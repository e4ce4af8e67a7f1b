/* rt3_main.cpp — command-line driver of the host backend: the shape of reference src/Main.cpp:246-315
 * (create renderer, camera, entities; prerender; render; save), with the scene chosen by name.
 *
 *   rt3_render [-W width] [-H height] [-s scene] [-o out.ppm|out.png] [--teddy path/to/teddy.obj]
 *              [--pathtrace] [--spp n] [--depth n] [--seed n] [--analytic] [--passes k] [--pfm out.pfm]
 *              [--aov DIR] [--aov-spp n] [--denoise]
 *   --pathtrace / --spp / --depth / --seed: CudaRenderSettings (default: the reference's ray caster); --analytic keeps
 *   ECS spheres analytic; --passes k renders k progressive passes of spp samples each (render_progressive) and writes
 *   the frame after every pass to <out>.<pass>.<ext>; --pfm also writes the linear float radiance (path tracing only); --aov writes the AOVs of the path tracer's primary
 *   rays (albedo.pfm, normal.pfm, depth.pfm: what a denoiser takes next to the colour) into DIR, from the first --aov-spp
 *   samples of every pixel (default: --spp); --denoise runs that AOV pass too and writes the frame denoised by it
 *   (CudaRenderer::denoise: edge-avoiding à-trous filter, SVGF's defaults) to <out> instead of the noisy one.
 *   scenes: default (reference Main.cpp:280-283, needs --teddy), triangle, sphere, rtiow (path traced, C1),
 *           or the path of a SceneLang file (*.scene)
 */
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

#include <CppDebugger.hpp>

#include "entities/Triangle.hpp"
#include "entities/Sphere.hpp"
#include "entities/Object.hpp"
#include "renderer/CudaRenderer.hpp"
#include "sceneparser/SceneParser.hpp"

using namespace RayTracer;

int main(int argc, const char** argv) {
    uint32_t width = 800, height = 600; /* reference defaults, Main.cpp:78-79 */
    std::string scene = "triangle", out = "result.ppm", teddy = "bin/objects/teddy.obj", pfm, aov_dir;
    bool pathtrace = false, analytic = false, denoise = false;
    uint32_t spp = 0, depth = 0, seed = 0, passes = 1, aov_spp = 0;
    for (int i = 1; i < argc; i++) {
        std::string a = argv[i];
        auto next = [&]() -> const char* { if (i + 1 >= argc) { std::fprintf(stderr, "missing value for %s\n", a.c_str()); std::exit(1); } return argv[++i]; };
        if (a == "-W") { width = (uint32_t) std::strtoul(next(), nullptr, 0); }
        else if (a == "-H") { height = (uint32_t) std::strtoul(next(), nullptr, 0); }
        else if (a == "-s") { scene = next(); }
        else if (a == "-o") { out = next(); }
        else if (a == "--teddy") { teddy = next(); }
        else if (a == "--pathtrace") { pathtrace = true; }
        else if (a == "--analytic") { analytic = true; }
        else if (a == "--spp") { spp = (uint32_t) std::strtoul(next(), nullptr, 0); pathtrace = true; }
        else if (a == "--depth") { depth = (uint32_t) std::strtoul(next(), nullptr, 0); }
        else if (a == "--seed") { seed = (uint32_t) std::strtoul(next(), nullptr, 0); }
        else if (a == "--pfm") { pfm = next(); pathtrace = true; }
        else if (a == "--aov") { aov_dir = next(); pathtrace = true; }
        else if (a == "--aov-spp") { aov_spp = (uint32_t) std::strtoul(next(), nullptr, 0); }
        else if (a == "--denoise") { denoise = true; pathtrace = true; }
        else if (a == "--passes") { passes = (uint32_t) std::strtoul(next(), nullptr, 0); pathtrace = true; }
        else { std::fprintf(stderr, "usage: %s [-W w] [-H h] [-s default|triangle|sphere|rtiow|file.scene] [-o out.ppm|out.png] [--teddy file] "
                               "[--pathtrace] [--spp n] [--depth n] [--seed n] [--analytic] [--passes k] [--pfm out.pfm] [--aov DIR] [--aov-spp n] [--denoise]\n", argv[0]); return a == "-h" ? 0 : 1; }
    }
    try {
        Renderer* renderer = initialize_renderer();
        CudaRenderer* cuda = (CudaRenderer*) renderer;
        Camera cam;
        Tools::Array<ECS::RenderEntity*> entities;
        if (scene == "default") {
            entities.push_back(ECS::create_object(teddy, {0.0f, 0.0f, -3.0f}, 1.0f / 17.0f, {1.0f, 0.0f, 0.0f}));
            entities.push_back(ECS::create_sphere({-2.0f, 0.0f, -5.0f}, 1.0f, 8, 8, {0.0f, 0.0f, 1.0f}));
        } else if (scene.size() > 6 && scene.compare(scene.size() - 6, 6, ".scene") == 0) {
            ParsedScene parsed;                                  /* SceneLang file (reference src/lib/sceneparser/SceneLang.md) */
            SceneParser::parse_file(scene, parsed);
            for (const std::string& w : parsed.warnings) { std::fprintf(stderr, "warning: %s\n", w.c_str()); }
            for (size_t i = 0; i < parsed.entities.size(); i++) { entities.push_back(parsed.entities[i]); }
        } else if (scene == "sphere") {
            entities.push_back(ECS::create_sphere({0.0f, 0.0f, -3.0f}, 1.0f, 8, 8, {1.0f, 0.0f, 0.0f}));
        } else if (scene == "rtiow") {
            entities.push_back(ECS::create_sphere({0.0f, -100.5f, -1.0f}, 100.0f, 8, 8, {0.8f, 0.8f, 0.0f}));
            entities.push_back(ECS::create_sphere({0.0f, 0.0f, -1.0f}, 0.5f, 8, 8, {0.1f, 0.2f, 0.5f}));
            entities.push_back(ECS::create_sphere({-1.0f, 0.0f, -1.0f}, 0.5f, 8, 8, {1.0f, 1.0f, 1.0f}));
            entities.push_back(ECS::create_sphere({1.0f, 0.0f, -1.0f}, 0.5f, 8, 8, {0.8f, 0.6f, 0.2f}));
            CudaRenderSettings st = cuda->get_settings();
            st.mode = RT3_MODE_PATHTRACE; st.analytic_spheres = true;
            cuda->set_settings(st);
            Material glass; glass.kind = Material::dielectric; glass.ior = 1.5f;
            Material gold; gold.kind = Material::metal; gold.albedo = glm::vec3(0.8f, 0.6f, 0.2f);
            cuda->set_material(2, glass);
            cuda->set_material(3, gold);
        } else {
            entities.push_back(ECS::create_triangle({1.0f, 0.0f, -3.0f}, {-1.0f, 0.0f, -3.0f}, {0.0f, 1.0f, -3.0f}, {1.0f, 0.0f, 0.0f}));
        }
        {
            CudaRenderSettings st = cuda->get_settings();
            if (pathtrace) { st.mode = RT3_MODE_PATHTRACE; }
            if (analytic) { st.analytic_spheres = true; }
            if (spp) { st.spp = spp; }
            if (depth) { st.max_depth = depth; }
            if (seed) { st.seed = seed; }
            st.aov_spp = aov_spp;
            cuda->set_settings(st);
        }
        if (scene == "rtiow") { cam.update(width, height, 1.0f, ((float) width / (float) height) * 2.0f, 2.0f); }
        else { cam.update(width, height, 2.0f, ((float) width / (float) height) * 2.0f, 2.0f); }
        auto save = [&](const Frame& frame, const std::string& path) {
            if (path.size() > 4 && path.compare(path.size() - 4, 4, ".png") == 0) { frame.to_png(path); } else { frame.to_ppm(path); }
        };
        renderer->prerender(entities);
        if (passes > 1) {
            struct Sink { const std::string* out; decltype(save)* writer; } sink = { &out, &save };
            cuda->render_progressive(cam, passes, [](uint32_t pass, const Frame& frame, void* user) {
                Sink* k = (Sink*) user;
                const size_t dot = k->out->find_last_of('.');
                const std::string stem = dot == std::string::npos ? *k->out : k->out->substr(0, dot), ext = dot == std::string::npos ? "" : k->out->substr(dot);
                (*k->writer)(frame, stem + "." + std::to_string(pass) + ext);
            }, &sink);
        } else {
            renderer->render(cam);
        }
        for (size_t i = 0; i < entities.size(); i++) {
            if (entities[i]->type == ECS::et_object) { delete (ECS::Object*) entities[i]; }
            else if (entities[i]->type == ECS::et_sphere) { delete (ECS::Sphere*) entities[i]; }
            else { delete (ECS::Triangle*) entities[i]; }
        }
        if (!denoise) { save(cam.get_frame(), out); }
        if (!pfm.empty()) { cuda->write_radiance_pfm(width, height, pfm); }
        std::printf("%s: %ux%u, %.3f ms on the device, %llu rays -> %s\n", scene.c_str(), width, height, cuda->stats().device_ms,
                    (unsigned long long) cuda->stats().rays, denoise ? "denoiser" : out.c_str());
        if (!aov_dir.empty() || denoise) {
            CudaPathAovs aovs;
            cuda->render_path_aovs(cam, aovs);
            if (!aov_dir.empty()) { cuda->write_path_aovs_pfm(aovs, aov_dir); }
            std::printf("AOVs: %u samples per pixel, %.3f ms on the device -> %s\n", cuda->get_settings().aov_spp ? cuda->get_settings().aov_spp : cuda->get_settings().spp,
                        cuda->stats().device_ms, aov_dir.empty() ? "denoiser" : (aov_dir + "/{albedo,normal,depth}.pfm").c_str());
        }
        if (denoise) {
            cuda->denoise(cam);
            save(cam.get_frame(), out);
            std::printf("denoised: %u kernels, %.3f ms on the device -> %s\n", cuda->stats().kernel_launches, cuda->stats().device_ms, out.c_str());
        }
        delete renderer;
    } catch (CppDebugger::Fatal& e) {
        std::fprintf(stderr, "fatal: %s\n", e.what());
        return -1;
    }
    return 0;
}
