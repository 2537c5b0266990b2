// crt — headless command-line host (replaces the GLFW/ImGui shell of reference src/main.cu:119-426):
//   main() -> config_task -> scene ingest -> set_BVH -> Render -> run_view -> save_frame_buffer,
// all through the C-ABI of include/crt.h.
#include <sys/stat.h>

#include <chrono>
#include <cmath>
#include <ctime>
#include <iostream>
#include <sstream>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/crt.h"

static bool exists(const std::string& p) { struct stat st; return stat(p.c_str(), &st) == 0; }
static std::string dir_of(const std::string& p) { size_t k = p.find_last_of('/'); return k == std::string::npos ? "." : p.substr(0, k); }
static std::string base_of(const std::string& p) {
    std::string q = p;
    while (!q.empty() && q.back() == '/') q.pop_back();
    size_t k = q.find_last_of('/');
    return k == std::string::npos ? q : q.substr(k + 1);
}
// The shipped configs name paths relative to build/Debug ("../../scenes/..."). The OBJ is looked up as
// given (cwd), under --root, next to the config file, and by file name next to the config file; MTL_dir
// is then taken relative to the same base (or is the config's directory).
static void resolve(const std::string& obj, const std::string& mtl, const std::string& root, const std::string& cfg_dir,
                    std::string* obj_out, std::string* mtl_out) {
    const bool absolute = !obj.empty() && obj[0] == '/';
    std::vector<std::string> bases = absolute ? std::vector<std::string>{""} : std::vector<std::string>{cfg_dir + "/", root + "/", ""};
    for (auto& b : bases) {
        if (!exists(b + obj)) continue;
        *obj_out = b + obj;
        std::string m = (!mtl.empty() && mtl[0] == '/') ? mtl : b + mtl;
        *mtl_out = exists(m) ? m : dir_of(*obj_out);
        return;
    }
    if (exists(cfg_dir + "/" + base_of(obj))) { *obj_out = cfg_dir + "/" + base_of(obj); *mtl_out = cfg_dir; return; }
    *obj_out = obj;
    *mtl_out = mtl;
}
// Little-endian PFM (scale -1.0), rows bottom first as the format requires; img is top row first, `channels` 3 (PF) or 1 (Pf).
static bool write_pfm(const std::string& path, const float* img, uint32_t width, uint32_t height, int channels) {
    FILE* f = fopen(path.c_str(), "wb");
    if (!f) return false;
    bool ok = fprintf(f, "%s\n%u %u\n-1.0\n", channels == 3 ? "PF" : "Pf", width, height) > 0;
    const size_t row = (size_t)width * channels;
    for (uint32_t y = height; ok && y-- > 0;) ok = fwrite(img + row * y, sizeof(float), row, f) == row;
    return (fclose(f) == 0) && ok;
}
// --aov PREFIX: PREFIX_albedo.pfm, PREFIX_normal.pfm, PREFIX_depth.pfm of the render (r) or group (g)
static int write_aov(const std::string& prefix, crt_render* r, crt_group* g, uint32_t width, uint32_t height) {
    const size_t n = (size_t)width * height;
    std::vector<float> albedo(3 * n), normal(3 * n), depth(n);
    const int rc = r ? crt_render_get_aov(r, albedo.data(), normal.data(), depth.data(), nullptr)
                     : crt_group_get_aov(g, albedo.data(), normal.data(), depth.data(), nullptr);
    if (rc != CRT_OK) { fprintf(stderr, "crt: get_aov failed: %s\n", crt_last_error()); return 1; }
    if (!write_pfm(prefix + "_albedo.pfm", albedo.data(), width, height, 3) || !write_pfm(prefix + "_normal.pfm", normal.data(), width, height, 3) ||
        !write_pfm(prefix + "_depth.pfm", depth.data(), width, height, 1)) {
        fprintf(stderr, "crt: cannot write %s_*.pfm\n", prefix.c_str());
        return 1;
    }
    return 0;
}
static double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// The reference's window without the window (src/main.cu:288-378): its widgets as commands read from stdin, the scene and the
// render object resident between frames as in its event loop. "render" is the Render button (main.cu:367-377: inverse view matrix
// from the current eye / lookat / up, run_view, "render cost"), "save" the Save button (main.cu:342-354: .tmp/<time>.png).
static int run_session(crt_render* render, crt_config cfg) {
    bool rendered = false;
    std::string line;
    auto fail = [](const char* what) { printf("{\"error\": \"%s: %s\"}\n", what, crt_last_error()); fflush(stdout); };
    while (std::getline(std::cin, line)) {
        std::istringstream in(line);
        std::string cmd;
        if (!(in >> cmd) || cmd[0] == '#') continue;
        if (cmd == "quit" || cmd == "exit") break;
        if (cmd == "eye" || cmd == "lookat" || cmd == "up") {
            float v[3];
            if (!(in >> v[0] >> v[1] >> v[2])) { printf("{\"error\": \"%s needs three numbers\"}\n", cmd.c_str()); fflush(stdout); continue; }
            float* dst = cmd == "eye" ? cfg.eye_pos : cmd == "lookat" ? cfg.lookat : cfg.up;
            memcpy(dst, v, sizeof(v));
            printf("{\"%s\": [%g, %g, %g]}\n", cmd.c_str(), v[0], v[1], v[2]);
        } else if (cmd == "spp" || cmd == "light_sample_n") {
            long n = 0;
            const long hi = cmd == "spp" ? 2048 : 64;                       // the sliders' ranges, main.cu:318,330
            if (!(in >> n) || n < 1) { printf("{\"error\": \"%s needs a positive integer\"}\n", cmd.c_str()); fflush(stdout); continue; }
            if (n > hi) fprintf(stderr, "crt: %s %ld is beyond the reference slider's range (%ld); accepted\n", cmd.c_str(), n, hi);
            if (cmd == "spp") { cfg.spp = (uint32_t)n; crt_render_set_spp(render, cfg.spp); }
            else { cfg.light_sample_n = (uint32_t)n; crt_render_set_light_sample_n(render, cfg.light_sample_n); }
            printf("{\"%s\": %ld}\n", cmd.c_str(), n);
        } else if (cmd == "p_rr" || cmd == "P_RR") {
            float p = 0;
            if (!(in >> p) || !(p >= 0.0f && p <= 1.0f)) { printf("{\"error\": \"p_rr needs a number in [0, 1]\"}\n"); fflush(stdout); continue; }
            cfg.p_rr = p;
            crt_render_set_p_rr(render, p);
            printf("{\"p_rr\": %g}\n", p);
        } else if (cmd == "render") {
            float M[9];
            crt_inverse_view_matrix(cfg.eye_pos, cfg.lookat, cfg.up, M);
            const double t0 = now_ms();
            if (crt_render_run_view(render, cfg.eye_pos, M, cfg.fov_y * (float)M_PI / 180.0f) != CRT_OK) { fail("run_view"); continue; }
            const double t1 = now_ms();
            crt_render_stats st;
            crt_render_get_stats(render, &st);
            rendered = true;
            printf("{\"render_cost_s\": %.6f, \"render_ms\": %.3f, \"msamples_per_s\": %.2f, \"spp\": %u}\n", (t1 - t0) * 1e-3, st.ms_total,
                   st.ms_total > 0 ? (double)st.samples / (st.ms_total * 1e3) : 0.0, cfg.spp);
        } else if (cmd == "save") {
            std::string path;
            if (!(in >> path)) {
                char stamp[64];
                const time_t now = time(nullptr);
                strftime(stamp, sizeof(stamp), "%Y-%m-%d-%H-%M-%S", localtime(&now));
                mkdir(".tmp", 0755);
                path = std::string(".tmp/") + stamp + ".png";
            }
            if (!rendered) { printf("{\"error\": \"save: nothing rendered yet\"}\n"); fflush(stdout); continue; }
            if (crt_render_save_png(render, path.c_str()) != CRT_OK) { fail("save_png"); continue; }
            printf("{\"saved\": \"%s\"}\n", path.c_str());
        } else {
            printf("{\"error\": \"unknown command %s\"}\n", cmd.c_str());
        }
        fflush(stdout);
    }
    return 0;
}

#define DIE_IF(rc, what) do { if ((rc) != CRT_OK) { fprintf(stderr, "crt: %s failed: %s\n", what, crt_last_error()); return 1; } } while (0)

int main(int argc, char** argv) {
    std::string config = "config.json", out = "out.png", root = ".";
    std::string checkpoint, aov;
    bool session = false;
    long spp = -1, seed = -1, width = -1, height = -1, chunk_spp = 64, stop_after = -1;
    int estimator = -1, device = 0, builder = CRT_BUILDER_PLOC8, gpus = 1;
    for (int i = 1; i < argc; ++i) {
        std::string a = argv[i];
        auto next = [&]() -> const char* { return i + 1 < argc ? argv[++i] : ""; };
        if (a == "--config") config = next();
        else if (a == "--out") out = next();
        else if (a == "--root") root = next();
        else if (a == "--spp") spp = atol(next());
        else if (a == "--seed") seed = atol(next());
        else if (a == "--width") width = atol(next());
        else if (a == "--height") height = atol(next());
        else if (a == "--device") device = atoi(next());
        else if (a == "--gpus") gpus = atoi(next());
        else if (a == "--estimator") { std::string e = next(); estimator = e == "mis" ? CRT_ESTIMATOR_MIS : CRT_ESTIMATOR_COMPAT; }
        else if (a == "--builder") { std::string e = next(); builder = e == "lbvh8" ? CRT_BUILDER_LBVH8 : e == "ploc" ? CRT_BUILDER_PLOC : e == "ploc8" ? CRT_BUILDER_PLOC8 : CRT_BUILDER_LBVH; }
        else if (a == "--checkpoint") checkpoint = next();
        else if (a == "--chunk-spp") chunk_spp = atol(next());
        else if (a == "--stop-after") stop_after = atol(next());
        else if (a == "--session") session = true;
        else if (a == "--aov") aov = next();
        else if (a == "--help" || a == "-h") {
            printf("usage: crt --config config.json [--root DIR] [--out image.png] [--spp N] [--seed S]\n"
                   "           [--width W --height H] [--estimator compat|mis] [--builder lbvh|lbvh8|ploc|ploc8] [--device D] [--gpus N]\n"
                   "           [--checkpoint FILE [--chunk-spp N] [--stop-after CHUNKS]] [--aov PREFIX]\n"
                   "  --checkpoint: progressive render in chunks of N samples per pixel (default 64); FILE is rewritten after\n"
                   "                every chunk and, if it exists at start, the render resumes from it (bit-identical image).\n"
                   "  --gpus N:     devices D .. D+N-1 render shares of the samples (the built scene is copied device to device), one\n"
                   "                NCCL reduce sums the accumulation buffers on device D; the image is the one a single GPU renders.\n"
                   "  --aov:        also write first-hit AOVs for a denoiser, over the same samples as the image: PREFIX_albedo.pfm,\n"
                   "                PREFIX_normal.pfm (3 channels) and PREFIX_depth.pfm (1 channel, +inf where no sample hit).\n"
                   "  --session:    the controls of the reference's window (src/main.cu:288-378) as commands on stdin, the scene staying\n"
                   "                resident between frames: eye X Y Z | lookat X Y Z | up X Y Z | spp N | p_rr P | light_sample_n N |\n"
                   "                render | save [FILE] (default .tmp/<time>.png) | quit. One JSON line per command on stdout.\n");
            return 0;
        } else { fprintf(stderr, "crt: unknown argument %s\n", a.c_str()); return 2; }
    }
    crt_config cfg;
    DIE_IF(crt_config_load(config.c_str(), &cfg), "config");
    if (spp > 0) cfg.spp = (uint32_t)spp;
    if (seed >= 0) cfg.seed = (uint32_t)seed;
    if (width > 0) cfg.width = (uint32_t)width;
    if (height > 0) cfg.height = (uint32_t)height;
    if (estimator >= 0) cfg.estimator = (uint32_t)estimator;
    const std::string cfg_dir = dir_of(config);

    crt_scene* scene = nullptr;
    DIE_IF(crt_scene_create(&scene), "scene_create");
    double t0 = now_ms();
    for (uint32_t k = 0; k < cfg.n_obj; ++k) {
        std::string obj, mtl;
        resolve(cfg.obj_path[k], cfg.mtl_dir[k], root, cfg_dir, &obj, &mtl);
        DIE_IF(crt_scene_add_obj(scene, obj.c_str(), mtl.c_str()), "add_obj");
    }
    double t1 = now_ms();
    float build_ms = 0;
    DIE_IF(crt_scene_build_bvh(scene, cfg.bvh_thresh_n, builder, device, &build_ms), "build_bvh");
    double t2 = now_ms();
    uint64_t n_tris = 0, n_nodes = 0; uint32_t n_mats = 0, n_lights = 0;
    crt_scene_counts(scene, &n_tris, &n_mats, &n_lights, &n_nodes);

    float M[9];
    crt_inverse_view_matrix(cfg.eye_pos, cfg.lookat, cfg.up, M);
    const float fovy_rad = cfg.fov_y * (float)M_PI / 180.0f;
    if (gpus > 1) {
        // several GPUs behind one handle (crt_group): this thread drives all of them
        if (!checkpoint.empty() || session) { fprintf(stderr, "crt: --checkpoint and --session render on one GPU (omit --gpus)\n"); return 2; }
        std::vector<int> devs;
        for (int k = 0; k < gpus; ++k) devs.push_back(device + k);
        crt_group* group = nullptr;
        double g0 = now_ms();
        DIE_IF(crt_group_create(scene, cfg.width, cfg.height, devs.data(), (uint32_t)devs.size(), &group), "group_create");
        DIE_IF(crt_group_set_params(group, cfg.spp, cfg.p_rr, cfg.light_sample_n, cfg.seed, (int)cfg.estimator), "group_set_params");
        if (!aov.empty()) DIE_IF(crt_group_set_aov(group, 1), "group_set_aov");
        double g1 = now_ms();
        DIE_IF(crt_group_run_view(group, cfg.eye_pos, M, fovy_rad), "group_run_view");
        double g2 = now_ms();
        DIE_IF(crt_group_save_png(group, out.c_str()), "group_save_png");
        if (!aov.empty() && write_aov(aov, nullptr, group, cfg.width, cfg.height) != 0) return 1;
        double g3 = now_ms();
        float reduce_ms = 0, slowest = 0;
        unsigned long long ext = 0, sh = 0, pr = 0;
        for (int k = 0; k < gpus; ++k) {
            crt_render_stats c;
            crt_group_get_stats(group, (uint32_t)k, &c, &reduce_ms);
            if (c.ms_total > slowest) slowest = c.ms_total;
            ext += c.extend_rays; sh += c.shadow_rays; pr += c.probe_rays;
        }
        const double total_samples = (double)cfg.width * cfg.height * cfg.spp;
        printf("{\"gpus\": %d, \"triangles\": %llu, \"nodes\": %llu, \"load_ms\": %.2f, \"bvh_build_gpu_ms\": %.3f, \"replicate_and_setup_ms\": %.2f, "
               "\"render_ms_slowest_gpu\": %.3f, \"reduce_ms\": %.3f, \"render_wall_ms\": %.2f, \"png_ms\": %.2f, \"msamples_per_s\": %.2f, "
               "\"extend_rays\": %llu, \"shadow_rays\": %llu, \"probe_rays\": %llu, \"out\": \"%s\"}\n",
               gpus, (unsigned long long)n_tris, (unsigned long long)n_nodes, t1 - t0, build_ms, g1 - g0, slowest, reduce_ms, g2 - g1, g3 - g2,
               total_samples / ((g2 - g1) * 1e3), ext, sh, pr, out.c_str());
        crt_group_destroy(group);
        crt_scene_destroy(scene);
        return 0;
    }
    crt_render* render = nullptr;
    DIE_IF(crt_render_create(scene, cfg.width, cfg.height, &render), "render_create");
    crt_render_set_spp(render, cfg.spp);
    crt_render_set_p_rr(render, cfg.p_rr);
    crt_render_set_light_sample_n(render, cfg.light_sample_n);
    crt_render_set_seed(render, cfg.seed);
    DIE_IF(crt_render_set_estimator(render, (int)cfg.estimator), "set_estimator");
    if (!aov.empty()) {
        if (session) { fprintf(stderr, "crt: --aov does not apply to --session\n"); return 2; }
        DIE_IF(crt_render_set_aov(render, 1), "set_aov");
    }
    if (session) {
        int rc = run_session(render, cfg);
        crt_render_destroy(render);
        crt_scene_destroy(scene);
        return rc;
    }
    double t3 = now_ms();
    crt_render_stats st;
    uint64_t samples_rendered = (uint64_t)cfg.width * cfg.height * cfg.spp, resumed_from = 0;
    if (checkpoint.empty()) {
        DIE_IF(crt_render_run_view(render, cfg.eye_pos, M, fovy_rad), "run_view");   // main.cu:372
        crt_render_get_stats(render, &st);
    } else {
        // progressive render with checkpoint / resume (SURVEY.md 8(f)2): chunks of the sample-major work index space
        const uint64_t npix = (uint64_t)cfg.width * cfg.height, total = npix * cfg.spp;
        const uint64_t chunk = npix * (uint64_t)(chunk_spp > 0 ? chunk_spp : 64);
        uint64_t done = 0;
        crt_render_set_accumulate(render, 1);
        if (exists(checkpoint)) {
            float ce[3], cM[9], cf;
            DIE_IF(crt_render_load_checkpoint(render, checkpoint.c_str(), &done, ce, cM, &cf), "load_checkpoint");
            if (memcmp(ce, cfg.eye_pos, sizeof(ce)) || memcmp(cM, M, sizeof(cM)) || memcmp(&cf, &fovy_rad, sizeof(cf))) {
                fprintf(stderr, "crt: checkpoint %s was rendered with a different camera\n", checkpoint.c_str());
                return 1;
            }
            resumed_from = done;
        } else {
            DIE_IF(crt_render_clear_accum(render), "clear_accum");
        }
        memset(&st, 0, sizeof(st));
        long chunks = 0;
        while (done < total) {
            const uint64_t end = done + chunk < total ? done + chunk : total;
            crt_render_set_work_range(render, done, end);
            DIE_IF(crt_render_run_view(render, cfg.eye_pos, M, fovy_rad), "run_view");
            crt_render_stats c;
            crt_render_get_stats(render, &c);
            st.ms_total += c.ms_total; st.extend_rays += c.extend_rays; st.shadow_rays += c.shadow_rays; st.probe_rays += c.probe_rays;
            st.iterations += c.iterations; st.kernel_launches += c.kernel_launches; st.samples += c.samples;
            done = end;
            DIE_IF(crt_render_save_checkpoint(render, checkpoint.c_str(), done), "save_checkpoint");
            if (stop_after > 0 && ++chunks >= stop_after) break;
        }
        samples_rendered = st.samples;
        if (done < total) {
            printf("{\"checkpoint\": \"%s\", \"work_done\": %llu, \"work_total\": %llu, \"resumed_from\": %llu, \"complete\": false}\n",
                   checkpoint.c_str(), (unsigned long long)done, (unsigned long long)total, (unsigned long long)resumed_from);
            crt_render_destroy(render);
            crt_scene_destroy(scene);
            return 0;
        }
    }
    double t4 = now_ms();
    DIE_IF(crt_render_save_png(render, out.c_str()), "save_png");
    if (!aov.empty() && write_aov(aov, render, nullptr, cfg.width, cfg.height) != 0) return 1;
    double t5 = now_ms();
    double msamples = st.ms_total > 0 ? (double)samples_rendered / (st.ms_total * 1e3) : 0.0;
    printf("{\"triangles\": %llu, \"nodes\": %llu, \"materials\": %u, \"lights\": %u, \"load_ms\": %.2f, \"bvh_build_gpu_ms\": %.3f, "
           "\"upload_and_build_ms\": %.2f, \"render_ms\": %.3f, \"render_wall_ms\": %.2f, \"png_ms\": %.2f, \"msamples_per_s\": %.2f, "
           "\"extend_rays\": %llu, \"shadow_rays\": %llu, \"probe_rays\": %llu, \"iterations\": %llu, \"resumed_from\": %llu, \"out\": \"%s\"}\n",
           (unsigned long long)n_tris, (unsigned long long)n_nodes, n_mats, n_lights, t1 - t0, build_ms, t2 - t1, st.ms_total, t4 - t3,
           t5 - t4, msamples, (unsigned long long)st.extend_rays, (unsigned long long)st.shadow_rays, (unsigned long long)st.probe_rays,
           (unsigned long long)st.iterations, (unsigned long long)resumed_from, out.c_str());
    crt_render_destroy(render);
    crt_scene_destroy(scene);
    return 0;
}
