// Camera rays of the AOV pass, stated with the CPU oracle's own pieces: orc::primary_ray (oracle/orc_render.cpp) and the
// Philox draw the oracle's estimators use for the camera jitter, draw(pixel, sample, kCameraBounce, 0, seed) with key
// (seed, "CRT1"). Built by tests/aov_reference.py against oracle/liborc.so; the rays are then traced by the oracle's
// closest-hit traversal (orc_trace).
#include "../oracle/orc_render.h"

using namespace orc;

extern "C" {

// Work items w in [w_begin, w_end) of the sample-major index space w = sample * W*H + pixel: ray k = w - w_begin as
// {o, FLT_MAX, d, 0} in rays[8k..8k+7], its pixel in pixel_out[k].
void aov_camera_rays(const float eye[3], const float M[9], float fovy_rad, int width, int height, uint64_t w_begin,
                     uint64_t w_end, uint32_t seed, float* rays, int32_t* pixel_out) {
    Camera cam;
    cam.eye = V3{eye[0], eye[1], eye[2]};
    for (int k = 0; k < 9; ++k) cam.M[k] = M[k];
    cam.tan_half = tanf(fovy_rad / 2);                    // Render.cuh:338, as crt_render_run_view evaluates it
    const uint64_t npix = (uint64_t)width * (uint64_t)height;
    for (uint64_t w = w_begin; w < w_end; ++w) {
        const uint32_t pixel = (uint32_t)(w % npix), sample = (uint32_t)(w / npix);
        const U4 r = philox4x32_10(U4{pixel, sample, 0xFFFFFFFFu, 0u}, seed, 0x43525431u);
        const Ray ray = primary_ray(cam, width, height, (int)(pixel % (uint32_t)width), (int)(pixel / (uint32_t)width), u01(r.x), u01(r.y));
        float* o = rays + 8 * (w - w_begin);
        o[0] = ray.o.x; o[1] = ray.o.y; o[2] = ray.o.z; o[3] = FLT_MAX;
        o[4] = ray.d.x; o[5] = ray.d.y; o[6] = ray.d.z; o[7] = 0.0f;
        pixel_out[w - w_begin] = (int32_t)pixel;
    }
}

}  // extern "C"
