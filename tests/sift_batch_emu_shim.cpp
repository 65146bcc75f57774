// csrc/sift.cu compiled for the host on top of tests/cuda_emu.h, with the extractor's handle exposed so that one object
// serves per-image calls (vo_sift_extract) and batched calls (vo_sift_extract_batch) in any order: the batch path, its
// scratch growth, its truncation and its flags run against the per-image path in tests/test_sift_batch_emulation.py.
// Test infrastructure only.
// Build: g++ -x c++ -std=c++17 -O2 -ffp-contract=off -fno-gnu-unique -pthread -DVO_HOST_EMU='"cuda_emu.h"' -I tests
#include "../visual-odometry-pipeline_b200/csrc/sift.cu"
#include <stdio.h>

namespace vo {
static char g_err[512];
void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
const char *get_error() { return g_err; }
void clear_error() { g_err[0] = 0; }
}  // namespace vo

static vo_ctx g_ctx;

extern "C" {
const char *emu_last_error() { return vo::get_error(); }
long long emu_launches() { return vo_emu::g_launches; }
void *emu_sift_create(int H, int W, int max_keypoints) {
    memset(&g_ctx, 0, sizeof(g_ctx));
    vo_sift_config cfg = {H, W, max_keypoints};
    vo_sift *s = nullptr;
    return vo_sift_create(&g_ctx, &cfg, &s) == VO_OK ? s : nullptr;
}
void emu_sift_destroy(void *s) { vo_sift_destroy((vo_sift *)s); }
int emu_sift_extract(void *s, const unsigned char *image, int channels, float *kp, float *desc, float *aux, int *count2) {
    return vo_sift_extract((vo_sift *)s, image, channels, kp, desc, aux, count2, nullptr);
}
int emu_sift_extract_batch(void *s, const unsigned char *images, int S, int channels, int out_rows, float *kp, float *desc,
                           float *aux, int *count) {
    return vo_sift_extract_batch((vo_sift *)s, images, S, channels, out_rows, kp, desc, aux, count, nullptr);
}
}
