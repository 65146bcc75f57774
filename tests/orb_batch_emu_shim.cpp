// csrc/orb.cu compiled for the host on top of tests/cuda_emu.h, with the extractor's handle exposed so that one object
// serves per-image calls (vo_orb_extract) and batched calls (vo_orb_extract_batch) in any order: the batch path, its
// scratch growth and its truncation run against the per-image path and the pinned CPU restatement in
// tests/test_orb_batch_emulation.py.  Test infrastructure only.
// Build: g++ -x c++ -std=c++17 -O2 -ffp-contract=off -pthread -DVO_HOST_EMU='"cuda_emu.h"' -I tests
#include "../visual-odometry-pipeline_b200/csrc/orb.cu"
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
void *emu_orb_create(int H, int W, int nfeatures, int nlevels, int fast_threshold) {
    memset(&g_ctx, 0, sizeof(g_ctx));
    vo_orb_config cfg = {H, W, nfeatures, nlevels, fast_threshold};
    vo_orb *o = nullptr;
    return vo_orb_create(&g_ctx, &cfg, &o) == VO_OK ? o : nullptr;
}
void emu_orb_destroy(void *o) { vo_orb_destroy((vo_orb *)o); }
int emu_orb_capacity(void *o) { return vo_orb_capacity((vo_orb *)o); }
int emu_orb_extract(void *o, const unsigned char *image, int channels, float *kp, unsigned char *desc, float *aux, int *count2) {
    return vo_orb_extract((vo_orb *)o, image, channels, kp, desc, aux, count2, nullptr);
}
int emu_orb_extract_batch(void *o, const unsigned char *images, int S, int channels, int out_rows, float *kp,
                          unsigned char *desc, float *aux, int *count) {
    return vo_orb_extract_batch((vo_orb *)o, images, S, channels, out_rows, kp, desc, aux, count, nullptr);
}
}
