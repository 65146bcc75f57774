// Float-descriptor matcher on the 5th-generation tensor cores (VO_PREC_TF32X3 / VO_PREC_TF32X1).
//
// Replaces `sim = d1 @ d2.t(); topk(sim, 2, dim=1); max(sim, dim=0)` of the reference's torch matchers
// (R2D2.py:56-60: cuBLAS SGEMM + two more passes over a materialised N x M matrix) and the brute-force
// distance matrix of cv2.BFMatcher.knnMatch (feature_extractors/SIFT.py:27).  Here the N x M similarity
// matrix lives only in tensor memory:
//
//   * one CTA owns a 128-row block of the reference descriptors (A).  A is written ONCE into tensor memory
//     (tcgen05.st, 128 columns for the tf32 "hi" part, 128 for the "lo" part) and stays there: the MMAs take
//     A from TMEM, so shared memory holds nothing but the B ring and the MMA reads only B from it;
//   * 128-column x 32-k boxes of the current-frame descriptors (B) stream through a 13-stage TMA/mbarrier
//     ring (208 KB in flight per SM).  Two CTAs (adjacent row blocks) form a cluster and each issues every other
//     box with .multicast::cluster, so each box crosses L2 -> SM once per pair of SMs;
//   * a single thread issues tcgen05.mma.cta_group::1.kind::tf32 (M=128, N=128, K=8) into one of two
//     128-column fp32 accumulators.  3xTF32: every k-step issues lo*hi, hi*hi and hi*lo, which restores
//     fp32-grade products; for integer-valued SIFT descriptors one pass is already exact (every product and
//     partial sum is an integer < 2^24);
//   * two groups of four epilogue warps (one group per accumulator) read the tile with tcgen05.ld and fold it
//     into a running top-2 per row (thread-private, one row per thread) and a per-column arg-max
//     (redux.sync.max.f32 + ballot across the 32 rows of a warp, 4 warps merged in shared memory, one 64-bit
//     atomicMin per column and CTA), while the MMA thread already fills the other accumulator.
//
// L2 mode uses the GEMM form -|a_i - b_j|^2 = (2 a_i.b_j - |b_j|^2) - |a_i|^2, evaluated per element in the
// epilogue (the row norm matters for the column arg-min, the column norm for the row arg-min).
//
// Operand arithmetic (template parameter PASSES):
//    3  3xTF32      hi/lo tf32 split, three kind::tf32 MMAs per 8 k            R2D2 default (fp32-grade)
//    1  1xTF32      single tf32 pass, column norm as an extra K-step           integer-valued data, rules with a column side
//   16  1xFP16      single fp16 pass (kind::f16, K = 16), 192-column tiles     integer-valued data: SIFT, ORB bytes (exact)
//   48  3xFP16      x * 2^8 = hi + lo in fp16, three kind::f16 MMAs per 16 k   the 22 operand bits of 3xTF32 at twice the rate
//    8  1xFP8/256   256-bit descriptors as 256-d rows of e4m3 -1 / +1         a.b = 256 - 2 Hamming (exact), kind::f8f6f4 (K = 32),
//                                                                              K = 256, no norms (as fp16 rows: twice the bytes and MMAs)
//    9  the same, row arg-max only (no second best)                            mutual-NN rule without k-NN output; the swapped pass
// The two fp16 modes use the all-warp epilogue (16 warps on every tile, accumulator released right after the TMEM read,
// the four threads of a row share their filter threshold); tools/probe/mma_issue_probe.cu has the pipe rates.
#include "common.cuh"
#include "tc_ptx.cuh"
#include <cuda_fp16.h>
#include <stdlib.h>

// Work items (row-block pair x column split x frame pair) with at most this many column tiles run on the persistent form of the
// fp16 / fp8 passes: at 11 tiles (2k x 2k) the per-CTA set-up and drain is as long as the tiles, at 105 (20k x 20k) it is 2 %
// and the plain form's steady state is 6 % faster (B200: 2k +9 %, 5k +5 % / +2 %, 20k -6 % persistent vs plain).
#ifndef VO_TC_PERSIST_MAX_TILES
#define VO_TC_PERSIST_MAX_TILES 64
#endif

namespace vo {
namespace {

constexpr int TC_BM = 128;      // rows of A per CTA (= TMEM lanes)
constexpr int TC_BN = 128;      // columns per B tile (= accumulator columns), 3xTF32; single pass uses TcCfg<1>::BN
constexpr int TC_D = 128;       // descriptor length
constexpr int TC_KB = 32;       // k elements per swizzle-128B row (32 fp32 = 128 B)
constexpr int TC_NKB = TC_D / TC_KB;
// the norm extension of the single passes (one more K-step: ones[128 x 8] * (-|b|^2 as three tf32 pieces, zeros)[8 x BN]) travels
// as 8 floats = 32 B per column through a SWIZZLE_32B box — a quarter of the bytes of a 128-byte row
constexpr int TC_EXT_K = 8;
// Per-mode tile geometry.  3xTF32: 128-column tiles, 13-stage ring of 16 KB boxes, TMEM = acc0 0 | acc1 128 | A_hi 256 |
// A_lo 384.  Single pass has no A_lo, so the accumulators can be wider: 160-column tiles (27 % fewer tcgen05.mma per
// FLOP — the single-pass kernel is bound by the MMA-issuing thread, not by the pipe), 10-stage ring of 20 KB boxes,
// TMEM = acc0 0 | acc1 160 | ones block of the norm extension 320 | A_hi 384.
// PASSES == 16 selects the fp16 single pass (VO_PREC_F16X1): operands rounded to fp16 (11 significant bits like tf32,
// so integer-valued SIFT descriptors stay exact), tcgen05.mma.kind::f16 with K = 16 per instruction at twice the tf32
// rate.  192-column tiles, 9-stage ring of 24 KB boxes ([192 rows x 64 k] fp16), A as 64 packed columns:
// TMEM = acc0 0 | acc1 192 | ones block 384 | A 416.
// PASSES == 48 is the split form of the same idea (VO_PREC_F16X3): x * 2^8 = hi + lo with hi, lo in fp16 carries the same
// 22 operand bits as the tf32 hi/lo split (the scaling keeps the lo parts of unit-norm descriptors out of the fp16
// subnormals; 2^-16 is taken off the accumulator in the epilogue, exactly), three kind::f16 MMAs per 16 k instead of
// three kind::tf32 MMAs per 8 k.  Tile geometry, ring and epilogue are those of 3xTF32.
template <int PASSES>
struct TcCfg {
    static constexpr bool F8 = PASSES == 8 || PASSES == 9;        // e4m3 operands, tcgen05.mma.kind::f8f6f4 (128 k per 128-byte box)
    static constexpr bool TOP1 = PASSES == 9;                     // row arg-max only: the fold keeps (s1, i1), half the filter hits
    static constexpr bool K256 = F8;                              // single pass over 256-d rows (bit descriptors as -1 / +1)
    static constexpr bool F16 = PASSES == 16 || K256;             // fp16 / fp8 single pass (own epilogue)
    static constexpr int KBOX = F8 ? 128 : 64;                    // k per box of the 16- and 8-bit passes
    static constexpr bool H16 = F16 || PASSES == 48;              // fp16 operands
    static constexpr bool THREE = PASSES == 3 || PASSES == 48;    // hi/lo split, three MMAs per k-step
    static constexpr bool ALLWARP_COLS = PASSES == 48;            // all-warp epilogue with the column side
    static constexpr int KDIM = K256 ? 256 : TC_D;                // descriptor length the kernel contracts over
    static constexpr bool SINGLE = !THREE;
    static constexpr int ALO = H16 ? 64 : TC_D;                   // TMEM columns from A_hi to A_lo
    static constexpr int BN = F16 ? 192 : (SINGLE ? 160 : 128);
    static constexpr int STAGES = F16 ? 9 : (SINGLE ? 10 : 13);
    static constexpr int BLOCK_BYTES = BN * 128;                  // one [BN rows x 128 B] box: 32 fp32 or 64 fp16 along k
    static constexpr int TMEM_A = K256 ? 384 : (F16 ? 416 : (SINGLE ? 384 : 256));  // first column of A_hi (A_lo follows in 3xTF32)
    static constexpr int TMEM_EXT = F16 ? 384 : 320;              // single pass only
    static constexpr int OFF_SCOL = STAGES * BLOCK_BYTES;         // [2 groups][2 bufs][4 quarters][BN] x (float, u32)
    // column scratch, (float, u32) per entry: [2 groups][2 bufs][4 quarters][BN]; the all-warp epilogue of the split fp16
    // pass needs [2 bufs][4][BN]; the fp16 single pass has no column side
    static constexpr int SCOL_N = F16 ? 0 : (ALLWARP_COLS ? 2 * 4 * BN : 2 * 2 * 4 * BN);
    static constexpr int OFF_ROW2 = OFF_SCOL + SCOL_N * 8;
    static constexpr int OFF_BAR = OFF_ROW2 + (H16 ? 4 * TC_BM * 4 : 0);        // [4 column quarters][128 rows] shared second-bests
    static constexpr int SMEM_BYTES = OFF_BAR + 512 + 1024;       // barriers + alignment slack
    static_assert(SMEM_BYTES <= 232448, "dynamic shared memory of one CTA (227 KB)");
    static constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
    // kind::f16: D = f32 [4,6) = 1, A = B = fp16 (format 0)
    static constexpr uint32_t IDESC16 = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
    static constexpr float ACC_SCALE = PASSES == 48 ? 1.0f / 65536.0f : 1.0f;  // accumulator -> a.b
};
constexpr int TC_THREADS = 576;              // warps 0..15 epilogue, warp 16 TMA, warp 17 MMA
constexpr int TC_WARP_TMA = 16, TC_WARP_MMA = 17;
constexpr int TC_TMEM_COLS = 512;            // 2 accumulators x 128 | A_hi 128 | A_lo 128
constexpr int TC_CLUSTER = 2;

using namespace tc;

// instruction descriptor (cute::UMMA::InstrDescriptor): D=f32 [4,6)=1, A=tf32 [7,10)=2, B=tf32 [10,13)=2,
// A,B K-major (bits 15,16 = 0), N>>3 [17,23), M>>4 [24,29) — TcCfg<>::IDESC

// ---------------------------------------------------------------- pre-pass: tf32 split + squared norms

// one warp per descriptor row (128 floats = 32 lanes x float4)
// ext (optional, [rows][32]): -|x|^2 split into three tf32 pieces in columns 0..2, zeros elsewhere — the extra
// K-step that lets the MMA itself subtract the column norm (single-pass L2 mode).
__global__ void __launch_bounds__(256)
prep_kernel(const float *__restrict__ x, long long rows, float *__restrict__ hi, float *__restrict__ lo,
            float *__restrict__ norm2, float *__restrict__ ext) {
    const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    const float4 v = reinterpret_cast<const float4 *>(x)[row * 32 + lane];
    float4 h = make_float4(to_tf32(v.x), to_tf32(v.y), to_tf32(v.z), to_tf32(v.w));
    reinterpret_cast<float4 *>(hi)[row * 32 + lane] = h;
    if (lo) {
        float4 l = make_float4(to_tf32(v.x - h.x), to_tf32(v.y - h.y), to_tf32(v.z - h.z), to_tf32(v.w - h.w));
        reinterpret_cast<float4 *>(lo)[row * 32 + lane] = l;
    }
    if (norm2) {
        float s = __fadd_rn(__fadd_rn(__fmul_rn(v.x, v.x), __fmul_rn(v.y, v.y)), __fadd_rn(__fmul_rn(v.z, v.z), __fmul_rn(v.w, v.w)));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s = __fadd_rn(s, __shfl_xor_sync(0xffffffffu, s, o));
        if (lane == 0) norm2[row] = s;
        if (ext) {
            float4 e = make_float4(0.f, 0.f, 0.f, 0.f);
            if (lane == 0) {
                const float n1 = to_tf32(s), n2 = to_tf32(__fsub_rn(s, n1));
                const float n3 = to_tf32(__fsub_rn(__fsub_rn(s, n1), n2));
                e = make_float4(-n1, -n2, -n3, 0.f);
            }
            if (lane < TC_EXT_K / 4) reinterpret_cast<float4 *>(ext)[row * (TC_EXT_K / 4) + lane] = e;
        }
    }
}

// fp16 single pass: x -> fp16 (round to nearest even), norms and extension rows as above (from the fp32 values)
__global__ void __launch_bounds__(256)
prep16_kernel(const float *__restrict__ x, long long rows, __half *__restrict__ h16, float *__restrict__ norm2,
              float *__restrict__ ext) {
    const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    const float4 v = reinterpret_cast<const float4 *>(x)[row * 32 + lane];
    const __half2 p0 = __floats2half2_rn(v.x, v.y), p1 = __floats2half2_rn(v.z, v.w);
    uint2 w;
    w.x = *reinterpret_cast<const uint32_t *>(&p0);
    w.y = *reinterpret_cast<const uint32_t *>(&p1);
    reinterpret_cast<uint2 *>(h16)[row * 32 + lane] = w;
    if (norm2) {
        float s = __fadd_rn(__fadd_rn(__fmul_rn(v.x, v.x), __fmul_rn(v.y, v.y)), __fadd_rn(__fmul_rn(v.z, v.z), __fmul_rn(v.w, v.w)));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s = __fadd_rn(s, __shfl_xor_sync(0xffffffffu, s, o));
        if (lane == 0) norm2[row] = s;
        if (ext) {
            float4 e = make_float4(0.f, 0.f, 0.f, 0.f);
            if (lane == 0) {
                const float n1 = to_tf32(s), n2 = to_tf32(__fsub_rn(s, n1));
                const float n3 = to_tf32(__fsub_rn(__fsub_rn(s, n1), n2));
                e = make_float4(-n1, -n2, -n3, 0.f);
            }
            if (lane < TC_EXT_K / 4) reinterpret_cast<float4 *>(ext)[row * (TC_EXT_K / 4) + lane] = e;
        }
    }
}

// byte descriptors as fp16 rows: ROW_BYTES = 32 (the reference's ORB semantics: BFMatcher NORM_L2 over byte values; the matcher
// treats them as 128-d rows that are zero beyond the 32nd element — TMA out-of-bounds fill for B, a bounds test in the A load)
// or 128 (SIFT descriptors shipped as uint8: they are integers 0..255, a quarter of the float32 bytes over the bus).  Every
// value, product and partial sum is an exact integer, as for float32 SIFT.
template <int ROW_BYTES>
__global__ void __launch_bounds__(256)
prep16_u8_kernel(const uint8_t *__restrict__ x, long long rows, __half *__restrict__ h16, float *__restrict__ norm2,
                 float *__restrict__ ext) {
    constexpr int LPR = ROW_BYTES / 4, RPW = 32 / LPR;   // lanes per row (4 bytes each), rows per warp
    const int lane = threadIdx.x & 31, sub = lane % LPR;
    const long long row = (long long)blockIdx.x * (8 * RPW) + (threadIdx.x >> 5) * RPW + lane / LPR;
    const bool ok = row < rows;
    float s = 0.f;
    if (ok) {  // compact fp16 rows of ROW_BYTES values
        const uchar4 v = reinterpret_cast<const uchar4 *>(x)[row * LPR + sub];
        const __half2 p0 = __floats2half2_rn((float)v.x, (float)v.y), p1 = __floats2half2_rn((float)v.z, (float)v.w);
        uint2 w;
        w.x = *reinterpret_cast<const uint32_t *>(&p0);
        w.y = *reinterpret_cast<const uint32_t *>(&p1);
        s = (float)((int)v.x * v.x + (int)v.y * v.y + (int)v.z * v.z + (int)v.w * v.w);
        reinterpret_cast<uint2 *>(h16)[row * LPR + sub] = w;
    }
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) s = __fadd_rn(s, __shfl_xor_sync(0xffffffffu, s, o));  // integers < 2^24: exact
    if (!ok) return;
    if (sub == 0) norm2[row] = s;
    if (ext && sub < TC_EXT_K / 4) {
        float4 e = make_float4(0.f, 0.f, 0.f, 0.f);
        if (sub == 0) {
            const float n1 = to_tf32(s), n2 = to_tf32(__fsub_rn(s, n1));
            const float n3 = to_tf32(__fsub_rn(__fsub_rn(s, n1), n2));
            e = make_float4(-n1, -n2, -n3, 0.f);
        }
        reinterpret_cast<float4 *>(ext)[row * (TC_EXT_K / 4) + sub] = e;
    }
}

// 256-bit descriptors (VO_NORM_HAMMING_TC) as 256-d rows of -1 / +1: a.b = (#equal bits) - (#different bits) =
// 256 - 2 popcount(a xor b), an exact small integer in the fp32 accumulator, and no norm enters: the matcher's cosine
// machinery (larger is closer) orders by Hamming distance.  The values are e4m3 bytes (+1.0 = 0x38, -1.0 = 0xb8; as fp16
// the pass moved twice the bytes and issued twice the MMAs: 5.40 -> 4.41 ms per 250 pairs of 5k x 5k): 256 B per
// descriptor, one warp per descriptor, one byte of bits -> 8 bytes per lane.
__global__ void __launch_bounds__(256)
prep_bits8_kernel(const uint8_t *__restrict__ x, long long rows, uint8_t *__restrict__ f8) {
    const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    const uint32_t v = x[row * 32 + lane];
    uint32_t w[2];
#pragma unroll
    for (int i = 0; i < 2; ++i) {   // bit set -> sign clear
        const uint32_t n = ~(v >> (4 * i));
        w[i] = 0x38383838u | ((n & 1u) << 7) | ((n & 2u) << 14) | ((n & 4u) << 21) | ((n & 8u) << 28);
    }
    *reinterpret_cast<uint2 *>(f8 + row * 256 + lane * 8) = make_uint2(w[0], w[1]);
}

// Second pass of the tensor-core Hamming matcher (roles swapped: current-frame descriptors as rows): the row arg-max of every
// current descriptor IS the column arg-min of the first pass.  Merges the per-split partials (ties -> lower reference row,
// the rule of the fused column arg-min) into the colkey format finalize reads: ordered(-score) << 32 | reference row.
__global__ void __launch_bounds__(256)
colkey_from_partials_kernel(const vo_row_best *__restrict__ part, int n_split, int m_stride, const int32_t *__restrict__ n_cur,
                            unsigned long long *__restrict__ colkey) {
    const int b = blockIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m_stride) return;
    const int M = n_cur ? min(n_cur[b], m_stride) : m_stride;
    unsigned long long best = ~0ull;
    if (j < M)
        for (int sp = 0; sp < n_split; ++sp) {
            const vo_row_best p = part[((size_t)b * n_split + sp) * m_stride + j];   // the swapped pass keeps row bests only
            if (p.i1 >= 0) {
                const unsigned long long key = ((unsigned long long)p.s1 << 32) | (unsigned long long)(uint32_t)p.i1;
                best = key < best ? key : best;
            }
        }
    colkey[(size_t)b * m_stride + j] = best;
}

// split fp16 (VO_PREC_F16X3): x * 2^8 = hi + lo, both fp16; squared norms of the unscaled rows
__global__ void __launch_bounds__(256)
prep16x3_kernel(const float *__restrict__ x, long long rows, __half *__restrict__ hi16, __half *__restrict__ lo16,
                float *__restrict__ norm2) {
    const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    const float4 v = reinterpret_cast<const float4 *>(x)[row * 32 + lane];
    const float e[4] = {v.x * 256.0f, v.y * 256.0f, v.z * 256.0f, v.w * 256.0f};  // exact scaling
    __half h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        h[i] = __float2half_rn(e[i]);
        l[i] = __float2half_rn(e[i] - __half2float(h[i]));  // the residual is exact in fp32
    }
    uint2 wh, wl;
    wh.x = (uint32_t)__half_as_ushort(h[0]) | ((uint32_t)__half_as_ushort(h[1]) << 16);
    wh.y = (uint32_t)__half_as_ushort(h[2]) | ((uint32_t)__half_as_ushort(h[3]) << 16);
    wl.x = (uint32_t)__half_as_ushort(l[0]) | ((uint32_t)__half_as_ushort(l[1]) << 16);
    wl.y = (uint32_t)__half_as_ushort(l[2]) | ((uint32_t)__half_as_ushort(l[3]) << 16);
    reinterpret_cast<uint2 *>(hi16)[row * 32 + lane] = wh;
    reinterpret_cast<uint2 *>(lo16)[row * 32 + lane] = wl;
    if (norm2) {
        float s = __fadd_rn(__fadd_rn(__fmul_rn(v.x, v.x), __fmul_rn(v.y, v.y)), __fadd_rn(__fmul_rn(v.z, v.z), __fmul_rn(v.w, v.w)));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s = __fadd_rn(s, __shfl_xor_sync(0xffffffffu, s, o));
        if (lane == 0) norm2[row] = s;
    }
}

// ---------------------------------------------------------------- epilogue helpers
// Fold one (score, column) into the row's running top-2 (larger is better), branch-free: 2 FSETP + 3 FMNMX + 3 SEL.
// Ties go to the lower column index without an index comparison, because every thread meets its columns in
// ascending order (tiles ascending, columns ascending inside a tile): a later column only ever replaces an entry
// it strictly beats.  An unset slot is (-inf, -1): a -inf (masked) or NaN score never enters.
__device__ __forceinline__ void row_insert(float s, int col, float &s1, float &s2, int32_t &i1, int32_t &i2) {
    const bool gt1 = s > s1;
    const bool gt2 = s > s2;
    i2 = gt1 ? i1 : (gt2 ? col : i2);
    i1 = gt1 ? col : i1;
    s2 = gt2 ? fminf(s1, s) : s2;  // (not fmaxf(s2, fminf(s1, s)): a NaN score must leave the slots untouched)
    s1 = gt1 ? s : s1;
}

// Filter threshold of a row.  The four threads that share a row (one per column quarter) publish their running
// second-best after every tile; `tau` = the best of the other three is a lower bound of the row's final second-best,
// so a column scoring below it can never reach the row's top-2, whichever thread owns it (two columns scoring >= tau
// exist).  A column scoring exactly tau must still enter (it may win a tie on the column index), hence the largest
// float below tau.  Sharing makes a thread filter as if it had seen four times as many columns: the warp-wide slow
// path (expected ~ 256/k per 4 columns after k columns) is hit ~ 60 % less often.  Stale reads are harmless (the
// published values only grow) and no barrier is involved.
__device__ __forceinline__ float row_threshold(float s2_own, float tau) {
    uint32_t tb = __float_as_uint(tau);
    tb = (tau > 0.f) ? tb - 1u : ((tau < 0.f) ? tb + 1u : 0x80000001u);
    const float below = (tau == -INFINITY) ? tau : __uint_as_float(tb);
    return fmaxf(s2_own, below);
}

// ---------------------------------------------------------------- epilogue: 8 accumulator columns
// v[] = 8 accumulator columns of this thread's row.  Updates the row top-2 and leaves, per column, the warp's
// maximum and the ballot of the lanes that attain it (both warp-uniform; lane 0 stores them as two vectors).
// ROW_MASK is set only for the last, partial row block: elsewhere every lane holds a valid row.
// Kept small on purpose (a rolled loop calls it 8 times per tile and warp): 16 warps share the instruction cache.
// COLFILT (all-warp epilogue of the split fp16 pass): the column side runs only for 4-column groups in which some row of
// the warp reaches `colthr`, a lower bound of what the warp's columns already hold in colkey (their best over the row
// blocks seen so far, weakest column; >= keeps exact ties, which a lower row index may still win).  Slots of skipped
// columns keep the zero ballot the caller wrote.  Needs row blocks of a pair that run at different times (pair_group).
template <int METRIC, bool MASK_COLS, bool ROW_MASK, bool COLS, bool EXT, bool SCALED = false, bool COLFILT = false, bool TOP1 = false>
__device__ __forceinline__ void epi_group8(const float (&v)[8], int cbase, int M, bool row_ok, float na,
                                           const float *__restrict__ cn, bool cn_vec, int lane, float *cv_out,
                                           uint32_t *cb_out, float &s1, float &s2, int32_t &i1, int32_t &i2, float &thr,
                                           float colthr = 0.f, bool *col_any = nullptr) {
    float sc[8], wm[8], nb[8];
    uint32_t bal[8];
    if (METRIC == VO_METRIC_L2 && !EXT) {
        if (!MASK_COLS && cn_vec) {  // warp-uniform: two 128-bit broadcast loads instead of eight scalar ones
            const float4 n0 = __ldg(reinterpret_cast<const float4 *>(cn + cbase));
            const float4 n1 = __ldg(reinterpret_cast<const float4 *>(cn + cbase) + 1);
            nb[0] = n0.x; nb[1] = n0.y; nb[2] = n0.z; nb[3] = n0.w;
            nb[4] = n1.x; nb[5] = n1.y; nb[6] = n1.z; nb[7] = n1.w;
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) nb[j] = (!MASK_COLS || cbase + j < M) ? __ldg(cn + cbase + j) : 0.0f;
        }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int col = cbase + j;
        float s = v[j];
        if (METRIC == VO_METRIC_L2) {
            // with a column arg-min the row norm orders rows inside a column; without one it is a per-row
            // constant that the caller subtracts once, after the scan (same two roundings either way)
            // EXT: the accumulator already holds 2 a.b - |b|^2 (A scaled by 2, norm folded in as one more K-step)
            if (!EXT) s = __fmaf_rn(SCALED ? 2.0f / 65536.0f : 2.0f, s, -nb[j]);  // SCALED: accumulator = 2^16 a.b
            if (COLS) s = __fsub_rn(s, na);
        } else if (SCALED) {
            s = __fmul_rn(s, 1.0f / 65536.0f);  // exact
        }
        if (MASK_COLS) s = (col < M) ? s : -INFINITY;
        sc[j] = s;
        if (COLS && !COLFILT) {
            const float sr = ROW_MASK ? (row_ok ? s : -INFINITY) : s;
            wm[j] = warp_max_f32(sr);
            bal[j] = __ballot_sync(0xffffffffu, sr == wm[j]);
        }
    }
    if (COLS && COLFILT) {
#pragma unroll
        for (int j0 = 0; j0 < 8; j0 += 4) {
            const float m4 = fmaxf(fmaxf(sc[j0], sc[j0 + 1]), fmaxf(sc[j0 + 2], sc[j0 + 3]));
            const bool reach = (!ROW_MASK || row_ok) && m4 >= colthr;
            if (__any_sync(0xffffffffu, reach)) {  // warp-uniform: the collectives below need every lane
#pragma unroll
                for (int j = j0; j < j0 + 4; ++j) {
                    const float sr = ROW_MASK ? (row_ok ? sc[j] : -INFINITY) : sc[j];
                    wm[j] = warp_max_f32(sr);
                    bal[j] = __ballot_sync(0xffffffffu, sr == wm[j]);
                }
                if (lane == 0) {
                    *reinterpret_cast<float4 *>(cv_out + j0) = make_float4(wm[j0], wm[j0 + 1], wm[j0 + 2], wm[j0 + 3]);
                    *reinterpret_cast<uint4 *>(cb_out + j0) = make_uint4(bal[j0], bal[j0 + 1], bal[j0 + 2], bal[j0 + 3]);
                }
                *col_any = true;
            }
        }
    }
    if (COLS && !COLFILT && lane == 0) {
        *reinterpret_cast<float4 *>(cv_out) = make_float4(wm[0], wm[1], wm[2], wm[3]);
        *reinterpret_cast<float4 *>(cv_out + 4) = make_float4(wm[4], wm[5], wm[6], wm[7]);
        *reinterpret_cast<uint4 *>(cb_out) = make_uint4(bal[0], bal[1], bal[2], bal[3]);
        *reinterpret_cast<uint4 *>(cb_out + 4) = make_uint4(bal[4], bal[5], bal[6], bal[7]);
    }
    // Row top-2: a 4-wide max filter, then a branch-free insert of the 4 candidates.  The branch is taken by the
    // whole warp if any lane needs it, so the filter is kept narrow (expected entries ~ 256/k per 4 columns and warp
    // once a row has seen k columns).  Measured alternative: descending to the halves / single columns that really
    // enter (one insert instead of four per hit) costs a third FMNMX per group and nested divergent branches — the
    // single-pass kernels lost 5-8 % (20k x 20k fp16 pass 910 -> 862 TF), so the four straight inserts stay.
#pragma unroll
    for (int j0 = 0; j0 < 8; j0 += 4) {
        const float m4 = fmaxf(fmaxf(sc[j0], sc[j0 + 1]), fmaxf(sc[j0 + 2], sc[j0 + 3]));
        if ((!ROW_MASK || row_ok) && m4 > thr) {  // thr >= s2 (TOP1: >= s1): see row_threshold()
            if (TOP1) {  // ascending columns: strict > keeps the lower column on ties
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const bool gt = sc[j0 + j] > s1;
                    i1 = gt ? cbase + j0 + j : i1;
                    s1 = gt ? sc[j0 + j] : s1;
                }
                thr = fmaxf(thr, s1);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) row_insert(sc[j0 + j], cbase + j0 + j, s1, s2, i1, i2);
                thr = fmaxf(thr, s2);
            }
        }
    }
}

// ---------------------------------------------------------------- A of the fp16 / fp8 single passes -> tensor memory
// One thread's 128 bytes of A (src; zero where !have or past row_elems) -> 32 TMEM columns, arrival on bar_a; the warps of the
// third column quarter (ones_warp) write the ones block of the norm extension.  wait_bar != 0: the loads are issued, then the
// mbarrier is waited for (the accumulator of the previous item's last tile: every MMA that reads the old A has retired), then
// the store happens.  Deliberately NOT inlined: it runs once per work item, and inlined into the tile loop its 32 registers
// pushed the loop's invariants out of the register file (rematerialised per tile: the pass lost 15 %).
template <bool EXT, bool F8>
__device__ __noinline__ void tc_a_to_tmem(const uint8_t *src, bool have, int k0, int row_elems, bool a_warp, bool ones_warp,
                                          uint32_t taddr_a, uint32_t taddr_ext, uint32_t bar_a, uint32_t wait_bar,
                                          uint32_t wait_parity, int lane) {
    constexpr int EPV = F8 ? 16 : 8;   // elements per 16-byte load
    float v[32];
    if (a_warp) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            uint4 x = (have && k0 + k * EPV < row_elems) ? __ldg(reinterpret_cast<const uint4 *>(src) + k) : make_uint4(0, 0, 0, 0);
            uint32_t wd[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if (EXT) {  // A scaled by 2 (exact): the accumulator holds 2 a.b - |b|^2
                    const __half2 d = __hmul2(*reinterpret_cast<const __half2 *>(&wd[i]), __floats2half2_rn(2.0f, 2.0f));
                    wd[i] = *reinterpret_cast<const uint32_t *>(&d);
                }
                v[4 * k + i] = __uint_as_float(wd[i]);
            }
        }
    }
    if (wait_bar) {
        tc::mbar_wait(wait_bar, wait_parity);
        tc::tc_fence_after();
    }
    if (a_warp) {
        tc::tc_st32(taddr_a, v);
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        tc::tc_fence_before();
        if (lane == 0) tc::mbar_arrive(bar_a);
    }
    if (EXT && ones_warp) {  // constant, but rewritten with every A: its warps arrive on bar_a too
        const float ones[8] = {1.f, 1.f, 1.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        tc::tc_st8(taddr_ext, ones);
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        tc::tc_fence_before();
        if (lane == 0) tc::mbar_arrive(bar_a);
    }
}

// ---------------------------------------------------------------- main kernel
// COLS = false drops the column arg-max (REDUX + ballot per column and warp, the per-tile merge and its barrier):
// the ratio / threshold / plain-NN acceptance rules never read it.
template <int PASSES, int METRIC, bool COLS, bool PERSIST_T = false>
__global__ void __cluster_dims__(TC_CLUSTER, 1, 1) __launch_bounds__(TC_THREADS, 1)
match_f32_tc_kernel(const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo,
                    const float *__restrict__ a_hi, const float *__restrict__ a_lo, int n_stride, int m_stride,
                    const int32_t *__restrict__ n_ref, const int32_t *__restrict__ n_cur,
                    const float *__restrict__ row_norm, const float *__restrict__ col_norm, int n_split,
                    vo_row_partial *__restrict__ part, unsigned long long *__restrict__ colkey,
                    int pair_group, int row_elems, int lgrid_x, int n_pairs) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t *smem = smem_raw + (base - smem_u32(smem_raw));

    // Launch order -> work.  Hardware hands out CTAs in x, y, z order, so with the plain mapping the row blocks of one pair
    // run together and march through the column tiles in lockstep.  The column filter of the split fp16 epilogue wants the
    // opposite (row blocks of a pair at different times, so that later ones see the earlier ones' column bests): inside a
    // set of `pair_group` consecutive pairs the clusters are dealt round-robin over the pairs.  The set is sized by the
    // host to keep its current-frame descriptors in L2.  A bijection; both CTAs of a cluster stay on one pair.
    int b = blockIdx.z, rblock = blockIdx.x;
    if (pair_group > 1) {
        const int clusters_x = gridDim.x / TC_CLUSTER;
        const int set0 = (blockIdx.z / pair_group) * pair_group;
        const int gs = min(pair_group, (int)gridDim.z - set0);
        const int l = (blockIdx.z - set0) * clusters_x + (int)(blockIdx.x / TC_CLUSTER);
        b = set0 + l % gs;
        rblock = (l / gs) * TC_CLUSTER + (int)(blockIdx.x % TC_CLUSTER);
    }
    const int split = blockIdx.y;
    const int N = n_ref ? min(n_ref[b], n_stride) : n_stride;
    const int M = n_cur ? min(n_cur[b], m_stride) : m_stride;
    const int row0 = rblock * TC_BM;
    using Cfg = TcCfg<PASSES>;
    constexpr int BN = Cfg::BN, STAGES = Cfg::STAGES, BLOCK_BYTES = Cfg::BLOCK_BYTES, HALF = BN / 2;
    constexpr int TMEM_A = Cfg::TMEM_A, TMEM_EXT = Cfg::TMEM_EXT;
    constexpr uint32_t IDESC = Cfg::IDESC;
    const int tiles_total = (M + BN - 1) / BN;
    const int tiles_per_split = (tiles_total + n_split - 1) / n_split;
    const int t_begin = min(tiles_total, split * tiles_per_split);
    const int t_end = min(tiles_total, t_begin + tiles_per_split);
    const int n_tiles = t_end - t_begin;  // identical in both CTAs of the cluster (same pair, same split)
    // The fp16 / fp8 single passes are PERSISTENT: the grid is one cluster per SM pair and every cluster walks the work items
    // (row-block pair, column split, frame pair) w = cluster, cluster + #clusters, ... in the order the hardware would have
    // handed out the CTAs of the logical grid (lgrid_x, n_split, n_pairs).  Barriers, the TMA ring and the two accumulators
    // run on across items; only A is replaced (by the epilogue warps, once the last MMA of the previous item has retired).
    // Per-CTA set-up / drain and the gap to the next CTA cost 14 k cycles against 27 tiles x 1.3 k at 5k x 5k (11 tiles at 2k x 2k).
    // The other passes run one item per CTA, taken from blockIdx (the variables above).
    constexpr bool PERSIST = PERSIST_T;
    static_assert(!PERSIST || Cfg::F16, "only the fp16 / fp8 single passes have the item loop in their epilogue");
    struct Item { int b, row0, split, N, M, t_begin, n_tiles; };
    const int w_step = PERSIST ? (int)gridDim.x / TC_CLUSTER : 1;
    const int w_first = PERSIST ? (int)blockIdx.x / TC_CLUSTER : 0;
    const int w_end = PERSIST ? (lgrid_x / TC_CLUSTER) * n_split * n_pairs : 1;
    auto item_at = [&](int w) {
        Item I;
        if (!PERSIST) { I.b = b; I.row0 = row0; I.split = split; I.N = N; I.M = M; I.t_begin = t_begin; I.n_tiles = n_tiles; return I; }
        const int cx = lgrid_x / TC_CLUSTER;
        I.b = w / (cx * n_split);
        I.split = (w / cx) % n_split;
        I.row0 = ((w % cx) * TC_CLUSTER + (int)(blockIdx.x % TC_CLUSTER)) * TC_BM;
        I.N = n_ref ? min(n_ref[I.b], n_stride) : n_stride;
        I.M = n_cur ? min(n_cur[I.b], m_stride) : m_stride;
        const int tt = (I.M + BN - 1) / BN, tps = (tt + n_split - 1) / n_split;
        I.t_begin = min(tt, I.split * tps);
        I.n_tiles = min(tt, I.t_begin + tps) - I.t_begin;
        return I;
    };
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t crank = cluster_rank();

    // single-pass L2: one extra box per tile carries -|b|^2 (three tf32 pieces), multiplied by a column block of ones in A
    constexpr bool F16 = Cfg::F16;
    constexpr bool H16 = Cfg::H16, THREE = Cfg::THREE, SCALED = PASSES == 48;
    constexpr bool EXT = !THREE && (METRIC == VO_METRIC_L2);
    constexpr int NKB = H16 ? Cfg::KDIM / Cfg::KBOX : TC_NKB;                           // k boxes per tile (128 B of k each)
    constexpr int ITEMS = THREE ? 2 * NKB : (EXT ? NKB + 1 : NKB);               // B boxes streamed per tile
    const uint32_t s_b = base;
    float *scol_v = reinterpret_cast<float *>(smem + Cfg::OFF_SCOL);                      // [2 groups][2 bufs][4][BN]
    uint32_t *scol_b = reinterpret_cast<uint32_t *>(smem + Cfg::OFF_SCOL + Cfg::SCOL_N * 4);
    const uint32_t s_bar = base + Cfg::OFF_BAR;
    // barrier slots (8 B each): full[S] empty[S] a_full tmem_full[2] tmem_empty[2]; then the TMEM base word
    auto bar_full = [&](int s) { return s_bar + 8u * s; };
    auto bar_empty = [&](int s) { return s_bar + 8u * (STAGES + s); };
    const uint32_t bar_a = s_bar + 8u * (2 * STAGES);
    auto bar_tfull = [&](int g) { return s_bar + 8u * (2 * STAGES + 1 + g); };
    auto bar_tempty = [&](int g) { return s_bar + 8u * (2 * STAGES + 3 + g); };
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + Cfg::OFF_BAR + 8 * (2 * STAGES + 5));
    volatile float *srow2 = reinterpret_cast<volatile float *>(smem + Cfg::OFF_ROW2);  // fp16 passes: row_threshold()
    if (Cfg::H16 && threadIdx.x < 4 * TC_BM) srow2[threadIdx.x] = -INFINITY;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(bar_full(s), 1);            // this CTA's producer arms it; TMA bytes complete it
            mbar_init(bar_empty(s), TC_CLUSTER);  // one commit from each CTA of the cluster
        }
        mbar_init(bar_a, THREE ? 16 : (EXT ? 12 : 8));   // warps that store a part of A (or the ones block)
        for (int g = 0; g < 2; ++g) { mbar_init(bar_tfull(g), 1); mbar_init(bar_tempty(g), H16 ? 16 : 8); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == TC_WARP_MMA) {  // TMEM allocation is warp-collective; this warp also frees it
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"((uint32_t)TC_TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();  // the peer's barriers exist before anything multicasts into this CTA
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    auto tile_of = [&](int lt) { return t_begin + lt; };

    if (warp == TC_WARP_TMA) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            int it = 0;
            for (int w = w_first; w < w_end; w += w_step) {
            const Item I = item_at(w);
            for (int lt = 0; lt < I.n_tiles; ++lt) {
                const int brow = I.b * m_stride + (I.t_begin + lt) * BN;
                for (int item = 0; item < ITEMS; ++item, ++it) {
                    const int stage = it % STAGES;
                    const uint32_t phase = (uint32_t)(it / STAGES) & 1u;
                    mbar_wait(bar_empty(stage), phase ^ 1u);  // both CTAs consumed the slot
                    const bool is_ext = EXT && item == NKB;  // map_b_lo is the extension map in that mode
                    mbar_expect_tx(bar_full(stage), is_ext ? BN * TC_EXT_K * 4 : BLOCK_BYTES);  // bytes arrive by multicast, whoever issues
                    if ((uint32_t)(it & 1) == crank) {
                        const int kb = is_ext ? 0 : (THREE ? (item >> 1) : item);
                        const bool is_lo = is_ext || (THREE && (item & 1));
                        tma_load_2d_mc(s_b + stage * BLOCK_BYTES, is_lo ? &map_b_lo : &map_b_hi, kb * (H16 ? Cfg::KBOX : TC_KB), brow,
                                       bar_full(stage), (uint16_t)((1u << TC_CLUSTER) - 1u));
                    }
                }
            }
            }
        }
    } else if (warp == TC_WARP_MMA) {
        // ===================== MMA issuer =====================
        // The warp stays converged (all lanes wait on the barriers); one elected lane issues.  Descriptors are a
        // constant upper word plus (smem address >> 4): one integer add per MMA, nothing else on the issue path.
        {
            uint32_t stage = 0, phase = 0, a_phase = 0;
            int gt = 0;  // tiles issued so far, over all items: accumulator buffer and its phase
            for (int w = w_first; w < w_end; w += w_step) {
            const Item I = item_at(w);
            if (I.n_tiles == 0) continue;
            mbar_wait(bar_a, a_phase);  // this item's A is in tensor memory
            a_phase ^= 1u;
            tc_fence_after();
            for (int lt = 0; lt < I.n_tiles; ++lt, ++gt) {
                const int buf = gt & 1;
                const uint32_t use = (uint32_t)(gt >> 1);
                mbar_wait(bar_tempty(buf), (use & 1u) ^ 1u);  // epilogue has drained this accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(buf * BN);
#pragma unroll
                for (int item = 0; item < ITEMS; ++item) {
                    mbar_wait(bar_full(stage), phase);
                    tc_fence_after();
                    if (elect_one()) {
                        const int kb = THREE ? (item >> 1) : item;       // compile-time after unrolling
                        const bool is_lo = THREE && (item & 1);
                        const uint32_t b_lo32 = (((s_b + stage * BLOCK_BYTES) & 0x3ffffu) >> 4) | (1u << 16);
                        const uint32_t a_hi_t = tmem_base + (uint32_t)(TMEM_A + kb * TC_KB);
                        if (EXT && item == NKB) {  // ones[128 x 8] * (-|b|^2 pieces)[8 x BN], always kind::tf32
                            const uint64_t bdesc = ((uint64_t)TC_SDESC_HI_32B << 32) | (uint64_t)b_lo32;
                            tc_mma_tf32_ts(d_tmem, tmem_base + (uint32_t)TMEM_EXT, bdesc, IDESC, 1u);
                        } else
#pragma unroll
                        for (int k8 = 0; k8 < TC_KB / 8; ++k8) {
                            const uint64_t bdesc = ((uint64_t)TC_SDESC_HI << 32) | (uint64_t)(b_lo32 + k8 * 2);
                            const uint32_t ahi = a_hi_t + k8 * 8;
                            if (Cfg::F8) {  // 32 k per instruction: again 32 B of B and 8 TMEM columns of A per step
                                tc_mma_f8_ts(d_tmem, ahi, bdesc, Cfg::IDESC16, (item | k8) ? 1u : 0u);  // e4m3 = format 0 as well
                            } else if (F16) {  // 16 k per instruction: the same 32 B of B and 8 TMEM columns of A per step
                                tc_mma_f16_ts(d_tmem, ahi, bdesc, Cfg::IDESC16, (item | k8) ? 1u : 0u);
                            } else if (H16) {  // split fp16: a_hi * b_lo on the lo boxes; a_lo * b_hi, a_hi * b_hi on the hi boxes
                                if (is_lo) {
                                    tc_mma_f16_ts(d_tmem, ahi, bdesc, Cfg::IDESC16, 1u);
                                } else {
                                    tc_mma_f16_ts(d_tmem, ahi + Cfg::ALO, bdesc, Cfg::IDESC16, (item | k8) ? 1u : 0u);
                                    tc_mma_f16_ts(d_tmem, ahi, bdesc, Cfg::IDESC16, 1u);
                                }
                            } else if (is_lo) {  // a_hi * b_lo
                                tc_mma_tf32_ts(d_tmem, ahi, bdesc, IDESC, 1u);
                            } else {
                                if (THREE)  // a_lo * b_hi first (small term), then a_hi * b_hi
                                    tc_mma_tf32_ts(d_tmem, ahi + TC_D, bdesc, IDESC, (item | k8) ? 1u : 0u);
                                tc_mma_tf32_ts(d_tmem, ahi, bdesc, IDESC, (THREE || (item | k8)) ? 1u : 0u);
                            }
                        }
                        // slot reusable (in BOTH CTAs' rings) once these MMAs retire
                        tc_commit_mc(bar_empty(stage), (uint16_t)((1u << TC_CLUSTER) - 1u));
                        if (item == ITEMS - 1) tc_commit(bar_tfull(buf));  // accumulator complete
                    }
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1u; }
                }
            }
            }
        }
    } else {
        if constexpr (Cfg::F16) {
        // ===================== fp16 pass epilogue: all 16 warps on every tile =====================
        // warp -> TMEM lane quarter q (hardware rule), column quarter cq of the tile (48 columns).  A thread pulls its
        // 48 accumulator columns into registers with three tcgen05.ld, hands the accumulator back to the MMA thread
        // at once, and only then folds them into its row's top-2: the accumulator is blocked for one TMEM read, not
        // for the fold (with two 8-warp groups the fold time of a tile sat on the critical path of its buffer).
        constexpr int QW = BN / 4;
        static_assert(QW == 48, "three 16-column reads per thread");
        const int cq = warp >> 2;
        const int q = warp & 3;
        const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
        const int rr = q * 32 + lane;  // row inside the CTA: index into the shared second-bests
        const bool a_warp = cq < Cfg::KDIM / Cfg::KBOX;   // this warp carries 128 B of k (one 32-column chunk) of A into tensor memory
        // A of an item: this thread's 128 bytes.  row_elems < 128: compact rows (byte descriptors: 32 values), the rest is zero.
        auto a_src = [&](int ib, int irow0) {
            const int row = irow0 + rr;
            return reinterpret_cast<const uint8_t *>(a_hi) +
                   (((size_t)ib * n_stride + min(row, n_stride - 1)) * row_elems + cq * Cfg::KBOX) * (Cfg::F8 ? 1 : 2);
        };
        auto a_put = [&](int ib, int irow0, uint32_t wait_bar, uint32_t wait_parity) {
            tc_a_to_tmem<EXT, Cfg::F8>(a_src(ib, irow0), irow0 + rr < n_stride, cq * Cfg::KBOX, row_elems, a_warp, cq == 2,
                                       lane_base + (uint32_t)(TMEM_A + cq * 32), lane_base + (uint32_t)TMEM_EXT, bar_a, wait_bar,
                                       wait_parity, lane);
        };
        // Register budget: 576 threads leave 96 registers each, and 48 of them hold the tile slice during the fold — so nothing
        // about the items stays live across the tile loop except (w, column count, first tile, tile count); whatever else is needed
        // once per item (pair, split, row block; the next item for the hand-over) is decoded again from w where it is used.
        int gt = 0;             // tiles consumed so far, over all items
        bool a_stored = false;  // the current item's A went in during the previous item's last tile
        for (int w = w_first; w < w_end; w += w_step) {
            int M, n_t, tile0;
            bool row_ok, partial_rows;
            float na = 0.0f;
            {
                const Item I = item_at(w);
                M = I.M; n_t = I.n_tiles; tile0 = I.t_begin;
                row_ok = I.row0 + rr < I.N;
                partial_rows = I.row0 + TC_BM > I.N;
                if (METRIC == VO_METRIC_L2 && row_ok) na = row_norm[(size_t)I.b * n_stride + I.row0 + rr];
                // every MMA of the earlier items has retired (their accumulators were all waited for below): A may be replaced
                if (n_t > 0 && !a_stored) a_put(I.b, I.row0, 0u, 0u);
            }
            a_stored = false;
            const bool has_next = PERSIST && w + w_step < w_end;
            if (has_next && a_warp) {   // the next item's A towards L2 (128 B per thread): it is wanted at this item's last tile
                const Item Nx = item_at(w + w_step);
                if (Nx.n_tiles > 0 && Nx.row0 + rr < n_stride) asm volatile("prefetch.global.L2 [%0];" ::"l"(a_src(Nx.b, Nx.row0)));
            }
            float s1 = -INFINITY, s2 = -INFINITY, thr = -INFINITY;
            int32_t i1 = -1, i2 = -1;
            // One tile: wait for its accumulator (unless the hand-over below already did), read it, fold it.
            auto tile = [&](int lt, bool waited) {
                const int buf = gt & 1;
                const uint32_t use = (uint32_t)(gt >> 1);
                const int col0 = (tile0 + lt) * BN + cq * QW;
                const bool full_tile = (tile0 + lt) * BN + BN <= M;
                if (!waited) {
                    mbar_wait(bar_tfull(buf), use & 1u);
                    tc_fence_after();
                }
                const uint32_t taddr = lane_base + (uint32_t)(buf * BN + cq * QW);
                // 48 columns per thread through 32 registers (four groups of 8): columns 0..31 are read; as the first two groups
                // are folded, columns 32..47 are read into their registers (the reads fly during the next group's fold), and
                // after the third group the accumulator is handed back — half a fold later than with 48 registers for the
                // slice, which did not leave room for the item loop (96 per thread: 5 warps share a 16 K register file; a few
                // spilled registers cost 10-40 % here, local memory has next to no L1 beside 220 KB of shared memory).
                // With two accumulators the MMA thread has (2 x fold - MMA) cycles of slack per tile, more than this delay.
                uint32_t g0[8], g1[8], g2[8], g3[8];
                tc_ld8_issue(taddr, g0);
                tc_ld8_issue(taddr + 8, g1);
                tc_ld8_issue(taddr + 16, g2);
                tc_ld8_issue(taddr + 24, g3);
                {  // the other three column quarters' second-bests of this row (read while the TMEM loads fly)
                    const float tau = fmaxf(fmaxf(srow2[((cq + 1) & 3) * TC_BM + rr], srow2[((cq + 2) & 3) * TC_BM + rr]),
                                            srow2[((cq + 3) & 3) * TC_BM + rr]);
                    thr = fmaxf(thr, row_threshold(Cfg::TOP1 ? s1 : s2, tau));   // TOP1: the slots hold running bests
                }
                tc_ld_wait8(g0);
                tc_ld_wait8(g1);
                tc_ld_wait8(g2);
                tc_ld_wait8(g3);
#define TC_FOLD8(BUF, J0, MASKC, MASKR)                                                                                    \
    {                                                                                                                      \
        float v[8];                                                                                                        \
        _Pragma("unroll") for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(BUF[i]);                                      \
        epi_group8<METRIC, MASKC, MASKR, false, EXT, false, false, Cfg::TOP1>(v, col0 + (J0), M, row_ok, na, nullptr, false,  \
                                                                              lane, nullptr, nullptr, s1, s2, i1, i2, thr); \
    }
#define TC_FOLD48(MASKC, MASKR)                                                                                            \
    TC_FOLD8(g0, 0, MASKC, MASKR)                                                                                          \
    tc_ld8_issue(taddr + 32, g0);                                                                                          \
    TC_FOLD8(g1, 8, MASKC, MASKR)                                                                                          \
    tc_ld8_issue(taddr + 40, g1);                                                                                          \
    TC_FOLD8(g2, 16, MASKC, MASKR)                                                                                         \
    tc_ld_wait8(g0);                                                                                                       \
    tc_ld_wait8(g1);                                                                                                       \
    tc_fence_before(); /* the whole tile slice has been read: hand the accumulator back */                                 \
    if (lane == 0) mbar_arrive(bar_tempty(buf));                                                                           \
    TC_FOLD8(g3, 24, MASKC, MASKR)                                                                                         \
    TC_FOLD8(g0, 32, MASKC, MASKR)                                                                                         \
    TC_FOLD8(g1, 40, MASKC, MASKR)
                if (full_tile && !partial_rows) { TC_FOLD48(false, false) } else { TC_FOLD48(true, true) }
#undef TC_FOLD48
#undef TC_FOLD8
                srow2[cq * TC_BM + rr] = Cfg::TOP1 ? s1 : s2;
                ++gt;
            };
            // all tiles but the last in a plain loop (the loop of the one-item-per-CTA kernel, and compiled like it); the last
            // tile of an item, with the hand-over of A to the next item, stands apart
            for (int lt = 0; lt < n_t - 1; ++lt) tile(lt, false);
            if (n_t > 0) {
                bool waited = false;
                if (has_next) {
                    // Once the last accumulator of the item is complete every MMA that reads this item's A has retired, so the
                    // next item's A goes in first (its loads fly during the wait for that accumulator; the tile slice is not in
                    // registers yet) and the tensor pipe restarts while this tile is still being folded.
                    const Item Nx = item_at(w + w_step);
                    if (Nx.n_tiles > 0) {   // warp-uniform (as is everything about an item)
                        a_put(Nx.b, Nx.row0, bar_tfull(gt & 1), (uint32_t)(gt >> 1) & 1u);
                        a_stored = waited = true;
                    }
                }
                tile(n_t - 1, waited);
            }
            if (METRIC == VO_METRIC_L2) {  // the deferred row norm (-inf stays -inf)
                s1 = __fsub_rn(s1, na); s2 = __fsub_rn(s2, na);
            }
            {
                const Item I = item_at(w);
                if (I.row0 + rr < n_stride) {  // four column quarters: four partials per (row, split), merged by finalize
                    const size_t at = ((size_t)I.b * (n_split * 4) + I.split * 4 + cq) * n_stride + I.row0 + rr;
                    if (Cfg::TOP1) {  // 8-byte partials (SCORE_COMPACT_PARTIALS)
                        vo_row_best q;
                        q.s1 = float_to_ordered(-s1); q.i1 = i1;
                        reinterpret_cast<vo_row_best *>(part)[at] = q;
                    } else {
                        vo_row_partial p;
                        p.s1 = float_to_ordered(-s1); p.s2 = float_to_ordered(-s2);
                        p.i1 = i1; p.i2 = i2;
                        part[at] = p;
                    }
                }
            }
            if (has_next) {
                // the shared second-bests belong to the item: clear the own slot (a quarter still inside this item then reads
                // -inf, which only loosens its filter), and nobody starts the next item before every slot is clear
                srow2[cq * TC_BM + rr] = -INFINITY;
                asm volatile("bar.sync 1, 512;" ::: "memory");
            }
        }
        } else if constexpr (Cfg::ALLWARP_COLS) {
        // ===================== split-fp16 epilogue: all 16 warps on every tile, with the column side =====================
        // Same idea as the fp16 single pass: lane quarter q x column quarter cq (32 columns per thread), the tile slice
        // goes to registers, the accumulator is released, then the fold.  Column arg-max: per warp and column
        // redux.max + ballot into shared memory (lane 0), a 128-thread named barrier per column quarter, and the q == 0
        // warp of the quarter merges its 32 columns (one per lane) over the four lane quarters -> one atomicMin each.
        constexpr int QW = BN / 4;
        static_assert(QW == 32, "two 16-column reads per thread, one merged column per lane");
        const int cq = warp >> 2;
        const int q = warp & 3;
        const int row = row0 + q * 32 + lane;
        const bool row_ok = row < N;
        const bool partial_rows = row0 + TC_BM > N;
        const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
        if (n_tiles > 0) {  // A -> tensor memory: column quarters 0,1 store the hi part (k 0..63, 64..127), 2,3 the lo part
            const __half *src = reinterpret_cast<const __half *>(cq < 2 ? a_hi : a_lo) +
                                ((size_t)b * n_stride + min(row, n_stride - 1)) * TC_D + (cq & 1) * 64;
            const bool have = row < n_stride;
            float v[32];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const uint4 x = have ? __ldg(reinterpret_cast<const uint4 *>(src) + k) : make_uint4(0, 0, 0, 0);
                v[4 * k] = __uint_as_float(x.x); v[4 * k + 1] = __uint_as_float(x.y);
                v[4 * k + 2] = __uint_as_float(x.z); v[4 * k + 3] = __uint_as_float(x.w);
            }
            tc_st32(lane_base + (uint32_t)(TMEM_A + cq * 32), v);
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            tc_fence_before();
            if (lane == 0) mbar_arrive(bar_a);
        }
        float s1 = -INFINITY, s2 = -INFINITY, thr = -INFINITY;
        int32_t i1 = -1, i2 = -1;
        const int rr = q * 32 + lane;  // row inside the CTA: index into the shared second-bests
        const float *cn = (METRIC == VO_METRIC_L2) ? col_norm + (size_t)b * m_stride : nullptr;
        const float na = (METRIC == VO_METRIC_L2 && row_ok) ? row_norm[(size_t)b * n_stride + row] : 0.0f;
        const bool cn_vec = (METRIC == VO_METRIC_L2) && ((reinterpret_cast<uintptr_t>(cn) & 15u) == 0);
        for (int lt = 0; lt < n_tiles; ++lt) {
            const int buf = lt & 1;
            const uint32_t use = (uint32_t)(lt >> 1);
            const int tcol0 = tile_of(lt) * BN;
            const int col0 = tcol0 + cq * QW;
            const bool full_tile = tcol0 + BN <= M;
            float *tile_cv = scol_v + buf * 4 * BN;      // [4 lane quarters][BN], alternating per tile
            uint32_t *tile_cb = scol_b + buf * 4 * BN;
            float *my_cv = tile_cv + q * BN + cq * QW;
            uint32_t *my_cb = tile_cb + q * BN + cq * QW;
            mbar_wait(bar_tfull(buf), use & 1u);
            tc_fence_after();
            const uint32_t taddr = lane_base + (uint32_t)(buf * BN + cq * QW);
            uint32_t ra[16], rb[16];
            tc_ld16_issue(taddr, ra);
            tc_ld16_issue(taddr + 16, rb);
            {  // the other three column quarters' second-bests of this row (read while the TMEM loads fly)
                const float tau = fmaxf(fmaxf(srow2[((cq + 1) & 3) * TC_BM + rr], srow2[((cq + 2) & 3) * TC_BM + rr]),
                                        srow2[((cq + 3) & 3) * TC_BM + rr]);
                thr = fmaxf(thr, row_threshold(s2, tau));
            }
            float colthr = -INFINITY;  // weakest current best among this warp's 32 columns (colkey: -score ordered << 32 | row)
            bool col_any = false;
            if (COLS) {
                const int c = col0 + lane;
                float cur_best = INFINITY;  // columns past M never lower the bound
                if (c < M) {
                    const unsigned long long key = *reinterpret_cast<const volatile unsigned long long *>(colkey + (size_t)b * m_stride + c);
                    cur_best = (key == ~0ull) ? -INFINITY : -ordered_to_float((uint32_t)(key >> 32));
                }
                colthr = -warp_max_f32(-cur_best);
                my_cb[lane] = 0u;  // empty ballot = "this warp has no candidate for the column"
                __syncwarp();
            }
            tc_ld_wait16(ra);
            tc_ld_wait16(rb);
            tc_fence_before();  // the tile slice is in registers: hand the accumulator back before folding
            if (lane == 0) mbar_arrive(bar_tempty(buf));
#define TC_FOLD16(BUF, J0, MASKC, MASKR)                                                                                   \
    _Pragma("unroll") for (int u = 0; u < 2; ++u) {                                                                        \
        float v[8];                                                                                                        \
        _Pragma("unroll") for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(BUF[8 * u + i]);                              \
        epi_group8<METRIC, MASKC, MASKR, COLS, false, SCALED, true>(v, col0 + (J0) + 8 * u, M, row_ok, na, cn, cn_vec, lane, \
                                                                  my_cv + (J0) + 8 * u, my_cb + (J0) + 8 * u, s1, s2, i1,  \
                                                                  i2, thr, colthr, &col_any);                              \
    }
            if (full_tile && !partial_rows) {
                TC_FOLD16(ra, 0, false, false) TC_FOLD16(rb, 16, false, false)
            } else {
                TC_FOLD16(ra, 0, true, true) TC_FOLD16(rb, 16, true, true)
            }
#undef TC_FOLD16
            srow2[cq * TC_BM + rr] = s2;
            if (COLS) {
                // the four lane quarters of this column quarter meet; the barrier also tells whether any of them left a
                // candidate (usually none: then there is nothing to merge)
                uint32_t merge;
                asm volatile("{\n\t.reg .pred p, r;\n\tsetp.ne.u32 p, %1, 0;\n\tbar.red.or.pred r, %2, 128, p;\n\tselp.u32 %0, 1, 0, r;\n\t}"
                             : "=r"(merge)
                             : "r"((uint32_t)col_any), "r"(1 + cq)
                             : "memory");
                if (q == 0 && merge) {  // one column per lane
                    const int j = cq * QW + lane;
                    const int col = tcol0 + j;
                    float best = -INFINITY;
                    int brow = -1;
#pragma unroll
                    for (int qq = 0; qq < 4; ++qq) {
                        const float val = tile_cv[qq * BN + j];
                        const uint32_t bal = tile_cb[qq * BN + j];
                        if (bal != 0u && val > best) { best = val; brow = qq * 32 + __ffs(bal) - 1; }
                    }
                    if (col < M && brow >= 0 && row0 + brow < N) {
                        const unsigned long long key =
                            ((unsigned long long)float_to_ordered(-best) << 32) | (unsigned long long)(uint32_t)(row0 + brow);
                        unsigned long long *dst = colkey + (size_t)b * m_stride + col;
                        if (key < *reinterpret_cast<volatile unsigned long long *>(dst)) atomicMin(dst, key);
                    }
                }
                // no second barrier: tile lt+1 writes the other scratch buffer, and tile lt+2 cannot be written before
                // the merging warp has arrived at the barrier of tile lt+1, i.e. after it has read this one
            }
        }
        if (METRIC == VO_METRIC_L2 && !COLS) {  // the deferred row norm (-inf stays -inf)
            s1 = __fsub_rn(s1, na); s2 = __fsub_rn(s2, na);
        }
        if (row < n_stride) {  // four column quarters: four partials per (row, split), merged by finalize
            vo_row_partial p;
            p.s1 = float_to_ordered(-s1); p.s2 = float_to_ordered(-s2);
            p.i1 = i1; p.i2 = i2;
            part[((size_t)b * (n_split * 4) + split * 4 + cq) * n_stride + row] = p;
        }
        } else {
        // ===================== epilogue: 2 groups (one per accumulator) x 8 warps =====================
        // warp -> lane quarter q (hardware rule: warp w may touch TMEM lanes 32*(w%4)..), column half h, group g
        const int g = warp >> 3;
        const int h = (warp >> 2) & 1;
        const int q = warp & 3;
        const int row = row0 + q * 32 + lane;
        const bool row_ok = row < N;
        const bool partial_rows = row0 + TC_BM > N;
        const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);

        // ---- A -> tensor memory, once: group 0 stores the tf32 hi part, group 1 the lo part; each warp 2 k-chunks
        if (n_tiles > 0 && (g == 0 || THREE)) {
            const float *src = (g == 0 ? a_hi : a_lo) + ((size_t)b * n_stride + min(row, n_stride - 1)) * TC_D;
            const bool have = row < n_stride;
#pragma unroll 1
            for (int c = 2 * h; c < 2 * h + 2; ++c) {
                float v[32];
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const float4 x = have ? __ldg(reinterpret_cast<const float4 *>(src + c * 32) + k) : make_float4(0, 0, 0, 0);
                    const float sc2 = EXT ? 2.0f : 1.0f;  // exact
                    v[4 * k] = sc2 * x.x; v[4 * k + 1] = sc2 * x.y; v[4 * k + 2] = sc2 * x.z; v[4 * k + 3] = sc2 * x.w;
                }
                tc_st32(lane_base + (uint32_t)(TMEM_A + g * TC_D + c * 32), v);
            }
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            tc_fence_before();
            if (lane == 0) mbar_arrive(bar_a);
        }

        if (EXT && n_tiles > 0 && g == 1 && h == 0) {  // the ones block of A (TMEM columns of the unused lo half)
            const float ones[8] = {1.f, 1.f, 1.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            tc_st8(lane_base + (uint32_t)TMEM_EXT, ones);
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            tc_fence_before();
            if (lane == 0) mbar_arrive(bar_a);
        }

        float s1 = -INFINITY, s2 = -INFINITY;  // running top-2 of -|a-b|^2 or a.b over this warp's columns
        float thr = -INFINITY;                 // filter threshold (= s2 here: no sharing between the two groups)
        int32_t i1 = -1, i2 = -1;
        float *grp_cv = scol_v + g * 2 * 4 * BN;
        uint32_t *grp_cb = scol_b + g * 2 * 4 * BN;
        const float *cn = (METRIC == VO_METRIC_L2) ? col_norm + (size_t)b * m_stride : nullptr;
        const float na = (METRIC == VO_METRIC_L2 && row_ok) ? row_norm[(size_t)b * n_stride + row] : 0.0f;
        const bool cn_vec = (METRIC == VO_METRIC_L2) && ((reinterpret_cast<uintptr_t>(cn) & 15u) == 0);

        for (int lt = g; lt < n_tiles; lt += 2) {
            const int col0 = tile_of(lt) * BN;
            const uint32_t use = (uint32_t)(lt >> 1);
            const bool full_tile = col0 + BN <= M;
            float *tile_cv = grp_cv + (use & 1u) * 4 * BN;   // this tile's column scratch (alternates per use)
            uint32_t *tile_cb = grp_cb + (use & 1u) * 4 * BN;
            float *my_cv = tile_cv + q * BN;
            uint32_t *my_cb = tile_cb + q * BN;
            mbar_wait(bar_tfull(g), use & 1u);
            tc_fence_after();
            const uint32_t taddr = lane_base + (uint32_t)(g * BN);
            // Three epilogue schedules.  3xTF32 is bound by the tensor pipe: plain load -> wait -> fold.  Single pass is
            // bound by the epilogue, whose cost per 8 columns was the TMEM read latency, so the read of the next
            // columns is kept in flight while the current ones are folded (two register buffers swapped by moves: the
            // loops stay rolled with one or two epi_group8 bodies, 16 warps share the instruction cache); without the
            // column arg-max there are registers to spare and the reads are 16 columns wide.
            if (THREE) {
#define TC_EPI_LOOP(MASKC, MASKR)                                                                                          \
    _Pragma("unroll 1") for (int j0 = HALF * h; j0 < HALF * h + HALF; j0 += 8) {                                                 \
        uint32_t cur[8];                                                                                                   \
        tc_ld8_issue(taddr + j0, cur);                                                                                     \
        tc_ld_wait8(cur);                                                                                                  \
        float v[8];                                                                                                        \
        _Pragma("unroll") for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(cur[i]);                                      \
        epi_group8<METRIC, MASKC, MASKR, COLS, EXT, SCALED>(v, col0 + j0, M, row_ok, na, cn, cn_vec, lane, my_cv + j0, my_cb + j0, \
                                                    s1, s2, i1, i2, thr);                                                       \
    }
                if (full_tile && !partial_rows) { TC_EPI_LOOP(false, false) } else { TC_EPI_LOOP(true, true) }
#undef TC_EPI_LOOP
            } else if (COLS) {
                uint32_t cur[8], nxt[8];
                tc_ld8_issue(taddr + HALF * h, cur);
                tc_ld_wait8(cur);
#define TC_EPI_LOOP(MASKC, MASKR)                                                                                          \
    _Pragma("unroll 1") for (int j0 = HALF * h; j0 < HALF * h + HALF; j0 += 8) {                                                 \
        const bool more = j0 + 8 < HALF * h + HALF;                                                                            \
        if (more) tc_ld8_issue(taddr + j0 + 8, nxt);                                                                       \
        float v[8];                                                                                                        \
        _Pragma("unroll") for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(cur[i]);                                      \
        epi_group8<METRIC, MASKC, MASKR, COLS, EXT>(v, col0 + j0, M, row_ok, na, cn, cn_vec, lane, my_cv + j0, my_cb + j0, \
                                                    s1, s2, i1, i2, thr);                                                       \
        if (more) {                                                                                                        \
            tc_ld_wait8(nxt);                                                                                              \
            _Pragma("unroll") for (int i = 0; i < 8; ++i) cur[i] = nxt[i];                                                 \
        }                                                                                                                  \
    }
                if (full_tile && !partial_rows) { TC_EPI_LOOP(false, false) } else { TC_EPI_LOOP(true, true) }
#undef TC_EPI_LOOP
            } else {
                // no column side: 16-column reads, two register buffers used alternately (unrolled by two, so no moves)
                uint32_t bufa[16], bufb[16];
                tc_ld16_issue(taddr + HALF * h, bufa);
                tc_ld_wait16(bufa);
#define TC_FOLD16(BUF, J0, MASKC, MASKR)                                                                                   \
    _Pragma("unroll") for (int u = 0; u < 2; ++u) {                                                                        \
        float v[8];                                                                                                        \
        _Pragma("unroll") for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(BUF[8 * u + i]);                              \
        epi_group8<METRIC, MASKC, MASKR, COLS, EXT>(v, col0 + (J0) + 8 * u, M, row_ok, na, cn, cn_vec, lane,               \
                                                    my_cv + (J0) + 8 * u, my_cb + (J0) + 8 * u, s1, s2, i1, i2, thr);           \
    }
#define TC_EPI_LOOP(MASKC, MASKR)                                                                                          \
    _Pragma("unroll 1") for (int j0 = HALF * h; j0 < HALF * h + HALF; j0 += 32) {                                          \
        const bool has_b = j0 + 16 < HALF * h + HALF;   /* HALF is a multiple of 16, not necessarily of 32 */               \
        if (has_b) tc_ld16_issue(taddr + j0 + 16, bufb);                                                                   \
        TC_FOLD16(bufa, j0, MASKC, MASKR)                                                                                  \
        if (has_b) {                                                                                                       \
            tc_ld_wait16(bufb);                                                                                            \
            const bool more = j0 + 32 < HALF * h + HALF;                                                                   \
            if (more) tc_ld16_issue(taddr + j0 + 32, bufa);                                                                \
            TC_FOLD16(bufb, j0 + 16, MASKC, MASKR)                                                                         \
            if (more) tc_ld_wait16(bufa);                                                                                  \
        }                                                                                                                  \
    }
                if (full_tile && !partial_rows) { TC_EPI_LOOP(false, false) } else { TC_EPI_LOOP(true, true) }
#undef TC_EPI_LOOP
#undef TC_FOLD16
            }
            tc_fence_before();  // this warp's share of the accumulator has been read: hand it back
            if (lane == 0) mbar_arrive(bar_tempty(g));
            if (COLS) group_bar(1 + g);
            if (COLS && (h * 4 + q) * 32 < BN) {  // one column per thread, merge the 4 lane quarters (ascending rows)
                const int j = (h * 4 + q) * 32 + lane;
                const int col = col0 + j;
                float best = -INFINITY;
                int brow = -1;
#pragma unroll
                for (int qq = 0; qq < 4; ++qq) {
                    const float val = tile_cv[qq * BN + j];
                    const uint32_t bal = tile_cb[qq * BN + j];
                    if (bal != 0u && val > best) { best = val; brow = qq * 32 + __ffs(bal) - 1; }
                }
                if (j < BN && col < M && brow >= 0 && row0 + brow < N) {
                    const unsigned long long key =
                        ((unsigned long long)float_to_ordered(-best) << 32) | (unsigned long long)(uint32_t)(row0 + brow);
                    unsigned long long *dst = colkey + (size_t)b * m_stride + col;
                    if (key < *reinterpret_cast<volatile unsigned long long *>(dst)) atomicMin(dst, key);
                }
            }
            // no second barrier: the next tile of this group writes the other scratch buffer, and the one after
            // next cannot start before every warp has passed the barrier above again
        }
        // four warps (2 groups x 2 column halves) saw disjoint columns of each row: four partials, merged by finalize
        if (METRIC == VO_METRIC_L2 && !COLS) {  // the deferred row norm (-inf stays -inf)
            s1 = __fsub_rn(s1, na); s2 = __fsub_rn(s2, na);
        }
        if (row < n_stride) {
            vo_row_partial p;
            p.s1 = float_to_ordered(-s1); p.s2 = float_to_ordered(-s2);
            p.i1 = i1; p.i2 = i2;
            part[((size_t)b * (n_split * 4) + split * 4 + g * 2 + h) * n_stride + row] = p;
        }
        }  // !F16
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();  // nobody leaves while the peer can still multicast into / arrive on this CTA
    if (warp == TC_WARP_MMA) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TC_TMEM_COLS)
                     : "memory");
    }
}

// [rows][row_elems] fp32 (or fp16 when `half`), box = 128 B of k x box_rows rows, SWIZZLE_128B
int make_map(vo_ctx *ctx, CUtensorMap *map, const void *ptr, long long rows, int box_rows, int row_elems = TC_D,
             bool half = false, bool bytes = false, bool narrow = false) {
    PFN_encodeTiled fn = (PFN_encodeTiled)ctx->encode_tiled;
    const size_t esz = bytes ? 1 : (half ? 2 : 4);
    cuuint64_t dims[2] = {(cuuint64_t)row_elems, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)row_elems * esz};
    cuuint32_t box[2] = {(cuuint32_t)((narrow ? 32 : 128) / esz), (cuuint32_t)box_rows};   // narrow: 32-byte rows, SWIZZLE_32B
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, bytes ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : (half ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32), 2, (void *)ptr, dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, narrow ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed (CUresult %d)", (int)r);
        return VO_ERR_CUDA;
    }
    return VO_OK;
}

template <int PASSES, int METRIC, bool COLS, bool PERSIST>
int launch_tc_kern(vo_ctx *ctx, dim3 grid, const CUtensorMap &bh, const CUtensorMap &bl, const float *a_hi, const float *a_lo,
                   int n_stride, int m_stride, const int32_t *n_ref, const int32_t *n_cur, const float *row_norm,
                   const float *col_norm, int n_split, vo_row_partial *part, unsigned long long *colkey, cudaStream_t st,
                   int row_elems) {
    auto kern = match_f32_tc_kernel<PASSES, METRIC, COLS, PERSIST>;
    VO_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<PASSES>::SMEM_BYTES));
    // split fp16 with the column side: interleave as many pairs as keep their current-frame descriptors (hi + lo fp16) in L2
    int pair_group = 1;
    if (TcCfg<PASSES>::ALLWARP_COLS && COLS && !getenv("VO_TC_NO_INTERLEAVE"))
        pair_group = (int)max(1ll, min(8ll, (64ll << 20) / ((long long)m_stride * TC_D * 4)));
    dim3 launch_grid = grid;
    if constexpr (PERSIST) {  // persistent: one cluster per SM pair (as many as can be resident), each walks the logical grid
        // resident clusters: asked once per kernel and context, since devices (and MIG slices) differ in SM count
        constexpr int slot = 2 * (PASSES == 16 ? 0 : PASSES - 7) + (METRIC == VO_METRIC_COSINE ? 1 : 0);
        static_assert(slot >= 0 && slot < VO_TC_PERSIST_KERNELS, "persistent passes 16, 8, 9 x metric");
        int &max_clusters = ctx->tc_max_clusters[slot];
        if (max_clusters == 0) {
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(TC_CLUSTER * 64);
            cfg.blockDim = dim3(TC_THREADS);
            cfg.dynamicSmemBytes = TcCfg<PASSES>::SMEM_BYTES;
            cudaLaunchAttribute at;
            at.id = cudaLaunchAttributeClusterDimension;
            at.val.clusterDim.x = TC_CLUSTER; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
            cfg.attrs = &at;
            cfg.numAttrs = 1;
            int n = 0;
            if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess || n <= 0) {
                (void)cudaGetLastError();
                n = ctx->sm_count / TC_CLUSTER;
            }
            max_clusters = n;
        }
        const long long items = (long long)(grid.x / TC_CLUSTER) * grid.y * grid.z;
        const long long clusters = items < max_clusters ? items : (long long)max_clusters;
        launch_grid = dim3((unsigned)(clusters * TC_CLUSTER), 1, 1);
    }
    kern<<<launch_grid, TC_THREADS, TcCfg<PASSES>::SMEM_BYTES, st>>>(bh, bl, a_hi, a_lo, n_stride, m_stride, n_ref, n_cur, row_norm, col_norm,
                                                  n_split, part, colkey, pair_group, row_elems, (int)grid.x, (int)grid.z);
    VO_LAUNCH_CHECK(ctx);
    return VO_OK;
}

template <int PASSES, int METRIC, bool COLS>
int launch_tc(vo_ctx *ctx, dim3 grid, const CUtensorMap &bh, const CUtensorMap &bl, const float *a_hi, const float *a_lo,
              int n_stride, int m_stride, const int32_t *n_ref, const int32_t *n_cur, const float *row_norm,
              const float *col_norm, int n_split, vo_row_partial *part, unsigned long long *colkey, cudaStream_t st,
              int row_elems = TC_D) {
#define TC_FWD ctx, grid, bh, bl, a_hi, a_lo, n_stride, m_stride, n_ref, n_cur, row_norm, col_norm, n_split, part, colkey, st, row_elems
    if constexpr (TcCfg<PASSES>::F16) {
        const int tiles_per_item = ceil_div(ceil_div(m_stride, TcCfg<PASSES>::BN), n_split);
        const char *e = getenv("VO_TC_PERSIST");   // VO_TC_PERSIST=0 / 1 forces the plain / the persistent form (comparison runs)
        const bool persist = e ? e[0] != '0' : tiles_per_item <= VO_TC_PERSIST_MAX_TILES;
        if (persist) return launch_tc_kern<PASSES, METRIC, COLS, true>(TC_FWD);
    }
    return launch_tc_kern<PASSES, METRIC, COLS, false>(TC_FWD);
#undef TC_FWD
}

}  // namespace

int match_f32_tc(vo_ctx *ctx, const float *ref, const float *cur, int B, int n_stride, int m_stride,
                 const int32_t *n_ref, const int32_t *n_cur, int metric, int passes, int need_cols,
                 vo_row_partial **part_out, int *n_split_out, unsigned long long *colkey, const float **row_norm_out,
                 cudaStream_t st, int src_u8) {
    // src_u8 = 32 / 128: ref / cur are byte descriptors (uint8 [rows][src_u8]) compared as byte values; only the fp16 single pass
    // without column side takes them
    if (src_u8 && (passes != 16 || need_cols || metric != VO_METRIC_L2 || (src_u8 != 32 && src_u8 != 128))) {
        set_error("match_f32_tc: byte descriptors (32 or 128 per row) run the fp16 single pass (L2, no column arg-min) only");
        return VO_ERR_ARG;
    }
    int rc = ensure_encode(ctx);
    if (rc) return rc;
    if (passes == 16 && need_cols) passes = 1;  // the fp16 pass has no column arg-max: same results from the tf32 pass
    const long long rows_a = (long long)B * n_stride, rows_b = (long long)B * m_stride;
    const bool l2 = metric == VO_METRIC_L2;
    // workspace: A_hi | A_lo  and  B_hi | B_lo  and  row norms | column norms
    float *split_a, *split_b, *norms;
    const bool f16 = passes == 16, h16 = passes == 16 || passes == 48, three = passes == 3 || passes == 48;
    const size_t esz = h16 ? sizeof(__half) : sizeof(float);
    const int row_elems = src_u8 ? src_u8 : TC_D;  // stored elements per descriptor row
    const bool ext = !three && l2;  // B extension rows [rows_b][32] live behind B_hi
    // Consecutive pairs of one frame sequence (pair i = frames i, i + 1: what sequence.FrameSequence hands over, and what a VO run
    // is): the current descriptors are the reference descriptors one frame on.  Then every frame is prepared ONCE — B + 1 frames
    // instead of 2 B — and the B side of the matcher is the A side shifted by a frame (prep is 16 % of a 2k-keypoint SIFT step).
    const size_t src_row_bytes = src_u8 ? (size_t)src_u8 : TC_D * sizeof(float);
    const bool chained = n_stride == m_stride && (n_stride & 3) == 0 && B > 0 && !getenv("VO_NO_CHAIN_PREP") &&
                         reinterpret_cast<const char *>(cur) == reinterpret_cast<const char *>(ref) + (size_t)n_stride * src_row_bytes;
    const long long rows_p = chained ? rows_a + n_stride : rows_a;   // rows prepared on the A side
    const size_t per_a = (size_t)rows_p * row_elems * esz, per_b = chained ? 0 : (size_t)rows_b * row_elems * esz;
    if ((rc = ws_get(ctx, WS_SPLIT_A, per_a * (three ? 2 : 1), (void **)&split_a))) return rc;
    const size_t per_ext = (size_t)(chained ? rows_p : rows_b) * TC_EXT_K * sizeof(float);
    if ((rc = ws_get(ctx, WS_SPLIT_B, per_b * (three ? 2 : 1) + (ext ? per_ext : 0) + 16, (void **)&split_b))) return rc;
    const long long rows_a4 = (rows_a + 3) & ~3ll;  // column norms start 16 B aligned (vector loads in the epilogue)
    if ((rc = ws_get(ctx, WS_NORMS, sizeof(float) * (size_t)(chained ? rows_p : rows_a4 + rows_b), (void **)&norms))) return rc;
    const size_t shift = (size_t)n_stride * row_elems * esz;   // one frame of prepared rows, bytes (chained)
    float *a_hi = split_a, *a_lo = three ? reinterpret_cast<float *>(reinterpret_cast<char *>(split_a) + per_a) : nullptr;
    float *b_hi = chained ? reinterpret_cast<float *>(reinterpret_cast<char *>(a_hi) + shift) : split_b;
    float *b_lo = !three ? nullptr : (chained ? reinterpret_cast<float *>(reinterpret_cast<char *>(a_lo) + shift)
                                              : reinterpret_cast<float *>(reinterpret_cast<char *>(split_b) + per_b));
    float *x_ext = ext ? reinterpret_cast<float *>(reinterpret_cast<char *>(split_b) + per_b * (three ? 2 : 1)) : nullptr;
    float *b_ext = (ext && chained) ? x_ext + (size_t)n_stride * TC_EXT_K : x_ext;
    float *row_norm = norms, *col_norm = chained ? norms + n_stride : norms + rows_a4;

    VO_PROF(ctx, st, VO_STAGE_PREP);
    // (side 0: reference rows — all prepared rows when chained, extension included; side 1: current rows, not run when chained)
    for (int side = 0; side < (chained ? 1 : 2); ++side) {
        const float *src = side ? cur : ref;
        const long long rows = side ? rows_b : rows_p;
        float *hi = side ? b_hi : a_hi, *lo = side ? b_lo : a_lo;
        float *nrm = l2 ? (side ? col_norm : row_norm) : nullptr;
        float *xe = (side || chained) ? x_ext : nullptr;
        const unsigned g8 = (unsigned)((rows + 7) / 8);
        if (passes == 48)
            prep16x3_kernel<<<g8, 256, 0, st>>>(src, rows, reinterpret_cast<__half *>(hi), reinterpret_cast<__half *>(lo), nrm);
        else if (f16 && src_u8 == 32)
            prep16_u8_kernel<32><<<(unsigned)((rows + 31) / 32), 256, 0, st>>>(reinterpret_cast<const uint8_t *>(src), rows, reinterpret_cast<__half *>(hi), side ? col_norm : row_norm, xe);
        else if (f16 && src_u8)
            prep16_u8_kernel<128><<<g8, 256, 0, st>>>(reinterpret_cast<const uint8_t *>(src), rows, reinterpret_cast<__half *>(hi), side ? col_norm : row_norm, xe);
        else if (f16)
            prep16_kernel<<<g8, 256, 0, st>>>(src, rows, reinterpret_cast<__half *>(hi), nrm, xe);
        else
            prep_kernel<<<g8, 256, 0, st>>>(src, rows, hi, lo, nrm, xe);
        VO_LAUNCH_CHECK(ctx);
    }

    CUtensorMap mbh, mbl;
    const int bn = three ? TcCfg<3>::BN : (f16 ? TcCfg<16>::BN : TcCfg<1>::BN);
    if ((rc = make_map(ctx, &mbh, b_hi, rows_b, bn, row_elems, h16))) return rc;
    if (ext) rc = make_map(ctx, &mbl, b_ext, rows_b, bn, TC_EXT_K, false, false, true);
    else rc = make_map(ctx, &mbl, three ? b_lo : b_hi, rows_b, bn, TC_D, h16);
    if (rc) return rc;

    const int row_blocks = ceil_div(n_stride, TC_BM);
    const int grid_x = ceil_div(row_blocks, TC_CLUSTER) * TC_CLUSTER;  // clusters pair adjacent row blocks
    const int n_split = pick_split(ctx, B, grid_x, ceil_div(m_stride, bn), 4);
    vo_row_partial *part;
    if ((rc = ws_get(ctx, WS_ROWPART, sizeof(vo_row_partial) * (size_t)B * n_split * 4 * n_stride, (void **)&part))) return rc;
    dim3 grid(grid_x, n_split, B);
    VO_PROF(ctx, st, VO_STAGE_MATCH);
#define TC_ARGS ctx, grid, mbh, mbl, a_hi, a_lo, n_stride, m_stride, n_ref, n_cur, row_norm, col_norm, n_split, part, colkey, st
#define TC_PICK(P, MET) (need_cols ? launch_tc<P, MET, true>(TC_ARGS) : launch_tc<P, MET, false>(TC_ARGS))
    if (passes == 3) rc = l2 ? TC_PICK(3, VO_METRIC_L2) : TC_PICK(3, VO_METRIC_COSINE);
    else if (passes == 48) rc = l2 ? TC_PICK(48, VO_METRIC_L2) : TC_PICK(48, VO_METRIC_COSINE);
    else if (f16) rc = l2 ? launch_tc<16, VO_METRIC_L2, false>(TC_ARGS, row_elems) : launch_tc<16, VO_METRIC_COSINE, false>(TC_ARGS);
    else rc = l2 ? TC_PICK(1, VO_METRIC_L2) : TC_PICK(1, VO_METRIC_COSINE);
#undef TC_PICK
#undef TC_ARGS
    if (rc) return rc;
    *part_out = part;
    *n_split_out = n_split * 4;  // 2 epilogue groups x 2 column halves -> four partials per (row, split)
    *row_norm_out = nullptr;     // scores already carry -|a-b|^2 in full
    return VO_OK;
}

// Tensor-core Hamming matcher (VO_NORM_HAMMING_TC): 256-bit descriptors -> e4m3 rows of -1 / +1 (once per frame set), then the
// single pass over K = 256 (8 kind::f8f6f4 MMAs of N = 192 per tile; row top-2, thread-private; with the e4m3 operands the
// fold, not the tensor pipe, bounds it) — once with the reference descriptors as rows, and, when the acceptance rule needs the
// column arg-min (mutual nearest neighbours, raw column output), once more with the roles swapped.  Scores are exact integers.
int match_bits_tc(vo_ctx *ctx, const uint8_t *ref, const uint8_t *cur, int B, int n_stride, int m_stride, const int32_t *n_ref,
                  const int32_t *n_cur, int need_cols, int need_second, vo_row_partial **part_out, int *n_split_out,
                  unsigned long long *colkey, cudaStream_t st) {
    int rc = ensure_encode(ctx);
    if (rc) return rc;
    constexpr int KD = 256, BN = TcCfg<8>::BN;
    const long long rows_a = (long long)B * n_stride, rows_b = (long long)B * m_stride;
    uint8_t *a8, *b8;
    // consecutive pairs of one frame sequence (cur = ref one frame on): every frame is expanded once (see match_f32_tc)
    const bool chained = n_stride == m_stride && B > 0 && !getenv("VO_NO_CHAIN_PREP") && cur == ref + (size_t)n_stride * 32;
    const long long rows_p = chained ? rows_a + n_stride : rows_a;
    if ((rc = ws_get(ctx, WS_SPLIT_A, (size_t)rows_p * KD, (void **)&a8))) return rc;
    if (chained) b8 = a8 + (size_t)n_stride * KD;
    else if ((rc = ws_get(ctx, WS_SPLIT_B, (size_t)rows_b * KD, (void **)&b8))) return rc;
    VO_PROF(ctx, st, VO_STAGE_PREP);
    prep_bits8_kernel<<<(unsigned)((rows_p + 7) / 8), 256, 0, st>>>(ref, rows_p, a8);
    VO_LAUNCH_CHECK(ctx);
    if (!chained) {
        prep_bits8_kernel<<<(unsigned)((rows_b + 7) / 8), 256, 0, st>>>(cur, rows_b, b8);
        VO_LAUNCH_CHECK(ctx);
    }

    // second == false: the acceptance rule reads the row arg-max only (mutual NN without k-NN output; always so for the swapped
    // pass) — the fold then keeps one (score, index) pair per row and its filter fires half as often
    auto pass = [&](const uint8_t *A, const uint8_t *Bm, int ns, int ms, const int32_t *na, const int32_t *nb, int slot,
                    vo_row_partial **part, int *n_split, bool second) -> int {
        CUtensorMap map;
        int r;
        if ((r = make_map(ctx, &map, Bm, (long long)B * ms, BN, KD, false, true))) return r;
        const int row_blocks = ceil_div(ns, TC_BM);
        const int grid_x = ceil_div(row_blocks, TC_CLUSTER) * TC_CLUSTER;
        const int ns_split = pick_split(ctx, B, grid_x, ceil_div(ms, BN), 4);
        if ((r = ws_get(ctx, slot, sizeof(vo_row_partial) * (size_t)B * ns_split * 4 * ns, (void **)part))) return r;
        dim3 grid(grid_x, ns_split, B);
        *n_split = ns_split * 4;
        if (second)
            return launch_tc<8, VO_METRIC_COSINE, false>(ctx, grid, map, map, reinterpret_cast<const float *>(A), nullptr, ns, ms, na, nb,
                                                         nullptr, nullptr, ns_split, *part, nullptr, st, KD);
        return launch_tc<9, VO_METRIC_COSINE, false>(ctx, grid, map, map, reinterpret_cast<const float *>(A), nullptr, ns, ms, na, nb,
                                                     nullptr, nullptr, ns_split, *part, nullptr, st, KD);
    };
    VO_PROF(ctx, st, VO_STAGE_MATCH);
    if ((rc = pass(a8, b8, n_stride, m_stride, n_ref, n_cur, WS_ROWPART, part_out, n_split_out, need_second != 0))) return rc;
    if (need_cols) {
        vo_row_partial *part2;
        int n_split2;
        if ((rc = pass(b8, a8, m_stride, n_stride, n_cur, n_ref, WS_ROWPART2, &part2, &n_split2, false))) return rc;
        colkey_from_partials_kernel<<<dim3(ceil_div(m_stride, 256), B), 256, 0, st>>>(reinterpret_cast<const vo_row_best *>(part2), n_split2,
                                                                                      m_stride, n_cur, colkey);
        VO_LAUNCH_CHECK(ctx);
    }
    return VO_OK;
}

}  // namespace vo
