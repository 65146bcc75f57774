// PnP-RANSAC on the GPU: hypothesis table -> P3P minimal solves -> one warp per hypothesis
// inlier counting over correspondences staged in shared memory -> packed atomic arg-max ->
// inlier mask of the winner -> Gauss-Newton refit on its inliers -> pose outputs.
//
// Replaces the 3x cv2.solvePnPRansac(iterationsCount=100, reprojectionError=1.5) loop,
// cv2.Rodrigues and the pose inversion of VisualOdometry.computepose_3D_2D
// (VisualOdometry_Stereo.py:120-144).  OpenCV semantics kept: inlier iff fp32 squared
// reprojection error <= thr^2; the returned inlier set is that of the best MINIMAL model; the
// final pose is a non-linear least-squares refit on exactly those inliers (SURVEY 3.4.1).
//
// Compile this file with -fmad=false (see pnp_math.cuh).
#include "common.cuh"
#include "pnp_math.cuh"
#include "tc_ptx.cuh"

namespace vo {
namespace {

struct IntrD {
    double fx, fy, cx, cy;
};

// ---------------------------------------------------------------- hypothesis table
// keys (optional): per-pair generator keys read from device memory (common.cuh: vo_pair_key); NULL = (seed, pair0 + b)
__global__ void hypotheses_kernel(const int32_t *__restrict__ n_pts, int B, int H, uint64_t seed, int64_t pair0,
                                  const vo_pair_key *__restrict__ keys, int32_t *__restrict__ hyp) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (long long)B * H) return;
    const int b = (int)(gid / H), h = (int)(gid % H);
    const int n = n_pts[b];
    int32_t idx[4] = {-1, -1, -1, -1};
    if (n >= 4) draw_hypothesis(keys ? keys[b].seed : seed, keys ? keys[b].pair : pair0 + b, h, n, idx);
    reinterpret_cast<int4 *>(hyp)[gid] = make_int4(idx[0], idx[1], idx[2], idx[3]);
}

// ---------------------------------------------------------------- minimal solves
// One thread per (pair, hypothesis).  Writes the fp32 pose the scorer uses; an inadmissible
// hypothesis gets a NaN pose, which can never count an inlier.
template <int MINB>
__global__ void __launch_bounds__(128, MINB)
p3p_kernel(const float *__restrict__ xyz, const float *__restrict__ uv, const int32_t *__restrict__ n_pts, int B,
           int cap, const int32_t *__restrict__ hyp, int H, IntrD k, float *__restrict__ poses) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (long long)B * H) return;
    const int b = (int)(gid / H);
    const int n = min(n_pts[b], cap);
    const int4 id = reinterpret_cast<const int4 *>(hyp)[gid];
    const int ids[4] = {id.x, id.y, id.z, id.w};
    bool ok = true;
    for (int s = 0; s < 4; ++s) ok = ok && ids[s] >= 0 && ids[s] < n;
    PoseD best;
    if (ok) {
        double P[4][3], q[4][2];
        for (int s = 0; s < 4; ++s) {
            const size_t o = (size_t)b * cap + ids[s];
            P[s][0] = xyz[o * 3 + 0]; P[s][1] = xyz[o * 3 + 1]; P[s][2] = xyz[o * 3 + 2];
            q[s][0] = uv[o * 2 + 0]; q[s][1] = uv[o * 2 + 1];
        }
        ok = p3p_solve4(P, q, k.fx, k.fy, k.cx, k.cy, best);
    }
    float *o = poses + gid * 12;
    if (ok) {
        for (int j = 0; j < 9; ++j) o[j] = (float)best.r[j];
        for (int j = 0; j < 3; ++j) o[9 + j] = (float)best.t[j];
    } else {
        const float qnan = __int_as_float(0x7fc00000);
        for (int j = 0; j < 12; ++j) o[j] = qnan;
    }
}

// ---------------------------------------------------------------- scoring
// One warp owns SC_HPW hypotheses (their scaled poses live in registers, each value duplicated into both halves of a
// 64-bit register pair); its lanes stride over PAIRS of correspondences.  The 15 fp32 operations of the inlier test
// (pnp_math.cuh, is_inlier) run as packed FFMA2 / FMUL2 (`fma.rn.f32x2`, sm_100): two points per instruction, every
// half rounded exactly like the scalar operation, so counts are bit-identical to the scalar rule the refit kernel and
// the oracle use.  FFMA2 needs half the issue slots of two FFMAs, which is what bounded the scalar kernel (0.76
// instructions per clock and scheduler at 55 % FMA-pipe utilisation): measured with tools/probe/ffma2_probe.cu,
// 8 FFMA2 + 2 LOP3 per round keep 118 of 128 FMA lanes per clock and SM busy, 8 FFMA + 2 LOP3 only 94.
//
// Correspondences reach shared memory by TMA: `score_prep_kernel` lays every 1024-point tile out once per pair as one
// contiguous 20 KB block in the packed order the lanes read ({X0 X1 Y0 Y1}, {Z0 Z1 u0-cx u1-cx}, {v0-cy v1-cy}; points
// past the end are NaN = never an inlier), and each scoring CTA pulls tiles through a two-slot `cp.async.bulk` /
// mbarrier ring, so the copy of tile t+1 overlaps the tests of tile t and no thread spends instructions on staging.
constexpr int SC_WARPS = 8;
constexpr int SC_TILE = 1024;                     // correspondences per staged tile; also the granularity of the pruning test
constexpr int SC_TILE_FLOATS = SC_TILE * 5;       // 20 KB
constexpr int SC_TILE_BYTES = SC_TILE_FLOATS * 4;

typedef unsigned long long f32x2;  // two fp32 in one 64-bit register pair
__device__ __forceinline__ f32x2 pk2(float lo, float hi) {
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpk2(f32x2 v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
    f32x2 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
    f32x2 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}

// is_inlier (pnp_math.cuh) for two points at once.  M = the ScoreModel with rows 0 and 1 negated (exact), every entry
// in both halves, so a = z*(u-cx) + (-x) is a single FFMA2.  Adds the number of inliers among the two points (0..2) to `count`.
__device__ __forceinline__ void inliers2(int &count, const f32x2 (&M)[12], f32x2 THR, f32x2 X, f32x2 Y, f32x2 Z, f32x2 U, f32x2 V) {
    const f32x2 nx = fma2(M[0], X, fma2(M[1], Y, fma2(M[2], Z, M[9])));
    const f32x2 ny = fma2(M[3], X, fma2(M[4], Y, fma2(M[5], Z, M[10])));
    const f32x2 z = fma2(M[6], X, fma2(M[7], Y, fma2(M[8], Z, M[11])));
    const f32x2 a = fma2(z, U, nx);
    const f32x2 b = fma2(z, V, ny);
    const f32x2 w = mul2(THR, z);
    const f32x2 l = fma2(a, a, mul2(b, b));
    const f32x2 r = mul2(w, w);
    float l0, l1, r0, r1;
    unpk2(l, l0, l1);
    unpk2(r, r0, r1);
    // ordered compare (NaN -> not an inlier) + predicated increment: two instructions per point
    asm("{\n\t.reg .pred p0, p1;\n\t"
        "setp.le.f32 p0, %1, %2;\n\t"
        "setp.le.f32 p1, %3, %4;\n\t"
        "@p0 add.s32 %0, %0, 1;\n\t"
        "@p1 add.s32 %0, %0, 1;\n\t}"
        : "+r"(count)
        : "f"(l0), "f"(r0), "f"(l1), "f"(r1));
}

// grid (tiles, B): tile t of pair b -> staged + (b * tiles + t) * SC_TILE_FLOATS
__global__ void __launch_bounds__(256)
score_prep_kernel(const float *__restrict__ xyz, const float *__restrict__ uv, const int32_t *__restrict__ n_pts, int cap,
                  IntrF k, float *__restrict__ staged) {
    const int b = blockIdx.y, t = blockIdx.x;
    const int n = min(n_pts[b], cap);
    const int p0 = t * SC_TILE;
    if (p0 >= n) return;  // never read
    const float *pxyz = xyz + (size_t)b * cap * 3;
    const float *puv = uv + (size_t)b * cap * 2;
    float *dst = staged + ((size_t)b * gridDim.x + t) * SC_TILE_FLOATS;
    const float qnan = __int_as_float(0x7fc00000);
    for (int j = threadIdx.x; j < SC_TILE / 2; j += 256) {
        float v[2][5];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int i = p0 + 2 * j + e;
            if (i < n) {
                const float2 q2 = *reinterpret_cast<const float2 *>(puv + (size_t)i * 2);
                v[e][0] = pxyz[(size_t)i * 3]; v[e][1] = pxyz[(size_t)i * 3 + 1]; v[e][2] = pxyz[(size_t)i * 3 + 2];
                v[e][3] = VO_FSUBF(q2.x, k.cx); v[e][4] = VO_FSUBF(q2.y, k.cy);
            } else {
#pragma unroll
                for (int c = 0; c < 5; ++c) v[e][c] = qnan;
            }
        }
        reinterpret_cast<float4 *>(dst)[j] = make_float4(v[0][0], v[1][0], v[0][1], v[1][1]);
        reinterpret_cast<float4 *>(dst + 2 * SC_TILE)[j] = make_float4(v[0][2], v[1][2], v[0][3], v[1][3]);
        reinterpret_cast<float2 *>(dst + 4 * SC_TILE)[j] = make_float2(v[0][4], v[1][4]);
    }
}

__device__ __forceinline__ void bulk_load(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    tc::mbar_expect_tx(bar, bytes);
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}

// Exact pruning: `lower[b]` is a running lower bound of the winning inlier count of pair b (every warp publishes its
// partial counts after each staged tile — a final count can only be larger).  A hypothesis whose count so far plus ALL
// remaining points is still below that bound can neither win nor tie, so the warp stops scoring it; the winner, its
// count and the tie rule (lowest index) are unchanged.  A CTA whose hypotheses are all out stops fetching tiles.  The
// host scores the first 32 hypotheses in a launch of their own so that the bulk starts with a bound that is already
// close to the final one (with ~60 % inliers a fifth of the random minimal samples is all-inlier).  Disabled when the
// caller wants every hypothesis' count.
//
// Order of the hypotheses.  With pruning, a CTA lives as long as its longest-lived hypothesis, and a fifth of random
// minimal samples is good: in index order practically every CTA keeps a few hypotheses to the very end while most of
// its warps idle at the tile barrier (ncu: barrier = top stall, FMA pipe 56 %).  So the pipeline first scores ALL
// hypotheses on tile 0 only (`t_limit` = 1, counts to `hyp_counts`, no key), sorts them by that count
// (`hyp_sort_kernel`), and scores the rest in sorted order (`perm`, counts carried over through `init`, tiles from
// `t_begin` = 1): CTAs are homogeneous — the good ones run dense to the end, the others leave together and free their
// SM slots.  The scouts are the 32 best-looking hypotheses, so the bound is near-final from the start.  The
// processing order changes nothing in the result: keys carry the original hypothesis index.
struct ScoreOrder {
    const int32_t *perm;   // [B][H] slot -> hypothesis, or null (identity)
    const int32_t *init;   // [B][H] counts of the tiles before t_begin, by hypothesis, or null
    int t_begin, t_limit;  // tiles [t_begin, min(T, t_limit)) are scored
    int write_key;         // 0: partial pass, counts only
};

// ORDERED = false compiles the order away (identity, all tiles, keys written): the unpruned / short-run kernel.
template <int SC_HPW, int MIN_CTAS, bool ORDERED>  // hypotheses per warp, resident CTAs per SM the register budget must allow
__global__ void __launch_bounds__(SC_WARPS * 32, MIN_CTAS)
score_kernel(const float *__restrict__ staged, int tiles, const int32_t *__restrict__ n_pts, int cap,
             const float *__restrict__ poses, int H, int h_begin, int h_end, IntrF k, float thr,
             unsigned long long *__restrict__ bestkey, unsigned int *__restrict__ lower, int32_t *__restrict__ hyp_counts,
             ScoreOrder ord_in) {
    const ScoreOrder ord = ORDERED ? ord_in : ScoreOrder{nullptr, nullptr, 0, 0x7fffffff, 1};
    __shared__ __align__(128) float sbuf[2][SC_TILE_FLOATS];
    __shared__ __align__(8) unsigned long long sbar[2];
    const int b = blockIdx.y;
    const int n = min(n_pts[b], cap);
    const int T = min((n + SC_TILE - 1) / SC_TILE, ord.t_limit);
    const int t0 = min(ord.t_begin, T);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int h0 = h_begin + (blockIdx.x * SC_WARPS + warp) * SC_HPW;  // this launch scores SLOTS [h_begin, h_end)
    const bool prune = hyp_counts == nullptr;
    const float *tiles_b = staged + (size_t)b * tiles * SC_TILE_FLOATS;
    const uint32_t bar0 = tc::smem_u32(&sbar[0]), buf0 = tc::smem_u32(&sbuf[0][0]);
    if (threadIdx.x == 0) {
        tc::mbar_init(bar0, 1);
        tc::mbar_init(bar0 + 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int s = 0; s < 2 && t0 + s < T; ++s)
            bulk_load(buf0 + s * SC_TILE_BYTES, tiles_b + (size_t)(t0 + s) * SC_TILE_FLOATS, SC_TILE_BYTES, bar0 + 8 * s);
    }
    // scaled poses, duplicated into both halves; rows 0 and 1 negated (exact), so that a = z*(u-cx) + (-x) is one FFMA2
    f32x2 M[SC_HPW][12];
    int count[SC_HPW];
#pragma unroll
    for (int q = 0; q < SC_HPW; ++q) {
        PoseF p;
        const int slot = min(h0 + q, H - 1);
        const int h = ord.perm ? ord.perm[(size_t)b * H + slot] : slot;
        count[q] = (ord.init && lane == 0) ? ord.init[(size_t)b * H + h] : 0;
        const float *src = poses + ((size_t)b * H + h) * 12;
#pragma unroll
        for (int j = 0; j < 9; ++j) p.r[j] = __ldg(src + j);
#pragma unroll
        for (int j = 0; j < 3; ++j) p.t[j] = __ldg(src + 9 + j);
        const ScoreModel m = score_model(p, k);
#pragma unroll
        for (int j = 0; j < 12; ++j) {
            const bool neg = (j < 6) || j == 9 || j == 10;
            const float v = neg ? -m.m[j] : m.m[j];
            M[q][j] = pk2(v, v);
        }
    }
    const f32x2 THR = pk2(thr, thr);
    unsigned alive = 0;  // warp-uniform mask of hypotheses still scored
#pragma unroll
    for (int q = 0; q < SC_HPW; ++q) alive |= (h0 + q < h_end) ? (1u << q) : 0u;
    constexpr unsigned ALL = (1u << SC_HPW) - 1u;

    for (int t = t0; t < T; ++t) {
        const int s = (t - t0) & 1;
        const int p0 = t * SC_TILE;
        const int cnt = min(SC_TILE, n - p0);
        const int np = (cnt + 1) >> 1;
        // the bound is read before the tile is scored, so its L2 latency hides behind the tests; a stale (smaller)
        // value only prunes later, never wrongly
        unsigned int lb = 0;
        if (prune && t + 1 < T) lb = *reinterpret_cast<volatile unsigned int *>(&lower[b]);
        tc::mbar_wait(bar0 + 8 * s, (uint32_t)((t - t0) >> 1) & 1u);
        const ulonglong2 *sA = reinterpret_cast<const ulonglong2 *>(&sbuf[s][0]);             // {X0 X1}, {Y0 Y1}
        const ulonglong2 *sB = reinterpret_cast<const ulonglong2 *>(&sbuf[s][2 * SC_TILE]);  // {Z0 Z1}, {uc0 uc1}
        const f32x2 *sC = reinterpret_cast<const f32x2 *>(&sbuf[s][4 * SC_TILE]);            // {vc0 vc1}
        if (alive == ALL) {  // common case: no per-hypothesis branches in the loop
#pragma unroll 2
            for (int j = lane; j < np; j += 32) {
                const ulonglong2 A = sA[j], Bv = sB[j];
                const f32x2 V = sC[j];
#pragma unroll
                for (int q = 0; q < SC_HPW; ++q) inliers2(count[q], M[q], THR, A.x, A.y, Bv.x, Bv.y, V);
            }
        } else if (alive) {
            for (int j = lane; j < np; j += 32) {
                const ulonglong2 A = sA[j], Bv = sB[j];
                const f32x2 V = sC[j];
#pragma unroll
                for (int q = 0; q < SC_HPW; ++q)
                    if (alive & (1u << q)) inliers2(count[q], M[q], THR, A.x, A.y, Bv.x, Bv.y, V);
            }
        }
        if (prune && alive && t + 1 < T) {  // between tiles: publish partial counts, drop the hopeless
            const int remaining = n - (p0 + cnt);
            int tot[SC_HPW], wbest = 0;
#pragma unroll
            for (int q = 0; q < SC_HPW; ++q) {
                tot[q] = (alive & (1u << q)) ? __reduce_add_sync(0xffffffffu, count[q]) : 0;
                wbest = max(wbest, tot[q]);
            }
            if (lane == 0 && wbest > (int)lb) atomicMax(&lower[b], (unsigned int)wbest);
            lb = max(lb, (unsigned int)wbest);
#pragma unroll
            for (int q = 0; q < SC_HPW; ++q)
                if ((alive & (1u << q)) && (unsigned int)(tot[q] + remaining) < lb) alive &= ~(1u << q);
        }
        if (t + 1 < T) {
            // every warp is done with slot s; if no hypothesis of the CTA is left, drain the copy in flight and stop
            const int any = __syncthreads_or(alive != 0u);
            if (!any) {
                if (threadIdx.x == 0) tc::mbar_wait(bar0 + 8 * (s ^ 1), (uint32_t)((t + 1 - t0) >> 1) & 1u);
                break;
            }
            if (threadIdx.x == 0 && t + 2 < T)
                bulk_load(buf0 + s * SC_TILE_BYTES, tiles_b + (size_t)(t + 2) * SC_TILE_FLOATS, SC_TILE_BYTES, bar0 + 8 * s);
        }
    }
#pragma unroll
    for (int q = 0; q < SC_HPW; ++q) {
        if (alive & (1u << q)) {
            const int c = __reduce_add_sync(0xffffffffu, count[q]);
            if (lane == 0) {
                const int h = ord.perm ? ord.perm[(size_t)b * H + h0 + q] : h0 + q;
                if (hyp_counts) hyp_counts[(size_t)b * H + h] = c;
                if (ord.write_key) {  // larger count wins; ties -> lowest hypothesis index
                    const unsigned long long key =
                        ((unsigned long long)(uint32_t)c << 32) | (unsigned long long)(0xffffffffu - (uint32_t)h);
                    atomicMax(&bestkey[b], key);
                }
                if (prune || !ord.write_key) atomicMax(&lower[b], (unsigned int)c);  // a partial count is a lower bound too
            }
        }
    }
}

// Orders the hypotheses of every pair by their tile-0 inlier count, descending (counting sort over 0..SC_TILE; the order
// inside a bin is whatever the atomics give — it only affects scheduling).  One CTA per pair.
__global__ void __launch_bounds__(1024)
hyp_sort_kernel(const int32_t *__restrict__ c0, int H, int32_t *__restrict__ perm) {
    __shared__ int hist[SC_TILE + 1];   // hist[c] = hypotheses with count c, then the first slot of bin c
    __shared__ int wsum[32];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int32_t *c = c0 + (size_t)b * H;
    for (int i = tid; i <= SC_TILE; i += 1024) hist[i] = 0;
    __syncthreads();
    for (int h = tid; h < H; h += 1024) atomicAdd(&hist[min(max(c[h], 0), SC_TILE)], 1);
    __syncthreads();
    // exclusive scan in descending count order: thread tid owns bin SC_TILE - tid (bin 0 comes last)
    const int mine = hist[SC_TILE - tid];
    int incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = wsum[lane], wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += v;
        }
        wsum[lane] = wi - w;  // exclusive
    }
    __syncthreads();
    const int excl = wsum[warp] + incl - mine;
    __syncthreads();
    hist[SC_TILE - tid] = excl;
    if (tid == 1023) hist[0] = excl + mine;  // bin 0 starts after bins SC_TILE..1
    __syncthreads();
    for (int h = tid; h < H; h += 1024) perm[(size_t)b * H + atomicAdd(&hist[min(max(c[h], 0), SC_TILE)], 1)] = h;
}

// ---------------------------------------------------------------- winner mask + refit + outputs
constexpr int RF_THREADS = 256;
constexpr int RF_ACC = 28;  // 21 (upper JtJ) + 6 (Jtr) + 1 (cost)

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ void so3_exp(const double w[3], double R[9]) {
    const double th2 = w[0] * w[0] + w[1] * w[1] + w[2] * w[2];
    const double th = sqrt(th2);
    double A, Bc;
    if (th < 1e-6) {
        A = 1.0 - th2 / 6.0;
        Bc = 0.5 - th2 / 24.0;
    } else {
        A = sin(th) / th;
        Bc = (1.0 - cos(th)) / th2;
    }
    const double wx = w[0], wy = w[1], wz = w[2];
    R[0] = 1.0 - Bc * (wy * wy + wz * wz); R[1] = -A * wz + Bc * wx * wy;      R[2] = A * wy + Bc * wx * wz;
    R[3] = A * wz + Bc * wx * wy;          R[4] = 1.0 - Bc * (wx * wx + wz * wz); R[5] = -A * wx + Bc * wy * wz;
    R[6] = -A * wy + Bc * wx * wz;         R[7] = A * wx + Bc * wy * wz;        R[8] = 1.0 - Bc * (wx * wx + wy * wy);
}

__device__ void so3_log(const double R[9], double w[3]) {
    double c = 0.5 * (R[0] + R[4] + R[8] - 1.0);
    c = fmin(1.0, fmax(-1.0, c));
    const double ax = R[7] - R[5], ay = R[2] - R[6], az = R[3] - R[1];
    const double s = 0.5 * sqrt(ax * ax + ay * ay + az * az);
    const double th = atan2(s, c);
    if (s < 1e-9) {
        if (c > 0.0) {  // theta ~ 0
            w[0] = 0.5 * ax; w[1] = 0.5 * ay; w[2] = 0.5 * az;
        } else {  // theta ~ pi: axis from the diagonal (cv::Rodrigues does the same)
            double x = sqrt(fmax((R[0] + 1.0) * 0.5, 0.0));
            double y = sqrt(fmax((R[4] + 1.0) * 0.5, 0.0)) * (R[1] < 0.0 ? -1.0 : 1.0);
            double z = sqrt(fmax((R[8] + 1.0) * 0.5, 0.0)) * (R[2] < 0.0 ? -1.0 : 1.0);
            if (fabs(x) < fabs(y) && fabs(x) < fabs(z) && (R[5] > 0.0) != (y * z > 0.0)) z = -z;
            const double nrm = sqrt(x * x + y * y + z * z);
            const double f = nrm > 0.0 ? th / nrm : 0.0;
            w[0] = f * x; w[1] = f * y; w[2] = f * z;
        }
        return;
    }
    const double f = 0.5 * th / s;
    w[0] = f * ax; w[1] = f * ay; w[2] = f * az;
}

// 6x6 SPD solve by Cholesky, in place on the packed upper triangle (row-major i<=j).
__device__ bool solve6(const double Hu[21], const double g[6], double x[6]) {
    double L[6][6];
    int idx = 0;
    double A[6][6];
    for (int i = 0; i < 6; ++i)
        for (int j = i; j < 6; ++j) { A[i][j] = Hu[idx]; A[j][i] = Hu[idx]; ++idx; }
    for (int i = 0; i < 6; ++i) {
        for (int j = 0; j <= i; ++j) {
            double s = A[i][j];
            for (int q = 0; q < j; ++q) s -= L[i][q] * L[j][q];
            if (i == j) {
                if (!(s > 0.0)) return false;
                L[i][i] = sqrt(s);
            } else {
                L[i][j] = s / L[j][j];
            }
        }
    }
    double y[6];
    for (int i = 0; i < 6; ++i) {
        double s = g[i];
        for (int q = 0; q < i; ++q) s -= L[i][q] * y[q];
        y[i] = s / L[i][i];
    }
    for (int i = 5; i >= 0; --i) {
        double s = y[i];
        for (int q = i + 1; q < 6; ++q) s -= L[q][i] * x[q];
        x[i] = s / L[i][i];
    }
    return true;
}

// Shared state of refit_pose; the kernel declares it __shared__.
struct RefitShared {
    double R[9], t[3];                    // current pose, seeded with the winning minimal model
    double Rp[9], tp[3], cost;            // last accepted pose and its cost
    double acc[RF_THREADS / 32][RF_ACC];  // per-warp partial sums of the normal equations
    int stop, bad;
};

// Gauss-Newton with a guard (the refined pose is chained into every later global pose, so it must never be worse
// than what RANSAC found): every pass evaluates the cost at the current pose first; a pose that is not finite or
// whose cost exceeds that of the last accepted pose is dropped for the last accepted one (at worst the minimal
// model itself) and the iteration stops.  One extra evaluate-only pass checks the last step.
// inlier(i, X, Y, Z, u, v) fetches correspondence i < n and says whether it is an inlier of the winning minimal model; only
// those enter the refit.  On entry s.R / s.t hold that model and s.stop = s.bad = 0, visible to every thread.  On return
// s.R / s.t hold the refined pose; a minimal model that is not finite sets s.bad and leaves the identity there instead (for
// thread 0, which writes the outputs).
template <class Inlier>
__device__ __forceinline__ void refit_pose(RefitShared &s, int n, int iters, IntrD kd, const Inlier &inlier) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int it = 0; it <= iters; ++it) {
        double acc[RF_ACC];
#pragma unroll
        for (int j = 0; j < RF_ACC; ++j) acc[j] = 0.0;
        double R[9], t[3];
        for (int j = 0; j < 9; ++j) R[j] = s.R[j];
        for (int j = 0; j < 3; ++j) t[j] = s.t[j];
        for (int i = threadIdx.x; i < n; i += RF_THREADS) {
            float Xf, Yf, Zf, uf, vf;
            if (!inlier(i, Xf, Yf, Zf, uf, vf)) continue;
            const double X = Xf, Y = Yf, Z = Zf;
            const double xr = R[0] * X + R[1] * Y + R[2] * Z;
            const double yr = R[3] * X + R[4] * Y + R[5] * Z;
            const double zr = R[6] * X + R[7] * Y + R[8] * Z;
            const double xc = xr + t[0], yc = yr + t[1], zc = zr + t[2];
            const double iz = 1.0 / zc;
            const double x = xc * iz, y = yc * iz;
            const double ru = kd.fx * x + kd.cx - (double)uf;
            const double rv = kd.fy * y + kd.cy - (double)vf;
            const double a0 = kd.fx * iz, a2 = -kd.fx * x * iz;
            const double b1 = kd.fy * iz, b2 = -kd.fy * y * iz;
            const double ju[6] = {a2 * yr, a0 * zr - a2 * xr, -a0 * yr, a0, 0.0, a2};
            const double jv[6] = {-b1 * zr + b2 * yr, -b2 * xr, b1 * xr, 0.0, b1, b2};
            int q = 0;
#pragma unroll
            for (int r = 0; r < 6; ++r)
#pragma unroll
                for (int c = r; c < 6; ++c) acc[q++] += ju[r] * ju[c] + jv[r] * jv[c];
#pragma unroll
            for (int r = 0; r < 6; ++r) acc[21 + r] += ju[r] * ru + jv[r] * rv;
            acc[27] += ru * ru + rv * rv;
        }
#pragma unroll
        for (int j = 0; j < RF_ACC; ++j) {
            const double v = warp_sum(acc[j]);
            if (lane == 0) s.acc[warp][j] = v;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            double tot[RF_ACC];
            for (int j = 0; j < RF_ACC; ++j) {
                double v = 0.0;
                for (int w = 0; w < RF_THREADS / 32; ++w) v += s.acc[w][j];
                tot[j] = v;
            }
            const double cost = tot[27];
            bool finite = cost == cost && cost < 1e300;
            for (int j = 0; j < 9; ++j) finite = finite && s.R[j] == s.R[j] && fabs(s.R[j]) < 2.0;
            for (int j = 0; j < 3; ++j) finite = finite && s.t[j] == s.t[j] && fabs(s.t[j]) < 1e300;
            if (it == 0 && !finite) {        // the minimal model itself is unusable: report "no model"
                s.bad = 1;
                s.stop = 1;
            } else if (it > 0 && !(finite && cost <= s.cost * (1.0 + 1e-12))) {   // worse than the last accepted pose: take that one back
                for (int j = 0; j < 9; ++j) s.R[j] = s.Rp[j];
                for (int j = 0; j < 3; ++j) s.t[j] = s.tp[j];
                s.stop = 1;
            } else {
                s.cost = cost;
                for (int j = 0; j < 9; ++j) s.Rp[j] = s.R[j];
                for (int j = 0; j < 3; ++j) s.tp[j] = s.t[j];
                if (it == iters) s.stop = 1;
            }
            double g[6], d[6];
            for (int j = 0; j < 6; ++j) g[j] = -tot[21 + j];
            // tiny relative damping keeps the factorisation defined for planar / weak geometry
            int dq = 0;
            for (int r = 0; r < 6; ++r) {
                tot[dq] += 1e-12 * tot[dq] + 1e-300;
                dq += 6 - r;
            }
            if (s.stop) {
            } else if (solve6(tot, g, d)) {
                double dR[9], Rn[9];
                so3_exp(d, dR);
                for (int i = 0; i < 3; ++i)
                    for (int j = 0; j < 3; ++j)
                        Rn[3 * i + j] = dR[3 * i] * s.R[j] + dR[3 * i + 1] * s.R[3 + j] + dR[3 * i + 2] * s.R[6 + j];
                for (int j = 0; j < 9; ++j) s.R[j] = Rn[j];
                for (int j = 0; j < 3; ++j) s.t[j] += d[3 + j];
                double mx = 0.0;
                for (int j = 0; j < 6; ++j) mx = fmax(mx, fabs(d[j]));
                if (mx < 1e-11) s.stop = 1;
            } else {
                s.stop = 1;
            }
        }
        __syncthreads();
        if (s.stop) break;
    }
    if (threadIdx.x == 0 && s.bad) {
        for (int j = 0; j < 9; ++j) s.R[j] = (j % 4 == 0) ? 1.0 : 0.0;
        for (int j = 0; j < 3; ++j) s.t[j] = 0.0;
    }
}

// The pose outputs of one pair: rt = [R|t], rvec_tvec = (Rodrigues vector, t), T_rel = [R|t]^-1.  A null output is skipped.
// (The identity written through here gets T_rel[3], [7], [11] = -0.0; write_no_pose writes +0.0.)
__device__ __forceinline__ void write_pose(const double *R, const double *t, double *rt, double *rvec_tvec, double *T_rel) {
    if (rt) {
        for (int j = 0; j < 9; ++j) rt[j] = R[j];
        for (int j = 0; j < 3; ++j) rt[9 + j] = t[j];
    }
    if (rvec_tvec) {
        double w[3];
        so3_log(R, w);
        for (int j = 0; j < 3; ++j) rvec_tvec[j] = w[j];
        for (int j = 0; j < 3; ++j) rvec_tvec[3 + j] = t[j];
    }
    if (T_rel) {  // inverse of [R|t]: [R^T | -R^T t]  (pose.pose = pose.inv_pose, :143)
        for (int i = 0; i < 3; ++i) {
            for (int j = 0; j < 3; ++j) T_rel[4 * i + j] = R[3 * j + i];
            T_rel[4 * i + 3] = -(R[i] * t[0] + R[3 + i] * t[1] + R[6 + i] * t[2]);
        }
        T_rel[12] = 0.0; T_rel[13] = 0.0; T_rel[14] = 0.0; T_rel[15] = 1.0;
    }
}

// The pose outputs of a pair without a model: identity rotation, zero translation and Rodrigues vector.
__device__ __forceinline__ void write_no_pose(double *rt, double *rvec_tvec, double *T_rel) {
    for (int j = 0; j < 16; ++j)
        if (T_rel) T_rel[j] = (j % 5 == 0) ? 1.0 : 0.0;
    for (int j = 0; j < 12; ++j)
        if (rt) rt[j] = (j == 0 || j == 4 || j == 8) ? 1.0 : 0.0;
    for (int j = 0; j < 6; ++j)
        if (rvec_tvec) rvec_tvec[j] = 0.0;
}

__global__ void __launch_bounds__(RF_THREADS)
refit_kernel(const float *__restrict__ xyz, const float *__restrict__ uv, const int32_t *__restrict__ n_pts, int cap,
             const float *__restrict__ poses, int H, IntrF kf, IntrD kd, float thr, int min_inliers, int iters,
             const unsigned long long *__restrict__ bestkey, double *__restrict__ rt_out,
             double *__restrict__ rvec_tvec, double *__restrict__ T_rel, int32_t *__restrict__ n_inl_out,
             int32_t *__restrict__ best_h_out, uint8_t *__restrict__ mask_out, int32_t *__restrict__ status,
             int accumulate_status) {
    const int b = blockIdx.x;
    const int n = min(n_pts[b], cap);
    const unsigned long long key = bestkey[b];
    const int count = (int)(uint32_t)(key >> 32);
    const int h = (int)(0xffffffffu - (uint32_t)(key & 0xffffffffull));
    const bool have = (n >= 4) && (key != 0ull) && (count > min_inliers);
    const float *pxyz = xyz + (size_t)b * cap * 3;
    const float *puv = uv + (size_t)b * cap * 2;
    if (rt_out) rt_out += (size_t)b * 12;
    if (rvec_tvec) rvec_tvec += (size_t)b * 6;
    if (T_rel) T_rel += (size_t)b * 16;
    if (mask_out) mask_out += (size_t)b * cap;

    __shared__ RefitShared s;

    if (!have) {
        if (mask_out)
            for (int i = threadIdx.x; i < cap; i += RF_THREADS) mask_out[i] = 0;
        if (threadIdx.x == 0) {
            int stt = (status && accumulate_status) ? status[b] : 0;
            stt |= (n < 4) ? VO_ST_TOO_FEW_POINTS : VO_ST_NO_MODEL;
            if (status) status[b] = stt;
            if (n_inl_out) n_inl_out[b] = (n >= 4 && key != 0ull) ? count : 0;
            if (best_h_out) best_h_out[b] = (n >= 4 && key != 0ull) ? h : -1;
            write_no_pose(rt_out, rvec_tvec, T_rel);
        }
        return;
    }

    PoseF p;
    {
        const float *src = poses + ((size_t)b * H + h) * 12;
        for (int j = 0; j < 9; ++j) p.r[j] = src[j];
        for (int j = 0; j < 3; ++j) p.t[j] = src[9 + j];
    }
    const ScoreModel sm = score_model(p, kf);
    if (threadIdx.x == 0) {
        // f64 start: the winning fp32 pose, rotation re-orthonormalised by two Newton polar steps
        double R[9];
        for (int j = 0; j < 9; ++j) R[j] = (double)p.r[j];
        for (int it = 0; it < 2; ++it) {
            double G[9];  // G = R^T R
            for (int i = 0; i < 3; ++i)
                for (int j = 0; j < 3; ++j) G[3 * i + j] = R[i] * R[j] + R[3 + i] * R[3 + j] + R[6 + i] * R[6 + j];
            double N[9];  // R (3I - G) / 2
            for (int i = 0; i < 3; ++i)
                for (int j = 0; j < 3; ++j) {
                    double v = 0.0;
                    for (int q = 0; q < 3; ++q) v += R[3 * i + q] * ((q == j ? 3.0 : 0.0) - G[3 * q + j]);
                    N[3 * i + j] = 0.5 * v;
                }
            for (int j = 0; j < 9; ++j) R[j] = N[j];
        }
        for (int j = 0; j < 9; ++j) s.R[j] = R[j];
        for (int j = 0; j < 3; ++j) s.t[j] = (double)p.t[j];
        s.stop = 0;
        s.bad = 0;
    }
    // identical arithmetic to score_kernel
    auto inlier = [&](int i, float &X, float &Y, float &Z, float &u, float &v) {
        X = pxyz[i * 3]; Y = pxyz[i * 3 + 1]; Z = pxyz[i * 3 + 2];
        u = puv[i * 2]; v = puv[i * 2 + 1];
        return is_inlier(sm, thr, X, Y, Z, VO_FSUBF(u, kf.cx), VO_FSUBF(v, kf.cy));
    };
    // inlier mask of the winning minimal model (the refit recomputes the flags instead of storing them per point)
    if (mask_out)
        for (int i = threadIdx.x; i < cap; i += RF_THREADS) {
            float X, Y, Z, u, v;
            mask_out[i] = (i < n && inlier(i, X, Y, Z, u, v)) ? 1 : 0;
        }
    __syncthreads();
    refit_pose(s, n, iters, kd, inlier);
    if (threadIdx.x == 0) {
        if (status) status[b] = (accumulate_status ? status[b] : 0) | (s.bad ? VO_ST_NO_MODEL : VO_ST_OK);
        if (n_inl_out) n_inl_out[b] = count;
        if (best_h_out) best_h_out[b] = h;
        write_pose(s.R, s.t, rt_out, rvec_tvec, T_rel);
    }
}

}  // namespace
}  // namespace vo

namespace vo {
int hypotheses_impl(vo_ctx *ctx, const int32_t *n_pts, int B, int H, uint64_t seed, int64_t pair0, const vo_pair_key *keys,
                    int32_t *hyp, void *stream) {
    VO_REQUIRE(ctx && n_pts && hyp, "vo_hypotheses: null argument");
    VO_REQUIRE(B >= 0 && H >= 0, "vo_hypotheses: negative size");
    VO_REQUIRE(((uintptr_t)hyp % 16) == 0, "vo_hypotheses: table must be 16B aligned");
    const long long total = (long long)B * H;
    if (total == 0) return VO_OK;
    VO_PROF(ctx, (cudaStream_t)stream, VO_STAGE_HYP);
    hypotheses_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(n_pts, B, H, seed, pair0, keys, hyp);
    VO_LAUNCH_CHECK(ctx);
    VO_PROF(ctx, (cudaStream_t)stream, -1);
    return VO_OK;
}
}  // namespace vo

extern "C" int vo_hypotheses(vo_ctx *ctx, const int32_t *n_pts, int B, int H, uint64_t seed, int64_t pair0,
                             int32_t *hyp, void *stream) {
    return vo::hypotheses_impl(ctx, n_pts, B, H, seed, pair0, nullptr, hyp, stream);
}

namespace vo {
int pnp_ransac_impl(vo_ctx *ctx, const float *xyz, const float *uv, const int32_t *n_pts, int B, int cap,
                    const double *K_h, const int32_t *hyp, int H, float thr_px, int min_inliers, int refine_iters,
                    double *rt, double *rvec_tvec, double *T_rel, int32_t *n_inl, int32_t *best_h,
                    uint8_t *inlier_mask, int32_t *hyp_counts, int32_t *status, int accumulate_status,
                    void *stream) {
    VO_REQUIRE(ctx && xyz && uv && n_pts && K_h && hyp, "vo_pnp_ransac: null argument");
    VO_REQUIRE(B >= 0 && cap >= 0 && H > 0, "vo_pnp_ransac: bad size");
    VO_REQUIRE(((uintptr_t)hyp % 16) == 0, "vo_pnp_ransac: hypothesis table must be 16B aligned");
    VO_REQUIRE(K_h[0] != 0.0 && K_h[4] != 0.0, "vo_pnp_ransac: zero focal length");
    cudaStream_t st = (cudaStream_t)stream;
    if (B == 0) return VO_OK;
    float *poses;
    unsigned long long *bestkey;
    int rc;
    const int tiles = ceil_div(cap, SC_TILE);
    const size_t pose_floats = ((size_t)12 * B * H + 31) & ~(size_t)31;  // staged tiles start 128 B aligned
    const size_t staged_floats = (size_t)B * tiles * SC_TILE_FLOATS;
    // sorted scoring (pruned runs with more than one tile and enough hypotheses): tile-0 counts + permutation, [B][H] each
    constexpr int SCOUTS = 32;
    // (worth its two extra launches from ~6 tiles on: c2-sized runs, 4 tiles x 1024 hypotheses, measured 0.41 -> 0.42 ms)
    const bool sorted = !hyp_counts && tiles >= 6 && H > 2 * SCOUTS;
    if ((rc = ws_get(ctx, WS_POSES, sizeof(float) * (pose_floats + staged_floats) + (sorted ? sizeof(int32_t) * 2 * (size_t)B * H : 0),
                     (void **)&poses)))
        return rc;
    float *staged = poses + pose_floats;
    int32_t *c0 = reinterpret_cast<int32_t *>(staged + staged_floats), *perm = c0 + (size_t)B * H;
    if ((rc = ws_get(ctx, WS_BESTKEY, (sizeof(unsigned long long) + sizeof(unsigned int)) * (size_t)B, (void **)&bestkey))) return rc;
    unsigned int *lower = reinterpret_cast<unsigned int *>(bestkey + B);  // running lower bound of the best count (pruning)
    VO_CUDA(cudaMemsetAsync(bestkey, 0, (sizeof(unsigned long long) + sizeof(unsigned int)) * (size_t)B, st));

    IntrD kd{K_h[0], K_h[4], K_h[2], K_h[5]};
    IntrF kf{(float)K_h[0], (float)K_h[4], (float)K_h[2], (float)K_h[5]};
    const long long total = (long long)B * H;
    VO_PROF(ctx, st, VO_STAGE_P3P);
    // occupancy over registers: the f64 solve is a long dependent chain, so 8 blocks per SM (64 registers, spills to L1)
    // beat 3 blocks at 136 registers: 0.270 -> 0.204 ms per 524 k hypotheses (3 / 4 / 5 / 6 / 8: 0.270 / 0.232 / 0.219 / 0.214 / 0.204)
    p3p_kernel<8><<<(unsigned)((total + 127) / 128), 128, 0, st>>>(xyz, uv, n_pts, B, cap, hyp, H, kd, poses);
    VO_LAUNCH_CHECK(ctx);
    VO_PROF(ctx, st, VO_STAGE_SCORE);
    if (tiles > 0) {
        score_prep_kernel<<<dim3(tiles, B), 256, 0, st>>>(xyz, uv, n_pts, cap, kf, staged);
        VO_LAUNCH_CHECK(ctx);
    }
    // 4 hypotheses per warp, 3 CTAs per SM.  Measured (B200, 32 pairs x 16 384 hypotheses x 13.7 k points, tools/score_bench.py):
    // 2 / 4 / 8 hypotheses per warp at 2-3 CTAs per SM: 2.73 / 2.52 / 2.70 ms pruned, 4.26 / 4.07 / 4.02 ms unpruned.
    constexpr int HPW = 4, CTAS = 3, PER_CTA = SC_WARPS * HPW;
    const int no_limit = 0x7fffffff;
    auto launch = [&](int hb, int he, int32_t *counts, const ScoreOrder &ord) {
        if (ord.perm || ord.t_limit != no_limit)
            score_kernel<HPW, CTAS, true><<<dim3(ceil_div(he - hb, PER_CTA), B), SC_WARPS * 32, 0, st>>>(
                staged, tiles, n_pts, cap, poses, H, hb, he, kf, thr_px, bestkey, lower, counts, ord);
        else
            score_kernel<HPW, CTAS, false><<<dim3(ceil_div(he - hb, PER_CTA), B), SC_WARPS * 32, 0, st>>>(
                staged, tiles, n_pts, cap, poses, H, hb, he, kf, thr_px, bestkey, lower, counts, ord);
    };
    if (sorted) {
        launch(0, H, c0, ScoreOrder{nullptr, nullptr, 0, 1, 0});  // every hypothesis on tile 0
        VO_LAUNCH_CHECK(ctx);
        hyp_sort_kernel<<<B, 1024, 0, st>>>(c0, H, perm);
        VO_LAUNCH_CHECK(ctx);
        const ScoreOrder rest{perm, c0, 1, no_limit, 1};
        launch(0, SCOUTS, nullptr, rest);                         // scouts: the 32 best-looking hypotheses, scored to the end
        VO_LAUNCH_CHECK(ctx);
        launch(SCOUTS, H, nullptr, rest);
        VO_LAUNCH_CHECK(ctx);
    } else {
        const ScoreOrder all{nullptr, nullptr, 0, no_limit, 1};
        const int h_first = (hyp_counts || H <= 2 * SCOUTS) ? 0 : SCOUTS;  // scouts: the first hypotheses of every pair
        if (h_first) {
            launch(0, h_first, hyp_counts, all);
            VO_LAUNCH_CHECK(ctx);
        }
        launch(h_first, H, hyp_counts, all);
        VO_LAUNCH_CHECK(ctx);
    }
    VO_PROF(ctx, st, VO_STAGE_REFIT);
    refit_kernel<<<B, RF_THREADS, 0, st>>>(xyz, uv, n_pts, cap, poses, H, kf, kd, thr_px, min_inliers, refine_iters,
                                           bestkey, rt, rvec_tvec, T_rel, n_inl, best_h, inlier_mask, status,
                                           accumulate_status);
    VO_LAUNCH_CHECK(ctx);
    VO_PROF(ctx, st, -1);
    return VO_OK;
}
}  // namespace vo

extern "C" int vo_pnp_ransac(vo_ctx *ctx, const float *xyz, const float *uv, const int32_t *n_pts, int B, int cap,
                             const double *K_h, const int32_t *hyp, int H, float thr_px, int min_inliers,
                             int refine_iters, double *rt, double *rvec_tvec, double *T_rel, int32_t *n_inl,
                             int32_t *best_h, uint8_t *inlier_mask, int32_t *hyp_counts, int32_t *status,
                             void *stream) {
    return vo::pnp_ransac_impl(ctx, xyz, uv, n_pts, B, cap, K_h, hyp, H, thr_px, min_inliers, refine_iters, rt,
                               rvec_tvec, T_rel, n_inl, best_h, inlier_mask, hyp_counts, status, 0, stream);
}

// =====================================================================================================================
// Reference-sampler PnP-RANSAC ("Mode R"): computepose_3D_2D lines :120-135 as the reference runs them — three bootstrap
// resamples (the index rows are an INPUT: the drop-in draws them with np.random.randint exactly like :122), each through
// the inside of cv2.solvePnPRansac(iterationsCount = 100, reprojectionError = 1.5): OpenCV's own sample table, EPnP on five
// points, projectPoints-style fp32 scoring, the adaptive iteration count, and the refit on the inliers of the best MINIMAL
// model (duplicates of the resample included); best of three by inlier count, > min_inliers.  Arithmetic: pnp_ref_math.cuh.
// All restarts x iterations minimal models are solved and scored in parallel; the sequential loop with its early stop is
// replayed over the counts afterwards (a model's count does not depend on the iterations before it).
// =====================================================================================================================
#include "pnp_ref_math.cuh"

namespace vo {
namespace {

constexpr int RP_MAX_RESTARTS = 8, RP_MAX_ITERS = 1024;

// refpnp::jacobi_eig12_rr (parallel-order Jacobi on the symmetric 12 x 12 M^T M) by one warp on shared memory: lanes 0..5 take
// the angles of the round's six disjoint pairs, then the 144 (pair, row, matrix) column updates and the 72 (pair, column) row
// updates are dealt over the lanes.  Every element goes through the same operations as in the serial loop (the two phases make
// them independent of the order of the pairs): bit-identical to it.  Eigenvalues / vectors are then sorted like jacobi_eig does.
// (The cyclic-by-row order, one rotation after the other with only its 12-element updates in parallel, took 340-400 k cycles per
// solve — 66 dependent f64 divide / square-root chains per sweep; this order has 11 per sweep.)
__device__ void jacobi12_warp(double (*A)[12], double (*V)[12], double *d, double (*cs)[2], int lane) {
    for (int i = lane; i < 144; i += 32) V[i / 12][i % 12] = (i / 12 == i % 12) ? 1.0 : 0.0;
    __syncwarp();
    for (int sweep = 0; sweep < 60; ++sweep) {
        double off = 0.0, diag = 0.0;
        for (int i = 0; i < 12; ++i) {          // every lane sums in jacobi_eig12_rr's order: a warp-uniform decision
            diag += A[i][i] * A[i][i];
            for (int jj = i + 1; jj < 12; ++jj) off += A[i][jj] * A[i][jj];
        }
        if (off <= 1e-30 * diag || off == 0.0) break;
        for (int round = 0; round < 11; ++round) {
            if (lane < 6) {
                int p, q;
                refpnp::jacobi12_pair(round, lane, p, q);
                refpnp::jacobi12_angle(A[p][p], A[q][q], A[p][q], cs[lane][0], cs[lane][1]);
            }
            __syncwarp();
            for (int t = lane; t < 144; t += 32) {      // columns p, q: (pair k, row i) of A, then of V
                const int k = (t % 72) / 12, i = t % 12;
                int p, q;
                refpnp::jacobi12_pair(round, k, p, q);
                const double c = cs[k][0], sn = cs[k][1];
                double (*Mx)[12] = t < 72 ? A : V;
                const double akp = Mx[i][p], akq = Mx[i][q];
                Mx[i][p] = c * akp - sn * akq;
                Mx[i][q] = sn * akp + c * akq;
            }
            __syncwarp();
            for (int t = lane; t < 72; t += 32) {       // rows p, q of A: (pair k, column j)
                const int k = t / 12, j = t % 12;
                int p, q;
                refpnp::jacobi12_pair(round, k, p, q);
                const double c = cs[k][0], sn = cs[k][1];
                const double apk = A[p][j], aqk = A[q][j];
                A[p][j] = c * apk - sn * aqk;
                A[q][j] = sn * apk + c * aqk;
            }
            __syncwarp();
        }
    }
    __syncwarp();
    if (lane == 0) {
        for (int i = 0; i < 12; ++i) d[i] = A[i][i];
        for (int i = 0; i < 11; ++i) {          // selection sort, descending (jacobi_eig)
            int m = i;
            for (int jj = i + 1; jj < 12; ++jj) m = (d[jj] > d[m]) ? jj : m;
            if (m != i) {
                const double td = d[i]; d[i] = d[m]; d[m] = td;
                for (int k = 0; k < 12; ++k) { const double tv = V[k][i]; V[k][i] = V[k][m]; V[k][m] = tv; }
            }
        }
    }
    __syncwarp();
}

// one WARP per (restart, iteration): lane 0 prepares (control points, barycentrics, M^T M), the 12 x 12 eigen-decomposition runs
// warp-wide in shared memory, and the three beta candidates (initialisation, five Gauss-Newton steps, orientation, error) run
// on lanes 0, 1, 2 at once.  Same operations in the same order per element as the serial refpnp::epnp5: identical results.
// (One thread per solve, the first version, took 1.05 ms per frame pair for the 300 solves — a chain of dependent f64
// operations on local-memory arrays; the warp-wide Jacobi brought it to 0.56 ms.)
//
// Batching: pair b of B owns xyz + b*cap*3, uv + b*cap*2, the bootstrap rows boot + b*restarts*cap (row stride cap) and the
// sample table table + b*table_stride (stride 0: one table shared by the batch, the single-pair entry's host-built one).
// pn[b] is the pair's point count once ref_prepare_kernel has checked it, -1 for a pair with bad input; pairs with fewer
// than EP_N points (or bad input) solve nothing and read no point.  Every kernel indexes (b, restart, iteration) the same way,
// so B = 1 with cap = n is exactly the single-pair computation.
constexpr int RP_PREP_THREADS = 128;
constexpr int32_t RP_BAD = -1;

// one CTA per pair: n_pts[b] (n_fixed when n_pts is NULL) must lie in [0, cap] and every index of the first n entries of each
// bootstrap row in [0, n); the verdict goes to pn[b].  With `table` set, thread 0 then builds the pair's OpenCV sample table
// (refpnp::mwc_table: one thread stepping the multiply-with-carry generator, 87 us at iters = 100) — on the device, so the
// batched entry needs no host staging and its table follows n_pts without a host read.
__global__ void __launch_bounds__(RP_PREP_THREADS)
ref_prepare_kernel(const int32_t *__restrict__ n_pts, int n_fixed, int cap, const int32_t *__restrict__ boot, int restarts,
                   int iters, int32_t *__restrict__ table, int32_t *__restrict__ pn) {
    const int b = blockIdx.x;
    const int n = n_pts ? n_pts[b] : n_fixed;
    int bad = (n < 0 || n > cap) ? 1 : 0;
    if (!bad) {                                 // block-uniform
        const int32_t *rows = boot + (size_t)b * restarts * cap;
        for (int r = 0; r < restarts; ++r)
            for (int i = threadIdx.x; i < n; i += RP_PREP_THREADS) {
                const int32_t v = rows[(size_t)r * cap + i];
                bad |= (v < 0 || v >= n) ? 1 : 0;
            }
    }
    bad = __syncthreads_or(bad);
    if (threadIdx.x == 0) {
        pn[b] = bad ? RP_BAD : n;
        if (table && !bad && n >= refpnp::EP_N) refpnp::mwc_table(n, iters, table + (size_t)b * iters * refpnp::EP_N);
    }
}

// The warps cover B x restarts x iterations; an iteration without a model (pair without a solve, repeated point, no finite
// candidate) writes valid 0 and a zero pose.
constexpr int RP_WARPS = 4;
__global__ void __launch_bounds__(32 * RP_WARPS)
ref_epnp_kernel(const float *__restrict__ xyz, const float *__restrict__ uv, const int32_t *__restrict__ boot,
                const int32_t *__restrict__ pn, int B, int cap, const int32_t *__restrict__ table, int table_stride, int restarts,
                int iters, IntrD kd, double *__restrict__ poses, int32_t *__restrict__ valid) {
    __shared__ double sA[RP_WARPS][12][12], sV[RP_WARPS][12][12], sd[RP_WARPS][12], sX[RP_WARPS][refpnp::EP_N][3], sv[RP_WARPS][4][12];
    __shared__ refpnp::EpnpState sS[RP_WARPS];
    __shared__ int s_mode[RP_WARPS];            // 0: repeated point (no model), 1: regular, 2: coplanar
    __shared__ double s_cs[RP_WARPS][6][2];     // the (cos, sin) of a Jacobi round's six rotations
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int per = restarts * iters;
    const int id = blockIdx.x * RP_WARPS + w;
    if (id >= B * per) return;                  // warp-uniform
    const int b = id / per, r = (id % per) / iters, h = id % iters;
    if (pn[b] < refpnp::EP_N) {                 // warp-uniform: too few points, or bad input
        if (lane == 0) valid[id] = 0;
        if (lane < 12) poses[(size_t)id * 12 + lane] = 0.0;
        return;
    }
    xyz += (size_t)b * cap * 3;
    uv += (size_t)b * cap * 2;
    const int32_t *row = boot + ((size_t)b * restarts + r) * cap;
    const int32_t *tab = table + (size_t)b * table_stride;
    if (lane == 0) {
        double q[refpnp::EP_N][2];
        int src[refpnp::EP_N];
        bool repeated = false;
        for (int j = 0; j < refpnp::EP_N; ++j) {
            const int idx = row[tab[h * refpnp::EP_N + j]];
            for (int k = 0; k < j; ++k) repeated = repeated || (src[k] == idx);
            src[j] = idx;
            for (int k = 0; k < 3; ++k) sX[w][j][k] = (double)xyz[(size_t)idx * 3 + k];
            q[j][0] = (double)uv[(size_t)idx * 2];
            q[j][1] = (double)uv[(size_t)idx * 2 + 1];
        }
        // The five sampled positions are distinct, but a bootstrap resample repeats points: a sample that holds the same
        // correspondence twice has four distinct points, M^T M a four-dimensional null space, and what OpenCV's EPnP returns
        // for it is arbitrary.  Such an iteration is spent without a model (0.7 % of the iterations at n = 1500) —
        // deterministic, and the same in the oracle.
        if (!repeated) refpnp::epnp5_prepare(sX[w], q, kd.fx, kd.fy, kd.cx, kd.cy, sS[w], sA[w]);
        s_mode[w] = repeated ? 0 : (sS[w].planar ? 2 : 1);
    }
    __syncwarp();
    const int mode = s_mode[w];
    if (mode == 1) jacobi12_warp(sA[w], sV[w], sd[w], s_cs[w], lane);
    if (lane == 0 && mode != 0) {
        if (mode == 2) refpnp::epnp5_basis_planar(sA[w], sv[w]);
        else refpnp::epnp5_basis_from_eig(sV[w], sv[w]);
    }
    __syncwarp();
    // the three candidates (find_betas_approx_1 / _2 / _3 + Gauss-Newton + orientation) are independent: lanes 0, 1, 2
    refpnp::Pose p;
    double err = 0.0;
    bool fin = false;
    if (mode != 0 && lane < 3) fin = refpnp::epnp5_candidate(sX[w], sS[w], sv[w], lane, p, err);
    const bool f1 = __shfl_sync(0xffffffffu, (int)fin, 1) != 0, f2 = __shfl_sync(0xffffffffu, (int)fin, 2) != 0;
    const double e1 = __shfl_sync(0xffffffffu, err, 1), e2 = __shfl_sync(0xffffffffu, err, 2);
    int pick = -1;                              // lowest error, the earlier candidate keeps ties (compute_pose)
    if (lane == 0) {
        double best = 0.0;
        if (fin) { pick = 0; best = err; }
        if (f1 && (pick < 0 || e1 < best)) { pick = 1; best = e1; }
        if (f2 && (pick < 0 || e2 < best)) { pick = 2; best = e2; }
        valid[id] = pick >= 0 ? 1 : 0;
    }
    pick = __shfl_sync(0xffffffffu, pick, 0);
    if (lane == pick) {
        for (int k = 0; k < 9; ++k) poses[(size_t)id * 12 + k] = p.R[k];
        for (int k = 0; k < 3; ++k) poses[(size_t)id * 12 + 9 + k] = p.t[k];
    }
    if (pick < 0 && lane < 12) poses[(size_t)id * 12 + lane] = 0.0;
}

// one warp per (pair, restart, iteration): inlier count over the n points of the restart's resample
__global__ void __launch_bounds__(256)
ref_score_kernel(const float *__restrict__ xyz, const float *__restrict__ uv, const int32_t *__restrict__ boot,
                 const int32_t *__restrict__ pn, int B, int cap, int restarts, int iters, IntrD kd, float thr2,
                 const double *__restrict__ poses, const int32_t *__restrict__ valid, int32_t *__restrict__ counts) {
    const int id = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    const int per = restarts * iters;
    if (id >= B * per) return;
    if (!valid[id]) {                           // (every iteration of a pair without a solve)
        if (lane == 0) counts[id] = -1;
        return;
    }
    const int pb = id / per, n = pn[pb];
    xyz += (size_t)pb * cap * 3;
    uv += (size_t)pb * cap * 2;
    refpnp::Pose p;
    for (int k = 0; k < 9; ++k) p.R[k] = poses[(size_t)id * 12 + k];
    for (int k = 0; k < 3; ++k) p.t[k] = poses[(size_t)id * 12 + 9 + k];
    const int32_t *b = boot + ((size_t)pb * restarts + (id % per) / iters) * cap;
    int c = 0;
    for (int i = lane; i < n; i += 32) {
        const int idx = b[i];
        c += refpnp::reproj_err2(p, kd.fx, kd.fy, kd.cx, kd.cy, xyz[(size_t)idx * 3], xyz[(size_t)idx * 3 + 1], xyz[(size_t)idx * 3 + 2],
                                 uv[(size_t)idx * 2], uv[(size_t)idx * 2 + 1]) <= thr2 ? 1 : 0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if (lane == 0) counts[id] = c;
}

// stopping rule per restart, best of the restarts, inlier mask of the winning minimal model, Gauss-Newton refit on those
// inliers (what cv2.solvePnP(ITERATIVE) converges to, SURVEY 3.4.1), Rodrigues vector and the pose the reference stores.
// One CTA per pair.  accumulate_status: OR into the soft bits an earlier stage set (vo_pipeline) instead of overwriting them.
__global__ void __launch_bounds__(RF_THREADS)
ref_select_refit_kernel(const float *__restrict__ xyz, const float *__restrict__ uv, const int32_t *__restrict__ boot,
                        const int32_t *__restrict__ pn, int cap, int restarts, int iters, IntrD kd, float thr2, double confidence,
                        int min_inliers, int refine_iters, const double *__restrict__ poses, const int32_t *__restrict__ counts,
                        double *__restrict__ rt_out, double *__restrict__ rvec_tvec, double *__restrict__ T_rel,
                        int32_t *__restrict__ n_inl_out, int32_t *__restrict__ best_out, uint8_t *__restrict__ mask_out,
                        int32_t *__restrict__ status, int accumulate_status) {
    __shared__ int s_best[RP_MAX_RESTARTS], s_cnt[RP_MAX_RESTARTS], s_run[RP_MAX_RESTARTS];
    __shared__ int s_r, s_h;
    __shared__ RefitShared s;
    const int pb = blockIdx.x, per = restarts * iters;
    const int n_chk = pn[pb];
    const bool bad_input = n_chk == RP_BAD;
    const int n = bad_input ? 0 : n_chk;
    xyz += (size_t)pb * cap * 3;
    uv += (size_t)pb * cap * 2;
    boot += (size_t)pb * restarts * cap;
    poses += (size_t)pb * per * 12;
    counts += (size_t)pb * per;
    if (rt_out) rt_out += (size_t)pb * 12;
    if (rvec_tvec) rvec_tvec += (size_t)pb * 6;
    if (T_rel) T_rel += (size_t)pb * 16;
    if (n_inl_out) n_inl_out += pb;
    if (best_out) best_out += (size_t)pb * 3;
    if (mask_out) mask_out += (size_t)pb * cap;
    if (status) status += pb;
    if (threadIdx.x < restarts) {
        int run = 0, cnt = 0;
        s_best[threadIdx.x] = refpnp::ransac_scan(counts + threadIdx.x * iters, n, iters, confidence, &run, &cnt);
        s_cnt[threadIdx.x] = cnt;
        s_run[threadIdx.x] = run;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int best = 0, rsel = -1;                             // :132-135: flag and inliers > best and inliers > 20, first restart keeps ties
        for (int r = 0; r < restarts; ++r)
            if (s_best[r] >= 0 && s_cnt[r] > best && s_cnt[r] > min_inliers) { best = s_cnt[r]; rsel = r; }
        s_r = rsel;
        s_h = rsel >= 0 ? s_best[rsel] : -1;
        s.stop = 0;
        s.bad = 0;
        if (rsel >= 0) {
            const double *p = poses + ((size_t)rsel * iters + s_h) * 12;
            for (int j = 0; j < 9; ++j) s.R[j] = p[j];
            for (int j = 0; j < 3; ++j) s.t[j] = p[9 + j];
        }
    }
    __syncthreads();
    const int rsel = s_r, hsel = s_h;
    if (rsel < 0) {                                         // (always so for a pair with bad input: all its counts are -1)
        if (mask_out)
            for (int i = threadIdx.x; i < (bad_input ? cap : n); i += RF_THREADS) mask_out[i] = 0;
        if (threadIdx.x == 0) {
            if (status)
                status[0] = (accumulate_status ? status[0] : 0) | VO_ST_NO_MODEL | (bad_input ? VO_ST_BAD_INPUT : 0);
            if (n_inl_out) n_inl_out[0] = 0;
            if (best_out) { best_out[0] = -1; best_out[1] = -1; best_out[2] = 0; }
            write_no_pose(rt_out, rvec_tvec, T_rel);
        }
        return;
    }
    const int32_t *b = boot + (size_t)rsel * cap;
    refpnp::Pose pm;                                        // the winning minimal model: its mask selects the refit's points
    for (int j = 0; j < 9; ++j) pm.R[j] = s.R[j];
    for (int j = 0; j < 3; ++j) pm.t[j] = s.t[j];
    auto inlier = [&](int i, float &X, float &Y, float &Z, float &u, float &v) {
        const int idx = b[i];
        X = xyz[(size_t)idx * 3]; Y = xyz[(size_t)idx * 3 + 1]; Z = xyz[(size_t)idx * 3 + 2];
        u = uv[(size_t)idx * 2]; v = uv[(size_t)idx * 2 + 1];
        return refpnp::reproj_err2(pm, kd.fx, kd.fy, kd.cx, kd.cy, X, Y, Z, u, v) <= thr2;
    };
    if (mask_out)
        for (int i = threadIdx.x; i < n; i += RF_THREADS) {
            float X, Y, Z, u, v;
            mask_out[i] = inlier(i, X, Y, Z, u, v) ? 1 : 0;
        }
    refit_pose(s, n, refine_iters, kd, inlier);
    if (threadIdx.x == 0) {
        if (status) status[0] = (accumulate_status ? status[0] : 0) | (s.bad ? VO_ST_NO_MODEL : VO_ST_OK);
        if (n_inl_out) n_inl_out[0] = s_cnt[rsel];
        if (best_out) { best_out[0] = rsel; best_out[1] = hsel; best_out[2] = s_run[rsel]; }
        write_pose(s.R, s.t, rt_out, rvec_tvec, T_rel);
    }
}

// ---------------------------------------------------------------- bootstrap rows
// boot[b][r][i] = draw_bootstrap(seed, pair0 + b, r, i, n_pts[b]) for i < n_pts[b] (pnp_math.cuh: keyed like the hypotheses,
// a pure function of the pair, not of its batch position), -1 for the padding i >= n_pts[b].  keys (optional) replaces
// (seed, pair0 + b) by (keys[b].seed, keys[b].pair).
__global__ void bootstrap_kernel(const int32_t *__restrict__ n_pts, int B, int restarts, int cap, uint64_t seed, int64_t pair0,
                                 const vo_pair_key *__restrict__ keys, int32_t *__restrict__ boot) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (long long)B * restarts * cap) return;
    const int i = (int)(gid % cap), r = (int)((gid / cap) % restarts), b = (int)(gid / ((long long)cap * restarts));
    const int n = n_pts[b];
    boot[gid] = i < n ? draw_bootstrap(keys ? keys[b].seed : seed, keys ? keys[b].pair : pair0 + b, r, i, n) : -1;
}

}  // namespace

int bootstrap_impl(vo_ctx *ctx, const int32_t *n_pts, int B, int restarts, int cap, uint64_t seed, int64_t pair0,
                   const vo_pair_key *keys, int32_t *boot, void *stream) {
    VO_REQUIRE(ctx && n_pts && boot, "vo_bootstrap: null argument");
    VO_REQUIRE(B >= 0 && restarts >= 0 && cap >= 0, "vo_bootstrap: negative size");
    const long long total = (long long)B * restarts * cap;
    if (total == 0) return VO_OK;
    VO_PROF(ctx, (cudaStream_t)stream, VO_STAGE_HYP);
    bootstrap_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(n_pts, B, restarts, cap, seed, pair0,
                                                                                      keys, boot);
    VO_LAUNCH_CHECK(ctx);
    VO_PROF(ctx, (cudaStream_t)stream, -1);
    return VO_OK;
}

// Both Mode R entries.  n_pts NULL: one pair (B = 1) of n_fixed points whose bootstrap rows have stride cap = n_fixed, with the
// sample table built on the host; otherwise B pairs, n_pts on the device, one table per pair built on the device.
int pnp_ransac_ref_impl(vo_ctx *ctx, const float *xyz, const float *uv, const int32_t *n_pts, int n_fixed, int B, int cap,
                        const double *K_h, const int32_t *boot_idx, int restarts, int iters, float thr_px, double confidence,
                        int min_inliers, int refine_iters, double *rt, double *rvec_tvec, double *T_rel, int32_t *n_inl,
                        int32_t *best, uint8_t *inlier_mask, int32_t *hyp_counts, double *hyp_poses, int32_t *status,
                        int accumulate_status, void *stream) {
    VO_REQUIRE(B >= 0 && cap >= 0 && restarts >= 1 && restarts <= RP_MAX_RESTARTS && iters >= 1 && iters <= RP_MAX_ITERS,
               "vo_pnp_ransac_ref: bad size (B %d, cap %d, restarts %d, iterations %d)", B, cap, restarts, iters);
    VO_REQUIRE(K_h[0] != 0.0 && K_h[4] != 0.0, "vo_pnp_ransac_ref: zero focal length");
    VO_REQUIRE((long long)B * restarts * iters <= 0x7fffffffLL, "vo_pnp_ransac_ref: %d pairs x %d x %d models exceed 2^31", B,
               restarts, iters);
    if (B == 0) return VO_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const bool host_table = n_pts == nullptr;
    const size_t per = (size_t)restarts * iters, total = (size_t)B * per;
    // workspace: sample tables | checked point counts | validity | counts | poses
    char *ws;
    int rc;
    const size_t table_ints = (size_t)(host_table ? 1 : B) * iters * refpnp::EP_N;
    const size_t off_pn = sizeof(int32_t) * table_ints, off_valid = off_pn + sizeof(int32_t) * (size_t)B,
                 off_counts = off_valid + sizeof(int32_t) * total;
    const size_t off_poses = (off_counts + sizeof(int32_t) * total + 15) & ~(size_t)15;
    if ((rc = ws_get(ctx, WS_POSES, off_poses + sizeof(double) * 12 * total, (void **)&ws))) return rc;
    int32_t *table = reinterpret_cast<int32_t *>(ws), *pn = reinterpret_cast<int32_t *>(ws + off_pn);
    int32_t *valid = reinterpret_cast<int32_t *>(ws + off_valid), *counts = reinterpret_cast<int32_t *>(ws + off_counts);
    double *poses = reinterpret_cast<double *>(ws + off_poses);
    const IntrD kd{K_h[0], K_h[4], K_h[2], K_h[5]};
    const float thr2 = (float)((double)thr_px * (double)thr_px);      // findInliers: float t = (float)(thresh * thresh)
    VO_PROF(ctx, st, VO_STAGE_HYP);
    if (host_table && n_fixed >= refpnp::EP_N) {
        // OpenCV's sample table is a function of the point count alone.  One pair: built on the host (the same
        // refpnp::mwc_table; on the device it is one thread, 87 us of the 470 us call) and copied in stream order — a
        // pageable source is staged by the driver before cudaMemcpyAsync returns, so the array may die here.  (Not
        // capture-safe; the batched entry builds its tables on the device.)
        int32_t table_h[RP_MAX_ITERS * refpnp::EP_N];
        refpnp::mwc_table(n_fixed, iters, table_h);
        VO_CUDA(cudaMemcpyAsync(table, table_h, sizeof(int32_t) * (size_t)iters * refpnp::EP_N, cudaMemcpyHostToDevice, st));
    }
    ref_prepare_kernel<<<B, RP_PREP_THREADS, 0, st>>>(n_pts, n_fixed, cap, boot_idx, restarts, iters, host_table ? nullptr : table, pn);
    VO_LAUNCH_CHECK(ctx);
    VO_PROF(ctx, st, VO_STAGE_P3P);
    const int table_stride = host_table ? 0 : iters * refpnp::EP_N;
    ref_epnp_kernel<<<(unsigned)((total + RP_WARPS - 1) / RP_WARPS), 32 * RP_WARPS, 0, st>>>(xyz, uv, boot_idx, pn, B, cap, table,
                                                                                            table_stride, restarts, iters, kd, poses, valid);
    VO_LAUNCH_CHECK(ctx);
    VO_PROF(ctx, st, VO_STAGE_SCORE);
    ref_score_kernel<<<(unsigned)((total + 7) / 8), 256, 0, st>>>(xyz, uv, boot_idx, pn, B, cap, restarts, iters, kd, thr2,
                                                                            poses, valid, counts);
    VO_LAUNCH_CHECK(ctx);
    VO_PROF(ctx, st, VO_STAGE_REFIT);
    ref_select_refit_kernel<<<B, RF_THREADS, 0, st>>>(xyz, uv, boot_idx, pn, cap, restarts, iters, kd, thr2, confidence, min_inliers,
                                                      refine_iters, poses, counts, rt, rvec_tvec, T_rel, n_inl, best, inlier_mask,
                                                      status, accumulate_status);
    VO_LAUNCH_CHECK(ctx);
    VO_PROF(ctx, st, -1);
    if (hyp_counts) VO_CUDA(cudaMemcpyAsync(hyp_counts, counts, sizeof(int32_t) * total, cudaMemcpyDeviceToDevice, st));
    if (hyp_poses) VO_CUDA(cudaMemcpyAsync(hyp_poses, poses, sizeof(double) * 12 * total, cudaMemcpyDeviceToDevice, st));
    return VO_OK;
}

}  // namespace vo

extern "C" int vo_pnp_ransac_ref(vo_ctx *ctx, const float *xyz, const float *uv, int n, const double *K_h, const int32_t *boot_idx,
                                 int restarts, int iters, float thr_px, double confidence, int min_inliers, int refine_iters,
                                 double *rt, double *rvec_tvec, double *T_rel, int32_t *n_inl, int32_t *best, uint8_t *inlier_mask,
                                 int32_t *hyp_counts, double *hyp_poses, int32_t *status, void *stream) {
    VO_REQUIRE(ctx && xyz && uv && K_h && boot_idx, "vo_pnp_ransac_ref: null argument");
    VO_REQUIRE(n >= 0, "vo_pnp_ransac_ref: bad size (n %d)", n);
    return vo::pnp_ransac_ref_impl(ctx, xyz, uv, nullptr, n, 1, n, K_h, boot_idx, restarts, iters, thr_px, confidence, min_inliers,
                                   refine_iters, rt, rvec_tvec, T_rel, n_inl, best, inlier_mask, hyp_counts, hyp_poses, status, 0,
                                   stream);
}

extern "C" int vo_pnp_ransac_ref_batch(vo_ctx *ctx, const float *xyz, const float *uv, const int32_t *n_pts, int B, int cap,
                                       const double *K_h, const int32_t *boot_idx, int restarts, int iters, float thr_px,
                                       double confidence, int min_inliers, int refine_iters, double *rt, double *rvec_tvec,
                                       double *T_rel, int32_t *n_inl, int32_t *best, uint8_t *inlier_mask, int32_t *hyp_counts,
                                       double *hyp_poses, int32_t *status, void *stream) {
    VO_REQUIRE(ctx && xyz && uv && n_pts && K_h && boot_idx && T_rel && status, "vo_pnp_ransac_ref_batch: null argument");
    return vo::pnp_ransac_ref_impl(ctx, xyz, uv, n_pts, 0, B, cap, K_h, boot_idx, restarts, iters, thr_px, confidence, min_inliers,
                                   refine_iters, rt, rvec_tvec, T_rel, n_inl, best, inlier_mask, hyp_counts, hyp_poses, status, 0,
                                   stream);
}

extern "C" int vo_bootstrap(vo_ctx *ctx, const int32_t *n_pts, int B, int restarts, int cap, uint64_t seed, int64_t pair0,
                            int32_t *boot, void *stream) {
    return vo::bootstrap_impl(ctx, n_pts, B, restarts, cap, seed, pair0, nullptr, boot, stream);
}
