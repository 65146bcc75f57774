// Per-hypothesis math of the PnP-RANSAC path, written once for device code (and compilable for
// the host so the build container, which has no GPU, can unit-test it against OpenCV).
//
//  * hypothesis generator: counter-based, integer-only (bit-exact everywhere)
//  * P3P minimal solver (Grunert's distance formulation, quartic by Ferrari with a bracketed
//    Newton resolvent root, rigid alignment of the two triangles, 4th point disambiguation —
//    the same contract as OpenCV's SOLVEPNP_P3P inside solvePnPRansac: 3 points + 1 to choose)
//  * fp32 inlier rule of OpenCV's RANSAC, err^2 <= thr^2 (ptsetreg.cpp semantics, SURVEY 3.4.1),
//    in a division-free form
//
// The f64 solver uses only + - * / sqrt, and this translation unit is compiled with
// -fmad=false, so the CPU oracle (gcc -ffp-contract=off) reproduces every bit of it.  The fp32
// scoring uses explicit fused multiply-adds on both sides (__fmaf_rn / fmaf).
#pragma once
#include <stdint.h>
#include <math.h>

#if defined(__CUDACC__)
#define VO_HD __host__ __device__ __forceinline__
#else
#define VO_HD inline
#endif

#if defined(__CUDA_ARCH__)
#define VO_FMAF(a, b, c) __fmaf_rn((a), (b), (c))
#define VO_FMULF(a, b) __fmul_rn((a), (b))
#define VO_FSUBF(a, b) __fsub_rn((a), (b))
#else
#define VO_FMAF(a, b, c) fmaf((a), (b), (c))
#define VO_FMULF(a, b) ((a) * (b))
#define VO_FSUBF(a, b) ((a) - (b))
#endif

namespace vo {

// ---------------------------------------------------------------- hypothesis generator
VO_HD uint64_t mix64(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// Mode R bootstrap entry i of restart r of pair `pair`, uniform in [0, n); requires n >= 1.  The pair key is the hypothesis
// generator's; the restart is mixed in XOR-ed into a domain constant whose high word is set, so no row key equals a hypothesis
// key of the same (seed, pair) (mix64 is a bijection and a hypothesis mixes in h < 2^32).  Range map: multiply-high of the high
// word u, (u * n) >> 32, which gives every value floor or ceil of 2^32 / n of the 2^32 words: relative bias below n / 2^32.
VO_HD int32_t draw_bootstrap(uint64_t seed, int64_t pair, int r, int i, int n) {
    uint64_t key = mix64(seed + 0x9E3779B97F4A7C15ull * (uint64_t)(pair + 1));
    key = mix64(key ^ 0xB0075742A9B5D0E1ull ^ (uint64_t)(uint32_t)r);
    const uint32_t u = (uint32_t)(mix64(key + (uint64_t)(uint32_t)i * 0xD1B54A32D192ED03ull) >> 32);
    return (int32_t)(((uint64_t)u * (uint64_t)(uint32_t)n) >> 32);
}

// 4 distinct indices in [0, n) for hypothesis h of pair `pair`; requires n >= 4.
VO_HD void draw_hypothesis(uint64_t seed, int64_t pair, int h, int n, int32_t out[4]) {
    uint64_t key = mix64(seed + 0x9E3779B97F4A7C15ull * (uint64_t)(pair + 1));
    key = mix64(key ^ (uint64_t)(uint32_t)h);
    uint64_t ctr = 0;
    for (int s = 0; s < 4; ++s) {
        int32_t v;
        bool dup;
        do {
            const uint64_t r = mix64(key + ctr * 0xD1B54A32D192ED03ull);
            ++ctr;
            v = (int32_t)((uint32_t)(r >> 32) % (uint32_t)n);
            dup = false;
            for (int q = 0; q < s; ++q) dup = dup || (out[q] == v);
        } while (dup);
        out[s] = v;
    }
}

// ---------------------------------------------------------------- fp32 scoring
struct PoseF {
    float r[9];
    float t[3];
};
struct IntrF {
    float fx, fy, cx, cy;
};

// Inlier rule of cv2.solvePnPRansac (ptsetreg.cpp / PnPRansacCallback::computeError, SURVEY 3.4.1):
//   Xc = R X + t ; u^ = fx Xc.x / Xc.z + cx ; inlier iff (u - u^)^2 + (v - v^)^2 <= thr^2.
// Evaluated division-free, multiplied through by Xc.z^2 (exact in real arithmetic, sign-independent):
//   a = z (u - cx) - fx x,  b = z (v - cy) - fy y,  inlier iff a^2 + b^2 <= (thr z)^2
// with fx, fy folded into the first two pose rows once per hypothesis (ScoreModel) and the principal
// point removed once per correspondence (uc = u - cx, vc = v - cy).  17 fp32 instructions per
// (hypothesis, point), every one an explicitly rounded mul / fma, so host and device agree bit for bit.
// A point exactly on the camera plane (Xc.z == 0, which projectPoints maps as if z were 1) and any
// NaN pose are never inliers.
struct ScoreModel {
    float m[12];  // rows 0,1 of [R|t] scaled by fx, fy; row 2 as is: m[0..2],m[9] | m[3..5],m[10] | m[6..8],m[11]
};

VO_HD ScoreModel score_model(const PoseF &p, const IntrF &k) {
    ScoreModel s;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        s.m[j] = VO_FMULF(k.fx, p.r[j]);
        s.m[3 + j] = VO_FMULF(k.fy, p.r[3 + j]);
        s.m[6 + j] = p.r[6 + j];
    }
    s.m[9] = VO_FMULF(k.fx, p.t[0]);
    s.m[10] = VO_FMULF(k.fy, p.t[1]);
    s.m[11] = p.t[2];
    return s;
}

// uc = u - cx, vc = v - cy (each rounded once); thr = reprojection threshold in pixels
VO_HD bool is_inlier(const ScoreModel &s, float thr, float X, float Y, float Z, float uc, float vc) {
    const float x = VO_FMAF(s.m[0], X, VO_FMAF(s.m[1], Y, VO_FMAF(s.m[2], Z, s.m[9])));
    const float y = VO_FMAF(s.m[3], X, VO_FMAF(s.m[4], Y, VO_FMAF(s.m[5], Z, s.m[10])));
    const float z = VO_FMAF(s.m[6], X, VO_FMAF(s.m[7], Y, VO_FMAF(s.m[8], Z, s.m[11])));
    const float a = VO_FMAF(z, uc, -x);
    const float b = VO_FMAF(z, vc, -y);
    const float w = VO_FMULF(thr, z);
    return VO_FMAF(a, a, VO_FMULF(b, b)) <= VO_FMULF(w, w);
}

// ---------------------------------------------------------------- quartic (f64, basic ops only)
// Real roots of x^4 + a x^3 + b x^2 + c x + d.  Returns the count (0..4).
VO_HD int solve_quartic_monic(double a, double b, double c, double d, double roots[4]) {
    const double a2 = a * a;
    const double p = b - 0.375 * a2;
    const double q = c - 0.5 * a * b + 0.125 * a2 * a;
    const double r = d - 0.25 * a * c + 0.0625 * a2 * b - (3.0 / 256.0) * a2 * a2;
    const double shift = -0.25 * a;
    int n = 0;
    const double scale = fabs(p) + fabs(r) + 1.0;
    if (fabs(q) <= 1e-14 * scale) {
        // biquadratic: y^2 = (-p +- sqrt(p^2 - 4 r)) / 2
        double disc = p * p - 4.0 * r;
        if (disc < 0.0) {
            if (disc > -1e-12 * scale * scale) disc = 0.0; else return 0;
        }
        const double sd = sqrt(disc);
        const double z[2] = {0.5 * (-p + sd), 0.5 * (-p - sd)};
        for (int k = 0; k < 2; ++k) {
            if (z[k] >= 0.0) {
                const double y = sqrt(z[k]);
                roots[n++] = y + shift;
                roots[n++] = -y + shift;
            }
        }
        return n;
    }
    // resolvent  f(m) = m^3 + p m^2 + (p^2/4 - r) m - q^2/8,  f(0) < 0: positive root in (0, hi]
    const double c2 = p, c1 = 0.25 * p * p - r, c0 = -0.125 * q * q;
    double lo = 0.0, hi = 1.0 + fmax(fabs(c2), fmax(fabs(c1), fabs(c0)));
    double m = hi;
    for (int it = 0; it < 200; ++it) {
        const double fm = ((m + c2) * m + c1) * m + c0;
        if (fm == 0.0) break;
        if (fm > 0.0) hi = m; else lo = m;
        const double dfm = (3.0 * m + 2.0 * c2) * m + c1;
        double mn = (dfm != 0.0) ? m - fm / dfm : lo;
        if (!(mn > lo && mn < hi)) mn = 0.5 * (lo + hi);
        if (mn == m || !(hi > lo)) break;
        m = mn;
        if (hi - lo <= 4e-16 * hi) break;
    }
    if (!(m > 0.0)) return 0;
    const double s = sqrt(2.0 * m);
    const double qs = q / (2.0 * s);
    const double hb = 0.5 * p + m;
    // y^2 - s y + (hb + qs) = 0   and   y^2 + s y + (hb - qs) = 0
    const double sgn[2] = {1.0, -1.0};
    for (int k = 0; k < 2; ++k) {
        const double cc = hb + sgn[k] * qs;
        double disc = s * s - 4.0 * cc;
        if (disc < 0.0) {
            if (disc > -1e-10 * (s * s + fabs(4.0 * cc) + 1e-300)) disc = 0.0; else continue;
        }
        const double sd = sqrt(disc);
        roots[n++] = 0.5 * (sgn[k] * s + sd) + shift;
        roots[n++] = 0.5 * (sgn[k] * s - sd) + shift;
    }
    return n;
}

// ---------------------------------------------------------------- P3P
struct PoseD {
    double r[9];
    double t[3];
};

VO_HD void cross3(const double a[3], const double b[3], double o[3]) {
    o[0] = a[1] * b[2] - a[2] * b[1];
    o[1] = a[2] * b[0] - a[0] * b[2];
    o[2] = a[0] * b[1] - a[1] * b[0];
}
VO_HD double dot3(const double a[3], const double b[3]) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }

// orthonormal frame of a triangle: e1 along P2-P1, e3 normal, e2 = e3 x e1.  false if degenerate.
VO_HD bool tri_frame(const double P1[3], const double P2[3], const double P3[3], double e[9]) {
    double d12[3] = {P2[0] - P1[0], P2[1] - P1[1], P2[2] - P1[2]};
    double d13[3] = {P3[0] - P1[0], P3[1] - P1[1], P3[2] - P1[2]};
    const double l1 = sqrt(dot3(d12, d12));
    if (!(l1 > 0.0)) return false;
    e[0] = d12[0] / l1; e[1] = d12[1] / l1; e[2] = d12[2] / l1;
    double nrm[3];
    cross3(e, d13, nrm);
    const double l3 = sqrt(dot3(nrm, nrm));
    if (!(l3 > 1e-12 * sqrt(dot3(d13, d13)))) return false;
    e[6] = nrm[0] / l3; e[7] = nrm[1] / l3; e[8] = nrm[2] / l3;
    cross3(e + 6, e, e + 3);
    return true;
}

// Up to 4 poses (X_cam = R X_world + t) from 3 world points / pixel observations.
// K = (fx, fy, cx, cy).  Returns the number of solutions written.
VO_HD int p3p_solve(const double P[3][3], const double uv[3][2], double fx, double fy, double cx, double cy,
                    PoseD sol[4]) {
    double f[3][3];
    for (int i = 0; i < 3; ++i) {
        const double x = (uv[i][0] - cx) / fx, y = (uv[i][1] - cy) / fy;
        const double inv = 1.0 / sqrt(x * x + y * y + 1.0);
        f[i][0] = x * inv; f[i][1] = y * inv; f[i][2] = inv;
    }
    double d23[3], d13[3], d12[3];
    for (int k = 0; k < 3; ++k) {
        d23[k] = P[1][k] - P[2][k];
        d13[k] = P[0][k] - P[2][k];
        d12[k] = P[0][k] - P[1][k];
    }
    const double a2 = dot3(d23, d23), b2 = dot3(d13, d13), c2 = dot3(d12, d12);
    if (!(a2 > 0.0 && b2 > 0.0 && c2 > 0.0)) return 0;
    const double ca = dot3(f[1], f[2]), cb = dot3(f[0], f[2]), cg = dot3(f[0], f[1]);

    // s2 = u s1, s3 = v s1;  u = n(v)/d(v);  quartic in v from  u^2 - 2 u cg + 1 = (c2/b2) q(v)
    const double K1 = (a2 - c2) / b2, rr = c2 / b2;
    const double n2 = K1 - 1.0, n1 = -2.0 * K1 * cb, n0 = 1.0 + K1;
    const double d1 = -2.0 * ca, d0 = 2.0 * cg;
    // w(v) = 1 - rr q(v),  q(v) = v^2 - 2 cb v + 1
    const double w2 = -rr, w1 = 2.0 * rr * cb, w0 = 1.0 - rr;
    const double dd2 = d1 * d1, dd1 = 2.0 * d1 * d0, dd0 = d0 * d0;
    // n^2 - 2 cg n d + d^2 w  (n d is cubic: it contributes to v^3..v^0 only)
    const double A4 = n2 * n2 + dd2 * w2;
    const double A3 = 2.0 * n2 * n1 - 2.0 * cg * (n2 * d1) + (dd2 * w1 + dd1 * w2);
    const double A2 = (n1 * n1 + 2.0 * n2 * n0) - 2.0 * cg * (n2 * d0 + n1 * d1) + (dd2 * w0 + dd1 * w1 + dd0 * w2);
    const double A1 = 2.0 * n1 * n0 - 2.0 * cg * (n1 * d0 + n0 * d1) + (dd1 * w0 + dd0 * w1);
    const double A0 = n0 * n0 - 2.0 * cg * (n0 * d0) + dd0 * w0;
    const double amax = fmax(fmax(fabs(A4), fabs(A3)), fmax(fmax(fabs(A2), fabs(A1)), fabs(A0)));
    if (!(fabs(A4) > 1e-12 * amax)) return 0;
    double roots[4];
    const int nr = solve_quartic_monic(A3 / A4, A2 / A4, A1 / A4, A0 / A4, roots);

    double eP[9];
    if (!tri_frame(P[0], P[1], P[2], eP)) return 0;
    int ns = 0;
    for (int k = 0; k < nr; ++k) {
        double v = roots[k];
        // two Newton polish steps on the un-normalised quartic
        for (int it = 0; it < 2; ++it) {
            const double fv = (((A4 * v + A3) * v + A2) * v + A1) * v + A0;
            const double dfv = ((4.0 * A4 * v + 3.0 * A3) * v + 2.0 * A2) * v + A1;
            if (dfv != 0.0) v -= fv / dfv;
        }
        if (!(v > 0.0)) continue;
        const double den = d1 * v + d0;
        if (!(fabs(den) > 1e-12)) continue;
        const double u = ((n2 * v + n1) * v + n0) / den;
        if (!(u > 0.0)) continue;
        const double qv = (v - 2.0 * cb) * v + 1.0;
        if (!(qv > 0.0)) continue;
        const double s1 = sqrt(b2 / qv), s2 = u * s1, s3 = v * s1;
        double Q[3][3];
        for (int c = 0; c < 3; ++c) {
            Q[0][c] = s1 * f[0][c]; Q[1][c] = s2 * f[1][c]; Q[2][c] = s3 * f[2][c];
        }
        double eQ[9];
        if (!tri_frame(Q[0], Q[1], Q[2], eQ)) continue;
        PoseD &o = sol[ns];
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) o.r[3 * i + j] = eQ[i] * eP[j] + eQ[3 + i] * eP[3 + j] + eQ[6 + i] * eP[6 + j];
        for (int i = 0; i < 3; ++i)
            o.t[i] = Q[0][i] - (o.r[3 * i] * P[0][0] + o.r[3 * i + 1] * P[0][1] + o.r[3 * i + 2] * P[0][2]);
        ++ns;
    }
    return ns;
}

// 3 points + 1: solve P3P on the first three, keep the solution with the smallest reprojection
// error of the 4th (positive depth required).  false when no admissible solution exists.
VO_HD bool p3p_solve4(const double P[4][3], const double uv[4][2], double fx, double fy, double cx, double cy,
                      PoseD &best) {
    PoseD sol[4];
    const int ns = p3p_solve(P, uv, fx, fy, cx, cy, sol);
    double best_err = 1e300;
    int best_k = -1;
    for (int k = 0; k < ns; ++k) {
        const PoseD &s = sol[k];
        const double x = s.r[0] * P[3][0] + s.r[1] * P[3][1] + s.r[2] * P[3][2] + s.t[0];
        const double y = s.r[3] * P[3][0] + s.r[4] * P[3][1] + s.r[5] * P[3][2] + s.t[1];
        const double z = s.r[6] * P[3][0] + s.r[7] * P[3][1] + s.r[8] * P[3][2] + s.t[2];
        if (!(z > 0.0)) continue;
        const double du = fx * (x / z) + cx - uv[3][0], dv = fy * (y / z) + cy - uv[3][1];
        const double e = du * du + dv * dv;
        if (e < best_err) { best_err = e; best_k = k; }
    }
    if (best_k < 0) return false;
    best = sol[best_k];
    return true;
}

}  // namespace vo
