// K2 geometry: per-sample decode -> colour -> Sampson gate -> DLT triangulation -> reprojection / cheirality /
//              parallax filters.  One thread per sampled pixel, grid = (128-sample tiles, reference views).
// K2b fix-up : the few samples whose null-vector iteration did not converge (grossly inconsistent matches)
//              are re-evaluated with a Jacobi eigen-solver from a device-side worklist.
// K3 pack    : ordered stream compaction of the kept samples into the packed point cloud, fully parallel
//              (grid = tiles x views) from per-tile group counts written by K2.
//
// Replaces reference core/pipeline.py:652-780 and core/geometry.py:58-141 (see the per-step citations).
// Arithmetic mirrors the reference's dtype flow and operation order (SURVEY.md 8a):
//   * decode / pixel scaling / DLT rows / reprojection / parallax in f32 with NO fused multiply-add
//     except where the reference's sgemm uses one (the 4-term projection dot products);
//   * Sampson distance and the bilinear colour weights in f64;
//   * the 4x4 null vector: the reference calls LAPACK's f32 SVD; here it is the eigenvector of the
//     smallest eigenvalue of A^T A in f64 (shifted inverse iteration; Jacobi fallback) -- both sit ~1e-7
//     relative from the exact singular vector of the same f32 matrix; tolerance 1e-4 rel / 1e-5 abs.
//   * threshold comparisons that the reference makes on a quotient or on arccos are made division-free /
//     arccos-free where a rigorous bound decides them, and exactly otherwise (same verdicts).
// Per-pair camera constants (P1,P2,C1,C2,F, pixel scales, group ids) are staged in shared memory.
#include "ldp_device.cuh"

namespace ldp {

#ifndef K2_TILE
#define K2_TILE 128
#endif
constexpr int K2_THREADS = K2_TILE;
#ifndef K2_MIN_BLOCKS
#define K2_MIN_BLOCKS 8
#endif
constexpr int K3_THREADS = K2_TILE;
constexpr int KFIX_BLOCKS = 148;
// np.degrees on float32 multiplies by f32(180) / f32(pi) evaluated in f32 (measured, DESIGN.md)
#define RAD2DEG_F32 57.295776367187500f

// The neighbours' constants, staged in shared memory as one table per field, each in the descriptor's own order: staging is a
// word copy with a few range checks (no divisions), rows of P2 stay 16-byte aligned (128-bit reads), and the lanes of a warp that
// read the same field of DIFFERENT neighbours hit different banks (row strides of 12 / 9 / 3 / 1 words).
struct PairTable {
    alignas(16) float P2[LDP_MAX_NN][12];
    float F[LDP_MAX_NN][9];
    float C2[LDP_MAX_NN][3];
    float sxB[LDP_MAX_NN], syB[LDP_MAX_NN];
    int group[LDP_MAX_NN];
    const float* warp[LDP_MAX_NN];
    const float* cert[LDP_MAX_NN];
};
struct PairView {           // neighbour k of the table
    const float* P2; const float* C2; const float* F;
    float sxB, syB;
    int group;
    const float* warp;
};
__device__ __forceinline__ PairView pair_view(const PairTable& pt, int k) {
    PairView v;
    v.P2 = pt.P2[k]; v.C2 = pt.C2[k]; v.F = pt.F[k];
    v.sxB = pt.sxB[k]; v.syB = pt.syB[k]; v.group = pt.group[k]; v.warp = pt.warp[k];
    return v;
}
struct RefConst {
    float P1[12];
    float C1[3];
    float sxA, syA, sx_img, sy_img;
    int img_w, img_h, nn;
    const uint8_t* image;
};
struct GeomArgs {           // launch-constant extras computed on the host
    float par_cos_max;      // parallax: keep iff clip(cos) <= par_cos_max  (== f32 arccos/degrees test, see ldp_api.cu)
    int have_bestk;
    int nb2;                // 128-sample tiles per view
    // test hook, read by the multiview instantiations only (ldp_debug_force_fixup): n > 0 sends every sample i with i % n == 0
    // to the fix-up as if its two-view solve (force_fix_two) / its multi-view solve (force_fix_mv) had not converged
    int force_fix_two, force_fix_mv;
};

// The workspace rows are dead once their last consumer ran; telling L2 so spares the write-back of lines
// that the next launch overwrites anyway (48 MB per 46-view step at 512^2; measured -4 us per step.  The same for
// the 12 MB of winning-neighbour rows measured no gain).
__device__ __forceinline__ void l2_discard_line(const void* p) {
    asm volatile("discard.global.L2 [%0], 128;" :: "l"(p) : "memory");
}

// The view's camera constants, descriptor -> shared memory, in ONE global round trip: the 451 words from sxA to group[] are
// contiguous in ldp_ref_desc, every thread loads its words (and pointers) before it stores any of them, and nothing depends
// on a loaded value (the rows beyond nn are copied too: never read).  A CTA's warps sit through this before they can do
// anything else, 3634 times per step: the per-field loops it replaces cost eight dependent round trips (4.7k cycles of 23k).
constexpr int DESC_WORDS = 4 + 12 + 3 + LDP_MAX_NN * (12 + 3 + 9 + 3);
static_assert(offsetof(ldp_ref_desc, group) + sizeof(int32_t) * LDP_MAX_NN - offsetof(ldp_ref_desc, sxA) == DESC_WORDS * 4, "descriptor layout");
static_assert(offsetof(RefConst, sy_img) - offsetof(RefConst, sxA) == 12, "RefConst layout");
__device__ __forceinline__ uint32_t* desc_word_slot(int e, RefConst& rc, PairTable& pt) {
    if (e < 4) return reinterpret_cast<uint32_t*>(&rc.sxA) + e;
    if (e < 16) return reinterpret_cast<uint32_t*>(rc.P1) + (e - 4);
    if (e < 19) return reinterpret_cast<uint32_t*>(rc.C1) + (e - 16);
    e -= 19;
    if (e < LDP_MAX_NN * 12) return reinterpret_cast<uint32_t*>(&pt.P2[0][0]) + e;
    e -= LDP_MAX_NN * 12;
    if (e < LDP_MAX_NN * 3) return reinterpret_cast<uint32_t*>(&pt.C2[0][0]) + e;
    e -= LDP_MAX_NN * 3;
    if (e < LDP_MAX_NN * 9) return reinterpret_cast<uint32_t*>(&pt.F[0][0]) + e;
    e -= LDP_MAX_NN * 9;
    if (e < LDP_MAX_NN) return reinterpret_cast<uint32_t*>(pt.sxB) + e;
    e -= LDP_MAX_NN;
    if (e < LDP_MAX_NN) return reinterpret_cast<uint32_t*>(pt.syB) + e;
    return reinterpret_cast<uint32_t*>(pt.group) + (e - LDP_MAX_NN);
}
// stage_load puts the loads in flight (registers), stage_store waits for them: a kernel issues its other independent loads in
// between.  slices > 0: the CTA also asks L2 for its share (slice of slices) of the view's reference image.
constexpr int DESC_PER = 4;                                   // words per thread: one pass for CTAs of >= 113 threads
struct StagedDesc {
    uint32_t v[DESC_PER];
    const float* p_warp; const float* p_cert; const uint8_t* p_img;
    int img_w, img_h, nn;
};
__device__ __forceinline__ void stage_load(const ldp_ref_desc* rd, int t, int nt, StagedDesc& sd) {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(&rd->sxA);
    sd.p_warp = nullptr; sd.p_cert = nullptr; sd.p_img = nullptr; sd.img_w = sd.img_h = sd.nn = 0;
    if (t < LDP_MAX_NN) { sd.p_warp = rd->warp[t]; sd.p_cert = rd->cert[t]; }
    if (t == LDP_MAX_NN) { sd.p_img = rd->image; sd.img_w = rd->img_w; sd.img_h = rd->img_h; sd.nn = rd->nn; }
#pragma unroll
    for (int q = 0; q < DESC_PER; ++q) sd.v[q] = (t + q * nt < DESC_WORDS) ? __ldg(src + t + q * nt) : 0u;
}
__device__ __forceinline__ void stage_store(const StagedDesc& sd, RefConst& rc, PairTable& pc, int t, int nt,
                                            int slice = 0, int slices = 0) {
#pragma unroll
    for (int q = 0; q < DESC_PER; ++q) if (t + q * nt < DESC_WORDS) *desc_word_slot(t + q * nt, rc, pc) = sd.v[q];
    if (t < LDP_MAX_NN) { pc.warp[t] = sd.p_warp; pc.cert[t] = sd.p_cert; }
    if (t == LDP_MAX_NN) {
        rc.image = sd.p_img; rc.img_w = sd.img_w; rc.img_h = sd.img_h; rc.nn = sd.nn;
        if (slices > 0) l2_prefetch_slice(sd.p_img, (size_t)sd.img_w * sd.img_h * 3, slice, slices);
    }
}
__device__ __forceinline__ void stage_constants(const ldp_ref_desc* rd, RefConst& rc, PairTable& pc, int t, int nt) {
    StagedDesc sd;
    stage_load(rd, t, nt, sd);
    stage_store(sd, rc, pc, t, nt);
}
static_assert(DESC_PER * 113 >= DESC_WORDS, "stage_load covers the descriptor in one pass");

// Cyclic Jacobi eigen-decomposition of the symmetric 4x4 M (f64): eigenvector of the smallest eigenvalue.
__device__ void jacobi_smallest_eigvec4(const double* __restrict__ Min, double* __restrict__ vout) {
    double a[4][4], V[4][4];
    a[0][0] = Min[0]; a[1][0] = a[0][1] = Min[1]; a[1][1] = Min[2];
    a[2][0] = a[0][2] = Min[3]; a[2][1] = a[1][2] = Min[4]; a[2][2] = Min[5];
    a[3][0] = a[0][3] = Min[6]; a[3][1] = a[1][3] = Min[7]; a[3][2] = a[2][3] = Min[8]; a[3][3] = Min[9];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) V[i][j] = (i == j) ? 1.0 : 0.0;
    const double tr = a[0][0] + a[1][1] + a[2][2] + a[3][3];
    const double tiny = tr * tr * 1e-28;      // off-diagonal mass: eigenvector good to ~1e-13 (quadratic convergence)
    for (int sweep = 0; sweep < 16; ++sweep) {
        const double off = a[0][1] * a[0][1] + a[0][2] * a[0][2] + a[0][3] * a[0][3] +
                           a[1][2] * a[1][2] + a[1][3] * a[1][3] + a[2][3] * a[2][3];
        if (!(off > tiny)) break;
#pragma unroll
        for (int p = 0; p < 3; ++p) {
#pragma unroll
            for (int q = p + 1; q < 4; ++q) {
                const double apq = a[p][q];
                if (fabs(apq) > 1e-300) {
                    const double tau = (a[q][q] - a[p][p]) / (2.0 * apq);
                    const double t = ((tau >= 0.0) ? 1.0 : -1.0) / (fabs(tau) + sqrt(1.0 + tau * tau));
                    const double c = rsqrt(1.0 + t * t), sn = t * c;
                    a[p][p] -= t * apq;
                    a[q][q] += t * apq;
                    a[p][q] = a[q][p] = 0.0;
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        if (k != p && k != q) {
                            const double akp = a[k][p], akq = a[k][q];
                            a[k][p] = a[p][k] = c * akp - sn * akq;
                            a[k][q] = a[q][k] = sn * akp + c * akq;
                        }
                    }
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const double vkp = V[k][p], vkq = V[k][q];
                        V[k][p] = c * vkp - sn * vkq;
                        V[k][q] = sn * vkp + c * vkq;
                    }
                }
            }
        }
    }
    int j = 0;
    double best = a[0][0];
    if (a[1][1] < best) { best = a[1][1]; j = 1; }
    if (a[2][2] < best) { best = a[2][2]; j = 2; }
    if (a[3][3] < best) { best = a[3][3]; j = 3; }
#pragma unroll
    for (int k = 0; k < 4; ++k) vout[k] = (j == 0) ? V[k][0] : (j == 1) ? V[k][1] : (j == 2) ? V[k][2] : V[k][3];
}

// 1/sqrt(s) and 1/v in f64 for s, v in the normal range, to within a few ulp: the hardware's 2^-22 estimate and two Newton steps,
// without the library routines' special-case paths (zero, infinity, denormals come out as NaN here: the callers' pivots are
// clamped positive, and a NaN eigenvector ends in the Jacobi fix-up like any other non-convergence).  Neither value needs to be
// correctly rounded: one scales an iterate, the other is multiplied and rounded to f32.
__device__ __forceinline__ double rsqrt_newton(double s) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(s));
#pragma unroll
    for (int q = 0; q < 2; ++q) { const double t = s * y; const double e = fma(-t, y, 1.0); y = fma(0.5 * y, e, y); }
    return y;
}
__device__ __forceinline__ double rcp_newton(double v) {
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(v));
#pragma unroll
    for (int q = 0; q < 2; ++q) { const double e = fma(-v, y, 1.0); y = fma(y, e, y); }
    return y;
}

// Smallest-eigenvalue eigenvector of M = A^T A (A 4x4 row-major, f32 values held in f64).
// ROBUST = false: inverse iteration on the Cholesky factor of M + mu*I (same eigenvectors; converges at
// (sigma_4/sigma_3)^2 per step: 3-5 steps on consistent matches); returns false if not converged in INVIT_MAX.
// ROBUST = true : Jacobi.
constexpr int INVIT_MAX = 24;     // slow convergers are rare; iterating on is far cheaper than the Jacobi fix-up
struct Gram { double m00, m10, m11, m20, m21, m22, m30, m31, m32, m33; };       // lower triangle of A^T A
__device__ __forceinline__ void gram_add_row(Gram& g, double a, double b, double c, double d) {
    g.m00 = fma(a, a, g.m00); g.m10 = fma(b, a, g.m10); g.m11 = fma(b, b, g.m11);
    g.m20 = fma(c, a, g.m20); g.m21 = fma(c, b, g.m21); g.m22 = fma(c, c, g.m22);
    g.m30 = fma(d, a, g.m30); g.m31 = fma(d, b, g.m31); g.m32 = fma(d, c, g.m32); g.m33 = fma(d, d, g.m33);
}
template <bool ROBUST>
__device__ __forceinline__ bool null_vector_gram(const Gram& g, double v[4]) {
    const double m00 = g.m00, m10 = g.m10, m11 = g.m11, m20 = g.m20, m21 = g.m21, m22 = g.m22;
    const double m30 = g.m30, m31 = g.m31, m32 = g.m32, m33 = g.m33;
    const double tr = m00 + m11 + m22 + m33;
    if (!(tr > 0.0) || !isfinite(tr)) { v[0] = v[1] = v[2] = 0.0; v[3] = 1.0; if (!(tr == tr)) v[0] = tr; return true; }
    if (ROBUST) {
        const double Ms[10] = {m00, m10, m11, m20, m21, m22, m30, m31, m32, m33};
        jacobi_smallest_eigvec4(Ms, v);
        return true;
    }
    // M + mu*I has the same eigenvectors; the shift keeps the Cholesky pivots positive when A is
    // numerically rank-3 (noise-free correspondences).
    const double mu = tr * 1e-13;
    const double i0 = rsqrt_newton(m00 + mu);
    const double l10 = m10 * i0, l20 = m20 * i0, l30 = m30 * i0;
    const double i1 = rsqrt_newton(fmax(m11 + mu - l10 * l10, mu * 1e-3));
    const double l21 = (m21 - l20 * l10) * i1, l31 = (m31 - l30 * l10) * i1;
    const double i2 = rsqrt_newton(fmax(m22 + mu - l20 * l20 - l21 * l21, mu * 1e-3));
    const double l32 = (m32 - l30 * l20 - l31 * l21) * i2;
    const double i3 = rsqrt_newton(fmax(m33 + mu - l30 * l30 - l31 * l31 - l32 * l32, mu * 1e-3));
    // Steps 1 and 2 are taken without normalising or testing: from x = e4 the forward solve is y = (0, 0, 0, i3), and two
    // steps grow the vector by at most 1 / mu^2 (far inside the f64 range for any tr that is not itself denormal-small;
    // an overflow would end in the Jacobi fix-up like any other non-convergence).  The test needs two normalised iterates
    // anyway, so nothing converges later than before.
    double x0, x1, x2, x3;
    {
        const double z3 = i3 * i3;
        const double z2 = (-l32 * z3) * i2;
        const double z1 = (-l21 * z2 - l31 * z3) * i1;
        const double z0 = (-l10 * z1 - l20 * z2 - l30 * z3) * i0;
        const double y0 = z0 * i0;
        const double y1 = (z1 - l10 * y0) * i1;
        const double y2 = (z2 - l20 * y0 - l21 * y1) * i2;
        const double y3 = (z3 - l30 * y0 - l31 * y1 - l32 * y2) * i3;
        const double w3 = y3 * i3;
        const double w2 = (y2 - l32 * w3) * i2;
        const double w1 = (y1 - l21 * w2 - l31 * w3) * i1;
        const double w0 = (y0 - l10 * w1 - l20 * w2 - l30 * w3) * i0;
        const double inv = rsqrt_newton(w0 * w0 + w1 * w1 + w2 * w2 + w3 * w3);
        x0 = w0 * inv; x1 = w1 * inv; x2 = w2 * inv; x3 = w3 * inv;
    }
    bool converged = false;
    for (int it = 2; it < INVIT_MAX; ++it) {
        const double y0 = x0 * i0;                                   // L y = x
        const double y1 = (x1 - l10 * y0) * i1;
        const double y2 = (x2 - l20 * y0 - l21 * y1) * i2;
        const double y3 = (x3 - l30 * y0 - l31 * y1 - l32 * y2) * i3;
        const double z3 = y3 * i3;                                   // L^T z = y
        const double z2 = (y2 - l32 * z3) * i2;
        const double z1 = (y1 - l21 * z2 - l31 * z3) * i1;
        const double z0 = (y0 - l10 * z1 - l20 * z2 - l30 * z3) * i0;
        // (no sign to fix: z . x = |L^-1 x|^2 >= 0, the factorised matrix is positive definite by construction)
        const double inv = rsqrt_newton(z0 * z0 + z1 * z1 + z2 * z2 + z3 * z3);
        const double n0 = z0 * inv, n1 = z1 * inv, n2 = z2 * inv, n3 = z3 * inv;
        const double e0 = n0 - x0, e1 = n1 - x1, e2 = n2 - x2, e3 = n3 - x3;
        x0 = n0; x1 = n1; x2 = n2; x3 = n3;
        if (e0 * e0 + e1 * e1 + e2 * e2 + e3 * e3 < 1e-26) { converged = true; break; }
    }
    v[0] = x0; v[1] = x1; v[2] = x2; v[3] = x3;
    return converged;
}
template <bool ROBUST>
__device__ __forceinline__ bool null_vector4(const double A[16], double v[4]) {
    Gram g = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int r = 0; r < 4; ++r) gram_add_row(g, A[4 * r], A[4 * r + 1], A[4 * r + 2], A[4 * r + 3]);
    return null_vector_gram<ROBUST>(g, v);
}

// X @ P^T row: the reference's sgemm accumulates the K=4 products with FMAs in index order
// (measured against numpy/OpenBLAS, DESIGN.md); same here.
__device__ __forceinline__ float proj_row(const float* p, float X0, float X1, float X2, float X3) {
    float acc = __fmul_rn(X0, p[0]);
    acc = __fmaf_rn(X1, p[1], acc);
    acc = __fmaf_rn(X2, p[2], acc);
    acc = __fmaf_rn(X3, p[3], acc);
    return acc;
}

// core/geometry.py:91-104
__device__ __forceinline__ float reproj_err(const float* P, float X0, float X1, float X2, float X3,
                                            float u, float v, float* zout) {
    const float q0 = proj_row(P, X0, X1, X2, X3), q1 = proj_row(P + 4, X0, X1, X2, X3), q2 = proj_row(P + 8, X0, X1, X2, X3);
    *zout = q2;
    const float z = fmaxf(q2, 1e-12f);
    const float du = __fsub_rn(__fdiv_rn(q0, z), u), dv = __fsub_rn(__fdiv_rn(q1, z), v);
    return __fsqrt_rn(__fadd_rn(__fmul_rn(du, du), __fmul_rn(dv, dv)));
}

// Three channels of the texels (x0,y) and (x0+1,y) of a [h,w,3] u8 image: 6 consecutive bytes starting at `off`,
// fetched as three aligned 32-bit words (instead of six byte loads) when the window stays inside the image.
__device__ __forceinline__ void fetch_texel_pair(const uint8_t* __restrict__ im, size_t off, size_t total, bool two,
                                                 float t0[3], float t1[3]) {
    const size_t base = off & ~(size_t)3;
    if ((reinterpret_cast<size_t>(im) & 3) == 0 && base + 12 <= total) {
        const uint32_t* wp = reinterpret_cast<const uint32_t*>(im + base);
        const uint32_t w0 = __ldg(wp), w1 = __ldg(wp + 1), w2 = __ldg(wp + 2);
        const unsigned sh = (unsigned)(off & 3) * 8u;
        const uint32_t a = __funnelshift_r(w0, w1, sh), b = __funnelshift_r(w1, w2, sh);   // bytes off..off+3, off+4..off+7
        t0[0] = (float)(a & 0xffu); t0[1] = (float)((a >> 8) & 0xffu); t0[2] = (float)((a >> 16) & 0xffu);
        if (two) { t1[0] = (float)(a >> 24); t1[1] = (float)(b & 0xffu); t1[2] = (float)((b >> 8) & 0xffu); }
        else { t1[0] = t0[0]; t1[1] = t0[1]; t1[2] = t0[2]; }
    } else {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            t0[c] = (float)__ldg(im + off + c);
            t1[c] = two ? (float)__ldg(im + off + 3 + c) : t0[c];
        }
    }
}

// ---- lens models (include/ldp_b200.h: ldp_lens).  Not in the reference, which triangulates every camera as a pinhole.
// The inversion is Newton's method in f64 from the distorted point; it stops when the step is below LENS_STEP_TOL normalised
// units, and fails (NaN) after LENS_MAX_ITERS steps, or when the Jacobian determinant (fisheye: d theta_d / d theta) is not
// positive at an iterate -- past the fold of the polynomial, where the inverse is not unique -- or when the fisheye angle
// it converges to lies outside [0, pi/2).  tests/lens_oracle.py restates the same rule.
constexpr int LENS_MAX_ITERS = 20;
constexpr double LENS_STEP_TOL = 1e-12;
constexpr double LENS_HALF_PI = 1.5707963267948966;
constexpr double LENS_FISHEYE_THETA0_MAX = 1.5707963267948966 - 1e-6;   // fisheye: the first iterate lies inside [0, pi/2)

__device__ __forceinline__ void lens_distort(const ldp_lens& L, double x, double y, double& xd, double& yd) {
    const double* k = L.k;
    const double r2 = x * x + y * y;
    if (L.model == LDP_LENS_FISHEYE) {
        const double r = sqrt(r2);
        const double th = atan(r), t2 = th * th;
        const double thd = th * (1.0 + t2 * (k[0] + t2 * (k[1] + t2 * (k[2] + t2 * k[3]))));
        const double s = (r > 0.0) ? thd / r : 1.0;
        xd = x * s; yd = y * s;
    } else {
        const double radial = (1.0 + r2 * (k[0] + r2 * (k[1] + r2 * k[4]))) / (1.0 + r2 * (k[5] + r2 * (k[6] + r2 * k[7])));
        xd = x * radial + 2.0 * k[2] * x * y + k[3] * (r2 + 2.0 * x * x);
        yd = y * radial + k[2] * (r2 + 2.0 * y * y) + 2.0 * k[3] * x * y;
    }
}

// normalised distorted (xd, yd) -> normalised ideal (x, y); false (and NaN) where there is no valid inverse
__device__ __forceinline__ bool lens_undistort(const ldp_lens& L, double xd, double yd, double& x, double& y) {
    const double* k = L.k;
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    if (L.model == LDP_LENS_FISHEYE) {
        const double rd = sqrt(xd * xd + yd * yd);
        if (rd == 0.0) { x = xd; y = yd; return true; }
        // start at r_d, clamped into the valid range like cv2.fisheye: when theta_d(pi/2) > pi/2 (positive coefficients) the
        // distorted radii in [pi/2, theta_d(pi/2)) have a solution inside it; only the solution's range is checked
        double th = fmin(rd, LENS_FISHEYE_THETA0_MAX);
        bool ok = false;
        for (int it = 0; it < LENS_MAX_ITERS; ++it) {
            const double t2 = th * th;
            const double f = th * (1.0 + t2 * (k[0] + t2 * (k[1] + t2 * (k[2] + t2 * k[3])))) - rd;
            const double d = 1.0 + t2 * (3.0 * k[0] + t2 * (5.0 * k[1] + t2 * (7.0 * k[2] + t2 * 9.0 * k[3])));
            if (!(d > 0.0)) break;
            const double step = f / d;
            th -= step;
            if (fabs(step) < LENS_STEP_TOL) { ok = th >= 0.0 && th < LENS_HALF_PI; break; }
        }
        if (!ok) { x = y = nan; return false; }
        const double s = tan(th) / rd;
        x = xd * s; y = yd * s;
        return true;
    }
    double u = xd, v = yd;
    for (int it = 0; it < LENS_MAX_ITERS; ++it) {
        const double r2 = u * u + v * v;
        const double a = 1.0 + r2 * (k[0] + r2 * (k[1] + r2 * k[4]));
        const double b = 1.0 + r2 * (k[5] + r2 * (k[6] + r2 * k[7]));
        const double da = k[0] + r2 * (2.0 * k[1] + r2 * 3.0 * k[4]);      // d a / d r2
        const double db = k[5] + r2 * (2.0 * k[6] + r2 * 3.0 * k[7]);
        const double radial = a / b;
        const double drad = (da * b - a * db) / (b * b);                     // d radial / d r2
        const double fx = u * radial + 2.0 * k[2] * u * v + k[3] * (r2 + 2.0 * u * u) - xd;
        const double fy = v * radial + k[2] * (r2 + 2.0 * v * v) + 2.0 * k[3] * u * v - yd;
        const double j00 = radial + 2.0 * u * u * drad + 2.0 * k[2] * v + 6.0 * k[3] * u;
        const double j01 = 2.0 * u * v * drad + 2.0 * k[2] * u + 2.0 * k[3] * v;
        const double j10 = 2.0 * u * v * drad + 2.0 * k[2] * u + 2.0 * k[3] * v;
        const double j11 = radial + 2.0 * v * v * drad + 6.0 * k[2] * v + 2.0 * k[3] * u;
        const double det = j00 * j11 - j01 * j10;
        if (!(det > 0.0)) break;
        const double du = (j11 * fx - j01 * fy) / det, dv = (j00 * fy - j10 * fx) / det;
        u -= du; v -= dv;
        if (du * du + dv * dv < LENS_STEP_TOL * LENS_STEP_TOL) { x = u; y = v; return true; }
    }
    x = y = nan;
    return false;
}

// f32 observed pixel -> f32 ideal pinhole pixel of the same camera (NaN where the lens has no valid inverse)
__device__ __forceinline__ void lens_undistort_px(const ldp_lens& L, float u, float v, float& ui, float& vi) {
    const double fx = L.fx, fy = L.fy, cx = L.cx, cy = L.cy;
    double x, y;
    lens_undistort(L, ((double)u - cx) / fx, ((double)v - cy) / fy, x, y);
    ui = (float)(fx * x + cx); vi = (float)(fy * y + cy);
}

// reprojection error in the distorted image: the f32 projection q (as reproj_err forms it) through the forward lens, in f64
__device__ __forceinline__ float lens_reproj_err(const ldp_lens& L, const float* P, float X0, float X1, float X2, float X3,
                                                 float u, float v, float* zout) {
    const float q0 = proj_row(P, X0, X1, X2, X3), q1 = proj_row(P + 4, X0, X1, X2, X3), q2 = proj_row(P + 8, X0, X1, X2, X3);
    *zout = q2;
    const double z = (double)fmaxf(q2, 1e-12f);
    const double fx = L.fx, fy = L.fy, cx = L.cx, cy = L.cy;
    double xd, yd;
    lens_distort(L, ((double)q0 / z - cx) / fx, ((double)q1 / z - cy) / fy, xd, yd);
    const double du = fx * xd + cx - (double)u, dv = fy * yd + cy - (double)v;
    return (float)sqrt(du * du + dv * dv);
}

// The Sampson gate, the dehomogenisation and the parallax test for the multi-view refinement (mv_refine): the same
// arithmetic as eval_sample's inline copies, which stay inline because factoring them out changes the two-view kernels'
// register allocation and spills (DESIGN.md 4.4).
// Sampson gate in f64: core/geometry.py:133-141, core/pipeline.py:708-727.  se < thr is decided on num^2 vs thr*den outside
// a 2^-50 band, by the reference's quotient inside it.
__device__ __forceinline__ int sampson_pass(const float* F, double a0, double a1, double b0, double b1, double thr) {
    const double l0 = (double)F[0] * a0 + (double)F[1] * a1 + (double)F[2];
    const double l1 = (double)F[3] * a0 + (double)F[4] * a1 + (double)F[5];
    const double l2 = (double)F[6] * a0 + (double)F[7] * a1 + (double)F[8];
    const double m0 = (double)F[0] * b0 + (double)F[3] * b1 + (double)F[6];
    const double m1 = (double)F[1] * b0 + (double)F[4] * b1 + (double)F[7];
    const double num = b0 * l0 + b1 * l1 + l2;
    const double den = l0 * l0 + l1 * l1 + m0 * m0 + m1 * m1 + 1e-12;
    const double n2 = num * num, td = thr * den;
    int good;
    if (n2 < td * (1.0 - 1.0 / 1125899906842624.0)) good = 1;
    else if (n2 > td * (1.0 + 1.0 / 1125899906842624.0)) good = 0;
    else good = (__ddiv_rn(n2, den) < thr) ? 1 : 0;
    if (!(n2 == n2) || !(den == den)) good = 0;                                  // NaN: comparison is False in numpy
    return good;
}

// core/geometry.py:85-87: w = where(|Xh3| < 1e-12, 1e-12, Xh3); X = Xh / w
__device__ __forceinline__ void dehomogenise(const double v[4], float& X0, float& X1, float& X2, float& X3) {
    const float w32 = (float)v[3];
    if (fabsf(w32) < 1e-12f) {
        X0 = __fdiv_rn((float)v[0], 1e-12f); X1 = __fdiv_rn((float)v[1], 1e-12f);
        X2 = __fdiv_rn((float)v[2], 1e-12f); X3 = __fdiv_rn(w32, 1e-12f);
    } else {
        const double iwv = rcp_newton(v[3]);
        X0 = (float)(v[0] * iwv); X1 = (float)(v[1] * iwv); X2 = (float)(v[2] * iwv); X3 = 1.0f;
    }
}

// parallax filter, core/geometry.py:113-119
__device__ __forceinline__ bool parallax_pass(float X0, float X1, float X2, const float* C1, const float* C2, float par_cos_max) {
    float a0 = __fsub_rn(X0, C1[0]), a1 = __fsub_rn(X1, C1[1]), a2 = __fsub_rn(X2, C1[2]);
    float b0 = __fsub_rn(X0, C2[0]), b1 = __fsub_rn(X1, C2[1]), b2 = __fsub_rn(X2, C2[2]);
    const float na = __fadd_rn(__fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(a0, a0), __fmul_rn(a1, a1)), __fmul_rn(a2, a2))), 1e-12f);
    const float nb = __fadd_rn(__fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(b0, b0), __fmul_rn(b1, b1)), __fmul_rn(b2, b2))), 1e-12f);
    a0 = __fdiv_rn(a0, na); a1 = __fdiv_rn(a1, na); a2 = __fdiv_rn(a2, na);
    b0 = __fdiv_rn(b0, nb); b1 = __fdiv_rn(b1, nb); b2 = __fdiv_rn(b2, nb);
    float d = __fadd_rn(__fadd_rn(__fmul_rn(a0, b0), __fmul_rn(a1, b1)), __fmul_rn(a2, b2));
    const bool dnan = (d != d);
    d = fminf(fmaxf(d, -1.0f), 1.0f);
    // degrees(arccos(d)) >= min_deg  <=>  d <= par_cos_max (arccos is monotone; threshold found on the host)
    return !dnan && d <= par_cos_max;
}

struct SampleResult {
    float X0, X1, X2, err;
    float z1;               // the reference camera's depth of the point (reproj_err's z), NaN where not triangulated
    float cr, cg, cb, dcert;
    float4 dbg;
    int keep, good, grp;
    bool converged;
};

#ifdef LDP_GEOM_CLOCKS   // dev (scratch/geom_clocks.py): cycles per phase of warp 0 of three CTAs of every view, in ws.dbgclk
#define GCLK_DECL long long gck[12] = {0,0,0,0,0,0,0,0,0,0,0,0}; long long gck_last = clock64();
#define GCLK_ARGS , long long* gck, long long& gck_last
#define GCLK_PASS , gck, gck_last
#define GCLK(slot) do { const long long t_ = clock64(); gck[slot] += t_ - gck_last; gck_last = t_; } while (0)
__device__ __forceinline__ void gclk_use(float x) { asm volatile("" :: "f"(x)); }
__device__ __forceinline__ void gclk_use(int x) { asm volatile("" :: "r"(x)); }
__device__ __forceinline__ void gclk_use(uint32_t x) { asm volatile("" :: "r"(x)); }
#define GCLK_USE(x) gclk_use(x)
#define GCLK_FLUSH do { if (threadIdx.x == 0 && (blockIdx.x == 5 || blockIdx.x == 40 || blockIdx.x == 70)) for (int q_ = 0; q_ < 12; ++q_) ws.dbgclk[(size_t)r * 32 + (blockIdx.x == 5 ? 0 : blockIdx.x == 40 ? 1 : 2) * 12 + q_] = gck[q_]; } while (0)   /* three CTAs per view, plain stores */
#else
#define GCLK_DECL
#define GCLK_ARGS
#define GCLK_PASS
#define GCLK(slot) do { } while (0)
#define GCLK_USE(x) do { } while (0)
#define GCLK_FLUSH do { } while (0)
#endif

// Per-sample inputs gathered by the geometry kernel; stored (pt0 / pt1) for the samples the fix-up re-evaluates.
struct SampleRec {
    float4 wv;              // winning neighbour's warp row: xA, yA, xB, yB in [-1, 1]
    uint32_t tex[3];        // the four bilinear texels, 3 bytes each: t00 t01 t10 t11
    uint32_t k_cert;        // bits 0..7 neighbour slot k; debug certainty is kept separately
};

// ---- gather: everything that needs a scattered load (core/pipeline.py:636-640,652-653,661-675)
// certainty of neighbour q at pixel idx as the path sees it: raw planes go through the reference's post-processing
__device__ __forceinline__ float cert_at(const ldp_params& P, const PairTable& pc, const ProView& pv, int q, int idx) {
    float c = __ldg(pc.cert[q] + idx);
    if (P.prologue) {
        const int y = idx / P.W;
        c = prologue_cert(c, q, idx, idx - y * P.W, y, P, pv);
    }
    return c;
}

__device__ __forceinline__ void gather_sample(const ldp_params& P, const RefConst& rc, const PairTable& pc, const ProView& pv,
                                              const GeomArgs& ga, int k_pre, int idx,
                                              SampleRec& rec, float& craw) {
    int k = 0;                                                                    // core/pipeline.py:634-635,652
    if (ga.have_bestk) {
        k = k_pre;                         // the stream kernel's winner byte at idx, fetched by the caller
    } else {                               // stage entry point: arg-max over neighbours at the sampled pixel only
        float best = cert_at(P, pc, pv, 0, idx);
        for (int q = 1; q < rc.nn; ++q) {
            const float c = cert_at(P, pc, pv, q, idx);
            if (c > best) { best = c; k = q; }
        }
    }
    const PairView pk = pair_view(pc, k);
    const float4 wv = __ldg(reinterpret_cast<const float4*>(pk.warp) + idx);      // core/pipeline.py:636-640,653
    craw = 0.f;
    if (P.collect_debug) craw = cert_at(P, pc, pv, k, idx);
    const float wm1 = (float)(P.w_match - 1), hm1 = (float)(P.h_match - 1);
    const float xA = __fmul_rn(__fmul_rn(__fadd_rn(wv.x, 1.0f), 0.5f), wm1);
    const float yA = __fmul_rn(__fmul_rn(__fadd_rn(wv.y, 1.0f), 0.5f), hm1);
    const float fx = __fmul_rn(xA, rc.sx_img), fy = __fmul_rn(yA, rc.sy_img);
    const int iw = rc.img_w, ih = rc.img_h;
    const int x0 = min(max((int)fminf(fmaxf(floorf(fx), -1.f), (float)iw), 0), iw - 1);
    const int y0 = min(max((int)fminf(fmaxf(floorf(fy), -1.f), (float)ih), 0), ih - 1);
    const int x1 = min(x0 + 1, iw - 1), y1 = min(y0 + 1, ih - 1);
    float t00[3], t01[3], t10[3], t11[3];
    const size_t img_bytes = (size_t)iw * ih * 3;
    fetch_texel_pair(rc.image, ((size_t)y0 * iw + x0) * 3, img_bytes, x1 != x0, t00, t01);
    fetch_texel_pair(rc.image, ((size_t)y1 * iw + x0) * 3, img_bytes, x1 != x0, t10, t11);
    rec.wv = wv;
    rec.tex[0] = (uint32_t)t00[0] | ((uint32_t)t00[1] << 8) | ((uint32_t)t00[2] << 16) | ((uint32_t)t01[0] << 24);
    rec.tex[1] = (uint32_t)t01[1] | ((uint32_t)t01[2] << 8) | ((uint32_t)t10[0] << 16) | ((uint32_t)t10[1] << 24);
    rec.tex[2] = (uint32_t)t10[2] | ((uint32_t)t11[0] << 8) | ((uint32_t)t11[1] << 16) | ((uint32_t)t11[2] << 24);
    rec.k_cert = (uint32_t)k;
}

// bilinear blend of the four texels at image position (fx, fy) with clipped corners (core/pipeline.py:661-679): f64 weights,
// left-to-right sum like the reference; /255.0 as an FMA-corrected reciprocal multiply.  Shared by eval_sample and the colour
// maps (ldp_depth_colors), so a kept map pixel gets the colour of a sampled pixel with the same winner.
__device__ __forceinline__ void bilinear_rgb(float fx, float fy, int x0, int y0, int x1, int y1, const float t00[3], const float t01[3],
                                             const float t10[3], const float t11[3], float col[3]) {
    const double dfx = (double)fx, dfy = (double)fy;
    const double ax = __dsub_rn((double)x1, dfx), bx = __dsub_rn(dfx, (double)x0);
    const double ay = __dsub_rn((double)y1, dfy), by = __dsub_rn(dfy, (double)y0);
    const double w00 = __dmul_rn(ax, ay), w01 = __dmul_rn(bx, ay), w10 = __dmul_rn(ax, by), w11 = __dmul_rn(bx, by);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        double acc = __dmul_rn((double)t00[c], w00);
        acc = __dadd_rn(acc, __dmul_rn((double)t01[c], w01));
        acc = __dadd_rn(acc, __dmul_rn((double)t10[c], w10));
        acc = __dadd_rn(acc, __dmul_rn((double)t11[c], w11));
        const double q0 = acc * (1.0 / 255.0);
        const double rr = fma(-q0, 255.0, acc);
        col[c] = (float)fma(rr, 1.0 / 255.0, q0);                                 // == acc / 255.0 rounded; .astype(f32) at :754
    }
}

// ---- compute: everything else the reference computes for one sampled pixel (core/pipeline.py:653-769)
// LENS: the launch has lens cameras (ldp_params.lens); lt = the view's staged lens table, [0] reference camera, [1 + k]
// neighbour k.  A lens camera's observed pixels are undistorted before the Sampson gate and the DLT, and its reprojection
// error is measured in the distorted image; a pinhole camera's arithmetic is the same as without LENS.
template <bool ROBUST, bool LENS>
__device__ __forceinline__ void eval_sample(const ldp_params& P, const RefConst& rc, const PairTable& pc, const GeomArgs& ga,
                                            const ldp_lens* lt, const SampleRec& rec, float craw, SampleResult& o GCLK_ARGS) {
    const int k = (int)(rec.k_cert & 0xffu);
    const PairView pk = pair_view(pc, k);
    o.grp = pk.group;
    const float4 wv = rec.wv;
    const float wm1 = (float)(P.w_match - 1), hm1 = (float)(P.h_match - 1);
    // core/pipeline.py:655-656 and 701-702: ((x + 1.0) * 0.5) * (w_match - 1), f32 op by op
    const float xA = __fmul_rn(__fmul_rn(__fadd_rn(wv.x, 1.0f), 0.5f), wm1);
    const float yA = __fmul_rn(__fmul_rn(__fadd_rn(wv.y, 1.0f), 0.5f), hm1);
    const float xB = __fmul_rn(__fmul_rn(__fadd_rn(wv.z, 1.0f), 0.5f), wm1);
    const float yB = __fmul_rn(__fmul_rn(__fadd_rn(wv.w, 1.0f), 0.5f), hm1);

    // ---- colour: core/pipeline.py:661-679 (f64 weights, clipped corners)
    const float fx = __fmul_rn(xA, rc.sx_img), fy = __fmul_rn(yA, rc.sy_img);
    const int iw = rc.img_w, ih = rc.img_h;
    // floor(...).astype(int32) then clip; clamp in float first so the cast cannot overflow
    const int x0 = min(max((int)fminf(fmaxf(floorf(fx), -1.f), (float)iw), 0), iw - 1);
    const int y0 = min(max((int)fminf(fmaxf(floorf(fy), -1.f), (float)ih), 0), ih - 1);
    const int x1 = min(x0 + 1, iw - 1), y1 = min(y0 + 1, ih - 1);
    float t00[3], t01[3], t10[3], t11[3];
    t00[0] = (float)(rec.tex[0] & 0xffu); t00[1] = (float)((rec.tex[0] >> 8) & 0xffu); t00[2] = (float)((rec.tex[0] >> 16) & 0xffu);
    t01[0] = (float)(rec.tex[0] >> 24);   t01[1] = (float)(rec.tex[1] & 0xffu);        t01[2] = (float)((rec.tex[1] >> 8) & 0xffu);
    t10[0] = (float)((rec.tex[1] >> 16) & 0xffu); t10[1] = (float)(rec.tex[1] >> 24);  t10[2] = (float)(rec.tex[2] & 0xffu);
    t11[0] = (float)((rec.tex[2] >> 8) & 0xffu);  t11[1] = (float)((rec.tex[2] >> 16) & 0xffu); t11[2] = (float)(rec.tex[2] >> 24);

    // ---- full-resolution pixel coordinates: core/pipeline.py:681-683, 697-703
    const float uA_obs = __fmul_rn(xA, rc.sxA), vA_obs = __fmul_rn(yA, rc.syA);
    const float uB_obs = __fmul_rn(xB, pk.sxB), vB_obs = __fmul_rn(yB, pk.syB);
    // the ideal pinhole pixels that P, F and the DLT assume
    float uA = uA_obs, vA = vA_obs, uB = uB_obs, vB = vB_obs;
    if constexpr (LENS) {
        if (lt[0].model != LDP_LENS_PINHOLE) lens_undistort_px(lt[0], uA_obs, vA_obs, uA, vA);
        if (lt[1 + k].model != LDP_LENS_PINHOLE) lens_undistort_px(lt[1 + k], uB_obs, vB_obs, uB, vB);
    }

    // ---- Sampson gate in f64: core/geometry.py:133-141, core/pipeline.py:708-727.  se < thr is decided on
    //      num^2 vs thr*den outside a 2^-50 band, by the reference's quotient inside it.
    o.good = 1;
    if (!P.no_filter && P.sampson_thresh > 0.0) {
        const double a0 = uA, a1 = vA, b0 = uB, b1 = vB;
        const float* F = pk.F;
        const double l0 = (double)F[0] * a0 + (double)F[1] * a1 + (double)F[2];
        const double l1 = (double)F[3] * a0 + (double)F[4] * a1 + (double)F[5];
        const double l2 = (double)F[6] * a0 + (double)F[7] * a1 + (double)F[8];
        const double m0 = (double)F[0] * b0 + (double)F[3] * b1 + (double)F[6];
        const double m1 = (double)F[1] * b0 + (double)F[4] * b1 + (double)F[7];
        const double num = b0 * l0 + b1 * l1 + l2;
        const double den = l0 * l0 + l1 * l1 + m0 * m0 + m1 * m1 + 1e-12;
        const double n2 = num * num, td = P.sampson_thresh * den;
        if (n2 < td * (1.0 - 1.0 / 1125899906842624.0)) o.good = 1;
        else if (n2 > td * (1.0 + 1.0 / 1125899906842624.0)) o.good = 0;
        else o.good = (__ddiv_rn(n2, den) < P.sampson_thresh) ? 1 : 0;
        if (!(n2 == n2) || !(den == den)) o.good = 0;                            // NaN: comparison is False in numpy
    }

    {
        float col[3];
        bilinear_rgb(fx, fy, x0, y0, x1, y1, t00, t01, t10, t11, col);
        o.cr = col[0]; o.cg = col[1]; o.cb = col[2];
    }

    GCLK_USE(o.cr); GCLK_USE(o.cg); GCLK_USE(o.cb); GCLK_USE(o.good); GCLK(3);
    o.X0 = o.X1 = o.X2 = 0.f;
    o.err = o.z1 = __int_as_float(0x7fc00000);
    o.keep = 0;
    o.converged = true;
    if (o.good) {          // the reference triangulates only the Sampson survivors (core/pipeline.py:721-733)
        // ---- DLT rows (f32, multiply then subtract): core/geometry.py:72-75
        double A[16];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            A[j]      = (double)__fsub_rn(__fmul_rn(uA, rc.P1[8 + j]), rc.P1[j]);
            A[4 + j]  = (double)__fsub_rn(__fmul_rn(vA, rc.P1[8 + j]), rc.P1[4 + j]);
            A[8 + j]  = (double)__fsub_rn(__fmul_rn(uB, pk.P2[8 + j]), pk.P2[j]);
            A[12 + j] = (double)__fsub_rn(__fmul_rn(vB, pk.P2[8 + j]), pk.P2[4 + j]);
        }
        double v[4];
        GCLK_USE(__double2hiint(A[0])); GCLK_USE(__double2hiint(A[15])); GCLK(4);
        o.converged = null_vector4<ROBUST>(A, v);
        GCLK_USE(__double2hiint(v[0])); GCLK_USE(__double2hiint(v[3])); GCLK(5);
        // core/geometry.py:85-87: w = where(|Xh3| < 1e-12, 1e-12, Xh3); X = Xh / w
        float X0, X1, X2, X3;
        {
            const float w32 = (float)v[3];
            if (fabsf(w32) < 1e-12f) {
                X0 = __fdiv_rn((float)v[0], 1e-12f); X1 = __fdiv_rn((float)v[1], 1e-12f);
                X2 = __fdiv_rn((float)v[2], 1e-12f); X3 = __fdiv_rn(w32, 1e-12f);
            } else {
                const double iwv = rcp_newton(v[3]);
                X0 = (float)(v[0] * iwv); X1 = (float)(v[1] * iwv); X2 = (float)(v[2] * iwv); X3 = 1.0f;
            }
        }
        // ---- reprojection errors + cheirality: core/geometry.py:91-110, core/pipeline.py:735-737
        float z1, z2;
        float e1, e2;
        if constexpr (LENS) {       // a lens camera's error is measured against its observed (distorted) pixel
            e1 = (lt[0].model != LDP_LENS_PINHOLE) ? lens_reproj_err(lt[0], rc.P1, X0, X1, X2, X3, uA_obs, vA_obs, &z1)
                                                   : reproj_err(rc.P1, X0, X1, X2, X3, uA, vA, &z1);
            e2 = (lt[1 + k].model != LDP_LENS_PINHOLE) ? lens_reproj_err(lt[1 + k], pk.P2, X0, X1, X2, X3, uB_obs, vB_obs, &z2)
                                                       : reproj_err(pk.P2, X0, X1, X2, X3, uB, vB, &z2);
        } else {
            e1 = reproj_err(rc.P1, X0, X1, X2, X3, uA, vA, &z1);
            e2 = reproj_err(pk.P2, X0, X1, X2, X3, uB, vB, &z2);
        }
        const float err = (e1 != e1 || e2 != e2) ? __int_as_float(0x7fc00000) : fmaxf(e1, e2);   // np.maximum propagates NaN
        int keep;
        if (P.no_filter) {                                                        // core/pipeline.py:739-743
            keep = (isfinite(X0) && isfinite(X1) && isfinite(X2) && isfinite(X3) && isfinite(err)) ? 1 : 0;
        } else {                                                                  // core/pipeline.py:745-749
            keep = (err <= P.reproj_thresh && z1 > 0.0f && z2 > 0.0f) ? 1 : 0;
            if (keep && P.min_parallax_deg > 0.0f) {                              // core/geometry.py:113-119
                float a0 = __fsub_rn(X0, rc.C1[0]), a1 = __fsub_rn(X1, rc.C1[1]), a2 = __fsub_rn(X2, rc.C1[2]);
                float b0 = __fsub_rn(X0, pk.C2[0]), b1 = __fsub_rn(X1, pk.C2[1]), b2 = __fsub_rn(X2, pk.C2[2]);
                const float na = __fadd_rn(__fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(a0, a0), __fmul_rn(a1, a1)), __fmul_rn(a2, a2))), 1e-12f);
                const float nb = __fadd_rn(__fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(b0, b0), __fmul_rn(b1, b1)), __fmul_rn(b2, b2))), 1e-12f);
                a0 = __fdiv_rn(a0, na); a1 = __fdiv_rn(a1, na); a2 = __fdiv_rn(a2, na);
                b0 = __fdiv_rn(b0, nb); b1 = __fdiv_rn(b1, nb); b2 = __fdiv_rn(b2, nb);
                float d = __fadd_rn(__fadd_rn(__fmul_rn(a0, b0), __fmul_rn(a1, b1)), __fmul_rn(a2, b2));
                const bool dnan = (d != d);
                d = fminf(fmaxf(d, -1.0f), 1.0f);
                // degrees(arccos(d)) >= min_deg  <=>  d <= par_cos_max (arccos is monotone; threshold found on the host)
                keep = (!dnan && d <= ga.par_cos_max) ? 1 : 0;
            }
        }
        o.X0 = X0; o.X1 = X1; o.X2 = X2; o.err = err; o.z1 = z1; o.keep = keep;
        GCLK_USE(o.X0); GCLK_USE(o.err); GCLK_USE(o.keep); GCLK(6);
    }
    o.dcert = 0.f;
    o.dbg = make_float4(0.f, 0.f, 0.f, 0.f);
    if (P.collect_debug) {                                                        // core/pipeline.py:761-769
        const float denom = (P.sample_cap > 1e-6f) ? P.sample_cap : 1.0f;
        o.dcert = fminf(fmaxf(__fdiv_rn(craw, denom), 0.f), 1.f);
        o.dbg = make_float4(fminf(fmaxf(xA, 0.f), wm1), fminf(fmaxf(yA, 0.f), hm1),
                            fminf(fmaxf(xB, 0.f), wm1), fminf(fmaxf(yB, 0.f), hm1));
    }
}

__device__ __forceinline__ void store_sample(const ldp_params& P, const Workspace& ws, const ldp_outputs& out,
                                             size_t o, const SampleResult& s) {
    ws.pt0[o] = make_float4(s.X0, s.X1, s.X2, s.err);
    ws.pt1[o] = make_float4(s.cr, s.cg, s.cb, s.dcert);
    if (P.collect_debug) ws.dbgm[o] = s.dbg;
    const uint8_t f = (uint8_t)(s.keep | (s.good << 1) | (s.grp << 2));
    ws.flags[o] = f;
    if (out.sample_flags) out.sample_flags[o] = f;
    if (out.sample_xyzerr) reinterpret_cast<float4*>(out.sample_xyzerr)[o] = make_float4(s.X0, s.X1, s.X2, s.err);
}

// ---- multi-view refinement (ldp_params.multiview; the semantics are stated in include/ldp_b200.h).  Not in the reference.
// It runs for a KEPT sample only, after its two-view verdict: the candidates' certainty words and warp rows are gathered
// then, so a launch pays for them at the kept samples alone and the plain path's load chain is untouched.  The candidate
// set lives in a bit mask; a candidate's pixel is re-decoded (its 8-byte warp half reloaded, from L1) in each pass
// instead of being kept in registers.
constexpr int MV_FIX = 1 << 30;     // fix_list entry: only the multi-view solve of a kept sample is to be redone

struct MvPix { float u_obs, v_obs, u, v; };      // observed pixel, ideal pinhole pixel

// neighbour q's pixel at map pixel idx (the xB, yB half of its warp row), decoded like eval_sample decodes the winner's
template <bool LENS>
__device__ __forceinline__ MvPix mv_pixel(const ldp_params& P, const PairTable& pc, const ldp_lens* lt, int q, int idx) {
    const float2 w = __ldg(reinterpret_cast<const float2*>(pc.warp[q] + (size_t)idx * 4 + 2));
    const float xB = __fmul_rn(__fmul_rn(__fadd_rn(w.x, 1.0f), 0.5f), (float)(P.w_match - 1));
    const float yB = __fmul_rn(__fmul_rn(__fadd_rn(w.y, 1.0f), 0.5f), (float)(P.h_match - 1));
    MvPix b;
    b.u_obs = __fmul_rn(xB, pc.sxB[q]); b.v_obs = __fmul_rn(yB, pc.syB[q]);
    b.u = b.u_obs; b.v = b.v_obs;
    if constexpr (LENS) {
        if (lt[1 + q].model != LDP_LENS_PINHOLE) lens_undistort_px(lt[1 + q], b.u_obs, b.v_obs, b.u, b.v);
    }
    return b;
}

// the two DLT rows of camera Pm at ideal pixel (u, v), f32 like the two-view rows, into the Gram matrix
__device__ __forceinline__ void gram_add_view(Gram& g, const float* Pm, float u, float v) {
    double ru[4], rv[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        ru[j] = (double)__fsub_rn(__fmul_rn(u, Pm[8 + j]), Pm[j]);
        rv[j] = (double)__fsub_rn(__fmul_rn(v, Pm[8 + j]), Pm[4 + j]);
    }
    gram_add_row(g, ru[0], ru[1], ru[2], ru[3]);
    gram_add_row(g, rv[0], rv[1], rv[2], rv[3]);
}

// reprojection error of one view (lens-aware like eval_sample's) and its depth
template <bool LENS>
__device__ __forceinline__ float mv_view_err(const ldp_lens* L, const float* Pm, float X0, float X1, float X2, float X3,
                                             const MvPix& b, float* z) {
    if constexpr (LENS) {
        if (L->model != LDP_LENS_PINHOLE) return lens_reproj_err(*L, Pm, X0, X1, X2, X3, b.u_obs, b.v_obs, z);
    }
    return reproj_err(Pm, X0, X1, X2, X3, b.u, b.v, z);
}

// Refines the kept two-view point (X, err) of the sample at map pixel idx, winner k, winner warp row wv.  On return X / err
// hold the point to emit and mask its view mask.  ROBUST = false: returns false if a solve did not converge (nothing is
// changed; the fix-up repeats the refinement with ROBUST = true, which always converges).  z_ref: when not null, receives the
// reference camera's depth of an accepted refined point (left alone otherwise).
template <bool ROBUST, bool LENS>
__device__ bool mv_refine(const ldp_params& P, const RefConst& rc, const PairTable& pc, const ProView& pv, const GeomArgs& ga,
                          const ldp_lens* lt, int idx, int k, float4 wv, float& X0, float& X1, float& X2, float& err, int& mask,
                          float* z_ref = nullptr) {
    mask = 1 << k;
    const float wm1 = (float)(P.w_match - 1), hm1 = (float)(P.h_match - 1);
    MvPix a, bk;
    {
        const float xA = __fmul_rn(__fmul_rn(__fadd_rn(wv.x, 1.0f), 0.5f), wm1);
        const float yA = __fmul_rn(__fmul_rn(__fadd_rn(wv.y, 1.0f), 0.5f), hm1);
        const float xB = __fmul_rn(__fmul_rn(__fadd_rn(wv.z, 1.0f), 0.5f), wm1);
        const float yB = __fmul_rn(__fmul_rn(__fadd_rn(wv.w, 1.0f), 0.5f), hm1);
        a.u_obs = __fmul_rn(xA, rc.sxA); a.v_obs = __fmul_rn(yA, rc.syA);
        bk.u_obs = __fmul_rn(xB, pc.sxB[k]); bk.v_obs = __fmul_rn(yB, pc.syB[k]);
        a.u = a.u_obs; a.v = a.v_obs; bk.u = bk.u_obs; bk.v = bk.v_obs;
        if constexpr (LENS) {
            if (lt[0].model != LDP_LENS_PINHOLE) lens_undistort_px(lt[0], a.u_obs, a.v_obs, a.u, a.v);
            if (lt[1 + k].model != LDP_LENS_PINHOLE) lens_undistort_px(lt[1 + k], bk.u_obs, bk.v_obs, bk.u, bk.v);
        }
    }
    // ---- candidates: one slot per neighbour uid, not the winner's, confident, finite, through the Sampson gate
    const int gk = pc.group[k];
    unsigned cand = 0;
    Gram g = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    gram_add_view(g, rc.P1, a.u, a.v);
    gram_add_view(g, pc.P2[k], bk.u, bk.v);
    const Gram g2v = g;
    for (int q = 0; q < rc.nn; ++q) {
        if (pc.group[q] != q || q == gk) continue;             // (also excludes k: group[k] == k means q == gk)
        if (!(cert_at(P, pc, pv, q, idx) >= P.multiview_min_cert)) continue;
        const MvPix b = mv_pixel<LENS>(P, pc, lt, q, idx);
        if (!isfinite(b.u) || !isfinite(b.v)) continue;
        if (P.sampson_thresh > 0.0 && !sampson_pass(pc.F[q], a.u, a.v, b.u, b.v, P.sampson_thresh)) continue;
        cand |= 1u << q;
        gram_add_view(g, pc.P2[q], b.u, b.v);
    }
    if (!cand) return true;
    // ---- solve, trim once, solve again if something was dropped
    double v[4];
    if (!null_vector_gram<ROBUST>(g, v)) return false;
    float Y0, Y1, Y2, Y3;
    dehomogenise(v, Y0, Y1, Y2, Y3);
    const float thr = P.reproj_thresh;
    unsigned used = cand;
    g = g2v;
    for (unsigned m = cand; m; m &= m - 1) {
        const int q = __ffs(m) - 1;
        const MvPix b = mv_pixel<LENS>(P, pc, lt, q, idx);
        float z;
        const float e = mv_view_err<LENS>(lt + 1 + q, pc.P2[q], Y0, Y1, Y2, Y3, b, &z);
        if (!(e <= thr) || !(z > 0.0f)) used &= ~(1u << q);
        else gram_add_view(g, pc.P2[q], b.u, b.v);
    }
    if (!used) return true;                                    // nothing left beside the winner: the two-view point stands
    if (used != cand) {
        if (!null_vector_gram<ROBUST>(g, v)) return false;
        dehomogenise(v, Y0, Y1, Y2, Y3);
    }
    // ---- accept: every included view within the threshold and in front, the reference-winner parallax still met
    float zA, zB;
    const float eA = mv_view_err<LENS>(lt, rc.P1, Y0, Y1, Y2, Y3, a, &zA);
    const float eB = mv_view_err<LENS>(lt + 1 + k, pc.P2[k], Y0, Y1, Y2, Y3, bk, &zB);
    bool ok = eA <= thr && zA > 0.0f && eB <= thr && zB > 0.0f;
    float emax = fmaxf(eA, eB);
    for (unsigned m = used; m && ok; m &= m - 1) {
        const int q = __ffs(m) - 1;
        const MvPix b = mv_pixel<LENS>(P, pc, lt, q, idx);
        float z;
        const float e = mv_view_err<LENS>(lt + 1 + q, pc.P2[q], Y0, Y1, Y2, Y3, b, &z);
        ok = e <= thr && z > 0.0f;
        emax = fmaxf(emax, e);
    }
    if (ok && P.min_parallax_deg > 0.0f) ok = parallax_pass(Y0, Y1, Y2, rc.C1, pc.C2[k], ga.par_cos_max);
    if (ok) { X0 = Y0; X1 = Y1; X2 = Y2; err = emax; mask |= (int)used; if (z_ref) *z_ref = zA; }
    return true;
}

// The view's lens table (lens_a, lens_b[]), descriptor -> shared memory, staged like the camera constants: loads first, stores
// after the caller's other loads are in flight.  Only the LENS instantiations declare and stage it.
constexpr int LENS_WORDS = (int)(sizeof(ldp_lens) * (LDP_MAX_NN + 1) / 4);
constexpr int LENS_PER = (LENS_WORDS + K2_THREADS - 1) / K2_THREADS;
static_assert(offsetof(ldp_ref_desc, lens_b) == offsetof(ldp_ref_desc, lens_a) + sizeof(ldp_lens) && sizeof(ldp_lens) % 8 == 0,
              "lens table layout");
struct StagedLens { uint32_t v[LENS_PER]; };
__device__ __forceinline__ void lens_load(const ldp_ref_desc* rd, int t, StagedLens& sl) {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(&rd->lens_a);
#pragma unroll
    for (int q = 0; q < LENS_PER; ++q) sl.v[q] = (t + q * K2_THREADS < LENS_WORDS) ? __ldg(src + t + q * K2_THREADS) : 0u;
}
__device__ __forceinline__ void lens_store(const StagedLens& sl, ldp_lens* dst, int t) {
    uint32_t* d = reinterpret_cast<uint32_t*>(dst);
#pragma unroll
    for (int q = 0; q < LENS_PER; ++q) if (t + q * K2_THREADS < LENS_WORDS) d[t + q * K2_THREADS] = sl.v[q];
}

// K2b compute: gathers each sample's inputs, per-sample result (in place) + per-tile group statistics out.
// MV: multiview launch: a kept sample's point is refined from its other confident neighbours (mv_refine).
template <bool LENS, bool MV>
__global__ void __launch_bounds__(K2_THREADS, K2_MIN_BLOCKS)
ldp_geometry_kernel(const ldp_params P, const ldp_ref_desc* __restrict__ refs, const Workspace ws, const ldp_outputs out,
                    const GeomArgs ga)
{
    __shared__ RefConst rc;
    __shared__ PairTable pc;
    __shared__ int s_cnt[LDP_MAX_NN], s_first[LDP_MAX_NN];
    __shared__ ProView pv;
    const int r = blockIdx.y;
    GCLK_DECL
    // host-written descriptors, no kernel produces them: their loads are put in flight first and collected after the sample
    // indices are requested, one round trip for both; the prefetches are hints (the winner row was written three kernels ago)
    StagedDesc sd;
    stage_load(refs + r, threadIdx.x, K2_THREADS, sd);
    const ldp_lens* lt = nullptr;
    StagedLens sl;
    if constexpr (LENS) lens_load(refs + r, threadIdx.x, sl);
    if (ga.have_bestk && threadIdx.x == LDP_MAX_NN + 32)
        l2_prefetch_slice(ws.bestk + (size_t)r * ws.n_pad, (size_t)P.H * P.W, blockIdx.x, gridDim.x);
    if (P.prologue) stage_proview(refs + r, pv, threadIdx.x);
    GCLK(0);
    grid_dependency_sync();
    GCLK(10);
    const int i0 = blockIdx.x * K2_THREADS;
    const int32_t* sel = (out.sel_idx ? out.sel_idx : ws.sel) + (size_t)r * ws.sel_cap;
    const int i = i0 + threadIdx.x;
    const int idx_f = (i < (int)ws.sel_cap) ? __ldg(sel + i) : 0;
    const int S = out.n_samples[r];
    stage_store(sd, rc, pc, threadIdx.x, K2_THREADS, blockIdx.x, (int)gridDim.x);
    if constexpr (LENS) {
        __shared__ __align__(8) ldp_lens s_lens[LDP_MAX_NN + 1];
        lens_store(sl, s_lens, threadIdx.x);
        lt = s_lens;
    }
    if (ga.have_bestk) {                    // the draw kernel of this launch was the last reader of the view's p row
        const char* row = reinterpret_cast<const char*>(ws.w + (size_t)r * ws.n_pad);
        const int nlines = (int)(ws.n_pad * sizeof(float) / 128);
        for (int l = i0 + threadIdx.x; l < nlines; l += gridDim.x * K2_THREADS) l2_discard_line(row + (size_t)l * 128);
    }
    if (i0 >= S) return;
    int k_pre = 0;                          // needs no staged constant: requested before the barrier
    if (ga.have_bestk && i0 + (int)threadIdx.x < S) k_pre = ws.bestk[(size_t)r * ws.n_pad + idx_f];
    if (threadIdx.x < LDP_MAX_NN) { s_cnt[threadIdx.x] = 0; s_first[threadIdx.x] = 0x7fffffff; }
    __syncthreads();
    GCLK_USE(idx_f); GCLK(1);
    const int lane = threadIdx.x & 31;
    int keep = 0, grp = -1;
    if (i < S) {
        const size_t o = (size_t)r * ws.sel_cap + i;
        SampleRec rec;
        float craw;
        gather_sample(P, rc, pc, pv, ga, k_pre, idx_f, rec, craw);
        GCLK_USE(rec.tex[0]); GCLK_USE(rec.tex[2]); GCLK_USE(rec.wv.x); GCLK(2);
        SampleResult s;
        eval_sample<false, LENS>(P, rc, pc, ga, lt, rec, craw, s GCLK_PASS);
        if constexpr (MV) {
            if (ga.force_fix_two > 0 && i % ga.force_fix_two == 0) s.converged = false;
        }
        if (!s.converged) {                 // rare: store the record for the fix-up (flag bit 7), keep = 0 for now
            ws.pt0[o] = rec.wv;
            ws.pt1[o] = make_float4(__uint_as_float(rec.tex[0]), __uint_as_float(rec.tex[1]), __uint_as_float(rec.tex[2]),
                                    __uint_as_float(rec.k_cert));
            if (P.collect_debug) ws.dbgm[o].x = craw;
            const int slot = atomicAdd(ws.fix_count, 1);
            ws.fix_list[slot] = make_int2(r, i);
            ws.flags[o] = (uint8_t)(0x80 | (s.grp << 2));
            s.keep = 0;
        } else {
            store_sample(P, ws, out, o, s);
            if constexpr (MV) {
                if (s.keep) {               // the verdict is final; only the point moves
                    float X0 = s.X0, X1 = s.X1, X2 = s.X2, err = s.err;
                    int mask;
                    const int k = (int)(rec.k_cert & 0xffu);
                    const bool conv = mv_refine<false, LENS>(P, rc, pc, pv, ga, lt, idx_f, k, rec.wv, X0, X1, X2, err, mask);
                    if (conv && !(ga.force_fix_mv > 0 && i % ga.force_fix_mv == 0)) {
                        ws.pt0[o] = make_float4(X0, X1, X2, err);
                        ws.vmask[o] = mask;
                    } else {                // rare: the fix-up redoes the multi-view solve from the winner's warp row and slot
                        ws.mvrec[o] = rec.wv;           //   (vmask holds the slot until then); pt0 is the fallback
                        ws.vmask[o] = k;
                        const int slot = atomicAdd(ws.fix_count, 1);
                        ws.fix_list[slot] = make_int2(r, i | MV_FIX);
                    }
                }
            }
        }
        keep = s.keep;
        grp = s.grp;
        GCLK(7);
    }
    // per-tile group statistics for the pack kernels: kept count and first sample position per group
    const unsigned same = __match_any_sync(0xffffffffu, grp);
    const unsigned kept_all = __ballot_sync(0xffffffffu, keep);
    if (grp >= 0 && lane == (__ffs(same) - 1)) {
        atomicMin(&s_first[grp], i);                                   // lowest lane of the group has the lowest index
        const unsigned kept_same = same & kept_all;
        if (kept_same) atomicAdd(&s_cnt[grp], __popc(kept_same));
    }
    if (lane == 0 && kept_all) atomicAdd(&ws.kept[r], __popc(kept_all));
    GCLK(8);
    __syncthreads();
    GCLK(9);
    if (threadIdx.x < LDP_MAX_NN) {
        const size_t t = ((size_t)r * ga.nb2 + blockIdx.x) * LDP_MAX_NN + threadIdx.x;
        ws.blk_cnt[t] = s_cnt[threadIdx.x];
        ws.blk_first[t] = s_first[threadIdx.x];
    }
    GCLK_FLUSH;
}

// K2c fix-up + plan: one CTA per view.  (1) The view's entries of the worklist (null-vector iteration not converged: grossly
// inconsistent matches) are re-evaluated with the Jacobi solver, one thread each - usually there are none.  (2) The view's
// output plan, once for all of its pack CTAs: kept points per neighbour group, groups in order of first appearance
// (reference core/pipeline.py:685-695), and for every 128-sample tile and group the row (relative to the view's first row)
// at which that tile's kept samples of that group start.
template <bool LENS, bool MV>
__global__ void __launch_bounds__(K2_THREADS)
ldp_fix_kernel(const ldp_params P, const ldp_ref_desc* __restrict__ refs, const Workspace ws, const ldp_outputs out,
               const GeomArgs ga)
{
    __shared__ RefConst rc;
    __shared__ PairTable pc;
    __shared__ int s_tot[LDP_MAX_NN], s_first[LDP_MAX_NN], s_base[LDP_MAX_NN];
    constexpr int TB = 128;                                 // tiles staged per block step
    __shared__ int s_c[TB * LDP_MAX_NN], s_f[TB * LDP_MAX_NN];
    grid_dependency_sync();
    const int r = blockIdx.x, tid = threadIdx.x;
    const int n = *ws.fix_count;
    if (n > 0) {
        stage_constants(refs + r, rc, pc, tid, K2_THREADS);
        const ldp_lens* lt = nullptr;
        if constexpr (LENS) {
            __shared__ __align__(8) ldp_lens s_lens[LDP_MAX_NN + 1];
            StagedLens sl;
            lens_load(refs + r, tid, sl);
            lens_store(sl, s_lens, tid);
            lt = s_lens;
        }
        const ProView* pv = nullptr;
        if constexpr (MV) {
            __shared__ ProView s_pv;
            if (P.prologue) stage_proview(refs + r, s_pv, tid);
            pv = &s_pv;
        }
        __syncthreads();
        for (int e = tid; e < n; e += K2_THREADS) {
            const int2 it = ws.fix_list[e];
            if (it.x != r) continue;
            const int i = MV ? (it.y & ~MV_FIX) : it.y;
            const size_t o = (size_t)r * ws.sel_cap + i;
            int idx = 0;
            if constexpr (MV) idx = ((out.sel_idx ? out.sel_idx : ws.sel) + (size_t)r * ws.sel_cap)[i];
            if (MV && (it.y & MV_FIX)) {    // kept, two-view result final (pt0): redo the multi-view solve alone
                const float4 x = ws.pt0[o];
                float X0 = x.x, X1 = x.y, X2 = x.z, err = x.w;
                int mask;
                mv_refine<true, LENS>(P, rc, pc, *pv, ga, lt, idx, ws.vmask[o], ws.mvrec[o], X0, X1, X2, err, mask);
                ws.pt0[o] = make_float4(X0, X1, X2, err);
                ws.vmask[o] = mask;
                continue;
            }
            SampleRec rec;                  // the record the geometry kernel stored
            rec.wv = ws.pt0[o];
            const float4 b = ws.pt1[o];
            rec.tex[0] = __float_as_uint(b.x); rec.tex[1] = __float_as_uint(b.y); rec.tex[2] = __float_as_uint(b.z);
            rec.k_cert = __float_as_uint(b.w);
            const float craw = P.collect_debug ? ws.dbgm[o].x : 0.f;
            SampleResult s;
            GCLK_DECL
            eval_sample<true, LENS>(P, rc, pc, ga, lt, rec, craw, s GCLK_PASS);
            store_sample(P, ws, out, o, s);
            if constexpr (MV) {
                if (s.keep) {
                    float X0 = s.X0, X1 = s.X1, X2 = s.X2, err = s.err;
                    int mask;
                    mv_refine<true, LENS>(P, rc, pc, *pv, ga, lt, idx, (int)(rec.k_cert & 0xffu), rec.wv, X0, X1, X2, err, mask);
                    ws.pt0[o] = make_float4(X0, X1, X2, err);
                    ws.vmask[o] = mask;
                }
            }
            if (s.keep) {
                atomicAdd(&ws.kept[r], 1);
                atomicAdd(&ws.blk_cnt[((size_t)r * ga.nb2 + i / K2_THREADS) * LDP_MAX_NN + s.grp], 1);
            }
        }
        __syncthreads();
    }
    // ---- plan.  Thread (part, g) owns group g over one eighth of the view's tiles; the tile statistics are staged in shared
    //      memory by all threads (coalesced, every load in flight at once, requested together with the sample count that says
    //      how many of them mean something: the tables are nb2 tiles long, always readable).
    constexpr int NPART = K2_THREADS / LDP_MAX_NN;
    __shared__ int s_ptot[NPART][LDP_MAX_NN], s_pfirst[NPART][LDP_MAX_NN];
    int32_t* cnt = ws.blk_cnt + (size_t)r * ga.nb2 * LDP_MAX_NN;
    int32_t* fst = ws.blk_first + (size_t)r * ga.nb2 * LDP_MAX_NN;
    const int g = tid % LDP_MAX_NN, part = tid / LDP_MAX_NN;
    const int first_block = min(TB, ga.nb2) * LDP_MAX_NN;
    for (int e = tid; e < first_block; e += K2_THREADS) {
        s_c[e] = __ldcg(cnt + e);
        s_f[e] = __ldcg(fst + e);
    }
    const int S = __ldcg(out.n_samples + r);
    const int nb = (S + K2_THREADS - 1) / K2_THREADS;
    int tot = 0, first = 0x7fffffff;                       // thread g < LDP_MAX_NN: the whole view
    for (int t0 = 0; t0 < nb; t0 += TB) {
        const int ntile = min(TB, nb - t0);
        if (t0 > 0) {
            __syncthreads();
            for (int e = tid; e < ntile * LDP_MAX_NN; e += K2_THREADS) {
                s_c[e] = __ldcg(cnt + t0 * LDP_MAX_NN + e);
                s_f[e] = __ldcg(fst + t0 * LDP_MAX_NN + e);
            }
        }
        __syncthreads();
        const int per = (ntile + NPART - 1) / NPART, ta = min(part * per, ntile), tb = min(ta + per, ntile);
        int pt = 0, pf = 0x7fffffff;
        for (int t = ta; t < tb; ++t) { pt += s_c[t * LDP_MAX_NN + g]; pf = min(pf, s_f[t * LDP_MAX_NN + g]); }
        s_ptot[part][g] = pt;
        s_pfirst[part][g] = pf;
        __syncthreads();
        if (tid < LDP_MAX_NN)
#pragma unroll
            for (int q = 0; q < NPART; ++q) { tot += s_ptot[q][tid]; first = min(first, s_pfirst[q][tid]); }
    }
    if (tid < LDP_MAX_NN) { s_tot[tid] = tot; s_first[tid] = first; }
    __syncthreads();
    if (tid == 0) {
        int order[LDP_MAX_NN];
        int m = 0;
        for (int q = 0; q < LDP_MAX_NN; ++q) { s_base[q] = 0; if (s_first[q] != 0x7fffffff) order[m++] = q; }
        for (int a = 1; a < m; ++a) {                       // insertion sort by first appearance
            const int gg = order[a];
            int q = a - 1;
            while (q >= 0 && s_first[order[q]] > s_first[gg]) { order[q + 1] = order[q]; --q; }
            order[q + 1] = gg;
        }
        int acc = 0;
        for (int a = 0; a < m; ++a) { const int gg = order[a]; s_base[gg] = acc; acc += s_tot[gg]; }
        for (int a = 0; a < LDP_MAX_NN; ++a) {
            out.group_order[(size_t)r * LDP_MAX_NN + a] = (a < m) ? order[a] : -1;
            out.group_count[(size_t)r * LDP_MAX_NN + a] = s_tot[a];
        }
    }
    __syncthreads();
    // tile t, group g: rows of the group in earlier tiles (+ the group's base) -> blk_first
    int carried = s_base[g];                                // rows of group g before the block of tiles at hand
    for (int t0 = 0; t0 < nb; t0 += TB) {
        const int ntile = min(TB, nb - t0);
        if (nb > TB) {                                      // (a single block of tiles is still in shared memory from the first pass)
            __syncthreads();
            for (int e = tid; e < ntile * LDP_MAX_NN; e += K2_THREADS) s_c[e] = __ldcg(cnt + t0 * LDP_MAX_NN + e);
            __syncthreads();
            const int per0 = (ntile + NPART - 1) / NPART, a0 = min(part * per0, ntile), b0 = min(a0 + per0, ntile);
            int pt = 0;
            for (int t = a0; t < b0; ++t) pt += s_c[t * LDP_MAX_NN + g];
            s_ptot[part][g] = pt;
            __syncthreads();
        }
        const int per = (ntile + NPART - 1) / NPART, ta = min(part * per, ntile), tb = min(ta + per, ntile);
        int run = carried, block_tot = 0;
#pragma unroll
        for (int q = 0; q < NPART; ++q) { const int v = s_ptot[q][g]; run += (q < part) ? v : 0; block_tot += v; }
        for (int t = ta; t < tb; ++t) { const int c = s_c[t * LDP_MAX_NN + g]; fst[(t0 + t) * LDP_MAX_NN + g] = run; run += c; }
        carried += block_tot;
    }
}

// ---------------------------------------------------------------------------------------------
// K3 scatter: grid (tiles, views).  Output order of the reference (core/pipeline.py:685-695,753-780): neighbour groups in
// order of first appearance over the sample order, sample order inside a group, kept samples only.
// dst = view base (kept counts of earlier views) + [plan of ldp_fix_kernel: group base + earlier tiles of the group]
//       + rank inside the tile.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(K3_THREADS)
ldp_pack_kernel(const ldp_params P, const ldp_ref_desc* __restrict__ refs, const Workspace ws, const ldp_outputs out,
                const GeomArgs ga)
{
    static_assert(K3_THREADS == K2_THREADS && K3_THREADS % LDP_MAX_NN == 0, "one pack CTA per geometry tile");
    __shared__ int s_start[LDP_MAX_NN];
    __shared__ int s_wcnt[K3_THREADS / 32][LDP_MAX_NN];
    __shared__ long long s_red[K3_THREADS / 32];
    __shared__ long long s_off;
    grid_dependency_sync();
    const int r = blockIdx.y, b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // ---- everything the CTA needs is requested in ONE batch, before the sample count that decides what is used.  Rows are
    //      sel_cap long and the tile tables nb2 long, so every address is valid; what lies beyond the view's samples is ignored.
    const int i = b * K2_THREADS + tid;
    const bool in_row = i < (int)ws.sel_cap;
    const size_t o = (size_t)r * ws.sel_cap + i;
    const int S = __ldcg(out.n_samples + r);
    const int f_raw = in_row ? __ldcg(ws.flags + o) : 0;
    float4 pa = make_float4(0.f, 0.f, 0.f, 0.f), pc4 = pa, pd = pa;
    if (in_row) { pa = __ldcg(ws.pt0 + o); pc4 = __ldcg(ws.pt1 + o); }
    if (in_row && P.collect_debug && out.dbg_matches) pd = __ldcg(ws.dbgm + o);
    const bool mv_out = P.multiview && out.view_mask;
    int vm = 0;
    if (in_row && mv_out) vm = __ldcg(ws.vmask + o);
    int start_g = 0;
    if (tid < LDP_MAX_NN) start_g = __ldcg(ws.blk_first + ((size_t)r * ga.nb2 + b) * LDP_MAX_NN + tid);
    long long partk = 0;
    for (int q = tid; q < r; q += K3_THREADS) partk += (long long)__ldcg(ws.kept + q);
    const int kept_r = __ldcg(ws.kept + r);
    const int nb = (S + K2_THREADS - 1) / K2_THREADS;
    if (b >= nb && b != 0) return;
#pragma unroll
    for (int oo = 16; oo > 0; oo >>= 1) partk += __shfl_xor_sync(0xffffffffu, partk, oo);
    if (lane == 0) s_red[warp] = partk;
    if (tid < LDP_MAX_NN) s_start[tid] = start_g;
    const int f = (i < S) ? f_raw : 0;
    const int keep = f & 1, g = (f >> 2) & 0x1f;
    const unsigned same = __match_any_sync(0xffffffffu, keep ? g : -1);
    const int rank_in_warp = __popc(same & ((1u << lane) - 1u));
    if (lane < LDP_MAX_NN) s_wcnt[warp][lane] = 0;
    __syncwarp();
    if (keep && rank_in_warp == 0) s_wcnt[warp][g] = __popc(same);
    __syncthreads();
    if (tid == 0) {
        long long v = 0;
        for (int q = 0; q < K3_THREADS / 32; ++q) v += s_red[q];
        s_off = v;
        if (b == 0) {
            out.ref_offset[r] = v;
            if (r == (int)gridDim.y - 1) out.ref_offset[r + 1] = v + kept_r;
        }
    }
    __syncthreads();
    if (b >= nb) return;
    if (keep) {
        int before = s_start[g];
        for (int ww = 0; ww < warp; ++ww) before += s_wcnt[ww][g];
        const long long dst = s_off + before + rank_in_warp;
        if (dst < out.capacity) {
            out.xyz[dst * 3 + 0] = pa.x; out.xyz[dst * 3 + 1] = pa.y; out.xyz[dst * 3 + 2] = pa.z;
            out.rgb[dst * 3 + 0] = pc4.x; out.rgb[dst * 3 + 1] = pc4.y; out.rgb[dst * 3 + 2] = pc4.z;
            out.err[dst] = pa.w;
            if (mv_out) out.view_mask[dst] = vm;
            if (P.collect_debug && out.dbg_matches) {
                reinterpret_cast<float4*>(out.dbg_matches)[dst] = pd;
                if (out.dbg_cert) out.dbg_cert[dst] = pc4.w;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// The post-processing alone (core/pipeline.py:405-430): grid (pixel blocks, neighbours, views).
// ---------------------------------------------------------------------------------------------
constexpr int KP_THREADS = 256;
__global__ void __launch_bounds__(KP_THREADS)
ldp_prologue_kernel(const ldp_params P, const ldp_ref_desc* __restrict__ refs, float* __restrict__ outp,
                    size_t ref_stride, size_t plane_stride)
{
    grid_dependency_sync();
    __shared__ ProView pv;
    const int r = blockIdx.z, k = blockIdx.y;
    const ldp_ref_desc* rd = refs + r;
    if (k >= rd->nn) return;
    stage_proview(rd, pv, threadIdx.x);
    __syncthreads();
    const float* __restrict__ c = rd->cert[k];
    const int N = P.H * P.W;
    float* __restrict__ o = outp + (size_t)r * ref_stride + (size_t)k * plane_stride;
    for (int px = blockIdx.x * KP_THREADS + threadIdx.x; px < N; px += gridDim.x * KP_THREADS) {
        const int y = px / P.W;
        o[px] = prologue_cert(__ldcs(c + px), k, px, px - y * P.W, y, P, pv);
    }
}

// ldp_undistort_points: the geometry kernels' lens inversion on a list of pixels
constexpr int KU_THREADS = 256;
__global__ void __launch_bounds__(KU_THREADS)
ldp_undistort_kernel(const ldp_lens L, long long n, const float2* __restrict__ in, float2* __restrict__ out) {
    for (long long i = (long long)blockIdx.x * KU_THREADS + threadIdx.x; i < n; i += (long long)gridDim.x * KU_THREADS) {
        const float2 p = in[i];
        float2 q = p;
        if (L.model != LDP_LENS_PINHOLE) lens_undistort_px(L, p.x, p.y, q.x, q.y);
        out[i] = q;
    }
}

// ---------------------------------------------------------------------------------------------
// Depth maps (ldp_depth_maps; the rule is stated in include/ldp_b200.h).  Not in the reference.
// KD1: one thread per map pixel, grid (CTAs per view, views); a CTA strides over its view's map, so the camera constants are
//      staged once per CTA and not once per 128 pixels.  The arg-max reads the neighbours' certainty words and a candidate
//      the winner's 16-byte warp row, both coalesced over the map.  A candidate is evaluated by eval_sample (and mv_refine)
//      like a sampled pixel; its texels are not gathered (zero records: the colour eval_sample computes from them is dead
//      code here).  A solve that does not converge puts the pixel on its view's worklist instead of writing it.
// KD2: the fix-up.  Redoes every worklist entry with Jacobi (ROBUST = true) and writes it.
// ---------------------------------------------------------------------------------------------
struct DepthArgs {
    float* depth;                    // [R][N]
    float* err;                      // [R][N] or null
    float* xyz;                      // [R][N][3] or null
    uint8_t* flags;                  // [R][N] or null
    unsigned long long* kept;        // [R], zeroed by the host
    uint32_t* fix_list;              // [R][N] worklist, pixel | MV_FIX (one entry per pixel at most: it cannot overflow)
    int32_t* fix_count;              // [R], zeroed by the host
    float min_cert;                  // f32(min_certainty)
    int N;                           // H * W
};
constexpr int KDF_BLOCKS = 16;       // fix-up CTAs per view

// best post-processed certainty over the view's nn >= 1 neighbours at pixel idx and its slot: first index on ties, NaN wins
// (the stream kernel's arg-max, core/pipeline.py:634-635)
__device__ __forceinline__ float depth_argmax(const ldp_params& P, const PairTable& pc, const ProView& pv, int nn, int idx, int& k) {
    k = 0;
    float best = cert_at(P, pc, pv, 0, idx);
    for (int q = 1; q < nn; ++q) {
        const float c = cert_at(P, pc, pv, q, idx);
        if (c > best || c != c) { best = c; k = q; }
    }
    return best;
}

__device__ __forceinline__ void depth_store(const DepthArgs& d, size_t o, int flags, float z, float err, float X0, float X1, float X2) {
    d.depth[o] = z;
    if (d.err) d.err[o] = err;
    if (d.xyz) { d.xyz[3 * o] = X0; d.xyz[3 * o + 1] = X1; d.xyz[3 * o + 2] = X2; }
    if (d.flags) d.flags[o] = (uint8_t)flags;
}

__device__ __forceinline__ void depth_push(const DepthArgs& d, int r, uint32_t entry) {
    const int slot = atomicAdd(d.fix_count + r, 1);
    d.fix_list[(size_t)r * d.N + slot] = entry;
}

__device__ __forceinline__ void depth_count_kept(const DepthArgs& d, int r, unsigned kept) {
    kept = __reduce_add_sync(0xffffffffu, kept);
    if ((threadIdx.x & 31) == 0 && kept) atomicAdd(d.kept + r, (unsigned long long)kept);
}

// the view's constants (and lens table, post-processing view) in shared memory
template <bool LENS>
__device__ __forceinline__ const ldp_lens* depth_stage(const ldp_params& P, const ldp_ref_desc* rd, RefConst& rc, PairTable& pc,
                                                       ProView& pv, ldp_lens* s_lens) {
    stage_constants(rd, rc, pc, threadIdx.x, K2_THREADS);
    if (P.prologue) stage_proview(rd, pv, threadIdx.x);
    if constexpr (LENS) {
        StagedLens sl;
        lens_load(rd, threadIdx.x, sl);
        lens_store(sl, s_lens, threadIdx.x);
        return s_lens;
    }
    return nullptr;
}

__device__ __forceinline__ SampleRec depth_record(const PairTable& pc, int k, int idx) {
    SampleRec rec;
    rec.wv = __ldg(reinterpret_cast<const float4*>(pc.warp[k]) + idx);
    rec.tex[0] = rec.tex[1] = rec.tex[2] = 0u;
    rec.k_cert = (uint32_t)k;
    return rec;
}

template <bool LENS, bool MV>
__global__ void __launch_bounds__(K2_THREADS, K2_MIN_BLOCKS)
ldp_depth_kernel(const ldp_params P, const ldp_ref_desc* __restrict__ refs, const GeomArgs ga, const DepthArgs d)
{
    __shared__ RefConst rc;
    __shared__ PairTable pc;
    __shared__ ProView pv;
    __shared__ __align__(8) ldp_lens s_lens[LENS ? LDP_MAX_NN + 1 : 1];
    const int r = blockIdx.y;
    grid_dependency_sync();
    const ldp_lens* lt = depth_stage<LENS>(P, refs + r, rc, pc, pv, s_lens);
    __syncthreads();
    const int nn = rc.nn, N = d.N;
    const float nan = __int_as_float(0x7fc00000);
    unsigned kept = 0;
    for (int base = blockIdx.x * K2_THREADS; base < N; base += gridDim.x * K2_THREADS) {
        const int idx = base + threadIdx.x;
        if (idx >= N) break;
        int k = 0;
        const float c = (nn > 0) ? depth_argmax(P, pc, pv, nn, idx, k) : nan;
        const int cand = (c >= d.min_cert) ? 1 : 0;
        int f = cand | (k << 4);
        float z = nan, err = nan, X0 = nan, X1 = nan, X2 = nan;
        if (cand) {
            const SampleRec rec = depth_record(pc, k, idx);
            SampleResult s;
            GCLK_DECL
            eval_sample<false, LENS>(P, rc, pc, ga, lt, rec, 0.f, s GCLK_PASS);
            if (!s.converged || (ga.force_fix_two > 0 && idx % ga.force_fix_two == 0)) {
                depth_push(d, r, (uint32_t)idx);
                continue;
            }
            f |= (s.good << 1) | (s.keep << 2);
            err = s.err;
            if (s.keep) { X0 = s.X0; X1 = s.X1; X2 = s.X2; z = s.z1; }
            if constexpr (MV) {
                if (s.keep) {
                    int mask;
                    if (!mv_refine<false, LENS>(P, rc, pc, pv, ga, lt, idx, k, rec.wv, X0, X1, X2, err, mask, &z) ||
                        (ga.force_fix_mv > 0 && idx % ga.force_fix_mv == 0)) {
                        depth_push(d, r, (uint32_t)idx | MV_FIX);
                        continue;
                    }
                }
            }
            kept += s.keep;
        }
        depth_store(d, (size_t)r * N + idx, f, z, err, X0, X1, X2);
    }
    depth_count_kept(d, r, kept);
}

template <bool LENS, bool MV>
__global__ void __launch_bounds__(K2_THREADS)
ldp_depth_fix_kernel(const ldp_params P, const ldp_ref_desc* __restrict__ refs, const GeomArgs ga, const DepthArgs d)
{
    __shared__ RefConst rc;
    __shared__ PairTable pc;
    __shared__ ProView pv;
    __shared__ __align__(8) ldp_lens s_lens[LENS ? LDP_MAX_NN + 1 : 1];
    const int r = blockIdx.y;
    grid_dependency_sync();
    const int n = d.fix_count[r];
    if ((int)blockIdx.x * K2_THREADS >= n) return;
    const ldp_lens* lt = depth_stage<LENS>(P, refs + r, rc, pc, pv, s_lens);
    __syncthreads();
    const float nan = __int_as_float(0x7fc00000);
    unsigned kept = 0;
    for (int base = blockIdx.x * K2_THREADS; base < n; base += gridDim.x * K2_THREADS) {
        const int e = base + threadIdx.x;
        if (e < n) {
            const uint32_t it = d.fix_list[(size_t)r * d.N + e];
            const int idx = (int)(it & ~(uint32_t)MV_FIX);
            int k;
            depth_argmax(P, pc, pv, rc.nn, idx, k);
            const SampleRec rec = depth_record(pc, k, idx);
            SampleResult s;
            GCLK_DECL
            if (MV && (it & MV_FIX)) eval_sample<false, LENS>(P, rc, pc, ga, lt, rec, 0.f, s GCLK_PASS);   // converged: as before
            else eval_sample<true, LENS>(P, rc, pc, ga, lt, rec, 0.f, s GCLK_PASS);
            float z = nan, err = s.err, X0 = nan, X1 = nan, X2 = nan;
            if (s.keep) { X0 = s.X0; X1 = s.X1; X2 = s.X2; z = s.z1; }
            if constexpr (MV) {
                if (s.keep) {
                    int mask;
                    mv_refine<true, LENS>(P, rc, pc, pv, ga, lt, idx, k, rec.wv, X0, X1, X2, err, mask, &z);
                }
            }
            depth_store(d, (size_t)r * d.N + idx, 1 | (s.good << 1) | (s.keep << 2) | (k << 4), z, err, X0, X1, X2);
            kept += s.keep;
        }
    }
    depth_count_kept(d, r, kept);
}

}  // namespace ldp
