// Cross-view depth consistency (ldp_depth_consistency; the rule is stated in include/ldp_b200.h, the structure in
// DESIGN.md §4.9).  Not in the reference.  Included by ldp_api.cu (unity build), after ldp_geometry.cu (lens_distort) and
// ldp_outlier.cu (the compaction's ldp_outlier_kept_kernel).
//
// KC1 ldp_consistency_check_kernel<OWNER>: status bit 1 for a coordinate that is not finite, bit 2 for an owner outside [-1, V).
// KC2 ldp_consistency_kernel<LENS>: one thread per point, grid-stride.  The view constants (map pointer, P, the two map
//     scales, and with LENS the lens) are staged in shared memory a chunk of views at a time; every thread of the CTA tests
//     its point against the staged views, so the reads of the constants are broadcasts.  A table that fits one chunk is
//     staged once per CTA.  The two counters stay in registers; the map read goes through the read-only path (the cloud
//     comes in emission order, so neighbouring threads read neighbouring pixels of a view).  Writes the counters and the
//     keep flag that the outlier filter's scan and ldp_outlier_kept_kernel compact into kept_idx.
#include "ldp_device.cuh"

namespace ldp {

constexpr int CS_THREADS = 256;
constexpr int CS_CHUNK_PINHOLE = 128;    // views staged at once: 72 B each (map pointer, P, scales)
constexpr int CS_CHUNK_LENS = 64;        // 160 B each (+ ldp_lens)

struct ConsistencyArgs {
    const float* xyz;                    // [n,3]
    const int* owner;                    // [n] or NULL
    const float* const* depth;           // [V] device pointers to [H*W] f32 maps
    const float* P;                      // [V,12]
    const double* scales;                // [V,2] (ax, ay)
    const ldp_lens* lens;                // [V] (LENS only)
    int* n_consistent;                   // [n] or NULL
    int* n_violations;                   // [n] or NULL
    int* flag;                           // [n] keep flag for the compaction
    int* status;                         // [2] bit mask, kept count (the scan's total)
    long long n;
    double rel_tol;
    int V, H, W;
    int min_views, max_violations;
};

// OWNER: an owner array is given (its range is checked)
template <bool OWNER>
__global__ void __launch_bounds__(CS_THREADS)
ldp_consistency_check_kernel(const float* __restrict__ xyz, const int* __restrict__ owner, long long n, int V, int* __restrict__ status)
{
    grid_dependency_sync();
    const long long i = (long long)blockIdx.x * CS_THREADS + threadIdx.x;
    int bad = 0;
    if (i < n) {
        const float x = xyz[3 * i], y = xyz[3 * i + 1], z = xyz[3 * i + 2];
        if (!(isfinite(x) && isfinite(y) && isfinite(z))) bad |= 1;
        if constexpr (OWNER) { const int o = owner[i]; if (o < -1 || o >= V) bad |= 2; }
    }
    bad = __reduce_or_sync(0xffffffffu, bad);
    if ((threadIdx.x & 31) == 0 && bad) atomicOr(status, bad);
}

// q = ((P[0] X + P[1] Y) + P[2] Z) + P[3] in f64 without contraction: every product of two f32 values is exact
__device__ __forceinline__ double cons_row(const float* p, double X, double Y, double Z) {
    return __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn((double)p[0], X), __dmul_rn((double)p[1], Y)), __dmul_rn((double)p[2], Z)),
                     (double)p[3]);
}

// Steps 1-3 of the rule for one point (X, Y, Z) and one view (its P rows p, map scales s, map D, lens L): ++nc where the view
// supports the point, ++nv where it looks through it; returns true iff it supports it, and then pix is the map pixel.
// Shared by ldp_consistency_kernel and the fusion kernels (ldp_fusion.cu), so both apply one test.
template <bool LENS>
__device__ __forceinline__ bool cons_test(const float* p, const double* s, const float* D, const ldp_lens& L, double X, double Y,
                                          double Z, int W, int H, double rel_tol, int& nc, int& nv, size_t& pix) {
    const double z = cons_row(p + 8, X, Y, Z);
    if (!(z > 0.0)) return false;
    double u = __ddiv_rn(cons_row(p, X, Y, Z), z), v = __ddiv_rn(cons_row(p + 4, X, Y, Z), z);
    if constexpr (LENS) {
        if (L.model != LDP_LENS_PINHOLE) {
            const double fx = L.fx, fy = L.fy, cx = L.cx, cy = L.cy;
            double xd, yd;
            lens_distort(L, (u - cx) / fx, (v - cy) / fy, xd, yd);
            u = fx * xd + cx; v = fy * yd + cy;
        }
    }
    const double fxm = floor(__dmul_rn(u, s[0])), fym = floor(__dmul_rn(v, s[1]));
    if (!(fxm >= 0.0 && fxm < (double)W && fym >= 0.0 && fym < (double)H)) return false;
    pix = (size_t)fym * (size_t)W + (size_t)fxm;
    const double Dp = (double)__ldg(D + pix);
    if (!(Dp > 0.0)) return false;               // NaN (no depth) or not in front: no evidence
    const double d = __dsub_rn(z, Dp), t = __dmul_rn(rel_tol, Dp);
    if (fabs(d) <= t) { ++nc; return true; }
    if (d < -t) ++nv;
    return false;
}

template <bool LENS>
__global__ void __launch_bounds__(CS_THREADS)
ldp_consistency_kernel(const ConsistencyArgs a)
{
    constexpr int CHUNK = LENS ? CS_CHUNK_LENS : CS_CHUNK_PINHOLE;
    __shared__ float s_P[CHUNK][12];
    __shared__ double s_S[CHUNK][2];
    __shared__ const float* s_D[CHUNK];
    __shared__ __align__(8) ldp_lens s_L[LENS ? CHUNK : 1];
    grid_dependency_sync();
    const bool bad = (*(volatile const int*)a.status & 1) != 0;     // written by the check kernel before this one
    const int W = a.W, H = a.H, V = a.V;
    int staged = -1;                                   // first view of the chunk in shared memory (uniform over the CTA)
    for (long long base = (long long)blockIdx.x * CS_THREADS; base < a.n; base += (long long)gridDim.x * CS_THREADS) {
        const long long i = base + threadIdx.x;
        const bool live = i < a.n;
        if (bad) {                                     // a coordinate is not finite: nothing is kept, nothing else written
            if (live) a.flag[i] = 0;
            continue;
        }
        double X = 0.0, Y = 0.0, Z = 0.0;
        int own = -1;
        if (live) {
            X = (double)a.xyz[3 * i]; Y = (double)a.xyz[3 * i + 1]; Z = (double)a.xyz[3 * i + 2];
            if (a.owner) own = a.owner[i];
        }
        int nc = 0, nv = 0;
        for (int c0 = 0; c0 < V; c0 += CHUNK) {
            const int cn = min(CHUNK, V - c0);
            if (staged != c0) {
                __syncthreads();
                for (int t = threadIdx.x; t < cn * 12; t += CS_THREADS) s_P[t / 12][t % 12] = a.P[(size_t)c0 * 12 + t];
                for (int t = threadIdx.x; t < cn * 2; t += CS_THREADS) s_S[t / 2][t % 2] = a.scales[(size_t)c0 * 2 + t];
                for (int t = threadIdx.x; t < cn; t += CS_THREADS) s_D[t] = a.depth[c0 + t];
                if constexpr (LENS) {
                    constexpr int WORDS = (int)(sizeof(ldp_lens) / 8);
                    const unsigned long long* src = reinterpret_cast<const unsigned long long*>(a.lens + c0);
                    unsigned long long* dst = reinterpret_cast<unsigned long long*>(s_L);
                    for (int t = threadIdx.x; t < cn * WORDS; t += CS_THREADS) dst[t] = src[t];
                }
                __syncthreads();
                staged = c0;
            }
            if (!live) continue;
            for (int j = 0; j < cn; ++j) {
                if (c0 + j == own) continue;           // a point is never checked against the view it came from
                size_t pix;
                cons_test<LENS>(s_P[j], s_S[j], s_D[j], s_L[LENS ? j : 0], X, Y, Z, W, H, a.rel_tol, nc, nv, pix);
            }
        }
        if (live) {
            if (a.n_consistent) a.n_consistent[i] = nc;
            if (a.n_violations) a.n_violations[i] = nv;
            a.flag[i] = (nc >= a.min_views && nv <= a.max_violations) ? 1 : 0;
        }
    }
}

}  // namespace ldp
