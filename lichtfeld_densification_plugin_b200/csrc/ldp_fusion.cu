// Depth-map fusion (ldp_depth_colors, ldp_fuse_depth_maps; the rules are stated in include/ldp_b200.h, the structure in
// DESIGN.md §4.10).  Not in the reference.  Included by ldp_api.cu (unity build), after ldp_geometry.cu (the colour blend) and
// ldp_consistency.cu (the per-view test, cons_test).
//
// KF0 ldp_depth_color_kernel: the colour maps.  One thread per map pixel, grid (CTAs per view, views) like ldp_depth_kernel;
//     a kept pixel decodes its winner's warp row, gathers the four texels and blends them with bilinear_rgb, as eval_sample
//     does for a sampled pixel.
// KF1 ldp_fusion_check_kernel: status bit 2 for a view whose depth, xyz, rgb or err pointer is NULL.
// KF2 ldp_fusion_verdict_kernel<LENS> (pass 1): one thread per map pixel of every view, grid-stride; a pixel with a finite
//     depth is tested against every other view with cons_test and gets its consistent count and keep flag.  The view
//     constants are staged in shared memory a chunk at a time, as ldp_consistency_kernel stages them.
// KF3 ldp_fusion_emit_kernel<LENS> (pass 2, views below the pixel's own): a kept pixel is emitted unless a lower view holds a
//     kept pixel that agrees with it; the walk stops at the first one, and a CTA stops staging chunks once none of its
//     threads needs them.  The emit flags are compacted by the outlier filter's scan and ldp_outlier_kept_kernel into the
//     ascending source list.
// KF4 ldp_fusion_sum_kernel<LENS> (pass 2, views above): one thread per emitted point, reading the source list; it adds the
//     members' xyz and rgb in ascending view order and writes the fused point at its rank.
#include "ldp_device.cuh"

namespace ldp {

struct FusionArgs {
    const float* const* depth;           // [V] device pointers to [N] f32 maps
    const float* const* xyz;             // [V] -> [N,3]
    const float* const* rgb;             // [V] -> [N,3]
    const float* const* err;             // [V] -> [N]
    const float* P;                      // [V,12]
    const double* scales;                // [V,2] (ax, ay)
    const ldp_lens* lens;                // [V] (LENS only)
    uint8_t* kept;                       // [V*N] pass 1's keep flag
    int* n_cons;                         // [V*N] pass 1's consistent count
    int* flag;                           // [V*N] emit flag for the compaction
    const long long* source;             // [m] the emitted pixels, ascending
    float* xyz_out;                      // [m,3]
    float* rgb_out;                      // [m,3]
    float* err_out;                      // [m]
    int* n_views_out;                    // [m]
    int* n_consistent_out;               // [m]
    int* status;                         // [2] bit mask, emitted count (the scan's total)
    long long total;                     // V * N
    double rel_tol;
    int V, H, W, N;
    int min_views, max_violations;
};

// one chunk of views in shared memory
template <bool LENS>
struct FuseViews {
    static constexpr int CHUNK = LENS ? CS_CHUNK_LENS : CS_CHUNK_PINHOLE;
    double S[CHUNK][2];
    ldp_lens L[LENS ? CHUNK : 1];
    float P[CHUNK][12];
    const float* D[CHUNK];
    const float* X[CHUNK];
    const float* C[CHUNK];
};

// stages views [c0, c0 + cn); every thread of the CTA calls it
template <bool LENS, bool MEMBERS>
__device__ __forceinline__ void fuse_stage(const FusionArgs& a, FuseViews<LENS>& sv, int c0, int cn) {
    __syncthreads();
    for (int t = threadIdx.x; t < cn * 12; t += CS_THREADS) sv.P[t / 12][t % 12] = a.P[(size_t)c0 * 12 + t];
    for (int t = threadIdx.x; t < cn * 2; t += CS_THREADS) sv.S[t / 2][t % 2] = a.scales[(size_t)c0 * 2 + t];
    for (int t = threadIdx.x; t < cn; t += CS_THREADS) {
        sv.D[t] = a.depth[c0 + t];
        if constexpr (MEMBERS) { sv.X[t] = a.xyz[c0 + t]; sv.C[t] = a.rgb[c0 + t]; }
    }
    if constexpr (LENS) {
        constexpr int WORDS = (int)(sizeof(ldp_lens) / 8);
        const unsigned long long* src = reinterpret_cast<const unsigned long long*>(a.lens + c0);
        unsigned long long* dst = reinterpret_cast<unsigned long long*>(sv.L);
        for (int t = threadIdx.x; t < cn * WORDS; t += CS_THREADS) dst[t] = src[t];
    }
    __syncthreads();
}

__global__ void __launch_bounds__(K2_THREADS)
ldp_depth_color_kernel(const ldp_params P, const ldp_ref_desc* __restrict__ refs, const uint8_t* __restrict__ flags,
                       float* __restrict__ rgb, int N)
{
    __shared__ RefConst rc;
    __shared__ PairTable pc;
    const int r = blockIdx.y;
    grid_dependency_sync();
    stage_constants(refs + r, rc, pc, threadIdx.x, K2_THREADS);
    __syncthreads();
    const float nan = __int_as_float(0x7fc00000);
    const float wm1 = (float)(P.w_match - 1), hm1 = (float)(P.h_match - 1);
    const int iw = rc.img_w, ih = rc.img_h;
    const size_t img_bytes = (size_t)iw * ih * 3;
    for (int base = blockIdx.x * K2_THREADS; base < N; base += gridDim.x * K2_THREADS) {
        const int idx = base + threadIdx.x;
        if (idx >= N) break;
        const size_t o = (size_t)r * N + idx;
        const int f = flags[o], k = f >> 4;
        float col[3] = {nan, nan, nan};
        if ((f & 4) && k < rc.nn) {             // kept; its winner's warp row, decoded as eval_sample decodes it
            const float4 wv = __ldg(reinterpret_cast<const float4*>(pc.warp[k]) + idx);
            const float xA = __fmul_rn(__fmul_rn(__fadd_rn(wv.x, 1.0f), 0.5f), wm1);
            const float yA = __fmul_rn(__fmul_rn(__fadd_rn(wv.y, 1.0f), 0.5f), hm1);
            const float fx = __fmul_rn(xA, rc.sx_img), fy = __fmul_rn(yA, rc.sy_img);
            const int x0 = min(max((int)fminf(fmaxf(floorf(fx), -1.f), (float)iw), 0), iw - 1);
            const int y0 = min(max((int)fminf(fmaxf(floorf(fy), -1.f), (float)ih), 0), ih - 1);
            const int x1 = min(x0 + 1, iw - 1), y1 = min(y0 + 1, ih - 1);
            float t00[3], t01[3], t10[3], t11[3];
            fetch_texel_pair(rc.image, ((size_t)y0 * iw + x0) * 3, img_bytes, x1 != x0, t00, t01);
            fetch_texel_pair(rc.image, ((size_t)y1 * iw + x0) * 3, img_bytes, x1 != x0, t10, t11);
            bilinear_rgb(fx, fy, x0, y0, x1, y1, t00, t01, t10, t11, col);
        }
        rgb[3 * o] = col[0]; rgb[3 * o + 1] = col[1]; rgb[3 * o + 2] = col[2];
    }
}

__global__ void __launch_bounds__(CS_THREADS)
ldp_fusion_check_kernel(const FusionArgs a)
{
    grid_dependency_sync();
    const int v = blockIdx.x * CS_THREADS + threadIdx.x;
    int bad = 0;
    if (v < a.V && !(a.depth[v] && a.xyz[v] && a.rgb[v] && a.err[v])) bad = 2;
    bad = __reduce_or_sync(0xffffffffu, bad);
    if ((threadIdx.x & 31) == 0 && bad) atomicOr(a.status, bad);
}

template <bool LENS>
__global__ void __launch_bounds__(CS_THREADS)
ldp_fusion_verdict_kernel(const FusionArgs a)
{
    constexpr int CHUNK = FuseViews<LENS>::CHUNK;
    __shared__ __align__(16) FuseViews<LENS> sv;
    grid_dependency_sync();
    if (*(volatile const int*)a.status & 2) return;     // written by the check kernel: a view table cannot be read
    const int V = a.V, N = a.N;
    int staged = -1;
    for (long long base = (long long)blockIdx.x * CS_THREADS; base < a.total; base += (long long)gridDim.x * CS_THREADS) {
        const long long s = base + threadIdx.x;
        const bool live = s < a.total;
        int r = -1;
        bool pt = false;
        double X = 0.0, Y = 0.0, Z = 0.0;
        if (live) {
            r = (int)(s / N);
            const int i = (int)(s - (long long)r * N);
            if (isfinite(__ldg(a.depth[r] + i))) {
                const float* xp = a.xyz[r] + 3 * (size_t)i;
                const float x = __ldg(xp), y = __ldg(xp + 1), z = __ldg(xp + 2);
                if (isfinite(x) && isfinite(y) && isfinite(z)) { pt = true; X = x; Y = y; Z = z; }
                else atomicOr(a.status, 1);
            }
        }
        int nc = 0, nv = 0;
        for (int c0 = 0; c0 < V; c0 += CHUNK) {
            const int cn = min(CHUNK, V - c0);
            if (staged != c0) { fuse_stage<LENS, false>(a, sv, c0, cn); staged = c0; }
            if (!pt) continue;
            for (int j = 0; j < cn; ++j) {
                if (c0 + j == r) continue;             // a pixel is never tested against its own view
                size_t pix;
                cons_test<LENS>(sv.P[j], sv.S[j], sv.D[j], sv.L[LENS ? j : 0], X, Y, Z, a.W, a.H, a.rel_tol, nc, nv, pix);
            }
        }
        if (live) {
            a.n_cons[s] = nc;
            a.kept[s] = (pt && nc >= a.min_views && nv <= a.max_violations) ? 1 : 0;
        }
    }
}

template <bool LENS>
__global__ void __launch_bounds__(CS_THREADS)
ldp_fusion_emit_kernel(const FusionArgs a)
{
    constexpr int CHUNK = FuseViews<LENS>::CHUNK;
    __shared__ __align__(16) FuseViews<LENS> sv;
    grid_dependency_sync();
    const bool bad = *(volatile const int*)a.status != 0;    // bit 1 from pass 1, bit 2 from the check kernel: emit nothing
    const int V = a.V, N = a.N;
    int staged = -1;
    for (long long base = (long long)blockIdx.x * CS_THREADS; base < a.total; base += (long long)gridDim.x * CS_THREADS) {
        const long long s = base + threadIdx.x;
        const bool live = s < a.total;
        int r = 0;
        bool need = false;
        double X = 0.0, Y = 0.0, Z = 0.0;
        if (live && !bad) {
            r = (int)(s / N);
            need = a.kept[s] != 0;
            if (need) {
                const float* xp = a.xyz[r] + 3 * (size_t)(s - (long long)r * N);
                X = __ldg(xp); Y = __ldg(xp + 1); Z = __ldg(xp + 2);
            }
        }
        for (int c0 = 0; c0 < V; c0 += CHUNK) {
            const bool want = need && c0 < r;          // a lower view may still hold a member
            if (!__syncthreads_or(want)) break;
            const int cn = min(CHUNK, V - c0);
            if (staged != c0) { fuse_stage<LENS, false>(a, sv, c0, cn); staged = c0; }
            if (!want) continue;
            const int jn = min(cn, r - c0);
            for (int j = 0; j < jn; ++j) {
                size_t pix;
                int nc = 0, nv = 0;                    // unused: only the verdict and the pixel matter here
                if (cons_test<LENS>(sv.P[j], sv.S[j], sv.D[j], sv.L[LENS ? j : 0], X, Y, Z, a.W, a.H, a.rel_tol, nc, nv, pix) && a.kept[(size_t)(c0 + j) * N + pix]) { need = false; break; }     // the lower view emits the point
            }
        }
        if (live) a.flag[s] = need ? 1 : 0;
    }
}

template <bool LENS>
__global__ void __launch_bounds__(CS_THREADS)
ldp_fusion_sum_kernel(const FusionArgs a)
{
    constexpr int CHUNK = FuseViews<LENS>::CHUNK;
    __shared__ __align__(16) FuseViews<LENS> sv;
    grid_dependency_sync();
    const long long m = *(volatile const int*)(a.status + 1);  // the emitted count, written by the scan
    const int V = a.V, N = a.N;
    int staged = -1;
    for (long long base = (long long)blockIdx.x * CS_THREADS; base < m; base += (long long)gridDim.x * CS_THREADS) {
        const long long k = base + threadIdx.x;
        const bool live = k < m;
        int r = V, i = 0, cnt = 0;
        long long s = 0;
        float x = 0.f, y = 0.f, z = 0.f;
        double sx = 0.0, sy = 0.0, sz = 0.0, sr = 0.0, sg = 0.0, sb = 0.0;
        if (live) {
            s = a.source[k];
            r = (int)(s / N);
            i = (int)(s - (long long)r * N);
            const float* xp = a.xyz[r] + 3 * (size_t)i;
            const float* cp = a.rgb[r] + 3 * (size_t)i;
            x = __ldg(xp); y = __ldg(xp + 1); z = __ldg(xp + 2);
            sx = x; sy = y; sz = z;
            sr = __ldg(cp); sg = __ldg(cp + 1); sb = __ldg(cp + 2);
        }
        const double X = x, Y = y, Z = z;
        for (int c0 = 0; c0 < V; c0 += CHUNK) {
            const int cn = min(CHUNK, V - c0);
            const bool want = live && c0 + cn > r + 1;     // the chunk holds views above the point's own
            if (!__syncthreads_or(want)) continue;
            if (staged != c0) { fuse_stage<LENS, true>(a, sv, c0, cn); staged = c0; }
            if (!want) continue;
            for (int j = max(0, r + 1 - c0); j < cn; ++j) {
                size_t pix;
                int nc = 0, nv = 0;                    // unused: only the verdict and the pixel matter here
                if (cons_test<LENS>(sv.P[j], sv.S[j], sv.D[j], sv.L[LENS ? j : 0], X, Y, Z, a.W, a.H, a.rel_tol, nc, nv, pix) && a.kept[(size_t)(c0 + j) * N + pix]) {
                    const float* mp = sv.X[j] + 3 * pix;
                    const float* mc = sv.C[j] + 3 * pix;
                    sx = __dadd_rn(sx, (double)__ldg(mp)); sy = __dadd_rn(sy, (double)__ldg(mp + 1)); sz = __dadd_rn(sz, (double)__ldg(mp + 2));
                    sr = __dadd_rn(sr, (double)__ldg(mc)); sg = __dadd_rn(sg, (double)__ldg(mc + 1)); sb = __dadd_rn(sb, (double)__ldg(mc + 2));
                    ++cnt;
                }
            }
        }
        if (live) {
            const double n = (double)(cnt + 1);
            a.xyz_out[3 * k] = (float)__ddiv_rn(sx, n); a.xyz_out[3 * k + 1] = (float)__ddiv_rn(sy, n); a.xyz_out[3 * k + 2] = (float)__ddiv_rn(sz, n);
            a.rgb_out[3 * k] = (float)__ddiv_rn(sr, n); a.rgb_out[3 * k + 1] = (float)__ddiv_rn(sg, n); a.rgb_out[3 * k + 2] = (float)__ddiv_rn(sb, n);
            a.err_out[k] = __ldg(a.err[r] + i);
            a.n_views_out[k] = cnt + 1;
            a.n_consistent_out[k] = a.n_cons[s];
        }
    }
}

}  // namespace ldp
