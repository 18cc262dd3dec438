// Depth-map fusion (ldp_depth_colors, ldp_fuse_depth_maps, ldp_fuse_depth_maps_oriented; the rules are stated in
// include/ldp_b200.h, the structure in DESIGN.md §4.10) and normal maps (ldp_depth_normals, DESIGN.md §4.11).  Not in the
// reference.  Included by ldp_api.cu (unity build), after ldp_geometry.cu (the colour blend), ldp_outlier.cu (the normal
// rule, normal_rule) and ldp_consistency.cu (the per-view test, cons_test).
//
// KF0 ldp_depth_color_kernel: the colour maps.  One thread per map pixel, grid (CTAs per view, views) like ldp_depth_kernel;
//     a kept pixel decodes its winner's warp row, gathers the four texels and blends them with bilinear_rgb, as eval_sample
//     does for a sampled pixel.
// KF1 ldp_fusion_check_kernel<NRM>: status bit 2 for a view whose depth, xyz, rgb or err pointer (with NRM: or normal map
//     pointer) is NULL.
// KF2 ldp_fusion_verdict_kernel<LENS> (pass 1): one thread per map pixel of every view, grid-stride; a pixel with a finite
//     depth is tested against every other view with cons_test and gets its consistent count and keep flag.  The view
//     constants are staged in shared memory a chunk at a time, as ldp_consistency_kernel stages them.
// KF3 ldp_fusion_emit_kernel<LENS> (pass 2, views below the pixel's own): a kept pixel is emitted unless a lower view holds a
//     kept pixel that agrees with it; the walk stops at the first one, and a CTA stops staging chunks once none of its
//     threads needs them.  The emit flags are compacted by the outlier filter's scan and ldp_outlier_kept_kernel into the
//     ascending source list.
// KF4 ldp_fusion_sum_kernel<LENS> (pass 2, views above): one thread per emitted point, reading the source list; it adds the
//     members' xyz and rgb in ascending view order and writes the fused point at its rank.
// KF2-KF4 take a second flag, NRM (ldp_fuse_depth_maps_oriented): a view's verdict is consistent only where its normal map
//     also agrees with the pixel's normal, and KF4 sums the members' normals too.  The <LENS, false> instantiations are the
//     kernels of ldp_fuse_depth_maps.
// KN1 ldp_depth_normals_check_kernel: status bit 2 for a NULL map pointer, bit 1 for a non-finite xyz under a finite depth.
// KN2 ldp_depth_normals_kernel<R>: one CTA per 16 x 16 output tile of one view, grid (tiles per view, views).  The tile's
//     (16 + 2R)^2 halo of depth and xyz is staged in shared memory; each of the 128 threads takes two pixels, lists each
//     one's window neighbourhood in shared memory (stride 128, the layout normal_epilogue reads) and calls normal_rule.
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
    const float* const* nrm;             // [V] -> [N,3] normal maps (NRM only)
    float* nrm_out;                      // [m,3] (NRM only)
    double cos_max;                      // (NRM only)
};

// the normal map pointers of a chunk (NRM only; the empty base adds nothing to the shared memory of the other kernels)
template <int CHUNK> struct FuseNormals { const float* Nm[CHUNK]; };
template <> struct FuseNormals<0> {};

// one chunk of views in shared memory
template <bool LENS, bool NRM = false>
struct FuseViews : FuseNormals<NRM ? (LENS ? CS_CHUNK_LENS : CS_CHUNK_PINHOLE) : 0> {
    static constexpr int CHUNK = LENS ? CS_CHUNK_LENS : CS_CHUNK_PINHOLE;
    double S[CHUNK][2];
    ldp_lens L[LENS ? CHUNK : 1];
    float P[CHUNK][12];
    const float* D[CHUNK];
    const float* X[CHUNK];
    const float* C[CHUNK];
};

// stages views [c0, c0 + cn); every thread of the CTA calls it
template <bool LENS, bool MEMBERS, bool NRM = false>
__device__ __forceinline__ void fuse_stage(const FusionArgs& a, FuseViews<LENS, NRM>& sv, int c0, int cn) {
    __syncthreads();
    for (int t = threadIdx.x; t < cn * 12; t += CS_THREADS) sv.P[t / 12][t % 12] = a.P[(size_t)c0 * 12 + t];
    for (int t = threadIdx.x; t < cn * 2; t += CS_THREADS) sv.S[t / 2][t % 2] = a.scales[(size_t)c0 * 2 + t];
    for (int t = threadIdx.x; t < cn; t += CS_THREADS) {
        sv.D[t] = a.depth[c0 + t];
        if constexpr (MEMBERS) { sv.X[t] = a.xyz[c0 + t]; sv.C[t] = a.rgb[c0 + t]; }
        if constexpr (NRM) sv.Nm[t] = a.nrm[c0 + t];
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

// the oriented rule's normal test: the view's normal at the pixel is finite and ((n0 m0 + n1 m1) + n2 m2) >= cos_max in f64
// without FMA (each product of two f32 values is exact)
__device__ __forceinline__ bool fuse_normal_agrees(const float* Nm, size_t pix, double n0, double n1, double n2, double cos_max) {
    const float* mp = Nm + 3 * pix;
    const float m0 = __ldg(mp), m1 = __ldg(mp + 1), m2 = __ldg(mp + 2);
    if (!(isfinite(m0) && isfinite(m1) && isfinite(m2))) return false;
    return __dadd_rn(__dadd_rn(__dmul_rn(n0, (double)m0), __dmul_rn(n1, (double)m1)), __dmul_rn(n2, (double)m2)) >= cos_max;
}

template <bool NRM>
__global__ void __launch_bounds__(CS_THREADS)
ldp_fusion_check_kernel(const FusionArgs a)
{
    grid_dependency_sync();
    const int v = blockIdx.x * CS_THREADS + threadIdx.x;
    int bad = 0;
    if (v < a.V && !(a.depth[v] && a.xyz[v] && a.rgb[v] && a.err[v])) bad = 2;
    if constexpr (NRM) { if (v < a.V && !a.nrm[v]) bad = 2; }
    bad = __reduce_or_sync(0xffffffffu, bad);
    if ((threadIdx.x & 31) == 0 && bad) atomicOr(a.status, bad);
}

template <bool LENS, bool NRM>
__global__ void __launch_bounds__(CS_THREADS)
ldp_fusion_verdict_kernel(const FusionArgs a)
{
    constexpr int CHUNK = FuseViews<LENS>::CHUNK;
    __shared__ __align__(16) FuseViews<LENS, NRM> sv;
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
        double n0 = 0.0, n1 = 0.0, n2 = 0.0;           // NRM: the pixel's own normal
        if (live) {
            r = (int)(s / N);
            const int i = (int)(s - (long long)r * N);
            if (isfinite(__ldg(a.depth[r] + i))) {
                const float* xp = a.xyz[r] + 3 * (size_t)i;
                const float x = __ldg(xp), y = __ldg(xp + 1), z = __ldg(xp + 2);
                if (isfinite(x) && isfinite(y) && isfinite(z)) { pt = true; X = x; Y = y; Z = z; }
                else atomicOr(a.status, 1);
                if constexpr (NRM) {
                    const float* np_ = a.nrm[r] + 3 * (size_t)i;
                    const float u0 = __ldg(np_), u1 = __ldg(np_ + 1), u2 = __ldg(np_ + 2);
                    if (isfinite(u0) && isfinite(u1) && isfinite(u2)) { n0 = u0; n1 = u1; n2 = u2; }
                    else pt = false;                   // no normal: not kept
                }
            }
        }
        int nc = 0, nv = 0;
        for (int c0 = 0; c0 < V; c0 += CHUNK) {
            const int cn = min(CHUNK, V - c0);
            if (staged != c0) { fuse_stage<LENS, false, NRM>(a, sv, c0, cn); staged = c0; }
            if (!pt) continue;
            for (int j = 0; j < cn; ++j) {
                if (c0 + j == r) continue;             // a pixel is never tested against its own view
                size_t pix;
                if constexpr (NRM) {
                    int dnc = 0;                       // consistent only where the normals agree too: counted here
                    if (cons_test<LENS>(sv.P[j], sv.S[j], sv.D[j], sv.L[LENS ? j : 0], X, Y, Z, a.W, a.H, a.rel_tol, dnc, nv, pix) &&
                        fuse_normal_agrees(sv.Nm[j], pix, n0, n1, n2, a.cos_max)) ++nc;
                } else {
                    cons_test<LENS>(sv.P[j], sv.S[j], sv.D[j], sv.L[LENS ? j : 0], X, Y, Z, a.W, a.H, a.rel_tol, nc, nv, pix);
                }
            }
        }
        if (live) {
            a.n_cons[s] = nc;
            a.kept[s] = (pt && nc >= a.min_views && nv <= a.max_violations) ? 1 : 0;
        }
    }
}

template <bool LENS, bool NRM>
__global__ void __launch_bounds__(CS_THREADS)
ldp_fusion_emit_kernel(const FusionArgs a)
{
    constexpr int CHUNK = FuseViews<LENS>::CHUNK;
    __shared__ __align__(16) FuseViews<LENS, NRM> sv;
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
        double n0 = 0.0, n1 = 0.0, n2 = 0.0;
        if (live && !bad) {
            r = (int)(s / N);
            need = a.kept[s] != 0;
            if (need) {
                const float* xp = a.xyz[r] + 3 * (size_t)(s - (long long)r * N);
                X = __ldg(xp); Y = __ldg(xp + 1); Z = __ldg(xp + 2);
                if constexpr (NRM) {
                    const float* np_ = a.nrm[r] + 3 * (size_t)(s - (long long)r * N);
                    n0 = __ldg(np_); n1 = __ldg(np_ + 1); n2 = __ldg(np_ + 2);
                }
            }
        }
        for (int c0 = 0; c0 < V; c0 += CHUNK) {
            const bool want = need && c0 < r;          // a lower view may still hold a member
            if (!__syncthreads_or(want)) break;
            const int cn = min(CHUNK, V - c0);
            if (staged != c0) { fuse_stage<LENS, false, NRM>(a, sv, c0, cn); staged = c0; }
            if (!want) continue;
            const int jn = min(cn, r - c0);
            for (int j = 0; j < jn; ++j) {
                size_t pix;
                int nc = 0, nv = 0;                    // unused: only the verdict and the pixel matter here
                bool agree = cons_test<LENS>(sv.P[j], sv.S[j], sv.D[j], sv.L[LENS ? j : 0], X, Y, Z, a.W, a.H, a.rel_tol, nc, nv, pix);
                if constexpr (NRM) agree = agree && fuse_normal_agrees(sv.Nm[j], pix, n0, n1, n2, a.cos_max);
                if (agree && a.kept[(size_t)(c0 + j) * N + pix]) { need = false; break; }     // the lower view emits the point
            }
        }
        if (live) a.flag[s] = need ? 1 : 0;
    }
}

template <bool LENS, bool NRM>
__global__ void __launch_bounds__(CS_THREADS)
ldp_fusion_sum_kernel(const FusionArgs a)
{
    constexpr int CHUNK = FuseViews<LENS>::CHUNK;
    __shared__ __align__(16) FuseViews<LENS, NRM> sv;
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
        double n0 = 0.0, n1 = 0.0, n2 = 0.0, snx = 0.0, sny = 0.0, snz = 0.0;     // NRM: own normal, normal sums
        if (live) {
            s = a.source[k];
            r = (int)(s / N);
            i = (int)(s - (long long)r * N);
            const float* xp = a.xyz[r] + 3 * (size_t)i;
            const float* cp = a.rgb[r] + 3 * (size_t)i;
            x = __ldg(xp); y = __ldg(xp + 1); z = __ldg(xp + 2);
            sx = x; sy = y; sz = z;
            sr = __ldg(cp); sg = __ldg(cp + 1); sb = __ldg(cp + 2);
            if constexpr (NRM) {
                const float* np_ = a.nrm[r] + 3 * (size_t)i;
                n0 = __ldg(np_); n1 = __ldg(np_ + 1); n2 = __ldg(np_ + 2);
                snx = n0; sny = n1; snz = n2;
            }
        }
        const double X = x, Y = y, Z = z;
        for (int c0 = 0; c0 < V; c0 += CHUNK) {
            const int cn = min(CHUNK, V - c0);
            const bool want = live && c0 + cn > r + 1;     // the chunk holds views above the point's own
            if (!__syncthreads_or(want)) continue;
            if (staged != c0) { fuse_stage<LENS, true, NRM>(a, sv, c0, cn); staged = c0; }
            if (!want) continue;
            for (int j = max(0, r + 1 - c0); j < cn; ++j) {
                size_t pix;
                int nc = 0, nv = 0;                    // unused: only the verdict and the pixel matter here
                bool member = cons_test<LENS>(sv.P[j], sv.S[j], sv.D[j], sv.L[LENS ? j : 0], X, Y, Z, a.W, a.H, a.rel_tol, nc, nv, pix);
                if constexpr (NRM) member = member && fuse_normal_agrees(sv.Nm[j], pix, n0, n1, n2, a.cos_max);
                if (member && a.kept[(size_t)(c0 + j) * N + pix]) {
                    const float* mp = sv.X[j] + 3 * pix;
                    const float* mc = sv.C[j] + 3 * pix;
                    sx = __dadd_rn(sx, (double)__ldg(mp)); sy = __dadd_rn(sy, (double)__ldg(mp + 1)); sz = __dadd_rn(sz, (double)__ldg(mp + 2));
                    sr = __dadd_rn(sr, (double)__ldg(mc)); sg = __dadd_rn(sg, (double)__ldg(mc + 1)); sb = __dadd_rn(sb, (double)__ldg(mc + 2));
                    if constexpr (NRM) {
                        const float* mn = sv.Nm[j] + 3 * pix;
                        snx = __dadd_rn(snx, (double)__ldg(mn)); sny = __dadd_rn(sny, (double)__ldg(mn + 1)); snz = __dadd_rn(snz, (double)__ldg(mn + 2));
                    }
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
            if constexpr (NRM) {                       // > 0: every member passed the angle test against the pixel, cos_max > 0
                const double len = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(snx, snx), __dmul_rn(sny, sny)), __dmul_rn(snz, snz)));
                a.nrm_out[3 * k] = (float)__ddiv_rn(snx, len); a.nrm_out[3 * k + 1] = (float)__ddiv_rn(sny, len);
                a.nrm_out[3 * k + 2] = (float)__ddiv_rn(snz, len);
            }
        }
    }
}

// ---- normal maps (ldp_depth_normals; rule in include/ldp_b200.h, DESIGN.md §4.11)
constexpr int DN_TILE = 16;             // output tile edge
constexpr int DN_THREADS = 128;         // two pixels of the tile per thread

struct DepthNormalArgs {
    const float* const* depth;          // [V] -> [N]
    const float* const* xyz;            // [V] -> [N,3]
    const float* centers;               // [V,3]
    float* normals;                     // [V*N,3]
    float* curvature;                   // [V*N] or NULL
    int* status;                        // [2]
    double rel_tol;
    int V, H, W, N;
    int tiles_x;
};

__global__ void __launch_bounds__(CS_THREADS)
ldp_depth_normals_check_kernel(const DepthNormalArgs a)
{
    grid_dependency_sync();
    const int v = blockIdx.y;
    const float* D = a.depth[v];
    const float* X = a.xyz[v];
    int bad = (D && X) ? 0 : 2;
    if (!bad)
        for (int i = blockIdx.x * CS_THREADS + threadIdx.x; i < a.N; i += gridDim.x * CS_THREADS)
            if (isfinite(__ldg(D + i)) &&
                !(isfinite(__ldg(X + 3 * (size_t)i)) && isfinite(__ldg(X + 3 * (size_t)i + 1)) && isfinite(__ldg(X + 3 * (size_t)i + 2))))
                bad = 1;
    bad = __reduce_or_sync(0xffffffffu, bad);
    if ((threadIdx.x & 31) == 0 && bad) atomicOr(a.status, bad);
}

template <int R>
__global__ void __launch_bounds__(DN_THREADS)
ldp_depth_normals_kernel(const DepthNormalArgs a)
{
    constexpr int HS = DN_TILE + 2 * R;                 // halo edge
    constexpr int WIN = (2 * R + 1) * (2 * R + 1);
    __shared__ float sX[HS * HS * 3];                   // [pixels][3]: normal_rule reads it directly
    __shared__ float sD[HS * HS];                       // NaN outside the map
    __shared__ int sI[WIN * DN_THREADS];                // entry j of this thread at sI[j * DN_THREADS + tid]
    grid_dependency_sync();
    if (*(volatile const int*)a.status) return;         // written by the check kernel: nothing else is written
    const int v = blockIdx.y;
    const int y0 = (blockIdx.x / a.tiles_x) * DN_TILE - R, x0 = (blockIdx.x % a.tiles_x) * DN_TILE - R;
    const float* D = a.depth[v];
    const float* X = a.xyz[v];
    const float nan = __int_as_float(0x7fc00000);
    for (int t = threadIdx.x; t < HS * HS; t += DN_THREADS) {
        const int gy = y0 + t / HS, gx = x0 + t % HS;
        sD[t] = (gy >= 0 && gy < a.H && gx >= 0 && gx < a.W) ? __ldg(D + (size_t)gy * a.W + gx) : nan;
    }
    for (int t = threadIdx.x; t < HS * HS * 3; t += DN_THREADS) {
        const int p = t / 3, gy = y0 + p / HS, gx = x0 + p % HS;
        sX[t] = (gy >= 0 && gy < a.H && gx >= 0 && gx < a.W) ? __ldg(X + 3 * ((size_t)gy * a.W + gx) + (t - 3 * p)) : nan;
    }
    __syncthreads();
    const float* centre = a.centers + 3 * (size_t)v;
    int* I = sI + threadIdx.x;
    int undefined = 0;
#pragma unroll 1
    for (int h = 0; h < 2; ++h) {
        const int pp = threadIdx.x + h * DN_THREADS, ty = pp / DN_TILE, tx = pp % DN_TILE;
        const int y = y0 + R + ty, x = x0 + R + tx;
        if (y >= a.H || x >= a.W) continue;
        const int p = (ty + R) * HS + (tx + R);
        const float dp = sD[p];
        double n[3] = {nan, nan, nan}, curv = nan;
        if (isfinite(dp)) {
            const double Dp = dp, t = __dmul_rn(a.rel_tol, Dp);
            int k = 0;
#pragma unroll
            for (int dy = -R; dy <= R; ++dy)
#pragma unroll
                for (int dx = -R; dx <= R; ++dx) {
                    const int q = p + dy * HS + dx;
                    const float dq = sD[q];             // NaN outside the map or without depth: fails the test
                    if (fabs(__dsub_rn((double)dq, Dp)) <= t) I[(k++) * DN_THREADS] = q;
                }
            const double xp[3] = {(double)sX[3 * p], (double)sX[3 * p + 1], (double)sX[3 * p + 2]};
            if (!normal_rule(sX, I, DN_THREADS, k, xp, centre, n, &curv)) {
                ++undefined;
                n[0] = n[1] = n[2] = nan;
            }
        }
        const size_t o = (size_t)v * a.N + (size_t)y * a.W + x;
        a.normals[3 * o] = (float)n[0]; a.normals[3 * o + 1] = (float)n[1]; a.normals[3 * o + 2] = (float)n[2];
        if (a.curvature) a.curvature[o] = (float)curv;
    }
    undefined = __reduce_add_sync(0xffffffffu, undefined);
    if ((threadIdx.x & 31) == 0 && undefined) atomicAdd(a.status + 1, undefined);
}

}  // namespace ldp
