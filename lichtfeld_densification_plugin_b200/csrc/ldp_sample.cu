// K1: certainty-weighted + coverage correspondence sampling, one CTA per reference view.
//
// Replaces, for every reference view of the launch,
//   * the per-pixel best neighbour           reference core/pipeline.py:634-635   (torch.max over neighbours)
//   * select_samples_with_coverage           reference core/sampling.py:8-53
//       - cap / border mask / f32 normalise  :12-14,23-29
//       - np.random.choice(replace=False, p) :31-32  == numpy legacy RandomState.choice: rejection rounds of
//         inverse-CDF draws on a sequential f64 cumsum (numpy/random/mtrand.pyx), restated in
//         oracle/densify_oracle.py:legacy_choice_no_replace
//       - per-tile best pixel ("coverage")   :34-50
//       - np.unique(concat)                  :52
//
// Data flow per view (N = H*W pixels, nn neighbours):
//   phase 1  stream nn certainty planes once (float4, evict-first)  -> w[N] f32, bestk[N] u8 in the
//            L2-resident workspace; block f64 sum -> s (or the caller's override)
//   phase 2  re-read w (L2): p = fl32(w/s) as f64, per-chunk sums in SHARED memory, per-tile arg-max
//   rounds   in-place f64 prefix over the chunk table (shared) -> per draw: binary search in shared
//            memory, then one 128-byte read of the chunk's weights and a <=chunk-long sequential scan
//            that reproduces numpy's `searchsorted(cdf/cdf[-1], u, 'right')` comparison exactly
//            (__ddiv_rn); first-occurrence dedupe by atomicOr on a bitmap; found pixels are zeroed
//            and their mass subtracted from the chunk table (exact, see DESIGN.md "exact f64 sums").
//   finish   coverage picks OR-ed into the bitmap; ordered bitmap compaction = sorted unique sel_idx.
#include <cooperative_groups.h>
#include "ldp_device.cuh"

namespace ldp {

constexpr int K1_THREADS = 1024;     // top-M kernel: one CTA per view
constexpr int KD_THREADS = 1024;     // draw kernel: 1024 threads x 64 registers, DRAW_PASS draws in flight per thread
constexpr int KS_THREADS = 256;      // stream / prep kernels: full grid
constexpr int KS_SPAN = 8192;        // pixels per CTA of the full-grid passes (multiple of every chunk size)

// (double)f without the conversion (XU) pipe for normal f (any sign): rebias the exponent, shift the mantissa.
// Zero, subnormal, inf and NaN inputs take the real conversion.
__device__ __forceinline__ double widen_f32(float f) {
    const uint32_t b = __float_as_uint(f);
    const uint32_t e = (b >> 23) & 0xffu;
    if (e == 0u || e == 0xffu) return (double)f;
    return __hiloint2double((int)((b & 0x80000000u) | (((b & 0x7fffffffu) >> 3) + 0x38000000u)), (int)(b << 29));
}

struct K1Shared {
    double red_d[32];
    int red_i[32];
    int n_found;
};

__device__ __forceinline__ unsigned long long cov_key(float p, int idx) {
    return ((unsigned long long)__float_as_uint(p) << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)idx);
}

// descending bitonic sort of n (power of two) 64-bit keys
__device__ void bitonic_sort_desc(unsigned long long* a, int n) {
    for (int k = 2; k <= n; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            // one compare-exchange per thread and step: pair p -> elements (i, i + j), i = p with a zero inserted at bit log2(j)
            for (int p = threadIdx.x; p < (n >> 1); p += blockDim.x) {
                const int i = ((p & ~(j - 1)) << 1) | (p & (j - 1)), l = i + j;
                const unsigned long long x = a[i], y = a[l];
                const bool desc = ((i & k) == 0);
                if (desc ? (x < y) : (x > y)) { a[i] = y; a[l] = x; }
            }
            __syncthreads();
        }
    }
}

// =============================================================================================
// K1a  stream: grid (ceil(N / KS_SPAN), n_refs).  Reads every certainty value once (float4, evict-first),
//      writes w = min(best, cap) * border_mask (f32) and the winning neighbour (u8) to the L2-resident
//      workspace, and one f64 partial weight sum + NaN/negative flags per CTA.
//      reference core/pipeline.py:634-635 (torch.max over neighbours), core/sampling.py:12-14,23-25
//      HBM-bound by design: the instruction budget per 4-pixel quad is kept small (plane pointers in
//      registers, magic-number row/column, interior fast path for the border mask, NaN found via the sum).
// =============================================================================================
__device__ __forceinline__ uint32_t div_magic(uint32_t n, unsigned long long magic) {     // floor(n / d), d's magic = ceil(2^40/d)
    return (uint32_t)(((unsigned long long)n * magic) >> 40);
}

__device__ __forceinline__ void quad_border_weights(float wv[4], int px, int x, int y, int W, int H, int border, int N) {
    if (x + 3 < W && px + 3 < N) {
        // the quad lies in one image row (always on the vector path): pixels j in [lo, hi] are inside, if the row is
        const bool row_ok = y >= border && y <= H - 1 - border;
        const int lo = border - x, hi = W - 1 - border - x;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float m = (row_ok && j >= lo && j <= hi) ? 1.f : 0.f;
            wv[j] = wv[j] * m;                                 // cert * inside.float(): inf * 0 = NaN like torch
        }
        return;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float m = (x >= border && x <= W - 1 - border && y >= border && y <= H - 1 - border) ? 1.f : 0.f;
        float v = wv[j] * m;
        if (px + j >= N) v = 0.f;
        wv[j] = v;
        if (++x == W) { x = 0; ++y; }
    }
}

#ifndef KS_MIN_BLOCKS
#define KS_MIN_BLOCKS 5
#endif
// NNMAX 1..4: plane pointers held in registers, loop fully unrolled, two quads per step; 5..8: one quad per step, NNMAX loads
// in flight; 0: any nn (pointers in shared memory).
// PRO: the planes are raw matcher outputs and the reference's post-processing (core/pipeline.py:405-430) is applied
//      to every value as it is read (ldp_device.cuh:prologue_cert).
//      PRO = 1: no view of the launch has a neighbour mask (ldp_params.no_warped_masks): clamp and reference-view mask only - no warp
//      row is read, registers and occupancy stay those of the plain kernel; PRO = 2: warped neighbour masks as well.
template <int NNMAX, int PRO>
__global__ void __launch_bounds__(KS_THREADS, PRO == 2 ? 3 : (NNMAX > 4 ? 4 : KS_MIN_BLOCKS))      // PRO 2 holds the warp rows too: more registers
ldp_stream_kernel(const ldp_params P, const ldp_ref_desc* __restrict__ refs, const Workspace ws, const SampleGeom G)
{
    grid_dependency_sync();
    __shared__ const float* s_cert[LDP_MAX_NN];
    __shared__ double red_d[32];
    __shared__ float red_f[32];
    __shared__ ProView s_pv;
    const int r = blockIdx.y, blk = blockIdx.x, tid = threadIdx.x;
    const int N = G.N;
    const ldp_ref_desc* rd = refs + r;
    const int nn = rd->nn;
    if (tid < LDP_MAX_NN) s_cert[tid] = (tid < nn) ? rd->cert[tid] : nullptr;
    if (PRO) stage_proview(rd, s_pv, tid);
    if (blk == 0) {          // per-view state consumed by the later kernels of this launch
        if (tid == 0) {
            ws.rstat[r].s = 0.f; ws.rstat[r].npos = 0; ws.rstat[r].emin_inv = 0; ws.rstat[r].bad = 0;
            ws.kept[r] = 0;
        }
        unsigned long long* gb = ws.gbins + (size_t)r * ws.bins_cap;
        for (int i = tid; i < (int)ws.bins_cap; i += KS_THREADS) gb[i] = 0ull;
    }
    __syncthreads();
    float* __restrict__ w = ws.w + (size_t)r * ws.n_pad;
    uint8_t* __restrict__ bk = ws.bestk + (size_t)r * ws.n_pad;
    const float cap = P.sample_cap;
    const int W = P.W, H = P.H, border = P.no_filter ? 0 : P.border;
    const int base = blk * KS_SPAN;
    double lsum = 0.0;
    float lmin = 0.f;                      // running minimum: negative weights (NaN is caught through the sum)
    if (nn > 0) {
        const float* c0 = s_cert[0];
        const float* c1 = (NNMAX >= 2) ? s_cert[min(1, nn - 1)] : nullptr;
        const float* c2 = (NNMAX >= 3) ? s_cert[min(2, nn - 1)] : nullptr;
        const float* c3 = (NNMAX >= 4) ? s_cert[min(3, nn - 1)] : nullptr;
        // finishes one quad: cap, border mask, flags, f64 sum, stores
        auto finish_quad_xy = [&](int px, int x, int y, float wv[4], const int bi[4]) {
#pragma unroll
            for (int j = 0; j < 4; ++j) wv[j] = (wv[j] > cap) ? cap : wv[j];          // torch.clamp(max=cap): NaN stays NaN
            const bool interior = y >= border && y <= H - 1 - border && x >= border && x + 3 <= W - 1 - border && px + 3 < N;
            if (!interior) quad_border_weights(wv, px, x, y, W, H, border, N);
            lmin = fminf(lmin, fminf(fminf(wv[0], wv[1]), fminf(wv[2], wv[3])));
            // hardware conversions here: 4 per quad on the conversion pipe cost this kernel ~2.6 us of that pipe, the integer
            // widening (widen_f32, right for the conversion-bound prep / draw kernels) a fifth of its issue slots
            lsum += ((double)wv[0] + (double)wv[1]) + ((double)wv[2] + (double)wv[3]);
            *reinterpret_cast<float4*>(w + px) = make_float4(wv[0], wv[1], wv[2], wv[3]);
            *reinterpret_cast<uint32_t*>(bk + px) = (uint32_t)bi[0] | ((uint32_t)bi[1] << 8) | ((uint32_t)bi[2] << 16) | ((uint32_t)bi[3] << 24);
        };
        auto finish_quad = [&](int px, float wv[4], const int bi[4]) {
            const int y = (int)div_magic((uint32_t)px, G.w_magic);
            finish_quad_xy(px, px - y * W, y, wv, bi);
        };
        auto take = [&](const float4& c, int k, float wv[4], int bi[4]) {              // NaN-propagating max, first index wins
            if (c.x > wv[0] || c.x != c.x) { wv[0] = c.x; bi[0] = k; }
            if (c.y > wv[1] || c.y != c.y) { wv[1] = c.y; bi[1] = k; }
            if (c.z > wv[2] || c.z != c.z) { wv[2] = c.z; bi[2] = k; }
            if (c.w > wv[3] || c.w != c.w) { wv[3] = c.w; bi[3] = k; }
        };
        // ---- raw planes (PRO): the reference's post-processing of one quad of neighbour k (core/pipeline.py:405-430);
        //      a quad lies in one image row on the vector path.  Same arithmetic as ldp_device.cuh:prologue_cert.
        const bool has_a = PRO && s_pv.mask_a != nullptr;
        const bool ident_a = has_a && s_pv.mask_w == W && s_pv.mask_h == H && (reinterpret_cast<uintptr_t>(s_pv.mask_a) & 3u) == 0;
        auto mask_a_quad = [&](int px, float ma[4]) {
            if (ident_a) {                                             // same resolution: 4 mask bytes in one load
                const uint32_t m = __ldg(reinterpret_cast<const uint32_t*>(s_pv.mask_a + px));
                ma[0] = (float)(m & 0xffu); ma[1] = (float)((m >> 8) & 0xffu); ma[2] = (float)((m >> 16) & 0xffu); ma[3] = (float)(m >> 24);
            } else {
                const int y = (int)div_magic((uint32_t)px, G.w_magic), x = px - y * W;
#pragma unroll
                for (int j = 0; j < 4; ++j) ma[j] = mask_at(s_pv.mask_a, x + j, y, s_pv);
            }
        };
        auto warped_mask = [&](const uint8_t* __restrict__ mb, const float2 g) {
            const float fx = rintf(__fsub_rn(__fmul_rn(__fadd_rn(g.x, 1.f), 0.5f * (float)W), 0.5f));
            const float fy = rintf(__fsub_rn(__fmul_rn(__fadd_rn(g.y, 1.f), 0.5f * (float)H), 0.5f));
            float m = 0.f;
            if (fx > -1.f && fx < (float)W && fy > -1.f && fy < (float)H) m = mask_at(mb, (int)fx, (int)fy, s_pv);
            return m;
        };
        auto pro_quad = [&](float4& c, int k, int px, const float ma[4]) {
            const float fl = P.certainty_floor;
            c.x = (c.x < fl) ? fl : c.x; c.y = (c.y < fl) ? fl : c.y;               // torch.clamp(min=): NaN stays NaN
            c.z = (c.z < fl) ? fl : c.z; c.w = (c.w < fl) ? fl : c.w;
            if (has_a) { c.x = __fmul_rn(c.x, ma[0]); c.y = __fmul_rn(c.y, ma[1]); c.z = __fmul_rn(c.z, ma[2]); c.w = __fmul_rn(c.w, ma[3]); }
            const uint8_t* mb = (PRO == 2) ? s_pv.mask_b[k] : nullptr;
            if (mb) {                                                              // (xB, yB) of the 4 rows: read once, evict-first
                const float2* g = reinterpret_cast<const float2*>(s_pv.warp[k] + (size_t)px * 4 + 2);
                const float2 g0 = __ldcs(g), g1 = __ldcs(g + 2), g2 = __ldcs(g + 4), g3 = __ldcs(g + 6);
                c.x = __fmul_rn(c.x, warped_mask(mb, g0)); c.y = __fmul_rn(c.y, warped_mask(mb, g1));
                c.z = __fmul_rn(c.z, warped_mask(mb, g2)); c.w = __fmul_rn(c.w, warped_mask(mb, g3));
            }
        };
        if (G.vec && NNMAX > 4 && !PRO) {
            // 5..8 neighbours: one quad per step, all NNMAX 128-bit loads issued before any of them is consumed
            for (int it = 0; it < KS_SPAN / (KS_THREADS * 4); ++it) {
                const int px = base + (it * KS_THREADS + tid) * 4;
                if (px >= N) break;
                float4 a[NNMAX > 4 ? NNMAX : 1];
#pragma unroll
                for (int k = 0; k < NNMAX; ++k) a[k] = ld_stream4(s_cert[min(k, nn - 1)] + px);    // clamp: a duplicate load, not a branch
                float wv[4] = {a[0].x, a[0].y, a[0].z, a[0].w};
                int bi[4] = {0, 0, 0, 0};
#pragma unroll
                for (int k = 1; k < NNMAX; ++k) if (k < nn) take(a[k], k, wv, bi);
                finish_quad(px, wv, bi);
            }
        } else if (G.vec && NNMAX > 0 && NNMAX <= 4) {
            // two quads per step: all 2*NNMAX 128-bit loads are issued before any of them is consumed
            constexpr int STEP = KS_THREADS * 4;
            // (x, y) of the thread's quad, advanced by the pass stride instead of divided out of the pixel index every time
            int qy = (int)div_magic((uint32_t)(base + tid * 4), G.w_magic), qx = base + tid * 4 - qy * W;
            auto advance = [&](int& x, int& y) { x += G.step_dx; y += G.step_dy; if (x >= W) { x -= W; ++y; } };
            for (int it = 0; it < KS_SPAN / STEP; it += 2) {
                const int pxa = base + it * STEP + tid * 4, pxb = pxa + STEP;
                const bool va = pxa < N, vb = pxb < N;
                if (!va) break;
                const int qb = vb ? pxb : pxa;                         // clamp: a duplicate load instead of a branch
                float4 a0, a1, a2, a3, b0, b1, b2, b3;
                a0 = ld_stream4(c0 + pxa); b0 = ld_stream4(c0 + qb);
                if (NNMAX >= 2) { a1 = ld_stream4(c1 + pxa); b1 = ld_stream4(c1 + qb); }
                if (NNMAX >= 3) { a2 = ld_stream4(c2 + pxa); b2 = ld_stream4(c2 + qb); }
                if (NNMAX >= 4) { a3 = ld_stream4(c3 + pxa); b3 = ld_stream4(c3 + qb); }
                if (PRO) {
                    float ma[4] = {1.f, 1.f, 1.f, 1.f}, mb[4] = {1.f, 1.f, 1.f, 1.f};
                    if (has_a) { mask_a_quad(pxa, ma); mask_a_quad(qb, mb); }
                    pro_quad(a0, 0, pxa, ma); pro_quad(b0, 0, qb, mb);
                    if (NNMAX >= 2 && nn >= 2) { pro_quad(a1, 1, pxa, ma); pro_quad(b1, 1, qb, mb); }
                    if (NNMAX >= 3 && nn >= 3) { pro_quad(a2, 2, pxa, ma); pro_quad(b2, 2, qb, mb); }
                    if (NNMAX >= 4 && nn >= 4) { pro_quad(a3, 3, pxa, ma); pro_quad(b3, 3, qb, mb); }
                }
                float wa[4] = {a0.x, a0.y, a0.z, a0.w}, wb[4] = {b0.x, b0.y, b0.z, b0.w};
                int ia[4] = {0, 0, 0, 0}, ib[4] = {0, 0, 0, 0};
                if (NNMAX >= 2) { take(a1, 1, wa, ia); take(b1, 1, wb, ib); }
                if (NNMAX >= 3) { take(a2, 2, wa, ia); take(b2, 2, wb, ib); }
                if (NNMAX >= 4) { take(a3, 3, wa, ia); take(b3, 3, wb, ib); }
                finish_quad_xy(pxa, qx, qy, wa, ia);
                advance(qx, qy);
                if (vb) finish_quad_xy(pxb, qx, qy, wb, ib);
                advance(qx, qy);
            }
        } else {
            for (int it = 0; it < KS_SPAN / (KS_THREADS * 4); ++it) {
                const int px = base + (it * KS_THREADS + tid) * 4;
                if (px >= N) break;
                float wv[4];
                int bi[4] = {0, 0, 0, 0};
                if (PRO) {
                    // raw planes: post-process each value, then the same first-index-wins maximum
                    int y = (int)div_magic((uint32_t)px, G.w_magic), x = px - y * W;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        float best = 0.f;
                        int bk = 0;
                        if (px + j < N) {
                            best = prologue_cert(__ldcs(c0 + px + j), 0, px + j, x, y, P, s_pv);
                            for (int k = 1; k < nn; ++k) {
                                const float c = prologue_cert(__ldcs(s_cert[k] + px + j), k, px + j, x, y, P, s_pv);
                                if (c > best || c != c) { best = c; bk = k; }
                            }
                        }
                        wv[j] = best; bi[j] = bk;
                        if (++x == W) { x = 0; ++y; }
                    }
                } else if (G.vec) {
                    const float4 v = ld_stream4(c0 + px);
                    wv[0] = v.x; wv[1] = v.y; wv[2] = v.z; wv[3] = v.w;
#pragma unroll 4
                    for (int k = 1; k < nn; ++k) take(ld_stream4(s_cert[k] + px), k, wv, bi);
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j) wv[j] = (px + j < N) ? __ldcs(c0 + px + j) : 0.f;
                    for (int k = 1; k < nn; ++k) {
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const float c = (px + j < N) ? __ldcs(s_cert[k] + px + j) : 0.f;
                            if (c > wv[j] || c != c) { wv[j] = c; bi[j] = k; }
                        }
                    }
                }
                finish_quad(px, wv, bi);
            }
        }
    }
    if (blk == (int)gridDim.x - 1) {       // keep the row padding [N, n_pad) zero: the draw kernel's 32-byte scans read it
        for (int i = ((N + 3) & ~3) + tid; i < (int)ws.n_pad; i += KS_THREADS) w[i] = 0.f;
    }
    const double bsum = block_sum(lsum, red_d);
    const float bmin = -block_sum_max(-lmin, red_f);
    if (tid == 0) {
        ws.partial[(size_t)r * ws.nblk + blk] = bsum;
        ws.bflags[(size_t)r * ws.nblk + blk] = ((bsum != bsum) ? 1 : 0) | ((bmin < 0.f) ? 2 : 0) | ((nn <= 0) ? 4 : 0);
    }
}

// =============================================================================================
// K1b  prep: same grid.  s = f32(sum of the f64 partials) (or the caller's override); p = fl32(w / s) is
//      written back IN PLACE over w (so the draw kernel never divides); f64 sums of p per chunk go to the
//      global chunk table; per-tile arg-max of p (the coverage picks); number of positive p and their smallest
//      exponent (exactness test); clears the selection bitmap.
//      reference core/sampling.py:26-29 (normalise), :34-50 (coverage walk == per-tile arg-max)
//      Issue-bound, so the per-pixel work is kept small:
//        * p = fl32(w / s) with the correctly rounded reciprocal of s hoisted out of the loop and two FMA residual
//          corrections per value (div_by); zeros and tiny quotients take the IEEE division.
//        * positives / smallest positive exponent from the quad minimum; zeros (border, masked) take a side path;
//        * per-tile arg-max as one 64-bit key (p bits << 32 | ~index) per tile in shared memory, raised by atomicMax
//          behind an exact pre-filter; one key per tile and CTA then goes to the global table.
//      CS = chunk_shift (5..7: chunk sums by shuffles inside a warp row of 128 pixels; 0: wider chunks, atomics).
//      COLS = how a quad's coverage tiles are found (PrepCols; launch_sample states when each mode applies).
// =============================================================================================
// fl32(a / b) for b > 0 with y = RN(1/b) hoisted: two residual corrections on the FMA pipe.  q1 is a faithful quotient
// (error <= 1/2 ulp + 2^-23 ulp), so by Markstein's theorem (y correctly rounded, residual exact) the second correction
// rounds to RN(a / b).  Requires exact residuals: a >= 2^-100 or a == 0, results in the normal range (callers guard).
// Checked against __fdiv_rn on 2^32 operand pairs by scratch/divcheck.cu.
__device__ __forceinline__ float div_by(float a, float b, float y) {
    const float q0 = __fmul_rn(a, y);
    const float r0 = __fmaf_rn(-b, q0, a);
    const float q1 = __fmaf_rn(r0, y, q0);
    const float r1 = __fmaf_rn(-b, q1, a);
    return __fmaf_rn(r1, y, q1);
}

#ifdef LDP_PHASE_CLOCKS
__device__ __forceinline__ long long gtimer() { long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#define LDP_PCLK(slot) do { if (threadIdx.x == 0 && (blockIdx.x == 3 || blockIdx.x == 31)) ws.dbgclk[(size_t)r * 32 + (blockIdx.x == 3 ? 18 : 24) + (slot)] = gtimer(); } while (0)
#else
#define LDP_PCLK(slot) do { } while (0)
#endif
#ifndef KP_MIN_BLOCKS
#define KP_MIN_BLOCKS 5
#endif
// How the prep kernel finds the coverage tiles of a quad's pixels.
enum class PrepCols {
    CONST,      // as QUAD, and a thread's quads all start in one pixel column: its tile split is computed once
    QUAD,       // a quad lies in one image row and in at most two tiles, whose columns umulhi(x, t_magic32) finds
    PIXEL,      // any map: a tile per pixel, through the 40-bit magic
};
template <int CS, PrepCols COLS>
__global__ void __launch_bounds__(KS_THREADS, KP_MIN_BLOCKS)
ldp_prep_kernel(const ldp_params P, const ldp_ref_desc* __restrict__ refs, const Workspace ws, const ldp_outputs out,
                const SampleGeom G)
{
    grid_dependency_sync();
    {   // the draw kernels' selection bitmap: cleared here, one kernel ahead of its first use
        uint32_t* bm = ws.bitmap + (size_t)blockIdx.y * ws.n_words;
        for (int i = blockIdx.x * KS_THREADS + threadIdx.x; i < (int)ws.n_words; i += gridDim.x * KS_THREADS) bm[i] = 0u;
    }
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int red_i[32];
    __shared__ float s_s;
    __shared__ int s_bad;
    constexpr int NIT = KS_SPAN / (KS_THREADS * 4);
    constexpr int STEP = KS_THREADS * 4;
    const int r = blockIdx.y, blk = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const int N = G.N, W = P.W;
    const ldp_ref_desc* rd = refs + r;
    LDP_PCLK(0);
    float* __restrict__ w = ws.w + (size_t)r * ws.n_pad;
    const int base = blk * KS_SPAN;
    int px = base + tid * 4;
    // the first quad's load is in flight while the normaliser is reduced
    float4 vnext = (px < N) ? __ldcg(reinterpret_cast<const float4*>(w + px)) : make_float4(0.f, 0.f, 0.f, 0.f);
    // ---- s: fixed-order reduction of the per-CTA partials (every CTA of the view computes the same value)
    if (tid < 32) {
        double a = 0.0;
        int f = 0;
        for (int i = lane; i < (int)ws.nblk; i += 32) {
            a += ws.partial[(size_t)r * ws.nblk + i];
            f |= ws.bflags[(size_t)r * ws.nblk + i];
        }
        a = warp_sum(a);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) f |= __shfl_xor_sync(0xffffffffu, f, o);
        if (lane == 0) {
            float s = (float)a;
            if (rd->weight_sum_override > 0.f) s = rd->weight_sum_override;
            s_s = s;
            s_bad = f;
            if (blk == 0) {
                ws.rstat[r].s = s;
                ws.rstat[r].bad = f;
                if (out.weight_sum) out.weight_sum[r] = s;
            }
        }
    }

    const int end = min(base + KS_SPAN, N);
    const int y_first = (int)div_magic((uint32_t)base, G.w_magic), y_last = (int)div_magic((uint32_t)(end - 1), G.w_magic);
    // tile rows: umulhi is exact for y * tile < N < 2^30, but one-pixel tiles (PIXEL only) have no 32-bit magic
    const int ty0 = (COLS == PrepCols::PIXEL) ? (int)div_magic((uint32_t)y_first, G.t_magic) : (int)__umulhi((uint32_t)y_first, G.t_magic32);
    const int ty1 = (COLS == PrepCols::PIXEL) ? (int)div_magic((uint32_t)y_last, G.t_magic) : (int)__umulhi((uint32_t)y_last, G.t_magic32);
    const int nlb = (ty1 - ty0 + 1) * G.nbx;
    unsigned long long* lb = reinterpret_cast<unsigned long long*>(smem_raw);            // [nlb] (p bits << 32) | ~index
    for (int i = tid; i < nlb; i += KS_THREADS) lb[i] = 0ull;
    __syncthreads();
    const float s = s_s;
    if (s_bad || !(s > 0.f)) return;       // the draw kernel reports the status
    const float yr = __frcp_rn(s);                     // correctly rounded reciprocal, once per thread
    const bool fast_div = (s >= 1.0f) && (s < 3.0e8f);  // then p >= 2^-90 implies w >= 2^-90: every residual of div_by is exact
    LDP_PCLK(1);

    double* __restrict__ csum = ws.csum + (size_t)r * ws.nchunk_pad;
    double* __restrict__ csum0 = ws.csum0 + (size_t)r * ws.nchunk_pad;      // the copy the first draw round searches (see Workspace)
    int lpos = 0;
    uint32_t lmin1 = 0xFFFFFFFFu;                      // (bit pattern - 1) of the smallest positive p; zeros wrap to the top
    int y = (int)div_magic((uint32_t)px, G.w_magic), x = px - y * W;
    // tile geometry of a CONST / QUAD quad: pixels [0, nsplit) lie in tile column tx0, the rest in tx0 + 1
    int tx0 = (int)__umulhi((uint32_t)x, G.t_magic32);
    int nsplit = (tx0 + 1) * G.tile - x;               // >= 4: no straddle
#pragma unroll
    for (int it = 0; it < NIT; ++it) {
        double a = 0.0;
        const float4 v = vnext;
        if (it + 1 < NIT) {
            const int qn = px + STEP;
            vnext = (qn < N) ? __ldcg(reinterpret_cast<const float4*>(w + qn)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (px < N) {
            // core/sampling.py:29 -- zeros (border, masked) divide to exact zeros on the fast path too
            float p0 = div_by(v.x, s, yr), p1 = div_by(v.y, s, yr), p2 = div_by(v.z, s, yr), p3 = div_by(v.w, s, yr);
            const uint32_t c0 = __float_as_uint(p0) - 1u, c1 = __float_as_uint(p1) - 1u, c2 = __float_as_uint(p2) - 1u, c3 = __float_as_uint(p3) - 1u;
            uint32_t cmin = min(min(c0, c1), min(c2, c3));
            if (cmin < 0x12000000u || !fast_div) {     // a non-zero quotient below 2^-91 (or an unusual s): IEEE division
                p0 = __fdiv_rn(v.x, s); p1 = __fdiv_rn(v.y, s); p2 = __fdiv_rn(v.z, s); p3 = __fdiv_rn(v.w, s);
                cmin = min(min(__float_as_uint(p0) - 1u, __float_as_uint(p1) - 1u), min(__float_as_uint(p2) - 1u, __float_as_uint(p3) - 1u));
            }
            lmin1 = min(lmin1, cmin);
            const float pmin = fminf(fminf(p0, p1), fminf(p2, p3));
            if (pmin > 0.f) lpos += 4;
            else lpos += ((p0 > 0.f) ? 1 : 0) + ((p1 > 0.f) ? 1 : 0) + ((p2 > 0.f) ? 1 : 0) + ((p3 > 0.f) ? 1 : 0);
            *reinterpret_cast<float4*>(w + px) = make_float4(p0, p1, p2, p3);
            a = ((double)p0 + (double)p1) + ((double)p2 + (double)p3);
            // ---- per-tile arg-max of p, lowest index on ties: 64-bit key, exact pre-filter, rare CAS
            if (COLS == PrepCols::PIXEL) {                 // the quad may wrap a row end or cover several tiles
                const float pv[4] = {p0, p1, p2, p3};
                int xx = x, yy = y;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (pv[j] > 0.f && px + j < N) {
                        const int b = ((int)div_magic((uint32_t)yy, G.t_magic) - ty0) * G.nbx + (int)div_magic((uint32_t)xx, G.t_magic);
                        const unsigned long long key = cov_key(pv[j], px + j);
                        if (lb[b] < key) atomicMax(&lb[b], key);
                    }
                    if (++xx == W) { xx = 0; ++yy; }
                }
            } else {
                if (COLS == PrepCols::QUAD) {
                    tx0 = (int)__umulhi((uint32_t)x, G.t_magic32);
                    nsplit = (tx0 + 1) * G.tile - x;
                }
                const int b0 = ((int)__umulhi((uint32_t)y, G.t_magic32) - ty0) * G.nbx + tx0;
                const bool s1 = nsplit > 1, s2 = nsplit > 2, s3 = nsplit > 3;               // pixel j belongs to the first tile
                const float m0 = fmaxf(fmaxf(p0, s1 ? p1 : 0.f), fmaxf(s2 ? p2 : 0.f, s3 ? p3 : 0.f));
                const unsigned long long k0 = ((unsigned long long)__float_as_uint(m0) << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)px);
                if (k0 > lb[b0]) {                         // could improve the tile (k0 bounds the exact key from above)
                    const int j0 = (p0 == m0) ? 0 : (s1 && p1 == m0) ? 1 : (s2 && p2 == m0) ? 2 : 3;
                    if (m0 > 0.f) atomicMax(&lb[b0], k0 - (unsigned long long)j0);
                }
                if (!s3) {                                 // the quad straddles a tile edge
                    const float m1 = fmaxf(fmaxf(s1 ? 0.f : p1, s2 ? 0.f : p2), p3);
                    const unsigned long long k1 = ((unsigned long long)__float_as_uint(m1) << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)px);
                    if (k1 > lb[b0 + 1]) {
                        const int j1 = (!s1 && p1 == m1) ? 1 : (!s2 && p2 == m1) ? 2 : 3;
                        if (m1 > 0.f) atomicMax(&lb[b0 + 1], k1 - (unsigned long long)j1);
                    }
                }
            }
        }
        // ---- chunk sums
        if (CS >= 5 && CS <= 7) {
            constexpr int GL = (CS >= 5 && CS <= 7) ? ((1 << CS) >> 2) : 1;
#pragma unroll
            for (int o = 1; o < GL; o <<= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
            if (px < N && (lane & (GL - 1)) == 0) { csum[px >> CS] = a; csum0[px >> CS] = a; }
        } else {
            const int cs = G.chunk_shift;          // chunks wider than a warp row (zeroed by the host memset)
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
            if (px < N && lane == 0) { atomicAdd(&csum[px >> cs], a); atomicAdd(&csum0[px >> cs], a); }
        }
        px += STEP;
        if (COLS == PrepCols::CONST) {
            y += G.step_dy;
        } else {
            x += G.step_dx; y += G.step_dy;
            if (x >= W) { x -= W; ++y; }
        }
    }
    LDP_PCLK(2);
    const int npos = block_sum(lpos, red_i);
    const uint32_t min1 = (uint32_t)block_min((int)(lmin1 ^ 0x80000000u), red_i) ^ 0x80000000u;   // unsigned order through the signed reduction
    if (tid == 0) {
        if (npos) atomicAdd(&ws.rstat[r].npos, npos);
        if (min1 != 0xFFFFFFFFu) atomicMax(&ws.rstat[r].emin_inv, 255 - (int)(((min1 + 1u) >> 23) & 0xffu));
    }
    __syncthreads();
    LDP_PCLK(3);
    unsigned long long* gb = ws.gbins + (size_t)r * ws.bins_cap;
    for (int i = tid; i < nlb; i += KS_THREADS) {
        const unsigned long long key = lb[i];
        if (key) atomicMax(&gb[(ty0 + i / G.nbx) * G.nbx + (i % G.nbx)], key);
    }
    LDP_PCLK(4);
}

// =============================================================================================
// K1c  draw: one thread-block CLUSTER of C CTAs per view.  numpy's legacy RandomState.choice(replace=False, p)
//      restated (oracle/densify_oracle.py:legacy_choice_no_replace): rejection rounds of inverse-CDF draws.
//
//      The kernel is bound by the SM's load/store wavefront rate, not by arithmetic (profiles/r01_*), so every
//      step is organised to touch few 128-byte wavefronts:
//        * every CTA keeps the view's f64 chunk-prefix table in shared memory, in a padded layout
//          (2 doubles after every 8) that makes the per-thread 8-entry prefix build conflict-free;
//        * a guide table (bucket of u -> first candidate chunk) cuts the binary search to 1-3 probes;
//        * the chunk's p values are scanned with 32-byte (LDG.256) loads and early exit;
//        * numpy's exact predicate fl64(cum / total) > u (__ddiv_rn) is evaluated once, at the first
//          approximate crossing (slow exact continuation otherwise);
//        * first-occurrence dedupe = atomicOr on the global selection bitmap; the found mass leaves the
//          global chunk sums through fire-and-forget f64 reductions at L2 (exact sums => order-free, DESIGN.md);
//          found p are zeroed by their finder after the round's cluster barrier.
//      Finally CTA 0 ORs the coverage picks in and an ordered bitmap compaction yields np.unique(concat).
//      reference core/sampling.py:31-32,34-52
// =============================================================================================
#ifndef LDP_NO_GUIDE
#define LDP_USE_GUIDE 1              // round 1 searches inside guide-table ranges (measured: 32.8 vs 41.0 us without the table)
#endif
constexpr int DRAW_PASS = 2;          // draws a thread keeps in flight (they share one Philox call): every phase is
                                      // batched over them so that its loads overlap -- the kernel is latency- and
                                      // LSU-wavefront-bound, not ALU-bound (profiles/r01_draw_*.md)

__device__ __forceinline__ int pad8(int i) { return i + ((i >> 3) << 1); }     // padded table index

__device__ __forceinline__ void ldg256(const float* p, float v[8]) {
    asm volatile("ld.global.cg.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]) : "l"(p));
}
__device__ __forceinline__ void ldg256u(const uint32_t* p, uint32_t v[8]) {
    asm volatile("ld.global.cg.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]) : "l"(p));
}
__device__ __forceinline__ void red_add_f64(double* addr, double v) {
    asm volatile("red.global.add.f64 [%0], %1;" :: "l"(addr), "d"(v) : "memory");
}

// (double)f for f >= 0 without the conversion (XU) pipe: rebias the exponent, shift the mantissa.
// Zero and subnormal inputs take the real conversion (never on the hot path: p >= 2^-126 there).
__device__ __forceinline__ double widen_pos(float f) {
    const uint32_t b = __float_as_uint(f);
    if ((b >> 23) == 0u && b != 0u) return (double)f;          // subnormal: never on the hot path
    const double d = __hiloint2double((int)((b >> 3) + 0x38000000u), (int)(b << 29));
    return (b == 0u) ? 0.0 : d;                                // zeros (border, already drawn) without a branch
}

// numpy's predicate fl64(x / total) > u, decided without dividing whenever x is outside a 2^-50 relative band
// around t = fl(u * total):  x > t(1+2^-50)  =>  x/total > u(1+2^-51) >= nextafter(u)  => true;
//                            x < t(1-2^-50)  =>  x/total < u                            => false.
__device__ __forceinline__ bool cdf_exceeds(double x, double total, double u, double t_hi, double t_lo) {
    if (x > t_hi) return true;
    if (x < t_lo) return false;
    return __ddiv_rn(x, total) > u;
}

// Exact continuation of a scan (rare: the approximate crossing was not the exact one, or inexact sums).
__device__ __noinline__ int slow_exact_scan(const float* __restrict__ w, const uint32_t* __restrict__ gone, int start, int N,
                                            double cum, double total, double u, int last, float* pout) {
    for (int i = start; i < N; ++i) {
        float p = __ldcg(w + i);
        if (gone && ((__ldcg(gone + (i >> 5)) >> (i & 31)) & 1u)) p = 0.f;         // drawn in round 1
        if (p > 0.f) {
            cum += (double)p;
            last = i;
            *pout = p;
            if (__ddiv_rn(cum, total) > u) return i;
        }
    }
    return last;
}

// MODE 1: the first rejection round only (all `size` draws), c_first INDEPENDENT CTAs per view -- they meet only in
//         the selection bitmap (atomicOr), the global chunk sums (red.add) and their own find lists, so no cluster is
//         needed and every SM of the device can take part;
// MODE 2: everything after it, one thread-block cluster per view: zero the found p, rounds 2.., coverage picks,
//         ordered compaction.  The kernel boundary is the barrier between round 1 and round 2.
template <int MODE>
__global__ void __launch_bounds__(KD_THREADS, 1)
ldp_draw_kernel(const ldp_params P, const ldp_ref_desc* __restrict__ refs, const double* __restrict__ uniforms,
                const Workspace ws, const ldp_outputs out, const SampleGeom G, const int c_first)
{
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* pre = reinterpret_cast<double*>(smem_raw);                         // [pad8(nchunk_ept)] padded prefix
    int* guide = reinterpret_cast<int*>(pre + G.draw_pre_cap);                 // [NG + 2]
    unsigned long long* bins = reinterpret_cast<unsigned long long*>(smem_raw);   // coverage sort reuses the table
    __shared__ K1Shared sh;

    const int C = (MODE == 1) ? c_first : (int)cluster.num_blocks();
    const int crank = (MODE == 1) ? (int)(blockIdx.x % (unsigned)C) : (int)cluster.block_rank();
    const int r = blockIdx.x / C;
    const int tid = threadIdx.x, lane = tid & 31;
    const int T = blockDim.x;
    const int gtid = crank * T + tid, GT = C * T;
    const int N = G.N;
    const int nchunk = G.nchunk;
    const int NG = G.draw_ng;
    const ldp_ref_desc* rd = refs + r;

    float* __restrict__ w = ws.w + (size_t)r * ws.n_pad;                 // holds p after the prep kernel
    uint32_t* __restrict__ bitmap = ws.bitmap + (size_t)r * ws.n_words;
    int32_t* __restrict__ flist = ws.found + ((size_t)r * ws.draw_cmax + crank) * ws.found_cap;
    int32_t* __restrict__ fcnt = ws.fcnt + (size_t)r * ws.draw_cmax;
    int32_t* __restrict__ sel = (out.sel_idx ? out.sel_idx : ws.sel) + (size_t)r * ws.sel_cap;
    double* __restrict__ gcsum = ws.csum + (size_t)r * ws.nchunk_pad;
    // Round 1 runs on independent CTAs that may start at different times - after their siblings' first finds have left the chunk
    // sums - and numpy's first round searches the cdf of ALL weights: they build their tables from the copy the prep kernel
    // made (csum0, never modified); every find is removed from csum, which the later rounds (one cluster, barriers between
    // rounds) search.
    const double* __restrict__ gtable = (MODE == 1) ? ws.csum0 + (size_t)r * ws.nchunk_pad : gcsum;
    const unsigned long long* __restrict__ gb = ws.gbins + (size_t)r * ws.bins_cap;
    const uint32_t* __restrict__ gone = (MODE == 2) ? ws.gone + (size_t)r * ws.n_words : nullptr;   // drawn in round 1

    auto finish_empty = [&](int status) {
        if (gtid == 0) {
            out.status[r] = status;
            out.n_samples[r] = 0;
            if (out.uniforms_used) out.uniforms_used[r] = 0;
            if (out.rounds) out.rounds[r] = 0;
        }
    };
    grid_dependency_sync();
    LDP_CLK(ws, r, 0);
    // MODE 2: everything the prologue needs is fetched in one batch (each L2 round trip costs ~0.75 us here)
    int ds = 0, nfc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (MODE == 2) {
        ds = __ldcg(ws.dstat + r);
#pragma unroll
        for (int c2 = 0; c2 < 8; ++c2) nfc[c2] = (c2 < c_first) ? __ldcg(fcnt + c2) : 0;
    }
    // every exit below is taken by all CTAs of the view alike (same inputs, same arithmetic); MODE 2 reports
    const RefStat st = ws.rstat[r];
    if (st.bad & 4) { if (MODE == 2) finish_empty(LDP_REF_NO_NEIGHBOURS); return; }
    if (st.bad & 1) { if (MODE == 2) finish_empty(LDP_REF_BAD_WEIGHTS); return; }          // NaN: `s <= 0` is False, choice raises
    if (!(st.s > 0.f)) { if (MODE == 2) finish_empty(LDP_REF_EMPTY); return; }             // core/sampling.py:27-28
    if (st.bad & 2) { if (MODE == 2) finish_empty(LDP_REF_BAD_WEIGHTS); return; }

    const int cs = G.chunk_shift;
    const int size = G.size;
    const int EPT = G.draw_ept;                     // table entries per thread (multiple of 8)
    int n_have = 0, drawn = 0, rounds = 0, fail = 0, inexact = 0;
    const double* U = uniforms ? uniforms + (size_t)r * (size_t)P.uniforms_per_ref : nullptr;
    const uint32_t rng_stream = rd->rng_stream;

    if (MODE == 2) {
        // ---- pick up after round 1: its verdict, its finds; the finders' p are zeroed here (the barrier before the
        //      next draws orders these stores)
        fail = ds & 0xff;
        inexact = (ds >> 8) & 1;
        if (fail) { finish_empty(fail); return; }
        drawn = size;
        rounds = 1;
#pragma unroll
        for (int c2 = 0; c2 < 8; ++c2) n_have += nfc[c2];
        if (n_have < size) {
            // The pixels drawn in round 1 must weigh nothing from now on.  Zeroing their p would be ~8500 scattered
            // 4-byte stores per view (one load/store wavefront each); instead the selection bitmap as round 1 left it
            // is copied (coalesced, 32 KB) and the scans of the later rounds mask by it.  The few pixels drawn in the
            // later rounds are zeroed in place as before.
            const uint4* src = reinterpret_cast<const uint4*>(bitmap);
            uint4* dst = reinterpret_cast<uint4*>(ws.gone + (size_t)r * ws.n_words);
            for (int i = gtid; i < (int)(ws.n_words / 4); i += GT) dst[i] = __ldcg(src + i);
        }
    }
    LDP_CLK(ws, r, 1);
    while (MODE == 1 || n_have < size) {
        if (MODE == 2 && rounds <= 4) LDP_CLK(ws, r, 18 + 2 * rounds);
        // ---- (a) padded inclusive prefix of the global chunk sums: 8-entry rows per thread, one block scan
        if (tid == 0) sh.n_found = 0;
        // coalesced copy of the global chunk sums into the padded table, then 8-entry rows per thread
        for (int i0 = 2 * tid; i0 < nchunk; i0 += 8 * T) {          // 4 loads in flight per thread (L2 latency, not bandwidth)
            double2 d[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int i = i0 + 2 * j * T;
                d[j] = (i < nchunk) ? __ldcg(reinterpret_cast<const double2*>(gtable + i)) : make_double2(0.0, 0.0);   // nchunk_pad is even
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int i = i0 + 2 * j * T;
                if (i < nchunk) *reinterpret_cast<double2*>(pre + pad8(i)) = make_double2(d[j].x, (i + 1 < nchunk) ? d[j].y : 0.0);
            }
        }
        if (rounds == 0) LDP_CLK(ws, r, 11);
        __syncthreads();
        if (rounds == 0) LDP_CLK(ws, r, 12);
        double run = 0.0;
        const int e0 = tid * EPT;
        for (int q = 0; q < EPT; q += 8) {
            const int i0 = e0 + q;
            if (i0 < nchunk) {
                double2* row = reinterpret_cast<double2*>(pre + pad8(i0));
                double v[8];
#pragma unroll
                for (int j = 0; j < 8; j += 2) {          // entries beyond the table are whatever shared memory held: mask both halves
                    const double2 d = row[j >> 1];
                    v[j] = (i0 + j < nchunk) ? d.x : 0.0;
                    v[j + 1] = (i0 + j + 1 < nchunk) ? d.y : 0.0;
                }
#pragma unroll
                for (int j = 0; j < 8; ++j) { run += v[j]; v[j] = run; }
#pragma unroll
                for (int j = 0; j < 8; j += 2) row[j >> 1] = make_double2(v[j], v[j + 1]);
            }
        }
        if (rounds == 0) LDP_CLK(ws, r, 14);
        double total;
        const double base = block_exclusive_scan(run, sh.red_d, &total);
        if (rounds == 0) LDP_CLK(ws, r, 15);
        for (int q = 0; q < EPT; q += 8) {
            const int i0 = e0 + q;
            if (i0 < nchunk) {
                double2* dst = reinterpret_cast<double2*>(pre + pad8(i0));
#pragma unroll
                for (int j = 0; j < 4; ++j) { double2 d = dst[j]; d.x += base; d.y += base; dst[j] = d; }
            }
        }
#ifdef LDP_USE_GUIDE
        if (rounds == 0) for (int i = tid; i < NG + 2; i += T) guide[i] = nchunk - 1;
#endif
        __syncthreads();
        if (rounds == 0) LDP_CLK(ws, r, 16);
        total = pre[pad8(nchunk - 1)];
        if (rounds == 0) {
            // numpy's checks in RandomState.choice, in numpy's order
            if (fabs(total - 1.0) > 3.4526698300124393e-4) { fail = LDP_REF_PSUM; break; }
            if (st.npos < size) { fail = LDP_REF_FEWER_NONZERO; break; }
            // exactness of every f64 partial sum: all p are multiples of 2^(emin-150) and the total stays below
            // 2^53 of those units  <=>  ilogb(total) - (emin - 150) < 53
            if (st.npos > 0) {
                const int etot = ilogb(total);
                const int emin = 255 - st.emin_inv;          // smallest biased exponent among the positive p
                if (emin <= 0 || etot - (emin - 150) >= 53) inexact = 1;
            }
            LDP_CLK(ws, r, 17);                        // (the selection bitmap was cleared by the prep kernel)
        }
        if (n_have >= size) break;
        const int cnt = size - n_have;
        if (P.rng_mode == LDP_RNG_EXPLICIT && (int64_t)drawn + cnt > P.uniforms_per_ref) { fail = LDP_REF_UNIFORMS_EXHAUSTED; break; }
        if (rounds >= 64) { fail = LDP_REF_ROUNDS_EXCEEDED; break; }
        // ---- (a') guide table: guide[k] ~ first chunk whose prefix reaches (k / NG) * total.  It only has to be
        //      approximately right: the exact fix-up after the search walks to numpy's chunk from any start.
        //      Built for the first round only (8500 draws); later rounds have a few hundred draws and search the
        //      whole table.
#ifdef LDP_USE_GUIDE
        if (rounds == 0) {
            const double ngt = (double)NG / total;
            int kprev = (e0 > 0 && e0 <= nchunk) ? min(NG, (int)(pre[pad8(e0 - 1)] * ngt)) : -1;
            for (int q = 0; q < EPT; ++q) {
                const int c = e0 + q;
                if (c < nchunk) {
                    int kc = min(NG, (int)(pre[pad8(c)] * ngt));
                    if (c == nchunk - 1) kc = NG + 1;
                    for (int k = max(kprev, -1) + 1; k <= kc; ++k) guide[k] = c;       // (max: never below the table, whatever the sums)
                    kprev = max(kprev, kc);
                }
            }
        }
#endif
        if (rounds > 0 && C > 1) cluster.sync(); else __syncthreads();    // B2: the p zeroed after the last round are visible
        if (MODE == 2 && rounds == 1) LDP_CLK(ws, r, 2);
        if (rounds == 0) LDP_CLK(ws, r, 3);
        // ---- (b) draws: each thread takes DRAW_PASS (=2) consecutive draws per pass (one Philox call)
        constexpr double EPS_UP = 1.0 + 1.0 / 1125899906842624.0, EPS_DN = 1.0 - 1.0 / 1125899906842624.0;
        // MODE 1 (8500 draws, issue bound): two draws per thread and pass, sharing one Philox call, 8 weights per scan step.
        // MODE 2 (a few hundred draws, latency bound): one draw per thread, a branch-free search over the whole table and
        // the whole 32-weight line of the chunk requested at once -- every dependent L2 round trip costs ~0.7 us here.
        constexpr int ND = (MODE == 2) ? 1 : 2;
        for (int dw = ND * (gtid - lane); dw < cnt; dw += ND * GT) {      // warp-uniform trip count (ballots inside)
            const int d0 = dw + ND * lane;
            double uu[2], tt[2], cum[2];
            int lo[2], hi[2], ii[2];
            float hp[2];
            bool valid[2], hit[2];
            cum[1] = 0.0; lo[1] = hi[1] = 0; ii[1] = -1; hp[1] = 0.f; hit[1] = true; tt[1] = 0.0;      // (absent when ND == 1)
            // 1. uniforms + guide lookups
            valid[0] = d0 < cnt;
            valid[1] = (ND == 2) && d0 + 1 < cnt;
            if (P.rng_mode == LDP_RNG_EXPLICIT) {
                uu[0] = valid[0] ? U[drawn + d0] : 0.5;
                uu[1] = valid[1] ? U[drawn + d0 + 1] : 0.5;
            } else if (ND == 1) {
                uu[0] = philox_uniform(P.seed, rng_stream, (uint32_t)(drawn + d0));
                uu[1] = 0.5;
            } else if (((drawn + d0) & 1) == 0) {
                philox_uniform2(P.seed, rng_stream, (uint32_t)(drawn + d0), uu);
            } else {
                uu[0] = philox_uniform(P.seed, rng_stream, (uint32_t)(drawn + d0));
                uu[1] = philox_uniform(P.seed, rng_stream, (uint32_t)(drawn + d0 + 1));
            }
#pragma unroll
            for (int k = 0; k < ND; ++k) {
                tt[k] = uu[k] * total;
#ifdef LDP_USE_GUIDE
                const int kb = min(NG - 1, (int)(uu[k] * (double)NG));
                lo[k] = (rounds == 0) ? guide[kb] : 0;
                hi[k] = (rounds == 0) ? max(lo[k], guide[kb + 1]) : nchunk - 1;
#else
                lo[k] = 0; hi[k] = nchunk - 1;
#endif
            }
            // 2. lock-step binary search inside the guide ranges: first chunk with prefix > u * total (approximate)
            if (MODE == 2 && rounds == 1 && dw == ND * (gtid - lane)) LDP_CLK(ws, r, 11);
#ifdef LDP_USE_GUIDE
            if (MODE == 2)
#endif
            {                           // branch-free upper bound over the whole table: #entries <= target, one probe per bit
                int pos[2] = {0, 0};    // (the probes of the two draws are independent and pipeline)
                for (int step = 1 << (31 - __clz(max(nchunk, 1))); step > 0; step >>= 1) {
#pragma unroll
                    for (int k = 0; k < ND; ++k) {
                        const int q = pos[k] + step;
                        if (q <= nchunk && !(pre[pad8(q - 1)] > tt[k])) pos[k] = q;
                    }
                }
#pragma unroll
                for (int k = 0; k < ND; ++k) lo[k] = min(pos[k], nchunk - 1);
            }
#ifdef LDP_USE_GUIDE
            else
            for (;;) {
                bool more = false;
#pragma unroll
                for (int k = 0; k < ND; ++k) {
                    if (lo[k] < hi[k]) {
                        const int mid = (lo[k] + hi[k]) >> 1;
                        if (pre[pad8(mid)] > tt[k]) hi[k] = mid; else lo[k] = mid + 1;
                        more |= lo[k] < hi[k];
                    }
                }
                if (!more) break;
            }
#endif
            // 3. exact predicate of searchsorted(cdf, u, 'right') on the chunk boundaries
            if (MODE == 2 && rounds == 1 && dw == ND * (gtid - lane)) LDP_CLK(ws, r, 12);
#pragma unroll
            for (int k = 0; k < ND; ++k) {
                int c = lo[k];
                const double thi = tt[k] * EPS_UP, tlo = tt[k] * EPS_DN;
                double below = (c > 0) ? pre[pad8(c - 1)] : 0.0;
                const double here = pre[pad8(c)];
                const bool down = (c > 0) && cdf_exceeds(below, total, uu[k], thi, tlo);
                const bool up = (c < nchunk - 1) && !cdf_exceeds(here, total, uu[k], thi, tlo);
                if (down || up) {                             // rare: walk to the exact chunk
                    while (c > 0 && cdf_exceeds(pre[pad8(c - 1)], total, uu[k], thi, tlo)) --c;
                    while (c < nchunk - 1 && !cdf_exceeds(pre[pad8(c)], total, uu[k], thi, tlo)) ++c;
                    below = (c > 0) ? pre[pad8(c - 1)] : 0.0;
                }
                lo[k] = c;
                cum[k] = below;
                hit[k] = !valid[k];
                ii[k] = -1;
                hp[k] = 0.f;
            }
            // 4. in-chunk scans: one 32-byte piece per draw per step, both loads in flight together.  The kernel is bound
            if (MODE == 2 && rounds == 1 && dw == ND * (gtid - lane)) LDP_CLK(ws, r, 14);
            //    by instruction issue here, so a piece costs 8 conversions + 8 DADD + 8 compares: p >= 0 makes the running
            //    sums monotone, hence the first pixel whose sum exceeds the target is found by COUNTING the sums that do
            //    not (its own weight is then necessarily positive).  A draw that hits keeps its piece in registers.
            constexpr int PW = (MODE == 2) ? 32 : 8;          // weights examined per step
            const int steps = (1 << cs) / PW;                 // chunks hold at least 32 weights
            float e[2][PW];
            int fm[2] = {-1, -1};
            for (int pc = 0; pc < steps; ++pc) {
                if (!__any_sync(0xffffffffu, !hit[0] || !hit[1])) break;
#pragma unroll
                uint32_t gm[2] = {0u, 0u};
#pragma unroll
                for (int k = 0; k < ND; ++k)
                    if (!hit[k]) {
#pragma unroll
                        for (int q = 0; q < PW; q += 8) ldg256(w + (lo[k] << cs) + pc * PW + q, e[k] + q);
                        if (MODE == 2) { const int b = (lo[k] << cs) + pc * PW; gm[k] = __ldcg(gone + (b >> 5)) >> (b & 31); }
                    }
                if (MODE == 2) {
#pragma unroll
                    for (int k = 0; k < ND; ++k)
                        if (!hit[k]) {
#pragma unroll
                            for (int m = 0; m < PW; ++m) if ((gm[k] >> m) & 1u) e[k][m] = 0.f;
                        }
                }
#pragma unroll
                for (int k = 0; k < ND; ++k) {
                    if (!hit[k]) {
                        const double tlo = tt[k] * EPS_DN;
                        const int b = (lo[k] << cs) + pc * PW;
                        if (cum[k] > tlo) {            // rare: the sum entered the piece inside the tolerance band already:
                            int f = -1;                // the first positive weight is the candidate
#pragma unroll
                            for (int m = PW - 1; m >= 0; --m) if (e[k][m] > 0.f) f = m;
                            if (f >= 0) { hit[k] = true; fm[k] = f; ii[k] = b + f; }
                        } else {
                            double c = cum[k];         // padding beyond N is zero (stream kernel)
                            int nle = 0;
#pragma unroll
                            for (int m = 0; m < PW; ++m) { c += (double)e[k][m]; nle += (c <= tlo) ? 1 : 0; }
                            if (nle < PW) { hit[k] = true; fm[k] = nle; ii[k] = b + nle; }     // cum stays the sum before the piece
                            else cum[k] = c;
                        }
                    }
                }
            }
            // 4b. running sum and weight at the candidate (once per draw)
            if (MODE == 2 && rounds == 1 && dw == ND * (gtid - lane)) LDP_CLK(ws, r, 15);
#pragma unroll
            for (int k = 0; k < ND; ++k) {
                if (fm[k] >= 0) {
                    double c = cum[k];
                    float h = 0.f;
#pragma unroll
                    for (int m = 0; m < PW; ++m) if (m <= fm[k]) { c += (double)e[k][m]; h = e[k][m]; }
                    cum[k] = c;
                    hp[k] = h;
                }
            }
            // 5. numpy's exact comparison at the approximate crossing (slow exact continuation otherwise)
#pragma unroll
            for (int k = 0; k < ND; ++k) {
                if (valid[k]) {
                    const double thi = tt[k] * EPS_UP, tlo = tt[k] * EPS_DN;
                    if (ii[k] >= 0) {
                        if (!cdf_exceeds(cum[k], total, uu[k], thi, tlo))
                            ii[k] = slow_exact_scan(w, gone, ii[k] + 1, N, cum[k], total, uu[k], ii[k], &hp[k]);
                    } else {
                        ii[k] = slow_exact_scan(w, gone, min(N, (lo[k] + 1) << cs), N, cum[k], total, uu[k], -1, &hp[k]);
                    }
                }
            }
            // 6. dedupe (both atomics in flight together), then warp-aggregated append + mass removal
            if (MODE == 2 && rounds == 1 && dw == ND * (gtid - lane)) LDP_CLK(ws, r, 16);
            uint32_t old[2] = {0xffffffffu, 0xffffffffu};
#pragma unroll
            for (int k = 0; k < ND; ++k)
#ifdef LDP_EXP_NOOR
                old[k] = (ii[k] >= 0) ? 0u : 0xffffffffu;
#else
                old[k] = (ii[k] >= 0) ? atomicOr(&bitmap[ii[k] >> 5], 1u << (ii[k] & 31)) : 0xffffffffu;
#endif
            // two draws of one thread may hit the same pixel: the second is then not fresh
            const bool fresh0 = ii[0] >= 0 && !(old[0] & (1u << (ii[0] & 31)));
            const bool fresh1 = ii[1] >= 0 && !(old[1] & (1u << (ii[1] & 31)));
            const unsigned fm0 = __ballot_sync(0xffffffffu, fresh0), fm1 = __ballot_sync(0xffffffffu, fresh1);
            if (fm0 | fm1) {
                const int n0 = __popc(fm0), n1 = __popc(fm1);
                int basepos = 0;
                if (lane == 0) basepos = atomicAdd(&sh.n_found, n0 + n1);
                basepos = __shfl_sync(0xffffffffu, basepos, 0);
                const unsigned below_mask = (1u << lane) - 1u;
                if (fresh0) {
                    flist[basepos + __popc(fm0 & below_mask)] = ii[0];
#ifndef LDP_EXP_NORED
                    red_add_f64(gcsum + (ii[0] >> cs), -widen_pos(hp[0]));      // the found mass leaves the chunk sum
#endif
                }
                if (fresh1) {
                    flist[basepos + n0 + __popc(fm1 & below_mask)] = ii[1];
#ifndef LDP_EXP_NORED
                    red_add_f64(gcsum + (ii[1] >> cs), -widen_pos(hp[1]));
#endif
                }
            }
        }
        __syncthreads();
        if (rounds == 0) LDP_CLK(ws, r, 4);
        if (MODE == 2 && rounds <= 4) LDP_CLK(ws, r, 19 + 2 * rounds);
        const int my_new = sh.n_found;
        if (tid == 0) fcnt[crank] = my_new;
        if (MODE == 1) {                   // round 1 ends with the kernel; MODE 2 continues
            if (gtid == 0) ws.dstat[r] = inexact << 8;
            return;
        }
        if (C > 1) cluster.sync(); else __syncthreads();          // B1: every draw of the round is done and published
        if (rounds == 0) LDP_CLK(ws, r, 6);
        int n_new = 0;
        for (int c2 = 0; c2 < C; ++c2) n_new += (C > 1) ? __ldcg(fcnt + c2) : my_new;
        drawn += cnt;
        ++rounds;
        n_have += n_new;
        if (n_have >= size) break;                        // done
        for (int e0z = 0; e0z < my_new; e0z += 8 * T) {                           // the finder zeroes its p
            int zi[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) { const int e = e0z + j * T + tid; zi[j] = (e < my_new) ? flist[e] : -1; }
#pragma unroll
            for (int j = 0; j < 8; ++j) if (zi[j] >= 0) w[zi[j]] = 0.f;
        }
        if (rounds == 1) LDP_CLK(ws, r, 7);
        // no barrier here: the chunk sums were complete at B1; the zeroing stores drain while the table is rebuilt and
        // are ordered before the next round's scans by the cluster barrier B2 above
    }
    LDP_CLK(ws, r, 8);
    if (MODE == 1) {                       // reached only through a failed check or size == 0: no draws were made
        if (tid == 0) fcnt[crank] = 0;
        if (gtid == 0) ws.dstat[r] = fail | (inexact << 8);
        return;
    }
    if (fail) { finish_empty(fail); return; }
    // The coverage picks are CTA 0's; the ordered compaction is shared by the CTAs of the cluster when its size divides
    // the 8 bitmap words a thread owns (every CTA scans the whole bitmap, each extracts a contiguous range of words).
    const bool share = (C == 2 || C == 4 || C == 8);
    if (crank != 0 && !share) return;
    __syncthreads();

    // ------------------------------------------------------------------ coverage picks (core/sampling.py:34-50)
    if (crank == 0) {
        int lp = 0;
        for (int i = tid; i < G.nbins; i += T) lp += (gb[i] != 0ull) ? 1 : 0;
        const int nb_pos = block_sum(lp, sh.red_i);
        if (nb_pos > G.cov_budget) {          // budget binds: keep the cov_budget best tiles (descending weight)
            int nb_pow2 = 1;
            while (nb_pow2 < G.nbins) nb_pow2 <<= 1;
            for (int i = tid; i < nb_pow2; i += T) bins[i] = (i < G.nbins) ? gb[i] : 0ull;
            __syncthreads();
            bitonic_sort_desc(bins, nb_pow2);
            for (int i = tid; i < G.cov_budget; i += T) {
                const unsigned long long key = bins[i];
                if (key != 0ull) {
                    const int idx = (int)(0xFFFFFFFFu - (uint32_t)(key & 0xFFFFFFFFull));
                    atomicOr(&bitmap[idx >> 5], 1u << (idx & 31));
                }
            }
        } else {
            for (int i = tid; i < G.nbins; i += T) {
                const unsigned long long key = gb[i];
                if (key != 0ull) {
                    const int idx = (int)(0xFFFFFFFFu - (uint32_t)(key & 0xFFFFFFFFull));
                    atomicOr(&bitmap[idx >> 5], 1u << (idx & 31));
                }
            }
        }
        __threadfence();
        __syncthreads();
    }
    if (share) cluster.sync();                            // the picks are in the bitmap before anybody counts it
    LDP_CLK(ws, r, 9);

    // ------------------------------------------------------------------ ordered compaction == np.unique(concat)
    // Two passes per tile of T*8 bitmap words.  (1) each thread counts the bits of 8 CONSECUTIVE words, one block scan
    // gives every word its output offset (shared memory).  (2) the CTA's range of words is walked again INTERLEAVED over
    // the threads (word t, t + T, ...): the selected pixels cluster in the confident regions of the map, and the bit
    // extraction of a thread that owns 256 consecutive pixels of such a region would serialise its whole warp.
    {
        const int nwords = (int)ws.n_words;                    // multiple of 8 (n_pad is a multiple of 256)
        int* woff = reinterpret_cast<int*>(smem_raw);          // the chunk table is dead: [T*8 + 1] per-word output offsets,
        const int wcap = min(nwords, T * 8) + 1;
        int* stage = woff + wcap;                              // then staged indices for coalesced stores
        const int stage_cap = (int)(G.draw_smem_bytes / sizeof(int)) - wcap;
        const int nshare = share ? C : 1;
        const int wpc = (T * 8) / nshare;                      // words of a tile this CTA extracts
        int carry = 0;
        for (int t0 = 0; t0 < nwords; t0 += T * 8) {
            const int w0 = t0 + tid * 8;
            uint32_t m[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            if (w0 < nwords) ldg256u(bitmap + w0, m);
            int cntb = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) cntb += __popc(m[j]);
            LDP_CLK(ws, r, 28);
            int tile_total;
            int pos = block_exclusive_scan(cntb, sh.red_i, &tile_total);
            LDP_CLK(ws, r, 29);
            const int tw = min(T * 8, nwords - t0);                              // words in this tile
            if (w0 < nwords) {
#pragma unroll
                for (int j = 0; j < 8; ++j) { woff[tid * 8 + j] = pos; pos += __popc(m[j]); }
            }
            if (tid == 0) woff[tw] = tile_total;                                 // sentinel
            __syncthreads();
            const int lo_w = min(crank * wpc, tw), hi_w = min(lo_w + wpc, tw);   // this CTA's words of the tile (tile-relative)
            const int out_lo = woff[lo_w], out_hi = woff[hi_w];
            const bool staged = (out_hi - out_lo) <= stage_cap;
            for (int jj = 0; jj < wpc; jj += T) {
                const int wr = lo_w + jj + tid;                                  // tile-relative word
                if (wr < hi_w) {
                    uint32_t mm = __ldcg(bitmap + t0 + wr);
                    int o = woff[wr];
                    while (mm) {
                        const int b = __ffs(mm) - 1;
                        mm &= mm - 1;
                        const int v = ((t0 + wr) << 5) + b;
                        if (staged) stage[o - out_lo] = v;
                        else if (carry + o < (int)ws.sel_cap) sel[carry + o] = v;
                        ++o;
                    }
                }
            }
            __syncthreads();
            LDP_CLK(ws, r, 30);
            if (staged)
                for (int i = tid; i < out_hi - out_lo; i += T)
                    if (carry + out_lo + i < (int)ws.sel_cap) sel[carry + out_lo + i] = stage[i];
            __syncthreads();
            carry += tile_total;
        }
        if (crank != 0) return;
        LDP_CLK(ws, r, 10);
        if (tid == 0) {
            out.status[r] = LDP_REF_OK | (inexact ? LDP_REF_INEXACT_SCAN : 0);
            out.n_samples[r] = min(carry, (int)ws.sel_cap);
            if (out.uniforms_used) out.uniforms_used[r] = drawn;
            if (out.rounds) out.rounds[r] = rounds;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// no_filter branch of the sampler (reference core/sampling.py:15-21): the M pixels of largest capped
// certainty, in descending order.  np.argsort is unstable, so the order among equal certainties is
// implementation-defined in the reference; here ties are broken by ascending pixel index.
// One CTA per view; runs after ldp_sample_kernel's phase 1 (w = capped certainty, no border mask).
//   1. 4-pass 8-bit radix select over the f32 keys -> value of the M-th largest, #strictly greater
//   2. ordered gather of {key > kth} U {first (M - #greater) pixels with key == kth}
//   3. bitonic sort of the M (key, ~index) pairs, descending
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t f32_order_key(float f) {
    if (f != f) return 0u;                      // numpy sorts NaN last in argsort(-x)
    const uint32_t b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

__global__ void __launch_bounds__(K1_THREADS, 1)
ldp_topm_generic_kernel(const ldp_params P, const ldp_ref_desc* __restrict__ refs, const Workspace ws,
                const ldp_outputs out, const SampleGeom G)
{
    grid_dependency_sync();
    __shared__ int hist[256];
    __shared__ int red_i[32];
    __shared__ uint32_t s_prefix;
    __shared__ int s_remaining;
    const int r = blockIdx.x, tid = threadIdx.x, T = blockDim.x, N = G.N;
    const float* __restrict__ w = ws.w + (size_t)r * ws.n_pad;
    int32_t* __restrict__ sel = (out.sel_idx ? out.sel_idx : ws.sel) + (size_t)r * ws.sel_cap;
    unsigned long long* keys = ws.topk_keys + (size_t)r * ws.topk_cap;
    const int M = min(P.matches_per_ref, N);
    if (refs[r].nn <= 0 || M <= 0) {
        if (tid == 0) { out.status[r] = (refs[r].nn <= 0) ? LDP_REF_NO_NEIGHBOURS : LDP_REF_EMPTY; out.n_samples[r] = 0; }
        return;
    }
    // 1. radix select (most significant byte first)
    if (tid == 0) { s_prefix = 0u; s_remaining = M; }
    __syncthreads();
    for (int pass = 0; pass < 4; ++pass) {
        const int shift = 24 - 8 * pass;
        for (int i = tid; i < 256; i += T) hist[i] = 0;
        __syncthreads();
        const uint32_t prefix = s_prefix;
        const uint32_t pmask = (pass == 0) ? 0u : (0xFFFFFFFFu << (shift + 8));
        for (int i = tid; i < N; i += T) {
            const uint32_t k = f32_order_key(w[i]);
            if ((k & pmask) == prefix) atomicAdd(&hist[(k >> shift) & 0xffu], 1);
        }
        __syncthreads();
        if (tid == 0) {
            int rem = s_remaining;
            int b = 255;
            for (; b > 0; --b) {
                if (hist[b] >= rem) break;
                rem -= hist[b];
            }
            s_prefix = prefix | ((uint32_t)b << shift);
            s_remaining = rem;            // how many of the elements equal-so-far are still needed
        }
        __syncthreads();
    }
    const uint32_t kth = s_prefix;
    const int need_eq = s_remaining;
    // 2. ordered gather
    const int Lp = (N + T - 1) / T;
    const int p0 = min(tid * Lp, N), p1 = min(p0 + Lp, N);
    int c_gt = 0, c_eq = 0;
    for (int i = p0; i < p1; ++i) {
        const uint32_t k = f32_order_key(w[i]);
        c_gt += (k > kth);
        c_eq += (k == kth);
    }
    int tot_gt, tot_eq;
    int o_gt = block_exclusive_scan(c_gt, red_i, &tot_gt);
    int o_eq = block_exclusive_scan(c_eq, red_i, &tot_eq);
    for (int i = p0; i < p1; ++i) {
        const uint32_t k = f32_order_key(w[i]);
        if (k > kth) { keys[o_gt++] = ((unsigned long long)k << 32) | (0xFFFFFFFFu - (uint32_t)i); }
        else if (k == kth) {
            if (o_eq < need_eq) keys[tot_gt + o_eq] = ((unsigned long long)k << 32) | (0xFFFFFFFFu - (uint32_t)i);
            ++o_eq;
        }
    }
    int n2 = 1;
    while (n2 < M) n2 <<= 1;
    for (int i = M + tid; i < n2; i += T) keys[i] = 0ull;
    __threadfence_block();
    __syncthreads();
    // 3. sort descending (global memory, L2-resident)
    bitonic_sort_desc(keys, n2);
    for (int i = tid; i < M; i += T) sel[i] = (int)(0xFFFFFFFFu - (uint32_t)(keys[i] & 0xFFFFFFFFull));
    if (tid == 0) {
        out.status[r] = LDP_REF_OK;
        out.n_samples[r] = M;
        if (out.uniforms_used) out.uniforms_used[r] = 0;
        if (out.rounds) out.rounds[r] = 0;
    }
}

// ---------------------------------------------------------------------------------------------
// no_filter, fast variant (M <= 16384): same result as ldp_topm_generic_kernel.  One thread-block CLUSTER of C CTAs per
// view (C = 1, 2, 4 or 8, chosen by the host so that the views fill the SMs): every pass over the view's pixels is
// split between the CTAs (contiguous slices of quads), the histograms meet through distributed shared memory, and the
// M selected keys are sorted by a bitonic network whose 64-bit keys live in the shared memory of the C CTAs.
//   1. 3-pass radix select (11 + 11 + 10 bits) of the M-th largest key: coalesced reads; one shared atomic per 128-pixel
//      row, per quad or per pixel depending on how many pixels share a bin (certainties saturated at the cap would
//      otherwise serialise on one bin); every CTA sums the C histograms and finds the crossing bin by a suffix scan;
//   2. if more pixels tie at that key than are needed, the ones with the lowest indices win (np.argsort is unstable in
//      the reference; ours is "ascending index"): the index of the last one taken is found by the same radix select
//      over the pixel index of the tied pixels (skipped when every tied pixel is taken);
//   3. unordered gather of the M keys (one counter in CTA 0, one atomic per warp, keys stored straight into the owning
//      CTA's slice), bitonic sort (two butterfly stages per shared-memory pass; the stages whose partner lives in
//      another CTA read it over DSMEM into a second buffer), write out.
// ---------------------------------------------------------------------------------------------
constexpr int KT_BINS = 2048;
constexpr int KT_UNROLL = 4;
// bins of the four pixels of a thread's quad (-1: not counted)
__device__ __forceinline__ void topm_hist_add4(int* hist, int b0, int b1, int b2, int b3) {
    const bool uni = (b0 == b1) && (b1 == b2) && (b2 == b3);
    const int v0 = __shfl_sync(0xffffffffu, b0, 0);
    if (__all_sync(0xffffffffu, uni && b0 == v0)) {                 // the warp's whole 128-pixel row in one bin (or in none)
        if (v0 >= 0 && (threadIdx.x & 31) == 0) atomicAdd(&hist[v0], 128);
    } else if (uni) {
        if (b0 >= 0) atomicAdd(&hist[b0], 4);
    } else {
        if (b0 >= 0) atomicAdd(&hist[b0], 1);
        if (b1 >= 0) atomicAdd(&hist[b1], 1);
        if (b2 >= 0) atomicAdd(&hist[b2], 1);
        if (b3 >= 0) atomicAdd(&hist[b3], 1);
    }
}
// Same, for passes in which a warp's 128 pixels fall into few distinct bins (the most significant key digit of
// certainties in [0, 1]): lanes with the same bin are found with match.any and their leader adds the group's count - one
// conflict-free atomic per distinct bin instead of up to 32 atomics colliding on one address.
__device__ __forceinline__ void topm_hist_add4_few(int* hist, int b0, int b1, int b2, int b3) {
    const int lane = threadIdx.x & 31;
    const bool uni = (b0 == b1) && (b1 == b2) && (b2 == b3);
    if (__all_sync(0xffffffffu, uni)) {                                // every thread's quad in one bin: one match for the four
        const unsigned m = __match_any_sync(0xffffffffu, b0);
        if (b0 >= 0 && (__ffs(m) - 1) == lane) atomicAdd(&hist[b0], 4 * __popc(m));
        return;
    }
    const int b[4] = {b0, b1, b2, b3};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const unsigned m = __match_any_sync(0xffffffffu, b[j]);
        if (b[j] >= 0 && (__ffs(m) - 1) == lane) atomicAdd(&hist[b[j]], __popc(m));
    }
}
// Waits for the C local histograms of the pass, sums them, and finds - scanning the bins from the top (DESC) or from the
// bottom - the bin in which the running count reaches `rem`; returns the bin, how many are still needed inside it
// (*rem_out) and how many it holds (*binc_out).  Every thread of every CTA gets the same result.
template <bool DESC>
__device__ __forceinline__ int topm_crossing_bin(cooperative_groups::cluster_group& cl, int C, int* hist, int nbins, int rem,
                                                 int* red_i, int* s3, int* rem_out, int* binc_out) {
    if (C > 1) cl.sync(); else __syncthreads();
    const int tid = threadIdx.x;                         // nbins is even and <= 2 * blockDim.x
    const int b0 = 2 * tid, b1 = 2 * tid + 1;
    const int i0 = DESC ? nbins - 1 - b0 : b0, i1 = DESC ? nbins - 1 - b1 : b1;
    int h0 = 0, h1 = 0;
    if (b1 < nbins) {
        if (C > 1) {
            for (int c = 0; c < C; ++c) { const int* rh = cl.map_shared_rank(hist, c); h0 += rh[i0]; h1 += rh[i1]; }
        } else { h0 = hist[i0]; h1 = hist[i1]; }
    }
    int total;
    const int before = block_exclusive_scan(h0 + h1, red_i, &total);
    if (before < rem && rem <= before + h0) { s3[0] = i0; s3[1] = rem - before; s3[2] = h0; }
    else if (before + h0 < rem && rem <= before + h0 + h1) { s3[0] = i1; s3[1] = rem - before - h0; s3[2] = h1; }
    __syncthreads();
    *rem_out = s3[1];
    *binc_out = s3[2];
    const int b = s3[0];
    __syncthreads();
    return b;
}
__device__ __forceinline__ void topm_cx(unsigned long long& x, unsigned long long& y, bool desc) {
    const bool sw = desc ? (x < y) : (x > y);
    const unsigned long long t = x;
    x = sw ? y : x;
    y = sw ? t : y;
}

// Stages jstart, jstart / 2, .., 1 (jstart <= 64) of merge k on a warp's 128-key block: x[m] is key e = lane + 32 m of
// the block, g0 the global position of key e = lane.
__device__ __forceinline__ void topm_tail(unsigned long long (&x)[4], int g0, int lane, int k, int jstart) {
#pragma unroll
    for (int j = 64; j >= 32; j >>= 1) {
        if (j > jstart) continue;
        const int mb = j >> 5;
#pragma unroll
        for (int m = 0; m < 4; ++m)
            if ((m & mb) == 0) topm_cx(x[m], x[m | mb], ((g0 + 32 * m) & k) == 0);
    }
#pragma unroll
    for (int j = 16; j >= 1; j >>= 1) {
        if (j > jstart) continue;
        const bool lower = (lane & j) == 0;
#pragma unroll
        for (int m = 0; m < 4; ++m) {
            const unsigned long long y = __shfl_xor_sync(0xffffffffu, x[m], j);
            const bool desc = ((g0 + 32 * m) & k) == 0;
            const bool take_max = (desc == lower);
            x[m] = ((x[m] > y) == take_max) ? x[m] : y;
        }
    }
}

// rows[rho] = number of pixels of row rho (32 consecutive quads = 128 pixels of the CTA's slice) whose key is `key`
// returns how many of this thread's pixels have a larger key
__device__ __forceinline__ int topm_count_rows(const float* __restrict__ w, int q_lo, int q_hi, int N, uint32_t key, int* rows) {
    const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31;
    int n_above = 0;
    for (int qb = q_lo; qb < q_hi; qb += KT_UNROLL * T) {
        float4 v[KT_UNROLL];
#pragma unroll
        for (int u = 0; u < KT_UNROLL; ++u) {
            const int q = qb + u * T + tid;
            v[u] = (q < q_hi) ? __ldcg(reinterpret_cast<const float4*>(w) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < KT_UNROLL; ++u) {
            const int qw = qb + u * T + (tid & ~31);                 // the row's first quad: warp-uniform
            if (qw >= q_hi) break;
            const int q = qw + lane;
            const float e[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
            int c = 0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t k = f32_order_key(e[j]);
                c += (4 * q + j < N && k == key) ? 1 : 0;
                n_above += (4 * q + j < N && k > key) ? 1 : 0;
            }
            const int tot = __popc(__ballot_sync(0xffffffffu, c & 1)) + 2 * __popc(__ballot_sync(0xffffffffu, c & 2)) +
                            4 * __popc(__ballot_sync(0xffffffffu, c & 4));
            if (lane == 0) rows[(qw - q_lo) >> 5] = tot;
        }
    }
    __syncthreads();
    return n_above;
}
// rows[] -> exclusive prefix sums in place; returns the CTA's total
__device__ __forceinline__ int topm_rows_prefix(int* rows, int nrows, int* red_i) {
    const int tid = threadIdx.x, T = blockDim.x;
    const int per_t = (nrows + T - 1) / T, r0 = min(tid * per_t, nrows), r1 = min(r0 + per_t, nrows);
    int s = 0;
    for (int i = r0; i < r1; ++i) s += rows[i];
    int total;
    int ex = block_exclusive_scan(s, red_i, &total);
    for (int i = r0; i < r1; ++i) { const int c = rows[i]; rows[i] = ex; ex += c; }
    __syncthreads();
    return total;
}

__global__ void __launch_bounds__(K1_THREADS, 1)
ldp_topm_kernel(const ldp_params P, const ldp_ref_desc* __restrict__ refs, const Workspace ws,
                const ldp_outputs out, const SampleGeom G, const int C)
{
    namespace cg = cooperative_groups;
    cg::cluster_group cl = cg::this_cluster();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int hist2[2][KT_BINS];
    __shared__ int red_i[32];
    __shared__ int s3[3];
    __shared__ int s_cnt, s_tot;
    grid_dependency_sync();
    const int rank = (C > 1) ? (int)cl.block_rank() : 0;
    const int r = (int)(blockIdx.x / (unsigned)C), tid = threadIdx.x, T = blockDim.x, N = G.N, lane = tid & 31;
    const float* __restrict__ w = ws.w + (size_t)r * ws.n_pad;
    int32_t* __restrict__ sel = (out.sel_idx ? out.sel_idx : ws.sel) + (size_t)r * ws.sel_cap;
    const int M = min(P.matches_per_ref, N);
    if (refs[r].nn <= 0 || M <= 0) {                    // the same for every CTA of the cluster
        if (tid == 0 && rank == 0) { out.status[r] = (refs[r].nn <= 0) ? LDP_REF_NO_NEIGHBOURS : LDP_REF_EMPTY; out.n_samples[r] = 0; }
        return;
    }
    int n2 = 1;
    while (n2 < M) n2 <<= 1;
    const int keys_cap = max(n2 / C, min(n2, 1024));    // keys per sort buffer (same formula on the host)
    unsigned long long* cur = reinterpret_cast<unsigned long long*>(smem_raw);        // [keys_cap]
    unsigned long long* nxt = cur + keys_cap;                                         // [keys_cap], only when C > 1
    int* rows = reinterpret_cast<int*>(cur + (C > 1 ? 2 : 1) * (size_t)keys_cap);     // [nrows] tie counts per 128-pixel row
    const int N4 = (int)(ws.n_pad / 4);                 // rows are padded to a multiple of 256 floats (padding is zero)
    const int per = (((N4 + C - 1) / C) + 31) & ~31;    // quads per CTA: whole warps
    const int q_lo = min(rank * per, N4), q_hi = min(q_lo + per, N4);
    const int nrows = (q_hi - q_lo) >> 5;
    if (tid == 0) s_cnt = 0;
#ifdef LDP_PHASE_CLOCKS
    if (tid == 0 && rank == 0) ws.dbgclk[(size_t)r * 32 + 0] = clock64();
#endif
    // ---- 0. certainties saturate at the cap (w = min(certainty, cap)): if at least M pixels sit there, the M-th largest
    // key is the cap itself and nothing is strictly greater - no selection and no sort, only the ordered emission of 3b.
    const uint32_t capkey = f32_order_key(P.sample_cap);
    uint32_t kth = capkey;
    int need_eq = M;                                     // pixels with key == kth that are taken (lowest indices first)
    int before_eq = 0;                                   // tied pixels in the slices of the lower-ranked CTAs
    int pc = 0;                                          // pass counter; pass p counts into hist2[p & 1]
    int cnt_gt = topm_count_rows(w, q_lo, q_hi, N, capkey, rows);      // 0: nothing exceeds the cap
    {
        const int mine = topm_rows_prefix(rows, nrows, red_i);
        int all = mine;
        if (C > 1) {
            if (tid == 0) s_tot = mine;
            cl.sync();
            all = 0;
            for (int c = 0; c < C; ++c) { const int t = *cl.map_shared_rank(&s_tot, c); all += t; before_eq += (c < rank) ? t : 0; }
        }
        if (all < M) need_eq = -1;                       // not enough: find the M-th largest key
    }
    if (need_eq < 0) {
        // ---- 1. the M-th largest key
        uint32_t prefix = 0u, pmask = 0u;
        int rem = M, binc = 0;
        const int shifts[3] = {21, 10, 0}, widths[3] = {11, 11, 10};
        for (int pass = 0; pass < 3; ++pass, ++pc) {
            const int shift = shifts[pass], nb = 1 << widths[pass];
            int* hist = hist2[pc & 1];                  // its readers of pass pc - 2 are past the barrier of pass pc - 1
            for (int i = tid; i < KT_BINS; i += T) hist[i] = 0;
            __syncthreads();
            int ncap = 0;
            for (int qb = q_lo; qb < q_hi; qb += KT_UNROLL * T) {        // KT_UNROLL loads in flight per thread
                float4 v[KT_UNROLL];
#pragma unroll
                for (int u = 0; u < KT_UNROLL; ++u) {
                    const int q = qb + u * T + tid;
                    v[u] = (q < q_hi) ? __ldcg(reinterpret_cast<const float4*>(w) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
                for (int u = 0; u < KT_UNROLL; ++u) {
                    const int q = qb + u * T + tid;
                    if (qb + u * T + (tid & ~31) >= q_hi) break;         // warp-uniform: the row lies beyond the slice
                    const float e[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
                    int b[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const uint32_t k = f32_order_key(e[j]);
                        const bool in = (4 * q + j < N) && (k & pmask) == prefix;
                        ncap += (in && k == capkey) ? 1 : 0;               // saturated certainties: counted in a register
                        b[j] = (in && k != capkey) ? (int)((k >> shift) & (uint32_t)(nb - 1)) : -1;
                    }
                    if (pass == 0) topm_hist_add4_few(hist, b[0], b[1], b[2], b[3]);
                    else topm_hist_add4(hist, b[0], b[1], b[2], b[3]);
                }
            }
            ncap = warp_sum(ncap);
            if (lane == 0 && ncap > 0) atomicAdd(&hist[(capkey >> shift) & (uint32_t)(nb - 1)], ncap);
            const int bsel = topm_crossing_bin<true>(cl, C, hist, nb, rem, red_i, s3, &rem, &binc);
            prefix |= (uint32_t)bsel << shift;
            pmask |= (uint32_t)(nb - 1) << shift;
        }
        kth = prefix;
        need_eq = rem;
#ifdef LDP_PHASE_CLOCKS
        if (tid == 0 && rank == 0) ws.dbgclk[(size_t)r * 32 + 1] = clock64();
#endif
        // ---- 2. where the pixels tied at that key lie (they are emitted in pixel order, the first need_eq of them)
        cnt_gt = topm_count_rows(w, q_lo, q_hi, N, kth, rows);
        const int mine = topm_rows_prefix(rows, nrows, red_i);
        before_eq = 0;
        if (C > 1) {
            if (tid == 0) s_tot = mine;                  // its readers of step 0 are past the barriers of step 1
            cl.sync();
            for (int c = 0; c < rank; ++c) before_eq += *cl.map_shared_rank(&s_tot, c);
        }
    }
#ifdef LDP_PHASE_CLOCKS
    else if (tid == 0 && rank == 0) ws.dbgclk[(size_t)r * 32 + 1] = clock64();
    if (tid == 0 && rank == 0) ws.dbgclk[(size_t)r * 32 + 2] = clock64();
#endif
    // ---- 3. the n_gt keys above kth are sorted; they go (any order) into the sort buffers: the CTAs share them when
    // there are enough keys, otherwise CTA 0 sorts alone
    const int n_gt = M - need_eq;
    int n2s = 1;
    while (n2s < n_gt) n2s <<= 1;
    const int Cs = (n2s >= 128 * C) ? C : 1;
    const int L = n2s / Cs, gbase = (Cs > 1 ? rank : 0) * L;
    int logL = 0;
    while ((1 << logL) < L) ++logL;
    const bool sorter = n_gt > 0 && (Cs > 1 || rank == 0);
    if (sorter) for (int i = tid; i < L; i += T) if (gbase + i >= n_gt) cur[i] = 0ull;      // padding sorts last
    int pos = 0;
    if (n_gt > 0) {                                      // 3a. slots for this thread's keys (counted by step 2's sweep): one reservation per warp
        const int cnt = cnt_gt;
        int inc = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int n = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += n;
        }
        int base = 0;
        if (lane == 31 && inc > 0) base = atomicAdd((C > 1) ? cl.map_shared_rank(&s_cnt, 0) : &s_cnt, inc);
        base = __shfl_sync(0xffffffffu, base, 31);
        pos = base + inc - cnt;
    }
    // 3b. one sweep: keys above kth into their slots; tied pixels straight to their final place, in pixel order:
    // rows[] holds how many tied pixels precede each 128-pixel row, ballots count the ones before a lane inside the row
    for (int qb = q_lo; qb < q_hi; qb += KT_UNROLL * T) {
        float4 v[KT_UNROLL];
#pragma unroll
        for (int u = 0; u < KT_UNROLL; ++u) {
            const int q = qb + u * T + tid;
            v[u] = (q < q_hi) ? __ldcg(reinterpret_cast<const float4*>(w) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < KT_UNROLL; ++u) {
            const int qw = qb + u * T + (tid & ~31);
            if (qw >= q_hi) break;
            const int q = qw + lane;
            const float e[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
            uint32_t kk[4];
            bool eq[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                kk[j] = f32_order_key(e[j]);
                eq[j] = (4 * q + j < N) && kk[j] == kth;
            }
            const unsigned m0 = __ballot_sync(0xffffffffu, eq[0]), m1 = __ballot_sync(0xffffffffu, eq[1]),
                           m2 = __ballot_sync(0xffffffffu, eq[2]), m3 = __ballot_sync(0xffffffffu, eq[3]);
            if (m0 | m1 | m2 | m3) {
                const unsigned lt = (1u << lane) - 1u;
                int ord = before_eq + rows[(qw - q_lo) >> 5] + __popc(m0 & lt) + __popc(m1 & lt) + __popc(m2 & lt) + __popc(m3 & lt);
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (eq[j]) { if (ord < need_eq) sel[n_gt + ord] = 4 * q + j; ++ord; }
            }
            if (n_gt > 0) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if ((4 * q + j < N) && kk[j] > kth) {
                        if (pos < n_gt) {
                            const int owner = pos >> logL, li = pos & (L - 1);
                            unsigned long long* dst = (Cs > 1) ? cl.map_shared_rank(cur, owner) : ((C > 1) ? cl.map_shared_rank(cur, 0) : cur);
                            dst[li] = ((unsigned long long)kk[j] << 32) | (0xFFFFFFFFu - (uint32_t)(4 * q + j));
                        }
                        ++pos;
                    }
                }
            }
        }
    }
#ifdef LDP_PHASE_CLOCKS
    if (tid == 0 && rank == 0) ws.dbgclk[(size_t)r * 32 + 3] = clock64();
#endif
    if (tid == 0 && rank == 0) {
        out.status[r] = LDP_REF_OK;
        out.n_samples[r] = M;
        if (out.uniforms_used) out.uniforms_used[r] = 0;
        if (out.rounds) out.rounds[r] = 0;
    }
#ifdef LDP_PHASE_CLOCKS
    if (tid == 0 && rank == 0 && n_gt == 0) ws.dbgclk[(size_t)r * 32 + 4] = clock64();
#endif
    if (n_gt == 0) {                                     // every CTA of the cluster takes this exit together ...
        if (C > 1) cl.sync();                            // ... and none before the others have read its s_tot (DSMEM of an exited CTA is gone)
        return;
    }
    if (C > 1) cl.sync(); else __syncthreads();          // every key is in its slice
    if (!sorter) return;                                 // CTA 0 sorts alone: nobody touches the others' memory any more
    // ---- bitonic sort, descending, over the Cs slices (element g = rank * L + i).  Stages by partner distance j:
    //   j >= L        partner in another CTA: read over DSMEM into the second buffer;
    //   128 <= j < L  two stages (j, j / 2) per shared-memory pass, 4 keys per thread, conflict-free;
    //   j <= 64       ("tail") a warp holds a 128-key block, key e = lane + 32 m in register m of lane: stages 64 and 32
    //                 are between registers, 16..1 between lanes (shuffles) - 7 stages in one conflict-free pass, and
    //                 the whole of the merges k <= 128 in the first one.
    const bool tails = L >= 128;
    if (tails) {
        for (int blk = (tid >> 5) * 128; blk < L; blk += (T >> 5) * 128) {
            unsigned long long x[4];
#pragma unroll
            for (int m = 0; m < 4; ++m) x[m] = cur[blk + lane + 32 * m];
            const int g0 = gbase + blk + lane;
            for (int k = 2; k <= 128 && k <= n2s; k <<= 1) topm_tail(x, g0, lane, k, k >> 1);
#pragma unroll
            for (int m = 0; m < 4; ++m) cur[blk + lane + 32 * m] = x[m];
        }
        __syncthreads();
    }
    for (int k = tails ? 256 : 2; k <= n2s; k <<= 1) {
        int j = k >> 1;
        if (j >= L) {                                    // partner in another CTA (Cs > 1 only)
            cl.sync();                                   // the partner's local stages of the previous merge are done
            for (; j >= L; j >>= 1) {
                const unsigned long long* rem_buf = cl.map_shared_rank(cur, rank ^ (j >> logL));
                for (int i = tid; i < L; i += T) {
                    const int g = gbase + i;
                    const unsigned long long x = cur[i], y = rem_buf[i];
                    const bool desc = (g & k) == 0, lower = (g & j) == 0;
                    const unsigned long long mx = x > y ? x : y, mn = x > y ? y : x;
                    nxt[i] = (desc == lower) ? mx : mn;
                }
                cl.sync();                               // everybody has read `cur`; `nxt` is complete
                unsigned long long* t = cur; cur = nxt; nxt = t;
            }
        }
        const int jstop = tails ? 128 : 2;               // stages below jstop are the tail's (or the single j == 1 stage)
        while (j >= jstop) {
            if (j >= 2 * jstop || !tails) {              // stages j and j / 2 in one shared-memory pass: 4 keys per thread
                const int h = j >> 1;
                for (int p = tid; p < (L >> 2); p += T) {
                    const int i0 = ((p & ~(h - 1)) << 2) | (p & (h - 1));
                    unsigned long long a = cur[i0], b = cur[i0 + h], c = cur[i0 + j], d = cur[i0 + j + h];
                    const bool desc = ((gbase + i0) & k) == 0;
                    topm_cx(a, c, desc); topm_cx(b, d, desc);
                    topm_cx(a, b, desc); topm_cx(c, d, desc);
                    cur[i0] = a; cur[i0 + h] = b; cur[i0 + j] = c; cur[i0 + j + h] = d;
                }
                j >>= 2;
            } else {                                     // j == 128 alone
                for (int p = tid; p < (L >> 1); p += T) {
                    const int i0 = ((p & ~(j - 1)) << 1) | (p & (j - 1));
                    unsigned long long a = cur[i0], b = cur[i0 + j];
                    topm_cx(a, b, ((gbase + i0) & k) == 0);
                    cur[i0] = a; cur[i0 + j] = b;
                }
                j >>= 1;
            }
            __syncthreads();
        }
        if (tails) {
            for (int blk = (tid >> 5) * 128; blk < L; blk += (T >> 5) * 128) {
                unsigned long long x[4];
#pragma unroll
                for (int m = 0; m < 4; ++m) x[m] = cur[blk + lane + 32 * m];
                topm_tail(x, gbase + blk + lane, lane, k, 64);
#pragma unroll
                for (int m = 0; m < 4; ++m) cur[blk + lane + 32 * m] = x[m];
            }
            __syncthreads();
        } else if (j == 1) {
            for (int p = tid; p < (L >> 1); p += T) {
                const int i0 = 2 * p;
                unsigned long long a = cur[i0], b = cur[i0 + 1];
                topm_cx(a, b, ((gbase + i0) & k) == 0);
                cur[i0] = a; cur[i0 + 1] = b;
            }
            __syncthreads();
        }
    }
#ifdef LDP_PHASE_CLOCKS
    if (tid == 0 && rank == 0) ws.dbgclk[(size_t)r * 32 + 4] = clock64();
#endif
    for (int i = tid; i < L; i += T) if (gbase + i < n_gt) sel[gbase + i] = (int)(0xFFFFFFFFu - (uint32_t)(cur[i] & 0xFFFFFFFFull));
}

}  // namespace ldp
