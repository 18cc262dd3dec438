// Internal device-side helpers shared by the densification kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/ldp_b200.h"

namespace ldp {

// ---------------------------------------------------------------------------------------------
// Workspace carved by the host (ldp_api.cu).  Everything is per reference view r; rows are padded so
// that float4 / 16-byte accesses stay aligned.
// ---------------------------------------------------------------------------------------------
struct RefStat {        // per-view scalars passed between the sampler kernels
    float s;            // f32 normaliser (core/sampling.py:26)
    int npos;           // number of p > 0
    int emin_inv;       // max over positive p of (255 - biased exponent); 0: no positive p (zero-initialisable, atomicMax)
    int bad;            // bit0 NaN weight, bit1 negative weight, bit2 no neighbours
};

struct Workspace {
    float* w;            // [R][n_pad]   stream: capped, border-masked weights; prep: overwritten by p = w / s
                         //              (zeroed as pixels get drawn)
    uint8_t* bestk;      // [R][n_pad]   winning neighbour per pixel
    uint32_t* bitmap;    // [R][n_words] selected-pixel bitmap
    uint32_t* gone;      // [R][n_words] the bitmap as the first draw round left it: those pixels weigh nothing afterwards
    int32_t* found;      // [R][draw_cmax][found_cap] pixel indices: per-CTA find lists of the current round
    int32_t* fcnt;       // [R][draw_cmax] entries in each list
    int32_t* sel;        // [R][sel_cap]  sample indices when the caller does not ask for them
    float4* pt0;         // [R][sel_cap]  X,Y,Z,err per sample
    float4* pt1;         // [R][sel_cap]  r,g,b,debug-cert per sample
    float4* dbgm;        // [R][sel_cap]  clipped match coords per sample (collect_debug)
    uint8_t* flags;      // [R][sel_cap]  bit0 keep, bit1 sampson-pass, bits2.. group
    int32_t* kept;       // [R]           kept points (atomic)
    unsigned long long* topk_keys;  // [R][topk_cap] no_filter candidate keys
    double* csum;        // [R][nchunk_pad] f64 sums of p per chunk
    double* csum0;       // [R][nchunk_pad] the same sums, written by the prep kernel and never modified: what the first draw round
                         //   searches.  Its independent CTAs start whenever an SM is free - also after their siblings have removed
                         //   their first finds from csum - and numpy's first round draws from the cdf of ALL weights
    double* partial;     // [R][nblk]    per-CTA f64 partial weight sums of the stream kernel
    int32_t* bflags;     // [R][nblk]    per-CTA NaN / negative flags
    RefStat* rstat;      // [R]
    unsigned long long* gbins;      // [R][bins_cap] per-tile arg-max keys (p bits << 32 | ~index)
    int32_t* blk_cnt;    // [R][nb2][LDP_MAX_NN] kept samples per 128-sample tile and group (geometry -> pack)
    int32_t* blk_first;  // [R][nb2][LDP_MAX_NN] first sample position per tile and group
    int2* fix_list;      // [R*sel_cap] (view, sample) pairs whose null-vector iteration did not converge
    int32_t* fix_count;  // [1]          entries in fix_list
    int32_t* dstat;      // [R] verdict of the first draw round for the rounds that follow: fail code | inexact << 8
    long long* dbgclk;   // [R][32] phase timestamps of the draw kernel (written only with -DLDP_PHASE_CLOCKS)
    size_t n_pad, n_words, found_cap, sel_cap, topk_cap, nchunk_pad, nblk, bins_cap, draw_cmax;
    // multiview launches only (NULL otherwise)
    int32_t* vmask;      // [R][sel_cap]  neighbour slots that contributed to the kept sample's point (geometry / fix -> pack)
    float4* mvrec;       // [R][sel_cap] winner's warp row of a kept sample whose multi-view solve did not converge (its
                         //   winner slot waits in vmask, its two-view result in pt0 / pt1 for the fix-up to fall back to)
};

struct SampleGeom {     // launch-constant shape of the sampler
    int N;              // H*W
    int chunk_shift;    // log2(pixels per chunk)
    int nchunk;
    int tile;           // max(1, W / tiles)
    int nbx, nby, nbins;
    int size;           // min(int(0.85*M), N)
    int cov_budget;     // max(1, M - size)
    int vec;            // cert planes are 16-B aligned and W % 4 == 0
    int prep_lb_cap;    // local tile bins per CTA of the prep kernel
    unsigned long long w_magic;   // ceil(2^40 / W): floor(n / W) = (n * w_magic) >> 40 for n < 2^21 * ...
    unsigned long long t_magic;   // ceil(2^40 / tile)
    uint32_t t_magic32;           // ceil(2^32 / tile) (0 for tile 1): floor(n / tile) = umulhi(n, t_magic32) for n * tile < 2^32
    int step_dx, step_dy;         // (KS_THREADS * 4) % W, (KS_THREADS * 4) / W: pixel step of the full-grid passes
    int draw_ept;       // draw kernel: chunk-table entries per thread (multiple of 8)
    int draw_pre_cap;   // draw kernel: doubles in the padded prefix table
    int draw_ng;        // draw kernel: guide-table buckets
    int draw_smem_bytes; // draw kernel: dynamic shared memory of the launch
};

// ---------------------------------------------------------------------------------------------
// Programmatic dependent launch (ldp_api.cu:launch_k): wait until the previous kernel of the stream has completed and
// its memory is visible, then allow the NEXT kernel's CTAs to be scheduled as soon as all CTAs of this grid are resident.
// Must precede the first access to anything another kernel of the stream writes or reads.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void grid_dependency_sync() {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

// ---------------------------------------------------------------------------------------------
// warp / block collectives (fixed reduction trees => run-to-run deterministic)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int warp_min(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// All threads get the block total.  scratch: >= 32 elements of T in shared memory.
template <typename T>
__device__ __forceinline__ T block_sum(T v, T* scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) scratch[warp] = v;
    __syncthreads();
    T r = (lane < nw) ? scratch[lane] : T(0);
    return warp_sum(r);
}
// block-wide maximum of a float (all threads get it)
__device__ __forceinline__ float block_sum_max(float v, float* scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    __syncthreads();
    if (lane == 0) scratch[warp] = v;
    __syncthreads();
    float r = (lane < nw) ? scratch[lane] : -3.0e38f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) r = fmaxf(r, __shfl_xor_sync(0xffffffffu, r, o));
    return r;
}
__device__ __forceinline__ int block_min(int v, int* scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_min(v);
    __syncthreads();
    if (lane == 0) scratch[warp] = v;
    __syncthreads();
    int r = (lane < nw) ? scratch[lane] : 0x7fffffff;
    return warp_min(r);
}

// Exclusive scan of one value per thread; *total receives the block sum.  scratch >= 32 elements.
template <typename T>
__device__ __forceinline__ T block_exclusive_scan(T v, T* scratch, T* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    T inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        T n = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += n;
    }
    __syncthreads();
    if (lane == 31) scratch[warp] = inc;
    __syncthreads();
    T wv = (lane < nw) ? scratch[lane] : T(0);
    T winc = wv;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        T n = __shfl_up_sync(0xffffffffu, winc, o);
        if (lane >= o) winc += n;
    }
    T wexc = winc - wv;
    T base = __shfl_sync(0xffffffffu, wexc, warp);
    *total = __shfl_sync(0xffffffffu, winc, 31);
    return base + inc - v;
}

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 counter-based generator (Salmon et al. 2011), used for the production uniforms.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                              uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// The d-th double of stream `stream`: 53-bit construction identical to numpy's random_sample
// ((a >> 5) * 2^26 + (b >> 6)) / 2^53, so explicit and Philox streams have the same lattice.
__device__ __forceinline__ double philox_uniform(uint64_t seed, uint32_t stream, uint32_t d) {
    uint32_t r[4];
    philox4x32_10(d >> 1, 0u, stream, 0x4c445031u, (uint32_t)seed, (uint32_t)(seed >> 32), r);
    const uint32_t a = (d & 1u) ? r[2] : r[0], b = (d & 1u) ? r[3] : r[1];
    return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) * (1.0 / 9007199254740992.0);
}

// ---------------------------------------------------------------------------------------------
// Certainty post-processing between the matcher and the path (reference core/pipeline.py:405-430), applied on the
// fly wherever a raw certainty value is read when ldp_params.prologue is set.
// ---------------------------------------------------------------------------------------------
struct ProView {            // per-view constants, staged in shared memory
    const uint8_t* mask_a;
    const uint8_t* mask_b[LDP_MAX_NN];
    const float* warp[LDP_MAX_NN];
    int mask_w, mask_h;
    float msx, msy;
};
__device__ __forceinline__ void stage_proview(const ldp_ref_desc* rd, ProView& pv, int t) {
    if (t < LDP_MAX_NN) { pv.mask_b[t] = rd->mask_b[t]; pv.warp[t] = rd->warp[t]; }
    if (t == 0) { pv.mask_a = rd->mask_a; pv.mask_w = rd->mask_w; pv.mask_h = rd->mask_h; pv.msx = rd->mask_sx; pv.msy = rd->mask_sy; }
}
// mask value at map pixel (ix, iy): F.interpolate(mode="nearest") to the map size, then .float()
__device__ __forceinline__ float mask_at(const uint8_t* __restrict__ m, int ix, int iy, const ProView& pv) {
    const int mx = min((int)floorf(__fmul_rn((float)ix, pv.msx)), pv.mask_w - 1);
    const int my = min((int)floorf(__fmul_rn((float)iy, pv.msy)), pv.mask_h - 1);
    return (float)__ldg(m + (size_t)my * pv.mask_w + mx);
}
// certainty of neighbour k at pixel px = (x, y) after clamp(min), x maskA, x grid_sample(maskB, warp[..., 2:4])
__device__ __forceinline__ float prologue_cert(float c, int k, int px, int x, int y, const ldp_params& P, const ProView& pv) {
    c = (c < P.certainty_floor) ? P.certainty_floor : c;                       // torch.clamp(min=): NaN stays NaN
    if (pv.mask_a) c = __fmul_rn(c, mask_at(pv.mask_a, x, y, pv));
    if (pv.mask_b[k]) {
        const float2 g = __ldg(reinterpret_cast<const float2*>(pv.warp[k] + (size_t)px * 4 + 2));
        // grid_sampler un-normalise (align_corners=False): (g + 1) * (size / 2) - 0.5, then nearbyint
        const float fx = rintf(__fsub_rn(__fmul_rn(__fadd_rn(g.x, 1.f), 0.5f * (float)P.W), 0.5f));
        const float fy = rintf(__fsub_rn(__fmul_rn(__fadd_rn(g.y, 1.f), 0.5f * (float)P.H), 0.5f));
        float m = 0.f;                                                         // padding_mode="zeros"; NaN coordinates fall outside
        if (fx > -1.f && fx < (float)P.W && fy > -1.f && fy < (float)P.H) m = mask_at(pv.mask_b[k], (int)fx, (int)fy, pv);
        c = __fmul_rn(c, m);
    }
    return c;
}

#ifdef LDP_PHASE_CLOCKS
#define LDP_CLK(ws, r, slot) do { if (threadIdx.x == 0 && (blockIdx.x % cooperative_groups::this_cluster().num_blocks()) == 0) (ws).dbgclk[(size_t)(r) * 32 + (slot)] = clock64(); } while (0)
#else
#define LDP_CLK(ws, r, slot) do { } while (0)
#endif

// Two consecutive draws (d even, d + 1) from ONE Philox call.
__device__ __forceinline__ void philox_uniform2(uint64_t seed, uint32_t stream, uint32_t d, double u[2]) {
    uint32_t r[4];
    philox4x32_10(d >> 1, 0u, stream, 0x4c445031u, (uint32_t)seed, (uint32_t)(seed >> 32), r);
    u[0] = ((double)(r[0] >> 5) * 67108864.0 + (double)(r[1] >> 6)) * (1.0 / 9007199254740992.0);
    u[1] = ((double)(r[2] >> 5) * 67108864.0 + (double)(r[3] >> 6)) * (1.0 / 9007199254740992.0);
}

// Slice i of n of [base, base + bytes) -> L2, as one bulk prefetch (whole 16-byte units inside the array only).  The sampled pixels
// of a view touch most sectors of its reference image and of its winner row in random order; read that way they are DRAM row
// misses, read once front to back they are a few hundred KB of streaming that the view's CTAs then hit in L2.
__device__ __forceinline__ void l2_prefetch_slice(const void* base, size_t bytes, int i, int n) {
    const size_t chunk = ((bytes + n - 1) / n + 15) & ~(size_t)15;
    const uintptr_t b0 = reinterpret_cast<uintptr_t>(base);
    const uintptr_t lo = (b0 + (size_t)i * chunk + 15) & ~(uintptr_t)15;
    uintptr_t hi = b0 + (size_t)(i + 1) * chunk;
    if (hi > b0 + bytes) hi = b0 + bytes;
    hi &= ~(uintptr_t)15;
    if (hi > lo) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" :: "l"(lo), "r"((uint32_t)(hi - lo)) : "memory");
}

__device__ __forceinline__ float4 ld_stream4(const float* p) {   // read-once data: evict-first
    return __ldcs(reinterpret_cast<const float4*>(p));
}

}  // namespace ldp
