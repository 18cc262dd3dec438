// Output contract on the device (SURVEY 8a row a15, 8f row 2): the reference turns the path's float colours into
// uint8 (core/image_utils.py:24-26) and writes one struct.pack per point (core/writers.py:15-46).  Here the records
// are built where the points are - 15 bytes per vertex for the binary PLY (27 with a normal), 43 bytes per point for COLMAP's
// points3D.bin - so a caller copies n * 15 bytes to the host and appends them to the header with one write; and the
// rows a point cap keeps (densify.py:110-120; the indices stay numpy's default_rng(seed).choice on the host) are
// gathered on the device.  Included by ldp_api.cu (unity build).
#include "ldp_device.cuh"

namespace ldp {

constexpr int KO_THREADS = 256;       // points per CTA: 256 * 15, 256 * 27 and 256 * 43 bytes are multiples of 16

// np.clip(np.round(c * 255.0), 0, 255).astype(np.uint8) on a float32 colour: the product stays float32 (NEP 50),
// np.round is half-to-even
__device__ __forceinline__ uint8_t to_u8(float c) {
    const float v = rintf(__fmul_rn(c, 255.0f));
    return (uint8_t)fminf(fmaxf(v, 0.0f), 255.0f);
}
__device__ __forceinline__ void put_bytes(uint8_t* dst, const void* src, int n) {
    const uint8_t* s = reinterpret_cast<const uint8_t*>(src);
#pragma unroll
    for (int i = 0; i < 8; ++i) if (i < n) dst[i] = s[i];
}
// copies `bytes` staged bytes to out (any alignment of the total; the CTA's first byte is 16-byte aligned when the
// buffer is)
__device__ __forceinline__ void flush_records(const uint8_t* smem, uint8_t* out, int bytes, bool aligned) {
    const int tid = threadIdx.x;
    if (aligned) {
        const int nw = bytes >> 2;
        const uint32_t* s = reinterpret_cast<const uint32_t*>(smem);
        uint32_t* o = reinterpret_cast<uint32_t*>(out);
        for (int i = tid; i < nw; i += KO_THREADS) o[i] = s[i];
        for (int i = (nw << 2) + tid; i < bytes; i += KO_THREADS) out[i] = smem[i];
    } else {
        for (int i = tid; i < bytes; i += KO_THREADS) out[i] = smem[i];
    }
}

// FORMAT 0: PLY vertex  <fff BBB            (core/writers.py:44-45)
// FORMAT 1: points3D    <Q id <ddd <BBB <d  (core/writers.py:23-26; ids are first_id + i, first_id = 1 for a whole file)
// FORMAT 2: PLY vertex with a normal  <fff xyz <fff nxyz BBB (core/writers.py write_ply(..., normals=))
template <int FORMAT>
__global__ void __launch_bounds__(KO_THREADS)
ldp_records_kernel(const float* __restrict__ xyz, const float* __restrict__ rgb, const float* __restrict__ err,
                   long long n_max, const long long* __restrict__ n_dev, unsigned long long first_id,
                   uint8_t* __restrict__ out, int aligned, const float* __restrict__ nrm)
{
    constexpr int REC = (FORMAT == 0) ? 15 : (FORMAT == 1) ? 43 : 27;
    __shared__ __align__(16) uint8_t rec[KO_THREADS * REC];
    grid_dependency_sync();
    long long n = n_max;
    if (n_dev) { const long long nd = *n_dev; n = nd < n ? nd : n; }
    const long long p0 = (long long)blockIdx.x * KO_THREADS;
    if (p0 >= n) return;
    const int cnt = (int)((n - p0 < KO_THREADS) ? (n - p0) : KO_THREADS), tid = threadIdx.x;
    if (tid < cnt) {
        const long long i = p0 + tid;
        const float x = xyz[3 * i], y = xyz[3 * i + 1], z = xyz[3 * i + 2];
        const uint8_t r8 = to_u8(rgb[3 * i]), g8 = to_u8(rgb[3 * i + 1]), b8 = to_u8(rgb[3 * i + 2]);
        uint8_t* d = rec + tid * REC;
        if (FORMAT == 0) {
            put_bytes(d, &x, 4); put_bytes(d + 4, &y, 4); put_bytes(d + 8, &z, 4);
            d[12] = r8; d[13] = g8; d[14] = b8;
        } else if (FORMAT == 2) {
            const float nx = nrm[3 * i], ny = nrm[3 * i + 1], nz = nrm[3 * i + 2];
            put_bytes(d, &x, 4); put_bytes(d + 4, &y, 4); put_bytes(d + 8, &z, 4);
            put_bytes(d + 12, &nx, 4); put_bytes(d + 16, &ny, 4); put_bytes(d + 20, &nz, 4);
            d[24] = r8; d[25] = g8; d[26] = b8;
        } else {
            const unsigned long long id = first_id + (unsigned long long)i;
            const double xd = (double)x, yd = (double)y, zd = (double)z, ed = err ? (double)err[i] : 0.0;
            put_bytes(d, &id, 8); put_bytes(d + 8, &xd, 8); put_bytes(d + 16, &yd, 8); put_bytes(d + 24, &zd, 8);
            d[32] = r8; d[33] = g8; d[34] = b8;
            put_bytes(d + 35, &ed, 8);
        }
    }
    __syncthreads();
    flush_records(rec, out + p0 * REC, cnt * REC, aligned != 0);
}

__global__ void __launch_bounds__(KO_THREADS)
ldp_rgb_u8_kernel(const float* __restrict__ rgb, long long n_values, uint8_t* __restrict__ out)
{
    grid_dependency_sync();
    for (long long i = (long long)blockIdx.x * KO_THREADS + threadIdx.x; i < n_values; i += (long long)gridDim.x * KO_THREADS)
        out[i] = to_u8(rgb[i]);
}

// rows sel[0..m) of (xyz, rgb, err): xyz[sel], rgb[sel], err[sel] (densify.py:118-119)
__global__ void __launch_bounds__(KO_THREADS)
ldp_gather_rows_kernel(const float* __restrict__ xyz, const float* __restrict__ rgb, const float* __restrict__ err,
                       const long long* __restrict__ sel, long long m, long long n,
                       float* __restrict__ xyz_out, float* __restrict__ rgb_out, float* __restrict__ err_out, int* __restrict__ bad)
{
    grid_dependency_sync();
    const long long i = (long long)blockIdx.x * KO_THREADS + threadIdx.x;
    if (i >= m) return;
    long long s = sel[i];
    if (s < 0) s += n;                                   // numpy's negative indices
    if (s < 0 || s >= n) { if (bad) atomicExch(bad, 1); return; }
    xyz_out[3 * i] = xyz[3 * s]; xyz_out[3 * i + 1] = xyz[3 * s + 1]; xyz_out[3 * i + 2] = xyz[3 * s + 2];
    rgb_out[3 * i] = rgb[3 * s]; rgb_out[3 * i + 1] = rgb[3 * s + 1]; rgb_out[3 * i + 2] = rgb[3 * s + 2];
    if (err && err_out) err_out[i] = err[s];
}

// out[i, :] = src[sel[i], :] for rows of `row_floats` floats (the debug preview's subsample of matches [K,4] and
// normalised certainties [K], core/pipeline.py:577-582)
__global__ void __launch_bounds__(KO_THREADS)
ldp_gather_f32_rows_kernel(const float* __restrict__ src, int row_floats, const long long* __restrict__ sel, long long m, long long n,
                           float* __restrict__ out, int* __restrict__ bad)
{
    grid_dependency_sync();
    const long long total = m * row_floats;
    for (long long e = (long long)blockIdx.x * KO_THREADS + threadIdx.x; e < total; e += (long long)gridDim.x * KO_THREADS) {
        const long long i = e / row_floats;
        const int c = (int)(e - i * row_floats);
        long long s = sel[i];
        if (s < 0) s += n;
        if (s < 0 || s >= n) { if (bad) atomicExch(bad, 1); continue; }
        out[e] = src[s * row_floats + c];
    }
}

// Concatenation of packed point segments without a host round trip (reference core/pipeline.py:914-928: np.concatenate of
// the per-view arrays, in arrival order).  Segment q holds *count[q] points at the start of its own padded arrays
// (the outputs of one launch, or one rank's block of an all-gather); segment q's rows land at sum(count[0..q)).
// grid = (row blocks of the largest segment, segments); every CTA sums the counts before its segment itself (a few
// hundred at most), so nothing synchronises: the counts stay on the device.
__global__ void __launch_bounds__(KO_THREADS)
ldp_concat_points_kernel(const float* const* __restrict__ xyz_src, const float* const* __restrict__ rgb_src,
                         const float* const* __restrict__ err_src, const long long* const* __restrict__ count_src,
                         int n_seg, long long seg_cap, float* __restrict__ xyz_out, float* __restrict__ rgb_out,
                         float* __restrict__ err_out, long long out_cap, long long* __restrict__ seg_offset_out,
                         long long* __restrict__ total_out)
{
    __shared__ long long red[KO_THREADS / 32];
    __shared__ long long s_base;
    grid_dependency_sync();
    const int q = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    long long part = 0;
    for (int j = tid; j < q; j += KO_THREADS) { const long long c = *count_src[j]; part += (c < 0) ? 0 : (c > seg_cap ? seg_cap : c); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if (lane == 0) red[warp] = part;
    __syncthreads();
    if (tid == 0) {
        long long b = 0;
        for (int w = 0; w < KO_THREADS / 32; ++w) b += red[w];
        s_base = b;
    }
    __syncthreads();
    const long long base = s_base;
    long long cnt = *count_src[q];
    cnt = (cnt < 0) ? 0 : (cnt > seg_cap ? seg_cap : cnt);
    if (blockIdx.x == 0 && tid == 0) {
        if (seg_offset_out) {
            seg_offset_out[q] = base;
            if (q == n_seg - 1) seg_offset_out[n_seg] = base + cnt;
        }
        if (total_out && q == n_seg - 1) *total_out = (base + cnt < out_cap) ? base + cnt : out_cap;
    }
    if (base + cnt > out_cap) cnt = (out_cap > base) ? out_cap - base : 0;
    const float* __restrict__ xs = xyz_src[q];
    const float* __restrict__ rs = rgb_src[q];
    const float* __restrict__ es = err_src[q];
    const long long n3 = cnt * 3;
    // flat copies.  The sources may be a peer GPU's memory (distributed.PeerClouds: the all-gather IS this kernel), so they are
    // read 16 bytes per request when aligned, several requests in flight per thread; the destination offset (base rows) is
    // arbitrary, hence scalar stores.
    const bool vec = ((reinterpret_cast<uintptr_t>(xs) | reinterpret_cast<uintptr_t>(rs) | reinterpret_cast<uintptr_t>(es)) & 15u) == 0;
    const long long stride = (long long)gridDim.x * KO_THREADS, t0 = (long long)blockIdx.x * KO_THREADS + tid;
    if (vec) {
        const long long n3v = n3 >> 2, nev = cnt >> 2;
        constexpr int UN = 4;                              // requests in flight per thread and array (a peer read costs microseconds)
        for (long long e0 = t0; e0 < n3v; e0 += UN * stride) {
            float4 a[UN], c[UN];
#pragma unroll
            for (int u = 0; u < UN; ++u) {
                const long long e = e0 + u * stride;
                if (e < n3v) { a[u] = __ldcs(reinterpret_cast<const float4*>(xs) + e); c[u] = __ldcs(reinterpret_cast<const float4*>(rs) + e); }
            }
#pragma unroll
            for (int u = 0; u < UN; ++u) {
                const long long e = e0 + u * stride;
                if (e < n3v) {
                    float* xo = xyz_out + base * 3 + 4 * e;
                    float* ro = rgb_out + base * 3 + 4 * e;
                    xo[0] = a[u].x; xo[1] = a[u].y; xo[2] = a[u].z; xo[3] = a[u].w;
                    ro[0] = c[u].x; ro[1] = c[u].y; ro[2] = c[u].z; ro[3] = c[u].w;
                }
            }
        }
        for (long long e = (n3v << 2) + t0; e < n3; e += stride) { xyz_out[base * 3 + e] = xs[e]; rgb_out[base * 3 + e] = rs[e]; }
        for (long long e = t0; e < nev; e += stride) {
            const float4 a = __ldcs(reinterpret_cast<const float4*>(es) + e);
            float* eo = err_out + base + 4 * e;
            eo[0] = a.x; eo[1] = a.y; eo[2] = a.z; eo[3] = a.w;
        }
        for (long long e = (nev << 2) + t0; e < cnt; e += stride) err_out[base + e] = es[e];
    } else {
        for (long long e = t0; e < n3; e += stride) { xyz_out[base * 3 + e] = xs[e]; rgb_out[base * 3 + e] = rs[e]; }
        for (long long e = t0; e < cnt; e += stride) err_out[base + e] = es[e];
    }
}

// The all-gather of the ranks' point clouds as a PUSH over NVLink peer memory (distributed.PeerClouds): every rank copies its
// own rows into EVERY rank's rank-ordered cloud, at the row given by the counts of the lower ranks.  Posted remote stores
// keep the links full where remote loads wait a round trip each (measured at 8 GPUs: 0.26 ms pulling, see profiles).
// grid = (row blocks, destination ranks).  count_src[q]: device pointer to rank q's point count (peer memory for q != rank).
__global__ void __launch_bounds__(KO_THREADS)
ldp_scatter_points_kernel(const float* __restrict__ xyz, const float* __restrict__ rgb, const float* __restrict__ err,
                          const long long* const* __restrict__ count_src, int rank, int world, long long seg_cap,
                          float* const* __restrict__ xyz_dst, float* const* __restrict__ rgb_dst, float* const* __restrict__ err_dst,
                          long long out_cap, long long* __restrict__ seg_offset_out, long long* __restrict__ total_out)
{
    __shared__ long long s_cnt[64];
    grid_dependency_sync();
    const int p = blockIdx.y, tid = threadIdx.x;
    if (tid < world) { const long long c = *count_src[tid]; s_cnt[tid] = (c < 0) ? 0 : (c > seg_cap ? seg_cap : c); }
    __syncthreads();
    long long base = 0, total = 0;
    for (int q = 0; q < world; ++q) { if (q < rank) base += s_cnt[q]; total += s_cnt[q]; }
    long long cnt = s_cnt[rank];
    if (blockIdx.x == 0 && p == rank && tid == 0) {          // this rank's own bookkeeping: offsets of every rank, total
        if (seg_offset_out) {
            long long run = 0;
            for (int q = 0; q < world; ++q) { seg_offset_out[q] = run; run += s_cnt[q]; }
            seg_offset_out[world] = run;
        }
        if (total_out) *total_out = (total < out_cap) ? total : out_cap;
    }
    if (base + cnt > out_cap) cnt = (out_cap > base) ? out_cap - base : 0;
    float* __restrict__ xo = xyz_dst[p] + base * 3;
    float* __restrict__ ro = rgb_dst[p] + base * 3;
    float* __restrict__ eo = err_dst[p] + base;
    const long long stride = (long long)gridDim.x * KO_THREADS, t0 = (long long)blockIdx.x * KO_THREADS + tid;
    // 16-byte stores on the (possibly remote) destination: the destination row offset is arbitrary, so the first few floats
    // up to a 16-byte boundary and the tail go one by one; the local source is read with whatever alignment results
    auto copy = [&](const float* __restrict__ src, float* __restrict__ dst, long long n) {
        const long long head = (long long)((16u - (unsigned)(reinterpret_cast<uintptr_t>(dst) & 15u)) & 15u) >> 2;
        const long long h = head < n ? head : n;
        if (t0 < h) dst[t0] = src[t0];
        const long long nv = (n - h) >> 2;
        float4* dv = reinterpret_cast<float4*>(dst + h);
        const float* sv = src + h;
        for (long long e = t0; e < nv; e += stride) {
            const float4 v = make_float4(sv[4 * e], sv[4 * e + 1], sv[4 * e + 2], sv[4 * e + 3]);
            dv[e] = v;
        }
        for (long long e = h + (nv << 2) + t0; e < n; e += stride) dst[e] = src[e];
    };
    copy(xyz, xo, cnt * 3);
    copy(rgb, ro, cnt * 3);
    copy(err, eo, cnt);
}

}  // namespace ldp
