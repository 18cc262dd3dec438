// Voxel-grid downsample on the device (SURVEY 8f row 2, reference densify.py:29-50 = Open3D's
// PointCloud::voxel_down_sample).  Open3D is not part of the reference tree or of this image: the algorithm below is
// restated from its published source (open3d/geometry/PointCloud.cpp, VoxelDownSample) and PARITY IS UNPINNED:
//   voxel_min_bound = min_bound - voxel_size / 2;  index = floor((p - voxel_min_bound) / voxel_size) per axis (f64);
//   every voxel keeps the mean of its points and of their colours, accumulated in f64 in point order.
// Open3D emits the voxels in the iteration order of a std::unordered_map (implementation-defined); here they come out
// in the order in which each voxel's first point appears.  No sort: a hash table finds the voxels, a prefix sum over the
// "first point of its voxel" flags ranks them, and each voxel's (few) points are summed in ascending point index so the
// f64 sums are the sequential ones.  Included by ldp_api.cu (unity build).
#include "ldp_device.cuh"

namespace ldp {

constexpr int KV_THREADS = 256;
constexpr unsigned long long VX_EMPTY = 0xFFFFFFFFFFFFFFFFull;

struct VoxelWs {
    double* bounds;                 // [8] min x,y,z (as doubles after the reduction), max colour, scratch
    unsigned int* bounds_u;         // [8] ordered-uint encodings while reducing: min x,y,z, max rgb, max x,y,z; [7] scratch
    unsigned long long* keys;       // [cap] voxel key per slot (VX_EMPTY = free)
    int* first;                     // [cap] smallest point index in the slot's voxel
    int* slot;                      // [n]   slot of each point
    int* flag;                      // [n]   1 if the point is the first of its voxel
    int* rank;                      // [n]   exclusive prefix of flag
    int* count;                     // [n+1] points per voxel (by rank), then exclusive prefix = segment starts
    int* cursor;                    // [n]   fill cursor per voxel
    int* seg;                       // [n]   first member of each voxel (exclusive prefix of count)
    int* members;                   // [n]   point indices grouped by voxel
    int* block_tot;                 // [ceil(n/1024)+1] scan scratch
    int* large;                     // [n+2] voxels with many points: [0] how many, [1] next to take, [2..] their ranks
    int* status;                    // [2]   0: key overflow flag, 1: number of voxels
    unsigned long long cap_mask;
};

__device__ __forceinline__ unsigned int f32_ordered(float f) {
    const unsigned int b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float f32_unordered(unsigned int k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

__global__ void __launch_bounds__(KV_THREADS)
ldp_voxel_bounds_kernel(const float* __restrict__ xyz, const float* __restrict__ rgb, long long n, VoxelWs ws)
{
    grid_dependency_sync();
    // rgb == nullptr (outlier filter): bounds_u[4 + c] = max of coordinate c instead of bounds_u[3] = max colour.  Both
    // maxima also catch a NaN with the sign bit clear; the minima catch one with it set.
    unsigned int mn[3] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu}, mx[3] = {0u, 0u, 0u};
    for (long long i = (long long)blockIdx.x * KV_THREADS + threadIdx.x; i < n; i += (long long)gridDim.x * KV_THREADS) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            mn[c] = min(mn[c], f32_ordered(xyz[3 * i + c]));
            if (rgb) mx[0] = max(mx[0], f32_ordered(rgb[3 * i + c]));
            else mx[c] = max(mx[c], f32_ordered(xyz[3 * i + c]));
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            mn[c] = min(mn[c], __shfl_xor_sync(0xffffffffu, mn[c], o));
            mx[c] = max(mx[c], __shfl_xor_sync(0xffffffffu, mx[c], o));
        }
    }
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int c = 0; c < 3; ++c) atomicMin(&ws.bounds_u[c], mn[c]);
        if (rgb) atomicMax(&ws.bounds_u[3], mx[0]);
        else for (int c = 0; c < 3; ++c) atomicMax(&ws.bounds_u[4 + c], mx[c]);
    }
}

__device__ __forceinline__ unsigned long long vx_hash(unsigned long long k) {
    k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
    return k;
}

// voxel index of every point, hash insert, smallest point index per voxel (the size is read from size_dev when given)
__global__ void __launch_bounds__(KV_THREADS)
ldp_voxel_insert_kernel(const float* __restrict__ xyz, long long n, double voxel_size, const double* __restrict__ size_dev, VoxelWs ws)
{
    grid_dependency_sync();
    const long long i = (long long)blockIdx.x * KV_THREADS + threadIdx.x;
    if (i >= n) return;
    if (size_dev) voxel_size = *size_dev;
    unsigned long long key = 0ull;
    bool bad = false;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const double vmin = (double)f32_unordered(ws.bounds_u[c]) - voxel_size * 0.5;
        const double ref = ((double)xyz[3 * i + c] - vmin) / voxel_size;
        const double fl = floor(ref);
        if (!(fl >= 0.0) || fl >= 2097152.0) bad = true;               // 21 bits per axis (also catches NaN)
        key |= (unsigned long long)(long long)(bad ? 0.0 : fl) << (21 * c);
    }
    if (bad) { atomicExch(&ws.status[0], 1); ws.slot[i] = -1; return; }
    unsigned long long h = vx_hash(key) & ws.cap_mask;
    for (;;) {
        const unsigned long long prev = atomicCAS(&ws.keys[h], VX_EMPTY, key);
        if (prev == VX_EMPTY || prev == key) break;
        h = (h + 1) & ws.cap_mask;
    }
    ws.slot[i] = (int)h;
    atomicMin(&ws.first[h], (int)i);
}

__global__ void __launch_bounds__(KV_THREADS)
ldp_voxel_flag_kernel(long long n, VoxelWs ws)
{
    grid_dependency_sync();
    const long long i = (long long)blockIdx.x * KV_THREADS + threadIdx.x;
    if (i >= n) return;
    const int s = ws.slot[i];
    ws.flag[i] = (s >= 0 && ws.first[s] == (int)i) ? 1 : 0;
}

// ---- exclusive prefix sum of n ints (three launches; the middle one is a single CTA walking the block totals)
constexpr int SC_THREADS = 1024;
__global__ void __launch_bounds__(SC_THREADS)
ldp_scan_blocks_kernel(const int* __restrict__ in, int* __restrict__ out, long long n, int* __restrict__ block_tot)
{
    __shared__ int red_i[32];
    grid_dependency_sync();
    const long long i = (long long)blockIdx.x * SC_THREADS + threadIdx.x;
    const int v = (i < n) ? in[i] : 0;
    int total;
    const int ex = block_exclusive_scan(v, red_i, &total);
    if (i < n) out[i] = ex;
    if (threadIdx.x == 0) block_tot[blockIdx.x] = total;
}
__global__ void __launch_bounds__(SC_THREADS)
ldp_scan_totals_kernel(int* __restrict__ block_tot, int nblocks, int* __restrict__ grand_total)
{
    __shared__ int red_i[32];
    __shared__ int carry;
    grid_dependency_sync();
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < nblocks; base += SC_THREADS) {
        const int i = base + threadIdx.x;
        const int v = (i < nblocks) ? block_tot[i] : 0;
        int total;
        const int ex = block_exclusive_scan(v, red_i, &total);
        const int c = carry;
        if (i < nblocks) block_tot[i] = c + ex;
        __syncthreads();
        if (threadIdx.x == 0) carry = c + total;
        __syncthreads();
    }
    if (threadIdx.x == 0 && grand_total) *grand_total = carry;
}
__global__ void __launch_bounds__(SC_THREADS)
ldp_scan_add_kernel(int* __restrict__ out, long long n, const int* __restrict__ block_tot)
{
    grid_dependency_sync();
    const long long i = (long long)blockIdx.x * SC_THREADS + threadIdx.x;
    if (i < n) out[i] += block_tot[blockIdx.x];
}

// points per voxel (indexed by the voxel's rank = number of voxels whose first point comes earlier)
__global__ void __launch_bounds__(KV_THREADS)
ldp_voxel_count_kernel(long long n, VoxelWs ws)
{
    grid_dependency_sync();
    const long long i = (long long)blockIdx.x * KV_THREADS + threadIdx.x;
    if (i >= n) return;
    const int s = ws.slot[i];
    if (s >= 0) atomicAdd(&ws.count[ws.rank[ws.first[s]]], 1);
}
// group the point indices by voxel (any order inside a voxel; the mean kernel orders them)
__global__ void __launch_bounds__(KV_THREADS)
ldp_voxel_group_kernel(long long n, VoxelWs ws, const int* __restrict__ seg_start)
{
    grid_dependency_sync();
    const long long i = (long long)blockIdx.x * KV_THREADS + threadIdx.x;
    if (i >= n) return;
    const int s = ws.slot[i];
    if (s < 0) return;
    const int v = ws.rank[ws.first[s]];
    ws.members[seg_start[v] + atomicAdd(&ws.cursor[v], 1)] = (int)i;
}
// The f64 sums run over a voxel's points in ascending point index (Open3D's loop order).  Voxels with up to
// KV_SMALL points: one thread orders the segment by insertion and sums; larger ones go to a work list for
// ldp_voxel_large_kernel (a CTA sorts the segment with a bitonic network, then one thread sums).
constexpr int KV_SMALL = 48;
__device__ __forceinline__ void voxel_emit(const float* __restrict__ xyz, const float* __restrict__ rgb, const int* m, int a, int b,
                                           bool scale, int v, float* __restrict__ xyz_out, float* __restrict__ rgb_out) {
    double sx = 0.0, sy = 0.0, sz = 0.0, sr = 0.0, sg = 0.0, sb = 0.0;
    for (int i = a; i < b; ++i) {
        const size_t p = (size_t)m[i] * 3;
        sx += (double)xyz[p]; sy += (double)xyz[p + 1]; sz += (double)xyz[p + 2];
        double r = (double)rgb[p], g = (double)rgb[p + 1], bl = (double)rgb[p + 2];
        if (scale) { r = r / 255.0; g = g / 255.0; bl = bl / 255.0; }      // densify.py:41-44: colours above 1 mean 0..255 input
        sr += r; sg += g; sb += bl;
    }
    const double cnt = (double)(b - a);
    xyz_out[3 * (size_t)v] = (float)(sx / cnt); xyz_out[3 * (size_t)v + 1] = (float)(sy / cnt); xyz_out[3 * (size_t)v + 2] = (float)(sz / cnt);
    rgb_out[3 * (size_t)v] = (float)(sr / cnt); rgb_out[3 * (size_t)v + 1] = (float)(sg / cnt); rgb_out[3 * (size_t)v + 2] = (float)(sb / cnt);
}

__global__ void __launch_bounds__(KV_THREADS)
ldp_voxel_mean_kernel(const float* __restrict__ xyz, const float* __restrict__ rgb, VoxelWs ws, const int* __restrict__ seg_start,
                      float* __restrict__ xyz_out, float* __restrict__ rgb_out)
{
    grid_dependency_sync();
    const int nv = ws.status[1];
    const int v = blockIdx.x * KV_THREADS + threadIdx.x;
    if (v >= nv) return;
    const int a = seg_start[v], b = a + ws.cursor[v];
    if (b - a > KV_SMALL) { ws.large[2 + atomicAdd(&ws.large[0], 1)] = v; return; }
    int* m = ws.members;
    for (int i = a + 1; i < b; ++i) {
        const int x = m[i];
        int j = i - 1;
        while (j >= a && m[j] > x) { m[j + 1] = m[j]; --j; }
        m[j + 1] = x;
    }
    voxel_emit(xyz, rgb, m, a, b, f32_unordered(ws.bounds_u[3]) > 1.0f, v, xyz_out, rgb_out);
}

__global__ void __launch_bounds__(SC_THREADS)
ldp_voxel_large_kernel(const float* __restrict__ xyz, const float* __restrict__ rgb, VoxelWs ws, const int* __restrict__ seg_start,
                       float* __restrict__ xyz_out, float* __restrict__ rgb_out)
{
    __shared__ int s_v;
    grid_dependency_sync();
    const int n_large = ws.large[0], tid = threadIdx.x;
    for (;;) {
        __syncthreads();
        if (tid == 0) { const int t = atomicAdd(&ws.large[1], 1); s_v = (t < n_large) ? ws.large[2 + t] : -1; }
        __syncthreads();
        const int v = s_v;
        if (v < 0) return;
        const int a = seg_start[v], len = ws.cursor[v];
        int* m = ws.members + a;
        int n2 = 1;
        while (n2 < len) n2 <<= 1;
        // ascending bitonic network with every compare-exchange in the same direction (the first step of a merge pairs
        // i with its mirror image), so the virtual +inf padding beyond len never moves
        for (int k = 2; k <= n2; k <<= 1) {
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int p = tid; p < (n2 >> 1); p += SC_THREADS) {
                    const int i = ((p & ~(j - 1)) << 1) | (p & (j - 1));
                    const int l = (j == (k >> 1)) ? (i ^ (k - 1)) : (i + j);
                    if (l < len && i < len) {
                        const int x = m[i], y = m[l];
                        if (x > y) { m[i] = y; m[l] = x; }
                    }
                }
                __syncthreads();
            }
        }
        if (tid == 0) voxel_emit(xyz, rgb, m, 0, len, f32_unordered(ws.bounds_u[3]) > 1.0f, v, xyz_out, rgb_out);
    }
}

}  // namespace ldp
