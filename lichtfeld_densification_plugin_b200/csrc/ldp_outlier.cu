// Statistical outlier removal on the device (Open3D's PointCloud::RemoveStatisticalOutliers, restated from its published
// source; PARITY UNPINNED, see include/ldp_b200.h for the rule and DESIGN.md §4.5 for the structure).
//
// The hot part is an exact k-nearest-neighbour search.  The points are grouped into a pyramid of grids built with the
// voxel filter's kernels (ldp_voxel.cu: bounds, hash insert, first-of-cell flags, scan, count, group), cell size
// h_l = h0 * 8^l, each with a cell-ordered float4 copy of the points (xyz, original index).  One thread per point, in the
// level-0 cell order, keeps a sorted list of its k smallest f64 d^2 in shared memory and visits shells of cells around its
// cell.  It skips a cell whose box distance is at least the current k-th value and stops when the k-th value is no larger
// than a lower bound on the distance to every cell not yet visited; that bound carries a margin far above the rounding of
// the cell-index computation, so the list holds exactly the k smallest distances.  After R shells without stopping the
// point starts again one level coarser; the coarsest level has at most 3 cells per axis and is searched to the end.
// Included by ldp_api.cu (unity build).
#include "ldp_device.cuh"

namespace ldp {

constexpr int OL_THREADS = 64;          // k-NN kernel: 64 threads x k f64 list entries of shared memory (<= 32 KB)
constexpr int OL_MAX_K = 64;
constexpr int OL_MAX_LEVELS = 8;        // h0 >= extent / 2^20, so h_7 >= 2 * extent: the coarsest level is never beyond 7
constexpr int OL_DEFAULT_SHELLS = 2;    // shells 0 and 1 (the query's cell and its 26 neighbours) per level
constexpr int OL_EXTEND_SHELLS = 6;     // with a full list, a level is searched on up to this many shells
constexpr int OL_CHUNK = 256;           // reductions: consecutive points per first-stage partial
constexpr int OL_FINAL = 1024;          // reductions: threads of the second stage
constexpr double OL_CELL_EPS = 1e-6;    // cell widths; the cell-index computation is off by < 1e-9 of a cell (t < 2^21)
constexpr double OL_D2_SLACK = 1.0 - 1e-9;   // relative; a computed d^2 is within 1e-15 of the exact one

struct OutlierLevel {
    const unsigned long long* keys;     // [cap] the level's hash table (ldp_voxel_insert_kernel)
    const int2* cell;                   // [cap] (first position in pts, point count) of the slot's cell
    const float4* pts;                  // [n]   xyz and original index (int bits), grouped by cell
    unsigned long long cap_mask;
    double h;                           // cell size
    double vmin[3];                     // min bound - h / 2, as the insert kernel computes it
    int gmax[3];                        // largest occupied cell index per axis
    int pad;
};

struct OutlierGrid { OutlierLevel lv[OL_MAX_LEVELS]; };

// the level descriptors into device memory, where the k-NN kernel indexes them by level
__global__ void ldp_outlier_levels_kernel(OutlierGrid g, int n_levels, OutlierLevel* __restrict__ out)
{
    grid_dependency_sync();
    for (int l = 0; l < n_levels; ++l) out[l] = g.lv[l];
}

// trial cell size for the first grid: a surface filling the bounding box would put about k/2 points in a cell
__global__ void ldp_outlier_trial_size_kernel(const unsigned int* __restrict__ bounds_u, long long n, int k_eff, double* __restrict__ h_out)
{
    grid_dependency_sync();
    double ext = 0.0;
    for (int c = 0; c < 3; ++c)
        ext = fmax(ext, (double)f32_unordered(bounds_u[4 + c]) - (double)f32_unordered(bounds_u[c]));
    double h = 1.0;
    if (ext > 0.0 && ext <= 1e300) h = fmax(ext * sqrt((double)k_eff / (2.0 * (double)n)), ext / 1048576.0);
    *h_out = h;
}

// cell[slot] = (segment start, point count) of every occupied slot of a level's hash table
__global__ void __launch_bounds__(KV_THREADS)
ldp_outlier_cells_kernel(VoxelWs ws, int2* __restrict__ cell)
{
    grid_dependency_sync();
    const long long s = (long long)blockIdx.x * KV_THREADS + threadIdx.x;
    if (s > (long long)ws.cap_mask || ws.keys[s] == VX_EMPTY) return;
    const int v = ws.rank[ws.first[s]];
    cell[s] = make_int2(ws.seg[v], ws.count[v]);
}

// cell-ordered copy of the points: pts[pos] = (xyz, index) of members[pos]
__global__ void __launch_bounds__(KV_THREADS)
ldp_outlier_pack_kernel(const float* __restrict__ xyz, long long n, const int* __restrict__ members, float4* __restrict__ pts)
{
    grid_dependency_sync();
    const long long p = (long long)blockIdx.x * KV_THREADS + threadIdx.x;
    if (p >= n) return;
    const int i = members[p];
    pts[p] = make_float4(xyz[3 * (size_t)i], xyz[3 * (size_t)i + 1], xyz[3 * (size_t)i + 2], __int_as_float(i));
}

__device__ __forceinline__ int2 outlier_find_cell(const OutlierLevel& lv, int ix, int iy, int iz) {
    const unsigned long long key = (unsigned long long)ix | ((unsigned long long)iy << 21) | ((unsigned long long)iz << 42);
    unsigned long long h = vx_hash(key) & lv.cap_mask;
    for (;;) {
        const unsigned long long k = lv.keys[h];
        if (k == key) return lv.cell[h];
        if (k == VX_EMPTY) return make_int2(0, 0);
        h = (h + 1) & lv.cap_mask;
    }
}

// d^2 = (dx*dx + dy*dy) + dz*dz in f64, no contraction
__device__ __forceinline__ double outlier_d2(double qx, double qy, double qz, float4 p) {
    const double dx = __dsub_rn((double)p.x, qx), dy = __dsub_rn((double)p.y, qy), dz = __dsub_rn((double)p.z, qz);
    return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}

// lower bound on the gap, in cell widths, between the query (at t, in cell c) and cell c + d along one axis
__device__ __forceinline__ double outlier_gap(int d, double f) {
    if (d == 0) return 0.0;
    const double g = (d > 0) ? ((double)d - f) : ((double)(-d - 1) + f);
    return fmax(g - OL_CELL_EPS, 0.0);
}

__global__ void __launch_bounds__(OL_THREADS)
ldp_outlier_knn_kernel(const OutlierLevel* __restrict__ levels, int n_levels, long long n, int k, int max_shells,
                       double* __restrict__ mean_dist, int* __restrict__ status)
{
    extern __shared__ double s_list[];                   // [k][OL_THREADS]: entry j of this thread at s_list[j * OL_THREADS + tid]
    grid_dependency_sync();
    const long long p = (long long)blockIdx.x * OL_THREADS + threadIdx.x;
    if (p >= n) return;
    double* L = s_list + threadIdx.x;
    const float4 q4 = levels[0].pts[p];
    const double q[3] = {(double)q4.x, (double)q4.y, (double)q4.z};
    int cnt = 0;
    bool done = false;
    for (int l = 0; l < n_levels && !done; ++l) {
        const OutlierLevel& lv = levels[l];
        const double h = lv.h;
        int c[3];
        double f[3], fedge = 0.5;          // distance of the query to the nearest face of its cell
#pragma unroll
        for (int a = 0; a < 3; ++a) {                    // the insert kernel's own expression: the query's cell is its key
            const double t = (q[a] - lv.vmin[a]) / h;
            const double fl = floor(t);
            c[a] = (int)fl;
            f[a] = t - fl;
            fedge = fmin(fedge, fmin(f[a], 1.0 - f[a]));
        }
        int R = (l == n_levels - 1) ? 0x7fffffff : max_shells;
        cnt = 0;                                         // a coarser level starts over (no candidate is counted twice)
        double kth = __longlong_as_double(0x7ff0000000000000ll);     // +inf; L[k - 1] once the list is full
        for (int r = 0; r < R && !done; ++r) {
            for (int dx = -r; dx <= r && !done; ++dx) {
                const int ix = c[0] + dx;
                if (ix < 0 || ix > lv.gmax[0]) continue;
                const double gx = outlier_gap(dx, f[0]);
                for (int dy = -r; dy <= r && !done; ++dy) {
                    const int iy = c[1] + dy;
                    if (iy < 0 || iy > lv.gmax[1]) continue;
                    const double gy = outlier_gap(dy, f[1]);
                    const bool edge = (dx == -r || dx == r || dy == -r || dy == r);
                    const int step = (edge || r == 0) ? 1 : 2 * r;     // inside the shell's x/y faces only dz = -r, r
                    for (int dz = -r; dz <= r && !done; dz += step) {
                        const int iz = c[2] + dz;
                        if (iz < 0 || iz > lv.gmax[2]) continue;
                        if (cnt == k) {
                            const double gz = outlier_gap(dz, f[2]);
                            const double box = __dmul_rn(__dmul_rn(h, h), __dadd_rn(__dadd_rn(__dmul_rn(gx, gx), __dmul_rn(gy, gy)), __dmul_rn(gz, gz)));
                            if (__dmul_rn(box, OL_D2_SLACK) >= kth) continue;
                        }
                        const int2 cs = outlier_find_cell(lv, ix, iy, iz);
                        for (int e = cs.x; e < cs.x + cs.y; ++e) {
                            const double d2 = outlier_d2(q[0], q[1], q[2], lv.pts[e]);
                            if (cnt == k && !(d2 < kth)) continue;
                            int j = (cnt < k) ? cnt++ : k - 1;
                            while (j > 0 && L[(j - 1) * OL_THREADS] > d2) { L[j * OL_THREADS] = L[(j - 1) * OL_THREADS]; --j; }
                            L[j * OL_THREADS] = d2;
                            if (cnt == k) {
                                kth = L[(k - 1) * OL_THREADS];
                                if (kth == 0.0) { done = true; break; }            // k duplicates: nothing can come closer
                            }
                        }
                    }
                }
            }
            if (done) break;
            // every occupied cell visited, or the k-th distance no larger than the distance to the unvisited cells
            if (c[0] - r <= 0 && c[0] + r >= lv.gmax[0] && c[1] - r <= 0 && c[1] + r >= lv.gmax[1] &&
                c[2] - r <= 0 && c[2] + r >= lv.gmax[2]) { done = true; break; }
            if (cnt == k) {
                const double b = __dmul_rn(h, __dsub_rn(__dadd_rn((double)r, fedge), OL_CELL_EPS));
                if (b > 0.0 && kth <= __dmul_rn(__dmul_rn(b, b), OL_D2_SLACK)) { done = true; break; }
                // a full list bounds the radius still to search: when a few more shells of this level cover it, stay (the
                // cells beyond the k-th distance are skipped before their lookup) rather than rescan 8x coarser cells
                if (r == R - 1) {
                    const double need = sqrt(kth) / h - fedge + 2.0 * OL_CELL_EPS;
                    if (need < (double)OL_EXTEND_SHELLS) R = max(R, (int)ceil(need) + 1);
                }
            }
        }
        if (!done && l == 0) atomicAdd(&status[2], 1);
    }
    double s = 0.0;
    for (int j = 0; j < k; ++j) s = __dadd_rn(s, __dsqrt_rn(L[j * OL_THREADS]));
    mean_dist[__float_as_int(q4.w)] = __ddiv_rn(s, (double)k);
}

// ---- the two sums of the threshold, in a fixed order (include/ldp_b200.h): stage 1 sums OL_CHUNK consecutive points
// sequentially; stage 2 (one CTA) lets thread t sum partials t, t + OL_FINAL, ... sequentially, then halves the
// OL_FINAL results pairwise (v[t] += v[t + s], s = 512, 256, ..., 1).  Terms of points with m_i <= 0 are skipped.
__global__ void __launch_bounds__(KV_THREADS)
ldp_outlier_partial_kernel(const double* __restrict__ m, long long n, const double* __restrict__ mean, double* __restrict__ part)
{
    grid_dependency_sync();
    const long long t = (long long)blockIdx.x * KV_THREADS + threadIdx.x;
    const long long a = t * OL_CHUNK;
    if (a >= n) return;
    const long long b = (a + OL_CHUNK < n) ? a + OL_CHUNK : n;
    const double mu = mean ? *mean : 0.0;
    double s = 0.0;
    for (long long i = a; i < b; ++i) {
        const double v = m[i];
        if (!(v > 0.0)) continue;
        if (mean) { const double d = __dsub_rn(v, mu); s = __dadd_rn(s, __dmul_rn(d, d)); }
        else s = __dadd_rn(s, v);
    }
    part[t] = s;
}

// stage 2; second == 0: stats[0] = mean = S / n.  second == 1: stats[1] = std = sqrt(Q / (n - 1)), stats[2] = mean + ratio * std
__global__ void __launch_bounds__(OL_FINAL)
ldp_outlier_stats_kernel(const double* __restrict__ part, long long n_part, long long n, double ratio, int second, double* __restrict__ stats)
{
    __shared__ double v[OL_FINAL];
    grid_dependency_sync();
    const int t = threadIdx.x;
    double s = 0.0;
    for (long long j = t; j < n_part; j += OL_FINAL) s = __dadd_rn(s, part[j]);
    v[t] = s;
    __syncthreads();
    for (int h = OL_FINAL / 2; h > 0; h >>= 1) {
        if (t < h) v[t] = __dadd_rn(v[t], v[t + h]);
        __syncthreads();
    }
    if (t != 0) return;
    if (!second) { stats[0] = __ddiv_rn(v[0], (double)n); return; }
    const double sd = __dsqrt_rn(__ddiv_rn(v[0], (double)(n - 1)));
    stats[1] = sd;
    stats[2] = __dadd_rn(stats[0], __dmul_rn(ratio, sd));
}

__global__ void __launch_bounds__(KV_THREADS)
ldp_outlier_flag_kernel(const double* __restrict__ m, long long n, const double* __restrict__ stats, int* __restrict__ flag)
{
    grid_dependency_sync();
    const long long i = (long long)blockIdx.x * KV_THREADS + threadIdx.x;
    if (i >= n) return;
    const double v = m[i];
    flag[i] = (v > 0.0 && v < stats[2]) ? 1 : 0;
}

__global__ void __launch_bounds__(KV_THREADS)
ldp_outlier_kept_kernel(const int* __restrict__ flag, const int* __restrict__ rank, long long n, long long* __restrict__ kept_idx)
{
    grid_dependency_sync();
    const long long i = (long long)blockIdx.x * KV_THREADS + threadIdx.x;
    if (i < n && flag[i]) kept_idx[rank[i]] = i;
}

}  // namespace ldp
