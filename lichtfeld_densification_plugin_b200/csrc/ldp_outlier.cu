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
// The same search with neighbour identities (NBR = true: (d^2, index) pairs, ties by index) ends in a PCA epilogue that
// gives oriented normals (ldp_estimate_normals, DESIGN.md §4.6).  Included by ldp_api.cu (unity build).
#include "ldp_device.cuh"

namespace ldp {

constexpr int OL_THREADS = 64;          // k-NN kernel: 64 threads x k list entries of shared memory (f64: <= 32 KB;
                                        // NBR, f64 + int32: <= 48 KB, the default limit)
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

// ---- oriented normals (ldp_estimate_normals; rule in include/ldp_b200.h, DESIGN.md §4.6): the k-NN kernel's NBR = true
// instantiation keeps (d^2, index) pairs and ends in this epilogue, in the same thread
struct NormalArgs {
    const float* xyz;                   // [n,3] the input: the neighbours' coordinates, gathered by index
    const float* centers;               // [n_centers,3] or NULL (no orientation)
    const int* center_idx;              // [n] or NULL (centers[0] for every point)
    float* normals;                     // [n,3]
    float* curvature;                   // [n] or NULL
    int* knn_idx;                       // [n,k] or NULL
    int n_centers;
    int pad;
};

// f64 arithmetic without contraction, on the device and on the host (where nothing contracts without FMA code generation)
__host__ __device__ __forceinline__ double nadd(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
__host__ __device__ __forceinline__ double nsub(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}
__host__ __device__ __forceinline__ double nmul(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
__host__ __device__ __forceinline__ double ndiv(double a, double b) {
#ifdef __CUDA_ARCH__
    return __ddiv_rn(a, b);
#else
    return a / b;
#endif
}

constexpr int NRM_MAX_SWEEPS = 32;      // cyclic Jacobi on 3x3 converges quadratically: a handful of sweeps in practice
constexpr double NRM_LINE = 1e-12;      // lambda1 <= NRM_LINE * lambda2: a line, the plane is not determined

// cyclic Jacobi on the symmetric 3x3 a (destroyed: its diagonal ends as the eigenvalues); v = the eigenvectors as columns.
// A rotation is skipped when |a_pq| <= 1e-20 * trace (the matrix is PSD): that perturbs an eigenvector by at most
// 1e-20 * trace / gap, far below what the f32 output resolves.
__host__ __device__ __forceinline__ void jacobi3(double a[3][3], double v[3][3]) {
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c) v[r][c] = (r == c) ? 1.0 : 0.0;
    const double tiny = 1e-20 * (fabs(a[0][0]) + fabs(a[1][1]) + fabs(a[2][2]));
    for (int sweep = 0; sweep < NRM_MAX_SWEEPS; ++sweep) {
        bool rotated = false;
#pragma unroll
        for (int pq = 0; pq < 3; ++pq) {
            const int p = (pq == 2) ? 1 : 0, q = (pq == 0) ? 1 : 2;
            const double apq = a[p][q];
            if (!(fabs(apq) > tiny)) continue;
            rotated = true;
            const double theta = (a[q][q] - a[p][p]) / (2.0 * apq);
            double t = (fabs(theta) > 1e150) ? 0.5 / theta
                                             : ((theta >= 0.0) ? 1.0 : -1.0) / (fabs(theta) + sqrt(1.0 + theta * theta));
            const double c = 1.0 / sqrt(1.0 + t * t), s = t * c;
            a[p][p] -= t * apq;
            a[q][q] += t * apq;
            a[p][q] = a[q][p] = 0.0;
            const int r = 3 - p - q;
            const double arp = a[r][p], arq = a[r][q];
            a[r][p] = a[p][r] = c * arp - s * arq;
            a[r][q] = a[q][r] = s * arp + c * arq;
#pragma unroll
            for (int m = 0; m < 3; ++m) {
                const double vp = v[m][p], vq = v[m][q];
                v[m][p] = c * vp - s * vq;
                v[m][q] = s * vp + c * vq;
            }
        }
        if (!rotated) break;
    }
}

// The rule of include/ldp_b200.h for one point x with neighbours idx[j * stride], j < k (ascending (d^2, index)):
// returns false for an undefined normal (n = 0, curvature NaN).  centre: f32 [3] or NULL.
__host__ __device__ __forceinline__ bool normal_rule(const float* __restrict__ xyz, const int* idx, int stride, int k,
                                                     const double x[3], const float* centre, double n[3], double* curv) {
    n[0] = n[1] = n[2] = 0.0;
    *curv = nan("");
    if (k < 3) return false;
    double mu[3] = {0.0, 0.0, 0.0};
    for (int j = 0; j < k; ++j) {
        const size_t e = 3 * (size_t)idx[j * stride];
#pragma unroll
        for (int a = 0; a < 3; ++a) mu[a] = nadd(mu[a], (double)xyz[e + a]);
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) mu[a] = ndiv(mu[a], (double)k);
    double c00 = 0.0, c01 = 0.0, c02 = 0.0, c11 = 0.0, c12 = 0.0, c22 = 0.0;
    for (int j = 0; j < k; ++j) {
        const size_t e = 3 * (size_t)idx[j * stride];
        const double d0 = nsub((double)xyz[e], mu[0]), d1 = nsub((double)xyz[e + 1], mu[1]), d2 = nsub((double)xyz[e + 2], mu[2]);
        c00 = nadd(c00, nmul(d0, d0)); c01 = nadd(c01, nmul(d0, d1)); c02 = nadd(c02, nmul(d0, d2));
        c11 = nadd(c11, nmul(d1, d1)); c12 = nadd(c12, nmul(d1, d2)); c22 = nadd(c22, nmul(d2, d2));
    }
    const double kd = (double)k;
    double a[3][3], v[3][3];
    a[0][0] = ndiv(c00, kd); a[0][1] = a[1][0] = ndiv(c01, kd); a[0][2] = a[2][0] = ndiv(c02, kd);
    a[1][1] = ndiv(c11, kd); a[1][2] = a[2][1] = ndiv(c12, kd); a[2][2] = ndiv(c22, kd);
    if (nadd(nadd(a[0][0], a[1][1]), a[2][2]) == 0.0) return false;          // all duplicates
    jacobi3(a, v);
    // ascending eigenvalues with their columns; constant indices only, so everything stays in registers
    double l0 = a[0][0], l1 = a[1][1], l2 = a[2][2];
    double m[3] = {v[0][0], v[1][0], v[2][0]}, m1[3] = {v[0][1], v[1][1], v[2][1]}, m2[3] = {v[0][2], v[1][2], v[2][2]};
    auto order = [](double& la, double* va, double& lb, double* vb) {
        if (!(lb < la)) return;
        const double t = la; la = lb; lb = t;
#pragma unroll
        for (int r = 0; r < 3; ++r) { const double u = va[r]; va[r] = vb[r]; vb[r] = u; }
    };
    order(l0, m, l1, m1);
    order(l1, m1, l2, m2);
    order(l0, m, l1, m1);
    if (!(l1 > NRM_LINE * l2)) return false;                                 // a line (or worse)
    const double len = sqrt(m[0] * m[0] + m[1] * m[1] + m[2] * m[2]);
    int big = 0;                                                              // canonical sign: largest |component| > 0,
    if (fabs(m[1]) > fabs(m[big])) big = 1;                                   // the lowest axis on ties
    if (fabs(m[2]) > fabs(m[big])) big = 2;
    double sgn = (m[big] < 0.0) ? -1.0 : 1.0;
    if (centre) {
        const double dot = nadd(nadd(nmul(m[0], nsub((double)centre[0], x[0])), nmul(m[1], nsub((double)centre[1], x[1]))),
                                nmul(m[2], nsub((double)centre[2], x[2])));
        if (sgn * dot < 0.0) sgn = -sgn;
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) n[r] = sgn * m[r] / len;
    *curv = l0 / (nadd(nadd(l0, l1), l2));
    return true;
}

__device__ __forceinline__ void normal_epilogue(const NormalArgs& na, int i, const double q[3], int k, const int* I, int* status)
{
    if (na.knn_idx)
        for (int j = 0; j < k; ++j) na.knn_idx[(size_t)i * k + j] = I[j * OL_THREADS];
    const float* centre = nullptr;
    if (na.centers) {
        const int ci = na.center_idx ? na.center_idx[i] : 0;
        if (ci >= 0 && ci < na.n_centers) centre = na.centers + 3 * (size_t)ci;
        else atomicOr(&status[0], 2);
    }
    double n[3], curv;
    if (!normal_rule(na.xyz, I, OL_THREADS, k, q, centre, n, &curv)) atomicAdd(&status[1], 1);
    na.normals[3 * (size_t)i] = (float)n[0];
    na.normals[3 * (size_t)i + 1] = (float)n[1];
    na.normals[3 * (size_t)i + 2] = (float)n[2];
    if (na.curvature) na.curvature[i] = (float)curv;
}

template <bool NBR>
__global__ void __launch_bounds__(OL_THREADS)
ldp_outlier_knn_kernel(const OutlierLevel* __restrict__ levels, int n_levels, long long n, int k, int max_shells,
                       double* __restrict__ mean_dist, int* __restrict__ status, NormalArgs na)
{
    extern __shared__ double s_list[];                   // [k][OL_THREADS]: entry j of this thread at s_list[j * OL_THREADS + tid]
    grid_dependency_sync();
    const long long p = (long long)blockIdx.x * OL_THREADS + threadIdx.x;
    if (p >= n) return;
    double* L = s_list + threadIdx.x;
    int* I = reinterpret_cast<int*>(s_list + (size_t)k * OL_THREADS) + threadIdx.x;   // NBR: the entries' original indices
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
        int kth_id = 0x7fffffff;                                          // NBR: I[k - 1] once the list is full
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
                        if constexpr (!NBR) {
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
                        } else {
                            // (d^2, index) pairs, lexicographic.  k duplicates of the query end the search only after the
                            // whole cell: every exact duplicate lies in the query's own cell, in atomic (not index) order
                            for (int e = cs.x; e < cs.x + cs.y; ++e) {
                                const float4 pe = lv.pts[e];
                                const double d2 = outlier_d2(q[0], q[1], q[2], pe);
                                const int id = __float_as_int(pe.w);
                                if (cnt == k && !(d2 < kth || (d2 == kth && id < kth_id))) continue;
                                int j = (cnt < k) ? cnt++ : k - 1;
                                while (j > 0 && (L[(j - 1) * OL_THREADS] > d2 ||
                                                 (L[(j - 1) * OL_THREADS] == d2 && I[(j - 1) * OL_THREADS] > id))) {
                                    L[j * OL_THREADS] = L[(j - 1) * OL_THREADS];
                                    I[j * OL_THREADS] = I[(j - 1) * OL_THREADS];
                                    --j;
                                }
                                L[j * OL_THREADS] = d2;
                                I[j * OL_THREADS] = id;
                                if (cnt == k) { kth = L[(k - 1) * OL_THREADS]; kth_id = I[(k - 1) * OL_THREADS]; }
                            }
                            if (cnt == k && kth == 0.0) done = true;
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
    if constexpr (!NBR) {
        double s = 0.0;
        for (int j = 0; j < k; ++j) s = __dadd_rn(s, __dsqrt_rn(L[j * OL_THREADS]));
        mean_dist[__float_as_int(q4.w)] = __ddiv_rn(s, (double)k);
    } else {
        normal_epilogue(na, __float_as_int(q4.w), q, k, I, status);
    }
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
