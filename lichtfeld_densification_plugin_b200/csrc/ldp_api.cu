// C ABI of the densification path (include/ldp_b200.h).  Unity build: the kernels live in the two
// included translation units; this file carves the workspace, picks launch geometry and enqueues.
#include <cstdio>
#include <cmath>
#include <cstring>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "ldp_sample.cu"
#include "ldp_geometry.cu"
#include "ldp_output.cu"
#include "ldp_select.cu"
#include "ldp_voxel.cu"
#include "ldp_outlier.cu"
#include "ldp_consistency.cu"
#include "ldp_fusion.cu"

namespace {

thread_local std::string g_last_error;
thread_local int g_launches = 0;

// ---- optional per-kernel timing (ldp_profile_enable / ldp_profile_read)
constexpr int MAX_PROF = 64;
thread_local bool g_prof_on = false;
thread_local cudaEvent_t g_prof_ev[2 * MAX_PROF];
thread_local bool g_prof_ev_ready = false;
thread_local int g_prof_n = 0;

thread_local const char* g_prof_name[MAX_PROF];

struct KernelTimer {
    cudaStream_t st;
    int slot;
    KernelTimer(cudaStream_t s, const char* name) : st(s), slot(-1) {
        if (!g_prof_on || g_prof_n >= MAX_PROF) return;
        if (!g_prof_ev_ready) {
            for (int i = 0; i < 2 * MAX_PROF; ++i) cudaEventCreate(&g_prof_ev[i]);
            g_prof_ev_ready = true;
        }
        slot = g_prof_n++;
        g_prof_name[slot] = name;
        cudaEventRecord(g_prof_ev[2 * slot], st);
    }
    ~KernelTimer() { if (slot >= 0) cudaEventRecord(g_prof_ev[2 * slot + 1], st); }
};

// First statement of every entry point that enqueues work: ldp_last_launch_count and the profile describe that call alone.
void begin_call() {
    g_launches = 0;
    g_prof_n = 0;
}

int fail(int code, const char* what) {
    g_last_error = what ? what : "";
    return code;
}
// Drops the error a failed runtime call left in this thread's last-error slot, so that a later, unrelated check (the
// caller's own, e.g. torch's after its next launch) does not report it again.
void clear_last_error() { (void)cudaGetLastError(); }
int cuda_fail(cudaError_t e, const char* where) {
    clear_last_error();
    g_last_error = std::string(where) + ": " + cudaGetErrorString(e);
    return LDP_ERR_CUDA;
}
int check(cudaError_t e, const char* where) { return e == cudaSuccess ? LDP_OK : cuda_fail(e, where); }

constexpr int MAX_DEVICES = 64;
int current_device() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { clear_last_error(); dev = 0; }
    return (dev >= 0 && dev < MAX_DEVICES) ? dev : 0;
}

// per device (a process may drive several, possibly different, GPUs) and per calling thread: no shared mutable state
int max_active_clusters(int csize, size_t smem) {
    thread_local int cache_all[MAX_DEVICES][9] = {};
    thread_local size_t cache_smem_all[MAX_DEVICES] = {};
    const int dev = current_device();
    int* cache = cache_all[dev];
    size_t& cache_smem = cache_smem_all[dev];
    if (cache_smem != smem) { for (int i = 0; i < 9; ++i) cache[i] = 0; cache_smem = smem; }
    if (cache[csize]) return cache[csize];
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(csize * 64));
    cfg.blockDim = dim3(ldp::KD_THREADS);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)csize;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, ldp::ldp_draw_kernel<2>, &cfg) != cudaSuccess) { clear_last_error(); n = 0; }
    cache[csize] = n > 0 ? n : -1;
    return cache[csize];
}

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

int g_force_cluster = 0;      // test hook (ldp_debug_set_cluster)
int g_force_fix_two = 0, g_force_fix_mv = 0;   // test hook (ldp_debug_force_fixup)
int g_sm_reserve = 0;         // ldp_set_sm_reserve
int g_last_cluster = 0;

int sm_count() {          // of the CURRENT device
    thread_local int cached[MAX_DEVICES] = {};
    const int dev = current_device();
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) cached[dev] = n;
        else { clear_last_error(); cached[dev] = 148; }
    }
    return cached[dev];
}

constexpr size_t K1_SMEM_BUDGET = 200 * 1024;
constexpr size_t PREP_SMEM_MAX = 64 * 1024;

// Every kernel is launched with programmatic dependent launch allowed: its CTAs may be scheduled while the previous
// kernel of the stream drains, and block in griddepcontrol.wait (ldp_device.cuh:grid_dependency_sync) until that kernel's
// memory is visible.  Hides the launch latency at each of the 6 kernel boundaries of a step.
// cluster > 0: the grid is launched as thread-block clusters of that many CTAs along x.
template <typename... KArgs, typename... Args>
cudaError_t launch_k(int cluster, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    attr[1].id = cudaLaunchAttributeClusterDimension;
    attr[1].val.clusterDim.x = (unsigned)cluster;
    attr[1].val.clusterDim.y = 1;
    attr[1].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = cluster > 0 ? 2 : 1;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// What the launch returned, counted in ldp_last_launch_count; a failure is reported under the kernel's name.
int launched(cudaError_t e, const char* name) {
    ++g_launches;
    return check(e, name);
}
template <typename... KArgs, typename... Args>
int launch(const char* name, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    return launched(launch_k(0, kernel, grid, block, smem, st, std::forward<Args>(args)...), name);
}

// A kernel launched as thread-block clusters: launch_at(c) enqueues it with clusters of c CTAs.  A size the device cannot
// schedule (odd sizes may not be) falls back to the largest power of two below it.  The size launched is what
// ldp_debug_last_cluster reports.
template <typename LaunchAt>
int launch_cluster(const char* name, int csize, LaunchAt launch_at) {
    cudaError_t e;
    while ((e = launch_at(csize)) != cudaSuccess && csize > 1) {
        clear_last_error();
        csize = csize > 4 ? 4 : (csize > 2 ? 2 : 1);
    }
    g_last_cluster = csize;
    return launched(e, name);
}

// ---- instantiations the host picks from
// [prologue mode][nn_max].  Mode 0: processed certainty planes; 1: raw matcher planes and no neighbour mask anywhere (no
// warp row is read); 2: raw planes whose post-processing samples the neighbour masks through the warp.  An nn_max outside
// the unrolled ones (0 = unknown) takes the generic <0, mode>.
using StreamKernel = decltype(&ldp::ldp_stream_kernel<0, 0>);
const StreamKernel k_stream[3][9] = {
    {ldp::ldp_stream_kernel<0, 0>, ldp::ldp_stream_kernel<1, 0>, ldp::ldp_stream_kernel<2, 0>, ldp::ldp_stream_kernel<3, 0>,
     ldp::ldp_stream_kernel<4, 0>, ldp::ldp_stream_kernel<5, 0>, ldp::ldp_stream_kernel<6, 0>, ldp::ldp_stream_kernel<7, 0>,
     ldp::ldp_stream_kernel<8, 0>},
    {ldp::ldp_stream_kernel<0, 1>, ldp::ldp_stream_kernel<1, 1>, ldp::ldp_stream_kernel<2, 1>, ldp::ldp_stream_kernel<3, 1>,
     ldp::ldp_stream_kernel<4, 1>, ldp::ldp_stream_kernel<0, 1>, ldp::ldp_stream_kernel<0, 1>, ldp::ldp_stream_kernel<0, 1>,
     ldp::ldp_stream_kernel<0, 1>},
    {ldp::ldp_stream_kernel<0, 2>, ldp::ldp_stream_kernel<1, 2>, ldp::ldp_stream_kernel<2, 2>, ldp::ldp_stream_kernel<3, 2>,
     ldp::ldp_stream_kernel<4, 2>, ldp::ldp_stream_kernel<0, 2>, ldp::ldp_stream_kernel<0, 2>, ldp::ldp_stream_kernel<0, 2>,
     ldp::ldp_stream_kernel<0, 2>},
};
// [chunk_shift 5, 6, 7, other][PrepCols]
using ldp::PrepCols;
using PrepKernel = decltype(&ldp::ldp_prep_kernel<5, PrepCols::CONST>);
const PrepKernel k_prep[4][3] = {
    {ldp::ldp_prep_kernel<5, PrepCols::CONST>, ldp::ldp_prep_kernel<5, PrepCols::QUAD>, ldp::ldp_prep_kernel<5, PrepCols::PIXEL>},
    {ldp::ldp_prep_kernel<6, PrepCols::CONST>, ldp::ldp_prep_kernel<6, PrepCols::QUAD>, ldp::ldp_prep_kernel<6, PrepCols::PIXEL>},
    {ldp::ldp_prep_kernel<7, PrepCols::CONST>, ldp::ldp_prep_kernel<7, PrepCols::QUAD>, ldp::ldp_prep_kernel<7, PrepCols::PIXEL>},
    {ldp::ldp_prep_kernel<0, PrepCols::CONST>, ldp::ldp_prep_kernel<0, PrepCols::QUAD>, ldp::ldp_prep_kernel<0, PrepCols::PIXEL>},
};

// Raises the dynamic shared memory limit of every kernel that takes more than the default 48 KB, once per device (a
// process may drive several).  Threads that make their first call at the same time wait for one configuration.
int configure_device() {
    static std::once_flag once[MAX_DEVICES];
    static cudaError_t result[MAX_DEVICES];
    const int dev = current_device();
    std::call_once(once[dev], [dev] {
        cudaError_t e = cudaSuccess;
        auto raise = [&e](const void* kernel, size_t bytes) {
            if (e == cudaSuccess) e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        };
        raise((const void*)ldp::ldp_draw_kernel<1>, K1_SMEM_BUDGET);
        raise((const void*)ldp::ldp_draw_kernel<2>, K1_SMEM_BUDGET);
        for (const auto& row : k_prep)
            for (PrepKernel k : row) raise((const void*)k, PREP_SMEM_MAX);
        raise((const void*)ldp::ldp_topm_kernel, K1_SMEM_BUDGET);
        raise((const void*)ldp::ldp_kcenters_kernel<true>, K1_SMEM_BUDGET);
        result[dev] = e;
    });
    return check(result[dev], "cudaFuncSetAttribute");
}

// Bump allocator over a workspace: consecutive blocks, the offset rounded up to `align` bytes after each; base = nullptr
// only measures.
struct Carver {
    char* base;
    size_t off = 0;
    template <typename T>
    T* take(size_t count, size_t align = 256) {
        T* q = base ? reinterpret_cast<T*>(base + off) : nullptr;
        off = align_up(off + count * sizeof(T), align);
        return q;
    }
};

struct Plan {
    ldp::Workspace ws;
    ldp::SampleGeom geom;
    size_t bytes;
    size_t k1_smem;
    size_t prep_smem;
    int nb2;
    void* zero_base;        // launch state that every call clears with ONE memset: counters, per-view statistics, coverage
    size_t zero_bytes;      //   keys, tile partial slots
};

int64_t sel_capacity(int32_t M) {
    const int64_t m_main = (int64_t)((double)M * 0.85);      // int(M * 0.85), reference core/sampling.py:31
    int64_t cap = (M > m_main + 1) ? M : m_main + 1;
    if (cap < 4) cap = 4;
    return (cap + 3) / 4 * 4;
}

int make_plan(const ldp_params* p, void* base, Plan* plan) {
    if (!p || p->n_refs < 0 || p->H <= 0 || p->W <= 0 || p->matches_per_ref < 0 || p->tiles <= 0 || p->border < 0 ||
        p->w_match <= 0 || p->h_match <= 0)
        return fail(LDP_ERR_INVALID, "bad ldp_params");
    const long long Nll = (long long)p->H * (long long)p->W;
    if (Nll > 0x3fffffffLL) return fail(LDP_ERR_INVALID, "map too large");
    const int N = (int)Nll;
    const size_t R = (size_t)p->n_refs;
    ldp::SampleGeom& g = plan->geom;
    g.N = N;
    g.tile = (p->W / p->tiles > 1) ? p->W / p->tiles : 1;
    g.nbx = (p->W + g.tile - 1) / g.tile;
    g.nby = (p->H + g.tile - 1) / g.tile;
    g.nbins = g.nbx * g.nby;
    if (g.nbins > LDP_MAX_BINS) return fail(LDP_ERR_INVALID, "too many coverage tiles for this aspect ratio");
    int nb_pow2 = 1;
    while (nb_pow2 < g.nbins) nb_pow2 <<= 1;
    const int m_main = (int)((double)p->matches_per_ref * 0.85);
    g.size = m_main < N ? m_main : N;
    g.cov_budget = (p->matches_per_ref - g.size > 1) ? p->matches_per_ref - g.size : 1;
    g.vec = 0;
    g.w_magic = ((1ull << 40) + (unsigned long long)p->W - 1) / (unsigned long long)p->W;
    g.t_magic = ((1ull << 40) + (unsigned long long)g.tile - 1) / (unsigned long long)g.tile;
    g.t_magic32 = (g.tile > 1) ? (uint32_t)(((1ull << 32) + (unsigned long long)g.tile - 1) / (unsigned long long)g.tile) : 0u;
    g.step_dx = (ldp::KS_THREADS * 4) % p->W;
    g.step_dy = (ldp::KS_THREADS * 4) / p->W;
    int cs = 5;
    for (;; ++cs) {
        const size_t nchunk = ((size_t)N + ((size_t)1 << cs) - 1) >> cs;
        const size_t ept = 8 * ((nchunk + 8 * ldp::KD_THREADS - 1) / (8 * ldp::KD_THREADS));
        const size_t pre_cap = ept * ldp::KD_THREADS / 8 * 10 + 16;            // padded: 10 doubles per 8 entries
        size_t ng = 1;
        while (ng * 2 <= nchunk / 2) ng *= 2;
        const size_t bytes = pre_cap * 8 + (ng + 2) * 4 + 16;
        if (bytes <= K1_SMEM_BUDGET && bytes >= (size_t)nb_pow2 * 8) {
            g.nchunk = (int)nchunk; g.draw_ept = (int)ept; g.draw_pre_cap = (int)pre_cap; g.draw_ng = (int)ng;
            plan->k1_smem = bytes;
            break;
        }
        if (bytes <= K1_SMEM_BUDGET) {      // tiny map: the coverage sort needs nb_pow2 keys
            g.nchunk = (int)nchunk; g.draw_ept = (int)ept; g.draw_pre_cap = (int)pre_cap; g.draw_ng = (int)ng;
            plan->k1_smem = (size_t)nb_pow2 * 8;
            break;
        }
        if (cs > 20) return fail(LDP_ERR_INVALID, "map too large for the chunk table");
    }
    g.chunk_shift = cs;
    {   // the ordered compaction keeps one output offset per bitmap word of a tile in shared memory, plus staging
        const size_t nw = (align_up((size_t)N, 256) + 31) / 32;
        const size_t need = (std::min(nw, (size_t)ldp::KD_THREADS * 8) + 1) * 4 + 4096;
        if (plan->k1_smem < need) plan->k1_smem = need;
    }
    g.draw_smem_bytes = (int)plan->k1_smem;

    ldp::Workspace& w = plan->ws;
    w.n_pad = align_up((size_t)N, 256);
    w.n_words = (w.n_pad + 31) / 32;
    w.found_cap = align_up((size_t)(g.size > 0 ? g.size : 1), 4);
    w.sel_cap = (size_t)sel_capacity(p->matches_per_ref);
    size_t tk = 1;
    const size_t Mn = (size_t)((p->matches_per_ref < N) ? p->matches_per_ref : N);
    while (tk < Mn) tk <<= 1;
    w.topk_cap = p->no_filter ? tk : 0;
    w.nchunk_pad = align_up((size_t)g.nchunk, 32);
    w.bins_cap = align_up((size_t)g.nbins, 32);
    {
        const int rows = (ldp::KS_SPAN + p->W - 1) / p->W + 1;
        long long lb = (long long)(rows / g.tile + 2) * g.nbx;
        if (lb > g.nbins) lb = g.nbins;
        g.prep_lb_cap = (int)align_up((size_t)lb, 4);
    }
    plan->prep_smem = (size_t)g.prep_lb_cap * 8;
    w.nblk = ((size_t)N + ldp::KS_SPAN - 1) / ldp::KS_SPAN;

    Carver c{static_cast<char*>(base)};
    w.w = c.take<float>(R * w.n_pad);
    w.bestk = c.take<uint8_t>(R * w.n_pad);
    w.bitmap = c.take<uint32_t>(R * w.n_words);
    w.gone = c.take<uint32_t>(R * w.n_words);
    w.draw_cmax = 8;
    w.found = c.take<int32_t>(R * w.draw_cmax * w.found_cap);
    w.fcnt = c.take<int32_t>(R * w.draw_cmax);
    w.sel = c.take<int32_t>(R * w.sel_cap);
    w.pt0 = c.take<float4>(R * w.sel_cap);
    w.pt1 = c.take<float4>(R * w.sel_cap);
    w.dbgm = c.take<float4>(p->collect_debug ? R * w.sel_cap : 0);
    w.flags = c.take<uint8_t>(R * w.sel_cap);
    w.topk_keys = c.take<unsigned long long>(R * w.topk_cap);
    w.csum = c.take<double>(R * w.nchunk_pad);
    w.csum0 = c.take<double>(R * w.nchunk_pad);
    w.dbgclk = c.take<long long>(R * 32);
    plan->nb2 = (int)((w.sel_cap + ldp::K2_THREADS - 1) / ldp::K2_THREADS);
    w.blk_cnt = c.take<int32_t>(R * plan->nb2 * LDP_MAX_NN);
    w.blk_first = c.take<int32_t>(R * plan->nb2 * LDP_MAX_NN);
    w.fix_list = c.take<int2>(R * w.sel_cap);
    w.dstat = c.take<int32_t>(R);
    const size_t mv_slots = p->multiview ? R * w.sel_cap : 0;
    w.vmask = c.take<int32_t>(mv_slots);
    w.mvrec = c.take<float4>(mv_slots);
    // ---- the zero block (one memset per call, clear_launch_state): 8-byte items first, packed on 8 bytes
    const size_t z0 = c.off;
    w.gbins = c.take<unsigned long long>(R * w.bins_cap, 8);
    w.partial = c.take<double>(R * w.nblk, 8);
    w.rstat = c.take<ldp::RefStat>(R, 8);
    w.bflags = c.take<int32_t>(R * w.nblk, 8);
    w.kept = c.take<int32_t>(R, 8);
    w.fix_count = c.take<int32_t>(1, 8);
    plan->zero_base = base ? static_cast<char*>(base) + z0 : nullptr;
    plan->zero_bytes = c.off - z0;
    plan->bytes = align_up(c.off, 256);
    return LDP_OK;
}

int clear_launch_state(const Plan& plan, cudaStream_t st) {
    return check(cudaMemsetAsync(plan.zero_base, 0, plan.zero_bytes, st), "cudaMemsetAsync(launch state)");
}

int check_outputs(const ldp_params* p, const ldp_outputs* o) {
    if (!o) return fail(LDP_ERR_INVALID, "null outputs");
    if (!o->xyz || !o->rgb || !o->err || !o->ref_offset || !o->status || !o->n_samples || !o->group_count || !o->group_order)
        return fail(LDP_ERR_INVALID, "a required output pointer is null");
    if (p->collect_debug && (!o->dbg_matches || !o->dbg_cert))
        return fail(LDP_ERR_INVALID, "collect_debug needs dbg_matches and dbg_cert");
    if (o->capacity < 0) return fail(LDP_ERR_INVALID, "negative capacity");
    if (o->view_mask && !p->multiview) return fail(LDP_ERR_INVALID, "view_mask is written by multiview launches only");
    if (p->multiview && p->no_filter) return fail(LDP_ERR_INVALID, "multiview needs the filters (no_filter = 0)");
    if (p->multiview && !(p->multiview_min_cert > 0.0f && p->multiview_min_cert <= 1.0f))
        return fail(LDP_ERR_INVALID, "multiview_min_cert must lie in (0, 1]");
    return LDP_OK;
}

// The sample kernels' vector loads: the host wrapper guarantees 16-byte aligned certainty planes when W % 4 == 0; the planes'
// addresses live in device memory, so alignment cannot be checked here without a copy.  Callers that cannot guarantee it
// set params->scalar_loads = 1 to force the scalar load path.
int vec_ok_for(const ldp_params* p) { return (p->W % 4 == 0 && p->scalar_loads == 0) ? 1 : 0; }

// The plan of `p` laid over the caller's workspace from its first 256-byte boundary, checked to fit in workspace_bytes (the
// read-back hooks, which reuse a launch's workspace, pass SIZE_MAX).
int bind_plan(const ldp_params* p, void* workspace, size_t workspace_bytes, Plan* plan) {
    if (!workspace) return fail(LDP_ERR_INVALID, "null workspace");
    char* base = reinterpret_cast<char*>(align_up(reinterpret_cast<size_t>(workspace), 256));
    const int rc = make_plan(p, base, plan);
    if (rc != LDP_OK) return rc;
    if (plan->bytes + (size_t)(base - static_cast<char*>(workspace)) > workspace_bytes) return fail(LDP_ERR_WORKSPACE, "workspace too small");
    plan->geom.vec = vec_ok_for(p);
    return LDP_OK;
}

// the first kernel of the path (also launched alone by ldp_debug_launch_stream for the roofline measurement)
int launch_stream(const ldp_params* p, const ldp_ref_desc* refs, const Plan& plan, cudaStream_t st) {
    const int mode = p->prologue ? (p->no_warped_masks ? 1 : 2) : 0;
    const int nn = (p->nn_max >= 1 && p->nn_max <= 8) ? p->nn_max : 0;
    return launch("ldp_stream_kernel", k_stream[mode][nn], dim3((unsigned)plan.ws.nblk, (unsigned)p->n_refs), dim3(ldp::KS_THREADS),
                  0, st, *p, refs, plan.ws, plan.geom);
}

int launch_sample(const ldp_params* p, const ldp_ref_desc* refs, const double* uniforms, const ldp_outputs* out,
                  const Plan& plan, cudaStream_t st) {
    int rc = configure_device();
    if (rc != LDP_OK) return rc;
    if (plan.prep_smem > PREP_SMEM_MAX) return fail(LDP_ERR_INVALID, "map too wide for the prep kernel tables");
    const int R = p->n_refs;
    const dim3 grid((unsigned)plan.ws.nblk, (unsigned)R);
    { KernelTimer kt(st, "ldp_stream_kernel");
      if ((rc = launch_stream(p, refs, plan, st)) != LDP_OK) return rc; }
    if (p->no_filter) {
        KernelTimer kt(st, "ldp_topm_kernel");
        size_t n2 = 1;
        const size_t Mn = (size_t)std::min((long long)p->matches_per_ref, (long long)plan.geom.N);
        while (n2 < Mn) n2 <<= 1;
        // dynamic shared memory of a CTA: its sort buffer(s) + one tie count per 128-pixel row of its slice
        const size_t n4 = plan.ws.n_pad / 4;
        auto topm_smem = [&](int c) {
            const size_t keys_cap = std::max(n2 / (size_t)c, std::min(n2, (size_t)1024));
            const size_t per = (((n4 + c - 1) / c) + 31) & ~(size_t)31;
            return (c > 1 ? 2 : 1) * keys_cap * 8 + (per / 32) * 4;
        };
        if (topm_smem(1) > K1_SMEM_BUDGET)
            return launch("ldp_topm_generic_kernel", ldp::ldp_topm_generic_kernel, dim3(R), dim3(ldp::K1_THREADS), 0, st, *p, refs,
                          plan.ws, *out, plan.geom);
        // one cluster of C CTAs per view: the largest C that keeps every view's cluster in one wave (one CTA per SM)
        int csize = 1;
        for (int c = 8; c > 1; c >>= 1)
            if ((long long)R * c <= sm_count() && (size_t)c * 1024 <= n2) { csize = c; break; }
        const int fc = g_force_cluster;              // test hook
        if ((fc == 1 || fc == 2 || fc == 4 || fc == 8) && (size_t)fc <= n2) csize = fc;
        while (csize > 1 && topm_smem(csize) > K1_SMEM_BUDGET) csize >>= 1;
        return launch_cluster("ldp_topm_kernel", csize, [&](int c) {
            return launch_k(c > 1 ? c : 0, ldp::ldp_topm_kernel, dim3((unsigned)(R * c)), dim3(ldp::K1_THREADS), topm_smem(c), st,
                            *p, refs, plan.ws, *out, plan.geom, c);
        });
    }
    if (plan.geom.chunk_shift > 7) {      // chunk sums are accumulated with atomics: start from zero
        const size_t bytes = (size_t)R * plan.ws.nchunk_pad * sizeof(double);
        if ((rc = check(cudaMemsetAsync(plan.ws.csum, 0, bytes, st), "cudaMemsetAsync(csum)")) != LDP_OK) return rc;
        if ((rc = check(cudaMemsetAsync(plan.ws.csum0, 0, bytes, st), "cudaMemsetAsync(csum0)")) != LDP_OK) return rc;
    }
    { KernelTimer kt(st, "ldp_prep_kernel");
      const ldp::SampleGeom& g = plan.geom;
      // QUAD needs every quad in one image row (W % 4 == 0) and in at most two tiles (tiles wider than one pixel), and
      // umulhi(x, t_magic32) exact for every column: (W - 1) * tile < 2^32.  CONST is the QUAD case in which W divides the
      // pass stride (step_dx == 0), so that a thread stays in one pixel column.  Every other map takes PIXEL.
      const bool quad = p->W % 4 == 0 && g.tile > 1 && (unsigned long long)(p->W - 1) * g.tile < (1ull << 32);
      const PrepCols cols = !quad ? PrepCols::PIXEL : g.step_dx == 0 ? PrepCols::CONST : PrepCols::QUAD;
      const int cs = g.chunk_shift;
      const PrepKernel kp = k_prep[(cs >= 5 && cs <= 7) ? cs - 5 : 3][(int)cols];
      if ((rc = launch("ldp_prep_kernel", kp, grid, dim3(ldp::KS_THREADS), plan.prep_smem, st, *p, refs, plan.ws, *out, plan.geom)) != LDP_OK)
          return rc; }
    // ---- round 1: independent CTAs, as many per view as the device has SMs for (one CTA per SM: the table fills it), less
    //      the SMs left to concurrent kernels (other launches in flight, communication)
    const int sm_reserve = p->sm_reserve >= 0 ? p->sm_reserve : g_sm_reserve;
    int c_first = (sm_count() - sm_reserve) / R;
    if (c_first < 1) c_first = 1;
    if (c_first > (int)plan.ws.draw_cmax) c_first = (int)plan.ws.draw_cmax;
    if (g_force_cluster > 0) c_first = g_force_cluster;
    { KernelTimer kt(st, "ldp_draw_kernel");
      if ((rc = launch("ldp_draw_kernel<1>", ldp::ldp_draw_kernel<1>, dim3((unsigned)(R * c_first)), dim3(ldp::KD_THREADS), plan.k1_smem,
                       st, *p, refs, uniforms, plan.ws, *out, plan.geom, c_first)) != LDP_OK)
          return rc; }
    // ---- rounds 2.., coverage, compaction: one cluster per view.  The kernel is a chain of latency-bound phases (table
    // rebuild, a few hundred draws per round, bitmap compaction): one CTA per 2^18 pixels is as fast as more of them
    // (measured: 46 views at 512^2, 1 vs 2 vs 4 CTAs: 24.9 / 24.9 / 37 us) and leaves the other SMs to the launches in
    // flight beside this one (3 in flight: 0.143 -> 0.136 ms per step; 640^2, 32 views: 4 -> 2 CTAs 1.33 -> 1.28 ms per
    // 250 views).  Capped by what is resident at once (GPC boundaries make that smaller than sm_count / n_refs: ask the
    // occupancy API).
    int want = 1;
    while (want < 8 && (long long)want * (1 << 18) < (long long)plan.geom.N) want <<= 1;
    int csize = 1;
    for (int c = want; c > 1; c >>= 1) {
        if ((long long)R * c > sm_count()) continue;
        if (max_active_clusters(c, plan.k1_smem) >= R) { csize = c; break; }
    }
    if (g_force_cluster > 0) csize = g_force_cluster;
    KernelTimer kt(st, "ldp_resume_kernel");
    return launch_cluster("ldp_draw_kernel<2>", csize, [&](int c) {
        return launch_k(c, ldp::ldp_draw_kernel<2>, dim3((unsigned)(R * c)), dim3(ldp::KD_THREADS), plan.k1_smem, st,
                        *p, refs, uniforms, plan.ws, *out, plan.geom, c_first);
    });
}

// Largest f32 cosine d for which the reference's parallax test passes, i.e. for which
// f32(arccos(d)) * f32(180/pi) >= min_deg in float32 (core/geometry.py:118-119, arccos correctly rounded).
// arccos is monotone, so `angle >= min_deg` is `d <= threshold`: the kernel compares cosines and never calls acos.
float parallax_cos_threshold(float min_deg) {
    auto pred = [&](float d) {
        const float a = (float)acos((double)d);
        const float ang = a * 57.2957763671875f;
        return ang >= min_deg;
    };
    auto ord = [](float f) { uint32_t b; memcpy(&b, &f, 4); return (b & 0x80000000u) ? ~b : (b | 0x80000000u); };
    auto unord = [](uint32_t k) { uint32_t b = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k; float f; memcpy(&f, &b, 4); return f; };
    if (!pred(-1.0f)) return -2.0f;
    if (pred(1.0f)) return 1.0f;
    uint32_t lo = ord(-1.0f), hi = ord(1.0f);           // pred(lo) true, pred(hi) false
    while (hi - lo > 1) {
        const uint32_t mid = lo + (hi - lo) / 2;
        if (pred(unord(mid))) lo = mid; else hi = mid;
    }
    return unord(lo);
}

ldp::GeomArgs make_geom_args(const ldp_params* p, int nb2, int have_bestk) {
    thread_local float cached_deg = -1.f, cached_cos = 1.f;
    if (p->min_parallax_deg != cached_deg) { cached_cos = parallax_cos_threshold(p->min_parallax_deg); cached_deg = p->min_parallax_deg; }
    ldp::GeomArgs ga;
    ga.par_cos_max = cached_cos;
    ga.have_bestk = have_bestk;
    ga.nb2 = nb2;
    ga.force_fix_two = g_force_fix_two;
    ga.force_fix_mv = g_force_fix_mv;
    return ga;
}

// gather + compute -> fix + plan, then the ordered scatter of all views of the launch (needs every view's kept count)
int launch_triangulate(const ldp_params* p, const ldp_ref_desc* refs, const ldp_outputs* out, const Plan& plan,
                       int have_bestk, cudaStream_t st) {
    ldp::GeomArgs ga = make_geom_args(p, plan.nb2, have_bestk);
    const dim3 grid((unsigned)plan.nb2, (unsigned)p->n_refs);
    int rc;
    // The order in which these instantiations are first named here steers the device compiler's inlining: as a [lens][mv]
    // table, ldp_fix_kernel<true, true> compiles to different code (166 instead of 158 registers, 272 bytes of stack).
    { KernelTimer kt(st, "ldp_geometry_kernel");
      auto* k2 =p->multiview ? (p->lens ? ldp::ldp_geometry_kernel<true, true> : ldp::ldp_geometry_kernel<false, true>)
                              : (p->lens ? ldp::ldp_geometry_kernel<true, false> : ldp::ldp_geometry_kernel<false, false>);
      if ((rc = launch("ldp_geometry_kernel", k2, grid, dim3(ldp::K2_THREADS), 0, st, *p, refs, plan.ws, *out, ga)) != LDP_OK) return rc; }
    { KernelTimer kt(st, "ldp_fix_kernel");
      auto* kf = p->multiview ? (p->lens ? ldp::ldp_fix_kernel<true, true> : ldp::ldp_fix_kernel<false, true>)
                              : (p->lens ? ldp::ldp_fix_kernel<true, false> : ldp::ldp_fix_kernel<false, false>);
      if ((rc = launch("ldp_fix_kernel", kf, dim3(p->n_refs), dim3(ldp::K2_THREADS), 0, st, *p, refs, plan.ws, *out, ga)) != LDP_OK) return rc; }
    ga.have_bestk = 1;
    KernelTimer kt(st, "ldp_pack_kernel");
    return launch("ldp_pack_kernel", ldp::ldp_pack_kernel, grid, dim3(ldp::K3_THREADS), 0, st, *p, refs, plan.ws, *out, ga);
}

// ---- depth maps: the worklist of the fix-up (one slot per pixel of every view) and its counters
struct DepthPlan {
    int32_t* fix_count;
    uint32_t* fix_list;
    size_t bytes;
};

int make_depth_plan(const ldp_params* p, void* base, DepthPlan* dp) {
    if (!p || p->n_refs < 0 || p->n_refs > 65535 || p->H <= 0 || p->W <= 0 || p->w_match <= 0 || p->h_match <= 0)
        return fail(LDP_ERR_INVALID, "bad ldp_params");
    const long long N = (long long)p->H * (long long)p->W;
    if (N > 0x3fffffffLL) return fail(LDP_ERR_INVALID, "map too large");
    const size_t R = (size_t)p->n_refs;
    Carver c{static_cast<char*>(base)};
    dp->fix_count = c.take<int32_t>(R);
    dp->fix_list = c.take<uint32_t>(R * (size_t)N);
    dp->bytes = align_up(c.off, 256);
    return LDP_OK;
}

}  // namespace

extern "C" {

int ldp_abi_version(void) { return LDP_ABI_VERSION; }

const char* ldp_last_error_string(void) { return g_last_error.c_str(); }

int64_t ldp_sel_capacity(int32_t matches_per_ref) { return sel_capacity(matches_per_ref); }

int ldp_last_launch_count(void) { return g_launches; }

int ldp_profile_enable(int on) { g_prof_on = (on != 0); g_prof_n = 0; return LDP_OK; }

int ldp_profile_read(float* ms_out, int max_n) {
    if (!ms_out || max_n < 0) return fail(LDP_ERR_INVALID, "bad profile buffer");
    const int n = g_prof_n < max_n ? g_prof_n : max_n;
    for (int i = 0; i < n; ++i) {
        cudaError_t e = cudaEventSynchronize(g_prof_ev[2 * i + 1]);
        if (e != cudaSuccess) return cuda_fail(e, "cudaEventSynchronize(profile)");
        e = cudaEventElapsedTime(&ms_out[i], g_prof_ev[2 * i], g_prof_ev[2 * i + 1]);
        if (e != cudaSuccess) return cuda_fail(e, "cudaEventElapsedTime(profile)");
    }
    return g_prof_n;
}

int ldp_debug_last_cluster(void) { return g_last_cluster; }

int ldp_debug_launch_stream(const ldp_params* params, const ldp_ref_desc* refs, void* workspace, size_t workspace_bytes,
                            void* stream, int reps) {
    begin_call();
    if (!params || !refs || !workspace || reps < 1) return fail(LDP_ERR_INVALID, "bad arguments");
    Plan plan;
    int rc = bind_plan(params, workspace, workspace_bytes, &plan);
    for (int i = 0; i < reps && rc == LDP_OK; ++i) rc = launch_stream(params, refs, plan, static_cast<cudaStream_t>(stream));
    return rc;
}

int ldp_debug_read_clocks(const ldp_params* params, void* workspace, long long* host_out) {
    if (!params || !workspace || !host_out) return fail(LDP_ERR_INVALID, "bad arguments");
    Plan plan;
    const int rc = bind_plan(params, workspace, SIZE_MAX, &plan);
    if (rc != LDP_OK) return rc;
    return check(cudaMemcpy(host_out, plan.ws.dbgclk, (size_t)params->n_refs * 32 * sizeof(long long), cudaMemcpyDeviceToHost),
                 "cudaMemcpy(dbgclk)");
}

int ldp_debug_force_fixup(int two_view_every, int multiview_every) {
    if (two_view_every < 0 || multiview_every < 0) return fail(LDP_ERR_INVALID, "force_fixup periods must be >= 0");
    g_force_fix_two = two_view_every;
    g_force_fix_mv = multiview_every;
    return LDP_OK;
}

int ldp_debug_read_fixups(const ldp_params* params, void* workspace, int32_t* host_out) {
    if (!params || !workspace || !host_out) return fail(LDP_ERR_INVALID, "bad arguments");
    Plan plan;
    int rc = bind_plan(params, workspace, SIZE_MAX, &plan);
    if (rc != LDP_OK) return rc;
    host_out[0] = host_out[1] = 0;
    int32_t count = 0;
    if ((rc = check(cudaMemcpy(&count, plan.ws.fix_count, sizeof(count), cudaMemcpyDeviceToHost), "cudaMemcpy(fix_count)")) != LDP_OK)
        return rc;
    if (count <= 0) return LDP_OK;
    std::vector<int2> list((size_t)count);
    if ((rc = check(cudaMemcpy(list.data(), plan.ws.fix_list, list.size() * sizeof(int2), cudaMemcpyDeviceToHost),
                    "cudaMemcpy(fix_list)")) != LDP_OK)
        return rc;
    host_out[0] = count;
    for (const int2& it : list) host_out[1] += (it.y & ldp::MV_FIX) ? 1 : 0;
    return LDP_OK;
}

int ldp_debug_set_cluster(int csize) {
    if (csize < 0 || csize > 8) return fail(LDP_ERR_INVALID, "cluster size must be 0 (auto) .. 8");
    g_force_cluster = csize;
    return LDP_OK;
}

const char* ldp_profile_name(int i) { return (i >= 0 && i < g_prof_n) ? g_prof_name[i] : ""; }

// ---- output contract on the device (ldp_output.cu)
// format 0: PLY, 1: points3D (err, first_id), 2: PLY with normals
static int pack_records(int format, const float* xyz, const float* rgb, const float* err, const float* normals, int64_t n,
                        const int64_t* n_dev, uint64_t first_id, uint8_t* out, void* stream) {
    begin_call();
    if (n < 0) return fail(LDP_ERR_INVALID, "negative point count");
    if (n == 0) return LDP_OK;
    if (format == 2 && !normals) return fail(LDP_ERR_INVALID, "null normals");
    if (!xyz || !rgb || !out) return fail(LDP_ERR_INVALID, "null pointer");
    static const decltype(&ldp::ldp_records_kernel<0>) k_records[3] = {ldp::ldp_records_kernel<0>, ldp::ldp_records_kernel<1>,
                                                                        ldp::ldp_records_kernel<2>};
    const unsigned grid = (unsigned)((n + ldp::KO_THREADS - 1) / ldp::KO_THREADS);
    const int aligned = (reinterpret_cast<uintptr_t>(out) & 15u) == 0;
    return launch("ldp_records_kernel", k_records[format], dim3(grid), dim3(ldp::KO_THREADS), 0, reinterpret_cast<cudaStream_t>(stream),
                  xyz, rgb, err, (long long)n, reinterpret_cast<const long long*>(n_dev), (unsigned long long)first_id, out, aligned,
                  normals);
}

int ldp_pack_ply_records(const float* xyz, const float* rgb, int64_t n, const int64_t* n_dev, uint8_t* records_out, void* stream) {
    return pack_records(0, xyz, rgb, nullptr, nullptr, n, n_dev, 0, records_out, stream);
}

int ldp_pack_ply_normal_records(const float* xyz, const float* rgb, const float* normals, int64_t n, const int64_t* n_dev,
                                uint8_t* records_out, void* stream) {
    return pack_records(2, xyz, rgb, nullptr, normals, n, n_dev, 0, records_out, stream);
}

int ldp_pack_points3d_records(const float* xyz, const float* rgb, const float* err, int64_t n, const int64_t* n_dev,
                              uint64_t first_id, uint8_t* records_out, void* stream) {
    return pack_records(1, xyz, rgb, err, nullptr, n, n_dev, first_id, records_out, stream);
}

int ldp_undistort_points(const ldp_lens* lens, int64_t n, const float* uv_in, float* uv_out, void* stream) {
    begin_call();
    if (!lens || n < 0) return fail(LDP_ERR_INVALID, "bad arguments");
    if (lens->model < LDP_LENS_PINHOLE || lens->model > LDP_LENS_FISHEYE) return fail(LDP_ERR_INVALID, "unknown lens model");
    if (n == 0) return LDP_OK;
    if (!uv_in || !uv_out) return fail(LDP_ERR_INVALID, "null pointer");
    if ((reinterpret_cast<size_t>(uv_in) | reinterpret_cast<size_t>(uv_out)) & 7) return fail(LDP_ERR_INVALID, "uv arrays must be 8-byte aligned");
    const long long blocks = (n + ldp::KU_THREADS - 1) / ldp::KU_THREADS;
    const unsigned grid = (unsigned)std::min<long long>(blocks, (long long)sm_count() * 16);
    return launch("ldp_undistort_kernel", ldp::ldp_undistort_kernel, dim3(grid), dim3(ldp::KU_THREADS), 0,
                  reinterpret_cast<cudaStream_t>(stream), *lens, (long long)n, reinterpret_cast<const float2*>(uv_in),
                  reinterpret_cast<float2*>(uv_out));
}

int ldp_rgb_to_uint8(const float* rgb, int64_t n_values, uint8_t* out, void* stream) {
    begin_call();
    if (n_values < 0) return fail(LDP_ERR_INVALID, "negative count");
    if (n_values == 0) return LDP_OK;
    if (!rgb || !out) return fail(LDP_ERR_INVALID, "null pointer");
    const long long blocks = (n_values + ldp::KO_THREADS - 1) / ldp::KO_THREADS;
    const unsigned grid = (unsigned)std::min<long long>(blocks, (long long)sm_count() * 16);
    return launch("ldp_rgb_u8_kernel", ldp::ldp_rgb_u8_kernel, dim3(grid), dim3(ldp::KO_THREADS), 0, reinterpret_cast<cudaStream_t>(stream),
                  rgb, (long long)n_values, out);
}

int ldp_gather_points(const float* xyz, const float* rgb, const float* err, const int64_t* sel, int64_t m, int64_t n,
                      float* xyz_out, float* rgb_out, float* err_out, int32_t* bad_index_flag, void* stream) {
    begin_call();
    if (m < 0 || n < 0) return fail(LDP_ERR_INVALID, "negative count");
    if (m == 0) return LDP_OK;
    if (!xyz || !rgb || !sel || !xyz_out || !rgb_out) return fail(LDP_ERR_INVALID, "null pointer");
    const unsigned grid = (unsigned)((m + ldp::KO_THREADS - 1) / ldp::KO_THREADS);
    return launch("ldp_gather_rows_kernel", ldp::ldp_gather_rows_kernel, dim3(grid), dim3(ldp::KO_THREADS), 0,
                  reinterpret_cast<cudaStream_t>(stream), xyz, rgb, err, reinterpret_cast<const long long*>(sel), (long long)m,
                  (long long)n, xyz_out, rgb_out, err_out, (int*)bad_index_flag);
}

int ldp_gather_rows(const float* src, int32_t row_floats, const int64_t* sel, int64_t m, int64_t n, float* out,
                    int32_t* bad_index_flag, void* stream) {
    begin_call();
    if (m < 0 || n < 0 || row_floats <= 0) return fail(LDP_ERR_INVALID, "bad row gather shape");
    if (m == 0) return LDP_OK;
    if (!src || !sel || !out) return fail(LDP_ERR_INVALID, "null pointer");
    const long long blocks = (m * row_floats + ldp::KO_THREADS - 1) / ldp::KO_THREADS;
    const unsigned grid = (unsigned)std::min<long long>(blocks, (long long)sm_count() * 16);
    return launch("ldp_gather_f32_rows_kernel", ldp::ldp_gather_f32_rows_kernel, dim3(grid), dim3(ldp::KO_THREADS), 0,
                  reinterpret_cast<cudaStream_t>(stream), src, (int)row_floats, reinterpret_cast<const long long*>(sel), (long long)m,
                  (long long)n, out, (int*)bad_index_flag);
}

int ldp_concat_points(const float* const* xyz_src, const float* const* rgb_src, const float* const* err_src,
                      const int64_t* const* count_src, int32_t n_seg, int64_t seg_cap, float* xyz_out, float* rgb_out,
                      float* err_out, int64_t out_capacity, int64_t* seg_offset_out, int64_t* total_out, void* stream) {
    begin_call();
    if (n_seg < 0 || seg_cap < 0 || out_capacity < 0) return fail(LDP_ERR_INVALID, "negative size");
    if (n_seg == 0) return LDP_OK;
    if (!xyz_src || !rgb_src || !err_src || !count_src || !xyz_out || !rgb_out || !err_out) return fail(LDP_ERR_INVALID, "null pointer");
    if (n_seg > 65535) return fail(LDP_ERR_INVALID, "too many segments");
    const long long blocks = (seg_cap * 3 + ldp::KO_THREADS * 4 - 1) / (ldp::KO_THREADS * 4);
    // enough CTAs to keep a few MB of (possibly remote) reads in flight: about four waves of CTAs over all segments
    const long long per_seg = std::max<long long>(64, (long long)sm_count() * 8 * 4 / std::max(1, n_seg));
    const unsigned gx = (unsigned)std::max<long long>(1, std::min<long long>(blocks, per_seg));
    return launch("ldp_concat_points_kernel", ldp::ldp_concat_points_kernel, dim3(gx, (unsigned)n_seg), dim3(ldp::KO_THREADS), 0,
                  reinterpret_cast<cudaStream_t>(stream), xyz_src, rgb_src, err_src, reinterpret_cast<const long long* const*>(count_src),
                  (int)n_seg, (long long)seg_cap, xyz_out, rgb_out, err_out, (long long)out_capacity,
                  reinterpret_cast<long long*>(seg_offset_out), reinterpret_cast<long long*>(total_out));
}

int ldp_scatter_points(const float* xyz, const float* rgb, const float* err, const int64_t* const* count_src, int32_t rank,
                       int32_t world, int64_t seg_cap, float* const* xyz_dst, float* const* rgb_dst, float* const* err_dst,
                       int64_t out_capacity, int64_t* seg_offset_out, int64_t* total_out, void* stream) {
    begin_call();
    if (world < 1 || world > 64 || rank < 0 || rank >= world || seg_cap < 0 || out_capacity < 0) return fail(LDP_ERR_INVALID, "bad rank / world / size");
    if (!xyz || !rgb || !err || !count_src || !xyz_dst || !rgb_dst || !err_dst) return fail(LDP_ERR_INVALID, "null pointer");
    const long long blocks = (seg_cap * 3 + ldp::KO_THREADS * 4 - 1) / (ldp::KO_THREADS * 4);
    const long long per_dst = std::max<long long>(32, (long long)sm_count() * 8 * 2 / world);
    const unsigned gx = (unsigned)std::max<long long>(1, std::min<long long>(blocks, per_dst));
    return launch("ldp_scatter_points_kernel", ldp::ldp_scatter_points_kernel, dim3(gx, (unsigned)world), dim3(ldp::KO_THREADS), 0,
                  reinterpret_cast<cudaStream_t>(stream), xyz, rgb, err, reinterpret_cast<const long long* const*>(count_src), (int)rank,
                  (int)world, (long long)seg_cap, xyz_dst, rgb_dst, err_dst, (long long)out_capacity,
                  reinterpret_cast<long long*>(seg_offset_out), reinterpret_cast<long long*>(total_out));
}

// ---- pair generation on the device (ldp_select.cu)
int ldp_select_kcenters(const float* flat_poses, int32_t n, int32_t k, float* scratch, int32_t* centers_sorted,
                        int32_t* centers_order, void* stream) {
    begin_call();
    if (n <= 0 || k <= 0 || k > n) return fail(LDP_ERR_INVALID, "k-centres needs 1 <= k <= n");
    if (n > ldp::KC_THREADS * ldp::KC_MAX_PER_THREAD) return fail(LDP_ERR_INVALID, "k-centres: more than 8192 views");
    if (!flat_poses || !scratch || !centers_sorted || !centers_order) return fail(LDP_ERR_INVALID, "null pointer");
    const size_t smem = (size_t)n * ldp::KC_PAD * sizeof(float);
    const bool in_smem = smem <= K1_SMEM_BUDGET;         // the poses fit in shared memory (n <= 3011)
    if (in_smem) {
        const int rc = configure_device();
        if (rc != LDP_OK) return rc;
    }
    return launch("ldp_kcenters_kernel", in_smem ? ldp::ldp_kcenters_kernel<true> : ldp::ldp_kcenters_kernel<false>, dim3(1),
                  dim3(ldp::KC_THREADS), in_smem ? smem : 0, reinterpret_cast<cudaStream_t>(stream), flat_poses, (int)n, (int)k, scratch,
                  centers_sorted, centers_order);
}

int ldp_nearest_neighbors(const float* flat_poses, int32_t n, int32_t k, int64_t* idx_out, void* stream) {
    begin_call();
    if (n < 0 || k < 0) return fail(LDP_ERR_INVALID, "negative size");
    if (n <= 1 || k == 0) return LDP_OK;
    if (k > n - 1 || k > ldp::KNN_MAX_K) return fail(LDP_ERR_INVALID, "nearest neighbours needs k <= min(n - 1, 16)");
    if (!flat_poses || !idx_out) return fail(LDP_ERR_INVALID, "null pointer");
    return launch("ldp_knn_kernel", ldp::ldp_knn_kernel, dim3((unsigned)n), dim3(ldp::KNN_THREADS), 0, reinterpret_cast<cudaStream_t>(stream),
                  flat_poses, (int)n, (int)k, reinterpret_cast<long long*>(idx_out));
}

// ---- voxel-grid downsample (ldp_voxel.cu)
static size_t voxel_cap(int64_t n) {
    size_t cap = 1024;
    while (cap < (size_t)n * 2) cap <<= 1;
    return cap;
}
static int voxel_plan(int64_t n, void* base, ldp::VoxelWs* ws, size_t* bytes) {
    if (n < 0 || n > 500000000ll) return fail(LDP_ERR_INVALID, "voxel downsample: bad point count");
    const size_t cap = voxel_cap(n), N = (size_t)std::max<int64_t>(n, 1);
    Carver c{static_cast<char*>(base)};
    ws->bounds = c.take<double>(8);
    ws->bounds_u = c.take<unsigned int>(8);
    ws->keys = c.take<unsigned long long>(cap);
    ws->first = c.take<int>(cap);
    ws->slot = c.take<int>(N);
    ws->flag = c.take<int>(N);
    ws->rank = c.take<int>(N);
    ws->count = c.take<int>(N + 1);
    ws->cursor = c.take<int>(N);
    ws->seg = c.take<int>(N);
    ws->members = c.take<int>(N);
    ws->block_tot = c.take<int>(N / ldp::SC_THREADS + 2);
    ws->large = c.take<int>(N + 2);
    ws->status = nullptr;
    ws->cap_mask = cap - 1;
    *bytes = c.off;
    return LDP_OK;
}

int ldp_voxel_workspace_bytes(int64_t n, size_t* bytes_out) {
    if (!bytes_out) return fail(LDP_ERR_INVALID, "null bytes_out");
    ldp::VoxelWs ws;
    return voxel_plan(n, nullptr, &ws, bytes_out);
}

static int scan_exclusive(const int* in, int* out, int64_t n, int* block_tot, int* grand_total, cudaStream_t st) {
    const int nblocks = (int)((n + ldp::SC_THREADS - 1) / ldp::SC_THREADS);
    int rc = launch("ldp_scan_blocks_kernel", ldp::ldp_scan_blocks_kernel, dim3(nblocks), dim3(ldp::SC_THREADS), 0, st, in, out,
                    (long long)n, block_tot);
    if (rc == LDP_OK)
        rc = launch("ldp_scan_totals_kernel", ldp::ldp_scan_totals_kernel, dim3(1), dim3(ldp::SC_THREADS), 0, st, block_tot, nblocks,
                    grand_total);
    if (rc == LDP_OK)
        rc = launch("ldp_scan_add_kernel", ldp::ldp_scan_add_kernel, dim3(nblocks), dim3(ldp::SC_THREADS), 0, st, out, (long long)n,
                    (const int*)block_tot);
    return rc;
}

int ldp_voxel_downsample(const float* xyz, const float* rgb, int64_t n, double voxel_size, float* xyz_out, float* rgb_out,
                         int32_t* status_out, void* workspace, size_t workspace_bytes, void* stream) {
    begin_call();
    if (!(voxel_size > 0.0)) return fail(LDP_ERR_INVALID, "voxel_size must be positive");       // Open3D: "voxel_size <= 0."
    if (!status_out) return fail(LDP_ERR_INVALID, "null status_out");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    int rc = check(cudaMemsetAsync(status_out, 0, 2 * sizeof(int32_t), st), "cudaMemsetAsync(status)");
    if (rc != LDP_OK || n == 0) return rc;
    if (!xyz || !rgb || !xyz_out || !rgb_out || !workspace) return fail(LDP_ERR_INVALID, "null pointer");
    ldp::VoxelWs ws;
    size_t need = 0;
    if ((rc = voxel_plan(n, workspace, &ws, &need)) != LDP_OK) return rc;
    if (workspace_bytes < need) return fail(LDP_ERR_INVALID, "voxel workspace too small");
    ws.status = status_out;
    const size_t cap = (size_t)ws.cap_mask + 1;
    cudaError_t e = cudaMemsetAsync(ws.bounds_u, 0xFF, 3 * sizeof(unsigned int), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(ws.bounds_u + 3, 0, sizeof(unsigned int), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(ws.keys, 0xFF, cap * sizeof(unsigned long long), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(ws.first, 0x7F, cap * sizeof(int), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(ws.count, 0, ((size_t)n + 1) * sizeof(int), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(ws.cursor, 0, (size_t)n * sizeof(int), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(ws.large, 0, 2 * sizeof(int), st);
    if ((rc = check(e, "cudaMemsetAsync(voxel workspace)")) != LDP_OK) return rc;
    const unsigned grid = (unsigned)((n + ldp::KV_THREADS - 1) / ldp::KV_THREADS);
    const unsigned rgrid = (unsigned)std::min<long long>(grid, (long long)sm_count() * 8);
    const dim3 block(ldp::KV_THREADS);
    rc = launch("ldp_voxel_bounds_kernel", ldp::ldp_voxel_bounds_kernel, dim3(rgrid), block, 0, st, xyz, rgb, (long long)n, ws);
    if (rc != LDP_OK) return rc;
    rc = launch("ldp_voxel_insert_kernel", ldp::ldp_voxel_insert_kernel, dim3(grid), block, 0, st, xyz, (long long)n, voxel_size,
                (const double*)nullptr, ws);
    if (rc != LDP_OK) return rc;
    rc = launch("ldp_voxel_flag_kernel", ldp::ldp_voxel_flag_kernel, dim3(grid), block, 0, st, (long long)n, ws);
    if (rc != LDP_OK) return rc;
    rc = scan_exclusive(ws.flag, ws.rank, n, ws.block_tot, ws.status + 1, st);
    if (rc != LDP_OK) return rc;
    rc = launch("ldp_voxel_count_kernel", ldp::ldp_voxel_count_kernel, dim3(grid), block, 0, st, (long long)n, ws);
    if (rc != LDP_OK) return rc;
    rc = scan_exclusive(ws.count, ws.seg, n, ws.block_tot, nullptr, st);
    if (rc != LDP_OK) return rc;
    rc = launch("ldp_voxel_group_kernel", ldp::ldp_voxel_group_kernel, dim3(grid), block, 0, st, (long long)n, ws, (const int*)ws.seg);
    if (rc != LDP_OK) return rc;
    rc = launch("ldp_voxel_mean_kernel", ldp::ldp_voxel_mean_kernel, dim3(grid), block, 0, st, xyz, rgb, ws, (const int*)ws.seg,
                xyz_out, rgb_out);
    if (rc != LDP_OK) return rc;
    return launch("ldp_voxel_large_kernel", ldp::ldp_voxel_large_kernel, dim3((unsigned)sm_count()), dim3(ldp::SC_THREADS), 0, st, xyz,
                  rgb, ws, (const int*)ws.seg, xyz_out, rgb_out);
}

// ---- statistical outlier removal (ldp_outlier.cu)
static int g_outlier_shells = 0;           // ldp_debug_outlier_max_shells; 0 = ldp::OL_DEFAULT_SHELLS

struct OutlierPlan {
    ldp::VoxelWs vws;                      // grid-building scratch, shared by the trial grid and every level
    int* vstat;                            // [2] status of the voxel kernels: overflow flag, cell count
    double* h_trial;                       // [1] trial cell size
    double* stats;                         // [3] used when the caller passes no stats_out
    double* m;                             // [n] used when the caller passes no mean_dist_out
    double* part;                          // [ceil(n / KS_CHUNK)] first-stage partial sums
    ldp::OutlierLevel* levels;             // [KS_MAX_LEVELS] level descriptors for the k-NN kernel
    unsigned long long* keys[ldp::OL_MAX_LEVELS];
    int2* cell[ldp::OL_MAX_LEVELS];
    float4* pts[ldp::OL_MAX_LEVELS];
};

// with_stats = false (the normal call) leaves out the per-point means and the partial sums
static int outlier_plan(int64_t n, void* base, OutlierPlan* pl, size_t* bytes, bool with_stats = true) {
    if (n < 0 || n > 500000000ll) return fail(LDP_ERR_INVALID, "k-NN search: bad point count");
    Carver c{static_cast<char*>(base)};
    int rc = voxel_plan(n, base, &pl->vws, &c.off);
    if (rc != LDP_OK) return rc;
    const size_t cap = voxel_cap(n), N = (size_t)std::max<int64_t>(n, 1);
    pl->vstat = c.take<int>(2);
    pl->h_trial = c.take<double>(1);
    pl->stats = c.take<double>(3);
    pl->m = c.take<double>(with_stats ? N : 0);
    pl->part = c.take<double>(with_stats ? N / ldp::OL_CHUNK + 1 : 0);
    pl->levels = c.take<ldp::OutlierLevel>(ldp::OL_MAX_LEVELS);
    for (int l = 0; l < ldp::OL_MAX_LEVELS; ++l) {
        pl->keys[l] = c.take<unsigned long long>(cap);
        pl->cell[l] = c.take<int2>(cap);
        pl->pts[l] = c.take<float4>(N);
    }
    *bytes = c.off;
    return LDP_OK;
}

int ldp_outlier_workspace_bytes(int64_t n, int32_t nb_neighbors, size_t* bytes_out) {
    if (!bytes_out) return fail(LDP_ERR_INVALID, "null bytes_out");
    if (nb_neighbors < 1 || nb_neighbors > ldp::OL_MAX_K) return fail(LDP_ERR_INVALID, "nb_neighbors must lie in [1, 64]");
    OutlierPlan pl;
    return outlier_plan(n, nullptr, &pl, bytes_out);
}

int ldp_debug_outlier_max_shells(int shells) {
    if (shells < 0) return fail(LDP_ERR_INVALID, "shells must be >= 0");
    g_outlier_shells = shells;
    return LDP_OK;
}

static float host_f32_unordered(unsigned int k) {          // ldp::f32_unordered on the host
    const unsigned int b = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
    float f;
    std::memcpy(&f, &b, sizeof(f));
    return f;
}

// hash insert, first-of-cell flags, ranks: the cells of a grid of size h (or *h_dev) in pl.vws.keys
static int outlier_insert(const float* xyz, int64_t n, double h, const double* h_dev, OutlierPlan& pl, unsigned grid, cudaStream_t st,
                          int* cells_out) {
    ldp::VoxelWs& ws = pl.vws;
    const size_t cap = (size_t)ws.cap_mask + 1;
    cudaError_t e = cudaMemsetAsync(ws.keys, 0xFF, cap * sizeof(unsigned long long), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(ws.first, 0x7F, cap * sizeof(int), st);
    int rc = check(e, "cudaMemsetAsync(outlier grid)");
    if (rc != LDP_OK) return rc;
    rc = launch("ldp_voxel_insert_kernel", ldp::ldp_voxel_insert_kernel, dim3(grid), dim3(ldp::KV_THREADS), 0, st, xyz, (long long)n, h,
                h_dev, ws);
    if (rc != LDP_OK) return rc;
    rc = launch("ldp_voxel_flag_kernel", ldp::ldp_voxel_flag_kernel, dim3(grid), dim3(ldp::KV_THREADS), 0, st, (long long)n, ws);
    if (rc != LDP_OK) return rc;
    return scan_exclusive(ws.flag, ws.rank, n, ws.block_tot, cells_out, st);
}

// Steps 1 and 2 of the k-NN search, shared by ldp_statistical_outliers, ldp_estimate_normals and ldp_gaussian_init: bounds and a trial grid,
// whose cell count sets the level-0 cell size (the one host synchronisation), then the pyramid and its level descriptors
// in pl.levels.  A coordinate that is not finite sets status_out[0] = 1 and leaves *n_levels_out = 0 (and returns LDP_OK);
// any CUDA failure returns LDP_ERR_CUDA.
static int knn_pyramid(const float* xyz, int64_t n, int k, OutlierPlan& pl, cudaStream_t st, int32_t* status_out, int* n_levels_out) {
    *n_levels_out = 0;
    cudaError_t e;
    int rc;
    ldp::VoxelWs& ws = pl.vws;
    ws.status = pl.vstat;
    const unsigned grid = (unsigned)((n + ldp::KV_THREADS - 1) / ldp::KV_THREADS);
    const unsigned rgrid = (unsigned)std::min<long long>(grid, (long long)sm_count() * 8);
    const size_t cap = (size_t)ws.cap_mask + 1;
    const unsigned cgrid = (unsigned)((cap + ldp::KV_THREADS - 1) / ldp::KV_THREADS);

    // 1. bounds and a trial grid; its cell count sets the level-0 cell size (the one host synchronisation)
    unsigned int bu[8];
    double h_trial = 0.0;
    {
        KernelTimer kt(st, "ldp_outlier_trial_grid");
        e = cudaMemsetAsync(ws.bounds_u, 0xFF, 3 * sizeof(unsigned int), st);
        if (e == cudaSuccess) e = cudaMemsetAsync(ws.bounds_u + 3, 0, 5 * sizeof(unsigned int), st);
        if ((rc = check(e, "cudaMemsetAsync(outlier bounds)")) != LDP_OK) return rc;
        rc = launch("ldp_voxel_bounds_kernel", ldp::ldp_voxel_bounds_kernel, dim3(rgrid), dim3(ldp::KV_THREADS), 0, st, xyz,
                    (const float*)nullptr, (long long)n, ws);
        if (rc != LDP_OK) return rc;
        rc = launch("ldp_outlier_trial_size_kernel", ldp::ldp_outlier_trial_size_kernel, dim3(1), dim3(1), 0, st,
                    (const unsigned int*)ws.bounds_u, (long long)n, k, pl.h_trial);
        if (rc != LDP_OK) return rc;
        rc = outlier_insert(xyz, n, 0.0, pl.h_trial, pl, grid, st, reinterpret_cast<int*>(ws.bounds_u + 7));
        if (rc != LDP_OK) return rc;
    }
    e = cudaMemcpyAsync(bu, ws.bounds_u, sizeof(bu), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&h_trial, pl.h_trial, sizeof(double), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if ((rc = check(e, "outlier trial grid")) != LDP_OK) return rc;
    double mn[3], mx[3], ext = 0.0;
    bool finite = true;
    for (int c = 0; c < 3; ++c) {
        mn[c] = (double)host_f32_unordered(bu[c]);
        mx[c] = (double)host_f32_unordered(bu[4 + c]);
        finite = finite && std::isfinite(mn[c]) && std::isfinite(mx[c]);
        ext = std::max(ext, mx[c] - mn[c]);
    }
    if (!finite)                                        // status_out[0] = 1 (little-endian int32, zeroed by the caller)
        return check(cudaMemsetAsync(status_out, 1, 1, st), "cudaMemsetAsync(status)");
    const double trial_cells = (double)std::max(1u, bu[7]);
    double h = 1.0;
    if (ext > 0.0) h = std::max(h_trial * std::sqrt(0.5 * k * trial_cells / (double)n), ext / 1048576.0);

    // 2. the pyramid: h_l = h0 * 8^l up to the first level with at most 3 cells per axis
    ldp::OutlierGrid lv;
    int n_levels = 0;
    {
        KernelTimer kt(st, "ldp_outlier_pyramid");
        for (;;) {
            ldp::OutlierLevel& L = lv.lv[n_levels];
            L.keys = pl.keys[n_levels]; L.cell = pl.cell[n_levels]; L.pts = pl.pts[n_levels];
            L.cap_mask = ws.cap_mask; L.h = h; L.pad = 0;
            for (int c = 0; c < 3; ++c) {
                L.vmin[c] = mn[c] - h * 0.5;                                  // ldp_voxel_insert_kernel's expression
                L.gmax[c] = (int)std::floor((mx[c] - L.vmin[c]) / h);
            }
            ws.keys = pl.keys[n_levels];
            e = cudaMemsetAsync(ws.count, 0, ((size_t)n + 1) * sizeof(int), st);
            if (e == cudaSuccess) e = cudaMemsetAsync(ws.cursor, 0, (size_t)n * sizeof(int), st);
            if ((rc = check(e, "cudaMemsetAsync(outlier level)")) != LDP_OK) return rc;
            if ((rc = outlier_insert(xyz, n, h, nullptr, pl, grid, st, pl.vstat + 1)) != LDP_OK) return rc;
            rc = launch("ldp_voxel_count_kernel", ldp::ldp_voxel_count_kernel, dim3(grid), dim3(ldp::KV_THREADS), 0, st, (long long)n, ws);
            if (rc != LDP_OK) return rc;
            if ((rc = scan_exclusive(ws.count, ws.seg, n, ws.block_tot, nullptr, st)) != LDP_OK) return rc;
            rc = launch("ldp_voxel_group_kernel", ldp::ldp_voxel_group_kernel, dim3(grid), dim3(ldp::KV_THREADS), 0, st, (long long)n, ws,
                        (const int*)ws.seg);
            if (rc != LDP_OK) return rc;
            rc = launch("ldp_outlier_cells_kernel", ldp::ldp_outlier_cells_kernel, dim3(cgrid), dim3(ldp::KV_THREADS), 0, st, ws,
                        pl.cell[n_levels]);
            if (rc != LDP_OK) return rc;
            rc = launch("ldp_outlier_pack_kernel", ldp::ldp_outlier_pack_kernel, dim3(grid), dim3(ldp::KV_THREADS), 0, st, xyz,
                        (long long)n, (const int*)ws.members, pl.pts[n_levels]);
            if (rc != LDP_OK) return rc;
            ++n_levels;
            if (n_levels == ldp::OL_MAX_LEVELS || !(ext / h > 2.0)) break;
            h *= 8.0;
        }
    }
    rc = launch("ldp_outlier_levels_kernel", ldp::ldp_outlier_levels_kernel, dim3(1), dim3(1), 0, st, lv, n_levels, pl.levels);
    if (rc != LDP_OK) return rc;
    *n_levels_out = n_levels;
    return LDP_OK;
}

int ldp_statistical_outliers(const float* xyz, int64_t n, int32_t nb_neighbors, double std_ratio, int64_t* kept_idx_out,
                             double* mean_dist_out, double* stats_out, int32_t* status_out, void* workspace, size_t workspace_bytes,
                             void* stream) {
    begin_call();
    if (nb_neighbors < 1 || nb_neighbors > ldp::OL_MAX_K) return fail(LDP_ERR_INVALID, "nb_neighbors must lie in [1, 64]");
    if (!(std_ratio > 0.0)) return fail(LDP_ERR_INVALID, "std_ratio must be positive");
    if (!status_out) return fail(LDP_ERR_INVALID, "null status_out");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    int rc = check(cudaMemsetAsync(status_out, 0, 3 * sizeof(int32_t), st), "cudaMemsetAsync(status)");
    if (rc != LDP_OK || n == 0) return rc;
    if (!xyz || !kept_idx_out || !workspace) return fail(LDP_ERR_INVALID, "null pointer");
    OutlierPlan pl;
    size_t need = 0;
    if ((rc = outlier_plan(n, workspace, &pl, &need)) != LDP_OK) return rc;
    if (workspace_bytes < need) return fail(LDP_ERR_WORKSPACE, "outlier workspace too small");
    const int k = (int)std::min<int64_t>(nb_neighbors, n);
    int n_levels = 0;
    if ((rc = knn_pyramid(xyz, n, k, pl, st, status_out, &n_levels)) != LDP_OK || n_levels == 0) return rc;
    ldp::VoxelWs& ws = pl.vws;
    const unsigned grid = (unsigned)((n + ldp::KV_THREADS - 1) / ldp::KV_THREADS);

    // 3. k nearest, per-point mean distance
    double* m = mean_dist_out ? mean_dist_out : pl.m;
    double* stats = stats_out ? stats_out : pl.stats;
    {
        KernelTimer kt(st, "ldp_outlier_knn_kernel");
        const unsigned kgrid = (unsigned)((n + ldp::OL_THREADS - 1) / ldp::OL_THREADS);
        rc = launch("ldp_outlier_knn_kernel", ldp::ldp_outlier_knn_kernel<ldp::KNN_MEAN>, dim3(kgrid), dim3(ldp::OL_THREADS),
                    (size_t)k * ldp::OL_THREADS * sizeof(double), st, (const ldp::OutlierLevel*)pl.levels, n_levels, (long long)n, k,
                    g_outlier_shells > 0 ? g_outlier_shells : ldp::OL_DEFAULT_SHELLS, m, (int*)status_out, ldp::NormalArgs{});
        if (rc != LDP_OK) return rc;
    }

    // 4. threshold (first pass: the mean; second: the spread around it, std and threshold), keep flags, kept indices
    KernelTimer kt(st, "ldp_outlier_threshold");
    const long long n_part = (n + ldp::OL_CHUNK - 1) / ldp::OL_CHUNK;
    const unsigned pgrid = (unsigned)((n_part + ldp::KV_THREADS - 1) / ldp::KV_THREADS);
    for (int second = 0; second < 2; ++second) {
        rc = launch("ldp_outlier_partial_kernel", ldp::ldp_outlier_partial_kernel, dim3(pgrid), dim3(ldp::KV_THREADS), 0, st,
                    (const double*)m, (long long)n, second ? (const double*)stats : nullptr, pl.part);
        if (rc != LDP_OK) return rc;
        rc = launch("ldp_outlier_stats_kernel", ldp::ldp_outlier_stats_kernel, dim3(1), dim3(ldp::OL_FINAL), 0, st, (const double*)pl.part,
                    n_part, (long long)n, std_ratio, second, stats);
        if (rc != LDP_OK) return rc;
    }
    rc = launch("ldp_outlier_flag_kernel", ldp::ldp_outlier_flag_kernel, dim3(grid), dim3(ldp::KV_THREADS), 0, st, (const double*)m,
                (long long)n, (const double*)stats, ws.flag);
    if (rc != LDP_OK) return rc;
    if ((rc = scan_exclusive(ws.flag, ws.rank, n, ws.block_tot, (int*)status_out + 1, st)) != LDP_OK) return rc;
    return launch("ldp_outlier_kept_kernel", ldp::ldp_outlier_kept_kernel, dim3(grid), dim3(ldp::KV_THREADS), 0, st, (const int*)ws.flag,
                  (const int*)ws.rank, (long long)n, reinterpret_cast<long long*>(kept_idx_out));
}

// ---- oriented normals (ldp_outlier.cu: ldp_outlier_knn_kernel<KNN_NORMALS> and its epilogue)
int ldp_normals_workspace_bytes(int64_t n, int32_t k, size_t* bytes_out) {
    if (!bytes_out) return fail(LDP_ERR_INVALID, "null bytes_out");
    if (k < 3 || k > ldp::OL_MAX_K) return fail(LDP_ERR_INVALID, "k must lie in [3, 64]");
    OutlierPlan pl;
    return outlier_plan(n, nullptr, &pl, bytes_out, false);
}

int ldp_estimate_normals(const float* xyz, int64_t n, int32_t k, const float* centers, int32_t n_centers, const int32_t* center_idx,
                         float* normals_out, float* curvature_out, int32_t* knn_idx_out, int32_t* status_out, void* workspace,
                         size_t workspace_bytes, void* stream) {
    begin_call();
    if (k < 3 || k > ldp::OL_MAX_K) return fail(LDP_ERR_INVALID, "k must lie in [3, 64]");
    if (center_idx && !centers) return fail(LDP_ERR_INVALID, "center_idx needs centers");
    if (centers && n_centers < 1) return fail(LDP_ERR_INVALID, "n_centers must be >= 1 when centers are given");
    if (!status_out) return fail(LDP_ERR_INVALID, "null status_out");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    int rc = check(cudaMemsetAsync(status_out, 0, 3 * sizeof(int32_t), st), "cudaMemsetAsync(status)");
    if (rc != LDP_OK || n == 0) return rc;
    if (!xyz || !normals_out || !workspace) return fail(LDP_ERR_INVALID, "null pointer");
    OutlierPlan pl;
    size_t need = 0;
    if ((rc = outlier_plan(n, workspace, &pl, &need, false)) != LDP_OK) return rc;
    if (workspace_bytes < need) return fail(LDP_ERR_WORKSPACE, "normals workspace too small");
    const int k_eff = (int)std::min<int64_t>(k, n);
    int n_levels = 0;
    if ((rc = knn_pyramid(xyz, n, k_eff, pl, st, status_out, &n_levels)) != LDP_OK || n_levels == 0) return rc;
    KernelTimer kt(st, "ldp_normals_knn_kernel");
    const ldp::NormalArgs na{xyz, centers, center_idx, normals_out, curvature_out, knn_idx_out, centers ? n_centers : 0, 0};
    const unsigned kgrid = (unsigned)((n + ldp::OL_THREADS - 1) / ldp::OL_THREADS);
    return launch("ldp_outlier_knn_kernel", ldp::ldp_outlier_knn_kernel<ldp::KNN_NORMALS>, dim3(kgrid), dim3(ldp::OL_THREADS),
                  (size_t)k_eff * ldp::OL_THREADS * (sizeof(double) + sizeof(int)), st, (const ldp::OutlierLevel*)pl.levels, n_levels,
                  (long long)n, k_eff, g_outlier_shells > 0 ? g_outlier_shells : ldp::OL_DEFAULT_SHELLS, (double*)nullptr,
                  (int*)status_out, na);
}

// ---- 3DGS initialisation (ldp_outlier.cu: ldp_outlier_knn_kernel<KNN_GAUSSIANS> and its epilogue; ldp_output.cu)
int ldp_gaussian_workspace_bytes(int64_t n, int32_t k, size_t* bytes_out) {
    if (!bytes_out) return fail(LDP_ERR_INVALID, "null bytes_out");
    if (k < 1 || k > ldp::OL_MAX_K - 1) return fail(LDP_ERR_INVALID, "k must lie in [1, 63]");
    OutlierPlan pl;
    return outlier_plan(n, nullptr, &pl, bytes_out, false);
}

int ldp_gaussian_init(const float* xyz, const float* rgb, const float* normals, int64_t n, int32_t k, double opacity, double flatten,
                      float* sh_dc_out, float* opacity_out, float* scales_out, float* rotations_out, float* dist2_out,
                      int32_t* status_out, void* workspace, size_t workspace_bytes, void* stream) {
    begin_call();
    if (k < 1 || k > ldp::OL_MAX_K - 1) return fail(LDP_ERR_INVALID, "k must lie in [1, 63]");
    if (!(opacity > 0.0 && opacity < 1.0)) return fail(LDP_ERR_INVALID, "opacity must lie in (0, 1)");
    if (!(flatten > 0.0 && flatten <= 1.0)) return fail(LDP_ERR_INVALID, "flatten must lie in (0, 1]");
    if (flatten < 1.0 && !normals) return fail(LDP_ERR_INVALID, "flatten < 1 needs normals");
    if (!status_out) return fail(LDP_ERR_INVALID, "null status_out");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    int rc = check(cudaMemsetAsync(status_out, 0, 3 * sizeof(int32_t), st), "cudaMemsetAsync(status)");
    if (rc != LDP_OK || n == 0) return rc;
    if (!xyz || !rgb || !sh_dc_out || !opacity_out || !scales_out || !rotations_out || !workspace)
        return fail(LDP_ERR_INVALID, "null pointer");
    OutlierPlan pl;
    size_t need = 0;
    if ((rc = outlier_plan(n, workspace, &pl, &need, false)) != LDP_OK) return rc;
    if (workspace_bytes < need) return fail(LDP_ERR_WORKSPACE, "gaussian workspace too small");
    const int kk = (int)std::min<int64_t>((int64_t)k + 1, n);          // k_eff + 1: the point itself and its k_eff nearest
    int n_levels = 0;
    if ((rc = knn_pyramid(xyz, n, kk, pl, st, status_out, &n_levels)) != LDP_OK || n_levels == 0) return rc;
    KernelTimer kt(st, "ldp_gaussian_knn_kernel");
    const ldp::GaussianArgs ga{rgb, normals, sh_dc_out, opacity_out, scales_out, rotations_out, dist2_out, std::log(flatten),
                               (float)std::log(opacity / (1.0 - opacity)), 0};
    const unsigned kgrid = (unsigned)((n + ldp::OL_THREADS - 1) / ldp::OL_THREADS);
    return launch("ldp_outlier_knn_kernel", ldp::ldp_outlier_knn_kernel<ldp::KNN_GAUSSIANS>, dim3(kgrid), dim3(ldp::OL_THREADS),
                  (size_t)kk * ldp::OL_THREADS * sizeof(double), st, (const ldp::OutlierLevel*)pl.levels, n_levels, (long long)n, kk,
                  g_outlier_shells > 0 ? g_outlier_shells : ldp::OL_DEFAULT_SHELLS, (double*)nullptr, (int*)status_out, ga);
}

int ldp_pack_gaussian_ply_records(const float* xyz, const float* normals, const float* sh_dc, const float* opacity, const float* scales,
                                  const float* rotations, int64_t n, const int64_t* n_dev, int32_t sh_degree, uint8_t* records_out,
                                  void* stream) {
    begin_call();
    if (n < 0) return fail(LDP_ERR_INVALID, "negative point count");
    if (sh_degree < 0 || sh_degree > 3) return fail(LDP_ERR_INVALID, "sh_degree must lie in [0, 3]");
    if (n == 0) return LDP_OK;
    if (!xyz || !sh_dc || !opacity || !scales || !rotations || !records_out) return fail(LDP_ERR_INVALID, "null pointer");
    if (reinterpret_cast<uintptr_t>(records_out) & 3u) return fail(LDP_ERR_INVALID, "records_out must be 4-byte aligned");
    static const decltype(&ldp::ldp_gaussian_records_kernel<0>) k_records[4] = {
        ldp::ldp_gaussian_records_kernel<0>, ldp::ldp_gaussian_records_kernel<1>, ldp::ldp_gaussian_records_kernel<2>,
        ldp::ldp_gaussian_records_kernel<3>};
    const long long floats = (long long)n * (17 + 3 * ((sh_degree + 1) * (sh_degree + 1) - 1));
    const unsigned grid = (unsigned)((floats + ldp::KO_THREADS - 1) / ldp::KO_THREADS);
    KernelTimer kt(reinterpret_cast<cudaStream_t>(stream), "ldp_gaussian_records_kernel");
    return launch("ldp_gaussian_records_kernel", k_records[sh_degree], dim3(grid), dim3(ldp::KO_THREADS), 0,
                  reinterpret_cast<cudaStream_t>(stream), xyz, normals, sh_dc, opacity, scales, rotations, (long long)n,
                  reinterpret_cast<const long long*>(n_dev), reinterpret_cast<float*>(records_out));
}

int ldp_set_sm_reserve(int n_sms) {
    if (n_sms < 0 || n_sms >= sm_count()) return fail(LDP_ERR_INVALID, "sm reserve out of range");
    g_sm_reserve = n_sms;
    return LDP_OK;
}

int64_t ldp_struct_size(int which) {
    switch (which) {
        case 0: return (int64_t)sizeof(ldp_params);
        case 1: return (int64_t)sizeof(ldp_ref_desc);
        case 2: return (int64_t)sizeof(ldp_outputs);
        case 3: return (int64_t)sizeof(ldp_lens);
        default: return -1;
    }
}

int ldp_workspace_bytes(const ldp_params* params, size_t* bytes_out) {
    if (!bytes_out) return fail(LDP_ERR_INVALID, "null bytes_out");
    Plan plan;
    int rc = make_plan(params, nullptr, &plan);
    if (rc != LDP_OK) return rc;
    *bytes_out = plan.bytes + 256;
    return LDP_OK;
}

int ldp_densify_refs(const ldp_params* params, const ldp_ref_desc* refs, const double* uniforms,
                     const ldp_outputs* out, void* workspace, size_t workspace_bytes, void* stream) {
    begin_call();
    int rc = check_outputs(params, out);
    if (rc != LDP_OK) return rc;
    if (params->n_refs == 0) return LDP_OK;
    if (!refs || !workspace) return fail(LDP_ERR_INVALID, "null refs/workspace");
    if (params->rng_mode == LDP_RNG_EXPLICIT && !params->no_filter && !uniforms)
        return fail(LDP_ERR_INVALID, "explicit rng mode needs a uniform stream");
    Plan plan;
    if ((rc = bind_plan(params, workspace, workspace_bytes, &plan)) != LDP_OK) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if ((rc = clear_launch_state(plan, st)) != LDP_OK) return rc;
    if ((rc = launch_sample(params, refs, uniforms, out, plan, st)) != LDP_OK) return rc;
    return launch_triangulate(params, refs, out, plan, 1, st);
}

int ldp_sample_refs(const ldp_params* params, const ldp_ref_desc* refs, const double* uniforms,
                    const ldp_outputs* out, void* workspace, size_t workspace_bytes, void* stream) {
    begin_call();
    if (!params || !out || !out->status || !out->n_samples || !out->sel_idx) return fail(LDP_ERR_INVALID, "sample stage needs status, n_samples, sel_idx");
    if (params->n_refs == 0) return LDP_OK;
    if (!refs || !workspace) return fail(LDP_ERR_INVALID, "null refs/workspace");
    if (params->rng_mode == LDP_RNG_EXPLICIT && !params->no_filter && !uniforms)
        return fail(LDP_ERR_INVALID, "explicit rng mode needs a uniform stream");
    Plan plan;
    int rc = bind_plan(params, workspace, workspace_bytes, &plan);
    if (rc != LDP_OK) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if ((rc = clear_launch_state(plan, st)) != LDP_OK) return rc;
    return launch_sample(params, refs, uniforms, out, plan, st);
}

int ldp_triangulate_samples(const ldp_params* params, const ldp_ref_desc* refs, const ldp_outputs* out,
                            void* workspace, size_t workspace_bytes, void* stream) {
    begin_call();
    int rc = check_outputs(params, out);
    if (rc != LDP_OK) return rc;
    if (!out->sel_idx) return fail(LDP_ERR_INVALID, "triangulate stage reads out->sel_idx / out->n_samples");
    if (params->n_refs == 0) return LDP_OK;
    if (!refs || !workspace) return fail(LDP_ERR_INVALID, "null refs/workspace");
    Plan plan;
    if ((rc = bind_plan(params, workspace, workspace_bytes, &plan)) != LDP_OK) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if ((rc = clear_launch_state(plan, st)) != LDP_OK) return rc;
    return launch_triangulate(params, refs, out, plan, 0, st);
}

int ldp_depth_workspace_bytes(const ldp_params* params, size_t* bytes_out) {
    if (!bytes_out) return fail(LDP_ERR_INVALID, "null bytes_out");
    DepthPlan dp;
    const int rc = make_depth_plan(params, nullptr, &dp);
    if (rc != LDP_OK) return rc;
    *bytes_out = dp.bytes + 256;
    return LDP_OK;
}

int ldp_depth_maps(const ldp_params* params, const ldp_ref_desc* refs, double min_certainty, float* depth, float* err, float* xyz,
                   uint8_t* flags, int64_t* kept, void* workspace, size_t workspace_bytes, void* stream) {
    begin_call();
    if (!params) return fail(LDP_ERR_INVALID, "null params");
    if (!(min_certainty > 0.0 && min_certainty <= 1.0)) return fail(LDP_ERR_INVALID, "min_certainty must lie in (0, 1]");
    if (params->multiview && params->no_filter) return fail(LDP_ERR_INVALID, "multiview needs the filters (no_filter = 0)");
    if (params->multiview && !(params->multiview_min_cert > 0.0f && params->multiview_min_cert <= 1.0f))
        return fail(LDP_ERR_INVALID, "multiview_min_cert must lie in (0, 1]");
    DepthPlan dp;
    int rc = make_depth_plan(params, nullptr, &dp);
    if (rc != LDP_OK) return rc;
    if (params->n_refs == 0) return LDP_OK;
    if (!refs || !depth || !kept || !workspace) return fail(LDP_ERR_INVALID, "null refs / depth / kept / workspace");
    char* base = reinterpret_cast<char*>(align_up(reinterpret_cast<size_t>(workspace), 256));
    if ((rc = make_depth_plan(params, base, &dp)) != LDP_OK) return rc;
    if (dp.bytes + (size_t)(base - static_cast<char*>(workspace)) > workspace_bytes) return fail(LDP_ERR_WORKSPACE, "workspace too small");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int R = params->n_refs, N = params->H * params->W;
    if ((rc = check(cudaMemsetAsync(kept, 0, (size_t)R * sizeof(int64_t), st), "cudaMemsetAsync(kept)")) != LDP_OK) return rc;
    if ((rc = check(cudaMemsetAsync(dp.fix_count, 0, (size_t)R * sizeof(int32_t), st), "cudaMemsetAsync(fix_count)")) != LDP_OK)
        return rc;
    const ldp::GeomArgs ga = make_geom_args(params, 0, 0);
    const ldp::DepthArgs d{depth, err, xyz, flags, reinterpret_cast<unsigned long long*>(kept), dp.fix_list, dp.fix_count,
                           (float)min_certainty, N};
    // enough CTAs per view for about 16 resident per SM over the launch; each strides over its share of the view's map
    const int tiles = (N + ldp::K2_THREADS - 1) / ldp::K2_THREADS;
    const int per_view = std::max(1, std::min(tiles, (sm_count() * 16 + R - 1) / R));
    { KernelTimer kt(st, "ldp_depth_kernel");
      auto* kd = params->multiview ? (params->lens ? ldp::ldp_depth_kernel<true, true> : ldp::ldp_depth_kernel<false, true>)
                                   : (params->lens ? ldp::ldp_depth_kernel<true, false> : ldp::ldp_depth_kernel<false, false>);
      if ((rc = launch("ldp_depth_kernel", kd, dim3((unsigned)per_view, (unsigned)R), dim3(ldp::K2_THREADS), 0, st, *params, refs, ga, d))
          != LDP_OK)
          return rc; }
    KernelTimer kt(st, "ldp_depth_fix_kernel");
    auto* kf = params->multiview ? (params->lens ? ldp::ldp_depth_fix_kernel<true, true> : ldp::ldp_depth_fix_kernel<false, true>)
                                 : (params->lens ? ldp::ldp_depth_fix_kernel<true, false> : ldp::ldp_depth_fix_kernel<false, false>);
    return launch("ldp_depth_fix_kernel", kf, dim3(ldp::KDF_BLOCKS, (unsigned)R), dim3(ldp::K2_THREADS), 0, st, *params, refs, ga, d);
}

int ldp_postprocess_certainty(const ldp_params* params, const ldp_ref_desc* refs, float* outp,
                              size_t ref_stride, size_t plane_stride, void* stream) {
    begin_call();
    if (!params || params->n_refs < 0 || params->H <= 0 || params->W <= 0) return fail(LDP_ERR_INVALID, "bad shape");
    if (params->n_refs == 0) return LDP_OK;
    if (!refs || !outp) return fail(LDP_ERR_INVALID, "null refs/out");
    if ((long long)params->H * params->W > (1ll << 24)) return fail(LDP_ERR_INVALID, "map too large");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int N = params->H * params->W;
    const int bx = std::min((N + ldp::KP_THREADS - 1) / ldp::KP_THREADS, 4 * sm_count());
    const dim3 grid((unsigned)bx, LDP_MAX_NN, (unsigned)params->n_refs);
    KernelTimer kt(st, "ldp_prologue_kernel");
    return launch("ldp_prologue_kernel", ldp::ldp_prologue_kernel, grid, dim3(ldp::KP_THREADS), 0, st, *params, refs, outp, ref_stride,
                  plane_stride);
}


// ---- cross-view depth consistency (ldp_consistency.cu; the compaction is the outlier filter's scan + ldp_outlier_kept_kernel).
// Last in the file: the device compiler places kernel instantiations in reverse order of first use, so the new kernels go
// ahead of all others and the layout of the existing kernels relative to one another does not change.
struct ConsistencyPlan {
    int* flag;                             // [n] keep flags
    int* rank;                             // [n] their exclusive prefix
    int* block_tot;                        // the scan's per-block totals
};

static int consistency_plan(int64_t n, void* base, ConsistencyPlan* pl, size_t* bytes) {
    if (n < 0 || n > 500000000ll) return fail(LDP_ERR_INVALID, "depth consistency: bad point count");
    const size_t N = (size_t)std::max<int64_t>(n, 1);
    Carver c{static_cast<char*>(base)};
    pl->flag = c.take<int>(N);
    pl->rank = c.take<int>(N);
    pl->block_tot = c.take<int>(N / ldp::SC_THREADS + 2);
    *bytes = c.off;
    return LDP_OK;
}

int ldp_consistency_workspace_bytes(int64_t n, size_t* bytes_out) {
    if (!bytes_out) return fail(LDP_ERR_INVALID, "null bytes_out");
    ConsistencyPlan pl;
    return consistency_plan(n, nullptr, &pl, bytes_out);
}

int ldp_depth_consistency(const float* xyz, int64_t n, const int32_t* owner, const float* const* depth_ptrs, int32_t H, int32_t W,
                          const float* P, const double* scales, const ldp_lens* lens, int32_t n_views, double rel_tol,
                          int32_t min_views, int32_t max_violations, int32_t* n_consistent_out, int32_t* n_violations_out,
                          int64_t* kept_idx_out, int32_t* status_out, void* workspace, size_t workspace_bytes, void* stream) {
    begin_call();
    if (!(rel_tol > 0.0 && rel_tol < 1.0)) return fail(LDP_ERR_INVALID, "rel_tol must lie in (0, 1)");
    if (min_views < 0 || max_violations < 0) return fail(LDP_ERR_INVALID, "min_views and max_violations must be >= 0");
    if (n_views < 0 || H <= 0 || W <= 0 || (long long)H * W > 0x3fffffffLL) return fail(LDP_ERR_INVALID, "bad view count or map shape");
    if (n_views > 0 && (!depth_ptrs || !P || !scales)) return fail(LDP_ERR_INVALID, "null depth_ptrs / P / scales");
    if (!status_out) return fail(LDP_ERR_INVALID, "null status_out");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    int rc = check(cudaMemsetAsync(status_out, 0, 2 * sizeof(int32_t), st), "cudaMemsetAsync(status)");
    if (rc != LDP_OK || n == 0) return rc;
    if (!xyz || !kept_idx_out || !workspace) return fail(LDP_ERR_INVALID, "null pointer");
    ConsistencyPlan pl;
    size_t need = 0;
    if ((rc = consistency_plan(n, workspace, &pl, &need)) != LDP_OK) return rc;
    if (workspace_bytes < need) return fail(LDP_ERR_WORKSPACE, "consistency workspace too small");
    const unsigned grid = (unsigned)((n + ldp::CS_THREADS - 1) / ldp::CS_THREADS);
    rc = launch("ldp_consistency_check_kernel", owner ? ldp::ldp_consistency_check_kernel<true> : ldp::ldp_consistency_check_kernel<false>,
                dim3(grid), dim3(ldp::CS_THREADS), 0, st, xyz, (const int*)owner, (long long)n, (int)n_views, (int*)status_out);
    if (rc != LDP_OK) return rc;
    const ldp::ConsistencyArgs a{xyz, (const int*)owner, depth_ptrs, P, scales, lens, (int*)n_consistent_out, (int*)n_violations_out,
                                 pl.flag, (int*)status_out, (long long)n, rel_tol, (int)n_views, (int)H, (int)W, (int)min_views,
                                 (int)max_violations};
    // a few resident CTAs per SM; each strides over the cloud, so a table of one chunk is staged once per CTA
    const unsigned cgrid = (unsigned)std::min<long long>(grid, (long long)sm_count() * 8);
    {
        KernelTimer kt(st, "ldp_consistency_kernel");
        rc = launch("ldp_consistency_kernel", lens ? ldp::ldp_consistency_kernel<true> : ldp::ldp_consistency_kernel<false>,
                    dim3(cgrid), dim3(ldp::CS_THREADS), 0, st, a);
        if (rc != LDP_OK) return rc;
    }
    if ((rc = scan_exclusive(pl.flag, pl.rank, n, pl.block_tot, (int*)status_out + 1, st)) != LDP_OK) return rc;
    const unsigned kgrid = (unsigned)((n + ldp::KV_THREADS - 1) / ldp::KV_THREADS);
    return launch("ldp_outlier_kept_kernel", ldp::ldp_outlier_kept_kernel, dim3(kgrid), dim3(ldp::KV_THREADS), 0, st, (const int*)pl.flag,
                  (const int*)pl.rank, (long long)n, reinterpret_cast<long long*>(kept_idx_out));
}

// ---- depth-map fusion (ldp_fusion.cu; the compaction is the outlier filter's scan + ldp_outlier_kept_kernel).  Last in the
// file for the reason given above the consistency check.
int ldp_depth_colors(const ldp_params* params, const ldp_ref_desc* refs, const uint8_t* flags, float* rgb_out, void* stream) {
    begin_call();
    DepthPlan dp;
    int rc = make_depth_plan(params, nullptr, &dp);
    if (rc != LDP_OK) return rc;
    if (params->n_refs == 0) return LDP_OK;
    if (!refs || !flags || !rgb_out) return fail(LDP_ERR_INVALID, "null refs / flags / rgb_out");
    const int R = params->n_refs, N = params->H * params->W;
    const int tiles = (N + ldp::K2_THREADS - 1) / ldp::K2_THREADS;
    const int per_view = std::max(1, std::min(tiles, (sm_count() * 16 + R - 1) / R));
    KernelTimer kt(static_cast<cudaStream_t>(stream), "ldp_depth_color_kernel");
    return launch("ldp_depth_color_kernel", ldp::ldp_depth_color_kernel, dim3((unsigned)per_view, (unsigned)R), dim3(ldp::K2_THREADS), 0,
                  static_cast<cudaStream_t>(stream), *params, refs, flags, rgb_out, N);
}

struct FusionPlan {
    uint8_t* kept;                         // [V*N] pass 1's keep flags
    int* n_cons;                           // [V*N] pass 1's consistent counts
    int* flag;                             // [V*N] emit flags
    int* rank;                             // [V*N] their exclusive prefix
    int* block_tot;                        // the scan's per-block totals
};

static int fusion_plan(int32_t n_views, int32_t H, int32_t W, void* base, FusionPlan* pl, size_t* bytes) {
    if (n_views < 0 || H <= 0 || W <= 0 || (long long)H * W > 0x3fffffffLL) return fail(LDP_ERR_INVALID, "bad view count or map shape");
    const long long total = (long long)n_views * H * W;
    if (total >= (1ll << 31)) return fail(LDP_ERR_INVALID, "fusion: n_views * H * W must be below 2^31 (int32 ranks)");
    const size_t T = (size_t)std::max<long long>(total, 1);
    Carver c{static_cast<char*>(base)};
    pl->kept = c.take<uint8_t>(T);
    pl->n_cons = c.take<int>(T);
    pl->flag = c.take<int>(T);
    pl->rank = c.take<int>(T);
    pl->block_tot = c.take<int>(T / ldp::SC_THREADS + 2);
    *bytes = c.off;
    return LDP_OK;
}

int ldp_fuse_workspace_bytes(int32_t n_views, int32_t H, int32_t W, size_t* bytes_out) {
    if (!bytes_out) return fail(LDP_ERR_INVALID, "null bytes_out");
    FusionPlan pl;
    return fusion_plan(n_views, H, W, nullptr, &pl, bytes_out);
}

// both fusion entry points; normal_ptrs = NULL: ldp_fuse_depth_maps (the <LENS, false> kernels)
static int fuse_maps(const float* const* depth_ptrs, const float* const* xyz_ptrs, const float* const* rgb_ptrs,
                     const float* const* err_ptrs, const float* const* normal_ptrs, int32_t n_views, int32_t H, int32_t W,
                     const float* P, const double* scales, const ldp_lens* lens, double rel_tol, double cos_max, int32_t min_views,
                     int32_t max_violations, float* xyz_out, float* rgb_out, float* err_out, float* normals_out,
                     int32_t* n_views_out, int32_t* n_consistent_out, int64_t* source_out, int32_t* status_out, void* workspace,
                     size_t workspace_bytes, void* stream) {
    if (!(rel_tol > 0.0 && rel_tol < 1.0)) return fail(LDP_ERR_INVALID, "rel_tol must lie in (0, 1)");
    if (min_views < 0 || max_violations < 0) return fail(LDP_ERR_INVALID, "min_views and max_violations must be >= 0");
    FusionPlan pl;
    size_t need = 0;
    int rc = fusion_plan(n_views, H, W, nullptr, &pl, &need);
    if (rc != LDP_OK) return rc;
    if (!status_out) return fail(LDP_ERR_INVALID, "null status_out");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    rc = check(cudaMemsetAsync(status_out, 0, 2 * sizeof(int32_t), st), "cudaMemsetAsync(status)");
    if (rc != LDP_OK || n_views == 0) return rc;
    if (!depth_ptrs || !xyz_ptrs || !rgb_ptrs || !err_ptrs || !P || !scales) return fail(LDP_ERR_INVALID, "null view table");
    if (!xyz_out || !rgb_out || !err_out || !n_views_out || !n_consistent_out || !source_out || !workspace)
        return fail(LDP_ERR_INVALID, "null output or workspace");
    if ((rc = fusion_plan(n_views, H, W, workspace, &pl, &need)) != LDP_OK) return rc;
    if (workspace_bytes < need) return fail(LDP_ERR_WORKSPACE, "fusion workspace too small");
    const long long total = (long long)n_views * H * W;
    const bool nrm = normal_ptrs != nullptr;
    const ldp::FusionArgs a{depth_ptrs, xyz_ptrs, rgb_ptrs, err_ptrs, P, scales, lens, pl.kept, pl.n_cons, pl.flag,
                            reinterpret_cast<const long long*>(source_out), xyz_out, rgb_out, err_out, (int*)n_views_out,
                            (int*)n_consistent_out, (int*)status_out, total, rel_tol, (int)n_views, (int)H, (int)W, (int)(H * W),
                            (int)min_views, (int)max_violations, normal_ptrs, normals_out, cos_max};
    rc = launch("ldp_fusion_check_kernel", nrm ? ldp::ldp_fusion_check_kernel<true> : ldp::ldp_fusion_check_kernel<false>,
                dim3((unsigned)((n_views + ldp::CS_THREADS - 1) / ldp::CS_THREADS)), dim3(ldp::CS_THREADS), 0, st, a);
    if (rc != LDP_OK) return rc;
    // a few resident CTAs per SM; each strides over the maps, so a table of one chunk is staged once per CTA
    const unsigned grid = (unsigned)std::min<long long>((total + ldp::CS_THREADS - 1) / ldp::CS_THREADS, (long long)sm_count() * 8);
    const int which = (lens ? 2 : 0) + (nrm ? 1 : 0);
    {
        KernelTimer kt(st, "ldp_fusion_verdict_kernel");
        auto* k = (which == 0) ? ldp::ldp_fusion_verdict_kernel<false, false> : (which == 1) ? ldp::ldp_fusion_verdict_kernel<false, true>
                : (which == 2) ? ldp::ldp_fusion_verdict_kernel<true, false> : ldp::ldp_fusion_verdict_kernel<true, true>;
        if ((rc = launch("ldp_fusion_verdict_kernel", k, dim3(grid), dim3(ldp::CS_THREADS), 0, st, a)) != LDP_OK) return rc;
    }
    {
        KernelTimer kt(st, "ldp_fusion_emit_kernel");
        auto* k = (which == 0) ? ldp::ldp_fusion_emit_kernel<false, false> : (which == 1) ? ldp::ldp_fusion_emit_kernel<false, true>
                : (which == 2) ? ldp::ldp_fusion_emit_kernel<true, false> : ldp::ldp_fusion_emit_kernel<true, true>;
        if ((rc = launch("ldp_fusion_emit_kernel", k, dim3(grid), dim3(ldp::CS_THREADS), 0, st, a)) != LDP_OK) return rc;
    }
    if ((rc = scan_exclusive(pl.flag, pl.rank, total, pl.block_tot, (int*)status_out + 1, st)) != LDP_OK) return rc;
    const unsigned kgrid = (unsigned)((total + ldp::KV_THREADS - 1) / ldp::KV_THREADS);
    rc = launch("ldp_outlier_kept_kernel", ldp::ldp_outlier_kept_kernel, dim3(kgrid), dim3(ldp::KV_THREADS), 0, st, (const int*)pl.flag,
                (const int*)pl.rank, total, reinterpret_cast<long long*>(source_out));
    if (rc != LDP_OK) return rc;
    KernelTimer kt(st, "ldp_fusion_sum_kernel");
    auto* k = (which == 0) ? ldp::ldp_fusion_sum_kernel<false, false> : (which == 1) ? ldp::ldp_fusion_sum_kernel<false, true>
            : (which == 2) ? ldp::ldp_fusion_sum_kernel<true, false> : ldp::ldp_fusion_sum_kernel<true, true>;
    return launch("ldp_fusion_sum_kernel", k, dim3(grid), dim3(ldp::CS_THREADS), 0, st, a);
}

int ldp_fuse_depth_maps(const float* const* depth_ptrs, const float* const* xyz_ptrs, const float* const* rgb_ptrs,
                        const float* const* err_ptrs, int32_t n_views, int32_t H, int32_t W, const float* P, const double* scales,
                        const ldp_lens* lens, double rel_tol, int32_t min_views, int32_t max_violations, float* xyz_out,
                        float* rgb_out, float* err_out, int32_t* n_views_out, int32_t* n_consistent_out, int64_t* source_out,
                        int32_t* status_out, void* workspace, size_t workspace_bytes, void* stream) {
    begin_call();
    return fuse_maps(depth_ptrs, xyz_ptrs, rgb_ptrs, err_ptrs, nullptr, n_views, H, W, P, scales, lens, rel_tol, 0.0, min_views,
                     max_violations, xyz_out, rgb_out, err_out, nullptr, n_views_out, n_consistent_out, source_out, status_out,
                     workspace, workspace_bytes, stream);
}

int ldp_fuse_depth_maps_oriented(const float* const* depth_ptrs, const float* const* xyz_ptrs, const float* const* rgb_ptrs,
                                 const float* const* err_ptrs, const float* const* normal_ptrs, int32_t n_views, int32_t H, int32_t W,
                                 const float* P, const double* scales, const ldp_lens* lens, double rel_tol, double cos_max,
                                 int32_t min_views, int32_t max_violations, float* xyz_out, float* rgb_out, float* err_out,
                                 float* normals_out, int32_t* n_views_out, int32_t* n_consistent_out, int64_t* source_out,
                                 int32_t* status_out, void* workspace, size_t workspace_bytes, void* stream) {
    begin_call();
    if (!(cos_max > 0.0 && cos_max < 1.0)) return fail(LDP_ERR_INVALID, "cos_max must lie in (0, 1)");
    if (n_views > 0 && (!normal_ptrs || !normals_out)) return fail(LDP_ERR_INVALID, "null normal_ptrs / normals_out");
    return fuse_maps(depth_ptrs, xyz_ptrs, rgb_ptrs, err_ptrs, normal_ptrs, n_views, H, W, P, scales, lens, rel_tol, cos_max,
                     min_views, max_violations, xyz_out, rgb_out, err_out, normals_out, n_views_out, n_consistent_out, source_out,
                     status_out, workspace, workspace_bytes, stream);
}

int ldp_depth_normals(const float* const* depth_ptrs, const float* const* xyz_ptrs, int32_t n_views, int32_t H, int32_t W,
                      const float* centers, int32_t radius, double rel_tol, float* normals_out, float* curvature_out,
                      int32_t* status_out, void* stream) {
    begin_call();
    if (radius < 1 || radius > 3) return fail(LDP_ERR_INVALID, "radius must lie in [1, 3]");
    if (!(rel_tol > 0.0 && rel_tol < 1.0)) return fail(LDP_ERR_INVALID, "rel_tol must lie in (0, 1)");
    if (n_views < 0 || n_views > 65535 || H <= 0 || W <= 0) return fail(LDP_ERR_INVALID, "bad view count or map shape");
    if ((long long)n_views * H * W >= (1ll << 31)) return fail(LDP_ERR_INVALID, "normal maps: n_views * H * W must be below 2^31");
    if (!status_out) return fail(LDP_ERR_INVALID, "null status_out");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    int rc = check(cudaMemsetAsync(status_out, 0, 2 * sizeof(int32_t), st), "cudaMemsetAsync(status)");
    if (rc != LDP_OK || n_views == 0) return rc;
    if (!depth_ptrs || !xyz_ptrs || !centers || !normals_out) return fail(LDP_ERR_INVALID, "null map table / centers / normals_out");
    const int N = H * W;
    const int tiles_x = (W + ldp::DN_TILE - 1) / ldp::DN_TILE, tiles = tiles_x * ((H + ldp::DN_TILE - 1) / ldp::DN_TILE);
    const ldp::DepthNormalArgs a{depth_ptrs, xyz_ptrs, centers, normals_out, curvature_out, (int*)status_out, rel_tol, (int)n_views,
                                 (int)H, (int)W, N, tiles_x};
    const int per_view = std::max(1, std::min((N + ldp::CS_THREADS - 1) / ldp::CS_THREADS, (sm_count() * 8 + n_views - 1) / n_views));
    {
        KernelTimer kt(st, "ldp_depth_normals_check_kernel");
        rc = launch("ldp_depth_normals_check_kernel", ldp::ldp_depth_normals_check_kernel, dim3((unsigned)per_view, (unsigned)n_views),
                    dim3(ldp::CS_THREADS), 0, st, a);
        if (rc != LDP_OK) return rc;
    }
    KernelTimer kt(st, "ldp_depth_normals_kernel");
    auto* k = (radius == 1) ? ldp::ldp_depth_normals_kernel<1> : (radius == 2) ? ldp::ldp_depth_normals_kernel<2>
                                                                                : ldp::ldp_depth_normals_kernel<3>;
    return launch("ldp_depth_normals_kernel", k, dim3((unsigned)tiles, (unsigned)n_views), dim3(ldp::DN_THREADS), 0, st, a);
}

}  // extern "C"
