// C ABI of the densification path (include/ldp_b200.h).  Unity build: the kernels live in the two
// included translation units; this file carves the workspace, picks launch geometry and enqueues.
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <string>
#include <utility>
#include <vector>

#include "ldp_sample.cu"
#include "ldp_front.cu"
#include "ldp_geometry.cu"
#include "ldp_output.cu"
#include "ldp_select.cu"
#include "ldp_voxel.cu"
#include "ldp_outlier.cu"

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

constexpr int MAX_DEVICES = 64;
int current_device() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { (void)cudaGetLastError(); dev = 0; }
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
    if (cudaOccupancyMaxActiveClusters(&n, ldp::ldp_draw_kernel<2>, &cfg) != cudaSuccess) { (void)cudaGetLastError(); n = 0; }
    cache[csize] = n > 0 ? n : -1;
    return cache[csize];
}

int fail(int code, const char* what) {
    g_last_error = what ? what : "";
    return code;
}
int cuda_fail(cudaError_t e, const char* where) {
    g_last_error = std::string(where) + ": " + cudaGetErrorString(e);
    return LDP_ERR_CUDA;
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
        else { (void)cudaGetLastError(); cached[dev] = 148; }
    }
    return cached[dev];
}

constexpr size_t K1_SMEM_BUDGET = 200 * 1024;

// Every kernel is launched with programmatic dependent launch allowed: its CTAs may be scheduled while the previous
// kernel of the stream drains, and block in griddepcontrol.wait (ldp_device.cuh:grid_dependency_sync) until that kernel's
// memory is visible.  Hides the launch latency at each of the 6 kernel boundaries of a step.  LDP_PDL=0 turns it off.
template <typename... KArgs, typename... Args>
cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    static const int pdl = [] { const char* e = getenv("LDP_PDL"); return e ? atoi(e) : 1; }();
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

struct Plan {
    ldp::Workspace ws;
    ldp::SampleGeom geom;
    size_t bytes;
    size_t k1_smem;
    size_t prep_smem;
    int nb2;
    void* zero_base;        // launch state that every call clears with ONE memset: counters, per-view statistics, coverage
    size_t zero_bytes;      //   keys, tile partial slots
    int use_front;          // the fused persistent front kernel replaces stream + prep
    int front_grid;
    size_t front_smem;
};

// CTAs of the front kernel that are resident at once (2 per SM for up to 4 neighbour planes per stage, else 1)
int front_grid_size(int nn_stage, size_t smem) {
    (void)nn_stage;
    const size_t per_sm = 227 * 1024;
    int per = (int)(per_sm / (smem + 2048));
    if (per > 2) per = 2;
    if (per < 1) per = 1;
    return per * sm_count();
}

int choose_subbatches(int n_refs);

int next_epoch() {
    static int epoch = 0;
    epoch = (epoch % 0x3fffffff) + 1;      // never 0: the counters are cleared to 0 at the start of every call
    return epoch;
}

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
    g.prep_lean = (p->W <= 8192 && p->H <= 8192 && g.tile > 1) ? 1 : 0;
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
    // ---- which first stage: the fused persistent front kernel (ldp_front.cu) needs the vector path (16-byte aligned rows of
    //      W % 4 == 0 pixels), coverage tiles wider than a pixel, a known neighbour count <= 8 per view, no warped masks,
    //      and few enough tiles per view that the resident CTAs can park a whole view (see the deadlock note there)
    //      MEASURED SLOWER than the two kernels it replaces and therefore OFF unless LDP_FRONT=1 (profiles/r02_summary.md):
    //      131-140 us against 41 + 27 us at the bench shape.  With one quad per thread and tile every per-tile step (stage
    //      selection, block reductions, announcement, barriers) is paid per quad: 84 M warp instructions against 25 M.
    static const int front_mode = [] { const char* e = getenv("LDP_FRONT"); return e ? atoi(e) : 0; }();
    g.front_nn = p->nn_max;
    g.front_cache = 0;
    plan->use_front = 0;
    plan->front_grid = 0;
    plan->front_smem = 0;
    if (front_mode && !p->no_filter && p->W % 4 == 0 && p->scalar_loads == 0 && g.prep_lean && p->nn_max >= 1 && p->nn_max <= 8 &&
        (!p->prologue || p->no_warped_masks) && choose_subbatches(p->n_refs) == 1 && plan->prep_smem <= 16 * 1024) {
        size_t smem = ((size_t)ldp::KF_STAGES * g.front_nn + ldp::KF_PARK) * ldp::KF_TILE * sizeof(float) + plan->prep_smem;
        const size_t cache = (size_t)p->n_refs * ((size_t)g.front_nn * sizeof(void*) + sizeof(int));
        g.front_cache = (cache <= 12 * 1024) ? 1 : 0;        // what is left of the SM's shared memory beside two CTAs' rings
        if (g.front_cache) smem += cache;
        const int grid = front_grid_size(g.front_nn, smem);
        const size_t tpv = ((size_t)N + ldp::KF_TILE - 1) / ldp::KF_TILE;
        if (smem <= 200 * 1024 && tpv <= (size_t)3 * grid) { plan->use_front = 1; plan->front_grid = grid; plan->front_smem = smem; }
    }
    w.nblk = plan->use_front ? ((size_t)N + ldp::KF_TILE - 1) / ldp::KF_TILE : ((size_t)N + ldp::KS_SPAN - 1) / ldp::KS_SPAN;

    size_t off = 0;
    char* b = static_cast<char*>(base);
    auto carve = [&](size_t bytes) { char* q = b ? b + off : nullptr; off = align_up(off + bytes, 256); return q; };
    w.w = reinterpret_cast<float*>(carve(R * w.n_pad * sizeof(float)));
    w.bestk = reinterpret_cast<uint8_t*>(carve(R * w.n_pad));
    w.bitmap = reinterpret_cast<uint32_t*>(carve(R * w.n_words * sizeof(uint32_t)));
    w.gone = reinterpret_cast<uint32_t*>(carve(R * w.n_words * sizeof(uint32_t)));
    w.draw_cmax = 8;
    w.found = reinterpret_cast<int32_t*>(carve(R * w.draw_cmax * w.found_cap * sizeof(int32_t)));
    w.fcnt = reinterpret_cast<int32_t*>(carve(R * w.draw_cmax * sizeof(int32_t)));
    w.sel = reinterpret_cast<int32_t*>(carve(R * w.sel_cap * sizeof(int32_t)));
    w.pt0 = reinterpret_cast<float4*>(carve(R * w.sel_cap * sizeof(float4)));
    w.pt1 = reinterpret_cast<float4*>(carve(R * w.sel_cap * sizeof(float4)));
    w.dbgm = reinterpret_cast<float4*>(carve(p->collect_debug ? R * w.sel_cap * sizeof(float4) : 0));
    w.flags = reinterpret_cast<uint8_t*>(carve(R * w.sel_cap));
    w.topk_keys = reinterpret_cast<unsigned long long*>(carve(R * w.topk_cap * sizeof(unsigned long long)));
    w.csum = reinterpret_cast<double*>(carve(R * w.nchunk_pad * sizeof(double)));
    w.csum0 = reinterpret_cast<double*>(carve(R * w.nchunk_pad * sizeof(double)));
    w.dbgclk = reinterpret_cast<long long*>(carve(R * 32 * sizeof(long long)));
    plan->nb2 = (int)((w.sel_cap + ldp::K2_THREADS - 1) / ldp::K2_THREADS);
    w.blk_cnt = reinterpret_cast<int32_t*>(carve(R * plan->nb2 * LDP_MAX_NN * sizeof(int32_t)));
    w.blk_first = reinterpret_cast<int32_t*>(carve(R * plan->nb2 * LDP_MAX_NN * sizeof(int32_t)));
    w.fix_list = reinterpret_cast<int2*>(carve(R * w.sel_cap * sizeof(int2)));
    w.dstat = reinterpret_cast<int32_t*>(carve(R * sizeof(int32_t)));
    const size_t mv_slots = p->multiview ? R * w.sel_cap : 0;
    w.vmask = reinterpret_cast<int32_t*>(carve(mv_slots * sizeof(int32_t)));
    w.mvrec = reinterpret_cast<float4*>(carve(mv_slots * sizeof(float4)));
    // ---- the zero block (one memset per call, clear_launch_state): 8-byte items first
    {
        const size_t z0 = off;
        auto sub = [&](size_t bytes) { char* q = b ? b + off : nullptr; off += align_up(bytes, 8); return q; };
        w.vword = reinterpret_cast<unsigned long long*>(sub(R * sizeof(unsigned long long)));
        w.gbins = reinterpret_cast<unsigned long long*>(sub(R * w.bins_cap * sizeof(unsigned long long)));
        w.partial = reinterpret_cast<double*>(sub(R * w.nblk * sizeof(double)));
        w.rstat = reinterpret_cast<ldp::RefStat*>(sub(R * sizeof(ldp::RefStat)));
        w.bflags = reinterpret_cast<int32_t*>(sub(R * w.nblk * sizeof(int32_t)));
        w.kept = reinterpret_cast<int32_t*>(sub(R * sizeof(int32_t)));
        w.fix_count = reinterpret_cast<int32_t*>(sub(ldp::LDP_MAX_SUB * sizeof(int32_t)));
        w.arrive = reinterpret_cast<int32_t*>(sub(R * sizeof(int32_t)));
        w.ticket = reinterpret_cast<int32_t*>(sub(8 * sizeof(int32_t)));
        plan->zero_base = b ? b + z0 : nullptr;
        plan->zero_bytes = off - z0;
        off = align_up(off, 256);
    }
    plan->bytes = off;
    return LDP_OK;
}

cudaError_t clear_launch_state(const Plan& plan, cudaStream_t st) {
    return cudaMemsetAsync(plan.zero_base, 0, plan.zero_bytes, st);
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

static int vec_ok_for(const ldp_params* p) { return (p->W % 4 == 0 && p->scalar_loads == 0) ? 1 : 0; }

// the fused first stage (ldp_front.cu): persistent CTAs, TMA ring, stream + normalise
cudaError_t launch_front(const ldp_params* p, const ldp_ref_desc* refs, const ldp_outputs* out, Plan& plan, cudaStream_t st) {
    static bool configured_dev[MAX_DEVICES] = {};
        bool& configured = configured_dev[current_device()];
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(ldp::ldp_front_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(ldp::ldp_front_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return e;
        configured = true;
    }
    plan.geom.epoch = next_epoch();
    const long long total = (long long)plan.ws.nblk * p->n_refs;
    const unsigned grid = (unsigned)std::min<long long>(plan.front_grid, total);
    if (p->prologue)
        return launch_k(ldp::ldp_front_kernel<true>, dim3(grid), dim3(ldp::KF_THREADS), plan.front_smem, st, *p, refs, plan.ws, *out, plan.geom);
    return launch_k(ldp::ldp_front_kernel<false>, dim3(grid), dim3(ldp::KF_THREADS), plan.front_smem, st, *p, refs, plan.ws, *out, plan.geom);
}

// the first kernel of the path (also launched alone by ldp_debug_launch_stream for the roofline measurement)
void launch_stream(const ldp_params* p, const ldp_ref_desc* refs, Plan& plan, cudaStream_t st, int nsubrefs) {
    const dim3 grid((unsigned)plan.ws.nblk, (unsigned)nsubrefs);
    if (p->prologue && !p->no_warped_masks) switch (p->nn_max) {      // raw matcher planes: post-processing fused into the read
          case 1: (void)launch_k(ldp::ldp_stream_kernel<1, 2>, dim3(grid), dim3(ldp::KS_THREADS), 0, st, *p, refs, plan.ws, plan.geom); break;
          case 2: (void)launch_k(ldp::ldp_stream_kernel<2, 2>, dim3(grid), dim3(ldp::KS_THREADS), 0, st, *p, refs, plan.ws, plan.geom); break;
          case 3: (void)launch_k(ldp::ldp_stream_kernel<3, 2>, dim3(grid), dim3(ldp::KS_THREADS), 0, st, *p, refs, plan.ws, plan.geom); break;
          case 4: (void)launch_k(ldp::ldp_stream_kernel<4, 2>, dim3(grid), dim3(ldp::KS_THREADS), 0, st, *p, refs, plan.ws, plan.geom); break;
          default: (void)launch_k(ldp::ldp_stream_kernel<0, 2>, dim3(grid), dim3(ldp::KS_THREADS), 0, st, *p, refs, plan.ws, plan.geom); break;
    } else if (p->prologue) switch (p->nn_max) {                      // ... and no neighbour mask anywhere: no warp row is read
          case 1: (void)launch_k(ldp::ldp_stream_kernel<1, 1>, dim3(grid), dim3(ldp::KS_THREADS), 0, st, *p, refs, plan.ws, plan.geom); break;
          case 2: (void)launch_k(ldp::ldp_stream_kernel<2, 1>, dim3(grid), dim3(ldp::KS_THREADS), 0, st, *p, refs, plan.ws, plan.geom); break;
          case 3: (void)launch_k(ldp::ldp_stream_kernel<3, 1>, dim3(grid), dim3(ldp::KS_THREADS), 0, st, *p, refs, plan.ws, plan.geom); break;
          case 4: (void)launch_k(ldp::ldp_stream_kernel<4, 1>, dim3(grid), dim3(ldp::KS_THREADS), 0, st, *p, refs, plan.ws, plan.geom); break;
          default: (void)launch_k(ldp::ldp_stream_kernel<0, 1>, dim3(grid), dim3(ldp::KS_THREADS), 0, st, *p, refs, plan.ws, plan.geom); break;
    } else switch (p->nn_max) {
          case 1: (void)launch_k(ldp::ldp_stream_kernel<1, 0>, dim3(grid), dim3(ldp::KS_THREADS), 0, st, *p, refs, plan.ws, plan.geom); break;
          case 2: (void)launch_k(ldp::ldp_stream_kernel<2, 0>, dim3(grid), dim3(ldp::KS_THREADS), 0, st, *p, refs, plan.ws, plan.geom); break;
          case 3: (void)launch_k(ldp::ldp_stream_kernel<3, 0>, dim3(grid), dim3(ldp::KS_THREADS), 0, st, *p, refs, plan.ws, plan.geom); break;
          case 4: (void)launch_k(ldp::ldp_stream_kernel<4, 0>, dim3(grid), dim3(ldp::KS_THREADS), 0, st, *p, refs, plan.ws, plan.geom); break;
          case 5: (void)launch_k(ldp::ldp_stream_kernel<5, 0>, dim3(grid), dim3(ldp::KS_THREADS), 0, st, *p, refs, plan.ws, plan.geom); break;
          case 6: (void)launch_k(ldp::ldp_stream_kernel<6, 0>, dim3(grid), dim3(ldp::KS_THREADS), 0, st, *p, refs, plan.ws, plan.geom); break;
          case 7: (void)launch_k(ldp::ldp_stream_kernel<7, 0>, dim3(grid), dim3(ldp::KS_THREADS), 0, st, *p, refs, plan.ws, plan.geom); break;
          case 8: (void)launch_k(ldp::ldp_stream_kernel<8, 0>, dim3(grid), dim3(ldp::KS_THREADS), 0, st, *p, refs, plan.ws, plan.geom); break;
          default: (void)launch_k(ldp::ldp_stream_kernel<0, 0>, dim3(grid), dim3(ldp::KS_THREADS), 0, st, *p, refs, plan.ws, plan.geom); break;
      }
}

int launch_sample(const ldp_params* p, const ldp_ref_desc* refs, const double* uniforms, const ldp_outputs* out,
                  Plan& plan, int vec_ok, cudaStream_t st, int ref0, int nsubrefs) {
    plan.geom.vec = vec_ok;
    plan.geom.ref0 = ref0;
    static bool configured_dev[MAX_DEVICES] = {};
        bool& configured = configured_dev[current_device()];
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(ldp::ldp_draw_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)K1_SMEM_BUDGET);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(ldp::ldp_draw_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)K1_SMEM_BUDGET);
        if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(draw)");
        e = cudaFuncSetAttribute(ldp::ldp_prep_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
        if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(prep)");
        e = cudaFuncSetAttribute(ldp::ldp_prep_kernel<5, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(ldp::ldp_prep_kernel<6, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(ldp::ldp_prep_kernel<7, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(ldp::ldp_prep_kernel<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(ldp::ldp_prep_kernel<5, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(ldp::ldp_prep_kernel<6, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(ldp::ldp_prep_kernel<7, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(ldp::ldp_prep_kernel<0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
        if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(prep lean)");
        configured = true;
    }
    if (plan.prep_smem > 64 * 1024) return fail(LDP_ERR_INVALID, "map too wide for the prep kernel tables");
    const dim3 grid((unsigned)plan.ws.nblk, (unsigned)nsubrefs);
    cudaError_t e;
    if (plan.use_front) {
        if (plan.geom.chunk_shift > 7) {      // chunk sums are accumulated with atomics: start from zero
            e = cudaMemsetAsync(plan.ws.csum, 0, (size_t)nsubrefs * plan.ws.nchunk_pad * sizeof(double), st);
            if (e == cudaSuccess) e = cudaMemsetAsync(plan.ws.csum0, 0, (size_t)nsubrefs * plan.ws.nchunk_pad * sizeof(double), st);
            if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(csum)");
        }
        { KernelTimer kt(st, "ldp_front_kernel");
          e = launch_front(p, refs, out, plan, st); }
        ++g_launches;
        if (e != cudaSuccess || (e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e, "ldp_front_kernel");
    } else {
    { KernelTimer kt(st, "ldp_stream_kernel");
      launch_stream(p, refs, plan, st, nsubrefs); }
    ++g_launches;
    if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e, "ldp_stream_kernel");
    }
    if (p->no_filter) {
        { KernelTimer kt(st, "ldp_topm_kernel");
          size_t n2 = 1;
          const size_t Mn = (size_t)std::min((long long)p->matches_per_ref, (long long)plan.geom.N);
          while (n2 < Mn) n2 <<= 1;
          static bool topm_configured_dev[MAX_DEVICES] = {};
        bool& topm_configured = topm_configured_dev[current_device()];
          if (!topm_configured) {
              (void)cudaFuncSetAttribute(ldp::ldp_topm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)K1_SMEM_BUDGET);
              topm_configured = true;
          }
          // dynamic shared memory of a CTA: its sort buffer(s) + one tie count per 128-pixel row of its slice
          const size_t n4 = plan.ws.n_pad / 4;
          auto topm_smem = [&](int c) {
              const size_t keys_cap = std::max(n2 / (size_t)c, std::min(n2, (size_t)1024));
              const size_t per = (((n4 + c - 1) / c) + 31) & ~(size_t)31;
              return (c > 1 ? 2 : 1) * keys_cap * 8 + (per / 32) * 4;
          };
          if (topm_smem(1) <= K1_SMEM_BUDGET && !getenv("LDP_TOPM_GENERIC")) {
              // one cluster of C CTAs per view: the largest C that keeps every view's cluster in one wave (one CTA per SM)
              int csize = 1;
              for (int c = 8; c > 1; c >>= 1)
                  if ((long long)nsubrefs * c <= sm_count() && (size_t)c * 1024 <= n2) { csize = c; break; }
              static const int env_c = [] { const char* e = getenv("LDP_TOPM_CLUSTER"); return e ? atoi(e) : 0; }();
              if ((env_c == 1 || env_c == 2 || env_c == 4 || env_c == 8) && (size_t)env_c <= n2) csize = env_c;
              const int fc = g_force_cluster;              // test hook
              if ((fc == 1 || fc == 2 || fc == 4 || fc == 8) && (size_t)fc <= n2) csize = fc;
              while (csize > 1 && topm_smem(csize) > K1_SMEM_BUDGET) csize >>= 1;
              static const int pdl = [] { const char* e = getenv("LDP_PDL"); return e ? atoi(e) : 1; }();
              for (;;) {
                  cudaLaunchConfig_t cfg = {};
                  cfg.gridDim = dim3((unsigned)(nsubrefs * csize));
                  cfg.blockDim = dim3(ldp::K1_THREADS);
                  cfg.dynamicSmemBytes = topm_smem(csize);
                  cfg.stream = st;
                  cudaLaunchAttribute attr[2];
                  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
                  attr[0].val.programmaticStreamSerializationAllowed = pdl;
                  attr[1].id = cudaLaunchAttributeClusterDimension;
                  attr[1].val.clusterDim.x = (unsigned)csize;
                  attr[1].val.clusterDim.y = 1;
                  attr[1].val.clusterDim.z = 1;
                  cfg.attrs = attr;
                  cfg.numAttrs = csize > 1 ? 2 : 1;
                  if (cudaLaunchKernelEx(&cfg, ldp::ldp_topm_kernel, *p, refs, plan.ws, *out, plan.geom, csize) == cudaSuccess || csize == 1) break;
                  (void)cudaGetLastError();
                  csize >>= 1;                             // cluster not schedulable: smaller one
              }
              g_last_cluster = csize;
          } else
              (void)launch_k(ldp::ldp_topm_generic_kernel, dim3(nsubrefs), dim3(ldp::K1_THREADS), 0, st, *p, refs, plan.ws, *out, plan.geom); }
        ++g_launches;
        if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e, "ldp_topm_kernel");
        return LDP_OK;
    }
    if (!plan.use_front) {
    if (plan.geom.chunk_shift > 7) {      // chunk sums are accumulated with atomics: start from zero
        e = cudaMemsetAsync(plan.ws.csum + (size_t)ref0 * plan.ws.nchunk_pad, 0, (size_t)nsubrefs * plan.ws.nchunk_pad * sizeof(double), st);
        if (e == cudaSuccess)
            e = cudaMemsetAsync(plan.ws.csum0 + (size_t)ref0 * plan.ws.nchunk_pad, 0, (size_t)nsubrefs * plan.ws.nchunk_pad * sizeof(double), st);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(csum)");
    }
    { KernelTimer kt(st, "ldp_prep_kernel");
      static const bool force_generic = getenv("LDP_PREP_GENERIC") != nullptr;
      if (vec_ok && plan.geom.prep_lean && !force_generic) {
          const bool xc = plan.geom.step_dx == 0;       // W divides the pass stride: a thread stays in one pixel column
#define LDP_PREP_LAUNCH(CSV) \
          do { if (xc) (void)launch_k(ldp::ldp_prep_kernel<CSV, true>, dim3(grid), dim3(ldp::KS_THREADS), plan.prep_smem, st, *p, refs, plan.ws, *out, plan.geom); \
               else (void)launch_k(ldp::ldp_prep_kernel<CSV, false>, dim3(grid), dim3(ldp::KS_THREADS), plan.prep_smem, st, *p, refs, plan.ws, *out, plan.geom); } while (0)
          switch (plan.geom.chunk_shift) {
              case 5: LDP_PREP_LAUNCH(5); break;
              case 6: LDP_PREP_LAUNCH(6); break;
              case 7: LDP_PREP_LAUNCH(7); break;
              default: LDP_PREP_LAUNCH(0); break;
          }
#undef LDP_PREP_LAUNCH
      } else {
          (void)launch_k(ldp::ldp_prep_generic_kernel, dim3(grid), dim3(ldp::KS_THREADS), plan.prep_smem, st, *p, refs, plan.ws, *out, plan.geom);
      } }
    ++g_launches;
    if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e, "ldp_prep_kernel");
    }
    // ---- round 1: independent CTAs, as many per view as the device has SMs for (one CTA per SM: the table fills it)
    static const int env_reserve = [] { const char* e = getenv("LDP_SM_RESERVE"); return e ? atoi(e) : -1; }();   // SMs left to concurrent
    const int sm_reserve = env_reserve >= 0 ? env_reserve : (p->sm_reserve >= 0 ? p->sm_reserve : g_sm_reserve);                                             // kernels (other launches in
    int c_first = (sm_count() - sm_reserve) / nsubrefs;                                                            // flight, communication)
    if (c_first < 1) c_first = 1;
    if (c_first > (int)plan.ws.draw_cmax) c_first = (int)plan.ws.draw_cmax;
    if (g_force_cluster > 0) c_first = g_force_cluster;
    { KernelTimer kt(st, "ldp_draw_kernel");
      (void)launch_k(ldp::ldp_draw_kernel<1>, dim3((unsigned)(nsubrefs * c_first)), dim3(ldp::KD_THREADS), plan.k1_smem, st,
                     *p, refs, uniforms, plan.ws, *out, plan.geom, c_first); }
    ++g_launches;
    if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e, "ldp_draw_kernel<1>");
    {
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
            if ((long long)nsubrefs * c > sm_count()) continue;
            if (max_active_clusters(c, plan.k1_smem) >= nsubrefs) { csize = c; break; }
        }
        if (g_force_cluster > 0) csize = g_force_cluster;
        static const int env_c = [] { const char* e = getenv("LDP_RESUME_CLUSTER"); return e ? atoi(e) : 0; }();
        if (env_c > 0) csize = env_c;
        KernelTimer kt(st, "ldp_resume_kernel");
        for (;;) {
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3((unsigned)(nsubrefs * csize));
            cfg.blockDim = dim3(ldp::KD_THREADS);
            cfg.dynamicSmemBytes = plan.k1_smem;
            cfg.stream = st;
            static const int pdl = [] { const char* e = getenv("LDP_PDL"); return e ? atoi(e) : 1; }();
            cudaLaunchAttribute attr[2];
            attr[0].id = cudaLaunchAttributeClusterDimension;
            attr[0].val.clusterDim.x = (unsigned)csize;
            attr[0].val.clusterDim.y = 1;
            attr[0].val.clusterDim.z = 1;
            attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            attr[1].val.programmaticStreamSerializationAllowed = pdl;
            cfg.attrs = attr;
            cfg.numAttrs = 2;
            e = cudaLaunchKernelEx(&cfg, ldp::ldp_draw_kernel<2>, *p, refs, uniforms, plan.ws, *out, plan.geom, c_first);
            if (e == cudaSuccess) break;
            (void)cudaGetLastError();
            if (csize == 1) return cuda_fail(e, "ldp_draw_kernel<2>");
            csize = (csize > 4) ? 4 : (csize > 2 ? 2 : 1);      // odd sizes may not be schedulable: fall back
        }
        g_last_cluster = csize;
    }
    ++g_launches;
    if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e, "ldp_draw_kernel");
    return LDP_OK;
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

ldp::GeomArgs make_geom_args(const ldp_params* p, const Plan& plan, int have_bestk, int ref0, int sub) {
    thread_local float cached_deg = -1.f, cached_cos = 1.f;
    if (p->min_parallax_deg != cached_deg) { cached_cos = parallax_cos_threshold(p->min_parallax_deg); cached_deg = p->min_parallax_deg; }
    ldp::GeomArgs ga;
    ga.par_cos_max = cached_cos;
    ga.have_bestk = have_bestk;
    ga.nb2 = plan.nb2;
    ga.ref0 = ref0;
    ga.sub = sub;
    static const int discard_mode = [] { const char* e = getenv("LDP_DISCARD"); return e ? atoi(e) : 1; }();
    ga.discard = have_bestk ? discard_mode : 0;
    static const int fuse_mode = [] { const char* e = getenv("LDP_FUSE_GATHER"); return e ? atoi(e) : 1; }();
    ga.fused = p->multiview ? 1 : fuse_mode;      // the refinement reads the sample index: a multiview launch always gathers itself
    static const int prefetch_mode = [] { const char* e = getenv("LDP_GEOM_PREFETCH"); return e ? atoi(e) : 1; }();
    ga.l2_prefetch = prefetch_mode;
    ga.force_fix_two = g_force_fix_two;
    ga.force_fix_mv = g_force_fix_mv;
    return ga;
}

// gather -> compute -> fix+plan for views [ref0, ref0 + nsubrefs)
int launch_geometry(const ldp_params* p, const ldp_ref_desc* refs, const ldp_outputs* out, Plan& plan,
                    int have_bestk, cudaStream_t st, int ref0, int nsubrefs, int sub) {
    const ldp::GeomArgs ga = make_geom_args(p, plan, have_bestk, ref0, sub);
    const dim3 grid((unsigned)plan.nb2, (unsigned)nsubrefs);
    const dim3 ggrid((unsigned)((plan.ws.sel_cap + ldp::KG_THREADS * KG_SPT - 1) / (ldp::KG_THREADS * KG_SPT)), (unsigned)nsubrefs);
    cudaError_t e;
    if (!ga.fused) {
        { KernelTimer kt(st, "ldp_gather_kernel");
          (void)launch_k(ldp::ldp_gather_kernel, dim3(ggrid), dim3(ldp::KG_THREADS), 0, st, *p, refs, plan.ws, *out, ga); }
        ++g_launches;
        if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e, "ldp_gather_kernel");
    }
    { KernelTimer kt(st, "ldp_geometry_kernel");
      auto* k2 = p->multiview ? (p->lens ? ldp::ldp_geometry_kernel<true, true> : ldp::ldp_geometry_kernel<false, true>)
                              : (p->lens ? ldp::ldp_geometry_kernel<true, false> : ldp::ldp_geometry_kernel<false, false>);
      (void)launch_k(k2, dim3(grid), dim3(ldp::K2_THREADS), 0, st, *p, refs, plan.ws, *out, ga); }
    ++g_launches;
    if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e, "ldp_geometry_kernel");
    { KernelTimer kt(st, "ldp_fix_kernel");
      auto* kf = p->multiview ? (p->lens ? ldp::ldp_fix_kernel<true, true> : ldp::ldp_fix_kernel<false, true>)
                              : (p->lens ? ldp::ldp_fix_kernel<true, false> : ldp::ldp_fix_kernel<false, false>);
      (void)launch_k(kf, dim3(nsubrefs), dim3(ldp::K2_THREADS), 0, st, *p, refs, plan.ws, *out, ga); }
    ++g_launches;
    if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e, "ldp_fix_kernel");
    return LDP_OK;
}

// ordered scatter of all views of the launch (needs every view's kept count)
int launch_pack(const ldp_params* p, const ldp_ref_desc* refs, const ldp_outputs* out, Plan& plan, cudaStream_t st) {
    const ldp::GeomArgs ga = make_geom_args(p, plan, 1, 0, 0);
    const dim3 grid((unsigned)plan.nb2, (unsigned)p->n_refs);
    { KernelTimer kt(st, "ldp_pack_kernel");
      (void)launch_k(ldp::ldp_pack_kernel, dim3(grid), dim3(ldp::K3_THREADS), 0, st, *p, refs, plan.ws, *out, ga); }
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "ldp_pack_kernel");
    return LDP_OK;
}

// Internal streams for pipelining a launch over sub-batches of views: the kernels of the path stress different
// resources (HBM stream, issue-bound prep, latency-bound draw, DRAM-latency gather, FP64 geometry), so the kernels of
// one sub-batch overlap those of the next.  Fork/join with events keeps the call stream-ordered for the caller.
struct SubStreams {
    cudaStream_t s[ldp::LDP_MAX_SUB];
    cudaEvent_t start, done[ldp::LDP_MAX_SUB];
    bool ok = false;
};
SubStreams& substreams() {
    static thread_local SubStreams ss;
    if (!ss.ok) {
        bool good = cudaEventCreateWithFlags(&ss.start, cudaEventDisableTiming) == cudaSuccess;
        for (int i = 0; i < ldp::LDP_MAX_SUB && good; ++i) {
            good = cudaStreamCreateWithFlags(&ss.s[i], cudaStreamNonBlocking) == cudaSuccess &&
                   cudaEventCreateWithFlags(&ss.done[i], cudaEventDisableTiming) == cudaSuccess;
        }
        ss.ok = good;
    }
    return ss;
}

int g_force_sub = -1;      // ldp_debug_set_subbatches; -1 = environment / default
int choose_subbatches(int n_refs) {
    int n = g_force_sub;
    if (n < 0) {
        static int env_n = -2;
        if (env_n == -2) { const char* e = getenv("LDP_SUBBATCH"); env_n = e ? atoi(e) : 0; }
        n = env_n;
    }
    if (n <= 0) n = 1;
    if (n > ldp::LDP_MAX_SUB) n = ldp::LDP_MAX_SUB;
    while (n > 1 && n_refs < 2 * n) --n;
    return n;
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

int ldp_debug_set_subbatches(int n) {
    if (n < -1 || n > ldp::LDP_MAX_SUB) return fail(LDP_ERR_INVALID, "sub-batches must be -1 (default) .. 8");
    g_force_sub = n;
    return LDP_OK;
}

int ldp_debug_launch_stream(const ldp_params* params, const ldp_ref_desc* refs, void* workspace, size_t workspace_bytes,
                            void* stream, int reps) {
    if (!params || !refs || !workspace || reps < 1) return fail(LDP_ERR_INVALID, "bad arguments");
    Plan plan;
    char* base = reinterpret_cast<char*>(align_up(reinterpret_cast<size_t>(workspace), 256));
    int rc = make_plan(params, base, &plan);
    if (rc != LDP_OK) return rc;
    if (plan.bytes + (size_t)(base - static_cast<char*>(workspace)) > workspace_bytes) return fail(LDP_ERR_WORKSPACE, "workspace too small");
    plan.geom.vec = vec_ok_for(params);
    plan.geom.ref0 = 0;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cudaError_t e;
    if (plan.use_front) {      // the fused front kernel is the first stage on this shape (it cleans its own counters up)
        ldp_outputs none = {};
        e = clear_launch_state(plan, st);
        for (int i = 0; i < reps && e == cudaSuccess; ++i) e = launch_front(params, refs, &none, plan, st);
        if (e != cudaSuccess) return cuda_fail(e, "ldp_front_kernel");
    } else {
        for (int i = 0; i < reps; ++i) launch_stream(params, refs, plan, st, params->n_refs);
    }
    e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "ldp_stream_kernel");
    return LDP_OK;
}

int ldp_debug_read_clocks(const ldp_params* params, void* workspace, long long* host_out) {
    Plan plan;
    char* base = reinterpret_cast<char*>(align_up(reinterpret_cast<size_t>(workspace), 256));
    int rc = make_plan(params, base, &plan);
    if (rc != LDP_OK) return rc;
    cudaError_t e = cudaMemcpy(host_out, plan.ws.dbgclk, (size_t)params->n_refs * 32 * sizeof(long long), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpy(dbgclk)");
    return LDP_OK;
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
    char* base = reinterpret_cast<char*>(align_up(reinterpret_cast<size_t>(workspace), 256));
    int rc = make_plan(params, base, &plan);
    if (rc != LDP_OK) return rc;
    host_out[0] = host_out[1] = 0;
    int32_t counts[ldp::LDP_MAX_SUB];
    cudaError_t e = cudaMemcpy(counts, plan.ws.fix_count, sizeof(counts), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpy(fix_count)");
    const int nsub = choose_subbatches(params->n_refs);
    std::vector<int2> list;
    for (int h = 0; h < nsub; ++h) {           // sub-batch h's worklist starts at its first view * sel_cap (launch_geometry)
        const int lo = (int)(((long long)h * params->n_refs) / nsub);
        if (counts[h] <= 0) continue;
        list.resize((size_t)counts[h]);
        e = cudaMemcpy(list.data(), plan.ws.fix_list + (size_t)lo * plan.ws.sel_cap, list.size() * sizeof(int2), cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpy(fix_list)");
        host_out[0] += counts[h];
        for (const int2& it : list) host_out[1] += (it.y & ldp::MV_FIX) ? 1 : 0;
    }
    return LDP_OK;
}

int ldp_debug_set_cluster(int csize) {
    if (csize < 0 || csize > 8) return fail(LDP_ERR_INVALID, "cluster size must be 0 (auto) .. 8");
    g_force_cluster = csize;
    return LDP_OK;
}

const char* ldp_profile_name(int i) { return (i >= 0 && i < g_prof_n) ? g_prof_name[i] : ""; }

// ---- output contract on the device (ldp_output.cu)
// format 2 takes the normals [n,3] in place of err
static int pack_records(int format, const float* xyz, const float* rgb, const float* err, int64_t n, const int64_t* n_dev,
                        uint64_t first_id, uint8_t* out, void* stream) {
    if (n < 0) return fail(LDP_ERR_INVALID, "negative point count");
    g_launches = 0;
    if (n == 0) return LDP_OK;
    if (!xyz || !rgb || !out) return fail(LDP_ERR_INVALID, "null pointer");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const unsigned grid = (unsigned)((n + ldp::KO_THREADS - 1) / ldp::KO_THREADS);
    const int aligned = (reinterpret_cast<uintptr_t>(out) & 15u) == 0;
    if (format == 0)
        (void)launch_k(ldp::ldp_records_kernel<0>, dim3(grid), dim3(ldp::KO_THREADS), 0, st, xyz, rgb, err, (long long)n,
                       reinterpret_cast<const long long*>(n_dev), (unsigned long long)first_id, out, aligned, (const float*)nullptr);
    else if (format == 1)
        (void)launch_k(ldp::ldp_records_kernel<1>, dim3(grid), dim3(ldp::KO_THREADS), 0, st, xyz, rgb, err, (long long)n,
                       reinterpret_cast<const long long*>(n_dev), (unsigned long long)first_id, out, aligned, (const float*)nullptr);
    else
        (void)launch_k(ldp::ldp_records_kernel<2>, dim3(grid), dim3(ldp::KO_THREADS), 0, st, xyz, rgb, (const float*)nullptr,
                       (long long)n, reinterpret_cast<const long long*>(n_dev), 0ull, out, aligned, err);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "ldp_records_kernel");
    return LDP_OK;
}

int ldp_pack_ply_records(const float* xyz, const float* rgb, int64_t n, const int64_t* n_dev, uint8_t* records_out, void* stream) {
    return pack_records(0, xyz, rgb, nullptr, n, n_dev, 0, records_out, stream);
}

int ldp_pack_ply_normal_records(const float* xyz, const float* rgb, const float* normals, int64_t n, const int64_t* n_dev,
                                uint8_t* records_out, void* stream) {
    if (n > 0 && !normals) return fail(LDP_ERR_INVALID, "null normals");
    return pack_records(2, xyz, rgb, normals, n, n_dev, 0, records_out, stream);
}

int ldp_pack_points3d_records(const float* xyz, const float* rgb, const float* err, int64_t n, const int64_t* n_dev,
                              uint64_t first_id, uint8_t* records_out, void* stream) {
    return pack_records(1, xyz, rgb, err, n, n_dev, first_id, records_out, stream);
}

int ldp_undistort_points(const ldp_lens* lens, int64_t n, const float* uv_in, float* uv_out, void* stream) {
    if (!lens || n < 0) return fail(LDP_ERR_INVALID, "bad arguments");
    if (lens->model < LDP_LENS_PINHOLE || lens->model > LDP_LENS_FISHEYE) return fail(LDP_ERR_INVALID, "unknown lens model");
    g_launches = 0;
    if (n == 0) return LDP_OK;
    if (!uv_in || !uv_out) return fail(LDP_ERR_INVALID, "null pointer");
    if ((reinterpret_cast<size_t>(uv_in) | reinterpret_cast<size_t>(uv_out)) & 7) return fail(LDP_ERR_INVALID, "uv arrays must be 8-byte aligned");
    const long long blocks = (n + ldp::KU_THREADS - 1) / ldp::KU_THREADS;
    const unsigned grid = (unsigned)std::min<long long>(blocks, (long long)sm_count() * 16);
    (void)launch_k(ldp::ldp_undistort_kernel, dim3(grid), dim3(ldp::KU_THREADS), 0, reinterpret_cast<cudaStream_t>(stream), *lens,
                   (long long)n, reinterpret_cast<const float2*>(uv_in), reinterpret_cast<float2*>(uv_out));
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "ldp_undistort_kernel");
    return LDP_OK;
}

int ldp_rgb_to_uint8(const float* rgb, int64_t n_values, uint8_t* out, void* stream) {
    if (n_values < 0) return fail(LDP_ERR_INVALID, "negative count");
    g_launches = 0;
    if (n_values == 0) return LDP_OK;
    if (!rgb || !out) return fail(LDP_ERR_INVALID, "null pointer");
    const long long blocks = (n_values + ldp::KO_THREADS - 1) / ldp::KO_THREADS;
    const unsigned grid = (unsigned)std::min<long long>(blocks, (long long)sm_count() * 16);
    (void)launch_k(ldp::ldp_rgb_u8_kernel, dim3(grid), dim3(ldp::KO_THREADS), 0, reinterpret_cast<cudaStream_t>(stream), rgb, (long long)n_values, out);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "ldp_rgb_u8_kernel");
    return LDP_OK;
}

int ldp_gather_points(const float* xyz, const float* rgb, const float* err, const int64_t* sel, int64_t m, int64_t n,
                      float* xyz_out, float* rgb_out, float* err_out, int32_t* bad_index_flag, void* stream) {
    if (m < 0 || n < 0) return fail(LDP_ERR_INVALID, "negative count");
    g_launches = 0;
    if (m == 0) return LDP_OK;
    if (!xyz || !rgb || !sel || !xyz_out || !rgb_out) return fail(LDP_ERR_INVALID, "null pointer");
    const unsigned grid = (unsigned)((m + ldp::KO_THREADS - 1) / ldp::KO_THREADS);
    (void)launch_k(ldp::ldp_gather_rows_kernel, dim3(grid), dim3(ldp::KO_THREADS), 0, reinterpret_cast<cudaStream_t>(stream), xyz, rgb, err,
                   reinterpret_cast<const long long*>(sel), (long long)m, (long long)n, xyz_out, rgb_out, err_out, (int*)bad_index_flag);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "ldp_gather_rows_kernel");
    return LDP_OK;
}

int ldp_gather_rows(const float* src, int32_t row_floats, const int64_t* sel, int64_t m, int64_t n, float* out,
                    int32_t* bad_index_flag, void* stream) {
    if (m < 0 || n < 0 || row_floats <= 0) return fail(LDP_ERR_INVALID, "bad row gather shape");
    g_launches = 0;
    if (m == 0) return LDP_OK;
    if (!src || !sel || !out) return fail(LDP_ERR_INVALID, "null pointer");
    const long long blocks = (m * row_floats + ldp::KO_THREADS - 1) / ldp::KO_THREADS;
    const unsigned grid = (unsigned)std::min<long long>(blocks, (long long)sm_count() * 16);
    (void)launch_k(ldp::ldp_gather_f32_rows_kernel, dim3(grid), dim3(ldp::KO_THREADS), 0, reinterpret_cast<cudaStream_t>(stream), src,
                   (int)row_floats, reinterpret_cast<const long long*>(sel), (long long)m, (long long)n, out, (int*)bad_index_flag);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "ldp_gather_f32_rows_kernel");
    return LDP_OK;
}

int ldp_concat_points(const float* const* xyz_src, const float* const* rgb_src, const float* const* err_src,
                      const int64_t* const* count_src, int32_t n_seg, int64_t seg_cap, float* xyz_out, float* rgb_out,
                      float* err_out, int64_t out_capacity, int64_t* seg_offset_out, int64_t* total_out, void* stream) {
    if (n_seg < 0 || seg_cap < 0 || out_capacity < 0) return fail(LDP_ERR_INVALID, "negative size");
    g_launches = 0;
    if (n_seg == 0) return LDP_OK;
    if (!xyz_src || !rgb_src || !err_src || !count_src || !xyz_out || !rgb_out || !err_out) return fail(LDP_ERR_INVALID, "null pointer");
    if (n_seg > 65535) return fail(LDP_ERR_INVALID, "too many segments");
    const long long blocks = (seg_cap * 3 + ldp::KO_THREADS * 4 - 1) / (ldp::KO_THREADS * 4);
    // enough CTAs to keep a few MB of (possibly remote) reads in flight: about four waves of CTAs over all segments
    const long long per_seg = std::max<long long>(64, (long long)sm_count() * 8 * 4 / std::max(1, n_seg));
    const unsigned gx = (unsigned)std::max<long long>(1, std::min<long long>(blocks, per_seg));
    (void)launch_k(ldp::ldp_concat_points_kernel, dim3(gx, (unsigned)n_seg), dim3(ldp::KO_THREADS), 0, reinterpret_cast<cudaStream_t>(stream),
                   xyz_src, rgb_src, err_src, reinterpret_cast<const long long* const*>(count_src), (int)n_seg, (long long)seg_cap,
                   xyz_out, rgb_out, err_out, (long long)out_capacity, reinterpret_cast<long long*>(seg_offset_out),
                   reinterpret_cast<long long*>(total_out));
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "ldp_concat_points_kernel");
    return LDP_OK;
}

int ldp_scatter_points(const float* xyz, const float* rgb, const float* err, const int64_t* const* count_src, int32_t rank,
                       int32_t world, int64_t seg_cap, float* const* xyz_dst, float* const* rgb_dst, float* const* err_dst,
                       int64_t out_capacity, int64_t* seg_offset_out, int64_t* total_out, void* stream) {
    if (world < 1 || world > 64 || rank < 0 || rank >= world || seg_cap < 0 || out_capacity < 0) return fail(LDP_ERR_INVALID, "bad rank / world / size");
    g_launches = 0;
    if (!xyz || !rgb || !err || !count_src || !xyz_dst || !rgb_dst || !err_dst) return fail(LDP_ERR_INVALID, "null pointer");
    const long long blocks = (seg_cap * 3 + ldp::KO_THREADS * 4 - 1) / (ldp::KO_THREADS * 4);
    const long long per_dst = std::max<long long>(32, (long long)sm_count() * 8 * 2 / world);
    const unsigned gx = (unsigned)std::max<long long>(1, std::min<long long>(blocks, per_dst));
    (void)launch_k(ldp::ldp_scatter_points_kernel, dim3(gx, (unsigned)world), dim3(ldp::KO_THREADS), 0, reinterpret_cast<cudaStream_t>(stream),
                   xyz, rgb, err, reinterpret_cast<const long long* const*>(count_src), (int)rank, (int)world, (long long)seg_cap,
                   xyz_dst, rgb_dst, err_dst, (long long)out_capacity, reinterpret_cast<long long*>(seg_offset_out),
                   reinterpret_cast<long long*>(total_out));
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "ldp_scatter_points_kernel");
    return LDP_OK;
}

// ---- pair generation on the device (ldp_select.cu)
int ldp_select_kcenters(const float* flat_poses, int32_t n, int32_t k, float* scratch, int32_t* centers_sorted,
                        int32_t* centers_order, void* stream) {
    g_launches = 0;
    if (n <= 0 || k <= 0 || k > n) return fail(LDP_ERR_INVALID, "k-centres needs 1 <= k <= n");
    if (n > ldp::KC_THREADS * ldp::KC_MAX_PER_THREAD) return fail(LDP_ERR_INVALID, "k-centres: more than 8192 views");
    if (!flat_poses || !scratch || !centers_sorted || !centers_order) return fail(LDP_ERR_INVALID, "null pointer");
    const size_t smem = (size_t)n * ldp::KC_PAD * sizeof(float);
    if (smem <= K1_SMEM_BUDGET) {                        // the poses fit in shared memory (n <= 3011)
        static bool configured_dev[MAX_DEVICES] = {};
        bool& configured = configured_dev[current_device()];
        if (!configured) {
            (void)cudaFuncSetAttribute(ldp::ldp_kcenters_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)K1_SMEM_BUDGET);
            configured = true;
        }
        (void)launch_k(ldp::ldp_kcenters_kernel<true>, dim3(1), dim3(ldp::KC_THREADS), smem, reinterpret_cast<cudaStream_t>(stream),
                       flat_poses, (int)n, (int)k, scratch, centers_sorted, centers_order);
    } else
        (void)launch_k(ldp::ldp_kcenters_kernel<false>, dim3(1), dim3(ldp::KC_THREADS), 0, reinterpret_cast<cudaStream_t>(stream),
                       flat_poses, (int)n, (int)k, scratch, centers_sorted, centers_order);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "ldp_kcenters_kernel");
    return LDP_OK;
}

int ldp_nearest_neighbors(const float* flat_poses, int32_t n, int32_t k, int64_t* idx_out, void* stream) {
    g_launches = 0;
    if (n < 0 || k < 0) return fail(LDP_ERR_INVALID, "negative size");
    if (n <= 1 || k == 0) return LDP_OK;
    if (k > n - 1 || k > ldp::KNN_MAX_K) return fail(LDP_ERR_INVALID, "nearest neighbours needs k <= min(n - 1, 16)");
    if (!flat_poses || !idx_out) return fail(LDP_ERR_INVALID, "null pointer");
    (void)launch_k(ldp::ldp_knn_kernel, dim3((unsigned)n), dim3(ldp::KNN_THREADS), 0, reinterpret_cast<cudaStream_t>(stream), flat_poses,
                   (int)n, (int)k, reinterpret_cast<long long*>(idx_out));
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "ldp_knn_kernel");
    return LDP_OK;
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
    size_t off = 0;
    auto carve = [&](size_t b) { void* p = base ? static_cast<char*>(base) + off : nullptr; off += align_up(b, 256); return p; };
    ws->bounds = reinterpret_cast<double*>(carve(8 * sizeof(double)));
    ws->bounds_u = reinterpret_cast<unsigned int*>(carve(8 * sizeof(unsigned int)));
    ws->keys = reinterpret_cast<unsigned long long*>(carve(cap * sizeof(unsigned long long)));
    ws->first = reinterpret_cast<int*>(carve(cap * sizeof(int)));
    ws->slot = reinterpret_cast<int*>(carve(N * sizeof(int)));
    ws->flag = reinterpret_cast<int*>(carve(N * sizeof(int)));
    ws->rank = reinterpret_cast<int*>(carve(N * sizeof(int)));
    ws->count = reinterpret_cast<int*>(carve((N + 1) * sizeof(int)));
    ws->cursor = reinterpret_cast<int*>(carve(N * sizeof(int)));
    ws->seg = reinterpret_cast<int*>(carve(N * sizeof(int)));
    ws->members = reinterpret_cast<int*>(carve(N * sizeof(int)));
    ws->block_tot = reinterpret_cast<int*>(carve((N / ldp::SC_THREADS + 2) * sizeof(int)));
    ws->large = reinterpret_cast<int*>(carve((N + 2) * sizeof(int)));
    ws->status = nullptr;
    ws->cap_mask = cap - 1;
    *bytes = off;
    return LDP_OK;
}

int ldp_voxel_workspace_bytes(int64_t n, size_t* bytes_out) {
    if (!bytes_out) return fail(LDP_ERR_INVALID, "null bytes_out");
    ldp::VoxelWs ws;
    return voxel_plan(n, nullptr, &ws, bytes_out);
}

static int scan_exclusive(const int* in, int* out, int64_t n, int* block_tot, int* grand_total, cudaStream_t st) {
    const int nblocks = (int)((n + ldp::SC_THREADS - 1) / ldp::SC_THREADS);
    (void)launch_k(ldp::ldp_scan_blocks_kernel, dim3(nblocks), dim3(ldp::SC_THREADS), 0, st, in, out, (long long)n, block_tot);
    (void)launch_k(ldp::ldp_scan_totals_kernel, dim3(1), dim3(ldp::SC_THREADS), 0, st, block_tot, nblocks, grand_total);
    (void)launch_k(ldp::ldp_scan_add_kernel, dim3(nblocks), dim3(ldp::SC_THREADS), 0, st, out, (long long)n, (const int*)block_tot);
    g_launches += 3;
    return LDP_OK;
}

int ldp_voxel_downsample(const float* xyz, const float* rgb, int64_t n, double voxel_size, float* xyz_out, float* rgb_out,
                         int32_t* status_out, void* workspace, size_t workspace_bytes, void* stream) {
    g_launches = 0;
    if (!(voxel_size > 0.0)) return fail(LDP_ERR_INVALID, "voxel_size must be positive");       // Open3D: "voxel_size <= 0."
    if (!status_out) return fail(LDP_ERR_INVALID, "null status_out");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    cudaError_t e = cudaMemsetAsync(status_out, 0, 2 * sizeof(int32_t), st);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(status)");
    if (n == 0) return LDP_OK;
    if (!xyz || !rgb || !xyz_out || !rgb_out || !workspace) return fail(LDP_ERR_INVALID, "null pointer");
    ldp::VoxelWs ws;
    size_t need = 0;
    int rc = voxel_plan(n, workspace, &ws, &need);
    if (rc != LDP_OK) return rc;
    if (workspace_bytes < need) return fail(LDP_ERR_INVALID, "voxel workspace too small");
    ws.status = status_out;
    const size_t cap = (size_t)ws.cap_mask + 1;
    e = cudaMemsetAsync(ws.bounds_u, 0xFF, 3 * sizeof(unsigned int), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(ws.bounds_u + 3, 0, sizeof(unsigned int), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(ws.keys, 0xFF, cap * sizeof(unsigned long long), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(ws.first, 0x7F, cap * sizeof(int), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(ws.count, 0, ((size_t)n + 1) * sizeof(int), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(ws.cursor, 0, (size_t)n * sizeof(int), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(ws.large, 0, 2 * sizeof(int), st);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(voxel workspace)");
    const unsigned grid = (unsigned)((n + ldp::KV_THREADS - 1) / ldp::KV_THREADS);
    const unsigned rgrid = (unsigned)std::min<long long>(grid, (long long)sm_count() * 8);
    (void)launch_k(ldp::ldp_voxel_bounds_kernel, dim3(rgrid), dim3(ldp::KV_THREADS), 0, st, xyz, rgb, (long long)n, ws);
    (void)launch_k(ldp::ldp_voxel_insert_kernel, dim3(grid), dim3(ldp::KV_THREADS), 0, st, xyz, (long long)n, voxel_size, (const double*)nullptr, ws);
    (void)launch_k(ldp::ldp_voxel_flag_kernel, dim3(grid), dim3(ldp::KV_THREADS), 0, st, (long long)n, ws);
    g_launches += 3;
    scan_exclusive(ws.flag, ws.rank, n, ws.block_tot, ws.status + 1, st);
    (void)launch_k(ldp::ldp_voxel_count_kernel, dim3(grid), dim3(ldp::KV_THREADS), 0, st, (long long)n, ws);
    ++g_launches;
    scan_exclusive(ws.count, ws.seg, n, ws.block_tot, nullptr, st);
    (void)launch_k(ldp::ldp_voxel_group_kernel, dim3(grid), dim3(ldp::KV_THREADS), 0, st, (long long)n, ws, (const int*)ws.seg);
    (void)launch_k(ldp::ldp_voxel_mean_kernel, dim3(grid), dim3(ldp::KV_THREADS), 0, st, xyz, rgb, ws, (const int*)ws.seg, xyz_out, rgb_out);
    (void)launch_k(ldp::ldp_voxel_large_kernel, dim3((unsigned)sm_count()), dim3(ldp::SC_THREADS), 0, st, xyz, rgb, ws, (const int*)ws.seg, xyz_out, rgb_out);
    g_launches += 3;
    if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e, "voxel downsample kernels");
    return LDP_OK;
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
    size_t off = 0;
    int rc = voxel_plan(n, base, &pl->vws, &off);
    if (rc != LDP_OK) return rc;
    const size_t cap = voxel_cap(n), N = (size_t)std::max<int64_t>(n, 1);
    auto carve = [&](size_t b) { void* p = base ? static_cast<char*>(base) + off : nullptr; off += align_up(b, 256); return p; };
    pl->vstat = reinterpret_cast<int*>(carve(2 * sizeof(int)));
    pl->h_trial = reinterpret_cast<double*>(carve(sizeof(double)));
    pl->stats = reinterpret_cast<double*>(carve(3 * sizeof(double)));
    pl->m = reinterpret_cast<double*>(carve(with_stats ? N * sizeof(double) : 0));
    pl->part = reinterpret_cast<double*>(carve(with_stats ? (N / ldp::OL_CHUNK + 1) * sizeof(double) : 0));
    pl->levels = reinterpret_cast<ldp::OutlierLevel*>(carve(ldp::OL_MAX_LEVELS * sizeof(ldp::OutlierLevel)));
    for (int l = 0; l < ldp::OL_MAX_LEVELS; ++l) {
        pl->keys[l] = reinterpret_cast<unsigned long long*>(carve(cap * sizeof(unsigned long long)));
        pl->cell[l] = reinterpret_cast<int2*>(carve(cap * sizeof(int2)));
        pl->pts[l] = reinterpret_cast<float4*>(carve(N * sizeof(float4)));
    }
    *bytes = off;
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
static void outlier_insert(const float* xyz, int64_t n, double h, const double* h_dev, OutlierPlan& pl, unsigned grid, cudaStream_t st,
                           int* cells_out) {
    ldp::VoxelWs& ws = pl.vws;
    const size_t cap = (size_t)ws.cap_mask + 1;
    (void)cudaMemsetAsync(ws.keys, 0xFF, cap * sizeof(unsigned long long), st);
    (void)cudaMemsetAsync(ws.first, 0x7F, cap * sizeof(int), st);
    (void)launch_k(ldp::ldp_voxel_insert_kernel, dim3(grid), dim3(ldp::KV_THREADS), 0, st, xyz, (long long)n, h, h_dev, ws);
    (void)launch_k(ldp::ldp_voxel_flag_kernel, dim3(grid), dim3(ldp::KV_THREADS), 0, st, (long long)n, ws);
    g_launches += 2;
    scan_exclusive(ws.flag, ws.rank, n, ws.block_tot, cells_out, st);
}

// Steps 1 and 2 of the k-NN search, shared by ldp_statistical_outliers and ldp_estimate_normals: bounds and a trial grid,
// whose cell count sets the level-0 cell size (the one host synchronisation), then the pyramid and its level descriptors
// in pl.levels.  A coordinate that is not finite sets status_out[0] = 1 and leaves *n_levels_out = 0.
static int knn_pyramid(const float* xyz, int64_t n, int k, OutlierPlan& pl, cudaStream_t st, int32_t* status_out, int* n_levels_out) {
    *n_levels_out = 0;
    cudaError_t e;
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
        if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(outlier bounds)");
        (void)launch_k(ldp::ldp_voxel_bounds_kernel, dim3(rgrid), dim3(ldp::KV_THREADS), 0, st, xyz, (const float*)nullptr, (long long)n, ws);
        (void)launch_k(ldp::ldp_outlier_trial_size_kernel, dim3(1), dim3(1), 0, st, (const unsigned int*)ws.bounds_u, (long long)n, k, pl.h_trial);
        g_launches += 2;
        outlier_insert(xyz, n, 0.0, pl.h_trial, pl, grid, st, reinterpret_cast<int*>(ws.bounds_u + 7));
    }
    e = cudaMemcpyAsync(bu, ws.bounds_u, sizeof(bu), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&h_trial, pl.h_trial, sizeof(double), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return cuda_fail(e, "outlier trial grid");
    double mn[3], mx[3], ext = 0.0;
    bool finite = true;
    for (int c = 0; c < 3; ++c) {
        mn[c] = (double)host_f32_unordered(bu[c]);
        mx[c] = (double)host_f32_unordered(bu[4 + c]);
        finite = finite && std::isfinite(mn[c]) && std::isfinite(mx[c]);
        ext = std::max(ext, mx[c] - mn[c]);
    }
    if (!finite) {                                      // status_out[0] = 1 (little-endian int32, zeroed by the caller)
        e = cudaMemsetAsync(status_out, 1, 1, st);
        return e == cudaSuccess ? LDP_OK : cuda_fail(e, "cudaMemsetAsync(status)");
    }
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
            if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(outlier level)");
            outlier_insert(xyz, n, h, nullptr, pl, grid, st, pl.vstat + 1);
            (void)launch_k(ldp::ldp_voxel_count_kernel, dim3(grid), dim3(ldp::KV_THREADS), 0, st, (long long)n, ws);
            ++g_launches;
            scan_exclusive(ws.count, ws.seg, n, ws.block_tot, nullptr, st);
            (void)launch_k(ldp::ldp_voxel_group_kernel, dim3(grid), dim3(ldp::KV_THREADS), 0, st, (long long)n, ws, (const int*)ws.seg);
            (void)launch_k(ldp::ldp_outlier_cells_kernel, dim3(cgrid), dim3(ldp::KV_THREADS), 0, st, ws, pl.cell[n_levels]);
            (void)launch_k(ldp::ldp_outlier_pack_kernel, dim3(grid), dim3(ldp::KV_THREADS), 0, st, xyz, (long long)n,
                           (const int*)ws.members, pl.pts[n_levels]);
            g_launches += 3;
            ++n_levels;
            if (n_levels == ldp::OL_MAX_LEVELS || !(ext / h > 2.0)) break;
            h *= 8.0;
        }
    }
    (void)launch_k(ldp::ldp_outlier_levels_kernel, dim3(1), dim3(1), 0, st, lv, n_levels, pl.levels);
    ++g_launches;
    *n_levels_out = n_levels;
    return LDP_OK;
}

int ldp_statistical_outliers(const float* xyz, int64_t n, int32_t nb_neighbors, double std_ratio, int64_t* kept_idx_out,
                             double* mean_dist_out, double* stats_out, int32_t* status_out, void* workspace, size_t workspace_bytes,
                             void* stream) {
    g_launches = 0;
    if (nb_neighbors < 1 || nb_neighbors > ldp::OL_MAX_K) return fail(LDP_ERR_INVALID, "nb_neighbors must lie in [1, 64]");
    if (!(std_ratio > 0.0)) return fail(LDP_ERR_INVALID, "std_ratio must be positive");
    if (!status_out) return fail(LDP_ERR_INVALID, "null status_out");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    cudaError_t e = cudaMemsetAsync(status_out, 0, 3 * sizeof(int32_t), st);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(status)");
    if (n == 0) return LDP_OK;
    if (!xyz || !kept_idx_out || !workspace) return fail(LDP_ERR_INVALID, "null pointer");
    OutlierPlan pl;
    size_t need = 0;
    int rc = outlier_plan(n, workspace, &pl, &need);
    if (rc != LDP_OK) return rc;
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
        (void)launch_k(ldp::ldp_outlier_knn_kernel<false>, dim3(kgrid), dim3(ldp::OL_THREADS), (size_t)k * ldp::OL_THREADS * sizeof(double), st,
                       (const ldp::OutlierLevel*)pl.levels, n_levels, (long long)n, k,
                       g_outlier_shells > 0 ? g_outlier_shells : ldp::OL_DEFAULT_SHELLS, m, (int*)status_out, ldp::NormalArgs{});
        ++g_launches;
    }

    // 4. threshold, keep flags, kept indices
    {
        KernelTimer kt(st, "ldp_outlier_threshold");
        const long long n_part = (n + ldp::OL_CHUNK - 1) / ldp::OL_CHUNK;
        const unsigned pgrid = (unsigned)((n_part + ldp::KV_THREADS - 1) / ldp::KV_THREADS);
        (void)launch_k(ldp::ldp_outlier_partial_kernel, dim3(pgrid), dim3(ldp::KV_THREADS), 0, st, (const double*)m, (long long)n,
                       (const double*)nullptr, pl.part);
        (void)launch_k(ldp::ldp_outlier_stats_kernel, dim3(1), dim3(ldp::OL_FINAL), 0, st, (const double*)pl.part, n_part, (long long)n,
                       std_ratio, 0, stats);
        (void)launch_k(ldp::ldp_outlier_partial_kernel, dim3(pgrid), dim3(ldp::KV_THREADS), 0, st, (const double*)m, (long long)n,
                       (const double*)stats, pl.part);
        (void)launch_k(ldp::ldp_outlier_stats_kernel, dim3(1), dim3(ldp::OL_FINAL), 0, st, (const double*)pl.part, n_part, (long long)n,
                       std_ratio, 1, stats);
        (void)launch_k(ldp::ldp_outlier_flag_kernel, dim3(grid), dim3(ldp::KV_THREADS), 0, st, (const double*)m, (long long)n,
                       (const double*)stats, ws.flag);
        g_launches += 5;
        scan_exclusive(ws.flag, ws.rank, n, ws.block_tot, (int*)status_out + 1, st);
        (void)launch_k(ldp::ldp_outlier_kept_kernel, dim3(grid), dim3(ldp::KV_THREADS), 0, st, (const int*)ws.flag, (const int*)ws.rank,
                       (long long)n, reinterpret_cast<long long*>(kept_idx_out));
        ++g_launches;
    }
    if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e, "statistical outlier kernels");
    return LDP_OK;
}

// ---- oriented normals (ldp_outlier.cu: ldp_outlier_knn_kernel<true> and its epilogue)
int ldp_normals_workspace_bytes(int64_t n, int32_t k, size_t* bytes_out) {
    if (!bytes_out) return fail(LDP_ERR_INVALID, "null bytes_out");
    if (k < 3 || k > ldp::OL_MAX_K) return fail(LDP_ERR_INVALID, "k must lie in [3, 64]");
    OutlierPlan pl;
    return outlier_plan(n, nullptr, &pl, bytes_out, false);
}

int ldp_estimate_normals(const float* xyz, int64_t n, int32_t k, const float* centers, int32_t n_centers, const int32_t* center_idx,
                         float* normals_out, float* curvature_out, int32_t* knn_idx_out, int32_t* status_out, void* workspace,
                         size_t workspace_bytes, void* stream) {
    g_launches = 0;
    if (k < 3 || k > ldp::OL_MAX_K) return fail(LDP_ERR_INVALID, "k must lie in [3, 64]");
    if (center_idx && !centers) return fail(LDP_ERR_INVALID, "center_idx needs centers");
    if (centers && n_centers < 1) return fail(LDP_ERR_INVALID, "n_centers must be >= 1 when centers are given");
    if (!status_out) return fail(LDP_ERR_INVALID, "null status_out");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    cudaError_t e = cudaMemsetAsync(status_out, 0, 3 * sizeof(int32_t), st);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(status)");
    if (n == 0) return LDP_OK;
    if (!xyz || !normals_out || !workspace) return fail(LDP_ERR_INVALID, "null pointer");
    OutlierPlan pl;
    size_t need = 0;
    int rc = outlier_plan(n, workspace, &pl, &need, false);
    if (rc != LDP_OK) return rc;
    if (workspace_bytes < need) return fail(LDP_ERR_WORKSPACE, "normals workspace too small");
    const int k_eff = (int)std::min<int64_t>(k, n);
    int n_levels = 0;
    if ((rc = knn_pyramid(xyz, n, k_eff, pl, st, status_out, &n_levels)) != LDP_OK || n_levels == 0) return rc;
    {
        KernelTimer kt(st, "ldp_normals_knn_kernel");
        ldp::NormalArgs na{xyz, centers, center_idx, normals_out, curvature_out, knn_idx_out, centers ? n_centers : 0, 0};
        const unsigned kgrid = (unsigned)((n + ldp::OL_THREADS - 1) / ldp::OL_THREADS);
        (void)launch_k(ldp::ldp_outlier_knn_kernel<true>, dim3(kgrid), dim3(ldp::OL_THREADS),
                       (size_t)k_eff * ldp::OL_THREADS * (sizeof(double) + sizeof(int)), st,
                       (const ldp::OutlierLevel*)pl.levels, n_levels, (long long)n, k_eff,
                       g_outlier_shells > 0 ? g_outlier_shells : ldp::OL_DEFAULT_SHELLS, (double*)nullptr, (int*)status_out, na);
        ++g_launches;
    }
    if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e, "normal kernels");
    return LDP_OK;
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

// vec_hint: the host wrapper guarantees 16-byte aligned certainty planes when W % 4 == 0; the planes'
// addresses live in device memory, so alignment cannot be checked here without a copy.  Callers that
// cannot guarantee it set params->scalar_loads = 1 to force the scalar load path.

// L2 residency for the inter-kernel workspace (weights / p, winning neighbour, sample records): the path re-reads
// them from several kernels of the same call while ~0.2 GB of certainty planes stream through the 126 MB L2.
// An access-policy window marks the hot prefix of the workspace as persisting for the kernels of this call.
struct L2Window {
    cudaStream_t st;
    bool active;
    L2Window(cudaStream_t s, void* base, size_t bytes) : st(s), active(false) {
        static int mode = -1;          // -1 unknown, 0 off, 1 on
        static size_t max_window = 0, persist_bytes = 0;
        if (mode < 0) {
            const char* env = getenv("LDP_L2_PERSIST");
            mode = (env && env[0] == '1') ? 1 : 0;
            if (mode) {
                int dev = 0;
                cudaDeviceProp prop;
                if (cudaGetDevice(&dev) != cudaSuccess || cudaGetDeviceProperties(&prop, dev) != cudaSuccess ||
                    prop.persistingL2CacheMaxSize <= 0) { mode = 0; }
                else {
                    persist_bytes = (size_t)prop.persistingL2CacheMaxSize;
                    max_window = (size_t)prop.accessPolicyMaxWindowSize;
                    if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, persist_bytes) != cudaSuccess) { (void)cudaGetLastError(); mode = 0; }
                }
            }
        }
        if (mode != 1 || bytes == 0) return;
        cudaStreamAttrValue v = {};
        v.accessPolicyWindow.base_ptr = base;
        v.accessPolicyWindow.num_bytes = bytes < max_window ? bytes : max_window;
        const double ratio = (double)persist_bytes / (double)v.accessPolicyWindow.num_bytes;
        v.accessPolicyWindow.hitRatio = ratio >= 1.0 ? 1.0f : (float)ratio;
        v.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        v.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
        if (cudaStreamSetAttribute(st, cudaStreamAttributeAccessPolicyWindow, &v) == cudaSuccess) active = true;
        else (void)cudaGetLastError();
    }
    ~L2Window() {
        if (!active) return;
        cudaStreamAttrValue v = {};
        v.accessPolicyWindow.num_bytes = 0;
        (void)cudaStreamSetAttribute(st, cudaStreamAttributeAccessPolicyWindow, &v);
    }
};

int ldp_densify_refs(const ldp_params* params, const ldp_ref_desc* refs, const double* uniforms,
                     const ldp_outputs* out, void* workspace, size_t workspace_bytes, void* stream) {
    g_launches = 0;
    g_prof_n = 0;
    int rc = check_outputs(params, out);
    if (rc != LDP_OK) return rc;
    if (params->n_refs == 0) return LDP_OK;
    if (!refs || !workspace) return fail(LDP_ERR_INVALID, "null refs/workspace");
    if (params->rng_mode == LDP_RNG_EXPLICIT && !params->no_filter && !uniforms)
        return fail(LDP_ERR_INVALID, "explicit rng mode needs a uniform stream");
    Plan plan;
    char* base = reinterpret_cast<char*>(align_up(reinterpret_cast<size_t>(workspace), 256));
    rc = make_plan(params, base, &plan);
    if (rc != LDP_OK) return rc;
    if (plan.bytes + (size_t)(base - static_cast<char*>(workspace)) > workspace_bytes) return fail(LDP_ERR_WORKSPACE, "workspace too small");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // the winning-neighbour plane is written by the first kernel and gathered (1 byte per sample, random) by the fifth
    L2Window l2(st, plan.ws.bestk, (size_t)params->n_refs * plan.ws.n_pad);      // winning-neighbour plane (1 B / px)
    cudaError_t e = clear_launch_state(plan, st);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(launch state)");
    const int nsub = choose_subbatches(params->n_refs);
    if (nsub == 1) {
        rc = launch_sample(params, refs, uniforms, out, plan, vec_ok_for(params), st, 0, params->n_refs);
        if (rc != LDP_OK) return rc;
        rc = launch_geometry(params, refs, out, plan, 1, st, 0, params->n_refs, 0);
        if (rc != LDP_OK) return rc;
        return launch_pack(params, refs, out, plan, st);
    }
    SubStreams& ss = substreams();
    if (!ss.ok) return fail(LDP_ERR_CUDA, "cannot create internal streams");
    if ((e = cudaEventRecord(ss.start, st)) != cudaSuccess) return cuda_fail(e, "cudaEventRecord(start)");
    for (int h = 0; h < nsub; ++h) {
        const int lo = (int)(((long long)h * params->n_refs) / nsub), hi = (int)(((long long)(h + 1) * params->n_refs) / nsub);
        cudaStream_t sh = ss.s[h];
        if ((e = cudaStreamWaitEvent(sh, ss.start, 0)) != cudaSuccess) return cuda_fail(e, "cudaStreamWaitEvent(start)");
        rc = launch_sample(params, refs, uniforms, out, plan, vec_ok_for(params), sh, lo, hi - lo);
        if (rc != LDP_OK) return rc;
        rc = launch_geometry(params, refs, out, plan, 1, sh, lo, hi - lo, h);
        if (rc != LDP_OK) return rc;
        if ((e = cudaEventRecord(ss.done[h], sh)) != cudaSuccess) return cuda_fail(e, "cudaEventRecord(done)");
        if ((e = cudaStreamWaitEvent(st, ss.done[h], 0)) != cudaSuccess) return cuda_fail(e, "cudaStreamWaitEvent(done)");
    }
    return launch_pack(params, refs, out, plan, st);
}

int ldp_sample_refs(const ldp_params* params, const ldp_ref_desc* refs, const double* uniforms,
                    const ldp_outputs* out, void* workspace, size_t workspace_bytes, void* stream) {
    g_launches = 0;
    g_prof_n = 0;
    if (!params || !out || !out->status || !out->n_samples || !out->sel_idx) return fail(LDP_ERR_INVALID, "sample stage needs status, n_samples, sel_idx");
    if (params->n_refs == 0) return LDP_OK;
    if (!refs || !workspace) return fail(LDP_ERR_INVALID, "null refs/workspace");
    if (params->rng_mode == LDP_RNG_EXPLICIT && !params->no_filter && !uniforms)
        return fail(LDP_ERR_INVALID, "explicit rng mode needs a uniform stream");
    Plan plan;
    char* base = reinterpret_cast<char*>(align_up(reinterpret_cast<size_t>(workspace), 256));
    int rc = make_plan(params, base, &plan);
    if (rc != LDP_OK) return rc;
    if (plan.bytes + (size_t)(base - static_cast<char*>(workspace)) > workspace_bytes) return fail(LDP_ERR_WORKSPACE, "workspace too small");
    cudaError_t e = clear_launch_state(plan, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(launch state)");
    return launch_sample(params, refs, uniforms, out, plan, vec_ok_for(params), static_cast<cudaStream_t>(stream), 0, params->n_refs);
}

int ldp_triangulate_samples(const ldp_params* params, const ldp_ref_desc* refs, const ldp_outputs* out,
                            void* workspace, size_t workspace_bytes, void* stream) {
    g_launches = 0;
    g_prof_n = 0;
    int rc = check_outputs(params, out);
    if (rc != LDP_OK) return rc;
    if (!out->sel_idx) return fail(LDP_ERR_INVALID, "triangulate stage reads out->sel_idx / out->n_samples");
    if (params->n_refs == 0) return LDP_OK;
    if (!refs || !workspace) return fail(LDP_ERR_INVALID, "null refs/workspace");
    Plan plan;
    char* base = reinterpret_cast<char*>(align_up(reinterpret_cast<size_t>(workspace), 256));
    rc = make_plan(params, base, &plan);
    if (rc != LDP_OK) return rc;
    if (plan.bytes + (size_t)(base - static_cast<char*>(workspace)) > workspace_bytes) return fail(LDP_ERR_WORKSPACE, "workspace too small");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cudaError_t e = clear_launch_state(plan, st);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(launch state)");
    rc = launch_geometry(params, refs, out, plan, 0, st, 0, params->n_refs, 0);
    if (rc != LDP_OK) return rc;
    return launch_pack(params, refs, out, plan, st);
}

int ldp_postprocess_certainty(const ldp_params* params, const ldp_ref_desc* refs, float* outp,
                              size_t ref_stride, size_t plane_stride, void* stream) {
    g_launches = 0;
    g_prof_n = 0;
    if (!params || params->n_refs < 0 || params->H <= 0 || params->W <= 0) return fail(LDP_ERR_INVALID, "bad shape");
    if (params->n_refs == 0) return LDP_OK;
    if (!refs || !outp) return fail(LDP_ERR_INVALID, "null refs/out");
    if ((long long)params->H * params->W > (1ll << 24)) return fail(LDP_ERR_INVALID, "map too large");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int N = params->H * params->W;
    const int bx = std::min((N + ldp::KP_THREADS - 1) / ldp::KP_THREADS, 4 * sm_count());
    const dim3 grid((unsigned)bx, LDP_MAX_NN, (unsigned)params->n_refs);
    { KernelTimer kt(st, "ldp_prologue_kernel");
      (void)launch_k(ldp::ldp_prologue_kernel, dim3(grid), dim3(ldp::KP_THREADS), 0, st, *params, refs, outp, ref_stride, plane_stride); }
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "ldp_prologue_kernel");
    return LDP_OK;
}

}  // extern "C"
