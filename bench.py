#!/usr/bin/env python
"""Benchmark of the post-matching densification hot path (BASELINE.json metric / config).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]

Workload (config.workload): BASELINE.json configs[1] -- MipNeRF360-garden-shaped scene, 185 views, RoMa 'fast'
(512x512 maps), reference fraction 0.25 -> 46 reference views, 4 neighbours each -> 184 view pairs, 10 000 matches
per reference, all filters on; synthetic matcher outputs (the RoMa network is out of scope).  One "step" = one pass
of sample -> triangulate -> filter -> colour over all 46 reference views (one launch sequence of the C-ABI call).

value      filtered 3D points / s, inputs resident in HBM, CUDA-event timed, max over ranks.  Weak scaling: every rank
           processes its own 46-view batches, each step in flight reads its OWN input tensors, and there is NO collective
           per step: the points stay on the rank that made them; the ranks' kept-point counts (what a rank needs to place
           its slice in the global output) are exchanged ONCE, after the last step, inside the timed region.
e2e        same metric through the public batched API from HOST buffers (pinned): certainty planes + reference images
           are copied host->device every step, the warp planes stay in pinned host memory and are gathered over PCIe at
           the sampled pixels only (zero-copy), results are read back device->host.
api        the drop-in entry point an integrator calls, core.pipeline.triangulate_refs (descriptors rebuilt per call,
           results returned as numpy arrays), with device-resident matcher outputs and with pageable host tensors.
roofline   dominant kernel (the fused front kernel: every certainty value read once, nn*H*W*4 bytes per view), duration
           from back-to-back launches of that kernel alone between two CUDA events; by_kernel: every kernel of the step
           (event-bracketed inside the step); path_frac: SURVEY 8d bytes of the whole step / step time / peak.
config5    BASELINE.json configs[4]: 1000-view scene, 'base' 640x640, 250 reference views sharded over the ranks
           (distributed.shard_bounds), Philox keyed by the global view index; timed region = every launch of the rank +
           ONE final point all-gather (single NCCL collective of the rank's packed cloud, counts in its header) + the
           device-side concatenation in rank order; checked bit-exact against the single-GPU result.
cpu_baseline / --impl reference
           the oracle port of the reference's CPU path (oracle/densify_oracle.py, bit-identical to the reference in
           the build container) on the host cores, one process per core, bounded sample.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import multiprocessing as mp
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOAD = dict(name="garden-shaped 185 views, RoMa fast 512x512, ref_fraction 0.25 (46 refs), 4 nn/ref (184 pairs), "
                     "M=10000, all filters on", n_views=185, setting="fast", ref_fraction=0.25, nn=4, M=10000)
CONFIG5 = dict(name="1000 views, RoMa base 640x640, ref_fraction 0.25 (250 refs), 4 nn/ref (1000 pairs), M=10000, all filters on",
               n_views=1000, setting="base", ref_fraction=0.25, nn=4, M=10000, refs_per_launch=84)
METRIC = "filtered_points_per_sec"
UNIT = "points/s"
CPU_SAMPLE = dict(steps=8, warmup=3)          # cpu_baseline inside the GPU arm: same code and sample shape as --impl reference


# ---------------------------------------------------------------------------------------------------------
# CPU arm: oracle port on host cores
# ---------------------------------------------------------------------------------------------------------
def _cpu_worker(wid: int, n_steps: int, ready, go, results, seed: int) -> None:
    import torch
    torch.set_num_threads(1)
    from lichtfeld_densification_plugin_b200 import synth
    from oracle import densify_oracle as O
    scene = synth.make_scene(WORKLOAD["n_views"], WORKLOAD["setting"], WORKLOAD["ref_fraction"], WORKLOAD["nn"])
    cams = scene.cameras
    rp = wid % scene.n_refs
    inp = synth.synth_ref_inputs(scene, rp, device="cpu", cert_family="R", seed=seed)
    oc = lambda c: O.OracleCamera(c.uid, c.width, c.height, c.K, c.R, c.t, c.P, c.C)
    cfg = O.OracleConfig(matches_per_ref=WORKLOAD["M"], w_match=scene.w_match, h_match=scene.h_match)
    nn = len(inp["nbr_indices"])
    certs = [inp["cert"][k] for k in range(nn)]
    warps = [inp["warp"][k] for k in range(nn)]
    img = inp["image"].numpy()
    rc, ncs = oc(cams[inp["ref_index"]]), [oc(cams[j]) for j in inp["nbr_indices"]]
    ready.put(wid)
    go.wait()
    stamps = []
    for s in range(n_steps):
        t0 = time.time()
        res = O.triangulate_ref(certs, warps, img, rc, ncs, cfg, rng=np.random.RandomState(1000 * wid + s))
        stamps.append((t0, time.time(), 0 if res is None else int(res.xyz.shape[0]), nn))
    results.put((wid, stamps))


def run_cpu_arm(workers: int, steps: int, warmup: int, seed: int = 0):
    """Every worker process runs `warmup + steps` reference views of the workload (one per step)."""
    ctx = mp.get_context("fork")
    ready, results, go = ctx.Queue(), ctx.Queue(), ctx.Event()
    procs = [ctx.Process(target=_cpu_worker, args=(w, warmup + steps, ready, go, results, seed)) for w in range(workers)]
    for p in procs:
        p.start()
    for _ in procs:
        ready.get()
    go.set()
    out = [results.get() for _ in procs]
    for p in procs:
        p.join()
    t_start = min(st[warmup][0] for _, st in out)
    t_end = max(st[-1][1] for _, st in out)
    pts = sum(s[2] for _, st in out for s in st[warmup:])
    pairs = sum(s[3] for _, st in out for s in st[warmup:])
    per_ref = [s[1] - s[0] for _, st in out for s in st[warmup:]]
    wall = t_end - t_start
    return dict(points_per_s=pts / wall, pairs_per_s=pairs / wall, wall_s=wall, refs=workers * steps,
                ms_per_ref_single_core=1e3 * float(np.median(per_ref)), points=pts)


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_sample_text(workers: int, steps: int, warmup: int) -> str:
    return (f"{workers} processes (one per host core, torch threads = 1) x {steps} timed reference views each of the workload "
            f"after {warmup} warm-up views (1 view per step per process)")


def reference_arm(args) -> None:
    """The reference's CPU implementation of the path (oracle port; the reference is pure Python and was checked
    bit-identical against it in the build container) on every host core.  --steps / --warmup are honoured as given:
    a step is one reference view per worker process (a bounded sample of the 46-view workload)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    workers = max(1, min(host_cores(), 32))
    steps = max(1, args.steps if args.steps is not None else 20)
    warmup = max(0, args.warmup if args.warmup is not None else 3)
    r = run_cpu_arm(workers, steps, warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["points_per_s"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": 1e3 * r["wall_s"] / steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32 geometry / f64 cdf, sampson, colour", "data": "synthetic",
        "config": {"workload": WORKLOAD["name"]},
        "pairs_per_sec": r["pairs_per_s"],
        "cpu_baseline": {"value": r["points_per_s"], "unit": UNIT, "cores": workers, "kind": "port",
                         "sample": cpu_sample_text(workers, steps, warmup),
                         "ms_per_ref_single_core": r["ms_per_ref_single_core"]},
        "e2e": {"value": r["points_per_s"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, index: int, period_s: float = 0.02) -> None:
        super().__init__(daemon=True)
        self.index, self.period = index, period_s
        self.samples, self.reasons, self.max_mhz, self.power = [], set(), None, []
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(t.strip().isdigit() for t in vis.split(",")) else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def run(self) -> None:
        if not self.ok:
            return
        nv = self.nv
        while not self._halt.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self) -> dict:
        self._halt.set()
        self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples), "power_w_max": max(self.power) if self.power else None}


# ---------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------
def measured_hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def recorded_traffic():
    """dram bytes per launch of the dominant kernel from the committed ncu capture, if any."""
    try:
        with open(os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")) as f:
            return json.load(f).get("dram_bytes_per_launch")
    except Exception:
        return None


def recorded_instructions():
    """warp instructions one step executes, from the committed ncu captures (profiles/dominant_kernel_traffic.json)."""
    try:
        with open(os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")) as f:
            d = json.load(f).get("warp_instructions_per_step") or {}
        return int(sum(v for v in d.values() if isinstance(v, (int, float)))), d.get("note")
    except Exception:
        return None, None


DUMP_MAX_BYTES = 64 << 20


def outputs_snapshot(o, R: int) -> dict:
    """What a caller of the timed path receives from one step, copied to the host: every kept point (xyz, rgb, err, rows of
    the views in order) and per view its row offset, status word and sample count.  More points than fit DUMP_MAX_BYTES
    are cut to a fixed seeded sample of rows (``point_rows`` lists them)."""
    K = o.total_points()
    rows = None
    per_row = 7 * 4 + 8
    if K * per_row > DUMP_MAX_BYTES - 64 * (R + 1):
        rows = np.sort(np.random.RandomState(0).choice(K, (DUMP_MAX_BYTES - 64 * (R + 1)) // per_row, replace=False))
    snap = {}
    for name in ("xyz", "rgb", "err"):
        a = getattr(o, name)[:K].cpu().numpy().astype(np.float32)
        snap[name] = a if rows is None else a[rows]
    if rows is not None:
        snap["point_rows"] = rows.astype(np.float64)
    snap["ref_offset"] = o.ref_offset[:R + 1].cpu().numpy().astype(np.float64)
    snap["status"] = o.status[:R].cpu().numpy().astype(np.float64)
    snap["n_samples"] = o.n_samples[:R].cpu().numpy().astype(np.float64)
    return snap


def write_outputs(out_dir: str, snap: dict) -> None:
    os.makedirs(out_dir, exist_ok=True)
    for name, a in snap.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def _dbg(msg: str) -> None:
    if os.environ.get("BENCH_DEBUG"):
        print(f"[bench rank {os.environ.get('RANK', '0')}] {msg}", file=sys.stderr, flush=True)


class SceneInputs:
    """Synthetic matcher outputs of `n` reference views of a scene, resident on one device."""

    def __init__(self, scene, ref_positions, dev, seed: int):
        import torch
        from lichtfeld_densification_plugin_b200 import synth
        n, nn, H, W = len(ref_positions), scene.nn, scene.H, scene.W
        self.cert = torch.empty((n, nn, H, W), dtype=torch.float32, device=dev)
        self.warp = torch.empty((n, nn, H, W, 4), dtype=torch.float32, device=dev)
        self.image = torch.empty((n, scene.h_match, scene.w_match, 3), dtype=torch.uint8, device=dev)
        self.table, self.positions = [], list(ref_positions)
        for i, rp in enumerate(ref_positions):
            inp = synth.synth_ref_inputs(scene, rp, device=dev, cert_family="R", seed=seed)
            self.cert[i], self.warp[i], self.image[i] = inp["cert"], inp["warp"], inp["image"]
            self.table.append((inp["ref_index"], inp["nbr_indices"]))

    def batch(self, eng, scene, lo: int, hi: int, stream_base: int, cert=None, warp=None, image=None):
        cert = self.cert if cert is None else cert
        warp = self.warp if warp is None else warp
        image = self.image if image is None else image
        cams, nn = scene.cameras, scene.nn
        b = eng.new_batch(scene.H, scene.W, scene.w_match, scene.h_match)
        for i in range(lo, hi):
            ri, nb = self.table[i]
            b.add([cert[i, k] for k in range(nn)], [warp[i, k] for k in range(nn)], image[i], cams[ri],
                  [cams[j] for j in nb], rng_stream=stream_base + self.positions[i])
        return b


def config5_block(args, dev, rank: int, world: int, ring) -> dict:
    """BASELINE.json configs[4]: the sharded scene with the final point all-gather (see the module docstring)."""
    import torch
    import torch.distributed as dist
    from lichtfeld_densification_plugin_b200 import distributed as D
    from lichtfeld_densification_plugin_b200 import synth
    from lichtfeld_densification_plugin_b200.engine import PathConfig
    from lichtfeld_densification_plugin_b200.output import ConcatPlan, PackedCloud

    scene = synth.make_scene(CONFIG5["n_views"], CONFIG5["setting"], CONFIG5["ref_fraction"], CONFIG5["nn"])
    # views per launch: at most CONFIG5["refs_per_launch"], the rank's views cut into launches of equal size (a launch of 84 views
    # at 640^2 fills the device better than three of 32: 1.0 vs 1.3 ms for the 250 views of one GPU)
    R_all, per_max = scene.n_refs, int(os.environ.get("BENCH_C5_REFS_PER_LAUNCH", CONFIG5["refs_per_launch"]))
    r_lo, r_hi = D.shard_bounds(R_all, rank, world)
    r_max = max(D.shard_bounds(R_all, q, world)[1] - D.shard_bounds(R_all, q, world)[0] for q in range(world))
    n_launch = max(1, -(-r_max // per_max))
    per = -(-r_max // n_launch)
    cfg = PathConfig(matches_per_ref=CONFIG5["M"], seed=5)
    eng0 = ring.engines[0]
    sel_cap = eng0.sel_capacity(cfg.matches_per_ref)
    depth = ring.depth

    class Shard:
        def __init__(self, lo, hi, cap_refs, cloud=None):
            self.lo, self.hi = lo, hi
            self.inputs = SceneInputs(scene, list(range(lo, hi)), dev, seed=500)
            self.chunks = [(a, min(a + per, hi - lo)) for a in range(0, hi - lo, per)]
            self.outs = [eng0.alloc_outputs(b - a, sel_cap) for a, b in self.chunks]
            self.prepared = []
            for c, (a, b) in enumerate(self.chunks):
                j = c % depth
                batch = self.inputs.batch(ring.engines[j], scene, a, b, stream_base=0)
                descs = ring.engines[j].upload_descs(batch)
                self.prepared.append((j, ring.engines[j].prepare(batch, cfg, descs_dev=descs, outputs=self.outs[c])))
            # the rank's cloud (the SAME capacity on every rank); N > 1: it lives in symmetric memory, where the peers read it
            self.cloud = cloud if cloud is not None else PackedCloud(cap_refs * sel_cap, dev)
            self.plan = ConcatPlan([o.xyz for o in self.outs], [o.rgb for o in self.outs], [o.err for o in self.outs],
                                   [o.ref_offset[o.n_refs:o.n_refs + 1] for o in self.outs], per * sel_cap)

        def launch_all(self):
            """every launch of the shard on the ring streams, then the rank's cloud on the main stream"""
            main = torch.cuda.current_stream(dev)
            for st in ring.streams:
                st.wait_stream(main)
            for j, p in self.prepared:
                with torch.cuda.stream(ring.streams[j]):
                    p.launch()
            for st in ring.streams:
                main.wait_stream(st)
            self.plan.run(self.cloud)

    cap_refs = max(D.shard_bounds(R_all, q, world)[1] - D.shard_bounds(R_all, q, world)[0] for q in range(world))
    lo, hi = D.shard_bounds(R_all, rank, world)
    # N > 1: the final all-gather is our own kernel reading the peers' clouds over NVLink (distributed.PeerClouds); the NCCL
    # collective + compaction (distributed.all_gather_cloud) is timed beside it, and is what runs if the node offers no
    # symmetric memory
    peer, peer_err = None, None
    if world > 1 and not int(os.environ.get("BENCH_NO_PEER", "0")):
        try:
            peer = D.PeerClouds(cap_refs * sel_cap, dev)
        except Exception as exc:      # no peer access on this node: the library collective remains
            peer_err = f"{type(exc).__name__}: {exc}"
        ok = torch.tensor([1 if peer is not None else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            peer = None
    shard = Shard(lo, hi, cap_refs, cloud=peer.cloud if peer is not None else None)
    gathered = PackedCloud(world * shard.cloud.capacity, dev) if world > 1 else None
    scratch = torch.empty((world, shard.cloud.packed.numel()), dtype=torch.uint8, device=dev) if world > 1 else None
    torch.cuda.synchronize(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def one_pass(use_peer: bool):
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record()
        shard.launch_all()
        e[1].record()
        if use_peer == "pull":
            total, offsets = peer.gather(out=gathered, mode="pull")
        elif use_peer:
            total, offsets = peer.gather()
        else:
            total, offsets = D.all_gather_cloud(shard.cloud, out=gathered, scratch=scratch)
        e[2].record()
        return e, total, offsets

    passes = max(3, min(10, args.steps))

    def timed_passes(use_peer: bool):
        for _ in range(2):
            one_pass(use_peer)
        barrier()
        ms_all, ms_compute, ms_gather = [], [], []
        total = offsets = None
        for _ in range(passes):
            barrier()
            e, total, offsets = one_pass(use_peer)
            torch.cuda.synchronize(dev)
            ms_all.append(e[0].elapsed_time(e[2]))
            ms_compute.append(e[0].elapsed_time(e[1]))
            ms_gather.append(e[1].elapsed_time(e[2]))
        t = torch.tensor([float(np.median(ms_all)), float(np.median(ms_compute)), float(np.median(ms_gather))], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()], total, offsets

    nccl_ms = pull_ms = None
    if world > 1 and peer is not None:
        nccl_ms, _, _ = timed_passes(False)            # the library collective, for comparison
        pull_ms, _, _ = timed_passes("pull")           # our kernel reading the peers instead of writing to them
    (ms, ms_c, ms_g), total, offsets = timed_passes(peer is not None)
    n_total = int(offsets[-1].item())
    # ---- bit-exact check against the single-GPU result: rank 0 recomputes the whole scene alone (outside the timed region)
    same = None
    sha = None
    if rank == 0:
        if world > 1:
            whole = Shard(0, R_all, R_all)
            whole.launch_all()
            torch.cuda.synchronize(dev)
            ref_cloud = whole.cloud
        else:                                   # N = 1: another cut into launches (46 views per launch) must give the same cloud
            per_alt = 46
            outs, preps = [], []
            for a in range(0, R_all, per_alt):
                b = min(a + per_alt, R_all)
                batch = shard.inputs.batch(eng0, scene, a, b, stream_base=0)
                o = eng0.alloc_outputs(b - a, sel_cap)
                preps.append(eng0.prepare(batch, cfg, outputs=o))
                preps[-1].launch()
                torch.cuda.synchronize(dev)
                outs.append(o)
            from lichtfeld_densification_plugin_b200.output import concat_launches
            ref_cloud = concat_launches(outs)
            torch.cuda.synchronize(dev)
        k = ref_cloud.total_points()
        same = bool(k == n_total and torch.equal(ref_cloud.xyz[:k], total.xyz[:k]) and torch.equal(ref_cloud.rgb[:k], total.rgb[:k])
                    and torch.equal(ref_cloud.err[:k], total.err[:k]))
        if not same and world == 1 and os.environ.get("BENCH_DEBUG"):
            def per_view(os_, chunks_):
                d = {}
                for o_, (a_, b_) in zip(os_, chunks_):
                    off_ = o_.ref_offset.cpu().numpy(); ns_ = o_.n_samples.cpu().numpy(); st_ = o_.status.cpu().numpy()
                    ws_ = o_.weight_sum.cpu().numpy(); uu_ = o_.uniforms_used.cpu().numpy(); rr_ = o_.rounds.cpu().numpy()
                    for r_ in range(b_ - a_):
                        d[a_ + r_] = (int(ns_[r_]), int(st_[r_]), int(off_[r_ + 1] - off_[r_]), float(ws_[r_]), int(uu_[r_]), int(rr_[r_]))
                return d
            mine = per_view(shard.outs, shard.chunks)
            alt = per_view(outs, [(a_, min(a_ + per_alt, R_all)) for a_ in range(0, R_all, per_alt)])
            bad = [v for v in range(R_all) if mine[v] != alt[v]]
            print("[bench] config5 cut check: views that differ (n_samples, status, kept):", [(v, mine[v], alt[v]) for v in bad[:10]],
                  "totals", n_total, k, file=sys.stderr)
        h = hashlib.sha1()
        for a in (total.xyz[:n_total], total.rgb[:n_total], total.err[:n_total]):
            h.update(a.cpu().numpy().tobytes())
        sha = h.hexdigest()
    pad_bytes = int(shard.cloud.packed.numel())
    return {
        "workload": CONFIG5["name"], "refs_total": R_all, "refs_this_rank": hi - lo, "refs_per_launch": per,
        "launches_per_rank": len(shard.chunks), "steps_in_flight": depth, "passes_timed": passes,
        "ms": ms, "ms_launches_and_local_concat": ms_c, "ms_all_gather_and_concat": ms_g,
        "points": n_total, "points_per_sec": n_total / (ms * 1e-3), "pairs_per_sec": R_all * scene.nn / (ms * 1e-3),
        "all_gather": {"collective": ("none (N = 1)" if world == 1 else
                                      "own kernel: ldp_scatter_points pushes this rank's rows (exactly its count; counts read from the peers' "
                                      "headers) into every rank's rank-ordered cloud over NVLink (symmetric memory), two device-side "
                                      "barriers; no padding moved" if peer is not None else
                                      "ncclAllGather (one call: count header + xyz | rgb | err, padded to capacity) + ldp_concat_points"),
                       "bytes_received_per_rank": (int(28 * n_total * (world - 1) / world) if peer is not None else pad_bytes * (world - 1)) if world > 1 else 0,
                       "payload_bytes_total": 28 * n_total, "ms": ms_g,
                       "gb_per_s_received_per_rank": ((28 * n_total * (world - 1) / world if peer is not None else pad_bytes * (world - 1)) / (ms_g * 1e-3) / 1e9) if world > 1 and ms_g > 0 else None,
                       "nccl_all_gather_plus_concat_ms": nccl_ms[2] if nccl_ms else None, "nccl_total_ms": nccl_ms[0] if nccl_ms else None,
                       "pull_variant_ms": pull_ms[2] if pull_ms else None,
                       "peer_memory_error": peer_err},
        "limiter": ("all-gather" if ms_g > ms_c else "launches") if world > 1 else "launches",
        "equals_single_gpu_result": same if world > 1 else None,
        "equals_other_cut_into_launches": same if world == 1 else None,
        "cloud_sha1": sha, "timing": "CUDA events on the main stream, median over the passes, max over ranks; host sync only between passes",
    }


def api_block(args, dev, scene, inputs, cfg_M: int) -> dict:
    """The drop-in entry point: core.pipeline.triangulate_refs on _MatchedReference objects (descriptors rebuilt per call,
    numpy results), with the matcher outputs on the device and with pageable host tensors (what the reference's
    .to('cpu') leaves behind, core/pipeline.py:432-442)."""
    import torch
    from lichtfeld_densification_plugin_b200.core import pipeline as PL
    from lichtfeld_densification_plugin_b200.core.config import DensePipelineConfig
    cams = scene.cameras
    cfg = DensePipelineConfig(output_path="/tmp/bench_api.ply", matches_per_ref=cfg_M)
    ctx = PL._TriangulationContext(cameras=PL._build_camera_lookup(cams), config=cfg, matcher_sample_cap=0.9,
                                   w_match=scene.w_match, h_match=scene.h_match)

    def matched(cert, warp, image_np):
        out = []
        for i, (ri, nb) in enumerate(inputs.table):
            packed = PL._PackedReferenceBatch(ref_id=cams[ri].uid, ref_path="", imA_np=image_np[i], maskA_np=None,
                                              wA_cam=cams[ri].width, hA_cam=cams[ri].height, nn_ids=[cams[j].uid for j in nb],
                                              nn_masks=[None] * len(nb), nn_arrays=[])
            out.append(PL._MatchedReference(packed=packed, warp_list_cpu=[warp[i, k] for k in range(len(nb))],
                                            cert_list_cpu=[cert[i, k] for k in range(len(nb))], pair_index_by_nbr={}, image_by_nbr={}))
        return out

    def run(mrs, n):
        streams = [int(mr.packed.ref_id) for mr in mrs]
        pts = 0
        res = None
        for _ in range(3):           # the previous call's results stay alive while the next one runs, as in the timed loop:
            res = PL.triangulate_refs(mrs, ctx, rng_streams=streams)      # both page-locked result blocks exist after this
        torch.cuda.synchronize(dev)
        per_call = []
        t0 = time.perf_counter()
        for _ in range(n):
            t1 = time.perf_counter()
            res = PL.triangulate_refs(mrs, ctx, rng_streams=streams)      # synchronises: the results are host arrays
            pts = sum(0 if r is None else int(r.xyz.shape[0]) for r in res)
            per_call.append(time.perf_counter() - t1)
        torch.cuda.synchronize(dev)
        if os.environ.get("BENCH_DEBUG"):
            print("[bench] api per-call ms:", [round(1e3 * t, 2) for t in per_call], file=sys.stderr)
        return (time.perf_counter() - t0) / n, pts, sorted(per_call)[len(per_call) // 2]

    image_dev_np = inputs.image            # device tensor: _to_device accepts tensors as well as numpy arrays
    n = max(3, min(args.steps, 20))
    s_dev, pts, med_dev = run(matched(inputs.cert, inputs.warp, image_dev_np), n)
    h_cert, h_warp, h_img = inputs.cert.cpu(), inputs.warp.cpu(), inputs.image.cpu().numpy()
    s_host, pts_h, med_host = run(matched(h_cert, h_warp, h_img), max(2, min(n, 5)))
    return {"entry_point": "core.pipeline.triangulate_refs (46 _MatchedReference per call, numpy results)",
            "device_resident_inputs": {"ms_per_step": 1e3 * s_dev, "ms_per_step_median": 1e3 * med_dev, "points_per_sec": pts / s_dev},
            "pageable_host_inputs": {"ms_per_step": 1e3 * s_host, "ms_per_step_median": 1e3 * med_host, "points_per_sec": pts_h / s_host,
                                     "h2d_bytes_per_step": int(h_cert.numel() * 4 + h_warp.numel() * 4 + h_img.size)},
            "points_per_step": pts}


def gpu_arm(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    steps = max(1, args.steps if args.steps is not None else 1000)
    warmup = max(3, args.warmup if args.warmup is not None else 10)
    args.steps, args.warmup = steps, warmup

    cpu_base = None
    if world == 1 and rank == 0 and not args.no_cpu_baseline and not args.quick:
        # before CUDA is initialised in this process (workers are forked)
        workers = max(1, min(host_cores(), 32))
        r = run_cpu_arm(workers, steps=CPU_SAMPLE["steps"], warmup=CPU_SAMPLE["warmup"])
        cpu_base = {"value": r["points_per_s"], "unit": UNIT, "cores": workers, "kind": "port",
                    "sample": cpu_sample_text(workers, CPU_SAMPLE["steps"], CPU_SAMPLE["warmup"]),
                    "ms_per_ref_single_core": r["ms_per_ref_single_core"], "pairs_per_sec": r["pairs_per_s"]}

    import torch
    import torch.distributed as dist
    from lichtfeld_densification_plugin_b200 import synth
    from lichtfeld_densification_plugin_b200.engine import DensifyRing, PathConfig

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # stdout carries ONE JSON line: whatever libraries write to file descriptor 1 while the run lasts (NCCL prints its version
    # there) goes to stderr; the descriptor is restored for the line itself
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj) -> None:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(obj), flush=True)
        os.dup2(2, 1)

    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    scene = synth.make_scene(WORKLOAD["n_views"], WORKLOAD["setting"], WORKLOAD["ref_fraction"], WORKLOAD["nn"])
    R, nn, H, W = scene.n_refs, scene.nn, scene.H, scene.W

    # Consecutive steps are independent batches: DEPTH of them are kept in flight (engine.DensifyRing: one workspace and
    # one CUDA stream per slot), each slot with its OWN input tensors (different synthetic matcher outputs), so the
    # HBM-bound first kernel of one step runs beside the latency-bound draw / geometry kernels of another and no step
    # can hit another step's lines in L2.  BENCH_PIPELINE_DEPTH=1 times one launch sequence at a time only.
    DEPTH = max(1, int(os.environ.get("BENCH_PIPELINE_DEPTH", "3")))
    ring = DensifyRing(dev, DEPTH)
    eng = ring.engines[0]
    cfg = PathConfig(matches_per_ref=WORKLOAD["M"], seed=0)
    # Weak scaling = the same work on every GPU: all ranks process the same synthetic batches (same seeds, same Philox streams).
    # Seeded by rank instead (BENCH_DATA_PER_RANK=1), the batches themselves differ in cost by up to 6 % (measured on ONE GPU:
    # 0.1366 ms per step with the seeds of ranks 0 / 6, 0.1447 / 0.1451 ms with those of ranks 3 / 7), and the slowest batch
    # would be reported as a scaling loss.
    data_rank = rank if int(os.environ.get("BENCH_DATA_PER_RANK", "0")) else int(os.environ.get("BENCH_DATA_RANK", "0"))
    slots = [SceneInputs(scene, list(range(R)), dev, seed=100 + data_rank + 1000 * j) for j in range(DEPTH)]
    torch.cuda.synchronize(dev)
    batches = [slots[j].batch(ring.engines[j], scene, 0, R, stream_base=data_rank * R) for j in range(DEPTH)]
    descs = [ring.engines[j].upload_descs(batches[j]) for j in range(DEPTH)]
    sel_cap = eng.sel_capacity(cfg.matches_per_ref)
    NBUF = max(2, DEPTH)      # output buffers in rotation
    outs = [eng.alloc_outputs(R, sel_cap) for _ in range(NBUF)]
    prepared = {}      # (engine slot, output buffer) -> PreparedLaunch: the host side of a step is one C call
    counts_all = torch.zeros((world, NBUF), dtype=torch.int64, device=dev) if world > 1 else None

    def step(i: int, depth: int):
        k = i % NBUF
        j = i % depth if depth > 1 else 0
        st = ring.streams[j] if depth > 1 else torch.cuda.current_stream(dev)
        if (j, k) not in prepared:
            prepared[(j, k)] = ring.engines[j].prepare(batches[j], cfg, descs_dev=descs[j], outputs=outs[k])
        with torch.cuda.stream(st):
            prepared[(j, k)].launch()
        return outs[k]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    _dbg("setup done")

    def timed(depth: int, n_steps: int):
        """n_steps steps, `depth` in flight, between two events on the main stream; returns (ms, last outputs).  N > 1: the
        ranks' kept-point counts of the last NBUF steps are exchanged once, after the last step, inside the timed region."""
        main = torch.cuda.current_stream(dev)
        for i in range(warmup):
            step(i, depth)
        if depth > 1:
            for st in ring.streams:
                main.wait_stream(st)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if depth > 1:
            for st in ring.streams:
                st.wait_event(e0)
        last = None
        t_host = time.perf_counter()
        for i in range(n_steps):
            last = step(i, depth)
        issue_ms[depth] = 1e3 * (time.perf_counter() - t_host)      # host time to enqueue the steps (the device runs behind)
        if depth > 1:
            for st in ring.streams:
                main.wait_stream(st)
        e_own = torch.cuda.Event(enable_timing=True)
        e_own.record()                                   # this rank's own steps are done (diagnostic: before the exchange)
        if world > 1:
            mine = torch.stack([o.ref_offset[R] for o in outs])
            dist.all_gather_into_tensor(counts_all.view(-1), mine)
        e1.record()
        barrier()
        own_ms[depth] = e0.elapsed_time(e_own)
        return e0.elapsed_time(e1), last

    own_ms = {}
    issue_ms = {}

    sampler = ClockSampler(local_rank)
    sampler.start()
    ring_reserve = [e.sm_reserve for e in ring.engines]

    def set_reserve(values):
        """(the reserve travels in ldp_params: prepared launches are rebuilt when it changes)"""
        for e, v in zip(ring.engines, values):
            e.sm_reserve = v
        prepared.clear()
    set_reserve([0] * DEPTH)                             # one launch sequence at a time: the first draw kernel takes every SM
    ms_single, o = timed(1, steps)
    ms_total = ms_single
    if DEPTH > 1:
        set_reserve(ring_reserve)                        # DensifyRing's setting (16): SMs for the other steps in flight
        ms_total, o = timed(DEPTH, steps)                # the headline: DEPTH steps in flight
    _dbg("timed loop done")
    # the last timed step's results, before the load loop below writes the output buffers again
    snap = outputs_snapshot(o, R) if args.dump_outputs and rank == 0 else None
    # keep the GPU under the same load a little longer so the clock sampler sees the loaded state
    t_end = time.time() + (0.0 if args.quick else max(0.0, 0.6 - ms_total / 1e3))
    j = 0
    while time.time() < t_end:
        # wall-clock bounded, so the ranks run different numbers of iterations: no collectives in here
        step(j, DEPTH)
        j += 1
        if j % 64 == 0:
            torch.cuda.synchronize(dev)
    torch.cuda.synchronize(dev)
    clocks = sampler.stop()

    _dbg("clock load loop done")
    launches_per_step = o.launches
    total_pts = o.total_points()
    S_total = int(o.n_samples.sum().item())
    per_rank_ms = None
    if world > 1:
        t = torch.tensor([ms_total, ms_single], dtype=torch.float64, device=dev)
        mine_t = torch.tensor([own_ms.get(DEPTH, ms_total), own_ms.get(1, ms_single), issue_ms.get(DEPTH, 0.0),
                               float(clocks.get("sm_mhz") or 0.0), float(clocks.get("power_w_max") or 0.0)], dtype=torch.float64, device=dev)
        allt = [torch.zeros_like(mine_t) for _ in range(world)]
        dist.all_gather(allt, mine_t)
        per_rank_ms = {"note": "each rank's own steps, before the count exchange that ends the timed region",
                       "ms_per_step": [round(float(x[0].item()) / steps, 5) for x in allt],
                       "ms_per_step_one_launch_at_a_time": [round(float(x[1].item()) / steps, 5) for x in allt],
                       "host_enqueue_ms_per_step": [round(float(x[2].item()) / steps, 5) for x in allt],
                       "sm_mhz_median_under_load": [float(x[3].item()) for x in allt],
                       "power_w_max": [round(float(x[4].item()), 1) for x in allt]}
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, ms_single = float(t[0].item()), float(t[1].item())
        c = torch.tensor([total_pts, S_total], dtype=torch.int64, device=dev)
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
        total_pts_all, S_all = int(c[0].item()), int(c[1].item())
    else:
        total_pts_all, S_all = total_pts, S_total
    ms_step = ms_total / steps
    ms_single_step = ms_single / steps
    value = total_pts_all / (ms_step / 1e3)
    pairs_per_s = world * scene.n_pairs / (ms_step / 1e3)

    # ---- per-kernel timing (after the timed region; CUDA events around each kernel on the launch stream)
    import ctypes as C
    set_reserve([0] * DEPTH)
    eng.lib.ldp_profile_enable(1)
    n_prof = 20
    buf = (C.c_float * 64)()
    kdict = {}
    for i in range(n_prof):
        eng.densify(batches[0], cfg, descs_dev=descs[0], outputs=outs[0])
        n = eng.lib.ldp_profile_read(buf, 64)
        for k in range(n):                       # kernels of all sub-batches, summed by name
            name = eng.lib.ldp_profile_name(k).decode()
            kdict[name] = kdict.get(name, 0.0) + float(buf[k]) / n_prof
    eng.lib.ldp_profile_enable(0)
    _dbg("per-kernel profile done")
    dom = "ldp_front_kernel" if "ldp_front_kernel" in kdict else "ldp_stream_kernel"
    peak, peak_src = measured_hbm_peak()
    k1_bytes = R * nn * H * W * 4                     # every certainty value read exactly once
    # The dominant kernel's average launch duration: `reps` back-to-back launches of that kernel alone between two CUDA
    # events on the launch stream (193 MB of inputs per launch, larger than L2).  Bracketing each launch inside the step
    # with its own event pair (kernels_ms above) adds ~4 us of event latency per kernel; that figure is reported too.
    params = eng._params(batches[0], cfg, False, 0, 0)
    ws_t = eng._ensure_workspace(params)
    cur = torch.cuda.current_stream(dev).cuda_stream

    def stream_only(reps):
        rc = eng.lib.ldp_debug_launch_stream(C.byref(params), C.c_void_p(descs[0].data_ptr()), C.c_void_p(ws_t.data_ptr()),
                                             C.c_size_t(ws_t.numel()), C.c_void_p(cur), C.c_int(reps))
        if rc != 0:
            raise RuntimeError(f"ldp_debug_launch_stream failed: {rc}")
    stream_only(5)
    torch.cuda.synchronize(dev)
    k_ev0, k_ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k_reps = 50
    k_ev0.record()
    stream_only(k_reps)
    k_ev1.record()
    torch.cuda.synchronize(dev)
    dom_ms = k_ev0.elapsed_time(k_ev1) / k_reps
    achieved = k1_bytes / (dom_ms * 1e-3) / 1e9
    K_pts = total_pts
    path_bytes = R * nn * H * W * 4 + S_total * 28 + K_pts * 28          # SURVEY 8d: B_ref summed over the views
    path_gbs = path_bytes / (ms_step * 1e-3) / 1e9
    path_gbs_single = path_bytes / (ms_single_step * 1e-3) / 1e9
    # every kernel of the step against the same peak, on the bytes it has to move (what each is bound by: DESIGN.md 4)
    nominal = {
        "ldp_front_kernel": (k1_bytes, "nn*H*W*4: every certainty value once (workspace writes, 5 B/px, not counted)"),
        "ldp_stream_kernel": (k1_bytes, "nn*H*W*4: every certainty value once"),
        "ldp_prep_kernel": (R * H * W * 8, "H*W*8: weights in, probabilities out (L2)"),
        "ldp_draw_kernel": (R * int(WORKLOAD["M"] * 0.85) * 136, "draws * (128-byte chunk line + 8-byte chunk sum), L2"),
        "ldp_resume_kernel": (R * (H * W // 8 + (S_total // max(R, 1)) * 4), "selection bitmap + sorted indices out, L2"),
        "ldp_geometry_kernel": (S_total * (16 + 12 + 1) + S_total * 33, "per sample: warp row 16 B + 4 texels 12 B + winner 1 B in, 33 B out"),
        "ldp_fix_kernel": (0, "worklist of non-converged samples (normally empty)"),
        "ldp_pack_kernel": (S_total * 33 + K_pts * 28, "per sample 33 B in, per kept point 28 B out"),
    }
    by_kernel = {}
    for name, ms_k in kdict.items():
        nb, what = nominal.get(name, (0, ""))
        by_kernel[name] = {"us_in_step_event_bracketed": 1e3 * ms_k, "bytes": int(nb), "what": what,
                           "frac": (nb / (ms_k * 1e-3) / 1e9 / peak) if ms_k > 0 else None}

    if snap is not None:
        write_outputs(args.dump_outputs, snap)

    if args.quick:
        if rank == 0:
            emit({"quick": True, "ms_per_step": ms_step, "ms_per_step_one_launch_at_a_time": ms_single_step,
                  "kernels_ms": kdict, "front_kernel_alone_ms": dom_ms, "per_rank": per_rank_ms,
                  "k1_frac": achieved / peak, "path_frac": path_gbs / peak, "path_frac_one_at_a_time": path_gbs_single / peak})
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    _dbg("stream-only timing done")

    # ---- BASELINE config 5 (sharded scene + final point all-gather)
    c5 = None
    if not args.no_config5:
        c5 = config5_block(args, dev, rank, world, ring)
        _dbg("config5 done")

    # ---- the drop-in entry point (rank 0 only: it is a per-process host path)
    api = None
    if rank == 0 and not args.no_api:
        api = api_block(args, dev, scene, slots[0], WORKLOAD["M"])
        _dbg("api block done")

    # ---- e2e through the public API from host buffers.  The views are handed over in E2E_CHUNKS groups: the pinned
    #      host->device copy of group g+1 (copy stream) overlaps the kernels of group g, whose warp rows are gathered
    #      straight from pinned host memory over PCIe (the 0.77 GB of warp planes are never uploaded).
    cert, warp, image = slots[0].cert, slots[0].warp, slots[0].image
    E2E_CHUNKS = int(os.environ.get("BENCH_E2E_CHUNKS", "4")) if R >= 8 else 1
    h_cert = cert.cpu().pin_memory()
    h_img = image.cpu().pin_memory()
    h_warp = warp.cpu().pin_memory()
    # Two sets of device buffers: the upload of step i + 1 starts the moment step i's upload ends (the link never idles between
    # steps), while step i's last kernels and its read-back are still running; every step's own H2D copies, kernels and D2H
    # read are inside the timed region, its result is read one step later (and the last one before the clock stops).
    SETS = 2
    d_cert = [torch.empty_like(cert) for _ in range(SETS)]
    d_img = [torch.empty_like(image) for _ in range(SETS)]
    bounds = [(R * g // E2E_CHUNKS, R * (g + 1) // E2E_CHUNKS) for g in range(E2E_CHUNKS)]
    e2e_batches = [[slots[0].batch(eng, scene, lo, hi, stream_base=data_rank * R, cert=d_cert[q], warp=h_warp, image=d_img[q])
                    for lo, hi in bounds] for q in range(SETS)]
    e2e_descs = [[eng.upload_descs(b) for b in e2e_batches[q]] for q in range(SETS)]
    e2e_outs = [[eng.alloc_outputs(hi - lo, sel_cap) for lo, hi in bounds] for q in range(SETS)]
    copy_stream = torch.cuda.Stream(dev)
    back_stream = torch.cuda.Stream(dev)
    copied = [[torch.cuda.Event() for _ in bounds] for _ in range(SETS)]
    computed = [[torch.cuda.Event() for _ in bounds] for _ in range(SETS)]
    read_back = [torch.cuda.Event() for _ in range(SETS)]
    # a group's whole packed result (offsets | xyz | rgb | err, padded to capacity) goes back in ONE device->host copy on
    # a third stream as soon as the group is done: no intermediate synchronisation to learn the counts first, and the
    # copy runs in the other PCIe direction while the next groups are still being uploaded
    h_packed = [[torch.empty_like(o.packed, device="cpu").pin_memory() for o in e2e_outs[q]] for q in range(SETS)]

    def e2e_submit(q):
        """enqueue one step on buffer set q: uploads, launches, read-back; no host synchronisation"""
        main = torch.cuda.current_stream(dev)
        copy_stream.wait_event(computed[q][-1])          # the set's previous user has read its inputs (no-op the first time)
        with torch.cuda.stream(copy_stream):
            for g, (lo, hi) in enumerate(bounds):
                d_cert[q][lo:hi].copy_(h_cert[lo:hi], non_blocking=True)
                d_img[q][lo:hi].copy_(h_img[lo:hi], non_blocking=True)
                copied[q][g].record(copy_stream)
        back_stream.wait_event(read_back[q])             # ... and its results have left (host buffers of the set are reused)
        for g in range(E2E_CHUNKS):
            main.wait_event(copied[q][g])
            eng.densify(e2e_batches[q][g], cfg, descs_dev=e2e_descs[q][g], outputs=e2e_outs[q][g])
            computed[q][g].record(main)
            with torch.cuda.stream(back_stream):
                back_stream.wait_event(computed[q][g])
                h_packed[q][g].copy_(e2e_outs[q][g].packed, non_blocking=True)
        read_back[q].record(back_stream)

    def e2e_finish(q):
        """the result the caller reads: per-group offsets from the host copy of set q"""
        read_back[q].synchronize()
        n = 0
        for g, (lo, hi) in enumerate(bounds):
            n += int(h_packed[q][g][:8 * (hi - lo + 1)].view(torch.int64)[-1])
        return n

    def e2e_run(n_steps):
        n = 0
        e2e_submit(0)
        for i in range(1, n_steps):
            e2e_submit(i % SETS)
            n = e2e_finish((i - 1) % SETS)
        n = e2e_finish((n_steps - 1) % SETS)
        return n

    _dbg("e2e setup done")
    e2e_steps = max(3, min(steps, 20))
    n_e2e = e2e_run(3)
    torch.cuda.synchronize(dev)
    barrier()
    t0 = time.perf_counter()
    n_e2e = e2e_run(e2e_steps)
    torch.cuda.synchronize(dev)
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    if world > 1:
        t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_outs_flat = e2e_outs[0]
    S_e2e = int(sum(int(o.n_samples.sum().item()) for o in e2e_outs_flat))
    e2e = {"value": world * n_e2e / e2e_s, "unit": UNIT,
           "h2d_bytes_per_step": int(h_cert.numel() * 4 + h_img.numel() + S_e2e * 16),
           "d2h_bytes_per_step": int(sum(h.numel() for h in h_packed[0])), "ms_per_step": 1e3 * e2e_s,
           "note": f"cert planes + ref images copied H2D from pinned memory in {E2E_CHUNKS} groups of views, the copy of a "
                   "group overlapping the kernels of the previous one; warp planes stay pinned on the host and only the "
                   "sampled rows (16 B each) are gathered over PCIe; each group's packed result (offsets, xyz, rgb, err, padded to "
                   "capacity) is copied D2H on a third stream as soon as the group is done; two sets of device buffers: a step's "
                   "upload starts when the previous step's upload ends, its result is read on the host one step later (every "
                   "step's H2D, kernels, D2H and host read are inside the timed region)"}

    # the second roofline of the path: it executes ~78 M warp instructions per step (f64 cdf arithmetic, exact comparisons,
    # per-sample eigenvectors), which bounds it by instruction issue well before HBM: 148 SMs x 4 schedulers x SM clock
    n_inst, inst_note = recorded_instructions()
    issue_roofline = None
    if n_inst:
        sm_clock = (clocks.get("sm_max_mhz") or 1965.0) * 1e6
        n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
        peak_issue = n_sm * 4 * sm_clock
        issue_roofline = {"bound": "instruction issue", "warp_instructions_per_step": n_inst, "peak_warp_instructions_per_s": peak_issue,
                          "floor_ms_per_step": 1e3 * n_inst / peak_issue, "frac": n_inst / (ms_step * 1e-3) / peak_issue,
                          "frac_one_launch_at_a_time": n_inst / (ms_single_step * 1e-3) / peak_issue, "source": inst_note}
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 geometry / f64 cdf, sampson, colour", "data": "synthetic",
            "config": {"workload": WORKLOAD["name"], "refs_per_gpu": R, "pairs_per_gpu": scene.n_pairs,
                       "l2_policy": "inputs larger than L2 (0.97 GB per step vs 126 MB); every step in flight has its own input tensors",
                       "steps_in_flight": DEPTH,
                       "per_gpu_work": ("every rank processes the same synthetic batches (same seeds): identical work per GPU"
                                        if not int(os.environ.get("BENCH_DATA_PER_RANK", "0")) else "batches seeded by rank (their cost differs by up to 6 %)"),
                       "rng": "philox4x32-10", "multi_gpu": ("views sharded, points stay on their rank, no collective per step; the "
                                      "ranks' kept-point counts (global row offsets) are exchanged once after the last step, inside "
                                      "the timed region" if world > 1 else "none")},
            "pairs_per_sec": pairs_per_s, "points_per_step": total_pts_all, "samples_per_step": S_all,
            "ms_per_step_one_launch_at_a_time": ms_single_step,
            "per_rank": per_rank_ms,          # every rank's own device-timed figures (value uses the maximum)
            "gpu_launches": launches_per_step * steps,
            "kernels_ms": kdict,
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": recorded_traffic(), "peak_source": peak_src,
                         "kernel_ms": dom_ms, "kernel_ms_in_step_event_bracketed": kdict[dom],
                         "timing": f"{k_reps} back-to-back launches of the kernel alone between two CUDA events",
                         "algorithmic_bytes_per_launch": k1_bytes,
                         "by_kernel": by_kernel,
                         "path_achieved": path_gbs, "path_frac": path_gbs / peak,
                         "path_frac_one_launch_at_a_time": path_gbs_single / peak,
                         "path_algorithmic_bytes_per_step": path_bytes,
                         "path_note": "per GPU: SURVEY 8d bytes of one step (nn*H*W*4 + S*28 + K*28 per view) / ms_per_step / peak",
                         "issue": issue_roofline},
            "e2e": e2e, "clocks": clocks,
        }
        if c5 is not None:
            line["config5"] = c5
        if api is not None:
            line["api"] = api
        if cpu_base is not None:
            line["cpu_baseline"] = cpu_base
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="default: 1000 (GPU arm), 20 (--impl reference)")
    ap.add_argument("--warmup", type=int, default=None, help="default: 10 (GPU arm), 3 (--impl reference)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config5", action="store_true")
    ap.add_argument("--no-api", action="store_true")
    ap.add_argument("--quick", action="store_true", help="profiling runs: skip cpu baseline, clock-load loop, config5, api and e2e")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (kept points and per-view offsets, status, sample counts) "
                         "as DIR/<name>.npy, float32 / float64, at most 64 MB; the inputs depend only on the arguments")
    args = ap.parse_args()
    if args.impl == "reference":
        reference_arm(args)
    else:
        gpu_arm(args)


if __name__ == "__main__":
    main()
