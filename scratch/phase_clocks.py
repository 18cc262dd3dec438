"""Dev tool: build with -DLDP_PHASE_CLOCKS, run the bench workload once, print per-phase SM-clock deltas of the draw kernel."""
import os, sys, subprocess, ctypes as C
sys.path.insert(0, "/root/repo")
import numpy as np, torch
from lichtfeld_densification_plugin_b200 import build as B
B.NVCC_FLAGS.append("-DLDP_PHASE_CLOCKS")
B.build(force=True)
from lichtfeld_densification_plugin_b200 import synth
from lichtfeld_densification_plugin_b200.engine import DensifyEngine, PathConfig
dev = torch.device("cuda", 0)
scene = synth.make_scene(185, "fast", 0.25, 4)
eng = DensifyEngine(dev)
batch = eng.new_batch(scene.H, scene.W, scene.w_match, scene.h_match)
keep = []
for rp in range(scene.n_refs):
    inp = synth.synth_ref_inputs(scene, rp, device=dev, cert_family="R", seed=100)
    keep.append(inp)
    nn = len(inp["nbr_indices"])
    batch.add([inp["cert"][k] for k in range(nn)], [inp["warp"][k] for k in range(nn)], inp["image"], scene.cameras[inp["ref_index"]],
              [scene.cameras[j] for j in inp["nbr_indices"]], rng_stream=rp)
cfg = PathConfig(matches_per_ref=10000)
for _ in range(3):
    out = eng.densify(batch, cfg)
torch.cuda.synchronize()
params = eng._params(batch, cfg, False, 0, 0)
host = (C.c_longlong * (len(batch) * 32))()
rc = eng.lib.ldp_debug_read_clocks(C.byref(params), C.c_void_p(eng._workspace.data_ptr()), host)
clk = np.array(host[:]).reshape(len(batch), 32)
print("cluster size used:", eng.lib.ldp_debug_last_cluster())
names = {0: "start", 1: "init done", 11: "csum copied", 12: "copy synced", 14: "csum loaded+local", 15: "block scan done", 16: "prefix stored+sync", 17: "after B0", 3: "guide built", 4: "draws 1 done", 6: "after B1", 7: "zeroed", 8: "rounds done", 9: "coverage done", 10: "compaction done"}
order = [0, 1, 11, 12, 14, 15, 16, 17, 3, 4, 6, 7, 8, 9, 10]
for a, b in zip(order[:-1], order[1:]):
    dd = clk[:, b] - clk[:, a]
    print(f"{names[a]:>20} -> {names[b]:<20} median {np.median(dd):9.0f}  max {dd.max():9.0f} cycles")
#print("thread0 first pass: searches", np.median(clk[:,11]-clk[:,3]), " scans", np.median(clk[:,12]-clk[:,11]), " atomics issue", np.median(clk[:,13]-clk[:,12]), " rest of round", np.median(clk[:,4]-clk[:,13]))
print("total median", np.median(clk[:, 10] - clk[:, 0]), "max", (clk[:, 10] - clk[:, 0]).max(), "cycles @1.963 GHz")
print("---- resume kernel (rounds 2..): cycles")
seq = [(0, "start"), (1, "round-1 finds zeroed"), (20, "round 2 top"), (2, "table rebuilt + B2"), (11, "r2 uniforms+guide"), (12, "r2 binary search"), (14, "r2 exact chunk"), (15, "r2 scans"), (16, "r2 exact crossing"), (21, "round 2 draws done"), (22, "round 3 top"), (23, "round 3 draws done"), (24, "round 4 top"), (25, "round 4 draws done"), (8, "rounds done"), (9, "coverage done"), (28, "bitmap loaded+popc"), (29, "block scan"), (30, "bits extracted+sync"), (10, "compaction done")]
for (a, na), (b, nb_) in zip(seq[:-1], seq[1:]):
    dd = clk[:, b] - clk[:, a]
    ok = (clk[:, b] > 0) & (clk[:, a] > 0) & (dd > 0) & (dd < 10**7)
    if ok.sum(): print(f"{na:>24} -> {nb_:<24} median {np.median(dd[ok]):9.0f}  max {dd[ok].max():9.0f}  (n={ok.sum()})")
sys.exit(0)
d = clk[:, 1:11] - clk[:, 0:10]
print("rounds per view:", clk[:, 20][:12], "...")
for i in range(10):
    print(f"{names[i]:>16} -> {names[i+1]:<16} median {np.median(d[:, i]):9.0f}  max {d[:, i].max():9.0f} cycles")
#print("thread0 first pass: searches", np.median(clk[:,11]-clk[:,3]), " scans", np.median(clk[:,12]-clk[:,11]), " atomics issue", np.median(clk[:,13]-clk[:,12]), " rest of round", np.median(clk[:,4]-clk[:,13]))
print("total median", np.median(clk[:, 10] - clk[:, 0]), "max", (clk[:, 10] - clk[:, 0]).max())
print("span over all views (first start .. last end):", clk[:, 10].max() - clk[:, 0].min())
