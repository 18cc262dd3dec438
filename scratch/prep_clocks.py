"""Dev tool: globaltimer phase stamps of the lean prep kernel (CTAs 3 and 31 of every view)."""
import os, sys, ctypes as C
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
for _ in range(4):
    out = eng.densify(batch, cfg)
torch.cuda.synchronize()
params = eng._params(batch, cfg, False, 0, 0)
host = (C.c_longlong * (len(batch) * 32))()
eng.lib.ldp_debug_read_clocks(C.byref(params), C.c_void_p(eng._workspace.data_ptr()), host)
clk = np.array(host[:]).reshape(len(batch), 32)
t0 = clk[:, 16].min()
names = ["start", "s reduced+bins zeroed", "main loop done", "reductions done", "flushed", "-"]
for base, label in ((16, "CTA 3"), (24, "CTA 31")):
    c = clk[:, base:base + 6] - t0
    print(label, "start times (ns) by view:", np.sort(c[:, 0])[::5])
    for k in range(4):
        d = c[:, k + 1] - c[:, k]
        print(f"  {names[k]:>20} -> {names[k+1]:<20} median {np.median(d):7.0f} ns  max {d.max():7.0f}")
    print("  CTA lifetime median", np.median(c[:, 4] - c[:, 0]), "ns; last end", c[:, 4].max(), "ns")
