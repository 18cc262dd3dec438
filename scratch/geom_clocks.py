"""Dev tool: build with -DLDP_GEOM_CLOCKS, run the bench workload, print the geometry kernel's warp-cycles per phase (summed over warps)."""
import os, sys, ctypes as C
sys.path.insert(0, "/root/repo")
import numpy as np, torch
from lichtfeld_densification_plugin_b200 import build as B
B.NVCC_FLAGS.append("-DLDP_GEOM_CLOCKS")
for f in sys.argv[1:]:
    B.NVCC_FLAGS.append(f)
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
NRUN = 3
out = eng.densify(batch, cfg)
torch.cuda.synchronize()
eng._workspace.zero_()
for _ in range(NRUN):
    out = eng.densify(batch, cfg)
torch.cuda.synchronize()
params = eng._params(batch, cfg, False, 0, 0)
host = (C.c_longlong * (len(batch) * 32))()
rc = eng.lib.ldp_debug_read_clocks(C.byref(params), C.c_void_p(eng._workspace.data_ptr()), host)
clk = np.array(host[:], dtype=np.float64).reshape(len(batch), 32)[:, :36 if False else 32]
names = {0: "stage constants", 10: "grid dependency sync", 1: "idx, S, barrier", 2: "gather (k, warp row, texels)", 3: "coords, Sampson, colour", 4: "DLT rows",
         5: "null vector", 6: "reproject, filters", 7: "store", 8: "tile statistics", 9: "final barrier"}
for which, bx in enumerate((5, 40)):
    c = clk[:, which * 12: which * 12 + 12]
    print("---- CTA", bx, "of every view: warp 0, cycles (median / mean / max over the", len(batch), "views)")
    for k in [0, 10, 1, 2, 3, 4, 5, 6, 7, 8, 9]:
        print(f"{names[k]:>32}: {np.median(c[:, k]):8.0f} {c[:, k].mean():8.0f} {c[:, k].max():8.0f}")
    print(f"{'total':>32}: {np.median(c.sum(1)):8.0f} {c.sum(1).mean():8.0f} {c.sum(1).max():8.0f}")
