import sys, ctypes as C
sys.path.insert(0, "/root/repo")
import numpy as np, torch
from lichtfeld_densification_plugin_b200 import build as B
B.NVCC_FLAGS.append("-DLDP_PHASE_CLOCKS"); B.build(force=True)
from lichtfeld_densification_plugin_b200 import synth
from lichtfeld_densification_plugin_b200.engine import DensifyEngine, PathConfig
dev = torch.device("cuda", 0)
FAM = sys.argv[1] if len(sys.argv) > 1 else "R"
scene = synth.make_scene(40, "fast", 0.8, 8)
eng = DensifyEngine(dev); b = eng.new_batch(scene.H, scene.W, scene.w_match, scene.h_match); keep = []
for rp in range(scene.n_refs):
    inp = synth.synth_ref_inputs(scene, rp, device=dev, cert_family=FAM, seed=100); keep.append(inp); k = len(inp["nbr_indices"])
    b.add([inp["cert"][q] for q in range(k)], [inp["warp"][q] for q in range(k)], inp["image"], scene.cameras[inp["ref_index"]], [scene.cameras[j] for j in inp["nbr_indices"]], rng_stream=rp)
cfg = PathConfig(matches_per_ref=10000, no_filter=True)
for _ in range(3): out = eng.densify(b, cfg)
torch.cuda.synchronize()
params = eng._params(b, cfg, False, 0, 0)
host = (C.c_longlong * (len(b) * 32))()
eng.lib.ldp_debug_read_clocks(C.byref(params), C.c_void_p(eng._workspace.data_ptr()), host)
clk = np.array(host[:]).reshape(len(b), 32)
for a, bb, nm in ((0, 1, "cap count (+ radix select)"), (1, 2, "tie rows"), (2, 3, "gather / ordered emit"), (3, 4, "sort"),):
    print(f"{nm:28s} median {np.median(clk[:, bb] - clk[:, a]):10.0f} cycles")
