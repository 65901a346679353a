"""Development: clock64 timeline of CTA 0 of the NeRFLE.second kernel with its real IO policy (IoNerfSecond) inside
nerfle_render (the first kernel's stamps are overwritten by the second's; slots 0 and 1 only).

--first: the NeRFLE.first kernel instead (only its launches stamp, nrtdbg_set_timeline_tag), in the fine pass of a
64 + 128 hierarchical frame (per-ray ts written by k_sample_pdf just before).  Needs a library built with
NRT_EXTRA_NVCC_FLAGS=-DNRT_DBG_BOUNDARY (csrc/tc_core.cuh), which stamps the tile boundary into row 0: output `done` seen,
outputs stored, inputs in registers, encoding stored, `ready` arrived for the next tile's init layer.  Prints the cycles
from a tile's output `done` to the next tile's init `ready`, per slot, against the cycles per tile.

--second: the same boundary of the NeRFLE.second kernel (only its launches stamp) in the same hierarchical frame: stage 9's
(the last hidden layer's) `done` seen, rgb stored, the next tile's direction / light code in registers, its encoding
stored, `ready` arrived for its init layer.  Same NRT_DBG_BOUNDARY build."""
import ctypes, sys, os
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests")); sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import numpy as np, torch
import helpers, synth
from neural_raytracing_b200 import ops, _native as N
FIRST = "--first" in sys.argv
SECOND = "--second" in sys.argv
BOUNDARY = FIRST or SECOND
w1, w2 = helpers.nerfle_weights(False)
m1, m2 = helpers.cuda_mlp(w1), helpers.cuda_mlp(w2)
R = 148 * 3 * 2 * 12
rays = torch.from_numpy(synth.camera_rays(4, R)).cuda()
ts = torch.linspace(0, 2.037, 64, device="cuda")
code = torch.tensor([[0.4, 1.0, 0.3]], device="cuda")
kw = dict(n_coarse=64, n_fine=128, t_near=0.0, t_far=2.037, jitter_seed=3) if BOUNDARY else {}
render = lambda: ops.nerfle_render(m1, m2, rays, None if BOUNDARY else ts, code, prec="f16", **kw)
render(); torch.cuda.synchronize()
STAGES = 8 if FIRST else 11
if BOUNDARY:
    tags = [N.lib().nrt_profile_tag_name(i).decode() for i in range(N.lib().nrt_profile_num_tags())]
    N.lib().nrtdbg_set_timeline_tag(ctypes.c_int(tags.index("mlp_tc_nerf_first" if FIRST else "mlp_tc_nerf_second")))
buf = torch.zeros(4 * STAGES * 2 * 8, dtype=torch.int64, device="cuda")
N.lib().nrtdbg_set_timeline(ctypes.c_void_p(buf.data_ptr()))
render(); torch.cuda.synchronize()
N.lib().nrtdbg_set_timeline(None)
if BOUNDARY:
    N.lib().nrtdbg_set_timeline_tag(ctypes.c_int(-1))
t = buf.cpu().numpy().reshape(4, STAGES, 2, 8)
t0 = t[:, :, :, 1:][t[:, :, :, 1:] > 0].min()
names = ["-", "ready", "committed", "wait_done", "done", "loaded", "stored", "arrived"]
bnames = ["-", "-", "-", "out_done", "out_stored", "inputs", "enc_stored", "init_ready"]
for it in range(1, 3):
    for st in range(STAGES):
        for slot in range(2):
            row = t[it, st, slot]
            nm = bnames if BOUNDARY and st == 0 else names
            print("it%d st%d slot%d " % (it, st, slot) + "  ".join("%s=%6d" % (nm[k], row[k] - t0) if row[k] > 0 else "%s=     -" % nm[k] for k in range(1, 8)))
if BOUNDARY:
    # row 0 of iteration it: out_done / out_stored of tile it; inputs / enc_stored / init_ready of tile it (its init hand-off)
    for slot in range(2):
        per_tile = t[1:, 1, slot, 1] - t[:-1, 1, slot, 1]          # init layer issued, tile to tile
        gap = t[1:, 0, slot, 7] - t[:-1, 0, slot, 3]               # output done of tile it -> init ready of tile it+1
        store = t[:, 0, slot, 4] - t[:, 0, slot, 3]                # output done -> outputs stored
        print("slot %d: cycles per tile %s; output done -> next init ready %s (%.1f %% of a tile); output done -> stored %s"
              % (slot, per_tile.tolist(), gap.tolist(), 100.0 * np.median(gap) / np.median(per_tile), store.tolist()))
else:
    print("cycles per slot iteration:", t[1:, 0, 0, 1] - t[:-1, 0, 0, 1])
