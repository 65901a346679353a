"""Development aid: prints the precision of the tensor-core paths (forward max-abs error vs the oracle, per-tensor
gradient cosines vs float64 autograd and vs the reference fixtures).  Run on a GPU box:  python tools/parity_diag.py"""
import os
import random
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "golden")]
import helpers  # noqa: E402
import synth  # noqa: E402
from oracle import c_oracle  # noqa: E402
from neural_raytracing_b200 import config, ops  # noqa: E402
import test_gpu_tc_train as T  # noqa: E402


def t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def forward_errors():
    cases = dict(helpers.MLP_CASES)
    cases["nerf_second_le"] = (T.LE_KW, None)
    for name in ("nerf_first", "nerf_second", "nerf_second_le", "neural_bsdf"):
        kw = cases[name][0]
        w = synth.mlp_weights(**kw)
        for scale in (0.1, 0.6, 2.0):
            x = (scale * np.random.RandomState(7).standard_normal((5000, kw["in_size"]))).astype(np.float32)
            yo = c_oracle.mlp_forward(helpers.oracle_mlp(w), x)
            m = helpers.cuda_mlp(w)
            e = {p: float(np.abs(ops.mlp_forward(m, t(x), prec=p).cpu().numpy() - yo).max()) for p in ("f16", "bf16")}
            print("fwd %-15s |x|~%.1f  f16 %.2e  bf16 %.2e" % (name, scale, e["f16"], e["bf16"]), flush=True)


def grad_cosines():
    for name, sig, need_x in (("nerf_first", False, False), ("nerf_second", True, True), ("nerf_second_le", True, True)):
        kw = T.LE_KW if name == "nerf_second_le" else helpers.MLP_CASES[name][0]
        w = synth.mlp_weights(**kw)
        m = helpers.cuda_mlp(w)
        M = 5000
        out_act = ops.OUT_SIGMOID if sig else ops.OUT_NONE
        g = torch.Generator(device="cuda").manual_seed(M + 5)
        x = (0.6 if name == "nerf_first" else 0.1) * torch.randn(M, kw["in_size"], device="cuda", generator=g)
        gy = torch.randn(M, kw["out"], device="cuda", generator=g) * 3e-4
        for prec in ("f16", "bf16"):
            out, ws = ops.mlp_forward_train_tc(m, x, out_act, prec=prec)
            gp, gx = ops.mlp_backward_tc(m, M, out, gy, ws, out_act, need_input_grad=need_x, prec=prec)
            gW, gb = m.unpack(gp)
            for quantised in (True, False):
                y, xr, Ws, bs = T._ref(w, x, sig, quantised, split_inputs=kw["in_size"] <= 5)
                (y * gy.double()).sum().backward()
                cw = [T._cos(a, r.grad) for a, r in zip(gW, Ws)]
                cb = [T._cos(a, r.grad) for a, r in zip(gb, bs)]
                cx = T._cos(gx, xr.grad) if need_x else float("nan")
                print("grad %-15s %-4s %s  fwd %.1e  minW %.5f minB %.5f gx %.5f  W: %s" % (
                    name, prec, "quant" if quantised else "exact", float((out.double() - y.detach()).abs().max()), min(cw), min(cb), cx,
                    " ".join("%.4f" % c for c in cw)), flush=True)


def fixture_cosines():
    from neural_raytracing_b200.pathtracer.lights import PointLights
    from neural_raytracing_b200.pathtracer.shapes.nerf import NeRFLE
    g = helpers.golden("nerfle_train")
    for envmap in (False, True):
        tag = "le" if envmap else "pt"
        random.random = lambda: float(g["fixed_random"])
        n = NeRFLE(envmap=envmap, device="cuda")
        w1, w2 = helpers.nerfle_weights(envmap)
        for mod, w in ((n.first, w1), (n.second, w2)):
            mod.basis_p = torch.from_numpy(w["basis"]).cuda()
            for lin, W, b in zip([mod.init] + list(mod.layers) + [mod.out], w["W"], w["b"]):
                with torch.no_grad():
                    lin.weight.copy_(torch.from_numpy(W)); lin.bias.copy_(torch.from_numpy(b))
        rays = torch.from_numpy(g[tag + "_rays"]).cuda()
        lights = PointLights(device="cuda", location=torch.from_numpy(g[tag + "_light_loc"]).cuda(), scale=10)
        target = torch.full(tuple(rays.shape[:-1]) + (3,), 0.5, device="cuda")
        for tprec in ("f32", "f16", "bf16"):
            n.zero_grad()
            try:
                config.set_train_precision(tprec)
                loss = torch.nn.functional.mse_loss(n(rays, lights), target)
                loss.backward()
            finally:
                config.set_train_precision("f32")
            msg = []
            for name, mod in (("first", n.first), ("second", n.second)):
                lins = [mod.init] + list(mod.layers) + [mod.out]
                for kind in ("w", "b"):
                    ref_all = synth.unpack_grad(g, "%s_g_%s_%s" % (tag, name, kind))
                    got_all = torch.cat([(l.weight if kind == "w" else l.bias).grad.reshape(-1) for l in lins]).cpu().numpy().astype(np.float64)
                    cos = float(got_all @ ref_all / (np.linalg.norm(got_all) * np.linalg.norm(ref_all)))
                    # per tensor
                    off, per = 0, []
                    for l in lins:
                        k = (l.weight if kind == "w" else l.bias).numel()
                        a, b = got_all[off:off + k], ref_all[off:off + k]
                        per.append(float(a @ b / (np.linalg.norm(a) * np.linalg.norm(b) + 1e-300)))
                        off += k
                    msg.append("%s.%s all %.5f per-tensor [%s]" % (name, kind, cos, " ".join("%.4f" % c for c in per)))
            print("fixture %s %-4s loss %.6f (ref %.6f)  %s" % (tag, tprec, float(loss.detach()), float(g[tag + "_loss"]), " | ".join(msg)), flush=True)


if __name__ == "__main__":
    forward_errors()
    grad_cosines()
    fixture_cosines()
