"""CPU tests (-m "not gpu") of NeRFLE's opt-in hierarchical sampling (pathtracer/shapes/nerf.py: HierarchicalSampling,
NeRFLE.sampling): validation of the sampling description, fake-tensor shapes of the two operators it adds
(torch.ops.nrt_b200.nerfle_sample_hierarchical and composite_ts), and that the attribute changes neither the
state_dict nor the loading of models pickled before it existed."""
import os
import pickle
import random
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

from neural_raytracing_b200 import ops, torch_ops  # noqa: E402,F401
from neural_raytracing_b200.pathtracer.shapes.nerf import HierarchicalSampling, NeRFLE  # noqa: E402


def test_defaults_are_baseline_config_2():
    s = HierarchicalSampling()
    assert (s.n_coarse, s.n_fine, s.t_near, s.t_far, s.jitter) == (64, 128, 0.0, 2.05, True)
    assert s.n_samples == 192 and s.render_seed != 0 and s.seed is None
    assert HierarchicalSampling(jitter=False).render_seed == 0
    assert HierarchicalSampling(n_coarse=1, n_fine=0).n_samples == 1      # a single stratified pass needs no interior bins


@pytest.mark.parametrize("kw,msg", [
    (dict(n_coarse=2, n_fine=8), "n_coarse must be >= 3 when n_fine > 0"),
    (dict(t_near=1.0, t_far=1.0), "t_far (1) must be greater than t_near (1)"),
    (dict(t_near=2.0, t_far=0.5), "must be greater than t_near"),
    (dict(n_coarse=192, n_fine=384), "n_coarse + n_fine = 576 exceeds 512"),
    (dict(n_coarse=0, n_fine=0), "n_coarse must be >= 1"),
    (dict(n_coarse=3, n_fine=61), "n_coarse = 3 must divide 64 or be a multiple of 64"),
    (dict(n_coarse=64, n_fine=96), "n_fine = 96 must divide 64 or be a multiple of 64"),
])
def test_validation_messages(kw, msg):
    with pytest.raises(ValueError) as e:
        HierarchicalSampling(**kw)
    assert msg in str(e.value)


def test_largest_accepted_sample_count():
    assert HierarchicalSampling(n_coarse=128, n_fine=384).n_samples == ops.N.MAX_HIER_SAMPLES == 512


def test_fake_shapes_of_the_new_operators():
    from torch._subclasses.fake_tensor import FakeTensorMode
    a1, a2 = [3, 0, 16, 128, 5, 3, 65, 0], [70, 0, 16, 64, 8, 3, 3, 0]
    np1 = sum(k * n + n for k, n in ops.mlp_layer_dims(*a1[:7]))
    np2 = sum(k * n + n for k, n in ops.mlp_layer_dims(*a2[:7]))
    with FakeTensorMode():
        rays = torch.empty(2, 7, 5, 1, 6, device="cuda")
        ts = torch.ops.nrt_b200.nerfle_sample_hierarchical(
            rays, torch.empty(2, 3, device="cuda"), torch.empty(70, dtype=torch.int32, device="cuda"),
            torch.empty(np1, device="cuda"), torch.empty(3, 16, device="cuda"), a1, torch.empty(np2, device="cuda"),
            torch.empty(70, 16, device="cuda"), a2, ops.PREC_F16, 64, 128, 0.0, 2.05, 0,
            torch.empty(1, dtype=torch.int64, device="cuda"))
        assert tuple(ts.shape) == (192, 70)
        sig, rgb = torch.empty(192, 70, device="cuda"), torch.empty(192, 70, 3, device="cuda")
        assert tuple(torch.ops.nrt_b200.composite_ts(sig, rgb, ts).shape) == (70, 3)
        gs, gc = torch.ops.nrt_b200.composite_ts_backward(sig, rgb, ts, torch.empty(70, 3, device="cuda"))
        assert tuple(gs.shape) == (192, 70) and tuple(gc.shape) == (192, 70, 3)


def test_sampling_is_not_state_and_pickles():
    plain, n = NeRFLE(device="cpu"), NeRFLE(device="cpu")
    assert n.sampling is None
    n.sampling = HierarchicalSampling(n_coarse=32, n_fine=64, t_near=0.1, t_far=3.0, jitter=False)
    assert list(n.state_dict()) == list(plain.state_dict())
    m = pickle.loads(pickle.dumps(n))
    s = m.sampling
    assert isinstance(s, HierarchicalSampling)
    assert (s.n_coarse, s.n_fine, s.t_near, s.t_far, s.jitter, s.render_seed) == (32, 64, 0.1, 3.0, False, 0)


def test_model_pickled_before_the_attribute_existed_behaves_as_none():
    from neural_raytracing_b200.pathtracer.lights import PointLights
    torch.manual_seed(0)
    n = NeRFLE(device="cpu")
    del n.__dict__["sampling"]          # what unpickling a model saved before `sampling` existed yields
    old = pickle.loads(pickle.dumps(n))
    assert "sampling" not in old.__dict__ and getattr(old, "sampling", None) is None
    new = pickle.loads(pickle.dumps(old))
    new.sampling = None
    rays = torch.randn(1, 3, 2, 1, 6)
    lights = PointLights(device="cpu", location=torch.randn(1, 3), scale=10)
    real_random = random.random
    try:
        random.random = lambda: 0.25
        a, b = old(rays, lights), new(rays, lights)
    finally:
        random.random = real_random
    assert tuple(a.shape) == (1, 3, 2, 1, 3) and torch.equal(a, b)


def test_sampling_on_cpu_rays_fails_loudly():
    """The hierarchical sampling has no CPU implementation: a CPU NeRFLE with `sampling` set raises a clear error
    instead of falling back to the reference's sampling."""
    from neural_raytracing_b200.pathtracer.lights import PointLights
    n = NeRFLE(device="cpu")
    n.sampling = HierarchicalSampling()
    lights = PointLights(device="cpu", location=torch.randn(1, 3), scale=10)
    for grad in (False, True):
        with torch.set_grad_enabled(grad), pytest.raises(ops.NrtError) as e:
            n(torch.randn(1, 2, 2, 1, 6), lights)
        assert "CUDA kernels only" in str(e.value)
