"""Occupancy grid without a GPU: the restatement's formulas on hand-made cases, argument validation, the fake
implementations of the operators, and NeRFLE's state_dict."""
import ctypes
import math

import numpy as np
import pytest
import torch

import occupancy_port as occ
from neural_raytracing_b200 import _native as N
from neural_raytracing_b200 import ops, torch_ops
from neural_raytracing_b200.pathtracer.shapes.nerf import NeRFLE, OccupancyGrid

LO, HI = (-1.0, -1.0, -1.0), (1.0, 1.0, 1.0)


def test_cell_lookup_boundaries_outside_nan():
    res = 16                                            # h = 0.125
    p = np.array([[-1.0, -1.0, -1.0],                   # lowest corner: cell 0
                  [0.0, 0.0, 0.0],                      # a shared corner belongs to the upper cell (floor)
                  [0.9999, 0.9999, 0.9999],             # the last cell
                  [1.0, 0.0, 0.0],                      # on the upper face: outside
                  [-1.0001, 0.0, 0.0],                  # below the box
                  [np.nan, 0.0, 0.0], [np.inf, 0.0, 0.0]], np.float32)
    inside, c = occ.cell_index(p, res, LO, HI)
    assert inside.tolist() == [True, True, True, False, False, False, False]
    assert c[0] == 0 and c[1] == (8 * 16 + 8) * 16 + 8 and c[2] == 16 ** 3 - 1
    assert (c[3:] == -1).all()


def test_keep_mask_outside_and_nonfinite_are_kept():
    res = 16
    words = occ.pack_bits(np.zeros(res ** 3, bool))     # every cell empty
    rays = np.array([[0, 0, 0, 1, 0, 0], [5, 5, 5, 1, 0, 0], [np.nan, 0, 0, 1, 0, 0], [0, 0, 0, np.inf, 0, 0]], np.float32)
    keep = occ.keep_mask(words, res, LO, HI, rays, np.array([0.0, 0.5], np.float32))
    assert keep.tolist() == [[False, False], [True, True], [True, True], [True, True]]
    full = occ.pack_bits(np.ones(res ** 3, bool))
    assert occ.keep_mask(full, res, LO, HI, rays, np.array([0.0, 0.5], np.float32)).all()


def test_bits_pack_roundtrip_and_order():
    rs = np.random.RandomState(3)
    for n in (16 ** 3, 17 ** 3):
        b = rs.rand(n) < 0.3
        w = occ.pack_bits(b)
        assert w.dtype == np.int32 and w.size == ops.occupancy_words(round(n ** (1 / 3)))
        assert np.array_equal(occ.unpack_bits(w, n), b)
    one = np.zeros(64, bool); one[33] = True
    assert occ.pack_bits(one).view(np.uint32).tolist() == [0, 2]


def test_update_rule():
    dens = np.array([0.0, 1.0, 4.0, 0.5], np.float32)
    sig = np.array([[-1.0, -2.0], [0.25, 3.0], [1.0, np.float32(0.5)], [0.005, 0.02]], np.float32)
    d, bits = occ.update_rule(dens, sig, 0.5, 0.01)
    assert d.tolist() == [0.0, 3.0, 2.0, 0.25] and bits.tolist() == [False, True, True, True]
    d0, _ = occ.update_rule(dens, sig, 0.0, 0.01)       # decay 0 rebuilds
    assert d0.tolist() == np.array([0.0, 3.0, 1.0, 0.02], np.float32).tolist()


def test_update_points_lie_in_their_cells():
    res = 16
    for seed, ppc in ((0, 1), (7, 4)):
        p = occ.update_points(res, (-1.5, -0.5, 0.0), (1.5, 2.5, 1.0), ppc, seed)
        inside, c = occ.cell_index(p, res, (-1.5, -0.5, 0.0), (1.5, 2.5, 1.0))
        want = np.repeat(np.arange(res ** 3), ppc)
        ok = inside & (c == want)
        face = occ.near_face(p, res, (-1.5, -0.5, 0.0), (1.5, 2.5, 1.0))
        assert (ok | face).all() and (~ok).sum() <= 1e-4 * p.shape[0]
    a = occ.update_points(res, LO, HI, 2, 5)
    assert np.array_equal(a, occ.update_points(res, LO, HI, 2, 5))
    assert not np.array_equal(a, occ.update_points(res, LO, HI, 2, 6))


@pytest.mark.parametrize("kw, msg", [
    (dict(resolution=15), "resolution"), (dict(resolution=513), "resolution"), (dict(resolution=64.0), "resolution"),
    (dict(bbox_min=(0, 0, 0), bbox_max=(1, 0, 1)), "bbox"), (dict(bbox_min=(0, -math.inf, 0)), "box"),
    (dict(bbox_max=(1, 1, math.nan)), "box"), (dict(bbox_min=(0, 0)), "3 entries"), (dict(threshold=-0.1), "threshold"),
    (dict(threshold=math.nan), "threshold")])
def test_grid_validation(kw, msg):
    with pytest.raises(ValueError, match=msg):
        OccupancyGrid(device="cpu", **kw)


@pytest.mark.parametrize("kw, msg", [(dict(points_per_cell=0), "points_per_cell"), (dict(points_per_cell=2.0), "points_per_cell"),
                                     (dict(decay=-0.1), "decay"), (dict(decay=1.5), "decay"), (dict(seed=-1), "seed"),
                                     (dict(seed=1.5), "seed")])
def test_update_validation(kw, msg):
    g = OccupancyGrid(resolution=16, device="cpu")
    with pytest.raises(ValueError, match=msg):
        g.update(None, **kw)


def test_grid_fields_and_repr():
    g = OccupancyGrid(resolution=20, bbox_min=(-1, -2, -3), bbox_max=(1, 2, 3), threshold=0.5, device="cpu")
    assert g.density.shape == (8000,) and g.density.dtype == torch.float32
    assert g.bits.shape == (250,) and g.bits.dtype == torch.int32
    assert g.occupied_fraction() == 0.0
    assert repr(g) == "OccupancyGrid(resolution=20, bbox_min=(-1.0, -2.0, -3.0), bbox_max=(1.0, 2.0, 3.0), threshold=0.5)"
    with pytest.raises(ops.NrtError, match="never updated"):
        g.check_current(None)


def test_cpu_tensors_raise():
    g = OccupancyGrid(resolution=16, device="cpu")
    with pytest.raises(ops.NrtError, match="CUDA"):
        ops.occupancy_struct(g.res, g.bbox_min, g.bbox_max, g.bits)
    with pytest.raises(ops.NrtError, match="CUDA"):
        ops.occupancy_mask(g, torch.zeros(4, 6), torch.zeros(8))


def test_library_validates_descriptors():
    L = N.lib()
    bad = [N.NrtOccupancy(15, (ctypes.c_float * 3)(*LO), (ctypes.c_float * 3)(*HI), None),
           N.NrtOccupancy(16, (ctypes.c_float * 3)(*HI), (ctypes.c_float * 3)(*HI), None),
           N.NrtOccupancy(16, (ctypes.c_float * 3)(-1, math.nan, -1), (ctypes.c_float * 3)(*HI), None)]
    for g in bad:
        assert L.nrt_occupancy_mask(ctypes.byref(g), None, 0, None, None, 1, None, None) == N.E_INVALID
    g = N.NrtOccupancy(16, (ctypes.c_float * 3)(*LO), (ctypes.c_float * 3)(*HI), None)     # bits NULL
    assert L.nrt_occupancy_mask(ctypes.byref(g), None, 0, None, None, 1, None, None) == N.E_INVALID
    assert L.nrt_occupancy_update_workspace(None, 1, 16, 1) == 0


def test_profile_tags_named():
    names = [N.lib().nrt_profile_tag_name(i).decode() for i in range(N.lib().nrt_profile_num_tags())]
    assert "occupancy_cull" in names and "occupancy_update" in names


def test_state_dict_unchanged():
    m = NeRFLE(device="cpu")
    keys = list(m.state_dict().keys())
    m.occupancy = OccupancyGrid(resolution=16, device="cpu")
    assert list(m.state_dict().keys()) == keys
    assert not any("occupancy" in k for k in keys)
    assert NeRFLE(device="cpu").occupancy is None


def test_fake_implementations():
    from torch._subclasses.fake_tensor import FakeTensorMode
    assert "occupancy_update" in torch_ops.OPERATORS
    with FakeTensorMode():
        dens = torch.empty(16 ** 3, device="cuda")
        bits = torch.empty(128, dtype=torch.int32, device="cuda")
        p = torch.empty(100, device="cuda")
        d2, b2 = torch.ops.nrt_b200.occupancy_update(dens, bits, p, torch.empty(3, 16, device="cuda"),
                                                    [3, 0, 16, 128, 5, 3, 65, 0], 16, [-1.0] * 3, [1.0] * 3, 4, 0.0,
                                                    0.01, 1, 1)
        assert d2.shape == dens.shape and b2.shape == bits.shape and b2.dtype == torch.int32
        rays = torch.empty(10, 6, device="cuda")
        ts = torch.empty(64, device="cuda")
        code = torch.empty(1, 3, device="cuda")
        arch1, arch2 = [3, 0, 16, 128, 5, 3, 65, 0], [70, 0, 16, 64, 8, 3, 3, 0]
        out = torch.ops.nrt_b200.nerfle_render(rays, ts, code, p, p, arch1, p, p, arch2, 1, bits, 16, [-1.0] * 3, [1.0] * 3)
        assert out.shape == (10, 3)
        img = torch.ops.nrt_b200.nerfle_render_camera(0, torch.empty(1, 4, 4, device="cuda"), None, 1.0, 1.0, 0, 0, 5, 7, 1,
                                                      0.0, 0, ts, code, p, p, arch1, p, p, arch2, 1, bits, 16, [-1.0] * 3,
                                                      [1.0] * 3)
        assert img.shape == (1, 5, 7, 1, 3)
