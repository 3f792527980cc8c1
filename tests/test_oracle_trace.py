"""The oracle's visit trace (Layer.integrate(..., trace=True)) and its replay (tests/visit_replay.py):
the float32 replay of the trace from the layer before the call must BE the oracle's layer after
it, bit for bit, and the float64 replay bounds how far the oracle's own float32 recurrence is
from exact.  These are what the per-path GPU tests (test_gpu_update_paths.py) measure the device
against.  CPU only."""
import numpy as np
import pytest

from tests import util
from tests import visit_replay as vr

U = 2.0 ** -24
# float32 recurrence vs float64, per voxel: bounded by C_ROUNDINGS roundings of size u on
# quantities near trunc (distance) or the weight, per update (see test_gpu_update_paths.py)
C_ROUNDINGS = 16

SCENES = {
    "merged": dict(),
    "simple": dict(method=0),
    "invz_dropoff_sparsity": dict(use_const_weight=0, use_weight_dropoff=1,
                                  use_sparsity_compensation_factor=1,
                                  sparsity_compensation_factor=20.0),
    "max_weight_4": dict(max_weight=4.0),
    "anti_grazing": dict(enable_anti_grazing=1),
    "freespace_points": dict(),
}


def _check_call(ocfg, ol, frame, freespace=False):
    prior = ol.download()
    trace = ol.integrate(ocfg, *frame, freespace=freespace, trace=True)
    after = vr.LayerIndex(ol.download())
    r32 = vr.replay(trace, prior, ocfg, np.float32)
    r64 = vr.replay(trace, prior, ocfg, np.float64)
    d, w, c, found = after.voxels(r32["idx"])
    assert found.all(), "a visited voxel is missing from the oracle's layer"
    assert np.array_equal(r32["distance"].view(np.uint32), d.view(np.uint32)), "distance bits"
    assert np.array_equal(r32["weight"].view(np.uint32), w.view(np.uint32)), "weight bits"
    assert np.array_equal(r32["rgba"], c), "colours"
    trunc = np.float64(np.float32(ocfg.default_truncation_distance))
    n = r64["n"].astype(np.float64)
    err_d = np.abs(d.astype(np.float64) - r64["distance"])
    err_w = np.abs(w.astype(np.float64) - r64["weight"])
    assert (err_d <= C_ROUNDINGS * n * U * trunc).all(), f"distance: max error {err_d.max()}"
    assert (err_w <= C_ROUNDINGS * n * U * r64["weight"]).all(), f"weight: max error {err_w.max()}"
    return trace, r32


@pytest.mark.parametrize("scene", list(SCENES))
def test_trace_replay_is_the_oracle(scene):
    from oracle import oracle_py as orc
    ocfg, _ = util.make_cfgs(**SCENES[scene])
    ol = orc.Layer(0.05)
    saturated = 0
    for frame in util.small_frames(3, stride=8):
        trace, r32 = _check_call(ocfg, ol, frame, freespace=scene == "freespace_points")
        assert len(trace) > 0
        if scene == "max_weight_4":
            saturated += int(((r32["weight"] == 4.0) & (r32["n"] > 4)).sum())
    if scene == "max_weight_4":
        assert saturated > 0


def test_trace_does_not_change_the_result():
    """The traced call computes what the plain call computes; anti-grazing skips are not visits."""
    from oracle import oracle_py as orc
    frames = util.small_frames(2, stride=8)
    lens = {}
    for over in (dict(), dict(enable_anti_grazing=1)):
        ocfg, _ = util.make_cfgs(**over)
        a, b = orc.Layer(0.05), orc.Layer(0.05)
        n = 0
        for f in frames:
            a.integrate(ocfg, *f)
            n += len(b.integrate(ocfg, *f, trace=True))
        util.compare_layers(b.download(), a.download(), str(over), exact=True, check_flags=True)
        lens[bool(over)] = n
    assert lens[True] < lens[False]


def test_trace_needs_the_single_threaded_path():
    from oracle import oracle_py as orc
    ocfg, _ = util.make_cfgs()
    with pytest.raises(ValueError):
        orc.Layer(0.05).integrate(ocfg, *util.small_frames(1, stride=16)[0], threads=2, trace=True)


def test_classify_paths():
    """classify() on a hand-made trace: counts, the general rule (in-band visit, or an existing
    voxel that is neither fresh nor at +trunc) and the size classes."""
    from oracle import oracle_py as orc
    ocfg, _ = util.make_cfgs(default_truncation_distance=0.1)
    rows = []

    def add(v, sdfs):
        for s in sdfs:
            rows.append((v, s, 1.0, (1, 2, 3, 255)))
    add((0, 0, 0), [0.5] * 5)                      # free, fresh
    add((1, 0, 0), [0.5] * 4 + [0.05])             # one in-band visit: general, short
    add((2, 0, 0), [0.5] * 100)                    # general by its prior state: warp
    add((3, 0, 0), [0.5] * 2048)                   # free, long
    add((4, 0, 0), [0.5] * 2047 + [-0.2])          # general, long
    add((5, 0, 0), [0.5] * 96)                     # existing voxel at +trunc: free
    t = np.zeros(len(rows), orc.VISIT_DTYPE)
    for i, (v, s, w, c) in enumerate(rows):
        t[i] = (v, s, w, c)
    vox = np.zeros((1, 4096), orc.VOXEL_DTYPE)
    vox["distance"][0, 2], vox["weight"][0, 2] = 0.03, 2.0
    vox["distance"][0, 5], vox["weight"][0, 5] = np.float32(0.1), 7.0
    prior = (np.zeros((1, 3), np.int32), vox, np.ones(1, np.uint8))
    cl = vr.classify(t, prior, prior[0], ocfg)
    assert cl["idx"][:, 0].tolist() == [0, 1, 2, 3, 4, 5]
    assert cl["n"].tolist() == [5, 5, 100, 2048, 2048, 96]
    assert cl["general"].tolist() == [False, True, True, False, True, False]
    assert [vr.PATHS[p] for p in cl["path"]] == ["free", "short", "warp", "free", "long", "free"]
    assert not cl["closed_form"].any()
