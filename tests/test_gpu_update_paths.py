"""Each voxel-update path of the integrator's back half against the oracle's own visits, replayed
in float64 (tests/visit_replay.py).

Every job starts from the same bits on both sides: the device layer is cleared and loaded with
the oracle's layer before the job, so one-ulp differences of an earlier job cannot make a later
exactness claim meaningless.  Per job, every visited voxel is classified by the path the back half
(integrate_back.cu) gives it, and checked against what that path promises:

- free-space sum (not general; fixed-point sum of ray weights, then D = trunc): distance exactly
  trunc, colour unchanged; the weight bit-identical to the oracle when every ray weight and the
  prior weight are integers, otherwise |W - W64| <= n 2^-(shift+1) + 2u W64 (the rounding of each
  ray weight to the fixed-point grid, then the conversion and the one addition).  The sequential
  reference itself can round just below trunc there, when an sdf is within a few ulps of trunc:
  those voxels are counted and must lie within 2 ulp of trunc.
- short replay (general, fewer than K_WIDE_SEGMENT updates; the reference's update, update by
  update): distance, weight and colour bit-identical to the oracle.
- warp tree / long lists (general, K_WIDE_SEGMENT or more updates; clamped affine maps composed as
  an ordered tree, weights by prefix sums): per voxel |D - D64| <= min(tol, C n u trunc) and
  |W - W64| <= min(tol, C n u W64), tol the BASELINE.json tolerance.  C = 16 counts the roundings
  one update costs on quantities the clamps keep near trunc (distance) or near W (weight): the
  prefix-sum additions into w_prev (up to 5 shuffle levels plus W + pre) and its clamp, the
  reciprocal, a = w_prev / w_new, b = (sdf w) / w_new (2), one composition per update on average
  (a 32-update tree has 31; 3 roundings each) and the final a D + b per chunk; the maps are
  contractions (a <= 1), so errors add rather than grow.  C is the same for every scene.  Per
  class, the device's largest error must also be within SYSTEMATIC times the oracle's own
  largest error against float64, plus 2 ulp — a small systematic error per voxel shows there.
  SYSTEMATIC = 8: the tree spends up to 4x the roundings per update of the sequential update
  (C = 16 against 4: two products, a sum and a quotient), and the largest of a few hundred errors
  is itself a sample; the largest ratio measured on a B200 is 4.3 (warp-tree distances of the
  300-frame cluster with carving).  Colours within 1 LSB.

Also: the visits of the voxels the classifier calls general sum to st.general_updates, which
checks walk_tail_visits and k_mark_existing exactly, and the oracle's visit count equals
st.voxel_updates — except with anti-grazing, where st.voxel_updates is the front half's count of
(ray, voxel) pairs, taken before the walk skips the grazing voxels, so it is larger.  Every job is one group (far below CG_MAX_GROUP_POINTS and CG_MAX_PAIRS):
the update lists are per group."""
import numpy as np
import pytest

from tests import util
from tests import visit_replay as vr

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
C_ROUNDINGS = 16
SYSTEMATIC = 8


def _ulp(x):
    return np.spacing(np.abs(np.float32(x))).astype(np.float64)


def _ceil_log2(v):
    return int(v - 1).bit_length() if v > 1 else 0


def _shift(max_weight, rays):
    """The fixed-point shift of the free-space sum (integrate_back.cu, run_back_half)."""
    wb = _ceil_log2(int(min(max(np.float32(max_weight), 1.0), 1.0e9)) + 1)
    return max(0, min(40 - wb, 62 - wb - _ceil_log2(int(rays) + 1)))


def _ns_tol(ref):
    return np.maximum(util.ATOL, util.RTOL * np.abs(ref))


class _Tally:
    """Per-path counts and margins over the jobs of one scene."""

    def __init__(self):
        self.n = {p: 0 for p in vr.PATHS}
        self.worst = {}          # name -> max error / bound
        self.dev = {}            # (path, field) -> max device error vs float64
        self.orc = {}            # (path, field) -> max oracle error vs float64
        self.mag = {}            # (path, field) -> max |float64 value|
        self.below_trunc = 0     # free voxels the sequential reference rounds below trunc
        self.closed_form = 0
        self.counts_mismatch = []

    def worst_of(self, name, ratio):
        if ratio.size:
            self.worst[name] = max(self.worst.get(name, 0.0), float(ratio.max()))

    def err(self, table, key, e):
        if e.size:
            table[key] = max(table.get(key, 0.0), float(e.max()))

    def record(self, scene):
        m = {"voxels": dict(self.n), "closed_form": self.closed_form,
             "free_below_trunc": self.below_trunc,
             "max_err_over_bound": self.worst,
             "device_vs_oracle_err": {f"{p}.{f}": [self.dev.get((p, f), 0.0),
                                                   self.orc.get((p, f), 0.0)]
                                      for p in ("warp", "long") for f in ("distance", "weight")}}
        util.record_margins(f"update_paths/{scene}", m)
        return m


def _check_job(ocfg, prior, trace, st, got, ref, tally, what):
    trunc = np.float32(ocfg.default_truncation_distance)
    assert np.array_equal(got[0], ref[0]), f"{what}: block sets differ"
    cl = vr.classify(trace, prior, prior[0], ocfg)
    n_gen = int(cl["n"][cl["general"]].sum())
    pairs_ok = (st.voxel_updates >= len(trace) if ocfg.enable_anti_grazing and ocfg.method == 1
                else st.voxel_updates == len(trace))
    if not pairs_ok or n_gen != st.general_updates:
        tally.counts_mismatch.append((what, len(trace), int(st.voxel_updates), n_gen,
                                      int(st.general_updates)))
    r64 = vr.replay(trace, prior, ocfg, np.float64)
    assert np.array_equal(r64["idx"], cl["idx"])
    gd, gw, gc, _ = vr.LayerIndex(got).voxels(cl["idx"])
    od, ow, oc, _ = vr.LayerIndex(ref).voxels(cl["idx"])
    n = cl["n"].astype(np.float64)
    path = cl["path"]
    for k, name in enumerate(vr.PATHS):
        tally.n[name] += int((path == k).sum())
    tally.closed_form += int(cl["closed_form"].sum())

    # short replay: bit for bit
    s = path == 1
    assert np.array_equal(gd[s].view(np.uint32), od[s].view(np.uint32)), \
        f"{what}: short replay, {int((gd[s] != od[s]).sum())} distances differ from the oracle"
    assert np.array_equal(gw[s].view(np.uint32), ow[s].view(np.uint32)), \
        f"{what}: short replay, {int((gw[s] != ow[s]).sum())} weights differ from the oracle"
    assert np.array_equal(gc[s], oc[s]), f"{what}: short replay, colours differ from the oracle"

    # free-space sum
    f = path == 0
    order = vr.group(trace)[3]
    start = vr.group(trace)[1]
    w_sorted = trace["weight"][order]
    any_w = np.logical_or.reduceat(w_sorted > 0, start)
    integral = np.logical_and.reduceat(w_sorted == np.floor(w_sorted), start) & \
        (r64["w0"] == np.floor(r64["w0"]))
    fw = f & any_w
    assert (gd[fw] == trunc).all(), f"{what}: free-space voxel with distance != trunc"
    assert np.array_equal(gc[f], r64["rgba0"][f]), f"{what}: free-space voxel changed colour"
    fi = fw & integral
    assert np.array_equal(gw[fi].view(np.uint32), ow[fi].view(np.uint32)), \
        f"{what}: free-space sum of integer weights differs from the oracle"
    sh = _shift(ocfg.max_weight, st.rays)
    bound = n[fw] * 2.0 ** -(sh + 1) + 2 * U * r64["weight"][fw]
    e = np.abs(gw[fw].astype(np.float64) - r64["weight"][fw])
    tally.worst_of("free.weight", e / np.maximum(bound, 1e-300))
    assert (e <= bound).all(), f"{what}: free-space weight off by {e.max()} (shift {sh})"
    below = fw & (od < trunc)
    tally.below_trunc += int(below.sum())
    assert (trunc.astype(np.float64) - od[below] <= 2 * _ulp(trunc)).all(), \
        f"{what}: the reference rounds a free-space voxel more than 2 ulp below trunc"

    # warp tree and long lists
    for k, name in ((2, "warp"), (3, "long")):
        m = path == k
        if not m.any():
            continue
        for field, g, o, scale in (("distance", gd, od, np.float64(trunc)),
                                   ("weight", gw, ow, r64["weight"][m])):
            ref64 = r64[field][m]
            bound = np.minimum(_ns_tol(ref64), C_ROUNDINGS * n[m] * U * scale)
            e_dev = np.abs(g[m].astype(np.float64) - ref64)
            e_orc = np.abs(o[m].astype(np.float64) - ref64)
            tally.worst_of(f"{name}.{field}", e_dev / np.maximum(bound, 1e-300))
            tally.err(tally.dev, (name, field), e_dev)
            tally.err(tally.orc, (name, field), e_orc)
            tally.err(tally.mag, (name, field), np.abs(ref64))
            assert (e_dev <= bound).all(), \
                f"{what}: {name} {field} off by {e_dev.max()} against float64 ({int((e_dev > bound).sum())} voxels)"
        dc = np.abs(gc[m].astype(np.int16) - oc[m].astype(np.int16))
        assert dc.max(initial=0) <= 1, f"{what}: {name} colour differs by {dc.max()} LSB"


def _class_systematic(tally, what):
    for (name, field), e_dev in tally.dev.items():
        e_orc = tally.orc[(name, field)]
        two_ulp = 2 * _ulp(tally.mag[(name, field)])
        assert e_dev <= SYSTEMATIC * e_orc + two_ulp, \
            f"{what}: {name} {field}: device error {e_dev} vs the oracle's own {e_orc}"


def _lockstep(gpu_ctx, scene, jobs, voxel_size=0.05, max_blocks=8192, freespace=False, **over):
    """Runs the jobs (lists of frames: one frame = integratePointCloud, more = integrateBatch) on
    both sides in lock step and checks every path; returns the tally."""
    from coxgraph_b200 import Layer, TsdfIntegrator
    from oracle import oracle_py as orc
    ocfg, gcfg = util.make_cfgs(**over)
    ol, gl = orc.Layer(voxel_size), Layer(gpu_ctx, voxel_size, max_blocks=max_blocks)
    integ = TsdfIntegrator(gcfg, gl)
    tally = _Tally()
    for j, frames in enumerate(jobs):
        prior = ol.download()
        gl.removeAllBlocks()
        if len(prior[0]):
            gl.upload(*prior)
        trace = np.concatenate([ol.integrate(ocfg, T, p, c, freespace=freespace, trace=True)
                                for (T, p, c) in frames])
        if len(frames) == 1:
            st = integ.integratePointCloud(*frames[0], freespace_points=freespace)
        else:
            offs = np.cumsum([0] + [len(p) for (_, p, _) in frames]).astype(np.uint64)
            st = integ.integrateBatch(np.stack([T for (T, _, _) in frames]),
                                      np.concatenate([p for (_, p, _) in frames]),
                                      np.concatenate([c for (_, _, c) in frames]), offs,
                                      freespace_points=freespace)
        _check_job(ocfg, prior, trace, st, gl.download(), ol.download(), tally, f"{scene} job {j}")
    gl.close()
    m = tally.record(scene)
    _class_systematic(tally, scene)
    # visits: the oracle's count of updateTsdfVoxel calls is the device's count of (ray, voxel)
    # pairs, and the general ones are those of the voxels classified general
    assert not tally.counts_mismatch, f"{scene}: visit counts (job, oracle, device, general " \
        f"oracle, general device): {tally.counts_mismatch}"
    return m


def _cluster(n_frames=300, n_points=200):
    """The scene of test_gpu_edge.py::test_thousands_of_updates_per_voxel: the same small cluster
    from the same pose, every frame — with 200 points a frame instead of 40, so that voxels of the
    band (general ones) get 2048 updates or more (about 3000) and take the long lists; with 40
    they get at most about 1400."""
    rng = np.random.default_rng(5)
    base = np.array([0.3, -0.2, 1.4])
    T = np.array([1, 0, 0, 0, 0.01, 0.02, 0.03], np.float32)
    frames = []
    for _ in range(n_frames):
        p = (base + rng.uniform(-0.08, 0.08, (n_points, 3))).astype(np.float32)
        c = rng.integers(0, 256, (n_points, 4), dtype=np.uint8)
        c[:, 3] = 255
        frames.append((T, p, c))
    return frames


def _full_res(n=16):
    """Full 640x480 frames of one submap in one batch: with 16 of them the band voxels get up to
    about 350 updates (with 3, fewer than 96: the merged rays are few per voxel and frame)."""
    return util.small_frames(n, stride=1, robot=1, submap=2)


def test_small_frames_short_and_free(gpu_ctx):
    frames = util.small_frames(3, stride=8)
    for method in (1, 0):
        m = _lockstep(gpu_ctx, f"small_frames_method{method}", [[f] for f in frames], method=method)
        assert m["voxels"]["short"] > 0 and m["voxels"]["free"] > 0
    _lockstep(gpu_ctx, "small_frames_batched", [frames[:2], frames[2:]])


@pytest.mark.parametrize("over", [dict(), dict(use_const_weight=0), dict(max_weight=4.0),
                                  dict(use_const_weight=0, max_weight=0.5)],
                         ids=["const", "invz", "max_weight_4", "invz_max_weight_0.5"])
def test_full_resolution_warp_tree(gpu_ctx, over):
    """Full-resolution frames in one batch: lists of hundreds of updates (the warp tree)."""
    m = _lockstep(gpu_ctx, "full_res_" + "_".join(f"{k}{v}" for k, v in over.items()),
                  [_full_res()], max_blocks=16384, default_truncation_distance=0.16, **over)
    assert m["voxels"]["warp"] > 0


@pytest.mark.parametrize("carving", [1, 0])
@pytest.mark.parametrize("over", [dict(), dict(use_const_weight=0), dict(max_weight=4.0),
                                  dict(use_const_weight=0, max_weight=0.5)],
                         ids=["const", "invz", "max_weight_4", "invz_max_weight_0.5"])
def test_cluster_long_lists(gpu_ctx, carving, over):
    """300 frames of one small cluster in one job, then the same again on the result: lists of
    2048 updates or more, from a fresh voxel and from one with history."""
    frames = _cluster()
    m = _lockstep(gpu_ctx, f"cluster_carving{carving}_" + "_".join(f"{k}{v}" for k, v in over.items()),
                  [frames, frames], voxel_carving_enabled=carving,
                  default_truncation_distance=0.16, **over)
    assert m["voxels"]["long"] > 0


def test_dropoff_and_sparsity(gpu_ctx):
    """Drop-off gives zero weights to visits far behind the surface (the first_ok skip of the warp
    replay when they come first); sparsity compensation scales the band weights by 20."""
    m = _lockstep(gpu_ctx, "dropoff_sparsity", [_full_res()], max_blocks=16384, use_const_weight=0,
                  use_weight_dropoff=1, use_sparsity_compensation_factor=1,
                  sparsity_compensation_factor=20.0, default_truncation_distance=0.16)
    assert m["voxels"]["warp"] > 0


def test_anti_grazing(gpu_ctx):
    _lockstep(gpu_ctx, "anti_grazing", [_full_res()], max_blocks=16384, use_const_weight=0,
              enable_anti_grazing=1)


def test_fine_voxels_720p(gpu_ctx):
    from coxgraph_b200 import synth
    frames = util.small_frames(2, stride=8, cam=synth.CAM_1280x720)
    _lockstep(gpu_ctx, "2cm_720p", [[f] for f in frames], voxel_size=0.02, max_blocks=16384,
              default_truncation_distance=0.06, max_ray_length_m=3.0)


def test_freespace_points(gpu_ctx):
    frames = util.small_frames(3, stride=8)
    _lockstep(gpu_ctx, "freespace_points", [[f] for f in frames], freespace=True)
