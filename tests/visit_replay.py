"""Replay of the oracle's visit trace (oracle_py.Layer.integrate(..., trace=True)) and the device
path each voxel takes — the plain reference the per-path tests compare the CUDA back half with.

replay() restates the second half of updateTsdfVoxel and Color::blendTwoColors (oracle/
tsdf_oracle.cc update_voxel / blend): the kEps skip, the clamp of the distance to +-trunc, the
clamp of the weight to max_weight and the colour blend inside the truncation band, rounded to a
byte after every blend (std::round: half away from zero).  In float32 it is the oracle, bit for
bit; in float64 it is the high-precision reference of the same recurrence on the same inputs
(sdf, effective weights and colours of the trace)."""
import numpy as np

VPS = 16
K_EPS = np.float32(1e-6)          # voxblox kEpsilon (tsdf_oracle.cc kEps, cg_math.cuh kEps)
# integrate_back.cu: update lists of kWideSegment updates or more are replayed by a warp
# (k_long_finish); kLongSegment or more are first reduced in sub-blocks (k_long_partials)
K_WIDE_SEGMENT = 96
K_LONG_SEGMENT = 2048
DEFAULT_RGBA = (0, 0, 0, 255)     # voxblox::Color() (ORC_DEFAULT_ALPHA / CG_DEFAULT_ALPHA)

PATHS = ("free", "short", "warp", "long")


def _voxel_keys(idx):
    i = np.asarray(idx, np.int64) + (1 << 20)
    return (i[:, 2] << 42) | (i[:, 1] << 21) | i[:, 0]


class LayerIndex:
    """Voxel lookup in a downloaded layer (idx [B,3], voxels [B,4096], flags)."""

    def __init__(self, layer):
        self.idx, self.vox = layer[0], layer[1]
        keys = _voxel_keys(self.idx)
        self.order = np.argsort(keys, kind="stable")
        self.keys = keys[self.order]

    def find(self, gvi):
        """global voxel indices [N,3] -> (found bool [N], block row [N], linear index [N])."""
        gvi = np.asarray(gvi, np.int64)
        blk = gvi >> 4                              # floor division by 16
        lin = (gvi[:, 0] & 15) + VPS * ((gvi[:, 1] & 15) + VPS * (gvi[:, 2] & 15))
        k = _voxel_keys(blk)
        pos = np.searchsorted(self.keys, k)
        pos_c = np.minimum(pos, max(len(self.keys) - 1, 0))
        found = (pos < len(self.keys)) & (self.keys[pos_c] == k) if len(self.keys) else \
            np.zeros(len(k), bool)
        row = np.where(found, self.order[pos_c] if len(self.keys) else 0, 0)
        return found, row, lin

    def voxels(self, gvi):
        """(distance f32, weight f32, rgba u8 [N,4], found) at the given voxels; voxels of
        missing blocks read as a default voxel."""
        found, row, lin = self.find(gvi)
        d = np.zeros(len(found), np.float32)
        w = np.zeros(len(found), np.float32)
        c = np.tile(np.array(DEFAULT_RGBA, np.uint8), (len(found), 1))
        if found.any():
            v = self.vox[row[found], lin[found]]
            d[found], w[found], c[found] = v["distance"], v["weight"], v["rgba"]
        return d, w, c, found


def group(trace):
    """Visits grouped by voxel with a stable sort (the call order is kept inside a voxel) ->
    (voxel idx [V,3], start [V], count [V], order [N]: trace rows voxel by voxel)."""
    keys = _voxel_keys(trace["idx"])
    order = np.argsort(keys, kind="stable")
    sk = keys[order]
    head = np.ones(len(sk), bool)
    head[1:] = sk[1:] != sk[:-1]
    start = np.flatnonzero(head)
    count = np.diff(np.append(start, len(sk)))
    return trace["idx"][order[start]], start, count, order


def _round_half_away(v):
    f = np.floor(v)
    return f + (v - f >= 0.5)


def replay(trace, prior, cfg, dtype=np.float32):
    """The recurrence of updateTsdfVoxel over the trace, starting from `prior` (the layer before
    the call, as downloaded; None for an empty one).  Rank by rank, vectorised over voxels: update
    k of every voxel with more than k updates.  -> dict(idx [V,3], n [V], distance, weight (dtype),
    rgba u8 [V,4], d0, w0, rgba0 (the state before the call))."""
    dt = np.dtype(dtype)
    vidx, start, count, order = group(trace)
    if prior is not None and len(prior[0]):
        d0, w0, c0, _ = LayerIndex(prior).voxels(vidx)
    else:
        d0 = np.zeros(len(vidx), np.float32)
        w0 = np.zeros(len(vidx), np.float32)
        c0 = np.tile(np.array(DEFAULT_RGBA, np.uint8), (len(vidx), 1))
    # voxels by decreasing update count: the voxels still active at rank k are a prefix
    by_n = np.argsort(-count, kind="stable")
    n_sorted = count[by_n]
    first = start[by_n]
    D = d0[by_n].astype(dt)
    W = w0[by_n].astype(dt)
    Cc = c0[by_n].astype(dt)
    trunc = dt.type(np.float32(cfg.default_truncation_distance))
    max_w = dt.type(np.float32(cfg.max_weight))
    eps = dt.type(K_EPS)
    sdf_all = trace["sdf"][order].astype(dt)
    w_all = trace["weight"][order].astype(dt)
    col_all = trace["rgba"][order].astype(dt)
    for k in range(int(n_sorted[0]) if len(n_sorted) else 0):
        m = int(np.searchsorted(-n_sorted, -k, side="left"))  # voxels with n > k
        rows = first[:m] + k
        sdf, w, col = sdf_all[rows], w_all[rows], col_all[rows]
        Dm, Wm = D[:m], W[:m]
        new_w = Wm + w
        ok = ~(new_w < eps)
        new_sdf = (sdf * w + Dm * Wm) / np.where(ok, new_w, dt.type(1))
        band = ok & (np.abs(sdf) < trunc)
        if band.any():
            total = Wm[band] + w[band]
            w1 = (Wm[band] / total)[:, None]
            w2 = (w[band] / total)[:, None]
            Cc[:m][band] = _round_half_away(Cc[:m][band] * w1 + col[band] * w2)
        clamped = np.where(new_sdf > 0, np.where(new_sdf < trunc, new_sdf, trunc),
                           np.where(-trunc < new_sdf, new_sdf, -trunc))
        D[:m] = np.where(ok, clamped, Dm)
        W[:m] = np.where(ok, np.where(new_w < max_w, new_w, max_w), Wm)
    inv = np.empty_like(by_n)
    inv[by_n] = np.arange(len(by_n))
    return dict(idx=vidx, n=count, distance=D[inv], weight=W[inv],
                rgba=Cc[inv].astype(np.uint8), d0=d0, w0=w0, rgba0=c0)


def classify(trace, prior, blocks_before, cfg):
    """For one job (one device call, one group): each voxel's update count n, whether the back
    half treats it as "general", and its path.

    General (integrate_back.cu): one of its visits has !(sdf >= trunc) (k_walk_segments marks the
    visits in the last walk_tail_visits() steps of a ray, which by construction hold every such
    visit), or its block existed before the job and it holds w > 0 && d != trunc
    (k_mark_existing).  Paths: "free" (not general: k_block_accumulate -> k_finalize_blocks),
    "short" (general, n < K_WIDE_SEGMENT: k_voxel_update), "warp" (K_WIDE_SEGMENT <= n <
    K_LONG_SEGMENT: k_long_finish), "long" (n >= K_LONG_SEGMENT: k_long_partials + k_long_finish).
    closed_form: a long list the closed form of k_long_finish takes (every update free space and
    the voxel fresh or at +trunc).  The general rule excludes it: a voxel general by a visit has
    a visit with !(sdf >= trunc), which k_long_partials flags the same way (a NaN sdf included),
    and one general by its prior state has w > 0 and d != trunc.
    -> dict(idx, n, general, path (index into PATHS), closed_form)."""
    vidx, start, count, order = group(trace)
    trunc = np.float32(cfg.default_truncation_distance)
    sdf = trace["sdf"][order]
    not_free = np.logical_or.reduceat(~(sdf >= trunc), start) if len(start) else np.zeros(0, bool)
    existed = np.zeros(len(vidx), bool)
    d0 = np.zeros(len(vidx), np.float32)
    w0 = np.zeros(len(vidx), np.float32)
    if prior is not None and len(prior[0]):
        d0, w0, _, found = LayerIndex(prior).voxels(vidx)
        if blocks_before is not None:
            bb = LayerIndex((np.asarray(blocks_before, np.int32).reshape(-1, 3), None))
            existed = bb.find(vidx)[0]
        else:
            existed = found
    general = not_free | (existed & (w0 > 0) & (d0 != trunc))
    path = np.where(~general, 0, np.where(count < K_WIDE_SEGMENT, 1,
                                          np.where(count < K_LONG_SEGMENT, 2, 3)))
    closed = (path == 3) & ~not_free & ((w0 == 0) | (d0 == trunc)) & (trunc > 0)
    return dict(idx=vidx, n=count, general=general, path=path, closed_form=closed)
