"""TEST INFRASTRUCTURE ONLY -- the CPU oracle of utilities.surface_metrics (DESIGN.md section 7d).

scipy.ndimage and numpy, with the rules they do not state:
  * a voxel is foreground when it is non-zero; edges = mask ^ binary_erosion(mask) (6-neighbourhood, voxels outside the
    volume are background);
  * d(A->B) = distance_transform_edt(~edges(B), sampling=spacing)[edges(A)];
  * dice = 2|P n T| / (|P| + |T|) from integer counts; hausdorff = max of both directed maxima; hausdorff_percentile =
    max of np.percentile(d, percentile) (method "linear") over both directions; assd = mean of both directed sets
    together; surface_dice = #{d <= tolerance} over both directions / (#edges(P) + #edges(T));
  * both masks empty: every value NaN; exactly one empty: dice and surface_dice 0, the three distances +inf (numpy alone
    would give NaN for a percentile of an all-inf array).
"""
import numpy as np
from scipy import ndimage

KEYS = ("dice", "hausdorff", "hausdorff_percentile", "assd", "surface_dice")


def edges(mask):
    m = np.asarray(mask) != 0
    return m ^ ndimage.binary_erosion(m)


def directed(edges_a, edges_b, spacing=None):
    """d(A->B): the distances from every edge voxel of A to the nearest edge voxel of B (B must have one)."""
    return ndimage.distance_transform_edt(~edges_b, sampling=spacing)[edges_a]


def volume_metrics(pred, target, spacing=None, percentile=95.0, tolerance=1.0):
    """The five values of one [D, H, W] pair as Python floats."""
    p, t = np.asarray(pred) != 0, np.asarray(target) != 0
    n_p, n_t = int(p.sum()), int(t.sum())
    if n_p == 0 and n_t == 0:
        return dict.fromkeys(KEYS, float("nan"))
    if n_p == 0 or n_t == 0:
        return dict(dice=0.0, hausdorff=float("inf"), hausdorff_percentile=float("inf"), assd=float("inf"),
                    surface_dice=0.0)
    ep, et = edges(p), edges(t)
    d_pt, d_tp = directed(ep, et, spacing), directed(et, ep, spacing)
    return dict(
        dice=2 * int((p & t).sum()) / (n_p + n_t),
        hausdorff=float(max(d_pt.max(), d_tp.max())),
        hausdorff_percentile=float(max(np.percentile(d_pt, percentile), np.percentile(d_tp, percentile))),
        assd=float(np.mean(np.concatenate([d_pt, d_tp]))),
        surface_dice=(int((d_pt <= tolerance).sum()) + int((d_tp <= tolerance).sum())) / (d_pt.size + d_tp.size),
    )


def surface_metrics(pred, target, spacing=None, percentile=95.0, tolerance=1.0):
    """[D, H, W] -> dict of float64 scalars; [B, D, H, W] -> dict of float64 arrays [B]."""
    p, t = np.asarray(pred), np.asarray(target)
    if p.ndim == 3:
        return {k: np.float64(v) for k, v in volume_metrics(p, t, spacing, percentile, tolerance).items()}
    rows = [volume_metrics(p[i], t[i], spacing, percentile, tolerance) for i in range(p.shape[0])]
    return {k: np.array([r[k] for r in rows], dtype=np.float64) for k in KEYS}


def linear_percentile(values, percentile):
    """numpy.percentile(values, percentile) (method "linear") written out: sort, then interpolate between the order
    statistics around (n - 1) q as numpy 2.3's _lerp does."""
    x = np.sort(np.asarray(values, dtype=np.float64))
    n = x.size
    vi = (n - 1) * (percentile / 100)
    if vi >= n - 1:
        return float(x[-1])
    lo = int(np.floor(vi))
    a, b, g = x[lo], x[lo + 1], vi - lo
    diff = b - a
    return float(b - diff * (1 - g) if g >= 0.5 else a + diff * g)
