"""TEST INFRASTRUCTURE ONLY -- the CPU oracle of connected-component labelling and the component filters
(preprocess.label_components / largest_component / remove_small_components, DESIGN.md section 7c).

scipy.ndimage.label and numpy.bincount, plus the rules scipy does not state:
  * a voxel is foreground when it is non-zero; connectivity 6 / 18 / 26 = generate_binary_structure(3, 1 / 2 / 3);
  * each volume of a [B, D, H, W] input is labelled on its own (numbering restarts at 1);
  * largest component: most voxels, ties to the lower label; an empty volume stays empty;
  * filters: the voxels of dropped components become 0, every other voxel keeps its input value.
"""
import numpy as np
from scipy import ndimage

RANK = {6: 1, 18: 2, 26: 3}


def structure(connectivity):
    return ndimage.generate_binary_structure(3, RANK[connectivity])


def _volumes(mask):
    m = np.asarray(mask)
    return (m[None] if m.ndim == 3 else m), m.ndim == 3


def label(mask, connectivity=6):
    """(labels int32 like ``mask``, counts int64 [B] -- a scalar for a [D, H, W] input)."""
    vols, single = _volumes(mask)
    labels = np.zeros(vols.shape, dtype=np.int32)
    counts = np.zeros(vols.shape[0], dtype=np.int64)
    for b, v in enumerate(vols):
        lab, n = ndimage.label(v != 0, structure(connectivity))
        labels[b], counts[b] = lab, n
    return (labels[0], counts[0]) if single else (labels, counts)


def _filter(mask, connectivity, keep_of_sizes):
    vols, single = _volumes(mask)
    out = vols.copy()
    for b, v in enumerate(vols):
        lab, n = ndimage.label(v != 0, structure(connectivity))
        sizes = np.bincount(lab.ravel(), minlength=n + 1)
        keep = keep_of_sizes(sizes)
        keep[0] = True                                    # background keeps its value
        out[b] = np.where(keep[lab], v, np.zeros_like(v))
    return out[0] if single else out


def largest(mask, connectivity=6):
    def keep(sizes):
        k = np.zeros(sizes.shape, dtype=bool)
        if sizes.size > 1:
            k[1 + int(np.argmax(sizes[1:]))] = True       # argmax: the first maximum = the lower label
        return k
    return _filter(mask, connectivity, keep)


def remove_small(mask, min_size, connectivity=6):
    return _filter(mask, connectivity, lambda sizes: sizes >= min_size)
