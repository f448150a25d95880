"""GPU versions of the hot-path helpers of ``ctunet.utilities`` / ``ctunet.pytorch.transforms``.

  hard_segm_from_tensor   ctunet/utilities.py:103-124
  shape_3d                ctunet/utilities.py:127-178
  random_blank_patch      ctunet/pytorch/transforms.py:241-300
  SkullRandomHole         ctunet/pytorch/transforms.py:52-94
  encode_flaprec_batch    ctunet/pytorch/datasets.py:195-235, :30-47 (one-hot targets, atlas channel)
  dice_coeff, hausdorff   ctunet/utilities.py:53-70 (reporting metrics; monai restated -> parity unpinned)
  surface_metrics         no reference counterpart: per-volume Dice, Hausdorff, percentile Hausdorff, ASSD and surface
                          Dice with voxel spacing (DESIGN.md section 7d; oracle tests/surface_oracle.py)
  SaltAndPepper           ctunet/pytorch/transforms.py:13-49
  RandomAffine,           no reference counterpart: seeded rotation, scaling, translation and flips of mask batches
  affine_masks            (DESIGN.md section 7e; oracle tests/affine_oracle.py)
  RandomCraniectomy       SkullRandomHole / random_blank_patch drawn on the device from a Philox stream, without host
                          synchronisation (DESIGN.md section 7f; oracle tests/craniectomy_oracle.py)

The 'flap' shape of shape_3d calls the un-vendored, unpinned ``raster_geometry`` package in the reference
(utilities.py:145-166); it is not installed here, so ``cylinder`` / ``cube`` are RESTATED from the package's published
algorithm (oracle/unet_oracle.py: ``rg_cylinder``, ``rg_cube``) -- sphere and box are pinned to the reference,
the flap shape is parity unpinned.
"""
from __future__ import annotations

import ctypes
import math
import random

import numpy as np
import torch

from ._lib import call, ptr_array, stream_ptr
from ._lib import load as _load
from .losses import dice_loss  # noqa: F401  (re-export: utils.dice_loss)

_SHAPES = {"circle": 0, "sphere": 0, "square": 1, "box": 1, "cube": 1, "flap": 2, "autoimplant": 2}


def _need_cuda(t, what):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError("%s runs on CUDA tensors only (no CPU fallback)" % what)


def hard_segm_from_tensor(prob_map: torch.Tensor, keep_dims: bool = False) -> torch.Tensor:
    """Channel argmax as float32; ties go to the lowest index (utilities.py:118-124)."""
    _need_cuda(prob_map, "hard_segm_from_tensor")
    x = prob_map.float().contiguous()
    five = x.dim() == 5
    if not five:
        x = x.unsqueeze(0)
    b, c = x.shape[0], x.shape[1]
    spatial = x[0, 0].numel()
    out = torch.empty((b,) + tuple(x.shape[2:]), dtype=torch.float32, device=x.device)
    call("ctu_argmax_channels", x.data_ptr(), out.data_ptr(), b, c, spatial, stream_ptr())
    if five:
        return out.unsqueeze(1) if keep_dims else out
    out = out[0]
    return out.unsqueeze(0) if keep_dims else out


def blank_patch(image: torch.Tensor, center, size, shape: str, c_diam=None):
    """``masked = image AND outside``, ``extracted = image AND inside`` (uint8), the arithmetic of
    transforms.py:286-296 for a given centre / radius / shape.  ``center`` is a host triple or a device int32[3].
    The 'flap' shape draws its cylinder radius ``c_diam`` from the numpy RNG as utilities.py:146-148 unless given."""
    _need_cuda(image, "blank_patch")
    if shape not in _SHAPES:
        raise ValueError("shape %r is not supported (sphere, box, flap)" % (shape,))
    if _SHAPES[shape] == 2 and c_diam is None:
        c_diam = np.random.uniform(0.25, 1) * size / 4
    img = image.to(torch.uint8).contiguous()
    if img.dim() != 3:
        raise ValueError("expected a [D, H, W] volume")
    if not isinstance(center, torch.Tensor):
        center = torch.tensor([int(c) for c in center], dtype=torch.int32, device=img.device)
    masked, extracted = torch.empty_like(img), torch.empty_like(img)
    d, h, w = img.shape
    call("ctu_flap_mask_u8", img.data_ptr(), masked.data_ptr(), extracted.data_ptr(), d, h, w, center.data_ptr(),
         float(size), _SHAPES[shape], float(c_diam or 0.0), stream_ptr())
    return masked, extracted


def shape_3d(center, size, image_size, shape="flap", device="cuda", c_diam=None) -> torch.Tensor:
    """utilities.py:127-178: 0 inside the shape (bounds inclusive), 1 outside; float64 for sphere / box, uint8 for
    the flap shape, as the reference returns them."""
    ones = torch.ones(tuple(image_size), dtype=torch.uint8, device=device)
    masked, _ = blank_patch(ones, center, size, shape, c_diam)
    return masked if _SHAPES[shape] == 2 else masked.to(torch.float64)


def count_nonzero(image: torch.Tensor) -> int:
    img = image.to(torch.uint8).contiguous()
    cnt = torch.empty(1, dtype=torch.int64, device=img.device)
    call("ctu_count_nonzero_u8", img.data_ptr(), img.numel(), cnt.data_ptr(), stream_ptr())
    return int(cnt.item())


def kth_nonzero(image: torch.Tensor, k: int) -> torch.Tensor:
    """Device int32[3] = ``np.argwhere(image > 0)[k]`` (C order), transforms.py:249-252."""
    img = image.to(torch.uint8).contiguous()
    d, h, w = img.shape
    scratch = torch.empty((img.numel() + 4095) // 4096 + 1, dtype=torch.int64, device=img.device)
    coords = torch.empty(3, dtype=torch.int32, device=img.device)
    call("ctu_kth_nonzero_u8", img.data_ptr(), d, h, w, int(k), scratch.data_ptr(), coords.data_ptr(), stream_ptr())
    return coords


def radius_bounds(image_size):
    """transforms.py:266-267"""
    min_radius = (int(np.min(image_size)) // 5) - 1
    max_radius = np.max([min_radius, np.max(image_size) // 3.5])
    return min_radius, max_radius


def random_blank_patch(image: torch.Tensor, prob=1, return_extracted=False, p_type="random",
                       valid_shapes=("sphere", "box", "flap")):
    """transforms.py:241-300 on a CUDA volume.  Consumes the host RNGs in the reference's order
    (random.uniform, np.random.choice, np.random.randint, np.random.randint, and np.random.uniform for the flap
    shape) so a seeded run picks the same voxel index, radius, shape index and cylinder radius as the reference would
    for the same nonzero count."""
    _need_cuda(image, "random_blank_patch")
    img = image.to(torch.uint8).contiguous()
    r = random.uniform(0, 1)
    if prob >= r:
        n = count_nonzero(img)
        if n:
            center = kth_nonzero(img, int(np.random.choice(n)))
            min_radius, max_radius = radius_bounds(tuple(img.shape))
            size = np.random.randint(min_radius, max_radius)
            if p_type not in valid_shapes:
                p_type = valid_shapes[np.random.randint(0, len(valid_shapes))]
            masked, extracted = blank_patch(img, center, size, p_type)
            return (masked, extracted) if return_extracted else masked
    return (img, torch.zeros_like(img)) if return_extracted else img


class SkullRandomHole(object):
    """transforms.py:52-94 for CUDA tensors: ``sample['image']`` is [D,H,W] or [B,D,H,W]."""

    def __init__(self, p=1, double_output=False):
        self.p = p
        self.double_output = double_output

    def __call__(self, sample):
        img = sample["image"]
        _need_cuda(img, "SkullRandomHole")
        is_batch = img.dim() == 4
        vols = img if is_batch else img.unsqueeze(0)
        full = vols.to(torch.uint8)
        brk, flap = [], []
        for i in range(vols.shape[0]):
            m, e = random_blank_patch(full[i], self.p, True)
            brk.append(m)
            flap.append(e)
        brk, flap = torch.stack(brk), torch.stack(flap)
        if not is_batch:
            brk, flap = brk[0], flap[0]
        if self.double_output:
            return {"image": brk, "target": (full, flap)}
        return {"image": brk, "target": flap}


def encode_flaprec_batch(broken: torch.Tensor, full: torch.Tensor, flap: torch.Tensor, atlas=None, out=None):
    """What ``FlapRecWShapePrior2OTrainDataset.__getitem__`` + the default collate hand the model
    (datasets.py:195-235), computed on the device from uint8 masks [B,D,H,W]:
    image [B,Cin,D,H,W] float32 (channel 0 = the broken skull, channel 1 = ``atlas`` [D,H,W] float32 as
    ``load_atlas_and_append_at_axis`` appends it, datasets.py:30-47) and the two targets
    ``one_hot(label, 2).movedim(-1, 1).float()`` [B,2,D,H,W] (datasets.py:209-214).  The host then ships 3 bytes per
    voxel instead of 24.  ``out = (image, (skull_target, flap_target))`` writes into existing tensors;
    ``out = (image, None)`` produces the image only (the fused head + loss kernels of the training step read the uint8
    label masks themselves)."""
    for t in (broken, full, flap):
        _need_cuda(t, "encode_flaprec_batch")
        if t.dtype != torch.uint8 or t.dim() != 4 or t.shape != broken.shape:
            raise TypeError("encode_flaprec_batch expects three uint8 [B, D, H, W] masks of one shape")
    b = broken.shape[0]
    vol = tuple(broken.shape[1:])
    spatial = broken[0].numel()
    cin = 1 if atlas is None else 2
    if atlas is not None and (atlas.dtype != torch.float32 or tuple(atlas.shape) != vol or not atlas.is_cuda):
        raise TypeError("atlas: float32 CUDA volume of the mask shape")
    if out is None:
        image = torch.empty((b, cin) + vol, dtype=torch.float32, device=broken.device)
        sk = torch.empty((b, 2) + vol, dtype=torch.float32, device=broken.device)
        fl = torch.empty_like(sk)
    elif out[1] is None:
        image, sk, fl = out[0], None, None
        if image.dtype != torch.float32 or tuple(image.shape) != (b, cin) + vol or not image.is_contiguous() or not image.is_cuda:
            raise TypeError("encode_flaprec_batch: out image must be contiguous float32 CUDA [B, C, D, H, W]")
    else:
        image, (sk, fl) = out
        for t, c in ((image, cin), (sk, 2), (fl, 2)):
            if t.dtype != torch.float32 or tuple(t.shape) != (b, c) + vol or not t.is_contiguous() or not t.is_cuda:
                raise TypeError("encode_flaprec_batch: out tensors must be contiguous float32 CUDA [B, C, D, H, W]")
    call("ctu_encode_flaprec_u8", broken.contiguous().data_ptr(), full.contiguous().data_ptr(),
         flap.contiguous().data_ptr(), atlas.contiguous().data_ptr() if atlas is not None else None, image.data_ptr(),
         sk.data_ptr() if sk is not None else None, fl.data_ptr() if fl is not None else None, b, cin, spatial, stream_ptr())
    return image, ((sk, fl) if sk is not None else None)


def pack_mask_bits(mask: torch.Tensor) -> torch.Tensor:
    """uint8 {0,1} mask [..., S] -> bit-packed uint8 [..., S / 8], voxel v = bit ``v & 7`` of byte ``v >> 3`` (numpy
    ``packbits(bitorder="little")``): the wire format of ``encode_flaprec_bits`` / ``TrainStep.step_from_bits``.  Works on
    host or device tensors (a data pipeline would emit this format directly)."""
    flat = (mask.reshape(mask.shape[0], -1) != 0).to(torch.uint8)
    if flat.shape[1] % 8:
        raise ValueError("the volume size must be a multiple of 8 voxels")
    w = torch.tensor([1, 2, 4, 8, 16, 32, 64, 128], dtype=torch.uint8, device=mask.device)
    return (flat.view(flat.shape[0], -1, 8) * w).sum(-1, dtype=torch.int32).to(torch.uint8).contiguous()


def encode_flaprec_bits(broken_bits, full_bits, flap_bits, vol_shape, atlas=None, out=None):
    """``encode_flaprec_batch`` from bit-packed masks ([B, D*H*W/8] uint8 each, ``pack_mask_bits``): returns / fills
    ``(image float32 [B,Cin,D,H,W], (full_mask, flap_mask) uint8 [B,D,H,W])`` -- the label masks are what the fused head +
    loss kernels of ``trainer.TrainStep`` take as targets."""
    for t in (broken_bits, full_bits, flap_bits):
        _need_cuda(t, "encode_flaprec_bits")
        if t.dtype != torch.uint8 or t.dim() != 2 or t.shape != broken_bits.shape or not t.is_contiguous():
            raise TypeError("encode_flaprec_bits expects three contiguous uint8 [B, D*H*W/8] bit volumes of one shape")
    b = broken_bits.shape[0]
    vol = tuple(vol_shape)
    spatial = vol[0] * vol[1] * vol[2]
    if broken_bits.shape[1] * 8 != spatial:
        raise ValueError("bit volumes of %d bytes do not match the volume shape %s" % (broken_bits.shape[1], vol))
    cin = 1 if atlas is None else 2
    if atlas is not None and (atlas.dtype != torch.float32 or tuple(atlas.shape) != vol or not atlas.is_cuda):
        raise TypeError("atlas: float32 CUDA volume of the mask shape")
    if out is None:
        image = torch.empty((b, cin) + vol, dtype=torch.float32, device=broken_bits.device)
        fm = torch.empty((b,) + vol, dtype=torch.uint8, device=broken_bits.device)
        lm = torch.empty_like(fm)
    else:
        image, (fm, lm) = out
        for t, shp, dt in ((image, (b, cin) + vol, torch.float32), (fm, (b,) + vol, torch.uint8), (lm, (b,) + vol, torch.uint8)):
            if t.dtype != dt or tuple(t.shape) != shp or not t.is_contiguous() or not t.is_cuda:
                raise TypeError("encode_flaprec_bits: out = (float32 image [B,C,D,H,W], (uint8 [B,D,H,W], uint8 [B,D,H,W]))")
    call("ctu_encode_flaprec_bits", broken_bits.data_ptr(), full_bits.data_ptr(), flap_bits.data_ptr(),
         atlas.contiguous().data_ptr() if atlas is not None else None, image.data_ptr(), fm.data_ptr(), lm.data_ptr(), b, cin,
         spatial, stream_ptr())
    return image, (fm, lm)


# ---------------------------------------------------------------------------------------------- reporting metrics
def _metric_pair(pred, target, what):
    _need_cuda(pred, what)
    _need_cuda(target, what)
    if pred.dim() != 5 or pred.shape != target.shape or not 2 <= pred.shape[1] <= 4:
        raise ValueError("%s expects prediction and one-hot target of one [B, C, D, H, W] shape, 2 <= C <= 4" % what)
    return pred.detach().float().contiguous(), target.detach().float().contiguous()


def dice_coeff(pred: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
    """``utils.dice_coeff`` (utilities.py:53-60): mean over (sample, foreground class) of the hard-label Dice coefficient
    ``2|P n T| / (|P| + |T|)`` with P = ``argmax(pred, 1) == class`` -- ``monai.metrics.compute_meandice(one_hot(argmax),
    target, include_background=False)`` restated (NaN where the target class is empty, which then propagates through the
    mean exactly as in the reference).  Returns a 0-dim float32 CUDA tensor; no host synchronisation.
    One divergence, documented: when NO voxel of the whole batch is predicted foreground the reference's
    ``one_hot(argmax)`` has a single channel and monai raises on the shape mismatch; here the class counts as empty."""
    p, t = _metric_pair(pred, target, "dice_coeff")
    b, c = p.shape[0], p.shape[1]
    counts = torch.empty(3 * b * (c - 1), dtype=torch.float64, device=p.device)
    out = torch.empty(1, dtype=torch.float32, device=p.device)
    call("ctu_dice_coeff", p.data_ptr(), t.data_ptr(), b, c, p[0, 0].numel(), counts.data_ptr(), out.data_ptr(), stream_ptr())
    return out[0]


def hausdorff(result_b: torch.Tensor, reference_b: torch.Tensor) -> torch.Tensor:
    """``utils.hausdorff`` (utilities.py:63-70): mean over (sample, foreground class) of the symmetric Hausdorff distance
    between the surfaces of ``argmax(result_b, 1) == class`` and ``reference_b[:, class] == 1``
    (``monai.metrics.compute_hausdorff_distance`` restated: surface = mask minus its 6-neighbourhood erosion, Euclidean
    distance in voxels); NaN / inf (an empty surface) become ``max(reference_b.shape)`` as utilities.py:64,69 do.
    Exact integer squared distance transform on the device; returns a 0-dim float64 CUDA tensor, no host sync."""
    p, t = _metric_pair(result_b, reference_b, "hausdorff")
    b, c, d, h, w = p.shape
    lib = _load()
    nbytes = lib.ctu_hausdorff_workspace_bytes(b, c, d, h, w)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=p.device)
    out = torch.empty(1, dtype=torch.float64, device=p.device)
    call("ctu_hausdorff", p.data_ptr(), t.data_ptr(), b, c, d, h, w, float(max(reference_b.shape)), ws.data_ptr(), nbytes,
         out.data_ptr(), stream_ptr())
    return out[0]


_MASK_DTYPES = {torch.uint8: 1, torch.bool: 1, torch.float32: 4}      # CTU_MASK_U8 / CTU_MASK_F32
SURFACE_METRIC_KEYS = ("dice", "hausdorff", "hausdorff_percentile", "assd", "surface_dice")


def _number(x):
    return isinstance(x, (int, float, np.integer, np.floating)) and not isinstance(x, bool)


def surface_metrics(pred: torch.Tensor, target: torch.Tensor, spacing=None, percentile: float = 95.0,
                    tolerance: float = 1.0) -> dict:
    """Surface-distance scores of a binary prediction against its ground truth, per volume (DESIGN.md section 7d).

    ``pred`` and ``target``: CUDA masks of one shape, [D, H, W] or [B, D, H, W], each uint8, bool or float32; a voxel is
    foreground when it is non-zero (for several classes pass ``labels == k``); every axis at most 1024.  Edges are the
    mask minus its 6-neighbourhood erosion (voxels outside the volume are background); d(A->B) are the Euclidean
    distances from each edge voxel of A to the nearest edge voxel of B, in voxels, or in the unit of ``spacing`` =
    (sz, sy, sx) in the D, H, W order.

    Returns float64 CUDA tensors ([B], or 0-dim for a [D, H, W] input), computed without a host synchronisation:
      dice                  2|P n T| / (|P| + |T|)
      hausdorff             max(max d(P->T), max d(T->P))
      hausdorff_percentile  max(pct(d(P->T)), pct(d(T->P))), pct = numpy.percentile(., percentile) (method "linear")
      assd                  mean of d(P->T) and d(T->P) together
      surface_dice          (#{d(P->T) <= tolerance} + #{d(T->P) <= tolerance}) / (#edges(P) + #edges(T))
    Both masks empty: every value is NaN.  One mask empty: dice and surface_dice are 0, the three distances +inf (a
    predicted structure that does not exist scores 0; unlike ``dice_coeff``, nothing is NaN)."""
    what = "surface_metrics"
    for t in (pred, target):
        if not isinstance(t, torch.Tensor):
            raise RuntimeError("%s runs on CUDA tensors only (no CPU fallback)" % what)
    if pred.dim() not in (3, 4):
        raise ValueError("%s expects [D, H, W] or [B, D, H, W] masks, got %d dimensions" % (what, pred.dim()))
    if pred.shape != target.shape:
        raise ValueError("%s: prediction %s and target %s differ in shape" % (what, tuple(pred.shape), tuple(target.shape)))
    if not all(1 <= n <= 1024 for n in pred.shape[-3:]) or pred.numel() >= 2 ** 31:
        raise ValueError("%s: every axis must be 1..1024 and B*D*H*W below 2^31, got %s" % (what, tuple(pred.shape)))
    for t in (pred, target):
        if t.dtype not in _MASK_DTYPES:
            raise TypeError("%s expects uint8, bool or float32 masks, got %s" % (what, t.dtype))
    sp = None
    if spacing is not None:
        sp = list(spacing) if isinstance(spacing, (tuple, list)) else None
        if sp is None or len(sp) != 3 or not all(_number(s) and math.isfinite(s) and s > 0 for s in sp):
            raise ValueError("%s: spacing must be three positive finite numbers (sz, sy, sx), got %r" % (what, spacing))
        sp = [float(s) for s in sp]
    if not _number(percentile) or not 0 <= percentile <= 100:
        raise ValueError("%s: percentile must be in [0, 100], got %r" % (what, percentile))
    if not _number(tolerance) or not tolerance >= 0:
        raise ValueError("%s: tolerance must be >= 0, got %r" % (what, tolerance))
    if not pred.is_cuda or not target.is_cuda:
        raise RuntimeError("%s runs on CUDA tensors only (no CPU fallback)" % what)
    if pred.device != target.device:
        raise ValueError("%s: prediction on %s, target on %s" % (what, pred.device, target.device))
    p, t = pred.contiguous(), target.contiguous()
    b = p.shape[0] if p.dim() == 4 else 1
    d, h, w = p.shape[-3:]
    nbytes = _load().ctu_surface_metrics_workspace_bytes(b, d, h, w, int(sp is not None))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=p.device)
    out = torch.empty((5, b), dtype=torch.float64, device=p.device)
    call("ctu_surface_metrics", _MASK_DTYPES[p.dtype], p.data_ptr(), _MASK_DTYPES[t.dtype], t.data_ptr(), b, d, h, w,
         (ctypes.c_double * 3)(*sp) if sp is not None else None, float(percentile), float(tolerance), out.data_ptr(),
         ws.data_ptr(), nbytes, stream_ptr())
    return {k: (out[i] if p.dim() == 4 else out[i, 0]) for i, k in enumerate(SURFACE_METRIC_KEYS)}


# ---------------------------------------------------------------------------------------------- SaltAndPepper
class SaltAndPepper(object):
    """transforms.py:13-49 for CUDA tensors ([D,H,W] or [B,D,H,W], any dtype; returns float32 like ``torch.FloatTensor``).

    Kept from the reference, in its order: ``self.noise_density`` is OVERWRITTEN by ``np.random.uniform(0, noise_density)``
    on every call and key (transforms.py:31 -- the noise decays towards zero over training, SURVEY App. D.12), then per
    image one ``random.uniform(0, 1)`` gate against ``p``.  The two per-voxel uniform fields come from a Philox
    counter-based generator on the device (seeded from the numpy RNG, one draw per noisy image) instead of 2 x D*H*W
    float64 draws from numpy's MT19937 stream on the host: same distribution, different stream.  ``fields=(u_black, u_white)``
    (float64 CUDA tensors of the batch shape) replaces the generator -- with the reference's own draws the output is
    bit-identical to the reference's."""

    def __init__(self, p=1, noise_density=0.2, salt_ratio=0.1, keyws=("image", "target"), apply_to=(True, False)):
        self.p = p
        self.noise_density = noise_density
        self.salt_ratio = salt_ratio
        self.keyws = keyws
        self.apply_to = apply_to

    def __call__(self, sample, fields=None):
        for i, keyw in enumerate(self.keyws):
            if not self.apply_to[i]:
                continue
            img = sample[keyw]
            _need_cuda(img, "SaltAndPepper")
            is_batch = img.dim() == 4
            vols = (img if is_batch else img.unsqueeze(0)).to(torch.uint8).contiguous()   # .astype(np.uint8), :29-30
            out = vols.clone()
            self.noise_density = np.random.uniform(0, self.noise_density)                # :31
            for j in range(vols.shape[0]):
                r = random.uniform(0, 1)                                                  # :33
                if self.p >= r:
                    ub = uw = None
                    seed = 0
                    if fields is not None:
                        ub = (fields[0] if is_batch else fields[0].unsqueeze(0))[j].contiguous()
                        uw = (fields[1] if is_batch else fields[1].unsqueeze(0))[j].contiguous()
                        if ub.dtype != torch.float64 or uw.dtype != torch.float64 or ub.shape != vols[j].shape:
                            raise TypeError("fields: two float64 CUDA tensors of the image shape")
                    else:
                        seed = int(np.random.randint(0, 2 ** 31 - 1)) | (int(np.random.randint(0, 2 ** 31 - 1)) << 32)
                    call("ctu_salt_pepper_u8", vols[j].data_ptr(), out[j].data_ptr(), vols[j].numel(),
                         float(self.noise_density), float(self.salt_ratio), ub.data_ptr() if ub is not None else None,
                         uw.data_ptr() if uw is not None else None, seed, 0, stream_ptr())
            out = out.float()
            sample[keyw] = out if is_batch else out[0]
        return sample


# ---------------------------------------------------------------------------------------------- RandomAffine
AFFINE_DOMAIN = 0xAFF1            # engine.philox_key domain of the affine draws (Dropout3d uses 0)
AFFINE_PARAM_KEYS = ("angle_d", "angle_h", "angle_w", "scale", "shift_z", "shift_y", "shift_x", "flip_z", "flip_y", "flip_x")


def _triple(v, what):
    t = tuple(v) if isinstance(v, (tuple, list)) else (v, v, v)
    if len(t) != 3 or not all(_number(x) and math.isfinite(x) for x in t):
        raise ValueError("%s must be a finite number or a (d, h, w) triple, got %r" % (what, v))
    return tuple(float(x) for x in t)


def _mask_batch(masks, what):
    """Validate a list of 1..3 uint8 / bool CUDA masks of one [B, D, H, W] shape (errors before any launch)."""
    if not isinstance(masks, (tuple, list)) or not 1 <= len(masks) <= 3:
        raise ValueError("%s expects a list of 1 to 3 masks" % what)
    for m in masks:
        if not isinstance(m, torch.Tensor):
            raise TypeError("%s expects tensors, got %s" % (what, type(m).__name__))
        if m.dim() != 4 or m.shape != masks[0].shape:
            raise ValueError("%s expects masks of one [B, D, H, W] shape, got %s" % (what, [tuple(t.shape) for t in masks]))
        if m.dtype not in (torch.uint8, torch.bool):
            raise TypeError("%s expects uint8 or bool masks, got %s" % (what, m.dtype))
    for m in masks:
        if not m.is_cuda or m.device != masks[0].device:
            raise RuntimeError("%s runs on CUDA tensors of one device only (no CPU fallback)" % what)


def _check_matrices(matrices, batch, device, what):
    if not isinstance(matrices, torch.Tensor) or matrices.dtype != torch.float32 or tuple(matrices.shape) != (batch, 3, 4):
        raise ValueError("%s: matrices must be a float32 [%d, 3, 4] tensor, got %s" % (
            what, batch, (matrices.dtype, tuple(matrices.shape)) if isinstance(matrices, torch.Tensor) else type(matrices)))
    if not matrices.is_cuda or matrices.device != device:
        raise RuntimeError("%s: the matrices must be on the masks' device %s" % (what, device))


def affine_masks(masks, matrices):
    """Transform 1 to 3 uint8 or bool CUDA masks [B, D, H, W] of one shape with the per-sample affine maps ``matrices``
    (float32 [B, 3, 4], e.g. ``RandomAffine.draw``): nearest neighbour, a source outside the volume reads 0, every mask of
    a sample takes the same source voxel (DESIGN.md section 7e).  Returns new masks of the input dtype and shape.  The
    matrix values are not checked (that would synchronise): a non-finite source coordinate reads 0."""
    _mask_batch(masks, "affine_masks")
    b, d, h, w = masks[0].shape
    _check_matrices(matrices, b, masks[0].device, "affine_masks")
    src = [m.contiguous() for m in masks]
    out = [torch.empty_like(m) for m in src]
    u8 = lambda t: t.view(torch.uint8)          # noqa: E731  (bool is one byte of 0 / 1)
    call("ctu_affine_masks_u8", len(src), ptr_array([u8(t).data_ptr() for t in src]),
         ptr_array([u8(t).data_ptr() for t in out]), matrices.contiguous().data_ptr(), b, d, h, w, stream_ptr())
    return out


class RandomAffine(object):
    """Random rotation, isotropic scaling, translation and flips of training masks on the device (DESIGN.md section 7e).

    ``rotate``: degrees, a number or a (d, h, w) triple; the angle about each axis is uniform in [-r, r], 0 <= r <= 180.
    ``scale``: (lo, hi), the scale is uniform in [lo, hi].  ``translate``: voxels, a number or a (z, y, x) triple; uniform
    in [-T, T].  ``flip``: per axis (d, h, w), an enabled axis flips with probability 1/2 (default: left-right only, the one
    symmetry of a skull).  ``RandomAffine(0, (1, 1), 0, (False, False, False))`` is the identity.

    Each sample's map sends output voxel p to source q = c + t + (1/s) R F (p - c) about the volume centre c, sampled with
    nearest neighbour, so binary masks stay binary and ``broken & flap == 0``, ``broken | flap == full`` are kept exactly.
    The draws come from a Philox stream on the device (``ctu_affine_draw``): the key is ``torch.initial_seed()`` when the
    transform first draws on a device, mixed with the device index, the ``torch.distributed`` rank and a constant of its
    own (``engine.philox_key``); the pass counter lives in device memory and each draw advances it.
    ``torch.manual_seed(s)`` before the first draw reproduces a run, ranks draw independent transforms.

    ``__call__(sample)`` takes the dict of ``SkullRandomHole`` (uint8 / bool CUDA ``image`` [B, D, H, W] or [D, H, W], a
    mask or a tuple of masks as ``target``), so ``RandomAffine()(SkullRandomHole(double_output=True)(s))`` composes.  The
    atlas channel of a shape-prior model is NOT transformed: it is the fixed prior in atlas space, and the misregistration
    between it and the skull is what the augmentation simulates (``TrainStep(augment=...)`` leaves it as it is)."""

    def __init__(self, rotate=15.0, scale=(0.9, 1.1), translate=8.0, flip=(False, False, True)):
        rot = _triple(rotate, "rotate")
        if not all(0 <= r <= 180 for r in rot):
            raise ValueError("rotate must be in [0, 180] degrees, got %r" % (rotate,))
        if not isinstance(scale, (tuple, list)) or len(scale) != 2 or not all(_number(x) and math.isfinite(x) for x in scale) \
                or not 0 < scale[0] <= scale[1] <= 1000:
            raise ValueError("scale must be (lo, hi) with 0 < lo <= hi <= 1000, got %r" % (scale,))
        tr = _triple(translate, "translate")
        if not all(0 <= t <= 1e6 for t in tr):
            raise ValueError("translate must be in [0, 1e6] voxels, got %r" % (translate,))
        if not isinstance(flip, (tuple, list)) or len(flip) != 3 or not all(isinstance(f, (bool, np.bool_)) for f in flip):
            raise ValueError("flip must be three booleans (d, h, w), got %r" % (flip,))
        self.rotate, self.scale, self.translate, self.flip = rot, (float(scale[0]), float(scale[1])), tr, tuple(map(bool, flip))
        # float32 ranges the kernel reads: angles in radians, rounded once
        self._ranges = [float(np.float32(math.radians(r))) for r in rot] + [float(np.float32(x)) for x in self.scale] + \
                       [float(np.float32(t)) for t in tr]
        self._flip_axes = sum(1 << k for k, f in enumerate(self.flip) if f)
        self._state = {}                   # device -> (key, int64 pass counter on the device)
        self.last = None                   # (params [B, 10], matrices [B, 3, 4]) of the latest draw

    def draw(self, batch: int, vol_shape, device):
        """Draw one transform per sample: ``(params, matrices)`` float32 CUDA tensors [B, 10] (angles about d, h, w in
        radians, scale, shifts along z, y, x in voxels, flip signs) and [B, 3, 4].  No host synchronisation."""
        d, h, w = (int(v) for v in vol_shape)
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("RandomAffine draws on CUDA devices only (no CPU fallback)")
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        st = self._state.get(device)
        if st is None:
            from .engine import philox_key
            st = self._state[device] = (philox_key(device, AFFINE_DOMAIN), torch.zeros(1, dtype=torch.int64, device=device))
        params = torch.empty((batch, 10), dtype=torch.float32, device=device)
        mats = torch.empty((batch, 3, 4), dtype=torch.float32, device=device)
        with torch.cuda.device(device):
            call("ctu_affine_draw", int(batch), d, h, w, (ctypes.c_float * 8)(*self._ranges), self._flip_axes, st[0],
                 st[1].data_ptr(), params.data_ptr(), mats.data_ptr(), stream_ptr())
        self.last = (params, mats)
        return self.last

    def __call__(self, sample):
        img = sample["image"]
        if not isinstance(img, torch.Tensor) or img.dtype not in (torch.uint8, torch.bool):
            raise ValueError("RandomAffine transforms binary masks (uint8 / bool): encode float images after it")
        tgt = sample.get("target")
        tgts = list(tgt) if isinstance(tgt, (tuple, list)) else ([] if tgt is None else [tgt])
        vols = [img] + tgts
        is_batch = img.dim() == 4
        if any(not isinstance(t, torch.Tensor) or t.dim() != img.dim() for t in vols) or img.dim() not in (3, 4):
            raise ValueError("RandomAffine expects [D, H, W] or [B, D, H, W] masks of one shape")
        batch = [t if is_batch else t.unsqueeze(0) for t in vols]
        _mask_batch(batch, "RandomAffine")
        _, mats = self.draw(batch[0].shape[0], batch[0].shape[1:], batch[0].device)
        out = affine_masks(batch, mats)
        if not is_batch:
            out = [t[0] for t in out]
        res = dict(sample)
        res["image"] = out[0]
        if isinstance(tgt, (tuple, list)):
            res["target"] = type(tgt)(out[1:])
        elif tgt is not None:
            res["target"] = out[1]
        return res


# ---------------------------------------------------------------------------------------------- RandomCraniectomy
CRANIECTOMY_DOMAIN = 0xC4A1       # engine.philox_key domain of the craniectomy draws
CRANIECTOMY_PARAM_KEYS = ("applied", "shape", "radius", "c_diam", "z", "y", "x")


class RandomCraniectomy(object):
    """The virtual craniectomy drawn and cut on the device (DESIGN.md section 7f): per sample the distribution of
    ``random_blank_patch(full, p, True, p_type="random", valid_shapes=shapes)`` (transforms.py:241-300) -- a gate
    ``u <= p``, a centre uniform over the skull's bone voxels, an integer radius uniform in ``radius_bounds``, a shape
    uniform over ``shapes`` (sphere, box, flap) and the flap's cylinder radius -- drawn from a Philox stream on the device
    instead of the host RNGs, so nothing synchronises with the host.  ``random_blank_patch`` / ``SkullRandomHole`` replay
    the reference's host draws; this transform has the same distribution, not the same stream.

    The key is ``engine.philox_key(device, CRANIECTOMY_DOMAIN)`` when the transform first draws on a device and the pass
    counter lives in device memory (as ``RandomAffine``): ``torch.manual_seed(s)`` before the first draw reproduces a run.

    ``__call__(sample)`` is the sync-free twin of ``SkullRandomHole(p, double_output=True)``: a uint8 / bool CUDA
    ``image`` [B, D, H, W] or [D, H, W] (the full skull, non-zero is bone) gives ``{"image": broken, "target": (full,
    flap)}`` as uint8, with ``broken & flap == 0`` and ``broken | flap == full``; ``RandomAffine()(RandomCraniectomy()(s))``
    composes.  ``TrainStep(craniectomy=...)`` fuses the cut into the batch encoding of the training step."""

    def __init__(self, p=1.0, shapes=("sphere", "box", "flap")):
        if not _number(p) or not 0 <= p <= 1:
            raise ValueError("p must be in [0, 1], got %r" % (p,))
        if isinstance(shapes, str) or not isinstance(shapes, (tuple, list)) or not shapes or \
                not all(isinstance(s, str) and s in _SHAPES for s in shapes):
            raise ValueError("shapes: a non-empty list of 'sphere', 'box', 'flap', got %r" % (shapes,))
        self.p = float(p)
        self.shapes = tuple(shapes)
        self._shape_bits = sum({1 << _SHAPES[s] for s in shapes})
        self._state = {}                   # device -> (key, int64 pass counter on the device)
        self.last = None                   # params [B, 7] of the latest draw

    def _full(self, full, vol_shape):
        """Validate the full skulls (errors before any launch) -> (bits, contiguous tensor, batch, (d, h, w), radius range)."""
        if not isinstance(full, torch.Tensor):
            raise TypeError("RandomCraniectomy expects a tensor, got %s" % type(full).__name__)
        if vol_shape is None:
            if full.dtype not in (torch.uint8, torch.bool):
                raise TypeError("RandomCraniectomy expects uint8 or bool skull masks, got %s" % full.dtype)
            if full.dim() not in (3, 4):
                raise ValueError("RandomCraniectomy expects [B, D, H, W] or [D, H, W] masks, got %s" % (tuple(full.shape),))
            bits, vol = 0, tuple(int(v) for v in full.shape[-3:])
            batch = full.shape[0] if full.dim() == 4 else 1
        else:
            vol = tuple(int(v) for v in vol_shape)
            if len(vol) != 3:
                raise ValueError("vol_shape: (D, H, W)")
            if full.dtype != torch.uint8 or full.dim() != 2 or full.shape[1] * 8 != vol[0] * vol[1] * vol[2]:
                raise ValueError("bit-packed skulls: uint8 [B, D*H*W/8] of the volume shape %s, got %s %s"
                                 % (vol, full.dtype, tuple(full.shape)))
            bits, batch = 1, full.shape[0]
        if not 1 <= batch <= 65535 or not all(1 <= v <= 16384 for v in vol):
            raise ValueError("RandomCraniectomy: batch 1..65535 and axes 1..16384, got %d x %s" % (batch, vol))
        min_r, max_r = (int(r) for r in radius_bounds(vol))
        if min_r >= max_r:                 # np.random.randint(min_r, max_r) raises in the reference
            raise ValueError("the radius range [%d, %d) of a %s volume is empty" % (min_r, max_r, vol))
        if not full.is_cuda:
            raise RuntimeError("RandomCraniectomy runs on CUDA tensors only (no CPU fallback)")
        return bits, full.contiguous(), batch, vol, (min_r, max_r)

    def draw(self, full: torch.Tensor, vol_shape=None) -> torch.Tensor:
        """Draw one hole per sample of ``full`` (uint8 / bool [B, D, H, W] or [D, H, W]; with ``vol_shape`` bit-packed
        [B, D*H*W/8], ``pack_mask_bits``): float64 CUDA params [B, 7] = ``CRANIECTOMY_PARAM_KEYS`` (applied 0 / 1, shape
        0 sphere / 1 box / 2 flap, radius, c_diam (flap; 0 otherwise), the centre voxel z, y, x (-1 when not applied)).
        No host synchronisation."""
        bits, src, batch, vol, (min_r, max_r) = self._full(full, vol_shape)
        device = src.device
        st = self._state.get(device)
        if st is None:
            from .engine import philox_key
            st = self._state[device] = (philox_key(device, CRANIECTOMY_DOMAIN), torch.zeros(1, dtype=torch.int64, device=device))
        with torch.cuda.device(device):
            nbytes = _load().ctu_craniectomy_workspace_bytes(batch, *vol)
            ws = torch.empty(nbytes, dtype=torch.uint8, device=device)
            params = torch.empty((batch, 7), dtype=torch.float64, device=device)
            call("ctu_craniectomy_draw", bits, src.data_ptr(), batch, *vol, self.p, self._shape_bits, min_r, max_r, st[0],
                 st[1].data_ptr(), params.data_ptr(), ws.data_ptr(), nbytes, stream_ptr())
        self.last = params
        return params

    def __call__(self, sample):
        img = sample["image"]
        _, full, batch, vol, _ = self._full(img, None)
        params = self.draw(full)
        u8 = full.view(torch.uint8) if full.dtype == torch.bool else full      # bool is one byte of 0 / 1
        out = [torch.empty(u8.shape, dtype=torch.uint8, device=u8.device) for _ in range(3)]
        with torch.cuda.device(u8.device):
            call("ctu_craniectomy_masks_u8", u8.data_ptr(), params.data_ptr(), *[t.data_ptr() for t in out], batch, *vol,
                 stream_ptr())
        res = dict(sample)
        res["image"], res["target"] = out[0], (out[1], out[2])
        return res
