"""Synthetic skull-CT training data generated on the GPU (SURVEY.md section 8d): an ellipsoidal bone
shell phantom, a seeded virtual craniectomy through the product's own masking kernels
(transforms.py:241-300 semantics), the atlas stand-in channel (datasets.py:30-47) and one-hot float32
targets (datasets.py:209-214).  Used by bench.py and the examples; there are no real datasets here."""
from __future__ import annotations

import random

import numpy as np
import torch

from .utilities import random_blank_patch


def skull_phantom(size: int, seed: int, device) -> torch.Tensor:
    """uint8 [S,S,S] binary skull: ellipsoidal shell, thickness ~4.5 voxels at 128^3."""
    g = torch.Generator().manual_seed(seed)
    jit = (0.03 * torch.rand(3, generator=g)).tolist()
    lin = torch.linspace(-1, 1, size, device=device)
    zz, yy, xx = torch.meshgrid(lin, lin, lin, indexing="ij")
    r = torch.sqrt((zz / (0.80 + jit[0])) ** 2 + (yy / (0.88 + jit[1])) ** 2 + (xx / (0.72 + jit[2])) ** 2)
    thick = max(3.0, 4.5 * size / 128.0) / (size / 2.0)
    return ((r >= 1.0 - thick) & (r <= 1.0)).to(torch.uint8)


def head_ct_hu(shape=(256, 512, 512), seed: int = 0, device="cuda") -> torch.Tensor:
    """int16 HU head CT: the phantom of scripts/bench_infer.py (brain at 40 HU in an ellipsoidal 1000 HU bone shell,
    Gaussian noise of 30 HU) plus what a bone threshold of a real scan also keeps: a scanner-table slab under the head
    (600 HU, not touching it) and sparse metal speckle (1500 HU, about one voxel in 10^4).  Thresholded at 300 HU it
    holds one large component (the skull), one slab and thousands of islands."""
    d, h, w = shape
    g = torch.Generator(device=device).manual_seed(seed)
    zz, yy, xx = torch.meshgrid(*[torch.linspace(-1, 1, n, device=device) for n in (d, h, w)], indexing="ij")
    r = torch.sqrt((zz / 0.8) ** 2 + (yy / 0.88) ** 2 + (xx / 0.72) ** 2)
    hu = torch.full(shape, -1000.0, device=device)
    hu[r <= 1.0] = 40
    hu[(r >= 0.93) & (r <= 1.0)] = 1000
    hu[(yy >= 0.95) & (yy <= 0.98) & (xx.abs() <= 0.9)] = 600
    del zz, yy, xx, r
    hu[torch.rand(shape, device=device, generator=g) < 1e-4] = 1500
    return (hu + 30 * torch.randn(shape, device=device, generator=g)).clamp(-1024, 3071).to(torch.int16)


def make_training_batch(batch: int, in_channels: int, size: int, seed: int, device="cuda"):
    """(image [B,Cin,S,S,S] float32 {0,1}, (skull_onehot, flap_onehot) each [B,2,S,S,S] float32)."""
    random.seed(seed)
    np.random.seed(seed)
    atlas = skull_phantom(size, 999, device).float()
    imgs, sks, fls = [], [], []
    for b in range(batch):
        full = skull_phantom(size, seed * 131 + b, device)
        broken, flap = random_blank_patch(full, 1, True)
        chans = [broken.float()]
        if in_channels > 1:
            chans.append(atlas)
        imgs.append(torch.stack(chans, 0))
        sks.append(torch.stack((1 - full, full), 0).float())
        fls.append(torch.stack((1 - flap, flap), 0).float())
    return torch.stack(imgs).contiguous(), (torch.stack(sks).contiguous(), torch.stack(fls).contiguous())
