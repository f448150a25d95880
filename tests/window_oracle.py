"""TEST INFRASTRUCTURE ONLY -- the CPU oracle of overlapping sliding-window inference (preprocess.sliding_window_predict).

Written from the semantics in DESIGN.md section 7b, independently of the product's helpers:
  * per axis of size S, patch p: step = max(1, floor(p (1 - overlap))); S <= p -> one origin 0; otherwise
    ceil((S - p) / step) + 1 origins min(i step, S - p); windows = z-major product of the three lists;
  * separable weights: "constant" 1, "gaussian" max(g / max g, 2^-6) with g(t) = exp(-(t - (p-1)/2)^2 / (2 sigma^2)),
    sigma = sigma_scale p;
  * each window: ``oracle.unet_oracle.unet_forward`` in eval mode on the zero-padded window, outputs past the volume dropped;
  * blended value = sum(w v) / sum(w) in float64; label = argmax over the channels, first maximum wins.
"""
import math

import torch
import torch.nn.functional as F

from oracle import unet_oracle as O


def axis_origins(size, patch, overlap):
    step = max(1, int(math.floor(patch * (1.0 - overlap))))
    if size <= patch:
        return [0]
    out, i = [], 0
    while True:
        o = i * step
        if o + patch >= size:
            out.append(size - patch)
            return out
        out.append(o)
        i += 1


def axis_weights(patch, blend, sigma_scale=0.125):
    if blend == "constant":
        return [1.0] * patch
    sigma = sigma_scale * patch
    c = (patch - 1) / 2.0
    g = [math.exp(-((t - c) ** 2) / (2.0 * sigma ** 2)) for t in range(patch)]
    peak = max(g)
    return [max(v / peak, 2.0 ** -6) for v in g]


def axis_normaliser(size, patch, origins, weights):
    n = [0.0] * size
    for o in origins:
        for t in range(patch):
            if o + t < size:
                n[o + t] += weights[t]
    return n


def predict(sd, cfg, vol, patch, overlap, blend, sigma_scale=0.125, batch=4):
    """vol: CPU float32 [Cin, D, H, W].  Returns (blended float64 [C, D, H, W] per output, float32 labels [D, H, W] per
    output, the window list)."""
    cin, d, h, w = vol.shape
    axes = [axis_origins(s, patch, overlap) for s in (d, h, w)]
    wins = [(z, y, x) for z in axes[0] for y in axes[1] for x in axes[2]]
    wt = torch.tensor(axis_weights(patch, blend, sigma_scale), dtype=torch.float64)
    w3 = wt.view(-1, 1, 1) * wt.view(1, -1, 1) * wt.view(1, 1, -1)
    pad = [max(o + patch for o in a) - s for a, s in zip(axes, (d, h, w))]
    vp = F.pad(vol, (0, pad[2], 0, pad[1], 0, pad[0]))
    acc = None
    for i in range(0, len(wins), batch):
        chunk = wins[i:i + batch]
        xb = torch.stack([vp[:, z:z + patch, y:y + patch, x:x + patch] for z, y, x in chunk])
        with torch.no_grad():
            out = O.unet_forward(sd, xb, cfg, training=False)
        out = out if isinstance(out, tuple) else (out,)
        if acc is None:
            acc = [torch.zeros((o.shape[1], d, h, w), dtype=torch.float64) for o in out]
        for k, o in enumerate(out):
            for j, (z, y, x) in enumerate(chunk):
                dz, dy, dx = min(patch, d - z), min(patch, h - y), min(patch, w - x)
                acc[k][:, z:z + dz, y:y + dy, x:x + dx] += (o[j].double() * w3)[:, :dz, :dy, :dx]
    nz, ny, nx = (torch.tensor(axis_normaliser(s, patch, a, wt.tolist()), dtype=torch.float64)
                  for s, a in zip((d, h, w), axes))
    norm = nz.view(-1, 1, 1) * ny.view(1, -1, 1) * nx.view(1, 1, -1)
    blended = [a / norm for a in acc]
    labels = [O.hard_segm_from_tensor(b) for b in blended]
    return blended, labels, wins


def margin(blended):
    """Per voxel: the gap between the largest and the second-largest channel (the label's distance from a tie)."""
    top = blended.topk(2, dim=0).values if blended.shape[0] > 1 else torch.cat((blended, blended - 1))
    return top[0] - top[1]
