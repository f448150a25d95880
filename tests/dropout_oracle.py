"""TEST INFRASTRUCTURE ONLY -- the CPU oracle (oracle/unet_oracle.py) with given Dropout3d masks.

``nn.Dropout3d(dropout_p)`` ends every block of the reference (models.py:34,46,411,438,492), right after the block's second
BatchNorm+ReLU.  ``unet_forward(..., dropout_keep=...)`` runs ``oracle.unet_oracle.unet_forward`` unchanged except at those
stages, where the caller's [N, C] keep factors (the masks a Dropout3d drew: 0 or 1/(1-p) per sample and channel) multiply
the ReLU output before the activation is stored (rounded once, as the product's kernels do).  The masks are keyed by the
Dropout3d module name, e.g. ``d_blocks.0.block.6``, ``u_blocks.3.block.7``, ``dblock2.6``, ``cblock_center.6``,
``ublock1.7`` -- the keys of ``net.dropout_keep()``.  Absent sites are the identity (dropout_p = 0 or eval mode)."""
import contextlib

import torch.nn.functional as F

from oracle import unet_oracle as O

# index of the second BatchNorm of a block -> index of the Dropout3d that follows it (down block / center: Conv, BN, ReLU,
# Conv, BN, ReLU, Dropout3d; up block: ConvTranspose3d first)
_SITE_OF_BN = {"4": "6", "5": "7"}


@contextlib.contextmanager
def _with_masks(keep):
    orig = O._bn_relu

    def bn_relu(sd, prefix, y, training, n_updates):
        base, idx = prefix.rsplit(".", 1)
        k = keep.get(base + "." + _SITE_OF_BN[idx]) if idx in _SITE_OF_BN else None
        if k is None:
            return orig(sd, prefix, y, training, n_updates)
        # O._bn_relu restated, with the keep factor applied before the storage rounding
        w, b = sd[prefix + ".weight"], sd[prefix + ".bias"]
        rm, rv = sd[prefix + ".running_mean"], sd[prefix + ".running_var"]
        if training:
            out = F.batch_norm(y, rm, rv, w, b, True, O.BN_MOMENTUM, O.BN_EPS)
            sd[prefix + ".num_batches_tracked"] += 1
            for _ in range(n_updates - 1):
                with O.torch.no_grad():
                    F.batch_norm(y.detach(), rm, rv, None, None, True, O.BN_MOMENTUM, O.BN_EPS)
                sd[prefix + ".num_batches_tracked"] += 1
        else:
            out = F.batch_norm(y, rm, rv, w, b, False, O.BN_MOMENTUM, O.BN_EPS)
        return O._store(F.relu(out) * k.to(out.dtype)[:, :, None, None, None])

    O._bn_relu = bn_relu
    try:
        yield
    finally:
        O._bn_relu = orig


def unet_forward(sd, x, cfg, training=False, dropout_keep=None, **kw):
    """``oracle.unet_oracle.unet_forward`` with the Dropout3d masks ``dropout_keep`` ({module name: [N, C]})."""
    if not dropout_keep:
        return O.unet_forward(sd, x, cfg, training, **kw)
    with _with_masks(dict(dropout_keep)):
        return O.unet_forward(sd, x, cfg, training, **kw)
