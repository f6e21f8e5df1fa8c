"""Drop-in for `custom_layers.RoiResizeConv` (reference: custom_layers.py:7-56).

The reference layer crops `img[:, y1:y2, x1:x2, :]` per RoI and bilinearly resizes the crop to
pool_size x pool_size with TF-1.3's legacy kernel (`align_corners=False`, no half-pixel
offset); there is no max pooling in it.  `mode="resize"` (default) reproduces that; `mode="max"`
is the max-pool variant specified in oracle/roi_oracle.py.  Forward and backward are the K-d
kernels of roi.cu; gradients flow to the feature map only (none to the RoIs, as in TF).

Keras / TensorFlow are not importable in this image, so the class mirrors the Keras layer
interface (`build`, `compute_output_shape`, `get_config`, `call`, `__call__`) without
subclassing it; tensors are numpy arrays (returned as numpy) or CUDA torch tensors (returned as
torch, differentiable through `torch.autograd`).  INTEGRATION.md shows the Keras-side binding.
"""
import numpy as np
import torch

from . import ops
from .runtime import get_context


class _RoiFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feat, rois, pool, mode):
        feat = feat.contiguous()
        if mode == "max":
            # the arg-max only feeds the backward: take the one-byte format whenever the bins allow it
            compact = rois.shape[1] < 65536 and ops.roi_compact_supported(feat.shape[1], feat.shape[2], feat.shape[3], pool)
            out, argmax = ops.roi_forward(feat, rois, pool, "max", compact=compact)
        else:
            out, argmax = ops.roi_forward(feat, rois, pool, "resize"), None
        ctx.mode, ctx.feat_shape = mode, tuple(feat.shape)
        if argmax is not None:
            ctx.save_for_backward(rois, argmax)
        else:
            ctx.save_for_backward(rois)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        saved = ctx.saved_tensors
        rois, argmax = saved[0], (saved[1] if len(saved) > 1 else None)
        grad_feat = ops.roi_backward(grad_out.contiguous(), rois, ctx.feat_shape, ctx.mode, argmax)
        return grad_feat, None, None, None


def roi_pool(feat, rois, pool_size, mode="resize", extents=None):
    """feat (B,H,W,C) f32 CUDA tensor, rois (B,N,4) int16/int32/float32 CUDA tensor (feature cells,
    x2/y2 excluded from the crop) -> (B,N,P,P,C) f32, differentiable w.r.t. feat.
    `extents` (B,2) i32 (rows, cols) on the device: feat is a padded batch of differently sized maps (ops.pad_batch);
    the RoIs are clamped to each image's own map first, so every image pools as on its own map and the gradient of the
    padding is zero."""
    if extents is not None:
        rois = ops.clip_rois(rois, extents)
    return _RoiFunction.apply(feat, rois, int(pool_size), mode)


class RoiResizeConv:
    """Region-of-interest layer: crop + bilinear resize to pool_size^2 (or max pool)."""

    def __init__(self, pool_size, num_rois, mode="resize", **kwargs):
        if mode not in ("resize", "max"):
            raise ValueError("mode must be 'resize' or 'max'")
        self.pool_size = pool_size
        self.num_rois = num_rois
        self.mode = mode
        self.name = kwargs.pop("name", "roi_resize_conv")
        self.trainable = kwargs.pop("trainable", True)
        self.built = False
        self.nb_channels = None

    def build(self, input_shape):
        self.nb_channels = input_shape[0][3]
        self.built = True

    def compute_output_shape(self, input_shape):
        return None, self.num_rois, self.pool_size, self.pool_size, self.nb_channels

    def get_config(self):
        config = {'pool_size': self.pool_size, 'num_rois': self.num_rois}
        if self.mode != "resize":
            config['mode'] = self.mode
        return config

    @classmethod
    def from_config(cls, config):
        return cls(**config)

    def call(self, x, mask=None):
        img, rois = x[0], x[1]
        as_numpy = not isinstance(img, torch.Tensor)
        ctx = get_context(None if as_numpy else img.device)
        if as_numpy:
            img = ctx.to_device(img, np.float32)
        if not isinstance(rois, torch.Tensor):
            rois = np.asarray(rois)
            if rois.dtype not in (np.int16, np.int32, np.float32):
                rois = rois.astype(np.float32 if rois.dtype.kind == 'f' else np.int32)
            rois = ctx.to_device(rois)
        if rois.shape[1] != self.num_rois:
            raise ValueError("expected %d rois, got %d" % (self.num_rois, rois.shape[1]))
        if img.shape[0] != rois.shape[0]:
            raise ValueError("img and rois must have the same batch size")
        out = roi_pool(img, rois, self.pool_size, self.mode)
        return ctx.to_host(out) if as_numpy else out

    def __call__(self, x, **kwargs):
        if not self.built:
            self.build([tuple(x[0].shape), tuple(x[1].shape)])
        return self.call(x, **kwargs)
