"""Drop-in for the reference's `rpn_util.py`: RPN training targets on the GPU.

Same call signatures, array layouts and RNG stream as the reference (citations: file:line under
/root/reference/faster_rcnn).  The anchor x GT labelling, the sampling switch-offs and the Keras
`y_true` packing run in libfrcnn_b200.so (label.cu); only the draws of Python's `random` stay
on the host, because bit-exact parity needs the reference's own MT19937 stream in its order.
`RpnTrainingManager.rpn_targets_device` draws with the same rule on the device instead (sample.cu).
"""
import random

import numpy as np
import torch

from . import ops
from .custom_decorators import profile
from .runtime import get_context
from .shared_constants import BBREG_MULTIPLIERS, DEFAULT_ANCHORS  # noqa: F401  (re-exported like the reference)
from .util import get_bbox_coords

POS_OVERLAP = 0.7          # rpn_util.py:11-15; compiled into label.cu as float32 constants
NEG_OVERLAP = 0.3
SAMPLE_SIZE = 256
MAX_POS_SAMPLES = 128


class RpnTrainingManager:
    """Generates RPN training targets for an image (reference: rpn_util.py:24-140)."""

    def __init__(self, calc_conv_dims, stride, preprocess_func, anchor_dims=DEFAULT_ANCHORS):
        self._cache = {}
        self.calc_conv_dims = calc_conv_dims
        self.stride = stride
        self.preprocess_func = preprocess_func
        self.anchor_dims = anchor_dims

    @profile
    def batched_image(self, image):
        """(1,H,W,3) network input (rpn_util.py:45-51)."""
        return np.expand_dims(self.preprocess_func(image.data), axis=0)

    # -- device side ----------------------------------------------------------------------------
    def _label_batch(self, images, extents=None, pad_to=None):
        """Labels a list of images that share one conv shape in a single launch sequence.
        Returns device tensors can_use (B,N) u8, is_pos (B,N) u8, bbreg (B,N,4) f32, counts (B,2).
        With `extents` ((B,2) i32 conv shapes of the images, a host array or a CUDA tensor) the images may differ: they are labelled as one
        batch padded to `pad_to` (rows, cols)."""
        ctx = get_context()
        rows, cols = pad_to if extents is not None else self.calc_conv_dims(images[0].height, images[0].width)
        g_max = max(len(img.gt_boxes) for img in images)
        if g_max == 0:
            raise ValueError("image without ground-truth boxes (the reference fails in np.amax here too)")
        gt = np.zeros((len(images), g_max, 4), dtype=np.float32)
        n_gt = np.zeros(len(images), dtype=np.int32)
        wh = np.zeros((len(images), 2), dtype=np.int32)
        for b, img in enumerate(images):
            if extents is None and tuple(self.calc_conv_dims(img.height, img.width)) != (rows, cols):
                raise ValueError("images of one batch must share the conv feature-map shape")
            if len(img.gt_boxes) == 0:
                raise ValueError("image without ground-truth boxes (the reference fails in np.amax here too)")
            n_gt[b] = len(img.gt_boxes)
            gt[b, :n_gt[b]] = get_bbox_coords(img.gt_boxes)
            wh[b] = img.width, img.height
        if extents is not None and not isinstance(extents, torch.Tensor):
            extents = ctx.to_device(extents)
        return ops.label_anchors(ctx.to_device(gt), ctx.to_device(n_gt), ctx.to_device(wh), rows, cols,
                                 self.anchor_dims, self.stride, extents=extents)

    @profile
    def _process(self, image):
        """Labels before sampling, cached like the reference (rpn_util.py:54-103)."""
        ctx = get_context()
        can_use, is_pos, bbreg, _ = self._label_batch([image])
        self._cache[image.cache_key] = {
            'can_use': ctx.to_host(can_use[0]).view(np.bool_),
            'is_pos': ctx.to_host(is_pos[0]).view(np.bool_),
            'bbreg_targets': ctx.to_host(bbreg[0]),
        }

    @profile
    def rpn_y_true(self, image):
        """(y_class (1,R,C,2A) bool, y_bbreg (1,R,C,8A) f32) for one image (rpn_util.py:106-140).
        The cache entry is consumed, as in the reference."""
        ctx = get_context()
        rows, cols = self.calc_conv_dims(image.height, image.width)
        n_anchors = len(self.anchor_dims)
        if image.cache_key in self._cache:
            res = self._cache.pop(image.cache_key)
            can_use = ctx.to_device(res['can_use'].view(np.uint8))[None]
            is_pos = ctx.to_device(res['is_pos'].view(np.uint8))[None]
            bbreg = ctx.to_device(res['bbreg_targets'])[None]
            counts = _host_counts(res['can_use'], res['is_pos'])
        else:
            can_use, is_pos, bbreg, counts = self._label_batch([image])
            res = None
        y_class, y_bbreg = self._sample_and_pack(can_use, is_pos, bbreg, counts, rows, cols, n_anchors)
        if res is not None:            # the reference mutates the cached can_use in _apply_sampling
            res['can_use'][...] = ctx.to_host(can_use[0]).view(np.bool_)
        return ctx.to_host(y_class).view(np.bool_), ctx.to_host(y_bbreg)

    def rpn_y_true_batch(self, images):
        """Batched variant (not in the reference): list of images with one conv shape ->
        y_class (B,R,C,2A) bool, y_bbreg (B,R,C,8A) f32.  RNG draws happen image by image in list
        order, so the result equals calling `rpn_y_true` on each image in turn."""
        ctx = get_context()
        rows, cols = self.calc_conv_dims(images[0].height, images[0].width)
        can_use, is_pos, bbreg, counts = self._label_batch(images)
        y_class, y_bbreg = self._sample_and_pack(can_use, is_pos, bbreg, counts, rows, cols, len(self.anchor_dims))
        return ctx.to_host(y_class).view(np.bool_), ctx.to_host(y_bbreg)

    def rpn_y_true_ragged(self, images, pad_to=None):
        """Batched variant for images of different conv shapes (not in the reference): list of images ->
        y_class (B,R,C,2A) bool, y_bbreg (B,R,C,8A) f32, extents (B,2) i32 (each image's conv rows, cols).  (R, C) are the
        largest conv shape of the batch or `pad_to`.  Image b's targets are y_class[b, :rows_b, :cols_b] (and the same of
        y_bbreg); the padding is zero, i.e. unusable anchors.  RNG draws happen image by image in list order, so the result
        equals calling `rpn_y_true` on each image in turn."""
        ctx = get_context()
        extents, rows, cols = self._padded_extents(images, pad_to)
        can_use, is_pos, bbreg, counts = self._label_batch(images, extents, (rows, cols))
        y_class, y_bbreg = self._sample_and_pack(can_use, is_pos, bbreg, counts, rows, cols, len(self.anchor_dims))
        return ctx.to_host(y_class).view(np.bool_), ctx.to_host(y_bbreg), extents

    def rpn_targets_device(self, images, state, pad_to=None):
        """RPN targets drawn on the device (not in the reference): list of images (any conv shapes) + the RNG state of
        ops.sampler_state -> can_use (B,N) u8, is_pos (B,N) u8, bbreg (B,N,4) f32, extents (B,2) i32, all CUDA tensors
        in the padded (R,C,A) layout of the largest conv shape or `pad_to`: exactly the inputs of
        loss_functions.rpn_losses(..., extents=extents, padded_shape=(R, C)).  The 256-anchor mini-batch follows the
        reference's rule with the counter-based RNG (ops.sample_rpn_), so nothing returns to the host; image b's draw
        depends on (seed, offset + b) only, and state's offset advances by B."""
        ext, rows, cols = self._padded_extents(images, pad_to)
        extents = get_context().to_device(ext)
        can_use, is_pos, bbreg, counts = self._label_batch(images, extents, (rows, cols))
        ops.sample_rpn_(can_use, is_pos, counts, state, extents=extents, padded_shape=(rows, cols),
                        n_anchors=len(self.anchor_dims), max_pos=MAX_POS_SAMPLES, sample_size=SAMPLE_SIZE)
        return can_use, is_pos, bbreg, extents

    def _padded_extents(self, images, pad_to):
        """(B,2) i32 host array of the images' conv shapes and the padded (rows, cols): the largest of them or `pad_to`"""
        extents = np.array([tuple(self.calc_conv_dims(img.height, img.width)) for img in images], np.int32).reshape(-1, 2)
        rows, cols = (int(v) for v in extents.max(axis=0))
        if pad_to is not None:
            if pad_to[0] < rows or pad_to[1] < cols:
                raise ValueError("pad_to %s is smaller than the largest conv shape (%d, %d)" % (tuple(pad_to), rows, cols))
            rows, cols = int(pad_to[0]), int(pad_to[1])
        return extents, rows, cols

    def _sample_and_pack(self, can_use, is_pos, bbreg, counts, rows, cols, n_anchors):
        ctx = get_context()
        if isinstance(counts, torch.Tensor):
            counts = ctx.to_host(counts)                  # (B,2): the only D2H before the final targets
        off_pos, off_neg = _draw_switch_offs(counts)
        return ops.pack_rpn_targets(can_use, is_pos, bbreg, rows, cols, n_anchors,
                                    _ranks_to_device(ctx, off_pos), _ranks_to_device(ctx, off_neg))


def _host_counts(can_use, is_pos):
    cu, ip = np.asarray(can_use) == 1, np.asarray(is_pos) == 1
    return np.array([[int(np.count_nonzero(cu & ip)), int(np.count_nonzero(cu & ~ip))]])


def _draw_switch_offs(counts):
    """Replays the RNG calls of _apply_sampling (rpn_util.py:338-348) for every image, in order."""
    off_pos, off_neg = [], []
    for num_pos, num_neg in counts.tolist():
        p, q = [], []
        if num_pos > MAX_POS_SAMPLES:
            p = random.sample(range(num_pos), num_pos - MAX_POS_SAMPLES)
            num_pos = MAX_POS_SAMPLES
        if num_neg + num_pos > SAMPLE_SIZE:
            q = random.sample(range(num_neg), num_neg + num_pos - SAMPLE_SIZE)
        off_pos.append(p)
        off_neg.append(q)
    return off_pos, off_neg


def _ranks_to_device(ctx, per_image):
    total = sum(len(r) for r in per_image)
    if total == 0:
        return None
    offsets = np.zeros(len(per_image) + 1, dtype=np.int32)
    offsets[1:] = np.cumsum([len(r) for r in per_image])
    ranks = np.fromiter((v for r in per_image for v in r), dtype=np.int32, count=total)
    return ctx.to_device(ranks), ctx.to_device(offsets)


# ---- module-level helpers with the reference's names ------------------------------------------
def _idx_to_conv(idx, conv_width, anchors_per_loc):
    """flat anchor index -> (row, col, anchor) (rpn_util.py:143-156)."""
    y, rem = divmod(idx, conv_width * anchors_per_loc)
    x, anchor_idx = divmod(rem, anchors_per_loc)
    return y, x, anchor_idx


def _get_conv_center(conv_x, conv_y, stride):
    """pixel centre of a conv cell (rpn_util.py:169-180)."""
    return int(stride * (conv_x + 0.5)), int(stride * (conv_y + 0.5))


@profile
def _get_all_anchor_coords(conv_rows, conv_cols, anchor_dims, stride):
    """(N,4) f32 pixel-space anchors, generated on the GPU (rpn_util.py:276-298)."""
    ctx = get_context()
    return ctx.to_host(ops.anchor_grid(anchor_dims, conv_rows, conv_cols, stride, pixel_space=True))


@profile
def _get_out_of_bounds_idxs(anchor_coords, img_width, img_height):
    """indices of anchors crossing the image border (rpn_util.py:302-310)."""
    a = anchor_coords
    return np.where((a[:, 0] < 0) | (a[:, 1] < 0) | (a[:, 2] >= img_width) | (a[:, 3] >= img_height))[0]


@profile
def _apply_sampling(is_pos, can_use):
    """256-anchor mini-batch balancing; mutates and returns `can_use` (rpn_util.py:324-350)."""
    ctx = get_context()
    cu_host, ip_host = np.asarray(can_use) == 1, np.asarray(is_pos) == 1
    off_pos, off_neg = _draw_switch_offs(_host_counts(cu_host, ip_host))
    cu = ctx.to_device(cu_host.view(np.uint8))[None]
    ip = ctx.to_device(ip_host.view(np.uint8))[None]
    n = cu.shape[1]
    scratch = ctx.empty((1, n, 4), torch.float32)
    ops.pack_rpn_targets(cu, ip, scratch, 1, n, 1, _ranks_to_device(ctx, off_pos), _ranks_to_device(ctx, off_neg))
    can_use[cu_host & (ctx.to_host(cu[0]) == 0)] = 0
    return can_use
