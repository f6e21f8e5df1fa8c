"""Drop-in for the reference's `loss_functions.py` (loss_functions.py:15-76), a widening row of the hot path
(SURVEY.md 8f-2): the masked RPN / detector losses evaluated by fused CUDA kernels (csrc/losses.cu) directly on
the targets the path produces.

Two surfaces:
  * the reference's factories `cls_loss_rpn`, `bbreg_loss_rpn`, `bbreg_loss_det`, `cls_loss_det` -- callables
    `(y_true, y_pred) -> float32 scalar` on numpy arrays in the Keras layouts (what Keras would report for that
    output, i.e. the mean of the loss tensor);
  * `rpn_losses` / `det_losses` -- differentiable torch functions on CUDA tensors that take the UNPACKED labels,
    so the `y_true` tensors never have to be built.
"""
import numpy as np
import torch

from . import ops
from .runtime import get_context
from .shared_constants import DEFAULT_ANCHORS_PER_LOC

N_CLS = 256            # loss_functions.py:8-12
N_REG = 2400
LAMBDA_REG = 10.0
LAMBDA_REG_DET = 1


class _RpnLosses(torch.autograd.Function):
    @staticmethod
    def forward(ctx, cls_pred, reg_pred, can_use, is_pos, bbreg, extents, padded_shape):
        loss, g_cls, g_reg = ops.rpn_losses(can_use, is_pos, bbreg, cls_pred.contiguous(), reg_pred.contiguous(), want_grad=True,
                                            extents=extents, padded_shape=padded_shape)
        ctx.save_for_backward(g_cls, g_reg)
        return loss

    @staticmethod
    def backward(ctx, grad_loss):
        g_cls, g_reg = ctx.saved_tensors
        return g_cls * grad_loss[:, 0:1], g_reg * grad_loss[:, 1].reshape(-1, 1, 1), None, None, None, None, None


class _DetLosses(torch.autograd.Function):
    @staticmethod
    def forward(ctx, cls_pred, reg_pred, y_class, y_transform):
        loss, g_cls, g_reg = ops.det_losses(y_class, y_transform, cls_pred.contiguous(), reg_pred.contiguous(), want_grad=True)
        ctx.save_for_backward(g_cls, g_reg)
        return loss

    @staticmethod
    def backward(ctx, grad_loss):
        g_cls, g_reg = ctx.saved_tensors
        return g_cls * grad_loss[:, 0].reshape(-1, 1, 1), g_reg * grad_loss[:, 1].reshape(-1, 1, 1), None, None


def rpn_losses(cls_pred, reg_pred, can_use, is_pos, bbreg, extents=None, padded_shape=None):
    """cls_pred (B,N) f32 sigmoid outputs, reg_pred (B,N,4) f32, labels as `ops.label_anchors` emits them ->
    loss (B,2) = (cls_loss_rpn, bbreg_loss_rpn), differentiable w.r.t. the two predictions.  A padded batch of
    differently sized maps passes `extents` and `padded_shape` as `ops.rpn_losses` takes them."""
    return _RpnLosses.apply(cls_pred, reg_pred, can_use, is_pos, bbreg, extents, padded_shape)


def det_losses(cls_pred, reg_pred, y_class_num, y_transform):
    """cls_pred (B,M,K), reg_pred (B,M,4(K-1)), targets as `ops.label_rois` emits them ->
    loss (B,2) = (cls_loss_det, bbreg_loss_det), differentiable w.r.t. the two predictions."""
    return _DetLosses.apply(cls_pred, reg_pred, y_class_num, y_transform)


# ---- the reference's factories (numpy, Keras layouts) ----------------------------------------------
def cls_loss_rpn(anchors_per_loc=DEFAULT_ANCHORS_PER_LOC):
    def cls_loss_rpn_internal(y_true, y_pred):
        ctx = get_context()
        a = anchors_per_loc
        y = np.asarray(y_true)
        can_use = ctx.to_device(np.ascontiguousarray(y[..., :a] != 0).reshape(1, -1).view(np.uint8))
        is_pos = ctx.to_device(np.ascontiguousarray(y[..., a:] != 0).reshape(1, -1).view(np.uint8))
        pred = ctx.to_device(np.asarray(y_pred, dtype=np.float32).reshape(1, -1))
        zeros = torch.zeros((1, pred.shape[1], 4), dtype=torch.float32, device=pred.device)
        return ctx.to_host(ops.rpn_losses(can_use, is_pos, zeros, pred, zeros))[0, 0]
    return cls_loss_rpn_internal


def bbreg_loss_rpn(anchors_per_loc=DEFAULT_ANCHORS_PER_LOC):
    def bbreg_loss_rpn_internal(y_true, y_pred):
        ctx = get_context()
        a4 = 4 * anchors_per_loc
        y = np.asarray(y_true, dtype=np.float32)
        sel = np.ascontiguousarray(y[..., :a4].reshape(-1, 4)[:, 0] != 0).reshape(1, -1).view(np.uint8)   # repeat(.., 4)
        targets = ctx.to_device(np.ascontiguousarray(y[..., a4:]).reshape(1, -1, 4))
        pred = ctx.to_device(np.asarray(y_pred, dtype=np.float32).reshape(1, -1, 4))
        flags = ctx.to_device(sel)
        half = torch.full((1, pred.shape[1]), 0.5, dtype=torch.float32, device=pred.device)
        return ctx.to_host(ops.rpn_losses(flags, flags, targets, half, pred))[0, 1]
    return bbreg_loss_rpn_internal


def bbreg_loss_det(num_classes):
    def class_loss_internal(y_true, y_pred):
        ctx = get_context()
        y = np.asarray(y_true, dtype=np.float32)
        m = y.shape[-2]
        yt = ctx.to_device(y.reshape(1, m, 8 * num_classes))
        pred = ctx.to_device(np.asarray(y_pred, dtype=np.float32).reshape(1, m, 4 * num_classes))
        k = num_classes + 1
        onehot = torch.zeros((1, m, k), dtype=torch.int32, device=pred.device)
        onehot[..., -1] = 1
        uniform = torch.full((1, m, k), 1.0 / k, dtype=torch.float32, device=pred.device)
        return ctx.to_host(ops.det_losses(onehot, yt, uniform, pred))[0, 1]
    return class_loss_internal


def cls_loss_det(y_true, y_pred):
    ctx = get_context()
    y = np.asarray(y_true)
    m, k = y.shape[-2], y.shape[-1]
    yc = ctx.to_device(y.reshape(-1, m, k)[:1].astype(np.int32))
    pred = ctx.to_device(np.asarray(y_pred, dtype=np.float32).reshape(-1, m, k)[:1])
    zeros_t = torch.zeros((1, m, 8 * (k - 1)), dtype=torch.float32, device=pred.device)
    zeros_p = torch.zeros((1, m, 4 * (k - 1)), dtype=torch.float32, device=pred.device)
    return ctx.to_host(ops.det_losses(yc, zeros_t, pred, zeros_p))[0, 0]
