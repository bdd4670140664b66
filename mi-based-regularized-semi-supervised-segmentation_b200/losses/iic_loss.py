"""Drop-in loss modules for the reference's ``contrastyou/losses/iic_loss.py`` -- B200 CUDA path.

Same class names, constructor arguments, call signatures, return values and exception types as the
reference; the arithmetic runs in libiic_b200.so (see ops.py / include/iic_b200.h).  The modules stay
parameter-free (empty ``state_dict``) so reference checkpoints load unchanged
(dc2:deepclustering2/trainer/_io.py:51-60).

Differences a caller can observe:
  * inputs must be float32 CUDA tensors -- there is no CPU path;
  * the simplex / NaN assertions are evaluated on the device and, in the default "strict" policy,
    read back once at the end of the call (checks.py) instead of once per assert;
  * ``padding`` up to 7 (the reference's own default) is supported.
"""
from __future__ import annotations

import sys
from itertools import repeat

import numpy as np
import torch
from torch import Tensor, nn

from .. import checks
from ..ops import (FusedShapeUnsupported, GlobalIICFunction, GlobalTerm, JointFunction, LocalIICFunction,
                   LocalIICLogitsFunction, LocalTerm, from_logits_covered, global_logits_covered, iic_terms)


def _pair(x):
    # contrastyou/losses/iic_loss.py:16-26
    if isinstance(x, (tuple, list)):
        return tuple(x)
    return tuple(repeat(x, 2))


class IIDLoss(nn.Module):
    """Global IIC loss on (N, K) simplex rows; mirrors contrastyou/losses/iic_loss.py:31-71."""

    def __init__(self, lamb: float = 1.0, eps: float = sys.float_info.epsilon):
        super().__init__()
        print(f"Initialize {self.__class__.__name__}.")
        self.lamb = float(lamb)
        self.eps = float(eps)          # stored but unused, as in the reference (:40; 1e-10 is hard-coded)
        self.torch_vision = torch.__version__

    def forward(self, x_out: Tensor, x_tf_out: Tensor):
        """Returns ``(loss, loss_no_lamb, p_i_j)`` (iic_loss.py:43-71)."""
        assert x_out.dim() == 2 and x_tf_out.shape == x_out.shape, (x_out.shape, x_tf_out.shape)
        # the simplex assertions of :50-51 run inside the joint kernel
        loss, loss_no_lamb, p_i_j = GlobalIICFunction.apply(x_out, x_tf_out, self.lamb,
                                                            checks.want_simplex_kernels())
        checks.finish(x_out.device, loss, "x_out / x_tf_out not normalized.")
        return loss, loss_no_lamb, p_i_j

    def from_logits(self, logits_out: Tensor, logits_tf_out: Tensor, T: float = 1.0):
        """``IIDLoss.forward(softmax(logits_out / T, 1), softmax(logits_tf_out / T, 1))`` -- the (N, K) rows of a
        ``ClusterHead`` before its ``SoftmaxWithT`` (contrastyou/trainer/_utils.py:15-23, ``ClusterHead.logits()``) --
        with the softmax inside the joint launch and its backward inside the gradient kernel.  Returns the same
        ``(loss, loss_no_lamb, p_i_j)``; the gradients are with respect to the logits.  Covered: N <= 4096 rows and
        K <= 128 clusters, float32 CUDA rows with unit inner stride (sub-head views of a wider head output included);
        anything else applies the softmax first."""
        assert logits_out.dim() == 2 and logits_tf_out.shape == logits_out.shape, (logits_out.shape, logits_tf_out.shape)
        if global_logits_covered(logits_out, logits_tf_out):
            t = GlobalTerm(logits_out, logits_tf_out, self.lamb, True, logits=True, inv_temperature=1.0 / float(T))
            (r,) = iic_terms([t])
            checks.finish(logits_out.device, r[0])
            return r
        return IIDLoss.forward(self, (logits_out / T).softmax(1), (logits_tf_out / T).softmax(1))


def compute_joint(x_out: Tensor, x_tf_out: Tensor, symmetric=True) -> Tensor:
    """Joint probability of two (N, K) simplex batches; mirrors iic_loss.py:74-94."""
    bn, k = x_out.shape
    assert x_tf_out.size(0) == bn and x_tf_out.size(1) == k
    # the simplex assertions of :82-83 run inside the joint kernel
    p_i_j = JointFunction.apply(x_out, x_tf_out, bool(symmetric), checks.want_simplex_kernels())
    checks.finish(x_out.device, None, "x_out / x_tf_out not normalized.")
    return p_i_j


class IIDSegmentationLoss(nn.Module):
    """Local (shifted-window) IIC loss on (B, K, H, W) maps; mirrors iic_loss.py:97-149."""

    def __init__(self, lamda=1.0, padding=7, eps: float = sys.float_info.epsilon) -> None:
        super().__init__()
        print(f"Initialize {self.__class__.__name__}.")
        self.lamda = lamda
        self.padding = padding
        self.eps = eps                 # unused in the reference too (1e-16 is hard-coded, :124,141-143)

    def _loss(self, x_out: Tensor, x_tf_out: Tensor, mask, patch, step) -> Tensor:
        assert x_out.requires_grad and x_tf_out.requires_grad        # :110
        if mask is not None:
            assert not mask.requires_grad                            # :112
        assert x_out.shape == x_tf_out.shape                         # :114
        # :113 asserts simplex(x_out) only; here it runs inside the joint kernel
        loss = LocalIICFunction.apply(x_out, x_tf_out, mask, int(self.padding), int(patch[0]), int(patch[1]),
                                      int(step[0]), int(step[1]), float(self.lamda),
                                      checks.want_simplex_kernels())
        checks.finish(x_out.device, loss, "x_out is not a simplex over dim 1")
        return loss

    # the reference overrides __call__ (not forward), so module hooks are bypassed there too (:107)
    def __call__(self, x_out: Tensor, x_tf_out: Tensor, mask: Tensor = None) -> Tensor:
        h, w = x_out.shape[2], x_out.shape[3]
        return self._loss(x_out, x_tf_out, mask, (h, w), (h, w))


def patch_generator(feature_map, patch_size=(32, 32), step_size=(16, 16)):
    """Yields the window views of iic_loss.py:152-160 (host-side helper; the loss itself tiles on the GPU)."""
    b, c, h, w = feature_map.shape
    hs = np.arange(0, h - patch_size[0], step_size[0])
    hs = np.append(hs, max(h - patch_size[0], 0))
    ws = np.arange(0, w - patch_size[1], step_size[1])
    ws = np.append(ws, max(w - patch_size[1], 0))
    for _h in hs:
        for _w in ws:
            yield feature_map[:, :, _h:min(_h + patch_size[0], h), _w:min(_w + patch_size[1], w)]


class IIDSegmentationSmallPathLoss(IIDSegmentationLoss):
    """Mean of the local loss over 50 %-overlapping patches; mirrors iic_loss.py:164-189.

    All patches are processed by ONE joint launch, one epilogue and one backward launch.
    """

    def __init__(self, lamda=1.0, padding=7, eps: float = sys.float_info.epsilon, patch_size=32) -> None:
        super().__init__(lamda, padding, eps)
        self._patch_size = _pair(patch_size)
        self._step_size = _pair(patch_size // 2)

    def __call__(self, x_out: Tensor, x_tf_out: Tensor, mask: Tensor = None):
        assert x_out.shape == x_tf_out.shape, (x_out.shape, x_tf_out.shape)
        return self._loss(x_out, x_tf_out, mask, self._patch_size, self._step_size)

    def __repr__(self):
        return f"{self.__class__.__name__} with patch_size={self._patch_size} and padding={self.padding}."

    def from_logits(self, logits_out: Tensor, logits_tf_out: Tensor, T: float = 1.0) -> Tensor:
        """``self(softmax(logits_out / T, 1), softmax(logits_tf_out / T, 1))`` with both softmaxes -- the
        ``SoftmaxWithT`` at the end of ``LocalClusterHead`` (contrastyou/trainer/_utils.py:15-23,137-168) --
        fused into the joint kernel and their backward into the gradient kernel, so the probability maps are
        never written to memory.  The gradient is returned with respect to the logits.

        The fused kernels cover one patch (the patch at least the map) and
          * 10 clusters: padding 1, width a multiple of 4 and at most 248 (the udaiic decoder shapes);
          * 16 to 24 clusters (the reference's 20): padding 3, or padding 1 on maps with enough row blocks to fill the
            GPU; width a multiple of 16;
          * 128 clusters (the wide heads): padding 1, width a multiple of 16 and at most 248.
        Both need 16-byte aligned rows.  Any other shape applies the softmax first and takes the probability path."""
        assert logits_out.shape == logits_tf_out.shape, (logits_out.shape, logits_tf_out.shape)
        assert logits_out.requires_grad and logits_tf_out.requires_grad        # :110
        h, w = logits_out.shape[2], logits_out.shape[3]
        one_patch = self._patch_size[0] >= h and self._patch_size[1] >= w
        if one_patch and logits_out.is_cuda:
            try:
                loss = LocalIICLogitsFunction.apply(logits_out, logits_tf_out, int(self.padding), float(self.lamda),
                                                    1.0 / float(T))
                checks.finish(logits_out.device, loss)
                return loss
            except FusedShapeUnsupported:
                pass
        return self((logits_out / T).softmax(1), (logits_tf_out / T).softmax(1))


def iic_losses(calls, from_logits: bool = False, T: float = 1.0):
    """Evaluate many loss calls of one iteration TOGETHER: ``calls`` is a sequence of ``(criterion, x_out, x_tf_out)`` or
    ``(criterion, x_out, x_tf_out, mask)`` with ``criterion`` an :class:`IIDLoss`, :class:`IIDSegmentationLoss` or
    :class:`IIDSegmentationSmallPathLoss` instance; the result is the list ``[criterion(x_out, x_tf_out), ...]`` -- same
    values, same autograd behaviour -- but computed with one joint kernel per call and ONE finish launch for all of
    them (csrc/finish.cu): one slot reduction, one epilogue and, under ``set_data_parallel(True)``, ONE exchange of all
    joints.  This is the batched form of the (feature layer x sub-head) loop of ``IICTrainEpocher.regularization``
    (semi_seg/epocher.py:249-277), where the reference issues S x L separate calls.

    ``from_logits=True``: every ``x_out`` / ``x_tf_out`` is a cluster head's LOGITS and the result is that of the calls
    on ``softmax(x / T, 1)`` (the heads' ``SoftmaxWithT``, contrastyou/trainer/_utils.py:15-23).  Local terms whose shape
    the fused kernels cover (:func:`from_logits_covered`, see :meth:`IIDSegmentationSmallPathLoss.from_logits`) take the
    softmax inside their kernels, and so do global terms of at most 4096 rows and 128 clusters (the finish launch
    normalises their rows, see :meth:`IIDLoss.from_logits`); the others get ``torch.softmax`` first.  Gradients are with
    respect to the logits.  Masks are not accepted with ``from_logits``."""
    terms, post = [], []
    inv_t = 1.0 / float(T)
    for c in calls:
        crit, x, y = c[0], c[1], c[2]
        mask = c[3] if len(c) > 3 else None
        if from_logits and mask is not None:
            raise ValueError("iic_losses(from_logits=True): masks are not supported; apply the softmax and pass the "
                             "probabilities with the mask")
        if isinstance(crit, IIDSegmentationLoss):
            assert x.requires_grad and y.requires_grad                   # iic_loss.py:110
            if mask is not None:
                assert not mask.requires_grad                            # :112
            assert x.shape == y.shape                                    # :114
            h, w = x.shape[2], x.shape[3]
            if isinstance(crit, IIDSegmentationSmallPathLoss):
                patch, step = crit._patch_size, crit._step_size
            else:
                patch, step = (h, w), (h, w)
            if from_logits:
                one_patch = patch[0] >= h and patch[1] >= w
                if one_patch and from_logits_covered(x, y, crit.padding):
                    terms.append(LocalTerm(x, y, None, crit.padding, (h, w), (h, w), crit.lamda, logits=True,
                                           inv_temperature=inv_t))
                    post.append(None)
                    continue
                x, y = (x / T).softmax(1), (y / T).softmax(1)          # on the autograd tape, before the batched call
            terms.append(LocalTerm(x, y, mask, crit.padding, patch, step, crit.lamda))
            post.append(None)
        elif isinstance(crit, IIDLoss):
            assert x.dim() == 2 and y.shape == x.shape, (x.shape, y.shape)
            if from_logits and global_logits_covered(x, y):
                terms.append(GlobalTerm(x, y, crit.lamb, True, logits=True, inv_temperature=inv_t))
                post.append(crit)
                continue
            if from_logits:
                x, y = (x / T).softmax(1), (y / T).softmax(1)
            terms.append(GlobalTerm(x, y, crit.lamb, True))
            post.append(crit)
        else:
            raise TypeError(f"iic_losses: unsupported criterion {type(crit).__name__}")
    if not terms:
        return []
    res = iic_terms(terms, checks.want_simplex_kernels())
    out = []
    for r, crit in zip(res, post):
        if crit is None:
            out.append(r)
        else:
            # semi_seg/_utils.py:12-15: the epocher's IIDLoss wrapper returns the loss only
            out.append(r[0] if getattr(crit, "_returns_loss_only", False) else r)
    checks.finish(terms[0].x.device, out[0] if not isinstance(out[0], tuple) else out[0][0],
                  "x_out / x_tf_out is not a simplex over dim 1")
    return out
