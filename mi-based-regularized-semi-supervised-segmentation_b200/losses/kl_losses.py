"""UDA consistency criteria on the B200 CUDA path.

``KL_div`` mirrors dc2:deepclustering2/loss/kl_losses.py:76-129; ``MSELoss`` is the twin of the
``torch.nn.MSELoss()`` the reference builds at semi_seg/trainer.py:137,194.  Both are called as
``criterion(softmax(tf_logits), softmax(logits_tf).detach())`` at semi_seg/epocher.py:221-224.
``uda_from_logits`` fuses those two softmaxes into the loss kernels.

``sup_kl_from_logits`` is the supervised branch of the same iteration (SURVEY.md section 8f row 4):
``KL_div()(label_logits.softmax(1), class2one_hot(labeled_target.squeeze(1), C))`` at
semi_seg/epocher.py:165-166, with the softmax and the one-hot fused into one pass that can also count
what the ``sup_dice`` meter needs (epocher.py:183-184).
"""
from __future__ import annotations

import numbers
from typing import List, Optional, Union

import torch
from torch import Tensor, nn

from .. import checks
from ..ops import SupervisedKLFunction, UDAFlipFunction, UDAFunction

_KIND = {"mse": 0, "kl": 1}


class KL_div(nn.Module):
    r"""KL(target || prob) = -\sum target * log((prob+eps)/(target+eps)); reduction "mean" or "sum".

    ``reduction="none"`` (the per-pixel map of dc2:loss/kl_losses.py:121-126) is accepted by the constructor like the
    reference's, but ``forward`` raises ``NotImplementedError`` for it: no caller on the udaiic path uses it
    (``semi_seg/trainer.py:137,194`` and ``semi_seg/main.py`` build ``KL_div()`` with the default), and the fused kernels
    never materialise the per-pixel map."""

    def __init__(self, reduction="mean", eps=1e-16, weight: Union[List[float], Tensor] = None, verbose=True):
        super().__init__()
        assert reduction in ("mean", "sum", "none"), reduction
        self._eps = eps
        self._reduction = reduction
        self._weight: Optional[Tensor] = weight
        if weight is not None:
            assert isinstance(weight, (list, Tensor)), type(weight)
            if isinstance(weight, list):
                assert all(isinstance(x, (int, float)) for x in weight)
                self._weight = torch.Tensor(weight).float()
            else:
                self._weight = weight.float()
            self._weight = self._weight / self._weight.sum() * len(self._weight)   # kl_losses.py:100
        if verbose:
            print(f"Initialized {self.__class__.__name__} \nwith weight={self._weight} and reduction={self._reduction}.")

    def forward(self, prob: Tensor, target: Tensor, **kwargs) -> Tensor:
        do_assert = not kwargs.get("disable_assert")
        if do_assert:
            assert prob.shape == target.shape
            assert not target.requires_grad
            assert prob.requires_grad
        if self._reduction == "none":
            raise NotImplementedError("KL_div(reduction='none') is not on the udaiic path; use the reference for it")
        if self._weight is not None:
            assert len(self._weight) == target.shape[1]
        if not target.is_floating_point():
            # the supervised call passes class2one_hot's `long` tensor (semi_seg/epocher.py:165-166); the reference's
            # `target + eps` promotes it to the default float dtype (kl_losses.py:115)
            target = target.to(prob.dtype)
        loss = UDAFunction.apply(prob, target, _KIND["kl"], float(self._eps), self._weight, False,
                                 bool(do_assert and checks.want_simplex_kernels()))
        if self._reduction == "sum":
            npix = prob.numel() // prob.shape[1]
            loss = loss * float(npix)
        if do_assert:
            checks.finish(prob.device, loss, "prob / target is not a simplex over dim 1")
        return loss

    def __repr__(self):
        return f"{self.__class__.__name__}\n, weight={self._weight}"


class MSELoss(nn.Module):
    """``torch.nn.MSELoss()`` (mean over every element) with the fused CUDA forward/backward."""

    def __init__(self, reduction: str = "mean") -> None:
        super().__init__()
        assert reduction in ("mean", "sum"), reduction
        self.reduction = reduction

    def forward(self, input: Tensor, target: Tensor) -> Tensor:
        assert input.shape == target.shape, (input.shape, target.shape)
        loss = UDAFunction.apply(input, target.detach(), _KIND["mse"], 0.0, None, False, False)
        if self.reduction == "sum":
            loss = loss * float(input.numel())
        return loss


def uda_from_logits(student_logits: Tensor, teacher_logits: Tensor, kind: str = "mse", eps: float = 1e-16,
                    teacher_flips: Optional[Tensor] = None) -> Tensor:
    """criterion(softmax(student_logits, 1), softmax(teacher_logits, 1).detach()) in one kernel each way
    (semi_seg/epocher.py:221-224); the gradient is returned w.r.t. ``student_logits``.

    ``teacher_flips`` (uint8 per sample, ``augment.draw_flip_flags``): the teacher is read through those flips, i.e.
    ``teacher_logits`` is the UNflipped ``unlabel_logits`` and the ``torch.stack([T(x) for x in unlabel_logits])`` of
    semi_seg/epocher.py:160-161 is folded into the loss kernels."""
    assert student_logits.shape == teacher_logits.shape
    if teacher_flips is not None:
        return UDAFlipFunction.apply(student_logits, teacher_logits.detach(),
                                     teacher_flips.to(student_logits.device, non_blocking=True), _KIND[kind],
                                     float(eps), True)
    return UDAFunction.apply(student_logits, teacher_logits.detach(), _KIND[kind], float(eps), None, True, False)


def _normalised_weight(weight) -> Optional[Tensor]:
    if weight is None:
        return None
    w = torch.as_tensor(weight).float()
    return w / w.sum() * len(w)                                                   # kl_losses.py:100


def sup_kl_from_logits(logits: Tensor, target: Tensor, weight: Union[List[float], Tensor] = None,
                       eps: float = 1e-16, return_dice: bool = False, ignore_index: Optional[int] = None):
    """``KL_div(weight=weight, eps=eps)(logits.softmax(1), class2one_hot(target, C))`` without the
    probability map or the one-hot tensor (semi_seg/epocher.py:165-166; dc2:loss/kl_losses.py:107-126).

    ``target`` holds int64 class indices, shaped (B, *spatial) or (B, 1, *spatial) as the loaders emit it.
    With ``return_dice`` the call also returns ``(intersection, union)``, the two (B, C) int64 tensors
    ``UniversalDice.add(logits.max(1)[1], target)`` would append (dc2:general_dice_meter.py:41-95), counted in
    the same pass.  A label outside [0, C) raises AssertionError like ``class2one_hot`` (per the check mode).

    ``ignore_index`` (an int, e.g. 255 for the Cityscapes / VOC void label, or torch's -100; a value inside [0, C)
    drops that class): pixels labelled with it add nothing to the loss, get a zero gradient and are left out of the
    Dice counts.  The loss is the sum over the other n pixels divided by n, also with ``weight``: this is
    ``KL_div``'s mean over the kept pixels, not ``F.cross_entropy``'s division by the summed weights of the kept
    labels.  n is counted on the GPU (no host synchronisation, so a CUDA graph can replay the call with a different
    number of ignored pixels); when every pixel is ignored the loss is 0 and the gradient is zero.  Any other label
    outside [0, C) still raises, and counts in n.
    """
    if ignore_index is not None:
        if isinstance(ignore_index, bool) or not isinstance(ignore_index, numbers.Integral):
            raise TypeError(f"sup_kl_from_logits: ignore_index must be None or an int, got "
                            f"{type(ignore_index).__name__}")
        ignore_index = int(ignore_index)
        if not -2 ** 63 <= ignore_index < 2 ** 63:
            raise ValueError(f"sup_kl_from_logits: ignore_index={ignore_index} is not an int64 label")
    if target.dim() == logits.dim() and target.shape[1] == 1:
        target = target.squeeze(1)
    assert not target.requires_grad
    if not eps > 0:
        raise ValueError("sup_kl_from_logits needs eps > 0 (the reference's loss is NaN at eps = 0)")
    loss, dice, _ = SupervisedKLFunction.apply(logits, target, float(eps), _normalised_weight(weight),
                                               bool(return_dice), ignore_index)
    checks.finish(logits.device, loss, "prob / target is not a simplex over dim 1")
    if return_dice:
        return loss, (dice[0], dice[1])
    return loss


def dice_from_counts(intersection: Tensor, union: Tensor) -> Tensor:
    """Per-class Dice of one group, as UniversalDice.log computes it from the summed counts
    (dc2:general_dice_meter.py:96-108): (2 * sum_b I + 1e-6) / (sum_b U + 1e-6)."""
    return (2 * intersection.sum(0) + 1e-6) / (union.sum(0) + 1e-6)
