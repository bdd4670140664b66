"""Loss plumbing of the reference's ``semi_seg/_utils.py`` that sits on the hot path.

``IIDLoss`` (semi_seg/_utils.py:12-15) returns the loss only; ``IICLossWrapper`` (:189-224) picks the
global loss for encoder features and the small-patch local loss for decoder features.
``average_iter`` / ``weighted_average_iter`` (contrastyou/helper/utils.py:46-47,54-56) are the two reductions the
epocher applies to those losses (semi_seg/epocher.py:275,277); ``combine_iic_losses`` does both in three launches.  The UNet block
names come from contrastyou/arch/unet.py:185-194 and are restated here so this module does not need
the backbone.
"""
from __future__ import annotations

from itertools import repeat
from typing import List, Sequence, Union

import torch
from torch import Tensor, nn

from ..losses.iic_loss import IIDLoss as _IIDLoss
from ..losses.iic_loss import IIDSegmentationSmallPathLoss, iic_losses

# contrastyou/arch/unet.py:185-194
ENCODER_NAMES = ["Conv1", "Conv2", "Conv3", "Conv4", "Conv5"]
DECODER_NAMES = ["Up5", "Up_conv5", "Up4", "Up_conv4", "Up3", "Up_conv3", "Up2", "Up_conv2", "DeConv_1x1"]


class IIDLoss(_IIDLoss):
    _returns_loss_only = True        # semi_seg/_utils.py:14-15; iic_losses() honours it too

    def forward(self, x_out: Tensor, x_tf_out: Tensor):
        return super().forward(x_out, x_tf_out)[0]

    def from_logits(self, logits_out: Tensor, logits_tf_out: Tensor, T: float = 1.0):
        return super().from_logits(logits_out, logits_tf_out, T)[0]


def _nlist(n):
    def parse(x):
        if isinstance(x, (list, tuple)):
            assert len(x) == n, (len(x), n)
            return x
        return list(repeat(x, n))
    return parse


class IICLossWrapper(nn.Module):
    def __init__(self, feature_names: Union[str, List[str]], paddings: Union[int, List[int]],
                 patch_sizes: Union[int, List[int]]) -> None:
        super().__init__()
        if isinstance(feature_names, str):
            feature_names = [feature_names]
        self._encoder_features = [f for f in feature_names if f in ENCODER_NAMES]
        self._decoder_features = [f for f in feature_names if f in DECODER_NAMES]
        assert len(feature_names) == len(self._encoder_features) + len(self._decoder_features)
        self._LossModuleDict = nn.ModuleDict()
        for f in self._encoder_features:
            self._LossModuleDict[f] = IIDLoss()
        if len(self._decoder_features) > 0:
            paddings = _nlist(len(self._decoder_features))(paddings)
            patch_sizes = _nlist(len(self._decoder_features))(patch_sizes)
            for f, p, size in zip(self._decoder_features, paddings, patch_sizes):
                self._LossModuleDict[f] = IIDSegmentationSmallPathLoss(padding=p, patch_size=size)

    def __getitem__(self, item):
        if item in self._LossModuleDict.keys():
            return self._LossModuleDict[item]
        raise IndexError(item)

    def __iter__(self):
        for k, v in self._LossModuleDict.items():
            yield v

    def items(self):
        return self._LossModuleDict.items()

    @property
    def feature_names(self):
        return self._encoder_features + self._decoder_features


def average_iter(a_list):
    """Mean over the sub-heads of one layer (contrastyou/helper/utils.py:46-47; semi_seg/epocher.py:275)."""
    a_list = list(a_list)
    return sum(a_list) / float(len(a_list))


def weighted_average_iter(a_list, weight_list):
    """sum_l w_l a_l / (sum_l w_l + 1e-16) over the feature layers (contrastyou/helper/utils.py:54-56;
    semi_seg/epocher.py:277; the weights are the normalised feature importances of semi_seg/trainer.py:46-49)."""
    a_list, weight_list = list(a_list), list(weight_list)
    assert len(a_list) == len(weight_list), (len(a_list), len(weight_list))
    return sum(a * w for a, w in zip(a_list, weight_list)) / (sum(weight_list) + 1e-16)


def combine_iic_losses(losses_per_layer: Sequence[Sequence[Tensor]], feature_importance: Sequence[float]):
    """``weighted_average_iter([average_iter(heads) for heads in losses_per_layer], feature_importance)`` -- the value
    ``IICTrainEpocher.regularization`` returns (semi_seg/epocher.py:274-277) -- as ONE stack, one weighted sum and one
    division instead of ~2*S*L scalar kernels.  Also returns the per-layer means (for the ``individual_mis`` meter,
    epocher.py:279-282) as one tensor, so they can be read with a single host transfer."""
    assert len(losses_per_layer) == len(feature_importance), (len(losses_per_layer), len(feature_importance))
    counts = [len(h) for h in losses_per_layer]
    assert all(c > 0 for c in counts), counts
    flat = torch.stack([l for heads in losses_per_layer for l in heads])
    # weight of one sub-head loss: importance of its layer / number of sub-heads of that layer
    w = torch.tensor([float(fi) / c for fi, c in zip(feature_importance, counts) for _ in range(c)],
                     dtype=flat.dtype).to(flat.device, non_blocking=True)
    total = (flat * w).sum() / (float(sum(feature_importance)) + 1e-16)
    seg = torch.tensor([1.0 / c for c in counts for _ in range(c)], dtype=flat.dtype).to(flat.device, non_blocking=True)
    index = torch.tensor([i for i, c in enumerate(counts) for _ in range(c)]).to(flat.device, non_blocking=True)
    per_layer = torch.zeros(len(counts), dtype=flat.dtype, device=flat.device).index_add(0, index, flat * seg)
    return total, per_layer


def iic_regularization(prob_pairs_per_layer: Sequence[Sequence], criteria: Sequence[nn.Module],
                       feature_importance: Sequence[float], from_logits: bool = False, T: float = 1.0):
    """The value ``IICTrainEpocher.regularization`` computes (semi_seg/epocher.py:249-277) from the cluster heads' outputs:
    ``prob_pairs_per_layer[l]`` is the list of ``(prob1, prob2)`` pairs of layer ``l`` (one per sub-head, epocher.py:
    269-273), ``criteria[l]`` that layer's loss module (``IICLossWrapper[l]``).  All S x L loss calls go through
    :func:`iic_losses` -- one finish launch, one multi-GPU exchange -- and are combined by :func:`combine_iic_losses`
    (``average_iter`` over sub-heads, ``weighted_average_iter`` over layers).  Returns ``(reg_loss, per_layer_losses)``.
    ``from_logits=True``: the pairs are the heads' logits, as for :func:`iic_losses`."""
    assert len(prob_pairs_per_layer) == len(criteria) == len(feature_importance)
    calls, counts = [], []
    for pairs, crit in zip(prob_pairs_per_layer, criteria):
        pairs = list(pairs)
        counts.append(len(pairs))
        calls += [(crit, a, b) for a, b in pairs]
    flat = iic_losses(calls, from_logits=from_logits, T=T)
    per_layer, k = [], 0
    for c in counts:
        per_layer.append([l[0] if isinstance(l, tuple) else l for l in flat[k:k + c]])
        k += c
    return combine_iic_losses(per_layer, feature_importance)
