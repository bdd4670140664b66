"""torch custom ops (namespace ``iic_b200``) over the C-ABI CUDA library, plus their autograd glue.

Every op is CUDA-only and calls straight into libiic_b200.so through ctypes with raw device pointers
and the current CUDA stream; there is no eager/PyTorch fallback.  Nothing here synchronises the host,
so a whole loss forward+backward can be captured in a CUDA graph.

The mathematical contract of each op (reference file:line) is stated in include/iic_b200.h.
"""
from __future__ import annotations

import math
from typing import Optional, Tuple

import torch

from . import _lib

_LIBDEF = torch.library.Library("iic_b200", "DEF")
_LIBDEF.define("local_joint(Tensor x, Tensor y, Tensor? mask, int pad, int patch_h, int patch_w, "
               "int step_h, int step_w, bool check_simplex=False) -> Tensor")
_LIBDEF.define("local_epilogue(Tensor J, int K, int pad, float lamda) -> (Tensor, Tensor, Tensor)")
_LIBDEF.define("local_backward(Tensor x, Tensor y, Tensor? mask, Tensor Wx, Tensor Wy, Tensor grad, int pad, "
               "int patch_h, int patch_w, int step_h, int step_w) -> (Tensor, Tensor)")
_LIBDEF.define("local_joint_logits(Tensor lx, Tensor ly, int pad, float inv_temperature) -> Tensor")
_LIBDEF.define("local_backward_logits(Tensor lx, Tensor ly, Tensor Wx, Tensor Wy, Tensor grad, int pad, "
               "float inv_temperature) -> (Tensor, Tensor)")
_LIBDEF.define("global_joint(Tensor x, Tensor y, bool check_simplex=False) -> Tensor")
_LIBDEF.define("global_epilogue(Tensor J, float lamb, bool symmetric, bool want_losses) -> (Tensor, Tensor)")
_LIBDEF.define("global_backward(Tensor x, Tensor y, Tensor J, float lamb, bool symmetric, Tensor? g_loss, "
               "Tensor? g_no_lamb, Tensor? gP) -> (Tensor, Tensor)")
_LIBDEF.define("uda_forward(Tensor prob, Tensor target, int kind, float eps, Tensor? weight, bool from_logits, "
               "bool check_simplex) -> Tensor")
_LIBDEF.define("uda_backward(Tensor prob, Tensor target, int kind, float eps, Tensor? weight, bool from_logits, "
               "Tensor grad) -> Tensor")
_LIBDEF.define("simplex_check(Tensor t, int axis) -> ()")
_LIBDEF.define("flip_batch(Tensor x, Tensor flips) -> Tensor")
_LIBDEF.define("uda_flip_forward(Tensor prob, Tensor target, Tensor flips, int kind, float eps, bool from_logits) -> Tensor")
_LIBDEF.define("uda_flip_backward(Tensor prob, Tensor target, Tensor flips, int kind, float eps, bool from_logits, "
               "Tensor grad) -> Tensor")
_LIBDEF.define("sup_forward(Tensor logits, Tensor labels, float eps, Tensor? weight, bool want_dice) -> (Tensor, Tensor)")
_LIBDEF.define("sup_backward(Tensor logits, Tensor labels, float eps, Tensor? weight, Tensor grad) -> Tensor")


# ---- per (device, stream) persistent state ---------------------------------------------------------
class _StreamState:
    """Sticky flag word + small zero-initialised, self-resetting kernel workspaces."""

    def __init__(self, device: torch.device):
        lib = _lib.load()
        self.flags = torch.zeros(1, dtype=torch.int32, device=device)
        self.uda_ws = torch.zeros(lib.iic_uda_workspace_bytes(device.index or 0), dtype=torch.uint8, device=device)
        self.epi_ws = {}
        self.sup_ws = None
        self.flip_ws = None
        self.fin_ws = torch.zeros(lib.iic_finish_workspace_bytes(), dtype=torch.uint8, device=device)

    def uda_flip_ws(self, outer: int, device) -> torch.Tensor:
        nbytes = _lib.load().iic_uda_flip_workspace_bytes(device.index or 0, outer)
        if self.flip_ws is None or self.flip_ws.numel() < nbytes:
            self.flip_ws = torch.zeros(nbytes, dtype=torch.uint8, device=device)
        return self.flip_ws

    def supervised_ws(self, outer: int, device) -> torch.Tensor:
        nbytes = _lib.load().iic_sup_workspace_bytes(device.index or 0, outer)
        if self.sup_ws is None or self.sup_ws.numel() < nbytes:
            self.sup_ws = torch.zeros(nbytes, dtype=torch.uint8, device=device)
        return self.sup_ws

    def epilogue_ws(self, K: int, pad: int, n_patches: int, device) -> torch.Tensor:
        key = (pad, n_patches)
        ws = self.epi_ws.get(key)
        if ws is None:
            nbytes = _lib.load().iic_local_epilogue_workspace_bytes(K, pad, n_patches)
            ws = torch.zeros(nbytes, dtype=torch.uint8, device=device)
            self.epi_ws[key] = ws
        return ws


_states = {}


def _state(device: torch.device) -> _StreamState:
    key = (device.index, torch.cuda.current_stream(device).cuda_stream)
    st = _states.get(key)
    if st is None:
        st = _StreamState(device)
        _states[key] = st
    return st


_side_streams = {}
overlap_global_backward = False    # run the small global-term gradient kernels beside the local ones (see IICTermsFunction.backward);
                                   # measured at config 2: no gain (0.1639 vs 0.1614-0.1626 ms per step), so off


def _side_stream(device: torch.device) -> "torch.cuda.Stream":
    """A second stream paired with the current stream of `device` (created once, outside any graph capture if the first
    backward runs eagerly, as every warm-up does)."""
    key = (device.index, torch.cuda.current_stream(device).cuda_stream)
    st = _side_streams.get(key)
    if st is None:
        st = torch.cuda.Stream(device=device)
        _side_streams[key] = st
    return st


def flags_tensor(device) -> torch.Tensor:
    """The sticky int32 flag word (IIC_FLAG_*) of the current stream of `device`."""
    return _state(torch.device(device)).flags


def _stream(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _require_cuda_f32(name: str, t: torch.Tensor):
    if not t.is_cuda:
        raise _lib.IICLibraryError(f"iic_b200: `{name}` must be a CUDA tensor (there is no CPU path); got {t.device}")
    if t.dtype != torch.float32:
        raise TypeError(f"iic_b200: `{name}` must be float32, got {t.dtype}")


def _w_contig(t: torch.Tensor) -> torch.Tensor:
    """The kernels need unit innermost stride; anything else is copied (patch views are fine)."""
    return t if t.stride(-1) == 1 else t.contiguous()


def _mask_args(mask: Optional[torch.Tensor], x: torch.Tensor):
    if mask is None:
        return None, 0, 0, 0
    _require_cuda_f32("mask", mask)
    B, K, H, W = x.shape
    if mask.dim() != 4 or mask.shape[0] != B or mask.shape[2:] != x.shape[2:] or mask.shape[1] not in (1, K):
        raise ValueError(f"iic_b200: mask shape {tuple(mask.shape)} does not broadcast to {tuple(x.shape)}")
    mask = _w_contig(mask)
    return mask, mask.stride(0), (0 if mask.shape[1] == 1 else mask.stride(1)), mask.stride(2)


# ---- op implementations ------------------------------------------------------------------------------
def _local_joint(x, y, mask, pad, patch_h, patch_w, step_h, step_w, check_simplex=False):
    lib = _lib.load()
    _require_cuda_f32("x_out", x)
    _require_cuda_f32("x_tf_out", y)
    if x.dim() != 4 or x.shape != y.shape:
        raise ValueError(f"iic_b200.local_joint: shapes {tuple(x.shape)} vs {tuple(y.shape)}")
    x, y = _w_contig(x), _w_contig(y)
    B, K, H, W = x.shape
    m, msn, msc, msh = _mask_args(mask, x)
    npatch = lib.iic_local_num_patches(H, W, patch_h, patch_w, step_h, step_w)
    if npatch <= 0:
        _lib.check(1, "iic_local_num_patches")
    T = 2 * pad + 1
    dev = x.device.index
    nbytes = lib.iic_local_joint_workspace_bytes(dev, B, K, H, W, pad, patch_h, patch_w, step_h, step_w)
    if nbytes == 0:
        _lib.check(1, "iic_local_joint_workspace_bytes")
    ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    J = torch.empty((npatch, T, T, K, K), dtype=torch.float64, device=x.device)
    flags = None
    if check_simplex:
        # the assertion on x_out (iic_loss.py:113) rides along with the joint kernel; rows that are not
        # dense (a sliced view) take the stand-alone streaming check instead
        if x.stride(2) == W:
            flags = _state(x.device).flags.data_ptr()
        else:
            _simplex_check(x, 1)
    with torch.cuda.device(x.device):
        rc = lib.iic_local_joint(x.data_ptr(), x.stride(0), x.stride(1), x.stride(2),
                                 y.data_ptr(), y.stride(0), y.stride(1), y.stride(2),
                                 _ptr(m), msn, msc, msh, B, K, H, W, pad, patch_h, patch_w, step_h, step_w,
                                 J.data_ptr(), ws.data_ptr(), nbytes, flags, _stream(x.device))
    _lib.check(rc, "iic_local_joint")
    return J


def _local_epilogue(J, K, pad, lamda):
    lib = _lib.load()
    if not J.is_cuda or J.dtype != torch.float64 or not J.is_contiguous():
        raise TypeError("iic_b200.local_epilogue: J must be a contiguous CUDA float64 tensor")
    npatch = J.shape[0]
    st = _state(J.device)
    loss = torch.empty((), dtype=torch.float32, device=J.device)
    n = lib.iic_local_coeff_floats(K, pad, npatch)
    Wx = torch.empty(n, dtype=torch.float32, device=J.device)
    Wy = torch.empty(n, dtype=torch.float32, device=J.device)
    ws = st.epilogue_ws(K, pad, npatch, J.device)
    with torch.cuda.device(J.device):
        rc = lib.iic_local_epilogue(J.data_ptr(), K, pad, npatch, float(lamda), loss.data_ptr(), None,
                                    Wx.data_ptr(), Wy.data_ptr(), None, st.flags.data_ptr(), ws.data_ptr(),
                                    _stream(J.device))
    _lib.check(rc, "iic_local_epilogue")
    return loss, Wx, Wy


def _local_backward_into(x, y, mask, Wx, Wy, grad, pad, patch_h, patch_w, step_h, step_w, gx, gy):
    """iic_local_backward writing into the given (B, K, H, W) tensors / channel-block views (dense rows and planes, any
    sample stride); with several patches they must be zero-filled (the patches accumulate)."""
    lib = _lib.load()
    x, y = _w_contig(x), _w_contig(y)
    B, K, H, W = x.shape
    m, msn, msc, msh = _mask_args(mask, x)
    for g in (gx, gy):
        assert g.shape == x.shape and g.stride(3) == 1 and g.stride(2) == W and g.stride(1) == H * W, (g.shape, g.stride())
    grad = grad.to(torch.float32).reshape(())
    with torch.cuda.device(x.device):
        rc = lib.iic_local_backward(x.data_ptr(), x.stride(0), x.stride(1), x.stride(2),
                                    y.data_ptr(), y.stride(0), y.stride(1), y.stride(2),
                                    _ptr(m), msn, msc, msh, B, K, H, W, pad, patch_h, patch_w, step_h, step_w,
                                    Wx.data_ptr(), Wy.data_ptr(), grad.data_ptr(), gx.data_ptr(), gy.data_ptr(),
                                    gx.stride(0), gy.stride(0), _stream(x.device))
    _lib.check(rc, "iic_local_backward")


def _local_backward(x, y, mask, Wx, Wy, grad, pad, patch_h, patch_w, step_h, step_w):
    B, K, H, W = x.shape
    npatch = _lib.load().iic_local_num_patches(H, W, patch_h, patch_w, step_h, step_w)
    alloc = torch.zeros if npatch > 1 else torch.empty
    gx = alloc((B, K, H, W), dtype=torch.float32, device=x.device)
    gy = alloc((B, K, H, W), dtype=torch.float32, device=x.device)
    _local_backward_into(x, y, mask, Wx, Wy, grad, pad, patch_h, patch_w, step_h, step_w, gx, gy)
    return gx, gy


class FusedShapeUnsupported(RuntimeError):
    """The fused from-logits kernels do not cover this shape; apply the softmax and use the probability path."""


def _logit_maps(lx, ly):
    _require_cuda_f32("logits_out", lx)
    _require_cuda_f32("logits_tf_out", ly)
    if lx.dim() != 4 or lx.shape != ly.shape:
        raise ValueError(f"iic_b200.local_joint_logits: shapes {tuple(lx.shape)} vs {tuple(ly.shape)}")
    return _w_contig(lx), _w_contig(ly)


def _local_joint_logits(lx, ly, pad, inv_temperature):
    lib = _lib.load()
    lx, ly = _logit_maps(lx, ly)
    B, K, H, W = lx.shape
    nbytes = lib.iic_b200_sm_count(lx.device.index or 0) * 9 * K * K * 4
    ws = torch.empty(max(nbytes, 4), dtype=torch.uint8, device=lx.device)
    J = torch.empty((1, 3, 3, K, K), dtype=torch.float64, device=lx.device)
    with torch.cuda.device(lx.device):
        rc = lib.iic_local_joint_from_logits(lx.data_ptr(), lx.stride(0), lx.stride(1), lx.stride(2),
                                             ly.data_ptr(), ly.stride(0), ly.stride(1), ly.stride(2),
                                             B, K, H, W, pad, float(inv_temperature), J.data_ptr(), ws.data_ptr(),
                                             ws.numel(), None, _stream(lx.device))
    if rc == _lib.UNSUPPORTED:
        raise FusedShapeUnsupported(lib.iic_b200_last_error().decode())
    _lib.check(rc, "iic_local_joint_from_logits")
    return J


def _local_backward_logits_into(lx, ly, Wx, Wy, grad, pad, inv_temperature, gx, gy):
    lib = _lib.load()
    lx, ly = _logit_maps(lx, ly)
    B, K, H, W = lx.shape
    grad = grad.to(torch.float32).reshape(())
    with torch.cuda.device(lx.device):
        rc = lib.iic_local_backward_from_logits(lx.data_ptr(), lx.stride(0), lx.stride(1), lx.stride(2),
                                                ly.data_ptr(), ly.stride(0), ly.stride(1), ly.stride(2),
                                                B, K, H, W, pad, float(inv_temperature), Wx.data_ptr(), Wy.data_ptr(),
                                                grad.data_ptr(), gx.data_ptr(), gy.data_ptr(), gx.stride(0), gy.stride(0),
                                                _stream(lx.device))
    if rc == _lib.UNSUPPORTED:
        raise FusedShapeUnsupported(lib.iic_b200_last_error().decode())
    _lib.check(rc, "iic_local_backward_from_logits")


def _local_backward_logits(lx, ly, Wx, Wy, grad, pad, inv_temperature):
    B, K, H, W = lx.shape
    gx = torch.empty((B, K, H, W), dtype=torch.float32, device=lx.device)
    gy = torch.empty((B, K, H, W), dtype=torch.float32, device=lx.device)
    _local_backward_logits_into(lx, ly, Wx, Wy, grad, pad, inv_temperature, gx, gy)
    return gx, gy


def _global_joint(x, y, check_simplex=False):
    lib = _lib.load()
    _require_cuda_f32("x_out", x)
    _require_cuda_f32("x_tf_out", y)
    if x.dim() != 2 or x.shape != y.shape:
        raise ValueError(f"iic_b200.global_joint: shapes {tuple(x.shape)} vs {tuple(y.shape)}")
    x, y = _w_contig(x), _w_contig(y)
    N, K = x.shape
    nbytes = lib.iic_global_joint_workspace_bytes(x.device.index, N, K)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    J = torch.empty((K, K), dtype=torch.float64, device=x.device)
    with torch.cuda.device(x.device):
        rc = lib.iic_global_joint(x.data_ptr(), x.stride(0), y.data_ptr(), y.stride(0), N, K, J.data_ptr(),
                                  ws.data_ptr(), nbytes,
                                  _state(x.device).flags.data_ptr() if check_simplex else None, _stream(x.device))
    _lib.check(rc, "iic_global_joint")
    return J


def _global_epilogue(J, lamb, symmetric, want_losses):
    lib = _lib.load()
    K = J.shape[0]
    st = _state(J.device)
    losses = torch.empty(2, dtype=torch.float32, device=J.device)
    P = torch.empty((K, K), dtype=torch.float32, device=J.device)
    with torch.cuda.device(J.device):
        rc = lib.iic_global_epilogue(J.data_ptr(), K, float(lamb), int(symmetric),
                                     losses.data_ptr() if want_losses else None, P.data_ptr(),
                                     st.flags.data_ptr(), _stream(J.device))
    _lib.check(rc, "iic_global_epilogue")
    return losses, P


def _global_backward(x, y, J, lamb, symmetric, g_loss, g_no_lamb, gP):
    N, K = x.shape
    gx = torch.empty((N, K), dtype=torch.float32, device=x.device)
    gy = torch.empty((N, K), dtype=torch.float32, device=x.device)
    _global_backward_into(x, y, J, lamb, symmetric, g_loss, g_no_lamb, gP, gx, gy)
    return gx, gy


def _global_backward_into(x, y, J, lamb, symmetric, g_loss, g_no_lamb, gP, gx, gy):
    lib = _lib.load()
    x, y = _w_contig(x), _w_contig(y)
    N, K = x.shape
    assert gx.shape == x.shape and gy.shape == x.shape and gx.stride(1) == 1 and gy.stride(1) == 1
    if g_loss is not None:
        g_loss = g_loss.to(torch.float32).reshape(())
    if g_no_lamb is not None:
        g_no_lamb = g_no_lamb.to(torch.float32).reshape(())
    if gP is not None:
        gP = gP.to(torch.float32).contiguous()
    with torch.cuda.device(x.device):
        rc = lib.iic_global_backward(x.data_ptr(), x.stride(0), y.data_ptr(), y.stride(0), N, K, J.data_ptr(),
                                     float(lamb), int(symmetric), _ptr(g_loss), _ptr(g_no_lamb), _ptr(gP),
                                     gx.data_ptr(), gy.data_ptr(), gx.stride(0), gy.stride(0),
                                     _stream(x.device))
    _lib.check(rc, "iic_global_backward")


def _as_oci(t: torch.Tensor) -> Tuple[int, int, int]:
    outer, C = t.shape[0], t.shape[1]
    inner = 1
    for s in t.shape[2:]:
        inner *= s
    return outer, C, inner


def _uda_forward(prob, target, kind, eps, weight, from_logits, check_simplex):
    lib = _lib.load()
    _require_cuda_f32("prob", prob)
    _require_cuda_f32("target", target)
    if prob.shape != target.shape or prob.dim() < 2:
        raise ValueError(f"iic_b200.uda_forward: shapes {tuple(prob.shape)} vs {tuple(target.shape)}")
    prob, target = prob.contiguous(), target.contiguous()
    outer, C, inner = _as_oci(prob)
    st = _state(prob.device)
    loss = torch.empty((), dtype=torch.float32, device=prob.device)
    if weight is not None:
        weight = weight.to(device=prob.device, dtype=torch.float32).contiguous()
    with torch.cuda.device(prob.device):
        rc = lib.iic_uda_forward(prob.data_ptr(), target.data_ptr(), outer, C, inner, kind, float(eps), _ptr(weight),
                                 int(from_logits), loss.data_ptr(), st.flags.data_ptr(), int(check_simplex),
                                 st.uda_ws.data_ptr(), _stream(prob.device))
    _lib.check(rc, "iic_uda_forward")
    return loss


def _uda_backward(prob, target, kind, eps, weight, from_logits, grad):
    lib = _lib.load()
    prob, target = prob.contiguous(), target.contiguous()
    outer, C, inner = _as_oci(prob)
    out = torch.empty_like(prob)
    grad = grad.to(torch.float32).reshape(())
    if weight is not None:
        weight = weight.to(device=prob.device, dtype=torch.float32).contiguous()
    with torch.cuda.device(prob.device):
        rc = lib.iic_uda_backward(prob.data_ptr(), target.data_ptr(), outer, C, inner, kind, float(eps), _ptr(weight),
                                  int(from_logits), grad.data_ptr(), out.data_ptr(), _stream(prob.device))
    _lib.check(rc, "iic_uda_backward")
    return out


def _simplex_check(t, axis):
    lib = _lib.load()
    _require_cuda_f32("tensor", t)
    if axis != 1:
        raise ValueError("iic_b200.simplex_check: only axis=1 is used by the reference path")
    t = t.contiguous()
    outer, C, inner = _as_oci(t)
    st = _state(t.device)
    with torch.cuda.device(t.device):
        rc = lib.iic_simplex_check(t.data_ptr(), outer, C, inner, C * inner, inner, st.flags.data_ptr(),
                                   _stream(t.device))
    _lib.check(rc, "iic_simplex_check")


def _flip_args(name, x, flips):
    _require_cuda_f32(name, x)
    if x.dim() != 4:
        raise ValueError(f"iic_b200.{name}: expected a (B, C, H, W) tensor, got {tuple(x.shape)}")
    if flips.dtype != torch.uint8 or flips.device != x.device or flips.shape != x.shape[:1]:
        raise TypeError(f"iic_b200.{name}: flips must be a uint8 tensor of shape ({x.shape[0]},) on {x.device}, got "
                        f"{flips.dtype} {tuple(flips.shape)} on {flips.device}")
    return x.contiguous(), flips.contiguous()


def _flip_batch(x, flips):
    lib = _lib.load()
    x, flips = _flip_args("flip_batch", x, flips)
    B, C, H, W = x.shape
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        rc = lib.iic_flip_batch(x.data_ptr(), out.data_ptr(), flips.data_ptr(), B, C, H, W, _stream(x.device))
    _lib.check(rc, "iic_flip_batch")
    return out


def _uda_flip_forward(prob, target, flips, kind, eps, from_logits):
    lib = _lib.load()
    prob, flips = _flip_args("uda_flip_forward", prob, flips)
    _require_cuda_f32("target", target)
    if prob.shape != target.shape:
        raise ValueError(f"iic_b200.uda_flip_forward: shapes {tuple(prob.shape)} vs {tuple(target.shape)}")
    target = target.contiguous()
    B, C, H, W = prob.shape
    st = _state(prob.device)
    loss = torch.empty((), dtype=torch.float32, device=prob.device)
    with torch.cuda.device(prob.device):
        rc = lib.iic_uda_flip_forward(prob.data_ptr(), target.data_ptr(), flips.data_ptr(), B, C, H, W, kind, float(eps),
                                      int(from_logits), loss.data_ptr(), st.flags.data_ptr(),
                                      st.uda_flip_ws(B, prob.device).data_ptr(), _stream(prob.device))
    _lib.check(rc, "iic_uda_flip_forward")
    return loss


def _uda_flip_backward(prob, target, flips, kind, eps, from_logits, grad):
    lib = _lib.load()
    prob, flips = _flip_args("uda_flip_backward", prob, flips)
    target = target.contiguous()
    B, C, H, W = prob.shape
    out = torch.empty_like(prob)
    grad = grad.to(torch.float32).reshape(())
    with torch.cuda.device(prob.device):
        rc = lib.iic_uda_flip_backward(prob.data_ptr(), target.data_ptr(), flips.data_ptr(), B, C, H, W, kind, float(eps),
                                       int(from_logits), grad.data_ptr(), out.data_ptr(), _stream(prob.device))
    _lib.check(rc, "iic_uda_flip_backward")
    return out


def _sup_args(logits, labels, weight):
    _require_cuda_f32("logits", logits)
    if labels.dtype != torch.int64 or labels.device != logits.device:
        raise TypeError(f"iic_b200.sup: labels must be an int64 tensor on {logits.device}, got {labels.dtype} on "
                        f"{labels.device}")
    if logits.dim() < 2 or labels.shape != logits.shape[:1] + logits.shape[2:]:
        raise ValueError(f"iic_b200.sup: logits {tuple(logits.shape)} need labels of shape "
                         f"{tuple(logits.shape[:1] + logits.shape[2:])}, got {tuple(labels.shape)}")
    if weight is not None:
        if weight.numel() != logits.shape[1]:
            raise ValueError(f"iic_b200.sup: {weight.numel()} class weights for {logits.shape[1]} classes")
        weight = weight.to(device=logits.device, dtype=torch.float32).contiguous()
    return logits.contiguous(), labels.contiguous(), weight


def _sup_forward(logits, labels, eps, weight, want_dice):
    lib = _lib.load()
    logits, labels, weight = _sup_args(logits, labels, weight)
    outer, C, inner = _as_oci(logits)
    st = _state(logits.device)
    loss = torch.empty((), dtype=torch.float32, device=logits.device)
    dice = torch.empty((2, outer, C) if want_dice else (0,), dtype=torch.int64, device=logits.device)
    with torch.cuda.device(logits.device):
        rc = lib.iic_sup_forward(logits.data_ptr(), labels.data_ptr(), outer, C, inner, float(eps), _ptr(weight),
                                 loss.data_ptr(), dice.data_ptr() if want_dice else None, st.flags.data_ptr(),
                                 st.supervised_ws(outer, logits.device).data_ptr(), _stream(logits.device))
    _lib.check(rc, "iic_sup_forward")
    return loss, dice


def _sup_backward(logits, labels, eps, weight, grad):
    lib = _lib.load()
    logits, labels, weight = _sup_args(logits, labels, weight)
    outer, C, inner = _as_oci(logits)
    out = torch.empty_like(logits)
    grad = grad.to(torch.float32).reshape(())
    with torch.cuda.device(logits.device):
        rc = lib.iic_sup_backward(logits.data_ptr(), labels.data_ptr(), outer, C, inner, float(eps), _ptr(weight),
                                  grad.data_ptr(), out.data_ptr(), _stream(logits.device))
    _lib.check(rc, "iic_sup_backward")
    return out


_LIBIMPL = torch.library.Library("iic_b200", "IMPL", "CUDA")
_LIBIMPL.impl("flip_batch", _flip_batch)
_LIBIMPL.impl("uda_flip_forward", _uda_flip_forward)
_LIBIMPL.impl("uda_flip_backward", _uda_flip_backward)
_LIBIMPL.impl("sup_forward", _sup_forward)
_LIBIMPL.impl("sup_backward", _sup_backward)
_LIBIMPL.impl("local_joint", _local_joint)
_LIBIMPL.impl("local_epilogue", _local_epilogue)
_LIBIMPL.impl("local_backward", _local_backward)
_LIBIMPL.impl("local_joint_logits", _local_joint_logits)
_LIBIMPL.impl("local_backward_logits", _local_backward_logits)
_LIBIMPL.impl("global_joint", _global_joint)
_LIBIMPL.impl("global_epilogue", _global_epilogue)
_LIBIMPL.impl("global_backward", _global_backward)
_LIBIMPL.impl("uda_forward", _uda_forward)
_LIBIMPL.impl("uda_backward", _uda_backward)
_LIBIMPL.impl("simplex_check", _simplex_check)


def _cpu_refusal(name):
    def fn(*a, **k):
        raise _lib.IICLibraryError(
            f"iic_b200::{name} has no CPU implementation: this package is the B200 CUDA path only. "
            "Move the tensors to a CUDA device.")
    return fn


_LIBCPU = torch.library.Library("iic_b200", "IMPL", "CPU")
for _n in ("local_joint", "local_epilogue", "local_backward", "local_joint_logits", "local_backward_logits", "global_joint", "global_epilogue",
           "global_backward", "uda_forward", "uda_backward", "simplex_check", "sup_forward", "sup_backward",
           "flip_batch", "uda_flip_forward", "uda_flip_backward"):
    _LIBCPU.impl(_n, _cpu_refusal(_n))

ops = torch.ops.iic_b200


# ---- data-parallel hook: one exchange of the partial joints ------------------------------------------
_process_group = None
_dist_enabled = False
_xchg = None          # PeerExchange, when the NVLink peer-memory exchange is set up
XCHG_CAPACITY = 1 << 18          # doubles per rank slot (2 MB): every joint of one iteration, e.g. config 3's 15 terms at K = 20
                                 # (118 k) or config 5's local + global joint at K = 128 (164 k)


class PeerExchange:
    """Exchange buffers of all ranks mapped into this process with CUDA IPC (csrc/xchg.cu).  Built collectively.

    Every rank runs the SAME sequence of collectives whatever fails locally (an allocation, an IPC import without peer
    access): local errors are recorded, the agreement all-reduce at the end decides for everybody, and a rank that
    failed releases what it had mapped.  ``ok`` tells whether the exchange is usable on ALL ranks."""

    def __init__(self, group, device: torch.device, capacity: int = None):
        import ctypes as C
        import torch.distributed as dist
        lib = _lib.load()
        capacity = XCHG_CAPACITY if capacity is None else capacity
        self.group, self.device, self.capacity = group, device, int(capacity)
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.ptrs = (C.c_void_p * self.world)()
        self._owned, self._imported, self.error = None, [], None
        handle = C.create_string_buffer(64)
        with torch.cuda.device(device):
            # phase 1 (local): allocate and export
            try:
                buf = C.c_void_p()
                _lib.check(lib.iic_xchg_create(self.world, self.capacity, C.byref(buf)), "iic_xchg_create")
                self._owned = buf.value
                _lib.check(lib.iic_xchg_export(buf, handle), "iic_xchg_export")
                mine = bytes(handle.raw)
            except Exception as e:  # noqa: BLE001
                self.error, mine = e, None
            # collective 1: everybody takes part, failed ranks contribute None
            handles = [None] * self.world
            dist.all_gather_object(handles, mine, group=group)
            # phase 2 (local): import the peers' buffers
            if self.error is None and all(h is not None for h in handles):
                try:
                    for r, h in enumerate(handles):
                        if r == self.rank:
                            self.ptrs[r] = self._owned
                        else:
                            peer = C.c_void_p()
                            _lib.check(lib.iic_xchg_import(C.create_string_buffer(h, 64), C.byref(peer)),
                                       f"iic_xchg_import(rank {r})")
                            self._imported.append(peer.value)
                            self.ptrs[r] = peer.value
                except Exception as e:  # noqa: BLE001
                    self.error = e
            elif self.error is None:
                self.error = RuntimeError("a peer could not create its exchange buffer")
            # collective 2: agreement (doubles as the barrier "every rank has mapped every buffer")
            ok = torch.tensor([0 if self.error is not None else 1], device=device)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
            self.ok = bool(int(ok.item()))
        if not self.ok:
            self.close()

    def close(self):
        """Unmap the peers' buffers and free the own one (idempotent)."""
        lib = _lib.load()
        with torch.cuda.device(self.device):
            for p in self._imported:
                lib.iic_xchg_release(p, 1)
            self._imported = []
            if self._owned is not None:
                torch.cuda.synchronize(self.device)
                lib.iic_xchg_release(self._owned, 0)
                self._owned = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def allreduce_(self, J: torch.Tensor) -> torch.Tensor:
        assert self.ok and J.dtype == torch.float64 and J.is_contiguous() and J.device == self.device
        lib = _lib.load()
        _lib.check(lib.iic_xchg_allreduce(J.data_ptr(), J.numel(), self.capacity, self.ptrs, self.rank, self.world,
                                          _state(self.device).flags.data_ptr(),
                                          torch.cuda.current_stream(self.device).cuda_stream), "iic_xchg_allreduce")
        return J


def set_data_parallel(enabled: bool, group=None, peer_memory=None):
    """When enabled, every joint (local and global) is summed over `group` with ONE exchange before
    the epilogue: each rank then holds the loss of the GLOBAL batch and the gradient of that loss with
    respect to its own shard (SURVEY.md section 8e).

    peer_memory: True  = the NVLink peer-memory exchange of csrc/xchg.cu (all ranks on one node, one GPU each;
                         collective call: every rank of `group` must make it), raising if it cannot be set up;
                 False = torch.distributed.all_reduce (NCCL);
                 None  = peer memory when the group is a single-node CUDA group of <= 16 ranks and the environment
                         variable IIC_B200_NO_P2P is unset, else NCCL."""
    global _process_group, _dist_enabled, _xchg
    _dist_enabled = bool(enabled)
    _process_group = group
    if _xchg is not None:
        _xchg.close()            # a previous call's buffers and IPC mappings
    _xchg = None
    if not _dist_enabled or peer_memory is False:
        return
    import os
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1):
        return
    auto = peer_memory is None
    if auto and (os.environ.get("IIC_B200_NO_P2P") or not torch.cuda.is_available() or dist.get_backend(group) != "nccl"
                 or dist.get_world_size(group) > 16
                 or int(os.environ.get("LOCAL_WORLD_SIZE", dist.get_world_size(group))) != dist.get_world_size(group)):
        return
    # PeerExchange runs the same collectives on every rank whatever fails locally and ends with an agreement step,
    # so either all ranks use peer memory or all of them fall back to NCCL
    px = PeerExchange(group, torch.device("cuda", torch.cuda.current_device()))
    if px.ok:
        _xchg = px
    elif not auto:
        raise RuntimeError(f"iic_b200: the peer-memory exchange could not be set up on every rank ({px.error})")


def ddp_loss_scale(group=None) -> float:
    """Factor for the IIC terms of a loss that is back-propagated under ``DistributedDataParallel``.

    With the joint exchange on, every rank holds the IIC loss L of the GLOBAL batch and its backward yields
    dL/d(activations of the local shard); the parameter gradient of L is therefore the SUM of the ranks' gradients
    (SURVEY.md section 7, "DDP semantics").  Stock DDP averages gradients, which is right for the per-rank means
    (supervised, UDA) and a factor world_size too small for L: multiply the IIC terms by this value.  1.0 when the
    exchange is off or no process group is up."""
    if not _dist_enabled:
        return 1.0
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return 1.0
    return float(dist.get_world_size(group if group is not None else _process_group))


def data_parallel_transport() -> str:
    """'peer_memory', 'nccl' or 'off' -- what _maybe_allreduce will use."""
    if not _dist_enabled:
        return "off"
    return "peer_memory" if _xchg is not None else "nccl"


def _maybe_allreduce(J: torch.Tensor) -> torch.Tensor:
    if _dist_enabled:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(_process_group) > 1:
            if _xchg is not None and J.is_cuda and J.numel() <= _xchg.capacity:
                return _xchg.allreduce_(J if J.is_contiguous() else J.contiguous())
            dist.all_reduce(J, op=dist.ReduceOp.SUM, group=_process_group)
    return J


# ---- one or many IIC terms through ONE finish launch (csrc/finish.cu) ------------------------------------
class LocalTerm:
    """One local IIC call: IIDSegmentationLoss / IIDSegmentationSmallPathLoss on (x, y[, mask]); `logits` = the inputs are
    the cluster head's logits and the softmax is fused into the kernels (one patch, no mask)."""
    __slots__ = ("x", "y", "mask", "pad", "patch", "step", "lamda", "logits", "inv_temperature")

    def __init__(self, x, y, mask, pad, patch, step, lamda, logits=False, inv_temperature=1.0):
        self.x, self.y, self.mask = x, y, mask
        self.pad, self.patch, self.step, self.lamda = int(pad), (int(patch[0]), int(patch[1])), (int(step[0]), int(step[1])), float(lamda)
        self.logits, self.inv_temperature = bool(logits), float(inv_temperature)


class GlobalTerm:
    """One global IIC call: IIDLoss / compute_joint on (N, K) rows."""
    __slots__ = ("x", "y", "lamb", "symmetric", "want_losses")

    def __init__(self, x, y, lamb=1.0, symmetric=True, want_losses=True):
        self.x, self.y, self.lamb, self.symmetric, self.want_losses = x, y, float(lamb), bool(symmetric), bool(want_losses)


MAX_TERMS_PER_FINISH = 32
GLOBAL_ROWS_MAX = 4096          # larger (N, K) inputs take the multi-CTA global joint kernel instead of iic_finish


def _world():
    if _dist_enabled:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            return dist.get_world_size(_process_group)
    return 1


def _finish_terms(terms, check_simplex):
    """Joint kernels of every term, then ONE iic_finish launch (slot reduction, the multi-GPU exchange of ALL joints,
    the epilogues).  Returns per term a dict of what its backward needs and its outputs."""
    import ctypes as C
    lib = _lib.load()
    assert 0 < len(terms) <= MAX_TERMS_PER_FINISH
    for t in terms:                      # before any device state is touched: CPU tensors are refused loudly
        _require_cuda_f32("x_out", t.x)
        _require_cuda_f32("x_tf_out", t.y)
    dev = terms[0].x.device
    st = _state(dev)
    flags = st.flags.data_ptr()
    items = (_lib.FinishItem * len(terms))()
    keep, recs, E_total = [], [], 0
    n_loss = sum(1 if isinstance(t, LocalTerm) else 2 for t in terms)
    loss_buf = torch.empty(n_loss, dtype=torch.float32, device=dev)
    lo = 0
    with torch.cuda.device(dev):
        for i, t in enumerate(terms):
            it = items[i]
            if isinstance(t, LocalTerm):
                _require_cuda_f32("x_out", t.x)
                _require_cuda_f32("x_tf_out", t.y)
                if t.x.dim() != 4 or t.x.shape != t.y.shape:
                    raise ValueError(f"iic_b200: local term shapes {tuple(t.x.shape)} vs {tuple(t.y.shape)}")
                x, y = _w_contig(t.x), _w_contig(t.y)
                B, K, H, W = x.shape
                info = _lib.SlotInfo()
                if t.logits:
                    nbytes = max(lib.iic_b200_sm_count(dev.index or 0) * 9 * K * K * 4, 4)
                    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
                    rc = lib.iic_local_joint_from_logits(x.data_ptr(), x.stride(0), x.stride(1), x.stride(2),
                                                         y.data_ptr(), y.stride(0), y.stride(1), y.stride(2),
                                                         B, K, H, W, t.pad, t.inv_temperature, None, ws.data_ptr(), nbytes,
                                                         C.byref(info), _stream(dev))
                    if rc == _lib.UNSUPPORTED:
                        raise FusedShapeUnsupported(lib.iic_b200_last_error().decode())
                    _lib.check(rc, "iic_local_joint_from_logits")
                    npatch, m = 1, None
                else:
                    m, msn, msc, msh = _mask_args(t.mask, x)
                    npatch = lib.iic_local_num_patches(H, W, t.patch[0], t.patch[1], t.step[0], t.step[1])
                    if npatch <= 0:
                        _lib.check(1, "iic_local_num_patches")
                    nbytes = lib.iic_local_joint_workspace_bytes(dev.index or 0, B, K, H, W, t.pad, t.patch[0], t.patch[1],
                                                                 t.step[0], t.step[1])
                    if nbytes == 0:
                        _lib.check(1, "iic_local_joint_workspace_bytes")
                    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
                    fl = None
                    if check_simplex:
                        if x.stride(2) == W:
                            fl = flags
                        else:
                            _simplex_check(x, 1)
                    _lib.check(lib.iic_local_joint_partials(
                        x.data_ptr(), x.stride(0), x.stride(1), x.stride(2), y.data_ptr(), y.stride(0), y.stride(1),
                        y.stride(2), _ptr(m), msn, msc, msh, B, K, H, W, t.pad, t.patch[0], t.patch[1], t.step[0], t.step[1],
                        ws.data_ptr(), nbytes, fl, C.byref(info), _stream(dev)), "iic_local_joint_partials")
                T = 2 * t.pad + 1
                ncoef = lib.iic_local_coeff_floats(K, t.pad, npatch)
                Wx = torch.empty(ncoef, dtype=torch.float32, device=dev)
                Wy = torch.empty(ncoef, dtype=torch.float32, device=dev)
                it.kind, it.K, it.lamda = _lib.ITEM_LOCAL, K, t.lamda
                it.slots, it.layout, it.n_slots, it.nb, it.slot_stride = ws.data_ptr(), info.layout, info.n_slots, info.nb, info.slot_stride
                it.pad, it.n_patches = t.pad, npatch
                it.epilogue_workspace = st.epilogue_ws(K, t.pad, npatch, dev).data_ptr()      # used when the epilogue is not fused
                it.loss_out, it.Wx, it.Wy = loss_buf[lo:].data_ptr(), Wx.data_ptr(), Wy.data_ptr()
                E = npatch * T * T * K * K
                recs.append(dict(kind="local", x=x, y=y, mask=m, Wx=Wx, Wy=Wy, loss=loss_buf[lo], K=K, T=T, npatch=npatch,
                                 joff=E_total, E=E))
                keep.append(ws)
                lo += 1
            else:
                _require_cuda_f32("x_out", t.x)
                _require_cuda_f32("x_tf_out", t.y)
                if t.x.dim() != 2 or t.x.shape != t.y.shape:
                    raise ValueError(f"iic_b200: global term shapes {tuple(t.x.shape)} vs {tuple(t.y.shape)}")
                x, y = _w_contig(t.x), _w_contig(t.y)
                N, K = x.shape
                P = torch.empty((K, K), dtype=torch.float32, device=dev)
                it.kind, it.K, it.lamda = _lib.ITEM_GLOBAL_ROWS, K, t.lamb
                it.x, it.x_sn, it.y, it.y_sn, it.N = x.data_ptr(), x.stride(0), y.data_ptr(), y.stride(0), N
                it.symmetric, it.check_simplex = int(t.symmetric), int(bool(check_simplex))
                it.loss_out, it.P_out = loss_buf[lo:].data_ptr(), P.data_ptr()
                E = K * K
                recs.append(dict(kind="global", x=x, y=y, P=P, loss=loss_buf[lo], loss_nl=loss_buf[lo + 1], K=K, joff=E_total,
                                 E=E))
                lo += 2
            E_total += E
        J_all = torch.empty(E_total, dtype=torch.float64, device=dev)
        world = _world()
        fused_xchg = world > 1 and _xchg is not None and E_total <= _xchg.capacity
        if world > 1 and not fused_xchg:
            # NCCL transport (or joints larger than the peer slots): reduce here, all-reduce, then the epilogue launches
            _lib.check(lib.iic_finish(items, len(terms), J_all.data_ptr(), E_total, flags, st.fin_ws.data_ptr(), None, 0, 1, 0,
                                      0, _stream(dev)), "iic_finish")
            import torch.distributed as dist
            dist.all_reduce(J_all, op=dist.ReduceOp.SUM, group=_process_group)
            for i, (t, r) in enumerate(zip(terms, recs)):
                Jv = J_all[r["joff"]:r["joff"] + r["E"]]
                if r["kind"] == "local":
                    _lib.check(lib.iic_local_epilogue(Jv.data_ptr(), r["K"], t.pad, r["npatch"], t.lamda, items[i].loss_out, None,
                                                      r["Wx"].data_ptr(), r["Wy"].data_ptr(), None, flags,
                                                      st.epilogue_ws(r["K"], t.pad, r["npatch"], dev).data_ptr(), _stream(dev)),
                               "iic_local_epilogue")
                else:
                    _lib.check(lib.iic_global_epilogue(Jv.data_ptr(), r["K"], t.lamb, int(t.symmetric), items[i].loss_out,
                                                       r["P"].data_ptr(), flags, _stream(dev)), "iic_global_epilogue")
        else:
            _lib.check(lib.iic_finish(items, len(terms), J_all.data_ptr(), E_total, flags, st.fin_ws.data_ptr(),
                                      _xchg.ptrs if fused_xchg else None, _xchg.rank if fused_xchg else 0,
                                      world if fused_xchg else 1, _xchg.capacity if fused_xchg else 0, 1, _stream(dev)),
                       "iic_finish")
    del keep
    for r in recs:
        r["J"] = J_all[r["joff"]:r["joff"] + r["E"]]
    return recs


def _block_of(t: torch.Tensor):
    """(base, n0, c0) when `t` is the block ``base.view(N, C, *spatial)[n0:n0+B, c0:c0+K]`` of a contiguous tensor it is a
    differentiable VIEW of -- what ``chunk`` / ``unbind`` / slicing of a batched cluster-head output give
    (contrastyou/trainer/_utils.py:137-168, semi_seg/epocher.py:269-273).  The gradient of such a view can be written
    straight into its block of the base's gradient instead of going through autograd's view backward (a zero-filled
    full-size tensor plus a copy per view).  None for leaves and for anything that is not such a block."""
    if t.is_leaf or t._base is None:
        return None
    base = t._base
    if not (base.requires_grad and base.is_contiguous() and base.dtype == t.dtype and base.dim() >= t.dim()):
        return None
    N = base.shape[0]
    if N == 0:
        return None
    if t.dim() == 4:
        B, K, H, W = t.shape
        if tuple(base.shape[-2:]) != (H, W):
            return None
        plane = H * W
        C = base.numel() // (N * plane)
        want = (C * plane, plane, W, 1)
    else:
        B, K = t.shape
        plane = 1
        C = base.numel() // N
        want = (C, 1)
    st = t.stride()
    if any(sz > 1 and a != b for sz, a, b in zip(t.shape, st, want)):
        return None
    off = t.storage_offset() - base.storage_offset()
    n0, rem = divmod(off, C * plane)
    c0, r2 = divmod(rem, plane)
    if off < 0 or r2 or n0 + B > N or c0 + K > C:
        return None
    return base, n0, c0


def _block_view(G: torch.Tensor, like: torch.Tensor, n0: int, c0: int) -> torch.Tensor:
    N = G.shape[0]
    if like.dim() == 4:
        B, K, H, W = like.shape
        return G.view(N, -1, H, W)[n0:n0 + B, c0:c0 + K]
    B, K = like.shape
    return G.view(N, -1)[n0:n0 + B, c0:c0 + K]


def _region(v: torch.Tensor, blk, src: torch.Tensor):
    """The part of `src` that the use `v` (block `blk` = (n0, c0) of it, or None = all of it) covers, as
    (first row, end row, first element, end element) with elements counted inside one row of `src`."""
    N = src.shape[0]
    if blk is None:
        return (0, N, 0, src.numel() // N if N else 0)
    B, K = v.shape[:2]
    plane = math.prod(v.shape[2:])
    return (blk[0], blk[0] + B, blk[1] * plane, (blk[1] + K) * plane)


def _intersect(a, b) -> bool:
    return (a[0] < a[1] and a[2] < a[3] and b[0] < b[1] and b[2] < b[3]
            and a[0] < b[1] and b[0] < a[1] and a[2] < b[3] and b[2] < a[3])


class IICTermsFunction(torch.autograd.Function):
    """The losses of one or many IIC terms -- local (iic_loss.py:107-149,171-186) and global (iic_loss.py:43-94) -- from
    ONE finish launch.  apply(terms, check_simplex, slots, *sources): `terms` carries geometry and the input views,
    `sources` the distinct differentiable tensors behind them, `slots[2*i]`, `slots[2*i+1]` = (source index, block or
    None) for x and y of term i.  Outputs per local term: loss; per global term: loss, loss_no_lamb, P.  In backward
    every term's gradient kernel writes directly into its block of the source's gradient -- or into a temporary that is
    added to the block, when the same block was written before or when the source's regions overlap."""

    @staticmethod
    def forward(ctx, terms, check_simplex, slots, *sources):
        recs = _finish_terms(terms, check_simplex)
        outs, saved = [], []
        for r in recs:
            if r["kind"] == "local":
                outs.append(r["loss"])
                saved += [r["x"], r["y"], r["Wx"], r["Wy"]] + ([r["mask"]] if r["mask"] is not None else [])
            else:
                outs += [r["loss"], r["loss_nl"], r["P"]]
                saved += [r["x"], r["y"], r["J"]]
        ctx.save_for_backward(*saved)
        ctx.meta = [(t.__class__, getattr(t, "pad", None), getattr(t, "patch", None), getattr(t, "step", None),
                     getattr(t, "logits", False), getattr(t, "inv_temperature", 1.0), getattr(t, "lamb", None),
                     getattr(t, "symmetric", True), r.get("mask") is not None, r.get("npatch", 1))
                    for t, r in zip(terms, recs)]
        ctx.slots = slots
        ctx.src_meta = [(tuple(s_.shape), s_.device) for s_ in sources]
        # a source whose distinct blocks tile it completely needs no zero fill
        cover = [0] * len(sources)
        seen = set()
        for k, (si, blk) in enumerate(slots):
            t = terms[k // 2]
            v = t.x if k % 2 == 0 else t.y
            if blk is not None and (si, blk) not in seen:
                seen.add((si, blk))
                cover[si] += v.numel()
        # a source with two distinct regions that intersect (overlapping blocks, or the whole tensor and a block of it):
        # every use then adds into a zero-filled buffer
        regions = [set() for _ in sources]
        for k, (si, blk) in enumerate(slots):
            t = terms[k // 2]
            regions[si].add(_region(t.x if k % 2 == 0 else t.y, blk, sources[si]))
        ctx.overlap = [any(_intersect(a, b) for a in rs for b in rs if a < b) for rs in regions]
        ctx.covered = [c == s_.numel() and not o for c, s_, o in zip(cover, sources, ctx.overlap)]
        ctx.set_materialize_grads(False)
        return tuple(outs)

    @staticmethod
    def backward(ctx, *grads):
        sv = list(ctx.saved_tensors)
        slots = ctx.slots
        n_src = len(ctx.src_meta)
        # which sources get a complete set of gradients (then their buffer need not be zeroed)
        gi, need_zero, any_grad = 0, [False] * n_src, [False] * n_src
        for ti, m in enumerate(ctx.meta):
            n_out = 1 if m[0] is LocalTerm else 3
            has = any(g is not None for g in grads[gi:gi + n_out])
            gi += n_out
            for k in (2 * ti, 2 * ti + 1):
                si, blk = slots[k]
                if has:
                    any_grad[si] = True
                if (blk is not None and not has) or (has and m[9] > 1):
                    need_zero[si] = True          # a block nobody writes, or patches that accumulate into their output
        G = [None] * n_src
        written = set()

        def target(k, like):
            """Where the gradient of input k goes: (tensor to write into, accumulate-from-temp?)."""
            si, blk = slots[k]
            shape, dev = ctx.src_meta[si]
            if G[si] is None:
                zero = need_zero[si] or ctx.overlap[si] or (blk is not None and not ctx.covered[si])
                G[si] = (torch.zeros if zero else torch.empty)(shape, dtype=torch.float32, device=dev)
            dst = G[si] if blk is None else _block_view(G[si], like, blk[0], blk[1])
            if ctx.overlap[si] or (si, blk) in written:
                # second use of the block, or a region that another use overlaps: add afterwards
                return torch.zeros_like(like, memory_format=torch.contiguous_format), dst
            written.add((si, blk))
            return dst, None

        # The global terms' gradient kernels are one small CTA each (~7 us of latency-bound work at (32, 10)); the local ones
        # fill the GPU for ~75 us with one persistent CTA per SM.  With both kinds present the global ones go to a side
        # stream that forks BEFORE the local launches and is joined after them: inside a captured CUDA graph they are
        # parallel branches, and the small CTA (128 threads) fits on an SM beside a local-backward CTA.  The global kernels
        # are launched after the local ones, so that they never hold an SM the persistent kernel is waiting for.
        n_local = sum(1 for m in ctx.meta if m[0] is LocalTerm)
        use_side = overlap_global_backward and n_local > 0 and n_local < len(ctx.meta)
        side, main, deferred, gjobs = None, None, [], []
        # saved-tensor and gradient offsets of every term
        offs, gi, si_ = [], 0, 0
        for m in ctx.meta:
            offs.append((si_, gi))
            if m[0] is LocalTerm:
                si_ += 4 + (1 if m[8] else 0)
                gi += 1
            else:
                si_ += 3
                gi += 3
        order = list(range(len(ctx.meta)))
        if use_side:
            # global terms first: their targets are allocated (and zero-filled where needed) on the main stream before the fork
            order.sort(key=lambda t_: ctx.meta[t_][0] is LocalTerm)
        for ti in order:
            cls, pad, patch, step, logits, inv_t, lamb, symmetric, has_mask, npatch = ctx.meta[ti]
            si_, gi = offs[ti]
            if cls is LocalTerm:
                if use_side and side is None and gjobs:
                    main = torch.cuda.current_stream(sv[si_].device)
                    side = _side_stream(sv[si_].device)
                    side.wait_stream(main)        # fork: upstream gradients and the global targets' zero fills are queued on main
                x, y, Wx, Wy = sv[si_:si_ + 4]
                mask = sv[si_ + 4] if has_mask else None
                g = grads[gi]
                if g is None:
                    continue
                (gx, ax), (gy, ay) = target(2 * ti, x), target(2 * ti + 1, y)
                if logits:
                    _local_backward_logits_into(x, y, Wx, Wy, g.contiguous(), pad, inv_t, gx, gy)
                else:
                    _local_backward_into(x, y, mask, Wx, Wy, g.contiguous(), pad, patch[0], patch[1], step[0], step[1], gx, gy)
            else:
                x, y, J = sv[si_:si_ + 3]
                g1, g2, gP = grads[gi:gi + 3]
                if g1 is None and g2 is None and gP is None:
                    continue
                (gx, ax), (gy, ay) = target(2 * ti, x), target(2 * ti + 1, y)
                if use_side:
                    gjobs.append((x, y, J, lamb, symmetric, g1, g2, gP, gx, gy, ax, ay))
                    continue
                _global_backward_into(x, y, J.view(x.shape[1], x.shape[1]), lamb, symmetric, g1, g2, gP, gx, gy)
            if ax is not None:
                ax += gx
            if ay is not None:
                ay += gy
        if gjobs:
            if side is None:                      # no local term had a gradient after all: plain launches
                for (x, y, J, lamb, symmetric, g1, g2, gP, gx, gy, ax, ay) in gjobs:
                    _global_backward_into(x, y, J.view(x.shape[1], x.shape[1]), lamb, symmetric, g1, g2, gP, gx, gy)
                    if ax is not None:
                        ax += gx
                    if ay is not None:
                        ay += gy
            else:
                with torch.cuda.stream(side):
                    for (x, y, J, lamb, symmetric, g1, g2, gP, gx, gy, ax, ay) in gjobs:
                        _global_backward_into(x, y, J.view(x.shape[1], x.shape[1]), lamb, symmetric, g1, g2, gP, gx, gy)
                        if ax is not None:
                            deferred.append((ax, gx))
                        if ay is not None:
                            deferred.append((ay, gy))
                main.wait_stream(side)            # join: every later reader (and the allocator) sees the side work done
                for acc, g_ in deferred:
                    acc += g_
        return (None, None, None, *[G[i] if any_grad[i] else None for i in range(n_src)])


def iic_terms(terms, check_simplex=False):
    """Evaluate many IIC terms together; returns a list with, per term, the loss (LocalTerm) or the tuple
    (loss, loss_no_lamb, P) (GlobalTerm).  Global terms with more than GLOBAL_ROWS_MAX rows and batches beyond
    MAX_TERMS_PER_FINISH are split off transparently."""
    terms = list(terms)
    out = [None] * len(terms)
    batch = [i for i, t in enumerate(terms) if isinstance(t, LocalTerm) or t.x.shape[0] <= GLOBAL_ROWS_MAX]
    for i, t in enumerate(terms):
        if i not in batch:
            out[i] = _GlobalIICMultiCTAFunction.apply(t.x, t.y, t.lamb, t.symmetric, check_simplex)
    for c0 in range(0, len(batch), MAX_TERMS_PER_FINISH):
        idx = batch[c0:c0 + MAX_TERMS_PER_FINISH]
        sub = [terms[i] for i in idx]
        sources, index, slots = [], {}, []
        for t in sub:
            for v in (t.x, t.y):
                blk = _block_of(v) if torch.is_grad_enabled() and v.requires_grad else None
                src = blk[0] if blk is not None else v
                if id(src) not in index:
                    index[id(src)] = len(sources)
                    sources.append(src)
                slots.append((index[id(src)], (blk[1], blk[2]) if blk is not None else None))
        res = list(IICTermsFunction.apply(sub, check_simplex, slots, *sources))
        for i, t in zip(idx, sub):
            if isinstance(t, LocalTerm):
                out[i] = res.pop(0)
            else:
                out[i] = (res.pop(0), res.pop(0), res.pop(0))
    return out


# ---- autograd ------------------------------------------------------------------------------------------
class LocalIICFunction(torch.autograd.Function):
    """loss = mean over patches of the shifted-window IIC loss (iic_loss.py:107-149, 171-186): joint kernel, one finish
    launch (slot reduction [+ exchange] + epilogue), and in backward one gradient kernel."""

    @staticmethod
    def forward(ctx, x, y, mask, pad, patch_h, patch_w, step_h, step_w, lamda, check_simplex=False):
        t = LocalTerm(x, y, mask, pad, (patch_h, patch_w), (step_h, step_w), lamda)
        (r,) = _finish_terms([t], check_simplex)
        ctx.save_for_backward(r["x"], r["y"], r["mask"], r["Wx"], r["Wy"])
        ctx.geom = (pad, patch_h, patch_w, step_h, step_w)
        return r["loss"]

    @staticmethod
    def backward(ctx, grad):
        x, y, mask, Wx, Wy = ctx.saved_tensors
        gx, gy = ops.local_backward(x, y, mask, Wx, Wy, grad.contiguous(), *ctx.geom)
        return gx, gy, None, None, None, None, None, None, None, None


class LocalIICLogitsFunction(torch.autograd.Function):
    """LocalIICFunction applied to softmax(logits / T, dim=1) of both maps, with the softmax and its
    backward fused into the joint and gradient kernels (contrastyou/trainer/_utils.py:15-23,137-168 feeding
    iic_loss.py:107-149); one patch = the whole map.  Raises FusedShapeUnsupported for other shapes."""

    @staticmethod
    def forward(ctx, lx, ly, pad, lamda, inv_temperature):
        t = LocalTerm(lx, ly, None, pad, lx.shape[2:], lx.shape[2:], lamda, logits=True, inv_temperature=inv_temperature)
        (r,) = _finish_terms([t], False)
        ctx.save_for_backward(r["x"], r["y"], r["Wx"], r["Wy"])
        ctx.cfg = (pad, inv_temperature)
        return r["loss"]

    @staticmethod
    def backward(ctx, grad):
        lx, ly, Wx, Wy = ctx.saved_tensors
        gx, gy = ops.local_backward_logits(lx, ly, Wx, Wy, grad.contiguous(), *ctx.cfg)
        return gx, gy, None, None, None


class _GlobalIICMultiCTAFunction(torch.autograd.Function):
    """(loss, loss_no_lamb, P) of IIDLoss.forward (iic_loss.py:43-71) for LARGE N: multi-CTA joint, exchange, epilogue."""

    @staticmethod
    def forward(ctx, x, y, lamb, symmetric=True, check_simplex=False):
        J = _maybe_allreduce(ops.global_joint(x, y, check_simplex))
        losses, P = ops.global_epilogue(J, lamb, symmetric, True)
        ctx.save_for_backward(x, y, J)
        ctx.cfg = (lamb, symmetric)
        ctx.set_materialize_grads(False)     # unused outputs arrive as None, not as zero tensors
        return losses[0], losses[1], P

    @staticmethod
    def backward(ctx, g1, g2, gP):
        x, y, J = ctx.saved_tensors
        gx, gy = ops.global_backward(x, y, J, ctx.cfg[0], ctx.cfg[1], g1, g2, gP)
        return gx, gy, None, None, None


class GlobalIICFunction(torch.autograd.Function):
    """(loss, loss_no_lamb, P) of IIDLoss.forward (iic_loss.py:43-71): for the udaiic sizes (N <= 4096 rows) ONE launch --
    iic_finish computes the joint from the rows, exchanges it under data parallelism and runs the epilogue."""

    @staticmethod
    def forward(ctx, x, y, lamb, check_simplex=False):
        ctx.set_materialize_grads(False)     # unused outputs arrive as None, not as zero tensors
        ctx.lamb = lamb
        if x.dim() == 2 and x.shape[0] > GLOBAL_ROWS_MAX:
            J = _maybe_allreduce(ops.global_joint(x, y, check_simplex))
            losses, P = ops.global_epilogue(J, lamb, True, True)
            ctx.save_for_backward(x, y, J)
            return losses[0], losses[1], P
        (r,) = _finish_terms([GlobalTerm(x, y, lamb, True)], check_simplex)
        ctx.save_for_backward(r["x"], r["y"], r["J"].view(r["K"], r["K"]))
        return r["loss"], r["loss_nl"], r["P"]

    @staticmethod
    def backward(ctx, g1, g2, gP):
        x, y, J = ctx.saved_tensors
        gx, gy = ops.global_backward(x, y, J, ctx.lamb, True, g1, g2, gP)
        return gx, gy, None, None


class JointFunction(torch.autograd.Function):
    """P = compute_joint(x, y, symmetric) (iic_loss.py:74-94)."""

    @staticmethod
    def forward(ctx, x, y, symmetric, check_simplex=False):
        J = _maybe_allreduce(ops.global_joint(x, y, check_simplex))
        _, P = ops.global_epilogue(J, 1.0, symmetric, False)
        ctx.save_for_backward(x, y, J)
        ctx.symmetric = symmetric
        return P

    @staticmethod
    def backward(ctx, gP):
        x, y, J = ctx.saved_tensors
        gx, gy = ops.global_backward(x, y, J, 1.0, ctx.symmetric, None, None, gP)
        return gx, gy, None, None


class UDAFunction(torch.autograd.Function):
    """MSE / KL consistency (semi_seg/epocher.py:221-224); the gradient flows to `prob` only."""

    @staticmethod
    def forward(ctx, prob, target, kind, eps, weight, from_logits, check_simplex):
        loss = ops.uda_forward(prob, target, kind, eps, weight, from_logits, check_simplex)
        ctx.save_for_backward(prob, target, weight)
        ctx.cfg = (kind, eps, from_logits)
        return loss

    @staticmethod
    def backward(ctx, grad):
        prob, target, weight = ctx.saved_tensors
        kind, eps, from_logits = ctx.cfg
        g = ops.uda_backward(prob, target, kind, eps, weight, from_logits, grad.contiguous())
        return g, None, None, None, None, None, None


class SupervisedKLFunction(torch.autograd.Function):
    """KL_div()(softmax(logits), one_hot(labels)) (semi_seg/epocher.py:165-166) and the Dice counts of the
    `sup_dice` meter (epocher.py:183-184) from one pass over the logits; the gradient flows to `logits` only."""

    @staticmethod
    def forward(ctx, logits, labels, eps, weight, want_dice):
        loss, dice = ops.sup_forward(logits, labels, eps, weight, want_dice)
        ctx.save_for_backward(logits, labels, weight)
        ctx.eps = eps
        ctx.mark_non_differentiable(dice)
        return loss, dice

    @staticmethod
    def backward(ctx, grad, _grad_dice):
        logits, labels, weight = ctx.saved_tensors
        g = ops.sup_backward(logits, labels, ctx.eps, weight, grad.contiguous())
        return g, None, None, None, None


class FlipBatchFunction(torch.autograd.Function):
    """Per-sample flips of a (B, C, H, W) batch in one launch (semi_seg/epocher.py:148-149,160-161,264-266).  A flip
    is a permutation and its own inverse, so the backward is the same kernel on the incoming gradient."""

    @staticmethod
    def forward(ctx, x, flips):
        ctx.save_for_backward(flips)
        return ops.flip_batch(x, flips)

    @staticmethod
    def backward(ctx, grad):
        (flips,) = ctx.saved_tensors
        return ops.flip_batch(grad.contiguous(), flips), None


class UDAFlipFunction(torch.autograd.Function):
    """UDAFunction with the target read through per-sample flips (the flipped copy is never materialised)."""

    @staticmethod
    def forward(ctx, prob, target, flips, kind, eps, from_logits):
        loss = ops.uda_flip_forward(prob, target, flips, kind, eps, from_logits)
        ctx.save_for_backward(prob, target, flips)
        ctx.cfg = (kind, eps, from_logits)
        return loss

    @staticmethod
    def backward(ctx, grad):
        prob, target, flips = ctx.saved_tensors
        kind, eps, from_logits = ctx.cfg
        g = ops.uda_flip_backward(prob, target, flips, kind, eps, from_logits, grad.contiguous())
        return g, None, None, None, None, None
