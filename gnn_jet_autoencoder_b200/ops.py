"""Thin torch custom-op layer over the C-ABI library (north star: "Python/PyTorch host code calls
hand-written sm_100a CUDA kernels through a thin C-ABI torch custom-op layer").

Two levels:
  * ``raw_*`` functions: pointer-level calls used by the captured training step (``trainer.py``);
    no allocation, no autograd, safe under CUDA-graph capture.
  * ``torch.ops.gnnjet.*`` custom ops (CUDA only -- there is no CPU implementation, so a CPU tensor
    raises) plus the autograd glue the nn.Modules use.
"""
from __future__ import annotations

import functools
from typing import List, Sequence, Tuple

import torch
from torch import Tensor

from . import _lib
from ._lib import GJ_METRIC_EUCLIDEAN, GJ_METRIC_MINKOWSKIAN, GJ_PREC_BF16, GJ_PREC_FP32  # noqa: F401

PRECISIONS = {"fp32": GJ_PREC_FP32, "float32": GJ_PREC_FP32, "bf16": GJ_PREC_BF16, "bfloat16": GJ_PREC_BF16}

# number of kernels of this library launched through this module (bench.py's "gpu_launches" claim)
LAUNCHES = {"count": 0}


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _on_device(fn):
    """Runs an op body with the operands' GPU as the current device (the C launchers use cudaGetDevice() and the current
    stream of the current device; the reference accepts e.g. ``device='cuda:1'`` while device 0 is current) and checks that
    all tensor operands live on one device."""
    @functools.wraps(fn)
    def wrapper(*args, **kw):
        tens = [a for a in list(args) + list(kw.values()) if isinstance(a, Tensor)]
        if not tens or not tens[0].is_cuda:
            return fn(*args, **kw)          # _req raises the "no CPU implementation" error
        dev = tens[0].device
        for t in tens[1:]:
            if t.device != dev:
                raise _lib.GnnJetError(f"all operands must live on one device: got {dev} and {t.device}")
        with torch.cuda.device(dev):
            return fn(*args, **kw)
    return wrapper


def _ptr(t):
    return None if t is None else t.data_ptr()


def _req(t: Tensor, name: str) -> Tensor:
    if not t.is_cuda:
        raise _lib.GnnJetError(f"{name} must be a CUDA tensor: the GraphNet path has no CPU implementation")
    if t.dtype != torch.float32:
        raise _lib.GnnJetError(f"{name} must be float32 (got {t.dtype})")
    return t.contiguous()


def metric_id(metric) -> int:
    """graphnet.py:314-327: only 'minkowskian' selects the Minkowskian form; unknown names fall back
    to euclidean (the reference logs a warning).  The width-4 gate of graphnet.py:155 is applied in
    the kernel."""
    return GJ_METRIC_MINKOWSKIAN if str(metric).lower() == "minkowskian" else GJ_METRIC_EUCLIDEAN


# --------------------------------------------------------------------------------------------------
# pointer-level calls
# --------------------------------------------------------------------------------------------------
def _step_launches(desc, backward: bool, saved: bool = False) -> int:
    """Kernel launches of one gj_mp_step_fwd / gj_mp_step_bwd call (the bench's gpu_launches claim), as the library counts
    them for this descriptor (gj_mp_step_launches)."""
    return int(_lib.load().gj_mp_step_launches(desc, 1 if backward else 0, 1 if saved else 0))


def raw_mp_fwd(desc, h_ptr, params_ptr, hout_ptr, e_ptr, ws_ptr, ws_bytes, stream, saved_ptr=None):
    lib = _lib.load()
    if saved_ptr:
        _lib.check(lib.gj_mp_step_fwd_saving(desc, h_ptr, params_ptr, hout_ptr, e_ptr, saved_ptr, ws_ptr, ws_bytes, stream),
                   "gj_mp_step_fwd_saving")
    else:
        _lib.check(lib.gj_mp_step_fwd(desc, h_ptr, params_ptr, hout_ptr, e_ptr, ws_ptr, ws_bytes, stream), "gj_mp_step_fwd")
    LAUNCHES["count"] += _step_launches(desc, False)


def raw_mp_bwd(desc, h_ptr, e_ptr, params_ptr, dhout_ptr, dh_ptr, dparams_ptr, ws_ptr, ws_bytes, stream, saved_ptr=None):
    lib = _lib.load()
    if saved_ptr:
        _lib.check(lib.gj_mp_step_bwd_saved(desc, h_ptr, e_ptr, params_ptr, dhout_ptr, dh_ptr, dparams_ptr, saved_ptr, ws_ptr,
                                            ws_bytes, stream), "gj_mp_step_bwd_saved")
    else:
        _lib.check(lib.gj_mp_step_bwd(desc, h_ptr, e_ptr, params_ptr, dhout_ptr, dh_ptr, dparams_ptr, ws_ptr, ws_bytes,
                                      stream), "gj_mp_step_bwd")
    LAUNCHES["count"] += _step_launches(desc, True, bool(saved_ptr))


# ---- a chain of steps with per-chain helper launches (include/gnnjet_b200.h: gj_mp_steps_pack / gj_mp_steps_reduce) ----
def _ptr_array(ptrs):
    return (_lib.C.c_void_p * len(ptrs))(*[int(p) for p in ptrs])


def _desc_array(descs):
    return (_lib.C.POINTER(_lib.MPDesc) * len(descs))(*[_lib.C.pointer(d) for d in descs])


def raw_mp_pack_steps(descs, params_ptrs, saved_ptrs, stream):
    """ONE launch packs the bf16 edge-parameter images of all steps into their ``saved`` buffers."""
    _lib.check(_lib.load().gj_mp_steps_pack(len(descs), _desc_array(descs), _ptr_array(params_ptrs), _ptr_array(saved_ptrs), stream),
               "gj_mp_steps_pack")
    LAUNCHES["count"] += 1 if descs else 0


def raw_mp_fwd_packed(desc, h_ptr, params_ptr, hout_ptr, e_ptr, ws_ptr, ws_bytes, stream, saved_ptr):
    _lib.check(_lib.load().gj_mp_step_fwd_packed(desc, h_ptr, params_ptr, hout_ptr, e_ptr, saved_ptr, ws_ptr, ws_bytes, stream),
               "gj_mp_step_fwd_packed")
    LAUNCHES["count"] += _step_launches(desc, False) - 1      # no packing launch


def raw_mp_bwd_deferred(desc, h_ptr, e_ptr, params_ptr, dhout_ptr, dh_ptr, ws_ptr, ws_bytes, stream, saved_ptr, partials_ptr):
    _lib.check(_lib.load().gj_mp_step_bwd_deferred(desc, h_ptr, e_ptr, params_ptr, dhout_ptr, dh_ptr, saved_ptr, partials_ptr, ws_ptr,
                                                   ws_bytes, stream), "gj_mp_step_bwd_deferred")
    LAUNCHES["count"] += _step_launches(desc, True, True) - 1      # no reduction launch


def raw_mp_reduce_steps(descs, partials_ptrs, dparams_ptrs, stream):
    """ONE launch reduces the parameter-gradient partials of all steps into their gradient blocks."""
    _lib.check(_lib.load().gj_mp_steps_reduce(len(descs), _desc_array(descs), _ptr_array(partials_ptrs), _ptr_array(dparams_ptrs), stream),
               "gj_mp_steps_reduce")
    LAUNCHES["count"] += 1 if descs else 0


# --------------------------------------------------------------------------------------------------
# custom ops
# --------------------------------------------------------------------------------------------------
def _desc_for(h: Tensor, num_nodes: int, node_in: int, edge_widths, node_widths, alpha, metric, precision):
    B, N, F = h.shape
    if N != num_nodes:
        raise _lib.GnnJetError(f"expected {num_nodes} nodes per jet, got {N}")
    return _lib.make_desc(B, N, node_in, edge_widths, node_widths, alpha, metric, precision,
                          h_ld=F, h_cols=min(F, node_in))


@torch.library.custom_op("gnnjet::mp_step_fwd", mutates_args=(), device_types="cuda")
@_on_device
def mp_step_fwd(h: Tensor, params: Tensor, num_nodes: int, node_in: int, edge_widths: List[int],
                node_widths: List[int], alpha: float, metric: int, precision: int) -> Tuple[Tensor, Tensor]:
    """One message-passing step (graphnet.py:154-168).  h (B,N,F) -> (h' (B,N,H'), e (B,N,E_last))."""
    h = _req(h, "h")
    params = _req(params, "params")
    d = _desc_for(h, num_nodes, node_in, edge_widths, node_widths, alpha, metric, precision)
    lib = _lib.load()
    need = lib.gj_mp_param_count(d)
    if need == 0 or params.numel() != need:
        raise _lib.GnnJetError(f"packed parameter block has {params.numel()} floats, the step needs {need}")
    B, N, _ = h.shape
    h_out = torch.empty((B, N, node_widths[-1]), device=h.device, dtype=torch.float32)
    e = torch.empty((B, N, edge_widths[-1]), device=h.device, dtype=torch.float32)
    ws_bytes = lib.gj_mp_step_fwd_workspace(d)
    ws = torch.empty((max(ws_bytes, 4) + 3) // 4, device=h.device, dtype=torch.float32)
    raw_mp_fwd(d, h.data_ptr(), params.data_ptr(), h_out.data_ptr(), e.data_ptr(), ws.data_ptr(), ws_bytes, _stream())
    return h_out, e


@mp_step_fwd.register_fake
def _(h, params, num_nodes, node_in, edge_widths, node_widths, alpha, metric, precision):
    B, N, _ = h.shape
    return h.new_empty((B, N, node_widths[-1])), h.new_empty((B, N, edge_widths[-1]))


@torch.library.custom_op("gnnjet::mp_step_bwd", mutates_args=(), device_types="cuda")
@_on_device
def mp_step_bwd(h: Tensor, e: Tensor, params: Tensor, dh_out: Tensor, num_nodes: int, node_in: int,
                edge_widths: List[int], node_widths: List[int], alpha: float, metric: int,
                precision: int) -> Tuple[Tensor, Tensor]:
    """Adjoint of one step: (dh (B,N,F), dparams packed like params)."""
    h = _req(h, "h")
    e = _req(e, "e")
    params = _req(params, "params")
    dh_out = _req(dh_out, "dh_out")
    d = _desc_for(h, num_nodes, node_in, edge_widths, node_widths, alpha, metric, precision)
    lib = _lib.load()
    B, N, F = h.shape
    # columns beyond h_cols (crop case) receive no gradient: start from zeros only then
    dh = torch.zeros_like(h) if F > node_in else torch.empty_like(h)
    dparams = torch.empty_like(params)
    ws_bytes = lib.gj_mp_step_bwd_workspace(d)
    ws = torch.empty((max(ws_bytes, 4) + 3) // 4, device=h.device, dtype=torch.float32)
    raw_mp_bwd(d, h.data_ptr(), e.data_ptr(), params.data_ptr(), dh_out.data_ptr(), dh.data_ptr(),
               dparams.data_ptr(), ws.data_ptr(), ws_bytes, _stream())
    return dh, dparams


@mp_step_bwd.register_fake
def _(h, e, params, dh_out, num_nodes, node_in, edge_widths, node_widths, alpha, metric, precision):
    return torch.empty_like(h), torch.empty_like(params)


class _MPStep(torch.autograd.Function):
    """Autograd node of one step.  ``flat`` is the packed parameter block the Linear parameters of the
    step are views of (see models/graphnet.py); the individual parameters are passed too so that
    autograd routes ``dparams`` back to them as views (no copy kernels)."""

    @staticmethod
    def forward(ctx, h, flat, cfg, *plist):
        num_nodes, node_in, ew, nw, alpha, metric, precision = cfg
        h_out, e = torch.ops.gnnjet.mp_step_fwd(h, flat, num_nodes, node_in, ew, nw, alpha, metric, precision)
        ctx.save_for_backward(h, e, flat)
        ctx.cfg = cfg
        ctx.shapes = [p.shape for p in plist]
        return h_out

    @staticmethod
    def backward(ctx, dh_out):
        h, e, flat = ctx.saved_tensors
        num_nodes, node_in, ew, nw, alpha, metric, precision = ctx.cfg
        dh, dparams = torch.ops.gnnjet.mp_step_bwd(h, e, flat, dh_out.contiguous(), num_nodes, node_in, ew, nw,
                                                    alpha, metric, precision)
        grads, off = [], 0
        for s in ctx.shapes:
            n = s.numel()
            grads.append(dparams[off:off + n].view(s))
            off += n
        return (dh, None, None, *grads)


def mp_step(h: Tensor, flat: Tensor, cfg, plist: Sequence[Tensor]) -> Tensor:
    return _MPStep.apply(h, flat, cfg, *plist)


# ---- Chamfer --------------------------------------------------------------------------------------
@torch.library.custom_op("gnnjet::chamfer", mutates_args=(), device_types="cuda")
@_on_device
def chamfer(p: Tensor, q: Tensor, norm: int, w_chamfer: float, w_jet: float) -> Tuple[Tensor, Tensor]:
    """(terms[3], dterms[2]/dp): terms = [chamfer, jet, w_chamfer*chamfer + w_jet*jet]
    (chamfer_loss.py:26-41, distance_sq.py:46-54)."""
    p = _req(p, "p")
    q = _req(q, "q")
    if p.dim() != 3 or q.dim() != 3 or p.shape[0] != q.shape[0]:
        raise ValueError(f"p and q must be (B,N,D) with equal batch sizes; got {tuple(p.shape)} and {tuple(q.shape)}")
    if p.shape[-1] not in (3, 4) or q.shape[-1] != p.shape[-1]:
        raise ValueError("p and q must both be 3- or 4-vectors (distance_sq.py:31-42)")
    B, Np, D = p.shape
    Nq = q.shape[1]
    if B == 0:
        return torch.zeros(3, device=p.device, dtype=torch.float32), torch.empty_like(p)
    terms = torch.empty(3, device=p.device, dtype=torch.float32)
    jet_terms = torch.empty((max(B, 1), 2), device=p.device, dtype=torch.float32)
    dp = torch.empty_like(p)
    lib = _lib.load()
    _lib.check(lib.gj_chamfer_fwd_bwd(B, Np, Nq, D, norm, w_chamfer, w_jet, p.data_ptr(), q.data_ptr(),
                                      jet_terms.data_ptr(), terms.data_ptr(), dp.data_ptr(), _stream()),
               "gj_chamfer_fwd_bwd")
    LAUNCHES["count"] += 2
    return terms, dp


@chamfer.register_fake
def _(p, q, norm, w_chamfer, w_jet):
    return p.new_empty(3), torch.empty_like(p)


class _Chamfer(torch.autograd.Function):
    @staticmethod
    def forward(ctx, p, q, norm, wc, wj):
        terms, dp = torch.ops.gnnjet.chamfer(p, q, norm, wc, wj)
        ctx.save_for_backward(dp)
        ctx.mark_non_differentiable(terms)
        return terms[2], terms

    @staticmethod
    def backward(ctx, g, _unused):
        (dp,) = ctx.saved_tensors
        return dp * g, None, None, None, None


def chamfer_loss(p: Tensor, q: Tensor, norm: int, w_chamfer: float, w_jet: float):
    """Returns (loss, terms); gradient flows to ``p`` (the reconstruction) only."""
    if q.requires_grad:
        raise NotImplementedError("the fused Chamfer kernel differentiates w.r.t. the reconstruction p only")
    return _Chamfer.apply(p, q.detach(), norm, float(w_chamfer), float(w_jet))


# ---- 'mean' latent map ----------------------------------------------------------------------------
@torch.library.custom_op("gnnjet::latent_mean_fwd", mutates_args=(), device_types="cuda")
@_on_device
def latent_mean_fwd(y: Tensor) -> Tensor:
    y = _req(y, "y")
    B, N, W = y.shape
    z = torch.empty((B, W), device=y.device, dtype=torch.float32)
    _lib.check(_lib.load().gj_latent_mean_fwd(B, N, W, y.data_ptr(), z.data_ptr(), _stream()), "gj_latent_mean_fwd")
    LAUNCHES["count"] += 1
    return z


@latent_mean_fwd.register_fake
def _(y):
    return y.new_empty((y.shape[0], y.shape[2]))


@torch.library.custom_op("gnnjet::latent_mean_bwd", mutates_args=(), device_types="cuda")
@_on_device
def latent_mean_bwd(dz: Tensor, num_nodes: int) -> Tensor:
    dz = _req(dz, "dz")
    B, W = dz.shape
    dy = torch.empty((B, num_nodes, W), device=dz.device, dtype=torch.float32)
    _lib.check(_lib.load().gj_latent_mean_bwd(B, num_nodes, W, dz.data_ptr(), dy.data_ptr(), _stream()),
               "gj_latent_mean_bwd")
    LAUNCHES["count"] += 1
    return dy


@latent_mean_bwd.register_fake
def _(dz, num_nodes):
    return dz.new_empty((dz.shape[0], num_nodes, dz.shape[1]))


class _LatentMean(torch.autograd.Function):
    @staticmethod
    def forward(ctx, y):
        ctx.n = y.shape[1]
        return torch.ops.gnnjet.latent_mean_fwd(y)

    @staticmethod
    def backward(ctx, dz):
        return torch.ops.gnnjet.latent_mean_bwd(dz.contiguous(), ctx.n)


def latent_mean(y: Tensor) -> Tensor:
    return _LatentMean.apply(y)


# ---- small dense layers ---------------------------------------------------------------------------
@torch.library.custom_op("gnnjet::linear_fwd", mutates_args=(), device_types="cuda")
@_on_device
def linear_fwd(x: Tensor, w: Tensor, b: Tensor | None) -> Tensor:
    x = _req(x, "x")
    w = _req(w, "w")
    if b is not None:
        b = _req(b, "b")
    rows, K = x.shape
    O = w.shape[0]
    y = torch.empty((rows, O), device=x.device, dtype=torch.float32)
    _lib.check(_lib.load().gj_linear_fwd(rows, K, O, x.data_ptr(), w.data_ptr(), _ptr(b), y.data_ptr(), _stream()),
               "gj_linear_fwd")
    LAUNCHES["count"] += 1
    return y


@linear_fwd.register_fake
def _(x, w, b):
    return x.new_empty((x.shape[0], w.shape[0]))


@torch.library.custom_op("gnnjet::linear_bwd", mutates_args=(), device_types="cuda")
@_on_device
def linear_bwd(x: Tensor, w: Tensor, dy: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    x = _req(x, "x")
    w = _req(w, "w")
    dy = _req(dy, "dy")
    rows, K = x.shape
    O = w.shape[0]
    lib = _lib.load()
    dx = torch.empty_like(x)
    dw = torch.empty_like(w)
    db = torch.empty(O, device=x.device, dtype=torch.float32)
    ws_bytes = lib.gj_linear_bwd_workspace(rows, K, O)
    ws = torch.empty((ws_bytes + 3) // 4, device=x.device, dtype=torch.float32)
    _lib.check(lib.gj_linear_bwd(rows, K, O, x.data_ptr(), w.data_ptr(), dy.data_ptr(), dx.data_ptr(), dw.data_ptr(),
                                 db.data_ptr(), ws.data_ptr(), ws_bytes, _stream()), "gj_linear_bwd")
    LAUNCHES["count"] += 3
    return dx, dw, db


@linear_bwd.register_fake
def _(x, w, dy):
    return torch.empty_like(x), torch.empty_like(w), x.new_empty(w.shape[0])


class _Linear(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w, b):
        ctx.save_for_backward(x, w)
        ctx.has_bias = b is not None
        return torch.ops.gnnjet.linear_fwd(x, w, b)

    @staticmethod
    def backward(ctx, dy):
        x, w = ctx.saved_tensors
        dx, dw, db = torch.ops.gnnjet.linear_bwd(x, w, dy.contiguous())
        return dx, dw, (db if ctx.has_bias else None)


def linear(x: Tensor, w: Tensor, b: Tensor | None) -> Tensor:
    """y = x W^T + b over the last axis (decoder.py:127-136, encoder.py:156-161)."""
    lead = x.shape[:-1]
    y = _Linear.apply(x.reshape(-1, x.shape[-1]), w, b)
    return y.view(*lead, w.shape[0])


# ---- optimiser ------------------------------------------------------------------------------------
@_on_device
def adam_step_flat_(param: Tensor, grad: Tensor, exp_avg: Tensor, exp_avg_sq: Tensor, step: int, lr: float = 1e-5,
                    betas=(0.9, 0.999), eps: float = 1e-8, grad_scale: float = 1.0, l1_lambda: float = 0.0,
                    l2_lambda: float = 0.0) -> None:
    """In-place fused Adam over flat fp32 buffers (torch.optim.Adam defaults, initialize.py:152-153) with the
    regulariser gradients of train.py:376-384 folded in."""
    for t, n in ((param, "param"), (grad, "grad"), (exp_avg, "exp_avg"), (exp_avg_sq, "exp_avg_sq")):
        if not t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous():
            raise _lib.GnnJetError(f"{n} must be a contiguous float32 CUDA tensor")
    _lib.check(_lib.load().gj_adam_step_flat(param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(),
                                             param.numel(), lr, betas[0], betas[1], eps, int(step), grad_scale,
                                             l1_lambda, l2_lambda, _stream()), "gj_adam_step_flat")
    LAUNCHES["count"] += 1


def set_deterministic(on: bool) -> bool:
    """Bitwise-reproducible parameter gradients in the bf16 mode (one tile group per CTA in the backward edge kernels, about
    2.5x their time); returns the previous setting.  Call it before building a GNNAETrainer CUDA graph."""
    return bool(_lib.load().gj_set_deterministic(1 if on else 0))


OPTIMIZERS = {"rmsprop": 1, "adagrad": 2, "sgd": 3}


def _optimizer_hparams(kind: str):
    """(kind id, (alpha, momentum, eps)) of the hyper-parameters utils/initialize.py:154-170 passes."""
    k = OPTIMIZERS[kind.lower()]
    return k, ((0.99, 0.9, 1e-16) if k == 1 else ((0.0, 0.0, 1e-16) if k == 2 else (0.0, 0.9, 0.0)))


@_on_device
def optimizer_step_flat_(kind: str, param: Tensor, grad: Tensor, momentum_buf: Tensor, sq_acc: Tensor, lr: float = 1e-5,
                         grad_scale: float = 1.0, l1_lambda: float = 0.0, l2_lambda: float = 0.0) -> None:
    """In-place fused RMSprop / Adagrad / SGD over flat fp32 buffers with the hyper-parameters utils/initialize.py:154-170 passes
    (RMSprop: eps 1e-16, momentum 0.9, torch's alpha 0.99; Adagrad: eps 1e-16; SGD: momentum 0.9)."""
    for t, n in ((param, "param"), (grad, "grad"), (momentum_buf, "momentum_buf"), (sq_acc, "sq_acc")):
        if not t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous():
            raise _lib.GnnJetError(f"{n} must be a contiguous float32 CUDA tensor")
    k, (alpha, momentum, eps) = _optimizer_hparams(kind)
    _lib.check(_lib.load().gj_optimizer_step_flat(k, param.data_ptr(), grad.data_ptr(), momentum_buf.data_ptr(), sq_acc.data_ptr(),
                                                  param.numel(), lr, alpha, momentum, eps, grad_scale, l1_lambda, l2_lambda, _stream()),
               "gj_optimizer_step_flat")
    LAUNCHES["count"] += 1


# ---- non-finite step guard (include/gnnjet_b200.h: gj_nonfinite_flag / gj_nonfinite_check / gj_*_step_flat_guarded) ----------
def _req_i32(t: Tensor, name: str, n: int) -> None:
    if not t.is_cuda or t.dtype != torch.int32 or not t.is_contiguous() or t.numel() < n:
        raise _lib.GnnJetError(f"{name} must be a contiguous int32 CUDA tensor of at least {n} elements")


def _req_f32(t: Tensor, name: str) -> None:
    if not t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous():
        raise _lib.GnnJetError(f"{name} must be a contiguous float32 CUDA tensor")


@_on_device
def nonfinite_flag_(terms: Tensor, out: Tensor) -> None:
    """out[0] = 0 if every element of ``terms`` (at most 64) is finite, else NaN: one launch, no host synchronisation."""
    _req_f32(terms, "terms")
    _req_f32(out, "out")
    _lib.check(_lib.load().gj_nonfinite_flag(terms.data_ptr(), terms.numel(), out.data_ptr(), _stream()), "gj_nonfinite_flag")
    LAUNCHES["count"] += 1


@_on_device
def nonfinite_check_(x: Tensor, skip: Tensor, flag: Tensor | None = None) -> None:
    """skip[0] = 1 if any element of ``x`` is not finite, else 0 (int32); ``flag[0]`` the same as 1.0 / 0.0: one launch, one CTA, no
    host synchronisation."""
    _req_f32(x, "x")
    _req_i32(skip, "skip", 1)
    if flag is not None:
        _req_f32(flag, "flag")
    _lib.check(_lib.load().gj_nonfinite_check(x.data_ptr(), x.numel(), skip.data_ptr(), _ptr(flag), _stream()), "gj_nonfinite_check")
    LAUNCHES["count"] += 1


@_on_device
def adam_step_flat_guarded_(param: Tensor, grad: Tensor, exp_avg: Tensor, exp_avg_sq: Tensor, skip: Tensor, step_state: Tensor,
                            lr: float = 1e-5, betas=(0.9, 0.999), eps: float = 1e-8, grad_scale: float = 1.0, l1_lambda: float = 0.0,
                            l2_lambda: float = 0.0) -> None:
    """``adam_step_flat_`` behind the device flag ``skip[0]`` (int32): nothing is written when it is set.  The step number is
    ``step_state[0] + 1`` (int32, two elements, zero-initialised; ``step_state[0]`` counts the updates applied and the launch advances
    it when it applies its update, ``step_state[1]`` is the kernel's arrival counter and stays 0)."""
    for t, n in ((param, "param"), (grad, "grad"), (exp_avg, "exp_avg"), (exp_avg_sq, "exp_avg_sq")):
        _req_f32(t, n)
    _req_i32(skip, "skip", 1)
    _req_i32(step_state, "step_state", 2)
    _lib.check(_lib.load().gj_adam_step_flat_guarded(param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(),
                                                     param.numel(), lr, betas[0], betas[1], eps, skip.data_ptr(), step_state.data_ptr(),
                                                     grad_scale, l1_lambda, l2_lambda, _stream()), "gj_adam_step_flat_guarded")
    LAUNCHES["count"] += 1


@_on_device
def optimizer_step_flat_guarded_(kind: str, param: Tensor, grad: Tensor, momentum_buf: Tensor, sq_acc: Tensor, skip: Tensor,
                                 step_state: Tensor | None = None, lr: float = 1e-5, grad_scale: float = 1.0, l1_lambda: float = 0.0,
                                 l2_lambda: float = 0.0) -> None:
    """``optimizer_step_flat_`` behind the device flag ``skip[0]``; ``step_state`` (optional, as for ``adam_step_flat_guarded_``)
    counts the updates applied."""
    for t, n in ((param, "param"), (grad, "grad"), (momentum_buf, "momentum_buf"), (sq_acc, "sq_acc")):
        _req_f32(t, n)
    _req_i32(skip, "skip", 1)
    if step_state is not None:
        _req_i32(step_state, "step_state", 2)
    k, (alpha, momentum, eps) = _optimizer_hparams(kind)
    _lib.check(_lib.load().gj_optimizer_step_flat_guarded(k, param.data_ptr(), grad.data_ptr(), momentum_buf.data_ptr(), sq_acc.data_ptr(),
                                                          param.numel(), lr, alpha, momentum, eps, grad_scale, l1_lambda, l2_lambda,
                                                          skip.data_ptr(), _ptr(step_state), _stream()), "gj_optimizer_step_flat_guarded")
    LAUNCHES["count"] += 1


@_on_device
def param_norms(param: Tensor) -> Tensor:
    """[sum |p|, sum p^2] of a flat buffer (encoder.py:173-179)."""
    param = _req(param, "param")
    lib = _lib.load()
    out = torch.empty(2, device=param.device, dtype=torch.float32)
    ws_bytes = lib.gj_param_norms_workspace(param.numel())
    ws = torch.empty((ws_bytes + 3) // 4, device=param.device, dtype=torch.float32)
    _lib.check(lib.gj_param_norms(param.data_ptr(), param.numel(), out.data_ptr(), ws.data_ptr(), ws_bytes, _stream()),
               "gj_param_norms")
    LAUNCHES["count"] += 2
    return out


@_on_device
def umma_selftest(a: Tensor, b: Tensor, a_mn_major: bool, b_mn_major: bool) -> Tensor:
    """D = A(m,k) B(n,k)^T on one CTA through tcgen05 (bf16 operands, fp32 TMEM accumulator)."""
    a = _req(a, "a")
    b = _req(b, "b")
    m, k = a.shape
    n = b.shape[0]
    out = torch.zeros((128, n), device=a.device, dtype=torch.float32)
    _lib.check(_lib.load().gj_umma_selftest(m, n, k, int(a_mn_major), int(b_mn_major), a.data_ptr(), b.data_ptr(),
                                            out.data_ptr(), _stream()), "gj_umma_selftest")
    return out
