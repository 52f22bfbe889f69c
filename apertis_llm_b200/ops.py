"""torch.autograd bindings of the C-ABI kernels (device memory, streams and autograd plumbing only;
all arithmetic on the hot path runs in libapertis_b200.so).

  causal_conv1d_silu   core.py:368-375
  selective_scan       core.py:324-353, 383, 394-396
  moe_experts          core.py:480-607 (router, plan, permute, expert MLPs, combine, aux losses)
"""
from __future__ import annotations

import ctypes
import math
import os
from typing import Optional

import torch

from . import _lib
from ._lib import AB_BF16, AB_F32, ROW_ALIGN, call, dt, ptr, query, stream_ptr

def _on_tensor_device(fn):
    """Runs an autograd Function's forward / backward with the device of its first CUDA tensor argument current: the C ABI
    launches on the current device and stream, so a module living on cuda:1 while cuda:0 is current must switch first."""
    def wrapper(ctx, *args):
        dev = next((a.device for a in args if torch.is_tensor(a) and a.is_cuda), None)
        if dev is None:
            return fn(ctx, *args)
        with torch.cuda.device(dev):
            return fn(ctx, *args)
    wrapper.__name__, wrapper.__doc__ = fn.__name__, fn.__doc__
    return wrapper


# --------------------------------------------------------------------------------------------
# workspaces
# --------------------------------------------------------------------------------------------
_scan_ws = {}       # (device index, stream, pipelined?) -> [tensor, epoch]
# APERTIS_B200_SCAN = auto (default) | rounds | pipelined | single | two_pass.  auto = the "rounds" schedule
# (csrc/ssm_scan_rounds.cu, every shape); the other values select the older schedules of csrc/ssm_scan*.cu.
_SCAN_ENV = os.environ.get("APERTIS_B200_SCAN", "auto")
SCAN_MODE = {"two_pass": _lib.SCAN_TWO_PASS, "single": _lib.SCAN_SINGLE_PASS, "pipelined": _lib.SCAN_PIPELINED,
             "rounds": _lib.SCAN_ROUNDS}.get(_SCAN_ENV)


def default_scan_mode(dtype: torch.dtype, Di: int, L: int = 1 << 20) -> int:
    """The "rounds" schedule (csrc/ssm_scan_rounds.cu) serves every shape; the older schedules stay selectable."""
    if SCAN_MODE is not None:
        return SCAN_MODE
    return _lib.SCAN_ROUNDS


def _scan_workspace(device, nbytes: int, mode: int = _lib.SCAN_SINGLE_PASS):
    """Persistent, zero-initialised hand-shake workspace per (device, stream) with its launch epoch.  The pipelined
    schedule keeps its epoch inside the workspace (valid under CUDA-graph replay) and gets a workspace of its own."""
    key = (device.index, torch.cuda.current_stream(device).cuda_stream, mode == _lib.SCAN_PIPELINED)
    ent = _scan_ws.get(key)
    if ent is None or ent[0].numel() < nbytes:
        epoch = ent[1] if ent is not None else 0
        ent = [torch.zeros(max(nbytes, 1 << 20), dtype=torch.uint8, device=device), epoch]
        _scan_ws[key] = ent
    ent[1] += 1
    if ent[1] >= (1 << 30) - 1:          # epoch wrap: start over on a clean buffer
        ent[0].zero_()
        ent[1] = 1
    return ent[0], ent[1]


_SCAN_CHECK = os.environ.get("APERTIS_B200_SCAN_CHECK", "0") == "1"


def _scan_check(ws: torch.Tensor, what: str):
    """Debug aid (APERTIS_B200_SCAN_CHECK=1, synchronises): the hand-shake waits of the scan kernels are bounded and raise a
    flag in the workspace instead of hanging; turn a raised flag into an exception."""
    if _SCAN_CHECK and not torch.cuda.is_current_stream_capturing() and int(ws[64:68].view(torch.int32).item()) != 0:
        ws[64:68].zero_()
        raise RuntimeError(f"{what}: a hand-shake wait of the selective scan timed out (protocol error)")


def scan_plan(B: int, L: int, Di: int, dtype: torch.dtype, mode: int = _lib.SCAN_SINGLE_PASS):
    """-> (tile rows, slab channels, saved states per sequence, workspace bytes, effective mode): a pipelined request
    the schedule does not cover comes back as single-pass."""
    t, s, n, m = ctypes.c_int(), ctypes.c_int(), ctypes.c_int(), ctypes.c_int(mode)
    ws = ctypes.c_size_t()
    call("ab_selective_scan_plan", B, L, Di, dt(dtype), ctypes.byref(m), ctypes.byref(t), ctypes.byref(s), ctypes.byref(n), ctypes.byref(ws))
    return t.value, s.value, n.value, ws.value, m.value


def _row_stride(t: torch.Tensor) -> int:
    """Row stride (elements) of a [B, L, C] tensor whose rows may be slices of a wider contiguous buffer."""
    B, L, C = t.shape
    assert t.stride(2) == 1 and (B == 1 or t.stride(0) == L * t.stride(1)), "unsupported layout"
    return t.stride(1)


def _rows(t: torch.Tensor) -> torch.Tensor:
    """Ensures a [B,L,C] tensor is usable as strided rows (last dim contiguous, batches back to back)."""
    B, L, C = t.shape
    if t.stride(2) == 1 and (B == 1 or t.stride(0) == L * t.stride(1)) and (L == 1 or t.stride(1) >= C):
        return t
    return t.contiguous()


# --------------------------------------------------------------------------------------------
# block-wrapper LayerNorm (pre_norm of ApertisAttention / ApertisFeedForward)
# --------------------------------------------------------------------------------------------
class _LayerNorm(torch.autograd.Function):
    @staticmethod
    @_on_tensor_device
    def forward(ctx, x, weight, bias, eps, out_dtype):
        _lib.ensure_device(x.device)
        shape = x.shape
        Dm = shape[-1]
        x2 = x.reshape(-1, Dm).contiguous()
        S = x2.shape[0]
        w, b = weight.float().contiguous(), bias.float().contiguous()
        y = torch.empty(S, Dm, dtype=out_dtype, device=x.device)
        stats = torch.empty(S, 2, dtype=torch.float32, device=x.device)
        call("ab_layernorm_fwd", ptr(x2), ptr(w), ptr(b), float(eps), ptr(y), ptr(stats), S, Dm, dt(x2), dt(out_dtype), stream_ptr())
        ctx.save_for_backward(x2, stats, w)
        ctx.shape = shape
        return y.view(shape)

    @staticmethod
    @_on_tensor_device
    def backward(ctx, dy):
        x2, stats, w = ctx.saved_tensors
        S, Dm = x2.shape
        dy2 = dy.reshape(S, Dm).contiguous()
        dx = torch.empty_like(x2)
        dw = torch.empty(Dm, dtype=torch.float32, device=x2.device)
        db = torch.empty(Dm, dtype=torch.float32, device=x2.device)
        nws = query("ab_layernorm_bwd_workspace_bytes", S, Dm)
        ws = torch.empty(max(nws, 16), dtype=torch.uint8, device=x2.device)
        call("ab_layernorm_bwd", ptr(dy2), ptr(x2), ptr(stats), ptr(w), None, ptr(dx), ptr(dw), ptr(db), ptr(ws), ws.numel(), S, Dm,
             dt(x2), dt(dy2), stream_ptr())
        return dx.view(ctx.shape), dw, db, None, None


class _LayerNormSkip(torch.autograd.Function):
    """LayerNorm that also hands its input on as the residual: x then has ONE consumer in the autograd graph, and the
    backward adds the residual path's gradient inside the LayerNorm-backward kernel (`dres` of ab_layernorm_bwd) instead of
    leaving the sum of the two branches to a separate elementwise pass over [tokens, Dm]."""

    @staticmethod
    @_on_tensor_device
    def forward(ctx, x, weight, bias, eps, out_dtype):
        _lib.ensure_device(x.device)
        shape = x.shape
        Dm = shape[-1]
        x2 = x.reshape(-1, Dm).contiguous()
        S = x2.shape[0]
        w, b = weight.float().contiguous(), bias.float().contiguous()
        y = torch.empty(S, Dm, dtype=out_dtype, device=x.device)
        stats = torch.empty(S, 2, dtype=torch.float32, device=x.device)
        call("ab_layernorm_fwd", ptr(x2), ptr(w), ptr(b), float(eps), ptr(y), ptr(stats), S, Dm, dt(x2), dt(out_dtype), stream_ptr())
        ctx.save_for_backward(x2, stats, w)
        ctx.shape = shape
        return y.view(shape), x.view_as(x)

    @staticmethod
    @_on_tensor_device
    def backward(ctx, dy, dskip):
        x2, stats, w = ctx.saved_tensors
        S, Dm = x2.shape
        if dy is None:
            return dskip, None, None, None, None
        dy2 = dy.reshape(S, Dm).contiguous()
        dres = dskip.reshape(S, Dm).to(x2.dtype).contiguous() if dskip is not None else None
        dx = torch.empty_like(x2)
        dw = torch.empty(Dm, dtype=torch.float32, device=x2.device)
        db = torch.empty(Dm, dtype=torch.float32, device=x2.device)
        nws = query("ab_layernorm_bwd_workspace_bytes", S, Dm)
        ws = torch.empty(max(nws, 16), dtype=torch.uint8, device=x2.device)
        call("ab_layernorm_bwd", ptr(dy2), ptr(x2), ptr(stats), ptr(w), ptr(dres), ptr(dx), ptr(dw), ptr(db), ptr(ws), ws.numel(), S, Dm,
             dt(x2), dt(dy2), stream_ptr())
        return dx.view(ctx.shape), dw, db, None, None


class _DropoutAdd(torch.autograd.Function):
    @staticmethod
    @_on_tensor_device
    def forward(ctx, sub, res, p):
        _lib.ensure_device(sub.device)
        sub = sub.contiguous()
        res = res.contiguous()
        out = torch.empty_like(res)
        seed = torch.randint(0, 2 ** 31 - 1, (2,), device=sub.device, dtype=torch.int32) if p > 0 else None
        call("ab_dropout_add", ptr(sub), ptr(res), ptr(out), float(p), ptr(seed), sub.numel(), dt(sub), dt(out), stream_ptr())
        ctx.p, ctx.seed, ctx.sub_dtype = p, seed, sub.dtype
        return out

    @staticmethod
    @_on_tensor_device
    def backward(ctx, dout):
        if ctx.p == 0:
            return dout.to(ctx.sub_dtype), dout, None
        dout = dout.contiguous()
        dsub = torch.empty(dout.shape, dtype=ctx.sub_dtype, device=dout.device)
        call("ab_dropout_add", ptr(dout), None, ptr(dsub), float(ctx.p), ptr(ctx.seed), dout.numel(), dt(dout), dt(dsub), stream_ptr())
        return dsub, dout, None


def dropout_add(sub, res, p: float, training: bool):
    """nn.Dropout(p)(sub) + res of the block wrappers (core.py:836-837, 918-919) as one kernel."""
    return _DropoutAdd.apply(sub, res, float(p) if training else 0.0)


def layer_norm(x, weight, bias, eps, out_dtype=None):
    """nn.LayerNorm over the last dim (core.py:694-695, 887-888) through the sm_100a kernel."""
    return _LayerNorm.apply(x, weight, bias, eps, out_dtype if out_dtype is not None else x.dtype)


def layer_norm_skip(x, weight, bias, eps, out_dtype=None):
    """(LayerNorm(x), x) for the pre-norm residual wrappers: use the second result as the residual operand, so that the
    two gradients meeting at x are added inside the LayerNorm-backward kernel."""
    return _LayerNormSkip.apply(x, weight, bias, eps, out_dtype if out_dtype is not None else x.dtype)


# --------------------------------------------------------------------------------------------
# causal conv1d + SiLU
# --------------------------------------------------------------------------------------------
class _CausalConv1dSiLU(torch.autograd.Function):
    @staticmethod
    @_on_tensor_device
    def forward(ctx, xp, weight, bias):
        _lib.ensure_device(xp.device)
        xp = _rows(xp)
        B, L, Di = xp.shape
        Kc = weight.shape[-1]
        w = weight.reshape(Di, Kc).float().contiguous()
        b = bias.float().contiguous()
        xa = torch.empty(B, L, Di, dtype=xp.dtype, device=xp.device)
        call("ab_causal_conv1d_silu_fwd", ptr(xp), _row_stride(xp), ptr(w), ptr(b), ptr(xa), B, L, Di, Kc, dt(xp), stream_ptr())
        ctx.save_for_backward(xp, w, b)
        ctx.wshape = weight.shape
        ctx.wdtype, ctx.bdtype = weight.dtype, bias.dtype
        return xa

    @staticmethod
    @_on_tensor_device
    def backward(ctx, dxa):
        xp, w, b = ctx.saved_tensors
        B, L, Di = xp.shape
        Kc = w.shape[-1]
        dxa = dxa.contiguous()
        dxp = torch.empty(B, L, Di, dtype=xp.dtype, device=xp.device)
        dw = torch.empty(Di, Kc, dtype=torch.float32, device=xp.device)
        db = torch.empty(Di, dtype=torch.float32, device=xp.device)
        nws = query("ab_causal_conv1d_silu_bwd_workspace_bytes", B, L, Di)
        ws = torch.empty(nws, dtype=torch.uint8, device=xp.device)
        call("ab_causal_conv1d_silu_bwd", ptr(xp), _row_stride(xp), ptr(dxa), ptr(w), ptr(b), ptr(dxp), Di, ptr(dw), ptr(db),
             ptr(ws), nws, B, L, Di, Kc, dt(xp), stream_ptr())
        return dxp, dw.reshape(ctx.wshape).to(ctx.wdtype), db.to(ctx.bdtype)


def causal_conv1d_silu(xp: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """xp [B,L,Di] (channels last), weight [Di,1,Kc] (2 <= Kc <= 8), bias [Di] -> silu(causal depthwise conv) [B,L,Di]."""
    return _CausalConv1dSiLU.apply(xp, weight, bias)


# --------------------------------------------------------------------------------------------
# selective scan
# --------------------------------------------------------------------------------------------
class _SelectiveScan(torch.autograd.Function):
    @staticmethod
    @_on_tensor_device
    def forward(ctx, xa, dlog, BC, z, A_log, D, h0, want_yssm, want_hlast, mode):
        _lib.ensure_device(xa.device)
        xa = xa.contiguous()
        dlog = dlog.contiguous()
        BC, z = BC.contiguous(), _rows(z)
        B, L, Di = xa.shape
        H = dlog.shape[-1]
        assert BC.shape == (B, L, 2 * Di)
        Bm, Cm = BC[..., :Di], BC[..., Di:]
        dev = xa.device
        A = A_log.reshape(-1).float().contiguous()
        Dv = D.float().contiguous()
        if want_yssm and mode == _lib.SCAN_PIPELINED:
            mode = _lib.SCAN_SINGLE_PASS                     # y_ssm (output_attentions) is not emitted by the pipelined kernels
        T, Cs, nchunks, nws, mode = scan_plan(B, L, Di, xa.dtype, mode)
        if mode != _lib.SCAN_PIPELINED and torch.cuda.is_current_stream_capturing():
            # the non-pipelined single pass validates its words with a launch epoch passed by value, which a replayed
            # CUDA graph would freeze: captured steps use the two-pass schedule (no inter-CTA waits, nothing to validate)
            mode = _lib.SCAN_TWO_PASS
        ws, epoch = _scan_workspace(dev, nws, mode)
        y = torch.empty_like(xa)
        y_ssm = torch.empty_like(xa) if want_yssm else None
        h_last = torch.empty(B, Di, dtype=torch.float32, device=dev) if want_hlast else None
        hstart = torch.empty(B, nchunks, Di, dtype=torch.float32, device=dev)
        h0c = h0.reshape(B, Di).float().contiguous() if h0 is not None else None
        call("ab_selective_scan_fwd", ptr(xa), ptr(dlog), ptr(Bm), ptr(Cm), 2 * Di, ptr(z), _row_stride(z), ptr(A),
             ptr(Dv), ptr(h0c), ptr(y), ptr(y_ssm), ptr(h_last), ptr(hstart), ptr(ws), ws.numel(), epoch, mode,
             B, L, Di, H, dt(xa), stream_ptr())
        _scan_check(ws, "ab_selective_scan_fwd")
        ctx.save_for_backward(xa, dlog, BC, z, A, Dv, hstart)
        ctx.mode = mode
        ctx.a_shape, ctx.want_yssm = A_log.shape, want_yssm
        if h_last is not None:
            ctx.mark_non_differentiable(h_last)
        return y, y_ssm, h_last

    @staticmethod
    @_on_tensor_device
    def backward(ctx, dy, dyssm, _dh):
        xa, dlog, BC, z, A, Dv, hstart = ctx.saved_tensors
        B, L, Di = xa.shape
        H = dlog.shape[-1]
        dev = xa.device
        Bm, Cm = BC[..., :Di], BC[..., Di:]
        dy = dy.contiguous()
        dys = dyssm.contiguous() if (dyssm is not None and ctx.want_yssm) else None
        T, Cs, nchunks, nws, _ = scan_plan(B, L, Di, xa.dtype, ctx.mode)
        ws, epoch = _scan_workspace(dev, nws, ctx.mode)
        dxa = torch.empty_like(xa)
        dz = torch.empty_like(xa)
        dbc = torch.empty(B, L, 2 * Di, dtype=xa.dtype, device=dev)       # [dB | dC] rows, ready for the x_param_proj GEMM
        parts = H if ctx.mode == _lib.SCAN_PIPELINED else Di // 4     # pipelined: d dlog comes back final
        ddl = torch.empty(B, L, parts, dtype=torch.float32, device=dev)
        dA = torch.empty(Di, dtype=torch.float32, device=dev)
        dD = torch.empty(Di, dtype=torch.float32, device=dev)
        dB, dC = dbc[..., :Di], dbc[..., Di:]
        call("ab_selective_scan_bwd", ptr(xa), ptr(dlog), ptr(Bm), ptr(Cm), 2 * Di, ptr(z), _row_stride(z), ptr(dy),
             ptr(dys), ptr(A), ptr(Dv), ptr(hstart), ptr(dxa), ptr(dB), ptr(dC), 2 * Di, ptr(dz), ptr(ddl), ptr(dA), ptr(dD),
             ptr(ws), ws.numel(), epoch, ctx.mode, B, L, Di, H, dt(xa), stream_ptr())
        _scan_check(ws, "ab_selective_scan_bwd")
        ddlog = (ddl if parts == H else ddl.view(B, L, H, parts // H).sum(-1)).to(dlog.dtype)
        return dxa, ddlog, dbc, dz, dA.reshape(ctx.a_shape), dD, None, None, None, None


def selective_scan(xa, dlog, BC, z, A_log, D, h0=None, want_yssm=False, want_hlast=False, mode: Optional[int] = None):
    """Fused softplus(dt) / discretise / scan / D skip / SiLU(z) gate.

    xa, z [B,L,Di]; BC [B,L,2*Di] = [B-term | C-term]; dlog [B,L,H]; A_log [H,16]; D [Di]; h0 [B,H,16] or None.
    Returns (y [B,L,Di], y_ssm | None, h_last [B,Di] fp32 | None)."""
    mode = default_scan_mode(xa.dtype, xa.shape[-1], xa.shape[1]) if mode is None else mode
    if mode == _lib.SCAN_ROUNDS:
        return _SelectiveScanRounds.apply(xa, dlog, None, BC, z, A_log, D, h0, want_yssm, want_hlast, dlog.shape[-1])
    return _SelectiveScan.apply(xa, dlog, BC, z, A_log, D, h0, want_yssm, want_hlast, mode)


# --------------------------------------------------------------------------------------------
# selective scan, "rounds" schedule (the default)
# --------------------------------------------------------------------------------------------
_rounds_ws = {}      # (device index, stream) -> workspace tensor


def _rounds_plan(B, L, Di, dtype):
    n, ws = ctypes.c_int64(), ctypes.c_size_t()
    call("ab_ssm_scan_plan", B, L, Di, dt(dtype), ctypes.byref(n), ctypes.byref(ws))
    return n.value, ws.value


def _rounds_workspace(device, nbytes):
    """One workspace per (device, stream): launches on a stream are ordered, and each launch leaves the counters zeroed."""
    key = (device.index, torch.cuda.current_stream(device).cuda_stream)
    t = _rounds_ws.get(key)
    if t is None or t.numel() < nbytes:
        t = torch.zeros(max(nbytes, 2 << 20), dtype=torch.uint8, device=device)      # zero-filled once (ABI contract)
        _rounds_ws[key] = t
    return t


def _cols(t, lo, hi):
    return t[..., lo:hi]


class _SelectiveScanRounds(torch.autograd.Function):
    """xa [B,L,Di] and z [B,L,Di] may be column slices of wider buffers (row stride arbitrary).
    fused layout (dlog is None): prm [B,L,Hp+2Di] = [dt (H, zero padded to Hp) | B | C], dt WITHOUT its bias (dt_bias given);
    split layout: dlog [B,L,H] contiguous (bias already in, or given separately), prm = [B | C] [B,L,2Di]."""

    @staticmethod
    def forward(ctx, xa, dlog, dt_bias, prm, z, A_log, D, h0, want_yssm, want_hlast, H):
        _lib.ensure_device(xa.device)
        with torch.cuda.device(xa.device):
            xa, z, prm = _rows(xa), _rows(z), _rows(prm)
            B, L, Di = xa.shape
            dev = xa.device
            fused = dlog is None
            W = prm.shape[-1]
            Hp = W - 2 * Di
            assert Hp >= (H if fused else 0) and (fused or Hp == 0), "bad [dt | B | C] layout"
            dl = prm if fused else dlog.contiguous()
            dl_stride = _row_stride(prm) if fused else H
            Bm, Cm = _cols(prm, Hp, Hp + Di), _cols(prm, Hp + Di, Hp + 2 * Di)
            A = A_log.reshape(-1).float().contiguous()
            Dv = D.float().contiguous()
            bias = dt_bias.float().contiguous() if dt_bias is not None else None
            nstate, nws = _rounds_plan(B, L, Di, xa.dtype)
            ws = _rounds_workspace(dev, nws)
            y = torch.empty(B, L, Di, dtype=xa.dtype, device=dev)
            y_ssm = torch.empty(B, L, Di, dtype=xa.dtype, device=dev) if want_yssm else None
            h_last = torch.empty(B, Di, dtype=torch.float32, device=dev) if want_hlast else None
            state = torch.empty(nstate, dtype=torch.float32, device=dev)
            h0c = h0.reshape(B, Di).float().contiguous() if h0 is not None else None
            call("ab_ssm_scan_fwd", ptr(xa), _row_stride(xa), ptr(dl), dl_stride, ptr(bias), ptr(Bm), ptr(Cm), _row_stride(prm),
                 ptr(z), _row_stride(z), ptr(A), ptr(Dv), ptr(h0c), ptr(y), ptr(y_ssm), ptr(h_last), ptr(state), ptr(ws), ws.numel(),
                 B, L, Di, H, dt(xa), stream_ptr(dev))
            ctx.save_for_backward(xa, prm, z, A, Dv, state)
            ctx.meta = (fused, H, Hp, want_yssm, A_log.shape, dlog.dtype if dlog is not None else None,
                        dt_bias is not None, dt_bias.dtype if dt_bias is not None else None)
            if h_last is not None:
                ctx.mark_non_differentiable(h_last)
            return y, y_ssm, h_last

    @staticmethod
    def backward(ctx, dy, dyssm, _dh):
        xa, prm, z, A, Dv, state = ctx.saved_tensors
        fused, H, Hp, want_yssm, a_shape, dlog_dtype, has_bias, bias_dtype = ctx.meta
        with torch.cuda.device(xa.device):
            B, L, Di = xa.shape
            dev = xa.device
            W = prm.shape[-1]
            Bm, Cm = _cols(prm, Hp, Hp + Di), _cols(prm, Hp + Di, Hp + 2 * Di)
            dy = dy.contiguous()
            dys = dyssm.contiguous() if (dyssm is not None and want_yssm) else None
            nstate, nws = _rounds_plan(B, L, Di, xa.dtype)
            ws = _rounds_workspace(dev, nws)
            dxa = torch.empty(B, L, Di, dtype=xa.dtype, device=dev)
            dz = torch.empty(B, L, Di, dtype=xa.dtype, device=dev)
            dprm = torch.empty(B, L, W, dtype=xa.dtype, device=dev)
            ddl = dprm if fused else torch.empty(B, L, H, dtype=xa.dtype, device=dev)
            dA = torch.empty(Di, dtype=torch.float32, device=dev)
            dD = torch.empty(Di, dtype=torch.float32, device=dev)
            dbias = torch.empty(H, dtype=torch.float32, device=dev) if has_bias else None
            dB, dC = _cols(dprm, Hp, Hp + Di), _cols(dprm, Hp + Di, Hp + 2 * Di)
            call("ab_ssm_scan_bwd", ptr(xa), _row_stride(xa), ptr(Bm), ptr(Cm), _row_stride(prm), ptr(z), _row_stride(z), ptr(dy),
                 ptr(dys), ptr(A), ptr(Dv), ptr(state), ptr(dxa), Di, ptr(dB), ptr(dC), W, ptr(dz), Di, ptr(ddl),
                 W if fused else H, Hp if fused else H, ptr(dbias), ptr(dA), ptr(dD), ptr(ws), ws.numel(), B, L, Di, H, dt(xa),
                 stream_ptr(dev))
            ddlog = None if fused else ddl.to(dlog_dtype)
            return (dxa, ddlog, dbias.to(bias_dtype) if has_bias else None, dprm, dz, dA.reshape(a_shape), dD,
                    None, None, None, None)


def selective_scan_fused(xa, prm, dt_bias, z, A_log, D, H, h0=None, want_yssm=False, want_hlast=False):
    """Scan over the fused projection output prm [B,L,Hp+2Di] = [dt (no bias) | B | C] (see _SelectiveScanRounds)."""
    return _SelectiveScanRounds.apply(xa, None, dt_bias, prm, z, A_log, D, h0, want_yssm, want_hlast, H)



# --------------------------------------------------------------------------------------------
# dense projections of the SSM layer on the tcgen05 GEMM kernel (core.py:366-367, 376-383, 397)
# --------------------------------------------------------------------------------------------
def _as_bf16(t):
    """bf16 GEMM operand of a contiguous tensor (fp32 masters are cast by the library's own kernel)."""
    if t.dtype == torch.bfloat16:
        return t.contiguous()
    if t.dtype == torch.float32 and t.is_contiguous() and t.numel() % 4 == 0:
        return _cast_bf16(t)
    return t.to(torch.bfloat16).contiguous()


def dense_nt(x2, w, precise, bias=None, out_dtype=None):
    """x2 [S,K] @ w[N,K]^T (+ bias) -> [S,N].  precise: fp32 in / out through the 3-product bf16 split."""
    S, K = x2.shape
    N = w.shape[0]
    dev = x2.device
    if precise:
        a, b, kk, od = _split_cols(x2.float().contiguous(), 0), _split_cols(w.float().contiguous(), 1), 3 * K, torch.float32
    else:
        a, b, kk, od = _as_bf16(x2), _as_bf16(w), K, (out_dtype or torch.bfloat16)
    c = torch.empty(S, N, dtype=od, device=dev)
    call("ab_dense_gemm_nt", ptr(a), ptr(b), ptr(bias), None, ptr(c), S, N, kk, _lib.EPI_BIAS if bias is not None else _lib.EPI_NONE,
         dt(od), stream_ptr(dev))
    return c


def dense_nn(dy2, w, precise, add=None, out_dtype=None):
    """dy2 [S,N] @ w[N,K] (+ add [S,K]) -> [S,K]: the input gradient of nn.Linear from the weight as stored."""
    S, N = dy2.shape
    K = w.shape[1]
    dev = dy2.device
    if precise:
        a, b, nn_, od = _split_cols(dy2.float().contiguous(), 0), _split_rows(w.float().contiguous(), 1, None, 1, N), 3 * N, torch.float32
    else:
        a, b, nn_, od = _as_bf16(dy2), _as_bf16(w), N, (out_dtype or torch.bfloat16)
    if add is not None:
        add = add.to(od).contiguous()
    c = torch.empty(S, K, dtype=od, device=dev)
    call("ab_dense_gemm_nn", ptr(a), ptr(b), None, ptr(add), ptr(c), S, K, nn_, _lib.EPI_ADD if add is not None else _lib.EPI_NONE,
         dt(od), stream_ptr(dev))
    return c


def dense_tn(dy2, x2, precise):
    """dy2 [S,N]^T @ x2 [S,K] -> fp32 [N,K]: the weight gradient of nn.Linear."""
    S, N = dy2.shape
    K = x2.shape[1]
    dev = dy2.device
    if precise:
        a, b, ss = _split_rows(dy2.float().contiguous(), 0, None, 1, S), _split_rows(x2.float().contiguous(), 1, None, 1, S), 3 * S
    else:
        a, b, ss = _as_bf16(dy2), _as_bf16(x2), S
    c = torch.empty(N, K, dtype=torch.float32, device=dev)
    nws = query("ab_dense_gemm_tn_workspace_bytes", ss, N, K)
    ws = torch.empty(nws, dtype=torch.uint8, device=dev) if nws else None
    call("ab_dense_gemm_tn", ptr(a), ptr(b), ptr(c), ptr(ws), nws, ss, N, K, stream_ptr(dev))
    return c


class _Linear(torch.autograd.Function):
    """nn.Linear (optionally several weights stacked along the output dim) on the library's GEMM: x [..., K] -> [..., N]."""

    @staticmethod
    def forward(ctx, x, bias, precise, *weights):
        _lib.ensure_device(x.device)
        with torch.cuda.device(x.device):
            K = x.shape[-1]
            x2 = x.reshape(-1, K)
            w = weights[0] if len(weights) == 1 else torch.cat([wi.reshape(-1, K) for wi in weights], 0)
            wb = w.float().contiguous() if precise else _as_bf16(w)
            xb = x2.float().contiguous() if precise else _as_bf16(x2)
            y = dense_nt(xb, wb, precise, bias=bias.float().contiguous() if bias is not None else None)
            ctx.save_for_backward(xb, wb)
            ctx.meta = (precise, x.shape, x.dtype, [wi.shape[0] for wi in weights], [wi.dtype for wi in weights],
                        bias.dtype if bias is not None else None)
            return y.view(*x.shape[:-1], w.shape[0])

    @staticmethod
    def backward(ctx, dy):
        xb, wb = ctx.saved_tensors
        precise, xshape, xdtype, splits, wdtypes, bdtype = ctx.meta
        with torch.cuda.device(dy.device):
            N = wb.shape[0]
            dy2 = dy.reshape(-1, N)
            dyb = dy2.float().contiguous() if precise else _as_bf16(dy2)
            dx = dense_nn(dyb, wb, precise).view(xshape) if ctx.needs_input_grad[0] else None
            dw = dense_tn(dyb, xb, precise)
            db = dy2.float().sum(0).to(bdtype) if bdtype is not None else None
            dws = [g.to(d) for g, d in zip(dw.split(splits, 0), wdtypes)]
            if dx is not None and dx.dtype != xdtype:
                dx = dx.to(xdtype)
            return (dx, db, None, *dws)


def linear(x, weights, bias=None, precise=False):
    """F.linear(x, cat(weights), bias) through ab_dense_gemm_*; `weights` is one tensor or a list stacked along dim 0."""
    if torch.is_tensor(weights):
        weights = [weights]
    return _Linear.apply(x, bias, precise, *weights)


class _SSMCore(torch.autograd.Function):
    """conv1d + SiLU -> fused parameter projection -> selective scan (core.py:368-396) as one autograd node, so that the
    intermediate gradients are written in place: the scan's dz and the conv's dxp land in the two halves of d[xp | z], the
    scan's direct d xa is added in the epilogue of the projection's input-gradient GEMM.

    xz [B,L,2Di] = [xp | z] (in-projection output); returns y [B,L,Di] (gated scan output)."""

    @staticmethod
    def forward(ctx, xz, conv_w, conv_b, Wp, Wdt, dt_bias, A_log, D, precise):
        _lib.ensure_device(xz.device)
        with torch.cuda.device(xz.device):
            dev = xz.device
            B, L, Di2 = xz.shape
            Di = Di2 // 2
            H, R = Wdt.shape
            Hp = (H + 7) // 8 * 8
            Kc = conv_w.shape[-1]
            W = Hp + 2 * Di
            cdt = torch.float32 if precise else torch.bfloat16
            xz = xz.to(cdt).contiguous()
            cw, cb = conv_w.reshape(Di, Kc).float().contiguous(), conv_b.float().contiguous()
            xp, z = xz[..., :Di], xz[..., Di:]
            xa = torch.empty(B, L, Di, dtype=cdt, device=dev)
            call("ab_causal_conv1d_silu_fwd", ptr(xp), Di2, ptr(cw), ptr(cb), ptr(xa), B, L, Di, Kc, dt(cdt), stream_ptr(dev))
            Wp32, Wdt32 = Wp.float().contiguous(), Wdt.float().contiguous()
            wcat = torch.empty(W, Di, dtype=cdt, device=dev)
            call("ab_dt_compose_fwd", ptr(Wp32), ptr(Wdt32), ptr(wcat), H, Hp, R, Di, dt(cdt), stream_ptr(dev))
            prm = dense_nt(xa.view(B * L, Di), wcat, precise).view(B, L, W)
            A = A_log.reshape(-1).float().contiguous()
            Dv = D.float().contiguous()
            bias = dt_bias.float().contiguous()
            nstate, nws = _rounds_plan(B, L, Di, cdt)
            ws = _rounds_workspace(dev, nws)
            y = torch.empty(B, L, Di, dtype=cdt, device=dev)
            state = torch.empty(nstate, dtype=torch.float32, device=dev)
            call("ab_ssm_scan_fwd", ptr(xa), Di, ptr(prm), W, ptr(bias), ptr(prm[..., Hp:]), ptr(prm[..., Hp + Di:]), W, ptr(z), Di2,
                 ptr(A), ptr(Dv), None, ptr(y), None, None, ptr(state), ptr(ws), ws.numel(), B, L, Di, H, dt(cdt), stream_ptr(dev))
            ctx.save_for_backward(xz, cw, cb, xa, wcat, prm, A, Dv, state, Wp32, Wdt32)
            ctx.meta = (precise, H, Hp, R, Kc, conv_w.shape, conv_w.dtype, conv_b.dtype, Wp.dtype, Wdt.dtype, dt_bias.dtype, A_log.shape)
            return y

    @staticmethod
    def backward(ctx, dy):
        xz, cw, cb, xa, wcat, prm, A, Dv, state, Wp32, Wdt32 = ctx.saved_tensors
        precise, H, Hp, R, Kc, cw_shape, cw_dtype, cb_dtype, wp_dtype, wdt_dtype, bias_dtype, a_shape = ctx.meta
        with torch.cuda.device(dy.device):
            dev = dy.device
            B, L, Di2 = xz.shape
            Di = Di2 // 2
            W = Hp + 2 * Di
            cdt = xz.dtype
            S = B * L
            dy = dy.to(cdt).contiguous()
            z = xz[..., Di:]
            nstate, nws = _rounds_plan(B, L, Di, cdt)
            ws = _rounds_workspace(dev, nws)
            dxz = torch.empty(B, L, Di2, dtype=cdt, device=dev)
            dxa_s = torch.empty(B, L, Di, dtype=cdt, device=dev)
            dprm = torch.empty(B, L, W, dtype=cdt, device=dev)
            dA = torch.empty(Di, dtype=torch.float32, device=dev)
            dD = torch.empty(Di, dtype=torch.float32, device=dev)
            dbias = torch.empty(H, dtype=torch.float32, device=dev)
            call("ab_ssm_scan_bwd", ptr(xa), Di, ptr(prm[..., Hp:]), ptr(prm[..., Hp + Di:]), W, ptr(z), Di2, ptr(dy), None, ptr(A),
                 ptr(Dv), ptr(state), ptr(dxa_s), Di, ptr(dprm[..., Hp:]), ptr(dprm[..., Hp + Di:]), W, ptr(dxz[..., Di:]), Di2,
                 ptr(dprm), W, Hp, ptr(dbias), ptr(dA), ptr(dD), ptr(ws), ws.numel(), B, L, Di, H, dt(cdt), stream_ptr(dev))
            # projection backward: d xa = d prm @ Wcat + (scan's direct d xa), d Wcat = d prm^T @ xa
            dprm2, xa2 = dprm.view(S, W), xa.view(S, Di)
            dxa = dense_nn(dprm2, wcat, precise, add=dxa_s.view(S, Di), out_dtype=cdt)
            dwcat = dense_tn(dprm2, xa2, precise)
            dWp = torch.empty(R + 2 * Di, Di, dtype=torch.float32, device=dev)
            dWdt = torch.empty(H, R, dtype=torch.float32, device=dev)
            call("ab_dt_compose_bwd", ptr(dwcat), ptr(Wp32), ptr(Wdt32), ptr(dWp), ptr(dWdt), H, Hp, R, Di, stream_ptr(dev))
            # conv backward writes d xp into the first half of d[xp | z]
            dcw = torch.empty(Di, Kc, dtype=torch.float32, device=dev)
            dcb = torch.empty(Di, dtype=torch.float32, device=dev)
            ncw = query("ab_causal_conv1d_silu_bwd_workspace_bytes", B, L, Di)
            cws = torch.empty(ncw, dtype=torch.uint8, device=dev)
            call("ab_causal_conv1d_silu_bwd", ptr(xz), Di2, ptr(dxa), ptr(cw), ptr(cb), ptr(dxz), Di2, ptr(dcw), ptr(dcb), ptr(cws), ncw,
                 B, L, Di, Kc, dt(cdt), stream_ptr(dev))
            return (dxz, dcw.reshape(cw_shape).to(cw_dtype), dcb.to(cb_dtype), dWp.to(wp_dtype), dWdt.to(wdt_dtype),
                    dbias.to(bias_dtype), dA.reshape(a_shape), dD, None)


class _DtCompose(torch.autograd.Function):
    """Wcat = [Wdt @ Wp[:R] ; 0 ; Wp[R:]] (csrc/ssm_proj.cu) with its gradient mapped back to the two parameters."""

    @staticmethod
    def forward(ctx, Wp, Wdt, precise):
        _lib.ensure_device(Wp.device)
        with torch.cuda.device(Wp.device):
            H, R = Wdt.shape
            Di = Wp.shape[1]
            Hp = (H + 7) // 8 * 8
            cdt = torch.float32 if precise else torch.bfloat16
            Wp32, Wdt32 = Wp.float().contiguous(), Wdt.float().contiguous()
            wcat = torch.empty(Hp + 2 * Di, Di, dtype=cdt, device=Wp.device)
            call("ab_dt_compose_fwd", ptr(Wp32), ptr(Wdt32), ptr(wcat), H, Hp, R, Di, dt(cdt), stream_ptr(Wp.device))
            ctx.save_for_backward(Wp32, Wdt32)
            ctx.meta = (H, Hp, R, Di, Wp.dtype, Wdt.dtype)
            return wcat

    @staticmethod
    def backward(ctx, dwcat):
        Wp32, Wdt32 = ctx.saved_tensors
        H, Hp, R, Di, wp_dtype, wdt_dtype = ctx.meta
        with torch.cuda.device(dwcat.device):
            dw = dwcat.float().contiguous()
            dWp = torch.empty(R + 2 * Di, Di, dtype=torch.float32, device=dw.device)
            dWdt = torch.empty(H, R, dtype=torch.float32, device=dw.device)
            call("ab_dt_compose_bwd", ptr(dw), ptr(Wp32), ptr(Wdt32), ptr(dWp), ptr(dWdt), H, Hp, R, Di, stream_ptr(dw.device))
            return dWp.to(wp_dtype), dWdt.to(wdt_dtype), None


def dt_compose(Wp, Wdt, precise=False):
    """Stacked weight of the fused parameter projection: [dt rows (H, padded to a multiple of 8) | B rows | C rows]."""
    return _DtCompose.apply(Wp, Wdt, precise)


def ssm_core(xz, conv_w, conv_b, Wp, Wdt, dt_bias, A_log, D, precise):
    return _SSMCore.apply(xz, conv_w, conv_b, Wp, Wdt, dt_bias, A_log, D, precise)


# --------------------------------------------------------------------------------------------
# language-model head + shifted cross-entropy (core.py:1412-1460)
# --------------------------------------------------------------------------------------------
class _LMHeadCE(torch.autograd.Function):
    """logits = hidden @ weight^T on the tcgen05 GEMM, loss = CrossEntropy(logits[:, :-1], labels[:, 1:]) (mean over the
    positions whose label is not ignore_index) with one read of the logits forward and one write of d logits backward.
    Returns (logits [B, L, V], loss); both are differentiable (a gradient arriving on the logits is added)."""

    @staticmethod
    @_on_tensor_device
    def forward(ctx, hidden, weight, labels, ignore_index, precise):
        _lib.ensure_device(hidden.device)
        dev = hidden.device
        B, L, Dm = hidden.shape
        V = weight.shape[0]
        h2 = hidden.reshape(B * L, Dm)
        hb = h2.float().contiguous() if precise else _as_bf16(h2)
        wb = weight.float().contiguous() if precise else _as_bf16(weight)
        logits = dense_nt(hb, wb, precise)                      # [B*L, V] fp32 | bf16
        labels = labels.to(torch.int64).contiguous()
        n = B * (L - 1)
        f32 = dict(dtype=torch.float32, device=dev)
        lse, row_loss, row_valid, sums = torch.empty(n, **f32), torch.empty(n, **f32), torch.empty(n, **f32), torch.empty(2, **f32)
        call("ab_shifted_ce_fwd", ptr(logits), ptr(labels), ptr(lse), ptr(row_loss), ptr(row_valid), ptr(sums), B, L, V, int(ignore_index),
             dt(logits), stream_ptr(dev))
        loss = sums[0] / sums[1]
        ctx.save_for_backward(hb, wb, logits, labels, lse, sums)
        ctx.meta = (B, L, V, Dm, int(ignore_index), precise, hidden.dtype, weight.dtype)
        return logits.view(B, L, V), loss

    @staticmethod
    @_on_tensor_device
    def backward(ctx, dlogits_ext, dloss):
        hb, wb, logits, labels, lse, sums = ctx.saved_tensors
        B, L, V, Dm, ignore_index, precise, hdtype, wdtype = ctx.meta
        dev = logits.device
        g = dloss.float() if dloss is not None else torch.zeros((), dtype=torch.float32, device=dev)
        scale = (g / sums[1]).reshape(1).contiguous()
        dl = torch.empty_like(logits)
        call("ab_shifted_ce_bwd", ptr(logits), ptr(labels), ptr(lse), ptr(scale), ptr(dl), B, L, V, ignore_index, dt(logits), stream_ptr(dev))
        if dlogits_ext is not None:
            dl += dlogits_ext.reshape(B * L, V).to(dl.dtype)
        dlb = dl if precise else _as_bf16(dl)
        dh = dense_nn(dlb, wb, precise).view(B, L, Dm).to(hdtype)
        dw = dense_tn(dlb, hb, precise).to(wdtype)
        return dh, dw, None, None, None


def lm_head_cross_entropy(hidden, weight, labels, ignore_index: int = -100, precise: bool = False):
    """(logits, loss) of the causal-LM head; see _LMHeadCE."""
    return _LMHeadCE.apply(hidden, weight, labels, ignore_index, precise)


# --------------------------------------------------------------------------------------------
# MoE
# --------------------------------------------------------------------------------------------
def _u8(n, dev):
    return torch.empty(max(int(n), 16), dtype=torch.uint8, device=dev)


_side_streams = {}


def _side_stream(device) -> torch.cuda.Stream:
    """One auxiliary stream per device for work that is off the critical path of the MoE (weight casts while the router
    and the plan run, bias column sums beside the gradient GEMMs).  Fork / join by stream waits: capturable in CUDA graphs."""
    st = _side_streams.get(device.index)
    if st is None:
        st = torch.cuda.Stream(device=device)
        _side_streams[device.index] = st
    return st


def moe_route(x2, ln_w, ln_b, eps, Wr, br, noise, noise_scale, K, quant=_lib.ROUTER_EXACT):
    """Router forward (no autograd).  Returns dict of routing tensors."""
    S, Dm = x2.shape
    E = Wr.shape[0]
    dev = x2.device
    f32 = dict(dtype=torch.float32, device=dev)
    r = dict(lclean=torch.empty(S, E, **f32), logits=torch.empty(S, E, **f32), gates=torch.empty(S, E, **f32),
             idx=torch.empty(S, K, dtype=torch.int32, device=dev), probs=torch.empty(S, K, **f32),
             w=torch.empty(S, K, **f32), lse=torch.empty(S, **f32), stats=torch.empty(S, 2, **f32),
             aux=torch.empty(2 * E + 1, **f32))
    nws = query("ab_moe_router_workspace_bytes", S, Dm, E)
    ws = _u8(nws, dev)
    call("ab_moe_router_fwd", ptr(x2), ptr(ln_w), ptr(ln_b), float(eps), ptr(Wr), ptr(br), ptr(noise), ptr(noise_scale),
         ptr(r["lclean"]), ptr(r["logits"]), ptr(r["gates"]), ptr(r["idx"]), ptr(r["probs"]), ptr(r["w"]), ptr(r["lse"]),
         ptr(r["stats"]), ptr(r["aux"]), ptr(ws), ws.numel(), S, Dm, E, K, dt(x2), quant, stream_ptr())
    return r


def moe_topk_from_logits(logits, K):
    S, E = logits.shape
    dev = logits.device
    f32 = dict(dtype=torch.float32, device=dev)
    gates, probs, w, lse = torch.empty(S, E, **f32), torch.empty(S, K, **f32), torch.empty(S, K, **f32), torch.empty(S, **f32)
    idx = torch.empty(S, K, dtype=torch.int32, device=dev)
    call("ab_moe_topk_from_logits", ptr(logits.contiguous()), ptr(gates), ptr(idx), ptr(probs), ptr(w), ptr(lse), S, E, K, stream_ptr())
    return gates, idx, probs, w, lse


def moe_plan(idx, w, E, cap, active=None, fixed_seg=0):
    """Capacity plan on the device (no host sync).  idx [S,K] int32, w [S,K] fp32.
    fixed_seg > 0: every expert segment is exactly fixed_seg rows (expert-parallel exchange layout)."""
    S, K = idx.shape
    dev = idx.device
    cap = int(min(cap, S))
    max_rows = E * fixed_seg if fixed_seg > 0 else int(query("ab_moe_max_rows", S, K, E, cap, ROW_ALIGN))
    i32 = dict(dtype=torch.int32, device=dev)
    p = dict(counts=torch.empty(E, **i32), seg_off=torch.empty(E + 1, **i32), row_of=torch.empty(S, K, **i32),
             tok_of_row=torch.empty(max_rows, **i32), slot_of_row=torch.empty(max_rows, **i32),
             tile_expert=torch.empty(max_rows // ROW_ALIGN, **i32), n_rows=torch.empty(2, **i32), max_rows=max_rows, cap=cap)
    nws = query("ab_moe_plan_workspace_bytes", S, K, E)
    ws = _u8(nws, dev)
    call("ab_moe_plan", ptr(idx), ptr(w), ptr(active), cap, ptr(p["counts"]), ptr(p["seg_off"]), ptr(p["row_of"]),
         ptr(p["tok_of_row"]), ptr(p["slot_of_row"]), ptr(p["tile_expert"]), ptr(p["n_rows"]), ptr(ws), ws.numel(),
         S, K, E, ROW_ALIGN, max_rows, fixed_seg, stream_ptr())
    return p


def _cast_bf16(t):
    out = torch.empty(t.shape, dtype=torch.bfloat16, device=t.device)
    call("ab_cast_f32_to_bf16", ptr(t), ptr(out), t.numel(), stream_ptr())
    return out


def _split_cols(t2d, which):
    rows, cols = t2d.shape
    out = torch.empty(rows, 3 * cols, dtype=torch.bfloat16, device=t2d.device)
    call("ab_split_f32_to_bf16x3", ptr(t2d), ptr(out), rows, cols, which, stream_ptr())
    return out


def _split_rows(t2d, which, seg_off=None, G=1, rows_per_group=0):
    rows, cols = t2d.shape
    out = torch.empty(3 * rows, cols, dtype=torch.bfloat16, device=t2d.device)
    call("ab_split_f32_to_bf16x3_rows", ptr(t2d), ptr(out), ptr(seg_off), G, rows_per_group, cols, which, stream_ptr())
    return out


def grouped_gemm(mode, A, W, plan, N, K, E, *, bias=None, aux=None, epi=_lib.EPI_NONE, act=0, out_dtype=torch.bfloat16,
                 want_c2=False, drop_p=0.0, drop_seed=None, out=None):
    """C = epi(A @ W[e]^T) ('nt', W [E,N,K]) or epi(A @ W[e]) ('nn', W [E,K,N]) over the permuted rows.
    out: write C into this [max_rows, N] tensor (e.g. a peer-mapped buffer) instead of a fresh one."""
    max_rows = A.shape[0]
    if out is not None:
        assert out.shape == (max_rows, N) and out.dtype == out_dtype and out.is_contiguous()
    c = out if out is not None else torch.empty(max_rows, N, dtype=out_dtype, device=A.device)
    c2 = torch.empty(max_rows, N, dtype=out_dtype, device=A.device) if want_c2 else None
    call("ab_grouped_gemm_" + mode, ptr(A), ptr(W), ptr(bias), ptr(aux), ptr(c), ptr(c2), ptr(plan["tile_expert"]),
         ptr(plan["n_rows"]), max_rows, N, K, E, epi, act, dt(out_dtype), float(drop_p), ptr(drop_seed), stream_ptr())
    return (c, c2) if want_c2 else c


def grouped_gemm_tn(A, Bm, seg_off, M, N, E, nsrc=1, src_stride=0):
    """Cw[e] = A[seg e]^T @ Bm[seg e]  -> fp32 [E, M, N]; with nsrc > 1 an expert's rows are nsrc strided blocks."""
    out = torch.empty(E, M, N, dtype=torch.float32, device=A.device)
    nws = query("ab_grouped_gemm_tn_workspace_bytes", M, N, E, nsrc)        # > 0: the contraction is cut over the source blocks
    ws = torch.empty(nws, dtype=torch.uint8, device=A.device) if nws else None
    call("ab_grouped_gemm_tn", ptr(A), ptr(Bm), ptr(out), ptr(seg_off), A.shape[0], M, N, E, nsrc, src_stride, ptr(ws), nws, stream_ptr())
    return out


def _colsum_side(side, main, a, plan, out, ws, C, E, max_rows, dev):
    """Column sums of `a` per expert segment on the side stream, after everything queued on the main stream so far."""
    side.wait_stream(main)
    with torch.cuda.stream(side):
        call("ab_moe_segment_colsum", ptr(a), ptr(plan["tile_expert"]), ptr(plan["n_rows"]), ptr(out), ptr(ws), ws.numel(), C, E,
             ROW_ALIGN, max_rows, dt(a), stream_ptr(dev))


class _MoEExperts(torch.autograd.Function):
    """Whole AdaptiveExpertSystem.forward as one autograd node.

    inputs: x2 [S,Dm]; router_norm weight/bias; router weight/bias; noise [S,E] | None; noise_scale [E] | None;
            stacked expert params ln_w/ln_b [E,Dm], W1 [E,I,Dm], b1 [E,I], W2 [E,Dm,I], b2 [E,Dm]
    cfg:    dict(K, eps, act, training, cap, lb_coef, rz_coef, active (int32 [E] | None), precise (fp32-accurate GEMMs))
    returns out [S,Dm], lb, rz, counts (non-differentiable int32 [E])"""

    @staticmethod
    @_on_tensor_device
    def forward(ctx, x2, rn_w, rn_b, Wr, br, noise, noise_scale, ln_w, ln_b, W1, b1, W2, b2, res, cfg):
        _lib.ensure_device(x2.device)
        dev = x2.device
        S, Dm = x2.shape
        E, I, _ = W1.shape
        K, act, training, precise = cfg["K"], cfg["act"], cfg["training"], cfg["precise"]
        x2 = x2.contiguous()
        f = lambda t: t.float().contiguous()
        rn_w, rn_b, Wr, br, ln_w, ln_b, b1, b2 = map(f, (rn_w, rn_b, Wr, br, ln_w, ln_b, b1, b2))
        W1, W2 = f(W1), f(W2)
        use_noise = noise is not None and noise_scale is not None
        main, side = torch.cuda.current_stream(dev), _side_stream(dev)
        w1 = w2 = None
        if not precise:
            # the bf16 shadows of the expert weights do not depend on the routing: cast them beside the router and the plan
            # (those are latency-bound kernels on a few SMs); buffers come from the main stream's pool
            w1, w2 = torch.empty(W1.shape, dtype=torch.bfloat16, device=dev), torch.empty(W2.shape, dtype=torch.bfloat16, device=dev)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                call("ab_cast_f32_to_bf16", ptr(W1), ptr(w1), W1.numel(), stream_ptr(dev))
                call("ab_cast_f32_to_bf16", ptr(W2), ptr(w2), W2.numel(), stream_ptr(dev))
        r = moe_route(x2, rn_w, rn_b, cfg["eps"], Wr, br, f(noise) if use_noise else None,
                      f(noise_scale) if use_noise else None, K, cfg.get("quant", _lib.ROUTER_EXACT))
        plan = moe_plan(r["idx"], r["w"], E, cfg["cap"], cfg["active"])
        max_rows = plan["max_rows"]
        cdt = torch.float32 if precise else torch.bfloat16         # dtype of the GEMM outputs that feed later GEMMs
        # ---- permute + per-expert LayerNorm
        xn = torch.empty(max_rows, Dm, dtype=cdt, device=dev)
        call("ab_moe_permute_ln", ptr(x2), ptr(r["stats"]), ptr(ln_w), ptr(ln_b), ptr(plan["tok_of_row"]), ptr(plan["tile_expert"]),
             ptr(plan["n_rows"]), ptr(xn), Dm, ROW_ALIGN, max_rows, dt(x2), dt(cdt), stream_ptr())
        if precise:
            a1 = _split_cols(xn, 0)
            w1 = _split_cols(W1.view(E * I, Dm), 1)
            k1 = 3 * Dm
        else:
            a1, k1 = xn, Dm
            main.wait_stream(side)
        drop_p = float(cfg.get("drop_p", 0.0)) if training else 0.0
        drop_seed = None
        if drop_p > 0.0:      # seed from torch's CUDA generator (restored by torch.utils.checkpoint on recompute), kept on device
            drop_seed = torch.randint(0, 2 ** 31 - 1, (2,), device=dev, dtype=torch.int32)
        h, hpre = grouped_gemm("nt", a1, w1, plan, I, k1, E, bias=b1, epi=_lib.EPI_BIAS_ACT, act=act, out_dtype=cdt, want_c2=True,
                               drop_p=drop_p, drop_seed=drop_seed)
        if precise:
            a2 = _split_cols(h, 0)
            w2 = _split_cols(W2.view(E * Dm, I), 1)
            k2 = 3 * I
        else:
            a2, k2 = h, I
        y = grouped_gemm("nt", a2, w2, plan, Dm, k2, E, bias=b2, epi=_lib.EPI_BIAS, out_dtype=cdt)
        # ---- combine (core.py:605) + the caller's output dropout and residual add (core.py:918-919) when it hands them in
        out_p = float(cfg.get("out_drop_p", 0.0)) if training else 0.0
        out_seed = torch.randint(0, 2 ** 31 - 1, (2,), device=dev, dtype=torch.int32) if out_p > 0.0 else None
        resc = res.reshape(S, Dm).float().contiguous() if res is not None else None
        out = torch.empty(S, Dm, dtype=x2.dtype if res is None else torch.float32, device=dev)
        call("ab_moe_unpermute", ptr(y), ptr(plan["row_of"]), ptr(r["w"]), ptr(resc), ptr(out), out_p, ptr(out_seed), S, K, Dm, dt(y), dt(out),
             stream_ptr())
        # ---- aux losses (core.py:499-505, 524-526) from the kernel's deterministic sums
        aux = r["aux"]
        zero = torch.zeros((), dtype=x2.dtype, device=dev)
        lb = (cfg["lb_coef"] * E / (S * S)) * (aux[:E] * aux[E:2 * E]).sum() if (training and cfg["lb_coef"] > 0) else zero
        rz = (cfg["rz_coef"] / S) * aux[2 * E] if (training and cfg["rz_coef"] > 0) else zero
        ctx.cfg = dict(cfg, S=S, Dm=Dm, E=E, I=I, use_noise=use_noise, max_rows=max_rows, cdt=cdt, drop_p=drop_p, out_p=out_p,
                       has_res=res is not None, res_shape=res.shape if res is not None else None,
                       res_dtype=res.dtype if res is not None else None)
        ctx.drop_seed = drop_seed
        ctx.out_seed = out_seed
        ctx.shadows = None if precise else (w1, w2)        # bf16 weight shadows cast in this forward, reused by the backward
        ctx.plan = {k: v for k, v in plan.items() if torch.is_tensor(v)}
        ctx.save_for_backward(x2, rn_w, rn_b, Wr, br, ln_w, W1, W2, noise if use_noise else None,
                              r["stats"], r["gates"], r["idx"], r["probs"], r["lse"], r["lclean"], r["w"], aux,
                              xn, h, hpre, y)
        ctx.routing = r
        counts = plan["counts"]
        ctx.mark_non_differentiable(counts)
        cfg["_routing"] = (r["idx"], plan["row_of"])     # for the caller's inspection: chosen experts, permuted row (-1 = dropped)
        return out, lb.to(x2.dtype) if torch.is_tensor(lb) else lb, rz.to(x2.dtype) if torch.is_tensor(rz) else rz, counts

    @staticmethod
    @_on_tensor_device
    def backward(ctx, dout, dlb, drz, _dcounts):
        (x2, rn_w, rn_b, Wr, br, ln_w, W1, W2, noise, stats, gates, idx, probs, lse, lclean, w, aux, xn, h, hpre, y) = ctx.saved_tensors
        cfg, plan = ctx.cfg, ctx.plan
        S, Dm, E, I, K = cfg["S"], cfg["Dm"], cfg["E"], cfg["I"], cfg["K"]
        act, precise, max_rows, cdt = cfg["act"], cfg["precise"], cfg["max_rows"], cfg["cdt"]
        dev = x2.device
        f32 = dict(dtype=torch.float32, device=dev)
        dout = dout.contiguous()
        # ---- combine backward: dY rows and d(gate weight)
        dy = torch.empty(max_rows, Dm, dtype=cdt, device=dev)
        dw_row = torch.empty(max_rows, **f32)
        call("ab_moe_unpermute_bwd", ptr(dout), ptr(y), ptr(w), ptr(plan["tok_of_row"]), ptr(plan["slot_of_row"]), ptr(plan["n_rows"]),
             ptr(dy), ptr(dw_row), cfg["out_p"], ptr(ctx.out_seed), K, Dm, max_rows, dt(dout), dt(y), dt(cdt), stream_ptr())
        seg = plan["seg_off"]
        # bias gradients (column sums of dY and dHpre over each expert's rows) run on the side stream beside the
        # latency-bound tail of this node (expert-LayerNorm backward, router backward); joined before the node returns
        main, side = torch.cuda.current_stream(dev), _side_stream(dev)
        db2 = torch.empty(E, Dm, **f32)
        db1 = torch.empty(E, I, **f32)
        ws_b2 = _u8(query("ab_moe_segment_colsum_workspace_bytes", Dm, ROW_ALIGN, max_rows), dev)
        ws_b1 = _u8(query("ab_moe_segment_colsum_workspace_bytes", I, ROW_ALIGN, max_rows), dev)
        if precise:
            seg3 = (seg * 3).contiguous()
            w2r = _split_rows(W2.view(E * Dm, I), 1, None, E, Dm)                 # [E, 3*Dm, I]
            dhpre = grouped_gemm("nn", _split_cols(dy, 0), w2r, plan, I, 3 * Dm, E, aux=hpre, epi=_lib.EPI_DACT, act=act, out_dtype=cdt,
                                 drop_p=cfg["drop_p"], drop_seed=ctx.drop_seed)
            dW2 = grouped_gemm_tn(_split_rows(dy, 0, seg, E), _split_rows(h, 1, seg, E), seg3, Dm, I, E)
            dW1 = grouped_gemm_tn(_split_rows(dhpre, 0, seg, E), _split_rows(xn, 1, seg, E), seg3, I, Dm, E)
            w1r = _split_rows(W1.view(E * I, Dm), 1, None, E, I)                  # [E, 3*I, Dm]
            dxn = grouped_gemm("nn", _split_cols(dhpre, 0), w1r, plan, Dm, 3 * I, E, out_dtype=torch.float32)
        else:
            w1b, w2b = ctx.shadows
            dhpre = grouped_gemm("nn", dy, w2b, plan, I, Dm, E, aux=hpre, epi=_lib.EPI_DACT, act=act, out_dtype=cdt,
                                 drop_p=cfg["drop_p"], drop_seed=ctx.drop_seed)
            dW2 = grouped_gemm_tn(dy, h, seg, Dm, I, E)
            dW1 = grouped_gemm_tn(dhpre, xn, seg, I, Dm, E)
            dxn = grouped_gemm("nn", dhpre, w1b, plan, Dm, I, E, out_dtype=torch.bfloat16)    # bf16 like the reference's autocast Linear backward
        # after the GEMMs (which fill every SM) come two latency-bound kernels: that is where the column sums run beside
        _colsum_side(side, main, dy, plan, db2, ws_b2, Dm, E, max_rows, dev)
        _colsum_side(side, main, dhpre, plan, db1, ws_b1, I, E, max_rows, dev)
        ws = _u8(query("ab_moe_permute_ln_bwd_workspace_bytes", Dm, ROW_ALIGN, max_rows), dev)
        # ---- per-expert LayerNorm backward on the permuted rows
        dxrow = torch.empty(max_rows, Dm, **f32)
        dln_w = torch.empty(E, Dm, **f32)
        dln_b = torch.empty(E, Dm, **f32)
        call("ab_moe_permute_ln_bwd", ptr(dxn), ptr(x2), ptr(stats), ptr(ln_w), ptr(plan["tok_of_row"]), ptr(plan["tile_expert"]),
             ptr(plan["n_rows"]), ptr(dxrow), ptr(dln_w), ptr(dln_b), ptr(ws), ws.numel(), Dm, E, ROW_ALIGN, max_rows, dt(x2),
             dt(dxn), stream_ptr())
        # ---- router backward (+ gather of the expert path into dx)
        training = cfg["training"]
        g_lb = (dlb.float() * (cfg["lb_coef"] * E / S)) if (training and cfg["lb_coef"] > 0) else torch.zeros((), **f32)
        g_rz = (drz.float() * (cfg["rz_coef"] / S)) if (training and cfg["rz_coef"] > 0) else torch.zeros((), **f32)
        scal = torch.stack([g_lb.reshape(()), g_rz.reshape(())]).contiguous()
        fvec = (aux[E:2 * E] / S).contiguous()
        dx = torch.empty_like(x2)
        dWr, dbr = torch.empty(E, Dm, **f32), torch.empty(E, **f32)
        drn_w, drn_b = torch.empty(Dm, **f32), torch.empty(Dm, **f32)
        dns = torch.empty(E, **f32) if cfg["use_noise"] else None
        nws = query("ab_moe_router_bwd_workspace_bytes", S, Dm, E)
        ws2 = _u8(nws, dev)
        call("ab_moe_router_bwd", ptr(x2), ptr(stats), ptr(rn_w), ptr(rn_b), ptr(Wr), ptr(br), ptr(gates), ptr(idx), ptr(probs),
             ptr(lse), ptr(lclean), ptr(noise.float().contiguous()) if cfg["use_noise"] else None, ptr(fvec), ptr(scal), ptr(dw_row),
             ptr(dxrow), ptr(plan["row_of"]), ptr(dx), ptr(dWr), ptr(dbr), ptr(drn_w), ptr(drn_b), ptr(dns), ptr(ws2), ws2.numel(),
             S, Dm, E, K, dt(x2), stream_ptr())
        dres = dout.reshape(cfg["res_shape"]).to(cfg["res_dtype"]) if cfg["has_res"] else None       # the residual passes the gradient on
        main.wait_stream(side)                                       # bias gradients
        return (dx, drn_w, drn_b, dWr, dbr, None, dns, dln_w, dln_b, dW1, db1, dW2, db2, dres, None)


def moe_experts(x2, rn_w, rn_b, Wr, br, noise, noise_scale, ln_w, ln_b, W1, b1, W2, b2, cfg, res=None):
    """res (optional, [S, Dm]): the caller's residual; with it the result is res + dropout(cfg['out_drop_p'])(moe(x2))."""
    return _MoEExperts.apply(x2, rn_w, rn_b, Wr, br, noise, noise_scale, ln_w, ln_b, W1, b1, W2, b2, res, cfg)


def moe_capacity(S: int, E: int, factor: float, training: bool, use_limit: bool) -> int:
    """core.py:508-511."""
    if use_limit and training and E > 0:
        return max(1, math.floor((S / E) * factor)) if S > 0 else 0
    return S
