"""Tensor-facing wrappers over the C ABI (one Python call = one kernel launch on the current
CUDA stream) and the host-side weight packers for adp_conv_gemm.

Activations are channels-last bf16 [B, T, C]; statistics fp64 [B, G, 2]; conditioning fp32.

`with ops.trace(timing=True) as tr:` records, for every launch made inside it, a label, the
algorithmic FLOPs / bytes of that launch and (optionally) CUDA events around it -- bench.py's
roofline and `gpu_launches` come from this, not from a side table.
"""
import ctypes as C
from typing import List, Optional, Sequence

import torch
from torch import Tensor

from . import _lib
from ._lib import (AttentionBwdArgs, ConvGemmArgs, NarrowConvArgs, NarrowConvBwdArgs, StemInArgs,
                   StemInBwdArgs, StemOutArgs, StemOutBwdArgs, WgradArgs)

ACT_NONE, ACT_GELU, ACT_SILU = 0, 1, 2


def _p(t: Optional[Tensor]):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def device_check() -> None:
    _lib.check(_lib.lib().adp_device_check(), "adp_device_check")


# -------------------------------------------------------------------------------- tracing
_TRACE = None


class trace:
    """Context manager collecting one record per kernel launch."""

    def __init__(self, timing: bool = False):
        self.timing, self.records = timing, []  # type: bool, List[dict]

    def __enter__(self):
        global _TRACE
        self._prev, _TRACE = _TRACE, self
        return self

    def __exit__(self, *exc):
        global _TRACE
        _TRACE = self._prev

    def table(self):
        """Aggregated by label: count, avg / total ms (after a sync), flops & bytes per launch."""
        if self.timing:
            torch.cuda.synchronize()
        out = {}
        for r in self.records:
            row = out.setdefault(r["name"], {"name": r["name"], "count": 0, "ms_total": 0.0,
                                             "flops": r["flops"], "bytes": r["bytes"]})
            row["count"] += 1
            if self.timing:
                row["ms_total"] += r["e0"].elapsed_time(r["e1"])
        for row in out.values():
            row["ms_avg"] = row["ms_total"] / row["count"]
        return out


def _launch(fn, what: str, meta):
    """meta: callable -> (label, flops, bytes); evaluated only while tracing."""
    tr = _TRACE
    if tr is None:
        _lib.check(fn(), what)
        return
    label, flops, nbytes = meta()
    rec = {"name": label, "flops": float(flops), "bytes": float(nbytes)}
    if tr.timing:
        rec["e0"] = torch.cuda.Event(enable_timing=True)
        rec["e1"] = torch.cuda.Event(enable_timing=True)
        rec["e0"].record()
    _lib.check(fn(), what)
    if tr.timing:
        rec["e1"].record()
    tr.records.append(rec)


def _nb(*tensors) -> int:
    return sum(t.numel() * t.element_size() for t in tensors if t is not None)


# ------------------------------------------------------------------------------ packers
def round_up(v: int, m: int) -> int:
    return (v + m - 1) // m * m


# storage type of packed GEMM operands: bf16 for the tensor-core path, fp32 while B200UNet packs
# for its fp32 verification mode (pack_dtype() context)
_PACK_DTYPE = [torch.bfloat16]


class pack_dtype:
    def __init__(self, dtype):
        self.dtype = dtype

    def __enter__(self):
        _PACK_DTYPE.append(self.dtype)

    def __exit__(self, *exc):
        _PACK_DTYPE.pop()


def packed_dtype():
    return _PACK_DTYPE[-1]


def _pad_rows(w2d: Tensor, n_pad: int) -> Tensor:
    out = torch.zeros(n_pad, w2d.shape[1], dtype=_PACK_DTYPE[-1], device=w2d.device)
    out[: w2d.shape[0]] = w2d.to(_PACK_DTYPE[-1])
    return out.contiguous()


def pack_conv(w: Tensor) -> Tensor:
    """Conv1d weight [co, ci, k] -> [n_pad, k*ci] (tap-major K), rows zero-padded to 16.
    Serves k=3 p=1 convs (taps -1,0,+1) and k=s=f downsample convs (1 tap over the
    [B, T/f, f*ci] view of the channels-last input)."""
    co, ci, k = w.shape
    return _pad_rows(w.permute(0, 2, 1).reshape(co, k * ci), round_up(co, 16))


def pack_linear(w: Tensor) -> Tensor:
    return _pad_rows(w, round_up(w.shape[0], 16))


def pack_upsample_conv(w: Tensor, f: int) -> Tensor:
    """nn.Upsample(nearest, f) -> Conv1d(k=3, p=1) folded into f output phases on the
    LOW-RES input: phase 0 = {W0 @ x[q-1], (W1+W2) @ x[q]}, phase f-1 = {(W0+W1) @ x[q],
    W2 @ x[q+1]}, interior phases = {(W0+W1+W2) @ x[q]}.  -> [f*n_pad, 2*ci]."""
    co, ci, k = w.shape
    assert k == 3 and f >= 2
    n_pad = round_up(co, 16)
    w = w.float()
    w0, w1, w2 = w[:, :, 0], w[:, :, 1], w[:, :, 2]
    out = torch.zeros(f, n_pad, 2 * ci, dtype=torch.float32, device=w.device)
    for p in range(f):
        if p == 0:
            out[p, :co, :ci], out[p, :co, ci:] = w0, w1 + w2
        elif p == f - 1:
            out[p, :co, :ci], out[p, :co, ci:] = w0 + w1, w2
        else:
            out[p, :co, :ci] = w0 + w1 + w2
    return out.reshape(f * n_pad, 2 * ci).to(_PACK_DTYPE[-1]).contiguous()


# ---------------------------------------------------------------------------------- ops
def conv_gemm(a: Tensor, w: Tensor, out: Tensor, *, c_in: int, n_valid: int,
              taps: Sequence[int] = (0,), up_factor: int = 0, bias: Optional[Tensor] = None,
              residual: Optional[Tensor] = None, gate: Optional[Tensor] = None,
              stats: Optional[Tensor] = None, groups: int = 8, block_n: int = 0) -> Tensor:
    """a: bf16 [B, T, lda]; w: packed bf16 [phases*n_pad, k_total]; out: [B, T, ldo]."""
    B, T, lda = a.shape
    phases = up_factor if up_factor > 1 else 1
    args = ConvGemmArgs()
    args.a, args.w, args.out = a.data_ptr(), w.data_ptr(), out.data_ptr()
    args.bias, args.residual, args.gate, args.stats = _p(bias), _p(residual), _p(gate), _p(stats)
    args.B, args.T, args.c_in, args.lda, args.ldo = B, T, c_in, lda, out.shape[-1]
    args.k_total = w.shape[1]
    args.n_pad, args.n_valid, args.phases = w.shape[0] // phases, n_valid, phases
    args.ntaps = len(taps)
    for i in range(3):
        args.tap_off[i] = taps[i] if i < len(taps) else 0
    args.up_factor, args.groups, args.block_n = up_factor, groups, block_n
    args.out_fp32 = 1 if out.dtype == torch.float32 else 0
    args.ld_gate = 0 if gate is None else gate.stride(0)

    def meta():
        rows = B * T
        tap_sum = len(taps) if up_factor <= 1 else (4 if up_factor == 2 else up_factor + 2)
        kind = "up%d" % up_factor if up_factor > 1 else "k%d" % len(taps)
        flops = 2.0 * rows * c_in * n_valid * tap_sum
        nbytes = rows * c_in * 2 + w.shape[0] * min(w.shape[1], tap_sum * c_in) * 2 \
            + rows * phases * n_valid * out.element_size() * (2 if residual is not None else 1)
        return f"conv_gemm[{kind} M={rows} K={c_in} N={n_valid}x{phases}]", flops, nbytes

    if a.dtype == torch.float32:       # fp32 verification mode (csrc/verify_f32.cu)
        assert w.dtype == torch.float32 and out.dtype == torch.float32
        assert residual is None or residual.dtype == torch.float32
        args.stats, args.out_fp32 = None, 0
        _launch(lambda: _lib.lib().adp_f32_conv_gemm(C.byref(args), _stream()), "adp_f32_conv_gemm", meta)
        if stats is not None:
            assert out.shape[-1] == phases * n_valid, "statistics need a dense output"
            gn_stats(out.reshape(B, -1, n_valid), stats, groups)
        return out
    _launch(lambda: _lib.lib().adp_conv_gemm(C.byref(args), _stream()), "adp_conv_gemm", meta)
    return out


def gn_silu(x: Tensor, y: Tensor, stats: Tensor, gamma: Tensor, beta: Tensor, groups: int,
            eps: float = 1e-5) -> Tensor:
    B, T, Cc = x.shape
    if x.dtype == torch.float32:
        _launch(lambda: _lib.lib().adp_f32_gn_silu(x.data_ptr(), y.data_ptr(), stats.data_ptr(), gamma.data_ptr(),
                                                   beta.data_ptr(), B, T, Cc, groups, eps, _stream()),
                "adp_f32_gn_silu", lambda: (f"f32_gn_silu[M={B * T} C={Cc}]", 0, _nb(x, y)))
        return y
    _launch(lambda: _lib.lib().adp_gn_silu(x.data_ptr(), y.data_ptr(), stats.data_ptr(),
                                           gamma.data_ptr(), beta.data_ptr(), B, T, Cc, groups,
                                           eps, _stream()), "adp_gn_silu",
            lambda: (f"gn_silu[M={B * T} C={Cc}]", 0, _nb(x, y)))
    return y


def gn_stats(x: Tensor, stats: Tensor, groups: int) -> Tensor:
    B, T, Cc = x.shape
    if x.dtype == torch.float32:
        assert x.is_contiguous()
        _launch(lambda: _lib.lib().adp_f32_gn_stats(x.data_ptr(), stats.data_ptr(), B, T, Cc, groups, _stream()),
                "adp_f32_gn_stats", lambda: (f"f32_gn_stats[M={B * T} C={Cc}]", 0, _nb(x)))
        return stats
    _launch(lambda: _lib.lib().adp_gn_stats(x.data_ptr(), stats.data_ptr(), B, T, Cc, groups,
                                            _stream()), "adp_gn_stats",
            lambda: (f"gn_stats[M={B * T} C={Cc}]", 0, _nb(x)))
    return stats


def ln_film(x: Tensor, y: Tensor, scale_shift: Optional[Tensor] = None, ss_stride: int = 0,
            stats_out: Optional[Tensor] = None, groups: int = 8, eps: float = 1e-6,
            y2: Optional[Tensor] = None, eps2: float = 1e-5) -> Tensor:
    """y = LN(x)*(1+scale)+shift; with y2 also y2 = LN(y; eps2) in the same pass."""
    B, T, Cc = x.shape
    if x.dtype == torch.float32:
        _launch(lambda: _lib.lib().adp_f32_ln_film(x.data_ptr(), y.data_ptr(), _p(y2), _p(scale_shift), ss_stride,
                                                   B, T, Cc, eps, eps2, _stream()),
                "adp_f32_ln_film", lambda: (f"f32_ln_film[M={B * T} C={Cc}]", 0, _nb(x, y, y2)))
        if stats_out is not None:
            gn_stats(y, stats_out, groups)
        return y
    if y2 is None:
        _launch(lambda: _lib.lib().adp_ln_film(x.data_ptr(), y.data_ptr(), _p(scale_shift), ss_stride,
                                               _p(stats_out), B, T, Cc, groups, eps, _stream()),
                "adp_ln_film", lambda: (f"ln_film[M={B * T} C={Cc}]", 0, _nb(x, y)))
    else:
        _launch(lambda: _lib.lib().adp_ln_film_dual(x.data_ptr(), y.data_ptr(), y2.data_ptr(),
                                                    _p(scale_shift), ss_stride, _p(stats_out), B, T, Cc,
                                                    groups, eps, eps2, _stream()),
                "adp_ln_film_dual", lambda: (f"ln_film_dual[M={B * T} C={Cc}]", 0, _nb(x, y, y2)))
    return y


def attention(q: Tensor, k: Tensor, v: Tensor, o: Tensor, heads: int, scale: float,
              lse: Optional[Tensor] = None) -> Tensor:
    """q: bf16 view [B, Tq, >=heads*64] (row pitch = stride(1)); k, v over Tk rows.
    lse: optional fp32 [B, heads, Tq] output (kept for attention_bwd)."""
    B, Tq = q.shape[0], q.shape[1]
    Tk = k.shape[1]
    if q.dtype == torch.float32:
        assert lse is None, "the fp32 verification mode covers inference only"
        _launch(lambda: _lib.lib().adp_f32_attention(q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(), B,
                                                     heads, Tq, Tk, q.stride(1), k.stride(1), v.stride(1),
                                                     o.stride(1), scale, _stream()),
                "adp_f32_attention", lambda: (f"f32_attention[B={B} H={heads} Tq={Tq} Tk={Tk}]",
                                              4.0 * B * heads * Tq * Tk * 64, 0))
        return o
    _launch(lambda: _lib.lib().adp_attention(q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(),
                                             B, heads, Tq, Tk, q.stride(1), k.stride(1),
                                             v.stride(1), o.stride(1), scale, _p(lse), _stream()),
            "adp_attention",
            lambda: (f"attention[B={B} H={heads} Tq={Tq} Tk={Tk}]", 4.0 * B * heads * Tq * Tk * 64,
                     (2 * B * Tq + 2 * B * Tk) * heads * 64 * 2))
    return o


def skinny_linear(x: Tensor, w: Tensor, bias: Optional[Tensor], y: Tensor, K: int, N: int,
                  in_act: int = ACT_NONE, out_act: int = ACT_NONE) -> Tensor:
    if w.dtype == torch.float32:
        _launch(lambda: _lib.lib().adp_f32_linear(x.data_ptr(), w.data_ptr(), _p(bias), y.data_ptr(), x.shape[0],
                                                  K, N, x.stride(0), w.stride(0), y.stride(0), in_act, out_act,
                                                  _stream()),
                "adp_f32_linear", lambda: (f"f32_linear[B={x.shape[0]} K={K} N={N}]", 2.0 * x.shape[0] * K * N,
                                           _nb(w)))
        return y
    _launch(lambda: _lib.lib().adp_skinny_linear(x.data_ptr(), w.data_ptr(), _p(bias), y.data_ptr(),
                                                 x.shape[0], K, N, x.stride(0), w.stride(0),
                                                 y.stride(0), in_act, out_act, _stream()),
            "adp_skinny_linear",
            lambda: (f"skinny_linear[B={x.shape[0]} K={K} N={N}]", 2.0 * x.shape[0] * K * N, _nb(w)))
    return y


def time_features(sigma: Tensor, freqs: Tensor, out: Tensor) -> Tensor:
    _launch(lambda: _lib.lib().adp_time_features(sigma.data_ptr(), freqs.data_ptr(), out.data_ptr(),
                                                 sigma.shape[0], freqs.shape[0], out.stride(0),
                                                 _stream()), "adp_time_features",
            lambda: ("time_features", 0, _nb(out)))
    return out


def silu_bf16(x: Tensor, y: Tensor) -> Tensor:
    if y.dtype == torch.float32:
        _launch(lambda: _lib.lib().adp_f32_silu(x.data_ptr(), y.data_ptr(), x.numel(), _stream()),
                "adp_f32_silu", lambda: ("f32_silu", 0, _nb(x, y)))
        return y
    _launch(lambda: _lib.lib().adp_silu_bf16(x.data_ptr(), y.data_ptr(), x.numel(), _stream()),
            "adp_silu_bf16", lambda: ("silu_bf16", 0, _nb(x, y)))
    return y


def stem_in(x: Tensor, w: Tensor, bias: Optional[Tensor], out: Tensor, f: int, *,
            append: Optional[Tensor] = None, noise: Optional[Tensor] = None,
            alpha: Optional[Tensor] = None, beta: Optional[Tensor] = None,
            stats: Optional[Tensor] = None, groups: int = 8) -> Tensor:
    a = StemInArgs()
    a.x, a.append, a.noise, a.alpha, a.beta = x.data_ptr(), _p(append), _p(noise), _p(alpha), _p(beta)
    a.w, a.bias, a.out, a.stats = w.data_ptr(), _p(bias), out.data_ptr(), _p(stats)
    a.B, a.cx, a.T = x.shape
    a.ca = 0 if append is None else append.shape[1]
    a.c0, a.f, a.groups = w.shape[0], f, groups
    if out.dtype == torch.float32:
        assert noise is None
        a.stats = None
        _launch(lambda: _lib.lib().adp_f32_stem_in(C.byref(a), _stream()), "adp_f32_stem_in",
                lambda: (f"f32_stem_in[B={x.shape[0]} T={x.shape[2]} c0={w.shape[0]}]", 0, _nb(x, append, out)))
        if stats is not None:
            gn_stats(out, stats, groups)
        return out
    _launch(lambda: _lib.lib().adp_stem_in(C.byref(a), _stream()), "adp_stem_in",
            lambda: (f"stem_in[B={x.shape[0]} T={x.shape[2]} c0={w.shape[0]}]",
                     2.0 * out.numel() * w.shape[1] * w.shape[2], _nb(x, append, noise, out)))
    return out


def stem_out(h: Tensor, x: Tensor, w: Tensor, bias: Optional[Tensor], gate: Tensor, f: int, *,
             append: Optional[Tensor] = None, w_adapt: Optional[Tensor] = None,
             b_adapt: Optional[Tensor] = None, v_out: Optional[Tensor] = None,
             x_next: Optional[Tensor] = None, ab: Optional[Tensor] = None,
             noise: Optional[Tensor] = None, alpha: Optional[Tensor] = None,
             beta: Optional[Tensor] = None, loss_sum: Optional[Tensor] = None,
             dv: Optional[Tensor] = None, cfg_scale: Optional[float] = None) -> None:
    a = StemOutArgs()
    a.h, a.x, a.append, a.w, a.bias = h.data_ptr(), x.data_ptr(), _p(append), w.data_ptr(), _p(bias)
    a.w_adapt, a.b_adapt, a.gate = _p(w_adapt), _p(b_adapt), gate.data_ptr()
    a.v_out, a.x_next, a.ab = _p(v_out), _p(x_next), _p(ab)
    a.noise, a.alpha, a.beta, a.loss_sum, a.dv = _p(noise), _p(alpha), _p(beta), _p(loss_sum), _p(dv)
    a.cfg = 0 if cfg_scale is None else 1
    a.cfg_scale = 1.0 if cfg_scale is None else cfg_scale
    a.B, a.cx, a.T = x.shape
    a.ca = 0 if append is None else append.shape[1]
    a.c0, a.co, a.f = h.shape[-1], w.shape[0], f
    a.ld_gate = gate.stride(0)
    if h.dtype == torch.float32:
        _launch(lambda: _lib.lib().adp_f32_stem_out(C.byref(a), _stream()), "adp_f32_stem_out",
                lambda: (f"f32_stem_out[B={x.shape[0]} T={x.shape[2]} c0={h.shape[-1]}]", 0, _nb(h, x, v_out)))
        return
    _launch(lambda: _lib.lib().adp_stem_out(C.byref(a), _stream()), "adp_stem_out",
            lambda: (f"stem_out[B={x.shape[0]} T={x.shape[2]} c0={h.shape[-1]}]",
                     2.0 * h.shape[0] * x.shape[2] * w.numel(),
                     _nb(h, x, append, noise, v_out, x_next, dv)))


def narrow_conv(x: Tensor, y: Tensor, stats_in: Tensor, gamma: Tensor, beta: Tensor, w: Tensor,
                bias: Optional[Tensor], groups: int, *, residual: Optional[Tensor] = None,
                scale_shift: Optional[Tensor] = None, ss_stride: int = 0,
                stats_out: Optional[Tensor] = None, gn_eps: float = 1e-5,
                ln_eps: float = 1e-6, w_packed: Optional[Tensor] = None) -> Tensor:
    a = NarrowConvArgs()
    a.w_packed = _p(w_packed)
    a.x, a.y, a.stats_in = x.data_ptr(), y.data_ptr(), stats_in.data_ptr()
    a.gamma, a.beta, a.w, a.bias = gamma.data_ptr(), beta.data_ptr(), w.data_ptr(), _p(bias)
    a.residual, a.scale_shift, a.stats_out = _p(residual), _p(scale_shift), _p(stats_out)
    a.ss_stride = ss_stride
    a.B, a.T, a.C = x.shape
    a.groups, a.gn_eps, a.ln_eps = groups, gn_eps, ln_eps
    _launch(lambda: _lib.lib().adp_narrow_conv(C.byref(a), _stream()), "adp_narrow_conv",
            lambda: (f"narrow_conv[M={x.shape[0] * x.shape[1]} C={x.shape[2]}"
                     f"{' +res+film' if residual is not None else ''}]",
                     2.0 * x.numel() * 3 * x.shape[2], _nb(x, y, residual)))
    return y   # C in (8, 32, 64): stem.cu narrow_conv_kernel / mid_conv.cu


def pack_mid_conv(w: Tensor) -> Tensor:
    """conv weight [C][C][3] (C = 32 / 64) -> bf16 [C][3*C], k = tap*C + ci: the smem image of
    adp_narrow_conv's B operand (adp_narrow_conv_args.w_packed)."""
    co, ci, k = w.shape
    return w.detach().permute(0, 2, 1).reshape(co, k * ci).to(torch.bfloat16).contiguous()


def sampler_step(x: Tensor, v: Tensor, ab: Tensor, x_next: Tensor) -> Tensor:
    _launch(lambda: _lib.lib().adp_sampler_step(x.data_ptr(), v.data_ptr(), ab.data_ptr(),
                                                x_next.data_ptr(), x.numel(), _stream()),
            "adp_sampler_step", lambda: ("sampler_step", 0, _nb(x, v, x_next)))
    return x_next


def step_select(step: Tensor, ctrl: Tensor, ab_table: Tensor, ab_out: Tensor, ss_out: Tensor) -> None:
    """ss_out <- table[step // ctrl[1]], ab_out <- ab_table[step]  (table address in ctrl[0])."""
    _launch(lambda: _lib.lib().adp_step_select(step.data_ptr(), ctrl.data_ptr(), ab_table.data_ptr(),
                                               ab_out.data_ptr(), ss_out.data_ptr(), ss_out.numel(), _stream()),
            "adp_step_select", lambda: ("step_select", 0, 2 * _nb(ss_out)))


def step_advance(step: Tensor) -> None:
    _launch(lambda: _lib.lib().adp_step_advance(step.data_ptr(), _stream()), "adp_step_advance",
            lambda: ("step_advance", 0, 4))


def inpaint_blend(x: Tensor, source: Tensor, noise: Tensor, mask_u8: Tensor, ab: Tensor) -> Tensor:
    """In place: x = ab[2]*source + ab[3]*noise where mask (VInpainter, reference diffusion.py:346-350)."""
    _launch(lambda: _lib.lib().adp_inpaint_blend(x.data_ptr(), source.data_ptr(), noise.data_ptr(),
                                                 mask_u8.data_ptr(), ab.data_ptr(), x.numel(), _stream()),
            "adp_inpaint_blend", lambda: ("inpaint_blend", 0, _nb(x, source, noise, mask_u8)))
    return x


def arv_step(chan: Tensor, v: Tensor, sig_next: Tensor) -> Tensor:
    """In place on chan [B, C+1, T] (current | sigma_i): the ARVSampler update with per-position
    noise levels (reference diffusion.py:231-235); channel C becomes sig_next [B, T]."""
    B, C1, T = chan.shape
    _launch(lambda: _lib.lib().adp_arv_step(chan.data_ptr(), v.data_ptr(), sig_next.data_ptr(), B, C1 - 1,
                                            T, _stream()),
            "adp_arv_step", lambda: ("arv_step", 0, 2 * _nb(chan) + _nb(v)))
    return chan


# ----------------------------------------------------------------------------- front-ends
def fir_resample(x: Tensor, bank: Tensor, factor_in: int, factor_out: int, half: int, t_out: int,
                 adjoint_of: Optional[int] = None) -> Tensor:
    """x fp32 [rows, t] -> [rows, t_out] through the polyphase bank [factor_out, taps]
    (adp_resample); with adjoint_of = t the transposed map [rows, t_out] -> [rows, t]."""
    rows = x.shape[0]
    taps = bank.shape[1]
    if adjoint_of is None:
        t = x.shape[1]
        y = torch.empty(rows, t_out, device=x.device, dtype=torch.float32)
        _launch(lambda: _lib.lib().adp_resample(x.data_ptr(), bank.data_ptr(), y.data_ptr(), rows, t, t_out,
                                                factor_in, factor_out, taps, half, _stream()),
                "adp_resample", lambda: (f"resample[{factor_in}->{factor_out}]", 2.0 * rows * t_out * taps,
                                         _nb(x, y)))
        return y
    t = adjoint_of
    dx = torch.empty(rows, t, device=x.device, dtype=torch.float32)
    _launch(lambda: _lib.lib().adp_resample_adjoint(x.data_ptr(), bank.data_ptr(), dx.data_ptr(), rows, t,
                                                    t_out, factor_in, factor_out, taps, half, _stream()),
            "adp_resample_adjoint", lambda: (f"resample_adjoint[{factor_in}->{factor_out}]",
                                             2.0 * rows * t_out * taps, _nb(x, dx)))
    return dx


def mel_spectrogram(wave: Tensor, window: Tensor, fb: Tensor, band: Tensor, n_fft: int, hop: int,
                    pad: int, apply_log: bool) -> Tensor:
    """wave fp32 [rows, t] -> mel fp32 [rows, n_mels, frames] (adp_mel_spectrogram)."""
    rows, t = wave.shape
    n_mels = fb.shape[1]
    frames = 1 + (t + 2 * pad - n_fft) // hop
    mel = torch.empty(rows, n_mels, frames, device=wave.device, dtype=torch.float32)
    _launch(lambda: _lib.lib().adp_mel_spectrogram(wave.data_ptr(), window.data_ptr(), fb.data_ptr(),
                                                   band.data_ptr(), mel.data_ptr(), rows, t, n_fft, hop, pad,
                                                   frames, n_mels, 1 if apply_log else 0, _stream()),
            "adp_mel_spectrogram", lambda: (f"mel_spectrogram[n_fft={n_fft}]", 0, _nb(wave, mel)))
    return mel


def to_flat(spec: Tensor, w: Tensor, hop: int, pad: int) -> Tensor:
    """spec fp32 [B, C, frames], w fp32 [C, win] -> [B, t_out] (adp_to_flat)."""
    B, Cc, frames = spec.shape
    win = w.shape[1]
    t_out = (frames - 1) * hop - 2 * pad + win
    out = torch.empty(B, t_out, device=spec.device, dtype=torch.float32)
    _launch(lambda: _lib.lib().adp_to_flat(spec.data_ptr(), w.data_ptr(), out.data_ptr(), B, Cc, frames, win,
                                           hop, pad, t_out, _stream()),
            "adp_to_flat", lambda: ("to_flat", 2.0 * B * t_out * Cc * (win // hop), _nb(spec, out)))
    return out


def to_flat_bwd(spec: Tensor, w: Tensor, dout: Tensor, hop: int, pad: int, need_dspec: bool,
                need_dw: bool):
    B, Cc, frames = spec.shape
    win = w.shape[1]
    t_out = dout.shape[1]
    dspec = torch.empty_like(spec) if need_dspec else None
    dw = torch.zeros_like(w) if need_dw else None
    _launch(lambda: _lib.lib().adp_to_flat_bwd(spec.data_ptr(), w.data_ptr(), dout.data_ptr(), _p(dspec),
                                               _p(dw), B, Cc, frames, win, hop, pad, t_out, _stream()),
            "adp_to_flat_bwd", lambda: ("to_flat_bwd", 4.0 * B * Cc * frames * win, _nb(spec, dout)))
    return dspec, dw


# ----------------------------------------------------------------------------- backward
def pack_conv_dgrad(w: Tensor) -> Tensor:
    """Weights of the data-gradient conv: dA[t] = sum_j dOut[t + o_j] @ Wt_j with the taps
    reversed and the matrices transposed ([co,ci,k] -> rows ci, K = (k reversed, co))."""
    return pack_conv(w.flip(2).transpose(0, 1).contiguous())


def wgrad(g: Tensor, x: Tensor, dw: Tensor, *, n: int, k: int, off: int = 0, g_col0: int = 0,
          x_col0: int = 0, ntaps: int = 1) -> Tensor:
    """dw[n_, k_] += sum_{b,t} g[b,t,g_col0+n_] * x[b,t+off,x_col0+k_]; g, x bf16 [B,T,ld].
    ntaps=3: dw is [3, n, k] and tap j uses row offset off + j (a whole k=3 conv in one launch)."""
    a = WgradArgs()
    a.ntaps = ntaps
    a.tap_stride = dw.stride(0) if ntaps == 3 else 0
    a.g, a.x, a.dw = g.data_ptr(), x.data_ptr(), dw.data_ptr()
    a.B, a.T = g.shape[0], g.shape[1]
    a.n, a.k = n, k
    a.ldg, a.ldx, a.ldw = g.stride(1), x.stride(1), dw.stride(-2)
    a.g_cols, a.x_cols = g.shape[2], x.shape[2]
    a.g_col0, a.x_col0, a.off = g_col0, x_col0, off
    _launch(lambda: _lib.lib().adp_wgrad(C.byref(a), _stream()), "adp_wgrad",
            lambda: (f"wgrad[M={g.shape[0] * g.shape[1]} n={n} k={k}{' x3' if ntaps == 3 else ''}]",
                     2.0 * g.shape[0] * g.shape[1] * n * k * ntaps, (g.shape[0] * g.shape[1]) * (n + k) * 2))
    return dw


def gn_silu_bwd(da: Tensor, x: Tensor, stats: Tensor, gamma: Tensor, beta: Tensor, dxh: Tensor,
                dgamma: Tensor, dbeta: Tensor, S: Tensor, groups: int, eps: float = 1e-5) -> Tensor:
    B, T, Cc = x.shape
    _launch(lambda: _lib.lib().adp_gn_silu_bwd(da.data_ptr(), x.data_ptr(), stats.data_ptr(),
                                               gamma.data_ptr(), beta.data_ptr(), dxh.data_ptr(),
                                               dgamma.data_ptr(), dbeta.data_ptr(), S.data_ptr(),
                                               B, T, Cc, groups, eps, _stream()),
            "adp_gn_silu_bwd", lambda: (f"gn_silu_bwd[M={B * T} C={Cc}]", 0, _nb(da, x, dxh)))
    return dxh


def gn_bwd_apply(dxh: Tensor, x: Tensor, stats: Tensor, S: Tensor, dx: Tensor, groups: int, *,
                 dres: Optional[Tensor] = None, colsum: Optional[Tensor] = None,
                 eps: float = 1e-5) -> Tensor:
    B, T, Cc = x.shape
    _launch(lambda: _lib.lib().adp_gn_bwd_apply(dxh.data_ptr(), x.data_ptr(), stats.data_ptr(),
                                                S.data_ptr(), _p(dres), dx.data_ptr(), _p(colsum),
                                                B, T, Cc, groups, eps, _stream()),
            "adp_gn_bwd_apply", lambda: (f"gn_bwd_apply[M={B * T} C={Cc}]", 0, _nb(dxh, x, dres, dx)))
    return dx


def ln_film_bwd(dy: Tensor, x: Tensor, scale_shift: Optional[Tensor], ss_stride: int, dx: Tensor, *,
                dss: Optional[Tensor] = None, dss_stride: int = 0,
                colsum: Optional[Tensor] = None, dres: Optional[Tensor] = None,
                eps: float = 1e-6) -> Tensor:
    B, T, Cc = x.shape
    _launch(lambda: _lib.lib().adp_ln_film_bwd(dy.data_ptr(), x.data_ptr(), _p(scale_shift),
                                               ss_stride, dx.data_ptr(), _p(dss), dss_stride,
                                               _p(colsum), _p(dres), B, T, Cc, eps, _stream()),
            "adp_ln_film_bwd", lambda: (f"ln_film_bwd[M={B * T} C={Cc}]", 0, _nb(dy, x, dx)))
    return dx


def colsum(x: Tensor, out: Tensor, gate: Optional[Tensor] = None) -> Tensor:
    B, T, Cc = x.shape
    _launch(lambda: _lib.lib().adp_colsum(x.data_ptr(), _p(gate), 0 if gate is None else gate.stride(0),
                                          out.data_ptr(), B, T, Cc, _stream()),
            "adp_colsum", lambda: (f"colsum[M={B * T} C={Cc}]", 0, _nb(x)))
    return out


def skip_gate(y: Tensor, skip: Tensor, gate: Tensor, out: Tensor, stats: Optional[Tensor],
              groups: int) -> Tensor:
    B, T, Cc = y.shape
    _launch(lambda: _lib.lib().adp_skip_gate(y.data_ptr(), skip.data_ptr(), gate.data_ptr(),
                                             gate.stride(0), out.data_ptr(), _p(stats), B, T, Cc,
                                             groups, _stream()),
            "adp_skip_gate", lambda: (f"skip_gate[M={B * T} C={Cc}]", 0, _nb(y, skip, out)))
    return out


def skip_gate_bwd(dout: Tensor, y: Tensor, gate: Tensor, dys: Tensor, dgate: Tensor) -> Tensor:
    B, T, Cc = y.shape
    _launch(lambda: _lib.lib().adp_skip_gate_bwd(dout.data_ptr(), y.data_ptr(), gate.data_ptr(),
                                                 gate.stride(0), dys.data_ptr(), dgate.data_ptr(),
                                                 dgate.stride(0), B, T, Cc, _stream()),
            "adp_skip_gate_bwd", lambda: (f"skip_gate_bwd[M={B * T} C={Cc}]", 0, _nb(dout, y, dys)))
    return dys


def cond_bwd(dss: Tensor, cond: Tensor, w: Tensor, dw: Tensor, dbias: Tensor, dcond: Optional[Tensor],
             N: int) -> None:
    B, K = cond.shape
    _launch(lambda: _lib.lib().adp_cond_bwd(dss.data_ptr(), dss.stride(0), cond.data_ptr(),
                                            w.data_ptr(), dw.data_ptr(), dbias.data_ptr(),
                                            _p(dcond), B, N, K, _stream()),
            "adp_cond_bwd", lambda: (f"cond_bwd[B={B} N={N} K={K}]", 4.0 * B * N * K, N * K * 6))


def narrow_conv_bwd(dy: Tensor, x: Tensor, stats_in: Tensor, gamma: Tensor, beta: Tensor,
                    w: Tensor, dxh: Tensor, dgamma: Tensor, dbeta: Tensor, S: Tensor, dw: Tensor,
                    dbias: Tensor, groups: int, gn_eps: float = 1e-5) -> Tensor:
    a = NarrowConvBwdArgs()
    a.dy, a.x, a.stats_in = dy.data_ptr(), x.data_ptr(), stats_in.data_ptr()
    a.gamma, a.beta, a.w = gamma.data_ptr(), beta.data_ptr(), w.data_ptr()
    a.dxh, a.dgamma, a.dbeta, a.S = dxh.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), S.data_ptr()
    a.dw, a.dbias = dw.data_ptr(), dbias.data_ptr()
    a.B, a.T, a.C = x.shape
    a.groups, a.gn_eps = groups, gn_eps
    _launch(lambda: _lib.lib().adp_narrow_conv_bwd(C.byref(a), _stream()), "adp_narrow_conv_bwd",
            lambda: (f"narrow_conv_bwd[M={x.shape[0] * x.shape[1]}]", 4.0 * x.numel() * 24, _nb(dy, x, dxh)))
    return dxh


def stem_out_bwd(dv: Tensor, h: Tensor, x: Tensor, w: Tensor, bias: Optional[Tensor], gate: Tensor,
                 f: int, dh: Tensor, dw: Tensor, dbias: Tensor, dgate: Tensor, *,
                 gscale: Optional[Tensor] = None, append: Optional[Tensor] = None,
                 noise: Optional[Tensor] = None, alpha: Optional[Tensor] = None,
                 beta: Optional[Tensor] = None, w_adapt: Optional[Tensor] = None,
                 dw_adapt: Optional[Tensor] = None, db_adapt: Optional[Tensor] = None,
                 dxin: Optional[Tensor] = None) -> Tensor:
    a = StemOutBwdArgs()
    a.dxin = _p(dxin)
    a.dv, a.gscale, a.h, a.x, a.append = dv.data_ptr(), _p(gscale), h.data_ptr(), x.data_ptr(), _p(append)
    a.noise, a.alpha, a.beta = _p(noise), _p(alpha), _p(beta)
    a.w, a.bias, a.w_adapt, a.gate = w.data_ptr(), _p(bias), _p(w_adapt), gate.data_ptr()
    a.dh, a.dw, a.dbias, a.dgate = dh.data_ptr(), dw.data_ptr(), dbias.data_ptr(), dgate.data_ptr()
    a.dw_adapt, a.db_adapt = _p(dw_adapt), _p(db_adapt)
    a.B, a.cx, a.T = x.shape
    a.ca = 0 if append is None else append.shape[1]
    a.c0, a.co, a.f = h.shape[-1], w.shape[0], f
    a.ld_gate, a.ld_dgate = gate.stride(0), dgate.stride(0)
    _launch(lambda: _lib.lib().adp_stem_out_bwd(C.byref(a), _stream()), "adp_stem_out_bwd",
            lambda: ("stem_out_bwd", 0, _nb(dv, h, x, dh)))
    return dh


def stem_in_bwd(dout: Tensor, x: Tensor, dw: Tensor, dbias: Tensor, f: int, *,
                append: Optional[Tensor] = None, noise: Optional[Tensor] = None,
                alpha: Optional[Tensor] = None, beta: Optional[Tensor] = None,
                w: Optional[Tensor] = None, dxin: Optional[Tensor] = None) -> None:
    a = StemInBwdArgs()
    a.w, a.dxin = _p(w), _p(dxin)
    a.dout, a.x, a.append = dout.data_ptr(), x.data_ptr(), _p(append)
    a.noise, a.alpha, a.beta = _p(noise), _p(alpha), _p(beta)
    a.dw, a.dbias = dw.data_ptr(), dbias.data_ptr()
    a.B, a.cx, a.T = x.shape
    a.ca = 0 if append is None else append.shape[1]
    a.c0, a.f = dout.shape[-1], f
    _launch(lambda: _lib.lib().adp_stem_in_bwd(C.byref(a), _stream()), "adp_stem_in_bwd",
            lambda: ("stem_in_bwd", 0, _nb(dout, x)))


def attention_bwd(q: Tensor, k: Tensor, v: Tensor, o: Tensor, d_o: Tensor, lse: Tensor, delta: Tensor,
                  dq: Tensor, dk: Tensor, dv: Tensor, heads: int, scale: float) -> None:
    """Backward of `attention`; all bf16 views [B, T, >=heads*64], lse / delta fp32 [B, heads, Tq]."""
    a = AttentionBwdArgs()
    a.q, a.k, a.v, a.o, a.d_o = q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(), d_o.data_ptr()
    a.lse, a.delta = lse.data_ptr(), delta.data_ptr()
    a.dq, a.dk, a.dv = dq.data_ptr(), dk.data_ptr(), dv.data_ptr()
    a.B, a.H, a.Tq, a.Tk = q.shape[0], heads, q.shape[1], k.shape[1]
    a.ldq, a.ldk, a.ldv, a.ldo, a.lddo = q.stride(1), k.stride(1), v.stride(1), o.stride(1), d_o.stride(1)
    a.lddq, a.lddk, a.lddv = dq.stride(1), dk.stride(1), dv.stride(1)
    a.scale = scale
    B, Tq, Tk = a.B, a.Tq, a.Tk
    _launch(lambda: _lib.lib().adp_attention_bwd(C.byref(a), _stream()), "adp_attention_bwd",
            lambda: (f"attention_bwd[B={B} H={heads} Tq={Tq} Tk={Tk}]", 14.0 * B * heads * Tq * Tk * 64,
                     (4 * B * Tq + 4 * B * Tk) * heads * 64 * 2))


def ln_fold_bwd(w: Tensor, g: Tensor, b: Tensor, dwf: Tensor, dbf: Tensor, dw: Tensor, dg: Tensor,
                db: Tensor) -> None:
    """Unfolds the gradient of a LayerNorm-affine-folded projection (see adp_ln_fold_bwd)."""
    N, Cc = w.shape
    _launch(lambda: _lib.lib().adp_ln_fold_bwd(w.data_ptr(), g.data_ptr(), b.data_ptr(), dwf.data_ptr(),
                                               dwf.stride(0), dbf.data_ptr(), dw.data_ptr(),
                                               dg.data_ptr(), db.data_ptr(), N, Cc, _stream()),
            "adp_ln_fold_bwd", lambda: (f"ln_fold_bwd[N={N} C={Cc}]", 0, 3 * N * Cc * 4))
