"""Per-kernel parity: every C-ABI entry point against a plain PyTorch fp32 restatement of
the a_unet / diffusion.py op it replaces (same bf16-rounded inputs, fp32 math).
Tolerances are written next to each check: outputs are bf16, so the bound is a few bf16
ulps (2^-8 relative) of the result plus accumulation-order noise."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda"
# the PyTorch restatements must be true fp32 (cuDNN/cuBLAS default to TF32 for conv/matmul)
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False


def bf(t):
    return t.to(torch.bfloat16)


def rnd(*shape, scale=1.0, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(DEV)


def assert_close(got, ref, rtol, atol, what):
    got, ref = got.float(), ref.float()
    err = (got - ref).abs()
    bound = atol + rtol * ref.abs()
    bad = err > bound
    msg = (f"{what}: max abs err {err.max().item():.4e}, ref max {ref.abs().max().item():.3e}, "
           f"violations {int(bad.sum())}/{bad.numel()}")
    print(msg)
    assert not bad.any(), msg


@pytest.fixture(scope="module")
def ops():
    from audio_diffusion_pytorch_b200 import ops
    ops.device_check()
    return ops


def stats_of(y, groups):
    """(sum, sumsq) per (batch, group) of a channels-last tensor."""
    B, T, Cc = y.shape
    yg = y.double().reshape(B, T, groups, Cc // groups)
    return torch.stack([yg.sum(dim=(1, 3)), (yg * yg).sum(dim=(1, 3))], dim=-1)


# ------------------------------------------------------------------------- conv_gemm
@pytest.mark.parametrize("B,T,cin,n", [
    (2, 256, 64, 64),      # SW128, one k-chunk
    (2, 384, 128, 256),    # SW128, two k-chunks, wide N
    (1, 128, 32, 32),      # SW64
    (3, 200, 16, 48),      # SW32, ragged T, n_pad 48
    (2, 40, 64, 8),        # T < tile, n_valid 8 (padded to 16)
    (1, 1024, 512, 1536),  # qkv-sized
    (2, 130, 1024, 128),   # long K pipeline (16 chunks > stages), ragged T
])
def test_conv_gemm_linear(ops, B, T, cin, n):
    a = bf(rnd(B, T, cin, seed=1))
    w = bf(rnd(n, cin, scale=cin ** -0.5, seed=2))
    bias = rnd(n, seed=3)
    out = torch.full((B, T, n), float("nan"), dtype=torch.bfloat16, device=DEV)
    ops.conv_gemm(a, ops.pack_linear(w), out, c_in=cin, n_valid=n, bias=bias)
    ref = a.float() @ w.float().t() + bias
    assert_close(out, ref, 2 ** -7, 1e-2, f"linear B{B} T{T} K{cin} N{n}")


@pytest.mark.parametrize("block_n", [16, 32, 64, 128, 256])
def test_conv_gemm_block_n(ops, block_n):
    B, T, cin, n = 2, 256, 128, 256
    a = bf(rnd(B, T, cin, seed=1))
    w = bf(rnd(n, cin, scale=cin ** -0.5, seed=2))
    out = torch.empty(B, T, n, dtype=torch.bfloat16, device=DEV)
    ops.conv_gemm(a, ops.pack_linear(w), out, c_in=cin, n_valid=n, block_n=block_n)
    assert_close(out, a.float() @ w.float().t(), 2 ** -7, 1e-2, f"block_n {block_n}")


def test_conv_gemm_fp32_out(ops):
    B, T, cin, n = 1, 8, 1024, 264
    a = bf(rnd(B, T, cin, seed=1))
    w = bf(rnd(n, cin, scale=cin ** -0.5, seed=2))
    bias = rnd(n, seed=3)
    out = torch.empty(B, T, n, dtype=torch.float32, device=DEV)
    ops.conv_gemm(a, ops.pack_linear(w), out, c_in=cin, n_valid=n, bias=bias)
    assert_close(out, a.float() @ w.float().t() + bias, 1e-4, 1e-4, "fp32 out")


@pytest.mark.parametrize("B,T,C,co", [(2, 512, 64, 64), (2, 300, 128, 128), (1, 256, 32, 32),
                                      (2, 100, 256, 256), (1, 128, 16, 16)])
def test_conv_gemm_conv3(ops, B, T, C, co):
    x = bf(rnd(B, T, C, seed=4))
    w = bf(rnd(co, C, 3, scale=(3 * C) ** -0.5, seed=5))
    bias = rnd(co, seed=6)
    res = bf(rnd(B, T, co, seed=7))
    groups = 8
    stats = torch.zeros(B, groups, 2, dtype=torch.float64, device=DEV)
    out = torch.empty(B, T, co, dtype=torch.bfloat16, device=DEV)
    ops.conv_gemm(x, ops.pack_conv(w), out, c_in=C, n_valid=co, taps=(-1, 0, 1), bias=bias,
                  residual=res, stats=stats, groups=groups)
    ref = F.conv1d(x.float().transpose(1, 2), w.float(), bias, padding=1).transpose(1, 2)
    ref = ref + res.float()
    assert_close(out, ref, 2 ** -7, 1e-2, f"conv3 C{C}")
    ref_stats = stats_of(out, groups)
    assert_close(stats, ref_stats, 1e-4, 1e-2, f"conv3 stats C{C}")


@pytest.mark.parametrize("B,T,C,co", [(2, 512, 64, 64), (1, 256, 1024, 1024), (8, 4096, 32, 32),
                                      (2, 300, 512, 128), (4, 640, 1024, 1024)])
def test_conv_gemm_early_weight_prefetch(ops, B, T, C, co):
    """adp_debug_set(2, 1): weight boxes of the first ring stages are issued before
    griddepcontrol.wait (graph-capture mode of the inference plans).  Same bits expected."""
    from audio_diffusion_pytorch_b200 import _lib
    x = bf(rnd(B, T, C, seed=4))
    w = bf(rnd(co, C, 3, scale=(3 * C) ** -0.5, seed=5))
    bias = rnd(co, seed=6)
    wp = ops.pack_conv(w)
    outs = []
    for flag in (0, 1):
        _lib.lib().adp_debug_set(2, flag)
        try:
            out = torch.empty(B, T, co, dtype=torch.bfloat16, device=DEV)
            for _ in range(3):      # back-to-back launches: the early fetch overlaps a predecessor
                ops.conv_gemm(x, wp, out, c_in=C, n_valid=co, taps=(-1, 0, 1), bias=bias)
            outs.append(out)
        finally:
            _lib.lib().adp_debug_set(2, 0)
    assert torch.equal(outs[0], outs[1])
    ref = F.conv1d(x.float().transpose(1, 2), w.float(), bias, padding=1).transpose(1, 2)
    assert_close(outs[1], ref, 2 ** -7, 1e-2, f"early-W conv3 C{C}")


@pytest.mark.parametrize("B,T,ci,co,f", [(2, 1024, 8, 32, 4), (2, 512, 32, 64, 4),
                                         (1, 256, 128, 256, 2), (2, 96, 64, 128, 2)])
def test_conv_gemm_downsample(ops, B, T, ci, co, f):
    x = bf(rnd(B, T, ci, seed=8))
    w = bf(rnd(co, ci, f, scale=(f * ci) ** -0.5, seed=9))
    bias = rnd(co, seed=10)
    out = torch.empty(B, T // f, co, dtype=torch.bfloat16, device=DEV)
    ops.conv_gemm(x.view(B, T // f, f * ci), ops.pack_conv(w), out, c_in=f * ci, n_valid=co,
                  bias=bias)
    ref = F.conv1d(x.float().transpose(1, 2), w.float(), bias, stride=f).transpose(1, 2)
    assert_close(out, ref, 2 ** -7, 1e-2, f"down ci{ci} f{f}")


@pytest.mark.parametrize("B,T,ci,co,f", [(2, 256, 32, 8, 4), (2, 256, 64, 32, 4),
                                         (1, 128, 256, 128, 2), (2, 200, 128, 64, 2),
                                         (1, 64, 1024, 512, 2)])
def test_conv_gemm_upsample(ops, B, T, ci, co, f):
    x = bf(rnd(B, T, ci, seed=11))
    w = bf(rnd(co, ci, 3, scale=(3 * ci) ** -0.5, seed=12))
    bias = rnd(co, seed=13)
    skip = bf(rnd(B, T * f, co, seed=14))
    gate = rnd(B, co, seed=15)
    groups = 8
    stats = torch.zeros(B, groups, 2, dtype=torch.float64, device=DEV)
    out = torch.empty(B, T * f, co, dtype=torch.bfloat16, device=DEV)
    ops.conv_gemm(x, ops.pack_upsample_conv(w, f), out.view(B, T, f * co), c_in=ci, n_valid=co,
                  up_factor=f, bias=bias, residual=skip.view(B, T, f * co), gate=gate,
                  stats=stats, groups=groups)
    up = F.interpolate(x.float().transpose(1, 2), scale_factor=f, mode="nearest")
    y = F.conv1d(up, w.float(), bias, padding=1).transpose(1, 2)
    ref = skip.float() + gate[:, None, :] * y
    # the phase decomposition sums taps in fp32 and rounds ONCE to bf16: slightly different
    # (more accurate) rounding than conv-ing with the three bf16 taps
    assert_close(out, ref, 2 ** -6, 3e-2, f"upsample ci{ci} co{co} f{f}")
    assert_close(stats, stats_of(out, groups), 1e-4, 1e-2, "upsample stats")


# -------------------------------------------------------------------------- row-wise
@pytest.mark.parametrize("B,T,C", [(2, 1000, 8), (2, 512, 32), (2, 300, 64), (1, 256, 512),
                                   (2, 128, 1024), (2, 100, 192)])
def test_gn_silu_and_stats(ops, B, T, C):
    x = bf(rnd(B, T, C, seed=16) * 1.5 + 0.3)
    gamma, beta = rnd(C, seed=17) * 0.2 + 1.0, rnd(C, seed=18) * 0.2
    groups = 8
    stats = torch.zeros(B, groups, 2, dtype=torch.float64, device=DEV)
    ops.gn_stats(x, stats, groups)
    assert_close(stats, stats_of(x, groups), 1e-4, 1e-2, f"gn_stats C{C}")
    y = torch.empty_like(x)
    ops.gn_silu(x, y, stats, gamma, beta, groups, 1e-5)
    ref = F.silu(F.group_norm(x.float().transpose(1, 2), groups, gamma, beta, 1e-5)).transpose(1, 2)
    assert_close(y, ref, 2 ** -7, 1e-2, f"gn_silu C{C}")


@pytest.mark.parametrize("B,T,C,film", [(2, 1000, 8, True), (2, 512, 32, True), (2, 300, 64, True),
                                        (1, 256, 512, True), (2, 128, 1024, True),
                                        (2, 64, 768, False), (2, 100, 128, False)])
def test_ln_film(ops, B, T, C, film):
    x = bf(rnd(B, T, C, seed=19) * 2.0 + 0.5)
    ss = rnd(B, 2 * C, seed=20) * 0.3 if film else None
    groups = 8
    stats = torch.zeros(B, groups, 2, dtype=torch.float64, device=DEV)
    y = torch.empty_like(x)
    ops.ln_film(x, y, ss, 2 * C if film else 0, stats, groups, 1e-6)
    ref = F.layer_norm(x.float(), (C,), eps=1e-6)
    if film:
        ref = ref * (1 + ss[:, None, :C]) + ss[:, None, C:]
    assert_close(y, ref, 2 ** -7, 1e-2, f"ln_film C{C}")
    assert_close(stats, stats_of(y, groups), 1e-4, 1e-2, f"ln_film stats C{C}")


@pytest.mark.parametrize("B,T,C", [(2, 300, 1024), (2, 257, 512), (1, 1000, 64), (2, 128, 256)])
def test_ln_film_dual(ops, B, T, C):
    """Modulation + attention pre-norm in one pass: y2 must equal LayerNorm of the STORED y."""
    x = bf(rnd(B, T, C, seed=26) * 2.0 + 0.5)
    ss = rnd(B, 2 * C, seed=27) * 0.3
    stats = torch.zeros(B, 8, 2, dtype=torch.float64, device=DEV)
    y, y2 = torch.empty_like(x), torch.empty_like(x)
    ops.ln_film(x, y, ss, 2 * C, stats, 8, 1e-6, y2=y2, eps2=1e-5)
    y_single = torch.empty_like(x)
    ops.ln_film(x, y_single, ss, 2 * C, None, 8, 1e-6)
    assert torch.equal(y, y_single), "dual pass changed the first output"
    ref2 = F.layer_norm(y.float(), (C,), eps=1e-5)
    assert_close(y2, ref2, 2 ** -7, 1e-2, f"ln_film_dual y2 C{C}")
    assert_close(stats, stats_of(y, 8), 1e-4, 1e-2, f"ln_film_dual stats C{C}")


@pytest.mark.parametrize("B,K,N,in_act,out_act", [(8, 1024, 1024, 0, 1), (3, 264, 1024, 0, 1),
                                                  (20, 1024, 520, 2, 0), (1, 64, 40, 1, 2)])
def test_skinny_linear(ops, B, K, N, in_act, out_act):
    x = rnd(B, K, seed=21)
    w = bf(rnd(N, K, scale=K ** -0.5, seed=22))
    bias = rnd(N, seed=23)
    y = torch.empty(B, N, dtype=torch.float32, device=DEV)
    ops.skinny_linear(x, w, bias, y, K, N, in_act, out_act)
    acts = {0: lambda t: t, 1: F.gelu, 2: F.silu}
    ref = acts[out_act](acts[in_act](x) @ w.float().t() + bias)
    assert_close(y, ref, 1e-4, 1e-4, f"skinny B{B} K{K} N{N}")


def test_time_features(ops):
    sigma = torch.rand(5, device=DEV)
    freqs = rnd(128, seed=24)
    out = torch.empty(5, 264, device=DEV)
    ops.time_features(sigma, freqs, out)
    fr = sigma[:, None] * freqs[None] * 2 * math.pi
    ref = torch.cat([sigma[:, None], fr.sin(), fr.cos(), torch.zeros(5, 7, device=DEV)], dim=-1)
    assert_close(out, ref, 1e-5, 2e-5, "time_features")


def test_sampler_step(ops):
    x, v = rnd(2, 2, 1000, seed=25), rnd(2, 2, 1000, seed=26)
    ab = torch.tensor([0.8, 0.6, 0.9, 0.43589], device=DEV)
    out = torch.empty_like(x)
    ops.sampler_step(x, v, ab, out)
    a0, b0, a1, b1 = ab.tolist()
    ref = a1 * (a0 * x - b0 * v) + b1 * (b0 * x + a0 * v)
    assert_close(out, ref, 1e-6, 1e-6, "sampler_step")


# ----------------------------------------------------------------------------- stems
@pytest.mark.parametrize("cx,ca,c0,f,noised", [(2, 0, 8, 1, False), (2, 2, 8, 1, True),
                                               (1, 1, 32, 4, False), (2, 0, 64, 2, True)])
def test_stem_in(ops, cx, ca, c0, f, noised):
    B, T = 2, 1000 * f
    x = rnd(B, cx, T, seed=27)
    app = rnd(B, ca, T, seed=28) if ca else None
    noise = rnd(B, cx, T, seed=29) if noised else None
    alpha = torch.rand(B, device=DEV) if noised else None
    beta = torch.rand(B, device=DEV) if noised else None
    w = rnd(c0, cx + ca, f, scale=((cx + ca) * f) ** -0.5, seed=30)
    bias = rnd(c0, seed=31)
    groups = 8
    stats = torch.zeros(B, groups, 2, dtype=torch.float64, device=DEV)
    out = torch.empty(B, T // f, c0, dtype=torch.bfloat16, device=DEV)
    ops.stem_in(x, w, bias, out, f, append=app, noise=noise, alpha=alpha, beta=beta, stats=stats,
                groups=groups)
    xin = x if not noised else alpha[:, None, None] * x + beta[:, None, None] * noise
    if ca:
        xin = torch.cat([xin, app], dim=1)
    ref = F.conv1d(xin, w, bias, stride=f).transpose(1, 2)
    assert_close(out, ref, 2 ** -7, 1e-2, f"stem_in cx{cx} ca{ca} c0{c0} f{f}")
    assert_close(stats, stats_of(out, groups), 1e-4, 1e-2, "stem_in stats")


@pytest.mark.parametrize("cx,ca,co,c0,f,mode", [(2, 0, 2, 8, 1, "v"), (2, 0, 2, 8, 1, "sample"),
                                                (2, 2, 2, 8, 1, "loss"), (1, 1, 1, 32, 4, "v"),
                                                (2, 0, 2, 8, 1, "cfg")])
def test_stem_out(ops, cx, ca, co, c0, f, mode):
    B, T = 2, 1200
    Bh = 2 * B if mode == "cfg" else B
    h = bf(rnd(Bh, T // f, c0, seed=32))
    x = rnd(B, cx, T, seed=33)
    app = rnd(B, ca, T, seed=34) if ca else None
    w = rnd(co, c0, 3, scale=(3 * c0) ** -0.5, seed=35)
    bias = rnd(co, seed=36)
    gate = rnd(Bh, co, seed=37)
    adapt = cx + ca != co
    wa = rnd(co, cx + ca, seed=38) if adapt else None
    ba = rnd(co, seed=39) if adapt else None
    kw = dict(append=app, w_adapt=wa, b_adapt=ba)
    v = torch.empty(B, co, T, device=DEV)
    noise = alpha = beta = None
    if mode == "loss":
        noise = rnd(B, cx, T, seed=40)
        alpha, beta = torch.rand(B, device=DEV), torch.rand(B, device=DEV)

    def branch(hh, gg, xin_full):
        up = F.interpolate(hh.float().transpose(1, 2), scale_factor=f, mode="nearest")
        y = F.conv1d(up, w, bias, padding=1)
        skip = F.conv1d(xin_full, wa[:, :, None], ba) if adapt else xin_full
        return skip + gg[:, :, None] * y

    xin = x if noise is None else alpha[:, None, None] * x + beta[:, None, None] * noise
    xin_full = torch.cat([xin, app], dim=1) if ca else xin
    if mode == "cfg":
        vc, vm = branch(h[:B], gate[:B], xin_full), branch(h[B:], gate[B:], xin_full)
        ref_v = vm + (vc - vm) * 5.0
    else:
        ref_v = branch(h, gate, xin_full)

    if mode in ("v", "cfg"):
        ops.stem_out(h, x, w, bias, gate, f, v_out=v, cfg_scale=5.0 if mode == "cfg" else None, **kw)
        assert_close(v, ref_v, 1e-4, 1e-4, f"stem_out {mode}")
    elif mode == "sample":
        ab = torch.tensor([0.8, 0.6, 0.9, 0.43589], device=DEV)
        xn = torch.empty_like(x)
        ops.stem_out(h, x, w, bias, gate, f, v_out=v, x_next=xn, ab=ab, **kw)
        a0, b0, a1, b1 = ab.tolist()
        ref = a1 * (a0 * x - b0 * ref_v) + b1 * (b0 * x + a0 * ref_v)
        assert_close(v, ref_v, 1e-4, 1e-4, "stem_out v (sample)")
        assert_close(xn, ref, 1e-4, 1e-4, "stem_out x_next")
    else:
        loss = torch.zeros(1, dtype=torch.float64, device=DEV)
        dv = torch.empty(B, co, T, device=DEV)
        ops.stem_out(h, x, w, bias, gate, f, v_out=v, noise=noise, alpha=alpha, beta=beta,
                     loss_sum=loss, dv=dv, **kw)
        vt = alpha[:, None, None] * noise - beta[:, None, None] * x
        ref_loss = F.mse_loss(ref_v, vt[:, :co])
        assert_close(v, ref_v, 1e-4, 1e-4, "stem_out v (loss)")
        assert_close(loss / ref_v.numel(), ref_loss.double().reshape(1), 1e-4, 1e-6, "loss")
        assert_close(dv, 2 * (ref_v - vt[:, :co]) / ref_v.numel(), 1e-3, 1e-8, "dv")


@pytest.mark.parametrize("C", [8, 32, 64])
@pytest.mark.parametrize("film,res", [(False, False), (True, True), (False, True)])
def test_narrow_conv(ops, film, res, C):
    B, T, groups = 2, 3000, 8
    x = bf(rnd(B, T, C, seed=41) * 1.3 + 0.2)
    stats_in = stats_of(x, groups).contiguous()
    gamma, beta = rnd(C, seed=42) * 0.2 + 1.0, rnd(C, seed=43) * 0.2
    w = rnd(C, C, 3, scale=(3 * C) ** -0.5, seed=44)
    bias = rnd(C, seed=45)
    resid = bf(rnd(B, T, C, seed=46)) if res else None
    ss = rnd(B, 2 * C, seed=47) * 0.3 if film else None
    stats_out = torch.zeros(B, groups, 2, dtype=torch.float64, device=DEV)
    y = torch.empty_like(x)
    ops.narrow_conv(x, y, stats_in, gamma, beta, w, bias, groups, residual=resid, scale_shift=ss,
                    ss_stride=2 * C, stats_out=stats_out)
    if C != 8:      # host-packed bf16 weights must give the identical result
        y_p = torch.empty_like(x)
        ops.narrow_conv(x, y_p, stats_in, gamma, beta, w, bias, groups, residual=resid, scale_shift=ss,
                        ss_stride=2 * C, w_packed=ops.pack_mid_conv(w))
        assert torch.equal(y, y_p), "w_packed path differs from the fp32-weight path"
    a = F.silu(F.group_norm(x.float().transpose(1, 2), groups, gamma, beta, 1e-5))
    ref = F.conv1d(a, w, bias, padding=1).transpose(1, 2)
    if res:
        ref = ref + resid.float()
    if film:
        ref = F.layer_norm(ref, (C,), eps=1e-6) * (1 + ss[:, None, :C]) + ss[:, None, C:]
    # activations AND weights enter the tensor core as bf16 (like every wider level), and the
    # LayerNorm of the film variant rescales the error by 1/std of an 8-channel row
    assert_close(y, ref, 2 ** -7, 3e-2 if film else 1e-2, f"narrow_conv film={film}")
    assert_close(stats_out, stats_of(y, groups), 1e-4, 1e-2, "narrow_conv stats")


# -------------------------------------------------------------------------- attention
@pytest.mark.parametrize("B,H,Tq,Tk", [(2, 8, 256, 256), (1, 2, 128, 128), (2, 8, 1024, 1024),
                                       (2, 4, 200, 200), (2, 8, 512, 64), (1, 2, 300, 8),
                                       (1, 1, 64, 384)])
def test_attention(ops, B, H, Tq, Tk):
    """softmax(q k^T / sqrt(64)) v per head, read straight out of packed projection buffers
    (q | k | v interleaved per row, as the fused qkv GEMM writes them)."""
    mid = H * 64
    self_attn = Tq == Tk
    if self_attn:
        qkv = bf(rnd(B, Tq, 3 * mid, seed=50))
        q, k, v = qkv[..., :mid], qkv[..., mid:2 * mid], qkv[..., 2 * mid:]
    else:
        q = bf(rnd(B, Tq, mid, seed=51))
        kv = bf(rnd(B, Tk, 2 * mid, seed=52))
        k, v = kv[..., :mid], kv[..., mid:]
    o = torch.full((B, Tq, mid), float("nan"), dtype=torch.bfloat16, device=DEV)
    ops.attention(q, k, v, o, H, 64 ** -0.5)

    def heads(t):
        return t.float().reshape(B, -1, H, 64).transpose(1, 2)
    ref = F.scaled_dot_product_attention(heads(q), heads(k), heads(v))
    ref = ref.transpose(1, 2).reshape(B, Tq, mid)
    assert_close(o, ref, 2 ** -6, 2e-2, f"attention B{B} H{H} Tq{Tq} Tk{Tk}")


@pytest.mark.parametrize("B,T,C,co,taps,extras", [
    (8, 256, 1024, 1024, 3, "res+stats"),    # README L7 conv3: one tile per CTA (8 drain warps)
    (8, 1024, 512, 512, 3, "res+stats"),     # README L5 conv3: two tiles per CTA (TMEM double buffer)
    (3, 128, 512, 256, 3, "res+stats"),      # odd number of M tiles
    (2, 200, 1024, 128, 3, "res+stats"),     # ragged T
    (1, 1024, 512, 1536, 1, "bias"),         # qkv projection (1 tap)
    (2, 384, 512, 256, 1, "gate+res"),       # MergeModulate epilogue
])
def test_conv_gemm_long_k(ops, B, T, C, co, taps, extras):
    """Long-K GEMMs of the deep levels with the 128-column N tile, each launched twice into the
    same buffers: against fp32 PyTorch, and the fused GroupNorm statistics of the result."""
    x = bf(rnd(B, T, C, seed=4))
    w = bf(rnd(co, C, taps, scale=(taps * C) ** -0.5, seed=5))
    bias = rnd(co, seed=6)
    res = bf(rnd(B, T, co, seed=7)) if "res" in extras else None
    gate = rnd(B, co, seed=8) if "gate" in extras else None
    groups = 8
    wp = ops.pack_conv(w)
    tp = (-1, 0, 1) if taps == 3 else (0,)
    st = torch.zeros(B, groups, 2, dtype=torch.float64, device=DEV) if "stats" in extras else None
    out = torch.full((B, T, co), float("nan"), dtype=torch.bfloat16, device=DEV)
    for _ in range(2):
        if st is not None:
            st.zero_()
        ops.conv_gemm(x, wp, out, c_in=C, n_valid=co, taps=tp, bias=bias, residual=res, gate=gate,
                      stats=st, groups=groups, block_n=128)
    torch.cuda.synchronize()
    ref = F.conv1d(x.float().transpose(1, 2), w.float(), bias, padding=taps // 2).transpose(1, 2)
    if gate is not None:
        ref = ref * gate[:, None, :]
    if res is not None:
        ref = ref + res.float()
    assert_close(out, ref, 2 ** -7, 1e-2, f"long-K GEMM B{B} T{T} K{C} N{co} taps{taps} {extras}")
    if st is not None:
        assert_close(st, stats_of(out, groups), 1e-4, 1e-2, "long-K GEMM stats")
