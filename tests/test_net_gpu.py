"""Whole-path parity on the GPU: the B200 UNetV0 / VSampler / model wrappers against
 (a) the committed golden vectors (made by oracle/make_golden.py from the UNMODIFIED
     reference files running on the a_unet shim), and
 (b) the CPU oracle port evaluated here on the same seeded inputs,
plus size-independent properties at the README (BASELINE) configuration.

Stated bf16 tolerance (north_star: "stated bf16 tolerance"): storage is bf16 with fp32
accumulation, so every activation carries ~2^-9 relative rounding.  The net output is
v = x + gate*branch with |branch| << |x| at initialisation, so two metrics are bounded:
  * rel-L2 error of v                      <= 1e-4   (10x inside the north star's fp32 rtol)
  * rel-L2 error of the branch (v - skip)  <= BRANCH_TOL = 1.2e-2 = 2x the error of the fp32
    oracle itself evaluated under bf16 autocast on CPU (5.8e-3 on the same metric, stored
    in the golden file as bf16_err_branch).  Measured on B200: 3.0e-3 (tiny), 4.4e-3 (README)."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda"
BRANCH_TOL = 1.2e-2
V_TOL = 1e-4

TINY = dict(in_channels=2, channels=[8, 32, 64], factors=[1, 4, 4], items=[1, 2, 2],
            attentions=[0, 0, 1], attention_heads=2, attention_features=64)
TINY_TEXT = dict(TINY, cross_attentions=[0, 1, 1], use_embedding_cfg=True,
                 embedding_max_length=8, embedding_features=32)
TINY_NOATT = dict(channels=[8, 32, 64], factors=[1, 4, 4], items=[1, 2, 2])


def rel_l2(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def fingerprint(module):
    ps = [p.detach().double() for p in module.parameters()]
    return np.array([sum(float(p.sum()) for p in ps), sum(float(p.abs().sum()) for p in ps),
                     float(sum(p.numel() for p in ps))])


@pytest.fixture(autouse=True)
def inference_mode():
    """This file tests the inference path (training parity: test_train_gpu.py)."""
    with torch.no_grad():
        yield


@pytest.fixture(scope="module")
def adp():
    import audio_diffusion_pytorch_b200 as adp
    return adp


def load(golden_dir, name):
    return {k: v for k, v in np.load(os.path.join(golden_dir, name)).items()}


def t(a):
    return torch.from_numpy(np.asarray(a)).to(DEV)


def check(v, v_ref, skip, what, branch_tol=BRANCH_TOL, v_tol=V_TOL):
    e_v, e_b = rel_l2(v, v_ref), rel_l2(v.cpu() - skip.cpu(), v_ref.cpu() - skip.cpu())
    print(f"{what}: rel-L2(v) {e_v:.3e}  rel-L2(branch) {e_b:.3e}")
    assert e_v <= v_tol, f"{what}: v error {e_v:.3e} > {v_tol}"
    assert e_b <= branch_tol, f"{what}: branch error {e_b:.3e} > {branch_tol}"


def test_unconditional_net_and_sampler_vs_golden(adp, oracle_port, golden_dir):
    g = load(golden_dir, "tiny_unconditional.npz")
    torch.manual_seed(0)
    ref = oracle_port.DiffusionModelPort(**TINY)
    np.testing.assert_allclose(fingerprint(ref), g["param_fingerprint"], rtol=1e-9)
    model = adp.DiffusionModel(net_t=adp.UNetV0, **TINY).to(DEV)
    model.net.load_reference_parameters(ref.net)
    x, sigma = t(g["x"]), t(g["sigma"])
    v_ref = torch.from_numpy(g["v"])
    print("oracle-under-bf16 errors stored in golden:", float(g["bf16_err_net"]),
          float(g["bf16_err_branch"]), float(g["bf16_err_sample5"]))
    for call in range(3):       # eager, graph capture, graph replay must agree
        v = model.net(x, sigma)
        check(v, v_ref, x, f"UNetV0 forward (call {call})")
    noise = t(g["noise"])
    s = model.sample(noise, num_steps=5)
    e = rel_l2(s, torch.from_numpy(g["sample5"]))
    print(f"VSampler 5 steps: rel-L2 {e:.3e}")
    assert e <= 5e-3
    assert torch.equal(noise, t(g["noise"])), "sample() must not mutate its input"
    # the conditioning table of the sampler in several blocks of steps: identical samples
    model.net.cond_table_rows = 4          # 2 steps per block at batch 2
    s_blocks = model.sample(noise, num_steps=5)
    # not bit-equal run to run: GroupNorm statistics are accumulated with atomics
    e_blocks = float((s_blocks.float().cpu() - s.float().cpu()).norm() / s.float().cpu().norm())
    print(f"blocked conditioning table: rel-L2 {e_blocks:.3e}")
    assert e_blocks <= 1e-4, "blocked conditioning table changed the sample"
    model.net.cond_table_rows = 4096


def test_text_cfg_vs_golden(adp, oracle_port, golden_dir):
    g = load(golden_dir, "tiny_text_cfg.npz")
    torch.manual_seed(0)
    ref = oracle_port.DiffusionModelPort(**TINY_TEXT)
    np.testing.assert_allclose(fingerprint(ref), g["param_fingerprint"], rtol=1e-9)
    model = adp.DiffusionModel(net_t=adp.UNetV0, **TINY_TEXT).to(DEV)
    model.net.load_reference_parameters(ref.net)
    x, sigma, emb = t(g["x"]), t(g["sigma"]), t(g["embedding"])
    with torch.no_grad():      # inference path (one 2B-row evaluation, guidance fused in the last kernel)
        v1 = model.net(x, sigma, embedding=emb)
        v5 = model.net(x, sigma, embedding=emb, embedding_scale=5.0)
    check(v1, torch.from_numpy(g["v_scale1"]), x, "text-cond forward, scale 1")
    # guidance extrapolates: v_m + 5 (v_c - v_m) amplifies the error of both passes (|1-s|+|s| = 9x)
    check(v5, torch.from_numpy(g["v_scale5"]), x, "text-cond forward, CFG 5", branch_tol=3e-2,
          v_tol=3e-4)
    s = model.sample(t(g["noise"]), num_steps=3, embedding=emb, embedding_scale=5.0)
    e = rel_l2(s, torch.from_numpy(g["sample3"]))
    print(f"CFG sampler 3 steps: rel-L2 {e:.3e}")
    assert e <= 5e-3


def test_upsampler_and_vocoder_sample_vs_golden(adp, oracle_port, golden_dir):
    g = load(golden_dir, "tiny_upsampler.npz")
    torch.manual_seed(0)
    ref = oracle_port.DiffusionUpsamplerPort(upsample_factor=16, in_channels=2, **TINY_NOATT)
    np.testing.assert_allclose(fingerprint(ref), g["param_fingerprint"], rtol=1e-9)
    model = adp.DiffusionUpsampler(net_t=adp.UNetV0, upsample_factor=16, in_channels=2,
                                   **TINY_NOATT).to(DEV)
    model.net.load_reference_parameters(ref.net)
    s = model.sample(t(g["low"]), num_steps=3, generator=torch.Generator().manual_seed(5))
    e = rel_l2(s, torch.from_numpy(g["sample3"]))
    print(f"DiffusionUpsampler.sample: rel-L2 {e:.3e}")
    assert e <= 5e-3
    e = rel_l2(model.reupsample(t(g["audio"])), torch.from_numpy(g["reupsampled"]))
    assert e <= 1e-5, f"reupsample {e}"

    g = load(golden_dir, "tiny_vocoder.npz")
    kw = dict(mel_n_fft=64, mel_channels=8, mel_sample_rate=48000, mel_normalize_log=True,
              **TINY_NOATT)
    torch.manual_seed(0)
    ref = oracle_port.DiffusionVocoderPort(**kw)
    np.testing.assert_allclose(fingerprint(ref), g["param_fingerprint"], rtol=1e-9)
    model = adp.DiffusionVocoder(net_t=adp.UNetV0, **kw).to(DEV)
    model.net.load_reference_parameters(ref.net)
    model.to_flat.load_state_dict(ref.to_flat.state_dict())
    s = model.sample(t(g["mel"]), num_steps=3, generator=torch.Generator().manual_seed(8))
    e = rel_l2(s, torch.from_numpy(g["sample3"]))
    print(f"DiffusionVocoder.sample: rel-L2 {e:.3e}")
    assert e <= 5e-3


def test_sampler_algebra_generic_net(adp, golden_dir):
    """VSampler around an arbitrary net (not the B200 U-Net): pins the fused step kernel."""
    g = load(golden_dir, "sampler_toy.npz")

    class Toy(torch.nn.Module):
        def forward(self, x, tt, **kw):
            return 0.5 * x * tt.view(-1, 1, 1) + torch.sin(x)

    out = adp.VSampler(net=Toy())(t(g["x"]), num_steps=7)
    np.testing.assert_allclose(out.cpu().numpy(), g["out7"], rtol=1e-4, atol=1e-5)


README = dict(in_channels=2, channels=[8, 32, 64, 128, 256, 512, 512, 1024, 1024],
              factors=[1, 4, 4, 4, 2, 2, 2, 2, 2], items=[1, 2, 2, 2, 2, 2, 2, 4, 4],
              attentions=[0, 0, 0, 0, 0, 1, 1, 1, 1], attention_heads=8, attention_features=64)


def test_readme_config_properties_full_size(adp, oracle_port):
    """BASELINE config at full size ([B,2,2^18]): properties that need no oracle run --
    batch independence, call-to-call reproducibility, finite output -- plus a level-by-level
    oracle comparison on a shorter clip of the SAME network (2^13 samples keeps the CPU
    oracle in seconds; every kernel shape class of the 9-level net is exercised)."""
    torch.manual_seed(0)
    ref = oracle_port.DiffusionModelPort(**README)
    model = adp.DiffusionModel(net_t=adp.UNetV0, **README).to(DEV)
    model.net.load_reference_parameters(ref.net)
    g = torch.Generator().manual_seed(11)
    x_small = torch.randn(2, 2, 2 ** 13, generator=g)
    sig = torch.rand(2, generator=g)
    with torch.no_grad():
        v_ref = ref.net(x_small, sig)
    v = model.net(x_small.to(DEV), sig.to(DEV))
    check(v, v_ref, x_small, "README net, T=2^13 vs CPU oracle")

    x = torch.randn(2, 2, 2 ** 18, generator=g).to(DEV)
    sig2 = torch.tensor([0.3, 0.8], device=DEV)
    v2 = model.net(x, sig2)
    assert torch.isfinite(v2).all()
    v2b = model.net(x, sig2)
    assert rel_l2(v2b - x, v2 - x) < 1e-3, "call-to-call reproducibility"
    v1 = model.net(x[:1], sig2[:1])
    e = rel_l2(v1 - x[:1], v2[:1] - x[:1])
    print(f"batch independence (branch rel-L2): {e:.3e}")
    assert e < 2e-2


# ------------------------------------------------------------------ BASELINE-size parity (r2)
CFG3 = dict(README, cross_attentions=[0, 0, 0, 1, 1, 1, 1, 1, 1], use_embedding_cfg=True,
            embedding_max_length=64, embedding_features=768)


def take_windows(t_, starts, win=1024):
    return torch.stack([t_[..., int(s):int(s) + win] for s in starts], dim=-2)


def test_tiny_sampler_50_steps_vs_golden(adp, oracle_port, golden_dir):
    """The headline metric is a 50-step sample: 50 steps against the reference's own output."""
    g = load(golden_dir, "tiny_sample50.npz")
    torch.manual_seed(0)
    ref = oracle_port.DiffusionModelPort(**TINY)
    np.testing.assert_allclose(fingerprint(ref), g["param_fingerprint"], rtol=1e-9)
    model = adp.DiffusionModel(net_t=adp.UNetV0, **TINY).to(DEV)
    model.net.load_reference_parameters(ref.net)
    noise = torch.randn(2, 2, 4096, generator=torch.Generator().manual_seed(int(g["noise_seed"])))
    s = model.sample(noise.to(DEV), num_steps=50)
    e = rel_l2(s, torch.from_numpy(g["sample50"]))
    print(f"VSampler 50 steps (tiny): rel-L2 {e:.3e}")
    assert e <= 1e-2


def test_readme_full_size_vs_golden(adp, oracle_port, golden_dir):
    """BASELINE configs[1] network at FULL length [1,2,2^18]: forward and a 10-step VSampler run
    against the unmodified reference (16 windows of 1024 samples spread over the clip)."""
    g = load(golden_dir, "readme_full_size.npz")
    torch.manual_seed(0)
    ref = oracle_port.DiffusionModelPort(**README)
    np.testing.assert_allclose(fingerprint(ref), g["param_fingerprint"], rtol=1e-9)
    model = adp.DiffusionModel(net_t=adp.UNetV0, **README).to(DEV)
    model.net.load_reference_parameters(ref.net)
    del ref
    x = torch.randn(1, 2, 2 ** 18, generator=torch.Generator().manual_seed(int(g["x_seed"])))
    starts = g["starts"]
    v = model.net(x.to(DEV), t(g["sigma"])).cpu()
    v_w, x_w, ref_w = take_windows(v, starts), take_windows(x, starts), torch.from_numpy(g["v_windows"])
    check(v_w, ref_w, x_w, "README net, full size 2^18 (windows)")
    s = model.sample(x.to(DEV), num_steps=10).cpu()
    e = rel_l2(take_windows(s, starts), torch.from_numpy(g["sample10_windows"]))
    print(f"README net, full size, VSampler 10 steps (windows): rel-L2 {e:.3e}")
    assert e <= 1e-2


def test_cfg3_readme_scale_vs_golden(adp, oracle_port, golden_dir):
    """BASELINE configs[2]: text-conditional README network (cross-attention at L3..L8, context
    [B,64,768], classifier-free guidance 5.0) against the unmodified reference."""
    g = load(golden_dir, "cfg3_readme_scale.npz")
    torch.manual_seed(0)
    ref = oracle_port.DiffusionModelPort(**CFG3)
    np.testing.assert_allclose(fingerprint(ref), g["param_fingerprint"], rtol=1e-9)
    model = adp.DiffusionModel(net_t=adp.UNetV0, **CFG3).to(DEV)
    model.net.load_reference_parameters(ref.net)
    del ref
    gen = torch.Generator().manual_seed(int(g["seed"]))
    x = torch.randn(1, 2, int(g["length"]), generator=gen)
    emb = torch.randn(1, 64, 768, generator=gen)
    sig = t(g["sigma"])
    with torch.no_grad():
        v1 = model.net(x.to(DEV), sig, embedding=emb.to(DEV))
        v5 = model.net(x.to(DEV), sig, embedding=emb.to(DEV), embedding_scale=5.0)
    check(v1, torch.from_numpy(g["v_scale1"]), x, "cfg3 README scale, guidance 1")
    # guidance extrapolates: v_m + 5 (v_c - v_m) amplifies both passes' error (|1-s| + |s| = 9x on
    # the conditional-unconditional difference); bound 2.5x the single-pass branch tolerance
    check(v5, torch.from_numpy(g["v_scale5"]), x, "cfg3 README scale, CFG 5", branch_tol=3e-2, v_tol=3e-4)
    s = model.sample(x.to(DEV), num_steps=3, embedding=emb.to(DEV), embedding_scale=5.0)
    e = rel_l2(s, torch.from_numpy(g["sample3"]))
    print(f"cfg3 README scale, CFG sampler 3 steps: rel-L2 {e:.3e}")
    assert e <= 5e-3


def test_vinpainter_vs_golden(adp, oracle_port, golden_dir, monkeypatch):
    """VInpainter (reference diffusion.py:306-354): the known region keeps the source, the rest is
    generated; 4 steps x 2 resamples against the unmodified reference.  torch.randn_like is fed the
    draws the reference run consumed (CUDA and CPU generators produce different streams)."""
    g = load(golden_dir, "tiny_inpaint.npz")
    torch.manual_seed(0)
    ref = oracle_port.DiffusionModelPort(**TINY)
    np.testing.assert_allclose(fingerprint(ref), g["param_fingerprint"], rtol=1e-9)
    model = adp.DiffusionModel(net_t=adp.UNetV0, **TINY).to(DEV)
    model.net.load_reference_parameters(ref.net)
    source = torch.randn(2, 2, 4096, generator=torch.Generator().manual_seed(int(g["source_seed"])))
    mask = torch.zeros(2, 2, 4096, dtype=torch.bool)
    for b_, lo, hi in g["mask_spans"]:
        mask[b_, :, lo:hi] = True
    steps, resamples = int(g["num_steps"]), int(g["num_resamples"])
    torch.manual_seed(int(g["rng_seed"]))                 # the reference run's CPU draws, in order
    draws = iter([torch.randn(2, 2, 4096) for _ in range(1 + steps * resamples)])
    monkeypatch.setattr(torch, "randn_like", lambda t_, **kw: next(draws).to(t_))
    inpainter = adp.VInpainter(net=model.net)
    out = inpainter(source.to(DEV), mask.to(DEV), num_steps=steps, num_resamples=resamples)
    e = rel_l2(out, torch.from_numpy(g["out"]))
    print(f"VInpainter 4 steps x 2 resamples: rel-L2 {e:.3e}")
    assert e <= 5e-3
    # the last step ends at sigma = 0: alpha = 1, beta = 0 -> the known region IS the source
    assert rel_l2(out.cpu()[mask], source[mask]) <= 1e-5


def test_autoencoder_decode_vs_golden(adp, oracle_port, golden_dir):
    """DiffusionAE (reference models.py:70-131): the latent of a (toy) encoder injected at depth 2
    by InjectChannelsItem (conv1x1 over cat([x, latent]) + x, here followed by attention);
    decode = 3-step VSampler conditioned on the latent, against the unmodified reference."""
    g = load(golden_dir, "tiny_autoencoder.npz")
    cfg = dict(TINY, inject_depth=2)
    torch.manual_seed(0)
    ref = oracle_port.DiffusionAEPort(encoder=oracle_port.ToyEncoder(), **cfg)
    np.testing.assert_allclose(fingerprint(ref), g["param_fingerprint"], rtol=1e-9)
    torch.manual_seed(0)
    model = adp.DiffusionAE(encoder=oracle_port.ToyEncoder(), net_t=adp.UNetV0, **cfg).to(DEV)
    model.net.load_reference_parameters(ref.net)
    model.encoder.load_state_dict(ref.encoder.state_dict())
    audio = torch.randn(2, 2, 4096, generator=torch.Generator().manual_seed(int(g["audio_seed"])))
    latent = model.encode(audio.to(DEV))
    assert rel_l2(latent, ref.encode(audio) if hasattr(ref, "encode") else ref.encoder(audio)) < 1e-5
    # the reference draws decode()'s noise on latent.device: feed the CPU draw of the golden run
    noise = torch.randn((2, 2, 4096), generator=torch.Generator().manual_seed(int(g["decode_seed"])))
    out = model.sampler(noise.to(DEV), num_steps=3, channels=[None, None, latent])
    e = rel_l2(out, torch.from_numpy(g["decode3"]))
    print(f"DiffusionAE decode (3 steps, latent injected at depth 2): rel-L2 {e:.3e}")
    assert e <= 5e-3
    assert model.decode(latent, num_steps=2).shape == (2, 2, 4096)      # closest_power_2(256 * 16)


TINY_AR = dict(TINY, in_channels=2, length=4096, num_splits=4)


def test_autoregressive_net_and_sampler_vs_golden(adp, oracle_port, golden_dir, monkeypatch):
    """DiffusionAR (reference models.py:227-250): the use_modulation=False net (SkipCat merges,
    sigma as an input channel) and ARVSampler (reference diffusion.py:193-298: start window +
    2 ladder shifts, 4 steps) against the unmodified reference.  torch.randn / randn_like are fed
    the reference run's CPU draws."""
    g = load(golden_dir, "tiny_autoregressive.npz")
    torch.manual_seed(0)
    ref = oracle_port.DiffusionARPort(**TINY_AR)
    np.testing.assert_allclose(fingerprint(ref), g["param_fingerprint"], rtol=1e-9)
    model = adp.DiffusionAR(net_t=adp.UNetV0, **TINY_AR).to(DEV)
    model.net.load_reference_parameters(ref.net)
    gen = torch.Generator().manual_seed(int(g["input_seed"]))
    audio = torch.randn(2, 2, 4096, generator=gen)
    chan = torch.cat([audio, torch.rand(2, 1, 4096, generator=gen)], dim=1)
    for _ in range(3):                       # eager, capture, replay
        v = model.net(chan.to(DEV))
    e = rel_l2(v, torch.from_numpy(g["v"]))
    print(f"use_modulation=False net forward: rel-L2 {e:.3e}")
    assert e <= 5e-3
    # draws of the reference run, in order: randn(start window), randn_like(start), one randn per shift
    torch.manual_seed(int(g["sample_seed"]))
    draws = iter([torch.randn(2, 2, 4096), torch.randn(2, 2, 4096)] + [torch.randn(2, 2, 1024) for _ in range(6)])
    monkeypatch.setattr(torch, "randn", lambda *a, **kw: next(draws).to(kw.get("device", "cpu")))
    monkeypatch.setattr(torch, "randn_like", lambda t_, **kw: next(draws).to(t_))
    out = model.sample(num_items=2, num_chunks=6, num_steps=4)
    monkeypatch.undo()
    assert out.shape == (2, 2, 6144)
    e = rel_l2(out, torch.from_numpy(g["sample"]))
    print(f"ARVSampler 6 chunks x 4 steps: rel-L2 {e:.3e}")
    assert e <= 1e-2


def close(got, want, what, rtol=1e-3, atol=1e-4):
    """The fp32 criterion of the north star: |got - want| <= atol + rtol * |want| elementwise."""
    got, want = got.detach().float().cpu(), want.detach().float().cpu()
    err = (got - want).abs()
    worst = float((err - rtol * want.abs()).max())
    print(f"{what}: max abs err {float(err.max()):.3e}, rel-L2 {rel_l2(got, want):.3e}, "
          f"max(err - rtol*|ref|) {worst:.3e} (atol {atol})")
    torch.testing.assert_close(got, want, rtol=rtol, atol=atol)


def test_fp32_verification_mode(adp, oracle_port, golden_dir):
    """B200UNet.verify_fp32: the SAME launch program, weight packs and folds as the bf16 path with
    fp32 storage and arithmetic (csrc/verify_f32.cu) meets rtol 1e-3 / atol 1e-4 against the
    unmodified reference's golden vectors -- net, 5-step sampler, cross-attention + guidance 5.0,
    the SkipCat (use_modulation=False) net -- and against the oracle on the 9-level README net."""
    g = load(golden_dir, "tiny_unconditional.npz")
    torch.manual_seed(0)
    ref = oracle_port.DiffusionModelPort(**TINY)
    model = adp.DiffusionModel(net_t=adp.UNetV0, **TINY).to(DEV)
    model.net.load_reference_parameters(ref.net)
    x, sigma = t(g["x"]), t(g["sigma"])
    v_bf16 = model.net(x, sigma).clone()
    model.net.verify_fp32 = True
    for call in range(3):                   # eager, capture, replay
        v = model.net(x, sigma)
    close(v, torch.from_numpy(g["v"]), "fp32 mode: tiny net forward")
    close(v - x, torch.from_numpy(g["v"]) - x.cpu(), "fp32 mode: tiny net branch (v - skip)")
    close(model.sample(t(g["noise"]), num_steps=5), torch.from_numpy(g["sample5"]), "fp32 mode: VSampler 5 steps")
    model.net.verify_fp32 = False           # and back: the tensor-core path is rebuilt
    assert rel_l2(model.net(x, sigma), v_bf16) <= 1e-4

    g = load(golden_dir, "tiny_text_cfg.npz")
    torch.manual_seed(0)
    ref = oracle_port.DiffusionModelPort(**TINY_TEXT)
    model = adp.DiffusionModel(net_t=adp.UNetV0, **TINY_TEXT).to(DEV)
    model.net.load_reference_parameters(ref.net)
    model.net.verify_fp32 = True
    x, sigma, emb = t(g["x"]), t(g["sigma"]), t(g["embedding"])
    close(model.net(x, sigma, embedding=emb), torch.from_numpy(g["v_scale1"]), "fp32 mode: text-cond, scale 1")
    close(model.net(x, sigma, embedding=emb, embedding_scale=5.0), torch.from_numpy(g["v_scale5"]),
          "fp32 mode: text-cond, CFG 5")
    close(model.sample(t(g["noise"]), num_steps=3, embedding=emb, embedding_scale=5.0),
          torch.from_numpy(g["sample3"]), "fp32 mode: CFG sampler 3 steps")

    g = load(golden_dir, "tiny_autoregressive.npz")
    torch.manual_seed(0)
    ref = oracle_port.DiffusionARPort(**TINY_AR)
    model = adp.DiffusionAR(net_t=adp.UNetV0, **TINY_AR).to(DEV)
    model.net.load_reference_parameters(ref.net)
    model.net.verify_fp32 = True
    gen = torch.Generator().manual_seed(int(g["input_seed"]))
    audio = torch.randn(2, 2, 4096, generator=gen)
    chan = torch.cat([audio, torch.rand(2, 1, 4096, generator=gen)], dim=1)
    close(model.net(chan.to(DEV)), torch.from_numpy(g["v"]), "fp32 mode: SkipCat net")

    torch.manual_seed(0)
    ref = oracle_port.DiffusionModelPort(**README)
    model = adp.DiffusionModel(net_t=adp.UNetV0, **README).to(DEV)
    model.net.load_reference_parameters(ref.net)
    model.net.verify_fp32 = True
    gen = torch.Generator().manual_seed(11)
    x_small = torch.randn(2, 2, 2 ** 13, generator=gen)
    sig = torch.rand(2, generator=gen)
    v_ref = ref.net(x_small, sig)
    v = model.net(x_small.to(DEV), sig.to(DEV))
    close(v, v_ref, "fp32 mode: README 9-level net (2^13 clip)")
    close(v.cpu() - x_small, v_ref - x_small, "fp32 mode: README net branch")


def test_fp32_verification_mode_model_wrappers(adp, oracle_port, golden_dir):
    """verify_fp32 through the model wrappers: appended channels (Upsampler, Vocoder) and the
    injected latent (DiffusionAE) take the fp32 stem / GEMM kernels; 3-step samples against the
    unmodified reference's vectors at rtol 1e-3 / atol 1e-4."""
    g = load(golden_dir, "tiny_upsampler.npz")
    torch.manual_seed(0)
    ref = oracle_port.DiffusionUpsamplerPort(upsample_factor=16, in_channels=2, **TINY_NOATT)
    model = adp.DiffusionUpsampler(net_t=adp.UNetV0, upsample_factor=16, in_channels=2, **TINY_NOATT).to(DEV)
    model.net.load_reference_parameters(ref.net)
    model.net.verify_fp32 = True
    s = model.sample(t(g["low"]), num_steps=3, generator=torch.Generator().manual_seed(5))
    close(s, torch.from_numpy(g["sample3"]), "fp32 mode: DiffusionUpsampler.sample")

    g = load(golden_dir, "tiny_vocoder.npz")
    kw = dict(mel_n_fft=64, mel_channels=8, mel_sample_rate=48000, mel_normalize_log=True, **TINY_NOATT)
    torch.manual_seed(0)
    ref = oracle_port.DiffusionVocoderPort(**kw)
    model = adp.DiffusionVocoder(net_t=adp.UNetV0, **kw).to(DEV)
    model.net.load_reference_parameters(ref.net)
    model.to_flat.load_state_dict(ref.to_flat.state_dict())
    model.net.verify_fp32 = True
    s = model.sample(t(g["mel"]), num_steps=3, generator=torch.Generator().manual_seed(8))
    close(s, torch.from_numpy(g["sample3"]), "fp32 mode: DiffusionVocoder.sample")

    g = load(golden_dir, "tiny_autoencoder.npz")
    cfg = dict(TINY, inject_depth=2)
    torch.manual_seed(0)
    ref = oracle_port.DiffusionAEPort(encoder=oracle_port.ToyEncoder(), **cfg)
    torch.manual_seed(0)
    model = adp.DiffusionAE(encoder=oracle_port.ToyEncoder(), net_t=adp.UNetV0, **cfg).to(DEV)
    model.net.load_reference_parameters(ref.net)
    model.encoder.load_state_dict(ref.encoder.state_dict())
    model.net.verify_fp32 = True
    audio = torch.randn(2, 2, 4096, generator=torch.Generator().manual_seed(int(g["audio_seed"])))
    latent = model.encode(audio.to(DEV))
    noise = torch.randn((2, 2, 4096), generator=torch.Generator().manual_seed(int(g["decode_seed"])))
    out = model.sampler(noise.to(DEV), num_steps=3, channels=[None, None, latent])
    close(out, torch.from_numpy(g["decode3"]), "fp32 mode: DiffusionAE decode")
