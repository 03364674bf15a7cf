"""UNetV0 on B200: the reference's `net_t` plugin slot (reference components.py:34-105),
rebuilt over the sm_100a kernels of libadp_b200.so.

`UNetV0(dim=1, in_channels=..., channels=[...], ...)` takes the reference's kwargs verbatim
and returns an nn.Module with the reference's call signature

    net(x[B,Cin,T], time[B], *, features=None, embedding=None, embedding_scale=1.0,
        embedding_mask_proba=0.0, channels=None[, append_channels]) -> [B,Cout,T]

Parameters keep PyTorch shapes (Conv1d [co,ci,k], Linear [out,in]) and are registered in
the same order as the a_unet module tree, so `load_reference_parameters` copies a reference
model's weights positionally.  The forward pass is a flat *program*: a list of kernel
launches over pre-allocated channels-last bf16 buffers, captured into one CUDA graph per
(batch, length) shape; nothing in it falls back to PyTorch ops or to the CPU.
"""
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F
from torch import Tensor, nn

from . import _lib, ops


def exists(v) -> bool:
    return v is not None


def default(v, d):
    return v if exists(v) else d


# ----------------------------------------------------------------------------- parameters
class ResnetParams(nn.Module):
    """a_unet ResnetBlock: (GroupNorm, SiLU, Conv1d k3) x 2 + identity shortcut."""

    def __init__(self, channels: int, groups: int):
        super().__init__()
        self.gn1 = nn.GroupNorm(groups, channels)
        self.conv1 = nn.Conv1d(channels, channels, 3, padding=1)
        self.gn2 = nn.GroupNorm(groups, channels)
        self.conv2 = nn.Conv1d(channels, channels, 3, padding=1)


class ModulationParams(nn.Module):
    """a_unet Modulation: Linear(SiLU(features)) -> (scale, shift); LayerNorm has no params."""

    def __init__(self, channels: int, features: int):
        super().__init__()
        self.proj = nn.Linear(features, 2 * channels)


class AttentionParams(nn.Module):
    """a_unet Attention: norm, norm_context, to_q, to_kv, to_out (no biases)."""

    def __init__(self, channels: int, head_features: int, heads: int,
                 context_features: Optional[int] = None):
        super().__init__()
        mid = head_features * heads
        ctx = default(context_features, channels)
        self.norm = nn.LayerNorm(channels)
        self.norm_context = nn.LayerNorm(ctx)
        self.to_q = nn.Linear(channels, mid, bias=False)
        self.to_kv = nn.Linear(ctx, 2 * mid, bias=False)
        self.to_out = nn.Linear(mid, channels, bias=False)


class ItemParams(nn.Module):
    """One repetition of [ResnetItem, ModulationItem, InjectChannelsItem?, AttentionItem?,
    CrossAttentionItem?] (reference components.py:89-95)."""

    def __init__(self, channels: int, groups: int, features: int, att: bool, cross: bool,
                 head_features: Optional[int], heads: Optional[int],
                 embedding_features: Optional[int], context: int = 0, modulation: bool = True):
        super().__init__()
        self.resnet = ResnetParams(channels, groups)
        self.modulation = ModulationParams(channels, features) if modulation else None
        # a_unet InjectChannelsItem: Conv1d(C + ctx -> C, k=1) over cat([x, channels[depth]]), + x
        self.inject = nn.Conv1d(channels + context, channels, 1) if context > 0 else None
        self.attention = AttentionParams(channels, head_features, heads) if att else None
        self.cross = (AttentionParams(channels, head_features, heads, embedding_features)
                      if cross else None)


class LevelParams(nn.Module):
    """a_unet Block: registration order = skip_adapter, (down, items, inner, items_up, up), merge."""

    def __init__(self, in_ch: int, out_ch: int, ch: int, factor: int, n_items: int, inner,
                 **item_kw):
        super().__init__()
        self.adapter = nn.Conv1d(in_ch, out_ch, 1) if in_ch != out_ch else None
        self.down = nn.Conv1d(in_ch, ch, factor, stride=factor)
        self.items_down = nn.ModuleList([ItemParams(ch, **item_kw) for _ in range(n_items)])
        self.inner = inner
        self.items_up = nn.ModuleList([ItemParams(ch, **item_kw) for _ in range(n_items)])
        self.up = nn.Conv1d(ch, out_ch, 3, padding=1)
        # a_unet SkipModulate (MergeModulate: Linear(features -> out)) or, with use_modulation=False,
        # SkipCat (MergeCat: Conv1d(2*out -> out, k=1) over cat([skip * 2^-0.5, y]))
        self.merge = (nn.Linear(item_kw["features"], out_ch) if item_kw.get("modulation", True)
                      else nn.Conv1d(2 * out_ch, out_ch, 1))
        self.in_ch, self.out_ch, self.ch, self.factor = in_ch, out_ch, ch, factor


class TimeParams(nn.Module):
    """a_unet TimeConditioningPlugin: NumberEmbedder + (Linear, GELU) applied twice (shared)."""

    def __init__(self, features: int, dim: int = 256):
        super().__init__()
        self.weights = nn.Parameter(torch.randn(dim // 2))
        self.to_out = nn.Linear(dim + 1, features)
        self.mlp = nn.Linear(features, features)


# -------------------------------------------------------------------------------- program
class _Pool:
    """Reuses activation buffers whose value is dead (better L2 residency than fresh ones)."""

    def __init__(self, device, reuse: bool, dtype=torch.bfloat16):
        self.device, self.reuse, self.dtype = device, reuse, dtype
        self.free: Dict[Tuple, List[Tensor]] = {}
        self.total_bytes = 0

    def get(self, *shape, dtype=None) -> Tensor:
        dtype = self.dtype if dtype is None else dtype
        key = (tuple(shape), dtype)
        lst = self.free.get(key)
        if self.reuse and lst:
            return lst.pop()
        t = torch.empty(*shape, dtype=dtype, device=self.device)
        self.total_bytes += t.numel() * t.element_size()
        return t

    def put(self, t: Optional[Tensor]) -> None:
        if t is not None and self.reuse:
            self.free.setdefault((tuple(t.shape), t.dtype), []).append(t)


class _Plan:
    """Everything tied to one input shape: static I/O buffers, workspaces, the launch list and
    (after warm-up) its CUDA graph."""

    def __init__(self):
        self.prog: List[Callable[[], None]] = []
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self.n_launches = 0
        self.n_kernels = 0
        self.runs = 0

    def add(self, fn: Callable[[], None]) -> None:
        self.prog.append(fn)
        self.n_launches += 1

    def run_eager(self) -> None:
        for fn in self.prog:
            fn()


class B200UNet(nn.Module):
    """See module docstring.  Reference parity notes per block are in include/adp_b200.h."""

    GN_EPS = 1e-5      # nn.GroupNorm default (a_unet ConvBlock)
    ATT_LN_EPS = 1e-5  # nn.LayerNorm default (a_unet Attention norms)
    MOD_LN_EPS = 1e-6  # a_unet Modulation LayerNorm

    def __init__(self, dim: int, in_channels: int, channels: Sequence[int],
                 factors: Sequence[int], items: Sequence[int],
                 attentions: Optional[Sequence[int]] = None,
                 cross_attentions: Optional[Sequence[int]] = None,
                 context_channels: Optional[Sequence[int]] = None,
                 attention_features: Optional[int] = None,
                 attention_heads: Optional[int] = None,
                 embedding_features: Optional[int] = None, resnet_groups: int = 8,
                 use_modulation: bool = True, modulation_features: int = 1024,
                 embedding_max_length: Optional[int] = None,
                 use_time_conditioning: bool = True, use_embedding_cfg: bool = False,
                 use_text_conditioning: bool = False, out_channels: Optional[int] = None,
                 append_channels: int = 0):
        super().__init__()
        n = len(channels)
        attentions = default(attentions, [0] * n)
        cross_attentions = default(cross_attentions, [0] * n)
        context_channels = default(context_channels, [0] * n)
        xs = (channels, factors, items, attentions, cross_attentions, context_channels)
        assert all(len(x) == n for x in xs)                       # reference components.py:61
        assert dim == 1, "the B200 path implements the 1-D (waveform) U-Net"
        if use_embedding_cfg:                                     # components.py:66-68
            assert exists(embedding_max_length), "use_embedding_cfg requires embedding_max_length"
        if use_time_conditioning:                                 # components.py:75
            assert use_modulation, "use_time_conditioning requires use_modulation=True"
        if use_text_conditioning:
            raise NotImplementedError(
                "use_text_conditioning builds a T5 encoder (a_unet TextConditioningPlugin); pass "
                "precomputed `embedding=` with use_text_conditioning=False (SURVEY.md 3.4)")
        for c, ctx in zip(channels, context_channels):
            assert ctx == 0 or c >= 16, "InjectChannelsItem is built for levels with >= 16 channels"
        if any(attentions) or any(cross_attentions):
            assert exists(attention_features) and exists(attention_heads), \
                "AttentionItem requires attention_features and attention_heads"
            assert attention_features == 64, "the tcgen05 attention kernel is built for head dim 64"
        if any(cross_attentions):
            assert exists(embedding_features), "CrossAttentionItem requires embedding_features"

        self.x_channels = in_channels - append_channels   # channels of `x` (rest is appended)
        self.append_channels = append_channels
        self.in_channels, self.out_channels = in_channels, default(out_channels, in_channels)
        self.channels, self.factors, self.items = list(channels), list(factors), list(items)
        self.attentions, self.cross_attentions = list(attentions), list(cross_attentions)
        self.context_channels = list(context_channels)
        self.groups, self.features = resnet_groups, modulation_features
        self.heads, self.head_features = attention_heads, attention_features
        self.embedding_features = embedding_features
        self.use_time_conditioning, self.use_embedding_cfg = use_time_conditioning, use_embedding_cfg
        self.use_modulation = use_modulation
        for c in self.channels:
            assert c % resnet_groups == 0 and c % 8 == 0, "channels must be multiples of 8 and groups"
        assert self.out_channels <= 4 and self.in_channels <= 8, "stem kernels: in<=8, out<=4 channels"

        # registration order mirrors a_unet: time plugin, cfg plugin, then the recursive blocks
        self.time = TimeParams(modulation_features) if use_time_conditioning else None
        self.fixed_embedding = (nn.Embedding(embedding_max_length, embedding_features)
                                if use_embedding_cfg else None)

        def build(i: int):
            if i == n:
                return None
            in_ch = in_channels if i == 0 else channels[i - 1]
            out_ch = self.out_channels if i == 0 else in_ch
            return LevelParams(in_ch, out_ch, channels[i], factors[i], items[i], build(i + 1),
                               groups=resnet_groups, features=modulation_features,
                               att=bool(attentions[i]), cross=bool(cross_attentions[i]),
                               head_features=attention_features, heads=attention_heads,
                               embedding_features=embedding_features, context=context_channels[i],
                               modulation=use_modulation)

        self.net = build(0)
        self._plans: Dict[Tuple, _Plan] = {}
        self._packed = None
        self._packed_version = None
        self._fingerprint = None
        self._storage_sig = None
        self._repack_graph = None
        self.use_cuda_graph = True
        # C = 32 / 64 ConvBlocks as ONE fused kernel (GroupNorm+SiLU -> conv3 -> +res -> LN/FiLM ->
        # statistics, csrc/mid_conv.cu) instead of three: those levels are HBM-bound
        self.fuse_thin_levels = True
        self.cond_table_rows = 4096    # sampler: rows (steps x batch) of conditioning per pass
        self.max_table_steps = 4096    # iterations per conditioning block (alpha/beta table rows)
        self.steps_per_graph = 10      # sampling steps captured back to back in one CUDA graph
        self._verify_fp32 = False

    @property
    def verify_fp32(self) -> bool:
        """fp32 VERIFICATION MODE (inference and sampling): the same launch program, packed-weight
        layouts and folds, with fp32 storage and fp32 arithmetic on the simple kernels of
        csrc/verify_f32.cu (the fused thin-level kernels are replaced by their unfused
        composition).  For checking the program against the reference at rtol 1e-3 / atol 1e-4;
        ~100x slower than the tensor-core path.  Switching drops every plan and pack."""
        return self._verify_fp32

    @verify_fp32.setter
    def verify_fp32(self, on: bool) -> None:
        if bool(on) != self._verify_fp32:
            self._verify_fp32 = bool(on)
            self.invalidate()

    def _act_dtype(self):
        return torch.float32 if self._verify_fp32 else torch.bfloat16

    # ------------------------------------------------------------------ weights
    def levels(self) -> List[LevelParams]:
        out, lvl = [], self.net
        while lvl is not None:
            out.append(lvl)
            lvl = lvl.inner
        return out

    @torch.no_grad()
    def load_reference_parameters(self, reference_net: nn.Module) -> None:
        """Positional copy from a reference UNetV0 (same kwargs): both trees register
        parameters in a_unet order, so shapes must line up one to one."""
        src, dst = list(reference_net.parameters()), list(self.parameters())
        assert len(src) == len(dst), f"parameter count {len(src)} != {len(dst)}"
        for s, d in zip(src, dst):
            assert s.shape == d.shape, f"shape mismatch {tuple(s.shape)} vs {tuple(d.shape)}"
            d.copy_(s)

    @torch.no_grad()
    def load_reference_state_dict(self, state_dict, prefix: str = "") -> None:
        """Loads the U-Net part of a reference checkpoint (`torch.save(model.state_dict())` of a
        reference model built with the same kwargs) without depending on a_unet's module NAMES:
        the keys under `prefix` are taken in checkpoint order, which is a_unet's registration
        order = this tree's parameter order, except that the time MLP's Linear is listed twice
        (a_unet repeats one module object inside a Sequential; both entries hold the same tensor).
        Shapes are checked entry by entry."""
        entries = [(k, v) for k, v in state_dict.items() if k.startswith(prefix)]
        mine = []
        for name, p in self.named_parameters():
            mine.append((name, p))
            if name == "time.mlp.bias":
                mine += mine[-2:]
        assert len(entries) == len(mine), \
            f"checkpoint has {len(entries)} tensors under '{prefix}', this net expects {len(mine)}"
        seen = {}
        for (key, src), (name, dst) in zip(entries, mine):
            assert tuple(src.shape) == tuple(dst.shape), \
                f"{key}: shape {tuple(src.shape)} does not match {name} {tuple(dst.shape)}"
            if name in seen:
                assert torch.equal(src, seen[name]), f"{key}: repeated module entries differ"
                continue
            seen[name] = src
            dst.copy_(src)

    def _version(self) -> int:
        return sum(p._version for p in self.parameters())

    def _storage_signature(self):
        return tuple((p.data_ptr(), p.dtype) for p in self.parameters())

    def invalidate(self) -> None:
        """Drops every packed weight, plan and captured graph.  Needed after a parameter was
        re-pointed (`p.data = ...`, `.to()`, `.half()`, `load_state_dict(assign=True)`); in-place
        updates through the Parameter (optimizers, `load_state_dict`, `copy_`) are tracked by the
        version counters and refresh the packs in place instead."""
        self._plans.clear()
        self._packed = None
        self._packed_version = None
        self._fingerprint = None
        self._repack_graph = None

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        if hasattr(self, "_plans"):
            self.invalidate()
        return out

    @torch.no_grad()
    def _check_untracked_updates(self) -> None:
        """`p.data.add_()` / `.data.copy_()` style updates (EMA wrappers, manual init, weight
        clipping) bump no version counter.  Inference entry points therefore compare a cheap device
        fingerprint of all parameters (one multi-tensor norm + one small device->host read per
        call, outside the step loop) and re-pack when it moved."""
        ps = [p for p in self.parameters()]
        if not ps or not ps[0].is_cuda:
            return
        fp = torch.stack(torch._foreach_norm(ps)).double().cpu()
        if self._fingerprint is not None and not torch.equal(fp, self._fingerprint):
            self._packed_version = None          # force an in-place re-pack
            for plan in self._plans.values():
                if hasattr(plan, "version"):
                    plan.version = None
        self._fingerprint = fp

    @torch.no_grad()
    def packed(self):
        """Kernel-layout copies of the weights (bf16 GEMM operands, folded LayerNorm affines,
        one concatenated conditioning projection).  Rebuilt when a parameter changes."""
        sig = self._storage_signature()
        if getattr(self, "_storage_sig", None) != sig:   # a parameter was re-pointed: addresses
            if getattr(self, "_storage_sig", None) is not None:   # baked into plans are stale
                self.invalidate()
            self._storage_sig = sig
        v = self._version()
        if self._packed is not None and self._packed_version == v:
            return self._packed
        if self._packed is not None:
            # weights changed (optimizer step): refresh the SAME tensors in place, so captured
            # CUDA graphs and plans that hold their addresses stay valid
            self._repack()
            self._packed_version = v
            return self._packed
        self._packed, self._packed_version = self._compute_packed(), v
        return self._packed

    @torch.no_grad()
    def _repack(self) -> None:
        """In-place refresh of every packed weight.  The re-layout is ~500 small permute / cast /
        fold launches whose HOST cost (12 ms per training step, profiles/r2_train_profile_start.txt)
        dwarfed their device time: sources (the parameters) and destinations (the packs) have
        fixed addresses, so the whole sequence is captured once into a CUDA graph and replayed."""
        if not (self.use_cuda_graph and self.net.down.weight.is_cuda):
            _copy_tree(self._packed, self._compute_packed())
            return
        if self._repack_graph is None:
            _copy_tree(self._packed, self._compute_packed())       # eager once: allocator warm
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                _copy_tree(self._packed, self._compute_packed())
            self._repack_graph = g
        else:
            self._repack_graph.replay()

    @torch.no_grad()
    def _compute_packed(self):
        with ops.pack_dtype(self._act_dtype()):
            return self._compute_packed_impl()

    def _compute_packed_impl(self):
        P: Dict = {}
        pd = self._act_dtype()
        f32 = lambda t: t.detach().float().contiguous()  # noqa: E731
        cond_w, cond_b, off = [], [], 0

        def add_cond(lin: nn.Linear) -> int:
            nonlocal off
            n_out = lin.weight.shape[0]
            pad = ops.round_up(n_out, 8)
            w = torch.zeros(pad, lin.weight.shape[1], device=lin.weight.device)
            b = torch.zeros(pad, device=lin.weight.device)
            w[:n_out], b[:n_out] = lin.weight.detach().float(), lin.bias.detach().float()
            cond_w.append(w)
            cond_b.append(b)
            start, off = off, off + pad
            return start

        def pack_att(a: AttentionParams, self_attn: bool) -> Dict:
            wq = a.to_q.weight.detach().float()
            wkv = a.to_kv.weight.detach().float()
            g1, b1 = a.norm.weight.detach().float(), a.norm.bias.detach().float()
            g2, b2 = a.norm_context.weight.detach().float(), a.norm_context.bias.detach().float()
            d: Dict = {"w_out": ops.pack_linear(a.to_out.weight.detach())}
            # LayerNorm affine folded into the projection: W (xhat*g + b) = (W*g) xhat + W b
            wq_f, bq = wq * g1[None, :], wq @ b1
            wkv_f, bkv = wkv * g2[None, :], wkv @ b2
            if self_attn:
                d["w_qkv"] = ops.pack_linear(torch.cat([wq_f, wkv_f], 0))
                d["b_qkv"] = torch.cat([bq, bkv]).contiguous()
            else:
                d["w_q"], d["b_q"] = ops.pack_linear(wq_f), bq.contiguous()
                d["w_kv"], d["b_kv"] = ops.pack_linear(wkv_f), bkv.contiguous()
            return d

        def pack_item(it: ItemParams, narrow: bool) -> Dict:
            r = it.resnet
            d: Dict = {"gn1": (f32(r.gn1.weight), f32(r.gn1.bias)),
                       "gn2": (f32(r.gn2.weight), f32(r.gn2.bias)),
                       "b1": f32(r.conv1.bias), "b2": f32(r.conv2.bias)}
            if it.modulation is not None:
                d["ss_off"] = add_cond(it.modulation.proj)
            if narrow:
                d["w1"], d["w2"] = f32(r.conv1.weight), f32(r.conv2.weight)
            else:
                d["w1"], d["w2"] = ops.pack_conv(r.conv1.weight.detach()), ops.pack_conv(r.conv2.weight.detach())
                if r.conv1.weight.shape[0] in (32, 64):    # thin levels: fused ConvBlock kernel
                    d["w1_raw"], d["w2_raw"] = f32(r.conv1.weight), f32(r.conv2.weight)
                    d["w1_mid"], d["w2_mid"] = ops.pack_mid_conv(r.conv1.weight), ops.pack_mid_conv(r.conv2.weight)
            if it.inject is not None:
                C_ = it.inject.weight.shape[0]
                wi = it.inject.weight.detach().float()[:, :, 0]
                ctx = wi.shape[1] - C_
                wc = torch.zeros(C_, ops.round_up(ctx, 16), device=wi.device)
                wc[:, :ctx] = wi[:, C_:]
                d["inj"] = {"w_x": ops.pack_linear(wi[:, :C_]), "w_c": ops.pack_linear(wc),
                            "b": f32(it.inject.bias)}
            if it.attention is not None:
                d["att"] = pack_att(it.attention, True)
            if it.cross is not None:
                d["cross"] = pack_att(it.cross, False)
            return d

        P["levels"] = []
        for i, lvl in enumerate(self.levels()):
            narrow = lvl.ch == 8 and not self._verify_fp32
            L: Dict = {"down_b": f32(lvl.down.bias), "up_b": f32(lvl.up.bias)}
            if i == 0:
                L["down_w"], L["up_w"] = f32(lvl.down.weight), f32(lvl.up.weight)
                if lvl.adapter is not None:
                    L["adapt_w"] = f32(lvl.adapter.weight[:, :, 0])
                    L["adapt_b"] = f32(lvl.adapter.bias)
            else:
                L["down_w"] = ops.pack_conv(lvl.down.weight.detach())
                L["up_w"] = (ops.pack_upsample_conv(lvl.up.weight.detach(), lvl.factor)
                             if lvl.factor > 1 else ops.pack_conv(lvl.up.weight.detach()))
            L["items_down"] = [pack_item(it, narrow) for it in lvl.items_down]
            L["items_up"] = [pack_item(it, narrow) for it in lvl.items_up]
            if self.use_modulation:
                L["gate_off"] = add_cond(lvl.merge)
            else:
                # SkipCat: out = Wc1 (skip * s) + Wc2 y + bc,  W = [Wc1 | Wc2]
                s_ = 2 ** -0.5
                wm = lvl.merge.weight.detach().float()[:, :, 0]
                co = wm.shape[0]
                wc1, wc2, bc = wm[:, :co] * s_, wm[:, co:], lvl.merge.bias.detach().float()
                if i > 0:
                    # the tensor-core GEMM needs K >= 16: an 8-channel level output is viewed as
                    # [B, T/2, 16] (two positions per row) against block-diagonal weights
                    rr = max(1, 16 // co)
                    L["cat_w1"] = ops.pack_linear(torch.block_diag(*[wc1] * rr))
                    L["cat_w2"] = ops.pack_linear(torch.block_diag(*[wc2] * rr))
                    L["cat_b"] = bc.repeat(rr).contiguous()
                else:
                    # level 0 runs in the stem kernel (skip adapter + upsample conv + merge): fold the
                    # 1x1 merge conv into both branches.  v = (Wc1 W_ad) x + Wc1 b_ad + conv'(h) + b',
                    # conv' = Wc2 o W_up, b' = Wc2 b_up + bc; the kernel's gate is 1.
                    w_up = lvl.up.weight.detach().float()
                    L["up_w"] = torch.einsum("om,mck->ock", wc2, w_up).contiguous()
                    L["up_b"] = (wc2 @ lvl.up.bias.detach().float() + bc).contiguous()
                    if lvl.adapter is not None:
                        L["adapt_w"] = (wc1 @ lvl.adapter.weight.detach().float()[:, :, 0]).contiguous()
                        L["adapt_b"] = (wc1 @ lvl.adapter.bias.detach().float()).contiguous()
                    else:
                        L["adapt_w"], L["adapt_b"] = wc1.contiguous(), torch.zeros_like(bc)
            P["levels"].append(L)
        n_tot = off
        if cond_w:
            w_all = torch.cat(cond_w, 0)
            n_pad = ops.round_up(n_tot, 256)
            w_pad = torch.zeros(n_pad, w_all.shape[1], dtype=pd, device=w_all.device)
            w_pad[:n_tot] = w_all.to(pd)
            P["cond_w"], P["cond_b"], P["cond_n"] = w_pad.contiguous(), torch.cat(cond_b).contiguous(), n_tot
        else:          # use_modulation=False: no conditioning linears at all
            P["cond_w"], P["cond_b"], P["cond_n"] = None, None, 0
        if self.time is not None:
            t = self.time
            kdim = t.to_out.weight.shape[1]
            kpad = ops.round_up(kdim, 8)
            w_emb = torch.zeros(self.features, kpad, dtype=pd, device=w_all.device)
            w_emb[:, :kdim] = t.to_out.weight.detach().to(pd)
            P["time"] = {"freqs": f32(t.weights), "w_emb": w_emb.contiguous(), "b_emb": f32(t.to_out.bias),
                         "w_mlp": t.mlp.weight.detach().to(pd).contiguous(),
                         "b_mlp": f32(t.mlp.bias), "kpad": kpad}
        return P

    def _add_conditioning(self, plan: _Plan, P: Dict, Bh: int) -> Tensor:
        """Appends the conditioning launches for Bh rows of (plan.sigma, plan.features_in) to
        `plan`; returns ss_all [Bh, n] fp32 (every Modulation / MergeModulate scale, shift and
        gate of the network, concatenated)."""
        dev = plan.sigma.device
        Fm = self.features
        n_tot = P["cond_n"]
        ss_all = torch.zeros(Bh, ops.round_up(n_tot, 8), device=dev)
        cond_bf = torch.zeros(1, Bh, Fm, dtype=self._act_dtype(), device=dev)
        fvec = torch.zeros(Bh, Fm, device=dev)
        plan.use_features_in = False
        if self.time is not None:
            tp = P["time"]
            feat = torch.zeros(Bh, tp["kpad"], device=dev)
            e0, e1 = torch.zeros(Bh, Fm, device=dev), torch.zeros(Bh, Fm, device=dev)
            plan.add(lambda: ops.time_features(plan.sigma, tp["freqs"], feat))
            plan.add(lambda: ops.skinny_linear(feat, tp["w_emb"], tp["b_emb"], e0, tp["kpad"], Fm,
                                               out_act=ops.ACT_GELU))
            plan.add(lambda: ops.skinny_linear(e0, tp["w_mlp"], tp["b_mlp"], e1, Fm, Fm,
                                               out_act=ops.ACT_GELU))
            plan.add(lambda: ops.skinny_linear(e1, tp["w_mlp"], tp["b_mlp"], fvec, Fm, Fm,
                                               out_act=ops.ACT_GELU))

            def add_features():
                if plan.use_features_in:
                    fvec.add_(plan.features_in)
            plan.add(add_features)
        else:
            plan.add(lambda: fvec.copy_(plan.features_in))
        plan.add(lambda: ops.silu_bf16(fvec, cond_bf))
        cond_bias = _pad_to(P["cond_b"], ss_all.shape[1])
        plan.add(lambda: ops.conv_gemm(cond_bf, P["cond_w"], ss_all.view(1, Bh, -1), c_in=Fm,
                                       n_valid=ss_all.shape[1], bias=cond_bias))
        return ss_all

    def _cond_table(self, sigmas: Tensor, features_in: Optional[Tensor]) -> Tensor:
        """ss_all for every row of `sigmas` [R] in one pass (the 97 MB of conditioning weights of
        the README network are read once per sample() call instead of once per step)."""
        R = sigmas.shape[0]
        key = ("cond", R)
        self.packed()
        if not self.use_modulation:       # nothing to evaluate: a dummy table keeps the step selector uniform
            plan = self._plans.get(key)
            if plan is None:
                plan = self._plans[key] = _Plan()
                plan.ss_all = torch.zeros(R, 8, device=sigmas.device)
            return plan.ss_all
        plan = self._plans.get(key)
        if plan is None:
            ops.device_check()
            plan = _Plan()
            plan.sigma = torch.zeros(R, device=sigmas.device)
            plan.features_in = torch.zeros(R, self.features, device=sigmas.device)
            plan.ss_all = self._add_conditioning(plan, self.packed(), R)
            self._plans[key] = plan
        plan.sigma.copy_(sigmas)
        plan.use_features_in = features_in is not None
        if features_in is not None:
            plan.features_in.copy_(features_in)
        plan.run_eager()
        return plan.ss_all

    # --------------------------------------------------------------------- plan
    def _build_plan(self, B: int, T: int, Bh: int, M: int, mode: str) -> _Plan:
        """B = batch of x; Bh = rows the trunk runs (2B under classifier-free guidance);
        M = embedding tokens (0 if none); mode in {'v', 'sample'}."""
        dev = self.net.down.weight.device
        P = self.packed()
        plan = _Plan()
        pool = _Pool(dev, reuse=True, dtype=self._act_dtype())
        G, Fm = self.groups, self.features
        levels = self.levels()
        total_f = 1
        for lv in levels:
            total_f *= lv.factor
        assert T % total_f == 0, f"length {T} must be divisible by the product of factors {total_f}"

        # ---- static I/O
        plan.x = torch.zeros(B, self.x_channels, T, device=dev)
        plan.append = torch.zeros(B, self.append_channels, T, device=dev) if self.append_channels else None
        plan.sigma = torch.zeros(Bh, device=dev)
        plan.features_in = torch.zeros(Bh, Fm, device=dev)
        plan.v = torch.zeros(B, self.out_channels, T, device=dev)
        plan.ab = torch.zeros(4, device=dev)
        adt = self._act_dtype()
        plan.embedding = torch.zeros(Bh, M, self.embedding_features, dtype=adt, device=dev) if M else None
        plan.cfg_scale = None
        plan.ctx = {i: torch.zeros(Bh, (T // _prod(self.factors[:i + 1])), ops.round_up(c, 16),
                                   dtype=adt, device=dev)
                    for i, c in enumerate(self.context_channels) if c > 0}
        plan.en = None                       # LayerNorm(embedding), shared by all cross-attentions
        plan.pre = []                        # step-invariant launches of a sampling plan
        add_ctx = plan.pre.append if mode == "sample" else plan.add

        # ---- statistics arena (zeroed once per forward)
        n_slots = 2 + sum(3 * (len(lv.items_down) + len(lv.items_up)) + 3 for lv in levels)
        arena = torch.zeros(n_slots, Bh, G, 2, dtype=torch.float64, device=dev)
        slot_i = [0]

        def new_stats() -> Tensor:
            s = arena[slot_i[0]]
            slot_i[0] += 1
            return s

        if mode == "sample":
            # the step's conditioning rows and alpha/beta are picked ON THE DEVICE from tables by a
            # step counter, so the captured graph is identical for every step (the host only
            # replays it, and several steps are captured back to back: _execute_steps)
            plan.step = torch.zeros(1, dtype=torch.int32, device=dev)
            plan.ctrl = torch.zeros(3, dtype=torch.int64, device=dev)
            plan.ab_table = torch.zeros(self.max_table_steps, 4, device=dev)
            plan.multi_graph, plan.multi_steps = None, 0
        plan.add(lambda: arena.zero_())

        # ---- conditioning: f = MLP(GELU(embed(sigma))) (+features); ss = W_all SiLU(f) + b.
        # The sampler knows every sigma_i up front and evaluates this ONCE for all steps
        # (_cond_table): its plan only receives the step's rows of the table.
        if mode == "sample":
            ss_all = torch.zeros(Bh, max(8, ops.round_up(P["cond_n"], 8)), device=dev)
            plan.ss_all = ss_all
            plan.use_features_in = False
            plan.add(lambda: ops.step_select(plan.step, plan.ctrl, plan.ab_table, plan.ab, ss_all))
        elif self.use_modulation:
            ss_all = self._add_conditioning(plan, P, Bh)
        else:
            ss_all = torch.zeros(Bh, 8, device=dev)
            plan.use_features_in = False
        ss_stride = ss_all.shape[1]
        mod = self.use_modulation

        # ---- one item chain
        def run_items(x: Tensor, x_stats: Tensor, items_p: List[Dict], lv: LevelParams, Tl: int,
                      last_needs_stats: bool, li: int = 0) -> Tuple[Tensor, Optional[Tensor]]:
            C = lv.ch
            narrow = C == 8 and not self._verify_fp32
            # thin levels (C = 32, 64) are HBM-bound: one fused ConvBlock kernel (mid_conv.cu)
            # instead of gn_silu -> conv_gemm (-> ln_film)
            thin = narrow or (self.fuse_thin_levels and C in (32, 64) and (C // G) % 4 == 0
                              and not self._verify_fp32)
            for idx, ip in enumerate(items_p):
                ss = ss_all[:, ip["ss_off"]:] if mod else None
                has_att, has_cross, has_inj = "att" in ip, "cross" in ip, "inj" in ip
                item_last = idx == len(items_p) - 1
                want_stats = (not item_last) or last_needs_stats
                mod_stats = new_stats() if (want_stats and not (has_att or has_cross or has_inj)) else None
                h_stats = new_stats()
                if thin:
                    h = pool.get(Bh, Tl, C)
                    y = pool.get(Bh, Tl, C)
                    w1, w2 = (ip["w1"], ip["w2"]) if narrow else (ip["w1_raw"], ip["w2_raw"])
                    p1, p2 = (None, None) if narrow else (ip["w1_mid"], ip["w2_mid"])
                    plan.add(lambda x=x, h=h, s=x_stats, hs=h_stats, ip=ip, w1=w1, p1=p1: ops.narrow_conv(
                        x, h, s, ip["gn1"][0], ip["gn1"][1], w1, ip["b1"], G, stats_out=hs,
                        gn_eps=self.GN_EPS, w_packed=p1))
                    plan.add(lambda x=x, h=h, y=y, hs=h_stats, ms=mod_stats, ip=ip, ss=ss, w2=w2, p2=p2:
                             ops.narrow_conv(h, y, hs, ip["gn2"][0], ip["gn2"][1], w2, ip["b2"], G,
                                             residual=x, scale_shift=ss, ss_stride=ss_stride, stats_out=ms,
                                             gn_eps=self.GN_EPS, ln_eps=self.MOD_LN_EPS, w_packed=p2))
                    pool.put(h)
                else:
                    h = pool.get(Bh, Tl, C)
                    r = pool.get(Bh, Tl, C)
                    y = pool.get(Bh, Tl, C) if mod else None
                    # use_modulation=False: the ResnetItem's output IS the item's output, so its
                    # GroupNorm statistics come out of conv2's epilogue
                    rs = None if mod else mod_stats
                    a = pool.get(Bh, Tl, C)
                    plan.add(lambda x=x, a=a, s=x_stats, ip=ip: ops.gn_silu(
                        x, a, s, ip["gn1"][0], ip["gn1"][1], G, self.GN_EPS))
                    plan.add(lambda a=a, h=h, hs=h_stats, ip=ip: ops.conv_gemm(
                        a, ip["w1"], h, c_in=C, n_valid=C, taps=(-1, 0, 1), bias=ip["b1"], stats=hs,
                        groups=G))
                    plan.add(lambda a=a, h=h, hs=h_stats, ip=ip: ops.gn_silu(
                        h, a, hs, ip["gn2"][0], ip["gn2"][1], G, self.GN_EPS))
                    plan.add(lambda x=x, a=a, r=r, ip=ip, rs=rs: ops.conv_gemm(
                        a, ip["w2"], r, c_in=C, n_valid=C, taps=(-1, 0, 1), bias=ip["b2"], residual=x,
                        stats=rs, groups=G))
                    pool.put(a)
                    xn_first = pool.get(Bh, Tl, C) if ((has_att or has_cross) and not has_inj and mod) else None
                    if mod:
                        # Modulation and the following attention pre-norm in ONE pass over the rows
                        plan.add(lambda r=r, y=y, ss=ss, ms=mod_stats, xn=xn_first: ops.ln_film(
                            r, y, ss, ss_stride, ms, G, self.MOD_LN_EPS, y2=xn, eps2=self.ATT_LN_EPS))
                        pool.put(r)
                    else:
                        y = r
                    pool.put(h)
                # the item's input is dead now (a level's skip is the chain's *output*)
                pool.put(x)
                x, x_stats = y, mod_stats
                if has_inj:
                    # InjectChannelsItem: conv1x1(cat([x, ctx])) + x as two accumulating GEMMs
                    # (W = [W_x | W_c]): tmp = ctx W_c^T + b + x ; out = x W_x^T + tmp
                    jp = ip["inj"]
                    ctxb = plan.ctx[li]
                    tmp, out_i = pool.get(Bh, Tl, C), pool.get(Bh, Tl, C)
                    inj_stats = new_stats() if (want_stats and not (has_att or has_cross)) else None
                    plan.add(lambda ctxb=ctxb, jp=jp, tmp=tmp, x=x: ops.conv_gemm(
                        ctxb, jp["w_c"], tmp, c_in=ctxb.shape[-1], n_valid=C, bias=jp["b"], residual=x))
                    plan.add(lambda x=x, jp=jp, tmp=tmp, o=out_i, st=inj_stats: ops.conv_gemm(
                        x, jp["w_x"], o, c_in=C, n_valid=C, residual=tmp, stats=st, groups=G))
                    pool.put(tmp)
                    pool.put(x)
                    x, x_stats = out_i, inj_stats
                mid = (self.heads or 0) * 64
                for kind in ("att", "cross"):
                    if kind not in ip:
                        continue
                    ap = ip[kind]
                    is_last_att = kind == "cross" or not has_cross
                    out_stats = new_stats() if (want_stats and is_last_att) else None
                    o = pool.get(Bh, Tl, mid)
                    y2 = pool.get(Bh, Tl, C)
                    if not thin and xn_first is not None:
                        xn, xn_first = xn_first, None      # produced by the fused Modulation pass
                    else:
                        xn = pool.get(Bh, Tl, C)
                        plan.add(lambda x=x, xn=xn: ops.ln_film(x, xn, None, 0, None, G, self.ATT_LN_EPS))
                    if kind == "att":
                        qkv = pool.get(Bh, Tl, 3 * mid)
                        plan.add(lambda xn=xn, qkv=qkv, ap=ap: ops.conv_gemm(
                            xn, ap["w_qkv"], qkv, c_in=C, n_valid=3 * mid, bias=ap["b_qkv"]))
                        plan.add(lambda qkv=qkv, o=o: ops.attention(
                            qkv[..., :mid], qkv[..., mid:2 * mid], qkv[..., 2 * mid:], o, self.heads,
                            64 ** -0.5))
                        pool.put(qkv)
                    else:
                        # context K/V do not depend on x or sigma: in sampling mode they are
                        # projected ONCE per sample() call (plan.pre), not once per step
                        E = self.embedding_features
                        q = pool.get(Bh, Tl, mid)
                        if plan.en is None:
                            plan.en = torch.empty(Bh, M, E, dtype=adt, device=dev)
                            add_ctx(lambda: ops.ln_film(plan.embedding, plan.en, None, 0, None, G,
                                                        self.ATT_LN_EPS))
                        kv = torch.empty(Bh, M, 2 * mid, dtype=adt, device=dev)
                        add_ctx(lambda kv=kv, ap=ap: ops.conv_gemm(
                            plan.en, ap["w_kv"], kv, c_in=E, n_valid=2 * mid, bias=ap["b_kv"]))
                        plan.add(lambda xn=xn, q=q, ap=ap: ops.conv_gemm(
                            xn, ap["w_q"], q, c_in=C, n_valid=mid, bias=ap["b_q"]))
                        plan.add(lambda q=q, kv=kv, o=o: ops.attention(
                            q, kv[..., :mid], kv[..., mid:], o, self.heads, 64 ** -0.5))
                        pool.put(q)
                    plan.add(lambda o=o, y2=y2, x=x, ap=ap, os_=out_stats: ops.conv_gemm(
                        o, ap["w_out"], y2, c_in=mid, n_valid=C, residual=x, stats=os_, groups=G))
                    pool.put(xn)
                    pool.put(o)
                    pool.put(x)
                    x, x_stats = y2, out_stats
            return x, x_stats

        # ---- recursive level walk
        def run_level(i: int, x_in: Optional[Tensor], T_in: int) -> Tuple[Tensor, Optional[Tensor]]:
            """Returns the level's output [Bh, T_in, out_ch] (+ its stats) for i >= 1;
            level 0 writes plan.v / x_next itself."""
            lv, Lp = levels[i], P["levels"][i]
            Tl = T_in // lv.factor
            C = lv.ch
            innermost = i == len(levels) - 1
            x = pool.get(Bh, Tl, C)
            st = new_stats()
            if i == 0:
                for half in range(Bh // B):
                    plan.add(lambda half=half, x=x, st=st: ops.stem_in(
                        plan.x, Lp["down_w"], Lp["down_b"], x[half * B:(half + 1) * B], lv.factor,
                        append=plan.append, stats=st[half * B:(half + 1) * B], groups=G))
            else:
                plan.add(lambda x=x, st=st: ops.conv_gemm(
                    x_in.view(Bh, Tl, lv.factor * lv.in_ch), Lp["down_w"], x, c_in=lv.factor * lv.in_ch,
                    n_valid=C, bias=Lp["down_b"], stats=st, groups=G))
            x, st = run_items(x, st, Lp["items_down"], lv, Tl, last_needs_stats=innermost, li=i)
            if not innermost:
                skip = x
                x, st = run_level(i + 1, skip, Tl)
                pool.put(skip)
            x, st = run_items(x, st, Lp["items_up"], lv, Tl, last_needs_stats=False, li=i)
            gate = ss_all[:, Lp["gate_off"]:] if mod else None
            if i == 0:
                plan.h0 = x
                plan.gate0 = gate if mod else torch.ones(Bh, 8, device=dev)
                plan.level0 = (lv, Lp)
                return x, None
            out = pool.get(Bh, T_in, lv.out_ch)
            ost = new_stats()
            if not mod:
                # SkipCat: y = upsample conv (+ bias); tmp = Wc1 (skip * s) + bc; out = Wc2 y + tmp
                Co = lv.out_ch
                rr = max(1, 16 // Co)
                assert T_in % rr == 0, "SkipCat merge of an 8-channel level needs an even length"
                y_up, tmp = pool.get(Bh, T_in, Co), pool.get(Bh, T_in, Co)

                def rows(t, rr=rr, Co=Co):
                    return t.view(Bh, T_in // rr, rr * Co)
                if lv.factor > 1:
                    plan.add(lambda x=x, y_up=y_up: ops.conv_gemm(
                        x, Lp["up_w"], y_up.view(Bh, Tl, lv.factor * lv.out_ch), c_in=C, n_valid=lv.out_ch,
                        up_factor=lv.factor, bias=Lp["up_b"]))
                else:
                    plan.add(lambda x=x, y_up=y_up: ops.conv_gemm(
                        x, Lp["up_w"], y_up, c_in=C, n_valid=lv.out_ch, taps=(-1, 0, 1), bias=Lp["up_b"]))
                plan.add(lambda tmp=tmp: ops.conv_gemm(rows(x_in), Lp["cat_w1"], rows(tmp), c_in=rr * Co,
                                                      n_valid=rr * Co, bias=Lp["cat_b"]))
                plan.add(lambda y_up=y_up, tmp=tmp, out=out, ost=ost: ops.conv_gemm(
                    rows(y_up), Lp["cat_w2"], rows(out), c_in=rr * Co, n_valid=rr * Co, residual=rows(tmp),
                    stats=ost if rr == 1 else None, groups=G))
                if rr > 1:           # the epilogue's group mapping does not see the paired layout
                    plan.add(lambda out=out, ost=ost: ops.gn_stats(out, ost, G))
                pool.put(y_up)
                pool.put(tmp)
                pool.put(x)
                return out, ost
            if lv.factor > 1:
                plan.add(lambda x=x, out=out, ost=ost: ops.conv_gemm(
                    x, Lp["up_w"], out.view(Bh, Tl, lv.factor * lv.out_ch), c_in=C, n_valid=lv.out_ch,
                    up_factor=lv.factor, bias=Lp["up_b"], residual=x_in.view(Bh, Tl, lv.factor * lv.out_ch),
                    gate=gate, stats=ost, groups=G))
            else:
                plan.add(lambda x=x, out=out, ost=ost: ops.conv_gemm(
                    x, Lp["up_w"], out, c_in=C, n_valid=lv.out_ch, taps=(-1, 0, 1), bias=Lp["up_b"],
                    residual=x_in, gate=gate, stats=ost, groups=G))
            pool.put(x)
            return out, ost

        run_level(0, None, T)
        lv0, L0 = plan.level0

        def final():
            kw = dict(append=plan.append, w_adapt=L0.get("adapt_w"), b_adapt=L0.get("adapt_b"),
                      cfg_scale=plan.cfg_scale)
            if mode == "sample":   # v and the VSampler update in one pass; x advanced in place
                ops.stem_out(plan.h0, plan.x, L0["up_w"], L0["up_b"], plan.gate0, lv0.factor,
                             x_next=plan.x, ab=plan.ab, **kw)
            else:
                ops.stem_out(plan.h0, plan.x, L0["up_w"], L0["up_b"], plan.gate0, lv0.factor,
                             v_out=plan.v, **kw)
        plan.add(final)
        if mode == "sample":
            plan.add(lambda: ops.step_advance(plan.step))
        plan.workspace_bytes = pool.total_bytes
        assert slot_i[0] <= n_slots
        return plan

    def _plan(self, B: int, T: int, Bh: int, M: int, mode: str, baked: Tuple = ()) -> _Plan:
        """`baked` = host-side values frozen into the captured graph (cfg scale, features flag)."""
        key = (B, T, Bh, M, mode, baked)
        self.packed()                      # refreshes the packed weights in place if needed
        plan = self._plans.get(key)
        if plan is None:
            ops.device_check()
            plan = self._plans[key] = self._build_plan(B, T, Bh, M, mode)
        return plan

    def profile_plan(self, plan: _Plan, iters: int = 5):
        """Instrumented eager passes of a plan: CUDA events around every launch, aggregated
        per kernel/shape -> {label: count per pass, avg/total ms per pass, flops, bytes}."""
        with ops.trace(timing=True) as tr:
            for _ in range(iters):
                if hasattr(plan, "step"):
                    plan.step.zero_()
                plan.run_eager()
        table = tr.table()
        for row in table.values():
            row["count"] //= iters
            row["ms_total"] /= iters
        return table

    def _execute(self, plan: _Plan) -> None:
        """First call eager (validates every launch), second call captures, then replays."""
        if not self.use_cuda_graph:
            plan.run_eager()
        elif plan.graph is not None:
            plan.graph.replay()
        elif plan.runs == 0:
            with ops.trace() as tr:          # also counts the kernels of one net evaluation
                plan.run_eager()
            plan.n_kernels = len(tr.records)
        else:
            g = torch.cuda.CUDAGraph()
            torch.cuda.synchronize()
            # inside the captured graph no kernel writes the packed weights, so the GEMMs may
            # fetch them before their programmatic-dependency wait (conv_gemm.cu, early_w)
            _lib.lib().adp_debug_set(2, 1)
            try:
                with torch.cuda.graph(g):
                    plan.run_eager()
            finally:
                _lib.lib().adp_debug_set(2, 0)
            plan.graph = g
            g.replay()
        plan.runs += 1

    def _execute_steps(self, plan: _Plan, n: int) -> None:
        """n consecutive sampling steps of a 'sample' plan.  Once the single-step graph exists, a
        second graph holding `steps_per_graph` steps back to back is captured and used for full
        groups: 5 graph launches instead of 50 per 50-step sample (host-side launch cost and its
        variance between boxes stay off the critical path)."""
        S = self.steps_per_graph
        while n > 0:
            if (self.use_cuda_graph and S > 1 and n >= S and plan.graph is not None):
                if plan.multi_graph is None or plan.multi_steps != S:
                    g = torch.cuda.CUDAGraph()
                    torch.cuda.synchronize()
                    _lib.lib().adp_debug_set(2, 1)
                    try:
                        with torch.cuda.graph(g):
                            for _ in range(S):
                                plan.run_eager()
                    finally:
                        _lib.lib().adp_debug_set(2, 0)
                    plan.multi_graph, plan.multi_steps = g, S
                plan.multi_graph.replay()
                plan.runs += S
                n -= S
            else:
                self._execute(plan)
                n -= 1

    def _set_step_tables(self, plan: _Plan, table: Tensor, ab_rows: Tensor, share: int = 1) -> None:
        """Points the plan's step selector at a block of conditioning rows [n, Bh, stride] and its
        alpha/beta rows [n_iterations, 4]; resets the device step counter."""
        assert ab_rows.shape[0] <= plan.ab_table.shape[0], "too many iterations per conditioning block"
        plan.ab_table[: ab_rows.shape[0]].copy_(ab_rows, non_blocking=True)
        plan.ctrl.copy_(torch.tensor([table.data_ptr(), share, table.shape[0]], dtype=torch.int64),
                        non_blocking=True)
        plan.step.zero_()

    def _stage_inputs(self, plan: _Plan, x: Tensor, time: Optional[Tensor], features, embedding,
                      embedding_scale: float, embedding_mask_proba: float, append_channels,
                      channels=None):
        B = x.shape[0]
        Bh = plan.sigma.shape[0]
        cfg = Bh == 2 * B
        for d, buf in plan.ctx.items():       # InjectChannelsItem context: [B, ctx, T_d] -> channels-last bf16
            assert channels is not None and channels[d] is not None, \
                f"context `channels[{d}]` is required (context_channels[{d}] > 0)"
            c = channels[d]
            assert c.shape[1] == self.context_channels[d] and c.shape[2] == buf.shape[1], \
                "context `channels` at depth must match resolution and context_channels"
            buf[:B, :, : c.shape[1]].copy_(c.transpose(1, 2))
            if cfg:
                buf[B:, :, : c.shape[1]].copy_(c.transpose(1, 2))
        if plan.x.data_ptr() != x.data_ptr():
            plan.x.copy_(x)
        if self.append_channels:
            assert exists(append_channels), "append_channels is required (AppendChannelsPlugin)"
            plan.append.copy_(append_channels)
        if self.time is not None:
            assert exists(time), "time conditioning requires the time argument"
            plan.sigma[:B].copy_(time.reshape(-1))
            if cfg:
                plan.sigma[B:].copy_(time.reshape(-1))
            plan.use_features_in = exists(features)
        elif self.use_modulation:
            assert exists(features), "use_time_conditioning=False needs features="
        if exists(features):
            plan.features_in[:B].copy_(features)
            if cfg:
                plan.features_in[B:].copy_(features)
        if plan.embedding is not None:
            assert exists(embedding), "ClassiferFreeGuidancePlugin requires embedding"
            emb = embedding
            if self.fixed_embedding is not None:
                fixed = self.fixed_embedding.weight[: emb.shape[1]].unsqueeze(0).expand_as(emb)
                if embedding_mask_proba > 0.0:          # a_unet CFG plugin, training-time masking
                    mask = torch.bernoulli(torch.full((B, 1, 1), embedding_mask_proba,
                                                      device=emb.device)).to(torch.bool)
                    emb = torch.where(mask, fixed, emb)
                if cfg:
                    plan.embedding[B:].copy_(fixed)
            plan.embedding[:B].copy_(emb)
        plan.cfg_scale = float(embedding_scale) if cfg else None

    def _shape_key(self, x: Tensor, embedding, embedding_scale: float):
        B, _, T = x.shape
        cfg = self.use_embedding_cfg and exists(embedding) and embedding_scale != 1.0
        M = embedding.shape[1] if (exists(embedding) and any(self.cross_attentions)) else 0
        return B, T, (2 * B if cfg else B), M

    def forward(self, x: Tensor, time: Optional[Tensor] = None, *, features: Optional[Tensor] = None,
                embedding: Optional[Tensor] = None, embedding_scale: float = 1.0,
                embedding_mask_proba: float = 0.0, channels=None,
                append_channels: Optional[Tensor] = None) -> Tensor:
        assert x.is_cuda, "the B200 path runs on a CUDA device only (no CPU fallback)"
        if self.use_embedding_cfg:
            assert exists(embedding), "ClassiferFreeGuidancePlugin requires embedding"
        ctx_list = [c for c in (channels or []) if exists(c)]
        if torch.is_grad_enabled() and (
                any(p.requires_grad for p in self.parameters()) or
                any(exists(t) and t.requires_grad for t in (x, features, embedding, append_channels, *ctx_list))):
            # differentiable: custom loss_fn / diffusion_t (reference models.py:28,37)
            from .training import differentiable_forward
            return differentiable_forward(self, x, time, features=features, embedding=embedding,
                                          embedding_scale=embedding_scale,
                                          embedding_mask_proba=embedding_mask_proba,
                                          append_channels=append_channels, channels=channels)
        return self._forward_inference(x, time, features, embedding, embedding_scale,
                                       embedding_mask_proba, append_channels, channels)

    @torch.no_grad()
    def _forward_inference(self, x, time, features, embedding, embedding_scale,
                           embedding_mask_proba, append_channels, channels=None) -> Tensor:
        self._check_untracked_updates()
        B, T, Bh, M = self._shape_key(x, embedding, embedding_scale)
        plan = self._plan(B, T, Bh, M, "v", (float(embedding_scale) if Bh != B else None,
                                             exists(features)))
        self._stage_inputs(plan, x.float(), time, features, embedding, embedding_scale,
                           embedding_mask_proba, append_channels, channels)
        self._execute(plan)
        return plan.v.clone().to(x.dtype)

    @torch.no_grad()
    def sample_loop(self, x_noisy: Tensor, sigmas: Tensor, alphas: Tensor, betas: Tensor,
                    progress=None, **kwargs) -> Tensor:
        """VSampler's loop (reference diffusion.py:183-188) with the per-step update fused into
        the net's last kernel: one graph launch per step, no host sync inside the loop."""
        assert x_noisy.is_cuda, "the B200 path runs on a CUDA device only (no CPU fallback)"
        self._check_untracked_updates()
        embedding = kwargs.get("embedding")
        scale = kwargs.get("embedding_scale", 1.0)
        B, T, Bh, M = self._shape_key(x_noisy, embedding, scale)
        plan = self._plan(B, T, Bh, M, "sample", (float(scale) if Bh != B else None,
                                                  exists(kwargs.get("features"))))
        self._stage_inputs(plan, x_noisy.float(), sigmas[0], kwargs.get("features"), embedding, scale,
                           kwargs.get("embedding_mask_proba", 0.0), kwargs.get("append_channels"),
                           kwargs.get("channels"))
        for fn in plan.pre:          # cross-attention context K/V: once per call
            fn()
        num_steps = sigmas.shape[0] - 1
        ab = torch.stack([alphas[:-1], betas[:-1], alphas[1:], betas[1:]], dim=1).float().contiguous()
        sig = sigmas.float().repeat(1, Bh // B).contiguous()      # [N+1, Bh]
        # conditioning table in blocks of <= ~4096 rows (190 KB of fp32 per row for the README net);
        # inside a block the device picks each step's rows: graph launches only, no host sync
        block = max(1, min(self.cond_table_rows // Bh, self.max_table_steps))
        it = iter(progress) if progress is not None else None
        for first in range(0, num_steps, block):
            n = min(block, num_steps - first)
            feats = plan.features_in.repeat(n, 1) if plan.use_features_in else None
            table = self._cond_table(sig[first:first + n].reshape(-1), feats).view(n, Bh, -1)
            self._set_step_tables(plan, table, ab[first:first + n])
            if it is None:
                self._execute_steps(plan, n)
            else:                      # progress bar: one graph launch per step
                for _ in range(n):
                    next(it)
                    self._execute(plan)
        if it is not None:
            for _ in it:               # let the progress generator finish (last description update)
                pass
        return plan.x.clone().to(x_noisy.dtype)


def _inpaint_loop(self, x_noisy: Tensor, source: Tensor, mask: Tensor, sigmas: Tensor, alphas: Tensor,
                  betas: Tensor, num_resamples: int, progress=None, **kwargs) -> Tensor:
    """VInpainter's loop (reference diffusion.py:338-352): per step `num_resamples` net evaluations;
    each one advances x to the level of the NEXT step only on the last resample (otherwise it is
    re-noised back to the current level), then the known region (mask) is replaced by the source
    noised to that level.  One graph launch + one blend kernel per evaluation; the noise is drawn
    with torch.randn_like(source) in the reference's order."""
    assert x_noisy.is_cuda, "the B200 path runs on a CUDA device only (no CPU fallback)"
    self._check_untracked_updates()
    embedding = kwargs.get("embedding")
    scale = kwargs.get("embedding_scale", 1.0)
    B, T, Bh, M = self._shape_key(x_noisy, embedding, scale)
    plan = self._plan(B, T, Bh, M, "sample", (float(scale) if Bh != B else None,
                                              exists(kwargs.get("features"))))
    self._stage_inputs(plan, x_noisy.float(), sigmas[0], kwargs.get("features"), embedding, scale,
                       kwargs.get("embedding_mask_proba", 0.0), kwargs.get("append_channels"),
                       kwargs.get("channels"))
    for fn in plan.pre:
        fn()
    num_steps = sigmas.shape[0] - 1
    a, b = alphas.float(), betas.float()
    # ab[i][j]: coefficients of a step from level i to level i + j (j = 0: stay, re-noise)
    ab = torch.stack([torch.stack([a[:-1], b[:-1], a[:-1], b[:-1]], 1),
                      torch.stack([a[:-1], b[:-1], a[1:], b[1:]], 1)], 1).contiguous()
    sig = sigmas.float().repeat(1, Bh // B).contiguous()
    src = source.float().expand_as(plan.x).contiguous()
    mask_u8 = mask.expand_as(plan.x).to(torch.uint8).contiguous()
    block = max(1, min(self.cond_table_rows // Bh, self.max_table_steps // max(1, num_resamples)))
    # per iteration (step i, resample r): alpha/beta row = ab[i][r is the last]
    last = torch.zeros(num_resamples, dtype=torch.long, device=ab.device)
    last[-1] = 1
    it = iter(progress) if progress is not None else None
    for first in range(0, num_steps, block):
        n = min(block, num_steps - first)
        feats = plan.features_in.repeat(n, 1) if plan.use_features_in else None
        table = self._cond_table(sig[first:first + n].reshape(-1), feats).view(n, Bh, -1)
        ab_rows = ab[first:first + n][:, last].reshape(n * num_resamples, 4)
        self._set_step_tables(plan, table, ab_rows, share=num_resamples)
        for _ in range(n):
            if it is not None:
                next(it)
            for r in range(num_resamples):
                self._execute(plan)
                ops.inpaint_blend(plan.x, src, torch.randn_like(source).float().expand_as(plan.x).contiguous(),
                                  mask_u8, plan.ab)
    if it is not None:
        for _ in it:
            pass
    return plan.x.clone().to(x_noisy.dtype)


B200UNet.inpaint_loop = torch.no_grad()(_inpaint_loop)


def _arv_loop(self, current: Tensor, sigmas: Tensor, progress=None, **kwargs) -> Tensor:
    """ARVSampler.sample_loop (reference diffusion.py:223-238): the net input is cat([current,
    sigma_i]) with a noise level PER POSITION (sigmas [N+1, B, 1, T]) and no time conditioning.
    The plan's input buffer holds that concatenation for the whole loop: one graph launch (the
    net) + one adp_arv_step (the update, which also writes sigma_{i+1} into the last channel)."""
    assert current.is_cuda, "the B200 path runs on a CUDA device only (no CPU fallback)"
    self._check_untracked_updates()
    embedding = kwargs.get("embedding")
    scale = kwargs.get("embedding_scale", 1.0)
    B, C, T = current.shape
    assert C + 1 == self.x_channels and sigmas.shape[1:] == (B, 1, T)
    plan_x = torch.cat([current.float(), sigmas[0].float()], dim=1)
    _, _, Bh, M = self._shape_key(plan_x, embedding, scale)
    plan = self._plan(B, T, Bh, M, "v", (float(scale) if Bh != B else None, exists(kwargs.get("features"))))
    self._stage_inputs(plan, plan_x, None, kwargs.get("features"), embedding, scale,
                       kwargs.get("embedding_mask_proba", 0.0), kwargs.get("append_channels"),
                       kwargs.get("channels"))
    sig = sigmas.float().reshape(sigmas.shape[0], B, T).contiguous()
    it = iter(progress) if progress is not None else None
    for i in range(sigmas.shape[0] - 1):
        if it is not None:
            next(it)
        self._execute(plan)
        ops.arv_step(plan.x, plan.v, sig[i + 1])
    if it is not None:
        for _ in it:
            pass
    return plan.x[:, :C].clone().to(current.dtype)


B200UNet.arv_loop = torch.no_grad()(_arv_loop)


def _copy_tree(dst, src) -> None:
    """In-place refresh of a nested dict/list/tuple of tensors (same structure)."""
    if isinstance(dst, Tensor):
        dst.copy_(src)
    elif isinstance(dst, dict):
        for k in dst:
            _copy_tree(dst[k], src[k])
    elif isinstance(dst, (list, tuple)):
        for d, s_ in zip(dst, src):
            _copy_tree(d, s_)


def _prod(vals) -> int:
    out = 1
    for v in vals:
        out *= v
    return out


def _pad_to(t: Tensor, n: int) -> Tensor:
    if t.shape[0] == n:
        return t
    out = torch.zeros(n, dtype=t.dtype, device=t.device)
    out[: t.shape[0]] = t
    return out


def UNetV0(dim: int, in_channels: int, channels: Sequence[int], factors: Sequence[int],
           items: Sequence[int], **kwargs) -> nn.Module:
    """Drop-in for reference components.py:34 `UNetV0` (same kwargs, asserts and call
    signature); returns the B200-native module."""
    return B200UNet(dim=dim, in_channels=in_channels, channels=channels, factors=factors,
                    items=items, **kwargs)
