"""MuseTalk on the B200 engine: VAE-encode -> audio-conditioned UNet -> VAE-decode -> blend paste-back.

The reference only *wraps* these networks (diffusers ``UNet2DConditionModel`` / ``AutoencoderKL``:
avatars/musetalk/models/unet.py:29-48, vae.py:10-38) and drives them from ``MuseReal.inference_batch``
(avatars/musetalk_avatar.py:130-152).  Here the host code (this file) assembles the same graphs out of the engine's
device operators — tcgen05 implicit-GEMM convs / linears / attention GEMMs, GroupNorm, LayerNorm, softmax, GEGLU ... —
captures them ONCE into a CUDA graph per batch size and replays the graph per step.  Weights are taken from state_dicts
with the diffusers key scheme (so a real ``unet.pth`` / ``sd-vae`` loads by name).

Load-time rewrites (exact up to fp16 rounding):
  * timestep is the constant 0 (musetalk_avatar.py:61): ``time_emb_proj(silu(time_embedding(t=0)))`` is folded into the
    bias of every ResnetBlock's conv1;
  * ``latents / scaling_factor`` (vae.py:102) is folded into ``post_quant_conv``; ``scaling_factor * mean`` (vae.py:93)
    into ``quant_conv``;
  * q/k/v projections are fused and every head is zero-padded to a multiple of 16 channels (head_dim 40 -> 48) so the
    attention GEMMs meet the tensor-core K granularity; ``to_out`` gets the matching zero columns.
"""
from __future__ import annotations

import os

import math
from typing import Dict, List, Optional, Sequence

import numpy as np

from . import _capi
from ._capi import LtbError
from .engine import mirror_index
from .ops import ConvWeight, Ctx, DevTensor

KEY_PAD = 64  # cross-attention keys (50 audio tokens) padded to a multiple of 16


def _np(t) -> np.ndarray:
    if hasattr(t, "detach"):
        t = t.detach().cpu().float().numpy()
    return np.asarray(t, dtype=np.float32)


def _ceil16(x: int) -> int:
    return (x + 15) // 16 * 16


def _silu(x):
    return x / (1.0 + np.exp(-x))


class _Norm:
    def __init__(self, ctx: Ctx, sd, p):
        self.gamma = ctx.upload(_np(sd[p + ".weight"]))
        self.beta = ctx.upload(_np(sd[p + ".bias"]))


def _pad_heads_rows(w: np.ndarray, heads: int, d: int, dp: int) -> np.ndarray:
    """[heads*d, cin] -> [heads*dp, cin] with zero rows after each head."""
    out = np.zeros((heads * dp, w.shape[1]), np.float32)
    for h in range(heads):
        out[h * dp:h * dp + d] = w[h * d:(h + 1) * d]
    return out


def _pad_heads_vec(b: np.ndarray, heads: int, d: int, dp: int) -> np.ndarray:
    out = np.zeros(heads * dp, np.float32)
    for h in range(heads):
        out[h * dp:h * dp + d] = b[h * d:(h + 1) * d]
    return out


def _pad_heads_cols(w: np.ndarray, heads: int, d: int, dp: int) -> np.ndarray:
    """[cout, heads*d] -> [cout, heads*dp] with zero columns after each head."""
    out = np.zeros((w.shape[0], heads * dp), np.float32)
    for h in range(heads):
        out[:, h * dp:h * dp + d] = w[:, h * d:(h + 1) * d]
    return out


class _Attn:
    """One diffusers ``Attention`` block (self or cross) in engine layout."""

    def __init__(self, ctx: Ctx, sd, p: str, C: int, heads: int, kv_dim: Optional[int]):
        d = C // heads
        dp = _ceil16(d)
        self.C, self.heads, self.d, self.dp = C, heads, d, dp
        self.self_attn = kv_dim is None
        bias = (p + ".to_q.bias") in sd
        wq, wk, wv = (_pad_heads_rows(_np(sd[f"{p}.{n}.weight"]), heads, d, dp) for n in ("to_q", "to_k", "to_v"))
        bq = bk = bv = None
        if bias:
            bq, bk, bv = (_pad_heads_vec(_np(sd[f"{p}.{n}.bias"]), heads, d, dp) for n in ("to_q", "to_k", "to_v"))
        if self.self_attn:
            self.qkv = ConvWeight(ctx, np.concatenate([wq, wk, wv], 0), np.concatenate([bq, bk, bv]) if bias else None, tap_major=False)
        else:
            self.q = ConvWeight(ctx, wq, bq, tap_major=False)
            self.kv = ConvWeight(ctx, np.concatenate([wk, wv], 0), np.concatenate([bk, bv]) if bias else None, tap_major=False)
        self.out = ConvWeight(ctx, _pad_heads_cols(_np(sd[p + ".to_out.0.weight"]), heads, d, dp), _np(sd[p + ".to_out.0.bias"]),
                              tap_major=False)


class _Resnet:
    def __init__(self, ctx: Ctx, sd, p: str, temb_act: Optional[np.ndarray]):
        w1 = _np(sd[p + ".conv1.weight"])
        b1 = _np(sd[p + ".conv1.bias"]).copy()
        if temb_act is not None:   # constant timestep: time_emb_proj(silu(emb)) is a per-channel bias after conv1
            b1 += _np(sd[p + ".time_emb_proj.weight"]) @ temb_act + _np(sd[p + ".time_emb_proj.bias"])
        self.cin, self.cout = w1.shape[1], w1.shape[0]
        self.norm1, self.norm2 = _Norm(ctx, sd, p + ".norm1"), _Norm(ctx, sd, p + ".norm2")
        self.conv1 = ConvWeight(ctx, w1, b1)
        self.conv2 = ConvWeight(ctx, _np(sd[p + ".conv2.weight"]), _np(sd[p + ".conv2.bias"]))
        self.shortcut = None
        if (p + ".conv_shortcut.weight") in sd:
            self.shortcut = ConvWeight(ctx, _np(sd[p + ".conv_shortcut.weight"]), _np(sd[p + ".conv_shortcut.bias"]), tap_major=False)


class _Transformer:
    def __init__(self, ctx: Ctx, sd, p: str, C: int, heads: int, ctx_dim: int):
        self.C = C
        self.norm = _Norm(ctx, sd, p + ".norm")
        self.proj_in = ConvWeight(ctx, _np(sd[p + ".proj_in.weight"]), _np(sd[p + ".proj_in.bias"]), tap_major=False)
        self.proj_out = ConvWeight(ctx, _np(sd[p + ".proj_out.weight"]), _np(sd[p + ".proj_out.bias"]), tap_major=False)
        b = p + ".transformer_blocks.0"
        self.ln1, self.ln2, self.ln3 = (_Norm(ctx, sd, f"{b}.norm{i}") for i in (1, 2, 3))
        self.attn1 = _Attn(ctx, sd, b + ".attn1", C, heads, None)
        self.attn2 = _Attn(ctx, sd, b + ".attn2", C, heads, ctx_dim)
        self.ff1 = ConvWeight(ctx, _np(sd[b + ".ff.net.0.proj.weight"]), _np(sd[b + ".ff.net.0.proj.bias"]), tap_major=False)
        self.ff2 = ConvWeight(ctx, _np(sd[b + ".ff.net.2.weight"]), _np(sd[b + ".ff.net.2.bias"]), tap_major=False)


class Builder:
    """Emits engine ops for the diffusers building blocks.  Tensors are NHWC fp16 ``DevTensor``s of shape (N,H,W,C)."""

    GN_GROUPS = 32   # every GroupNorm of the diffusers UNet / VAE uses 32 groups
    # Fusing the GroupNorm statistics into the producing conv's epilogue (ltb_conv_op.gn_stats) is implemented and parity-tested,
    # but measured SLOWER on B200 (MuseTalk B=8: 15.6 -> 17.6 ms/step): the extra shuffles/atomics make the 0.9 PFLOP/s VAE convs
    # epilogue-bound, which costs more than the separate statistics pass (1.0 ms) saves.  Off by default.
    FUSE_GN_STATS = os.environ.get("LTB_FUSE_GN", "0") == "1"

    def __init__(self, ctx: Ctx):
        self.ctx = ctx
        self.temps: List[DevTensor] = []

    def _stats_for(self, out: DevTensor, n_img: int):
        """Ask the producing conv to also emit the GroupNorm statistics of `out` (fused into its epilogue when possible)."""
        if not self.FUSE_GN_STATS or out.C % self.GN_GROUPS or out.pitch != out.C or out.c_off:
            return None
        st = self.new(n_img * self.GN_GROUPS * 4)                  # n_img * groups * 2 floats
        out.stats = (st, self.GN_GROUPS)
        return st

    def new(self, *shape) -> DevTensor:
        t = self.ctx.alloc(shape, np.float16, zero=True)
        self.temps.append(t)
        return t

    # -- primitives
    def conv3(self, x: DevTensor, w: ConvWeight, res: Optional[DevTensor] = None, stride: int = 1, pad=(1, 1), out: Optional[DevTensor] = None,
              stats: bool = False):
        N, H, W, _ = x.shape
        OH = (H + (2 if pad == (1, 1) else 1) - 3) // stride + 1
        OW = (W + (2 if pad == (1, 1) else 1) - 3) // stride + 1
        if out is None:
            out = self.new(N, OH, OW, w.cout)
        st = self._stats_for(out, N) if stats else None
        self.ctx.conv(x, w, out, N=N, IH=H, IW=W, OH=OH, OW=OW, stride=(stride, stride), pad=pad, res=res,
                      gn_stats=st, gn_groups=self.GN_GROUPS if st is not None else 0, gn_hw=OH * OW)
        return out

    def linear(self, x: DevTensor, w: ConvWeight, res: Optional[DevTensor] = None, out: Optional[DevTensor] = None, stats_imgs: int = 0):
        """x (..., Cin) -> (..., Cout) ; also 1x1 convs.  stats_imgs > 0: also produce GroupNorm statistics (rows/stats_imgs pixels per image)."""
        rows = x.rows
        if out is None:
            out = self.new(*x.shape[:-1], w.cout)
        st = self._stats_for(out, stats_imgs) if stats_imgs else None
        self.ctx.conv(x, w, out, N=1, IH=1, IW=rows, OH=1, OW=rows, res=res,
                      gn_stats=st, gn_groups=self.GN_GROUPS if st is not None else 0, gn_hw=(rows // stats_imgs) if stats_imgs else 0)
        return out

    def groupnorm(self, x: DevTensor, n: _Norm, groups: int, eps: float, silu: bool):
        N, H, W, C = x.shape
        out = self.new(N, H, W, C)
        if x.stats is not None and x.stats[1] == groups:
            self.ctx.groupnorm_apply(x, N, H * W, groups, eps, x.stats[0], n.gamma, n.beta, silu, out)
        else:
            self.ctx.groupnorm(x, N, H * W, groups, eps, n.gamma, n.beta, silu, out)
        return out

    def layernorm(self, x: DevTensor, n: _Norm, eps: float = 1e-5):
        out = self.new(*x.shape)
        self.ctx.layernorm(x, x.rows, x.C, eps, n.gamma, n.beta, out)
        return out

    # -- blocks
    def resnet(self, x: DevTensor, r: _Resnet, groups: int, eps: float):
        h = self.conv3(self.groupnorm(x, r.norm1, groups, eps, True), r.conv1, stats=True)
        h = self.groupnorm(h, r.norm2, groups, eps, True)
        skip = self.linear(x, r.shortcut) if r.shortcut is not None else x
        return self.conv3(h, r.conv2, res=skip, stats=True)

    # softmax(QK^T)V as one tcgen05 kernel (scores never reach HBM); LTB_FUSE_ATTENTION=0 restores GEMM + softmax + GEMM
    FUSE_ATTENTION = os.environ.get("LTB_FUSE_ATTENTION", "1") == "1"

    def attention(self, a, xq: DevTensor, B: int, nq: int, res: DevTensor, kv_src: Optional[DevTensor] = None, n_keys: Optional[int] = None,
                  n_valid: Optional[int] = None, stats_imgs: int = 0):
        """xq: (B*nq, C) normalised tokens.  Self-attention when kv_src is None, else keys/values from kv_src (B*n_keys, kv_dim).
        Key counts are padded to a multiple of 16 (tensor-core N / K granularity); padded keys get probability 0."""
        ctx, H, dp, d = self.ctx, a.heads, a.dp, a.d
        Hdp = H * dp
        if a.self_attn:
            nk = _ceil16(nq)
            valid = nq
            if nk != nq:
                assert B == 1, "key padding of self-attention needs per-batch row padding"
            qkv = self.new(B * nq + (nk - nq), 3 * Hdp)                   # padded key rows stay zero
            self.linear(xq, a.qkv, out=DevTensor(qkv.ptr, (B * nq, 3 * Hdp)))
            q_ptr, q_pitch = qkv.ptr, 3 * Hdp
            k_ptr, v_ptr, kv_pitch = qkv.offset(Hdp), qkv.offset(2 * Hdp), 3 * Hdp
            kv_rows = nq
        else:
            q = self.linear(xq, a.q)                                      # (B*nq, Hdp)
            kv = self.linear(kv_src, a.kv)                                # (B*n_keys, 2*Hdp)
            q_ptr, q_pitch = q.ptr, Hdp
            k_ptr, v_ptr, kv_pitch = kv.ptr, kv.offset(Hdp), 2 * Hdp
            nk, valid, kv_rows = n_keys, n_valid, n_keys
        if self.FUSE_ATTENTION and dp % 16 == 0 and dp <= 160:
            VT = self.new(B * H, dp, nk)
            ctx.transpose_heads(v_ptr, B, kv_rows, kv_pitch, H, dp, nk, VT)
            O = self.new(B * nq, Hdp)
            ctx.attention(q_ptr, q_pitch, k_ptr, kv_pitch, kv_rows, VT, nk, B, H, nq, valid, dp, float(d) ** -0.5, O)
            return self.linear(O, a.out, res=res, stats_imgs=stats_imgs)
        S = self.new(B * H, nq, nk)
        qv = DevTensor(q_ptr, (nq, dp), pitch=q_pitch)
        sv = DevTensor(S.ptr, (nq, nk), pitch=nk)
        ctx.conv(qv, None, sv, N=1, IH=1, IW=nq, OH=1, OW=nq, cin=dp, cout=nk, w_ptr=k_ptr, ktot=kv_pitch,
                 zbatch=B * H, zdiv=H, in_z=(nq * q_pitch, dp), w_z=(kv_rows * kv_pitch, dp), out_z=(H * nq * nk, nq * nk))
        ctx.softmax(S, B * H * nq, nk, valid, float(d) ** -0.5)
        VT = self.new(B * H, dp, nk)
        ctx.transpose_heads(v_ptr, B, kv_rows, kv_pitch, H, dp, nk, VT)
        O = self.new(B * nq, Hdp)
        ov = DevTensor(O.ptr, (nq, dp), pitch=Hdp)
        ctx.conv(sv, None, ov, N=1, IH=1, IW=nq, OH=1, OW=nq, cin=nk, cout=dp, w_ptr=VT.ptr, ktot=nk,
                 zbatch=B * H, zdiv=H, in_z=(H * nq * nk, nq * nk), w_z=(H * dp * nk, dp * nk), out_z=(nq * Hdp, dp))
        return self.linear(O, a.out, res=res, stats_imgs=stats_imgs)

    def transformer(self, x: DevTensor, t: _Transformer, audio: DevTensor, groups: int):
        N, H, W, C = x.shape
        tok = self.linear(self.groupnorm(x, t.norm, groups, 1e-6, False), t.proj_in)       # (N,H,W,C) == tokens (N*HW, C)
        tok = self.attention(t.attn1, self.layernorm(tok, t.ln1), N, H * W, res=tok)
        tok = self.attention(t.attn2, self.layernorm(tok, t.ln2), N, H * W, res=tok, kv_src=audio, n_keys=KEY_PAD, n_valid=50)
        g = self.linear(self.layernorm(tok, t.ln3), t.ff1)                                 # (.., 8C)
        gg = self.new(N, H, W, 4 * C)
        self.ctx.geglu(g, N * H * W, 4 * C, gg)
        tok = self.linear(gg, t.ff2, res=tok)
        return self.linear(tok, t.proj_out, res=x)

    # Upsample2D (nearest 2x + conv3x3) as ONE kernel: four 2x2 sub-pixel convs over the low-res map (ops.ConvWeight.upconv).
    FUSE_UPSAMPLE = os.environ.get("LTB_FUSE_UPSAMPLE", "1") == "1"

    def upsample(self, x: DevTensor, w: ConvWeight):
        N, H, W, C = x.shape
        if self.FUSE_UPSAMPLE and w.upconv_supported() and x.pitch % 8 == 0 and x.c_off % 8 == 0:
            out = self.new(N, 2 * H, 2 * W, w.cout)
            self.ctx.conv(x, w, out, N=N, IH=H, IW=W, OH=2 * H, OW=2 * W, pad=(1, 1), upsample2x=True)
            return out
        up = self.new(N, 2 * H, 2 * W, C)
        self.ctx.upsample2x(x, N, H, W, up)
        return self.conv3(up, w, stats=True)

    def concat(self, a: DevTensor, b: DevTensor):
        N, H, W, _ = a.shape
        out = self.new(N, H, W, a.C + b.C)
        self.ctx.copy_channels(a, DevTensor(out.ptr, (N, H, W, a.C), pitch=out.C, c_off=0))
        self.ctx.copy_channels(b, DevTensor(out.ptr, (N, H, W, b.C), pitch=out.C, c_off=a.C))
        return out


class MuseTalkModel:
    """Device-resident UNet + VAE weights (replaces load_model()'s vae/unet/pe, musetalk_avatar.py:57-67)."""

    def __init__(self, ctx: Ctx, unet_sd: Dict, vae_sd: Dict, ucfg, vcfg, with_encoder: bool = True):
        self.ctx, self.ucfg, self.vcfg = ctx, ucfg, vcfg
        sd = unet_sd
        boc = ucfg.block_out_channels
        heads = ucfg.num_heads
        # constant timestep embedding (t = 0): [cos(0)..., sin(0)...] = [1]*half + [0]*half
        half = boc[0] // 2
        temb = np.concatenate([np.ones(half, np.float32), np.zeros(half, np.float32)])
        temb = _np(sd["time_embedding.linear_1.weight"]) @ temb + _np(sd["time_embedding.linear_1.bias"])
        temb = _np(sd["time_embedding.linear_2.weight"]) @ _silu(temb) + _np(sd["time_embedding.linear_2.bias"])
        ta = _silu(temb)
        self.u_conv_in = ConvWeight(ctx, _np(sd["conv_in.weight"]), _np(sd["conv_in.bias"]), pad_cin=16)
        self.u_down = []
        for i in range(len(boc)):
            blk = {"res": [], "attn": [], "down": None}
            for j in range(ucfg.layers_per_block):
                blk["res"].append(_Resnet(ctx, sd, f"down_blocks.{i}.resnets.{j}", ta))
                if ucfg.down_has_attn[i]:
                    blk["attn"].append(_Transformer(ctx, sd, f"down_blocks.{i}.attentions.{j}", boc[i], heads, ucfg.cross_attention_dim))
            if i < len(boc) - 1:
                p = f"down_blocks.{i}.downsamplers.0.conv"
                blk["down"] = ConvWeight(ctx, _np(sd[p + ".weight"]), _np(sd[p + ".bias"]), tap_major=False)
            self.u_down.append(blk)
        self.u_mid = (_Resnet(ctx, sd, "mid_block.resnets.0", ta),
                      _Transformer(ctx, sd, "mid_block.attentions.0", boc[-1], heads, ucfg.cross_attention_dim),
                      _Resnet(ctx, sd, "mid_block.resnets.1", ta))
        rev = list(reversed(boc))
        self.u_up = []
        for i in range(len(boc)):
            blk = {"res": [], "attn": [], "up": None}
            for j in range(ucfg.layers_per_block + 1):
                blk["res"].append(_Resnet(ctx, sd, f"up_blocks.{i}.resnets.{j}", ta))
                if ucfg.up_has_attn[i]:
                    blk["attn"].append(_Transformer(ctx, sd, f"up_blocks.{i}.attentions.{j}", rev[i], heads, ucfg.cross_attention_dim))
            if i < len(boc) - 1:
                p = f"up_blocks.{i}.upsamplers.0.conv"
                blk["up"] = ConvWeight(ctx, _np(sd[p + ".weight"]), _np(sd[p + ".bias"]))
            self.u_up.append(blk)
        self.u_norm_out = _Norm(ctx, sd, "conv_norm_out")
        self.u_conv_out = ConvWeight(ctx, _np(sd["conv_out.weight"]), _np(sd["conv_out.bias"]), pad_cout=32)   # 32: TMA halo kernel

        # ---- VAE decoder
        sd = vae_sd
        sf = vcfg.scaling_factor
        self.v_post_quant = ConvWeight(ctx, _np(sd["post_quant_conv.weight"]) / sf, _np(sd["post_quant_conv.bias"]), pad_cin=16, pad_cout=16,
                                       tap_major=False)
        self.v_dec_in = ConvWeight(ctx, _np(sd["decoder.conv_in.weight"]), _np(sd["decoder.conv_in.bias"]), pad_cin=16)
        self.v_dec_mid = self._vae_mid(ctx, sd, "decoder.mid_block")
        vrev = list(reversed(vcfg.block_out_channels))
        self.v_dec_up = []
        for i in range(len(vrev)):
            blk = {"res": [_Resnet(ctx, sd, f"decoder.up_blocks.{i}.resnets.{j}", None) for j in range(vcfg.layers_per_block + 1)], "up": None}
            if i < len(vrev) - 1:
                p = f"decoder.up_blocks.{i}.upsamplers.0.conv"
                blk["up"] = ConvWeight(ctx, _np(sd[p + ".weight"]), _np(sd[p + ".bias"]))
            self.v_dec_up.append(blk)
        self.v_dec_norm_out = _Norm(ctx, sd, "decoder.conv_norm_out")
        self.v_dec_out = ConvWeight(ctx, _np(sd["decoder.conv_out.weight"]), _np(sd["decoder.conv_out.bias"]), pad_cout=32)
        # ---- VAE encoder (BASELINE config 3; offline in the reference: avatars/musetalk/genavatar.py:126-128)
        self.with_encoder = with_encoder
        if with_encoder:
            vb = vcfg.block_out_channels
            self.v_enc_in = ConvWeight(ctx, _np(sd["encoder.conv_in.weight"]), _np(sd["encoder.conv_in.bias"]), pad_cin=16)
            self.v_enc_down = []
            for i in range(len(vb)):
                blk = {"res": [_Resnet(ctx, sd, f"encoder.down_blocks.{i}.resnets.{j}", None) for j in range(vcfg.layers_per_block)], "down": None}
                if i < len(vb) - 1:
                    p = f"encoder.down_blocks.{i}.downsamplers.0.conv"
                    blk["down"] = ConvWeight(ctx, _np(sd[p + ".weight"]), _np(sd[p + ".bias"]), tap_major=False)
                self.v_enc_down.append(blk)
            self.v_enc_mid = self._vae_mid(ctx, sd, "encoder.mid_block")
            self.v_enc_norm_out = _Norm(ctx, sd, "encoder.conv_norm_out")
            self.v_enc_out = ConvWeight(ctx, _np(sd["encoder.conv_out.weight"]), _np(sd["encoder.conv_out.bias"]), pad_cout=32)
            L = vcfg.latent_channels
            qw, qb = _np(sd["quant_conv.weight"])[:L, :, 0, 0] * sf, _np(sd["quant_conv.bias"])[:L] * sf   # mean rows, x scaling_factor
            w_lo = np.zeros((16, 16), np.float32)
            b_lo = np.zeros(16, np.float32)
            w_lo[:L, :2 * L] = qw
            b_lo[:L] = qb
            w_hi = np.zeros((16, 16), np.float32)
            b_hi = np.zeros(16, np.float32)
            w_hi[L:2 * L, :2 * L] = qw
            b_hi[L:2 * L] = qb
            self.v_quant_masked = ConvWeight(ctx, w_lo, b_lo, tap_major=False)    # masked latents -> channels [0, L)
            self.v_quant_ref = ConvWeight(ctx, w_hi, b_hi, tap_major=False)       # reference latents -> channels [L, 2L)
        # positional encoding table (unet.py:12-27), rows >= 50 zero (key padding)
        pe = np.zeros((KEY_PAD, ucfg.cross_attention_dim), np.float32)
        pos = np.arange(50, dtype=np.float32)[:, None]
        D = ucfg.cross_attention_dim
        div = np.exp(np.arange(0, D, 2, dtype=np.float32) * np.float32(-math.log(10000.0) / D))
        pe[:50, 0::2] = np.sin(pos * div)
        pe[:50, 1::2] = np.cos(pos * div)
        self.pe = ctx.upload(pe.astype(np.float16))
        ctx.sync()

    @staticmethod
    def _vae_mid(ctx, sd, p):
        a = p + ".attentions.0"
        C = _np(sd[a + ".to_q.weight"]).shape[0]
        return (_Resnet(ctx, sd, p + ".resnets.0", None), _Norm(ctx, sd, a + ".group_norm"), _Attn(ctx, sd, a, C, 1, None),
                _Resnet(ctx, sd, p + ".resnets.1", None))

    # ------------------------------------------------------------------------------------------ graph emitters
    def emit_unet(self, b: Builder, latents16: DevTensor, audio_pe: DevTensor, taps: Optional[dict] = None) -> DevTensor:
        """latents16 (B,h,w,16) [8 real channels], audio_pe (B*64, 384) -> predicted latents (B,h,w,16) [4 real channels]."""
        cfg = self.ucfg
        G, eps = cfg.norm_groups, cfg.norm_eps
        h = b.conv3(latents16, self.u_conv_in, stats=True)
        skips = [h]
        for i, blk in enumerate(self.u_down):
            for j, r in enumerate(blk["res"]):
                h = b.resnet(h, r, G, eps)
                if blk["attn"]:
                    h = b.transformer(h, blk["attn"][j], audio_pe, G)
                skips.append(h)
            if blk["down"] is not None:
                h = b.conv3(h, blk["down"], stride=2)
                skips.append(h)
            if taps is not None:
                taps[f"down{i}"] = h
        h = b.resnet(h, self.u_mid[0], G, eps)
        h = b.transformer(h, self.u_mid[1], audio_pe, G)
        h = b.resnet(h, self.u_mid[2], G, eps)
        if taps is not None:
            taps["mid"] = h
        for i, blk in enumerate(self.u_up):
            for j, r in enumerate(blk["res"]):
                h = b.resnet(b.concat(h, skips.pop()), r, G, eps)
                if blk["attn"]:
                    h = b.transformer(h, blk["attn"][j], audio_pe, G)
            if blk["up"] is not None:
                h = b.upsample(h, blk["up"])
            if taps is not None:
                taps[f"up{i}"] = h
        return b.conv3(b.groupnorm(h, self.u_norm_out, G, eps, True), self.u_conv_out)

    def _emit_vae_mid(self, b: Builder, h: DevTensor, mid, G, eps):
        r0, gn, attn, r1 = mid
        h = b.resnet(h, r0, G, eps)
        N, H, W, C = h.shape
        h = b.attention(attn, b.groupnorm(h, gn, G, eps, False), N, H * W, res=h, stats_imgs=N)
        st = h.stats
        h = DevTensor(h.ptr, (N, H, W, C))
        h.stats = st
        return b.resnet(h, r1, G, eps)

    def emit_vae_decode(self, b: Builder, pred16: DevTensor, out_u8: DevTensor, taps: Optional[dict] = None) -> DevTensor:
        """pred16 (B,h,w,16) latents [4 real channels] -> uint8 BGR image written to out_u8 (B,8h,8w,3)."""
        cfg = self.vcfg
        G, eps = cfg.norm_groups, cfg.norm_eps
        h = b.conv3(b.linear(DevTensor(pred16.ptr, (*pred16.shape[:-1], 16), pitch=pred16.pitch), self.v_post_quant), self.v_dec_in, stats=True)
        h = self._emit_vae_mid(b, h, self.v_dec_mid, G, eps)
        if taps is not None:
            taps["dec_mid"] = h
        for i, blk in enumerate(self.v_dec_up):
            for r in blk["res"]:
                h = b.resnet(h, r, G, eps)
            if blk["up"] is not None:
                h = b.upsample(h, blk["up"])
            if taps is not None:
                taps[f"dec_up{i}"] = h
        img = b.conv3(b.groupnorm(h, self.v_dec_norm_out, G, eps, True), self.v_dec_out)   # (B,H,W,16), RGB in channels 0..2
        N, H, W, _ = img.shape
        b.ctx.vae_post(img, N * H * W, out_u8)
        return img

    def emit_vae_encode(self, b: Builder, img_u8: DevTensor, out_latents16: DevTensor):
        """img_u8 (B,H,W,3) uint8 BGR -> get_latents_for_unet (vae.py:110-122, latent_dist.mode()): (B,H/8,W/8,16) [8 real]."""
        assert self.with_encoder
        cfg = self.vcfg
        G, eps = cfg.norm_groups, cfg.norm_eps
        B, H, W, _ = img_u8.shape
        x = b.new(2 * B, H, W, 16)
        b.ctx.vae_pre(img_u8, B, H, W, True, DevTensor(x.ptr, (B, H, W, 16)))                                  # masked copies
        b.ctx.vae_pre(img_u8, B, H, W, False, DevTensor(x.offset(B * H * W * 16), (B, H, W, 16)))              # reference copies
        h = b.conv3(x, self.v_enc_in, stats=True)
        for blk in self.v_enc_down:
            for r in blk["res"]:
                h = b.resnet(h, r, G, eps)
            if blk["down"] is not None:
                h = b.conv3(h, blk["down"], stride=2, pad=(0, 0), stats=True)     # F.pad(x,(0,1,0,1)) + conv s2 p0
        h = self._emit_vae_mid(b, h, self.v_enc_mid, G, eps)
        m = b.conv3(b.groupnorm(h, self.v_enc_norm_out, G, eps, True), self.v_enc_out)   # (2B,h,w,16): moments in 0..7
        _, lh, lw, mc = m.shape
        half = B * lh * lw * mc
        tmp = b.linear(DevTensor(m.ptr, (B, lh, lw, 16), pitch=mc), self.v_quant_masked)
        b.linear(DevTensor(m.offset(half), (B, lh, lw, 16), pitch=mc), self.v_quant_ref, res=tmp, out=out_latents16)
        return out_latents16


class MuseTalkAvatar:
    """Avatar assets resident in HBM (replaces load_avatar's lists, musetalk_avatar.py:69-91): full frames, bbox
    (x1,y1,x2,y2), mask crop boxes (x_s,y_s,x_e,y_e), 3-channel blend masks and the pre-computed UNet input latents.

    frames_resident=False: a frame-free avatar — instead of the full frames only their crop boxes (the "body crops", packed like the
    masks) go to the device (``frames`` is None, ``body`` holds them); sessions composite the blended crop box (the *_region methods)
    and the host writes it into a copy of its own frame (engine.paste_region).  get_image_blending changes nothing outside it."""

    def __init__(self, ctx: Ctx, frames, masks, coords, crop_boxes, latents, frames_resident: bool = True):
        self.ctx = ctx
        self.frames_resident = bool(frames_resident)
        if self.frames_resident:
            frames = np.ascontiguousarray(np.asarray(frames), np.uint8)
            self.n, self.H, self.W = frames.shape[0], frames.shape[1], frames.shape[2]
        else:
            self.n, (self.H, self.W) = len(frames), np.shape(frames[0])[:2]
        self.frames_host = frames
        self.coords_host = np.ascontiguousarray(np.asarray(coords), np.int32).reshape(self.n, 4)
        self.crop_host = np.ascontiguousarray(np.asarray(crop_boxes), np.int32).reshape(self.n, 4)
        offs, blobs, o = [], [], 0
        for i in range(self.n):
            xs, ys, xe, ye = self.crop_host[i]
            x1, y1, x2, y2 = self.coords_host[i]
            m = np.ascontiguousarray(masks[i], np.uint8)
            if m.shape != (ye - ys, xe - xs, 3):
                raise ValueError(f"mask {i} has shape {m.shape}, crop box needs {(ye - ys, xe - xs, 3)}")
            if not (0 <= xs <= x1 < x2 <= xe <= self.W and 0 <= ys <= y1 < y2 <= ye <= self.H):
                raise ValueError(f"avatar frame {i}: bbox / crop box outside the frame")
            offs.append(o)
            blobs.append(m.reshape(-1))
            o += m.size
        self.masks_host = [np.asarray(m, np.uint8) for m in masks]
        c = self.crop_host
        self.region_max = (int((c[:, 3] - c[:, 1]).max()), int((c[:, 2] - c[:, 0]).max()))
        self.frames = ctx.upload(frames) if self.frames_resident else None
        self.body = None if self.frames_resident else ctx.upload(np.concatenate(
            [np.ascontiguousarray(frames[i][ys:ye, xs:xe], np.uint8).reshape(-1) for i, (xs, ys, xe, ye) in enumerate(c)]))
        self.coords = ctx.upload(self.coords_host)
        self.crop = ctx.upload(self.crop_host)
        self.masks = ctx.upload(np.concatenate(blobs))
        self.mask_off = ctx.upload(np.asarray(offs, np.int64))
        # latents: list of (1,8,h,w) arrays (latents.pt) -> NHWC fp16 padded to 16 channels
        lat = np.concatenate([_np(l) for l in latents], 0)
        self.lat_hw = lat.shape[2]
        lat16 = np.zeros((lat.shape[0], lat.shape[2], lat.shape[3], 16), np.float16)
        lat16[..., :8] = lat.transpose(0, 2, 3, 1)
        self.latents = ctx.upload(lat16)

    def box(self, idx: int):
        """The crop box of frame idx as (y1, y2, x1, x2), the order engine.paste_region takes."""
        xs, ys, xe, ye = (int(v) for v in self.crop_host[idx])
        return (ys, ye, xs, xe)

    def paste_op(self, pred: DevTensor, out: DevTensor, slot0: int, index: int, explicit_idx: int, count: int):
        """The ltb_op_mt_paste descriptor of `count` jobs: full frames into out (count, H, W, 3), or for a frame-free avatar the
        blended crop boxes into out (count, rh_max, rw_max, 3)."""
        op = _capi.MtPasteOp()
        op.coords, op.crop, op.masks, op.mask_off = self.coords.ptr, self.crop.ptr, self.masks.ptr, self.mask_off.ptr
        if self.frames_resident:
            op.frames = self.frames.ptr
        else:
            op.body, (op.region_h, op.region_w) = self.body.ptr, self.region_max
        op.pred, op.out = pred.ptr, out.ptr
        op.nf, op.H, op.W = self.n, self.H, self.W
        op.index, op.explicit_idx, op.slot0, op.count = index, explicit_idx, slot0, count
        op.pred_hw = self.lat_hw * 8
        return op

    def out_shape(self, count: int) -> tuple:
        """Shape of the paste output of `count` jobs: full frames, or crop boxes packed at region_max for a frame-free avatar."""
        return (count, self.H, self.W, 3) if self.frames_resident else (count, *self.region_max, 3)


class MuseTalkSession:
    """One avatar stream at a fixed batch size: the captured UNet + VAE-decode graph and the paste-back buffers."""

    def __init__(self, model: MuseTalkModel, avatar: MuseTalkAvatar, batch: int, keep_taps: bool = False, ctx: Optional[Ctx] = None,
                 paste_only: bool = False):
        """ctx: the session's own stream + scratch (created here unless given).  Sessions never share a ctx: the reference
        opens up to max_session of them concurrently (app.py:76-100), each driven by its own three threads, and capturing /
        synchronising a stream another session is using would corrupt both.
        paste_only: no network graph and no activation arena — only paste_pred() works (cross-session mode: the UNet / VAE pass of
        this session's frames runs in a shared MuseTalkBatchSession)."""
        self.model, self.avatar, self.B = model, avatar, int(batch)
        self._own_ctx = ctx is None
        self._paste_ctx = None
        self.graph = None
        if paste_only:
            self.ctx, self._own_ctx = None, False
            return
        ctx = self.ctx = Ctx() if ctx is None else ctx
        B, hw = self.B, avatar.lat_hw
        self.builder = Builder(ctx)
        self.d_index = ctx.alloc((4,), np.int32, zero=True)
        self.audio_in = ctx.alloc((B, KEY_PAD, model.ucfg.cross_attention_dim), np.float16, zero=True)
        self.audio_pe = ctx.alloc((B * KEY_PAD, model.ucfg.cross_attention_dim), np.float16, zero=True)
        self.latents16 = ctx.alloc((B, hw, hw, 16), np.float16, zero=True)
        self.image_u8 = ctx.alloc((B, hw * 8, hw * 8, 3), np.uint8, zero=True)
        self.frames_out = ctx.alloc(avatar.out_shape(B), np.uint8, zero=True)
        self.taps = {} if keep_taps else None
        self._paste_ctx = None
        self._audio_host = np.zeros((B, KEY_PAD, model.ucfg.cross_attention_dim), np.float16)

        def emit():
            ctx.gather_rows(avatar.latents, avatar.latents.shape[0], self.d_index, B, hw * hw * 16, self.latents16)
            ctx.eltwise(self.audio_in, model.pe, self.audio_in.rows * self.audio_in.C, KEY_PAD * self.audio_in.C, 0, self.audio_pe)
            self.pred16 = model.emit_unet(self.builder, self.latents16, self.audio_pe, self.taps)
            self.image16 = model.emit_vae_decode(self.builder, self.pred16, self.image_u8, self.taps)

        emit()                       # eager pass: allocates every intermediate and warms the kernels up
        ctx.sync()
        temps, self.builder.temps = self.builder.temps, []
        self.builder.new = _Replay(temps)   # the captured pass reuses exactly the same buffers, in the same order
        with ctx.capture() as cap:
            emit()
        self.graph = cap.graph
        self.graph_launches = None

    # ---- MuseReal.inference_batch (musetalk_avatar.py:130-152)
    def infer_async(self, index: int, audio_feats: Optional[np.ndarray] = None):
        if self.graph is None:
            raise RuntimeError("MuseTalkSession: paste-only (or closed) session has no network graph")
        if audio_feats is not None:
            a = np.asarray(audio_feats)
            if a.shape != (self.B, 50, self._audio_host.shape[2]):
                raise ValueError(f"audio features must be ({self.B},50,{self._audio_host.shape[2]}), got {a.shape}")
            self._audio_host[:, :50] = a.astype(np.float16)
            self.ctx.h2d(self.audio_in, self._audio_host, sync=False)
        self.ctx.set_i32(self.d_index, index)
        self.graph.launch()

    def infer(self, index: int, audio_feats: Optional[np.ndarray] = None, want_pred: bool = True):
        with self.ctx.lock:       # h2d -> index -> graph -> d2h is one critical section (inference vs process_frames thread)
            self.infer_async(index, audio_feats)
            if want_pred:
                return self.ctx.download(self.image_u8)          # uint8 (B,hw*8,hw*8,3) BGR, as vae.decode_latents returns
            self.ctx.sync()
            return None

    # ---- MuseReal.paste_back_frame (musetalk_avatar.py:154-164)
    def _need_frames(self, what: str):
        if not self.avatar.frames_resident:
            raise LtbError(f"{what}: the avatar was created frame-free (frames_resident=False); use the *_region methods")

    def _paste_op(self, pred: DevTensor, slot0: int, index: int, explicit_idx: int, count: int):
        self.ctx.mt_paste(self.avatar.paste_op(pred, self.frames_out, slot0, index, explicit_idx, count))

    def paste(self, slot: int, idx: int) -> np.ndarray:
        self._need_frames("paste")
        if not (0 <= slot < self.B and 0 <= idx < self.avatar.n):
            raise ValueError("paste: slot / idx out of range")
        with self.ctx.lock:
            self._paste_op(self.image_u8, slot, 0, idx, 1)
            one = DevTensor(self.frames_out.ptr, (self.avatar.H, self.avatar.W, 3), np.uint8)
            return self.ctx.download(one)

    def paste_pred(self, pred_u8: np.ndarray, idx: int) -> np.ndarray:
        """paste_back_frame for a host prediction (S,S,3) uint8 — the reference's exact argument.  Runs on its own small
        ctx (stream + scratch prediction + output frame): process_frames calls it while inference_batch is in flight."""
        self._need_frames("paste_pred")
        return self._paste_pred(pred_u8, idx, "paste_pred")

    def paste_pred_region(self, pred_u8: np.ndarray, idx: int):
        """paste_pred for a frame-free avatar: -> (the blended crop box uint8 (y_e-y_s, x_e-x_s, 3), box (y_s, y_e, x_s, x_e))."""
        if self.avatar.frames_resident:
            raise LtbError("paste_pred_region: the avatar holds full frames; use paste_pred")
        region = self._paste_pred(pred_u8, idx, "paste_pred_region")
        box = self.avatar.box(idx)
        return region[:box[1] - box[0], :box[3] - box[2]], box

    def _paste_pred(self, pred_u8: np.ndarray, idx: int, what: str) -> np.ndarray:
        S = self.avatar.lat_hw * 8
        pred_u8 = np.ascontiguousarray(pred_u8, np.uint8)
        if pred_u8.shape != (S, S, 3):
            raise ValueError(f"{what}: prediction must be ({S},{S},3) uint8, got {pred_u8.shape}")
        if not 0 <= idx < self.avatar.n:
            raise ValueError(f"{what}: idx out of range")
        if self._paste_ctx is None:
            self._paste_ctx = Ctx()
            self._pred_scratch = self._paste_ctx.alloc((1, S, S, 3), np.uint8)
            self._paste_out = self._paste_ctx.alloc(self.avatar.out_shape(1)[1:], np.uint8)
        pc = self._paste_ctx
        with pc.lock:
            pc.h2d(self._pred_scratch, pred_u8, sync=False)
            pc.mt_paste(self.avatar.paste_op(self._pred_scratch, self._paste_out, 0, 0, idx, 1))
            return pc.download(self._paste_out)

    def paste_batch_async(self, index: int):
        self._paste_op(self.image_u8, 0, index, -1, self.B)

    def paste_batch_region(self, index: int, out: Optional[np.ndarray] = None):
        """paste_batch for a frame-free avatar: -> (regions uint8 (B, rh_max, rw_max, 3), boxes); slot i's blended crop box is
        regions[i, :y_e-y_s, :x_e-x_s] of frame mirror_index(n, index + i)."""
        if self.avatar.frames_resident:
            raise LtbError("paste_batch_region: the avatar holds full frames; use paste_batch")
        a = self.avatar
        with self.ctx.lock:
            self.paste_batch_async(index)
            regions = self.ctx.download(self.frames_out, out)
        return regions, [a.box(mirror_index(a.n, index + i)) for i in range(self.B)]

    def paste_batch(self, index: int, out: Optional[np.ndarray] = None) -> np.ndarray:
        self._need_frames("paste_batch")
        with self.ctx.lock:
            self.paste_batch_async(index)
            return self.ctx.download(self.frames_out, out)

    def close(self):
        """Release the session's graph, streams and device buffers (one WebRTC connection = one session: no HBM leak)."""
        if getattr(self, "graph", None) is not None:
            self.graph.close()
            self.graph = None
        if self._paste_ctx is not None:
            self._paste_ctx.close()
            self._paste_ctx = None
        if self._own_ctx and self.ctx is not None:
            self.ctx.close()
        self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def step_async(self, index: int):
        """Everything resident (audio features already on the device): UNet + VAE decode + blend paste-back."""
        self._need_frames("step_async")
        self.infer_async(index, None)
        self.paste_batch_async(index)


class MuseTalkBatchSession:
    """Cross-session batching for MuseTalk (SURVEY 8(f) rank 1, the MuseTalk twin of ltb_w2l_infer_slots): up to G sessions x Bs
    frames run as ONE captured PE + UNet + VAE-decode graph of batch G*Bs.  A *group request* is (avatar, first frame index,
    Whisper features (Bs, 50, 384) or None): group g's latents are gathered from ITS avatar's table (mirror-indexed, outside the
    graph, so any session may occupy any group of any round), its features occupy rows [g*Bs, (g+1)*Bs) of audio_in.
    The reference serves every session with its own B-frame forward (avatars/musetalk_avatar.py:130-152 under app.py:76-100's
    max_session connections); at batch 8 the UNet is launch-latency bound on a B200 (64 M-tiles per layer), so four sessions per
    launch cost far less than four launches.  `batch` / `infer_slots` make it a mux for plugin.batcher.CrossSessionBatcher."""

    def __init__(self, model: MuseTalkModel, lat_hw: int, groups: int, frames_per_session: int, ctx: Optional[Ctx] = None):
        self.model, self.lat_hw, self.Bs, self.G = model, int(lat_hw), int(frames_per_session), int(groups)
        self.batch = self.G                                  # CrossSessionBatcher: requests per engine call
        self.B = B = self.G * self.Bs
        self._own_ctx = ctx is None
        ctx = self.ctx = Ctx() if ctx is None else ctx
        Bs, hw, cad = self.Bs, self.lat_hw, model.ucfg.cross_attention_dim
        self.builder = Builder(ctx)
        self._d_index = ctx.alloc((4 * self.G,), np.int32, zero=True)
        self.d_index = [DevTensor(self._d_index.ptr + 16 * g, (4,), np.int32) for g in range(self.G)]
        self.audio_in = ctx.alloc((B, KEY_PAD, cad), np.float16, zero=True)
        self.audio_in_of = [DevTensor(self.audio_in.ptr + g * Bs * KEY_PAD * cad * 2, (Bs, KEY_PAD, cad)) for g in range(self.G)]
        self.audio_pe = ctx.alloc((B * KEY_PAD, cad), np.float16, zero=True)
        self.latents16 = ctx.alloc((B, hw, hw, 16), np.float16, zero=True)
        self.latents16_of = [DevTensor(self.latents16.ptr + g * Bs * hw * hw * 16 * 2, (Bs, hw, hw, 16)) for g in range(self.G)]
        self.image_u8 = ctx.alloc((B, hw * 8, hw * 8, 3), np.uint8, zero=True)
        self._frames_out: Dict[tuple, DevTensor] = {}
        self._audio_host = np.zeros((B, KEY_PAD, cad), np.float16)

        def emit():
            ctx.eltwise(self.audio_in, model.pe, self.audio_in.rows * self.audio_in.C, KEY_PAD * self.audio_in.C, 0, self.audio_pe)
            self.pred16 = model.emit_unet(self.builder, self.latents16, self.audio_pe, None)
            self.image16 = model.emit_vae_decode(self.builder, self.pred16, self.image_u8, None)

        emit()
        ctx.sync()
        temps, self.builder.temps = self.builder.temps, []
        self.builder.new = _Replay(temps)
        with ctx.capture() as cap:
            emit()
        self.graph = cap.graph

    def _check(self, requests):
        if not 1 <= len(requests) <= self.G:
            raise ValueError(f"1..{self.G} group requests per call, got {len(requests)}")
        for r in requests:
            if r[0].lat_hw != self.lat_hw:
                raise ValueError("avatar latent size does not match the batch session")

    def infer_async(self, requests: Sequence[tuple]):
        """requests[g] = (MuseTalkAvatar, first frame index, features (Bs,50,384) | None = resident in audio_in_of[g])."""
        self._check(requests)
        ctx, Bs, row = self.ctx, self.Bs, self.lat_hw * self.lat_hw * 16
        stage = False
        for g, (av, index, feats) in enumerate(requests):
            if feats is not None:
                a = np.asarray(feats)
                if a.shape != (Bs, 50, self._audio_host.shape[2]):
                    raise ValueError(f"group features must be ({Bs},50,{self._audio_host.shape[2]}), got {a.shape}")
                self._audio_host[g * Bs:(g + 1) * Bs, :50] = a.astype(np.float16)
                stage = True
            ctx.set_i32(self.d_index[g], int(index))
            ctx.gather_rows(av.latents, av.latents.shape[0], self.d_index[g], Bs, row, self.latents16_of[g])
        if stage:
            n = len(requests) * Bs
            ctx.h2d(DevTensor(self.audio_in.ptr, (n,) + self.audio_in.shape[1:]), self._audio_host[:n], sync=False)
        self.graph.launch()

    def infer_groups(self, requests: Sequence[tuple]) -> List[np.ndarray]:
        """-> per request its (Bs, S, S, 3) uint8 BGR predictions (what MuseReal.inference_batch returns for that session)."""
        with self.ctx.lock:
            self.infer_async(requests)
            n = len(requests) * self.Bs
            S = self.lat_hw * 8
            pred = self.ctx.download(DevTensor(self.image_u8.ptr, (n, S, S, 3), np.uint8))
        return [pred[g * self.Bs:(g + 1) * self.Bs] for g in range(len(requests))]

    infer_slots = infer_groups

    def _out(self, g: int, av: MuseTalkAvatar) -> DevTensor:
        shape = av.out_shape(self.Bs)
        key = (g, *shape)
        if key not in self._frames_out:
            self._frames_out[key] = self.ctx.alloc(shape, np.uint8, zero=True)
        return self._frames_out[key]

    def paste_async(self, requests: Sequence[tuple]) -> List[DevTensor]:
        """Blend paste-back of every group's predictions into its own avatar frames (device resident; MuseReal.paste_back_frame x Bs).
        A frame-free avatar's group gets its blended crop boxes instead, (Bs, rh_max, rw_max, 3) (see MuseTalkAvatar.box)."""
        self._check(requests)
        outs = []
        for g, (a, index, _f) in enumerate(requests):
            out = self._out(g, a)
            self.ctx.mt_paste(a.paste_op(self.image_u8, out, g * self.Bs, int(index), -1, self.Bs))
            outs.append(out)
        return outs

    def step_async(self, requests: Sequence[tuple]):
        self.infer_async(requests)
        self.paste_async(requests)

    def step(self, requests: Sequence[tuple]) -> List[np.ndarray]:
        """One batched round: returns, per session, its Bs composited frames (Bs, H, W, 3) uint8 — for a frame-free avatar its Bs
        blended crop boxes (Bs, rh_max, rw_max, 3), crop box of frame mirror_index(n, index + i) = MuseTalkAvatar.box."""
        with self.ctx.lock:
            self.infer_async(requests)
            outs = [self.ctx.download(t, sync=False) for t in self.paste_async(requests)]
            self.ctx.sync()
            return outs

    def close(self):
        if getattr(self, "graph", None) is not None:
            self.graph.close()
            self.graph = None
        if self._own_ctx and self.ctx is not None:
            self.ctx.close()
        self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _Replay:
    """Hands back the buffers of the eager pass, in order, while the same op sequence is being captured."""

    def __init__(self, temps):
        self.temps, self.i = temps, 0

    def __call__(self, *shape):
        t = self.temps[self.i]
        self.i += 1
        assert t.shape == tuple(shape), (t.shape, shape)
        return t


def encode_avatar_latents(model: MuseTalkModel, images_u8: np.ndarray) -> np.ndarray:
    """GPU get_latents_for_unet for a stack of (n,256,256,3) uint8 BGR crops -> (n,8,h,w) float16 (latents.pt content,
    avatars/musetalk/genavatar.py:126-128 with the deterministic latent_dist.mode())."""
    ctx = model.ctx
    imgs = np.ascontiguousarray(images_u8, np.uint8)
    n, H, W, _ = imgs.shape
    d_img = ctx.upload(imgs)
    out = ctx.alloc((n, H // 8, W // 8, 16), np.float16, zero=True)
    b = Builder(ctx)
    model.emit_vae_encode(b, d_img, out)
    lat = ctx.download(out)
    for t in b.temps:
        ctx.free(t)
    ctx.free(d_img)
    ctx.free(out)
    return np.ascontiguousarray(lat[..., :8].transpose(0, 3, 1, 2))
