"""GPU: every kernel wrapper of geo4d_b200.ops checked at the shapes, strides and scalars the product actually uses,
plus targeted edge and adversarial cases, against plain high-precision references.

Part A records every call the full-width U-Net (benchmark latent 1x20x16x40x64, context 77 + 16*16 tokens), the
full-size VAE (decode + confidence head and encode at 320x512) and the image-token resampler make, deduplicates the
call signatures (tensor shapes / strides / dtypes, scalar arguments, which optional operands are present) and
replays each unique signature on seeded inputs laid out with the same strides, against an fp64 torch reference of
the same op computed from the same bf16-rounded inputs.  It also records statistics of the ACTUAL activations --
the largest |mean| / std of a GroupNorm group and the largest per-row logit spread of an attention call -- and
asserts that the adversarial cases of part B reach at least those values.  The weights are seeded, not a
checkpoint, so those statistics are a floor for what real activations reach, not a bound.

Part B: softmax / transpose / GroupNorm (fused and two-kernel paths) / attention needle and peaked cases / temporal
attention / DDIM update / tap-GEMM addressing edges, against fp64 references.

Bars (the ones tests/test_ops_gpu.py states): bf16 output 2.5e-3 relative L2 (one bf16 rounding of the result),
fp32 output 1e-5, attention 4e-3 (P is rounded to bf16 before PV), data movement exact.

The reference helpers are plain torch and device-agnostic; tests/test_kernel_sweep_cpu.py checks each of them
against torch's own op on the CPU, so a wrong reference cannot make a wrong kernel pass.
"""
import inspect
import time
from collections import defaultdict

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

BF16_TOL = 2.5e-3     # one bf16 rounding of the output
FP32_TOL = 1e-5       # fp32 accumulation order of a GEMM with an fp32 output
ATTN_TOL = 4e-3       # P is rounded to bf16 before the PV product
BF16_ULP = 2.0 ** -8  # one bf16 rounding, elementwise (round-to-nearest is within half of this)

# adversarial ranges of part B; part A asserts that the production activations stay inside them
GN_OFFSET_RATIOS = (0.0, 16.0, 64.0)   # |mean| / std of every group of the offset-dominated GroupNorm inputs
PEAKED_LOGIT_SPREAD = 32.0             # the peaked attention cases reach at least this max-min logit spread per row

WRAPPERS = ("linear", "conv3x3", "temporal_conv3", "bmm_nt", "groupnorm", "layernorm", "attention",
            "cross_attention2", "temporal_attention", "softmax_rows", "transpose_bf16", "concat_rows", "upsample2x",
            "im2col_s2")


def rel_l2(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / (b.norm() + 1e-30))


# ================================================================================================ references
# Every reference takes the kernel's operands (bf16 / fp32 tensors, any device) and returns float64.
def ref_linear(x, w, bias=None, act=0, residual=None, alpha=1.0):
    """act: 0 none, 1 SiLU, 2 GEGLU (weight rows interleaved in blocks of [32 value | 32 gate]), 3 GELU (erf)."""
    y = alpha * (x.double() @ w.double().t())
    if bias is not None:
        y = y + bias.double()
    if act == 1:
        y = F.silu(y)
    elif act == 3:
        y = F.gelu(y)
    elif act == 2:
        blk = y.reshape(y.shape[0], -1, 2, 32)
        y = (blk[:, :, 0] * F.gelu(blk[:, :, 1])).reshape(y.shape[0], -1)
    if residual is not None:
        y = y + residual.double()
    return y


def _tap_sum(x4, w_taps, taps):
    """x4 [N, H, W, C] -> sum over taps (dx, dy) of x[n, y+dy, x+dx] @ w^T with zero padding (float64)."""
    N, H, W, _ = x4.shape
    xp = F.pad(x4.double(), (0, 0, 1, 1, 1, 1))
    out = 0
    for (dx, dy), w in zip(taps, w_taps):
        out = out + xp[:, 1 + dy:1 + dy + H, 1 + dx:1 + dx + W, :] @ w.double().t()
    return out


def ref_conv3x3(x, N, H, W, w9, bias=None, row_bias=None, rows_per_bias=0, residual=None):
    taps = [(dx, dy) for dy in (-1, 0, 1) for dx in (-1, 0, 1)]
    y = _tap_sum(x.reshape(N, H, W, -1), list(w9), taps).reshape(N * H * W, -1)
    if bias is not None:
        y = y + bias.double()
    if row_bias is not None:
        y = y + row_bias.double()[torch.arange(N * H * W, device=x.device) // rows_per_bias]
    if residual is not None:
        y = y + residual.double()
    return y


def ref_temporal_conv3(x, B, T, HW, w3, bias=None, residual=None):
    taps = [(0, -1), (0, 0), (0, 1)]      # the frame axis plays the role of H
    y = _tap_sum(x.reshape(B, T, HW, -1), list(w3), taps).reshape(B * T * HW, -1)
    if bias is not None:
        y = y + bias.double()
    if residual is not None:
        y = y + residual.double()
    return y


def ref_bmm_nt(a, b, alpha=1.0):
    return alpha * torch.einsum("bmk,bnk->bmn", a.double(), b.double())


def ref_groupnorm(x, S, rows, gamma, beta, eps, silu):
    C = x.shape[1]
    g = x.double().reshape(S, rows, 32, C // 32)
    mean = g.mean(dim=(1, 3), keepdim=True)
    var = ((g - mean) ** 2).mean(dim=(1, 3), keepdim=True)
    y = ((g - mean) / torch.sqrt(var + eps)).reshape(S * rows, C) * gamma.double() + beta.double()
    return F.silu(y) if silu else y


def ref_layernorm(x, gamma, beta, eps):
    x = x.double()
    mean = x.mean(1, keepdim=True)
    var = ((x - mean) ** 2).mean(1, keepdim=True)
    return (x - mean) / torch.sqrt(var + eps) * gamma.double() + beta.double()


def ref_attention(q, k, v, B, H, Lq, Lk, kv_batch_div=1, scale=0.125):
    """q [B*Lq, >=H*64] rows, k / v [ceil(B/div)*Lk, >=H*64] rows -> [B*Lq, H*64] float64 (one batch at a time)."""
    inner = H * 64
    out = []
    for b in range(B):
        bk = b // kv_batch_div
        qh = q[b * Lq:(b + 1) * Lq, :inner].double().reshape(Lq, H, 64).transpose(0, 1)
        kh = k[bk * Lk:(bk + 1) * Lk, :inner].double().reshape(Lk, H, 64).transpose(0, 1)
        vh = v[bk * Lk:(bk + 1) * Lk, :inner].double().reshape(Lk, H, 64).transpose(0, 1)
        p = torch.softmax(qh @ kh.transpose(1, 2) * scale, dim=-1)
        out.append((p @ vh).transpose(0, 1).reshape(Lq, inner))
    return torch.cat(out, 0)


def ref_temporal_attention(q, k, v, B, T, HW, heads, scale=0.125):
    """attention over the T frames of each pixel: rows are (b, t, p)."""
    inner = heads * 64

    def seq(x):
        return x[:, :inner].double().reshape(B, T, HW, heads, 64).permute(0, 2, 3, 1, 4)   # [B, HW, heads, T, 64]
    p = torch.softmax(seq(q) @ seq(k).transpose(-1, -2) * scale, dim=-1)
    return (p @ seq(v)).permute(0, 3, 1, 2, 4).reshape(B * T * HW, inner)


def ref_softmax_rows(s):
    return torch.softmax(s.double(), dim=1)


def ref_transpose(x, batch, R, Cc):
    return x[:batch * R, :Cc].reshape(batch, R, Cc).transpose(1, 2)


def ref_upsample2x(x, N, H, W):
    return x.reshape(N, H, W, -1).repeat_interleave(2, 1).repeat_interleave(2, 2).reshape(N * 4 * H * W, -1)


def ref_im2col_s2(x, N, H, W, pad_before, Ho, Wo):
    C = x.shape[1]
    xp = torch.zeros(N, H + 3, W + 3, C, dtype=x.dtype, device=x.device)
    xp[:, pad_before:pad_before + H, pad_before:pad_before + W] = x.reshape(N, H, W, C)
    cols = [xp[:, ky:ky + 2 * Ho:2, kx:kx + 2 * Wo:2] for ky in range(3) for kx in range(3)]
    return torch.stack(cols, 3).reshape(N * Ho * Wo, 9 * C)


def ref_ddim(x, v, coef_row, noise=None):
    """v-parameterised DDIM update; coef row {sa, s1, rescale, sqrt_a_prev, dir, sigma} -> (x_prev, pred_x0)."""
    sa, s1, rs, sap, dr, sg = [float(c) for c in coef_row]
    x, v = x.double(), v.double()
    e_t = sa * v + s1 * x
    x0 = (sa * x - s1 * v) * rs
    xp = sap * x0 + dr * e_t
    if noise is not None:
        xp = xp + sg * noise.double()
    return xp, x0


# ================================================================================================ part A: recording
class TSpec:
    """shape / stride / dtype of a recorded tensor argument (stride(0) is its row pitch)."""

    def __init__(self, t):
        self.shape, self.stride, self.dtype = tuple(t.shape), tuple(t.stride()), t.dtype

    def key(self):
        return ("T", self.shape, self.stride, str(self.dtype).replace("torch.", ""))

    def make(self, gen, scale=1.0, offset=0.0):
        """seeded values in a buffer laid out with the recorded strides (views such as qkv[:, :inner] included)"""
        span = 1 + sum((s - 1) * st for s, st in zip(self.shape, self.stride))
        buf = torch.randn(span, device="cuda", generator=gen) * scale + offset
        return buf.to(self.dtype).as_strided(self.shape, self.stride)

    def empty(self):
        span = 1 + sum((s - 1) * st for s, st in zip(self.shape, self.stride))
        return torch.full((span,), float("nan"), device="cuda", dtype=self.dtype).as_strided(self.shape, self.stride)


def _describe(v):
    if isinstance(v, torch.Tensor):
        return TSpec(v)
    return v


def _sig_key(name, bound):
    return (name,) + tuple((k, v.key() if isinstance(v, TSpec) else v) for k, v in bound.items())


def _short(bound):
    parts = []
    for k, v in bound.items():
        if isinstance(v, TSpec):
            pitch = v.stride[-2] if len(v.shape) >= 2 else 1
            parts.append(f"{k}={'x'.join(map(str, v.shape))}@{pitch}{'' if v.dtype == torch.bfloat16 else ':' + str(v.dtype)[6:]}")
        elif v is not None and k != "workspace":
            parts.append(f"{k}={v}")
    return " ".join(parts)


def _gn_ratio(x, S, rows):
    g = x[:S * rows].double().reshape(S, rows, 32, -1)
    mean = g.mean(dim=(1, 3))
    std = g.std(dim=(1, 3), unbiased=False)
    return float((mean.abs() / std.clamp_min(1e-30)).max())


def _logit_spread(q, k, nq, Lk, H, scale):
    """max over a sample of query rows (first batch, every head) of max - min of the scaled logits"""
    rows = torch.linspace(0, nq - 1, min(nq, 64), device=q.device).long()
    qs = q[rows, :H * 64].double().reshape(-1, H, 64).transpose(0, 1)
    ks = k[:Lk, :H * 64].double().reshape(Lk, H, 64).transpose(0, 1)
    s = qs @ ks.transpose(1, 2) * scale
    return float((s.amax(-1) - s.amin(-1)).max())


class Recorder:
    def __init__(self):
        self.sigs = {}                      # key -> (name, bound specs)
        self.calls = defaultdict(int)
        self.stats = {"gn_ratio": (0.0, ""), "logit_spread": (0.0, "")}

    def _stat(self, key, value, where):
        if value > self.stats[key][0]:
            self.stats[key] = (value, where)

    def wrap(self, name, fn):
        sig = inspect.signature(fn)

        def recorded(*args, **kwargs):
            b = sig.bind(*args, **kwargs)
            b.apply_defaults()
            bound = {k: _describe(v) for k, v in b.arguments.items()}
            self.sigs.setdefault(_sig_key(name, bound), (name, bound))
            self.calls[name] += 1
            a = b.arguments
            if name == "groupnorm":
                self._stat("gn_ratio", _gn_ratio(a["x"], a["num_stats"], a["rows_per_stat"]), _short(bound))
            elif name == "attention":
                self._stat("logit_spread", _logit_spread(a["q"], a["k"], a["Lq"], a["Lk"], a["H"], a["scale"]),
                           _short(bound))
            elif name == "cross_attention2":
                for kk, L in (("k", a["Lk"]), ("k2", a["Lk2"])):
                    self._stat("logit_spread", _logit_spread(a["q"], a[kk], a["Lq"], L, a["H"], a["scale"]),
                               _short(bound))
            elif name == "temporal_attention":
                # the T keys of pixel 0 of the first clip: rows t * HW
                T, HW = a["T"], a["HW"]
                rows = torch.arange(T, device=a["q"].device) * HW
                self._stat("logit_spread", _logit_spread(a["q"][rows], a["k"][rows], T, T, a["heads"], a["scale"]),
                           _short(bound))
            return fn(*args, **kwargs)
        return recorded


@pytest.fixture(scope="module")
def production_calls(cuda_device, golden_dir):
    """Record every ops.* wrapper call of one U-Net forward, one VAE decode + encode and one resampler forward."""
    import os
    from geo4d_b200 import ops
    from oracle import unet as ou, vae as ov
    from tests.test_unet_gpu import make_unet
    from tests.test_vae_gpu import make_vae
    from geo4d_b200.resampler import Resampler
    from oracle.gen_golden_resampler import seeded_state
    t0 = time.time()
    rec = Recorder()
    sd = ou.init_params(ou.param_shapes(ou.UNetConfig()), seed=21)
    net = make_unet(dict(model_channels=320, context_dim=1024, temporal_length=16), sd, cuda_device)
    del sd
    vsd = ou.init_params(ov.param_shapes(ov.VAEConfig()), seed=31)
    vae = make_vae(dict(ch=128, adaptor_ch=128), vsd, cuda_device)
    del vsd
    gres = torch.load(os.path.join(golden_dir, "resampler_ref.pt"))
    rs = Resampler(**gres["kw"])
    rs.load_state_dict(seeded_state(gres["shapes"], seed=gres["seed"]), strict=True)
    rs = rs.to(cuda_device).prepare()
    g = torch.Generator().manual_seed(5)
    x = torch.randn(1, 20, 16, 40, 64, generator=g).to(cuda_device)
    ctx = torch.randn(1, 77 + 16 * 16, 1024, generator=g).to(cuda_device)
    z = torch.randn(1, 4, 40, 64, generator=g).to(cuda_device)
    img = torch.tanh(torch.randn(1, 3, 320, 512, generator=g)).to(cuda_device)
    tok = torch.randn(1, 257, 1280, generator=g).to(cuda_device)
    with pytest.MonkeyPatch.context() as mp:
        for name in WRAPPERS:
            mp.setattr(ops, name, rec.wrap(name, getattr(ops, name)))
        with torch.no_grad():
            net(x, torch.tensor([481], device=cuda_device), context=ctx, fs=torch.tensor([24], device=cuda_device))
            vae.decode_with_conf_adaptor(z)
            vae.encode_moments(img)
            rs(tok)
    torch.cuda.synchronize()
    del net, vae, rs
    torch.cuda.empty_cache()
    print(f"\n[kernel sweep] recorded {sum(rec.calls.values())} calls, {len(rec.sigs)} unique signatures "
          f"in {time.time() - t0:.1f} s")
    return rec


# ---------------------------------------------------------------------------------------------- replays
# Each replay builds seeded inputs with the recorded layout, runs the real wrapper and returns (error, bar).
def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _out_bar(dtype):
    return FP32_TOL if dtype == torch.float32 else BF16_TOL


def _opt(spec, g, scale=1.0):
    return None if spec is None else spec.make(g, scale)


def _ret_or_out(ret, out):
    return ret if out is None else out


def replay_linear(ops, a, g):
    x = a["x"].make(g)
    K = a["x"].shape[1]
    w = a["w"].make(g, K ** -0.5)
    bias, res = _opt(a["bias"], g), _opt(a["residual"], g)
    out = a["out"].empty() if a["out"] is not None else None
    y = ops.linear(x, w, bias, out=out, act=a["act"], residual=res, alpha=a["alpha"], out_dtype=a["out_dtype"])
    return rel_l2(y, ref_linear(x, w, bias, a["act"], res, a["alpha"])), _out_bar(y.dtype)


def replay_conv3x3(ops, a, g):
    x = a["x"].make(g)
    w9 = a["w9"].make(g, (9 * a["x"].shape[1]) ** -0.5)
    bias, rb, res = _opt(a["bias"], g), _opt(a["row_bias"], g), _opt(a["residual"], g)
    out = a["out"].empty() if a["out"] is not None else None
    y = ops.conv3x3(x, a["N"], a["H"], a["W"], w9, bias, out=out, row_bias=rb, rows_per_bias=a["rows_per_bias"],
                    residual=res, out_dtype=a["out_dtype"])
    ref = ref_conv3x3(x, a["N"], a["H"], a["W"], w9, bias, rb, a["rows_per_bias"], res)
    return rel_l2(y, ref), _out_bar(y.dtype)


def replay_temporal_conv3(ops, a, g):
    x = a["x"].make(g)
    w3 = a["w3"].make(g, (3 * a["x"].shape[1]) ** -0.5)
    bias, res = _opt(a["bias"], g), _opt(a["residual"], g)
    out = a["out"].empty() if a["out"] is not None else None
    y = ops.temporal_conv3(x, a["B"], a["T"], a["HW"], w3, bias, out=out, residual=res)
    return rel_l2(y, ref_temporal_conv3(x, a["B"], a["T"], a["HW"], w3, bias, res)), BF16_TOL


def replay_bmm_nt(ops, a, g):
    x, y = a["a"].make(g), a["b"].make(g)
    out = a["out"].empty() if a["out"] is not None else None
    o = ops.bmm_nt(x, y, out=out, alpha=a["alpha"], out_dtype=a["out_dtype"])
    return rel_l2(o, ref_bmm_nt(x, y, a["alpha"])), _out_bar(o.dtype)


def replay_groupnorm(ops, a, g):
    x = a["x"].make(g, 1.5, 0.3)
    gamma, beta = a["gamma"].make(g), a["beta"].make(g)
    out = a["out"].empty() if a["out"] is not None else None
    y = ops.groupnorm(x, a["num_stats"], a["rows_per_stat"], gamma, beta, a["eps"], a["silu"], out=out)
    return rel_l2(y, ref_groupnorm(x, a["num_stats"], a["rows_per_stat"], gamma, beta, a["eps"], a["silu"])), BF16_TOL


def replay_layernorm(ops, a, g):
    x = a["x"].make(g, 2.0, 0.5)
    gamma, beta = a["gamma"].make(g), a["beta"].make(g)
    out = a["out"].empty() if a["out"] is not None else None
    y = ops.layernorm(x, gamma, beta, a["eps"], out=out)
    return rel_l2(y, ref_layernorm(x, gamma, beta, a["eps"])), BF16_TOL


def replay_attention(ops, a, g):
    q, k, v = a["q"].make(g), a["k"].make(g), a["v"].make(g)
    B, H, Lq, Lk, div = a["B"], a["H"], a["Lq"], a["Lk"], a["kv_batch_div"]
    out = a["out"].make(g) if a["accumulate"] else a["out"].empty()
    prev = out[:, :H * 64].double().clone()
    ops.attention(q, k, v, out, B, H, Lq, Lk, kv_batch_div=div, accumulate=a["accumulate"], scale=a["scale"])
    ref = ref_attention(q, k, v, B, H, Lq, Lk, div, a["scale"])
    if a["accumulate"]:
        ref = ref + prev
    return rel_l2(out[:, :H * 64], ref), ATTN_TOL


def replay_cross_attention2(ops, a, g):
    q, k, v, k2, v2 = (a[n].make(g) for n in ("q", "k", "v", "k2", "v2"))
    B, H, Lq = a["B"], a["H"], a["Lq"]
    out = a["out"].empty()
    ops.cross_attention2(q, k, v, a["Lk"], a["div"], k2, v2, a["Lk2"], a["div2"], out, B, H, Lq, scale=a["scale"])
    ref = (ref_attention(q, k, v, B, H, Lq, a["Lk"], a["div"], a["scale"])
           + ref_attention(q, k2, v2, B, H, Lq, a["Lk2"], a["div2"], a["scale"]))
    return rel_l2(out[:, :H * 64], ref), ATTN_TOL


def replay_temporal_attention(ops, a, g):
    q, k, v = a["q"].make(g), a["k"].make(g), a["v"].make(g)
    out = a["out"].empty()
    ops.temporal_attention(q, k, v, out, a["B"], a["T"], a["HW"], a["heads"], scale=a["scale"])
    ref = ref_temporal_attention(q, k, v, a["B"], a["T"], a["HW"], a["heads"], a["scale"])
    return rel_l2(out[:, :a["heads"] * 64], ref), ATTN_TOL


def replay_softmax_rows(ops, a, g):
    s = a["scores"].make(g, 3.0)
    out = a["out"].empty() if a["out"] is not None else None
    p = ops.softmax_rows(s, out=out)
    return rel_l2(p, ref_softmax_rows(s)), BF16_TOL


def _exact(y, ref):
    return 0.0 if torch.equal(y, ref.to(y.dtype)) else float("inf")


def replay_transpose_bf16(ops, a, g):
    x = a["x"].make(g)
    out = a["out"].empty() if a["out"] is not None else None
    y = ops.transpose_bf16(x, a["batch"], a["R"], a["Cc"], out=out)
    return _exact(y, ref_transpose(x, a["batch"], a["R"], a["Cc"])), 0.0


def replay_concat_rows(ops, a, g):
    x, y = a["a"].make(g), a["b"].make(g)
    out = a["out"].empty() if a["out"] is not None else None
    o = ops.concat_rows(x, y, out=out)
    return _exact(o, torch.cat([x, y], 1)), 0.0


def replay_upsample2x(ops, a, g):
    x = a["x"].make(g)
    out = a["out"].empty() if a["out"] is not None else None
    y = ops.upsample2x(x, a["N"], a["H"], a["W"], out=out)
    return _exact(y, ref_upsample2x(x, a["N"], a["H"], a["W"])), 0.0


def replay_im2col_s2(ops, a, g):
    x = a["x"].make(g)
    out = a["out"].empty() if a["out"] is not None else None
    y = ops.im2col_s2(x, a["N"], a["H"], a["W"], a["pad_before"], a["Ho"], a["Wo"], out=out)
    return _exact(y, ref_im2col_s2(x, a["N"], a["H"], a["W"], a["pad_before"], a["Ho"], a["Wo"])), 0.0


REFERENCES = {
    "linear": replay_linear, "conv3x3": replay_conv3x3, "temporal_conv3": replay_temporal_conv3,
    "bmm_nt": replay_bmm_nt, "groupnorm": replay_groupnorm, "layernorm": replay_layernorm,
    "attention": replay_attention, "cross_attention2": replay_cross_attention2,
    "temporal_attention": replay_temporal_attention, "softmax_rows": replay_softmax_rows,
    "transpose_bf16": replay_transpose_bf16, "concat_rows": replay_concat_rows, "upsample2x": replay_upsample2x,
    "im2col_s2": replay_im2col_s2,
}


def test_every_production_call_matches_its_reference(production_calls):
    """Part A: each unique production signature, replayed on seeded inputs with the same strides."""
    from geo4d_b200 import ops
    t0 = time.time()
    rec = production_calls
    called = sorted(rec.calls)
    missing = [n for n in called if n not in REFERENCES]
    assert not missing, f"wrappers called by the forwards without a reference in this file: {missing}"
    per_op = defaultdict(lambda: [0, -1.0, None])
    failures = []
    for i, (key, (name, bound)) in enumerate(sorted(rec.sigs.items(), key=lambda kv: repr(kv[0]))):
        err, bar = REFERENCES[name](ops, bound, _gen(1000 + i))
        torch.cuda.synchronize()
        row = per_op[name]
        row[0] += 1
        if err > row[1]:
            row[1], row[2] = err, _short(bound)
        if not err <= bar:
            failures.append(f"{name} [{_short(bound)}]: error {err:.3e} > {bar:.1e}")
    print(f"\n{'wrapper':<20}{'calls':>7}{'unique':>8}{'worst err':>12}  worst signature")
    for name in WRAPPERS:
        if name in per_op:
            n, worst, where = per_op[name]
            print(f"{name:<20}{rec.calls[name]:>7}{n:>8}{worst:>12.3e}  {where}")
    gn, gn_where = rec.stats["gn_ratio"]
    sp, sp_where = rec.stats["logit_spread"]
    print(f"GroupNorm max |mean|/std of a group: {gn:.3f}  ({gn_where})")
    print(f"attention max logit spread of a row: {sp:.3f}  ({sp_where})")
    print(f"replayed {len(rec.sigs)} signatures in {time.time() - t0:.1f} s")
    assert not failures, "\n".join(failures)
    assert sorted(per_op) == sorted(WRAPPERS), f"wrappers never called: {sorted(set(WRAPPERS) - set(per_op))}"
    # the adversarial cases of part B must reach what the production activations reach
    assert gn <= max(GN_OFFSET_RATIOS), f"GroupNorm |mean|/std {gn:.2f} above the tested {max(GN_OFFSET_RATIOS)}"
    assert sp <= PEAKED_LOGIT_SPREAD, f"logit spread {sp:.2f} above the tested {PEAKED_LOGIT_SPREAD}"


# ================================================================================================ part B
@pytest.mark.parametrize("rows,cols,pad", [(37, 4, 0), (37, 4, 4), (1001, 2560, 0), (13, 4100, 12)])
def test_softmax_rows_edges(cuda_device, rows, cols, pad):
    from geo4d_b200 import ops
    g = _gen(rows + cols)
    buf = torch.randn(rows, cols + pad, device="cuda", generator=g) * 4
    s = buf[:, :cols]                                          # lds = cols + pad
    s[0, cols // 2] = 80.0 + float(s[0].max())                 # one dominant logit
    s[1 % rows].fill_(3.25)                                    # a constant row
    s[2 % rows] = s[2 % rows] - 1e4                            # large negative values
    p = ops.softmax_rows(s)
    ref = ref_softmax_rows(s)
    # within one bf16 rounding of the fp64 probability (the tiny absolute term only matters near fp32 underflow)
    bad = ((p.double() - ref).abs() > BF16_ULP * ref + 1e-37).nonzero()
    assert bad.numel() == 0, f"{bad.shape[0]} entries off, first {bad[:4].tolist()}"


@pytest.mark.parametrize("batch,R,Cc,ldin", [(1, 45, 70, 72), (3, 33, 31 * 8, 31 * 8 + 40), (2, 2560, 512, 1536)])
def test_transpose_bf16_edges(cuda_device, batch, R, Cc, ldin):
    from geo4d_b200 import ops
    x = torch.randn(batch * R, ldin, device="cuda", generator=_gen(R)).bfloat16()
    y = ops.transpose_bf16(x[:, :Cc], batch, R, Cc)
    assert torch.equal(y, ref_transpose(x, batch, R, Cc))


@pytest.fixture(params=["fused", "two-kernel"])
def gn_path(request, cuda_device):
    from geo4d_b200 import ops
    lib = ops.lib()
    lib.geo4d_debug_groupnorm_two_kernels(1 if request.param == "two-kernel" else 0)
    try:
        yield request.param
    finally:
        lib.geo4d_debug_groupnorm_two_kernels(0)


@pytest.mark.parametrize("ratio", GN_OFFSET_RATIOS)
@pytest.mark.parametrize("S,rows,C,silu,eps", [
    (2, 1000, 32, True, 1e-5), (3, 77, 320, False, 1e-6), (16, 160, 2560, True, 1e-5), (16, 40, 2560, True, 1e-5),
    (16, 2560, 320, True, 1e-5), (1, 40960, 320, True, 1e-5),      # U-Net: per-frame and per-clip statistics
    (1, 163840, 128, True, 1e-6),                                   # VAE at 320x512
])
def test_groupnorm_offset_dominated(gn_path, S, rows, C, silu, eps, ratio):
    """E[x^2] - mean^2 in fp32 cancels when |mean| >> std: inputs whose every group has |mean| / std = ratio."""
    from geo4d_b200 import ops
    g = _gen(S * 7 + C + int(ratio))
    std = 0.5 + torch.rand(S, 1, 32, 1, device="cuda", generator=g)               # per group
    sign = torch.where(torch.rand(S, 1, 32, 1, device="cuda", generator=g) < 0.5, -1.0, 1.0)
    x = (torch.randn(S, rows, 32, C // 32, device="cuda", generator=g) * std + sign * ratio * std)
    x = x.reshape(S * rows, C).bfloat16()
    gamma = torch.randn(C, device="cuda", generator=g)
    beta = torch.randn(C, device="cuda", generator=g)
    assert _gn_ratio(x, S, rows) >= 0.95 * ratio
    y = ops.groupnorm(x, S, rows, gamma, beta, eps, silu)
    y2 = ops.groupnorm(x, S, rows, gamma, beta, eps, silu)
    assert torch.equal(y, y2)                                   # fixed-order reduction: bit-reproducible
    assert rel_l2(y, ref_groupnorm(x, S, rows, gamma, beta, eps, silu)) < BF16_TOL


# ---------------------------------------------------------------------------------------------- attention
def _strided(rows, inner, g, scale=1.0):
    """three [rows, inner] column blocks of one [rows, 3 * inner] buffer, as the fused qkv projection lays them out"""
    buf = (torch.randn(rows, 3 * inner, device="cuda", generator=g) * scale).bfloat16()
    return buf, buf[:, :inner], buf[:, inner:2 * inner], buf[:, 2 * inner:]


def _needle_inputs(B, H, Lq, Lk, pos, scale, g):
    """Key j* = pos holds c * e0 and every query has q[0] = 4, while every other key has a zero in dimension 0:
    the needle's logit is exactly 26 and every other logit is N(0, 63 scale^2).  Returns q, k, v views."""
    inner = H * 64
    _, q, _, _ = _strided(B * Lq, inner, g)
    _, _, k, v = _strided(B * Lk, inner, g)
    qh, kh = q.view(B * Lq, H, 64)[:, :, 0], k.view(B * Lk, H, 64)
    qh.fill_(4.0)
    kh[:, :, 0] = 0.0
    for b in range(B):
        kh[b * Lk + pos] = 0.0
        kh[b * Lk + pos, :, 0] = 26.0 / (4.0 * scale)
    return q, k, v


@pytest.mark.parametrize("Lq", [1, 129])
@pytest.mark.parametrize("Lk", [1, 127, 128, 129, 255, 257, 2560])
@pytest.mark.parametrize("where", ["first-tile", "last-tile"])
def test_attention_needle(cuda_device, Lq, Lk, where):
    """One key dominates every row by ~20 logits: the output row is that key's value.  With the key in the last
    key tile the running max moves late, so the O rescale in TMEM (alpha << 1) is what makes the result right."""
    from geo4d_b200 import ops
    B, H, scale = 2, 2, 0.125
    pos = 0 if where == "first-tile" else Lk - 1
    g = _gen(Lq * 10000 + Lk)
    q, k, v = _needle_inputs(B, H, Lq, Lk, pos, scale, g)
    inner = H * 64
    obuf = torch.full((B * Lq, 3 * inner), 7.0, device="cuda", dtype=torch.bfloat16)
    out = obuf[:, inner:2 * inner]                                # out written with ld = 3 * inner
    ops.attention(q, k, v, out, B, H, Lq, Lk, scale=scale)
    logits = torch.einsum("qhd,khd->hqk", q.double().view(B, Lq, H, 64)[0], k.double().view(B, Lk, H, 64)[0]) * scale
    if Lk > 1:
        others = torch.cat([logits[..., :pos], logits[..., pos + 1:]], -1)
        assert float((logits[..., pos] - others.amax(-1)).min()) > 16.0     # the construction is a needle
    want = torch.stack([v[b * Lk + pos] for b in range(B) for _ in range(Lq)])
    assert torch.equal(obuf[:, :inner], torch.full_like(obuf[:, :inner], 7.0))
    assert torch.equal(obuf[:, 2 * inner:], torch.full_like(obuf[:, 2 * inner:], 7.0))
    err = (out.double() - want.double()).abs()
    assert bool((err <= BF16_ULP * want.double().abs() + 1e-6).all()), f"max err {float(err.max()):.3e}"


@pytest.mark.parametrize("B,H,Lq,Lk,div,scale,qmul", [
    (2, 2, 129, 2560, 1, 0.125, 6.0),     # peaked: q x 6, logits ~ N(0, 36)
    (2, 3, 257, 257, 1, 0.2, 1.0),        # non-default scale
    (4, 2, 130, 77, 3, 0.125, 1.0),       # kv_batch_div that does not divide B
    (2, 2, 200, 300, 1, 0.125, 1.0),      # single set, Lk off a multiple of 128
    (3, 5, 16, 273, 1, 0.125, 1.0),       # the resampler: Lk = L + nq
])
def test_attention_vs_fp64(cuda_device, B, H, Lq, Lk, div, scale, qmul):
    from geo4d_b200 import ops
    g = _gen(B * 1000 + Lk)
    inner = H * 64
    _, q, _, _ = _strided(B * Lq, inner, g, qmul)
    _, _, k, v = _strided(-(-B // div) * Lk, inner, g)
    obuf = torch.full((B * Lq, 3 * inner), 7.0, device="cuda", dtype=torch.bfloat16)
    out = obuf[:, :inner]
    ops.attention(q, k, v, out, B, H, Lq, Lk, kv_batch_div=div, scale=scale)
    if qmul > 1:
        assert _logit_spread(q, k, Lq, Lk, H, scale) >= PEAKED_LOGIT_SPREAD
    assert torch.equal(obuf[:, inner:], torch.full_like(obuf[:, inner:], 7.0))
    assert rel_l2(out, ref_attention(q, k, v, B, H, Lq, Lk, div, scale)) < ATTN_TOL


@pytest.mark.parametrize("peaked", ["first-set", "second-set"])
@pytest.mark.parametrize("Lk1,Lk2", [(1, 257), (257, 1)])
def test_cross_attention2_edges(cuda_device, Lk1, Lk2, peaked):
    """two independent softmaxes in one launch, one key set peaked (q direction planted in a late key), one flat"""
    from geo4d_b200 import ops
    B, T, H, Lq, scale = 4, 2, 2, 129, 0.125
    inner = H * 64
    g = _gen(Lk1 * 7 + Lk2)
    _, q, _, _ = _strided(B * Lq, inner, g)
    _, _, k1, v1 = _strided((B // T) * Lk1, inner, g)
    _, _, k2, v2 = _strided(B * Lk2, inner, g)
    kp, Lp = (k1, Lk1) if peaked == "first-set" else (k2, Lk2)
    kp.mul_(6.0)                                   # peaked: logits ~ N(0, 36)
    out = torch.empty(B * Lq, inner, device="cuda", dtype=torch.bfloat16)
    ops.cross_attention2(q, k1, v1, Lk1, T, k2, v2, Lk2, 1, out, B, H, Lq, scale=scale)
    ref = ref_attention(q, k1, v1, B, H, Lq, Lk1, T, scale) + ref_attention(q, k2, v2, B, H, Lq, Lk2, 1, scale)
    assert rel_l2(out, ref) < ATTN_TOL


@pytest.mark.parametrize("T", [1, 2, 15, 16])
@pytest.mark.parametrize("qmul", [1.0, 6.0])
def test_temporal_attention_edges(cuda_device, T, qmul):
    from geo4d_b200 import ops
    B, HW, heads = 2, 37, 3                        # HW not a multiple of the 4 pixels a block handles
    inner = heads * 64
    g = _gen(T * 10 + int(qmul))
    buf = torch.randn(B * T * HW, 3 * inner, device="cuda", generator=g)
    buf[:, :inner] *= qmul
    buf = buf.bfloat16()
    q, k, v = buf[:, :inner], buf[:, inner:2 * inner], buf[:, 2 * inner:]
    out = torch.empty(B * T * HW, inner, device="cuda", dtype=torch.bfloat16)
    ops.temporal_attention(q, k, v, out, B, T, HW, heads)
    assert rel_l2(out, ref_temporal_attention(q, k, v, B, T, HW, heads)) < ATTN_TOL


# ---------------------------------------------------------------------------------------------- DDIM update
@pytest.mark.parametrize("with_noise,with_x0", [(True, True), (True, False), (False, False)])
def test_ddim_step_noise_and_optional_outputs(cuda_device, with_noise, with_x0):
    from geo4d_b200 import ops
    g = _gen(9)
    n = 1000 + 77                                            # not a multiple of the 256-thread block
    x = torch.randn(n, device="cuda", generator=g)
    v = torch.randn(n, device="cuda", generator=g)
    noise = torch.randn(n, device="cuda", generator=g) if with_noise else None
    coef = torch.tensor([[0.9, 0.4, 1.0, 0.8, 0.6, 0.0], [0.5, 0.85, 0.98, 0.7, 0.7, 0.3]], device="cuda")
    idx = torch.ones(1, dtype=torch.int32, device="cuda")
    x1 = x.clone()
    p0 = torch.empty_like(x) if with_x0 else None
    ops.ddim_step(x1, v, coef, idx, pred_x0=p0, noise=noise)
    xp, x0 = ref_ddim(x, v, coef[1], noise)
    assert rel_l2(x1, xp) < 1e-6                             # a few fp32 roundings of the formula
    if with_x0:
        assert rel_l2(p0, x0) < 1e-6


# ---------------------------------------------------------------------------------------------- tap-GEMM addressing
from tests.test_ops_gpu import gemm_mode  # noqa: E402,F401  (the four kernel modes: single / pair x TMA / direct store)


@pytest.mark.parametrize("M,K,n,act,out_dtype", [(300, 320, 320, 0, torch.bfloat16), (1000, 640, 96, 1, torch.bfloat16),
                                                  (257, 128, 64, 0, torch.float32)])
def test_linear_strided_operands(gemm_mode, M, K, n, act, out_dtype):
    """A view with lda > K, output into a column slice of a wider buffer, residual with ldr != n, alpha = 0.5"""
    from geo4d_b200 import ops
    g = _gen(M + K + n)
    xbuf = torch.randn(M, K + 64, device="cuda", generator=g).bfloat16()
    x = xbuf[:, 64:]
    w = (torch.randn(n, K, device="cuda", generator=g) / K ** 0.5).bfloat16()
    b = torch.randn(n, device="cuda", generator=g)
    rbuf = torch.randn(M, n + 40, device="cuda", generator=g).bfloat16()
    res = rbuf[:, 8:8 + n]
    obuf = torch.full((M, n + 96), 7.0, device="cuda", dtype=out_dtype)
    out = obuf[:, 32:32 + n]
    ops.linear(x, w, b, out=out, act=act, residual=res, alpha=0.5)
    torch.cuda.synchronize()
    assert torch.equal(obuf[:, :32], torch.full_like(obuf[:, :32], 7.0))
    assert torch.equal(obuf[:, 32 + n:], torch.full_like(obuf[:, 32 + n:], 7.0))
    assert rel_l2(out, ref_linear(x, w, b, act, res, 0.5)) < _out_bar(out_dtype)


def test_bmm_nt_vae_attention_shapes(gemm_mode):
    """the VAE mid-block attention at 320x512: S = (q k^T) / sqrt(C) in fp32 from a strided q, then P V^T in bf16"""
    from geo4d_b200 import ops
    g = _gen(2560)
    L, C = 2560, 512
    qkv = torch.randn(L, 3 * C, device="cuda", generator=g).bfloat16()
    q = qkv[:, :C].unflatten(0, (1, L))
    kc = qkv[:, C:2 * C].contiguous().unflatten(0, (1, L))
    s = ops.bmm_nt(q, kc, alpha=float(C) ** -0.5, out_dtype=torch.float32)
    torch.cuda.synchronize()
    assert rel_l2(s, ref_bmm_nt(q, kc, float(C) ** -0.5)) < FP32_TOL
    p = torch.softmax(s.double(), -1).bfloat16()
    vt = qkv[:, 2 * C:].t().contiguous().unsqueeze(0)                 # [1, C, L]
    o = ops.bmm_nt(p, vt)
    torch.cuda.synchronize()
    assert o.dtype == torch.bfloat16 and rel_l2(o, ref_bmm_nt(p, vt)) < BF16_TOL


@pytest.mark.parametrize("T", [1, 16])
def test_temporal_conv3_clip_edges(gemm_mode, T):
    """T = 1: both temporal taps fall off the clip; T = 16: the full clip."""
    from geo4d_b200 import ops
    g = _gen(T)
    B, HW, Cin, Cout = 2, 160, 128, 192
    x = torch.randn(B * T * HW, Cin, device="cuda", generator=g).bfloat16()
    w3 = (torch.randn(3, Cout, Cin, device="cuda", generator=g) / (3 * Cin) ** 0.5).bfloat16()
    b = torch.randn(Cout, device="cuda", generator=g)
    res = torch.randn(B * T * HW, Cout, device="cuda", generator=g).bfloat16()
    y = ops.temporal_conv3(x, B, T, HW, w3, b, residual=res)
    torch.cuda.synchronize()
    assert rel_l2(y, ref_temporal_conv3(x, B, T, HW, w3, b, res)) < BF16_TOL


def test_conv3x3_vae_full_resolution(gemm_mode):
    """N = 1, 320 x 512 (W = 512 > the 128-row box), Cin = Cout = 128"""
    from geo4d_b200 import ops
    g = _gen(320)
    N, H, W, C = 1, 320, 512, 128
    x = torch.randn(N * H * W, C, device="cuda", generator=g).bfloat16()
    w9 = (torch.randn(9, C, C, device="cuda", generator=g) / (9 * C) ** 0.5).bfloat16()
    b = torch.randn(C, device="cuda", generator=g)
    y = ops.conv3x3(x, N, H, W, w9, b)
    torch.cuda.synchronize()
    assert rel_l2(y, ref_conv3x3(x, N, H, W, w9, b)) < BF16_TOL
