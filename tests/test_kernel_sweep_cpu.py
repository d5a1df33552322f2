"""CPU: the fp64 reference helpers of tests/test_kernel_sweep_gpu.py against torch's own ops, so that a wrong
reference cannot make a wrong kernel pass.  Inputs are bf16-rounded like the kernels' operands; agreement is to
fp64 rounding (1e-10 relative) unless stated."""
import pytest
import torch
import torch.nn.functional as F

from tests.test_kernel_sweep_gpu import (ref_attention, ref_bmm_nt, ref_conv3x3, ref_ddim, ref_groupnorm,
                                         ref_im2col_s2, ref_layernorm, ref_linear, ref_softmax_rows,
                                         ref_temporal_attention, ref_temporal_conv3, ref_transpose, ref_upsample2x,
                                         _gn_ratio, rel_l2)

TOL = 1e-10


def _g(seed):
    return torch.Generator().manual_seed(seed)


def _bf(*shape, g, scale=1.0, offset=0.0):
    return (torch.randn(*shape, generator=g) * scale + offset).bfloat16()


@pytest.mark.parametrize("act", [0, 1, 2, 3])
def test_ref_linear(act):
    g = _g(act)
    M, K, n = 37, 128, 128
    x, w = _bf(M, K, g=g), _bf(n, K, g=g, scale=K ** -0.5)
    b, res = torch.randn(n, generator=g), _bf(M, n // 2 if act == 2 else n, g=g)
    got = ref_linear(x, w, b, act, res, alpha=0.5)
    y = F.linear(x.double(), w.double(), None) * 0.5 + b.double()
    if act == 1:
        y = F.silu(y)
    elif act == 3:
        y = F.gelu(y)
    elif act == 2:
        # kernel layout: weight rows in blocks [32 value | 32 gate]; value column j pairs with gate column j
        idx = torch.arange(n).reshape(-1, 2, 32)
        y = y[:, idx[:, 0].reshape(-1)] * F.gelu(y[:, idx[:, 1].reshape(-1)])
    assert rel_l2(got, y + res.double()) < TOL


def test_ref_conv3x3():
    g = _g(1)
    N, H, W, Cin, Cout = 3, 5, 7, 16, 24
    x = _bf(N, Cin, H, W, g=g)
    w = _bf(Cout, Cin, 3, 3, g=g)
    b, rb = torch.randn(Cout, generator=g), torch.randn(N, Cout, generator=g)
    res = _bf(N * H * W, Cout, g=g)
    rows = x.permute(0, 2, 3, 1).reshape(N * H * W, Cin)
    w9 = w.permute(2, 3, 0, 1).reshape(9, Cout, Cin)
    got = ref_conv3x3(rows, N, H, W, w9, b, rb, H * W, res)
    want = F.conv2d(x.double(), w.double(), b.double(), padding=1) + rb.double()[:, :, None, None]
    assert rel_l2(got, want.permute(0, 2, 3, 1).reshape(N * H * W, Cout) + res.double()) < TOL


@pytest.mark.parametrize("T", [1, 2, 5])
def test_ref_temporal_conv3(T):
    g = _g(T)
    B, HW, Cin, Cout = 2, 6, 16, 8
    x = _bf(B, Cin, T, HW, 1, g=g)
    w = _bf(Cout, Cin, 3, 1, 1, g=g)
    b = torch.randn(Cout, generator=g)
    got = ref_temporal_conv3(x[..., 0].permute(0, 2, 3, 1).reshape(-1, Cin), B, T, HW,
                             w[:, :, :, 0, 0].permute(2, 0, 1), b)
    want = F.conv3d(x.double(), w.double(), b.double(), padding=(1, 0, 0))[..., 0].permute(0, 2, 3, 1)
    assert rel_l2(got, want.reshape(-1, Cout)) < TOL


def test_ref_bmm_nt():
    g = _g(2)
    a, b = _bf(3, 40, 64, g=g), _bf(3, 24, 64, g=g)
    assert rel_l2(ref_bmm_nt(a, b, 0.25), 0.25 * torch.bmm(a.double(), b.double().transpose(1, 2))) < TOL


@pytest.mark.parametrize("offset", [0.0, 64.0])
@pytest.mark.parametrize("silu", [False, True])
def test_ref_groupnorm(offset, silu):
    g = _g(3)
    S, rows, C = 3, 50, 64
    x = _bf(S * rows, C, g=g, scale=1.5, offset=offset)
    gamma, beta = torch.randn(C, generator=g), torch.randn(C, generator=g)
    want = F.group_norm(x.double().reshape(S, rows, C).permute(0, 2, 1), 32, gamma.double(), beta.double(), 1e-5)
    want = want.permute(0, 2, 1).reshape(S * rows, C)
    if silu:
        want = F.silu(want)
    assert rel_l2(ref_groupnorm(x, S, rows, gamma, beta, 1e-5, silu), want) < TOL
    # |mean| / std of a group, as the production recorder measures it
    grp = x.double().reshape(S, rows, 32, 2)
    want_ratio = max(float(grp[s, :, k].mean().abs() / grp[s, :, k].std(unbiased=False))
                     for s in range(S) for k in range(32))
    assert abs(_gn_ratio(x, S, rows) - want_ratio) < 1e-9 * max(1.0, want_ratio)


def test_ref_layernorm():
    g = _g(4)
    x = _bf(33, 320, g=g, scale=2.0, offset=0.5)
    gamma, beta = torch.randn(320, generator=g), torch.randn(320, generator=g)
    want = F.layer_norm(x.double(), (320,), gamma.double(), beta.double(), 1e-5)
    assert rel_l2(ref_layernorm(x, gamma, beta, 1e-5), want) < TOL


@pytest.mark.parametrize("B,div", [(4, 1), (4, 3)])
def test_ref_attention(B, div):
    g = _g(B + div)
    H, Lq, Lk, scale = 2, 9, 13, 0.2
    Bk = -(-B // div)
    q, k, v = _bf(B * Lq, H * 64, g=g), _bf(Bk * Lk, H * 64, g=g), _bf(Bk * Lk, H * 64, g=g)
    got = ref_attention(q, k, v, B, H, Lq, Lk, div, scale)
    idx = torch.arange(B) // div
    qh = q.double().reshape(B, Lq, H, 64).transpose(1, 2)
    kh = k.double().reshape(Bk, Lk, H, 64).transpose(1, 2)[idx]
    vh = v.double().reshape(Bk, Lk, H, 64).transpose(1, 2)[idx]
    want = F.scaled_dot_product_attention(qh, kh, vh, scale=scale).transpose(1, 2).reshape(B * Lq, H * 64)
    assert rel_l2(got, want) < TOL


def test_ref_temporal_attention():
    g = _g(5)
    B, T, HW, heads = 2, 5, 7, 2
    inner = heads * 64
    q, k, v = (_bf(B * T * HW, inner, g=g) for _ in range(3))
    got = ref_temporal_attention(q, k, v, B, T, HW, heads, 0.125)
    for b, t, p in [(0, 0, 0), (1, 4, 6), (1, 2, 3)]:
        row = (b * T + t) * HW + p
        keys = [(b * T + s) * HW + p for s in range(T)]
        for h in range(heads):
            sl = slice(h * 64, (h + 1) * 64)
            w = torch.softmax(k.double()[keys, sl] @ q.double()[row, sl] * 0.125, 0)
            assert rel_l2(got[row, sl], w @ v.double()[keys, sl]) < TOL


def test_ref_softmax_rows():
    g = _g(6)
    s = torch.randn(5, 12, generator=g) * 4
    s[0, 3] = 80.0
    s[2] -= 1e4
    e = torch.exp(s.double() - s.double().amax(1, keepdim=True))
    assert rel_l2(ref_softmax_rows(s), e / e.sum(1, keepdim=True)) < TOL


def test_ref_data_movement():
    g = _g(7)
    x = _bf(2 * 5, 20, g=g)
    t = ref_transpose(x, 2, 5, 12)
    assert t.shape == (2, 12, 5) and all(torch.equal(t[b], x[b * 5:(b + 1) * 5, :12].t()) for b in range(2))
    N, H, W, C = 2, 3, 4, 8
    u = _bf(N * H * W, C, g=g)
    want = F.interpolate(u.float().reshape(N, H, W, C).permute(0, 3, 1, 2), scale_factor=2, mode="nearest")
    assert torch.equal(ref_upsample2x(u, N, H, W).float(), want.permute(0, 2, 3, 1).reshape(-1, C))
    for H, W, pad in [(6, 8, 1), (7, 5, 1), (6, 8, 0), (7, 5, 0)]:
        x = _bf(N * H * W, C, g=g)
        x4 = x.float().reshape(N, H, W, C).permute(0, 3, 1, 2)
        xp = F.pad(x4, (1, 1, 1, 1)) if pad == 1 else F.pad(x4, (0, 1, 0, 1))   # U-Net / VAE downsample padding
        Ho, Wo = (xp.shape[2] - 3) // 2 + 1, (xp.shape[3] - 3) // 2 + 1
        cols = F.unfold(xp, 3, stride=2)                                            # [N, C*9 (c, ky, kx), L]
        want = cols.reshape(N, C, 9, Ho * Wo).permute(0, 3, 2, 1).reshape(N * Ho * Wo, 9 * C)
        assert torch.equal(ref_im2col_s2(x, N, H, W, pad, Ho, Wo).float(), want)


def test_ref_ddim():
    coef = torch.tensor([0.5, 0.85, 0.98, 0.7, 0.7, 0.3])
    x, v, nz = torch.tensor([1.5, -2.0]), torch.tensor([0.25, 3.0]), torch.tensor([-1.0, 0.5])
    xp, x0 = ref_ddim(x, v, coef, nz)
    sa, s1, rs, sap, dr, sg = coef.double().tolist()
    for i in range(2):
        xi, vi = float(x[i]), float(v[i])
        x0i = (sa * xi - s1 * vi) * rs
        assert abs(float(x0[i]) - x0i) < 1e-12
        assert abs(float(xp[i]) - (sap * x0i + dr * (sa * vi + s1 * xi) + sg * float(nz[i]))) < 1e-12
