"""Every dropout site against the host reference of the counter-based mask (tests/dropout_ref.py), and head_dim-64
attention in the regimes that need many work items per CTA or several images with several key tiles.

1. Extraction: inputs are built so that each output element is (keep ? known value * inv_keep : 0), so the realised
   keep / drop decisions of the kernel are read off its output and compared with the reference by exact equality;
   the kept values carry the inv_keep rescale within one bf16 ulp.
2. Parity: random inputs against a float64 autograd reference that applies the reference mask, with a global and a
   per-(image, head, 128-row tile) rel-L2; a mask from another seed (and, for attention, a backward mask shifted by one
   16-key group) must fail the same comparison by a wide margin.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import dropout_ref as dr

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

ULP = 2.0 ** -7          # one bf16 ulp, relative


def _ops():
    from sfcvit import ops
    return ops


def _mask_t(m):
    return torch.from_numpy(np.ascontiguousarray(m)).cuda()


def _assert_rescale(vals, expect, what, ulps=1.0):
    """vals (kernel, bf16) == expect (float64) within `ulps` bf16 ulps."""
    expect = torch.as_tensor(expect, dtype=torch.float64, device=vals.device)
    err = (vals.double() - expect).abs()
    bound = ulps * ULP * expect.abs() + 1e-30
    assert bool((err <= bound).all()), (what, float((err / bound).max()))


# ---------------------------------------------------------------------------------------------------------------- attention
def _attn_extract(B, H, N, dh, seed, p, epoch=None):
    """Realised masks of attention forward (probabilities as applied to V) and backward (as applied to dO -> dV)."""
    ops = _ops()
    D = H * dh
    inv = dr.inv_keep(p)
    fwd = torch.zeros(B, H, N, N, dtype=torch.bool, device="cuda")
    bwd = torch.zeros(B, H, N, N, dtype=torch.bool, device="cuda")
    qkv0 = torch.zeros(B * N, 3 * D, dtype=torch.bfloat16, device="cuda")        # Q = K = 0: P = 1 / N exactly
    _, lse = ops.attn_fwd(qkv0, B, H, N, drop_p=p, drop_seed=seed)
    out0 = torch.zeros(B * N, D, dtype=torch.bfloat16, device="cuda")             # V = 0: O = 0, delta = 0
    assert torch.allclose(lse, torch.full_like(lse, float(np.log(N))), atol=2e-3)
    for w in range((N + dh - 1) // dh):
        ks = torch.arange(w * dh, min(N, (w + 1) * dh), device="cuda")
        # forward: V one-hot over the key window -> out[q, d] = keep(q, w*dh + d) * inv / N
        qkv = qkv0.clone().view(B, N, 3, H, dh)
        qkv[:, ks, 2, :, ks - w * dh] = 1.0
        out, _ = ops.attn_fwd(qkv.view(B * N, 3 * D), B, H, N, drop_p=p, drop_seed=seed)
        o = out.view(B, N, H, dh).permute(0, 2, 1, 3)                            # [B, H, q, d]
        assert not bool(o[..., len(ks):].any()), "columns past the last key must be 0"
        o = o[..., :len(ks)]
        fwd[:, :, :, ks] = o != 0
        _assert_rescale(o[o != 0], inv / N, ("fwd", N, w))
        # backward: dO one-hot over the query window -> dV[k, d] = keep(w*dh + d, k) * inv / N
        dout = torch.zeros(B, N, H, dh, dtype=torch.bfloat16, device="cuda")
        dout[:, ks, :, ks - w * dh] = 1.0
        dqkv = ops.attn_bwd(qkv0, out0, dout.view(B * N, D), lse, B, H, N, drop_p=p, drop_seed=seed)
        dv = dqkv.view(B, N, 3, H, dh)[:, :, 2].permute(0, 2, 1, 3)               # [B, H, k, d]
        assert not bool(dv[..., len(ks):].any())
        dv = dv[..., :len(ks)]
        bwd[:, :, ks, :] = (dv != 0).transpose(-1, -2)
        _assert_rescale(dv[dv != 0], inv / N, ("bwd", N, w))
        assert not bool(dqkv.view(B, N, 3, H, dh)[:, :, :2].any()), "dQ, dK must be 0 when V = 0"
    return fwd, bwd


def _check_masks(got, ref, what):
    bad = (got != ref)
    if bool(bad.any()):
        where = torch.nonzero(bad)[:8].tolist()
        pytest.fail(f"{what}: {int(bad.sum())} of {bad.numel()} keep decisions differ from the reference, first at {where}")


# (N, comment): forward tile plan from fwd_layout, backward key tiles of <= 128 keys
TC_SHAPES = [1, 17, 128, 196, 197, 209, 577, 1025]


@pytest.mark.parametrize("N", TC_SHAPES)
def test_attention_tcgen05_mask_is_the_reference(cuda_device, N):
    B, H, seed, p = 2, 2, 0xC0FFEE + N, 0.3
    fwd, bwd = _attn_extract(B, H, N, 64, seed, p)
    ref = _mask_t(dr.attn_mask(B, H, N, seed, p))
    _check_masks(fwd, ref, f"attention forward N={N}")
    _check_masks(bwd, ref, f"attention backward N={N}")


def test_attention_tcgen05_mask_is_the_reference_n4096(cuda_device):
    B, H, N, seed, p = 2, 2, 4096, (1 << 64) - 3, 0.1
    fwd, bwd = _attn_extract(B, H, N, 64, seed, p)
    ref = _mask_t(dr.attn_mask(B, H, N, seed, p))
    _check_masks(fwd, ref, "attention forward N=4096")
    _check_masks(bwd, ref, "attention backward N=4096")


GENERIC_SHAPES = [(64, 192), (50, 32), (128, 96), (17, 16), (100, 48), (9, 128), (40, 24)]


@pytest.mark.parametrize("mma", [True, False])
@pytest.mark.parametrize("N,dh", GENERIC_SHAPES)
def test_attention_generic_mask_is_the_reference(cuda_device, monkeypatch, mma, N, dh):
    monkeypatch.setenv("SFC_ATTN_NO_MMA", "0" if mma else "1")
    B, H, seed, p = 2, 2, 77 + N, 0.25
    fwd, bwd = _attn_extract(B, H, N, dh, seed, p)
    ref = _mask_t(dr.attn_mask(B, H, N, seed, p))
    _check_masks(fwd, ref, f"generic attention forward N={N} dh={dh}")
    _check_masks(bwd, ref, f"generic attention backward N={N} dh={dh}")


def _rel(a, b):
    return float((a.double() - b).norm() / b.norm().clamp_min(1e-12))


def _tile_rel(x, ref, B, N, H, dh):
    """max over (image, head, 128-row tile) of the rel-L2 of [B*N, H*dh] tensors."""
    xa = x.double().reshape(B, N, H, dh)
    ra = ref.reshape(B, N, H, dh)
    worst = 0.0
    for t in range(0, N, 128):
        d = (xa[:, t:t + 128] - ra[:, t:t + 128]).pow(2).sum(dim=(1, 3)).sqrt()
        r = ra[:, t:t + 128].pow(2).sum(dim=(1, 3)).sqrt().clamp_min(1e-12)
        worst = max(worst, float((d / r).max()))
    return worst


def _attn_ref(qkv, dout, B, H, N, dh, mask_fwd, mask_bwd, inv):
    """float64 (softmax(S) * M * inv) V: out with M = mask_fwd, the gradients of the same expression with M = mask_bwd."""
    D = H * dh

    def run(mask):
        q, k, v = [t.reshape(B, N, H, dh).permute(0, 2, 1, 3).double().requires_grad_(True) for t in qkv.double().split(D, dim=1)]
        s = (q @ k.transpose(-1, -2)) * dh ** -0.5
        out = ((torch.softmax(s, dim=-1) * (mask.double() * inv)) @ v).permute(0, 2, 1, 3).reshape(B * N, D)
        out.backward(dout.double())
        return out.detach(), torch.logsumexp(s, dim=-1).detach(), [t.grad.permute(0, 2, 1, 3).reshape(B * N, D) for t in (q, k, v)]

    out, lse, grads = run(mask_bwd)
    if mask_fwd is not mask_bwd:
        out, _, _ = run(mask_fwd)
    return out, lse, grads


def _attn_errors(res, ref, B, H, N, dh):
    out, lse, dqkv = res
    rout, rlse, rg = ref
    D = H * dh
    e = {"out": (_rel(out, rout), _tile_rel(out, rout, B, N, H, dh)),
         "lse": float((lse.double() - rlse).abs().max())}
    for i, name in enumerate(("dq", "dk", "dv")):
        g = dqkv[:, i * D:(i + 1) * D]
        e[name] = (_rel(g, rg[i]), _tile_rel(g, rg[i], B, N, H, dh))
    return e


TOL = {"out": 1e-2, "dq": 2e-2, "dk": 2e-2, "dv": 2e-2}


def _attn_ok(e):
    return e["lse"] < 2e-3 and all(e[k][0] < t and e[k][1] < 3 * t for k, t in TOL.items())


def _attn_parity(B, H, N, dh, p, seed, controls=True):
    ops = _ops()
    D = H * dh
    g = torch.Generator(device="cuda").manual_seed(N * 7 + B)
    qkv = torch.randn(B * N, 3 * D, generator=g, device="cuda").bfloat16()
    dout = torch.randn(B * N, D, generator=g, device="cuda").bfloat16()
    out, lse = ops.attn_fwd(qkv, B, H, N, drop_p=p, drop_seed=seed)
    dqkv = ops.attn_bwd(qkv, out, dout, lse, B, H, N, drop_p=p, drop_seed=seed)
    res = (out, lse, dqkv)
    inv = dr.inv_keep(p)
    m = _mask_t(dr.attn_mask(B, H, N, seed, p)) if p > 0 else torch.ones((), dtype=torch.bool, device="cuda")
    e = _attn_errors(res, _attn_ref(qkv, dout, B, H, N, dh, m, m, inv), B, H, N, dh)
    assert _attn_ok(e), e
    if p > 0 and controls:
        # a mask of another seed must fail by a wide margin (out and all gradients)
        m2 = _mask_t(dr.attn_mask(B, H, N, seed + 1, p))
        e2 = _attn_errors(res, _attn_ref(qkv, dout, B, H, N, dh, m2, m2, inv), B, H, N, dh)
        for k, t in TOL.items():
            assert e2[k][0] > 5 * t, ("wrong-seed control passed", k, e2)
        # a backward mask shifted by one 16-key group against the right forward mask: the gradients must fail
        m3 = torch.roll(m, 16, dims=-1)
        e3 = _attn_errors(res, _attn_ref(qkv, dout, B, H, N, dh, m, m3, inv), B, H, N, dh)
        assert e3["out"][0] < TOL["out"]
        for k in ("dq", "dk", "dv"):
            assert e3[k][0] > 5 * TOL[k], ("shifted-backward-mask control passed", k, e3)
    return e


@pytest.mark.parametrize("N", TC_SHAPES[1:] + [4096])
def test_attention_tcgen05_dropout_parity(cuda_device, N):
    B, H = (2, 2) if N < 4096 else (1, 2)
    _attn_parity(B, H, N, 64, 0.1, 1234 + N)


def test_attention_tcgen05_dropout_parity_many_items(cuda_device):
    """B * H = 384 items in both directions on 148 SMs: persistent CTAs run several items each."""
    _attn_parity(64, 6, 197, 64, 0.1, 99)


@pytest.mark.parametrize("mma", [True, False])
@pytest.mark.parametrize("N,dh", GENERIC_SHAPES)
def test_attention_generic_dropout_parity(cuda_device, monkeypatch, mma, N, dh):
    monkeypatch.setenv("SFC_ATTN_NO_MMA", "0" if mma else "1")
    _attn_parity(2, 2, N, dh, 0.25, 4321 + N)


@pytest.mark.parametrize("B,H,N", [(64, 6, 197), (3, 2, 209), (2, 3, 577), (2, 2, 1025), (4, 2, 4096)])
def test_attention_tcgen05_no_dropout_per_tile(cuda_device, B, H, N):
    """Without dropout: many persistent items per CTA (B * H = 384), and B >= 2 with several forward key tiles (keys past
    N of image b must not pick up image b + 1's rows), each 128-row tile of each (image, head) checked on its own."""
    _attn_parity(B, H, N, 64, 0.0, 0)


# --------------------------------------------------------------------------------------------------------------------- GEMM
GEMM_VARIANTS = {
    # name: (N options, kwargs builder key) -- the comment names the epilogue the dispatcher picks
    "ncols_odd": "EPI 0 (N % 32 != 0)",
    "gelu": "EPI 0 (GELU)",
    "fp32": "EPI 1 (fp32 out)",
    "res_aux": "EPI 1 (residual + aux)",
    "plain": "EPI 2 (TMA store)",
    "res": "EPI 3 (TMA store + residual)",
    "aux": "EPI 4 (TMA store + ReLU-mask aux)",
}


def _gemm_case(M, N, variant, seed, p=0.3, epoch=None):
    """Runs one dropout GEMM whose pre-dropout values are all ~16 and returns (observed keep, reference keep)."""
    ops = _ops()
    K = 256
    g = torch.Generator(device="cuda").manual_seed(M * 1000 + N)
    a = (torch.randn(M, K, generator=g, device="cuda") * 0.05).bfloat16()
    w = (torch.randn(N, K, generator=g, device="cuda") * 0.05).bfloat16()
    bias = torch.full((N,), 16.0, dtype=torch.bfloat16, device="cuda")
    kw = dict(bias=bias, drop_p=p, drop_seed=seed)
    res = aux = None
    if variant in ("res", "res_aux"):
        res = torch.randn(M, N, generator=g, device="cuda").bfloat16()
        kw["residual"] = res
    if variant in ("aux", "res_aux"):
        aux = (torch.rand(M, N, generator=g, device="cuda") - 0.2).bfloat16()        # ~20 % ReLU-masked
        kw.update(aux=aux, aux_mode=ops.AUX_RELU_MASK)
    if variant == "gelu":
        kw["act"] = ops.ACT_GELU
    if variant == "fp32":
        kw["out_dtype"] = torch.float32
    out = ops.gemm(a, w, **kw)
    pre = a.double() @ w.double().t() + 16.0
    if variant == "gelu":
        pre = torch.nn.functional.gelu(pre)
    ref_keep = _mask_t(dr.gemm_mask(M, N, seed, p, epoch))
    live = torch.ones(M, N, dtype=torch.bool, device="cuda") if aux is None else aux > 0
    base = torch.zeros(M, N, dtype=torch.float64, device="cuda") if res is None else res.double()
    got_keep = out.double() != base
    _check_masks(got_keep & live, ref_keep & live, f"GEMM {variant} M={M} N={N}")
    assert not bool((got_keep & ~live).any()), "ReLU-masked elements must carry the residual only"
    expect = pre * dr.inv_keep(p) + base
    tol = (2.0 ** -23 if variant == "fp32" else ULP) * expect.abs() + 1e-5
    kept = ref_keep & live
    assert bool(((out.double() - expect).abs() <= tol)[kept].all()), (variant, M, N)
    return got_keep, ref_keep


@pytest.mark.parametrize("M", [100, 300])             # one CTA per tile / CTA pairs (fast epilogues only)
@pytest.mark.parametrize("N", [640, 768])             # column tiles of 128 / 256 (gemm_pick_bn)
@pytest.mark.parametrize("variant", ["gelu", "fp32", "res_aux", "plain", "res", "aux"])
def test_gemm_epilogue_mask_is_the_reference(cuda_device, variant, M, N):
    _gemm_case(M, N, variant, seed=(1 << 32) + 5 + M + N)


@pytest.mark.parametrize("M", [100, 300])
@pytest.mark.parametrize("N", [600, 200])             # N % 32 != 0: 128- and 256-column tiles
def test_gemm_epilogue_mask_is_the_reference_ncols_odd(cuda_device, M, N):
    _gemm_case(M, N, "ncols_odd", seed=17 + M + N)


# ------------------------------------------------------------------------------------------------- act_bwd / layernorm_bwd
@pytest.mark.parametrize("n", [8 * 1000 + 8, 4096 * 3 + 72])           # multiples of 8, not of 64
@pytest.mark.parametrize("mode", ["none", "gelu_grad", "relu_mask"])
def test_act_bwd_mask_is_the_reference(cuda_device, mode, n):
    ops = _ops()
    p, seed, alpha = 0.3, 2024 + n, 0.75
    g = torch.Generator(device="cuda").manual_seed(n)
    dy = torch.ones(n, dtype=torch.bfloat16, device="cuda")
    code = {"none": ops.AUX_NONE, "gelu_grad": ops.AUX_GELU_GRAD, "relu_mask": ops.AUX_RELU_MASK}[mode]
    aux = None
    if mode == "gelu_grad":
        aux = (torch.rand(n, generator=g, device="cuda") * 3 + 1).bfloat16()          # gelu'(a) in (1.0, 1.09)
    elif mode == "relu_mask":
        aux = (torch.rand(n, generator=g, device="cuda") - 0.2).bfloat16()
    out = ops.act_bwd(dy, aux, code, alpha=alpha, drop_p=p, drop_seed=seed)
    live = torch.ones(n, dtype=torch.bool, device="cuda") if mode != "relu_mask" else aux > 0
    ref = _mask_t(dr.flat_mask(n, seed, p))
    _check_masks((out != 0) & live, ref & live, f"act_bwd {mode} n={n}")
    assert not bool((out != 0)[~live].any())
    fprime = torch.ones(n, dtype=torch.float64, device="cuda")
    if mode == "gelu_grad":
        a = aux.double()
        fprime = 0.5 * (1 + torch.erf(a / 2 ** 0.5)) + a * torch.exp(-0.5 * a * a) / (2 * np.pi) ** 0.5
    kept = ref & live
    _assert_rescale(out[kept], (alpha * dr.inv_keep(p) * fprime)[kept], f"act_bwd {mode}")


@pytest.mark.parametrize("rows,D", [(333, 192), (77, 1024), (5, 2048)])
def test_layernorm_bwd_dropout_mask_and_colsum(cuda_device, rows, D):
    ops = _ops()
    p, seed = 0.25, 555 + D
    g = torch.Generator(device="cuda").manual_seed(rows)
    x = (torch.randn(rows, D, generator=g, device="cuda") * 2 + 0.5).bfloat16()
    gamma = (1 + 0.1 * torch.randn(D, generator=g, device="cuda")).bfloat16()
    beta = (0.1 * torch.randn(D, generator=g, device="cuda")).bfloat16()
    dy = torch.randn(rows, D, generator=g, device="cuda").bfloat16()
    _, mean, rstd = ops.layernorm_fwd(x, gamma, beta)
    dx, _, _, dxd, cs = ops.layernorm_bwd(dy, x, mean, rstd, gamma, torch.float32, drop_p=p, drop_seed=seed, want_colsum=True)
    ref = _mask_t(dr.ln_mask(rows, D, seed, p))
    nz = dx != 0
    _check_masks((dxd != 0) & nz, ref & nz, f"layernorm_bwd rows={rows} D={D}")
    assert not bool((dxd != 0)[~nz].any())
    kept = ref & nz
    # dx and dxd are two roundings of the same fp32 value: within one ulp of each other after the rescale
    _assert_rescale(dxd[kept], dx.double()[kept] * dr.inv_keep(p), "layernorm_bwd dx_drop", ulps=1.5)
    csum_ref = dxd.double().sum(0)
    assert _rel(cs, csum_ref) < 2e-3, _rel(cs, csum_ref)


# -------------------------------------------------------------------------------------------------------------------- epoch
def test_graph_epoch_is_mixed_into_every_site(cuda_device):
    """In a child process (the epoch counter is process-wide): epoch 0, then 7 via graphs.dropout_epoch; the masks of
    attention, GEMM and act_bwd follow seed + epoch * 0xD1B54A32D192ED03."""
    code = r"""
import sys; sys.path[:0] = ['tests', 'space-filling-curves-for-vision-transformers_b200']
import torch, dropout_ref as dr, test_gpu_dropout as t
from sfcvit import ops
from src.training import graphs
ep = graphs.dropout_epoch('cuda')
for e in (0, 7):
    ep.fill_(e); torch.cuda.synchronize()
    assert dr.current_epoch() == e
    seed, p = 31337, 0.3
    fwd, bwd = t._attn_extract(2, 2, 197, 64, seed, p)
    ref = t._mask_t(dr.attn_mask(2, 2, 197, seed, p))
    t._check_masks(fwd, ref, f'attention fwd epoch {e}'); t._check_masks(bwd, ref, f'attention bwd epoch {e}')
    assert torch.equal(ref, t._mask_t(dr.attn_mask(2, 2, 197, seed + e * dr.EPOCH_MUL, p, epoch=0)))
    t._gemm_case(300, 768, 'plain', seed)
    t._gemm_case(100, 640, 'res', seed)
    out = ops.act_bwd(torch.ones(4104, dtype=torch.bfloat16, device='cuda'), None, ops.AUX_NONE, drop_p=p, drop_seed=seed)
    t._check_masks(out != 0, t._mask_t(dr.flat_mask(4104, seed, p)), f'act_bwd epoch {e}')
print('ok')
"""
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout[-2000:] + r.stderr[-4000:]


# ------------------------------------------------------------------------------------------------- encoder layer / head
def _ln64(x, g, b, eps):
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    return (x - mu) / torch.sqrt(var + eps) * g + b


def _encoder_ref(x, P, B, N, D, H, eps, masks, invs):
    """float64 post-norm ReLU encoder layer (torch.nn.TransformerEncoderLayer, batch_first) with explicit masks."""
    in_w, in_b, out_w, out_b, w1, b1, w2, b2, g1, be1, g2, be2 = P
    m_attn, m_d1, m_ff, m_d2 = masks
    i_attn, i_d1, i_ff, i_d2 = invs
    dh = D // H
    x2 = x.reshape(B * N, D)
    qkv = x2 @ in_w.t() + in_b
    q, k, v = [t.reshape(B, N, H, dh).permute(0, 2, 1, 3) for t in qkv.split(D, dim=1)]
    pr = torch.softmax((q @ k.transpose(-1, -2)) * dh ** -0.5, dim=-1) * (m_attn * i_attn)
    attn = (pr @ v).permute(0, 2, 1, 3).reshape(B * N, D)
    y1 = x2 + (attn @ out_w.t() + out_b) * (m_d1 * i_d1)
    x1 = _ln64(y1, g1, be1, eps)
    h = torch.relu(x1 @ w1.t() + b1) * (m_ff * i_ff)
    y2 = x1 + (h @ w2.t() + b2) * (m_d2 * i_d2)
    return _ln64(y2, g2, be2, eps).reshape(B, N, D)


def test_encoder_layer_training_mode_matches_float64(cuda_device):
    """SF.encoder_layer with all four dropout sites on (seeds seed + 0..3) against a float64 restatement that applies the
    four reference masks: output, input gradient and the 12 parameter gradients. The FFN backward takes its ReLU mask
    from the post-dropout h (h == 0: ReLU-zero or dropped), which this covers."""
    from sfcvit import functional as SF
    B, N, D, H, F, eps = 8, 197, 192, 3, 384, 1e-5
    drops = (0.1, 0.1, 0.2, 0.1)
    seed = (1 << 63) + 12345
    torch.manual_seed(0)
    layer = torch.nn.TransformerEncoderLayer(D, H, F, dropout=0.1, batch_first=True).cuda()
    with torch.no_grad():                                   # bf16-exact parameters: both sides see the same numbers
        for prm in layer.parameters():
            prm.copy_(prm.bfloat16().float())
            if prm.dim() == 1:
                prm.add_(0.05 * torch.randn_like(prm)).copy_(prm.bfloat16().float())
    params = [layer.self_attn.in_proj_weight, layer.self_attn.in_proj_bias, layer.self_attn.out_proj.weight,
              layer.self_attn.out_proj.bias, layer.linear1.weight, layer.linear1.bias, layer.linear2.weight, layer.linear2.bias,
              layer.norm1.weight, layer.norm1.bias, layer.norm2.weight, layer.norm2.bias]
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(B, N, D, generator=g, device="cuda").bfloat16().float().requires_grad_(True)
    dout = torch.randn(B, N, D, generator=g, device="cuda").bfloat16().float()
    out = SF.encoder_layer(x, layer, H, eps, drops, seed)
    out.backward(dout)
    got = [out.detach(), x.grad] + [prm.grad for prm in params]

    def ref_run(sd):
        masks = (_mask_t(dr.attn_mask(B, H, N, sd, drops[0])).double(), _mask_t(dr.gemm_mask(B * N, D, sd + 1, drops[1])).double(),
                 _mask_t(dr.gemm_mask(B * N, F, sd + 2, drops[2])).double(), _mask_t(dr.gemm_mask(B * N, D, sd + 3, drops[3])).double())
        xr = x.detach().double().requires_grad_(True)
        pr = [prm.detach().double().requires_grad_(True) for prm in params]
        o = _encoder_ref(xr, pr, B, N, D, H, eps, masks, [dr.inv_keep(pp) for pp in drops])
        o.backward(dout.double())
        return [o.detach(), xr.grad] + [t.grad for t in pr]

    names = ["out", "dx", "in_w", "in_b", "out_w", "out_b", "w1", "b1", "w2", "b2", "g1", "be1", "g2", "be2"]
    tol = {"out": 2e-2}
    errs = {n: _rel(a, r) for n, a, r in zip(names, got, ref_run(seed))}
    assert all(errs[n] < tol.get(n, 5e-2) for n in names), errs
    # masks of other seeds: out and dx fail their tolerances, by at least 10x the error of the right masks
    wrong = {n: _rel(a, r) for n, a, r in zip(names, got, ref_run(seed + 4))}
    for n in ("out", "dx"):
        assert wrong[n] > max(tol.get(n, 5e-2), 10 * errs[n]), ("wrong-seed control passed", n, wrong, errs)


@pytest.mark.parametrize("M", [4, 256])
def test_head_linear_gelu_dropout_matches_float64(cuda_device, M):
    """The factorised head's hidden layer: SF.linear with GELU and p = 0.5 at K = 12544, N = 1536, forward and backward."""
    from sfcvit import functional as SF
    K, N, p, seed = 12544, 1536, 0.5, 2 ** 40 + M
    g = torch.Generator(device="cuda").manual_seed(M)
    x = (torch.randn(M, K, generator=g, device="cuda")).bfloat16().float().requires_grad_(True)
    w = (torch.randn(N, K, generator=g, device="cuda") * K ** -0.5).bfloat16().float().requires_grad_(True)
    b = (torch.randn(N, generator=g, device="cuda") * 0.1).bfloat16().float().requires_grad_(True)
    dy = torch.randn(M, N, generator=g, device="cuda").bfloat16().float()
    y = SF.linear(x, w, b, act=SF.ACT_GELU, drop_p=p, seed=seed)
    y.backward(dy)
    got = [y.detach(), x.grad, w.grad, b.grad]

    def ref_run(sd):
        m = _mask_t(dr.gemm_mask(M, N, sd, p)).double() * dr.inv_keep(p)
        xr, wr, br = [t.detach().double().requires_grad_(True) for t in (x, w, b)]
        yr = torch.nn.functional.gelu(xr @ wr.t() + br) * m
        yr.backward(dy.double())
        return [yr.detach(), xr.grad, wr.grad, br.grad]

    names = ["y", "dx", "dw", "db"]
    errs = {n: _rel(a, r) for n, a, r in zip(names, got, ref_run(seed))}
    assert errs["y"] < 1e-2 and all(errs[n] < 2e-2 for n in names[1:]), errs
    wrong = {n: _rel(a, r) for n, a, r in zip(names, got, ref_run(seed + 1))}
    assert all(wrong[n] > 0.2 for n in names), ("wrong-seed control passed", wrong)
