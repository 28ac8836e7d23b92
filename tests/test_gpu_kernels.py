"""Kernel-level parity through the C ABI: attention (K4), fused patch embed (K2), LayerNorm / column sums (K5),
fused clip + AdamW (K6), each against torch fp32 math on the same bf16 inputs (tolerances inside kernel_selftest)."""
import os
import sys

import pytest

pytestmark = pytest.mark.gpu
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))


@pytest.mark.parametrize("args", [(1, 1, 128), (2, 3, 196), (2, 2, 64), (1, 2, 576), (1, 1, 1), (3, 1, 129)])
def test_attention_fwd_bwd(cuda_device, args):
    import kernel_selftest as ks
    r = ks.check_attn(*args)
    assert r["ok"], r


def test_attention_dropout_mask_consistent(cuda_device):
    import kernel_selftest as ks
    r = ks.check_attn(2, 3, 196, 0.1)
    assert r["ok"], r


def test_attention_rejects_unsupported_shapes(cuda_device):
    """head_dim 64 runs on tensor cores for any N; other head dims need head_dim % 8 == 0 and N <= 128 (generic path)."""
    import torch
    from sfcvit import ops
    with pytest.raises(RuntimeError):       # head_dim 20
        ops.attn_fwd(torch.zeros(16, 3 * 60, dtype=torch.bfloat16, device="cuda"), 1, 3, 16)
    with pytest.raises(RuntimeError):       # head_dim 32 with 196 tokens
        ops.attn_fwd(torch.zeros(196, 3 * 96, dtype=torch.bfloat16, device="cuda"), 1, 3, 196)


@pytest.mark.parametrize("args", [(3, 3, 224, 16, 1, 768, "hilbert", "fp32"), (3, 3, 224, 16, 1, 384, "hilbert", "bf16"),
                                  (5, 3, 32, 4, 1, 192, "z", "fp32"), (5, 3, 32, 1, 16, 256, "hilbert", "fp32"),
                                  (5, 3, 32, 2, 4, 256, "peano", "fp32"), (2, 3, 64, 8, 2, 128, "moore", "bf16"),
                                  (2, 3, 384, 16, 1, 1024, "peano", "fp32"),
                                  # p == 4: 8-element chunks are two 4-element patch rows (vectorised half-row gather)
                                  (6, 3, 32, 4, 1, 192, "hilbert", "bf16"), (3, 3, 64, 4, 4, 128, "hilbert", "fp32"),
                                  (3, 1, 32, 4, 2, 128, "moore", "bf16"), (130, 3, 32, 4, 1, 256, "peano", "fp32"),
                                  # one k-block per tile: both warp sets of the split epilogue, 1 / 2 / 6 / 8 column chunks
                                  (2, 3, 16, 4, 1, 32, "z", "fp32"), (40, 3, 32, 4, 1, 64, "hilbert", "fp32"),
                                  (300, 3, 32, 4, 1, 192, "hilbert", "fp32")])
def test_patch_embed(cuda_device, args):
    import kernel_selftest as ks
    r = ks.check_patch(*args)
    assert r["ok"], r


# The TMEM-resident kernel (K <= 768, p % 8 == 0, D % 128 == 0): odd / even k-block counts, group changes inside a row,
# one channel, partial last tile, fewer tiles than a cluster, several tiles per CTA (> 148 tiles), fused position
# embedding behind a class-token row; cluster sizes 4 / 2 / 1 (>= 4 / 2-3 / 1 row tiles) for fp32 and bf16 input.
@pytest.mark.parametrize("args", [(4, 3, 64, 8, 1, 256, "hilbert", "fp32"), (2, 1, 64, 16, 1, 128, "z", "bf16"),
                                  (1, 3, 32, 16, 1, 128, "hilbert", "fp32"), (3, 3, 64, 8, 4, 384, "moore", "fp32"),
                                  (100, 3, 224, 16, 1, 256, "hilbert", "bf16"), (7, 3, 224, 16, 1, 768, "hilbert", "fp32"),
                                  (3, 3, 64, 8, 1, 256, "peano", "bf16"),
                                  (9, 3, 32, 4, 1, 192, "hilbert", "fp32"), (9, 3, 32, 4, 1, 320, "moore", "bf16")])
def test_patch_embed_tmem_resident(cuda_device, args):
    import kernel_selftest as ks
    r = ks.check_patch(*args, pos_cls=True)
    assert r["ok"], r


# The shared-memory kernel on the vectorised p % 8 == 0 gather, for shapes the TMEM-resident kernel does not take:
# D % 128 != 0 (fp32 and bf16 input; ViT-Tiny/16 has D = 192) and K > 768 (K = 1536: 24 k-blocks).
@pytest.mark.parametrize("args", [(3, 3, 224, 16, 1, 192, "hilbert", "fp32"), (2, 3, 64, 8, 1, 320, "moore", "bf16"),
                                  (2, 3, 64, 16, 2, 256, "z", "fp32")])
def test_patch_embed_smem_vectorised_gather(cuda_device, args):
    import kernel_selftest as ks
    r = ks.check_patch(*args, pos_cls=True)
    assert r["ok"], r


@pytest.mark.parametrize("args", [(1000, 768), (333, 192), (77, 1024), (5, 2048)])
def test_layernorm_and_colsum(cuda_device, args):
    import kernel_selftest as ks
    r = ks.check_ln(*args)
    assert r["ok"], r


def test_fused_clip_adamw_matches_torch(cuda_device):
    import kernel_selftest as ks
    r = ks.check_adamw()
    assert r["ok"], r


@pytest.mark.parametrize("mma", [True, False])
@pytest.mark.parametrize("B,H,N,dh,drop", [(2, 4, 64, 192, 0.0), (3, 2, 50, 32, 0.0), (1, 3, 128, 96, 0.0), (2, 4, 64, 192, 0.1),
                                           (2, 2, 17, 16, 0.0), (1, 2, 100, 48, 0.0), (2, 1, 9, 128, 0.0), (1, 2, 40, 24, 0.0)])
def test_attention_generic_head_dim(cuda_device, monkeypatch, mma, B, H, N, dh, drop):
    """head_dim != 64 (main.py builds 768 / 4 heads = 192 on 64 tokens): attention_generic.cu — the warp-MMA kernels
    (head_dim % 16 == 0) and the CUDA-core kernels (any head_dim % 8 == 0; forced with SFC_ATTN_NO_MMA=1)."""
    import torch
    from sfcvit import ops
    monkeypatch.setenv("SFC_ATTN_NO_MMA", "0" if mma else "1")
    g = torch.Generator(device="cuda").manual_seed(3)
    D = H * dh
    qkv = torch.randn(B * N, 3 * D, generator=g, device="cuda").bfloat16()
    out, lse = ops.attn_fwd(qkv, B, H, N, drop_p=drop, drop_seed=11)
    q, k, v = [t.reshape(B, N, H, dh).permute(0, 2, 1, 3).float().requires_grad_(True) for t in qkv.float().split(D, dim=1)]
    s = (q @ k.transpose(-1, -2)) * dh ** -0.5
    assert (lse - torch.logsumexp(s, dim=-1)).abs().max() < 2e-3
    dout = torch.randn(B * N, D, generator=g, device="cuda").bfloat16()
    dqkv = ops.attn_bwd(qkv, out, dout, lse, B, H, N, drop_p=drop, drop_seed=11)
    if drop == 0.0:
        ref = (torch.softmax(s, dim=-1) @ v).permute(0, 2, 1, 3).reshape(B * N, D)
        rel = lambda a, b: float((a.float() - b).norm() / b.norm())
        assert rel(out, ref) < 1e-2
        ref.backward(dout.float())
        ref_d = torch.cat([t.grad.permute(0, 2, 1, 3).reshape(B * N, D) for t in (q, k, v)], dim=1)
        for i, name in enumerate("qkv"):
            assert rel(dqkv[:, i * D:(i + 1) * D], ref_d[:, i * D:(i + 1) * D]) < 2e-2, name
    else:
        out2, _ = ops.attn_fwd(qkv, B, H, N, drop_p=drop, drop_seed=11)
        assert torch.equal(out, out2)
        # adjoint check along V: out is linear in V for a fixed mask, so <out(V'), dout> == <dV, V'>
        vdir = torch.randn(B * N, D, generator=g, device="cuda").bfloat16()
        qkv2 = qkv.clone(); qkv2[:, 2 * D:] = vdir
        out_dir, _ = ops.attn_fwd(qkv2, B, H, N, drop_p=drop, drop_seed=11)
        lhs = float((out_dir.float() * dout.float()).sum()); rhs = float((dqkv[:, 2 * D:].float() * vdir.float()).sum())
        assert abs(lhs - rhs) / max(abs(lhs), 1e-6) < 3e-2
        assert torch.isfinite(dqkv.float()).all()


@pytest.mark.parametrize("B,H,N,dh", [(2, 4, 64, 192), (1, 2, 100, 48), (2, 2, 128, 32), (3, 1, 23, 16)])
def test_attention_generic_paths_share_the_dropout_mask(cuda_device, monkeypatch, B, H, N, dh):
    """With dropout the warp-MMA and the CUDA-core kernels must draw the SAME mask (one counter-based definition,
    indexed by (image, head, query, key)): outputs and all three gradients agree to bf16 rounding; a different mask
    would differ by O(1)."""
    import torch
    from sfcvit import ops
    g = torch.Generator(device="cuda").manual_seed(5)
    D = H * dh
    qkv = torch.randn(B * N, 3 * D, generator=g, device="cuda").bfloat16()
    dout = torch.randn(B * N, D, generator=g, device="cuda").bfloat16()
    res = {}
    for mma in ("0", "1"):
        monkeypatch.setenv("SFC_ATTN_NO_MMA", mma)
        out, lse = ops.attn_fwd(qkv, B, H, N, drop_p=0.25, drop_seed=99)
        res[mma] = (out, lse, ops.attn_bwd(qkv, out, dout, lse, B, H, N, drop_p=0.25, drop_seed=99))
    rel = lambda a, b: float((a.float() - b.float()).norm() / b.float().norm())
    assert rel(res["0"][0], res["1"][0]) < 1e-2
    assert (res["0"][1] - res["1"][1]).abs().max() < 1e-4
    for i, name in enumerate("qkv"):
        assert rel(res["0"][2][:, i * D:(i + 1) * D], res["1"][2][:, i * D:(i + 1) * D]) < 2e-2, name


# K7: token-axis linear resampling into a concat slice vs torch (F.interpolate(mode="linear", align_corners=False) on the
# same bf16 inputs in fp32; output rounded to bf16: rel-L2 <= 4e-3), and the transposed operator vs autograd of torch's.
@pytest.mark.parametrize("lens", [(64, [64, 16, 4]), (196, [196, 49, 7]), (49, [49, 196]), (100, [100, 37, 1]), (16, [16, 16])])
def test_interp_concat_matches_torch(cuda_device, lens):
    import torch
    from sfcvit import functional as SF
    n, ns = lens
    B, dims = 3, [64, 32, 8][:len(ns)]
    g = torch.Generator(device="cuda").manual_seed(1)
    streams = [torch.randn(B, s, d, generator=g, device="cuda").bfloat16().requires_grad_(True) for s, d in zip(ns, dims)]
    out = SF.concat_streams(streams, n)
    ref_in = [s.detach().float().requires_grad_(True) for s in streams]
    ref = torch.cat([r if r.shape[1] == n else torch.nn.functional.interpolate(r.transpose(1, 2), size=n, mode="linear",
                                                                              align_corners=False).transpose(1, 2)
                     for r in ref_in], dim=-1)
    assert out.shape == ref.shape and out.dtype == torch.bfloat16
    assert float((out.float() - ref).norm() / ref.norm()) < 4e-3
    off = 0
    for s in streams:                                      # equal-length streams are copied bit-exactly
        if s.shape[1] == n:
            assert torch.equal(out[:, :, off:off + s.shape[2]], s.detach())
        off += s.shape[2]
    w = torch.randn(ref.shape, generator=g, device="cuda").bfloat16()
    (out.float() * w.float()).sum().backward()
    (ref * w.float()).sum().backward()
    for s, r in zip(streams, ref_in):
        assert s.grad.dtype == torch.bfloat16
        assert float((s.grad.float() - r.grad).norm() / r.grad.norm()) < 4e-3


def test_interp_concat_rejects_bad_layout(cuda_device):
    import torch
    from sfcvit import ops
    with pytest.raises(RuntimeError):
        ops.interp_concat_fwd(torch.zeros(1, 4, 12, dtype=torch.bfloat16, device="cuda"),
                              torch.zeros(1, 8, 12, dtype=torch.bfloat16, device="cuda"), 0)


@pytest.mark.parametrize("B,C,dt", [(512, 10, "bf16"), (256, 1000, "bf16"), (37, 1000, "fp32"), (1, 3, "fp32"), (4096, 100, "bf16")])
def test_soft_target_cross_entropy_matches_reference_formula(cuda_device, B, C, dt):
    """csrc/softce.cu vs the reference criterion (/root/reference/main.py:45-51) evaluated by torch on the same inputs:
    loss (fp32), gradient w.r.t. the logits (in the logits' dtype), deterministic from run to run; mixup-style targets
    (two-hot rows) and rows that do not sum to one."""
    import torch
    import torch.nn.functional as F
    from src.training.losses import SoftTargetCrossEntropy
    g = torch.Generator(device="cuda").manual_seed(B * 31 + C)
    dtype = torch.bfloat16 if dt == "bf16" else torch.float32
    x = (torch.randn(B, C, generator=g, device="cuda") * 3).to(dtype).requires_grad_(True)
    ya, yb = torch.randint(0, C, (B,), generator=g, device="cuda"), torch.randint(0, C, (B,), generator=g, device="cuda")
    t = 0.3 * F.one_hot(ya, C).float() + 0.7 * F.one_hot(yb, C).float()
    t[0] *= 0.5                                                     # a row that does not sum to one
    loss = SoftTargetCrossEntropy()(x, t)
    (loss * 2.0).backward()
    xr = x.detach().clone().requires_grad_(True)
    ref = -(t * F.log_softmax(xr.float(), dim=-1)).sum(dim=-1).mean()
    (ref * 2.0).backward()
    assert loss.dtype == torch.float32 and loss.dim() == 0
    assert abs(float(loss) - float(ref)) < 2e-5 * max(1.0, abs(float(ref)))
    assert x.grad.dtype == dtype
    tol = 1e-5 if dt == "fp32" else 4e-3
    assert float((x.grad.float() - xr.grad.float()).norm() / xr.grad.float().norm()) < tol
    again = SoftTargetCrossEntropy()(x.detach(), t)
    assert float(again) == float(loss.detach())
