"""The numpy dropout reference (tests/dropout_ref.py) against the C++ definition the kernels compile
(csrc/gemm_epilogue.cuh, built for the host by nvcc): keep decisions bit for bit on a few million random indices, thr16
and the float32 rescale, for both group sizes, the thr16 edge cases, 64-bit seeds and a non-zero graph epoch."""
import os
import shutil
import subprocess

import numpy as np
import pytest

import dropout_ref as dr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PK = os.path.join(ROOT, "space-filling-curves-for-vision-transformers_b200")


def _nvcc():
    cand = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    return cand if os.path.exists(cand) else shutil.which("nvcc")


@pytest.fixture(scope="module")
def host_exe(tmp_path_factory):
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip("nvcc not found")
    out = str(tmp_path_factory.mktemp("dropout_host") / "dropout_host")
    subprocess.check_call([nvcc, "-std=c++17", "-O2", "--expt-relaxed-constexpr", "-gencode", "arch=compute_100a,code=sm_100a",
                           "-I", os.path.join(ROOT, "include"), "-I", os.path.join(PK, "csrc"), "-o", out,
                           os.path.join(ROOT, "tests", "host", "dropout_host.cu")])
    return out


def _run(exe, seed, epoch, p, G, idx):
    r = subprocess.run([exe, str(seed), str(epoch), repr(float(p)), str(G)], input=idx.astype("<u8").tobytes(),
                       capture_output=True, check=True)
    thr = int(np.frombuffer(r.stdout[:4], "<u4")[0])
    inv = float(np.frombuffer(r.stdout[4:8], "<f4")[0])
    keep = np.frombuffer(r.stdout[8:], np.uint8).astype(bool)
    assert keep.size == idx.size
    return thr, inv, keep


def _indices(n, seed):
    rng = np.random.default_rng(seed)
    # small indices (first groups), contiguous runs (whole groups), and indices above 2^32 (high word of the pair hash)
    return np.concatenate([np.arange(4096, dtype=np.uint64),
                           rng.integers(0, 1 << 31, n // 2, dtype=np.uint64),
                           rng.integers(0, 1 << 62, n // 2, dtype=np.uint64),
                           np.uint64((1 << 40) + 3) + np.arange(1000, dtype=np.uint64)])


SEEDS = [0, (1 << 32) + 5, (1 << 64) - 1]
PS = [1e-6, 0.1, 0.3, 0.5, 0.99999]


@pytest.mark.parametrize("G", [8, 16])
@pytest.mark.parametrize("seed", SEEDS)
def test_keep_mask_matches_cuda_definition(host_exe, G, seed):
    idx = _indices(1 << 20, seed & 0xFFFF)
    for p in PS:
        for epoch in (0, 7):
            thr, inv, keep = _run(host_exe, seed, epoch, p, G, idx)
            assert thr == dr.thr16(p), (p, thr)
            assert inv == dr.inv_keep_f32(p), (p, inv)
            ref = dr.keep_mask(seed, p, idx, G, epoch)
            bad = np.flatnonzero(keep != ref)
            assert bad.size == 0, (p, epoch, bad[:8], idx[bad[:8]])


def test_thresholds_and_rescale():
    assert dr.thr16(1e-6) == 0 and dr.thr16(0.5) == 32768 and dr.thr16(0.99999) == 65535
    assert dr.thr16(0.3) == 19660                    # 0.3 * 65536 = 19660.8 rounds down
    assert dr.inv_keep(0.0) == 1.0 and dr.inv_keep(0.5) == 2.0
    assert dr.inv_keep(0.3) == 65536.0 / (65536 - 19660)
    # thr16 == 0 keeps everything; the keep rate otherwise is 1 - thr16 / 65536
    idx = np.arange(1 << 20, dtype=np.uint64)
    assert dr.keep_mask(3, 1e-6, idx, 8).all()
    for p, G in ((0.1, 8), (0.5, 16), (0.3, 16)):
        rate = dr.keep_mask(3, p, idx, G).mean()
        assert abs(rate - (1 - dr.thr16(p) / 65536)) < 4e-3, (p, G, rate)


def test_inv_keep_matches_ops():
    pytest.importorskip("torch")
    from sfcvit import ops
    for p in [0.0, 1e-6, 0.1, 0.25, 0.3, 0.5, 0.99999]:
        assert dr.inv_keep(p) == ops.drop_inv_keep(p), p


def test_seed_is_taken_modulo_2_64():
    idx = np.arange(4096, dtype=np.uint64)
    assert np.array_equal(dr.keep_mask(-1, 0.5, idx, 8), dr.keep_mask((1 << 64) - 1, 0.5, idx, 8))
    assert np.array_equal(dr.keep_mask(1 << 64, 0.5, idx, 8), dr.keep_mask(0, 0.5, idx, 8))
    # epoch e is seed + e * 0xD1B54A32D192ED03
    assert np.array_equal(dr.keep_mask(11, 0.5, idx, 16, epoch=7), dr.keep_mask(11 + 7 * dr.EPOCH_MUL, 0.5, idx, 16))
    assert not np.array_equal(dr.keep_mask(11, 0.5, idx, 16, epoch=7), dr.keep_mask(11, 0.5, idx, 16))


def test_attention_index_space():
    """((b * H + h) * N + q) * ceil16(N) + k: rows padded to 16 keys, so 16-key groups never straddle two rows."""
    B, H, N = 2, 3, 17
    idx = dr.attn_index(B, H, N)
    assert idx.shape == (B, H, N, N)
    assert int(idx[1, 2, 16, 16]) == ((1 * H + 2) * N + 16) * 32 + 16
    assert int(idx[0, 0, 1, 0]) == 32
    assert np.array_equal(dr.attn_mask(B, H, N, 5, 0.3, epoch=0), dr.keep_mask(5, 0.3, idx, 16))
    assert np.array_equal(dr.gemm_mask(3, 24, 5, 0.3, epoch=0).ravel(), dr.flat_mask(72, 5, 0.3, epoch=0))
