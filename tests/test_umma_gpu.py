"""The tcgen05 building block of csrc/policy_umma.cu in isolation: one 128 x N x K product through the hand-packed
shared-memory / instruction descriptors, tcgen05.mma, tcgen05.commit and tcgen05.ld, against a float64 product.
A wrong descriptor field, operand layout or TMEM lane mapping shows up here as a structured error (the failing run
keeps A, W and D in its tmp_path for inspection) instead of as a wrong policy mean."""
import ctypes as C

import numpy as np
import pytest


def _probe(N, K, three_pass, seed):
    import torch
    from reinforcementlearningplatform_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(seed)
    A = rng.normal(0, 1, (128, K)).astype(np.float32)
    W = rng.normal(0, 1, (N, K)).astype(np.float32)
    a, w = torch.from_numpy(A).cuda(), torch.from_numpy(W).cuda()
    d = torch.full((128, N), float("nan"), dtype=torch.float32, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())
    _lib.check(lib.b200_umma_probe(p(a), p(w), p(d), N, K, three_pass, None), "b200_umma_probe")
    torch.cuda.synchronize()
    return A, W, d.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("N,K", [(16, 8), (64, 64), (32, 16), (256, 32), (128, 64)])
def test_umma_three_pass_product_is_fp32_accurate(N, K, tmp_path):
    A, W, D = _probe(N, K, 1, seed=N * 100 + K)
    ref = A.astype(np.float64) @ W.astype(np.float64).T
    # fp32-level accuracy: the error of each element relative to sum_k |a||w| (what an fp32 dot product is judged by);
    # 3xTF32 with fp32 accumulation measures ~5e-7, one TF32 pass ~3e-4
    err = (np.abs(D - ref) / (np.abs(A).astype(np.float64) @ np.abs(W).astype(np.float64).T)).max()
    if not err <= 1.5e-6:
        np.savez(tmp_path / f"umma_probe_fail_{N}_{K}.npz", A=A, W=W, D=D, ref=ref)
    assert err <= 1.5e-6, f"N={N} K={K}: max |D - A W^T| / (|A| |W|^T) = {err} (operands in {tmp_path})"


@pytest.mark.gpu
def test_umma_single_pass_is_tf32_accurate_only():
    """one TF32 pass: error ~2^-11 per product -- shows that the 3-pass split, not luck, gives the 2e-5 above"""
    A, W, D = _probe(64, 64, 0, seed=9)
    ref = A.astype(np.float64) @ W.astype(np.float64).T
    err = (np.abs(D - ref) / (np.abs(A).astype(np.float64) @ np.abs(W).astype(np.float64).T)).max()
    assert 2e-5 < err < 2e-3, err
