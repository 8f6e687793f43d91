"""Full-size parity at the BASELINE.json sizes (VERDICT r1, "parity holes").

  * U1M / BC4M / P4096 A*A against the REFERENCE'S OWN CUDA operator (oracle/_ref/ref_spgemm, the reference sources compiled for
    sm_100): C.keys / C.bmps / C.offsets bit for bit through the SHA-256 of the complete arrays (the reference driver hashes its
    arrays, we hash ours), values element-wise on three windows of C blocks (first / middle / last 200 000) within the
    fp16-rounded-product tolerance of the reference kernel (1.5e-3 * sum |a||b|, SPGEMM.cu:271).
  * BC4M (full size) and R-MAT-16: conversion, SpMV and A*A against the oracle's OpenMP variants (oracle/bmsp_oracle.c;
    pinned to the scalar, reference-following functions in tests/test_oracle_golden.py): structure bit-exact, values within
    1e-3 * sum |a||b| (fp16 inputs, fp32 accumulation vs the oracle's double sums).
  * U1M / BC4M / P4096 A*A without the reference's build: the same SHA-256 digests and values at 4096 fixed positions, stored
    under tests/golden/ by tests/golden/make_fullsize_golden.py from the oracle's OpenMP product (whose C counts equal the
    reference's on these inputs).
"""
import os

import numpy as np
import pytest
import torch

from tests.util import GOLDEN, load_golden

pytestmark = pytest.mark.gpu

WINDOW = 200_000


@pytest.fixture(scope="module")
def B():
    import bmsparse_spgemm_spmv_b200 as B
    return B


@pytest.fixture(scope="module")
def refbin(oracle):
    if oracle.ref_cuda_bin("ref_spgemm") is None:
        pytest.skip("oracle/_ref/ref_spgemm not built (reference tree absent at build time)")
    return True


def _gen(B, name):
    G = B.generators
    if name == "u1m":
        nr, nc, rp, ci, v = G.uniform_random(1_000_000, 16, seed=2)
        return nr, nc, torch.from_numpy(rp).cuda(), torch.from_numpy(ci).cuda(), torch.from_numpy(v).cuda()
    if name == "p4096":
        nr, nc, rp, ci, v = G.poisson5pt(4096, 4096)
        return nr, nc, torch.from_numpy(rp).cuda(), torch.from_numpy(ci).cuda(), torch.from_numpy(v).cuda()
    if name == "bc4m":
        return G.block_clustered_torch(524288, device="cuda")
    if name == "rmat16":
        return G.rmat_torch(16, device="cuda")
    raise KeyError(name)


def _abs_matrix(B, M):
    """same structure, |values| (for the magnitude bound sum |a||b|)"""
    return B.bmSpMatrix.from_arrays(M.num_rows, M.num_cols, M.block_num, M.keys, M.bmps, M.offsets, M.values.abs(), transpose=M.transposed)


def _as_oracle(O, M, dtype):
    k, b, o, v = M.download()
    return O.OracleMatrix(M.num_rows, M.num_cols, k, b, o, v.astype(dtype), M.transposed)


@pytest.mark.parametrize("name", ["p4096", "u1m", "bc4m"])
def test_spgemm_full_size_vs_reference_cuda(B, oracle, refbin, tmp_path, name):
    O = oracle
    nr, nc, rp, ci, v = _gen(B, name)
    A = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v); Bt = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, transpose=True)
    del rp, ci, v
    # the reference indexes a compacted block-row array: only valid without empty block rows (SURVEY Appendix B)
    assert bool((A.block_row_ptr[1:] > A.block_row_ptr[:-1]).all()) and bool((Bt.block_row_ptr[1:] > Bt.block_row_ptr[:-1]).all())
    ref = O.run_ref_spgemm_digest(_as_oracle(O, A, np.float16), _as_oracle(O, Bt, np.float16), str(tmp_path), sample_blocks=WINDOW)
    C, info = B.bmSparse_mult(A, Bt)
    assert (C.block_num, C.nnz) == (ref["c_blocks"], ref["c_nnz"])
    k, b, o, vals = C.download()
    assert ref["offsets_len"] == C.block_num + 1 == o.size          # SPGEMM.cu:1087
    assert O.sha256_u64(k) == ref["sha256"]["keys"], "C.keys differ from the reference's CUDA output"
    assert O.sha256_u64(b) == ref["sha256"]["bmps"], "C.bmps differ from the reference's CUDA output"
    assert O.sha256_u64(o) == ref["sha256"]["offsets"], "C.offsets differ from the reference's CUDA output"
    # values on the sampled windows: magnitude bound from the product of the |.| matrices (same structure)
    Cm, _ = B.bmSparse_mult(_abs_matrix(B, A), _abs_matrix(B, Bt))
    mag = Cm.values
    assert Cm.block_num == C.block_num and Cm.nnz == C.nnz
    assert len(ref["windows"]) >= 1
    for w in ref["windows"]:
        b0, n = w["first_block"], w["keys"].size
        assert np.array_equal(w["keys"], k[b0:b0 + n]) and np.array_equal(w["bmps"], b[b0:b0 + n])
        assert np.array_equal(w["offsets"][:n], o[b0:b0 + n])
        v0, nv = w["first_value"], w["values"].size
        ours = vals[v0:v0 + nv].astype(np.float64)
        bound = 1.5e-3 * mag[v0:v0 + nv].cpu().numpy().astype(np.float64) + 1e-6
        assert np.all(np.abs(ours - w["values"].astype(np.float64)) <= bound), f"{name}: values differ beyond the fp16-product tolerance"


@pytest.mark.parametrize("name", ["p4096", "u1m", "bc4m"])
def test_spgemm_full_size_vs_stored_digests(B, oracle, name):
    """the products of test_spgemm_full_size_vs_reference_cuda against tests/golden/fullsize_spgemm.json and
    fullsize_spgemm_samples.npz: C.keys / C.bmps / C.offsets bit for bit through the SHA-256 of the complete arrays, values at 4096
    fixed positions within 1e-3 * sum |a||b| (fp16 inputs, fp32 accumulation vs the oracle's double sums)"""
    O = oracle
    rec = load_golden("fullsize_spgemm.json")["configs"][name]
    smp = np.load(os.path.join(GOLDEN, "fullsize_spgemm_samples.npz"))
    nr, nc, rp, ci, v = _gen(B, name)
    A = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v); Bt = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, transpose=True)
    del rp, ci, v
    C, info = B.bmSparse_mult(A, Bt)
    assert (C.block_num, C.nnz) == (rec["c_blocks"], rec["c_nnz"])
    k, b, o, vals = C.download()
    assert o.size == rec["offsets_len"]
    assert O.sha256_u64(k) == rec["sha256"]["keys"], "C.keys differ from the stored digest"
    assert O.sha256_u64(b) == rec["sha256"]["bmps"], "C.bmps differ from the stored digest"
    assert O.sha256_u64(o) == rec["sha256"]["offsets"], "C.offsets differ from the stored digest"
    del k, b, o
    pos = smp[f"{name}_pos"]
    err = np.abs(vals[pos].astype(np.float64) - smp[f"{name}_values"])
    assert np.all(err <= 1e-3 * smp[f"{name}_mag"] + 1e-30), f"{name}: max err/mag {float(np.max(err / np.maximum(smp[f'{name}_mag'], 1e-30)))}"


@pytest.mark.parametrize("name", ["rmat16", "bc4m"])
def test_full_size_vs_openmp_oracle(B, oracle, name):
    """conversion (both orientations), SpMV and A*A against the oracle at full size; R-MAT has empty block rows (the reference itself
    cannot run it), BC4M is the dense-block config (mma.sync numeric path)"""
    O = oracle
    O.use_all_cores()
    nr, nc, rp, ci, v = _gen(B, name)
    A = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v); Bt = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, transpose=True)
    rp_h, ci_h, v_h = rp.cpu().numpy(), ci.cpu().numpy(), v.cpu().numpy()
    del rp, ci, v
    oA = O.csr_to_bmsp_omp(nr, nc, rp_h, ci_h, v_h); oB = O.csr_to_bmsp_omp(nr, nc, rp_h, ci_h, v_h, transposed=True)
    for M, e in ((A, oA), (Bt, oB)):
        k, b, o, vals = M.download()
        assert np.array_equal(k, e.keys) and np.array_equal(b, e.bmps) and np.array_equal(o, e.offsets)
        assert np.array_equal(vals.astype(np.float32), e.values)
    # SpMV
    x = B.generators.x_vector(nc)
    y = B.bmSparse_SpMV(A, torch.from_numpy(x).cuda()).cpu().numpy().astype(np.float64)
    ref = O.spmv_omp(oA, x)
    absref = O.spmv_omp(O.OracleMatrix(nr, nc, oA.keys, oA.bmps, oA.offsets, np.abs(oA.values)), np.abs(x))
    assert np.all(np.abs(y - ref) <= 1e-5 * absref + 1e-30)
    # A*A
    C, info = B.bmSparse_mult(A, Bt)
    eC = O.spgemm_omp(oA, oB)
    k, b, o, vals = C.download()
    assert np.array_equal(k, eC.keys) and np.array_equal(b, eC.bmps) and np.array_equal(o, eC.offsets)
    # magnitude bound sum |a||b| per C value: our product of the |.| matrices (its structure was just shown to be the oracle's)
    Cm, _ = B.bmSparse_mult(_abs_matrix(B, A), _abs_matrix(B, Bt))
    assert Cm.block_num == C.block_num and Cm.nnz == C.nnz
    mag = Cm.values.cpu().numpy()
    err = np.abs(vals - eC.values)
    assert np.all(err <= 1e-3 * mag + 1e-30), f"max err/mag {float(np.max(err / np.maximum(mag, 1e-30)))}"
    if name == "bc4m":
        assert info.numeric_path == 1          # dense blocks: the mma.sync pass
