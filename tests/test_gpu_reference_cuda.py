"""GPU box only: pin the oracle (and through it the B200 kernels) to the REFERENCE'S OWN CUDA operators, compiled for
sm_100 from the reference tree into oracle/_ref/ (make -C oracle refcuda).  The reference is only valid on inputs with
no empty 8-row block row (SURVEY.md Appendix B), so only such inputs are used.  Results are also written to
gpurun_out/ref_cuda_golden.json; a copy is committed as tests/golden/ref_cuda_golden.json and checked on CPU."""
import json
import os

import numpy as np
import pytest

from tests.util import hex_to_u64, load_golden, random_csr

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def refbin(oracle):
    if oracle.ref_cuda_bin("ref_spgemm") is None or oracle.ref_cuda_bin("ref_spmv") is None:
        pytest.skip("oracle/_ref/ref_spgemm not built (reference tree absent at build time)")
    return True


def _values_close(ref_v, exp_v, mag):
    # the reference (multiplyV15) rounds every product to fp16 before the fp32 add (SPGEMM.cu:271): allow 2^-10 per term
    # (plus the fp16 subnormal spacing 2^-24 per term for products below 6e-5)
    return np.all(np.abs(ref_v.astype(np.float64) - exp_v) <= 1.5e-3 * mag + 1e-6)


def test_reference_cuda_matches_oracle(oracle, refbin, tmp_path):
    O = oracle
    g = load_golden("ragusa16.json")
    cases = {}
    crashed = []
    # 1. the reference's only fixture
    A = O.coo_to_bmsp(24, 24, g["A"]["rows"], g["A"]["cols"], g["A"]["vals"])
    Bt = O.coo_to_bmsp(24, 24, g["B"]["rows"], g["B"]["cols"], g["B"]["vals"], transposed=True)
    mats = {"ragusa16_AxB": (A, Bt)}
    # 2. poisson 64x64 (A*A) and a random matrix without empty block rows
    rp, ci, v = O.poisson5pt(64, 64)
    mats["poisson64_AxA"] = (O.csr_to_bmsp(4096, 4096, rp, ci, v), O.csr_to_bmsp(4096, 4096, rp, ci, v, transposed=True))
    rp, ci, v = random_csr(256, 256, 0.06, seed=77)
    mats["random256_AxA"] = (O.csr_to_bmsp(256, 256, rp, ci, v), O.csr_to_bmsp(256, 256, rp, ci, v, transposed=True))
    for name, (a, bt) in mats.items():
        assert np.all(np.diff(np.unique(a.keys >> np.uint64(32))) == 1) and (a.keys[0] >> np.uint64(32)) == 0
        exp = O.spgemm(a, bt)
        mag = O.spgemm(O.OracleMatrix(a.num_rows, a.num_cols, a.keys, a.bmps, a.offsets, np.abs(a.values)),
                       O.OracleMatrix(bt.num_rows, bt.num_cols, bt.keys, bt.bmps, bt.offsets, np.abs(bt.values), True)).values
        ran = []
        for tc, mode in ((5, 0), (4, 0), (5, 1)):     # default multiplyV15; wmma variant V14; bb_segsort route
            try:
                ref, us = O.run_ref_spgemm(a, bt, str(tmp_path), tc_version=tc, mode=mode)
            except RuntimeError as e:       # the reference itself faults on some small inputs (SURVEY.md Appendix B)
                crashed.append((name, tc, mode, str(e).splitlines()[0][:80]))
                continue
            ran.append((tc, mode))
            assert np.array_equal(ref.keys, exp.keys), (name, tc, mode)
            assert np.array_equal(ref.bmps[:exp.block_num], exp.bmps), (name, tc, mode)
            assert np.array_equal(ref.offsets[:exp.block_num + 1], exp.offsets), (name, tc, mode)
            # multiplyV15 launches C_size/2 two-warp CTAs with a grid-stride loop: every block is computed
            if tc == 5:
                assert _values_close(ref.values, exp.values, mag), (name, tc, mode)
                keep = ref
        if not ran or (5, 0) not in ran:
            continue
        ref = keep
        cases[name] = dict(C_blocks=int(exp.block_num), C_nnz=int(exp.nnz), keys_crc=int(np.bitwise_xor.reduce(ref.keys)),
                           bmps_crc=int(np.bitwise_xor.reduce(ref.bmps[:exp.block_num])), offsets_last=int(ref.offsets[exp.block_num]),
                           values_sum=float(ref.values.astype(np.float64).sum()))
    assert len(cases) >= 2, f"reference ran on too few inputs: {crashed}"
    # 3. SpMV: the shipped instantiation is fp32 matrix, x = ones
    rp, ci, v = O.poisson5pt(64, 64)
    a32 = O.csr_to_bmsp(4096, 4096, rp, ci, v, f16=False)
    y, us = O.run_ref_spmv(a32, str(tmp_path))
    exp_y = O.spmv(a32, np.ones(4096, np.float32))
    assert np.array_equal(y.astype(np.float64), exp_y)      # small integers: exact
    cases["poisson64_spmv_ones"] = dict(y_sum=float(y.sum()), y_abs_sum=float(np.abs(y).sum()))
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    json.dump(dict(source="oracle/_ref/ref_spgemm + ref_spmv = reference src/bmSparse_SPGEMM.cu, bmSparse_SPMV.cu, bmSpMatrix.cu "
                          "compiled for sm_100 and run on the B200 box", cases=cases, reference_faulted_on=crashed),
              open(os.path.join(ROOT, "gpurun_out", "ref_cuda_golden.json"), "w"), indent=1)


def test_b200_kernels_match_reference_cuda(oracle, refbin, tmp_path):
    """our CUDA path vs the reference's CUDA path directly (structure bit-exact, values within the fp16-product tolerance)"""
    import bmsparse_spgemm_spmv_b200 as B
    O = oracle
    nr, nc, rp, ci, v = B.generators.poisson5pt(96, 96)
    a = O.csr_to_bmsp(nr, nc, rp, ci, v); bt = O.csr_to_bmsp(nr, nc, rp, ci, v, transposed=True)
    ref, _ = O.run_ref_spgemm(a, bt, str(tmp_path))
    A = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v); Bt = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, transpose=True)
    for path in (0, 1):
        C, _ = B.bmSparse_mult(A, Bt, numeric_path=path)
        k, b, o, vals = C.download()
        assert np.array_equal(k, ref.keys) and np.array_equal(b, ref.bmps[:k.size]) and np.array_equal(o, ref.offsets[:k.size + 1])
        assert np.array_equal(vals, ref.values)      # integer-valued stencil: exact on both sides


def test_b200_kernels_match_stored_reference_outputs(oracle):
    """our CUDA path without the reference's build, on both numeric paths:
      * the reference's own outputs recorded in tests/golden/ref_cuda_golden.json: block and nonzero counts and the XOR of
        keys and bitmaps exact, the value sum within the fp16-product tolerance; the fp32 SpMV sums exact;
      * the 96 x 96 stencil of test_b200_kernels_match_reference_cuda: the SHA-256 of all four C arrays (integer values: exact),
        stored in tests/golden/fullsize_spgemm.json by tests/golden/make_fullsize_golden.py from the oracle."""
    import hashlib
    import torch
    import bmsparse_spgemm_spmv_b200 as B
    O = oracle
    rec = load_golden("ref_cuda_golden.json")["cases"]
    g = load_golden("ragusa16.json")
    rp, ci, v = random_csr(256, 256, 0.06, seed=77)
    _, _, prp, pci, pv = B.generators.poisson5pt(64, 64)
    mats = {"ragusa16_AxB": (B.bmSpMatrix.from_coo(24, 24, g["A"]["rows"], g["A"]["cols"], g["A"]["vals"]),
                             B.bmSpMatrix.from_coo(24, 24, g["B"]["rows"], g["B"]["cols"], g["B"]["vals"], transpose=True)),
            "poisson64_AxA": (B.bmSpMatrix.from_csr(4096, 4096, prp, pci, pv), B.bmSpMatrix.from_csr(4096, 4096, prp, pci, pv, transpose=True)),
            "random256_AxA": (B.bmSpMatrix.from_csr(256, 256, rp, ci, v), B.bmSpMatrix.from_csr(256, 256, rp, ci, v, transpose=True))}
    for name, (A, Bt) in mats.items():
        r = rec[name]
        for path in (0, 1):
            C, _ = B.bmSparse_mult(A, Bt, numeric_path=path)
            k, b, o, vals = C.download()
            assert (C.block_num, C.nnz, int(o[-1])) == (r["C_blocks"], r["C_nnz"], r["offsets_last"]), (name, path)
            assert int(np.bitwise_xor.reduce(k)) == r["keys_crc"] and int(np.bitwise_xor.reduce(b)) == r["bmps_crc"], (name, path)
            vals = vals.astype(np.float64)
            assert abs(float(vals.sum()) - r["values_sum"]) <= 2e-3 * float(np.abs(vals).sum()) + 1e-6, (name, path)
    A32 = B.bmSpMatrix.from_csr(4096, 4096, prp, pci, pv, dtype=torch.float32)
    y = B.bmSparse_SpMV(A32, torch.ones(4096, dtype=torch.float32, device="cuda")).cpu().numpy().astype(np.float64)
    assert float(y.sum()) == rec["poisson64_spmv_ones"]["y_sum"] and float(np.abs(y).sum()) == rec["poisson64_spmv_ones"]["y_abs_sum"]
    s96 = load_golden("fullsize_spgemm.json")["poisson96_AxA"]
    nr, nc, rp, ci, v = B.generators.poisson5pt(96, 96)
    A = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v); Bt = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, transpose=True)
    for path in (0, 1):
        C, _ = B.bmSparse_mult(A, Bt, numeric_path=path)
        k, b, o, vals = C.download()
        assert (C.block_num, C.nnz) == (s96["c_blocks"], s96["c_nnz"]), path
        assert (O.sha256_u64(k), O.sha256_u64(b), O.sha256_u64(o)) == (s96["sha256"]["keys"], s96["sha256"]["bmps"], s96["sha256"]["offsets"]), path
        assert hashlib.sha256(np.ascontiguousarray(vals, np.float32).tobytes()).hexdigest() == s96["sha256"]["values_f32"], path
