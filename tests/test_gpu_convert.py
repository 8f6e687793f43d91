"""GPU parity: CSR/COO/MTX -> bmSparse through the C ABI vs the oracle (bit-exact structure and values)."""
import os

import numpy as np
import pytest
import torch

from tests.util import assert_structure_equal, csr_rows, hex_to_u64, load_golden, random_csr

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def B():
    import bmsparse_spgemm_spmv_b200 as B
    return B


def _check(B, O, nr, nc, rp, ci, v, transposed, dtype=torch.float16, device_input=False):
    if device_input:
        M = B.bmSpMatrix.from_csr(nr, nc, torch.tensor(rp, device="cuda"), torch.tensor(ci, device="cuda"),
                                  torch.tensor(v, device="cuda"), transpose=transposed, dtype=dtype)
    else:
        M = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, transpose=transposed, dtype=dtype)
    exp = O.csr_to_bmsp(nr, nc, rp, ci, v, transposed=transposed, f16=(dtype == torch.float16))
    k, b, o, vals = M.download()
    assert_structure_equal((k, b, o), exp, f"{nr}x{nc} t={transposed}")
    assert np.array_equal(vals.astype(np.float32), exp.values), "values differ"
    # derived compact arrays
    brp = M.block_row_ptr.cpu().numpy()
    nbr = (nr + 7) // 8
    exp_brp = np.searchsorted(exp.keys >> np.uint64(32), np.arange(nbr + 1, dtype=np.uint64), side="left")
    assert np.array_equal(brp, exp_brp)
    assert np.array_equal(M.block_col.cpu().numpy(), (exp.keys & np.uint64(0xFFFFFFFF)).astype(np.int32))
    return M, exp


def test_fixture(B, oracle):
    g = load_golden("ragusa16.json")
    for name, tr in (("A", False), ("B", True)):
        M = B.bmSpMatrix.from_coo(g["num_rows"], g["num_cols"], g[name]["rows"], g[name]["cols"], g[name]["vals"], transpose=tr)
        k, b, o, v = M.download()
        pre = "A" if name == "A" else "Bt"
        assert np.array_equal(k, hex_to_u64(g[f"{pre}_keys"]))
        assert np.array_equal(b, hex_to_u64(g[f"{pre}_bmps"]))
        assert o.tolist() == g[f"{pre}_offsets"]
        assert M.num_rows == 24 and M.nnz == 81 and M.block_num == 9


@pytest.mark.parametrize("shape", [(24, 24), (61, 29), (100, 7), (7, 300), (257, 513), (1000, 1000)])
@pytest.mark.parametrize("transposed", [False, True])
def test_random(B, oracle, shape, transposed):
    nr, nc = shape
    rp, ci, v = random_csr(nr, nc, 0.08, seed=nr * 31 + nc, empty_block_rows=(1,) if nr > 24 else ())
    _check(B, oracle, nr, nc, rp, ci, v, transposed)
    _check(B, oracle, nr, nc, rp, ci, v, transposed, device_input=True)


def test_fp32_values_and_dense_blocks(B, oracle):
    rp, ci, v = random_csr(200, 200, 0.6, seed=5, fp16=False)
    _check(B, oracle, 200, 200, rp, ci, v, False, dtype=torch.float32)
    _check(B, oracle, 200, 200, rp, ci, v, True, dtype=torch.float16)


@pytest.mark.parametrize("vals_dtype", [np.float16, np.float32])
@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
@pytest.mark.parametrize("transposed", [False, True])
def test_value_dtype_pairs(B, oracle, vals_dtype, dtype, transposed):
    """every (input values, stored values) dtype pair, host and device input; fp32 values that fp16 cannot hold exactly, so the
    rounding on ingest is compared too"""
    rp, ci, v = random_csr(203, 171, 0.1, seed=31, empty_block_rows=(2,), fp16=False)
    v = v.astype(vals_dtype)
    _check(B, oracle, 203, 171, rp, ci, v, transposed, dtype=dtype)
    _check(B, oracle, 203, 171, rp, ci, v, transposed, dtype=dtype, device_input=True)


def test_poisson_and_long_rows(B, oracle):
    nr, nc, rp, ci, v = B.generators.poisson5pt(64, 48)
    _check(B, oracle, nr, nc, rp, ci, v, False)
    _check(B, oracle, nr, nc, rp, ci, v, True)
    # one very long row and empty rows around it
    rng = np.random.default_rng(3)
    cols = np.sort(rng.choice(20000, 6000, replace=False)).astype(np.int32)
    rp = np.zeros(41, np.int32); rp[18:] = 6000
    rp2 = rp.copy(); extra = np.array([5, 9, 19999], np.int32)
    ci = np.concatenate([cols, extra]); rp2[31:] += 3
    v = np.arange(1, ci.size + 1, dtype=np.float32) % 7 + 1
    _check(B, oracle, 40, 20000, rp2, ci, v, False)
    _check(B, oracle, 40, 20000, rp2, ci, v, True)


def test_empty_and_tiny(B, oracle):
    M = B.bmSpMatrix.from_csr(16, 16, np.zeros(17, np.int32), np.zeros(0, np.int32), np.zeros(0, np.float32))
    assert M.block_num == 0 and M.nnz == 0
    rp = np.array([0, 1], np.int32); ci = np.array([0], np.int32); v = np.array([2.0], np.float32)
    M, exp = _check(B, oracle, 1, 1, rp, ci, v, False)
    assert M.download()[1][0] == np.uint64(1 << 63)


def test_rejects_bad_input(B):
    rp = np.array([0, 2], np.int32)
    with pytest.raises(B.BmspError) as e:
        B.bmSpMatrix.from_csr(1, 8, rp, np.array([3, 3], np.int32), np.ones(2, np.float32))
    assert e.value.code == 4       # duplicate
    with pytest.raises(B.BmspError) as e:
        B.bmSpMatrix.from_csr(1, 8, rp, np.array([5, 3], np.int32), np.ones(2, np.float32))
    assert e.value.code == 3       # unsorted
    with pytest.raises(B.BmspError) as e:
        B.bmSpMatrix.from_csr(1, 8, rp, np.array([5, 8], np.int32), np.ones(2, np.float32))
    assert e.value.code == 8       # range


def test_mtx_symmetric_and_roundtrip(B, oracle, tmp_path):
    p = tmp_path / "s.mtx"
    p.write_text("%%MatrixMarket matrix coordinate real symmetric\n% c\n5 5 4\n1 1 2.5\n3 1 -1\n5 4 7\n5 5 1e-3\n")
    M = B.bmSpMatrix(str(p), False)
    nr, nc, r, c, v = oracle.read_mtx(str(p))
    exp = oracle.coo_to_bmsp(nr, nc, r, c, v)
    k, b, o, vals = M.download()
    assert_structure_equal((k, b, o), exp)
    assert M.nnz == 6
    rr, cc, vv = M.generate_coo()
    er, ec, ev = oracle.bmsp_to_coo(exp)
    assert np.array_equal(rr, er) and np.array_equal(cc, ec) and np.array_equal(vv, ev)
    assert M.compare(er, ec, ev) == (0, 0, 0.0, 0.0)


def test_from_arrays_and_block_transpose(B, oracle):
    rp, ci, v = random_csr(150, 90, 0.15, seed=9)
    A = oracle.csr_to_bmsp(150, 90, rp, ci, v, transposed=False)
    At = oracle.csr_to_bmsp(150, 90, rp, ci, v, transposed=True)
    M = B.bmSpMatrix.from_arrays(150, 90, A.block_num, A.keys, A.bmps, A.offsets, A.values.astype(np.float16))
    k, b, o, vals = M.download()
    assert_structure_equal((k, b, o), A)
    T = M.block_transpose()
    assert T.transposed
    k, b, o, vals = T.download()
    assert_structure_equal((k, b, o), At)
    assert np.array_equal(vals.astype(np.float32), At.values)
    k2, b2, o2, v2 = T.block_transpose().download()
    assert_structure_equal((k2, b2, o2), A)
    assert np.array_equal(v2.astype(np.float32), A.values)
    # slicing block rows
    S = M.slice_block_rows(3, 11)
    ks, bs, os_, vs = S.download()
    sel = (A.keys >> np.uint64(32) >= 3) & (A.keys >> np.uint64(32) < 11)
    assert np.array_equal(ks, A.keys[sel]) and np.array_equal(bs, A.bmps[sel])
    assert np.array_equal(os_, A.offsets[sel] - A.offsets[sel][0])


@pytest.mark.parametrize("in_dtype", [torch.float16, torch.float32])
@pytest.mark.parametrize("out_dtype", [torch.float16, torch.float32])
@pytest.mark.parametrize("src_transposed", [False, True])
def test_block_transpose_dtype_pairs(B, oracle, in_dtype, out_dtype, src_transposed):
    """block_transpose from and to either dtype equals the oracle's other form of the source's stored values"""
    rp, ci, v = random_csr(150, 90, 0.15, seed=9, fp16=False)
    M = B.bmSpMatrix.from_csr(150, 90, rp, ci, v, transpose=src_transposed, dtype=in_dtype)
    stored = oracle.f16_round(v) if in_dtype == torch.float16 else v
    exp = oracle.csr_to_bmsp(150, 90, rp, ci, stored, transposed=not src_transposed, f16=(out_dtype == torch.float16))
    T = M.block_transpose(dtype=out_dtype)
    assert T.transposed != src_transposed and T.dtype == out_dtype
    k, b, o, vals = T.download()
    assert_structure_equal((k, b, o), exp)
    assert np.array_equal(vals.astype(np.float32), exp.values)


def test_device_csr_row_ptr_is_validated(B):
    """ADVICE r1: a device CSR with a bad row_ptr must be rejected, not binary-searched out of bounds."""
    import bmsparse_spgemm_spmv_b200._lib as L
    nr, nc = 64, 64
    ci = torch.arange(64, dtype=torch.int32, device="cuda"); v = torch.ones(64, device="cuda")
    good = torch.arange(65, dtype=torch.int32, device="cuda")
    assert B.bmSpMatrix.from_csr(nr, nc, good, ci, v).nnz == 64
    swapped = good.clone(); swapped[10], swapped[11] = good[11].item(), good[10].item()      # decreases once
    short = good.clone(); short[-1] = 63                                                       # does not end at nnz
    for bad in (good + 1, swapped, short, -good):
        with pytest.raises(L.BmspError) as e:
            B.bmSpMatrix.from_csr(nr, nc, bad, ci, v)
        assert e.value.code == 1


def _write(path, banner, size, lines):
    with open(path, "w") as f:
        f.write(banner + "\n% a comment\n" + size + "\n" + "\n".join(lines) + "\n")


def test_matrix_market_banners(B, tmp_path):
    """MatrixMarket parity (cusp/io/detail/matrix_market.inl:155-330 is the behavioural spec): pattern / integer / real, general /
    symmetric / skew-symmetric against scipy.io.mmread; complex, hermitian and array storage are refused; indices are range-checked;
    duplicates are rejected unless merging is asked for."""
    import scipy.io
    import scipy.sparse as sp
    import bmsparse_spgemm_spmv_b200._lib as L
    rng = np.random.default_rng(5)
    n = 37
    ent = sorted({(int(r), int(c)) for r, c in zip(rng.integers(0, n, 300), rng.integers(0, n, 300)) if r > c})     # strictly lower triangle
    diag = [(i, i) for i in range(0, n, 3)]
    cases = {
        "real general": ([(r, c) for r, c in ent] + [(c, r) for r, c in ent[:40]] + diag, False),
        "integer symmetric": (ent + diag, False),
        "real skew-symmetric": (ent, False),
        "pattern symmetric": (ent + diag, True),
        "pattern general": (ent, True),
    }
    for kind, (entries, pattern) in cases.items():
        path = str(tmp_path / (kind.replace(" ", "_") + ".mtx"))
        typ = kind.split()[0]
        lines = []
        for k, (r, c) in enumerate(entries):
            val = "" if pattern else (f" {(k % 7) - 3 or 2}" if typ == "integer" else f" {((k * 37) % 17 - 8) / 4.0 or 0.5}")
            lines.append(f"{r + 1} {c + 1}{val}")
        _write(path, f"%%MatrixMarket matrix coordinate {kind}", f"{n} {n} {len(entries)}", lines)
        ref = sp.coo_matrix(scipy.io.mmread(path)).tocsr()
        ref.sort_indices()
        M = B.bmSpMatrix(path, False, dtype=torch.float32)
        rp, ci, v = M.to_csr()
        assert np.array_equal(rp.cpu().numpy(), ref.indptr) and np.array_equal(ci.cpu().numpy(), ref.indices), kind
        assert np.array_equal(v.cpu().numpy(), ref.data.astype(np.float32)), kind
        # the device-side compare agrees: nothing missing on either side, zero error
        assert M.compare_csr(torch.from_numpy(ref.indptr).cuda(), torch.from_numpy(ref.indices).cuda(), torch.from_numpy(ref.data.astype(np.float32)).cuda()) == (0, 0, 0.0, 0.0)
    for banner in ("coordinate complex general", "coordinate real hermitian", "array real general"):
        path = str(tmp_path / "bad.mtx")
        _write(path, f"%%MatrixMarket matrix {banner}", "3 3 1", ["1 1 1.0 0.0"])
        with pytest.raises(L.BmspError) as e:
            B.bmSpMatrix(path, False)
        assert e.value.code == 7, banner                                        # BMSP_ERR_UNSUPPORTED
    path = str(tmp_path / "range.mtx")
    _write(path, "%%MatrixMarket matrix coordinate real general", "3 3 2", ["1 1 1.0", "4 2 1.0"])
    with pytest.raises(L.BmspError) as e:
        B.bmSpMatrix(path, False)
    assert e.value.code == 8                                                    # BMSP_ERR_RANGE
    path = str(tmp_path / "short.mtx")
    _write(path, "%%MatrixMarket matrix coordinate real general", "3 3 3", ["1 1 1.0", "2 2 1.0"])
    with pytest.raises(L.BmspError) as e:
        B.bmSpMatrix(path, False)
    assert e.value.code == 5                                                    # BMSP_ERR_IO
    path = str(tmp_path / "dup.mtx")
    _write(path, "%%MatrixMarket matrix coordinate real general", "9 9 4", ["1 1 1.5", "2 3 2.0", "1 1 0.25", "2 3 -2.0"])
    with pytest.raises(L.BmspError) as e:
        B.bmSpMatrix(path, False)
    assert e.value.code == 4                                                    # BMSP_ERR_DUPLICATE
    M = B.bmSpMatrix(path, False, dtype=torch.float32, merge_duplicates=True)
    rp, ci, v = M.to_csr()
    assert rp.cpu().tolist()[:3] == [0, 1, 2] and ci.cpu().tolist() == [0, 2] and v.cpu().tolist() == [1.75, 0.0]


def test_large_mtx_is_parsed_in_parallel(B, oracle, tmp_path):
    """a file above the one-thread threshold (1 MB): the sliced parse must give the same matrix as the oracle's conversion"""
    rp, ci, v = random_csr(3000, 3000, 0.02, seed=11)
    rows = csr_rows(rp)
    path = str(tmp_path / "big.mtx")
    with open(path, "w") as f:
        f.write("%%MatrixMarket matrix coordinate real general\n")
        f.write(f"3000 3000 {ci.size}\n")
        f.write("".join(f"{r + 1} {c + 1} {float(x)!r}\n" for r, c, x in zip(rows.tolist(), ci.tolist(), v.tolist())))
    assert os.path.getsize(path) > (1 << 20)
    M = B.bmSpMatrix(path, False)
    exp = oracle.csr_to_bmsp(3000, 3000, rp, ci, v)
    k, b, o, vals = M.download()
    assert_structure_equal((k, b, o), exp, "big.mtx")
    assert np.array_equal(vals.astype(np.float32), exp.values)


@pytest.mark.parametrize("gen", ["poisson", "random", "rmat", "clustered"])
def test_to_csr_and_device_compare(B, gen):
    """bmSparse -> CSR on the device gives back the CSR the matrix was built from (fp16-rounded values), and the device-side
    compare reports real numbers: missing entries on either side and the relative error of a perturbed copy"""
    G = B.generators
    if gen == "poisson": nr, nc, rp, ci, v = G.poisson5pt(70, 53)
    elif gen == "rmat": nr, nc, rp, ci, v = G.rmat(12)
    elif gen == "clustered": nr, nc, rp, ci, v = G.block_clustered(200)
    else:
        nr, nc = 1001, 777
        rp, ci, v = random_csr(nr, nc, 0.03, seed=3, empty_block_rows=(1, 5))
    M = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v)
    rp2, ci2, v2 = M.to_csr()
    assert np.array_equal(rp2.cpu().numpy(), rp) and np.array_equal(ci2.cpu().numpy(), ci)
    assert np.array_equal(v2.cpu().numpy(), v.astype(np.float16).astype(np.float32))
    assert M.compare_csr(rp2, ci2, v2) == (0, 0, 0.0, 0.0)
    # drop two entries of the other side, perturb one value
    keep = np.ones(ci.size, bool); keep[[3, ci.size // 2]] = False
    rows = csr_rows(rp)
    rp3 = np.zeros(nr + 1, np.int64); np.cumsum(np.bincount(rows[keep], minlength=nr), out=rp3[1:])
    v3 = v2.cpu().numpy()[keep].copy(); v3[10] *= 1.5
    a, b, mean, mx = M.compare_csr(torch.from_numpy(rp3.astype(np.int32)).cuda(), torch.from_numpy(ci[keep]).cuda(), torch.from_numpy(v3).cuda())
    assert (a, b) == (2, 0) and abs(mx - 1.0 / 3.0) < 1e-6 and abs(mean - (1.0 / 3.0) / (ci.size - 2)) < 1e-9
    # the host-COO entry point (any order) goes through the same device comparison
    perm = np.random.default_rng(0).permutation(ci.size)
    assert M.compare(rows[perm], ci[perm], v2.cpu().numpy()[perm]) == (0, 0, 0.0, 0.0)
    with pytest.raises(Exception):
        B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, transpose=True).to_csr()
