"""Generate tests/golden/fullsize_spgemm.json and fullsize_spgemm_samples.npz: what the GPU parity tests compare the B200
SpGEMM against when the reference's own CUDA build (oracle/_ref) is absent.

  python tests/golden/make_fullsize_golden.py        (after __graft_entry__.build(); CPU only, about 60 GB of RAM)

For P4096 / U1M / BC4M A*A (the inputs of tests/test_gpu_fullsize.py) the CPU oracle's OpenMP product (oracle/bmsp_oracle.c)
gives the SHA-256 of the complete C.keys / C.bmps / C.offsets and, at 4096 fixed, seeded value positions, the value and the
magnitude sum |a||b| (from the product of the |.| matrices).  Before anything is written, the oracle's C block and nonzero
counts must equal the ones the reference's CUDA operator produced on a B200 (REF_COUNTS, recorded in
profiles/r1_compare_baselines.json).  For the 96 x 96 stencil of tests/test_gpu_reference_cuda.py (integer values: exact)
it gives the SHA-256 of all four C arrays, values as float32.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from oracle import oracle as O  # noqa: E402
from bmsparse_spgemm_spmv_b200 import generators as G  # noqa: E402

REF_COUNTS = {"p4096": (23038980, 218021892), "u1m": (253900089, 255969153), "bc4m": (23304023, 1433780174)}
GENS = {"p4096": lambda: G.poisson5pt(4096, 4096), "u1m": lambda: G.uniform_random(1_000_000, 16, seed=2),
        "bc4m": lambda: G.block_clustered(524288)}
SAMPLES = 4096


def sample_positions(nnz):
    return np.unique(np.random.default_rng(20261020).integers(0, nnz, SAMPLES))


def fullsize(name):
    nr, nc, rp, ci, v = GENS[name]()
    a = O.csr_to_bmsp_omp(nr, nc, rp, ci, v); bt = O.csr_to_bmsp_omp(nr, nc, rp, ci, v, transposed=True)
    del rp, ci, v
    C = O.spgemm_omp(a, bt)
    assert (C.block_num, C.nnz) == REF_COUNTS[name], (name, C.block_num, C.nnz)
    rec = {"c_blocks": C.block_num, "c_nnz": C.nnz, "offsets_len": int(C.offsets.size),
           "sha256": {"keys": O.sha256_u64(C.keys), "bmps": O.sha256_u64(C.bmps), "offsets": O.sha256_u64(C.offsets)}}
    pos = sample_positions(C.nnz)
    vals = C.values[pos].astype(np.float64)
    del C
    absm = lambda m: O.OracleMatrix(m.num_rows, m.num_cols, m.keys, m.bmps, m.offsets, np.abs(m.values), m.transposed)
    Cm = O.spgemm_omp(absm(a), absm(bt))
    assert (Cm.block_num, Cm.nnz) == REF_COUNTS[name]
    mag = Cm.values[pos].astype(np.float64)
    return rec, pos, vals, mag


def stencil96():
    nr, nc, rp, ci, v = G.poisson5pt(96, 96)
    C = O.spgemm(O.csr_to_bmsp(nr, nc, rp, ci, v), O.csr_to_bmsp(nr, nc, rp, ci, v, transposed=True))
    vals = C.values.astype(np.float32)
    assert np.array_equal(vals.astype(np.float64), C.values)          # integer-valued: exact in float32
    import hashlib
    return {"c_blocks": C.block_num, "c_nnz": C.nnz,
            "sha256": {"keys": O.sha256_u64(C.keys), "bmps": O.sha256_u64(C.bmps), "offsets": O.sha256_u64(C.offsets),
                       "values_f32": hashlib.sha256(vals.tobytes()).hexdigest()}}


if __name__ == "__main__":
    O.use_all_cores()
    out = {"source": "CPU oracle (oracle/bmsp_oracle.c, OpenMP variants) on the inputs of tests/test_gpu_fullsize.py; C counts checked "
                     "against those of the reference's CUDA operator (profiles/r1_compare_baselines.json) before writing; "
                     "written by tests/golden/make_fullsize_golden.py",
           "samples_seed": 20261020, "configs": {}, "poisson96_AxA": stencil96()}
    arrays = {}
    for name in ("p4096", "u1m", "bc4m"):
        rec, pos, vals, mag = fullsize(name)
        out["configs"][name] = rec
        arrays[f"{name}_pos"], arrays[f"{name}_values"], arrays[f"{name}_mag"] = pos, vals, mag
        print(name, rec, flush=True)
    np.savez_compressed(os.path.join(HERE, "fullsize_spgemm_samples.npz"), **arrays)
    json.dump(out, open(os.path.join(HERE, "fullsize_spgemm.json"), "w"), indent=1)
    print("golden written")
