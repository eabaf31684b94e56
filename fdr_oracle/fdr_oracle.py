"""ctypes binding of the CPU FDR oracle (fdr_oracle/fdr_oracle.cpp): sage's score_psms, spectrum_q_value and picked peptide / protein
competitions restated on the host, with the integer-key interface of sage_b200_assign_fdr.

TEST INFRASTRUCTURE ONLY: imported by tests/ and tools/bench_fdr.py, never by the sage_b200 package."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from sage_b200.api import FDR_DTYPE, FEATURE_DTYPE, CFdrParams, CFdrSummary, Tolerance

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "fdr_oracle.cpp")
_HDR = os.path.join(os.path.dirname(_HERE), "include", "sage_b200.h")
_SO = os.path.join(_HERE, "_build", "libfdr_oracle.so")
# as oracle/Makefile: no FMA contraction, no fast-math: every f32 / f64 operation stays separately rounded, as rustc emits for the reference
CXXFLAGS = ["-O3", "-march=x86-64-v3", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC", "-Wall", "-shared"]
NO_KEY = 0xFFFFFFFF


def build(force: bool = False) -> str:
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < max(os.path.getmtime(_SRC), os.path.getmtime(_HDR)):
        os.makedirs(os.path.dirname(_SO), exist_ok=True)
        env = dict(os.environ)
        env.pop("CXX", None)
        subprocess.check_call(["/usr/bin/g++"] + CXXFLAGS + ["-o", _SO, _SRC], env=env)
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        for f in ("fo_sort_spectrum_q", "fo_competition"):
            getattr(L, f).restype = C.c_uint64
        L.fo_posterior_error.restype = C.c_double
        L.fo_posterior_error.argtypes = [C.c_void_p, C.c_uint64, C.c_double, C.c_double, C.c_double]
        _lib = L
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def set_block(block: int):
    """0: sequential f64 sums (the reference's order); B > 0: every f64 sum in blocks of B terms (a second summation order)."""
    lib().fo_set_block(C.c_uint64(int(block)))


def set_threads(n: int):
    lib().fo_set_threads(C.c_int(int(n)))


def gauss_solve(left, right):
    left = np.ascontiguousarray(left, np.float64)
    right = np.ascontiguousarray(right, np.float64)
    d = len(right)
    out = np.zeros(d)
    return out if lib().fo_gauss_solve(_p(left), _p(right), C.c_int(d), _p(out)) else None


def lda_fit(rows, decoy):
    rows = np.ascontiguousarray(rows, np.float64)
    n, d = rows.shape
    dec = np.ascontiguousarray(decoy, np.uint8)
    coef = np.zeros(d)
    return coef if lib().fo_lda_fit(_p(rows), C.c_uint64(n), C.c_int(d), _p(dec), _p(coef)) else None


def kde(scores, decoy, bins=1000, monotonic=True, bw_mul=1.0):
    """Builder::build -> (bins, min_score, score_step)."""
    s = np.ascontiguousarray(scores, np.float64)
    d = np.ascontiguousarray(decoy, np.uint8)
    out, meta = np.zeros(bins), np.zeros(2)
    lib().fo_kde(_p(s), _p(d), C.c_uint64(len(s)), C.c_uint64(bins), C.c_int(int(monotonic)), C.c_double(bw_mul), _p(out), _p(meta))
    return out, float(meta[0]), float(meta[1])


def posterior_error(bins, min_score, score_step, score) -> float:
    b = np.ascontiguousarray(bins, np.float64)
    return float(lib().fo_posterior_error(_p(b), C.c_uint64(len(b)), C.c_double(min_score), C.c_double(score_step), C.c_double(score)))


def sort_spectrum_q(disc, decoy):
    """runner.rs:289-290 (ties by input index) + spectrum_q_value -> (order, q at each rank, passing)."""
    disc = np.ascontiguousarray(disc, np.float32)
    dec = np.ascontiguousarray(decoy, np.uint8)
    n = len(disc)
    order, q = np.zeros(n, np.uint32), np.zeros(n, np.float32)
    passing = lib().fo_sort_spectrum_q(_p(disc), _p(dec), C.c_uint64(n), _p(order), _p(q))
    return order, q, int(passing)


def competition(disc, decoy, key, n_keys):
    """Competition::assign_q_value over per-feature keys (NO_KEY = not competing) -> (q per feature, passing targets)."""
    disc = np.ascontiguousarray(disc, np.float32)
    dec = np.ascontiguousarray(decoy, np.uint8)
    key = np.ascontiguousarray(key, np.uint32)
    q = np.ones(len(disc), np.float32)
    passing = lib().fo_competition(_p(disc), _p(dec), _p(key), C.c_uint64(len(disc)), C.c_uint64(int(n_keys)), _p(q))
    return q, int(passing)


def assign_fdr(features, precursor_tol: Tolerance, peptide_key=None, protein_key=None, aligned_rt=None, delta_rt_model=None, delta_ims_model=None,
               n_peptides=None, n_peptide_keys=None, n_protein_keys=None):
    """Same arguments and results as sage_b200.assign_fdr, computed on the host."""
    f = np.ascontiguousarray(features)
    assert f.dtype == FEATURE_DTYPE
    n = len(f)
    keep = []

    def arr(x, dt):
        if x is None:
            return None
        a = np.ascontiguousarray(x, dtype=dt)
        keep.append(a)
        return a

    pk, prk = arr(peptide_key, np.uint32), arr(protein_key, np.uint32)
    p = CFdrParams()
    p.precursor_tol = precursor_tol._c()
    tables = [t for t in (pk, prk) if t is not None]
    p.n_peptides = int(n_peptides if n_peptides is not None else (len(tables[0]) if tables else 0))
    if pk is not None:
        p.peptide_key = _p(pk)
        p.n_peptide_keys = int(n_peptide_keys if n_peptide_keys is not None else (int(pk.max()) + 1 if len(pk) else 0))
    if prk is not None:
        p.protein_key = _p(prk)
        valid = prk[prk != NO_KEY]
        p.n_protein_keys = int(n_protein_keys if n_protein_keys is not None else (int(valid.max()) + 1 if len(valid) else 0))
    for name, x in (("aligned_rt", aligned_rt), ("delta_rt_model", delta_rt_model), ("delta_ims_model", delta_ims_model)):
        setattr(p, name, _p(arr(x, np.float32)))
    rows = np.zeros(n, FDR_DTYPE)
    order = np.zeros(n, np.uint32)
    s = CFdrSummary()
    rc = lib().fo_assign_fdr(_p(f), C.c_uint64(n), C.byref(p), _p(rows), _p(order), C.byref(s))
    if rc != 0:
        raise ValueError(f"fdr oracle: invalid input (code {rc})")
    summary = {k: getattr(s, k) for k, _ in CFdrSummary._fields_ if k != "coef"}
    summary["coef"] = np.array(s.coef[:], np.float64)
    summary["lda_fitted"] = bool(s.lda_fitted)
    return rows, order, summary


# ------------------------------------------------------------------------------------------------ competition keys
def peptide_keys(seq_off, seq, mods, nterm, decoy, generate_decoys=True) -> np.ndarray:
    """picked_peptide's key (fdr.rs:126-131) interned to dense ids: the Display string (peptide.rs:390-407), of Peptide::reverse() for a decoy
    when the database generated its decoys (reverse keeps the first and last residue and reverses the rest, peptide.rs:307-318). Two
    peptides print the same string exactly when their N-terminal mod, residues and per-residue modification masses are equal, so those are
    the interned values."""
    ids: dict = {}
    out = np.empty(len(decoy), np.uint32)
    seq = np.asarray(seq, np.uint8)
    mods = np.asarray(mods, np.float32) + np.float32(0.0)   # -0.0 prints like 0.0 (no modification)
    for i in range(len(decoy)):
        a, b = int(seq_off[i]), int(seq_off[i + 1])
        s, m = seq[a:b], mods[a:b]
        if generate_decoys and decoy[i] and b - a - 1 > 1:
            s = np.concatenate([s[:1], s[1:-1][::-1], s[-1:]])
            m = np.concatenate([m[:1], m[1:-1][::-1], m[-1:]])
        nt = None if np.isnan(nterm[i]) else float(nterm[i])
        out[i] = ids.setdefault((nt, s.tobytes(), m.tobytes()), len(ids))
    return out


def protein_keys(proteins) -> np.ndarray:
    """picked_protein's key (fdr.rs:159-165) interned to dense ids: the Peptide::proteins vector, NO_KEY unless it has exactly one entry.
    Generated decoys keep their target's protein names, so a target and its decoy share a key."""
    ids: dict = {}
    out = np.empty(len(proteins), np.uint32)
    for i, p in enumerate(proteins):
        out[i] = ids.setdefault(tuple(p), len(ids)) if len(p) == 1 else NO_KEY
    return out


def picked_keys(odb, generate_decoys=True):
    """(peptide_key, protein_key) of an oracle.OracleDB's own peptide table (`generate_decoys` as the database was built)."""
    e = odb.export()
    pk = peptide_keys(e["seq_off"], e["seq"], e["mods"], e["nterm"], e["decoy"], generate_decoys)
    prk = protein_keys([odb.peptide_proteins(i) for i in range(odb.n_peptides)])
    return pk, prk
