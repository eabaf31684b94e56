"""The kernels rank candidates by hyperscore = ln((Σb+1)(Σy+1)) + lnfact(nb) + lnfact(ny) (scoring.rs:179-201, 495) where `ln` is the host
libm's log(). sage_b200 reproduces glibc's log() operation by operation (sage_b200/csrc/glibc_log.cuh); these tests pin that claim:
the host evaluation of both variants against libm (CPU), the device evaluation against libm (GPU), and ranks / hyperscore bits for
candidates whose products differ by one ulp (GPU)."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def log_inputs(n, seed):
    rng = np.random.default_rng(seed)
    parts = [
        (rng.integers(0, 1 << 24, n).astype(np.float32) * np.float32(0.37) + np.float32(1)).astype(np.float64) *
        (rng.integers(0, 1 << 24, n).astype(np.float32) * np.float32(1.91) + np.float32(1)).astype(np.float64),   # (Σb+1)(Σy+1): products of two f32
        0.93 + rng.random(n) * 0.15,                       # around 1: the separate near-1 branch and its edges
        rng.random(n) * 64.0,                              # lambda = matched_peaks / scored_candidates
        np.exp((rng.random(n) - 0.5) * 1400.0),            # the whole exponent range
        rng.integers(1, 1 << 52, n).astype(np.uint64).view(np.float64),   # subnormals
        np.array([0.0, 1.0, np.inf, 0.9375, 1.064697265625, np.nextafter(0.9375, 0), np.nextafter(1.064697265625, 2), 5e-324, 1.7976931348623157e308]),
    ]
    return np.concatenate(parts)


def test_host_variant_matches_libm(tmp_path):
    """CPU: the variant the library selects equals this host's libm log() bit for bit on 3e6 inputs (the C++ evaluation is the same
    template the device compiles)."""
    from sage_b200 import api
    v = api.host_log_variant()
    assert v in (0, 1), "host libm is neither glibc log variant: f64 scores are only guaranteed to 1 ulp here"
    src = os.path.join(ROOT, "tests", "glibc_log_check.cpp")
    exe = str(tmp_path / "sage_b200_glibc_log_check")
    subprocess.check_call(["g++", "-O2", "-I", os.path.join(ROOT, "sage_b200", "csrc"), src, "-o", exe])
    out = subprocess.check_output([exe, "3000000"]).decode()
    mism = dict(tok.split("=") for tok in out.split() if "=" in tok)
    assert int(mism["variant%d" % v]) == 0, out


def test_host_log1pf_matches_libm_on_every_float(tmp_path):
    """CPU, exhaustive: the log1pf the kernels evaluate (OpenMS hyperscore, f32::ln_1p) equals this host's libm log1pf on all 2^32 floats."""
    from sage_b200 import api
    assert api.host_log1pf_exact()
    src = os.path.join(ROOT, "tests", "glibc_log1pf_check.cpp")
    exe = str(tmp_path / "sage_b200_glibc_log1pf_check")
    subprocess.check_call(["g++", "-O2", "-fopenmp", "-I", os.path.join(ROOT, "sage_b200", "csrc"), src, "-o", exe])
    out = subprocess.check_output([exe]).decode()
    assert "tested 4294967296 bad 0" in out, out


@pytest.mark.gpu
def test_device_log1pf_equals_host_libm():
    from sage_b200 import api
    rng = np.random.default_rng(9)
    x = np.concatenate([rng.integers(0, 1 << 31, 300_000).astype(np.uint32).view(np.float32), (rng.random(100_000) * 2 - 0.95).astype(np.float32),
                        (rng.integers(0, 1 << 24, 100_000) * 3.7).astype(np.float32)]).astype(np.float64)
    got = api.device_log(x, 2).astype(np.float32)
    libm = ctypes.CDLL("libm.so.6")
    libm.log1pf.restype, libm.log1pf.argtypes = ctypes.c_float, [ctypes.c_float]
    sel = np.arange(0, len(x), 5)
    want = np.array([libm.log1pf(float(t)) for t in x[sel]], np.float32)
    g = got[sel]
    same = (g.view(np.uint32) == want.view(np.uint32)) | (np.isnan(g) & np.isnan(want))
    assert same.all(), f"{int((~same).sum())} differ, e.g. x={x[sel][~same][:3]}"


@pytest.mark.gpu
def test_device_log_equals_host_libm():
    from sage_b200 import api
    v = api.host_log_variant()
    assert v in (0, 1)
    x = log_inputs(400_000, 5)
    got = api.device_log(x, v)
    want = np.log(x)   # numpy's f64 log: check below that it is libm's on this build, else call libm through ctypes
    libm = ctypes.CDLL("libm.so.6")
    libm.log.restype, libm.log.argtypes = ctypes.c_double, [ctypes.c_double]
    probe = x[:: max(1, len(x) // 2000)]
    ref_probe = np.array([libm.log(float(t)) for t in probe])
    if not np.array_equal(ref_probe.view(np.uint64), np.log(probe).view(np.uint64)):
        sel = np.arange(0, len(x), max(1, len(x) // 200_000))
        x, got = x[sel], got[sel]
        want = np.array([libm.log(float(t)) for t in x])
    same = (got.view(np.uint64) == want.view(np.uint64)) | (np.isnan(got) & np.isnan(want))
    assert same.all(), f"{int((~same).sum())} of {len(x)} differ, e.g. x={x[~same][:3]} device={got[~same][:3]} libm={want[~same][:3]}"
    other = api.device_log(x, 1 - v)   # the two variants are different functions (they differ near 1): the probe is meaningful
    assert (other.view(np.uint64) != want.view(np.uint64)).any()


def near_tie_spectra(pep, n, seed):
    """Spectra built so that two candidate peptides A and B of the same precursor window match 4 b + 4 y peaks each with
    (Σb+1, Σy+1) = (a, a) for A and (a + u, a - u) for B: the f64 products a² and a² - u² differ by ~2^-47 relative, i.e. the two
    hyperscores are equal or 1-2 ulp apart and their order is decided by the last bit of log(). All sums are exact in f32 (integers and
    halves below 2^23), so the construction does not depend on summation order."""
    from sage_b200 import SpectraBatch
    from sage_b200.synth import MAX_LEN, MONO, PROTON
    rng = np.random.default_rng(seed)
    ln_all = np.diff(pep.seq_off.astype(np.int64))
    cand = np.nonzero((ln_all[:-1] >= 12) & (ln_all[1:] >= 12) & (np.diff(pep.mono) < 1.0))[0]
    pa = rng.choice(cand, size=n)
    pb = pa + 1

    def ions(choice):
        ln = ln_all[choice]
        idx = np.minimum(pep.seq_off[choice].astype(np.int64)[:, None] + np.arange(MAX_LEN)[None, :], len(pep.seq) - 1)
        rm = np.where(np.arange(MAX_LEN)[None, :] < ln[:, None], MONO[pep.seq[idx]] + pep.mods[idx], np.float32(0)).astype(np.float32)
        b = np.cumsum(rm, axis=1, dtype=np.float32)
        return b, pep.mono[choice][:, None] - b

    (ba, ya), (bb, yb) = ions(pa), ions(pb)
    cols = np.array([3, 4, 5, 6])
    masses = np.concatenate([ba[:, cols], ya[:, cols], bb[:, cols], yb[:, cols]], axis=1).astype(np.float32)    # 16 peaks
    a = rng.integers((1 << 22) + 8, (1 << 23) - 8, n).astype(np.float64)   # f32 ulp is 0.5 here: a +- 0.5 are neighbours of a
    u = rng.choice([0.5, 0.5, 1.0, 1.5], n)                                 # products differ by u^2 / a^2 ~ 2^-47 .. 2^-44 relative

    def split(total):   # 4 positive parts summing exactly to total (three integers + the remainder; multiples of 0.5, exact in f32)
        parts = rng.integers(1000, 200000, (n, 3)).astype(np.float64)
        return np.concatenate([parts, (total - parts.sum(axis=1))[:, None]], axis=1)

    inten = np.concatenate([split(a - 1), split(a - 1), split(a - 1 + u), split(a - 1 - u)], axis=1)
    assert (inten > 0).all() and np.array_equal(inten.astype(np.float32).astype(np.float64), inten)
    order = np.argsort(masses, axis=1, kind="stable")
    masses = np.take_along_axis(masses, order, axis=1)
    inten = np.take_along_axis(inten.astype(np.float32), order, axis=1)
    tic = np.cumsum(inten, axis=1, dtype=np.float32)[:, -1]
    z = np.full(n, 2, np.uint8)
    prec_mz = ((pep.mono[pa].astype(np.float64) + 2 * float(PROTON)) / 2).astype(np.float32)
    return SpectraBatch(peak_off=np.arange(n + 1, dtype=np.uint64) * np.uint64(16), masses=masses.ravel(), intensities=inten.ravel(), prec_mz=prec_mz,
                        prec_charge=z, iso_lo=np.full(n, np.nan, np.float32), iso_hi=np.full(n, np.nan, np.float32), tic=tic,
                        level=np.full(n, 2, np.uint8), rt=np.zeros(n, np.float32), ims=np.full(n, np.nan, np.float32))


def test_near_tie_construction_on_the_oracle():
    """CPU: the constructed spectra do produce top-2 candidates within a few ulp of each other in the reference algorithm (the oracle),
    including cases where glibc's log() separates them by exactly one ulp — the situation a different log() could reorder."""
    from helpers import oracle_cfg, oracle_db_from_peptides
    from sage_b200 import Tolerance, synth
    pep = synth.make_peptides(6000, seed=77)
    sp = near_tie_spectra(pep, 1500, 79)
    odb = oracle_db_from_peptides(pep)
    kw = dict(precursor_tol=Tolerance.da(-3.0, 3.0), fragment_tol=Tolerance.ppm(-10, 10), report_psms=2, min_matched_peaks=8)
    of, oc, _, _ = odb.score_batch(oracle_cfg(**kw), sp.as_dict())
    two = oc == 2
    h = of["hyperscore"].reshape(-1, 2)[two]
    d = np.abs(h[:, 0].view(np.int64) - h[:, 1].view(np.int64))
    assert two.sum() > 800 and (d <= 2).sum() > 400 and ((d >= 1) & (d <= 2)).sum() > 50 and (d == 0).sum() > 50, (two.sum(), np.bincount(np.minimum(d, 9)))


@pytest.mark.gpu
def test_rank_under_one_ulp_near_ties():
    """GPU: ranks and hyperscore / delta bits of candidates whose products differ by the minimum possible amount equal the CPU path
    (VERDICT r1 next-round item 2). With CUDA's own log() the one-ulp cases can come out in the other order."""
    from helpers import assert_features_equal, oracle_cfg, oracle_db_from_peptides
    from sage_b200 import IndexedDatabase, Scorer, Tolerance, synth
    pep = synth.make_peptides(6000, seed=77)
    sp = near_tie_spectra(pep, 4000, 80)
    gdb, odb = IndexedDatabase.build_from_peptides(pep), oracle_db_from_peptides(pep)
    kw = dict(precursor_tol=Tolerance.da(-3.0, 3.0), fragment_tol=Tolerance.ppm(-10, 10), report_psms=3, min_matched_peaks=8)
    gf, gc = Scorer(gdb, **kw).score_batch(sp)
    of, oc, _, _ = odb.score_batch(oracle_cfg(**kw), sp.as_dict())
    total = assert_features_equal(gf, gc, of, oc, 3, what="near ties", f64_exact=True)
    sel = (np.arange(len(gf)) % 3) < np.repeat(gc, 3)
    assert np.array_equal(gf["peptide_idx"][sel], of["peptide_idx"][sel]) and np.array_equal(gf["rank"][sel], of["rank"][sel])
    h = of["hyperscore"].reshape(-1, 3)[oc >= 2]
    d = np.abs(h[:, 0].view(np.int64) - h[:, 1].view(np.int64))
    assert total > 4000 and ((d >= 1) & (d <= 2)).sum() > 100 and (d == 0).sum() > 100
