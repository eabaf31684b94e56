"""CPU checks of the FDR oracle (fdr_oracle/fdr_oracle.cpp), the authority for the device's assign_fdr: the reference's own LDA known answer,
Gauss::solve edge cases, KDE bins against a direct evaluation, Estimator::posterior_error's casts, hand-worked q-value tables, the
competition keys of a digested FASTA, and the ctypes mirrors of the new C structs."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from fdr_oracle import fdr_oracle as fo
from sage_b200 import Tolerance, api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# linear_discriminant.rs:248-280
LDA_ROWS = np.array([[5., 4., 3., 2.], [4., 5., 4., 3.], [6., 3., 4., 5.], [1., 0., 2., 9.], [5., 4., 4., 3.], [2., 1., 1., 9.5], [1., 0., 2., 8.],
                     [3., 2., -2., 10.]])
LDA_DECOY = np.array([0, 0, 0, 1, 0, 1, 1, 1], np.uint8)
LDA_EXPECTED = np.array([0.49706043, 0.48920177, 0.48920177, -0.07209359, 0.51204672, -0.02849527, -0.04924864, -0.06055943])


def test_lda_known_answer():
    coef = fo.lda_fit(LDA_ROWS, LDA_DECOY)
    s = LDA_ROWS @ coef
    assert np.all(np.abs(s / np.sqrt(np.sum(s * s)) - LDA_EXPECTED) <= 1e-8)


def test_lda_needs_both_classes():
    assert fo.lda_fit(LDA_ROWS, np.zeros(8, np.uint8)) is None
    assert fo.lda_fit(LDA_ROWS, np.ones(8, np.uint8)) is None


def test_gauss_zero_column():
    # a feature that never varies leaves a zero row and column: fill_zero's eps makes the system solvable, that coefficient is 0
    a = np.diag([2.0, 0.0, 4.0])
    x = fo.gauss_solve(a, np.array([1.0, 0.0, 2.0]))
    assert x is not None and x[1] == 0.0
    assert np.allclose(x, [1 / (2 + 1e-8), 0.0, 2 / (4 + 1e-8)], rtol=1e-15)


def test_gauss_eps_escalation():
    # 1e10 + 1e-8 == 1e10: the first eps leaves the system singular (left side not the identity); a larger eps on the ladder solves it
    a = np.full((2, 2), 1e10)
    b = np.array([1.0, 1.0])
    assert np.linalg.matrix_rank(a + 1e-8 * np.eye(2)) == 1
    x = fo.gauss_solve(a, b)
    assert x is not None and np.all(np.isfinite(x))
    ladder = []
    eps = 1e-8
    while eps <= 1.0:
        ladder.append(eps)
        eps *= 10.0
    assert any(np.allclose((a + e * np.eye(2)) @ x, b, rtol=1e-3, atol=1e-3) for e in ladder[1:])


def test_gauss_failure_and_fallback():
    assert fo.gauss_solve(np.array([[np.nan, 0.0], [0.0, 1.0]]), np.array([1.0, 1.0])) is None
    # one NaN feature poisons the scatter matrix: score_psms returns None and runner.rs falls back to the heuristic score
    f = synthetic_features(400, seed=3)
    f["hyperscore"][5] = np.nan
    rows, order, s = fo.assign_fdr(f, Tolerance.ppm(-20, 20))
    assert not s["lda_fitted"] and np.all(np.isnan(s["coef"]))
    heur = np.log1p((-f["poisson"]).astype(np.float32)) + f["longest_y_pct"] / np.float32(3.0)
    assert np.allclose(rows["discriminant_score"], heur, rtol=1e-6)   # numpy's log1pf is not glibc's; the device test compares bits
    assert np.all(rows["posterior_error"] == 1.0)


def direct_bins(scores, decoy, nbins, bw_mul, monotonic):
    d, t = scores[decoy == 1], scores[decoy == 0]

    def kde(sample):
        m = math.fsum(sample) / len(sample)
        sd = math.sqrt(math.fsum((sample - m) ** 2) / len(sample))
        h = sd * (4.0 / 3.0 / len(sample)) ** 0.2 * bw_mul
        return lambda x: math.fsum(np.exp(-0.5 * ((x - sample) / h) ** 2)) / (math.sqrt(2 * math.pi) * h * len(sample))

    kd, kt = kde(d), kde(t)
    pi = len(d) / len(scores)
    lo, hi = scores.min(), scores.max()
    step = (hi - lo) / (nbins - 1)
    out = np.array([kd(b * step + lo) * pi / (kt(b * step + lo) * (1 - pi) + kd(b * step + lo) * pi) for b in range(nbins)])
    if monotonic:
        out = np.maximum.accumulate(out[::-1])[::-1]
    return out, lo, step


@pytest.mark.parametrize("nbins,bw,mono", [(1000, 1.0, True), (100, 2.0, False), (1000, 0.1, False)])
def test_kde_bins_direct(nbins, bw, mono):
    rng = np.random.default_rng(11)
    dec = (rng.random(3000) < 0.4).astype(np.uint8)
    s = np.where(dec == 1, rng.normal(0, 1, 3000), rng.normal(2.5, 1.2, 3000))
    bins, lo, step = fo.kde(s, dec, nbins, mono, bw)
    want, wlo, wstep = direct_bins(s, dec, nbins, bw, mono)
    assert lo == wlo and step == wstep
    assert np.allclose(bins, want, rtol=1e-11, atol=1e-300)


def test_posterior_error_casts():
    bins = np.array([0.9, 0.5, 0.2, 0.1])
    pe = lambda s, step=1.0: fo.posterior_error(bins, 10.0, step, s)  # noqa: E731
    assert pe(11.25) == pytest.approx(0.5 - 0.3 * 0.25)
    # below min: (score - min) / step < 0 saturates to bin 0 and extrapolates from bins 0..1
    assert pe(8.0) == pytest.approx(0.9 + (0.5 - 0.9) * -2.0)
    # above the last bin: bin_lo = bin_hi = last
    assert pe(1e300) == 0.1
    # NaN score: `NaN as usize` == 0, the interpolation then yields NaN
    assert math.isnan(pe(float("nan")))
    # step == 0 (all scores equal): 0 / 0 -> bin 0 and a NaN interpolation
    assert math.isnan(pe(10.0, step=0.0))


def spectrum_q_reference(labels_sorted):
    """qvalue.rs:8-36 restated with numpy f32 scalars."""
    q, d, t = [], 1, 0
    for is_decoy in labels_sorted:
        d, t = (d + 1, t) if is_decoy else (d, t + 1)
        with np.errstate(divide="ignore"):
            q.append(np.float32(d) / np.float32(t))
    out, q_min, passing = [], np.float32(1.0), 0
    for v in reversed(q):
        q_min = min(q_min, v)
        out.append(q_min)
        passing += q_min <= np.float32(0.01)
    return np.array(out[::-1], np.float32), passing


def test_spectrum_q_hand_table():
    disc = np.float32([5, 4, 3, 2, 1])
    dec = np.uint8([0, 0, 1, 0, 1])
    order, q, passing = fo.sort_spectrum_q(disc, dec)
    assert list(order) == [0, 1, 2, 3, 4]
    # decoy/target: 1/1, 1/2, 2/2, 2/3, 3/3 -> reverse cumulative min from 1.0
    assert np.array_equal(q, np.float32([0.5, 0.5, 2 / 3, 2 / 3, 1.0]))
    assert passing == 0


def test_spectrum_q_ties_and_decoys_count():
    # 300 targets above one decoy: every q <= 0.01, and spectrum_q_value counts the decoy row as passing too
    disc = np.concatenate([np.linspace(10, 5, 300), [1.0]]).astype(np.float32)
    dec = np.concatenate([np.zeros(300), [1]]).astype(np.uint8)
    order, q, passing = fo.sort_spectrum_q(disc, dec)
    want, wp = spectrum_q_reference(dec[order])
    assert np.array_equal(q, want) and passing == wp == 301
    # equal scores keep input order
    order, _, _ = fo.sort_spectrum_q(np.float32([1, 2, 2, 1, 2]), np.zeros(5, np.uint8))
    assert list(order) == [1, 2, 4, 0, 3]


def competition_reference(disc, dec, key, n_keys):
    """fdr.rs:59-120 restated: keys in order, rows sorted stably by score, PEP from the oracle's KDE."""
    fwd, rev = {}, {}
    for s, d, k in zip(disc, dec, key):
        if k == fo.NO_KEY:
            continue
        side = rev if d else fwd
        side[k] = max(side.get(k, np.float32(-3.4028235e38)), s)
    keys = sorted(set(fwd) | set(rev))
    lo = np.float32(-3.4028235e38)
    scores = [float(max(fwd.get(k, lo), rev.get(k, lo))) for k in keys]
    isdec = [rev.get(k, lo) >= fwd.get(k, lo) for k in keys]
    bins, mn, step = fo.kde(np.array(scores), np.array(isdec, np.uint8), 1000, True, 1.0)
    rows = [(k, False, fwd[k]) for k in keys if k in fwd] + [(k, True, rev[k]) for k in keys if k in rev]
    rows.sort(key=lambda r: (r[0], r[1]))
    rows.sort(key=lambda r: -float(r[2]))
    dsum, tsum, q = np.float32(1.0), np.float32(0.0), []
    for k, d, s in rows:
        dsum = np.float32(dsum + np.float32(fo.posterior_error(bins, mn, step, float(s))))
        tsum = np.float32(tsum + (0 if d else 1))
        with np.errstate(divide="ignore"):
            q.append(dsum / tsum)
    q_min, passing, qs = np.float32(1.0), 0, {}
    for (k, d, s), v in zip(reversed(rows), reversed(q)):
        q_min = min(q_min, v)
        qs[(k, d)] = q_min
        passing += (q_min <= np.float32(0.01)) and not d
    return np.array([qs[(k, d)] if k != fo.NO_KEY else 1.0 for k, d in zip(key, dec)], np.float32), passing


def test_competition_hand_table():
    rng = np.random.default_rng(5)
    # 400 keys: 300 confident targets, decoys mostly low; some keys have both sides, some PSMs have no key
    n = 2000
    key = rng.integers(0, 400, n).astype(np.uint32)
    dec = (rng.random(n) < 0.3).astype(np.uint8)
    disc = np.where(dec == 1, rng.normal(0, 1, n), rng.normal(4, 1.5, n)).astype(np.float32)
    key[rng.random(n) < 0.05] = fo.NO_KEY
    q, passing = fo.competition(disc, dec, key, 400)
    want_q, want_p = competition_reference(disc, dec, key, 400)
    assert np.array_equal(q, want_q)
    assert passing == want_p
    # decoy rows may reach q <= 0.01 but never count as passing
    assert passing < int(np.sum(q[dec == 0] <= 0.01)) + int(np.sum(q[dec == 1] <= 0.01)) or not np.any(q[dec == 1] <= 0.01)


def test_competition_decoys_do_not_pass():
    # 1000 target keys, 30 low decoy keys and one decoy key among the best targets: the reverse cumulative min gives that decoy row a
    # q <= 0.01, which spectrum_q_value would count, but the competition counts targets only
    disc = np.concatenate([np.linspace(10, 5, 1000), np.linspace(0, -3, 30), [9.9]]).astype(np.float32)
    dec = np.concatenate([np.zeros(1000), np.ones(31)]).astype(np.uint8)
    key = np.arange(1031, dtype=np.uint32)
    q, passing = fo.competition(disc, dec, key, 1031)
    want_q, want_p = competition_reference(disc, dec, key, 1031)
    assert np.array_equal(q, want_q) and passing == want_p
    assert q[1030] <= 0.01 and 0 < passing == int(np.sum(q[:1000] <= 0.01))


def test_picked_keys_from_fasta():
    from oracle import oracle as O
    fasta = (">sp|P1|A\nMKWVTFISLLLLFSSAYSRGVFRRDTHKSEIAHRFKDLGEEHFKGLVLIAFSQYLQQCPFDEHVK\n"
             ">sp|P2|B\nMKWVTFISLLLLFSSAYSRGVFRRAAAPEPTTKLLLQQWK\n")
    odb = O.OracleDB.from_fasta(fasta)
    pk, prk = fo.picked_keys(odb)
    e = odb.export()
    seqs = [odb.sequence(i) for i in range(odb.n_peptides)]
    for i, s in enumerate(seqs):
        if e["decoy"][i]:
            twin = s[0] + s[1:-1][::-1] + s[-1]    # Peptide::reverse of the decoy is its target
            j = seqs.index(twin)
            assert not e["decoy"][j] and pk[i] == pk[j] and prk[i] == prk[j]
    assert len(set(pk[e["decoy"] == 0])) == int(np.sum(e["decoy"] == 0))   # targets are distinct
    shared = seqs.index("WVTFISLLLLFSSAYSR")
    assert odb.peptide_proteins(shared) == ["sp|P1|A", "sp|P2|B"] and prk[shared] == fo.NO_KEY
    one = seqs.index("AAAPEPTTK")
    assert prk[one] != fo.NO_KEY and prk[one] != prk[seqs.index("SEIAHR")]


def test_fdr_struct_layouts_match_header(tmp_path):
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu %%zu %%zu %%zu %%zu\\n", sizeof(sage_b200_fdr_params),'
                   'sizeof(sage_b200_fdr_row), sizeof(sage_b200_fdr_summary), offsetof(sage_b200_fdr_summary, lda_fitted),'
                   'offsetof(sage_b200_fdr_summary, ms_wall));return 0;}\n' % os.path.join(ROOT, "include", "sage_b200.h"))
    exe = tmp_path / "sz"
    subprocess.check_call(["/usr/bin/gcc", str(src), "-o", str(exe)])
    sizes = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert sizes == [C.sizeof(api.CFdrParams), api.FDR_DTYPE.itemsize, C.sizeof(api.CFdrSummary), api.CFdrSummary.lda_fitted.offset,
                     api.CFdrSummary.ms_wall.offset]


def test_oracle_validation():
    f = synthetic_features(100, seed=2)
    with pytest.raises(ValueError):
        fo.assign_fdr(f, Tolerance.pct(-1, 1))
    with pytest.raises(ValueError):
        fo.assign_fdr(f, Tolerance.ppm(-20, 20), peptide_key=np.zeros(10, np.uint32))   # peptide_idx >= n_peptides
    rows, order, s = fo.assign_fdr(f[:0], Tolerance.ppm(-20, 20))
    assert len(rows) == 0 and s["spectrum_passing"] == 0


def synthetic_features(n, seed):
    """Feature rows with target / decoy score distributions that differ (no search involved)."""
    rng = np.random.default_rng(seed)
    f = np.zeros(n, api.FEATURE_DTYPE)
    dec = rng.random(n) < 0.35
    f["label"] = np.where(dec, -1, 1)
    f["peptide_idx"] = rng.integers(0, 50, n)
    f["rank"] = 1
    f["charge"] = rng.integers(2, 4, n)
    f["peptide_len"] = rng.integers(7, 30, n)
    f["hyperscore"] = np.where(dec, rng.normal(20, 4, n), rng.normal(30, 6, n)).clip(1)
    f["delta_next"] = rng.exponential(2, n) + np.where(dec, 0, 3)
    f["delta_best"] = 0.0
    f["delta_mass"] = np.where(dec, rng.uniform(-20, 20, n), rng.normal(0, 3, n))
    f["expmass"], f["calcmass"] = 1500.0, 1500.0
    f["matched_peaks"] = rng.integers(4, 30, n)
    f["longest_b"], f["longest_y"] = rng.integers(0, 6, n), rng.integers(0, 8, n)
    f["longest_y_pct"] = (f["longest_y"] / f["peptide_len"]).astype(np.float32)
    f["matched_intensity_pct"] = rng.uniform(5, 60, n)
    f["poisson"] = -np.where(dec, rng.uniform(1, 5, n), rng.uniform(3, 15, n))
    f["rt"] = rng.uniform(0, 60, n)
    return f


def test_summation_order_spread():
    # the oracle with a second summation order (blocks of 64) stays within the device tolerances (DESIGN.md records the spread)
    f = synthetic_features(20000, seed=9)
    a, oa, sa = fo.assign_fdr(f, Tolerance.ppm(-20, 20))
    try:
        fo.set_block(64)
        b, ob, sb = fo.assign_fdr(f, Tolerance.ppm(-20, 20))
    finally:
        fo.set_block(0)
    assert sa["lda_fitted"] and sb["lda_fitted"]
    s = a["discriminant_score"].astype(np.float64)
    assert np.all(np.abs(s - b["discriminant_score"]) <= 1e-5 * np.maximum(1, np.abs(s)))
    assert np.max(np.abs(a["posterior_error"] - b["posterior_error"])) <= 1e-5
    assert abs(int(sa["spectrum_passing"]) - int(sb["spectrum_passing"])) <= 2
