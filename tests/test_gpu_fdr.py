"""sage_b200_assign_fdr / sage_b200_lda_fit on the device against the CPU FDR oracle (fdr_oracle/).

Bit-exact: given the device's own discriminant scores, the order, every spectrum_q and the spectrum passing count; the whole heuristic
fallback path. Within the DESIGN.md tolerances: what follows from f64 sums in another order and the device's exp / log1p / pow / log10."""
import ctypes as C

import numpy as np
import pytest

import fdr_data as D
from fdr_oracle import fdr_oracle as fo
from helpers import oracle_cfg
from sage_b200 import IndexedDatabase, SageB200Error, Scorer, Tolerance, api

pytestmark = pytest.mark.gpu

LDA_ROWS = np.array([[5., 4., 3., 2.], [4., 5., 4., 3.], [6., 3., 4., 5.], [1., 0., 2., 9.], [5., 4., 4., 3.], [2., 1., 1., 9.5], [1., 0., 2., 8.],
                     [3., 2., -2., 10.]])
LDA_DECOY = np.array([0, 0, 0, 1, 0, 1, 1, 1], np.uint8)
LDA_EXPECTED = np.array([0.49706043, 0.48920177, 0.48920177, -0.07209359, 0.51204672, -0.02849527, -0.04924864, -0.06055943])


def test_lda_known_answer_on_device():
    coef = api.lda_fit(LDA_ROWS, LDA_DECOY)
    s = LDA_ROWS @ coef
    assert np.all(np.abs(s / np.sqrt(np.sum(s * s)) - LDA_EXPECTED) <= 1e-8)
    ref = fo.lda_fit(LDA_ROWS, LDA_DECOY)
    assert np.all(np.abs(coef - ref) <= 1e-9 * np.max(np.abs(ref)))
    assert api.lda_fit(LDA_ROWS, np.zeros(8, np.uint8)) is None


def check_exact_spectrum_q(rows, order, summary, features):
    dec = (features["label"] == -1).astype(np.uint8)
    o_order, o_q, o_pass = fo.sort_spectrum_q(rows["discriminant_score"], dec)
    assert np.array_equal(order, o_order)
    assert np.array_equal(rows["spectrum_q"][order].view(np.uint32), o_q.view(np.uint32))
    assert summary["spectrum_passing"] == o_pass


def constant_columns(f, given):
    """LDA feature columns (linear_discriminant.rs:171-192) that do not vary; column 5 (the mass model's PEP) is taken to vary."""
    cols = {0: f["rank"], 1: f["charge"], 2: f["hyperscore"], 3: f["delta_next"], 4: f["delta_best"], 6: f["isotope_error"], 7: f["average_ppm"],
            8: f["poisson"], 9: f["matched_intensity_pct"], 10: f["matched_peaks"], 11: f["longest_b"], 12: f["longest_y"],
            13: f["longest_y"] / f["peptide_len"], 14: f["peptide_len"], 15: f["missed_cleavages"], 16: given.get("aligned_rt", f["rt"]), 17: f["ims"],
            18: given.get("delta_rt_model", np.full(len(f), 0.999)), 19: given.get("delta_ims_model", np.full(len(f), 0.999))}
    return {j for j, c in cols.items() if np.nanmin(c) == np.nanmax(c)}


def oracle_stable(f, tol, keys, opt, os_):
    """Whether the reference algorithm's LDA outcome survives other summation orders (the oracle with sums in blocks of 64, 1000 and 7 terms).
    Gauss::solve pivots on the largest signed value, so with exactly-constant feature columns it can take or skip a pivot on rounding
    residue: whether the fit succeeds, and its coefficients, then depend on the order of the f64 sums alone (DESIGN.md §10), and no other
    order can be held to it."""
    for block in (64, 1000, 7):
        try:
            fo.set_block(block)
            _, _, ob = fo.assign_fdr(f, tol, *(keys or (None, None)), **opt)
        finally:
            fo.set_block(0)
        if ob["lda_fitted"] != os_["lda_fitted"]:
            return False
        if os_["lda_fitted"] and not np.all(np.abs(ob["coef"] - os_["coef"]) <= 1e-10 * np.max(np.abs(os_["coef"]))):
            return False
    return True


def compare(f, tol, keys=None, **opt):
    pk, prk = keys if keys is not None else (None, None)
    g, go, gs = api.assign_fdr(f, tol, pk, prk, **opt)
    o, oo, os_ = fo.assign_fdr(f, tol, pk, prk, **opt)
    check_exact_spectrum_q(g, go, gs, f)
    if not oracle_stable(f, tol, keys, opt, os_):
        return g, gs, False
    assert gs["lda_fitted"] == os_["lda_fitted"]
    s = o["discriminant_score"].astype(np.float64)
    assert np.all(np.abs(g["discriminant_score"] - s) <= 1e-5 * np.maximum(1.0, np.abs(s)))
    a, b = g["posterior_error"], o["posterior_error"]
    both = (a > -300) & (b > -300)
    assert np.all(np.abs(a[both] - b[both]) <= 1e-4)
    assert np.array_equal(a[~both], b[~both]) or np.all(np.isnan(a[~both]) == np.isnan(b[~both]))
    if gs["lda_fitted"]:
        const = constant_columns(f, opt)
        var = [j for j in range(20) if j not in const]
        scale = np.max(np.abs(os_["coef"][var]))
        assert np.all(np.abs(gs["coef"][var] - os_["coef"][var]) <= 1e-9 * scale), (gs["coef"], os_["coef"])
    for k in ("spectrum_passing", "peptide_passing", "protein_passing"):
        assert abs(int(gs[k]) - int(os_[k])) <= max(2, 0.001 * os_[k]), (k, gs[k], os_[k])
    for k in ("spectrum_q", "peptide_q", "protein_q"):
        assert np.mean(np.abs(g[k] - o[k]) <= 1e-4) >= 0.999, k
    return g, gs, True


@pytest.fixture(scope="module")
def fasta_data():
    odb, full, sub, rows, spectra = D.fasta_dataset(400, 6000, seed=21)
    gdb = IndexedDatabase.build_from_peptides(sub)
    keys = fo.picked_keys(odb)
    return dict(odb=odb, full=full, rows=rows, spectra=spectra, gdb=gdb, keys=keys)


def device_features(data, tol, report_psms):
    sc = Scorer(data["gdb"], precursor_tol=tol, fragment_tol=Tolerance.ppm(-20, 20), report_psms=report_psms,
                min_isotope_err=-1 if tol.kind == api.DA else 0, max_isotope_err=1 if tol.kind == api.DA else 0)
    f, c = sc.score_batch(data["spectra"])
    return D.remap(D.valid_features(f, c, report_psms), data["rows"])


@pytest.mark.parametrize("tol", [Tolerance.ppm(-20, 20), Tolerance.da(-500, 500)], ids=["ppm20", "da500"])
@pytest.mark.parametrize("report_psms", [1, 5])
@pytest.mark.parametrize("with_keys", [False, True], ids=["nokeys", "keys"])
@pytest.mark.parametrize("with_models", [False, True], ids=["norTIM", "rtim"])
def test_end_to_end_against_oracle(fasta_data, tol, report_psms, with_keys, with_models):
    f = device_features(fasta_data, tol, report_psms)
    assert len(f) > 1000 and 0 < np.sum(f["label"] == -1) < len(f)
    opt = {}
    if with_models:
        rng = np.random.default_rng(len(f))
        opt = dict(aligned_rt=rng.uniform(0, 1, len(f)).astype(np.float32), delta_rt_model=rng.uniform(0, 0.2, len(f)).astype(np.float32),
                   delta_ims_model=rng.uniform(0, 1.2, len(f)).astype(np.float32))
    g, gs, _ = compare(f, tol, fasta_data["keys"] if with_keys else None, **opt)
    assert gs["spectrum_passing"] > 0
    if with_keys:
        assert gs["peptide_passing"] > 0
        shared = fasta_data["keys"][1][f["peptide_idx"]] == fo.NO_KEY
        assert np.any(shared) and np.all(g["protein_q"][shared] == 1.0)
    else:
        assert np.all(g["peptide_q"] == 1.0) and np.all(g["protein_q"] == 1.0)


def test_fallback_is_exact(fasta_data):
    f = device_features(fasta_data, Tolerance.ppm(-20, 20), 1)
    for case in (f[f["label"] == 1], f[f["label"] == -1]):   # no decoys / no targets: score_psms returns None
        g, go, gs = api.assign_fdr(case, Tolerance.ppm(-20, 20), *fasta_data["keys"])
        o, oo, os_ = fo.assign_fdr(case, Tolerance.ppm(-20, 20), *fasta_data["keys"])
        assert not gs["lda_fitted"] and not os_["lda_fitted"]
        assert np.array_equal(g["discriminant_score"].view(np.uint32), o["discriminant_score"].view(np.uint32))
        assert np.all(g["posterior_error"] == 1.0)
        assert np.array_equal(go, oo)
        assert np.array_equal(g["spectrum_q"].view(np.uint32), o["spectrum_q"].view(np.uint32))
        assert gs["spectrum_passing"] == os_["spectrum_passing"]
    nan = f.copy()
    nan["hyperscore"][3] = np.nan   # a non-finite row makes the fit fail
    g, go, gs = api.assign_fdr(nan, Tolerance.ppm(-20, 20))
    o, oo, os_ = fo.assign_fdr(nan, Tolerance.ppm(-20, 20))
    assert not gs["lda_fitted"] and np.array_equal(g["discriminant_score"].view(np.uint32), o["discriminant_score"].view(np.uint32))
    assert np.array_equal(go, oo) and np.array_equal(g["spectrum_q"].view(np.uint32), o["spectrum_q"].view(np.uint32))


def test_small_and_degenerate_inputs(fasta_data):
    f = device_features(fasta_data, Tolerance.ppm(-20, 20), 1)
    rows, order, s = api.assign_fdr(f[:0], Tolerance.ppm(-20, 20))
    assert len(rows) == 0 and s["spectrum_passing"] == 0
    rows, order, s = api.assign_fdr(f[:1], Tolerance.ppm(-20, 20), *fasta_data["keys"])
    o, oo, os_ = fo.assign_fdr(f[:1], Tolerance.ppm(-20, 20), *fasta_data["keys"])
    assert list(order) == [0] and rows.tobytes() == o.tobytes()
    # identical rows in both classes: zero scatter, all discriminants equal, KDE step 0 -> NaN PEP; ties keep input order
    same = np.repeat(f[:1], 64)
    same["label"][::3] = -1
    rows, order, s = api.assign_fdr(same, Tolerance.ppm(-20, 20))
    o, oo, os_ = fo.assign_fdr(same, Tolerance.ppm(-20, 20))
    assert np.array_equal(order, np.arange(64)) and np.array_equal(order, oo)
    assert np.array_equal(rows["spectrum_q"].view(np.uint32), o["spectrum_q"].view(np.uint32))
    assert np.array_equal(np.isnan(rows["posterior_error"]), np.isnan(o["posterior_error"]))


def test_invalid_inputs(fasta_data):
    f = device_features(fasta_data, Tolerance.ppm(-20, 20), 1)
    pk, prk = fasta_data["keys"]
    with pytest.raises(SageB200Error) as e:
        api.assign_fdr(f, Tolerance.ppm(-20, 20), pk[:10])   # peptide_idx >= n_peptides
    assert e.value.code == -1
    with pytest.raises(SageB200Error) as e:
        api.assign_fdr(f, Tolerance.ppm(-20, 20), pk, n_peptide_keys=int(pk.max()))   # a key >= its count
    assert e.value.code == -1
    with pytest.raises(SageB200Error) as e:
        api.assign_fdr(f, Tolerance.ppm(-20, 20), None, prk, n_protein_keys=1)
    assert e.value.code == -1
    with pytest.raises(SageB200Error) as e:
        api.assign_fdr(f, Tolerance.pct(-1, 1))
    assert e.value.code == -1
    # n >= 2^32 is refused before anything is read
    p = api.CFdrParams()
    p.precursor_tol = Tolerance.ppm(-20, 20)._c()
    rc = api.load_library().sage_b200_assign_fdr(C.c_int(0), api._ptr(f), C.c_uint64(1 << 32), C.byref(p), None, None, None)
    assert rc == -5


def test_two_calls_identical(fasta_data):
    f = device_features(fasta_data, Tolerance.da(-500, 500), 5)
    a, ao, asum = api.assign_fdr(f, Tolerance.da(-500, 500), *fasta_data["keys"])
    b, bo, bsum = api.assign_fdr(f, Tolerance.da(-500, 500), *fasta_data["keys"])
    assert a.tobytes() == b.tobytes() and np.array_equal(ao, bo)
    assert np.array_equal(asum["coef"].view(np.uint64), bsum["coef"].view(np.uint64))


def test_at_size_against_oracle():
    f, full = D.at_size_features(n_batches=20, batch=50_000)
    assert len(f) > 800_000   # 1 M spectra; those without a candidate above min_matched_peaks yield no PSM
    keys = D.synthetic_keys(full)
    g, gs, _ = compare(f, Tolerance.ppm(-20, 20), keys)
    assert gs["lda_fitted"] and gs["spectrum_passing"] > 0 and gs["peptide_passing"] > 0 and gs["protein_passing"] > 0


def test_well_conditioned_against_oracle():
    # every LDA feature varies, so the solve is far from a pivot decision and the full tolerance contract applies
    from test_fdr_oracle import synthetic_features
    rng = np.random.default_rng(31)
    n = 300_000
    f = synthetic_features(n, seed=30)
    f["rank"] = rng.integers(1, 4, n)
    f["delta_best"] = rng.exponential(1, n)
    f["isotope_error"] = rng.integers(0, 2, n)
    f["missed_cleavages"] = rng.integers(0, 2, n)
    f["ims"] = rng.uniform(0.7, 1.3, n)
    f["expmass"] = f["calcmass"] + np.where(f["label"] == -1, rng.uniform(-400, 400, n), rng.normal(0, 0.01, n))
    # target peptide 2k and its decoy 2k + 1 share peptide key k; ten keys make a protein, every 17th key is shared (no protein key)
    f["peptide_idx"] = 2 * rng.integers(0, 200_000, n) + (f["label"] == -1)
    pk = (np.arange(400_000) // 2).astype(np.uint32)
    prk = np.where(pk % 17 == 0, fo.NO_KEY, pk // 10).astype(np.uint32)
    opt = dict(delta_rt_model=rng.uniform(0, 0.3, n).astype(np.float32), delta_ims_model=rng.uniform(0, 0.3, n).astype(np.float32))
    for tol in (Tolerance.ppm(-20, 20), Tolerance.da(-500, 500)):
        g, gs, stable = compare(f, tol, (pk, prk), **opt)
        assert stable and gs["lda_fitted"] and gs["peptide_passing"] > 0 and gs["protein_passing"] > 0
