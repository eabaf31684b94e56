"""The FDR stages of sage_b200_assign_fdr one by one, each against the CPU oracle (fdr_oracle/) given the device's own discriminant scores.

check_given_scores() holds any assign_fdr result to what follows from its discriminant_score column alone: the spectrum order, spectrum_q and
passing count bit for bit, and the picked peptide / protein q-values within bounds derived below, against a numpy restatement of the device's
arithmetic (tight) and against fo.competition (the reference's f32 accumulation). The heuristic fallback gives scores the caller chooses
exactly (poisson = 0 and a failed fit: disc = fl32(longest_y_pct / 3)), so crafted tables drive the sort, the competitions and the scans
through their edges: chunk and scan-tile boundaries, ties, missing sides, sparse keys, NaN / inf / ±0 / subnormal scores.

GPU tests are marked `gpu`; the restatement, its bounds and the oracle's own NaN results are checked on the CPU in the same file."""
import numpy as np
import pytest

from fdr_oracle import fdr_oracle as fo
from sage_b200 import Tolerance, api

PPM = Tolerance.ppm(-20, 20)
F32_MIN = np.float32(-3.4028235e38)
NO_KEY = fo.NO_KEY
PICK_CHUNK, SCAN_THREADS = 32, 1024   # fdr.cuh: rows per thread of the PEP-sum scan, threads of k_pick_chunk_scan


def bits(x):
    return np.asarray(x, np.float32).view(np.uint32)


def f32(b):
    return np.array(b, np.uint32).view(np.float32)


# ------------------------------------------------------------------------------------------------ numpy restatement
def total_key(x):
    u = np.asarray(x, np.float32).view(np.uint32)
    return np.where(u & 0x80000000, ~u, u | 0x80000000).astype(np.uint32)


def from_total_key(k):
    k = np.asarray(k, np.uint32)
    return np.where(k & 0x80000000, k & 0x7FFFFFFF, ~k).astype(np.uint32).view(np.float32)


def kde_pep(bins, mn, step, score):
    """Estimator::posterior_error (kde.rs:148-168) in f64, `as usize` saturating (NaN and negatives -> 0), no contraction (as the device)."""
    score = np.asarray(score, np.float64)
    last = len(bins) - 1
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        f = np.floor((score - mn) / step)
        lo = np.where(f > 0, np.minimum(np.nan_to_num(f, nan=0.0), last), 0).astype(np.int64)
        hi = np.minimum(lo + 1, last)
        lower, upper = bins[lo], bins[hi]
        linear = (score - (lo.astype(np.float64) * step + mn)) / step
        return lower + (upper - lower) * linear


def restate_competition(disc, dec, key, n_keys):
    """Competition::assign_q_value (fdr.rs:59-120) with the arithmetic the device declares (fdr.cuh k_comp_* / k_pick_*): per-key maxima in
    f32 total order with NaN skipped (so +0 beats -0); one row per present side, key by key, target first, then a stable sort by descending
    total order; the PEP from fo.kde's bins interpolated in f64, rounded to f32; the PEP prefix sum in f64; q = fl32(1 + s) / fl32(t); a
    reverse NaN-skipping min-scan from 1.0; passing counts targets. Returns per-feature q, the passing count and the sorted rows."""
    disc = np.asarray(disc, np.float32)
    dec = np.asarray(dec).astype(bool)
    key = np.asarray(key, np.uint32)
    ok = key != NO_KEY
    k, side, tk = key[ok].astype(np.int64), dec[ok].astype(np.int64), total_key(disc[ok])
    live = ~np.isnan(disc[ok])
    best = np.full((n_keys, 2), total_key(F32_MIN), np.uint32)
    np.maximum.at(best, (k[live], side[live]), tk[live])
    has = np.zeros((n_keys, 2), bool)
    has[k, side] = True
    present = np.nonzero(has.any(1))[0]
    fw, rv = best[present, 0], best[present, 1]
    kx = from_total_key(np.maximum(fw, rv)).astype(np.float64)
    kdec = from_total_key(rv) >= from_total_key(fw)
    m = has[present].ravel()
    rkey, rside, rtk = np.repeat(present, 2)[m], np.tile([0, 1], len(present))[m], best[present].ravel()[m]
    if len(rkey) == 0:
        return dict(q=np.ones(len(disc), np.float32), passing=0, rows=0)
    o = np.argsort(~rtk, kind="stable")
    rkey, rside, rtk = rkey[o], rside[o], rtk[o]
    bins, mn, step = fo.kde(kx, kdec.astype(np.uint8), 1000, True, 1.0)
    pep = kde_pep(bins, mn, step, from_total_key(rtk).astype(np.float64)).astype(np.float32)
    s = np.cumsum(pep.astype(np.float64))
    t = np.cumsum(rside == 0)
    with np.errstate(divide="ignore", invalid="ignore"):
        qpre = np.float32(1.0 + s) / t.astype(np.float32)
    qrow = np.fmin(np.float32(1.0), np.fmin.accumulate(qpre[::-1])[::-1])
    passing = int(np.sum((qrow <= np.float32(0.01)) & (rside == 0)))
    qside = np.ones(2 * n_keys, np.float32)
    qside[2 * rkey + rside] = qrow
    q = np.ones(len(disc), np.float32)
    q[ok] = qside[2 * k + side]
    return dict(q=q, passing=passing, rows=len(rkey), rkey=rkey, rside=rside, pep=pep, s=s, t=t, qpre=qpre, qrow=qrow)


def q_bounds(r):
    """Per sorted row, bounds on |Δq| before the min-scan, in two versions: (device vs restatement, oracle vs restatement).

    Before the scan, q = fl32(fl32(1 + s) / t). A change Δ in s moves it by at most Δ / t + 3 ulp(q): ½ ulp(1 + s) / t ≤ ulp(q) from each
    of the two roundings of 1 + s, and ½ ulp(q) from each of the two roundings of the quotient.
      device: its KDE bins come from another summation order and its own exp, which leaves every f32 PEP within one ulp of the
              restatement's, Δ_r ≤ Σ_{i≤r} ulp(pep_i); its f64 prefix sums run in another order, r · 2⁻⁵² · (1 + s_r) more.
      oracle: the same PEPs (fo.kde is its KDE) accumulated as `decoy += pep` in f32 from 1.0, each add within ½ ulp of its result:
              Δ_r ≤ E_r = Σ_{i≤r} ½ ulp(dsum32_i), dsum32 the sequential f32 sum.
    A NaN PEP makes every later q NaN on both sides; the scan skips those rows, and they get no term."""
    pep = np.nan_to_num(r["pep"], nan=0.0, posinf=0.0)
    n = len(pep)
    f64 = np.arange(1, n + 1) * 2.0 ** -52 * (1.0 + np.nan_to_num(r["s"], nan=0.0, posinf=0.0))
    dev = np.cumsum(np.spacing(np.abs(pep)).astype(np.float64)) + f64
    dsum32 = np.cumsum(np.concatenate([[np.float32(1.0)], pep]).astype(np.float32), dtype=np.float32)[1:]
    orc = np.cumsum(0.5 * np.spacing(np.abs(dsum32)).astype(np.float64)) + f64
    t = r["t"].astype(np.float64)
    q_ulp = 3.0 * np.spacing(np.abs(r["qpre"])).astype(np.float64)
    out = []
    for d in (dev, orc):
        with np.errstate(divide="ignore", invalid="ignore"):
            b = d / t + q_ulp
        out.append(np.where(np.isfinite(b), b, 0.0))
    return out


def q_interval(r, b):
    """Where the post-scan q of each sorted row can lie when every pre-scan q_j may move by b_j: the reverse min-scan is monotone in
    each input, so min(1, min_{j≥r} (q_j - b_j)) <= q_r <= min(1, min_{j≥r} (q_j + b_j)) (NaN rows skipped)."""
    q = np.where(np.isnan(r["qpre"]), np.inf, r["qpre"].astype(np.float64))
    scan = lambda x: np.minimum(1.0, np.minimum.accumulate(x[::-1])[::-1])   # noqa: E731
    return scan(q - b), scan(q + b)


def per_feature(r, row_values, key, dec, n_keys):
    qb = np.zeros(2 * n_keys)
    qb[2 * r["rkey"] + r["rside"]] = row_values
    out = np.ones(len(key))
    ok = key != NO_KEY
    out[ok] = qb[2 * key[ok].astype(np.int64) + dec[ok]]
    return out


def check_interval(q, passing, r, b, key, dec, n_keys, what):
    """q per feature inside the interval of b around the restatement; the passing count exact except for targets whose interval
    straddles 0.01."""
    lo, hi = q_interval(r, b)
    flo, fhi = per_feature(r, lo, key, dec, n_keys), per_feature(r, hi, key, dec, n_keys)
    q = q.astype(np.float64)
    width = np.maximum(fhi - r["q"], r["q"] - flo)
    err = np.abs(q - r["q"])
    print(f"{what}: {r['rows']} rows, max |Δq| = {float(np.max(err, initial=0)):.3g}, at most {float(np.max(err / np.maximum(width, 1e-300), initial=0)):.3g} "
          f"of its bound (max bound {float(np.max(width, initial=0)):.3g})")
    bad = (q < flo) | (q > fhi)
    assert not np.any(bad), (what, np.nonzero(bad)[0][:5], q[bad][:5], flo[bad][:5], fhi[bad][:5])
    cut = np.float64(np.float32(0.01))
    ambiguous = int(np.sum((r["rside"] == 0) & (lo <= cut) & (hi > cut)))
    assert abs(int(passing) - r["passing"]) <= ambiguous, (what, passing, r["passing"], ambiguous)


def check_competition(q, passing, disc, dec, key, n_keys, what=""):
    """Device q per feature and passing count of one picked competition against the restatement (device bound) and, through it, the
    oracle (device + oracle bounds); the oracle is checked against the restatement on the way."""
    dec = np.asarray(dec).astype(np.int64)
    key = np.asarray(key, np.uint32)
    r = restate_competition(disc, dec, key, n_keys)
    oq, opass = fo.competition(disc, dec.astype(np.uint8), key, n_keys)
    if r["rows"] == 0:
        assert np.all(q == 1.0) and passing == 0 == opass and np.all(oq == 1.0), what
        return r
    dev_b, orc_b = q_bounds(r)
    check_interval(oq, opass, r, orc_b, key, dec, n_keys, what + " oracle vs restatement")
    check_interval(q, passing, r, dev_b, key, dec, n_keys, what + " device vs restatement")
    check_interval(q, passing, r, dev_b + orc_b, key, dec, n_keys, what + " device vs restatement, with the oracle's f32 drift")
    assert np.all(q[key == NO_KEY] == 1.0)
    return r


def key_tables(pk, prk):
    n_pk = int(pk.max()) + 1 if pk is not None and len(pk) else 0
    valid = prk[prk != NO_KEY] if prk is not None else np.zeros(0, np.uint32)
    return n_pk, int(valid.max()) + 1 if len(valid) else 0


def check_given_scores(f, g, order, summary, pk=None, prk=None, n_pk=None, n_prk=None):
    """Everything that follows from the device's discriminant scores: spectrum order / q / passing exact, picked competitions bounded."""
    dec = (f["label"] == -1).astype(np.uint8)
    disc = g["discriminant_score"]
    o_order, o_q, o_pass = fo.sort_spectrum_q(disc, dec)
    assert np.array_equal(order, o_order)
    assert np.array_equal(bits(g["spectrum_q"][order]), bits(o_q))
    assert summary["spectrum_passing"] == o_pass
    d_pk, d_prk = key_tables(pk, prk)
    for table, nk, field, count in ((pk, n_pk or d_pk, "peptide_q", "peptide_passing"), (prk, n_prk or d_prk, "protein_q", "protein_passing")):
        if table is None:
            assert np.all(g[field] == 1.0) and summary[count] == 0
            continue
        check_competition(g[field], summary[count], disc, dec, table[f["peptide_idx"]], nk, field)


# ------------------------------------------------------------------------------------------------ posterior error
def posterior_error_bound(disc32, dec):
    """The oracle's log10 PEP on disc32 (fo.kde + the posterior-error interpolation) and an interval the device's value must lie in.

    The device fits its KDE to the f64 discriminants of which disc32 is the rounding, so every sample, the sample min / max and every bin
    centre can sit up to δ = ½ ulp(max |disc32|) away (bin centres 3δ: min, and b · Δstep with |Δstep| ≤ 2δ / 999).
      position: the device's PEP at its own score is the oracle's interpolation at a score within 4δ of disc32; the PEP is monotone
                (a monotone KDE), so the ends of that interval bound it.
      bins:     each Gaussian term exp(-u²/2) moves by |Δ ln| ≤ |u| · 4δ / h + u² · |η|, with |η| ≤ 2δ / σ the relative change of the
                bandwidth (σ moves by at most 2δ); a class density's relative change is the kernel-weighted mean of that, plus |η| for its
                constant. A bin = πD / (πD + (1 - π) T) moves by at most twice the larger class term, the monotone running max and the
                convex interpolation keep a relative bound (taken as the suffix maximum over bins), and reordered f64 sums add n · 2⁻⁵⁰.
    Returns (oracle log10 PEP as the device writes it, lower, upper)."""
    x = np.asarray(disc32, np.float32).astype(np.float64)
    d = np.asarray(dec).astype(bool)
    n = len(x)
    bins, mn, step = fo.kde(x, d.astype(np.uint8), 1000, True, 1.0)
    delta = 0.5 * float(np.spacing(np.float32(np.max(np.abs(x)))))
    centres = np.arange(1000) * step + mn
    eps = np.zeros(1000)
    for cls in (d, ~d):
        xs = x[cls]
        sigma = np.sqrt(np.sum((xs - np.sum(xs) / len(xs)) ** 2) / len(xs))
        h = sigma * (4.0 / 3.0 / len(xs)) ** 0.2
        eta = 2 * delta / sigma
        w = np.zeros(1000)
        a = np.zeros(1000)
        for c0 in range(0, len(xs), 1 << 15):
            u = (centres[:, None] - xs[None, c0:c0 + (1 << 15)]) / h
            k = np.exp(-0.5 * u * u)
            w += k.sum(1)
            a += (k * (np.abs(u) * 4 * delta / h + u * u * eta)).sum(1)
        with np.errstate(invalid="ignore", divide="ignore"):
            eps = np.maximum(eps, np.nan_to_num(a / w, nan=0.0, posinf=0.0) + eta)
    eps = 2 * np.maximum.accumulate(eps[::-1])[::-1] + n * 2.0 ** -50
    lo_idx = np.clip(np.floor(np.nan_to_num((x - 4 * delta - mn) / step, nan=0.0)), 0, 999).astype(np.int64)
    e = eps[lo_idx]
    with np.errstate(divide="ignore", invalid="ignore"):
        pe = np.log10(kde_pep(bins, mn, step, x)).astype(np.float32)
        hi = np.log10(kde_pep(bins, mn, step, x - 4 * delta) * (1 + e))
        lo = np.log10(kde_pep(bins, mn, step, x + 4 * delta) * (1 - e))
    pe[np.isinf(pe)] = -324.0
    lo = lo.astype(np.float32) - np.spacing(np.abs(lo).astype(np.float32))
    hi = hi.astype(np.float32) + np.spacing(np.abs(hi).astype(np.float32))
    return pe, lo, hi


def check_posterior_error(g, f):
    pe, lo, hi = posterior_error_bound(g["discriminant_score"], f["label"] == -1)
    a = g["posterior_error"]
    both = (a > -300) & (pe > -300)
    inside = (a[both] >= lo[both]) & (a[both] <= hi[both])
    half = np.maximum(hi[both] - pe[both], pe[both] - lo[both])
    print(f"posterior_error: max |Δ| {float(np.max(np.abs(a[both] - pe[both]), initial=0)):.3g}, bound median {float(np.median(half)):.3g} "
          f"max {float(np.max(half, initial=0)):.3g}")
    assert np.all(inside), np.nonzero(~inside)[0][:5]
    assert np.array_equal(np.isnan(a), np.isnan(pe))
    assert np.array_equal(a[~both & ~np.isnan(a)] <= -300, pe[~both & ~np.isnan(pe)] <= -300)


# ------------------------------------------------------------------------------------------------ crafted inputs
def fallback_features(lyp, label, poisson=None):
    """Feature rows whose fallback score is fl32(lyp / 3) (poisson = 0: log1pf(-0) = -0 adds nothing, and keeps a -0 quotient -0); one
    NaN hyperscore makes the LDA fit fail wherever both classes are present. peptide_idx = row, so the key tables are per feature."""
    n = len(lyp)
    f = np.zeros(n, api.FEATURE_DTYPE)
    f["label"] = label
    f["peptide_idx"] = np.arange(n)
    f["peptide_len"], f["charge"], f["rank"] = 7, 2, 1
    f["longest_y_pct"] = lyp
    if poisson is not None:
        f["poisson"] = poisson
    f["hyperscore"][0] = np.nan
    return f


def fallback_score(lyp):
    with np.errstate(invalid="ignore"):
        return np.float32(-0.0) + np.asarray(lyp, np.float32) / np.float32(3.0)


def competition_case(n_rows, seed, ties=None):
    """n_rows rows in one competition: n_rows // 2 keys with a target and a decoy, one more with a target alone when n_rows is odd; targets
    score higher on the whole. ties = k draws every score from k values, so equal scores cross keys and chunk boundaries."""
    rng = np.random.default_rng(seed)
    nk = n_rows // 2
    key = np.concatenate([np.repeat(np.arange(nk), 2), [nk] * (n_rows % 2)]).astype(np.uint32)
    label = np.where(np.arange(n_rows) % 2 == 1, -1, 1)
    label[2 * nk:] = 1
    if ties:
        vals = np.float32(rng.normal(0, 6, ties))
        lyp = vals[rng.integers(0, ties, n_rows)] + np.where(label == 1, np.float32(0), vals.min() - 1)
    else:
        lyp = np.where(label == 1, rng.normal(9, 3, n_rows), rng.normal(0, 3, n_rows))
    return np.float32(lyp), label, key


C, CS = PICK_CHUNK, PICK_CHUNK * SCAN_THREADS
ROW_COUNTS = [1, 2, C - 1, C, C + 1, CS - 1, CS, CS + 1, 3 * CS + 17]
BIG_ROWS = 64 * CS + 2 * 1024 + 1   # 2.1 M rows: more than 64 chunks per thread of the one-block chunk scan


def shapes_case():
    """Keys with a target only, a decoy only or both; features without a key; 10 000 features on one key (atomicMax contention); the same
    key space seen sparsely by the protein table; equal scores across keys; a target equal to its decoy (the decoy takes the KDE label);
    NaN (skipped by the maximum, the side is still present), -inf (the side stays f32::MIN), subnormals, ±0 in both orders."""
    rng = np.random.default_rng(11)
    parts = []   # (lyp, label, key)

    def add(lyp, label, key):
        parts.append((np.float32(lyp), np.asarray(label), np.asarray(key, np.uint32)))

    add(rng.normal(9, 3, 3000), 1, np.arange(0, 3000))                    # targets only
    add(rng.normal(0, 3, 2000), -1, np.arange(3000, 5000))                # decoys only
    k = np.arange(5000, 9000)
    add(rng.normal(8, 3, 4000), 1, k)                                     # both sides
    add(rng.normal(1, 3, 4000), -1, k)
    add(rng.normal(5, 3, 10_000), np.where(rng.random(10_000) < 0.3, -1, 1), np.full(10_000, 9000))   # one key, 10 000 features
    add(np.full(500, 12.0), 1, np.arange(9001, 9501))                     # equal scores across keys
    add(np.full(500, 12.0), -1, np.arange(9251, 9751))                    # ... and a target equal to its decoy on 250 keys
    add([np.nan, np.nan, 7.5, np.nan], [1, -1, -1, 1], [9800, 9800, 9801, 9802])   # NaN: the side stays present at f32::MIN
    add([-np.inf, -np.inf, 3.0], [1, -1, 1], [9803, 9804, 9804])         # -inf stays f32::MIN
    sub = np.float32(3) * f32([1, 7, 0x007fffff]) * np.float32(1)       # lyp / 3 = subnormal
    add(np.concatenate([sub, -sub]), [1, -1, 1, -1, 1, -1], [9805, 9805, 9806, 9806, 9807, 9807])
    add([0.0, -0.0, -0.0, 0.0, -0.0, -0.0, 0.0, 0.0], [1, 1, 1, 1, -1, -1, -1, -1], [9808, 9808, 9809, 9809, 9808, 9810, 9810, 9811])
    add(rng.normal(4, 3, 300), np.where(rng.random(300) < 0.5, -1, 1), np.full(300, NO_KEY))   # no key
    lyp = np.concatenate([p[0] for p in parts])
    label = np.concatenate([np.broadcast_to(p[1], len(p[0])) for p in parts])
    key = np.concatenate([p[2] for p in parts])
    perm = rng.permutation(len(lyp))
    return lyp[perm], label[perm], key[perm]


DEGENERATE = {   # lyp, label, key, n_keys: every per-key score equal (KDE step 0), no decoy side, a single key, +inf in the sample
    "all_equal": (np.full(64, 18.0), np.where(np.arange(64) % 3 == 0, -1, 1), np.arange(64) // 2, 32),
    "no_decoys": (np.arange(50) * 3.0, np.ones(50, int), np.arange(50), 50),
    "one_key": (np.array([9.0, 27.0, 3.0]), np.array([1, -1, 1]), np.zeros(3), 1),
    "plus_inf": (np.array([np.inf, 9.0, 3.0, 6.0]), np.array([1, -1, 1, -1]), np.arange(4), 4),
}


def crafted_tables():
    """(name, scores, decoy, key, n_keys) for the CPU check of the restatement against the oracle."""
    out = []
    for n in ROW_COUNTS[:5] + [4096]:
        lyp, label, key = competition_case(n, seed=n)
        out.append((f"rows{n}", lyp, label, key, int(key.max()) + 1))
    lyp, label, key = competition_case(4096, seed=3, ties=8)
    out.append(("ties", lyp, label, key, int(key.max()) + 1))
    lyp, label, key = shapes_case()
    out.append(("shapes", lyp, label, key, 10_000))
    out += [(name, *c) for name, c in DEGENERATE.items()]
    return [(name, fallback_score(lyp), np.asarray(label) == -1, np.asarray(key, np.uint32), nk) for name, lyp, label, key, nk in out]


# ------------------------------------------------------------------------------------------------ CPU: the restatement and its bounds
def test_kde_pep_matches_oracle():
    rng = np.random.default_rng(4)
    x = rng.normal(0, 2, 3000)
    bins, mn, step = fo.kde(x, (rng.random(3000) < 0.4).astype(np.uint8), 1000, True, 1.0)
    s = np.concatenate([rng.uniform(mn - 1, mn + 1000 * step + 1, 2000), [mn, mn + 999 * step, np.nan, np.inf, -np.inf, -1e300]])
    want = np.array([fo.posterior_error(bins, mn, step, float(v)) for v in s])
    got = kde_pep(bins, mn, step, s)
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64)) or np.array_equal(got, want, equal_nan=True)


@pytest.mark.parametrize("case", crafted_tables(), ids=lambda c: c[0])
def test_restatement_against_oracle(case):
    name, disc, dec, key, nk = case
    r = restate_competition(disc, dec, key, nk)
    oq, opass = fo.competition(disc, dec.astype(np.uint8), key, nk)
    if r["rows"] == 0:
        assert np.all(oq == 1.0) and opass == 0
        return
    _, orc_b = q_bounds(r)
    check_interval(oq, opass, r, orc_b, key, dec.astype(np.int64), nk, name)
    if name == "plus_inf":   # +inf in the KDE sample: every PEP NaN, every q 1.0 (the reference's too)
        assert np.all(oq == 1.0) and np.all(r["q"] == 1.0)
    if name in ("all_equal", "no_decoys"):   # step 0 / an empty class: NaN PEPs again
        assert np.all(r["q"][key != NO_KEY] == 1.0)


def test_restatement_at_a_million_rows():
    lyp, label, key = competition_case(1_000_000, seed=77)
    disc, dec, nk = fallback_score(lyp), (label == -1).astype(np.int64), int(key.max()) + 1
    r = restate_competition(disc, dec, key, nk)
    oq, opass = fo.competition(disc, dec.astype(np.uint8), key, nk)
    _, orc_b = q_bounds(r)
    check_interval(oq, opass, r, orc_b, key, dec, nk, "1e6 rows")
    assert r["passing"] > 0


@pytest.mark.parametrize("n", [1000, 10_000])
def test_bounds_are_tight_on_small_tables(n):
    # the bounds must stay far below what a wrong PEP sum would move where q crosses 0.01
    lyp, label, key = competition_case(n, seed=n + 5)
    r = restate_competition(fallback_score(lyp), label == -1, key, int(key.max()) + 1)
    dev_b, orc_b = q_bounds(r)
    lo, hi = q_interval(r, dev_b + orc_b)
    near = np.abs(r["qrow"] - 0.01) <= 0.005
    assert np.any(near)
    assert np.max((hi - lo)[near]) < 1e-5


def test_oracle_fallback_nan_bits():
    """The host's fallback score (fo.assign_fdr, x86-64 SSE arithmetic) on NaN and invalid inputs: these bits are what the device
    reproduces. log1pf of a value below -1 (poisson > 1) is the default NaN 0xffc00000; a NaN keeps its sign and payload, quieted, through
    the f64 negation and f32 conversion, log1pf, the division and the sum; with both addends NaN the quotient's is returned."""
    f64 = lambda b: np.array([b], np.uint64).view(np.float64)[0]   # noqa: E731
    cases = [  # poisson, longest_y_pct bits, expected discriminant bits
        (0.0, 0x7fc00000, 0x7fc00000), (0.0, 0x7fc12345, 0x7fc12345), (0.0, 0x7f812345, 0x7fc12345), (0.0, 0xff800001, 0xffc00001),
        (2.0, 0x3f800000, 0xffc00000), (np.inf, 0x3f800000, 0xffc00000), (2.0, 0x7fc12345, 0x7fc12345), (2.0, 0xffc12345, 0xffc12345),
        (f64(0x7ff8000000000000), 0x3f800000, 0xffc00000), (f64(0x7ff8000123456789), 0x3f800000, 0xffc00009),
        (f64(0xfff0000123456789), 0x3f800000, 0x7fc00009), (f64(0x7ff8000123456789), 0x7fc54321, 0x7fc54321),
        (-np.inf, 0x3f800000, 0x7f800000), (-np.inf, 0xff800000, 0xffc00000), (1.0, 0x00000000, 0xff800000),
        (0.0, 0x00000000, 0x00000000), (0.0, 0x80000000, 0x80000000), (-0.0, 0x80000000, 0x00000000),
    ]
    f = fallback_features(f32([c[1] for c in cases]), np.ones(len(cases), int), poisson=[c[0] for c in cases])
    o, _, s = fo.assign_fdr(f, PPM)
    assert not s["lda_fitted"]
    assert [hex(b) for b in bits(o["discriminant_score"])] == [hex(c[2]) for c in cases]


def test_oracle_signed_zero_maximum():
    # +0 and -0 on one side of a key, in both orders: the maximum is +0 either way, so the competition does not depend on the input order
    disc = np.float32([0.0, -0.0, 1.0, 2.0, -1.0, 5.0])
    dec = np.uint8([0, 0, 1, 1, 1, 0])
    key = np.uint32([0, 0, 1, 2, 3, 4])
    a, pa = fo.competition(disc, dec, key, 5)
    p = [1, 0, 2, 3, 4, 5]
    b, pb = fo.competition(disc[p], dec[p], key[p], 5)
    assert np.array_equal(bits(a[p]), bits(b)) and pa == pb
    r = restate_competition(disc, dec, key, 5)
    assert np.array_equal(bits(r["q"]), bits(a))


# ------------------------------------------------------------------------------------------------ GPU
def run_fallback(lyp, label, pk=None, prk=None, poisson=None, **kw):
    f = fallback_features(lyp, label, poisson)
    g, order, s = api.assign_fdr(f, PPM, pk, prk, **kw)
    assert not s["lda_fitted"] and np.all(g["posterior_error"] == 1.0)
    return f, g, order, s


@pytest.mark.gpu
@pytest.mark.parametrize("n_rows", ROW_COUNTS + [BIG_ROWS])
def test_competition_row_counts(n_rows):
    lyp, label, key = competition_case(n_rows, seed=n_rows)
    f, g, order, s = run_fallback(lyp, label, key)
    assert np.array_equal(bits(g["discriminant_score"]), bits(fallback_score(lyp)))
    check_given_scores(f, g, order, s, key)
    if n_rows >= 1000:
        assert s["peptide_passing"] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("ties", [1, 3, 50])
def test_competition_ties_across_chunks(ties):
    lyp, label, key = competition_case(3 * 32 * 1024 + 17, seed=ties, ties=ties)
    f, g, order, s = run_fallback(lyp, label, key)
    check_given_scores(f, g, order, s, key)


@pytest.mark.gpu
def test_competition_key_shapes_and_special_values():
    lyp, label, key = shapes_case()
    pk = key.copy()
    # the same features in a sparse table: 20 M peptide keys of which ~10 k are present, and a 3-key protein table
    # (a peptide table has no NO_KEY: those features take peptide key 0 there)
    sparse = np.where(key == NO_KEY, NO_KEY, key.astype(np.int64) * 2003 % 20_000_000).astype(np.uint32)
    small = np.where(key == NO_KEY, NO_KEY, key % 3).astype(np.uint32)
    as_pk = lambda t: np.where(t == NO_KEY, 0, t).astype(np.uint32)   # noqa: E731
    f, g, order, s = run_fallback(lyp, label, as_pk(sparse), small, n_peptide_keys=20_000_000)
    check_given_scores(f, g, order, s, as_pk(sparse), small, n_pk=20_000_000)
    f, g, order, s = run_fallback(lyp, label, as_pk(small), sparse, n_protein_keys=20_000_000)   # and the other way round
    check_given_scores(f, g, order, s, as_pk(small), sparse, n_prk=20_000_000)
    f, g, order, s = run_fallback(lyp, label, None, pk)   # one table only, with NO_KEY features
    check_given_scores(f, g, order, s, None, pk)
    f, g, order, s = run_fallback(lyp, label, as_pk(pk), np.full(len(pk), NO_KEY, np.uint32))   # every protein key NO_KEY
    check_given_scores(f, g, order, s, as_pk(pk), np.full(len(pk), NO_KEY, np.uint32))
    assert s["protein_passing"] == 0 and np.all(g["protein_q"] == 1.0)


@pytest.mark.gpu
def test_one_key_table_alone():
    # the table not given has an empty device slot: its key check must not read the buffer that slot aliases (a protein table alone was
    # refused with "a peptide_key is >= n_peptide_keys (0)"; a peptide table alone read stale competition maxima as protein keys)
    lyp, label, key = competition_case(5000, seed=12)
    for pk, prk in ((key, None), (None, key), (key, None)):
        f, g, order, s = run_fallback(lyp, label, pk, prk)
        check_given_scores(f, g, order, s, pk, prk)
        assert s["peptide_passing" if prk is None else "protein_passing"] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["all_equal", "no_decoys", "one_key", "plus_inf"])
def test_competition_degenerate_kde(case):
    lyp, label, key, _ = DEGENERATE[case]
    key = np.asarray(key, np.uint32)
    f, g, order, s = run_fallback(np.float32(lyp), label, key)
    check_given_scores(f, g, order, s, key)
    assert np.all(g["peptide_q"] == 1.0)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 255, 256, 257, 4095, 4096, 4097, 5_000_000])
def test_spectrum_q_sizes(n):
    rng = np.random.default_rng(n)
    label = np.where(rng.random(n) < 0.3, -1, 1)
    lyp = np.float32(np.where(label == 1, rng.normal(6, 3, n), rng.normal(0, 3, n)))
    lyp[rng.random(n) < 0.2] = np.float32(4.5)   # long runs of ties
    f, g, order, s = run_fallback(lyp, label)
    assert np.array_equal(bits(g["discriminant_score"]), bits(fallback_score(lyp)))
    check_given_scores(f, g, order, s)


@pytest.mark.gpu
def test_fallback_special_values_bit_exact():
    # NaN scores of several payloads and both signs (a NaN longest_y_pct, poisson > 1, a NaN poisson), ±inf and ±0, between ordinary
    # scores of both classes: the discriminant bits are the host's, and so the order and every spectrum q
    rng = np.random.default_rng(8)
    n = 3000
    label = np.where(rng.random(n) < 0.4, -1, 1)
    lyp = np.float32(rng.normal(3, 3, n))
    poisson = np.zeros(n)
    i = rng.permutation(n)[:60]
    lyp[i[:5]] = f32([0x7fc00000, 0x7fc12345, 0x7f800001, 0xffc00001, 0xffd00000])
    poisson[i[5:10]] = [2.0, 7.5, np.inf, np.nan, -np.nan]
    lyp[i[10:14]] = [np.inf, -np.inf, 0.0, -0.0]
    poisson[i[14]], lyp[i[14]] = 2.0, f32(0x7fc00042)   # both NaN
    f, g, order, s = run_fallback(lyp, label, np.arange(n, dtype=np.uint32) // 2, poisson=poisson)
    o, oo, os_ = fo.assign_fdr(f, PPM, np.arange(n, dtype=np.uint32) // 2)
    assert np.array_equal(bits(g["discriminant_score"]), bits(o["discriminant_score"]))
    assert np.array_equal(order, oo) and np.array_equal(bits(g["spectrum_q"]), bits(o["spectrum_q"]))
    assert s["spectrum_passing"] == os_["spectrum_passing"]
    assert np.array_equal(bits(g["peptide_q"]), bits(o["peptide_q"])) and s["peptide_passing"] == os_["peptide_passing"]
    check_given_scores(f, g, order, s, np.arange(n, dtype=np.uint32) // 2)


def lda_rows(n, d, seed, n_decoy=None):
    """Random rows with every column varying on its own scale and the classes separated."""
    rng = np.random.default_rng(seed)
    dec = np.zeros(n, np.uint8)
    dec[rng.permutation(n)[:n_decoy if n_decoy is not None else max(1, int(0.35 * n))]] = 1
    scale = rng.uniform(0.5, 20, d)
    rows = rng.normal(0, 1, (n, d)) * scale + rng.uniform(-50, 50, d) + np.where(dec[:, None] == 1, 0.0, 0.7 * scale)
    return rows, dec


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, 255, 256, 257, 151_552, 151_553, 1_000_000])
def test_lda_fit_edges(n):
    # TILE = 256 rows per CTA and LDA_MAX_BLOCKS = 592 CTAs (151 552 rows) before the grid-stride; d < 20 pads the rows with zeros
    for d in (1, 2, 5, 19, 20):
        for n_decoy in ([None, 1] if n == 257 else [None]):
            rows, dec = lda_rows(n, d, seed=n * 31 + d, n_decoy=n_decoy)
            ref = fo.lda_fit(rows, dec)
            assert ref is not None
            for block in (64, 1000, 7):   # the oracle's answer does not depend on its summation order
                try:
                    fo.set_block(block)
                    other = fo.lda_fit(rows, dec)
                finally:
                    fo.set_block(0)
                assert np.all(np.abs(other - ref) <= 1e-10 * np.max(np.abs(ref))), (n, d, block)
            got = api.lda_fit(rows, dec)
            assert got is not None and np.all(np.abs(got - ref) <= 1e-9 * np.max(np.abs(ref))), (n, d, n_decoy, got, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("tol", [Tolerance.da(-1500, 1500), Tolerance.ppm(-10, 200), Tolerance.da(-0.5, 0.5)], ids=["da3000", "ppm210", "da_floor"])
def test_mass_model_bin_counts(tol):
    # 3000 bins (12 bin blocks of k_kde_bins), 210 bins, and the 1000-bin floor of a narrow Da window
    from test_gpu_fdr import compare, well_conditioned_case
    f, keys, opt = well_conditioned_case()
    g, gs, stable = compare(f, tol, keys, **opt)
    assert stable and gs["lda_fitted"] and gs["peptide_passing"] > 0 and gs["protein_passing"] > 0
