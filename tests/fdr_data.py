"""Feature tables with a realistic target / decoy mix for the FDR tests and tools/bench_fdr.py.

A seeded multi-protein FASTA (with segments copied between proteins, so some peptides are shared) is digested by the oracle with generated
decoys; spectra are drawn from its target peptides, but about 30 % of the target peptides are left out of the searched index, so their
spectra match random targets and decoys. Feature.peptide_idx is mapped back to the full table, which the competition keys describe."""
import numpy as np

from oracle import oracle as O

AA = np.frombuffer(b"ACDEFGHIKLMNPQRSTVWY", np.uint8)
FREQ = np.array([8.3, 1.4, 5.5, 6.8, 3.9, 7.1, 2.3, 5.9, 5.8, 9.7, 2.4, 4.1, 4.7, 3.9, 5.5, 6.6, 5.4, 6.9, 1.1, 2.9])


def make_fasta(n_proteins: int, seed: int, mean_len: int = 350, shared_fraction: float = 0.1) -> str:
    rng = np.random.default_rng(seed)
    prots = [rng.choice(AA, size=max(60, int(rng.lognormal(np.log(mean_len), 0.4))), p=FREQ / FREQ.sum()) for _ in range(n_proteins)]
    for i in rng.choice(n_proteins, size=int(n_proteins * shared_fraction), replace=False):   # shared peptides: copy a segment
        j = int(rng.integers(n_proteins))
        a = int(rng.integers(0, len(prots[j]) - 40))
        b = int(rng.integers(0, len(prots[i]) - 40))
        prots[i] = prots[i].copy()
        prots[i][b:b + 40] = prots[j][a:a + 40]
    return "".join(f">sp|P{i:05d}|PROT{i}\n{bytes(p).decode()}\n" for i, p in enumerate(prots))


def searched_subset(decoy: np.ndarray, seed: int, drop: float = 0.3) -> np.ndarray:
    """Rows of the full table that go into the searched index: every decoy, and the targets left after dropping `drop` of them."""
    rng = np.random.default_rng(seed)
    keep = (decoy != 0) | (rng.random(len(decoy)) >= drop)
    return np.nonzero(keep)[0]


def subset_peptides(pep, rows):
    from sage_b200 import Peptides
    ln = np.diff(pep.seq_off.astype(np.int64))[rows]
    starts = pep.seq_off[:-1].astype(np.int64)[rows]
    off = np.concatenate([[0], np.cumsum(ln)])
    idx = np.repeat(starts - off[:-1], ln) + np.arange(off[-1])
    return Peptides(seq_off=np.concatenate([[0], np.cumsum(ln)]).astype(np.uint32), seq=pep.seq[idx], mods=pep.mods[idx], nterm=pep.nterm[rows],
                    mono=pep.mono[rows], decoy=pep.decoy[rows], missed=pep.missed[rows])


def valid_features(features, counts, report_psms):
    k = np.arange(len(features)) % report_psms
    return features[k < np.repeat(np.asarray(counts), report_psms)].copy()


def fasta_dataset(n_proteins=300, n_spectra=3000, seed=7):
    """(full oracle db, full Peptides, searched Peptides, subset rows, spectra) for a synthetic FASTA."""
    from sage_b200 import synth
    from helpers import peptides_from_oracle
    odb = O.OracleDB.from_fasta(make_fasta(n_proteins, seed))
    full = peptides_from_oracle(odb)
    rows = searched_subset(full.decoy, seed + 1)
    spectra = synth.make_spectra(full, n_spectra, seed=seed + 2)
    return odb, full, subset_peptides(full, rows), rows, spectra


def score_with_oracle(searched, rows, spectra, cfg):
    """Feature rows from the CPU oracle's search of `searched`, peptide_idx mapped to the full table."""
    from helpers import oracle_db_from_peptides
    sdb = oracle_db_from_peptides(searched)
    f, c, _, _ = sdb.score_batch(cfg, spectra.as_dict())
    return remap(valid_features(f, c, cfg.report_psms), rows)


def remap(features, rows):
    """Oracle Feature rows (its own dtype) or device Feature rows -> FEATURE_DTYPE with peptide_idx in the full table."""
    from sage_b200.api import FEATURE_DTYPE
    out = np.zeros(len(features), FEATURE_DTYPE)
    for name in FEATURE_DTYPE.names:
        if name in features.dtype.names and not name.startswith("_"):
            out[name] = features[name]
    if "rt" not in features.dtype.names:
        out["rt"] = 0.0
    out["peptide_idx"] = rows[features["peptide_idx"]]
    return out


def synthetic_keys(pep, proteins_per_key: int = 8, shared_fraction: float = 0.05, seed: int = 0):
    """Competition keys for a synth.make_peptides table, which has no protein names: the peptide key interns the sequence, of the reversed
    decoy for decoys (its modifications are fixed by residue, so the sequence decides the Display string); peptide keys are grouped into
    synthetic proteins of `proteins_per_key` keys, and a seeded `shared_fraction` of the peptide keys count as shared (no protein key)."""
    from sage_b200.synth import MAX_LEN
    n = len(pep)
    col = np.arange(MAX_LEN)[None, :]
    mat = np.zeros((n, MAX_LEN), np.uint8)
    for a in range(0, n, 1 << 18):   # in slices: the index arrays are 8 bytes per residue slot
        b = min(n, a + (1 << 18))
        ln = np.diff(pep.seq_off[a:b + 1].astype(np.int64))[:, None]
        # Peptide::reverse (peptide.rs:307-318): for a decoy, position j in 1..len-2 takes residue len-1-j
        inner = (col >= 1) & (col < ln - 1) & (pep.decoy[a:b, None] != 0) & (ln > 2)
        src = np.where(inner, ln - 1 - col, col)
        idx = np.minimum(pep.seq_off[a:b].astype(np.int64)[:, None] + src, max(len(pep.seq) - 1, 0))
        mat[a:b] = np.where(col < ln, pep.seq[idx], 0)
    _, pk = np.unique(np.ascontiguousarray(mat).view(f"S{MAX_LEN}").ravel(), return_inverse=True)
    pk = pk.astype(np.uint32)
    n_pk = int(pk.max()) + 1 if n else 0
    rng = np.random.default_rng(seed)
    shared = rng.random(n_pk) < shared_fraction
    prk = np.where(shared[pk], np.uint32(0xFFFFFFFF), pk // np.uint32(proteins_per_key)).astype(np.uint32)
    return pk, prk


def at_size_features(n_batches=20, batch=50_000, n_peptides=2_000_000, seed=0x5A6E, precursor_tol=(0, -20.0, 20.0), report_psms=1, device=0):
    """~n_batches x batch PSMs: spectra of the cfg2-sized synthetic table scored on the device in batches against an index without ~30 %
    of its targets. Returns (features FEATURE_DTYPE with peptide_idx in the full table, full Peptides)."""
    from sage_b200 import IndexedDatabase, Scorer, Tolerance, synth
    full = synth.make_peptides(n_peptides, seed=seed)
    rows = searched_subset(full.decoy, seed + 1)
    gdb = IndexedDatabase.build_from_peptides(subset_peptides(full, rows), device=device)
    sc = Scorer(gdb, precursor_tol=Tolerance(*precursor_tol), fragment_tol=Tolerance.ppm(-20, 20), report_psms=report_psms)
    out = []
    for b in range(n_batches):
        sp = synth.make_spectra(full, batch, seed=seed + 100 + b)
        f, c = sc.score_batch(sp)
        out.append(remap(valid_features(f, c, report_psms), rows))
    return np.concatenate(out), full
