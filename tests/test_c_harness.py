"""The drop-in boundary exercised by something other than Python: tests/c_harness/harness.c (gcc, links libsage_b200.so through
include/sage_b200.h) takes array-of-structs peptides / spectra, flattens them into malloc'd SoA arrays as the Rust shim of INTEGRATION.md
does, keeps ONE scorer handle across batches, and writes the Feature rows back; this test compares them with the oracle."""
import ctypes as C
import os
import struct
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def build_harness(out_dir):
    from sage_b200.build import build_library, library_path
    build_library()
    libdir = os.path.dirname(library_path())
    exe = os.path.join(out_dir, "sage_b200_c_harness")
    subprocess.check_call(["/usr/bin/gcc", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "c_harness", "harness.c"),
                           "-L", libdir, "-lsage_b200", f"-Wl,-rpath,{libdir}", "-o", exe])
    return exe


def test_harness_compiles_and_links_against_the_header(tmp_path):
    """CPU: the C program builds against include/sage_b200.h and resolves every symbol it uses from libsage_b200.so (no GPU call)."""
    exe = build_harness(tmp_path)
    out = subprocess.run(["ldd", exe], capture_output=True, text=True).stdout
    assert "libsage_b200.so" in out and "not found" not in out.split("libsage_b200.so")[1].splitlines()[0]


def write_input(path, pep, params, batches):
    with open(path, "wb") as f:
        n = len(pep)
        f.write(struct.pack("<Q", n))
        off = pep.seq_off.astype(np.int64)
        for i in range(n):
            a, b = off[i], off[i + 1]
            f.write(struct.pack("<IBBff", b - a, int(pep.decoy[i]), int(pep.missed[i]), float(pep.mono[i]), float(pep.nterm[i])))
            f.write(pep.seq[a:b].tobytes())
            f.write(pep.mods[a:b].astype("<f4").tobytes())
        f.write(bytes(params))
        f.write(struct.pack("<Q", len(batches)))
        for sp in batches:
            f.write(struct.pack("<Q", len(sp)))
            po = sp.peak_off.astype(np.int64)
            for i in range(len(sp)):
                a, b = po[i], po[i + 1]
                f.write(struct.pack("<IfBBfffff", b - a, float(sp.prec_mz[i]), int(sp.prec_charge[i]), int(sp.level[i]), float(sp.iso_lo[i]), float(sp.iso_hi[i]),
                                    float(sp.tic[i]), float(sp.rt[i]), float(sp.ims[i])))
                f.write(sp.masses[a:b].astype("<f4").tobytes())
                f.write(sp.intensities[a:b].astype("<f4").tobytes())


def read_output(path, report_psms):
    from sage_b200 import api
    res = []
    with open(path, "rb") as f:
        while True:
            h = f.read(4)
            if len(h) < 4:
                break
            rc = struct.unpack("<i", h)[0]
            if rc != 0:
                ln = struct.unpack("<I", f.read(4))[0]
                res.append((rc, f.read(ln).decode(errors="replace")))
                continue
            n = struct.unpack("<Q", f.read(8))[0]
            counts = np.frombuffer(f.read(4 * n), np.uint32)
            feats = np.frombuffer(f.read(128 * n * report_psms), api.FEATURE_DTYPE)
            nfr = struct.unpack("<Q", f.read(8))[0]
            frags = np.frombuffer(f.read(24 * nfr), api.FRAGMENT_DTYPE)
            res.append((0, counts, feats, frags))
    return res


@pytest.mark.gpu
def test_c_harness_results_equal_the_oracle(tmp_path):
    from helpers import assert_features_equal, oracle_cfg, oracle_db_from_peptides
    from sage_b200 import Scorer, SpectraBatch, Tolerance, api, synth
    exe = build_harness(tmp_path)
    pep = synth.make_peptides(5000, seed=31, static_c=True)
    spectra = synth.make_spectra(pep, 900, seed=32)
    kw = dict(precursor_tol=Tolerance.ppm(-20, 20), fragment_tol=Tolerance.ppm(-10, 10), report_psms=2, min_isotope_err=-1, max_isotope_err=2, annotate_matches=True)
    p = api.CScorerParams()
    p.precursor_tol, p.fragment_tol = kw["precursor_tol"]._c(), kw["fragment_tol"]._c()
    p.min_matched_peaks, p.min_isotope_err, p.max_isotope_err = 4, -1, 2
    p.min_precursor_charge, p.max_precursor_charge, p.override_precursor_charge, p.max_fragment_charge = 2, 4, 0, -1
    p.chimera, p.wide_window, p.annotate_matches, p.score_type, p.report_psms = 0, 0, 1, 0, 2
    bad = SpectraBatch(**{**spectra.slice(0, 5).__dict__, "level": np.array([2, 2, 1, 2, 2], np.uint8)})     # third batch: a non-MS2 scan -> error code
    batches = [spectra.slice(0, 500), spectra.slice(500, 900), bad, spectra.slice(100, 130)]
    write_input(tmp_path / "in.bin", pep, p, batches)
    subprocess.check_call([exe, str(tmp_path / "in.bin"), str(tmp_path / "out.bin")])
    res = read_output(tmp_path / "out.bin", 2)
    assert len(res) == 4
    odb = oracle_db_from_peptides(pep)
    total = 0
    for bi in (0, 1, 3):
        rc, counts, feats, frags = res[bi]
        assert rc == 0
        of, oc, ofr, _ = odb.score_batch(oracle_cfg(**kw), batches[bi].as_dict())
        total += assert_features_equal(feats, counts, of, oc, 2, what=f"C harness batch {bi}")
        # Fragments re-attached per PSM (scoring.rs:738-751): same rows as the oracle's, in the reported order
        sel = (np.arange(len(feats)) % 2) < np.repeat(counts, 2)
        g, o = feats[sel], of[sel]
        assert len(frags) == len(ofr) == int(g["fragment_count"].sum())
        for a, b_ in zip(g, o):
            x = frags[a["fragment_offset"]:a["fragment_offset"] + a["fragment_count"]]
            y = ofr[b_["frag_offset"]:b_["frag_offset"] + b_["frag_count"]]
            assert a["fragment_count"] == b_["frag_count"] == a["matched_peaks"]
            for k in ("kind", "charge", "ordinal"):
                assert np.array_equal(x[k], y[k]), k
            for k in ("intensity", "mz_calculated", "mz_experimental"):
                assert np.array_equal(x[k].view(np.uint32), y[k].view(np.uint32)), k
    assert total > 700
    assert res[2][0] == -3   # SAGE_B200_ENOTMS2
    assert "non-MS2" in res[2][1]
