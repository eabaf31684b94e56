"""Python mirror of the reference interface for the hot path, bound to libsage_b200.so through the C ABI
(include/sage_b200.h) with ctypes. Names and argument meaning follow sage-core:

    Tolerance          crates/sage/src/mass.rs:10-16
    Precursor / ProcessedSpectrum   crates/sage/src/spectrum.rs:47-79
    IndexedDatabase    crates/sage/src/database.rs:384-395   (device-resident here)
    Scorer             crates/sage/src/scoring.rs:210-232    (.score(spectrum) -> [Feature], plus .score_batch)

There is no CPU fallback: loading fails if the CUDA library is missing and every call fails if no GPU is present.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field

import numpy as np

from .build import build_library, library_path

PPM, PCT, DA = 0, 1, 2
KIND = {"a": 0, "b": 1, "c": 2, "x": 3, "y": 4, "z": 5}


class SageB200Error(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"sage_b200 error {code}: {message}")
        self.code = code
        self.message = message


# ------------------------------------------------------------------------------------------------ C structs
class CTol(C.Structure):
    _fields_ = [("kind", C.c_int32), ("lo", C.c_float), ("hi", C.c_float)]


class CPeptides(C.Structure):
    _fields_ = [("n_peptides", C.c_uint64), ("residue_offsets", C.c_void_p), ("sequence", C.c_void_p), ("modifications", C.c_void_p),
                ("nterm", C.c_void_p), ("monoisotopic", C.c_void_p), ("decoy", C.c_void_p), ("missed_cleavages", C.c_void_p)]


class CIndex(C.Structure):
    _fields_ = [("n_fragments", C.c_uint64), ("fragment_peptide", C.c_void_p), ("fragment_mz", C.c_void_p), ("n_buckets", C.c_uint64),
                ("bucket_min", C.c_void_p), ("bucket_size", C.c_uint64), ("ion_kinds", C.c_void_p), ("n_ion_kinds", C.c_uint64)]


class CDbInfo(C.Structure):
    _fields_ = [("n_peptides", C.c_uint64), ("n_fragments", C.c_uint64), ("n_buckets", C.c_uint64), ("bucket_size", C.c_uint64),
                ("n_ion_kinds", C.c_uint64), ("total_residues", C.c_uint64), ("device_bytes", C.c_uint64), ("device", C.c_int32)]


class CScorerParams(C.Structure):
    _fields_ = [("precursor_tol", CTol), ("fragment_tol", CTol), ("min_matched_peaks", C.c_uint16), ("min_isotope_err", C.c_int8),
                ("max_isotope_err", C.c_int8), ("min_precursor_charge", C.c_uint8), ("max_precursor_charge", C.c_uint8),
                ("override_precursor_charge", C.c_uint8), ("max_fragment_charge", C.c_int8), ("chimera", C.c_uint8), ("wide_window", C.c_uint8),
                ("annotate_matches", C.c_uint8), ("score_type", C.c_uint8), ("report_psms", C.c_uint32)]


class CSpectra(C.Structure):
    _fields_ = [("n", C.c_uint64), ("peak_offsets", C.c_void_p), ("masses", C.c_void_p), ("intensities", C.c_void_p), ("precursor_mz", C.c_void_p),
                ("precursor_charge", C.c_void_p), ("isolation_lo", C.c_void_p), ("isolation_hi", C.c_void_p), ("total_ion_current", C.c_void_p),
                ("level", C.c_void_p), ("scan_start_time", C.c_void_p), ("inverse_ion_mobility", C.c_void_p)]


COUNTER_U64 = ["spectra", "peaks", "queries", "tasks", "pages", "entries_scanned", "matched_fragments", "candidates_scored", "peptide_record_floats",
               "psms", "wide_queries", "pep_queries", "pep_fallbacks", "wide_overflows", "algorithmic_bytes", "prelim_bytes", "score_bytes", "h2d_bytes", "d2h_bytes", "kernel_launches", "chunk_retries"]
COUNTER_F32 = ["ms_total", "ms_h2d", "ms_setup", "ms_prelim", "ms_score", "ms_d2h", "ms_prelim_count", "ms_wall"]


class CCounters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in COUNTER_U64] + [(n, C.c_float) for n in COUNTER_F32]


# layout == sage_b200_feature (include/sage_b200.h)
FEATURE_DTYPE = np.dtype([
    ("spectrum", "<u4"), ("peptide_idx", "<u4"), ("peptide_len", "<u4"), ("rank", "<u4"), ("label", "<i4"), ("expmass", "<f4"), ("calcmass", "<f4"),
    ("charge", "<u4"), ("rt", "<f4"), ("ims", "<f4"), ("delta_mass", "<f4"), ("isotope_error", "<f4"), ("average_ppm", "<f4"), ("_pad0", "<u4"),
    ("hyperscore", "<f8"), ("delta_next", "<f8"), ("delta_best", "<f8"), ("matched_peaks", "<u4"), ("longest_b", "<u4"), ("longest_y", "<u4"),
    ("longest_y_pct", "<f4"), ("missed_cleavages", "<u4"), ("matched_intensity_pct", "<f4"), ("scored_candidates", "<u4"), ("ms2_intensity", "<f4"),
    ("poisson", "<f8"), ("fragment_offset", "<u4"), ("fragment_count", "<u4"),
])
assert FEATURE_DTYPE.itemsize == 128
FRAGMENT_DTYPE = np.dtype([("kind", "<i4"), ("charge", "<i4"), ("ordinal", "<i4"), ("intensity", "<f4"), ("mz_calculated", "<f4"),
                           ("mz_experimental", "<f4")])

EXPORTED_SYMBOLS = [
    "sage_b200_device_count", "sage_b200_db_create", "sage_b200_db_build", "sage_b200_db_get_info", "sage_b200_db_export_index", "sage_b200_db_destroy",
    "sage_b200_scorer_create", "sage_b200_scorer_destroy", "sage_b200_scorer_set_option", "sage_b200_score_batch", "sage_b200_batch_upload", "sage_b200_batch_run",
    "sage_b200_batch_download", "sage_b200_score_batch_multi", "sage_b200_quick_score", "sage_b200_initial_hits", "sage_b200_counters_get",
    "sage_b200_process_spectra", "sage_b200_find_reporter_ions", "sage_b200_host_alloc", "sage_b200_host_free", "sage_b200_last_error",
    "sage_b200_host_log_variant", "sage_b200_host_log1pf_exact", "sage_b200_device_log", "sage_b200_bind_thread_to_device", "sage_b200_host_alloc_blocks",
    "sage_b200_assign_fdr", "sage_b200_lda_fit",
]

_lib = None


def load_library(build: bool = True):
    """Loads the in-tree CUDA library. Raises (never falls back) if it cannot be built/loaded."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        if not build:
            raise FileNotFoundError(f"{path} not built; run `python -m sage_b200.build`")
        build_library()
    lib = C.CDLL(path)
    for s in EXPORTED_SYMBOLS:
        getattr(lib, s)
    lib.sage_b200_host_alloc.restype = C.c_void_p
    lib.sage_b200_host_alloc.argtypes = [C.c_size_t]
    lib.sage_b200_host_free.argtypes = [C.c_void_p]
    lib.sage_b200_host_alloc_blocks.restype = C.c_void_p
    lib.sage_b200_host_alloc_blocks.argtypes = [C.c_size_t, C.c_void_p, C.c_int]
    lib.sage_b200_last_error.restype = C.c_size_t
    lib.sage_b200_initial_hits.restype = C.c_int64
    lib.sage_b200_db_destroy.argtypes = [C.c_void_p]
    lib.sage_b200_scorer_destroy.argtypes = [C.c_void_p]
    _lib = lib
    return lib


def _last_error() -> str:
    buf = C.create_string_buffer(2048)
    load_library().sage_b200_last_error(buf, C.c_size_t(2048))
    return buf.value.decode(errors="replace")


def _check(rc: int):
    if rc != 0:
        raise SageB200Error(int(rc), _last_error())


def device_count() -> int:
    return int(load_library().sage_b200_device_count())


def bind_thread_to_device(device: int) -> int:
    """Pins the calling thread to the CPUs of the GPU's NUMA node (-1: topology unknown, nothing changed)."""
    return int(load_library().sage_b200_bind_thread_to_device(C.c_int(device)))


def host_log_variant() -> int:
    """Which build of glibc's log() the host libm is (0 FMA-contracted, 1 plain, -1 unknown); the kernels reproduce that one (glibc_log.cuh)."""
    return int(load_library().sage_b200_host_log_variant())


def host_log1pf_exact() -> bool:
    """True when the host libm's log1pf is the function the kernels reproduce for the OpenMS score type."""
    return bool(load_library().sage_b200_host_log1pf_exact())


def device_log(x: np.ndarray, variant: int, device: int = 0) -> np.ndarray:
    """The device's evaluation of f64 log for every x (test hook for the glibc log() emulation)."""
    x = np.ascontiguousarray(x, np.float64)
    out = np.zeros_like(x)
    _check(load_library().sage_b200_device_log(C.c_int(device), C.c_int(variant), _ptr(x), C.c_uint64(len(x)), _ptr(out)))
    return out


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def pinned_empty(shape, dtype) -> np.ndarray:
    """numpy array backed by page-locked memory from sage_b200_host_alloc (release with pinned_free)."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    p = load_library().sage_b200_host_alloc(C.c_size_t(max(n, 16)))
    if not p:
        raise SageB200Error(-2, _last_error())
    buf = (C.c_ubyte * max(n, 16)).from_address(p)
    arr = np.frombuffer(buf, dtype=np.uint8, count=n).view(dtype).reshape(shape)
    _PINNED[arr.ctypes.data] = p
    return arr


def pinned_empty_blocks(shape, dtype, devices) -> np.ndarray:
    """Page-locked array whose i-th of len(devices) equal parts sits on the NUMA node next to devices[i] (sage_b200_host_alloc_blocks): the
    input / output buffers of a score_batch_multi call."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    dev = (C.c_int * len(devices))(*[int(d) for d in devices])
    p = load_library().sage_b200_host_alloc_blocks(C.c_size_t(max(n, 16)), dev, C.c_int(len(devices)))
    if not p:
        raise SageB200Error(-2, _last_error())
    buf = (C.c_ubyte * max(n, 16)).from_address(p)
    arr = np.frombuffer(buf, dtype=np.uint8, count=n).view(dtype).reshape(shape)
    _PINNED[arr.ctypes.data] = p
    return arr


_PINNED: dict = {}


def pinned_free(arr: np.ndarray):
    p = _PINNED.pop(arr.ctypes.data, None)
    if p is not None:
        load_library().sage_b200_host_free(C.c_void_p(p))


# ------------------------------------------------------------------------------------------------ reference-shaped types
@dataclass(frozen=True)
class Tolerance:
    """mass.rs:10-16. Tolerance.ppm(-10, 10) / .da(-500, 100) / .pct(..)."""
    kind: int
    lo: float
    hi: float

    @staticmethod
    def ppm(lo, hi):
        return Tolerance(PPM, float(lo), float(hi))

    @staticmethod
    def da(lo, hi):
        return Tolerance(DA, float(lo), float(hi))

    @staticmethod
    def pct(lo, hi):
        return Tolerance(PCT, float(lo), float(hi))

    def as_tuple(self):
        return (self.kind, self.lo, self.hi)

    def _c(self):
        return CTol(self.kind, self.lo, self.hi)


@dataclass
class Precursor:
    """spectrum.rs:47-55"""
    mz: float = 0.0
    charge: int | None = None
    isolation_window: Tolerance | None = None
    inverse_ion_mobility: float | None = None


@dataclass
class ProcessedSpectrum:
    """spectrum.rs:58-79"""
    level: int = 2
    id: str = ""
    file_id: int = 0
    scan_start_time: float = 0.0
    precursors: list = field(default_factory=list)
    masses: np.ndarray = field(default_factory=lambda: np.zeros(0, np.float32))
    intensities: np.ndarray = field(default_factory=lambda: np.zeros(0, np.float32))
    total_ion_current: float = 0.0


@dataclass
class SpectraBatch:
    """&[ProcessedSpectrum] flattened to the SoA the C ABI takes (sage_b200_spectra)."""
    peak_off: np.ndarray
    masses: np.ndarray
    intensities: np.ndarray
    prec_mz: np.ndarray
    prec_charge: np.ndarray
    iso_lo: np.ndarray
    iso_hi: np.ndarray
    tic: np.ndarray
    level: np.ndarray | None = None
    rt: np.ndarray | None = None
    ims: np.ndarray | None = None

    def __len__(self):
        return len(self.prec_mz)

    @staticmethod
    def from_spectra(spectra) -> "SpectraBatch":
        n = len(spectra)
        off = np.zeros(n + 1, np.uint64)
        for i, s in enumerate(spectra):
            off[i + 1] = off[i] + len(s.masses)
        masses = np.concatenate([np.asarray(s.masses, np.float32) for s in spectra]) if n else np.zeros(0, np.float32)
        intens = np.concatenate([np.asarray(s.intensities, np.float32) for s in spectra]) if n else np.zeros(0, np.float32)
        pmz, chg = np.full(n, np.nan, np.float32), np.zeros(n, np.uint8)
        ilo, ihi, ims = np.full(n, np.nan, np.float32), np.full(n, np.nan, np.float32), np.full(n, np.nan, np.float32)
        for i, s in enumerate(spectra):
            if s.precursors:
                p = s.precursors[0]
                pmz[i] = p.mz
                chg[i] = p.charge or 0
                if p.isolation_window is not None:
                    assert p.isolation_window.kind == DA
                    ilo[i], ihi[i] = p.isolation_window.lo, p.isolation_window.hi
                if p.inverse_ion_mobility is not None:
                    ims[i] = p.inverse_ion_mobility
        return SpectraBatch(off, masses, intens, pmz, chg, ilo, ihi, np.array([s.total_ion_current for s in spectra], np.float32),
                            np.array([s.level for s in spectra], np.uint8), np.array([s.scan_start_time for s in spectra], np.float32), ims)

    def as_dict(self) -> dict:
        return dict(peak_off=self.peak_off, masses=self.masses, intensities=self.intensities, prec_mz=self.prec_mz, prec_charge=self.prec_charge,
                    iso_lo=self.iso_lo, iso_hi=self.iso_hi, tic=self.tic, level=self.level, ims=self.ims)

    def slice(self, a: int, b: int) -> "SpectraBatch":
        p0, p1 = int(self.peak_off[a]), int(self.peak_off[b])
        opt = lambda x: None if x is None else x[a:b]  # noqa: E731
        return SpectraBatch(self.peak_off[a:b + 1] - self.peak_off[a], self.masses[p0:p1], self.intensities[p0:p1], self.prec_mz[a:b],
                            self.prec_charge[a:b], self.iso_lo[a:b], self.iso_hi[a:b], self.tic[a:b], opt(self.level), opt(self.rt), opt(self.ims))

    def _c(self, keep: list) -> CSpectra:
        def arr(x, dt):
            if x is None:
                return None
            a = np.ascontiguousarray(x, dtype=dt)
            keep.append(a)
            return _ptr(a)
        cs = CSpectra()
        cs.n = len(self)
        cs.peak_offsets = arr(self.peak_off, np.uint64)
        cs.masses = arr(self.masses, np.float32)
        cs.intensities = arr(self.intensities, np.float32)
        cs.precursor_mz = arr(self.prec_mz, np.float32)
        cs.precursor_charge = arr(self.prec_charge, np.uint8)
        cs.isolation_lo = arr(self.iso_lo, np.float32)
        cs.isolation_hi = arr(self.iso_hi, np.float32)
        cs.total_ion_current = arr(self.tic, np.float32)
        cs.level = arr(self.level, np.uint8)
        cs.scan_start_time = arr(self.rt, np.float32)
        cs.inverse_ion_mobility = arr(self.ims, np.float32)
        return cs


@dataclass
class Peptides:
    """The Peptide fields the hot path reads (peptide.rs:13-31), flattened. Row index == PeptideIx."""
    seq_off: np.ndarray
    seq: np.ndarray
    mods: np.ndarray
    nterm: np.ndarray
    mono: np.ndarray
    decoy: np.ndarray
    missed: np.ndarray

    def __len__(self):
        return len(self.mono)

    def sequence(self, i: int) -> str:
        return bytes(self.seq[self.seq_off[i]:self.seq_off[i + 1]]).decode()

    def _c(self, keep: list) -> CPeptides:
        def arr(x, dt):
            a = np.ascontiguousarray(x, dtype=dt)
            keep.append(a)
            return _ptr(a)
        cp = CPeptides()
        cp.n_peptides = len(self.mono)
        cp.residue_offsets = arr(self.seq_off, np.uint32)
        cp.sequence = arr(self.seq, np.uint8)
        cp.modifications = arr(self.mods, np.float32)
        cp.nterm = arr(self.nterm, np.float32)
        cp.monoisotopic = arr(self.mono, np.float32)
        cp.decoy = arr(self.decoy, np.uint8)
        cp.missed_cleavages = arr(self.missed, np.uint8)
        return cp


def _kinds(ion_kinds):
    return np.array([KIND[k] if isinstance(k, str) else int(k) for k in ion_kinds], dtype=np.uint8)


class IndexedDatabase:
    """Device-resident IndexedDatabase (database.rs:384-395)."""

    def __init__(self, handle, peptides: Peptides):
        self._h = C.c_void_p(handle)
        self.peptides = peptides
        info = CDbInfo()
        _check(load_library().sage_b200_db_get_info(self._h, C.byref(info)))
        self.info = {k: getattr(info, k) for k, _ in CDbInfo._fields_}

    def device_bytes(self) -> int:
        """HBM held by the index right now, including the block-major copies scorers have built on first use."""
        info = CDbInfo()
        _check(load_library().sage_b200_db_get_info(self._h, C.byref(info)))
        return int(info.device_bytes)

    def __del__(self):
        try:
            if self._h:
                load_library().sage_b200_db_destroy(self._h)
                self._h = None
        except Exception:
            pass

    @staticmethod
    def from_reference_layout(peptides: Peptides, frag_pep, frag_mz, bucket_min, bucket_size, ion_kinds=("b", "y"), device=0) -> "IndexedDatabase":
        """Upload an index already built by the reference's Parameters::build (database.rs:260)."""
        keep: list = []
        cp = peptides._c(keep)
        ci = CIndex()
        fp = np.ascontiguousarray(frag_pep, np.uint32)
        fm = np.ascontiguousarray(frag_mz, np.float32)
        bm = np.ascontiguousarray(bucket_min, np.float32)
        kinds = _kinds(ion_kinds)
        ci.n_fragments, ci.fragment_peptide, ci.fragment_mz = len(fp), _ptr(fp), _ptr(fm)
        ci.n_buckets, ci.bucket_min, ci.bucket_size = len(bm), _ptr(bm), int(bucket_size)
        ci.ion_kinds, ci.n_ion_kinds = _ptr(kinds), len(kinds)
        h = C.c_void_p()
        _check(load_library().sage_b200_db_create(C.byref(cp), C.byref(ci), C.c_int(device), C.byref(h)))
        return IndexedDatabase(h.value, peptides)

    @staticmethod
    def build_from_peptides(peptides: Peptides, bucket_size=8192, ion_kinds=("b", "y"), min_ion_index=2, device=0) -> "IndexedDatabase":
        """Parameters::build_from_peptides (database.rs:265-365) executed on the device."""
        keep: list = []
        cp = peptides._c(keep)
        kinds = _kinds(ion_kinds)
        h = C.c_void_p()
        _check(load_library().sage_b200_db_build(C.byref(cp), C.c_uint64(int(bucket_size)), _ptr(kinds), C.c_uint64(len(kinds)),
                                                 C.c_uint64(int(min_ion_index)), C.c_int(device), C.byref(h)))
        return IndexedDatabase(h.value, peptides)

    def export_index(self):
        nf, nb = self.info["n_fragments"], self.info["n_buckets"]
        fp, fm, bm = np.empty(nf, np.uint32), np.empty(nf, np.float32), np.empty(nb, np.float32)
        _check(load_library().sage_b200_db_export_index(self._h, _ptr(fp), _ptr(fm), _ptr(bm)))
        return fp, fm, bm


class Scorer:
    """Scorer (scoring.rs:210-232): same public fields; `db` is a device-resident IndexedDatabase."""

    def __init__(self, db: IndexedDatabase, precursor_tol: Tolerance, fragment_tol: Tolerance, min_matched_peaks=4, min_isotope_err=0,
                 max_isotope_err=0, min_precursor_charge=2, max_precursor_charge=4, override_precursor_charge=False, max_fragment_charge=None,
                 chimera=False, report_psms=1, wide_window=False, annotate_matches=False, score_type=0):
        self.db = db
        self.report_psms = int(report_psms)
        self.fragment_capacity = None   # annotate_matches: size of the fragments array (default: generous estimate)
        self.last_fragments = None      # Fragments rows of the last score_batch (Feature.fragment_offset/count index into it)
        p = CScorerParams()
        p.precursor_tol, p.fragment_tol = precursor_tol._c(), fragment_tol._c()
        p.min_matched_peaks = min_matched_peaks
        p.min_isotope_err, p.max_isotope_err = min_isotope_err, max_isotope_err
        p.min_precursor_charge, p.max_precursor_charge = min_precursor_charge, max_precursor_charge
        p.override_precursor_charge = int(override_precursor_charge)
        p.max_fragment_charge = -1 if max_fragment_charge is None else int(max_fragment_charge)
        p.chimera, p.wide_window, p.annotate_matches = int(chimera), int(wide_window), int(annotate_matches)
        p.score_type = int(score_type)
        p.report_psms = self.report_psms
        self._params = p
        h = C.c_void_p()
        _check(load_library().sage_b200_scorer_create(db._h, C.byref(p), C.byref(h)))
        self._h = h

    def set_option(self, name: str, value: int):
        _check(load_library().sage_b200_scorer_set_option(self._h, name.encode(), C.c_int64(int(value))))

    def __del__(self):
        try:
            if self._h:
                load_library().sage_b200_scorer_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def score_batch(self, batch: SpectraBatch, out: np.ndarray | None = None, counts: np.ndarray | None = None):
        """`spectra.par_iter().flat_map(|s| scorer.score(s))` (runner.rs:311-325). Returns (features[n*report_psms], counts[n])."""
        n = len(batch)
        if out is None:
            out = np.zeros(n * self.report_psms, FEATURE_DTYPE)
        if counts is None:
            counts = np.zeros(n, np.uint32)
        keep: list = []
        cs = batch._c(keep)
        used = C.c_uint64(0)
        if self._params.annotate_matches:
            cap = int(self.fragment_capacity or (n * self.report_psms * 128 + 1024))
            frags = np.zeros(cap, FRAGMENT_DTYPE)
            _check(load_library().sage_b200_score_batch(self._h, C.byref(cs), _ptr(out), _ptr(counts), _ptr(frags), C.c_uint64(cap), C.byref(used)))
            self.last_fragments = frags[:used.value]
            return out, counts
        _check(load_library().sage_b200_score_batch(self._h, C.byref(cs), _ptr(out), _ptr(counts), None, C.c_uint64(0), C.byref(used)))
        return out, counts

    # device-resident phases of score_batch (one chunk): upload once, run many times, download
    def upload(self, batch: SpectraBatch):
        keep: list = []
        cs = batch._c(keep)
        self._resident_n = len(batch)
        _check(load_library().sage_b200_batch_upload(self._h, C.byref(cs)))

    def run(self):
        _check(load_library().sage_b200_batch_run(self._h))

    def download(self, out: np.ndarray | None = None, counts: np.ndarray | None = None):
        n = self._resident_n
        if out is None:
            out = np.zeros(n * self.report_psms, FEATURE_DTYPE)
        if counts is None:
            counts = np.zeros(n, np.uint32)
        _check(load_library().sage_b200_batch_download(self._h, _ptr(out), _ptr(counts)))
        return out, counts

    def quick_score(self, batch: SpectraBatch, prefilter_low_memory: bool, keep: np.ndarray | None = None) -> np.ndarray:
        """Scorer::quick_score (scoring.rs:255-298) over a batch: keep[PeptideIx] (uint8) is OR-ed and returned."""
        if keep is None:
            keep = np.zeros(self.db.info["n_peptides"], np.uint8)
        keep_c = np.ascontiguousarray(keep, dtype=np.uint8)
        kl: list = []
        cs = batch._c(kl)
        _check(load_library().sage_b200_quick_score(self._h, C.byref(cs), C.c_int(int(prefilter_low_memory)), _ptr(keep_c)))
        return keep_c

    def score(self, spectrum: ProcessedSpectrum):
        """Scorer::score (scoring.rs:300): one spectrum -> list of Feature rows."""
        out, counts = self.score_batch(SpectraBatch.from_spectra([spectrum]))
        return out[:counts[0]]

    def initial_hits(self, batch: SpectraBatch):
        assert len(batch) == 1
        cap = 256
        m, p = np.zeros(cap, np.uint16), np.zeros(cap, np.uint32)
        c, i = np.zeros(cap, np.uint8), np.zeros(cap, np.int8)
        mp, scd = C.c_uint64(0), C.c_uint64(0)
        keep: list = []
        cs = batch._c(keep)
        n = load_library().sage_b200_initial_hits(self._h, C.byref(cs), _ptr(m), _ptr(p), _ptr(c), _ptr(i), C.c_uint64(cap), C.byref(mp), C.byref(scd))
        if n < 0:
            raise SageB200Error(int(n), _last_error())
        return dict(matched=m[:n].copy(), peptide=p[:n].copy(), charge=c[:n].copy(), iso=i[:n].copy(), matched_peaks=mp.value, scored_candidates=scd.value)

    def counters(self) -> dict:
        cc = CCounters()
        _check(load_library().sage_b200_counters_get(self._h, C.byref(cc)))
        return {k: getattr(cc, k) for k, _ in CCounters._fields_}


def score_batch_multi(scorers, batch: SpectraBatch, out: np.ndarray | None = None, counts: np.ndarray | None = None):
    """sage_b200_score_batch_multi: one process, one Scorer per GPU (same settings), spectra split into contiguous blocks."""
    n, r = len(batch), scorers[0].report_psms
    if out is None:
        out = np.zeros(n * r, FEATURE_DTYPE)
    if counts is None:
        counts = np.zeros(n, np.uint32)
    keep: list = []
    cs = batch._c(keep)
    arr = (C.c_void_p * len(scorers))(*[s._h for s in scorers])
    _check(load_library().sage_b200_score_batch_multi(arr, C.c_int(len(scorers)), C.byref(cs), _ptr(out), _ptr(counts)))
    return out, counts


class CProcessorParams(C.Structure):
    _fields_ = [("take_top_n", C.c_uint64), ("deisotope", C.c_uint8), ("min_deisotope_mz", C.c_float)]


class CRawSpectra(C.Structure):
    _fields_ = [("n", C.c_uint64), ("peak_offsets", C.c_void_p), ("mz", C.c_void_p), ("intensity", C.c_void_p), ("precursor_charge", C.c_void_p),
                ("level", C.c_void_p)]


class SpectrumProcessor:
    """SpectrumProcessor::new(take_top_n, deisotope, min_deisotope_mz) (spectrum.rs:271); process() runs on the device."""

    def __init__(self, take_top_n: int, deisotope: bool, min_deisotope_mz: float, device: int = 0):
        self.take_top_n, self.deisotope, self.min_deisotope_mz, self.device = int(take_top_n), bool(deisotope), float(min_deisotope_mz), device

    def process_batch(self, peak_off, mz, intensity, precursor_charge):
        """Raw centroided MS2 spectra (CSR) -> (peak_off[n+1], masses, intensities, tic[n]) of the ProcessedSpectrum batch."""
        peak_off = np.ascontiguousarray(peak_off, np.uint64)
        mz, intensity = np.ascontiguousarray(mz, np.float32), np.ascontiguousarray(intensity, np.float32)
        chg = np.ascontiguousarray(precursor_charge, np.uint8)
        n = len(chg)
        pp = CProcessorParams(self.take_top_n, int(self.deisotope), self.min_deisotope_mz)
        raw = CRawSpectra(n, _ptr(peak_off), _ptr(mz), _ptr(intensity), _ptr(chg), None)
        out_off = np.zeros(n + 1, np.uint64)
        om, oi, tic = np.zeros(max(1, len(mz)), np.float32), np.zeros(max(1, len(mz)), np.float32), np.zeros(n, np.float32)
        _check(load_library().sage_b200_process_spectra(C.c_int(self.device), C.byref(pp), C.byref(raw), _ptr(out_off), _ptr(om), _ptr(oi), _ptr(tic)))
        k = int(out_off[-1])
        return out_off, om[:k].copy(), oi[:k].copy(), tic


TMT6PLEX = np.float32([126.127726, 127.124761, 128.134436, 129.131471, 130.141145, 131.138180])   # tmt.rs:213-215


def find_reporter_ions(peak_off, masses, intensities, labels, label_tolerance: Tolerance, device: int = 0) -> np.ndarray:
    """tmt::find_reporter_ions (tmt.rs:193-211) over a batch of ProcessedSpectrum -> float32 [n, n_labels]."""
    peak_off = np.ascontiguousarray(peak_off, np.uint64)
    masses, intensities, labels = (np.ascontiguousarray(x, np.float32) for x in (masses, intensities, labels))
    n = len(peak_off) - 1
    out = np.zeros((n, len(labels)), np.float32)
    _check(load_library().sage_b200_find_reporter_ions(C.c_int(device), C.c_uint64(n), _ptr(peak_off), _ptr(masses), _ptr(intensities), _ptr(labels),
                                                       C.c_uint64(len(labels)), label_tolerance._c(), _ptr(out)))
    return out


# ------------------------------------------------------------------------------------------------ rescoring + FDR
class CFdrParams(C.Structure):
    _fields_ = [("precursor_tol", CTol), ("n_peptides", C.c_uint64), ("peptide_key", C.c_void_p), ("n_peptide_keys", C.c_uint64),
                ("protein_key", C.c_void_p), ("n_protein_keys", C.c_uint64), ("aligned_rt", C.c_void_p), ("delta_rt_model", C.c_void_p),
                ("delta_ims_model", C.c_void_p)]


FDR_SUMMARY_F32 = ["ms_h2d", "ms_lda", "ms_pep", "ms_spectrum_q", "ms_picked", "ms_d2h", "ms_wall"]


class CFdrSummary(C.Structure):
    _fields_ = [("spectrum_passing", C.c_uint64), ("peptide_passing", C.c_uint64), ("protein_passing", C.c_uint64), ("coef", C.c_double * 20),
                ("lda_fitted", C.c_uint32)] + [(n, C.c_float) for n in FDR_SUMMARY_F32]


# layout == sage_b200_fdr_row (include/sage_b200.h)
FDR_DTYPE = np.dtype([("discriminant_score", "<f4"), ("posterior_error", "<f4"), ("spectrum_q", "<f4"), ("peptide_q", "<f4"), ("protein_q", "<f4")])


def assign_fdr(features: np.ndarray, precursor_tol: Tolerance, peptide_key=None, protein_key=None, aligned_rt=None, delta_rt_model=None,
               delta_ims_model=None, device: int = 0, *, n_peptides: int | None = None, n_peptide_keys: int | None = None, n_protein_keys: int | None = None):
    """spectrum_fdr + picked_peptide + picked_protein (runner.rs:533-537) over Feature rows (FEATURE_DTYPE, any order).

    peptide_key / protein_key: uint32 per PeptideIx (see include/sage_b200.h); None skips that stage. The key counts default to max + 1 and
    n_peptides to the key table length. aligned_rt / delta_rt_model / delta_ims_model: optional float32 per feature (LDA features 16, 18, 19).
    Returns (rows FDR_DTYPE[n] in input order, order uint32[n] = input index at each rank, summary dict)."""
    f = np.ascontiguousarray(features)
    if f.dtype != FEATURE_DTYPE:
        raise TypeError("features must be FEATURE_DTYPE")
    n = len(f)
    keep: list = []

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
        p.peptide_key = _ptr(pk)
        p.n_peptide_keys = int(n_peptide_keys if n_peptide_keys is not None else (int(pk.max()) + 1 if len(pk) else 0))
    if prk is not None:
        p.protein_key = _ptr(prk)
        valid = prk[prk != 0xFFFFFFFF]
        p.n_protein_keys = int(n_protein_keys if n_protein_keys is not None else (int(valid.max()) + 1 if len(valid) else 0))
    for name, x in (("aligned_rt", aligned_rt), ("delta_rt_model", delta_rt_model), ("delta_ims_model", delta_ims_model)):
        a = arr(x, np.float32)
        if a is not None and len(a) != n:
            raise ValueError(f"{name} must have one value per feature")
        setattr(p, name, _ptr(a))
    rows = np.zeros(n, FDR_DTYPE)
    order = np.zeros(n, np.uint32)
    s = CFdrSummary()
    _check(load_library().sage_b200_assign_fdr(C.c_int(device), _ptr(f), C.c_uint64(n), C.byref(p), _ptr(rows), _ptr(order), C.byref(s)))
    summary = {k: getattr(s, k) for k, _ in CFdrSummary._fields_ if k != "coef"}
    summary["coef"] = np.array(s.coef[:], np.float64)
    summary["lda_fitted"] = bool(s.lda_fitted)
    return rows, order, summary


def lda_fit(rows: np.ndarray, decoy: np.ndarray, device: int = 0):
    """LinearDiscriminantAnalysis::train (linear_discriminant.rs:63-124) on caller rows [n, d <= 20] through the device reductions:
    the coefficients, or None when the model cannot be fitted."""
    x = np.ascontiguousarray(rows, np.float64)
    n, d = x.shape
    dec = np.ascontiguousarray(decoy, np.uint8)
    coef = np.zeros(d, np.float64)
    rc = load_library().sage_b200_lda_fit(C.c_int(device), _ptr(x), C.c_uint64(n), C.c_uint32(d), _ptr(dec), _ptr(coef))
    if rc == 1:
        return None
    _check(rc)
    return coef


Feature = FEATURE_DTYPE
