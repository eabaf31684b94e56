#!/usr/bin/env python
"""bench.py — spectra/sec of the fragment-index search-and-score hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one process per GPU under torchrun for N>1)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm (oracle port, all host threads), rank 0 only
    python bench.py ... --dump-outputs DIR                   # also writes the PSM table of the last timed step as DIR/<field>.npy (dump_outputs)

A "step" is one pass of the hot path over one batch of synthetic spectra. The headline workload is `cfg2` = BASELINE.json configs[1]:
50k MS2 spectra x 200 peaks vs a ~2M-peptide tryptic index, +-20 ppm precursor / +-20 ppm fragment; per GPU the work is fixed (weak
scaling: every rank scores its own 50k spectra against a replicated index; no collective on the data path).

  value      spectra/s with the spectra already resident in HBM: K x (k_setup_queries -> k_prelim_* -> k_replay -> k_score [-> k_fold -> k_features -> k_rows]), timed with CUDA
             events on the launching stream (sage_b200_batch_run), max over ranks.
  e2e        spectra/s through the C-ABI call sage_b200_score_batch with pinned HOST buffers: H2D of the spectra and D2H of the Feature rows
             inside the timed region; `e2e.pageable` is the same call with ordinary (malloc'd) host arrays, as a Rust Vec<f32> would be.
             `ms_per_call_median_rank0` / `ms_in_library_median_rank0`: per-call wall clock at the Python caller / inside the C call.
  roofline   the kernel that takes longest in a step: its share of the SURVEY.md §8d algorithmic bytes / its CUDA-event duration vs the
             measured HBM peak (`frac`), and the same with the DRAM bytes ncu measured for that kernel (`dram_frac`, from profiles/traffic.json
             when that capture belongs to the sources being timed); `kernels` lists both for every kernel of the step. The algorithmic bytes
             are the reference algorithm's work terms, collected by ONE untimed step in the reference's loop order (option narrow_index = 0):
             the timed steps count narrow windows against a small-block copy of the index and never visit those pages.
  cpu_baseline  the CPU oracle (bit-faithful port of sage-core's path; OpenMP over spectra) on this box's host cores.
  extra      the other BASELINE.json configurations, each with its own value / e2e / parity check, so that they are driver-run numbers too:
             cfg4 (open search), cfg5 (chimeric, report_psms 5) and cfg3 (15 M-peptide index with two variable modifications); their spectra
             totals are fixed (50k / 100k / 200k) and sharded over the N GPUs, i.e. strong scaling across the driver's N = 1, 2, 4, 8 runs.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

VAR_MODS_CFG3 = (("M", 15.9949), ("STY", 79.9663))
WORKLOADS = {
    # n_spectra: per GPU when scaling == "weak", total over all GPUs when "strong"
    "cfg2": dict(desc="50k synthetic MS2 spectra (200 peaks) per GPU vs ~2M-peptide tryptic index, +-20 ppm precursor, +-20 ppm fragment", n_spectra=50_000,
                 scaling="weak", n_peptides=2_000_000, scorer=dict(precursor_tol=(0, -20.0, 20.0), fragment_tol=(0, -20.0, 20.0)), spectra={}, cpu_sample=50_000),
    "cfg3": dict(desc="200k spectra (sharded over the GPUs) vs tryptic index + 2 variable mods (M+15.9949, STY+79.9663, max 2 per peptide: ~16M peptides, "
                      "~680M fragments) + static C, +-20 ppm / +-20 ppm", n_spectra=200_000, scaling="strong", n_peptides=2_000_000,
                 peptides=dict(var_mods=VAR_MODS_CFG3, max_variable_mods=2, static_c=True),
                 scorer=dict(precursor_tol=(0, -20.0, 20.0), fragment_tol=(0, -20.0, 20.0)), spectra={}, cpu_sample=2_000),
    "cfg4": dict(desc="open search: 50k spectra (sharded over the GPUs), -500..+500 Da precursor window, ~2M-peptide tryptic index, +-20 ppm fragment",
                 n_spectra=50_000, scaling="strong", n_peptides=2_000_000, scorer=dict(precursor_tol=(2, -500.0, 500.0), fragment_tol=(0, -20.0, 20.0)),
                 spectra={}, cpu_sample=512),
    "cfg5": dict(desc="chimeric search (report_psms=5) on 100k co-fragmenting spectra (sharded over the GPUs), +-20 ppm / +-20 ppm", n_spectra=100_000,
                 scaling="strong", n_peptides=2_000_000, scorer=dict(precursor_tol=(0, -20.0, 20.0), fragment_tol=(0, -20.0, 20.0), chimera=True, report_psms=5),
                 spectra=dict(chimeric=True), cpu_sample=10_000),
    "small": dict(desc="smoke-size: 4k spectra vs 100k peptides, +-20 ppm / +-20 ppm", n_spectra=4_000, scaling="weak", n_peptides=100_000,
                  scorer=dict(precursor_tol=(0, -20.0, 20.0), fragment_tol=(0, -20.0, 20.0)), spectra={}, cpu_sample=4_000),
}
EXTRAS = {"cfg2": ["cfg4", "cfg5", "cfg3"]}   # extra workloads run after the headline one (each with its own steps, see EXTRA_STEPS)
EXTRA_STEPS = {"cfg4": (3, 3), "cfg5": (5, 3), "cfg3": (5, 3)}   # (steps, warmup)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def spectra_per_rank(wl, world):
    return wl["n_spectra"] if wl["scaling"] == "weak" else max(1, wl["n_spectra"] // max(1, world))


def load_or_make(name, wl, rank, world):
    """Synthetic peptide table (shared by all ranks; rank 0 generates and caches it in the temporary directory, the others wait for the file) and
    this rank's spectra. The cache belongs to this user and to the generator sources it was made by, so a table left by another user or by another
    version of the generator is never read back."""
    from sage_b200 import Peptides, synth
    pk = dict(wl.get("peptides", {}))
    h = hashlib.sha1(json.dumps([wl["n_peptides"], sorted((k, str(v)) for k, v in pk.items())]).encode())
    for f in ("synth.py", os.path.join("csrc", "synth_expand.cpp")):
        h.update(open(os.path.join(ROOT, "sage_b200", f), "rb").read())
    cache = os.path.join(tempfile.gettempdir(), f"sage_b200_pep_{os.getuid()}_{h.hexdigest()[:12]}.npz")
    t0 = time.time()
    pep = None
    if rank != 0 and world > 1:
        for _ in range(1800):   # wait for rank 0 (up to 15 min)
            if os.path.exists(cache):
                break
            time.sleep(0.5)
    if os.path.exists(cache):
        try:
            z = np.load(cache)
            pep = Peptides(**{k: z[k] for k in ("seq_off", "seq", "mods", "nterm", "mono", "decoy", "missed")})
        except Exception:
            pep = None
    if pep is None:
        pep = synth.make_peptides(wl["n_peptides"], **pk)
        if rank == 0:
            tmp = cache + f".{os.getpid()}.tmp.npz"
            try:
                np.savez(tmp, **pep.__dict__)
                os.replace(tmp, cache)
            except OSError as e:   # the cache only saves time: a full or read-only temporary directory does not stop the run
                log(f"[rank 0] peptide table not cached ({e})")
                if os.path.exists(tmp):
                    os.unlink(tmp)
    spectra = synth.make_spectra(pep, spectra_per_rank(wl, world), seed=0xB200 + 2 + 1000 * rank, **wl["spectra"])
    log(f"[rank {rank}] {name} data: {len(pep)} peptides, {len(spectra)} spectra in {time.time() - t0:.1f}s")
    return pep, spectra


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed regions (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu):
        self.gpu, self.rows, self.proc, self.path = gpu, [], None, None

    def __enter__(self):
        # ONE nvidia-smi process polling every 50 ms, started (and past its driver initialisation) before the timed regions begin: spawning
        # a fresh nvidia-smi per sample put its start-up (NVML init takes driver locks) inside the timed e2e calls.
        import tempfile
        fd, self.path = tempfile.mkstemp(prefix="sage_b200_clocks_", suffix=".csv")
        os.close(fd)
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
            t0 = time.time()
            while time.time() - t0 < 5.0 and os.path.getsize(self.path) == 0:
                time.sleep(0.02)
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc is not None:
            time.sleep(0.06)   # one more sample after the last timed call
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        try:
            for ln in open(self.path).read().strip().splitlines():
                self.rows.append([x.strip() for x in ln.split(",")])
            os.unlink(self.path)
        except Exception:
            pass

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(self.rows)}


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def kernel_sources_sha():
    """Hash of the DEVICE code the library is built from (DRAM traffic is a property of the kernels, not of the host runtime):
    profiles/traffic.json is only trusted when it was captured from these sources."""
    h = hashlib.sha256()
    for f in ("kernels.cuh", "device_common.cuh", "glibc_log.cuh", "glibc_log_data.cuh"):
        h.update(open(os.path.join(ROOT, "sage_b200", "csrc", f), "rb").read())
    return h.hexdigest()[:16]


def committed_traffic(workload, kernel):
    """dram bytes (read + write) per launch of `kernel` from the committed `ncu --set full` capture (profiles/traffic.json). Returns
    (bytes or None, note): a capture taken from other sources than the ones being timed is reported as stale, not used."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None, "no capture committed"
    try:
        t = json.load(open(p))
    except Exception:
        return None, "unreadable profiles/traffic.json"
    if t.get("_sources_sha") != kernel_sources_sha():
        return None, f"stale: profiles/traffic.json was captured from sources {t.get('_sources_sha')}, timing {kernel_sources_sha()}"
    return (t.get(workload) or {}).get(kernel), t.get("_source", "")


def host_threads():
    """All host cores this process may use (torchrun exports OMP_NUM_THREADS=1, so the count is passed to the oracle explicitly)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def oracle_throughput(pep, spectra, wl, steps, warmup, threads=0, check=None):
    """Times the CPU oracle (OpenMP over spectra) on a bounded sample of the same workload. Returns (rates, sample size, threads used[, PSMs checked])."""
    threads = threads or host_threads()
    from oracle import oracle as O
    from helpers import oracle_db_from_peptides
    t0 = time.time()
    odb = oracle_db_from_peptides(pep)
    log(f"oracle index built in {time.time() - t0:.1f}s ({odb.n_fragments} fragments)")
    cfg = O.ScorerConfig(**wl["scorer"])
    ns = min(wl["cpu_sample"], len(spectra))
    sub = spectra.slice(0, ns).as_dict()
    # give the CPU its best shot: SMT siblings often hurt this memory-bound code, so try all threads and half, keep the faster
    best = None
    for cand in sorted({threads, max(1, threads // 2)}, reverse=True):
        odb.score_batch(cfg, sub, nthreads=cand)  # warm the index
        t = time.perf_counter()
        odb.score_batch(cfg, sub, nthreads=cand)
        dt = time.perf_counter() - t
        if best is None or dt < best[0]:
            best = (dt, cand)
    threads = best[1]
    log(f"oracle threads: using {threads} (probe {best[0]:.3f}s per {ns} spectra)")
    rates = []
    for i in range(warmup + steps):
        t = time.perf_counter()
        odb.score_batch(cfg, sub, nthreads=threads)
        dt = time.perf_counter() - t
        if i >= warmup:
            rates.append(ns / dt)
    if check is not None:   # parity of the measured GPU results against the oracle on the CPU sample (same run, same inputs)
        from helpers import assert_features_equal
        gf, gc = check
        r = cfg.report_psms
        of, oc, _, _ = odb.score_batch(cfg, sub, nthreads=threads)
        check_n = assert_features_equal(gf[:ns * r], gc[:ns], of, oc, r, what="bench parity check")
        log(f"parity check: {check_n} PSMs of {ns} spectra identical to the oracle")
        return rates, ns, threads, check_n
    return rates, ns, threads


CPU_BUILD = "oracle/Makefile: g++ -O3 -march=x86-64-v3 -ffp-contract=off -fopenmp (no per-candidate allocation; parallel index build)"


def cpu_baseline_obj(rates, ns, threads, best=True):
    return {"value": float(max(rates) if best else np.mean(rates)), "unit": "spectra/s", "cores": host_threads(), "threads": threads, "kind": "port",
            "build": CPU_BUILD,
            "sample": f"{ns} spectra of the same workload per step; C++ port of sage-core's Scorer::score (oracle/), OpenMP dynamic over spectra; "
                      f"`cores` = host cores available to this process, `threads` = OpenMP threads of the faster of {{all, half}}"}


class Dist:
    """torch.distributed plumbing (NCCL): barrier + max/sum over ranks. No collective touches the data path."""

    def __init__(self, world, local_rank):
        import torch
        self.torch, self.world = torch, world
        torch.cuda.set_device(local_rank)
        if world > 1:
            import torch.distributed as dist
            self.dist = dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def _red(self, x, op):
        if self.world == 1:
            return float(x)
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=op)
        return float(t.item())

    def max(self, x):
        return self._red(x, self.dist.ReduceOp.MAX if self.world > 1 else None)

    def sum(self, x):
        return self._red(x, self.dist.ReduceOp.SUM if self.world > 1 else None)

    def close(self):
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


def base_config(name, wl, gpus, world):
    return {"workload": f"{name}: {wl['desc']}", "spectra_per_gpu": spectra_per_rank(wl, world), "peaks_per_spectrum": 200, "scaling": wl["scaling"],
            "sharding": f"spectra sharded across {gpus} GPU(s), index replicated, no collective",
            "l2": "per-step working set (index + ion tables >= 0.7 GB, spectra >= 40 MB) exceeds the 126 MB L2; no flush needed"}


DUMP_BYTES = 64 << 20


def dump_outputs(path, features, counts, report_psms):
    """Writes a PSM table as the arrays a caller receives: <field>.npy for every Feature field, shape (spectra, report_psms), float32 for the f32
    fields and float64 for the others (their integers are exact in it), and counts.npy. Rows past a spectrum's count are never written by the
    library and are zeroed here. spectra.npy holds the spectrum indices the rows belong to: all of them, or a fixed seeded sample when the table
    would exceed DUMP_BYTES."""
    fields = [f for f in features.dtype.names if not f.startswith("_")]
    n = len(counts)
    feats = features.reshape(n, report_psms).copy()
    feats[np.arange(report_psms)[None, :] >= np.asarray(counts)[:, None]] = np.zeros((), features.dtype)
    per_spectrum = 16 + report_psms * sum(4 if features.dtype[f] == np.float32 else 8 for f in fields)
    budget = DUMP_BYTES - 4096 * (len(fields) + 2)   # room for the .npy headers
    idx = np.arange(n)
    if n * per_spectrum > budget:
        idx = np.sort(np.random.default_rng(0).choice(n, budget // per_spectrum, replace=False))
    os.makedirs(path, exist_ok=True)
    for f in fields:
        a = feats[f][idx]
        np.save(os.path.join(path, f"{f}.npy"), a if a.dtype == np.float32 else a.astype(np.float64))
    np.save(os.path.join(path, "counts.npy"), np.asarray(counts)[idx].astype(np.float64))
    np.save(os.path.join(path, "spectra.npy"), idx.astype(np.float64))
    log(f"outputs of the last timed step ({len(idx)} of {n} spectra) written to {path}")


def run_workload(name, wl, steps, warmup, rank, local_rank, world, gpus, D, cpu, pageable=True, dump=None):
    """One workload on this repo's CUDA path. Returns the JSON-line dict (rank 0's view; all ranks must call it). dump: directory that receives
    rank 0's outputs of the last timed step of the resident path (dump_outputs)."""
    from sage_b200 import IndexedDatabase, Scorer, SpectraBatch, Tolerance, api
    pep, spectra = load_or_make(name, wl, rank, world)
    t0 = time.time()
    gdb = IndexedDatabase.build_from_peptides(pep, device=local_rank)
    build_s = time.time() - t0
    config = base_config(name, wl, gpus, world)
    config["n_peptides"] = len(pep)
    kw = dict(wl["scorer"])
    kw["precursor_tol"], kw["fragment_tol"] = Tolerance(*kw["precursor_tol"]), Tolerance(*kw["fragment_tol"])
    scorer = Scorer(gdb, **kw)
    n = len(spectra)

    # pinned host copies of the inputs/outputs (the e2e path DMA-copies straight from/to these); allocated after the NUMA binding in main()
    def pin(a):
        p = api.pinned_empty(a.shape, a.dtype)
        p[...] = a
        return p
    hspec = SpectraBatch(peak_off=spectra.peak_off, masses=pin(spectra.masses), intensities=pin(spectra.intensities), prec_mz=spectra.prec_mz,
                         prec_charge=spectra.prec_charge, iso_lo=spectra.iso_lo, iso_hi=spectra.iso_hi, tic=spectra.tic, level=spectra.level, rt=spectra.rt,
                         ims=spectra.ims)
    out = api.pinned_empty((n * scorer.report_psms,), api.FEATURE_DTYPE)
    counts = api.pinned_empty((n,), np.uint32)

    # ---- warm-up (both paths)
    for _ in range(warmup):
        scorer.score_batch(hspec, out, counts)
    scorer.upload(hspec)
    for _ in range(warmup):
        scorer.run()
    # One UNTIMED step in the reference's loop order (option narrow_index = 0) collects the work terms of SURVEY.md §8(d) — pages visited, index
    # entries scanned — that define the algorithmic bytes of this workload; the timed steps run the default path (narrow windows are counted against
    # the small-block copy of the index and never visit those pages).
    scorer.set_option("narrow_index", 0)
    scorer.run()
    work = scorer.counters()
    scorer.set_option("narrow_index", int(os.environ.get("SAGE_B200_NARROW_INDEX", "1") != "0"))   # (the env switch is for A/B runs of the old path)
    scorer.run()

    with ClockSampler(local_rank) as clocks:
        # ---- timed: K steps with the spectra resident in HBM; CUDA events on the launching stream (inside the library)
        D.barrier()
        ph = dict(total=0.0, prelim=0.0, score=0.0, setup=0.0, count=0.0)
        t0 = time.perf_counter()
        for _ in range(steps):
            scorer.run()
            c = scorer.counters()
            ph["total"] += c["ms_total"]; ph["prelim"] += c["ms_prelim"]; ph["score"] += c["ms_score"]; ph["setup"] += c["ms_setup"]; ph["count"] += c["ms_prelim_count"]
        D.barrier()
        wall_resident = time.perf_counter() - t0
        last = scorer.counters()
        resident_out = scorer.download() if dump else None   # untimed: the last timed step's results, as a caller of run() receives them
        # ---- timed: K steps end to end through sage_b200_score_batch (pinned host in, pinned host out)
        D.barrier()
        t0 = time.perf_counter()
        per_call, in_lib = [], []
        for _ in range(steps):
            t1 = time.perf_counter()
            scorer.score_batch(hspec, out, counts)
            per_call.append(time.perf_counter() - t1)
            in_lib.append(scorer.counters()["ms_wall"])
        D.barrier()
        wall_e2e = time.perf_counter() - t0
        e2e_c = scorer.counters()
        # ---- the same call with pageable host arrays (what a Rust Vec<f32> is): the library stages them through its own pinned buffers
        wall_page = None
        if pageable:
            pout, pcounts = np.zeros(n * scorer.report_psms, api.FEATURE_DTYPE), np.zeros(n, np.uint32)
            scorer.score_batch(spectra, pout, pcounts)
            D.barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                scorer.score_batch(spectra, pout, pcounts)
            D.barrier()
            wall_page = time.perf_counter() - t0
    dev_s = D.max(ph["total"] / 1000.0)
    wall_e2e = D.max(wall_e2e)
    wall_resident = D.max(wall_resident)
    if wall_page is not None:
        wall_page = D.max(wall_page)
    total_spectra = D.sum(n) * steps
    value = total_spectra / dev_s
    e2e_value = total_spectra / wall_e2e
    psms = int(counts.sum())

    peak, peak_src = measured_hbm_peak()
    # Kernels of one step, each with its CUDA-event time (per step) and its share of the SURVEY.md §8d algorithmic bytes; the roofline object
    # describes the one that takes longest. Open search: k_prelim_wide (timed together with its small replay kernel).
    count_s, replay_s, score_s = ph["count"] / 1000.0 / steps, (ph["prelim"] - ph["count"]) / 1000.0 / steps, ph["score"] / 1000.0 / steps
    if last["wide_queries"]:
        kernels = [("k_prelim_wide", ph["prelim"] / 1000.0 / steps, work["prelim_bytes"]), ("k_score", score_s, work["score_bytes"])]
    else:
        kernels = [("k_prelim_narrow_warp", count_s, work["prelim_bytes"]), ("k_replay", replay_s, 0), ("k_score", score_s, work["score_bytes"])]
    per_kernel = []
    for k, t, nb in kernels:
        tr, tr_note = committed_traffic(name, k)
        per_kernel.append({"kernel": k, "launch_ms": t * 1e3, "algorithmic_bytes_per_launch": int(nb), "achieved": (nb / t / 1e9 if t > 0 else 0.0),
                           "frac": (nb / t / 1e9 / peak if t > 0 else 0.0), "traffic": tr,
                           "dram_frac": (tr / t / 1e9 / peak if (tr and t > 0) else None), "traffic_note": tr_note})
    dom = max(per_kernel, key=lambda r: r["launch_ms"])
    step_s = dev_s / steps
    notes = {"k_score": "the scoring phase: k_score<true> (matching, one CTA per spectrum) + k_fold + k_features + k_rows (one thread per candidate / row) for non-chimeric "
                        "searches, the fused k_score otherwise. Instruction-issue / latency bound, not byte bound: per candidate ~2(L-1)Z sorted-array lookups in shared memory; its algorithmic bytes "
                        "(candidate records + intensities) are small, see DESIGN.md",
             "k_prelim_narrow_warp": "dependent-probe (latency / divergent-issue) bound, not stream bound: `frac` counts the REFERENCE algorithm's probe bytes "
                                     "(work terms of one untimed step in the reference's loop order) and can exceed 1 because the timed path answers the probes "
                                     "from the small-block copy of the index without visiting those pages; `dram_frac` is what DRAM really moved; see DESIGN.md",
             "k_prelim_wide": "open-search counting kernel; see DESIGN.md"}
    roofline = {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["achieved"], "peak": peak, "unit": "GB/s", "frac": dom["frac"],
                "traffic": dom["traffic"], "dram_frac": dom["dram_frac"], "traffic_note": dom["traffic_note"], "peak_source": peak_src,
                "algorithmic_bytes_per_launch": dom["algorithmic_bytes_per_launch"],
                "launch_ms": dom["launch_ms"], "note": notes.get(dom["kernel"], ""), "kernels": per_kernel,
                "step": {"algorithmic_bytes": int(work["algorithmic_bytes"]), "device_ms": step_s * 1e3,
                         "achieved": work["algorithmic_bytes"] / step_s / 1e9, "frac": work["algorithmic_bytes"] / step_s / 1e9 / peak}}
    e2e = {"value": e2e_value, "unit": "spectra/s", "h2d_bytes_per_step": int(e2e_c["h2d_bytes"]), "d2h_bytes_per_step": int(e2e_c["d2h_bytes"]),
           "ms_per_step": wall_e2e * 1000.0 / steps, "ms_per_call_median_rank0": float(np.median(per_call)) * 1000.0,
           "ms_per_call_max_rank0": float(np.max(per_call)) * 1000.0, "ms_in_library_median_rank0": float(np.median(in_lib))}
    if wall_page is not None:
        e2e["pageable"] = {"value": total_spectra / wall_page, "unit": "spectra/s", "ms_per_step": wall_page * 1000.0 / steps,
                           "note": "same C-ABI call with ordinary (unpinned) host arrays in and out"}
    result = {"metric": "spectra/sec", "value": value, "unit": "spectra/s", "n_gpus": gpus, "steps": steps, "warmup": warmup,
              "ms_per_step": dev_s * 1000.0 / steps, "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None, "dtype": "f32",
              "data": "synthetic", "config": config, "e2e": e2e,
              "gpu_launches": (int(last["kernel_launches"]) + int(e2e_c["kernel_launches"])) * steps * gpus,   # own kernels in both timed regions (cub sorts not counted)
              "roofline": roofline, "clocks": clocks.summary(),
              "index": {"n_peptides": len(pep), "n_fragments": int(gdb.info["n_fragments"]), "hbm_bytes": int(gdb.device_bytes()), "hbm_bytes_page_index": int(gdb.info["device_bytes"]), "build_s": round(build_s, 2)},
              "phases_ms_per_step": {"setup": ph["setup"] / steps, "prelim": ph["prelim"] / steps, "prelim_count": ph["count"] / steps, "score": ph["score"] / steps,
                                     "resident_wall": wall_resident * 1000.0 / steps, "e2e_h2d": e2e_c["ms_h2d"], "e2e_d2h": e2e_c["ms_d2h"]},
              "work_per_step": {k: int(work[k]) for k in ("queries", "tasks", "pages", "entries_scanned", "matched_fragments", "candidates_scored", "psms",
                                                          "algorithmic_bytes", "wide_queries", "wide_overflows", "pep_queries", "pep_fallbacks")},
              "psms_per_step_rank0": psms, "host_log_variant": api.host_log_variant()}

    if rank == 0 and cpu:
        rates, ns, threads, check_n = oracle_throughput(pep, spectra, wl, steps=2, warmup=1, check=(np.array(out), np.array(counts)))
        from helpers import f64_exact_default
        result["parity_checked"] = {"spectra": ns, "psms_identical_to_oracle": check_n,
                                    "tolerance": "every field bit-exact, incl. the f64 scores (device log == host libm log)" if f64_exact_default()
                                                 else "integer/f32 fields bit-exact; f64 scores rtol 1e-6 (tests/helpers.py)"}
        result["cpu_baseline"] = cpu_baseline_obj(rates, ns, threads)
    if dump and rank == 0:
        dump_outputs(dump, *resident_out, scorer.report_psms)
    del scorer, gdb
    for a in (hspec.masses, hspec.intensities, out, counts):
        api.pinned_free(a)
    return result


def slim(r):
    """The part of a workload's result that goes under `extra`."""
    keep = ("value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "config", "e2e", "index", "phases_ms_per_step", "parity_checked", "cpu_baseline",
            "psms_per_step_rank0")
    o = {k: r[k] for k in keep if k in r}
    o["roofline"] = {k: r["roofline"][k] for k in ("kernel", "achieved", "peak", "unit", "frac", "traffic", "dram_frac", "launch_ms", "algorithmic_bytes_per_launch")}
    return o


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="sage_b200", choices=["sage_b200", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra workloads (cfg4 / cfg5 / cfg3) that follow the headline one")
    ap.add_argument("--extras", default="", help="comma-separated subset of the extra workloads to run")
    ap.add_argument("--spectra", type=int, default=0, help="override the number of spectra per GPU (profiling only; invalidates the metric)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the PSM table the last timed step of the headline workload computed (rank 0) as DIR/<name>.npy, "
                         "at most 64 MB; the inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "sage_b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl sage_b200)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    wl = dict(WORKLOADS[args.workload])
    if args.spectra:
        wl["n_spectra"], wl["scaling"] = args.spectra, "weak"
        wl["desc"] += f" [PROFILING RUN: {args.spectra} spectra]"
    warmup = max(3, args.warmup)

    # ------------------------------------------------------------------ reference arm: CPU oracle port, rank 0 only
    if args.impl == "reference":
        if rank != 0:
            return
        pep, spectra = load_or_make(args.workload, wl, 0, world)
        rates, ns, threads = oracle_throughput(pep, spectra, wl, args.steps, warmup)
        v = float(np.mean(rates))
        config = base_config(args.workload, wl, args.gpus, world)
        config["n_peptides"] = len(pep)
        cb = cpu_baseline_obj(rates, ns, threads, best=False)
        out = {"impl": "reference", "metric": "spectra/sec", "value": v, "unit": "spectra/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": warmup,
               "ms_per_step": 1000.0 * ns / v, "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
               "config": config, "cpu_baseline": cb, "e2e": {"value": v, "unit": "spectra/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(out), flush=True)
        return

    # ------------------------------------------------------------------ this repo's arm
    from sage_b200 import api
    if api.device_count() == 0:
        raise SystemExit("bench.py: no CUDA device — sage_b200 has no CPU fallback")
    # this rank's host thread (and the pinned buffers it is about to allocate) on the NUMA node next to its GPU
    node = api.bind_thread_to_device(local_rank)
    D = Dist(world, local_rank)
    result = run_workload(args.workload, wl, args.steps, warmup, rank, local_rank, world, args.gpus, D, cpu=(args.gpus == 1 and not args.no_cpu_baseline),
                          dump=args.dump_outputs)
    result["numa_node"] = node
    extras = [] if (args.no_extras or args.spectra) else EXTRAS.get(args.workload, [])
    if args.extras:
        extras = [e for e in args.extras.split(",") if e in WORKLOADS]
    if extras:
        result["extra"] = {}
    for ex in extras:
        st, wu = EXTRA_STEPS.get(ex, (5, 3))
        # the oracle needs its own index of the extra workload: affordable for the 2M-peptide tables at N = 1, and for cfg3 only where
        # BASELINE.json places it (8 GPUs); elsewhere the at-size parity of cfg3 is covered by tests/test_gpu_fullsize.py
        cpu = rank == 0 and not args.no_cpu_baseline and ((ex != "cfg3" and args.gpus == 1) or (ex == "cfg3" and args.gpus == 8))
        try:
            r = run_workload(ex, dict(WORKLOADS[ex]), st, wu, rank, local_rank, world, args.gpus, D, cpu=cpu, pageable=False)
            result["extra"][ex] = slim(r)
        except Exception as e:   # an extra workload never takes the headline line down with it
            result["extra"][ex] = {"error": f"{type(e).__name__}: {e}"}
            if world > 1:
                raise
    if rank == 0:
        print(json.dumps(result), flush=True)
    D.close()


if __name__ == "__main__":
    main()
