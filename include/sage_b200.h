/* sage_b200.h — C ABI of the B200-native fragment-index search-and-score library.
 *
 * Drop-in boundary for ONE path of lazear/sage (reference @0639176): sage-core's
 *   IndexedDatabase::query / IndexedQuery::page_search   crates/sage/src/database.rs:402-536
 *   Scorer::score (score_standard / score_chimera_fast)   crates/sage/src/scoring.rs:300-767
 * A Rust shim (INTEGRATION.md) keeps `Scorer` / `IndexedDatabase` / `ProcessedSpectrum` as they are and forwards
 * `Scorer::score` / a new `Scorer::score_batch` to these entry points. Plain pointers and sizes only; no C++ or
 * torch types cross this boundary. All functions return 0 on success and a negative SAGE_B200_E* code on failure
 * (never unwind; the reference panics instead — see sage_b200_last_error for the message).
 *
 * Ownership: the caller owns every input/output buffer for the duration of a call; the library copies what it needs
 * to the device and keeps no host pointers. Thread-safety: one sage_b200_scorer may be used by one host thread at a
 * time (calls are serialised internally by a per-scorer mutex); distinct scorers on the same db are independent.
 */
#ifndef SAGE_B200_H
#define SAGE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SAGE_B200_OK 0
#define SAGE_B200_EINVAL (-1)     /* bad argument */
#define SAGE_B200_ECUDA (-2)      /* CUDA runtime error (message has the cudaError string) */
#define SAGE_B200_ENOTMS2 (-3)    /* reference: assert_eq!(query.level, 2)            scoring.rs:301-304 */
#define SAGE_B200_ENOPRECURSOR (-4) /* reference: panic!("missing MS1 precursor")      scoring.rs:466-468 */
#define SAGE_B200_ELIMIT (-5)     /* a documented capacity limit was exceeded */

typedef struct sage_b200_db sage_b200_db;         /* replaces &IndexedDatabase (device-resident)  database.rs:384-395 */
typedef struct sage_b200_scorer sage_b200_scorer; /* replaces Scorer<'db>                          scoring.rs:210-232 */

/* mass.rs:10-16  Tolerance::{Ppm,Pct,Da}(lo,hi) */
enum { SAGE_B200_TOL_PPM = 0, SAGE_B200_TOL_PCT = 1, SAGE_B200_TOL_DA = 2 };
typedef struct { int32_t kind; float lo, hi; } sage_b200_tolerance;

/* ion_series.rs:8-15  Kind */
enum { SAGE_B200_KIND_A = 0, SAGE_B200_KIND_B = 1, SAGE_B200_KIND_C = 2, SAGE_B200_KIND_X = 3, SAGE_B200_KIND_Y = 4, SAGE_B200_KIND_Z = 5 };

/* Peptides as the hot path reads them (peptide.rs:13-31), flattened CSR/SoA. `PeptideIx` == row index. */
typedef struct {
    uint64_t n_peptides;
    const uint32_t* residue_offsets; /* n_peptides+1; residues of peptide i are [off[i], off[i+1]) */
    const uint8_t* sequence;         /* Peptide::sequence bytes, concatenated */
    const float* modifications;      /* Peptide::modifications, parallel to sequence */
    const float* nterm;              /* Peptide::nterm, NaN = None */
    const float* monoisotopic;       /* Peptide::monoisotopic, ascending (database.rs:226-230) */
    const uint8_t* decoy;            /* Peptide::decoy */
    const uint8_t* missed_cleavages; /* Peptide::missed_cleavages */
} sage_b200_peptides;

/* The fragment index exactly as IndexedDatabase holds it (database.rs:378-395). */
typedef struct {
    uint64_t n_fragments;
    const uint32_t* fragment_peptide; /* Theoretical::peptide_index */
    const float* fragment_mz;         /* Theoretical::fragment_mz   */
    uint64_t n_buckets;
    const float* bucket_min;          /* IndexedDatabase::min_value */
    uint64_t bucket_size;             /* IndexedDatabase::bucket_size */
    const uint8_t* ion_kinds;         /* IndexedDatabase::ion_kinds (SAGE_B200_KIND_*) */
    uint64_t n_ion_kinds;
} sage_b200_index;

typedef struct {
    uint64_t n_peptides, n_fragments, n_buckets, bucket_size, n_ion_kinds, total_residues;
    uint64_t device_bytes; /* HBM held by this db */
    int32_t device;
} sage_b200_db_info;

/* Mirror of Scorer's public fields (scoring.rs:210-232). */
typedef struct {
    sage_b200_tolerance precursor_tol, fragment_tol;
    uint16_t min_matched_peaks;
    int8_t min_isotope_err, max_isotope_err;
    uint8_t min_precursor_charge, max_precursor_charge, override_precursor_charge;
    int8_t max_fragment_charge; /* Option<u8>: <0 = None */
    uint8_t chimera, wide_window, annotate_matches;
    uint8_t score_type; /* 0 = SageHyperScore, 1 = OpenMSHyperScore (scoring.rs:10-14) */
    uint32_t report_psms;
} sage_b200_scorer_params;

/* &[ProcessedSpectrum] flattened (spectrum.rs:47-79); only precursors.first() is read (scoring.rs:466). */
typedef struct {
    uint64_t n;
    const uint64_t* peak_offsets;     /* n+1 */
    const float* masses;              /* ProcessedSpectrum::masses (ascending) */
    const float* intensities;         /* ProcessedSpectrum::intensities */
    const float* precursor_mz;        /* Precursor::mz; NaN = spectrum has no precursor */
    const uint8_t* precursor_charge;  /* Precursor::charge; 0 = None */
    const float* isolation_lo;        /* Precursor::isolation_window = Some(Da(lo,hi)); NaN = None. May be NULL (all None) */
    const float* isolation_hi;
    const float* total_ion_current;   /* ProcessedSpectrum::total_ion_current */
    const uint8_t* level;             /* ProcessedSpectrum::level; NULL = all 2 */
    const float* scan_start_time;     /* -> Feature::rt / aligned_rt; NULL = 0 */
    const float* inverse_ion_mobility;/* Precursor::inverse_ion_mobility, NaN/NULL = None -> Feature::ims = 0 */
} sage_b200_spectra;

/* Numeric fields of Feature that the path computes (scoring.rs:69-149, 535-593). spec_id/file_id are re-attached by
 * the caller from `spectrum`; psm_id (global atomic, scoring.rs:163-167) is assigned by the caller after the call. */
typedef struct {
    uint32_t spectrum;      /* index into the batch */
    uint32_t peptide_idx;   /* PeptideIx */
    uint32_t peptide_len;
    uint32_t rank;
    int32_t label;          /* -1 decoy, 1 target */
    float expmass, calcmass;
    uint32_t charge;
    float rt, ims;
    float delta_mass, isotope_error, average_ppm;
    double hyperscore, delta_next, delta_best;
    uint32_t matched_peaks, longest_b, longest_y;
    float longest_y_pct;
    uint32_t missed_cleavages;
    float matched_intensity_pct;
    uint32_t scored_candidates;
    float ms2_intensity;
    double poisson;
    uint32_t fragment_offset, fragment_count; /* into the fragments array when annotate_matches */
} sage_b200_feature;

/* One matched fragment (scoring.rs:152-161, 738-751). */
typedef struct { int32_t kind, charge, ordinal; float intensity, mz_calculated, mz_experimental; } sage_b200_fragment;

/* Work counters of the last score_batch (SURVEY.md §8d algorithmic-bytes terms) + device timings (CUDA events, ms). */
typedef struct {
    uint64_t spectra, peaks, queries, tasks /* (peak,fragment-charge) probes */, pages, entries_scanned, matched_fragments,
        candidates_scored, peptide_record_floats, psms, wide_queries,
        pep_queries /* narrow queries counted peptide-centrically (pages/entries_scanned are then not visited, see DESIGN.md) */, pep_fallbacks,
        wide_overflows /* open-search queries whose survivor list overflowed (replayed inside the counting kernel) */;
    uint64_t algorithmic_bytes;    /* SURVEY.md §8d formula, whole batch */
    uint64_t prelim_bytes;         /* the part of it the preliminary-scoring kernel(s) move: peak masses, bucket / page probes, entries scanned */
    uint64_t score_bytes;          /* the part k_score moves: peak intensities, candidate peptide records, PSM rows */
    uint64_t h2d_bytes, d2h_bytes; /* bytes copied across PCIe for the batch */
    uint64_t kernel_launches;
    uint64_t chunk_retries;        /* chunks re-run because a device work list was sized too small (first batches of a scorer; see DESIGN.md) */
    float ms_total, ms_h2d, ms_setup, ms_prelim, ms_score, ms_d2h; /* summed over chunks */
    float ms_prelim_count;         /* the part of ms_prelim before the heap-replay kernels: k_prelim_narrow_warp + k_prelim_narrow */
    float ms_wall;                 /* host wall clock of the last score_batch call, entry to return (includes every copy and wait) */
} sage_b200_counters;

int sage_b200_device_count(void);

/* IndexedDatabase -> device. `index` as built by Parameters::build (database.rs:260-365). */
int sage_b200_db_create(const sage_b200_peptides* peptides, const sage_b200_index* index, int device, sage_b200_db** out);

/* Parameters::build_from_peptides on the device (database.rs:265-365): fragment generation for `ion_kinds` with the
 * `min_ion_index` filter, global sort by fragment m/z, bucketing, per-bucket sort by PeptideIx. */
int sage_b200_db_build(const sage_b200_peptides* peptides, uint64_t bucket_size, const uint8_t* ion_kinds, uint64_t n_ion_kinds,
                       uint64_t min_ion_index, int device, sage_b200_db** out);

int sage_b200_db_get_info(const sage_b200_db* db, sage_b200_db_info* info);
/* Copies the index back in the reference layout (IndexedDatabase::fragments / min_value); any pointer may be NULL. */
int sage_b200_db_export_index(const sage_b200_db* db, uint32_t* fragment_peptide, float* fragment_mz, float* bucket_min);
void sage_b200_db_destroy(sage_b200_db* db);

int sage_b200_scorer_create(const sage_b200_db* db, const sage_b200_scorer_params* params, sage_b200_scorer** out);
void sage_b200_scorer_destroy(sage_b200_scorer* scorer);
/* Tuning knobs that do not change results.
 *   "pep_cap"         precursor windows with at most this many peptides are counted by streaming the candidates' ion tables instead of
 *                     probing the fragment index (default 0 = always probe the index, the reference's loop order)
 *   "sort_spectra"    1 (default): process spectra in ascending precursor order for cache locality; results are returned in input order
 *   "pipeline_chunks" cut every batch into at least this many pipelined chunks (default 1: chunks of <= 65536 spectra)
 *   "narrow_index"    1 (default): narrow precursor windows (up to 8192 peptides) are counted against a second, peptide-block-major copy of the
 *                     fragment index (one short m/z run per probe); 0: the reference's loop order against the page index — identical results,
 *                     and the only mode that fills the counters `pages` / `entries_scanned` (the reference algorithm's work terms)
 *   "score_split"     1 (default): non-chimeric scoring runs as three kernels (match per spectrum; fold and rank / rows one thread per candidate);
 *                     0: one fused kernel per spectrum (always used for chimera, annotate_matches, quick_score) — identical results
 *   "mass_parts"      1..4 (default 2): the peak-mass copy of a chunk from PINNED caller memory is cut into this many runs of spectra and the
 *                     counting kernel is queued once per run, so it starts while the rest of the copy is in flight
 *   "wide_tile", "wide_lmax", "worklist_reset", "narrow_block"   test hooks (tile size / survivor-list size of the open-search kernel; forget learned
 *                     list sizes; peptides per block of the narrow-search copy, 0 = sized by the average precursor window) */
int sage_b200_scorer_set_option(sage_b200_scorer* scorer, const char* name, int64_t value);

/* Scorer::score over a batch (runner.rs:311-325 `par_iter().flat_map(|s| scorer.score(s))`).
 * features: caller-allocated, n * report_psms entries; spectrum i's PSMs are features[i*report_psms .. +counts[i]).
 * fragments/fragment_capacity/fragments_used: only with annotate_matches (may be NULL otherwise). */
int sage_b200_score_batch(sage_b200_scorer* scorer, const sage_b200_spectra* spectra, sage_b200_feature* features, uint32_t* counts,
                          sage_b200_fragment* fragments, uint64_t fragment_capacity, uint64_t* fragments_used);

/* Same result as sage_b200_score_batch, computed by several GPUs of one box from one host process: contiguous blocks of spectra go to
 * scorers[0..n) (one per device, each on its own index replica, one host thread each); no collective. annotate_matches is not supported here. */
int sage_b200_score_batch_multi(sage_b200_scorer* const* scorers, int n_scorers, const sage_b200_spectra* spectra, sage_b200_feature* features,
                                uint32_t* counts);

/* Pins the calling host thread to the CPUs of the NUMA node next to `device` (PCI topology from sysfs): call it on the thread that will
 * allocate pinned buffers for and submit batches to that GPU (score_batch_multi does it for its own worker threads; a rayon pool would do it in
 * its start handler). Returns the NUMA node, or -1 when the topology is unknown (nothing changed). */
int sage_b200_bind_thread_to_device(int device);

/* Scorer::quick_score over a batch (scoring.rs:255-298; prefilter of runner.rs:143-278). keep has one byte per peptide of the db and is
 * OR-ed (the reference stores `true` into &[AtomicBool]). prefilter_low_memory selects the branch of scoring.rs:270. */
int sage_b200_quick_score(sage_b200_scorer* scorer, const sage_b200_spectra* spectra, int prefilter_low_memory, uint8_t* keep);

/* The same call split in phases for device-resident reuse (one batch of <= 262144 spectra / 2^26 peaks):
 * upload makes the spectra resident in HBM, run launches the kernels (results stay on the device; may be repeated),
 * download copies the Feature rows back. score_batch == upload + run + download per chunk. */
int sage_b200_batch_upload(sage_b200_scorer* scorer, const sage_b200_spectra* spectra);
int sage_b200_batch_run(sage_b200_scorer* scorer);
int sage_b200_batch_download(sage_b200_scorer* scorer, sage_b200_feature* features, uint32_t* counts);

/* Scorer::initial_hits for one spectrum (scoring.rs:418-462): the preliminary list in the reference's heap order.
 * White-box hook used by the parity tests. Returns the list length (<= cap written) or a negative error. */
int64_t sage_b200_initial_hits(sage_b200_scorer* scorer, const sage_b200_spectra* one_spectrum, uint16_t* matched, uint32_t* peptide,
                               uint8_t* charge, int8_t* isotope_error, uint64_t cap, uint64_t* matched_peaks, uint64_t* scored_candidates);

int sage_b200_counters_get(const sage_b200_scorer* scorer, sage_b200_counters* out);

/* SpectrumProcessor (spectrum.rs:39-44, 263-412) for centroided MS2 spectra — the step right before the hot path (SURVEY.md §8 row f2). */
typedef struct { uint64_t take_top_n; uint8_t deisotope; float min_deisotope_mz; } sage_b200_processor_params;
typedef struct {                    /* &[RawSpectrum] flattened (spectrum.rs:81-106) */
    uint64_t n;
    const uint64_t* peak_offsets;   /* n+1 */
    const float* mz;                /* RawSpectrum::mz (ascending) */
    const float* intensity;         /* RawSpectrum::intensity */
    const uint8_t* precursor_charge;/* precursors.first().charge, 0 = None (deisotoping then assumes up to 3+, spectrum.rs:289-293) */
    const uint8_t* level;           /* ms_level; NULL = all 2; other levels are rejected */
} sage_b200_raw_spectra;
/* process(): out_peak_offsets[n+1]; out_masses / out_intensities sized for the raw peak count (at most min(raw, take_top_n) are kept per spectrum);
 * out_tic[n] = ProcessedSpectrum::total_ion_current. */
int sage_b200_process_spectra(int device, const sage_b200_processor_params* processor, const sage_b200_raw_spectra* raw, uint64_t* out_peak_offsets,
                              float* out_masses, float* out_intensities, float* out_tic);

/* tmt::find_reporter_ions (tmt.rs:193-211) over a batch: out[i * n_labels + l] = intensity of the most intense peak of spectrum i within
 * label_tolerance of labels[l] (offset -PROTON, as the reference), 0 where none (the unwrap_or_default of tmt::quantify, tmt.rs:333). */
int sage_b200_find_reporter_ions(int device, uint64_t n, const uint64_t* peak_offsets, const float* masses, const float* intensities, const float* labels,
                                 uint64_t n_labels, sage_b200_tolerance label_tolerance, float* out);

/* Which build of glibc's log() the host libm is (replaces Rust's f64::ln, scoring.rs:179-201 / :512): the kernels reproduce that function
 * operation by operation so that hyperscore, poisson and ranks under near-ties carry the same bits as the CPU path on this host.
 * 0 = x86-64 glibc on a CPU with FMA+AVX2 (`__log_fma`), 1 = the uncontracted build (`__log_sse2`/`__log_avx`, musl, aarch64),
 * -1 = neither matched std::log on the probe inputs (the device then uses variant 0; f64 fields agree to <= 1 ulp). */
int sage_b200_host_log_variant(void);
/* 1 when the host libm's log1pf (Rust's f32::ln_1p: OpenMS hyperscore, scoring.rs:190-197) is the glibc / fdlibm function the kernels reproduce. */
int sage_b200_host_log1pf_exact(void);
/* Test hook: out[i] = the device's evaluation of log(x[i]) with `variant` (0/1), or of (double)log1pf((float)x[i]) with variant 2 — compared bit for bit with the host libm by tests/test_glibc_log.py. */
int sage_b200_device_log(int device, int variant, const double* x, uint64_t n, double* out);

/* ---- Rescoring and FDR: the three steps the reference runs right after the search (runner.rs:533-537):
 *   spectrum_fdr   LDA discriminant (linear_discriminant.rs:133-231), posterior error (kde.rs), sort, spectrum_q_value   runner.rs:280-291, qvalue.rs:8-36
 *   picked_peptide / picked_protein   fdr.rs:16-190
 * Strings never cross this boundary: the caller interns the reference's competition keys once per database (INTEGRATION.md). */
typedef struct {
    sage_b200_tolerance precursor_tol;  /* Scorer's precursor tolerance: Ppm or Da (Pct is rejected, as the reference's unreachable!) */
    uint64_t n_peptides;                /* rows of the peptide table; when > 0 every Feature::peptide_idx must be below it (required with keys) */
    const uint32_t* peptide_key;        /* [n_peptides] picked-peptide key per PeptideIx (fdr.rs:126-131); NULL skips picked_peptide */
    uint64_t n_peptide_keys;            /* every peptide_key is < n_peptide_keys */
    const uint32_t* protein_key;        /* [n_peptides] id of Peptide::proteins, UINT32_MAX when proteins.len() != 1 (fdr.rs:160-162); NULL skips picked_protein */
    uint64_t n_protein_keys;            /* every other protein_key is < n_protein_keys */
    const float* aligned_rt;            /* [n] Feature::aligned_rt (LDA feature 16); NULL = Feature::rt (scoring.rs:583) */
    const float* delta_rt_model;        /* [n] Feature::delta_rt_model (feature 18); NULL = 0.999 (scoring.rs:584) */
    const float* delta_ims_model;       /* [n] Feature::delta_ims_model (feature 19); NULL = 0.999 (scoring.rs:585) */
} sage_b200_fdr_params;

/* The Feature fields the three steps write, for features[i] (input order). peptide_q / protein_q stay 1.0 where that stage is skipped
 * (and protein_q for peptides without a protein key); posterior_error stays 1.0 when the LDA cannot be fitted (scoring.rs:576-580). */
typedef struct { float discriminant_score, posterior_error, spectrum_q, peptide_q, protein_q; } sage_b200_fdr_row;

typedef struct {
    uint64_t spectrum_passing, peptide_passing, protein_passing; /* the usize each step returns (q <= 0.01) */
    double coef[20];                   /* LDA coefficients (NaN when not fitted) */
    uint32_t lda_fitted;               /* 0: score_psms returned None and the heuristic score was used (runner.rs:284-287) */
    float ms_h2d, ms_lda, ms_pep, ms_spectrum_q, ms_picked, ms_d2h; /* CUDA-event times of the phases, ms */
    float ms_wall;                     /* host wall clock of the call, entry to return */
} sage_b200_fdr_summary;

/* Runs spectrum_fdr, picked_peptide and picked_protein over n Feature rows (any order: one score_batch result, or several concatenated).
 * out[i] holds the fields for features[i]; order[r] (may be NULL) is the input index at rank r of the reference's sort (discriminant score
 * descending, ties by input index), which a caller applies to its Vec<Feature>. summary may be NULL. n = 0 does nothing.
 * Errors: EINVAL for a peptide_idx >= n_peptides, a key >= its count, keys without n_peptides, or a Pct tolerance; ELIMIT for n >= 2^32. */
int sage_b200_assign_fdr(int device, const sage_b200_feature* features, uint64_t n, const sage_b200_fdr_params* params, sage_b200_fdr_row* out,
                         uint32_t* order, sage_b200_fdr_summary* summary);

/* LinearDiscriminantAnalysis::train (linear_discriminant.rs:63-124) on caller rows: rows is n x d row-major (d <= 20), decoy[i] != 0 for
 * class 0. The same device reductions and host Gauss::solve as sage_b200_assign_fdr. Returns 0 with coef[0..d) written, 1 when the model
 * cannot be fitted (an empty class, a failed solve or non-finite coefficients; coef is then NaN), or a negative error. */
int sage_b200_lda_fit(int device, const double* rows, uint64_t n, uint32_t d, const uint8_t* decoy, double* coef);

/* Page-locked host buffers: spectra/feature arrays placed here are copied by DMA without a staging memcpy. */
void* sage_b200_host_alloc(size_t bytes);
/* The same for a batch sage_b200_score_batch_multi cuts into n_devices contiguous blocks: the i-th of n equal parts of the buffer is placed on the
 * NUMA node next to devices[i] (first touch by a bound thread), then the region is registered with CUDA. Release with sage_b200_host_free. */
void* sage_b200_host_alloc_blocks(size_t bytes, const int* devices, int n_devices);
void sage_b200_host_free(void* p);

/* Message of the last failure on the calling thread. Returns the message length. */
size_t sage_b200_last_error(char* buf, size_t cap);

#ifdef __cplusplus
}
#endif
#endif /* SAGE_B200_H */
