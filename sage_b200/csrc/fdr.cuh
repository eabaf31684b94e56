// fdr.cuh — rescoring and FDR after the search, on the device (included by sage_b200.cu after its error helpers):
//
//   spectrum_fdr     runner.rs:280-291: ml::linear_discriminant::score_psms (linear_discriminant.rs:133-231) or the heuristic score, the sort,
//                    ml::qvalue::spectrum_q_value (qvalue.rs:8-36)
//   picked_peptide   fdr.rs:123-153      picked_protein   fdr.rs:155-190      (both through Competition::assign_q_value, fdr.rs:59-120)
//
//   k_fdr_prep        mass-error sample, decoy flags, class counts, input validation
//   k_moments         per-class count / sum (or squared deviation) / min / max of a sample for Kde::new + Builder::build (kde.rs:21-32, 83-111)
//   k_kde_bins        bins x n Gaussian kernels (kde.rs:34-48, 113-120); bins are spread over CTAs, samples over chunks
//   k_lda_pass        LDA class sums / per-class scatter (linear_discriminant.rs:63-110); feature rows are built in shared memory per tile
//   k_lda_project     Σ w·x (linear_discriminant.rs:127-130), posterior error (kde.rs:148-168, linear_discriminant.rs:217-228)
//   k_spectrum_q      integer prefix counts, f32 divide; reverse cumulative min via cub
//   k_comp_*          per-key forward / reverse maxima (atomicMax on the total-order image), compaction, sort, PEP-sum q-values
//
// Determinism: every f64 sum runs over a grid whose shape depends on the input size only, in a fixed order; there are no f64 atomics, so two
// calls give identical bits. Integer atomics (counts, maxima on the ordered-int image) are exact in any order.
#pragma once

namespace sb {
namespace fdr {

constexpr int NF = 20;                  // linear_discriminant.rs:19
constexpr int RED_BLOCKS = 512;         // grid of the moment reductions (fixed: the summation tree depends on n only)
constexpr int RED_THREADS = 256;
constexpr int TILE = 256;               // rows per LDA tile (one per thread)
constexpr int LDA_MAX_BLOCKS = 592;     // 4 CTAs per SM
constexpr int KDE_THREADS = 256;        // bins per CTA of k_kde_bins
constexpr int PICK_CHUNK = 32;          // rows per thread in the PEP-sum scan

// f32::total_cmp as an unsigned ascending key (negative values flip every bit, positive ones the sign bit)
__host__ __device__ __forceinline__ uint32_t total_key(float x) {
    uint32_t u;
    memcpy(&u, &x, 4);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ __forceinline__ float from_total_key(uint32_t k) {
    const uint32_t u = (k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k;
    float x;
    memcpy(&x, &u, 4);
    return x;
}

// A fitted Kde pair + Estimator (kde.rs:14-32, 139-143); filled on the device by k_kde_mean / k_kde_setup.
struct Kde {
    double cnt[2];      // class 0 = decoy sample, 1 = target sample
    double mean[2];
    double h[2], cst[2];
    double pi, min, max, step;
    uint32_t bins;
};

// Estimator::posterior_error (kde.rs:148-168), `as usize` with Rust's saturating semantics (NaN and negatives -> 0)
__device__ __forceinline__ double kde_pep(const double* bins, const Kde& k, double score) {
    const double f = floor((score - k.min) / k.step);
    uint64_t lo;
    if (!(f > 0.0)) lo = 0;
    else if (f >= 18446744073709551616.0) lo = ~0ull;
    else lo = (uint64_t)f;
    const uint64_t last = k.bins ? k.bins - 1 : 0;
    lo = lo < last ? lo : last;
    const uint64_t hi = lo + 1 < last ? lo + 1 : last;
    const double lower = bins[lo], upper = bins[hi];
    const double lo_score = (double)lo * k.step + k.min;
    const double linear = (score - lo_score) / k.step;
    return lower + (upper - lower) * linear;
}

// ------------------------------------------------------------------------------------------------ prep / validation
__global__ void k_fdr_prep(const sage_b200_feature* __restrict__ f, uint64_t n, int is_da, uint64_t n_peptides, double* __restrict__ mass_err,
                           uint8_t* __restrict__ dec, unsigned long long* __restrict__ n_decoy, unsigned* __restrict__ err) {
    unsigned local = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const sage_b200_feature& x = f[i];
        // linear_discriminant.rs:140-144: delta_mass for Ppm, (expmass - calcmass) in f32 for Da
        mass_err[i] = is_da ? (double)__fsub_rn(x.expmass, x.calcmass) : (double)x.delta_mass;
        const bool d = x.label == -1;
        dec[i] = d;
        local += d;
        if (n_peptides && x.peptide_idx >= n_peptides) atomicOr(err, 1u);
    }
    if (local) atomicAdd(n_decoy, (unsigned long long)local);
}

__global__ void k_check_keys(const uint32_t* __restrict__ pk, uint64_t npk, const uint32_t* __restrict__ prk, uint64_t nprk, uint64_t n_peptides,
                             unsigned* __restrict__ err) {
    for (uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n_peptides; p += (uint64_t)gridDim.x * blockDim.x) {
        if (pk && pk[p] >= npk) atomicOr(err, 2u);
        if (prk && prk[p] != 0xFFFFFFFFu && prk[p] >= nprk) atomicOr(err, 4u);
    }
}

// ------------------------------------------------------------------------------------------------ KDE
// Partials per block: {cnt0, cnt1, s0, s1, min, max}. With mean == nullptr s_c = Σ x, else Σ (x - mean_c)^2 (ml/mod.rs:24-32).
// min/max over both classes use f64::min/max (NaN is skipped), kde.rs:104-109.
__global__ void __launch_bounds__(RED_THREADS) k_moments(const double* __restrict__ x, const uint8_t* __restrict__ dec, uint64_t n, const Kde* kde,
                                                         double* __restrict__ partials) {
    double c0 = 0, c1 = 0, s0 = 0, s1 = 0, mn = 1.7976931348623157e308, mx = -1.7976931348623157e308;
    const bool sq = kde != nullptr;
    const double m0 = sq ? kde->mean[0] : 0.0, m1 = sq ? kde->mean[1] : 0.0;
    for (uint64_t i = (uint64_t)blockIdx.x * RED_THREADS + threadIdx.x; i < n; i += (uint64_t)RED_BLOCKS * RED_THREADS) {
        const double v = x[i];
        if (dec[i]) { c0 += 1.0; s0 += sq ? (v - m0) * (v - m0) : v; }
        else { c1 += 1.0; s1 += sq ? (v - m1) * (v - m1) : v; }
        mn = fmin(mn, v);
        mx = fmax(mx, v);
    }
    __shared__ double sm[6][RED_THREADS];
    sm[0][threadIdx.x] = c0; sm[1][threadIdx.x] = c1; sm[2][threadIdx.x] = s0; sm[3][threadIdx.x] = s1; sm[4][threadIdx.x] = mn; sm[5][threadIdx.x] = mx;
    __syncthreads();
    for (int w = RED_THREADS / 2; w > 0; w >>= 1) {
        if (threadIdx.x < w) {
            const int a = threadIdx.x, b = threadIdx.x + w;
            for (int q = 0; q < 4; q++) sm[q][a] += sm[q][b];
            sm[4][a] = fmin(sm[4][a], sm[4][b]);
            sm[5][a] = fmax(sm[5][a], sm[5][b]);
        }
        __syncthreads();
    }
    if (threadIdx.x < 6) partials[blockIdx.x * 6 + threadIdx.x] = sm[threadIdx.x][0];
}

// Fixed-tree reduction of the RED_BLOCKS partials of k_moments (one block of RED_BLOCKS threads).
__device__ void reduce_moments(const double* partials, double out[6]) {
    __shared__ double sm[6][RED_BLOCKS];
    for (int q = 0; q < 6; q++) sm[q][threadIdx.x] = partials[threadIdx.x * 6 + q];
    __syncthreads();
    for (int w = RED_BLOCKS / 2; w > 0; w >>= 1) {
        if (threadIdx.x < w) {
            const int a = threadIdx.x, b = threadIdx.x + w;
            for (int q = 0; q < 4; q++) sm[q][a] += sm[q][b];
            sm[4][a] = fmin(sm[4][a], sm[4][b]);
            sm[5][a] = fmax(sm[5][a], sm[5][b]);
        }
        __syncthreads();
    }
    for (int q = 0; q < 6; q++) out[q] = sm[q][0];
}

// mean (ml/mod.rs:24-26), min/max (kde.rs:104-109)
__global__ void __launch_bounds__(RED_BLOCKS) k_kde_mean(const double* partials, Kde* k) {
    double m[6];
    reduce_moments(partials, m);
    if (threadIdx.x == 0) {
        k->cnt[0] = m[0]; k->cnt[1] = m[1];
        k->mean[0] = m[2] / m[0]; k->mean[1] = m[3] / m[1];
        k->min = m[4];
        k->max = m[5];
    }
}

// std (ml/mod.rs:28-32), Kde::new (kde.rs:21-32), P(decoy) and the bin step (kde.rs:98-110)
__global__ void __launch_bounds__(RED_BLOCKS) k_kde_setup(const double* partials, Kde* k, double bw_mul, uint32_t bins) {
    double m[6];
    reduce_moments(partials, m);
    if (threadIdx.x == 0) {
        for (int c = 0; c < 2; c++) {
            const double len = k->cnt[c];
            const double sigma = sqrt(m[2 + c] / len);
            k->h[c] = sigma * pow(4.0 / 3.0 / len, 1.0 / 5.0) * bw_mul;
            k->cst[c] = sqrt(2.0 * 3.141592653589793) * k->h[c] * len;
        }
        k->pi = k->cnt[0] / (k->cnt[0] + k->cnt[1]);
        k->step = (k->max - k->min) / (double)(bins - 1);
        k->bins = bins;
    }
}

// partial[chunk][bin][class] = Σ over the chunk's samples of the class of exp(-0.5 ((score_bin - x) / h)^2)   (kde.rs:34-48, 115)
__global__ void __launch_bounds__(KDE_THREADS) k_kde_bins(const double* __restrict__ x, const uint8_t* __restrict__ dec, uint64_t n, uint64_t chunk,
                                                          const Kde* kde, double* __restrict__ partial) {
    __shared__ double sx[KDE_THREADS];
    __shared__ uint8_t sd[KDE_THREADS];
    const Kde k = *kde;
    const uint32_t bin = blockIdx.x * KDE_THREADS + threadIdx.x;
    const double score = (double)bin * k.step + k.min;
    const uint64_t a = (uint64_t)blockIdx.y * chunk, b = a + chunk < n ? a + chunk : n;
    double acc0 = 0.0, acc1 = 0.0;
    for (uint64_t t = a; t < b; t += KDE_THREADS) {
        const uint64_t i = t + threadIdx.x;
        if (i < b) { sx[threadIdx.x] = x[i]; sd[threadIdx.x] = dec[i]; }
        __syncthreads();
        const int m = (int)(b - t < (uint64_t)KDE_THREADS ? b - t : (uint64_t)KDE_THREADS);
        for (int j = 0; j < m; j++) {
            const int c = sd[j] ? 0 : 1;
            const double u = (score - sx[j]) / k.h[c];
            const double e = exp(-0.5 * (u * u));
            if (c == 0) acc0 += e; else acc1 += e;
        }
        __syncthreads();
    }
    if (bin < k.bins) {
        partial[((uint64_t)blockIdx.y * k.bins + bin) * 2 + 0] = acc0;
        partial[((uint64_t)blockIdx.y * k.bins + bin) * 2 + 1] = acc1;
    }
}

// bins[b] = decoy / (target + decoy) with pdf = Σ / constant (kde.rs:38-48, 113-119), chunks summed in order
__global__ void k_kde_finish(const double* __restrict__ partial, uint32_t nchunks, const Kde* kde, double* __restrict__ bins) {
    const Kde k = *kde;
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= k.bins) return;
    double s0 = 0.0, s1 = 0.0;
    for (uint32_t c = 0; c < nchunks; c++) {
        s0 += partial[((uint64_t)c * k.bins + b) * 2 + 0];
        s1 += partial[((uint64_t)c * k.bins + b) * 2 + 1];
    }
    const double decoy = s0 / k.cst[0] * k.pi;
    const double target = s1 / k.cst[1] * (1.0 - k.pi);
    bins[b] = decoy / (target + decoy);
}

// kde.rs:122-129: reverse running max (f64::max skips NaN)
__global__ void k_kde_monotonic(const Kde* kde, double* bins) {
    const uint32_t nb = kde->bins;
    double acc = bins[nb - 1];
    for (uint32_t i = nb; i-- > 0;) {
        acc = fmax(acc, bins[i]);
        bins[i] = acc;
    }
}

// ------------------------------------------------------------------------------------------------ LDA rows
// score_psms' compute_features (linear_discriminant.rs:162-193), exactly as the code builds the row.
struct FeatureRows {
    const sage_b200_feature* f;
    const double* mass_err;
    const uint8_t* dec;
    const float *aligned_rt, *delta_rt, *delta_ims;
    const double* mass_bins;
    const Kde* mass_kde;
    __device__ __forceinline__ bool decoy(uint64_t i) const { return dec[i]; }
    __device__ __forceinline__ void row(uint64_t i, const Kde& mk, double* r) const {
        const sage_b200_feature& x = f[i];
        double poisson = log1p(-x.poisson);
        if (!isfinite(poisson)) poisson = 3.5;
        auto clamp_sqrt = [](double v) { v = v < 0.001 ? 0.001 : (v > 0.999 ? 0.999 : v); return sqrt(v); };   // f64::clamp keeps NaN
        r[0] = (double)x.rank;
        r[1] = (double)x.charge;
        r[2] = log1p(x.hyperscore);
        r[3] = log1p(x.delta_next);
        r[4] = log1p(x.delta_best);
        r[5] = kde_pep(mass_bins, mk, mass_err[i]);
        r[6] = (double)x.isotope_error;
        r[7] = (double)x.average_ppm;
        r[8] = poisson;
        r[9] = log1p((double)x.matched_intensity_pct);
        r[10] = (double)x.matched_peaks;
        r[11] = log1p((double)x.longest_b);
        r[12] = log1p((double)x.longest_y);
        r[13] = (double)x.longest_y / (double)x.peptide_len;
        r[14] = log1p((double)x.peptide_len);
        r[15] = (double)x.missed_cleavages;
        r[16] = (double)(aligned_rt ? aligned_rt[i] : x.rt);
        r[17] = (double)x.ims;
        r[18] = clamp_sqrt((double)(delta_rt ? delta_rt[i] : 0.999f));
        r[19] = clamp_sqrt((double)(delta_ims ? delta_ims[i] : 0.999f));
    }
};

// Caller rows (sage_b200_lda_fit): n x d, zero-padded to NF columns
struct MatrixRows {
    const double* rows;
    const uint8_t* dec;
    uint32_t d;
    const Kde* mass_kde;   // unused
    __device__ __forceinline__ bool decoy(uint64_t i) const { return dec[i] != 0; }
    __device__ __forceinline__ void row(uint64_t i, const Kde&, double* r) const {
        for (int j = 0; j < NF; j++) r[j] = j < (int)d ? rows[i * d + j] : 0.0;
    }
};

__constant__ uint8_t c_pair_j[210], c_pair_k[210];   // the 210 entries j <= k of a 20 x 20 symmetric matrix

// pass 0: partials[block][class][j] = Σ row_j; pass 1: partials[block][class][pair] = Σ (row_j - mu_j)(row_k - mu_k)  (linear_discriminant.rs:72-105)
template <class Rows>
__global__ void __launch_bounds__(TILE) k_lda_pass(Rows rows, uint64_t n, int pass, const double* __restrict__ mean, double* __restrict__ partials) {
    __shared__ double sx[TILE][NF + 1];
    __shared__ uint8_t scls[TILE];
    Kde mk;
    if (rows.mass_kde) mk = *rows.mass_kde;
    const uint64_t ntiles = (n + TILE - 1) / TILE;
    double acc0 = 0.0, acc1 = 0.0;
    const int j = pass == 0 ? threadIdx.x % NF : (threadIdx.x < 210 ? c_pair_j[threadIdx.x] : 0);
    const int k = pass == 0 ? 0 : (threadIdx.x < 210 ? c_pair_k[threadIdx.x] : 0);
    const bool active = pass == 0 ? threadIdx.x < NF : threadIdx.x < 210;
    for (uint64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const uint64_t i = t * TILE + threadIdx.x;
        if (i < n) {
            double r[NF];
            rows.row(i, mk, r);
            const int c = rows.decoy(i) ? 0 : 1;
            if (pass == 1)
#pragma unroll
                for (int q = 0; q < NF; q++) r[q] = r[q] - mean[c * NF + q];
#pragma unroll
            for (int q = 0; q < NF; q++) sx[threadIdx.x][q] = r[q];
            scls[threadIdx.x] = (uint8_t)c;
        } else {
            scls[threadIdx.x] = 2;
        }
        __syncthreads();
        if (active) {
            for (int m = 0; m < TILE; m++) {
                const int c = scls[m];
                if (c == 2) break;
                const double v = pass == 0 ? sx[m][j] : sx[m][j] * sx[m][k];
                if (c == 0) acc0 += v; else acc1 += v;
            }
        }
        __syncthreads();
    }
    const int width = pass == 0 ? NF : 210;
    if (active) {
        const int e = pass == 0 ? j : threadIdx.x;
        partials[((uint64_t)blockIdx.x * 2 + 0) * width + e] = acc0;
        partials[((uint64_t)blockIdx.x * 2 + 1) * width + e] = acc1;
    }
}

// out[e] = Σ_blocks partials[block][e], blocks in order
__global__ void k_sum_blocks(const double* __restrict__ partials, uint32_t nblocks, uint32_t width, double* __restrict__ out) {
    const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= width) return;
    double s = 0.0;
    for (uint32_t b = 0; b < nblocks; b++) s += partials[(uint64_t)b * width + e];
    out[e] = s;
}

struct Coef { double w[NF]; };

// LinearDiscriminantAnalysis::score (Σ w·x in index order from 0.0) -> discriminant as f64 (for the KDE) and f32 (the Feature field)
__global__ void k_lda_project(FeatureRows rows, uint64_t n, Coef coef, double* __restrict__ disc64, float* __restrict__ disc32) {
    const Kde mk = *rows.mass_kde;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        double r[NF];
        rows.row(i, mk, r);
        double s = 0.0;
#pragma unroll
        for (int q = 0; q < NF; q++) s += coef.w[q] * r[q];
        disc64[i] = s;
        disc32[i] = (float)s;
    }
}

// linear_discriminant.rs:217-228: posterior_error = log10(pep) as f32, -324 for an infinite result
__global__ void k_posterior_error(const double* __restrict__ disc64, uint64_t n, const double* __restrict__ bins, const Kde* kde, float* __restrict__ pe) {
    const Kde k = *kde;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        float v = (float)log10(kde_pep(bins, k, disc64[i]));
        if (isinf(v)) v = -324.0f;
        pe[i] = v;
    }
}

// runner.rs:284-287: (-poisson as f32).ln_1p() + longest_y_pct / 3.0 in f32 (log1pf as glibc computes it); posterior_error keeps 1.0.
// NaN bits as the x86-64 host leaves them, where the device's own arithmetic would give its canonical 0x7fffffff: `-` flips a NaN's sign,
// the f64 -> f32 conversion keeps the top 23 payload bits and quiets, `/` and `+` with one NaN operand return it quieted, an invalid `+`
// (inf - inf) gives 0xffc00000, and when both addends are NaN the quotient's is returned (the host's operand order, pinned by a CPU test).
__global__ void k_fallback(const sage_b200_feature* __restrict__ f, uint64_t n, float* __restrict__ disc32, float* __restrict__ pe) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const double poisson = f[i].poisson;
        const uint64_t nb = (uint64_t)__double_as_longlong(poisson) ^ 0x8000000000000000ull;   // -poisson
        const float p = isnan(poisson) ? __uint_as_float((uint32_t)(nb >> 32 & 0x80000000u) | 0x7fc00000u | (uint32_t)(nb >> 29 & 0x7fffffu))
                                       : __double2float_rn(-poisson);
        const float l = glog::glibc_log1pf(p), y = f[i].longest_y_pct;
        const float q = isnan(y) ? __uint_as_float(__float_as_uint(y) | 0x00400000u) : __fdiv_rn(y, 3.0f);
        const float s = __fadd_rn(l, q);
        disc32[i] = isnan(q) ? q : isnan(l) ? l : isnan(s) ? __uint_as_float(0xffc00000u) : s;
        pe[i] = 1.0f;
    }
}

// ------------------------------------------------------------------------------------------------ sort + spectrum q
__global__ void k_sort_keys(const float* __restrict__ disc32, uint64_t n, uint32_t* __restrict__ key, uint32_t* __restrict__ idx) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        key[i] = total_key(disc32[i]);
        idx[i] = (uint32_t)i;
    }
}

__global__ void k_rank_decoy(const uint32_t* __restrict__ order, const uint8_t* __restrict__ dec, uint64_t n, uint32_t* __restrict__ flag) {
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (uint64_t)gridDim.x * blockDim.x) flag[r] = dec[order[r]];
}

// qvalue.rs:14-23: decoy = 1 + #decoys, target = #targets up to rank r; q = decoy as f32 / target as f32. Stored reversed for the min-scan.
__global__ void k_spectrum_q(const uint32_t* __restrict__ ndec, uint64_t n, float* __restrict__ qrev) {
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t d = 1ull + ndec[r], t = r + 1 - ndec[r];
        qrev[n - 1 - r] = __fdiv_rn(__ull2float_rn(d), __ull2float_rn(t));
    }
}

struct MinF32 {
    __device__ __forceinline__ float operator()(float a, float b) const { return fminf(a, b); }   // f32::min (NaN skipped)
};

// qvalue.rs:25-34: q at rank r = min(1, min over ranks >= r); passing counts every row (decoys too) with q <= 0.01
__global__ void k_spectrum_q_final(const float* __restrict__ qscan, const uint32_t* __restrict__ order, uint64_t n, sage_b200_fdr_row* __restrict__ out,
                                   unsigned long long* __restrict__ passing) {
    unsigned local = 0;
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (uint64_t)gridDim.x * blockDim.x) {
        const float q = fminf(1.0f, qscan[n - 1 - r]);
        out[order[r]].spectrum_q = q;
        local += q <= 0.01f;
    }
    if (local) atomicAdd(passing, (unsigned long long)local);
}

__global__ void k_write_scores(const float* __restrict__ disc32, const float* __restrict__ pe, uint64_t n, sage_b200_fdr_row* __restrict__ out) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        sage_b200_fdr_row o;
        o.discriminant_score = disc32[i];
        o.posterior_error = pe[i];
        o.spectrum_q = 1.0f;
        o.peptide_q = 1.0f;
        o.protein_q = 1.0f;
        out[i] = o;
    }
}

// ------------------------------------------------------------------------------------------------ picked competitions
__global__ void k_comp_init(uint64_t nk, uint32_t* __restrict__ fwd, uint32_t* __restrict__ rev, uint32_t* __restrict__ flags) {
    const uint32_t lowest = total_key(-3.40282347e38f);   // Competition::default: f32::MIN (fdr.rs:31-40)
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < nk; k += (uint64_t)gridDim.x * blockDim.x) {
        fwd[k] = lowest;
        rev[k] = lowest;
        flags[k] = 0;
    }
}

// fdr.rs:125-144 / 160-177: per key, forward / reverse = f32::max of the discriminant scores (NaN skipped), and which sides are present.
// Equal values of opposite sign (±0) are ordered as f32::total_cmp orders them, +0 above -0, whatever order the features come in; the
// reference's f32::max leaves that choice open, and fdr_oracle.cpp makes the same one.
__global__ void k_comp_max(const sage_b200_feature* __restrict__ f, const float* __restrict__ disc32, uint64_t n, const uint32_t* __restrict__ key_of,
                           uint32_t* __restrict__ fwd, uint32_t* __restrict__ rev, uint32_t* __restrict__ flags) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t key = key_of[f[i].peptide_idx];
        if (key == 0xFFFFFFFFu) continue;
        const int side = f[i].label == -1;
        atomicOr(&flags[key], 1u << side);
        const float s = disc32[i];
        if (!isnan(s)) atomicMax(side ? &rev[key] : &fwd[key], total_key(s));
    }
}

__global__ void k_comp_counts(const uint32_t* __restrict__ flags, uint64_t nk, uint32_t* __restrict__ nrows, uint32_t* __restrict__ present) {
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < nk; k += (uint64_t)gridDim.x * blockDim.x) {
        nrows[k] = __popc(flags[k]);
        present[k] = flags[k] != 0;
    }
}

// One KDE sample per present key (Competition::score / is_decoy, fdr.rs:43-57) and one row per present side, in key order, target first.
__global__ void k_comp_emit(const uint32_t* __restrict__ flags, const uint32_t* __restrict__ fwd, const uint32_t* __restrict__ rev, uint64_t nk,
                            const uint32_t* __restrict__ row_pos, const uint32_t* __restrict__ key_pos, double* __restrict__ kx, uint8_t* __restrict__ kdec,
                            uint32_t* __restrict__ row_key, uint32_t* __restrict__ row_id) {
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < nk; k += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t fl = flags[k];
        if (!fl) continue;
        const float fw = from_total_key(fwd[k]), rv = from_total_key(rev[k]);
        kx[key_pos[k]] = (double)from_total_key(max(fwd[k], rev[k]));   // in total order, as the per-side maxima: +0 above -0
        kdec[key_pos[k]] = rv >= fw;
        uint32_t p = row_pos[k];
        if (fl & 1u) { row_key[p] = fwd[k]; row_id[p] = (uint32_t)(2 * k); p++; }
        if (fl & 2u) { row_key[p] = rev[k]; row_id[p] = (uint32_t)(2 * k + 1); }
    }
}

// fdr.rs:89-100, per chunk of PICK_CHUNK sorted rows: pep = posterior_error(score) as f32; chunk sums of pep (f64) and of targets
__global__ void k_pick_chunk(const uint32_t* __restrict__ skey, const uint32_t* __restrict__ sid, uint64_t nr, const double* __restrict__ bins,
                             const Kde* kde, float* __restrict__ pep, double* __restrict__ csum, uint32_t* __restrict__ ctgt) {
    const Kde k = *kde;
    const uint64_t nch = (nr + PICK_CHUNK - 1) / PICK_CHUNK;
    for (uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; c < nch; c += (uint64_t)gridDim.x * blockDim.x) {
        double s = 0.0;
        uint32_t t = 0;
        const uint64_t e = (c + 1) * PICK_CHUNK < nr ? (c + 1) * PICK_CHUNK : nr;
        for (uint64_t r = c * PICK_CHUNK; r < e; r++) {
            const float p = (float)kde_pep(bins, k, (double)from_total_key(skey[r]));
            pep[r] = p;
            s += (double)p;
            t += (sid[r] & 1u) == 0;
        }
        csum[c] = s;
        ctgt[c] = t;
    }
}

// Exclusive prefix of the chunk sums, in a fixed order: one block, each thread a contiguous run of chunks.
__global__ void __launch_bounds__(1024) k_pick_chunk_scan(double* __restrict__ csum, uint32_t* __restrict__ ctgt, uint64_t nch) {
    __shared__ double ss[1024];
    __shared__ uint32_t st[1024];
    const uint64_t per = (nch + 1023) / 1024, a = threadIdx.x * per, b = a + per < nch ? a + per : nch;
    double s = 0.0;
    uint32_t t = 0;
    for (uint64_t c = a; c < b; c++) { s += csum[c]; t += ctgt[c]; }
    ss[threadIdx.x] = s;
    st[threadIdx.x] = t;
    __syncthreads();
    if (threadIdx.x == 0) {
        double run = 0.0;
        uint32_t trun = 0;
        for (int q = 0; q < 1024; q++) {
            const double v = ss[q];
            const uint32_t w = st[q];
            ss[q] = run;
            st[q] = trun;
            run += v;
            trun += w;
        }
    }
    __syncthreads();
    s = ss[threadIdx.x];
    t = st[threadIdx.x];
    for (uint64_t c = a; c < b; c++) {
        const double v = csum[c];
        const uint32_t w = ctgt[c];
        csum[c] = s;
        ctgt[c] = t;
        s += v;
        t += w;
    }
}

// q = (1 + Σ pep) / #targets in f32 (fdr.rs:89-100), stored reversed for the min-scan
__global__ void k_pick_q(const uint32_t* __restrict__ sid, const float* __restrict__ pep, uint64_t nr, const double* __restrict__ csum,
                         const uint32_t* __restrict__ ctgt, float* __restrict__ qrev) {
    const uint64_t nch = (nr + PICK_CHUNK - 1) / PICK_CHUNK;
    for (uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; c < nch; c += (uint64_t)gridDim.x * blockDim.x) {
        double s = csum[c];
        uint32_t t = ctgt[c];
        const uint64_t e = (c + 1) * PICK_CHUNK < nr ? (c + 1) * PICK_CHUNK : nr;
        for (uint64_t r = c * PICK_CHUNK; r < e; r++) {
            s += (double)pep[r];
            t += (sid[r] & 1u) == 0;
            qrev[nr - 1 - r] = __fdiv_rn((float)(1.0 + s), (float)t);
        }
    }
}

// fdr.rs:103-111: reverse cumulative min from 1.0; passing counts targets only
__global__ void k_pick_final(const float* __restrict__ qscan, const uint32_t* __restrict__ sid, uint64_t nr, float* __restrict__ qside,
                             unsigned long long* __restrict__ passing) {
    unsigned local = 0;
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < nr; r += (uint64_t)gridDim.x * blockDim.x) {
        const float q = fminf(1.0f, qscan[nr - 1 - r]);
        qside[sid[r]] = q;
        local += q <= 0.01f && (sid[r] & 1u) == 0;
    }
    if (local) atomicAdd(passing, (unsigned long long)local);
}

__global__ void k_pick_write(const sage_b200_feature* __restrict__ f, uint64_t n, const uint32_t* __restrict__ key_of, const float* __restrict__ qside,
                             int protein, sage_b200_fdr_row* __restrict__ out) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t key = key_of[f[i].peptide_idx];
        if (key == 0xFFFFFFFFu) continue;
        const float q = qside[2 * (uint64_t)key + (f[i].label == -1)];
        if (protein) out[i].protein_q = q; else out[i].peptide_q = q;
    }
}

}  // namespace fdr
}  // namespace sb

// ================================================================================================ host side
namespace {

using namespace sb::fdr;

// Gauss::solve (gauss.rs:26-165) on a d x d system with one right-hand column, row-major; restated operation by operation.
struct Gauss {
    int n;
    std::vector<double> L, R;
    double& l(int i, int j) { return L[(size_t)i * n + j]; }
    void swap_rows(int i, int j) {
        for (int k = 0; k < n; k++) std::swap(l(i, k), l(j, k));
        std::swap(R[i], R[j]);
    }
    void echelon() {
        int h = 0, k = 0;
        while (h < n && k < n) {
            int imax = 0;
            double vmax = -1.7976931348623157e308;
            for (int i = h; i < n; i++)
                if (l(i, k) >= vmax) { imax = i; vmax = l(i, k); }
            const int i = imax;
            if (l(i, k) == 0.0) { k++; continue; }
            if (h != imax) swap_rows(h, i);
            for (int r = h + 1; r < n; r++) {
                const double factor = l(r, k) / l(h, k);
                l(r, k) = 0.0;
                for (int j = k + 1; j < n; j++) l(r, j) -= l(h, j) * factor;
                R[r] -= R[h] * factor;
            }
            h++;
            k++;
        }
    }
    void reduce() {
        for (int i = n - 1; i >= 0; i--)
            for (int j = 0; j < n; j++) {
                const double x = l(i, j);
                if (x == 0.0) continue;
                for (int k = j; k < n; k++) l(i, k) /= x;
                R[i] /= x;
                break;
            }
    }
    void backfill() {
        for (int i = n - 1; i >= 0; i--)
            for (int j = 0; j < n; j++) {
                if (l(i, j) == 0.0) continue;
                for (int k = 0; k < i; k++) {
                    const double factor = l(k, j) / l(i, j);
                    for (int h = 0; h < n; h++) l(k, h) -= l(i, h) * factor;
                    R[k] -= R[i] * factor;
                }
                break;
            }
    }
    bool left_solved() {
        for (int i = 0; i < n; i++)
            for (int j = 0; j < n; j++) {
                const double x = l(i, j);
                if (i == j) { if (x != 1.0 && x != 0.0) return false; }
                else if (x > 1e-8) return false;
            }
        return true;
    }
    static bool solve(const std::vector<double>& left, const std::vector<double>& right, int n, std::vector<double>& out) {
        double eps = 1e-8;
        while (eps <= 1.0) {
            Gauss g{n, left, right};
            for (int i = 0; i < n; i++) g.l(i, i) += eps;   // fill_zero
            g.echelon();
            g.reduce();
            g.backfill();
            if (g.left_solved()) { out = g.R; return true; }
            eps *= 10.0;
        }
        return false;
    }
};

struct FdrDevice {
    std::mutex mu;
    bool init = false;
    cudaStream_t st = nullptr;
    cudaEvent_t ev[7] = {};
    DevBuf arena, temp;
    PinBuf stage;
    StagePool pool;
};
FdrDevice g_fdr[64];

// Carves one allocation into aligned pieces; pass 1 (base == nullptr) only measures.
struct Carve {
    char* base;
    size_t off = 0;
    template <class T>
    T* take(uint64_t count) {
        off = (off + 255) / 256 * 256;
        T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
        off += sizeof(T) * count;
        return p;
    }
};

unsigned grid_for(uint64_t n, unsigned threads = 256, unsigned cap = 148 * 8) {
    const uint64_t g = (n + threads - 1) / threads;
    return (unsigned)std::max<uint64_t>(1, std::min<uint64_t>(g, cap));
}

// Device buffers of one assign_fdr / lda_fit call
struct FdrBufs {
    sage_b200_feature* f;
    sage_b200_fdr_row* out;
    double *mass_err, *disc64, *mom, *kde_part, *mass_bins, *disc_bins, *lda_part, *lda_sum, *mean, *kx, *csum;
    float *disc32, *pe, *qa, *qb, *pep, *qside;
    uint8_t *dec, *kdec;
    uint32_t *key, *key_out, *idx, *order, *flag, *ndec, *pk, *prk, *fwd, *rev, *kflags, *nrows, *present, *row_pos, *key_pos, *ctgt;
    float *art, *drt, *dims;
    double* rows;
    Kde* kde;   // [0] mass model, [1] discriminant, [2] picked
    unsigned long long* counters;   // [0] decoys, [1] spectrum passing, [2] peptide passing, [3] protein passing
    unsigned* err;
};

uint32_t kde_chunks(uint64_t n, uint32_t bins) {
    const uint64_t bin_blocks = (bins + KDE_THREADS - 1) / KDE_THREADS;
    const uint64_t want = std::max<uint64_t>(1, (148 * 8 + bin_blocks - 1) / bin_blocks);
    return (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(want, (n + KDE_THREADS - 1) / KDE_THREADS));
}

// k_kde_bins partials for any bin count <= max_bins: chunks x bins <= (1184 + bin blocks) x 256
uint64_t kde_partials(uint32_t max_bins) { return 2ull * (148 * 8 + (max_bins + KDE_THREADS - 1) / KDE_THREADS) * KDE_THREADS; }

// Builder::build (kde.rs:83-136) over x[0..n) with decoy flags: fills kde[slot] and bins[0..bins)
int kde_build(cudaStream_t st, const double* x, const uint8_t* dec, uint64_t n, uint32_t bins, bool monotonic, double bw_mul, Kde* kde, double* mom,
              double* part, double* out_bins) {
    k_moments<<<RED_BLOCKS, RED_THREADS, 0, st>>>(x, dec, n, nullptr, mom);
    k_kde_mean<<<1, RED_BLOCKS, 0, st>>>(mom, kde);
    k_moments<<<RED_BLOCKS, RED_THREADS, 0, st>>>(x, dec, n, kde, mom);
    k_kde_setup<<<1, RED_BLOCKS, 0, st>>>(mom, kde, bw_mul, bins);
    const uint32_t nch = kde_chunks(n, bins);
    const uint64_t chunk = ((n + nch - 1) / nch + KDE_THREADS - 1) / KDE_THREADS * KDE_THREADS;
    k_kde_bins<<<dim3((bins + KDE_THREADS - 1) / KDE_THREADS, nch), KDE_THREADS, 0, st>>>(x, dec, n, chunk, kde, part);
    k_kde_finish<<<(bins + 255) / 256, 256, 0, st>>>(part, nch, kde, out_bins);
    if (monotonic) k_kde_monotonic<<<1, 1, 0, st>>>(kde, out_bins);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// LinearDiscriminantAnalysis::train (linear_discriminant.rs:63-124): device class sums and scatter, host solve. Returns 1 = fitted.
template <class Rows>
int lda_train(cudaStream_t st, const Rows& rows, uint64_t n, uint64_t n_decoy, uint32_t d, const FdrBufs& B, std::vector<double>& coef) {
    const uint64_t cnt[2] = {n_decoy, n - n_decoy};
    coef.assign(d, NAN);
    if (cnt[0] == 0 || cnt[1] == 0) return 0;
    const uint32_t nb = (uint32_t)std::min<uint64_t>((n + TILE - 1) / TILE, LDA_MAX_BLOCKS);
    k_lda_pass<<<nb, TILE, 0, st>>>(rows, n, 0, nullptr, B.lda_part);
    k_sum_blocks<<<1, 64, 0, st>>>(B.lda_part, nb, 2 * NF, B.lda_sum);
    CUDA_TRY(cudaGetLastError());
    double sums[2 * NF];
    CUDA_TRY(cudaMemcpyAsync(sums, B.lda_sum, sizeof sums, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    double mean[2 * NF];
    for (int c = 0; c < 2; c++)
        for (int j = 0; j < NF; j++) mean[c * NF + j] = sums[c * NF + j] / (double)cnt[c];
    CUDA_TRY(cudaMemcpyAsync(B.mean, mean, sizeof mean, cudaMemcpyHostToDevice, st));
    k_lda_pass<<<nb, TILE, 0, st>>>(rows, n, 1, B.mean, B.lda_part);
    k_sum_blocks<<<2, 256, 0, st>>>(B.lda_part, nb, 2 * 210, B.lda_sum);
    CUDA_TRY(cudaGetLastError());
    double scat[2 * 210];
    CUDA_TRY(cudaMemcpyAsync(scat, B.lda_sum, sizeof scat, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    // scatter_within = 0 + S_decoy / n_decoy + S_target / n_target; mu_diff = mu_target - mu_decoy
    std::vector<double> sw((size_t)d * d, 0.0), mu(d);
    int e = 0;
    for (int j = 0; j < NF; j++)
        for (int k = j; k < NF; k++, e++) {
            if (j >= (int)d || k >= (int)d) continue;
            double v = 0.0;
            for (int c = 0; c < 2; c++) v += scat[c * 210 + e] / (double)cnt[c];
            sw[(size_t)j * d + k] = v;
            sw[(size_t)k * d + j] = v;
        }
    for (uint32_t j = 0; j < d; j++) mu[j] = mean[NF + j] - mean[j];
    std::vector<double> w;
    if (!Gauss::solve(sw, mu, (int)d, w)) return 0;
    for (double v : w)
        if (!std::isfinite(v)) return 0;   // score_psms: non-finite coefficients count as a failed fit (linear_discriminant.rs:196-208)
    coef = w;
    return 1;
}

void init_pairs() {
    static std::once_flag once;
    static uint8_t pj[210], pk[210];
    std::call_once(once, [] {
        int e = 0;
        for (int j = 0; j < NF; j++)
            for (int k = j; k < NF; k++, e++) { pj[e] = (uint8_t)j; pk[e] = (uint8_t)k; }
    });
    cudaMemcpyToSymbol(c_pair_j, pj, sizeof pj);
    cudaMemcpyToSymbol(c_pair_k, pk, sizeof pk);
}

int fdr_device(int device, FdrDevice** out) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(SAGE_B200_ECUDA, "no CUDA device available: sage_b200 has no CPU fallback");
    if (device < 0 || device >= ndev || device >= 64) return fail(SAGE_B200_EINVAL, "device out of range");
    CUDA_TRY(cudaSetDevice(device));
    FdrDevice& D = g_fdr[device];
    static std::mutex init_mu;
    std::lock_guard<std::mutex> g(init_mu);
    if (!D.init) {
        CUDA_TRY(cudaStreamCreateWithFlags(&D.st, cudaStreamNonBlocking));
        for (auto& e : D.ev) CUDA_TRY(cudaEventCreate(&e));
        init_pairs();
        CUDA_TRY(cudaGetLastError());
        D.init = true;
    }
    *out = &D;
    return 0;
}

// Competition::assign_q_value (fdr.rs:59-120) for one key table; q per (key, side) then per feature
int picked(cudaStream_t st, const FdrBufs& B, uint64_t n, const uint32_t* key_of, uint64_t nk, int protein, size_t temp_bytes, void* temp) {
    const unsigned g = grid_for(nk);
    k_comp_init<<<g, 256, 0, st>>>(nk, B.fwd, B.rev, B.kflags);
    k_comp_max<<<grid_for(n), 256, 0, st>>>(B.f, B.disc32, n, key_of, B.fwd, B.rev, B.kflags);
    k_comp_counts<<<g, 256, 0, st>>>(B.kflags, nk, B.nrows, B.present);
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(temp, temp_bytes, B.nrows, B.row_pos, (int64_t)nk + 1, st));
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(temp, temp_bytes, B.present, B.key_pos, (int64_t)nk + 1, st));
    uint32_t tot[2];
    CUDA_TRY(cudaMemcpyAsync(&tot[0], B.row_pos + nk, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(&tot[1], B.key_pos + nk, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    const uint64_t nr = tot[0], nkp = tot[1];
    if (nr == 0) return 0;
    k_comp_emit<<<g, 256, 0, st>>>(B.kflags, B.fwd, B.rev, nk, B.row_pos, B.key_pos, B.kx, B.kdec, B.key, B.idx);
    int rc = kde_build(st, B.kx, B.kdec, nkp, 1000, true, 1.0, B.kde + 2, B.mom, B.kde_part, B.disc_bins);
    if (rc) return rc;
    // descending by score; rows were emitted key-major, target first, and the radix sort is stable
    CUDA_TRY(cub::DeviceRadixSort::SortPairsDescending(temp, temp_bytes, B.key, B.key_out, B.idx, B.order + 0, (int64_t)nr, 0, 32, st));
    uint32_t* sid = B.order;   // reused: the spectrum order has been copied out already
    const uint64_t nch = (nr + PICK_CHUNK - 1) / PICK_CHUNK;
    k_pick_chunk<<<grid_for(nch), 256, 0, st>>>(B.key_out, sid, nr, B.disc_bins, B.kde + 2, B.pep, B.csum, B.ctgt);
    k_pick_chunk_scan<<<1, 1024, 0, st>>>(B.csum, B.ctgt, nch);
    k_pick_q<<<grid_for(nch), 256, 0, st>>>(sid, B.pep, nr, B.csum, B.ctgt, B.qa);
    CUDA_TRY(cub::DeviceScan::InclusiveScan(temp, temp_bytes, B.qa, B.qb, MinF32(), (int64_t)nr, st));
    k_pick_final<<<grid_for(nr), 256, 0, st>>>(B.qb, sid, nr, B.qside, B.counters + 2 + protein);
    k_pick_write<<<grid_for(n), 256, 0, st>>>(B.f, n, key_of, B.qside, protein, B.out);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

size_t cub_temp_bytes(uint64_t n) {
    size_t a = 0, b = 0, c = 0, d = 0;
    cub::DeviceRadixSort::SortPairsDescending((void*)nullptr, a, (uint32_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr,
                                              (int64_t)n, 0, 32);
    cub::DeviceScan::InclusiveSum((void*)nullptr, b, (uint32_t*)nullptr, (uint32_t*)nullptr, (int64_t)n);
    cub::DeviceScan::InclusiveScan((void*)nullptr, c, (float*)nullptr, (float*)nullptr, MinF32(), (int64_t)n);
    cub::DeviceScan::ExclusiveSum((void*)nullptr, d, (uint32_t*)nullptr, (uint32_t*)nullptr, (int64_t)n);
    return std::max(std::max(a, b), std::max(c, d));
}

}  // namespace

extern "C" int sage_b200_assign_fdr(int device, const sage_b200_feature* features, uint64_t n, const sage_b200_fdr_params* P, sage_b200_fdr_row* out,
                                    uint32_t* order, sage_b200_fdr_summary* summary) {
    const auto t0 = std::chrono::steady_clock::now();
    if (!P) return fail(SAGE_B200_EINVAL, "assign_fdr: null params");
    if (P->precursor_tol.kind != SAGE_B200_TOL_PPM && P->precursor_tol.kind != SAGE_B200_TOL_DA)
        return fail(SAGE_B200_EINVAL, "assign_fdr: precursor tolerance must be Ppm or Da (Pct is never used on m/z, linear_discriminant.rs:142)");
    if (n >= (1ull << 32)) return fail(SAGE_B200_ELIMIT, "assign_fdr: %llu features; at most 2^32 - 1 per call", (unsigned long long)n);
    if ((P->peptide_key || P->protein_key) && P->n_peptides == 0) return fail(SAGE_B200_EINVAL, "assign_fdr: keys given without n_peptides");
    if ((P->peptide_key && P->n_peptide_keys > (1ull << 31)) || (P->protein_key && P->n_protein_keys > (1ull << 31)))
        return fail(SAGE_B200_ELIMIT, "assign_fdr: at most 2^31 competition keys");
    if (P->n_peptides > 0xFFFFFFFFull) return fail(SAGE_B200_EINVAL, "assign_fdr: n_peptides must fit 32 bits (PeptideIx is u32)");
    sage_b200_fdr_summary S{};
    for (double& c : S.coef) c = NAN;
    if (n == 0) {
        if (summary) { S.ms_wall = 0.0f; *summary = S; }
        return 0;
    }
    if (!features || !out) return fail(SAGE_B200_EINVAL, "assign_fdr: null argument");
    FdrDevice* Dp = nullptr;
    int rc = fdr_device(device, &Dp);
    if (rc) return rc;
    FdrDevice& D = *Dp;
    std::lock_guard<std::mutex> lk(D.mu);
    cudaStream_t st = D.st;
    const bool is_da = P->precursor_tol.kind == SAGE_B200_TOL_DA;
    // linear_discriminant.rs:146-150 (f32 arithmetic on the tolerance bounds)
    const float span = std::max(P->precursor_tol.hi - P->precursor_tol.lo, is_da ? 1000.0f : 100.0f);
    const uint32_t mass_bins = (uint32_t)std::fabs(std::ceil(span));
    const double bw_mul = is_da ? 0.1 : 2.0;
    const uint64_t npk = P->peptide_key ? P->n_peptide_keys : 0, nprk = P->protein_key ? P->n_protein_keys : 0;
    const uint64_t nk = std::max<uint64_t>(std::max(npk, nprk), 1), npep = P->n_peptides;
    const uint32_t max_bins = std::max<uint32_t>(mass_bins, 1000);

    FdrBufs B{};
    auto layout = [&](Carve& c) {
        B.f = c.take<sage_b200_feature>(n);
        B.out = c.take<sage_b200_fdr_row>(n);
        B.mass_err = c.take<double>(n);
        B.disc64 = c.take<double>(n);
        B.mom = c.take<double>(RED_BLOCKS * 6);
        B.kde_part = c.take<double>(kde_partials(max_bins));
        B.mass_bins = c.take<double>(max_bins);
        B.disc_bins = c.take<double>(1000);
        B.lda_part = c.take<double>((uint64_t)LDA_MAX_BLOCKS * 2 * 210);
        B.lda_sum = c.take<double>(2 * 210);
        B.mean = c.take<double>(2 * NF);
        B.kx = c.take<double>(nk);
        B.csum = c.take<double>(2 * nk / PICK_CHUNK + 2);
        B.disc32 = c.take<float>(n);
        B.pe = c.take<float>(n);
        B.qa = c.take<float>(std::max<uint64_t>(n, 2 * nk));
        B.qb = c.take<float>(std::max<uint64_t>(n, 2 * nk));
        B.pep = c.take<float>(2 * nk);
        B.qside = c.take<float>(2 * nk);
        B.dec = c.take<uint8_t>(n);
        B.kdec = c.take<uint8_t>(nk);
        B.key = c.take<uint32_t>(std::max<uint64_t>(n, 2 * nk));
        B.key_out = c.take<uint32_t>(std::max<uint64_t>(n, 2 * nk));
        B.idx = c.take<uint32_t>(std::max<uint64_t>(n, 2 * nk));
        B.order = c.take<uint32_t>(std::max<uint64_t>(n, 2 * nk));
        B.flag = c.take<uint32_t>(n);
        B.ndec = c.take<uint32_t>(n);
        B.pk = c.take<uint32_t>(P->peptide_key ? npep : 0);
        B.prk = c.take<uint32_t>(P->protein_key ? npep : 0);
        B.fwd = c.take<uint32_t>(nk);
        B.rev = c.take<uint32_t>(nk);
        B.kflags = c.take<uint32_t>(nk);
        B.nrows = c.take<uint32_t>(nk + 1);
        B.present = c.take<uint32_t>(nk + 1);
        B.row_pos = c.take<uint32_t>(nk + 1);
        B.key_pos = c.take<uint32_t>(nk + 1);
        B.ctgt = c.take<uint32_t>(2 * nk / PICK_CHUNK + 2);
        B.art = c.take<float>(P->aligned_rt ? n : 0);
        B.drt = c.take<float>(P->delta_rt_model ? n : 0);
        B.dims = c.take<float>(P->delta_ims_model ? n : 0);
        B.kde = c.take<Kde>(3);
        B.counters = c.take<unsigned long long>(4);
        B.err = c.take<unsigned>(1);
    };
    Carve measure{nullptr};
    layout(measure);
    if ((rc = D.arena.reserve(measure.off))) return rc;
    const size_t temp_bytes = cub_temp_bytes(std::max<uint64_t>(n, 2 * nk + 1));
    if ((rc = D.temp.reserve(temp_bytes))) return rc;
    Carve carve{D.arena.as<char>()};
    layout(carve);

    CUDA_TRY(cudaEventRecord(D.ev[0], st));
    if (is_pinned(features)) CUDA_TRY(cudaMemcpyAsync(B.f, features, n * sizeof(sage_b200_feature), cudaMemcpyHostToDevice, st));
    else if ((rc = staged_h2d(B.f, features, n * sizeof(sage_b200_feature), D.stage, D.pool, st))) return rc;
    // the small inputs go straight from pageable memory
    if (P->peptide_key) CUDA_TRY(cudaMemcpyAsync(B.pk, P->peptide_key, 4 * npep, cudaMemcpyHostToDevice, st));
    if (P->protein_key) CUDA_TRY(cudaMemcpyAsync(B.prk, P->protein_key, 4 * npep, cudaMemcpyHostToDevice, st));
    if (P->aligned_rt) CUDA_TRY(cudaMemcpyAsync(B.art, P->aligned_rt, 4 * n, cudaMemcpyHostToDevice, st));
    if (P->delta_rt_model) CUDA_TRY(cudaMemcpyAsync(B.drt, P->delta_rt_model, 4 * n, cudaMemcpyHostToDevice, st));
    if (P->delta_ims_model) CUDA_TRY(cudaMemcpyAsync(B.dims, P->delta_ims_model, 4 * n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemsetAsync(B.counters, 0, 4 * sizeof(unsigned long long), st));
    CUDA_TRY(cudaMemsetAsync(B.err, 0, sizeof(unsigned), st));
    CUDA_TRY(cudaEventRecord(D.ev[1], st));

    // ---- validation, class counts, mass-error sample
    k_fdr_prep<<<grid_for(n), 256, 0, st>>>(B.f, n, is_da, npep, B.mass_err, B.dec, B.counters, B.err);
    // a table the caller did not give has a zero-length slot, which aliases the next buffer: pass null for it
    if (P->peptide_key || P->protein_key)
        k_check_keys<<<grid_for(npep), 256, 0, st>>>(P->peptide_key ? B.pk : nullptr, npk, P->protein_key ? B.prk : nullptr, nprk, npep, B.err);
    CUDA_TRY(cudaGetLastError());
    unsigned long long n_decoy = 0;
    unsigned err = 0;
    CUDA_TRY(cudaMemcpyAsync(&n_decoy, B.counters, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(&err, B.err, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (err & 1u) return fail(SAGE_B200_EINVAL, "assign_fdr: a Feature::peptide_idx is >= n_peptides (%llu)", (unsigned long long)npep);
    if (err & 2u) return fail(SAGE_B200_EINVAL, "assign_fdr: a peptide_key is >= n_peptide_keys (%llu)", (unsigned long long)npk);
    if (err & 4u) return fail(SAGE_B200_EINVAL, "assign_fdr: a protein_key is >= n_protein_keys (%llu)", (unsigned long long)nprk);

    // ---- score_psms: mass model, LDA fit, projection (linear_discriminant.rs:133-212)
    FeatureRows rows{B.f, B.mass_err, B.dec, P->aligned_rt ? B.art : nullptr, P->delta_rt_model ? B.drt : nullptr,
                     P->delta_ims_model ? B.dims : nullptr, B.mass_bins, B.kde + 0};
    std::vector<double> coef;
    int fitted = 0;
    if (n_decoy > 0 && n_decoy < n) {
        if ((rc = kde_build(st, B.mass_err, B.dec, n, mass_bins, false, bw_mul, B.kde + 0, B.mom, B.kde_part, B.mass_bins))) return rc;
        fitted = lda_train(st, rows, n, n_decoy, NF, B, coef);
        if (fitted < 0) return fitted;
    }
    if (fitted) {
        Coef c;
        for (int j = 0; j < NF; j++) { c.w[j] = coef[j]; S.coef[j] = coef[j]; }
        k_lda_project<<<grid_for(n), 256, 0, st>>>(rows, n, c, B.disc64, B.disc32);
        CUDA_TRY(cudaGetLastError());
    }
    CUDA_TRY(cudaEventRecord(D.ev[2], st));
    if (fitted) {
        if ((rc = kde_build(st, B.disc64, B.dec, n, 1000, true, 1.0, B.kde + 1, B.mom, B.kde_part, B.disc_bins))) return rc;
        k_posterior_error<<<grid_for(n), 256, 0, st>>>(B.disc64, n, B.disc_bins, B.kde + 1, B.pe);
    } else {
        k_fallback<<<grid_for(n), 256, 0, st>>>(B.f, n, B.disc32, B.pe);
    }
    k_write_scores<<<grid_for(n), 256, 0, st>>>(B.disc32, B.pe, n, B.out);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(D.ev[3], st));

    // ---- sort + spectrum_q_value (runner.rs:289-290, qvalue.rs:8-36)
    void* temp = D.temp.p;
    size_t tb = D.temp.cap;
    k_sort_keys<<<grid_for(n), 256, 0, st>>>(B.disc32, n, B.key, B.idx);
    CUDA_TRY(cub::DeviceRadixSort::SortPairsDescending(temp, tb, B.key, B.key_out, B.idx, B.order, (int64_t)n, 0, 32, st));
    k_rank_decoy<<<grid_for(n), 256, 0, st>>>(B.order, B.dec, n, B.flag);
    CUDA_TRY(cub::DeviceScan::InclusiveSum(temp, tb, B.flag, B.ndec, (int64_t)n, st));
    k_spectrum_q<<<grid_for(n), 256, 0, st>>>(B.ndec, n, B.qa);
    CUDA_TRY(cub::DeviceScan::InclusiveScan(temp, tb, B.qa, B.qb, MinF32(), (int64_t)n, st));
    k_spectrum_q_final<<<grid_for(n), 256, 0, st>>>(B.qb, B.order, n, B.out, B.counters + 1);
    CUDA_TRY(cudaGetLastError());
    if (order) CUDA_TRY(cudaMemcpyAsync(order, B.order, 4 * n, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaEventRecord(D.ev[4], st));

    // ---- picked_peptide, picked_protein (fdr.rs:123-190)
    if (P->peptide_key && (rc = picked(st, B, n, B.pk, npk, 0, tb, temp))) return rc;
    if (P->protein_key && (rc = picked(st, B, n, B.prk, nprk, 1, tb, temp))) return rc;
    CUDA_TRY(cudaEventRecord(D.ev[5], st));

    unsigned long long cnt[4];
    CUDA_TRY(cudaMemcpyAsync(out, B.out, n * sizeof(sage_b200_fdr_row), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(cnt, B.counters, sizeof cnt, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaEventRecord(D.ev[6], st));
    CUDA_TRY(cudaStreamSynchronize(st));
    S.spectrum_passing = cnt[1];
    S.peptide_passing = cnt[2];
    S.protein_passing = cnt[3];
    S.lda_fitted = (uint32_t)fitted;
    float* ms[6] = {&S.ms_h2d, &S.ms_lda, &S.ms_pep, &S.ms_spectrum_q, &S.ms_picked, &S.ms_d2h};
    for (int p = 0; p < 6; p++) CUDA_TRY(cudaEventElapsedTime(ms[p], D.ev[p], D.ev[p + 1]));
    S.ms_wall = (float)std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (summary) *summary = S;
    return 0;
}

extern "C" int sage_b200_lda_fit(int device, const double* rows, uint64_t n, uint32_t d, const uint8_t* decoy, double* coef) {
    if (!coef || d == 0 || d > NF) return fail(SAGE_B200_EINVAL, "lda_fit: need 1 <= d <= 20 and a coef buffer");
    for (uint32_t j = 0; j < d; j++) coef[j] = NAN;
    if (n >= (1ull << 32)) return fail(SAGE_B200_ELIMIT, "lda_fit: at most 2^32 - 1 rows");
    if (n == 0) return 1;
    if (!rows || !decoy) return fail(SAGE_B200_EINVAL, "lda_fit: null argument");
    FdrDevice* Dp = nullptr;
    int rc = fdr_device(device, &Dp);
    if (rc) return rc;
    FdrDevice& D = *Dp;
    std::lock_guard<std::mutex> lk(D.mu);
    cudaStream_t st = D.st;
    FdrBufs B{};
    auto layout = [&](Carve& c) {
        B.rows = c.take<double>(n * d);
        B.dec = c.take<uint8_t>(n);
        B.lda_part = c.take<double>((uint64_t)LDA_MAX_BLOCKS * 2 * 210);
        B.lda_sum = c.take<double>(2 * 210);
        B.mean = c.take<double>(2 * NF);
    };
    Carve measure{nullptr};
    layout(measure);
    if ((rc = D.arena.reserve(measure.off))) return rc;
    Carve carve{D.arena.as<char>()};
    layout(carve);
    CUDA_TRY(cudaMemcpyAsync(B.rows, rows, 8 * n * d, cudaMemcpyHostToDevice, st));
    uint64_t n_decoy = 0;
    std::vector<uint8_t> dec(n);
    for (uint64_t i = 0; i < n; i++) { dec[i] = decoy[i] != 0; n_decoy += dec[i]; }
    CUDA_TRY(cudaMemcpyAsync(B.dec, dec.data(), n, cudaMemcpyHostToDevice, st));
    MatrixRows mr{B.rows, B.dec, d, nullptr};
    std::vector<double> w;
    const int fitted = lda_train(st, mr, n, n_decoy, d, B, w);
    if (fitted < 0) return fitted;
    CUDA_TRY(cudaStreamSynchronize(st));
    if (!fitted) return 1;
    for (uint32_t j = 0; j < d; j++) coef[j] = w[j];
    return 0;
}
