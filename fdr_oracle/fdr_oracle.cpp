// fdr_oracle.cpp — CPU restatement of sage's rescoring and FDR steps (reference @0639176), the authority the device path is tested against.
//
//   score_psms               crates/sage/src/ml/linear_discriminant.rs:133-231 (train :63-124, score :127-130)
//   Gauss::solve             crates/sage/src/ml/gauss.rs:26-165
//   Kde / Builder / Estimator crates/sage/src/ml/kde.rs:14-169, mean / std ml/mod.rs:24-32
//   spectrum_fdr             crates/sage-cli/src/runner.rs:280-291, spectrum_q_value ml/qvalue.rs:8-36
//   picked_peptide / protein crates/sage/src/fdr.rs:16-190 (Competition::assign_q_value :59-120)
//
// Test infrastructure only. Sums are sequential, as in the reference. Two things the reference leaves open are fixed here the way the device
// library fixes them: the order among equal discriminant scores (par_sort_unstable_by) is ascending input index, the competition rows,
// which the reference collects from a hash map, start in key order (target before decoy) before the stable sort by score, and the per-key
// maximum of +0 and -0 is +0 (max_total).
// fo_set_block(B > 0) switches every f64 sum to blocks of B terms (a second summation order, used to measure how much the results move
// under reordering; the reference's own KDE sums are rayon folds whose order changes from run to run).
#include <omp.h>

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <numeric>
#include <vector>

#include "../include/sage_b200.h"

namespace {

uint64_t g_block = 0;

struct Sum {
    double total = 0.0, blk = 0.0;
    uint64_t k = 0;
    void add(double x) {
        if (!g_block) { total += x; return; }
        blk += x;
        if (++k == g_block) { total += blk; blk = 0.0; k = 0; }
    }
    double get() const { return g_block ? total + blk : total; }
};

uint32_t total_key(float x) {
    uint32_t u;
    memcpy(&u, &x, 4);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// ---------------------------------------------------------------------------------------------------------------- ml/mod.rs, kde.rs
double mean_of(const std::vector<double>& v) {
    Sum s;
    for (double x : v) s.add(x);
    return s.get() / (double)v.size();
}
double std_of(const std::vector<double>& v) {
    const double m = mean_of(v);
    Sum s;
    for (double x : v) s.add((x - m) * (x - m));
    return std::sqrt(s.get() / (double)v.size());
}

struct Kde {
    const std::vector<double>* sample;
    double bandwidth, constant;
    Kde(const std::vector<double>& s, double bw_mul) : sample(&s) {
        const double sigma = std_of(s);
        bandwidth = sigma * std::pow(4.0 / 3.0 / (double)s.size(), 1.0 / 5.0) * bw_mul;
        constant = std::sqrt(2.0 * M_PI) * bandwidth * (double)s.size();
    }
    double pdf(double x) const {
        Sum s;
        for (double xi : *sample) {
            const double u = (x - xi) / bandwidth;
            s.add(std::exp(-0.5 * (u * u)));
        }
        return s.get() / constant;
    }
};

struct Estimator {
    std::vector<double> bins;
    double min_score = 0, score_step = 0;
    double posterior_error(double score) const {
        const double f = std::floor((score - min_score) / score_step);
        uint64_t lo;
        if (!(f > 0.0)) lo = 0;                               // `as usize`: NaN and negatives saturate to 0
        else if (f >= 18446744073709551616.0) lo = ~0ull;
        else lo = (uint64_t)f;
        const uint64_t last = bins.empty() ? 0 : bins.size() - 1;
        lo = std::min(last, lo);
        const uint64_t hi = std::min(last, lo + 1);
        const double lower = bins[lo], upper = bins[hi];
        const double bin_lo_score = (double)lo * score_step + min_score;
        const double linear = (score - bin_lo_score) / score_step;
        return lower + (upper - lower) * linear;
    }
};

Estimator kde_build(const std::vector<double>& scores, const std::vector<uint8_t>& decoys, size_t nbins, bool monotonic, double bw_mul) {
    std::vector<double> d, t;
    for (size_t i = 0; i < scores.size(); i++) (decoys[i] ? d : t).push_back(scores[i]);
    const double pi = (double)d.size() / (double)scores.size();
    const Kde kd(d, bw_mul), kt(t, bw_mul);
    double mn = DBL_MAX, mx = -DBL_MAX;
    for (double s : scores) { mn = std::fmin(mn, s); mx = std::fmax(mx, s); }
    Estimator e;
    e.min_score = mn;
    e.score_step = (mx - mn) / (double)(nbins - 1);
    e.bins.resize(nbins);
#pragma omp parallel for schedule(dynamic, 1)
    for (int64_t b = 0; b < (int64_t)nbins; b++) {
        const double score = (double)b * e.score_step + mn;
        const double decoy = kd.pdf(score) * pi;
        const double target = kt.pdf(score) * (1.0 - pi);
        e.bins[b] = decoy / (target + decoy);
    }
    if (monotonic) {
        double acc = e.bins.back();
        for (size_t i = nbins; i-- > 0;) { acc = std::fmax(acc, e.bins[i]); e.bins[i] = acc; }
    }
    return e;
}

// ---------------------------------------------------------------------------------------------------------------- gauss.rs
bool gauss_solve(const std::vector<double>& left, const std::vector<double>& right, int n, std::vector<double>& out) {
    for (double eps = 1e-8; eps <= 1.0; eps *= 10.0) {
        std::vector<double> L = left, R = right;
        auto l = [&](int i, int j) -> double& { return L[(size_t)i * n + j]; };
        for (int i = 0; i < n; i++) l(i, i) += eps;
        int h = 0, k = 0;
        while (h < n && k < n) {
            int imax = 0;
            double vmax = -DBL_MAX;
            for (int i = h; i < n; i++)
                if (l(i, k) >= vmax) { imax = i; vmax = l(i, k); }
            if (l(imax, k) == 0.0) { k++; continue; }
            if (h != imax) {
                for (int c = 0; c < n; c++) std::swap(l(h, c), l(imax, c));
                std::swap(R[h], R[imax]);
            }
            for (int i = h + 1; i < n; i++) {
                const double factor = l(i, k) / l(h, k);
                l(i, k) = 0.0;
                for (int j = k + 1; j < n; j++) l(i, j) -= l(h, j) * factor;
                R[i] -= R[h] * factor;
            }
            h++;
            k++;
        }
        for (int i = n - 1; i >= 0; i--)   // reduce
            for (int j = 0; j < n; j++) {
                const double x = l(i, j);
                if (x == 0.0) continue;
                for (int c = j; c < n; c++) l(i, c) /= x;
                R[i] /= x;
                break;
            }
        for (int i = n - 1; i >= 0; i--)   // backfill
            for (int j = 0; j < n; j++) {
                if (l(i, j) == 0.0) continue;
                for (int r = 0; r < i; r++) {
                    const double factor = l(r, j) / l(i, j);
                    for (int c = 0; c < n; c++) l(r, c) -= l(i, c) * factor;
                    R[r] -= R[i] * factor;
                }
                break;
            }
        bool ok = true;   // left_solved
        for (int i = 0; i < n && ok; i++)
            for (int j = 0; j < n; j++) {
                const double x = l(i, j);
                if (i == j ? (x != 1.0 && x != 0.0) : x > 1e-8) { ok = false; break; }
            }
        if (ok) { out = R; return true; }
    }
    return false;
}

// ---------------------------------------------------------------------------------------------------------------- linear_discriminant.rs
template <class RowFn>
bool lda_train(uint64_t n, int d, const std::vector<uint8_t>& decoy, RowFn row, std::vector<double>& coef) {
    std::vector<Sum> class_sum(2 * d);
    uint64_t count[2] = {0, 0};
    std::vector<double> r(d);
    for (uint64_t i = 0; i < n; i++) {
        row(i, r.data());
        const int c = decoy[i] ? 0 : 1;
        for (int j = 0; j < d; j++) class_sum[c * d + j].add(r[j]);
        count[c]++;
    }
    if (count[0] == 0 || count[1] == 0) return false;
    std::vector<double> mean(2 * d);
    for (int c = 0; c < 2; c++)
        for (int j = 0; j < d; j++) mean[c * d + j] = class_sum[c * d + j].get() / (double)count[c];
    std::vector<Sum> scatter(2 * d * d);
    std::vector<double> centered(d);
    for (uint64_t i = 0; i < n; i++) {
        row(i, r.data());
        const int c = decoy[i] ? 0 : 1;
        for (int j = 0; j < d; j++) centered[j] = r[j] - mean[c * d + j];
        for (int j = 0; j < d; j++)
            for (int k = 0; k < d; k++) scatter[((size_t)c * d + j) * d + k].add(centered[j] * centered[k]);
    }
    std::vector<double> sw((size_t)d * d, 0.0), mu(d);
    for (int c = 0; c < 2; c++)
        for (int e = 0; e < d * d; e++) sw[e] += scatter[(size_t)c * d * d + e].get() / (double)count[c];
    for (int j = 0; j < d; j++) mu[j] = mean[d + j] - mean[j];
    return gauss_solve(sw, mu, d, coef);
}

// score_psms: fills disc64 / posterior_error; false when the fit fails (runner.rs then uses the heuristic score)
bool score_psms(const sage_b200_feature* f, uint64_t n, const sage_b200_fdr_params* P, const std::vector<uint8_t>& decoys, std::vector<double>& disc,
                std::vector<float>& pe, std::vector<double>& coef) {
    const bool is_da = P->precursor_tol.kind == SAGE_B200_TOL_DA;
    auto mass_error = [&](uint64_t i) { return is_da ? (double)(f[i].expmass - f[i].calcmass) : (double)f[i].delta_mass; };
    const float span = std::max(P->precursor_tol.hi - P->precursor_tol.lo, is_da ? 1000.0f : 100.0f);
    std::vector<double> delta_mass(n);
    for (uint64_t i = 0; i < n; i++) delta_mass[i] = mass_error(i);
    const Estimator mass_model = kde_build(delta_mass, decoys, (size_t)std::fabs(std::ceil(span)), false, is_da ? 0.1 : 2.0);
    auto clamp_sqrt = [](double v) { v = v < 0.001 ? 0.001 : (v > 0.999 ? 0.999 : v); return std::sqrt(v); };
    auto features = [&](uint64_t i, double* r) {
        const sage_b200_feature& x = f[i];
        double poisson = std::log1p(-x.poisson);
        if (!std::isfinite(poisson)) poisson = 3.5;
        r[0] = (double)x.rank;
        r[1] = (double)x.charge;
        r[2] = std::log1p(x.hyperscore);
        r[3] = std::log1p(x.delta_next);
        r[4] = std::log1p(x.delta_best);
        r[5] = mass_model.posterior_error(mass_error(i));
        r[6] = (double)x.isotope_error;
        r[7] = (double)x.average_ppm;
        r[8] = poisson;
        r[9] = std::log1p((double)x.matched_intensity_pct);
        r[10] = (double)x.matched_peaks;
        r[11] = std::log1p((double)x.longest_b);
        r[12] = std::log1p((double)x.longest_y);
        r[13] = (double)x.longest_y / (double)x.peptide_len;
        r[14] = std::log1p((double)x.peptide_len);
        r[15] = (double)x.missed_cleavages;
        r[16] = (double)(P->aligned_rt ? P->aligned_rt[i] : x.rt);
        r[17] = (double)x.ims;
        r[18] = clamp_sqrt((double)(P->delta_rt_model ? P->delta_rt_model[i] : 0.999f));
        r[19] = clamp_sqrt((double)(P->delta_ims_model ? P->delta_ims_model[i] : 0.999f));
    };
    if (!lda_train(n, 20, decoys, features, coef)) return false;
    for (double c : coef)
        if (!std::isfinite(c)) return false;
    disc.resize(n);
#pragma omp parallel for
    for (int64_t i = 0; i < (int64_t)n; i++) {
        double r[20];
        features((uint64_t)i, r);
        double s = 0.0;
        for (int j = 0; j < 20; j++) s += coef[j] * r[j];
        disc[i] = s;
    }
    const Estimator kde = kde_build(disc, decoys, 1000, true, 1.0);
    pe.resize(n);
    for (uint64_t i = 0; i < n; i++) {
        float v = (float)std::log10(kde.posterior_error(disc[i]));
        if (std::isinf(v)) v = -324.0f;
        pe[i] = v;
    }
    return true;
}

// runner.rs:289 with ties by input index, then qvalue.rs:8-36 over the sorted labels
uint64_t sort_spectrum_q(const float* disc, const uint8_t* decoy, uint64_t n, uint32_t* order, float* q_rank) {
    std::iota(order, order + n, 0u);
    std::stable_sort(order, order + n, [&](uint32_t a, uint32_t b) { return total_key(disc[a]) > total_key(disc[b]); });
    uint64_t dcount = 1, tcount = 0;
    for (uint64_t r = 0; r < n; r++) {
        if (decoy[order[r]]) dcount++; else tcount++;
        q_rank[r] = (float)dcount / (float)tcount;
    }
    float q_min = 1.0f;
    uint64_t passing = 0;
    for (uint64_t r = n; r-- > 0;) {
        q_min = std::fmin(q_min, q_rank[r]);
        q_rank[r] = q_min;
        if (q_min <= 0.01f) passing++;
    }
    return passing;
}

// f32::max with NaN skipped; equal values of opposite sign (±0) are ordered as f32::total_cmp orders them, +0 above -0, so the result does
// not depend on the order the features come in (the reference leaves that choice open; the device makes the same one)
float max_total(float a, float b) {
    if (std::isnan(b)) return a;
    if (std::isnan(a)) return b;
    return total_key(b) > total_key(a) ? b : a;
}

// fdr.rs:16-190 with integer keys: q per feature written to q (features without a key are left alone)
uint64_t competition(const float* disc, const uint8_t* decoy, const uint32_t* key, uint64_t n, uint64_t n_keys, float* q) {
    const float lowest = -FLT_MAX;
    std::vector<float> fwd(n_keys, lowest), rev(n_keys, lowest);
    std::vector<uint8_t> has(n_keys, 0);
    for (uint64_t i = 0; i < n; i++) {
        const uint32_t k = key[i];
        if (k == 0xFFFFFFFFu) continue;
        if (decoy[i]) { rev[k] = max_total(rev[k], disc[i]); has[k] |= 2; }
        else { fwd[k] = max_total(fwd[k], disc[i]); has[k] |= 1; }
    }
    std::vector<double> scores;
    std::vector<uint8_t> is_decoy;
    struct Row { uint64_t key; bool decoy; float score; float q; };
    std::vector<Row> rows;
    for (uint64_t k = 0; k < n_keys; k++) {
        if (!has[k]) continue;
        scores.push_back((double)max_total(fwd[k], rev[k]));
        is_decoy.push_back(rev[k] >= fwd[k]);
        if (has[k] & 1) rows.push_back({k, false, fwd[k], 1.0f});
        if (has[k] & 2) rows.push_back({k, true, rev[k], 1.0f});
    }
    if (rows.empty()) return 0;
    const Estimator est = kde_build(scores, is_decoy, 1000, true, 1.0);
    std::stable_sort(rows.begin(), rows.end(), [](const Row& a, const Row& b) { return total_key(a.score) > total_key(b.score); });
    float dsum = 1.0f, tsum = 0.0f;
    for (Row& r : rows) {
        const float pep = (float)est.posterior_error((double)r.score);
        dsum += pep;
        if (!r.decoy) tsum += 1.0f;
        r.q = dsum / tsum;
    }
    float q_min = 1.0f;
    uint64_t passing = 0;
    for (size_t i = rows.size(); i-- > 0;) {
        q_min = std::fmin(q_min, rows[i].q);
        rows[i].q = q_min;
        if (q_min <= 0.01f && !rows[i].decoy) passing++;
    }
    std::vector<float> qside(2 * n_keys, 1.0f);
    for (const Row& r : rows) qside[2 * r.key + r.decoy] = r.q;
    for (uint64_t i = 0; i < n; i++)
        if (key[i] != 0xFFFFFFFFu) q[i] = qside[2 * (uint64_t)key[i] + decoy[i]];
    return passing;
}

}  // namespace

extern "C" {

void fo_set_block(uint64_t block) { g_block = block; }
void fo_set_threads(int n) { if (n > 0) omp_set_num_threads(n); }

// Gauss::solve on a d x d system (row-major) with one right-hand column; 1 when solved
int fo_gauss_solve(const double* left, const double* right, int d, double* out) {
    std::vector<double> L(left, left + (size_t)d * d), R(right, right + d), x;
    if (!gauss_solve(L, R, d, x)) return 0;
    std::copy(x.begin(), x.end(), out);
    return 1;
}

// LinearDiscriminantAnalysis::train on rows [n x d]; 1 when fitted (coef written)
int fo_lda_fit(const double* rows, uint64_t n, int d, const uint8_t* decoy, double* coef) {
    std::vector<uint8_t> dec(decoy, decoy + n);
    std::vector<double> c;
    if (!lda_train(n, d, dec, [&](uint64_t i, double* r) { for (int j = 0; j < d; j++) r[j] = rows[i * d + j]; }, c)) return 0;
    std::copy(c.begin(), c.end(), coef);
    return 1;
}

// Builder::build: out_bins[nbins], meta = {min_score, score_step}
void fo_kde(const double* scores, const uint8_t* decoy, uint64_t n, uint64_t nbins, int monotonic, double bw_mul, double* out_bins, double* meta) {
    std::vector<double> s(scores, scores + n);
    std::vector<uint8_t> d(decoy, decoy + n);
    const Estimator e = kde_build(s, d, nbins, monotonic != 0, bw_mul);
    std::copy(e.bins.begin(), e.bins.end(), out_bins);
    meta[0] = e.min_score;
    meta[1] = e.score_step;
}

double fo_posterior_error(const double* bins, uint64_t nbins, double min_score, double score_step, double score) {
    Estimator e;
    e.bins.assign(bins, bins + nbins);
    e.min_score = min_score;
    e.score_step = score_step;
    return e.posterior_error(score);
}

uint64_t fo_sort_spectrum_q(const float* disc, const uint8_t* decoy, uint64_t n, uint32_t* order, float* q_rank) {
    return sort_spectrum_q(disc, decoy, n, order, q_rank);
}

uint64_t fo_competition(const float* disc, const uint8_t* decoy, const uint32_t* key, uint64_t n, uint64_t n_keys, float* q) {
    return competition(disc, decoy, key, n, n_keys, q);
}

// The three steps end to end, the same contract as sage_b200_assign_fdr (validation included).
int fo_assign_fdr(const sage_b200_feature* f, uint64_t n, const sage_b200_fdr_params* P, sage_b200_fdr_row* out, uint32_t* order, sage_b200_fdr_summary* S) {
    if (P->precursor_tol.kind != SAGE_B200_TOL_PPM && P->precursor_tol.kind != SAGE_B200_TOL_DA) return SAGE_B200_EINVAL;
    if (n >= (1ull << 32)) return SAGE_B200_ELIMIT;
    if ((P->peptide_key || P->protein_key) && P->n_peptides == 0) return SAGE_B200_EINVAL;
    *S = sage_b200_fdr_summary{};
    for (double& c : S->coef) c = NAN;
    if (n == 0) return 0;
    for (uint64_t i = 0; i < n; i++)
        if (P->n_peptides && f[i].peptide_idx >= P->n_peptides) return SAGE_B200_EINVAL;
    for (uint64_t p = 0; p < ((P->peptide_key || P->protein_key) ? P->n_peptides : 0); p++) {
        if (P->peptide_key && P->peptide_key[p] >= P->n_peptide_keys) return SAGE_B200_EINVAL;
        if (P->protein_key && P->protein_key[p] != 0xFFFFFFFFu && P->protein_key[p] >= P->n_protein_keys) return SAGE_B200_EINVAL;
    }
    std::vector<uint8_t> decoy(n);
    for (uint64_t i = 0; i < n; i++) decoy[i] = f[i].label == -1;
    std::vector<double> disc64, coef;
    std::vector<float> pe, disc(n);
    const bool fitted = score_psms(f, n, P, decoy, disc64, pe, coef);
    for (uint64_t i = 0; i < n; i++) {
        if (fitted) {
            disc[i] = (float)disc64[i];
        } else {   // runner.rs:284-287
            disc[i] = std::log1p((float)(-f[i].poisson)) + f[i].longest_y_pct / 3.0f;
        }
        out[i] = {disc[i], fitted ? pe[i] : 1.0f, 1.0f, 1.0f, 1.0f};
    }
    S->lda_fitted = fitted;
    if (fitted)
        for (int j = 0; j < 20; j++) S->coef[j] = coef[j];
    std::vector<float> q_rank(n);
    S->spectrum_passing = sort_spectrum_q(disc.data(), decoy.data(), n, order, q_rank.data());
    for (uint64_t r = 0; r < n; r++) out[order[r]].spectrum_q = q_rank[r];
    std::vector<uint32_t> key(n);
    std::vector<float> q(n);
    for (int stage = 0; stage < 2; stage++) {
        const uint32_t* table = stage == 0 ? P->peptide_key : P->protein_key;
        if (!table) continue;
        for (uint64_t i = 0; i < n; i++) { key[i] = table[f[i].peptide_idx]; q[i] = 1.0f; }
        const uint64_t passing = competition(disc.data(), decoy.data(), key.data(), n, stage == 0 ? P->n_peptide_keys : P->n_protein_keys, q.data());
        for (uint64_t i = 0; i < n; i++) (stage == 0 ? out[i].peptide_q : out[i].protein_q) = q[i];
        (stage == 0 ? S->peptide_passing : S->protein_passing) = passing;
    }
    return 0;
}

}  // extern "C"
