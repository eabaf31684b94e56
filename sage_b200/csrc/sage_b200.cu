// sage_b200.cu — host runtime and C ABI (include/sage_b200.h) of the B200-native search-and-score library.
//
// Host side of the boundary, written in C++ because the reference (Rust) toolchain is absent in this image; it
// mirrors the reference's call structure: IndexedDatabase (database.rs:384-395) -> sage_b200_db, Scorer
// (scoring.rs:210-232) -> sage_b200_scorer, `par_iter().flat_map(|s| scorer.score(s))` (runner.rs:311-325) ->
// sage_b200_score_batch. No CPU fallback exists: every entry point fails loudly when CUDA is unavailable.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cuda_runtime.h>

#include <pthread.h>
#include <sched.h>

#include <algorithm>
#include <atomic>
#include <cctype>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <condition_variable>
#include <memory>
#include <mutex>
#include <thread>
#include <string>
#include <vector>

#include "../../include/sage_b200.h"
#include "kernels.cuh"

using namespace sb;

// ------------------------------------------------------------------------------------------------ errors
static thread_local std::string g_last_error;
static int fail(int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return code;
}
#define CUDA_TRY(expr)                                                                                         \
    do {                                                                                                       \
        cudaError_t _e = (expr);                                                                               \
        if (_e != cudaSuccess) return fail(SAGE_B200_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

// mass.rs:64-76
static const float kResidueMass[26] = {71.03711f, 0.0f,      103.00919f, 115.02694f, 129.04259f, 147.0684f, 57.02146f,  137.05891f, 113.08406f,
                                       0.0f,      128.09496f, 113.08406f, 131.0405f,  114.04293f, 237.14774f, 97.05276f, 128.05858f, 156.1011f,
                                       87.03203f, 101.04768f, 150.95363f, 99.06841f,  186.07932f, 0.0f,       163.06332f, 0.0f};

// ------------------------------------------------------------------------------------------- device buffers
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return 0;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) return fail(SAGE_B200_ECUDA, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
        cap = want;
        return 0;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <class T>
    T* as() const { return reinterpret_cast<T*>(p); }
};
struct PinBuf {
    void* p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return 0;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocPortable);
        if (e != cudaSuccess) return fail(SAGE_B200_ECUDA, "cudaHostAlloc(%zu) failed: %s", want, cudaGetErrorString(e));
        cap = want;
        return 0;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
};

// Host -> device copy of a PAGEABLE array (a Rust Vec<f32>, a numpy array) through a pinned staging buffer: a few pool threads copy 2 MB pieces
// into the staging buffer while the calling thread submits each piece's DMA as soon as it is staged, so the memcpy (one core moves ~10 GB/s,
// PCIe 5 x16 ~55 GB/s) overlaps the transfer instead of preceding it. The pool threads are persistent (one pool per pipeline lane, started by
// the first pageable chunk): creating 6 threads per array cost ~0.25 ms of a 6 ms call. Measured on cfg2 (ms per 50k-spectrum call, 2 MB pieces):
// 3 threads 6.5 | 6 -> 6.0 | 12 -> 7.2 | 16 x 1 MB 9.0 | 24 x 512 KB 9.5 (spawned per call; more copy threads only fight the DMA reads for the
// memory controllers).
struct StagePool {
    std::vector<std::thread> th;
    std::mutex mu;
    std::condition_variable cv;
    uint64_t gen = 0;
    bool quit = false;
    const char* src = nullptr;
    char* dst = nullptr;
    size_t bytes = 0, piece = 0, np = 0, done_cap = 0;
    std::atomic<size_t> next{0};
    std::atomic<int> busy{0};
    std::unique_ptr<std::atomic<unsigned char>[]> done;

    void worker() {
        uint64_t seen = 0;
        for (;;) {
            {
                std::unique_lock<std::mutex> lk(mu);
                cv.wait(lk, [&] { return quit || gen != seen; });
                if (quit) return;
                seen = gen;
            }
            for (;;) {
                const size_t i = next.fetch_add(1, std::memory_order_relaxed);
                if (i >= np) break;
                const size_t off = i * piece, len = std::min(piece, bytes - off);
                memcpy(dst + off, src + off, len);
                done[i].store(1, std::memory_order_release);
            }
            busy.fetch_sub(1, std::memory_order_release);
        }
    }
    // Copies src -> stage in pieces with the pool and submits piece i's DMA (stage -> device) as soon as pieces 0..i are staged.
    cudaError_t run(void* dev, const void* s, size_t n, void* stage, size_t piece_bytes, size_t nthreads, cudaStream_t st) {
        if (th.size() < nthreads) {
            const size_t have = th.size();
            for (size_t t = have; t < nthreads; t++) th.emplace_back([this] { worker(); });
        }
        const size_t pieces = (n + piece_bytes - 1) / piece_bytes;
        if (pieces > done_cap) { done.reset(new std::atomic<unsigned char>[pieces]); done_cap = pieces; }
        for (size_t i = 0; i < pieces; i++) done[i].store(0, std::memory_order_relaxed);
        {
            std::lock_guard<std::mutex> lk(mu);
            src = (const char*)s; dst = (char*)stage; bytes = n; piece = piece_bytes; np = pieces;
            next.store(0, std::memory_order_relaxed);
            busy.store((int)th.size(), std::memory_order_relaxed);
            gen++;
        }
        cv.notify_all();
        cudaError_t e = cudaSuccess;
        for (size_t i = 0; i < pieces; i++) {
            while (!done[i].load(std::memory_order_acquire)) std::this_thread::yield();
            const size_t off = i * piece_bytes, len = std::min(piece_bytes, n - off);
            if (e == cudaSuccess) e = cudaMemcpyAsync((char*)dev + off, (char*)stage + off, len, cudaMemcpyHostToDevice, st);
        }
        while (busy.load(std::memory_order_acquire) != 0) std::this_thread::yield();   // every worker has left the job: its fields may change
        return e;
    }
    ~StagePool() {
        {
            std::lock_guard<std::mutex> lk(mu);
            quit = true;
        }
        cv.notify_all();
        for (auto& t : th) t.join();
    }
};

static int staged_h2d(void* dst, const void* src, size_t bytes, PinBuf& stage, StagePool& pool, cudaStream_t st) {
    if (bytes == 0) return 0;
    int rc = stage.reserve(bytes);
    if (rc) return rc;
    static const size_t piece = []() { const char* e = getenv("SAGE_B200_STAGE_PIECE_KB"); return (size_t)std::max(64, e ? atoi(e) : 2048) << 10; }();
    static const size_t max_threads = []() { const char* e = getenv("SAGE_B200_STAGE_THREADS"); return (size_t)std::max(1, e ? atoi(e) : 6); }();
    const size_t np = (bytes + piece - 1) / piece;
    if (np <= 2) {   // small: a plain copy is cheaper than waking threads
        memcpy(stage.p, src, bytes);
        CUDA_TRY(cudaMemcpyAsync(dst, stage.p, bytes, cudaMemcpyHostToDevice, st));
        return 0;
    }
    const unsigned hw = std::max(2u, std::thread::hardware_concurrency());
    const size_t nthreads = std::min<size_t>(max_threads, (size_t)hw - 1);
    const cudaError_t e = pool.run(dst, src, bytes, stage.p, piece, nthreads, st);
    if (e != cudaSuccess) return fail(SAGE_B200_ECUDA, "staged host-to-device copy failed: %s", cudaGetErrorString(e));
    return 0;
}

static bool is_pinned(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

// sage_b200_assign_fdr / sage_b200_lda_fit (uses fail, DevBuf, staged_h2d above)
#include "fdr.cuh"

// ------------------------------------------------------------------------------------------------ db
struct BlockIndexSlot {
    WideIndexView v{};
    void *d_frag = nullptr, *d_blk = nullptr, *d_lut = nullptr;
    int failed = 0;
    uint64_t bytes = 0;
    std::vector<void*> retired;   // arrays of earlier builds: another scorer of the same db may still hold a view of them (freed with the db)
    uint64_t retired_bytes = 0;
    void release() {
        for (void** p : {&d_frag, &d_blk, &d_lut}) { if (*p) cudaFree(*p); *p = nullptr; }
        for (void* p : retired) cudaFree(p);
        retired.clear();
        retired_bytes = 0;
        v = WideIndexView{};
        bytes = 0;
    }
    // A rebuild with another block size keeps the old arrays alive: a chunk of another scorer, queued with the old view, may still run.
    void retire() {
        for (void** p : {&d_frag, &d_blk, &d_lut}) { if (*p) retired.push_back(*p); *p = nullptr; }
        retired_bytes += bytes;
        v = WideIndexView{};
        bytes = 0;
    }
};

struct sage_b200_db {
    int device = 0;
    DbView v{};
    void *d_page_grid = nullptr, *d_bucket_lut = nullptr, *d_pep_lut = nullptr;
    void *d_frag = nullptr, *d_bucket_min = nullptr, *d_pep_mono = nullptr, *d_ion_off = nullptr, *d_ions = nullptr, *d_pep_len = nullptr,
         *d_pep_flags = nullptr, *d_pep_missed = nullptr;
    uint64_t total_residues = 0, device_bytes = 0;
    int sm_count = 148;
    // secondary copies of the fragments in peptide-block-major order (WideIndexView), built lazily and guarded by wmu: `wide` (blocks = the
    // open-search count tile, built by the first scorer that meets a wide window) and `narrow` (small blocks, built by the first narrow chunk)
    mutable std::mutex wmu;
    mutable BlockIndexSlot wide, narrow;
};

static int dmalloc(sage_b200_db* db, void** p, size_t bytes) {
    if (bytes == 0) bytes = 16;
    CUDA_TRY(cudaMalloc(p, bytes));
    db->device_bytes += bytes;
    return 0;
}

static uint32_t ceil_log2_u64(uint64_t n) {
    uint32_t l = 0;
    while ((1ull << l) < n) l++;
    return l;
}

// Uploads the peptide table and builds the per-peptide ion tables. On return tmp_* hold device copies still needed by db_build.
static int db_upload_peptides(sage_b200_db* db, const sage_b200_peptides* P, const uint8_t* kinds, uint64_t n_kinds) {
    if (!P || (P->n_peptides && (!P->residue_offsets || !P->sequence || !P->modifications || !P->nterm || !P->monoisotopic || !P->decoy || !P->missed_cleavages)))
        return fail(SAGE_B200_EINVAL, "peptides: null array");
    if (n_kinds == 0 || n_kinds > MAX_KINDS) return fail(SAGE_B200_EINVAL, "ion_kinds: need 1..%d kinds", MAX_KINDS);
    if (P->n_peptides >= 0xFFFFFFFEull) return fail(SAGE_B200_ELIMIT, "too many peptides for u32 PeptideIx");
    const uint64_t n = P->n_peptides;
    db->v.n_pep = (uint32_t)n;
    db->v.n_kinds = (uint32_t)n_kinds;
    for (uint64_t k = 0; k < n_kinds; k++) {
        if (kinds[k] > 5) return fail(SAGE_B200_EINVAL, "ion kind %u out of range", kinds[k]);
        db->v.kinds[k] = kinds[k];
        if (kinds[k] <= 2) db->v.nterm_mask |= 1u << k;
    }
    const uint64_t nres = n ? P->residue_offsets[n] : 0;
    db->total_residues = nres;
    std::vector<uint8_t> len(n), flags(n);
    std::vector<uint32_t> ion_off(n + 1);
    uint64_t acc = 0;
    for (uint64_t i = 0; i < n; i++) {
        const uint64_t L = P->residue_offsets[i + 1] - P->residue_offsets[i];
        if (L == 0 || L > 255) return fail(SAGE_B200_ELIMIT, "peptide %llu has length %llu (supported 1..255)", (unsigned long long)i, (unsigned long long)L);
        len[i] = (uint8_t)L;
        flags[i] = P->decoy[i] ? 1 : 0;
        ion_off[i] = (uint32_t)acc;
        acc += n_kinds * (L - 1);
        if (acc > 0xFFFFFFFFull) return fail(SAGE_B200_ELIMIT, "ion table exceeds 2^32 entries");
    }
    ion_off[n] = (uint32_t)acc;
    int rc;
    if ((rc = dmalloc(db, &db->d_pep_mono, 4 * n))) return rc;
    if ((rc = dmalloc(db, &db->d_pep_len, n))) return rc;
    if ((rc = dmalloc(db, &db->d_pep_flags, n))) return rc;
    if ((rc = dmalloc(db, &db->d_pep_missed, n))) return rc;
    if ((rc = dmalloc(db, &db->d_ion_off, 4 * (n + 1)))) return rc;
    if ((rc = dmalloc(db, &db->d_ions, 4 * acc))) return rc;
    CUDA_TRY(cudaMemcpy(db->d_pep_mono, P->monoisotopic, 4 * n, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(db->d_pep_len, len.data(), n, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(db->d_pep_flags, flags.data(), n, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(db->d_pep_missed, P->missed_cleavages, n, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(db->d_ion_off, ion_off.data(), 4 * (n + 1), cudaMemcpyHostToDevice));
    // temporaries for ion generation
    void *t_off = nullptr, *t_seq = nullptr, *t_mods = nullptr, *t_nterm = nullptr, *t_res = nullptr;
    struct Temps {   // freed on every exit of this function
        void **a, **b, **c, **d, **e;
        ~Temps() { for (void** p : {a, b, c, d, e}) if (*p) cudaFree(*p); }
    } temps{&t_off, &t_seq, &t_mods, &t_nterm, &t_res};
    CUDA_TRY(cudaMalloc(&t_off, 4 * (n + 1) + 16));
    CUDA_TRY(cudaMalloc(&t_seq, nres + 16));
    CUDA_TRY(cudaMalloc(&t_mods, 4 * nres + 16));
    CUDA_TRY(cudaMalloc(&t_nterm, 4 * n + 16));
    CUDA_TRY(cudaMalloc(&t_res, sizeof kResidueMass));
    if (n) {
        CUDA_TRY(cudaMemcpy(t_off, P->residue_offsets, 4 * (n + 1), cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(t_seq, P->sequence, nres, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(t_mods, P->modifications, 4 * nres, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(t_nterm, P->nterm, 4 * n, cudaMemcpyHostToDevice));
    }
    CUDA_TRY(cudaMemcpy(t_res, kResidueMass, sizeof kResidueMass, cudaMemcpyHostToDevice));
    db->v.pep_mono = (const float*)db->d_pep_mono;
    db->v.pep_len = (const uint8_t*)db->d_pep_len;
    db->v.pep_flags = (const uint8_t*)db->d_pep_flags;
    db->v.pep_missed = (const uint8_t*)db->d_pep_missed;
    db->v.ion_off = (const uint32_t*)db->d_ion_off;
    db->v.ions = (const float*)db->d_ions;
    if (n) {
        k_build_ions<<<(unsigned)((n + 127) / 128), 128>>>((uint32_t)n, (const uint32_t*)t_off, (const uint8_t*)t_seq, (const float*)t_mods,
                                                           (const float*)t_nterm, (const float*)db->d_pep_mono, (const uint32_t*)db->d_ion_off,
                                                           (uint32_t)n_kinds, db->v, (float*)db->d_ions, (const float*)t_res);
        CUDA_TRY(cudaGetLastError());
    }
    CUDA_TRY(cudaDeviceSynchronize());
    return 0;
}

static int db_new(int device, sage_b200_db** out) {
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(SAGE_B200_ECUDA, "no CUDA device available (%s): sage_b200 has no CPU fallback", e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail(SAGE_B200_EINVAL, "device %d out of range (0..%d)", device, ndev - 1);
    CUDA_TRY(cudaSetDevice(device));
    sage_b200_db* db = new sage_b200_db();
    db->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) db->sm_count = prop.multiProcessorCount;
    *out = db;
    return 0;
}

extern "C" int sage_b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

extern "C" void sage_b200_db_destroy(sage_b200_db* db) {
    if (!db) return;
    cudaSetDevice(db->device);
    db->wide.release();
    db->narrow.release();
    void* ps[] = {db->d_page_grid, db->d_bucket_lut, db->d_pep_lut, db->d_frag, db->d_bucket_min, db->d_pep_mono, db->d_ion_off, db->d_ions, db->d_pep_len, db->d_pep_flags, db->d_pep_missed};
    for (void* p : ps)
        if (p) cudaFree(p);
    delete db;
}

// Search directories over the finished index (see DbView). Skipped (plain binary searches are used) when the shapes do not fit.
static int db_build_directories(sage_b200_db* db) {
    DbView& v = db->v;
    v.page_grid = nullptr; v.bucket_lut = nullptr; v.pep_lut = nullptr;
    if (v.n_frag == 0 || v.n_bucket == 0 || v.n_pep == 0 || (getenv("SAGE_B200_NO_DIRECTORIES") && getenv("SAGE_B200_NO_DIRECTORIES")[0] == '1')) return 0;
    int rc;
    if (v.bucket_size <= 65535u) {
        // cells per page ~ bucket_size / entries-per-cell: the in-cell search that follows a grid lookup is a chain of dependent loads
        uint32_t epc = 2;   // measured on cfg2 (preliminary scoring, ms): 32 entries per cell 1.87, 8: 1.83, 4: 1.82, 2: 1.81 (CTA kernel); 0.905 -> 0.876 (warp kernel); +6 % index memory
        if (const char* e = getenv("SAGE_B200_GRID_ENTRIES")) epc = (uint32_t)std::min(1024, std::max(1, atoi(e)));
        uint32_t cells = 64;
        while (cells < 16384 && (uint64_t)cells * epc < v.bucket_size) cells <<= 1;
        uint32_t shift = 0;
        while (((uint64_t)v.n_pep >> shift) >= cells) shift++;
        const uint32_t gn = (uint32_t)(((uint64_t)v.n_pep - 1) >> shift) + 1;   // cells 0..gn-1 cover every PeptideIx
        const uint64_t total = (uint64_t)v.n_bucket * (gn + 1);
        if ((rc = dmalloc(db, &db->d_page_grid, 2 * total))) return rc;
        k_build_page_grid<<<(unsigned)((total + 255) / 256), 256>>>(v, shift, gn, (uint16_t*)db->d_page_grid);
        CUDA_TRY(cudaGetLastError());
        v.grid_shift = shift; v.grid_n = gn;
    }
    float ends[2] = {0.f, 0.f};
    CUDA_TRY(cudaMemcpy(&ends[0], db->d_bucket_min, 4, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(&ends[1], (const float*)db->d_bucket_min + (v.n_bucket - 1), 4, cudaMemcpyDeviceToHost));
    bool lut_ok = ends[0] > 0.0f && std::isfinite(ends[0]) && std::isfinite(ends[1]);   // positive finite m/z: float order == total_cmp order
    if (lut_ok) {
        const float w = (ends[1] - ends[0]) / (float)BUCKET_LUT_CELLS;
        const float inv_w = (w > 0.0f && w < 3.0e38f) ? 1.0f / w : 0.0f;
        if ((rc = dmalloc(db, &db->d_bucket_lut, 4 * BUCKET_LUT_CELLS))) return rc;
        k_build_bucket_lut<<<BUCKET_LUT_CELLS / 256, 256>>>(v, ends[0], inv_w, (uint32_t*)db->d_bucket_lut);
        CUDA_TRY(cudaGetLastError());
        v.blut_base = ends[0]; v.blut_inv_w = inv_w;
    }
    // precursor-mass LUT over peptides[].monoisotopic (sorted ascending; needs positive finite ends like the bucket LUT)
    float pe[2] = {0.f, 0.f};
    CUDA_TRY(cudaMemcpy(&pe[0], db->d_pep_mono, 4, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(&pe[1], (const float*)db->d_pep_mono + (v.n_pep - 1), 4, cudaMemcpyDeviceToHost));
    const float pw = (pe[1] - pe[0]) / (float)PEP_LUT_CELLS;
    bool plut_ok = pe[0] > 0.0f && std::isfinite(pe[1]) && pw > 0.0f && pw < 3.0e38f;
    if (plut_ok) {   // only for a table the reference's binary search is well defined on: ascending, positive, finite
        uint32_t* d_bad = nullptr;
        uint32_t h_bad = 1;
        CUDA_TRY(cudaMalloc(&d_bad, 4));
        cudaMemset(d_bad, 0, 4);
        k_check_ascending<<<(v.n_pep + 255) / 256, 256>>>(v.n_pep, (const float*)db->d_pep_mono, d_bad);
        cudaMemcpy(&h_bad, d_bad, 4, cudaMemcpyDeviceToHost);
        cudaFree(d_bad);
        plut_ok = h_bad == 0;
    }
    if (plut_ok) {
        if ((rc = dmalloc(db, &db->d_pep_lut, 4 * (PEP_LUT_CELLS + 1)))) return rc;
        k_build_pep_lut<<<(PEP_LUT_CELLS + 256) / 256, 256>>>(v, pe[0], 1.0f / pw, (uint32_t*)db->d_pep_lut);
        CUDA_TRY(cudaGetLastError());
        v.plut_base = pe[0]; v.plut_inv_w = 1.0f / pw;
    }
    CUDA_TRY(cudaDeviceSynchronize());
    if (plut_ok) v.pep_lut = (const uint32_t*)db->d_pep_lut;
    if (db->d_page_grid) v.page_grid = (const uint16_t*)db->d_page_grid;
    if (lut_ok) v.bucket_lut = (const uint32_t*)db->d_bucket_lut;
    return 0;
}

extern "C" int sage_b200_db_create(const sage_b200_peptides* peptides, const sage_b200_index* index, int device, sage_b200_db** out) {
    if (!out || !index) return fail(SAGE_B200_EINVAL, "db_create: null argument");
    if (index->bucket_size == 0 || index->bucket_size > 0x7FFFFFFFull) return fail(SAGE_B200_EINVAL, "bucket_size out of range");
    if (index->n_fragments && (!index->fragment_peptide || !index->fragment_mz || !index->bucket_min)) return fail(SAGE_B200_EINVAL, "index: null array");
    const uint64_t nb_expect = (index->n_fragments + index->bucket_size - 1) / index->bucket_size;
    if (index->n_buckets != nb_expect) return fail(SAGE_B200_EINVAL, "n_buckets %llu != ceil(n_fragments/bucket_size) %llu", (unsigned long long)index->n_buckets, (unsigned long long)nb_expect);
    sage_b200_db* db = nullptr;
    int rc = db_new(device, &db);
    if (rc) return rc;
    if ((rc = db_upload_peptides(db, peptides, index->ion_kinds, index->n_ion_kinds))) { sage_b200_db_destroy(db); return rc; }
    const uint64_t nf = index->n_fragments;
    db->v.n_frag = nf;
    db->v.n_bucket = (uint32_t)index->n_buckets;
    db->v.bucket_size = (uint32_t)index->bucket_size;
    if ((rc = dmalloc(db, &db->d_frag, 8 * nf + 64))) { sage_b200_db_destroy(db); return rc; }
    if ((rc = dmalloc(db, &db->d_bucket_min, 4 * index->n_buckets))) { sage_b200_db_destroy(db); return rc; }
    void *t_pep = nullptr, *t_mz = nullptr;
    auto cleanup = [&]() { if (t_pep) cudaFree(t_pep); if (t_mz) cudaFree(t_mz); };
    if (nf) {
        if (cudaMalloc(&t_pep, 4 * nf) != cudaSuccess || cudaMalloc(&t_mz, 4 * nf) != cudaSuccess) { cleanup(); sage_b200_db_destroy(db); return fail(SAGE_B200_ECUDA, "cudaMalloc of upload temporaries failed"); }
        cudaError_t ce = cudaMemcpy(t_pep, index->fragment_peptide, 4 * nf, cudaMemcpyHostToDevice);
        if (ce == cudaSuccess) ce = cudaMemcpy(t_mz, index->fragment_mz, 4 * nf, cudaMemcpyHostToDevice);
        if (ce == cudaSuccess) ce = cudaMemcpy(db->d_bucket_min, index->bucket_min, 4 * index->n_buckets, cudaMemcpyHostToDevice);
        if (ce != cudaSuccess) {   // these errors are not sticky: a later synchronize would not report them and the index would be garbage
            cleanup(); sage_b200_db_destroy(db);
            return fail(SAGE_B200_ECUDA, "index upload failed: %s", cudaGetErrorString(ce));
        }
        k_pack_fragments_soa<<<(unsigned)((nf + 255) / 256), 256>>>(nf, (const uint32_t*)t_pep, (const float*)t_mz, (uint2*)db->d_frag);
    }
    cudaError_t e = cudaDeviceSynchronize();
    cleanup();
    if (e != cudaSuccess) { sage_b200_db_destroy(db); return fail(SAGE_B200_ECUDA, "index upload failed: %s", cudaGetErrorString(e)); }
    db->v.frag = (const uint2*)db->d_frag;
    db->v.bucket_min = (const float*)db->d_bucket_min;
    // IndexedDatabase does not carry min_ion_index (it lives in Parameters, database.rs:128): infer it from the fragment count and
    // verify the index content against the ion table; only then may narrow windows be counted peptide-centrically.
    db->v.pep_centric_ok = 0;
    db->v.min_ion_index = 0;
    if (peptides->n_peptides && nf) {
        const uint64_t n = peptides->n_peptides;
        int found = -1;
        for (uint32_t m = 0; m <= 64 && found < 0; m++) {
            uint64_t tot = 0;
            for (uint64_t i = 0; i < n; i++) {
                const uint64_t L = peptides->residue_offsets[i + 1] - peptides->residue_offsets[i];
                tot += index->n_ion_kinds * ((L - 1) > m ? (L - 1) - m : 0);
            }
            if (tot == nf) found = (int)m;
            if (tot < nf) break;
        }
        if (found >= 0) {
            void *acc = nullptr, *mis = nullptr;
            uint32_t mismatch = 1;
            if (cudaMalloc(&acc, 8 * n) == cudaSuccess && cudaMalloc(&mis, 4) == cudaSuccess && cudaMemset(acc, 0, 8 * n) == cudaSuccess &&
                cudaMemset(mis, 0, 4) == cudaSuccess) {
                k_index_signature<<<(unsigned)((nf + 255) / 256), 256>>>(nf, db->v.frag, (uint32_t)n, (uint32_t*)acc);
                k_index_verify<<<(unsigned)((n + 127) / 128), 128>>>((uint32_t)n, db->v.pep_len, db->v.ion_off, db->v.ions, db->v.n_kinds, db->v, (uint32_t)found,
                                                                    (const uint32_t*)acc, (uint32_t*)mis);
                if (cudaMemcpy(&mismatch, mis, 4, cudaMemcpyDeviceToHost) != cudaSuccess) mismatch = 1;
            }
            if (acc) cudaFree(acc);
            if (mis) cudaFree(mis);
            cudaGetLastError();
            if (mismatch == 0) { db->v.min_ion_index = (uint32_t)found; db->v.pep_centric_ok = 1; }
        }
    }
    if ((rc = db_build_directories(db))) { sage_b200_db_destroy(db); return rc; }
    *out = db;
    return 0;
}

extern "C" int sage_b200_db_build(const sage_b200_peptides* peptides, uint64_t bucket_size, const uint8_t* ion_kinds, uint64_t n_ion_kinds,
                                  uint64_t min_ion_index, int device, sage_b200_db** out) {
    if (!out || !peptides || !ion_kinds) return fail(SAGE_B200_EINVAL, "db_build: null argument");
    if (bucket_size == 0 || (bucket_size & (bucket_size - 1)) || bucket_size > (1ull << 30))
        return fail(SAGE_B200_EINVAL, "bucket_size must be a power of two (Builder::make_parameters rounds up, database.rs:97)");
    sage_b200_db* db = nullptr;
    int rc = db_new(device, &db);
    if (rc) return rc;
    if ((rc = db_upload_peptides(db, peptides, ion_kinds, n_ion_kinds))) { sage_b200_db_destroy(db); return rc; }
    const uint64_t n = peptides->n_peptides;
    // fragments kept per peptide: n_kinds * max(0, L-1-min_ion_index)   (database.rs:281-291)
    std::vector<uint64_t> frag_off(n + 1);
    uint64_t nf = 0;
    for (uint64_t i = 0; i < n; i++) {
        frag_off[i] = nf;
        const uint64_t L = peptides->residue_offsets[i + 1] - peptides->residue_offsets[i];
        const uint64_t keep = (L - 1) > min_ion_index ? (L - 1) - min_ion_index : 0;
        nf += n_ion_kinds * keep;
    }
    frag_off[n] = nf;
    const uint32_t shift = ceil_log2_u64(bucket_size);
    const uint64_t nb = (nf + bucket_size - 1) / bucket_size;
    if (nb > 0xFFFFFFFFull) { sage_b200_db_destroy(db); return fail(SAGE_B200_ELIMIT, "too many buckets"); }
    db->v.n_frag = nf;
    db->v.n_bucket = (uint32_t)nb;
    db->v.bucket_size = (uint32_t)bucket_size;
    db->v.min_ion_index = (uint32_t)std::min<uint64_t>(min_ion_index, 0xFFFFFFFFull);
    db->v.pep_centric_ok = 1;  // the index is generated from the ion table with this filter by construction
    if ((rc = dmalloc(db, &db->d_frag, 8 * nf + 64))) { sage_b200_db_destroy(db); return rc; }
    if ((rc = dmalloc(db, &db->d_bucket_min, 4 * nb))) { sage_b200_db_destroy(db); return rc; }
    db->v.frag = (const uint2*)db->d_frag;
    db->v.bucket_min = (const float*)db->d_bucket_min;
    if (nf == 0) { *out = db; return 0; }

    void *d_off = nullptr, *k32a = nullptr, *k32b = nullptr, *pa = nullptr, *pb = nullptr, *k64a = nullptr, *k64b = nullptr, *mza = nullptr, *mzb = nullptr, *tmp = nullptr;
    auto cleanup = [&]() { for (void* p : {d_off, k32a, k32b, pa, pb, k64a, k64b, mza, mzb, tmp}) if (p) cudaFree(p); };
#define TRY_BUILD(expr)                                                                                                    \
    do {                                                                                                                   \
        cudaError_t _e = (expr);                                                                                           \
        if (_e != cudaSuccess) { cleanup(); sage_b200_db_destroy(db); return fail(SAGE_B200_ECUDA, "%s failed: %s", #expr, cudaGetErrorString(_e)); } \
    } while (0)
    TRY_BUILD(cudaMalloc(&d_off, 8 * (n + 1)));
    TRY_BUILD(cudaMemcpy(d_off, frag_off.data(), 8 * (n + 1), cudaMemcpyHostToDevice));
    TRY_BUILD(cudaMalloc(&k32a, 4 * nf)); TRY_BUILD(cudaMalloc(&k32b, 4 * nf));
    TRY_BUILD(cudaMalloc(&pa, 4 * nf)); TRY_BUILD(cudaMalloc(&pb, 4 * nf));
    k_gen_fragments<<<(unsigned)((n + 127) / 128), 128>>>((uint32_t)n, db->v.pep_len, db->v.ion_off, db->v.ions, db->v.n_kinds, db->v, (uint32_t)std::min<uint64_t>(min_ion_index, 0xFFFFFFFFull),
                                                          nullptr, (const uint64_t*)d_off, (uint32_t*)k32a, (uint32_t*)pa);
    TRY_BUILD(cudaGetLastError());
    // (1) stable LSD radix sort by fragment m/z (par_sort_unstable_by fragment_mz, database.rs:301; ties keep PeptideIx order)
    size_t tb = 0;
    if (nf > 0x7FFFFFFFull) { cleanup(); sage_b200_db_destroy(db); return fail(SAGE_B200_ELIMIT, "more than 2^31 fragments: sort in slabs not implemented"); }
    TRY_BUILD(cub::DeviceRadixSort::SortPairs(nullptr, tb, (const uint32_t*)k32a, (uint32_t*)k32b, (const uint32_t*)pa, (uint32_t*)pb, (int)nf));
    TRY_BUILD(cudaMalloc(&tmp, tb + 16));
    TRY_BUILD(cub::DeviceRadixSort::SortPairs(tmp, tb, (const uint32_t*)k32a, (uint32_t*)k32b, (const uint32_t*)pa, (uint32_t*)pb, (int)nf));
    cudaFree(tmp); tmp = nullptr;
    cudaFree(k32a); k32a = nullptr; cudaFree(pa); pa = nullptr;
    // (2) bucket minima + (bucket, PeptideIx) keys, then a stable sort inside buckets (database.rs:337-346)
    TRY_BUILD(cudaMalloc(&k64a, 8 * nf)); TRY_BUILD(cudaMalloc(&k64b, 8 * nf));
    TRY_BUILD(cudaMalloc(&mza, 4 * nf)); TRY_BUILD(cudaMalloc(&mzb, 4 * nf));
    k_bucket_keys<<<(unsigned)((nf + 255) / 256), 256>>>(nf, shift, (const uint32_t*)k32b, (const uint32_t*)pb, (uint64_t*)k64a, (uint32_t*)mza, (float*)db->d_bucket_min);
    TRY_BUILD(cudaGetLastError());
    const int end_bit = std::min<int>(64, 32 + (int)ceil_log2_u64(nb + 1) + 1);
    TRY_BUILD(cub::DeviceRadixSort::SortPairs(nullptr, tb, (const uint64_t*)k64a, (uint64_t*)k64b, (const uint32_t*)mza, (uint32_t*)mzb, (int)nf, 0, end_bit));
    TRY_BUILD(cudaMalloc(&tmp, tb + 16));
    TRY_BUILD(cub::DeviceRadixSort::SortPairs(tmp, tb, (const uint64_t*)k64a, (uint64_t*)k64b, (const uint32_t*)mza, (uint32_t*)mzb, (int)nf, 0, end_bit));
    k_pack_fragments<<<(unsigned)((nf + 255) / 256), 256>>>(nf, (const uint64_t*)k64b, (const uint32_t*)mzb, (uint2*)db->d_frag);
    TRY_BUILD(cudaGetLastError());
    TRY_BUILD(cudaDeviceSynchronize());
    cleanup();
#undef TRY_BUILD
    if ((rc = db_build_directories(db))) { sage_b200_db_destroy(db); return rc; }
    *out = db;
    return 0;
}

extern "C" int sage_b200_db_get_info(const sage_b200_db* db, sage_b200_db_info* info) {
    if (!db || !info) return fail(SAGE_B200_EINVAL, "db_info: null argument");
    info->n_peptides = db->v.n_pep; info->n_fragments = db->v.n_frag; info->n_buckets = db->v.n_bucket; info->bucket_size = db->v.bucket_size;
    info->n_ion_kinds = db->v.n_kinds; info->total_residues = db->total_residues; info->device = db->device;
    {   // + the lazily built block-major copies (open search / narrow search), as far as they exist now
        std::lock_guard<std::mutex> lock(db->wmu);
        info->device_bytes = db->device_bytes + db->wide.bytes + db->narrow.bytes + db->wide.retired_bytes + db->narrow.retired_bytes;
    }
    return 0;
}

extern "C" int sage_b200_db_export_index(const sage_b200_db* db, uint32_t* fragment_peptide, float* fragment_mz, float* bucket_min) {
    if (!db) return fail(SAGE_B200_EINVAL, "db_export_index: null db");
    CUDA_TRY(cudaSetDevice(db->device));
    const uint64_t nf = db->v.n_frag;
    if (nf && (fragment_peptide || fragment_mz)) {
        void *t_pep = nullptr, *t_mz = nullptr;
        CUDA_TRY(cudaMalloc(&t_pep, 4 * nf));
        CUDA_TRY(cudaMalloc(&t_mz, 4 * nf));
        k_unpack_fragments<<<(unsigned)((nf + 255) / 256), 256>>>(nf, db->v.frag, (uint32_t*)t_pep, (float*)t_mz);
        cudaError_t e = cudaDeviceSynchronize();
        if (e == cudaSuccess && fragment_peptide) e = cudaMemcpy(fragment_peptide, t_pep, 4 * nf, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess && fragment_mz) e = cudaMemcpy(fragment_mz, t_mz, 4 * nf, cudaMemcpyDeviceToHost);
        cudaFree(t_pep); cudaFree(t_mz);
        if (e != cudaSuccess) return fail(SAGE_B200_ECUDA, "export failed: %s", cudaGetErrorString(e));
    }
    if (bucket_min && db->v.n_bucket) CUDA_TRY(cudaMemcpy(bucket_min, db->d_bucket_min, 4ull * db->v.n_bucket, cudaMemcpyDeviceToHost));
    return 0;
}

// Secondary index for open search (device_common.cuh: WideIndexView): fragments keyed by (PeptideIx / block, m/z), one LSD radix sort, block
// offsets and a per-block m/z LUT. `block` = the scorer's count-tile size. Returns a view with frag == nullptr when the index cannot be built
// (out of memory, SAGE_B200_NO_WIDE_INDEX=1): k_prelim_wide then streams the page slices as the reference does.
// Builds (or returns) one block-major copy of the fragments. `cells_for(entries per block)` picks the LUT resolution; wmu must be held.
static WideIndexView build_block_index(const sage_b200_db* db, BlockIndexSlot& slot, uint32_t block, uint32_t cells) {
    WideIndexView none{};
    if (slot.v.frag != nullptr && slot.v.block == block) return slot.v;
    if (slot.failed || block == 0 || db->v.n_frag == 0 || db->v.n_pep == 0) return none;
    const uint64_t nf = db->v.n_frag;
    slot.retire();   // a rebuild with another block size (tests, scorers with very different tolerances): see BlockIndexSlot::retire
    void *k_a = nullptr, *k_b = nullptr, *p_a = nullptr, *p_b = nullptr, *tmp = nullptr, *d_rng = nullptr;
    auto cleanup = [&]() { for (void* p : {k_a, k_b, p_a, p_b, tmp, d_rng}) if (p) cudaFree(p); };
    auto give_up = [&]() { cleanup(); for (void** p : {&slot.d_frag, &slot.d_blk, &slot.d_lut}) { if (*p) cudaFree(*p); *p = nullptr; } slot.v = WideIndexView{}; slot.bytes = 0; cudaGetLastError(); slot.failed = 1; return WideIndexView{}; };
    const uint32_t n_block = (db->v.n_pep + block - 1) / block;
    while (cells > 256 && (uint64_t)n_block * (cells + 1) * 4 > (1024ull << 20)) cells >>= 1;   // at most 1 GB of LUT
    if (cudaMalloc(&slot.d_frag, 8 * nf + 64) != cudaSuccess || cudaMalloc(&slot.d_blk, 8 * ((size_t)n_block + 1)) != cudaSuccess ||
        cudaMalloc(&slot.d_lut, 4 * (size_t)n_block * (cells + 1)) != cudaSuccess)
        return give_up();
    if (cudaMalloc(&k_a, 8 * nf) != cudaSuccess || cudaMalloc(&k_b, 8 * nf) != cudaSuccess || cudaMalloc(&p_a, 4 * nf) != cudaSuccess ||
        cudaMalloc(&p_b, 4 * nf) != cudaSuccess || cudaMalloc(&d_rng, 8) != cudaSuccess)
        return give_up();
    k_wide_keys<<<(unsigned)((nf + 255) / 256), 256>>>(nf, db->v.frag, block, (uint64_t*)k_a, (uint32_t*)p_a);
    int nb_bits = 1;
    while (nb_bits < 32 && (n_block >> nb_bits)) nb_bits++;
    size_t tb = 0;
    if (nf > 0x7FFFFFFFull) return give_up();
    if (cub::DeviceRadixSort::SortPairs(nullptr, tb, (const uint64_t*)k_a, (uint64_t*)k_b, (const uint32_t*)p_a, (uint32_t*)p_b, (int)nf, 0, 32 + nb_bits) != cudaSuccess ||
        cudaMalloc(&tmp, tb + 16) != cudaSuccess ||
        cub::DeviceRadixSort::SortPairs(tmp, tb, (const uint64_t*)k_a, (uint64_t*)k_b, (const uint32_t*)p_a, (uint32_t*)p_b, (int)nf, 0, 32 + nb_bits) != cudaSuccess)
        return give_up();
    k_wide_pack<<<(unsigned)((nf + 255) / 256), 256>>>(nf, (const uint64_t*)k_b, (const uint32_t*)p_b, (uint2*)slot.d_frag);
    k_wide_block_offsets<<<(n_block + 1 + 255) / 256, 256>>>(nf, (const uint64_t*)k_b, n_block, (uint64_t*)slot.d_blk);
    // m/z range of the index (positive floats order like their bit patterns)
    const uint32_t rng0[2] = {0xFFFFFFFFu, 0u};
    if (cudaMemcpy(d_rng, rng0, 8, cudaMemcpyHostToDevice) != cudaSuccess) return give_up();
    k_frag_mz_range<<<(unsigned)std::min<uint64_t>((nf + 255) / 256, 4096), 256>>>(nf, db->v.frag, (uint32_t*)d_rng);
    uint32_t rng[2];
    if (cudaMemcpy(rng, d_rng, 8, cudaMemcpyDeviceToHost) != cudaSuccess) return give_up();
    cleanup();
    k_a = k_b = p_a = p_b = tmp = d_rng = nullptr;
    float lo, hi;
    memcpy(&lo, &rng[0], 4); memcpy(&hi, &rng[1], 4);
    WideIndexView w{};
    w.frag = (const uint2*)slot.d_frag; w.blk_off = (const uint64_t*)slot.d_blk; w.lut = (const uint32_t*)slot.d_lut;
    w.block = block; w.n_block = n_block; w.cells = cells;
    const float width = (hi - lo) / (float)cells;
    w.base = (std::isfinite(lo) && lo > 0.0f) ? lo : 0.0f;
    w.inv_w = (std::isfinite(width) && width > 0.0f && lo > 0.0f) ? 1.0f / width : 0.0f;
    if (w.inv_w > 0.0f) {
        const uint64_t total = (uint64_t)n_block * (cells + 1);
        k_wide_lut<<<(unsigned)((total + 255) / 256), 256>>>(w, (uint32_t*)slot.d_lut);
    } else if (cudaMemset(slot.d_lut, 0, 4 * (size_t)n_block * (cells + 1)) != cudaSuccess) return give_up();   // degenerate range: every walk starts at the block start
    if (cudaDeviceSynchronize() != cudaSuccess) return give_up();
    slot.v = w;
    slot.bytes = 8 * nf + 8 * ((uint64_t)n_block + 1) + 4ull * n_block * (cells + 1);
    return w;
}

static WideIndexView db_wide_index(const sage_b200_db* db, uint32_t block) {
    std::lock_guard<std::mutex> lock(db->wmu);
    if (const char* e = getenv("SAGE_B200_NO_WIDE_INDEX")) if (e[0] == '1') return WideIndexView{};   // A/B + tests: stream the page slices instead
    // ~2 M entries per 80 k-peptide block, most of them inside a third of the m/z range: 2^18 cells leave a few dozen entries per cell there,
    // so the conservative (one cell early) start of a walk costs about one extra 32-entry fetch (measured: 2^16 cells -> ~8 extra fetches)
    return build_block_index(db, db->wide, block, 1u << 18);
}

// The narrow-search copy: blocks of `block` peptides (a +-20 ppm window holds a few hundred), LUT cells ~ `cells_x` per block entry.
static WideIndexView db_narrow_index(const sage_b200_db* db, uint32_t block, uint32_t cells_x, bool exact) {
    std::lock_guard<std::mutex> lock(db->wmu);
    // an automatically sized request accepts an existing copy whose blocks are within a factor of two (scorers with different tolerances
    // sharing one index must not rebuild it in turns)
    if (!exact && db->narrow.v.frag != nullptr && db->narrow.v.block * 2 >= block && db->narrow.v.block <= block * 2) return db->narrow.v;
    const uint32_t n_block = (db->v.n_pep + block - 1) / std::max(block, 1u);
    const uint64_t per_block = n_block ? db->v.n_frag / n_block : 0;
    uint32_t cells = 1024;
    while (cells < (1u << 18) && (uint64_t)cells < per_block * cells_x) cells <<= 1;
    return build_block_index(db, db->narrow, block, cells);
}

// Dynamic shared-memory opt-in of the kernels that need more than 48 KB: set ONCE per device to the device maximum (the attribute is per-function,
// per-device state; setting it per launch to the launch's own size would let two scorers with different shapes undo each other's setting).
static int ensure_kernel_attributes(int device) {
    static std::mutex mu;
    static bool done[64] = {};
    std::lock_guard<std::mutex> lock(mu);
    if (device >= 0 && device < 64 && done[device]) return 0;
    int optin = 0;
    CUDA_TRY(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    auto raise = [&](const void* fn) -> cudaError_t {   // dynamic limit = opt-in maximum minus the kernel's static shared memory
        cudaFuncAttributes fa;
        cudaError_t e = cudaFuncGetAttributes(&fa, fn);
        if (e != cudaSuccess) return e;
        return cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - (int)fa.sharedSizeBytes);
    };
    CUDA_TRY(raise((const void*)k_prelim_narrow));
    CUDA_TRY(raise((const void*)k_replay<true>));
    CUDA_TRY(raise((const void*)k_replay<false>));
    CUDA_TRY(raise((const void*)k_prelim_wide));
    CUDA_TRY(raise((const void*)k_score<false>));
    CUDA_TRY(raise((const void*)k_score<true>));
    CUDA_TRY(raise((const void*)k_process_ms2));
    if (device >= 0 && device < 64) done[device] = true;
    return 0;
}

// Which build of glibc's log() is the host libm (glibc_log.cuh)? Both variants are evaluated on the CPU and compared with std::log bit for bit
// on a few thousand inputs of the kinds the path feeds it: hyperscore products, lambda, arguments near 1 (the only region where the two
// variants differ). Returns 0 (FMA-contracted), 1 (plain), or -1 when neither matches (non-glibc libm: the device then uses variant 0 and
// hyperscore / poisson agree with the host to <= 1 ulp instead of bit for bit).
extern "C" int sage_b200_host_log_variant(void) {
    static int cached = -2;
    if (cached != -2) return cached;
    uint64_t st = 0x9E3779B97F4A7C15ull;
    auto next = [&]() { st ^= st << 13; st ^= st >> 7; st ^= st << 17; return st; };
    bool ok[2] = {true, true};
    for (int i = 0; i < 6000; i++) {
        const uint64_t u = next();
        double x;
        switch (i % 3) {
            case 0: x = (double)((float)(u & 0xffffff) * 0.37f + 1.0f) * (double)((float)((u >> 24) & 0xffffff) * 1.91f + 1.0f); break;
            case 1: x = 0.93 + (double)(u >> 11) * 0x1p-53 * 0.15; break;
            default: x = (double)(u >> 11) * 0x1p-53 * 64.0; break;
        }
        volatile double vx = x;   // keep the compiler from folding std::log
        const double ref = std::log(vx);
        const double a = glog::glibc_log<true>(x), b = glog::glibc_log<false>(x);
        if (memcmp(&a, &ref, 8)) ok[0] = false;
        if (memcmp(&b, &ref, 8)) ok[1] = false;
    }
    cached = ok[0] ? 0 : (ok[1] ? 1 : -1);
    return cached;
}

// 1 when the host libm's log1pf (Rust's f32::ln_1p, OpenMS hyperscore) is the fdlibm/glibc function the kernels reproduce (glibc_log.cuh).
extern "C" int sage_b200_host_log1pf_exact(void) {
    static int cached = -1;
    if (cached >= 0) return cached;
    uint64_t st = 0x2545F4914F6CDD1Dull;
    auto next = [&]() { st ^= st << 13; st ^= st >> 7; st ^= st << 17; return st; };
    int ok = 1;
    for (int i = 0; i < 20000 && ok; i++) {
        const uint64_t u = next();
        float x;
        switch (i % 3) {
            case 0: x = (float)(u & 0xffffff) * 3.7f; break;                                  // summed intensities
            case 1: x = (float)((double)(u >> 11) * 0x1p-53 * 2.0 - 0.9); break;            // around the branch points
            default: { uint32_t b = (uint32_t)(u >> 33); memcpy(&x, &b, 4); break; }          // any non-negative float
        }
        volatile float vx = x;
        const float ref = log1pf(vx), got = glog::glibc_log1pf(x);
        if (memcmp(&ref, &got, 4) && !(ref != ref && got != got)) ok = 0;
    }
    cached = ok;
    return cached;
}

// ------------------------------------------------------------------------------------------------ scorer
constexpr int MASS_PARTS = 4;   // the masses copy of a chunk is cut into at most this many parts, each followed by its own counting launch

struct ChunkState {
    bool loaded = false;
    uint32_t nparts = 1, part_lo[MASS_PARTS + 1] = {0, 0, 0, 0, 0};   // spectra [part_lo[p], part_lo[p+1]) belong to part p of the masses copy
    uint32_t n = 0, pmax = 2, zmax = 1, base = 0;
    uint64_t npk = 0;
    size_t nitems = 0, smem = 0, small_bytes = 0;
    size_t o_off = 0, o_pmz = 0, o_tic = 0, o_ilo = 0, o_ihi = 0, o_rt = 0, o_ims = 0, o_chg = 0;
    bool timed_upload = false;
    uint64_t hits_cap = 0, force_hits = 0;   // split scoring: entries of the hit arena / exact need of a re-run
    uint64_t nlist_cap = 0, force_nlist = 0, force_wide = 0;   // work-list capacities of the current attempt / exact needs for a re-run
    uint32_t wide_cap = 0;
    double t_issue0 = 0, t_issue1 = 0;   // host time (ms since the call started) when queueing this chunk began / ended (trace only)
};

// One in-flight chunk: its own stream, device buffers, pinned staging and pending-download bookkeeping. score_batch alternates
// between two lanes so that the H2D copy of chunk i+1 and the D2H of chunk i-1 overlap the kernels of chunk i.
struct Lane {
    cudaStream_t stream = nullptr;   // kernels + D2H
    cudaStream_t copy = nullptr;     // H2D: masses first (all the counting kernels need), intensities behind them, overlapping setup + preliminary scoring
    cudaEvent_t ev[9] = {};   // 0/1 H2D, 6 run start, 2 setup end, 8 counting kernels end, 3 replay end, 4 k_score end, 7/5 D2H
    cudaStream_t copy2 = nullptr;    // (unused: a second H2D stream did not overtake the queued bulk copies, see chunk_upload)
    cudaEvent_t ev_masses = nullptr, ev_intens = nullptr, ev_small = nullptr;
    cudaEvent_t ev_part[MASS_PARTS] = {};   // masses of the spectra [part_lo[p], part_lo[p+1]) are on the device
    DevBuf d_small, d_masses, d_intens, d_queries, d_hits, d_keys, d_features, d_counts, d_counters, d_dbgk, d_dbgm, d_sort, d_sorttmp, d_wlist, d_wslots,
        d_witems, d_citems, d_nlist, d_nslots;
    PinBuf h_small, h_masses, h_intens, h_features, h_counts, h_counters;
    DevBuf d_frags;
    DevBuf d_cand, d_meta, d_recs, d_hkey, d_emit, d_hitk, d_hiti, d_hitt;   // split scoring (k_score<true> -> k_fold -> k_features)
    ChunkState chunk;
    // pending work of the chunk in flight
    bool ran = false, downloading = false, dbg = false;
    uint64_t launches = 0;
    sage_b200_feature* fdst = nullptr;
    uint32_t* cdst = nullptr;
    bool f_pinned = false, c_pinned = false;
    // helper thread staging the intensities of a chunk whose caller arrays are pageable (chunk_upload starts it, chunk_run joins it)
    std::thread stager;
    std::unique_ptr<StagePool> pool{new StagePool};   // copy threads of staged_h2d (started by the first pageable chunk)
    int stager_rc = 0;
    char stager_msg[256] = {0};
    void release() {
        if (stager.joinable()) stager.join();
        for (DevBuf* b : {&d_small, &d_masses, &d_intens, &d_queries, &d_hits, &d_keys, &d_features, &d_counts, &d_counters, &d_dbgk, &d_dbgm, &d_sort, &d_sorttmp,
                          &d_wlist, &d_wslots, &d_witems, &d_citems, &d_nlist, &d_nslots, &d_frags, &d_cand, &d_meta, &d_recs, &d_hkey, &d_emit, &d_hitk, &d_hiti, &d_hitt}) b->release();
        for (PinBuf* b : {&h_small, &h_masses, &h_intens, &h_features, &h_counts, &h_counters}) b->release();
        for (auto& e : ev) if (e) cudaEventDestroy(e);
        if (ev_masses) cudaEventDestroy(ev_masses);
        if (ev_intens) cudaEventDestroy(ev_intens);
        if (ev_small) cudaEventDestroy(ev_small);
        for (auto& e : ev_part) if (e) cudaEventDestroy(e);
        if (copy2) cudaStreamDestroy(copy2);
        if (stream) cudaStreamDestroy(stream);
        if (copy) cudaStreamDestroy(copy);
    }
};

struct sage_b200_scorer {
    const sage_b200_db* db = nullptr;
    int device = 0;   // copy of db->device: scorer_destroy must not touch a db that was destroyed first
    sage_b200_scorer_params params{};
    ScorerView sv{};
    std::mutex mu;
    Lane lanes[2];
    DevBuf d_lnfact, d_keep;
    uint32_t quick_mode = 0;   // != 0 only inside sage_b200_quick_score
    int sort_spectra = 1;
    // annotate_matches: caller's fragment array for the current call and the running global offset
    sage_b200_fragment* frag_dst = nullptr;
    uint64_t frag_cap = 0, frag_used = 0;
    int pipeline_chunks = 1;   // score_batch cuts a batch into at least this many chunks (tuning / tests; large batches are cut at 65536 spectra anyway)
    // learned work-list sizes (per spectrum of a chunk): narrow key-list arena entries and open-search queries. A chunk that needs more than
    // its capacity is re-run once with the exact sizes it counted, and the estimates grow.
    double nlist_per_spectrum = 512.0, wide_per_spectrum = 0.0;
    // narrow windows are counted against the small-block copy of the index (block_probe) unless narrow_index == 0: then the reference's loop
    // order probes the page index and the page / entry work counters are produced (tests, bench's work_per_step pass)
    int score_split = 1;            // non-chimeric scoring runs as k_score<true> -> k_fold -> k_features -> k_rows (0: the fused kernel; tests compare both)
    double hits_per_spectrum = 0.0; // learned: hit-arena entries (= scoring tasks) a spectrum needs
    int narrow_index = 1;
    uint32_t narrow_block_auto = 0;   // block size narrow_block_for chose for this scorer's precursor tolerance
    int narrow_cta = 1;   // windows of WARPQ_CAP+1..NARROW_CAP peptides (one CTA per query) use the copy too
    uint32_t narrow_block = 0 /* 0 = sized by the average precursor window, see narrow_block_for */, narrow_cells_x = 4;   // measured on cfg2 (counting kernel ms; page index 0.628): 1024 x2 0.736 | 512 x2 0.644 | 1024 x4 0.637 |
                                                       // 512 x4 0.585 | 256 x2 0.585 | 256 x4 0.546 | 256 x8 0.546 | 128 x4 0.555 (profiles/r02_nblk*)
    int mass_parts = 2;        // measured on cfg2 (e2e ms per 50k-spectrum call, profiles/r02_parts): 1 part 3.24 | 2 -> 3.17 | 3 -> 3.38 | 4 -> 3.41
    int first_chunk_pct = 0;   // measured on cfg2 (e2e ms per 50k-spectrum call): 0 -> 3.44, 10 -> 3.46, 20 -> 3.52, 35 -> 3.53 (profiles/r02_e_*)
    // SAGE_B200_TRACE=1: per-chunk device timeline (ms since the start of the call) on stderr
    bool trace = false;
    cudaEvent_t ev_base = nullptr;
    std::chrono::steady_clock::time_point t_base;
    sage_b200_counters last{};
};

extern "C" int sage_b200_scorer_create(const sage_b200_db* db, const sage_b200_scorer_params* p, sage_b200_scorer** out) {
    if (!db || !p || !out) return fail(SAGE_B200_EINVAL, "scorer_create: null argument");
    if (p->report_psms == 0) return fail(SAGE_B200_EINVAL, "report_psms must be >= 1");
    if (p->report_psms > K_MAX / 2) return fail(SAGE_B200_ELIMIT, "report_psms %u > %d not supported", p->report_psms, K_MAX / 2);
    if (p->precursor_tol.kind < 0 || p->precursor_tol.kind > 2 || p->fragment_tol.kind < 0 || p->fragment_tol.kind > 2) return fail(SAGE_B200_EINVAL, "bad tolerance kind");
    if (p->score_type > 1) return fail(SAGE_B200_EINVAL, "bad score_type");
    CUDA_TRY(cudaSetDevice(db->device));
    { int rc_attr = ensure_kernel_attributes(db->device); if (rc_attr) return rc_attr; }
    sage_b200_scorer* s = new sage_b200_scorer();
    s->db = db;
    s->device = db->device;
    s->params = *p;
    ScorerView& v = s->sv;
    v.precursor_tol = {p->precursor_tol.kind, p->precursor_tol.lo, p->precursor_tol.hi};
    v.fragment_tol = {p->fragment_tol.kind, p->fragment_tol.lo, p->fragment_tol.hi};
    v.min_matched_peaks = p->min_matched_peaks;
    v.min_iso = p->min_isotope_err; v.max_iso = p->max_isotope_err;
    v.min_charge = p->min_precursor_charge; v.max_charge = p->max_precursor_charge;
    v.override_charge = p->override_precursor_charge; v.max_fragment_charge_opt = p->max_fragment_charge;
    v.chimera = p->chimera; v.wide_window = p->wide_window; v.annotate = p->annotate_matches; v.score_type = p->score_type;
    v.report_psms = p->report_psms;
    v.kparam = std::max<uint32_t>(50, 2 * p->report_psms);  // trim_hits (scoring.rs:323-326): k = min(len, max(50, 2*report_psms))
    v.n_iso = (v.min_iso != v.max_iso) ? (uint32_t)std::max(0, v.max_iso - v.min_iso + 1) : 1;
    v.n_ch_max = v.max_charge >= v.min_charge ? v.max_charge - v.min_charge + 1 : 0;
    if (v.n_ch_max < 1) v.n_ch_max = 1;  // known-charge spectra still need one slot
    if (v.n_iso > 32 || v.n_ch_max > 16) { delete s; return fail(SAGE_B200_ELIMIT, "isotope range > 32 or charge range > 16 not supported"); }
    v.qmax = std::max<uint32_t>(1, v.n_iso) * v.n_ch_max;
    v.lcap = std::max<uint32_t>(std::max<uint32_t>(v.n_iso, v.n_ch_max), 1) * v.kparam;
    v.wide_tile = WIDE_TILE;
    v.wide_lmax = WIDE_LMAX;
    v.wide_variant = 0;  // measured: float compares 142 ms vs unsigned bit-window 150 ms on cfg4
    if (const char* e = getenv("SAGE_B200_WIDE_VARIANT")) v.wide_variant = (uint32_t)atoi(e);
    v.pep_cap = 0;   // peptide-centric counting of small windows is opt-in: with the dense page grid the index path wins on cfg2 at every cap (0: 1.71 ms, 32: 1.74, 64: 1.82)
    if (const char* e = getenv("SAGE_B200_PEP_CAP")) v.pep_cap = (uint32_t)std::min<long>(std::max<long>(atol(e), 0), (long)NARROW_CAP);
    {   // lnfact table with the host libm (the reference's f64::ln): Stirling form of scoring.rs:170-177
        const uint32_t N = 4096;
        std::vector<double> tab(N);
        tab[0] = 1.0;
        for (uint32_t n = 1; n < N; n++) {
            const double x = (double)n;
            tab[n] = x * std::log(x) - x + 0.5 * std::log(x) + 0.5 * std::log(3.14159265358979323846 * 2.0 * x);
        }
        int rc2 = s->d_lnfact.reserve(8 * N);
        if (rc2) { delete s; return rc2; }
        CUDA_TRY(cudaMemcpy(s->d_lnfact.p, tab.data(), 8 * N, cudaMemcpyHostToDevice));
        v.lnfact_tab = s->d_lnfact.as<double>();
        v.lnfact_n = N;
    }
    v.log_variant = (uint32_t)std::max(0, sage_b200_host_log_variant());
    v.score_fast = 1;
    if (const char* e = getenv("SAGE_B200_SCORE_FAST")) v.score_fast = atoi(e) != 0;
    if (const char* e = getenv("SAGE_B200_SORT")) s->sort_spectra = atoi(e);
    for (Lane& L : s->lanes) {
        CUDA_TRY(cudaStreamCreateWithFlags(&L.stream, cudaStreamNonBlocking));
        CUDA_TRY(cudaStreamCreateWithFlags(&L.copy, cudaStreamNonBlocking));
        for (auto& e : L.ev) CUDA_TRY(cudaEventCreate(&e));
        CUDA_TRY(cudaEventCreate(&L.ev_masses));
        CUDA_TRY(cudaEventCreate(&L.ev_intens));
        CUDA_TRY(cudaEventCreate(&L.ev_small));
        for (auto& e : L.ev_part) CUDA_TRY(cudaEventCreate(&e));
        CUDA_TRY(cudaStreamCreateWithFlags(&L.copy2, cudaStreamNonBlocking));
    }
    if (const char* e = getenv("SAGE_B200_PIPELINE_CHUNKS")) s->pipeline_chunks = std::max(1, atoi(e));
    if (const char* e = getenv("SAGE_B200_TRACE")) s->trace = e[0] == '1';
    if (const char* e = getenv("SAGE_B200_SCORE_SPLIT")) s->score_split = atoi(e) != 0;
    if (const char* e = getenv("SAGE_B200_NARROW_INDEX")) s->narrow_index = atoi(e) != 0;
    if (const char* e = getenv("SAGE_B200_NARROW_CTA")) s->narrow_cta = atoi(e) != 0;
    if (const char* e = getenv("SAGE_B200_NARROW_BLOCK")) s->narrow_block = (uint32_t)std::max(0, atoi(e));
    if (const char* e = getenv("SAGE_B200_NARROW_CELLS_X")) s->narrow_cells_x = (uint32_t)std::max(1, atoi(e));
    if (const char* e = getenv("SAGE_B200_MASS_PARTS")) s->mass_parts = std::min(MASS_PARTS, std::max(1, atoi(e)));
    if (const char* e = getenv("SAGE_B200_FIRST_CHUNK_PCT")) s->first_chunk_pct = std::min(50, std::max(0, atoi(e)));
    CUDA_TRY(cudaEventCreate(&s->ev_base));
    *out = s;
    return 0;
}

extern "C" int sage_b200_scorer_set_option(sage_b200_scorer* s, const char* name, int64_t value) {
    if (!s || !name) return fail(SAGE_B200_EINVAL, "scorer_set_option: null argument");
    std::lock_guard<std::mutex> lock(s->mu);
    if (!strcmp(name, "sort_spectra")) { s->sort_spectra = value != 0; return 0; }
    if (!strcmp(name, "pipeline_chunks")) { s->pipeline_chunks = (int)std::max<int64_t>(1, value); return 0; }
    if (!strcmp(name, "score_split")) { s->score_split = value != 0; return 0; }
    if (!strcmp(name, "narrow_index")) { s->narrow_index = value != 0; return 0; }
    if (!strcmp(name, "narrow_block")) {   // test hook: peptides per block of the narrow-search copy (rebuilds it on the next batch)
        if (value != 0 && (value < 64 || value > (1 << 20))) return fail(SAGE_B200_EINVAL, "narrow_block must be 0 (automatic) or 64..1048576");
        s->narrow_block = (uint32_t)value;
        return 0;
    }
    if (!strcmp(name, "mass_parts")) {
        if (value < 1 || value > MASS_PARTS) return fail(SAGE_B200_EINVAL, "mass_parts must be 1..%d", MASS_PARTS);
        s->mass_parts = (int)value;
        return 0;
    }
    if (!strcmp(name, "wide_lmax")) {  // test hook: a tiny survivor list forces the overflow -> in-kernel serial replay path
        if (value < (int64_t)K_MAX || value > (int64_t)WIDE_LMAX) return fail(SAGE_B200_EINVAL, "wide_lmax must be in %d..%u", K_MAX, WIDE_LMAX);
        s->sv.wide_lmax = (uint32_t)value;
        return 0;
    }
    if (!strcmp(name, "wide_tile")) {  // test hook: smaller tiles exercise the multi-tile path on small databases
        if (value < 256 || value > (int64_t)WIDE_TILE || (value & 1)) return fail(SAGE_B200_EINVAL, "wide_tile must be even and in 256..%u", WIDE_TILE);
        s->sv.wide_tile = (uint32_t)value;
        return 0;
    }
    if (!strcmp(name, "worklist_reset")) {   // test hook: forget the learned work-list sizes; value = narrow arena entries per spectrum to start from
        if (value < 0) return fail(SAGE_B200_EINVAL, "worklist_reset takes a non-negative entry count");
        s->nlist_per_spectrum = (double)value;
        s->wide_per_spectrum = 0.0;
        s->hits_per_spectrum = value > 0 ? (double)value : 0.0;   // > 0: start the split scorer's hit arena at that many entries per spectrum too
        return 0;
    }
    if (!strcmp(name, "score_fast")) {  // 0: k_score always takes the generic task body (tests compare both)
        s->sv.score_fast = value != 0;
        return 0;
    }
    if (!strcmp(name, "log_variant")) {  // test hook: 0 = glibc log() as built with FMA contraction, 1 = without (default: whichever the host libm is)
        if (value < 0 || value > 1) return fail(SAGE_B200_EINVAL, "log_variant must be 0 or 1");
        s->sv.log_variant = (uint32_t)value;
        return 0;
    }
    if (!strcmp(name, "pep_cap")) {  // 0 (default) = always probe the fragment index (reference loop order)
        if (value < 0 || value > (int64_t)NARROW_CAP) return fail(SAGE_B200_EINVAL, "pep_cap must be 0..%u", NARROW_CAP);
        s->sv.pep_cap = (uint32_t)value;
        return 0;
    }
    return fail(SAGE_B200_EINVAL, "unknown option '%s'", name);
}

extern "C" void sage_b200_scorer_destroy(sage_b200_scorer* s) {
    if (!s) return;
    cudaSetDevice(s->device);
    for (Lane& L : s->lanes) L.release();
    if (s->ev_base) cudaEventDestroy(s->ev_base);
    s->d_lnfact.release();
    s->d_keep.release();
    delete s;
}

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Peptides per block of the narrow-search copy of the index: the power of two at or above the average precursor window of this scorer
// (sampled on the device from the peptide masses themselves), 128..4096. A probe then reads one or two short m/z runs. Measured (counting
// kernels, ms per step): cfg2 (windows ~180 peptides) 128 -> 0.555, 256 -> 0.546, 512 -> 0.585, 1024 -> 0.637; cfg3 (windows ~1500) 256 -> 20.4,
// 512 -> 14.0, 1024 -> 10.4, 2048 -> 9.0 (page index: 22-28).
static int narrow_block_for(sage_b200_scorer* S) {
    if (S->narrow_block_auto) return 0;
    const uint32_t samples = 4096;
    unsigned long long* d_sum = nullptr;
    unsigned long long sum = 0;
    CUDA_TRY(cudaMalloc(&d_sum, 8));
    cudaError_t e = cudaMemset(d_sum, 0, 8);
    if (e == cudaSuccess) {
        k_window_sample<<<(samples + 255) / 256, 256>>>(S->db->v, S->sv.precursor_tol, samples, d_sum);
        e = cudaMemcpy(&sum, d_sum, 8, cudaMemcpyDeviceToHost);
    }
    cudaFree(d_sum);
    if (e != cudaSuccess) return fail(SAGE_B200_ECUDA, "window sampling failed: %s", cudaGetErrorString(e));
    const double avg = (double)sum / samples;
    uint32_t block = 128;
    while (block < 4096 && (double)block < avg) block <<= 1;
    S->narrow_block_auto = block;
    return 0;
}

// Waits for the lane's staging thread (if one is running) and reports its error as this thread's.
static int lane_join_stager(Lane& L) {
    if (!L.stager.joinable()) return 0;
    L.stager.join();
    if (L.stager_rc) return fail(L.stager_rc, "%s", L.stager_msg);
    return 0;
}

// ---- one chunk of spectra through the device pipeline, in three phases:
//   chunk_upload   pack + H2D (spectra become device-resident)
//   chunk_run      k_setup_queries -> k_prelim_{narrow,wide} -> k_score (results stay on the device)
//   chunk_download D2H of Feature rows + counts
static int chunk_upload(sage_b200_scorer* S, Lane& L, const sage_b200_spectra* sp, uint64_t c0, uint64_t c1) {
    const ScorerView& sv = S->sv;
    ChunkState& C = L.chunk;
    C.loaded = false;
    const uint32_t n = (uint32_t)(c1 - c0);
    const uint64_t pk0 = sp->peak_offsets[c0], pk1 = sp->peak_offsets[c1];
    const uint64_t npk = pk1 - pk0;
    if (npk > 0xFFFFFFF0ull) return fail(SAGE_B200_ELIMIT, "chunk has too many peaks");
    C.n = n; C.npk = npk; C.base = (uint32_t)c0;
    // small per-spectrum arrays -> one pinned blob -> one H2D
    C.o_off = 0;
    C.o_pmz = align_up(C.o_off + 4 * (size_t)(n + 1), 16);
    C.o_tic = align_up(C.o_pmz + 4 * (size_t)n, 16);
    C.o_ilo = align_up(C.o_tic + 4 * (size_t)n, 16);
    C.o_ihi = align_up(C.o_ilo + 4 * (size_t)n, 16);
    C.o_rt = align_up(C.o_ihi + 4 * (size_t)n, 16);
    C.o_ims = align_up(C.o_rt + 4 * (size_t)n, 16);
    C.o_chg = align_up(C.o_ims + 4 * (size_t)n, 16);
    C.small_bytes = align_up(C.o_chg + n, 16);
    int rc;
    if ((rc = L.h_small.reserve(C.small_bytes))) return rc;
    if ((rc = L.d_small.reserve(C.small_bytes))) return rc;
    if ((rc = L.d_masses.reserve(4 * npk + 16))) return rc;
    if ((rc = L.d_intens.reserve(4 * npk + 16))) return rc;
    // Copy order on the lane's copy stream (one DMA queue, served in issue order):
    //   pinned caller arrays:   first quarter of the peak masses (needs no host preparation; in flight while the per-spectrum arrays are
    //                           validated and packed) -> per-spectrum blob -> rest of the masses -> intensities.  k_setup_queries + the
    //                           precursor sort need only the blob, so they run under the rest of the masses copy instead of after it.
    //   pageable caller arrays: blob first (the host, not the link, is the bottleneck: nothing is lost by packing before the first DMA),
    //                           then the masses through the staging buffer, then the intensities staged by a helper thread while this
    //                           thread already queues the kernels (chunk_run joins it before k_score is queued).
    cudaStream_t cp = L.copy;
    if ((rc = lane_join_stager(L))) return rc;
    CUDA_TRY(cudaEventRecord(L.ev[0], cp));
    const float* src_m = sp->masses + pk0;
    const float* src_i = sp->intensities + pk0;
    const bool pin_m = npk == 0 || is_pinned(src_m), pin_i = npk == 0 || is_pinned(src_i);
    // Pinned masses are also cut into `nparts` runs of spectra (caller order), each followed by its own event: the counting kernel is queued
    // once per part and starts on part p while part p + 1 is still in flight (it walks its spectra in precursor order either way).
    C.nparts = (pin_m && npk > (1u << 21) && n >= 4096) ? (uint32_t)S->mass_parts : 1u;
    for (uint32_t q = 0; q <= C.nparts; q++) C.part_lo[q] = (uint32_t)((uint64_t)n * q / C.nparts);
    // (clamped: the offsets are only validated by pack() below, and a copy must never leave the caller's array)
    auto part_off = [&](uint32_t q) -> uint64_t { const uint64_t o = sp->peak_offsets[c0 + C.part_lo[q]]; return o < pk0 ? 0 : std::min(o - pk0, npk); };
    // floats of the masses sent ahead of the blob: half of part 0 (a quarter of everything when there is one part)
    const uint64_t npk_a = !pin_m ? 0 : (npk > (1u << 21) ? (C.nparts > 1 ? part_off(1) / 2 : npk / 4) : npk);
    if (npk_a) CUDA_TRY(cudaMemcpyAsync(L.d_masses.p, src_m, 4 * npk_a, cudaMemcpyHostToDevice, cp));
    unsigned char* hs = (unsigned char*)L.h_small.p;
    auto pack = [&]() -> int {   // small per-spectrum arrays -> one pinned blob -> one H2D
        uint32_t* h_off = (uint32_t*)(hs + C.o_off);
        uint32_t pmax = 2, zmax = sv.max_charge;
        for (uint32_t i = 0; i <= n; i++) h_off[i] = (uint32_t)(sp->peak_offsets[c0 + i] - pk0);
        for (uint32_t i = 0; i < n; i++) {
            zmax = std::max<uint32_t>(zmax, sp->precursor_charge[c0 + i]);
            if (sp->peak_offsets[c0 + i + 1] < sp->peak_offsets[c0 + i]) return fail(SAGE_B200_EINVAL, "peak_offsets not monotone at spectrum %llu", (unsigned long long)(c0 + i));
            pmax = std::max(pmax, h_off[i + 1] - h_off[i]);
            if (sp->level && sp->level[c0 + i] != 2)
                return fail(SAGE_B200_ENOTMS2, "internal bug, trying to score a non-MS2 scan! (spectrum %llu has level %u)", (unsigned long long)(c0 + i), sp->level[c0 + i]);
            if (std::isnan(sp->precursor_mz[c0 + i])) return fail(SAGE_B200_ENOPRECURSOR, "missing MS1 precursor for spectrum %llu", (unsigned long long)(c0 + i));
        }
        C.pmax = (pmax + 3) & ~3u;   // multiple of 4 floats: the staged copies in k_score are 16-byte granular
        C.zmax = zmax;
        memcpy(hs + C.o_pmz, sp->precursor_mz + c0, 4 * (size_t)n);
        memcpy(hs + C.o_tic, sp->total_ion_current + c0, 4 * (size_t)n);
        float* h_ilo = (float*)(hs + C.o_ilo);
        float* h_ihi = (float*)(hs + C.o_ihi);
        float* h_rt = (float*)(hs + C.o_rt);
        float* h_ims = (float*)(hs + C.o_ims);
        for (uint32_t i = 0; i < n; i++) {
            h_ilo[i] = sp->isolation_lo ? sp->isolation_lo[c0 + i] : NAN;
            h_ihi[i] = sp->isolation_hi ? sp->isolation_hi[c0 + i] : NAN;
            h_rt[i] = sp->scan_start_time ? sp->scan_start_time[c0 + i] : 0.0f;
            h_ims[i] = sp->inverse_ion_mobility ? sp->inverse_ion_mobility[c0 + i] : NAN;
        }
        memcpy(hs + C.o_chg, sp->precursor_charge + c0, n);
        C.smem = (size_t)(C.pmax + 4) * 8 + (size_t)sv.lcap * 16 + (size_t)sv.kparam * (sizeof(ScoreRec) + 4) + C.pmax + 32;   // peaks, lists, records, order, marks
        if (C.smem + sizeof(ScoreTile) > 200 * 1024) return fail(SAGE_B200_ELIMIT, "spectrum with %u peaks exceeds the shared-memory budget", C.pmax);
        C.nitems = (size_t)n * sv.qmax;
        if (C.nitems > 0x7FFFFFFFull) return fail(SAGE_B200_ELIMIT, "too many queries in one chunk");
        int r;
        if ((r = L.d_queries.reserve(C.nitems * sizeof(QueryDesc)))) return r;
        if ((r = L.d_hits.reserve(C.nitems * sizeof(QueryHits)))) return r;
        if ((r = L.d_keys.reserve(C.nitems * sv.kparam * 8))) return r;
        if ((r = L.d_features.reserve((size_t)n * sv.report_psms * sizeof(FeatureOut)))) return r;
        if ((r = L.d_counts.reserve(4 * (size_t)n))) return r;
        if ((r = L.d_counters.reserve(8 * (C_COUNT + (size_t)sv.qmax)))) return r;   // + one in-use flag per query slot
        if ((r = L.h_counters.reserve(8 * C_COUNT + 32))) return r;
        return 0;
    };
    if ((rc = pack())) {
        cudaStreamSynchronize(cp);   // the masses copy may still be reading the caller's array
        return rc;
    }
    // The blob travels on the SAME stream as the bulk copies. Measured (profiles/r02_final_trace_cfg2.txt): on a second stream it is not served
    // by a second copy engine ahead of the queued bulk copies — it landed after BOTH of them and the whole pipeline started 0.75 ms later.
    CUDA_TRY(cudaMemcpyAsync(L.d_small.p, hs, C.small_bytes, cudaMemcpyHostToDevice, cp));
    CUDA_TRY(cudaEventRecord(L.ev_small, cp));
    if (!pin_m) {
        if (npk && (rc = staged_h2d(L.d_masses.p, src_m, 4 * npk, L.h_masses, *L.pool, cp))) { cudaStreamSynchronize(cp); return rc; }   // pageable caller memory: staged + overlapped
        CUDA_TRY(cudaEventRecord(L.ev_part[0], cp));
    } else {
        uint64_t sent = npk_a;
        for (uint32_t q = 0; q < C.nparts; q++) {
            const uint64_t end = q + 1 == C.nparts ? npk : part_off(q + 1);
            if (end > sent) {
                CUDA_TRY(cudaMemcpyAsync(L.d_masses.as<float>() + sent, src_m + sent, 4 * (end - sent), cudaMemcpyHostToDevice, cp));
                sent = end;
            }
            CUDA_TRY(cudaEventRecord(L.ev_part[q], cp));
        }
    }
    CUDA_TRY(cudaEventRecord(L.ev_masses, cp));   // preliminary scoring can start: it never reads intensities
    if (npk && !pin_i) {
        if ((rc = L.h_intens.reserve(4 * npk))) { cudaStreamSynchronize(cp); return rc; }
        L.stager_rc = 0;
        L.stager_msg[0] = 0;
        const int device = S->device;
        void* dst = L.d_intens.p;
        Lane* lane = &L;
        L.stager = std::thread([lane, device, dst, src_i, npk, cp]() {
            cudaSetDevice(device);
            int r = staged_h2d(dst, src_i, 4 * npk, lane->h_intens, *lane->pool, cp);
            if (r == 0 && (cudaEventRecord(lane->ev_intens, cp) != cudaSuccess || cudaEventRecord(lane->ev[1], cp) != cudaSuccess)) r = fail(SAGE_B200_ECUDA, "event record failed after the staged copy");
            if (r) snprintf(lane->stager_msg, sizeof lane->stager_msg, "%s", g_last_error.c_str());
            lane->stager_rc = r;
        });
    } else {
        if (npk) CUDA_TRY(cudaMemcpyAsync(L.d_intens.p, src_i, 4 * npk, cudaMemcpyHostToDevice, cp));
        CUDA_TRY(cudaEventRecord(L.ev_intens, cp));
        CUDA_TRY(cudaEventRecord(L.ev[1], cp));
    }
    S->last.h2d_bytes += C.small_bytes + 8 * npk;
    C.loaded = true;
    C.force_nlist = C.force_wide = 0;
    C.force_hits = 0;
    C.timed_upload = true;
    L.ran = false;
    L.downloading = false;
    return 0;
}

static int chunk_run(sage_b200_scorer* S, Lane& L, bool dbg) {
    const sage_b200_db* db = S->db;
    const ScorerView& sv = S->sv;
    cudaStream_t st = L.stream;
    ChunkState& C = L.chunk;
    if (!C.loaded) return fail(SAGE_B200_EINVAL, "no spectra resident on the device (call batch_upload first)");
    cudaGetLastError();   // a stale non-sticky error left by another user of the runtime must not be blamed on the launches below
    const uint32_t n = C.n;
    int rc;
    if (dbg) {
        if ((rc = L.d_dbgk.reserve((size_t)n * sv.kparam * 8))) return rc;
        if ((rc = L.d_dbgm.reserve((size_t)n * 16))) return rc;
    }
    BatchView bv{};
    unsigned char* ds = (unsigned char*)L.d_small.p;
    bv.n = n;
    bv.spectrum_base = C.base;
    bv.peak_off = (const uint32_t*)(ds + C.o_off);
    bv.masses = L.d_masses.as<float>();
    bv.intens = L.d_intens.as<float>();
    bv.prec_mz = (const float*)(ds + C.o_pmz);
    bv.prec_charge = (const uint8_t*)(ds + C.o_chg);
    bv.iso_lo = (const float*)(ds + C.o_ilo);
    bv.iso_hi = (const float*)(ds + C.o_ihi);
    bv.tic = (const float*)(ds + C.o_tic);
    bv.rt = (const float*)(ds + C.o_rt);
    bv.ims = (const float*)(ds + C.o_ims);
    bv.queries = L.d_queries.as<QueryDesc>();
    bv.hits = L.d_hits.as<QueryHits>();
    bv.hit_keys = L.d_keys.as<uint64_t>();
    bv.counters = L.d_counters.as<unsigned long long>();

    // kernels of the two lanes never overlap (measured: k_score of one chunk next to k_prelim_narrow of the other slows both); only
    // copies overlap kernels. ev[4] = end of the other lane's k_score (a never-recorded event counts as complete).
    CUDA_TRY(cudaStreamWaitEvent(st, S->lanes[(&L - S->lanes) ^ 1].ev[4], 0));
    CUDA_TRY(cudaStreamWaitEvent(st, L.ev_small, 0));
    CUDA_TRY(cudaEventRecord(L.ev[6], st));
    CUDA_TRY(cudaMemsetAsync(L.d_counters.p, 0, 8 * (C_COUNT + (size_t)sv.qmax), st));
    const bool annotate = sv.annotate && S->frag_dst != nullptr;
    if (annotate) {   // fragment offsets are global across the chunks of one call: start this chunk's counter at what was used so far
        if ((rc = L.d_frags.reserve(S->frag_cap * sizeof(sage_b200_fragment) + 64))) return rc;
        unsigned long long* hbase = (unsigned long long*)L.h_counters.p + C_COUNT + 1;
        *hbase = S->frag_used;
        CUDA_TRY(cudaMemcpyAsync(L.d_counters.as<unsigned long long>() + C_FRAGS, hbase, 8, cudaMemcpyHostToDevice, st));
    }
    // ---- setup: resolve precursor windows. Peptide-centric counting needs LO/HI bound arrays of nfc_max * pmax floats in smem.
    ScorerView svq = sv;
    uint32_t mfc = sv.max_fragment_charge_opt >= 0 ? std::min<uint32_t>(C.zmax, (uint32_t)(sv.max_fragment_charge_opt + 1) & 0xFF) : C.zmax;
    if (mfc < 2) mfc = 2;
    size_t pep_smem = (size_t)(mfc - 1) * (2 * (size_t)C.pmax * sizeof(float) + 2 * LUT_CELLS * sizeof(uint16_t));
    if (mfc - 1 > 8) pep_smem = 200 * 1024;
    if (pep_smem > 96 * 1024) { svq.pep_cap = 0; pep_smem = 0; }
    if (svq.pep_cap == 0) pep_smem = 0;
    uint32_t *sk_in = nullptr, *sk_out = nullptr, *sv_in = nullptr, *sv_out = nullptr;
    int sort_bits = 1;   // keys are PeptideIx < n_pep (spectra without a query sort last within those bits: the order only matters for locality)
    while (sort_bits < 32 && (db->v.n_pep >> sort_bits)) sort_bits++;
    // the top 16 bits are enough for that (two 8-bit radix passes instead of three on a 2M-peptide index: windows span hundreds of peptides)
    const int sort_lo = std::max(0, sort_bits - 16);
    size_t sort_tmp = 0;
    if (S->sort_spectra && n > 1) {  // process spectra in ascending precursor-window order: neighbouring CTAs then touch the same index lines
        if ((rc = L.d_sort.reserve(16 * (size_t)n))) return rc;
        sk_in = L.d_sort.as<uint32_t>(); sk_out = sk_in + n; sv_in = sk_out + n; sv_out = sv_in + n;
        CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, sort_tmp, sk_in, sk_out, sv_in, sv_out, (int)n, sort_lo, sort_bits, st));
        if ((rc = L.d_sorttmp.reserve(sort_tmp + 16))) return rc;
    }
    // Work-list capacities come from what earlier chunks needed (S->nlist_per_spectrum / wide_per_spectrum) or, on a re-run, from the
    // exact need the failed attempt counted: nothing in a chunk waits for the host, so chunks of both lanes queue back to back.
    C.nlist_cap = std::max<uint64_t>(C.force_nlist, (uint64_t)std::ceil(S->nlist_per_spectrum * (double)n) + 4096);
    C.wide_cap = (uint32_t)std::min<uint64_t>(C.nitems, std::max<uint64_t>(C.force_wide, S->wide_per_spectrum > 0.0
                                                                               ? (uint64_t)std::ceil(S->wide_per_spectrum * 1.1 * (double)n) + 64 : 0));
    if ((rc = L.d_nlist.reserve(8 * (C.nlist_cap + 16)))) return rc;
    if ((rc = L.d_nslots.reserve(C.nitems * sizeof(ReplaySlot)))) return rc;
    if (C.wide_cap) {
        if ((rc = L.d_witems.reserve(4 * (size_t)C.wide_cap))) return rc;
        if ((rc = L.d_wlist.reserve((size_t)C.wide_cap * WIDE_LMAX * 8))) return rc;
        if ((rc = L.d_wslots.reserve((size_t)C.wide_cap * sizeof(WideSlot)))) return rc;
    }
    if ((rc = L.d_citems.reserve(4 * C.nitems))) return rc;
    bv.cta_items = L.d_citems.as<uint32_t>();
    bv.nslots = L.d_nslots.as<ReplaySlot>();
    bv.wide_items = L.d_witems.as<uint32_t>();
    bv.wide_cap = C.wide_cap;
    bv.nlist_cap = C.nlist_cap;
    k_setup_queries<<<(n + 127) / 128, 128, 0, st>>>(db->v, svq, bv, sk_in, sv_in);
    CUDA_TRY(cudaGetLastError());
    if (sk_in) {
        CUDA_TRY(cub::DeviceRadixSort::SortPairs(L.d_sorttmp.p, sort_tmp, sk_in, sk_out, sv_in, sv_out, (int)n, sort_lo, sort_bits, st));
        bv.order = sv_out;
    }
    CUDA_TRY(cudaEventRecord(L.ev[2], st));
    if (C.nparts <= 1) CUDA_TRY(cudaStreamWaitEvent(st, L.ev_masses, 0));   // the counting kernels read the peak masses
    uint64_t launches = 1;

    // ---- preliminary scoring. Both kernels are always queued: CTAs whose query belongs to the other kernel (or to nobody) exit at once.
    const size_t rsm = (size_t)sv.kparam * REPLAY_THREADS * 8;
    // the small-block copy of the index: built on first use; never for wide-window (DIA) scorers
    // (nor for open-search tolerances, whose windows exceed the warp kernel's cap: the copy would only cost memory)
    const float ptol_span = std::max(std::fabs(sv.precursor_tol.lo), std::fabs(sv.precursor_tol.hi));
    const bool narrow_tol = ptol_span <= (sv.precursor_tol.kind == 0 ? 2000.0f : sv.precursor_tol.kind == 1 ? 0.2f : 5.0f);   // ppm / percent / Da
    WideIndexView nv{};
    if (S->narrow_index && !sv.wide_window && narrow_tol) {
        if (S->narrow_block == 0 && (rc = narrow_block_for(S))) return rc;
        nv = db_narrow_index(db, S->narrow_block ? S->narrow_block : S->narrow_block_auto, S->narrow_cells_x, S->narrow_block != 0);
    }
    for (uint32_t q = 0; q < C.nparts; q++) {   // one launch per part of the masses copy (a resident batch has one part)
        if (C.nparts > 1) CUDA_TRY(cudaStreamWaitEvent(st, L.ev_part[q], 0));
        const dim3 wgrid((n + WARPQ_WARPS - 1) / WARPQ_WARPS, sv.qmax);
        if (nv.frag != nullptr) k_prelim_narrow_warp<true><<<wgrid, WARPQ_WARPS * 32, 0, st>>>(db->v, svq, bv, L.d_nlist.as<uint64_t>(), C.part_lo[q], C.part_lo[q + 1], nv);
        else k_prelim_narrow_warp<false><<<wgrid, WARPQ_WARPS * 32, 0, st>>>(db->v, svq, bv, L.d_nlist.as<uint64_t>(), C.part_lo[q], C.part_lo[q + 1], nv);
        CUDA_TRY(cudaGetLastError());
        launches += q > 0;
    }
    if (C.nparts > 1) CUDA_TRY(cudaStreamWaitEvent(st, L.ev_masses, 0));
    k_prelim_narrow<<<(unsigned)std::min<uint64_t>(C.nitems, (uint64_t)db->sm_count * 6), PRELIM_THREADS, pep_smem, st>>>(db->v, svq, bv, C.pmax, L.d_nlist.as<uint64_t>(),
                                                                                                                         S->narrow_cta ? nv : WideIndexView{});
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(L.ev[8], st));   // narrow counting kernels done (the open-search kernel, when present, is timed with the replays)
    // narrow windows (<= NARROW_CAP peptides): 32-bit heap keys, half the shared memory
    k_replay<true><<<(unsigned)((C.nitems + REPLAY_THREADS - 1) / REPLAY_THREADS), REPLAY_THREADS, rsm / 2, st>>>(sv, bv, L.d_nlist.as<uint64_t>(), L.d_nslots.as<ReplaySlot>(),
                                                                                                                 (uint32_t)C.nitems, nullptr, n);
    CUDA_TRY(cudaGetLastError());
    launches += 3;
    if (C.wide_cap) {
        const int ctas = (int)std::min<uint64_t>((uint64_t)db->sm_count * WIDE_CTAS, C.wide_cap);
        const WideIndexView wv = db_wide_index(db, sv.wide_tile);   // built on first use (the first open-search chunk of a scorer is a re-run anyway)
        k_prelim_wide<<<ctas, WIDE_THREADS, sizeof(WideSmem), st>>>(db->v, sv, bv, (uint32_t)C.nitems, L.d_wlist.as<uint64_t>(), L.d_wslots.as<WideSlot>(), wv);
        CUDA_TRY(cudaGetLastError());
        if (wv.frag != nullptr) {   // reference-terms work counters of the queries the block-index path counted (no index entry is read)
            k_wide_account<<<(C.wide_cap + 7) / 8, 256, 0, st>>>(db->v, sv, bv);
            CUDA_TRY(cudaGetLastError());
            launches++;
        }
        k_replay<false><<<(unsigned)((C.wide_cap + REPLAY_THREADS - 1) / REPLAY_THREADS), REPLAY_THREADS, rsm, st>>>(
            sv, bv, L.d_wlist.as<uint64_t>(), L.d_wslots.as<WideSlot>(), C.wide_cap, L.d_counters.as<unsigned long long>() + C_WIDE, 0u);
        CUDA_TRY(cudaGetLastError());
        launches += 2;
    }
    CUDA_TRY(cudaEventRecord(L.ev[3], st));

    // ---- candidate scoring + feature assembly (first reader of the intensities)
    if ((rc = lane_join_stager(L))) return rc;   // ev_intens is recorded by the staging thread of a pageable chunk
    CUDA_TRY(cudaStreamWaitEvent(st, L.ev_intens, 0));
    const bool split = S->score_split && !sv.chimera && !annotate && !dbg && S->quick_mode == 0;
    if (split) {
        // hit arena: one entry per scoring task is reserved (sparsely used); sized from what earlier chunks needed, exact on a re-run
        C.hits_cap = std::max<uint64_t>(C.force_hits, (uint64_t)std::ceil((S->hits_per_spectrum > 0.0 ? S->hits_per_spectrum : 4096.0) * (double)n) + 65536);
        if ((rc = L.d_cand.reserve((size_t)n * sv.kparam * sizeof(CandOut)))) return rc;
        if ((rc = L.d_meta.reserve((size_t)n * sizeof(SpecMeta)))) return rc;
        if ((rc = L.d_recs.reserve((size_t)n * sv.kparam * sizeof(ScoreRec)))) return rc;
        if ((rc = L.d_hkey.reserve((size_t)n * sv.kparam * 8))) return rc;
        if ((rc = L.d_emit.reserve((size_t)n * sv.report_psms * 4 + 16))) return rc;
        if ((rc = L.d_hitk.reserve(2 * C.hits_cap + 16))) return rc;
        if ((rc = L.d_hiti.reserve(4 * C.hits_cap + 16))) return rc;
        if ((rc = L.d_hitt.reserve(4 * C.hits_cap + 16))) return rc;
        SplitOut so{};
        so.cand = L.d_cand.as<CandOut>(); so.meta = L.d_meta.as<SpecMeta>(); so.hit_k = L.d_hitk.as<uint16_t>(); so.hit_i = L.d_hiti.as<float>();
        so.hit_t = L.d_hitt.as<float>(); so.hit_cap = C.hits_cap; so.recs = L.d_recs.as<ScoreRec>(); so.hkey = L.d_hkey.as<unsigned long long>(); so.counters = bv.counters;
        // k_score<true> stages the peaks and the hit lists only (no records / order / marks)
        const size_t smem_split = (size_t)(C.pmax + 4) * 8 + (size_t)sv.lcap * 16 + 32;
        k_score<true><<<n, SCORE_THREADS, smem_split, st>>>(db->v, sv, bv, L.d_features.as<FeatureOut>(), L.d_counts.as<uint32_t>(), C.pmax, nullptr, nullptr, nullptr, 0ull, 0u,
                                                            nullptr, so);
        CUDA_TRY(cudaGetLastError());
        const uint64_t nthr = (uint64_t)n * sv.kparam, nrow = (uint64_t)n * sv.report_psms;
        CUDA_TRY(cudaMemsetAsync(L.d_emit.p, 0xFF, 4 * nrow, st));   // rank slots: RANK_EMPTY
        k_fold<<<(unsigned)((nthr + 127) / 128), 128, 0, st>>>(db->v, sv, so, n);
        CUDA_TRY(cudaGetLastError());
        k_features<<<(unsigned)((nthr + 127) / 128), 128, 0, st>>>(sv, n, so, L.d_emit.as<uint32_t>());
        CUDA_TRY(cudaGetLastError());
        k_rows<<<(unsigned)((nrow + 127) / 128), 128, 0, st>>>(db->v, sv, bv, so, L.d_emit.as<uint32_t>(), L.d_counts.as<uint32_t>(), L.d_features.as<FeatureOut>());
        CUDA_TRY(cudaGetLastError());
        launches += 4;
    } else {
        C.hits_cap = 0;
        k_score<false><<<n, SCORE_THREADS, C.smem, st>>>(db->v, sv, bv, L.d_features.as<FeatureOut>(), L.d_counts.as<uint32_t>(), C.pmax,
                                                        dbg ? L.d_dbgk.as<uint64_t>() : nullptr, dbg ? L.d_dbgm.as<uint32_t>() : nullptr,
                                                        annotate ? L.d_frags.as<FragmentOut>() : nullptr, (unsigned long long)S->frag_cap, S->quick_mode,
                                                        S->d_keep.as<uint8_t>(), SplitOut{});
        CUDA_TRY(cudaGetLastError());
        launches++;
    }
    CUDA_TRY(cudaEventRecord(L.ev[4], st));
    CUDA_TRY(cudaMemcpyAsync(L.h_counters.p, L.d_counters.p, 8 * C_COUNT, cudaMemcpyDeviceToHost, st));
    L.launches = launches;
    L.dbg = dbg;
    L.ran = true;
    return 0;
}

static int chunk_download(sage_b200_scorer* S, Lane& L, sage_b200_feature* fdst, uint32_t* cdst) {
    const ScorerView& sv = S->sv;
    cudaStream_t st = L.stream;
    ChunkState& C = L.chunk;
    if (!C.loaded) return fail(SAGE_B200_EINVAL, "no results on the device");
    const uint32_t n = C.n;
    int rc;
    const size_t fbytes = (size_t)n * sv.report_psms * sizeof(sage_b200_feature);
    const bool f_pinned = is_pinned(fdst), c_pinned = is_pinned(cdst);
    if (!f_pinned && (rc = L.h_features.reserve(fbytes))) return rc;
    if (!c_pinned && (rc = L.h_counts.reserve(4 * (size_t)n))) return rc;
    CUDA_TRY(cudaEventRecord(L.ev[7], st));
    CUDA_TRY(cudaMemcpyAsync(f_pinned ? (void*)fdst : L.h_features.p, L.d_features.p, fbytes, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(c_pinned ? (void*)cdst : L.h_counts.p, L.d_counts.p, 4 * (size_t)n, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaEventRecord(L.ev[5], st));
    L.fdst = fdst; L.cdst = cdst; L.f_pinned = f_pinned; L.c_pinned = c_pinned;
    L.downloading = true;
    S->last.d2h_bytes += fbytes + 4 * (size_t)n;
    return 0;
}

// Open search keeps one survivor list (WIDE_LMAX keys, 96 KiB) per wide query and lane. The arena is bounded by a memory budget: a chunk whose
// wide queries would need more is not re-run at its size — the call restarts with chunks small enough for the budget (internal code ERECHUNK).
constexpr int SAGE_B200_ERECHUNK = -100;   // never returned to callers
static uint64_t wide_arena_budget() {
    if (const char* e = getenv("SAGE_B200_WIDE_ARENA_MB")) return std::max<uint64_t>(1, (uint64_t)atoll(e)) << 20;   // (tests use a tiny budget)
    return 8ull << 30;
}
static uint64_t wide_max_chunk(double wide_per_spectrum, uint64_t otherwise) {
    if (!(wide_per_spectrum > 0.0)) return otherwise;
    const double per_spectrum = wide_per_spectrum * 1.1 * (double)WIDE_LMAX * 8.0;
    const uint64_t fit = (uint64_t)std::max(1.0, (double)wide_arena_budget() / per_spectrum);
    return std::min<uint64_t>(32768, std::max<uint64_t>(64, fit));   // open search: at most 32768 spectra per chunk
}

// Waits for everything queued on the lane and folds its counters / timings into S->last.
static int lane_finish(sage_b200_scorer* S, Lane& L) {
    ChunkState& C = L.chunk;
    if (!C.loaded) return 0;
    { const int jrc = lane_join_stager(L); if (jrc) return jrc; }
    CUDA_TRY(cudaStreamSynchronize(L.copy));
    CUDA_TRY(cudaStreamSynchronize(L.copy2));
    for (int attempt = 0;; attempt++) {
        CUDA_TRY(cudaStreamSynchronize(L.stream));
        if (!L.ran) break;
        const unsigned long long* hc = (const unsigned long long*)L.h_counters.p;
        const uint64_t need = hc[C_NLIST_NEED], nw = hc[C_WIDE], nh = C.hits_cap ? hc[C_HITS] : 0;
        if (nh) S->hits_per_spectrum = std::max(S->hits_per_spectrum, 1.25 * (double)nh / (double)C.n);
        if (need <= C.nlist_cap && nw <= C.wide_cap && nh <= C.hits_cap) {   // the chunk fitted its work lists: remember what it needed
            S->nlist_per_spectrum = std::max(S->nlist_per_spectrum, 1.25 * (double)need / (double)C.n);
            S->wide_per_spectrum = std::max(S->wide_per_spectrum, (double)nw / (double)C.n);
            break;
        }
        if (attempt >= 2) return fail(SAGE_B200_ECUDA, "internal error: chunk re-run with exact work-list sizes did not fit");
        S->nlist_per_spectrum = std::max(S->nlist_per_spectrum, 1.25 * (double)need / (double)C.n);
        S->wide_per_spectrum = std::max(S->wide_per_spectrum, (double)nw / (double)C.n);
        if (nw > C.wide_cap && nw * (uint64_t)WIDE_LMAX * 8 > wide_arena_budget() && C.n > wide_max_chunk(S->wide_per_spectrum, 65536))
            return fail(SAGE_B200_ERECHUNK, "open-search chunk of %u spectra needs %llu survivor lists: restarting with smaller chunks", C.n, (unsigned long long)nw);
        // a work list was too small: the queries it could not hold reported no hits. Re-run the chunk with the sizes just counted.
        C.force_nlist = need;
        C.force_wide = nw;
        C.force_hits = nh;
        S->last.chunk_retries++;
        int rc;
        if ((rc = chunk_run(S, L, L.dbg))) return rc;
        if (L.downloading) {
            S->last.d2h_bytes -= (uint64_t)C.n * S->sv.report_psms * sizeof(sage_b200_feature) + 4 * (uint64_t)C.n;
            if ((rc = chunk_download(S, L, L.fdst, L.cdst))) return rc;
        }
    }
    if (S->trace && L.ran && L.downloading) {
        float t[8];
        const int order[8] = {0, 1, 6, 2, 3, 4, 7, 5};
        for (int i = 0; i < 8; i++) cudaEventElapsedTime(&t[i], S->ev_base, L.ev[order[i]]);
        const double now = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - S->t_base).count();
        float tm = 0;
        cudaEventElapsedTime(&tm, S->ev_base, L.ev_masses);
        fprintf(stderr, "[sage_b200 trace] chunk base=%u n=%u | host issue %.3f..%.3f, finished %.3f | dev h2d %.3f..(masses %.3f)..%.3f run %.3f setup-end %.3f prelim-end %.3f score-end %.3f d2h %.3f..%.3f\n",
                C.base, C.n, C.t_issue0, C.t_issue1, now, t[0], tm, t[1], t[2], t[3], t[4], t[5], t[6], t[7]);
    }
    sage_b200_counters& T = S->last;
    float ms;
    if (C.timed_upload) { cudaEventElapsedTime(&ms, L.ev[0], L.ev[1]); T.ms_h2d += ms; T.ms_total += ms; C.timed_upload = false; }
    if (L.ran) {
        const unsigned long long* hc = (const unsigned long long*)L.h_counters.p;
        cudaEventElapsedTime(&ms, L.ev[6], L.ev[2]); T.ms_setup += ms;
        cudaEventElapsedTime(&ms, L.ev[2], L.ev[3]); T.ms_prelim += ms;
        cudaEventElapsedTime(&ms, L.ev[2], L.ev[8]); T.ms_prelim_count += ms;
        cudaEventElapsedTime(&ms, L.ev[3], L.ev[4]); T.ms_score += ms;
        cudaEventElapsedTime(&ms, L.ev[6], L.ev[4]); T.ms_total += ms;
        T.spectra += C.n; T.peaks += C.npk; T.queries += hc[C_QUERIES]; T.tasks += hc[C_TASKS]; T.pages += hc[C_PAGES]; T.entries_scanned += hc[C_ENTRIES];
        T.matched_fragments += hc[C_MATCHED]; T.candidates_scored += hc[C_CANDS]; T.peptide_record_floats += hc[C_PEPFLOATS]; T.psms += hc[C_PSMS];
        T.wide_queries += hc[C_WIDE]; T.pep_queries += hc[C_PEPQ]; T.pep_fallbacks += hc[C_PEPFALLBACK]; T.wide_overflows += hc[C_WOVERFLOW];
        T.d2h_bytes += 2 * 8 * C_COUNT;
        T.kernel_launches += L.launches;
        if (S->sv.annotate && S->frag_dst != nullptr) {
            const uint64_t end = hc[C_FRAGS], begin = S->frag_used;
            const uint64_t lim = std::min<uint64_t>(end, S->frag_cap);
            if (lim > begin) {
                CUDA_TRY(cudaMemcpy(S->frag_dst + begin, L.d_frags.as<sage_b200_fragment>() + begin, (lim - begin) * sizeof(sage_b200_fragment), cudaMemcpyDeviceToHost));
                T.d2h_bytes += (lim - begin) * sizeof(sage_b200_fragment);
            }
            S->frag_used = end;
        }
        L.ran = false;
    }
    if (L.downloading) {
        const size_t fbytes = (size_t)C.n * S->sv.report_psms * sizeof(sage_b200_feature);
        if (!L.f_pinned) memcpy(L.fdst, L.h_features.p, fbytes);
        if (!L.c_pinned) memcpy(L.cdst, L.h_counts.p, 4 * (size_t)C.n);
        cudaEventElapsedTime(&ms, L.ev[7], L.ev[5]); T.ms_d2h += ms; T.ms_total += ms;
        L.downloading = false;
    }
    return 0;
}

static void finish_counters(sage_b200_scorer* S) {
    // SURVEY.md §8(d): B = 8*P + sum_q[8*ceil(log2 N_pep)] + sum_tasks[8*ceil(log2 N_bucket)] + sum_pages[8*ceil(log2 bucket_size) + 8*entries]
    //                    + sum_candidates 4*(2L+2) + 64*n_psm
    sage_b200_counters& L = S->last;
    const DbView& v = S->db->v;
    const uint64_t lp = ceil_log2_u64(v.n_pep), lb = ceil_log2_u64(v.n_bucket), ls = ceil_log2_u64(v.bucket_size);
    L.prelim_bytes = 4 * L.peaks + 8 * lb * L.tasks + 8 * ls * L.pages + 8 * L.entries_scanned;
    L.score_bytes = 4 * L.peaks + 4 * L.peptide_record_floats + 64 * L.psms;
    L.algorithmic_bytes = 8 * L.peaks + 8 * lp * L.queries + 8 * lb * L.tasks + 8 * ls * L.pages + 8 * L.entries_scanned + 4 * L.peptide_record_floats + 64 * L.psms;
}

static int check_spectra(const sage_b200_spectra* sp) {
    if (!sp) return fail(SAGE_B200_EINVAL, "spectra: null");
    if (sp->n && (!sp->peak_offsets || !sp->precursor_mz || !sp->precursor_charge || !sp->total_ion_current)) return fail(SAGE_B200_EINVAL, "spectra: null array");
    if (sp->n && sp->peak_offsets[sp->n] > sp->peak_offsets[0] && (!sp->masses || !sp->intensities)) return fail(SAGE_B200_EINVAL, "spectra: null peak arrays");
    return 0;
}

// Error exit of a batch call: the other lane may still have an H2D reading the caller's arrays or a D2H writing into them. Drain both lanes
// before the error is returned, so the caller may free or reuse its buffers at once; the error message of the failure is preserved.
static int drain_lanes(sage_b200_scorer* S, int rc) {
    const std::string msg = g_last_error;
    for (Lane& L : S->lanes) {
        if (L.stager.joinable()) L.stager.join();   // it reads the caller's arrays
        if (L.copy) cudaStreamSynchronize(L.copy);
        if (L.copy2) cudaStreamSynchronize(L.copy2);
        if (L.stream) cudaStreamSynchronize(L.stream);
        L.chunk.loaded = false; L.ran = false; L.downloading = false;
    }
    cudaGetLastError();
    S->frag_dst = nullptr;
    g_last_error = msg;
    return rc;
}

static int score_batch_chunks(sage_b200_scorer* S, const sage_b200_spectra* sp, sage_b200_feature* features, uint32_t* counts, bool annotate);

extern "C" int sage_b200_score_batch(sage_b200_scorer* S, const sage_b200_spectra* sp, sage_b200_feature* features, uint32_t* counts,
                                     sage_b200_fragment* fragments, uint64_t fragment_capacity, uint64_t* fragments_used) {
    if (!S) return fail(SAGE_B200_EINVAL, "score_batch: null scorer");
    const auto t_call = std::chrono::steady_clock::now();
    int rc = check_spectra(sp);
    if (rc) return rc;
    if (sp->n && (!features || !counts)) return fail(SAGE_B200_EINVAL, "score_batch: null output");
    std::lock_guard<std::mutex> lock(S->mu);
    CUDA_TRY(cudaSetDevice(S->db->device));
    S->last = sage_b200_counters{};
    if (fragments_used) *fragments_used = 0;
    const bool annotate = S->sv.annotate != 0;
    if (annotate && (!fragments || !fragments_used)) return fail(SAGE_B200_EINVAL, "annotate_matches needs a fragments array and fragments_used");
    S->frag_dst = annotate ? fragments : nullptr;
    S->frag_cap = annotate ? fragment_capacity : 0;
    S->frag_used = 0;
    for (Lane& L : S->lanes) {   // a previous call may have failed half-way: make sure nothing is still queued on the lanes
        CUDA_TRY(cudaStreamSynchronize(L.copy));
        CUDA_TRY(cudaStreamSynchronize(L.copy2));
        CUDA_TRY(cudaStreamSynchronize(L.stream));
        L.chunk.loaded = false; L.ran = false; L.downloading = false;
    }
    if (S->trace) { S->t_base = std::chrono::steady_clock::now(); CUDA_TRY(cudaEventRecord(S->ev_base, S->lanes[0].stream)); }
    for (int restart = 0;; restart++) {
        rc = score_batch_chunks(S, sp, features, counts, annotate);
        if (rc != SAGE_B200_ERECHUNK) break;
        drain_lanes(S, rc);   // nothing of this call is kept: the first chunk that needs the re-chunking is the first open-search chunk of the handle
        if (restart >= 3) return fail(SAGE_B200_ELIMIT, "open search: survivor lists do not fit the arena budget even with the smallest chunks");
        const uint64_t retries = S->last.chunk_retries;
        S->last = sage_b200_counters{};
        S->last.chunk_retries = retries + 1;
        S->frag_dst = annotate ? fragments : nullptr;
        S->frag_used = 0;
    }
    if (rc) return drain_lanes(S, rc);
    finish_counters(S);
    S->last.ms_wall = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t_call).count();
    if (annotate) {
        *fragments_used = S->frag_used;
        S->frag_dst = nullptr;
        if (S->frag_used > fragment_capacity)
            return fail(SAGE_B200_ELIMIT, "fragment_capacity %llu too small: %llu fragments matched (features are complete; re-run with a larger array)",
                        (unsigned long long)fragment_capacity, (unsigned long long)S->frag_used);
    }
    return 0;
}

// The chunk loop of score_batch (two pipelined lanes). Returns SAGE_B200_ERECHUNK when an open-search chunk must be cut smaller.
static int score_batch_chunks(sage_b200_scorer* S, const sage_b200_spectra* sp, sage_b200_feature* features, uint32_t* counts, bool annotate) {
    int rc = 0;
    const uint64_t max_peaks = 1ull << 25;
    // Chunks are as large as the staging bounds allow: on cfg2 one 50k chunk computes in 3.6 ms, two 25k chunks in 4.2 ms (the kernels process
    // spectra in precursor order, so a denser chunk shares more index lines). Inside a chunk the intensities copy overlaps setup + preliminary
    // scoring; across chunks (two lanes) the whole H2D of chunk i+1 and the D2H of chunk i-1 overlap the kernels of chunk i.
    const uint64_t max_chunk = wide_max_chunk(S->wide_per_spectrum, 65536);   // open search: one ~100 KB survivor list per query, bounded by the arena budget
    // A short first chunk (first_chunk_pct of the batch, at most 16384 spectra) lets the kernels start while most of the H2D is still in flight.
    uint64_t first = 0, rest = sp->n;
    if (S->pipeline_chunks <= 1 && sp->n >= 16384) { first = std::min<uint64_t>(sp->n * (uint64_t)S->first_chunk_pct / 100, 16384); rest = sp->n - first; }
    const uint64_t nchunks = std::max<uint64_t>((uint64_t)S->pipeline_chunks, (rest + max_chunk - 1) / max_chunk);
    uint64_t target = (rest + nchunks - 1) / nchunks;
    target = std::min<uint64_t>(std::max<uint64_t>(target, 1), max_chunk);
    uint64_t c0 = 0;
    int li = 0;
    while (c0 < sp->n) {
        uint64_t c1 = std::min<uint64_t>(sp->n, c0 + (c0 == 0 && first ? first : target));
        while (c1 > c0 + 1 && sp->peak_offsets[c1] - sp->peak_offsets[c0] > max_peaks) c1 = c0 + (c1 - c0) / 2;
        Lane& L = S->lanes[li];
        if ((rc = lane_finish(S, L))) return rc;   // the chunk that used this lane two iterations ago
        const double ti0 = S->trace ? std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - S->t_base).count() : 0.0;
        if ((rc = chunk_upload(S, L, sp, c0, c1))) return rc;
        if ((rc = chunk_run(S, L, false))) return rc;
        if ((rc = chunk_download(S, L, features + c0 * S->sv.report_psms, counts + c0))) return rc;
        if (S->trace) { L.chunk.t_issue0 = ti0; L.chunk.t_issue1 = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - S->t_base).count(); }
        if (annotate && (rc = lane_finish(S, L))) return rc;   // fragment offsets are global: chunks run one after another
        c0 = c1;
        if (!annotate) li ^= 1;
    }
    for (Lane& L : S->lanes) {
        if ((rc = lane_finish(S, L))) return rc;
        L.chunk.loaded = false;
    }
    return 0;
}

// Pins the calling host thread to the CPUs of the NUMA node the GPU hangs off (sysfs: PCI device -> numa_node -> cpulist), so that the thread's
// pinned staging buffers (first touch) and its cudaMemcpyAsync submissions stay on the socket next to the GPU. Returns the node (>= 0), or -1
// when the topology cannot be read (single-node hosts, containers without sysfs): the thread is left alone.
static int device_numa_cpus(int device, cpu_set_t* want_out);

extern "C" int sage_b200_bind_thread_to_device(int device) {
    // topology lookups (sysfs) are cached per device: score_batch_multi binds its worker threads on every call
    static std::mutex mu;
    static int node_of[64];
    static cpu_set_t cpus_of[64];
    static bool known[64] = {};
    cpu_set_t want;
    int node;
    {
        std::lock_guard<std::mutex> lock(mu);
        if (device >= 0 && device < 64 && known[device]) { node = node_of[device]; want = cpus_of[device]; }
        else {
            node = device_numa_cpus(device, &want);
            if (device >= 0 && device < 64) { known[device] = true; node_of[device] = node; cpus_of[device] = want; }
        }
    }
    if (node < 0) return -1;
    if (pthread_setaffinity_np(pthread_self(), sizeof want, &want) != 0) return -1;
    return node;
}

// NUMA node of the GPU and the CPUs of that node this process may run on (-1: unknown).
static int device_numa_cpus(int device, cpu_set_t* want_out) {
    char bus[64] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, device) != cudaSuccess) { cudaGetLastError(); return -1; }
    for (char* c = bus; *c; c++) *c = (char)tolower(*c);
    char path[256];
    snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
    FILE* f = fopen(path, "r");
    if (!f) return -1;
    int node = -1;
    if (fscanf(f, "%d", &node) != 1) node = -1;
    fclose(f);
    if (node < 0) return -1;
    snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
    f = fopen(path, "r");
    if (!f) return -1;
    char list[4096] = {0};
    const size_t got = fread(list, 1, sizeof list - 1, f);
    fclose(f);
    if (got == 0) return -1;
    // CPUs the process was given when the library was loaded (before any thread was bound by us): never widen that set
    static const cpu_set_t initial = []() { cpu_set_t c; CPU_ZERO(&c); sched_getaffinity(0, sizeof c, &c); return c; }();
    cpu_set_t cur = initial, want;
    CPU_ZERO(&want);
    if (CPU_COUNT(&cur) == 0) return -1;
    int n_set = 0;
    for (char* tok = strtok(list, ",\n"); tok; tok = strtok(nullptr, ",\n")) {   // "0-31,64-95"
        int a = 0, b = 0;
        const int k = sscanf(tok, "%d-%d", &a, &b);
        if (k == 1) b = a;
        if (k < 1) continue;
        for (int c = a; c <= b && c < CPU_SETSIZE; c++)
            if (CPU_ISSET(c, &cur)) { CPU_SET(c, &want); n_set++; }   // never widen the affinity the process was given
    }
    if (n_set == 0) return -1;
    *want_out = want;
    return node;
}

// One process, several GPUs (SURVEY.md §8e): spectra are independent, so the batch is cut into contiguous blocks, block g goes to
// scorers[g] (each bound to its own device and index replica) on its own host thread; Feature.spectrum stays batch-relative.
// No collective and no peer traffic: results land directly in the caller's arrays.
extern "C" int sage_b200_score_batch_multi(sage_b200_scorer* const* scorers, int n_scorers, const sage_b200_spectra* sp, sage_b200_feature* features,
                                           uint32_t* counts) {
    if (!scorers || n_scorers <= 0) return fail(SAGE_B200_EINVAL, "score_batch_multi: no scorers");
    int rc = check_spectra(sp);
    if (rc) return rc;
    if (sp->n && (!features || !counts)) return fail(SAGE_B200_EINVAL, "score_batch_multi: null output");
    for (int g = 0; g < n_scorers; g++) {
        if (!scorers[g]) return fail(SAGE_B200_EINVAL, "score_batch_multi: null scorer %d", g);
        if (scorers[g]->sv.report_psms != scorers[0]->sv.report_psms || scorers[g]->sv.annotate)
            return fail(SAGE_B200_EINVAL, "score_batch_multi: scorers must share report_psms and not annotate matches");
    }
    const uint32_t r = scorers[0]->sv.report_psms;
    std::vector<int> rcs(n_scorers, 0);
    std::vector<std::string> msgs(n_scorers);
    std::vector<std::thread> th;
    for (int g = 0; g < n_scorers; g++) {
        const uint64_t a = sp->n * (uint64_t)g / (uint64_t)n_scorers, b = sp->n * (uint64_t)(g + 1) / (uint64_t)n_scorers;
        th.emplace_back([&, g, a, b]() {
            if (a == b) return;
            sage_b200_bind_thread_to_device(scorers[g]->db->device);   // worker + its staging copies on the GPU's NUMA node
            sage_b200_spectra sub = *sp;   // a view: same arrays, shifted per-spectrum pointers (peak_offsets stay absolute)
            sub.n = b - a;
            sub.peak_offsets = sp->peak_offsets + a;
            sub.precursor_mz = sp->precursor_mz + a;
            sub.precursor_charge = sp->precursor_charge + a;
            sub.isolation_lo = sp->isolation_lo ? sp->isolation_lo + a : nullptr;
            sub.isolation_hi = sp->isolation_hi ? sp->isolation_hi + a : nullptr;
            sub.total_ion_current = sp->total_ion_current + a;
            sub.level = sp->level ? sp->level + a : nullptr;
            sub.scan_start_time = sp->scan_start_time ? sp->scan_start_time + a : nullptr;
            sub.inverse_ion_mobility = sp->inverse_ion_mobility ? sp->inverse_ion_mobility + a : nullptr;
            rcs[g] = sage_b200_score_batch(scorers[g], &sub, features + a * r, counts + a, nullptr, 0, nullptr);
            if (rcs[g]) msgs[g] = g_last_error;
            else
                for (uint64_t i = a; i < b; i++)
                    for (uint32_t k = 0; k < counts[i]; k++) features[i * r + k].spectrum += (uint32_t)a;
        });
    }
    for (auto& x : th) x.join();
    for (int g = 0; g < n_scorers; g++)
        if (rcs[g]) return fail(rcs[g], "scorer %d (device %d): %s", g, scorers[g]->db->device, msgs[g].c_str());
    return 0;
}

// Scorer::quick_score over a batch (scoring.rs:255-298), the prefilter used by runner.rs:143-278: keep[PeptideIx] |= peptide identified.
// prefilter_low_memory != 0: peptides of the report_psms "largest" scored candidates per spectrum (see k_score); == 0: every preliminary hit.
extern "C" int sage_b200_quick_score(sage_b200_scorer* S, const sage_b200_spectra* sp, int prefilter_low_memory, uint8_t* keep) {
    if (!S || !keep) return fail(SAGE_B200_EINVAL, "quick_score: null argument");
    int rc = check_spectra(sp);
    if (rc) return rc;
    std::lock_guard<std::mutex> lock(S->mu);
    CUDA_TRY(cudaSetDevice(S->db->device));
    const size_t npep = S->db->v.n_pep;
    if ((rc = S->d_keep.reserve(npep + 16))) return rc;
    CUDA_TRY(cudaMemset(S->d_keep.p, 0, npep + 16));
    S->last = sage_b200_counters{};
    S->frag_dst = nullptr;
    for (Lane& L : S->lanes) { L.chunk.loaded = false; L.ran = false; L.downloading = false; }
    S->quick_mode = prefilter_low_memory ? 2u : 1u;
    const uint64_t max_peaks = 1ull << 25;
    Lane& L = S->lanes[0];
    for (int restart = 0; restart < 4; restart++) {
        uint64_t c0 = 0;
        rc = 0;
        const uint64_t max_chunk = wide_max_chunk(S->wide_per_spectrum, 32768);
        while (c0 < sp->n && rc == 0) {
            uint64_t c1 = std::min<uint64_t>(sp->n, c0 + max_chunk);
            while (c1 > c0 + 1 && sp->peak_offsets[c1] - sp->peak_offsets[c0] > max_peaks) c1 = c0 + (c1 - c0) / 2;
            if ((rc = chunk_upload(S, L, sp, c0, c1)) == 0 && (rc = chunk_run(S, L, false)) == 0) rc = lane_finish(S, L);
            c0 = c1;
        }
        if (rc != SAGE_B200_ERECHUNK) break;
        drain_lanes(S, rc);   // overflowed attempts leave no keep[] marks (k_score), so the marks of the finished chunks stay valid
        S->quick_mode = prefilter_low_memory ? 2u : 1u;
        CUDA_TRY(cudaMemset(S->d_keep.p, 0, npep + 16));
    }
    if (rc == SAGE_B200_ERECHUNK) rc = fail(SAGE_B200_ELIMIT, "open search: survivor lists do not fit the arena budget even with the smallest chunks");
    S->quick_mode = 0;
    L.chunk.loaded = false;
    if (rc) return drain_lanes(S, rc);
    std::vector<uint8_t> h(npep);
    CUDA_TRY(cudaMemcpy(h.data(), S->d_keep.p, npep, cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < npep; i++) keep[i] |= h[i];
    finish_counters(S);
    return 0;
}

// Device-resident variant of score_batch, split in phases (single chunk, lane 0): upload once, run the kernels any number of
// times (bench.py times this with the inputs already in HBM), download the Feature rows.
extern "C" int sage_b200_batch_upload(sage_b200_scorer* S, const sage_b200_spectra* sp) {
    if (!S) return fail(SAGE_B200_EINVAL, "batch_upload: null scorer");
    int rc = check_spectra(sp);
    if (rc) return rc;
    if (sp->n == 0 || sp->n > (1u << 18) || sp->peak_offsets[sp->n] - sp->peak_offsets[0] > (1ull << 26))
        return fail(SAGE_B200_ELIMIT, "batch_upload takes 1..262144 spectra and at most 2^26 peaks (use score_batch for larger batches)");
    std::lock_guard<std::mutex> lock(S->mu);
    CUDA_TRY(cudaSetDevice(S->db->device));
    S->last = sage_b200_counters{};
    Lane& L = S->lanes[0];
    if ((rc = chunk_upload(S, L, sp, 0, sp->n))) return rc;
    if ((rc = lane_finish(S, L))) return rc;
    L.chunk.nparts = 1;   // everything is resident: batch_run queues one counting launch
    L.chunk.part_lo[1] = L.chunk.n;
    return 0;
}
extern "C" int sage_b200_batch_run(sage_b200_scorer* S) {
    if (!S) return fail(SAGE_B200_EINVAL, "batch_run: null scorer");
    std::lock_guard<std::mutex> lock(S->mu);
    CUDA_TRY(cudaSetDevice(S->db->device));
    const uint64_t h2d = S->last.h2d_bytes;
    S->last = sage_b200_counters{};
    S->last.h2d_bytes = h2d;
    Lane& L = S->lanes[0];
    int rc = chunk_run(S, L, false);
    if (rc) return rc;
    if ((rc = lane_finish(S, L))) {
        if (rc == SAGE_B200_ERECHUNK) rc = fail(SAGE_B200_ELIMIT, "batch_run: the resident batch needs more open-search survivor lists than the arena budget allows; use score_batch");
        return rc;
    }
    finish_counters(S);
    return 0;
}
extern "C" int sage_b200_batch_download(sage_b200_scorer* S, sage_b200_feature* features, uint32_t* counts) {
    if (!S || !features || !counts) return fail(SAGE_B200_EINVAL, "batch_download: null argument");
    std::lock_guard<std::mutex> lock(S->mu);
    CUDA_TRY(cudaSetDevice(S->db->device));
    Lane& L = S->lanes[0];
    int rc = chunk_download(S, L, features, counts);
    if (rc) return rc;
    return lane_finish(S, L);
}

extern "C" int64_t sage_b200_initial_hits(sage_b200_scorer* S, const sage_b200_spectra* sp, uint16_t* matched, uint32_t* peptide, uint8_t* charge,
                                          int8_t* isotope_error, uint64_t cap, uint64_t* matched_peaks, uint64_t* scored_candidates) {
    if (!S) return fail(SAGE_B200_EINVAL, "initial_hits: null scorer");
    int rc = check_spectra(sp);
    if (rc) return rc;
    if (sp->n != 1) return fail(SAGE_B200_EINVAL, "initial_hits takes exactly one spectrum");
    std::lock_guard<std::mutex> lock(S->mu);
    if (cudaSetDevice(S->db->device) != cudaSuccess) return fail(SAGE_B200_ECUDA, "cudaSetDevice failed");
    S->last = sage_b200_counters{};
    std::vector<sage_b200_feature> f(S->sv.report_psms);
    uint32_t cnt = 0;
    Lane& L = S->lanes[0];
    if ((rc = chunk_upload(S, L, sp, 0, 1))) return rc;
    if ((rc = chunk_run(S, L, true))) return rc;
    if ((rc = chunk_download(S, L, f.data(), &cnt))) return rc;
    if ((rc = lane_finish(S, L))) return rc;
    L.chunk.loaded = false;
    std::vector<uint64_t> keys(S->sv.kparam);
    uint32_t meta[4] = {0, 0, 0, 0};
    if (cudaMemcpy(keys.data(), L.d_dbgk.p, 8 * (size_t)S->sv.kparam, cudaMemcpyDeviceToHost) != cudaSuccess ||
        cudaMemcpy(meta, L.d_dbgm.p, 16, cudaMemcpyDeviceToHost) != cudaSuccess)
        return fail(SAGE_B200_ECUDA, "initial_hits: readback failed");
    const uint32_t nk = meta[0];
    for (uint32_t i = 0; i < nk && i < cap; i++) {
        const uint64_t k = keys[i];
        if (matched) matched[i] = (uint16_t)(k >> 48);
        if (peptide) peptide[i] = (uint32_t)(k >> 16);
        if (charge) charge[i] = (uint8_t)(k >> 8);
        if (isotope_error) isotope_error[i] = (int8_t)((int)(k & 0xFF) - 128);
    }
    if (matched_peaks) *matched_peaks = meta[1];
    if (scored_candidates) *scored_candidates = meta[2];
    return (int64_t)nk;
}

// SpectrumProcessor::new(take_top_n, deisotope, min_deisotope_mz).process(..) for a batch of centroided MS2 RawSpectrum (spectrum.rs:271-412).
extern "C" int sage_b200_process_spectra(int device, const sage_b200_processor_params* pr, const sage_b200_raw_spectra* raw, uint64_t* out_peak_offsets,
                                         float* out_masses, float* out_intensities, float* out_tic) {
    if (!pr || !raw || !out_peak_offsets || !out_tic) return fail(SAGE_B200_EINVAL, "process_spectra: null argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(SAGE_B200_ECUDA, "no CUDA device available: sage_b200 has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(SAGE_B200_EINVAL, "device out of range");
    CUDA_TRY(cudaSetDevice(device));
    cudaGetLastError();   // a stale non-sticky error left by another user of the runtime must not be blamed on the launches below
    const uint64_t n = raw->n;
    out_peak_offsets[0] = 0;
    if (n == 0) return 0;
    if (!raw->peak_offsets || !raw->precursor_charge) return fail(SAGE_B200_EINVAL, "process_spectra: null array");
    const uint64_t pk0 = raw->peak_offsets[0], npk = raw->peak_offsets[n] - pk0;
    if (npk && (!raw->mz || !raw->intensity || !out_masses || !out_intensities)) return fail(SAGE_B200_EINVAL, "process_spectra: null peak arrays");
    if (n > 0x7FFFFFFFull || npk > 0xFFFFFFF0ull) return fail(SAGE_B200_ELIMIT, "process_spectra: batch too large");
    std::vector<uint32_t> off(n + 1);
    uint32_t pmax = 1;
    for (uint64_t i = 0; i <= n; i++) off[i] = (uint32_t)(raw->peak_offsets[i] - pk0);
    for (uint64_t i = 0; i < n; i++) {
        if (raw->level && raw->level[i] != 2) return fail(SAGE_B200_ENOTMS2, "process_spectra handles MS2 spectra only (spectrum %llu has level %u)", (unsigned long long)i, raw->level[i]);
        pmax = std::max(pmax, off[i + 1] - off[i]);
    }
    uint32_t p2 = 1;
    while (p2 < pmax) p2 <<= 1;
    const size_t smem = (size_t)p2 * 12 + (size_t)pmax * (5 * 4 + 2) + 32;
    if (smem > 200 * 1024) return fail(SAGE_B200_ELIMIT, "spectrum with %u raw peaks exceeds the shared-memory budget of the preprocessing kernel", pmax);
    void *d_off = nullptr, *d_mz = nullptr, *d_int = nullptr, *d_chg = nullptr, *d_om = nullptr, *d_oi = nullptr, *d_cnt = nullptr, *d_tic = nullptr;
    auto cleanup = [&]() { for (void* p : {d_off, d_mz, d_int, d_chg, d_om, d_oi, d_cnt, d_tic}) if (p) cudaFree(p); };
#define TRY_P(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) { cleanup(); return fail(SAGE_B200_ECUDA, "%s failed: %s", #expr, cudaGetErrorString(_e)); } } while (0)
    TRY_P(cudaMalloc(&d_off, 4 * (n + 1))); TRY_P(cudaMalloc(&d_mz, 4 * npk + 16)); TRY_P(cudaMalloc(&d_int, 4 * npk + 16)); TRY_P(cudaMalloc(&d_chg, n));
    TRY_P(cudaMalloc(&d_om, 4 * npk + 16)); TRY_P(cudaMalloc(&d_oi, 4 * npk + 16)); TRY_P(cudaMalloc(&d_cnt, 4 * n)); TRY_P(cudaMalloc(&d_tic, 4 * n));
    TRY_P(cudaMemcpy(d_off, off.data(), 4 * (n + 1), cudaMemcpyHostToDevice));
    if (npk) { TRY_P(cudaMemcpy(d_mz, raw->mz + pk0, 4 * npk, cudaMemcpyHostToDevice)); TRY_P(cudaMemcpy(d_int, raw->intensity + pk0, 4 * npk, cudaMemcpyHostToDevice)); }
    TRY_P(cudaMemcpy(d_chg, raw->precursor_charge, n, cudaMemcpyHostToDevice));
    ProcParams pp{(uint32_t)std::min<uint64_t>(pr->take_top_n, 0xFFFFFFFFull), pr->deisotope ? 1u : 0u, pr->min_deisotope_mz};
    { int rc_attr = ensure_kernel_attributes(device); if (rc_attr) { cleanup(); return rc_attr; } }
    k_process_ms2<<<(unsigned)n, 32, smem>>>(pp, (uint32_t)n, (const uint32_t*)d_off, (const float*)d_mz, (const float*)d_int, (const uint8_t*)d_chg, pmax, p2,
                                            (float*)d_om, (float*)d_oi, (uint32_t*)d_cnt, (float*)d_tic);
    TRY_P(cudaGetLastError());
    std::vector<uint32_t> cnt(n);
    std::vector<float> om(npk), oi(npk);
    TRY_P(cudaMemcpy(cnt.data(), d_cnt, 4 * n, cudaMemcpyDeviceToHost));
    TRY_P(cudaMemcpy(out_tic, d_tic, 4 * n, cudaMemcpyDeviceToHost));
    if (npk) { TRY_P(cudaMemcpy(om.data(), d_om, 4 * npk, cudaMemcpyDeviceToHost)); TRY_P(cudaMemcpy(oi.data(), d_oi, 4 * npk, cudaMemcpyDeviceToHost)); }
#undef TRY_P
    cleanup();
    uint64_t w = 0;   // compact: spectrum i keeps cnt[i] <= raw count peaks
    for (uint64_t i = 0; i < n; i++) {
        memcpy(out_masses + w, om.data() + off[i], 4 * (size_t)cnt[i]);
        memcpy(out_intensities + w, oi.data() + off[i], 4 * (size_t)cnt[i]);
        w += cnt[i];
        out_peak_offsets[i + 1] = w;
    }
    return 0;
}

// tmt::find_reporter_ions over a batch of ProcessedSpectrum (tmt.rs:193-211, called from tmt::quantify tmt.rs:322-333).
extern "C" int sage_b200_find_reporter_ions(int device, uint64_t n, const uint64_t* peak_offsets, const float* masses, const float* intensities, const float* labels,
                                            uint64_t n_labels, sage_b200_tolerance label_tolerance, float* out) {
    if (n == 0 || n_labels == 0) return 0;
    if (!peak_offsets || !labels || !out) return fail(SAGE_B200_EINVAL, "find_reporter_ions: null argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(SAGE_B200_ECUDA, "no CUDA device available: sage_b200 has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(SAGE_B200_EINVAL, "device out of range");
    if (label_tolerance.kind < 0 || label_tolerance.kind > 2) return fail(SAGE_B200_EINVAL, "bad tolerance kind");
    CUDA_TRY(cudaSetDevice(device));
    const uint64_t pk0 = peak_offsets[0], npk = peak_offsets[n] - pk0;
    if (npk && (!masses || !intensities)) return fail(SAGE_B200_EINVAL, "find_reporter_ions: null peak arrays");
    if (n > 0x7FFFFFFFull || npk > 0xFFFFFFF0ull || n_labels > 4096) return fail(SAGE_B200_ELIMIT, "find_reporter_ions: batch too large");
    std::vector<uint32_t> off(n + 1);
    for (uint64_t i = 0; i <= n; i++) off[i] = (uint32_t)(peak_offsets[i] - pk0);
    void *d_off = nullptr, *d_m = nullptr, *d_i = nullptr, *d_l = nullptr, *d_o = nullptr;
    auto cleanup = [&]() { for (void* p : {d_off, d_m, d_i, d_l, d_o}) if (p) cudaFree(p); };
#define TRY_R(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) { cleanup(); return fail(SAGE_B200_ECUDA, "%s failed: %s", #expr, cudaGetErrorString(_e)); } } while (0)
    TRY_R(cudaMalloc(&d_off, 4 * (n + 1))); TRY_R(cudaMalloc(&d_m, 4 * npk + 16)); TRY_R(cudaMalloc(&d_i, 4 * npk + 16));
    TRY_R(cudaMalloc(&d_l, 4 * n_labels)); TRY_R(cudaMalloc(&d_o, 4 * n * n_labels));
    TRY_R(cudaMemcpy(d_off, off.data(), 4 * (n + 1), cudaMemcpyHostToDevice));
    if (npk) { TRY_R(cudaMemcpy(d_m, masses + pk0, 4 * npk, cudaMemcpyHostToDevice)); TRY_R(cudaMemcpy(d_i, intensities + pk0, 4 * npk, cudaMemcpyHostToDevice)); }
    TRY_R(cudaMemcpy(d_l, labels, 4 * n_labels, cudaMemcpyHostToDevice));
    const uint64_t total = n * n_labels;
    k_find_reporter_ions<<<(unsigned)((total + 255) / 256), 256>>>((uint32_t)n, (uint32_t)n_labels, (const uint32_t*)d_off, (const float*)d_m, (const float*)d_i,
                                                                  (const float*)d_l, Tol{label_tolerance.kind, label_tolerance.lo, label_tolerance.hi}, (float*)d_o);
    TRY_R(cudaGetLastError());
    TRY_R(cudaMemcpy(out, d_o, 4 * total, cudaMemcpyDeviceToHost));
#undef TRY_R
    cleanup();
    return 0;
}

__global__ void k_device_log(int variant, const double* x, uint64_t n, double* out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = variant == 2 ? (double)glog::glibc_log1pf((float)x[i]) : glog::glibc_log_v(x[i], variant);
}
extern "C" int sage_b200_device_log(int device, int variant, const double* x, uint64_t n, double* out) {
    if (n == 0) return 0;
    if (!x || !out || variant < 0 || variant > 2) return fail(SAGE_B200_EINVAL, "device_log: bad argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(SAGE_B200_ECUDA, "no CUDA device available: sage_b200 has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(SAGE_B200_EINVAL, "device out of range");
    CUDA_TRY(cudaSetDevice(device));
    double *dx = nullptr, *dy = nullptr;
    CUDA_TRY(cudaMalloc(&dx, 8 * n));
    if (cudaMalloc(&dy, 8 * n) != cudaSuccess) { cudaFree(dx); return fail(SAGE_B200_ECUDA, "device_log: cudaMalloc failed"); }
    cudaError_t e = cudaMemcpy(dx, x, 8 * n, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        k_device_log<<<(unsigned)((n + 255) / 256), 256>>>(variant, dx, n, dy);
        e = cudaMemcpy(out, dy, 8 * n, cudaMemcpyDeviceToHost);
    }
    cudaFree(dx); cudaFree(dy);
    if (e != cudaSuccess) return fail(SAGE_B200_ECUDA, "device_log failed: %s", cudaGetErrorString(e));
    return 0;
}

extern "C" int sage_b200_counters_get(const sage_b200_scorer* S, sage_b200_counters* out) {
    if (!S || !out) return fail(SAGE_B200_EINVAL, "counters_get: null argument");
    *out = S->last;
    return 0;
}

// Page-locked buffer for a batch that sage_b200_score_batch_multi will cut into n contiguous blocks: block i is first-touched by a thread bound to
// the NUMA node of devices[i] and then the whole region is registered with CUDA, so every GPU DMA-reads its block from the memory next to it
// (one buffer allocated by one thread would sit on a single node and half of the GPUs of a two-socket box would pull across the socket link).
static std::mutex g_blocks_mu;
static std::vector<std::pair<void*, size_t>> g_blocks;
extern "C" void* sage_b200_host_alloc_blocks(size_t bytes, const int* devices, int n_devices) {
    if (bytes == 0) bytes = 16;
    const size_t page = 4096, total = (bytes + page - 1) / page * page;
    void* p = aligned_alloc(page, total);
    if (!p) { fail(SAGE_B200_ECUDA, "host_alloc_blocks: out of memory (%zu bytes)", total); return nullptr; }
    const int n = (devices && n_devices > 0) ? n_devices : 1;
    std::vector<std::thread> th;
    for (int g = 0; g < n; g++) {
        const size_t a = (total / page) * (size_t)g / (size_t)n * page, b = (total / page) * (size_t)(g + 1) / (size_t)n * page;
        th.emplace_back([=]() {
            if (devices) sage_b200_bind_thread_to_device(devices[g]);
            memset((char*)p + a, 0, b - a);   // first touch places the pages
        });
    }
    for (auto& t : th) t.join();
    if (cudaHostRegister(p, total, cudaHostRegisterPortable) != cudaSuccess) {
        cudaGetLastError();
        free(p);
        fail(SAGE_B200_ECUDA, "host_alloc_blocks: cudaHostRegister(%zu) failed", total);
        return nullptr;
    }
    std::lock_guard<std::mutex> lock(g_blocks_mu);
    g_blocks.emplace_back(p, total);
    return p;
}

extern "C" void* sage_b200_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 16, cudaHostAllocPortable) != cudaSuccess) {
        fail(SAGE_B200_ECUDA, "cudaHostAlloc(%zu) failed", bytes);
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
extern "C" void sage_b200_host_free(void* p) {
    if (!p) return;
    {
        std::lock_guard<std::mutex> lock(g_blocks_mu);
        for (size_t i = 0; i < g_blocks.size(); i++)
            if (g_blocks[i].first == p) {
                cudaHostUnregister(p);
                free(p);
                g_blocks.erase(g_blocks.begin() + i);
                return;
            }
    }
    cudaFreeHost(p);
}

extern "C" size_t sage_b200_last_error(char* buf, size_t cap) {
    if (buf && cap) {
        snprintf(buf, cap, "%s", g_last_error.c_str());
    }
    return g_last_error.size();
}

#if SAGE_B200_PHASE_CLOCKS
// variant builds only (not declared in the header): cycles per k_score phase summed over CTAs since the last reset
extern "C" int sage_b200_debug_phase_cycles(unsigned long long* out16, int reset) {
    if (out16) CUDA_TRY(cudaMemcpyFromSymbol(out16, g_phase, sizeof(unsigned long long) * 16));
    if (reset) { unsigned long long z[16] = {0}; CUDA_TRY(cudaMemcpyToSymbol(g_phase, z, sizeof z)); }
    return 0;
}
#endif
