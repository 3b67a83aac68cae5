// C-ABI of libscanfold_b200.so (include/scanfold_b200.h).  Host-side orchestration only: every fold,
// shuffle and accumulation runs in the CUDA kernels of mfe.cu / pf.cu / shuffle.cu.  No CPU fallback.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstddef>
#include <cstring>
#include <dlfcn.h>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/scanfold_b200.h"
#include "device_common.cuh"

namespace {

using namespace sfb;

struct Context {
    bool ready = false;
    int device = -1, n_sm = 0;
    HostParams hp;
    double pf_temperature = -1e9;
    MfeTables *d_mfe = nullptr;
    PfTables *d_pf = nullptr;
    cudaStream_t stream = nullptr;      // stream every launch / copy goes to (own_stream unless sfb_set_stream)
    cudaStream_t own_stream = nullptr;
};

Context g_ctx;
std::mutex g_mu;
thread_local std::string g_err;

int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}

struct CudaError : std::runtime_error {
    using std::runtime_error::runtime_error;
};
#define CK(expr)                                                                                         \
    do {                                                                                                 \
        cudaError_t e__ = (expr);                                                                        \
        if (e__ != cudaSuccess)                                                                          \
            throw CudaError(std::string(#expr) + ": " + cudaGetErrorString(e__));                        \
    } while (0)

// Device-memory cache: a scan plan needs several hundred MB of scratch (shuffles, energies) and callers create one
// plan per record, so freed blocks are kept (up to POOL_CAP bytes) and handed out again instead of going through
// cudaFree / cudaMalloc, which cost tens to hundreds of milliseconds at these sizes.
struct DevPool {
    static constexpr size_t POOL_CAP = (size_t)3 << 30;
    std::mutex mu;
    std::vector<std::pair<size_t, void *>> blocks;   // (bytes, pointer) of cached blocks
    size_t cached = 0;
    void *take(size_t bytes) {
        std::lock_guard<std::mutex> lk(mu);
        int best = -1;
        for (int k = 0; k < (int)blocks.size(); k++)
            if (blocks[k].first >= bytes && blocks[k].first <= 2 * bytes + 4096 &&
                (best < 0 || blocks[k].first < blocks[best].first))
                best = k;
        if (best < 0) return nullptr;
        void *p = blocks[best].second;
        cached -= blocks[best].first;
        blocks.erase(blocks.begin() + best);
        return p;
    }
    bool give(size_t bytes, void *p) {
        std::lock_guard<std::mutex> lk(mu);
        if (cached + bytes > POOL_CAP) return false;
        blocks.emplace_back(bytes, p);
        cached += bytes;
        return true;
    }
    void clear() {
        std::lock_guard<std::mutex> lk(mu);
        for (auto &b : blocks) cudaFree(b.second);
        blocks.clear();
        cached = 0;
    }
};
DevPool &g_pool = *new DevPool;   // never destroyed: buffers may be released during interpreter shutdown

template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t n = 0, cap_bytes = 0;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { release(); }
    void alloc(size_t count) {
        release();
        n = count;
        if (!count) return;
        const size_t bytes = ((count * sizeof(T) + 511) / 512) * 512;
        if (void *q = g_pool.take(bytes)) {
            p = static_cast<T *>(q);
            cap_bytes = bytes;   // the cached block may be larger; only its first `bytes` are used
            return;
        }
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) {   // out of memory: drop the cache and try once more
            cudaGetLastError();
            g_pool.clear();
            CK(cudaMalloc(&p, bytes));
        }
        cap_bytes = bytes;
    }
    void release() {
        if (p) {
            // the block may be handed to another buffer at once: work queued on it must have finished
            if (g_ctx.ready) cudaStreamSynchronize(g_ctx.stream);
            if (!g_pool.give(cap_bytes, p)) cudaFree(p);
        }
        p = nullptr;
        n = cap_bytes = 0;
    }
};

std::string default_par_path() {
    Dl_info info;
    if (dladdr((void *)&sfb_version, &info) && info.dli_fname) {
        std::string so = info.dli_fname;
        size_t k = so.find_last_of('/');
        std::string dir = k == std::string::npos ? "." : so.substr(0, k);
        return dir + "/params/rna_turner2004_besteffort.par";
    }
    return "rna_turner2004_besteffort.par";
}

void upload_mfe_tables() {
    CK(cudaMemcpy(g_ctx.d_mfe, &g_ctx.hp.mfe, sizeof(MfeTables), cudaMemcpyHostToDevice));
    mfe2_upload_tables(g_ctx.hp.mfe);
    mfe3_upload_tables(g_ctx.hp.mfe);
    mfe4_upload_tables(g_ctx.hp.mfe);
    CK(cudaGetLastError());
}

// md.temperature (ScanFold.py:213, ScanFoldFunctions.py:777): every energy table is rescaled from the 37 C values and
// the enthalpies of the parameter file, then the device copies (integer tables of the four MFE kernels, Boltzmann
// factors of the two PF kernels) are replaced.  Work queued on the stream still uses the old tables: drain it first.
void ensure_temperature(double temperature) {
    if (g_ctx.d_pf && g_ctx.pf_temperature == temperature && g_ctx.hp.temperature == temperature) return;
    CK(cudaStreamSynchronize(g_ctx.stream));
    if (g_ctx.hp.temperature != temperature) {
        set_temperature(g_ctx.hp, temperature);
        upload_mfe_tables();
    }
    static PfTables host_pf;
    make_pf_tables(g_ctx.hp, temperature, host_pf);
    if (!g_ctx.d_pf) CK(cudaMalloc(&g_ctx.d_pf, sizeof(PfTables)));
    CK(cudaMemcpy(g_ctx.d_pf, &host_pf, sizeof(PfTables), cudaMemcpyHostToDevice));
    pf2_upload_tables(host_pf);
    g_ctx.pf_temperature = temperature;
}
void ensure_pf_tables(double temperature) { ensure_temperature(temperature); }

int check_model(const sfb_model *m) {
    if (!g_ctx.ready) return fail(SFB_E_STATE, "sfb_init has not been called");
    if (m && !(m->temperature > -273.0 && m->temperature < 1000.0)) return fail(SFB_E_ARG, "temperature out of range");
    return 0;
}

// hard constraints without enforced pairs: only per-nucleotide flags, which the fast kernels fold in
bool hc_is_simple(const uint8_t *hc, size_t n) {
    for (size_t k = 0; k < n; k++)
        if (hc[k] == '(' || hc[k] == ')') return false;
    return true;
}

void encode_host(const uint8_t *ascii, size_t n, std::vector<uint8_t> &codes) {
    codes.resize(n);
    for (size_t k = 0; k < n; k++) codes[k] = (uint8_t)encode_nt(ascii[k]);
}

// ---------------------------------------------------------------------------------------------
constexpr int MFE4_MIN_W = 301;                       // windows the shared-memory kernels do not take (mfe3: <= 300 nt)
constexpr size_t MFE4_SCRATCH_CAP = (size_t)24 << 30;  // HBM the blocked kernel may use for the matrices of one batch

struct FoldWork {  // device scratch for one MFE launch
    DevBuf<int32_t> scratch, scratch2;
    DevBuf<char> scratch4;   // mfe4: C / FML / split matrices of the folds in flight
    int mode = 0;
    size_t per_cta = 0, per_warp2 = 0;
    static bool use4(int W) { return engine() >= 3 && W >= MFE4_MIN_W && mfe4_supports(W); }
    void prepare(int W, int n_fold) {
        if (use4(W)) {
            const size_t per = mfe4_bytes_per_fold(W);
            size_t folds = std::max<size_t>(1, std::min<size_t>((size_t)std::max(n_fold, 1), MFE4_SCRATCH_CAP / per));
            if (folds * per > scratch4.n) scratch4.alloc(folds * per);
            return;
        }
        per_cta = mfe_scratch_ints_per_cta(W, &mode);
        size_t need = per_cta * (size_t)mfe_grid_size(W, g_ctx.n_sm, n_fold);
        if (need > scratch.n) scratch.alloc(need);
        if (mfe2_supports(W) || mfe3_supports(W)) {
            per_warp2 = mfe3_supports(W) ? mfe3_scratch_shorts_per_cta(W) : mfe2_scratch_shorts_per_warp(W);
            size_t rows = (size_t)mfe3_max_ctas(g_ctx.n_sm, W);
            if (mfe2_supports(W)) rows = std::max(rows, (size_t)4 * mfe2_grid_size(g_ctx.n_sm, n_fold));
            size_t need2 = (per_warp2 * rows + 1) / 2;
            if (need2 > scratch2.n) scratch2.alloc(need2);
        }
    }
    static int &engine() {  // sfb_set_engines / SFB_MFE_ENGINE: which energy-only kernel generation may run
        static int e = getenv("SFB_MFE_ENGINE") ? atoi(getenv("SFB_MFE_ENGINE")) : 3;
        return e;
    }
    // energy-only unconstrained folds: int16 warp-per-fold kernel, then the int32 kernel on whatever it flagged
    // any fold above 300 nt (energy only or native with structure, constraints, span): blocked kernel
    void launch4(const MfeLaunch &L, cudaStream_t st, int *n_launch) const {
        const int32_t *hp = reinterpret_cast<const int32_t *>(reinterpret_cast<const char *>(g_ctx.d_mfe) +
                                                              offsetof(MfeTables, hairpin_len));
        launch_mfe4(L, g_ctx.d_mfe, hp, scratch4.p, scratch4.n, nullptr, g_ctx.n_sm, st, n_launch);
    }
    // native fold with enforced pairs / span (everything the fast kernels do not take)
    void launch_general(MfeLaunch L, cudaStream_t st, int *n_launch) const {
        if (use4(L.W)) {
            launch4(L, st, n_launch);
            return;
        }
        fill(L);
        launch_mfe(L, g_ctx.d_mfe, g_ctx.n_sm, st, n_launch);
    }
    void launch_energy_only(MfeLaunch L, cudaStream_t st, int *n_launch) const {
        if (use4(L.W)) {
            launch4(L, st, n_launch);
            return;
        }
        const bool use3 = engine() == 3 && mfe3_supports(L.W), use2 = engine() != 1 && mfe2_supports(L.W) && !L.pair_tbl;
        const bool hc3 = L.hc && L.hc_simple && use3;   // per-nucleotide hard constraints: folded into mfe3
        // mfe3 also traces the structure back and takes stacking pseudo-energies (Deigan)
        if ((use3 || (use2 && !L.sc)) && (!L.hc || hc3) && L.max_span <= 0) {
            MfeLaunch L2 = L;
            L2.gscratch = scratch2.p;
            L2.gscratch_per_cta = (long long)per_warp2;
            if (use3 && (!L.hc || hc3))
                launch_mfe3(L2, g_ctx.d_mfe, g_ctx.n_sm, st, n_launch);
            else
                launch_mfe2(L2, g_ctx.d_mfe, g_ctx.n_sm, st, n_launch);
            L.redo_only = 1;
            static const bool no_redo = getenv("SFB_DEBUG_NO_REDO") != nullptr;  // debugging: leave MFE_REDO markers
            if (no_redo) return;
        }
        fill(L);
        launch_mfe(L, g_ctx.d_mfe, g_ctx.n_sm, st, n_launch);
    }
    void fill(MfeLaunch &L) const {
        L.gscratch = scratch.p;
        L.gscratch_per_cta = (long long)per_cta;
        L.mats_in_gmem = mode;
    }
};

struct PfWork {
    DevBuf<double> scratch;
    size_t per_cta = 0;
    void prepare(int W, int n_fold, bool pairprob = false) {
        per_cta = pf_scratch_doubles_per_cta(W, pairprob);
        size_t need = per_cta * (size_t)pf_grid_size(W, g_ctx.n_sm, n_fold);
        if (need > scratch.n) scratch.alloc(need);
    }
};

// The PF kernels scale every nucleotide by the tables' fixed pf_scale (ViennaRNA's default).  Z of a strongly folding
// window can leave the fp64 range under it (GC-rich windows of 400 nt at 37 C, 300 nt at 10 C): the kernels then
// write a non-finite dG or ED and count the fold.  Such a window is folded again on pf.cu with the scale ViennaRNA's
// exp_params_rescale derives from the window's MFE under the constraints the partition function sees,
// pf_scale = exp(-1.07 mfe / (kT n)); the results do not depend on the scale beyond rounding.  One window per call
// (they are rare); the outputs of `L` are overwritten.  Tables must be at `temperature`.
void pf_rescaled_retry(PfLaunch L, double temperature, FoldWork &fw, cudaStream_t st, const PairProbCommit &pp = {}) {
    DevBuf<int32_t> d_e;
    d_e.alloc(1);
    MfeLaunch M{};
    M.seqs = L.seqs;
    M.hc = L.hc;
    M.hc_simple = L.hc_simple;
    M.sc = L.sc;
    M.n_fold = 1;
    M.W = L.W;
    M.max_span = L.max_span;
    M.e_out = d_e.p;
    if ((!L.hc || L.hc_simple) && L.max_span <= 0)
        fw.launch_energy_only(M, st, nullptr);
    else
        fw.launch_general(M, st, nullptr);
    int32_t e = 0;
    CK(cudaMemcpyAsync(&e, d_e.p, sizeof e, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const double kT = (temperature + 273.15) * 1.98717;
    L.n_fold = 1;
    L.pf_scale = std::exp(-1.07 * e * 10. / (kT * L.W));
    L.n_out_of_range = nullptr;
    launch_pf(L, g_ctx.d_mfe, g_ctx.d_pf, g_ctx.n_sm, st, nullptr, pp);
    CK(cudaGetLastError());
}

}  // namespace

// =================================================================================================
struct sfb_pairprob_table {
    PairProbDense D{};
    int L = 0, first_window = 0, n_windows = 0;   // the record and the shard of windows the table covers
    DevBuf<long long> cells;
    DevBuf<double> paired, prob;
    DevBuf<int32_t> npairs, pi, pj;
    DevBuf<long long> offsets;
    int c_rows = 0;
    long long n_pairs = -1;
};

struct sfb_scan_plan {
    sfb_scan_args a;
    int n_slots = 0;        // n_windows + final
    int chunk = 0;          // windows per chunk
    bool constrained = false;
    bool hc_simple = false;   // the record's constraint line has no '(' ')': the fast kernels take it
    std::vector<uint8_t> parity_host;  // not owned copy avoided: pointer kept in a.parity_shuffles
    DevBuf<uint8_t> seq, hc, nat, shuf, hc_win, parity_ascii;
    DevBuf<int32_t> es1, sc_win;
    DevBuf<int32_t> mfe, nat_unc, shuf_e, e_tmp;
    DevBuf<int16_t> pair_tbl, centroid;
    DevBuf<double> ed, dG;
    DevBuf<int32_t> n_out_of_range;   // PF windows whose Z left the fp64 range in the last run (see pf_rescaled_retry)
    DevBuf<uint8_t> shuf_all;  // only when shuffles_out requested at fetch time (kept per chunk -> full)
    FoldWork fw;
    PfWork pw;
    bool keep_shuffles = false;
    sfb_pairprob_table *pp = nullptr;   // sfb_scan_plan_pairprob: every run adds its regular windows' probabilities
    float stage_ms[4] = {0.f, 0.f, 0.f, 0.f};   // last run: gather + shuffles, MFE, PF, rest
};

struct sfb_partner_table {
    AccumDense D{};
    DevBuf<int32_t> count, first;
    DevBuf<long long> sums;
    DevBuf<int32_t> nparts, c_partner, c_count, c_first;
    DevBuf<long long> offsets, c_sums;
    int c_row0 = 0, c_rows = 0;
    long long n_entries = -1;
    int n_launches = 0;
};

extern "C" {

int sfb_version(void) { return SFB_VERSION; }

const char *sfb_last_error(void) { return g_err.c_str(); }

int sfb_params_besteffort(void) { return g_ctx.ready && g_ctx.hp.besteffort ? 1 : 0; }

int sfb_init(int device_ordinal, const char *par_file_or_null) {
    std::lock_guard<std::mutex> lk(g_mu);
    try {
        std::string path = par_file_or_null && *par_file_or_null ? par_file_or_null : default_par_path();
        try {
            load_params(path, g_ctx.hp);
        } catch (const std::exception &e) {
            return fail(SFB_E_PARAMS, e.what());
        }
        int n_dev = 0;
        cudaError_t e = cudaGetDeviceCount(&n_dev);
        if (e != cudaSuccess || n_dev == 0)
            return fail(SFB_E_CUDA, std::string("no CUDA device available: ") + cudaGetErrorString(e) +
                                        " (this library has no CPU fallback)");
        if (device_ordinal < 0 || device_ordinal >= n_dev) return fail(SFB_E_ARG, "device ordinal out of range");
        CK(cudaSetDevice(device_ordinal));
        cudaDeviceProp prop;
        CK(cudaGetDeviceProperties(&prop, device_ordinal));
        g_ctx.device = device_ordinal;
        g_ctx.n_sm = prop.multiProcessorCount;
        if (!g_ctx.own_stream) CK(cudaStreamCreateWithFlags(&g_ctx.own_stream, cudaStreamNonBlocking));
        if (!g_ctx.stream) g_ctx.stream = g_ctx.own_stream;
        if (!g_ctx.d_mfe) CK(cudaMalloc(&g_ctx.d_mfe, sizeof(MfeTables)));
        upload_mfe_tables();
        g_ctx.pf_temperature = -1e9;
        g_ctx.ready = true;
        ensure_temperature(37.0);
        return 0;
    } catch (const CudaError &e) {
        return fail(SFB_E_CUDA, e.what());
    }
}

void sfb_shutdown(void) {
    std::lock_guard<std::mutex> lk(g_mu);
    g_pool.clear();
    if (g_ctx.d_mfe) cudaFree(g_ctx.d_mfe);
    if (g_ctx.d_pf) cudaFree(g_ctx.d_pf);
    if (g_ctx.own_stream) cudaStreamDestroy(g_ctx.own_stream);
    g_ctx = Context();
}

int sfb_set_engines(int mfe_engine, int pf_engine) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (mfe_engine > 3 || pf_engine > 2) return fail(SFB_E_ARG, "sfb_set_engines: unknown engine");
    if (mfe_engine > 0) FoldWork::engine() = mfe_engine;
    if (pf_engine > 0) pf2_set_enabled(pf_engine >= 2);
    return 0;
}

int sfb_set_stream(void *cuda_stream_or_null) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!g_ctx.ready) return fail(SFB_E_STATE, "sfb_init has not been called");
    g_ctx.stream = cuda_stream_or_null ? (cudaStream_t)cuda_stream_or_null : g_ctx.own_stream;
    return 0;
}

int sfb_deigan(const double *react1, int n, double m, double b, int32_t *es1) {
    if (!react1 || !es1 || n < 0) return fail(SFB_E_ARG, "sfb_deigan: bad argument");
    es1[0] = 0;
    for (int i = 1; i <= n; i++) {
        double v = react1[i] < 0 ? 0. : m * std::log(react1[i] + 1) + b;
        es1[i] = (int32_t)roundf((float)(v * 100.));
    }
    return 0;
}

int sfb_fold_batch(const uint8_t *seqs, int n_seq, int len, const sfb_model *model, const uint8_t *hc,
                   const int32_t *sc, int32_t *e_dcal, int16_t *pair_tbl) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (int rc = check_model(model)) return rc;
    if (!seqs || !e_dcal || n_seq < 0 || len < 1) return fail(SFB_E_ARG, "sfb_fold_batch: bad argument");
    if (len > MAX_W) return fail(SFB_E_RANGE, "fold length exceeds MAX_W");
    if (n_seq == 0) return 0;
    try {
        CK(cudaSetDevice(g_ctx.device));
        ensure_temperature(model ? model->temperature : 37.0);
        std::vector<uint8_t> codes;
        encode_host(seqs, (size_t)n_seq * len, codes);
        DevBuf<uint8_t> d_seq, d_hc;
        DevBuf<int32_t> d_sc, d_e;
        DevBuf<int16_t> d_pt;
        d_seq.alloc(codes.size());
        CK(cudaMemcpyAsync(d_seq.p, codes.data(), codes.size(), cudaMemcpyHostToDevice, g_ctx.stream));
        if (hc) {
            d_hc.alloc((size_t)n_seq * len);
            CK(cudaMemcpyAsync(d_hc.p, hc, (size_t)n_seq * len, cudaMemcpyHostToDevice, g_ctx.stream));
        }
        if (sc) {
            d_sc.alloc((size_t)n_seq * (len + 1));
            CK(cudaMemcpyAsync(d_sc.p, sc, sizeof(int32_t) * (size_t)n_seq * (len + 1), cudaMemcpyHostToDevice,
                               g_ctx.stream));
        }
        d_e.alloc(n_seq);
        if (pair_tbl) d_pt.alloc((size_t)n_seq * len);
        FoldWork fw;
        fw.prepare(len, n_seq);
        MfeLaunch L{};
        L.seqs = d_seq.p;
        L.hc = d_hc.p;
        L.hc_simple = hc && hc_is_simple(hc, (size_t)n_seq * len);
        L.sc = d_sc.p;
        L.n_fold = n_seq;
        L.W = len;
        L.max_span = model ? model->max_bp_span : 0;
        L.e_out = d_e.p;
        L.pair_tbl = d_pt.p;
        fw.launch_energy_only(L, g_ctx.stream, nullptr);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(e_dcal, d_e.p, sizeof(int32_t) * n_seq, cudaMemcpyDeviceToHost, g_ctx.stream));
        if (pair_tbl)
            CK(cudaMemcpyAsync(pair_tbl, d_pt.p, sizeof(int16_t) * (size_t)n_seq * len, cudaMemcpyDeviceToHost,
                               g_ctx.stream));
        CK(cudaStreamSynchronize(g_ctx.stream));
        for (int k = 0; k < n_seq; k++)
            if (e_dcal[k] >= SFB_INF) return fail(SFB_E_CUDA, "traceback failed for fold " + std::to_string(k));
        return 0;
    } catch (const CudaError &e) {
        return fail(SFB_E_CUDA, e.what());
    }
}

int sfb_fold_long(const uint8_t *seq, int n, const sfb_model *model, const uint8_t *hc, int32_t *e_dcal, int32_t *pair_tbl) {
    if (n >= 1 && n < MFE4_MIN_W) {   // short sequences: the batch path (its pair table is 16 bit)
        if (!seq || !e_dcal || !pair_tbl) return fail(SFB_E_ARG, "sfb_fold_long: bad argument");
        std::vector<int16_t> pt16((size_t)n);
        const int rc = sfb_fold_batch(seq, 1, n, model, hc, nullptr, e_dcal, pt16.data());
        for (int k = 0; k < n && !rc; k++) pair_tbl[k] = pt16[k];
        return rc;
    }
    std::lock_guard<std::mutex> lk(g_mu);
    if (int rc = check_model(model)) return rc;
    if (!seq || !e_dcal || !pair_tbl || n < 1) return fail(SFB_E_ARG, "sfb_fold_long: bad argument");
    if (n > SFB_MAX_LONG) return fail(SFB_E_RANGE, "sequence exceeds SFB_MAX_LONG");
    if (!mfe4_supports(n)) return fail(SFB_E_PARAMS, "the loaded energy table does not fit the blocked kernel's packed fields");
    try {
        CK(cudaSetDevice(g_ctx.device));
        ensure_temperature(model ? model->temperature : 37.0);
        cudaStream_t st = g_ctx.stream;
        std::vector<uint8_t> codes;
        encode_host(seq, (size_t)n, codes);
        std::vector<int32_t> hp((size_t)n + 1);   // hairpin initiation by loop size, as load_params extrapolates it
        for (int u = 0; u <= n; u++)
            hp[u] = u <= 30 ? g_ctx.hp.mfe.hairpin[u] : g_ctx.hp.mfe.hairpin[30] + (int)(g_ctx.hp.lxc * std::log(u / 30.));
        DevBuf<uint8_t> d_seq, d_hc;
        DevBuf<int32_t> d_hp, d_e, d_pt;
        DevBuf<char> scratch;
        d_seq.alloc(n);
        d_hp.alloc((size_t)n + 1);
        d_e.alloc(1);
        d_pt.alloc(n);
        scratch.alloc(mfe4_bytes_per_fold(n));
        CK(cudaMemcpyAsync(d_seq.p, codes.data(), n, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(d_hp.p, hp.data(), sizeof(int32_t) * ((size_t)n + 1), cudaMemcpyHostToDevice, st));
        if (hc) {
            d_hc.alloc(n);
            CK(cudaMemcpyAsync(d_hc.p, hc, n, cudaMemcpyHostToDevice, st));
        }
        MfeLaunch L{};
        L.seqs = d_seq.p;
        L.hc = d_hc.p;
        L.hc_simple = hc && hc_is_simple(hc, (size_t)n);
        L.n_fold = 1;
        L.W = n;
        L.max_span = model ? model->max_bp_span : 0;
        L.e_out = d_e.p;
        launch_mfe4(L, g_ctx.d_mfe, d_hp.p, scratch.p, scratch.n, d_pt.p, g_ctx.n_sm, st, nullptr);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(e_dcal, d_e.p, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(pair_tbl, d_pt.p, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (*e_dcal >= SFB_INF) return fail(SFB_E_CUDA, "traceback failed");
        return 0;
    } catch (const CudaError &e) {
        return fail(SFB_E_CUDA, e.what());
    }
}

int sfb_pf_batch(const uint8_t *seqs, int n_seq, int len, const sfb_model *model, const uint8_t *hc,
                 const int32_t *sc, double *ensemble_dG, double *ed, int16_t *centroid_tbl, double *bpp) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (int rc = check_model(model)) return rc;
    if (!seqs || !ed || !ensemble_dG || !centroid_tbl || n_seq < 0 || len < 1)
        return fail(SFB_E_ARG, "sfb_pf_batch: bad argument");
    if (len > MAX_W) return fail(SFB_E_RANGE, "fold length exceeds MAX_W");
    if (n_seq == 0) return 0;
    try {
        CK(cudaSetDevice(g_ctx.device));
        ensure_pf_tables(model ? model->temperature : 37.0);
        std::vector<uint8_t> codes;
        encode_host(seqs, (size_t)n_seq * len, codes);
        DevBuf<uint8_t> d_seq, d_hc;
        DevBuf<int32_t> d_sc;
        DevBuf<double> d_dG, d_ed, d_bpp;
        DevBuf<int16_t> d_cen;
        d_seq.alloc(codes.size());
        CK(cudaMemcpyAsync(d_seq.p, codes.data(), codes.size(), cudaMemcpyHostToDevice, g_ctx.stream));
        if (hc) {
            d_hc.alloc((size_t)n_seq * len);
            CK(cudaMemcpyAsync(d_hc.p, hc, (size_t)n_seq * len, cudaMemcpyHostToDevice, g_ctx.stream));
        }
        if (sc) {
            d_sc.alloc((size_t)n_seq * (len + 1));
            CK(cudaMemcpyAsync(d_sc.p, sc, sizeof(int32_t) * (size_t)n_seq * (len + 1), cudaMemcpyHostToDevice,
                               g_ctx.stream));
        }
        d_dG.alloc(n_seq);
        d_ed.alloc(n_seq);
        d_cen.alloc((size_t)n_seq * len);
        if (bpp) {
            d_bpp.alloc((size_t)n_seq * len * len);
            CK(cudaMemsetAsync(d_bpp.p, 0, sizeof(double) * d_bpp.n, g_ctx.stream));
        }
        PfWork pw;
        pw.prepare(len, n_seq);
        PfLaunch L{};
        L.seqs = d_seq.p;
        L.hc = d_hc.p;
        L.hc_simple = hc && hc_is_simple(hc, (size_t)n_seq * len);
        L.sc = d_sc.p;
        L.n_fold = n_seq;
        L.W = len;
        L.max_span = model ? model->max_bp_span : 0;
        L.dG = d_dG.p;
        L.ed = d_ed.p;
        L.centroid = d_cen.p;
        L.bpp = d_bpp.p;
        L.gscratch = pw.scratch.p;
        L.gscratch_per_cta = (long long)pw.per_cta;
        launch_pf(L, g_ctx.d_mfe, g_ctx.d_pf, g_ctx.n_sm, g_ctx.stream, nullptr);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(ensemble_dG, d_dG.p, sizeof(double) * n_seq, cudaMemcpyDeviceToHost, g_ctx.stream));
        CK(cudaMemcpyAsync(ed, d_ed.p, sizeof(double) * n_seq, cudaMemcpyDeviceToHost, g_ctx.stream));
        CK(cudaMemcpyAsync(centroid_tbl, d_cen.p, sizeof(int16_t) * (size_t)n_seq * len, cudaMemcpyDeviceToHost,
                           g_ctx.stream));
        if (bpp)
            CK(cudaMemcpyAsync(bpp, d_bpp.p, sizeof(double) * d_bpp.n, cudaMemcpyDeviceToHost, g_ctx.stream));
        CK(cudaStreamSynchronize(g_ctx.stream));
        FoldWork fw;   // prepared on the first window that needs the retry
        for (int k = 0, prepared = 0; k < n_seq; k++) {
            if (std::isfinite(ensemble_dG[k]) && std::isfinite(ed[k])) continue;
            if (!prepared++) fw.prepare(len, 1);
            PfLaunch R = L;
            R.seqs = d_seq.p + (size_t)k * len;
            R.hc = hc ? d_hc.p + (size_t)k * len : nullptr;
            R.sc = sc ? d_sc.p + (size_t)k * (len + 1) : nullptr;
            R.dG = d_dG.p + k;
            R.ed = d_ed.p + k;
            R.centroid = d_cen.p + (size_t)k * len;
            R.bpp = bpp ? d_bpp.p + (size_t)k * len * len : nullptr;
            if (bpp) CK(cudaMemsetAsync(R.bpp, 0, sizeof(double) * len * len, g_ctx.stream));
            pf_rescaled_retry(R, model ? model->temperature : 37.0, fw, g_ctx.stream);
            CK(cudaMemcpyAsync(ensemble_dG + k, R.dG, sizeof(double), cudaMemcpyDeviceToHost, g_ctx.stream));
            CK(cudaMemcpyAsync(ed + k, R.ed, sizeof(double), cudaMemcpyDeviceToHost, g_ctx.stream));
            CK(cudaMemcpyAsync(centroid_tbl + (size_t)k * len, R.centroid, sizeof(int16_t) * len, cudaMemcpyDeviceToHost,
                               g_ctx.stream));
            if (bpp)
                CK(cudaMemcpyAsync(bpp + (size_t)k * len * len, R.bpp, sizeof(double) * len * len, cudaMemcpyDeviceToHost,
                                   g_ctx.stream));
            CK(cudaStreamSynchronize(g_ctx.stream));
            if (!(std::isfinite(ensemble_dG[k]) && std::isfinite(ed[k])))
                return fail(SFB_E_RANGE, "partition function of fold " + std::to_string(k) + " out of the fp64 range after rescaling");
        }
        return 0;
    } catch (const CudaError &e) {
        return fail(SFB_E_CUDA, e.what());
    }
}

// -------------------------------------------------------------------------------------------------
int sfb_scan_plan_create(const sfb_scan_args *args, sfb_scan_plan **plan_out) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!args || !plan_out) return fail(SFB_E_ARG, "sfb_scan_plan_create: null argument");
    if (int rc = check_model(&args->model)) return rc;
    const sfb_scan_args &a = *args;
    if (!a.seq || a.L < 1 || a.W < 1 || a.W > a.L || a.step < 1 || a.r < 0 || a.n_windows < 0 || a.first_window < 0)
        return fail(SFB_E_ARG, "sfb_scan_plan_create: bad geometry");
    if (a.W > MAX_W) return fail(SFB_E_RANGE, "window exceeds MAX_W");
    const int total_windows = (a.L - a.W) / a.step + 1;
    if (a.first_window + a.n_windows > total_windows) return fail(SFB_E_ARG, "window range exceeds the record");
    if (a.final_window && (a.n_windows == 0 || a.first_window + a.n_windows != total_windows))
        return fail(SFB_E_ARG, "final_window requires the shard that holds the last regular window");
    if (a.shuffle_type != SFB_SHUFFLE_MONO && a.shuffle_type != SFB_SHUFFLE_DI)
        return fail(SFB_E_ARG, "unknown shuffle type");
    try {
        CK(cudaSetDevice(g_ctx.device));
        ensure_pf_tables(a.model.temperature);
        auto *P = new sfb_scan_plan();
        std::unique_ptr<sfb_scan_plan> guard(P);
        P->a = a;
        P->n_slots = a.n_windows + (a.final_window ? 1 : 0);
        P->constrained = a.hc || a.react;
        P->hc_simple = a.hc && hc_is_simple(a.hc, (size_t)a.L);
        const int n = P->n_slots;
        long long per_win = (long long)std::max(a.r, 1) * a.W;
        long long chunk = (768ll << 20) / std::max(per_win, 1ll);
        chunk = std::max(1ll, std::min<long long>(chunk, 65536));
        P->chunk = (int)std::min<long long>(chunk, std::max(n, 1));
        const size_t cap = (size_t)P->chunk + 1;  // the final-window slot may ride on the last chunk

        std::vector<uint8_t> codes;
        encode_host(a.seq, a.L, codes);
        P->seq.alloc(a.L);
        CK(cudaMemcpyAsync(P->seq.p, codes.data(), a.L, cudaMemcpyHostToDevice, g_ctx.stream));
        if (a.hc) {
            P->hc.alloc(a.L);
            CK(cudaMemcpyAsync(P->hc.p, a.hc, a.L, cudaMemcpyHostToDevice, g_ctx.stream));
            P->hc_win.alloc(cap * a.W);
        }
        if (a.react) {
            std::vector<int32_t> es(a.L + 1);
            sfb_deigan(a.react, a.L, a.shape_m, a.shape_b, es.data());
            P->es1.alloc(a.L + 1);
            CK(cudaMemcpyAsync(P->es1.p, es.data(), sizeof(int32_t) * (a.L + 1), cudaMemcpyHostToDevice, g_ctx.stream));
            CK(cudaStreamSynchronize(g_ctx.stream));
            P->sc_win.alloc(cap * (a.W + 1));
        }
        CK(cudaStreamSynchronize(g_ctx.stream));
        P->nat.alloc(cap * a.W);
        P->shuf.alloc(cap * std::max(a.r, 1) * a.W);
        if (a.parity_shuffles) P->parity_ascii.alloc(cap * std::max(a.r, 1) * a.W);
        P->mfe.alloc(std::max(n, 1));
        P->nat_unc.alloc(std::max(n, 1));
        P->shuf_e.alloc((size_t)std::max(n, 1) * std::max(a.r, 1));
        P->pair_tbl.alloc((size_t)std::max(n, 1) * a.W);
        P->centroid.alloc((size_t)std::max(n, 1) * a.W);
        P->ed.alloc(std::max(n, 1));
        P->dG.alloc(std::max(n, 1));
        P->n_out_of_range.alloc(1);
        CK(cudaMemset(P->centroid.p, 0, sizeof(int16_t) * P->centroid.n));
        CK(cudaMemset(P->ed.p, 0, sizeof(double) * P->ed.n));
        CK(cudaMemset(P->dG.p, 0, sizeof(double) * P->dG.n));
        P->fw.prepare(a.W, (int)cap * std::max(a.r, 1));
        if (a.want_pf) P->pw.prepare(a.W, (int)cap);
        *plan_out = guard.release();
        return 0;
    } catch (const CudaError &e) {
        return fail(SFB_E_CUDA, e.what());
    } catch (const std::bad_alloc &) {
        return fail(SFB_E_CUDA, "out of host memory");
    }
}

void sfb_scan_plan_keep_shuffles(sfb_scan_plan *plan) {
    if (!plan || plan->keep_shuffles) return;
    plan->keep_shuffles = true;
    plan->shuf_all.alloc((size_t)std::max(plan->n_slots, 1) * std::max(plan->a.r, 1) * plan->a.W);
}

__global__ void encode_ascii_kernel(const uint8_t *in, uint8_t *out, long long n) {
    long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    uint8_t c = in[k];
    out[k] = (c == 'A' || c == 'a') ? 1 : (c == 'C' || c == 'c') ? 2 : (c == 'G' || c == 'g') ? 3
           : (c == 'U' || c == 'u' || c == 'T' || c == 't') ? 4 : 0;
}

__global__ void copy_last_slot_kernel(int32_t *mfe, int16_t *pair_tbl, int16_t *centroid, double *ed, double *dG,
                                      int last, int fin, int W, int copy_pf) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k == 0) {
        mfe[fin] = mfe[last];
        if (copy_pf) {
            ed[fin] = ed[last];
            dG[fin] = dG[last];
        }
    }
    if (k < W) {
        pair_tbl[(long long)fin * W + k] = pair_tbl[(long long)last * W + k];
        if (copy_pf) centroid[(long long)fin * W + k] = centroid[(long long)last * W + k];
    }
}

// The slots of the last run whose PF left the fp64 range, again with a per-window scale (pf_rescaled_retry).  A regular
// window is gathered from the record with its constraint slice; the final-window slot either re-ran pf() on the last
// regular window with its soft constraints or copied that window's results (Q5), and follows it.
static void pf_retry_out_of_range(sfb_scan_plan *P) {
    const sfb_scan_args &a = P->a;
    const int n = P->n_slots, W = a.W;
    cudaStream_t st = g_ctx.stream;
    ensure_temperature(a.model.temperature);
    std::vector<double> dG(n), ed(n);
    CK(cudaMemcpyAsync(dG.data(), P->dG.p, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(ed.data(), P->ed.p, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    DevBuf<uint8_t> seq, hc;
    DevBuf<int32_t> sc;
    seq.alloc(W);
    if (a.hc) hc.alloc(W);
    if (a.react) sc.alloc(W + 1);
    for (int s = 0; s < n; s++) {
        if (std::isfinite(dG[s]) && std::isfinite(ed[s])) continue;
        const bool final_slot = a.final_window && s == n - 1;
        if (final_slot && !a.react) {
            copy_last_slot_kernel<<<(W + 127) / 128, 128, 0, st>>>(P->mfe.p, P->pair_tbl.p, P->centroid.p, P->ed.p, P->dG.p,
                                                                   s - 1, s, W, 1);
            CK(cudaGetLastError());
            continue;
        }
        const int w = a.first_window + (final_slot ? s - 1 : s);
        PfLaunch L{};
        launch_gather_windows(P->seq.p, a.L, W, a.step, w, 1, 0, seq.p, st, nullptr);
        L.seqs = seq.p;
        if (a.hc && !final_slot) {
            launch_slice_hc(P->hc.p, a.L, W, a.step, w, 1, 0, hc.p, st, nullptr);
            L.hc = hc.p;
            L.hc_simple = P->hc_simple;
        }
        if (final_slot) {
            launch_slice_sc(P->es1.p, a.L, W, a.step, w, 1, 0, sc.p, st, nullptr);
            L.sc = sc.p;
        }
        L.W = W;
        L.max_span = a.model.max_bp_span;
        L.dG = P->dG.p + s;
        L.ed = P->ed.p + s;
        L.centroid = P->centroid.p + (size_t)s * W;
        L.gscratch = P->pw.scratch.p;
        L.gscratch_per_cta = (long long)P->pw.per_cta;
        PairProbCommit pp{};
        if (P->pp && !final_slot)   // the first attempt added nothing: this run is the window's only contribution
            pp = PairProbCommit{P->pp->cells.p, (long long)w * a.step - P->pp->D.nt0, a.step};
        pf_rescaled_retry(L, a.model.temperature, P->fw, st, pp);
    }
    CK(cudaStreamSynchronize(st));
}

int sfb_scan_plan_run(sfb_scan_plan *P, float *ms_total, float *ms_mfe, int32_t *n_launches_out) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!P) return fail(SFB_E_ARG, "null plan");
    if (!g_ctx.ready) return fail(SFB_E_STATE, "sfb_init has not been called");
    const sfb_scan_args &a = P->a;
    cudaStream_t st = g_ctx.stream;
    int n_launch = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, em0 = nullptr, em1 = nullptr, es0 = nullptr, ep1 = nullptr;
    try {
        CK(cudaSetDevice(g_ctx.device));
        CK(cudaEventCreate(&ev0));
        CK(cudaEventCreate(&ev1));
        CK(cudaEventCreate(&em0));
        CK(cudaEventCreate(&em1));
        CK(cudaEventCreate(&es0));
        CK(cudaEventCreate(&ep1));
        float mfe_ms = 0.f, shuf_ms = 0.f, pf_ms = 0.f;
        CK(cudaEventRecord(ev0, st));
        CK(cudaMemsetAsync(P->n_out_of_range.p, 0, sizeof(int32_t), st));
        const int n = P->n_slots, r = a.r, W = a.W;
        const double t_model = a.model.temperature, t_bg = a.background_temperature != 0. ? a.background_temperature : t_model;
        for (int c0 = 0, cn = 0; c0 < n; c0 += cn) {
            cn = std::min(P->chunk, n - c0);
            if (a.final_window && n - (c0 + cn) == 1) cn++;  // never leave the final-window slot alone
            const bool has_final = a.final_window && (c0 + cn == n);
            const int cn_regular = cn - (has_final ? 1 : 0);
            CK(cudaEventRecord(es0, st));
            // natives (final slot = seq[L-W:L])
            launch_gather_windows(P->seq.p, a.L, W, a.step, a.first_window + c0, cn, has_final, P->nat.p, st, &n_launch);
            // background sequences
            if (r > 0) {
                if (a.parity_shuffles) {
                    size_t bytes = (size_t)cn * r * W;
                    CK(cudaMemcpyAsync(P->parity_ascii.p, a.parity_shuffles + (size_t)c0 * r * W, bytes,
                                       cudaMemcpyHostToDevice, st));
                    encode_ascii_kernel<<<(unsigned)((bytes + 255) / 256), 256, 0, st>>>(P->parity_ascii.p, P->shuf.p,
                                                                                       (long long)bytes);
                    n_launch++;
                } else {
                    ShuffleLaunch S{};
                    S.seq_codes = P->seq.p;
                    S.L = a.L;
                    S.W = W;
                    S.step = a.step;
                    S.r = r;
                    S.type = a.shuffle_type;
                    S.seed = a.seed;
                    S.first_window = a.first_window + c0;
                    S.n_windows = cn;
                    S.final_slot = has_final;
                    S.global_window_base = a.first_window + c0;
                    S.out = P->shuf.p;
                    launch_shuffle(S, st, &n_launch);
                }
                if (P->keep_shuffles)
                    CK(cudaMemcpyAsync(P->shuf_all.p + (size_t)c0 * r * W, P->shuf.p, (size_t)cn * r * W,
                                       cudaMemcpyDeviceToDevice, st));
            }
            CK(cudaEventRecord(em0, st));
            ensure_temperature(t_bg);
            // r background folds per window, energy only (ScanFoldFunctions.py:805-814)
            if (r > 0) {
                MfeLaunch L{};
                L.seqs = P->shuf.p;
                L.n_fold = cn * r;
                L.W = W;
                L.max_span = 0;
                L.e_out = P->shuf_e.p + (size_t)c0 * r;
                P->fw.launch_energy_only(L, st, &n_launch);
            }
            // energy_list[0]: native without constraints / span (ScanFoldFunctions.py:774-789)
            const bool need_unc = P->constrained || a.model.max_bp_span > 0 || t_bg != t_model;
            {
                MfeLaunch L{};
                L.seqs = P->nat.p;
                L.n_fold = cn;
                L.W = W;
                L.max_span = 0;
                L.e_out = P->nat_unc.p + c0;
                L.pair_tbl = need_unc ? nullptr : P->pair_tbl.p + (size_t)c0 * W;
                P->fw.launch_energy_only(L, st, &n_launch);
            }
            ensure_temperature(t_model);
            // native fold with md / hc / sc and structure (ScanFold.py:494-497,512-513,534-541)
            if (need_unc && cn_regular > 0) {
                if (a.hc) launch_slice_hc(P->hc.p, a.L, W, a.step, a.first_window + c0, cn_regular, 0, P->hc_win.p, st, &n_launch);
                if (a.react)
                    launch_slice_sc(P->es1.p, a.L, W, a.step, a.first_window + c0, cn_regular, 0, P->sc_win.p, st, &n_launch);
                MfeLaunch L{};
                L.seqs = P->nat.p;
                L.hc = a.hc ? P->hc_win.p : nullptr;
                L.sc = a.react ? P->sc_win.p : nullptr;
                L.n_fold = cn_regular;
                L.W = W;
                L.max_span = a.model.max_bp_span;
                L.e_out = P->mfe.p + c0;
                L.pair_tbl = P->pair_tbl.p + (size_t)c0 * W;
                L.hc_simple = P->hc_simple;
                if ((!a.hc || P->hc_simple) && a.model.max_bp_span <= 0) {
                    P->fw.launch_energy_only(L, st, &n_launch);   // flags / Deigan only: mfe3 (+ int32 redo)
                } else {
                    P->fw.launch_general(L, st, &n_launch);
                }
            } else if (!need_unc) {
                CK(cudaMemcpyAsync(P->mfe.p + c0, P->nat_unc.p + c0, sizeof(int32_t) * cn, cudaMemcpyDeviceToDevice, st));
            }
            CK(cudaEventRecord(em1, st));
            // partition function of the native window: sees hc (ScanFold.py:512-514) but not sc (:525)
            if (a.want_pf && cn_regular > 0) {
                PfLaunch L{};
                L.seqs = P->nat.p;
                L.hc = a.hc ? P->hc_win.p : nullptr;
                L.hc_simple = P->hc_simple;
                L.n_fold = cn_regular;
                L.W = W;
                L.max_span = a.model.max_bp_span;
                L.dG = P->dG.p + c0;
                L.ed = P->ed.p + c0;
                L.centroid = P->centroid.p + (size_t)c0 * W;
                L.gscratch = P->pw.scratch.p;
                L.gscratch_per_cta = (long long)P->pw.per_cta;
                L.n_out_of_range = P->n_out_of_range.p;
                PairProbCommit pp{};
                if (P->pp) pp = PairProbCommit{P->pp->cells.p, (long long)(a.first_window + c0) * a.step - P->pp->D.nt0, a.step};
                launch_pf(L, g_ctx.d_mfe, g_ctx.d_pf, g_ctx.n_sm, st, &n_launch, pp);
            }
            CK(cudaEventRecord(ep1, st));
            if (has_final) {
                // Q5: the final-window block re-evaluates the STALE fold compound of the last regular window
                const int last = n - 2, fin = n - 1;
                int copy_pf = 1;
                if (a.want_pf && a.react) {  // stale fc now carries the soft constraints: pf() sees them
                    PfLaunch L{};
                    L.seqs = P->nat.p + (size_t)(cn_regular - 1) * W;
                    L.sc = P->sc_win.p + (size_t)(cn_regular - 1) * (W + 1);
                    L.n_fold = 1;
                    L.W = W;
                    L.max_span = a.model.max_bp_span;
                    L.dG = P->dG.p + fin;
                    L.ed = P->ed.p + fin;
                    L.centroid = P->centroid.p + (size_t)fin * W;
                    L.gscratch = P->pw.scratch.p;
                    L.gscratch_per_cta = (long long)P->pw.per_cta;
                    L.n_out_of_range = P->n_out_of_range.p;
                    launch_pf(L, g_ctx.d_mfe, g_ctx.d_pf, g_ctx.n_sm, st, &n_launch);
                    copy_pf = 0;
                }
                copy_last_slot_kernel<<<(W + 127) / 128, 128, 0, st>>>(P->mfe.p, P->pair_tbl.p, P->centroid.p, P->ed.p,
                                                                       P->dG.p, last, fin, W, copy_pf);
                n_launch++;
            }
            CK(cudaEventSynchronize(ep1));
            float ms = 0.f;
            CK(cudaEventElapsedTime(&ms, em0, em1));
            mfe_ms += ms;
            CK(cudaEventElapsedTime(&ms, es0, em0));
            shuf_ms += ms;
            CK(cudaEventElapsedTime(&ms, em1, ep1));
            pf_ms += ms;
        }
        int32_t n_out_of_range = 0;
        if (a.want_pf)
            CK(cudaMemcpyAsync(&n_out_of_range, P->n_out_of_range.p, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        CK(cudaEventRecord(ev1, st));
        CK(cudaEventSynchronize(ev1));
        CK(cudaGetLastError());
        if (n_out_of_range > 0) pf_retry_out_of_range(P);
        float tot = 0.f;
        CK(cudaEventElapsedTime(&tot, ev0, ev1));
        if (ms_total) *ms_total = tot;
        if (ms_mfe) *ms_mfe = mfe_ms;
        P->stage_ms[0] = shuf_ms;
        P->stage_ms[1] = mfe_ms;
        P->stage_ms[2] = pf_ms;
        P->stage_ms[3] = tot - shuf_ms - mfe_ms - pf_ms;
        if (n_launches_out) *n_launches_out = n_launch;
        cudaEventDestroy(ev0);
        cudaEventDestroy(ev1);
        cudaEventDestroy(em0);
        cudaEventDestroy(em1);
        cudaEventDestroy(es0);
        cudaEventDestroy(ep1);
        return 0;
    } catch (const CudaError &e) {
        if (es0) cudaEventDestroy(es0);
        if (ep1) cudaEventDestroy(ep1);
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        if (em0) cudaEventDestroy(em0);
        if (em1) cudaEventDestroy(em1);
        return fail(SFB_E_CUDA, e.what());
    }
}

int sfb_scan_plan_fetch(sfb_scan_plan *P, sfb_scan_out *out) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!P || !out) return fail(SFB_E_ARG, "null argument");
    try {
        CK(cudaSetDevice(g_ctx.device));
        const int n = P->n_slots, W = P->a.W, r = P->a.r;
        cudaStream_t st = g_ctx.stream;
        auto d2h = [&](void *dst, const void *src, size_t bytes) {
            if (dst && bytes) CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st));
        };
        d2h(out->mfe_dcal, P->mfe.p, sizeof(int32_t) * n);
        d2h(out->native_unconstrained_dcal, P->nat_unc.p, sizeof(int32_t) * n);
        d2h(out->shuffle_dcal, P->shuf_e.p, sizeof(int32_t) * (size_t)n * r);
        d2h(out->pair_tbl, P->pair_tbl.p, sizeof(int16_t) * (size_t)n * W);
        d2h(out->centroid_tbl, P->centroid.p, sizeof(int16_t) * (size_t)n * W);
        d2h(out->ed, P->ed.p, sizeof(double) * n);
        d2h(out->ensemble_dG, P->dG.p, sizeof(double) * n);
        if (out->shuffles_out) {
            if (!P->keep_shuffles) return fail(SFB_E_STATE, "shuffles were not kept: call sfb_scan_plan_keep_shuffles before run");
            d2h(out->shuffles_out, P->shuf_all.p, (size_t)n * r * W);
        }
        CK(cudaStreamSynchronize(st));
        if (out->shuffles_out) {
            static const char dec[5] = {'N', 'A', 'C', 'G', 'U'};
            size_t m = (size_t)n * r * W;
            for (size_t k = 0; k < m; k++) out->shuffles_out[k] = (uint8_t)dec[out->shuffles_out[k] % 5];
        }
        if (out->mfe_dcal)
            for (int k = 0; k < n; k++)
                if (out->mfe_dcal[k] >= SFB_INF) return fail(SFB_E_CUDA, "traceback failed in window slot " + std::to_string(k));
        return 0;
    } catch (const CudaError &e) {
        return fail(SFB_E_CUDA, e.what());
    }
}

int sfb_scan_plan_stage_ms(const sfb_scan_plan *plan, float ms[4]) {
    if (!plan || !ms) return fail(SFB_E_ARG, "null argument");
    for (int k = 0; k < 4; k++) ms[k] = plan->stage_ms[k];
    return 0;
}

void sfb_scan_plan_destroy(sfb_scan_plan *plan) {
    std::lock_guard<std::mutex> lk(g_mu);
    delete plan;
}

int sfb_scan(const sfb_scan_args *args, sfb_scan_out *out) {
    sfb_scan_plan *P = nullptr;
    int rc = sfb_scan_plan_create(args, &P);
    if (rc) return rc;
    if (out && out->shuffles_out) sfb_scan_plan_keep_shuffles(P);
    rc = sfb_scan_plan_run(P, nullptr, nullptr, nullptr);
    if (!rc) rc = sfb_scan_plan_fetch(P, out);
    sfb_scan_plan_destroy(P);
    return rc;
}

int sfb_accumulate_begin(const sfb_accum_args *args, sfb_partner_table **out) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!g_ctx.ready) return fail(SFB_E_STATE, "sfb_init has not been called");
    if (!args || !out) return fail(SFB_E_ARG, "null argument");
    const sfb_accum_args &a = *args;
    if (a.L < 1 || a.W < 1 || a.W > a.L || a.step < 1 || a.n_windows < 1 || a.first_window < 0)
        return fail(SFB_E_ARG, "sfb_accumulate_begin: bad geometry");
    if (!a.pair_tbl || !a.z100 || !a.mfe_dcal || !a.ed100) return fail(SFB_E_ARG, "sfb_accumulate_begin: null input");
    if ((long long)(a.first_window + a.n_windows - 1) * a.step + a.W > a.L)
        return fail(SFB_E_ARG, "window range exceeds the record");
    try {
        CK(cudaSetDevice(g_ctx.device));
        cudaStream_t st = g_ctx.stream;
        auto *T = new sfb_partner_table();
        std::unique_ptr<sfb_partner_table> guard(T);
        T->D.W = a.W;
        T->D.nt0 = a.first_window * a.step;
        T->D.n_nt = (a.n_windows - 1) * a.step + a.W;
        const size_t cells = (size_t)T->D.n_nt * (2 * a.W - 1);
        T->count.alloc(cells);
        T->first.alloc(cells);
        T->sums.alloc(6 * cells);
        T->D.count = T->count.p;
        T->D.first_seen = T->first.p;
        T->D.sums = T->sums.p;
        CK(cudaMemsetAsync(T->count.p, 0, cells * 4, st));
        CK(cudaMemsetAsync(T->first.p, 0x7F, cells * 4, st));
        CK(cudaMemsetAsync(T->sums.p, 0, 6 * cells * 8, st));
        DevBuf<int16_t> d_pt;
        DevBuf<int32_t> d_z100, d_mfe, d_ed100;
        const size_t nw = a.n_windows;
        d_pt.alloc(nw * a.W);
        d_z100.alloc(nw);
        d_mfe.alloc(nw);
        d_ed100.alloc(nw);
        CK(cudaMemcpyAsync(d_pt.p, a.pair_tbl, sizeof(int16_t) * nw * a.W, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(d_z100.p, a.z100, sizeof(int32_t) * nw, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(d_mfe.p, a.mfe_dcal, sizeof(int32_t) * nw, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(d_ed100.p, a.ed100, sizeof(int32_t) * nw, cudaMemcpyHostToDevice, st));
        AccumLaunch A{};
        A.step = a.step;
        A.first_window = a.first_window;
        A.n_windows = a.n_windows;
        A.pair_tbl = d_pt.p;
        A.z100 = d_z100.p;
        A.mfe = d_mfe.p;
        A.ed100 = d_ed100.p;
        A.D = T->D;
        launch_accumulate(A, st, &T->n_launches);
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(st));  // the staging buffers above die with this scope
        *out = guard.release();
        return 0;
    } catch (const CudaError &e) {
        return fail(SFB_E_CUDA, e.what());
    }
}

int sfb_accumulate_geometry(const sfb_partner_table *T, int32_t *nt0, int32_t *n_nt) {
    if (!T) return fail(SFB_E_ARG, "null table");
    if (nt0) *nt0 = T->D.nt0;
    if (n_nt) *n_nt = T->D.n_nt;
    return 0;
}

static int check_rows(const sfb_partner_table *T, int row0, int n_rows) {
    if (!T) return fail(SFB_E_ARG, "null table");
    if (row0 < 0 || n_rows < 0 || row0 + n_rows > T->D.n_nt) return fail(SFB_E_ARG, "row range outside the table");
    return 0;
}

int sfb_accumulate_export(sfb_partner_table *T, int row0, int n_rows, int32_t *d_count, int32_t *d_first,
                          int64_t *d_sums) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (int rc = check_rows(T, row0, n_rows)) return rc;
    if (!d_count || !d_first || !d_sums) return fail(SFB_E_ARG, "null buffer");
    try {
        CK(cudaSetDevice(g_ctx.device));
        cudaStream_t st = g_ctx.stream;
        const size_t ncol = 2 * T->D.W - 1, n = (size_t)n_rows * ncol, off = (size_t)row0 * ncol;
        const size_t plane = (size_t)T->D.n_nt * ncol;
        CK(cudaMemcpyAsync(d_count, T->count.p + off, n * 4, cudaMemcpyDeviceToDevice, st));
        CK(cudaMemcpyAsync(d_first, T->first.p + off, n * 4, cudaMemcpyDeviceToDevice, st));
        for (int q = 0; q < 6; q++)
            CK(cudaMemcpyAsync(d_sums + q * n, T->sums.p + q * plane + off, n * 8, cudaMemcpyDeviceToDevice, st));
        CK(cudaStreamSynchronize(st));
        return 0;
    } catch (const CudaError &e) {
        return fail(SFB_E_CUDA, e.what());
    }
}

int sfb_accumulate_merge(sfb_partner_table *T, int row0, int n_rows, const int32_t *d_count, const int32_t *d_first,
                         const int64_t *d_sums) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (int rc = check_rows(T, row0, n_rows)) return rc;
    if (!d_count || !d_first || !d_sums) return fail(SFB_E_ARG, "null buffer");
    try {
        CK(cudaSetDevice(g_ctx.device));
        launch_accum_merge(T->D, row0, n_rows, d_count, d_first, (const long long *)d_sums, g_ctx.stream, &T->n_launches);
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(g_ctx.stream));
        return 0;
    } catch (const CudaError &e) {
        return fail(SFB_E_CUDA, e.what());
    }
}

int sfb_accumulate_compact(sfb_partner_table *T, int row0, int n_rows, int64_t *n_entries) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (int rc = check_rows(T, row0, n_rows)) return rc;
    if (!n_entries) return fail(SFB_E_ARG, "null argument");
    try {
        CK(cudaSetDevice(g_ctx.device));
        cudaStream_t st = g_ctx.stream;
        T->c_row0 = row0;
        T->c_rows = n_rows;
        T->nparts.alloc(std::max(n_rows, 1));
        T->offsets.alloc((size_t)n_rows + 1);
        launch_accum_count(T->D, row0, n_rows, T->nparts.p, T->offsets.p, st, &T->n_launches);
        long long total = 0;
        if (n_rows > 0)
            CK(cudaMemcpyAsync(&total, T->offsets.p + n_rows, 8, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        T->n_entries = total;
        const size_t m = (size_t)std::max<long long>(total, 1);
        T->c_partner.alloc(m);
        T->c_count.alloc(m);
        T->c_first.alloc(m);
        T->c_sums.alloc(6 * m);
        launch_accum_emit(T->D, row0, n_rows, T->offsets.p, T->c_partner.p, T->c_count.p, T->c_first.p, T->c_sums.p, total,
                          st, &T->n_launches);
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(st));
        *n_entries = total;
        return 0;
    } catch (const CudaError &e) {
        return fail(SFB_E_CUDA, e.what());
    }
}

int sfb_accumulate_fetch(sfb_partner_table *T, int32_t *nparts, int32_t *partner, int32_t *count, int32_t *first_seen,
                         int64_t *sums) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!T || T->n_entries < 0) return fail(SFB_E_STATE, "sfb_accumulate_compact has not been called");
    if (!nparts || !partner || !count || !first_seen || !sums) return fail(SFB_E_ARG, "null buffer");
    try {
        CK(cudaSetDevice(g_ctx.device));
        cudaStream_t st = g_ctx.stream;
        const size_t m = (size_t)T->n_entries;
        if (T->c_rows) CK(cudaMemcpyAsync(nparts, T->nparts.p, sizeof(int32_t) * T->c_rows, cudaMemcpyDeviceToHost, st));
        if (m) {
            CK(cudaMemcpyAsync(partner, T->c_partner.p, 4 * m, cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(count, T->c_count.p, 4 * m, cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(first_seen, T->c_first.p, 4 * m, cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(sums, T->c_sums.p, 8 * 6 * m, cudaMemcpyDeviceToHost, st));
        }
        CK(cudaStreamSynchronize(st));
        return 0;
    } catch (const CudaError &e) {
        return fail(SFB_E_CUDA, e.what());
    }
}

int sfb_accumulate_launches(const sfb_partner_table *T) { return T ? T->n_launches : 0; }

// -------------------------------------------------------------------------------------------------
int sfb_pairprob_begin(int32_t L, int32_t W, int32_t step, int32_t first_window, int32_t n_windows,
                       sfb_pairprob_table **out) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!g_ctx.ready) return fail(SFB_E_STATE, "sfb_init has not been called");
    if (!out) return fail(SFB_E_ARG, "null argument");
    if (L < 1 || W < 1 || W > L || step < 1 || n_windows < 1 || first_window < 0)
        return fail(SFB_E_ARG, "sfb_pairprob_begin: bad geometry");
    if (W > MAX_W) return fail(SFB_E_RANGE, "window exceeds MAX_W");
    const int total = (L - W) / step + 1;
    if (first_window + n_windows > total) return fail(SFB_E_ARG, "window range exceeds the record");
    try {
        CK(cudaSetDevice(g_ctx.device));
        auto *T = new sfb_pairprob_table();
        std::unique_ptr<sfb_pairprob_table> guard(T);
        T->L = L;
        T->first_window = first_window;
        T->n_windows = n_windows;
        T->D.nt0 = first_window * step;
        T->D.n_nt = (n_windows - 1) * step + W;
        T->D.W = W;
        T->D.step = step;
        T->D.n_windows = total;
        T->cells.alloc((size_t)T->D.n_nt * W);
        T->D.cells = T->cells.p;
        CK(cudaMemsetAsync(T->cells.p, 0, sizeof(long long) * T->cells.n, g_ctx.stream));
        CK(cudaStreamSynchronize(g_ctx.stream));
        *out = guard.release();
        return 0;
    } catch (const CudaError &e) {
        return fail(SFB_E_CUDA, e.what());
    }
}

int sfb_scan_plan_pairprob(sfb_scan_plan *P, sfb_pairprob_table *T) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!P || !T) return fail(SFB_E_ARG, "null argument");
    const sfb_scan_args &a = P->a;
    if (!a.want_pf) return fail(SFB_E_ARG, "sfb_scan_plan_pairprob: the plan computes no partition function (want_pf = 0)");
    if (a.L != T->L || a.W != T->D.W || a.step != T->D.step)
        return fail(SFB_E_ARG, "sfb_scan_plan_pairprob: record length, window or step differ from the table's");
    if (a.first_window < T->first_window || a.first_window + a.n_windows > T->first_window + T->n_windows)
        return fail(SFB_E_ARG, "sfb_scan_plan_pairprob: the plan's windows lie outside the table's range");
    try {
        CK(cudaSetDevice(g_ctx.device));
        P->pw.prepare(a.W, P->chunk + 1, true);   // pf2 stages the probabilities of a fold in its scratch
        P->pp = T;
        return 0;
    } catch (const CudaError &e) {
        return fail(SFB_E_CUDA, e.what());
    }
}

static int check_pp_rows(const sfb_pairprob_table *T, int row0, int n_rows) {
    if (!T) return fail(SFB_E_ARG, "null table");
    if (row0 < 0 || n_rows < 0 || row0 + n_rows > T->D.n_nt) return fail(SFB_E_ARG, "row range outside the table");
    return 0;
}

int sfb_pairprob_export(sfb_pairprob_table *T, int row0, int n_rows, int64_t *d_rows) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (int rc = check_pp_rows(T, row0, n_rows)) return rc;
    if (!d_rows) return fail(SFB_E_ARG, "null buffer");
    try {
        CK(cudaSetDevice(g_ctx.device));
        const size_t n = (size_t)n_rows * T->D.W;
        if (n)
            CK(cudaMemcpyAsync(d_rows, T->cells.p + (size_t)row0 * T->D.W, n * 8, cudaMemcpyDeviceToDevice, g_ctx.stream));
        CK(cudaStreamSynchronize(g_ctx.stream));
        return 0;
    } catch (const CudaError &e) {
        return fail(SFB_E_CUDA, e.what());
    }
}

int sfb_pairprob_merge(sfb_pairprob_table *T, int row0, int n_rows, const int64_t *d_rows) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (int rc = check_pp_rows(T, row0, n_rows)) return rc;
    if (!d_rows) return fail(SFB_E_ARG, "null buffer");
    try {
        CK(cudaSetDevice(g_ctx.device));
        launch_pairprob_merge(T->D, row0, n_rows, (const long long *)d_rows, g_ctx.stream, nullptr);
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(g_ctx.stream));
        return 0;
    } catch (const CudaError &e) {
        return fail(SFB_E_CUDA, e.what());
    }
}

int sfb_pairprob_compact(sfb_pairprob_table *T, int row0, int n_rows, double cutoff, int64_t *n_pairs) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (int rc = check_pp_rows(T, row0, n_rows)) return rc;
    if (!n_pairs) return fail(SFB_E_ARG, "null argument");
    if (!(cutoff > 0.)) return fail(SFB_E_ARG, "sfb_pairprob_compact: cutoff must be positive");
    try {
        CK(cudaSetDevice(g_ctx.device));
        cudaStream_t st = g_ctx.stream;
        T->c_rows = n_rows;
        T->paired.alloc(std::max(n_rows, 1));
        T->npairs.alloc(std::max(n_rows, 1));
        T->offsets.alloc((size_t)n_rows + 1);
        launch_pairprob_count(T->D, row0, n_rows, cutoff, T->paired.p, T->npairs.p, T->offsets.p, st, nullptr);
        long long total = 0;
        if (n_rows > 0) CK(cudaMemcpyAsync(&total, T->offsets.p + n_rows, 8, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        const size_t m = (size_t)std::max<long long>(total, 1);
        T->pi.alloc(m);
        T->pj.alloc(m);
        T->prob.alloc(m);
        if (total > 0)
            launch_pairprob_emit(T->D, row0, n_rows, cutoff, T->offsets.p, T->pi.p, T->pj.p, T->prob.p, st, nullptr);
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(st));
        T->n_pairs = total;
        *n_pairs = total;
        return 0;
    } catch (const CudaError &e) {
        return fail(SFB_E_CUDA, e.what());
    }
}

int sfb_pairprob_fetch(sfb_pairprob_table *T, double *paired, int32_t *i, int32_t *j, double *p) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!T || T->n_pairs < 0) return fail(SFB_E_STATE, "sfb_pairprob_compact has not been called");
    if ((T->c_rows && !paired) || (T->n_pairs && (!i || !j || !p))) return fail(SFB_E_ARG, "null buffer");
    try {
        CK(cudaSetDevice(g_ctx.device));
        cudaStream_t st = g_ctx.stream;
        const size_t m = (size_t)T->n_pairs;
        if (T->c_rows) CK(cudaMemcpyAsync(paired, T->paired.p, sizeof(double) * T->c_rows, cudaMemcpyDeviceToHost, st));
        if (m) {
            CK(cudaMemcpyAsync(i, T->pi.p, 4 * m, cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(j, T->pj.p, 4 * m, cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(p, T->prob.p, 8 * m, cudaMemcpyDeviceToHost, st));
        }
        CK(cudaStreamSynchronize(st));
        return 0;
    } catch (const CudaError &e) {
        return fail(SFB_E_CUDA, e.what());
    }
}

void sfb_pairprob_free(sfb_pairprob_table *T) {
    std::lock_guard<std::mutex> lk(g_mu);
    delete T;
}

void sfb_accumulate_free(sfb_partner_table *T) {
    std::lock_guard<std::mutex> lk(g_mu);
    delete T;
}

}  // extern "C"
