// C ABI of the engine (include/triceratops_b200.h): device context, light-curve upload,
// staging of host columns, kernel launches, result read-back.  No CPU compute path: every entry
// point fails with TRI_ENODEVICE / TRI_ECUDA when there is no usable GPU.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <numeric>
#include <string>
#include <thread>
#include <vector>

#include "../../include/triceratops_b200.h"
#include "tri_kernels.cuh"
#include "tri_sampler.cuh"

namespace {

using namespace tri;

// Error text: per calling thread (the thread that got the error code reads its own message even
// when other threads use the engine in between) with the engine's most recent error as the
// answer for a thread that has none of its own.
thread_local std::string g_err;
std::mutex g_err_mutex;
std::string g_err_engine;

int fail(int code, const std::string& msg) {
    g_err = msg;
    std::lock_guard<std::mutex> lock(g_err_mutex);
    g_err_engine = msg;
    return code;
}

#define CU(call)                                                                         \
    do {                                                                                 \
        cudaError_t e_ = (call);                                                         \
        if (e_ != cudaSuccess)                                                           \
            return fail(TRI_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
    } while (0)

// grow-only device arena, bump-allocated per call
struct Arena {
    char* base = nullptr;
    size_t cap = 0, used = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return TRI_OK;
        if (base) CU(cudaFree(base));
        base = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 4;
        CU(cudaMalloc(&base, want));
        cap = want;
        return TRI_OK;
    }
    void reset() { used = 0; }
    template <typename T>
    T* take(size_t n) {
        size_t off = (used + 255) & ~size_t(255);
        used = off + n * sizeof(T);
        return reinterpret_cast<T*>(base + off);
    }
};

// grow-only pinned host arena: pageable caller columns are copied here by a few host threads so
// that their transfer is a true asynchronous DMA (a cudaMemcpyAsync from pageable memory keeps
// the calling thread busy for the whole transfer, at a fraction of the PCIe rate)
struct HostArena {
    char* base = nullptr;
    size_t cap = 0, used = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return TRI_OK;
        if (base) CU(cudaFreeHost(base));
        base = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 8;
        CU(cudaHostAlloc(&base, want, cudaHostAllocDefault));
        cap = want;
        return TRI_OK;
    }
    void reset() { used = 0; }
    char* take(size_t bytes) {
        size_t off = (used + 255) & ~size_t(255);
        if (off + bytes > cap) return nullptr;
        used = off + bytes;
        return base + off;
    }
};

constexpr size_t kPinnedLimit = (size_t)3 << 30;   // per slot; larger calls copy the rest directly
constexpr size_t kPinnedMinCopy = (size_t)256 << 10;

int host_threads() {
    static int n = [] {
        const char* e = std::getenv("TRI_B200_HOST_THREADS");
        int v = e ? std::atoi(e) : 0;
        if (v <= 0) {   // half the cores, shared between the ranks of the node
            const char* w = std::getenv("LOCAL_WORLD_SIZE");
            int ranks = std::max(1, w ? std::atoi(w) : 1);
            v = (int)std::thread::hardware_concurrency() / (2 * ranks);
        }
        return std::max(1, std::min(v, 8));
    }();
    return n;
}

void parallel_memcpy(void* dst, const void* src, size_t bytes) {
    int T = host_threads();
    if (T <= 1 || bytes < ((size_t)2 << 20)) {
        std::memcpy(dst, src, bytes);
        return;
    }
    size_t chunk = ((bytes / T) + 4095) & ~size_t(4095);
    std::vector<std::thread> th;
    for (int t = 1; t < T; ++t) {
        size_t lo = std::min(bytes, chunk * t), hi = std::min(bytes, chunk * (t + 1));
        if (hi > lo)
            th.emplace_back([=] { std::memcpy((char*)dst + lo, (const char*)src + lo, hi - lo); });
    }
    std::memcpy(dst, src, std::min(bytes, chunk));
    for (auto& x : th) x.join();
}

bool is_pinned(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeManaged;
}

constexpr int kSlots = TRI_MAX_INFLIGHT;

// One evaluation in flight: its device scratch, its staged columns, and the pinned landing zone
// of its small result record.  Slot kSlots is the private one of the synchronous helpers
// (tri_lnl_*, tri_simulate_*, tri_log_mean_exp).
struct Slot {
    Arena scratch;   // kernel scratch (a, p, lnl, items, partials)
    Arena staging;   // device copies of host columns
    HostArena pinned;   // pinned copies of pageable host columns, on their way to `staging`
    unsigned long long* d_counters = nullptr;  // [8]
    unsigned long long* h_counters = nullptr;  // pinned [8]
    LsePartial* d_lse_out = nullptr;           // [2], then s2 and T of the two branches
    LsePartial* h_lse_out = nullptr;           // pinned, same layout (kLseOutBytes)
    unsigned int* d_mom_done = nullptr;        // moments_kernel's block counter
    unsigned int* d_post_done = nullptr;       // [2] posterior_sums_kernel's block counters
    int64_t* d_post_idx[2] = {nullptr, nullptr};   // [g.post_cap] posterior samples per branch
    int64_t* h_post_idx[2] = {nullptr, nullptr};   // pinned landing zone, same size
    TopkState* d_topk = nullptr;               // [2]
    TopkState* h_topk = nullptr;               // pinned [2]
    unsigned int* d_hist16 = nullptr;          // [2][kTopkBins], zero between calls
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};   // geometry | lnl | finalize
    cudaEvent_t copied = nullptr, done = nullptr;
    int launches = 0;
    // the call in flight
    int64_t ticket = 0;   // 0 = free
    int branches = 0;     // 1 = TP-type, 2 = EB-type
    int64_t N = 0;
    bool moments = false; // tri_set_moments at submission: s2 follows the records
    double s2[2] = {NAN, NAN};
    int64_t post_K = 0;   // tri_set_posterior at submission (0: off)
    unsigned long long post_seed = 0, post_stream = 0;
    double post_T[2] = {NAN, NAN};
    bool host = false;    // host-buffer call: best-draw candidates are sorted in tri_wait
    bool want_top[2] = {false, false};
    tri_result want[2];   // the caller's records: its pointers go back into the results
    const double* lnl[2] = {nullptr, nullptr};   // device lnL arrays of the call
    // host-buffer calls: what tri_wait copies into the caller's (pageable) buffers -- a
    // cudaMemcpyAsync into pageable memory would make tri_submit_* wait for the kernels
    int64_t* h_tidx[2] = {nullptr, nullptr};     // pinned landing zone of the candidates
    double* h_tval[2] = {nullptr, nullptr};
    int64_t h_top_cap = 0;
    const double* d_out_lnl[2] = {nullptr, nullptr};    // device copies of lnL_out / mask_out
    const uint8_t* d_out_mask[2] = {nullptr, nullptr};
};

struct Ctx {
    bool ready = false;
    int device = -1;
    int sm_count = 0;
    int lnl_blocks_per_sm = 0;
    bool count_work = false;   // tri_set_counting: run the instantiation with work counters
    bool moments = false;      // tri_set_moments: second moment of the weights per branch
    size_t lnl_smem = 0;   // dynamic shared memory used to stage the light curve (0 = none)
    cudaStream_t stream = nullptr;        // kernels and result read-back
    cudaStream_t copy_stream = nullptr;   // host columns -> staging (overlaps the kernels)
    double* d_tae = nullptr;
    OrbitTable tab{};
    // light curve
    bool have_lc = false;
    double *d_time = nullptr, *d_flux = nullptr, *d_prefix = nullptr, *d_weight = nullptr;
    int* d_perm = nullptr;   // sorted stamp -> caller's stamp
    size_t lc_cap = 0;
    LightCurve lc{};
    CadenceTable cad{};   // n > 1: mixed cadence (lnl_kernel<*, true>), else n == 1
    Slot slots[kSlots + 1];
    int64_t next_ticket = 1;
    Slot* last = nullptr;    // the call completed last (tri_last_timing, tri_fetch_lnl)
    double last_s2[2] = {NAN, NAN};   // s2 of the evaluation tri_wait returned last
    // posterior samples (tri_set_posterior): K of the next submissions, and the capacity of
    // every slot's index buffers (grown only by tri_set_posterior)
    int64_t post_K = 0, post_cap = 0;
    unsigned long long post_seed = 0, post_stream = 0;
    // the samples of the evaluation tri_wait returned last: its slot's pinned buffers are
    // swapped in here, so that the slot can be reused at once
    int64_t* h_post_last[2] = {nullptr, nullptr};
    int64_t last_post_K = 0;
    int last_branches = 0;
    double last_post_T[2] = {NAN, NAN};
};

// d_lse_out / h_lse_out: the branches' evidence records, then their s2 (moments_kernel), then
// their T (posterior_sums_kernel)
constexpr size_t kLseS2Bytes = 2 * sizeof(LsePartial) + 2 * sizeof(double);
constexpr size_t kLseOutBytes = kLseS2Bytes + 2 * sizeof(double);

Ctx g;

// ---- orbit table (same construction as oracle/quadmodel.py make_orbit_table) ---------------
double ta_newton(double ma, double e) {
    double ea = ma, err = 0.05;
    int k = 0;
    while (std::fabs(err) > 1e-8 && k < 1000) {
        err = ea - e * std::sin(ea) - ma;
        ea = ea - err / (1.0 - e * std::cos(ea));
        k++;
    }
    double sta = std::sqrt(1.0 - e * e) * std::sin(ea) / (1.0 - e * std::cos(ea));
    double cta = (std::cos(ea) - e) / (1.0 - e * std::cos(ea));
    return std::atan2(sta, cta);
}

void linspace(double start, double stop, int n, std::vector<double>& out) {
    out.resize(n);
    double step = (stop - start) / (double)(n - 1);
    for (int i = 0; i < n; i++) out[i] = start + (double)i * step;
    out[n - 1] = stop;
}

int need_ready(bool need_lc) {
    if (!g.ready) return fail(TRI_ESTATE, "tri_init has not been called");
    if (need_lc && !g.have_lc) return fail(TRI_ESTATE, "tri_set_lightcurve has not been called");
    return TRI_OK;
}

Col to_col(const tri_col& c) { return Col{c.ptr, c.stride}; }

// Source pointer for an H2D copy of `bytes` from the caller's `src`: the caller's buffer when it
// is page-locked (or small, or the pinned arena is full), else a pinned copy of it.
const void* via_pinned(Slot& S, const void* src, size_t bytes) {
    if (bytes < kPinnedMinCopy || !S.pinned.base || is_pinned(src)) return src;
    char* hp = S.pinned.take(bytes);
    if (!hp) return src;
    parallel_memcpy(hp, src, bytes);
    return hp;
}

// copy one host column (if any) to the slot's staging arena: `c` then names the device copy
int stage(Slot& S, tri_col& c, int64_t N, cudaStream_t s) {
    if (c.ptr == nullptr) return TRI_OK;
    size_t n = c.stride ? (size_t)N : 1;
    double* p = S.staging.take<double>(n);
    CU(cudaMemcpyAsync(p, via_pinned(S, c.ptr, n * sizeof(double)), n * sizeof(double),
                       cudaMemcpyHostToDevice, s));
    c.ptr = p;
    return TRI_OK;
}

// One evaluation as the submission path sees it, whichever public layout it came in: 1 branch
// (tri_tp_args) or 2 (tri_eb_args: the EB and EBx2P branches), body = rp or reb.  A TP-type
// call has no ebfr and q (NULL) and scalar_loop 0.
struct Call {
    int branches;
    int64_t N;
    tri_col body, ebfr, q, P, inc, ecc, argp, mtot, rhost, u1, u2, cfr, lnprior;
    const uint8_t* extra_mask;
    int companion_is_host, scalar_loop;
};

// The adapters of the two public layouts (nullptr for a NULL argument).
const Call* as_call(const tri_tp_args* a, Call& c) {
    if (!a) return nullptr;
    c = Call{1, a->N, a->rp, {}, {}, a->P_orb, a->inc, a->ecc, a->argp, a->mtot, a->rhost, a->u1,
             a->u2, a->cfr, a->lnprior, a->extra_mask, a->companion_is_host, 0};
    return &c;
}

const Call* as_call(const tri_eb_args* a, Call& c) {
    if (!a) return nullptr;
    c = Call{2, a->N, a->reb, a->ebfr, a->q, a->P_orb, a->inc, a->ecc, a->argp, a->mtot,
             a->rhost, a->u1, a->u2, a->cfr, a->lnprior, a->extra_mask, a->companion_is_host,
             a->scalar_loop};
    return &c;
}

// The columns of a call in staging order, and which calls require each: `need` 1 every call,
// 2 EB-type calls only, 0 none (lnprior is optional).
struct CallCol {
    tri_col Call::*col;
    int need;
};
constexpr CallCol kCallCols[] = {
    {&Call::body, 1}, {&Call::ebfr, 2}, {&Call::q, 2},     {&Call::P, 1},   {&Call::inc, 1},
    {&Call::ecc, 1},  {&Call::argp, 1}, {&Call::mtot, 1},  {&Call::rhost, 1}, {&Call::u1, 1},
    {&Call::u2, 1},   {&Call::cfr, 1},  {&Call::lnprior, 0}};

// copy the call's host columns to the slot's staging arena: `c` then names the device copies
int stage_call(Slot& S, Call& c, cudaStream_t s) {
    for (const CallCol& k : kCallCols) {
        int rc = stage(S, c.*k.col, c.N, s);
        if (rc) return rc;
    }
    return TRI_OK;
}

int lnl_grid() { return g.sm_count * std::max(1, g.lnl_blocks_per_sm); }

size_t lnl_smem_bytes() { return g.lnl_smem; }

struct Scratch {
    double *a = nullptr, *cval = nullptr;
    double* lnl[2] = {nullptr, nullptr};   // per branch
    int64_t* items = nullptr;
    LsePartial* partials = nullptr;   // [2][lnl_grid()]
};

int lse_blocks(int64_t N) {
    int64_t b = (N + 4095) / 4096;
    return (int)std::max<int64_t>(1, std::min<int64_t>(b, 4 * (int64_t)g.sm_count));
}

int64_t post_tiles(int64_t N) { return (N + kPostTile - 1) / kPostTile; }

// (sized for an EB-type call: a slot serves both kinds in turn)
size_t scratch_bytes(int64_t N) {
    size_t n = (size_t)N;
    size_t b = 0;
    b += (n * 8 + 256) * 4;              // a, p, lnl of the two branches
    b += (n * 8 + 256) * 2;              // items, cval
    b += (size_t)lnl_grid() * sizeof(LsePartial) * 2 + 512;
    b += (size_t)lse_blocks(N) * sizeof(double) * 2 + 256;   // moments_kernel partials
    if (g.post_K > 0) b += (size_t)(2 * post_tiles(N) + 1) * sizeof(double) * 2 + 512;
    return b + 4096;
}

void finish_result(const LsePartial& r, int64_t N, tri_result* out) {
    out->m = r.m;
    out->s = r.s;
    out->n_finite = (int64_t)r.n_finite;
    out->n_posinf = (int64_t)r.n_posinf;
    if (r.n_posinf > 0) out->lnZ = INFINITY;
    else if (r.n_finite == 0) out->lnZ = -INFINITY;
    else out->lnZ = r.m + std::log(r.s) - std::log((double)N);
}

// the light-curve instantiation for the current light curve and counting switch
void (*lnl_instance())(LnlArgs) {
    const bool seg = g.cad.n > 1;   // mixed cadence: the segmented instantiation
    if (g.count_work) return seg ? lnl_kernel<true, true> : lnl_kernel<true, false>;
    return seg ? lnl_kernel<false, true> : lnl_kernel<false, false>;
}

int launch_lnl(Slot& S, LnlArgs& A, cudaStream_t s) {
    if (g.cad.n > 1) A.cad = g.cad;
    lnl_instance()<<<lnl_grid(), kLnlThreads, lnl_smem_bytes(), s>>>(A);
    S.launches += 1;
    CU(cudaGetLastError());
    return TRI_OK;
}

// evidence records and best draws of the call's branches: one block per branch
int launch_finalize(Slot& S, const Scratch& W, int64_t N, int branches, const tri_result* r,
                    cudaStream_t s) {
    FinalizeArgs F{};
    F.partials = W.partials;
    F.n_partials = lnl_grid();
    F.lse_out = S.d_lse_out;
    F.items = W.items;
    F.cval = W.cval;
    F.cap = N;
    F.count_dev = S.d_counters + 0;
    F.hist16 = S.d_hist16;
    for (int b = 0; b < branches; ++b) {
        S.want_top[b] = r[b].top_cap > 0 && r[b].top_idx && r[b].top_lnL;
        F.top_cap[b] = S.want_top[b] ? r[b].top_cap : 0;
        F.top_idx[b] = r[b].top_idx;
        F.top_val[b] = r[b].top_lnL;
    }
    if (branches == 1) S.want_top[1] = false;
    F.st = S.d_topk;
    finalize_kernel<<<branches, kFinThreads, 0, s>>>(F);
    S.launches += 1;
    CU(cudaGetLastError());
    return TRI_OK;
}

// s2 of the call's branches after finalize_kernel (only with tri_set_moments on)
int launch_moments(Slot& S, const Scratch& W, int64_t N, int branches, Col lnprior,
                   cudaStream_t s) {
    MomentsArgs M{};
    M.lnl[0] = W.lnl[0];
    M.lnl[1] = W.lnl[1];
    M.lnprior = lnprior;
    M.N = N;
    M.branches = branches;
    M.lse = S.d_lse_out;
    M.partials = S.scratch.take<double>(2 * (size_t)lse_blocks(N));
    M.done = S.d_mom_done;
    M.s2_out = reinterpret_cast<double*>(S.d_lse_out + 2);
    moments_kernel<<<lse_blocks(N), kMomThreads, 0, s>>>(M);
    S.launches += 1;
    CU(cudaGetLastError());
    return TRI_OK;
}

// posterior samples of the call's branches after finalize_kernel (and moments_kernel): tile sums
// and offsets, then the selection; the indices travel to the slot's pinned landing zone
int launch_posterior(Slot& S, const Scratch& W, int64_t N, int branches, Col lnprior,
                     cudaStream_t s) {
    PosteriorArgs P{};
    P.lnl[0] = W.lnl[0];
    P.lnl[1] = W.lnl[1];
    P.lnprior = lnprior;
    P.N = N;
    P.tiles = post_tiles(N);
    P.lse = S.d_lse_out;
    P.tile_sum = S.scratch.take<double>(2 * (size_t)P.tiles);
    P.tile_off = S.scratch.take<double>(2 * (size_t)(P.tiles + 1));
    P.done = S.d_post_done;
    P.total = reinterpret_cast<double*>(S.d_lse_out + 2) + 2;
    P.idx[0] = S.d_post_idx[0];
    P.idx[1] = S.d_post_idx[1];
    P.K = S.post_K;
    P.seed = S.post_seed;
    P.stream = S.post_stream;
    dim3 grid((unsigned)P.tiles, (unsigned)branches);
    posterior_sums_kernel<<<grid, kPostThreads, 0, s>>>(P);
    CU(cudaGetLastError());
    posterior_select_kernel<<<grid, kPostThreads, 0, s>>>(P);
    S.launches += 2;
    CU(cudaGetLastError());
    for (int b = 0; b < branches; ++b)
        CU(cudaMemcpyAsync(S.h_post_idx[b], S.d_post_idx[b], (size_t)S.post_K * sizeof(int64_t),
                           cudaMemcpyDeviceToHost, s));
    return TRI_OK;
}

// bytes of d_lse_out that a call's read-back needs
size_t lse_out_bytes(const Slot& S, int branches) {
    return S.post_K > 0 ? kLseOutBytes : S.moments ? kLseS2Bytes
                                                   : branches * sizeof(LsePartial);
}

// The LnlArgs fields that every launch of the light-curve kernel sets alike: light curve, orbit
// table, kind and the model columns of `c` (device pointers), with the period column P and the
// semi-major axis a given apart.  The caller adds its work list and its outputs.
LnlArgs lnl_args(const Call& c, Col P, Col a) {
    LnlArgs A{};
    A.lc = g.lc; A.tab = g.tab; A.eb = c.branches - 1; A.companion_is_host = c.companion_is_host;
    A.body = to_col(c.body); A.ebfr = to_col(c.ebfr);
    A.P = P; A.inc = to_col(c.inc); A.a = a; A.rhost = to_col(c.rhost);
    A.u1 = to_col(c.u1); A.u2 = to_col(c.u2); A.ecc = to_col(c.ecc); A.argp = to_col(c.argp);
    A.cfr = to_col(c.cfr);
    A.scalar_rule = c.scalar_loop ? 1 : 0;
    return A;
}

// Queue one evaluation on `s` for slot S: every pointer in `c` and in r[0 .. c.branches - 1]
// (lnL_out, mask_out, top_idx, top_lnL) is a device pointer.  The two branches of an EB-type
// call, EB (period P) and EBx2P (period 2P), share one geometry launch and one work list.
// Nothing here waits for the GPU; the small result record lands in the slot's pinned buffers and
// is read by finish_slot.
int enqueue(Slot& S, const Call& c, const tri_result* r, cudaStream_t s) {
    const int64_t N = c.N;
    const bool eb = c.branches == 2;
    S.scratch.reset();
    int rc = S.scratch.reserve(scratch_bytes(N));
    if (rc) return rc;
    Scratch W;
    W.a = S.scratch.take<double>(N);
    double* p = S.scratch.take<double>(N);   // EB-type: the period of each draw's branch
    for (int b = 0; b < c.branches; ++b)
        W.lnl[b] = r[b].lnL_out ? r[b].lnL_out : S.scratch.take<double>(N);
    W.items = S.scratch.take<int64_t>(N);
    W.cval = S.scratch.take<double>(N);
    W.partials = S.scratch.take<LsePartial>(2 * (size_t)lnl_grid());
    S.launches = 0;
    CU(cudaMemsetAsync(S.d_counters, 0, 8 * sizeof(unsigned long long), s));
    CU(cudaEventRecord(S.ev[0], s));
    int gb = std::max(1, (int)std::min<int64_t>((N + 255) / 256, (int64_t)g.sm_count * 8));
    if (eb) {
        GeomEb G{};
        G.N = N;
        G.reb = to_col(c.body); G.q = to_col(c.q); G.P = to_col(c.P); G.inc = to_col(c.inc);
        G.ecc = to_col(c.ecc); G.argp = to_col(c.argp); G.mtot = to_col(c.mtot);
        G.rhost = to_col(c.rhost);
        G.extra_mask = c.extra_mask;
        G.scalar_loop = c.scalar_loop;
        G.a_out = W.a; G.p_out = p; G.lnl_out = W.lnl[0]; G.lnl_twin_out = W.lnl[1];
        G.mask_out = r[0].mask_out; G.mask_twin_out = r[1].mask_out;
        G.items = W.items; G.n_items = S.d_counters + 0;
        geometry_eb_kernel<<<gb, 256, 0, s>>>(G);
    } else {
        GeomTp G{};
        G.N = N;
        G.rp = to_col(c.body); G.P = to_col(c.P); G.inc = to_col(c.inc); G.ecc = to_col(c.ecc);
        G.argp = to_col(c.argp); G.mtot = to_col(c.mtot); G.rhost = to_col(c.rhost);
        G.extra_mask = c.extra_mask;
        G.a_out = W.a; G.lnl_out = W.lnl[0]; G.mask_out = r[0].mask_out;
        G.items = W.items; G.n_items = S.d_counters + 0;
        geometry_tp_kernel<<<gb, 256, 0, s>>>(G);
    }
    S.launches += 1;
    CU(cudaGetLastError());
    CU(cudaEventRecord(S.ev[1], s));

    // the work-list length stays on the device: no host round trip between the two kernels
    LnlArgs A = lnl_args(c, eb ? Col{p, 1} : to_col(c.P), Col{W.a, 1});
    A.items = W.items; A.items_cap = N; A.count_dev = S.d_counters + 0;
    A.next = S.d_counters + 2;
    A.out = W.lnl[0]; A.out_twin = W.lnl[1]; A.counters = S.d_counters + 4;
    A.lnprior = to_col(c.lnprior); A.lse_partials = W.partials; A.cval = W.cval;
    A.hist16 = S.d_hist16;
    rc = launch_lnl(S, A, s);
    if (rc) return rc;
    CU(cudaEventRecord(S.ev[2], s));
    rc = launch_finalize(S, W, N, c.branches, r, s);
    if (rc) return rc;
    if (S.moments) {
        rc = launch_moments(S, W, N, c.branches, to_col(c.lnprior), s);
        if (rc) return rc;
    }
    if (S.post_K > 0) {
        rc = launch_posterior(S, W, N, c.branches, to_col(c.lnprior), s);
        if (rc) return rc;
    }
    CU(cudaMemcpyAsync(S.h_topk, S.d_topk, c.branches * sizeof(TopkState),
                       cudaMemcpyDeviceToHost, s));
    S.lnl[0] = W.lnl[0]; S.lnl[1] = W.lnl[1];
    CU(cudaEventRecord(S.ev[3], s));
    CU(cudaMemcpyAsync(S.h_lse_out, S.d_lse_out, lse_out_bytes(S, c.branches),
                       cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(S.h_counters, S.d_counters, 8 * sizeof(unsigned long long),
                       cudaMemcpyDeviceToHost, s));
    return TRI_OK;
}

// best first, ties by ascending index: the order of a stable sort of -lnL
void sort_candidates(int64_t n, int64_t* idx, double* val) {
    std::vector<std::pair<double, int64_t>> v((size_t)n);
    for (int64_t i = 0; i < n; ++i) v[(size_t)i] = {val[i], idx[i]};
    std::sort(v.begin(), v.end(), [](const std::pair<double, int64_t>& x,
                                     const std::pair<double, int64_t>& y) {
        return x.first > y.first || (x.first == y.first && x.second < y.second);
    });
    for (int64_t i = 0; i < n; ++i) { val[i] = v[(size_t)i].first; idx[i] = v[(size_t)i].second; }
}

// After the slot's `done` event: turn the pinned landing zone into the caller's records.
void finish_slot(Slot& S, tri_result* out) {
    const double* h_s2 = reinterpret_cast<const double*>(S.h_lse_out + 2);
    for (int b = 0; b < 2; ++b)
        S.s2[b] = !S.moments || b >= S.branches ? NAN : S.N == 0 ? 0.0 : h_s2[b];
    for (int b = 0; b < 2; ++b)   // (N == 0: no draw, an empty posterior)
        S.post_T[b] = S.post_K == 0 || b >= S.branches ? NAN : S.N == 0 ? 0.0 : h_s2[2 + b];
    for (int b = 0; b < S.branches; ++b) {
        tri_result r = S.want[b];   // keeps the caller's pointers and top_cap
        if (S.N == 0) {
            LsePartial z{-INFINITY, 0.0, 0, 0};
            finish_result(z, 0, &r);
            r.n_pass = r.n_stamps = r.n_interior = r.n_limb = r.n_top = 0;
            r.n_evaluated = 0;
            out[b] = r;
            continue;
        }
        finish_result(S.h_lse_out[b], S.N, &r);
        // work items: [0] at the front of the list, [3] at the back (short chords)
        const int64_t n_items = (int64_t)S.h_counters[0] + (int64_t)S.h_counters[3];
        if (S.branches == 1) {
            r.n_pass = n_items;
        } else {   // twins are counted separately by the geometry kernel
            r.n_pass = b ? (int64_t)S.h_counters[1] : n_items - (int64_t)S.h_counters[1];
        }
        // the two EB branches share one launch: these totals are joint
        r.n_stamps = (int64_t)S.h_counters[5];
        r.n_interior = (int64_t)S.h_counters[6];
        r.n_limb = (int64_t)S.h_counters[7];
        r.n_top = S.want_top[b]
            ? (int64_t)std::min<unsigned long long>(S.h_topk[b].n_out,
                                                    (unsigned long long)r.top_cap)
            : 0;
        r.n_evaluated = (int64_t)S.h_topk[b].n_finite;
        if (S.host && S.want_top[b]) {
            std::memcpy(r.top_idx, S.h_tidx[b], (size_t)r.n_top * 8);
            std::memcpy(r.top_lnL, S.h_tval[b], (size_t)r.n_top * 8);
            sort_candidates(r.n_top, r.top_idx, r.top_lnL);
        }
        out[b] = r;
    }
}

Slot* free_slot() {
    for (int i = 0; i < kSlots; ++i)
        if (g.slots[i].ticket == 0) return &g.slots[i];
    return nullptr;
}

// Arenas only grow, and growing one means cudaFree (a device-wide synchronisation).  When a call
// needs more than its slot holds, every free slot is grown to the new size in the same breath,
// so that a run of equally large calls pays for it once and not once per slot of the ring.
int grow_slots(Slot& S, size_t scratch, size_t staging, size_t pinned) {
    if (scratch <= S.scratch.cap && staging <= S.staging.cap && pinned <= S.pinned.cap)
        return TRI_OK;
    for (int i = 0; i < kSlots; ++i) {
        Slot& T = g.slots[i];
        if (T.ticket != 0 && &T != &S) continue;
        int rc = T.scratch.reserve(scratch);
        if (!rc && staging) rc = T.staging.reserve(staging);
        if (!rc && pinned) rc = T.pinned.reserve(pinned);
        if (rc) return rc;
    }
    return TRI_OK;
}

// A submission that fails after its first asynchronous copy leaves work queued on the two
// streams that refers to the slot's arenas: let it finish before the slot is handed out again.
int abandon(Slot& S, int rc) {
    cudaStreamSynchronize(g.copy_stream);
    cudaStreamSynchronize(g.stream);
    cudaGetLastError();
    S.ticket = 0;
    S.staging.reset();
    S.pinned.reset();
    S.scratch.reset();
    return rc;
}

Slot* find_slot(int64_t ticket) {
    if (ticket <= 0) return nullptr;
    for (int i = 0; i < kSlots; ++i)
        if (g.slots[i].ticket == ticket) return &g.slots[i];
    return nullptr;
}

int no_slot() {
    return fail(TRI_ESTATE, "TRI_MAX_INFLIGHT evaluations are already in flight: tri_wait one");
}

// The checks of every submission (before anything is queued), then a free slot that holds the
// call's switches: tri_set_moments and tri_set_posterior as they are now.
int open_slot(const Call* c, const tri_result* want, const int64_t* ticket, Slot** out) {
    int rc = need_ready(true);
    if (rc) return rc;
    if (!c || !want || !ticket) return fail(TRI_EINVAL, "NULL argument");
    if (c->N < 0) return fail(TRI_EINVAL, "N must be >= 0");
    for (const CallCol& k : kCallCols) {
        const tri_col& x = c->*k.col;
        if (x.ptr == nullptr) {
            if (k.need && c->branches >= k.need)
                return fail(TRI_EINVAL, "a required column is NULL");
        } else if (x.stride != 0 && x.stride != 1) {
            return fail(TRI_EINVAL, "column stride must be 0 or 1");
        }
    }
    Slot* S = free_slot();
    if (!S) return no_slot();
    CU(cudaSetDevice(g.device));
    S->moments = g.moments;
    S->post_K = g.post_K;
    S->post_seed = g.post_seed;
    S->post_stream = g.post_stream;
    *out = S;
    return TRI_OK;
}

// mark the slot in flight and hand out its ticket
void commit(Slot& S, const Call& c, bool host, const tri_result* want, int64_t* ticket) {
    S.branches = c.branches;
    S.N = c.N;
    S.host = host;
    for (int b = 0; b < c.branches; ++b) S.want[b] = want[b];
    S.ticket = g.next_ticket++;
    *ticket = S.ticket;
}

}  // namespace

extern "C" {

const char* tri_last_error(void) {
    if (g_err.empty()) {
        std::lock_guard<std::mutex> lock(g_err_mutex);
        g_err = g_err_engine;
    }
    return g_err.c_str();
}

int tri_init(int device) {
    if (g.ready && g.device == device) return TRI_OK;
    if (g.ready) tri_shutdown();
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(TRI_ENODEVICE,
                    std::string("no CUDA device available (there is no CPU fallback): ") +
                        (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0"));
    if (device < 0 || device >= n) return fail(TRI_EINVAL, "device index out of range");
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    g.device = device;
    g.sm_count = prop.multiProcessorCount;
    CU(cudaStreamCreateWithFlags(&g.stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&g.copy_stream, cudaStreamNonBlocking));
    // orbit table
    // (+1: z_sub may read one element behind the last row with weight 0, see tri_model.cuh)
    std::vector<double> es, ms, tae((size_t)kTableNe * kTableNm + 1, 0.0);
    linspace(0.0, kTableMaxE, kTableNe, es);
    linspace(0.0, kPi, kTableNm, ms);
    for (int i = 0; i < kTableNe; i++)
        for (int j = 0; j < kTableNm; j++)
            tae[(size_t)i * kTableNm + j] = ta_newton(ms[j], es[i]) - ms[j];
    CU(cudaMalloc(&g.d_tae, tae.size() * sizeof(double)));
    CU(cudaMemcpy(g.d_tae, tae.data(), tae.size() * sizeof(double), cudaMemcpyHostToDevice));
    g.tab.tae = g.d_tae;
    g.tab.de = es[1] - es[0];
    g.tab.dm = ms[1] - ms[0];
    g.tab.inv_dm = 1.0 / g.tab.dm;
    for (Slot& S : g.slots) {
        CU(cudaMalloc(&S.d_counters, 8 * sizeof(unsigned long long)));
        CU(cudaMalloc(&S.d_lse_out, kLseOutBytes));
        CU(cudaMallocHost(&S.h_lse_out, kLseOutBytes));
        CU(cudaMalloc(&S.d_mom_done, sizeof(unsigned int)));
        CU(cudaMemset(S.d_mom_done, 0, sizeof(unsigned int)));
        CU(cudaMalloc(&S.d_post_done, 2 * sizeof(unsigned int)));
        CU(cudaMemset(S.d_post_done, 0, 2 * sizeof(unsigned int)));
        CU(cudaMallocHost(&S.h_counters, 8 * sizeof(unsigned long long)));
        CU(cudaMalloc(&S.d_topk, 2 * sizeof(TopkState)));
        CU(cudaMalloc(&S.d_hist16, 2 * (size_t)kTopkBins * sizeof(unsigned int)));
        CU(cudaMemset(S.d_hist16, 0, 2 * (size_t)kTopkBins * sizeof(unsigned int)));
        CU(cudaMallocHost(&S.h_topk, 2 * sizeof(TopkState)));
        for (auto& ev : S.ev) CU(cudaEventCreate(&ev));
        CU(cudaEventCreateWithFlags(&S.copied, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&S.done, cudaEventDisableTiming));
    }
    // occupancy of the persistent light-curve kernel
    int bps = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, lnl_kernel<false, false>, kLnlThreads,
                                                     0));
    g.lnl_blocks_per_sm = std::max(1, bps);
    g.lnl_smem = 0;
    g.ready = true;
    g.have_lc = false;
    return TRI_OK;
}

int tri_shutdown(void) {
    if (!g.ready) return TRI_OK;
    cudaSetDevice(g.device);
    cudaDeviceSynchronize();   // evaluations may still be running on caller streams
    cudaFree(g.d_tae);
    cudaFree(g.d_time);
    cudaFree(g.d_flux);
    cudaFree(g.d_prefix);
    cudaFree(g.d_weight);
    cudaFree(g.d_perm);
    for (Slot& S : g.slots) {
        cudaFree(S.d_counters);
        cudaFree(S.d_lse_out);
        cudaFreeHost(S.h_lse_out);
        cudaFree(S.d_mom_done);
        cudaFree(S.d_post_done);
        cudaFreeHost(S.h_counters);
        cudaFree(S.d_topk);
        cudaFree(S.d_hist16);
        cudaFreeHost(S.h_topk);
        if (S.scratch.base) cudaFree(S.scratch.base);
        if (S.staging.base) cudaFree(S.staging.base);
        if (S.pinned.base) cudaFreeHost(S.pinned.base);
        for (int b = 0; b < 2; ++b) {
            if (S.h_tidx[b]) cudaFreeHost(S.h_tidx[b]);
            if (S.h_tval[b]) cudaFreeHost(S.h_tval[b]);
            if (S.d_post_idx[b]) cudaFree(S.d_post_idx[b]);
            if (S.h_post_idx[b]) cudaFreeHost(S.h_post_idx[b]);
        }
        for (auto& ev : S.ev) cudaEventDestroy(ev);
        cudaEventDestroy(S.copied);
        cudaEventDestroy(S.done);
    }
    for (int b = 0; b < 2; ++b)
        if (g.h_post_last[b]) cudaFreeHost(g.h_post_last[b]);
    cudaStreamDestroy(g.copy_stream);
    cudaStreamDestroy(g.stream);
    g = Ctx{};
    return TRI_OK;
}

int tri_struct_sizes(int64_t* out, int32_t n) {
    const int64_t sizes[8] = {sizeof(tri_col), sizeof(tri_tp_args), sizeof(tri_eb_args),
                              sizeof(tri_result), sizeof(tri_powerlaw), sizeof(tri_spline),
                              sizeof(tri_bound_prior), sizeof(tri_sampler_args)};
    if (!out || n < 0 || n > 8) return fail(TRI_EINVAL, "bad argument");
    for (int i = 0; i < n; ++i) out[i] = sizes[i];
    return TRI_OK;
}

int tri_set_counting(int32_t on) {
    int rc = need_ready(false);
    if (rc) return rc;
    g.count_work = on != 0;
    return TRI_OK;
}

int tri_set_moments(int32_t on) {
    int rc = need_ready(false);
    if (rc) return rc;
    g.moments = on != 0;
    return TRI_OK;
}

int tri_last_moments(double s2[2]) {
    int rc = need_ready(false);
    if (rc) return rc;
    if (!s2) return fail(TRI_EINVAL, "NULL argument");
    s2[0] = g.last_s2[0];
    s2[1] = g.last_s2[1];
    return TRI_OK;
}

// Grow the index buffers of every slot (and the landing zone of the last result) to K per
// branch.  The evaluations in flight finish first; the indices they already returned move over.
static int grow_posterior(int64_t K) {
    CU(cudaDeviceSynchronize());
    auto grow_host = [&](int64_t*& p) -> int {
        int64_t* q = nullptr;
        CU(cudaMallocHost(&q, (size_t)K * sizeof(int64_t)));
        if (p) {
            std::memcpy(q, p, (size_t)g.post_cap * sizeof(int64_t));
            cudaFreeHost(p);
        }
        p = q;
        return TRI_OK;
    };
    for (int i = 0; i < kSlots; ++i) {
        Slot& S = g.slots[i];
        for (int b = 0; b < 2; ++b) {
            if (S.d_post_idx[b]) cudaFree(S.d_post_idx[b]);
            S.d_post_idx[b] = nullptr;
            CU(cudaMalloc(&S.d_post_idx[b], (size_t)K * sizeof(int64_t)));
            int rc = grow_host(S.h_post_idx[b]);
            if (rc) return rc;
        }
    }
    for (int b = 0; b < 2; ++b) {
        int rc = grow_host(g.h_post_last[b]);
        if (rc) return rc;
    }
    g.post_cap = K;
    return TRI_OK;
}

int tri_set_posterior(int64_t K, uint64_t seed, uint64_t stream) {
    int rc = need_ready(false);
    if (rc) return rc;
    if (K < 0 || K > TRI_MAX_POSTERIOR)
        return fail(TRI_EINVAL, "posterior sample count K must be in [0, TRI_MAX_POSTERIOR]");
    CU(cudaSetDevice(g.device));
    if (K > g.post_cap) {
        rc = grow_posterior(K);
        if (rc) return rc;
    }
    g.post_K = K;
    g.post_seed = seed;
    g.post_stream = stream;
    return TRI_OK;
}

int tri_last_posterior(int32_t branch, int64_t* idx, int64_t cap, int64_t* n, double* total) {
    int rc = need_ready(false);
    if (rc) return rc;
    if (!n || !total || (!idx && cap > 0)) return fail(TRI_EINVAL, "NULL argument");
    if (branch < 0 || branch > 1 || (g.last_branches > 0 && branch >= g.last_branches))
        return fail(TRI_EINVAL, "bad branch");
    const double T = g.last_post_T[branch];
    const int64_t k = g.last_post_K > 0 && T > 0.0 && std::isfinite(T) ? g.last_post_K : 0;
    if (cap < k) return fail(TRI_EINVAL, "cap is smaller than the posterior sample count");
    if (k) std::memcpy(idx, g.h_post_last[branch], (size_t)k * sizeof(int64_t));
    *n = k;
    *total = T;
    return TRI_OK;
}

int tri_sm_count(int32_t* n) {
    int rc = need_ready(false);
    if (rc) return rc;
    *n = g.sm_count;
    return TRI_OK;
}

// `grp` (mixed cadence, tri_set_lightcurve_cadence): cadence group of every stamp, whose
// exposure and sample count `groups` holds (groups->n >= 2); exptime / nsamples are then the
// largest of the groups.  nullptr: one cadence (exptime, nsamples).
static int set_lightcurve(const double* time, const double* flux, const double* err,
                          int64_t npts, double sigma, double exptime, int32_t nsamples,
                          const int* grp = nullptr, const CadenceTable* groups = nullptr) {
    int rc = need_ready(false);
    if (rc) return rc;
    if (!time || !flux || npts <= 0) return fail(TRI_EINVAL, "empty light curve");
    if (npts > (int64_t)1 << 28) return fail(TRI_EINVAL, "light curve too long");
    if (err) {   // per-point errors: the reference scalar is their mean
        long double acc = 0.0L;
        for (int64_t j = 0; j < npts; j++) {
            if (!(err[j] > 0.0) || !std::isfinite(err[j]))
                return fail(TRI_EINVAL, "per-point errors must be finite and > 0");
            acc += err[j];
        }
        sigma = (double)(acc / (long double)npts);
    }
    if (!(sigma > 0.0) || nsamples < 1 || !(exptime >= 0.0))
        return fail(TRI_EINVAL, "sigma must be > 0, nsamples >= 1, exptime >= 0");
    for (int64_t j = 0; j < npts; j++)
        if (std::isnan(time[j]) || std::isnan(flux[j]))
            return fail(TRI_EINVAL, "NaN in light curve (calc_probs drops them, triceratops.py:709)");
    // chi^2 is a plain sum over stamps, so the stamps may be visited in time order
    std::vector<int64_t> order(npts);
    std::iota(order.begin(), order.end(), 0);
    if (grp)   // (group, time): each group is one contiguous, time-sorted slice
        std::stable_sort(order.begin(), order.end(), [&](int64_t x, int64_t y) {
            return grp[x] < grp[y] || (grp[x] == grp[y] && time[x] < time[y]);
        });
    else
        std::stable_sort(order.begin(), order.end(),
                         [&](int64_t x, int64_t y) { return time[x] < time[y]; });
    std::vector<double> t(npts), f(npts), pre(npts + 1), wgt(err ? npts : 0);
    long double run = 0.0L;
    pre[0] = 0.0;
    for (int64_t j = 0; j < npts; j++) {
        t[j] = time[order[j]];
        f[j] = flux[order[j]];
        long double d = (long double)f[j] - 1.0L;
        double term = (double)d * (double)d;
        if (err) {
            wgt[j] = 1.0 / (err[order[j]] * err[order[j]]);
            term = ((double)d * wgt[j]) * (double)d;     // as the kernel forms w r^2
        }
        run += (long double)term;
        pre[j + 1] = (double)run;
    }
    CU(cudaSetDevice(g.device));
    // evaluations still in flight read the current light curve: let them finish first
    for (int i = 0; i < kSlots; ++i)
        if (g.slots[i].ticket != 0) CU(cudaEventSynchronize(g.slots[i].done));
    CU(cudaStreamSynchronize(g.stream));
    if ((size_t)npts > g.lc_cap) {
        cudaFree(g.d_time); cudaFree(g.d_flux); cudaFree(g.d_prefix); cudaFree(g.d_perm);
        cudaFree(g.d_weight);
        g.d_time = g.d_flux = g.d_prefix = g.d_weight = nullptr;
        g.d_perm = nullptr;
        g.lc_cap = 0;
        CU(cudaMalloc(&g.d_perm, npts * sizeof(int)));
        CU(cudaMalloc(&g.d_time, npts * sizeof(double)));
        CU(cudaMalloc(&g.d_flux, npts * sizeof(double)));
        CU(cudaMalloc(&g.d_prefix, (npts + 1) * sizeof(double)));
        CU(cudaMalloc(&g.d_weight, npts * sizeof(double)));
        g.lc_cap = (size_t)npts;
    }
    CU(cudaMemcpy(g.d_time, t.data(), npts * sizeof(double), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(g.d_flux, f.data(), npts * sizeof(double), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(g.d_prefix, pre.data(), (npts + 1) * sizeof(double), cudaMemcpyHostToDevice));
    if (err) CU(cudaMemcpy(g.d_weight, wgt.data(), npts * sizeof(double), cudaMemcpyHostToDevice));
    {
        std::vector<int> perm(npts);
        for (int64_t j = 0; j < npts; j++) perm[j] = (int)order[j];
        CU(cudaMemcpy(g.d_perm, perm.data(), npts * sizeof(int), cudaMemcpyHostToDevice));
    }
    g.lc.time = g.d_time; g.lc.flux = g.d_flux; g.lc.prefix = g.d_prefix;
    g.lc.weight = err ? g.d_weight : nullptr;
    g.lc.npts = (int)npts; g.lc.nsamples = nsamples; g.lc.sigma = sigma; g.lc.exptime = exptime;
    g.lc.tmin = t.front(); g.lc.tmax = t.back();
    g.cad = CadenceTable{};
    g.cad.n = 1;
    if (grp) {
        g.cad = *groups;
        g.lc.tmin = *std::min_element(t.begin(), t.end());
        g.lc.tmax = *std::max_element(t.begin(), t.end());
        int j = 0;
        for (int c = 0; c < g.cad.n; ++c) {
            g.cad.off[c] = j;
            while (j < npts && grp[order[j]] == c) ++j;
            g.cad.tmin[c] = t[g.cad.off[c]];
            g.cad.tmax[c] = t[j - 1];
        }
        g.cad.off[g.cad.n] = j;
    }
    // stage the light curve in shared memory only when that costs no occupancy (of the
    // instantiation that will run)
    {
        void (*kern)(LnlArgs) = lnl_instance();
        int bps0 = 0, bps1 = 0;
        size_t need = (size_t)(3 * (size_t)npts + 1) * sizeof(double);
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps0, kern, kLnlThreads, 0));
        g.lnl_smem = 0;
        if (need <= 48 * 1024) {
            CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps1, kern, kLnlThreads, need));
            if (bps1 >= bps0) g.lnl_smem = need;
        }
        g.lnl_blocks_per_sm = std::max(1, bps0);
    }
    g.have_lc = true;
    return TRI_OK;
}

int tri_set_lightcurve(const double* time, const double* flux, int64_t npts, double sigma,
                       double exptime, int32_t nsamples) {
    return set_lightcurve(time, flux, nullptr, npts, sigma, exptime, nsamples);
}

int tri_set_lightcurve_err(const double* time, const double* flux, const double* flux_err,
                           int64_t npts, double exptime, int32_t nsamples) {
    if (!flux_err) return fail(TRI_EINVAL, "flux_err is NULL");
    return set_lightcurve(time, flux, flux_err, npts, 0.0, exptime, nsamples);
}

static_assert(kMaxCadences == TRI_MAX_CADENCES, "cadence table size");

int tri_set_lightcurve_cadence(const double* time, const double* flux, const double* flux_err,
                               double sigma, const double* exptime, const int32_t* nsamples,
                               int64_t npts) {
    int rc = need_ready(false);
    if (rc) return rc;
    if (!time || !flux || npts <= 0) return fail(TRI_EINVAL, "empty light curve");
    if (!exptime || !nsamples) return fail(TRI_EINVAL, "exptime or nsamples is NULL");
    if (npts > (int64_t)1 << 28) return fail(TRI_EINVAL, "light curve too long");
    // distinct (exptime, nsamples) pairs, compared exactly
    std::vector<std::pair<double, int32_t>> pairs;
    for (int64_t j = 0; j < npts; j++) {
        const double e = exptime[j];
        const int32_t n = nsamples[j];
        if (!std::isfinite(e) || e < 0.0)
            return fail(TRI_EINVAL, "exptime must be finite and >= 0 at every stamp");
        if (n < 1) return fail(TRI_EINVAL, "nsamples must be >= 1 at every stamp");
        const std::pair<double, int32_t> pr(e, n);
        if (std::find(pairs.begin(), pairs.end(), pr) != pairs.end()) continue;
        if ((int)pairs.size() == TRI_MAX_CADENCES)
            return fail(TRI_EINVAL, "more than TRI_MAX_CADENCES distinct (exptime, nsamples) "
                                    "pairs: round the exposure times to their cadences");
        pairs.push_back(pr);
    }
    const double sig = flux_err ? 0.0 : sigma;
    if (pairs.size() == 1)   // one cadence: exactly the scalar calls
        return set_lightcurve(time, flux, flux_err, npts, sig, pairs[0].first, pairs[0].second);
    std::sort(pairs.begin(), pairs.end());
    CadenceTable cad{};
    cad.n = (int)pairs.size();
    double emax = 0.0;
    int32_t nmax = 1;
    for (int c = 0; c < cad.n; ++c) {
        cad.exptime[c] = pairs[c].first;
        cad.nsamples[c] = pairs[c].second;
        emax = std::max(emax, pairs[c].first);
        nmax = std::max(nmax, pairs[c].second);
    }
    std::vector<int> grp(npts);
    for (int64_t j = 0; j < npts; j++)
        grp[j] = (int)(std::find(pairs.begin(), pairs.end(),
                                 std::pair<double, int32_t>(exptime[j], nsamples[j]))
                       - pairs.begin());
    return set_lightcurve(time, flux, flux_err, npts, sig, emax, nmax, grp.data(), &cad);
}

// ---- submit / wait --------------------------------------------------------------------------
// Device-pointer submission: the kernels go on the caller's stream.
static int submit_dev(const Call* c, const tri_result* want, void* stream, int64_t* ticket) {
    Slot* S = nullptr;
    int rc = open_slot(c, want, ticket, &S);
    if (rc) return rc;
    cudaStream_t s = (cudaStream_t)stream;   // NULL is the CUDA default stream, as everywhere
    if (c->N > 0) {
        rc = grow_slots(*S, scratch_bytes(c->N), 0, 0);
        if (!rc) rc = enqueue(*S, *c, want, s);
        if (rc) { cudaStreamSynchronize(s); return abandon(*S, rc); }
    }
    CU(cudaEventRecord(S->done, s));
    commit(*S, *c, false, want, ticket);
    return TRI_OK;
}

int tri_submit_tp_dev(const tri_tp_args* a, const tri_result* want, void* stream,
                      int64_t* ticket) {
    Call c;
    return submit_dev(as_call(a, c), want, stream, ticket);
}

int tri_submit_eb_dev(const tri_eb_args* a, const tri_result want[2], void* stream,
                      int64_t* ticket) {
    Call c;
    return submit_dev(as_call(a, c), want, stream, ticket);
}

// device-side landing buffers of one branch's outputs, and the copies back to the caller's
static int stage_outputs(Slot& S, int64_t N, const tri_result& want, tri_result& r) {
    const bool top = want.top_cap > 0 && want.top_idx && want.top_lnL;
    r = want;
    r.lnL_out = want.lnL_out ? S.staging.take<double>(N) : nullptr;
    r.mask_out = want.mask_out ? S.staging.take<uint8_t>(N) : nullptr;
    r.top_cap = top ? want.top_cap : 0;
    r.top_idx = top ? S.staging.take<int64_t>(want.top_cap) : nullptr;
    r.top_lnL = top ? S.staging.take<double>(want.top_cap) : nullptr;
    return TRI_OK;
}

// queue the read-back of branch b's candidates into the slot's pinned landing zone, and note
// the device arrays tri_wait copies into the caller's lnL_out / mask_out
static int queue_outputs(Slot& S, int b, const tri_result& want, const tri_result& r,
                         cudaStream_t s) {
    S.d_out_lnl[b] = want.lnL_out ? r.lnL_out : nullptr;
    S.d_out_mask[b] = want.mask_out ? r.mask_out : nullptr;
    if (r.top_cap > 0) {   // n_top is not known yet: the whole candidate buffer travels
        CU(cudaMemcpyAsync(S.h_tidx[b], r.top_idx, (size_t)r.top_cap * 8,
                           cudaMemcpyDeviceToHost, s));
        CU(cudaMemcpyAsync(S.h_tval[b], r.top_lnL, (size_t)r.top_cap * 8,
                           cudaMemcpyDeviceToHost, s));
    }
    return TRI_OK;
}

// pinned landing zone for `cap` candidates per branch (grow-only)
static int reserve_top(Slot& S, int64_t cap) {
    if (cap <= S.h_top_cap) return TRI_OK;
    for (int b = 0; b < 2; ++b) {
        if (S.h_tidx[b]) cudaFreeHost(S.h_tidx[b]);
        if (S.h_tval[b]) cudaFreeHost(S.h_tval[b]);
        S.h_tidx[b] = nullptr;
        S.h_tval[b] = nullptr;
    }
    S.h_top_cap = 0;
    for (int b = 0; b < 2; ++b) {
        CU(cudaMallocHost(&S.h_tidx[b], (size_t)cap * 8));
        CU(cudaMallocHost(&S.h_tval[b], (size_t)cap * 8));
    }
    S.h_top_cap = cap;
    return TRI_OK;
}

// Host-buffer submission into slot S: the columns go to the slot's staging arena on the copy
// stream, the kernels follow on the compute stream.
static int submit_host_body(Slot& S, const Call& h, const tri_result* want, int64_t* ticket) {
    int rc;
    const int64_t N = h.N;
    if (N > 0) {
        cudaStream_t cs = g.copy_stream;
        int64_t top_cap = 0;
        for (int b = 0; b < h.branches; ++b) top_cap = std::max(top_cap, want[b].top_cap);
        // pageable caller columns go through the pinned arena (sized for the EB-type column
        // set too: a slot serves both kinds in turn)
        rc = grow_slots(S, scratch_bytes(N),
                        (size_t)N * 8 * 16 + (size_t)N * 3 + 8192 + (size_t)top_cap * 32,
                        is_pinned(h.inc.ptr)
                            ? 0 : std::min(kPinnedLimit, (size_t)N * 8 * 14 + (size_t)N + 8192));
        if (rc) return rc;
        S.staging.reset();
        S.pinned.reset();
        Call d = h;
        rc = stage_call(S, d, cs);
        if (rc) return rc;
        if (h.extra_mask) {
            uint8_t* m = S.staging.take<uint8_t>(N);
            CU(cudaMemcpyAsync(m, via_pinned(S, h.extra_mask, (size_t)N), (size_t)N,
                               cudaMemcpyHostToDevice, cs));
            d.extra_mask = m;
        }
        rc = reserve_top(S, top_cap);
        if (rc) return rc;
        tri_result r[2];
        for (int b = 0; b < h.branches; ++b) {
            stage_outputs(S, N, want[b], r[b]);
            if (r[b].top_cap > 0) {
                CU(cudaMemsetAsync(r[b].top_idx, 0, (size_t)r[b].top_cap * 8, cs));
                CU(cudaMemsetAsync(r[b].top_lnL, 0, (size_t)r[b].top_cap * 8, cs));
            }
        }
        // the kernels start when the columns have landed; the next call's copies overlap them
        CU(cudaEventRecord(S.copied, cs));
        CU(cudaStreamWaitEvent(g.stream, S.copied, 0));
        rc = enqueue(S, d, r, g.stream);
        if (rc) return rc;
        for (int b = 0; b < h.branches; ++b) {
            rc = queue_outputs(S, b, want[b], r[b], g.stream);
            if (rc) return rc;
        }
    }
    CU(cudaEventRecord(S.done, g.stream));
    commit(S, h, true, want, ticket);
    return TRI_OK;
}

static int submit_host(const Call* h, const tri_result* want, int64_t* ticket) {
    Slot* S = nullptr;
    int rc = open_slot(h, want, ticket, &S);
    if (rc) return rc;
    rc = submit_host_body(*S, *h, want, ticket);
    return rc ? abandon(*S, rc) : TRI_OK;
}

int tri_submit_tp(const tri_tp_args* a, const tri_result* want, int64_t* ticket) {
    Call c;
    return submit_host(as_call(a, c), want, ticket);
}

int tri_submit_eb(const tri_eb_args* a, const tri_result want[2], int64_t* ticket) {
    Call c;
    return submit_host(as_call(a, c), want, ticket);
}

int tri_wait(int64_t ticket, tri_result* out) {
    int rc = need_ready(false);
    if (rc) return rc;
    if (!out) return fail(TRI_EINVAL, "NULL argument");
    Slot* S = find_slot(ticket);
    if (!S) return fail(TRI_EINVAL, "unknown ticket (already waited for?)");
    CU(cudaSetDevice(g.device));
    cudaError_t e = cudaEventSynchronize(S->done);
    if (e != cudaSuccess) {
        S->ticket = 0;
        return fail(TRI_ECUDA, std::string("cudaEventSynchronize: ") + cudaGetErrorString(e));
    }
    finish_slot(*S, out);
    S->ticket = 0;
    g.last = S;
    g.last_s2[0] = S->s2[0];
    g.last_s2[1] = S->s2[1];
    g.last_branches = S->branches;
    g.last_post_K = S->post_K;
    for (int b = 0; b < 2; ++b) {
        g.last_post_T[b] = S->post_T[b];
        if (S->post_K > 0) std::swap(S->h_post_idx[b], g.h_post_last[b]);
    }
    if (S->host && S->N > 0) {   // per-draw outputs (parity runs): copied now, synchronously
        for (int b = 0; b < S->branches; ++b) {
            if (S->d_out_lnl[b])
                CU(cudaMemcpy(S->want[b].lnL_out, S->d_out_lnl[b], (size_t)S->N * 8,
                              cudaMemcpyDeviceToHost));
            if (S->d_out_mask[b])
                CU(cudaMemcpy(S->want[b].mask_out, S->d_out_mask[b], (size_t)S->N,
                              cudaMemcpyDeviceToHost));
        }
    }
    return TRI_OK;
}

// ---- the synchronous forms: submit, then wait ------------------------------------------------
int tri_eval_tp_dev(const tri_tp_args* a, tri_result* out, void* stream) {
    int64_t t = 0;
    int rc = tri_submit_tp_dev(a, out, stream, &t);
    return rc ? rc : tri_wait(t, out);
}

int tri_eval_eb_dev(const tri_eb_args* a, tri_result out[2], void* stream) {
    int64_t t = 0;
    int rc = tri_submit_eb_dev(a, out, stream, &t);
    return rc ? rc : tri_wait(t, out);
}

int tri_eval_tp(const tri_tp_args* a, tri_result* out) {
    int64_t t = 0;
    int rc = tri_submit_tp(a, out, &t);
    return rc ? rc : tri_wait(t, out);
}

int tri_eval_eb(const tri_eb_args* a, tri_result out[2]) {
    int64_t t = 0;
    int rc = tri_submit_eb(a, out, &t);
    return rc ? rc : tri_wait(t, out);
}

static int lnl_seam(int eb, int64_t n, const double* body, const double* ebfr, const double* P,
                    const double* inc, const double* a, const double* R_s, const double* u1,
                    const double* u2, const double* ecc, const double* argp, const double* cfr,
                    int32_t is_host, int32_t twin, double* out, double* model_out = nullptr,
                    double* secdepth_out = nullptr, int scalar_rule = 0) {
    int rc = need_ready(true);
    if (rc) return rc;
    if (n < 0) return fail(TRI_EINVAL, "n must be >= 0");
    if (n == 0) return TRI_OK;
    if (!body || !P || !inc || !a || !R_s || !u1 || !u2 || !ecc || !argp || !cfr ||
        (!out && !model_out) || (eb && !ebfr))
        return fail(TRI_EINVAL, "NULL array");
    const size_t npts = (size_t)g.lc.npts;
    if (model_out && (size_t)n * npts > ((size_t)1 << 28))
        return fail(TRI_EINVAL, "model matrix too large (n * npts > 2^28): simulate fewer draws");
    CU(cudaSetDevice(g.device));
    cudaStream_t s = g.stream;
    Slot& S = g.slots[kSlots];
    S.staging.reset();
    rc = S.staging.reserve((size_t)n * 8 * 14 + 8192 + (model_out ? (size_t)n * npts * 8 : 0));
    if (rc) return rc;
    // (no mass, q or prior: the caller gives the semi-major axis, and there is no evidence)
    Call c{eb ? 2 : 1, n, {body, 1}, {ebfr, 1}, {}, {P, 1}, {inc, 1}, {ecc, 1}, {argp, 1}, {},
           {R_s, 1}, {u1, 1}, {u2, 1}, {cfr, 1}, {}, nullptr, is_host, scalar_rule};
    tri_col d_a{a, 1};
    rc = stage_call(S, c, s);
    if (!rc) rc = stage(S, d_a, n, s);
    if (rc) return rc;
    LnlArgs A = lnl_args(c, to_col(c.P), to_col(d_a));
    A.raw = 1;
    A.twin_uniform = twin ? 1 : 0;
    double* d_out = S.staging.take<double>(n);
    double* d_model = model_out ? S.staging.take<double>((size_t)n * npts) : nullptr;
    double* d_sec = secdepth_out ? S.staging.take<double>(n) : nullptr;
    S.launches = 0;
    CU(cudaMemsetAsync(S.d_counters, 0, 8 * sizeof(unsigned long long), s));
    A.count = n; A.next = S.d_counters + 2;
    A.out = d_out; A.counters = S.d_counters + 4;
    A.model_out = d_model; A.secdepth_out = d_sec; A.perm = g.d_perm;
    CU(cudaEventRecord(S.ev[0], s));
    CU(cudaEventRecord(S.ev[1], s));
    rc = launch_lnl(S, A, s);
    if (rc) return rc;
    CU(cudaEventRecord(S.ev[2], s));
    CU(cudaEventRecord(S.ev[3], s));
    if (out) CU(cudaMemcpyAsync(out, d_out, (size_t)n * 8, cudaMemcpyDeviceToHost, s));
    if (model_out)
        CU(cudaMemcpyAsync(model_out, d_model, (size_t)n * npts * 8, cudaMemcpyDeviceToHost, s));
    if (secdepth_out)
        CU(cudaMemcpyAsync(secdepth_out, d_sec, (size_t)n * 8, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    S.lnl[0] = S.lnl[1] = nullptr;
    S.N = n;
    g.last = &S;
    return TRI_OK;
}

int tri_lnl_tp(int64_t n, const double* R_p, const double* P_orb, const double* inc,
               const double* a, const double* R_s, const double* u1, const double* u2,
               const double* ecc, const double* argp, const double* cfr, int32_t is_host,
               double* out) {
    return lnl_seam(0, n, R_p, nullptr, P_orb, inc, a, R_s, u1, u2, ecc, argp, cfr, is_host, 0,
                    out);
}

int tri_lnl_eb(int64_t n, const double* R_EB, const double* EB_fluxratio, const double* P_orb,
               const double* inc, const double* a, const double* R_s, const double* u1,
               const double* u2, const double* ecc, const double* argp, const double* cfr,
               int32_t is_host, int32_t twin, double* out) {
    return lnl_seam(1, n, R_EB, EB_fluxratio, P_orb, inc, a, R_s, u1, u2, ecc, argp, cfr,
                    is_host, twin, out);
}

int tri_simulate_tp(int64_t n, const double* R_p, const double* P_orb, const double* inc,
                    const double* a, const double* R_s, const double* u1, const double* u2,
                    const double* ecc, const double* argp, const double* cfr, int32_t is_host,
                    double* flux_out) {
    if (!flux_out) return fail(TRI_EINVAL, "flux_out is NULL");
    return lnl_seam(0, n, R_p, nullptr, P_orb, inc, a, R_s, u1, u2, ecc, argp, cfr, is_host, 1,
                    nullptr, flux_out, nullptr);
}

int tri_simulate_eb(int64_t n, const double* R_EB, const double* EB_fluxratio,
                    const double* P_orb, const double* inc, const double* a, const double* R_s,
                    const double* u1, const double* u2, const double* ecc, const double* argp,
                    const double* cfr, int32_t is_host, int32_t scalar_rule, double* flux_out,
                    double* secdepth_out) {
    if (!flux_out) return fail(TRI_EINVAL, "flux_out is NULL");
    // twin = 1: the secondary-depth cut belongs to lnL_EB_p, not to the simulation
    return lnl_seam(1, n, R_EB, EB_fluxratio, P_orb, inc, a, R_s, u1, u2, ecc, argp, cfr,
                    is_host, 1, nullptr, flux_out, secdepth_out, scalar_rule ? 1 : 0);
}

int tri_fetch_lnl(int32_t branch, double* out, int64_t N) {
    int rc = need_ready(false);
    if (rc) return rc;
    if (branch < 0 || branch > 1 || !out) return fail(TRI_EINVAL, "bad argument");
    if (!g.last || !g.last->lnl[branch] || N != g.last->N)
        return fail(TRI_ESTATE, "no lnL array of that size from the last completed evaluation");
    CU(cudaSetDevice(g.device));
    CU(cudaMemcpy(out, g.last->lnl[branch], (size_t)N * 8, cudaMemcpyDeviceToHost));
    return TRI_OK;
}

int tri_log_mean_exp(const double* logw, int64_t n, tri_result* out) {
    int rc = need_ready(false);
    if (rc) return rc;
    if (!out || n < 0 || (n > 0 && !logw)) return fail(TRI_EINVAL, "bad argument");
    LsePartial z{-INFINITY, 0.0, 0, 0};
    if (n == 0) {
        finish_result(z, 0, out);
        return TRI_OK;
    }
    CU(cudaSetDevice(g.device));
    cudaStream_t s = g.stream;
    Slot& S = g.slots[kSlots];
    S.staging.reset();
    rc = S.staging.reserve((size_t)n * 8 + (size_t)lse_blocks(n) * sizeof(LsePartial) + 8192);
    if (rc) return rc;
    double* d = S.staging.take<double>(n);
    LsePartial* parts = S.staging.take<LsePartial>(lse_blocks(n));
    CU(cudaMemcpyAsync(d, logw, (size_t)n * 8, cudaMemcpyHostToDevice, s));
    {
        int nb = lse_blocks(n);
        lse_partial_kernel<<<nb, kLseThreads, 0, s>>>(d, Col{nullptr, 0}, n, parts);
        lse_final_kernel<<<1, kLseThreads, 0, s>>>(parts, nb, S.d_lse_out);
        CU(cudaGetLastError());
    }
    CU(cudaMemcpyAsync(S.h_lse_out, S.d_lse_out, sizeof(LsePartial), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    finish_result(S.h_lse_out[0], n, out);
    return TRI_OK;
}

int tri_last_timing(double* geometry_ms, double* lnl_ms, double* lse_ms, int32_t* launches) {
    int rc = need_ready(false);
    if (rc) return rc;
    if (!g.last || g.last->N == 0) return fail(TRI_ESTATE, "no timed call yet");
    float a = 0, b = 0, c = 0;
    CU(cudaEventElapsedTime(&a, g.last->ev[0], g.last->ev[1]));
    CU(cudaEventElapsedTime(&b, g.last->ev[1], g.last->ev[2]));
    CU(cudaEventElapsedTime(&c, g.last->ev[2], g.last->ev[3]));
    if (geometry_ms) *geometry_ms = a;
    if (lnl_ms) *lnl_ms = b;
    if (lse_ms) *lse_ms = c;
    if (launches) *launches = g.last->launches;
    return TRI_OK;
}

int tri_dev_splev(const double* t, const double* c, int32_t n, int32_t k, const double* x,
                  double* y, int64_t N, void* stream) {
    int rc = need_ready(false);
    if (rc) return rc;
    if (!t || !c || N < 0 || (N > 0 && (!x || !y))) return fail(TRI_EINVAL, "NULL argument");
    if (k < 1 || k > 5 || n < 2 * (k + 1) || n > kSplevMaxKnots)
        return fail(TRI_EINVAL, "spline degree must be 1..5 and 2(k+1) <= knots <= 512");
    if (N == 0) return TRI_OK;
    CU(cudaSetDevice(g.device));
    cudaStream_t s = (cudaStream_t)stream;   // NULL is the CUDA default stream, as everywhere
    int blocks = (int)std::min<int64_t>((N + 255) / 256, (int64_t)g.sm_count * 8);
    switch (k) {
        case 1: splev_kernel<1><<<blocks, 256, 0, s>>>(t, c, n, x, y, N); break;
        case 2: splev_kernel<2><<<blocks, 256, 0, s>>>(t, c, n, x, y, N); break;
        case 3: splev_kernel<3><<<blocks, 256, 0, s>>>(t, c, n, x, y, N); break;
        case 4: splev_kernel<4><<<blocks, 256, 0, s>>>(t, c, n, x, y, N); break;
        default: splev_kernel<5><<<blocks, 256, 0, s>>>(t, c, n, x, y, N); break;
    }
    CU(cudaGetLastError());
    return TRI_OK;
}

int tri_dev_sample(const tri_sampler_args* a, void* stream) {
    int rc = need_ready(false);
    if (rc) return rc;
    if (!a || a->n < 0) return fail(TRI_EINVAL, "bad argument");
    if (a->n == 0) return TRI_OK;
    if (!a->o_body || !a->o_P || !a->o_inc || !a->o_ecc || !a->o_argp || !a->o_mtot)
        return fail(TRI_EINVAL, "a required output column is NULL");
    if ((a->diluter == 2 && (!a->bg_fr_tess || a->idx_hi <= 0)) ||
        (a->host == 1 && (!a->ldc_u1 || !a->ldc_u2 || !a->err_flag)) ||
        (a->prior_mode != 0 && (!a->cc_sep || !a->cc_con || a->cc_n < 1)))
        return fail(TRI_EINVAL, "a table the scenario needs is NULL");
    if (a->prop && (a->prop_bins < 1 || (a->prop_bins & (a->prop_bins - 1)) != 0 ||
                    !(a->prop_alpha > 0.0 && a->prop_alpha <= 1.0) || !a->o_lnprior))
        return fail(TRI_EINVAL, "a proposal needs a power-of-two bin count, alpha in (0, 1] "
                                "and the lnprior column");
    CU(cudaSetDevice(g.device));
    cudaStream_t s = (cudaStream_t)stream;
    int blocks = (int)std::min<int64_t>((a->n + 255) / 256, (int64_t)g.sm_count * 8);
    sampler_kernel<<<blocks, 256, 0, s>>>(*a);
    CU(cudaGetLastError());
    return TRI_OK;
}

int tri_fp64_peak(double* dfma_per_s) {
    int rc = need_ready(false);
    if (rc) return rc;
    if (!dfma_per_s) return fail(TRI_EINVAL, "NULL argument");
    CU(cudaSetDevice(g.device));
    const int threads = 256, blocks = g.sm_count * 8, iters = 1 << 15;
    double* d = nullptr;
    CU(cudaMalloc(&d, (size_t)threads * blocks * sizeof(double)));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        CU(cudaEventRecord(e0, g.stream));
        dfma_peak_kernel<<<blocks, threads, 0, g.stream>>>(d, iters);
        CU(cudaEventRecord(e1, g.stream));
        CU(cudaEventSynchronize(e1));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, e0, e1));
        double rate = (double)threads * blocks * 8.0 * iters / (ms * 1e-3);
        if (rep > 0 && rate > best) best = rate;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d);
    *dfma_per_s = best;
    return TRI_OK;
}

}  // extern "C"
