// C ABI of libppgpu (include/ppgpu.h): handle management and the level-wise entry points.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/ppgpu.h"
#include "common.cuh"
#include "host_math.hpp"
#include "launch.h"

using namespace ppgpu;

static thread_local std::string g_err;

struct ppgpu_program {
    ReducedProgram host;
    DevProgram dev;
    int device = 0;
    int sm_count = 0;
    std::vector<void*> allocs;
    unsigned long long* d_counters = nullptr;  // CNT_COUNT
    unsigned long long* d_queue = nullptr;     // work-queue heads, one per launch in flight
    int queue_slot = 0;
    long long launches = 0;
    // optional per-family kernel timing (CUDA events on the launch stream)
    bool profiling = false;
    struct Span { int family; cudaEvent_t a, b; };
    std::vector<Span> spans;
    std::vector<cudaEvent_t> event_pool;
    // K2a -> K2 warm hand-over buffers (grown on demand)
    long long warm_cap = 0;
    double* d_warm_resid = nullptr;
    long long* d_warm_idx = nullptr;
    unsigned long long* d_warm_count = nullptr;
    int* d_k2w_order = nullptr;   // scratch for the cost order of the walk's work items (grown on demand)
    size_t k2w_order_cap = 0;
    long long k2w_min = 100000;   // smallest launch the vertex walk (K2w) is used for (ppgpu_set_option)
    bool k2w_ref = false;         // K2w with the reference dictionary updates (PPGPU_OPT_K2W_REF)
    double prof_ms[PPGPU_NUM_FAMILIES] = {0};
    long long prof_launches[PPGPU_NUM_FAMILIES] = {0};
};

struct ProfScope {
    ppgpu_program* p; cudaStream_t st; int family; cudaEvent_t a = nullptr, b = nullptr;
    static cudaEvent_t get(ppgpu_program* p) {
        if (!p->event_pool.empty()) { cudaEvent_t e = p->event_pool.back(); p->event_pool.pop_back(); return e; }
        cudaEvent_t e; cudaEventCreate(&e); return e;
    }
    ProfScope(ppgpu_program* p_, cudaStream_t st_, int fam) : p(p_), st(st_), family(fam) {
        if (p->profiling) { a = get(p); b = get(p); cudaEventRecord(a, st); }
    }
    ~ProfScope() {
        if (a) { cudaEventRecord(b, st); p->spans.push_back({family, a, b}); }
    }
};

static const int QUEUE_SLOTS = 64;
extern "C" { static void warm_release(ppgpu_program* p); }

static int fail(const char* where, cudaError_t e) {
    g_err = std::string(where) + ": " + cudaGetErrorString(e);
    return -1;
}
static int fail_msg(const std::string& m) { g_err = m; return -2; }

template <class T>
static cudaError_t upload(ppgpu_program* p, const std::vector<T>& v, const T** out) {
    void* d = nullptr;
    // 1 KiB zero tail: K2a reads 32-wide row segments of Gam without clamping the last one (k2a_relax.cu)
    const size_t bytes = v.size() * sizeof(T) + 1024;
    cudaError_t e = cudaMalloc(&d, bytes);
    if (e != cudaSuccess) return e;
    p->allocs.push_back(d);
    if ((e = cudaMemset(d, 0, bytes)) != cudaSuccess) return e;
    if (v.size()) e = cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
    *out = (const T*)d;
    return e;
}

static unsigned long long* next_queue(ppgpu_program* p, cudaStream_t st) {
    unsigned long long* q = p->d_queue + p->queue_slot;
    p->queue_slot = (p->queue_slot + 1) % QUEUE_SLOTS;
    cudaMemsetAsync(q, 0, sizeof(unsigned long long), st);
    return q;
}

extern "C" {

const char* ppgpu_last_error(void) { return g_err.c_str(); }
int ppgpu_version(void) { return 100; }

int ppgpu_program_create(const ppgpu_dims* d, const double* A, const double* b, const double* F, const double* A_t,
                         const double* b_t, const double* Q, const double* c, const double* H, int device,
                         ppgpu_program** out) {
    if (!d || !out) return fail_msg("null argument");
    if (d->is_qp && !Q) return fail_msg("is_qp set but Q is NULL");
    ppgpu_program* p = new ppgpu_program();
    if (!reduce_program(d->n, d->t, d->m, d->q, d->n_eq, d->is_qp, A, b, F, A_t, b_t, Q, c, H, p->host)) {
        std::string m = "program reduction failed: " + p->host.error;
        delete p;
        return fail_msg(m);
    }
    const ReducedProgram& R = p->host;
    if (R.W > 4) { delete p; return fail_msg("more than 256 inequality rows are not supported"); }
    if (R.R0 > 256) { delete p; return fail_msg("more than 256 region rows ((m - n_eq) + q) are not supported"); }
    if (k2_pad_columns(R.nfree + 2) < 0) { delete p; return fail_msg("n - n_eq + t + 2 > 64 columns are not supported"); }
    if (R.t + 2 > 16) { delete p; return fail_msg("more than 14 parameters are not supported"); }
    if (R.np > 64) { delete p; return fail_msg("n - n_eq > 64 is not supported"); }
    {
        // region emission (K5) factors the (n + k) x (n + k) KKT matrix of a candidate in shared memory: check the deepest level
        // now instead of failing with "invalid argument" in the middle of a solve (k5_emit.cu::launch_k5_t)
        const int depth = (R.n > R.t ? R.n : R.t) - R.ne, k = R.ne + (depth > 0 ? depth : 0), N = R.n + k, ld = N + R.t + 1;
        const size_t smem = ((size_t)N * ld + (size_t)R.R0 * (R.t + 1)) * sizeof(double) + (size_t)(2 * R.R0 + k + 2) * sizeof(int);
        if (smem > 200 * 1024) {
            delete p;
            return fail_msg("region emission needs " + std::to_string(smem / 1024) + " KB of shared memory at the deepest level (n + k = " +
                            std::to_string(N) + "); the limit is 200 KB (about n + k <= 150)");
        }
    }
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) { delete p; return fail("cudaSetDevice", e); }
    p->device = device;
    cudaDeviceGetAttribute(&p->sm_count, cudaDevAttrMultiProcessorCount, device);
    DevProgram& D = p->dev;
    D.n = R.n; D.t = R.t; D.m = R.m; D.q = R.q; D.ne = R.ne; D.is_qp = R.is_qp;
    D.mi = R.mi; D.np = R.np; D.W = R.W; D.R0 = R.R0; D.nfree = R.nfree; D.use_gram = R.use_gram;
    D.dc0 = R.nfree + 2;
#define UP(field, vecname) if ((e = upload(p, R.vecname, &D.field)) != cudaSuccess) { ppgpu_program_destroy(p); return fail("upload " #field, e); }
    UP(At, At) UP(C1, C1) UP(T0, T0) UP(Gam, Gam) UP(G, G) UP(V, V) UP(th_lo, th_lo) UP(th_hi, th_hi) UP(A, A) UP(b, b) UP(F, F) UP(A_t, At_theta) UP(b_t, bt) UP(Q, Q) UP(c, c) UP(H, H)
    UP(Xp, Xp) UP(K, K) UP(Pm, Pm)
#undef UP
    D.wk_ok = R.wk_ok; D.wk_nb = R.wk_nb; D.wk_ld = R.wk_ld; D.wk_D0 = nullptr; D.wk_bvar = nullptr; D.wk_nvar = nullptr;
    if (R.wk_ok) {
        if ((e = upload(p, R.wk_D0, &D.wk_D0)) != cudaSuccess || (e = upload(p, R.wk_bvar, &D.wk_bvar)) != cudaSuccess ||
            (e = upload(p, R.wk_nvar, &D.wk_nvar)) != cudaSuccess) { ppgpu_program_destroy(p); return fail("upload walk dictionary", e); }
    }
    D.lp_ok = R.lp_ok; D.lp_ld = R.lp_ld; D.lp_D0 = nullptr; D.lp_bvar = nullptr; D.lp_nvar = nullptr; D.lp_obj = nullptr;
    D.X0t = nullptr; D.Q2 = nullptr;
    if (R.lp_ok) {
        if ((e = upload(p, R.lp_D0, &D.lp_D0)) != cudaSuccess || (e = upload(p, R.lp_bvar, &D.lp_bvar)) != cudaSuccess ||
            (e = upload(p, R.lp_nvar, &D.lp_nvar)) != cudaSuccess || (e = upload(p, R.lp_obj, &D.lp_obj)) != cudaSuccess ||
            (e = upload(p, R.X0t, &D.X0t)) != cudaSuccess || (e = upload(p, R.Q2, &D.Q2)) != cudaSuccess) {
            ppgpu_program_destroy(p);
            return fail("upload LP start dictionary", e);
        }
    }
    void* dc = nullptr;
    if ((e = cudaMalloc(&dc, (CNT_COUNT + QUEUE_SLOTS) * sizeof(unsigned long long))) != cudaSuccess) {
        ppgpu_program_destroy(p);
        return fail("cudaMalloc counters", e);
    }
    p->allocs.push_back(dc);
    cudaMemset(dc, 0, (CNT_COUNT + QUEUE_SLOTS) * sizeof(unsigned long long));
    p->d_counters = (unsigned long long*)dc;
    p->d_queue = p->d_counters + CNT_COUNT;
    *out = p;
    return 0;
}

int ppgpu_program_destroy(ppgpu_program* p) {
    if (!p) return 0;
    for (void* d : p->allocs) cudaFree(d);
    if (p->d_k2w_order) cudaFree(p->d_k2w_order);
    warm_release(p);
    for (auto& s : p->spans) { cudaEventDestroy(s.a); cudaEventDestroy(s.b); }
    for (cudaEvent_t e : p->event_pool) cudaEventDestroy(e);
    delete p;
    return 0;
}

int ppgpu_set_option(ppgpu_program* p, int32_t option, int64_t value) {
    if (!p) return fail_msg("null argument");
    switch (option) {
        case PPGPU_OPT_K2W_MIN: p->k2w_min = value; return 0;
        case PPGPU_OPT_K2W_REF: p->k2w_ref = value != 0; return 0;
        default: return fail_msg("unknown option");
    }
}

int ppgpu_program_info(const ppgpu_program* p, ppgpu_info* o) {
    if (!p || !o) return fail_msg("null argument");
    const ReducedProgram& R = p->host;
    o->words = R.W; o->n_ineq = R.mi; o->region_rows = R.R0; o->use_gram = R.use_gram;
    o->max_depth = (R.n > R.t ? R.n : R.t) - R.ne;
    o->sm_count = p->sm_count;
    o->lp_columns = k2_pad_columns(R.nfree + 2);
    o->reserved = R.wk_ok;
    return 0;
}

int ppgpu_root_level(ppgpu_program* p, uint64_t* d_masks, int64_t* h_count, ppgpu_stream stream) {
    if (!p || !h_count) return fail_msg("null argument");
    long long cnt = 0;
    cudaError_t e = root_level(p->dev, d_masks, &cnt, (cudaStream_t)stream);
    if (e != cudaSuccess) return fail("root_level", e);
    p->launches += cnt > 0;
    *h_count = cnt;
    return 0;
}

// candidates of one ppgpu_level_eval call are processed in chunks of this many, so that the K2a -> K2 hand-over buffers
// (one residual vector per uncertified candidate) stay bounded however large the level is
static long long level_chunk() {
    static const long long c = getenv("PPGPU_CHUNK") ? atoll(getenv("PPGPU_CHUNK")) : (1ll << 22);
    return c < 1024 ? 1024 : c;
}
// with the vertex walk in front, the relaxation leaves next to nothing for the hand-over: the level can be one launch
// (one kernel tail per level instead of one per 2^22 candidates, and the walk's longest-first scheduling sees every prefix)
static long long walk_chunk() {
    static const long long c = getenv("PPGPU_WALK_CHUNK") ? atoll(getenv("PPGPU_WALK_CHUNK")) : (1ll << 27);
    return c < 1024 ? 1024 : c;
}

// Hand-over buffers are recycled through a small process-wide pool: a solve creates a program, runs a handful of levels
// and destroys it, and cudaMalloc/cudaFree of a few hundred MB per solve cost more than the kernels of small programs.
// A buffer belongs to exactly one live program at a time.
struct WarmBuf { int device; size_t resid_bytes, idx_bytes; double* resid; long long* idx; };
static std::mutex g_pool_mu;
static std::vector<WarmBuf> g_pool;

static void warm_release(ppgpu_program* p) {
    if (!p->d_warm_resid) return;
    std::lock_guard<std::mutex> lk(g_pool_mu);
    if (g_pool.size() < 4) {
        g_pool.push_back({p->device, (size_t)p->warm_cap * p->dev.R0 * sizeof(double),
                          (size_t)p->warm_cap * sizeof(long long), p->d_warm_resid, p->d_warm_idx});
    } else {
        cudaFree(p->d_warm_resid);
        cudaFree(p->d_warm_idx);
    }
    p->d_warm_resid = nullptr; p->d_warm_idx = nullptr; p->warm_cap = 0;
}

static cudaError_t ensure_warm(ppgpu_program* p, long long cap, cudaStream_t st) {
    if (!p->d_warm_count) {
        cudaError_t e = cudaMalloc((void**)&p->d_warm_count, sizeof(unsigned long long));
        if (e != cudaSuccess) return e;
        p->allocs.push_back(p->d_warm_count);
    }
    if (cap <= p->warm_cap) return cudaSuccess;
    // two sizes only (small levels / full chunks), so a solve grows its buffers at most twice
    const long long full = 4096 + level_chunk() / 8;
    const long long want = cap <= 65536 ? 65536 : (cap > full ? cap : full);   // (walked launches: n / 64 <= 2^27 / 64 = 4 full)
    cudaError_t e = cudaStreamSynchronize(st);   // earlier launches may still read the old buffers
    if (e != cudaSuccess) return e;
    warm_release(p);
    const size_t rb = (size_t)want * p->dev.R0 * sizeof(double), ib = (size_t)want * sizeof(long long);
    {
        std::lock_guard<std::mutex> lk(g_pool_mu);
        for (size_t i = 0; i < g_pool.size(); ++i) {
            if (g_pool[i].device == p->device && g_pool[i].resid_bytes >= rb && g_pool[i].idx_bytes >= ib) {
                p->d_warm_resid = g_pool[i].resid; p->d_warm_idx = g_pool[i].idx; p->warm_cap = want;
                g_pool.erase(g_pool.begin() + i);
                return cudaSuccess;
            }
        }
    }
    if ((e = cudaMalloc((void**)&p->d_warm_resid, rb)) != cudaSuccess) return e;
    if ((e = cudaMalloc((void**)&p->d_warm_idx, ib)) != cudaSuccess) { cudaFree(p->d_warm_resid); p->d_warm_resid = nullptr; return e; }
    p->warm_cap = want;
    return cudaSuccess;
}

static_assert(PPGPU_WITNESS_SLOTS == PPG_WITNESS_SLOTS, "witness slots: include/ppgpu.h and csrc/tolerances.h disagree");
// what ppgpu_level_eval_w adds to a level evaluation (all optional)
struct WitnessIo {
    uint64_t* out = nullptr;                 // n x slots x W: witnesses of the candidates the walk certifies / that inherit one
    const uint64_t* parent_feas = nullptr;   // parent level: feasible masks (nf x W), K6 workspace with their group index,
    long long parent_nf = 0;                 // and the witnesses of those parents in the same order
    const void* parent_ws = nullptr;
    const uint64_t* parent_wit = nullptr;
};

static int level_eval_chunk(ppgpu_program* p, const uint64_t* d_masks, int64_t n, int32_t k_act, uint8_t* d_status,
                            int32_t stages, cudaStream_t st, const WitnessIo& wio) {
    cudaError_t e;
    if (stages & 1) {
        ProfScope ps(p, st, 0);
        // K1 is two passes over the same bytes (thread-per-candidate prefilter, then QR of what it could not clear): in
        // pieces of 2^22 candidates the second pass finds masks and status in L2 (one 70 M-candidate launch: 9.8 vs 7.0 ms)
        const long long piece = 1ll << 22;
        for (long long off = 0; off < n; off += piece) {
            const long long nn = n - off < piece ? n - off : piece;
            e = launch_k1(p->dev, d_masks + (size_t)off * p->dev.W, nn, k_act, d_status + off, p->d_counters, p->sm_count, st);
            if (e != cudaSuccess) return fail("K1 rank", e);
            if (k_act >= 1 && k_act <= 8) p->launches++;  // prefilter + QR
            p->launches++;
            if (k_act >= 2 && k_act <= p->dev.np) p->launches++;   // singular-value re-check of borderline decisions
        }
    }
    if ((stages & 2) && !(stages & 8) && wio.parent_feas && wio.parent_wit && wio.parent_ws && wio.parent_nf > 0) {
        // certificates inherited from the parents' witness vertices: what they cover never reaches the walk
        ProfScope ps(p, st, 9);
        e = launch_inherit(p->dev, d_masks, n, d_status, wio.out, wio.parent_feas, wio.parent_nf, wio.parent_ws,
                           wio.parent_wit, p->d_counters, st);
        if (e != cudaSuccess) return fail("witness inheritance", e);
        p->launches++;
    }
    static const int warm_on = getenv("PPGPU_WARM") ? atoi(getenv("PPGPU_WARM")) : 1;
    p->dev.warm_count = nullptr; p->dev.warm_resid = nullptr; p->dev.warm_idx = nullptr; p->dev.warm_cap = 0;
    // (measured: leaving what inheritance does not cover at the last level to the relaxation instead of the walk is slower -
    // the 14 % of level 5 of the bench program that no parent covers cost K2a + K2 134 ms against the walk's 111)
    if ((stages & 2) && !(stages & 8) && k_act >= 1 && p->k2w_min >= 0 && n >= p->k2w_min) {
        // certificates shared between the candidates of a prefix (vertex walk); the relaxation only sees what is left
        ProfScope ps(p, st, 8);
        bool handled = false;
        const size_t want = k2w_order_scratch_ints(walk_chunk());   // one allocation per handle, sized for the largest launch
        if (want > p->k2w_order_cap) {
            // (earlier launches may still read the old buffer)
            if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return fail("K2w order scratch", e);
            if (p->d_k2w_order) cudaFree(p->d_k2w_order);
            p->d_k2w_order = nullptr; p->k2w_order_cap = 0;
            if ((e = cudaMalloc((void**)&p->d_k2w_order, want * sizeof(int))) != cudaSuccess) return fail("K2w order scratch", e);
            p->k2w_order_cap = want;
        }
        e = launch_k2w(p->dev, d_masks, n, k_act, d_status, next_queue(p, st), p->d_counters, p->sm_count, st, &handled, wio.out, p->d_k2w_order,
                       p->k2w_ref);
        if (e != cudaSuccess) return fail("K2w vertex walk", e);
        if (handled) p->launches += (n > 128ll * 8 * p->sm_count) ? 4 : 1;   // + the three kernels that order the work items
    }
    if ((stages & 2) && !(stages & 8)) {
        // feasibility certificates first (cheap); the simplex only sees what is left, and starts from K2a's last iterate
        ProfScope ps(p, st, 7);
        static const int iters = getenv("PPGPU_K2A_ITERS") ? atoi(getenv("PPGPU_K2A_ITERS")) : 96;
        if (iters > 0 && k_act >= 0) {
            if (warm_on) {
                const bool walked = k_act >= 1 && p->dev.wk_ok && p->k2w_min >= 0 && n >= p->k2w_min;
                const long long cap = n < 4096 ? n : 4096 + n / (walked ? 64 : 8);
                if ((e = ensure_warm(p, cap, st)) != cudaSuccess) return fail("warm-start buffers", e);
                p->dev.warm_count = p->d_warm_count; p->dev.warm_resid = p->d_warm_resid;
                p->dev.warm_idx = p->d_warm_idx; p->dev.warm_cap = cap;
                cudaMemsetAsync(p->d_warm_count, 0, sizeof(unsigned long long), st);
            }
            e = launch_k2a(p->dev, d_masks, n, k_act, d_status, next_queue(p, st), p->d_counters, iters,
                           p->sm_count, st);
            if (e != cudaSuccess) return fail("K2a relaxation", e);
            p->launches++;
        }
    }
    if (stages & 2) {
        ProfScope ps(p, st, 1);
        e = launch_k2(p->dev, d_masks, n, d_status, next_queue(p, st), p->d_counters, p->sm_count, st);
        if (e != cudaSuccess) return fail("K2 feasibility", e);
        p->launches++;
        if (p->dev.warm_count) {
            // candidates the warm solve found infeasible keep their hand-over mark until here, so that the cold scan of
            // the same launch does not solve them a second time
            if ((e = launch_clear_bits(d_status, n, PPG_ST_PRE, st)) != cudaSuccess) return fail("status clean-up", e);
            p->launches++;
        }
    }
    if (stages & 4) {
        ProfScope ps(p, st, 2);
        if (p->dev.is_qp && p->dev.use_gram) {
            e = launch_k34(p->dev, d_masks, n, k_act, d_status, next_queue(p, st), p->d_counters, p->sm_count, st);
            if (k_act >= 1 && k_act <= 8) p->launches++;  // the thread-per-candidate prefilter is a launch of its own
        } else {
            e = launch_mark_general(p->dev, n, k_act, d_status, st);
        }
        if (e != cudaSuccess) return fail("K3/K4 optimality screen", e);
        p->launches++;
    }
    return 0;
}

int ppgpu_level_eval(ppgpu_program* p, const uint64_t* d_masks, int64_t n, int32_t k_act, uint8_t* d_status,
                     int32_t stages, ppgpu_stream stream) {
    return ppgpu_level_eval_w(p, d_masks, n, k_act, d_status, stages, nullptr, nullptr, 0, nullptr, nullptr, stream);
}

int ppgpu_level_eval_w(ppgpu_program* p, const uint64_t* d_masks, int64_t n, int32_t k_act, uint8_t* d_status,
                       int32_t stages, uint64_t* d_witness, const uint64_t* d_parent_feas, int64_t parent_nf,
                       const void* d_parent_ws, const uint64_t* d_parent_wit, ppgpu_stream stream) {
    if (!p) return fail_msg("null argument");
    if (n <= 0) return 0;
    WitnessIo wio;
    wio.parent_feas = d_parent_feas; wio.parent_nf = parent_nf; wio.parent_ws = d_parent_ws; wio.parent_wit = d_parent_wit;
    const bool walk = (stages & 2) && !(stages & 8) && k_act >= 1 && p->dev.wk_ok && p->k2w_min >= 0 && n >= p->k2w_min;
    const long long chunk = walk ? walk_chunk() : level_chunk();
    for (int64_t off = 0; off < n; off += chunk) {
        const int64_t nn = n - off < chunk ? n - off : chunk;
        wio.out = d_witness ? d_witness + (size_t)off * PPGPU_WITNESS_SLOTS * p->dev.W : nullptr;
        const int rc = level_eval_chunk(p, d_masks + (size_t)off * p->dev.W, nn, k_act, d_status + off, stages,
                                        (cudaStream_t)stream, wio);
        if (rc) return rc;
    }
    return 0;
}

size_t ppgpu_scan_workspace_bytes(int64_t n) { return scan_workspace_bytes(n); }
size_t ppgpu_select_workspace_bytes(int64_t n) { return select_workspace_bytes(n); }

int ppgpu_level_select(ppgpu_program* p, const uint8_t* d_status, int64_t n, uint8_t bits, uint8_t value,
                       int64_t* d_idx_out, int64_t* h_count, void* d_ws, size_t ws_bytes, ppgpu_stream stream) {
    if (!p || !h_count) return fail_msg("null argument");
    *h_count = 0;
    if (n <= 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    // the count lands in the last workspace word, then comes back to the host
    if (ws_bytes < select_workspace_bytes(n)) return fail_msg("workspace too small");
    long long* d_count = (long long*)d_ws + (select_workspace_bytes(n) / sizeof(long long) - 1);
    cudaError_t e;
    {
        ProfScope ps(p, st, 6);
        e = select_indices(d_status, n, bits, value, (long long*)d_idx_out, d_count, d_ws, ws_bytes - sizeof(long long), st);
    }
    if (e != cudaSuccess) return fail("select", e);
    p->launches += 5;
    long long cnt = 0;
    e = cudaMemcpyAsync(&cnt, d_count, sizeof(long long), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return fail("select count", e);
    *h_count = cnt;
    return 0;
}

int ppgpu_regions_emit(ppgpu_program* p, const uint64_t* d_masks, const int64_t* d_sel, int64_t n_sel, int32_t k_act,
                       double* d_laws, double* d_rows, int32_t* d_flags, double* d_info, uint8_t* d_status,
                       ppgpu_stream stream) {
    if (!p) return fail_msg("null argument");
    if (n_sel <= 0) return 0;
    cudaError_t e;
    {
        ProfScope ps(p, (cudaStream_t)stream, 3);
        e = launch_k5(p->dev, d_masks, (const long long*)d_sel, n_sel, k_act, d_laws, d_rows, d_flags, d_info, d_status,
                      next_queue(p, (cudaStream_t)stream), p->d_counters, p->sm_count, (cudaStream_t)stream);
    }
    if (e != cudaSuccess) return fail("K5 emit", e);
    p->launches += k5_launches(p->dev.t);
    return 0;
}

int ppgpu_children_count(ppgpu_program* p, const uint64_t* d_masks, const int64_t* d_feas_idx, int64_t nf,
                         int32_t k_act, uint64_t* d_feas_masks, uint64_t* d_survive, int64_t* d_offsets,
                         int64_t* h_total, void* d_ws, size_t ws_bytes, ppgpu_stream stream) {
    if (!p || !h_total) return fail_msg("null argument");
    *h_total = 0;
    if (nf <= 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e;
    {
        ProfScope ps(p, st, 4);
        e = children_count(p->dev, d_masks, (const long long*)d_feas_idx, nf, k_act, d_feas_masks, d_survive,
                           (long long*)d_offsets, d_ws, ws_bytes, p->d_counters, st);
    }
    if (e != cudaSuccess) return fail("K6 count", e);
    p->launches += 12;   // prepare 8, count 1, scan 3
    long long tot = 0, disorder = 0;
    e = cudaMemcpyAsync(&tot, (long long*)d_offsets + nf, sizeof(long long), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&disorder, children_order_flag(d_ws, nf), sizeof(long long), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return fail("K6 total", e);
    if (disorder) return fail_msg("K6: the feasible parents are not one level's sets in lexicographic order");
    *h_total = tot;
    return 0;
}

int ppgpu_children_prepare(ppgpu_program* p, const uint64_t* d_masks, const int64_t* d_feas_idx, int64_t nf,
                           uint64_t* d_feas_masks, void* d_ws, size_t ws_bytes, ppgpu_stream stream) {
    if (!p) return fail_msg("null argument");
    if (nf <= 0) return 0;
    cudaError_t e;
    {
        ProfScope ps(p, (cudaStream_t)stream, 4);
        e = children_prepare(p->dev, d_masks, (const long long*)d_feas_idx, nf, d_feas_masks, d_ws, ws_bytes, (cudaStream_t)stream);
    }
    if (e != cudaSuccess) return fail("K6 prepare", e);
    p->launches += 8;    // gather, run flags, scan 3, groups, table clear, table insert (+ a memset)
    return 0;
}

int ppgpu_children_count_range(ppgpu_program* p, const uint64_t* d_feas_masks, int64_t nf, int32_t k_act,
                               uint64_t* d_survive, int64_t* d_counts, int64_t p_lo, int64_t p_hi, void* d_ws,
                               size_t ws_bytes, ppgpu_stream stream) {
    if (!p) return fail_msg("null argument");
    if (p_lo < 0 || p_hi > nf || p_lo > p_hi) return fail_msg("parent range outside [0, nf]");
    if (nf <= 0 || p_hi == p_lo) return 0;
    if (ws_bytes < scan_workspace_bytes(nf)) return fail_msg("workspace too small");
    cudaError_t e;
    {
        ProfScope ps(p, (cudaStream_t)stream, 4);
        e = children_count_range(p->dev, d_feas_masks, nf, k_act, d_survive, (long long*)d_counts, p_lo, p_hi, d_ws,
                                 p->d_counters, (cudaStream_t)stream);
    }
    if (e != cudaSuccess) return fail("K6 count", e);
    p->launches++;
    return 0;
}

int ppgpu_children_scan(ppgpu_program* p, int64_t* d_counts_to_offsets, int64_t nf, int64_t* h_total, void* d_ws,
                        size_t ws_bytes, ppgpu_stream stream) {
    if (!p || !h_total) return fail_msg("null argument");
    *h_total = 0;
    if (nf <= 0) return 0;
    if (ws_bytes < scan_workspace_bytes(nf)) return fail_msg("workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e;
    {
        ProfScope ps(p, st, 4);
        e = children_scan((long long*)d_counts_to_offsets, nf, d_ws, st);
    }
    if (e != cudaSuccess) return fail("K6 scan", e);
    p->launches += 2;
    long long tot = 0, disorder = 0;
    e = cudaMemcpyAsync(&tot, (long long*)d_counts_to_offsets + nf, sizeof(long long), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&disorder, children_order_flag(d_ws, nf), sizeof(long long), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return fail("K6 total", e);
    if (disorder) return fail_msg("K6: the feasible parents are not one level's sets in lexicographic order");
    *h_total = tot;
    return 0;
}

int ppgpu_children_write(ppgpu_program* p, const uint64_t* d_feas_masks, const uint64_t* d_survive,
                         const int64_t* d_offsets, int64_t nf, uint64_t* d_children, ppgpu_stream stream) {
    if (!p) return fail_msg("null argument");
    cudaError_t e;
    {
        ProfScope ps(p, (cudaStream_t)stream, 5);
        e = children_write(p->dev, d_feas_masks, d_survive, (const long long*)d_offsets, nf, d_children, (cudaStream_t)stream);
    }
    if (e != cudaSuccess) return fail("K6 write", e);
    p->launches += nf > 0;
    return 0;
}

int ppgpu_counters(ppgpu_program* p, uint64_t* h_out, int32_t reset, ppgpu_stream stream) {
    if (!p || !h_out) return fail_msg("null argument");
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemcpyAsync(h_out, p->d_counters, CNT_COUNT * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e == cudaSuccess && reset) e = cudaMemsetAsync(p->d_counters, 0, CNT_COUNT * sizeof(unsigned long long), st);
    if (e != cudaSuccess) return fail("counters", e);
    return 0;
}

int64_t ppgpu_launch_count(const ppgpu_program* p) { return p ? p->launches : 0; }

int ppgpu_profile_enable(ppgpu_program* p, int32_t on) {
    if (!p) return fail_msg("null argument");
    p->profiling = on != 0;
    return 0;
}

int ppgpu_profile_read(ppgpu_program* p, double* h_ms, int64_t* h_launches, int32_t reset) {
    if (!p || !h_ms || !h_launches) return fail_msg("null argument");
    for (auto& s : p->spans) {
        cudaError_t e = cudaEventSynchronize(s.b);
        if (e != cudaSuccess) return fail("profile sync", e);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, s.a, s.b);
        p->prof_ms[s.family] += ms;
        p->prof_launches[s.family] += 1;
        p->event_pool.push_back(s.a);
        p->event_pool.push_back(s.b);
    }
    p->spans.clear();
    for (int f = 0; f < PPGPU_NUM_FAMILIES; ++f) { h_ms[f] = p->prof_ms[f]; h_launches[f] = p->prof_launches[f]; }
    if (reset) for (int f = 0; f < PPGPU_NUM_FAMILIES; ++f) { p->prof_ms[f] = 0; p->prof_launches[f] = 0; }
    return 0;
}

int ppgpu_locate_points(const double* d_theta, int64_t n_points, int32_t t, const double* d_rows, const int64_t* d_row_off,
                        int64_t n_regions, const double* d_laws, int32_t n_x, int32_t use_tol, double tol, int32_t overlap,
                        const double* d_Q, const double* d_H, const double* d_c, int32_t* d_region, double* d_x,
                        ppgpu_stream stream) {
    if (n_points < 0 || n_regions < 0 || n_x < 0) return fail_msg("negative size");
    if (n_points == 0) return 0;
    if (!d_theta || !d_region || !d_row_off || (n_regions > 0 && !d_rows)) return fail_msg("null argument");
    if ((d_x || overlap) && n_x > 0 && n_regions > 0 && !d_laws) return fail_msg("laws needed (d_x or overlap) but d_laws is NULL");
    if (t < 1 || t > 32) return fail_msg("point location supports 1 <= t <= 32 parameters");
    if (overlap && (n_x < 1 || n_x > 128)) return fail_msg("the overlapping rule supports 1 <= n_x <= 128 variables");
    if (overlap && (!d_H || !d_c)) return fail_msg("the overlapping rule needs the objective (d_H, d_c; d_Q for an mpQP)");
    int dev = 0, sms = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return fail("device query", e);
    e = launch_locate(d_theta, n_points, t, d_rows, (const long long*)d_row_off, n_regions, d_laws, n_x, use_tol, tol,
                      overlap ? 1 : 0, d_Q, d_H, d_c, d_region, d_x, sms, (cudaStream_t)stream);
    if (e != cudaSuccess) return fail("K7 point location", e);
    return 0;
}

int ppgpu_solve_theta_batch(ppgpu_program* p, const double* d_theta, int64_t n_points, uint8_t* d_status, double* d_x,
                            double* d_dual, uint64_t* d_active, int32_t* d_iters, ppgpu_stream stream) {
    if (!p) return fail_msg("null argument");
    if (!p->dev.is_qp || !p->dev.use_gram)
        return fail_msg("solve_theta needs an mpQP whose Hessian is positive definite on the reduced space (use_gram = 0)");
    if (n_points < 0) return fail_msg("negative size");
    if (n_points == 0) return 0;
    if (!d_theta || !d_status) return fail_msg("null argument");
    cudaError_t e = cudaSetDevice(p->device);
    if (e == cudaSuccess)
        e = launch_theta_qp(p->dev, d_theta, n_points, d_status, d_x, d_dual, d_active, d_iters, p->sm_count, (cudaStream_t)stream);
    if (e != cudaSuccess) return fail("K8 fixed-theta QP", e);
    p->launches++;
    return 0;
}

int ppgpu_solve_theta_lp_batch(ppgpu_program* p, const double* d_theta, int64_t n_points, uint8_t* d_status, double* d_x,
                               double* d_dual, uint64_t* d_active, int32_t* d_iters, ppgpu_stream stream) {
    if (!p) return fail_msg("null argument");
    if (p->dev.is_qp) return fail_msg("solve_theta_lp needs an mpLP handle (this one is an mpQP: ppgpu_solve_theta_batch)");
    if (!p->dev.lp_ok) return fail_msg("solve_theta_lp: the reduced inequality rows have rank below n - n_eq, the LP has no vertex");
    if (n_points < 0) return fail_msg("negative size");
    if (n_points == 0) return 0;
    if (!d_theta || !d_status) return fail_msg("null argument");
    cudaError_t e = cudaSetDevice(p->device);
    if (e == cudaSuccess)
        e = launch_theta_lp(p->dev, d_theta, n_points, d_status, d_x, d_dual, d_active, d_iters, p->sm_count, (cudaStream_t)stream);
    if (e != cudaSuccess) return fail("K9 fixed-theta LP", e);
    p->launches++;
    return 0;
}

int ppgpu_chebyshev_batch(const double* d_rows, const int64_t* d_row_off, int64_t n_polytopes, int32_t t, int32_t max_rows,
                          double* d_radius, int32_t* d_code, ppgpu_stream stream) {
    if (n_polytopes < 0) return fail_msg("negative size");
    if (n_polytopes == 0) return 0;
    if (!d_rows || !d_row_off || !d_radius || !d_code) return fail_msg("null argument");
    if (t < 1 || t > 30) return fail_msg("the Chebyshev batch supports 1 <= t <= 30 parameters");
    if (max_rows < 1 || max_rows > 1024) return fail_msg("the Chebyshev batch supports 1..1024 rows per polytope");
    int dev = 0, sms = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return fail("device query", e);
    e = launch_cheb_batch(d_rows, (const long long*)d_row_off, n_polytopes, t, max_rows, d_radius, d_code, sms, (cudaStream_t)stream);
    if (e != cudaSuccess) return fail("Chebyshev batch", e);
    return 0;
}

}  // extern "C"

// ---- K11: the relaxation tree of a mixed-integer program (a handle of its own: none of the path's limits apply)
struct ppgpu_tree {
    TreeProgram host;
    DevTree dev;
    int device = 0;
    int sm_count = 0;
    bool inherit = false;
    std::vector<void*> allocs;
};

template <class T>
static cudaError_t tree_upload(ppgpu_tree* h, const std::vector<T>& v, const T** out) {
    void* d = nullptr;
    const size_t bytes = (v.size() ? v.size() : 1) * sizeof(T);
    cudaError_t e = cudaMalloc(&d, bytes);
    if (e != cudaSuccess) return e;
    h->allocs.push_back(d);
    if (v.size()) e = cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
    *out = (const T*)d;
    return e;
}

extern "C" {

int ppgpu_tree_create(const ppgpu_dims* d, const int32_t* binary_indices, int32_t nb, const double* A, const double* b,
                      const double* F, const double* A_t, const double* b_t, int device, ppgpu_tree** out) {
    if (!d || !out || (nb > 0 && !binary_indices)) return fail_msg("null argument");
    if (nb < 0 || nb > 63) return fail_msg("the tree supports 0 <= nb <= 63 binaries (a node is one uint64 of fixed bits)");
    ppgpu_tree* h = new ppgpu_tree();
    std::vector<int> bin(binary_indices, binary_indices + nb);
    if (!build_tree_dictionary(d->n, d->t, d->m, d->q, d->n_eq, nb, bin.data(), A, b, F, A_t, b_t, h->host)) {
        std::string m = "tree: " + h->host.error;
        delete h;
        return fail_msg(m);
    }
    const TreeProgram& R = h->host;
    // K11 keeps a node's dictionary in the shared memory of one warp: K9's envelope
    if (R.rows > 256) {
        std::string m = "tree: the lifted system has " + std::to_string(R.rows) +
                        " inequality rows ((m - n_eq) + q + 2 nb); at most 256 are supported";
        delete h;
        return fail_msg(m);
    }
    if (R.cols > 64) {
        std::string m = "tree: the lifted system has " + std::to_string(R.cols) +
                        " free variables (n + t - n_eq); at most 64 are supported";
        delete h;
        return fail_msg(m);
    }
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) { delete h; return fail("cudaSetDevice", e); }
    h->device = device;
    cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device);
    const char* env = getenv("PPGPU_TREE_INHERIT");
    h->inherit = env && atoi(env) != 0;
    DevTree& D = h->dev;
    D.nv = R.nv; D.rows = R.rows; D.cols = R.cols; D.rb0 = R.rb0; D.tp = R.tp; D.ld = R.ld; D.ne = R.ne; D.nb = R.nb;
#define UP(field, vecname) if ((e = tree_upload(h, R.vecname, &D.field)) != cudaSuccess) { ppgpu_tree_destroy(h); return fail("tree upload " #field, e); }
    UP(D0, D0) UP(bvar, bvar) UP(nvar, nvar) UP(hs, hs) UP(z0, z0) UP(Q2, Q2) UP(Arows, Arows) UP(brows, brows) UP(bin, bin)
#undef UP
    *out = h;
    return 0;
}

int ppgpu_tree_destroy(ppgpu_tree* h) {
    if (!h) return 0;
    for (void* d : h->allocs) cudaFree(d);
    delete h;
    return 0;
}

int ppgpu_tree_set_option(ppgpu_tree* h, int32_t option, int64_t value) {
    if (!h) return fail_msg("null argument");
    switch (option) {
        case PPGPU_TREE_OPT_INHERIT: h->inherit = value != 0; return 0;
        default: return fail_msg("unknown option");
    }
}

int ppgpu_tree_eval(ppgpu_tree* h, const uint64_t* d_nodes, int64_t n, int32_t depth, uint8_t* d_status, double* d_point,
                    const double* d_parent_point, const int64_t* d_parent_of, int32_t* d_iters, ppgpu_stream stream) {
    if (!h) return fail_msg("null argument");
    if (n < 0) return fail_msg("negative size");
    if (depth < 0 || depth > h->host.nb) return fail_msg("depth outside [0, nb]");
    if (n == 0) return 0;
    if (!d_nodes || !d_status) return fail_msg("null argument");
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaSetDevice(h->device);
    if (e != cudaSuccess) return fail("cudaSetDevice", e);
    const bool inherit = h->inherit && depth >= 1 && d_parent_point && d_parent_of;
    if (inherit) {
        e = launch_tree_inherit(h->dev, d_nodes, n, depth, d_parent_point, (const long long*)d_parent_of, d_status, d_point,
                                d_iters, st);
        if (e != cudaSuccess) return fail("K11 inheritance", e);
    }
    e = launch_tree_node(h->dev, d_nodes, n, depth, d_status, d_point, d_iters, inherit ? 1 : 0, h->sm_count, st);
    if (e != cudaSuccess) return fail("K11 tree node LP", e);
    return 0;
}

int ppgpu_tree_children(ppgpu_tree* h, const uint64_t* d_nodes, const uint8_t* d_status, int64_t n, int32_t depth,
                        int64_t* d_idx, uint64_t* d_children, int64_t* d_parent_of, int64_t* h_count, void* d_ws,
                        size_t ws_bytes, ppgpu_stream stream) {
    if (!h || !h_count) return fail_msg("null argument");
    *h_count = 0;
    if (n < 0) return fail_msg("negative size");
    if (depth < 0 || depth >= h->host.nb) return fail_msg("children need a depth in [0, nb)");
    if (n == 0) return 0;
    if (!d_nodes || !d_status || !d_idx || !d_children || !d_parent_of || !d_ws) return fail_msg("null argument");
    if (ws_bytes < select_workspace_bytes(n)) return fail_msg("workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaSetDevice(h->device);
    if (e != cudaSuccess) return fail("cudaSetDevice", e);
    long long* d_count = (long long*)d_ws + (select_workspace_bytes(n) / sizeof(long long) - 1);
    e = select_indices(d_status, n, 0xff, PPG_TREE_FEASIBLE, (long long*)d_idx, d_count, d_ws, ws_bytes - sizeof(long long), st);
    if (e != cudaSuccess) return fail("K11 select", e);
    e = launch_tree_children(d_nodes, (const long long*)d_idx, d_count, n, depth, d_children, (long long*)d_parent_of, st);
    if (e != cudaSuccess) return fail("K11 children", e);
    long long cnt = 0;
    e = cudaMemcpyAsync(&cnt, d_count, sizeof(long long), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return fail("K11 children count", e);
    *h_count = cnt;
    return 0;
}

int ppgpu_measure_fp64_peak(int32_t iters, double* h_tflops, ppgpu_stream stream) {
    if (!h_tflops) return fail_msg("null argument");
    cudaError_t e = measure_fp64_peak(iters, h_tflops, (cudaStream_t)stream);
    if (e != cudaSuccess) return fail("fp64 peak", e);
    return 0;
}

}  // extern "C"
