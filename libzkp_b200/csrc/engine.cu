// engine.cu — host side of the engine and the C ABI of include/lzkp_b200.h.
//
// One process drives one GPU (torchrun launches one rank per device); the proving key,
// its fixed-base window tables, the R1CS matrices and the NTT tables stay resident in
// HBM from lzkp_pk_load / lzkp_circuit_load until lzkp_pk_free (the reference keeps the
// same objects in process-wide OnceLocks, src/backend/snark.rs:295-339).
#include <cuda_runtime.h>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

#include "common.h"
#include "host_util.h"
#include "kernels_prove.cuh"
#include "tables.h"
#include "large.h"
#include "setup.h"
#include "verify.h"

using namespace lzkp;
using namespace lzkp::eng;

// ------------------------------------------------------------------------ plumbing
static thread_local std::string g_err;
static std::mutex g_mu;
static int g_device = -1;                       // primary device (devices[0] of lzkp_init)
static std::vector<int> g_devices;               // every device lzkp_init named: a proving key is replicated on each
static thread_local int t_device = -1;           // DeviceScope: the replica device this worker thread is bound to
static uint64_t g_mimc_uploaded = 0;             // bit d: c_mimc has been uploaded to device d (constants are per device)
static std::atomic<int> g_profile{0};

namespace lzkp {
namespace eng {
std::atomic<uint64_t> g_launches{0};
int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}
int DBuf::alloc(size_t n) {
    release();
    if (n == 0) n = 16;
    cudaError_t e = cudaMalloc(&p, n);
    if (e != cudaSuccess) {
        p = nullptr;
        cudaGetLastError();
        return fail(LZKP_E_NOMEM, "cudaMalloc(" + std::to_string(n) + "): " + cudaGetErrorString(e));
    }
    bytes = n;
    return LZKP_OK;
}
void DBuf::release() {
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
}
int ensure_device() {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_device < 0) {
        int n = 0;
        cudaError_t e = cudaGetDeviceCount(&n);
        if (e != cudaSuccess || n == 0) {
            cudaGetLastError();
            return fail(LZKP_E_NO_DEVICE, "no CUDA device: this engine has no CPU fallback");
        }
        int dev = 0;
        if (const char *lr = getenv("LOCAL_RANK")) dev = atoi(lr) % n;
        g_device = dev;
    }
    const int dev = t_device >= 0 ? t_device : g_device;
    CUDA_TRY(cudaSetDevice(dev));
    if (!(g_mimc_uploaded >> (dev & 63) & 1)) {
        std::vector<Fr> c(110);
        for (uint32_t i = 0; i < 110; i++) c[i] = host::mimc_constant(i);
        CUDA_TRY(cudaMemcpyToSymbol(c_mimc, c.data(), sizeof(Fr) * 110));
        g_mimc_uploaded |= 1ull << (dev & 63);
    }
    return LZKP_OK;
}
int current_device() { return t_device >= 0 ? t_device : g_device; }
DeviceScope::DeviceScope(int dev) : prev(t_device) {
    t_device = dev;
    cudaSetDevice(dev);
}
DeviceScope::~DeviceScope() {
    t_device = prev;
    const int back = prev >= 0 ? prev : g_device;
    if (back >= 0) cudaSetDevice(back);
}
}  // namespace eng
}  // namespace lzkp


// ------------------------------------------------------------------------ pk object
struct MsmPlan {                 // one curve
    DBuf table;                  // Affine<F>[rows * W * N]
    DBuf unit_dig, unit_tbl;     // uint32[n_units]
    DBuf items[4];               // uint2[n_items[v]] for the four granularities
    DBuf msm_items[4];           // uint2[n_msm]: item range of each MSM
    uint32_t n_items[4] = {0, 0, 0, 0};
    uint32_t item_len[4] = {8, 32, 128, 512};   // units per item of each granularity
    uint32_t n_units = 0, n_rows = 0, n_msm = 0;
    std::vector<uint32_t> msm_unit_begin;   // host: first unit of each MSM (+ end)
    std::vector<uint2> msm_items_host[4];   // host copy of msm_items per granularity
};

// Host memory the device can DMA to without an intermediate copy (results of a chunk land here asynchronously).
struct HBuf {
    void *p = nullptr;
    size_t bytes = 0;
    int ensure(size_t n) {
        if (n <= bytes) return LZKP_OK;
        if (p) cudaFreeHost(p);
        p = nullptr;
        bytes = 0;
        cudaError_t err = cudaMallocHost(&p, n);
        if (err != cudaSuccess) { p = nullptr; cudaGetLastError(); return fail(LZKP_E_NOMEM, "cudaMallocHost failed"); }
        bytes = n;
        return LZKP_OK;
    }
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
    ~HBuf() { if (p) cudaFreeHost(p); }
};
// Per-chunk device workspace.  A proving key owns two, so that two chunks of a batch are in flight on two
// streams: the latency-bound stages of one chunk (witness generation, witness map, recoding, assembly)
// run under the MSM kernels of the other.
struct Workspace {
    uint32_t chunk = 0;            // proofs the buffers are sized for
    DBuf z, abc, tmp, h, dig, r, s, rs, part1, part2, res1, res2, proofs, status, a, b, commit, sets, setlen, env, envlen;
    HBuf h_proofs, h_status, h_commit, h_env, h_envlen;
    // Last use of these buffers, on whatever stream it was enqueued (the *_device entry points run on the caller's
    // stream and return before the work has finished).  Every user waits on it before touching the workspace and
    // re-records it when its own work is enqueued: ws_acquire / ws_release.  pk->mu only orders the ENQUEUES.
    cudaEvent_t last_use = nullptr;
    ~Workspace() { if (last_use) cudaEventDestroy(last_use); }
};
static int ws_acquire(Workspace &ws, cudaStream_t st) { return event_acquire(ws.last_use, st); }
static int ws_release(Workspace &ws, cudaStream_t st) { return event_release(ws.last_use, st); }

// pk->stream is a BLOCKING stream on purpose: setup-time uploads use synchronous cudaMemcpy from pageable
// memory, whose DMA tail is only ordered against the legacy default stream and streams that synchronise
// with it; a non-blocking stream could run the first kernel before the bytes have landed.
struct lzkp_pk {
    std::mutex mu;
    int device = 0;                          // the device every buffer below lives on
    std::vector<lzkp_pk *> replicas;         // the same key on the other devices of lzkp_init's list (owned)
    uint32_t n_vars = 0, n_inst = 0, n_wit = 0, n = 0, log_n = 0, m = 0;
    bool has_circuit = false;
    int kind = -1;
    uint32_t kind_param = 0;
    int c = 16;
    uint32_t W = 16, N = 32768;
    uint64_t table_bytes = 0;
    uint32_t max_chunk = 8192;
    uint32_t n_dig_rows = 0, nz = 0;
    MsmPlan g1, g2;
    // Latency form for small calls (P <= latency_limit()): s*A and r*B1 of the assembly become two more fixed-base table
    // MSMs over the a / b1 rows with the scalars s*z_i / r*z_i (digit rows row_sz / row_rz), so the proof's tail is
    // a handful of additions and three inversions instead of two 254-bit variable-base scalar multiplications.
    MsmPlan g1_lat;                 // six MSMs: a, b1, l, h, s*A, r*B1 (shares g1.table)
    uint32_t row_sz = 0, row_rz = 0;
    bool has_lat = false;
    ProofConsts consts;
    // circuit
    DBuf csr_rowptr[3], csr_col[3], csr_val[3];
    CsrDev csr[3];
    DBuf tw_fwd, tw_inv, coset_br, uncoset_br;
    NttTables ntt;
    Workspace ws[2];
    // large mode (domain above 2^12): Pippenger MSMs over resident window-shifted bases, tiled NTTs
    bool large = false;
    bool tiled_wm = false;     // witness map on the tiled multi-pass NTT (domain above 2^12)
    MsmBases *L_a = nullptr, *L_b1 = nullptr, *L_b2 = nullptr, *L_l = nullptr, *L_h = nullptr;
    DBuf L_sa, L_sb, L_sl, L_sb1;
    // the five MSMs of one large proof run on side streams (each MsmBases has its own workspace), so the
    // latency-bound tail of one (bucket reduction, a few CTAs) runs under the accumulation of another
    cudaStream_t L_st[3] = {nullptr, nullptr, nullptr}, L_st_scale = nullptr;
    cudaEvent_t L_ev_in = nullptr, L_ev_done[3] = {nullptr, nullptr, nullptr}, L_ev_a = nullptr, L_ev_scale = nullptr;
    // single-proof sharding across GPUs (SURVEY.md §8e): this rank's point range [lo, lo + cnt) of each query,
    // in the order a, b1, l, h, b2 (extras +-delta included); unsharded = the full ranges
    uint32_t shard_index = 0, shard_count = 1, map_ranks = 1;
    bool L_scaled = false;            // this proof's k_scale_a share is pending in res1[4]
    uint32_t L_lo[5] = {0, 0, 0, 0, 0}, L_cnt[5] = {0, 0, 0, 0, 0};
    cudaStream_t stream = nullptr, stream2 = nullptr;      // chunk i of a batch runs on streams[i & 1]
    cudaEvent_t ev_fork = nullptr, ev_join[2] = {nullptr, nullptr};
    cudaStream_t chunk_stream(int i) const { return (i & 1) ? stream2 : stream; }
    // optional per-region CUDA-event timing (lzkp_profile_*): pairs recorded on the launching stream
    struct Mark { int region; cudaEvent_t a, b; };
    std::vector<Mark> marks;
    double prof_ms[LZKP_PROFILE_REGIONS] = {0};
    uint64_t prof_count[LZKP_PROFILE_REGIONS] = {0};
    ~lzkp_pk() {
        // (the caller has bound the thread to `device`: lzkp_pk_free / the replica loop below wrap the whole delete)
        for (lzkp_pk *r : replicas) { DeviceScope ds(r->device); delete r; }
        for (auto &m : marks) { cudaEventDestroy(m.a); cudaEventDestroy(m.b); }
        for (MsmBases *b : {L_a, L_b1, L_b2, L_l, L_h}) if (b) msm_bases_free(b);
        for (auto s_ : L_st) if (s_) cudaStreamDestroy(s_);
        if (L_ev_in) cudaEventDestroy(L_ev_in);
        if (L_ev_a) cudaEventDestroy(L_ev_a);
        if (L_ev_scale) cudaEventDestroy(L_ev_scale);
        if (L_st_scale) cudaStreamDestroy(L_st_scale);
        for (auto ev : L_ev_done) if (ev) cudaEventDestroy(ev);
        if (ev_fork) cudaEventDestroy(ev_fork);
        for (auto ev : ev_join) if (ev) cudaEventDestroy(ev);
        if (stream2) cudaStreamDestroy(stream2);
        if (stream) cudaStreamDestroy(stream);
    }
};

// ------------------------------------------------------------------------ lookup plans
struct BaseRef { uint32_t dig_row, tbl_row; };
static int finish_plan(MsmPlan &pl, const std::vector<std::vector<BaseRef>> &msms, uint32_t W) {
    std::vector<uint32_t> ud, ut;
    pl.msm_unit_begin.clear();
    for (auto &ms : msms) {
        pl.msm_unit_begin.push_back((uint32_t)ud.size());
        for (auto &b : ms)
            for (uint32_t w = 0; w < W; w++) {
                ud.push_back(b.dig_row * W + w);
                ut.push_back(b.tbl_row * W + w);
            }
    }
    pl.msm_unit_begin.push_back((uint32_t)ud.size());
    pl.n_units = (uint32_t)ud.size();
    pl.n_msm = (uint32_t)msms.size();
    TRY(upload(pl.unit_dig, ud));
    TRY(upload(pl.unit_tbl, ut));
    for (int v = 0; v < 4; v++) {
        std::vector<uint2> items, mi;
        for (uint32_t q = 0; q < pl.n_msm; q++) {
            uint32_t first = (uint32_t)items.size();
            for (uint32_t u = pl.msm_unit_begin[q]; u < pl.msm_unit_begin[q + 1]; u += pl.item_len[v])
                items.push_back(make_uint2(u, std::min(u + pl.item_len[v], pl.msm_unit_begin[q + 1])));
            mi.push_back(make_uint2(first, (uint32_t)items.size()));
        }
        pl.n_items[v] = (uint32_t)items.size();
        pl.msm_items_host[v] = mi;
        TRY(upload(pl.items[v], items));
        TRY(upload(pl.msm_items[v], mi));
    }
    return LZKP_OK;
}

// Units per item of the large-batch G1 grid (granularity 2: dim3(P / 128, items) of 128-thread CTAs of nearly equal
// length).  Such a grid runs in whole waves of the resident CTAs, so a last wave that is barely filled costs as much
// as a full one: the length is the one in [96, 192] with the least (waves rounded up) x (units per item), summed over
// batches of 1024 to 8192 proofs.  (The equality key at c = 17 with 128-unit items: 5312 CTAs = 8.97 waves of 592;
// after the shared A/B1 terms 4928 = 8.32 waves, still paying for 9; at 133 units 4736 = 8.00 waves.)
static uint32_t fit_item_len(const std::vector<std::vector<BaseRef>> &msms, uint32_t W, uint32_t resident) {
    uint32_t best = 128;
    uint64_t best_cost = UINT64_MAX;
    for (uint32_t len = 96; len <= 192; len++) {
        uint64_t items = 0, cost = 0;
        for (auto &ms : msms) items += ((uint64_t)ms.size() * W + len - 1) / len;
        for (uint64_t gx : {8u, 16u, 32u, 64u}) cost += (gx * items + resident - 1) / resident * len * (64 / gx);
        if (cost < best_cost) { best_cost = cost; best = len; }
    }
    return best;
}

// Signed c-bit windows of an Fr scalar by the offset trick (dev_util.cuh recode_offset): s + K must stay below
// 2^(c*W) with K = sum_w 2^(c*w + c-1) < 2^(c*W - 1) * (1 + 2^(1-c)).  BN254's r is 0.756 * 2^254, so c * W >= 255
// is enough: W = ceil(255 / c) (15 windows at c = 17, 16 at c = 16, 17 at c = 15).
static inline uint32_t window_count(int c) { return (uint32_t)((255 + c - 1) / c); }

// ------------------------------------------------------------------------ pk load
namespace {
struct Reader {
    const uint8_t *p, *end;
    bool take(size_t n, const uint8_t **out) {
        if ((size_t)(end - p) < n) return false;
        *out = p;
        p += n;
        return true;
    }
    bool g1(host::G1Canon &o) { const uint8_t *b; return take(64, &b) && host::read_g1(b, o); }
    bool g2(host::G2Canon &o) { const uint8_t *b; return take(128, &b) && host::read_g2(b, o); }
    bool vec_g1(std::vector<host::G1Canon> &v) {
        const uint8_t *b;
        if (!take(8, &b)) return false;
        uint64_t len;
        memcpy(&len, b, 8);
        if (len > (uint64_t)(end - p) / 64) return false;
        v.resize(len);
        for (auto &x : v) if (!g1(x)) return false;
        return true;
    }
    bool vec_g2(std::vector<host::G2Canon> &v) {
        const uint8_t *b;
        if (!take(8, &b)) return false;
        uint64_t len;
        memcpy(&len, b, 8);
        if (len > (uint64_t)(end - p) / 128) return false;
        v.resize(len);
        for (auto &x : v) if (!g2(x)) return false;
        return true;
    }
};
host::G1Canon neg_canon(const host::G1Canon &p) {
    host::G1Canon r = p;
    if (!host::is_inf(p)) {
        Fq m = Fq::modulus();
        sub8(r.y.l, m.l, p.y.l);
    }
    return r;
}
}  // namespace

static int pk_load_impl(const uint8_t *bytes, size_t len, int validate, const lzkp_pk_options *opt, lzkp_pk *pk) {
    static_assert(sizeof(host::G1Canon) == sizeof(G1Affine) && sizeof(host::G2Canon) == sizeof(G2Affine), "layout");
    Reader rd{bytes, bytes + len};
    host::G1Canon alpha_g1, beta_g1, delta_g1;
    host::G2Canon beta_g2, gamma_g2, delta_g2;
    std::vector<host::G1Canon> gamma_abc, a_q, b1_q, h_q, l_q;
    std::vector<host::G2Canon> b2_q;
    bool ok = rd.g1(alpha_g1) && rd.g2(beta_g2) && rd.g2(gamma_g2) && rd.g2(delta_g2) && rd.vec_g1(gamma_abc) &&
              rd.g1(beta_g1) && rd.g1(delta_g1) && rd.vec_g1(a_q) && rd.vec_g1(b1_q) && rd.vec_g2(b2_q) &&
              rd.vec_g1(h_q) && rd.vec_g1(l_q);
    if (!ok || rd.p != rd.end) return fail(LZKP_E_INVALID, "proving key: malformed ark-serialize bytes");
    const uint32_t nv = (uint32_t)a_q.size();
    if (nv < 2 || b1_q.size() != nv || b2_q.size() != nv || l_q.size() >= nv || gamma_abc.size() + l_q.size() != nv)
        return fail(LZKP_E_INVALID, "proving key: inconsistent query lengths");
    const uint32_t n = (uint32_t)h_q.size() + 1;
    if (n < 2 || (n & (n - 1))) return fail(LZKP_E_INVALID, "proving key: h_query length + 1 is not a power of two");
    pk->n_vars = nv;
    pk->n_wit = (uint32_t)l_q.size();
    pk->n_inst = nv - pk->n_wit;
    pk->n = n;
    pk->log_n = 0;
    while ((1u << pk->log_n) < n) pk->log_n++;
    pk->nz = nv - 1;
    pk->n_dig_rows = pk->nz + 3 + (n - 1);
    const uint32_t ROW_R = pk->nz, ROW_S = pk->nz + 1, ROW_RS = pk->nz + 2, ROW_H = pk->nz + 3;

    // Resident window tables (batched proving) while the domain is at most 2^16 and the tables fit the memory
    // budget at some c >= 8; beyond that, one proof per pass over Pippenger MSMs ("large" mode).
    {
        size_t free_b0 = 0, total_b0 = 0;
        CUDA_TRY(cudaMemGetInfo(&free_b0, &total_b0));
        const uint64_t budget0 = opt && opt->table_budget_bytes ? opt->table_budget_bytes : (uint64_t)(free_b0 * 0.6);
        const uint64_t rows1_max = 2ull * nv + pk->n_wit + n + 2, rows2_max = (uint64_t)nv + 1;
        const uint64_t min_table = (rows1_max * 64 + rows2_max * 128) * 32 * 128;      // c = 8: W = 32, N = 128
        pk->large = pk->log_n > 16 || min_table > budget0 || getenv("LZKP_FORCE_LARGE") != nullptr;
    }
    if (pk->large) {
        // A = alpha + a_q[0] + sum_{j>=1} z_j a_q[j] + r delta: delta rides along as one more base (scalar r / s / rs)
        CUDA_TRY(cudaStreamCreate(&pk->stream));
    CUDA_TRY(cudaStreamCreate(&pk->stream2));
    CUDA_TRY(cudaEventCreateWithFlags(&pk->ev_fork, cudaEventDisableTiming));
    for (auto &ev : pk->ev_join) CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        const int wb = opt && opt->window_bits ? opt->window_bits : 0;
        pk->shard_count = opt && opt->shard_count > 1 ? opt->shard_count : 1;
        pk->shard_index = pk->shard_count > 1 ? opt->shard_index : 0;
        if (pk->shard_index >= pk->shard_count) return fail(LZKP_E_INVALID, "shard_index >= shard_count");
        // Cost-weighted split (a G2 point costs ~3.2 G1 points in the sort-based MSM, fixed costs included; weights and
        // the map cost below were fitted with tools/shard_balance.py: slowest shard of 8 at 2^20 5.02 -> 4.5 ms).  The witness map is NOT distributed and h is NOT
        // broadcast: the first k ranks ("map ranks") each run the map themselves and share the H query between them;
        // the z-only queries a | b1 | l | b2 are cut over all ranks so that every rank ends up with the same load
        //   T = (W_z + W_h + k M) / G,     map rank: M + W_h / k + z-share,     other ranks: z-share = T
        // with M the cost of one witness map in MSM weight units (2.6 ms against 23.4 ms of MSMs at 2^20, less what
        // overlaps with the z-only MSMs on the side streams).
        // k is the smallest count whose spare capacity k (T - M) covers W_h (1 up to 4 GPUs, 3 at 8).
        // (every MSM call also carries ~0.55 ms (G1) / ~1 ms (G2) that does not scale with its range, so the best
        // weights drift with the shard count: fitted at 2, 4 and 8 shards)
        const uint32_t G_ = pk->shard_count;
        const uint64_t w_g2 = getenv("LZKP_SHARD_G2_WEIGHT") ? (uint64_t)atoi(getenv("LZKP_SHARD_G2_WEIGHT")) : (G_ > 2 ? 32 : 28);
        const uint64_t sizes[5] = {nv, nv, (uint64_t)pk->n_wit + 1, (uint64_t)n - 1, nv}, wts[5] = {10, 10, 10, 10, w_g2};
        const double Wh = (double)sizes[3] * wts[3];
        double Wz = 0;
        for (int q : {0, 1, 2, 4}) Wz += (double)sizes[q] * wts[q];
        const double map_frac = getenv("LZKP_SHARD_MAP_COST") ? atof(getenv("LZKP_SHARD_MAP_COST")) : (G_ > 4 ? 0.085 : 0.11);
        const double M = G_ > 1 ? map_frac * (Wz + Wh) : 0.0;
        uint32_t k = 1;
        while (k < G_ && k * ((Wz + Wh + k * M) / G_ - M) < Wh) k++;
        const double T = (Wz + Wh + k * M) / G_;
        std::vector<double> cutz(G_ + 1, 0.0), share(G_, 0.0);
        for (uint32_t i = 0; i < G_; i++) share[i] = i < k ? std::max(0.0, T - M - Wh / k) : T;
        // A rank whose share straddles a query boundary runs one MSM call more than its neighbours, and a call carries
        // ~0.25 ms that does not depend on its range (sort floor, segment and bucket reductions; tools/shard_balance.py:
        // the rank holding the end of l and the start of b2 was the slowest of 8 at every weight).  Shares of such ranks
        // shrink by that much per extra piece, the others absorb it; three rounds settle the cuts.  Slowest shard 4.64 -> 4.42 ms
        // at 8 shards, 7.37 -> 7.14 ms at 4 (with the G2 weight of 8 shards); two shards keep the plain split (the adjustment
        // only moved a sliver across and made it worse).
        const double piece_cost = G_ > 2 ? (getenv("LZKP_SHARD_PIECE_COST") ? atof(getenv("LZKP_SHARD_PIECE_COST")) : (G_ > 4 ? 0.25 : 0.45)) * 2.76e6 : 0.0;
        std::vector<double> adj(share);
        for (int round = 0; round < 4; round++) {
            double tot = 0;
            for (uint32_t i = 0; i < G_; i++) tot += adj[i];
            for (uint32_t i = 0; i < G_; i++) cutz[i + 1] = cutz[i] + adj[i] * Wz / tot;   // (clamping may leave a remainder)
            double bounds[5] = {0, 0, 0, 0, 0};                                             // weighted ends of a | b1 | l | b2
            { int j = 0; for (int q : {0, 1, 2, 4}) { bounds[j + 1] = bounds[j] + (double)sizes[q] * wts[q]; j++; } }
            if (piece_cost != 0.0)                      // a sliver of a query next to a boundary is not worth an MSM call: snap
                for (uint32_t i = 1; i < G_; i++)
                    for (int j = 1; j < 4; j++)
                        if (std::fabs(cutz[i] - bounds[j]) < 1.0e5) cutz[i] = bounds[j];        // < 10 k G1 points
            if (round == 3 || piece_cost == 0.0) break;
            double extra_total = 0;
            std::vector<double> extra(G_, 0.0);
            for (uint32_t i = 0; i < G_; i++) {
                int pieces = 0;
                for (int j = 0; j < 4; j++)
                    if (std::min(cutz[i + 1], bounds[j + 1]) - std::max(cutz[i], bounds[j]) > 1e-6 * Wz) pieces++;
                extra[i] = piece_cost * std::max(0, pieces - 1);
                extra_total += extra[i];
            }
            for (uint32_t i = 0; i < G_; i++) adj[i] = std::max(0.0, share[i] - extra[i] + extra_total / G_);
        }
        pk->map_ranks = k;
        const uint32_t me = pk->shard_index;
        if (me < k) {
            pk->L_lo[3] = (uint32_t)(sizes[3] * me / k);
            pk->L_cnt[3] = (uint32_t)(sizes[3] * (me + 1) / k) - pk->L_lo[3];
        } else {
            pk->L_lo[3] = 0;
            pk->L_cnt[3] = 0;
        }
        double acc_w = 0;
        for (int q : {0, 1, 2, 4}) {
            auto first_at = [&](double w) -> uint64_t {          // first point of query q at or after weighted position w
                if (w <= acc_w) return 0;
                return std::min<uint64_t>((uint64_t)std::ceil((w - acc_w) / wts[q]), sizes[q]);
            };
            uint64_t lo = first_at(cutz[me]), hi = me + 1 == G_ ? sizes[q] : first_at(cutz[me + 1]);
            pk->L_lo[q] = (uint32_t)lo;
            pk->L_cnt[q] = (uint32_t)(hi - lo);
            acc_w += (double)sizes[q] * wts[q];
        }
        auto load1 = [&](std::vector<host::G1Canon> v, size_t skip, const host::G1Canon *extra, int q, MsmBases **out) {
            v.erase(v.begin(), v.begin() + skip);
            if (extra) v.push_back(*extra);
            return msm_bases_load(1, reinterpret_cast<const uint8_t *>(v.data() + pk->L_lo[q]), pk->L_cnt[q], wb, 1, validate, out, 1);
        };
        host::G1Canon nd1 = neg_canon(delta_g1);
        TRY(load1(a_q, 1, &delta_g1, 0, &pk->L_a));
        TRY(load1(b1_q, 1, &delta_g1, 1, &pk->L_b1));
        TRY(load1(l_q, 0, &nd1, 2, &pk->L_l));
        TRY(load1(h_q, 0, nullptr, 3, &pk->L_h));
        {
            std::vector<host::G2Canon> v(b2_q.begin() + 1, b2_q.end());
            v.push_back(delta_g2);
            TRY(msm_bases_load(2, reinterpret_cast<const uint8_t *>(v.data() + pk->L_lo[4]), pk->L_cnt[4], wb, 1, validate, &pk->L_b2, 1));
        }
        {   // the A-sum feeds the one serial chain left (k_scale_a, 0.8 ms): their stream goes first
            int prio_lo = 0, prio_hi = 0;
            CUDA_TRY(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
            const bool prio = !(getenv("LZKP_NO_STREAM_PRIORITY") && atoi(getenv("LZKP_NO_STREAM_PRIORITY")));
            for (int i = 0; i < 3; i++)
                CUDA_TRY(cudaStreamCreateWithPriority(&pk->L_st[i], cudaStreamNonBlocking, prio_lo));
            CUDA_TRY(cudaStreamCreateWithPriority(&pk->L_st_scale, cudaStreamNonBlocking, prio ? prio_hi : prio_lo));
        }
        CUDA_TRY(cudaEventCreateWithFlags(&pk->L_ev_in, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&pk->L_ev_a, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&pk->L_ev_scale, cudaEventDisableTiming));
        for (auto &ev : pk->L_ev_done) CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        pk->c = wb ? wb : 16;
        pk->W = (255 + pk->c - 1) / pk->c;
        pk->max_chunk = 1;
        pk->table_bytes = ((uint64_t)(a_q.size() + b1_q.size() + l_q.size() + 1 + h_q.size()) * 64 + (uint64_t)b2_q.size() * 128) * pk->W;
        // constant terms alpha + a_q[0], beta + b_q[0] (G1 and G2)
        std::vector<host::G1Canon> misc1 = {alpha_g1, beta_g1, a_q[0], b1_q[0]};
        std::vector<host::G2Canon> misc2 = {beta_g2, b2_q[0]};
        DBuf d_misc1, d_misc2, d_out1, d_out2;
        cudaStream_t st = pk->stream;
        TRY(upload(d_misc1, misc1)); TRY(upload(d_misc2, misc2));
        LAUNCH(k_fq_to_mont, 1, 128, 0, st, d_misc1.as<Fq>(), misc1.size() * 2);
        LAUNCH(k_fq_to_mont, 1, 128, 0, st, d_misc2.as<Fq>(), misc2.size() * 4);
        if (validate) {
            // the queries were checked by msm_bases_load; here the remaining points deserialize_uncompressed validates
            std::vector<host::G1Canon> v1 = gamma_abc;
            v1.push_back(alpha_g1); v1.push_back(beta_g1); v1.push_back(delta_g1); v1.push_back(a_q[0]); v1.push_back(b1_q[0]);
            std::vector<host::G2Canon> v2 = {beta_g2, gamma_g2, delta_g2, b2_q[0]};
            DBuf d_v1, d_v2, d_bad;
            TRY(upload(d_v1, v1)); TRY(upload(d_v2, v2)); TRY(d_bad.alloc(sizeof(int)));
            CUDA_TRY(cudaMemsetAsync(d_bad.p, 0, sizeof(int), st));
            LAUNCH(k_fq_to_mont, (unsigned)((v1.size() * 2 + 127) / 128), 128, 0, st, d_v1.as<Fq>(), v1.size() * 2);
            LAUNCH(k_fq_to_mont, 1, 128, 0, st, d_v2.as<Fq>(), v2.size() * 4);
            LAUNCH(k_check_g1, (unsigned)((v1.size() + 63) / 64), 64, 0, st, d_v1.as<G1Affine>(), (uint32_t)v1.size(), d_bad.as<int>());
            LAUNCH(k_check_g2, 1, 64, 0, st, d_v2.as<G2Affine>(), (uint32_t)v2.size(), d_bad.as<int>());
            int bad = 0;
            CUDA_TRY(cudaMemcpyAsync(&bad, d_bad.p, sizeof(int), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            if (bad) return fail(LZKP_E_INVALID, "proving key: " + std::to_string(bad) + " point(s) off-curve or outside the subgroup");
        }
        TRY(d_out1.alloc(2 * sizeof(G1Affine))); TRY(d_out2.alloc(sizeof(G2Affine)));
        LAUNCH((k_affine_add<Fq>), 1, 1, 0, st, d_misc1.as<G1Affine>() + 0, d_misc1.as<G1Affine>() + 2, d_out1.as<G1Affine>() + 0, 0);
        LAUNCH((k_affine_add<Fq>), 1, 1, 0, st, d_misc1.as<G1Affine>() + 1, d_misc1.as<G1Affine>() + 3, d_out1.as<G1Affine>() + 1, 0);
        LAUNCH((k_affine_add<Fq2>), 1, 1, 0, st, d_misc2.as<G2Affine>() + 0, d_misc2.as<G2Affine>() + 1, d_out2.as<G2Affine>(), 0);
        G1Affine c1[2];
        G2Affine c2;
        CUDA_TRY(cudaMemcpyAsync(c1, d_out1.p, sizeof(c1), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaMemcpyAsync(&c2, d_out2.p, sizeof(c2), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        pk->consts.a0 = c1[0]; pk->consts.b0 = c1[1]; pk->consts.b2 = c2;
        CUDA_TRY(cudaGetLastError());
        return LZKP_OK;
    }

    // --- base lists (identity points are dropped: they contribute nothing to any MSM) ---
    // A variable whose A and B1 query points are the same point adds the same term z_j a_j to the A sum and to the
    // B1 sum (every MiMC-5 round of libzkp's circuits: A column = B column for t2 = t*t): the batch form computes it
    // once, in MSM 4 ("shared", one table row), and k_assemble adds that sum to both.
    std::vector<host::G1Canon> rows1;
    std::vector<host::G2Canon> rows2;
    std::vector<std::vector<BaseRef>> msm1(5), msm2(1);
    std::vector<BaseRef> a_all, b1_all;              // every a / b1 term, shared ones included (latency form)
    auto add1 = [&](const host::G1Canon &p) { rows1.push_back(p); return (uint32_t)rows1.size() - 1; };
    auto same_point = [](const host::G1Canon &u, const host::G1Canon &v) {
        return memcmp(&u.x, &v.x, sizeof(Fq)) == 0 && memcmp(&u.y, &v.y, sizeof(Fq)) == 0;
    };
    for (uint32_t j = 1; j < nv; j++) {
        const bool has_a = !host::is_inf(a_q[j]), has_b = !host::is_inf(b1_q[j]);
        if (has_a && has_b && same_point(a_q[j], b1_q[j])) {
            const BaseRef ref{j - 1, add1(a_q[j])};
            msm1[4].push_back(ref); a_all.push_back(ref); b1_all.push_back(ref);
            continue;
        }
        if (has_a) { msm1[0].push_back({j - 1, add1(a_q[j])}); a_all.push_back(msm1[0].back()); }
        if (has_b) { msm1[1].push_back({j - 1, add1(b1_q[j])}); b1_all.push_back(msm1[1].back()); }
    }
    for (uint32_t j = 0; j < pk->n_wit; j++) if (!host::is_inf(l_q[j])) msm1[2].push_back({pk->n_inst + j - 1, add1(l_q[j])});
    for (uint32_t i = 0; i + 1 < n; i++) if (!host::is_inf(h_q[i])) msm1[3].push_back({ROW_H + i, add1(h_q[i])});
    if (!host::is_inf(delta_g1)) {
        uint32_t rd1 = add1(delta_g1), rnd1 = add1(neg_canon(delta_g1));
        msm1[0].push_back({ROW_R, rd1});      // A  += r * delta_g1
        msm1[1].push_back({ROW_S, rd1});      // B1 += s * delta_g1
        msm1[2].push_back({ROW_RS, rnd1});    // C  -= rs * delta_g1 (folded into the L sum)
        a_all.push_back({ROW_R, rd1});
    }
    // latency form: C = s*(alpha + a0) + r*(beta + b0) + sum (s z_i) a_i + sum (r z_i) b_i + 2 rs delta + [L - rs delta] + H.
    // The proof needs the A sum itself (slot 0, whole: no shared MSM) but B1 only as r*B1 (slot 5), so slot 1 stays empty.
    std::vector<std::vector<BaseRef>> msm1_lat(6);
    {
        pk->row_sz = pk->n_dig_rows;
        pk->row_rz = pk->n_dig_rows + pk->nz;
        msm1_lat[0] = a_all;
        msm1_lat[2] = msm1[2];
        msm1_lat[3] = msm1[3];
        for (auto &b : a_all) if (b.dig_row < pk->nz) msm1_lat[4].push_back({pk->row_sz + b.dig_row, b.tbl_row});
        for (auto &b : b1_all) msm1_lat[5].push_back({pk->row_rz + b.dig_row, b.tbl_row});
        // the three constant points, computed with the host build of the same field / curve code
        auto mont = [](const host::G1Canon &c) { return G1Affine{Fq::from_canonical(c.x), Fq::from_canonical(c.y)}; };
        auto canon = [](const G1Affine &m) { host::G1Canon c; c.x = m.x.to_canonical(); c.y = m.y.to_canonical(); return c; };
        auto sum2 = [&](const host::G1Canon &u, const host::G1Canon &v) {
            G1XYZZ t = host::is_inf(u) ? G1XYZZ::inf() : G1XYZZ::from_affine(mont(u));
            if (!host::is_inf(v)) t.madd(mont(v));
            return t.is_inf() ? host::G1Canon{Fq::zero(), Fq::zero()} : canon(t.to_affine());
        };
        const host::G1Canon a0c = sum2(alpha_g1, a_q[0]), b0c = sum2(beta_g1, b1_q[0]), d2c = sum2(delta_g1, delta_g1);
        if (!host::is_inf(a0c)) msm1_lat[4].push_back({ROW_S, add1(a0c)});
        if (!host::is_inf(b0c)) msm1_lat[5].push_back({ROW_R, add1(b0c)});
        if (!host::is_inf(d2c)) msm1_lat[5].push_back({ROW_RS, add1(d2c)});
        pk->n_dig_rows += 2 * pk->nz;
        pk->has_lat = true;
    }
    for (uint32_t j = 1; j < nv; j++)
        if (!host::is_inf(b2_q[j])) { rows2.push_back(b2_q[j]); msm2[0].push_back({j - 1, (uint32_t)rows2.size() - 1}); }
    if (!host::is_inf(delta_g2)) { rows2.push_back(delta_g2); msm2[0].push_back({ROW_S, (uint32_t)rows2.size() - 1}); }
    pk->g1.n_rows = (uint32_t)rows1.size();
    pk->g2.n_rows = (uint32_t)rows2.size();

    // --- window size from the memory budget ---
    size_t free_b = 0, total_b = 0;
    CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
    uint64_t budget = opt && opt->table_budget_bytes ? opt->table_budget_bytes : (uint64_t)(free_b * 0.6);
    int c = opt && opt->window_bits ? opt->window_bits : 0;
    if (const char *e = getenv("LZKP_WINDOW_BITS")) if (!c) c = atoi(e);
    auto bytes_for = [&](int cc) {
        uint64_t W = window_count(cc), N = 1ull << (cc - 1);
        return (rows1.size() * 64ull + rows2.size() * 128ull) * W * N;
    };
    if (c == 0) {
        c = 16;
        while (c > 8 && bytes_for(c) > budget) c--;
    }
    if (c < 8 || c > 17) return fail(LZKP_E_INVALID, "window_bits must be in [8,17]");
    if (bytes_for(c) > free_b) return fail(LZKP_E_NOMEM, "window tables do not fit in device memory");
    pk->c = c;
    pk->W = window_count(c);
    pk->N = 1u << (c - 1);
    pk->table_bytes = bytes_for(c);
    pk->max_chunk = opt && opt->max_chunk ? opt->max_chunk : 8192;
    if (pk->max_chunk > 32768) pk->max_chunk = 32768;

    CUDA_TRY(cudaStreamCreate(&pk->stream));
    CUDA_TRY(cudaStreamCreate(&pk->stream2));
    CUDA_TRY(cudaEventCreateWithFlags(&pk->ev_fork, cudaEventDisableTiming));
    for (auto &ev : pk->ev_join) CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    // side stream of the latency form (small calls: the G2 MSM beside the witness map and the G1 MSMs)
    CUDA_TRY(cudaStreamCreateWithFlags(&pk->L_st[0], cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreateWithFlags(&pk->L_ev_in, cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&pk->L_ev_done[0], cudaEventDisableTiming));
    cudaStream_t st = pk->stream;

    // --- upload points, to Montgomery, optional validation ---
    std::vector<host::G1Canon> misc1 = {alpha_g1, beta_g1, delta_g1, a_q[0], b1_q[0]};
    std::vector<host::G2Canon> misc2 = {beta_g2, gamma_g2, delta_g2, b2_q[0]};
    DBuf d_rows1, d_rows2, d_misc1, d_misc2, d_out1, d_out2;
    TRY(upload(d_rows1, rows1)); TRY(upload(d_rows2, rows2)); TRY(upload(d_misc1, misc1)); TRY(upload(d_misc2, misc2));
    auto to_mont = [&](DBuf &b, size_t n_fq) {
        if (n_fq) LAUNCH(k_fq_to_mont, (unsigned)((n_fq + 127) / 128), 128, 0, st, b.as<Fq>(), n_fq);
    };
    to_mont(d_rows1, rows1.size() * 2); to_mont(d_rows2, rows2.size() * 4);
    to_mont(d_misc1, misc1.size() * 2); to_mont(d_misc2, misc2.size() * 4);
    if (validate) {
        // everything deserialize_uncompressed would check: all vk and query points
        std::vector<host::G1Canon> all1 = gamma_abc;
        std::vector<host::G2Canon> all2;
        DBuf d_all1, d_bad;
        TRY(upload(d_all1, all1));
        to_mont(d_all1, all1.size() * 2);
        TRY(d_bad.alloc(sizeof(int)));
        CUDA_TRY(cudaMemsetAsync(d_bad.p, 0, sizeof(int), st));
        auto chk1 = [&](DBuf &b, size_t cnt) {
            if (cnt) LAUNCH(k_check_g1, (unsigned)((cnt + 63) / 64), 64, 0, st, b.as<G1Affine>(), (uint32_t)cnt, d_bad.as<int>());
        };
        auto chk2 = [&](DBuf &b, size_t cnt) {
            if (cnt) LAUNCH(k_check_g2, (unsigned)((cnt + 63) / 64), 64, 0, st, b.as<G2Affine>(), (uint32_t)cnt, d_bad.as<int>());
        };
        chk1(d_rows1, rows1.size()); chk1(d_misc1, misc1.size()); chk1(d_all1, all1.size());
        chk2(d_rows2, rows2.size()); chk2(d_misc2, misc2.size());
        int bad = 0;
        CUDA_TRY(cudaMemcpyAsync(&bad, d_bad.p, sizeof(int), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        if (bad) return fail(LZKP_E_INVALID, "proving key: " + std::to_string(bad) + " point(s) off-curve or outside the subgroup");
    }
    // --- constant terms of calculate_coeff: vk_param + query[0] ---
    TRY(d_out1.alloc(2 * sizeof(G1Affine))); TRY(d_out2.alloc(sizeof(G2Affine)));
    LAUNCH((k_affine_add<Fq>), 1, 1, 0, st, d_misc1.as<G1Affine>() + 0, d_misc1.as<G1Affine>() + 3, d_out1.as<G1Affine>() + 0, 0);
    LAUNCH((k_affine_add<Fq>), 1, 1, 0, st, d_misc1.as<G1Affine>() + 1, d_misc1.as<G1Affine>() + 4, d_out1.as<G1Affine>() + 1, 0);
    LAUNCH((k_affine_add<Fq2>), 1, 1, 0, st, d_misc2.as<G2Affine>() + 0, d_misc2.as<G2Affine>() + 3, d_out2.as<G2Affine>(), 0);
    G1Affine c1[2];
    G2Affine c2;
    CUDA_TRY(cudaMemcpyAsync(c1, d_out1.p, sizeof(c1), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(&c2, d_out2.p, sizeof(c2), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    pk->consts.a0 = c1[0]; pk->consts.b0 = c1[1]; pk->consts.b2 = c2;

    // --- resident window tables + lookup plans ---
    TRY(pk->g1.table.alloc((size_t)rows1.size() * pk->W * pk->N * sizeof(G1Affine)));
    TRY(pk->g2.table.alloc((size_t)rows2.size() * pk->W * pk->N * sizeof(G2Affine)));
    if (!rows1.empty())
        TRY(build_table_g1(d_rows1.p, (uint32_t)rows1.size(), c, pk->W, pk->N, pk->g1.table.p, st));
    if (!rows2.empty())
        TRY(build_table_g2(d_rows2.p, (uint32_t)rows2.size(), c, pk->W, pk->N, pk->g2.table.p, st));
    {
        uint32_t resident = 0;
        TRY(batch_msm_g1_resident(c > 16 ? 4 : 2, &resident));
        pk->g1.item_len[2] = fit_item_len(msm1, pk->W, resident);
    }
    TRY(finish_plan(pk->g1, msm1, pk->W));
    TRY(finish_plan(pk->g1_lat, msm1_lat, pk->W));
    TRY(finish_plan(pk->g2, msm2, pk->W));
    // proofs per device pass: two workspaces must fit beside the tables
    {
        const uint64_t per_proof = (uint64_t)nv * 32 + 7ull * n * 32 + (uint64_t)pk->n_dig_rows * pk->W * (c > 16 ? 4 : 2) +
                                   (uint64_t)pk->g1.n_items[2] * sizeof(G1XYZZ) + (uint64_t)pk->g2.n_items[1] * sizeof(G2XYZZ) +
                                   4 * sizeof(G1XYZZ) + sizeof(G2XYZZ) + 1024;
        size_t free_now = 0, total_now = 0;
        CUDA_TRY(cudaMemGetInfo(&free_now, &total_now));
        uint64_t fit = (uint64_t)(free_now * 0.4) / (2 * per_proof);
        fit = std::max<uint64_t>(32, fit / 32 * 32);
        if (pk->max_chunk > fit) pk->max_chunk = (uint32_t)fit;
    }
    CUDA_TRY(cudaGetLastError());
    return LZKP_OK;
}

// ------------------------------------------------------------------------ circuit load
static int circuit_install(lzkp_pk *pk, uint32_t m, uint32_t n_inst, uint32_t n_wit, const uint32_t *const rowptr[3],
                           const uint32_t *const col[3], const uint8_t *const val[3]) {
    if (n_inst != pk->n_inst || n_wit != pk->n_wit) return fail(LZKP_E_INVALID, "circuit shape does not match the proving key");
    uint64_t need = (uint64_t)m + n_inst;
    uint32_t n = 1;
    while (n < need) n <<= 1;
    if (n != pk->n) return fail(LZKP_E_INVALID, "circuit domain size does not match the proving key's h_query");
    pk->tiled_wm = pk->large || pk->log_n > 12;      // above 2^12 a polynomial no longer fits one CTA's shared memory
    cudaStream_t st = pk->stream;
    for (int k = 0; k < 3; k++) {
        uint32_t nnz = rowptr[k][m];
        for (uint32_t i = 0; i < nnz; i++) if (col[k][i] >= pk->n_vars) return fail(LZKP_E_INVALID, "matrix column out of range");
        TRY(pk->csr_rowptr[k].alloc(sizeof(uint32_t) * (m + 1)));
        TRY(pk->csr_col[k].alloc(sizeof(uint32_t) * nnz));
        TRY(pk->csr_val[k].alloc(sizeof(Fr) * (size_t)nnz));
        CUDA_TRY(cudaMemcpy(pk->csr_rowptr[k].p, rowptr[k], sizeof(uint32_t) * (m + 1), cudaMemcpyHostToDevice));
        if (nnz) {
            CUDA_TRY(cudaMemcpy(pk->csr_col[k].p, col[k], sizeof(uint32_t) * nnz, cudaMemcpyHostToDevice));
            CUDA_TRY(cudaMemcpy(pk->csr_val[k].p, val[k], 32 * (size_t)nnz, cudaMemcpyHostToDevice));
            LAUNCH(k_to_r2_form, (nnz + 127) / 128, 128, 0, st, pk->csr_val[k].as<Fr>(), nnz);
        }
        pk->csr[k] = CsrDev{pk->csr_rowptr[k].as<uint32_t>(), pk->csr_col[k].as<uint32_t>(), pk->csr_val[k].as<Fr>()};
    }
    pk->m = m;
    // NTT tables: w = ROOT28^(2^(28-log n)); host arithmetic for the handful of scalars
    Fr w, wi, g, gi;
    for (int i = 0; i < 8; i++) { w.l[i] = FrParams::ROOT28(i); wi.l[i] = FrParams::ROOT28_INV(i); g.l[i] = FrParams::GEN(i); gi.l[i] = FrParams::GEN_INV(i); }
    for (uint32_t i = pk->log_n; i < 28; i++) { w = w.sqr(); wi = wi.sqr(); }
    Fr ninv = host::fr_from_u64(n).inverse();
    Fr gn = g;
    for (uint32_t i = 0; i < pk->log_n; i++) gn = gn.sqr();
    Fr zinv = (gn - Fr::one()).inverse();
    if (pk->tiled_wm) {       // transforms come from ntt_large.cu's cached plans; only Z(g)^-1 is needed here
        pk->ntt = NttTables{nullptr, nullptr, nullptr, nullptr, nullptr, ninv, zinv};
        CUDA_TRY(cudaStreamSynchronize(st));
        CUDA_TRY(cudaGetLastError());
        pk->has_circuit = true;
        return LZKP_OK;
    }
    TRY(pk->tw_fwd.alloc(sizeof(Fr) * (n / 2))); TRY(pk->tw_inv.alloc(sizeof(Fr) * (n / 2)));
    TRY(pk->coset_br.alloc(sizeof(Fr) * n)); TRY(pk->uncoset_br.alloc(sizeof(Fr) * n));
    LAUNCH(k_pow_table, (n / 2 + 127) / 128, 128, 0, st, pk->tw_fwd.as<Fr>(), w, Fr::one(), n / 2, 0u);
    LAUNCH(k_pow_table, (n / 2 + 127) / 128, 128, 0, st, pk->tw_inv.as<Fr>(), wi, Fr::one(), n / 2, 0u);
    LAUNCH(k_pow_table, (n + 127) / 128, 128, 0, st, pk->coset_br.as<Fr>(), g, ninv, n, pk->log_n);
    LAUNCH(k_pow_table, (n + 127) / 128, 128, 0, st, pk->uncoset_br.as<Fr>(), gi, ninv.to_canonical(), n, pk->log_n);
    pk->ntt = NttTables{pk->tw_fwd.as<Fr>(), pk->tw_inv.as<Fr>(), pk->coset_br.as<Fr>(), pk->uncoset_br.as<Fr>(), nullptr, ninv, zinv};
    size_t smem = (size_t)32 * n;
    if (smem > 48 * 1024) {
        CUDA_TRY(cudaFuncSetAttribute(k_ntt_icoset, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(cudaFuncSetAttribute(k_ntt_final, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    pk->has_circuit = true;
    return LZKP_OK;
}

// ------------------------------------------------------------------------ proving pipeline
// Item granularity: many more CTAs than the 148 x 3 resident ones, so the last wave of a launch is a small
// fraction of the kernel (measured: 512-unit items left the G1 kernel at 3.4 waves = 0.87 of peak).
// Calls of at most small_batch_limit() proofs are latency-bound: 8-unit items and a tree reduction keep the serial chain per thread
// short (msm_batch.cu kSmallBatch).
static inline int item_variant(uint32_t P) {
    return P > small_batch_limit() ? (P >= 256 ? 2 : 1) : 0;
}
// the item index is the grid's y dimension (<= 65535): very wide keys fall back to coarser items
static inline int fit_variant(const MsmPlan &pl, int v) {
    while (v < 3 && pl.n_items[v] > 65535u) v++;
    return v;
}
// Calls of at most this many proofs take the latency form (fixed-base s*A + r*B1, k_assemble_sums): +47 % G1 MSM work,
// which is free while the call is latency-bound (measured: 192 / 256 / 384 proofs 2.34 / 2.88 / 4.04 ms against 2.94 / 3.26 /
// 4.30 ms in the batch form; level at 512).  LZKP_LATENCY_BATCH overrides (0 disables).
static inline uint32_t latency_limit() {
    static const uint32_t v = getenv("LZKP_LATENCY_BATCH") ? (uint32_t)atoi(getenv("LZKP_LATENCY_BATCH")) : 384u;
    return v;
}
static inline bool use_lat(const lzkp_pk *pk, uint32_t P) { return pk->has_lat && P <= latency_limit() && P <= small_batch_limit(); }
static inline int item_variant_g2(uint32_t P) {
    // 32-unit items at every batch size: the G2 grid then is several waves of its 148 x 6 resident CTAs (with 128-unit
    // items a 4096-proof batch was 1.87 waves and paid for 2: measured 7.59 -> 7.06 ms; lengths 24..37 are within 2 %)
    return P > small_batch_limit() ? 1 : 0;
}
static int ensure_workspace(lzkp_pk *pk, Workspace &ws, uint32_t P) {
    if (P <= ws.chunk) return LZKP_OK;
    size_t part1 = 0, part2 = 0;       // worst case over the batch sizes <= P
    for (uint32_t pp : {std::min(P, small_batch_limit()), std::min(P, std::max(latency_limit(), 1u)), std::min(P, 255u), std::min(P, 2047u), P}) {
        part1 = std::max(part1, (size_t)pk->g1.n_items[fit_variant(pk->g1, item_variant(pp))] * pp);
        if (use_lat(pk, pp)) part1 = std::max(part1, (size_t)pk->g1_lat.n_items[fit_variant(pk->g1_lat, item_variant(pp))] * pp);
        part2 = std::max(part2, (size_t)pk->g2.n_items[fit_variant(pk->g2, item_variant_g2(pp))] * pp);
    }
    const size_t nv = pk->n_vars, n = pk->n;
    TRY(ws.z.ensure(P * nv * 32));
    TRY(ws.abc.ensure(3 * P * n * 32));
    TRY(ws.h.ensure(P * n * 32));
    if (pk->tiled_wm) TRY(ws.tmp.ensure(3 * P * n * 32));
    if (pk->large) {
        TRY(pk->L_sa.ensure(nv * 32)); TRY(pk->L_sb.ensure(nv * 32)); TRY(pk->L_sb1.ensure(nv * 32)); TRY(pk->L_sl.ensure(((size_t)pk->n_wit + 1) * 32));
    } else {
        TRY(ws.dig.ensure((size_t)pk->n_dig_rows * pk->W * P * (pk->c > 16 ? 4 : 2)));
    }
    TRY(ws.r.ensure(P * 32)); TRY(ws.s.ensure(P * 32)); TRY(ws.rs.ensure(P * 32));
    TRY(ws.part1.ensure(part1 * sizeof(G1XYZZ)));
    TRY(ws.part2.ensure(part2 * sizeof(G2XYZZ)));
    TRY(ws.res1.ensure((size_t)6 * P * sizeof(G1XYZZ)));
    TRY(ws.res2.ensure((size_t)P * sizeof(G2XYZZ)));
    TRY(ws.proofs.ensure((size_t)P * 256));
    TRY(ws.status.ensure((size_t)P * sizeof(int32_t)));
    TRY(ws.a.ensure(P * 8)); TRY(ws.b.ensure(P * 8)); TRY(ws.commit.ensure(P * 32));
    ws.chunk = P;
    return LZKP_OK;
}

static inline void wires_to_canonical(Fr *z, uint32_t P, uint32_t nv, uint32_t first, uint32_t count, cudaStream_t st) {
    const size_t total = (size_t)P * count;
    LAUNCH(k_wires_to_canonical, (unsigned)((total + 127) / 128), 128, 0, st, z, P, nv, first, count);
}

struct Region {           // RAII: brackets the kernels of one pipeline stage with two events when profiling is on
    lzkp_pk *pk;
    cudaStream_t st;
    cudaEvent_t b = nullptr;
    Region(lzkp_pk *pk_, int region, cudaStream_t st_) : pk(pk_), st(st_) {
        if (!g_profile.load(std::memory_order_relaxed) || pk->marks.size() > 65536) return;
        cudaEvent_t a;
        if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) { b = nullptr; return; }
        cudaEventRecord(a, st);
        pk->marks.push_back({region, a, b});
    }
    ~Region() { if (b) cudaEventRecord(b, st); }
};

// Witness map on P assignments already in ws_z (canonical): fills ws_h (canonical).
static int run_witness_map(lzkp_pk *pk, Workspace &ws, uint32_t P, cudaStream_t st) {
    const uint32_t n = pk->n, threads = std::max(32u, std::min(n / 2, 512u));
    const size_t smem = (size_t)32 * n;
    Region reg(pk, LZKP_REGION_WITNESS_MAP, st);
    if (pk->tiled_wm) {
        // a3-a7 on a domain above 2^12: SpMV, then all 3P polynomials through iNTT -> coset NTT as ONE batch of
        // tiled passes, pointwise (ab - c) / Z(g), coset iNTT of the P quotients, conversion of h to canonical form
        Fr *abc = ws.abc.as<Fr>(), *tmp = ws.tmp.as<Fr>(), *h = ws.h.as<Fr>();
        const size_t plane = (size_t)P * n;
        LAUNCH(k_spmv_abc, dim3((n + 127) / 128, P), 128, 0, st, pk->csr[0], pk->csr[1], pk->csr[2], ws.z.as<Fr>(), abc, P,
               pk->n_vars, pk->m, pk->n_inst, n);
        TRY(large_ntt_device(abc, tmp, pk->log_n, 1, 0, st, 3 * P, n));
        TRY(large_ntt_device(tmp, abc, pk->log_n, 0, 1, st, 3 * P, n));
        LAUNCH(k_pointwise_h, (unsigned)((plane + 127) / 128), 128, 0, st, abc, abc + plane, abc + 2 * plane, tmp, pk->ntt.zinv,
               plane);
        TRY(large_ntt_device(tmp, h, pk->log_n, 1, 1, st, P, n));
        LAUNCH(k_fr_to_canonical, (unsigned)((plane + 127) / 128), 128, 0, st, h, plane);
        return LZKP_OK;
    }
    LAUNCH(k_spmv_abc, dim3((n + 127) / 128, P), 128, 0, st, pk->csr[0], pk->csr[1], pk->csr[2], ws.z.as<Fr>(),
           ws.abc.as<Fr>(), P, pk->n_vars, pk->m, pk->n_inst, n);
    LAUNCH(k_ntt_icoset, dim3(P, 3), threads, smem, st, ws.abc.as<Fr>(), pk->ntt, P, pk->log_n);
    LAUNCH(k_ntt_final, P, threads, smem, st, ws.abc.as<Fr>(), ws.h.as<Fr>(), pk->ntt, P, pk->log_n);
    return LZKP_OK;
}

// From ws_z, r, s (device, canonical) to proofs (device).  status must be initialised by the caller.
// phase (large mode, sharded proving): 1 = inputs + the z-only MSMs on the side streams, 2 = the H MSM + join,
// 3 = both (default).
static int run_prove(lzkp_pk *pk, Workspace &ws, uint32_t P, const Fr *d_r, const Fr *d_s, uint8_t *d_proofs,
                     int32_t *d_status, cudaStream_t st, bool have_h = false, int phase = 3) {
    if (pk->large) {
        if (P != 1) return fail(LZKP_E_STATE, "large-domain proving runs one proof per pass");
        const uint32_t nv = pk->n_vars, ni = pk->n_inst, nw = pk->n_wit;
        const uint8_t *z = ws.z.as<uint8_t>();
        uint8_t *sa = pk->L_sa.as<uint8_t>(), *sb = pk->L_sb.as<uint8_t>(), *sl = pk->L_sl.as<uint8_t>();
        G1XYZZ *res1 = ws.res1.as<G1XYZZ>();
        const uint32_t *lo = pk->L_lo, *cnt = pk->L_cnt;
        if (phase & 1) {
        LAUNCH(k_fr_mul_canonical, 1, 128, 0, st, d_r, d_s, ws.rs.as<Fr>(), 1u);
        LAUNCH(k_check_canonical, (nv + 127) / 128, 128, 0, st, ws.z.as<Fr>(), nv, d_status);
        LAUNCH(k_check_canonical, 1, 32, 0, st, d_r, 1u, d_status);
        LAUNCH(k_check_canonical, 1, 32, 0, st, d_s, 1u, d_status);
        // scalar vectors: z[1..] || r, z[1..] || s, z[n_inst..] || rs (the last entry multiplies +-delta)
        const cudaMemcpyKind dd = cudaMemcpyDeviceToDevice;
        CUDA_TRY(cudaMemcpyAsync(sa, z + 32, (size_t)(nv - 1) * 32, dd, st));
        CUDA_TRY(cudaMemcpyAsync(sa + (size_t)(nv - 1) * 32, d_r, 32, dd, st));
        CUDA_TRY(cudaMemcpyAsync(sb, z + 32, (size_t)(nv - 1) * 32, dd, st));
        CUDA_TRY(cudaMemcpyAsync(sb + (size_t)(nv - 1) * 32, d_s, 32, dd, st));
        CUDA_TRY(cudaMemcpyAsync(sl, z + (size_t)ni * 32, (size_t)nw * 32, dd, st));
        CUDA_TRY(cudaMemcpyAsync(sl + (size_t)nw * 32, ws.rs.p, 32, dd, st));
        // fork: the z-only MSMs (a, l | b1 | b2) on three side streams; this stream runs the witness map, then h
        CUDA_TRY(cudaEventRecord(pk->L_ev_in, st));
        for (auto s_ : pk->L_st) CUDA_TRY(cudaStreamWaitEvent(s_, pk->L_ev_in, 0));
        CUDA_TRY(cudaStreamWaitEvent(pk->L_st_scale, pk->L_ev_in, 0));
        // The A-sum feeds the one serial chain left: slot 4 <- s * A-sum (+ the constant terms on shard 0), k_scale_a.  Both
        // run on the priority stream, so the chain (0.8 ms) ends under the other MSMs instead of after them.
        TRY(msm_device_raw(pk->L_a, sa + (size_t)lo[0] * 32, cnt[0], res1 + 0, pk->L_st_scale));
        pk->L_scaled = cnt[0] || pk->shard_index == 0;
        if (pk->L_scaled) LAUNCH(k_scale_a, 1, 128, 0, pk->L_st_scale, res1, pk->consts, d_r, d_s, pk->shard_index == 0 ? 1 : 0);
        CUDA_TRY(cudaEventRecord(pk->L_ev_scale, pk->L_st_scale));
        {
            Region reg(pk, LZKP_REGION_MSM_G1, pk->L_st[0]);
            TRY(msm_device_raw(pk->L_l, sl + (size_t)lo[2] * 32, cnt[2], res1 + 2, pk->L_st[0]));
        }
        // B1 only enters the proof as r * B1: its MSM runs on r * z_i (the delta extra: r * s), so no scalar multiplication
        // follows it; s * A-sum and the constant terms are scaled beside the remaining MSMs (k_scale_a).
        if (cnt[1]) {
            uint8_t *sb1 = pk->L_sb1.as<uint8_t>();
            const uint32_t last = nv - 1, hi = lo[1] + cnt[1], zc = std::min(hi, last) - lo[1];
            if (zc) LAUNCH(k_scalars_times, (zc + 127) / 128, 128, 0, pk->L_st[1], (const Fr *)(sb + (size_t)lo[1] * 32), d_r,
                           (Fr *)(sb1 + (size_t)lo[1] * 32), zc);
            if (hi > last) CUDA_TRY(cudaMemcpyAsync(sb1 + (size_t)last * 32, ws.rs.p, 32, dd, pk->L_st[1]));
            TRY(msm_device_raw(pk->L_b1, sb1 + (size_t)lo[1] * 32, cnt[1], res1 + 1, pk->L_st[1]));
        } else {
            TRY(msm_device_raw(pk->L_b1, sb, 0, res1 + 1, pk->L_st[1]));
        }
        {
            Region reg(pk, LZKP_REGION_MSM_G2, pk->L_st[2]);
            TRY(msm_device_raw(pk->L_b2, sb + (size_t)lo[4] * 32, cnt[4], ws.res2.p, pk->L_st[2]));
        }
        }
        if (!(phase & 2)) return LZKP_OK;
        if (!have_h && cnt[3]) TRY(run_witness_map(pk, ws, P, st));      // a shard without h_query points skips the map
        TRY(msm_device_raw(pk->L_h, ws.h.as<uint8_t>() + (size_t)lo[3] * 32, cnt[3], res1 + 3, st));
        for (int i = 0; i < 3; i++) {
            CUDA_TRY(cudaEventRecord(pk->L_ev_done[i], pk->L_st[i]));
            CUDA_TRY(cudaStreamWaitEvent(st, pk->L_ev_done[i], 0));
        }
        CUDA_TRY(cudaStreamWaitEvent(st, pk->L_ev_scale, 0));
        if (pk->L_scaled) LAUNCH(k_add_slot, 1, 1, 0, st, res1, 1, 4);
        if (!d_proofs) return LZKP_OK;           // partial sums only (sharded proving): the caller combines
        Region reg(pk, LZKP_REGION_ASSEMBLE, st);
        LAUNCH(k_assemble_sums, 1, 96, 0, st, res1, ws.res2.as<G2XYZZ>(), pk->consts, 1u, d_proofs, 1, -1);
        return LZKP_OK;
    }
    const uint32_t c = pk->c, W = pk->W, gx = (P + 127) / 128;
    void *dig = ws.dig.p;
    const uint32_t dig_bytes = pk->c > 16 ? 4u : 2u;      // signed c-bit digits: int16 up to c = 16
    const bool lat = use_lat(pk, P);
    const uint32_t ymax = 32768u;
    // digits of z, r, s, rs (everything but h); the latency form adds the rows s * z_i and r * z_i
    auto digits_z = [&](auto *dg) -> int {
        using DigT = std::remove_pointer_t<decltype(dg)>;
        LAUNCH(k_digits<DigT>, dim3(gx, std::min(pk->nz, ymax)), 128, 0, st, ws.z.as<Fr>(), pk->n_vars, 1u, dg, 0u, P, c, W, d_status, pk->nz);
        LAUNCH(k_digits<DigT>, dim3(gx, 1), 128, 0, st, d_r, 1u, 0u, dg, pk->nz, P, c, W, d_status, 1u);
        LAUNCH(k_digits<DigT>, dim3(gx, 1), 128, 0, st, d_s, 1u, 0u, dg, pk->nz + 1, P, c, W, d_status, 1u);
        LAUNCH(k_digits<DigT>, dim3(gx, 1), 128, 0, st, ws.rs.as<Fr>(), 1u, 0u, dg, pk->nz + 2, P, c, W, d_status, 1u);
        if (lat) {
            LAUNCH(k_digits_scaled<DigT>, dim3(gx, std::min(pk->nz, ymax)), 128, 0, st, ws.z.as<Fr>(), pk->n_vars, 1u, d_s, dg, pk->row_sz, P, c, W, pk->nz);
            LAUNCH(k_digits_scaled<DigT>, dim3(gx, std::min(pk->nz, ymax)), 128, 0, st, ws.z.as<Fr>(), pk->n_vars, 1u, d_r, dg, pk->row_rz, P, c, W, pk->nz);
        }
        return LZKP_OK;
    };
    auto digits_h = [&](auto *dg) -> int {
        using DigT = std::remove_pointer_t<decltype(dg)>;
        LAUNCH(k_digits<DigT>, dim3(gx, std::min(pk->n - 1, ymax)), 128, 0, st, ws.h.as<Fr>(), pk->n, 0u, dg, pk->nz + 3, P, c, W, d_status,
               pk->n - 1);
        return LZKP_OK;
    };
    auto args = [&](MsmPlan &pl, int iv, void *partial, void *out) {
        return BatchMsmArgs{pl.table.p, pk->N, pl.unit_dig.as<uint32_t>(), pl.unit_tbl.as<uint32_t>(), pl.items[iv].p,
                            pl.n_items[iv], pl.msm_items[iv].p, pl.n_msm, dig, dig_bytes, P, partial, out};
    };
    // Latency form: the G2 MSM only needs the digits of z and s, so it runs on a side stream beside the witness map, the
    // digits of h and the G1 MSMs (all of them latency-bound at these sizes) and joins before the assembly.
    cudaStream_t st_g2 = st;
    if (lat) {
        {
            Region reg(pk, LZKP_REGION_DIGITS, st);
            LAUNCH(k_fr_mul_canonical, gx, 128, 0, st, d_r, d_s, ws.rs.as<Fr>(), P);
            if (dig_bytes == 2) TRY(digits_z((int16_t *)dig)); else TRY(digits_z((int32_t *)dig));
        }
        st_g2 = pk->L_st[0];
        CUDA_TRY(cudaEventRecord(pk->L_ev_in, st));
        CUDA_TRY(cudaStreamWaitEvent(st_g2, pk->L_ev_in, 0));
        { Region reg(pk, LZKP_REGION_MSM_G2, st_g2); batch_msm_g2(args(pk->g2, fit_variant(pk->g2, item_variant_g2(P)), ws.part2.p, ws.res2.p), st_g2); }
        CUDA_TRY(cudaEventRecord(pk->L_ev_done[0], st_g2));
        if (!have_h) TRY(run_witness_map(pk, ws, P, st));
        { Region reg(pk, LZKP_REGION_DIGITS, st); if (dig_bytes == 2) TRY(digits_h((int16_t *)dig)); else TRY(digits_h((int32_t *)dig)); }
    } else {
        // One stream, stage after stage.  (Measured on B200: running the witness map and the G1 half of the assembly on
        // a side stream underneath the MSM kernels gains < 2 % without stream priority - their CTAs only get SMs in the
        // MSM kernel's last wave - and LOSES 2 % with priority, because a latency-bound CTA that holds 17k registers
        // displaces a quarter of an SM's MSM warps while issuing almost nothing.  Overlap happens across chunks instead.)
        if (!have_h) TRY(run_witness_map(pk, ws, P, st));
        Region reg(pk, LZKP_REGION_DIGITS, st);
        LAUNCH(k_fr_mul_canonical, gx, 128, 0, st, d_r, d_s, ws.rs.as<Fr>(), P);
        if (dig_bytes == 2) { TRY(digits_z((int16_t *)dig)); TRY(digits_h((int16_t *)dig)); }
        else { TRY(digits_z((int32_t *)dig)); TRY(digits_h((int32_t *)dig)); }
    }
    MsmPlan &pl1 = lat ? pk->g1_lat : pk->g1;
    // A/B switch (LZKP_G2_CONCURRENT=1): large batches run the G2 MSM on the side stream beside the G1 MSMs.  Measured
    // 23.84 -> 23.48 ms per 4096-proof step (the two kernels only mix where one drains: each alone fills the register
    // file); capping their residency with shared-memory padding so that they truly co-reside is slower (24.1 - 28.2 ms).
    // Off by default: +1.5 % is not worth losing per-stage timing (the regions overlap) in the bench's roofline.
    static const bool g2_conc = getenv("LZKP_G2_CONCURRENT") && atoi(getenv("LZKP_G2_CONCURRENT")) != 0;
    if (!lat && g2_conc) {
        CUDA_TRY(cudaEventRecord(pk->L_ev_in, st));
        CUDA_TRY(cudaStreamWaitEvent(pk->L_st[0], pk->L_ev_in, 0));
        { Region reg(pk, LZKP_REGION_MSM_G2, pk->L_st[0]); batch_msm_g2(args(pk->g2, fit_variant(pk->g2, item_variant_g2(P)), ws.part2.p, ws.res2.p), pk->L_st[0]); }
        CUDA_TRY(cudaEventRecord(pk->L_ev_done[0], pk->L_st[0]));
    }
    {
        Region reg(pk, LZKP_REGION_MSM_G1, st);
        BatchMsmArgs a1 = args(pl1, fit_variant(pl1, item_variant(P)), ws.part1.p, ws.res1.p);
        a1.table = pk->g1.table.p;                        // the latency plan walks the same tables
        batch_msm_g1(a1, st);
    }
    if (lat || g2_conc) CUDA_TRY(cudaStreamWaitEvent(st, pk->L_ev_done[0], 0));
    else { Region reg(pk, LZKP_REGION_MSM_G2, st); batch_msm_g2(args(pk->g2, fit_variant(pk->g2, item_variant_g2(P)), ws.part2.p, ws.res2.p), st); }
    Region reg(pk, LZKP_REGION_ASSEMBLE, st);
    if (lat) {
        LAUNCH(k_assemble_sums, (P + 31) / 32, 96, 0, st, ws.res1.as<G1XYZZ>(), ws.res2.as<G2XYZZ>(), pk->consts, P, d_proofs, 4, 5);
        return LZKP_OK;
    }
    LAUNCH(k_assemble, (P + 31) / 32, 128, 0, st, ws.res1.as<G1XYZZ>(), ws.res2.as<G2XYZZ>(), pk->consts, d_r, d_s, P, d_proofs);
    return LZKP_OK;
}

static void blank_failed(size_t n, const int32_t *status, uint8_t *proofs) {
    for (size_t i = 0; i < n; i++)
        if (status[i]) memset(proofs + 256 * i, 0, 256);
}

// ------------------------------------------------------------------------ stand-alone small NTT
// n <= 4096: one CTA, whole vector in shared memory (k_ntt_small).  Larger sizes: ntt_large.cu.
static int small_ntt_host(uint8_t *data, uint32_t log_n, int inverse, int coset) {
    const uint32_t n = 1u << log_n;
    DBuf d, tw_f, tw_i, cbr, ubr;
    TRY(d.alloc((size_t)n * 32));
    TRY(tw_f.alloc(sizeof(Fr) * std::max(1u, n / 2))); TRY(tw_i.alloc(sizeof(Fr) * std::max(1u, n / 2)));
    TRY(cbr.alloc(sizeof(Fr) * n)); TRY(ubr.alloc(sizeof(Fr) * n));
    Fr w, wi, g, gi;
    for (int i = 0; i < 8; i++) { w.l[i] = FrParams::ROOT28(i); wi.l[i] = FrParams::ROOT28_INV(i); g.l[i] = FrParams::GEN(i); gi.l[i] = FrParams::GEN_INV(i); }
    for (uint32_t i = log_n; i < 28; i++) { w = w.sqr(); wi = wi.sqr(); }
    Fr ninv = host::fr_from_u64(n).inverse();
    cudaStream_t st = nullptr;
    if (n >= 2) {
        LAUNCH(k_pow_table, (n / 2 + 127) / 128, 128, 0, st, tw_f.as<Fr>(), w, Fr::one(), n / 2, 0u);
        LAUNCH(k_pow_table, (n / 2 + 127) / 128, 128, 0, st, tw_i.as<Fr>(), wi, Fr::one(), n / 2, 0u);
    }
    LAUNCH(k_pow_table, (n + 127) / 128, 128, 0, st, cbr.as<Fr>(), g, ninv, n, log_n);
    LAUNCH(k_pow_table, (n + 127) / 128, 128, 0, st, ubr.as<Fr>(), gi, ninv.to_canonical(), n, log_n);
    NttTables T{tw_f.as<Fr>(), tw_i.as<Fr>(), cbr.as<Fr>(), ubr.as<Fr>(), nullptr, ninv, Fr::zero()};
    CUDA_TRY(cudaMemcpy(d.p, data, (size_t)n * 32, cudaMemcpyHostToDevice));
    size_t smem = (size_t)32 * n;
    if (smem > 48 * 1024) CUDA_TRY(cudaFuncSetAttribute(k_ntt_small, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    LAUNCH(k_ntt_small, 1, std::max(32u, std::min(n / 2, 512u)), smem, st, d.as<Fr>(), T, log_n, inverse, coset);
    CUDA_TRY(cudaMemcpy(data, d.p, (size_t)n * 32, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaGetLastError());
    return LZKP_OK;
}

// ------------------------------------------------------------------------ C ABI
// ---- chunked, double-buffered batches
// A batch is cut into chunks; chunk i uses workspace i & 1 on stream i & 1, so two chunks are in flight.
static uint32_t chunk_size(const lzkp_pk *pk, size_t n) {
    if (pk->large) return 1;
    uint32_t c = pk->max_chunk;
    static const int split = getenv("LZKP_BATCH_SPLIT") ? atoi(getenv("LZKP_BATCH_SPLIT")) : 1;
    if (split > 1 && n >= 1024) {         // cut one batch into `split` chunks so that two are in flight
        uint32_t q = (uint32_t)((n + split - 1) / split);
        q = (q + 127) / 128 * 128;
        c = std::min(c, std::max(256u, q));
    }
    return c;
}
struct HostOut {
    uint8_t *proofs; int32_t *status; uint8_t *commit;
    // libzkp envelopes instead of bare proofs (proofs == nullptr): scheme id, per-proof stride, lengths out
    uint8_t *env = nullptr; uint32_t *env_len = nullptr; uint32_t env_stride = 0, scheme = 0; bool with_sets = false;
    uint32_t set_stride = 0;
};
// Host-buffer batch: `prep(ws, off, P, st)` enqueues the chunk's input copies and witness generation.
template <class Prep>
static int run_batch_host(lzkp_pk *pk, size_t n, const uint8_t *r, const uint8_t *s, HostOut out, Prep prep) {
    const uint32_t C = chunk_size(pk, n);
    struct Pending { size_t off; uint32_t P; int w; };
    std::vector<Pending> pend;
    auto drain = [&](int w) -> int {       // copy finished chunks of workspace w from pinned staging to the caller
        CUDA_TRY(cudaStreamSynchronize(pk->chunk_stream(w)));
        for (auto it = pend.begin(); it != pend.end();) {
            if (it->w != w) { ++it; continue; }
            Workspace &ws = pk->ws[w];
            if (out.proofs) memcpy(out.proofs + it->off * 256, ws.h_proofs.p, (size_t)it->P * 256);
            if (out.env) {
                memcpy(out.env + it->off * out.env_stride, ws.h_env.p, (size_t)it->P * out.env_stride);
                memcpy(out.env_len + it->off, ws.h_envlen.p, (size_t)it->P * 4);
            }
            memcpy(out.status + it->off, ws.h_status.p, (size_t)it->P * 4);
            if (out.commit) memcpy(out.commit + it->off * 32, ws.h_commit.p, (size_t)it->P * 32);
            it = pend.erase(it);
        }
        return LZKP_OK;
    };
    int i = 0;
    for (size_t off = 0; off < n; off += C, i++) {
        const int w = pk->large ? 0 : (i & 1);
        const uint32_t P = (uint32_t)std::min<size_t>(C, n - off);
        Workspace &ws = pk->ws[w];
        cudaStream_t st = pk->chunk_stream(w);
        TRY(drain(w));                                    // the staging buffers of this workspace are free again
        TRY(ws_acquire(ws, st));                          // ... and so are its device buffers (a *_device call may still run)
        TRY(ensure_workspace(pk, ws, P));
        TRY(ws.h_proofs.ensure((size_t)ws.chunk * 256)); TRY(ws.h_status.ensure((size_t)ws.chunk * 4));
        TRY(ws.h_commit.ensure((size_t)ws.chunk * 32));
        CUDA_TRY(cudaMemcpyAsync(ws.r.p, r + off * 32, (size_t)P * 32, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(ws.s.p, s + off * 32, (size_t)P * 32, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemsetAsync(ws.status.p, 0, (size_t)P * 4, st));
        TRY(prep(ws, off, P, st));
        TRY(run_prove(pk, ws, P, ws.r.as<Fr>(), ws.s.as<Fr>(), ws.proofs.as<uint8_t>(), ws.status.as<int32_t>(), st));
        if (out.proofs) CUDA_TRY(cudaMemcpyAsync(ws.h_proofs.p, ws.proofs.p, (size_t)P * 256, cudaMemcpyDeviceToHost, st));
        if (out.env) {
            TRY(ws.env.ensure((size_t)ws.chunk * out.env_stride)); TRY(ws.envlen.ensure((size_t)ws.chunk * 4));
            TRY(ws.h_env.ensure((size_t)ws.chunk * out.env_stride)); TRY(ws.h_envlen.ensure((size_t)ws.chunk * 4));
            LAUNCH(k_envelope, (P * 32 + 127) / 128, 128, 0, st, ws.proofs.as<uint8_t>(), ws.commit.as<uint8_t>(),
                   ws.status.as<int32_t>(), out.with_sets ? ws.sets.as<uint64_t>() : nullptr, ws.setlen.as<uint32_t>(),
                   out.set_stride, out.scheme, P, ws.env.as<uint8_t>(), out.env_stride, ws.envlen.as<uint32_t>());
            CUDA_TRY(cudaMemcpyAsync(ws.h_env.p, ws.env.p, (size_t)P * out.env_stride, cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaMemcpyAsync(ws.h_envlen.p, ws.envlen.p, (size_t)P * 4, cudaMemcpyDeviceToHost, st));
        }
        CUDA_TRY(cudaMemcpyAsync(ws.h_status.p, ws.status.p, (size_t)P * 4, cudaMemcpyDeviceToHost, st));
        if (out.commit) CUDA_TRY(cudaMemcpyAsync(ws.h_commit.p, ws.commit.p, (size_t)P * 32, cudaMemcpyDeviceToHost, st));
        TRY(ws_release(ws, st));
        pend.push_back({off, P, w});
    }
    TRY(drain(0));
    TRY(drain(1));
    CUDA_TRY(cudaGetLastError());
    if (out.proofs) blank_failed(n, out.status, out.proofs);
    return LZKP_OK;
}
// Device-buffer batch on the caller's stream: fork to the two engine streams, join back.
template <class Prep>
static int run_batch_device(lzkp_pk *pk, size_t n, const void *d_r, const void *d_s, void *d_proofs, void *d_status,
                            cudaStream_t caller, Prep prep) {
    const uint32_t C = chunk_size(pk, n);
    const bool fork = !pk->large && n > C;               // a single chunk runs directly on the caller's stream
    if (fork) {
        CUDA_TRY(cudaEventRecord(pk->ev_fork, caller));
        CUDA_TRY(cudaStreamWaitEvent(pk->stream, pk->ev_fork, 0));
        CUDA_TRY(cudaStreamWaitEvent(pk->stream2, pk->ev_fork, 0));
    }
    int i = 0;
    for (size_t off = 0; off < n; off += C, i++) {
        const int w = fork ? (i & 1) : 0;
        const uint32_t P = (uint32_t)std::min<size_t>(C, n - off);
        Workspace &ws = pk->ws[w];
        cudaStream_t st = fork ? pk->chunk_stream(w) : caller;
        TRY(ws_acquire(ws, st));
        TRY(ensure_workspace(pk, ws, P));
        int32_t *stat = (int32_t *)d_status + off;
        CUDA_TRY(cudaMemsetAsync(stat, 0, (size_t)P * 4, st));
        TRY(prep(ws, off, P, stat, st));
        TRY(run_prove(pk, ws, P, (const Fr *)d_r + off, (const Fr *)d_s + off, (uint8_t *)d_proofs + off * 256, stat, st));
        TRY(ws_release(ws, st));
    }
    if (fork) {
        for (int w = 0; w < 2; w++) {
            CUDA_TRY(cudaEventRecord(pk->ev_join[w], pk->chunk_stream(w)));
            CUDA_TRY(cudaStreamWaitEvent(caller, pk->ev_join[w], 0));
        }
    }
    CUDA_TRY(cudaGetLastError());
    return LZKP_OK;
}

// ---- one call, every device: a replicated key cuts a host-buffer batch into one contiguous block per device and
// runs each block on its own host thread (streams, workspaces and staging buffers are per replica); results land in
// disjoint slices of the caller's buffers, so order is preserved and there is no gather step.
static constexpr size_t kFanMinBlock = 256;      // below this a block is latency-bound: fewer devices are used
static thread_local bool t_in_fan = false;       // set while a thread runs ONE block of a fan-out (the primary's block must not fan out again)
static inline bool should_fan(const lzkp_pk *pk, size_t n) {
    return !t_in_fan && !pk->replicas.empty() && n >= 2 * kFanMinBlock;
}
static HostOut slice(HostOut o, size_t off) {
    if (o.proofs) o.proofs += off * 256;
    o.status += off;
    if (o.commit) o.commit += off * 32;
    if (o.env) { o.env += off * o.env_stride; o.env_len += off; }
    return o;
}
template <class Fn>
static int fan_out(lzkp_pk *pk, size_t n, Fn fn) {
    const size_t G = std::min<size_t>(1 + pk->replicas.size(), std::max<size_t>(1, n / kFanMinBlock));
    const size_t base = n / G, rem = n % G;
    auto begin = [&](size_t g) { return g * base + std::min(g, rem); };
    std::vector<int> rcs(G, LZKP_OK);
    std::vector<std::string> errs(G);
    std::vector<std::thread> th;
    for (size_t g = 1; g < G; g++)
        th.emplace_back([&, g] {
            lzkp_pk *q = pk->replicas[g - 1];
            DeviceScope ds(q->device);
            t_in_fan = true;
            rcs[g] = fn(q, begin(g), begin(g + 1) - begin(g));
            if (rcs[g] != LZKP_OK) errs[g] = g_err;
        });
    t_in_fan = true;
    rcs[0] = fn(pk, 0, begin(1));
    t_in_fan = false;
    if (rcs[0] != LZKP_OK) errs[0] = g_err;
    for (auto &t : th) t.join();
    for (size_t g = 0; g < G; g++)
        if (rcs[g] != LZKP_OK) return fail(rcs[g], errs[g]);
    return LZKP_OK;
}

#pragma GCC visibility push(default)
extern "C" {

int lzkp_init(const int *devices, int n_devices) {
    if (devices && n_devices > 0) {
        int visible = 0;
        if (cudaGetDeviceCount(&visible) != cudaSuccess || visible == 0) {
            cudaGetLastError();
            return fail(LZKP_E_NO_DEVICE, "no CUDA device: this engine has no CPU fallback");
        }
        if (n_devices > 64) return fail(LZKP_E_INVALID, "at most 64 devices");
        for (int i = 0; i < n_devices; i++) {
            if (devices[i] < 0 || devices[i] >= visible) return fail(LZKP_E_INVALID, "device index out of range");
            for (int j = 0; j < i; j++) if (devices[j] == devices[i]) return fail(LZKP_E_INVALID, "device listed twice");
        }
        std::lock_guard<std::mutex> lk(g_mu);
        if (g_device >= 0 && g_device != devices[0]) return fail(LZKP_E_STATE, "device already selected");
        g_device = devices[0];
        // the list may grow on a later call (keys loaded before it keep the replicas they were loaded with)
        if ((size_t)n_devices > g_devices.size()) g_devices.assign(devices, devices + n_devices);
    }
    TRY(ensure_device());
    std::vector<int> devs;
    { std::lock_guard<std::mutex> lk(g_mu); devs = g_devices; }
    for (size_t i = 1; i < devs.size(); i++) {           // contexts + constants of the other devices, now rather than mid-batch
        DeviceScope ds(devs[i]);
        TRY(ensure_device());
    }
    return LZKP_OK;
}
int lzkp_device_count(void) {
    std::lock_guard<std::mutex> lk(g_mu);
    return g_devices.empty() ? (g_device >= 0 ? 1 : 0) : (int)g_devices.size();
}
int lzkp_shutdown(void) {        // releases the process-wide caches (NTT plans, generator tables); keys are freed by lzkp_pk_free
    if (g_device >= 0) cudaSetDevice(g_device);
    ntt_plans_free();                  // (plans of every device: each is freed under its own device)
    generator_tables_free();
    return LZKP_OK;
}
const char *lzkp_last_error(void) { return g_err.c_str(); }
uint64_t lzkp_kernel_launches(void) { return g_launches.load(); }

int lzkp_profile_enable(int on) {
    g_profile.store(on ? 1 : 0);
    return LZKP_OK;
}
int lzkp_profile_read(lzkp_pk *pk, double ms[LZKP_PROFILE_REGIONS], uint64_t count[LZKP_PROFILE_REGIONS], int reset) {
    if (!pk || !ms || !count) return fail(LZKP_E_INVALID, "null argument");
    TRY(ensure_device());
    std::lock_guard<std::mutex> lk(pk->mu);
    for (auto &m : pk->marks) {
        float t = 0;
        CUDA_TRY(cudaEventSynchronize(m.b));
        CUDA_TRY(cudaEventElapsedTime(&t, m.a, m.b));
        pk->prof_ms[m.region] += t;
        pk->prof_count[m.region]++;
        cudaEventDestroy(m.a);
        cudaEventDestroy(m.b);
    }
    pk->marks.clear();
    for (int i = 0; i < LZKP_PROFILE_REGIONS; i++) {
        ms[i] = pk->prof_ms[i];
        count[i] = pk->prof_count[i];
        if (reset) { pk->prof_ms[i] = 0; pk->prof_count[i] = 0; }
    }
    return LZKP_OK;
}

int lzkp_pk_load_ex(const uint8_t *pk_bytes, size_t len, int validate, const lzkp_pk_options *opt, lzkp_pk **out) {
    if (!pk_bytes || !out) return fail(LZKP_E_INVALID, "null argument");
    *out = nullptr;
    TRY(ensure_device());
    lzkp_pk *pk = new (std::nothrow) lzkp_pk();
    if (!pk) return fail(LZKP_E_NOMEM, "host allocation failed");
    pk->device = current_device();
    int rc = pk_load_impl(pk_bytes, len, validate, opt, pk);
    if (rc != LZKP_OK) {
        delete pk;
        return rc;
    }
    // In-process multi-GPU (SURVEY.md 8e "Batched proving"; the reference's batch path is ONE process,
    // src/advanced/batch.rs:110-140): the key, its tables and workspaces are replicated on every other device of
    // lzkp_init's list, each replica loaded by its own host thread with the window size the primary chose.
    std::vector<int> devs;
    { std::lock_guard<std::mutex> lk(g_mu); devs = g_devices; }
    const bool sharded = opt && opt->shard_count > 1;
    if (devs.size() > 1 && !sharded && !pk->large && pk->device == devs[0]) {
        lzkp_pk_options ro{};
        if (opt) ro = *opt;
        ro.window_bits = pk->c;
        ro.max_chunk = pk->max_chunk;
        const size_t R = devs.size() - 1;
        std::vector<lzkp_pk *> reps(R, nullptr);
        std::vector<int> rcs(R, LZKP_OK);
        std::vector<std::string> errs(R);
        std::vector<std::thread> th;
        for (size_t i = 0; i < R; i++)
            th.emplace_back([&, i] {
                DeviceScope ds(devs[i + 1]);
                int rc_ = ensure_device();
                lzkp_pk *r = rc_ == LZKP_OK ? new (std::nothrow) lzkp_pk() : nullptr;
                if (rc_ == LZKP_OK && !r) rc_ = fail(LZKP_E_NOMEM, "host allocation failed");
                if (rc_ == LZKP_OK) {
                    r->device = devs[i + 1];
                    rc_ = pk_load_impl(pk_bytes, len, 0 /* the primary validated these bytes */, &ro, r);
                }
                if (rc_ != LZKP_OK) { errs[i] = g_err; delete r; r = nullptr; }
                reps[i] = r;
                rcs[i] = rc_;
            });
        for (auto &t : th) t.join();
        for (size_t i = 0; i < R; i++)
            if (rcs[i] != LZKP_OK) {
                for (lzkp_pk *r : reps) if (r) { DeviceScope ds(r->device); delete r; }
                delete pk;
                return fail(rcs[i], "replica on device " + std::to_string(devs[i + 1]) + ": " + errs[i]);
            }
        pk->replicas = reps;
    }
    *out = pk;
    return LZKP_OK;
}
int lzkp_pk_load(const uint8_t *pk_bytes, size_t len, int validate, lzkp_pk **out) {
    return lzkp_pk_load_ex(pk_bytes, len, validate, nullptr, out);
}
void lzkp_pk_free(lzkp_pk *pk) {
    if (!pk) return;
    DeviceScope ds(pk->device);
    delete pk;
}
int lzkp_pk_info(const lzkp_pk *pk, uint64_t info[8]) {
    if (!pk || !info) return fail(LZKP_E_INVALID, "null argument");
    info[0] = pk->n_vars; info[1] = pk->n_inst; info[2] = pk->n_wit; info[3] = pk->n;
    info[4] = (uint64_t)pk->c; info[5] = pk->W; info[6] = pk->table_bytes; info[7] = pk->max_chunk;
    if (pk->large) info[7] = 1;
    return LZKP_OK;
}

int lzkp_pk_shard_info(const lzkp_pk *pk, uint32_t first[5], uint32_t count[5], uint32_t *map_ranks) {
    if (!pk || !first || !count) return fail(LZKP_E_INVALID, "null argument");
    if (!pk->large) return fail(LZKP_E_STATE, "not a large-domain proving key");
    for (int q = 0; q < 5; q++) { first[q] = pk->L_lo[q]; count[q] = pk->L_cnt[q]; }
    if (map_ranks) *map_ranks = pk->map_ranks;
    return LZKP_OK;
}

int lzkp_pk_work(const lzkp_pk *pk, uint64_t work[4]) {
    if (!pk || !work) return fail(LZKP_E_INVALID, "null argument");
    work[0] = pk->g1.n_units; work[1] = pk->g2.n_units; work[2] = pk->g1.n_rows; work[3] = pk->g2.n_rows;
    return LZKP_OK;
}

int lzkp_circuit_load(lzkp_pk *pk, uint32_t m, uint32_t n_inst, uint32_t n_wit, const uint32_t *a_rowptr,
                      const uint32_t *a_col, const uint8_t *a_val, const uint32_t *b_rowptr, const uint32_t *b_col,
                      const uint8_t *b_val, const uint32_t *c_rowptr, const uint32_t *c_col, const uint8_t *c_val) {
    if (!pk || !a_rowptr || !b_rowptr || !c_rowptr) return fail(LZKP_E_INVALID, "null argument");
    TRY(ensure_device());
    std::lock_guard<std::mutex> lk(pk->mu);
    const uint32_t *rp[3] = {a_rowptr, b_rowptr, c_rowptr}, *cl[3] = {a_col, b_col, c_col};
    const uint8_t *vl[3] = {a_val, b_val, c_val};
    pk->kind = -1;
    TRY(circuit_install(pk, m, n_inst, n_wit, rp, cl, vl));
    for (lzkp_pk *q : pk->replicas) {
        DeviceScope ds(q->device);
        TRY(ensure_device());
        std::lock_guard<std::mutex> lq(q->mu);
        q->kind = -1;
        TRY(circuit_install(q, m, n_inst, n_wit, rp, cl, vl));
    }
    return LZKP_OK;
}
static host::R1cs synth(int kind, uint32_t param) {
    return kind == LZKP_CIRCUIT_EQUALITY ? host::synth_equality(param) : host::synth_membership(param);
}
int lzkp_circuit_builtin(lzkp_pk *pk, int kind, uint32_t param) {
    if (!pk || (kind != LZKP_CIRCUIT_EQUALITY && kind != LZKP_CIRCUIT_MEMBERSHIP) || param == 0)
        return fail(LZKP_E_INVALID, "bad circuit kind / parameter");
    TRY(ensure_device());
    std::lock_guard<std::mutex> lk(pk->mu);
    host::R1cs cs = synth(kind, param);
    const host::Csr *M[3] = {&cs.A, &cs.B, &cs.C};
    const uint32_t *rp[3], *cl[3];
    const uint8_t *vl[3];
    for (int k = 0; k < 3; k++) {
        rp[k] = M[k]->rowptr.data(); cl[k] = M[k]->col.data();
        vl[k] = reinterpret_cast<const uint8_t *>(M[k]->val.data());
    }
    TRY(circuit_install(pk, cs.m, cs.n_inst, cs.n_wit, rp, cl, vl));
    pk->kind = kind;
    pk->kind_param = param;
    for (lzkp_pk *q : pk->replicas) {
        DeviceScope ds(q->device);
        TRY(ensure_device());
        std::lock_guard<std::mutex> lq(q->mu);
        TRY(circuit_install(q, cs.m, cs.n_inst, cs.n_wit, rp, cl, vl));
        q->kind = kind;
        q->kind_param = param;
    }
    return LZKP_OK;
}
int lzkp_builtin_circuit_csr(int kind, uint32_t param, uint64_t shape[6], uint32_t *rowptr[3], uint32_t *col[3],
                             uint8_t *val[3]) {
    if ((kind != LZKP_CIRCUIT_EQUALITY && kind != LZKP_CIRCUIT_MEMBERSHIP) || param == 0 || !shape)
        return fail(LZKP_E_INVALID, "bad circuit kind / parameter");
    host::R1cs cs = synth(kind, param);
    const host::Csr *M[3] = {&cs.A, &cs.B, &cs.C};
    shape[0] = cs.m; shape[1] = cs.n_inst; shape[2] = cs.n_wit;
    for (int k = 0; k < 3; k++) shape[3 + k] = M[k]->col.size();
    if (rowptr && col && val)
        for (int k = 0; k < 3; k++) {
            memcpy(rowptr[k], M[k]->rowptr.data(), sizeof(uint32_t) * (cs.m + 1));
            memcpy(col[k], M[k]->col.data(), sizeof(uint32_t) * M[k]->col.size());
            memcpy(val[k], M[k]->val.data(), 32 * M[k]->col.size());
        }
    return LZKP_OK;
}

int lzkp_key_sizes(uint32_t m, uint32_t n_inst, uint32_t n_wit, size_t *pk_len, size_t *vk_len) {
    if (!pk_len || !vk_len || n_inst < 1) return fail(LZKP_E_INVALID, "bad argument");
    uint64_t need = (uint64_t)m + n_inst, n = 2;
    while (n < need) n <<= 1;
    const size_t nv = (size_t)n_inst + n_wit;
    *vk_len = 64 + 3 * 128 + 8 + 64 * (size_t)n_inst;
    *pk_len = *vk_len + 128 + 5 * 8 + 64 * (2 * nv + (n - 1) + n_wit) + 128 * nv;
    return LZKP_OK;
}
static int setup_common(uint32_t m, uint32_t n_inst, uint32_t n_wit, const uint32_t *const rp[3],
                        const uint32_t *const cl[3], const uint8_t *const vl[3], const uint8_t *toxic, uint8_t *pk_out,
                        size_t pk_cap, uint8_t *vk_out, size_t vk_cap) {
    if (!toxic || !pk_out || !vk_out) return fail(LZKP_E_INVALID, "null argument");
    size_t pl, vl_;
    TRY(lzkp_key_sizes(m, n_inst, n_wit, &pl, &vl_));
    if (pk_cap < pl || vk_cap < vl_) return fail(LZKP_E_INVALID, "setup: output buffer too small (see lzkp_key_sizes)");
    TRY(ensure_device());
    std::vector<uint8_t> pk, vk;
    TRY(setup_run(m, n_inst, n_wit, rp, cl, vl, toxic, pk, vk));
    if (pk.size() != pl || vk.size() != vl_) return fail(LZKP_E_STATE, "setup: size mismatch");
    memcpy(pk_out, pk.data(), pl);
    memcpy(vk_out, vk.data(), vl_);
    return LZKP_OK;
}
int lzkp_setup(uint32_t m, uint32_t n_inst, uint32_t n_wit, const uint32_t *a_rowptr, const uint32_t *a_col,
               const uint8_t *a_val, const uint32_t *b_rowptr, const uint32_t *b_col, const uint8_t *b_val,
               const uint32_t *c_rowptr, const uint32_t *c_col, const uint8_t *c_val, const uint8_t toxic[160],
               uint8_t *pk_out, size_t pk_cap, uint8_t *vk_out, size_t vk_cap) {
    if (!a_rowptr || !b_rowptr || !c_rowptr) return fail(LZKP_E_INVALID, "null argument");
    const uint32_t *rp[3] = {a_rowptr, b_rowptr, c_rowptr}, *cl[3] = {a_col, b_col, c_col};
    const uint8_t *vl[3] = {a_val, b_val, c_val};
    return setup_common(m, n_inst, n_wit, rp, cl, vl, toxic, pk_out, pk_cap, vk_out, vk_cap);
}
int lzkp_setup_builtin(int kind, uint32_t param, const uint8_t toxic[160], uint8_t *pk_out, size_t pk_cap,
                       uint8_t *vk_out, size_t vk_cap) {
    if ((kind != LZKP_CIRCUIT_EQUALITY && kind != LZKP_CIRCUIT_MEMBERSHIP) || param == 0)
        return fail(LZKP_E_INVALID, "bad circuit kind / parameter");
    host::R1cs cs = synth(kind, param);
    const host::Csr *M[3] = {&cs.A, &cs.B, &cs.C};
    const uint32_t *rp[3], *cl[3];
    const uint8_t *vl[3];
    for (int k = 0; k < 3; k++) {
        rp[k] = M[k]->rowptr.data(); cl[k] = M[k]->col.data();
        vl[k] = reinterpret_cast<const uint8_t *>(M[k]->val.data());
    }
    return setup_common(cs.m, cs.n_inst, cs.n_wit, rp, cl, vl, toxic, pk_out, pk_cap, vk_out, vk_cap);
}

int lzkp_generator_mul(int group, const uint8_t *scalars, size_t n, uint8_t *out_affine) {
    if ((group != 1 && group != 2) || (n && (!scalars || !out_affine))) return fail(LZKP_E_INVALID, "bad argument");
    return generator_mul(group, scalars, n, out_affine);
}

int lzkp_prove_batch(lzkp_pk *pk, size_t n_proofs, const uint8_t *z, const uint8_t *r, const uint8_t *s,
                     uint8_t *proofs_out, int32_t *status) {
    if (!pk || (n_proofs && (!z || !r || !s || !proofs_out || !status))) return fail(LZKP_E_INVALID, "null argument");
    if (should_fan(pk, n_proofs)) {
        const size_t zrow = (size_t)pk->n_vars * 32;
        return fan_out(pk, n_proofs, [&](lzkp_pk *q, size_t off, size_t cnt) {
            return lzkp_prove_batch(q, cnt, z + off * zrow, r + off * 32, s + off * 32, proofs_out + off * 256, status + off);
        });
    }
    TRY(ensure_device());
    std::lock_guard<std::mutex> lk(pk->mu);
    if (!pk->has_circuit) return fail(LZKP_E_STATE, "lzkp_circuit_load has not been called");
    const size_t nv = pk->n_vars;
    return run_batch_host(pk, n_proofs, r, s, HostOut{proofs_out, status, nullptr},
                          [&](Workspace &ws, size_t off, uint32_t P, cudaStream_t st) -> int {
        CUDA_TRY(cudaMemcpyAsync(ws.z.p, z + off * nv * 32, (size_t)P * nv * 32, cudaMemcpyHostToDevice, st));
        return LZKP_OK;
    });
}

int lzkp_prove_batch_device(lzkp_pk *pk, size_t n_proofs, const void *d_z, const void *d_r, const void *d_s,
                            void *d_proofs, void *d_status, void *stream) {
    if (!pk || (n_proofs && (!d_z || !d_r || !d_s || !d_proofs || !d_status))) return fail(LZKP_E_INVALID, "null argument");
    TRY(ensure_device());
    std::lock_guard<std::mutex> lk(pk->mu);
    if (!pk->has_circuit) return fail(LZKP_E_STATE, "lzkp_circuit_load has not been called");
    const size_t nv = pk->n_vars;
    return run_batch_device(pk, n_proofs, d_r, d_s, d_proofs, d_status, (cudaStream_t)stream,
                            [&](Workspace &ws, size_t off, uint32_t P, int32_t *, cudaStream_t st) -> int {
        CUDA_TRY(cudaMemcpyAsync(ws.z.p, (const uint8_t *)d_z + off * nv * 32, (size_t)P * nv * 32, cudaMemcpyDeviceToDevice, st));
        return LZKP_OK;
    });
}

int lzkp_builtin_witness(int kind, uint32_t param, uint64_t value, uint64_t other, const uint64_t *set,
                         uint32_t set_len, const uint8_t *commitment, uint8_t *z_out, size_t z_cap) {
    if (!z_out || param == 0) return fail(LZKP_E_INVALID, "bad argument");
    std::vector<Fr> z;
    if (kind == LZKP_CIRCUIT_EQUALITY) z = host::assign_equality(param, value, other, commitment);
    else if (kind == LZKP_CIRCUIT_MEMBERSHIP) {
        if (!set) return fail(LZKP_E_INVALID, "null set");
        z = host::assign_membership(param, value, set, set_len, commitment);
        if (z.empty()) return fail(LZKP_E_INVALID, "membership inputs rejected (empty / oversized set or value not in set)");
    } else return fail(LZKP_E_INVALID, "bad circuit kind");
    if (z_cap < z.size() * 32) return fail(LZKP_E_INVALID, "z_out too small");
    memcpy(z_out, z.data(), z.size() * 32);
    return LZKP_OK;
}

static int equality_batch_impl(lzkp_pk *pk, size_t n_proofs, const uint64_t *a, const uint64_t *b,
                               const uint8_t *commitments, const uint8_t *r, const uint8_t *s, HostOut out) {
    if (!pk || (n_proofs && (!a || !b || !r || !s || !out.status || (!out.proofs && !out.env)))) return fail(LZKP_E_INVALID, "null argument");
    if (should_fan(pk, n_proofs))
        return fan_out(pk, n_proofs, [&](lzkp_pk *q, size_t off, size_t cnt) {
            return equality_batch_impl(q, cnt, a + off, b + off, commitments ? commitments + off * 32 : nullptr, r + off * 32,
                                       s + off * 32, slice(out, off));
        });
    TRY(ensure_device());
    std::lock_guard<std::mutex> lk(pk->mu);
    if (!pk->has_circuit || pk->kind != LZKP_CIRCUIT_EQUALITY) return fail(LZKP_E_STATE, "pk is not bound to the builtin equality circuit");
    return run_batch_host(pk, n_proofs, r, s, out,
                          [&](Workspace &ws, size_t off, uint32_t P, cudaStream_t st) -> int {
        CUDA_TRY(cudaMemcpyAsync(ws.a.p, a + off, (size_t)P * 8, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(ws.b.p, b + off, (size_t)P * 8, cudaMemcpyHostToDevice, st));
        if (commitments) CUDA_TRY(cudaMemcpyAsync(ws.commit.p, commitments + off * 32, (size_t)P * 32, cudaMemcpyHostToDevice, st));
        Region reg(pk, LZKP_REGION_WITGEN, st);
        LAUNCH(k_witgen_equality, (P + 127) / 128, 128, 0, st, ws.a.as<uint64_t>(), ws.b.as<uint64_t>(),
               commitments ? ws.commit.as<Fr>() : nullptr, ws.z.as<Fr>(), ws.commit.as<Fr>(), ws.status.as<int32_t>(), P,
               pk->kind_param, pk->n_vars);
        wires_to_canonical(ws.z.as<Fr>(), P, pk->n_vars, 4u, 3u * pk->kind_param, st);
        return LZKP_OK;
    });
}

int lzkp_prove_equality_batch(lzkp_pk *pk, size_t n_proofs, const uint64_t *a, const uint64_t *b,
                              const uint8_t *commitments, const uint8_t *r, const uint8_t *s, uint8_t *proofs_out,
                              uint8_t *commitments_out, int32_t *status) {
    if (n_proofs && !proofs_out) return fail(LZKP_E_INVALID, "null argument");
    HostOut out{proofs_out, status, commitments_out};
    return equality_batch_impl(pk, n_proofs, a, b, commitments, r, s, out);
}
int lzkp_prove_equality_enveloped(lzkp_pk *pk, size_t n_proofs, const uint64_t *a, const uint64_t *b, const uint8_t *r,
                                  const uint8_t *s, uint8_t *envelopes_out, uint32_t *envelope_len, int32_t *status) {
    if (n_proofs && (!envelopes_out || !envelope_len)) return fail(LZKP_E_INVALID, "null argument");
    HostOut out{nullptr, status, nullptr};
    out.env = envelopes_out; out.env_len = envelope_len; out.env_stride = 298; out.scheme = 2;
    return equality_batch_impl(pk, n_proofs, a, b, nullptr, r, s, out);
}

static int membership_batch_impl(lzkp_pk *pk, size_t n_proofs, const uint64_t *value, const uint64_t *sets,
                                 const uint32_t *set_len, uint32_t set_stride, const uint8_t *commitments,
                                 const uint8_t *r, const uint8_t *s, HostOut out) {
    if (!pk || (n_proofs && (!value || !sets || !set_len || !r || !s || !out.status || (!out.proofs && !out.env))))
        return fail(LZKP_E_INVALID, "null argument");
    if (n_proofs && set_stride == 0) return fail(LZKP_E_INVALID, "set_stride must be at least 1");
    if (should_fan(pk, n_proofs))
        return fan_out(pk, n_proofs, [&](lzkp_pk *q, size_t off, size_t cnt) {
            return membership_batch_impl(q, cnt, value + off, sets + off * set_stride, set_len + off, set_stride,
                                         commitments ? commitments + off * 32 : nullptr, r + off * 32, s + off * 32, slice(out, off));
        });
    TRY(ensure_device());
    std::lock_guard<std::mutex> lk(pk->mu);
    if (!pk->has_circuit || pk->kind != LZKP_CIRCUIT_MEMBERSHIP) return fail(LZKP_E_STATE, "pk is not bound to the builtin membership circuit");
    return run_batch_host(pk, n_proofs, r, s, out,
                          [&](Workspace &ws, size_t off, uint32_t P, cudaStream_t st) -> int {
        TRY(ws.sets.ensure((size_t)ws.chunk * set_stride * 8));
        TRY(ws.setlen.ensure((size_t)ws.chunk * 4));
        CUDA_TRY(cudaMemcpyAsync(ws.a.p, value + off, (size_t)P * 8, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(ws.sets.p, sets + off * set_stride, (size_t)P * set_stride * 8, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(ws.setlen.p, set_len + off, (size_t)P * 4, cudaMemcpyHostToDevice, st));
        if (commitments) CUDA_TRY(cudaMemcpyAsync(ws.commit.p, commitments + off * 32, (size_t)P * 32, cudaMemcpyHostToDevice, st));
        Region reg(pk, LZKP_REGION_WITGEN, st);
        LAUNCH(k_witgen_membership, (P + 127) / 128, 128, 0, st, ws.a.as<uint64_t>(), ws.sets.as<uint64_t>(),
               ws.setlen.as<uint32_t>(), set_stride, commitments ? ws.commit.as<Fr>() : nullptr, ws.z.as<Fr>(),
               ws.commit.as<Fr>(), ws.status.as<int32_t>(), P, pk->kind_param, pk->n_vars);
        wires_to_canonical(ws.z.as<Fr>(), P, pk->n_vars, 2u + 2u * pk->kind_param + 1u, 330u, st);
        return LZKP_OK;
    });
}

int lzkp_prove_membership_batch(lzkp_pk *pk, size_t n_proofs, const uint64_t *value, const uint64_t *sets,
                                const uint32_t *set_len, uint32_t set_stride, const uint8_t *commitments,
                                const uint8_t *r, const uint8_t *s, uint8_t *proofs_out, uint8_t *commitments_out,
                                int32_t *status) {
    if (n_proofs && !proofs_out) return fail(LZKP_E_INVALID, "null argument");
    HostOut out{proofs_out, status, commitments_out};
    return membership_batch_impl(pk, n_proofs, value, sets, set_len, set_stride, commitments, r, s, out);
}
int lzkp_prove_membership_enveloped(lzkp_pk *pk, size_t n_proofs, const uint64_t *value, const uint64_t *sets,
                                    const uint32_t *set_len, uint32_t set_stride, const uint8_t *r, const uint8_t *s,
                                    uint8_t *envelopes_out, uint32_t envelope_stride, uint32_t *envelope_len,
                                    int32_t *status) {
    if (n_proofs && (!envelopes_out || !envelope_len)) return fail(LZKP_E_INVALID, "null argument");
    if (!pk) return fail(LZKP_E_INVALID, "null argument");
    if (pk->kind != LZKP_CIRCUIT_MEMBERSHIP) return fail(LZKP_E_STATE, "pk is not bound to the builtin membership circuit");
    if (envelope_stride < 10 + 4 + 8 * std::max(pk->kind_param, set_stride) + 256 + 32)
        return fail(LZKP_E_INVALID, "envelope_stride below 302 + 8 * set slots");
    HostOut out{nullptr, status, nullptr};
    out.env = envelopes_out; out.env_len = envelope_len; out.env_stride = envelope_stride; out.scheme = 4;
    out.with_sets = true; out.set_stride = set_stride;
    return membership_batch_impl(pk, n_proofs, value, sets, set_len, set_stride, nullptr, r, s, out);
}

int lzkp_prove_equality_batch_device(lzkp_pk *pk, size_t n_proofs, const void *d_a, const void *d_b, const void *d_r,
                                     const void *d_s, void *d_proofs, void *d_status, void *stream) {
    if (!pk || !d_a || !d_b || !d_r || !d_s || !d_proofs || !d_status) return fail(LZKP_E_INVALID, "null argument");
    TRY(ensure_device());
    std::lock_guard<std::mutex> lk(pk->mu);
    if (!pk->has_circuit || pk->kind != LZKP_CIRCUIT_EQUALITY) return fail(LZKP_E_STATE, "pk is not bound to the builtin equality circuit");
    return run_batch_device(pk, n_proofs, d_r, d_s, d_proofs, d_status, (cudaStream_t)stream,
                            [&](Workspace &ws, size_t off, uint32_t P, int32_t *stat, cudaStream_t st) -> int {
        Region reg(pk, LZKP_REGION_WITGEN, st);
        LAUNCH(k_witgen_equality, (P + 127) / 128, 128, 0, st, (const uint64_t *)d_a + off, (const uint64_t *)d_b + off,
               (const Fr *)nullptr, ws.z.as<Fr>(), ws.commit.as<Fr>(), stat, P, pk->kind_param, pk->n_vars);
        wires_to_canonical(ws.z.as<Fr>(), P, pk->n_vars, 4u, 3u * pk->kind_param, st);
        return LZKP_OK;
    });
}

int lzkp_witness_map(lzkp_pk *pk, size_t n_proofs, const uint8_t *z, uint8_t *h_out) {
    if (!pk || (n_proofs && (!z || !h_out))) return fail(LZKP_E_INVALID, "null argument");
    TRY(ensure_device());
    std::lock_guard<std::mutex> lk(pk->mu);
    if (!pk->has_circuit) return fail(LZKP_E_STATE, "lzkp_circuit_load has not been called");
    cudaStream_t st = pk->stream;
    Workspace &ws = pk->ws[0];
    const size_t nv = pk->n_vars, n = pk->n;
    for (size_t off = 0; off < n_proofs; off += pk->max_chunk) {
        uint32_t P = (uint32_t)std::min<size_t>(pk->max_chunk, n_proofs - off);
        TRY(ws_acquire(ws, st));
        TRY(ensure_workspace(pk, ws, P));
        CUDA_TRY(cudaMemcpyAsync(ws.z.p, z + off * nv * 32, (size_t)P * nv * 32, cudaMemcpyHostToDevice, st));
        TRY(run_witness_map(pk, ws, P, st));
        CUDA_TRY(cudaMemcpyAsync(h_out + off * n * 32, ws.h.p, (size_t)P * n * 32, cudaMemcpyDeviceToHost, st));
        TRY(ws_release(ws, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        CUDA_TRY(cudaGetLastError());
    }
    return LZKP_OK;
}

int lzkp_witness_map_device(lzkp_pk *pk, const void *d_z, void *d_h, void *stream) {
    if (!pk || !d_z || !d_h) return fail(LZKP_E_INVALID, "null argument");
    TRY(ensure_device());
    std::lock_guard<std::mutex> lk(pk->mu);
    if (!pk->has_circuit) return fail(LZKP_E_STATE, "lzkp_circuit_load has not been called");
    cudaStream_t st = (cudaStream_t)stream;
    Workspace &ws = pk->ws[0];
    TRY(ws_acquire(ws, st));
    TRY(ensure_workspace(pk, ws, 1));
    CUDA_TRY(cudaMemcpyAsync(ws.z.p, d_z, (size_t)pk->n_vars * 32, cudaMemcpyDeviceToDevice, st));
    TRY(run_witness_map(pk, ws, 1, st));
    CUDA_TRY(cudaMemcpyAsync(d_h, ws.h.p, (size_t)pk->n * 32, cudaMemcpyDeviceToDevice, st));
    TRY(ws_release(ws, st));
    return LZKP_OK;
}

int lzkp_prove_partial_device(lzkp_pk *pk, const void *d_z, const void *d_r, const void *d_s, const void *d_h,
                              void *d_partial, void *d_status, void *stream, int phase) {
    if (phase == 0) phase = 3;
    if (!pk || !d_r || !d_s || !d_status || ((phase & 1) && !d_z) || ((phase & 2) && !d_partial))
        return fail(LZKP_E_INVALID, "null argument");
    TRY(ensure_device());
    std::lock_guard<std::mutex> lk(pk->mu);
    if (!pk->large) return fail(LZKP_E_STATE, "sharded proving needs a large-domain proving key");
    if ((phase & 2) && !d_h && pk->L_cnt[3] && !pk->has_circuit)
        return fail(LZKP_E_STATE, "this shard holds h_query points: pass h, or bind the circuit so that it runs the witness map itself");
    cudaStream_t st = (cudaStream_t)stream;
    Workspace &ws = pk->ws[0];
    TRY(ws_acquire(ws, st));
    TRY(ensure_workspace(pk, ws, 1));
    if (phase & 1) {
        // the side streams of the previous proof must have left the scalar vectors (their join events are recorded
        // in phase 2; waiting on a never-recorded event is a no-op)
        for (auto ev : pk->L_ev_done) CUDA_TRY(cudaStreamWaitEvent(st, ev, 0));
        if (pk->L_ev_scale) CUDA_TRY(cudaStreamWaitEvent(st, pk->L_ev_scale, 0));
        CUDA_TRY(cudaMemsetAsync(d_status, 0, 4, st));
        CUDA_TRY(cudaMemcpyAsync(ws.z.p, d_z, (size_t)pk->n_vars * 32, cudaMemcpyDeviceToDevice, st));
    }
    if ((phase & 2) && d_h) CUDA_TRY(cudaMemcpyAsync(ws.h.p, d_h, (size_t)pk->n * 32, cudaMemcpyDeviceToDevice, st));
    TRY(run_prove(pk, ws, 1, (const Fr *)d_r, (const Fr *)d_s, nullptr, (int32_t *)d_status, st, d_h != nullptr, phase));
    if (!(phase & 2)) { TRY(ws_release(ws, st)); return LZKP_OK; }
    uint8_t *out = (uint8_t *)d_partial;
    CUDA_TRY(cudaMemcpyAsync(out, ws.res1.p, 4 * sizeof(G1XYZZ), cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(out + 4 * sizeof(G1XYZZ), ws.res2.p, sizeof(G2XYZZ), cudaMemcpyDeviceToDevice, st));
    TRY(ws_release(ws, st));
    return LZKP_OK;
}

int lzkp_prove_combine_device(lzkp_pk *pk, const void *d_partials, int n_partials, const void *d_r, const void *d_s,
                              void *d_proof, void *stream) {
    if (!pk || !d_partials || n_partials < 1 || !d_r || !d_s || !d_proof) return fail(LZKP_E_INVALID, "bad argument");
    TRY(ensure_device());
    std::lock_guard<std::mutex> lk(pk->mu);
    if (!pk->large) return fail(LZKP_E_STATE, "sharded proving needs a large-domain proving key");
    cudaStream_t st = (cudaStream_t)stream;
    Workspace &ws = pk->ws[0];
    TRY(ws_acquire(ws, st));
    TRY(ensure_workspace(pk, ws, 1));
    LAUNCH(k_sum_partials, 1, 160, 0, st, (const uint8_t *)d_partials, (uint32_t)n_partials, ws.res1.as<G1XYZZ>(),
           ws.res2.as<G2XYZZ>());
    // slot 1 of every partial already holds the shard's s * A + r * B1 share (k_scale_ab): the tail is three conversions
    LAUNCH(k_assemble_sums, 1, 96, 0, st, ws.res1.as<G1XYZZ>(), ws.res2.as<G2XYZZ>(), pk->consts, 1u, (uint8_t *)d_proof, 1, -1);
    TRY(ws_release(ws, st));
    CUDA_TRY(cudaGetLastError());
    return LZKP_OK;
}

int lzkp_msm_g1(const uint8_t *bases_affine, const uint8_t *scalars, size_t n, uint8_t *out_affine) {
    if (!out_affine || (n && (!bases_affine || !scalars))) return fail(LZKP_E_INVALID, "null argument");
    TRY(ensure_device());
    return large_msm_g1_host(bases_affine, scalars, n, out_affine);
}
int lzkp_msm_g2(const uint8_t *bases_affine, const uint8_t *scalars, size_t n, uint8_t *out_affine) {
    if (!out_affine || (n && (!bases_affine || !scalars))) return fail(LZKP_E_INVALID, "null argument");
    TRY(ensure_device());
    return large_msm_g2_host(bases_affine, scalars, n, out_affine);
}
struct lzkp_bases { MsmBases *b; };
int lzkp_bases_load(int group, const uint8_t *bases_affine, size_t n, int window_bits, int resident_windows,
                    int validate, lzkp_bases **out) {
    if (!out || (group != 1 && group != 2) || (n && !bases_affine)) return fail(LZKP_E_INVALID, "bad argument");
    *out = nullptr;
    TRY(ensure_device());
    MsmBases *b = nullptr;
    TRY(msm_bases_load(group, bases_affine, n, window_bits, resident_windows, validate, &b));
    *out = new lzkp_bases{b};
    return LZKP_OK;
}
void lzkp_bases_free(lzkp_bases *b) {
    if (!b) return;
    if (g_device >= 0) cudaSetDevice(g_device);
    msm_bases_free(b->b);
    delete b;
}
int lzkp_msm(lzkp_bases *b, const uint8_t *scalars, size_t n, uint8_t *out_affine) {
    if (!b || !out_affine || (n && !scalars)) return fail(LZKP_E_INVALID, "null argument");
    TRY(ensure_device());
    return msm_host(b->b, scalars, n, out_affine);
}
int lzkp_msm_device(lzkp_bases *b, const void *d_scalars, size_t n, void *d_out_affine, void *stream) {
    if (!b || !d_out_affine || (n && !d_scalars)) return fail(LZKP_E_INVALID, "null argument");
    TRY(ensure_device());
    return msm_device(b->b, d_scalars, n, d_out_affine, (cudaStream_t)stream);
}

int lzkp_ntt(uint8_t *data, uint32_t log_n, int inverse, int coset) {
    if (!data || log_n > 28) return fail(LZKP_E_INVALID, "bad argument");
    TRY(ensure_device());
    if (log_n <= 12 && !getenv("LZKP_NTT_FORCE_TILED")) return small_ntt_host(data, log_n, inverse, coset);
    return large_ntt_host(data, log_n, inverse, coset);
}

int lzkp_ntt_device(void *d_in, void *d_out, uint32_t log_n, int inverse, int coset, void *stream) {
    if (!d_in || !d_out || log_n > 28) return fail(LZKP_E_INVALID, "bad argument");
    if (log_n > 11 && d_in == d_out) return fail(LZKP_E_INVALID, "lzkp_ntt_device: d_out must differ from d_in above 2^11");
    TRY(ensure_device());
    return large_ntt_device(d_in, d_out, log_n, inverse, coset, (cudaStream_t)stream);
}

struct lzkp_vk { VerifyingKeyDev *v; };
int lzkp_vk_load(const uint8_t *vk_bytes, size_t len, lzkp_vk **out) {
    if (!vk_bytes || !out) return fail(LZKP_E_INVALID, "null argument");
    *out = nullptr;
    TRY(ensure_device());
    VerifyingKeyDev *v = nullptr;
    TRY(vk_load(vk_bytes, len, &v));
    *out = new lzkp_vk{v};
    return LZKP_OK;
}
int lzkp_vk_info(const lzkp_vk *vk, uint64_t info[4]) {
    if (!vk || !info) return fail(LZKP_E_INVALID, "null argument");
    vk_info(vk->v, info);
    return LZKP_OK;
}
void lzkp_vk_free(lzkp_vk *vk) {
    if (!vk) return;
    if (g_device >= 0) cudaSetDevice(g_device);
    vk_free(vk->v);
    delete vk;
}
int lzkp_verify_batch(lzkp_vk *vk, size_t n, const uint8_t *proofs, const uint8_t *public_inputs, size_t n_pub,
                      uint8_t *ok_out) {
    if (!vk || (n && (!proofs || !ok_out || (n_pub && !public_inputs)))) return fail(LZKP_E_INVALID, "null argument");
    TRY(ensure_device());
    return verify_batch(vk->v, n, proofs, public_inputs, n_pub, ok_out);
}
int lzkp_verify_batch_device(lzkp_vk *vk, size_t n, const void *d_proofs, const void *d_public_inputs, size_t n_pub,
                             void *d_ok, void *stream) {
    if (!vk || (n && (!d_proofs || !d_ok || (n_pub && !d_public_inputs)))) return fail(LZKP_E_INVALID, "null argument");
    TRY(ensure_device());
    return verify_batch_device(vk->v, n, (const uint8_t *)d_proofs, (const uint8_t *)d_public_inputs, n_pub, (uint8_t *)d_ok,
                               (cudaStream_t)stream);
}

int lzkp_commit_value_snark(uint64_t value, uint8_t out[32]) {
    if (!out) return fail(LZKP_E_INVALID, "null argument");
    static std::mutex mu;
    std::lock_guard<std::mutex> lk(mu);
    host::commit_value_snark(value, out);
    return LZKP_OK;
}

}  // extern "C"
#pragma GCC visibility pop
