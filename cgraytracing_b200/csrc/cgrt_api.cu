// cgrt_api.cu — the C ABI of include/cgrt.h: host-side orchestration of the sm_100a kernels.
// There is NO CPU fallback anywhere in this file: without a CUDA device cgrt_create fails with CGRT_ERR_NO_DEVICE.
#include "../../include/cgrt.h"

#include <unistd.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

#include "cgrt_passes.cuh"

#include <dlfcn.h>

using namespace cgrt;

namespace {

struct HostTexture {
    std::vector<uint8_t> rgb;
    int w, h, isbump;
    double n[3], p[3], lenx, leny;
};
struct HostObject {
    int kind;
    double a[3], b[3], r, col[3], refl, transp;
    int tex, objtype;
    std::vector<double> tri9;  // mesh
    std::vector<double> cp;    // bezier
};

struct BvhBuild {
    double *tri9 = nullptr;  // original order, device
    int ntris = 0;
};

// Process-wide cache of the photon pass's large buffers (deposit tables 2 x 8.4 GB, suspended-photon queues 2 x 2.1 GB at 16 Mi
// photons per launch). A render() creates and destroys a context; handing 20 GB back to the stream-ordered pool and carving it up
// again for the next context was measured to cost up to 0.4 s per render. Blocks parked here are plain cudaMalloc allocations that
// the next context of the same device takes over as they are; they are only freed at process exit.
struct ArenaBlock {
    int device;
    size_t bytes;
    void *ptr;
};
std::mutex g_arena_mutex;
std::vector<ArenaBlock> g_arena;

void *arena_take(int device, size_t bytes) {
    {
        std::lock_guard<std::mutex> lk(g_arena_mutex);
        size_t best = g_arena.size();
        for (size_t i = 0; i < g_arena.size(); i++)
            if (g_arena[i].device == device && g_arena[i].bytes >= bytes && (best == g_arena.size() || g_arena[i].bytes < g_arena[best].bytes)) best = i;
        if (best != g_arena.size() && g_arena[best].bytes <= bytes + bytes / 4 + (1u << 20)) {  // close fit only
            void *p = g_arena[best].ptr;
            g_arena.erase(g_arena.begin() + (long)best);
            return p;
        }
    }
    void *p = nullptr;
    if (cudaMalloc(&p, bytes) == cudaSuccess) return p;
    cudaGetLastError();
    // Out of memory while blocks of other sizes sit parked: hand them back to the driver, largest first, until the request fits.
    for (;;) {
        void *victim = nullptr;
        {
            std::lock_guard<std::mutex> lk(g_arena_mutex);
            size_t big = g_arena.size();
            for (size_t i = 0; i < g_arena.size(); i++)
                if (g_arena[i].device == device && (big == g_arena.size() || g_arena[i].bytes > g_arena[big].bytes)) big = i;
            if (big == g_arena.size()) return nullptr;  // nothing left to release: genuinely out of memory
            victim = g_arena[big].ptr;
            g_arena.erase(g_arena.begin() + (long)big);
        }
        cudaFree(victim);
        if (cudaMalloc(&p, bytes) == cudaSuccess) return p;
        cudaGetLastError();
    }
}
// bytes parked for `device` (the photon pass sizes its launches from free + parked memory)
size_t arena_held(int device) {
    std::lock_guard<std::mutex> lk(g_arena_mutex);
    size_t held = 0;
    for (const ArenaBlock &b : g_arena) held += b.device == device ? b.bytes : 0;
    return held;
}
// cudaFree every parked block of `device` (all devices when device < 0) -> bytes released
size_t arena_trim(int device) {
    std::vector<ArenaBlock> victims;
    {
        std::lock_guard<std::mutex> lk(g_arena_mutex);
        for (size_t i = 0; i < g_arena.size();)
            if (device < 0 || g_arena[i].device == device) { victims.push_back(g_arena[i]); g_arena.erase(g_arena.begin() + (long)i); }
            else i++;
    }
    size_t freed = 0;
    int cur = 0;
    cudaGetDevice(&cur);
    for (const ArenaBlock &b : victims) { cudaSetDevice(b.device); cudaFree(b.ptr); freed += b.bytes; }
    cudaSetDevice(cur);
    return freed;
}
void arena_give(int device, size_t bytes, void *p) {
    if (!p) return;
    std::lock_guard<std::mutex> lk(g_arena_mutex);
    size_t held = 0;
    for (const ArenaBlock &b : g_arena) held += b.device == device ? b.bytes : 0;
    if (held + bytes > ((size_t)120 << 30)) { cudaFree(p); return; }  // park at most 120 GB per device
    g_arena.push_back(ArenaBlock{device, bytes, p});
}

// NCCL is bound at run time, never at link time: the communicator a host hands to cgrt_allreduce_accum must be driven by the SAME
// NCCL build that created it, and a process may already hold one (a framework's bundled copy). The copy already loaded in the
// process wins (dlopen with RTLD_NOLOAD finds it by its soname), else the system's libnccl.so.2 is loaded.
struct NcclUniqueId { char internal[128]; };  // ncclUniqueId (nccl.h: NCCL_UNIQUE_ID_BYTES = 128), passed by value
struct NcclApi {
    void *handle = nullptr;
    int (*GetUniqueId)(NcclUniqueId *) = nullptr;
    int (*CommInitRank)(void **, int, NcclUniqueId, int) = nullptr;
    int (*CommInitAll)(void **, int, const int *) = nullptr;
    int (*CommDestroy)(void *) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, void *, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    std::string why;
    bool ok = false;
};
enum { NCCL_UINT8 = 1, NCCL_INT64 = 4, NCCL_FLOAT32 = 7, NCCL_FLOAT64 = 8, NCCL_SUM = 0 };  // ncclDataType_t / ncclRedOp_t values (nccl.h)
NcclApi &nccl_api() {
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        const char *names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char *n : names) if (!api.handle) api.handle = dlopen(n, RTLD_NOW | RTLD_NOLOAD);
        for (const char *n : names) if (!api.handle) api.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (!api.handle) { api.why = "libnccl.so.2 not found (dlopen)"; return; }
        auto sym = [&](const char *n) { void *p = dlsym(api.handle, n); if (!p) api.why = std::string("missing NCCL symbol ") + n; return p; };
        api.GetUniqueId = (decltype(api.GetUniqueId))sym("ncclGetUniqueId");
        api.CommInitRank = (decltype(api.CommInitRank))sym("ncclCommInitRank");
        api.CommInitAll = (decltype(api.CommInitAll))sym("ncclCommInitAll");
        api.CommDestroy = (decltype(api.CommDestroy))sym("ncclCommDestroy");
        api.AllReduce = (decltype(api.AllReduce))sym("ncclAllReduce");
        api.AllGather = (decltype(api.AllGather))sym("ncclAllGather");
        api.GetErrorString = (decltype(api.GetErrorString))sym("ncclGetErrorString");
        api.ok = api.why.empty();
    });
    return api;
}

// ping-pong buffers of the radix sort
template <typename K>
struct SortScratch {
    K *kb[2] = {nullptr, nullptr};
    uint32_t *vb[2] = {nullptr, nullptr};
    uint32_t *counts = nullptr;
    size_t cap = 0;
};

}  // namespace

struct cgrt_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    std::string err = "";
    cgrt_config cfg;
    PassParams P;
    std::vector<HostTexture> textures;
    std::vector<HostObject> objects;
    bool committed = false;
    bool bvh_f32 = true;  // every tree within CGRT_F32_BOUND (set by cgrt_commit_scene): the traversal without fp64 box arithmetic
    SceneDev S;
    BvhBuild bvh_src[CGRT_MAX_BVH];
    int obj_bvh[CGRT_MAX_OBJECTS];
    std::vector<void *> allocs;
    std::vector<std::pair<void *, size_t>> big_allocs;  // arena blocks (see dalloc)
    // CGRT_GUARD=1 (dev): every device buffer is allocated with CGRT_GUARD_BYTES of 0xA5 on both sides; the fences are verified when
    // the buffer is released and by cgrt_check_guards. user pointer -> (base pointer, user bytes)
    std::unordered_map<void *, std::pair<void *, size_t>> guarded;
    uint64_t guard_violations = 0;

    // hitpoints
    double *hp_rec = nullptr;  // raw records (12 doubles each), creation order of the wavefront
    unsigned int hp_cap = 0, hp_count = 0;
    unsigned int *d_hp_count = nullptr;
    bool grid_built = false;
    unsigned int nhp = 0;
    HpArrays A;
    void *acc = nullptr;
    uint32_t *cell_start = nullptr, *pix_start = nullptr, *pix_perm = nullptr;

    // queues
    RayQueue q[2];       // eye pass only: the photon pass keeps its rays in registers
    size_t q_cap[2] = {0, 0};
    unsigned int *d_qcount = nullptr;  // [0],[1]: eye ray queues; [2..7]: suspended-photon queues of the photon pass; [8..13]: work cursors of its 6 trace launches
    // photon pass buffers
    // Deposit tables are double-buffered: the trace kernels of chunk k+1 (stream `tstream`) run while the sort + deposit kernels of
    // chunk k (stream `stream`) drain the other buffer — the latency-bound gather and the fp64-bound tracer share the SMs.
    struct DepBuf {
        char *rec = nullptr;          // deposit table: slots x deposit_rec_bytes(compact)
        size_t rec_bytes = 0;         // bytes of one slot in this table
        uint32_t *keys = nullptr;     // bin per slot (CGRT_KEY_INVALID = empty)
        uint32_t *perm = nullptr;     // cell-grouped order of the valid slots
        uint32_t *hist = nullptr;     // bin counters -> cursors (P.bin_mask + 1 of them in use)
        uint32_t *bsum = nullptr;     // per-4096-bin block totals
        uint32_t *nvalid = nullptr;
        cudaEvent_t traced = nullptr, drained = nullptr;
        bool drained_valid = false;
        size_t cap = 0;               // slots
    } dep[2];
    unsigned int chunk_seq = 0;
    cudaStream_t tstream = nullptr;
    // The per-round tail (all-reduce of the accumulators when a communicator is attached, then round_update_kernel) runs on its own stream:
    // it only has to finish before the NEXT round's sort + deposit, so the next round's trace launches — which never read a radius or an
    // accumulator — run underneath it. `updated` is what every reader of hitpoint state waits for (join_update).
    cudaStream_t ustream = nullptr;
    cudaEvent_t ev_tail = nullptr, ev_updated = nullptr;
    bool update_pending = false;
    void *comm = nullptr;   // ncclComm_t attached by cgrt_set_comm (not owned)
    int comm_world = 1;
    // peer-memory exchange (cgrt_peer_export / cgrt_peer_attach): this rank's shared block = two accumulator buffers (round parity), flag
    // arrays for rounds and for shutdown, an error word; and the mapped blocks of the other ranks
    struct Peer {
        char *block = nullptr;          // own block (cudaMalloc)
        size_t acc_bytes = 0, bytes = 0;
        int rank = -1, world = 0;
        int round = 0, parity = 0;
        bool attached = false;
        char *base[CGRT_MAX_PEERS] = {};    // every rank's block as mapped here (own included)
        bool ipc[CGRT_MAX_PEERS] = {};      // opened with cudaIpcOpenMemHandle (to be closed)
    } peer;
    int sm_count = 148;
    int overlap = 0;  // cgrt_set_overlap: off by default; its measurements are in DESIGN.md section 4
    // resident-grid sizes of the persistent photon kernels (SMs x occupancy), so that static striding leaves no tail of late blocks
    unsigned int grid_first = 592, grid_cont = 592;
    PhotonState *pq[2] = {nullptr, nullptr};
    size_t pq_cap = 0;
    uint32_t *reach = nullptr;        // reach bitmap (cells within 2 cells of a hitpoint), built with the grid
    int cull = 1;
    Counters *d_ctr = nullptr;
    TravCounters *d_tc = nullptr;
    int *d_fxerr = nullptr;  // fixed-point accumulators: FIX_ERR_* bits raised by the deposit and update kernels; stays raised
    uint64_t launches = 0;
    unsigned int deposit_grid = 148 * 8;  // resident deposit blocks: 8 x 256 threads per SM
    int profiling = 0;   // 1: time every photon kernel with events (serialises host and device at the end of each pass)
    double ms[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    cudaEvent_t ev[2] = {nullptr, nullptr};
    // photons per trace launch: bounds the deposit table (chunk * max_depth * 104 B) and the two photon queues (chunk * 128 B each).
    // 0 = as many as fit in 60 % of the device's memory, at most 128 Mi: the deposit kernel amortises a cell's candidate list over the
    // hits of one chunk that fall into it, so at 4096^2 (16x the cells of 1024^2) a 16 Mi chunk left ~2 hits per cell group and the
    // kernel re-read 88 GB of candidates per chunk
    size_t photon_chunk = 0;
    // per-photon update (update_mode 0): r2 after n accepted photons, the reference's recurrence r2 *= (n a + a) / (n a + 1) run on the host
    double *r2tab = nullptr;
    int r2cap = 0;
    int *d_maxcnt = nullptr;
    size_t auto_chunk = 0;
    int counting = 0;  // 1: photon trace kernels also count BVH node visits / triangle tests (roofline accounting)
    // stochastic PPM (cgrt_set_sppm): per-pixel statistics, and the visible-point count the per-round buffers are sized for. Every
    // round rebuilds the grid; sizing its buffers from this capacity (grown with headroom, never shrunk) instead of the round's exact
    // count makes every round ask the pool and the arena for the same sizes, so device memory reaches a steady state.
    int sppm = CGRT_SPPM_OFF;
    uint32_t sppm_round = 0;    // the round whose camera stream the eye pass draws
    double *pix_tau = nullptr;  // [W*H][4] tau (+pad)
    double *pix_r2 = nullptr;   // [W*H]
    int *pix_cnt = nullptr;     // [W*H]
    size_t sppm_cap = 0;
    bool sppm_traced = false;   // cgrt_sppm_eye_pass has traced this round's visible points and cgrt_build_grid has not run yet
    size_t gather_cap = 0;      // SPPM: records per rank the all-gather's buffers are sized for (grown with headroom, never shrunk)
};

namespace {

#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e__ = (call);                                                                        \
        if (e__ != cudaSuccess) {                                                                        \
            char b__[512];                                                                               \
            snprintf(b__, sizeof b__, "%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            ctx->err = b__;                                                                              \
            return CGRT_ERR_CUDA;                                                                        \
        }                                                                                                \
    } while (0)
#define CKS(expr)                \
    do {                         \
        int s__ = (expr);        \
        if (s__ != 0) return s__; \
    } while (0)
#define FAIL(code, msg)   \
    do {                  \
        ctx->err = (msg); \
        return (code);    \
    } while (0)

// Everything that reads or writes hitpoint state on the main stream first waits for the pending per-round update (stream-side wait, the
// host is not blocked).
int join_update(cgrt_ctx *ctx) {
    if (ctx->update_pending) {
        CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_updated, 0));
        ctx->update_pending = false;
    }
    return 0;
}

// Small and medium buffers come from the stream-ordered pool (no device-wide sync, memory is reused); buffers of CGRT_ARENA_MIN bytes
// or more (ray queues, hitpoint records) come from the process-wide arena of plain cudaMalloc blocks: growing the pool by gigabytes
// was measured at 150-400 ms per context, a cudaMalloc of the same size at a few ms, and a parked block costs nothing.
#define CGRT_ARENA_MIN ((size_t)32 << 20)
#define CGRT_GUARD_BYTES ((size_t)4096)
bool guard_mode() {
    static const bool on = [] { const char *e = getenv("CGRT_GUARD"); return e && atoi(e) != 0; }();
    return on;
}
// fences of one guarded buffer -> number of damaged bytes (synchronises the context's streams)
uint64_t guard_damage(cgrt_ctx *ctx, void *base, size_t bytes) {
    std::vector<unsigned char> h(2 * CGRT_GUARD_BYTES);
    if (ctx->tstream) cudaStreamSynchronize(ctx->tstream);
    if (ctx->ustream) cudaStreamSynchronize(ctx->ustream);
    cudaStreamSynchronize(ctx->stream);
    cudaMemcpy(h.data(), base, CGRT_GUARD_BYTES, cudaMemcpyDeviceToHost);
    cudaMemcpy(h.data() + CGRT_GUARD_BYTES, (char *)base + CGRT_GUARD_BYTES + bytes, CGRT_GUARD_BYTES, cudaMemcpyDeviceToHost);
    uint64_t bad = 0;
    for (unsigned char c : h) bad += c != 0xA5;
    return bad;
}
// user pointer of a freshly allocated base block of bytes + 2 fences
void *guard_wrap(cgrt_ctx *ctx, void *base, size_t bytes) {
    cudaMemsetAsync(base, 0xA5, CGRT_GUARD_BYTES, ctx->stream);
    cudaMemsetAsync((char *)base + CGRT_GUARD_BYTES + bytes, 0xA5, CGRT_GUARD_BYTES, ctx->stream);
    void *user = (char *)base + CGRT_GUARD_BYTES;
    ctx->guarded[user] = std::make_pair(base, bytes);
    return user;
}
// base pointer of a guarded user pointer about to be released (fences verified); the pointer itself when guard mode is off
void *guard_unwrap(cgrt_ctx *ctx, void *user) {
    auto it = ctx->guarded.find(user);
    if (it == ctx->guarded.end()) return user;
    void *base = it->second.first;
    ctx->guard_violations += guard_damage(ctx, base, it->second.second);
    ctx->guarded.erase(it);
    return base;
}
// the photon pass's tables: always arena blocks
void *big_take(cgrt_ctx *ctx, size_t bytes) {
    if (!guard_mode()) return arena_take(ctx->device, bytes);
    void *base = arena_take(ctx->device, bytes + 2 * CGRT_GUARD_BYTES);
    return base ? guard_wrap(ctx, base, bytes) : nullptr;
}
void big_give(cgrt_ctx *ctx, size_t bytes, void *p) {
    if (!p) return;
    const bool g = ctx->guarded.count(p) != 0;
    arena_give(ctx->device, bytes + (g ? 2 * CGRT_GUARD_BYTES : 0), guard_unwrap(ctx, p));
}
template <typename T>
int dalloc(cgrt_ctx *ctx, T **p, size_t n) {
    *p = nullptr;
    if (n == 0) n = 1;
    const size_t user_bytes = (n * sizeof(T) + 15) & ~(size_t)15;
    const size_t bytes = user_bytes + (guard_mode() ? 2 * CGRT_GUARD_BYTES : 0);
    void *q = nullptr;
    if (bytes >= CGRT_ARENA_MIN) {
        q = arena_take(ctx->device, bytes);
        if (!q) FAIL(CGRT_ERR_CUDA, "out of device memory");
        ctx->big_allocs.push_back(std::make_pair(q, bytes));
    } else {
        CK(cudaMallocAsync(&q, bytes, ctx->stream));
        ctx->allocs.push_back(q);
    }
    *p = (T *)(guard_mode() ? guard_wrap(ctx, q, user_bytes) : q);
    return 0;
}
int dfree(cgrt_ctx *ctx, void *p) {
    if (!p) return 0;
    p = guard_unwrap(ctx, p);
    for (size_t i = 0; i < ctx->big_allocs.size(); i++)
        if (ctx->big_allocs[i].first == p) {
            CK(cudaStreamSynchronize(ctx->stream));  // the next owner may be another context on another stream
            arena_give(ctx->device, ctx->big_allocs[i].second, p);
            ctx->big_allocs[i] = ctx->big_allocs.back();
            ctx->big_allocs.pop_back();
            return 0;
        }
    for (size_t i = 0; i < ctx->allocs.size(); i++)
        if (ctx->allocs[i] == p) {
            ctx->allocs[i] = ctx->allocs.back();
            ctx->allocs.pop_back();
            break;
        }
    CK(cudaFreeAsync(p, ctx->stream));
    return 0;
}
inline unsigned int nblk(size_t n, unsigned int b) { return (unsigned int)((n + b - 1) / b); }

struct PhaseTimer {
    cgrt_ctx *ctx;
    int slot;
    bool on;
    PhaseTimer(cgrt_ctx *c, int s, bool enabled = true) : ctx(c), slot(s), on(enabled) {
        if (on) cudaEventRecord(ctx->ev[0], ctx->stream);
    }
    void stop() {
        if (!on) return;
        cudaEventRecord(ctx->ev[1], ctx->stream);
        cudaEventSynchronize(ctx->ev[1]);
        float t = 0;
        cudaEventElapsedTime(&t, ctx->ev[0], ctx->ev[1]);
        ctx->ms[slot] += t;
    }
};

// ---- radix sort driver: keys (dev) -> sorted keys + permutation (dev). nbits rounded up to whole 8-bit digits.
// `scratch` (optional) supplies the ping-pong buffers so that a hot caller (the per-round deposit sort) allocates nothing.
template <typename K>
int sort_scratch_reserve(cgrt_ctx *ctx, SortScratch<K> &sc, size_t n) {
    if (n <= sc.cap) return 0;
    if (sc.cap) { CKS(dfree(ctx, sc.kb[0])); CKS(dfree(ctx, sc.kb[1])); CKS(dfree(ctx, sc.vb[0])); CKS(dfree(ctx, sc.vb[1])); CKS(dfree(ctx, sc.counts)); }
    size_t ntiles = (n + RS_TILE - 1) / RS_TILE;
    CKS(dalloc(ctx, &sc.kb[0], n)); CKS(dalloc(ctx, &sc.kb[1], n)); CKS(dalloc(ctx, &sc.vb[0], n)); CKS(dalloc(ctx, &sc.vb[1], n));
    CKS(dalloc(ctx, &sc.counts, (size_t)256 * ntiles));
    sc.cap = n;
    return 0;
}
template <typename K>
int sort_scratch_release(cgrt_ctx *ctx, SortScratch<K> &sc) {
    if (!sc.cap) return 0;
    CKS(dfree(ctx, sc.kb[0])); CKS(dfree(ctx, sc.kb[1])); CKS(dfree(ctx, sc.vb[0])); CKS(dfree(ctx, sc.vb[1])); CKS(dfree(ctx, sc.counts));
    sc = SortScratch<K>();
    return 0;
}
// Asynchronous on the ctx stream. Results are left in the scratch buffers: *keys_sorted / *perm point at them.
template <typename K>
int radix_sort_async(cgrt_ctx *ctx, SortScratch<K> &sc, size_t n, const K *keys_in, int nbits, const K **keys_sorted, const uint32_t **perm) {
    if (n >= (1ull << 32)) FAIL(CGRT_ERR_CAPACITY, "radix sort: more than 2^32 keys");
    CKS(sort_scratch_reserve(ctx, sc, n));
    int passes = (nbits + 7) / 8;
    if (passes < 1) passes = 1;
    int ntiles = (int)((n + RS_TILE - 1) / RS_TILE);
    const K *src_k = keys_in;
    const uint32_t *src_v = nullptr;
    int cur = 0;
    for (int p = 0; p < passes; p++) {
        int shift = 8 * p;
        rs_hist_kernel<K><<<ntiles, RS_THREADS, 0, ctx->stream>>>(src_k, (int64_t)n, shift, sc.counts, ntiles);
        rs_scan_kernel<<<1, 1024, 0, ctx->stream>>>(sc.counts, (int64_t)256 * ntiles);
        rs_scatter_kernel<K><<<ntiles, RS_THREADS, 0, ctx->stream>>>(src_k, src_v, sc.kb[cur], sc.vb[cur], (int64_t)n, shift, sc.counts, ntiles, p == 0);
        ctx->launches += 3;
        src_k = sc.kb[cur];
        src_v = sc.vb[cur];
        cur ^= 1;
    }
    CK(cudaGetLastError());
    *keys_sorted = src_k;
    *perm = src_v;
    return 0;
}
// reserve > n: the scratch is allocated for `reserve` keys (stable allocation sizes from call to call)
int radix_sort_dev(cgrt_ctx *ctx, size_t n, const uint64_t *keys_in, int nbits, uint64_t *keys_out, uint32_t *perm_out, size_t reserve = 0) {
    if (n == 0) return 0;
    SortScratch<uint64_t> sc;
    if (reserve > n) CKS(sort_scratch_reserve(ctx, sc, reserve));
    const uint64_t *ks;
    const uint32_t *pm;
    CKS(radix_sort_async(ctx, sc, n, keys_in, nbits, &ks, &pm));
    CK(cudaMemcpyAsync(keys_out, ks, n * sizeof(uint64_t), cudaMemcpyDeviceToDevice, ctx->stream));
    CK(cudaMemcpyAsync(perm_out, pm, n * sizeof(uint32_t), cudaMemcpyDeviceToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return sort_scratch_release(ctx, sc);
}

// ---- LBVH build over n triangles already on the device (tri9, original order)
int build_bvh(cgrt_ctx *ctx, double *tri9_dev, int n, double orient_sign, int slot) {
    BvhDev &B = ctx->S.bvh[slot];
    memset(&B, 0, sizeof B);
    B.ntris = n;
    B.orient_sign = orient_sign;
    B.root_is_leaf = (n == 1);
    ctx->bvh_src[slot].tri9 = tri9_dev;
    ctx->bvh_src[slot].ntris = n;
    if (n <= 0) FAIL(CGRT_ERR_INVALID, "mesh with no triangles");
    const unsigned int T = 256;
    uint32_t *bounds;
    uint64_t *keys, *keys_sorted;
    uint32_t *perm;
    CKS(dalloc(ctx, &bounds, 6));
    CKS(dalloc(ctx, &keys, (size_t)n));
    CKS(dalloc(ctx, &keys_sorted, (size_t)n));
    CKS(dalloc(ctx, &perm, (size_t)n));
    uint32_t init[6] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u};
    CK(cudaMemcpyAsync(bounds, init, sizeof init, cudaMemcpyHostToDevice, ctx->stream));
    lbvh_bounds_kernel<<<nblk(n, T), T, 0, ctx->stream>>>(tri9_dev, n, bounds);
    lbvh_morton_kernel<<<nblk(n, T), T, 0, ctx->stream>>>(tri9_dev, n, bounds, keys);
    ctx->launches += 2;
    CKS(radix_sort_dev(ctx, (size_t)n, keys, 30, keys_sorted, perm));

    TriRec *tris;
    int *tri_id;
    float *box;
    int *left, *right, *parent;
    unsigned int *flags;
    int ninternal = n > 1 ? n - 1 : 0;
    CKS(dalloc(ctx, &tris, (size_t)n));
    CKS(dalloc(ctx, &tri_id, (size_t)n));
    CKS(dalloc(ctx, &box, (size_t)(2 * n) * 6));
    CKS(dalloc(ctx, &left, (size_t)n));
    CKS(dalloc(ctx, &right, (size_t)n));
    CKS(dalloc(ctx, &parent, (size_t)(2 * n)));
    CKS(dalloc(ctx, &flags, (size_t)n));
    CK(cudaMemsetAsync(flags, 0, sizeof(unsigned int) * n, ctx->stream));
    CK(cudaMemsetAsync(parent, 0xff, sizeof(int) * 2 * n, ctx->stream));
    lbvh_leaves_kernel<<<nblk(n, T), T, 0, ctx->stream>>>(tri9_dev, perm, n, tris, tri_id, box);
    ctx->launches++;
    if (ninternal > 0) {
        lbvh_hierarchy_kernel<<<nblk(ninternal, T), T, 0, ctx->stream>>>(keys_sorted, n, left, right, parent);
        lbvh_refit_kernel<<<nblk(n, T), T, 0, ctx->stream>>>(n, left, right, parent, box, flags);
        ctx->launches += 2;
    }
    // ---- 4-wide nodes: collapse level by level (the host only reads one counter per level)
    BvhNode4 *nodes4;
    int *wqueue, *wcounter;
    CKS(dalloc(ctx, &nodes4, (size_t)(ninternal > 0 ? ninternal : 1)));
    CKS(dalloc(ctx, &wqueue, (size_t)(ninternal > 0 ? ninternal : 1)));
    CKS(dalloc(ctx, &wcounter, 1));
    int wide_levels = 0;
    if (ninternal > 0) {
        int one = 1, zero = 0;
        CK(cudaMemcpyAsync(wqueue, &zero, sizeof zero, cudaMemcpyHostToDevice, ctx->stream));  // wide node 0 = binary root 0
        CK(cudaMemcpyAsync(wcounter, &one, sizeof one, cudaMemcpyHostToDevice, ctx->stream));
        int begin = 0, end = 1;
        while (begin < end) {
            lbvh_collapse_kernel<<<nblk(end - begin, T), T, 0, ctx->stream>>>(n, begin, end, left, right, box, wqueue, wcounter, nodes4);
            ctx->launches++;
            int total = 0;
            CK(cudaMemcpyAsync(&total, wcounter, sizeof total, cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            begin = end; end = total;
            wide_levels++;
        }
    }
    // traversal stack: at most three pushes per wide level (CGRT_BVH_STACK entries)
    if (3 * wide_levels + 4 > CGRT_BVH_STACK) FAIL(CGRT_ERR_CAPACITY, "mesh hierarchy too deep for the traversal stack");
    float root[6];  // box 0 is the root (the only leaf when n == 1)
    CK(cudaMemcpyAsync(root, box, sizeof root, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaGetLastError());
    B.f32_ok = 1;
    for (int a = 0; a < 3; a++) {
        B.root_lo[a] = root[a]; B.root_hi[a] = root[3 + a];
        if (!(std::fabs(root[a]) <= CGRT_F32_BOUND && std::fabs(root[3 + a]) <= CGRT_F32_BOUND)) B.f32_ok = 0;
    }
    B.nodes4 = nodes4;
    B.tris = tris;
    B.tri_id = tri_id;
    CKS(dfree(ctx, bounds)); CKS(dfree(ctx, keys)); CKS(dfree(ctx, keys_sorted)); CKS(dfree(ctx, perm));
    CKS(dfree(ctx, wqueue)); CKS(dfree(ctx, wcounter));
    CKS(dfree(ctx, box)); CKS(dfree(ctx, left)); CKS(dfree(ctx, right)); CKS(dfree(ctx, parent)); CKS(dfree(ctx, flags));
    return 0;
}

// Per-mesh orientation sign (SURVEY Q8): sum of pa . (pb x pc) in triangle order; >= 0 -> winding normals point outward.
double orientation_sign(const double *tri9, size_t n) {
    double vol = 0.0;
    for (size_t i = 0; i < n; i++) {
        const double *t = tri9 + 9 * i;
        d3 pa = mk(t[0], t[1], t[2]), pb = mk(t[3], t[4], t[5]), pc = mk(t[6], t[7], t[8]);
        vol += dot(pa, cross(pb, pc));
    }
    return (vol >= 0.0) ? 1.0 : -1.0;
}

int alloc_queue(cgrt_ctx *ctx, RayQueue &q, size_t cap, bool with_aux) {
    double *base;
    CKS(dalloc(ctx, &base, cap * 9));
    q.ox = base; q.oy = base + cap; q.oz = base + 2 * cap;
    q.dx = base + 3 * cap; q.dy = base + 4 * cap; q.dz = base + 5 * cap;
    q.wx = base + 6 * cap; q.wy = base + 7 * cap; q.wz = base + 8 * cap;
    CKS(dalloc(ctx, &q.id, cap));
    q.aux = nullptr;
    if (with_aux) CKS(dalloc(ctx, &q.aux, cap));
    return 0;
}
int free_queue(cgrt_ctx *ctx, RayQueue &q) {
    CKS(dfree(ctx, q.ox)); CKS(dfree(ctx, q.id)); CKS(dfree(ctx, q.aux));
    memset(&q, 0, sizeof q);
    return 0;
}
// Only the OUTPUT queue of a bounce may be (re)allocated: the input queue holds the live rays of the current wavefront.
int ensure_queue(cgrt_ctx *ctx, int which, size_t cap) {
    if (cap <= ctx->q_cap[which]) return 0;
    if (ctx->q_cap[which]) CKS(free_queue(ctx, ctx->q[which]));
    CKS(alloc_queue(ctx, ctx->q[which], cap, true));
    ctx->q_cap[which] = cap;
    return 0;
}
// float or fixed-point accumulators with the per-round update: the 64-byte record (DepositRecC) of the float walk; everything else keeps
// the 96-byte fp64 record
inline bool compact_records(const cgrt_ctx *ctx) { return ctx->cfg.accum_mode != 0 && ctx->cfg.update_mode != 0; }
// bytes of one accumulator lane: fp64 (accum_mode 0), float (1), int64 fixed point (2)
inline size_t acc_elem(const cgrt_ctx *ctx) { return ctx->cfg.accum_mode == 1 ? sizeof(float) : sizeof(double); }
// The fixed-point mode's error word; the streams that write it must have been synchronised.
int check_fixed(cgrt_ctx *ctx) {
    if (ctx->cfg.accum_mode != 2) return 0;
    int e = 0;
    CK(cudaMemcpy(&e, ctx->d_fxerr, sizeof e, cudaMemcpyDeviceToHost));
    if (e & FIX_ERR_VALUE)
        FAIL(CGRT_ERR_CAPACITY, "fixed-point accumulators: a deposit value f * flux / pi above 2^16 (or not a number); the flux sums are invalid");
    if (e & FIX_ERR_COUNT)
        FAIL(CGRT_ERR_CAPACITY, "fixed-point accumulators: more than 2^24 photons accepted by one hitpoint (SPPM: one pixel) in one round; "
                                "the flux sums are invalid");
    return 0;
}
int ensure_photon_buffers(cgrt_ctx *ctx, size_t photons, size_t slots) {
    const size_t rb = deposit_rec_bytes(compact_records(ctx));
    bool fresh = false;
    const int nbuf = ctx->overlap ? 2 : 1;  // the second deposit table only exists while the two-stream pipeline is on
    for (int bi = 0; bi < nbuf; bi++) {
        auto &b = ctx->dep[bi];
        if (slots <= b.cap && b.rec_bytes == rb) continue;
        CK(cudaStreamSynchronize(ctx->tstream));
        CK(cudaStreamSynchronize(ctx->stream));
        if (b.cap) {
            big_give(ctx, b.cap * b.rec_bytes, b.rec);
            big_give(ctx, b.cap * sizeof(uint32_t), b.keys);
            big_give(ctx, b.cap * sizeof(uint32_t), b.perm);
        }
        b.cap = 0; b.rec = nullptr; b.keys = nullptr; b.perm = nullptr;  // nothing dangles if a block below cannot be had
        char *nrec = (char *)big_take(ctx, slots * rb);
        uint32_t *nkeys = (uint32_t *)big_take(ctx, slots * sizeof(uint32_t));
        uint32_t *nperm = (uint32_t *)big_take(ctx, slots * sizeof(uint32_t));
        if (!nrec || !nkeys || !nperm) {
            big_give(ctx, slots * rb, nrec);
            big_give(ctx, slots * sizeof(uint32_t), nkeys);
            big_give(ctx, slots * sizeof(uint32_t), nperm);
            FAIL(CGRT_ERR_CUDA, "out of device memory for the deposit tables");
        }
        b.rec = nrec; b.keys = nkeys; b.perm = nperm;
        b.cap = slots; b.rec_bytes = rb;
        b.drained_valid = false;
        fresh = true;
    }
    photons += CGRT_QHOLE_MARGIN;  // room for the slots warps reserve and do not use
    if (photons > ctx->pq_cap) {
        CK(cudaStreamSynchronize(ctx->tstream));
        for (int k = 0; k < 2; k++) {
            if (ctx->pq_cap) big_give(ctx, ctx->pq_cap * sizeof(PhotonState), ctx->pq[k]);
            ctx->pq[k] = nullptr;
        }
        ctx->pq_cap = 0;
        for (int k = 0; k < 2; k++) {
            ctx->pq[k] = (PhotonState *)big_take(ctx, photons * sizeof(PhotonState));
            if (!ctx->pq[k]) {
                if (k == 1) { big_give(ctx, photons * sizeof(PhotonState), ctx->pq[0]); ctx->pq[0] = nullptr; }
                FAIL(CGRT_ERR_CUDA, "out of device memory for the photon queues");
            }
        }
        ctx->pq_cap = photons;
        fresh = true;
    }
    if (!ctx->dep[0].hist) {
        for (auto &b : ctx->dep) {
            CKS(dalloc(ctx, &b.hist, (size_t)1 << CGRT_BIN_BITS_MAX));
            CKS(dalloc(ctx, &b.bsum, ((size_t)1 << CGRT_BIN_BITS_MAX) / (CGRT_SCAN_BLOCK * CGRT_SCAN_ITEMS)));
            CKS(dalloc(ctx, &b.nvalid, 2));
            CK(cudaEventCreateWithFlags(&b.traced, cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&b.drained, cudaEventDisableTiming));
        }
        fresh = true;
    }
    if (fresh) CK(cudaStreamSynchronize(ctx->stream));  // the pool allocations are ordered on `stream`; `tstream` uses them too
    return 0;
}

int ensure_hp_capacity(cgrt_ctx *ctx, size_t need) {
    if (need <= ctx->hp_cap) return 0;
    size_t cap = ctx->hp_cap ? ctx->hp_cap : 1024;
    while (cap < need) cap = cap + cap / 2 + 1024;
    if (cap >= (1ull << 32)) FAIL(CGRT_ERR_CAPACITY, "more than 2^32 hitpoints");
    double *nrec;
    CKS(dalloc(ctx, &nrec, cap * CGRT_HP_RECORD_DOUBLES));
    if (ctx->hp_rec) {
        CK(cudaMemcpyAsync(nrec, ctx->hp_rec, (size_t)ctx->hp_count * CGRT_HP_RECORD_DOUBLES * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        CKS(dfree(ctx, ctx->hp_rec));
    }
    ctx->hp_rec = nrec;
    ctx->hp_cap = (unsigned int)cap;
    return 0;
}

void derive_params(cgrt_ctx *ctx) {
    const cgrt_config &c = ctx->cfg;
    PassParams &P = ctx->P;
    P.width = c.width; P.height = c.height; P.max_depth = c.max_depth; P.samples = c.num_of_samples; P.use_dof = c.use_dof;
    P.hashsize = (uint32_t)c.hashsize;
    P.bin_mask = (1u << (c.hashsize > (4 << 20) ? CGRT_BIN_BITS_MAX : CGRT_BIN_BITS_MIN)) - 1u;
    // Hashtable(hashsize, r): hash.h:22-30 with r = 200.0/height (main.cpp:183)
    double r = 200.0 / c.height;
    int cells = (int)(std::ceil(70.0 / r));
    P.celllength = 70.0 / cells;
    P.inv_celllength = 1.0 / P.celllength;
    P.r2_init = r * r;
    P.alpha = c.alpha; P.focus_plane = c.focus_plane; P.lens_radius = c.lens_radius;
    for (int i = 0; i < 3; i++) { P.cam[i] = c.camorg[i]; P.light[i] = c.lightorg[i]; }
    P.seed = c.seed;
}

}  // namespace

namespace {
template <typename T>
int upload(cgrt_ctx *ctx, T **d, const T *h, size_t n) {
    CKS(dalloc(ctx, d, n));
    CK(cudaMemcpyAsync(*d, h, n * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
    return 0;
}
template <typename T>
int download_free(cgrt_ctx *ctx, T *h, T *d, size_t n) {
    if (h) CK(cudaMemcpyAsync(h, d, n * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return dfree(ctx, d);
}
}  // namespace

// ---- peer-memory exchange -------------------------------------------------------------------------------------------------------------
namespace {
struct PeerBlob {  // CGRT_PEER_HANDLE_BYTES = 128
    cudaIpcMemHandle_t handle;  // 64 bytes
    uint64_t pid, ptr, bytes, acc_bytes;
    int32_t device, nhp, accum_mode, magic;
    char pad[128 - 64 - 4 * 8 - 4 * 4];
};
static_assert(sizeof(PeerBlob) == 128, "peer handle blob is 128 bytes");
inline size_t peer_flags_off(const cgrt_ctx::Peer &p) { return 2 * p.acc_bytes; }                                   // int[CGRT_MAX_PEERS]: rounds
inline size_t peer_done_off(const cgrt_ctx::Peer &p) { return 2 * p.acc_bytes + CGRT_MAX_PEERS * sizeof(int); }      // int[CGRT_MAX_PEERS]: shutdown
inline size_t peer_err_off(const cgrt_ctx::Peer &p) { return 2 * p.acc_bytes + 2 * CGRT_MAX_PEERS * sizeof(int); }   // int
const unsigned long long PEER_TIMEOUT_NS = 20ull * 1000 * 1000 * 1000;

// Shutdown handshake + unmapping (cgrt_destroy): a rank may only free its block when no peer can still be reading it.
void peer_release(cgrt_ctx *ctx) {
    cgrt_ctx::Peer &P = ctx->peer;
    if (!P.block) return;
    cudaSetDevice(ctx->device);
    if (ctx->ustream) cudaStreamSynchronize(ctx->ustream);
    cudaStreamSynchronize(ctx->stream);
    if (P.attached) {
        PeerPtrs done;
        for (int g = 0; g < CGRT_MAX_PEERS; g++) done.p[g] = g < P.world ? P.base[g] + peer_done_off(P) : nullptr;
        peer_signal_kernel<<<1, 32, 0, ctx->stream>>>(done, P.rank, P.world, 1);
        peer_wait_kernel<<<1, 32, 0, ctx->stream>>>(reinterpret_cast<const int *>(P.block + peer_done_off(P)), P.world, 1, PEER_TIMEOUT_NS,
                                                  reinterpret_cast<int *>(P.block + peer_err_off(P)));
        cudaStreamSynchronize(ctx->stream);
        for (int g = 0; g < P.world; g++)
            if (P.ipc[g]) cudaIpcCloseMemHandle(P.base[g]);
    }
    cudaFree(P.block);
    P = cgrt_ctx::Peer();
}
}  // namespace

// =================================================================================================================
extern "C" {

int cgrt_version(void) { return 103; }

void cgrt_default_config(cgrt_config *c) {
    memset(c, 0, sizeof *c);
    c->width = 1024; c->height = 768; c->max_depth = 5; c->num_of_samples = 1; c->use_dof = 0; c->hashsize = 1000001;
    c->accum_mode = 0;
    c->update_mode = 1;
    c->alpha = 0.7; c->focus_plane = 20.0; c->lens_radius = 1.5;
    c->lightorg[0] = 0; c->lightorg[1] = 19.999; c->lightorg[2] = 20;
    c->camorg[0] = 0; c->camorg[1] = 0; c->camorg[2] = -10;
    c->seed = 20261018ull;
}

int cgrt_create(int device, cgrt_ctx **out) {
    if (!out) return CGRT_ERR_INVALID;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return CGRT_ERR_NO_DEVICE;
    if (cudaSetDevice(device) != cudaSuccess) return CGRT_ERR_NO_DEVICE;
    cgrt_ctx *ctx = new cgrt_ctx();
    ctx->device = device;
    {
        int sms = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && sms > 0) {
            ctx->sm_count = sms;
            ctx->deposit_grid = (unsigned int)sms * 8u;
        }
    }
    {
        int sms = 148, nb = 0;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
        auto occ = [&](const void *k) { return (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k, CGRT_PHOTON_BLOCK, 0) == cudaSuccess && nb > 0) ? (unsigned int)(nb * sms) : 592u; };
        ctx->grid_first = occ((const void *)photon_trace_kernel<true>);
        ctx->grid_cont = occ((const void *)photon_trace_kernel<false>);
        if (const char *e = getenv("CGRT_PHOTON_CHUNK")) { long long c = atoll(e); if (c > 0) ctx->photon_chunk = (size_t)c; }  // tests: force multi-chunk passes
        cudaGetLastError();
    }
    cgrt_default_config(&ctx->cfg);
    derive_params(ctx);
    memset(&ctx->S, 0, sizeof ctx->S);
    memset(&ctx->A, 0, sizeof ctx->A);
    memset(ctx->q, 0, sizeof ctx->q);
    {   // keep freed blocks in the device's default pool instead of returning them to the OS at every synchronize
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            uint64_t keep = UINT64_MAX;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
    }
    // (the side stream of the round's tail at the highest stream priority was measured on 8 GPUs: c2 8.06 vs 5.17 ms per round with the
    // peer exchange — default priority it is)
    if (cudaStreamCreateWithFlags(&ctx->tstream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ctx->ustream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_tail, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_updated, cudaEventDisableTiming) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess || cudaEventCreate(&ctx->ev[0]) != cudaSuccess ||
        cudaEventCreate(&ctx->ev[1]) != cudaSuccess) {
        delete ctx;
        return CGRT_ERR_CUDA;
    }
    if (dalloc(ctx, &ctx->d_hp_count, 1) || dalloc(ctx, &ctx->d_qcount, 16) || dalloc(ctx, &ctx->d_ctr, 1) || dalloc(ctx, &ctx->d_tc, 1) ||
        dalloc(ctx, &ctx->d_fxerr, 1)) {
        delete ctx;
        return CGRT_ERR_CUDA;
    }
    cudaMemsetAsync(ctx->d_hp_count, 0, sizeof(unsigned int), ctx->stream);
    cudaMemsetAsync(ctx->d_qcount, 0, 16 * sizeof(unsigned int), ctx->stream);
    cudaMemsetAsync(ctx->d_ctr, 0, sizeof(Counters), ctx->stream);
    cudaMemsetAsync(ctx->d_tc, 0, sizeof(TravCounters), ctx->stream);
    cudaMemsetAsync(ctx->d_fxerr, 0, sizeof(int), ctx->stream);
    cudaStreamSynchronize(ctx->stream);
    *out = ctx;
    return CGRT_OK;
}

int cgrt_destroy(cgrt_ctx *ctx) {
    if (!ctx) return CGRT_OK;
    cudaSetDevice(ctx->device);
    if (ctx->tstream) cudaStreamSynchronize(ctx->tstream);
    if (ctx->ustream) cudaStreamSynchronize(ctx->ustream);
    cudaStreamSynchronize(ctx->stream);
    peer_release(ctx);  // shutdown handshake with the other ranks, unmap their blocks, free ours
    for (auto &b : ctx->dep) {
        if (b.traced) cudaEventDestroy(b.traced);
        if (b.drained) cudaEventDestroy(b.drained);
        if (b.cap) {
            big_give(ctx, b.cap * b.rec_bytes, b.rec);
            big_give(ctx, b.cap * sizeof(uint32_t), b.keys);
            big_give(ctx, b.cap * sizeof(uint32_t), b.perm);
        }
    }
    for (int k = 0; k < 2; k++) big_give(ctx, ctx->pq_cap * sizeof(PhotonState), ctx->pq[k]);
    if (!ctx->guarded.empty()) {
        uint64_t bad = ctx->guard_violations;
        for (auto &g : ctx->guarded) bad += guard_damage(ctx, g.second.first, g.second.second);
        if (bad) fprintf(stderr, "cgrt: CGRT_GUARD found %llu damaged fence bytes in this context\n", (unsigned long long)bad);
    }
    for (auto &b : ctx->big_allocs) arena_give(ctx->device, b.second, b.first);
    for (void *p : ctx->allocs) cudaFreeAsync(p, ctx->stream);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->ev[0]) cudaEventDestroy(ctx->ev[0]);
    if (ctx->ev[1]) cudaEventDestroy(ctx->ev[1]);
    if (ctx->ev_tail) cudaEventDestroy(ctx->ev_tail);
    if (ctx->ev_updated) cudaEventDestroy(ctx->ev_updated);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->tstream) cudaStreamDestroy(ctx->tstream);
    if (ctx->ustream) cudaStreamDestroy(ctx->ustream);
    delete ctx;
    return CGRT_OK;
}

const char *cgrt_last_error(const cgrt_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int cgrt_set_config(cgrt_ctx *ctx, const cgrt_config *cfg) {
    if (!ctx || !cfg) return CGRT_ERR_INVALID;
    if (cfg->width <= 0 || cfg->height <= 0 || cfg->hashsize <= 0 || cfg->num_of_samples <= 0 || cfg->max_depth <= 0)
        FAIL(CGRT_ERR_INVALID, "config: non-positive size");
    if ((uint64_t)cfg->width * cfg->height * cfg->num_of_samples >= (1ull << 28))
        FAIL(CGRT_ERR_CAPACITY, "config: width*height*samples must be < 2^28 (creation sequence is 32 bits)");
    if (cfg->max_depth > 5) FAIL(CGRT_ERR_CAPACITY, "config: max_depth > 5 needs more than 4 DFS bits");
    if (ctx->hp_count) FAIL(CGRT_ERR_INVALID, "config cannot change after the eye pass");
    if (ctx->sppm) FAIL(CGRT_ERR_INVALID, "config cannot change while SPPM is on (the pixel statistics are sized and seeded from it)");
    if (cfg->update_mode != 0 && cfg->update_mode != 1) FAIL(CGRT_ERR_INVALID, "config: update_mode must be 0 (per photon) or 1 (per round)");
    if (cfg->accum_mode < 0 || cfg->accum_mode > 2) FAIL(CGRT_ERR_INVALID, "config: accum_mode must be 0 (fp64), 1 (float) or 2 (fixed point)");
    if (cfg->update_mode == 0 && ctx->comm) FAIL(CGRT_ERR_INVALID, "config: the per-photon update is not shard-invariant (one GPU only)");
    ctx->cfg = *cfg;
    if (cfg->update_mode == 0) ctx->cfg.accum_mode = 0;  // per-photon update: fp64 sums S = sum c / r2_old in the accumulator buffer
    derive_params(ctx);
    return CGRT_OK;
}
int cgrt_get_stream(cgrt_ctx *ctx, void **stream) {
    if (!ctx || !stream) return CGRT_ERR_INVALID;
    *stream = (void *)ctx->stream;
    return CGRT_OK;
}
int cgrt_synchronize(cgrt_ctx *ctx) {
    if (!ctx) return CGRT_ERR_INVALID;
    CK(cudaStreamSynchronize(ctx->tstream));
    CKS(join_update(ctx));
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->peer.attached) {  // did a wait for the other ranks give up?
        int perr = 0;
        CK(cudaMemcpy(&perr, ctx->peer.block + peer_err_off(ctx->peer), sizeof perr, cudaMemcpyDeviceToHost));
        if (perr) FAIL(CGRT_ERR_NCCL, "peer exchange: rank " + std::to_string(perr - 1) + " did not publish its round in time");
    }
    return check_fixed(ctx);
}

// ---- scene ---------------------------------------------------------------------------------------------------------
int cgrt_add_texture(cgrt_ctx *ctx, const uint8_t *rgb, int w, int h, const double n[3], const double p[3], double lenx, double leny,
                     int isbump, int *tex_id) {
    if (!ctx || !rgb || w <= 0 || h <= 0) return CGRT_ERR_INVALID;
    if (ctx->committed) FAIL(CGRT_ERR_INVALID, "scene already committed");
    if (ctx->textures.size() >= CGRT_MAX_TEX) FAIL(CGRT_ERR_CAPACITY, "too many textures");
    HostTexture t;
    t.rgb.assign(rgb, rgb + (size_t)w * h * 3);
    t.w = w; t.h = h; t.isbump = isbump != 0; t.lenx = lenx; t.leny = leny;
    for (int i = 0; i < 3; i++) { t.n[i] = n[i]; t.p[i] = p[i]; }
    ctx->textures.push_back(std::move(t));
    if (tex_id) *tex_id = (int)ctx->textures.size() - 1;
    return CGRT_OK;
}
static int add_object(cgrt_ctx *ctx, HostObject &&o, int *obj_id) {
    if (ctx->committed) FAIL(CGRT_ERR_INVALID, "scene already committed");
    if (ctx->objects.size() >= CGRT_MAX_OBJECTS) FAIL(CGRT_ERR_CAPACITY, "too many objects");
    ctx->objects.push_back(std::move(o));
    if (obj_id) *obj_id = (int)ctx->objects.size() - 1;
    return CGRT_OK;
}
int cgrt_add_sphere(cgrt_ctx *ctx, const double c[3], double r, const double col[3], double refl, double transp, int *obj_id) {
    if (!ctx || !c || !col) return CGRT_ERR_INVALID;
    HostObject o{};
    o.kind = OBJ_SPHERE; o.r = r; o.refl = refl; o.transp = transp; o.tex = -1; o.objtype = 0;
    for (int i = 0; i < 3; i++) { o.a[i] = c[i]; o.col[i] = col[i]; }
    return add_object(ctx, std::move(o), obj_id);
}
int cgrt_add_plane(cgrt_ctx *ctx, const double p[3], const double n[3], const double col[3], double refl, double transp, int tex_id, int *obj_id) {
    if (!ctx || !p || !n || !col) return CGRT_ERR_INVALID;
    if (tex_id >= (int)ctx->textures.size()) FAIL(CGRT_ERR_INVALID, "unknown texture id");
    HostObject o{};
    o.kind = OBJ_PLANE; o.refl = refl; o.transp = transp; o.tex = tex_id < 0 ? -1 : tex_id; o.objtype = 0;
    for (int i = 0; i < 3; i++) { o.a[i] = p[i]; o.b[i] = n[i]; o.col[i] = col[i]; }
    return add_object(ctx, std::move(o), obj_id);
}
int cgrt_add_mesh(cgrt_ctx *ctx, const double *tri9, int ntri, const double col[3], double refl, double transp, int objtype, int *obj_id) {
    if (!ctx || !tri9 || ntri <= 0 || !col) return CGRT_ERR_INVALID;
    HostObject o{};
    o.kind = OBJ_MESH; o.refl = refl; o.transp = transp; o.tex = -1; o.objtype = objtype;
    for (int i = 0; i < 3; i++) o.col[i] = col[i];
    o.tri9.assign(tri9, tri9 + (size_t)ntri * 9);
    return add_object(ctx, std::move(o), obj_id);
}
int cgrt_add_bezier(cgrt_ctx *ctx, const double *cp3, int ncp, const double pos[3], const double col[3], double refl, double transp, int *obj_id) {
    if (!ctx || !cp3 || ncp < 2 || ncp > CGRT_MAX_CP || !pos || !col) return CGRT_ERR_INVALID;
    HostObject o{};
    o.kind = OBJ_BEZIER; o.refl = refl; o.transp = transp; o.tex = -1; o.objtype = 0;
    for (int i = 0; i < 3; i++) { o.a[i] = pos[i]; o.col[i] = col[i]; }
    o.cp.assign(cp3, cp3 + (size_t)ncp * 3);
    return add_object(ctx, std::move(o), obj_id);
}

int cgrt_commit_scene(cgrt_ctx *ctx) {
    if (!ctx) return CGRT_ERR_INVALID;
    if (ctx->committed) FAIL(CGRT_ERR_INVALID, "scene already committed");
    CK(cudaSetDevice(ctx->device));
    SceneDev &S = ctx->S;
    memset(&S, 0, sizeof S);
    std::vector<double *> heights(ctx->textures.size(), nullptr);
    // textures (K5) + height tables (texture.h:27-37; exp() on the host so the table is bit-identical to the reference's)
    for (size_t t = 0; t < ctx->textures.size(); t++) {
        const HostTexture &ht = ctx->textures[t];
        size_t nt = (size_t)ht.w * ht.h;
        uint8_t *raw;
        uchar4 *tex;
        CKS(dalloc(ctx, &raw, nt * 3));
        CKS(dalloc(ctx, &tex, nt));
        CK(cudaMemcpyAsync(raw, ht.rgb.data(), nt * 3, cudaMemcpyHostToDevice, ctx->stream));
        texture_stage_kernel<<<nblk(nt, 256), 256, 0, ctx->stream>>>(raw, (int64_t)nt, tex);
        ctx->launches++;
        CK(cudaStreamSynchronize(ctx->stream));
        CKS(dfree(ctx, raw));
        TexDev &T = S.tex[t];
        T.texels = tex; T.W = ht.w; T.H = ht.h; T.isbump = ht.isbump; T.lenx = ht.lenx; T.leny = ht.leny;
        for (int i = 0; i < 3; i++) { T.n[i] = ht.n[i]; T.p[i] = ht.p[i]; }
        if (ht.isbump) {
            std::vector<double> hh(nt);
            const double coeff = 0.5;
            for (size_t i = 0; i < nt; i++) {
                double r = (double)ht.rgb[3 * i] / (double)256, g = (double)ht.rgb[3 * i + 1] / (double)256, b = (double)ht.rgb[3 * i + 2] / (double)256;
                double v = (0.299 * r + 0.587 * g + 0.114 * b);
                v = 1 - std::exp(-3.3 * v);
                v *= coeff;
                hh[i] = v;
            }
            CKS(dalloc(ctx, &heights[t], nt));
            CK(cudaMemcpyAsync(heights[t], hh.data(), nt * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
        }
    }
    S.ntex = (int)ctx->textures.size();
    int nbvh = 0, nbez = 0;
    S.nobj = (int)ctx->objects.size();
    for (int i = 0; i < S.nobj; i++) {
        const HostObject &ho = ctx->objects[i];
        ObjDev &O = S.obj[i];
        O.kind = ho.kind; O.tex = ho.tex; O.bvh = -1; O.objtype = ho.objtype; O.aux = 0;
        O.r = ho.r; O.r2 = ho.r * ho.r; O.refl = ho.refl; O.transp = ho.transp;
        for (int k = 0; k < 3; k++) { O.a[k] = ho.a[k]; O.b[k] = ho.b[k]; O.col[k] = ho.col[k]; }
        // main.cpp:82,129,135
        O.material = (ho.refl < CGRT_EPS && ho.transp < CGRT_EPS) ? MAT_DIFFUSE : (ho.transp < CGRT_EPS ? MAT_MIRROR : MAT_GLASS);
        ctx->obj_bvh[i] = -1;
        if (ho.kind == OBJ_MESH) {
            if (nbvh >= CGRT_MAX_BVH) FAIL(CGRT_ERR_CAPACITY, "too many meshes");
            int n = (int)(ho.tri9.size() / 9);
            double *tri9;
            CKS(dalloc(ctx, &tri9, ho.tri9.size()));
            CK(cudaMemcpyAsync(tri9, ho.tri9.data(), ho.tri9.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
            CKS(build_bvh(ctx, tri9, n, orientation_sign(ho.tri9.data(), (size_t)n), nbvh));
            O.bvh = nbvh; ctx->obj_bvh[i] = nbvh; nbvh++;
        } else if (ho.kind == OBJ_PLANE && ho.tex >= 0) {
            const HostTexture &ht = ctx->textures[ho.tex];
            // objects.h:482: only an n.y == 1 plane with a bump texture gets the displaced mesh
            if (std::fabs(ho.b[1] - 1.0) < 1e-5 && ht.isbump && ht.h / 3 - 1 > 0 && ht.w / 3 - 1 > 0) {
                if (nbvh >= CGRT_MAX_BVH) FAIL(CGRT_ERR_CAPACITY, "too many meshes");
                int ncell = (ht.h / 3 - 1) * (ht.w / 3 - 1);
                int n = 2 * ncell;
                double *tri9;
                CKS(dalloc(ctx, &tri9, (size_t)n * 9));
                bump_triangles_kernel<<<nblk(ncell, 256), 256, 0, ctx->stream>>>(heights[ho.tex], ht.h, ht.w, ht.p[0], ht.p[2], ht.lenx, ht.leny, ho.a[1], tri9);
                ctx->launches++;
                std::vector<double> host((size_t)n * 9);
                CK(cudaMemcpyAsync(host.data(), tri9, host.size() * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
                CK(cudaStreamSynchronize(ctx->stream));
                CKS(build_bvh(ctx, tri9, n, orientation_sign(host.data(), (size_t)n), nbvh));
                O.bvh = nbvh; ctx->obj_bvh[i] = nbvh; nbvh++;
            }
        } else if (ho.kind == OBJ_BEZIER) {
            if (nbez >= CGRT_MAX_BEZIER) FAIL(CGRT_ERR_CAPACITY, "too many Bezier objects");
            BezDev &Z = S.bez[nbez];
            Z.ncp = (int)(ho.cp.size() / 3);
            double max_z = -1e10, max_y = -1e10, min_y = 1e10;  // bezier.h:50-63
            for (int k = 0; k < Z.ncp; k++) {
                for (int c = 0; c < 3; c++) Z.cp[k][c] = ho.cp[3 * k + c];
                if (Z.cp[k][2] > max_z) max_z = Z.cp[k][2];
                if (Z.cp[k][1] > max_y) max_y = Z.cp[k][1];
                if (Z.cp[k][1] < min_y) min_y = Z.cp[k][1];
            }
            for (int c = 0; c < 3; c++) Z.pos[c] = ho.a[c];
            Z.box[0] = max_z + ho.a[0]; Z.box[1] = -max_z + ho.a[0];
            Z.box[2] = max_y + ho.a[1]; Z.box[3] = min_y + ho.a[1];
            Z.box[4] = max_z + ho.a[2]; Z.box[5] = -max_z + ho.a[2];
            double rz = Z.cp[Z.ncp - 1][2];
            Z.umin_r2 = rz * rz;
            bez_binomials(Z.ncp, Z.C, Z.Cm);
            O.aux = nbez++;
        }
    }
    S.nbvh = nbvh;
    S.nbez = nbez;
    for (int b = 0; b < nbvh; b++) ctx->bvh_f32 = ctx->bvh_f32 && S.bvh[b].f32_ok;
    S.nplane = S.nsphere = S.ndeferred = 0;
    for (int i = 0; i < S.nobj; i++) {
        if (S.obj[i].kind == OBJ_PLANE) S.plane_ix[S.nplane++] = (unsigned char)i;
        if (S.obj[i].kind == OBJ_SPHERE) S.sphere_ix[S.nsphere++] = (unsigned char)i;
        if (S.obj[i].bvh >= 0 || S.obj[i].kind == OBJ_BEZIER) S.deferred_ix[S.ndeferred++] = (unsigned char)i;
    }
    for (double *h : heights) CKS(dfree(ctx, h));
    ctx->committed = true;
    return CGRT_OK;
}

// ---- parity hooks ------------------------------------------------------------------------------------------------

static int intersect_impl(cgrt_ctx *ctx, int64_t n, const double *org, const double *dir, double *t, double *nrm, double *nrm_raw, int32_t *obj,
                          int32_t *into, int32_t *prim, bool count, uint64_t *nv, uint64_t *tt) {
    if (!ctx || n < 0 || !org || !dir) return CGRT_ERR_INVALID;
    if (!ctx->committed) FAIL(CGRT_ERR_INVALID, "commit the scene first");
    if (n == 0) return CGRT_OK;
    CK(cudaSetDevice(ctx->device));
    double *d_org, *d_dir, *d_t, *d_n, *d_nr;
    int *d_obj, *d_into, *d_prim;
    CKS(upload(ctx, &d_org, org, (size_t)n * 3));
    CKS(upload(ctx, &d_dir, dir, (size_t)n * 3));
    CKS(dalloc(ctx, &d_t, (size_t)n)); CKS(dalloc(ctx, &d_n, (size_t)n * 3)); CKS(dalloc(ctx, &d_nr, (size_t)n * 3));
    CKS(dalloc(ctx, &d_obj, (size_t)n)); CKS(dalloc(ctx, &d_into, (size_t)n)); CKS(dalloc(ctx, &d_prim, (size_t)n));
    CK(cudaMemsetAsync(ctx->d_tc, 0, sizeof(TravCounters), ctx->stream));
    if (count) intersect_batch_kernel<true><<<nblk(n, 128), 128, 0, ctx->stream>>>(ctx->S, n, d_org, d_dir, d_t, d_n, d_nr, d_obj, d_into, d_prim, ctx->d_tc);
    else intersect_batch_kernel<false><<<nblk(n, 128), 128, 0, ctx->stream>>>(ctx->S, n, d_org, d_dir, d_t, d_n, d_nr, d_obj, d_into, d_prim, ctx->d_tc);
    ctx->launches++;
    CK(cudaGetLastError());
    CKS(download_free(ctx, t, d_t, (size_t)n));
    CKS(download_free(ctx, nrm, d_n, (size_t)n * 3));
    CKS(download_free(ctx, nrm_raw, d_nr, (size_t)n * 3));
    CKS(download_free(ctx, (int *)obj, d_obj, (size_t)n));
    CKS(download_free(ctx, (int *)into, d_into, (size_t)n));
    CKS(download_free(ctx, (int *)prim, d_prim, (size_t)n));
    CKS(dfree(ctx, d_org)); CKS(dfree(ctx, d_dir));
    if (count) {
        TravCounters tc;
        CK(cudaMemcpy(&tc, ctx->d_tc, sizeof tc, cudaMemcpyDeviceToHost));
        if (nv) *nv = tc.node_visits;
        if (tt) *tt = tc.tri_tests;
    }
    return CGRT_OK;
}
int cgrt_intersect_batch(cgrt_ctx *ctx, int64_t n, const double *org, const double *dir, double *t, double *nrm, double *nrm_raw, int32_t *obj,
                         int32_t *into, int32_t *prim) {
    return intersect_impl(ctx, n, org, dir, t, nrm, nrm_raw, obj, into, prim, false, nullptr, nullptr);
}
int cgrt_count_traversal(cgrt_ctx *ctx, int64_t n, const double *org, const double *dir, uint64_t *node_visits, uint64_t *tri_tests) {
    return intersect_impl(ctx, n, org, dir, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, true, node_visits, tri_tests);
}

int cgrt_hash_keys(cgrt_ctx *ctx, int64_t n, const double *pos, int hashsize, double celllength_in, uint32_t *key, int32_t *ixyz) {
    if (!ctx || n < 0 || !pos || hashsize <= 0 || !(celllength_in > 0)) return CGRT_ERR_INVALID;
    if (n == 0) return CGRT_OK;
    CK(cudaSetDevice(ctx->device));
    int cells = (int)(std::ceil(70.0 / celllength_in));  // hash.h:25-26
    double cl = 70.0 / cells;
    double *d_pos;
    uint32_t *d_key;
    int *d_ixyz;
    CKS(upload(ctx, &d_pos, pos, (size_t)n * 3));
    CKS(dalloc(ctx, &d_key, (size_t)n)); CKS(dalloc(ctx, &d_ixyz, (size_t)n * 3));
    hash_keys_kernel<<<nblk(n, 256), 256, 0, ctx->stream>>>(n, d_pos, (uint32_t)hashsize, cl, d_key, d_ixyz);
    ctx->launches++;
    CK(cudaGetLastError());
    CKS(download_free(ctx, key, d_key, (size_t)n));
    CKS(download_free(ctx, (int *)ixyz, d_ixyz, (size_t)n * 3));
    CKS(dfree(ctx, d_pos));
    return CGRT_OK;
}

int cgrt_surface_color(cgrt_ctx *ctx, int obj, int64_t n, const double *pos, double *col) {
    if (!ctx || n < 0 || !pos || !col) return CGRT_ERR_INVALID;
    if (!ctx->committed || obj < 0 || obj >= ctx->S.nobj) FAIL(CGRT_ERR_INVALID, "bad object id / scene not committed");
    if (n == 0) return CGRT_OK;
    double *d_pos, *d_col;
    CKS(upload(ctx, &d_pos, pos, (size_t)n * 3));
    CKS(dalloc(ctx, &d_col, (size_t)n * 3));
    surface_color_kernel<<<nblk(n, 256), 256, 0, ctx->stream>>>(ctx->S, obj, n, d_pos, d_col);
    ctx->launches++;
    CK(cudaGetLastError());
    CKS(download_free(ctx, col, d_col, (size_t)n * 3));
    CKS(dfree(ctx, d_pos));
    return CGRT_OK;
}

int cgrt_object_triangles(cgrt_ctx *ctx, int obj, double *tri9, int64_t cap, int64_t *ntri) {
    if (!ctx || !ntri) return CGRT_ERR_INVALID;
    if (!ctx->committed || obj < 0 || obj >= ctx->S.nobj) FAIL(CGRT_ERR_INVALID, "bad object id / scene not committed");
    int b = ctx->obj_bvh[obj];
    *ntri = b < 0 ? 0 : ctx->bvh_src[b].ntris;
    if (tri9 && b >= 0) {
        int64_t n = *ntri < cap ? *ntri : cap;
        CK(cudaStreamSynchronize(ctx->stream));
        CK(cudaMemcpy(tri9, ctx->bvh_src[b].tri9, (size_t)n * 9 * sizeof(double), cudaMemcpyDeviceToHost));
    }
    return CGRT_OK;
}

int cgrt_sample(cgrt_ctx *ctx, uint64_t seed, uint32_t pass, uint64_t path, uint32_t dim, int what, const double aux[3], double out[3]) {
    if (!ctx || !out) return CGRT_ERR_INVALID;
    double *d_out;
    CKS(dalloc(ctx, &d_out, 3));
    double a0 = aux ? aux[0] : 0, a1 = aux ? aux[1] : 0, a2 = aux ? aux[2] : 0;
    sample_kernel<<<1, 1, 0, ctx->stream>>>(seed, pass, path, dim, what, a0, a1, a2, d_out);
    ctx->launches++;
    CK(cudaGetLastError());
    return download_free(ctx, out, d_out, 3);
}

int cgrt_radix_sort(cgrt_ctx *ctx, int64_t n, const uint64_t *key_in, int nbits, uint64_t *key_out, uint32_t *perm) {
    if (!ctx || n < 0 || !key_in || nbits <= 0 || nbits > 64) return CGRT_ERR_INVALID;
    if (n == 0) return CGRT_OK;
    uint64_t *d_in, *d_out;
    uint32_t *d_perm;
    CKS(upload(ctx, &d_in, key_in, (size_t)n));
    CKS(dalloc(ctx, &d_out, (size_t)n)); CKS(dalloc(ctx, &d_perm, (size_t)n));
    CKS(radix_sort_dev(ctx, (size_t)n, d_in, nbits, d_out, d_perm));
    CKS(download_free(ctx, key_out, d_out, (size_t)n));
    CKS(download_free(ctx, perm, d_perm, (size_t)n));
    return dfree(ctx, d_in);
}

// The per-depth wavefront of the eye half of trace() over the n rays in ray queue 0 (or, generate = true, the camera rays of the rows from r0).
static int eye_wavefront(cgrt_ctx *ctx, size_t n, int depth0, int r0, bool generate) {
    const PassParams &P = ctx->P;
    size_t max_rays = 4u << 20;
    int cur = 0;
    for (int depth = depth0; depth < P.max_depth && n > 0; depth++) {
        CKS(ensure_queue(ctx, cur ^ 1, 2 * n > max_rays ? 2 * n : max_rays));  // glass splits: at most two children per ray
        CKS(ensure_hp_capacity(ctx, (size_t)ctx->hp_count + n));
        CK(cudaMemsetAsync(ctx->d_qcount + (cur ^ 1), 0, sizeof(unsigned int), ctx->stream));
        const bool f32 = ctx->bvh_f32;
#define LAUNCH_EYE(FIRSTV, F32V, SPPMV)                                                                                                      \
    eye_bounce_kernel<FIRSTV, F32V, SPPMV><<<nblk(n, 128), 128, 0, ctx->stream>>>(ctx->S, P, depth, ctx->q[cur], (unsigned int)n, r0, ctx->q[cur ^ 1], \
                                                                          ctx->d_qcount + (cur ^ 1), ctx->hp_rec, ctx->d_hp_count, ctx->hp_cap, ctx->d_ctr, \
                                                                          ctx->sppm_round)
        if (generate && depth == depth0 && ctx->sppm == CGRT_SPPM_JITTER) { if (f32) LAUNCH_EYE(true, true, CGRT_SPPM_JITTER); else LAUNCH_EYE(true, false, CGRT_SPPM_JITTER); }
        else if (generate && depth == depth0 && ctx->sppm == CGRT_SPPM_CORNER) { if (f32) LAUNCH_EYE(true, true, CGRT_SPPM_CORNER); else LAUNCH_EYE(true, false, CGRT_SPPM_CORNER); }
        else if (generate && depth == depth0) { if (f32) LAUNCH_EYE(true, true, 0); else LAUNCH_EYE(true, false, 0); }
        else { if (f32) LAUNCH_EYE(false, true, 0); else LAUNCH_EYE(false, false, 0); }
#undef LAUNCH_EYE
        ctx->launches++;
        CK(cudaGetLastError());
        unsigned int counts[2];
        CK(cudaMemcpyAsync(&counts[0], ctx->d_qcount + (cur ^ 1), sizeof(unsigned int), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(&counts[1], ctx->d_hp_count, sizeof(unsigned int), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        n = counts[0];
        ctx->hp_count = counts[1];
        cur ^= 1;
    }
    return CGRT_OK;
}

// ---- eye pass ------------------------------------------------------------------------------------------------------
static int eye_pass_impl(cgrt_ctx *ctx, int y0, int y1);
int cgrt_eye_pass(cgrt_ctx *ctx, int y0, int y1) {
    if (!ctx) return CGRT_ERR_INVALID;
    if (ctx->sppm) FAIL(CGRT_ERR_INVALID, "SPPM is on: cgrt_sppm_begin_round / cgrt_sppm_eye_pass trace the eye pass of every round");
    return eye_pass_impl(ctx, y0, y1);
}
static int eye_pass_impl(cgrt_ctx *ctx, int y0, int y1) {
    if (!ctx->committed) FAIL(CGRT_ERR_INVALID, "commit the scene first");
    if (ctx->grid_built) FAIL(CGRT_ERR_INVALID, "grid already built");
    const PassParams &P = ctx->P;
    if (y1 < 0) y1 = P.height;
    if (y0 < 0 || y1 > P.height || y0 >= y1) FAIL(CGRT_ERR_INVALID, "bad row range");
    CK(cudaSetDevice(ctx->device));
    PhaseTimer timer(ctx, 0);
    size_t per_row = (size_t)P.width * P.samples;
    size_t max_rays = 4u << 20;
    if (const char *e = getenv("CGRT_EYE_CHUNK")) { long long c = atoll(e); if (c > 0) max_rays = (size_t)c; }  // tests: force many chunks / queue growth
    int rows_per_chunk = (int)(max_rays / per_row);
    if (rows_per_chunk < 1) rows_per_chunk = 1;
    for (int r0 = y0; r0 < y1; r0 += rows_per_chunk) {
        int r1 = r0 + rows_per_chunk < y1 ? r0 + rows_per_chunk : y1;
        size_t n = (size_t)(r1 - r0) * per_row;
        CKS(eye_wavefront(ctx, n, 0, r0, true));
    }
    timer.stop();
    return CGRT_OK;
}

int cgrt_export_hitpoints_dev(cgrt_ctx *ctx, void **records_dev, int64_t *count) {
    if (!ctx || !records_dev || !count) return CGRT_ERR_INVALID;
    *records_dev = ctx->hp_rec;
    *count = ctx->hp_count;
    return CGRT_OK;
}
int cgrt_import_hitpoints_dev(cgrt_ctx *ctx, const void *records_dev, int64_t count) {
    if (!ctx || count < 0 || (count > 0 && !records_dev)) return CGRT_ERR_INVALID;
    if (ctx->sppm && !ctx->sppm_traced)
        FAIL(CGRT_ERR_INVALID, "SPPM is on: import the round's visible points between cgrt_sppm_eye_pass and cgrt_build_grid");
    if (ctx->grid_built) FAIL(CGRT_ERR_INVALID, "grid already built");
    CK(cudaSetDevice(ctx->device));
    if (count >= (1ll << 32)) FAIL(CGRT_ERR_INVALID, "more hitpoint records than one import holds");
    if (count) {  // the records come from the caller: checked before they replace anything (see hp_validate_kernel)
        unsigned int *d_bad, bad = 0;
        CKS(dalloc(ctx, &d_bad, 1));
        CK(cudaMemsetAsync(d_bad, 0, sizeof(unsigned int), ctx->stream));
        hp_validate_kernel<<<nblk((size_t)count, 256), 256, 0, ctx->stream>>>(static_cast<const double *>(records_dev), (unsigned int)count, ctx->P.celllength,
                                                                           ctx->P.hashsize, ctx->P.width, ctx->P.height, d_bad);
        ctx->launches++;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(&bad, d_bad, sizeof bad, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        CKS(dfree(ctx, d_bad));
        if (bad & 1u) FAIL(CGRT_ERR_INVALID, "import: a record's bucket key is >= hashsize");
        if (bad & 2u) FAIL(CGRT_ERR_INVALID, "import: a record's bucket key is not the cell key of its position");
        if (bad & 4u) FAIL(CGRT_ERR_INVALID, "import: a record's pixel lies outside the image");
    }
    // replaces the current set (the caller passes the all-gathered union, which includes this rank's own records)
    ctx->hp_count = 0;
    CKS(ensure_hp_capacity(ctx, (size_t)count));
    if (count) CK(cudaMemcpyAsync(ctx->hp_rec, records_dev, (size_t)count * CGRT_HP_RECORD_DOUBLES * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    unsigned int c = (unsigned int)count;
    CK(cudaMemcpyAsync(ctx->d_hp_count, &c, sizeof c, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->hp_count = c;
    return CGRT_OK;
}

// Per-photon update: (re)build the table r2(n), n < cap, with the reference's own statements (main.cpp:119-120) on the host.
static int build_r2_table(cgrt_ctx *ctx, int cap) {
    std::vector<double> t((size_t)cap);
    double r2 = ctx->P.r2_init;
    const double alpha = ctx->P.alpha;
    for (int n = 0; n < cap; n++) {
        t[(size_t)n] = r2;
        double g = (n * alpha + alpha) / (n * alpha + 1.0);
        r2 *= g;
    }
    if (ctx->r2tab) CKS(dfree(ctx, ctx->r2tab));
    CKS(dalloc(ctx, &ctx->r2tab, (size_t)cap));
    CK(cudaMemcpyAsync(ctx->r2tab, t.data(), (size_t)cap * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->r2cap = cap;
    return CGRT_OK;
}

// ---- grid ----------------------------------------------------------------------------------------------------------
static int build_grid_impl(cgrt_ctx *ctx);
int cgrt_build_grid(cgrt_ctx *ctx) {
    if (!ctx) return CGRT_ERR_INVALID;
    if (ctx->sppm && !ctx->sppm_traced) FAIL(CGRT_ERR_INVALID, "SPPM is on: trace the round's visible points first (cgrt_sppm_eye_pass)");
    return build_grid_impl(ctx);
}
static int build_grid_impl(cgrt_ctx *ctx) {
    if (ctx->grid_built) FAIL(CGRT_ERR_INVALID, "grid already built");
    CK(cudaSetDevice(ctx->device));
    PhaseTimer timer(ctx, 1);
    const PassParams &P = ctx->P;
    unsigned int n = ctx->hp_count;
    ctx->nhp = n;
    // buffers are sized for m >= n hitpoints: m = n, except under SPPM (see cgrt_ctx::sppm_cap)
    if (ctx->sppm && n > ctx->sppm_cap) ctx->sppm_cap = (size_t)n + n / 8 + 4096;
    const size_t m = ctx->sppm ? ctx->sppm_cap : (size_t)n;
    size_t npix = (size_t)P.width * P.height;
    CKS(dalloc(ctx, &ctx->cell_start, (size_t)P.hashsize + 1));
    CKS(dalloc(ctx, &ctx->pix_start, npix + 1));
    CKS(dalloc(ctx, &ctx->pix_perm, m));
    // The arrays the deposit kernel gathers from — prefilter, exact records, f, accumulators — live in one slab. (Marking the slab
    // persisting in L2 with an access-policy window was measured: the deposit kernel did not move (11.0 ms, it is not bound by L2
    // misses) while the counting sort lost its L2-resident cursors (1.2 -> 4.2 ms), so no window is set.)
    size_t acc_bytes = (size_t)n * 4 * acc_elem(ctx);
    {
        auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
        const size_t acc_cap = m * 4 * acc_elem(ctx);
        size_t o_pre = 0, o_pren = o_pre + up(m * sizeof(float4)), o_pref = o_pren + up(m * sizeof(float4));
        size_t o_hot = o_pref + up(m * sizeof(float4)), o_f = o_hot + up(m * sizeof(HpHot));
        size_t o_acc = o_f + up(m * 4 * sizeof(double)), total = o_acc + up(acc_cap);
        char *slab;
        CKS(dalloc(ctx, &slab, total));
        ctx->A.pre = reinterpret_cast<float4 *>(slab + o_pre);
        ctx->A.pre_n = reinterpret_cast<float4 *>(slab + o_pren);
        ctx->A.pre_f = reinterpret_cast<float4 *>(slab + o_pref);
        ctx->A.hot = reinterpret_cast<HpHot *>(slab + o_hot);
        ctx->A.f = reinterpret_cast<double *>(slab + o_f);
        ctx->acc = slab + o_acc;
        CK(cudaMemsetAsync(ctx->acc, 0, acc_bytes ? acc_bytes : 1, ctx->stream));
    }
    if (ctx->cfg.update_mode == 0) {
        CKS(build_r2_table(ctx, 1 << 20));
        CKS(dalloc(ctx, &ctx->d_maxcnt, 1));
        CK(cudaMemsetAsync(ctx->d_maxcnt, 0, sizeof(int), ctx->stream));
    }
    CKS(dalloc(ctx, &ctx->A.flux, m * 4));
    CKS(dalloc(ctx, &ctx->A.cnt, m));
    CKS(dalloc(ctx, &ctx->A.hw, m * 2));
    CKS(dalloc(ctx, &ctx->A.key, m));
    CKS(dalloc(ctx, &ctx->A.seq, m));
    if (n > 0) {
        uint64_t *keys, *keys_sorted, *pixkeys, *pixkeys_sorted;
        uint32_t *perm;
        CKS(dalloc(ctx, &keys, m)); CKS(dalloc(ctx, &keys_sorted, m)); CKS(dalloc(ctx, &perm, m));
        CKS(dalloc(ctx, &pixkeys, m)); CKS(dalloc(ctx, &pixkeys_sorted, m));
        hp_extract_keys_kernel<<<nblk(n, 256), 256, 0, ctx->stream>>>(ctx->hp_rec, n, keys);
        ctx->launches++;
        int kbits = 32;
        while (kbits > 1 && !(((uint64_t)P.hashsize - 1) >> (kbits - 1))) kbits--;
        CKS(radix_sort_dev(ctx, n, keys, 32 + kbits, keys_sorted, perm, m));
        hp_gather_sorted_kernel<<<nblk(n, 256), 256, 0, ctx->stream>>>(ctx->hp_rec, perm, n, P.r2_init, ctx->A, pixkeys, P.width);
        if (ctx->sppm) {
            sppm_visible_radius_kernel<<<nblk(n, 256), 256, 0, ctx->stream>>>(n, ctx->A, ctx->pix_r2, P.width);
            ctx->launches++;
        }
        lower_bound_table_kernel<<<nblk((size_t)n + 1, 256), 256, 0, ctx->stream>>>(ctx->A.key, nullptr, n, P.hashsize, ctx->cell_start);
        CKS(dalloc(ctx, &ctx->reach, (size_t)1 << (CGRT_REACH_BITS - 5)));
        CK(cudaMemsetAsync(ctx->reach, 0, sizeof(uint32_t) << (CGRT_REACH_BITS - 5), ctx->stream));
        reach_mark_kernel<<<nblk(n, 256), 256, 0, ctx->stream>>>(ctx->A.hot, n, P.celllength, ctx->reach);
        ctx->launches++;
        ctx->launches += 2;
        int pbits = 1;
        while (pbits < 40 && ((uint64_t)npix >> pbits)) pbits++;
        CKS(radix_sort_dev(ctx, n, pixkeys, pbits, pixkeys_sorted, ctx->pix_perm, m));
        lower_bound_table_kernel<<<nblk((size_t)n + 1, 256), 256, 0, ctx->stream>>>(nullptr, pixkeys_sorted, n, (unsigned int)npix, ctx->pix_start);
        ctx->launches++;
        CK(cudaStreamSynchronize(ctx->stream));
        CK(cudaGetLastError());
        CKS(dfree(ctx, keys)); CKS(dfree(ctx, keys_sorted)); CKS(dfree(ctx, perm)); CKS(dfree(ctx, pixkeys)); CKS(dfree(ctx, pixkeys_sorted));
    } else {
        CK(cudaMemsetAsync(ctx->cell_start, 0, ((size_t)P.hashsize + 1) * sizeof(uint32_t), ctx->stream));
        CK(cudaMemsetAsync(ctx->pix_start, 0, (npix + 1) * sizeof(uint32_t), ctx->stream));
    }
    // the raw records are no longer needed (SPPM keeps the buffer at its capacity for the next round's eye pass)
    if (!ctx->sppm) {
        CKS(dfree(ctx, ctx->hp_rec));
        ctx->hp_rec = nullptr;
        ctx->hp_cap = 0;
    }
    ctx->grid_built = true;
    ctx->sppm_traced = false;
    timer.stop();
    return CGRT_OK;
}

// SPPM: release the grid and the visible points of the last round (every buffer build_grid_impl allocated).
static int release_grid(cgrt_ctx *ctx) {
    HpArrays &A = ctx->A;
    CKS(dfree(ctx, A.pre));  // the slab: pre, pre_n, pre_f, hot, f, accumulators
    CKS(dfree(ctx, A.flux)); CKS(dfree(ctx, A.cnt)); CKS(dfree(ctx, A.hw)); CKS(dfree(ctx, A.key)); CKS(dfree(ctx, A.seq));
    CKS(dfree(ctx, ctx->cell_start)); CKS(dfree(ctx, ctx->pix_start)); CKS(dfree(ctx, ctx->pix_perm)); CKS(dfree(ctx, ctx->reach));
    memset(&A, 0, sizeof A);
    ctx->acc = nullptr;
    ctx->cell_start = ctx->pix_start = ctx->pix_perm = ctx->reach = nullptr;
    ctx->grid_built = false;
    ctx->nhp = 0;
    return CGRT_OK;
}

// ---- photon pass ---------------------------------------------------------------------------------------------------
// Per chunk: max_depth trace launches (the first emits and runs the analytic fast path, the others resume the photons that
// were suspended in front of a mesh), a 24-bit radix sort of the deposit keys, and the cell-grouped deposit kernel. No host
// synchronisation anywhere: the pass is asynchronous on the ctx stream unless profiling is on (then the phases are
// bracketed by events and the pass ends with one synchronise).
// inj_* != nullptr: the photons are the caller's rays (device arrays, cgrt_trace) instead of emissions from the light; one launch.
static int photon_pass_impl(cgrt_ctx *ctx, uint64_t first, uint64_t count, const double *inj_org, const double *inj_dir, const double *inj_flux, int inj_depth) {
    if (!ctx) return CGRT_ERR_INVALID;
    if (!ctx->grid_built) FAIL(CGRT_ERR_INVALID, "build the grid first");
    CK(cudaSetDevice(ctx->device));
    const PassParams &P = ctx->P;
    size_t chunk = ctx->photon_chunk ? ctx->photon_chunk : ctx->auto_chunk;
    if (chunk == 0) {  // once per context: cudaMemGetInfo is not free
        size_t free_b = 0, total_b = 0;
        CK(cudaMemGetInfo(&free_b, &total_b));
        const size_t per_photon = (size_t)P.max_depth * (deposit_rec_bytes(compact_records(ctx)) + 2 * sizeof(uint32_t)) * (ctx->overlap ? 2 : 1) + 2 * sizeof(PhotonState);
        // what this context can actually get: free memory plus the blocks the arena holds for this device (a parked block is either
        // reused as it is or released on demand by arena_take), not the device's total — other contexts and frameworks share the GPU
        const size_t avail_b = free_b + arena_held(ctx->device);
        (void)total_b;
        chunk = (avail_b / 10 * 6) / per_photon;
        chunk &= ~(((size_t)1 << 20) - 1);
        if (chunk > ((size_t)128 << 20)) chunk = (size_t)128 << 20;
        if (chunk < ((size_t)1 << 20)) chunk = (size_t)1 << 20;
        ctx->auto_chunk = chunk;
    }
    const size_t first_chunk = count < chunk ? (size_t)count : chunk;
    if (first_chunk == 0) return CGRT_OK;
    CKS(ensure_photon_buffers(ctx, first_chunk, first_chunk * (size_t)P.max_depth));
    if (inj_org && first_chunk != count) FAIL(CGRT_ERR_CAPACITY, "cgrt_trace: more rays than one launch holds");
    const unsigned int resume_grid = (unsigned int)ctx->sm_count * 8u;  // 8 resident blocks per SM, grid-stride over the queue
    const bool overlap = ctx->overlap && !ctx->profiling;
    cudaStream_t D = ctx->stream, T = overlap ? ctx->tstream : ctx->stream;
    // Profiling runs on one stream and keeps one list of (event, timing slot) stamps: a stamp charges the time since the stamp before
    // it to its slot, and a chunk opens with slot -1, so the gap between chunks is not charged. Slot 2 (the chunk's whole trace) gets
    // the memsets and, in the reduction below, every emission (9), Bezier + traversal (7) and continuation (8) interval as well.
    std::vector<std::pair<cudaEvent_t, int>> marks;
    auto stamp = [&](int slot) {
        cudaEvent_t ev;
        if (ctx->profiling && cudaEventCreate(&ev) == cudaSuccess) {
            cudaEventRecord(ev, D);
            marks.push_back(std::make_pair(ev, slot));
        }
    };
    for (uint64_t done = 0; done < count; done += chunk) {
        const size_t n = (size_t)((count - done) < chunk ? (count - done) : chunk);
        const uint64_t base = first + done;
        const size_t slots = n * (size_t)P.max_depth;
        cgrt_ctx::DepBuf &B = ctx->dep[overlap ? (ctx->chunk_seq++ & 1u) : 0u];
        stamp(-1);
        // ---- trace (stream T): may not overwrite the buffer before its previous deposit pass has drained it
        if (B.drained_valid) CK(cudaStreamWaitEvent(T, B.drained, 0));
        CK(cudaMemsetAsync(B.keys, 0xff, slots * sizeof(uint32_t), T));
        CK(cudaMemsetAsync(B.hist, 0, ((size_t)P.bin_mask + 1) * sizeof(uint32_t), T));
        CK(cudaMemsetAsync(ctx->d_qcount + 2, 0, 12 * sizeof(unsigned int), T));
        stamp(2);
        unsigned int *qc = ctx->d_qcount + 2;
#define LAUNCH_PT(F, GRID, QIN, NIN, QOUT, NOUT, CURSOR)                                                                            \
    photon_trace_kernel<F><<<GRID, CGRT_PHOTON_BLOCK, 0, T>>>(ctx->S, P, base, (unsigned int)n, QIN, NIN, QOUT, NOUT, B.rec, compact_records(ctx) ? 1 : 0, B.keys, B.hist, \
                                                             ctx->cull ? ctx->reach : nullptr, ctx->d_ctr, CURSOR)
        if (inj_org) {
            photon_inject_kernel<<<nblk(n, 128), 128, 0, T>>>(ctx->S, (unsigned int)n, inj_depth, inj_org, inj_dir, inj_flux, ctx->pq[0], qc);
        } else {
            unsigned int want = nblk(n, CGRT_PHOTON_BLOCK);
            LAUNCH_PT(true, (want < ctx->grid_first ? want : ctx->grid_first), nullptr, nullptr, ctx->pq[0], qc, qc + 6);
        }
        stamp(9);
        ctx->launches++;
        if (inj_org || ctx->S.nbvh > 0 || ctx->S.nbez > 0) {
            for (int pass = 1; pass <= P.max_depth; pass++) {  // a resumed photon advances at least one segment per pass
                PhotonState *qin = ctx->pq[(pass - 1) & 1];
                PhotonState *qout = ctx->pq[pass & 1];
                const unsigned int *nin = qc + pass - 1;
                if (ctx->S.nbez > 0) {
                    photon_bezier_kernel<<<resume_grid, 128, 0, T>>>(ctx->S, qin, nin);
                    ctx->launches++;
                }
                if (ctx->S.nbvh > 0) {
                    static const bool trav_exact = getenv("CGRT_TRAV_EXACT") != nullptr;  // dev: force the fp64-slab instantiation
                    const bool f32 = ctx->bvh_f32 && !trav_exact;  // true on all BASELINE scenes
                    if (ctx->counting) {
                        if (f32) photon_traverse_kernel<true, true><<<resume_grid, 128, 0, T>>>(ctx->S, qin, nin, ctx->d_tc);
                        else photon_traverse_kernel<true, false><<<resume_grid, 128, 0, T>>>(ctx->S, qin, nin, ctx->d_tc);
                    } else {
                        if (f32) photon_traverse_kernel<false, true><<<resume_grid, 128, 0, T>>>(ctx->S, qin, nin, ctx->d_tc);
                        else photon_traverse_kernel<false, false><<<resume_grid, 128, 0, T>>>(ctx->S, qin, nin, ctx->d_tc);
                    }
                    ctx->launches++;
                }
                stamp(7);
                LAUNCH_PT(false, ctx->grid_cont, qin, nin, qout, qc + pass, qc + 6 + pass);
                stamp(8);
                ctx->launches++;
            }
        }
#undef LAUNCH_PT
        // ---- sort + deposit (stream D) after the trace of this buffer
        if (overlap) {
            CK(cudaEventRecord(B.traced, T));
            CK(cudaStreamWaitEvent(D, B.traced, 0));
        }
        // the trace launches above read neither radii nor accumulators; the gather does: the previous round's update must have landed
        CKS(join_update(ctx));
        if (ctx->nhp > 0) {
            const int nsb = (int)(((size_t)P.bin_mask + 1) / (CGRT_SCAN_BLOCK * CGRT_SCAN_ITEMS));
            bin_scan_blocks_kernel<<<nsb, CGRT_SCAN_BLOCK, 0, D>>>(B.hist, B.bsum);
            bin_scan_sums_kernel<<<1, CGRT_SCAN_BLOCK, 0, D>>>(B.bsum, nsb, B.nvalid);
            bin_scatter_kernel<<<ctx->deposit_grid, 256, 0, D>>>(B.keys, slots, B.hist, B.bsum, B.perm);
            ctx->launches += 3;
            stamp(6);
            size_t spans = (slots + CGRT_DEPOSIT_SPAN - 1) / CGRT_DEPOSIT_SPAN;
            size_t want = (spans * 32 + CGRT_DEPOSIT_BLOCK - 1) / CGRT_DEPOSIT_BLOCK;
            unsigned int dblocks = (unsigned int)(want < (size_t)ctx->deposit_grid ? want : (size_t)ctx->deposit_grid);
            U1State U1;
            U1.cnt = ctx->A.cnt; U1.r2tab = ctx->r2tab; U1.cap = ctx->r2cap; U1.err = ctx->d_fxerr;
            if (ctx->cfg.update_mode == 0)
                photon_deposit_kernel<2><<<dblocks, CGRT_DEPOSIT_BLOCK, 0, D>>>(P, reinterpret_cast<const DepositRec *>(B.rec), B.perm, B.nvalid, ctx->cell_start, ctx->A.pre, ctx->A.pre_n,
                                                                                ctx->A.pre_f, ctx->A.hot, ctx->A.f, ctx->acc, ctx->d_ctr, U1);
            else if (ctx->cfg.accum_mode == 0)
                photon_deposit_kernel<0><<<dblocks, CGRT_DEPOSIT_BLOCK, 0, D>>>(P, reinterpret_cast<const DepositRec *>(B.rec), B.perm, B.nvalid, ctx->cell_start, ctx->A.pre, ctx->A.pre_n,
                                                                                ctx->A.pre_f, ctx->A.hot, ctx->A.f, ctx->acc, ctx->d_ctr, U1);
            else if (ctx->cfg.accum_mode == 1)
                photon_deposit_kernel<1><<<dblocks, CGRT_DEPOSIT_BLOCK, 0, D>>>(P, reinterpret_cast<const DepositRec *>(B.rec), B.perm, B.nvalid, ctx->cell_start, ctx->A.pre, ctx->A.pre_n,
                                                                                ctx->A.pre_f, ctx->A.hot, ctx->A.f, ctx->acc, ctx->d_ctr, U1);
            else
                photon_deposit_kernel<ACC_FIXED><<<dblocks, CGRT_DEPOSIT_BLOCK, 0, D>>>(P, reinterpret_cast<const DepositRec *>(B.rec), B.perm, B.nvalid, ctx->cell_start,
                                                                                        ctx->A.pre, ctx->A.pre_n, ctx->A.pre_f, ctx->A.hot, ctx->A.f, ctx->acc, ctx->d_ctr, U1);
            ctx->launches++;
        } else {
            stamp(6);
        }
        stamp(3);
        if (overlap) {
            CK(cudaEventRecord(B.drained, D));
            B.drained_valid = true;
        }
        CK(cudaGetLastError());
    }
    if (ctx->profiling) {
        CK(cudaStreamSynchronize(ctx->stream));
        for (size_t k = 1; k < marks.size(); k++) {
            const int slot = marks[k].second;
            if (slot < 0) continue;
            float t = 0;
            cudaEventElapsedTime(&t, marks[k - 1].first, marks[k].first);
            ctx->ms[slot] += t;
            if (slot == 9 || slot == 7 || slot == 8) ctx->ms[2] += t;
        }
        for (auto &m : marks) cudaEventDestroy(m.first);
    }
    return CGRT_OK;
}

int cgrt_photon_pass(cgrt_ctx *ctx, uint64_t first, uint64_t count) { return photon_pass_impl(ctx, first, count, nullptr, nullptr, nullptr, 0); }

int cgrt_trace(cgrt_ctx *ctx, int64_t n, const double *org, const double *dir, const double *weight, int flag, int depth, const int32_t *x, const int32_t *y,
               uint64_t first_index) {
    if (!ctx || n < 0 || (n > 0 && (!org || !dir || !weight))) return CGRT_ERR_INVALID;
    if (!ctx->committed) FAIL(CGRT_ERR_INVALID, "commit the scene first");
    if (depth < 0) FAIL(CGRT_ERR_INVALID, "negative depth");
    if (flag && ctx->sppm) FAIL(CGRT_ERR_INVALID, "SPPM is on: cgrt_sppm_begin_round makes every round's visible points");
    if (n == 0 || depth >= ctx->P.max_depth) return CGRT_OK;  // main.cpp:46: nothing is traced beyond MAX_DEPTH
    if (n >= (1ll << 28)) FAIL(CGRT_ERR_CAPACITY, "cgrt_trace: at most 2^28 rays per call");
    CK(cudaSetDevice(ctx->device));
    double *d_org, *d_dir, *d_w;
    CKS(upload(ctx, &d_org, org, (size_t)n * 3)); CKS(upload(ctx, &d_dir, dir, (size_t)n * 3)); CKS(upload(ctx, &d_w, weight, (size_t)n * 3));
    int rc = CGRT_OK;
    if (flag) {  // eye ray: hitpoints are created (main.cpp:85-99), children followed (main.cpp:129-157)
        if (ctx->grid_built) FAIL(CGRT_ERR_INVALID, "eye rays add hitpoints: trace them before cgrt_build_grid");
        if (!x || !y) FAIL(CGRT_ERR_INVALID, "eye rays need their pixel (x, y)");
        for (int64_t i = 0; i < n; i++)
            if (x[i] < 0 || x[i] >= ctx->P.width || y[i] < 0 || y[i] >= ctx->P.height) FAIL(CGRT_ERR_INVALID, "pixel outside the image");
        int32_t *d_x, *d_y;
        CKS(upload(ctx, &d_x, x, (size_t)n)); CKS(upload(ctx, &d_y, y, (size_t)n));
        CKS(ensure_queue(ctx, 0, (size_t)n));
        eye_inject_kernel<<<nblk(n, 256), 256, 0, ctx->stream>>>((unsigned int)n, ctx->P.width, ctx->P.samples, d_org, d_dir, d_w, d_x, d_y, ctx->q[0]);
        ctx->launches++;
        rc = eye_wavefront(ctx, (size_t)n, depth, 0, false);
        CKS(dfree(ctx, d_x)); CKS(dfree(ctx, d_y));
    } else {     // photon: deposits into the per-round accumulators (main.cpp:101-128), bounces followed
        CK(cudaStreamSynchronize(ctx->stream));  // the uploads, whichever stream the trace kernels run on
        rc = photon_pass_impl(ctx, first_index, (uint64_t)n, d_org, d_dir, d_w, depth);
        if (rc == CGRT_OK) CK(cudaStreamSynchronize(ctx->stream));
    }
    CKS(dfree(ctx, d_org)); CKS(dfree(ctx, d_dir)); CKS(dfree(ctx, d_w));
    return rc;
}

int cgrt_accum_dev(cgrt_ctx *ctx, void **ptr_dev, int64_t *n_elems) {
    if (!ctx || !ptr_dev || !n_elems) return CGRT_ERR_INVALID;
    if (!ctx->grid_built) FAIL(CGRT_ERR_INVALID, "build the grid first");
    CKS(join_update(ctx));
    *ptr_dev = ctx->acc;
    *n_elems = (int64_t)ctx->nhp * 4;
    return CGRT_OK;
}

static int nccl_fail(cgrt_ctx *ctx, int r, const char *what) {
    NcclApi &N = nccl_api();
    ctx->err = std::string(what) + ": " + (N.GetErrorString ? N.GetErrorString(r) : "NCCL error");
    return CGRT_ERR_NCCL;
}
static int allreduce_on(cgrt_ctx *ctx, void *comm, cudaStream_t st) {
    NcclApi &N = nccl_api();
    if (!N.ok) FAIL(CGRT_ERR_NCCL, "NCCL is not available: " + N.why);
    if (ctx->nhp == 0) return CGRT_OK;
    const int type = ctx->cfg.accum_mode == 0 ? NCCL_FLOAT64 : ctx->cfg.accum_mode == 1 ? NCCL_FLOAT32 : NCCL_INT64;
    int r = N.AllReduce(ctx->acc, ctx->acc, (size_t)ctx->nhp * 4, type, NCCL_SUM, comm, st);
    if (r != 0) return nccl_fail(ctx, r, "ncclAllReduce");
    ctx->launches++;
    return CGRT_OK;
}

int cgrt_allreduce_accum(cgrt_ctx *ctx, void *nccl_comm) {
    if (!ctx) return CGRT_ERR_INVALID;
    if (!nccl_comm) return CGRT_OK;
    if (!ctx->grid_built) FAIL(CGRT_ERR_INVALID, "build the grid first");
    CK(cudaSetDevice(ctx->device));
    CKS(join_update(ctx));
    return allreduce_on(ctx, nccl_comm, ctx->stream);  // asynchronous, ordered on the ctx stream
}


// The peer block holds the accumulators of a fixed hitpoint set; under SPPM the visible-point count changes every round.
#define SPPM_NO_PEER "multi-GPU SPPM exchanges over NCCL (cgrt_set_comm); the peer exchange is not supported (its block is sized for a fixed hitpoint count)"
int cgrt_peer_export(cgrt_ctx *ctx, void *handle128) {
    if (!ctx || !handle128) return CGRT_ERR_INVALID;
    if (ctx->sppm) FAIL(CGRT_ERR_INVALID, SPPM_NO_PEER);
    if (!ctx->grid_built) FAIL(CGRT_ERR_INVALID, "build the grid first");
    if (ctx->cfg.update_mode == 0) FAIL(CGRT_ERR_INVALID, "the per-photon update is not shard-invariant (one GPU only)");
    if (ctx->peer.block) FAIL(CGRT_ERR_INVALID, "peer block already exported");
    CK(cudaSetDevice(ctx->device));
    CKS(join_update(ctx));
    CK(cudaStreamSynchronize(ctx->stream));
    cgrt_ctx::Peer &P = ctx->peer;
    const size_t elem = acc_elem(ctx);
    P.acc_bytes = (((size_t)ctx->nhp * 4 * elem) + 255) & ~(size_t)255;
    if (P.acc_bytes == 0) P.acc_bytes = 256;
    P.bytes = 2 * P.acc_bytes + 2 * CGRT_MAX_PEERS * sizeof(int) + 256;
    // a plain cudaMalloc block: pool (cudaMallocAsync) memory cannot be exported
    if (cudaMalloc(&P.block, P.bytes) != cudaSuccess) { P = cgrt_ctx::Peer(); cudaGetLastError(); FAIL(CGRT_ERR_CUDA, "out of device memory for the peer block"); }
    CK(cudaMemset(P.block, 0, P.bytes));
    // carry over what has been accumulated so far (normally nothing)
    CK(cudaMemcpy(P.block, ctx->acc, (size_t)ctx->nhp * 4 * elem, cudaMemcpyDeviceToDevice));
    ctx->acc = P.block;
    PeerBlob b;
    memset(&b, 0, sizeof b);
    CK(cudaIpcGetMemHandle(&b.handle, P.block));
    b.pid = (uint64_t)getpid(); b.ptr = (uint64_t)(uintptr_t)P.block; b.bytes = P.bytes; b.acc_bytes = P.acc_bytes;
    b.device = ctx->device; b.nhp = (int32_t)ctx->nhp; b.accum_mode = ctx->cfg.accum_mode; b.magic = 0x43475250;
    memcpy(handle128, &b, sizeof b);
    return CGRT_OK;
}

int cgrt_peer_attach(cgrt_ctx *ctx, int rank, int world, const void *handles) {
    if (!ctx || !handles || world < 1 || world > CGRT_MAX_PEERS || rank < 0 || rank >= world) return CGRT_ERR_INVALID;
    if (ctx->sppm) FAIL(CGRT_ERR_INVALID, SPPM_NO_PEER);
    cgrt_ctx::Peer &P = ctx->peer;
    if (!P.block) FAIL(CGRT_ERR_INVALID, "cgrt_peer_export first");
    if (P.attached) FAIL(CGRT_ERR_INVALID, "peers already attached");
    CK(cudaSetDevice(ctx->device));
    const PeerBlob *B = reinterpret_cast<const PeerBlob *>(handles);
    for (int g = 0; g < world; g++) {
        if (B[g].magic != 0x43475250) FAIL(CGRT_ERR_INVALID, "not a peer handle");
        if (B[g].nhp != (int32_t)ctx->nhp || B[g].accum_mode != ctx->cfg.accum_mode || B[g].acc_bytes != P.acc_bytes)
            FAIL(CGRT_ERR_INVALID, "peer " + std::to_string(g) + " holds a different hitpoint set or accumulator type");
    }
    if (B[rank].ptr != (uint64_t)(uintptr_t)P.block) FAIL(CGRT_ERR_INVALID, "handles[rank] is not this context's own handle");
    for (int g = 0; g < world; g++) {
        if (g == rank) { P.base[g] = P.block; continue; }
        if (B[g].pid == (uint64_t)getpid()) {  // another context of this process: peer access, the pointer is valid as it is
            if (B[g].device != ctx->device) {
                int can = 0;
                CK(cudaDeviceCanAccessPeer(&can, ctx->device, B[g].device));
                if (!can) FAIL(CGRT_ERR_CUDA, "no peer access between devices " + std::to_string(ctx->device) + " and " + std::to_string(B[g].device));
                cudaError_t e = cudaDeviceEnablePeerAccess(B[g].device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); FAIL(CGRT_ERR_CUDA, "cudaDeviceEnablePeerAccess failed"); }
                cudaGetLastError();
            }
            P.base[g] = reinterpret_cast<char *>((uintptr_t)B[g].ptr);
        } else {
            void *q = nullptr;
            cudaError_t e = cudaIpcOpenMemHandle(&q, B[g].handle, cudaIpcMemLazyEnablePeerAccess);
            if (e != cudaSuccess) { cudaGetLastError(); FAIL(CGRT_ERR_CUDA, std::string("cudaIpcOpenMemHandle: ") + cudaGetErrorString(e)); }
            P.base[g] = reinterpret_cast<char *>(q);
            P.ipc[g] = true;
        }
    }
    P.rank = rank; P.world = world; P.round = 0; P.parity = 0; P.attached = true;
    return CGRT_OK;
}

int cgrt_set_comm(cgrt_ctx *ctx, void *nccl_comm, int world) {
    if (!ctx || world < 1) return CGRT_ERR_INVALID;
    if (nccl_comm && ctx->sppm) FAIL(CGRT_ERR_INVALID, "multi-GPU SPPM: attach the communicator before cgrt_set_sppm");
    if (nccl_comm && ctx->cfg.update_mode == 0) FAIL(CGRT_ERR_INVALID, "the per-photon update is not shard-invariant (one GPU only)");
    if (nccl_comm && !nccl_api().ok) FAIL(CGRT_ERR_NCCL, "NCCL is not available: " + nccl_api().why);
    CKS(join_update(ctx));
    ctx->comm = nccl_comm;
    ctx->comm_world = nccl_comm ? world : 1;
    return CGRT_OK;
}

int cgrt_comm_unique_id(void *id128) {
    NcclApi &N = nccl_api();
    if (!id128) return CGRT_ERR_INVALID;
    if (!N.ok) return CGRT_ERR_NCCL;
    return N.GetUniqueId((NcclUniqueId *)id128) == 0 ? CGRT_OK : CGRT_ERR_NCCL;
}
int cgrt_comm_init_rank(int device, int rank, int world, const void *id128, void **comm) {
    NcclApi &N = nccl_api();
    if (!id128 || !comm || world < 1 || rank < 0 || rank >= world) return CGRT_ERR_INVALID;
    if (!N.ok) return CGRT_ERR_NCCL;
    if (cudaSetDevice(device) != cudaSuccess) return CGRT_ERR_NO_DEVICE;
    NcclUniqueId id;
    memcpy(&id, id128, sizeof id);
    return N.CommInitRank(comm, world, id, rank) == 0 ? CGRT_OK : CGRT_ERR_NCCL;
}
int cgrt_comm_init_all(int n, const int *devices, void **comms) {
    NcclApi &N = nccl_api();
    if (n < 1 || !comms) return CGRT_ERR_INVALID;
    if (!N.ok) return CGRT_ERR_NCCL;
    return N.CommInitAll(comms, n, devices) == 0 ? CGRT_OK : CGRT_ERR_NCCL;
}
int cgrt_comm_destroy(void *comm) {
    NcclApi &N = nccl_api();
    if (!comm) return CGRT_OK;
    if (!N.ok) return CGRT_ERR_NCCL;
    return N.CommDestroy(comm) == 0 ? CGRT_OK : CGRT_ERR_NCCL;
}

// Tile-sharded eye pass, the exchange step: every rank contributes the records of its rows; all ranks end up with the same union (rank
// order = row order, so the union is in creation order; the grid's sort key makes the order irrelevant anyway).
int cgrt_allgather_hitpoints(cgrt_ctx *ctx, void *nccl_comm, int world) {
    if (!ctx || world < 1) return CGRT_ERR_INVALID;
    if (ctx->sppm && !ctx->sppm_traced) FAIL(CGRT_ERR_INVALID, "multi-GPU SPPM: all-gather between cgrt_sppm_eye_pass and cgrt_build_grid");
    if (ctx->grid_built) FAIL(CGRT_ERR_INVALID, "grid already built");
    if (!nccl_comm || world == 1) return CGRT_OK;
    NcclApi &N = nccl_api();
    if (!N.ok) FAIL(CGRT_ERR_NCCL, "NCCL is not available: " + N.why);
    CK(cudaSetDevice(ctx->device));
    PhaseTimer timer(ctx, 10);
    long long *d_counts;
    CKS(dalloc(ctx, &d_counts, (size_t)world + 1));
    long long mine = (long long)ctx->hp_count;
    CK(cudaMemcpyAsync(d_counts + world, &mine, sizeof mine, cudaMemcpyHostToDevice, ctx->stream));
    int r = N.AllGather(d_counts + world, d_counts, 1, NCCL_INT64, nccl_comm, ctx->stream);
    if (r != 0) return nccl_fail(ctx, r, "ncclAllGather(counts)");
    std::vector<long long> counts((size_t)world);
    CK(cudaMemcpyAsync(counts.data(), d_counts, sizeof(long long) * world, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    long long cap = 0, total = 0;
    for (long long c : counts) { cap = c > cap ? c : cap; total += c; }
    if (total >= (1ll << 32)) FAIL(CGRT_ERR_CAPACITY, "more than 2^32 hitpoints");
    const size_t rec_bytes = (size_t)CGRT_HP_RECORD_DOUBLES * sizeof(double);
    // SPPM gathers every round: the buffers are sized from a capacity that only grows, so that every round asks for the same sizes
    // (the records still travel in slots of `cap`, the largest tile of this round)
    size_t slots = (size_t)(cap ? cap : 1);
    if (ctx->sppm) {
        if ((size_t)cap > ctx->gather_cap) ctx->gather_cap = (size_t)cap + (size_t)cap / 8 + 4096;
        slots = ctx->gather_cap;
    }
    double *send, *recv;
    CKS(dalloc(ctx, &send, slots * CGRT_HP_RECORD_DOUBLES));
    CKS(dalloc(ctx, &recv, slots * CGRT_HP_RECORD_DOUBLES * world));
    if (mine) CK(cudaMemcpyAsync(send, ctx->hp_rec, (size_t)mine * rec_bytes, cudaMemcpyDeviceToDevice, ctx->stream));
    if (cap) {
        r = N.AllGather(send, recv, (size_t)cap * rec_bytes, NCCL_UINT8, nccl_comm, ctx->stream);  // equal-size slots, ranks pad to the largest tile
        if (r != 0) return nccl_fail(ctx, r, "ncclAllGather(records)");
    }
    ctx->hp_count = 0;
    CKS(ensure_hp_capacity(ctx, (size_t)total));
    size_t at = 0;
    for (int k = 0; k < world; k++) {
        if (counts[k]) CK(cudaMemcpyAsync(ctx->hp_rec + at * CGRT_HP_RECORD_DOUBLES, recv + (size_t)k * cap * CGRT_HP_RECORD_DOUBLES, (size_t)counts[k] * rec_bytes,
                                         cudaMemcpyDeviceToDevice, ctx->stream));
        at += (size_t)counts[k];
    }
    unsigned int c = (unsigned int)total;
    CK(cudaMemcpyAsync(ctx->d_hp_count, &c, sizeof c, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->hp_count = c;
    ctx->launches += 2;
    CKS(dfree(ctx, send)); CKS(dfree(ctx, recv)); CKS(dfree(ctx, d_counts));
    timer.stop();
    return CGRT_OK;
}

int cgrt_round_update(cgrt_ctx *ctx) {
    if (!ctx) return CGRT_ERR_INVALID;
    if (!ctx->grid_built) FAIL(CGRT_ERR_INVALID, "build the grid first");
    CK(cudaSetDevice(ctx->device));
    CKS(join_update(ctx));
    PhaseTimer timer(ctx, 4, ctx->profiling != 0);  // asynchronous unless profiling
    unsigned int n = ctx->nhp;
    if (ctx->sppm) {  // fold the round into the pixels, in stream order: the next round's eye pass waits for it anyway
        const unsigned int npix = (unsigned int)((size_t)ctx->P.width * ctx->P.height);
        // several GPUs: every rank holds the same sorted union, so the accumulators line up and every rank folds the same sums
        if (ctx->comm) CKS(allreduce_on(ctx, ctx->comm, ctx->stream));
        if (n > 0) {
            if (ctx->cfg.accum_mode == 0)
                sppm_fold_kernel<0><<<nblk(npix, 256), 256, 0, ctx->stream>>>(npix, ctx->P.alpha, ctx->pix_start, ctx->pix_perm, ctx->acc, ctx->pix_tau, ctx->pix_r2, ctx->pix_cnt);
            else if (ctx->cfg.accum_mode == 1)
                sppm_fold_kernel<1><<<nblk(npix, 256), 256, 0, ctx->stream>>>(npix, ctx->P.alpha, ctx->pix_start, ctx->pix_perm, ctx->acc, ctx->pix_tau, ctx->pix_r2, ctx->pix_cnt);
            else
                sppm_fold_fixed_kernel<<<nblk(npix, 256), 256, 0, ctx->stream>>>(npix, ctx->P.alpha, ctx->pix_start, ctx->pix_perm, reinterpret_cast<long long *>(ctx->acc),
                                                                                 ctx->pix_tau, ctx->pix_r2, ctx->pix_cnt, ctx->d_fxerr);
            ctx->launches++;
            CK(cudaGetLastError());
        }
        timer.stop();
        return CGRT_OK;
    }
    // the tail of a round on its own stream (see cgrt_ctx::ustream); on the main stream while profiling so that its events bracket it —
    // and when an NCCL all-reduce is part of it: measured on 8 GPUs, the collective on the side stream is SLOWER than in stream order
    // (c2: 5.40 vs 4.93 ms per round, c1: 5.72 vs 5.54): NCCL's blocks cannot become resident next to the persistent emission kernel of
    // the next round (4 blocks x 114 registers fill an SM), so the all-reduce starts late on some rank and every rank waits for it
    cudaStream_t U = (ctx->profiling || ctx->comm) ? ctx->stream : ctx->ustream;
    if (U != ctx->stream) {
        CK(cudaEventRecord(ctx->ev_tail, ctx->stream));
        CK(cudaStreamWaitEvent(U, ctx->ev_tail, 0));
    }
    if (ctx->peer.attached) {
        // the exchange over peer memory fused with the update (see peer_reduce_update_kernel); always on the side stream
        cgrt_ctx::Peer &P = ctx->peer;
        timer.stop();
        const int value = ++P.round;
        PeerPtrs flags, accs;
        for (int g = 0; g < CGRT_MAX_PEERS; g++) {
            flags.p[g] = g < P.world ? P.base[g] + peer_flags_off(P) : nullptr;
            accs.p[g] = g < P.world ? P.base[g] + (size_t)P.parity * P.acc_bytes : nullptr;
        }
        peer_signal_kernel<<<1, 32, 0, ctx->stream>>>(flags, P.rank, P.world, value);
        cudaStream_t V = ctx->ustream;
        CK(cudaEventRecord(ctx->ev_tail, ctx->stream));
        CK(cudaStreamWaitEvent(V, ctx->ev_tail, 0));
        peer_wait_kernel<<<1, 32, 0, V>>>(reinterpret_cast<const int *>(P.block + peer_flags_off(P)), P.world, value, PEER_TIMEOUT_NS,
                                         reinterpret_cast<int *>(P.block + peer_err_off(P)));
        void *clear_next = P.block + (size_t)(P.parity ^ 1) * P.acc_bytes;
        if (n > 0) {
            if (ctx->cfg.accum_mode == 0) peer_reduce_update_kernel<0><<<nblk(n, 64), 64, 0, V>>>(n, ctx->P.alpha, ctx->A, accs, P.world, clear_next);
            else if (ctx->cfg.accum_mode == 1) peer_reduce_update_kernel<1><<<nblk(n, 64), 64, 0, V>>>(n, ctx->P.alpha, ctx->A, accs, P.world, clear_next);
            else peer_reduce_update_fixed_kernel<<<nblk(n, 64), 64, 0, V>>>(n, ctx->P.alpha, ctx->A, accs, P.world, reinterpret_cast<long long *>(clear_next),
                                                                            ctx->d_fxerr);
        }
        ctx->launches += 3;
        CK(cudaGetLastError());
        CK(cudaEventRecord(ctx->ev_updated, V));
        ctx->update_pending = true;
        P.parity ^= 1;
        ctx->acc = P.block + (size_t)P.parity * P.acc_bytes;  // the next round deposits into the other buffer
        return CGRT_OK;
    }
    if (ctx->comm) CKS(allreduce_on(ctx, ctx->comm, U));
    if (n > 0 && ctx->cfg.update_mode == 0) {
        // per-photon update: fold the live counts into r2 / flux / filter radii; grow the r2 table before any count can reach its end
        round_update_u1_kernel<<<nblk(n, 256), 256, 0, U>>>(n, ctx->A, reinterpret_cast<const double *>(ctx->acc), ctx->r2tab, ctx->r2cap, ctx->d_maxcnt);
        ctx->launches++;
        int maxcnt = 0;
        CK(cudaMemcpyAsync(&maxcnt, ctx->d_maxcnt, sizeof maxcnt, cudaMemcpyDeviceToHost, U));
        CK(cudaStreamSynchronize(U));
        if (maxcnt >= ctx->r2cap - 1) FAIL(CGRT_ERR_CAPACITY, "per-photon update: a hitpoint accepted more photons in one round than the r2 table holds");
        if (maxcnt > ctx->r2cap / 4) {
            CK(cudaStreamSynchronize(ctx->stream));
            int cap = ctx->r2cap;
            while (maxcnt > cap / 4 && cap < (1 << 28)) cap *= 2;
            CKS(build_r2_table(ctx, cap));
        }
    } else if (n > 0) {
        if (ctx->cfg.accum_mode == 0) round_update_kernel<0><<<nblk(n, 256), 256, 0, U>>>(n, ctx->P.alpha, ctx->A, ctx->acc);
        else if (ctx->cfg.accum_mode == 1) round_update_kernel<1><<<nblk(n, 256), 256, 0, U>>>(n, ctx->P.alpha, ctx->A, ctx->acc);
        else round_update_fixed_kernel<<<nblk(n, 256), 256, 0, U>>>(n, ctx->P.alpha, ctx->A, reinterpret_cast<long long *>(ctx->acc), ctx->d_fxerr);
        ctx->launches++;
        CK(cudaGetLastError());
    }
    if (U != ctx->stream) {
        CK(cudaEventRecord(ctx->ev_updated, U));
        ctx->update_pending = true;
    }
    timer.stop();
    return CGRT_OK;
}

int cgrt_gather_image(cgrt_ctx *ctx, double n_emitted, double *rgb, uint8_t *rgb8) {
    if (!ctx || !rgb) return CGRT_ERR_INVALID;
    if (!ctx->grid_built) FAIL(CGRT_ERR_INVALID, "build the grid first");
    CK(cudaSetDevice(ctx->device));
    CKS(join_update(ctx));
    PhaseTimer timer(ctx, 5);
    const PassParams &P = ctx->P;
    size_t npix = (size_t)P.width * P.height;
    double *d_rgb;
    uint8_t *d_rgb8 = nullptr;
    CKS(dalloc(ctx, &d_rgb, npix * 3));
    if (rgb8) CKS(dalloc(ctx, &d_rgb8, npix * 3));
    // main.cpp:256 divides by num_photon*num_threads*num_of_samples: the caller states the photons, the samples factor comes from the config
    if (ctx->sppm)
        sppm_image_kernel<<<nblk(npix, 256), 256, 0, ctx->stream>>>(P.width, P.height, n_emitted * (double)P.samples, ctx->pix_tau, ctx->pix_r2, d_rgb, d_rgb8);
    else
        image_gather_kernel<<<nblk(npix, 256), 256, 0, ctx->stream>>>(P.width, P.height, n_emitted * (double)P.samples, ctx->pix_start, ctx->pix_perm, ctx->A.hot,
                                                                      ctx->A.flux, d_rgb, d_rgb8);
    ctx->launches++;
    CK(cudaGetLastError());
    CKS(download_free(ctx, rgb, d_rgb, npix * 3));
    if (rgb8) CKS(download_free(ctx, rgb8, d_rgb8, npix * 3));
    timer.stop();
    return check_fixed(ctx);
}

// ---- stochastic progressive photon mapping --------------------------------------------------------------------------
int cgrt_set_sppm(cgrt_ctx *ctx, int mode) {
    if (!ctx) return CGRT_ERR_INVALID;
    if (mode != CGRT_SPPM_OFF && mode != CGRT_SPPM_JITTER && mode != CGRT_SPPM_CORNER) FAIL(CGRT_ERR_INVALID, "SPPM mode must be 0 (off), 1 (jitter) or 2 (corner)");
    if (!ctx->committed) FAIL(CGRT_ERR_INVALID, "commit the scene first");
    if (ctx->hp_count || ctx->grid_built) FAIL(CGRT_ERR_INVALID, "SPPM must be chosen before any eye pass or grid");
    if (mode && ctx->cfg.update_mode == 0) FAIL(CGRT_ERR_INVALID, "SPPM needs the per-round update (update_mode 1)");
    if (mode && ctx->peer.block) FAIL(CGRT_ERR_INVALID, SPPM_NO_PEER);
    CK(cudaSetDevice(ctx->device));
    CKS(dfree(ctx, ctx->pix_tau)); CKS(dfree(ctx, ctx->pix_r2)); CKS(dfree(ctx, ctx->pix_cnt));
    ctx->pix_tau = ctx->pix_r2 = nullptr;
    ctx->pix_cnt = nullptr;
    ctx->sppm = mode;
    ctx->sppm_round = 0;
    if (!mode) return CGRT_OK;
    const size_t npix = (size_t)ctx->P.width * ctx->P.height;
    CKS(dalloc(ctx, &ctx->pix_tau, npix * 4));
    CKS(dalloc(ctx, &ctx->pix_r2, npix));
    CKS(dalloc(ctx, &ctx->pix_cnt, npix));
    std::vector<double> r2(npix, ctx->P.r2_init);  // (200/height)^2, main.cpp:84,94
    CK(cudaMemsetAsync(ctx->pix_tau, 0, npix * 4 * sizeof(double), ctx->stream));
    CK(cudaMemsetAsync(ctx->pix_cnt, 0, npix * sizeof(int), ctx->stream));
    CK(cudaMemcpyAsync(ctx->pix_r2, r2.data(), npix * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return CGRT_OK;
}

int cgrt_sppm_eye_pass(cgrt_ctx *ctx, uint32_t round, int y0, int y1) {
    if (!ctx) return CGRT_ERR_INVALID;
    if (!ctx->sppm) FAIL(CGRT_ERR_INVALID, "SPPM is off: cgrt_set_sppm first");
    if (y1 < 0) y1 = ctx->P.height;
    if (y0 < 0 || y1 > ctx->P.height || y0 > y1) FAIL(CGRT_ERR_INVALID, "bad row range");
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->tstream));
    CKS(join_update(ctx));
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->grid_built) CKS(release_grid(ctx));
    ctx->sppm_traced = false;
    ctx->hp_count = 0;
    CK(cudaMemsetAsync(ctx->d_hp_count, 0, sizeof(unsigned int), ctx->stream));
    ctx->sppm_round = round;
    if (y1 > y0) CKS(eye_pass_impl(ctx, y0, y1));  // an empty tile (more ranks than rows) contributes no visible points
    ctx->sppm_traced = true;
    return CGRT_OK;
}

int cgrt_sppm_begin_round(cgrt_ctx *ctx, uint32_t round) {
    CKS(cgrt_sppm_eye_pass(ctx, round, 0, -1));
    return build_grid_impl(ctx);
}

int cgrt_sppm_download_pixels(cgrt_ctx *ctx, double *tau, double *r2, int32_t *n) {
    if (!ctx) return CGRT_ERR_INVALID;
    if (!ctx->sppm) FAIL(CGRT_ERR_INVALID, "SPPM is off: cgrt_set_sppm first");
    CK(cudaSetDevice(ctx->device));
    CKS(join_update(ctx));
    CK(cudaStreamSynchronize(ctx->stream));
    const size_t npix = (size_t)ctx->P.width * ctx->P.height;
    if (tau) {
        std::vector<double> t(npix * 4);
        CK(cudaMemcpy(t.data(), ctx->pix_tau, npix * 4 * sizeof(double), cudaMemcpyDeviceToHost));
        for (size_t p = 0; p < npix; p++) { tau[3 * p] = t[4 * p]; tau[3 * p + 1] = t[4 * p + 1]; tau[3 * p + 2] = t[4 * p + 2]; }
    }
    if (r2) CK(cudaMemcpy(r2, ctx->pix_r2, npix * sizeof(double), cudaMemcpyDeviceToHost));
    if (n) CK(cudaMemcpy(n, ctx->pix_cnt, npix * sizeof(int), cudaMemcpyDeviceToHost));
    return check_fixed(ctx);
}

// ---- multi-run averaging (average.cpp) ------------------------------------------------------------------------------
int cgrt_average_u8(cgrt_ctx *ctx, int n, const uint8_t *const *imgs, int64_t nbytes, uint8_t *out) {
    if (!ctx || n <= 0 || n > 255 || !imgs || nbytes < 0 || !out) return CGRT_ERR_INVALID;
    if (nbytes == 0) return CGRT_OK;
    CK(cudaSetDevice(ctx->device));
    uint8_t *d_in, *d_out;
    CKS(dalloc(ctx, &d_in, (size_t)n * (size_t)nbytes));
    CKS(dalloc(ctx, &d_out, (size_t)nbytes));
    for (int k = 0; k < n; k++) {
        if (!imgs[k]) FAIL(CGRT_ERR_INVALID, "null image");
        CK(cudaMemcpyAsync(d_in + (size_t)k * (size_t)nbytes, imgs[k], (size_t)nbytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    average_u8_kernel<<<nblk((size_t)nbytes, 256), 256, 0, ctx->stream>>>(d_in, n, nbytes, d_out);
    ctx->launches++;
    CK(cudaGetLastError());
    CKS(download_free(ctx, out, d_out, (size_t)nbytes));
    return dfree(ctx, d_in);
}

int cgrt_average_f64(cgrt_ctx *ctx, int n, const double *const *imgs, int64_t nvalues, double *mean, uint8_t *rgb8) {
    if (!ctx || n <= 0 || !imgs || nvalues < 0 || !mean) return CGRT_ERR_INVALID;
    if (nvalues == 0) return CGRT_OK;
    CK(cudaSetDevice(ctx->device));
    double *d_in, *d_mean;
    uint8_t *d_rgb8 = nullptr;
    CKS(dalloc(ctx, &d_in, (size_t)n * (size_t)nvalues));
    CKS(dalloc(ctx, &d_mean, (size_t)nvalues));
    if (rgb8) CKS(dalloc(ctx, &d_rgb8, (size_t)nvalues));
    for (int k = 0; k < n; k++) {
        if (!imgs[k]) FAIL(CGRT_ERR_INVALID, "null image");
        CK(cudaMemcpyAsync(d_in + (size_t)k * (size_t)nvalues, imgs[k], (size_t)nvalues * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    }
    average_f64_kernel<<<nblk((size_t)nvalues, 256), 256, 0, ctx->stream>>>(d_in, n, nvalues, d_mean, d_rgb8);
    ctx->launches++;
    CK(cudaGetLastError());
    CKS(download_free(ctx, mean, d_mean, (size_t)nvalues));
    if (rgb8) CKS(download_free(ctx, rgb8, d_rgb8, (size_t)nvalues));
    return dfree(ctx, d_in);
}

// ---- downloads -----------------------------------------------------------------------------------------------------
int cgrt_num_hitpoints(cgrt_ctx *ctx, int64_t *n) {
    if (!ctx || !n) return CGRT_ERR_INVALID;
    *n = ctx->grid_built ? ctx->nhp : ctx->hp_count;
    return CGRT_OK;
}

int cgrt_download_hitpoints(cgrt_ctx *ctx, double *pos, double *normal, double *f, double *flux, double *r2, int32_t *n, int32_t *hw, uint32_t *key,
                            uint32_t *seq) {
    if (!ctx) return CGRT_ERR_INVALID;
    if (!ctx->grid_built) FAIL(CGRT_ERR_INVALID, "build the grid first");
    size_t m = ctx->nhp;
    if (m == 0) return CGRT_OK;
    CKS(join_update(ctx));
    CK(cudaStreamSynchronize(ctx->stream));
    std::vector<HpHot> hot(m);
    std::vector<double> tmp(m * 4);
    CK(cudaMemcpy(hot.data(), ctx->A.hot, m * sizeof(HpHot), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < m; i++) {
        if (pos) { pos[3 * i] = hot[i].px; pos[3 * i + 1] = hot[i].py; pos[3 * i + 2] = hot[i].pz; }
        if (normal) { normal[3 * i] = hot[i].nx; normal[3 * i + 1] = hot[i].ny; normal[3 * i + 2] = hot[i].nz; }
        if (r2) r2[i] = hot[i].r2;
    }
    if (f) {
        CK(cudaMemcpy(tmp.data(), ctx->A.f, m * 4 * sizeof(double), cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < m; i++) { f[3 * i] = tmp[4 * i]; f[3 * i + 1] = tmp[4 * i + 1]; f[3 * i + 2] = tmp[4 * i + 2]; }
    }
    if (flux) {
        CK(cudaMemcpy(tmp.data(), ctx->A.flux, m * 4 * sizeof(double), cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < m; i++) { flux[3 * i] = tmp[4 * i]; flux[3 * i + 1] = tmp[4 * i + 1]; flux[3 * i + 2] = tmp[4 * i + 2]; }
    }
    if (n) CK(cudaMemcpy(n, ctx->A.cnt, m * sizeof(int), cudaMemcpyDeviceToHost));
    if (hw) CK(cudaMemcpy(hw, ctx->A.hw, m * 2 * sizeof(int), cudaMemcpyDeviceToHost));
    if (key) CK(cudaMemcpy(key, ctx->A.key, m * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    if (seq) CK(cudaMemcpy(seq, ctx->A.seq, m * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return check_fixed(ctx);
}

int cgrt_download_accum(cgrt_ctx *ctx, double *dflux, double *mcount) {
    if (!ctx) return CGRT_ERR_INVALID;
    if (!ctx->grid_built) FAIL(CGRT_ERR_INVALID, "build the grid first");
    size_t m = ctx->nhp;
    if (m == 0) return CGRT_OK;
    CKS(join_update(ctx));
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->cfg.accum_mode == 0) {
        std::vector<double> a(m * 4);
        CK(cudaMemcpy(a.data(), ctx->acc, m * 4 * sizeof(double), cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < m; i++) {
            if (dflux) { dflux[3 * i] = a[4 * i]; dflux[3 * i + 1] = a[4 * i + 1]; dflux[3 * i + 2] = a[4 * i + 2]; }
            if (mcount) mcount[i] = a[4 * i + 3];
        }
    } else if (ctx->cfg.accum_mode == 1) {
        std::vector<float> a(m * 4);
        CK(cudaMemcpy(a.data(), ctx->acc, m * 4 * sizeof(float), cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < m; i++) {
            if (dflux) { dflux[3 * i] = a[4 * i]; dflux[3 * i + 1] = a[4 * i + 1]; dflux[3 * i + 2] = a[4 * i + 2]; }
            if (mcount) mcount[i] = a[4 * i + 3];
        }
    } else {  // fixed point: sum q * 2^-22 and M, as the round update reads them
        std::vector<long long> a(m * 4);
        CK(cudaMemcpy(a.data(), ctx->acc, m * 4 * sizeof(long long), cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < m; i++) {
            if (dflux)
                for (int c = 0; c < 3; c++) dflux[3 * i + c] = (double)a[4 * i + c] * CGRT_FIX_INV_SCALE;
            if (mcount) mcount[i] = (double)a[4 * i + 3];
        }
    }
    return check_fixed(ctx);
}

int cgrt_download_grid(cgrt_ctx *ctx, uint32_t *cell_start) {
    if (!ctx || !cell_start) return CGRT_ERR_INVALID;
    if (!ctx->grid_built) FAIL(CGRT_ERR_INVALID, "build the grid first");
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaMemcpy(cell_start, ctx->cell_start, ((size_t)ctx->P.hashsize + 1) * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return CGRT_OK;
}

int cgrt_get_counters(cgrt_ctx *ctx, cgrt_counters *out) {
    if (!ctx || !out) return CGRT_ERR_INVALID;
    Counters c;
    CK(cudaStreamSynchronize(ctx->tstream));
    CKS(join_update(ctx));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaMemcpy(&c, ctx->d_ctr, sizeof c, cudaMemcpyDeviceToHost));
    memset(out, 0, sizeof *out);
    out->eye_segments = c.eye_segments;
    out->photon_segments = c.photon_segments;
    out->diffuse_hits = c.diffuse_hits;
    out->candidates = c.candidates;
    out->deposits = c.deposits;
    out->gathered_hits = c.gathered_hits;
    out->exact_tests = c.exact_tests;
    out->cell_groups = c.cell_groups;
    out->staged_candidates = c.staged_candidates;
    {
        TravCounters tc;
        CK(cudaMemcpy(&tc, ctx->d_tc, sizeof tc, cudaMemcpyDeviceToHost));
        out->node_visits = tc.node_visits;
        out->tri_tests = tc.tri_tests;
    }
    out->hitpoints = ctx->grid_built ? ctx->nhp : ctx->hp_count;
    out->gpu_launches = ctx->launches;
    return CGRT_OK;
}

int cgrt_set_counting(cgrt_ctx *ctx, int on) {
    if (!ctx) return CGRT_ERR_INVALID;
    ctx->counting = on != 0;
    CK(cudaMemset(ctx->d_tc, 0, sizeof(TravCounters)));
    return CGRT_OK;
}

int cgrt_set_overlap(cgrt_ctx *ctx, int on) {
    if (!ctx) return CGRT_ERR_INVALID;
    CK(cudaStreamSynchronize(ctx->tstream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->overlap = on != 0;
    ctx->auto_chunk = 0;  // two deposit tables: the chunk is sized again
    return CGRT_OK;
}

int cgrt_release_cached_memory(int device, uint64_t *bytes_released) {
    const size_t freed = arena_trim(device);
    if (bytes_released) *bytes_released = (uint64_t)freed;
    return CGRT_OK;
}

int cgrt_deposit_record_bytes(const cgrt_ctx *ctx) { return (int)deposit_rec_bytes(ctx != nullptr && compact_records(ctx)); }

int cgrt_photon_chunk(cgrt_ctx *ctx, uint64_t *photons_per_launch) {
    if (!ctx || !photons_per_launch) return CGRT_ERR_INVALID;
    *photons_per_launch = (uint64_t)(ctx->photon_chunk ? ctx->photon_chunk : ctx->auto_chunk);
    return CGRT_OK;
}

int cgrt_check_guards(cgrt_ctx *ctx, uint64_t *damaged) {
    if (!ctx || !damaged) return CGRT_ERR_INVALID;
    uint64_t bad = ctx->guard_violations;
    for (auto &g : ctx->guarded) bad += guard_damage(ctx, g.second.first, g.second.second);
    *damaged = bad;
    return CGRT_OK;
}

int cgrt_set_culling(cgrt_ctx *ctx, int on) {
    if (!ctx) return CGRT_ERR_INVALID;
    ctx->cull = on != 0;
    return CGRT_OK;
}

int cgrt_set_profiling(cgrt_ctx *ctx, int on) {
    if (!ctx) return CGRT_ERR_INVALID;
    ctx->profiling = on != 0;
    return CGRT_OK;
}

int cgrt_get_timings(cgrt_ctx *ctx, double ms[12]) {
    if (!ctx || !ms) return CGRT_ERR_INVALID;
    for (int i = 0; i < 12; i++) ms[i] = ctx->ms[i];
    return CGRT_OK;
}

}  // extern "C"
