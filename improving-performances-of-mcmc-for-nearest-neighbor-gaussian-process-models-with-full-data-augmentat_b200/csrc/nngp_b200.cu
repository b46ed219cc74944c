// nngp_b200.cu -- context management and the C-ABI entry points of libnngp_b200.so (see include/nngp_b200.h).
//
// One context = one model's graph structure resident on one B200 plus the device-resident state of one chain
// (current + proposal factor, field, residual r = L^-1 (field - beta_0)).  Only scalars and explicitly requested vectors
// cross PCIe.  There is no CPU fallback: every compute entry point needs a CUDA device.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nvtx3/nvToolsExt.h>   // header-only; a no-op unless a profiler injects its library (SURVEY.md section 5: one range per phase A-F)

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <numeric>
#include <string>
#include <thread>
#include <vector>

#include "../../include/nngp_b200.h"
#include "kernels.cuh"
#include "nngp_internal.h"

namespace nngp {

// ------------------------------------------------------------------------------------------------------------------
// errors, launch counter
// ------------------------------------------------------------------------------------------------------------------
// Kernels of several contexts of ONE process may wait for each other from inside the device (shards of one field connected with
// nngp_shard_connect_local).  CUDA's default lazy module loading loads a kernel at its first launch and may need the device to
// drain to do so: a host thread stuck in such a load while its stream's previous kernel waits for a peer whose host thread
// needs the same lock is a deadlock.  Ask for eager loading before this library makes its first CUDA call (no effect, and no
// harm, when the process has already initialised CUDA: then there is one context per process and nothing to deadlock with).
static const int g_eager_loading = (setenv("CUDA_MODULE_LOADING", "EAGER", 0), 0);
// ... which comes too late when the host process initialised CUDA before this library was loaded (e.g. a Python process that
// asked torch.cuda.is_available() first): the loading mode is fixed at cuInit.  preload_device_code() (below, after the kernels
// are declared) then loads every kernel of this library explicitly before contexts that wait for each other are connected.

static std::mutex g_err_mu;
static char g_err[1024] = "";
static thread_local char t_err[1024] = "";   // the calling thread's last message (chains run on worker threads)
static std::atomic<long long> g_launches{0};

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(t_err, sizeof(t_err), fmt, ap);
    va_end(ap);
    std::lock_guard<std::mutex> lk(g_err_mu);
    std::memcpy(g_err, t_err, sizeof(g_err));
}

struct CudaFail {};
#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e__ = (call);                                                                        \
        if (e__ != cudaSuccess) {                                                                        \
            nngp::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__));       \
            throw nngp::CudaFail();                                                                      \
        }                                                                                                \
    } while (0)
#define LAUNCHED(c) do { nngp::g_launches.fetch_add(1, std::memory_order_relaxed); (c)->launches_in_op++; } while (0)

struct NcclFail {};
struct ArgFail {};
#define REQUIRE(cond, ...)                    \
    do {                                      \
        if (!(cond)) {                        \
            nngp::set_error(__VA_ARGS__);     \
            throw nngp::ArgFail();            \
        }                                     \
    } while (0)
struct StateFail {};

// ------------------------------------------------------------------------------------------------------------------
// NCCL, resolved at run time (dlopen): the library must not pin a second copy of libnccl.so.2 next to the one a host
// process (e.g. PyTorch) may already have loaded, so nothing is linked; whichever libnccl.so.2 is resident is used.
// Only the sharded contexts need it: per-colour halo exchange (ncclSend / ncclRecv) and scalar all-reduces.
// ------------------------------------------------------------------------------------------------------------------
struct NcclApi {
    typedef struct { char internal[128]; } UniqueId;
    typedef void *Comm;
    int (*GetUniqueId)(UniqueId *) = nullptr;
    int (*CommInitRank)(Comm *, int, UniqueId, int) = nullptr;
    int (*CommDestroy)(Comm) = nullptr;
    int (*Send)(const void *, size_t, int, int, Comm, cudaStream_t) = nullptr;
    int (*Recv)(void *, size_t, int, int, Comm, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, Comm, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    bool ok = false;
};
static NcclApi g_nccl;
static const int kNcclFloat64 = 8, kNcclSum = 0;   // ncclDataType_t / ncclRedOp_t values (nccl.h)

static void nccl_load() {
    if (g_nccl.ok) return;
    void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) { set_error("cannot load libnccl.so.2: %s", dlerror()); throw NcclFail(); }
#define NCCL_SYM(field, name) *(void **)(&g_nccl.field) = dlsym(h, name); if (!g_nccl.field) { set_error("libnccl: missing %s", name); throw NcclFail(); }
    NCCL_SYM(GetUniqueId, "ncclGetUniqueId") NCCL_SYM(CommInitRank, "ncclCommInitRank") NCCL_SYM(CommDestroy, "ncclCommDestroy")
    NCCL_SYM(Send, "ncclSend") NCCL_SYM(Recv, "ncclRecv") NCCL_SYM(GroupStart, "ncclGroupStart") NCCL_SYM(GroupEnd, "ncclGroupEnd")
    NCCL_SYM(AllReduce, "ncclAllReduce") NCCL_SYM(GetErrorString, "ncclGetErrorString")
#undef NCCL_SYM
    g_nccl.ok = true;
}
#define NCK(call)                                                                                              \
    do {                                                                                                       \
        int r__ = (call);                                                                                      \
        if (r__ != 0) {                                                                                        \
            nngp::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, nngp::g_nccl.GetErrorString(r__));    \
            throw nngp::NcclFail();                                                                            \
        }                                                                                                      \
    } while (0)

// Loads every kernel of this library on the current device now (driver API, resolved with dlopen so that the library still
// loads on a machine without a driver): cuModuleEnumerateFunctions + cuFuncLoad over the module that holds the kernels
// (CUDA >= 12.4).  A no-op when the driver is too old; eager module loading (above) is then the only protection.
static void preload_device_code(int device) {
    static std::mutex mu;
    static bool done[64] = {false};
    std::lock_guard<std::mutex> lk(mu);
    if (device < 0 || device >= 64 || done[device]) return;
    done[device] = true;
    void *h = dlopen("libcuda.so.1", RTLD_NOW | RTLD_GLOBAL);
    if (!h) return;
    typedef int (*GetModuleFn)(void **, void *);
    typedef int (*CountFn)(unsigned int *, void *);
    typedef int (*EnumFn)(void **, unsigned int, void *);
    typedef int (*LoadFn)(void *);
    GetModuleFn get_module = (GetModuleFn)dlsym(h, "cuFuncGetModule");
    CountFn count = (CountFn)dlsym(h, "cuModuleGetFunctionCount");
    EnumFn enumerate = (EnumFn)dlsym(h, "cuModuleEnumerateFunctions");
    LoadFn load = (LoadFn)dlsym(h, "cuFuncLoad");
    if (!get_module || !count || !enumerate || !load) return;
    cudaFunction_t f = nullptr;
    if (cudaGetFuncBySymbol(&f, (const void *)fill_u64_kernel) != cudaSuccess || !f) { cudaGetLastError(); return; }
    void *mod = nullptr;
    if (get_module(&mod, (void *)f) != 0 || !mod) return;
    unsigned int nf = 0;
    if (count(&nf, mod) != 0 || nf == 0) return;
    std::vector<void *> fs(nf, nullptr);
    if (enumerate(fs.data(), nf, mod) != 0) return;
    int loaded = 0;
    for (void *fn : fs) if (fn && load(fn) == 0) loaded++;
    if (std::getenv("NNGP_VERBOSE")) std::fprintf(stderr, "[nngp_b200] device %d: %d / %u kernels loaded ahead of use\n", device, loaded, nf);
}

// ------------------------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------------------------
template <class T>
struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    void alloc(size_t count) {
        release();
        n = count;
        if (count) CK(cudaMalloc(&p, count * sizeof(T)));
    }
    void upload(const std::vector<T> &h, cudaStream_t s) {
        alloc(h.size());
        if (!h.empty()) CK(cudaMemcpyAsync(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, s));
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
    }
};

struct Ctx {
    int device = 0, layout = NNGP_LAYOUT_MORTON;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;    // nngp_sweep_loglik_host: the field's way back to the host overlaps the log-lik pass
    cudaEvent_t ev_copy = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    int n = 0, d = 0, m = 0, M = 0, ld = 0, n_obs = 0, covfun = 0, dt = 0, K = 0, n_levels = 0, max_col = 0;
    // ---- sharding (one spatial block of a larger field; SURVEY.md 8e) ----
    bool sharded = false;
    int world = 1, rank = 0, n_owned = 0;
    long long n_global = 0;            // sites of the whole field (= n on an unsharded context)
    NcclApi::Comm comm = nullptr;
    std::vector<int> send_ptr, recv_ptr;   // [(colour, peer)] segments of the packed halo buffers
    std::vector<int> gstart;               // processing-index range of the ghost sites of each colour
    // peer-to-peer transport: own area + the peers' areas (CUDA IPC mappings, or direct pointers inside one process)
    bool p2p = false;
    double *p2p_area = nullptr;            // [16 halo flags | 16 reduction flags | 2 x 32 reduction slots | recv values x 2 parities]
    size_t p2p_flag_off = 0, p2p_rflag_off = 16, p2p_slot_off = 32, p2p_hdr_off = 96, p2p_val_off = 112, p2p_doubles = 0, p2p_parity_stride = 0;
    unsigned int peer_stride[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // parity stride of every peer's receive values (read from its area header)
    PeerTable peers{};
    void *peer_mapped[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    unsigned long long red_epoch = 0;
    int graph_launches = 0;
    std::vector<int> send_proc;            // processing id of every entry of the send lists
    std::vector<int> send_storage_h;       // storage id of the same
    std::vector<int> btile_count;          // per colour: tiles that hold boundary sites (they come first inside the colour)
    DevBuf<unsigned long long> d_shard_state;         // [0] sweeps since connect, [1 + colour] boundary tiles done
    DevBuf<int> d_bptr;
    DevBuf<int2> d_bdst;
    long long nnz = 0;
    int n_sm = 148;
    long long launches_in_op = 0;

    // host-side structure
    std::vector<int> i2g, g2i, cstart, lvl_ptr, partial_rows;   // i2g / g2i: storage id <-> reference (0-based) id
    struct Seg { int l0, l1; bool single_block; };
    std::vector<Seg> solve_plan;
    // tiles of the sweep: runs of consecutive same-colour sites with <= 128 sites and <= 1024 CSC entries
    std::vector<int> tile_ptr;             // per colour, into d_tiles
    // 0 = PDL chain of 128x8 tiles (blocked segmented reduction, L2 eviction hints), 5 CTAs/SM, and the 6-CTAs/SM build for
    //     colours whose tile count would otherwise spill into a second wave (default; profiles/r01_explore_sweep_occupancy.txt)
    // 1 = the same chain with 5 CTAs/SM everywhere; 2 = the same tiles as plain launches (no PDL); 3 = thread per site;
    // 4 = as 0, each colour triggers its dependent only after its own wait (at most two colours resident per stream)
    int sweep_variant = 0;
    int solve_variant = 0;                 // 0 sync-free single launch, 1 level-scheduled launches
    int commit_variant = 0;                // 0 tiled transposition, 1 thread per column
    // 1 plain coalesced loads (default), 0 TMA-staged ring.  Measured on B200 (profiles/r01_explore_final.txt): the TMA ring is
    // SLOWER (44.7 vs 37.3 us at n = 1M, 128 vs 100 us at 4M, 96 vs 55 us at m = 20): the pass is bound by the latency of
    // the 8-byte field gathers, which wants 2048 resident threads per SM; a 100 KB ring leaves room for 512.
    int loglik_variant = 1;
    // 1 = a log-lik of the current factor and field right after a sweep sums the sweep's residual r instead of rebuilding it
    // (default); 0 = always the full pass (comparison)
    bool loglik_from_residual = true;
    int n_slots = 0;                       // padded length of the level-ordered row list
    int solve_ctas_per_sm = 1;             // window of the sync-free solve = n_sm * this * 256 rows
    int solve_window_ctas = 0;             // if > 0: absolute number of CTAs (overrides the per-SM setting)
    int solve_sleep_ns = 0;                // back-off between polls
    // sharded sweep: at most this many ghost CTAs (4 ghost sites in flight each) per colour launch, placed at the end of the grid (0)
    // or at its head (1).  2 GPUs x 1M sites, m = 10 (profiles/r02_shard_explore_2gpu.txt): 32 CTAs 231 us, 96: 194, 148: 186 (one
    // round of polls instead of three); at the head of the grid 194 us -- the spinning CTAs take tile slots of the first wave
    // 8 GPUs x 1M sites (profiles/r02_shard_explore_8gpu.txt): 32 CTAs 309 us, 74: 241, 148: 215, 296: 202, 592: 202
    int shard_ghost_ctas = 296;
    // 0 end of the grid (default), 1 head, 2 = per colour: head iff tiles + ghost CTAs are co-resident.  After the prologue work of
    // round 2 (2 GPUs x 1M sites): end 167 us, auto 168, head 180
    int shard_ghost_first = 0;

    // device structure
    DevBuf<int> d_psite, d_gid, d_i2g, d_g2i, d_nn, d_colptr, d_crow, d_csrc, d_zpos, d_lvl_rows, d_lvl_ptr, d_lm, d_optr, d_oidx, d_cstart,
        d_partial_rows, d_nbad;
    // prediction (new sites appended after n0 observed ones): level-ordered, warp-padded list of the NEW rows only
    int pred_n0 = -1, pred_slots = 0, pred_levels = 0;
    DevBuf<int> d_pred_rows;
    DevBuf<double> d_frec;                 // device-side record store of the last chain_run: n_frec x n, column-major
    // regressors of the Gaussian model (nngp_regressors_set): design matrices resident in HBM
    int reg_p = -1, reg_q = 0;             // ncol(X$X) (-1 = none set); 1 + length(X$locs) (0 = no location-level regressors)
    std::vector<int> reg_xlocs;            // 0-based columns of X$X listed in X$locs
    DevBuf<double> d_Xa;                   // cbind(1, X$X): n_obs x (p+1), column-major, observation order
    DevBuf<double> d_Xl;                   // cbind(1, X$X[hctam_scol_1, X$locs]): n x q, column-major, storage order
    DevBuf<double> d_B;                    // sparse_chol %*% d_Xl of the current factor (sparse_chol_X_locs)
    DevBuf<double> d_yobs, d_robs, d_coef, d_atb_part, d_atb_out;
    int frec_rows = 0;
    DevBuf<double> d_mtab;
    bool matern_table = true;              // tabulate the Matern kernel per factor build (false: evaluate K_nu per pair)
    DevBuf<double> d_locs, d_tl, d_linv[2], d_valT, d_pd, d_nobs, d_ymx, d_S, d_field, d_newfield, d_r, d_tmp1, d_tmp2, d_io,
        d_zbuf, d_partials, d_scalars, d_flush;
    DevBuf<SweepParams> d_sp;
    DevBuf<int> d_send_storage, d_recv_proc;
    DevBuf<int4> d_ginfo;
    DevBuf<unsigned long long> d_shard_tl;   // development aid: per-colour time stamps of one sharded sweep (nngp_shard_timeline)
    bool shard_tl_on = false;
    DevBuf<double> d_sendbuf, d_recvbuf;
    DevBuf<unsigned char> d_owned;         // per storage id: 1 = owned row (reductions skip ghost rows)
    DevBuf<int4> d_tiles;
    DevBuf<unsigned char> d_cloc;          // per tile (padded to 1024): local site id of every CSC entry, 255 = padding
    DevBuf<int> d_rows_padded, d_ticket;
    DevBuf<int> d_nn_lvl, d_lpos;          // triangular solve: neighbour table in row-list (DAG level) order; position of every row in the list
    DevBuf<double> d_linv_lvl[2];          // ... and the factor values in the same order, written by the factor build next to d_linv
    bool level_copy = true;
    int factor_variant = 0;                // 0 = thread per row everywhere (default), 1 = warp-per-row kernel where it exists (m = 20)
    DevBuf<unsigned long long> d_solve_tl;   // development aid: per-chunk completion times of the sync-free solve
    bool solve_tl_on = false;
    double *h_pinned = nullptr;       // 64 doubles of pinned scratch for scalar results
    double *h_stage = nullptr;        // pinned staging for vectors (n doubles at least)
    size_t h_stage_n = 0;

    int cur = 0;                      // which linv buffer is the current factor (slot 0); the other one is the proposal
    // d_r = linv[cur] (d_field - r_beta0): set by refresh_r and kept by the sweeps that follow it (they patch r with the same beta_0);
    // cleared on entry to every ABI call that is not known to leave d_field, d_r, linv[cur] and cur alone (get_ctx)
    bool r_valid = false;
    double r_beta0 = 0.0;
    bool have_factor[2] = {false, false};
    bool committed = false;           // valT / pd correspond to linv[cur]
    bool have_field = false, have_obs = false, have_newfield = false;
    bool can_sweep = true;            // false: created without a colouring (prediction context)
    bool can_solve = true;            // false: sharded context created without the whole field's DAG levels
    // sharded triangular solve: two solution buffers inside the peer-mapped area (peers store ghost values straight into them)
    size_t p2p_x_off = 0, p2p_x_stride = 0, p2p_tab_off = 0;
    unsigned int peer_x_off[8] = {0, 0, 0, 0, 0, 0, 0, 0}, peer_x_stride[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    unsigned long long solve_epoch = 0;
    DevBuf<int> d_sxptr;
    DevBuf<int2> d_sxdst;
    std::vector<int> recv_storage;    // storage id of every ghost site, receive order
    double n_obs_global = -1.0;       // observations of the whole field (sharded contexts: all-reduced on first use)
    CovConst last_cc{};
    bool have_cc = false;
    unsigned long long sweep_counter = 0;
    cudaGraphExec_t sweep_graph = nullptr;
    bool use_graph = true;

    double *linv_slot(int slot) { return d_linv[slot == NNGP_SLOT_CURRENT ? cur : 1 - cur].p; }
    bool &have_slot(int slot) { return have_factor[slot == NNGP_SLOT_CURRENT ? cur : 1 - cur]; }
};

static std::mutex g_ctx_mu;
static std::vector<Ctx *> g_ctx;

// keep_r: the calling entry point leaves the residual's validity as it is (reads only, or sets it itself after a sweep); every
// other entry point may change the field, the residual or the current factor, so it forgets that r is current
static Ctx *get_ctx(const int *id, bool keep_r = false) {
    REQUIRE(id != nullptr, "null ctx_id");
    std::lock_guard<std::mutex> lk(g_ctx_mu);
    REQUIRE(*id >= 0 && *id < (int)g_ctx.size() && g_ctx[*id] != nullptr, "unknown context id %d", *id);
    Ctx *c = g_ctx[*id];
    if (!keep_r) c->r_valid = false;
    return c;
}

static void use(Ctx *c) { CK(cudaSetDevice(c->device)); }

static int grid_for(Ctx *c, long long work, int block, int per_sm = 8) {
    long long b = (work + block - 1) / block;
    long long cap = (long long)c->n_sm * per_sm;
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (int)b;
}

static void ensure_stage(Ctx *c, size_t count) {
    if (c->h_stage_n >= count) return;
    if (c->h_stage) cudaFreeHost(c->h_stage);
    c->h_stage = nullptr;
    c->h_stage_n = 0;
    CK(cudaMallocHost(&c->h_stage, count * sizeof(double)));
    c->h_stage_n = count;
}

// Is `p` page-locked host memory (cudaMallocHost / nngp_host_alloc / cudaHostRegister)?  Then the DMA engine can read or
// write it directly and the staging copy is skipped.
static bool is_pinned(const void *p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
}

// multi-threaded memcpy between pageable caller memory and the pinned staging buffer (a single thread moves ~8 GB/s,
// which made the staging copy of an 8 MB vector the largest term of an end-to-end step)
static void par_memcpy(void *dst, const void *src, size_t bytes) {
    const size_t chunk = (size_t)1 << 20;
    const long long nchunks = (long long)((bytes + chunk - 1) / chunk);
#pragma omp parallel for schedule(static) if (nchunks >= 4)
    for (long long k = 0; k < nchunks; k++) {
        const size_t off = (size_t)k * chunk;
        std::memcpy((char *)dst + off, (const char *)src + off, std::min(chunk, bytes - off));
    }
}

// host vector (reference order) -> device vector (internal order)
static void upload_site_vector(Ctx *c, const double *host, double *dev) {
    if (is_pinned(host)) {
        CK(cudaMemcpyAsync(c->d_io.p, host, sizeof(double) * c->n, cudaMemcpyHostToDevice, c->stream));
    } else {
        ensure_stage(c, c->n);
        par_memcpy(c->h_stage, host, sizeof(double) * c->n);
        CK(cudaMemcpyAsync(c->d_io.p, c->h_stage, sizeof(double) * c->n, cudaMemcpyHostToDevice, c->stream));
    }
    gather_f64_kernel<<<grid_for(c, c->n, 256), 256, 0, c->stream>>>(dev, c->d_io.p, c->d_i2g.p, c->n);
    LAUNCHED(c);
    if (is_pinned(host)) CK(cudaStreamSynchronize(c->stream));   // the caller may reuse its buffer as soon as we return
}

// device vector (internal order) -> host vector (reference order)
static void download_site_vector(Ctx *c, const double *dev, double *host) {
    gather_f64_kernel<<<grid_for(c, c->n, 256), 256, 0, c->stream>>>(c->d_io.p, dev, c->d_g2i.p, c->n);
    LAUNCHED(c);
    if (is_pinned(host)) {
        CK(cudaMemcpyAsync(host, c->d_io.p, sizeof(double) * c->n, cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        return;
    }
    ensure_stage(c, c->n);
    CK(cudaMemcpyAsync(c->h_stage, c->d_io.p, sizeof(double) * c->n, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    par_memcpy(host, c->h_stage, sizeof(double) * c->n);
}

static uint32_t morton2(uint32_t x, uint32_t y) {
    auto spread = [](uint32_t v) {
        v &= 0xffffu;
        v = (v | (v << 8)) & 0x00ff00ffu;
        v = (v | (v << 4)) & 0x0f0f0f0fu;
        v = (v | (v << 2)) & 0x33333333u;
        v = (v | (v << 1)) & 0x55555555u;
        return v;
    };
    return spread(x) | (spread(y) << 1);
}

static CovConst make_cov(Ctx *c, const double *cp, int ncp) {
    CovConst cc{};
    cc.mtab = nullptr;
    cc.linv_lvl = nullptr; cc.lpos = nullptr; cc.nsl = 0;
    cc.covfun = c->covfun;
    cc.d = c->d;
    cc.dt = c->dt;
    const bool matern = c->covfun >= NNGP_MATERN_ISOTROPIC;
    int n_range;
    switch (c->covfun) {
        case NNGP_EXPONENTIAL_SCALEDIM: case NNGP_MATERN_SCALEDIM: n_range = c->d; break;
        case NNGP_EXPONENTIAL_SPACETIME: case NNGP_MATERN_SPACETIME: n_range = 2; break;
        default: n_range = 1;
    }
    REQUIRE(ncp == 2 + n_range + (matern ? 1 : 0), "covparms has %d entries, covfun %d with d=%d needs %d", ncp, c->covfun, c->d,
            2 + n_range + (matern ? 1 : 0));
    cc.variance = cp[0];
    cc.nugget = cp[ncp - 1] * cp[0];
    cc.smooth = matern ? cp[ncp - 2] : 0.0;
    cc.normcon = matern ? cc.variance / (std::pow(2.0, cc.smooth - 1.0) * std::tgamma(cc.smooth)) : 0.0;
    for (int k = 0; k < 4; k++) cc.range[k] = 1.0;
    switch (c->covfun) {
        case NNGP_EXPONENTIAL_SCALEDIM: case NNGP_MATERN_SCALEDIM:
            for (int k = 0; k < c->d; k++) cc.range[k] = cp[1 + k];
            break;
        case NNGP_EXPONENTIAL_SPACETIME: case NNGP_MATERN_SPACETIME:
            for (int k = 0; k < c->d - 1; k++) cc.range[k] = cp[1];
            cc.range[c->d - 1] = cp[2];
            break;
        default:
            for (int k = 0; k < 4; k++) cc.range[k] = cp[1];
    }
    return cc;
}

// ------------------------------------------------------------------------------------------------------------------
// device ops (all asynchronous on c->stream unless they return a scalar)
// ------------------------------------------------------------------------------------------------------------------
template <bool MATERN>
static void launch_factor(Ctx *c, double *linv, const CovConst &cc) {
    const int n = c->n, ld = c->ld, M = c->M;
    bool specialised = false;
    const int blk = 128, grd = (n + blk - 1) / blk;
#define FACTOR_CASE(MM, DD)                                                                                              \
    if (!specialised && M == MM && c->dt == DD) {                                                                                        \
        vecchia_factor_reg_kernel<MM, DD, MATERN><<<grd, blk, 0, c->stream>>>(c->d_nn.p, c->d_tl.p, linv, n, ld, cc, c->d_nbad.p); \
        specialised = true;                                                                                              \
    }
    FACTOR_CASE(6, 2)
    FACTOR_CASE(6, 3)
    FACTOR_CASE(11, 2)
    FACTOR_CASE(11, 3)
    if (!specialised && M == 21 && (c->dt == 2 || c->dt == 3) && c->factor_variant == 1) {   // m = 20: one warp per row (see kernels.cuh; measured option)
        const size_t smem = sizeof(double) * ((MATERN ? 8 * MTS_SEGS : 0) + 8 * 21 * 21 + 21 * 32) + sizeof(int) * 21 * 32;
        const int blocks = std::max(1, std::min((n + 31) / 32, c->n_sm * 2));
        if (c->dt == 2) {
            CK(cudaFuncSetAttribute(vecchia_factor_warp_kernel<21, 2, MATERN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            vecchia_factor_warp_kernel<21, 2, MATERN><<<blocks, 256, smem, c->stream>>>(c->d_nn.p, c->d_tl.p, linv, n, ld, cc, c->d_nbad.p);
        } else {
            CK(cudaFuncSetAttribute(vecchia_factor_warp_kernel<21, 3, MATERN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            vecchia_factor_warp_kernel<21, 3, MATERN><<<blocks, 256, smem, c->stream>>>(c->d_nn.p, c->d_tl.p, linv, n, ld, cc, c->d_nbad.p);
        }
        LAUNCHED(c);
        return;
    }
    if (!specialised && M == 21 && c->dt == 2) {   // thread per row, 231-entry triangle: all 255 registers and spills to L1 beyond (comparison)
        vecchia_factor_reg_kernel<21, 2, MATERN, 1><<<grd, blk, 0, c->stream>>>(c->d_nn.p, c->d_tl.p, linv, n, ld, cc, c->d_nbad.p);
        specialised = true;
    }
#undef FACTOR_CASE
    if (specialised) {
        LAUNCHED(c);
        const int np = M <= 24 ? 0 : (int)c->partial_rows.size();   // partial rows ride along in the main launch
        if (np > 0) {
            vecchia_factor_generic_kernel<24, MATERN><<<(np + blk - 1) / blk, blk, 0, c->stream>>>(c->d_nn.p, c->d_tl.p, linv, c->d_partial_rows.p, np, ld, M, cc, c->d_nbad.p);
            LAUNCHED(c);
        }
        return;
    }
    if (M <= 8) vecchia_factor_generic_kernel<8, MATERN><<<grd, blk, 0, c->stream>>>(c->d_nn.p, c->d_tl.p, linv, nullptr, n, ld, M, cc, c->d_nbad.p);
    else if (M <= 16) vecchia_factor_generic_kernel<16, MATERN><<<grd, blk, 0, c->stream>>>(c->d_nn.p, c->d_tl.p, linv, nullptr, n, ld, M, cc, c->d_nbad.p);
    else if (M <= 24) vecchia_factor_generic_kernel<24, MATERN><<<grd, blk, 0, c->stream>>>(c->d_nn.p, c->d_tl.p, linv, nullptr, n, ld, M, cc, c->d_nbad.p);
    else vecchia_factor_generic_kernel<32, MATERN><<<grd, blk, 0, c->stream>>>(c->d_nn.p, c->d_tl.p, linv, nullptr, n, ld, M, cc, c->d_nbad.p);
    LAUNCHED(c);
}

static void op_factor_build(Ctx *c, int slot, const CovConst &cc_in) {
    CovConst cc = cc_in;
    cc.mtab = nullptr;
    if (c->covfun >= NNGP_MATERN_ISOTROPIC && c->matern_table) {
        if (c->d_mtab.n == 0) c->d_mtab.alloc((size_t)MT_SEGS * 8);
        matern_table_kernel<<<(MT_SEGS + 15) / 16, 128, 0, c->stream>>>(c->d_mtab.p, cc.smooth, cc.normcon);
        LAUNCHED(c);
        cc.mtab = c->d_mtab.p;
    }
    CK(cudaMemsetAsync(c->d_nbad.p, 0, 2 * sizeof(int), c->stream));
    transform_locs_kernel<<<grid_for(c, c->n, 256), 256, 0, c->stream>>>(c->d_locs.p, c->d_tl.p, c->n, cc);
    LAUNCHED(c);
    double *linv = c->linv_slot(slot);
    if (c->level_copy && c->d_lpos.p) {
        cc.linv_lvl = c->d_linv_lvl[slot == NNGP_SLOT_CURRENT ? c->cur : 1 - c->cur].p;
        cc.lpos = c->d_lpos.p;
        cc.nsl = c->n_slots;
    }
    if (c->covfun >= NNGP_MATERN_ISOTROPIC) launch_factor<true>(c, linv, cc);
    else launch_factor<false>(c, linv, cc);
    CK(cudaGetLastError());
    c->have_slot(slot) = true;
    if (slot == NNGP_SLOT_CURRENT) c->committed = false;
}

#define DISPATCH_MT(M, CALL)          \
    switch (M) {                      \
        case 6: { constexpr int MT = 6; CALL; } break;   \
        case 11: { constexpr int MT = 11; CALL; } break; \
        case 21: { constexpr int MT = 21; CALL; } break; \
        default: { constexpr int MT = 0; CALL; } break;  \
    }

static const int kReduceBlocks = 148 * 8;

// sharded field: every rank holds the partial sums of its owned rows / observations; the scalars are summed over ranks
static void allreduce_scalars(Ctx *c, int off, int count);
static int op_halo_exchange(Ctx *c, int col);

template <int MT, int STAGES>
static bool launch_loglik_tma(Ctx *c, const double *linv, const double *field, double shift, int *blocks_out) {
    const size_t smem = (size_t)STAGES * MT * 256 * 12 + 64;
    CK(cudaFuncSetAttribute(loglik_tma_kernel<MT, STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));   // per device
    const int per_sm = std::max(1, (int)((size_t)220 * 1024 / smem));
    const int blocks = std::max(1, std::min(c->n_sm * per_sm, (c->n + 255) / 256));
    loglik_tma_kernel<MT, STAGES><<<blocks, 256, smem, c->stream>>>(c->d_nn.p, linv, field, shift, c->n, c->ld, c->sharded ? c->d_owned.p : nullptr, reinterpret_cast<double2 *>(c->d_partials.p));
    *blocks_out = blocks;
    return true;
}

// partial sums -> d_scalars[off..off+1].  allow_residual: the caller accepts the sums taken from the sweep's residual when it is
// current for exactly this factor, field and beta_0 (an unsharded context); they differ from the full pass by the rounding the
// sweep's incremental updates of r accumulated
static void op_loglik_sums(Ctx *c, const double *linv, const double *field, double shift, int scal_off, bool allow_residual) {
    int blocks = std::min(kReduceBlocks, (c->n + 255) / 256);
    if (allow_residual && c->loglik_from_residual && !c->sharded && c->r_valid && linv == c->d_linv[c->cur].p && field == c->d_field.p &&
        std::memcmp(&shift, &c->r_beta0, sizeof(double)) == 0) {
        loglik_residual_kernel<<<blocks, 256, 0, c->stream>>>(linv, c->d_r.p, c->n, reinterpret_cast<double2 *>(c->d_partials.p),
                                                              reinterpret_cast<unsigned int *>(c->d_ticket.p + 1), c->d_scalars.p + scal_off);
        LAUNCHED(c);
        return;
    }
    bool done = false;
    if (c->loglik_variant == 0) {   // TMA-staged ring (specialised neighbour counts only)
        if (c->M == 6) done = launch_loglik_tma<6, 4>(c, linv, field, shift, &blocks);
        else if (c->M == 11) done = launch_loglik_tma<11, 3>(c, linv, field, shift, &blocks);
        else if (c->M == 21) done = launch_loglik_tma<21, 2>(c, linv, field, shift, &blocks);
    }
    if (!done) {
        DISPATCH_MT(c->M, (loglik_partial_kernel<MT><<<blocks, 256, 0, c->stream>>>(c->d_nn.p, linv, field, shift, c->n, c->ld, c->M, c->sharded ? c->d_owned.p : nullptr, reinterpret_cast<double2 *>(c->d_partials.p))));
    }
    LAUNCHED(c);
    reduce_partials_kernel<2><<<1, 1024, 0, c->stream>>>(c->d_partials.p, blocks, c->d_scalars.p + scal_off);
    LAUNCHED(c);
    allreduce_scalars(c, scal_off, 2);
}

static void op_spmv(Ctx *c, const double *linv, const double *v, double shift, double *out) {
    DISPATCH_MT(c->M, (spmv_rows_kernel<MT><<<grid_for(c, c->n, 256), 256, 0, c->stream>>>(c->d_nn.p, linv, v, shift, c->n, c->ld, c->M, out)));
    LAUNCHED(c);
}

// the level-ordered copy of the factor that `linv` points to (nullptr: none kept, or the option is off)
static const double *level_linv(Ctx *c, const double *linv) {
    if (!c->level_copy || !c->d_lpos.p) return nullptr;
    if (linv == c->d_linv[0].p) return c->d_linv_lvl[0].p;
    if (linv == c->d_linv[1].p) return c->d_linv_lvl[1].p;
    return nullptr;
}

// x = solve(linv, b); optional y = shift + scale * x
static void op_sptrsv(Ctx *c, const double *linv, const double *b, double *x, double *y, double shift, double scale) {
    if (c->sharded && c->world > 1) {
        // One spatial block of a larger field: every rank solves its owned rows, in the order of the whole field's DAG levels, with
        // the same synchronisation-free kernel; a ghost parent is awaited like a local one, because its owner stores the value
        // straight into this rank's solution buffer over NVLink.  Two buffers alternate: buffer e & 1 serves solve e and is
        // re-armed ("pending" everywhere) at the start of solve e - 1; the all-reduce that closes every solve keeps any rank from
        // starting solve e + 1 -- and storing into a peer's buffer -- before every rank has finished solve e.
        if (!c->p2p || !c->can_solve) { set_error("triangular solves on a sharded field need the peer-to-peer transport (nngp_shard_p2p_connect / nngp_shard_connect_local) and the whole field's DAG levels (global_level of nngp_ctx_create_sharded)"); throw StateFail(); }
        const unsigned long long e = c->solve_epoch++;
        unsigned long long *xs = reinterpret_cast<unsigned long long *>(c->p2p_area + c->p2p_x_off + (size_t)(e & 1ull) * c->p2p_x_stride);
        unsigned long long *xs_next = reinterpret_cast<unsigned long long *>(c->p2p_area + c->p2p_x_off + (size_t)((e + 1ull) & 1ull) * c->p2p_x_stride);
        CK(cudaMemsetAsync(c->d_ticket.p, 0, sizeof(int), c->stream));
        fill_u64_kernel<<<grid_for(c, c->n, 256), 256, 0, c->stream>>>(xs_next, NNGP_SOLVE_SENTINEL, c->n);
        LAUNCHED(c);
        ShardSolve ss{};
        ss.peers = c->peers;
        ss.sxptr = c->d_sxptr.p;
        ss.sxdst = c->d_sxdst.p;
        for (int h = 0; h < c->world; h++) ss.x_off[h] = c->peer_x_off[h] + (unsigned int)(e & 1ull) * c->peer_x_stride[h];
        if (c->n_slots > 0) {
            const int want = c->solve_window_ctas > 0 ? c->solve_window_ctas : c->n_sm * c->solve_ctas_per_sm;
            const int blocks = std::max(1, std::min((c->n_slots + 255) / 256, want));
            const double *lv = level_linv(c, linv);
            if (lv) { DISPATCH_MT(c->M, (sptrsv_syncfree_kernel<MT, true, true><<<blocks, 256, 0, c->stream>>>(c->d_nn_lvl.p, lv, c->d_rows_padded.p, c->n_slots, b, xs, y, shift, scale, c->n_slots, c->M, c->d_ticket.p, c->d_nbad.p + 1, (unsigned int)c->solve_sleep_ns, ss))); }
            else { DISPATCH_MT(c->M, (sptrsv_syncfree_kernel<MT, true><<<blocks, 256, 0, c->stream>>>(c->d_nn.p, linv, c->d_rows_padded.p, c->n_slots, b, xs, y, shift, scale, c->ld, c->M, c->d_ticket.p, c->d_nbad.p + 1, (unsigned int)c->solve_sleep_ns, ss))); }
            LAUNCHED(c);
        }
        allreduce_scalars(c, 60, 1);   // barrier: every rank has finished this solve (and its stores into the peers' buffers)
        shard_solve_ghosts_kernel<<<grid_for(c, c->n, 256), 256, 0, c->stream>>>(xs, c->d_owned.p, c->n, x, y, shift, scale);
        LAUNCHED(c);
        return;
    }
    if (c->solve_variant == 0) {
        CK(cudaMemsetAsync(c->d_ticket.p, 0, sizeof(int), c->stream));
        fill_u64_kernel<<<grid_for(c, c->n, 256), 256, 0, c->stream>>>(reinterpret_cast<unsigned long long *>(x), NNGP_SOLVE_SENTINEL, c->n);
        LAUNCHED(c);
        const int want = c->solve_window_ctas > 0 ? c->solve_window_ctas : c->n_sm * c->solve_ctas_per_sm;
        const int blocks = std::max(1, std::min((c->n_slots + 255) / 256, want));
        const double *lv = level_linv(c, linv);
        const int slot0 = 0;
        const int blocks_rest = std::max(1, std::min((c->n_slots - slot0 + 255) / 256, want));
        if (lv) { DISPATCH_MT(c->M, (sptrsv_syncfree_kernel<MT, false, true><<<blocks_rest, 256, 0, c->stream>>>(c->d_nn_lvl.p, lv, c->d_rows_padded.p, c->n_slots, b, reinterpret_cast<unsigned long long *>(x), y, shift, scale, c->n_slots, c->M, c->d_ticket.p, c->d_nbad.p + 1, (unsigned int)c->solve_sleep_ns, ShardSolve{}, slot0, c->solve_tl_on ? c->d_solve_tl.p : nullptr))); }
        else { DISPATCH_MT(c->M, (sptrsv_syncfree_kernel<MT><<<blocks, 256, 0, c->stream>>>(c->d_nn.p, linv, c->d_rows_padded.p, c->n_slots, b, reinterpret_cast<unsigned long long *>(x), y, shift, scale, c->ld, c->M, c->d_ticket.p, c->d_nbad.p + 1, (unsigned int)c->solve_sleep_ns, ShardSolve{}))); }
        LAUNCHED(c);
        return;
    }
    for (const auto &s : c->solve_plan) {
        if (s.single_block) {
            sptrsv_multilevel_kernel<<<1, 1024, 0, c->stream>>>(c->d_nn.p, linv, c->d_lvl_rows.p, c->d_lvl_ptr.p, s.l0, s.l1, b, x, y, shift, scale, c->ld, c->M);
        } else {
            const int lo = c->lvl_ptr[s.l0], hi = c->lvl_ptr[s.l0 + 1];
            sptrsv_level_kernel<<<(hi - lo + 255) / 256, 256, 0, c->stream>>>(c->d_nn.p, linv, c->d_lvl_rows.p, lo, hi, b, x, y, shift, scale, c->ld, c->M);
        }
        LAUNCHED(c);
    }
}

static void op_commit(Ctx *c) {
    const int n_tiled = c->sharded ? c->n_owned : c->n;   // tiles cover the owned sites; ghost columns follow in processing order
    if (c->commit_variant == 0) {
        const int nt = c->tile_ptr[c->K];   // every tile of every colour
        if (nt > 0) {
            transpose_tile2_kernel<128><<<nt, 128, 0, c->stream>>>(c->d_tiles.p, c->d_colptr.p, c->d_csrc.p, c->d_cloc.p, c->d_linv[c->cur].p, c->d_valT.p, c->d_pd.p);
            LAUNCHED(c);
        }
    } else {
        transpose_values_kernel<<<grid_for(c, n_tiled, 256), 256, 0, c->stream>>>(c->d_colptr.p, c->d_csrc.p, c->d_linv[c->cur].p, 0, n_tiled, c->d_valT.p, c->d_pd.p);
        LAUNCHED(c);
    }
    if (n_tiled < c->n) {   // values of the ghost sites' local columns (the halo apply patches r along them)
        transpose_values_kernel<<<grid_for(c, c->n - n_tiled, 256), 256, 0, c->stream>>>(c->d_colptr.p, c->d_csrc.p, c->d_linv[c->cur].p, n_tiled, c->n, c->d_valT.p, c->d_pd.p);
        LAUNCHED(c);
    }
    c->committed = true;
}

static ShardConst shard_const(Ctx *c) {
    ShardConst sc{};
    sc.peers = c->peers;
    sc.bptr = c->d_bptr.p;
    sc.bdst = c->d_bdst.p;
    sc.ginfo = c->d_ginfo.p;
    sc.tl = c->shard_tl_on ? c->d_shard_tl.p : nullptr;
    sc.state = c->d_shard_state.p;
    sc.err = c->d_nbad.p + 1;
    sc.world = c->world; sc.rank = c->rank; sc.K = c->K;
    sc.val_off = (unsigned int)c->p2p_val_off;
    for (int h = 0; h < 8; h++) sc.peer_stride[h] = c->peer_stride[h];
    return sc;
}

// One launch per colour.  Unsharded field or a sharded one with the peer-to-peer transport: a chain of programmatic
// dependent launches (colour c+1's r-independent prologue overlaps colour c); with the peer-to-peer transport the same kernel
// also pushes the boundary values to the peers and applies the ghost values that arrive (gibbs_tile2_kernel<.., SHARD>).
// Returns the number of kernels launched.
static int launch_sweep_colors(Ctx *c) {
    const bool fused_halo = c->sharded && c->p2p && c->world > 1;
    const ShardConst sc = fused_halo ? shard_const(c) : ShardConst{};
    int launched = 0;
    for (int col = 0; col < c->K; col++) {
        if (c->sweep_variant == 3 && !c->sharded) {
            const int q0 = c->cstart[col], q1 = c->cstart[col + 1];
            if (q1 > q0) {
                gibbs_color_kernel<<<(q1 - q0 + 255) / 256, 256, 0, c->stream>>>(c->d_colptr.p, c->d_crow.p, c->d_valT.p, c->d_pd.p, c->d_nobs.p, c->d_S.p, c->d_zpos.p, c->d_gid.p, c->d_psite.p, c->d_zbuf.p, c->d_sp.p, c->d_field.p, c->d_r.p, q0, q1);
                launched++;
            }
            continue;
        }
        const int t0 = c->tile_ptr[col], nt = c->tile_ptr[col + 1] - t0;
        ShardColour cl{};
        int grid = nt;
        if (fused_halo) {
            const int W = c->world;
            cl.n_tiles = nt;
            cl.n_btiles = c->btile_count[col];
            cl.g0 = c->recv_ptr[(size_t)col * W];
            cl.g1 = c->recv_ptr[(size_t)(col + 1) * W];
            cl.col = col;
            const int ng = cl.g1 - cl.g0;
            const int n_gcta = ng > 0 ? std::min(c->shard_ghost_ctas, (ng + 3) / 4) : 0;   // ghost CTAs: one warp per ghost site, 4 warps per CTA
            grid += n_gcta;
            // at the head of the grid the ghost CTAs are resident, with their columns and old values loaded, when the peers' values
            // land; that only pays when they do not push tiles of this colour into a second wave (auto: head iff everything fits)
            const int slots = c->n_sm * ((nt > 5 * c->n_sm && nt <= 6 * c->n_sm) ? 6 : 5);
            cl.ghost_first = c->shard_ghost_first == 2 ? (nt + n_gcta <= slots ? 1 : 0) : c->shard_ghost_first;
        }
        if (grid == 0) continue;
        const bool pdl = c->sweep_variant != 2 && !(c->sharded && !fused_halo);
        cudaLaunchConfig_t lc = {};
        lc.gridDim = dim3(grid);
        lc.blockDim = dim3(128);
        lc.stream = c->stream;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        lc.attrs = at;
        lc.numAttrs = (pdl && launched > 0) ? 1 : 0;   // the first colour of a sweep is an ordinary launch: it must see the counter update
#define NNGP_T2_ARGS (const int4 *)(c->d_tiles.p + t0), t0, (const int *)c->d_colptr.p, (const int *)c->d_crow.p, (const unsigned char *)c->d_cloc.p, (const double *)c->d_valT.p, (const double *)c->d_pd.p, (const double *)c->d_nobs.p, (const double *)c->d_S.p, (const int *)c->d_zpos.p, (const int *)c->d_gid.p, (const int *)c->d_psite.p, (const double *)c->d_zbuf.p, (const SweepParams *)c->d_sp.p, c->d_field.p, c->d_r.p, sc, cl
        // a colour with slightly more tiles than 5 CTAs/SM can hold (a 6 % tail wave that costs a whole extra gather -> sum ->
        // scatter round) runs the 6-CTAs/SM build (80 registers) so that all its tiles are co-resident
        const bool six = (c->sweep_variant == 0 || c->sweep_variant == 4) && nt > 5 * c->n_sm && nt <= 6 * c->n_sm;
        if (fused_halo && c->shard_tl_on) {   // development aid: the time-stamped build
            CK(cudaLaunchKernelEx(&lc, gibbs_tile2_kernel<128, true, 5, 2, true, true, true>, NNGP_T2_ARGS));
        } else if (fused_halo) {
            if (six) CK(cudaLaunchKernelEx(&lc, gibbs_tile2_kernel<128, true, 6, 2, true>, NNGP_T2_ARGS));
            else CK(cudaLaunchKernelEx(&lc, gibbs_tile2_kernel<128, true, 5, 2, true>, NNGP_T2_ARGS));
        } else if (!pdl) {
            CK(cudaLaunchKernelEx(&lc, gibbs_tile2_kernel<128, false, 5, 2>, NNGP_T2_ARGS));
        } else if (c->sweep_variant == 4) {   // as 0, dependents triggered after the wait (see LATE in kernels.cuh)
            if (six) CK(cudaLaunchKernelEx(&lc, gibbs_tile2_kernel<128, true, 6, 2, false, true>, NNGP_T2_ARGS));
            else CK(cudaLaunchKernelEx(&lc, gibbs_tile2_kernel<128, true, 5, 2, false, true>, NNGP_T2_ARGS));
        } else {
            if (six) CK(cudaLaunchKernelEx(&lc, gibbs_tile2_kernel<128, true, 6, 2>, NNGP_T2_ARGS));
            else CK(cudaLaunchKernelEx(&lc, gibbs_tile2_kernel<128, true, 5, 2>, NNGP_T2_ARGS));
        }
#undef NNGP_T2_ARGS
        launched++;
        if (c->sharded && !fused_halo) launched += op_halo_exchange(c, col);
    }
    advance_sweep_kernel<<<1, 32, 0, c->stream>>>(c->d_sp.p, (unsigned long long)c->n_global, fused_halo ? c->d_shard_state.p : nullptr);
    return launched + 1;
}

// n_sweeps sweeps over all colours; scalar parameters are read from d_sp.  Nothing in the sequence depends on host-side values
// (the NCCL transport excepted), so one sweep is captured once and replayed as a CUDA graph: K + 1 plain launches per sweep were
// CPU-submission bound.
static void op_sweeps(Ctx *c, int n_sweeps) {
    if (n_sweeps <= 0) return;
    const bool graphable = c->use_graph && !(c->sharded && c->world > 1 && !c->p2p);
    for (int s = 0; s < n_sweeps; s++) {
        int nl;
        if (graphable) {
            if (!c->sweep_graph) {
                cudaGraph_t g;
                CK(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
                c->graph_launches = launch_sweep_colors(c);
                CK(cudaStreamEndCapture(c->stream, &g));
                CK(cudaGraphInstantiate(&c->sweep_graph, g, 0));
                CK(cudaGraphDestroy(g));
            }
            CK(cudaGraphLaunch(c->sweep_graph, c->stream));
            nl = c->graph_launches;
        } else {
            nl = launch_sweep_colors(c);
            CK(cudaGetLastError());
        }
        g_launches.fetch_add(nl, std::memory_order_relaxed);
        c->launches_in_op += nl;
    }
}

static void set_sweep_params(Ctx *c, double beta0, double log_scale, double log_noise_variance, int rng_mode, double seed) {
    SweepParams *sp = reinterpret_cast<SweepParams *>(c->h_pinned + 32);
    sp->beta0 = beta0;
    sp->e_ls = std::exp(-log_scale);
    sp->e_ln = std::exp(-log_noise_variance);
    sp->sweep_counter = c->sweep_counter;
    sp->z_offset = 0;
    const unsigned long long s = (unsigned long long)(long long)seed;
    sp->key0 = (unsigned int)(s & 0xffffffffull);
    sp->key1 = (unsigned int)(s >> 32) ^ 0x5eed5eedu;
    sp->rng_mode = rng_mode;
    CK(cudaMemcpyAsync(c->d_sp.p, sp, sizeof(SweepParams), cudaMemcpyHostToDevice, c->stream));
}

static void fetch_scalars(Ctx *c, int count) {
    CK(cudaMemcpyAsync(c->h_pinned, c->d_scalars.p, sizeof(double) * count, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
}

// the sync-free solve raises a device flag instead of spinning forever on a corrupted structure
static void check_solve_flag(Ctx *c) {
    int flag = 0;
    CK(cudaMemcpyAsync(c->h_pinned + 9, c->d_nbad.p + 1, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    std::memcpy(&flag, c->h_pinned + 9, sizeof(int));
    if (flag == 2) {
        unsigned long long dbg[4] = {0, 0, 0, 0};
        if (c->d_shard_state.p) cudaMemcpy(dbg, c->d_shard_state.p, sizeof(dbg), cudaMemcpyDeviceToHost);
        int sdbg[3] = {0, 0, 0};
        cudaMemcpy(sdbg, c->d_nbad.p + 3, sizeof(sdbg), cudaMemcpyDeviceToHost);
        set_error("sharded field: rank %d timed out waiting for a peer's halo value / reduction flag (a rank died or fell out of step); last halo wait recorded: colour %llu, ghost slot %llu, sweep %llu (this rank is at sweep %llu); last solve wait recorded: row %d for site %d in chunk %d",
                  c->rank, dbg[1] + 1, dbg[2], dbg[3], dbg[0], sdbg[0], sdbg[1], sdbg[2]);
        throw NcclFail();
    }
    if (flag) {
        int dbg[3] = {0, 0, 0};
        cudaMemcpy(dbg, c->d_nbad.p + 3, sizeof(dbg), cudaMemcpyDeviceToHost);
        set_error("triangular solve: dependency wait timed out (corrupted neighbour structure, or a peer of a sharded field that never delivered): rank %d, row (storage id) %d waited for site %d in chunk %d; owned = %d / %d",
                  c->rank, dbg[0], dbg[1], dbg[2], c->sharded && c->d_owned.p ? 1 : 0, c->n);
        throw CudaFail();
    }
}

static double ll_from_sums(Ctx *c, double sum_log, double sum_sq, double log_scale) {
    return sum_log - (double)c->n_global * 0.5 * log_scale - 0.5 * sum_sq / std::exp(log_scale);
}

static void op_obs_sq(Ctx *c, const double *fnew, const double *f, int scal_off) {
    const int blocks = std::min(kReduceBlocks, (c->n_obs + 255) / 256);
    obs_sq_partial_kernel<<<blocks, 256, 0, c->stream>>>(c->d_lm.p, c->d_ymx.p, fnew, f, c->n_obs, reinterpret_cast<double2 *>(c->d_partials.p));
    LAUNCHED(c);
    reduce_partials_kernel<2><<<1, 1024, 0, c->stream>>>(c->d_partials.p, blocks, c->d_scalars.p + scal_off);
    LAUNCHED(c);
    allreduce_scalars(c, scal_off, 2);
}

static void op_beta0_sums(Ctx *c, int scal_off) {
    const int blocks = std::min(kReduceBlocks, (c->n + 255) / 256);
    DISPATCH_MT(c->M, (beta0_partial_kernel<MT><<<blocks, 256, 0, c->stream>>>(c->d_nn.p, c->d_linv[c->cur].p, c->d_field.p, c->n, c->ld, c->M, c->sharded ? c->d_owned.p : nullptr, reinterpret_cast<double2 *>(c->d_partials.p))));
    LAUNCHED(c);
    reduce_partials_kernel<2><<<1, 1024, 0, c->stream>>>(c->d_partials.p, blocks, c->d_scalars.p + scal_off);
    LAUNCHED(c);
    allreduce_scalars(c, scal_off, 2);
}

static void allreduce_scalars(Ctx *c, int off, int count) {
    if (c->sharded && c->world > 1 && c->p2p) {
        c->red_epoch++;
        allreduce_p2p_kernel<<<1, 32, 0, c->stream>>>(c->peers, c->d_scalars.p + off, count, c->world, c->rank, c->p2p_slot_off, c->p2p_rflag_off, c->red_epoch, c->d_nbad.p + 1, c->d_scalars.p + off);
        LAUNCHED(c);
        return;
    }
    if (!c->sharded || c->world == 1 || !c->comm) return;   // without a communicator the caller sums the per-rank partials
    NCK(g_nccl.AllReduce(c->d_scalars.p + off, c->d_scalars.p + off, (size_t)count, kNcclFloat64, kNcclSum, c->comm, c->stream));
}

// halo exchange for colour `col` (0-based) of a sharded field over NCCL (the fallback transport; the peer-to-peer transport is
// fused into the sweep kernel): pack, one send/recv group, apply.  Returns the number of kernels launched.
static int op_halo_exchange(Ctx *c, int col) {
    if (!c->sharded || c->world == 1) return 0;
    if (!c->comm) { set_error("this sharded context has no transport: connect its peers (nngp_shard_p2p_connect / nngp_shard_connect_local), give it an NCCL id, or drive it with the nngp_shard_* colour-stepping entry points"); throw StateFail(); }
    const int W = c->world;
    const int s0 = c->send_ptr[(size_t)col * W], s1 = c->send_ptr[(size_t)(col + 1) * W];
    const int r0 = c->recv_ptr[(size_t)col * W], r1 = c->recv_ptr[(size_t)(col + 1) * W];
    int launched = 0;
    if (s1 > s0) {
        halo_pack_kernel<<<(s1 - s0 + 255) / 256, 256, 0, c->stream>>>(c->d_send_storage.p, c->d_field.p, s0, s1, c->d_sendbuf.p);
        launched++;
    }
    NCK(g_nccl.GroupStart());
    for (int h = 0; h < W; h++) {
        if (h == c->rank) continue;
        const int a = c->send_ptr[(size_t)col * W + h], b = c->send_ptr[(size_t)col * W + h + 1];
        const int ra = c->recv_ptr[(size_t)col * W + h], rb = c->recv_ptr[(size_t)col * W + h + 1];
        if (b > a) NCK(g_nccl.Send(c->d_sendbuf.p + a, (size_t)(b - a), kNcclFloat64, h, c->comm, c->stream));
        if (rb > ra) NCK(g_nccl.Recv(c->d_recvbuf.p + ra, (size_t)(rb - ra), kNcclFloat64, h, c->comm, c->stream));
    }
    NCK(g_nccl.GroupEnd());
    if (r1 > r0) {
        halo_apply_kernel<<<(r1 - r0 + 255) / 256, 256, 0, c->stream>>>(c->d_recv_proc.p, c->d_recvbuf.p, r0, r1, c->d_colptr.p, c->d_crow.p, c->d_valT.p, c->d_psite.p, c->d_field.p, c->d_r.p);
        launched++;
    }
    return launched;
}

static void ensure_zbuf(Ctx *c, size_t count) {
    if (c->d_zbuf.n >= count) return;
    CK(cudaStreamSynchronize(c->stream));
    c->d_zbuf.alloc(count);
    if (c->sweep_graph) { cudaGraphExecDestroy(c->sweep_graph); c->sweep_graph = nullptr; }  // zbuf pointer is baked in
}

static void refresh_r(Ctx *c, double beta0) {
    op_spmv(c, c->d_linv[c->cur].p, c->d_field.p, beta0, c->d_r.p);
    c->r_valid = !c->sharded;   // a sharded field's ghost rows are not kept current by its own sweep
    c->r_beta0 = beta0;
}

// ---- dense products with the resident design matrices (update_Gaussian.R:226-246) ----
static const int kAtbRowsPerChunk = 4096;

// host_out (qa x qb, column-major) = A^T B over `rows` rows; returns after the result is on the host
static void op_atb(Ctx *c, const double *A, int qa, const double *B, int qb, int rows, double *host_out) {
    const int chunks = std::max(1, (rows + kAtbRowsPerChunk - 1) / kAtbRowsPerChunk);
    const size_t qq = (size_t)qa * qb;
    if (c->d_atb_part.n < qq * chunks) c->d_atb_part.alloc(qq * chunks);
    if (c->d_atb_out.n < qq) c->d_atb_out.alloc(qq);
    dim3 grid((qa + 15) / 16, (qb + 15) / 16, chunks);
    atb_partial_kernel<<<grid, 256, 0, c->stream>>>(A, qa, B, qb, rows, kAtbRowsPerChunk, c->d_atb_part.p);
    LAUNCHED(c);
    atb_reduce_kernel<<<grid_for(c, (long long)qq, 256), 256, 0, c->stream>>>(c->d_atb_part.p, chunks, (int)qq, c->d_atb_out.p);
    LAUNCHED(c);
    CK(cudaMemcpyAsync(host_out, c->d_atb_out.p, qq * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
}

// in place: lower Cholesky factor of the symmetric positive definite q x q matrix A (column-major), upper part zeroed;
// false when a pivot falls below 1e-13 of its diagonal entry
static bool dense_chol_lower(std::vector<double> &A, int q) {
    for (int j = 0; j < q; j++) {
        const double ajj = A[(size_t)j + (size_t)q * j];
        double dj = ajj;
        for (int k = 0; k < j; k++) dj -= A[(size_t)j + (size_t)q * k] * A[(size_t)j + (size_t)q * k];
        if (!(dj > 1e-13 * ajj)) return false;                        // numerically singular (e.g. collinear regressors)
        dj = std::sqrt(dj);
        A[(size_t)j + (size_t)q * j] = dj;
        for (int i = j + 1; i < q; i++) {
            double v = A[(size_t)i + (size_t)q * j];
            for (int k = 0; k < j; k++) v -= A[(size_t)i + (size_t)q * k] * A[(size_t)j + (size_t)q * k];
            A[(size_t)i + (size_t)q * j] = v / dj;
        }
        for (int i = 0; i < j; i++) A[(size_t)i + (size_t)q * j] = 0.0;
    }
    return true;
}

// inverse of a symmetric positive definite matrix through its Cholesky factor: P = L L^T, P^-1 = L^-T L^-1
static bool dense_spd_inverse(const std::vector<double> &P, int q, std::vector<double> &inv) {
    std::vector<double> L(P);
    if (!dense_chol_lower(L, q)) return false;
    std::vector<double> Li((size_t)q * q, 0.0);                       // L^-1, lower triangular, column by column
    for (int j = 0; j < q; j++) {
        Li[(size_t)j + (size_t)q * j] = 1.0 / L[(size_t)j + (size_t)q * j];
        for (int i = j + 1; i < q; i++) {
            double v = 0.0;
            for (int k = j; k < i; k++) v -= L[(size_t)i + (size_t)q * k] * Li[(size_t)k + (size_t)q * j];
            Li[(size_t)i + (size_t)q * j] = v / L[(size_t)i + (size_t)q * i];
        }
    }
    inv.assign((size_t)q * q, 0.0);
    for (int a = 0; a < q; a++)
        for (int b = 0; b <= a; b++) {
            double v = 0.0;
            for (int k = a; k < q; k++) v += Li[(size_t)k + (size_t)q * a] * Li[(size_t)k + (size_t)q * b];
            inv[(size_t)a + (size_t)q * b] = v;
            inv[(size_t)b + (size_t)q * a] = v;
        }
    return true;
}

// mu = beta_0 + X$X %*% beta (:249) enters every later step as observed_field - mu + beta_0 = y - X beta: refresh d_ymx and
// the per-site sums residuals_sum (:260)
static void op_set_beta(Ctx *c, const double *beta) {
    CK(cudaMemcpyAsync(c->d_coef.p, beta, sizeof(double) * c->reg_p, cudaMemcpyHostToDevice, c->stream));
    obs_minus_xb_kernel<<<grid_for(c, c->n_obs, 256), 256, 0, c->stream>>>(c->d_Xa.p + c->n_obs, c->d_coef.p, c->reg_p, c->d_yobs.p, c->n_obs, c->d_ymx.p);
    LAUNCHED(c);
    site_obs_sum_kernel<<<grid_for(c, c->n, 256), 256, 0, c->stream>>>(c->d_optr.p, c->d_oidx.p, c->d_ymx.p, c->n, c->d_S.p);
    LAUNCHED(c);
    CK(cudaStreamSynchronize(c->stream));                              // `beta` may live on the caller's stack
}

// :77-83 (and after every accepted proposal :145-151, :200-206): sparse_chol_X_locs = sparse_chol %*% cbind(1, X_locs),
// beta_interweaved_covmat = solve(crossprod(.)), and the lower Cholesky factor of the latter (= t(chol(.)) in R)
static void op_interweave(Ctx *c, std::vector<double> &cov, std::vector<double> &chol_lower) {
    const int q = c->reg_q, n = c->n;
    for (int l = 0; l < q; l++) op_spmv(c, c->d_linv[c->cur].p, c->d_Xl.p + (size_t)l * n, 0.0, c->d_B.p + (size_t)l * n);
    std::vector<double> prec((size_t)q * q);
    op_atb(c, c->d_B.p, q, c->d_B.p, q, n, prec.data());
    if (!dense_spd_inverse(prec, q, cov)) { set_error("interweaving: crossprod(sparse_chol %%*%% cbind(1, X_locs)) is not positive definite (collinear location regressors?)"); throw StateFail(); }
    chol_lower = cov;
    if (!dense_chol_lower(chol_lower, q)) { set_error("interweaving: beta_interweaved_covmat is not positive definite"); throw StateFail(); }
}

static void flush_l2(Ctx *c) {
    if (c->d_flush.n == 0) c->d_flush.alloc((size_t)32 << 20);  // 256 MB of doubles
    fill_f64_kernel<<<c->n_sm * 8, 256, 0, c->stream>>>(c->d_flush.p, 1.0, c->d_flush.n);
}

static void destroy_ctx(Ctx *c) {
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->sweep_graph) cudaGraphExecDestroy(c->sweep_graph);
    if (c->comm && g_nccl.ok) g_nccl.CommDestroy(c->comm);
    for (int h = 0; h < 8; h++) if (c->peer_mapped[h]) cudaIpcCloseMemHandle(c->peer_mapped[h]);
    c->d_recvbuf.p = nullptr;
    if (c->p2p_area) cudaFree(c->p2p_area);
    c->d_shard_state.release(); c->d_bptr.release(); c->d_bdst.release(); c->d_sxptr.release(); c->d_sxdst.release();
    c->d_ginfo.release(); c->d_shard_tl.release();
    c->d_send_storage.release(); c->d_recv_proc.release(); c->d_sendbuf.release(); c->d_owned.release();
    DevBuf<int> *ib[] = {&c->d_psite, &c->d_gid, &c->d_i2g, &c->d_g2i, &c->d_nn, &c->d_colptr, &c->d_crow, &c->d_csrc, &c->d_zpos, &c->d_lvl_rows, &c->d_lvl_ptr,
                         &c->d_lm, &c->d_optr, &c->d_oidx, &c->d_cstart, &c->d_partial_rows, &c->d_nbad};
    for (auto *b : ib) b->release();
    DevBuf<double> *db[] = {&c->d_locs, &c->d_tl, &c->d_linv[0], &c->d_linv[1], &c->d_valT, &c->d_pd, &c->d_nobs, &c->d_ymx, &c->d_S,
                            &c->d_field, &c->d_newfield, &c->d_r, &c->d_tmp1, &c->d_tmp2, &c->d_io, &c->d_zbuf, &c->d_partials,
                            &c->d_scalars, &c->d_flush};
    for (auto *b : db) b->release();
    c->d_mtab.release();
    c->d_frec.release();
    c->d_Xa.release(); c->d_Xl.release(); c->d_B.release(); c->d_yobs.release(); c->d_robs.release(); c->d_coef.release(); c->d_atb_part.release(); c->d_atb_out.release();
    c->d_pred_rows.release();
    c->d_sp.release();
    c->d_tiles.release();
    c->d_rows_padded.release(); c->d_ticket.release(); c->d_cloc.release();
    c->d_nn_lvl.release(); c->d_lpos.release(); c->d_linv_lvl[0].release(); c->d_linv_lvl[1].release();
    if (c->h_pinned) cudaFreeHost(c->h_pinned);
    if (c->h_stage) cudaFreeHost(c->h_stage);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->ev_copy) cudaEventDestroy(c->ev_copy);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

}  // namespace nngp

using namespace nngp;

// every ABI function runs its body through this wrapper: exceptions never cross the C boundary
#define ABI_BEGIN try {
#define ABI_END                                                   \
    if (status) *status = NNGP_OK;                                \
    }                                                             \
    catch (const nngp::ArgFail &) { if (status) *status = NNGP_ERR_ARG; }     \
    catch (const nngp::CudaFail &) { if (status) *status = NNGP_ERR_CUDA; }   \
    catch (const nngp::StateFail &) { if (status) *status = NNGP_ERR_STATE; } \
    catch (const nngp::NcclFail &) { if (status) *status = NNGP_ERR_NCCL; } \
    catch (const std::bad_alloc &) { nngp::set_error("host allocation failed"); if (status) *status = NNGP_ERR_ALLOC; } \
    catch (...) { nngp::set_error("unexpected exception"); if (status) *status = NNGP_ERR_ARG; }
#define NEED(cond, msg) do { if (!(cond)) { nngp::set_error(msg); throw nngp::StateFail(); } } while (0)

extern "C" {

void nngp_version(int *major, int *minor) { if (major) *major = 0; if (minor) *minor = 1; }

void nngp_last_error(char *buf, const int *len) {
    if (!buf || !len || *len <= 0) return;
    std::lock_guard<std::mutex> lk(g_err_mu);
    std::strncpy(buf, g_err, (size_t)*len - 1);
    buf[*len - 1] = '\0';
}

// R's .C() hands a character vector over as char **: the message goes into the first string, which the caller has sized
// (e.g. strrep(" ", 1024)) -- writing through nngp_last_error's char * there would overwrite the pointer slot itself
void nngp_last_error_r(char **buf, const int *len) {
    if (!buf || !buf[0] || !len || *len <= 0) return;
    nngp_last_error(buf[0], len);
}

void nngp_host_alloc(const double *n_bytes, void **ptr, int *status) {
    ABI_BEGIN
    REQUIRE(n_bytes && ptr && *n_bytes >= 0, "nngp_host_alloc: bad argument");
    void *p = nullptr;
    CK(cudaMallocHost(&p, (size_t)std::max(*n_bytes, 8.0)));
    *ptr = p;
    ABI_END
}

void nngp_host_free(void **ptr, int *status) {
    ABI_BEGIN
    REQUIRE(ptr != nullptr, "nngp_host_free: null argument");
    if (*ptr) CK(cudaFreeHost(*ptr));
    *ptr = nullptr;
    ABI_END
}

void nngp_launch_count(double *count) { if (count) *count = (double)g_launches.load(); }

void nngp_device_count(int *count, int *status) {
    ABI_BEGIN
    REQUIRE(count != nullptr, "null count");
    int k = 0;
    cudaError_t e = cudaGetDeviceCount(&k);
    if (e != cudaSuccess) { k = 0; set_error("cudaGetDeviceCount: %s", cudaGetErrorString(e)); *count = 0; throw CudaFail(); }
    *count = k;
    ABI_END
}

struct ShardArgs {
    const int *owned, *global_id, *global_zpos, *global_level, *send_site, *send_ptr, *recv_site, *recv_ptr;
    int n_colors, world, rank;
    long long n_global;
    const char *comm_id;
};

static void create_ctx_impl(const int *n_, const int *d_, const int *m_, const double *locs, const int *NNarray, const int *coloring,
                            const int *n_obs_, const int *locs_match, const int *covfun_id, const int *device, const int *layout,
                            const ShardArgs *sh, int *ctx_id, int *status) {
    Ctx *c = nullptr;
    ABI_BEGIN
    REQUIRE(n_ && d_ && m_ && locs && NNarray && coloring && n_obs_ && (locs_match || *n_obs_ == 0) && covfun_id && device && layout && ctx_id, "nngp_ctx_create: null argument");
    const int n = *n_, d = *d_, m = *m_, M = m + 1, n_obs = *n_obs_;
    REQUIRE(n >= 1 && d >= 1 && d <= 4 && m >= 1 && m <= 31 && n_obs >= 0, "nngp_ctx_create: need n>=1, 1<=d<=4, 1<=m<=31 (got n=%d d=%d m=%d)", n, d, m);
    REQUIRE(*covfun_id >= 0 && *covfun_id <= 7, "unknown covfun_id %d", *covfun_id);
    REQUIRE((long long)n * M < 2147483647LL, "n*(m+1) must fit int32");
    if ((*covfun_id == NNGP_EXPONENTIAL_SPHERE || *covfun_id == NNGP_MATERN_SPHERE)) REQUIRE(d == 2, "*_sphere needs lon/lat (d=2)");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { set_error("no CUDA device: libnngp_b200 has no CPU fallback"); throw CudaFail(); }
    REQUIRE(*device >= 0 && *device < ndev, "device %d out of range (%d devices)", *device, ndev);

    const bool prof_create = std::getenv("NNGP_PROFILE_CREATE") != nullptr;
    auto t_create = std::chrono::steady_clock::now();
    auto phase = [&](const char *what) {
        if (!prof_create) return;
        const auto now = std::chrono::steady_clock::now();
        std::fprintf(stderr, "[nngp ctx_create] %-28s %8.1f ms\n", what, 1e3 * std::chrono::duration<double>(now - t_create).count());
        t_create = now;
    };
    c = new Ctx();
    c->device = *device;
    c->layout = (*layout == NNGP_LAYOUT_COLOR || *layout == NNGP_LAYOUT_COLOR_MORTON) ? *layout : NNGP_LAYOUT_MORTON;
    c->n = n; c->d = d; c->m = m; c->M = M; c->n_obs = n_obs; c->covfun = *covfun_id;
    c->dt = (*covfun_id == NNGP_EXPONENTIAL_SPHERE || *covfun_id == NNGP_MATERN_SPHERE) ? 3 : d;
    c->ld = (n + 31) / 32 * 32;
    use(c);
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, c->device));
    c->n_sm = prop.multiProcessorCount;
    CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&c->ev_copy, cudaEventDisableTiming));
    CK(cudaEventCreate(&c->ev0));
    CK(cudaEventCreate(&c->ev1));
    CK(cudaMallocHost(&c->h_pinned, 64 * sizeof(double)));

    phase("cuda stream / events");
    // ---- validate structure, colour classes ----
    // coloring all zero = "no colouring": a context that never sweeps (the joint observed ++ predicted site set of
    // mcmc_nngp_predict_field, predict.R:4-8, has none).  Internally one colour class; every sweep entry point refuses.
    std::vector<int> no_colour;
    if (!sh) {
        bool all_zero = true;
        for (int i = 0; i < n && all_zero; i++) all_zero = coloring[i] == 0;
        if (all_zero) { no_colour.assign(n, 1); coloring = no_colour.data(); c->can_sweep = false; }
    }
    int K = 0;
    for (int i = 0; i < n; i++) { REQUIRE(coloring[i] >= 1, "coloring[%d] = %d (colours are 1..K; all zero = context without sweeps)", i, coloring[i]); K = std::max(K, coloring[i]); }
    if (sh) {   // a shard sees only some of the field's colours but must walk all of them in step with its peers
        REQUIRE(sh->n_colors >= K && sh->world >= 1 && sh->rank >= 0 && sh->rank < sh->world && sh->owned && sh->global_id && sh->global_zpos && sh->send_ptr && sh->recv_ptr && sh->comm_id,
                "nngp_ctx_create_sharded: bad sharding arguments");
        K = sh->n_colors;
        c->sharded = true; c->world = sh->world; c->rank = sh->rank;
    }
    c->n_global = sh ? sh->n_global : n;
    c->K = K;
    auto is_ghost = [&](int ref) { return sh != nullptr && sh->owned[ref] == 0; };
    for (int i = 0; i < n; i++) {
        REQUIRE(NNarray[i] == i + 1, "NNarray[%d,1] must be the row itself", i + 1);
        bool seen_na = false;
        for (int j = 1; j < M; j++) {
            const int v = NNarray[(size_t)i + (size_t)n * j];
            if (v == NNGP_NA_INT) { seen_na = true; continue; }
            REQUIRE(!seen_na, "NNarray row %d has a neighbour after an NA", i + 1);
            REQUIRE(v >= 1 && v <= i, "NNarray[%d,%d] = %d is not a previous site", i + 1, j + 1, v);
        }
    }
    // The sweep kernels update all sites of a colour concurrently and patch r without atomics: that is only race-free if no
    // two sites of one colour appear in the same row (= the colouring is proper for the moral graph, initialize.R:103-110).
    // Checked here, once, instead of trusting the caller (compute-sanitizer's racecheck is not available on this pool).
    if (c->can_sweep) {
        std::vector<int> seen(K + 1, -1);
        for (int i = 0; i < n; i++) {
            for (int j = 0; j < M; j++) {
                const int v = NNarray[(size_t)i + (size_t)n * j];
                if (v == NNGP_NA_INT) continue;
                const int col = coloring[v - 1];
                REQUIRE(seen[col] != i, "coloring is not proper: row %d contains two sites of colour %d (they would be updated concurrently)", i + 1, col);
                seen[col] = i;
            }
        }
    }
    phase("validation");
    // ---- numberings ----
    // storage order: NNGP_LAYOUT_MORTON = Z-curve over all sites; NNGP_LAYOUT_COLOR[_MORTON] = colour-major (reference / Z-curve
    // order inside a colour).  processing order (sweep) = colour-major, storage order inside a colour.
    std::vector<uint32_t> key(n, 0);
    if (c->layout != NNGP_LAYOUT_COLOR) {
        double lo[2] = {INFINITY, INFINITY}, hi[2] = {-INFINITY, -INFINITY};
        const int dd = std::min(d, 2);
        for (int k = 0; k < dd; k++)
            for (int i = 0; i < n; i++) { const double x = locs[(size_t)i + (size_t)n * k]; lo[k] = std::min(lo[k], x); hi[k] = std::max(hi[k], x); }
        for (int i = 0; i < n; i++) {
            uint32_t g[2] = {0, 0};
            for (int k = 0; k < dd; k++) {
                const double ext = hi[k] - lo[k];
                double t = ext > 0 ? (locs[(size_t)i + (size_t)n * k] - lo[k]) / ext : 0.0;
                g[k] = (uint32_t)std::min(65535.0, std::max(0.0, t * 65536.0));
            }
            key[i] = morton2(g[0], g[1]);
        }
    }
    c->i2g.resize(n);
    const bool color_major_storage = (c->layout != NNGP_LAYOUT_MORTON);
    {   // stable order by (colour if colour-major, key): one sort of packed 64-bit words -- (key, reference id) for the default
        // Morton layout, (colour, key) with the id carried alongside otherwise
        if (!color_major_storage) {
            std::vector<unsigned long long> w(n);
            for (int i = 0; i < n; i++) w[i] = ((unsigned long long)key[i] << 32) | (unsigned int)i;
            std::sort(w.begin(), w.end());
            for (int q = 0; q < n; q++) c->i2g[q] = (int)(w[q] & 0xffffffffull);
        } else {
            std::iota(c->i2g.begin(), c->i2g.end(), 0);
            std::stable_sort(c->i2g.begin(), c->i2g.end(), [&](int a, int b) {
                if (coloring[a] != coloring[b]) return coloring[a] < coloring[b];
                return key[a] < key[b];
            });
        }
    }
    c->g2i.resize(n);
    for (int q = 0; q < n; q++) c->g2i[c->i2g[q]] = q;
    // processing order: storage ids sorted by colour (stable => storage order inside a colour)
    std::vector<int> psite(n), pof(n);   // psite[p] = storage id of processing site p; pof = inverse
    // (owned sites colour by colour -- inside a colour of a sharded field the boundary sites, i.e. those some peer ghosts, come
    // first so that their tiles run, and push their values to the peers, before the interior tiles; then the ghost sites)
    std::vector<unsigned char> is_boundary(n, 0);   // by reference id
    if (sh)
        for (int k = 0; k < sh->send_ptr[(size_t)K * sh->world]; k++) {
            const int ref = sh->send_site[k] - 1;
            REQUIRE(ref >= 0 && ref < n && sh->owned[ref], "send_site[%d] is not an owned local site", k + 1);
            is_boundary[ref] = 1;
        }
    {   // stable counting sort of the storage ids by bucket = (ghost, colour, interior)
        auto bucket = [&](int q) {
            const int ref = c->i2g[q];
            return (is_ghost(ref) ? 2 * K : 0) + 2 * (coloring[ref] - 1) + (is_boundary[ref] ? 0 : 1);
        };
        std::vector<int> start((size_t)4 * K + 1, 0);
        for (int q = 0; q < n; q++) start[bucket(q) + 1]++;
        for (int b = 0; b < 4 * K; b++) start[b + 1] += start[b];
        for (int q = 0; q < n; q++) psite[start[bucket(q)]++] = q;
    }
    for (int p = 0; p < n; p++) pof[psite[p]] = p;
    c->cstart.assign(K + 1, 0);
    c->gstart.assign(K + 1, 0);
    for (int i = 0; i < n; i++) (is_ghost(i) ? c->gstart : c->cstart)[coloring[i]]++;
    for (int k = 0; k < K; k++) c->cstart[k + 1] += c->cstart[k];
    c->n_owned = c->cstart[K];
    c->gstart[0] = c->n_owned;
    for (int k = 0; k < K; k++) c->gstart[k + 1] += c->gstart[k];
    // position of each site inside the reference's rnorm() hand-out order: colour 1..K, ascending reference index
    std::vector<int> zpos(n), gid(n);
    {
        if (sh) {   // Philox keys and the position in the rnorm() hand-out order refer to the WHOLE field
            for (int p = 0; p < n; p++) { const int ref = c->i2g[psite[p]]; gid[p] = sh->global_id[ref]; zpos[p] = sh->global_zpos[ref]; }
        } else {
            std::vector<int> next(c->cstart.begin(), c->cstart.end() - 1);
            std::vector<int> zg(n);
            for (int i = 0; i < n; i++) zg[i] = next[coloring[i] - 1]++;
            for (int p = 0; p < n; p++) { gid[p] = c->i2g[psite[p]]; zpos[p] = zg[gid[p]]; }
        }
    }

    phase("orderings (2 sorts)");
    // ---- row structure in storage numbering ----
    const int ld = c->ld;
    std::vector<int> nn((size_t)ld * M, -1);
    std::vector<unsigned char> is_partial(n, 0);
#pragma omp parallel for schedule(static)
    for (int q = 0; q < n; q++) {
        const int i = c->i2g[q];
        for (int j = 0; j < M; j++) {
            const int v = NNarray[(size_t)i + (size_t)n * j];
            if (v == NNGP_NA_INT) is_partial[q] = 1;
            else nn[(size_t)j * ld + q] = c->g2i[v - 1];
        }
    }
    for (int q = 0; q < n; q++) if (is_partial[q]) c->partial_rows.push_back(q);
    std::vector<double> locs_int((size_t)n * d);
#pragma omp parallel for schedule(static)
    for (int q = 0; q < n; q++)
        for (int k = 0; k < d; k++) locs_int[(size_t)q * d + k] = locs[(size_t)c->i2g[q] + (size_t)n * k];
    phase("row structure");
    // ---- transpose (CSC) structure: columns in processing order, row ids in storage numbering ----
    std::vector<int> colptr(n + 1, 0);
    for (int q = 0; q < n; q++)
        for (int j = 0; j < M; j++) { const int v = nn[(size_t)j * ld + q]; if (v >= 0) colptr[pof[v] + 1]++; }
    for (int p = 0; p < n; p++) { c->max_col = std::max(c->max_col, colptr[p + 1]); colptr[p + 1] += colptr[p]; }
    c->nnz = colptr[n];
    std::vector<int> crow(c->nnz), csrc(c->nnz);
    {
        std::vector<int> pos(colptr.begin(), colptr.end() - 1);
        for (int q = 0; q < n; q++)  // rows ascending => every column's entries are sorted by (storage) row
            for (int j = 0; j < M; j++) {
                const int v = nn[(size_t)j * ld + q];
                if (v >= 0) { const int p = pof[v]; crow[pos[p]] = q; csrc[pos[p]] = j * ld + q; pos[p]++; }
            }
    }
    phase("transpose structure");
    // ---- solve DAG levels ----
    // A sharded field solves its OWNED rows only, and every rank must walk them in the order of the WHOLE field's levels: with
    // local levels (ghost sites' rows are cut) a rank could schedule a row before an owned row it transitively depends on through
    // a peer, and the bounded window of the sync-free solve would deadlock.  Without global levels the solves are unavailable.
    std::vector<int> level;
    const bool shard_levels = sh && sh->global_level;
    c->can_solve = !sh || shard_levels;
    if (shard_levels) {
        level.assign(sh->global_level, sh->global_level + n);
        c->n_levels = 0;
        for (int i = 0; i < n; i++) { REQUIRE(level[i] >= 0, "global_level[%d] < 0", i); if (sh->owned[i]) c->n_levels = std::max(c->n_levels, level[i] + 1); }
    } else {
        c->n_levels = solve_levels(NNarray, n, m, level);
    }
    auto solved_here = [&](int ref) { return !shard_levels || sh->owned[ref]; };
    c->lvl_ptr.assign(c->n_levels + 1, 0);
    for (int i = 0; i < n; i++) if (solved_here(i)) c->lvl_ptr[level[i] + 1]++;
    for (int l = 0; l < c->n_levels; l++) c->lvl_ptr[l + 1] += c->lvl_ptr[l];
    std::vector<int> lvl_rows(c->lvl_ptr[c->n_levels]);
    {
        std::vector<int> pos(c->lvl_ptr.begin(), c->lvl_ptr.end() - 1);
        for (int q = 0; q < n; q++) if (solved_here(c->i2g[q])) lvl_rows[pos[level[c->i2g[q]]]++] = q;  // internal ids ascending inside a level
    }
    // plan: runs of narrow levels -> one single-CTA launch; wide levels -> one launch each
    for (int l = 0; l < c->n_levels;) {
        const int w = c->lvl_ptr[l + 1] - c->lvl_ptr[l];
        if (w <= 4096) {
            int l1 = l;
            while (l1 < c->n_levels && (c->lvl_ptr[l1 + 1] - c->lvl_ptr[l1]) <= 4096) l1++;
            c->solve_plan.push_back({l, l1, true});
            l = l1;
        } else {
            c->solve_plan.push_back({l, l + 1, false});
            l++;
        }
    }
    // level-ordered row list, every level padded to a warp multiple (sync-free solve)
    std::vector<int> rows_padded;
    rows_padded.reserve((size_t)n + 32 * (size_t)c->n_levels);
    for (int l = 0; l < c->n_levels; l++) {
        for (int t = c->lvl_ptr[l]; t < c->lvl_ptr[l + 1]; t++) rows_padded.push_back(lvl_rows[t]);
        while (rows_padded.size() % 32) rows_padded.push_back(-1);
    }
    c->n_slots = (int)rows_padded.size();
    phase("solve levels");
    // ---- sweep tiles: runs of consecutive same-colour sites with <= 128 sites and <= 1024 CSC entries; a tile never mixes
    // boundary and interior sites ----
    std::vector<int4> tiles;
    {
        const int T = 128, ECAP = 1024;
        // sites per BOUNDARY tile of a sharded field.  A boundary tile is on the critical path of the colour (tile -> NVLink hop -> ghost
        // patch on the peer -> next colour): nngp_shard_timeline showed the last push 5 us after the launch's wait with 128-site tiles
        // (eight gathers per thread in the crowd of the interior tiles) and 2.5 us with 4-site tiles.  2 GPUs x 1M sites: 128 sites
        // 176 us / sweep, 32: 171, 16: 158, 8: 154, 4: 152, 2: 163 (profiles/r02_shard_boundary_cycle_2gpu.txt); NNGP_BTILE_SITES overrides
        int Tb = 8;
        if (const char *e = std::getenv("NNGP_BTILE_SITES")) Tb = std::max(1, std::min(128, std::atoi(e)));
        c->tile_ptr.assign(K + 1, 0);
        c->btile_count.assign(K, 0);
        for (int col = 0; col < K; col++) {
            int s0 = c->cstart[col];
            const int send = c->cstart[col + 1];
            int bend = s0;   // end of the colour's boundary sites
            while (bend < send && is_boundary[c->i2g[psite[bend]]]) bend++;
            while (s0 < send) {
                const int lim = s0 < bend ? bend : send;
                int s1 = s0 + 1;   // at least one site (an oversize column is handled inside the kernel)
                const int Tt = s0 < bend ? Tb : T;
                while (s1 < lim && s1 - s0 < Tt && colptr[s1 + 1] - colptr[s0] <= ECAP) s1++;
                tiles.push_back(make_int4(s0, s1, colptr[s0], colptr[s1]));
                if (s0 < bend) c->btile_count[col]++;
                s0 = s1;
            }
            c->tile_ptr[col + 1] = (int)tiles.size();
        }
    }
    // local site id of every entry of a tile, one padded block of 1024 bytes per tile (blocked reduction of
    // gibbs_tile2_kernel); an oversize single-site tile does not use it
    std::vector<unsigned char> cloc((size_t)tiles.size() * 1024, (unsigned char)255);
#pragma omp parallel for schedule(static)
    for (long long t = 0; t < (long long)tiles.size(); t++) {
        const int4 tl = tiles[t];
        if (tl.w - tl.z > 1024) continue;
        for (int q = tl.x; q < tl.y; q++)
            for (int e = colptr[q]; e < colptr[q + 1]; e++) cloc[(size_t)t * 1024 + (size_t)(e - tl.z)] = (unsigned char)(q - tl.x);
    }
    phase("tiles");
    // ---- observations: lm in storage numbering (gathers of field); per-site lists / counts in processing order ----
    std::vector<int> lm(n_obs), optr(n + 1, 0), oidx(n_obs);
    for (int o = 0; o < n_obs; o++) {
        REQUIRE(locs_match[o] >= 1 && locs_match[o] <= n, "locs_match[%d] = %d out of range", o + 1, locs_match[o]);
        lm[o] = c->g2i[locs_match[o] - 1];
        optr[pof[lm[o]] + 1]++;
    }
    std::vector<double> nobs(n);
    for (int p = 0; p < n; p++) { nobs[p] = optr[p + 1]; optr[p + 1] += optr[p]; }
    {
        std::vector<int> pos(optr.begin(), optr.end() - 1);
        for (int o = 0; o < n_obs; o++) oidx[pos[pof[lm[o]]]++] = o;
    }
    phase("observations");
    // ---- upload ----
    cudaStream_t s = c->stream;
    c->d_psite.upload(psite, s); c->d_gid.upload(gid, s);
    c->d_i2g.upload(c->i2g, s); c->d_g2i.upload(c->g2i, s); c->d_nn.upload(nn, s); c->d_colptr.upload(colptr, s);
    { std::vector<int> crow_padded(crow); crow_padded.resize(crow.size() + 4, 0); c->d_crow.upload(crow_padded, s); }   // + 4: see d_valT
    c->d_csrc.upload(csrc, s); c->d_zpos.upload(zpos, s); c->d_lvl_rows.upload(lvl_rows, s);
    c->d_lvl_ptr.upload(c->lvl_ptr, s); c->d_lm.upload(lm, s); c->d_optr.upload(optr, s); c->d_oidx.upload(oidx, s);
    c->d_cstart.upload(c->cstart, s); c->d_locs.upload(locs_int, s); c->d_nobs.upload(nobs, s);
    if (!c->partial_rows.empty()) c->d_partial_rows.upload(c->partial_rows, s);
    c->d_nbad.alloc(8);   // [0] rows with a non-PD block, [1] wait timed out (1 solve, 2 halo / reduction), [3..5] which solve row waited for what
    CK(cudaMemsetAsync(c->d_nbad.p, 0, 8 * sizeof(int), s));
    c->d_ticket.alloc(2);   // [0] the triangular solve's chunk tickets, [1] the residual log-lik's CTA count (back to 0 after every launch)
    CK(cudaMemsetAsync(c->d_ticket.p, 0, 2 * sizeof(int), s));
    c->d_rows_padded.upload(rows_padded, s);
    {   // level-ordered copies for the triangular solve: static neighbour table now, factor values at every factor build
        std::vector<int> lpos(n, -1), nn_lvl((size_t)c->n_slots * M, -1);
        for (int t = 0; t < c->n_slots; t++) {
            const int q = rows_padded[t];
            if (q < 0) continue;
            lpos[q] = t;
            for (int j = 0; j < M; j++) nn_lvl[(size_t)j * c->n_slots + t] = nn[(size_t)j * ld + q];
        }
        c->d_lpos.upload(lpos, s);
        c->d_nn_lvl.upload(nn_lvl, s);
        for (int k = 0; k < 2; k++) {
            c->d_linv_lvl[k].alloc((size_t)std::max(c->n_slots, 1) * M);
            CK(cudaMemsetAsync(c->d_linv_lvl[k].p, 0, sizeof(double) * (size_t)std::max(c->n_slots, 1) * M, s));
        }
        CK(cudaStreamSynchronize(s));
    }
    c->d_tiles.upload(tiles, s);
    c->d_cloc.upload(cloc, s);
    c->d_tl.alloc((size_t)n * c->dt);
    for (int k = 0; k < 2; k++) { c->d_linv[k].alloc((size_t)ld * M); CK(cudaMemsetAsync(c->d_linv[k].p, 0, sizeof(double) * ld * M, s)); }
    c->d_valT.alloc((size_t)c->nnz + 2);
    CK(cudaMemsetAsync(c->d_valT.p + c->nnz, 0, 2 * sizeof(double), s));
    c->d_pd.alloc(n); c->d_ymx.alloc(std::max(n_obs, 1)); c->d_S.alloc(n); c->d_field.alloc(n);
    c->d_newfield.alloc(n); c->d_r.alloc(n); c->d_tmp1.alloc(n); c->d_tmp2.alloc(n); c->d_io.alloc((size_t)std::max(n, n_obs));
    c->d_zbuf.alloc(n); c->d_partials.alloc((size_t)kReduceBlocks * 4); c->d_scalars.alloc(64); c->d_sp.alloc(1);
    CK(cudaMemsetAsync(c->d_S.p, 0, sizeof(double) * n, s));
    if (sh) {
        const int W = sh->world;
        c->send_ptr.assign(sh->send_ptr, sh->send_ptr + (size_t)K * W + 1);
        c->recv_ptr.assign(sh->recv_ptr, sh->recv_ptr + (size_t)K * W + 1);
        std::vector<int> send_storage(c->send_ptr.back()), recv_proc(c->recv_ptr.back());
        c->send_proc.resize(send_storage.size());
        for (size_t k = 0; k < send_storage.size(); k++) {
            const int ref = sh->send_site[k] - 1;   // (range and ownership were checked when the boundary sites were marked)
            send_storage[k] = c->g2i[ref];
            c->send_proc[k] = pof[send_storage[k]];
        }
        c->send_storage_h = send_storage;
        for (size_t k = 0; k < recv_proc.size(); k++) {
            const int ref = sh->recv_site[k] - 1;
            REQUIRE(ref >= 0 && ref < n && !sh->owned[ref], "recv_site[%d] is not a ghost site", (int)k + 1);
            recv_proc[k] = pof[c->g2i[ref]];
        }
        REQUIRE(W <= 8, "at most 8 ranks per field");
        std::vector<unsigned char> owned_storage(n);
        for (int q = 0; q < n; q++) owned_storage[q] = sh->owned[c->i2g[q]] ? 1 : 0;
        c->d_send_storage.upload(send_storage, s);
        c->d_recv_proc.upload(recv_proc, s);
        {   // (storage id, first entry, end of the column) of every ghost site in receive order: one load in the ghost CTAs' prologue
            std::vector<int4> ginfo(std::max<size_t>(recv_proc.size(), 1), make_int4(0, 0, 0, 0));
            for (size_t k = 0; k < recv_proc.size(); k++) { const int pp = recv_proc[k]; ginfo[k] = make_int4(psite[pp], colptr[pp], colptr[pp + 1], pp); }
            c->d_ginfo.upload(ginfo, s);
        }
        c->d_owned.upload(owned_storage, s);
        c->d_sendbuf.alloc(std::max<size_t>(send_storage.size(), 1));
        // the receive values live in one plain cudaMalloc area that peers can map through CUDA IPC.  Fixed header so that every
        // rank knows where its peers' flags are: [16 halo flags | 16 reduction flags | 2 x 32 reduction slots | receive values of
        // even sweeps | receive values of odd sweeps] (two parities: a peer one sweep ahead never overwrites unread values)
        const size_t nrecv = (std::max<size_t>(recv_proc.size(), 1) + 15) / 16 * 16;
        c->p2p_parity_stride = nrecv;
        // ... | 2 solution buffers of the sharded triangular solve (n local sites each) | storage id of every ghost site (int32) ]
        c->p2p_x_off = c->p2p_val_off + 2 * nrecv;
        c->p2p_x_stride = ((size_t)n + 15) / 16 * 16;
        c->p2p_tab_off = c->p2p_x_off + 2 * c->p2p_x_stride;
        c->p2p_doubles = std::max<size_t>(c->p2p_tab_off + (recv_proc.size() + 1) / 2 + 16, (size_t)1 << 18);   // >= 2 MB: a whole allocation of its own
        CK(cudaMalloc(&c->p2p_area, c->p2p_doubles * sizeof(double)));
        CK(cudaMemsetAsync(c->p2p_area, 0, c->p2p_doubles * sizeof(double), s));
        {   // header: what a peer must know about this rank's area (read by the peers when they connect)
            unsigned long long *hdr = reinterpret_cast<unsigned long long *>(c->h_pinned + 40);
            hdr[0] = (unsigned long long)nrecv;
            hdr[1] = (unsigned long long)recv_proc.size();
            hdr[2] = (unsigned long long)c->p2p_x_off;
            hdr[3] = (unsigned long long)c->p2p_x_stride;
            hdr[4] = (unsigned long long)c->p2p_tab_off;
            CK(cudaMemcpyAsync(c->p2p_area + c->p2p_hdr_off, hdr, 5 * sizeof(unsigned long long), cudaMemcpyHostToDevice, s));
            c->recv_storage.resize(recv_proc.size());
            for (size_t k = 0; k < recv_proc.size(); k++) c->recv_storage[k] = psite[recv_proc[k]];
            if (!c->recv_storage.empty())
                CK(cudaMemcpyAsync(c->p2p_area + c->p2p_tab_off, c->recv_storage.data(), c->recv_storage.size() * sizeof(int), cudaMemcpyHostToDevice, s));
        }
        c->d_recvbuf.p = c->p2p_area + c->p2p_val_off;      // not owned by the DevBuf (released with the area)
        c->d_recvbuf.n = 0;
        ensure_stage(c, (size_t)std::max(n, n_obs));   // no page-locked allocation (a device-synchronising call) once peers may be waiting on this rank
        c->d_shard_state.alloc(4);
        CK(cudaMemsetAsync(c->d_shard_state.p, 0, 4 * sizeof(unsigned long long), s));
        CK(cudaStreamSynchronize(s));
        if (W > 1 && sh->comm_id[0] != '\0') {   // collective: every rank of the field creates its context at the same time
            nccl_load();
            NcclApi::UniqueId id;
            std::memcpy(id.internal, sh->comm_id, 128);
            NCK(g_nccl.CommInitRank(&c->comm, W, id, sh->rank));
        }
    }
    CK(cudaStreamSynchronize(s));   // host vectors go out of scope below
    phase("allocations + uploads");
    {
        std::lock_guard<std::mutex> lk(g_ctx_mu);
        int id = -1;
        for (size_t k = 0; k < g_ctx.size(); k++) if (!g_ctx[k]) { id = (int)k; break; }
        if (id < 0) { g_ctx.push_back(nullptr); id = (int)g_ctx.size() - 1; }
        g_ctx[id] = c;
        *ctx_id = id;
    }
    c = nullptr;
    ABI_END
    if (c) destroy_ctx(c);
}

void nngp_ctx_create(const int *n_, const int *d_, const int *m_, const double *locs, const int *NNarray, const int *coloring,
                     const int *n_obs_, const int *locs_match, const int *covfun_id, const int *device, const int *layout,
                     int *ctx_id, int *status) {
    create_ctx_impl(n_, d_, m_, locs, NNarray, coloring, n_obs_, locs_match, covfun_id, device, layout, nullptr, ctx_id, status);
}

void nngp_comm_unique_id(char *id128, int *status) {
    ABI_BEGIN
    REQUIRE(id128 != nullptr, "nngp_comm_unique_id: null buffer");
    nccl_load();
    NcclApi::UniqueId id;
    NCK(g_nccl.GetUniqueId(&id));
    std::memcpy(id128, id.internal, 128);
    ABI_END
}

void nngp_ctx_create_sharded(const int *n_, const int *d_, const int *m_, const double *locs, const int *NNarray, const int *coloring,
                             const int *n_colors, const int *owned, const int *global_id, const int *global_zpos, const int *global_level,
                             const double *n_global,
                             const int *n_obs_, const int *locs_match, const int *covfun_id, const int *device, const int *layout,
                             const int *world, const int *rank, const int *send_site, const int *send_ptr, const int *recv_site,
                             const int *recv_ptr, const char *comm_id128, int *ctx_id, int *status) {
    if (!n_colors || !world || !rank || !n_global) { set_error("nngp_ctx_create_sharded: null argument"); if (status) *status = NNGP_ERR_ARG; return; }
    ShardArgs sh{owned, global_id, global_zpos, global_level, send_site, send_ptr, recv_site, recv_ptr, *n_colors, *world, *rank, (long long)*n_global, comm_id128};
    create_ctx_impl(n_, d_, m_, locs, NNarray, coloring, n_obs_, locs_match, covfun_id, device, layout, &sh, ctx_id, status);
}

void nngp_ctx_destroy(const int *ctx_id, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    { std::lock_guard<std::mutex> lk(g_ctx_mu); g_ctx[*ctx_id] = nullptr; }
    destroy_ctx(c);
    ABI_END
}

void nngp_ctx_set_option(const int *ctx_id, const int *key, const int *value, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(key && value, "nngp_ctx_set_option: null argument");
    use(c);
    CK(cudaStreamSynchronize(c->stream));
    switch (*key) {
        case NNGP_OPT_SWEEP_VARIANT: REQUIRE(*value >= 0 && *value <= 4, "sweep variant must be 0..4"); c->sweep_variant = *value; break;
        case NNGP_OPT_SOLVE_VARIANT: REQUIRE(*value >= 0 && *value <= 1, "solve variant must be 0..1"); c->solve_variant = *value; break;
        case NNGP_OPT_USE_GRAPH: c->use_graph = (*value != 0); break;
        case NNGP_OPT_SOLVE_CTAS_PER_SM: REQUIRE(*value >= 1 && *value <= 8, "solve CTAs per SM must be 1..8"); c->solve_ctas_per_sm = *value; break;
        case NNGP_OPT_LOGLIK_VARIANT: REQUIRE(*value >= 0 && *value <= 1, "loglik variant must be 0..1"); c->loglik_variant = *value; break;
        case NNGP_OPT_LOGLIK_FROM_RESIDUAL: c->loglik_from_residual = (*value != 0); break;
        case NNGP_OPT_MATERN_TABLE: c->matern_table = (*value != 0); break;
        case NNGP_OPT_COMMIT_VARIANT: REQUIRE(*value >= 0 && *value <= 1, "commit variant must be 0..1"); c->commit_variant = *value; break;
        case NNGP_OPT_SOLVE_WINDOW_CTAS: REQUIRE(*value >= 0 && *value <= 4096, "solve window must be 0..4096 CTAs"); c->solve_window_ctas = *value; break;
        case NNGP_OPT_SOLVE_LEVEL_COPY: c->level_copy = (*value != 0); c->have_factor[0] = c->have_factor[1] = false; c->committed = false; break;
        case NNGP_OPT_SHARD_GHOST_CTAS: REQUIRE(*value >= 1 && *value <= 1024, "ghost CTAs must be 1..1024"); c->shard_ghost_ctas = *value; if (c->sweep_graph) { cudaGraphExecDestroy(c->sweep_graph); c->sweep_graph = nullptr; } break;
        case NNGP_OPT_SHARD_GHOST_FIRST: REQUIRE(*value >= 0 && *value <= 2, "ghost placement must be 0..2"); c->shard_ghost_first = *value; if (c->sweep_graph) { cudaGraphExecDestroy(c->sweep_graph); c->sweep_graph = nullptr; } break;
        case NNGP_OPT_FACTOR_VARIANT: REQUIRE(*value >= 0 && *value <= 1, "factor variant must be 0..1"); c->factor_variant = *value; break;
        case NNGP_OPT_SOLVE_SLEEP_NS: REQUIRE(*value >= 0 && *value <= 100000, "solve sleep must be 0..100000 ns"); c->solve_sleep_ns = *value; break;
        default: REQUIRE(false, "unknown option key %d", *key);
    }
    if (c->sweep_graph) { cudaGraphExecDestroy(c->sweep_graph); c->sweep_graph = nullptr; }
    ABI_END
}

// development aid: one sweep of a peer-to-peer connected sharded field (every rank calls it together) with six %globaltimer stamps
// per colour (see NNGP_TL_MIN / NNGP_TL_MAX in kernels.cuh); out_ns[K][6], ns relative to this rank's first stamp, -1 = never set
void nngp_shard_timeline(const int *ctx_id, const double *beta_0, const double *log_scale, const double *log_noise_variance, double *out_ns, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(beta_0 && log_scale && log_noise_variance && out_ns, "nngp_shard_timeline: null argument");
    NEED(c->sharded && c->p2p && c->world > 1 && c->have_field && c->have_obs && c->have_slot(NNGP_SLOT_CURRENT), "nngp_shard_timeline: needs a connected sharded context with factor, field and observations");
    use(c);
    const size_t cnt = (size_t)c->K * 6;
    std::vector<unsigned long long> init(cnt);
    for (size_t i = 0; i < cnt; i++) init[i] = (i % 6 == 0 || i % 6 == 2) ? ~0ull : 0ull;   // min-stamps start at +inf
    c->d_shard_tl.upload(init, c->stream);
    if (c->sweep_graph) { cudaGraphExecDestroy(c->sweep_graph); c->sweep_graph = nullptr; }
    c->shard_tl_on = true;
    if (!c->committed) op_commit(c);
    set_sweep_params(c, *beta_0, *log_scale, *log_noise_variance, NNGP_RNG_PHILOX, 1.0);
    refresh_r(c, *beta_0);
    op_sweeps(c, 1);
    c->sweep_counter += 1ull;
    c->shard_tl_on = false;
    std::vector<unsigned long long> t(cnt);
    CK(cudaMemcpyAsync(t.data(), c->d_shard_tl.p, sizeof(unsigned long long) * cnt, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    if (c->sweep_graph) { cudaGraphExecDestroy(c->sweep_graph); c->sweep_graph = nullptr; }
    unsigned long long t0 = ~0ull;
    for (size_t i = 0; i < cnt; i++) if (t[i] != 0ull && t[i] != ~0ull && t[i] < t0) t0 = t[i];
    for (size_t i = 0; i < cnt; i++) out_ns[i] = (t[i] == 0ull || t[i] == ~0ull) ? -1.0 : (double)(t[i] - t0);
    check_solve_flag(c);
    ABI_END
}

// development aid: one SpMV + triangular solve with the completion time of every 256-slot chunk of the level-ordered row list
// recorded (%globaltimer, ns, relative to the first); out_ns[k] for chunk k of the part the sync-free kernel walks, level_of_chunk[k]
// = DAG level of the chunk's first row; *n_chunks in: capacity, out: count
void nngp_solve_timeline(const int *ctx_id, double *out_ns, int *level_of_chunk, int *n_chunks, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(out_ns && level_of_chunk && n_chunks, "nngp_solve_timeline: null argument");
    NEED(!c->sharded && c->have_slot(NNGP_SLOT_CURRENT) && c->have_field, "nngp_solve_timeline: needs an unsharded context with a factor and a field");
    use(c);
    const int slot0 = 0;
    const int nc = (c->n_slots - slot0 + 255) / 256;
    REQUIRE(*n_chunks >= nc, "nngp_solve_timeline: need room for %d chunks", nc);
    c->d_solve_tl.alloc((size_t)nc + 1);
    CK(cudaMemsetAsync(c->d_solve_tl.p, 0, sizeof(unsigned long long) * ((size_t)nc + 1), c->stream));
    c->solve_tl_on = true;
    op_spmv(c, c->linv_slot(NNGP_SLOT_CURRENT), c->d_field.p, 0.0, c->d_tmp1.p);
    op_sptrsv(c, c->linv_slot(NNGP_SLOT_CURRENT), c->d_tmp1.p, c->d_tmp2.p, nullptr, 0.0, 1.0);
    c->solve_tl_on = false;
    std::vector<unsigned long long> t((size_t)nc);
    CK(cudaMemcpyAsync(t.data(), c->d_solve_tl.p, sizeof(unsigned long long) * nc, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    unsigned long long t0 = ~0ull;
    for (int k = 0; k < nc; k++) if (t[k] && t[k] < t0) t0 = t[k];
    // level of a slot: levels are padded to warps, so walk the padded level starts
    std::vector<int> slot_level((size_t)c->n_slots, 0);
    { int tpos = 0; for (int l = 0; l < c->n_levels; l++) { const int w = c->lvl_ptr[l + 1] - c->lvl_ptr[l]; const int wp = (w + 31) / 32 * 32; for (int u = 0; u < wp && tpos < c->n_slots; u++) slot_level[tpos++] = l; } }
    for (int k = 0; k < nc; k++) { out_ns[k] = t[k] ? (double)(t[k] - t0) : -1.0; level_of_chunk[k] = slot_level[(size_t)slot0 + (size_t)k * 256]; }
    *n_chunks = nc;
    ABI_END
}

void nngp_ctx_info(const int *ctx_id, int *info8, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(info8 != nullptr, "null info");
    info8[0] = c->n; info8[1] = c->m; info8[2] = c->K; info8[3] = c->n_levels; info8[4] = (int)c->nnz; info8[5] = c->max_col;
    info8[6] = c->device; info8[7] = c->layout;
    ABI_END
}

void nngp_factor_build(const int *ctx_id, const int *slot, const double *covparms, const int *n_covparms, int *n_not_pd, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(slot && covparms && n_covparms && (*slot == 0 || *slot == 1), "nngp_factor_build: bad argument");
    use(c);
    const CovConst cc = make_cov(c, covparms, *n_covparms);
    c->last_cc = cc; c->have_cc = true;
    op_factor_build(c, *slot, cc);
    int bad = 0;
    CK(cudaMemcpyAsync(c->h_pinned, c->d_nbad.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    std::memcpy(&bad, c->h_pinned, sizeof(int));
    if (n_not_pd) *n_not_pd = bad;
    ABI_END
}

void nngp_factor_get(const int *ctx_id, const int *slot, double *Linv, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(slot && Linv && (*slot == 0 || *slot == 1), "nngp_factor_get: bad argument");
    NEED(c->have_slot(*slot), "nngp_factor_get: that slot holds no factor");
    use(c);
    DevBuf<double> tmp;
    tmp.alloc((size_t)c->n * c->M);
    linv_to_host_order_kernel<<<grid_for(c, c->n, 256), 256, 0, c->stream>>>(tmp.p, c->linv_slot(*slot), c->d_g2i.p, c->n, c->ld, c->M);
    LAUNCHED(c);
    CK(cudaMemcpyAsync(Linv, tmp.p, sizeof(double) * (size_t)c->n * c->M, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    tmp.release();
    ABI_END
}

void nngp_factor_accept(const int *ctx_id, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    NEED(c->have_slot(NNGP_SLOT_PROPOSAL), "nngp_factor_accept: no proposal factor");
    use(c);
    c->cur = 1 - c->cur;
    op_commit(c);
    ABI_END
}

void nngp_factor_commit(const int *ctx_id, const int *slot, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(slot && (*slot == 0 || *slot == 1), "nngp_factor_commit: bad slot");
    NEED(c->have_slot(*slot), "nngp_factor_commit: that slot holds no factor");
    use(c);
    if (*slot == NNGP_SLOT_PROPOSAL) c->cur = 1 - c->cur;
    op_commit(c);
    ABI_END
}

void nngp_precision_diag(const int *ctx_id, double *out, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(out != nullptr, "null out");
    NEED(c->have_slot(NNGP_SLOT_CURRENT), "nngp_precision_diag: no current factor");
    use(c);
    if (!c->committed) op_commit(c);
    scatter_f64_kernel<<<grid_for(c, c->n, 256), 256, 0, c->stream>>>(c->d_tmp1.p, c->d_pd.p, c->d_psite.p, c->n);   // processing -> storage order
    LAUNCHED(c);
    download_site_vector(c, c->d_tmp1.p, out);
    ABI_END
}

void nngp_field_set(const int *ctx_id, const double *field, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(field != nullptr, "null field");
    use(c);
    upload_site_vector(c, field, c->d_field.p);
    CK(cudaStreamSynchronize(c->stream));
    c->have_field = true;
    ABI_END
}

void nngp_field_get(const int *ctx_id, double *field, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id, true);
    REQUIRE(field != nullptr, "null field");
    NEED(c->have_field, "nngp_field_get: no field on the device");
    use(c);
    download_site_vector(c, c->d_field.p, field);
    ABI_END
}

void nngp_obs_set(const int *ctx_id, const double *y_minus_xb, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(y_minus_xb != nullptr || c->n_obs == 0, "null observations");
    use(c);
    if (c->n_obs > 0) {
        ensure_stage(c, std::max(c->n_obs, c->n));
        std::memcpy(c->h_stage, y_minus_xb, sizeof(double) * c->n_obs);
        CK(cudaMemcpyAsync(c->d_ymx.p, c->h_stage, sizeof(double) * c->n_obs, cudaMemcpyHostToDevice, c->stream));
        site_obs_sum_kernel<<<grid_for(c, c->n, 256), 256, 0, c->stream>>>(c->d_optr.p, c->d_oidx.p, c->d_ymx.p, c->n, c->d_S.p);
        LAUNCHED(c);
        CK(cudaStreamSynchronize(c->stream));
    }
    c->have_obs = true;
    ABI_END
}

void nngp_loglik(const int *ctx_id, const int *slot, const double *beta_0, const double *log_scale, double *ll, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id, true);
    REQUIRE(slot && beta_0 && log_scale && ll && (*slot == 0 || *slot == 1), "nngp_loglik: bad argument");
    NEED(c->have_slot(*slot), "nngp_loglik: that slot holds no factor");
    NEED(c->have_field, "nngp_loglik: no field on the device");
    use(c);
    op_loglik_sums(c, c->linv_slot(*slot), c->d_field.p, *beta_0, 0, true);
    fetch_scalars(c, 2);
    *ll = ll_from_sums(c, c->h_pinned[0], c->h_pinned[1], *log_scale);
    ABI_END
}

void nngp_loglik_host(const int *ctx_id, const int *slot, const double *z, const double *log_scale, double *ll, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(slot && z && log_scale && ll && (*slot == 0 || *slot == 1), "nngp_loglik_host: bad argument");
    NEED(c->have_slot(*slot), "nngp_loglik_host: that slot holds no factor");
    use(c);
    upload_site_vector(c, z, c->d_tmp1.p);
    op_loglik_sums(c, c->linv_slot(*slot), c->d_tmp1.p, 0.0, 0, false);
    fetch_scalars(c, 2);
    *ll = ll_from_sums(c, c->h_pinned[0], c->h_pinned[1], *log_scale);
    ABI_END
}

void nngp_spmv(const int *ctx_id, const int *slot, const double *v, double *out, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(slot && v && out && (*slot == 0 || *slot == 1), "nngp_spmv: bad argument");
    NEED(c->have_slot(*slot), "nngp_spmv: that slot holds no factor");
    use(c);
    upload_site_vector(c, v, c->d_tmp1.p);
    op_spmv(c, c->linv_slot(*slot), c->d_tmp1.p, 0.0, c->d_tmp2.p);
    download_site_vector(c, c->d_tmp2.p, out);
    ABI_END
}

void nngp_sptmv(const int *ctx_id, const int *slot, const double *u, double *out, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    NEED(!c->sharded, "nngp_sptmv: not available on a sharded context (sweep, log-lik, factor build and the scalar reductions are)");
    REQUIRE(slot && u && out && (*slot == 0 || *slot == 1), "nngp_sptmv: bad argument");
    NEED(c->have_slot(*slot), "nngp_sptmv: that slot holds no factor");
    use(c);
    upload_site_vector(c, u, c->d_tmp1.p);
    sptmv_kernel<<<grid_for(c, c->n, 256), 256, 0, c->stream>>>(c->d_colptr.p, c->d_crow.p, c->d_csrc.p, c->d_psite.p, c->linv_slot(*slot), c->d_tmp1.p, c->n, c->d_tmp2.p);
    LAUNCHED(c);
    download_site_vector(c, c->d_tmp2.p, out);
    ABI_END
}

void nngp_sptrsv(const int *ctx_id, const int *slot, const double *b, double *x, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(slot && b && x && (*slot == 0 || *slot == 1), "nngp_sptrsv: bad argument");
    NEED(c->have_slot(*slot), "nngp_sptrsv: that slot holds no factor");
    use(c);
    upload_site_vector(c, b, c->d_tmp1.p);
    op_sptrsv(c, c->linv_slot(*slot), c->d_tmp1.p, c->d_tmp2.p, nullptr, 0.0, 1.0);
    CK(cudaGetLastError());
    download_site_vector(c, c->d_tmp2.p, x);
    check_solve_flag(c);
    ABI_END
}

void nngp_gibbs_sweep(const int *ctx_id, const int *n_sweeps, const double *beta_0, const double *log_scale,
                      const double *log_noise_variance, const int *rng_mode, const double *z, const double *seed, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(n_sweeps && beta_0 && log_scale && log_noise_variance && rng_mode && *n_sweeps >= 0, "nngp_gibbs_sweep: bad argument");
    REQUIRE(*rng_mode == NNGP_RNG_PHILOX || (*rng_mode == NNGP_RNG_SUPPLIED && z != nullptr), "nngp_gibbs_sweep: rng_mode 0 needs z");
    NEED(c->can_sweep, "this context was created without a colouring (all-zero coloring): it cannot run Gibbs sweeps");
    NEED(c->have_slot(NNGP_SLOT_CURRENT), "nngp_gibbs_sweep: no current factor");
    NEED(c->have_field && c->have_obs, "nngp_gibbs_sweep: field and observations must be set first");
    use(c);
    if (!c->committed) op_commit(c);
    const size_t nz = (size_t)c->n_global * (size_t)std::max(1, *n_sweeps);   // normals are indexed by the position in the whole field
    if (*rng_mode == NNGP_RNG_SUPPLIED) {
        ensure_zbuf(c, nz);
        CK(cudaMemcpyAsync(c->d_zbuf.p, z, sizeof(double) * nz, cudaMemcpyHostToDevice, c->stream));
    }
    set_sweep_params(c, *beta_0, *log_scale, *log_noise_variance, *rng_mode, seed ? *seed : 0.0);
    refresh_r(c, *beta_0);
    op_sweeps(c, *n_sweeps);
    c->sweep_counter += (unsigned long long)*n_sweeps;
    CK(cudaStreamSynchronize(c->stream));
    if (c->p2p) check_solve_flag(c);
    ABI_END
}

// One sampler step for a caller that keeps the field on the host: field_io goes up, n_sweeps sweeps run, the Vecchia log-likelihood of
// the new field is taken on the device (the field is already there: nngp_field_set + nngp_gibbs_sweep + nngp_field_get +
// nngp_loglik_host would send it over PCIe a second time), the new field comes down.
void nngp_sweep_loglik_host(const int *ctx_id, const int *n_sweeps, const double *beta_0, const double *log_scale,
                            const double *log_noise_variance, const int *rng_mode, const double *z, const double *seed,
                            double *field_io, double *ll, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(n_sweeps && beta_0 && log_scale && log_noise_variance && rng_mode && field_io && ll && *n_sweeps >= 0, "nngp_sweep_loglik_host: bad argument");
    REQUIRE(*rng_mode == NNGP_RNG_PHILOX || (*rng_mode == NNGP_RNG_SUPPLIED && z != nullptr), "nngp_sweep_loglik_host: rng_mode 0 needs z");
    NEED(c->can_sweep, "this context was created without a colouring (all-zero coloring): it cannot run Gibbs sweeps");
    NEED(c->have_slot(NNGP_SLOT_CURRENT) && c->have_obs, "nngp_sweep_loglik_host: factor and observations must be set first");
    use(c);
    if (!c->committed) op_commit(c);
    const bool pinned = is_pinned(field_io);
    if (pinned) {   // as upload_site_vector, without its synchronisation: the buffer is not handed back before the download below
        CK(cudaMemcpyAsync(c->d_io.p, field_io, sizeof(double) * c->n, cudaMemcpyHostToDevice, c->stream));
        gather_f64_kernel<<<grid_for(c, c->n, 256), 256, 0, c->stream>>>(c->d_field.p, c->d_io.p, c->d_i2g.p, c->n);
        LAUNCHED(c);
    } else {
        upload_site_vector(c, field_io, c->d_field.p);
    }
    c->have_field = true;
    const size_t nz = (size_t)c->n_global * (size_t)std::max(1, *n_sweeps);
    if (*rng_mode == NNGP_RNG_SUPPLIED) {
        ensure_zbuf(c, nz);
        CK(cudaMemcpyAsync(c->d_zbuf.p, z, sizeof(double) * nz, cudaMemcpyHostToDevice, c->stream));
    }
    set_sweep_params(c, *beta_0, *log_scale, *log_noise_variance, *rng_mode, seed ? *seed : 0.0);
    refresh_r(c, *beta_0);
    op_sweeps(c, *n_sweeps);
    c->sweep_counter += (unsigned long long)*n_sweeps;
    if (pinned) {   // the new field leaves on a second stream while the log-lik pass reads it on the first
        gather_f64_kernel<<<grid_for(c, c->n, 256), 256, 0, c->stream>>>(c->d_io.p, c->d_field.p, c->d_g2i.p, c->n);
        LAUNCHED(c);
        CK(cudaEventRecord(c->ev_copy, c->stream));
        CK(cudaStreamWaitEvent(c->copy_stream, c->ev_copy, 0));
        CK(cudaMemcpyAsync(field_io, c->d_io.p, sizeof(double) * c->n, cudaMemcpyDeviceToHost, c->copy_stream));
        op_loglik_sums(c, c->linv_slot(NNGP_SLOT_CURRENT), c->d_field.p, *beta_0, 0, true);
        CK(cudaMemcpyAsync(c->h_pinned, c->d_scalars.p, sizeof(double) * 2, cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        CK(cudaStreamSynchronize(c->copy_stream));
    } else {
        op_loglik_sums(c, c->linv_slot(NNGP_SLOT_CURRENT), c->d_field.p, *beta_0, 0, true);
        CK(cudaMemcpyAsync(c->h_pinned, c->d_scalars.p, sizeof(double) * 2, cudaMemcpyDeviceToHost, c->stream));
        download_site_vector(c, c->d_field.p, field_io);   // synchronises
    }
    *ll = ll_from_sums(c, c->h_pinned[0], c->h_pinned[1], *log_scale);
    if (c->p2p) check_solve_flag(c);
    ABI_END
}

void nngp_shard_p2p_export(const int *ctx_id, char *handle64, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(handle64 != nullptr, "nngp_shard_p2p_export: null buffer");
    NEED(c->sharded && c->p2p_area, "nngp_shard_p2p_export: not a sharded context");
    use(c);
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, c->p2p_area));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle size");
    std::memcpy(handle64, &h, 64);
    ABI_END
}

// after the peers' areas are known: destinations of every boundary site's value (peer, slot inside the peer's receive values)
static void finish_p2p_connect(Ctx *c, const int *peer_recv_base) {
    const int W = c->world, K = c->K;
    std::vector<std::vector<int>> peer_tab(W);   // storage id, on peer h, of every ghost site of peer h (its receive order)
    for (int h = 0; h < W; h++) {   // what every peer's (mapped) area says about itself
        unsigned long long hdr[5] = {0, 0, 0, 0, 0};
        CK(cudaMemcpy(hdr, c->peers.area[h] + c->p2p_hdr_off, sizeof(hdr), cudaMemcpyDeviceToHost));
        REQUIRE(hdr[0] >= 16 && hdr[0] < (1ull << 31) && hdr[2] < (1ull << 32) && hdr[3] < (1ull << 32), "peer %d: implausible area header (was its context created?)", h);
        c->peer_stride[h] = (unsigned int)hdr[0];
        c->peer_x_off[h] = (unsigned int)hdr[2];
        c->peer_x_stride[h] = (unsigned int)hdr[3];
        peer_tab[h].resize((size_t)hdr[1]);
        if (h != c->rank && hdr[1] > 0) CK(cudaMemcpy(peer_tab[h].data(), c->peers.area[h] + hdr[4], (size_t)hdr[1] * sizeof(int), cudaMemcpyDeviceToHost));
    }
    {   // sharded solve: an owned boundary site's solution value goes to x[storage id on the peer] of every peer that ghosts it
        std::vector<int> sxptr((size_t)c->n + 1, 0);
        for (size_t k = 0; k < c->send_proc.size(); k++) sxptr[(size_t)c->send_storage_h[k] + 1]++;
        for (int q = 0; q < c->n; q++) sxptr[q + 1] += sxptr[q];
        std::vector<int2> sxdst(std::max<size_t>(c->send_proc.size(), 1));
        std::vector<int> pos(sxptr.begin(), sxptr.end() - 1);
        for (int col = 0; col < K; col++)
            for (int h = 0; h < W; h++) {
                const int a = c->send_ptr[(size_t)col * W + h], b = c->send_ptr[(size_t)col * W + h + 1];
                for (int k = a; k < b; k++) {
                    const size_t slot = (size_t)peer_recv_base[(size_t)col * W + h] + (size_t)(k - a);
                    REQUIRE(slot < peer_tab[h].size(), "halo lists of rank %d and rank %d do not match", c->rank, h);
                    sxdst[pos[c->send_storage_h[k]]++] = make_int2(h, peer_tab[h][slot]);
                }
            }
        c->d_sxptr.upload(sxptr, c->stream);
        c->d_sxdst.upload(sxdst, c->stream);
        // both solution buffers start "pending"; buffer e & 1 serves solve e and is re-armed at the start of solve e - 1
        fill_u64_kernel<<<grid_for(c, (long long)(2 * c->p2p_x_stride), 256), 256, 0, c->stream>>>(reinterpret_cast<unsigned long long *>(c->p2p_area + c->p2p_x_off), NNGP_SOLVE_SENTINEL, (int)(2 * c->p2p_x_stride));
        c->solve_epoch = 0;
    }
    std::vector<int> bptr((size_t)c->n_owned + 1, 0);
    for (size_t k = 0; k < c->send_proc.size(); k++) bptr[(size_t)c->send_proc[k] + 1]++;
    for (int q = 0; q < c->n_owned; q++) bptr[q + 1] += bptr[q];
    std::vector<int2> bdst(std::max<size_t>(c->send_proc.size(), 1));
    std::vector<int> pos(bptr.begin(), bptr.end() - 1);
    for (int col = 0; col < K; col++)
        for (int h = 0; h < W; h++) {
            const int a = c->send_ptr[(size_t)col * W + h], b = c->send_ptr[(size_t)col * W + h + 1];
            for (int k = a; k < b; k++) bdst[pos[c->send_proc[k]]++] = make_int2(h, peer_recv_base[(size_t)col * W + h] + (k - a));
        }
    c->d_bptr.upload(bptr, c->stream);
    c->d_bdst.upload(bdst, c->stream);
    CK(cudaMemsetAsync(c->d_shard_state.p, 0, 4 * sizeof(unsigned long long), c->stream));
    // every ghost slot (both parities) starts EMPTY: the value itself is the message (see NNGP_HALO_EMPTY)
    fill_u64_kernel<<<grid_for(c, (long long)(2 * c->p2p_parity_stride), 256), 256, 0, c->stream>>>(reinterpret_cast<unsigned long long *>(c->p2p_area + c->p2p_val_off), NNGP_HALO_EMPTY, (int)(2 * c->p2p_parity_stride));
    CK(cudaStreamSynchronize(c->stream));
    if (c->sweep_graph) { cudaGraphExecDestroy(c->sweep_graph); c->sweep_graph = nullptr; }
    c->p2p = true;
}

void nngp_shard_p2p_connect(const int *ctx_id, const char *all_handles, const int *peer_recv_base, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(all_handles && peer_recv_base, "nngp_shard_p2p_connect: null argument");
    NEED(c->sharded && c->p2p_area, "nngp_shard_p2p_connect: not a sharded context");
    use(c);
    const int W = c->world;
    for (int h = 0; h < W; h++) {
        if (h == c->rank) { c->peers.area[h] = c->p2p_area; continue; }
        cudaIpcMemHandle_t hd;
        std::memcpy(&hd, all_handles + (size_t)h * 64, 64);
        void *p = nullptr;
        CK(cudaIpcOpenMemHandle(&p, hd, cudaIpcMemLazyEnablePeerAccess));
        c->peer_mapped[h] = p;
        c->peers.area[h] = static_cast<double *>(p);
    }
    finish_p2p_connect(c, peer_recv_base);
    ABI_END
}

// single-process form: the W contexts of the field live in this process (one per GPU -- what an R session with several GPUs
// has -- or several on one GPU); their areas are addressed directly, peer access is enabled between distinct devices
void nngp_shard_connect_local(const int *ctx_ids, const int *world, int *status) {
    ABI_BEGIN
    REQUIRE(ctx_ids && world && *world >= 1 && *world <= 8, "nngp_shard_connect_local: bad argument");
    const int W = *world;
    std::vector<Ctx *> cs(W);
    for (int h = 0; h < W; h++) {
        cs[h] = get_ctx(ctx_ids + h);
        NEED(cs[h]->sharded && cs[h]->p2p_area && cs[h]->world == W && cs[h]->rank == h, "nngp_shard_connect_local: context h must be rank h of a W-rank sharded field");
        NEED(cs[h]->K == cs[0]->K, "nngp_shard_connect_local: the contexts belong to different fields");
    }
    for (int g = 0; g < W; g++) {
        Ctx *c = cs[g];
        use(c);
        preload_device_code(c->device);   // members wait for each other inside kernels: no lazy module load may happen from now on
        std::vector<int> base((size_t)c->K * W, 0);
        for (int h = 0; h < W; h++) {
            c->peers.area[h] = cs[h]->p2p_area;
            if (h == g) continue;
            if (cs[h]->device != c->device) {
                int can = 0;
                CK(cudaDeviceCanAccessPeer(&can, c->device, cs[h]->device));
                REQUIRE(can, "device %d cannot access device %d", c->device, cs[h]->device);
                cudaError_t e = cudaDeviceEnablePeerAccess(cs[h]->device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CK(e);
                cudaGetLastError();
            }
            for (int col = 0; col < c->K; col++) {
                const int mine = c->send_ptr[(size_t)col * W + h + 1] - c->send_ptr[(size_t)col * W + h];
                const int theirs = cs[h]->recv_ptr[(size_t)col * W + g + 1] - cs[h]->recv_ptr[(size_t)col * W + g];
                REQUIRE(mine == theirs, "nngp_shard_connect_local: rank %d sends %d values of colour %d to rank %d, which expects %d", g, mine, col + 1, h, theirs);
                base[(size_t)col * W + h] = cs[h]->recv_ptr[(size_t)col * W + g];
            }
        }
        finish_p2p_connect(c, base.data());
    }
    ABI_END
}

// enqueues n_sweeps sweeps on every member of a locally connected field, then waits for all of them (the members exchange
// their halos among themselves while they run)
void nngp_shard_group_sweep(const int *ctx_ids, const int *world, const int *n_sweeps, const double *beta_0, const double *log_scale,
                            const double *log_noise_variance, const int *rng_mode, const double *z, const double *seed, int *status) {
    ABI_BEGIN
    REQUIRE(ctx_ids && world && n_sweeps && beta_0 && log_scale && log_noise_variance && rng_mode && *world >= 1 && *world <= 8 && *n_sweeps >= 0, "nngp_shard_group_sweep: bad argument");
    REQUIRE(*rng_mode == NNGP_RNG_PHILOX || (*rng_mode == NNGP_RNG_SUPPLIED && z != nullptr), "nngp_shard_group_sweep: rng_mode 0 needs z");
    const int W = *world;
    std::vector<Ctx *> cs(W);
    for (int h = 0; h < W; h++) {
        cs[h] = get_ctx(ctx_ids + h);
        NEED(cs[h]->sharded && (cs[h]->p2p || W == 1), "nngp_shard_group_sweep: the contexts are not connected (nngp_shard_connect_local)");
        NEED(cs[h]->have_slot(NNGP_SLOT_CURRENT) && cs[h]->have_field && cs[h]->have_obs, "nngp_shard_group_sweep: factor, field and observations must be set first");
    }
    for (Ctx *c : cs) {
        use(c);
        if (!c->committed) op_commit(c);
        const size_t nz = (size_t)c->n_global * (size_t)std::max(1, *n_sweeps);
        if (*rng_mode == NNGP_RNG_SUPPLIED) {
            ensure_zbuf(c, nz);
            CK(cudaMemcpyAsync(c->d_zbuf.p, z, sizeof(double) * nz, cudaMemcpyHostToDevice, c->stream));
        }
        set_sweep_params(c, *beta_0, *log_scale, *log_noise_variance, *rng_mode, seed ? *seed : 0.0);
        refresh_r(c, *beta_0);
    }
    for (int s = 0; s < *n_sweeps; s++)       // sweep by sweep over the members: no stream runs far ahead of its peers
        for (Ctx *c : cs) { use(c); op_sweeps(c, 1); }
    for (Ctx *c : cs) {
        use(c);
        c->sweep_counter += (unsigned long long)*n_sweeps;
        CK(cudaStreamSynchronize(c->stream));
    }
    for (Ctx *c : cs) { use(c); check_solve_flag(c); }
    ABI_END
}

// all-reduced scalars of a locally connected field: [sum log diag, sum u^2] of the log-likelihood -> ll (identical on every member)
void nngp_shard_group_loglik(const int *ctx_ids, const int *world, const int *slot, const double *beta_0, const double *log_scale,
                             double *ll, int *status) {
    ABI_BEGIN
    REQUIRE(ctx_ids && world && slot && beta_0 && log_scale && ll && *world >= 1 && *world <= 8 && (*slot == 0 || *slot == 1), "nngp_shard_group_loglik: bad argument");
    const int W = *world;
    std::vector<Ctx *> cs(W);
    for (int h = 0; h < W; h++) {
        cs[h] = get_ctx(ctx_ids + h);
        NEED(cs[h]->sharded && (cs[h]->p2p || W == 1), "nngp_shard_group_loglik: the contexts are not connected (nngp_shard_connect_local)");
        NEED(cs[h]->have_slot(*slot) && cs[h]->have_field, "nngp_shard_group_loglik: factor and field must be set first");
    }
    for (Ctx *c : cs) { use(c); op_loglik_sums(c, c->linv_slot(*slot), c->d_field.p, *beta_0, 0, false); }
    for (int h = 0; h < W; h++) {
        Ctx *c = cs[h];
        use(c);
        fetch_scalars(c, 2);
        ll[h] = ll_from_sums(c, c->h_pinned[0], c->h_pinned[1], *log_scale);
    }
    for (Ctx *c : cs) { use(c); check_solve_flag(c); }
    ABI_END
}

// ---- colour-stepping form of the sharded sweep: the caller moves the halo (any transport), the library does the rest ----
void nngp_shard_sweep_begin(const int *ctx_id, const double *beta_0, const double *log_scale, const double *log_noise_variance,
                            const int *rng_mode, const double *z, const double *seed, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(beta_0 && log_scale && log_noise_variance && rng_mode, "nngp_shard_sweep_begin: bad argument");
    REQUIRE(*rng_mode == NNGP_RNG_PHILOX || (*rng_mode == NNGP_RNG_SUPPLIED && z != nullptr), "nngp_shard_sweep_begin: rng_mode 0 needs z");
    NEED(c->sharded, "nngp_shard_sweep_begin: not a sharded context");
    NEED(c->have_slot(NNGP_SLOT_CURRENT) && c->have_field && c->have_obs, "nngp_shard_sweep_begin: factor, field and observations must be set first");
    use(c);
    if (!c->committed) op_commit(c);
    if (*rng_mode == NNGP_RNG_SUPPLIED) {
        ensure_zbuf(c, (size_t)c->n_global);
        CK(cudaMemcpyAsync(c->d_zbuf.p, z, sizeof(double) * (size_t)c->n_global, cudaMemcpyHostToDevice, c->stream));
    }
    set_sweep_params(c, *beta_0, *log_scale, *log_noise_variance, *rng_mode, seed ? *seed : 0.0);
    refresh_r(c, *beta_0);
    CK(cudaStreamSynchronize(c->stream));
    ABI_END
}

void nngp_shard_sweep_colour(const int *ctx_id, const int *colour, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(colour && *colour >= 1 && *colour <= c->K, "nngp_shard_sweep_colour: colour out of range");
    NEED(c->sharded, "nngp_shard_sweep_colour: not a sharded context");
    use(c);
    const int col = *colour - 1;
    const int t0 = c->tile_ptr[col], nt = c->tile_ptr[col + 1] - t0;
    if (nt > 0) {
        gibbs_tile2_kernel<128, false, 5, 2><<<nt, 128, 0, c->stream>>>(c->d_tiles.p + t0, t0, c->d_colptr.p, c->d_crow.p, c->d_cloc.p, c->d_valT.p, c->d_pd.p, c->d_nobs.p, c->d_S.p, c->d_zpos.p, c->d_gid.p, c->d_psite.p, c->d_zbuf.p, c->d_sp.p, c->d_field.p, c->d_r.p, ShardConst{}, ShardColour{});
        LAUNCHED(c);
    }
    CK(cudaGetLastError());
    ABI_END
}

void nngp_shard_halo_get(const int *ctx_id, const int *colour, double *out, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(colour && *colour >= 1 && *colour <= c->K, "nngp_shard_halo_get: colour out of range");
    NEED(c->sharded, "nngp_shard_halo_get: not a sharded context");
    use(c);
    const int W = c->world, col = *colour - 1;
    const int s0 = c->send_ptr[(size_t)col * W], s1 = c->send_ptr[(size_t)(col + 1) * W];
    if (s1 > s0) {
        REQUIRE(out != nullptr, "nngp_shard_halo_get: null buffer");
        halo_pack_kernel<<<(s1 - s0 + 255) / 256, 256, 0, c->stream>>>(c->d_send_storage.p, c->d_field.p, s0, s1, c->d_sendbuf.p);
        LAUNCHED(c);
        CK(cudaMemcpyAsync(out, c->d_sendbuf.p + s0, sizeof(double) * (size_t)(s1 - s0), cudaMemcpyDeviceToHost, c->stream));
    }
    CK(cudaStreamSynchronize(c->stream));
    ABI_END
}

void nngp_shard_halo_put(const int *ctx_id, const int *colour, const double *in, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(colour && *colour >= 1 && *colour <= c->K, "nngp_shard_halo_put: colour out of range");
    NEED(c->sharded, "nngp_shard_halo_put: not a sharded context");
    use(c);
    const int W = c->world, col = *colour - 1;
    const int r0 = c->recv_ptr[(size_t)col * W], r1 = c->recv_ptr[(size_t)(col + 1) * W];
    if (r1 > r0) {
        REQUIRE(in != nullptr, "nngp_shard_halo_put: null buffer");
        CK(cudaMemcpyAsync(c->d_recvbuf.p + r0, in, sizeof(double) * (size_t)(r1 - r0), cudaMemcpyHostToDevice, c->stream));
        halo_apply_kernel<<<(r1 - r0 + 255) / 256, 256, 0, c->stream>>>(c->d_recv_proc.p, c->d_recvbuf.p, r0, r1, c->d_colptr.p, c->d_crow.p, c->d_valT.p, c->d_psite.p, c->d_field.p, c->d_r.p);
        LAUNCHED(c);
    }
    CK(cudaStreamSynchronize(c->stream));
    ABI_END
}

void nngp_shard_sweep_end(const int *ctx_id, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    NEED(c->sharded, "nngp_shard_sweep_end: not a sharded context");
    use(c);
    advance_sweep_kernel<<<1, 32, 0, c->stream>>>(c->d_sp.p, (unsigned long long)c->n_global, nullptr);
    LAUNCHED(c);
    c->sweep_counter += 1ull;
    CK(cudaStreamSynchronize(c->stream));
    ABI_END
}

void nngp_ancillary_propose(const int *ctx_id, const double *beta_0, const double *delta_log_scale,
                            const double *log_noise_variance, double *field_response_ratio, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(beta_0 && delta_log_scale && log_noise_variance && field_response_ratio, "nngp_ancillary_propose: bad argument");
    NEED(c->have_slot(NNGP_SLOT_CURRENT) && c->have_slot(NNGP_SLOT_PROPOSAL), "nngp_ancillary_propose: needs current and proposal factors");
    NEED(c->have_field && c->have_obs, "nngp_ancillary_propose: field and observations must be set first");
    use(c);
    // tmp1 = current %*% (field - beta_0); tmp2 = solve(proposal, tmp1); newfield = beta_0 + exp(.5 dls) * tmp2
    op_spmv(c, c->linv_slot(NNGP_SLOT_CURRENT), c->d_field.p, *beta_0, c->d_tmp1.p);
    op_sptrsv(c, c->linv_slot(NNGP_SLOT_PROPOSAL), c->d_tmp1.p, c->d_tmp2.p, c->d_newfield.p, *beta_0, std::exp(0.5 * *delta_log_scale));
    op_obs_sq(c, c->d_newfield.p, c->d_field.p, 0);
    CK(cudaGetLastError());
    fetch_scalars(c, 2);
    check_solve_flag(c);
    // sum(dnorm(y, new) - dnorm(y, old)) = -(SSR_new - SSR_old) / (2 tau^2)
    *field_response_ratio = -0.5 * (c->h_pinned[0] - c->h_pinned[1]) * std::exp(-*log_noise_variance);
    c->have_newfield = true;
    ABI_END
}

void nngp_ancillary_accept(const int *ctx_id, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    NEED(c->have_newfield, "nngp_ancillary_accept: no proposal field");
    use(c);
    // D2D copy (16 MB of traffic at n = 1M) rather than a pointer swap: the captured sweep graph bakes the field pointer in
    CK(cudaMemcpyAsync(c->d_field.p, c->d_newfield.p, sizeof(double) * c->n, cudaMemcpyDeviceToDevice, c->stream));
    c->have_newfield = false;
    c->cur = 1 - c->cur;
    op_commit(c);
    ABI_END
}

void nngp_beta0_moments(const int *ctx_id, const double *log_scale, double *mean, double *var, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(log_scale && mean && var, "nngp_beta0_moments: bad argument");
    NEED(c->have_slot(NNGP_SLOT_CURRENT) && c->have_field, "nngp_beta0_moments: needs a current factor and a field");
    use(c);
    op_beta0_sums(c, 0);
    fetch_scalars(c, 2);
    const double vv = c->h_pinned[0], uv = c->h_pinned[1];
    *var = (1.0 / vv) * std::exp(*log_scale);
    *mean = std::exp(-*log_scale) * uv * *var;
    ABI_END
}

void nngp_ssr(const int *ctx_id, double *ssr, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(ssr != nullptr, "null ssr");
    NEED(c->have_field && c->have_obs, "nngp_ssr: field and observations must be set first");
    use(c);
    op_obs_sq(c, c->d_field.p, c->d_field.p, 0);
    fetch_scalars(c, 2);
    *ssr = c->h_pinned[0];
    ABI_END
}

void nngp_field_init(const int *ctx_id, const int *slot, const double *beta_0, const double *log_scale, const double *z, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(slot && beta_0 && log_scale && z && (*slot == 0 || *slot == 1), "nngp_field_init: bad argument");
    NEED(c->have_slot(*slot), "nngp_field_init: that slot holds no factor");
    use(c);
    upload_site_vector(c, z, c->d_tmp1.p);
    op_sptrsv(c, c->linv_slot(*slot), c->d_tmp1.p, c->d_tmp2.p, c->d_field.p, *beta_0, std::sqrt(std::exp(*log_scale)));
    CK(cudaGetLastError());
    check_solve_flag(c);
    c->have_field = true;
    ABI_END
}

void nngp_predict_sample(const int *ctx_id, const int *slot, const int *n_obs_sites, const double *field, const double *beta_0,
                         const double *log_scale, const double *z_pred, double *out, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    NEED(!c->sharded, "nngp_predict_sample: not available on a sharded context (sweep, log-lik, factor build and the scalar reductions are)");
    REQUIRE(slot && n_obs_sites && field && beta_0 && log_scale && z_pred && out && (*slot == 0 || *slot == 1), "nngp_predict_sample: bad argument");
    REQUIRE(*n_obs_sites >= 0 && *n_obs_sites <= c->n, "nngp_predict_sample: n_obs_sites out of range");
    NEED(c->have_slot(*slot), "nngp_predict_sample: that slot holds no factor");
    use(c);
    // predict.R:43-53 solves the joint system with rhs c(sparse_chol[1:n,1:n] %*% (field - beta_0)/sd, z): its first n0 unknowns
    // are (field - beta_0)/sd again, so only the new rows are solved:  x_i = (z_i - sum_j Linv[i,j] x[nn(i,j)]) / Linv[i,1].
    const int n0 = *n_obs_sites, np = c->n - n0, n = c->n;
    const double sd = std::exp(0.5 * *log_scale);
    if (c->pred_n0 != n0) {   // level schedule of the new rows (a new row waits only for new-site parents)
        std::vector<int> nn((size_t)c->ld * c->M);
        CK(cudaMemcpy(nn.data(), c->d_nn.p, sizeof(int) * nn.size(), cudaMemcpyDeviceToHost));
        std::vector<int> lvl(n, -1);
        int depth = 0;
        for (int i = n0; i < n; i++) {
            const int q = c->g2i[i];
            int l = 0;
            for (int j = 1; j < c->M; j++) {
                const int p = nn[(size_t)j * c->ld + q];
                if (p >= 0 && lvl[p] >= 0) l = std::max(l, lvl[p] + 1);
            }
            lvl[q] = l;
            depth = std::max(depth, l + 1);
        }
        std::vector<std::vector<int>> by_level(depth);
        for (int q = 0; q < n; q++) if (lvl[q] >= 0) by_level[lvl[q]].push_back(q);
        std::vector<int> rows;
        rows.reserve((size_t)np + 32 * (size_t)depth);
        for (auto &v : by_level) { for (int q : v) rows.push_back(q); while (rows.size() % 32) rows.push_back(-1); }
        c->d_pred_rows.upload(rows, c->stream);
        CK(cudaStreamSynchronize(c->stream));
        c->pred_slots = (int)rows.size();
        c->pred_levels = depth;
        c->pred_n0 = n0;
    }
    std::vector<double> host(n);
    for (int i = 0; i < n0; i++) host[i] = (field[i] - *beta_0) / sd;
    for (int i = 0; i < np; i++) host[n0 + i] = z_pred[i];
    upload_site_vector(c, host.data(), c->d_tmp1.p);     // known x on the observed rows, rhs z on the new rows
    predict_prepare_kernel<<<grid_for(c, n, 256), 256, 0, c->stream>>>(reinterpret_cast<unsigned long long *>(c->d_tmp2.p), c->d_tmp1.p, c->d_i2g.p, n0, n);
    LAUNCHED(c);
    if (c->pred_slots > 0) {
        CK(cudaMemsetAsync(c->d_ticket.p, 0, sizeof(int), c->stream));
        const int want = c->solve_window_ctas > 0 ? c->solve_window_ctas : c->n_sm * c->solve_ctas_per_sm;
        const int blocks = std::max(1, std::min((c->pred_slots + 255) / 256, want));
        const double *linv = c->linv_slot(*slot);
        DISPATCH_MT(c->M, (sptrsv_syncfree_kernel<MT><<<blocks, 256, 0, c->stream>>>(c->d_nn.p, linv, c->d_pred_rows.p, c->pred_slots, c->d_tmp1.p, reinterpret_cast<unsigned long long *>(c->d_tmp2.p), nullptr, 0.0, 1.0, c->ld, c->M, c->d_ticket.p, c->d_nbad.p + 1, (unsigned int)c->solve_sleep_ns, ShardSolve{})));
        LAUNCHED(c);
    }
    CK(cudaGetLastError());
    download_site_vector(c, c->d_tmp2.p, host.data());
    check_solve_flag(c);
    for (int i = 0; i < np; i++) out[i] = sd * host[n0 + i];
    ABI_END
}

}  // extern "C"

// Buffers a chain needs beyond the context's own (the supplied-normals block, the device-side record store).  Allocating or
// freeing device memory synchronises the device, which must not happen while a peer of a sharded field waits on this rank from
// inside a kernel: the group entry points call this for every member BEFORE they start the chain threads.
static bool prepare_chain_buffers(Ctx *c, int n_iter, double thin, int n_chromatic, int rng_mode, bool want_field_records) {
    use(c);
    if (rng_mode == NNGP_RNG_SUPPLIED) ensure_zbuf(c, (size_t)c->n_global * (size_t)std::max(1, n_chromatic));
    const int n_frec = (int)std::nearbyint(n_iter * thin);
    bool on_device = false;
    if (want_field_records && n_frec > 0) {
        size_t free_b = 0, total_b = 0;
        CK(cudaMemGetInfo(&free_b, &total_b));
        const size_t need = (size_t)n_frec * c->n * sizeof(double);
        if (c->d_frec.n >= (size_t)n_frec * c->n || need + ((size_t)2 << 30) < free_b + c->d_frec.n * sizeof(double)) {
            if (c->d_frec.n < (size_t)n_frec * c->n) c->d_frec.alloc((size_t)n_frec * c->n);
            on_device = true;
            c->frec_rows = n_frec;
        }
    }
    return on_device;
}

// regression part of one chain (nngp_chain_run_regressors); nullptr = the no-regressor model
struct RegRun {
    double *beta_io;              // p: state$params$beta in, out
    const double *solve_1XT1X;    // (p+1) x (p+1): X$solve_1XT1X      (initialize.R:135)
    const double *chol_1XT1X;     // (p+1) x (p+1): X$chol_solve_1XT1X (initialize.R:136; upper factor)
    double *beta_records;         // n_iter x p column-major, or NULL
};

// The loop of Scripts/mcmc_nngp_update_Gaussian.R:101-314 for one chain, entirely on the device side of the ABI.
static void chain_run_impl(Ctx *c, const int *n_shape_, double *params_io, const int *n_iter_, const double *thin_,
                           const int *n_chromatic_, const int *iter_start_, const int *chain_index_, const int *rng_mode_,
                           const double *var_y_, double *records_out, double *field_records_out, int *accept_out, const RegRun *reg) {
    const int ns = *n_shape_, n_iter = *n_iter_, n_chromatic = *n_chromatic_, iter_start = *iter_start_, rng_mode = *rng_mode_;
    const double thin = *thin_, var_y = *var_y_;
    REQUIRE(ns >= 1 && ns <= 5 && n_iter >= 0 && n_chromatic >= 0, "nngp_chain_run: bad sizes");
    NEED(c->can_sweep, "this context was created without a colouring (all-zero coloring): it cannot run Gibbs sweeps");
    use(c);
    // the loop refreshes r before its sweeps and changes the field and the factor after them: however it ends, r is not left
    // marked current
    struct ForgetR { Ctx *c; ~ForgetR() { c->r_valid = false; } } forget_r{c};
    // regressors: beta, the interweaving matrices (:77-83) and scratch for the (p+1)- and q-vectors
    const int reg_p = reg ? c->reg_p : 0, reg_q = reg ? c->reg_q : 0, P1 = reg_p + 1;
    std::vector<double> beta, iw_cov, iw_chol, gvec, bmean, zz, innov, coefl;
    if (reg) {
        beta.assign(reg->beta_io, reg->beta_io + reg_p);
        const size_t w = (size_t)std::max(P1, reg_q);
        gvec.resize(w); bmean.resize(w); zz.resize(w); innov.resize(w); coefl.resize(w);
    }
    const int n = c->n;
    const long long nz = c->n_global;   // normals of a sweep are indexed by the position in the WHOLE field's hand-out order
    const bool matern = c->covfun >= NNGP_MATERN_ISOTROPIC;
    // a sharded field: every rank runs this loop on its block with the same scalar state and the same R stream; all scalars
    // that enter a decision are all-reduced (rank-ordered sums, identical everywhere), so the ranks stay in step
    if (c->n_obs_global < 0) {
        if (c->sharded && c->world > 1) {
            c->h_pinned[16] = (double)c->n_obs;
            CK(cudaMemcpyAsync(c->d_scalars.p + 16, c->h_pinned + 16, sizeof(double), cudaMemcpyHostToDevice, c->stream));
            allreduce_scalars(c, 16, 1);
            CK(cudaMemcpyAsync(c->h_pinned + 16, c->d_scalars.p + 16, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
            CK(cudaStreamSynchronize(c->stream));
            c->n_obs_global = c->h_pinned[16];
        } else {
            c->n_obs_global = (double)c->n_obs;
        }
    }
    const double n_obs = c->n_obs_global;
    const int n_obs_local = c->n_obs;
    double beta_0 = params_io[0], log_scale = params_io[1], lnv = params_io[2], logvar_suf = params_io[3], logvar_anc = params_io[4];
    double shape[5], new_shape[5], cp[8], innovation[6];
    for (int k = 0; k < ns; k++) shape[k] = params_io[5 + k];
    auto to_covparms = [&](const double *sh) {   // update_Gaussian.R:67-71,117-122,173-178
        cp[0] = 1.0;
        for (int j = 0; j < ns; j++) cp[1 + j] = (matern && j == ns - 1) ? 0.5 + 0.5 / (1.0 + std::exp(-sh[j])) : std::exp(sh[j]);
        cp[1 + ns] = 0.0;
        return make_cov(c, cp, ns + 2);
    };
    auto n_bad = [&]() {   // rows whose block was not positive definite; also surfaces a solve / halo wait that timed out
        int bad[2];
        const bool reduce = c->sharded && c->world > 1;
        if (reduce) {   // the accept / reject decision must be the same on every rank: sum the counts over the ranks
            int_to_f64_kernel<<<1, 32, 0, c->stream>>>(c->d_nbad.p, c->d_scalars.p + 17);
            LAUNCHED(c);
            allreduce_scalars(c, 17, 1);
            CK(cudaMemcpyAsync(c->h_pinned + 17, c->d_scalars.p + 17, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
        }
        CK(cudaMemcpyAsync(c->h_pinned + 8, c->d_nbad.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        std::memcpy(bad, c->h_pinned + 8, 2 * sizeof(int));
        if (reduce) bad[0] = (int)std::min(2.0e9, c->h_pinned[17]);
        if (bad[1] == 2) { set_error("sharded field: timed out waiting for a peer's halo / reduction flag (a rank died or fell out of step)"); throw NcclFail(); }
        if (bad[1]) { set_error("triangular solve: dependency wait timed out (corrupted neighbour structure?)"); throw CudaFail(); }
        return bad[0];
    };
    RStream rs;
    rs.set_seed((uint32_t)(iter_start + *chain_index_));                         // :36
    op_factor_build(c, NNGP_SLOT_CURRENT, to_covparms(shape));                   // :72
    op_commit(c);                                                                // :73-74
    std::vector<double> zhost;
    // :75 current_p = rnorm(n_locs) is dead code in the reference but consumes n draws of R's stream.  In NNGP_RNG_SUPPLIED mode
    // (bit-comparable with R) they are consumed too; in Philox mode the field draws differ from R's anyway, so the 15-20 ms of
    // host RNG per call (n = 1M) are skipped and the scalar draws simply continue from the seeded state.
    if (rng_mode == NNGP_RNG_SUPPLIED) { zhost.resize((size_t)nz); rs.rnorm(zhost.data(), nz); }
    std::vector<int> acc_anc(n_iter + 1, 0), acc_suf(n_iter + 1, 0);
    if (reg_q > 0) op_interweave(c, iw_cov, iw_chol);                            // :77-83
    if (reg) op_set_beta(c, beta.data());                                        // :85
    const int n_frec = (int)std::nearbyint(n_iter * thin);
    // stored field samples stay in HBM, already in R's n_frec x n column-major layout, and leave in one copy at the end
    const bool frec_on_device = prepare_chain_buffers(c, n_iter, thin, n_chromatic, rng_mode, field_records_out != nullptr);
    const unsigned long long philox_seed = ((unsigned long long)(uint32_t)iter_start << 20) ^ (unsigned long long)(uint32_t)*chain_index_;
    // development aid: NNGP_CHAIN_PROFILE=1 synchronises at the phase boundaries and prints host wall-clock per phase
    const bool prof = std::getenv("NNGP_CHAIN_PROFILE") != nullptr;
    double phase_s[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    auto t_last = std::chrono::steady_clock::now();
    auto mark = [&](int k) {
        if (!prof) return;
        CK(cudaStreamSynchronize(c->stream));
        const auto t = std::chrono::steady_clock::now();
        phase_s[k] += std::chrono::duration<double>(t - t_last).count();
        t_last = t;
    };
    if (prof) { CK(cudaStreamSynchronize(c->stream)); t_last = std::chrono::steady_clock::now(); }
    for (int iter = 1; iter <= n_iter; iter++) {
        // ---- (A) ancillary :113-157 ----
        nvtxRangePushA("nngp A ancillary covariance update");
        const double sd_anc = std::exp(.5 * logvar_anc);
        for (int k = 0; k < ns + 1; k++) innovation[k] = 0.0 + sd_anc * rs.norm_rand();
        double new_log_scale = log_scale + innovation[0];
        for (int k = 0; k < ns; k++) new_shape[k] = shape[k] + innovation[1 + k];
        op_factor_build(c, NNGP_SLOT_PROPOSAL, to_covparms(new_shape));          // :123
        op_spmv(c, c->linv_slot(NNGP_SLOT_CURRENT), c->d_field.p, beta_0, c->d_tmp1.p);
        op_sptrsv(c, c->linv_slot(NNGP_SLOT_PROPOSAL), c->d_tmp1.p, c->d_tmp2.p, c->d_newfield.p, beta_0, std::exp(.5 * (new_log_scale - log_scale)));  // :127
        op_obs_sq(c, c->d_newfield.p, c->d_field.p, 0);
        fetch_scalars(c, 2);
        const int bad_a = n_bad();
        const double ratio = -0.5 * (c->h_pinned[0] - c->h_pinned[1]) * std::exp(-lnv);   // :129-131
        if (ratio + 0.0 > std::log(rs.unif_rand()) && bad_a == 0) {              // :133
            std::memcpy(shape, new_shape, sizeof(double) * ns);
            log_scale = new_log_scale;
            CK(cudaMemcpyAsync(c->d_field.p, c->d_newfield.p, sizeof(double) * n, cudaMemcpyDeviceToDevice, c->stream));
            c->cur = 1 - c->cur;
            op_commit(c);
            acc_anc[iter] = 1;
            if (reg_q > 0) op_interweave(c, iw_cov, iw_chol);                    // :145-151
        }
        if (iter_start >= 0 && iter_start <= 2000 && iter % 25 == 0) {           // :153-157
            int a = 0;
            for (int k = iter - 24; k <= iter; k++) a += acc_anc[k];
            const double mean_acc = a / 25.0;
            if (mean_acc < .05) logvar_anc -= (.4 + .05 * rs.norm_rand());
            if (mean_acc > .15) logvar_anc += (.4 + .05 * rs.norm_rand());
        }
        mark(0);
        nvtxRangePop();
        // ---- (B) sufficient :165-213 ----
        nvtxRangePushA("nngp B sufficient covariance update");
        const double sd_suf = std::exp(.5 * logvar_suf);
        for (int k = 0; k < ns + 1; k++) innovation[k] = 0.0 + sd_suf * rs.norm_rand();
        new_log_scale = log_scale + innovation[0];
        if (std::exp(new_log_scale) < var_y) {                                    // :167
            for (int k = 0; k < ns; k++) new_shape[k] = shape[k] + innovation[1 + k];
            op_factor_build(c, NNGP_SLOT_PROPOSAL, to_covparms(new_shape));      // :179
            op_loglik_sums(c, c->linv_slot(NNGP_SLOT_PROPOSAL), c->d_field.p, beta_0, 0, false);
            op_loglik_sums(c, c->linv_slot(NNGP_SLOT_CURRENT), c->d_field.p, beta_0, 2, false);
            fetch_scalars(c, 4);
            const int bad_s = n_bad();
            const double GP_ratio = ll_from_sums(c, c->h_pinned[0], c->h_pinned[1], new_log_scale) -
                                    ll_from_sums(c, c->h_pinned[2], c->h_pinned[3], log_scale);   // :184-186
            if (GP_ratio > std::log(rs.unif_rand()) && bad_s == 0) {              // :189
                std::memcpy(shape, new_shape, sizeof(double) * ns);
                log_scale = new_log_scale;
                c->cur = 1 - c->cur;
                op_commit(c);
                acc_suf[iter] = 1;
                if (reg_q > 0) op_interweave(c, iw_cov, iw_chol);                // :200-206
            }
        }
        if (iter_start >= 0 && iter_start <= 2000 && iter % 25 == 0) {           // :209-213
            int a = 0;
            for (int k = iter - 24; k <= iter; k++) a += acc_suf[k];
            const double mean_acc = a / 25.0;
            if (mean_acc < .05) logvar_suf -= (.2 + .05 * rs.norm_rand());
            if (mean_acc > .15) logvar_suf += (.2 + .05 * rs.norm_rand());
        }
        mark(1);
        nvtxRangePop();
        // ---- (C) beta_0 :219-224 (no location-level regressors) ----
        nvtxRangePushA("nngp C mean parameters");
        if (reg_q == 0) {
            op_beta0_sums(c, 0);
            fetch_scalars(c, 2);
            const double bvar = (1.0 / c->h_pinned[0]) * std::exp(log_scale);
            const double b0mean = std::exp(-log_scale) * c->h_pinned[1] * bvar;
            beta_0 = b0mean + std::sqrt(bvar) * rs.norm_rand();
        }
        // ---- (C') regression coefficients :226-250 ----
        if (reg) {
            // :229 beta_mean = crossprod(observed_field - field[locs_match] + beta_0, cbind(1, X$X)) %*% X$solve_1XT1X
            obs_resid_kernel<<<grid_for(c, n_obs_local, 256), 256, 0, c->stream>>>(c->d_lm.p, c->d_yobs.p, c->d_field.p, beta_0, n_obs_local, c->d_robs.p);
            LAUNCHED(c);
            op_atb(c, c->d_Xa.p, P1, c->d_robs.p, 1, n_obs_local, gvec.data());
            for (int j = 0; j < P1; j++) {
                double v = 0.0;
                for (int k = 0; k < P1; k++) v += gvec[k] * reg->solve_1XT1X[(size_t)k + (size_t)P1 * j];
                bmean[j] = v;
            }
            for (int k = 0; k < P1; k++) zz[k] = rs.norm_rand();                 // :231 rnorm(ncol(X$X) + 1)
            const double sd_noise = std::exp(.5 * lnv);
            for (int j = 0; j < P1; j++) {                                       // t(chol) %*% z
                double v = 0.0;
                for (int k = 0; k <= j; k++) v += reg->chol_1XT1X[(size_t)k + (size_t)P1 * j] * zz[k];
                innov[j] = bmean[j] + sd_noise * v;
            }
            shift_kernel<<<grid_for(c, n, 256), 256, 0, c->stream>>>(c->d_field.p, n, beta_0, innov[0]);   // :232
            LAUNCHED(c);
            beta_0 = innov[0];
            for (int k = 0; k < reg_p; k++) beta[k] = innov[1 + k];
            if (reg_q > 0) {                                                     // :237-246 interweaving
                coefl[0] = 0.0;
                for (int l = 1; l < reg_q; l++) coefl[l] = beta[c->reg_xlocs[l - 1]];
                CK(cudaMemcpyAsync(c->d_coef.p, coefl.data(), sizeof(double) * reg_q, cudaMemcpyHostToDevice, c->stream));
                site_design_axpy_kernel<<<grid_for(c, n, 256), 256, 0, c->stream>>>(c->d_Xl.p, c->d_coef.p, reg_q, n, 1.0, c->d_field.p, c->d_tmp1.p);   // other_field
                LAUNCHED(c);
                op_spmv(c, c->d_linv[c->cur].p, c->d_tmp1.p, 0.0, c->d_tmp2.p);
                op_atb(c, c->d_B.p, reg_q, c->d_tmp2.p, 1, n, gvec.data());      // crossprod(sparse_chol %*% other_field, sparse_chol_X_locs)
                for (int j = 0; j < reg_q; j++) {
                    double v = 0.0;
                    for (int k = 0; k < reg_q; k++) v += iw_cov[(size_t)j + (size_t)reg_q * k] * gvec[k];
                    bmean[j] = v;
                }
                for (int k = 0; k < reg_q; k++) zz[k] = rs.norm_rand();          // :242 rnorm(length(X$locs) + 1)
                const double sd_scale = std::exp(.5 * log_scale);
                for (int j = 0; j < reg_q; j++) {                                // t(beta_interweaved_covmat_chol) %*% z
                    double v = 0.0;
                    for (int k = 0; k <= j; k++) v += iw_chol[(size_t)j + (size_t)reg_q * k] * zz[k];
                    innov[j] = bmean[j] + sd_scale * v;
                }
                beta_0 = innov[0];
                for (int l = 1; l < reg_q; l++) { beta[c->reg_xlocs[l - 1]] = innov[l]; coefl[l] = innov[l]; }
                CK(cudaMemcpyAsync(c->d_coef.p, coefl.data(), sizeof(double) * reg_q, cudaMemcpyHostToDevice, c->stream));
                site_design_axpy_kernel<<<grid_for(c, n, 256), 256, 0, c->stream>>>(c->d_Xl.p, c->d_coef.p, reg_q, n, -1.0, c->d_tmp1.p, c->d_field.p);  // :245
                LAUNCHED(c);
                CK(cudaStreamSynchronize(c->stream));                            // coefl is reused by the next iteration
            }
            op_set_beta(c, beta.data());                                         // :249 mu
        }
        mark(2);
        nvtxRangePop();
        // ---- (D) chromatic sweeps :257-275 ----
        nvtxRangePushA("nngp D chromatic Gibbs sweeps");
        if (rng_mode == NNGP_RNG_SUPPLIED) {
            ensure_zbuf(c, (size_t)nz * std::max(1, n_chromatic));
            zhost.resize((size_t)nz * std::max(1, n_chromatic));
            rs.rnorm(zhost.data(), (int64_t)nz * n_chromatic);
            CK(cudaMemcpyAsync(c->d_zbuf.p, zhost.data(), sizeof(double) * (size_t)nz * n_chromatic, cudaMemcpyHostToDevice, c->stream));
        }
        set_sweep_params(c, beta_0, log_scale, lnv, rng_mode, (double)philox_seed);
        refresh_r(c, beta_0);
        op_sweeps(c, n_chromatic);
        c->sweep_counter += (unsigned long long)n_chromatic;
        mark(3);
        nvtxRangePop();
        // ---- (E) noise variance :281-293 ----
        nvtxRangePushA("nngp E noise variance");
        op_obs_sq(c, c->d_field.p, c->d_field.p, 0);
        fetch_scalars(c, 2);
        const double ssr = c->h_pinned[0];
        for (int k = 0; k < 10; k++) {
            const double inn = 0.0 + .01 * rs.norm_rand();
            if (std::exp(lnv + inn) < var_y) {
                if (-.5 * n_obs * inn - .5 * ssr * (std::exp(-lnv - inn) - std::exp(-lnv)) > std::log(rs.unif_rand())) lnv += inn;
            }
        }
        mark(4);
        nvtxRangePop();
        // ---- (F) records :305-311 ----
        nvtxRangePushA("nngp F records");
        if (records_out) {
            records_out[(size_t)(iter - 1)] = beta_0;
            records_out[(size_t)(iter - 1) + (size_t)n_iter] = log_scale;
            records_out[(size_t)(iter - 1) + (size_t)n_iter * 2] = lnv;
            for (int k = 0; k < ns; k++) records_out[(size_t)(iter - 1) + (size_t)n_iter * (3 + k)] = shape[k];
        }
        if (reg && reg->beta_records)
            for (int k = 0; k < reg_p; k++) reg->beta_records[(size_t)(iter - 1) + (size_t)n_iter * k] = beta[k];
        if (field_records_out) {
            const double t = iter * thin;
            if (std::nearbyint(t) == t) {
                const int row = (int)t - 1;
                if (row >= 0 && row < n_frec) {
                    if (frec_on_device) {
                        record_field_kernel<<<grid_for(c, n, 256), 256, 0, c->stream>>>(c->d_frec.p, c->d_field.p, c->d_g2i.p, row, n_frec, n);
                        LAUNCHED(c);
                    } else {   // record store does not fit next to the model: one download per stored sample
                        std::vector<double> f(n);
                        download_site_vector(c, c->d_field.p, f.data());
                        for (int s = 0; s < n; s++) field_records_out[(size_t)row + (size_t)n_frec * s] = f[s];
                    }
                }
            }
        }
        if (accept_out) { accept_out[iter - 1] = acc_anc[iter]; accept_out[n_iter + iter - 1] = acc_suf[iter]; }
        mark(5);
        nvtxRangePop();
    }
    if (prof && n_iter > 0)
        std::fprintf(stderr, "[nngp chain profile] per iteration, us: ancillary %.1f  sufficient %.1f  mean-params %.1f  sweeps(%d) %.1f  noise %.1f  records %.1f\n",
                     1e6 * phase_s[0] / n_iter, 1e6 * phase_s[1] / n_iter, 1e6 * phase_s[2] / n_iter, n_chromatic, 1e6 * phase_s[3] / n_iter,
                     1e6 * phase_s[4] / n_iter, 1e6 * phase_s[5] / n_iter);
    if (frec_on_device) CK(cudaMemcpyAsync(field_records_out, c->d_frec.p, (size_t)n_frec * n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    params_io[0] = beta_0; params_io[1] = log_scale; params_io[2] = lnv; params_io[3] = logvar_suf; params_io[4] = logvar_anc;
    for (int k = 0; k < ns; k++) params_io[5 + k] = shape[k];
    if (reg) std::memcpy(reg->beta_io, beta.data(), sizeof(double) * reg_p);
}

extern "C" {

void nngp_chain_run(const int *ctx_id, const int *n_shape_, double *params_io, const int *n_iter_, const double *thin_,
                    const int *n_chromatic_, const int *iter_start_, const int *chain_index_, const int *rng_mode_,
                    const double *var_y_, double *records_out, double *field_records_out, int *accept_out, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(n_shape_ && params_io && n_iter_ && thin_ && n_chromatic_ && iter_start_ && chain_index_ && rng_mode_ && var_y_, "nngp_chain_run: null argument");
    NEED(c->have_field && c->have_obs, "nngp_chain_run: field and observations must be set first");
    chain_run_impl(c, n_shape_, params_io, n_iter_, thin_, n_chromatic_, iter_start_, chain_index_, rng_mode_, var_y_, records_out,
                   field_records_out, accept_out, nullptr);
    ABI_END
}

void nngp_regressors_set(const int *ctx_id, const int *p_, const double *X, const double *observed_field, const int *n_xlocs_,
                         const int *xlocs, const int *first_obs, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    NEED(!c->sharded, "nngp_regressors_set: not available on a sharded context");
    REQUIRE(p_ && X && observed_field && n_xlocs_, "nngp_regressors_set: null argument");
    const int p = *p_, nx = *n_xlocs_, n = c->n, n_obs = c->n_obs;
    REQUIRE(p >= 1 && nx >= 0 && nx <= p, "nngp_regressors_set: need p >= 1 and 0 <= n_xlocs <= p (got p=%d n_xlocs=%d)", p, nx);
    REQUIRE(n_obs >= 1, "nngp_regressors_set: the context has no observations");
    REQUIRE(nx == 0 || (xlocs && first_obs), "nngp_regressors_set: X$locs given without xlocs / first_obs");
    for (int l = 0; l < nx; l++) REQUIRE(xlocs[l] >= 1 && xlocs[l] <= p, "nngp_regressors_set: xlocs[%d] = %d outside 1..%d", l, xlocs[l], p);
    if (nx > 0)
        for (int i = 0; i < n; i++) REQUIRE(first_obs[i] >= 1 && first_obs[i] <= n_obs, "nngp_regressors_set: first_obs[%d] = %d outside 1..%d", i, first_obs[i], n_obs);
    use(c);
    c->reg_p = -1;
    const size_t P1 = (size_t)p + 1;
    c->d_Xa.alloc(P1 * n_obs);
    {
        std::vector<double> ones((size_t)n_obs, 1.0);
        CK(cudaMemcpyAsync(c->d_Xa.p, ones.data(), sizeof(double) * n_obs, cudaMemcpyHostToDevice, c->stream));
        CK(cudaMemcpyAsync(c->d_Xa.p + n_obs, X, sizeof(double) * (size_t)p * n_obs, cudaMemcpyHostToDevice, c->stream));
        CK(cudaStreamSynchronize(c->stream));
    }
    c->d_yobs.alloc(n_obs);
    CK(cudaMemcpyAsync(c->d_yobs.p, observed_field, sizeof(double) * n_obs, cudaMemcpyHostToDevice, c->stream));
    c->d_robs.alloc(n_obs);
    c->d_coef.alloc(P1 + 1);
    c->reg_xlocs.clear();
    if (nx > 0) {
        const int q = nx + 1;
        std::vector<double> Xl((size_t)n * q);
        for (int s = 0; s < n; s++) {
            const size_t row = (size_t)first_obs[c->i2g[s]] - 1;
            Xl[s] = 1.0;
            for (int l = 1; l < q; l++) Xl[(size_t)l * n + s] = X[row + (size_t)n_obs * (xlocs[l - 1] - 1)];
        }
        c->d_Xl.alloc((size_t)n * q);
        CK(cudaMemcpyAsync(c->d_Xl.p, Xl.data(), sizeof(double) * (size_t)n * q, cudaMemcpyHostToDevice, c->stream));
        c->d_B.alloc((size_t)n * q);
        CK(cudaStreamSynchronize(c->stream));
        for (int l = 0; l < nx; l++) c->reg_xlocs.push_back(xlocs[l] - 1);
        c->reg_q = q;
    } else {
        c->reg_q = 0;
    }
    CK(cudaStreamSynchronize(c->stream));
    c->reg_p = p;
    ABI_END
}

void nngp_chain_run_regressors(const int *ctx_id, const int *n_shape_, double *params_io, double *beta_io, const double *solve_1XT1X,
                               const double *chol_solve_1XT1X, const int *n_iter_, const double *thin_, const int *n_chromatic_,
                               const int *iter_start_, const int *chain_index_, const int *rng_mode_, const double *var_y_,
                               double *records_out, double *beta_records_out, double *field_records_out, int *accept_out, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    NEED(!c->sharded, "nngp_chain_run_regressors: not available on a sharded context");
    REQUIRE(n_shape_ && params_io && beta_io && solve_1XT1X && chol_solve_1XT1X && n_iter_ && thin_ && n_chromatic_ && iter_start_ && chain_index_ && rng_mode_ && var_y_,
            "nngp_chain_run_regressors: null argument");
    NEED(c->reg_p >= 1, "nngp_chain_run_regressors: nngp_regressors_set must be called first");
    NEED(c->have_field, "nngp_chain_run_regressors: the field must be set first");
    RegRun reg{beta_io, solve_1XT1X, chol_solve_1XT1X, beta_records_out};
    chain_run_impl(c, n_shape_, params_io, n_iter_, thin_, n_chromatic_, iter_start_, chain_index_, rng_mode_, var_y_, records_out,
                   field_records_out, accept_out, &reg);
    c->have_obs = true;                                                          // d_ymx / residuals_sum now hold y - X beta of the final state
    ABI_END
}

// ---- several chains at once (mclapply over chains, Scripts/mcmc_nngp_update_Gaussian.R:22-26; mcmc_nngp_run.R n_cores) ----
// One blocking call (so that it works through R's .C(), whose argument copies do not outlive a call): chain k runs on context
// ctx_ids[k] -- its own device, stream and device-resident state -- driven by its own host thread; at most max_concurrent chains
// are in flight.  Chains on different GPUs run in parallel; chains that share a GPU overlap on it (a sweep is a chain of
// latency-bound colour stages that leaves most of the memory system idle, so co-scheduled chains fill each other's gaps).
// Every chain's result is the one the sequential call gives: all random draws are keyed by (iter_start, chain_index).
struct ChainJob {
    Ctx *c;
    double *params, *beta, *records, *beta_records, *field_records;
    int *accept;
    int chain_index, status;
    std::string error;
};

static void run_chain_jobs(std::vector<ChainJob> &jobs, int max_concurrent, const int *n_shape, const int *n_iter, const double *thin,
                           const int *n_chromatic, const int *iter_start, const int *rng_mode, const double *var_y,
                           const double *solve_1XT1X, const double *chol_1XT1X) {
    std::atomic<int> next{0};
    auto worker = [&]() {
        for (;;) {
            const int k = next.fetch_add(1);
            if (k >= (int)jobs.size()) return;
            ChainJob &j = jobs[k];
            int *status = &j.status;
            ABI_BEGIN
            if (solve_1XT1X) {
                RegRun reg{j.beta, solve_1XT1X, chol_1XT1X, j.beta_records};
                chain_run_impl(j.c, n_shape, j.params, n_iter, thin, n_chromatic, iter_start, &j.chain_index, rng_mode, var_y, j.records,
                               j.field_records, j.accept, &reg);
                j.c->have_obs = true;
            } else {
                chain_run_impl(j.c, n_shape, j.params, n_iter, thin, n_chromatic, iter_start, &j.chain_index, rng_mode, var_y, j.records,
                               j.field_records, j.accept, nullptr);
            }
            ABI_END
            if (j.status != NNGP_OK) j.error = t_err;
        }
    };
    const int n_threads = std::max(1, std::min(max_concurrent, (int)jobs.size()));
    std::vector<std::thread> pool;
    for (int w = 1; w < n_threads; w++) pool.emplace_back(worker);
    worker();
    for (auto &th : pool) th.join();
}

static void chains_run_common(const int *n_chains_, const int *ctx_ids, const int *n_shape, double *params_io, double *beta_io,
                              const double *solve_1XT1X, const double *chol_1XT1X, const int *n_iter, const double *thin,
                              const int *n_chromatic, const int *iter_start, const int *chain_index, const int *rng_mode,
                              const double *var_y, const int *max_concurrent, double *records_out, double *beta_records_out,
                              double *field_records_out, int *accept_out, bool with_reg, int *status) {
    ABI_BEGIN
    REQUIRE(n_chains_ && ctx_ids && n_shape && params_io && n_iter && thin && n_chromatic && iter_start && chain_index && rng_mode && var_y && max_concurrent,
            "nngp_chains_run: null argument");
    REQUIRE(!with_reg || (beta_io && solve_1XT1X && chol_1XT1X), "nngp_chains_run_regressors: null argument");
    const int nc = *n_chains_, ns = *n_shape, ni = *n_iter;
    REQUIRE(nc >= 1 && ns >= 1 && ns <= 5 && ni >= 0 && *max_concurrent >= 1, "nngp_chains_run: bad sizes");
    const long long n_frec = (long long)std::nearbyint(ni * *thin);
    std::vector<ChainJob> jobs(nc);
    for (int k = 0; k < nc; k++) {
        Ctx *c = get_ctx(ctx_ids + k);
        for (int l = 0; l < k; l++) REQUIRE(jobs[l].c != c, "nngp_chains_run: chains %d and %d share context %d (a context holds the state of ONE chain)", l + 1, k + 1, ctx_ids[k]);
        NEED(!c->sharded, "nngp_chains_run: not available on a sharded context");
        NEED(c->have_field && (with_reg || c->have_obs), "nngp_chains_run: field and observations must be set first on every context");
        if (with_reg) NEED(c->reg_p >= 1, "nngp_chains_run_regressors: nngp_regressors_set must be called first on every context");
        if (with_reg && k > 0) REQUIRE(c->reg_p == jobs[0].c->reg_p, "nngp_chains_run_regressors: the contexts hold different numbers of regressors");
        ChainJob &j = jobs[k];
        j.c = c;
        j.params = params_io + (size_t)k * (5 + ns);
        j.beta = with_reg ? beta_io + (size_t)k * c->reg_p : nullptr;
        j.records = records_out ? records_out + (size_t)k * ni * (3 + ns) : nullptr;
        j.beta_records = (with_reg && beta_records_out) ? beta_records_out + (size_t)k * ni * c->reg_p : nullptr;
        j.field_records = field_records_out ? field_records_out + (size_t)k * n_frec * c->n : nullptr;
        j.accept = accept_out ? accept_out + (size_t)k * 2 * ni : nullptr;
        j.chain_index = chain_index[k];
        j.status = NNGP_OK;
    }
    run_chain_jobs(jobs, *max_concurrent, n_shape, n_iter, thin, n_chromatic, iter_start, rng_mode, var_y, with_reg ? solve_1XT1X : nullptr, chol_1XT1X);
    for (int k = 0; k < nc; k++)
        if (jobs[k].status != NNGP_OK) {
            set_error("chain %d: %s", k + 1, jobs[k].error.c_str());
            switch (jobs[k].status) {
                case NNGP_ERR_CUDA: throw CudaFail();
                case NNGP_ERR_STATE: throw StateFail();
                case NNGP_ERR_NCCL: throw NcclFail();
                case NNGP_ERR_ALLOC: throw std::bad_alloc();
                default: throw ArgFail();
            }
        }
    ABI_END
}

void nngp_chains_run(const int *n_chains, const int *ctx_ids, const int *n_shape, double *params_io, const int *n_iter, const double *thin,
                     const int *n_chromatic, const int *iter_start, const int *chain_index, const int *rng_mode, const double *var_y,
                     const int *max_concurrent, double *records_out, double *field_records_out, int *accept_out, int *status) {
    chains_run_common(n_chains, ctx_ids, n_shape, params_io, nullptr, nullptr, nullptr, n_iter, thin, n_chromatic, iter_start, chain_index,
                      rng_mode, var_y, max_concurrent, records_out, nullptr, field_records_out, accept_out, false, status);
}

void nngp_chains_run_regressors(const int *n_chains, const int *ctx_ids, const int *n_shape, double *params_io, double *beta_io,
                                const double *solve_1XT1X, const double *chol_solve_1XT1X, const int *n_iter, const double *thin,
                                const int *n_chromatic, const int *iter_start, const int *chain_index, const int *rng_mode,
                                const double *var_y, const int *max_concurrent, double *records_out, double *beta_records_out,
                                double *field_records_out, int *accept_out, int *status) {
    chains_run_common(n_chains, ctx_ids, n_shape, params_io, beta_io, solve_1XT1X, chol_solve_1XT1X, n_iter, thin, n_chromatic, iter_start,
                      chain_index, rng_mode, var_y, max_concurrent, records_out, beta_records_out, field_records_out, accept_out, true, status);
}

// One chain on a field sharded over the GPUs of THIS process (nngp_shard_connect_local): every member runs the reference loop on its
// block, on its own host thread, with the same scalar state and the same R stream; the scalars that enter a decision are all-reduced
// between the members, so they stay in step.  params_io: one parameter vector (in / out, identical on every member);
// records_out / accept_out: the scalar records (identical on every member; member 0's are returned); field_records_out: member h's
// block after member h - 1's, each round(n_iter * thin) x n_local(h), or NULL.
void nngp_shard_group_chain_run(const int *ctx_ids, const int *world, const int *n_shape, double *params_io, const int *n_iter,
                                const double *thin, const int *n_chromatic, const int *iter_start, const int *chain_index, const int *rng_mode,
                                const double *var_y, double *records_out, double *field_records_out, int *accept_out, int *status) {
    ABI_BEGIN
    REQUIRE(ctx_ids && world && n_shape && params_io && n_iter && thin && n_chromatic && iter_start && chain_index && rng_mode && var_y && *world >= 1 && *world <= 8,
            "nngp_shard_group_chain_run: bad argument");
    const int W = *world, ns = *n_shape, ni = *n_iter;
    REQUIRE(ns >= 1 && ns <= 5 && ni >= 0, "nngp_shard_group_chain_run: bad sizes");
    const long long n_frec = (long long)std::nearbyint(ni * *thin);
    std::vector<ChainJob> jobs(W);
    std::vector<std::vector<double>> p(W), rec(W);
    std::vector<std::vector<int>> acc(W);
    size_t foff = 0;
    for (int h = 0; h < W; h++) {
        Ctx *c = get_ctx(ctx_ids + h);
        NEED(c->sharded && c->world == W && c->rank == h && (c->p2p || W == 1), "nngp_shard_group_chain_run: context h must be rank h of a locally connected W-rank field");
        NEED(c->have_field && c->have_obs, "nngp_shard_group_chain_run: field and observations must be set first on every member");
        p[h].assign(params_io, params_io + 5 + ns);
        rec[h].assign((size_t)ni * (3 + ns), 0.0);
        acc[h].assign((size_t)2 * ni, 0);
        ChainJob &j = jobs[h];
        j.c = c;
        j.params = p[h].data();
        j.beta = nullptr; j.beta_records = nullptr;
        j.records = rec[h].data();
        j.field_records = field_records_out ? field_records_out + foff : nullptr;
        foff += (size_t)n_frec * c->n;
        j.accept = acc[h].data();
        j.chain_index = *chain_index;
        j.status = NNGP_OK;
    }
    for (int h = 0; h < W; h++) prepare_chain_buffers(jobs[h].c, ni, *thin, *n_chromatic, *rng_mode, field_records_out != nullptr);
    run_chain_jobs(jobs, W, n_shape, n_iter, thin, n_chromatic, iter_start, rng_mode, var_y, nullptr, nullptr);   // all members at once
    for (int h = 0; h < W; h++)
        if (jobs[h].status != NNGP_OK) {
            set_error("member %d: %s", h, jobs[h].error.c_str());
            switch (jobs[h].status) {
                case NNGP_ERR_CUDA: throw CudaFail();
                case NNGP_ERR_STATE: throw StateFail();
                case NNGP_ERR_NCCL: throw NcclFail();
                case NNGP_ERR_ALLOC: throw std::bad_alloc();
                default: throw ArgFail();
            }
        }
    for (int h = 1; h < W; h++) {
        REQUIRE(p[h] == p[0] && rec[h] == rec[0] && acc[h] == acc[0], "nngp_shard_group_chain_run: member %d fell out of step with member 0 (their scalar records differ)", h);
    }
    std::memcpy(params_io, p[0].data(), sizeof(double) * (5 + ns));
    if (records_out) std::memcpy(records_out, rec[0].data(), sizeof(double) * rec[0].size());
    if (accept_out) std::memcpy(accept_out, acc[0].data(), sizeof(int) * acc[0].size());
    ABI_END
}

void nngp_records_summary(const int *ctx_id, const int *first_row, const int *n_rows, const double *offsets, double *out, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id);
    REQUIRE(first_row && n_rows && out && *first_row >= 1 && *n_rows >= 1, "nngp_records_summary: bad argument");
    NEED(c->frec_rows > 0 && c->d_frec.p, "nngp_records_summary: no device-resident field records (run nngp_chain_run with field records first)");
    REQUIRE(*first_row - 1 + *n_rows <= c->frec_rows, "nngp_records_summary: rows %d..%d exceed the %d stored samples", *first_row, *first_row + *n_rows - 1, c->frec_rows);
    use(c);
    const int n = c->n, k = *n_rows;
    DevBuf<double> scratch, dout, doff;
    scratch.alloc((size_t)n * k);
    dout.alloc((size_t)n * 5);
    if (offsets) { doff.alloc(k); CK(cudaMemcpyAsync(doff.p, offsets, sizeof(double) * k, cudaMemcpyHostToDevice, c->stream)); }
    records_summary_kernel<<<(n + 127) / 128, 128, 0, c->stream>>>(c->d_frec.p, c->frec_rows, *first_row - 1, k, offsets ? doff.p : nullptr, n, dout.p, scratch.p);
    LAUNCHED(c);
    CK(cudaMemcpyAsync(out, dout.p, sizeof(double) * (size_t)n * 5, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    scratch.release(); dout.release(); doff.release();
    ABI_END
}

void nngp_time_op(const int *ctx_id, const int *op_, const int *reps_, const int *flush_l2_, double *ms_out, int *launches_out, int *status) {
    ABI_BEGIN
    Ctx *c = get_ctx(ctx_id, true);   // no timed op writes the field, r or the current factor; the sweeps keep r current
    NEED(!c->sharded || *op_ != 4 || c->world == 1 || (c->p2p && c->can_solve), "nngp_time_op: the triangular solve of a sharded context needs the peer-to-peer transport");
    REQUIRE(op_ && reps_ && flush_l2_ && ms_out && *reps_ >= 1, "nngp_time_op: bad argument");
    const int op = *op_;
    use(c);
    NEED(c->have_slot(NNGP_SLOT_CURRENT), "nngp_time_op: build and commit a factor first");
    if (!c->committed) op_commit(c);
    if (op == 0) NEED(c->have_cc, "nngp_time_op(factor): call nngp_factor_build once first");
    if (op == 2 || op == 6) {
        NEED(c->can_sweep, "this context was created without a colouring (all-zero coloring): it cannot run Gibbs sweeps");
        NEED(c->have_field && c->have_obs, "nngp_time_op(sweep): field and observations must be set first");
        const SweepParams *sp = reinterpret_cast<SweepParams *>(c->h_pinned + 32);
        set_sweep_params(c, sp->beta0, -std::log(sp->e_ls > 0 ? sp->e_ls : 1.0), -std::log(sp->e_ln > 0 ? sp->e_ln : 1.0), NNGP_RNG_PHILOX, 12345.0);
        refresh_r(c, sp->beta0);
    }
    if (op == 1 || op == 3 || op == 4 || op == 6) NEED(c->have_field, "nngp_time_op: field must be set first");
    CK(cudaStreamSynchronize(c->stream));
    for (int r = 0; r < *reps_; r++) {
        if (*flush_l2_) flush_l2(c);
        c->launches_in_op = 0;
        CK(cudaEventRecord(c->ev0, c->stream));
        switch (op) {
            case 0: op_factor_build(c, NNGP_SLOT_PROPOSAL, c->last_cc); break;
            case 1: op_loglik_sums(c, c->linv_slot(NNGP_SLOT_CURRENT), c->d_field.p, 0.0, 0, false); break;
            case 2: op_sweeps(c, 1); c->sweep_counter++; break;
            case 3: op_spmv(c, c->linv_slot(NNGP_SLOT_CURRENT), c->d_field.p, 0.0, c->d_tmp1.p); break;
            case 4: op_spmv(c, c->linv_slot(NNGP_SLOT_CURRENT), c->d_field.p, 0.0, c->d_tmp1.p);
                    op_sptrsv(c, c->linv_slot(NNGP_SLOT_CURRENT), c->d_tmp1.p, c->d_tmp2.p, nullptr, 0.0, 1.0); break;
            case 5: op_commit(c); break;
            case 6: op_sweeps(c, 1); c->sweep_counter++;
                    op_loglik_sums(c, c->linv_slot(NNGP_SLOT_CURRENT), c->d_field.p, 0.0, 0, true); break;
            default: REQUIRE(false, "nngp_time_op: unknown op %d", op);
        }
        CK(cudaEventRecord(c->ev1, c->stream));
        CK(cudaEventSynchronize(c->ev1));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
        ms_out[r] = ms;
        if (launches_out) *launches_out = (int)c->launches_in_op;
    }
    CK(cudaGetLastError());
    ABI_END
}

// Times `reps` repetitions of one op enqueued on SEVERAL contexts at once (their streams run concurrently on the device(s)):
// how much chains that share a GPU overlap.  op: 2 = one Gibbs sweep, 6 = sweep + log-lik.  ms_out[0] = time from the first
// context's start event to the last context's end event, measured with CUDA events per stream (max over the contexts of a
// common-origin interval); the contexts must live on ONE device.
void nngp_time_op_group(const int *ctx_ids, const int *n_ctx, const int *op_, const int *reps_, double *ms_out, int *status) {
    ABI_BEGIN
    REQUIRE(ctx_ids && n_ctx && op_ && reps_ && ms_out && *n_ctx >= 1 && *n_ctx <= 16 && *reps_ >= 1 && (*op_ == 2 || *op_ == 6), "nngp_time_op_group: bad argument");
    const int nc = *n_ctx;
    std::vector<Ctx *> cs(nc);
    for (int k = 0; k < nc; k++) {
        cs[k] = get_ctx(ctx_ids + k, true);
        NEED(!cs[k]->sharded && cs[k]->can_sweep && cs[k]->have_slot(NNGP_SLOT_CURRENT) && cs[k]->have_field && cs[k]->have_obs, "nngp_time_op_group: every context needs a factor, a field and observations");
        REQUIRE(cs[k]->device == cs[0]->device, "nngp_time_op_group: the contexts must share a device");
    }
    use(cs[0]);
    for (Ctx *c : cs) {
        if (!c->committed) op_commit(c);
        const SweepParams *sp = reinterpret_cast<SweepParams *>(c->h_pinned + 32);
        set_sweep_params(c, sp->beta0, -std::log(sp->e_ls > 0 ? sp->e_ls : 1.0), -std::log(sp->e_ln > 0 ? sp->e_ln : 1.0), NNGP_RNG_PHILOX, 12345.0);
        refresh_r(c, sp->beta0);
        op_sweeps(c, 1);   // instantiates the graph outside the timed region
        c->sweep_counter++;
        CK(cudaStreamSynchronize(c->stream));
    }
    // a common origin: every stream waits for one event recorded on the first stream
    CK(cudaEventRecord(cs[0]->ev0, cs[0]->stream));
    for (int k = 1; k < nc; k++) CK(cudaStreamWaitEvent(cs[k]->stream, cs[0]->ev0, 0));
    for (int r = 0; r < *reps_; r++)
        for (Ctx *c : cs) {
            op_sweeps(c, 1);
            c->sweep_counter++;
            if (*op_ == 6) op_loglik_sums(c, c->linv_slot(NNGP_SLOT_CURRENT), c->d_field.p, 0.0, 0, true);
        }
    for (Ctx *c : cs) CK(cudaEventRecord(c->ev1, c->stream));
    double worst = 0.0;
    for (Ctx *c : cs) {
        CK(cudaEventSynchronize(c->ev1));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, cs[0]->ev0, c->ev1));
        worst = std::max(worst, (double)ms);
    }
    ms_out[0] = worst;
    ABI_END
}

// measured FP64 FMA throughput of the device (GFLOP/s, 2 flops per DFMA): dependent-free DFMA chains on every SM, best of 5
void nngp_fp64_peak(const int *device, double *gflops, int *status) {
    ABI_BEGIN
    REQUIRE(device && gflops, "nngp_fp64_peak: null argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { set_error("no CUDA device: libnngp_b200 has no CPU fallback"); throw CudaFail(); }
    REQUIRE(*device >= 0 && *device < ndev, "device %d out of range (%d devices)", *device, ndev);
    CK(cudaSetDevice(*device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, *device));
    double *d_out = nullptr;
    CK(cudaMalloc(&d_out, sizeof(double)));
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    const int blocks = prop.multiProcessorCount * 8, iters = 4096;
    double best = 0.0;
    for (int rep = 0; rep < 6; rep++) {
        CK(cudaEventRecord(e0, 0));
        fp64_peak_kernel<<<blocks, 256>>>(d_out, iters, 1.0000001, 1e-9);
        CK(cudaEventRecord(e1, 0));
        CK(cudaEventSynchronize(e1));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        g_launches.fetch_add(1, std::memory_order_relaxed);
        const double flops = (double)blocks * 256.0 * iters * 64.0 * 2.0;
        if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e9);
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d_out);
    *gflops = best;
    ABI_END
}

}  // extern "C"
