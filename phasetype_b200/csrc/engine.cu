/*
 * engine.cu -- lifecycle and sweep orchestration of the B200 Gibbs engine (layer 2 of
 * include/pht_b200.h).  One engine = one GPU = one shard of the observations.
 *
 * A sweep is the body of the reference's iteration loop (src/PHT_MCMC_Aslett.c:268-405):
 *     k_assemble -> [k_spectral] -> path kernel of the selected method -> [all-reduce of
 *     the statistics block over NCCL] -> k_update
 * enqueued on one stream with no host synchronisation in between, and captured once into
 * a CUDA graph that is replayed per sweep (the sweep index lives in device memory).
 */
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cstdarg>
#include <cmath>
#include <string>
#include <vector>
#include <algorithm>
#include <thread>
#include <dlfcn.h>
#include <unistd.h>
#include <time.h>
#include "engine_internal.h"
#include "pht_unif.h"

/* ---------------------------------------------------------------- errors */
static thread_local char g_err[512] = "";
static int fail(const char *fmt, ...) {
    va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof(g_err), fmt, ap); va_end(ap);
    return -1;
}
extern "C" const char *pht_last_error(void) { return g_err; }
#define CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); } while (0)

/* ---------------------------------------------------------------- NCCL (loaded lazily) */
typedef struct ncclComm *ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
struct NcclApi {
    void *h = nullptr;
    int (*GetUniqueId)(ncclUniqueId *) = nullptr;
    int (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    int (*CommDestroy)(ncclComm_t) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
};
static NcclApi g_nccl;
static int nccl_load() {
    if (g_nccl.h) return 0;
    const char *names[] = { "libnccl.so.2", "libnccl.so" };
    for (const char *nm : names) { g_nccl.h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL); if (g_nccl.h) break; }
    if (!g_nccl.h) return fail("NCCL not found: %s", dlerror());
    g_nccl.GetUniqueId = (int (*)(ncclUniqueId *))dlsym(g_nccl.h, "ncclGetUniqueId");
    g_nccl.CommInitRank = (int (*)(ncclComm_t *, int, ncclUniqueId, int))dlsym(g_nccl.h, "ncclCommInitRank");
    g_nccl.CommDestroy = (int (*)(ncclComm_t))dlsym(g_nccl.h, "ncclCommDestroy");
    g_nccl.AllReduce = (int (*)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t))dlsym(g_nccl.h, "ncclAllReduce");
    g_nccl.GetErrorString = (const char *(*)(int))dlsym(g_nccl.h, "ncclGetErrorString");
    if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.CommDestroy || !g_nccl.AllReduce)
        return fail("NCCL symbols missing");
    return 0;
}
static const int NCCL_INT64 = 4, NCCL_SUM = 0;     /* ncclInt64, ncclSum (stable enum values of nccl.h) */

/* ---------------------------------------------------------------- engine */
/* method 64 with visits: the observations without visits in the ordinary layout of their own (y, flags, u, local index and
 * group offsets), run by the per-observation kernels; the panel observations in theirs (the same, plus chunk offsets and
 * the visit CSR) and the beta scratch of k_unif_panel_paths, with its hand-out counter; both by group, then by decreasing y */
struct PanelBufs {
    double *py = nullptr, *pu = nullptr; uint8_t *pc = nullptr; uint32_t *pperm = nullptr; unsigned long long *pgofs = nullptr;
    double *vy = nullptr, *vu = nullptr, *vt = nullptr, *beta = nullptr; uint8_t *vc = nullptr; uint32_t *vperm = nullptr, *vm = nullptr;
    unsigned long long *vgofs = nullptr, *vcoff = nullptr, *voff = nullptr, *vnext = nullptr;
    long n_plain = 0, n_panel = 0;
};

struct pht_engine {
    pht_config cfg;
    std::vector<int> T; std::vector<double> C, nu, zeta;
    long l_local = 0;
    cudaStream_t stream = nullptr;
    /* device buffers */
    double *d_y = nullptr; uint8_t *d_cens = nullptr;
    double *d_ys = nullptr; uint8_t *d_cs = nullptr; uint32_t *d_perm = nullptr;   /* MHRS: the same observations by decreasing y */
    uint32_t *d_glist = nullptr; XchgWindow *d_xw = nullptr;                        /* MHRS global tail */
    XchgWindow *xpeer[PHT_MAX_WORLD] = {}; std::vector<void *> ipc_opened; bool peers_attached = false;
    bool peer_reduce = false;          /* statistics all-reduced by k_allreduce_peer through the windows (else NCCL, if a communicator exists) */
    uint32_t k_switch = 1u << 15;
    double *d_model = nullptr; long long *d_stats = nullptr; DevState *d_state = nullptr;
    int *d_T = nullptr; double *d_C = nullptr, *d_nu = nullptr, *d_zeta = nullptr;
    int *d_var_ptr = nullptr, *d_cell_i = nullptr, *d_cell_j = nullptr;
    TailItem *d_items = nullptr; uint32_t *d_pend0 = nullptr, *d_pend1 = nullptr, *d_done = nullptr;
    unsigned long long *d_found = nullptr; uint32_t item_cap = 0;
    double *d_res = nullptr; int res_rows = 0;
    double *d_beta = nullptr, *d_pires = nullptr;      /* Dirichlet prior of pi (n) and the pi draws of the last run (res_rows x n) */
    uint32_t *d_idx_exact = nullptr, *d_idx_cens = nullptr; unsigned long long n_exact = 0, n_cens = 0;   /* ECS launch lists */
    std::vector<uint8_t> h_cens;       /* host copy of the flags (ECS parity ranges) */
    double *d_inject = nullptr;        /* host-supplied evals | Q | Qinv (parity hook), else nullptr */
    void *d_flush = nullptr; size_t flush_bytes = 0;   /* L2 flush scratch (measurement aid) */
    ModelLayout L;
    int grid_blocks = 0, tail_blocks = 0, replay_blocks = 0;
    uint4 *d_recs = nullptr;           /* MHRS search -> replay records, one per observation position */
    /* MHRS interval bounds (pht_engine_set_upper): u in upload order, u in the sorted layout, u of each tail item; the
     * grids of the kernel instances that read them */
    double *d_u = nullptr, *d_us = nullptr, *d_item_u = nullptr;
    int iv_blocks[3] = { 0, 0, 0 };
    /* method 64: the uniformisation table (pht_unif.h) and the longest time span it must cover (max of y and of u - y) */
    double *d_unif = nullptr; double unif_tmax = 0.0;
    /* method 64, several chains (pht_engine_set_chains): model, stats, table, res and pires hold `chains` blocks, chain 0
     * first; the chains' Philox keys (2 x u32 each) and observation counters; the seed that NULL keys count from */
    int chains = 1; uint32_t *d_keys = nullptr; unsigned long long *d_cnext = nullptr; uint64_t base_seed = 0;
    int chain_blocks = 0;              /* grid of the several-chain path kernel */
    /* method 64, groups (pht_engine_set_groups): G structures in d_T / d_C and the (group, cell) CSR; model, stats, table and
     * counters per (chain, group) unit, block c G + g.  With G > 1: each group's table span (gtmax), its range of the
     * grouped layout (gofs, G + 1 offsets), the layout itself (by group, then by decreasing y: y, flags, permutation and u
     * when bounds are set) and the host copy of the group ids in upload order */
    int groups = 1;
    double *d_gtmax = nullptr; unsigned long long *d_gofs = nullptr;
    double *d_gys = nullptr, *d_gus = nullptr; uint8_t *d_gcs = nullptr; uint32_t *d_gperm = nullptr;
    std::vector<uint8_t> h_group;
    /* method 64, delayed entry (pht_engine_set_entry): the ages in upload order (device and host), the truncated
     * observations (a > 0) by decreasing a with their local indices, their ghost counts and offsets, the entry tables,
     * the ghost counter, the scan's scratch and the ghost kernel's grid */
    bool entry_set = false; std::vector<double> h_entry;
    double *d_entry = nullptr, *d_ea = nullptr; uint32_t *d_eobs = nullptr; long n_trunc = 0;
    unsigned *d_eM = nullptr; unsigned long long *d_eoff = nullptr, *d_enext = nullptr; double *d_etab = nullptr;
    void *d_escan = nullptr; size_t escan_bytes = 0; int ghost_blocks = 0, count_blocks = 0;
    /* method 64, counts (pht_engine_set_counts): the counts in upload order; the records below the threshold expanded into
     * the ordinary layout (y, flags, u, the expanded index of every unit) with its group offsets, run by the per-observation
     * kernels; the records at or above it (y, flags, u, expanded index of unit 0) and their work items, run by
     * k_unif_records; its hand-out counter and grid; the threshold and the chunk size */
    bool counts_set = false; std::vector<uint32_t> h_counts;
    double *d_cy = nullptr, *d_cu = nullptr; uint8_t *d_cc = nullptr; uint32_t *d_cperm = nullptr; unsigned long long *d_cgofs = nullptr;
    long n_low = 0;
    double *d_ry = nullptr, *d_ru = nullptr; uint8_t *d_rc = nullptr; uint32_t *d_rbase = nullptr; uint4 *d_ritems = nullptr;
    long n_items = 0; unsigned long long *d_rnext = nullptr; int rec_blocks = 0;
    uint32_t counts_threshold = 0, counts_chunk = 0;
    /* method 64, panel observations (pht_engine_set_visits): the visits in upload order (host CSR) and the two layouts
     * (PanelBufs below); the panel kernel's grid */
    bool visits_set = false; std::vector<int64_t> h_voff; std::vector<double> h_vt; std::vector<uint32_t> h_vm;
    PanelBufs pan; int panel_blocks = 0;
    /* method 64, misclassified panel observations (pht_engine_set_stage_visits; h_vm then holds stage indices): the stages
     * (0: mask visits), the support of each column of E as a phase mask, E and K per chain (chains x n x stages), the prior
     * (nullptr: E fixed), the E draws of the last run (chains x eres_rows x n x stages) and the kernel's grid */
    int stages = 0; std::vector<uint32_t> h_colmask;
    double *d_E = nullptr, *d_alpha = nullptr, *d_Eres = nullptr; unsigned long long *d_K = nullptr;
    int eres_rows = 0, emis_blocks = 0;
    /* graph */
    cudaGraphExec_t graph_exec = nullptr; int graph_res_rows = -1; double *graph_res = nullptr;
    unsigned long long graph_launches = 0;      /* kernels one replay of the captured sweep launches */
    /* nccl */
    ncclComm_t comm = nullptr;
    /* timing */
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::vector<cudaEvent_t> kev; int kev_used = 0;
    unsigned long long launches = 0;
};

extern "C" int pht_device_count(void) {
    int c = 0;
    if (cudaGetDeviceCount(&c) != cudaSuccess) { cudaGetLastError(); return 0; }
    return c;
}

extern "C" int pht_choose_zbits(double sum_y) {
    if (!(sum_y > 0.0) || !std::isfinite(sum_y)) return 30;
    int b = 62 - (int)std::ceil(std::log2(16.0 * sum_y + 1.0));
    if (b > 52) b = 52;
    if (b < 0) b = 0;
    return b;
}

static SweepParams sweep_params(pht_engine *e) {
    SweepParams p; memset(&p, 0, sizeof(p));
    p.y = e->d_y; p.cens = e->d_cens; p.l_local = e->l_local;
    p.obs_rank = (uint32_t)e->cfg.rank; p.obs_world = (uint32_t)e->cfg.world;
    p.model = e->d_model; p.stats = e->d_stats; p.state = e->d_state;
    p.n = e->cfg.n; p.m = e->cfg.m; p.mhit = e->cfg.mhit; p.zbits = e->cfg.zbits;
    p.k0 = (uint32_t)e->cfg.seed; p.k1 = (uint32_t)(e->cfg.seed >> 32);
    pht_roundkeys_init(&p.rk, p.k0, p.k1);
    p.items = e->d_items; p.pend0 = e->d_pend0; p.pend1 = e->d_pend1; p.done = e->d_done; p.found = e->d_found;
    p.item_cap = e->item_cap; p.mhrs_cap = e->cfg.mhrs_cap;
    if (e->d_ys) { p.y = e->d_ys; p.cens = e->d_cs; p.perm = e->d_perm; }      /* production layout: decreasing y */
    p.glist = e->d_glist; p.k_switch = e->k_switch; p.recs = e->d_recs;
    if (e->peers_attached) { p.xw = e->d_xw; for (int r = 0; r < e->cfg.world && r < PHT_MAX_WORLD; r++) p.xpeer[r] = e->xpeer[r]; }
    if (e->d_u) { p.u = e->d_ys ? e->d_us : e->d_u; p.item_u = e->d_item_u; }
    p.chains = e->chains; p.ckeys = e->d_keys; p.cnext = e->d_cnext;
    p.groups = e->groups;
    if (e->groups > 1) {                           /* the grouped layout: each group a contiguous range (e->d_gofs) */
        p.y = e->d_gys; p.cens = e->d_gcs; p.perm = e->d_gperm;
        if (e->d_u) p.u = e->d_gus;
    }
    return p;
}
static UpdateParams update_params(pht_engine *e, double *res, int res_rows) {
    UpdateParams u; memset(&u, 0, sizeof(u));
    u.model = e->d_model; u.stats = e->d_stats; u.state = e->d_state; u.res = res; u.res_rows = res_rows;
    u.T = e->d_T; u.C = e->d_C; u.nu = e->d_nu; u.zeta = e->d_zeta;
    u.var_ptr = e->d_var_ptr; u.cell_i = e->d_cell_i; u.cell_j = e->d_cell_j;
    u.n = e->cfg.n; u.m = e->cfg.m; u.zbits = e->cfg.zbits;
    u.k0 = (uint32_t)e->cfg.seed; u.k1 = (uint32_t)(e->cfg.seed >> 32);
    u.beta = e->d_beta; u.pires = (e->d_beta && res) ? e->d_pires : nullptr;
    u.chains = e->chains; u.ckeys = e->d_keys; u.cnext = e->d_cnext;
    u.groups = e->groups; u.gtmax = e->groups > 1 ? e->d_gtmax : nullptr;
    return u;
}

/* ---- device memory for the large per-call buffers (observations, sorted layout, records, tail lists): stream-ordered
 * allocations from the device's default pool, whose release threshold is raised so that the memory of a finished call
 * is reused by the next one.  Two reasons: a call allocates ~0.5 GB, and once peer access is on (several GPUs in one
 * process) every plain cudaMalloc/cudaFree also maps/unmaps the block on the peers -- 100..700 ms per call measured on
 * 2 GPUs.  Pool memory is not peer-mapped; the exchange window, which must be, stays a plain allocation.
 * PHT_B200_NO_POOL=1 goes back to cudaMalloc/cudaFree; pht_release_device_memory() hands the cached memory back. */
static bool pool_off() { static const bool off = getenv("PHT_B200_NO_POOL") != nullptr; return off; }
cudaError_t pht_dev_alloc(void **p, size_t bytes, cudaStream_t st) {
    if (pool_off()) return cudaMalloc(p, bytes);
    return cudaMallocAsync(p, bytes, st);
}
cudaError_t pht_dev_free(void *p, cudaStream_t st) {
    if (!p) return cudaSuccess;
    if (pool_off()) return cudaFree(p);
    return cudaFreeAsync(p, st);
}
static void pool_keep(int dev) {
    cudaMemPool_t pool;
    if (!pool_off() && cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
        unsigned long long thr = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    cudaGetLastError();
}
extern "C" int pht_release_device_memory(void) {
    int ndev = 0, cur = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess) { cudaGetLastError(); return 0; }
    cudaGetDevice(&cur);
    for (int d = 0; d < ndev; d++) {
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, d) == cudaSuccess) { cudaSetDevice(d); cudaDeviceSynchronize(); cudaMemPoolTrimTo(pool, 0); }
    }
    cudaSetDevice(cur); cudaGetLastError();
    return 0;
}

static int method_of(const pht_config &c) {       /* dispatch priority of src/PHT_MCMC_Aslett.c:325-337 */
    if (c.method & PHT_METHOD_MHRS) return PHT_METHOD_MHRS;
    if (c.method & PHT_METHOD_DCS) return PHT_METHOD_DCS;
    if (c.method & PHT_METHOD_ECS) return PHT_METHOD_ECS;
    if (c.method & PHT_METHOD_MHS_HOBOLTH) return PHT_METHOD_MHS_HOBOLTH;      /* the engine's extension (pht_b200.h) */
    if (c.method & PHT_METHOD_MHS_ASLETT) return PHT_METHOD_MHS_ASLETT;
    if (c.method & PHT_METHOD_UNIF) return PHT_METHOD_UNIF;
    return 0;
}

static int counts_build(pht_engine *e);      /* pht_engine_set_counts: the counted records' layouts */
static int visits_build(pht_engine *e);      /* pht_engine_set_visits: the panel and plain layouts */
static int engine_visits_reachable(pht_engine *e, const int64_t *off, const double *t, const uint32_t *mask, const double *pi,
                                   int G, const int *T, const double *C, const uint8_t *gid);

static UnifPanel panel_args(const PanelBufs &b) {
    UnifPanel V; memset(&V, 0, sizeof(V));
    V.y = b.vy; V.u = b.vu; V.cens = b.vc; V.perm = b.vperm; V.gofs = b.vgofs; V.coff = b.vcoff;
    V.voff = b.voff; V.vt = b.vt; V.vm = b.vm; V.beta = b.beta; V.next = b.vnext;
    return V;
}

/* the observation process of stage visits; the E draws recorded only when the sweep records its rows */
static UnifEmis emis_args(const pht_engine *e, bool record) {
    UnifEmis X; memset(&X, 0, sizeof(X));
    X.E = e->d_E; X.alpha = e->d_alpha; X.K = e->d_K; X.Eres = record ? e->d_Eres : nullptr; X.S = e->stages;
    return X;
}

/* the panel kernel of the visits set: k_unif_emis_paths for stage visits, else k_unif_panel_paths */
static cudaError_t launch_panel_kernel(pht_engine *e, const SweepParams &p, const UnifPanel &V) {
    if (e->stages) return pht_launch_unif_emis(p, e->d_unif, V, emis_args(e, false), e->emis_blocks, e->stream);
    return pht_launch_unif_panel(p, e->d_unif, V, e->panel_blocks, e->stream);
}

/* the phase mask of every visit: the masks themselves (colmask empty), or for stage visits the support of the stage's
 * column of E (colmask[o]) */
static std::vector<uint32_t> visit_masks(const uint32_t *v, size_t count, const std::vector<uint32_t> &colmask) {
    std::vector<uint32_t> mk(v, v + count);
    if (!colmask.empty()) for (uint32_t &x : mk) x = colmask[x];
    return mk;
}

/* method 64 with visits: the observations without visits through the per-observation kernels (their own layout and group
 * offsets), then k_unif_panel_paths over the panel observations; both add to the same statistics blocks */
static int enqueue_panel(pht_engine *e, const SweepParams &p) {
    const PanelBufs &b = e->pan;
    if (b.n_plain > 0) {
        SweepParams q = p;
        q.y = b.py; q.cens = b.pc; q.perm = b.pperm; q.u = b.pu; q.l_local = b.n_plain;
        CU(pht_launch_unif(q, e->d_unif, q.groups > 1 ? b.pgofs : nullptr, q.chains > 1 || q.groups > 1 ? e->chain_blocks : e->grid_blocks, e->stream));
        e->launches++;
    }
    CU(launch_panel_kernel(e, p, panel_args(b)));
    return 0;                                      /* enqueue_paths counts the panel kernel */
}

/* method 64 with counts: the expanded records below the threshold through the per-observation kernels (their own layout
 * and group offsets), then k_unif_records over the items of the others; both add to the same statistics blocks */
static int enqueue_counts(pht_engine *e, const SweepParams &p) {
    if (e->n_low > 0) {
        SweepParams q = p;
        q.y = e->d_cy; q.cens = e->d_cc; q.perm = e->d_cperm; q.u = e->d_cu; q.l_local = e->n_low;
        CU(pht_launch_unif(q, e->d_unif, q.groups > 1 ? e->d_cgofs : nullptr, q.chains > 1 || q.groups > 1 ? e->chain_blocks : e->grid_blocks, e->stream));
        e->launches++;
    }
    if (e->n_items > 0) {
        UnifRecords R; memset(&R, 0, sizeof(R));
        R.y = e->d_ry; R.u = e->d_ru; R.cens = e->d_rc; R.base = e->d_rbase; R.items = e->d_ritems; R.n_items = e->n_items; R.next = e->d_rnext;
        CU(pht_launch_unif_records(p, e->d_unif, R, e->rec_blocks, e->stream));
        e->launches++;
    }
    e->launches--;                                 /* enqueue_paths counts one */
    return 0;
}

/* enqueue the path kernel of the configured method */
static int enqueue_paths(pht_engine *e, const SweepParams &p, const uint32_t *idx_exact = nullptr, unsigned long long n_exact = 0,
                         const uint32_t *idx_cens = nullptr, unsigned long long n_cens = 0, bool lists_given = false) {
    switch (method_of(e->cfg)) {
    case PHT_METHOD_ECS:
        if (lists_given) CU(pht_launch_ecs(p, e->grid_blocks, idx_exact, n_exact, idx_cens, n_cens, e->stream));
        else CU(pht_launch_ecs(p, e->grid_blocks, e->d_idx_exact, e->n_exact, e->d_idx_cens, e->n_cens, e->stream));
        e->launches += (lists_given ? (n_exact != 0) + (n_cens != 0) : (e->n_exact != 0) + (e->n_cens != 0)) - 1;
        break;
    case PHT_METHOD_MHRS:
        if (p.u) CU(pht_launch_mhrs(p, e->iv_blocks[0], e->iv_blocks[1], e->iv_blocks[2], e->stream));
        else CU(pht_launch_mhrs(p, e->grid_blocks, e->tail_blocks, e->replay_blocks, e->stream));
        e->launches += 2; break;
    case PHT_METHOD_DCS: CU(pht_launch_dcs(p, e->grid_blocks, e->stream)); e->launches++; break;           /* unit machine + complex-spectrum kernel */
    case PHT_METHOD_MHS_HOBOLTH: CU(pht_launch_dcs(p, e->grid_blocks, e->stream, true)); e->launches++; break;
    case PHT_METHOD_UNIF:
        if (e->counts_set) { if (enqueue_counts(e, p)) return -1; break; }
        if (e->visits_set && p.outB == nullptr) { if (enqueue_panel(e, p)) return -1; break; }   /* (pht_engine_paths: panel_window) */
        CU(pht_launch_unif(p, e->d_unif, p.groups > 1 ? e->d_gofs : nullptr, p.chains > 1 || p.groups > 1 ? e->chain_blocks : e->grid_blocks, e->stream));
        break;
    case PHT_METHOD_MHS_ASLETT:
        /* every observation through one kernel: the window list in parity mode, else the whole shard (identity) */
        if (lists_given) CU(pht_launch_mhs_aslett(p, e->grid_blocks, idx_exact, n_exact, e->stream));
        else CU(pht_launch_mhs_aslett(p, e->grid_blocks, nullptr, (unsigned long long)e->l_local, e->stream));
        break;
    default: return fail("sampling method %d has no kernel in this build", e->cfg.method);
    }
    e->launches++;
    return 0;
}

/* k_assemble (+ spectral data for ECS / DCS, the uniformisation table for method 64): everything the path kernels read
 * from the model block */
static int enqueue_model(pht_engine *e, const UpdateParams &u) {
    CU(pht_launch_assemble(u, e->stream)); e->launches++;
    if (method_of(e->cfg) == PHT_METHOD_UNIF) {
        CU(pht_launch_unif_table(u, e->d_unif, e->unif_tmax, e->stream)); e->launches++;
    } else if (method_of(e->cfg) != PHT_METHOD_MHRS) {
        CU(pht_launch_spectral(u, e->d_inject, e->stream)); e->launches++;
    }
    return 0;
}

/* method 64 with entry ages: entry tables, ghost counts, their scan and the ghost paths of the truncated observations,
 * reduced into the same statistics block (nothing is launched without truncated observations) */
static int enqueue_entry(pht_engine *e, const UpdateParams &u, const SweepParams &p) {
    if (!e->entry_set || e->n_trunc == 0) return 0;
    UnifEntry E; memset(&E, 0, sizeof(E));
    E.a = e->d_ea; E.obs = e->d_eobs; E.first = 0; E.count = e->n_trunc; E.M = e->d_eM; E.off = e->d_eoff;
    E.etab = e->d_etab; E.next = e->d_enext; E.scan_tmp = e->d_escan; E.scan_bytes = e->escan_bytes;
    E.count_blocks = e->count_blocks;
    CU(pht_launch_unif_entry(u, p, e->d_unif, E, e->ghost_blocks, PHT_ENTRY_COUNTS | PHT_ENTRY_GHOSTS, e->stream));
    e->launches += 5;
    return 0;
}

static int enqueue_sweep(pht_engine *e, double *res, int res_rows, bool time_kernel) {
    UpdateParams u = update_params(e, res, res_rows);
    if (enqueue_model(e, u)) return -1;
    SweepParams p = sweep_params(e);
    if (time_kernel && e->kev_used + 2 <= (int)e->kev.size()) CU(cudaEventRecord(e->kev[e->kev_used++], e->stream));
    if (enqueue_paths(e, p)) return -1;
    if (enqueue_entry(e, u, p)) return -1;          /* the ghost pass is path work: inside the path-kernel timing */
    if (time_kernel && (e->kev_used & 1)) CU(cudaEventRecord(e->kev[e->kev_used++], e->stream));
    if (e->peer_reduce) {
        ReduceParams r; memset(&r, 0, sizeof(r));
        r.stats = e->d_stats; r.len = stats_len(e->cfg.n); r.state = e->d_state; r.xw = e->d_xw;
        r.rank = (uint32_t)e->cfg.rank; r.world = (uint32_t)e->cfg.world;
        for (int k = 0; k < e->cfg.world && k < PHT_MAX_WORLD; k++) r.xpeer[k] = e->xpeer[k];
        CU(pht_launch_peer_allreduce(r, e->stream)); e->launches++;
    } else if (e->comm) {
        CU(pht_launch_pack_error(u, e->stream)); e->launches++;
        int rc = g_nccl.AllReduce(e->d_stats, e->d_stats, (size_t)stats_len(e->cfg.n), NCCL_INT64, NCCL_SUM, e->comm, e->stream);
        if (rc != 0) return fail("ncclAllReduce failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?");
    }
    CU(pht_launch_update(u, e->stream)); e->launches++;
    if (e->stages && e->d_alpha) { CU(pht_launch_emis_update(u, emis_args(e, res != nullptr), e->stream)); e->launches++; }
    return 0;
}

extern "C" void pht_engine_destroy(pht_engine *e) {
    if (!e) return;
    const bool timing = getenv("PHT_B200_TIMING") != nullptr;
    struct timespec ts0; clock_gettime(CLOCK_MONOTONIC, &ts0);
    auto stage = [&](const char *what) {
        if (!timing) return;
        struct timespec t; clock_gettime(CLOCK_MONOTONIC, &t);
        fprintf(stderr, "[pht_engine_destroy] %-27s %8.3f ms\n", what, (t.tv_sec - ts0.tv_sec) * 1e3 + (t.tv_nsec - ts0.tv_nsec) * 1e-6);
        ts0 = t;
    };
    cudaSetDevice(e->cfg.device);
    if (e->stream) cudaStreamSynchronize(e->stream);
    /* the graph holds captured NCCL work: it must go before the communicator it refers to */
    if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }
    stage("sync, graph");
    if (e->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(e->comm);
    for (cudaEvent_t ev : e->kev) cudaEventDestroy(ev);
    if (e->ev0) cudaEventDestroy(e->ev0);
    if (e->ev1) cudaEventDestroy(e->ev1);
    for (void *q : e->ipc_opened) cudaIpcCloseMemHandle(q);
    stage("events, ipc");
    { const PanelBufs &b = e->pan;
      void *pb[] = { b.py, b.pu, b.pc, b.pperm, b.pgofs, b.vy, b.vu, b.vt, b.beta, b.vc, b.vperm, b.vm, b.vgofs, b.vcoff, b.voff, b.vnext };
      for (void *q : pb) pht_dev_free(q, e->stream); }
    { void *eb[] = { e->d_E, e->d_alpha, e->d_Eres, e->d_K };
      for (void *q : eb) pht_dev_free(q, e->stream); }
    void *big[] = { e->d_cy, e->d_cu, e->d_cc, e->d_cperm, e->d_cgofs, e->d_ry, e->d_ru, e->d_rc, e->d_rbase, e->d_ritems, e->d_rnext, e->d_gtmax, e->d_gofs, e->d_gys, e->d_gus, e->d_gcs, e->d_gperm, e->d_keys, e->d_cnext, e->d_entry, e->d_ea, e->d_eobs, e->d_eM, e->d_eoff, e->d_enext, e->d_etab, e->d_escan, e->d_unif, e->d_u, e->d_us, e->d_item_u, e->d_recs, e->d_ys, e->d_cs, e->d_perm, e->d_y, e->d_cens, e->d_items /* arena: found, pend0, pend1, done live inside */, e->d_idx_exact, e->d_idx_cens,
                    e->d_glist, e->d_model, e->d_stats, e->d_state, e->d_T, e->d_C, e->d_nu, e->d_zeta, e->d_var_ptr, e->d_cell_i, e->d_cell_j, e->d_pires, e->d_res };
    for (void *b : big) pht_dev_free(b, e->stream);
    if (e->stream) cudaStreamSynchronize(e->stream);
    stage("pool frees");
    void *bufs[] = { e->d_xw /* mapped by the peers: a plain allocation */, e->d_beta, e->d_inject, e->d_flush };
    for (void *b : bufs) if (b) cudaFree(b);
    stage("plain frees");
    if (e->stream) cudaStreamDestroy(e->stream);
    stage("stream");
    delete e;
}

extern "C" int pht_engine_create(pht_engine **out, const pht_config *cfg, const double *y_local,
                                 const int *cens_local, long l_local) {
    if (!out || !cfg) return fail("null argument");
    *out = nullptr;
    const int n = cfg->n, m = cfg->m, n1 = n + 1;
    if (n < 1 || n > PHT_MAX_PHASES) return fail("n = %d outside 1..%d", n, PHT_MAX_PHASES);
    if (m < 1 || m > n * n1) return fail("m = %d outside 1..n(n+1)", m);
    if (method_of(*cfg) == 0) return fail("unknown sampling method (code = %d)", cfg->method);
    if (cfg->mhit < 0 || cfg->mhit > 65535) return fail("mhit = %d outside 0..65535", cfg->mhit);
    if (cfg->world < 1 || cfg->rank < 0 || cfg->rank >= cfg->world) return fail("bad shard (rank %d of %d)", cfg->rank, cfg->world);
    if (cfg->zbits < 0 || cfg->zbits > 52) return fail("zbits = %d outside 0..52", cfg->zbits);
    if (l_local < 0 || l_local > 0x7fffffffL) return fail("l_local out of range");
    if ((double)l_local * cfg->world > 4.0e9) return fail("global observation index exceeds 32 bits");
    for (int i = 0; i < n1 * n1; i++) if (cfg->T[i] < 0 || cfg->T[i] > m) return fail("T[%d] = %d outside 0..m", i, cfg->T[i]);
    /* the absorbing state has no exits: a parameter in row n would make the update read beyond N and z */
    for (int j = 0; j < n1; j++) if (cfg->T[n + j * n1] != 0) return fail("T[%d, %d] = %d: row n+1 (the absorbing state) must be all zero", n, j, cfg->T[n + j * n1]);
    if (cfg->world > PHT_MAX_WORLD) return fail("world = %d exceeds %d", cfg->world, PHT_MAX_WORLD);

    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return fail("no CUDA device available (this library has no CPU path)"); }
    if (cfg->device < 0 || cfg->device >= ndev) return fail("device %d not present (%d devices)", cfg->device, ndev);
    CU(cudaSetDevice(cfg->device));
    /* (cudaGetDeviceProperties takes 2-13 ms per call here; two attributes take microseconds) */
    int cc_major = 0, cc_minor = 0;
    CU(cudaDeviceGetAttribute(&cc_major, cudaDevAttrComputeCapabilityMajor, cfg->device));
    CU(cudaDeviceGetAttribute(&cc_minor, cudaDevAttrComputeCapabilityMinor, cfg->device));
    if (cc_major < 10) return fail("device %d is sm_%d%d; this library is built for sm_100a only", cfg->device, cc_major, cc_minor);

    /* PHT_B200_TIMING=1: stage times of the set-up on stderr (tools/e2e_breakdown.py) */
    const bool timing = getenv("PHT_B200_TIMING") != nullptr;
    struct timespec ts0; clock_gettime(CLOCK_MONOTONIC, &ts0);
    auto stage = [&](const char *what) {
        if (!timing) return;
        struct timespec t; clock_gettime(CLOCK_MONOTONIC, &t);
        fprintf(stderr, "[pht_engine_create] %-28s %8.3f ms\n", what, (t.tv_sec - ts0.tv_sec) * 1e3 + (t.tv_nsec - ts0.tv_nsec) * 1e-6);
        ts0 = t;
    };
    pht_engine *e = new pht_engine();
    e->cfg = *cfg;
    e->T.assign(cfg->T, cfg->T + n1 * n1); e->C.assign(cfg->C, cfg->C + n1 * n1);
    e->nu.assign(cfg->nu, cfg->nu + m); e->zeta.assign(cfg->zeta, cfg->zeta + m);
    e->cfg.T = e->T.data(); e->cfg.C = e->C.data(); e->cfg.nu = e->nu.data(); e->cfg.zeta = e->zeta.data();
    const bool auto_cap = e->cfg.mhrs_cap <= 0;
    if (auto_cap) e->cfg.mhrs_cap = 256;
    e->l_local = l_local;
    e->base_seed = cfg->seed;
    e->L = ModelLayout::make(n, m);
#define CUE(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { fail("%s failed: %s", #call, cudaGetErrorString(e_)); pht_engine_destroy(e); return -1; } } while (0)
    CUE(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    CUE(cudaEventCreate(&e->ev0)); CUE(cudaEventCreate(&e->ev1));

    /* observations: y as is, censoring flags repacked int32 -> uint8 (9 B per path in HBM) */
    const size_t ln = (size_t)(l_local > 0 ? l_local : 1);
    pool_keep(cfg->device);
    CUE(pht_dev_alloc((void **)&e->d_y, ln * sizeof(double), e->stream));
    CUE(pht_dev_alloc((void **)&e->d_cens, ln, e->stream));
    stage("stream, events, 2 mallocs");
    if (l_local > 0) {
        /* the int32 flags are repacked to bytes by two helper threads while this one feeds y to the copy engine (a copy
         * from pageable memory occupies the calling thread): 7 ms each at 1e7 observations, now side by side.
         * (a pageable staging vector: pinning 10 MB per call cost more than the copy it would speed up) */
        std::vector<uint8_t> hc((size_t)l_local);
        uint8_t *hcp = hc.data();
        const long half = l_local / 2;
        std::thread r0([=] { for (long i = 0; i < half; i++) hcp[i] = cens_local[i] != 0; });
        std::thread r1([=] { for (long i = half; i < l_local; i++) hcp[i] = cens_local[i] != 0; });
        const cudaError_t ey = cudaMemcpyAsync(e->d_y, y_local, (size_t)l_local * sizeof(double), cudaMemcpyHostToDevice, e->stream);
        r0.join(); r1.join();
        CUE(ey);
        stage("y upload | flag repack");
        CUE(cudaMemcpyAsync(e->d_cens, hc.data(), (size_t)l_local, cudaMemcpyHostToDevice, e->stream));
        CUE(cudaStreamSynchronize(e->stream));
        stage("flag upload + sync");
        if (method_of(e->cfg) == PHT_METHOD_ECS) e->h_cens.swap(hc);
    }

    /* parameter -> cells CSR in the reference's insertion order (row-major walk of T, src/PHT_MCMC_Aslett.c:210-228) */
    std::vector<int> var_ptr(m + 1, 0), cell_i, cell_j;
    for (int i = 0; i < n1; i++) for (int j = 0; j < n1; j++) { int v = e->T[i + j * n1]; if (v) var_ptr[v]++; }
    for (int v = 0; v < m; v++) var_ptr[v + 1] += var_ptr[v];
    cell_i.resize(var_ptr[m] > 0 ? var_ptr[m] : 1); cell_j.resize(cell_i.size());
    { std::vector<int> fill(var_ptr.begin(), var_ptr.end() - 1);
      for (int i = 0; i < n1; i++) for (int j = 0; j < n1; j++) { int v = e->T[i + j * n1]; if (v) { int c = fill[v - 1]++; cell_i[c] = i; cell_j[c] = j; } } }

    /* the small buffers too come from the pool (a plain cudaFree per buffer cost up to 66 ms per call inside a process that
     * holds other allocations: PHT_B200_TIMING); the host vectors they are filled from live until the synchronize below */
#define SMALL(ptr, bytes) CUE(pht_dev_alloc((void **)&(ptr), (bytes), e->stream))
    SMALL(e->d_model, sizeof(double) * e->L.total); CUE(cudaMemsetAsync(e->d_model, 0, sizeof(double) * e->L.total, e->stream));
    SMALL(e->d_stats, sizeof(long long) * stats_len(n)); CUE(cudaMemsetAsync(e->d_stats, 0, sizeof(long long) * stats_len(n), e->stream));
    SMALL(e->d_state, sizeof(DevState)); CUE(cudaMemsetAsync(e->d_state, 0, sizeof(DevState), e->stream));
    SMALL(e->d_T, sizeof(int) * n1 * n1); CUE(cudaMemcpyAsync(e->d_T, e->T.data(), sizeof(int) * n1 * n1, cudaMemcpyHostToDevice, e->stream));
    SMALL(e->d_C, sizeof(double) * n1 * n1); CUE(cudaMemcpyAsync(e->d_C, e->C.data(), sizeof(double) * n1 * n1, cudaMemcpyHostToDevice, e->stream));
    SMALL(e->d_nu, sizeof(double) * m); CUE(cudaMemcpyAsync(e->d_nu, e->nu.data(), sizeof(double) * m, cudaMemcpyHostToDevice, e->stream));
    SMALL(e->d_zeta, sizeof(double) * m); CUE(cudaMemcpyAsync(e->d_zeta, e->zeta.data(), sizeof(double) * m, cudaMemcpyHostToDevice, e->stream));
    SMALL(e->d_var_ptr, sizeof(int) * (m + 1)); CUE(cudaMemcpyAsync(e->d_var_ptr, var_ptr.data(), sizeof(int) * (m + 1), cudaMemcpyHostToDevice, e->stream));
    SMALL(e->d_cell_i, sizeof(int) * cell_i.size()); CUE(cudaMemcpyAsync(e->d_cell_i, cell_i.data(), sizeof(int) * cell_i.size(), cudaMemcpyHostToDevice, e->stream));
    SMALL(e->d_cell_j, sizeof(int) * cell_j.size()); CUE(cudaMemcpyAsync(e->d_cell_j, cell_j.data(), sizeof(int) * cell_j.size(), cudaMemcpyHostToDevice, e->stream));
#undef SMALL
    CUE(cudaStreamSynchronize(e->stream));
    stage("model buffers");
    if (cfg->world > 1) {
        /* this rank's exchange window: all-reduce slots (every method) and the global MHRS tail (flags 0, found words NONE) */
        CUE(cudaMalloc(&e->d_xw, sizeof(XchgWindow)));
        CUE(cudaMemsetAsync(e->d_xw, 0, sizeof(XchgWindow), e->stream));
        CUE(cudaMemsetAsync(e->d_xw->gfound, 0xFF, sizeof(e->d_xw->gfound), e->stream));
        CUE(cudaStreamSynchronize(e->stream));
    }
    if (method_of(e->cfg) == PHT_METHOD_UNIF) {
        /* the table (capacity PHT_UNIF_CAP powers; log k! filled once here), the y-descending layout so that the lanes of
         * a warp run similar Poisson truncations (parity hooks keep the upload order), and the longest span y */
        CUE(pht_dev_alloc((void **)&e->d_unif, sizeof(double) * pht_unif_table_doubles(n, PHT_UNIF_CAP), e->stream));
        CUE(pht_unif_init(e->d_unif, n, PHT_UNIF_CAP, 1, e->stream));
        /* chain 0's key and observation counter (pht_engine_set_chains adds more) */
        const uint32_t key[2] = { (uint32_t)cfg->seed, (uint32_t)(cfg->seed >> 32) };
        CUE(pht_dev_alloc((void **)&e->d_keys, sizeof(key), e->stream));
        CUE(cudaMemcpyAsync(e->d_keys, key, sizeof(key), cudaMemcpyHostToDevice, e->stream));
        CUE(pht_dev_alloc((void **)&e->d_cnext, sizeof(unsigned long long), e->stream));
        CUE(cudaMemsetAsync(e->d_cnext, 0, sizeof(unsigned long long), e->stream));
        for (long i = 0; i < l_local; i++) if (y_local[i] > e->unif_tmax) e->unif_tmax = y_local[i];
        if (l_local > 1 && !getenv("PHT_B200_NO_SORT")) {
            CUE(pht_dev_alloc((void **)&e->d_ys, ln * sizeof(double), e->stream)); CUE(pht_dev_alloc((void **)&e->d_cs, ln, e->stream));
            CUE(pht_dev_alloc((void **)&e->d_perm, ln * sizeof(uint32_t), e->stream));
            CUE(pht_sort_by_y_desc(e->d_y, e->d_cens, l_local, e->d_ys, e->d_cs, e->d_perm, e->stream));
        }
        CUE(cudaStreamSynchronize(e->stream));
        e->grid_blocks = pht_unif_grid_blocks(cfg->device, n, false);
        if (e->grid_blocks <= 0) { fail("the uniformisation kernel does not fit on the device: %s", cudaGetErrorString(cudaGetLastError())); pht_engine_destroy(e); return -1; }
    }
    if (method_of(e->cfg) == PHT_METHOD_MHRS) {
        /* Tail work lists: one arena with room for a quarter of the shard (at least 2^20 observations, at most all of
         * them).  In practice ~1 % of the observations plus one per resident lane are handed over; if the lists ever
         * fill up, lanes simply keep their observation (k_mhrs.cu), so the size is a speed matter, not a limit. */
        size_t slots = ln / 4 > ((size_t)1 << 20) ? ln / 4 : ((size_t)1 << 20);
        if (slots > ln) slots = ln;
        if (const char *ev = getenv("PHT_B200_TAIL_SLOTS")) { const long v = atol(ev); if (v >= 1 && (size_t)v < slots) slots = (size_t)v; }
        e->item_cap = (uint32_t)slots;
        unsigned char *arena = nullptr;
        CUE(pht_dev_alloc((void **)&arena, slots * (sizeof(TailItem) + sizeof(unsigned long long) + 3 * sizeof(uint32_t)), e->stream));
        e->d_items = reinterpret_cast<TailItem *>(arena); arena += slots * sizeof(TailItem);
        e->d_found = reinterpret_cast<unsigned long long *>(arena); arena += slots * sizeof(unsigned long long);
        e->d_pend0 = reinterpret_cast<uint32_t *>(arena); arena += slots * sizeof(uint32_t);
        e->d_pend1 = reinterpret_cast<uint32_t *>(arena); arena += slots * sizeof(uint32_t);
        e->d_done = reinterpret_cast<uint32_t *>(arena);
        stage("tail arena");
        /* the production layout: observations by decreasing y (k_sort.cu); parity hooks keep using the upload order */
        if (l_local > 1 && !getenv("PHT_B200_NO_SORT")) {
            CUE(pht_dev_alloc((void **)&e->d_ys, ln * sizeof(double), e->stream)); CUE(pht_dev_alloc((void **)&e->d_cs, ln, e->stream));
            CUE(pht_dev_alloc((void **)&e->d_perm, ln * sizeof(uint32_t), e->stream));
            stage("sorted-layout mallocs");
            CUE(pht_sort_by_y_desc(e->d_y, e->d_cens, l_local, e->d_ys, e->d_cs, e->d_perm, e->stream));
            stage("sort by y");
        }
        /* global tail: the canonical list */
        if (const char *ev = getenv("PHT_B200_KSWITCH")) { const long v = atol(ev); if (v >= 512 && v <= (1l << 24)) e->k_switch = (uint32_t)v; }
        if (cfg->world > 1) CUE(pht_dev_alloc((void **)&e->d_glist, sizeof(uint32_t) * 2 * PHT_MAX_WORLD * PHT_GCAP, e->stream));      /* double buffered */
        CUE(pht_dev_alloc((void **)&e->d_recs, ln * sizeof(uint4), e->stream));
        stage("record list");
        if (pht_mhrs_grid_blocks(cfg->device, n, false, &e->grid_blocks, &e->tail_blocks, &e->replay_blocks) != 0) e->grid_blocks = 0;
        if (e->grid_blocks <= 0) { fail("MHRS kernel does not fit on the device: %s", cudaGetErrorString(cudaGetLastError())); pht_engine_destroy(e); return -1; }
        if (auto_cap) {
            /* Attempts a lane spends on one observation before it hands it to the tail.  A lane is a slow worker (one
             * attempt is ~9 dependent jump-steps of ~0.9 us each with the SM full), so an observation that runs to the cap
             * occupies its lane for cap x 8 us, and the lane phase cannot end sooner: 2 ms at 256 -- nothing against the
             * 4.3 ms the lane phase of 10^7 observations takes anyway, twice the whole lane phase of a 1.25 x 10^6 shard
             * (one GPU's share of the 8-GPU run).  But the tail is the slower searcher per attempt (24 warps per SM, whole
             * warps per observation), so handing over early only pays at small shards.  Measured (tools/gpu_r2_capsweep.sh,
             * ms per sweep at cap 256 / 64 / 32): 1.25e6 observations 3.57 / 3.07 / 3.20; 2.5e6: 5.05 / 5.07 / 5.43; 5e6:
             * 7.45 / 8.16 / 9.02; 1e7: 13.9 / 15.5 / 17.3.  Rule: cap = 8 x observations per resident lane, as a power of
             * two between 32 and 256.  Results do not depend on it. */
            const double per_lane = (double)l_local / ((double)e->grid_blocks * 256.0);
            int cap = 32; while (cap < 1024 && (double)(cap * 2) <= 8.0 * per_lane) cap *= 2;
            e->cfg.mhrs_cap = cap;
        }
    }
    if (method_of(e->cfg) == PHT_METHOD_ECS) {
        std::vector<uint32_t> ie, ic;
        for (long i = 0; i < l_local; i++) (e->h_cens[i] ? ic : ie).push_back((uint32_t)i);
        e->n_exact = ie.size(); e->n_cens = ic.size();
        CUE(pht_dev_alloc((void **)&e->d_idx_exact, sizeof(uint32_t) * (ie.size() + 1), e->stream)); CUE(pht_dev_alloc((void **)&e->d_idx_cens, sizeof(uint32_t) * (ic.size() + 1), e->stream));
        if (!ie.empty()) CUE(cudaMemcpyAsync(e->d_idx_exact, ie.data(), sizeof(uint32_t) * ie.size(), cudaMemcpyHostToDevice, e->stream));
        if (!ic.empty()) CUE(cudaMemcpyAsync(e->d_idx_cens, ic.data(), sizeof(uint32_t) * ic.size(), cudaMemcpyHostToDevice, e->stream));
        CUE(cudaStreamSynchronize(e->stream));
        e->grid_blocks = pht_ecs_grid_blocks(cfg->device, n);
        if (e->grid_blocks <= 0) { fail("ECS kernels do not fit on the device: %s", cudaGetErrorString(cudaGetLastError())); pht_engine_destroy(e); return -1; }
    }
    if (method_of(e->cfg) == PHT_METHOD_MHS_HOBOLTH || method_of(e->cfg) == PHT_METHOD_MHS_ASLETT) {
        e->grid_blocks = method_of(e->cfg) == PHT_METHOD_MHS_HOBOLTH ? pht_dcs_grid_blocks(cfg->device, n, true) : pht_mhs_aslett_grid_blocks(cfg->device, n);
        if (e->grid_blocks <= 0) { fail("the MH sampler variant does not fit on the device: %s", cudaGetErrorString(cudaGetLastError())); pht_engine_destroy(e); return -1; }
    }
    if (method_of(e->cfg) == PHT_METHOD_DCS) {
        e->grid_blocks = pht_dcs_grid_blocks(cfg->device, n);
        if (e->grid_blocks <= 0) { fail("DCS kernel does not fit on the device: %s", cudaGetErrorString(cudaGetLastError())); pht_engine_destroy(e); return -1; }
    }
    { const double one = 1.0;         /* start distribution e1, as the reference fixes it (src/PHT_MCMC_Aslett.c:190-193) */
      CUE(cudaMemcpyAsync(e->d_model + e->L.pi, &one, sizeof(double), cudaMemcpyHostToDevice, e->stream)); CUE(cudaStreamSynchronize(e->stream)); }
    /* sweep index 1, start-value assembly (src/PHT_MCMC_Aslett.c:268) */
    DevState st; memset(&st, 0, sizeof(st)); st.iter = 1; st.first_assembly = 1;
    CUE(cudaMemcpyAsync(e->d_state, &st, sizeof(st), cudaMemcpyHostToDevice, e->stream));
    CUE(cudaStreamSynchronize(e->stream));
#undef CUE
    stage("occupancy queries, state");
    *out = e;
    return 0;
}

extern "C" int pht_comm_unique_id(void *id128) {
    if (nccl_load()) return -1;
    ncclUniqueId id; int rc = g_nccl.GetUniqueId(&id);
    if (rc != 0) return fail("ncclGetUniqueId failed (%d)", rc);
    memcpy(id128, &id, sizeof(id));
    return 0;
}
extern "C" int pht_engine_comm_init(pht_engine *e, const void *id128) {
    if (!e) return fail("null engine");
    if (e->cfg.world == 1) return 0;
    if (nccl_load()) return -1;
    CU(cudaSetDevice(e->cfg.device));
    ncclUniqueId id; memcpy(&id, id128, sizeof(id));
    int rc = g_nccl.CommInitRank(&e->comm, e->cfg.world, id, e->cfg.rank);
    if (rc != 0) return fail("ncclCommInitRank failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?");
    /* one collective outside any graph capture: NCCL connects its transports lazily on first use */
    CU(cudaMemsetAsync(e->d_stats, 0, sizeof(long long) * stats_len(e->cfg.n), e->stream));
    rc = g_nccl.AllReduce(e->d_stats, e->d_stats, (size_t)stats_len(e->cfg.n), NCCL_INT64, NCCL_SUM, e->comm, e->stream);
    if (rc != 0) return fail("ncclAllReduce (warm-up) failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?");
    CU(cudaStreamSynchronize(e->stream));
    return 0;
}

/* ---------------------------------------------------------------- peer exchange windows (MHRS global tail) */
struct PeerHandle { unsigned long long pid; unsigned long long ptr; int device; int valid; cudaIpcMemHandle_t ipc; unsigned long long cfg_hash; };
/* what every rank of a run must agree on (the chain is one chain): key, shape, sampler, fixed-point scale, world size,
 * whether interval bounds are set (a global tail round searches every rank's items with one kernel instance) and whether
 * entry ages are set */
static unsigned long long cfg_hash(const pht_engine *e) {
    const pht_config &c = e->cfg;
    unsigned long long h = 0xcbf29ce484222325ULL;
    const unsigned long long v[] = { c.seed, (unsigned long long)c.n, (unsigned long long)c.m, (unsigned long long)c.method, (unsigned long long)c.mhit,
                                     (unsigned long long)c.zbits, (unsigned long long)c.world, e->d_u ? 1ull : 0ull,
                                     e->entry_set ? 1ull : 0ull };
    for (unsigned long long x : v) for (int b = 0; b < 8; b++) { h ^= (x >> (8 * b)) & 0xffull; h *= 0x100000001b3ULL; }
    return h;
}
static_assert(sizeof(PeerHandle) <= PHT_PEER_HANDLE_BYTES, "peer handle does not fit its ABI slot");

extern "C" int pht_engine_peer_handle(pht_engine *e, void *handle) {
    if (!e || !handle) return fail("null argument");
    memset(handle, 0, PHT_PEER_HANDLE_BYTES);
    PeerHandle h; memset(&h, 0, sizeof(h));
    if (e->d_xw) {
        CU(cudaSetDevice(e->cfg.device));
        h.pid = (unsigned long long)getpid(); h.ptr = (unsigned long long)(uintptr_t)e->d_xw; h.device = e->cfg.device; h.valid = 1;
        h.cfg_hash = cfg_hash(e);
        CU(cudaIpcGetMemHandle(&h.ipc, e->d_xw));
    }
    memcpy(handle, &h, sizeof(h));
    return 0;
}

extern "C" int pht_engine_peer_attach(pht_engine *e, const void *handles) {
    if (!e || !handles) return fail("null argument");
    if (e->cfg.world == 1 || !e->d_xw) return 0;           /* nothing to share (single rank) */
    CU(cudaSetDevice(e->cfg.device));
    for (int r = 0; r < e->cfg.world; r++) {
        PeerHandle h; memcpy(&h, (const char *)handles + (size_t)r * PHT_PEER_HANDLE_BYTES, sizeof(h));
        if (!h.valid) return fail("rank %d offers no exchange window", r);
        if (h.cfg_hash != cfg_hash(e)) return fail("rank %d runs a different configuration (seed, n, m, method, mhit, zbits, world or the presence of interval bounds or of entry ages differ from rank %d's): the ranks of a run share one chain", r, e->cfg.rank);
        if (r == e->cfg.rank) { e->xpeer[r] = e->d_xw; continue; }
        if (h.pid == (unsigned long long)getpid()) {
            /* same process (one host thread per GPU): the peer's pointer is valid here once peer access is on */
            if (h.device != e->cfg.device) {
                int can = 0; CU(cudaDeviceCanAccessPeer(&can, e->cfg.device, h.device));
                if (!can) return fail("device %d cannot access device %d", e->cfg.device, h.device);
                cudaError_t pe = cudaDeviceEnablePeerAccess(h.device, 0);
                if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) return fail("cudaDeviceEnablePeerAccess(%d): %s", h.device, cudaGetErrorString(pe));
                cudaGetLastError();
            }
            e->xpeer[r] = reinterpret_cast<XchgWindow *>((uintptr_t)h.ptr);
        } else {
            void *q = nullptr;
            CU(cudaIpcOpenMemHandle(&q, h.ipc, cudaIpcMemLazyEnablePeerAccess));
            e->ipc_opened.push_back(q);
            e->xpeer[r] = reinterpret_cast<XchgWindow *>(q);
        }
    }
    e->peers_attached = true;
    /* the statistics go through the windows too, unless the launcher asks for the NCCL all-reduce (PHT_B200_NCCL=1) */
    { const char *ev = getenv("PHT_B200_NCCL"); e->peer_reduce = !(ev && *ev && *ev != '0'); }
    if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }     /* kernel parameters change */
    return 0;
}

/* the next sweep gets index next_iter and assembles its model from start values (src/PHT_MCMC_Aslett.c:268) */
static int set_next_iter(pht_engine *e, uint32_t next_iter) {
    DevState st; CU(cudaMemcpy(&st, e->d_state, sizeof(st), cudaMemcpyDeviceToHost));
    st.iter = next_iter; st.first_assembly = 1;
    CU(cudaMemcpy(e->d_state, &st, sizeof(st), cudaMemcpyHostToDevice));
    return 0;
}

extern "C" int pht_engine_set_theta(pht_engine *e, const double *theta, uint32_t next_iter) {
    if (!e || !theta) return fail("null argument");
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    for (int c = 0; c < e->chains * e->groups; c++)           /* every chain, in every group's block */
        CU(cudaMemcpy(e->d_model + (size_t)c * e->L.total + e->L.theta, theta, sizeof(double) * e->cfg.m, cudaMemcpyHostToDevice));
    return set_next_iter(e, next_iter);
}
extern "C" int pht_engine_get_theta(pht_engine *e, double *theta) {
    if (!e || !theta) return fail("null argument");
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    CU(cudaMemcpy(theta, e->d_model + e->L.theta, sizeof(double) * e->cfg.m, cudaMemcpyDeviceToHost));
    return 0;
}

extern "C" int pht_engine_set_pi(pht_engine *e, const double *pi, const double *beta) {
    if (!e) return fail("null engine");
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    const int n = e->cfg.n;
    if (pi) {
        double sum = 0.0;
        for (int i = 0; i < n; i++) { if (!(pi[i] >= 0.0)) return fail("pi[%d] = %g is not a probability", i, pi[i]); sum += pi[i]; }
        if (!(sum > 0.999999 && sum < 1.000001)) return fail("pi sums to %g, not 1", sum);
        if (e->visits_set && engine_visits_reachable(e, e->h_voff.data(), e->h_vt.data(), visit_masks(e->h_vm.data(), e->h_vm.size(), e->h_colmask).data(),
                                                     pi, 0, nullptr, nullptr, nullptr))
            return -1;                             /* (pht_engine_set_visits: a visit sequence this pi cannot start) */
        for (int c = 0; c < e->chains * e->groups; c++)       /* every chain, in every group's block */
            CU(cudaMemcpy(e->d_model + (size_t)c * e->L.total + e->L.pi, pi, sizeof(double) * n, cudaMemcpyHostToDevice));
    }
    if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }     /* kernel parameters change */
    if (beta) {
        /* The update needs start states drawn from their conditional law given y.  MHRS does that by construction (a
         * rejection sampler from pi).  The reference's ECS and DCS samplers draw the start state from pi itself
         * (src/Simulate_AbsCTMC_eq_Aslett_ECS.c:231-238, src/Simulate_AbsCTMC_gt_Hobolth_DCS.c:88-95) -- exact only for
         * the degenerate pi the reference always uses -- so B carries no information about pi there. */
        if (method_of(e->cfg) != PHT_METHOD_MHRS && method_of(e->cfg) != PHT_METHOD_UNIF)
            return fail("the start-distribution update needs method MHRS or 64 (ECS and DCS draw the start state from pi, not from its conditional law given y)");
        for (int i = 0; i < n; i++) if (!(beta[i] > 0.0)) return fail("beta[%d] = %g: Dirichlet parameters must be positive", i, beta[i]);
        if (!e->d_beta) CU(cudaMalloc(&e->d_beta, sizeof(double) * n));
        CU(cudaMemcpy(e->d_beta, beta, sizeof(double) * n, cudaMemcpyHostToDevice));
    } else if (e->d_beta) { CU(cudaFree(e->d_beta)); e->d_beta = nullptr; }
    return 0;
}
extern "C" int pht_engine_get_pi(pht_engine *e, double *pi) {
    if (!e || !pi) return fail("null argument");
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    CU(cudaMemcpy(pi, e->d_model + e->L.pi, sizeof(double) * e->cfg.n, cudaMemcpyDeviceToHost));
    return 0;
}
extern "C" int pht_engine_pi_rows(pht_engine *e, int rows, double *out) {
    if (!e || !out || rows < 0) return fail("bad argument");
    if (!e->d_beta || !e->d_pires) return fail("pi is not being inferred (pht_engine_set_pi with a prior first)");
    if (rows > e->res_rows) return fail("%d rows asked, the last run produced at most %d", rows, e->res_rows);
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    if (rows) CU(cudaMemcpy(out, e->d_pires, sizeof(double) * (size_t)rows * e->cfg.n, cudaMemcpyDeviceToHost));
    return 0;
}

/* ---------------------------------------------------------------- several chains (method 64) */
extern "C" int pht_engine_set_chains(pht_engine *e, int chains, const uint64_t *keys) {
    if (!e) return fail("null engine");
    if (method_of(e->cfg) != PHT_METHOD_UNIF)
        return fail("several chains per engine need method 64 (the uniformisation sampler); MHRS, ECS, DCS and the MH variants run one chain per engine");
    if (e->cfg.world > 1)
        return fail("several chains per engine need world = 1: the statistics all-reduce of a multi-rank run carries one chain's block");
    if (chains < 1 || chains > PHT_MAX_CHAINS) return fail("chains = %d outside 1..%d", chains, PHT_MAX_CHAINS);
    if ((long)chains * e->groups > PHT_MAX_CHAINS)
        return fail("chains x groups = %d x %d exceeds %d (pht_engine_set_groups)", chains, e->groups, PHT_MAX_CHAINS);
    if (chains > 1 && e->entry_set)
        return fail("%d chains asked while entry ages (delayed entry) are set: the ghost paths are drawn for one chain; clear them with pht_engine_set_entry(e, NULL) first", chains);
    std::vector<uint64_t> k((size_t)chains);
    for (int c = 0; c < chains; c++) k[(size_t)c] = keys ? keys[c] : e->base_seed + (uint64_t)c;
    { std::vector<uint64_t> sorted(k); std::sort(sorted.begin(), sorted.end());
      for (size_t i = 1; i < sorted.size(); i++) if (sorted[i] == sorted[i - 1])
          return fail("duplicate key 0x%llx: two chains with one key would be one chain drawn twice", (unsigned long long)sorted[i]); }
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    const int n = e->cfg.n;
    const int G = e->groups, units = chains * G;
    if (units > 1 && !e->chain_blocks) {
        e->chain_blocks = pht_unif_grid_blocks(e->cfg.device, n, true);
        if (e->chain_blocks <= 0) { e->chain_blocks = 0; return fail("the several-chain path kernel does not fit on the device: %s", cudaGetErrorString(cudaGetLastError())); }
    }
    const size_t total = (size_t)e->L.total, slen = (size_t)stats_len(n), tab = pht_unif_table_doubles(n, PHT_UNIF_CAP);
    /* the new buffers first: a failed allocation leaves the engine as it was */
    double *model = nullptr, *unif = nullptr; long long *stats = nullptr; uint32_t *dkeys = nullptr; unsigned long long *cnext = nullptr;
    const size_t bytes[] = { sizeof(double) * units * total, sizeof(long long) * units * slen, sizeof(double) * units * tab,
                             sizeof(uint32_t) * 2 * chains, sizeof(unsigned long long) * units };
    void **ptrs[] = { (void **)&model, (void **)&stats, (void **)&unif, (void **)&dkeys, (void **)&cnext };
    for (int b = 0; b < 5; b++) {
        const cudaError_t ce = pht_dev_alloc(ptrs[b], bytes[b], e->stream);
        if (ce != cudaSuccess) {
            cudaGetLastError();
            for (int f = 0; f < b; f++) pht_dev_free(*ptrs[f], e->stream);
            cudaStreamSynchronize(e->stream); cudaGetLastError();
            return fail("cannot allocate device memory for %d chains (%.1f MB, of which the uniformisation tables take %.1f MB per chain and group): %s",
                        chains, (bytes[0] + bytes[1] + bytes[2] + bytes[3] + bytes[4]) / 1e6, sizeof(double) * tab / 1e6, cudaGetErrorString(ce));
        }
    }
    /* stage visits: E and K per chain, every chain starting from chain 0's E */
    double *dE = nullptr; unsigned long long *dK = nullptr;
    const size_t nS = (size_t)n * e->stages;
    if (e->stages) {
        cudaError_t ce = pht_dev_alloc((void **)&dE, sizeof(double) * chains * nS, e->stream);
        if (ce == cudaSuccess) ce = pht_dev_alloc((void **)&dK, sizeof(unsigned long long) * chains * nS, e->stream);
        if (ce != cudaSuccess) {
            cudaGetLastError();
            for (int f = 0; f < 5; f++) pht_dev_free(*ptrs[f], e->stream);
            pht_dev_free(dE, e->stream);
            cudaStreamSynchronize(e->stream); cudaGetLastError();
            return fail("cannot allocate device memory for the emission matrices of %d chains: %s", chains, cudaGetErrorString(ce));
        }
        for (int c = 0; c < chains; c++) CU(cudaMemcpyAsync(dE + c * nS, e->d_E, sizeof(double) * nS, cudaMemcpyDeviceToDevice, e->stream));
        CU(cudaMemsetAsync(dK, 0, sizeof(unsigned long long) * chains * nS, e->stream));
    }
    /* every chain starts from chain 0's current theta and pi (the rest of a model block is rebuilt every sweep) */
    for (int c = 0; c < units; c++)
        CU(cudaMemcpyAsync(model + (size_t)c * total, e->d_model, sizeof(double) * total, cudaMemcpyDeviceToDevice, e->stream));
    CU(cudaMemsetAsync(stats, 0, bytes[1], e->stream));
    CU(pht_unif_init(unif, n, PHT_UNIF_CAP, units, e->stream));       /* log k! in every unit's table */
    std::vector<uint32_t> hk(2 * (size_t)chains);
    for (int c = 0; c < chains; c++) { hk[2 * (size_t)c] = (uint32_t)k[(size_t)c]; hk[2 * (size_t)c + 1] = (uint32_t)(k[(size_t)c] >> 32); }
    CU(cudaMemcpyAsync(dkeys, hk.data(), bytes[3], cudaMemcpyHostToDevice, e->stream));
    CU(cudaMemsetAsync(cnext, 0, bytes[4], e->stream));
    void *old[] = { e->d_model, e->d_stats, e->d_unif, e->d_keys, e->d_cnext, e->d_res, e->d_pires, e->d_E, e->d_K, e->d_Eres };
    for (void *b : old) CU(pht_dev_free(b, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    e->d_model = model; e->d_stats = stats; e->d_unif = unif; e->d_keys = dkeys; e->d_cnext = cnext;
    e->d_res = nullptr; e->d_pires = nullptr; e->res_rows = 0;
    e->d_E = dE; e->d_K = dK; e->d_Eres = nullptr; e->eres_rows = 0;
    e->chains = chains;
    e->cfg.seed = k[0];                            /* chain 0's key is the engine's key (the ghost kernels read it) */
    if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }     /* kernel parameters change */
    return 0;
}

extern "C" int pht_engine_set_chain_theta(pht_engine *e, const double *theta, uint32_t next_iter) {
    if (!e || !theta) return fail("null argument");
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    for (int c = 0; c < e->chains * e->groups; c++)            /* chain c / groups, in every group's block */
        CU(cudaMemcpy(e->d_model + (size_t)c * e->L.total + e->L.theta, theta + (size_t)(c / e->groups) * e->cfg.m, sizeof(double) * e->cfg.m, cudaMemcpyHostToDevice));
    return set_next_iter(e, next_iter);
}

extern "C" int pht_engine_get_chain_theta(pht_engine *e, double *theta) {
    if (!e || !theta) return fail("null argument");
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    for (int c = 0; c < e->chains; c++)
        CU(cudaMemcpy(theta + (size_t)c * e->cfg.m, e->d_model + (size_t)c * e->groups * e->L.total + e->L.theta, sizeof(double) * e->cfg.m, cudaMemcpyDeviceToHost));
    return 0;
}

extern "C" int pht_engine_chain_rows(pht_engine *e, int rows, double *theta_out, double *pi_out) {
    if (!e || rows < 0) return fail("bad argument");
    if (rows > e->res_rows) return fail("%d rows asked, the last run produced at most %d", rows, e->res_rows);
    if (pi_out && (!e->d_beta || !e->d_pires)) return fail("pi is not being inferred (pht_engine_set_pi with a prior first)");
    if (rows == 0) return 0;
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    const size_t m = (size_t)e->cfg.m, n = (size_t)e->cfg.n, R = (size_t)e->res_rows;
    if (theta_out) CU(cudaMemcpy2D(theta_out, sizeof(double) * rows * m, e->d_res, sizeof(double) * R * m, sizeof(double) * rows * m, e->chains, cudaMemcpyDeviceToHost));
    if (pi_out) CU(cudaMemcpy2D(pi_out, sizeof(double) * rows * n, e->d_pires, sizeof(double) * R * n, sizeof(double) * rows * n, e->chains, cudaMemcpyDeviceToHost));
    return 0;
}

/* ---------------------------------------------------------------- groups (method 64) */
/* each group's table span: the largest y and u - y (finite u) over its observations, as pht_engine_set_upper takes it */
static int group_tmax(pht_engine *e, const std::vector<uint8_t> &gid, int G, std::vector<double> &tmax) {
    const long l = e->l_local;
    std::vector<double> y((size_t)(l > 0 ? l : 1)), u;
    if (l > 0) CU(cudaMemcpy(y.data(), e->d_y, sizeof(double) * (size_t)l, cudaMemcpyDeviceToHost));
    if (l > 0 && e->d_u) { u.resize((size_t)l); CU(cudaMemcpy(u.data(), e->d_u, sizeof(double) * (size_t)l, cudaMemcpyDeviceToHost)); }
    tmax.assign((size_t)G, 0.0);
    for (long i = 0; i < l; i++) {
        double &t = tmax[gid[(size_t)i]];
        if (y[(size_t)i] > t) t = y[(size_t)i];
        if (!u.empty() && u[(size_t)i] < INFINITY && u[(size_t)i] - y[(size_t)i] > t) t = u[(size_t)i] - y[(size_t)i];
    }
    return 0;
}

/* after the interval bounds change: the groups' table spans and u in the grouped layout */
static int group_refresh(pht_engine *e) {
    if (e->groups <= 1) return 0;
    std::vector<double> t;
    if (group_tmax(e, e->h_group, e->groups, t)) return -1;
    CU(cudaMemcpy(e->d_gtmax, t.data(), sizeof(double) * t.size(), cudaMemcpyHostToDevice));
    const long l = e->l_local;
    if (e->d_u) {
        if (!e->d_gus) CU(pht_dev_alloc((void **)&e->d_gus, sizeof(double) * (size_t)(l > 0 ? l : 1), e->stream));
        CU(pht_gather_f64(e->d_u, e->d_gperm, e->d_gus, l, e->stream));
    } else if (e->d_gus) { CU(pht_dev_free(e->d_gus, e->stream)); e->d_gus = nullptr; }
    CU(cudaStreamSynchronize(e->stream));
    return 0;
}

extern "C" int pht_engine_set_groups(pht_engine *e, int G, const int *T, const double *C, const int *group_local) {
    if (!e) return fail("null engine");
    if (method_of(e->cfg) != PHT_METHOD_UNIF)
        return fail("groups with their own structure need method 64 (the uniformisation sampler): MHRS, ECS, DCS and the MH variants run one structure per engine");
    if (e->cfg.world > 1)
        return fail("groups need world = 1: the statistics all-reduce of a multi-rank run carries one statistics block");
    const int n = e->cfg.n, m = e->cfg.m, n1 = n + 1, nn1 = n1 * n1;
    const long l = e->l_local;
    const bool clear = T == nullptr;
    std::vector<uint8_t> gid((size_t)(l > 0 ? l : 1), 0);
    if (clear) { G = 1; T = e->T.data(); C = e->C.data(); }
    else {
        if (!C || (!group_local && l > 0)) return fail("null argument");
        if (G < 1 || G > PHT_MAX_GROUPS) return fail("groups = %d outside 1..%d", G, PHT_MAX_GROUPS);
    }
    if ((long)e->chains * G > PHT_MAX_CHAINS)
        return fail("chains x groups = %d x %d exceeds %d", e->chains, G, PHT_MAX_CHAINS);
    if (G > 1 && e->entry_set)
        return fail("%d groups asked while entry ages (delayed entry) are set: the ghost paths are drawn on one model; clear them with pht_engine_set_entry(e, NULL) first", G);
    if (!clear) {
        std::vector<char> used((size_t)m, 0);
        for (int g = 0; g < G; g++) {
            const int *Tg = T + (size_t)g * nn1;
            for (int i = 0; i < nn1; i++) {
                if (Tg[i] < 0 || Tg[i] > m) return fail("group %d: T[%d] = %d outside 0..m", g, i, Tg[i]);
                if (Tg[i]) used[(size_t)Tg[i] - 1] = 1;
            }
            for (int j = 0; j < n1; j++) if (Tg[n + j * n1] != 0)
                return fail("group %d: T[%d, %d] = %d: row n+1 (the absorbing state) must be all zero", g, n, j, Tg[n + j * n1]);
        }
        for (int v = 0; v < m; v++) if (!used[(size_t)v])
            return fail("parameter %d is used by no group's structure: nothing in the data would inform it", v + 1);
        for (long k = 0; k < l; k++) {
            if (group_local[k] < 0 || group_local[k] >= G) return fail("group[%ld] = %d outside 0..%d", k, group_local[k], G - 1);
            gid[(size_t)k] = (uint8_t)group_local[k];
        }
    }
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    if (e->visits_set && engine_visits_reachable(e, e->h_voff.data(), e->h_vt.data(), visit_masks(e->h_vm.data(), e->h_vm.size(), e->h_colmask).data(), nullptr, G, T, C,
                                                 G > 1 ? gid.data() : nullptr)) return -1;
    if (G > 1 && !e->chain_blocks) {
        e->chain_blocks = pht_unif_grid_blocks(e->cfg.device, n, true);
        if (e->chain_blocks <= 0) { e->chain_blocks = 0; return fail("the several-unit path kernel does not fit on the device: %s", cudaGetErrorString(cudaGetLastError())); }
    }
    /* parameter -> cells CSR over (group, parameter): row g m + v lists group g's cells of parameter v in the reference's
     * insertion order (row-major walk of T_g, as pht_engine_create builds it for one structure) */
    std::vector<int> var_ptr((size_t)G * m + 1, 0), cell_i, cell_j;
    for (int g = 0; g < G; g++) for (int i = 0; i < n1; i++) for (int j = 0; j < n1; j++) {
        const int v = T[(size_t)g * nn1 + i + j * n1]; if (v) var_ptr[(size_t)g * m + v]++;
    }
    for (size_t r = 0; r + 1 < var_ptr.size(); r++) var_ptr[r + 1] += var_ptr[r];
    cell_i.resize(var_ptr.back() > 0 ? var_ptr.back() : 1); cell_j.resize(cell_i.size());
    { std::vector<int> fill(var_ptr.begin(), var_ptr.end() - 1);
      for (int g = 0; g < G; g++) for (int i = 0; i < n1; i++) for (int j = 0; j < n1; j++) {
          const int v = T[(size_t)g * nn1 + i + j * n1];
          if (v) { const int c = fill[(size_t)g * m + v - 1]++; cell_i[c] = i; cell_j[c] = j; }
      } }
    std::vector<double> tmax; std::vector<unsigned long long> gofs((size_t)G + 1, 0ull);
    if (G > 1) {
        if (group_tmax(e, gid, G, tmax)) return -1;
        for (long k = 0; k < l; k++) gofs[(size_t)gid[(size_t)k] + 1]++;
        for (int g = 0; g < G; g++) gofs[(size_t)g + 1] += gofs[(size_t)g];
    }
    /* the new buffers first: a failed allocation (or sort) leaves the engine as it was */
    const int units = e->chains * G, old_G = e->groups;
    const size_t total = (size_t)e->L.total, slen = (size_t)stats_len(n), tab = pht_unif_table_doubles(n, PHT_UNIF_CAP);
    const size_t ln = (size_t)(l > 0 ? l : 1);
    int *dT = nullptr, *dvp = nullptr, *dci = nullptr, *dcj = nullptr; double *dC = nullptr, *dtmax = nullptr;
    unsigned long long *dgofs = nullptr, *cnext = nullptr; double *model = nullptr, *unif = nullptr; long long *stats = nullptr;
    double *gys = nullptr, *gus = nullptr; uint8_t *gcs = nullptr, *dgid = nullptr; uint32_t *gperm = nullptr;
    struct Buf { void **p; size_t bytes; };
    std::vector<Buf> bufs = { { (void **)&dT, sizeof(int) * G * nn1 }, { (void **)&dC, sizeof(double) * G * nn1 },
                              { (void **)&dvp, sizeof(int) * var_ptr.size() }, { (void **)&dci, sizeof(int) * cell_i.size() },
                              { (void **)&dcj, sizeof(int) * cell_j.size() }, { (void **)&model, sizeof(double) * units * total },
                              { (void **)&stats, sizeof(long long) * units * slen }, { (void **)&unif, sizeof(double) * units * tab },
                              { (void **)&cnext, sizeof(unsigned long long) * units } };
    if (G > 1) {
        bufs.push_back({ (void **)&dtmax, sizeof(double) * G }); bufs.push_back({ (void **)&dgofs, sizeof(unsigned long long) * (G + 1) });
        bufs.push_back({ (void **)&gys, sizeof(double) * ln }); bufs.push_back({ (void **)&gcs, ln });
        bufs.push_back({ (void **)&gperm, sizeof(uint32_t) * ln }); bufs.push_back({ (void **)&dgid, ln });
        if (e->d_u) bufs.push_back({ (void **)&gus, sizeof(double) * ln });
    }
    auto undo = [&](size_t upto) { for (size_t f = 0; f < upto; f++) pht_dev_free(*bufs[f].p, e->stream); cudaStreamSynchronize(e->stream); cudaGetLastError(); };
    size_t bytes_all = 0;
    for (const Buf &b : bufs) bytes_all += b.bytes;
    for (size_t b = 0; b < bufs.size(); b++) {
        const cudaError_t ce = pht_dev_alloc(bufs[b].p, bufs[b].bytes, e->stream);
        if (ce != cudaSuccess) {
            cudaGetLastError(); undo(b);
            return fail("cannot allocate device memory for %d groups x %d chains (%.1f MB, of which the uniformisation tables take %.1f MB per chain and group): %s",
                        G, e->chains, bytes_all / 1e6, sizeof(double) * tab / 1e6, cudaGetErrorString(ce));
        }
    }
    cudaError_t ce = cudaSuccess;
#define STEP(call) do { if (ce == cudaSuccess) ce = (call); } while (0)
    STEP(cudaMemcpyAsync(dT, T, bufs[0].bytes, cudaMemcpyHostToDevice, e->stream));
    STEP(cudaMemcpyAsync(dC, C, bufs[1].bytes, cudaMemcpyHostToDevice, e->stream));
    STEP(cudaMemcpyAsync(dvp, var_ptr.data(), bufs[2].bytes, cudaMemcpyHostToDevice, e->stream));
    STEP(cudaMemcpyAsync(dci, cell_i.data(), bufs[3].bytes, cudaMemcpyHostToDevice, e->stream));
    STEP(cudaMemcpyAsync(dcj, cell_j.data(), bufs[4].bytes, cudaMemcpyHostToDevice, e->stream));
    /* unit (c, g) starts from chain c's current theta and pi (the rest of a model block is rebuilt every sweep) */
    for (int u = 0; u < units && ce == cudaSuccess; u++)
        STEP(cudaMemcpyAsync(model + (size_t)u * total, e->d_model + (size_t)(u / G) * old_G * total, sizeof(double) * total, cudaMemcpyDeviceToDevice, e->stream));
    STEP(cudaMemsetAsync(stats, 0, bufs[6].bytes, e->stream));
    STEP(pht_unif_init(unif, n, PHT_UNIF_CAP, units, e->stream));      /* log k! in every unit's table */
    STEP(cudaMemsetAsync(cnext, 0, bufs[8].bytes, e->stream));
    if (G > 1) {
        STEP(cudaMemcpyAsync(dtmax, tmax.data(), sizeof(double) * G, cudaMemcpyHostToDevice, e->stream));
        STEP(cudaMemcpyAsync(dgofs, gofs.data(), sizeof(unsigned long long) * (G + 1), cudaMemcpyHostToDevice, e->stream));
        if (l > 0) {
            STEP(cudaMemcpyAsync(dgid, gid.data(), (size_t)l, cudaMemcpyHostToDevice, e->stream));
            STEP(pht_sort_by_group(e->d_perm, dgid, e->d_y, e->d_cens, l, gys, gcs, gperm, e->stream));
            if (e->d_u) STEP(pht_gather_f64(e->d_u, gperm, gus, l, e->stream));
        }
    }
    STEP(cudaStreamSynchronize(e->stream));
#undef STEP
    if (ce != cudaSuccess) { undo(bufs.size()); return fail("setting up %d groups failed: %s", G, cudaGetErrorString(ce)); }
    pht_dev_free(dgid, e->stream);
    void *old[] = { e->d_T, e->d_C, e->d_var_ptr, e->d_cell_i, e->d_cell_j, e->d_model, e->d_stats, e->d_unif, e->d_cnext,
                    e->d_gtmax, e->d_gofs, e->d_gys, e->d_gcs, e->d_gperm, e->d_gus };
    for (void *b : old) CU(pht_dev_free(b, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    e->d_T = dT; e->d_C = dC; e->d_var_ptr = dvp; e->d_cell_i = dci; e->d_cell_j = dcj;
    e->d_model = model; e->d_stats = stats; e->d_unif = unif; e->d_cnext = cnext;
    e->d_gtmax = dtmax; e->d_gofs = dgofs; e->d_gys = gys; e->d_gcs = gcs; e->d_gperm = gperm; e->d_gus = gus;
    e->groups = G;
    if (G > 1) e->h_group.assign(gid.begin(), gid.begin() + l); else e->h_group.clear();
    if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }     /* kernel parameters change */
    if (e->visits_set) return visits_build(e);     /* the panel layouts follow the grouped layout */
    return e->counts_set ? counts_build(e) : 0;      /* the counted records follow the grouped layout */
}

/* ---------------------------------------------------------------- counts (method 64) */
/* Records at or above the threshold go to k_unif_records in items of at most the chunk size; the others are expanded once
 * into the ordinary layout.  Chosen from the "sweep" lines of profiles/counts_bench.jsonl (NVIDIA B200, 1000 W; C3 shape,
 * 1e7 units, ms per sweep at chunk 32 / 64 / 256 / 1024): exact times rounded to 0.01 (501 records) 8.62 / 11.80 / 15.26 /
 * 22.64 at any threshold; rounded to 1e-4 (50001 records of ~200 units) at threshold 64: 9.24 / 11.53 / 13.81 / 24.15,
 * against 9.51 at 16, 9.48 at 256 and 10.47 at 1024 with chunk 32.  One item per warp round keeps every warp busy to the
 * end of the sweep, which outweighs preparing a record once per 32 units instead of once per 1024.
 * PHT_B200_COUNTS_THRESHOLD and PHT_B200_COUNTS_CHUNK override them for that sweep; the results do not depend on either. */
#define PHT_COUNTS_THRESHOLD 64
#define PHT_COUNTS_CHUNK 32

static int counts_free(pht_engine *e) {
    void *bufs[] = { e->d_cy, e->d_cu, e->d_cc, e->d_cperm, e->d_cgofs, e->d_ry, e->d_ru, e->d_rc, e->d_rbase, e->d_ritems, e->d_rnext };
    for (void *b : bufs) CU(pht_dev_free(b, e->stream));
    e->d_cy = e->d_cu = e->d_ry = e->d_ru = nullptr; e->d_cc = e->d_rc = nullptr; e->d_cperm = e->d_rbase = nullptr;
    e->d_cgofs = e->d_rnext = nullptr; e->d_ritems = nullptr; e->n_low = 0; e->n_items = 0;
    CU(cudaStreamSynchronize(e->stream));
    return 0;
}

/* both layouts of the counted records from e->h_counts, in the engine's layout order (by group, then by decreasing y);
 * unit j of record k is expanded observation base_k + j, base the exclusive prefix sum of the counts in upload order */
static int counts_build(pht_engine *e) {
    const long l = e->l_local;
    const int G = e->groups;
    const size_t ln = (size_t)(l > 0 ? l : 1);
    std::vector<double> y(ln), u; std::vector<uint8_t> c(ln); std::vector<uint32_t> order(ln);
    const uint32_t *dperm = G > 1 ? e->d_gperm : e->d_perm;
    if (l > 0) {
        CU(cudaMemcpy(y.data(), e->d_y, sizeof(double) * (size_t)l, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(c.data(), e->d_cens, (size_t)l, cudaMemcpyDeviceToHost));
        if (e->d_u) { u.resize(ln); CU(cudaMemcpy(u.data(), e->d_u, sizeof(double) * (size_t)l, cudaMemcpyDeviceToHost)); }
        if (dperm) CU(cudaMemcpy(order.data(), dperm, sizeof(uint32_t) * (size_t)l, cudaMemcpyDeviceToHost));
        else for (long i = 0; i < l; i++) order[(size_t)i] = (uint32_t)i;
    }
    std::vector<uint32_t> base(ln);
    { uint64_t acc = 0; for (long i = 0; i < l; i++) { base[(size_t)i] = (uint32_t)acc; acc += e->h_counts[(size_t)i]; } }
    const uint32_t thr = e->counts_threshold, ch = e->counts_chunk;
    std::vector<double> ly, lu, ry, ru; std::vector<uint8_t> lc, rc; std::vector<uint32_t> lperm, rbase; std::vector<uint4> items;
    std::vector<unsigned long long> lgofs((size_t)G + 1, 0ull);
    for (long pos = 0; pos < l; pos++) {
        const uint32_t k = order[(size_t)pos], w = e->h_counts[k];
        if (w == 0u) continue;
        const uint32_t g = G > 1 ? e->h_group[k] : 0u;
        if (w >= thr) {
            const uint32_t r = (uint32_t)ry.size();
            ry.push_back(y[k]); rc.push_back(c[k]); rbase.push_back(base[k]);
            if (!u.empty()) ru.push_back(u[k]);
            for (uint32_t j0 = 0; j0 < w; j0 += ch) { items.push_back(make_uint4(r, j0, w - j0 < ch ? w - j0 : ch, g)); if (w - j0 <= ch) break; }
        } else {
            for (uint32_t j = 0; j < w; j++) {
                ly.push_back(y[k]); lc.push_back(c[k]); lperm.push_back(base[k] + j);
                if (!u.empty()) lu.push_back(u[k]);
            }
            lgofs[(size_t)g + 1] += w;
        }
    }
    for (int g = 0; g < G; g++) lgofs[(size_t)g + 1] += lgofs[(size_t)g];
    if (counts_free(e)) return -1;
    auto up = [&](void **dst, const void *src, size_t bytes) -> cudaError_t {
        cudaError_t ce = pht_dev_alloc(dst, bytes ? bytes : 1, e->stream);
        if (ce == cudaSuccess && bytes) ce = cudaMemcpyAsync(*dst, src, bytes, cudaMemcpyHostToDevice, e->stream);
        return ce;
    };
    CU(up((void **)&e->d_cy, ly.data(), sizeof(double) * ly.size()));
    CU(up((void **)&e->d_cc, lc.data(), lc.size()));
    CU(up((void **)&e->d_cperm, lperm.data(), sizeof(uint32_t) * lperm.size()));
    if (!u.empty()) CU(up((void **)&e->d_cu, lu.data(), sizeof(double) * lu.size()));
    CU(up((void **)&e->d_cgofs, lgofs.data(), sizeof(unsigned long long) * lgofs.size()));
    CU(up((void **)&e->d_ry, ry.data(), sizeof(double) * ry.size()));
    CU(up((void **)&e->d_rc, rc.data(), rc.size()));
    CU(up((void **)&e->d_rbase, rbase.data(), sizeof(uint32_t) * rbase.size()));
    if (!u.empty()) CU(up((void **)&e->d_ru, ru.data(), sizeof(double) * ru.size()));
    CU(up((void **)&e->d_ritems, items.data(), sizeof(uint4) * items.size()));
    CU(pht_dev_alloc((void **)&e->d_rnext, sizeof(unsigned long long), e->stream));
    CU(cudaStreamSynchronize(e->stream));
    e->n_low = (long)ly.size(); e->n_items = (long)items.size();
    if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }     /* kernel parameters change */
    return 0;
}

extern "C" int pht_engine_set_counts(pht_engine *e, const uint32_t *counts_local) {
    if (!e) return fail("null engine");
    if (method_of(e->cfg) != PHT_METHOD_UNIF)
        return fail("counts (tied observations as records) need method 64 (the uniformisation sampler): MHRS, ECS, DCS and the MH variants draw one path per observation");
    if (e->peers_attached) return fail("counts cannot be set after the exchange windows are attached (counts need a single-rank engine)");
    if (e->cfg.world > 1) return fail("counts need world = 1: the expanded index of a unit is a single-rank numbering");
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    if (!counts_local) {
        if (!e->counts_set) return 0;
        e->counts_set = false; e->h_counts.clear();
        if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }
        return counts_free(e);
    }
    if (e->visits_set)
        return fail("counts are not supported with visits (panel observations): the units of a record would share their visits; clear the visits with pht_engine_set_visits(e, NULL, NULL, NULL) first");
    if (e->entry_set)
        return fail("counts are not supported with entry ages (delayed entry): a record's ghost count would be a sum of w Geometric draws; clear the ages with pht_engine_set_entry(e, NULL) first");
    const long l = e->l_local;
    unsigned long long total = 0;
    for (long i = 0; i < l; i++) total += counts_local[i];
    if (total >= (1ull << 32))
        return fail("the counts sum to %llu: the expanded observation index (Philox counter word 2) is 32 bits, so the sum must stay below 2^32", total);
    /* every unit's path ends by max(y, u): the fixed-point scale must leave room for sum_k w_k max(y_k, u_k) */
    std::vector<double> y((size_t)(l > 0 ? l : 1)), u;
    if (l > 0) CU(cudaMemcpy(y.data(), e->d_y, sizeof(double) * (size_t)l, cudaMemcpyDeviceToHost));
    if (l > 0 && e->d_u) { u.resize((size_t)l); CU(cudaMemcpy(u.data(), e->d_u, sizeof(double) * (size_t)l, cudaMemcpyDeviceToHost)); }
    double sum = 0.0;
    for (long i = 0; i < l; i++) {
        const double ui = u.empty() ? INFINITY : u[(size_t)i];
        sum += (double)counts_local[i] * (ui < INFINITY ? ui : y[(size_t)i]);
    }
    if (sum > 0.0 && e->cfg.zbits > pht_choose_zbits(sum))
        return fail("zbits = %d is too fine for these counts: sum of count x max(y, u) = %g allows at most %d", e->cfg.zbits, sum, pht_choose_zbits(sum));
    if (!e->rec_blocks) {
        e->rec_blocks = pht_unif_records_grid_blocks(e->cfg.device, e->cfg.n);
        if (e->rec_blocks <= 0) { e->rec_blocks = 0; return fail("the record kernel does not fit on the device: %s", cudaGetErrorString(cudaGetLastError())); }
    }
    e->counts_threshold = PHT_COUNTS_THRESHOLD; e->counts_chunk = PHT_COUNTS_CHUNK;
    if (const char *ev = getenv("PHT_B200_COUNTS_THRESHOLD")) { const long v = atol(ev); if (v >= 1) e->counts_threshold = (uint32_t)v; }
    if (const char *ev = getenv("PHT_B200_COUNTS_CHUNK")) { const long v = atol(ev); if (v >= 1 && v <= (1l << 24)) e->counts_chunk = (uint32_t)v; }
    std::vector<uint32_t> old; old.swap(e->h_counts);
    const bool had = e->counts_set;
    e->h_counts.assign(counts_local, counts_local + l);
    e->counts_set = true;
    if (counts_build(e)) {                          /* a failed allocation: back to the previous counts */
        const std::string msg = g_err;
        e->h_counts.swap(old); e->counts_set = had;
        if (had) counts_build(e); else counts_free(e);
        return fail("%s", msg.c_str());
    }
    return 0;
}

/* ---------------------------------------------------------------- panel observations (method 64) */
static void panel_free(PanelBufs &b, cudaStream_t st) {
    void *bufs[] = { b.py, b.pu, b.pc, b.pperm, b.pgofs, b.vy, b.vu, b.vt, b.beta, b.vc, b.vperm, b.vm, b.vgofs, b.vcoff, b.voff, b.vnext };
    for (void *q : bufs) pht_dev_free(q, st);
    b = PanelBufs();
    cudaStreamSynchronize(st);
}

/* Both layouts from the visits in e->h_voff / h_vt / h_vm, in the engine's layout order (by group, then by decreasing y):
 * y, flags, u, local index and group offsets of each; the panel observations' chunk offsets and visits; the beta scratch
 * ((most visits + 1) n doubles per resident lane of the panel kernel).  A failed allocation leaves e->pan as it was. */
static int visits_build(pht_engine *e) {
    const long l = e->l_local;
    const int G = e->groups, n = e->cfg.n;
    const size_t ln = (size_t)(l > 0 ? l : 1);
    std::vector<double> y(ln), u; std::vector<uint8_t> c(ln); std::vector<uint32_t> order(ln);
    const uint32_t *dperm = G > 1 ? e->d_gperm : e->d_perm;
    if (l > 0) {
        CU(cudaMemcpy(y.data(), e->d_y, sizeof(double) * (size_t)l, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(c.data(), e->d_cens, (size_t)l, cudaMemcpyDeviceToHost));
        if (e->d_u) { u.resize(ln); CU(cudaMemcpy(u.data(), e->d_u, sizeof(double) * (size_t)l, cudaMemcpyDeviceToHost)); }
        if (dperm) CU(cudaMemcpy(order.data(), dperm, sizeof(uint32_t) * (size_t)l, cudaMemcpyDeviceToHost));
        else for (long i = 0; i < l; i++) order[(size_t)i] = (uint32_t)i;
    }
    std::vector<double> py, pu, vy, vu, vt; std::vector<uint8_t> pc, vc; std::vector<uint32_t> pperm, vperm, vm;
    std::vector<unsigned long long> pgofs((size_t)G + 1, 0ull), vgofs((size_t)G + 1, 0ull), vcoff((size_t)G + 1, 0ull), voff(1, 0ull);
    long mmax = 0;
    for (long pos = 0; pos < l; pos++) {
        const uint32_t k = order[(size_t)pos], g = G > 1 ? e->h_group[k] : 0u;
        const long m = (long)(e->h_voff[k + 1] - e->h_voff[k]);
        if (m == 0) {
            py.push_back(y[k]); pc.push_back(c[k]); pperm.push_back(k);
            if (!u.empty()) pu.push_back(u[k]);
            pgofs[(size_t)g + 1]++;
            continue;
        }
        vy.push_back(y[k]); vc.push_back(c[k]); vperm.push_back(k);
        if (!u.empty()) vu.push_back(u[k]);
        vgofs[(size_t)g + 1]++;
        for (int64_t q = e->h_voff[k]; q < e->h_voff[k + 1]; q++) { vt.push_back(e->h_vt[(size_t)q]); vm.push_back(e->h_vm[(size_t)q]); }
        voff.push_back(vt.size());
        if (m > mmax) mmax = m;
    }
    for (int g = 0; g < G; g++) {
        vcoff[(size_t)g + 1] = vcoff[(size_t)g] + (vgofs[(size_t)g + 1] + 31) / 32;
        pgofs[(size_t)g + 1] += pgofs[(size_t)g]; vgofs[(size_t)g + 1] += vgofs[(size_t)g];
    }
    PanelBufs b;
    cudaError_t ce = cudaSuccess;
    auto up = [&](void **dst, const void *src, size_t bytes) {
        if (ce == cudaSuccess) ce = pht_dev_alloc(dst, bytes ? bytes : 1, e->stream);
        if (ce == cudaSuccess && bytes && src) ce = cudaMemcpyAsync(*dst, src, bytes, cudaMemcpyHostToDevice, e->stream);
    };
    up((void **)&b.py, py.data(), sizeof(double) * py.size()); up((void **)&b.pc, pc.data(), pc.size());
    up((void **)&b.pperm, pperm.data(), sizeof(uint32_t) * pperm.size()); up((void **)&b.pgofs, pgofs.data(), sizeof(unsigned long long) * pgofs.size());
    up((void **)&b.vy, vy.data(), sizeof(double) * vy.size()); up((void **)&b.vc, vc.data(), vc.size());
    up((void **)&b.vperm, vperm.data(), sizeof(uint32_t) * vperm.size()); up((void **)&b.vgofs, vgofs.data(), sizeof(unsigned long long) * vgofs.size());
    up((void **)&b.vcoff, vcoff.data(), sizeof(unsigned long long) * vcoff.size()); up((void **)&b.voff, voff.data(), sizeof(unsigned long long) * voff.size());
    up((void **)&b.vt, vt.data(), sizeof(double) * vt.size()); up((void **)&b.vm, vm.data(), sizeof(uint32_t) * vm.size());
    if (!u.empty()) { up((void **)&b.pu, pu.data(), sizeof(double) * pu.size()); up((void **)&b.vu, vu.data(), sizeof(double) * vu.size()); }
    up((void **)&b.vnext, nullptr, sizeof(unsigned long long));
    const size_t beta_bytes = sizeof(double) * (size_t)e->panel_blocks * PHT_UNIF_PANEL_THREADS * (size_t)(mmax + 1) * (size_t)n;
    up((void **)&b.beta, nullptr, beta_bytes);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(e->stream);
    if (ce != cudaSuccess) {
        cudaGetLastError(); panel_free(b, e->stream); cudaGetLastError();
        return fail("cannot allocate device memory for the panel observations (%.1f MB of beta scratch for %ld visits per observation at most): %s",
                    beta_bytes / 1e6, mmax, cudaGetErrorString(ce));
    }
    panel_free(e->pan, e->stream);
    b.n_plain = (long)py.size(); b.n_panel = (long)vy.size();
    e->pan = b;
    if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }     /* kernel parameters change */
    return 0;
}

/* for every phase, the phases reachable from it through the nonzero cells of the structure (itself included); bit n: an exit */
static void reach_sets(int n, const int *T, const double *C, std::vector<uint64_t> &reach) {
    const int n1 = n + 1;
    reach.assign((size_t)n, 0ull);
    for (int i = 0; i < n; i++) {
        reach[(size_t)i] = 1ull << i;
        for (int j = 0; j <= n; j++) if (j != i && T[i + j * n1] != 0 && C[i + j * n1] != 0.0) reach[(size_t)i] |= 1ull << j;
    }
    for (bool grew = true; grew;) {
        grew = false;
        for (int i = 0; i < n; i++) {
            uint64_t r = reach[(size_t)i];
            for (int j = 0; j < n; j++) if ((r >> j) & 1ull) r |= reach[(size_t)j];
            if (r != reach[(size_t)i]) { reach[(size_t)i] = r; grew = true; }
        }
    }
}

/* Whether every observation's visits can happen: the phases it can be in at each visit, starting from the support of pi
 * (the start state itself when t_1 = 0) and moving along the nonzero cells of its group's structure (T, C: G structures of
 * (n+1)^2, gid: the group of every observation, or nullptr for one group), and for exact and interval data an exit after
 * the last visit (from the phase at y itself when an exact observation's last visit is at y).  0, or fail() naming the
 * first observation that cannot be drawn (its first draw would find only zero weights: error word 512). */
static int visits_reachable(int n, int G, const int *T, const double *C, const uint8_t *gid, const double *pi, long l,
                            const double *y, const uint8_t *c, const double *u, const int64_t *off, const double *t,
                            const uint32_t *mask) {
    const int n1 = n + 1;
    std::vector<std::vector<uint64_t>> reach((size_t)G);
    for (int g = 0; g < G; g++) reach_sets(n, T + (size_t)g * n1 * n1, C + (size_t)g * n1 * n1, reach[(size_t)g]);
    uint64_t start = 0;
    for (int i = 0; i < n; i++) if (pi[i] > 0.0) start |= 1ull << i;
    for (long k = 0; k < l; k++) {
        const int64_t v0 = off[k], m = off[k + 1] - v0;
        if (m == 0) continue;
        const size_t g = gid ? (size_t)gid[k] : 0;
        const std::vector<uint64_t> &R = reach[g];
        auto step = [&](uint64_t from) { uint64_t r = 0; for (int i = 0; i < n; i++) if ((from >> i) & 1ull) r |= R[(size_t)i]; return r; };
        uint64_t cur = (t[v0] == 0.0 ? start : step(start)) & mask[v0];
        for (int64_t q = v0 + 1; q < v0 + m && cur; q++) cur = step(cur) & mask[q];
        if (!cur) return fail("observation %ld: the start distribution and the structure cannot produce its visit sequence (no path from pi's support through the masks' phases)", k);
        const bool iv = u && u[k] < INFINITY;
        if (!c[k] || iv) {
            const size_t g0 = g * n1 * n1;
            const bool direct = !c[k] && t[v0 + m - 1] == y[k];
            bool ok = false;
            for (int i = 0; i < n; i++) {
                if (!((cur >> i) & 1ull)) continue;
                if (direct) ok = ok || (T[g0 + i + n * n1] != 0 && C[g0 + i + n * n1] != 0.0);
                else ok = ok || ((R[(size_t)i] >> n) & 1ull);
            }
            if (!ok) return fail("observation %ld: the structure cannot absorb after its last visit (no exit from the phases its visits allow)", k);
        }
    }
    return 0;
}

/* visits_reachable for the engine's visits (or the given ones) and data, against its structures and the given pi (nullptr:
 * chain 0's current pi), T / C / gid (nullptr: the engine's own) */
static int engine_visits_reachable(pht_engine *e, const int64_t *off, const double *t, const uint32_t *mask, const double *pi,
                                   int G, const int *T, const double *C, const uint8_t *gid) {
    const long l = e->l_local;
    const int n = e->cfg.n, n1 = n + 1;
    const size_t ln = (size_t)(l > 0 ? l : 1);
    std::vector<double> y(ln), u, p((size_t)n); std::vector<uint8_t> c(ln);
    std::vector<int> Th; std::vector<double> Ch;
    if (l > 0) {
        CU(cudaMemcpy(y.data(), e->d_y, sizeof(double) * (size_t)l, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(c.data(), e->d_cens, (size_t)l, cudaMemcpyDeviceToHost));
        if (e->d_u) { u.resize(ln); CU(cudaMemcpy(u.data(), e->d_u, sizeof(double) * (size_t)l, cudaMemcpyDeviceToHost)); }
    }
    if (pi) p.assign(pi, pi + n);
    else CU(cudaMemcpy(p.data(), e->d_model + e->L.pi, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost));
    if (!T) {
        G = e->groups;
        Th.resize((size_t)G * n1 * n1); Ch.resize(Th.size());
        CU(cudaMemcpy(Th.data(), e->d_T, sizeof(int) * Th.size(), cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(Ch.data(), e->d_C, sizeof(double) * Ch.size(), cudaMemcpyDeviceToHost));
        T = Th.data(); C = Ch.data();
        gid = G > 1 ? e->h_group.data() : nullptr;
    }
    return visits_reachable(n, G, T, C, gid, p.data(), l, y.data(), c.data(), u.empty() ? nullptr : u.data(), off, t, mask);
}

/* the engine refusals common to mask and stage visits */
static int visits_refused(const pht_engine *e) {
    if (method_of(e->cfg) != PHT_METHOD_UNIF)
        return fail("visits (panel observations) need method 64 (the uniformisation sampler): MHRS, ECS, DCS and the MH variants draw paths given the absorption time alone");
    if (e->peers_attached) return fail("visits cannot be set after the exchange windows are attached (visits need a single-rank engine)");
    if (e->cfg.world > 1) return fail("visits need world = 1: the panel observations are laid out and handed out on one rank");
    return 0;
}

/* pht_engine_set_visits and pht_engine_set_stage_visits: checks and stores the visits; val holds masks (colmask empty) or
 * stage indices into colmask, the support of every column of E.  The caller keeps the observation process. */
static int visits_upload(pht_engine *e, const int64_t *offsets_local, const double *t, const uint32_t *val, const std::vector<uint32_t> &colmask) {
    if (visits_refused(e)) return -1;
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    if (!offsets_local) {
        if (!e->visits_set) return 0;
        e->visits_set = false; e->h_voff.clear(); e->h_vt.clear(); e->h_vm.clear();
        panel_free(e->pan, e->stream);
        if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }
        return 0;
    }
    if (e->counts_set)
        return fail("visits are not supported with counts: the units of a record would share their visits; clear the counts with pht_engine_set_counts(e, NULL) first");
    const long l = e->l_local;
    const int n = e->cfg.n;
    if (offsets_local[0] != 0) return fail("offsets[0] = %lld: the visit offsets start at 0", (long long)offsets_local[0]);
    for (long k = 0; k < l; k++) {
        const int64_t m = offsets_local[k + 1] - offsets_local[k];
        if (m < 0) return fail("offsets[%ld] = %lld is below offsets[%ld] = %lld: the visit offsets must not decrease", k + 1, (long long)offsets_local[k + 1], k, (long long)offsets_local[k]);
        if (m > PHT_MAX_VISITS) return fail("observation %ld has %lld visits, more than PHT_MAX_VISITS = %d", k, (long long)m, PHT_MAX_VISITS);
    }
    const size_t ln = (size_t)(l > 0 ? l : 1);
    std::vector<double> y(ln);
    if (l > 0) CU(cudaMemcpy(y.data(), e->d_y, sizeof(double) * (size_t)l, cudaMemcpyDeviceToHost));
    const uint32_t all = n == 32 ? 0xffffffffu : (1u << n) - 1u;
    bool any = false;
    for (long k = 0; k < l; k++) {
        const int64_t v0 = offsets_local[k], m = offsets_local[k + 1] - v0;
        if (m == 0) continue;
        any = true;
        const double yk = y[(size_t)k];
        if (yk == 0.0 && (m > 1 || t[v0] != 0.0))
            return fail("observation %ld has y = 0: it takes a single visit at t = 0 (the stage at the start), no other", k);
        for (int64_t q = v0; q < v0 + m; q++) {
            if (!(t[q] >= 0.0)) return fail("visit %lld of observation %ld: t = %g is negative or NaN", (long long)(q - v0), k, t[q]);
            if (t[q] > yk) return fail("visit %lld of observation %ld: t = %g is above y = %g", (long long)(q - v0), k, t[q], yk);
            if (q > v0 && !(t[q] > t[q - 1])) return fail("visit %lld of observation %ld: t = %g does not follow t = %g (the times must increase)", (long long)(q - v0), k, t[q], t[q - 1]);
            if (!colmask.empty()) {
                if (val[q] >= colmask.size()) return fail("visit %lld of observation %ld: stage %u is not below stages = %d", (long long)(q - v0), k, val[q], (int)colmask.size());
                continue;
            }
            if (val[q] == 0u) return fail("visit %lld of observation %ld has an empty mask", (long long)(q - v0), k);
            if (val[q] & ~all) return fail("visit %lld of observation %ld: mask 0x%x has bits at or above n = %d", (long long)(q - v0), k, val[q], n);
        }
        if (e->entry_set && t[v0] < e->h_entry[(size_t)k])
            return fail("observation %ld: its first visit t = %g is before its entry age a = %g", k, t[v0], e->h_entry[(size_t)k]);
    }
    if (any && engine_visits_reachable(e, offsets_local, t, visit_masks(val, (size_t)offsets_local[l], colmask).data(), nullptr, 0, nullptr, nullptr, nullptr))
        return -1;
    if (!e->panel_blocks) {
        e->panel_blocks = pht_unif_panel_grid_blocks(e->cfg.device, n);
        if (e->panel_blocks <= 0) { e->panel_blocks = 0; return fail("the panel path kernel does not fit on the device: %s", cudaGetErrorString(cudaGetLastError())); }
    }
    if (!any) {                                    /* no visits at all: the plain engine */
        if (e->visits_set) { e->visits_set = false; e->h_voff.clear(); e->h_vt.clear(); e->h_vm.clear(); panel_free(e->pan, e->stream); }
        if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }
        return 0;
    }
    const int64_t total = offsets_local[l];
    std::vector<int64_t> ovoff; std::vector<double> ovt; std::vector<uint32_t> ovm;
    ovoff.swap(e->h_voff); ovt.swap(e->h_vt); ovm.swap(e->h_vm);
    e->h_voff.assign(offsets_local, offsets_local + l + 1);
    e->h_vt.assign(t, t + total); e->h_vm.assign(val, val + total);
    if (visits_build(e)) {                          /* a failed allocation: back to the previous visits */
        e->h_voff.swap(ovoff); e->h_vt.swap(ovt); e->h_vm.swap(ovm);
        return -1;
    }
    e->visits_set = true;
    return 0;
}

/* back to mask visits (or none): the observation process of stage visits goes */
static void emission_free(pht_engine *e) {
    void *bufs[] = { e->d_E, e->d_alpha, e->d_Eres, e->d_K };
    for (void *q : bufs) pht_dev_free(q, e->stream);
    cudaStreamSynchronize(e->stream);
    e->d_E = e->d_alpha = e->d_Eres = nullptr; e->d_K = nullptr;
    e->stages = 0; e->h_colmask.clear(); e->eres_rows = 0;
}

extern "C" int pht_engine_set_visits(pht_engine *e, const int64_t *offsets_local, const double *t, const uint32_t *mask) {
    if (!e) return fail("null engine");
    if (visits_upload(e, offsets_local, t, mask, std::vector<uint32_t>())) return -1;
    emission_free(e);
    return 0;
}

/* alpha (n x S) checked as pht_engine_set_stage_visits states, against the support of E (n x S) */
static int alpha_check(int n, int S, const double *E, const double *alpha) {
    for (int c = 0; c < n; c++)
        for (int o = 0; o < S; o++) {
            const double a = alpha[c * S + o], v = E[c * S + o];
            if (!(a >= 0.0) || !std::isfinite(a)) return fail("alpha[%d, %d] = %g: Dirichlet parameters must be finite and not negative", c, o, a);
            if (a > 0.0 && a < 0.1) return fail("alpha[%d, %d] = %g is below 0.1: Gamma draws of such shapes underflow to 0 often enough to make a visit impossible mid-run (0 is a structural zero)", c, o, a);
            if ((a > 0.0) != (v > 0.0)) return fail("alpha[%d, %d] = %g but E[%d, %d] = %g: E's support must equal alpha's (alpha = 0 is a structural zero)", c, o, a, c, o, v);
        }
    return 0;
}

/* E (n x S) and alpha (n x S or nullptr) checked as pht_engine_set_stage_visits states; colmask receives E's column supports */
static int emission_check(int n, int S, const double *E, const double *alpha, std::vector<uint32_t> &colmask) {
    colmask.assign((size_t)S, 0u);
    for (int c = 0; c < n; c++) {
        double sum = 0.0;
        for (int o = 0; o < S; o++) {
            const double v = E[c * S + o];
            if (!(v >= 0.0) || !std::isfinite(v)) return fail("E[%d, %d] = %g is not a probability", c, o, v);
            sum += v;
            if (v > 0.0) colmask[(size_t)o] |= 1u << c;
        }
        if (!(std::fabs(sum - 1.0) <= 1e-12)) return fail("row %d of E sums to %.17g, not 1 (within 1e-12)", c, sum);
    }
    return alpha ? alpha_check(n, S, E, alpha) : 0;
}

static int emis_grid(pht_engine *e, int S) {
    const int b = pht_unif_emis_grid_blocks(e->cfg.device, e->cfg.n, S);
    if (b <= 0) return fail("the stage-visit path kernel does not fit on the device: %s", cudaGetErrorString(cudaGetLastError()));
    return b;
}

extern "C" int pht_engine_set_stage_visits(pht_engine *e, int stages, const double *E, const double *alpha, const int64_t *offsets_local,
                                           const double *t, const uint32_t *stage) {
    if (!e) return fail("null engine");
    if (!offsets_local) {
        if (visits_upload(e, nullptr, nullptr, nullptr, std::vector<uint32_t>())) return -1;
        emission_free(e);
        return 0;
    }
    if (visits_refused(e)) return -1;
    if (stages < 1 || stages > PHT_MAX_STAGES) return fail("stages = %d outside 1..%d", stages, PHT_MAX_STAGES);
    if (!E) return fail("null emission matrix");
    const int n = e->cfg.n, S = stages;
    const size_t nS = (size_t)n * S, chains = (size_t)e->chains;
    std::vector<uint32_t> colmask;
    if (emission_check(n, S, E, alpha, colmask)) return -1;
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    if (!e->panel_blocks) {
        e->panel_blocks = pht_unif_panel_grid_blocks(e->cfg.device, n);
        if (e->panel_blocks <= 0) { e->panel_blocks = 0; return fail("the panel path kernel does not fit on the device: %s", cudaGetErrorString(cudaGetLastError())); }
    }
    const int blocks = emis_grid(e, S);
    if (blocks < 0) return -1;
    /* the new observation process first: a refusal or a failed allocation leaves the engine as it was */
    double *dE = nullptr, *dalpha = nullptr; unsigned long long *dK = nullptr;
    cudaError_t ce = pht_dev_alloc((void **)&dE, sizeof(double) * chains * nS, e->stream);
    if (ce == cudaSuccess) ce = pht_dev_alloc((void **)&dK, sizeof(unsigned long long) * chains * nS, e->stream);
    if (ce == cudaSuccess && alpha) ce = pht_dev_alloc((void **)&dalpha, sizeof(double) * nS, e->stream);
    for (size_t c = 0; c < chains && ce == cudaSuccess; c++) ce = cudaMemcpyAsync(dE + c * nS, E, sizeof(double) * nS, cudaMemcpyHostToDevice, e->stream);
    if (ce == cudaSuccess) ce = cudaMemsetAsync(dK, 0, sizeof(unsigned long long) * chains * nS, e->stream);
    if (ce == cudaSuccess && alpha) ce = cudaMemcpyAsync(dalpha, alpha, sizeof(double) * nS, cudaMemcpyHostToDevice, e->stream);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(e->stream);
    auto drop = [&]() { void *b[] = { dE, dK, dalpha }; for (void *q : b) pht_dev_free(q, e->stream); cudaStreamSynchronize(e->stream); };
    if (ce != cudaSuccess) {
        cudaGetLastError(); drop(); cudaGetLastError();
        return fail("cannot allocate device memory for the emission matrices: %s", cudaGetErrorString(ce));
    }
    if (visits_upload(e, offsets_local, t, stage, colmask)) { drop(); return -1; }
    emission_free(e);
    if (!e->visits_set) { drop(); return 0; }      /* no visits at all: the plain engine */
    e->d_E = dE; e->d_K = dK; e->d_alpha = dalpha;
    e->stages = S; e->h_colmask = colmask; e->emis_blocks = std::min(blocks, e->panel_blocks);
    if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }
    return 0;
}

/* E NULL keeps every chain's own E (a prior is then checked against each of them); the new buffers are filled before
 * the old ones go, so a refusal or a failed copy leaves the engine as it was */
extern "C" int pht_engine_set_emission(pht_engine *e, const double *E, const double *alpha) {
    if (!e) return fail("null engine");
    if (!e->stages) return fail("the emission matrix belongs to stage visits: set them with pht_engine_set_stage_visits first");
    const int n = e->cfg.n, S = e->stages;
    const size_t nS = (size_t)n * S, chains = (size_t)e->chains;
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    std::vector<uint32_t> colmask = e->h_colmask;
    if (E) {
        if (emission_check(n, S, E, alpha, colmask)) return -1;
        if (colmask != e->h_colmask &&
            engine_visits_reachable(e, e->h_voff.data(), e->h_vt.data(), visit_masks(e->h_vm.data(), e->h_vm.size(), colmask).data(), nullptr, 0, nullptr, nullptr, nullptr))
            return -1;
    } else if (alpha) {
        std::vector<double> cur(chains * nS);
        CU(cudaMemcpy(cur.data(), e->d_E, sizeof(double) * cur.size(), cudaMemcpyDeviceToHost));
        for (size_t c = 0; c < chains; c++)
            if (alpha_check(n, S, cur.data() + c * nS, alpha)) {
                const std::string msg = pht_last_error();
                return fail("%s (chain %zu's E)", msg.c_str(), c);
            }
    }
    double *dE = nullptr, *dalpha = nullptr;
    cudaError_t ce = cudaSuccess;
    if (E) ce = pht_dev_alloc((void **)&dE, sizeof(double) * chains * nS, e->stream);
    for (size_t c = 0; c < chains && E && ce == cudaSuccess; c++) ce = cudaMemcpyAsync(dE + c * nS, E, sizeof(double) * nS, cudaMemcpyHostToDevice, e->stream);
    if (alpha && ce == cudaSuccess) ce = pht_dev_alloc((void **)&dalpha, sizeof(double) * nS, e->stream);
    if (alpha && ce == cudaSuccess) ce = cudaMemcpyAsync(dalpha, alpha, sizeof(double) * nS, cudaMemcpyHostToDevice, e->stream);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(e->stream);
    if (ce != cudaSuccess) {
        cudaGetLastError();
        pht_dev_free(dE, e->stream); pht_dev_free(dalpha, e->stream);
        cudaStreamSynchronize(e->stream); cudaGetLastError();
        return fail("cannot set the emission matrix or its prior: %s", cudaGetErrorString(ce));
    }
    if (E) { pht_dev_free(e->d_E, e->stream); e->d_E = dE; }
    pht_dev_free(e->d_alpha, e->stream); e->d_alpha = dalpha;
    cudaStreamSynchronize(e->stream);
    e->h_colmask = colmask;
    if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }     /* new pointers; the update comes or goes */
    return 0;
}

extern "C" int pht_engine_get_emission(pht_engine *e, double *E) {
    if (!e || !E) return fail("null argument");
    if (!e->stages) return fail("no stage visits are set (pht_engine_set_stage_visits)");
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    CU(cudaMemcpy(E, e->d_E, sizeof(double) * (size_t)e->cfg.n * e->stages, cudaMemcpyDeviceToHost));
    return 0;
}

extern "C" int pht_engine_emission_rows(pht_engine *e, int rows, double *out) {
    if (!e || rows < 0) return fail("bad argument");
    if (!e->stages || !e->d_alpha) return fail("E is not being inferred (pht_engine_set_stage_visits or pht_engine_set_emission with a prior first)");
    if (rows > e->eres_rows || !e->d_Eres) return fail("%d rows asked, the last run produced at most %d", rows, e->d_Eres ? e->eres_rows : 0);
    if (rows == 0) return 0;
    if (!out) return fail("null argument");
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    const size_t nS = (size_t)e->cfg.n * e->stages, R = (size_t)e->eres_rows;
    CU(cudaMemcpy2D(out, sizeof(double) * rows * nS, e->d_Eres, sizeof(double) * R * nS, sizeof(double) * rows * nS, e->chains, cudaMemcpyDeviceToHost));
    return 0;
}

/* pht_engine_paths with visits: the window's panel observations through k_unif_panel_paths (chain 0, every group on its own
 * model and table), recorded at their window positions over what the plain kernels recorded there */
static int panel_window(pht_engine *e, long first, long count, int *B, int *N, double *z) {
    const int n = e->cfg.n, G = e->groups;
    std::vector<std::vector<uint32_t>> byg((size_t)G);
    for (long k = first; k < first + count; k++)
        if (e->h_voff[(size_t)k + 1] > e->h_voff[(size_t)k]) byg[G > 1 ? e->h_group[(size_t)k] : 0].push_back((uint32_t)k);
    std::vector<uint32_t> perm; std::vector<unsigned long long> gofs((size_t)G + 1, 0ull), coff((size_t)G + 1, 0ull), voff(1, 0ull);
    std::vector<double> vt; std::vector<uint32_t> vm;
    for (int g = 0; g < G; g++) {
        for (uint32_t k : byg[(size_t)g]) {
            perm.push_back(k);
            for (int64_t q = e->h_voff[k]; q < e->h_voff[(size_t)k + 1]; q++) { vt.push_back(e->h_vt[(size_t)q]); vm.push_back(e->h_vm[(size_t)q]); }
            voff.push_back(vt.size());
        }
        gofs[(size_t)g + 1] = perm.size();
        coff[(size_t)g + 1] = coff[(size_t)g] + (byg[(size_t)g].size() + 31) / 32;
    }
    const long cnt = (long)perm.size();
    if (cnt == 0) return 0;
    std::vector<double> yw((size_t)count), uw, y((size_t)cnt), u; std::vector<uint8_t> cw((size_t)count), c((size_t)cnt);
    CU(cudaMemcpy(yw.data(), e->d_y + first, sizeof(double) * count, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(cw.data(), e->d_cens + first, (size_t)count, cudaMemcpyDeviceToHost));
    if (e->d_u) { uw.resize((size_t)count); u.resize((size_t)cnt); CU(cudaMemcpy(uw.data(), e->d_u + first, sizeof(double) * count, cudaMemcpyDeviceToHost)); }
    for (long j = 0; j < cnt; j++) {
        const size_t wpos = (size_t)(perm[(size_t)j] - first);
        y[(size_t)j] = yw[wpos]; c[(size_t)j] = cw[wpos];
        if (!u.empty()) u[(size_t)j] = uw[wpos];
    }
    PanelBufs w;
    int *dB = nullptr, *dN = nullptr; double *dz = nullptr;
    int rc = -1;
#define CUP(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { fail("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); goto out; } } while (0)
    {
        auto up = [&](void **dst, const void *src, size_t bytes) -> cudaError_t {
            cudaError_t ce = cudaMalloc(dst, bytes ? bytes : 1);
            if (ce == cudaSuccess && bytes && src) ce = cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice);
            return ce;
        };
        CUP(up((void **)&w.vy, y.data(), sizeof(double) * cnt)); CUP(up((void **)&w.vc, c.data(), (size_t)cnt));
        if (!u.empty()) CUP(up((void **)&w.vu, u.data(), sizeof(double) * cnt));
        CUP(up((void **)&w.vperm, perm.data(), sizeof(uint32_t) * cnt)); CUP(up((void **)&w.vgofs, gofs.data(), sizeof(unsigned long long) * gofs.size()));
        CUP(up((void **)&w.vcoff, coff.data(), sizeof(unsigned long long) * coff.size())); CUP(up((void **)&w.voff, voff.data(), sizeof(unsigned long long) * voff.size()));
        CUP(up((void **)&w.vt, vt.data(), sizeof(double) * vt.size())); CUP(up((void **)&w.vm, vm.data(), sizeof(uint32_t) * vm.size()));
        CUP(up((void **)&w.vnext, nullptr, sizeof(unsigned long long)));
        w.beta = e->pan.beta;                       /* sized for the longest panel of the engine */
        CUP(cudaMalloc(&dB, sizeof(int) * count)); CUP(cudaMalloc(&dN, sizeof(int) * count * n * n)); CUP(cudaMalloc(&dz, sizeof(double) * count * n));
        CUP(cudaMemset(dN, 0, sizeof(int) * count * n * n));
        UpdateParams up_ = update_params(e, nullptr, 0);
        up_.chains = 1;
        if (enqueue_model(e, up_)) goto out;
        SweepParams p = sweep_params(e);
        p.chains = 1;
        p.outB = dB; p.outN = dN; p.outz = dz; p.first = first; p.count = count;
        CUP(launch_panel_kernel(e, p, panel_args(w)));
        e->launches++;
        if (pht_engine_sync(e)) goto out;
        std::vector<int> hB((size_t)count), hN((size_t)count * n * n); std::vector<double> hz((size_t)count * n);
        CUP(cudaMemcpy(hB.data(), dB, sizeof(int) * count, cudaMemcpyDeviceToHost));
        CUP(cudaMemcpy(hN.data(), dN, sizeof(int) * count * n * n, cudaMemcpyDeviceToHost));
        CUP(cudaMemcpy(hz.data(), dz, sizeof(double) * count * n, cudaMemcpyDeviceToHost));
        for (uint32_t k : perm) {
            const size_t wpos = (size_t)(k - first);
            B[wpos] = hB[wpos];
            memcpy(N + wpos * n * n, hN.data() + wpos * n * n, sizeof(int) * n * n);
            memcpy(z + wpos * n, hz.data() + wpos * n, sizeof(double) * n);
        }
        rc = 0;
    }
#undef CUP
out:
    void *bufs[] = { w.vy, w.vc, w.vu, w.vperm, w.vgofs, w.vcoff, w.voff, w.vt, w.vm, w.vnext, dB, dN, dz };
    for (void *q : bufs) if (q) cudaFree(q);
    return rc;
}

extern "C" int pht_engine_set_upper(pht_engine *e, const double *upper_local) {
    if (!e) return fail("null engine");
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    if (e->peers_attached) return fail("the interval bounds of a multi-rank run are set on every rank before the exchange windows are attached");
    if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }     /* kernel parameters change */
    if (!upper_local) {
        double *bufs[] = { e->d_u, e->d_us, e->d_item_u };
        for (double *b : bufs) CU(pht_dev_free(b, e->stream));
        e->d_u = e->d_us = e->d_item_u = nullptr;
        CU(cudaStreamSynchronize(e->stream));
        if (method_of(e->cfg) == PHT_METHOD_UNIF) {
            std::vector<double> y((size_t)(e->l_local > 0 ? e->l_local : 1));
            if (e->l_local > 0) CU(cudaMemcpy(y.data(), e->d_y, sizeof(double) * (size_t)e->l_local, cudaMemcpyDeviceToHost));
            e->unif_tmax = 0.0;
            for (long i = 0; i < e->l_local; i++) if (y[(size_t)i] > e->unif_tmax) e->unif_tmax = y[(size_t)i];
        }
        if (group_refresh(e)) return -1;
        if (e->visits_set) return visits_build(e);
        return e->counts_set ? counts_build(e) : 0;
    }
    const bool unif = method_of(e->cfg) == PHT_METHOD_UNIF;
    if (method_of(e->cfg) != PHT_METHOD_MHRS && !unif)
        return fail("interval-censored observations need method MHRS or 64 (ECS, DCS and the MH variants have no conditional law for a bounded absorption time)");
    const long l = e->l_local;
    std::vector<double> y((size_t)(l > 0 ? l : 1)); std::vector<uint8_t> c((size_t)(l > 0 ? l : 1));
    if (l > 0) {
        CU(cudaMemcpy(y.data(), e->d_y, sizeof(double) * (size_t)l, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(c.data(), e->d_cens, (size_t)l, cudaMemcpyDeviceToHost));
    }
    /* an interval path ends by u, not by y: the fixed-point scale must leave room for sum max(y, u) (each record counted
     * as often as its count, when counts are set) */
    double sum = 0.0, tmax = 0.0;
    for (long i = 0; i < l; i++) {
        const double u = upper_local[i], wgt = e->counts_set ? (double)e->h_counts[(size_t)i] : 1.0;
        if (y[(size_t)i] > tmax) tmax = y[(size_t)i];
        if (std::isnan(u)) return fail("upper[%ld] is NaN", i);
        if (u == INFINITY) { sum += wgt * y[(size_t)i]; continue; }
        if (!(u > y[(size_t)i])) return fail("upper[%ld] = %g is not above y = %g", i, u, y[(size_t)i]);
        if (!c[(size_t)i]) return fail("upper[%ld] = %g on an exact observation: a finite bound needs the censoring flag", i, u);
        /* (the rejection loop `while (t < y || t > u)` runs no attempt at all when y = 0; method 64 takes y = 0 as a
         * failure before the first inspection: left-censored) */
        if (!unif && !(y[(size_t)i] > 0.0)) return fail("upper[%ld] = %g with y = %g: an interval needs y > 0 (a tiny y for a failure before the first inspection)", i, u, y[(size_t)i]);
        if (unif && !(y[(size_t)i] >= 0.0)) return fail("upper[%ld] = %g with y = %g: an interval needs y >= 0", i, u, y[(size_t)i]);
        if (u - y[(size_t)i] > tmax) tmax = u - y[(size_t)i];
        sum += wgt * u;
    }
    for (double a : e->h_entry) sum += a;           /* ghost paths of delayed-entry observations (pht_engine_set_entry) */
    if (sum > 0.0 && e->cfg.zbits > pht_choose_zbits(sum))
        return fail("zbits = %d is too fine for these bounds: interval paths end by u, and sum of max(y, u) (plus the entry ages, when set; times the counts, when set) = %g allows at most %d",
                    e->cfg.zbits, sum, pht_choose_zbits(sum));
    const size_t ln = (size_t)(l > 0 ? l : 1);
    if (unif) e->unif_tmax = tmax;
    if (!unif && !e->iv_blocks[0] && pht_mhrs_grid_blocks(e->cfg.device, e->cfg.n, true, &e->iv_blocks[0], &e->iv_blocks[1], &e->iv_blocks[2]) != 0) {
        e->iv_blocks[0] = 0;
        return fail("MHRS interval kernels do not fit on the device: %s", cudaGetErrorString(cudaGetLastError()));
    }
    if (!e->d_u) CU(pht_dev_alloc((void **)&e->d_u, ln * sizeof(double), e->stream));
    if (e->d_ys && !e->d_us) CU(pht_dev_alloc((void **)&e->d_us, ln * sizeof(double), e->stream));
    if (!unif && !e->d_item_u) CU(pht_dev_alloc((void **)&e->d_item_u, (size_t)e->item_cap * sizeof(double), e->stream));
    if (l > 0) {
        CU(cudaMemcpyAsync(e->d_u, upper_local, sizeof(double) * (size_t)l, cudaMemcpyHostToDevice, e->stream));
        if (e->d_ys) CU(pht_gather_f64(e->d_u, e->d_perm, e->d_us, l, e->stream));
    }
    CU(cudaStreamSynchronize(e->stream));
    if (group_refresh(e)) return -1;
    if (e->visits_set) return visits_build(e);     /* u in the panel layouts */
    return e->counts_set ? counts_build(e) : 0;
}

static int entry_free(pht_engine *e) {
    void *bufs[] = { e->d_entry, e->d_ea, e->d_eobs, e->d_eM, e->d_eoff, e->d_enext, e->d_etab, e->d_escan };
    for (void *b : bufs) CU(pht_dev_free(b, e->stream));
    e->d_entry = e->d_ea = e->d_etab = nullptr; e->d_eobs = nullptr; e->d_eM = nullptr; e->d_eoff = e->d_enext = nullptr;
    e->d_escan = nullptr; e->escan_bytes = 0; e->n_trunc = 0;
    e->entry_set = false; e->h_entry.clear();
    CU(cudaStreamSynchronize(e->stream));
    return 0;
}

extern "C" int pht_engine_set_entry(pht_engine *e, const double *entry_local) {
    if (!e) return fail("null engine");
    if (method_of(e->cfg) != PHT_METHOD_UNIF)
        return fail("delayed entry (entry ages, left truncation) needs method 64: the units lost before entry are drawn as left-censored paths of the uniformisation sampler");
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    if (e->peers_attached) return fail("the entry ages of a multi-rank run are set on every rank before the exchange windows are attached");
    if (entry_local && e->chains > 1)
        return fail("entry ages (delayed entry) are not supported with %d chains: the ghost paths are drawn for one chain; pht_engine_set_chains(e, 1, ...) first", e->chains);
    if (entry_local && e->counts_set)
        return fail("entry ages (delayed entry) are not supported with counts: a record's ghost count would be a sum of w Geometric draws; clear the counts with pht_engine_set_counts(e, NULL) first");
    if (entry_local && e->groups > 1)
        return fail("entry ages (delayed entry) are not supported with %d groups: the ghost paths are drawn on one model; pht_engine_set_groups(e, 1, ...) or (e, 0, NULL, ...) first", e->groups);
    if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }     /* the sweep changes shape */
    if (!entry_local) return entry_free(e);
    const long l = e->l_local;
    const size_t ln = (size_t)(l > 0 ? l : 1);
    std::vector<double> y(ln), u(ln, INFINITY);
    if (l > 0) {
        CU(cudaMemcpy(y.data(), e->d_y, sizeof(double) * (size_t)l, cudaMemcpyDeviceToHost));
        if (e->d_u) CU(cudaMemcpy(u.data(), e->d_u, sizeof(double) * (size_t)l, cudaMemcpyDeviceToHost));
    }
    /* ghost paths end by their entry age: the fixed-point scale must leave room for sum of max(y, u) + a */
    double sum = 0.0;
    std::vector<uint32_t> trunc;
    for (long i = 0; i < l; i++) {
        const double a = entry_local[i], yi = y[(size_t)i], ui = u[(size_t)i];
        if (!std::isfinite(a)) return fail("entry[%ld] = %g: an entry age must be finite", i, a);
        if (a < 0.0) return fail("entry[%ld] = %g is negative", i, a);
        if (a > yi) return fail("entry[%ld] = %g is above y = %g: a unit enters before its failure or censoring time (a left-censored record, y = 0, takes no entry age)", i, a, yi);
        if (e->visits_set && e->h_voff[(size_t)i + 1] > e->h_voff[(size_t)i] && e->h_vt[(size_t)e->h_voff[(size_t)i]] < a)
            return fail("entry[%ld] = %g is after the observation's first visit t = %g", i, a, e->h_vt[(size_t)e->h_voff[(size_t)i]]);
        sum += (ui < INFINITY && ui > yi ? ui : yi) + a;
        if (a > 0.0) trunc.push_back((uint32_t)i);
    }
    if (sum > 0.0 && e->cfg.zbits > pht_choose_zbits(sum))
        return fail("zbits = %d is too fine for these entry ages: ghost paths end by a, and sum of max(y, u) + a = %g allows at most %d",
                    e->cfg.zbits, sum, pht_choose_zbits(sum));
    if (!e->ghost_blocks) {
        e->ghost_blocks = pht_unif_ghost_grid_blocks(e->cfg.device, e->cfg.n);
        if (e->ghost_blocks <= 0) { e->ghost_blocks = 0; return fail("the ghost-path kernel does not fit on the device: %s", cudaGetErrorString(cudaGetLastError())); }
        int sms = 0;
        CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->cfg.device));
        e->count_blocks = 8 * sms;                   /* the count kernel is grid-stride: 8 blocks of 256 per SM */
    }
    if (entry_free(e)) return -1;
    /* the truncated observations by decreasing a (ties by index), so that the lanes of a warp run similar truncations */
    std::stable_sort(trunc.begin(), trunc.end(), [&](uint32_t i, uint32_t j) { return entry_local[i] > entry_local[j]; });
    const long nt = (long)trunc.size();
    std::vector<double> ea((size_t)(nt > 0 ? nt : 1));
    for (long k = 0; k < nt; k++) ea[(size_t)k] = entry_local[trunc[(size_t)k]];
    CU(pht_dev_alloc((void **)&e->d_entry, ln * sizeof(double), e->stream));
    CU(pht_dev_alloc((void **)&e->d_ea, ea.size() * sizeof(double), e->stream));
    CU(pht_dev_alloc((void **)&e->d_eobs, ea.size() * sizeof(uint32_t), e->stream));
    CU(pht_dev_alloc((void **)&e->d_eM, (size_t)(nt + 1) * sizeof(unsigned), e->stream));
    CU(pht_dev_alloc((void **)&e->d_eoff, (size_t)(nt + 1) * sizeof(unsigned long long), e->stream));
    CU(pht_dev_alloc((void **)&e->d_enext, sizeof(unsigned long long), e->stream));
    CU(pht_dev_alloc((void **)&e->d_etab, 2 * PHT_UNIF_CAP * sizeof(double), e->stream));
    e->escan_bytes = pht_unif_entry_scan_bytes(nt);
    CU(pht_dev_alloc(&e->d_escan, e->escan_bytes ? e->escan_bytes : 1, e->stream));
    if (l > 0) CU(cudaMemcpyAsync(e->d_entry, entry_local, sizeof(double) * (size_t)l, cudaMemcpyHostToDevice, e->stream));
    if (nt > 0) {
        CU(cudaMemcpyAsync(e->d_ea, ea.data(), sizeof(double) * (size_t)nt, cudaMemcpyHostToDevice, e->stream));
        CU(cudaMemcpyAsync(e->d_eobs, trunc.data(), sizeof(uint32_t) * (size_t)nt, cudaMemcpyHostToDevice, e->stream));
    }
    CU(cudaStreamSynchronize(e->stream));
    e->h_entry.assign(entry_local, entry_local + l);
    e->n_trunc = nt; e->entry_set = true;
    return 0;
}

extern "C" int pht_engine_entry_paths(pht_engine *e, long first, long count, int *M, long total, int *B, int *N, double *z) {
    if (!e || !M) return fail("null argument");
    if (method_of(e->cfg) != PHT_METHOD_UNIF) return fail("delayed entry (entry ages, left truncation) needs method 64");
    if (first < 0 || count < 0 || first + count > e->l_local) return fail("range [%ld, %ld) outside the shard", first, first + count);
    if (B && (!N || !z)) return fail("null argument");
    if (count == 0 || !e->entry_set) {
        for (long i = 0; i < count; i++) M[i] = 0;
        if (B && total != 0) return fail("%ld ghost paths asked, the window has none (no entry ages set)", total);
        return 0;
    }
    CU(cudaSetDevice(e->cfg.device));
    const int n = e->cfg.n;
    unsigned *dM = nullptr; unsigned long long *doff = nullptr; void *tmp = nullptr;
    int *dB = nullptr, *dN = nullptr; double *dz = nullptr;
    int rc = -1;
#define CUP(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { fail("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); goto out; } } while (0)
    {
        UnifEntry E; memset(&E, 0, sizeof(E));
        E.scan_bytes = pht_unif_entry_scan_bytes(count);
        CUP(cudaMalloc(&dM, sizeof(unsigned) * (count + 1))); CUP(cudaMalloc(&doff, sizeof(unsigned long long) * (count + 1)));
        CUP(cudaMalloc(&tmp, E.scan_bytes ? E.scan_bytes : 1));
        /* the window in upload order: entry ages d_entry[first + i], local observation first + i */
        E.a = e->d_entry + first; E.obs = nullptr; E.first = first; E.count = count; E.M = dM; E.off = doff;
        E.etab = e->d_etab; E.next = e->d_enext; E.scan_tmp = tmp; E.count_blocks = e->count_blocks;
        UpdateParams u = update_params(e, nullptr, 0);
        u.chains = 1;
        if (enqueue_model(e, u)) goto out;
        SweepParams p = sweep_params(e);
        p.chains = 1;
        CUP(pht_launch_unif_entry(u, p, e->d_unif, E, e->ghost_blocks, PHT_ENTRY_COUNTS, e->stream));
        if (pht_engine_sync(e)) goto out;
        std::vector<unsigned> hM((size_t)count);
        unsigned long long G = 0;
        CUP(cudaMemcpy(hM.data(), dM, sizeof(unsigned) * count, cudaMemcpyDeviceToHost));
        CUP(cudaMemcpy(&G, doff + count, sizeof(G), cudaMemcpyDeviceToHost));
        for (long i = 0; i < count; i++) M[i] = (int)hM[(size_t)i];
        if (B) {
            if ((unsigned long long)total != G) { fail("total = %ld, but the window's ghost counts sum to %llu", total, G); goto out; }
            if (G > 0) {
                CUP(cudaMalloc(&dB, sizeof(int) * G)); CUP(cudaMalloc(&dN, sizeof(int) * G * n * n)); CUP(cudaMalloc(&dz, sizeof(double) * G * n));
                CUP(cudaMemsetAsync(dN, 0, sizeof(int) * G * n * n, e->stream));
                p.outB = dB; p.outN = dN; p.outz = dz; p.first = 0; p.count = (long)G;
                CUP(pht_launch_unif_entry(u, p, e->d_unif, E, e->ghost_blocks, PHT_ENTRY_GHOSTS, e->stream));
                if (pht_engine_sync(e)) goto out;
                CUP(cudaMemcpy(B, dB, sizeof(int) * G, cudaMemcpyDeviceToHost));
                CUP(cudaMemcpy(N, dN, sizeof(int) * G * n * n, cudaMemcpyDeviceToHost));
                CUP(cudaMemcpy(z, dz, sizeof(double) * G * n, cudaMemcpyDeviceToHost));
            }
        }
        rc = 0;
    }
#undef CUP
out:
    cudaFree(dM); cudaFree(doff); cudaFree(tmp);
    if (dB) cudaFree(dB);
    if (dN) cudaFree(dN);
    if (dz) cudaFree(dz);
    return rc;
}

/* rows x m draws of theta and rows x n of pi per chain, chain 0 first (chain c's rows start at c x res_rows) */
static int ensure_res(pht_engine *e, int rows) {
    if (rows <= e->res_rows) return 0;
    CU(cudaStreamSynchronize(e->stream));
    if (e->d_res) { CU(pht_dev_free(e->d_res, e->stream)); e->d_res = nullptr; }
    CU(pht_dev_alloc((void **)&e->d_res, sizeof(double) * (size_t)e->chains * rows * e->cfg.m, e->stream));
    if (e->d_pires) { CU(pht_dev_free(e->d_pires, e->stream)); e->d_pires = nullptr; }
    CU(pht_dev_alloc((void **)&e->d_pires, sizeof(double) * (size_t)e->chains * rows * e->cfg.n, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    e->res_rows = rows;
    return 0;
}

extern "C" int pht_engine_enqueue(pht_engine *e, int nsweeps) {
    if (!e || nsweeps < 0) return fail("bad argument");
    CU(cudaSetDevice(e->cfg.device));
    if (ensure_res(e, nsweeps > 0 ? nsweeps : 1)) return -1;
    if (e->stages && e->d_alpha && (!e->d_Eres || e->eres_rows != e->res_rows)) {    /* rows of the E draws, like res */
        CU(cudaStreamSynchronize(e->stream));
        if (e->d_Eres) { CU(pht_dev_free(e->d_Eres, e->stream)); e->d_Eres = nullptr; e->eres_rows = 0; }
        CU(pht_dev_alloc((void **)&e->d_Eres, sizeof(double) * (size_t)e->chains * e->res_rows * e->cfg.n * e->stages, e->stream));
        CU(cudaStreamSynchronize(e->stream));
        e->eres_rows = e->res_rows;
        if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }
    }
    CU(cudaMemsetAsync(&e->d_state->res_row, 0, sizeof(uint32_t), e->stream));
    e->kev_used = 0;
    const bool graph = e->cfg.use_graph != 0;
    if (!graph) {
        const int want = 2 * (nsweeps < 64 ? nsweeps : 64);
        while ((int)e->kev.size() < want) { cudaEvent_t ev; CU(cudaEventCreate(&ev)); e->kev.push_back(ev); }
    }
    if (graph && (e->graph_exec == nullptr || e->graph_res != e->d_res || e->graph_res_rows != e->res_rows)) {
        if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }
        cudaGraph_t g = nullptr;
        CU(cudaStreamBeginCapture(e->stream, cudaStreamCaptureModeThreadLocal));
        const unsigned long long before = e->launches;
        int rc = enqueue_sweep(e, e->d_res, e->res_rows, false);
        e->graph_launches = e->launches - before; e->launches = before;      /* counted per replay below */
        cudaError_t ce = cudaStreamEndCapture(e->stream, &g);
        if (rc != 0) { if (g) cudaGraphDestroy(g); return -1; }
        if (ce != cudaSuccess) return fail("graph capture failed: %s", cudaGetErrorString(ce));
        ce = cudaGraphInstantiate(&e->graph_exec, g, 0);
        cudaGraphDestroy(g);
        if (ce != cudaSuccess) return fail("graph instantiate failed: %s", cudaGetErrorString(ce));
        e->graph_res = e->d_res; e->graph_res_rows = e->res_rows;
    }
    CU(cudaEventRecord(e->ev0, e->stream));
    for (int k = 0; k < nsweeps; k++) {
        if (e->d_flush) CU(cudaMemsetAsync(e->d_flush, k & 0xff, e->flush_bytes, e->stream));
        if (graph) { CU(cudaGraphLaunch(e->graph_exec, e->stream)); e->launches += e->graph_launches; }
        else if (enqueue_sweep(e, e->d_res, e->res_rows, k < 64)) return -1;
    }
    CU(cudaEventRecord(e->ev1, e->stream));
    return 0;
}

static int check_state(pht_engine *e) {
    DevState st; CU(cudaMemcpy(&st, e->d_state, sizeof(st), cudaMemcpyDeviceToHost));
    if (st.error) {
        int err = st.error;
        cudaMemsetAsync(&e->d_state->error, 0, sizeof(int), e->stream);
        cudaStreamSynchronize(e->stream);
        return fail("device error word 0x%x (%s%s%s%s%s%s%s%s%s%s)", err, (err & 2) ? "sojourn total overflows the fixed-point range (lower PHT_B200_ZBITS); " : "",
                    (err & 4) ? "MHRS tail list overflow; " : "",
                    (err & 8) ? "an observation's survival probability is too small for rejection sampling (more than 4e9 attempts); " : "",
                    (err & 16) ? "(unused) " : "",
                    (err & 32) ? "spectral decomposition failed; " : "",
                    (err & 64) ? "a peer GPU did not arrive at a barrier of the global MHRS tail; " : "",
                    (err & 128) ? "another rank of the run raised its error word; " : "",
                    (err & PHT_UNIF_ERR_TABLE) ? "the uniformisation sampler needs more powers of R than its table holds (a stiff generator or a very long y); " : "",
                    (err & PHT_UNIF_ERR_ZERO) ? "every weight of a uniformisation draw underflowed to zero; " : "",
                    (err & PHT_UNIF_ERR_ENTRY) ? "the model leaves (almost) no survival at an observation's entry age: S(a) underflowed or more than 2^20 units would have been lost before entry; " : "");
    }
    return 0;
}

extern "C" int pht_engine_sync(pht_engine *e) {
    if (!e) return fail("null engine");
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    return check_state(e);
}

extern "C" int pht_engine_set_l2_flush(pht_engine *e, unsigned long long bytes) {
    if (!e) return fail("null engine");
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    if (e->d_flush) { CU(cudaFree(e->d_flush)); e->d_flush = nullptr; e->flush_bytes = 0; }
    if (bytes) { CU(cudaMalloc(&e->d_flush, (size_t)bytes)); e->flush_bytes = (size_t)bytes; }
    return 0;
}

extern "C" int pht_engine_last_ms(pht_engine *e, float *total_ms, float *path_kernel_ms) {
    if (!e) return fail("null engine");
    if (total_ms) CU(cudaEventElapsedTime(total_ms, e->ev0, e->ev1));
    if (path_kernel_ms) {
        float acc = 0.f; int pairs = e->kev_used / 2;
        for (int i = 0; i < pairs; i++) { float ms; CU(cudaEventElapsedTime(&ms, e->kev[2 * i], e->kev[2 * i + 1])); acc += ms; }
        *path_kernel_ms = pairs ? acc / pairs : -1.f;
    }
    return 0;
}

extern "C" int pht_engine_run(pht_engine *e, int nsweeps, double *out) {
    if (pht_engine_enqueue(e, nsweeps)) return -1;
    if (pht_engine_sync(e)) return -1;
    if (out && nsweeps > 0) CU(cudaMemcpy(out, e->d_res, sizeof(double) * (size_t)nsweeps * e->cfg.m, cudaMemcpyDeviceToHost));
    return 0;
}

/* one sweep of chain 0 at the current parameters without updating them: its statistics blocks (one per group) into h */
static int chain0_stats(pht_engine *e, std::vector<long long> &h) {
    CU(cudaSetDevice(e->cfg.device));
    UpdateParams u = update_params(e, nullptr, 0);
    u.chains = 1;                                  /* chain 0 only */
    if (enqueue_model(e, u)) return -1;
    SweepParams p = sweep_params(e);
    p.chains = 1;
    if (enqueue_paths(e, p)) return -1;
    if (enqueue_entry(e, u, p)) return -1;
    if (pht_engine_sync(e)) return -1;
    h.resize((size_t)e->groups * stats_len(e->cfg.n));
    CU(cudaMemcpy(h.data(), e->d_stats, sizeof(long long) * h.size(), cudaMemcpyDeviceToHost));
    return 0;
}

/* N, B and the fixed-point totals of statistics blocks [g0, g1) of h, summed */
static int unpack_stats(const pht_engine *e, const long long *h, int blocks, long long *N, long long *B, long long *zfix) {
    const int n = e->cfg.n, len = stats_len(n);
    for (int i = 0; i < n * n; i++) { long long a = 0; for (int g = 0; g < blocks; g++) a += h[(size_t)g * len + i]; if (N) N[i] = a; }
    for (int i = 0; i < n; i++) {
        long long b = 0; __int128 tot = 0;
        for (int g = 0; g < blocks; g++) {
            const long long *q = h + (size_t)g * len;
            b += q[n * n + i];
            tot += ((__int128)q[n * n + 2 * n + i] << 32) + (__int128)(unsigned long long)q[n * n + n + i];
        }
        if (B) B[i] = b;
        if (tot > (__int128)0x7fffffffffffffffLL || tot < -(__int128)0x7fffffffffffffffLL) return fail("sojourn total of state %d overflows the fixed-point range (zbits = %d)", i, e->cfg.zbits);
        if (zfix) zfix[i] = (long long)tot;
    }
    return 0;
}

extern "C" int pht_engine_sweep_stats(pht_engine *e, long long *N, long long *B, long long *zfix) {
    if (!e) return fail("null engine");
    std::vector<long long> h;
    if (chain0_stats(e, h)) return -1;
    return unpack_stats(e, h.data(), e->groups, N, B, zfix);     /* the sum over the groups */
}

extern "C" int pht_engine_emission_stats(pht_engine *e, long long *K) {
    if (!e || !K) return fail("null argument");
    if (!e->stages) return fail("no stage visits are set (pht_engine_set_stage_visits)");
    std::vector<long long> h;
    if (chain0_stats(e, h)) return -1;
    CU(cudaMemcpy(K, e->d_K, sizeof(long long) * (size_t)e->cfg.n * e->stages, cudaMemcpyDeviceToHost));
    return 0;
}

extern "C" int pht_engine_group_stats(pht_engine *e, long long *N, long long *B, long long *zfix) {
    if (!e) return fail("null engine");
    if (method_of(e->cfg) != PHT_METHOD_UNIF) return fail("groups with their own structure need method 64");
    std::vector<long long> h;
    if (chain0_stats(e, h)) return -1;
    const int n = e->cfg.n;
    for (int g = 0; g < e->groups; g++)
        if (unpack_stats(e, h.data() + (size_t)g * stats_len(n), 1, N ? N + (size_t)g * n * n : nullptr, B ? B + (size_t)g * n : nullptr,
                         zfix ? zfix + (size_t)g * n : nullptr)) return -1;
    return 0;
}

/* pht_engine_paths of a grouped engine: one k_unif_paths launch per group with observations in the window, over that
 * group's observations of the window (in upload order) on chain 0's model and table of the group; each path is recorded
 * at its window position */
static int group_paths(pht_engine *e, long first, long count, int *B, int *N, double *z) {
    const int n = e->cfg.n, G = e->groups;
    const size_t tabd = pht_unif_table_doubles(n, PHT_UNIF_CAP);
    std::vector<double> y((size_t)count), u;
    std::vector<uint8_t> c((size_t)count);
    CU(cudaMemcpy(y.data(), e->d_y + first, sizeof(double) * count, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(c.data(), e->d_cens + first, (size_t)count, cudaMemcpyDeviceToHost));
    if (e->d_u) { u.resize((size_t)count); CU(cudaMemcpy(u.data(), e->d_u + first, sizeof(double) * count, cudaMemcpyDeviceToHost)); }
    UpdateParams up = update_params(e, nullptr, 0);
    up.chains = 1;                                 /* chain 0 only: its G models and tables */
    if (enqueue_model(e, up)) return -1;
    double *dy = nullptr, *du = nullptr, *dz = nullptr; uint8_t *dc = nullptr; uint32_t *dperm = nullptr; int *dB = nullptr, *dN = nullptr;
    int rc = -1;
#define CUP(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { fail("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); goto out; } } while (0)
    {
        CUP(cudaMalloc(&dy, sizeof(double) * count)); CUP(cudaMalloc(&dc, (size_t)count)); CUP(cudaMalloc(&dperm, sizeof(uint32_t) * count));
        if (e->d_u) CUP(cudaMalloc(&du, sizeof(double) * count));
        CUP(cudaMalloc(&dB, sizeof(int) * count)); CUP(cudaMalloc(&dN, sizeof(int) * count * n * n)); CUP(cudaMalloc(&dz, sizeof(double) * count * n));
        for (int g = 0; g < G; g++) {
            std::vector<long> pos;
            for (long k = 0; k < count; k++) if (e->h_group[(size_t)(first + k)] == g) pos.push_back(k);
            if (pos.empty()) continue;
            const long cnt = (long)pos.size();
            std::vector<double> yg((size_t)cnt), ug((size_t)cnt); std::vector<uint8_t> cg((size_t)cnt); std::vector<uint32_t> ig((size_t)cnt);
            for (long k = 0; k < cnt; k++) {
                const long w = pos[(size_t)k];
                yg[(size_t)k] = y[(size_t)w]; cg[(size_t)k] = c[(size_t)w]; ig[(size_t)k] = (uint32_t)(first + w);
                if (du) ug[(size_t)k] = u[(size_t)w];
            }
            CUP(cudaMemcpyAsync(dy, yg.data(), sizeof(double) * cnt, cudaMemcpyHostToDevice, e->stream));
            CUP(cudaMemcpyAsync(dc, cg.data(), (size_t)cnt, cudaMemcpyHostToDevice, e->stream));
            CUP(cudaMemcpyAsync(dperm, ig.data(), sizeof(uint32_t) * cnt, cudaMemcpyHostToDevice, e->stream));
            if (du) CUP(cudaMemcpyAsync(du, ug.data(), sizeof(double) * cnt, cudaMemcpyHostToDevice, e->stream));
            CUP(cudaMemsetAsync(dN, 0, sizeof(int) * cnt * n * n, e->stream));
            CUP(cudaMemsetAsync(&e->d_state->next_obs, 0, sizeof(unsigned long long), e->stream));   /* each launch hands out from 0 */
            SweepParams p = sweep_params(e);
            p.chains = 1; p.groups = 1;
            p.model = e->d_model + (size_t)g * e->L.total;
            p.y = dy; p.cens = dc; p.perm = dperm; p.u = du; p.l_local = cnt;
            p.outB = dB; p.outN = dN; p.outz = dz; p.first = 0; p.count = cnt;
            CUP(pht_launch_unif(p, e->d_unif + (size_t)g * tabd, nullptr, e->grid_blocks, e->stream));
            e->launches++;
            if (pht_engine_sync(e)) goto out;
            std::vector<int> hB((size_t)cnt), hN((size_t)cnt * n * n); std::vector<double> hz((size_t)cnt * n);
            CUP(cudaMemcpy(hB.data(), dB, sizeof(int) * cnt, cudaMemcpyDeviceToHost));
            CUP(cudaMemcpy(hN.data(), dN, sizeof(int) * cnt * n * n, cudaMemcpyDeviceToHost));
            CUP(cudaMemcpy(hz.data(), dz, sizeof(double) * cnt * n, cudaMemcpyDeviceToHost));
            for (long k = 0; k < cnt; k++) {
                const long w = pos[(size_t)k];
                B[w] = hB[(size_t)k];
                memcpy(N + (size_t)w * n * n, hN.data() + (size_t)k * n * n, sizeof(int) * n * n);
                memcpy(z + (size_t)w * n, hz.data() + (size_t)k * n, sizeof(double) * n);
            }
        }
        rc = 0;
    }
#undef CUP
out:
    cudaFree(dy); cudaFree(dc); cudaFree(dperm); cudaFree(dB); cudaFree(dN); cudaFree(dz);
    if (du) cudaFree(du);
    return rc;
}

extern "C" int pht_engine_paths(pht_engine *e, long first, long count, int *B, int *N, double *z) {
    if (!e || !B || !N || !z) return fail("null argument");
    if (first < 0 || count < 0 || first + count > e->l_local) return fail("range [%ld, %ld) outside the shard", first, first + count);
    if (e->counts_set) return fail("per-observation paths are not recorded while counts are set: compare with an engine on the expanded data instead");
    if (count == 0) return 0;
    CU(cudaSetDevice(e->cfg.device));
    if (e->groups > 1) {
        if (group_paths(e, first, count, B, N, z)) return -1;
        return e->visits_set ? panel_window(e, first, count, B, N, z) : 0;
    }
    const int n = e->cfg.n;
    int *dB = nullptr, *dN = nullptr; double *dz = nullptr;
    uint32_t *t_exact = nullptr, *t_cens = nullptr;
    /* every exit goes through `out`, which releases the temporaries */
    int rc = -1;
#define CUP(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { fail("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); goto out; } } while (0)
    {
        CUP(cudaMalloc(&dB, sizeof(int) * count)); CUP(cudaMalloc(&dN, sizeof(int) * count * n * n)); CUP(cudaMalloc(&dz, sizeof(double) * count * n));
        CUP(cudaMemsetAsync(dB, 0, sizeof(int) * count, e->stream)); CUP(cudaMemsetAsync(dN, 0, sizeof(int) * count * n * n, e->stream));
        CUP(cudaMemsetAsync(dz, 0, sizeof(double) * count * n, e->stream));
        UpdateParams u = update_params(e, nullptr, 0);
        u.chains = 1;                              /* chain 0 only */
        if (enqueue_model(e, u)) goto out;
        SweepParams p = sweep_params(e);
        p.chains = 1;
        p.y = e->d_y; p.cens = e->d_cens; p.perm = nullptr;         /* the window [first, first + count) is in upload order */
        if (p.u) p.u = e->d_u;
        p.outB = dB; p.outN = dN; p.outz = dz; p.first = first; p.count = count;
        if (method_of(e->cfg) == PHT_METHOD_ECS) {
            std::vector<uint32_t> ie, ic;
            for (long i = first; i < first + count; i++) (e->h_cens[i] ? ic : ie).push_back((uint32_t)i);
            CUP(cudaMalloc(&t_exact, sizeof(uint32_t) * (ie.size() + 1))); CUP(cudaMalloc(&t_cens, sizeof(uint32_t) * (ic.size() + 1)));
            if (!ie.empty()) CUP(cudaMemcpy(t_exact, ie.data(), sizeof(uint32_t) * ie.size(), cudaMemcpyHostToDevice));
            if (!ic.empty()) CUP(cudaMemcpy(t_cens, ic.data(), sizeof(uint32_t) * ic.size(), cudaMemcpyHostToDevice));
            if (enqueue_paths(e, p, t_exact, ie.size(), t_cens, ic.size(), true)) goto out;
        } else if (method_of(e->cfg) == PHT_METHOD_MHS_ASLETT) {
            std::vector<uint32_t> all((size_t)count);
            for (long i = 0; i < count; i++) all[(size_t)i] = (uint32_t)(first + i);
            CUP(cudaMalloc(&t_exact, sizeof(uint32_t) * all.size()));
            CUP(cudaMemcpy(t_exact, all.data(), sizeof(uint32_t) * all.size(), cudaMemcpyHostToDevice));
            if (enqueue_paths(e, p, t_exact, all.size(), nullptr, 0, true)) goto out;
        } else if (enqueue_paths(e, p)) goto out;
        if (pht_engine_sync(e)) goto out;
        CUP(cudaMemcpy(B, dB, sizeof(int) * count, cudaMemcpyDeviceToHost));
        CUP(cudaMemcpy(N, dN, sizeof(int) * count * n * n, cudaMemcpyDeviceToHost));
        CUP(cudaMemcpy(z, dz, sizeof(double) * count * n, cudaMemcpyDeviceToHost));
        rc = 0;
    }
#undef CUP
out:
    cudaFree(dB); cudaFree(dN); cudaFree(dz);
    if (t_exact) cudaFree(t_exact);
    if (t_cens) cudaFree(t_cens);
    if (rc == 0 && e->visits_set) rc = panel_window(e, first, count, B, N, z);
    return rc;
}

extern "C" int pht_engine_set_spectral(pht_engine *e, const double *evals, const double *Q, const double *Qinv) {
    if (!e) return fail("null engine");
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    const int n = e->cfg.n;
    if (method_of(e->cfg) == PHT_METHOD_UNIF && evals && Q && Qinv)
        return fail("method 64 uses no spectral data (it samples through the uniformised chain)");
    if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }     /* the sweep changes shape */
    if (!evals || !Q || !Qinv) {
        if (e->d_inject) { CU(cudaFree(e->d_inject)); e->d_inject = nullptr; }
        return 0;
    }
    if (!e->d_inject) CU(cudaMalloc(&e->d_inject, sizeof(double) * (n + 2 * n * n)));
    CU(cudaMemcpy(e->d_inject, evals, sizeof(double) * n, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(e->d_inject + n, Q, sizeof(double) * n * n, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(e->d_inject + n + n * n, Qinv, sizeof(double) * n * n, cudaMemcpyHostToDevice));
    return 0;
}

extern "C" int pht_engine_get_model(pht_engine *e, double *S, double *s, double *P, double *Pfull,
                                    double *evals, double *Q, double *Qinv) {
    if (!e) return fail("null engine");
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    const int n = e->cfg.n;
    std::vector<double> h(e->L.total);
    CU(cudaMemcpy(h.data(), e->d_model, sizeof(double) * h.size(), cudaMemcpyDeviceToHost));
    if (S) memcpy(S, &h[e->L.S], sizeof(double) * n * n);
    if (s) memcpy(s, &h[e->L.s], sizeof(double) * n);
    if (P) memcpy(P, &h[e->L.P], sizeof(double) * n * n);
    if (Pfull) memcpy(Pfull, &h[e->L.Pfull], sizeof(double) * n * (n + 1));
    if (evals) memcpy(evals, &h[e->L.evals], sizeof(double) * n);
    if (Q) memcpy(Q, &h[e->L.Q], sizeof(double) * n * n);
    if (Qinv) memcpy(Qinv, &h[e->L.Qinv], sizeof(double) * n * n);
    return 0;
}

extern "C" int pht_engine_round_trace(pht_engine *e, unsigned long long *out) {
    if (!e || !out) return fail("null argument");
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    DevState *st = new DevState; cudaError_t ce = cudaMemcpy(st, e->d_state, sizeof(*st), cudaMemcpyDeviceToHost);
    if (ce == cudaSuccess) memcpy(out, st->round_trace, sizeof(st->round_trace));
    delete st;
    CU(ce);
    return 0;
}

extern "C" int pht_engine_counters(pht_engine *e, unsigned long long *out) {
    if (!e || !out) return fail("null argument");
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->stream));
    DevState st; CU(cudaMemcpy(&st, e->d_state, sizeof(st), cudaMemcpyDeviceToHost));
    memcpy(out, st.counters, sizeof(st.counters));
    out[PHT_CNT_LAUNCHES] = e->launches;
    return 0;
}
