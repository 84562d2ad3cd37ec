// api.cu -- C-ABI (include/rri_b200.h) and sweep orchestration of the B200-native RRI engine.
#include <dlfcn.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/rri_b200.h"
#include "gemm_tf32_sm100.h"
#include "common.cuh"
#include "devmem.h"
#include "kernels.h"
#include "wrri_tc_sm100.h"

using namespace rri;

// -------------------------------------------------------------------------------------------------
// errors
// -------------------------------------------------------------------------------------------------
static thread_local char g_err[1024] = "";
static int fail(const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return 1;
}
#define CK(call)                                                                                \
    do {                                                                                        \
        cudaError_t e_ = (call);                                                                \
        if (e_ != cudaSuccess)                                                                  \
            return fail("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)
#define CKL() CK(cudaGetLastError())

extern "C" const char* rri_last_error(void) { return g_err; }
extern "C" const char* rri_version(void) { return "rri_b200 0.1 (sm_100a; tcgen05 tf32 + simt f32/f64)"; }

// -------------------------------------------------------------------------------------------------
// NCCL through dlsym (no link-time dependency: the library must load on a CPU-only host)
// -------------------------------------------------------------------------------------------------
struct Id128 { char b[128]; };
struct NcclApi {
    void* lib = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    int (*GetUniqueId)(void*) = nullptr;
    int (*CommInitRank)(void**, int, /* ncclUniqueId by value: 128 bytes */ Id128, int) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
static NcclApi g_nccl;

static int nccl_load(const char* path)
{
    if (g_nccl.lib) return 0;
    void* lib = nullptr;
    if (path && *path) lib = dlopen(path, RTLD_NOW | RTLD_GLOBAL);
    if (!lib) lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) return fail("cannot load NCCL (%s): %s", path ? path : "libnccl.so.2", dlerror());
    g_nccl.AllReduce = (decltype(g_nccl.AllReduce))dlsym(lib, "ncclAllReduce");
    g_nccl.GetUniqueId = (decltype(g_nccl.GetUniqueId))dlsym(lib, "ncclGetUniqueId");
    g_nccl.CommInitRank = (decltype(g_nccl.CommInitRank))dlsym(lib, "ncclCommInitRank");
    g_nccl.CommDestroy = (decltype(g_nccl.CommDestroy))dlsym(lib, "ncclCommDestroy");
    g_nccl.GetErrorString = (decltype(g_nccl.GetErrorString))dlsym(lib, "ncclGetErrorString");
    if (!g_nccl.AllReduce || !g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.CommDestroy)
        return fail("NCCL symbols missing in %s", path ? path : "libnccl.so.2");
    g_nccl.lib = lib;
    return 0;
}
#define NCK(call)                                                                                \
    do {                                                                                         \
        int r_ = (call);                                                                         \
        if (r_ != 0)                                                                             \
            return fail("%s failed: %s", #call, g_nccl.GetErrorString ? g_nccl.GetErrorString(r_) : "?"); \
    } while (0)

extern "C" int rri_nccl_unique_id(char id_out[128], const char* nccl_lib_path)
{
    if (nccl_load(nccl_lib_path)) return 1;
    NCK(g_nccl.GetUniqueId(id_out));
    return 0;
}
extern "C" int rri_nccl_comm_create(void** comm_out, const char id[128], int32_t rank, int32_t world,
                                    int32_t device, const char* nccl_lib_path)
{
    if (nccl_load(nccl_lib_path)) return 1;
    CK(cudaSetDevice(device));
    Id128 u;
    memcpy(u.b, id, 128);
    NCK(g_nccl.CommInitRank(comm_out, world, u, rank));
    return 0;
}
extern "C" int rri_nccl_comm_destroy(void* comm)
{
    if (!g_nccl.lib) return fail("NCCL not loaded");
    NCK(g_nccl.CommDestroy(comm));
    return 0;
}

// -------------------------------------------------------------------------------------------------
// handle
// -------------------------------------------------------------------------------------------------
// Exchange buffers and their peer mappings outlive the handle: cudaMalloc + CUDA-IPC export / open of a fresh buffer
// cost ~0.2 s per engine (longer than 40 sweeps of the headline configuration at two GPUs), and every nmf() call
// creates a new engine.  A destroyed handle parks its buffer here; the next handle of the same geometry on the same
// device takes it over, and when all ranks present the same IPC handles again the mappings are reused as they are
// (the epoch counter continues, so stale flags can never satisfy a wait).  Entries are only released by
// rri_cache_trim -- to be called on all ranks together -- so no rank ever frees a buffer a peer still has mapped.
struct PeerGroup {
    bool used = false;
    int device = -1, world = 0, rank = 0;
    void* xbuf = nullptr; size_t bytes = 0;
    void* peer_base[16] = {nullptr}; bool peer_open[16] = {false};
    char handles[16 * 64] = {0};
    bool mapped = false;
    unsigned epoch = 0;
};


struct rri_handle_s {
    int64_t n = 0, d = 0;
    int k = 0, dtype = 0, math = 0, order = 0, device = 0, sm_count = 148;
    size_t es = 4;
    // data
    const void* X = nullptr; int64_t ldx = 0;
    const void* M = nullptr; int mk = 0; int64_t ldm = 0;
    // comm
    void* comm = nullptr; int rank = 0, world = 1;
    // peer-memory exchange of the T half-step (multi-GPU hals): every rank exports one buffer
    //   [2 epochs][d*k + k*k] partial statistic | T' replica [d,k] | T replica [k,ldtk] | slice sums [16][k] | flags
    // and all ranks map all buffers (CUDA IPC); see hals_kernels.cu: peer_update_rows_kernel
    void* xbuf = nullptr; size_t xbuf_bytes = 0, xslot_elems = 0;
    size_t x_off_tt = 0, x_off_tk = 0, x_off_tsum = 0, x_off_flags = 0;
    int64_t ldtk = 0;
    void* peer_base[16] = {nullptr}; bool peer_open[16] = {false};
    void* Tt_own = nullptr;            // the handle's private T' (used again when the exchange is switched off)
    unsigned epoch = 0;
    bool p2p = false, peer_mapped = false;
    int* p2p_err = nullptr;
    char handles[16 * 64] = {0};       // the IPC handles the current mappings were opened from
    PeerGroup parked; bool have_parked = false;     // parked group taken over by rri_peer_export
    unsigned* counters = nullptr;      // [8] arrival counters of the "last block finalises" kernels (zero between launches)
    // workspace
    std::vector<void*> allocs;
    int64_t ws_bytes = 0, launches = 0;
    // rri order
    PassPlan pp{};
    int hb = 0, gbw = 0;
    void *ypart = nullptr, *ppart = nullptr, *gpart = nullptr, *hpart = nullptr, *stat = nullptr;
    // hals order
    void *Xt = nullptr; int64_t ldxt = 0, ldwt = 0;
    void* Xt_ext = nullptr; int64_t ldxt_ext = 0;      // caller-provided storage for the transposed copy (optional)
    void *Wt = nullptr, *Tt = nullptr, *Cpart = nullptr, *cg = nullptr /* [max(n,d)*k | k*k] */, *Hm = nullptr;
    void *gram_part = nullptr, *colsum_part = nullptr;
    int splits_t = 1, splits_w = 1, ub_blocks_t = 1, ub_blocks_w = 1, gchunks_w = 1, gchunks_t = 1;
    double* sx_slots = nullptr;        // grid-reduction scratch of the constrained T update (simplex_T)
    Tf32Gemm* tf32 = nullptr;
    bool fixT_cached = false;
    // masked
    TilePlan tpl{}, wpl{};
    void *numer_part = nullptr, *denom_part = nullptr, *mstat = nullptr;
    WrriTc* wtc = nullptr; int wtc_groups_t = 1, wtc_groups_w = 1;
    // observed-entries (sparse) binding: CSR given by the caller, CSC built by rri_bind_csr
    bool sparse = false; int64_t nnz = 0;
    SpSide csr{}, csc{};
    void *sp_quad = nullptr;           // [max(n,d)] packed gather records of one pass
    void *sp_told = nullptr;           // [2][d] T[t,:] before its T-step (two topics in flight)
    void *sp_wold = nullptr;           // [2][n] W[:,t] before its W-step
    void *sp_npart = nullptr, *sp_dpart = nullptr;     // per-block partial sums of a pass: [nblk][nseg] each
    uint32_t* sp_perm = nullptr;       // [nnz] CSR position of every CSC entry
    int sp_ldt = 0;                    // row stride of T' [d, sp_ldt] (k rounded up to 16 bytes: vector gathers)
    bool sp_refresh_v2 = true;         // residual restart: row copy from the factors, column copy gathered from it
    bool sp_batched_sums = true;       // per-topic sums once per sweep (2 launches) instead of once per half-step (2k)
    int* sp_err = nullptr;
    // zero-filled sparse binding (rri_bind_csr_zero): the rows and the columns with their chunk plans; the block-order
    // half-steps take X T' / X' W from launch_spmm instead of the dense contraction
    bool zero_csr = false;
    SpmmPlan zrow{}, zcol{};
    // common
    double* sums = nullptr;    // [2k] device
    int* flags = nullptr;      // device
    double *obj_part = nullptr, *obj_out = nullptr;
    int oblocks = 1;
    // objective through the contraction: ||X||^2 is computed once per binding; c2_valid = Cpart still holds X T' of
    // the current T (and Tt its transpose): true right after a block-order sweep
    bool xsq_valid = false, c2_valid = false;
    void* Gobj = nullptr;
};

static int ws_alloc(rri_handle_t h, void** p, size_t bytes)
{
    if (bytes == 0) bytes = 16;
    CK(cached_malloc(p, bytes));
    CK(cudaMemsetAsync(*p, 0, bytes, 0));          // blocks come back from the cache with old contents
    h->allocs.push_back(*p);
    h->ws_bytes += (int64_t)bytes;
    return 0;
}

extern "C" int rri_create(rri_handle_t* out, int64_t n_local, int64_t d, int32_t k, int32_t dtype,
                          int32_t math, int32_t order, int32_t device)
{
    if (!out) return fail("null handle pointer");
    if (n_local <= 0 || d <= 0) return fail("n_local and d must be positive (got %lld, %lld)", (long long)n_local, (long long)d);
    if (k <= 0 || k > 256) return fail("k must be in [1,256] (got %d)", k);
    if (dtype != RRI_F32 && dtype != RRI_F64) return fail("bad dtype %d", dtype);
    if (order != RRI_ORDER_RRI && order != RRI_ORDER_HALS) return fail("bad order %d", order);
    if (math != RRI_MATH_IEEE && math != RRI_MATH_TF32) return fail("bad math %d", math);
    if (math == RRI_MATH_TF32 && dtype != RRI_F32) return fail("TF32 math needs f32 data");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail("no CUDA device available (%s); this library has no CPU fallback", cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail("bad device %d", device);
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail("device %d is sm_%d%d; this build contains sm_100a code only", device, prop.major, prop.minor);
    rri_handle_t h = new rri_handle_s();
    h->n = n_local; h->d = d; h->k = k; h->dtype = dtype; h->math = math; h->order = order;
    h->device = device; h->sm_count = prop.multiProcessorCount;
    h->es = dtype == RRI_F32 ? 4 : 8;
    if (ws_alloc(h, (void**)&h->sums, sizeof(double) * 2 * k) || ws_alloc(h, (void**)&h->flags, sizeof(int) * 4) ||
        ws_alloc(h, (void**)&h->counters, sizeof(unsigned) * 8)) {
        rri_destroy(h);
        return 1;
    }
    cudaStreamSynchronize(0);
    *out = h;
    return 0;
}

static void peer_release(rri_handle_t h);

extern "C" int rri_destroy(rri_handle_t h)
{
    if (!h) return 0;
    cudaSetDevice(h->device);
    // Workspace blocks are parked for the next handle, which zero-fills them on the legacy default stream: nothing of
    // this handle may still be in flight on a (possibly non-blocking) caller stream when they are handed out again.
    cudaDeviceSynchronize();
    peer_release(h);
    for (void* p : h->allocs) cached_free(p);
    if (h->tf32) tf32_gemm_destroy(h->tf32);
    if (h->wtc) wrri_tc_destroy(h->wtc);
    delete h;
    return 0;
}

extern "C" int rri_set_comm(rri_handle_t h, void* nccl_comm, int32_t rank, int32_t world, const char* nccl_lib_path)
{
    if (!h) return fail("null handle");
    if (world > 1) {
        if (!nccl_comm) return fail("world > 1 needs a communicator");
        if (nccl_load(nccl_lib_path)) return 1;
    }
    h->comm = nccl_comm; h->rank = rank; h->world = world;
    return 0;
}

// -------------------------------------------------------------------------------------------------
// peer-memory exchange (the NCCL all-reduce of the block-order T half-step replaced by NVLink loads / stores inside
// the update kernel: hals_kernels.cu peer_update_rows_kernel)
// -------------------------------------------------------------------------------------------------
static size_t round_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

static PeerGroup g_groups[64];

static PeerGroup* group_take(int device, size_t bytes)
{
    for (PeerGroup& g : g_groups)
        if (g.used && g.device == device && g.bytes == bytes) { g.used = false; return &g; }
    return nullptr;
}
static PeerGroup* group_slot()
{
    for (PeerGroup& g : g_groups) if (!g.used) return &g;
    return nullptr;
}

static bool peer_rank_supported(rri_handle_t h)
{
    return h->dtype == RRI_F32 ? h->k <= 128 : h->k <= 64;      // the thread-per-row update kernel
}

extern "C" int rri_peer_export(rri_handle_t h, char handle_out[64])
{
    if (!h) return fail("null handle");
    if (!h->X) return fail("rri_bind has not been called");
    if (h->order != RRI_ORDER_HALS || h->mk != MK_NONE) return fail("the peer-memory exchange serves unmasked hals handles");
    if (h->zero_csr) return fail("the peer-memory exchange serves dense data; zero-filled sparse handles use the NCCL all-reduce");
    if (!peer_rank_supported(h)) return fail("the fused peer-memory T update supports k <= 128 (f32) / 64 (f64)");
    CK(cudaSetDevice(h->device));
    if (!h->xbuf) {
        const size_t es = h->es;
        const int64_t v = 16 / (int64_t)es;
        h->ldtk = (h->d + v - 1) / v * v;
        h->xslot_elems = ((size_t)h->d * h->k + (size_t)h->k * h->k + 63) / 64 * 64;
        h->x_off_tt = round_up(2 * h->xslot_elems * es, 256);
        h->x_off_tk = round_up(h->x_off_tt + (size_t)h->d * h->k * es, 256);
        h->x_off_tsum = round_up(h->x_off_tk + (size_t)h->k * h->ldtk * es, 256);
        h->x_off_flags = round_up(h->x_off_tsum + (size_t)16 * h->k * es, 256);
        h->xbuf_bytes = h->x_off_flags + 2 * 16 * 32 * sizeof(unsigned);
        if (PeerGroup* g = group_take(h->device, h->xbuf_bytes)) {
            // a parked buffer of the same geometry: same IPC handle as before, mappings kept for rri_peer_import
            h->xbuf = g->xbuf;
            h->parked = *g;
            h->have_parked = true;
            *g = PeerGroup();
        } else {
            CK(cudaMalloc(&h->xbuf, h->xbuf_bytes));
            CK(cudaMemset(h->xbuf, 0, h->xbuf_bytes));
            CK(cudaDeviceSynchronize());
        }
    }
    cudaIpcMemHandle_t mh;
    CK(cudaIpcGetMemHandle(&mh, h->xbuf));
    static_assert(sizeof(mh) == 64, "cudaIpcMemHandle_t is 64 bytes");
    memcpy(handle_out, &mh, 64);
    return 0;
}

extern "C" int rri_peer_import(rri_handle_t h, const char* handles, int32_t rank, int32_t world)
{
    if (!h) return fail("null handle");
    if (!h->xbuf) return fail("rri_peer_export must be called first");
    if (world < 2 || world > 16 || rank < 0 || rank >= world) return fail("bad rank/world %d/%d", rank, world);
    CK(cudaSetDevice(h->device));
    if (h->have_parked) {
        PeerGroup& g = h->parked;
        h->have_parked = false;
        if (g.mapped && g.world == world && g.rank == rank && memcmp(g.handles, handles, (size_t)64 * world) == 0) {
            // every rank came back with the buffer it had: nothing to map, the flags continue from the old epoch
            for (int r = 0; r < 16; ++r) { h->peer_base[r] = g.peer_base[r]; h->peer_open[r] = g.peer_open[r]; }
            memcpy(h->handles, handles, (size_t)64 * world);
            if (!h->p2p_err && ws_alloc(h, (void**)&h->p2p_err, sizeof(int))) return 1;
            CK(cudaStreamSynchronize(0));
            h->rank = rank; h->world = world; h->epoch = g.epoch; h->p2p = false; h->peer_mapped = true;
            return 0;
        }
        // some rank has a new buffer: drop the old mappings, restart the flags of this one
        for (int r = 0; r < 16; ++r)
            if (g.peer_open[r] && g.peer_base[r]) cudaIpcCloseMemHandle(g.peer_base[r]);
        CK(cudaMemset((char*)h->xbuf + h->x_off_flags, 0, 2 * 16 * 32 * sizeof(unsigned)));
        CK(cudaDeviceSynchronize());
    }
    memcpy(h->handles, handles, (size_t)64 * world);
    for (int r = 0; r < world; ++r) {
        if (r == rank) { h->peer_base[r] = h->xbuf; continue; }
        cudaIpcMemHandle_t mh;
        memcpy(&mh, handles + 64 * r, 64);
        void* p = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&p, mh, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail("cudaIpcOpenMemHandle for rank %d failed: %s", r, cudaGetErrorString(e));
        }
        h->peer_base[r] = p; h->peer_open[r] = true;
    }
    if (!h->p2p_err && ws_alloc(h, (void**)&h->p2p_err, sizeof(int))) return 1;
    CK(cudaStreamSynchronize(0));
    h->rank = rank; h->world = world; h->epoch = 0; h->p2p = false;     // enabled by rri_peer_enable on ALL ranks
    h->peer_mapped = true;
    return 0;
}

// parks the exchange buffer and its mappings for the next handle (or really releases them when the table is full)
static void peer_release(rri_handle_t h)
{
    if (!h->xbuf) return;
    if (h->have_parked) {                       // exported from a parked group but never imported: put it back
        if (PeerGroup* g = group_slot()) { *g = h->parked; g->used = true; h->xbuf = nullptr; h->have_parked = false; return; }
    }
    PeerGroup* g = group_slot();
    if (g) {
        g->used = true; g->device = h->device; g->world = h->world; g->rank = h->rank;
        g->xbuf = h->xbuf; g->bytes = h->xbuf_bytes; g->mapped = h->peer_mapped; g->epoch = h->epoch;
        for (int r = 0; r < 16; ++r) { g->peer_base[r] = h->peer_base[r]; g->peer_open[r] = h->peer_open[r]; }
        memcpy(g->handles, h->handles, sizeof(g->handles));
    } else {
        for (int r = 0; r < 16; ++r)
            if (h->peer_open[r] && h->peer_base[r]) cudaIpcCloseMemHandle(h->peer_base[r]);
        cudaFree(h->xbuf);
    }
    h->xbuf = nullptr; h->peer_mapped = false;
    for (int r = 0; r < 16; ++r) { h->peer_open[r] = false; h->peer_base[r] = nullptr; }
}

extern "C" int rri_peer_close(rri_handle_t h)
{
    if (!h) return fail("null handle");
    CK(cudaSetDevice(h->device));
    h->p2p = false;
    if (h->Tt_own) { h->Tt = h->Tt_own; h->Tt_own = nullptr; }
    peer_release(h);
    return 0;
}

extern "C" int rri_peer_enable(rri_handle_t h, int32_t on)
{
    if (!h) return fail("null handle");
    if (on && !h->peer_mapped) return fail("rri_peer_import has not succeeded on this rank");
    h->p2p = on != 0;
    // with the exchange on, the T' copy of this handle IS its replica inside the exchange buffer (the peers write
    // the rows they own straight into it)
    if (h->p2p) {
        if (!h->Tt_own) h->Tt_own = h->Tt;
        h->Tt = (char*)h->xbuf + h->x_off_tt;
    } else if (h->Tt_own) {
        h->Tt = h->Tt_own; h->Tt_own = nullptr;
    }
    return 0;
}

// rows of T' (columns of T) that rank r updates in the fused exchange: 128-row blocks dealt out evenly
static void peer_row_range(int64_t d, int world, int r, int64_t& lo, int64_t& hi)
{
    const int64_t nb = (d + 127) / 128;
    const int64_t q = nb / world, rem = nb % world;
    const int64_t b0 = q * r + (r < rem ? r : rem), b1 = b0 + q + (r < rem ? 1 : 0);
    lo = b0 * 128 < d ? b0 * 128 : d;
    hi = b1 * 128 < d ? b1 * 128 : d;
}

static PeerExchange peer_args(rri_handle_t h, unsigned epoch)
{
    PeerExchange px;
    memset(&px, 0, sizeof(px));
    px.world = h->world; px.rank = h->rank; px.epoch = epoch; px.ldtk = h->ldtk; px.err = h->p2p_err;
    peer_row_range(h->d, h->world, h->rank, px.row_lo, px.row_hi);
    const int b = (int)(epoch & 1u);
    for (int r = 0; r < h->world; ++r) {
        char* base = (char*)h->peer_base[r];
        px.part[r] = base + (size_t)b * h->xslot_elems * h->es;
        px.Tt[r] = base + h->x_off_tt;
        px.Tk[r] = base + h->x_off_tk;
        px.tsum[r] = base + h->x_off_tsum;
        px.flag1[r] = (unsigned*)(base + h->x_off_flags);
        px.flag2[r] = (unsigned*)(base + h->x_off_flags) + 16 * 32;
    }
    return px;
}

static int allreduce(rri_handle_t h, void* buf, size_t count, cudaStream_t st)
{
    if (h->world <= 1) return 0;
    NCK(g_nccl.AllReduce(buf, buf, count, h->dtype == RRI_F32 ? 7 : 8, /*ncclSum*/ 0, h->comm, st));
    h->launches++;
    return 0;
}

// Workspace of the block-order half-steps downstream of the contraction (and of the contraction's output): both the
// dense binding and the zero-filled sparse one.  splits_w / splits_t (K-slices of the two contractions) are set first.
static int alloc_halfstep_ws(rri_handle_t h)
{
    const int64_t n = h->n, d = h->d;
    const int k = h->k;
    const size_t es = h->es;
    const size_t a = (size_t)h->splits_w * n * k, b = (size_t)h->splits_t * d * k;
    if (ws_alloc(h, &h->Cpart, es * (a > b ? a : b))) return 1;
    const int64_t m = n > d ? n : d;
    if (ws_alloc(h, &h->cg, es * ((size_t)m * k + (size_t)k * k))) return 1;
    if (ws_alloc(h, &h->Hm, es * (size_t)k * k)) return 1;
    {   // rows of W' are TMA operands in tf32 mode: keep them 16-byte aligned
        const int64_t v = 16 / (int64_t)es;
        h->ldwt = (n + v - 1) / v * v;
    }
    if (ws_alloc(h, &h->Wt, es * (size_t)k * h->ldwt) || ws_alloc(h, &h->Tt, es * (size_t)d * k)) return 1;
    h->gchunks_w = gram_chunks(n, k, h->sm_count);
    h->gchunks_t = gram_chunks(d, k, h->sm_count);
    const int gc = h->gchunks_w > h->gchunks_t ? h->gchunks_w : h->gchunks_t;
    if (ws_alloc(h, &h->gram_part, es * (size_t)gc * k * k)) return 1;
    h->ub_blocks_w = update_rows_blocks(n, h->sm_count);
    h->ub_blocks_t = update_rows_blocks(d, h->sm_count);
    int ubm = h->ub_blocks_w > h->ub_blocks_t ? h->ub_blocks_w : h->ub_blocks_t;
    {   // the multi-GPU T update works in 32-row blocks (peer_update_blocks)
        const int pb = peer_update_blocks(d, h->sm_count);
        if (pb > ubm) ubm = pb;
    }
    if (ws_alloc(h, &h->colsum_part, es * (size_t)ubm * k)) return 1;
    if (h->order == RRI_ORDER_HALS && ws_alloc(h, (void**)&h->sx_slots, sizeof(double) * (size_t)simplex_T_slots(d))) return 1;
    return 0;
}

template <typename T>
static int bind_impl(rri_handle_t h, cudaStream_t st)
{
    const int64_t n = h->n, d = h->d;
    const int k = h->k, ks = k + 1;
    const size_t es = sizeof(T);
    h->oblocks = obj_blocks(n, d, h->sm_count);
    if (!h->obj_part) {
        size_t op = 2 * (size_t)(h->oblocks > 256 ? h->oblocks : 256);
        if (op < (size_t)8 * h->sm_count) op = (size_t)8 * h->sm_count;
        if (ws_alloc(h, (void**)&h->obj_part, sizeof(double) * op)) return 1;
        if (ws_alloc(h, (void**)&h->obj_out, sizeof(double) * 16)) return 1;
    }
    if (h->mk != MK_NONE) {
        if (!h->numer_part) {
            h->tpl = plan_tstats(n, d, h->sm_count);
            h->wpl = plan_wstats(n, d, h->sm_count);
            size_t a = (size_t)h->tpl.groups * d, b = (size_t)h->wpl.groups * n;
            if (h->math == RRI_MATH_TF32) {
                // fp32 data: the W T product of every tile goes through the tensor cores
                std::string err;
                h->wtc = wrri_tc_create(h->sm_count, n, d, k, err);
                if (!h->wtc) return fail("tensor-core WRRI path unavailable: %s", err.c_str());
                h->wtc_groups_t = wrri_tc_groups(h->wtc, 0);
                h->wtc_groups_w = wrri_tc_groups(h->wtc, 1);
                const size_t a2 = (size_t)h->wtc_groups_t * d, b2 = (size_t)h->wtc_groups_w * n;
                if (a2 > a) a = a2;
                if (b2 > b) b = b2;
            }
            const size_t m = a > b ? a : b;
            if (ws_alloc(h, &h->numer_part, es * m) || ws_alloc(h, &h->denom_part, es * m)) return 1;
            if (ws_alloc(h, &h->mstat, es * 2 * (size_t)d)) return 1;
        }
        return 0;
    }
    // the W-only half-step (fix_T, i.e. transform()) always goes through the contraction path
    if (!h->Cpart) {
        h->splits_w = simt_gemm_splits(n, d, h->sm_count);
        h->splits_t = simt_gemm_splits(d, n, h->sm_count);
        if (h->math == RRI_MATH_TF32) { h->splits_w = 1; h->splits_t = 1; }
        if (alloc_halfstep_ws(h)) return 1;
        if (h->math == RRI_MATH_TF32) {
            std::string err;
            // (k + 16: the device-resident NNDSVD runs its randomized SVD with k + 10 columns through this kernel)
            h->tf32 = tf32_gemm_create(h->sm_count, k + 16 < 256 ? k + 16 : 256, err);
            if (!h->tf32) return fail("tf32 contraction unavailable: %s", err.c_str());
        }
    }
    if (h->order == RRI_ORDER_HALS) {
        // transposed copy of the data for the T half-step (X' W): both contractions then read
        // K-contiguous operands
        const int64_t v = 16 / (int64_t)es;
        h->ldxt = (n + v - 1) / v * v;
        if (h->Xt_ext) {
            if (h->ldxt_ext < h->ldxt || h->ldxt_ext % v != 0 || (reinterpret_cast<uintptr_t>(h->Xt_ext) & 15) != 0)
                return fail("caller-provided X' storage needs a 16-byte aligned base and a row stride >= %lld, multiple of %lld",
                            (long long)h->ldxt, (long long)v);
            h->Xt = h->Xt_ext; h->ldxt = h->ldxt_ext;
        } else if (!h->Xt) {
            CK(cached_malloc(&h->Xt, es * (size_t)d * h->ldxt));    // (no memset: fully overwritten by the transpose)
            h->allocs.push_back(h->Xt);
            h->ws_bytes += (int64_t)(es * (size_t)d * h->ldxt);
        }
        launch_transpose<T>((const T*)h->X, n, d, h->ldx, (T*)h->Xt, h->ldxt, st);
        h->launches++;
        CKL();
    } else {
        h->pp = plan_pass(n, d, h->ldx, h->X, (int)es, h->sm_count);
        h->hb = tstep_blocks(d);
        h->gbw = wstep_blocks(n, h->sm_count);
        if (!h->ypart) {
            if (ws_alloc(h, &h->ypart, es * (size_t)h->pp.ct * n)) return 1;
            if (ws_alloc(h, &h->ppart, es * (size_t)h->pp.rg * d)) return 1;
            if (ws_alloc(h, &h->gpart, es * (size_t)h->gbw * ks)) return 1;
            if (ws_alloc(h, &h->hpart, es * (size_t)h->hb * ks)) return 1;
            if (ws_alloc(h, &h->stat, es * (size_t)(d + ks))) return 1;
        }
    }
    return 0;
}

extern "C" int rri_set_transpose_storage(rri_handle_t h, void* Xt_dev, int64_t ldXt)
{
    if (!h) return fail("null handle");
    if (h->X) return fail("rri_set_transpose_storage must be called before rri_bind");
    h->Xt_ext = Xt_dev; h->ldxt_ext = ldXt;
    return 0;
}

extern "C" int rri_bind(rri_handle_t h, const void* X_dev, int64_t ldX, const void* mask_dev,
                        int32_t mask_kind, int64_t ldM, void* stream)
{
    if (!h) return fail("null handle");
    if (!X_dev) return fail("X is null");
    if (ldX < h->d) return fail("ldX (%lld) < d (%lld)", (long long)ldX, (long long)h->d);
    if (mask_kind != RRI_MASK_NONE && !mask_dev) return fail("mask kind %d without a mask pointer", mask_kind);
    if (mask_kind != RRI_MASK_NONE && ldM < h->d) return fail("ldM < d");
    if (mask_kind < 0 || mask_kind > 2) return fail("bad mask kind %d", mask_kind);
    if (h->sparse) return fail("this handle is bound to observed-entries (CSR) data; create a new one for dense data");
    if (h->zero_csr) return fail("this handle is bound to zero-filled sparse (CSR) data; create a new one for dense data");
    if (h->X && ((h->mk != MK_NONE) != (mask_kind != RRI_MASK_NONE)))
        return fail("a handle cannot switch between masked and unmasked data; create a new one");
    CK(cudaSetDevice(h->device));
    h->X = X_dev; h->ldx = ldX;
    h->M = mask_kind == RRI_MASK_NONE ? nullptr : mask_dev;
    h->mk = mask_kind; h->ldm = ldM;
    h->fixT_cached = false;
    h->xsq_valid = false; h->c2_valid = false;
    cudaStream_t st = (cudaStream_t)stream;
    int rc = h->dtype == RRI_F32 ? bind_impl<float>(h, st) : bind_impl<double>(h, st);
    if (rc) return rc;
    // workspace zero-fills were issued on the legacy default stream: finish them before the caller's (possibly
    // non-blocking) stream starts using the buffers
    CK(cudaStreamSynchronize(0));
    return 0;
}

// -------------------------------------------------------------------------------------------------
// observed-entries (sparse) binding
// -------------------------------------------------------------------------------------------------
template <typename T>
static int bind_csr_impl(rri_handle_t h, const int64_t* rowptr, const int32_t* col, const T* val, const T* wgt,
                         cudaStream_t st)
{
    const int64_t n = h->n, d = h->d, nnz = h->nnz;
    const int k = h->k;
    const size_t es = sizeof(T);
    const int64_t m = n > d ? n : d;
    const size_t ne = (size_t)(nnz > 0 ? nnz : 1);
    void *E_csr = nullptr, *E_csc = nullptr, *x_csc = nullptr, *w_csc = nullptr, *csc_row = nullptr, *colptr = nullptr;
    if (ws_alloc(h, (void**)&h->obj_part, sizeof(double) * 2 * 256) || ws_alloc(h, (void**)&h->obj_out, sizeof(double) * 8)) return 1;
    if (ws_alloc(h, &E_csr, es * ne) || ws_alloc(h, &E_csc, es * ne) || ws_alloc(h, &x_csc, es * ne)) return 1;
    if (wgt && ws_alloc(h, &w_csc, es * ne)) return 1;
    if (ws_alloc(h, &csc_row, sizeof(int32_t) * ne) || ws_alloc(h, &colptr, sizeof(int64_t) * (size_t)(d + 1))) return 1;
    if (ws_alloc(h, &h->sp_quad, 4 * es * (size_t)m) || ws_alloc(h, &h->sp_told, es * 2 * (size_t)d) ||
        ws_alloc(h, &h->sp_wold, es * 2 * (size_t)n) || ws_alloc(h, &h->mstat, es * 2 * (size_t)m) ||
        ws_alloc(h, (void**)&h->sp_err, sizeof(int)))
        return 1;
    {
        const int64_t v = 16 / (int64_t)es;
        h->ldwt = (n + v - 1) / v * v;
    }
    {
        const char* env = getenv("RRI_SP_REFRESH_V2");
        h->sp_refresh_v2 = !(env && *env == '0');
        const char* envb = getenv("RRI_SP_BATCHED_SUMS");
        h->sp_batched_sums = !(envb && *envb == '0');        // measured: 30.8 -> 29.8 ms per config-4 sweep
        const int v = 16 / (int)es;
        h->sp_ldt = h->sp_refresh_v2 ? (k + v - 1) / v * v : k;
    }
    if (ws_alloc(h, &h->Wt, es * (size_t)k * h->ldwt) || ws_alloc(h, &h->Tt, es * (size_t)d * h->sp_ldt)) return 1;
    if (ws_alloc(h, (void**)&h->sp_perm, sizeof(uint32_t) * ne)) return 1;
    CK(cudaStreamSynchronize(0));          // the zero-fills above ran on the legacy default stream
    const int rc = sp_build_csc<T>(rowptr, col, val, wgt, n, d, nnz, (int64_t*)colptr, (int32_t*)csc_row, (T*)x_csc,
                                   (T*)w_csc, h->sp_perm, h->sm_count, h->sp_err, st);
    if (rc < 0)
        return fail("malformed CSR input:%s%s%s", (-rc & 1) ? " rowptr is not a monotone [0..nnz] sequence;" : "",
                    (-rc & 2) ? " column index outside [0,d);" : "",
                    (-rc & 4) ? " column indices must be strictly ascending inside every row (sort and merge duplicates);" : "");
    if (rc > 0) return fail("building the column orientation failed: %s", cudaGetErrorString((cudaError_t)rc));
    h->csr = SpSide{n, rowptr, col, val, wgt, E_csr, nnz / n >= 512 ? 256 : 32, nullptr, 1, 0, d, nullptr};
    h->csc = SpSide{d, (const int64_t*)colptr, (const int32_t*)csc_row, x_csc, w_csc, E_csc, nnz / d >= 512 ? 256 : 32,
                    nullptr, 1, 0, n, nullptr};
    h->launches += 8;
    // blocked passes: the gathered factor is staged through shared memory in blocks of nb records
    const char* env = getenv("RRI_SP_BLOCKED");
    const bool blocked = !(env && *env == '0');
    const char* env16 = getenv("RRI_SP_IDX16");
    const bool use16 = !(env16 && *env16 == '0');
    size_t part_elems = (size_t)m;
    for (SpSide* sd : {&h->csr, &h->csc}) {
        int nblk = 1;
        const int nb = sp_block_len((int)es, sd->nother, &nblk);
        if (!blocked || nblk > 64) continue;          // (a very long factor would make the sub-segments too short)
        void* p2 = nullptr;
        void* i16 = nullptr;
        if (ws_alloc(h, &p2, sizeof(int64_t) * (size_t)sd->nseg * (size_t)(nblk + 1))) return 1;
        if (use16 && ws_alloc(h, &i16, sizeof(uint16_t) * ne)) return 1;
        CK(cudaStreamSynchronize(0));
        launch_sp_subptr(sd->ptr, sd->idx, sd->nseg, nblk, nb, (int64_t*)p2, h->sm_count, st);
        if (use16 && nnz > 0) {
            launch_sp_local_index(sd->idx, nnz, nb, (uint16_t*)i16, h->sm_count, st);
            sd->idx16 = (const uint16_t*)i16;
            h->launches++;
        }
        sd->ptr2 = (const int64_t*)p2; sd->nblk = nblk; sd->nb = nb;
        if ((size_t)nblk * (size_t)sd->nseg > part_elems) part_elems = (size_t)nblk * (size_t)sd->nseg;
        h->launches++;
    }
    if (ws_alloc(h, &h->sp_npart, es * part_elems) || ws_alloc(h, &h->sp_dpart, es * part_elems)) return 1;
    CK(cudaStreamSynchronize(0));
    CKL();
    CK(cudaStreamSynchronize(st));
    return 0;
}

extern "C" int rri_bind_csr(rri_handle_t h, int64_t nnz, const int64_t* rowptr_dev, const int32_t* col_dev,
                            const void* val_dev, const void* weight_dev, void* stream)
{
    if (!h) return fail("null handle");
    if (h->X) return fail("the handle is already bound; create a new one");
    if (nnz < 0 || nnz >= ((int64_t)1 << 31)) return fail("nnz must be in [0, 2^31) (got %lld)", (long long)nnz);
    if (!rowptr_dev) return fail("rowptr is null");
    if (nnz > 0 && (!col_dev || !val_dev)) return fail("col/val is null");
    if (h->math == RRI_MATH_TF32) return fail("the observed-entries path has no contraction: create the handle with RRI_MATH_IEEE");
    CK(cudaSetDevice(h->device));
    h->nnz = nnz;
    cudaStream_t st = (cudaStream_t)stream;
    const int rc = h->dtype == RRI_F32
                       ? bind_csr_impl<float>(h, rowptr_dev, col_dev, (const float*)val_dev, (const float*)weight_dev, st)
                       : bind_csr_impl<double>(h, rowptr_dev, col_dev, (const double*)val_dev, (const double*)weight_dev, st);
    if (rc) return rc;
    h->sparse = true;
    h->mk = MK_SPARSE;
    h->X = val_dev ? val_dev : (const void*)rowptr_dev;      // "bound" marker; the dense kernels never see it
    return 0;
}

// -------------------------------------------------------------------------------------------------
// zero-filled sparse binding: the block order with a sparse x dense contraction (spmm_kernels.cu)
// -------------------------------------------------------------------------------------------------
// Chunk plan of one orientation: segments longer than SPMM_CHUNK are cut into chunks whose partials are added in chunk
// order by the last one to arrive.  Built on the host from the segment pointers, once per binding.
static int build_spmm_plan(rri_handle_t h, SpmmPlan& pl, int64_t nseg, const int64_t* ptr_dev, const int32_t* idx,
                           const void* val)
{
    std::vector<int64_t> ptr((size_t)nseg + 1);
    CK(cudaMemcpy(ptr.data(), ptr_dev, sizeof(int64_t) * ptr.size(), cudaMemcpyDeviceToHost));
    std::vector<int32_t> lseg;
    std::vector<int64_t> lslot;
    std::vector<int2> litem;
    for (int64_t s = 0; s < nseg; ++s) {
        const int64_t len = ptr[s + 1] - ptr[s];
        if (len <= SPMM_CHUNK) continue;
        const int j = (int)lseg.size();
        lseg.push_back((int32_t)s);
        lslot.push_back((int64_t)litem.size());
        for (int64_t c = 0; c * SPMM_CHUNK < len; ++c) litem.push_back(make_int2(j, (int)c));
    }
    pl = SpmmPlan{};
    pl.nseg = nseg; pl.ptr = ptr_dev; pl.idx = idx; pl.val = val;
    pl.nlong_items = (int64_t)litem.size();
    void *a = nullptr, *b = nullptr, *c = nullptr;
    if (ws_alloc(h, &a, sizeof(int2) * litem.size()) || ws_alloc(h, &b, sizeof(int32_t) * lseg.size()) ||
        ws_alloc(h, &c, sizeof(int64_t) * lslot.size()) || ws_alloc(h, &pl.slots, h->es * litem.size() * (size_t)h->k) ||
        ws_alloc(h, (void**)&pl.counters, sizeof(unsigned) * lseg.size()))
        return 1;
    CK(cudaStreamSynchronize(0));          // (the zero-fills above ran on the legacy default stream)
    if (!litem.empty()) {
        CK(cudaMemcpy(a, litem.data(), sizeof(int2) * litem.size(), cudaMemcpyHostToDevice));
        CK(cudaMemcpy(b, lseg.data(), sizeof(int32_t) * lseg.size(), cudaMemcpyHostToDevice));
        CK(cudaMemcpy(c, lslot.data(), sizeof(int64_t) * lslot.size(), cudaMemcpyHostToDevice));
    }
    pl.litem = (const int2*)a; pl.lseg = (const int32_t*)b; pl.lslot = (const int64_t*)c;
    return 0;
}

template <typename T>
static int bind_csr_zero_impl(rri_handle_t h, const int64_t* rowptr, const int32_t* col, const T* val, cudaStream_t st)
{
    const int64_t n = h->n, d = h->d, nnz = h->nnz;
    const size_t ne = (size_t)(nnz > 0 ? nnz : 1);
    size_t op = 8 * (size_t)h->sm_count;
    if (op < 512) op = 512;
    if (ws_alloc(h, (void**)&h->obj_part, sizeof(double) * op) || ws_alloc(h, (void**)&h->obj_out, sizeof(double) * 16)) return 1;
    void *csc_row = nullptr, *x_csc = nullptr, *colptr = nullptr;
    if (ws_alloc(h, &csc_row, sizeof(int32_t) * ne) || ws_alloc(h, &x_csc, sizeof(T) * ne) ||
        ws_alloc(h, &colptr, sizeof(int64_t) * (size_t)(d + 1)) || ws_alloc(h, (void**)&h->sp_err, sizeof(int)))
        return 1;
    h->splits_w = 1; h->splits_t = 1;
    if (alloc_halfstep_ws(h)) return 1;
    CK(cudaStreamSynchronize(0));
    // the CSR position of every CSC entry is only needed while the column orientation is built
    uint32_t* perm = nullptr;
    CK(cudaMalloc(&perm, sizeof(uint32_t) * ne));
    const int rc = sp_build_csc<T>(rowptr, col, val, nullptr, n, d, nnz, (int64_t*)colptr, (int32_t*)csc_row, (T*)x_csc,
                                   nullptr, perm, h->sm_count, h->sp_err, st);
    cudaFree(perm);
    if (rc < 0)
        return fail("malformed CSR input:%s%s%s", (-rc & 1) ? " rowptr is not a monotone [0..nnz] sequence;" : "",
                    (-rc & 2) ? " column index outside [0,d);" : "",
                    (-rc & 4) ? " column indices must be strictly ascending inside every row (sort and merge duplicates);" : "");
    if (rc > 0) return fail("building the column orientation failed: %s", cudaGetErrorString((cudaError_t)rc));
    h->launches += 8;
    if (build_spmm_plan(h, h->zrow, n, rowptr, col, val) ||
        build_spmm_plan(h, h->zcol, d, (const int64_t*)colptr, (const int32_t*)csc_row, x_csc))
        return 1;
    CKL();
    CK(cudaStreamSynchronize(st));
    return 0;
}

extern "C" int rri_bind_csr_zero(rri_handle_t h, int64_t nnz, const int64_t* rowptr_dev, const int32_t* col_dev,
                                 const void* val_dev, void* stream)
{
    if (!h) return fail("null handle");
    if (h->X) return fail("the handle is already bound; create a new one");
    if (nnz < 0 || nnz >= ((int64_t)1 << 31)) return fail("nnz must be in [0, 2^31) (got %lld)", (long long)nnz);
    if (!rowptr_dev) return fail("rowptr is null");
    if (nnz > 0 && (!col_dev || !val_dev)) return fail("col/val is null");
    if (h->order != RRI_ORDER_HALS) return fail("zero-filled sparse data runs in block order: create the handle with RRI_ORDER_HALS");
    if (h->math != RRI_MATH_IEEE) return fail("zero-filled sparse data runs with RRI_MATH_IEEE (the sparse contraction is not compute-bound)");
    CK(cudaSetDevice(h->device));
    h->nnz = nnz;
    cudaStream_t st = (cudaStream_t)stream;
    const int rc = h->dtype == RRI_F32 ? bind_csr_zero_impl<float>(h, rowptr_dev, col_dev, (const float*)val_dev, st)
                                       : bind_csr_zero_impl<double>(h, rowptr_dev, col_dev, (const double*)val_dev, st);
    if (rc) return rc;
    h->zero_csr = true;
    h->X = val_dev ? val_dev : (const void*)rowptr_dev;      // "bound" marker; the dense kernels never see it
    return 0;
}

static SolveArgs solve_args(const rri_params_t* p, bool forT)
{
    SolveArgs a;
    a.reg_l1 = forT ? p->reg_t_l1 : p->reg_w_l1;
    a.reg_l2 = forT ? p->reg_t_l2 : p->reg_w_l2;
    a.eps = p->eps;
    const double ub = forT ? p->ub_t : p->ub_w;
    a.has_ub = ub > 0 ? 1 : 0;
    a.ub = ub > 0 ? ub : 0.0;
    return a;
}

static int check_params(rri_handle_t h, const rri_params_t* p)
{
    if (!p) return fail("null params");
    if (!h->X) return fail("rri_bind has not been called");
    if (p->fix_W && p->fix_T) return fail("fix_W and fix_T both set: nothing to update");
    if (p->fix_W) return fail("fix_W=True is not supported on the device path (the reference's T-only sweep also rescales W, nmf.py:450-452)");
    // simplex_T, unmasked: Euclidean projection of the row onto the simplex (optimization.py:58-59); masked / observed
    // entries: the vector-c branch rescales the clipped solution to the sum (optimization.py:85-87)
    if (p->simplex_T && !(p->ub_t > 0)) return fail("simplex_T needs t_row_sum > 0");
    return 0;
}

// -------------------------------------------------------------------------------------------------
// rri order, unmasked
// -------------------------------------------------------------------------------------------------
template <typename T>
static int rri_prologue(rri_handle_t h, T* W, int t0, const rri_params_t* p, cudaStream_t st)
{
    // p = w_t0' X and g = w_t0' W for the first T-step (nmf.py:672-673)
    launch_rri_pass<T>((const T*)h->X, h->ldx, h->n, h->d, nullptr, W, h->k, t0, (T*)h->ypart, (T*)h->ppart,
                       false, true, h->pp, st);
    launch_rri_wstep<T>(W, h->n, h->k, 0, t0, (const T*)h->ypart, h->pp.ct, h->n, (const T*)h->hpart, h->hb,
                        solve_args(p, false), (T*)h->gpart, h->sums, h->flags, false, h->gbw, st);
    h->launches += 2;
    CKL();
    return 0;
}

template <typename T>
static int rri_finish(rri_handle_t h, int t_last, cudaStream_t st)
{
    // the sum of the last updated W column has no consumer kernel: finalize it here
    if (h->world > 1) {
        launch_reduce_stat<T>((const T*)h->ppart, 0, 0, (const T*)h->gpart, h->gbw, h->k, (T*)h->stat, st);
        if (allreduce(h, h->stat, (size_t)(h->k + 1), st)) return 1;
        launch_finalize_sums<T>((const T*)h->stat, 1, h->k, t_last, h->sums, h->flags, st);
        h->launches += 2;
    } else {
        launch_finalize_sums<T>((const T*)h->gpart, h->gbw, h->k, t_last, h->sums, h->flags, st);
        h->launches++;
    }
    CKL();
    return 0;
}

template <typename T>
static int rri_topic_range(rri_handle_t h, T* W, T* Tm, int t0, int t1, bool first_has_prev,
                           const rri_params_t* p, cudaStream_t st)
{
    const int k = h->k;
    const int64_t n = h->n, d = h->d;
    const SolveArgs at = solve_args(p, true), aw = solve_args(p, false);
    for (int t = t0; t < t1; ++t) {
        const int tn = (t + 1) % k;
        const int t_prev = ((t == t0 && !first_has_prev) || k == 1) ? -1 : (t + k - 1) % k;
        const T* pp = (const T*)h->ppart; int rg = h->pp.rg;
        const T* gp = (const T*)h->gpart; int gb = h->gbw;
        if (h->world > 1) {
            launch_reduce_stat<T>(pp, rg, d, gp, gb, k, (T*)h->stat, st);
            h->launches++;
            if (allreduce(h, h->stat, (size_t)(d + k + 1), st)) return 1;
            pp = (const T*)h->stat; rg = 1;
            gp = (const T*)h->stat + d; gb = 1;
        }
        launch_rri_tstep<T>(Tm, d, k, t, pp, rg, d, gp, gb, at, (T*)h->hpart, h->sums, t_prev, h->flags, true, st);
        if (p->simplex_T) {
            // qf_min with s = t_row_sum projects the scalar-c solution onto the simplex
            // (optimization.py:58-59); h = T T_t' must then be taken from the projected row
            launch_project_rows_simplex<T>(Tm + (int64_t)t * d, 1, d, p->ub_t, st);
            launch_rri_tstep<T>(Tm, d, k, t, pp, rg, d, gp, gb, at, (T*)h->hpart, h->sums, -1, h->flags, false, st);
            h->launches += 2;
        }
        // k == 1: the look-ahead statistic p = w_tn'X would be taken from the column this very topic is
        // about to overwrite, so it is recomputed after the W-step instead
        launch_rri_pass<T>((const T*)h->X, h->ldx, n, d, Tm + (int64_t)t * d, W, k, tn, (T*)h->ypart,
                           (T*)h->ppart, true, k > 1, h->pp, st);
        launch_rri_wstep<T>(W, n, k, t, tn, (const T*)h->ypart, h->pp.ct, n, (const T*)h->hpart, h->hb, aw,
                            (T*)h->gpart, h->sums, h->flags, true, h->gbw, st);
        h->launches += 3;
        if (k == 1) {
            if (rri_finish<T>(h, 0, st)) return 1;
            if (rri_prologue<T>(h, W, 0, p, st)) return 1;
        }
    }
    CKL();
    return 0;
}

// -------------------------------------------------------------------------------------------------
// hals order, unmasked
// -------------------------------------------------------------------------------------------------
// C = A B' over the data (A = X or X'), plus -- TF32 path, G != null -- the Gram matrix G = B B' of the factor as one
// more row tile of the same launch
template <typename T>
static int contraction(rri_handle_t h, const T* A, int64_t lda, const T* B, int64_t ldb, T* Cpart,
                       int64_t M, int N, int64_t K, int splits, cudaStream_t st, T* G = nullptr)
{
    if (h->math == RRI_MATH_TF32) {
        std::string err;
        int nl = tf32_gemm_run(h->tf32, (const float*)A, lda, (const float*)B, ldb, (float*)Cpart, N, M, N, K, st, err,
                               G ? (const float*)B : nullptr, ldb, G ? N : 0, (float*)G, N);
        if (nl < 0) return fail("tf32 contraction failed: %s", err.c_str());
        h->launches += nl;
    } else {
        launch_simt_gemm_nt<T>(A, lda, B, ldb, Cpart, M, N, K, splits, st);
        h->launches++;
    }
    return 0;
}

// the Gram matrix of a half-step: on the tensor cores inside the contraction launch (TF32 math, RRI_TC_GRAM=0 to
// switch off), otherwise the IEEE gram_kernel + fixed-order reduce
static bool gram_in_contraction(rri_handle_t h)
{
    static const bool off = [] { const char* e = getenv("RRI_TC_GRAM"); return e && *e == '0'; }();
    return h->math == RRI_MATH_TF32 && !off;
}

template <typename T>
static int hals_W_half(rri_handle_t h, T* W, const T* Tk, int64_t ldtk, const rri_params_t* p, bool recompute, cudaStream_t st)
{
    const int k = h->k;
    const int64_t n = h->n, d = h->d;
    if (recompute) {
        // C2 = X T' and H = T T' (from the d x k transposed copy, or as the Gram tile of the contraction)
        const bool tc_gram = gram_in_contraction(h);
        if (!tc_gram) { launch_gram<T>((const T*)h->Tt, d, k, (T*)h->gram_part, h->gchunks_t, (T*)h->Hm, st); h->launches += 2; }
        if (h->zero_csr) {
            launch_spmm<T>(h->zrow, (const T*)h->Tt, k, (T*)h->Cpart, st);
            h->launches++;
        } else if (contraction<T>(h, (const T*)h->X, h->ldx, Tk, ldtk, (T*)h->Cpart, n, k, d, h->splits_w, st, tc_gram ? (T*)h->Hm : nullptr)) {
            return 1;
        }
    }
    const int parts = h->math == RRI_MATH_TF32 ? 1 : h->splits_w;
    // the zero-column test of nmf.py:793 is over ALL rows: with row shards the sums are all-reduced once per call
    // (the per-topic sums and the zero-topic flags are taken once per call from W' and T: hals_finish_sums)
    launch_update_rows<T>(W, n, k, (const T*)h->Cpart, parts, n * k, nullptr, (const T*)h->Hm, solve_args(p, false),
                          (T*)h->Wt, h->ldwt, (T*)h->colsum_part, h->flags, h->ub_blocks_w,
                          ColsumOut{nullptr, k, 0, h->counters + 0}, st);
    h->launches++;
    CKL();
    return 0;
}

// Tk [k, ldtk]: where T is written (the caller's T, or this rank's replica inside the peer-exchange buffer)
template <typename T>
static int hals_T_half(rri_handle_t h, T* W, T* Tk, int64_t ldtk, const rri_params_t* p, cudaStream_t st)
{
    const int k = h->k;
    const int64_t n = h->n, d = h->d;
    T* cg = (T*)h->cg;                 // [d*k | k*k]: X'W partial followed by W'W partial, all-reduced together
    T* G = cg + (size_t)d * k;
    const bool tc_gram = gram_in_contraction(h);
    const int psplits = h->math == RRI_MATH_TF32 ? 1 : h->splits_t;
    if (h->world > 1 && h->p2p && !p->simplex_T) {
        // Exchange over NVLink peer memory fused with the update: this rank's partials [X_i'W_i | W_i'W_i] are
        // produced straight into its exported slot, then ONE kernel publishes / waits, adds the slices it owns over
        // all ranks in rank order, updates those rows of T' and stores them into every rank's replicas.
        const unsigned e = ++h->epoch;
        const int b = (int)(e & 1u);
        T* myC = (T*)((char*)h->xbuf + (size_t)b * h->xslot_elems * h->es);      // partial  [d*k | k*k]
        T* myG = myC + (size_t)d * k;
        if (!tc_gram) { launch_gram<T>(W, n, k, (T*)h->gram_part, h->gchunks_w, myG, st); h->launches += 2; }
        T* Cdst = psplits == 1 ? myC : (T*)h->Cpart;
        if (contraction<T>(h, (const T*)h->Xt, h->ldxt, (const T*)h->Wt, h->ldwt, Cdst, d, k, n, h->splits_t, st,
                           tc_gram ? myG : nullptr)) return 1;
        if (psplits > 1) { launch_reduce_parts<T>((const T*)h->Cpart, psplits, d * k, d * k, myC, st); h->launches++; }
        const PeerExchange px = peer_args(h, e);
        const int blocks = peer_update_blocks(px.row_hi - px.row_lo, h->sm_count);
        const int nl = launch_peer_update_rows<T>(px, d, k, solve_args(p, true), G, (T*)h->colsum_part, h->flags, h->sums,
                                                  h->counters + 1, blocks, st);
        if (!nl) return fail("the fused peer-memory T update does not support k = %d", k);
        h->launches += nl;
        CKL();
        return 0;
    }
    if (!tc_gram) { launch_gram<T>(W, n, k, (T*)h->gram_part, h->gchunks_w, G, st); h->launches += 2; }
    // (one rank, TF32: the Gram tile lands right behind the contraction output, as the all-reduce wants it)
    T* Cout = (h->world > 1 && psplits == 1) ? cg : (T*)h->Cpart;
    if (h->zero_csr) {
        launch_spmm<T>(h->zcol, W, k, Cout, st);
        h->launches++;
    } else if (contraction<T>(h, (const T*)h->Xt, h->ldxt, (const T*)h->Wt, h->ldwt, Cout, d, k, n, h->splits_t, st,
                              tc_gram ? G : nullptr)) {
        return 1;
    }
    const T* C = Cout;
    int parts = psplits;
    if (h->world > 1) {
        if (psplits > 1) { launch_reduce_parts<T>(C, parts, d * k, d * k, cg, st); h->launches++; }
        if (allreduce(h, cg, (size_t)d * k + (size_t)k * k, st)) return 1;
        C = cg; parts = 1;
    }
    if (p->simplex_T) {
        // the projection couples the columns of T: one cooperative launch, or a chain of per-topic launches where
        // the grid cannot be co-resident or k is outside the fused kernel's register range (RRI_SIMPLEX_FUSED=0
        // forces the chain; read per call so that one process can time both)
        const char* e = getenv("RRI_SIMPLEX_FUSED");
        int nl = 0;
        const int rc = launch_simplex_T_update<T>((T*)h->Tt, d, k, C, parts, d * k, G, solve_args(p, true), p->ub_t, Tk,
                                                  ldtk, h->sx_slots, h->flags, h->sm_count, !(e && *e == '0'), &nl, st);
        if (rc) return fail("constrained T update failed: %s", cudaGetErrorString((cudaError_t)rc));
        h->launches += nl;
        return 0;
    }
    // Tt (d x k) is updated in place; its transpose is written straight into the caller's T (k x d)
    launch_update_rows<T>((T*)h->Tt, d, k, C, parts, d * k, nullptr, G, solve_args(p, true), Tk, ldtk, (T*)h->colsum_part,
                          h->flags, h->ub_blocks_t, ColsumOut{nullptr, 0, 0, h->counters + 2}, st);
    h->launches++;
    CKL();
    return 0;
}

// Once per call: sum(T[t,:]) and sum(W[:,t]) (nmf.py:757, :793) with the zero-topic flags, from the rows of T and of
// W' -- a topic that empties inside a call makes the next half-step's denominator zero and raises the unbounded flag
// anyway, so nothing is lost by not looking after every half-step.  On row shards the test on W is over ALL rows: the
// shard sums are all-reduced.  t_sums: take the T sums here (false where the peer exchange finalised them itself).
template <typename T>
static int hals_finish_sums(rri_handle_t h, const T* Tm, bool t_sums, cudaStream_t st)
{
    launch_rowsum_flag<T>((const T*)h->Wt, h->k, h->n, h->ldwt, h->sums, h->k, h->world > 1 ? 0 : 2, h->flags, st);
    h->launches++;
    if (t_sums) {
        launch_rowsum_flag<T>(Tm, h->k, h->d, h->d, h->sums, 0, 1, h->flags, st);
        h->launches++;
    }
    if (h->world <= 1) return 0;
    NCK(g_nccl.AllReduce(h->sums + h->k, h->sums + h->k, (size_t)h->k, 8, 0, h->comm, st));
    launch_flag_from_sums(h->sums, h->k, h->k, 2, h->flags, st);
    h->launches += 2;
    return 0;
}

// -------------------------------------------------------------------------------------------------
// masked WRRI (both orders)
// -------------------------------------------------------------------------------------------------
// vector-c solve with a sum constraint (optimization.py:85-87): x <- s x / sum(x), with sum(x) = sums[t] taken
// after the ub clip; the copy the next pass reads (row2, stride ld2) is rescaled as well, and sums[t] becomes the
// sum AFTER the rescaling -- the nt1 that the zero-topic test of nmf.py:757 sees
template <typename T>
static void scale_row_to_sum(rri_handle_t h, T* row, T* row2, int64_t ld2, int t, const rri_params_t* p, cudaStream_t st)
{
    launch_vec_scale_to_sum<T>(row, h->d, 1, h->sums, t, p->ub_t, st);
    if (row2) { launch_vec_scale_to_sum<T>(row2, h->d, ld2, h->sums, t, p->ub_t, st); h->launches++; }
    launch_vec_sum_flag<T>(row, h->d, 1, h->sums, t, 1, h->flags, st);
    h->launches += 2;
}

template <typename T>
static int wrri_T_step(rri_handle_t h, T* W, T* Tm, int t, const rri_params_t* p, cudaStream_t st)
{
    const int64_t n = h->n, d = h->d;
    int parts = h->tpl.groups;
    if (h->wtc) {
        std::string err;
        parts = h->wtc_groups_t;
        if (wrri_tc_stats(h->wtc, 0, (const float*)h->X, h->ldx, h->M, h->mk, h->ldm, t, (const float*)Tm + (int64_t)t * d, (float*)h->numer_part,
                          (float*)h->denom_part, parts, st, err) < 0)
            return fail("tensor-core WRRI T statistics failed: %s", err.c_str());
    } else {
        launch_wrri_tstats<T>((const T*)h->X, h->ldx, h->M, h->mk, h->ldm, W, Tm, n, d, h->k, t, (T*)h->numer_part,
                              (T*)h->denom_part, h->tpl, st);
    }
    h->launches++;
    const T* nu = (const T*)h->numer_part; const T* de = (const T*)h->denom_part;
    if (h->world > 1) {
        T* ms = (T*)h->mstat;
        launch_reduce_parts<T>(nu, parts, d, d, ms, st);
        launch_reduce_parts<T>(de, parts, d, d, ms + d, st);
        h->launches += 2;
        if (allreduce(h, ms, (size_t)2 * d, st)) return 1;
        nu = ms; de = ms + d; parts = 1;
    }
    T* tp2 = h->wtc ? (T*)wrri_tc_Tp(h->wtc) + t : nullptr;       // keep the padded T' operand in step
    launch_wrri_final<T>(nu, de, parts, d, solve_args(p, true), Tm + (int64_t)t * d, 1, tp2,
                         h->wtc ? wrri_tc_KP(h->wtc) : 0, h->flags, st);
    launch_vec_sum_flag<T>(Tm + (int64_t)t * d, d, 1, h->sums, t, p->simplex_T ? 0 : 1, h->flags, st);
    h->launches += 2;
    if (p->simplex_T) scale_row_to_sum<T>(h, Tm + (int64_t)t * d, tp2, h->wtc ? wrri_tc_KP(h->wtc) : 0, t, p, st);
    return 0;
}

template <typename T>
static int wrri_W_step(rri_handle_t h, T* W, T* Tm, int t, const rri_params_t* p, cudaStream_t st)
{
    const int64_t n = h->n, d = h->d;
    int parts = h->wpl.groups;
    if (h->wtc) {
        std::string err;
        parts = h->wtc_groups_w;
        if (wrri_tc_stats(h->wtc, 1, (const float*)h->X, h->ldx, h->M, h->mk, h->ldm, t, (const float*)Tm + (int64_t)t * d, (float*)h->numer_part,
                          (float*)h->denom_part, parts, st, err) < 0)
            return fail("tensor-core WRRI W statistics failed: %s", err.c_str());
    } else {
        launch_wrri_wstats<T>((const T*)h->X, h->ldx, h->M, h->mk, h->ldm, W, Tm, n, d, h->k, t, (T*)h->numer_part,
                              (T*)h->denom_part, h->wpl, st);
    }
    T* wp2 = h->wtc ? (T*)wrri_tc_Wp(h->wtc) + t : nullptr;       // keep the padded W operand in step
    launch_wrri_final<T>((const T*)h->numer_part, (const T*)h->denom_part, parts, n, solve_args(p, false),
                         W + t, h->k, wp2, h->wtc ? wrri_tc_KP(h->wtc) : 0, h->flags, st);
    launch_vec_sum_flag<T>(W + t, n, h->k, h->sums, h->k + t, h->world > 1 ? 0 : 2, h->flags, st);
    h->launches += 3;
    if (h->world > 1) {
        // the zero-column test of nmf.py:793 is over ALL rows: all-reduce the shard sum (a double)
        NCK(g_nccl.AllReduce(h->sums + h->k + t, h->sums + h->k + t, 1, 8, 0, h->comm, st));
        launch_flag_from_sums(h->sums, h->k + t, 1, 2, h->flags, st);
        h->launches += 2;
    }
    return 0;
}

// -------------------------------------------------------------------------------------------------
// observed-entries WRRI (both orders): one streaming pass over the CSC copy per T-step, over the CSR copy
// per W-step (sparse_kernels.cu)
// -------------------------------------------------------------------------------------------------
struct SpPending {             // rank-one change  wo to' - wn tn'  a residual copy has not absorbed yet
    const void *wo = nullptr, *wn = nullptr, *to = nullptr, *tn = nullptr;
};
struct SpState {
    SpPending csr, csc;
    int ct = 0, cw = 0;                 // parity of the told / wold buffers
    const void* told_cur = nullptr;     // T[t,:] before this topic's T-step (null: no T-step preceded the W-step)
};

template <typename T>
static void sp_refresh(rri_handle_t h, bool need_csr, bool need_csc, const T* W, cudaStream_t st)
{
    // E = X - W T on the observed entries, from the current factors
    if (h->sp_refresh_v2) {
        // the row copy from the factors (16-byte gathers of T' rows), the column copy as a permutation of it
        launch_sp_residual_rows<T>(h->csr, W, h->k, (const T*)h->Tt, h->sp_ldt, h->k, h->sm_count, st);
        h->launches++;
        if (need_csc && h->nnz > 0) {
            launch_sp_gather<T>(h->sp_perm, (const T*)h->csr.E, (T*)h->csc.E, h->nnz, h->sm_count, st);
            h->launches++;
        }
        return;
    }
    if (need_csc) { launch_sp_residual<T>(h->csc, (const T*)h->Tt, W, h->k, h->sm_count, st); h->launches++; }
    if (need_csr) { launch_sp_residual<T>(h->csr, W, (const T*)h->Tt, h->k, h->sm_count, st); h->launches++; }
}

template <typename T>
static int sp_T_step(rri_handle_t h, T* W, T* Tm, int t, const rri_params_t* p, SpState& S, cudaStream_t st)
{
    const int64_t n = h->n, d = h->d;
    const T* wt = (const T*)h->Wt + (int64_t)t * h->ldwt;            // W[:,t], contiguous
    T* trow = Tm + (int64_t)t * d;
    T* told = (T*)h->sp_told + (int64_t)(S.ct & 1) * d;
    T* ms = (T*)h->mstat;                                            // [numer(d) | denom(d)] for the all-reduce
    launch_sp_pack<T>((const T*)S.csc.wo, (const T*)S.csc.wn, wt, wt, h->sp_quad, n, st);
    const T* nu = (const T*)h->sp_npart; const T* de = (const T*)h->sp_dpart;
    int parts = launch_sp_pass<T>(h->csc, h->sp_quad, (const T*)S.csc.to, (const T*)S.csc.tn, trow, told, (T*)h->sp_npart,
                                  (T*)h->sp_dpart, h->sm_count, st);
    h->launches += 2;
    if (h->world > 1) {
        launch_reduce_parts<T>(nu, parts, d, d, ms, st);
        launch_reduce_parts<T>(de, parts, d, d, ms + d, st);
        h->launches += 2;
        if (allreduce(h, ms, (size_t)2 * d, st)) return 1;
        nu = ms; de = ms + d; parts = 1;
    }
    launch_wrri_final<T>(nu, de, parts, d, solve_args(p, true), trow, 1, (T*)h->Tt + t, h->sp_ldt, h->flags, st);
    h->launches++;
    if (!h->sp_batched_sums || p->simplex_T) {
        launch_vec_sum_flag<T>(trow, d, 1, h->sums, t, p->simplex_T ? 0 : 1, h->flags, st);
        h->launches++;
    }
    if (p->simplex_T) scale_row_to_sum<T>(h, trow, (T*)h->Tt + t, h->sp_ldt, t, p, st);
    S.csc = SpPending{wt, wt, told, trow};       // w_t (told - tnew)'; merged with the W-step's change if one follows
    S.told_cur = told;
    S.ct++;
    return 0;
}

template <typename T>
static int sp_W_step(rri_handle_t h, T* W, T* Tm, int t, const rri_params_t* p, SpState& S, cudaStream_t st)
{
    const int64_t n = h->n, d = h->d;
    T* wt = (T*)h->Wt + (int64_t)t * h->ldwt;
    const T* trow = Tm + (int64_t)t * d;
    const T* told = S.told_cur ? (const T*)S.told_cur : trow;
    T* wold = (T*)h->sp_wold + (int64_t)(S.cw & 1) * n;
    launch_sp_pack<T>((const T*)S.csr.to, (const T*)S.csr.tn, told, trow, h->sp_quad, d, st);
    const int parts = launch_sp_pass<T>(h->csr, h->sp_quad, (const T*)S.csr.wo, (const T*)S.csr.wn, wt, wold,
                                        (T*)h->sp_npart, (T*)h->sp_dpart, h->sm_count, st);
    launch_wrri_final<T>((const T*)h->sp_npart, (const T*)h->sp_dpart, parts, n, solve_args(p, false), W + t, h->k, wt, 1,
                         h->flags, st);
    h->launches += 3;
    if (!h->sp_batched_sums) {
        launch_vec_sum_flag<T>(wt, n, 1, h->sums, h->k + t, h->world > 1 ? 0 : 2, h->flags, st);
        h->launches++;
        if (h->world > 1) {
            NCK(g_nccl.AllReduce(h->sums + h->k + t, h->sums + h->k + t, 1, 8, 0, h->comm, st));
            launch_flag_from_sums(h->sums, h->k + t, 1, 2, h->flags, st);
            h->launches += 2;
        }
    }
    // both copies now lag by  wold told' - wnew tnew'  (one record even when a T-step preceded: the terms in
    // w_old t_new' cancel)
    S.csr = SpPending{wold, wt, told, trow};
    if (S.told_cur) S.csc = S.csr;
    S.told_cur = nullptr;
    S.cw++;
    return 0;
}

// The 2k single-block column-sum launches of a sweep (13.6 us each at config-4 shape) replaced by two launches at its
// end -- row t of T and of W' is final once its step has run (RRI_SP_BATCHED_SUMS=0 restores the per-step sums).
template <typename T>
static int sp_topic_sums(rri_handle_t h, const T* Tm, int t0, int t1, bool did_T, bool did_W, cudaStream_t st)
{
    if (!h->sp_batched_sums) return 0;
    if (did_T) { launch_rowsum_flag<T>(Tm + (int64_t)t0 * h->d, t1 - t0, h->d, h->d, h->sums, t0, 1, h->flags, st); h->launches++; }
    if (did_W) {
        launch_rowsum_flag<T>((const T*)h->Wt + (int64_t)t0 * h->ldwt, t1 - t0, h->n, h->ldwt, h->sums, h->k + t0,
                              h->world > 1 ? 0 : 2, h->flags, st);
        h->launches++;
        if (h->world > 1) {
            NCK(g_nccl.AllReduce(h->sums + h->k + t0, h->sums + h->k + t0, (size_t)(t1 - t0), 8, 0, h->comm, st));
            launch_flag_from_sums(h->sums, h->k + t0, t1 - t0, 2, h->flags, st);
            h->launches += 2;
        }
    }
    return 0;
}

template <typename T>
static int sp_load_factors(rri_handle_t h, const T* W, const T* Tm, cudaStream_t st)
{
    launch_transpose<T>(Tm, h->k, h->d, h->d, (T*)h->Tt, h->sp_ldt, st);     // T' [d,k] (padded row stride)
    launch_transpose<T>(W, h->n, h->k, h->k, (T*)h->Wt, h->ldwt, st);        // W' [k,ldwt]
    h->launches += 2;
    CKL();
    return 0;
}

template <typename T>
static int sp_topic_range(rri_handle_t h, T* W, T* Tm, int t0, int t1, const rri_params_t* p, cudaStream_t st,
                          SpState* carried = nullptr, bool restart = true)
{
    // reference order (nmf.py:415-476).  restart: both residual copies are rebuilt from the current factors (always at
    // the start of a call); otherwise they continue from the previous sweep with its pending rank-one record
    SpState local;
    SpState& S = carried ? *carried : local;
    if (restart) { S = SpState(); sp_refresh<T>(h, true, true, W, st); }
    for (int t = t0; t < t1; ++t) {
        if (sp_T_step<T>(h, W, Tm, t, p, S, st)) return 1;
        if (sp_W_step<T>(h, W, Tm, t, p, S, st)) return 1;
    }
    if (sp_topic_sums<T>(h, Tm, t0, t1, true, true, st)) return 1;
    CKL();
    return 0;
}

template <typename T>
static int sp_sweeps(rri_handle_t h, T* W, T* Tm, int n_sweeps, const rri_params_t* p, cudaStream_t st)
{
    const int k = h->k;
    if (sp_load_factors<T>(h, W, Tm, st)) return 1;
    // residual restart period inside one call (rri_params_t.sp_refresh_every; 0 or 1 = every sweep, which makes
    // N sweeps in one call == N calls of one sweep bit for bit).  The restart costs 17 % of a config-4 sweep; with a
    // longer period the two residual copies are carried from sweep to sweep (interleaved order only: in block order
    // each half updates one copy k times while the other stands still).
    const int every = p->sp_refresh_every > 1 ? p->sp_refresh_every : 1;
    SpState carried;
    for (int s = 0; s < n_sweeps; ++s) {
        if (!p->fix_T && h->order == RRI_ORDER_RRI) {
            if (sp_topic_range<T>(h, W, Tm, 0, k, p, st, &carried, s % every == 0)) return 1;
            continue;
        }
        if (!p->fix_T) {                       // block order, T half: only the column copy is read
            SpState S;
            sp_refresh<T>(h, false, true, W, st);
            for (int t = 0; t < k; ++t) {
                if (sp_T_step<T>(h, W, Tm, t, p, S, st)) return 1;
                S.told_cur = nullptr;
            }
        }
        SpState S;                             // W half (also transform(): fix_T): only the row copy is read
        sp_refresh<T>(h, true, false, W, st);
        for (int t = 0; t < k; ++t)
            if (sp_W_step<T>(h, W, Tm, t, p, S, st)) return 1;
        if (sp_topic_sums<T>(h, Tm, 0, k, !p->fix_T, true, st)) return 1;
    }
    CKL();
    return 0;
}

// -------------------------------------------------------------------------------------------------
// sweeps
// -------------------------------------------------------------------------------------------------
template <typename T>
static int sweeps_impl(rri_handle_t h, T* W, T* Tm, int n_sweeps, const rri_params_t* p, cudaStream_t st)
{
    const int k = h->k;
    const int64_t n = h->n, d = h->d;
    if (h->sparse) return sp_sweeps<T>(h, W, Tm, n_sweeps, p, st);
    if (h->mk != MK_NONE) {
        if (h->wtc) { wrri_tc_load_factors(h->wtc, (const float*)W, (const float*)Tm, st); h->launches += 2; }
        for (int s = 0; s < n_sweeps; ++s) {
            if (h->order == RRI_ORDER_RRI) {
                for (int t = 0; t < k; ++t) {
                    if (!p->fix_T && wrri_T_step<T>(h, W, Tm, t, p, st)) return 1;
                    if (!p->fix_W && wrri_W_step<T>(h, W, Tm, t, p, st)) return 1;
                }
            } else {
                if (!p->fix_T) for (int t = 0; t < k; ++t) if (wrri_T_step<T>(h, W, Tm, t, p, st)) return 1;
                if (!p->fix_W) for (int t = 0; t < k; ++t) if (wrri_W_step<T>(h, W, Tm, t, p, st)) return 1;
            }
        }
        CKL();
        return 0;
    }
    if (p->fix_T) {
        // W-only sweeps (transform(): sklearn_interface.py:327-334): X T' and T T' are constant, so
        // one pass over X serves every sweep; both update orders coincide here
        launch_transpose<T>(Tm, k, d, d, (T*)h->Tt, k, st);
        h->launches++;
        for (int s = 0; s < n_sweeps; ++s)
            if (hals_W_half<T>(h, W, Tm, d, p, s == 0, st)) return 1;
        return n_sweeps > 0 ? hals_finish_sums<T>(h, Tm, false, st) : 0;
    }
    if (h->order == RRI_ORDER_HALS) {
        launch_transpose<T>(Tm, k, d, d, (T*)h->Tt, k, st);
        launch_transpose<T>(W, n, k, k, (T*)h->Wt, h->ldwt, st);
        h->launches += 2;
        const bool px = h->world > 1 && h->p2p;
        // with the peer exchange the current T lives in this rank's replica inside the exchange buffer (the peers
        // store the rows they update into it); the caller's T is loaded into it here and read back at the end
        T* Tk = px ? (T*)((char*)h->xbuf + h->x_off_tk) : Tm;
        const int64_t ldtk = px ? h->ldtk : d;
        if (px) CK(cudaMemcpy2DAsync(Tk, (size_t)ldtk * sizeof(T), Tm, (size_t)d * sizeof(T), (size_t)d * sizeof(T), (size_t)k,
                                     cudaMemcpyDeviceToDevice, st));
        for (int s = 0; s < n_sweeps; ++s) {
            if (hals_T_half<T>(h, W, Tk, ldtk, p, st)) return 1;
            if (hals_W_half<T>(h, W, Tk, ldtk, p, true, st)) return 1;
        }
        if (px) CK(cudaMemcpy2DAsync(Tm, (size_t)d * sizeof(T), Tk, (size_t)ldtk * sizeof(T), (size_t)d * sizeof(T), (size_t)k,
                                     cudaMemcpyDeviceToDevice, st));
        h->c2_valid = n_sweeps > 0;            // Cpart = X T' for the T just written, Tt = its transpose
        return n_sweeps > 0 ? hals_finish_sums<T>(h, Tm, !(px && !p->simplex_T), st) : 0;
    }
    if (rri_prologue<T>(h, W, 0, p, st)) return 1;
    for (int s = 0; s < n_sweeps; ++s)
        if (rri_topic_range<T>(h, W, Tm, 0, k, s > 0, p, st)) return 1;
    return k == 1 ? 0 : rri_finish<T>(h, k - 1, st);     // (k == 1 finalises inside the topic loop)
}

static int read_flags(rri_handle_t h, int32_t* flags_host, cudaStream_t st)
{
    if (!flags_host) return 0;
    CK(cudaMemcpyAsync(flags_host, h->flags, sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return 0;
}

extern "C" int rri_sweeps(rri_handle_t h, void* W_dev, void* T_dev, int32_t n_sweeps, const rri_params_t* p,
                          int32_t* flags_host, void* stream)
{
    if (!h) return fail("null handle");
    if (!W_dev || !T_dev) return fail("W or T is null");
    if (n_sweeps < 0) return fail("n_sweeps < 0");
    if (check_params(h, p)) return 1;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    CK(cudaMemsetAsync(h->flags, 0, sizeof(int), st));
    h->c2_valid = false;
    if (n_sweeps > 0) {
        int rc = h->dtype == RRI_F32 ? sweeps_impl<float>(h, (float*)W_dev, (float*)T_dev, n_sweeps, p, st)
                                     : sweeps_impl<double>(h, (double*)W_dev, (double*)T_dev, n_sweeps, p, st);
        if (rc) return rc;
    }
    return read_flags(h, flags_host, st);
}

template <typename T>
static int topics_impl(rri_handle_t h, T* W, T* Tm, int t0, int t1, const rri_params_t* p, cudaStream_t st)
{
    if (h->sparse) {
        if (sp_load_factors<T>(h, W, Tm, st)) return 1;
        return sp_topic_range<T>(h, W, Tm, t0, t1, p, st);
    }
    if (h->mk != MK_NONE) {
        if (h->wtc) { wrri_tc_load_factors(h->wtc, (const float*)W, (const float*)Tm, st); h->launches += 2; }
        for (int t = t0; t < t1; ++t) {
            if (wrri_T_step<T>(h, W, Tm, t, p, st)) return 1;
            if (wrri_W_step<T>(h, W, Tm, t, p, st)) return 1;
        }
        CKL();
        return 0;
    }
    if (rri_prologue<T>(h, W, t0, p, st)) return 1;
    if (rri_topic_range<T>(h, W, Tm, t0, t1, false, p, st)) return 1;
    return h->k == 1 ? 0 : rri_finish<T>(h, t1 - 1, st);
}

extern "C" int rri_topics(rri_handle_t h, void* W_dev, void* T_dev, int32_t t_begin, int32_t t_end,
                          const rri_params_t* p, int32_t* flags_host, void* stream)
{
    if (!h) return fail("null handle");
    if (!W_dev || !T_dev) return fail("W or T is null");
    if (check_params(h, p)) return 1;
    if (h->zero_csr) return fail("rri_topics does not serve zero-filled sparse handles (block order only)");
    if (h->order != RRI_ORDER_RRI) return fail("rri_topics needs a handle created with RRI_ORDER_RRI");
    if (p->fix_T) return fail("rri_topics does not take fix_T");
    if (t_begin < 0 || t_end > h->k || t_begin >= t_end) return fail("bad topic range [%d,%d)", t_begin, t_end);
    CK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    CK(cudaMemsetAsync(h->flags, 0, sizeof(int), st));
    int rc = h->dtype == RRI_F32 ? topics_impl<float>(h, (float*)W_dev, (float*)T_dev, t_begin, t_end, p, st)
                                 : topics_impl<double>(h, (double*)W_dev, (double*)T_dev, t_begin, t_end, p, st);
    if (rc) return rc;
    return read_flags(h, flags_host, st);
}

extern "C" int rri_topic_sums(rri_handle_t h, double* sum_T_host, double* sum_W_host, void* stream)
{
    if (!h) return fail("null handle");
    cudaStream_t st = (cudaStream_t)stream;
    CK(cudaSetDevice(h->device));
    if (sum_T_host) CK(cudaMemcpyAsync(sum_T_host, h->sums, sizeof(double) * h->k, cudaMemcpyDeviceToHost, st));
    if (sum_W_host) CK(cudaMemcpyAsync(sum_W_host, h->sums + h->k, sizeof(double) * h->k, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return 0;
}

// -------------------------------------------------------------------------------------------------
// objective, partial statistic, misc
// -------------------------------------------------------------------------------------------------
template <typename T>
static int objective_contraction_impl(rri_handle_t h, const T* W, const T* Tm, bool reuse, cudaStream_t st);

template <typename T>
static int objective_impl(rri_handle_t h, const T* W, const T* Tm, cudaStream_t st)
{
    if (h->zero_csr) return objective_contraction_impl<T>(h, W, Tm, false, st);     // (no pass over n x d entries)
    if (h->sparse) {
        launch_transpose<T>(Tm, h->k, h->d, h->d, (T*)h->Tt, h->sp_ldt, st);
        sp_refresh<T>(h, true, false, W, st);
        launch_sp_objective<T>(h->csr, h->nnz, h->obj_part, h->obj_out, st);
        launch_norms<T>(W, h->n * h->k, h->obj_part, h->obj_out + 2, st);
        launch_norms<T>(Tm, (int64_t)h->k * h->d, h->obj_part, h->obj_out + 4, st);
        h->launches += 7;
        CKL();
        return 0;
    }
    launch_objective<T>((const T*)h->X, h->ldx, h->M, h->mk, h->ldm, W, Tm, h->n, h->d, h->k, h->obj_part,
                        h->oblocks, h->obj_out, st);
    launch_norms<T>(W, h->n * h->k, h->obj_part, h->obj_out + 2, st);
    launch_norms<T>(Tm, (int64_t)h->k * h->d, h->obj_part, h->obj_out + 4, st);
    h->launches += 6;
    CKL();
    return 0;
}

extern "C" int rri_objective(rri_handle_t h, const void* W_dev, const void* T_dev, double* out_host, void* stream)
{
    if (!h) return fail("null handle");
    if (!h->X) return fail("rri_bind has not been called");
    if (!W_dev || !T_dev || !out_host) return fail("null argument");
    CK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    int rc = h->dtype == RRI_F32 ? objective_impl<float>(h, (const float*)W_dev, (const float*)T_dev, st)
                                 : objective_impl<double>(h, (const double*)W_dev, (const double*)T_dev, st);
    if (rc) return rc;
    CK(cudaMemcpyAsync(out_host, h->obj_out, sizeof(double) * 6, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return 0;
}

// Objective through the contraction (unmasked dense data):  ||X - W T||^2 = ||X||^2 - 2 <X T', W> + <W'W, T T'>.
// reuse != 0: the caller states that W and T are exactly what the last rri_sweeps call (block order) left, so the
// contraction X T' of its last W half-step is still in the workspace; otherwise one contraction pass is made.
template <typename T>
static int objective_contraction_impl(rri_handle_t h, const T* W, const T* Tm, bool reuse, cudaStream_t st)
{
    const int64_t n = h->n, d = h->d;
    const int k = h->k;
    if (!h->Gobj && ws_alloc(h, &h->Gobj, sizeof(T) * 2 * (size_t)k * k)) return 1;
    CK(cudaStreamSynchronize(0));
    double* acc = h->obj_out + 8;                       // {||X||^2, <X T', W>}
    if (!h->xsq_valid) {
        if (h->zero_csr) launch_sumsq_rows<T>((const T*)h->zrow.val, 1, h->nnz, h->nnz, h->obj_part, acc, h->sm_count, st);
        else launch_sumsq_rows<T>((const T*)h->X, n, d, h->ldx, h->obj_part, acc, h->sm_count, st);
        h->xsq_valid = true;
        h->launches += 2;
    }
    if (!(reuse && h->c2_valid)) {
        launch_transpose<T>(Tm, k, d, d, (T*)h->Tt, k, st);
        h->launches++;
        if (h->zero_csr) {
            launch_spmm<T>(h->zrow, (const T*)h->Tt, k, (T*)h->Cpart, st);
            h->launches++;
        } else if (contraction<T>(h, (const T*)h->X, h->ldx, Tm, d, (T*)h->Cpart, n, k, d, h->splits_w, st)) {
            return 1;
        }
        h->c2_valid = false;                            // (the caller's T may change before the next call)
    }
    const int parts = h->math == RRI_MATH_TF32 ? 1 : h->splits_w;      // (1 on zero-filled sparse handles)
    launch_dot_parts<T>((const T*)h->Cpart, parts, n * k, W, n * k, h->obj_part, acc + 1, h->sm_count, st);
    T* G = (T*)h->Gobj;
    T* H = G + (size_t)k * k;
    launch_gram<T>(W, n, k, (T*)h->gram_part, h->gchunks_w, G, st);                 // IEEE Gram products
    launch_gram<T>((const T*)h->Tt, d, k, (T*)h->gram_part, h->gchunks_t, H, st);
    launch_objective_identity<T>(G, H, k, acc, h->obj_out, st);
    launch_norms<T>(W, n * k, h->obj_part, h->obj_out + 2, st);
    launch_norms<T>(Tm, (int64_t)k * d, h->obj_part, h->obj_out + 4, st);
    h->launches += 11;
    CKL();
    return 0;
}

extern "C" int rri_objective_contraction(rri_handle_t h, const void* W_dev, const void* T_dev, int32_t reuse_last_sweep,
                                         double* out_host, void* stream)
{
    if (!h) return fail("null handle");
    if (!h->X) return fail("rri_bind has not been called");
    if (!W_dev || !T_dev || !out_host) return fail("null argument");
    if (h->sparse || h->mk != MK_NONE) return fail("the objective through the contraction needs unmasked dense data");
    if (!h->Cpart) return fail("no contraction workspace on this handle");
    CK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (h->world > 1 && h->p2p && h->order == RRI_ORDER_HALS && !(reuse_last_sweep && h->c2_valid))
        return fail("with the peer exchange on, the objective through the contraction is available right after rri_sweeps");
    int rc = h->dtype == RRI_F32 ? objective_contraction_impl<float>(h, (const float*)W_dev, (const float*)T_dev, reuse_last_sweep != 0, st)
                                 : objective_contraction_impl<double>(h, (const double*)W_dev, (const double*)T_dev, reuse_last_sweep != 0, st);
    if (rc) return rc;
    CK(cudaMemcpyAsync(out_host, h->obj_out, sizeof(double) * 6, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return 0;
}

// p[c * pstride] = (X' w_t)[c], g[j] = (W' w_t)[j]
template <typename T>
__global__ void partials_unmasked_kernel(const T* __restrict__ p, int64_t pstride, const T* __restrict__ g,
                                         const T* __restrict__ Tm, int64_t d, int k, int t, T* __restrict__ wR,
                                         T* __restrict__ nw)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c < d) {
        T dot = T(0);
        for (int j = 0; j < k; ++j)
            if (j != t) dot = fma(g[j], Tm[(int64_t)j * d + c], dot);            // nmf.py:674-675
        wR[c] = p[c * pstride] - dot;
    }
    if (c == 0) nw[0] = g[t];                                                       // nmf.py:676
}

template <typename T>
static int partials_impl(rri_handle_t h, const T* W, const T* Tm, int t, T* wR, T* nw, cudaStream_t st)
{
    const int64_t d = h->d;
    rri_params_t p;
    memset(&p, 0, sizeof(p));
    if (h->sparse) {
        if (sp_load_factors<T>(h, W, Tm, st)) return 1;
        sp_refresh<T>(h, false, true, W, st);
        const T* wt = (const T*)h->Wt + (int64_t)t * h->ldwt;
        launch_sp_pack<T>(nullptr, nullptr, wt, wt, h->sp_quad, h->n, st);
        const int parts = launch_sp_pass<T>(h->csc, h->sp_quad, nullptr, nullptr, Tm + (int64_t)t * d, (T*)h->sp_told,
                                            (T*)h->sp_npart, (T*)h->sp_dpart, h->sm_count, st);
        launch_reduce_parts<T>((const T*)h->sp_npart, parts, d, d, wR, st);
        launch_reduce_parts<T>((const T*)h->sp_dpart, parts, d, d, nw, st);
        h->launches += 4;
        CKL();
        return 0;
    }
    if (h->zero_csr) {
        // X' W and W'W of the T half-step, then the statistic of topic t from column t of both
        const int k = h->k;
        T* G = (T*)h->cg + (size_t)d * k;
        launch_spmm<T>(h->zcol, W, k, (T*)h->Cpart, st);
        launch_gram<T>(W, h->n, k, (T*)h->gram_part, h->gchunks_w, G, st);
        partials_unmasked_kernel<T><<<(unsigned)((d + 255) / 256), 256, 0, st>>>((const T*)h->Cpart + t, k, G + (size_t)t * k,
                                                                                  Tm, d, k, t, wR, nw);
        h->launches += 4;
        CKL();
        return 0;
    }
    if (h->mk != MK_NONE) {
        launch_wrri_tstats<T>((const T*)h->X, h->ldx, h->M, h->mk, h->ldm, W, Tm, h->n, d, h->k, t,
                              (T*)h->numer_part, (T*)h->denom_part, h->tpl, st);
        launch_reduce_parts<T>((const T*)h->numer_part, h->tpl.groups, d, d, wR, st);
        launch_reduce_parts<T>((const T*)h->denom_part, h->tpl.groups, d, d, nw, st);
        h->launches += 3;
    } else {
        if (h->order != RRI_ORDER_RRI) return fail("rri_partials_T (unmasked) needs a handle created with RRI_ORDER_RRI");
        if (rri_prologue<T>(h, const_cast<T*>(W), t, &p, st)) return 1;     // prologue does not write W
        launch_reduce_stat<T>((const T*)h->ppart, h->pp.rg, d, (const T*)h->gpart, h->gbw, h->k, (T*)h->stat, st);
        partials_unmasked_kernel<T><<<(unsigned)((d + 255) / 256), 256, 0, st>>>((const T*)h->stat, 1, (const T*)h->stat + d,
                                                                                  Tm, d, h->k, t, wR, nw);
        h->launches += 2;
    }
    CKL();
    return 0;
}

extern "C" int rri_partials_T(rri_handle_t h, const void* W_dev, const void* T_dev, int32_t t, void* out_wR_dev,
                              void* out_nw_dev, void* stream)
{
    if (!h) return fail("null handle");
    if (!h->X) return fail("rri_bind has not been called");
    if (t < 0 || t >= h->k) return fail("bad topic %d", t);
    CK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    return h->dtype == RRI_F32
               ? partials_impl<float>(h, (const float*)W_dev, (const float*)T_dev, t, (float*)out_wR_dev, (float*)out_nw_dev, st)
               : partials_impl<double>(h, (const double*)W_dev, (const double*)T_dev, t, (double*)out_wR_dev, (double*)out_nw_dev, st);
}

extern "C" int rri_project_rows_simplex(rri_handle_t h, void* A_dev, int64_t rows, int64_t cols, double s, void* stream)
{
    if (!h) return fail("null handle");
    if (!A_dev || rows <= 0 || cols <= 0) return fail("bad matrix");
    if (!(s > 0)) return fail("Radius s must be strictly positive");          // matrixops.py:42
    CK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (h->dtype == RRI_F32) launch_project_rows_simplex<float>((float*)A_dev, rows, cols, s, st);
    else launch_project_rows_simplex<double>((double*)A_dev, rows, cols, s, st);
    h->launches++;
    CKL();
    return 0;
}

extern "C" int rri_cache_trim(int32_t device)
{
    CK(cudaSetDevice(device));
    cache_trim();
    // parked exchange buffers: on row shards every rank must trim at the same point (a peer may have this buffer mapped)
    for (PeerGroup& g : g_groups) {
        if (!g.used || g.device != device) continue;
        for (int r = 0; r < 16; ++r)
            if (g.peer_open[r] && g.peer_base[r]) cudaIpcCloseMemHandle(g.peer_base[r]);
        cudaFree(g.xbuf);
        g = PeerGroup();
    }
    return 0;
}

extern "C" int rri_stats(rri_handle_t h, int64_t* kernel_launches, int64_t* workspace_bytes)
{
    if (!h) return fail("null handle");
    if (kernel_launches) *kernel_launches = h->launches;
    if (workspace_bytes) *workspace_bytes = h->ws_bytes;
    return 0;
}

extern "C" int rri_gemm_nt(rri_handle_t h, const void* A_dev, int64_t lda, const void* B_dev, int64_t ldb,
                           void* C_dev, int64_t ldc, int64_t M, int32_t N, int64_t K, void* stream)
{
    if (!h) return fail("null handle");
    if (N <= 0 || N > 256 || M <= 0 || K <= 0) return fail("bad shape");
    if (ldc != N) return fail("ldc must equal N");
    CK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (h->math == RRI_MATH_TF32) {
        if (!h->tf32) {
            std::string err;
            h->tf32 = tf32_gemm_create(h->sm_count, N > h->k ? N : h->k, err);
            if (!h->tf32) return fail("tf32 contraction unavailable: %s", err.c_str());
        }
        std::string err;
        int nl = tf32_gemm_run(h->tf32, (const float*)A_dev, lda, (const float*)B_dev, ldb, (float*)C_dev, N, M, N, K, st, err);
        if (nl < 0) return fail("tf32 contraction failed: %s", err.c_str());
        h->launches += nl;
    } else if (h->dtype == RRI_F32) {
        launch_simt_gemm_nt<float>((const float*)A_dev, lda, (const float*)B_dev, ldb, (float*)C_dev, M, N, K, 1, st);
        h->launches++;
    } else {
        launch_simt_gemm_nt<double>((const double*)A_dev, lda, (const double*)B_dev, ldb, (double*)C_dev, M, N, K, 1, st);
        h->launches++;
    }
    CKL();
    return 0;
}

template <typename T>
static int profile_impl(rri_handle_t h, int which, const T* W, const T* Tm, int iters, float* avg_ms, cudaStream_t st)
{
    const int64_t n = h->n, d = h->d;
    const int k = h->k;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    if (which == 2 && h->mk == MK_NONE && h->order == RRI_ORDER_HALS) {
        launch_transpose<T>(W, n, k, k, (T*)h->Wt, h->ldwt, st);
        h->launches++;
    }
    if (which == 1 && h->zero_csr) {              // the W-half contraction gathers rows of T'
        launch_transpose<T>(Tm, k, d, d, (T*)h->Tt, k, st);
        h->launches++;
    }
    rri_params_t prm;
    memset(&prm, 0, sizeof(prm));
    prm.eps = 1.7763568394002505e-15;
    const bool halves = which == 3 || which == 4;
    T* Tk = const_cast<T*>(Tm);
    int64_t ldtk = d;
    if (halves) {
        if (h->mk != MK_NONE || h->order != RRI_ORDER_HALS) return fail("which=3/4 need an unmasked hals-order handle");
        launch_transpose<T>(Tm, k, d, d, (T*)h->Tt, k, st);
        launch_transpose<T>(W, n, k, k, (T*)h->Wt, h->ldwt, st);
        h->launches += 2;
        if (h->world > 1 && h->p2p) {
            Tk = (T*)((char*)h->xbuf + h->x_off_tk); ldtk = h->ldtk;
            CK(cudaMemcpy2DAsync(Tk, (size_t)ldtk * sizeof(T), Tm, (size_t)d * sizeof(T), (size_t)d * sizeof(T), (size_t)k,
                                 cudaMemcpyDeviceToDevice, st));
        }
    }
    SpState spS;
    if (which == 5 || which == 6) {
        // one masked / observed-entries half-step of topic 0 (statistics pass + solve): the pass kernel dominates
        if (h->mk == MK_NONE) return fail("which=5/6 need a masked or observed-entries handle");
        prm.ub_t = 1.0;
        if (h->sparse) {
            if (sp_load_factors<T>(h, W, Tm, st)) return 1;
            sp_refresh<T>(h, true, true, W, st);
        } else if (h->wtc) {
            wrri_tc_load_factors(h->wtc, (const float*)W, (const float*)Tm, st);
            h->launches += 2;
        }
    }
    for (int it = -1; it < iters; ++it) {          // one untimed warm-up launch
        if (it == 0) CK(cudaEventRecord(e0, st));
        if (which == 5 || which == 6) {
            T* Wm = const_cast<T*>(W); T* Tw = const_cast<T*>(Tm);
            int rc;
            if (h->sparse) rc = which == 5 ? sp_T_step<T>(h, Wm, Tw, 0, &prm, spS, st) : sp_W_step<T>(h, Wm, Tw, 0, &prm, spS, st);
            else rc = which == 5 ? wrri_T_step<T>(h, Wm, Tw, 0, &prm, st) : wrri_W_step<T>(h, Wm, Tw, 0, &prm, st);
            if (rc) return 1;
            continue;
        }
        if (which == 0) {
            if (h->mk != MK_NONE || h->order != RRI_ORDER_RRI) return fail("which=0 needs an unmasked rri-order handle");
            launch_rri_pass<T>((const T*)h->X, h->ldx, n, d, Tm, W, k, 1 % k, (T*)h->ypart, (T*)h->ppart, true, true, h->pp, st);
            h->launches++;
        } else if (which == 1) {
            if (h->mk != MK_NONE) return fail("which=1 needs an unmasked handle");
            if (h->zero_csr) { launch_spmm<T>(h->zrow, (const T*)h->Tt, k, (T*)h->Cpart, st); h->launches++; continue; }
            if (contraction<T>(h, (const T*)h->X, h->ldx, Tm, d, (T*)h->Cpart, n, k, d, h->splits_w, st)) return 1;
        } else if (which == 2) {
            if (h->mk != MK_NONE || h->order != RRI_ORDER_HALS) return fail("which=2 needs an unmasked hals-order handle");
            if (h->zero_csr) { launch_spmm<T>(h->zcol, W, k, (T*)h->Cpart, st); h->launches++; continue; }
            if (contraction<T>(h, (const T*)h->Xt, h->ldxt, (const T*)h->Wt, h->ldwt, (T*)h->Cpart, d, k, n, h->splits_t, st)) return 1;
        } else if (which == 3) {
            // the whole T half-step (contraction + Gram + exchange + update); collective on row shards
            if (hals_T_half<T>(h, const_cast<T*>(W), Tk, ldtk, &prm, st)) return 1;
        } else if (which == 4) {
            if (hals_W_half<T>(h, const_cast<T*>(W), Tk, ldtk, &prm, true, st)) return 1;
        } else {
            return fail("bad kernel selector %d", which);
        }
    }
    CK(cudaEventRecord(e1, st));
    CK(cudaEventSynchronize(e1));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    CK(cudaEventDestroy(e0));
    CK(cudaEventDestroy(e1));
    CKL();
    *avg_ms = ms / (float)iters;
    return 0;
}

extern "C" int rri_profile_kernel(rri_handle_t h, int32_t which, const void* W_dev, const void* T_dev, int32_t iters,
                                  float* avg_ms_host, void* stream)
{
    if (!h) return fail("null handle");
    if (!h->X) return fail("rri_bind has not been called");
    if (!W_dev || !T_dev || !avg_ms_host || iters <= 0) return fail("bad argument");
    CK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    return h->dtype == RRI_F32 ? profile_impl<float>(h, which, (const float*)W_dev, (const float*)T_dev, iters, avg_ms_host, st)
                               : profile_impl<double>(h, which, (const double*)W_dev, (const double*)T_dev, iters, avg_ms_host, st);
}
