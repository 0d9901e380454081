// sqrn_abi.cu -- kernels + host side of the C ABI declared in include/sqrn.h.
//
// Host responsibilities (everything here is orchestration, none of it scores a
// stem): digest parameter sets into tables, move CSR batches to the GPU, run the
// structure-pool loop of SQRNdbnseq.py:1102-1199 as rounds of batched kernel
// launches, de-duplicate / rank the finished structures (seq.py:1201-1224) and
// hand back caller-owned buffers.
#include <cuda_runtime.h>
#include <pthread.h>
#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <string>
#include <unordered_map>
#include <vector>
#include "sqrn_params.h"
#include "sqrn_nussinov.cuh"
#include "sqrn_hungarian.cuh"
#include "sqrn_edmonds.cuh"

using namespace sqrn;

// ------------------------------------------------------------------ kernel
// Persistent teams pull work items from a global counter (length-sorted by the
// host, longest first), so a batch of mixed lengths keeps every SM busy.
template <class C>
__device__ __forceinline__ void work_loop(const DevParams *__restrict__ Pg, const DevBatch &B, const DevWork &Wk,
                                          const Layout &L, unsigned char *smem)
{
    constexpr int TW = C::TW;
    __shared__ DevParams Psh;
    {
        const int *src = reinterpret_cast<const int *>(Pg);
        int *dst = reinterpret_cast<int *>(&Psh);
        #pragma unroll 1
        for (int k = threadIdx.x; k < (int)(sizeof(DevParams) / 4); k += blockDim.x) dst[k] = src[k];
    }
    __syncthreads();
    const int team = (TW == 1) ? (threadIdx.x >> 5) : 0;
    State S = bind_state(smem + (size_t)team * L.total, L);
    if (TW > 1 && !C::PERSIST) {
        // the two staging barriers of the base-list sweep (team_scan): one arrival each, the elected producer's
        if (threadIdx.x == 0) { mbar_init(S.stage, 1); mbar_init(S.stage + 8, 1); mbar_fence_init(); }
        __syncthreads();
    }
    const int n_items = Wk.n_items_dev ? *Wk.n_items_dev : Wk.n_items;
    for (;;) {
        int item = 0;
        if (TW == 1) {
            if ((threadIdx.x & 31) == 0) item = atomicAdd(Wk.counter, 1);
            item = __shfl_sync(0xffffffffu, item, 0);
        } else {
            if (threadIdx.x == 0) S.misc[1] = atomicAdd(Wk.counter, 1);
            __syncthreads();
            item = S.misc[1];
            __syncthreads();
        }
        if (item >= n_items) break;
        item = Wk.order ? Wk.order[item] : item + Wk.item_base;
        team_run_item<C>(S, Psh, B, Wk, L, item);
    }
}

// Cluster flavour for a FEW LONG sequences (rRNA scale): one thread-block cluster per sequence.
// Each CTA (1024 threads) holds a full replica of the sequence state -- bit masks, partners, stems:
// tens of KB, the N x N matrices never exist -- and scans every CS-th anti-diagonal; the per-CTA
// winners are exchanged through distributed shared memory (cluster_best) and every replica applies
// the same stem.  Rank 0 fetches the work items and writes the results.
// GL: the cluster shares ONE global candidate list (gl_build / gl_step): its CTAs take anti-diagonals (build) and
// record chunks (sweeps) from counters in global memory and meet through the same DSMEM exchange twice per step.
template <bool PLAIN, bool STDP, bool GL = false>
__global__ void __launch_bounds__(1024, 1)
k_cluster(const DevParams *__restrict__ Pg, DevBatch B, DevWork Wk, Layout L)
{
    namespace cg = cooperative_groups;
    using C = Cfg<32, PLAIN, STDP, MODE_TAIL, -1, true, GL>;
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ DevParams Psh;
    {
        const int *src = reinterpret_cast<const int *>(Pg);
        int *dst = reinterpret_cast<int *>(&Psh);
        for (int k = threadIdx.x; k < (int)(sizeof(DevParams) / 4); k += blockDim.x) dst[k] = src[k];
    }
    __syncthreads();
    cg::cluster_group cl = cg::this_cluster();
    const unsigned cr = cl.block_rank(), cs = cl.num_blocks();
    State S = bind_state(smem, L);
    S.dstride = (int)cs; S.doffset = (int)cr;
    cl.sync();                              // every CTA of the cluster is resident before anyone writes into its shared memory
    for (;;) {
        if (cr == 0 && threadIdx.x == 0) {
            int it = atomicAdd(Wk.counter, 1);
            for (unsigned q = 0; q < cs; q++) *cl.map_shared_rank(&S.misc[1], q) = it;      // DSMEM broadcast
        }
        cl.sync();
        int item = S.misc[1];
        cl.sync();                          // everyone has read it before rank 0 may overwrite it
        if (item >= Wk.n_items) break;
        item = Wk.order ? Wk.order[item] : item + Wk.item_base;
        team_run_item<C>(S, Psh, B, Wk, L, item);
    }
}

// general flavour: any batch, any mode, shared-memory layout chosen per launch
template <int TW>
__global__ void __launch_bounds__(TW == 1 ? 256 : TW * 32, TW == 1 ? 3 : 1)
k_work(const DevParams *__restrict__ Pg, DevBatch B, DevWork Wk, Layout L)
{
    extern __shared__ __align__(16) unsigned char smem[];
    work_loop<Cfg<TW>>(Pg, B, Wk, L, smem);
}

// Long sequences, run to completion (MODE_TAIL): CTA teams over the persistent candidate list in
// global memory (gl_build / gl_step): one enumeration per sequence, cached adjusted scores.  Items
// whose list overflows its slot go to DevWork::ovf_list and are redone by k_work<TW> behind it.
template <int TW, bool SIMPLE = false>
__global__ void __launch_bounds__(TW * 32, TW == 8 ? 4 : 1)
k_long(const DevParams *__restrict__ Pg, DevBatch B, DevWork Wk, Layout L)
{
    extern __shared__ __align__(16) unsigned char smem[];
    work_loop<Cfg<TW, false, false, MODE_TAIL, -1, false, true, SIMPLE ? 2 : -1>>(Pg, B, Wk, L, smem);
}

// Fast lane (`byseq pl=1` shape): one warp per sequence, plain sequences (no reactivities,
// restraints, alignment weights), the standard {GC, AU, GU} pairing table, single-path greedy to
// completion.  The shared-memory layout is a compile-time constant, so every array address is
// "team base + immediate" and the code stays small enough for the instruction cache.
constexpr int FAST_TEAMS = 8, FAST_CCAP = 128, FAST_RCAP = 256;
// persistent run list: ~0.003 N^2 entries on random RNA with minlen 4 (measured; DESIGN.md)
__host__ __device__ constexpr int fast_pcap(int ncap) { return ncap <= 128 ? 128 : ncap <= 224 ? 272 : 448; }
template <int NCAP> __host__ __device__ constexpr Layout fast_layout()
{
    return make_layout(NCAP, 0, FAST_CCAP, 4, 1, FAST_RCAP, -1, 0, NCAP / 4 + 2, fast_pcap(NCAP), 2);
}
template <int NCAP> __host__ __device__ constexpr Layout rescan_layout()
{
    return make_layout(NCAP, 0, FAST_CCAP, 4, 1, FAST_RCAP, -1, 0, NCAP / 4 + 2, 0, 2);
}
template <int NCAP, int IO = 1>
__global__ void __launch_bounds__(32 * FAST_TEAMS, 4)
k_fast(const DevParams *__restrict__ Pg, DevBatch B, DevWork Wk)
{
    extern __shared__ __align__(16) unsigned char smem[];
    constexpr Layout L = fast_layout<NCAP>();
    work_loop<Cfg<1, true, true, MODE_TAIL, -1, false, true, -1, IO>>(Pg, B, Wk, L, smem);
}
// The same lane without the persistent run list: every greedy step re-enumerates the anti-diagonals.
// Runs behind k_fast on the items whose list overflowed (DevWork::ovf_list), normally none.
template <int NCAP>
__global__ void __launch_bounds__(32 * FAST_TEAMS, 4)
k_fast_rescan(const DevParams *__restrict__ Pg, DevBatch B, DevWork Wk)
{
    extern __shared__ __align__(16) unsigned char smem[];
    constexpr Layout L = rescan_layout<NCAP>();
    work_loop<Cfg<1, true, true, MODE_TAIL>>(Pg, B, Wk, L, smem);          // (either boundary format, decided at run time)
}

// ----------------------------------------------------------------- context
struct DBuf {
    void *p = nullptr; size_t cap = 0;
    cudaError_t ensure(size_t n)
    {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = n + n / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

constexpr int FAST_MAX_CHUNKS = 20;

struct PEntry {
    sqrn_paramset ps; int nmax; DevParams hp; DevParams *d_p; double *d_lut;
};

struct Stem3 { int32_t i, j, len; };

struct CachedResult {           // result of the last sqrn_predict_batch, kept for the E_CAPACITY retry
    bool valid = false;
    int64_t n_seqs = 0, total_len = 0;
    std::vector<int64_t> struct_offsets, stem_offsets, dbn_offsets;
    std::vector<double> scores; std::vector<uint8_t> isint0; std::vector<uint64_t> psmask;
    std::vector<int32_t> n_total, stems; std::vector<int8_t> dbn, cons;
};
struct CachedStems {
    bool valid = false; int64_t n_seqs = 0;
    std::vector<int64_t> off; std::vector<int32_t> stems; std::vector<double> scores;
};

enum { B_OFF, B_OFF32, B_SYM, B_RCODE, B_RVALS, B_RFPOS, B_RFNEG, B_RCLASS, B_RBOFF, B_RB, B_SMAT, B_COLS, B_BPP, B_BPPOFF,
       W_ORDER, W_ISEQ, W_IOFF, W_ISTEMS, W_SUBOPT, W_COUNTER, W_OOFF, W_OSTEMS, W_ON, W_OFIN, W_ORAW,
       W_OFLAGS, W_DOFF, W_DBNA, W_DBNC, W_NCALLS, W_OVF, W_GENT, W_GBPS, W_GQB, W_GCNT, W_GCNT2, W_GSTAT, W_OVF2, W_RNDC, W_RNDL, W_BASE, W_BASEOFF, W_BASEN, W_BASEBEND, W_MAT, W_CELLCNT, W_CELLS, W_CELLS2,
       NU_COLPTR, NU_PK, NU_PE, NU_ORDER, NU_OUTBASE, NU_OUTP, NU_OUTN, NU_CNT,
       HU_ROWPTR, HU_ACOL, HU_ACOST, HU_ORDER, HU_OUTBASE, HU_OUTP, HU_OUTN, HU_CNT,
       ED_VBASE, ED_EBASE, ED_ROWPTR, ED_POS, ED_ADJ, ED_EP, ED_WT, ED_MAXW, ED_ORDER, ED_OUTBASE, ED_OUTP, ED_OUTN, ED_CNT, NBUF };

// ------------------------------------------------------------- launch plan
struct Plan { int tw, threads, tpc, grid; size_t smem; Layout L; int fast_ncap = 0; int cluster = 0; bool cl_plain = false;
              size_t smem_rescan = 0; int grid_rescan = 0;
              bool glist = false; Layout Lg; size_t smem_g = 0; int grid_g = 0; long long gcap = 0; int grid_classic = 0; };

struct sqrn_ctx {
    int device = 0;
    cudaStream_t stream = nullptr; bool own_stream = false;
    cudaStream_t s_in = nullptr, s_out = nullptr, s_k2 = nullptr;       // copy-in, copy-out, second kernel stream
    cudaEvent_t ev0 = nullptr, ev1 = nullptr; bool ev_valid = false;
    cudaEvent_t ev_start = nullptr, ev_out = nullptr, ev_k2done = nullptr;
    cudaEvent_t ev_in[FAST_MAX_CHUNKS] = {}, ev_k0[FAST_MAX_CHUNKS] = {}, ev_k1[FAST_MAX_CHUNKS] = {}, ev_o[FAST_MAX_CHUNKS] = {};
    cudaEvent_t ev_l0[FAST_MAX_CHUNKS] = {}, ev_l1[FAST_MAX_CHUNKS] = {};   // the CTA-team launch of a chunk of mixed lengths
    uint8_t *hflags = nullptr; size_t hflags_cap = 0;                    // pinned staging for the result flags
    int32_t *horder = nullptr; size_t horder_cap = 0;                   // pinned: processing order of the fast-lane chunks
    Plan fast_plans[3]; bool fast_plan_ok[3] = {false, false, false};   // the three length classes of the fast kernels
    std::string err;
    int sm_count = 0; size_t smem_optin = 0;
    std::vector<PEntry> pcache;
    DBuf buf[NBUF];
    int64_t n_launches = 0, n_calls = 0; double kernel_ms = 0.0;
    int region_mode = REGION_AUTO;
    int no_fast_kernel = 0;      // tuning knob: route the fast lane through the general kernel
    int no_cluster = 0, force_cluster = 0;   // tuning knobs: never / always (with this size) use k_cluster for long sequences
    int64_t n_cluster_launches = 0, n_glist_launches = 0;
    int no_glist = 0;            // tuning knob: CTA teams rescan every step (no global persistent list)
    int gl_rebuild = 0;          // tuning knob: rebuild period of the binned global list in passes (0: the default)
    CachedResult cres; CachedStems cstems;
    void *nu_ws = nullptr; size_t nu_ws_bytes = 0;   // workspace of sqrn_nussinov_batch (exact size, grown on demand)
    void *hu_ws = nullptr; size_t hu_ws_bytes = 0;   // global-tier slots of sqrn_hungarian_batch (grown on demand)
    void *ed_ws = nullptr; size_t ed_ws_bytes = 0;   // team slots of sqrn_edmonds_batch (grown on demand)
};

static std::string g_create_err;

#define TRY(x) do { int r_ = (x); if (r_ != SQRN_OK) return r_; } while (0)
#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { \
    ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_); return SQRN_E_CUDA; } } while (0)

// No exception crosses the C boundary: host allocation failures inside an entry point come back as SQRN_E_NOMEM.
template <class F>
static int guarded(sqrn_ctx *ctx, F &&body)
{
    try { return body(); }
    catch (const std::bad_alloc &) { if (ctx) ctx->err = "out of host memory"; return SQRN_E_NOMEM; }
    catch (const std::exception &e) { if (ctx) ctx->err = std::string("internal error: ") + e.what(); return SQRN_E_NOMEM; }
    catch (...) { if (ctx) ctx->err = "internal error"; return SQRN_E_NOMEM; }
}

extern "C" int sqrn_abi_version(void) { return SQRN_ABI_VERSION; }

extern "C" int sqrn_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

extern "C" const char *sqrn_last_error(const sqrn_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

extern "C" int sqrn_ctx_create(int device, sqrn_ctx **out)
{
    if (!out) return SQRN_E_BADARG;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        g_create_err = std::string("no usable CUDA device (libsqrn_b200 has no CPU fallback): ") + cudaGetErrorString(e);
        cudaGetLastError();
        return SQRN_E_CUDA;
    }
    if (device < 0 || device >= n) { g_create_err = "device index out of range"; return SQRN_E_BADARG; }
    sqrn_ctx *ctx = new sqrn_ctx();
    ctx->device = device;
    if ((e = cudaSetDevice(device)) != cudaSuccess ||
        (e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess ||
        (e = cudaEventCreate(&ctx->ev0)) != cudaSuccess || (e = cudaEventCreate(&ctx->ev1)) != cudaSuccess) {
        g_create_err = std::string("context creation failed: ") + cudaGetErrorString(e);
        delete ctx; return SQRN_E_CUDA;
    }
    ctx->own_stream = true;
    bool ok = cudaStreamCreateWithFlags(&ctx->s_in, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&ctx->s_out, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&ctx->s_k2, cudaStreamNonBlocking) == cudaSuccess &&
              cudaEventCreateWithFlags(&ctx->ev_start, cudaEventDisableTiming) == cudaSuccess &&
              cudaEventCreateWithFlags(&ctx->ev_out, cudaEventDisableTiming) == cudaSuccess &&
              cudaEventCreateWithFlags(&ctx->ev_k2done, cudaEventDisableTiming) == cudaSuccess;
    for (int c = 0; c < FAST_MAX_CHUNKS && ok; c++)
        ok = cudaEventCreateWithFlags(&ctx->ev_in[c], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreate(&ctx->ev_k0[c]) == cudaSuccess && cudaEventCreate(&ctx->ev_k1[c]) == cudaSuccess &&
             cudaEventCreate(&ctx->ev_l0[c]) == cudaSuccess && cudaEventCreate(&ctx->ev_l1[c]) == cudaSuccess &&
             cudaEventCreateWithFlags(&ctx->ev_o[c], cudaEventDisableTiming) == cudaSuccess;
    if (!ok) { g_create_err = std::string("context creation failed: ") + cudaGetErrorString(cudaGetLastError()); delete ctx; return SQRN_E_CUDA; }
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    if (const char *e = getenv("SQRN_GL_REBUILD")) ctx->gl_rebuild = std::max(0, atoi(e));      // experiment knob (SQRN_TUNE_GL_REBUILD)
    *out = ctx;
    return SQRN_OK;
}

extern "C" void sqrn_ctx_destroy(sqrn_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (auto &b : ctx->buf) b.release();
    for (auto &p : ctx->pcache) { cudaFree(p.d_p); cudaFree(p.d_lut); }
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    cudaStreamDestroy(ctx->s_in); cudaStreamDestroy(ctx->s_out); cudaStreamDestroy(ctx->s_k2);
    cudaEventDestroy(ctx->ev0); cudaEventDestroy(ctx->ev1);
    cudaEventDestroy(ctx->ev_start); cudaEventDestroy(ctx->ev_out); cudaEventDestroy(ctx->ev_k2done);
    for (int c = 0; c < FAST_MAX_CHUNKS; c++) { cudaEventDestroy(ctx->ev_in[c]); cudaEventDestroy(ctx->ev_k0[c]); cudaEventDestroy(ctx->ev_k1[c]); cudaEventDestroy(ctx->ev_o[c]); cudaEventDestroy(ctx->ev_l0[c]); cudaEventDestroy(ctx->ev_l1[c]); }
    if (ctx->hflags) cudaFreeHost(ctx->hflags);
    if (ctx->horder) cudaFreeHost(ctx->horder);
    if (ctx->nu_ws) cudaFree(ctx->nu_ws);
    if (ctx->hu_ws) cudaFree(ctx->hu_ws);
    if (ctx->ed_ws) cudaFree(ctx->ed_ws);
    delete ctx;
}

extern "C" int sqrn_ctx_set_stream(sqrn_ctx *ctx, void *cuda_stream)
{
    if (!ctx) return SQRN_E_BADARG;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    ctx->stream = (cudaStream_t)cuda_stream; ctx->own_stream = false;
    return SQRN_OK;
}

extern "C" int sqrn_ctx_set_tuning(sqrn_ctx *ctx, int what, int value)
{
    if (!ctx) return SQRN_E_BADARG;
    if (what == SQRN_TUNE_REGION && value >= 0 && value <= 2) { ctx->region_mode = value; return SQRN_OK; }
    if (what == SQRN_TUNE_NO_FAST_KERNEL) { ctx->no_fast_kernel = value != 0; return SQRN_OK; }
    if (what == SQRN_TUNE_NO_GLIST) { ctx->no_glist = value != 0; return SQRN_OK; }
    if (what == SQRN_TUNE_GL_REBUILD && value >= 0) { ctx->gl_rebuild = value; return SQRN_OK; }
    if (what == SQRN_TUNE_CLUSTER && (value == 0 || value == 1 || value == 2 || value == 4 || value == 8 || value == 16)) {
        ctx->no_cluster = value == 1; ctx->force_cluster = value > 1 ? value : 0; return SQRN_OK;   // 0 automatic, 1 never, 2..16 always
    }
    ctx->err = "unknown tuning knob";
    return SQRN_E_BADARG;
}

extern "C" int sqrn_ctx_last_stats(const sqrn_ctx *ctx, int64_t *n_launches, double *kernel_ms, int64_t *n_optimal_calls)
{
    if (!ctx) return SQRN_E_BADARG;
    if (n_launches) *n_launches = ctx->n_launches;
    if (kernel_ms) *kernel_ms = ctx->kernel_ms;
    if (n_optimal_calls) *n_optimal_calls = ctx->n_calls;
    return SQRN_OK;
}

// parameter-set digest, cached per (paramset, length class)
static int get_params(sqrn_ctx *ctx, const sqrn_paramset &ps, int nmax, const PEntry **out)
{
    for (auto &e : ctx->pcache)
        if (e.nmax >= nmax && !memcmp(&e.ps, &ps, sizeof ps)) { *out = &e; return SQRN_OK; }
    int ncap = (nmax + 1023) / 1024 * 1024;
    HostParams H;
    if (!build_host_params(ps, ncap, H, ctx->err)) return SQRN_E_UNSUPPORTED;
    PEntry e; memcpy(&e.ps, &ps, sizeof ps); e.nmax = ncap; e.d_p = nullptr; e.d_lut = nullptr;
    CK(cudaMalloc(&e.d_lut, H.lut.size() * sizeof(double)));
    CK(cudaMalloc(&e.d_p, sizeof(DevParams)));
    H.p.sdf_lut = e.d_lut + H.sdf_off; H.p.of_lut = e.d_lut + H.of_off; H.p.pw17_lut = e.d_lut + H.pw17_off;
    e.hp = H.p;
    CK(cudaMemcpy(e.d_lut, H.lut.data(), H.lut.size() * sizeof(double), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(e.d_p, &H.p, sizeof(DevParams), cudaMemcpyHostToDevice));
    ctx->pcache.push_back(e);
    *out = &ctx->pcache.back();
    return SQRN_OK;
}

// ------------------------------------------------------------- launch plan
static int next_pow2(int x) { int p = 1; while (p < x) p <<= 1; return p; }

template <int TW>
static int plan_for(sqrn_ctx *ctx, Plan &pl)
{
    CK(cudaFuncSetAttribute(k_work<TW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
    int nb = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_work<TW>, pl.threads, pl.smem));
    if (nb < 1) { ctx->err = "kernel does not fit on an SM"; return SQRN_E_UNSUPPORTED; }
    pl.grid = nb * ctx->sm_count;
    return SQRN_OK;
}

// choose the team shape for sequences up to nmax symbols.  keep_all: the mode needs every
// survivor of a scan in the list (MODE_STEP); otherwise the lists are flushed when they fill up
// and their sizes only set the flush granularity.
// small_lists: the items sweep a base list (only in-range survivors stay in the list between flushes).
static int make_plan(sqrn_ctx *ctx, const PEntry &P, int nmax, int rbmax, int min_ccap, bool keep_all, bool extras,
                     int max_init, Plan &pl, bool small_lists = false)
{
    const int m = P.hp.m, npc = P.hp.npc;
    // every stem the greedy adds has >= m pairs (AnnotateStems' minlen filter, seq.py:492); max_init < 0: unknown
    const int scap = max_init < 0 ? 0 : max_init + nmax / (2 * m) + 2;
    double dens = m >= 4 ? 0.004 : (m == 3 ? 0.01 : 0.025);         // candidate stems / N^2 on random RNA
    int est = (int)(dens * nmax * (double)nmax) + 32;
    const size_t budget = ctx->smem_optin - sizeof(DevParams) - 1024;
    if (nmax <= 320 && min_ccap <= 1024) {
        pl.tw = 1;
        int ccap = keep_all ? std::max(std::min(next_pow2(est), 1024), 64) : 128;
        if (ccap < min_ccap) ccap = next_pow2(min_ccap);
        pl.L = make_layout(nmax, rbmax, ccap, npc, 1, 256, extras, keep_all, scap);
        pl.tpc = (int)std::max<size_t>(1, std::min<size_t>(8, (96 * 1024) / pl.L.total));
        pl.threads = 32 * pl.tpc;
        pl.smem = (size_t)pl.tpc * pl.L.total;
        return plan_for<1>(ctx, pl);
    }
    pl.tw = nmax <= 2048 ? 8 : 32;
    // at least two rounds of survivors (one per thread and round) must fit between flushes
    int ccap = keep_all ? std::max(std::min(next_pow2(est), 4096), 1024 * (pl.tw / 8)) : (pl.tw == 8 ? 2048 : 8192);
    if (small_lists) ccap = 1024 * (pl.tw / 8);             // (more CTAs per SM; an item whose window holds more is redone with min_ccap)
    if (ccap < min_ccap) ccap = next_pow2(min_ccap);
    for (;;) {
        pl.L = make_layout(nmax, rbmax, ccap, npc, pl.tw, 4096, extras, keep_all, scap);
        if ((size_t)pl.L.total <= budget || ccap <= 64 * pl.tw) break;
        ccap >>= 1;
    }
    if ((size_t)pl.L.total > budget) { ctx->err = "sequence too long for one CTA's shared memory"; return SQRN_E_UNSUPPORTED; }
    pl.tpc = 1; pl.threads = 32 * pl.tw; pl.smem = pl.L.total;
    return pl.tw == 8 ? plan_for<8>(ctx, pl) : plan_for<32>(ctx, pl);
}

// CTA teams in MODE_TAIL: plan the global-list kernel next to the rescanning one (which stays as its fallback)
template <int TW>
static int plan_glist_t(sqrn_ctx *ctx, Plan &pl)
{
    CK(cudaFuncSetAttribute(k_long<TW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem_g));
    if (TW == 8) CK(cudaFuncSetAttribute(k_long<8, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem_g));
    int nb = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_long<TW>, TW * 32, pl.smem_g));
    if (nb < 1) return SQRN_E_UNSUPPORTED;
    if (const char *e = getenv("SQRN_LONG_PER_SM")) nb = std::max(1, std::min(nb, atoi(e)));      // experiment: fewer resident CTAs
    pl.grid_g = nb * ctx->sm_count;
    return SQRN_OK;
}

static void maybe_glist(sqrn_ctx *ctx, const PEntry &P, Plan &pl, int nmax, int rbmax, bool extras, int max_init, bool tail_mode)
{
    if (pl.tw == 1 || !tail_mode || ctx->no_glist || !P.hp.ub_ok || !(P.hp.loopbonus >= 0.0) || nmax > 32767) return;
    const int m = P.hp.m;
    const int scap = max_init < 0 ? 0 : max_init + nmax / (2 * m) + 2;
    pl.Lg = make_layout(nmax, rbmax, 128 * pl.tw, P.hp.npc, pl.tw, 64, extras, 0, scap, -1);   // Ccap: 2 x 64 list slots per warp
    pl.smem_g = pl.Lg.total;
    if (pl.smem_g + sizeof(DevParams) + 1024 > ctx->smem_optin) return;
    if ((pl.tw == 8 ? plan_glist_t<8>(ctx, pl) : plan_glist_t<32>(ctx, pl)) != SQRN_OK) { cudaGetLastError(); return; }
    // entries per slot: runs whose positive part reaches minbpscore, ~0.02 N^2 for minlen 2 on random RNA (DESIGN.md)
    const double dens = m >= 4 ? 0.003 : (m == 3 ? 0.008 : 0.02);
    pl.gcap = (long long)(1.5 * dens * nmax * (double)nmax) + 4096;
    // a slot is two halves of gcap records (16-byte record + bp score + bin = 25 bytes); at most ~16 GB of list
    // space: fewer resident CTAs rather than smaller slots
    const long long budget = 16ll << 30;
    if (pl.gcap * 50 * pl.grid_g > budget) pl.grid_g = (int)std::max<long long>(1, budget / (pl.gcap * 50));
    pl.glist = true;
}

// the compile-time-layout fast kernel, when the parameter set and the lengths allow it
template <int NCAP>
static int plan_fast(sqrn_ctx *ctx, Plan &pl)
{
    constexpr Layout L = fast_layout<NCAP>();
    pl.tw = 1; pl.tpc = FAST_TEAMS; pl.threads = 32 * FAST_TEAMS; pl.L = L; pl.smem = (size_t)FAST_TEAMS * L.total;
    pl.fast_ncap = NCAP;
    CK(cudaFuncSetAttribute(k_fast<NCAP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
    CK(cudaFuncSetAttribute(k_fast<NCAP, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
    int nb = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_fast<NCAP>, pl.threads, pl.smem));
    if (nb < 1) { ctx->err = "kernel does not fit on an SM"; return SQRN_E_UNSUPPORTED; }
    pl.grid = nb * ctx->sm_count;
    constexpr Layout L2 = rescan_layout<NCAP>();
    pl.smem_rescan = (size_t)FAST_TEAMS * L2.total;
    CK(cudaFuncSetAttribute(k_fast_rescan<NCAP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem_rescan));
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_fast_rescan<NCAP>, pl.threads, pl.smem_rescan));
    if (nb < 1) { ctx->err = "kernel does not fit on an SM"; return SQRN_E_UNSUPPORTED; }
    pl.grid_rescan = nb * ctx->sm_count;
    return SQRN_OK;
}

static void maybe_cluster(sqrn_ctx *ctx, const PEntry &P, Plan &pl, int n_items, bool plain, bool tail_mode);

static bool fast_eligible(const PEntry &P, int nmax) { return P.hp.std_pairs && P.hp.m >= 2 && nmax <= 320; }

static int make_fast_plan(sqrn_ctx *ctx, const PEntry &P, int nmax, int n_items, Plan &pl)
{
    if (fast_eligible(P, nmax) && !ctx->no_fast_kernel) {
        // (the attributes and occupancy of the three length classes are looked up once per context)
        const int cls = nmax <= 128 ? 0 : nmax <= 224 ? 1 : 2;
        if (!ctx->fast_plan_ok[cls]) {
            Plan q;
            TRY(cls == 0 ? plan_fast<128>(ctx, q) : cls == 1 ? plan_fast<224>(ctx, q) : plan_fast<320>(ctx, q));
            ctx->fast_plans[cls] = q; ctx->fast_plan_ok[cls] = true;
        }
        pl = ctx->fast_plans[cls];
        return SQRN_OK;
    }
    TRY(make_plan(ctx, P, nmax, 0, 0, false, false, 0, pl));
    maybe_glist(ctx, P, pl, nmax, 0, false, 0, true);
    maybe_cluster(ctx, P, pl, n_items, true, true);
    return SQRN_OK;
}

// Few long sequences: give each one a thread-block cluster instead of a single CTA (k_cluster).
// n_items = work items of the launch; plain = no reactivities / restraints / smat / interchainonly.
template <bool PLAIN, bool STDP, bool GL = false>
static int plan_cluster_t(sqrn_ctx *ctx, Plan &pl, int cs)
{
    auto kern = k_cluster<PLAIN, STDP, GL>;
    const size_t smem = GL ? pl.smem_g : pl.smem;
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(cs * ctx->sm_count)); cfg.blockDim = dim3(1024); cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = (unsigned)cs; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int ncl = 0;
    cudaError_t e = cudaOccupancyMaxActiveClusters(&ncl, kern, &cfg);
    if (e != cudaSuccess || ncl < 1) { cudaGetLastError(); return SQRN_E_UNSUPPORTED; }
    pl.cluster = cs; pl.grid = ncl;          // grid counts clusters here
    return SQRN_OK;
}

static void maybe_cluster(sqrn_ctx *ctx, const PEntry &P, Plan &pl, int n_items, bool plain, bool tail_mode)
{
    if (pl.tw != 32 || !tail_mode || ctx->no_cluster || n_items < 1) return;
    int want = ctx->force_cluster;
    if (!want) {
        if (2 * n_items > ctx->sm_count) return;             // enough sequences to fill the SMs one CTA each
        want = 8;
        while (want > 2 && want * n_items > ctx->sm_count) want >>= 1;
    }
    pl.cl_plain = plain && P.hp.std_pairs;
    pl.grid_classic = pl.grid;
    for (int cs = want; cs >= 2; cs >>= 1) {
        // with a global candidate list planned (k_long), the cluster shares one list; else it rescans
        int rc = pl.glist && pl.tw == 32 ? plan_cluster_t<false, false, true>(ctx, pl, cs)
               : pl.cl_plain ? plan_cluster_t<true, true>(ctx, pl, cs) : plan_cluster_t<false, false>(ctx, pl, cs);
        if (rc == SQRN_OK) return;
    }
    pl.cluster = 0;
}

template <class T>
static int upload(sqrn_ctx *ctx, int slot, const T *h, size_t count, T **d)
{
    CK(ctx->buf[slot].ensure(std::max<size_t>(count, 1) * sizeof(T)));
    *d = (T *)ctx->buf[slot].p;
    if (count) CK(cudaMemcpyAsync(*d, h, count * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
    return SQRN_OK;
}
template <class T>
static int dalloc(sqrn_ctx *ctx, int slot, size_t count, T **d)
{
    CK(ctx->buf[slot].ensure(std::max<size_t>(count, 1) * sizeof(T)));
    *d = (T *)ctx->buf[slot].p;
    return SQRN_OK;
}

// one launch of the work kernel the plan names
static int dispatch(sqrn_ctx *ctx, const PEntry &P, const Plan &pl, cudaStream_t st, const DevBatch &B, const DevWork &W)
{
    static const bool glist_init = getenv("SQRN_GLIST_INIT") != nullptr;       // experiment: the list also for pool tails
    const bool use_glist = pl.glist && W.mode == MODE_TAIL && (!W.init_off || glist_init);
    if (pl.cluster && use_glist && pl.tw == 32) {
        // a thread-block cluster per sequence over ONE shared candidate list; overflowed items go to k_work<32> behind it
        const int ncl = std::min(pl.grid, std::max(W.n_items, 1));
        GEnt *ge; double *gb; uint8_t *gq; int32_t *ovf; int *cnt, *gcnt;
        TRY(dalloc(ctx, W_GENT, (size_t)2 * ncl * pl.gcap, &ge));
        TRY(dalloc(ctx, W_GBPS, (size_t)2 * ncl * pl.gcap, &gb));
        TRY(dalloc(ctx, W_GQB, (size_t)2 * ncl * pl.gcap, &gq));
        TRY(dalloc(ctx, W_OVF2, (size_t)W.n_items, &ovf));      // not W_OVF: fast-lane chunks on the other stream use that one
        TRY(dalloc(ctx, W_GCNT, 4, &cnt));
        TRY(dalloc(ctx, W_GCNT2, (size_t)GL_CNT_INTS * ncl, &gcnt));
        CK(cudaMemsetAsync(cnt, 0, 4 * sizeof(int), st));
        CK(cudaMemsetAsync(gcnt, 0, (size_t)GL_CNT_INTS * ncl * sizeof(int), st));
        DevWork W1 = W; W1.g_ent = ge; W1.g_bps = gb; W1.g_qb = gq; W1.g_cap = pl.gcap; W1.g_cnt = gcnt; W1.g_rebuild = ctx->gl_rebuild;
        W1.ovf_count = cnt; W1.ovf_list = ovf;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(ncl * pl.cluster)); cfg.blockDim = dim3(1024); cfg.dynamicSmemBytes = pl.smem_g; cfg.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = (unsigned)pl.cluster; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        const DevParams *dp = P.d_p;
        CK(cudaLaunchKernelEx(&cfg, k_cluster<false, false, true>, dp, B, W1, pl.Lg));
        DevWork W2 = W; W2.order = ovf; W2.n_items_dev = cnt; W2.counter = cnt + 1;
        int g2 = pl.grid_classic > 0 ? pl.grid_classic : ctx->sm_count;
        k_work<32><<<g2, pl.threads, pl.smem, st>>>(P.d_p, B, W2, pl.L);
        CK(cudaGetLastError());
        ctx->n_launches++; ctx->n_cluster_launches++; ctx->n_glist_launches++;
        return SQRN_OK;
    }
    if (pl.cluster) {
        int ncl = std::min(pl.grid, std::max(W.n_items, 1));
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(ncl * pl.cluster)); cfg.blockDim = dim3(1024); cfg.dynamicSmemBytes = pl.smem; cfg.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = (unsigned)pl.cluster; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        const DevParams *dp = P.d_p;
        if (pl.cl_plain) CK(cudaLaunchKernelEx(&cfg, k_cluster<true, true>, dp, B, W, pl.L));
        else CK(cudaLaunchKernelEx(&cfg, k_cluster<false, false>, dp, B, W, pl.L));
        ctx->n_cluster_launches++;
        return SQRN_OK;
    }
    int grid = pl.grid;
    int teams = (W.n_items + pl.tpc - 1) / pl.tpc;
    if (grid > teams) grid = std::max(teams, 1);
    if (use_glist) {       // items with pre-selected stems (pool tails) have few steps left: they rescan
        const int gg = std::max(1, std::min(pl.grid_g, W.n_items));
        GEnt *ge; double *gb; uint8_t *gq; int32_t *ovf; int *cnt;
        TRY(dalloc(ctx, W_GENT, (size_t)2 * gg * pl.gcap, &ge));
        TRY(dalloc(ctx, W_GBPS, (size_t)2 * gg * pl.gcap, &gb));
        TRY(dalloc(ctx, W_GQB, (size_t)2 * gg * pl.gcap, &gq));
        TRY(dalloc(ctx, W_OVF2, (size_t)W.n_items, &ovf));      // not W_OVF: fast-lane chunks on the other stream use that one
        TRY(dalloc(ctx, W_GCNT, 4, &cnt));
        CK(cudaMemsetAsync(cnt, 0, 4 * sizeof(int), st));
        DevWork W1 = W; W1.g_ent = ge; W1.g_bps = gb; W1.g_qb = gq; W1.g_cap = pl.gcap; W1.g_rebuild = ctx->gl_rebuild;
        const bool trace = getenv("SQRN_TRACE") != nullptr;
        unsigned long long *d_stat = nullptr;
        if (trace) { TRY(dalloc(ctx, W_GSTAT, 16, &d_stat)); CK(cudaMemsetAsync(d_stat, 0, 16 * sizeof(unsigned long long), st)); W1.g_stat = d_stat; }
        W1.ovf_count = cnt; W1.ovf_list = ovf;
        // (lists of a few thousand records -- 256-thread CTAs on parameter sets with minlen >= 3, or short sequences: the
        //  flavour that sweeps the whole list every pass; its smaller code keeps four CTAs per SM inside the instruction cache)
        static const bool no_simple = getenv("SQRN_NO_LONG_SIMPLE") != nullptr;
        if (pl.tw == 8 && !no_simple && pl.gcap <= 24576) k_long<8, true><<<gg, 256, pl.smem_g, st>>>(P.d_p, B, W1, pl.Lg);
        else if (pl.tw == 8) k_long<8><<<gg, 256, pl.smem_g, st>>>(P.d_p, B, W1, pl.Lg);
        else k_long<32><<<gg, 1024, pl.smem_g, st>>>(P.d_p, B, W1, pl.Lg);
        CK(cudaGetLastError());
        DevWork W2 = W; W2.order = ovf; W2.n_items_dev = cnt; W2.counter = cnt + 1;
        if (pl.tw == 8) k_work<8><<<grid, pl.threads, pl.smem, st>>>(P.d_p, B, W2, pl.L);
        else k_work<32><<<grid, pl.threads, pl.smem, st>>>(P.d_p, B, W2, pl.L);
        CK(cudaGetLastError());
        ctx->n_launches++; ctx->n_glist_launches++;
        if (trace) {
            unsigned long long h[16]; int hc[4];
            CK(cudaStreamSynchronize(st));
            CK(cudaMemcpy(h, d_stat, sizeof h, cudaMemcpyDeviceToHost));
            CK(cudaMemcpy(hc, cnt, sizeof hc, cudaMemcpyDeviceToHost));
            fprintf(stderr, "[sqrn] k_long<%d>: %d items (%d overflowed), %d CTAs x %lld entries; steps %llu (level changes %llu), "
                    "entries swept %llu, evaluations %llu, cache resets %llu, cuts %llu, rebuilds %llu\n", pl.tw, W.n_items, hc[0], gg, pl.gcap,
                    h[3], h[4], h[0], h[1], h[2], h[5], h[12]);
            fprintf(stderr, "[sqrn]   cycles (thread 0, summed over CTAs, M): build %.1f, loop %.1f = levels %.1f + sweep1 %.1f + sweep2 %.1f + apply %.1f + rest\n",
                    h[9] / 1e6, h[8] / 1e6, h[10] / 1e6, h[6] / 1e6, h[7] / 1e6, h[11] / 1e6);
        }
        return SQRN_OK;
    }
    if (pl.fast_ncap) {
        if (!W.ovf_list || !W.ovf_count || !W.n_items_dev) { ctx->err = "fast lane launched without an overflow list"; return SQRN_E_BADARG; }
        DevWork W1 = W; W1.n_items_dev = nullptr;
        if (B.sym_packed) {
            if (pl.fast_ncap == 128) k_fast<128, 2><<<grid, pl.threads, pl.smem, st>>>(P.d_p, B, W1);
            else if (pl.fast_ncap == 224) k_fast<224, 2><<<grid, pl.threads, pl.smem, st>>>(P.d_p, B, W1);
            else k_fast<320, 2><<<grid, pl.threads, pl.smem, st>>>(P.d_p, B, W1);
        }
        else if (pl.fast_ncap == 128) k_fast<128><<<grid, pl.threads, pl.smem, st>>>(P.d_p, B, W1);
        else if (pl.fast_ncap == 224) k_fast<224><<<grid, pl.threads, pl.smem, st>>>(P.d_p, B, W1);
        else k_fast<320><<<grid, pl.threads, pl.smem, st>>>(P.d_p, B, W1);
        CK(cudaGetLastError());
        // the items whose run list overflowed (usually none: the CTAs then leave at once)
        DevWork W2 = W; W2.order = W.ovf_list; W2.counter = W.ovf_count + 1; W2.ovf_list = nullptr; W2.ovf_count = nullptr;
        const int g2 = std::min(grid, pl.grid_rescan);
        if (pl.fast_ncap == 128) k_fast_rescan<128><<<g2, pl.threads, pl.smem_rescan, st>>>(P.d_p, B, W2);
        else if (pl.fast_ncap == 224) k_fast_rescan<224><<<g2, pl.threads, pl.smem_rescan, st>>>(P.d_p, B, W2);
        else k_fast_rescan<320><<<g2, pl.threads, pl.smem_rescan, st>>>(P.d_p, B, W2);
        ctx->n_launches++;
    }
    else if (pl.tw == 1) k_work<1><<<grid, pl.threads, pl.smem, st>>>(P.d_p, B, W, pl.L);
    else if (pl.tw == 8) k_work<8><<<grid, pl.threads, pl.smem, st>>>(P.d_p, B, W, pl.L);
    else k_work<32><<<grid, pl.threads, pl.smem, st>>>(P.d_p, B, W, pl.L);
    CK(cudaGetLastError());
    return SQRN_OK;
}

static int launch(sqrn_ctx *ctx, const PEntry &P, const Plan &pl, const DevBatch &B, DevWork &W)
{
    CK(cudaMemsetAsync(W.counter, 0, sizeof(int), ctx->stream));
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    TRY(dispatch(ctx, P, pl, ctx->stream, B, W));
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    ctx->ev_valid = true;
    ctx->n_launches++;
    return SQRN_OK;
}

// ------------------------------------------------ fast lane (byseq pl=1 shape)
// one launch over items [item_base, item_base + n_items) of a resident CSR batch
// compact device outputs of the packed lane (NULL members: the byte lane)
struct PackedOut { uint8_t *nib = nullptr; int32_t *milli = nullptr; uint16_t *ns16 = nullptr; int *rnd_count = nullptr; double *rnd_list = nullptr; int rnd_cap = 0; };

static int fast_launch(sqrn_ctx *ctx, const PEntry &P, const Plan &pl, cudaStream_t st, int64_t item_base, int64_t n_items,
                       const int64_t *d_offsets, const uint8_t *d_symbols, uint8_t *d_dbn_ascii, double *d_scores,
                       int32_t *d_n_stems, uint8_t *d_flags, int *d_counter, int32_t *d_ovf, unsigned long long *d_ncalls, int round3,
                       cudaEvent_t e0, cudaEvent_t e1, const int32_t *d_order = nullptr, const PackedOut *pk = nullptr, int64_t n_batch = -1)
{
    DevBatch B; memset(&B, 0, sizeof B);
    B.n_seqs = n_batch >= 0 ? n_batch : item_base + n_items; B.off = d_offsets; B.sym = d_symbols; B.sym_packed = pk != nullptr;
    DevWork W; memset(&W, 0, sizeof W);
    W.n_items = (int)n_items; W.item_base = (int)item_base; W.mode = MODE_TAIL; W.region_mode = ctx->region_mode;
    W.round3 = round3; W.counter = d_counter; W.out_flags = d_flags; W.n_calls = d_ncalls;
    if (pl.fast_ncap) {          // [counter, overflow count, counter of the rescanning kernel]; list slots of this item range
        W.ovf_count = d_counter + 1; W.n_items_dev = d_counter + 1; W.ovf_list = d_ovf + item_base;
    }
    W.out_nstems = d_n_stems; W.out_raw = d_scores; W.dbn_off = d_offsets; W.out_dbn_ascii = d_dbn_ascii;
    if (pk) { W.out_dbn_ascii = nullptr; W.out_raw = nullptr; W.out_nstems = nullptr; W.out_dbn_nib = pk->nib; W.out_milli = pk->milli; W.out_ns16 = pk->ns16; W.rnd_count = pk->rnd_count; W.rnd_list = pk->rnd_list; W.rnd_cap = pk->rnd_cap; }
    W.order = d_order;             // absolute item ids, or NULL: items item_base .. item_base + n_items - 1 in order
    if (e0) CK(cudaEventRecord(e0, st));
    TRY(dispatch(ctx, P, pl, st, B, W));
    if (e1) CK(cudaEventRecord(e1, st));
    ctx->n_launches++;
    return SQRN_OK;
}

static int sqrn_fast_predict_device_impl(sqrn_ctx *ctx, const sqrn_paramset *ps, int64_t n_seqs, int64_t total_len,
                                        int32_t max_len, const int64_t *d_offsets, const uint8_t *d_symbols,
                                        uint8_t *d_dbn_ascii, double *d_scores, int32_t *d_n_stems)
{
    if (!ctx || !ps || n_seqs < 0 || n_seqs > 0x7fffffff || max_len > SQRN_MAX_LEN) return SQRN_E_BADARG;
    (void)total_len;
    cudaSetDevice(ctx->device);
    if (n_seqs == 0) return SQRN_OK;
    const PEntry *P;
    TRY(get_params(ctx, *ps, max_len, &P));
    Plan pl;
    TRY(make_fast_plan(ctx, *P, max_len, (int)n_seqs, pl));
    int *d_counter; uint8_t *d_flags; unsigned long long *d_nc;
    int32_t *d_ovf;
    TRY(dalloc(ctx, W_COUNTER, 4 * FAST_MAX_CHUNKS, &d_counter));
    TRY(dalloc(ctx, W_OVF, (size_t)n_seqs, &d_ovf));
    TRY(dalloc(ctx, W_OFLAGS, (size_t)n_seqs, &d_flags));
    TRY(dalloc(ctx, W_NCALLS, 1, &d_nc));
    CK(cudaMemsetAsync(d_counter, 0, 4 * sizeof(int), ctx->stream));
    CK(cudaMemsetAsync(d_nc, 0, sizeof(unsigned long long), ctx->stream));
    int rc = fast_launch(ctx, *P, pl, ctx->stream, 0, n_seqs, d_offsets, d_symbols, d_dbn_ascii, d_scores, d_n_stems,
                         d_flags, d_counter, d_ovf, d_nc, 0, ctx->ev0, ctx->ev1);
    if (rc == SQRN_OK) ctx->ev_valid = true;
    return rc;
}

extern "C" int sqrn_fast_predict_device(sqrn_ctx *ctx, const sqrn_paramset *ps, int64_t n_seqs, int64_t total_len,
                                        int32_t max_len, const int64_t *d_offsets, const uint8_t *d_symbols,
                                        uint8_t *d_dbn_ascii, double *d_scores, int32_t *d_n_stems)
{
    return guarded(ctx, [&] { return sqrn_fast_predict_device_impl(ctx, ps, n_seqs, total_len, max_len, d_offsets, d_symbols, d_dbn_ascii, d_scores, d_n_stems); });
}

static int sqrn_fast_predict_packed_device_impl(sqrn_ctx *ctx, const sqrn_paramset *ps, int64_t n_seqs, int64_t total_len,
                                               int32_t max_len, const int64_t *d_offsets, const uint8_t *d_packed,
                                               uint8_t *d_dbn_nib, int32_t *d_score_milli, uint16_t *d_n_stems, uint8_t *d_flags)
{
    if (!ctx || !ps || !d_score_milli || !d_flags || n_seqs < 0 || n_seqs > 0x7fffffff || max_len > SQRN_MAX_LEN) return SQRN_E_BADARG;
    (void)total_len;
    cudaSetDevice(ctx->device);
    if (n_seqs == 0) return SQRN_OK;
    const PEntry *P;
    TRY(get_params(ctx, *ps, max_len, &P));
    Plan pl;
    TRY(make_fast_plan(ctx, *P, max_len, (int)n_seqs, pl));
    int *d_counter; unsigned long long *d_nc; int32_t *d_ovf; int *d_rnd; PackedOut pk;
    constexpr int RND_CAP = 4096;
    TRY(dalloc(ctx, W_COUNTER, 4 * FAST_MAX_CHUNKS, &d_counter));
    TRY(dalloc(ctx, W_OVF, (size_t)n_seqs, &d_ovf));
    TRY(dalloc(ctx, W_NCALLS, 1, &d_nc));
    TRY(dalloc(ctx, W_RNDC, 1, &d_rnd));
    TRY(dalloc(ctx, W_RNDL, (size_t)4 * RND_CAP, &pk.rnd_list));
    CK(cudaMemsetAsync(d_counter, 0, 4 * sizeof(int), ctx->stream));
    CK(cudaMemsetAsync(d_nc, 0, sizeof(unsigned long long), ctx->stream));
    CK(cudaMemsetAsync(d_rnd, 0, sizeof(int), ctx->stream));
    pk.nib = d_dbn_nib; pk.milli = d_score_milli; pk.ns16 = d_n_stems; pk.rnd_count = d_rnd; pk.rnd_cap = RND_CAP;
    // (scores next to a rounding tie keep FLAG_ROUND in d_flags and their thousandths unset: the host variant redoes those)
    int rc = fast_launch(ctx, *P, pl, ctx->stream, 0, n_seqs, d_offsets, d_packed, nullptr, nullptr, nullptr,
                         d_flags, d_counter, d_ovf, d_nc, 0, ctx->ev0, ctx->ev1, nullptr, &pk);
    if (rc == SQRN_OK) ctx->ev_valid = true;
    return rc;
}

extern "C" int sqrn_fast_predict_packed_device(sqrn_ctx *ctx, const sqrn_paramset *ps, int64_t n_seqs, int64_t total_len,
                                               int32_t max_len, const int64_t *d_offsets, const uint8_t *d_packed,
                                               uint8_t *d_dbn_nib, int32_t *d_score_milli, uint16_t *d_n_stems, uint8_t *d_flags)
{
    return guarded(ctx, [&] { return sqrn_fast_predict_packed_device_impl(ctx, ps, n_seqs, total_len, max_len, d_offsets, d_packed, d_dbn_nib, d_score_milli, d_n_stems, d_flags); });
}

// Host buffers in, host buffers out.  The batch is cut into chunks that flow through three
// stages on separate streams -- host->device copy, kernel, device->host copy -- so PCIe traffic
// in both directions overlaps the kernels of the neighbouring chunks.
//
// Two boundary formats share the pipeline.  Bytes: ASCII symbols + int64 offsets in, ASCII dot-bracket + three rounded
// float64 scores + int32 stem counts out.  Packed (`off32` set): 2-bit base codes + uint32 offsets in (offsets are
// widened on the device), 4-bit bracket codes + two int32 scores in thousandths + uint16 stem counts + flags out --
// 0.11 GB instead of 0.30 GB over PCIe per million 130-nt sequences.
__global__ void k_widen_offsets(const uint32_t *__restrict__ in, int64_t *__restrict__ out, int64_t n)
{
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) out[k] = (int64_t)in[k];
}

struct FastIO {
    const int64_t *off64 = nullptr; const uint32_t *off32 = nullptr; const uint8_t *symbols = nullptr;
    uint8_t *dbn = nullptr;            // ASCII (bytes) or 4-bit codes (packed)
    double *scores = nullptr; int32_t *n_stems = nullptr;                     // bytes
    int32_t *milli = nullptr; uint16_t *ns16 = nullptr; uint8_t *flags = nullptr;   // packed
};

static int fast_predict_host_impl(sqrn_ctx *ctx, const sqrn_paramset *ps, int64_t n_seqs, const FastIO &io)
{
    const bool packed = io.off32 != nullptr;
    const int64_t *offsets = io.off64; const uint8_t *symbols = io.symbols; uint8_t *dbn_ascii = io.dbn;
    double *scores = io.scores; int32_t *n_stems = io.n_stems;
    auto OFF = [&](int64_t b) -> int64_t { return packed ? (int64_t)io.off32[b] : offsets[b]; };
    cudaSetDevice(ctx->device);
    ctx->n_launches = 0; ctx->n_calls = 0; ctx->kernel_ms = 0; ctx->n_cluster_launches = 0;
    if (n_seqs == 0) return SQRN_OK;
    const bool trace = getenv("SQRN_TRACE") != nullptr;
    auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t_0 = now();
    const int64_t total = OFF(n_seqs);
    int64_t *d_off; uint8_t *d_sym, *d_dbn, *d_flags; double *d_sc = nullptr; int32_t *d_ns = nullptr; int *d_counter; unsigned long long *d_nc;
    uint32_t *d_off32 = nullptr; PackedOut pk; int *d_rnd = nullptr;
    constexpr int RND_CAP = 4096;
    TRY(dalloc(ctx, B_OFF, (size_t)n_seqs + 1, &d_off));
    if (packed) {
        TRY(dalloc(ctx, B_OFF32, (size_t)n_seqs + 1, &d_off32));
        TRY(dalloc(ctx, B_SYM, (size_t)(total + 3) / 4 + 1, &d_sym));
        TRY(dalloc(ctx, W_DBNA, (size_t)(total / 2 + n_seqs + 1), &d_dbn));
        TRY(dalloc(ctx, W_ORAW, (size_t)n_seqs, &d_sc));              // 2 int32 per sequence
        TRY(dalloc(ctx, W_ON, (size_t)(n_seqs + 1) / 2, &d_ns));      // uint16 per sequence
        TRY(dalloc(ctx, W_RNDC, 1, &d_rnd));
        TRY(dalloc(ctx, W_RNDL, (size_t)4 * RND_CAP, &pk.rnd_list));
        pk.nib = d_dbn; pk.milli = (int32_t *)d_sc; pk.ns16 = io.ns16 ? (uint16_t *)d_ns : nullptr; pk.rnd_count = d_rnd; pk.rnd_cap = RND_CAP;
    } else {
        TRY(dalloc(ctx, B_SYM, (size_t)std::max<int64_t>(total, 1), &d_sym));
        TRY(dalloc(ctx, W_DBNA, (size_t)std::max<int64_t>(total, 1), &d_dbn));
        TRY(dalloc(ctx, W_ORAW, (size_t)n_seqs * 3, &d_sc));
        TRY(dalloc(ctx, W_ON, (size_t)n_seqs, &d_ns));
    }
    TRY(dalloc(ctx, W_OFLAGS, (size_t)n_seqs, &d_flags));
    int32_t *d_ovf;
    TRY(dalloc(ctx, W_COUNTER, 4 * FAST_MAX_CHUNKS, &d_counter));
    TRY(dalloc(ctx, W_OVF, (size_t)n_seqs, &d_ovf));
    TRY(dalloc(ctx, W_NCALLS, 1, &d_nc));
    if (ctx->hflags_cap < (size_t)n_seqs) {
        if (ctx->hflags) cudaFreeHost(ctx->hflags);
        ctx->hflags = nullptr; ctx->hflags_cap = 0;
        CK(cudaMallocHost(&ctx->hflags, (size_t)n_seqs + 64));
        ctx->hflags_cap = (size_t)n_seqs + 64;
    }
    const double t_1 = now();
    // chunks of at least 64 Ki sequences; the first and the last one are cut again (1/4 + 3/4, 2/3 + 1/3) so that
    // the pipeline fills and drains on small pieces
    int nbase = (int)std::min<int64_t>(FAST_MAX_CHUNKS - 2, std::max<int64_t>(1, n_seqs / 65536));
    if (const char *e = getenv("SQRN_FAST_CHUNKS")) nbase = std::max(1, std::min(FAST_MAX_CHUNKS - 2, atoi(e)));
    int64_t bounds[FAST_MAX_CHUNKS + 1];
    int nchunks = 0;
    bounds[0] = 0;
    for (int c = 0; c < nbase; c++) {
        const int64_t lo = n_seqs * c / nbase, hi = n_seqs * (c + 1) / nbase;
        if (nbase >= 4 && c == 0) bounds[++nchunks] = lo + (hi - lo) / 4;
        if (nbase >= 4 && c == nbase - 1) bounds[++nchunks] = lo + (hi - lo) * 2 / 3;
        bounds[++nchunks] = hi;
    }
    cudaStream_t s_main = ctx->stream;
    CK(cudaMemsetAsync(d_counter, 0, 4 * FAST_MAX_CHUNKS * sizeof(int), s_main));
    CK(cudaMemsetAsync(d_nc, 0, sizeof(unsigned long long), s_main));
    if (packed) CK(cudaMemsetAsync(d_rnd, 0, sizeof(int), s_main));
    CK(cudaEventRecord(ctx->ev_start, s_main));
    CK(cudaStreamWaitEvent(ctx->s_in, ctx->ev_start, 0));
    Plan plans[4]; bool have_plan[4] = {false, false, false, false};
    if (ctx->horder_cap < (size_t)n_seqs) {
        if (ctx->horder) cudaFreeHost(ctx->horder);
        ctx->horder = nullptr; ctx->horder_cap = 0;
        CK(cudaMallocHost(&ctx->horder, ((size_t)n_seqs + 64) * sizeof(int32_t)));
        ctx->horder_cap = (size_t)n_seqs + 64;
    }
    std::vector<int64_t> len_count;
    bool split_chunk[FAST_MAX_CHUNKS] = {};
    const bool no_order = getenv("SQRN_FAST_NO_ORDER") != nullptr;
    for (int c = 0; c < nchunks; c++) {
        const int64_t b0 = bounds[c], b1 = bounds[c + 1];
        const int64_t t0 = OFF(b0), t1 = OFF(b1);
        cudaStream_t s_k = (c & 1) ? ctx->s_k2 : s_main;
        // the chunk's longest sequence picks its kernel (scanned while the earlier chunks are in flight); a chunk that
        // mixes sequences of up to 320 symbols with longer ones is dealt to two launches (warp teams / CTA teams)
        int max_len = 0, short_max = 0;
        int64_t n_long = 0;
        for (int64_t b = b0; b < b1; b++) {
            int64_t n = OFF(b + 1) - OFF(b);
            if (n < 0 || n > SQRN_MAX_LEN) { ctx->err = "sequence length out of range"; cudaDeviceSynchronize(); return SQRN_E_BADARG; }
            if (n > max_len) max_len = (int)n;
            if (n > 320) n_long++; else if (n > short_max) short_max = (int)n;
        }
        static const bool no_split = getenv("SQRN_FAST_NO_SPLIT") != nullptr;
        const bool split = n_long > 0 && n_long < b1 - b0 && !no_split;
        const int64_t n_short = split ? (b1 - b0) - n_long : 0;
        const PEntry *P;
        TRY(get_params(ctx, *ps, max_len, &P));
        const int cls = max_len <= 128 ? 0 : max_len <= 224 ? 1 : max_len <= 320 ? 2 : 3;
        // (plans of the three short classes are kept for the call: they are laid out for the class limit, not this chunk's maximum)
        static const int cls_cap[3] = {128, 224, 320};
        if (cls == 3 || !have_plan[cls]) { TRY(make_fast_plan(ctx, *P, cls == 3 ? max_len : cls_cap[cls], (int)(split ? n_long : b1 - b0), plans[cls])); have_plan[cls] = true; }
        const Plan &pl = plans[cls];
        const int scls = short_max <= 128 ? 0 : short_max <= 224 ? 1 : 2;
        if (split && !have_plan[scls]) { TRY(make_fast_plan(ctx, *P, cls_cap[scls], (int)n_short, plans[scls])); have_plan[scls] = true; }
        // CTA-team plans share per-context scratch (candidate lists, counters): their launches all go to one stream
        if (pl.tw > 1 && !split) s_k = s_main;
        // Long sequences: longest first (a counting sort by length, done while the earlier chunks run), so that the
        // last CTAs to finish are not the longest items and the SM slots the next chunk's kernel is waiting for
        // free up together instead of trailing behind one long sequence each.
        const int32_t *d_order = nullptr;
        // (warp-team chunks are taken in input order: measured, the order list bought nothing there -- 11.3 ms either way per
        //  1 M sequences -- and cost the host 5 ms of counting sort per step plus 4 MB of copies)
        static const bool order_short = getenv("SQRN_FAST_ORDER_SHORT") != nullptr;
        if (split) {
            // [short items in input order | long items, longest first]
            int32_t *ord = ctx->horder + b0;
            len_count.assign((size_t)max_len + 2, 0);
            int64_t ks = 0;
            for (int64_t b = b0; b < b1; b++) {
                const int64_t n = OFF(b + 1) - OFF(b);
                if (n > 320) len_count[(size_t)(max_len - n) + 1]++; else ord[ks++] = (int32_t)b;
            }
            for (int l = 0; l <= max_len; l++) len_count[(size_t)l + 1] += len_count[(size_t)l];
            for (int64_t b = b0; b < b1; b++) {
                const int64_t n = OFF(b + 1) - OFF(b);
                if (n > 320) ord[n_short + len_count[(size_t)(max_len - n)]++] = (int32_t)b;
            }
            int32_t *d_o;
            TRY(dalloc(ctx, W_ORDER, (size_t)n_seqs, &d_o));
            CK(cudaMemcpyAsync(d_o + b0, ord, (size_t)(b1 - b0) * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->s_in));
            d_order = d_o + b0;
        }
        else if (b1 - b0 > 1 && (pl.tw > 1 || (order_short && b1 - b0 >= 4096)) && !no_order) {
            int32_t *ord = ctx->horder + b0;      // pinned, one region per chunk: the copy below is truly asynchronous
            len_count.assign((size_t)max_len + 2, 0);
            for (int64_t b = b0; b < b1; b++) len_count[(size_t)(max_len - (OFF(b + 1) - OFF(b))) + 1]++;
            for (int l = 0; l <= max_len; l++) len_count[(size_t)l + 1] += len_count[(size_t)l];
            for (int64_t b = b0; b < b1; b++) ord[len_count[(size_t)(max_len - (OFF(b + 1) - OFF(b)))]++] = (int32_t)b;
            int32_t *d_o;
            TRY(dalloc(ctx, W_ORDER, (size_t)n_seqs, &d_o));
            CK(cudaMemcpyAsync(d_o + b0, ord, (size_t)(b1 - b0) * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->s_in));
            d_order = d_o + b0;
        }
        // stage 1: inputs of the chunk
        const int64_t o_lo = b0 + (c ? 1 : 0), o_n = b1 - b0 + (c ? 0 : 1);      // offsets this chunk adds
        if (packed) {
            CK(cudaMemcpyAsync(d_off32 + o_lo, io.off32 + o_lo, (size_t)o_n * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->s_in));
            k_widen_offsets<<<(unsigned)std::min<int64_t>(256, (o_n + 255) / 256), 256, 0, ctx->s_in>>>(d_off32 + o_lo, d_off + o_lo, o_n);
            CK(cudaGetLastError());
            if (t1 > t0) CK(cudaMemcpyAsync(d_sym + t0 / 4, symbols + t0 / 4, (size_t)((t1 + 3) / 4 - t0 / 4), cudaMemcpyHostToDevice, ctx->s_in));
        } else {
            CK(cudaMemcpyAsync(d_off + o_lo, offsets + o_lo, (size_t)o_n * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->s_in));
            if (t1 > t0) CK(cudaMemcpyAsync(d_sym + t0, symbols + t0, (size_t)(t1 - t0), cudaMemcpyHostToDevice, ctx->s_in));
        }
        CK(cudaEventRecord(ctx->ev_in[c], ctx->s_in));
        // stage 2: kernel
        CK(cudaStreamWaitEvent(s_k, ctx->ev_in[c], 0));
        if (c == 1) CK(cudaStreamWaitEvent(s_k, ctx->ev_start, 0));
        if (split) {
            // the short items through their warp-team kernel on the chunk's stream, the long ones through CTA teams on the
            // main stream (counter: the spare word of the chunk's four); the chunk's outputs wait for both
            TRY(fast_launch(ctx, *P, plans[scls], s_k, b0, n_short, d_off, d_sym, d_dbn, d_sc, d_ns, d_flags, d_counter + 4 * c, d_ovf, d_nc, 1,
                            ctx->ev_k0[c], ctx->ev_k1[c], d_order, packed ? &pk : nullptr, b1));
            if (s_k != s_main) CK(cudaStreamWaitEvent(s_main, ctx->ev_in[c], 0));
            TRY(fast_launch(ctx, *P, pl, s_main, b0, n_long, d_off, d_sym, d_dbn, d_sc, d_ns, d_flags, d_counter + 4 * c + 3, d_ovf, d_nc, 1,
                            ctx->ev_l0[c], ctx->ev_l1[c], d_order + n_short, packed ? &pk : nullptr, b1));
            CK(cudaStreamWaitEvent(ctx->s_out, ctx->ev_l1[c], 0));
            split_chunk[c] = true;
        }
        else
        TRY(fast_launch(ctx, *P, pl, s_k, b0, b1 - b0, d_off, d_sym, d_dbn, d_sc, d_ns, d_flags, d_counter + 4 * c, d_ovf, d_nc, 1,
                        ctx->ev_k0[c], ctx->ev_k1[c], d_order, packed ? &pk : nullptr));
        // stage 3: outputs of the chunk
        CK(cudaStreamWaitEvent(ctx->s_out, ctx->ev_k1[c], 0));
        if (packed) {
            const int64_t y0 = t0 / 2 + b0, y1 = t1 / 2 + b1;                     // bytes of the chunk's 4-bit codes
            if (y1 > y0) CK(cudaMemcpyAsync(dbn_ascii + y0, d_dbn + y0, (size_t)(y1 - y0), cudaMemcpyDeviceToHost, ctx->s_out));
            CK(cudaMemcpyAsync(io.milli + 2 * b0, (int32_t *)d_sc + 2 * b0, (size_t)(b1 - b0) * 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->s_out));
            if (io.ns16) CK(cudaMemcpyAsync(io.ns16 + b0, (uint16_t *)d_ns + b0, (size_t)(b1 - b0) * sizeof(uint16_t), cudaMemcpyDeviceToHost, ctx->s_out));
        } else {
            if (t1 > t0) CK(cudaMemcpyAsync(dbn_ascii + t0, d_dbn + t0, (size_t)(t1 - t0), cudaMemcpyDeviceToHost, ctx->s_out));
            CK(cudaMemcpyAsync(scores + 3 * b0, d_sc + 3 * b0, (size_t)(b1 - b0) * 3 * sizeof(double), cudaMemcpyDeviceToHost, ctx->s_out));
            if (n_stems) CK(cudaMemcpyAsync(n_stems + b0, d_ns + b0, (size_t)(b1 - b0) * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->s_out));
        }
        CK(cudaMemcpyAsync(ctx->hflags + b0, d_flags + b0, (size_t)(b1 - b0), cudaMemcpyDeviceToHost, ctx->s_out));
        CK(cudaEventRecord(ctx->ev_o[c], ctx->s_out));
    }
    const double t_2 = now();
    CK(cudaEventRecord(ctx->ev_out, ctx->s_out));
    CK(cudaEventRecord(ctx->ev_k2done, ctx->s_k2));
    CK(cudaStreamWaitEvent(s_main, ctx->ev_out, 0));          // later work on the context's stream sees the results
    CK(cudaStreamWaitEvent(s_main, ctx->ev_k2done, 0));
    // ScoreStruct's round(x, 3) (seq.py:899) was done on the device except next to rounding ties: the flags of
    // each chunk are checked as soon as its results are back, while the later chunks are still in flight
    bool too_many_levels = false;
    for (int c = 0; c < nchunks; c++) {
        CK(cudaEventSynchronize(ctx->ev_o[c]));
        const uint8_t *fl = ctx->hflags;
        for (int64_t b = bounds[c]; b < bounds[c + 1]; ) {
            if (b + 8 <= bounds[c + 1]) {
                uint64_t w; memcpy(&w, fl + b, 8);
                if (!(w & 0x0a0a0a0a0a0a0a0aull)) { b += 8; continue; }
            }
            if ((fl[b] & FLAG_ROUND) && !packed) for (int t = 0; t < 3; t++) scores[3 * b + t] = pyround3(scores[3 * b + t]);
            if (fl[b] & FLAG_LEVELS) too_many_levels = true;
            b++;
        }
    }
    CK(cudaStreamSynchronize(s_main));
    if (packed) {
        // scores next to a rounding tie came back unrounded through the side list: CPython's round() on the host
        int nr = 0;
        CK(cudaMemcpy(&nr, d_rnd, sizeof nr, cudaMemcpyDeviceToHost));
        if (nr > RND_CAP) { ctx->err = "too many scores next to a rounding tie"; return SQRN_E_UNSUPPORTED; }
        if (nr > 0) {
            std::vector<double> rl((size_t)4 * nr);
            CK(cudaMemcpy(rl.data(), pk.rnd_list, rl.size() * sizeof(double), cudaMemcpyDeviceToHost));
            for (int k = 0; k < nr; k++) {
                const int64_t b = (int64_t)rl[4 * (size_t)k];
                for (int t = 0; t < 2; t++) {
                    const double q = pyround3(rl[4 * (size_t)k + 1 + t]) * 1000.0;
                    if (!(fabs(q) < 2147483000.0)) { ctx->err = "score out of the range of the packed format"; return SQRN_E_UNSUPPORTED; }
                    io.milli[2 * b + t] = (int32_t)llrint(q);
                }
            }
        }
        if (io.flags) memcpy(io.flags, ctx->hflags, (size_t)n_seqs);
        too_many_levels = false;          // the caller reads the flags: bit 1 = the sequence needs the byte lane (more than 7 levels)
    }
    const double t_3 = now();
    for (int c = 0; c < nchunks; c++) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, ctx->ev_k0[c], ctx->ev_k1[c]) == cudaSuccess) ctx->kernel_ms += ms;
        if (split_chunk[c] && cudaEventElapsedTime(&ms, ctx->ev_l0[c], ctx->ev_l1[c]) == cudaSuccess) ctx->kernel_ms += ms;
    }
    {
        unsigned long long c = 0;
        CK(cudaMemcpy(&c, d_nc, sizeof c, cudaMemcpyDeviceToHost));
        ctx->n_calls = (int64_t)c;
    }
    if (too_many_levels) { ctx->err = "more than 30 pseudoknot levels: use sqrn_predict_batch"; return SQRN_E_UNSUPPORTED; }
    if (trace) {
        fprintf(stderr, "[sqrn] fast_predict_host: prepare %.2f ms, enqueue %.2f ms, wait %.2f ms, finish %.2f ms\n",
                t_1 - t_0, t_2 - t_1, t_3 - t_2, now() - t_3);
        {
            std::vector<int> hc(4 * FAST_MAX_CHUNKS);
            cudaMemcpy(hc.data(), d_counter, hc.size() * sizeof(int), cudaMemcpyDeviceToHost);
            long long ovf = 0;
            for (int c = 0; c < nchunks; c++) ovf += hc[4 * c + 1];
            fprintf(stderr, "[sqrn]   items sent to the rescanning kernel (run-list overflow): %lld of %lld\n", ovf, (long long)n_seqs);
        }
        for (int c = 0; c < nchunks; c++) {
            float a = 0, b = 0;
            cudaEventElapsedTime(&a, ctx->ev_k0[0], ctx->ev_k0[c]); cudaEventElapsedTime(&b, ctx->ev_k0[0], ctx->ev_k1[c]);
            fprintf(stderr, "[sqrn]   chunk %2d kernel %.3f .. %.3f ms\n", c, a, b);
        }
    }
    return SQRN_OK;
}

extern "C" int sqrn_fast_predict_host(sqrn_ctx *ctx, const sqrn_paramset *ps, int64_t n_seqs, const int64_t *offsets,
                                      const uint8_t *symbols, uint8_t *dbn_ascii, double *scores, int32_t *n_stems)
{
    if (!ctx || !ps || !offsets || n_seqs < 0 || n_seqs > 0x7fffffff) return SQRN_E_BADARG;
    FastIO io; io.off64 = offsets; io.symbols = symbols; io.dbn = dbn_ascii; io.scores = scores; io.n_stems = n_stems;
    return guarded(ctx, [&] { return fast_predict_host_impl(ctx, ps, n_seqs, io); });
}

extern "C" int sqrn_fast_predict_packed_host(sqrn_ctx *ctx, const sqrn_paramset *ps, int64_t n_seqs, const uint32_t *offsets,
                                             const uint8_t *packed, uint8_t *dbn_nib, int32_t *score_milli, uint16_t *n_stems,
                                             uint8_t *flags)
{
    if (!ctx || !ps || !offsets || !score_milli || n_seqs < 0 || n_seqs > 0x7fffffff) return SQRN_E_BADARG;
    FastIO io; io.off32 = offsets; io.symbols = packed; io.dbn = dbn_nib; io.milli = score_milli; io.ns16 = n_stems; io.flags = flags;
    return guarded(ctx, [&] { return fast_predict_host_impl(ctx, ps, n_seqs, io); });
}

extern "C" int sqrn_fast_last_flags(const sqrn_ctx *ctx, int64_t n_seqs, uint8_t *flags)
{
    if (!ctx || !flags || n_seqs < 0 || (size_t)n_seqs > ctx->hflags_cap) return SQRN_E_BADARG;
    memcpy(flags, ctx->hflags, (size_t)n_seqs);
    return SQRN_OK;
}

// ------------------------------------------------------ general work runner
struct DeviceBatch {                 // an uploaded sqrn_batch
    DevBatch B; std::vector<int> len; int nmax = 0, rbmax = 0;
    std::vector<int32_t> rb_sorted;
};

static int upload_batch(sqrn_ctx *ctx, const sqrn_batch *in, DeviceBatch &D)
{
    DevBatch &B = D.B; memset(&B, 0, sizeof B);
    const int64_t n = in->n_seqs;
    if (n < 0 || n > 0x7fffffff || !in->offsets || (!in->symbols && n)) { ctx->err = "bad batch"; return SQRN_E_BADARG; }
    D.len.resize((size_t)n); D.nmax = 0; D.rbmax = 0;
    for (int64_t b = 0; b < n; b++) {
        int64_t l = in->offsets[b + 1] - in->offsets[b];
        if (l < 0 || l > SQRN_MAX_LEN) { ctx->err = "sequence length out of range"; return SQRN_E_BADARG; }
        D.len[b] = (int)l; D.nmax = std::max(D.nmax, (int)l);
    }
    const int64_t total = in->offsets[n];
    B.n_seqs = n; B.interchainonly = in->interchainonly; B.react_comp = in->react_sum_compensated;
    int64_t *d_off; uint8_t *d_sym;
    TRY(upload(ctx, B_OFF, in->offsets, (size_t)n + 1, &d_off)); B.off = d_off;
    TRY(upload(ctx, B_SYM, in->symbols, (size_t)total, &d_sym)); B.sym = d_sym;
    if (in->react_code) {
        int R = in->n_react_values;
        if (R < 1 || R > 65535 || !in->react_values) { ctx->err = "bad reactivity table"; return SQRN_E_BADARG; }
        uint16_t *d_rc; double *d_rv;
        TRY(upload(ctx, B_RCODE, in->react_code, (size_t)total, &d_rc));
        TRY(upload(ctx, B_RVALS, in->react_values, (size_t)R, &d_rv));
        B.rcode = d_rc; B.rvals = d_rv; B.R = R;
        if (R <= SQRN_MAX_REACT_LUT) {               // host libm pow() table; above that the device uses sqrt
            std::vector<double> pos, neg;
            build_react_lut(in->react_values, R, pos, neg);
            double *d_p, *d_n;
            TRY(upload(ctx, B_RFPOS, pos.data(), pos.size(), &d_p));
            TRY(upload(ctx, B_RFNEG, neg.data(), neg.size(), &d_n));
            B.rf_pos = d_p; B.rf_neg = d_n;
        }
    }
    if (in->restr_class) { uint8_t *d; TRY(upload(ctx, B_RCLASS, in->restr_class, (size_t)total, &d)); B.rclass = d; }
    if (in->rbp_offsets && in->rbp_offsets[n] > 0) {
        for (int64_t b = 0; b < n; b++) {
            int64_t q = in->rbp_offsets[b + 1] - in->rbp_offsets[b];
            if (q < 0 || q > D.len[b]) { ctx->err = "bad restraint pair list"; return SQRN_E_BADARG; }
            D.rbmax = std::max(D.rbmax, (int)q);
            for (int64_t k = in->rbp_offsets[b]; k < in->rbp_offsets[b + 1]; k++) {
                int v = in->rbps[2 * k], w = in->rbps[2 * k + 1];
                if (v < 0 || w <= v || w >= D.len[b]) { ctx->err = "restraint pair out of range"; return SQRN_E_BADARG; }
            }
        }
        sort_rbps(n, in->rbp_offsets, in->rbps, D.rb_sorted);
        int64_t *d_o; int32_t *d_r;
        TRY(upload(ctx, B_RBOFF, in->rbp_offsets, (size_t)n + 1, &d_o));
        TRY(upload(ctx, B_RB, D.rb_sorted.data(), D.rb_sorted.size(), &d_r));
        B.rbp_off = d_o; B.rbp = d_r;
    }
    if (in->smat) {
        if (!in->cols || in->smat_L <= 0) { ctx->err = "smat without column map"; return SQRN_E_BADARG; }
        double *d_s; int32_t *d_c;
        TRY(upload(ctx, B_SMAT, in->smat, (size_t)in->smat_L * in->smat_L, &d_s));
        TRY(upload(ctx, B_COLS, in->cols, (size_t)total, &d_c));
        B.smat = d_s; B.L = in->smat_L; B.cols = d_c;
    }
    if (in->bpp_mode) {
        if ((in->bpp_mode != 1 && in->bpp_mode != 2) || !in->bpp_term || !in->bpp_offsets) { ctx->err = "bad bpp term"; return SQRN_E_BADARG; }
        for (int64_t b = 0; b < n; b++)
            if (in->bpp_offsets[b + 1] - in->bpp_offsets[b] != (int64_t)D.len[b] * D.len[b]) { ctx->err = "bpp term: need one N x N matrix per sequence"; return SQRN_E_BADARG; }
        double *d_t; int64_t *d_o;
        TRY(upload(ctx, B_BPP, in->bpp_term, (size_t)in->bpp_offsets[n], &d_t));
        TRY(upload(ctx, B_BPPOFF, in->bpp_offsets, (size_t)n + 1, &d_o));
        B.bpp = d_t; B.bpp_off = d_o; B.bpp_mode = in->bpp_mode;
    }
    return SQRN_OK;
}

// base lists of the batch for the current parameter set (device pointers; DevWork::base_*)
struct BaseDev { BEnt *ent = nullptr; int64_t *off = nullptr; int32_t *n = nullptr; int32_t *bend = nullptr; bool valid = false; };

struct HostWork {
    int mode = MODE_TAIL;
    const BaseDev *base = nullptr;
    std::vector<int32_t> item_seq; std::vector<int64_t> init_off; std::vector<int32_t> init_stems;
    std::vector<double> subopt; std::vector<int64_t> out_cap;        // per item stem capacity
    bool want_dbn = false, want_fin = false;
    bool keep_on_device = false;     // leave stems / scores in the context's device buffers (only the counts come back)
    // device copies of the outputs after run_items (valid until the context's scratch is reused)
    const int32_t *d_out_stems = nullptr; const double *d_out_fin = nullptr; const int32_t *d_out_n = nullptr; const int64_t *d_out_off = nullptr;
    // outputs
    std::vector<int64_t> out_off, dbn_off;
    std::vector<int32_t> out_stems, out_n; std::vector<double> out_fin, out_raw;
    std::vector<uint8_t> flags; std::vector<int8_t> dbn;
};

// run all items of W (any mix of sequence lengths) and bring the outputs back
static int run_items(sqrn_ctx *ctx, const sqrn_paramset &ps, const DeviceBatch &D, HostWork &W, int min_ccap = 0)
{
    const int n = (int)W.item_seq.size();
    W.out_n.assign((size_t)n, 0);
    W.out_off.assign((size_t)n + 1, 0);
    for (int k = 0; k < n; k++) W.out_off[k + 1] = W.out_off[k] + W.out_cap[k];
    const int64_t tot_stems = W.out_off[n];
    W.out_stems.assign(W.keep_on_device ? 0 : (size_t)tot_stems * 3, 0);
    if (W.want_fin || W.mode == MODE_YIELD) W.out_fin.assign(W.keep_on_device ? 1 : (size_t)tot_stems, 0.0);
    const bool fin = (W.mode == MODE_TAIL || W.mode == MODE_FINAL);
    if (fin) { W.out_raw.assign((size_t)n * 3, 0.0); W.flags.assign((size_t)n, 0); }
    int64_t tot_dbn = 0;
    if (fin && W.want_dbn) {
        W.dbn_off.assign((size_t)n + 1, 0);
        for (int k = 0; k < n; k++) W.dbn_off[k + 1] = W.dbn_off[k] + D.len[W.item_seq[k]];
        tot_dbn = W.dbn_off[n];
        W.dbn.assign((size_t)tot_dbn, 0);
    }
    if (n == 0) return SQRN_OK;

    DevWork G; memset(&G, 0, sizeof G);
    G.mode = W.mode; G.region_mode = ctx->region_mode;
    int32_t *d_iseq; TRY(upload(ctx, W_ISEQ, W.item_seq.data(), (size_t)n, &d_iseq)); G.item_seq = d_iseq;
    if (!W.init_off.empty() && !W.init_stems.empty()) {
        int64_t *d_io; int32_t *d_is;
        TRY(upload(ctx, W_IOFF, W.init_off.data(), (size_t)n + 1, &d_io));
        TRY(upload(ctx, W_ISTEMS, W.init_stems.data(), W.init_stems.size(), &d_is));
        G.init_off = d_io; G.init_stems = d_is;
    }
    if (W.mode == MODE_STEP) { double *d; TRY(upload(ctx, W_SUBOPT, W.subopt.data(), (size_t)n, &d)); G.item_subopt = d; }
    int64_t *d_oo; TRY(upload(ctx, W_OOFF, W.out_off.data(), (size_t)n + 1, &d_oo)); G.out_off = d_oo;
    TRY(dalloc(ctx, W_OSTEMS, (size_t)tot_stems * 3, &G.out_stems));
    TRY(dalloc(ctx, W_ON, (size_t)n, &G.out_nstems));
    if (!W.out_fin.empty()) TRY(dalloc(ctx, W_OFIN, (size_t)tot_stems, &G.out_stemfin));
    if (fin) { TRY(dalloc(ctx, W_ORAW, (size_t)n * 3, &G.out_raw)); TRY(dalloc(ctx, W_OFLAGS, (size_t)n, &G.out_flags)); }
    if (tot_dbn || (fin && W.want_dbn)) {
        int64_t *d_do; TRY(upload(ctx, W_DOFF, W.dbn_off.data(), (size_t)n + 1, &d_do)); G.dbn_off = d_do;
        TRY(dalloc(ctx, W_DBNC, (size_t)tot_dbn, &G.out_dbn_code));
    }
    TRY(dalloc(ctx, W_COUNTER, 1, &G.counter));
    TRY(dalloc(ctx, W_NCALLS, 1, &G.n_calls));
    CK(cudaMemsetAsync(G.n_calls, 0, sizeof(unsigned long long), ctx->stream));
    const bool have_base = W.base && W.base->valid && (W.mode == MODE_STEP || W.mode == MODE_TAIL || W.mode == MODE_BASE);
    if (have_base) { G.base_ent = W.base->ent; G.base_off = W.base->off; G.base_n = W.base->n; G.base_bend = W.base->bend; }

    // length classes: warp teams (<= 320), 256-thread CTAs (<= 2048), 1024-thread CTAs
    std::vector<int32_t> order((size_t)n);
    for (int k = 0; k < n; k++) order[k] = k;
    auto cls = [&](int k) { int l = D.len[W.item_seq[k]]; return (l <= 320 && min_ccap <= 1024) ? 0 : (l <= 2048 ? 1 : 2); };
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
        int ca = cls(a), cb = cls(b);
        if (ca != cb) return ca < cb;
        return D.len[W.item_seq[a]] > D.len[W.item_seq[b]];          // longest first inside a class
    });
    int32_t *d_order; TRY(upload(ctx, W_ORDER, order.data(), (size_t)n, &d_order));
    const PEntry *P; TRY(get_params(ctx, ps, std::max(D.nmax, 1), &P));
    // most pre-selected stems of any item; MODE_FINAL gets structures of other parameter sets: no bound from m
    int max_init = 0;
    if (W.mode == MODE_FINAL) max_init = -1;
    else if (!W.init_off.empty())
        for (int k = 0; k < n; k++) max_init = std::max<int>(max_init, (int)(W.init_off[k + 1] - W.init_off[k]));
    int pos = 0;
    while (pos < n) {
        int c = cls(order[pos]), end = pos;
        while (end < n && cls(order[end]) == c) end++;
        int nmax_c = D.len[W.item_seq[order[pos]]];
        Plan pl; TRY(make_plan(ctx, *P, std::max(nmax_c, 1), D.rbmax, min_ccap, W.mode == MODE_STEP, D.B.rcode != nullptr, max_init, pl,
                               have_base && c > 0));
        {
            const bool plain = !D.B.rcode && !D.B.rclass && !D.B.rbp_off && !D.B.smat && !D.B.interchainonly && !D.B.bpp;
            maybe_glist(ctx, *P, pl, std::max(nmax_c, 1), D.rbmax, D.B.rcode != nullptr, max_init, W.mode == MODE_TAIL);
            maybe_cluster(ctx, *P, pl, end - pos, plain, W.mode == MODE_TAIL);
        }
        DevWork Gc = G; Gc.order = d_order + pos; Gc.n_items = end - pos;
        TRY(launch(ctx, *P, pl, D.B, Gc));
        pos = end;
    }
    CK(cudaMemcpyAsync(W.out_n.data(), G.out_nstems, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    W.d_out_stems = G.out_stems; W.d_out_fin = G.out_stemfin; W.d_out_n = G.out_nstems; W.d_out_off = G.out_off;
    if (tot_stems && !W.keep_on_device) CK(cudaMemcpyAsync(W.out_stems.data(), G.out_stems, (size_t)tot_stems * 3 * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (!W.out_fin.empty() && tot_stems && !W.keep_on_device) CK(cudaMemcpyAsync(W.out_fin.data(), G.out_stemfin, (size_t)tot_stems * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    if (fin) {
        CK(cudaMemcpyAsync(W.out_raw.data(), G.out_raw, (size_t)n * 3 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(W.flags.data(), G.out_flags, (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (tot_dbn) CK(cudaMemcpyAsync(W.dbn.data(), G.out_dbn_code, (size_t)tot_dbn, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    unsigned long long c = 0;
    CK(cudaMemcpy(&c, G.n_calls, sizeof c, cudaMemcpyDeviceToHost));
    ctx->n_calls += (int64_t)c;
    if (ctx->ev_valid) { float ms = 0; if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->kernel_ms += ms; }
    return SQRN_OK;
}

// Base lists for the pool rounds of one parameter set: every sequence served by CTA teams (> 320 nt) gets a slot sized
// from the run density of random RNA (a slot that turns out too small just leaves its sequence to the enumerating path).
static int build_base(sqrn_ctx *ctx, const sqrn_paramset &ps, const DeviceBatch &D, BaseDev &bd)
{
    bd = BaseDev();
    static const bool off_knob = getenv("SQRN_NO_BASE") != nullptr;
    if (off_knob) return SQRN_OK;
    const int64_t nseq = (int64_t)D.len.size();
    const PEntry *P; TRY(get_params(ctx, ps, std::max(D.nmax, 1), &P));
    if (!P->hp.ub_ok || !(P->hp.loopbonus >= 0.0)) return SQRN_OK;
    const int m = P->hp.m;
    const double dens = m >= 4 ? 0.003 : (m == 3 ? 0.008 : 0.02);
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); return SQRN_OK; }
    const int64_t budget = (int64_t)std::min<size_t>(free_b / 2, (size_t)48 << 30) / (int64_t)sizeof(BEnt);
    std::vector<int64_t> off((size_t)nseq + 1, 0);
    HostWork W; W.mode = MODE_BASE;
    for (int64_t b = 0; b < nseq; b++) {
        int64_t cap = 0;
        if (D.len[b] > 320) cap = (int64_t)(1.5 * dens * D.len[b] * (double)D.len[b]) + 1024;
        if (off[b] + cap > budget) cap = 0;
        off[b + 1] = off[b] + cap;
        if (cap) { W.item_seq.push_back((int32_t)b); W.out_cap.push_back(0); }
    }
    if (W.item_seq.empty()) return SQRN_OK;
    TRY(dalloc(ctx, W_BASE, (size_t)off[nseq], &bd.ent));
    TRY(upload(ctx, W_BASEOFF, off.data(), (size_t)nseq + 1, &bd.off));
    TRY(dalloc(ctx, W_BASEN, (size_t)nseq, &bd.n));
    TRY(dalloc(ctx, W_BASEBEND, (size_t)nseq * (GL_NBIN + 1), &bd.bend));
    CK(cudaMemsetAsync(bd.n, 0xff, (size_t)nseq * sizeof(int32_t), ctx->stream));
    bd.valid = true;
    W.base = &bd;
    return run_items(ctx, ps, D, W);
}

// MODE_STEP with retries: grows the per-item output capacity / candidate list
// until every item fits (no approximation is ever returned)
static int run_step_items(sqrn_ctx *ctx, const sqrn_paramset &ps, const DeviceBatch &D, HostWork &W)
{
    const int n = (int)W.item_seq.size();
    W.out_cap.assign((size_t)n, 16);
    TRY(run_items(ctx, ps, D, W));
    std::vector<int> redo;
    for (int k = 0; k < n; k++) if (W.out_n[k] < 0 || W.out_n[k] > W.out_cap[k]) redo.push_back(k);
    if (redo.empty()) return SQRN_OK;
    int min_ccap = 0;
    // ChooseStems returns a set of pairwise-conflicting alternatives (seq.py:783-787): it is bounded by the number of
    // candidates, not by N / 2.  team_choose reports the true count even when it could only write `cap` triples, so an
    // item is done only when its count fits the capacity it ran with; otherwise it runs again with exactly that count.
    std::vector<int64_t> want((size_t)n, 0);
    for (int k : redo) want[k] = std::max<int64_t>(D.len[W.item_seq[k]] / 2 + 1, W.out_n[k]);
    for (int attempt = 0; attempt < 5 && !redo.empty(); attempt++) {
        HostWork R; R.mode = MODE_STEP; R.base = W.base;
        bool list_overflow = false;
        for (int k : redo) {
            R.item_seq.push_back(W.item_seq[k]);
            R.subopt.push_back(W.subopt[k]);
            if (W.out_n[k] < 0) list_overflow = true;
        }
        if (!W.init_off.empty()) {
            R.init_off.push_back(0);
            for (int k : redo) {
                for (int64_t q = W.init_off[k]; q < W.init_off[k + 1]; q++)
                    for (int t = 0; t < 3; t++) R.init_stems.push_back(W.init_stems[3 * q + t]);
                R.init_off.push_back((int64_t)R.init_stems.size() / 3);
            }
        }
        for (int k : redo) R.out_cap.push_back(want[k]);
        if (list_overflow) min_ccap = min_ccap ? min_ccap * 4 : 4096;
        TRY(run_items(ctx, ps, D, R, min_ccap));
        std::vector<int> still;
        // splice the re-run results back: rebuild W's CSR with the larger capacities
        std::vector<int64_t> new_off((size_t)n + 1, 0);
        std::vector<int64_t> new_cap = W.out_cap;
        auto fits = [&](size_t q) { return R.out_n[q] >= 0 && R.out_n[q] <= R.out_cap[q]; };
        for (size_t q = 0; q < redo.size(); q++) if (fits(q)) new_cap[redo[q]] = std::max<int64_t>(W.out_cap[redo[q]], R.out_n[q]);
        for (int k = 0; k < n; k++) new_off[k + 1] = new_off[k] + new_cap[k];
        std::vector<int32_t> new_stems((size_t)new_off[n] * 3, 0);
        for (int k = 0; k < n; k++) {
            int64_t cnt = std::min<int64_t>(std::max(W.out_n[k], 0), W.out_cap[k]);
            std::copy(W.out_stems.begin() + 3 * W.out_off[k], W.out_stems.begin() + 3 * (W.out_off[k] + cnt), new_stems.begin() + 3 * new_off[k]);
        }
        for (size_t q = 0; q < redo.size(); q++) {
            int k = redo[q];
            if (!fits(q)) {
                W.out_n[k] = R.out_n[q];                                // < 0: list overflow again; > cap: the count to run with
                if (R.out_n[q] > 0) want[k] = R.out_n[q];
                still.push_back(k);
                continue;
            }
            std::copy(R.out_stems.begin() + 3 * R.out_off[q], R.out_stems.begin() + 3 * (R.out_off[q] + R.out_n[q]), new_stems.begin() + 3 * new_off[k]);
            W.out_n[k] = R.out_n[q];
        }
        W.out_stems.swap(new_stems); W.out_off.swap(new_off); W.out_cap.swap(new_cap);
        redo.swap(still);
    }
    if (!redo.empty()) { ctx->err = "candidate list overflow: too many tied stems for one CTA"; return SQRN_E_UNSUPPORTED; }
    return SQRN_OK;
}

// ---------------------------------------------------- PairsToDBN on the host
// Generic per-pair restatement of SQRNdbnseq.py:114-161 for pair sets that are
// not a stem list (consensus intersections, hardrest forced pairs).
static void pairs_to_codes(std::vector<std::pair<int, int>> pairs, int N, int8_t *codes)
{
    for (auto &p : pairs) if (p.first > p.second) std::swap(p.first, p.second);
    std::sort(pairs.begin(), pairs.end());
    pairs.erase(std::unique(pairs.begin(), pairs.end()), pairs.end());
    const int n = (int)pairs.size();
    auto X = [&](int a, int b) {
        int i = pairs[a].first, j = pairs[a].second, k = pairs[b].first, l = pairs[b].second;
        return (i < k && k < j && j < l) || (k < i && i < l && l < j);
    };
    std::vector<int> cc((size_t)n, 0), ord((size_t)n), grp((size_t)n, -1), gsz;
    for (int a = 0; a < n; a++) for (int b = 0; b < n; b++) if (a != b && X(a, b)) cc[a]++;
    for (int a = 0; a < n; a++) ord[a] = a;
    std::stable_sort(ord.begin(), ord.end(), [&](int a, int b) {
        if (cc[a] != cc[b]) return cc[a] < cc[b];
        return pairs[a].first < pairs[b].first; });
    std::vector<std::vector<int>> groups;
    for (int a = 0; a < n; a++) {
        int x = ord[a], g = -1;
        for (size_t h = 0; h < groups.size() && g < 0; h++) {
            bool clash = false;
            for (int y : groups[h]) if (X(x, y)) { clash = true; break; }
            if (!clash) g = (int)h;
        }
        if (g < 0) { g = (int)groups.size(); groups.emplace_back(); }
        groups[g].push_back(x);
    }
    std::vector<int> gord(groups.size());
    for (size_t g = 0; g < groups.size(); g++) gord[g] = (int)g;
    std::stable_sort(gord.begin(), gord.end(), [&](int a, int b) { return groups[a].size() > groups[b].size(); });
    for (int p = 0; p < N; p++) codes[p] = 0;
    for (size_t r = 0; r < gord.size(); r++) {
        int lev = (int)std::min<size_t>(r + 1, 127);
        for (int x : groups[gord[r]]) { codes[pairs[x].first] = (int8_t)lev; codes[pairs[x].second] = (int8_t)-lev; }
    }
}

// fn(b) for b in [0, n) on a few host threads (per-sequence bookkeeping of big batches: each b touches only its own
// data).  The workers are started once per process and sleep between jobs (a pool round posts three jobs; starting
// fifteen threads for each cost as much as it saved).  Exceptions never leave a worker: they are reported by the caller.
namespace {
struct HostPool {
    std::vector<std::thread> th;
    std::mutex mu; std::condition_variable cv_job, cv_done;
    std::function<void()> job; uint64_t generation = 0; int pending = 0; bool stop = false;
    HostPool()
    {
        int nt = (int)std::thread::hardware_concurrency();
        nt = std::max(1, std::min(nt, 16));
        try { for (int t = 1; t < nt; t++) th.emplace_back([this] { loop(); }); } catch (...) {}
    }
    ~HostPool()
    {
        { std::lock_guard<std::mutex> g(mu); stop = true; }
        cv_job.notify_all();
        for (auto &x : th) x.join();
    }
    void loop()
    {
        uint64_t seen = 0;
        for (;;) {
            std::function<void()> f;
            {
                std::unique_lock<std::mutex> g(mu);
                cv_job.wait(g, [&] { return stop || generation != seen; });
                if (stop) return;
                seen = generation; f = job;
            }
            f();
            { std::lock_guard<std::mutex> g(mu); if (--pending == 0) cv_done.notify_all(); }
        }
    }
    // every worker and the caller run f once (f pulls its share from a shared counter)
    void run(const std::function<void()> &f)
    {
        { std::lock_guard<std::mutex> g(mu); job = f; pending = (int)th.size(); generation++; }
        cv_job.notify_all();
        f();
        std::unique_lock<std::mutex> g(mu);
        cv_done.wait(g, [&] { return pending == 0; });
    }
};
std::mutex g_pool_guard;              // one job at a time (contexts of several GPUs may call from several host threads)
std::atomic<bool> g_forked(false);    // a fork()ed child has no workers: it runs its jobs on the calling thread
// (never destroyed: the workers end with the process; a destructor would have to join threads a forked child does not have)
HostPool &host_pool()
{
    static HostPool *p = [] { pthread_atfork(nullptr, nullptr, [] { g_forked.store(true); }); return new HostPool; }();
    return *p;
}
}  // namespace

template <class F>
static void parallel_for(int64_t n, F &&fn)
{
    if (n < 64 || g_forked.load()) { for (int64_t b = 0; b < n; b++) fn(b); return; }
    std::unique_lock<std::mutex> only(g_pool_guard, std::try_to_lock);
    if (!only.owns_lock()) { for (int64_t b = 0; b < n; b++) fn(b); return; }      // (another GPU's host thread has the workers)
    std::atomic<int64_t> next(0);
    std::atomic<bool> failed(false);
    host_pool().run([&] {
        try {
            for (;;) {
                const int64_t b0 = next.fetch_add(16);
                if (b0 >= n || failed.load()) break;
                for (int64_t b = b0; b < std::min(n, b0 + 16); b++) fn(b);
            }
        } catch (...) { failed.store(true); }          // (out of host memory in a worker: reported by the calling thread)
    });
    if (failed.load()) throw std::bad_alloc();
}

// ------------------------------------------------------------ full G path
struct Struct {
    std::vector<Stem3> stems; uint64_t psmask; double score[3]; uint8_t isint0;
    std::vector<std::pair<int, int>> bps;      // sorted
    std::vector<int8_t> dbn;
};

static void stems_to_bps(const std::vector<Stem3> &st, std::vector<std::pair<int, int>> &bps)
{
    bps.clear();
    for (auto &s : st) for (int k = 0; k < s.len; k++) bps.emplace_back(s.i + k, s.j - k);
    std::sort(bps.begin(), bps.end());
}

struct Pool {                      // the pool of partial structures of one sequence (one paramset)
    std::vector<std::vector<Stem3>> cur;
    int cursize = 1; double cursubopt = 0; bool tail = false, done = false;
    std::vector<std::vector<Stem3>> fin;     // in finalisation order
};

static int copy_result(sqrn_ctx *ctx, sqrn_result *out)
{
    CachedResult &C = ctx->cres;
    out->need_structs = (int64_t)C.scores.size() / 3;
    out->need_stems = (int64_t)C.stems.size() / 3;
    out->need_dbn = (int64_t)C.dbn.size();
    if (out->cap_structs < out->need_structs || out->cap_stems < out->need_stems || out->cap_dbn < out->need_dbn) {
        ctx->err = "output capacity too small"; return SQRN_E_CAPACITY;
    }
    const size_t ns = (size_t)out->need_structs;
    memcpy(out->struct_offsets, C.struct_offsets.data(), C.struct_offsets.size() * sizeof(int64_t));
    if (ns) {
        memcpy(out->scores, C.scores.data(), ns * 3 * sizeof(double));
        memcpy(out->struct_is_int0, C.isint0.data(), ns);
        memcpy(out->psmask, C.psmask.data(), ns * sizeof(uint64_t));
        memcpy(out->dbn_offsets, C.dbn_offsets.data(), ns * sizeof(int64_t));
    }
    memcpy(out->stem_offsets, C.stem_offsets.data(), (ns + 1) * sizeof(int64_t));
    if (out->n_total) memcpy(out->n_total, C.n_total.data(), C.n_total.size() * sizeof(int32_t));
    if (!C.stems.empty()) memcpy(out->stems, C.stems.data(), C.stems.size() * sizeof(int32_t));
    if (!C.dbn.empty()) memcpy(out->dbn, C.dbn.data(), C.dbn.size());
    if (out->cons && !C.cons.empty()) memcpy(out->cons, C.cons.data(), C.cons.size());
    return SQRN_OK;
}

static int sqrn_predict_batch_impl(sqrn_ctx *ctx, const sqrn_paramset *ps, int n_ps, const sqrn_batch *in, sqrn_result *out)
{
    if (!ctx || !out) return SQRN_E_BADARG;
    cudaSetDevice(ctx->device);
    if (!in) {                                   // E_CAPACITY retry: hand out the cached result
        if (!ctx->cres.valid) { ctx->err = "no cached result"; return SQRN_E_BADARG; }
        return copy_result(ctx, out);
    }
    if (!ps || n_ps < 1 || n_ps > 64) { ctx->err = "need 1..64 parameter sets"; return SQRN_E_BADARG; }
    if (in->bpp_mode && n_ps != 1) { ctx->err = "a bpp term belongs to one parameter set: call with n_ps == 1"; return SQRN_E_BADARG; }
    ctx->cres.valid = false;
    ctx->n_launches = 0; ctx->n_calls = 0; ctx->kernel_ms = 0; ctx->n_cluster_launches = 0;
    const bool trace = getenv("SQRN_TRACE") != nullptr;
    auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    double t_mark = now(), t_upload = 0, t_base = 0, t_gather = 0, t_step = 0, t_scatter = 0, t_tail = 0, t_dedupe = 0, t_final = 0;
    auto lap = [&](double &acc) { const double t = now(); acc += t - t_mark; t_mark = t; };
    int n_rounds = 0;
    DeviceBatch D;
    TRY(upload_batch(ctx, in, D));
    const int64_t nseq = in->n_seqs;
    const int poollim = in->poollim;
    lap(t_upload);
    std::vector<std::vector<Struct>> uniq((size_t)nseq);
    std::vector<std::unordered_map<uint64_t, std::vector<int>>> index((size_t)nseq);

    for (int psi = 0; psi < n_ps; psi++) {
        const sqrn_paramset &P = ps[psi];
        const double inc = (P.suboptmax - P.suboptmin) / P.suboptsteps;          // seq.py:1071
        std::vector<Pool> pools((size_t)nseq);
        for (auto &pl : pools) { pl.cur.assign(1, {}); pl.cursize = 1; pl.cursubopt = P.suboptmin; }
        BaseDev base;
        if (poollim > 1) TRY(build_base(ctx, P, D, base));      // (pl = 1: the structures run to completion on their own persistent lists)
        lap(t_base);
        std::vector<std::pair<int, int>> tail_items;      // (seq, index in its pool) run to completion
        for (;;) {
            // round prologue per pool, seq.py:1161-1174 (per sequence, on a few host threads); then where every pool's
            // items and their pre-selected stems start in the flat arrays of the launch, and the fill (threads again)
            HostWork W; W.mode = MODE_STEP; W.base = &base;
            std::vector<int64_t> item0((size_t)nseq + 1, 0), stem0((size_t)nseq + 1, 0);
            parallel_for(nseq, [&](int64_t b) {
                Pool &pl = pools[b];
                if (pl.done || pl.tail) return;
                if (pl.cur.empty()) { pl.done = true; return; }
                if ((int)pl.cur.size() > pl.cursize) {
                    pl.cursize = (int)pl.cur.size();
                    if (pl.cursubopt < P.suboptmax) pl.cursubopt += inc;
                }
                std::vector<std::vector<Stem3>> keep;
                for (auto &st : pl.cur) {
                    if ((double)st.size() == P.maxstemnum) pl.fin.push_back(std::move(st));
                    else keep.push_back(std::move(st));
                }
                pl.cur.swap(keep);
                if (pl.cur.empty()) { pl.done = true; return; }
                if (pl.cursize >= poollim) { pl.tail = true; return; }    // stopper == 1 from now on
                int64_t ns = 0;
                for (auto &st : pl.cur) ns += (int64_t)st.size();
                item0[b + 1] = (int64_t)pl.cur.size(); stem0[b + 1] = ns;
            });
            for (int64_t b = 0; b < nseq; b++) { item0[b + 1] += item0[b]; stem0[b + 1] += stem0[b]; }
            const int64_t n_it = item0[nseq];
            if (n_it == 0) break;
            std::vector<std::pair<int, int>> owner((size_t)n_it);        // item -> (seq, pool index)
            W.item_seq.resize((size_t)n_it); W.subopt.resize((size_t)n_it);
            W.init_off.resize((size_t)n_it + 1); W.init_stems.resize((size_t)stem0[nseq] * 3);
            W.init_off[(size_t)n_it] = stem0[nseq];
            parallel_for(nseq, [&](int64_t b) {
                if (item0[b + 1] == item0[b]) return;
                Pool &pl = pools[b];
                int64_t k = item0[b], so = stem0[b];
                for (size_t q = 0; q < pl.cur.size(); q++, k++) {
                    W.item_seq[(size_t)k] = (int32_t)b; W.subopt[(size_t)k] = pl.cursubopt; owner[(size_t)k] = std::make_pair((int)b, (int)q);
                    W.init_off[(size_t)k] = so;
                    for (auto &st : pl.cur[q]) { W.init_stems[3 * (size_t)so] = st.i; W.init_stems[3 * (size_t)so + 1] = st.j; W.init_stems[3 * (size_t)so + 2] = st.len; so++; }
                }
            });
            lap(t_gather); n_rounds++;
            TRY(run_step_items(ctx, P, D, W));
            lap(t_step);
            // seq.py:1179-1199: children in pool order, or finalise (per sequence, on a few host threads)
            parallel_for(nseq, [&](int64_t b) {
                if (item0[b + 1] == item0[b]) return;
                Pool &pl = pools[b];
                std::vector<std::vector<Stem3>> next;
                for (int64_t k = item0[b]; k < item0[b + 1]; k++) {
                    auto &st = pl.cur[(size_t)(k - item0[b])];
                    const int nnew = W.out_n[(size_t)k];
                    if (nnew == 0) { pl.fin.push_back(std::move(st)); continue; }
                    for (int q = 0; q < nnew; q++) {
                        const int32_t *o = &W.out_stems[3 * (W.out_off[(size_t)k] + q)];
                        if (q + 1 == nnew) { st.push_back(Stem3{ o[0], o[1], o[2] }); next.push_back(std::move(st)); break; }   // the last child takes the parent's storage
                        std::vector<Stem3> child; child.reserve(st.size() + 1);
                        child = st;
                        child.push_back(Stem3{ o[0], o[1], o[2] });
                        next.push_back(std::move(child));
                    }
                }
                pl.cur.swap(next);
            });
            lap(t_scatter);
        }
        lap(t_gather);
        // tail phase: every remaining structure runs to completion on its own (items and results per sequence, on the
        // host threads)
        {
            HostWork W; W.mode = MODE_TAIL; W.base = &base;
            std::vector<int64_t> item0((size_t)nseq + 1, 0), stem0((size_t)nseq + 1, 0);
            for (int64_t b = 0; b < nseq; b++) {
                const Pool &pl = pools[b];
                int64_t ni = 0, ns = 0;
                if (pl.tail) { ni = (int64_t)pl.cur.size(); for (auto &st : pl.cur) ns += (int64_t)st.size(); }
                item0[b + 1] = item0[b] + ni; stem0[b + 1] = stem0[b] + ns;
            }
            const int64_t n_it = item0[nseq];
            if (n_it > 0) {
                W.item_seq.resize((size_t)n_it); W.out_cap.resize((size_t)n_it);
                W.init_off.resize((size_t)n_it + 1); W.init_stems.resize((size_t)stem0[nseq] * 3);
                W.init_off[(size_t)n_it] = stem0[nseq];
                parallel_for(nseq, [&](int64_t b) {
                    if (item0[b + 1] == item0[b]) return;
                    const Pool &pl = pools[b];
                    int64_t k = item0[b], so = stem0[b];
                    for (size_t q = 0; q < pl.cur.size(); q++, k++) {
                        W.item_seq[(size_t)k] = (int32_t)b; W.out_cap[(size_t)k] = D.len[b] / 2 + 1;
                        W.init_off[(size_t)k] = so;
                        for (auto &st : pl.cur[q]) { W.init_stems[3 * (size_t)so] = st.i; W.init_stems[3 * (size_t)so + 1] = st.j; W.init_stems[3 * (size_t)so + 2] = st.len; so++; }
                    }
                });
                TRY(run_items(ctx, P, D, W));
                // finalisation order inside the tail: by round (= stems added), structures that hit
                // maxstemnum before those that ran dry, then pool order (seq.py:1168-1196)
                struct Key { int round, kind, idx; size_t item; };
                parallel_for(nseq, [&](int64_t b) {
                    if (item0[b + 1] == item0[b]) return;
                    Pool &pl = pools[b];
                    std::vector<Key> kv;
                    kv.reserve((size_t)(item0[b + 1] - item0[b]));
                    for (int64_t k = item0[b]; k < item0[b + 1]; k++) {
                        const int q = (int)(k - item0[b]);
                        const int n0 = (int)pl.cur[(size_t)q].size(), n1 = W.out_n[(size_t)k];
                        kv.push_back(Key{ n1 - n0, ((double)n1 == P.maxstemnum) ? 0 : 1, q, (size_t)k });
                    }
                    std::stable_sort(kv.begin(), kv.end(), [](const Key &x, const Key &y) {
                        if (x.round != y.round) return x.round < y.round;
                        if (x.kind != y.kind) return x.kind < y.kind;
                        return x.idx < y.idx; });
                    for (auto &key : kv) {
                        std::vector<Stem3> st((size_t)W.out_n[key.item]);
                        for (int q = 0; q < W.out_n[key.item]; q++) {
                            const int32_t *o = &W.out_stems[3 * (W.out_off[key.item] + q)];
                            st[(size_t)q] = Stem3{ o[0], o[1], o[2] };
                        }
                        pl.fin.push_back(std::move(st));
                    }
                });
            }
        }
        lap(t_tail);
        // dedupe by bp set across parameter sets, seq.py:1201-1212
        parallel_for(nseq, [&](int64_t b) {
            for (auto &st : pools[b].fin) {
                std::vector<std::pair<int, int>> bps;
                stems_to_bps(st, bps);
                uint64_t h = 1469598103934665603ull;
                for (auto &p : bps) { h = (h ^ (uint64_t)p.first) * 1099511628211ull; h = (h ^ (uint64_t)p.second) * 1099511628211ull; }
                int hit = -1;
                for (int cand : index[b][h]) if (uniq[b][cand].bps == bps) { hit = cand; break; }
                if (hit >= 0) { uniq[b][hit].psmask |= 1ull << psi; continue; }
                Struct S; S.stems = std::move(st); S.psmask = 1ull << psi; S.bps.swap(bps);
                S.score[0] = S.score[1] = S.score[2] = 0; S.isint0 = 1;
                index[b][h].push_back((int)uniq[b].size());
                uniq[b].push_back(std::move(S));
            }
        });
    }

    lap(t_dedupe);
    // ScoreStruct + dbn of every unique structure on the device (MODE_FINAL)
    {
        HostWork W; W.mode = MODE_FINAL; W.want_dbn = true;
        std::vector<size_t> first((size_t)nseq + 1, 0);
        std::vector<int64_t> stem0((size_t)nseq + 1, 0);
        for (int64_t b = 0; b < nseq; b++) {
            first[b + 1] = first[b] + uniq[b].size();
            int64_t ns = 0;
            for (auto &S : uniq[b]) ns += (int64_t)S.stems.size();
            stem0[b + 1] = stem0[b] + ns;
        }
        const size_t n_it = first[(size_t)nseq];
        W.item_seq.resize(n_it); W.out_cap.assign(n_it, 0);
        W.init_off.resize(n_it + 1); W.init_stems.resize((size_t)stem0[nseq] * 3);
        W.init_off[n_it] = stem0[nseq];
        parallel_for(nseq, [&](int64_t b) {
            size_t k = first[b]; int64_t so = stem0[b];
            for (auto &S : uniq[b]) {
                W.item_seq[k] = (int32_t)b; W.init_off[k] = so;
                for (auto &st : S.stems) { W.init_stems[3 * (size_t)so] = st.i; W.init_stems[3 * (size_t)so + 1] = st.j; W.init_stems[3 * (size_t)so + 2] = st.len; so++; }
                k++;
            }
        });
        TRY(run_items(ctx, ps[0], D, W));
        parallel_for(nseq, [&](int64_t b) {
            size_t k = first[b];
            for (auto &S : uniq[b]) {
                for (int t = 0; t < 3; t++) S.score[t] = pyround3(W.out_raw[3 * k + t]);     // seq.py:899
                S.isint0 = W.flags[k] & 1;       // (flag 2, more than 30 levels: the int8 level codes of this output go up to 127)
                S.dbn.assign(W.dbn.begin() + W.dbn_off[k], W.dbn.begin() + W.dbn_off[k + 1]);
                k++;
            }
        });
    }

    lap(t_final);
    // rank (RankStructs, seq.py:902-955), forced pairs, consensus, truncate
    CachedResult &C = ctx->cres;
    C = CachedResult();
    C.n_seqs = nseq; C.total_len = in->offsets[nseq];
    C.struct_offsets.assign((size_t)nseq + 1, 0);
    C.n_total.assign((size_t)nseq, 0);
    C.cons.assign((size_t)C.total_len, 0);
    const int *rb = in->rankby;
    if (!(rb[0] >= 0 && rb[0] < 3 && rb[1] >= 0 && rb[1] < 3 && rb[2] >= 0 && rb[2] < 3 && rb[0] != rb[1] && rb[0] != rb[2] && rb[1] != rb[2])) {
        ctx->err = "Invalid ranking indices"; return SQRN_E_BADARG;
    }
    HostParams HP;           // symbol codes of the last paramset, for the hardrest key test
    if (in->hardrest) { std::string e; if (!build_host_params(ps[n_ps - 1], 16, HP, e)) { ctx->err = e; return SQRN_E_UNSUPPORTED; } }
    // pass 1 (per sequence, in parallel): the final order; pass 2: where every sequence's output starts; pass 3 (in
    // parallel): the output arrays
    std::vector<std::vector<int>> order((size_t)nseq);
    std::vector<int> keepn((size_t)nseq, 0);
    std::vector<int64_t> stems_of((size_t)nseq + 1, 0);
    parallel_for(nseq, [&](int64_t b) {
        auto &U = uniq[b];
        const int n = (int)U.size(), N = D.len[b];
        std::vector<int> &idx = order[b];
        idx.resize((size_t)n);
        for (int k = 0; k < n; k++) idx[k] = k;
        auto keycmp = [&](int x, int y) {      // > 0 when x ranks before y
            for (int t = 0; t < 3; t++) {
                double a = U[x].score[rb[t]], c = U[y].score[rb[t]];
                if (a > c) return 1;
                if (a < c) return -1;
            }
            return 0;
        };
        std::stable_sort(idx.begin(), idx.end(), [&](int x, int y) { return keycmp(x, y) > 0; });
        std::stable_partition(idx.begin(), idx.end(), [&](int x) { return (U[x].psmask & in->priority_mask) != 0; });
        if (in->rankbydiff && n >= 3) {
            std::vector<uint8_t> seen((size_t)N * N, 0), all((size_t)N * N, 0);
            size_t nall = 0, nseen = 0;
            for (auto &S : U) for (auto &p : S.bps) { size_t c = (size_t)p.first * N + p.second; if (!all[c]) { all[c] = 1; nall++; } }
            auto mark = [&](const Struct &S) { for (auto &p : S.bps) { size_t c = (size_t)p.first * N + p.second; if (!seen[c]) { seen[c] = 1; nseen++; } } };
            mark(U[idx[0]]);
            int cur = 1;
            std::vector<int> extra((size_t)n, 0);
            while (nseen != nall && cur < n - 1) {
                for (int k = cur; k < n; k++) {
                    int e = 0;
                    for (auto &p : U[idx[k]].bps) if (!seen[(size_t)p.first * N + p.second]) e++;
                    extra[idx[k]] = e;
                }
                std::stable_sort(idx.begin() + cur, idx.end(), [&](int x, int y) {
                    if (extra[x] != extra[y]) return extra[x] > extra[y];
                    return keycmp(x, y) > 0; });
                mark(U[idx[cur]]);
                cur++;
            }
            std::stable_sort(idx.begin() + cur, idx.end(), [&](int x, int y) { return keycmp(x, y) > 0; });
        }
        C.n_total[b] = n;
        keepn[b] = (in->max_structs > 0 && in->max_structs < n) ? in->max_structs : n;
        int64_t ns = 0;
        for (int r = 0; r < keepn[b]; r++) ns += (int64_t)U[idx[r]].stems.size();
        stems_of[b + 1] = ns;
    });
    for (int64_t b = 0; b < nseq; b++) {
        C.struct_offsets[b + 1] = C.struct_offsets[b] + keepn[b];
        stems_of[b + 1] += stems_of[b];
    }
    const int64_t n_out = C.struct_offsets[nseq];
    C.scores.resize((size_t)n_out * 3); C.isint0.resize((size_t)n_out); C.psmask.resize((size_t)n_out);
    C.stem_offsets.resize((size_t)n_out + 1); C.dbn_offsets.resize((size_t)n_out);
    C.stems.resize((size_t)stems_of[nseq] * 3);
    std::vector<int64_t> dbn_of((size_t)nseq + 1, 0);
    for (int64_t b = 0; b < nseq; b++) dbn_of[b + 1] = dbn_of[b] + (int64_t)keepn[b] * D.len[b];
    C.dbn.resize((size_t)dbn_of[nseq]);
    C.stem_offsets[(size_t)n_out] = stems_of[nseq];
    parallel_for(nseq, [&](int64_t b) {
        auto &U = uniq[b];
        const int n = (int)U.size(), N = D.len[b];
        const std::vector<int> &idx = order[b];
        // forced pairs, seq.py:1226-1228
        std::vector<std::pair<int, int>> forced;
        if (in->hardrest && in->rbp_offsets) {
            const uint8_t *sym = in->symbols + in->offsets[b];
            for (int64_t k = in->rbp_offsets[b]; k < in->rbp_offsets[b + 1]; k++) {
                int v = in->rbps[2 * k], w = in->rbps[2 * k + 1];
                // "seq[v]+seq[w] in bpweights" on the normalised symbols == the pair mask of the digest
                int cv = HP.p.code_table[sym[v]], cw = HP.p.code_table[sym[w]];
                if (HP.p.pairmask[cv] >> cw & 1) forced.emplace_back(v, w);
            }
        }
        int64_t so = stems_of[b];
        for (int r = 0; r < keepn[b]; r++) {
            Struct &S = U[idx[r]];
            const size_t k = (size_t)(C.struct_offsets[b] + r);
            for (int t = 0; t < 3; t++) C.scores[3 * k + t] = S.score[t];
            C.isint0[k] = S.isint0; C.psmask[k] = S.psmask;
            C.stem_offsets[k] = so;
            for (auto &st : S.stems) { C.stems[3 * (size_t)so] = st.i; C.stems[3 * (size_t)so + 1] = st.j; C.stems[3 * (size_t)so + 2] = st.len; so++; }
            const int64_t o = dbn_of[b] + (int64_t)r * N;
            C.dbn_offsets[k] = o;
            if (forced.empty()) { if (N) memcpy(C.dbn.data() + o, S.dbn.data(), (size_t)N); }
            else {
                std::vector<std::pair<int, int>> pp = S.bps; pp.insert(pp.end(), forced.begin(), forced.end());
                pairs_to_codes(pp, N, C.dbn.data() + o);
            }
        }
        // consensus of the top conslim structures, seq.py:845-858, 1236
        {
            int top = std::min(std::max(in->conslim, 0), n);
            std::vector<std::pair<int, int>> cb;
            if (top > 0) {
                cb = U[idx[0]].bps;
                for (int r = 1; r < top; r++) {
                    std::vector<std::pair<int, int>> t;
                    std::set_intersection(cb.begin(), cb.end(), U[idx[r]].bps.begin(), U[idx[r]].bps.end(), std::back_inserter(t));
                    cb.swap(t);
                }
            }
            int8_t *dst = C.cons.data() + in->offsets[b];
            if (top == 1 && forced.empty()) { if (N) memcpy(dst, U[idx[0]].dbn.data(), (size_t)N); }
            else { cb.insert(cb.end(), forced.begin(), forced.end()); pairs_to_codes(cb, N, dst); }
        }
    });
    C.valid = true;
    if (trace) {
        double t_rank = 0; lap(t_rank);
        fprintf(stderr, "[sqrn] predict_batch: %lld sequences x %d parameter sets, %d rounds, %lld launches, kernels %.1f ms; host ms: upload %.1f, "
                "base lists %.1f, gather %.1f, step rounds %.1f, scatter %.1f, tails %.1f, dedupe %.1f, final %.1f, rank + output %.1f\n",
                (long long)nseq, n_ps, n_rounds, (long long)ctx->n_launches, ctx->kernel_ms, t_upload, t_base, t_gather, t_step, t_scatter,
                t_tail, t_dedupe, t_final, t_rank);
    }
    return copy_result(ctx, out);
}

extern "C" int sqrn_predict_batch(sqrn_ctx *ctx, const sqrn_paramset *ps, int n_ps, const sqrn_batch *in, sqrn_result *out)
{
    return guarded(ctx, [&] { return sqrn_predict_batch_impl(ctx, ps, n_ps, in, out); });
}

// ------------------------------------------------- alignment step 1 on the device
// SQRNdbnali (ali.py:211-242) sums the score of every stem of every sequence into the cells of its base pairs, sequence
// after sequence -- and float64 addition order is observable.  Here every CTA owns a band of matrix ROWS and walks the
// stems of ALL sequences in sequence order (they sit in device memory, written by the YieldStems kernel; the stream of
// (i, j, len, score) records is read through L2 by every band); within one sequence a cell belongs to at most one stem,
// so the threads of a CTA never meet on a cell, and a barrier per sequence keeps the order: the additions every cell sees
// are exactly the reference's, without atomics or sorting.  Only the upper triangle is accumulated (the reference adds the
// same value to [v, w] and [w, v]); k_mirror fills the rest.
__global__ void __launch_bounds__(256)
k_stem_matrix(int64_t n_seqs, const int64_t *__restrict__ seq_off, const int32_t *__restrict__ cols,
              const int64_t *__restrict__ st_off, const int32_t *__restrict__ st_n, const int32_t *__restrict__ stems,
              const double *__restrict__ score, int L, int rows_per_band, double *__restrict__ mat)
{
    const int r0 = blockIdx.x * rows_per_band, r1 = min(L, r0 + rows_per_band);
    for (int64_t b = 0; b < n_seqs; b++) {
        const int32_t *cb = cols + seq_off[b];
        const int64_t o = st_off[b];
        const int ns = st_n[b];
        for (int k = threadIdx.x; k < ns; k += blockDim.x) {
            const int i = stems[3 * (o + k)], j = stems[3 * (o + k) + 1], len = stems[3 * (o + k) + 2];
            // rows of the stem's cells: cols[i] .. cols[i + len - 1], increasing
            if (cb[i] >= r1 || cb[i + len - 1] < r0) continue;
            const double sc = score[o + k];
            for (int q = 0; q < len; q++) {
                const int v = cb[i + q], w = cb[j - q];
                if (v >= r0 && v < r1) mat[(int64_t)v * L + w] += sc;          // (v < w: i + q < j - q and cols increase)
            }
        }
        __syncthreads();
    }
}

__global__ void k_mirror(int L, double *__restrict__ mat)
{
    const int64_t n = (int64_t)L * L;
    for (int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; c < n; c += (int64_t)gridDim.x * blockDim.x) {
        const int v = (int)(c / L), w = (int)(c % L);
        if (v > w) mat[c] = mat[(int64_t)w * L + v];
    }
}

// MatrixToDBNs (ali.py:133-150) looks at the cells in stable descending order of their value, stops below the threshold
// and skips w - v < 4: the cells that pass both tests are collected, then ranked by counting (value descending, flat
// index ascending) -- a few hundred conserved pairs on real alignments.
__global__ void k_cells_collect(int L, const double *__restrict__ mat, double thr, int cap, int *__restrict__ count, int32_t *__restrict__ cells)
{
    const int64_t n = (int64_t)L * L;
    for (int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; c < n; c += (int64_t)gridDim.x * blockDim.x) {
        const int v = (int)(c / L), w = (int)(c % L);
        if (w - v >= 4 && !(mat[c] < thr)) { const int slot = atomicAdd(count, 1); if (slot < cap) cells[slot] = (int32_t)c; }
    }
}
__global__ void k_cells_rank(int m, const double *__restrict__ mat, const int32_t *__restrict__ cells, int32_t *__restrict__ sorted)
{
    for (int a = blockIdx.x * blockDim.x + threadIdx.x; a < m; a += gridDim.x * blockDim.x) {
        const int32_t ca = cells[a]; const double va = mat[ca];
        int rank = 0;
        for (int b = 0; b < m; b++) { const int32_t c = cells[b]; const double v = mat[c]; if (v > va || (v == va && c < ca)) rank++; }
        sorted[rank] = ca;
    }
}

static int sqrn_stem_matrix_batch_impl(sqrn_ctx *ctx, const sqrn_paramset *ps, const sqrn_batch *in, double *matrix,
                                      double threshold, int64_t cap_cells, int64_t *n_cells, int32_t *cells)
{
    if (!ctx || !ps || !in || !matrix || !n_cells) return SQRN_E_BADARG;
    if (in->smat || !in->cols || in->smat_L <= 0) { ctx->err = "stem matrix: need the column map (cols, smat_L = alignment length) and no smat"; return SQRN_E_BADARG; }
    cudaSetDevice(ctx->device);
    ctx->n_launches = 0; ctx->n_calls = 0; ctx->kernel_ms = 0; ctx->n_cluster_launches = 0;
    const int L = in->smat_L;
    const int64_t nseq = in->n_seqs, total = in->offsets[nseq];
    for (int64_t b = 0; b < nseq; b++)                 // columns of a row: inside the alignment, strictly increasing
        for (int64_t k = in->offsets[b]; k < in->offsets[b + 1]; k++)
            if (in->cols[k] < 0 || in->cols[k] >= L || (k > in->offsets[b] && in->cols[k] <= in->cols[k - 1])) {
                ctx->err = "stem matrix: the column map of a row must be strictly increasing and inside the alignment"; return SQRN_E_BADARG;
            }
    DeviceBatch D;
    TRY(upload_batch(ctx, in, D));
    HostWork W; W.mode = MODE_YIELD; W.keep_on_device = true;
    for (int64_t b = 0; b < nseq; b++) {
        W.item_seq.push_back((int32_t)b);
        const double n = D.len[b];
        W.out_cap.push_back((int64_t)(0.03 * n * n) + 64);
    }
    TRY(run_items(ctx, *ps, D, W));
    bool redo = false;
    for (int64_t b = 0; b < nseq; b++) if (W.out_n[b] > W.out_cap[b]) { W.out_cap[b] = W.out_n[b]; redo = true; }
    if (redo) TRY(run_items(ctx, *ps, D, W));
    int32_t *d_cols; double *d_mat; int *d_cnt; int32_t *d_cells, *d_sorted;
    TRY(upload(ctx, B_COLS, in->cols, (size_t)total, &d_cols));
    TRY(dalloc(ctx, W_MAT, (size_t)L * L, &d_mat));
    const int cap = (int)std::min<int64_t>(std::max<int64_t>(cap_cells, 0), 1 << 16);
    TRY(dalloc(ctx, W_CELLCNT, 1, &d_cnt));
    TRY(dalloc(ctx, W_CELLS, (size_t)std::max(cap, 1), &d_cells));
    TRY(dalloc(ctx, W_CELLS2, (size_t)std::max(cap, 1), &d_sorted));
    cudaStream_t st = ctx->stream;
    CK(cudaMemsetAsync(d_mat, 0, (size_t)L * L * sizeof(double), st));
    CK(cudaMemsetAsync(d_cnt, 0, sizeof(int), st));
    const int bands = std::max(1, std::min(L, 2 * ctx->sm_count)), rpb = (L + bands - 1) / bands;
    k_stem_matrix<<<(L + rpb - 1) / rpb, 256, 0, st>>>(nseq, D.B.off, d_cols, W.d_out_off, W.d_out_n, W.d_out_stems, W.d_out_fin, L, rpb, d_mat);
    CK(cudaGetLastError());
    k_mirror<<<2 * ctx->sm_count, 256, 0, st>>>(L, d_mat);
    k_cells_collect<<<2 * ctx->sm_count, 256, 0, st>>>(L, d_mat, threshold, cap, d_cnt, d_cells);
    CK(cudaGetLastError());
    int m = 0;
    CK(cudaMemcpyAsync(&m, d_cnt, sizeof m, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(matrix, d_mat, (size_t)L * L * sizeof(double), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    ctx->n_launches += 3;
    *n_cells = m;
    if (m > cap) { *n_cells = -1; return SQRN_OK; }      // more cells than the caller (or the device ranking) takes: the caller sorts the matrix itself
    if (m > 0) {
        if (!cells) return SQRN_E_BADARG;
        k_cells_rank<<<std::min(2 * ctx->sm_count, (m + 255) / 256), 256, 0, st>>>(m, d_mat, d_cells, d_sorted);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(cells, d_sorted, (size_t)m * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        ctx->n_launches++;
    }
    return SQRN_OK;
}

extern "C" int sqrn_stem_matrix_batch(sqrn_ctx *ctx, const sqrn_paramset *ps, const sqrn_batch *in, double *matrix,
                                      double threshold, int64_t cap_cells, int64_t *n_cells, int32_t *cells)
{
    return guarded(ctx, [&] { return sqrn_stem_matrix_batch_impl(ctx, ps, in, matrix, threshold, cap_cells, n_cells, cells); });
}

// ------------------------------------------------------------- YieldStems
static int sqrn_yield_stems_batch_impl(sqrn_ctx *ctx, const sqrn_paramset *ps, const sqrn_batch *in, sqrn_stems *out)
{
    if (!ctx || !out) return SQRN_E_BADARG;
    cudaSetDevice(ctx->device);
    CachedStems &C = ctx->cstems;
    if (in) {
        if (!ps) return SQRN_E_BADARG;
        C.valid = false;
        ctx->n_launches = 0; ctx->n_calls = 0; ctx->kernel_ms = 0; ctx->n_cluster_launches = 0;
        DeviceBatch D;
        TRY(upload_batch(ctx, in, D));
        const int64_t nseq = in->n_seqs;
        HostWork W; W.mode = MODE_YIELD;
        for (int64_t b = 0; b < nseq; b++) {
            W.item_seq.push_back((int32_t)b);
            double n = D.len[b];
            W.out_cap.push_back((int64_t)(0.03 * n * n) + 64);
        }
        TRY(run_items(ctx, *ps, D, W));
        bool redo = false;
        for (int64_t b = 0; b < nseq; b++) if (W.out_n[b] > W.out_cap[b]) { W.out_cap[b] = W.out_n[b]; redo = true; }
        if (redo) TRY(run_items(ctx, *ps, D, W));
        C.n_seqs = nseq; C.off.assign((size_t)nseq + 1, 0); C.stems.clear(); C.scores.clear();
        for (int64_t b = 0; b < nseq; b++) {
            int n = W.out_n[b];
            C.off[b + 1] = C.off[b] + n;
            C.stems.insert(C.stems.end(), W.out_stems.begin() + 3 * W.out_off[b], W.out_stems.begin() + 3 * (W.out_off[b] + n));
            C.scores.insert(C.scores.end(), W.out_fin.begin() + W.out_off[b], W.out_fin.begin() + W.out_off[b] + n);
        }
        C.valid = true;
    } else if (!C.valid) { ctx->err = "no cached result"; return SQRN_E_BADARG; }
    out->need_stems = (int64_t)C.scores.size();
    if (out->cap_stems < out->need_stems) { ctx->err = "output capacity too small"; return SQRN_E_CAPACITY; }
    memcpy(out->stem_offsets, C.off.data(), C.off.size() * sizeof(int64_t));
    if (!C.scores.empty()) {
        memcpy(out->stems, C.stems.data(), C.stems.size() * sizeof(int32_t));
        memcpy(out->scores, C.scores.data(), C.scores.size() * sizeof(double));
    }
    return SQRN_OK;
}

extern "C" int sqrn_yield_stems_batch(sqrn_ctx *ctx, const sqrn_paramset *ps, const sqrn_batch *in, sqrn_stems *out)
{
    return guarded(ctx, [&] { return sqrn_yield_stems_batch_impl(ctx, ps, in, out); });
}

// ------------------------------------------------------------- test seam
// One launch of the work kernel on host buffers, any mode: lets the GPU tests
// check AnnotateStems / OptimalStems seams against the oracle with arbitrary
// pre-selected stems.  Same argument meaning as the DevWork fields.
static int sqrn_debug_run_impl(sqrn_ctx *ctx, const sqrn_paramset *ps, const sqrn_batch *in, int mode, int n_items,
                              const int32_t *item_seq, const int64_t *init_off, const int32_t *init_stems,
                              const double *item_subopt, const int64_t *out_cap, int32_t *out_stems, int32_t *out_n,
                              double *out_fin, double *out_raw, uint8_t *out_flags, int8_t *dbn_code, int min_ccap)
{
    if (!ctx || !ps || !in) return SQRN_E_BADARG;
    cudaSetDevice(ctx->device);
    ctx->n_launches = 0; ctx->n_calls = 0; ctx->kernel_ms = 0; ctx->n_cluster_launches = 0;
    DeviceBatch D;
    TRY(upload_batch(ctx, in, D));
    HostWork W; W.mode = mode; W.want_dbn = dbn_code != nullptr; W.want_fin = out_fin != nullptr;
    for (int k = 0; k < n_items; k++) {
        W.item_seq.push_back(item_seq ? item_seq[k] : k);
        W.out_cap.push_back(out_cap[k]);
        if (item_subopt) W.subopt.push_back(item_subopt[k]);
    }
    if (mode == MODE_STEP && !item_subopt) W.subopt.assign((size_t)n_items, 1.0);
    if (init_off) {
        W.init_off.assign(init_off, init_off + n_items + 1);
        W.init_stems.assign(init_stems, init_stems + 3 * init_off[n_items]);
    }
    TRY(run_items(ctx, *ps, D, W, min_ccap));
    memcpy(out_n, W.out_n.data(), (size_t)n_items * sizeof(int32_t));
    if (!W.out_stems.empty()) memcpy(out_stems, W.out_stems.data(), W.out_stems.size() * sizeof(int32_t));
    if (out_fin && !W.out_fin.empty()) memcpy(out_fin, W.out_fin.data(), W.out_fin.size() * sizeof(double));
    if (out_raw && !W.out_raw.empty()) memcpy(out_raw, W.out_raw.data(), W.out_raw.size() * sizeof(double));
    if (out_flags && !W.flags.empty()) memcpy(out_flags, W.flags.data(), W.flags.size());
    if (dbn_code && !W.dbn.empty()) memcpy(dbn_code, W.dbn.data(), W.dbn.size());
    return SQRN_OK;
}

extern "C" int sqrn_debug_run(sqrn_ctx *ctx, const sqrn_paramset *ps, const sqrn_batch *in, int mode, int n_items,
                              const int32_t *item_seq, const int64_t *init_off, const int32_t *init_stems,
                              const double *item_subopt, const int64_t *out_cap, int32_t *out_stems, int32_t *out_n,
                              double *out_fin, double *out_raw, uint8_t *out_flags, int8_t *dbn_code, int min_ccap)
{
    return guarded(ctx, [&] { return sqrn_debug_run_impl(ctx, ps, in, mode, n_items, item_seq, init_off, init_stems, item_subopt, out_cap, out_stems, out_n, out_fin, out_raw, out_flags, dbn_code, min_ccap); });
}

// ------------------------------------------------------------- Nussinov
// The DP and the backtrack of sqrn_nussinov.cuh.  Persistent CTAs, each with its own workspace slot, take the
// sequences of a tier longest first from a counter.  Shared-memory tier: the whole triangle in shared memory, for
// sequences up to nu_smem_max_n(opt-in limit) positions; global tier: the triangle in the CTA's slot in HBM.  K (int16)
// is in the slot for both.  The whole workspace (the global tier's slots and the shared-memory tier's K) takes at most
// NU_WORKSPACE_CAP bytes, but at least one global slot (1.28 GB at 16 000 nt; 11 MB at 1 500 nt).  The context keeps
// it between calls at the exact size the largest call needed (re-allocating 4 GiB per call cost more than the 500 x
// 300-1500 nt DP itself) and frees it in sqrn_ctx_destroy.  The two tiers run concurrently on two streams, so the short
// sequences do not wait for the longest long one.
constexpr int64_t NU_WORKSPACE_CAP = (int64_t)4 << 30;

template <int TW, bool SMEM>
__global__ void __launch_bounds__(TW * 32, 1)
k_nussinov(NuBatch nb, NuLayout L)
{
    extern __shared__ __align__(16) unsigned char smem[];
    int *s_item = (int *)(smem + L.item_off);
    const int64_t slot = blockIdx.x;
    double *tri = SMEM ? (double *)smem : nb.wd + slot * nb.slot_d;
    double *prevbuf = SMEM ? nullptr : (double *)(smem + L.prev_off);
    int16_t *K = nb.wk + slot * nb.slot_k;
    double *sb = SMEM ? nullptr : nb.wbest + slot * nb.slot_s;
    int16_t *sk = SMEM ? nullptr : nb.wbk + slot * nb.slot_s;
    for (;;) {
        if (threadIdx.x == 0) *s_item = atomicAdd(nb.counter, 1);
        __syncthreads();
        const int item = *s_item;
        __syncthreads();
        if (item >= nb.n_items) break;
        nu_item<TW>(nb, nb.order[item], tri, prevbuf, L, smem, K, sb, sk);
    }
}

static int64_t nu_round8(int64_t x) { return (x + 7) & ~(int64_t)7; }

static int sqrn_nussinov_batch_impl(sqrn_ctx *ctx, int64_t n_seqs, const int64_t *offsets, const uint8_t *symbols,
                                    const int64_t *stem_offsets, const int32_t *stems, const double *scores,
                                    int32_t minloop, int64_t *pair_offsets, int32_t *pairs)
{
    if (!ctx) return SQRN_E_BADARG;
    if (n_seqs < 0 || n_seqs >= (1LL << 31) || !offsets || !stem_offsets || !pair_offsets || minloop < 0 || offsets[0] != 0) {
        ctx->err = "nussinov: bad arguments (offsets / stem_offsets / pair_offsets must be given, offsets[0] == 0, minloop >= 0)";
        return SQRN_E_BADARG;
    }
    cudaSetDevice(ctx->device);
    ctx->n_launches = 0; ctx->n_calls = 0; ctx->kernel_ms = 0; ctx->n_cluster_launches = 0;
    std::vector<int64_t> out_base((size_t)n_seqs + 1, 0);
    for (int64_t b = 0; b < n_seqs; b++) {
        const int64_t n = offsets[b + 1] - offsets[b], ns = stem_offsets[b + 1] - stem_offsets[b];
        if (n < 0 || n > SQRN_MAX_LEN || ns < 0) {
            ctx->err = "nussinov: offsets must not decrease and a sequence may have at most SQRN_MAX_LEN positions";
            return SQRN_E_BADARG;
        }
        if (ns > 0 && (!stems || !scores)) { ctx->err = "nussinov: stems / scores missing"; return SQRN_E_BADARG; }
        if (ns > 0 && !nu_stems_ok((int)n, stems + 3 * stem_offsets[b], ns)) {
            ctx->err = "nussinov: a stem of sequence " + std::to_string(b) + " leaves [0, N) or has len < 1";
            return SQRN_E_BADARG;
        }
        out_base[(size_t)b + 1] = out_base[(size_t)b] + n / 2;
    }
    const int64_t total = offsets[n_seqs], cap = out_base[(size_t)n_seqs];
    if ((total > 0 && !symbols) || (cap > 0 && !pairs)) { ctx->err = "nussinov: symbols / pairs missing"; return SQRN_E_BADARG; }
    pair_offsets[0] = 0;
    if (n_seqs == 0) return SQRN_OK;

    // candidate lists P(j) per sequence (host threads), then one flat CSR: sequence b's column pointers at offsets[b] + b
    std::vector<std::vector<int64_t>> cnt((size_t)n_seqs);
    std::vector<std::vector<int16_t>> lk((size_t)n_seqs);
    std::vector<std::vector<double>> le((size_t)n_seqs);
    parallel_for(n_seqs, [&](int64_t b) {
        nu_seq_lists((int)(offsets[b + 1] - offsets[b]), stems ? stems + 3 * stem_offsets[b] : nullptr,
                     scores ? scores + stem_offsets[b] : nullptr, stem_offsets[b + 1] - stem_offsets[b], cnt[(size_t)b], lk[(size_t)b], le[(size_t)b]);
    });
    std::vector<int64_t> pbase((size_t)n_seqs + 1, 0);
    for (int64_t b = 0; b < n_seqs; b++) pbase[(size_t)b + 1] = pbase[(size_t)b] + (int64_t)lk[(size_t)b].size();
    std::vector<int64_t> colptr((size_t)(total + n_seqs));
    std::vector<int16_t> pk((size_t)std::max<int64_t>(pbase[(size_t)n_seqs], 1));
    std::vector<double> pe(pk.size());
    parallel_for(n_seqs, [&](int64_t b) {
        int64_t *cp = colptr.data() + offsets[b] + b, at = pbase[(size_t)b];
        const int N = (int)(offsets[b + 1] - offsets[b]);
        for (int j = 0; j < N; j++) { cp[j] = at; at += cnt[(size_t)b][(size_t)j]; }
        cp[N] = at;
        std::copy(lk[(size_t)b].begin(), lk[(size_t)b].end(), pk.begin() + pbase[(size_t)b]);
        std::copy(le[(size_t)b].begin(), le[(size_t)b].end(), pe.begin() + pbase[(size_t)b]);
    });

    // the two tiers, each longest first; sequences of < 2 positions have no pair and are not launched
    const int smax = nu_smem_max_n(ctx->smem_optin);
    std::vector<int32_t> ord_g, ord_s;
    for (int64_t b = 0; b < n_seqs; b++) {
        const int64_t n = offsets[b + 1] - offsets[b];
        if (n >= 2) (n <= smax ? ord_s : ord_g).push_back((int32_t)b);
    }
    auto longest_first = [&](int32_t a, int32_t c) { return offsets[a + 1] - offsets[a] > offsets[c + 1] - offsets[c]; };
    std::stable_sort(ord_g.begin(), ord_g.end(), longest_first);
    std::stable_sort(ord_s.begin(), ord_s.end(), longest_first);
    std::vector<int32_t> order(ord_g);
    order.insert(order.end(), ord_s.begin(), ord_s.end());

    cudaStream_t st = ctx->stream;
    NuBatch nb{};
    int64_t *d_off, *d_colptr, *d_obase; uint8_t *d_sym; int16_t *d_pk; double *d_pe; int32_t *d_order, *d_outp, *d_outn; int *d_cnt;
    TRY(upload(ctx, B_OFF, offsets, (size_t)n_seqs + 1, &d_off));
    TRY(upload(ctx, B_SYM, symbols, (size_t)total, &d_sym));
    TRY(upload(ctx, NU_COLPTR, colptr.data(), colptr.size(), &d_colptr));
    TRY(upload(ctx, NU_PK, pk.data(), (size_t)pbase[(size_t)n_seqs], &d_pk));
    TRY(upload(ctx, NU_PE, pe.data(), (size_t)pbase[(size_t)n_seqs], &d_pe));
    TRY(upload(ctx, NU_ORDER, order.data(), order.size(), &d_order));
    TRY(upload(ctx, NU_OUTBASE, out_base.data(), (size_t)n_seqs, &d_obase));
    TRY(dalloc(ctx, NU_OUTP, (size_t)(2 * cap), &d_outp));
    TRY(dalloc(ctx, NU_OUTN, (size_t)n_seqs, &d_outn));
    TRY(dalloc(ctx, NU_CNT, 2, &d_cnt));
    CK(cudaMemsetAsync(d_outn, 0, (size_t)n_seqs * sizeof(int32_t), st));
    CK(cudaMemsetAsync(d_cnt, 0, 2 * sizeof(int), st));
    nb.off = d_off; nb.sym = d_sym; nb.colptr = d_colptr; nb.pk = d_pk; nb.pe = d_pe; nb.minloop = minloop;
    nb.out_base = d_obase; nb.out_pairs = d_outp; nb.out_n = d_outn;

    // launch geometry first: one workspace for both tiers
    const int ng = (int)ord_g.size(), nsm = (int)ord_s.size();
    NuLayout Lg{}, Ls{};
    int grid_g = 0, grid_s = 0;
    int64_t kg = 0, ks = 0, slot_d = 0, slot_s = 0;
    auto kern_g = k_nussinov<NU_GLOB_TW, false>;
    auto kern_s = k_nussinov<NU_SMEM_TW, true>;
    if (ng) {
        const int nmax = (int)(offsets[ord_g[0] + 1] - offsets[ord_g[0]]);
        Lg = nu_layout(nmax, false);
        CK(cudaFuncSetAttribute(kern_g, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Lg.total));
        int occ = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern_g, NU_GLOB_TW * 32, Lg.total));
        slot_d = nu_round8(nu_cells(nmax)); kg = nu_round8(nu_cells(nmax)); slot_s = nu_round8(nmax);
        grid_g = (int)std::min<int64_t>((int64_t)ng, (int64_t)ctx->sm_count * std::max(occ, 1));
    }
    if (nsm) {
        const int nmax = (int)(offsets[ord_s[0] + 1] - offsets[ord_s[0]]);
        Ls = nu_layout(nmax, true);
        CK(cudaFuncSetAttribute(kern_s, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Ls.total));
        int occ = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern_s, NU_SMEM_TW * 32, Ls.total));
        ks = nu_round8(nu_cells(nmax));
        grid_s = (int)std::min<int64_t>((int64_t)nsm, (int64_t)ctx->sm_count * std::max(occ, 1));
    }
    if (ng) {                                         // the global slots get what the shared tier's K leaves of the cap
        const int64_t slot_bytes = 8 * slot_d + 2 * kg + 10 * slot_s;
        grid_g = (int)std::min<int64_t>(grid_g, std::max<int64_t>(1, (NU_WORKSPACE_CAP - 2 * grid_s * ks) / slot_bytes));
    }
    // workspace: global-tier triangles | row best values | K of both tiers | row best k (each part 8-element aligned)
    const int64_t n_wd = grid_g * slot_d, n_wb = grid_g * slot_s, n_wk = grid_g * kg + grid_s * ks, n_wbk = grid_g * slot_s;
    const size_t ws_bytes = (size_t)(8 * (n_wd + n_wb) + 2 * (n_wk + n_wbk) + 16);
    if (ws_bytes > ctx->nu_ws_bytes) {
        if (ctx->nu_ws) cudaFree(ctx->nu_ws);
        ctx->nu_ws = nullptr; ctx->nu_ws_bytes = 0;
        CK(cudaMalloc(&ctx->nu_ws, ws_bytes));
        ctx->nu_ws_bytes = ws_bytes;
    }
    double *d_wd = (double *)ctx->nu_ws, *d_wb = d_wd + n_wd;
    int16_t *d_wk = (int16_t *)(d_wb + n_wb), *d_wbk = d_wk + n_wk;
    CK(cudaEventRecord(ctx->ev0, st));
    CK(cudaEventRecord(ctx->ev_start, st));          // the uploads are done: where the second stream starts
    if (ng) {
        NuBatch g = nb;
        g.n_items = ng; g.order = d_order; g.counter = d_cnt;
        g.wd = d_wd; g.wk = d_wk; g.wbest = d_wb; g.wbk = d_wbk; g.slot_d = slot_d; g.slot_k = kg; g.slot_s = slot_s;
        kern_g<<<grid_g, NU_GLOB_TW * 32, Lg.total, st>>>(g, Lg);
        CK(cudaGetLastError());
        ctx->n_launches++;
    }
    if (nsm) {
        // on the second stream, behind the uploads of the first: the two tiers share the SMs
        NuBatch s = nb;
        s.n_items = nsm; s.order = d_order + ng; s.counter = d_cnt + 1;
        s.wk = d_wk + grid_g * kg; s.slot_k = ks;
        CK(cudaStreamWaitEvent(ctx->s_k2, ctx->ev_start, 0));
        kern_s<<<grid_s, NU_SMEM_TW * 32, Ls.total, ctx->s_k2>>>(s, Ls);
        CK(cudaGetLastError());
        CK(cudaEventRecord(ctx->ev_k2done, ctx->s_k2));
        CK(cudaStreamWaitEvent(st, ctx->ev_k2done, 0));
        ctx->n_launches++;
    }
    CK(cudaEventRecord(ctx->ev1, st));
    std::vector<int32_t> outn((size_t)n_seqs);
    CK(cudaMemcpyAsync(outn.data(), d_outn, (size_t)n_seqs * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (cap > 0) CK(cudaMemcpyAsync(pairs, d_outp, (size_t)(2 * cap) * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->kernel_ms = ms;
    // sequence b's pairs were written at out_base[b]; pack them in sequence order (in place: never moves right)
    int64_t at = 0;
    for (int64_t b = 0; b < n_seqs; b++) {
        pair_offsets[b] = at;
        const int64_t m = outn[(size_t)b];
        if (m && at != out_base[(size_t)b]) memmove(pairs + 2 * at, pairs + 2 * out_base[(size_t)b], (size_t)m * 2 * sizeof(int32_t));
        at += m;
    }
    pair_offsets[n_seqs] = at;
    if (cap > at) memset(pairs + 2 * at, 0, (size_t)(cap - at) * 2 * sizeof(int32_t));     // (no stale device memory)
    return SQRN_OK;
}

extern "C" int sqrn_nussinov_batch(sqrn_ctx *ctx, int64_t n_seqs, const int64_t *offsets, const uint8_t *symbols,
                                   const int64_t *stem_offsets, const int32_t *stems, const double *scores,
                                   int32_t minloop, int64_t *pair_offsets, int32_t *pairs)
{
    return guarded(ctx, [&] { return sqrn_nussinov_batch_impl(ctx, n_seqs, offsets, symbols, stem_offsets, stems, scores, minloop, pair_offsets, pairs); });
}

// ------------------------------------------------------------- Hungarian
// The assignment and the filter of sqrn_hungarian.cuh.  Three tiers by length, each a persistent kernel whose teams
// take the tier's sequences longest first from a counter: a warp per sequence up to HU_WARP_MAX_N positions (HU_WPC
// states in a CTA's shared memory), a CTA with its state in shared memory up to hu_smem_max_n(opt-in limit), and a CTA
// with its state in a slot of a device workspace beyond that (at most one slot per SM: 1.4 MB at SQRN_MAX_LEN).  The
// warp tier runs on the second stream, concurrently with the other two.
template <int TW, bool SMEM>
__global__ void __launch_bounds__(TW == 1 ? HU_WPC * 32 : TW * 32, 1)
k_hungarian(HuBatch hb, HuLayout L)
{
    extern __shared__ __align__(16) unsigned char smem[];
    if (TW == 1) {
        unsigned char *st = smem + (threadIdx.x >> 5) * L.total;
        for (;;) {
            int item = 0;
            if ((threadIdx.x & 31) == 0) item = atomicAdd(hb.counter, 1);
            item = __shfl_sync(0xffffffffu, item, 0);
            if (item >= hb.n_items) break;
            hu_item<HuTeam<1>>(hb, hb.order[item], st, L, nullptr);
        }
        return;
    }
    const size_t base = SMEM ? L.total : 0;
    HuKey *red = (HuKey *)(smem + base);
    int *s_item = (int *)(smem + base + 16 * HU_CTA_TW);
    unsigned char *st = SMEM ? smem : hb.ws + (int64_t)blockIdx.x * hb.slot_bytes;
    for (;;) {
        if (threadIdx.x == 0) *s_item = atomicAdd(hb.counter, 1);
        __syncthreads();
        const int item = *s_item;
        __syncthreads();
        if (item >= hb.n_items) break;
        hu_item<HuTeam<TW>>(hb, hb.order[item], st, L, red);
    }
}

static int sqrn_hungarian_batch_impl(sqrn_ctx *ctx, int64_t n_seqs, const int64_t *offsets, const uint8_t *symbols,
                                     const int64_t *stem_offsets, const int32_t *stems, const double *scores,
                                     int32_t minloop, double power, int64_t *pair_offsets, int32_t *pairs)
{
    if (!ctx) return SQRN_E_BADARG;
    if (n_seqs < 0 || n_seqs >= (1LL << 31) || !offsets || !stem_offsets || !pair_offsets || minloop < 0 || offsets[0] != 0) {
        ctx->err = "hungarian: bad arguments (offsets / stem_offsets / pair_offsets must be given, offsets[0] == 0, minloop >= 0)";
        return SQRN_E_BADARG;
    }
    cudaSetDevice(ctx->device);
    ctx->n_launches = 0; ctx->n_calls = 0; ctx->kernel_ms = 0; ctx->n_cluster_launches = 0;
    std::vector<int64_t> out_base((size_t)n_seqs + 1, 0);
    for (int64_t b = 0; b < n_seqs; b++) {
        const int64_t n = offsets[b + 1] - offsets[b], ns = stem_offsets[b + 1] - stem_offsets[b];
        if (n < 0 || n > SQRN_MAX_LEN || ns < 0) {
            ctx->err = "hungarian: offsets must not decrease and a sequence may have at most SQRN_MAX_LEN positions";
            return SQRN_E_BADARG;
        }
        if (ns > 0 && (!stems || !scores)) { ctx->err = "hungarian: stems / scores missing"; return SQRN_E_BADARG; }
        if (ns > 0 && !hu_stems_ok((int)n, stems + 3 * stem_offsets[b], ns)) {
            ctx->err = "hungarian: a stem of sequence " + std::to_string(b) + " leaves [0, N), has len < 1 or a pair (v, w) with v >= w";
            return SQRN_E_BADARG;
        }
        out_base[(size_t)b + 1] = out_base[(size_t)b] + n / 2;
    }
    const int64_t total = offsets[n_seqs], cap = out_base[(size_t)n_seqs];
    if ((total > 0 && !symbols) || (cap > 0 && !pairs)) { ctx->err = "hungarian: symbols / pairs missing"; return SQRN_E_BADARG; }
    pair_offsets[0] = 0;
    if (n_seqs == 0) return SQRN_OK;

    // weights and adjacency per sequence (host threads), then one flat CSR: sequence b's row pointers at offsets[b] + b
    std::vector<std::vector<int64_t>> rows((size_t)n_seqs);
    std::vector<std::vector<int16_t>> acol((size_t)n_seqs);
    std::vector<std::vector<double>> acost((size_t)n_seqs);
    std::vector<char> bad((size_t)n_seqs, 0);
    parallel_for(n_seqs, [&](int64_t b) {
        const int64_t ns = stem_offsets[b + 1] - stem_offsets[b];
        std::vector<double> w;
        if (ns > 0 && !hu_weights(scores + stem_offsets[b], ns, power, w)) { bad[(size_t)b] = 1; return; }
        hu_seq_adjacency((int)(offsets[b + 1] - offsets[b]), ns > 0 ? stems + 3 * stem_offsets[b] : nullptr, w.data(), ns,
                         rows[(size_t)b], acol[(size_t)b], acost[(size_t)b]);
    });
    for (int64_t b = 0; b < n_seqs; b++)
        if (bad[(size_t)b]) {
            ctx->err = "hungarian: sequence " + std::to_string(b) + " has a negative or NaN score or a non-finite score ** power";
            return SQRN_E_BADARG;
        }
    std::vector<int64_t> abase((size_t)n_seqs + 1, 0);
    for (int64_t b = 0; b < n_seqs; b++) abase[(size_t)b + 1] = abase[(size_t)b] + (int64_t)acol[(size_t)b].size();
    std::vector<int64_t> rowptr((size_t)(total + n_seqs));
    std::vector<int16_t> ac((size_t)std::max<int64_t>(abase[(size_t)n_seqs], 1));
    std::vector<double> ae(ac.size());
    parallel_for(n_seqs, [&](int64_t b) {
        int64_t *rp = rowptr.data() + offsets[b] + b;
        const int N = (int)(offsets[b + 1] - offsets[b]);
        for (int p = 0; p <= N; p++) rp[p] = abase[(size_t)b] + rows[(size_t)b][(size_t)p];
        std::copy(acol[(size_t)b].begin(), acol[(size_t)b].end(), ac.begin() + abase[(size_t)b]);
        std::copy(acost[(size_t)b].begin(), acost[(size_t)b].end(), ae.begin() + abase[(size_t)b]);
    });

    // the three tiers, each longest first; a sequence without stem pairs has no pair to keep and is not launched
    const int smax = hu_smem_max_n(ctx->smem_optin);
    std::vector<int32_t> ord[3];                      // global, CTA, warp
    for (int64_t b = 0; b < n_seqs; b++) {
        const int64_t n = offsets[b + 1] - offsets[b];
        if (abase[(size_t)b + 1] > abase[(size_t)b]) ord[n > smax ? 0 : n > HU_WARP_MAX_N ? 1 : 2].push_back((int32_t)b);
    }
    auto longest_first = [&](int32_t a, int32_t c) { return offsets[a + 1] - offsets[a] > offsets[c + 1] - offsets[c]; };
    std::vector<int32_t> order;
    for (auto &o : ord) { std::stable_sort(o.begin(), o.end(), longest_first); order.insert(order.end(), o.begin(), o.end()); }

    cudaStream_t st = ctx->stream;
    int64_t *d_off, *d_rowptr, *d_obase; uint8_t *d_sym; int16_t *d_ac; double *d_ae; int32_t *d_order, *d_outp, *d_outn; int *d_cnt;
    TRY(upload(ctx, B_OFF, offsets, (size_t)n_seqs + 1, &d_off));
    TRY(upload(ctx, B_SYM, symbols, (size_t)total, &d_sym));
    TRY(upload(ctx, HU_ROWPTR, rowptr.data(), rowptr.size(), &d_rowptr));
    TRY(upload(ctx, HU_ACOL, ac.data(), (size_t)abase[(size_t)n_seqs], &d_ac));
    TRY(upload(ctx, HU_ACOST, ae.data(), (size_t)abase[(size_t)n_seqs], &d_ae));
    TRY(upload(ctx, HU_ORDER, order.data(), order.size(), &d_order));
    TRY(upload(ctx, HU_OUTBASE, out_base.data(), (size_t)n_seqs, &d_obase));
    TRY(dalloc(ctx, HU_OUTP, (size_t)(2 * cap), &d_outp));
    TRY(dalloc(ctx, HU_OUTN, (size_t)n_seqs, &d_outn));
    TRY(dalloc(ctx, HU_CNT, 3, &d_cnt));
    CK(cudaMemsetAsync(d_outn, 0, (size_t)n_seqs * sizeof(int32_t), st));
    CK(cudaMemsetAsync(d_cnt, 0, 3 * sizeof(int), st));
    HuBatch hb{};
    hb.off = d_off; hb.sym = d_sym; hb.rowptr = d_rowptr; hb.acol = d_ac; hb.acost = d_ae; hb.minloop = minloop;
    hb.out_base = d_obase; hb.out_pairs = d_outp; hb.out_n = d_outn;

    const int ng = (int)ord[0].size(), nc = (int)ord[1].size(), nw = (int)ord[2].size();
    auto nmax = [&](const std::vector<int32_t> &o) { return (int)(offsets[o[0] + 1] - offsets[o[0]]); };
    CK(cudaEventRecord(ctx->ev0, st));
    CK(cudaEventRecord(ctx->ev_start, st));          // the uploads are done: where the second stream starts
    if (nw) {                                         // warp tier, on the second stream
        auto kern = k_hungarian<1, true>;
        const HuLayout L = hu_layout(nmax(ord[2]));
        const size_t sm = hu_warp_smem(nmax(ord[2]));
        CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
        int occ = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, HU_WPC * 32, sm));
        HuBatch w = hb;
        w.n_items = nw; w.order = d_order + ng + nc; w.counter = d_cnt + 2;
        const int grid = (int)std::min<int64_t>((nw + HU_WPC - 1) / HU_WPC, (int64_t)ctx->sm_count * std::max(occ, 1));
        CK(cudaStreamWaitEvent(ctx->s_k2, ctx->ev_start, 0));
        kern<<<grid, HU_WPC * 32, sm, ctx->s_k2>>>(w, L);
        CK(cudaGetLastError());
        CK(cudaEventRecord(ctx->ev_k2done, ctx->s_k2));
        ctx->n_launches++;
    }
    if (ng) {                                         // global tier: one slot per CTA, at most one CTA per SM
        auto kern = k_hungarian<HU_CTA_TW, false>;
        const HuLayout L = hu_layout(nmax(ord[0]));
        const size_t sm = hu_cta_smem(0, false);
        const int grid = std::min(ng, ctx->sm_count);
        const size_t ws_bytes = (size_t)grid * L.total;
        if (ws_bytes > ctx->hu_ws_bytes) {
            if (ctx->hu_ws) cudaFree(ctx->hu_ws);
            ctx->hu_ws = nullptr; ctx->hu_ws_bytes = 0;
            CK(cudaMalloc(&ctx->hu_ws, ws_bytes));
            ctx->hu_ws_bytes = ws_bytes;
        }
        HuBatch g = hb;
        g.n_items = ng; g.order = d_order; g.counter = d_cnt; g.ws = (unsigned char *)ctx->hu_ws; g.slot_bytes = (int64_t)L.total;
        kern<<<grid, HU_CTA_TW * 32, sm, st>>>(g, L);
        CK(cudaGetLastError());
        ctx->n_launches++;
    }
    if (nc) {                                         // CTA tier
        auto kern = k_hungarian<HU_CTA_TW, true>;
        const HuLayout L = hu_layout(nmax(ord[1]));
        const size_t sm = hu_cta_smem(nmax(ord[1]), true);
        CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
        int occ = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, HU_CTA_TW * 32, sm));
        HuBatch c = hb;
        c.n_items = nc; c.order = d_order + ng; c.counter = d_cnt + 1;
        const int grid = (int)std::min<int64_t>((int64_t)nc, (int64_t)ctx->sm_count * std::max(occ, 1));
        kern<<<grid, HU_CTA_TW * 32, sm, st>>>(c, L);
        CK(cudaGetLastError());
        ctx->n_launches++;
    }
    if (nw) CK(cudaStreamWaitEvent(st, ctx->ev_k2done, 0));
    CK(cudaEventRecord(ctx->ev1, st));
    std::vector<int32_t> outn((size_t)n_seqs);
    CK(cudaMemcpyAsync(outn.data(), d_outn, (size_t)n_seqs * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (cap > 0) CK(cudaMemcpyAsync(pairs, d_outp, (size_t)(2 * cap) * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->kernel_ms = ms;
    // sequence b's pairs were written at out_base[b]; pack them in sequence order (in place: never moves right)
    int64_t at = 0;
    for (int64_t b = 0; b < n_seqs; b++) {
        pair_offsets[b] = at;
        const int64_t m = outn[(size_t)b];
        if (m < 0) {
            ctx->err = "hungarian: sequence " + std::to_string(b) + ": the cost matrix is infeasible (a reduced cost overflows)";
            return SQRN_E_BADARG;
        }
        if (m && at != out_base[(size_t)b]) memmove(pairs + 2 * at, pairs + 2 * out_base[(size_t)b], (size_t)m * 2 * sizeof(int32_t));
        at += m;
    }
    pair_offsets[n_seqs] = at;
    if (cap > at) memset(pairs + 2 * at, 0, (size_t)(cap - at) * 2 * sizeof(int32_t));     // (no stale device memory)
    return SQRN_OK;
}

extern "C" int sqrn_hungarian_batch(sqrn_ctx *ctx, int64_t n_seqs, const int64_t *offsets, const uint8_t *symbols,
                                    const int64_t *stem_offsets, const int32_t *stems, const double *scores,
                                    int32_t minloop, double power, int64_t *pair_offsets, int32_t *pairs)
{
    return guarded(ctx, [&] { return sqrn_hungarian_batch_impl(ctx, n_seqs, offsets, symbols, stem_offsets, stems, scores, minloop, power, pair_offsets, pairs); });
}

// ------------------------------------------------------------- Edmonds
// The matching of sqrn_edmonds.cuh.  Three tiers by length, each a persistent kernel whose teams take the tier's
// sequences longest first from a counter: a warp per sequence up to ED_WARP_MAX_N positions (ED_WPC node states in a
// CTA's shared memory), a CTA with its node state in shared memory up to ed_smem_max_n(opt-in limit), and a CTA with its
// node state in its workspace slot beyond that.  Every team also has the edge state of its sequences (allowed-edge
// stamps, the mybestedges arena) in its slot.  Slots are sized from the V and E of the launch's sequences; the whole
// workspace takes at most ED_WORKSPACE_CAP bytes but at least one slot per tier, and the context keeps it between calls.
// The adjacency is read-only, in global memory.  The warp tier runs on the second stream, concurrently with the others.
constexpr int64_t ED_WORKSPACE_CAP = (int64_t)4 << 30;

template <int TW, bool SMEM>
__global__ void __launch_bounds__(TW == 1 ? ED_WPC * 32 : TW * 32, 1)
k_edmonds(EdBatch eb, int64_t vbytes)
{
    extern __shared__ __align__(16) unsigned char smem[];
    if (TW == 1) {
        const int w = threadIdx.x >> 5;
        unsigned char *st = smem + w * vbytes;
        int32_t *est = (int32_t *)(eb.ws + ((int64_t)blockIdx.x * ED_WPC + w) * eb.slot_bytes);
        for (;;) {
            int item = 0;
            if ((threadIdx.x & 31) == 0) item = atomicAdd(eb.counter, 1);
            item = __shfl_sync(0xffffffffu, item, 0);
            if (item >= eb.n_items) break;
            ed_item<HuTeam<1>>(eb, eb.order[item], st, est, nullptr);
        }
        return;
    }
    const size_t base = SMEM ? vbytes : 0;
    HuKey *red = (HuKey *)(smem + base);
    int *s_item = (int *)(smem + base + 16 * ED_CTA_TW);
    unsigned char *slot = eb.ws + (int64_t)blockIdx.x * eb.slot_bytes;
    unsigned char *st = SMEM ? smem : slot;
    int32_t *est = (int32_t *)(SMEM ? slot : slot + vbytes);
    for (;;) {
        if (threadIdx.x == 0) *s_item = atomicAdd(eb.counter, 1);
        __syncthreads();
        const int item = *s_item;
        __syncthreads();
        if (item >= eb.n_items) break;
        ed_item<HuTeam<TW>>(eb, eb.order[item], st, est, red);
    }
}

static int sqrn_edmonds_batch_impl(sqrn_ctx *ctx, int64_t n_seqs, const int64_t *offsets, const int64_t *stem_offsets,
                                   const int32_t *stems, const double *scores, double power, int64_t *pair_offsets,
                                   int32_t *pairs)
{
    if (!ctx) return SQRN_E_BADARG;
    if (n_seqs < 0 || n_seqs >= (1LL << 31) || !offsets || !stem_offsets || !pair_offsets || offsets[0] != 0) {
        ctx->err = "edmonds: bad arguments (offsets / stem_offsets / pair_offsets must be given, offsets[0] == 0)";
        return SQRN_E_BADARG;
    }
    cudaSetDevice(ctx->device);
    ctx->n_launches = 0; ctx->n_calls = 0; ctx->kernel_ms = 0; ctx->n_cluster_launches = 0;
    std::vector<int64_t> out_base((size_t)n_seqs + 1, 0);
    for (int64_t b = 0; b < n_seqs; b++) {
        const int64_t n = offsets[b + 1] - offsets[b], ns = stem_offsets[b + 1] - stem_offsets[b];
        if (n < 0 || n > SQRN_MAX_LEN || ns < 0) {
            ctx->err = "edmonds: offsets must not decrease and a sequence may have at most SQRN_MAX_LEN positions";
            return SQRN_E_BADARG;
        }
        if (ns > 0 && (!stems || !scores)) { ctx->err = "edmonds: stems / scores missing"; return SQRN_E_BADARG; }
        if (ns > 0 && !hu_stems_ok((int)n, stems + 3 * stem_offsets[b], ns)) {
            ctx->err = "edmonds: a stem of sequence " + std::to_string(b) + " leaves [0, N), has len < 1 or a pair (v, w) with v >= w";
            return SQRN_E_BADARG;
        }
        out_base[(size_t)b + 1] = out_base[(size_t)b] + n / 2;
    }
    const int64_t cap = out_base[(size_t)n_seqs];
    if (cap > 0 && !pairs) { ctx->err = "edmonds: pairs missing"; return SQRN_E_BADARG; }
    pair_offsets[0] = 0;
    if (n_seqs == 0) return SQRN_OK;

    // the graph of each sequence (host threads), then flat arrays: nodes at vbase[b], edges at ebase[b], row pointers
    // at vbase[b] + b holding offsets into the flat adjacency
    std::vector<std::vector<int32_t>> pos((size_t)n_seqs), adj((size_t)n_seqs), ep((size_t)n_seqs);
    std::vector<std::vector<int64_t>> rows((size_t)n_seqs);
    std::vector<std::vector<double>> wt((size_t)n_seqs);
    std::vector<double> maxw((size_t)n_seqs, 0.0);
    std::vector<char> bad((size_t)n_seqs, 0);
    parallel_for(n_seqs, [&](int64_t b) {
        const int64_t ns = stem_offsets[b + 1] - stem_offsets[b];
        std::vector<double> w;
        if (ns > 0 && !ed_weights(scores + stem_offsets[b], ns, power, w)) { bad[(size_t)b] = 1; return; }
        maxw[(size_t)b] = ed_seq_graph((int)(offsets[b + 1] - offsets[b]), ns > 0 ? stems + 3 * stem_offsets[b] : nullptr,
                                       w.data(), ns, pos[(size_t)b], rows[(size_t)b], adj[(size_t)b], ep[(size_t)b], wt[(size_t)b]);
    });
    for (int64_t b = 0; b < n_seqs; b++)
        if (bad[(size_t)b]) {
            ctx->err = "edmonds: sequence " + std::to_string(b) + " has a negative or NaN score or a non-finite or huge score ** power";
            return SQRN_E_BADARG;
        }
    std::vector<int64_t> vbase((size_t)n_seqs + 1, 0), ebase((size_t)n_seqs + 1, 0);
    for (int64_t b = 0; b < n_seqs; b++) {
        vbase[(size_t)b + 1] = vbase[(size_t)b] + (int64_t)pos[(size_t)b].size();
        ebase[(size_t)b + 1] = ebase[(size_t)b] + (int64_t)wt[(size_t)b].size();
    }
    const int64_t nv = vbase[(size_t)n_seqs], ne = ebase[(size_t)n_seqs];
    std::vector<int64_t> rowptr((size_t)(nv + n_seqs));
    std::vector<int32_t> fpos((size_t)std::max<int64_t>(nv, 1)), fadj((size_t)std::max<int64_t>(2 * ne, 1)), fep(fadj.size());
    std::vector<double> fwt((size_t)std::max<int64_t>(ne, 1));
    parallel_for(n_seqs, [&](int64_t b) {
        const size_t B = (size_t)b;
        int64_t *rp = rowptr.data() + vbase[B] + b;
        for (size_t x = 0; x < rows[B].size(); x++) rp[x] = 2 * ebase[B] + rows[B][x];
        std::copy(pos[B].begin(), pos[B].end(), fpos.begin() + vbase[B]);
        std::copy(adj[B].begin(), adj[B].end(), fadj.begin() + 2 * ebase[B]);
        std::copy(ep[B].begin(), ep[B].end(), fep.begin() + 2 * ebase[B]);
        std::copy(wt[B].begin(), wt[B].end(), fwt.begin() + ebase[B]);
    });

    // the three tiers, each longest first; a sequence without an edge has no pair and is not launched
    const int smax = ed_smem_max_n(ctx->smem_optin);
    std::vector<int32_t> ord[3];                      // global, CTA, warp
    for (int64_t b = 0; b < n_seqs; b++) {
        const int64_t n = offsets[b + 1] - offsets[b];
        if (ebase[(size_t)b + 1] > ebase[(size_t)b]) ord[n > smax ? 0 : n > ED_WARP_MAX_N ? 1 : 2].push_back((int32_t)b);
    }
    auto longest_first = [&](int32_t a, int32_t c) { return offsets[a + 1] - offsets[a] > offsets[c + 1] - offsets[c]; };
    std::vector<int32_t> order;
    for (auto &o : ord) { std::stable_sort(o.begin(), o.end(), longest_first); order.insert(order.end(), o.begin(), o.end()); }

    cudaStream_t st = ctx->stream;
    int64_t *d_vb, *d_eb, *d_rowptr, *d_obase; int32_t *d_pos, *d_adj, *d_ep; double *d_wt, *d_maxw;
    int32_t *d_order, *d_outp, *d_outn; int *d_cnt;
    TRY(upload(ctx, ED_VBASE, vbase.data(), vbase.size(), &d_vb));
    TRY(upload(ctx, ED_EBASE, ebase.data(), ebase.size(), &d_eb));
    TRY(upload(ctx, ED_ROWPTR, rowptr.data(), rowptr.size(), &d_rowptr));
    TRY(upload(ctx, ED_POS, fpos.data(), (size_t)nv, &d_pos));
    TRY(upload(ctx, ED_ADJ, fadj.data(), (size_t)(2 * ne), &d_adj));
    TRY(upload(ctx, ED_EP, fep.data(), (size_t)(2 * ne), &d_ep));
    TRY(upload(ctx, ED_WT, fwt.data(), (size_t)ne, &d_wt));
    TRY(upload(ctx, ED_MAXW, maxw.data(), maxw.size(), &d_maxw));
    TRY(upload(ctx, ED_ORDER, order.data(), order.size(), &d_order));
    TRY(upload(ctx, ED_OUTBASE, out_base.data(), (size_t)n_seqs, &d_obase));
    TRY(dalloc(ctx, ED_OUTP, (size_t)(2 * cap), &d_outp));
    TRY(dalloc(ctx, ED_OUTN, (size_t)n_seqs, &d_outn));
    TRY(dalloc(ctx, ED_CNT, 3, &d_cnt));
    CK(cudaMemsetAsync(d_outn, 0, (size_t)n_seqs * sizeof(int32_t), st));
    CK(cudaMemsetAsync(d_cnt, 0, 3 * sizeof(int), st));
    EdBatch eb{};
    eb.vbase = d_vb; eb.ebase = d_eb; eb.rowptr = d_rowptr; eb.pos = d_pos; eb.adj = d_adj; eb.ep = d_ep;
    eb.wt = d_wt; eb.maxw = d_maxw; eb.out_base = d_obase; eb.out_pairs = d_outp; eb.out_n = d_outn;

    // launch geometry per tier: the node-state bytes a team needs (the most nodes of the tier), its slot (node state
    // for the global tier, then the edge state of the tier's largest graph), the number of teams
    struct Tier { int n = 0, grid = 0, teams_per_cta = 1; int64_t vbytes = 0, slot = 0; size_t smem = 0; };
    Tier T3[3];
    for (int t = 0; t < 3; t++) {
        Tier &ti = T3[t];
        ti.n = (int)ord[t].size();
        if (!ti.n) continue;
        int vmax = 0; int64_t ewords = 0;
        for (const int32_t b : ord[t]) {
            const int v = (int)(vbase[(size_t)b + 1] - vbase[(size_t)b]);
            vmax = std::max(vmax, v);
            ewords = std::max(ewords, ed_edge_words(v, ebase[(size_t)b + 1] - ebase[(size_t)b]));
        }
        ti.vbytes = (int64_t)ed_layout(vmax).total;
        ti.slot = (t == 0 ? ti.vbytes : 0) + 4 * ewords;
        int occ = 0;
        if (t == 2) {
            ti.teams_per_cta = ED_WPC;
            ti.smem = ed_warp_smem(vmax);
            CK(cudaFuncSetAttribute(k_edmonds<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ti.smem));
            CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_edmonds<1, true>, ED_WPC * 32, ti.smem));
            ti.grid = (int)std::min<int64_t>((ti.n + ED_WPC - 1) / ED_WPC, (int64_t)ctx->sm_count * std::max(occ, 1));
        } else if (t == 1) {
            ti.smem = ed_cta_smem(vmax, true);
            CK(cudaFuncSetAttribute(k_edmonds<ED_CTA_TW, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ti.smem));
            CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_edmonds<ED_CTA_TW, true>, ED_CTA_TW * 32, ti.smem));
            ti.grid = (int)std::min<int64_t>((int64_t)ti.n, (int64_t)ctx->sm_count * std::max(occ, 1));
        } else {
            ti.smem = ed_cta_smem(0, false);
            ti.grid = std::min(ti.n, ctx->sm_count);
        }
    }
    // the cap: each tier gets a third of it, and at least one CTA
    int64_t ws_bytes = 0, at[3];
    for (int t = 0; t < 3; t++) {
        Tier &ti = T3[t];
        at[t] = ws_bytes;
        if (!ti.n) continue;
        const int64_t per_cta = ti.slot * ti.teams_per_cta;
        ti.grid = (int)std::min<int64_t>(ti.grid, std::max<int64_t>(1, ED_WORKSPACE_CAP / 3 / per_cta));
        ws_bytes += ((int64_t)ti.grid * per_cta + 255) & ~(int64_t)255;
    }
    if ((size_t)ws_bytes > ctx->ed_ws_bytes) {
        if (ctx->ed_ws) cudaFree(ctx->ed_ws);
        ctx->ed_ws = nullptr; ctx->ed_ws_bytes = 0;
        CK(cudaMalloc(&ctx->ed_ws, (size_t)ws_bytes));
        ctx->ed_ws_bytes = (size_t)ws_bytes;
    }
    unsigned char *ws = (unsigned char *)ctx->ed_ws;
    const int ng = T3[0].n, nc = T3[1].n, nw = T3[2].n;
    CK(cudaEventRecord(ctx->ev0, st));
    CK(cudaEventRecord(ctx->ev_start, st));          // the uploads are done: where the second stream starts
    if (nw) {                                         // warp tier, on the second stream
        EdBatch w = eb;
        w.n_items = nw; w.order = d_order + ng + nc; w.counter = d_cnt + 2; w.ws = ws + at[2]; w.slot_bytes = T3[2].slot;
        CK(cudaStreamWaitEvent(ctx->s_k2, ctx->ev_start, 0));
        k_edmonds<1, true><<<T3[2].grid, ED_WPC * 32, T3[2].smem, ctx->s_k2>>>(w, T3[2].vbytes);
        CK(cudaGetLastError());
        CK(cudaEventRecord(ctx->ev_k2done, ctx->s_k2));
        ctx->n_launches++;
    }
    if (ng) {                                         // global tier
        EdBatch g = eb;
        g.n_items = ng; g.order = d_order; g.counter = d_cnt; g.ws = ws + at[0]; g.slot_bytes = T3[0].slot;
        k_edmonds<ED_CTA_TW, false><<<T3[0].grid, ED_CTA_TW * 32, T3[0].smem, st>>>(g, T3[0].vbytes);
        CK(cudaGetLastError());
        ctx->n_launches++;
    }
    if (nc) {                                         // CTA tier
        EdBatch c = eb;
        c.n_items = nc; c.order = d_order + ng; c.counter = d_cnt + 1; c.ws = ws + at[1]; c.slot_bytes = T3[1].slot;
        k_edmonds<ED_CTA_TW, true><<<T3[1].grid, ED_CTA_TW * 32, T3[1].smem, st>>>(c, T3[1].vbytes);
        CK(cudaGetLastError());
        ctx->n_launches++;
    }
    if (nw) CK(cudaStreamWaitEvent(st, ctx->ev_k2done, 0));
    CK(cudaEventRecord(ctx->ev1, st));
    std::vector<int32_t> outn((size_t)n_seqs);
    CK(cudaMemcpyAsync(outn.data(), d_outn, (size_t)n_seqs * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (cap > 0) CK(cudaMemcpyAsync(pairs, d_outp, (size_t)(2 * cap) * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->kernel_ms = ms;
    for (int64_t b = 0; b < n_seqs; b++)
        if (outn[(size_t)b] < 0) {
            ctx->err = "edmonds: sequence " + std::to_string(b) + ": internal capacity exceeded";
            return SQRN_E_UNSUPPORTED;
        }
    // sequence b's pairs were written at out_base[b] in node order: sort them by v, then pack them in sequence order
    // (in place: never moves right)
    parallel_for(n_seqs, [&](int64_t b) {
        int32_t *p = pairs + 2 * out_base[(size_t)b];
        std::vector<std::pair<int32_t, int32_t>> pr((size_t)outn[(size_t)b]);
        for (size_t k = 0; k < pr.size(); k++) pr[k] = {p[2 * k], p[2 * k + 1]};
        std::sort(pr.begin(), pr.end());
        for (size_t k = 0; k < pr.size(); k++) { p[2 * k] = pr[k].first; p[2 * k + 1] = pr[k].second; }
    });
    int64_t atp = 0;
    for (int64_t b = 0; b < n_seqs; b++) {
        pair_offsets[b] = atp;
        const int64_t m = outn[(size_t)b];
        if (m && atp != out_base[(size_t)b]) memmove(pairs + 2 * atp, pairs + 2 * out_base[(size_t)b], (size_t)m * 2 * sizeof(int32_t));
        atp += m;
    }
    pair_offsets[n_seqs] = atp;
    if (cap > atp) memset(pairs + 2 * atp, 0, (size_t)(cap - atp) * 2 * sizeof(int32_t));     // (no stale device memory)
    return SQRN_OK;
}

extern "C" int sqrn_edmonds_batch(sqrn_ctx *ctx, int64_t n_seqs, const int64_t *offsets, const int64_t *stem_offsets,
                                  const int32_t *stems, const double *scores, double power, int64_t *pair_offsets,
                                  int32_t *pairs)
{
    return guarded(ctx, [&] { return sqrn_edmonds_batch_impl(ctx, n_seqs, offsets, stem_offsets, stems, scores, power, pair_offsets, pairs); });
}
