// pcb200 -- C ABI (include/pcb200.h) over the sm_100a kernels.  No CPU path: a context can only be
// created on a CUDA device (the PCB_EMU build of this same file is test infrastructure, see tests/emu).
#include "pcb_block.cuh"
#include "../../include/pcb200.h"

#include <cstdarg>
#include <vector>
#ifndef PCB_EMU
#include <dlfcn.h>
#endif

// ---- error string ---------------------------------------------------------------------------------------
static thread_local char g_err[1024] = "";
void pcb_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}

// ---- plan registry --------------------------------------------------------------------------------------
#define PCB_PLAN(N, R1, R2) extern const PcbOpLaunch pcb_plan_##N;
#include <pcb_plans.inc>
#undef PCB_PLAN
static const PcbOpLaunch* const g_plans[] = {
#define PCB_PLAN(N, R1, R2) &pcb_plan_##N,
#include <pcb_plans.inc>
#undef PCB_PLAN
};
static const int g_nplans = (int)(sizeof g_plans / sizeof g_plans[0]);
const PcbOpLaunch* pcb_find_plan(int N) {
    for (int i = 0; i < g_nplans; ++i)
        if (g_plans[i]->N == N) return g_plans[i];
    return nullptr;
}

// ---- objects ----------------------------------------------------------------------------------------------
// ---- collectives of the large-grid mode: NCCL resolved at run time (dlopen), host callbacks in the emulation build ----
struct PcbNcclId { char internal[128]; };      // ncclUniqueId
struct PcbNccl {
    void* lib = nullptr;
    int (*GetUniqueId)(PcbNcclId*) = nullptr;
    int (*CommInitRank)(void**, int, PcbNcclId, int) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
    int (*Send)(const void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    int (*Recv)(void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
enum { PCB_NCCL_FLOAT64 = 8, PCB_NCCL_UINT8 = 1, PCB_NCCL_SUM = 0 };
typedef int (*pcb_allreduce_cb)(double* buf, long long count);
typedef int (*pcb_p2p_cb)(int nops, const int* is_send, const int* peer, void* const* ptr, const long long* bytes);
struct PcbComm {
    int rank = 0, world = 1;
    void* nccl = nullptr;              // ncclComm_t
    pcb_allreduce_cb allreduce_cb = nullptr;
    pcb_p2p_cb p2p_cb = nullptr;
};
static PcbNccl g_nccl;

#define PCB_ORDER_EVENTS 16
struct pcb_ctx {
    int device = 0;
    int N = 0;
    int z0 = 0, z1 = 0;             // i2 planes owned by this context (0..N on a full context)
    long long nloc = 0;             // cells owned = (z1 - z0) N^2
    PcbComm* comm = nullptr;        // collectives (slab contexts of the large-grid mode)
    long long nn = 0, R = 0;        // N^3; rows of a column on this context = 3 * nloc
    cudaStream_t stream = nullptr;
    const PcbOpLaunch* plan = nullptr;
    cplx* tw = nullptr;             // [R1][R2] forward twiddles exp(-2 pi i k1 n2 / N)
    double pending_norms[32];       // pcb_update_resid_start / _wait: norms of a fused update whose result has not been fetched yet
    int pending_state = 0;          // 0 none, 1 on their way into hstage (stream not yet synchronised), 2 ready in pending_norms
    int pending_m = 0;
    PcbDist* ddist = nullptr;       // large-grid mode over peer memory: device copy of the slab pointer table of the current apply
    int* ctab = nullptr;            // plane mode: slot -> index and index -> slot tables of the plan (k_coord_tables)
    double* partial = nullptr;      // reduction partials (device)
    size_t partial_bytes = 0;
    void* hstage = nullptr;         // pinned host staging for small results / E matrices
    size_t hstage_bytes = 0;
    void* dsmall = nullptr;         // small device buffer (E matrix, reduced results)
    size_t dsmall_bytes = 0;
    cplx* scratch = nullptr;        // work columns (cross-DoF dielectric, block transposes)
    size_t scratch_bytes = 0;
    cplx* bv_buf = nullptr;         // pcb_band_velocity: the tau tables + E^ of its columns; released by pcb_ctx_trim
    size_t bv_bytes = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaEvent_t order_ev[PCB_ORDER_EVENTS] = {};   // pcb_ctx_record / pcb_ctx_wait: stream ordering between contexts, created on first use
    long long launches = 0;
    char blk_name[32] = "";         // the last tiled block kernel (Gram / update) planned on this context: pcb_block_launch_info
    long long blk_grid = 0, blk_tiles = 0;
    int sms = 148;
    int use_plane = 1;              // PCB200_PLANE=0 forces the five-pass operator (A/B measurements)
    int use_plane_coupled = 1;      // PCB200_PLANE_COUPLED=0: coupled 3x3 dielectric on the five-pass path
    int use_plane_cross = 1;        // cross-DoF dielectric: 1 = plane halves with the stencil fused into the inverse half as a gather on load
                                    // (4 kernels, 9 column transfers, default: 2.73 ms per 16 columns at N = 120), 2 = plane halves around the
                                    // stencil kernel on the slot layout (5 kernels, 2.97 ms), 0 = split five-pass path (7 kernels, 3.54 ms)
    int zsplit = 0;                 // plane mode in its z-split form (half planes): the only plane mode of N = 128, 144, 160; PCB200_PLANE_SPLIT=1 /
                                    // pcb_ctx_option "plane_split" select it for the smaller sizes that have it (A/B measurements, tests)
    int use_mid_five = -1;          // five-sweep plane pass k_mid2: -1 where it is the faster form (R2 >= 15), 0 never, 1 wherever it exists
    // pcb_apply_host pipeline: copy streams, two slots of (row-major staging in/out, planar columns in/out), events
    cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
    cplx* hp_buf = nullptr;         // one allocation: 2 slots x 4 regions of R x hp_cols elements
    int hp_cols = 0;                // columns per pipeline chunk the staging was sized for (<= PCB_HOST_CH)
    cudaEvent_t hp_ev[2][4] = {{nullptr, nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr, nullptr}};
};
struct pcb_diel {
    pcb_ctx* ctx;
    int kind;
    unsigned char* mask;    // [nn] (padded to 4)
    unsigned* mbits;        // plane mode: per-item dielectric bit words (k_mask_bits); null when the size has no plane pass
    unsigned* mbits2;       // five-sweep plane pass: bit words in its item order (k_mask_bits2); else null
    unsigned char* maskp2;  // five-sweep plane pass, coupled dielectric: byte mask in its slot order (k_mask_plane2); else null
    unsigned char* maskp;   // plane mode, coupled dielectric: byte mask in plane-slot order (k_mask_plane); else null
    unsigned char* maskp_fe; // the same mask for pcb_field_energy where maskp does not exist: built by its first call in the plane layout
    int zsplit;             // the plane-mode form (ctx->zsplit) the slot-ordered masks were built for
    unsigned char* matp;    // materials, plane mode: the index bytes in the item order of the plane pass (k_mat_bytes); else null
    double* inv_eps;        // materials: [n_mat] 1 / eps on the device (mask then holds the [3 nn] index bytes); else null
    int n_mat;              // materials: entries of inv_eps; else 0
    double ediag[3];
    cplx eoff[3];
    PcbStencil st;
};
struct pcb_op {
    pcb_ctx* ctx;
    cplx* T;                // [3][3][N] device
    PcbOp d;                // kernel-side description
    pcb_diel* diel;
};

#define PCB_CHECK_ARG(cond, msg)               \
    do {                                       \
        if (!(cond)) {                         \
            pcb_set_error("%s: %s", __func__, msg); \
            return -2;                         \
        }                                      \
    } while (0)

static int ensure(pcb_ctx*, void** p, size_t* have, size_t want, bool host) {
    if (*have >= want) return 0;
    if (*p) {
        if (host) PCB_CUDA_OK(cudaFreeHost(*p)); else PCB_CUDA_OK(cudaFree(*p));
        *p = nullptr; *have = 0;
    }
    if (host) PCB_CUDA_OK(cudaMallocHost(p, want)); else PCB_CUDA_OK(cudaMalloc(p, want));
    *have = want;
    return 0;
}
static int ensure_partial(pcb_ctx* c, size_t bytes) { return ensure(c, (void**)&c->partial, &c->partial_bytes, bytes, false); }
static int ensure_hstage(pcb_ctx* c, size_t bytes) { return ensure(c, &c->hstage, &c->hstage_bytes, bytes, true); }
static int ensure_dsmall(pcb_ctx* c, size_t bytes) { return ensure(c, &c->dsmall, &c->dsmall_bytes, bytes, false); }
static int ensure_scratch(pcb_ctx* c, size_t bytes) { return ensure(c, (void**)&c->scratch, &c->scratch_bytes, bytes, false); }

#define PCB_HOST_CH 8      // columns per pipeline chunk: 8 x 16 B = 128-byte rows, the narrowest 2-D copy that still runs at PCIe speed

static void note_block(pcb_ctx* c, const char* name, long long grid, long long tiles) {
    snprintf(c->blk_name, sizeof c->blk_name, "%s", name);
    c->blk_grid = grid; c->blk_tiles = tiles;
}

static int grid_for(pcb_ctx* c, long long items, int per_block, int waves) {
    long long b = (items + per_block - 1) / per_block;
    long long cap = (long long)c->sms * waves;
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (int)b;
}

// Sum `count` doubles over all ranks, in place on the device, ordered on the context's stream.  No-op without a communicator.
static int comm_allreduce(pcb_ctx* c, double* dbuf, long long count) {
    PcbComm* cm = c->comm;
    if (!cm || cm->world <= 1) return 0;
#ifdef PCB_EMU
    if (!cm->allreduce_cb) { pcb_set_error("host-emu communicator has no allreduce callback"); return -4; }
    if (cm->allreduce_cb(dbuf, count) != 0) { pcb_set_error("allreduce callback failed"); return -4; }
    return 0;
#else
    const int rc = g_nccl.AllReduce(dbuf, dbuf, (size_t)count, PCB_NCCL_FLOAT64, PCB_NCCL_SUM, cm->nccl, c->stream);
    if (rc != 0) { pcb_set_error("ncclAllReduce failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?"); return -4; }
    return 0;
#endif
}

extern "C" {

const char* pcb_last_error(void) { return g_err; }
const char* pcb_backend(void) {
#ifdef PCB_EMU
    return "host-emu";
#else
    return "cuda-sm_100a";
#endif
}
int pcb_device_count(int* n) {
    PCB_CHECK_ARG(n, "null");
    PCB_CUDA_OK(cudaGetDeviceCount(n));
    return 0;
}
int pcb_supported_sizes(int* sizes, int cap) {
    for (int i = 0; i < g_nplans && i < cap; ++i) sizes[i] = g_plans[i]->N;
    return g_nplans;
}

static int ctx_create(int device, int N, int z0, int z1, pcb_ctx** out);
void pcb_ctx_destroy(pcb_ctx* c);
int pcb_ctx_create(int device, int N, pcb_ctx** out) { return ctx_create(device, N, 0, N, out); }
int pcb_ctx_create_slab(int device, int N, int z0, int z1, pcb_ctx** out) {
    if (z0 < 0 || z1 > N || z0 >= z1) { pcb_set_error("pcb_ctx_create_slab: need 0 <= z0 < z1 <= N"); return -2; }
    return ctx_create(device, N, z0, z1, out);
}
}  // extern "C"
// slot <-> index tables of the plane layout in the context's plane-mode form
static int ctx_coord_tables(pcb_ctx* c) {
    PcbOp tmp; memset(&tmp, 0, sizeof tmp);
    tmp.N = c->N; tmp.ctab = c->ctab; tmp.zsplit = c->zsplit;
    PcbCols none; memset(&none, 0, sizeof none);
    if (c->plan->pass(tmp, none, 1, PCB_PASS_COORDTAB, c->tw, c->stream, c->sms)) return -1;
    PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
    return 0;
}
static int ctx_create(int device, int N, int z0, int z1, pcb_ctx** out) {
    PCB_CHECK_ARG(out, "null");
    const PcbOpLaunch* plan = pcb_find_plan(N);
    if (!plan) { pcb_set_error("pcb_ctx_create: no FFT plan for N = %d (see pcb_supported_sizes)", N); return -2; }
    int ndev = 0;
    PCB_CUDA_OK(cudaGetDeviceCount(&ndev));
    if (ndev <= 0 || device < 0 || device >= ndev) { pcb_set_error("pcb_ctx_create: CUDA device %d not available (%d devices)", device, ndev); return -3; }
    PCB_CUDA_OK(cudaSetDevice(device));
    pcb_ctx* c = new pcb_ctx;
    c->device = device; c->N = N; c->nn = (long long)N * N * N; c->plan = plan;
    c->z0 = z0; c->z1 = z1; c->nloc = (long long)(z1 - z0) * N * N; c->R = 3 * c->nloc;
    { const char* e = getenv("PCB200_PLANE"); c->use_plane = (plan->plane_mode && !(e && e[0] == '0')) ? 1 : 0; }
    { const char* e = getenv("PCB200_PLANE_COUPLED"); c->use_plane_coupled = !(e && e[0] == '0'); }
    { const char* e = getenv("PCB200_PLANE_CROSS"); c->use_plane_cross = e ? (e[0] == '0' ? 0 : (e[0] == '2' ? 2 : 1)) : 1; }
    { const char* e = getenv("PCB200_MID_FIVE"); c->use_mid_five = e ? (e[0] == '0' ? 0 : 1) : -1; }
    { const char* e = getenv("PCB200_PLANE_SPLIT"); c->zsplit = (plan->plane_split == 2 || (plan->plane_split == 1 && e && e[0] == '1')) ? 1 : 0; }
    // cross-DoF M at N >= 160: the stencil as its own kernel between the plane halves (5 kernels) -- gathered on load in the inverse half it
    // takes 4.06 ms of an 8.84 ms apply at N = 160 (bcc_dg, 16 columns), as a kernel 1.46 ms of 7.79 ms; below that the fused form wins or ties
    if (!getenv("PCB200_PLANE_CROSS") && c->zsplit && N >= 160) c->use_plane_cross = 2;
#ifndef PCB_EMU
    cudaDeviceProp prop;
    PCB_CUDA_OK_OR(cudaGetDeviceProperties(&prop, device), delete c);
    c->sms = prop.multiProcessorCount;
    // the binary holds sm_100a code only (arch-specific, not forward compatible): refuse every other part cleanly
    if (prop.major != 10 || prop.minor != 0) { pcb_set_error("pcb_ctx_create: device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor); delete c; return -3; }
#else
    c->sms = 2;
#endif
    PCB_CUDA_OK_OR(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking), delete c);
    PCB_CUDA_OK_OR(cudaEventCreate(&c->ev0), pcb_ctx_destroy(c));
    PCB_CUDA_OK_OR(cudaEventCreate(&c->ev1), pcb_ctx_destroy(c));
    // [0, N): twiddles of the plan; z-split plane mode: [N, N + N/2) twiddles of the plan of N/2, [N + N/2, 2N) the split twiddles w_N^n
    std::vector<cplx> tw((size_t)2 * N, cmake(0.0, 0.0));
    for (int k1 = 0; k1 < plan->r1; ++k1)
        for (int n2 = 0; n2 < plan->r2; ++n2) {
            const double ang = -2.0 * M_PI * (double)((long long)k1 * n2 % N) / (double)N;
            tw[(size_t)k1 * plan->r2 + n2] = cmake(cos(ang), sin(ang));
        }
    if (plan->plane_split) {
        const int nz = N / 2;
        for (int k1 = 0; k1 < plan->zr1; ++k1)
            for (int n2 = 0; n2 < plan->zr2; ++n2) {
                const double ang = -2.0 * M_PI * (double)((long long)k1 * n2 % nz) / (double)nz;
                tw[(size_t)N + (size_t)k1 * plan->zr2 + n2] = cmake(cos(ang), sin(ang));
            }
        for (int n = 0; n < nz; ++n) {
            const double ang = -2.0 * M_PI * (double)n / (double)N;
            tw[(size_t)N + nz + n] = cmake(cos(ang), sin(ang));
        }
    }
    PCB_CUDA_OK_OR(cudaMalloc(&c->tw, sizeof(cplx) * 2 * N), pcb_ctx_destroy(c));
    PCB_CUDA_OK_OR(cudaMemcpy(c->tw, tw.data(), sizeof(cplx) * 2 * N, cudaMemcpyHostToDevice), pcb_ctx_destroy(c));
    if (plan->plane_mode) {
        PCB_CUDA_OK_OR(cudaMalloc(&c->ctab, sizeof(int) * 4 * N), pcb_ctx_destroy(c));
        if (ctx_coord_tables(c)) { pcb_ctx_destroy(c); return -1; }
    }
    *out = c;
    return 0;
}
extern "C" {
void pcb_ctx_destroy(pcb_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->tw) cudaFree(c->tw);
    if (c->ctab) cudaFree(c->ctab);
    if (c->ddist) cudaFree(c->ddist);
    if (c->partial) cudaFree(c->partial);
    if (c->dsmall) cudaFree(c->dsmall);
    if (c->scratch) cudaFree(c->scratch);
    if (c->bv_buf) cudaFree(c->bv_buf);
    if (c->hstage) cudaFreeHost(c->hstage);
    if (c->hp_buf) cudaFree(c->hp_buf);
    if (c->s_h2d) cudaStreamDestroy(c->s_h2d);
    if (c->s_d2h) cudaStreamDestroy(c->s_d2h);
    for (int a = 0; a < 2; ++a) for (int b = 0; b < 4; ++b) if (c->hp_ev[a][b]) cudaEventDestroy(c->hp_ev[a][b]);
    for (int i = 0; i < PCB_ORDER_EVENTS; ++i) if (c->order_ev[i]) cudaEventDestroy(c->order_ev[i]);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}
long long pcb_ctx_trim(pcb_ctx* c) {
    if (!c || !c->bv_buf) return 0;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    cudaFree(c->bv_buf);
    const long long freed = (long long)c->bv_bytes;
    c->bv_buf = nullptr; c->bv_bytes = 0;
    return freed;
}
int pcb_sync(pcb_ctx* c) { PCB_CUDA_OK(cudaStreamSynchronize(c->stream)); PCB_CUDA_OK(cudaGetLastError()); return 0; }
int pcb_launch_count(pcb_ctx* c, long long* n) { *n = c->launches; return 0; }
/* Pass-structure switches of a context (defaults come from the PCB200_* environment variables at pcb_ctx_create; operators
 * created or updated afterwards see the new value): "plane", "plane_coupled", "plane_cross" (0 / 1), "mid_five" (-1 auto, 0, 1). */
int pcb_ctx_option(pcb_ctx* c, const char* name, int value) {
    PCB_CHECK_ARG(c && name, "null");
    if (!strcmp(name, "plane")) c->use_plane = (value && c->plan->plane_mode) ? 1 : 0;
    else if (!strcmp(name, "plane_coupled")) c->use_plane_coupled = value ? 1 : 0;
    else if (!strcmp(name, "plane_cross")) c->use_plane_cross = (value == 2) ? 2 : (value ? 1 : 0);
    else if (!strcmp(name, "mid_five")) c->use_mid_five = value < 0 ? -1 : (value ? 1 : 0);
    else if (!strcmp(name, "plane_split")) {
        // the form of the plane mode (0 whole planes, 1 z-split half planes) where the size has both; dielectrics carry masks in the slot
        // order of the form they were created under and must be re-created after a change (pcb_op_create / _update check)
        const int want = (c->plan->plane_split == 2 || (c->plan->plane_split == 1 && value)) ? 1 : 0;
        if (want != c->zsplit) {
            PCB_CUDA_OK(cudaSetDevice(c->device));
            PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
            c->zsplit = want;
            if (c->ctab && ctx_coord_tables(c)) return -1;
        }
    }
    else { pcb_set_error("pcb_ctx_option: unknown option %s", name); return -2; }
    return 0;
}
/* Stream ordering between two contexts of one process (large-grid mode: the slab context's exchange and the full context's
 * operator run on their own streams): pcb_ctx_record marks "everything enqueued on ctx so far" in slot idx; pcb_ctx_wait makes
 * all LATER work of `waiter` start only after that mark.  No host synchronisation. */
int pcb_ctx_record(pcb_ctx* c, int idx) {
    PCB_CHECK_ARG(c && idx >= 0 && idx < PCB_ORDER_EVENTS, "bad arguments");
    PCB_CUDA_OK(cudaSetDevice(c->device));
    if (!c->order_ev[idx]) PCB_CUDA_OK(cudaEventCreateWithFlags(&c->order_ev[idx], cudaEventDisableTiming));
    PCB_CUDA_OK(cudaEventRecord(c->order_ev[idx], c->stream));
    return 0;
}
int pcb_ctx_wait(pcb_ctx* waiter, pcb_ctx* owner, int idx) {
    PCB_CHECK_ARG(waiter && owner && idx >= 0 && idx < PCB_ORDER_EVENTS && owner->order_ev[idx], "bad arguments / slot never recorded");
    PCB_CUDA_OK(cudaSetDevice(waiter->device));
    PCB_CUDA_OK(cudaStreamWaitEvent(waiter->stream, owner->order_ev[idx], 0));
    return 0;
}
int pcb_mem_info(pcb_ctx* c, size_t* f, size_t* t) { PCB_CUDA_OK(cudaSetDevice(c->device)); PCB_CUDA_OK(cudaMemGetInfo(f, t)); return 0; }
int pcb_timer_start(pcb_ctx* c) { PCB_CUDA_OK(cudaEventRecord(c->ev0, c->stream)); return 0; }
int pcb_timer_stop(pcb_ctx* c, float* ms) {
    PCB_CUDA_OK(cudaEventRecord(c->ev1, c->stream));
    PCB_CUDA_OK(cudaEventSynchronize(c->ev1));
    PCB_CUDA_OK(cudaEventElapsedTime(ms, c->ev0, c->ev1));
    return 0;
}

// ---- memory -------------------------------------------------------------------------------------------------
int pcb_malloc(pcb_ctx* c, size_t bytes, void** dptr) {
    PCB_CUDA_OK(cudaSetDevice(c->device));
    PCB_CUDA_OK(cudaMalloc(dptr, bytes));
    return 0;
}
int pcb_free(pcb_ctx* c, void* dptr) {
    PCB_CUDA_OK(cudaSetDevice(c->device));
    PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
    PCB_CUDA_OK(cudaFree(dptr));
    return 0;
}
int pcb_host_alloc(size_t bytes, void** hptr) { PCB_CUDA_OK(cudaMallocHost(hptr, bytes)); return 0; }
int pcb_host_free(void* hptr) { PCB_CUDA_OK(cudaFreeHost(hptr)); return 0; }
int pcb_memcpy_h2d(pcb_ctx* c, void* dst, const void* src, size_t bytes) {
    PCB_CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream));
    PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
    return 0;
}
int pcb_memcpy_d2h(pcb_ctx* c, void* dst, const void* src, size_t bytes) {
    PCB_CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
    PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
    return 0;
}
int pcb_memcpy_d2d(pcb_ctx* c, void* dst, const void* src, size_t bytes) {
    PCB_CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, c->stream));
    return 0;
}
int pcb_memset_zero(pcb_ctx* c, void* dst, size_t bytes) { PCB_CUDA_OK(cudaMemsetAsync(dst, 0, bytes, c->stream)); return 0; }

static int transpose_cols(pcb_ctx* c, cplx* rm, long long ld, int k, void* const* cols, bool to_cols) {
    PcbColListW L;
    for (int j0 = 0; j0 < k; j0 += PCB_MAXL) {
        const int kk = (k - j0 < PCB_MAXL) ? k - j0 : PCB_MAXL;
        for (int j = 0; j < kk; ++j) L.p[j] = (cplx*)cols[j0 + j];
        dim3 grid((unsigned)((c->R + 31) / 32), (unsigned)((kk + 31) / 32), 1);
        if (to_cols) PCB_LAUNCH(k_transpose<1>, grid, dim3(256, 1, 1), 0, c->stream, rm + j0, ld, L, kk, c->R);
        else PCB_LAUNCH(k_transpose<0>, grid, dim3(256, 1, 1), 0, c->stream, rm + j0, ld, L, kk, c->R);
        PCB_CUDA_OK(cudaGetLastError());
        c->launches++;
    }
    return 0;
}
// The block travels as one (R, kc) slab per chunk of columns: host row-major -> device staging -> planar columns.
int pcb_block_upload(pcb_ctx* c, const void* host_rm, long long ld, int k, void* const* cols) {
    PCB_CHECK_ARG(host_rm && cols && k > 0 && ld >= k, "bad arguments");
    PCB_CUDA_OK(cudaSetDevice(c->device));
    if (ensure_scratch(c, sizeof(cplx) * (size_t)c->R * (size_t)k)) return -1;
    if (ld == k) {
        PCB_CUDA_OK(cudaMemcpyAsync(c->scratch, host_rm, sizeof(cplx) * (size_t)c->R * k, cudaMemcpyHostToDevice, c->stream));
    } else {
        PCB_CUDA_OK(cudaMemcpy2DAsync(c->scratch, sizeof(cplx) * k, host_rm, sizeof(cplx) * ld, sizeof(cplx) * k, (size_t)c->R,
                                      cudaMemcpyHostToDevice, c->stream));
    }
    if (transpose_cols(c, c->scratch, k, k, cols, true)) return -1;
    PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
    return 0;
}
int pcb_block_download(pcb_ctx* c, void* host_rm, long long ld, int k, const void* const* cols) {
    PCB_CHECK_ARG(host_rm && cols && k > 0 && ld >= k, "bad arguments");
    PCB_CUDA_OK(cudaSetDevice(c->device));
    if (ensure_scratch(c, sizeof(cplx) * (size_t)c->R * (size_t)k)) return -1;
    if (transpose_cols(c, c->scratch, k, k, (void* const*)cols, false)) return -1;
    if (ld == k) {
        PCB_CUDA_OK(cudaMemcpyAsync(host_rm, c->scratch, sizeof(cplx) * (size_t)c->R * k, cudaMemcpyDeviceToHost, c->stream));
    } else {
        PCB_CUDA_OK(cudaMemcpy2DAsync(host_rm, sizeof(cplx) * ld, c->scratch, sizeof(cplx) * k, sizeof(cplx) * k, (size_t)c->R,
                                      cudaMemcpyDeviceToHost, c->stream));
    }
    PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
    return 0;
}
int pcb_fill_uniform(pcb_ctx* c, int k, void* const* cols, unsigned long long seed) {
    PCB_CHECK_ARG(cols && k > 0, "bad arguments");
    PcbColListW L;
    for (int j0 = 0; j0 < k; j0 += PCB_MAXL) {
        const int kk = (k - j0 < PCB_MAXL) ? k - j0 : PCB_MAXL;
        for (int j = 0; j < kk; ++j) L.p[j] = (cplx*)cols[j0 + j];
        dim3 grid((unsigned)grid_for(c, c->R, 256, 8), (unsigned)kk, 1);
        PCB_LAUNCH(k_fill_uniform, grid, dim3(256, 1, 1), 0, c->stream, L, c->nloc, c->nn, (long long)c->z0 * c->N * c->N, j0, seed);
        PCB_CUDA_OK(cudaGetLastError());
        c->launches++;
    }
    return 0;
}

// ---- geometry -------------------------------------------------------------------------------------------------
int pcb_geometry_mask(pcb_ctx* c, int kind, const double* minv, unsigned char* host_mask, unsigned char* host_amb) {
    PCB_CHECK_ARG(c && minv && host_mask && host_amb && kind >= PCB_GEOM_SC_FLAT1 && kind <= PCB_GEOM_FCC, "bad arguments");
    PCB_CUDA_OK(cudaSetDevice(c->device));
    const size_t nn = (size_t)c->nn;
    if (ensure_scratch(c, 2 * nn + 256)) return -1;
    unsigned char* dm = reinterpret_cast<unsigned char*>(c->scratch);
    unsigned char* da = dm + ((nn + 127) / 128) * 128;
    PcbGeom g;
    g.kind = kind;
    for (int i = 0; i < 9; ++i) g.minv[i] = minv[i];
    PCB_LAUNCH(k_geom_mask, dim3((unsigned)((nn + 255) / 256), 1, 1), dim3(256, 1, 1), 0, c->stream, g, c->N, dm, da);
    PCB_CUDA_OK(cudaGetLastError());
    c->launches++;
    PCB_CUDA_OK(cudaMemcpyAsync(host_mask, dm, nn, cudaMemcpyDeviceToHost, c->stream));
    PCB_CUDA_OK(cudaMemcpyAsync(host_amb, da, nn, cudaMemcpyDeviceToHost, c->stream));
    PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
    return 0;
}

// ---- dielectric -----------------------------------------------------------------------------------------------
void pcb_diel_destroy(pcb_diel* d);
int pcb_diel_create(pcb_ctx* c, int kind, const int64_t* ind_e, long long n_e, const int64_t* ind_v, long long n_v,
                    const double* ediag, const double* eoff, int k, const double* stencil, pcb_diel** out) {
    PCB_CHECK_ARG(out && kind >= PCB_DIEL_NONE && kind <= PCB_DIEL_CROSSDOF, "bad kind");
    PCB_CUDA_OK(cudaSetDevice(c->device));
    pcb_diel* d = new pcb_diel;
    d->ctx = c; d->kind = kind; d->mask = nullptr; d->mbits = nullptr; d->mbits2 = nullptr; d->maskp = nullptr; d->maskp2 = nullptr; d->maskp_fe = nullptr;
    d->matp = nullptr; d->inv_eps = nullptr; d->n_mat = 0;
    for (int i = 0; i < 3; ++i) { d->ediag[i] = ediag ? ediag[i] : 1.0; d->eoff[i] = eoff ? cmake(eoff[2 * i], eoff[2 * i + 1]) : cmake(0.0, 0.0); }
    d->st.k = 1; for (int i = 0; i < 8; ++i) d->st.w[i] = 0.0;
    if (kind == PCB_DIEL_CROSSDOF) {
        if (k < 1 || k > 4 || !stencil) { pcb_set_error("pcb_diel_create: crossdof needs 1 <= k <= 4 and the 2k stencil weights"); delete d; return -2; }
        d->st.k = k;
        for (int i = 0; i < 2 * k; ++i) d->st.w[i] = stencil[i];
    }
    const size_t mbytes = (size_t)((c->nn + 3) / 4) * 4;
    PCB_CUDA_OK_OR(cudaMalloc(&d->mask, mbytes), pcb_diel_destroy(d));
    PCB_CUDA_OK_OR(cudaMemsetAsync(d->mask, 0, mbytes, c->stream), pcb_diel_destroy(d));
    const int64_t* lists[2] = {ind_e, ind_v};
    const long long counts[2] = {n_e, (kind == PCB_DIEL_TRIVIAL) ? n_v : 0};
    for (int which = 0; which < 2; ++which) {
        const long long n = counts[which];
        if (n <= 0 || !lists[which]) continue;
        long long* dind = nullptr;
        PCB_CUDA_OK_OR(cudaMalloc(&dind, sizeof(long long) * (size_t)n), pcb_diel_destroy(d));
#define PCB_DIEL_FAIL do { cudaStreamSynchronize(c->stream); cudaFree(dind); pcb_diel_destroy(d); } while (0)
        PCB_CUDA_OK_OR(cudaMemcpyAsync(dind, lists[which], sizeof(long long) * (size_t)n, cudaMemcpyHostToDevice, c->stream), PCB_DIEL_FAIL);
        dim3 grid((unsigned)((n + 255) / 256), 1, 1);
        PCB_LAUNCH(k_mask_from_index, grid, dim3(256, 1, 1), 0, c->stream, (const long long*)dind, n, c->nn, which, (unsigned*)d->mask);
        PCB_CUDA_OK_OR(cudaGetLastError(), PCB_DIEL_FAIL);
        c->launches++;
        PCB_CUDA_OK_OR(cudaStreamSynchronize(c->stream), PCB_DIEL_FAIL);
#undef PCB_DIEL_FAIL
        PCB_CUDA_OK_OR(cudaFree(dind), pcb_diel_destroy(d));
    }
    d->zsplit = c->zsplit;
    const bool whole = !c->zsplit;      // whole-plane forms only: five-sweep pass, clusters for the coupled dielectric
    if (c->plan->plane_mode) {
        const size_t words = c->zsplit ? (size_t)2 * c->plan->zr1 : (size_t)c->plan->r1;
        PCB_CUDA_OK_OR(cudaMalloc(&d->mbits, sizeof(unsigned) * 3 * (size_t)c->N * c->N * words), pcb_diel_destroy(d));
        PcbOp tmp;
        memset(&tmp, 0, sizeof tmp);
        tmp.N = c->N; tmp.nn = c->nn; tmp.nloc = c->nloc; tmp.mask = d->mask; tmp.mbits = d->mbits; tmp.zsplit = c->zsplit;
        PcbCols none;
        memset(&none, 0, sizeof none);
        if (c->plan->pass(tmp, none, 1, PCB_PASS_MASKBITS, c->tw, c->stream, c->sms)) { pcb_diel_destroy(d); return -1; }
        c->launches++;
        if (whole && c->plan->plane_five && c->plan->plane_coupled && kind == PCB_DIEL_TRIVIAL) {
            PCB_CUDA_OK_OR(cudaMalloc(&d->maskp2, (size_t)c->nn), pcb_diel_destroy(d));
            tmp.maskp2 = d->maskp2;
            if (c->plan->pass(tmp, none, 1, PCB_PASS_MASKPLANE2, c->tw, c->stream, c->sms)) { pcb_diel_destroy(d); return -1; }
            c->launches++;
        }
        if (whole && c->plan->plane_five && (kind == PCB_DIEL_CHIRAL || (kind == PCB_DIEL_TRIVIAL && c->plan->plane_coupled))) {
            PCB_CUDA_OK_OR(cudaMalloc(&d->mbits2, sizeof(unsigned) * 3 * (size_t)c->N * c->N * 8), pcb_diel_destroy(d));
            tmp.mbits2 = d->mbits2;
            if (c->plan->pass(tmp, none, 1, PCB_PASS_MASKBITS2, c->tw, c->stream, c->sms)) { pcb_diel_destroy(d); return -1; }
            c->launches++;
        }
        const bool coupled_plane = whole ? c->plan->plane_coupled : c->plan->plane_split_coupled;
        if ((coupled_plane && kind == PCB_DIEL_TRIVIAL) || kind == PCB_DIEL_CROSSDOF) {
            PCB_CUDA_OK_OR(cudaMalloc(&d->maskp, (size_t)c->nn), pcb_diel_destroy(d));
            tmp.maskp = d->maskp;
            if (c->plan->pass(tmp, none, 1, PCB_PASS_MASKPLANE, c->tw, c->stream, c->sms)) { pcb_diel_destroy(d); return -1; }
            c->launches++;
            if (kind == PCB_DIEL_CROSSDOF) {
                // bits 4-6: where each component has a coupling term at all (the fused stencil-on-load skips the rest)
                unsigned char* withact = nullptr;
                PCB_CUDA_OK_OR(cudaMalloc(&withact, (size_t)c->nn), pcb_diel_destroy(d));
                tmp.ctab = c->ctab; tmp.sten = d->st;
                for (int i = 0; i < 3; ++i) tmp.eoff[i] = d->eoff[i];
                PCB_LAUNCH(k_mask_active, dim3((unsigned)((c->nn + 255) / 256), 1, 1), dim3(256, 1, 1), 0, c->stream, tmp, (const unsigned char*)d->maskp, withact);
                PCB_CUDA_OK_OR(cudaGetLastError(), { cudaFree(withact); pcb_diel_destroy(d); });
                PCB_CUDA_OK_OR(cudaStreamSynchronize(c->stream), { cudaFree(withact); pcb_diel_destroy(d); });
                cudaFree(d->maskp);
                d->maskp = withact;
                c->launches++;
            }
        }
    }
    PCB_CUDA_OK_OR(cudaStreamSynchronize(c->stream), pcb_diel_destroy(d));
    *out = d;
    return 0;
}
int pcb_diel_create_materials(pcb_ctx* c, const uint8_t* mat, long long n, const double* inv_eps, int n_mat, pcb_diel** out) {
    PCB_CHECK_ARG(c && mat && inv_eps && out, "null");
    if (c->nloc != c->nn) {
        pcb_set_error("pcb_diel_create_materials: needs whole columns; a slab context has no dielectric of this kind");
        return -2;
    }
    // the whole input is checked before anything is allocated
    if (n != 3 * c->nn) { pcb_set_error("pcb_diel_create_materials: n = %lld, expected 3 N^3 = %lld", n, 3 * c->nn); return -1; }
    if (n_mat < 1 || n_mat > 256) { pcb_set_error("pcb_diel_create_materials: n_mat = %d, expected 1 ... 256", n_mat); return -1; }
    for (int i = 0; i < n_mat; ++i)
        if (!std::isfinite(inv_eps[i]) || !(inv_eps[i] > 0.0)) { pcb_set_error("pcb_diel_create_materials: inv_eps[%d] = %g is not finite and > 0", i, inv_eps[i]); return -1; }
    unsigned char top = 0;
    for (long long r = 0; r < n; ++r) top = mat[r] > top ? mat[r] : top;
    if (top >= n_mat) {
        long long r = 0;
        while (mat[r] < n_mat) ++r;
        pcb_set_error("pcb_diel_create_materials: mat[%lld] = %d >= n_mat = %d", r, (int)mat[r], n_mat);
        return -1;
    }
    PCB_CUDA_OK(cudaSetDevice(c->device));
    pcb_diel* d = new pcb_diel;
    d->ctx = c; d->kind = PCB_DIEL_MATERIALS; d->mask = nullptr; d->mbits = nullptr; d->mbits2 = nullptr; d->maskp = nullptr; d->maskp2 = nullptr; d->maskp_fe = nullptr;
    d->matp = nullptr; d->inv_eps = nullptr; d->n_mat = n_mat; d->zsplit = c->zsplit;
    for (int i = 0; i < 3; ++i) { d->ediag[i] = 1.0; d->eoff[i] = cmake(0.0, 0.0); }
    d->st.k = 1; for (int i = 0; i < 8; ++i) d->st.w[i] = 0.0;
    PCB_CUDA_OK_OR(cudaMalloc(&d->mask, (size_t)n), pcb_diel_destroy(d));
    PCB_CUDA_OK_OR(cudaMalloc(&d->inv_eps, sizeof(double) * (size_t)n_mat), pcb_diel_destroy(d));
    PCB_CUDA_OK_OR(cudaMemcpyAsync(d->mask, mat, (size_t)n, cudaMemcpyHostToDevice, c->stream), pcb_diel_destroy(d));
    PCB_CUDA_OK_OR(cudaMemcpyAsync(d->inv_eps, inv_eps, sizeof(double) * (size_t)n_mat, cudaMemcpyHostToDevice, c->stream), pcb_diel_destroy(d));
    if (c->plan->plane_mode) {
        // the index bytes of every z item of the plane pass, padded to pcb_mat_pad(ZR2) bytes (whole or half planes, as mbits)
        const int zr1 = c->zsplit ? c->plan->zr1 : c->plan->r1, zr2 = c->zsplit ? c->plan->zr2 : c->plan->r2;
        const size_t bytes = 3 * (size_t)c->N * c->N * (c->zsplit ? 2 : 1) * zr1 * pcb_mat_pad(zr2);
        PCB_CUDA_OK_OR(cudaMalloc(&d->matp, bytes), pcb_diel_destroy(d));
        PcbOp tmp;
        memset(&tmp, 0, sizeof tmp);
        tmp.N = c->N; tmp.nn = c->nn; tmp.nloc = c->nloc; tmp.mat = d->mask; tmp.matp = d->matp; tmp.zsplit = c->zsplit;
        PcbCols none;
        memset(&none, 0, sizeof none);
        if (c->plan->pass(tmp, none, 1, PCB_PASS_MATBYTES, c->tw, c->stream, c->sms)) { pcb_diel_destroy(d); return -1; }
        c->launches++;
    }
    PCB_CUDA_OK_OR(cudaStreamSynchronize(c->stream), pcb_diel_destroy(d));
    *out = d;
    return 0;
}
// A new 1 / eps table in the same allocation: the operators built on d read it from their next launch.  Stream-ordered behind the
// work already queued, and synchronous, so that the host array may be reused on return.
int pcb_diel_set_inv_eps(pcb_diel* d, const double* inv_eps, int n_mat) {
    PCB_CHECK_ARG(d && inv_eps, "null");
    if (d->kind != PCB_DIEL_MATERIALS) { pcb_set_error("pcb_diel_set_inv_eps: dielectric kind %d is not PCB_DIEL_KIND_MATERIALS", d->kind); return -1; }
    if (n_mat != d->n_mat) { pcb_set_error("pcb_diel_set_inv_eps: n_mat = %d, the dielectric has %d materials", n_mat, d->n_mat); return -1; }
    for (int i = 0; i < n_mat; ++i)
        if (!std::isfinite(inv_eps[i]) || !(inv_eps[i] > 0.0)) { pcb_set_error("pcb_diel_set_inv_eps: inv_eps[%d] = %g is not finite and > 0", i, inv_eps[i]); return -1; }
    pcb_ctx* c = d->ctx;
    PCB_CUDA_OK(cudaSetDevice(c->device));
    PCB_CUDA_OK(cudaMemcpyAsync(d->inv_eps, inv_eps, sizeof(double) * (size_t)n_mat, cudaMemcpyHostToDevice, c->stream));
    PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
    return 0;
}
void pcb_diel_destroy(pcb_diel* d) {
    if (!d) return;
    cudaSetDevice(d->ctx->device);
    cudaStreamSynchronize(d->ctx->stream);
    if (d->mask) cudaFree(d->mask);
    if (d->mbits) cudaFree(d->mbits);
    if (d->maskp) cudaFree(d->maskp);
    if (d->mbits2) cudaFree(d->mbits2);
    if (d->maskp2) cudaFree(d->maskp2);
    if (d->maskp_fe) cudaFree(d->maskp_fe);
    if (d->matp) cudaFree(d->matp);
    if (d->inv_eps) cudaFree(d->inv_eps);
    delete d;
}

// ---- operator ---------------------------------------------------------------------------------------------------
static void op_fill(pcb_op* o, double gamma, double shift, double pshift, pcb_diel* diel) {
    pcb_ctx* c = o->ctx;
    o->diel = diel;
    o->d.N = c->N; o->d.nn = c->nn; o->d.nloc = c->nloc; o->d.z0 = c->z0; o->d.T = o->T;
    o->d.gamma = gamma; o->d.shift = shift; o->d.pshift = pshift;
    o->d.inv_n3 = 1.0 / (double)c->nn;
    o->d.diel = diel ? diel->kind : PCB_DIEL_NONE;
    o->d.mask = diel ? diel->mask : nullptr;
    o->d.mbits = diel ? diel->mbits : nullptr;
    o->d.maskp = diel ? diel->maskp : nullptr;
    o->d.mbits2 = diel ? diel->mbits2 : nullptr;
    o->d.maskp2 = diel ? diel->maskp2 : nullptr;
    if (diel && diel->kind == PCB_DIEL_MATERIALS) { o->d.matp = diel->matp; o->d.inv_eps = diel->inv_eps; }
    if (diel) o->d.sten = diel->st; else { o->d.sten.k = 1; for (int i = 0; i < 8; ++i) o->d.sten.w[i] = 0.0; }
    o->d.ctab = c->ctab;
    o->d.zsplit = c->zsplit;
    o->d.dist = nullptr;
    // five-sweep plane pass: where it is the faster form -- N = 8 x 15 with the identity / isotropic M (0.80 vs 0.815 ms); the coupled M
    // on clusters is faster in the seven-sweep kernel (1.20 vs 1.44 ms: with 8 warps the split sweep C and the DSMEM step cost more)
    o->d.mid_five = (c->plan->plane_five && !c->zsplit && (c->use_mid_five == 1 ||
                     (c->use_mid_five == -1 && c->plan->r2 >= 15 && o->d.diel != PCB_DIEL_TRIVIAL))) ? 1 : 0;
    for (int i = 0; i < 3; ++i) {
        o->d.ediag[i] = diel ? diel->ediag[i] : 1.0;
        o->d.eoff[i] = diel ? diel->eoff[i] : cmake(0.0, 0.0);
    }
}
int pcb_op_update(pcb_op* o, const double* tables, double gamma, double shift, double pshift, pcb_diel* diel) {
    PCB_CHECK_ARG(o && tables, "null");
    pcb_ctx* c = o->ctx;
    PCB_CHECK_ARG(!diel || diel->ctx == c, "dielectric belongs to another context");
    PCB_CHECK_ARG(!diel || diel->zsplit == c->zsplit, "dielectric was created under the other plane-mode form (plane_split); re-create it");
    PCB_CUDA_OK(cudaSetDevice(c->device));
    const size_t bytes = sizeof(cplx) * 9 * (size_t)c->N;
    if (ensure_hstage(c, bytes > 65536 ? bytes : 65536)) return -1;
    PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
    memcpy(c->hstage, tables, bytes);
    PCB_CUDA_OK(cudaMemcpyAsync(o->T, c->hstage, bytes, cudaMemcpyHostToDevice, c->stream));
    PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
    op_fill(o, gamma, shift, pshift, diel);
    return 0;
}
int pcb_op_create(pcb_ctx* c, const double* tables, double gamma, double shift, double pshift, pcb_diel* diel, pcb_op** out) {
    PCB_CHECK_ARG(c && tables && out, "null");
    PCB_CUDA_OK(cudaSetDevice(c->device));
    pcb_op* o = new pcb_op;
    o->ctx = c; o->T = nullptr; o->diel = nullptr;
    PCB_CUDA_OK(cudaMalloc(&o->T, sizeof(cplx) * 9 * (size_t)c->N));
    if (int rc = pcb_op_update(o, tables, gamma, shift, pshift, diel)) { cudaFree(o->T); delete o; return rc; }
    *out = o;
    return 0;
}
void pcb_op_destroy(pcb_op* o) {
    if (!o) return;
    cudaSetDevice(o->ctx->device);
    cudaStreamSynchronize(o->ctx->stream);
    if (o->T) cudaFree(o->T);
    delete o;
}

// Y_j = M_CrossDoF X_j for kc columns in one launch (blockIdx.y = column)
static int launch_crossdof(pcb_op* o, int kc, const cplx* const* X, cplx* const* Y) {
    pcb_ctx* c = o->ctx;
    PcbCols cols;
    for (int j = 0; j < kc; ++j) { cols.in[j] = X[j]; cols.out[j] = Y[j]; }
    dim3 grid((unsigned)((c->nn + 255) / 256), (unsigned)kc, 1);
    if (o->diel->st.k == 1) PCB_LAUNCH(k_diel_crossdof<1>, grid, dim3(256, 1, 1), 0, c->stream, o->d, o->diel->st, cols);
    else if (o->diel->st.k == 2) PCB_LAUNCH(k_diel_crossdof<2>, grid, dim3(256, 1, 1), 0, c->stream, o->d, o->diel->st, cols);
    else PCB_LAUNCH(k_diel_crossdof<0>, grid, dim3(256, 1, 1), 0, c->stream, o->d, o->diel->st, cols);
    PCB_CUDA_OK(cudaGetLastError());
    c->launches++;
    return 0;
}

// the same on the plane-slot layout: cols.wrk -> cols.out (between the halves of the plane pass)
static int launch_crossdof_t(pcb_op* o, int kc, const PcbCols& cols) {
    pcb_ctx* c = o->ctx;
    dim3 grid((unsigned)((c->nn + 255) / 256), (unsigned)kc, 1);
    if (o->diel->st.k == 1) PCB_LAUNCH(k_diel_crossdof_t<1>, grid, dim3(256, 1, 1), 0, c->stream, o->d, o->diel->st, cols);
    else if (o->diel->st.k == 2) PCB_LAUNCH(k_diel_crossdof_t<2>, grid, dim3(256, 1, 1), 0, c->stream, o->d, o->diel->st, cols);
    else PCB_LAUNCH(k_diel_crossdof_t<0>, grid, dim3(256, 1, 1), 0, c->stream, o->d, o->diel->st, cols);
    PCB_CUDA_OK(cudaGetLastError());
    c->launches++;
    return 0;
}

// Pass structure of an A / H apply (DESIGN.md 3): 0 plane mode (3 passes), 1 five passes, 2 five passes split around the
// cross-DoF stencil (7 kernels), 3 plane mode split around the stencil on the slot layout (5 kernels), 4 plane halves with the
// stencil fused into the inverse half (4 kernels)
enum { PCB_STRUCT_PLANE = 0, PCB_STRUCT_FIVE = 1, PCB_STRUCT_CROSS7 = 2, PCB_STRUCT_CROSS5 = 3, PCB_STRUCT_CROSS4 = 4 };
// A / H of this context run on the plane layout (transposed scratch columns) for every dielectric kind that has a plane structure
static bool plane_layout(const pcb_ctx* c) { return c->use_plane && (c->zsplit || c->plan->plane_split != 2); }
static int apply_structure(const pcb_op* o) {
    const pcb_ctx* c = o->ctx;
    const int diel = o->d.diel;
    if (plane_layout(c)) {
        if (diel == PCB_DIEL_NONE || diel == PCB_DIEL_CHIRAL || diel == PCB_DIEL_MATERIALS) return PCB_STRUCT_PLANE;
        if (diel == PCB_DIEL_TRIVIAL && c->use_plane_coupled && (c->zsplit ? c->plan->plane_split_coupled : c->plan->plane_coupled)) return PCB_STRUCT_PLANE;
        if (diel == PCB_DIEL_CROSSDOF && c->use_plane_cross) return c->use_plane_cross == 2 ? PCB_STRUCT_CROSS5 : PCB_STRUCT_CROSS4;
    }
    return diel == PCB_DIEL_CROSSDOF ? PCB_STRUCT_CROSS7 : PCB_STRUCT_FIVE;
}

// In-place columns (in[j] == out[j]) are refused where the pass structure re-reads X after writing `out` (H outside the plane
// mode) or uses `out` as work space (cross-DoF plane halves, cross-DoF M).  Every column is checked before anything is enqueued:
// a refused call returns -2 with all output columns untouched, also when the aliased column sits in a later launch chunk.
// PCB_APPLY_DFIELD / PCB_APPLY_EFIELD read x only in their first pass (the cross-DoF stencil of EFIELD reads the forward passes'
// output from the scratch), so they take in[j] == out[j] in every pass structure.
static bool refuses_inplace_AH(int mode, int st) {
    return (mode == PCB_APPLY_H && st != PCB_STRUCT_PLANE) || st == PCB_STRUCT_CROSS5 || st == PCB_STRUCT_CROSS4;
}
static int check_inplace(const pcb_op* o, int mode, int ncols, const void* const* in, void* const* out, const char* fn) {
    bool refused = false;
    if (mode == PCB_APPLY_M) refused = (o->d.diel == PCB_DIEL_CROSSDOF);
    else if (mode == PCB_APPLY_A || mode == PCB_APPLY_H) refused = refuses_inplace_AH(mode, apply_structure(o));
    else if (mode == PCB_APPLY_EFOURIER) refused = refuses_inplace_AH(PCB_APPLY_A, apply_structure(o));      // A's passes, A's rule
    if (!refused) return 0;
    for (int j = 0; j < ncols; ++j)
        if (in[j] == out[j]) {
            pcb_set_error("%s: in[%d] == out[%d]; this mode re-reads X / uses out as work space here, use distinct columns", fn, j, j);
            return -2;
        }
    return 0;
}

// One kernel of an apply: a pass id, or the cross-DoF stencil on the natural layout (STENCIL: scratch -> out) or on the
// plane-slot layout (STENCIL_T: cols.wrk -> out).  The columns it runs on: IO in -> out; SCR in -> the scratch (a natural-layout
// pass with the scratch as its `out`); WRK in / out with the scratch as the transposed work columns cols.wrk (plane layout).
enum { PCB_STEP_STENCIL = -1, PCB_STEP_STENCIL_T = -2 };
enum { PCB_COLS_IO = 0, PCB_COLS_SCR = 1, PCB_COLS_WRK = 2 };
struct PcbStep { int kern, cols; };
struct PcbSteps { int n; PcbStep s[7]; };

// mode PCB_APPLY_EFOURIER runs the passes of A with a plain inverse x pass last (no K_A): out = IFFT3(M FFT3(K_A^H x)).
// dist bit 0: the first x pass reads the input slabs of all ranks through o->d.dist, bit 1: the last x pass writes the output slabs.
static int last_pass(int mode, bool dout, bool trn) {
    if (mode == PCB_APPLY_EFOURIER) return trn ? PCB_PASS_XINV_T : PCB_PASS_XINV;
    if (mode == PCB_APPLY_A) return trn ? (dout ? PCB_PASS_XINV_A_TD : PCB_PASS_XINV_A_T) : (dout ? PCB_PASS_XINV_A_D : PCB_PASS_XINV_A);
    return trn ? (dout ? PCB_PASS_XINV_H_TD : PCB_PASS_XINV_H_T) : (dout ? PCB_PASS_XINV_H_D : PCB_PASS_XINV_H);
}
static PcbSteps structure_steps(int st, int mode, int dist) {
    const bool din = dist & 1, dout = dist & 2;
    const int first = din ? PCB_PASS_XFWD_SYM_D : PCB_PASS_XFWD_SYM, first_t = din ? PCB_PASS_XFWD_SYM_TD : PCB_PASS_XFWD_SYM_T;
    const int last = last_pass(mode, dout, false), last_t = last_pass(mode, dout, true);
    enum { IO = PCB_COLS_IO, SCR = PCB_COLS_SCR, WRK = PCB_COLS_WRK };
    switch (st) {
        case PCB_STRUCT_PLANE:      // x forward -> transposed scratch, fused y/z/M/z/y on (i1,i2) planes, x inverse -> out
            // (Round 2, measured and removed: running the three passes on chunks of 1 / 2 / 4 columns so that the scratch of a chunk
            // (83 MB per column) could stay in the 126 MB L2 between the passes: 2.76 / 2.44 / 2.22 ms instead of 2.02 ms per 16
            // columns -- the per-chunk launches lose more in partial waves (360 planes per column on 148 SMs) than L2 residency returns.)
            return {3, {{first_t, WRK}, {PCB_PASS_MID, WRK}, {last_t, WRK}}};
        case PCB_STRUCT_CROSS4:     // x forward -> scratch, forward half of the plane pass scratch -> out (real-space planes, slot
                                    // layout), inverse half with the stencil applied on load out -> scratch, x inverse scratch -> out
            return {4, {{first_t, WRK}, {PCB_PASS_MID_FWD_O, WRK}, {PCB_PASS_MID_INV_ST, WRK}, {last_t, WRK}}};
        case PCB_STRUCT_CROSS5:     // x forward -> scratch, forward half of the plane pass in place, stencil scratch -> out (slot
                                    // layout), inverse half out -> scratch, x inverse scratch -> out
            return {5, {{first_t, WRK}, {PCB_PASS_MID_FWD, WRK}, {PCB_STEP_STENCIL_T, WRK}, {PCB_PASS_MID_INV, WRK}, {last_t, WRK}}};
        case PCB_STRUCT_CROSS7:     // cross-DoF M is a stencil in real space: forward passes into scratch, M scratch -> out, inverse in place
            return {7, {{first, SCR}, {PCB_PASS_YFWD, SCR}, {PCB_PASS_ZFWD, SCR}, {PCB_STEP_STENCIL, SCR},
                        {PCB_PASS_ZINV, IO}, {PCB_PASS_YINV, IO}, {last, IO}}};
        default:
            return {5, {{first, IO}, {PCB_PASS_YFWD, IO}, {PCB_PASS_ZMID, IO}, {PCB_PASS_YINV, IO}, {last, IO}}};
    }
}
// The kernels of an A / H / EFOURIER apply in launch order
static PcbSteps apply_steps(const pcb_op* o, int mode, int dist) {
    int st = apply_structure(o);
    if (dist && o->ctx->zsplit) st = (o->d.diel == PCB_DIEL_CROSSDOF) ? PCB_STRUCT_CROSS7 : PCB_STRUCT_FIVE;      // no peer-memory x passes on split tiles
    return structure_steps(st, mode, dist);
}
// The forward half of a layout, D = FFT3(K_A^H x): the steps of its split structure (CROSS5 on the plane layout, CROSS7 on the
// natural layout) before the stencil
static PcbSteps forward_steps(bool plane) {
    PcbSteps p = structure_steps(plane ? PCB_STRUCT_CROSS5 : PCB_STRUCT_CROSS7, PCB_APPLY_A, 0);
    p.n = 0;
    while (p.s[p.n].kern >= 0) ++p.n;
    return p;
}

// Runs the steps on kc columns (cols.in -> cols.out) with the context's scratch where a step uses it, counting one launch per
// kernel.  ev (pcb_apply_timed): ev[0] is recorded once the scratch is set up, ev[i + 1] after step i.
static int run_steps(pcb_op* o, const PcbSteps& p, PcbCols cols, int kc, cudaEvent_t* ev = nullptr) {
    pcb_ctx* c = o->ctx;
    bool scratch = false;
    for (int i = 0; i < p.n; ++i) scratch |= (p.s[i].cols != PCB_COLS_IO);
    PcbCols sc = cols;
    if (scratch) {
        if (ensure_scratch(c, sizeof(cplx) * (size_t)c->R * (size_t)kc)) return -1;
        for (int j = 0; j < kc; ++j) cols.wrk[j] = sc.wrk[j] = sc.out[j] = c->scratch + (size_t)j * c->R;
    }
    if (ev) PCB_CUDA_OK(cudaEventRecord(ev[0], c->stream));
    for (int i = 0; i < p.n; ++i) {
        const int k = p.s[i].kern;
        if (k == PCB_STEP_STENCIL) { if (launch_crossdof(o, kc, sc.out, cols.out)) return -1; }
        else if (k == PCB_STEP_STENCIL_T) { if (launch_crossdof_t(o, kc, cols)) return -1; }
        else {
            if (c->plan->pass(o->d, p.s[i].cols == PCB_COLS_SCR ? sc : cols, kc, k, c->tw, c->stream, c->sms)) return -1;
            c->launches++;
        }
        if (ev) PCB_CUDA_OK(cudaEventRecord(ev[i + 1], c->stream));
    }
    return 0;
}

// A / H on kc columns (cols.in -> cols.out).  dist: the x passes read / write the slabs of all ranks through o->d.dist
// (large-grid mode over peer memory); cols.in then holds the local X copies and cols.out local work columns.
static int apply_AH(pcb_op* o, int mode, const PcbCols& cols, int kc, int j0, int dist) {
    if (refuses_inplace_AH(mode, apply_structure(o)) || dist)      // (pcb_apply has checked all its columns already; pcb_apply_dist has not)
        for (int j = 0; j < kc; ++j)
            if (cols.in[j] == cols.out[j]) {
                pcb_set_error("pcb_apply: in[%d] == out[%d]; this pass structure re-reads X / uses out as work space, use distinct columns", j0 + j, j0 + j);
                return -2;
            }
    return run_steps(o, apply_steps(o, mode, dist), cols, kc);
}

// Y = M X for one column of a point-wise dielectric (none / chiral / trivial / materials), in place allowed
static int launch_point_diel(pcb_op* o, const cplx* X, cplx* Y) {
    pcb_ctx* c = o->ctx;
    dim3 grid((unsigned)grid_for(c, c->nn, 256, 8), 1, 1);
    if (o->d.diel == PCB_DIEL_MATERIALS) PCB_LAUNCH(k_diel_mat, grid, dim3(256, 1, 1), 0, c->stream, o->d, X, Y);
    else PCB_LAUNCH(k_diel_point, grid, dim3(256, 1, 1), 0, c->stream, o->d, X, Y);
    PCB_CUDA_OK(cudaGetLastError());
    c->launches++;
    return 0;
}

// D = FFT3(K_A^H x) (DFIELD) or E = M D (EFIELD) in the natural layout: the forward half, then for E the point-wise M in place
// on out, or the cross-DoF stencil from the scratch into out.
static int apply_field(pcb_op* o, int mode, const PcbCols& cols, int kc) {
    pcb_ctx* c = o->ctx;
    const bool stencil = (mode == PCB_APPLY_EFIELD && o->d.diel == PCB_DIEL_CROSSDOF);
    PcbSteps p = forward_steps(false);
    if (stencil) p.s[p.n++] = {PCB_STEP_STENCIL, PCB_COLS_SCR};
    else for (int i = 0; i < p.n; ++i) p.s[i].cols = PCB_COLS_IO;      // D straight into out
    if (run_steps(o, p, cols, kc)) return -1;
    if (mode != PCB_APPLY_EFIELD || o->d.diel == PCB_DIEL_NONE || stencil) return 0;
    for (int j = 0; j < kc; ++j)
        if (launch_point_diel(o, cols.out[j], cols.out[j])) return -1;
    return 0;
}

int pcb_apply(pcb_op* o, int mode, int ncols, const void* const* in, void* const* out) {
    PCB_CHECK_ARG(o && in && out && ncols > 0, "bad arguments");
    pcb_ctx* c = o->ctx;
    PCB_CUDA_OK(cudaSetDevice(c->device));
    const PcbOpLaunch* pl = c->plan;
    const bool cross = (o->d.diel == PCB_DIEL_CROSSDOF);
    if (c->nloc != c->nn && mode != PCB_APPLY_P) {
        pcb_set_error("pcb_apply: mode %d needs whole columns; a slab context only supports PCB_APPLY_P (gather with pcb_slab_exchange)", mode);
        return -2;
    }
    if (int rc = check_inplace(o, mode, ncols, in, out, "pcb_apply")) return rc;
    for (int j0 = 0; j0 < ncols; j0 += PCB_MAXC) {
        const int kc = (ncols - j0 < PCB_MAXC) ? ncols - j0 : PCB_MAXC;
        PcbCols cols;
        for (int j = 0; j < kc; ++j) { cols.in[j] = (const cplx*)in[j0 + j]; cols.out[j] = (cplx*)out[j0 + j]; }
        switch (mode) {
            case PCB_APPLY_FFT: case PCB_APPLY_IFFT:
                // plain transforms are in place on `out`; copy first when out of place
                for (int j = 0; j < kc; ++j)
                    if (cols.in[j] != cols.out[j]) PCB_CUDA_OK(cudaMemcpyAsync(cols.out[j], cols.in[j], sizeof(cplx) * (size_t)c->R, cudaMemcpyDeviceToDevice, c->stream));
                if (pl->apply(o->d, cols, kc, mode == PCB_APPLY_FFT ? 0 : 1, c->tw, c->stream, c->sms)) return -1;
                c->launches += 3;
                break;
            case PCB_APPLY_A: case PCB_APPLY_H: case PCB_APPLY_EFOURIER:
                if (int rc = apply_AH(o, mode, cols, kc, j0, 0)) return rc;
                break;
            case PCB_APPLY_P: {
                PcbResidArgs a;
                for (int j = 0; j < kc; ++j) { a.x[j] = cols.in[j]; a.hx[j] = nullptr; a.w[j] = cols.out[j]; a.lambda[j] = 0.0; }
                const int gx = grid_for(c, c->nloc, 256, 4);
                if (ensure_partial(c, sizeof(double) * (size_t)gx * PCB_MAXC_RP)) return -1;
                dim3 grid((unsigned)gx, (unsigned)((kc + PCB_RP_CH - 1) / PCB_RP_CH), 1);
                PCB_LAUNCH(k_resid_precond<2>, grid, dim3(256, 1, 1), 0, c->stream, o->d, a, kc, c->partial);
                PCB_CUDA_OK(cudaGetLastError());
                c->launches++;
            } break;
            case PCB_APPLY_M:
                if (cross && launch_crossdof(o, kc, cols.in, cols.out)) return -1;      // (in place refused by check_inplace)
                for (int j = 0; j < kc && !cross; ++j)
                    if (launch_point_diel(o, cols.in[j], cols.out[j])) return -1;
                break;
            case PCB_APPLY_DFIELD: case PCB_APPLY_EFIELD:
                if (int rc = apply_field(o, mode, cols, kc)) return rc;
                break;
            case PCB_APPLY_KA: case PCB_APPLY_KAH: case PCB_APPLY_KB: {
                dim3 grid((unsigned)grid_for(c, c->nn, 256, 8), (unsigned)kc, 1);
                if (mode == PCB_APPLY_KA) PCB_LAUNCH(k_symbol_point<0>, grid, dim3(256, 1, 1), 0, c->stream, o->d, cols);
                else if (mode == PCB_APPLY_KAH) PCB_LAUNCH(k_symbol_point<1>, grid, dim3(256, 1, 1), 0, c->stream, o->d, cols);
                else PCB_LAUNCH(k_symbol_point<2>, grid, dim3(256, 1, 1), 0, c->stream, o->d, cols);
                PCB_CUDA_OK(cudaGetLastError());
                c->launches++;
            } break;
            default:
                pcb_set_error("pcb_apply: unknown mode %d", mode);
                return -2;
        }
    }
    return 0;
}

int pcb_apply_timed(pcb_op* o, int mode, int ncols, const void* const* in, void* const* out, float* pass_ms, int* npass) {
    PCB_CHECK_ARG(o && in && out && pass_ms && npass && ncols > 0 && ncols <= PCB_MAXC, "bad arguments (ncols <= 32)");
    PCB_CHECK_ARG(mode == PCB_APPLY_A || mode == PCB_APPLY_H, "mode must be PCB_APPLY_A or PCB_APPLY_H");
    if (int rc = check_inplace(o, mode, ncols, in, out, "pcb_apply_timed")) return rc;
    pcb_ctx* c = o->ctx;
    PCB_CUDA_OK(cudaSetDevice(c->device));
    PcbCols cols;
    for (int j = 0; j < ncols; ++j) { cols.in[j] = (const cplx*)in[j]; cols.out[j] = (cplx*)out[j]; }
    const PcbSteps p = apply_steps(o, mode, 0);
    cudaEvent_t ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
#define PCB_EV_FREE do { for (int q = 0; q < 8; ++q) if (ev[q]) cudaEventDestroy(ev[q]); } while (0)
    for (int i = 0; i < 8; ++i) PCB_CUDA_OK_OR(cudaEventCreate(&ev[i]), PCB_EV_FREE);
    if (run_steps(o, p, cols, ncols, ev)) { cudaStreamSynchronize(c->stream); PCB_EV_FREE; return -1; }
    PCB_CUDA_OK_OR(cudaEventSynchronize(ev[p.n]), PCB_EV_FREE);
    for (int i = 0; i < p.n; ++i) PCB_CUDA_OK_OR(cudaEventElapsedTime(&pass_ms[i], ev[i], ev[i + 1]), PCB_EV_FREE);
    PCB_EV_FREE;
#undef PCB_EV_FREE
    *npass = p.n;
    return 0;
}

// ---- electric energy of modes in the dielectric -------------------------------------------------------------------
// The slot-ordered byte mask the plane-layout energy kernel reads: the dielectric's own maskp where it has one (coupled M on
// clusters, cross-DoF: bits 0-3 are k_mask_plane's), else built here once and kept until pcb_diel_destroy.
static const unsigned char* energy_slot_mask(pcb_op* o) {
    pcb_diel* d = o->diel;
    if (d->maskp) return d->maskp;
    if (d->maskp_fe) return d->maskp_fe;
    pcb_ctx* c = o->ctx;
    unsigned char* mp = nullptr;
    if (cudaMalloc(&mp, (size_t)c->nn) != cudaSuccess) { (void)cudaGetLastError(); pcb_set_error("pcb_field_energy: cudaMalloc of the slot mask failed"); return nullptr; }
    PcbOp tmp;
    memset(&tmp, 0, sizeof tmp);
    tmp.N = c->N; tmp.nn = c->nn; tmp.nloc = c->nloc; tmp.mask = d->mask; tmp.maskp = mp; tmp.zsplit = d->zsplit;
    PcbCols none;
    memset(&none, 0, sizeof none);
    if (c->plan->pass(tmp, none, 1, PCB_PASS_MASKPLANE, c->tw, c->stream, c->sms)) { cudaStreamSynchronize(c->stream); cudaFree(mp); return nullptr; }
    c->launches++;
    d->maskp_fe = mp;
    return mp;
}

// e_in / e_tot of kc columns: forward passes into the scratch (the plane layout where A / H run in plane mode, else the natural
// layout), the energy kernel over a fixed grid of gx CTAs per column, then the fixed-order sum of the partials into `dout`.
static int field_energy_chunk(pcb_op* o, const PcbCols& cols, int kc, bool plane, const unsigned char* smask, int gx, double* dout) {
    pcb_ctx* c = o->ctx;
    if (run_steps(o, forward_steps(plane), cols, kc)) return -1;
    PcbCols e;
    memset(&e, 0, sizeof e);
    for (int j = 0; j < kc; ++j) e.in[j] = c->scratch + (size_t)j * c->R;
    PcbOp d = o->d;
    if (plane) d.maskp = smask;
    const PcbStencil st = d.sten;
    const int k = st.k;
    dim3 grid((unsigned)gx, (unsigned)kc, 1), blk(256, 1, 1);
    double* part = c->partial;
#define PCB_FE_GO(KERN)                                                                                             \
    do {                                                                                                            \
        switch (d.diel) {                                                                                           \
            case PCB_DIEL_NONE: PCB_LAUNCH((KERN<0, 1>), grid, blk, 0, c->stream, d, st, e, kc, part); break;       \
            case PCB_DIEL_CHIRAL: PCB_LAUNCH((KERN<1, 1>), grid, blk, 0, c->stream, d, st, e, kc, part); break;     \
            case PCB_DIEL_TRIVIAL: PCB_LAUNCH((KERN<2, 1>), grid, blk, 0, c->stream, d, st, e, kc, part); break;    \
            case PCB_DIEL_MATERIALS: PCB_LAUNCH((KERN<4, 1>), grid, blk, 0, c->stream, d, st, e, kc, part); break;  \
            default:                                                                                                \
                if (k == 1) PCB_LAUNCH((KERN<3, 1>), grid, blk, 0, c->stream, d, st, e, kc, part);                  \
                else if (k == 2) PCB_LAUNCH((KERN<3, 2>), grid, blk, 0, c->stream, d, st, e, kc, part);             \
                else PCB_LAUNCH((KERN<3, 0>), grid, blk, 0, c->stream, d, st, e, kc, part);                         \
        }                                                                                                           \
    } while (0)
    if (plane) PCB_FE_GO(k_field_energy_t);
    else PCB_FE_GO(k_field_energy);
#undef PCB_FE_GO
    PCB_CUDA_OK(cudaGetLastError());
    PCB_LAUNCH(k_sum_partials, dim3(1, 1, 1), dim3(64, 1, 1), 0, c->stream, (const double*)part, gx, 2 * kc, dout);
    PCB_CUDA_OK(cudaGetLastError());
    c->launches += 2;
    return 0;
}

int pcb_field_energy(pcb_op* o, int ncols, const void* const* x, double* e_in, double* e_tot) {
    PCB_CHECK_ARG(o && x && e_in && e_tot && ncols > 0, "bad arguments");
    pcb_ctx* c = o->ctx;
    PCB_CUDA_OK(cudaSetDevice(c->device));
    if (c->nloc != c->nn) {
        pcb_set_error("pcb_field_energy: needs whole columns; a slab context only supports PCB_APPLY_P (gather with pcb_slab_exchange)");
        return -2;
    }
    PCB_CHECK_ARG(!o->diel || o->diel->zsplit == c->zsplit, "dielectric was created under the other plane-mode form (plane_split); re-create it");
    const bool plane = plane_layout(c);
    const unsigned char* smask = nullptr;
    if (plane && o->d.diel != PCB_DIEL_NONE && o->d.diel != PCB_DIEL_MATERIALS && !(smask = energy_slot_mask(o))) return -1;
    const int gx = grid_for(c, c->nn, 256, 4);      // fixed for the context: the same partials for a column at any width
    const int kmax = ncols < PCB_MAXC ? ncols : PCB_MAXC;
    if (ensure_partial(c, sizeof(double) * ((size_t)gx + 1) * 2 * PCB_MAXC)) return -1;
    if (ensure_hstage(c, 65536)) return -1;
    if (ensure_scratch(c, sizeof(cplx) * (size_t)c->R * (size_t)kmax)) return -1;
    double* dout = c->partial + (size_t)gx * 2 * PCB_MAXC;
    for (int j0 = 0; j0 < ncols; j0 += PCB_MAXC) {
        const int kc = (ncols - j0 < PCB_MAXC) ? ncols - j0 : PCB_MAXC;
        PcbCols cols;
        memset(&cols, 0, sizeof cols);
        for (int j = 0; j < kc; ++j) cols.in[j] = (const cplx*)x[j0 + j];
        if (field_energy_chunk(o, cols, kc, plane, smask, gx, dout)) return -1;
        PCB_CUDA_OK(cudaMemcpyAsync(c->hstage, dout, sizeof(double) * 2 * kc, cudaMemcpyDeviceToHost, c->stream));
        PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
        const double* h = (const double*)c->hstage;
        for (int j = 0; j < kc; ++j) { e_in[j0 + j] = h[2 * j] / (double)c->nn; e_tot[j0 + j] = h[2 * j + 1] / (double)c->nn; }
    }
    return 0;
}

// e_m per material of a materials dielectric: the forward passes of pcb_field_energy's layout into the scratch, k_material_energy[_t]
// over the same fixed grid, the fixed-order sum of the [CTA][column][n_mat] partials.  Every check comes before any output.
int pcb_material_energy(pcb_op* o, int ncols, const void* const* x, int n_mat, double* e_mat) {
    PCB_CHECK_ARG(o && x && e_mat && ncols > 0, "bad arguments");
    pcb_ctx* c = o->ctx;
    PCB_CUDA_OK(cudaSetDevice(c->device));
    if (c->nloc != c->nn) {
        pcb_set_error("pcb_material_energy: needs whole columns; a slab context only supports PCB_APPLY_P (gather with pcb_slab_exchange)");
        return -2;
    }
    if (!o->diel || o->d.diel != PCB_DIEL_MATERIALS) {
        pcb_set_error("pcb_material_energy: the operator has no materials dielectric (PCB_DIEL_KIND_MATERIALS)");
        return -1;
    }
    if (n_mat != o->diel->n_mat) { pcb_set_error("pcb_material_energy: n_mat = %d, the dielectric has %d materials", n_mat, o->diel->n_mat); return -1; }
    PCB_CHECK_ARG(o->diel->zsplit == c->zsplit, "dielectric was created under the other plane-mode form (plane_split); re-create it");
    const bool plane = plane_layout(c);
    const int gx = grid_for(c, c->nn, 256, 4);      // fixed for the context: the same partials for a column at any width
    const int kmax = ncols < PCB_MAXC ? ncols : PCB_MAXC;
    const size_t E = (size_t)PCB_MAXC * (size_t)n_mat;
    if (ensure_partial(c, sizeof(double) * ((size_t)gx + 1) * E)) return -1;
    if (ensure_scratch(c, sizeof(cplx) * (size_t)c->R * (size_t)kmax)) return -1;
    std::vector<double> h(E);
    double* dout = c->partial + (size_t)gx * E;
    for (int j0 = 0; j0 < ncols; j0 += PCB_MAXC) {
        const int kc = (ncols - j0 < PCB_MAXC) ? ncols - j0 : PCB_MAXC;
        PcbCols cols;
        memset(&cols, 0, sizeof cols);
        for (int j = 0; j < kc; ++j) cols.in[j] = (const cplx*)x[j0 + j];
        if (run_steps(o, forward_steps(plane), cols, kc)) return -1;
        PcbCols e;
        memset(&e, 0, sizeof e);
        for (int j = 0; j < kc; ++j) e.in[j] = c->scratch + (size_t)j * c->R;
        const int ne = kc * n_mat;
        dim3 grid((unsigned)gx, (unsigned)kc, 1), blk(256, 1, 1);
        const bool reg = n_mat <= PCB_ME_REG;      // bins in registers, else the match path
        if (plane && reg) PCB_LAUNCH(k_material_energy_t<PCB_ME_REG>, grid, blk, 0, c->stream, o->d, e, kc, n_mat, c->partial);
        else if (plane) PCB_LAUNCH(k_material_energy_t<0>, grid, blk, 0, c->stream, o->d, e, kc, n_mat, c->partial);
        else if (reg) PCB_LAUNCH(k_material_energy<PCB_ME_REG>, grid, blk, 0, c->stream, o->d, e, kc, n_mat, c->partial);
        else PCB_LAUNCH(k_material_energy<0>, grid, blk, 0, c->stream, o->d, e, kc, n_mat, c->partial);
        PCB_CUDA_OK(cudaGetLastError());
        PCB_LAUNCH(k_sum_partials, dim3((unsigned)((ne + 63) / 64), 1, 1), dim3(64, 1, 1), 0, c->stream, (const double*)c->partial, gx, ne, dout);
        PCB_CUDA_OK(cudaGetLastError());
        c->launches += 2;
        PCB_CUDA_OK(cudaMemcpyAsync(h.data(), dout, sizeof(double) * (size_t)ne, cudaMemcpyDeviceToHost, c->stream));
        PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
        for (int i = 0; i < ne; ++i) e_mat[(size_t)j0 * n_mat + i] = h[i] / (double)c->nn;
    }
    return 0;
}

// ---- band velocity matrices (Hellmann-Feynman) ---------------------------------------------------------------------
// E^ = PCB_APPLY_EFOURIER of the ncols columns into the context's bv_buf (behind the tau tables), k_band_velocity over a grid
// fixed by the context, the fixed-order sum of its partials; V_d = W_d + W_d^H is formed on the host.
int pcb_band_velocity(pcb_op* o, int ncols, const void* const* x, const double* dtables, void* V, double* xx, double* xax) {
    PCB_CHECK_ARG(o && x && dtables && V && xx && xax && ncols > 0, "bad arguments");
    PCB_CHECK_ARG(ncols <= PCB_MAXC, "ncols > 32: call per block of at most 32 columns");
    pcb_ctx* c = o->ctx;
    PCB_CUDA_OK(cudaSetDevice(c->device));
    if (c->nloc != c->nn) {
        pcb_set_error("pcb_band_velocity: needs whole columns; a slab context only supports PCB_APPLY_P (gather with pcb_slab_exchange)");
        return -2;
    }
    PCB_CHECK_ARG(!o->diel || o->diel->zsplit == c->zsplit, "dielectric was created under the other plane-mode form (plane_split); re-create it");
    const int N = c->N;
    const size_t need = sizeof(cplx) * (3 * (size_t)N + (size_t)c->R * (size_t)ncols);      // grows with the widest call so far
    if (c->bv_bytes < need) {
        if (c->bv_buf) { PCB_CUDA_OK(cudaStreamSynchronize(c->stream)); PCB_CUDA_OK(cudaFree(c->bv_buf)); c->bv_buf = nullptr; c->bv_bytes = 0; }
        PCB_CUDA_OK(cudaMalloc(&c->bv_buf, need));
        c->bv_bytes = need;
    }
    cplx* tau = c->bv_buf;
    cplx* ehat = c->bv_buf + 3 * (size_t)N;
    const long long nchunks = (c->nn + PCB_BV_P - 1) / PCB_BV_P;
    const int gx = (int)(nchunks < 2LL * c->sms ? nchunks : 2LL * c->sms);      // fixed for the context: the same partials at any width
    const int nb = (ncols + PCB_BV_B - 1) / PCB_BV_B;
    const long long E = 6LL * ncols * ncols + 2LL * ncols;
    if (ensure_partial(c, sizeof(double) * ((size_t)gx + 1) * (size_t)E)) return -1;
    double* dout = c->partial + (size_t)gx * (size_t)E;
    PCB_CUDA_OK(cudaMemcpyAsync(tau, dtables, sizeof(cplx) * 3 * (size_t)N, cudaMemcpyHostToDevice, c->stream));
    PcbCols cols;
    memset(&cols, 0, sizeof cols);
    for (int j = 0; j < ncols; ++j) { cols.in[j] = (const cplx*)x[j]; cols.out[j] = ehat + (size_t)j * c->R; }
    if (int rc = apply_AH(o, PCB_APPLY_EFOURIER, cols, ncols, 0, 0)) return rc;
    PcbCols bv;
    memset(&bv, 0, sizeof bv);
    for (int j = 0; j < ncols; ++j) { bv.in[j] = cols.in[j]; bv.out[j] = cols.out[j]; }
    if (PCB_BV_SMEM > 48 * 1024) PCB_CUDA_OK(cudaFuncSetAttribute(k_band_velocity, cudaFuncAttributeMaxDynamicSharedMemorySize, PCB_BV_SMEM));
    PCB_LAUNCH(k_band_velocity, dim3((unsigned)gx, (unsigned)(nb * nb), 1), dim3(PCB_BV_NT, 1, 1), (size_t)PCB_BV_SMEM, c->stream,
               o->d, bv, (const cplx*)tau, ncols, nb, c->partial);
    PCB_CUDA_OK(cudaGetLastError());
    PCB_LAUNCH(k_sum_partials, dim3((unsigned)((E + 63) / 64), 1, 1), dim3(64, 1, 1), 0, c->stream, (const double*)c->partial, gx, (int)E, dout);
    PCB_CUDA_OK(cudaGetLastError());
    c->launches += 2;
    std::vector<double> h((size_t)E);
    PCB_CUDA_OK(cudaMemcpyAsync(h.data(), dout, sizeof(double) * (size_t)E, cudaMemcpyDeviceToHost, c->stream));
    PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
    double* v = (double*)V;
    const size_t n = (size_t)ncols;
    for (size_t d = 0; d < 3; ++d)
        for (size_t i = 0; i < n; ++i)
            for (size_t j = 0; j < n; ++j) {
                const double* wij = &h[2 * ((d * n + i) * n + j)];
                const double* wji = &h[2 * ((d * n + j) * n + i)];
                v[2 * ((d * n + i) * n + j)] = wij[0] + wji[0];          // V = W + W^H
                v[2 * ((d * n + i) * n + j) + 1] = wij[1] - wji[1];
            }
    for (size_t j = 0; j < n; ++j) { xx[j] = h[6 * n * n + j]; xax[j] = h[6 * n * n + n + j]; }
    return 0;
}

// Host-buffer apply (the reference-facing call with NumPy arrays): Y_host = op(X_host) for row-major (R, k) host blocks.
// The block travels in chunks of PCB_HOST_CH columns (2-D copies of 128-byte rows run at full PCIe speed) through a
// three-stream pipeline -- H2D of chunk c+1, transpose + apply + transpose of chunk c, D2H of chunk c-1 overlap -- so both PCIe
// directions are busy at once; with pinned host memory a 16-column block at N = 120 takes ~3 instead of 4 chunk-copy times.
static int apply_host_pipeline(pcb_op* o, int mode, int k, const void* x_host, long long ldx, void* y_host, long long ldy);
int pcb_apply_host(pcb_op* o, int mode, int k, const void* x_host, long long ldx, void* y_host, long long ldy) {
    PCB_CHECK_ARG(o && x_host && y_host && k > 0 && ldx >= k && ldy >= k, "bad arguments");
    pcb_ctx* c = o->ctx;
    PCB_CUDA_OK(cudaSetDevice(c->device));
    if (!c->s_h2d) {
        PCB_CUDA_OK(cudaStreamCreateWithFlags(&c->s_h2d, cudaStreamNonBlocking));
        PCB_CUDA_OK(cudaStreamCreateWithFlags(&c->s_d2h, cudaStreamNonBlocking));
        for (int a = 0; a < 2; ++a) for (int b = 0; b < 4; ++b) PCB_CUDA_OK(cudaEventCreateWithFlags(&c->hp_ev[a][b], cudaEventDisableTiming));
    }
    // staging: 2 slots x 4 regions of R x min(k, CH) elements (a single-vector call takes 1/8 of the block-call size)
    static const char* ev_ch = getenv("PCB200_HOST_CH");      // columns per pipeline chunk (default 8 = 128-byte rows of the 2-D copies)
    int chmax = ev_ch ? atoi(ev_ch) : PCB_HOST_CH;
    if (chmax < 1 || chmax > PCB_HOST_CH) chmax = PCB_HOST_CH;
    const int chw = k < chmax ? k : chmax;
    if (chw != c->hp_cols) {
        if (c->hp_buf) { PCB_CUDA_OK(cudaStreamSynchronize(c->stream)); PCB_CUDA_OK(cudaFree(c->hp_buf)); c->hp_buf = nullptr; c->hp_cols = 0; }
        PCB_CUDA_OK(cudaMalloc(&c->hp_buf, sizeof(cplx) * (size_t)c->R * (size_t)chw * 8));
        c->hp_cols = chw;
    }
    const int rc = apply_host_pipeline(o, mode, k, x_host, ldx, y_host, ldy);
    if (rc != 0) {      // no copy may still target the caller's buffers when an error is reported
        cudaStreamSynchronize(c->s_h2d); cudaStreamSynchronize(c->stream); cudaStreamSynchronize(c->s_d2h);
        (void)cudaGetLastError();
    }
    return rc;
}
static int apply_host_pipeline(pcb_op* o, int mode, int k, const void* x_host, long long ldx, void* y_host, long long ldy) {
    pcb_ctx* c = o->ctx;
    const size_t R = (size_t)c->R, CH = (size_t)c->hp_cols;
    PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
    enum { EV_H2D = 0, EV_INFREE = 1, EV_CMP = 2, EV_OUTFREE = 3 };
    const int nchunks = (int)((k + CH - 1) / CH);
    for (int ch = 0; ch < nchunks; ++ch) {
        const int slot = ch & 1;
        const int j0 = ch * (int)CH, kc = (k - j0 < (int)CH) ? k - j0 : (int)CH;
        cplx* st_in = c->hp_buf + (size_t)(slot * 4 + 0) * R * CH;
        cplx* st_out = c->hp_buf + (size_t)(slot * 4 + 1) * R * CH;
        cplx* col_in = c->hp_buf + (size_t)(slot * 4 + 2) * R * CH;
        cplx* col_out = c->hp_buf + (size_t)(slot * 4 + 3) * R * CH;
        // H2D (waits until the staging slot has been consumed by the transpose of chunk ch-2)
        if (ch >= 2) PCB_CUDA_OK(cudaStreamWaitEvent(c->s_h2d, c->hp_ev[slot][EV_INFREE], 0));
        PCB_CUDA_OK(cudaMemcpy2DAsync(st_in, sizeof(cplx) * kc, (const cplx*)x_host + j0, sizeof(cplx) * ldx, sizeof(cplx) * kc, R,
                                      cudaMemcpyHostToDevice, c->s_h2d));
        PCB_CUDA_OK(cudaEventRecord(c->hp_ev[slot][EV_H2D], c->s_h2d));
        // compute stream: transpose in, apply, transpose out
        PCB_CUDA_OK(cudaStreamWaitEvent(c->stream, c->hp_ev[slot][EV_H2D], 0));
        void* pin[PCB_HOST_CH]; void* pout[PCB_HOST_CH];
        for (int j = 0; j < kc; ++j) { pin[j] = col_in + (size_t)j * R; pout[j] = col_out + (size_t)j * R; }
        if (transpose_cols(c, st_in, kc, kc, pin, true)) return -1;
        PCB_CUDA_OK(cudaEventRecord(c->hp_ev[slot][EV_INFREE], c->stream));
        if (ch >= 2) PCB_CUDA_OK(cudaStreamWaitEvent(c->stream, c->hp_ev[slot][EV_OUTFREE], 0));
        if (int rc = pcb_apply(o, mode, kc, pin, pout)) return rc;
        if (transpose_cols(c, st_out, kc, kc, pout, false)) return -1;
        PCB_CUDA_OK(cudaEventRecord(c->hp_ev[slot][EV_CMP], c->stream));
        // D2H
        PCB_CUDA_OK(cudaStreamWaitEvent(c->s_d2h, c->hp_ev[slot][EV_CMP], 0));
        PCB_CUDA_OK(cudaMemcpy2DAsync((cplx*)y_host + j0, sizeof(cplx) * ldy, st_out, sizeof(cplx) * kc, sizeof(cplx) * kc, R,
                                      cudaMemcpyDeviceToHost, c->s_d2h));
        PCB_CUDA_OK(cudaEventRecord(c->hp_ev[slot][EV_OUTFREE], c->s_d2h));
    }
    PCB_CUDA_OK(cudaStreamSynchronize(c->s_d2h));
    PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
    return 0;
}

// ---- block kernels ----------------------------------------------------------------------------------------------
int pcb_residual(pcb_op* o, int precond, int ncols, const void* const* x, const void* const* hx, void* const* w,
                 const double* lambda, double* norms2) {
    PCB_CHECK_ARG(o && x && hx && w && lambda && norms2 && ncols > 0 && precond >= 0 && precond <= 3, "bad arguments");
    pcb_ctx* c = o->ctx;
    PCB_CUDA_OK(cudaSetDevice(c->device));
    const int gx = grid_for(c, c->nloc, 256, 4);
    if (ensure_partial(c, sizeof(double) * (size_t)gx * PCB_MAXC_RP + sizeof(double) * PCB_MAXC_RP)) return -1;
    if (ensure_hstage(c, 65536)) return -1;
    for (int j0 = 0; j0 < ncols; j0 += PCB_MAXC_RP) {
        const int kc = (ncols - j0 < PCB_MAXC_RP) ? ncols - j0 : PCB_MAXC_RP;
        PcbResidArgs a;
        for (int j = 0; j < kc; ++j) {
            a.x[j] = (const cplx*)x[j0 + j]; a.hx[j] = (const cplx*)hx[j0 + j]; a.w[j] = (cplx*)w[j0 + j]; a.lambda[j] = lambda[j0 + j];
        }
        dim3 grid((unsigned)gx, (unsigned)((kc + PCB_RP_CH - 1) / PCB_RP_CH), 1);
        if (precond == 1) PCB_LAUNCH(k_resid_precond<1>, grid, dim3(256, 1, 1), 0, c->stream, o->d, a, kc, c->partial);
        else if (precond == 2) PCB_LAUNCH((k_resid_precond<1, true>), grid, dim3(256, 1, 1), 0, c->stream, o->d, a, kc, c->partial);
        else if (precond == 3) PCB_LAUNCH((k_resid_precond<0, true>), grid, dim3(256, 1, 1), 0, c->stream, o->d, a, kc, c->partial);
        else PCB_LAUNCH(k_resid_precond<0>, grid, dim3(256, 1, 1), 0, c->stream, o->d, a, kc, c->partial);
        PCB_CUDA_OK(cudaGetLastError());
        double* dout = c->partial + (size_t)gx * PCB_MAXC_RP;
        PCB_LAUNCH(k_sum_partials, dim3(1, 1, 1), dim3(64, 1, 1), 0, c->stream, (const double*)c->partial, gx, kc, dout);
        PCB_CUDA_OK(cudaGetLastError());
        c->launches += 2;
        if (comm_allreduce(c, dout, kc)) return -1;
        PCB_CUDA_OK(cudaMemcpyAsync(c->hstage, dout, sizeof(double) * kc, cudaMemcpyDeviceToHost, c->stream));
        PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
        memcpy(norms2 + j0, c->hstage, sizeof(double) * kc);
    }
    return 0;
}

int pcb_gram2(pcb_ctx* c, int n, const void* const* s, const void* const* hs, void* G, void* T) {
    return pcb_gram2_top(c, n, n, s, hs, G, T);
}
int pcb_gram2_top(pcb_ctx* c, int n, int ntop, const void* const* s, const void* const* hs, void* G, void* T) {
    PCB_CHECK_ARG(c && s && hs && G && T && n > 0 && n <= PCB_MAXL && ntop > 0 && ntop <= n, "bad arguments (n <= 96, 0 < ntop <= n)");
    PCB_CUDA_OK(cudaSetDevice(c->device));
    const int nt = (n + 7) / 8, nc = 8 * nt;
    const int ttop = (ntop + 7) / 8;                       // leading tile rows to accumulate
    PcbColList S, HS;
    for (int j = 0; j < PCB_MAXL; ++j) { S.p[j] = (j < n) ? (const cplx*)s[j] : nullptr; HS.p[j] = (j < n) ? (const cplx*)hs[j] : nullptr; }
    const int npairs = ttop * nt - ttop * (ttop - 1) / 2;  // pairs (ta < ttop, tb >= ta) = a prefix of the row-major upper triangle
    const bool tside = ttop < nt;                          // leading rows only: T = (HS_top)^H S, the other HS columns are not read
    const size_t smem = sizeof(cplx) * 4 * (size_t)nc * PCB_GM_LD;
    const long long ntiles = (c->R + PCB_GM_TR - 1) / PCB_GM_TR;
    // One launch covers at most PCB_GM_MAXW * PCB_GM_PPW tile pairs (n <= 64); wider blocks take several launches over equal
    // shares of the pair list, all writing disjoint entries of the same per-CTA partial matrices (the kernel is DMMA-bound, so
    // re-reading the columns costs little).  Warps per CTA: every warp gets the same number of pairs where possible (all warps
    // meet at one barrier per row tile, the slowest one sets the pace), as many warps as that allows.
    const int cap = PCB_GM_MAXW * PCB_GM_PPW;
    const int nlaunch = (npairs + cap - 1) / cap, share = (npairs + nlaunch - 1) / nlaunch;
    long long gx = 0;
    for (int l = 0; l < nlaunch; ++l) {
        const int pair0 = l * share, np = (npairs - pair0 < share) ? npairs - pair0 : share;
        int W = 0;
        for (int ppw = 1; ppw <= PCB_GM_PPW && W == 0; ++ppw) {
            const int w = (np + ppw - 1) / ppw;                 // fewest warps with <= ppw pairs each
            if (w <= PCB_GM_MAXW && ((w * ppw - np) * 8 <= np || ppw == PCB_GM_PPW)) W = w;   // <= 12.5 % idle pair slots
        }
        if (W < 4) W = 4;
        { static const char* ev = getenv("PCB200_GRAM_W"); if (ev && atoi(ev) >= 4 && atoi(ev) <= PCB_GM_MAXW && (np + atoi(ev) - 1) / atoi(ev) <= PCB_GM_PPW) W = atoi(ev); }
        const int ppw = (np + W - 1) / W;
        void (*kern)(PcbColList, PcbColList, int, int, int, int, int, long long, cplx*) =
            W <= 12 ? (tside ? (ppw <= 1 ? k_gram2<1, true, 12> : k_gram2<2, true, 12>) : (ppw <= 1 ? k_gram2<1, false, 12> : k_gram2<2, false, 12>))
                    : (tside ? (ppw <= 1 ? k_gram2<1, true, PCB_GM_MAXW> : k_gram2<2, true, PCB_GM_MAXW>)
                             : (ppw <= 1 ? k_gram2<1, false, PCB_GM_MAXW> : k_gram2<2, false, PCB_GM_MAXW>));
        if (l == 0) {
            int per_sm = (int)((size_t)224 * 1024 / (smem + 1024)); if (per_sm < 1) per_sm = 1;
            const int by_threads = 2048 / (32 * W); if (per_sm > by_threads) per_sm = by_threads;
            if (per_sm > 4) per_sm = 4;
#ifndef PCB_EMU
            if (smem > 48 * 1024) PCB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            PCB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
            { int occ = 0; PCB_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, 32 * W, smem)); if (occ >= 1 && occ < per_sm) per_sm = occ; }
#endif
            gx = (long long)c->sms * per_sm; if (gx > ntiles) gx = ntiles;
            if (ensure_partial(c, sizeof(cplx) * (size_t)gx * 2 * nc * nc)) return -1;
            if (ensure_dsmall(c, sizeof(cplx) * 2 * PCB_MAXL * PCB_MAXL + 65536)) return -1;
            if (ensure_hstage(c, sizeof(cplx) * 2 * PCB_MAXL * PCB_MAXL + 65536)) return -1;
        }
#ifndef PCB_EMU
        else {
            if (smem > 48 * 1024) PCB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            PCB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
        }
#endif
        PCB_LAUNCH(kern, dim3((unsigned)gx, 1, 1), dim3(32 * W, 1, 1), smem, c->stream, S, HS, n, 8 * ttop, nt, pair0, np, c->R, (cplx*)c->partial);
        PCB_CUDA_OK(cudaGetLastError());
        c->launches++;
    }
    note_block(c, "k_gram2", gx, ntiles);
    cplx* dout = (cplx*)c->dsmall;
    const int ne = 2 * nc * nc;
    PCB_LAUNCH(k_gram_finish, dim3((unsigned)((ne + 127) / 128), 1, 1), dim3(128, 1, 1), 0, c->stream, (const cplx*)c->partial, (int)gx, nt, ttop, dout);
    PCB_CUDA_OK(cudaGetLastError());
    c->launches += 1;
    if (comm_allreduce(c, (double*)dout, 2LL * ne)) return -1;      // large-grid mode: sum of the per-slab Gram pairs (NCCL)
    PCB_CUDA_OK(cudaMemcpyAsync(c->hstage, dout, sizeof(cplx) * ne, cudaMemcpyDeviceToHost, c->stream));
    PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
    const cplx* h = (const cplx*)c->hstage;
    cplx* g = (cplx*)G; cplx* t = (cplx*)T;
    // hermitize on the host (hermitize(), orthogonalization.py:26-33): (M + M^H)/2
    for (int a = 0; a < n; ++a)
        for (int b = 0; b < n; ++b) {
            const cplx gab = h[a * nc + b], gba = h[b * nc + a];
            const cplx tab = h[nc * nc + a * nc + b], tba = h[nc * nc + b * nc + a];
            g[a * n + b] = cmake(0.5 * (gab.x + gba.x), 0.5 * (gab.y - gba.y));
            t[a * n + b] = cmake(0.5 * (tab.x + tba.x), 0.5 * (tab.y - tba.y));
        }
    return 0;
}

static int update_impl(pcb_ctx* c, pcb_op* o, int m, int nl, void* const* s, void* const* hs, void* const* p_out, void* const* hp_out, const void* E,
                       const double* lambda, void* const* w_out, double* norms2);
int pcb_update(pcb_ctx* c, int m, int nl, void* const* s, void* const* hs, void* const* p_out, void* const* hp_out, const void* E) {
    return update_impl(c, nullptr, m, nl, s, hs, p_out, hp_out, E, nullptr, nullptr, nullptr);
}
/* pcb_update followed by pcb_residual(precond = 1) on the new X, HX with the new Ritz values `lambda`: w_out_j = K_P^-1 (lambda_j x_j - hx_j),
 * norms2[j] = ||lambda_j x_j - hx_j||^2 (HOST).  For m <= 16 one kernel does both (k_update_res: the residual is formed from the
 * accumulator fragments, X and HX are not re-read); wider blocks run the two kernels back to back. */
int pcb_update_resid(pcb_op* o, int m, int nl, void* const* s, void* const* hs, void* const* p_out, void* const* hp_out, const void* E,
                     const double* lambda, void* const* w_out, double* norms2) {
    PCB_CHECK_ARG(o && lambda && w_out && norms2, "bad arguments");
    return update_impl(o->ctx, o, m, nl, s, hs, p_out, hp_out, E, lambda, w_out, norms2);
}
static int update_impl(pcb_ctx* c, pcb_op* o, int m, int nl, void* const* s, void* const* hs, void* const* p_out, void* const* hp_out, const void* E,
                       const double* lambda, void* const* w_out, double* norms2) {
    PCB_CHECK_ARG(c && s && hs && p_out && hp_out && E && m > 0 && nl >= m && nl <= PCB_MAXL && m <= 32, "bad arguments");
    PCB_CUDA_OK(cudaSetDevice(c->device));
    const int MP = 8 * ((m + 7) / 8), MPp = MP + 2, JT = MP / 4;       // output columns padded to 8; E' row stride (conflict-free)
    const int kx = (m + 1) & ~1, kp = (nl - m + 1) & ~1, nlp = kx + kp; // even column counts: a k-step covers two columns
    PCB_CHECK_ARG(nlp <= PCB_MAXL + 2, "too many columns");
    if (ensure_hstage(c, sizeof(cplx) * 2 * PCB_MAXL * PCB_MAXL + 65536)) return -1;
    if (ensure_dsmall(c, sizeof(cplx) * 2 * PCB_MAXL * PCB_MAXL + 65536)) return -1;
    PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
    cplx* he = (cplx*)c->hstage;
    const cplx* e = (const cplx*)E;
    PcbColList Sin, HSin;
    PcbColListW X, HX, P, HP;
    for (int k = 0; k < PCB_MAXL; ++k) {
        Sin.p[k] = nullptr; HSin.p[k] = nullptr;
        X.p[k] = (k < m) ? (cplx*)s[k] : nullptr; HX.p[k] = (k < m) ? (cplx*)hs[k] : nullptr;
        P.p[k] = (k < m) ? (cplx*)p_out[k] : nullptr; HP.p[k] = (k < m) ? (cplx*)hp_out[k] : nullptr;
    }
    for (int k = 0; k < nlp; ++k) {
        const int src = (k < kx) ? (k < m ? k : -1) : (k - kx + m < nl ? k - kx + m : -1);   // input column or zero padding
        if (k < PCB_MAXL) { Sin.p[k] = src >= 0 ? (const cplx*)s[src] : nullptr; HSin.p[k] = src >= 0 ? (const cplx*)hs[src] : nullptr; }
        else if (src >= 0) { pcb_set_error("pcb_update: column list overflow"); return -2; }
        for (int j = 0; j < MPp; ++j) he[k * MPp + j] = (src >= 0 && j < m) ? e[src * m + j] : cmake(0.0, 0.0);
    }
    PCB_CUDA_OK(cudaMemcpyAsync(c->dsmall, he, sizeof(cplx) * nlp * MPp, cudaMemcpyHostToDevice, c->stream));
    const cplx* dE = (const cplx*)c->dsmall;
    // rows per tile: 32 when the double-buffered stage fits in shared memory, else 16
    const size_t smem32 = sizeof(cplx) * (2 * (size_t)nlp * MPp + 4 * (size_t)nlp * PcbUpd<32>::LD);
    const size_t smem16 = sizeof(cplx) * (2 * (size_t)nlp * MPp + 4 * (size_t)nlp * PcbUpd<16>::LD);
    const size_t smem48 = sizeof(cplx) * (2 * (size_t)nlp * MPp + 4 * (size_t)nlp * PcbUpd<48>::LD);
    const bool big = smem32 <= (size_t)224 * 1024;
    // 48-row tiles with 24 warps (6 row tiles x 4 column tiles) when they fit: more thin warps overlap the stage barriers better
    static const char* ev_tr = getenv("PCB200_UPD_TR");
    const bool wide = JT == 4 && smem48 <= (size_t)224 * 1024 && !(ev_tr && atoi(ev_tr) == 32);
    static const char* ev_nst = getenv("PCB200_UPD_NST");
    const size_t smem32x3 = sizeof(cplx) * (2 * (size_t)nlp * MPp + 6 * (size_t)nlp * PcbUpd<32>::LD);
    // m = 16: three 32-row stages with one barrier per tile (2.71 ms at n_loc = 48; 48-row tiles x 24 warps 2.76, two stages 2.77)
    const bool deep = !(ev_nst && atoi(ev_nst) == 2) && JT == 4 && smem32x3 <= (size_t)224 * 1024;
    const int TR = deep ? 32 : wide ? 48 : big ? 32 : 16;
    const size_t smem = deep ? smem32x3 : wide ? smem48 : big ? smem32 : smem16;
    const int JW = (deep || wide || (TR / 8) * JT <= 16) ? 1 : 2;  // one column tile per warp while that keeps <= 16 warps per CTA
    const int warps = (TR / 8) * (JT / JW);
    const long long ntiles = (c->R + TR - 1) / TR;
    if (o) {
        // fused form: 3 components x 16 cells per tile, 24 warps, two stages + 12 KB for the raw residual of the tile
        const size_t smem_f = smem48 + sizeof(cplx) * 2 * 48 * 17;
        static const char* ev_f = getenv("PCB200_FUSED_RESID");
        if (JT == 4 && m <= 16 && smem_f <= (size_t)226 * 1024 && !(ev_f && ev_f[0] == '0')) {
            PcbUpdRes rs;
            for (int j = 0; j < 16; ++j) { rs.w[j] = j < m ? (cplx*)w_out[j] : nullptr; rs.lambda[j] = j < m ? lambda[j] : 0.0; }
            const long long nt = (c->nloc + 15) / 16;
            long long gxf = c->sms; if (gxf > nt) gxf = nt;
            if (ensure_partial(c, sizeof(double) * ((size_t)gxf * 16 + 16))) return -1;
#ifndef PCB_EMU
            if (smem_f > 48 * 1024) PCB_CUDA_OK(cudaFuncSetAttribute(k_update_res, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_f));
#endif
            note_block(c, "k_update_res", gxf, nt);
            PCB_LAUNCH(k_update_res, dim3((unsigned)gxf, 1, 1), dim3(PCB_UPDRES_THREADS, 1, 1), smem_f, c->stream, o->d, Sin, HSin, X, HX, P, HP, rs, dE, m, kx, kp, MPp, c->partial);
            PCB_CUDA_OK(cudaGetLastError());
            double* dout = c->partial + (size_t)gxf * 16;
            PCB_LAUNCH(k_sum_partials, dim3(1, 1, 1), dim3(64, 1, 1), 0, c->stream, (const double*)c->partial, (int)gxf, 16, dout);
            PCB_CUDA_OK(cudaGetLastError());
            c->launches += 2;
            if (comm_allreduce(c, dout, m)) return -1;
            char* hn = (char*)c->hstage + sizeof(cplx) * 2 * PCB_MAXL * PCB_MAXL;      // behind the E staging area
            PCB_CUDA_OK(cudaMemcpyAsync(hn, dout, sizeof(double) * m, cudaMemcpyDeviceToHost, c->stream));
            if (!norms2) { c->pending_state = 1; c->pending_m = m; return 0; }      // pcb_update_resid_start: fetched by _wait
            PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
            memcpy(norms2, hn, sizeof(double) * m);
            return 0;
        }
    }
    int per_sm = (int)((size_t)224 * 1024 / (smem + 1024)); if (per_sm < 1) per_sm = 1; if (per_sm > 4) per_sm = 4;
    long long gx = (long long)c->sms * per_sm; if (gx > ntiles) gx = ntiles;
    dim3 grid((unsigned)gx, 1, 1), block((unsigned)(32 * warps), 1, 1);
#ifndef PCB_EMU
#define PCB_UPD_GO(K)                                                                                              \
    do {                                                                                                           \
        if (smem > 48 * 1024) PCB_CUDA_OK(cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        PCB_LAUNCH(K, grid, block, smem, c->stream, Sin, HSin, X, HX, P, HP, dE, m, kx, kp, MPp, c->R);            \
    } while (0)
#else
#define PCB_UPD_GO(K) PCB_LAUNCH(K, grid, block, smem, c->stream, Sin, HSin, X, HX, P, HP, dE, m, kx, kp, MPp, c->R)
#endif
    if (deep) { PCB_UPD_GO((k_update<32, 1, 3>)); note_block(c, "k_update<32,1,3>", gx, ntiles); }
    else if (wide) { PCB_UPD_GO((k_update<48, 1>)); note_block(c, "k_update<48,1>", gx, ntiles); }
    else if (big && JW == 1) { PCB_UPD_GO((k_update<32, 1>)); note_block(c, "k_update<32,1>", gx, ntiles); }
    else if (big) { PCB_UPD_GO((k_update<32, 2>)); note_block(c, "k_update<32,2>", gx, ntiles); }
    else if (JW == 1) { PCB_UPD_GO((k_update<16, 1>)); note_block(c, "k_update<16,1>", gx, ntiles); }
    else { PCB_UPD_GO((k_update<16, 2>)); note_block(c, "k_update<16,2>", gx, ntiles); }
    PCB_CUDA_OK(cudaGetLastError());
    c->launches++;
    if (o) {      // wide blocks: two kernels
        double* dst = norms2 ? norms2 : c->pending_norms;
        const int rc = pcb_residual(o, 1, m, (const void* const*)s, (const void* const*)hs, w_out, lambda, dst);
        if (!norms2 && rc == 0) { c->pending_state = 2; c->pending_m = m; }
        return rc;
    }
    return 0;
}
/* pcb_update_resid in two halves: _start enqueues everything and returns while the GPU works (the caller's host-side
 * bookkeeping -- the rotated Gram blocks of the incremental Gram pair -- overlaps the kernel), _wait returns the norms. */
int pcb_update_resid_start(pcb_op* o, int m, int nl, void* const* s, void* const* hs, void* const* p_out, void* const* hp_out, const void* E,
                           const double* lambda, void* const* w_out) {
    PCB_CHECK_ARG(o && lambda && w_out, "bad arguments");
    o->ctx->pending_state = 0;
    return update_impl(o->ctx, o, m, nl, s, hs, p_out, hp_out, E, lambda, w_out, nullptr);
}
int pcb_update_resid_wait(pcb_op* o, int m, double* norms2) {
    PCB_CHECK_ARG(o && norms2 && o->ctx->pending_state != 0 && o->ctx->pending_m == m, "no pending pcb_update_resid_start of this width");
    pcb_ctx* c = o->ctx;
    if (c->pending_state == 1) {
        PCB_CUDA_OK(cudaSetDevice(c->device));
        PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
        memcpy(norms2, (char*)c->hstage + sizeof(cplx) * 2 * PCB_MAXL * PCB_MAXL, sizeof(double) * m);
    } else memcpy(norms2, c->pending_norms, sizeof(double) * m);
    c->pending_state = 0;
    return 0;
}

int pcb_block_launch_info(pcb_ctx* c, char* name, int cap, long long* grid, long long* tiles) {
    PCB_CHECK_ARG(c && name && cap > 0 && grid && tiles, "bad arguments");
    snprintf(name, (size_t)cap, "%s", c->blk_name);
    *grid = c->blk_grid; *tiles = c->blk_tiles;
    return 0;
}

int pcb_coldots(pcb_ctx* c, int ncols, const void* const* a, const void* const* b, void* out) {
    PCB_CHECK_ARG(c && a && b && out && ncols > 0 && ncols <= PCB_MAXL, "bad arguments");
    PCB_CUDA_OK(cudaSetDevice(c->device));
    const int gx = grid_for(c, c->R, 256, 4);
    if (ensure_partial(c, sizeof(cplx) * ((size_t)gx + 1) * PCB_MAXL)) return -1;
    if (ensure_hstage(c, 65536)) return -1;
    PcbColList A, B;
    for (int j = 0; j < PCB_MAXL; ++j) { A.p[j] = (j < ncols) ? (const cplx*)a[j] : nullptr; B.p[j] = (j < ncols) ? (const cplx*)b[j] : nullptr; }
    dim3 grid((unsigned)gx, (unsigned)ncols, 1);
    PCB_LAUNCH(k_coldots, grid, dim3(256, 1, 1), 0, c->stream, A, B, ncols, c->R, (cplx*)c->partial);
    PCB_CUDA_OK(cudaGetLastError());
    double* dout = c->partial + 2 * (size_t)gx * PCB_MAXL;
    PCB_LAUNCH(k_sum_partials, dim3((unsigned)((2 * ncols + 63) / 64), 1, 1), dim3(64, 1, 1), 0, c->stream, (const double*)c->partial, gx, 2 * ncols, dout);
    PCB_CUDA_OK(cudaGetLastError());
    c->launches += 2;
    if (comm_allreduce(c, dout, 2LL * ncols)) return -1;
    PCB_CUDA_OK(cudaMemcpyAsync(c->hstage, dout, sizeof(cplx) * ncols, cudaMemcpyDeviceToHost, c->stream));
    PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
    memcpy(out, c->hstage, sizeof(cplx) * ncols);
    return 0;
}

int pcb_axpby(pcb_ctx* c, int ncols, const void* const* x, void* const* y, double alpha, double beta) {
    PCB_CHECK_ARG(c && x && y && ncols > 0, "bad arguments");
    PCB_CUDA_OK(cudaSetDevice(c->device));
    for (int j = 0; j < ncols; ++j) {
        dim3 grid((unsigned)grid_for(c, c->R, 256, 8), 1, 1);
        PCB_LAUNCH(k_axpby, grid, dim3(256, 1, 1), 0, c->stream, (const cplx*)x[j], (cplx*)y[j], alpha, beta, c->R);
        PCB_CUDA_OK(cudaGetLastError());
        c->launches++;
    }
    return 0;
}


// ---- large-grid mode: communicator and slab <-> full-column exchange -------------------------------------------------
#ifndef PCB_EMU
static int nccl_load() {
    if (g_nccl.lib) return 0;
    // Order: PCB200_NCCL_LIB (explicit path), a copy the process has already mapped (e.g. torch's bundled NCCL: RTLD_NOLOAD, so
    // that two different NCCL builds never coexist), then the default search path.  RTLD_LOCAL: nothing else resolves against it.
    const char* names[] = {"libnccl.so.2", "libnccl.so", nullptr};
    if (const char* ev = getenv("PCB200_NCCL_LIB")) {
        g_nccl.lib = dlopen(ev, RTLD_NOW | RTLD_LOCAL);
        if (!g_nccl.lib) { pcb_set_error("cannot dlopen PCB200_NCCL_LIB=%s: %s", ev, dlerror()); return -4; }
    }
    for (int i = 0; names[i] && !g_nccl.lib; ++i) g_nccl.lib = dlopen(names[i], RTLD_NOW | RTLD_LOCAL | RTLD_NOLOAD);
    for (int i = 0; names[i] && !g_nccl.lib; ++i) g_nccl.lib = dlopen(names[i], RTLD_NOW | RTLD_LOCAL);
    if (!g_nccl.lib) { pcb_set_error("cannot dlopen libnccl.so.2: %s", dlerror()); return -4; }
#define PCB_SYM(field, name)                                                        \
    *(void**)(&g_nccl.field) = dlsym(g_nccl.lib, name);                             \
    if (!g_nccl.field) { pcb_set_error("libnccl: missing symbol %s", name); return -4; }
    PCB_SYM(GetUniqueId, "ncclGetUniqueId") PCB_SYM(CommInitRank, "ncclCommInitRank") PCB_SYM(CommDestroy, "ncclCommDestroy")
    PCB_SYM(AllReduce, "ncclAllReduce") PCB_SYM(AllGather, "ncclAllGather") PCB_SYM(Send, "ncclSend") PCB_SYM(Recv, "ncclRecv")
    PCB_SYM(GroupStart, "ncclGroupStart") PCB_SYM(GroupEnd, "ncclGroupEnd") PCB_SYM(GetErrorString, "ncclGetErrorString")
#undef PCB_SYM
    return 0;
}
#endif

int pcb_comm_unique_id(void* id128) {
    PCB_CHECK_ARG(id128, "null");
    memset(id128, 0, 128);
#ifndef PCB_EMU
    if (nccl_load()) return -4;
    const int rc = g_nccl.GetUniqueId((PcbNcclId*)id128);
    if (rc != 0) { pcb_set_error("ncclGetUniqueId failed: %s", g_nccl.GetErrorString(rc)); return -4; }
#endif
    return 0;
}
int pcb_comm_init(pcb_ctx* c, const void* id128, int rank, int world) {
    PCB_CHECK_ARG(c && id128 && world >= 1 && rank >= 0 && rank < world, "bad arguments");
    if (c->comm) { pcb_set_error("pcb_comm_init: context already has a communicator"); return -2; }
    PcbComm* cm = new PcbComm;
    cm->rank = rank; cm->world = world;
#ifndef PCB_EMU
    PCB_CUDA_OK(cudaSetDevice(c->device));
    if (nccl_load()) { delete cm; return -4; }
    PcbNcclId id;
    memcpy(&id, id128, 128);
    const int rc = g_nccl.CommInitRank(&cm->nccl, world, id, rank);
    if (rc != 0) { pcb_set_error("ncclCommInitRank failed: %s", g_nccl.GetErrorString(rc)); delete cm; return -4; }
#endif
    c->comm = cm;
    return 0;
}
/* host-emulation build only (tests): collectives through host callbacks, e.g. torch.distributed gloo */
int pcb_comm_set_host_callbacks(pcb_ctx* c, void* allreduce_cb, void* p2p_cb) {
#ifdef PCB_EMU
    PCB_CHECK_ARG(c && c->comm, "call pcb_comm_init first");
    c->comm->allreduce_cb = (pcb_allreduce_cb)allreduce_cb;
    c->comm->p2p_cb = (pcb_p2p_cb)p2p_cb;
    return 0;
#else
    (void)c; (void)allreduce_cb; (void)p2p_cb;
    pcb_set_error("pcb_comm_set_host_callbacks exists in the host-emulation test build only; the CUDA build uses NCCL");
    return -2;
#endif
}
int pcb_comm_destroy(pcb_ctx* c) {
    if (!c || !c->comm) return 0;
#ifndef PCB_EMU
    PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
    if (c->comm->nccl) g_nccl.CommDestroy(c->comm->nccl);
#endif
    delete c->comm;
    c->comm = nullptr;
    return 0;
}

/* ---- large-grid mode over peer memory ------------------------------------------------------------------------------
 * pcb_comm_share: map one allocation of every rank into every rank (CUDA IPC; the handles travel by ncclAllGather).
 * dptr must be the base of a pcb_malloc allocation; peers[g] receives rank g's allocation as seen from this process
 * (peers[rank] = dptr).  Collective over the communicator. */
int pcb_comm_share(pcb_ctx* c, void* dptr, void** peers) {
    PCB_CHECK_ARG(c && c->comm && dptr && peers, "bad arguments / no communicator");
#ifdef PCB_EMU
    pcb_set_error("pcb_comm_share: peer memory needs the CUDA build (the host-emulation build uses the slab exchange)");
    return -2;
#else
    PcbComm* cm = c->comm;
    PCB_CHECK_ARG(cm->world <= PCB_MAXW, "at most 8 ranks");
    PCB_CUDA_OK(cudaSetDevice(c->device));
    cudaIpcMemHandle_t h;
    PCB_CUDA_OK(cudaIpcGetMemHandle(&h, dptr));
    const size_t hs = sizeof(cudaIpcMemHandle_t);
    if (ensure_dsmall(c, sizeof(cplx) * 2 * PCB_MAXL * PCB_MAXL + 65536)) return -1;
    if (ensure_hstage(c, sizeof(cplx) * 2 * PCB_MAXL * PCB_MAXL + 65536)) return -1;
    char* dall = (char*)c->dsmall;
    PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
    memcpy(c->hstage, &h, hs);
    PCB_CUDA_OK(cudaMemcpyAsync(dall + cm->rank * hs, c->hstage, hs, cudaMemcpyHostToDevice, c->stream));
    const int rc = g_nccl.AllGather(dall + cm->rank * hs, dall, hs, PCB_NCCL_UINT8, cm->nccl, c->stream);
    if (rc != 0) { pcb_set_error("ncclAllGather failed: %s", g_nccl.GetErrorString(rc)); return -4; }
    PCB_CUDA_OK(cudaMemcpyAsync(c->hstage, dall, hs * cm->world, cudaMemcpyDeviceToHost, c->stream));
    PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
    for (int g = 0; g < cm->world; ++g) {
        if (g == cm->rank) { peers[g] = dptr; continue; }
        cudaIpcMemHandle_t hg;
        memcpy(&hg, (char*)c->hstage + g * hs, hs);
        PCB_CUDA_OK(cudaIpcOpenMemHandle(&peers[g], hg, cudaIpcMemLazyEnablePeerAccess));
    }
    return 0;
#endif
}
int pcb_comm_unshare(pcb_ctx* c, void** peers) {
    PCB_CHECK_ARG(c && c->comm && peers, "bad arguments / no communicator");
#ifndef PCB_EMU
    PCB_CUDA_OK(cudaSetDevice(c->device));
    PCB_CUDA_OK(cudaStreamSynchronize(c->stream));
    for (int g = 0; g < c->comm->world; ++g)
        if (g != c->comm->rank && peers[g]) { PCB_CUDA_OK(cudaIpcCloseMemHandle(peers[g])); peers[g] = nullptr; }
#endif
    return 0;
}
/* Stream-ordered barrier over the communicator (a one-element all-reduce on the context's stream): work enqueued behind it
 * starts only after every rank's work enqueued before its own barrier call has finished. */
int pcb_comm_barrier(pcb_ctx* c) {
    PCB_CHECK_ARG(c && c->comm, "no communicator");
    PCB_CUDA_OK(cudaSetDevice(c->device));
    if (ensure_dsmall(c, sizeof(cplx) * 2 * PCB_MAXL * PCB_MAXL + 65536)) return -1;
    return comm_allreduce(c, (double*)((char*)c->dsmall + sizeof(cplx) * 2 * PCB_MAXL * PCB_MAXL), 1);
}
/* A / H on whole columns whose data live as slabs on the `world` ranks: src[j * world + g] / dst[j * world + g] = column j's slab
 * on rank g as mapped by pcb_comm_share (zb: slab boundaries).  xcopy[j] and work[j] are LOCAL full columns of this context
 * (copy of X for the last pass; work space).  The slab gather / scatter of pcb_slab_exchange is fused into the first and the
 * last FFT pass, which read and write peer memory over NVLink tile by tile.  Caller: order the ranks with pcb_comm_barrier. */
int pcb_apply_dist(pcb_op* o, int mode, int ncols, const void* const* src, void* const* dst, const int* zb, int world,
                   void* const* xcopy, void* const* work) {
    PCB_CHECK_ARG(o && dst && zb && xcopy && work && ncols > 0 && ncols <= PCB_MAXC_DIST && world >= 1 && world <= PCB_MAXW, "bad arguments");
    PCB_CHECK_ARG(mode == PCB_APPLY_A || mode == PCB_APPLY_H, "mode must be PCB_APPLY_A or PCB_APPLY_H");
    pcb_ctx* c = o->ctx;
    PCB_CHECK_ARG(c->nloc == c->nn, "needs a full (non-slab) context");
    PCB_CHECK_ARG(c->N % c->plan->lx == 0, "grid size not supported by the peer-memory passes (x tiles must not straddle planes)");
    PCB_CHECK_ARG(zb[0] == 0 && zb[world] == c->N, "zb must cover [0, N]");
    PCB_CUDA_OK(cudaSetDevice(c->device));
    if (!c->ddist) PCB_CUDA_OK(cudaMalloc(&c->ddist, sizeof(PcbDist)));
    if (ensure_hstage(c, sizeof(cplx) * 2 * PCB_MAXL * PCB_MAXL + 65536)) return -1;
    PCB_CUDA_OK(cudaStreamSynchronize(c->stream));      // the staging table of the previous call has been consumed
    PcbDist* hd = (PcbDist*)c->hstage;
    memset(hd, 0, sizeof(PcbDist));
    hd->world = world;
    for (int g = 0; g <= world; ++g) hd->zb[g] = zb[g];
    PcbCols cols;
    memset(&cols, 0, sizeof cols);
    for (int j = 0; j < ncols; ++j) {
        for (int g = 0; g < world; ++g) { hd->src[j][g] = src ? (const cplx*)src[j * world + g] : nullptr; hd->dst[j][g] = (cplx*)dst[j * world + g]; }
        cols.in[j] = (const cplx*)xcopy[j];
        cols.out[j] = (cplx*)work[j];
    }
    PCB_CUDA_OK(cudaMemcpyAsync(c->ddist, hd, sizeof(PcbDist), cudaMemcpyHostToDevice, c->stream));
    o->d.dist = c->ddist;
    const int rc = apply_AH(o, mode, cols, ncols, 0, src ? 3 : 2);      // src == null: xcopy[] already holds the whole input columns
    o->d.dist = nullptr;
    return rc;
}

/* Measurement aid: `reps` all-reduces (sum) of `count` doubles over the communicator on the context's stream, timed with CUDA
 * events; *ms = average device time of one all-reduce (the latency the Gram pair of the large-grid mode pays per iteration). */
int pcb_comm_allreduce_timed(pcb_ctx* c, long long count, int reps, float* ms) {
    PCB_CHECK_ARG(c && c->comm && count > 0 && reps > 0 && ms, "bad arguments / no communicator");
    PCB_CUDA_OK(cudaSetDevice(c->device));
    if (ensure_dsmall(c, sizeof(double) * (size_t)count > sizeof(cplx) * 2 * PCB_MAXL * PCB_MAXL + 65536 ? sizeof(double) * (size_t)count : sizeof(cplx) * 2 * PCB_MAXL * PCB_MAXL + 65536)) return -1;
    PCB_CUDA_OK(cudaMemsetAsync(c->dsmall, 0, sizeof(double) * (size_t)count, c->stream));
    if (comm_allreduce(c, (double*)c->dsmall, count)) return -4;      // warm-up (first call sets up the NCCL channels)
    PCB_CUDA_OK(cudaEventRecord(c->ev0, c->stream));
    for (int i = 0; i < reps; ++i) if (comm_allreduce(c, (double*)c->dsmall, count)) return -4;
    PCB_CUDA_OK(cudaEventRecord(c->ev1, c->stream));
    PCB_CUDA_OK(cudaEventSynchronize(c->ev1));
    PCB_CUDA_OK(cudaEventElapsedTime(ms, c->ev0, c->ev1));
    *ms /= (float)reps;
    return 0;
}

/* Exchange between the row-sharded (slab) layout of the dense phase and whole columns for the operator (SURVEY 8e-ii).
 * zb[0..world]: i2-plane boundaries of the slabs (zb[rank] == ctx z0).  Column j lives as a slab column slab_cols[j] on
 * every rank and as a whole column full_cols[j] on rank owners[j] only (ignored elsewhere).
 * to_full = 1: every rank sends its three component segments of column j to owners[j];  to_full = 0: the reverse. */
int pcb_slab_exchange(pcb_ctx* c, int to_full, int ncols, const int* owners, const int* zb, void* const* slab_cols, void* const* full_cols) {
    PCB_CHECK_ARG(c && c->comm && owners && zb && slab_cols && full_cols && ncols > 0, "bad arguments / no communicator");
    PcbComm* cm = c->comm;
    const long long plane = (long long)c->N * c->N;
    PCB_CHECK_ARG(zb[cm->rank] == c->z0 && zb[cm->rank + 1] == c->z1, "zb does not match this slab context");
    PCB_CUDA_OK(cudaSetDevice(c->device));
    std::vector<int> is_send, peer;
    std::vector<void*> ptr;
    std::vector<long long> bytes;
    for (int j = 0; j < ncols; ++j) {
        const int o = owners[j];
        PCB_CHECK_ARG(o >= 0 && o < cm->world, "owner out of range");
        for (int comp = 0; comp < 3; ++comp) {
            cplx* mine = (cplx*)slab_cols[j] + comp * c->nloc;
            if (o == cm->rank) {
                cplx* full = (cplx*)full_cols[j] + comp * c->nn;
                for (int g = 0; g < cm->world; ++g) {
                    cplx* seg = full + (long long)zb[g] * plane;
                    const long long nb = (long long)(zb[g + 1] - zb[g]) * plane * (long long)sizeof(cplx);
                    if (g == cm->rank) {
                        if (to_full) PCB_CUDA_OK(cudaMemcpyAsync(seg, mine, nb, cudaMemcpyDeviceToDevice, c->stream));
                        else PCB_CUDA_OK(cudaMemcpyAsync(mine, seg, nb, cudaMemcpyDeviceToDevice, c->stream));
                    } else {
                        is_send.push_back(to_full ? 0 : 1); peer.push_back(g); ptr.push_back(seg); bytes.push_back(nb);
                    }
                }
            } else {
                is_send.push_back(to_full ? 1 : 0); peer.push_back(o); ptr.push_back(mine);
                bytes.push_back(c->nloc * (long long)sizeof(cplx));
            }
        }
    }
    const int nops = (int)is_send.size();
    if (nops == 0) return 0;
#ifdef PCB_EMU
    if (!cm->p2p_cb) { pcb_set_error("host-emu communicator has no p2p callback"); return -4; }
    if (cm->p2p_cb(nops, is_send.data(), peer.data(), ptr.data(), bytes.data()) != 0) { pcb_set_error("p2p callback failed"); return -4; }
#else
    int rc = g_nccl.GroupStart();
    for (int i = 0; i < nops && rc == 0; ++i)
        rc = is_send[i] ? g_nccl.Send(ptr[i], (size_t)bytes[i], PCB_NCCL_UINT8, peer[i], cm->nccl, c->stream)
                        : g_nccl.Recv(ptr[i], (size_t)bytes[i], PCB_NCCL_UINT8, peer[i], cm->nccl, c->stream);
    const int rc2 = g_nccl.GroupEnd();
    if (rc != 0 || rc2 != 0) { pcb_set_error("NCCL send/recv group failed: %s", g_nccl.GetErrorString(rc ? rc : rc2)); return -4; }
#endif
    return 0;
}

}  // extern "C"
