// pcb200 -- per-grid-size instantiation of the operator passes.
// Compiled once per supported N with -DPCB_N=.. -DPCB_R1=.. -DPCB_R2=.. (see build.py), so the
// sizes build in parallel and each object only carries the codelets it needs.
#include "pcb_operator.cuh"

#ifndef PCB_NTP
#define PCB_NTP 256
#endif
#ifndef PCB_N
#error "compile with -DPCB_N -DPCB_R1 -DPCB_R2"
#endif

namespace {

typedef Plan<PCB_N, PCB_R1, PCB_R2> P;
constexpr int NT = 128;      // y lines and split z passes (one CTA per tile)
constexpr int NTP = PCB_NTP;     // persistent z-mid kernel: 2 CTAs/SM of 256 threads when two stages fit twice in shared memory,
constexpr int kRowBytes = 3 * P::R1 * P::R2P * (int)sizeof(cplx);
constexpr int LX = (8 * kRowBytes <= 65536) ? 8 : (4 * kRowBytes <= 65536) ? 4 : (2 * kRowBytes <= 65536) ? 2 : 1;
constexpr int kStageX = LX * kRowBytes;               // one x-tile (three components)
// forward x pass: 64-thread CTAs where the first radix step has at most 64 items (LX * R2: N = 192, 240, 256) -- with 128 threads
// half of them would sit out the phase that issues the loads (N = 256, 8 columns: 4.48 -> 2.69 ms; the inverse pass, whose
// loading phase has 3 LX R1 items, gets slower with 64 threads, 4.40 -> 5.01 ms, and keeps 128)
constexpr int NTX = (LX * P::R2 <= 64) ? 64 : NT;
constexpr int kSmemL = 3 * P::N * 8 * (int)sizeof(cplx);
constexpr int kSmemZ = 2 * kSmemL;                       // two stages
// ... else (N >= 160) single-stage tiles with 2-3 CTAs of 256 threads per SM.  (Round 2, measured and removed: when two stages still
// fit ONCE, one CTA of 512 threads per SM with the cp.async double buffer -- the same 16 warps and pipeline depth per SM as the small
// sizes, no spills -- is slower: N = 160, 16 columns 2.09 vs 1.79 ms, N = 256, 8 columns 4.08 vs 3.31 ms.)
constexpr bool kZTwice = 2 * (kSmemZ + 1024) <= 224 * 1024;
constexpr int NSTZ = kZTwice ? 2 : 1;         // ... else single-stage tiles, still several CTAs per SM
constexpr int kSmemZU = NSTZ * kSmemL;

template <class K>
int set_smem(K kern, int bytes) {
    if (bytes > 48 * 1024) PCB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    return 0;
}
inline int ctas_per_sm(int smem, int regs_hint_threads) {
    int n = (224 * 1024) / (smem + 1024);
    if (n < 1) n = 1;
    if (n > regs_hint_threads) n = regs_hint_threads;
    return n;
}

// one CTA per tile (y lines and the split z passes)
#define PCB_GO(KERN, GRIDX, SMEM)                                                   \
    do {                                                                            \
        auto kfn = KERN;                                                            \
        if (set_smem(kfn, (SMEM))) return -1;                                       \
        dim3 grid((unsigned)(GRIDX), (unsigned)ncols, 1);                           \
        PCB_LAUNCH(kfn, grid, dim3(NT, 1, 1), (size_t)(SMEM), s, op, cols, tw);      \
        PCB_CUDA_OK(cudaGetLastError());                                            \
    } while (0)
#define PCB_GO_X(KERN, GRIDX, SMEM)                                                 \
    do {                                                                            \
        auto kfn = KERN;                                                            \
        if (set_smem(kfn, (SMEM))) return -1;                                       \
        dim3 grid((unsigned)(GRIDX), (unsigned)ncols, 1);                           \
        PCB_LAUNCH(kfn, grid, dim3(NTX, 1, 1), (size_t)(SMEM), s, op, cols, tw);     \
        PCB_CUDA_OK(cudaGetLastError());                                            \
    } while (0)
// persistent CTAs striding over (column, tile)
#define PCB_GO_P(KERN, NTHR, TILES, SMEM, MAXCTA)                                   \
    do {                                                                            \
        auto kfn = KERN;                                                            \
        if (set_smem(kfn, (SMEM))) return -1;                                       \
        long long gx = (long long)sms * ctas_per_sm((SMEM), (MAXCTA));              \
        const long long tot = (long long)(TILES) * ncols;                           \
        if (gx > tot) gx = tot;                                                     \
        dim3 grid((unsigned)gx, 1, 1);                                              \
        PCB_LAUNCH(kfn, grid, dim3((NTHR), 1, 1), (size_t)(SMEM), s, op, cols, tw, ncols); \
        PCB_CUDA_OK(cudaGetLastError());                                            \
    } while (0)

// plane mode: N % 8 == 0, tiles of 8 rows must not straddle an i2 plane, and N x (N+1) complex fit in one CTA's shared memory
constexpr bool kPlane = (P::N % 8 == 0) && (LX == 8) && ((long long)P::N * (P::N + 1) * 16 <= 232448);
constexpr int kSmemMid = P::N * (P::N + 1) * (int)sizeof(cplx);
// z-split plane mode (half planes of N/2 x N; ZSplit in pcb_operator.cuh): N % 16 == 0, a plan for N/2, the half plane fits.  The only
// plane mode of N = 128, 144, 160; selectable (PCB200_PLANE_SPLIT=1 / pcb_ctx_set "plane_split") for the smaller sizes as well
constexpr bool kPlaneSplit = (P::N % 16 == 0) && (LX == 8) && PlanOf<P::N / 2>::ok && ((long long)(P::N / 2) * (P::N + 1) * 16 + 128 <= 232448);
constexpr bool kPlaneFive = kPlane && Mid2<P>::OK;
#ifdef PCB_EMU
constexpr bool kPlaneCoupled = false;      // thread-block clusters are not emulated: the coupled dielectric keeps the five-pass path there
#else
constexpr bool kPlaneCoupled = kPlane && P::N % 3 == 0 && kSmemMid + 128 <= 232448;
#endif
#ifdef PCB_EMU
constexpr bool kPlaneSplitCoupled = false;
#else
constexpr bool kPlaneSplitCoupled = kPlaneSplit;      // coupled 3x3 M on clusters of three CTAs, one half plane per cluster
#endif
// plane passes (k_mid / k_mid2) move their rows by TMA bulk copies on the device (one mbarrier per warp behind the plane, at most
// 128 bytes) and by row loops under host emulation
#ifdef PCB_EMU
constexpr int kTma = 0;
#else
constexpr int kTma = 1;
#endif
static_assert(!kPlane || kSmemMid + 128 <= 232448, "whole plane + mbarriers exceed a CTA's shared memory");
static_assert(!kPlaneSplit || (P::N / 2) * (P::N + 1) * (int)sizeof(cplx) + 128 <= 232448, "half plane + mbarriers exceed a CTA's shared memory");
constexpr int kStageXT = 3 * LX * (P::R1 * P::R2P + 1) * (int)sizeof(cplx);

constexpr int GX = (P::N * P::N + LX - 1) / LX;          // x tiles per column
constexpr int GL = ((P::N + 7) / 8) * P::N;              // strided-line tiles per column

#ifndef PCB_EMU
// persistent launch on clusters of three CTAs (one per component): as many clusters as can be co-resident
template <class K>
int launch_cluster3(K kfn, int threads, int smem, int planes, const PcbOp& op, const PcbCols& cols, const cplx* tw, int ncols, cudaStream_t s, int sms, int N) {
    if (set_smem(kfn, smem)) return -1;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cudaLaunchAttribute at;
    at.id = cudaLaunchAttributeClusterDimension;
    at.val.clusterDim.x = 3; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
    cfg.blockDim = dim3((unsigned)threads, 1, 1);
    cfg.dynamicSmemBytes = (size_t)smem;
    cfg.stream = s;
    cfg.attrs = &at; cfg.numAttrs = 1;
    static int max_clusters = 0;      // per kernel instantiation: co-resident clusters (a 3-CTA cluster needs three free SMs of one GPC)
    if (max_clusters == 0) {
        cfg.gridDim = dim3(3 * 148, 1, 1);
        PCB_CUDA_OK(cudaOccupancyMaxActiveClusters(&max_clusters, kfn, &cfg));
        if (getenv("PCB200_DEBUG")) fprintf(stderr, "[pcb200] plane pass, coupled M, N = %d, %d threads: %d co-resident clusters of 3 CTAs (%d SMs)\n", N, threads, max_clusters, sms);
        if (max_clusters < 1) { pcb_set_error("plane mode: no 3-CTA cluster of the plane pass fits on this device"); max_clusters = 0; return -1; }
    }
    long long ncl = max_clusters;
    if (ncl > planes) ncl = planes;
    cfg.gridDim = dim3((unsigned)(3 * ncl), 1, 1);
    PCB_CUDA_OK(cudaLaunchKernelEx(&cfg, kfn, op, cols, tw, ncols));
    PCB_CUDA_OK(cudaGetLastError());
    return 0;
}
#endif

// five-sweep plane pass (k_mid2): instantiated only for the plans it supports
template <bool ENABLED, class PP>
struct PlaneFive {
    static int go(const PcbOp&, const PcbCols&, int, int, const cplx*, cudaStream_t, int) {
        pcb_set_error("the five-sweep plane pass is not available for N = %d", PP::N);
        return -1;
    }
};
template <class PP>
struct PlaneFive<true, PP> {
    static int go(const PcbOp& op, const PcbCols& cols, int ncols, int pass_id, const cplx* tw, cudaStream_t s, int sms) {
        typedef Mid2<PP> M2;
        if (pass_id == PCB_PASS_MASKBITS2) {
            const long long total = 3LL * PP::N * 8 * PP::N;
            PCB_LAUNCH((k_mask_bits2<PP>), dim3((unsigned)((total + 255) / 256), 1, 1), dim3(256, 1, 1), 0, s, op, const_cast<unsigned*>(op.mbits2));
            PCB_CUDA_OK(cudaGetLastError());
            return 0;
        }
        constexpr int smem = PP::N * (PP::N + 1) * (int)sizeof(cplx) + (kTma ? 128 : 0);
        if (pass_id == PCB_PASS_MASKPLANE2) {
            const long long total = (long long)PP::N * PP::N * PP::N;
            PCB_LAUNCH((k_mask_plane2<PP>), dim3((unsigned)((total + 255) / 256), 1, 1), dim3(256, 1, 1), 0, s, op, const_cast<unsigned char*>(op.maskp2));
            PCB_CUDA_OK(cudaGetLastError());
            return 0;
        }
#ifndef PCB_EMU
        if (op.diel == PCB_DIEL_TRIVIAL) {
            if (PP::N % 3 != 0) { pcb_set_error("five-sweep plane pass: coupled M not available for N = %d", PP::N); return -1; }
            return launch_cluster3(k_mid2<PP, 2, 1>, M2::NTHR, smem, PP::N * ncols, op, cols, tw, ncols, s, sms, PP::N);
        }
#endif
        if (op.diel == PCB_DIEL_NONE) PCB_GO_P((k_mid2<PP, 0, kTma>), M2::NTHR, 3 * PP::N, smem, 1);
        else PCB_GO_P((k_mid2<PP, 1, kTma>), M2::NTHR, 3 * PP::N, smem, 1);
        return 0;
    }
};

// coupled 3x3 M on clusters of three CTAs / peer-memory x passes: full planes only (not in the z-split plane mode)
template <bool OK, class PP, int ZS>
struct Coupled {
    static int go(const PcbOp&, const PcbCols&, int, int, const cplx*, cudaStream_t, int) {
        pcb_set_error("plane mode: no cluster form of the coupled dielectric for N = %d", PP::N);
        return -1;
    }
};
#ifndef PCB_EMU
template <class PP, int ZS>
struct Coupled<true, PP, ZS> {
    static int go(const PcbOp& op, const PcbCols& cols, int ncols, int pass_id, const cplx* tw, cudaStream_t s, int sms) {
        if (ZS == 1 && kPlaneFive && op.mid_five && op.mbits2 != nullptr && op.maskp2 != nullptr)
            return PlaneFive<(kPlaneFive && ZS == 1), PP>::go(op, cols, ncols, pass_id, tw, s, sms);
        // (z-split: one cluster per HALF plane -- the three components of the half plane h of (column, i0))
        return launch_cluster3(k_mid<PP, 2, 1, 0, 0, ZS>, PP::N / ZS / 8 * 32, PP::N / ZS * (PP::N + 1) * (int)sizeof(cplx) + 128, PP::N * ZS * ncols,
                               op, cols, tw, ncols, s, sms, PP::N);
    }
};
#endif
template <bool OK, class PP>
struct XDist {
    static int go(const PcbOp&, const PcbCols&, int, int, const cplx*, cudaStream_t) {
        pcb_set_error("z-split plane mode has no peer-memory x passes (N = %d)", PP::N);
        return -1;
    }
};
template <class PP>
struct XDist<true, PP> {
    static int go(const PcbOp& op, const PcbCols& cols, int ncols, int pass_id, const cplx* tw, cudaStream_t s) {
        if (pass_id == PCB_PASS_XFWD_SYM_TD) PCB_GO((k_xfwd<PP, LX, NT, 1, 1, 1>), GX, kStageXT);
        else if (pass_id == PCB_PASS_XINV_A_TD) PCB_GO((k_xinv<PP, LX, NT, 1, 1, 1>), GX, kStageXT);
        else PCB_GO((k_xinv<PP, LX, NT, 2, 1, 1>), GX, kStageXT);
        return 0;
    }
};

// plane-mode passes exist only for sizes with kPlane (the kernels are not even instantiated otherwise)
template <bool ENABLED, class PP, int ZS>
struct PlanePass {
    static int go(const PcbOp&, const PcbCols&, int, int, const cplx*, cudaStream_t, int) {
        pcb_set_error("plane mode is not available for N = %d", PP::N);
        return -1;
    }
};
template <class PP, int ZS>
struct PlanePass<true, PP, ZS> {
    static int go(const PcbOp& op, const PcbCols& cols, int ncols, int pass_id, const cplx* tw, cudaStream_t s, int sms) {
        constexpr int kSmemMidZ = PP::N / ZS * (PP::N + 1) * (int)sizeof(cplx);
        if (pass_id == PCB_PASS_MASKBITS) {
            const long long total = 3LL * PP::N * PP::N * ZS * ZSplit<PP, ZS>::PZ::R1;
            PCB_LAUNCH((k_mask_bits<PP, ZS>), dim3((unsigned)((total + 255) / 256), 1, 1), dim3(256, 1, 1), 0, s, op, const_cast<unsigned*>(op.mbits));
            PCB_CUDA_OK(cudaGetLastError());
            return 0;
        }
        if (pass_id == PCB_PASS_MATBYTES) {
            const long long total = 3LL * PP::N * PP::N * ZS * ZSplit<PP, ZS>::PZ::R1;
            PCB_LAUNCH((k_mat_bytes<PP, ZS>), dim3((unsigned)((total + 255) / 256), 1, 1), dim3(256, 1, 1), 0, s, op, const_cast<unsigned char*>(op.matp));
            PCB_CUDA_OK(cudaGetLastError());
            return 0;
        }
        if (pass_id == PCB_PASS_MASKPLANE) {
            const long long total = (long long)PP::N * PP::N * PP::N;
            PCB_LAUNCH((k_mask_plane<PP, ZS>), dim3((unsigned)((total + 255) / 256), 1, 1), dim3(256, 1, 1), 0, s, op, const_cast<unsigned char*>(op.maskp));
            PCB_CUDA_OK(cudaGetLastError());
            return 0;
        }
        if (pass_id == PCB_PASS_COORDTAB) {
            PCB_LAUNCH((k_coord_tables<PP, ZS>), dim3((unsigned)((PP::N + 127) / 128), 1, 1), dim3(128, 1, 1), 0, s, const_cast<int*>(op.ctab));
            PCB_CUDA_OK(cudaGetLastError());
            return 0;
        }
// plane pass on whole (ZS = 1) or half (ZS = 2) planes: one CTA per plane, N / ZS / 8 warps
#define PCB_GO_MID(DIEL, HALF, STEN) PCB_GO_P((k_mid<PP, DIEL, kTma, HALF, STEN, ZS>), PP::N / ZS / 8 * 32, 3 * PP::N * ZS, kSmemMidZ + (kTma ? 128 : 0), 1)
        if (pass_id == PCB_PASS_MID_FWD_O || pass_id == PCB_PASS_MID_INV_ST) {      // ... with the stencil fused into the inverse half
            const int k = op.sten.k;
            if (pass_id == PCB_PASS_MID_FWD_O) PCB_GO_MID(0, 1, 1);
            else if (k == 1) PCB_GO_MID(0, 2, 3);
            else if (k == 2) PCB_GO_MID(0, 2, 5);
            else PCB_GO_MID(0, 2, 1);
            return 0;
        }
        if (pass_id == PCB_PASS_MID_FWD || pass_id == PCB_PASS_MID_INV) {      // halves of the plane pass (cross-DoF dielectric)
            if (pass_id == PCB_PASS_MID_FWD) PCB_GO_MID(0, 1, 0);
            else PCB_GO_MID(0, 2, 0);
            return 0;
        }
#ifndef PCB_EMU
        if (pass_id == PCB_PASS_MID && op.diel == PCB_DIEL_TRIVIAL) {
            // coupled 3x3 M: clusters of three CTAs (one component each) exchanging the coupled points through DSMEM
            return Coupled<(ZS == 1 ? kPlaneCoupled : kPlaneSplitCoupled), PP, ZS>::go(op, cols, ncols, pass_id, tw, s, sms);
        }
#endif
        if (pass_id == PCB_PASS_XFWD_SYM_TD || pass_id == PCB_PASS_XINV_A_TD || pass_id == PCB_PASS_XINV_H_TD)
            return XDist<ZS == 1, PP>::go(op, cols, ncols, pass_id, tw, s);
        if constexpr (ZS == 2) {      // z-split plane mode: x passes with the split tiles, plane pass on half planes
            if (pass_id == PCB_PASS_XFWD_SYM_T) PCB_GO((k_xfwd<PP, LX, NT, 1, 1, 0, ZS>), GX, kStageXT);
            else if (pass_id == PCB_PASS_XINV_A_T) PCB_GO((k_xinv<PP, LX, NT, 1, 1, 0, ZS>), GX, kStageXT);
            else if (pass_id == PCB_PASS_XINV_H_T) PCB_GO((k_xinv<PP, LX, NT, 2, 1, 0, ZS>), GX, kStageXT);
            else if (pass_id == PCB_PASS_XINV_T) PCB_GO((k_xinv<PP, LX, NT, 0, 1, 0, ZS>), GX, kStageXT);
            else if (pass_id == PCB_PASS_MID && op.diel == PCB_DIEL_NONE) PCB_GO_MID(0, 0, 0);
            else if (pass_id == PCB_PASS_MID && op.diel == PCB_DIEL_CHIRAL) PCB_GO_MID(1, 0, 0);
            else if (pass_id == PCB_PASS_MID && op.diel == PCB_DIEL_MATERIALS) PCB_GO_MID(4, 0, 0);
            else { pcb_set_error("z-split plane mode: pass %d / dielectric type %d not supported", pass_id, op.diel); return -1; }
            return 0;
        }
        if (pass_id == PCB_PASS_XFWD_SYM_T) {
            // from N = 64 on two tiles per CTA, the second tile's loads behind the first tile's radix-R2 phase (N = 48: 0.058 vs
            // 0.051 ms -- below N = 64 one tile per CTA stays)
            if constexpr (LX * PP::R2 <= NT && PP::N >= 64 && ZS == 1) PCB_GO((k_xfwd2<PP, LX, NT>), (GX + 1) / 2, kStageXT);
            else PCB_GO((k_xfwd<PP, LX, NT, 1, 1>), GX, kStageXT);
        }
        else if (pass_id == PCB_PASS_XINV_A_T) PCB_GO((k_xinv<PP, LX, NT, 1, 1>), GX, kStageXT);
        else if (pass_id == PCB_PASS_XINV_H_T) PCB_GO((k_xinv<PP, LX, NT, 2, 1>), GX, kStageXT);
        else if (pass_id == PCB_PASS_XINV_T) PCB_GO((k_xinv<PP, LX, NT, 0, 1>), GX, kStageXT);
        else if (pass_id == PCB_PASS_MASKBITS2 || pass_id == PCB_PASS_MASKPLANE2) return PlaneFive<(kPlaneFive && ZS == 1), PP>::go(op, cols, ncols, pass_id, tw, s, sms);
        else if (op.diel == PCB_DIEL_NONE || op.diel == PCB_DIEL_CHIRAL) {
            if (kPlaneFive && ZS == 1 && op.mid_five && (op.diel == PCB_DIEL_NONE || op.mbits2 != nullptr)) return PlaneFive<(kPlaneFive && ZS == 1), PP>::go(op, cols, ncols, pass_id, tw, s, sms);
            if (op.diel == PCB_DIEL_NONE) PCB_GO_MID(0, 0, 0);
            else PCB_GO_MID(1, 0, 0);
        }
        else if (op.diel == PCB_DIEL_MATERIALS) PCB_GO_MID(4, 0, 0);      // seven sweeps: k_mid2 has no materials form
        else { pcb_set_error("plane mode: dielectric type %d not supported", op.diel); return -1; }
        return 0;
#undef PCB_GO_MID
    }
};

int run_pass(const PcbOp& op, const PcbCols& cols, int ncols, int pass_id, const cplx* tw, cudaStream_t s, int sms) {
    switch (pass_id) {
        case PCB_PASS_XFWD_SYM: PCB_GO_X((k_xfwd<P, LX, NTX, 1>), GX, kStageX); break;
        case PCB_PASS_XFWD:     PCB_GO_X((k_xfwd<P, LX, NTX, 0>), GX, kStageX); break;
        case PCB_PASS_YFWD:     PCB_GO((k_line<P, 1, -1, NT>), GL, kSmemL); break;
        case PCB_PASS_ZFWD:     PCB_GO((k_line<P, 2, -1, NT>), GL, kSmemL); break;
        case PCB_PASS_ZINV:     PCB_GO((k_line<P, 2, +1, NT>), GL, kSmemL); break;
        case PCB_PASS_YINV:     PCB_GO((k_line<P, 1, +1, NT>), GL, kSmemL); break;
        case PCB_PASS_XINV:     PCB_GO((k_xinv<P, LX, NT, 0>), GX, kStageX); break;
        case PCB_PASS_XINV_A:   PCB_GO((k_xinv<P, LX, NT, 1>), GX, kStageX); break;
        case PCB_PASS_XINV_H:   PCB_GO((k_xinv<P, LX, NT, 2>), GX, kStageX); break;
        case PCB_PASS_XFWD_SYM_D: PCB_GO_X((k_xfwd<P, LX, NTX, 1, 0, 1>), GX, kStageX); break;
        case PCB_PASS_XINV_A_D:   PCB_GO((k_xinv<P, LX, NT, 1, 0, 1>), GX, kStageX); break;
        case PCB_PASS_XINV_H_D:   PCB_GO((k_xinv<P, LX, NT, 2, 0, 1>), GX, kStageX); break;
        case PCB_PASS_ZMID:
            if (op.diel == PCB_DIEL_NONE) PCB_GO_P((k_zmid<P, 0, NTP, NSTZ>), NTP, GL, kSmemZU, 3);
            else if (op.diel == PCB_DIEL_CHIRAL) PCB_GO_P((k_zmid<P, 1, NTP, NSTZ>), NTP, GL, kSmemZU, 3);
            else if (op.diel == PCB_DIEL_TRIVIAL) PCB_GO_P((k_zmid<P, 2, NTP, NSTZ>), NTP, GL, kSmemZU, 2);
            else if (op.diel == PCB_DIEL_MATERIALS) PCB_GO_P((k_zmid<P, 4, NTP, NSTZ>), NTP, GL, kSmemZU, 3);
            else { pcb_set_error("zmid: dielectric type %d has no fused z pass", op.diel); return -1; }
            break;
        case PCB_PASS_XFWD_SYM_T: case PCB_PASS_MID: case PCB_PASS_XINV_A_T: case PCB_PASS_XINV_H_T: case PCB_PASS_MASKBITS:
        case PCB_PASS_MID_FWD: case PCB_PASS_MID_INV: case PCB_PASS_MASKPLANE: case PCB_PASS_COORDTAB: case PCB_PASS_MASKBITS2:
        case PCB_PASS_XFWD_SYM_TD: case PCB_PASS_XINV_A_TD: case PCB_PASS_XINV_H_TD: case PCB_PASS_MID_FWD_O: case PCB_PASS_MID_INV_ST: case PCB_PASS_MASKPLANE2:
        case PCB_PASS_XINV_T: case PCB_PASS_MATBYTES:
            if (op.zsplit) return PlanePass<kPlaneSplit, P, 2>::go(op, cols, ncols, pass_id, tw, s, sms);
            return PlanePass<kPlane, P, 1>::go(op, cols, ncols, pass_id, tw, s, sms);
        default: pcb_set_error("unknown pass id %d", pass_id); return -1;
    }
    return 0;
}

int run_apply(const PcbOp& op, const PcbCols& cols, int ncols, int mode, const cplx* tw, cudaStream_t s, int sms) {
    static const int fwd[] = {PCB_PASS_XFWD, PCB_PASS_YFWD, PCB_PASS_ZFWD};
    static const int inv[] = {PCB_PASS_ZINV, PCB_PASS_YINV, PCB_PASS_XINV};
    static const int opA[] = {PCB_PASS_XFWD_SYM, PCB_PASS_YFWD, PCB_PASS_ZMID, PCB_PASS_YINV, PCB_PASS_XINV_A};
    static const int opH[] = {PCB_PASS_XFWD_SYM, PCB_PASS_YFWD, PCB_PASS_ZMID, PCB_PASS_YINV, PCB_PASS_XINV_H};
    const int* seq;
    int n;
    switch (mode) {
        case 0: seq = fwd; n = 3; break;
        case 1: seq = inv; n = 3; break;
        case 2: seq = opA; n = 5; break;
        case 3: seq = opH; n = 5; break;
        default: pcb_set_error("unknown apply mode %d", mode); return -1;
    }
    for (int i = 0; i < n; ++i)
        if (run_pass(op, cols, ncols, seq[i], tw, s, sms)) return -1;
    return 0;
}

}  // namespace

#define PCB_CAT2(a, b) a##b
#define PCB_CAT(a, b) PCB_CAT2(a, b)
extern const PcbOpLaunch PCB_CAT(pcb_plan_, PCB_N) = {PCB_N, PCB_R1, PCB_R2, (kPlane || kPlaneSplit) ? 1 : 0, kPlaneCoupled ? 1 : 0, kPlaneFive ? 1 : 0, LX,
                                                      kPlaneSplit ? (kPlane ? 1 : 2) : 0, kPlaneSplit ? PlanOf<(kPlaneSplit ? P::N / 2 : P::N)>::type::R1 : 0,
                                                      kPlaneSplit ? PlanOf<(kPlaneSplit ? P::N / 2 : P::N)>::type::R2 : 0, kPlaneSplitCoupled ? 1 : 0, run_apply, run_pass};
