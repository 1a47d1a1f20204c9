// pcb200 -- the matrix-free operator  H x = K_A IFFT3( M FFT3( K_A^H x ) ) + gamma K_B x + shift x
// (reference: pcfft.py:130-181, _kernels.py:13-71, discretization.py:352-401) as hand-written
// mixed-radix complex128 FFT passes with the Fourier symbols and the dielectric multiply fused in.
//
// Two pass structures (chosen per call in pcb_capi.cu):
//
// PLANE MODE -- three global passes, 7 column transfers per op-apply (N % 8 == 0, N <= 120; N = 128, 144, 160 in the z-split form, ZSplit below):
//   k_xfwd<T>  x-lines:  y = (-conj k) x x fused on load, forward FFT along i0, stored TRANSPOSED as W'[c][i0][i2][i1]
//   k_mid      one (i1,i2) plane per CTA in shared memory: forward y, forward z, M, inverse z, inverse y, in place
//   k_xinv<T>  x-lines:  inverse FFT along i0 from W', 1/N^3, k x v, + gamma conj(k)(k.x) + shift x, natural layout
//
// FIVE PASSES -- 11 column transfers (any N with a plan, coupled 3x3 M; the cross-DoF M splits pass 3 around a stencil kernel):
//   k_xfwd     x-lines:  y = (-conj k) x x  fused on load, forward FFT along i0          (K_A^H, pass 1)
//   k_line     y-lines:  forward FFT along i1                                            (pass 2)
//   k_zmid     z-lines:  forward FFT along i2, M (point-wise, real space), inverse FFT   (pass 3)
//   k_line     y-lines:  inverse FFT along i1                                            (pass 4)
//   k_xinv     x-lines:  inverse FFT along i0, 1/N^3, k x v, + gamma conj(k)(k.x) + shift x on store
//
// Every 1-D FFT of length N = R1*R2 is two in-register radix codelets (pcb_codelets.cuh) with one shared-memory
// exchange between them.  y/z lines are processed for 8 consecutive i0 at once (128-byte segments, fully coalesced);
// coprime factorisations use the Good-Thomas maps there (no twiddles), x-lines always use Cooley-Tukey so that global
// accesses stay contiguous.  Around M the data stays in registers between the last forward and the first inverse radix.
#pragma once
#include "pcb_common.cuh"
#include <type_traits>

#define PCB_MAXC 32   // columns per launch (pointer lists travel in kernel parameter space)

struct PcbCols {
    const cplx* in[PCB_MAXC];   // source columns (X)
    cplx* out[PCB_MAXC];        // destination / work columns
    cplx* wrk[PCB_MAXC];        // plane mode: scratch columns holding the transposed layout W'[c][i0][i2][i1]
};

// occupancy hint of the x passes: ask for `want` CTAs/SM (caps registers) only where the tile is small enough to allow it
constexpr int pcb_min_ctas(int stage_bytes, int r1, int want) { return (want * stage_bytes <= 200 * 1024 && r1 <= 8) ? want : 1; }
// inverse x pass with a first radix above 8: three CTAs per SM where they fit -- uncapped, N = 256 takes 174 registers, which the
// allocation granularity (8 per thread) turns into two resident CTAs of four warps instead of three
constexpr int pcb_min_ctas_inv(int stage_bytes, int r1, int want) {
    return r1 <= 8 ? pcb_min_ctas(stage_bytes, r1, want) : (3 * stage_bytes <= 200 * 1024 ? 3 : 1);
}
constexpr int pcb_gcd(int a, int b) { return b == 0 ? a : pcb_gcd(b, a % b); }
constexpr int pcb_modinv(int a, int m) {   // a^-1 mod m (m small)
    for (int x = 1; x < m; ++x) if ((a * x) % m == 1) return x;
    return 1;
}

template <int N_, int R1_, int R2_>
struct Plan {
    static constexpr int N = N_, R1 = R1_, R2 = R2_;
    static_assert(R1_ * R2_ == N_, "N = R1 * R2");
    static constexpr bool PFA = pcb_gcd(R1_, R2_) == 1;
    static constexpr int U = pcb_modinv(R2_ % R1_, R1_);   // R2^-1 mod R1
    static constexpr int V = pcb_modinv(R1_ % R2_, R2_);   // R1^-1 mod R2
    static constexpr int R2P = R2_ | 1;                    // odd stride: conflict-free strided smem access
    // index maps of the strided (y/z) passes
    PCB_HD static int lin(int n1, int n2) { return PFA ? (R2 * n1 + R1 * n2) % N : n1 * R2 + n2; }
    PCB_HD static int lout(int k1, int k2) { return PFA ? (R2 * U * k1 + R1 * V * k2) % N : k1 + R1 * k2; }
    // the same maps split into a per-digit part (a compile-time constant in unrolled loops, or computed once per item)
    // and a conditional subtract instead of a modulo per element
    PCB_HD static int lin1(int n1) { return PFA ? (R2 * n1) % N : n1 * R2; }
    PCB_HD static int lin2(int n2) { return PFA ? (R1 * n2) % N : n2; }
    PCB_HD static int lout1(int k1) { return PFA ? (R2 * U * k1) % N : k1; }
    PCB_HD static int lout2(int k2) { return PFA ? (R1 * V * k2) % N : R1 * k2; }
    PCB_HD static int wrap(int s) { return PFA ? (s >= N ? s - N : s) : s; }
    // output index held by slot s after a forward transform whose digits (k1, k2) sit in slot lin(k1, k2)
    PCB_HD static int coord(int s) {
        return PFA ? lout(((s % R1) * U) % R1, ((s % R2) * V) % R2) : (s / R2) + R1 * (s % R2);
    }
};

// the plan of a grid size by number (pcb_plans.inc): the z-split plane mode needs the plan of N / 2 next to the one of N
template <int N_>
struct PlanOf { static constexpr bool ok = false; typedef Plan<N_, N_, 1> type; };
#define PCB_PLAN(n, r1, r2) template <> struct PlanOf<n> { static constexpr bool ok = true; typedef Plan<n, r1, r2> type; };
#include "pcb_plans.inc"
#undef PCB_PLAN

// Z-SPLIT PLANE MODE (ZS = 2; N = 128, 144, 160, where an N x (N+1) plane no longer fits one SM's shared memory): the first
// radix-2 step of the z transform -- decimation in frequency, pairs (i2', i2' + N/2) -- is done by the forward x pass, whose
// tiles then hold 4 consecutive i1 of BOTH planes i2' and i2' + N/2:
//     E_h[i2'] = (x[i2'] + (-1)^h x[i2' + N/2]) w_N^(h i2'),   h = 0, 1,
// stored at plane row h N/2 + i2' (the position the inputs came from), so that every (i1, i2) plane falls into two independent
// HALF planes of N/2 x N elements whose z transform has length N/2 (output k' of half h is grid index i2 = 2 k' + h).  The
// plane pass runs on half planes (one per CTA, N/16 warps, 16 columns per warp in the z steps), and the inverse x pass undoes
// the split on load: x[i2' + j N/2] = e[i2'] + (-1)^j conj(w_N^i2') o[i2'].  Three passes and 7 column transfers as in plane
// mode proper, instead of the five passes / 11 transfers these sizes had.  tw: [0, N) twiddles of the plan of N, [N, N + N/2)
// those of the plan of N/2, [N + N/2, 2N) the split twiddles w_N^n.
template <class P, int ZS>
struct ZSplit {
    static constexpr int N = P::N, NZ = N / ZS;
    typedef typename PlanOf<NZ>::type PZ;
    // row r of x tile `tile` (LX rows: LX / ZS consecutive i1 of each of the ZS planes i2' + h NZ) -> i1 + N i2
    template <int LX> PCB_HD static int row(int tile, int r) {
        constexpr int LH = LX / ZS;
        return ZS == 1 ? tile * LX + r : ((tile / (N / LH)) + (r / LH) * NZ) * N + (tile % (N / LH)) * LH + r % LH;
    }
    // grid index i2 of plane row rho (= h NZ + slot of the plan of NZ)
    PCB_HD static int coord_row(int rho) { return ZS == 1 ? P::coord(rho) : ZS * PZ::coord(rho % NZ) + rho / NZ; }
};

// z = a x v  (cross product, _kernels.py:51-66)
PCB_HD void pcb_cross(const cplx a[3], const cplx v[3], cplx z[3]) {
    z[0] = csub(cmul(a[1], v[2]), cmul(a[2], v[1]));
    z[1] = csub(cmul(a[2], v[0]), cmul(a[0], v[2]));
    z[2] = csub(cmul(a[0], v[1]), cmul(a[1], v[0]));
}

// ---- cp.async (LDGSTS) helpers: global -> shared without staging in registers ------------------------
#ifdef PCB_EMU
PCB_D void pcb_cp16(cplx* dst, const cplx* src) { *dst = *src; }
PCB_D void pcb_cp8(void* dst, const void* src) { memcpy(dst, src, 8); }
PCB_D void pcb_cp_commit() {}
template <int N> PCB_D void pcb_cp_wait() {}
#else
PCB_D void pcb_cp16(cplx* dst, const cplx* src) {
    unsigned d = (unsigned)__cvta_generic_to_shared(dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(src));
}
PCB_D void pcb_cp8(void* dst, const void* src) {
    unsigned d = (unsigned)__cvta_generic_to_shared(dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(d), "l"(src));
}
PCB_D void pcb_cp_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N> PCB_D void pcb_cp_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }
#endif

// ---- bulk (TMA, 1-D) copies with mbarrier completion: one thread moves a whole row, no LSU instructions per element ----
#ifndef PCB_EMU
PCB_D unsigned pcb_smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
PCB_D void pcb_mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(pcb_smem_u32(bar)), "r"(count));
}
PCB_D void pcb_mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(pcb_smem_u32(bar)), "r"(bytes) : "memory");
}
PCB_D void pcb_mbar_wait(unsigned long long* bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "PCB_MBAR_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra PCB_MBAR_DONE;\n"
        "bra PCB_MBAR_WAIT;\n"
        "PCB_MBAR_DONE:\n"
        "}\n" ::"r"(pcb_smem_u32(bar)), "r"(parity) : "memory");
}
PCB_D void pcb_bulk_load(void* smem_dst, const void* gsrc, unsigned bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                 ::"r"(pcb_smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(pcb_smem_u32(bar)) : "memory");
}
PCB_D void pcb_bulk_store(void* gdst, const void* smem_src, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n" ::"l"(gdst), "r"(pcb_smem_u32(smem_src)), "r"(bytes) : "memory");
}
PCB_D void pcb_bulk_commit() { asm volatile("cp.async.bulk.commit_group;\n" ::: "memory"); }
PCB_D void pcb_bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory"); }
PCB_D void pcb_fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }
PCB_D void pcb_fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory"); }
// ---- thread-block clusters: distributed shared memory (the coupled 3x3 dielectric of the plane pass) ----
PCB_D unsigned pcb_cluster_ctarank() { unsigned r; asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r)); return r; }
PCB_D unsigned pcb_cluster_id() { unsigned r; asm volatile("mov.u32 %0, %%clusterid.x;\n" : "=r"(r)); return r; }
PCB_D unsigned pcb_cluster_count() { unsigned r; asm volatile("mov.u32 %0, %%nclusterid.x;\n" : "=r"(r)); return r; }
PCB_D unsigned pcb_mapa(unsigned smem_addr, unsigned rank) {      // the same shared-memory offset in CTA `rank` of the cluster
    unsigned r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;\n" : "=r"(r) : "r"(smem_addr), "r"(rank));
    return r;
}
PCB_D cplx pcb_ld_cluster(unsigned addr) {
    cplx v;
    asm volatile("ld.shared::cluster.v2.f64 {%0, %1}, [%2];\n" : "=d"(v.x), "=d"(v.y) : "r"(addr) : "memory");
    return v;
}
PCB_D void pcb_st_cluster(unsigned addr, cplx v) {
    asm volatile("st.shared::cluster.v2.f64 [%0], {%1, %2};\n" ::"r"(addr), "d"(v.x), "d"(v.y) : "memory");
}
PCB_D void pcb_cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
#endif

#ifdef PCB_EMU
PCB_D void pcb_prefetch_l2(const void*) {}
#else
PCB_D void pcb_prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];\n" ::"l"(p)); }
#endif

// ---------------------------------------------------------------------------------------
// Pass 1: x-lines forward.  SYM: 0 plain FFT, 1 multiply by K_A^H = (-conj k) x . on load.
// Tile = LX consecutive rows (a row = all i0 for one (i1,i2)), all three components; one CTA per tile, registers stage the
// radix-R1 input, shared memory the exchange.  Measured alternatives on B200 (N = 120, 16 columns): a persistent cp.async
// double-buffered variant 0.63 ms and a three-phase variant with a coalesced point-wise prologue 0.53 ms, vs 0.51 ms for this
// form with the 4-CTAs/SM register cap (plane mode: 4-row tiles with 64 threads and 8 CTAs/SM 0.55 ms, 16-row tiles with 256 threads and 2 CTAs/SM 0.57 ms, persistent CTAs
// with TMA bulk row copies into one in-place tile buffer and the next tile issued behind the second radix step 0.64 ms) -- so the simple form
// stays (the inverse pass, which also re-reads X, does gain from
// the three-phase structure; the z pass, with twice the arithmetic per byte, from the cp.async pipeline).
// ---------------------------------------------------------------------------------------
// TRN = 1 (plane mode): the output goes to the scratch column in the transposed layout W'[c][k][i2][i1] (8 consecutive i1 of
// one k = a 128-byte segment), so that the fused y/z pass finds every (i1, i2) plane contiguous; rows get one element of
// padding in shared memory (RS) to keep the row-fastest reads of that store pattern conflict-free.
// (Round 2, measured and removed: every CTA asking L2 -- prefetch.global.L2 -- for the rows of the tile 296 / 592 / 1184 blocks ahead,
// i.e. what a successor CTA on the same SM loads one CTA lifetime later: 0.57-0.59 ms instead of 0.53 ms at N = 120, 16 columns.)
// DIST = 1 (large-grid mode over peer memory): the input column is not local -- its i2 planes are slabs on the ranks of the job,
// read here through the IPC-mapped pointers of op.dist (a tile of rows lies in one plane, hence in one rank's slab); the tile is
// also copied to the local column cols.in[col], which the inverse x pass re-reads for the gamma K_B x + shift x term, so every
// element crosses NVLink once per direction.  The slab gather of the exchange path is fused into this pass.
// z-split forward x pass: three CTAs per SM (168 registers) where the first radix is at most 10 -- N = 160: 1.28 vs 1.35 ms per
// 16 columns, N = 128: 0.62 vs 0.68; with R1 = 12 (N = 144) the cap spills and loses (1.22 vs 1.10 ms)
#ifndef PCB_XFWD_ZS_CTAS
#define PCB_XFWD_ZS_CTAS 3
#endif
// ZS = 2 (with TRN): z-split plane mode, see ZSplit -- the tile's rows are 4 consecutive i1 of the planes i2' and i2' + N/2, and
// the radix-2 butterfly of the z transform is applied where the second radix step reads the exchange buffer.
template <class P, int LX, int NT, int SYM, int TRN = 0, int DIST = 0, int ZS = 1>
__global__ void __launch_bounds__(NT, (ZS == 2 ? (P::R1 <= 10 ? PCB_XFWD_ZS_CTAS : 1) : pcb_min_ctas(3 * LX * (P::R1 * P::R2P + TRN) * 16, P::R1, 4))) k_xfwd(PcbOp op, PcbCols cols, const cplx* __restrict__ tw) {
    constexpr int N = P::N, R1 = P::R1, R2 = P::R2, R2P = P::R2P;
    constexpr int RS = R1 * R2P + TRN;      // row stride in shared memory
    static_assert(ZS == 1 || (TRN == 1 && DIST == 0 && ZS == 2 && LX % 2 == 0 && N % (8 * ZS) == 0), "z-split: plane mode only");
    typedef ZSplit<P, ZS> ZSP;
    PCB_DYN_SMEM(cplx, sm);   // [3][LX][RS]
    const int col = blockIdx.y;
    const cplx* __restrict__ X = cols.in[col];
    cplx* __restrict__ Y = TRN ? cols.wrk[col] : cols.out[col];
    const long long nn = op.nn;
    const int row0 = blockIdx.x * LX;
    const int nrows = N * N;
    const int tid = threadIdx.x;
    const cplx* __restrict__ Xs = X;      // where the tile is read from, component stride cs
    long long cs = nn;
    cplx* __restrict__ Xc = nullptr;      // DIST: local copy of the column
    if (DIST) {
        const PcbDist* __restrict__ d = op.dist;
        const int i2t = row0 / N;
        int g = 0;
        while (g + 1 < d->world && i2t >= d->zb[g + 1]) ++g;
        cs = (long long)(d->zb[g + 1] - d->zb[g]) * N * N;
        Xs = d->src[col][g] - (long long)d->zb[g] * N * N;
        Xc = const_cast<cplx*>(X);
    }

    for (int item = tid; item < LX * R2; item += NT) {
        const int r = item / R2, n2 = item % R2;
        const int row = ZS == 1 ? row0 + r : ZSP::template row<LX>(blockIdx.x, r);
        if (row >= nrows) continue;
        const int i1 = row % N, i2 = row / N;
        cplx v[3][R1];
        cplx kc[3];
        if (SYM) {
            PCB_UNROLL
            for (int c = 0; c < 3; ++c) {
                const cplx b = __ldg(op.T + (c * 3 + 1) * N + i1);
                const cplx d = __ldg(op.T + (c * 3 + 2) * N + i2);
                kc[c] = cadd(b, d);
            }
        }
        PCB_UNROLL
        for (int n1 = 0; n1 < R1; ++n1) {
            const int i0 = n1 * R2 + n2;
            const long long e = (long long)row * N + i0;
            cplx x[3];
            PCB_UNROLL
            for (int c = 0; c < 3; ++c) x[c] = Xs[c * cs + e];
            if (DIST) {
                PCB_UNROLL
                for (int c = 0; c < 3; ++c) Xc[c * nn + e] = x[c];
            }
            if (SYM) {
                cplx a[3], z[3];
                PCB_UNROLL
                for (int c = 0; c < 3; ++c) {
                    const cplx k = cadd(kc[c], __ldg(op.T + (c * 3 + 0) * N + i0));
                    a[c] = cmake(-k.x, k.y);   // -conj(k)
                }
                pcb_cross(a, x, z);
                PCB_UNROLL
                for (int c = 0; c < 3; ++c) v[c][n1] = z[c];
            } else {
                PCB_UNROLL
                for (int c = 0; c < 3; ++c) v[c][n1] = x[c];
            }
        }
        PCB_UNROLL
        for (int c = 0; c < 3; ++c) {
            Dft<R1, -1>::run(v[c]);
            PCB_UNROLL
            for (int k1 = 0; k1 < R1; ++k1) {
                cplx val = v[c][k1];
                if (k1 > 0) val = cmul(val, __ldg(tw + k1 * R2 + n2));
                sm[(c * LX + r) * RS + k1 * R2P + n2] = val;
            }
        }
    }
    __syncthreads();
    for (int item = tid; item < 3 * LX * R1; item += NT) {
        const int k1 = TRN ? (item / LX) % R1 : item % R1;
        const int r = TRN ? item % LX : (item / R1) % LX;
        const int c = item / (R1 * LX);
        const int row = ZS == 1 ? row0 + r : ZSP::template row<LX>(blockIdx.x, r);
        if (row >= nrows) continue;
        cplx v[R2];
        if (ZS == 2) {      // E_h = (a + (-1)^h b) w_N^(h i2'): a, b = the rows of the planes i2', i2' + N/2 with this row's i1
            constexpr int LH = LX / 2;
            const int ra = r % LH, h = r / LH;
            const cplx* __restrict__ pa = sm + (c * LX + ra) * RS + k1 * R2P;
            const cplx wz = h ? __ldg(tw + N + N / 2 + (row / N - N / 2)) : cmake(1.0, 0.0);
            PCB_UNROLL
            for (int n2 = 0; n2 < R2; ++n2) {
                const cplx a = pa[n2], b = pa[LH * RS + n2];
                v[n2] = h ? cmul(csub(a, b), wz) : cadd(a, b);
            }
        } else {
            PCB_UNROLL
            for (int n2 = 0; n2 < R2; ++n2) v[n2] = sm[(c * LX + r) * RS + k1 * R2P + n2];
        }
        Dft<R2, -1>::run(v);
        if (TRN) {      // W'[c][k][i2][i1], k = k1 + R1*k2: consecutive threads = consecutive i1
            cplx* __restrict__ dst = Y + c * nn + (long long)k1 * N * N + row;      // row = i1 + N*i2
            PCB_UNROLL
            for (int k2 = 0; k2 < R2; ++k2) dst[(long long)R1 * k2 * N * N] = v[k2];
        } else {
            cplx* __restrict__ dst = Y + c * nn + (long long)row * N + k1;
            PCB_UNROLL
            for (int k2 = 0; k2 < R2; ++k2) dst[R1 * k2] = v[k2];
        }
    }
}

// Plane-mode forward x pass on TWO consecutive tiles per CTA (K_A^H on load, transposed store): the raw loads of the second
// tile are issued before the radix-R2 phase of the first, so a CTA has loads in flight for about a third of its life instead of a
// fifth (ncu of k_xfwd<T>: long_scoreboard 69 %, DRAM 61 %); the price is 3 instead of 4 CTAs per SM (24 complex values wait in
// registers through a phase that needs R2 more).  One phase-1 item per thread (LX R2 <= NT).
// (Longer chains -- 4, 8, 16 tiles per CTA with the same ping-pong -- spill 1.3-10 KB per thread whether the loop is unrolled
// or not and run at 0.85-0.91 ms; two tiles: 0.50 ms against 0.53 ms for k_xfwd<T> at N = 120, 16 columns.)
template <class P, int LX, int NT>
__global__ void __launch_bounds__(NT, 3) k_xfwd2(PcbOp op, PcbCols cols, const cplx* __restrict__ tw) {
    constexpr int N = P::N, R1 = P::R1, R2 = P::R2, R2P = P::R2P;
    constexpr int RS = R1 * R2P + 1;
    static_assert(LX * R2 <= NT, "one radix-R1 item per thread");
    PCB_DYN_SMEM(cplx, sm);   // [3][LX][RS]
    const int col = blockIdx.y;
    const cplx* __restrict__ X = cols.in[col];
    cplx* __restrict__ Y = cols.wrk[col];
    const long long nn = op.nn;
    const int nrows = N * N;
    const int tid = threadIdx.x;
    const int r = tid / R2, n2 = tid % R2;      // phase-1 item of this thread
    const bool has1 = tid < LX * R2;

    auto load_raw = [&](int row0, cplx (&x)[3][R1]) {
        const int row = row0 + r;
        if (has1 && row < nrows) {
            PCB_UNROLL
            for (int n1 = 0; n1 < R1; ++n1) {
                const long long e = (long long)row * N + n1 * R2 + n2;
                PCB_UNROLL
                for (int c = 0; c < 3; ++c) x[c][n1] = X[c * nn + e];
            }
        }
    };
    auto phase1 = [&](int row0, cplx (&x)[3][R1]) {      // (-conj k) x . on the loaded values, radix R1, twiddles -> shared memory
        const int row = row0 + r;
        if (!(has1 && row < nrows)) return;
        const int i1 = row % N, i2 = row / N;
        cplx kc[3];
        PCB_UNROLL
        for (int c = 0; c < 3; ++c) kc[c] = cadd(__ldg(op.T + (c * 3 + 1) * N + i1), __ldg(op.T + (c * 3 + 2) * N + i2));
        PCB_UNROLL
        for (int n1 = 0; n1 < R1; ++n1) {
            const int i0 = n1 * R2 + n2;
            cplx a[3], xin[3] = {x[0][n1], x[1][n1], x[2][n1]}, z[3];
            PCB_UNROLL
            for (int c = 0; c < 3; ++c) {
                const cplx k = cadd(kc[c], __ldg(op.T + (c * 3 + 0) * N + i0));
                a[c] = cmake(-k.x, k.y);
            }
            pcb_cross(a, xin, z);
            PCB_UNROLL
            for (int c = 0; c < 3; ++c) x[c][n1] = z[c];
        }
        PCB_UNROLL
        for (int c = 0; c < 3; ++c) {
            Dft<R1, -1>::run(x[c]);
            PCB_UNROLL
            for (int k1 = 0; k1 < R1; ++k1) {
                cplx val = x[c][k1];
                if (k1 > 0) val = cmul(val, __ldg(tw + k1 * R2 + n2));
                sm[(c * LX + r) * RS + k1 * R2P + n2] = val;
            }
        }
    };
    auto phase2 = [&](int row0) {      // radix R2 from shared memory, transposed store W'[c][k][i2][i1]
        for (int item = tid; item < 3 * LX * R1; item += NT) {
            const int k1 = (item / LX) % R1, rr = item % LX, c = item / (R1 * LX);
            const int row = row0 + rr;
            if (row >= nrows) continue;
            cplx v[R2];
            PCB_UNROLL
            for (int m2 = 0; m2 < R2; ++m2) v[m2] = sm[(c * LX + rr) * RS + k1 * R2P + m2];
            Dft<R2, -1>::run(v);
            cplx* __restrict__ dst = Y + c * nn + (long long)k1 * N * N + row;
            PCB_UNROLL
            for (int k2 = 0; k2 < R2; ++k2) dst[(long long)R1 * k2 * N * N] = v[k2];
        }
    };

    const int row0 = blockIdx.x * (2 * LX);
    cplx xa[3][R1], xb[3][R1];
    load_raw(row0, xa);
    phase1(row0, xa);
    load_raw(row0 + LX, xb);       // in flight during the radix-R2 phase of the first tile
    __syncthreads();
    phase2(row0);
    __syncthreads();
    phase1(row0 + LX, xb);
    __syncthreads();
    phase2(row0 + LX);
}

// ---------------------------------------------------------------------------------------
// Pass 5: x-lines inverse.  MODE 0: plain IFFT * 1/N^3;  1: A = K_A . ;  2: H = K_A . + gamma K_B x + shift x
// Reads the work column W (in Fourier-x order), the source column X (MODE 2) and writes OUT
// (OUT may alias W: each CTA only touches its own rows).
// ---------------------------------------------------------------------------------------
// DIST = 1 (large-grid mode over peer memory): the result rows go straight into the output column's slab on the rank that owns
// their i2 plane (IPC-mapped pointers of op.dist) -- the slab scatter of the exchange path fused into this pass; X is re-read
// from the local copy the forward pass left in cols.in[col].
#ifndef PCB_XINV_CTAS
#define PCB_XINV_CTAS 4
#endif
// ZS = 2 (with TRN): z-split plane mode (ZSplit) -- tiles as in k_xfwd<.., ZS = 2>; the epilogue recombines the two half planes,
// x[i2' + j N/2] = e[i2'] + (-1)^j conj(w_N^i2') o[i2'], while it reads the transformed tile.
// (z-split sizes: the uncapped kernel takes 170-172 registers, which the allocation granularity turns into TWO resident CTAs of four
// warps; asking for three caps it at 168.  Measured on one box: N = 128 (R1 = 8) 1.02 -> 0.91 ms per 16 columns, but N = 160 (R1 = 10)
// 1.97 -> 2.01 ms -- that pass is insensitive to occupancy, to the L2 prefetch of X and to the epilogue batch (PB = 2 / 4 / 8:
// 2.03 / 2.01 / 2.02 ms) -- so the cap applies where the first radix is 8.)
#ifndef PCB_XINV_ZS_CTAS
#define PCB_XINV_ZS_CTAS 3
#endif
template <class P, int LX, int NT, int MODE, int TRN = 0, int DIST = 0, int ZS = 1>
__global__ void __launch_bounds__(NT, (ZS == 2 ? (P::R1 <= 8 ? PCB_XINV_ZS_CTAS : 1) : pcb_min_ctas_inv(3 * LX * (P::R1 * P::R2P + TRN) * 16, P::R1, (TRN ? PCB_XINV_CTAS : 4)))) k_xinv(PcbOp op, PcbCols cols, const cplx* __restrict__ tw) {
    constexpr int N = P::N, R1 = P::R1, R2 = P::R2, R2P = P::R2P;
    constexpr int RS = R1 * R2P + TRN;      // row stride in shared memory (see k_xfwd)
    static_assert(ZS == 1 || (TRN == 1 && DIST == 0 && ZS == 2 && LX % 2 == 0 && N % (8 * ZS) == 0), "z-split: plane mode only");
    typedef ZSplit<P, ZS> ZSP;
    constexpr int LH = LX / ZS;             // z-split: the tile is ZS chunks of LH consecutive rows
    PCB_DYN_SMEM(cplx, sm);   // [3][LX][RS]
    const int col = blockIdx.y;
    const cplx* __restrict__ X = cols.in[col];
    cplx* __restrict__ W = cols.out[col];
    const cplx* __restrict__ WT = cols.wrk[col];      // TRN: transposed work column W'[c][k][i2][i1]
    const long long nn = op.nn;
    const int row0 = blockIdx.x * LX;
    const int nrows = N * N;
    const int nr = (nrows - row0 < LX) ? nrows - row0 : LX;      // rows of this tile
    const int tid = threadIdx.x;
    cplx* __restrict__ Wd = W;            // where the tile is stored, component stride cs
    long long cs = nn;
    if (DIST) {
        const PcbDist* __restrict__ d = op.dist;
        const int i2t = row0 / N;
        int g = 0;
        while (g + 1 < d->world && i2t >= d->zb[g + 1]) ++g;
        cs = (long long)(d->zb[g + 1] - d->zb[g]) * N * N;
        Wd = d->dst[col][g] - (long long)d->zb[g] * N * N;
    }

    if (MODE == 2 && ZS == 1) {   // the epilogue re-reads X: pull this tile's lines (3 contiguous chunks) towards L2 now
        const int lines = (nr * N * (int)sizeof(cplx) + 127) / 128;
        for (int l = tid; l < 3 * lines; l += NT)
            pcb_prefetch_l2(reinterpret_cast<const char*>(X + (l / lines) * nn + (long long)row0 * N) + (l % lines) * 128);
    }
    if (MODE == 2 && ZS == 2) {   // ... 3 x ZS chunks of LH rows
        constexpr int lines = (LH * N * (int)sizeof(cplx) + 127) / 128;
        for (int l = tid; l < 3 * ZS * lines; l += NT) {
            const int ch = l / lines;
            pcb_prefetch_l2(reinterpret_cast<const char*>(X + (ch / ZS) * nn + (long long)ZSP::template row<LX>(blockIdx.x, (ch % ZS) * LH) * N) + (l % lines) * 128);
        }
    }
    // inverse radix R2 over k2 (fixed k1): global (Fourier order, k = k1 + R1*k2) -> registers -> shared
    for (int item = tid; item < 3 * LX * R1; item += NT) {
        const int k1 = TRN ? (item / LX) % R1 : item % R1;
        const int r = TRN ? item % LX : (item / R1) % LX;
        const int c = item / (R1 * LX);
        const int cr = c * LX + r;
        if (r >= nr) continue;
        cplx v[R2];
        if (TRN) {
            const cplx* __restrict__ src = WT + c * nn + (long long)k1 * N * N + (ZS == 1 ? row0 + r : ZSP::template row<LX>(blockIdx.x, r));
            PCB_UNROLL
            for (int k2 = 0; k2 < R2; ++k2) v[k2] = src[(long long)R1 * k2 * N * N];
        } else {
            const cplx* __restrict__ src = W + c * nn + (long long)(row0 + r) * N + k1;
            PCB_UNROLL
            for (int k2 = 0; k2 < R2; ++k2) v[k2] = src[R1 * k2];
        }
        Dft<R2, +1>::run(v);
        PCB_UNROLL
        for (int n2 = 0; n2 < R2; ++n2) {
            cplx val = v[n2];
            if (k1 > 0) { const cplx t = __ldg(tw + k1 * R2 + n2); val = cmul(val, cmake(t.x, -t.y)); }
            sm[cr * RS + k1 * R2P + n2] = val;
        }
    }
    __syncthreads();
    // inverse radix R1 over k1 (fixed n2), in place: slot (n1, n2) <-> i0 = n1*R2 + n2
    for (int item = tid; item < 3 * LX * R2; item += NT) {
        const int n2 = item % R2, cr = item / R2;
        if (cr % LX >= nr) continue;
        cplx v[R1];
        PCB_UNROLL
        for (int k1 = 0; k1 < R1; ++k1) v[k1] = sm[cr * RS + k1 * R2P + n2];
        Dft<R1, +1>::run(v);
        PCB_UNROLL
        for (int n1 = 0; n1 < R1; ++n1) sm[cr * RS + n1 * R2P + n2] = v[n1];
    }
    __syncthreads();
    // point-wise epilogue, fully coalesced: 1/N^3, k x v, (+ gamma conj(k)(k.x) + shift x), store
#ifndef PCB_XINV_PB
#define PCB_XINV_PB 4
#endif
    constexpr int PB = PCB_XINV_PB;     // points per thread and batch: all X loads of a batch are issued before they are used
    // global position of tile element e (row-major over the tile's rows): contiguous from row0 N, or ZS chunks of LH rows
    auto gpos = [&](int e) -> long long {
        return ZS == 1 ? (long long)row0 * N + e : (long long)ZSP::template row<LX>(blockIdx.x, (e / (LH * N)) * LH) * N + e % (LH * N);
    };
    for (int e0 = tid; e0 < nr * N; e0 += PB * NT) {
        cplx x[PB][3];
        if (MODE == 2) {
            PCB_UNROLL
            for (int q = 0; q < PB; ++q) {
                const int e = e0 + q * NT;
                if (e < nr * N) {
                    const long long g = gpos(e);
                    PCB_UNROLL
                    for (int c = 0; c < 3; ++c) x[q][c] = X[c * nn + g];
                }
            }
        }
        PCB_UNROLL
        for (int q = 0; q < PB; ++q) {
            const int e = e0 + q * NT;
            if (e >= nr * N) continue;
            const int r = e / N, i0 = e % N;
            const int row = ZS == 1 ? row0 + r : ZSP::template row<LX>(blockIdx.x, r);
            const int slot = (ZS == 1 ? r : r % LH) * RS + (i0 / R2) * R2P + i0 % R2;
            cplx u[3], z[3];
            if (ZS == 2) {      // x[i2' + j N/2] = e + (-1)^j conj(w_N^i2') o
                const int j = r / LH;
                const cplx t = __ldg(tw + N + N / 2 + (row / N - j * (N / 2)));
                const cplx wc = j ? cmake(-t.x, t.y) : cmake(t.x, -t.y);
                PCB_UNROLL
                for (int c = 0; c < 3; ++c) u[c] = cscale(cfma(wc, sm[(c * LX + LH) * RS + slot], sm[c * LX * RS + slot]), op.inv_n3);
            } else {
                PCB_UNROLL
                for (int c = 0; c < 3; ++c) u[c] = cscale(sm[c * LX * RS + slot], op.inv_n3);
            }
            if (MODE) {
                const Sym3 sy = pcb_symbol(op.T, N, i0, row % N, row / N);
                pcb_cross(sy.k, u, z);
                if (MODE == 2) {
                    // gamma K_B x = gamma conj(k) (k . x)   (h_block with D_B, pcfft.py:176)
                    cplx dot = cadd(cadd(cmul(sy.k[0], x[q][0]), cmul(sy.k[1], x[q][1])), cmul(sy.k[2], x[q][2]));
                    dot = cscale(dot, op.gamma);
                    PCB_UNROLL
                    for (int c = 0; c < 3; ++c) {
                        cplx t = cfmac(sy.k[c], dot, z[c]);
                        t.x = fma(op.shift, x[q][c].x, t.x);
                        t.y = fma(op.shift, x[q][c].y, t.y);
                        z[c] = t;
                    }
                }
            } else {
                PCB_UNROLL
                for (int c = 0; c < 3; ++c) z[c] = u[c];
            }
            const long long g = gpos(e);
            PCB_UNROLL
            for (int c = 0; c < 3; ++c) Wd[c * cs + g] = z[c];
        }
    }
}

// (Round 2, measured and removed: the inverse x pass on two consecutive tiles per CTA, the counterpart of k_xfwd2 -- the second
// tile's scattered radix-R2 loads issued before the first tile's point-wise epilogue.  The 15 complex values waiting through an
// epilogue that itself holds 4 x 3 X values spill 450-670 bytes at 3 CTAs per SM: 0.871 vs 0.693 ms at N = 120, 16 columns.)

// ---------------------------------------------------------------------------------------
// Passes 2/4 (and the split z passes of the cross-DoF variant): strided lines, in place.
// DIM 1: lines along i1 (tile = 8 i0 x one i2);  DIM 2: lines along i2 (tile = 8 i0 x one i1).
// A CTA handles the three components of one tile.
// ---------------------------------------------------------------------------------------
template <class P, int DIM, int DIR, int NT>
__global__ void __launch_bounds__(NT) k_line(PcbOp op, PcbCols cols, const cplx* __restrict__ tw) {
    constexpr int N = P::N, R1 = P::R1, R2 = P::R2;
    PCB_DYN_SMEM(cplx, sm);   // [3][N][8]
    const int col = blockIdx.y;
    cplx* __restrict__ Y = cols.out[col];
    const long long nn = op.nn;
    constexpr int NT0 = (N + 7) / 8;
    const int t0 = blockIdx.x % NT0, other = blockIdx.x / NT0;
    const long long sline = (DIM == 1) ? N : (long long)N * N;
    const long long sother = (DIM == 1) ? (long long)N * N : N;
    const int tid = threadIdx.x;

    for (int item = tid; item < 3 * R2 * 8; item += NT) {
        const int i0l = item % 8, n2 = (item / 8) % R2, c = item / (8 * R2);
        const int i0 = t0 * 8 + i0l;
        if (i0 >= N) continue;
        cplx* __restrict__ base = Y + c * nn + other * sother + i0;
        cplx v[R1];
        PCB_UNROLL
        for (int n1 = 0; n1 < R1; ++n1) v[n1] = base[P::lin(n1, n2) * sline];
        Dft<R1, DIR>::run(v);
        PCB_UNROLL
        for (int k1 = 0; k1 < R1; ++k1) {
            cplx val = v[k1];
            if (!P::PFA && k1 > 0) {
                const cplx t = __ldg(tw + k1 * R2 + n2);
                val = cmul(val, cmake(t.x, DIR < 0 ? t.y : -t.y));
            }
            sm[(c * N + k1 * R2 + n2) * 8 + i0l] = val;
        }
    }
    __syncthreads();
    for (int item = tid; item < 3 * R1 * 8; item += NT) {
        const int i0l = item % 8, k1 = (item / 8) % R1, c = item / (8 * R1);
        const int i0 = t0 * 8 + i0l;
        if (i0 >= N) continue;
        cplx v[R2];
        PCB_UNROLL
        for (int n2 = 0; n2 < R2; ++n2) v[n2] = sm[(c * N + k1 * R2 + n2) * 8 + i0l];
        Dft<R2, DIR>::run(v);
        cplx* __restrict__ base = Y + c * nn + other * sother + i0;
        PCB_UNROLL
        for (int k2 = 0; k2 < R2; ++k2) base[P::lout(k1, k2) * sline] = v[k2];
    }
}

// Point-wise dielectric multiply on the three components at one grid point (real space).
// chiral: rows in Omega_1 scaled by 1/eps (discretization.py:352-366); trivial: Hermitian 3x3
// with diagonal eps_cc on edge DoFs and off-diagonals on the cell's volume DoF (:368-401).
PCB_HD void pcb_diel_point(const PcbOp& op, unsigned m, cplx u[3]) {
    const double d0 = (m & 1u) ? op.ediag[0] : 1.0;
    const double d1 = (m & 2u) ? op.ediag[1] : 1.0;
    const double d2 = (m & 4u) ? op.ediag[2] : 1.0;
    cplx y0 = cscale(u[0], d0), y1 = cscale(u[1], d1), y2 = cscale(u[2], d2);
    if (m & 8u) {
        y0 = cfma(op.eoff[0], u[1], cfma(op.eoff[1], u[2], y0));
        y1 = cfmac(op.eoff[0], u[0], cfma(op.eoff[2], u[2], y1));
        y2 = cfmac(op.eoff[1], u[0], cfmac(op.eoff[2], u[1], y2));
    }
    u[0] = y0; u[1] = y1; u[2] = y2;
}

// Materials dielectric (PCB_DIEL_MATERIALS): M is diagonal, (M x)_r = inv_eps[mat[r]] x_r.  In the plane pass each z item's ZR2
// index bytes are stored padded to pcb_mat_pad(ZR2) bytes (k_mat_bytes), so that one aligned vector load of ZP / 4 words fetches
// them; the 2 KB table of 1 / eps is read through __ldg and stays L1-resident (the plane leaves no room for it in shared memory).
PCB_HD constexpr int pcb_mat_pad(int r2) { return r2 <= 4 ? 4 : (r2 <= 8 ? 8 : 16); }
template <int W>
PCB_D void pcb_ldg_words(unsigned* w, const unsigned char* __restrict__ p) {
#ifdef PCB_EMU
    memcpy(w, p, 4 * W);
#else
    if constexpr (W == 4) { const uint4 u = __ldg(reinterpret_cast<const uint4*>(p)); w[0] = u.x; w[1] = u.y; w[2] = u.z; w[3] = u.w; }
    else if constexpr (W == 2) { const uint2 u = __ldg(reinterpret_cast<const uint2*>(p)); w[0] = u.x; w[1] = u.y; }
    else w[0] = __ldg(reinterpret_cast<const unsigned*>(p));
#endif
}
// v[k] *= inv_eps[index byte k of the packed words w]
template <int R>
PCB_D void pcb_mat_scale(const PcbOp& op, const unsigned* w, cplx* v) {
    PCB_UNROLL
    for (int k = 0; k < R; ++k) v[k] = cscale(v[k], __ldg(op.inv_eps + ((w[k / 4] >> (8 * (k % 4))) & 0xffu)));
}

// ---------------------------------------------------------------------------------------
// Pass 3: z-lines: forward FFT, dielectric multiply M in real space, inverse FFT; in place.
// DIEL: 0 identity, 1 component-wise (chiral), 2 coupled 3x3 at a point (trivial), 4 materials (index bytes gathered per item).
// Persistent CTAs; tile = 8 consecutive i0 x one i1, all i2, three components (3*N segments of 128 B), streamed into
// one of two shared-memory stages with cp.async while the previous tile is transformed.  The line element with
// digits (a, b) always lives in slot P::lin(a, b) of its stage, so all four radix steps exchange in place.
// ---------------------------------------------------------------------------------------
template <class P, int NT>
PCB_D void pcb_ztile_load(cplx* __restrict__ st, const cplx* __restrict__ Y, long long nn, int t0, int i1, int tid) {
    constexpr int N = P::N;
    const int i0l = tid % 8, i0 = t0 * 8 + i0l;
    if (i0 >= N) return;
    const cplx* __restrict__ src = Y + (long long)i1 * N + i0;
    PCB_UNROLL
    for (int c = 0; c < 3; ++c)
        for (int i2 = tid / 8; i2 < N; i2 += NT / 8)
            pcb_cp16(st + (c * N + i2) * 8 + i0l, src + c * nn + (long long)i2 * N * N);
}

// NSTAGE = 2: the next tile streams into the other stage while this one is transformed; NSTAGE = 1 (large N, where two stages
// would leave one CTA per SM): load, wait, transform in the single stage and rely on the co-resident CTAs for overlap.
template <class P, int DIEL, int NT, int NSTAGE = 2>
__global__ void __launch_bounds__(NT, (NT > 256 ? 1 : 2)) k_zmid(PcbOp op, PcbCols cols, const cplx* __restrict__ tw, int ncols) {
    constexpr int N = P::N, R1 = P::R1, R2 = P::R2;
    constexpr int STAGE = 3 * N * 8;
    PCB_DYN_SMEM(cplx, sm);   // [NSTAGE][3][N][8]
    const long long nn = op.nn;
    constexpr int NT0 = (N + 7) / 8;
    const int tpc = NT0 * N;
    const int total = tpc * ncols;
    const int tid = threadIdx.x;

    int tile = blockIdx.x, stage = 0;
    if (NSTAGE == 2 && tile < total) {
        pcb_ztile_load<P, NT>(sm, cols.out[tile / tpc], nn, (tile % tpc) % NT0, (tile % tpc) / NT0, tid);
        pcb_cp_commit();
    }
    for (; tile < total; tile += gridDim.x) {
        const int next = tile + gridDim.x;
        if (NSTAGE == 1) {
            pcb_ztile_load<P, NT>(sm, cols.out[tile / tpc], nn, (tile % tpc) % NT0, (tile % tpc) / NT0, tid);
            pcb_cp_commit();
            pcb_cp_wait<0>();
        } else if (next < total) {
            pcb_ztile_load<P, NT>(sm + (stage ^ 1) * STAGE, cols.out[next / tpc], nn, (next % tpc) % NT0, (next % tpc) / NT0, tid);
            pcb_cp_commit();
            pcb_cp_wait<1>();
        } else {
            pcb_cp_wait<0>();
        }
        const int t0 = (tile % tpc) % NT0, i1 = (tile % tpc) / NT0;
        // dielectric bits of this thread's radix-R2 items (bit k2 = component c of point (i0, i1, i2 = lout(k1,k2)) in Omega_1),
        // fetched before the barrier so that the mask latency hides behind the tile load and the first radix step
        constexpr int ZI = (3 * R1 * 8 + NT - 1) / NT;
        unsigned mbits[ZI];
        if (DIEL == 1) {
            PCB_UNROLL
            for (int q = 0; q < ZI; ++q) {
                const int item = tid + NT * q;
                unsigned w = 0u;
                const int i0 = t0 * 8 + item % 8;
                if (item < 3 * R1 * 8 && i0 < N) {
                    const int o1 = P::lout1((item / 8) % R1), cc = item / (8 * R1);
                    const unsigned char* __restrict__ mp = op.mask + (long long)i1 * N + i0;
                    PCB_UNROLL
                    for (int k2 = 0; k2 < R2; ++k2) w |= ((unsigned)(__ldg(mp + P::wrap(o1 + P::lout2(k2)) * (N * N)) >> cc) & 1u) << k2;
                }
                mbits[q] = w;
            }
        }
        __syncthreads();
        cplx* __restrict__ st = sm + stage * STAGE;
        cplx* __restrict__ Y = cols.out[tile / tpc];

        // forward radix R1 over n1 (fixed n2)
        for (int item = tid; item < 3 * R2 * 8; item += NT) {
            const int i0l = item % 8, n2 = (item / 8) % R2, c = item / (8 * R2);
            if (t0 * 8 + i0l >= N) continue;
            cplx* __restrict__ sc = st + c * N * 8 + i0l;
            const int b2 = P::lin2(n2);
            cplx v[R1];
            PCB_UNROLL
            for (int n1 = 0; n1 < R1; ++n1) v[n1] = sc[P::wrap(P::lin1(n1) + b2) * 8];
            Dft<R1, -1>::run(v);
            PCB_UNROLL
            for (int k1 = 0; k1 < R1; ++k1) {
                cplx val = v[k1];
                if (!P::PFA && k1 > 0) val = cmul(val, __ldg(tw + k1 * R2 + n2));
                sc[P::wrap(P::lin1(k1) + b2) * 8] = val;
            }
        }
        __syncthreads();
        // forward radix R2 (-> real space), M, inverse radix R2
        if (DIEL == 2) {
            // coupled 3x3 M: the three components of a point meet in shared memory.  Per-component radix items (as for the
            // other dielectrics, v[R2] registers instead of v[3][R2]) around a point-wise phase; the real-space value with
            // digits (k1, k2) sits in slot lin(k1, k2) and belongs to grid index i2 = lout(k1, k2).
            for (int item = tid; item < 3 * R1 * 8; item += NT) {
                const int i0l = item % 8, k1 = (item / 8) % R1, c = item / (8 * R1);
                if (t0 * 8 + i0l >= N) continue;
                const int b1 = P::lin1(k1);
                cplx* __restrict__ sc = st + c * N * 8 + i0l;
                cplx v[R2];
                PCB_UNROLL
                for (int n2 = 0; n2 < R2; ++n2) v[n2] = sc[P::wrap(b1 + P::lin2(n2)) * 8];
                Dft<R2, -1>::run(v);
                PCB_UNROLL
                for (int k2 = 0; k2 < R2; ++k2) sc[P::wrap(b1 + P::lin2(k2)) * 8] = v[k2];
            }
            __syncthreads();
            for (int e = tid; e < N * 8; e += NT) {
                const int i0l = e % 8, slot = e / 8;
                const int i0 = t0 * 8 + i0l;
                if (i0 >= N) continue;
                const int i2 = P::coord(slot);
                const unsigned mk = __ldg(op.mask + ((long long)i2 * N + i1) * N + i0);
                cplx u[3] = {st[slot * 8 + i0l], st[(N + slot) * 8 + i0l], st[(2 * N + slot) * 8 + i0l]};
                pcb_diel_point(op, mk, u);
                st[slot * 8 + i0l] = u[0]; st[(N + slot) * 8 + i0l] = u[1]; st[(2 * N + slot) * 8 + i0l] = u[2];
            }
            __syncthreads();
            for (int item = tid; item < 3 * R1 * 8; item += NT) {
                const int i0l = item % 8, k1 = (item / 8) % R1, c = item / (8 * R1);
                if (t0 * 8 + i0l >= N) continue;
                const int b1 = P::lin1(k1);
                cplx* __restrict__ sc = st + c * N * 8 + i0l;
                cplx v[R2];
                PCB_UNROLL
                for (int k2 = 0; k2 < R2; ++k2) v[k2] = sc[P::wrap(b1 + P::lin2(k2)) * 8];
                Dft<R2, +1>::run(v);
                PCB_UNROLL
                for (int n2 = 0; n2 < R2; ++n2) {
                    cplx val = v[n2];
                    if (!P::PFA && k1 > 0) { const cplx t = __ldg(tw + k1 * R2 + n2); val = cmul(val, cmake(t.x, -t.y)); }
                    sc[P::wrap(b1 + P::lin2(n2)) * 8] = val;
                }
            }
        } else {
            PCB_UNROLL
            for (int q = 0; q < ZI; ++q) {
                const int item = tid + NT * q;
                if (item >= 3 * R1 * 8) break;
                const int i0l = item % 8, k1 = (item / 8) % R1, c = item / (8 * R1);
                const int i0 = t0 * 8 + i0l;
                if (i0 >= N) continue;
                const int b1 = P::lin1(k1);
                cplx* __restrict__ sc = st + c * N * 8 + i0l;
                // materials: the item's R2 index bytes gathered from the natural-order map and packed four to a word, issued ahead
                // of the column loads and the radix step (gathered before the barrier as the chiral bits are, the ZI x R2 / 4 words
                // spill from N = 120 on)
                constexpr int MW = (DIEL == 4) ? (R2 + 3) / 4 : 1;
                unsigned mw[MW];
                if (DIEL == 4) {
                    PCB_UNROLL
                    for (int w = 0; w < MW; ++w) mw[w] = 0u;
                    const unsigned char* __restrict__ mp = op.mat + c * nn + (long long)i1 * N + i0;
                    const int o1 = P::lout1(k1);      // real-space digits (k1, k2) belong to grid index i2 = lout(k1, k2)
                    PCB_UNROLL
                    for (int k2 = 0; k2 < R2; ++k2) mw[k2 / 4] |= (unsigned)__ldg(mp + P::wrap(o1 + P::lout2(k2)) * (N * N)) << (8 * (k2 % 4));
                }
                cplx v[R2];
                PCB_UNROLL
                for (int n2 = 0; n2 < R2; ++n2) v[n2] = sc[P::wrap(b1 + P::lin2(n2)) * 8];
                Dft<R2, -1>::run(v);
                if (DIEL == 1) {
                    const double scl = op.ediag[c];
                    const unsigned w = mbits[q];
                    PCB_UNROLL
                    for (int k2 = 0; k2 < R2; ++k2) v[k2] = cscale(v[k2], ((w >> k2) & 1u) ? scl : 1.0);   // branch-free
                }
                if (DIEL == 4) pcb_mat_scale<R2>(op, mw, v);
                Dft<R2, +1>::run(v);
                PCB_UNROLL
                for (int n2 = 0; n2 < R2; ++n2) {
                    cplx val = v[n2];
                    if (!P::PFA && k1 > 0) { const cplx t = __ldg(tw + k1 * R2 + n2); val = cmul(val, cmake(t.x, -t.y)); }
                    sc[P::wrap(b1 + P::lin2(n2)) * 8] = val;
                }
            }
        }
        __syncthreads();
        // inverse radix R1 and store
        for (int item = tid; item < 3 * R2 * 8; item += NT) {
            const int i0l = item % 8, n2 = (item / 8) % R2, c = item / (8 * R2);
            const int i0 = t0 * 8 + i0l;
            if (i0 >= N) continue;
            const cplx* __restrict__ sc = st + c * N * 8 + i0l;
            const int b2 = P::lin2(n2);
            cplx v[R1];
            PCB_UNROLL
            for (int k1 = 0; k1 < R1; ++k1) v[k1] = sc[P::wrap(P::lin1(k1) + b2) * 8];
            Dft<R1, +1>::run(v);
            cplx* __restrict__ base = Y + c * nn + (long long)i1 * N + i0;
            PCB_UNROLL
            for (int n1 = 0; n1 < R1; ++n1) base[(long long)P::wrap(P::lin1(n1) + b2) * (N * N)] = v[n1];
        }
        __syncthreads();
        if (NSTAGE == 2) stage ^= 1;
    }
}

// Plane mode set-up (once per dielectric): mbits[c][i0][slot][k1], bit k2 = "component c of grid point
// (i0, i1 = coord(slot), i2 = lout(k1, k2)) lies in Omega_1" -- exactly the 15 (R2) flags one radix-R2 item of k_mid needs.
template <class P, int ZS = 1>
__global__ void k_mask_bits(PcbOp op, unsigned* __restrict__ out) {
    // z-split (ZS = 2): mbits[c][i0][slot][h][k1], bit k2 = (i0, i1 = coord(slot), i2 = ZS lout_z(k1, k2) + h), digits of the plan of N / ZS
    typedef typename ZSplit<P, ZS>::PZ PZ;
    constexpr int N = P::N, R1 = PZ::R1, R2 = PZ::R2;
    const long long total = 3LL * N * N * ZS * R1;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const int k1 = (int)(t % R1), h = (int)((t / R1) % ZS), slot = (int)((t / (R1 * ZS)) % N), i0 = (int)((t / ((long long)R1 * ZS * N)) % N),
              c = (int)(t / ((long long)R1 * ZS * N * N));
    const int i1 = P::coord(slot), o1 = PZ::lout1(k1);
    unsigned w = 0u;
    for (int k2 = 0; k2 < R2; ++k2) {
        const int i2 = ZS * PZ::wrap(o1 + PZ::lout2(k2)) + h;
        w |= ((unsigned)(op.mask[((long long)i2 * N + i1) * N + i0] >> c) & 1u) << k2;
    }
    out[t] = w;
}
// The same for the materials dielectric: matp[item t of k_mask_bits][k2] = mat[c nn + (i2 N + i1) N + i0], the ZR2 index bytes of
// the item padded with zeros to pcb_mat_pad(ZR2)
template <class P, int ZS = 1>
__global__ void k_mat_bytes(PcbOp op, unsigned char* __restrict__ out) {
    typedef typename ZSplit<P, ZS>::PZ PZ;
    constexpr int N = P::N, R1 = PZ::R1, R2 = PZ::R2, ZP = pcb_mat_pad(R2);
    const long long total = 3LL * N * N * ZS * R1;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const int k1 = (int)(t % R1), h = (int)((t / R1) % ZS), slot = (int)((t / (R1 * ZS)) % N), i0 = (int)((t / ((long long)R1 * ZS * N)) % N),
              c = (int)(t / ((long long)R1 * ZS * N * N));
    const int i1 = P::coord(slot), o1 = PZ::lout1(k1);
    for (int k2 = 0; k2 < ZP; ++k2) {
        const int i2 = ZS * PZ::wrap(o1 + PZ::lout2(k2 < R2 ? k2 : 0)) + h;
        out[t * ZP + k2] = k2 < R2 ? op.mat[c * op.nn + ((long long)i2 * N + i1) * N + i0] : (unsigned char)0;
    }
}

// ---------------------------------------------------------------------------------------
// Plane mode, pass 2 of 3: forward y, forward z, M, inverse z, inverse y on one (i1, i2) plane held in shared memory.
// (Measured alternative, B200, N = 120, 16 columns: moving the radix-8 step of the y transform into the x passes -- whose
// thread mapping already holds a tile's 8 rows in 8 adjacent lanes, so the step is three shuffle butterflies per value --
// takes this kernel from 0.90 to 0.745 ms (five shared-memory sweeps instead of seven), but the 180 SHFL per thread-item cost
// the x passes more: 0.53 -> 0.72 ms and 0.70 -> 0.82 ms, 2.27 ms per apply instead of 2.09.  Reverted; git history has it.)
// The x pass wrote the transposed layout W'[c][i0][i2][i1], so the plane of (c, i0) is one contiguous chunk of N^2 elements;
// a CTA (N/8 warps, one per SM, persistent) keeps it in shared memory with row stride N+1 (row-fastest accesses of the y
// steps stay conflict-free; N = 120: 232 320 B of the 232 448 B a CTA can have).  Warp w owns rows i2 in [8w, 8w+8) for the
// y steps and slots i1 in [8w, 8w+8) for the z steps, so only two CTA-wide barriers per plane are needed (row -> column
// ownership and back); loading, the y steps and storing of different warps overlap each other.  HBM traffic of the whole
// operator drops from 11 to 7 column transfers per op-apply.  DIEL: 0 identity, 1 component-wise (chiral), 4 materials; the coupled
// 3x3 dielectrics need all three components of a point and stay on the five-pass path.
// ---------------------------------------------------------------------------------------
// TMA = 1 (the device build): the rows of a plane are moved by bulk copies -- cp.async.bulk, one elected lane per warp
// issues eight row copies against the warp's own mbarrier; the store goes back the same way after a proxy fence -- instead
// of per-element cp.async / LDS + STG loops: 960 LDGSTS and 960 LDS+STG per warp and plane leave the LSU queue, which the
// radix steps need (N = 120, 16 columns: 0.884 -> 0.818 ms).  TMA = 0, the loop form, is what the host-emulation build runs.
// (Round 2, measured and removed: the radix-R1 steps with two items per lane in flight -- either both loaded before both
// butterflies, or software-pipelined so that item i+1's loads go out before item i's stores; the shared-memory plane carries no
// restrict information, so the compiler keeps each trip's loads behind the previous trip's stores.  At the 128-register cap of
// 15 warps either form spills 400-800 bytes per thread and the pass takes 1.17 instead of 0.82 ms at N = 120, 16 columns.)
// Cross-DoF dielectric (discretization.py:403-453) on the PLANE-SLOT layout, one output component at one point: the
// off-diagonal part  sum_b eps_cb (S_cb x_b)(p)  with S_ab = (I_a T_ab + T_ab I_b)/2, T_ab = c (x) c^T on two axes (2k taps each).
// X: a column in the slot layout W'[c][i0][row][col] (point (i0, coord(col), coord(row))), maskp the byte mask in the same
// order, ctab the slot <-> index tables.  i[] = grid indices of the point, mp = its mask byte.
// (N and the stencil half-width are compile-time here and all index arithmetic is 32-bit with conditional wraps: written with
// runtime N, 64-bit indices and % the ~1000 instructions per coupled point made the fused pass issue-bound -- 1.33 ms instead of
// the 1.19 ms of the two separate kernels at N = 120.)
// `live` = false: nothing is loaded (predicated loads) and zero comes back -- lets the caller batch several points per trip.
template <int N, int K>
PCB_D cplx pcb_crossdof_couple(const PcbOp& op, int c, const int i[3], unsigned mp, const cplx* __restrict__ X, bool live = true) {
    const int nn = N * N * N;
    const int* __restrict__ ctab = op.ctab;
    const unsigned char* __restrict__ maskp = op.maskp;
    constexpr int PA[3] = {0, 0, 1}, PB[3] = {1, 2, 2}, CAX[3] = {2, 2, 1}, TAX[3] = {1, 0, 0};
    const int kk = K > 0 ? K : op.sten.k;
    cplx out = cmake(0.0, 0.0);
    const double Ic = (double)((mp >> c) & 1u);
    PCB_UNROLL
    for (int pr = 0; pr < 3; ++pr) {
        const cplx e = op.eoff[pr];
        const int a = PA[pr], b = PB[pr], cax = CAX[pr], tax = TAX[pr];
        if ((c != a && c != b) || (e.x == 0.0 && e.y == 0.0)) continue;
        const bool first = (c == a);                 // y_a += e S x_b   |   y_b += conj(e) S^T x_a
        const int other = first ? b : a;
        const cplx* __restrict__ Xo = X + other * nn;
        cplx sacc = cmake(0.0, 0.0);
#ifndef PCB_EMU
#pragma unroll
#endif
        for (int j1 = 0; j1 < (K > 0 ? 2 * K : 2 * kk); ++j1) {
            const int oc = first ? 1 - kk + j1 : -(1 - kk + j1);
            int qc = i[cax] + oc;
            qc += (qc < 0) ? N : 0; qc -= (qc >= N) ? N : 0;
            // slot-layout position contributed by the c-axis index (axis 0: plane, 1: column, 2: row)
            const int pc = cax == 0 ? qc * (N * N) : (cax == 1 ? __ldg(ctab + N + qc) : __ldg(ctab + 3 * N + qc) * N);
#ifndef PCB_EMU
#pragma unroll
#endif
            for (int j2 = 0; j2 < (K > 0 ? 2 * K : 2 * kk); ++j2) {
                const int ot = first ? -(1 - kk + j2) : 1 - kk + j2;
                int qt = i[tax] + ot;
                qt += (qt < 0) ? N : 0; qt -= (qt >= N) ? N : 0;
                const int pt = tax == 0 ? qt * (N * N) : (tax == 1 ? __ldg(ctab + N + qt) : __ldg(ctab + 3 * N + qt) * N);
                // the third axis keeps the point's own index
                const int rest = 3 - cax - tax;
                const int po = rest == 0 ? i[0] * (N * N) : (rest == 1 ? __ldg(ctab + N + i[1]) : __ldg(ctab + 3 * N + i[2]) * N);
                const int qs = pc + pt + po;
                const double w = op.sten.w[j1] * op.sten.w[j2] * 0.5;
                const unsigned mq = live ? (unsigned)__ldg(maskp + qs) : 0u;
                const cplx xq = live ? Xo[qs] : cmake(0.0, 0.0);
                const double Io = (double)((mq >> other) & 1u);
                sacc = cadd(sacc, cscale(xq, w * (Ic + Io)));
            }
        }
        out = first ? cfma(e, sacc, out) : cfmac(e, sacc, out);
    }
    return out;
}

// DIEL = 2 (coupled 3x3 point-wise M, discretization.py:368-401): the kernel is launched as CLUSTERS OF THREE CTAs, one per
// component of the same (column, i0) plane.  The fused z step is split at real space: (A) forward radix R2 and the diagonal
// entries (bit words as for DIEL = 1) -> own plane; cluster barrier; (B) every CTA takes a third of the rows and, at the
// points whose volume DoF lies in Omega_1 (byte mask in plane-slot order, k_mask_plane), reads the three components -- one
// local, two through distributed shared memory --, adds the off-diagonal terms and writes all three back; cluster barrier;
// (C) inverse radix R2.  With u~ = D u stored by (A), y_a = u~_a + sum_b eps_ab (u~_b / d_b).  Only the coupled points cross
// the SM-to-SM network (bcc gyroids: 10-20 % of the cells), so the 3x3 dielectric costs one extra shared-memory sweep
// and two cluster barriers per plane instead of the two extra global passes of the five-pass structure.
// HALF = 1 / 2: only the forward (y, z) / inverse (z, y) transforms of the plane, M left out -- the cross-DoF dielectric is a
// stencil across planes and runs as its own kernel on the real-space planes in between (k_diel_crossdof_t, pcb_block.cuh).
// HALF = 2 loads from cols.out (the stencil's output) and stores to cols.wrk.
// STEN (with the halves): the stencil is FUSED into the inverse half instead -- HALF = 1 then stores its real-space planes to
// cols.out, and HALF = 2, once a warp's rows have landed, applies M to them in shared memory: the diagonal entry, and at the
// points flagged by k_mask_active (a quarter of the cells for the gyroids) the coupling terms, whose taps it gathers from the
// real-space planes of the other components in cols.out (same or neighbouring i0; L2 hits, the planes of a wave of CTAs are
// adjacent).  Four kernels, 9 column transfers instead of five kernels / 11.  STEN = 2 * K + 1 encodes the stencil half-width
// K at compile time (K = 1, 2), STEN = 1 reads it from op.sten.
// ZS = 2: z-split plane mode (ZSplit) -- the CTA holds a HALF plane of NZ = N/2 rows (plane rows h NZ .. h NZ + NZ - 1) and N
// columns; NZ / 8 warps own 8 rows each in the y steps (plan of N) and CW = 16 columns each in the z steps (plan PZ of N/2,
// twiddles at tw + N); the z output (k1, k2) of half h is grid index i2 = 2 lout_z(k1, k2) + h.
template <class P, int DIEL, int TMA = 0, int HALF = 0, int STEN = 0, int ZS = 1>
__global__ void __launch_bounds__(P::N / ZS / 8 * 32, 1) k_mid(PcbOp op, PcbCols cols, const cplx* __restrict__ tw, int ncols) {
    typedef typename ZSplit<P, ZS>::PZ PZ;
    constexpr int N = P::N, R1 = P::R1, R2 = P::R2;
    constexpr int NZ = N / ZS, ZR1 = PZ::R1, ZR2 = PZ::R2;      // rows of the CTA's (half) plane and the radices of the z transform
    constexpr int NW = NZ / 8, CW = N / NW;                     // warps; columns a warp owns in the z steps
    constexpr int LD = N + 1;                    // row stride (complex)
    constexpr bool FWD = HALF != 2, INV = HALF != 1;
    static_assert(N % 8 == 0 && NZ % 8 == 0 && N % NW == 0, "plane mode needs N % 8 == 0 (z-split: N % 16 == 0)");
    static_assert(HALF == 0 || DIEL == 0, "the half passes carry no dielectric");
    const cplx* __restrict__ twz = ZS == 1 ? tw : tw + N;      // twiddles of the z plan
    PCB_DYN_SMEM(cplx, pl);   // [NZ rows][LD] (+ one mbarrier per warp behind it when TMA)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long nn = op.nn;
    cplx* __restrict__ myrows = pl + (8 * warp) * LD;
#ifndef PCB_EMU
    unsigned long long* mybar = reinterpret_cast<unsigned long long*>(pl + (size_t)NZ * LD) + warp;
    unsigned phase = 0;
    if (TMA) {
        if (lane == 0) { pcb_mbar_init(mybar, 1); pcb_fence_mbar_init(); }
        __syncthreads();
    }
#endif
    // plane enumeration: (column, component, i0) over the CTAs, or (column, i0) over the clusters with the component = cluster rank
    int first = blockIdx.x, stride = gridDim.x, total = 3 * N * ZS * ncols, crank = 0;
#ifndef PCB_EMU
    unsigned pbase[3] = {0u, 0u, 0u};
    double inv_d[3] = {1.0, 1.0, 1.0};
    if (DIEL == 2) {
        crank = (int)pcb_cluster_ctarank(); first = (int)pcb_cluster_id(); stride = (int)pcb_cluster_count(); total = N * ZS * ncols;
        PCB_UNROLL
        for (int r = 0; r < 3; ++r) { pbase[r] = pcb_mapa(pcb_smem_u32(pl), (unsigned)r); inv_d[r] = 1.0 / op.ediag[r]; }
    }
#endif

    for (int pid = first; pid < total; pid += stride) {
        // z-split: (column, i0, component, half) -- the half planes of all three components of one i0 are in flight together, so the
        // cross-DoF gathers of the fused stencil find the other components' planes in L2 (a column no longer fits L2 for N > 128)
        const int col = (DIEL == 2) ? pid / (N * ZS) : pid / (3 * N * ZS);
        const int c = (DIEL == 2) ? crank : (ZS == 1 ? (pid / N) % 3 : (pid / ZS) % 3);
        const int i0 = (DIEL == 2) ? (pid / ZS) % N : (ZS == 1 ? pid % N : (pid / (3 * ZS)) % N);
        const int hz = ZS == 1 ? 0 : pid % ZS, prow = hz * NZ + 8 * warp;      // half plane; first plane row of this warp
        const long long poff = c * nn + (long long)i0 * N * N + (long long)prow * N;      // this warp's 8 rows
        cplx* __restrict__ base = ((STEN && HALF == 1) ? cols.out[col] : cols.wrk[col]) + poff;
        const cplx* __restrict__ src = (HALF == 2) ? cols.out[col] + poff : cols.wrk[col] + poff;
        // ---- load own rows (contiguous 8*N elements) ----
#ifndef PCB_EMU
        if (TMA) {
            if (lane == 0) {
                pcb_bulk_wait_read();                       // the previous plane's bulk stores have read these rows
                pcb_mbar_expect_tx(mybar, 8u * N * (unsigned)sizeof(cplx));
                PCB_UNROLL
                for (int r = 0; r < 8; ++r) pcb_bulk_load(myrows + r * LD, src + r * N, N * (unsigned)sizeof(cplx), mybar);
            }
        } else
#endif
        {
            for (int e = lane; e < 8 * N; e += 32) pcb_cp16(myrows + (e / N) * LD + e % N, src + e);
            pcb_cp_commit();
        }
        // dielectric bits this lane needs in the z step (items it = lane + 32 q: slot 8w + it%8, digit k1 = it/8): one precomputed
        // word per item (k_mask_bits), fetched now so that its latency hides behind the row loads
        constexpr int ZI = (CW * ZR1 + 31) / 32;
        unsigned mbits[ZI];
        if (DIEL == 1 || DIEL == 2) {
            PCB_UNROLL
            for (int q = 0; q < ZI; ++q) {
                const int it = lane + 32 * q;
                mbits[q] = (it < CW * ZR1) ? __ldg(op.mbits + (((((long long)c * N + i0) * N + CW * warp + it % CW) * ZS + hz) * ZR1 + it / CW)) : 0u;
            }
        }
        // coupled dielectric: mask bytes of this thread's points in step (B), point e = threadIdx.x + q * blockDim.x of the CTA's
        // third of the rows -- also fetched here, ten independent loads whose latency the plane's transforms hide
        constexpr int NTHR = NW * 32, PBQ = (DIEL == 2) ? ((NZ + 2) / 3 * N + NTHR - 1) / NTHR : 1;
        unsigned pmask[(PBQ + 3) / 4];
        int prow0 = 0, pcnt = 0;
        if (DIEL == 2) {
            prow0 = (crank * NZ) / 3;      // rows of the CTA's (half) plane
            pcnt = (((crank + 1) * NZ) / 3 - prow0) * N;
            const unsigned char* __restrict__ mp = op.maskp + (long long)i0 * N * N + (hz * NZ + prow0) * N;
            PCB_UNROLL
            for (int w = 0; w < (PBQ + 3) / 4; ++w) pmask[w] = 0u;
            PCB_UNROLL
            for (int q = 0; q < PBQ; ++q) {
                const int e = threadIdx.x + q * NTHR;
                if (e < pcnt) pmask[q / 4] |= (unsigned)__ldg(mp + e) << (8 * (q % 4));
            }
        }
#ifndef PCB_EMU
        if (TMA) { pcb_mbar_wait(mybar, phase); phase ^= 1u; } else
#endif
        pcb_cp_wait<0>();
        __syncwarp();
        if (STEN && HALF == 2) {
            // ---- M on own rows (real space): diagonal, and the cross-DoF coupling gathered from the other components' planes ----
            const unsigned char* __restrict__ mrow = op.maskp + ((long long)i0 * N + prow) * N;
            const cplx* __restrict__ Xcol = cols.out[col];
            const int* __restrict__ ctab = op.ctab;
            // pass 1: the diagonal entry, and a bit per element of this lane that has a coupling term (k_mask_active)
            static_assert(8 * N <= 32 * 64, "one bit per element of a lane");
            typedef typename std::conditional<(8 * N > 32 * 32), unsigned long long, unsigned>::type abits_t;
            abits_t actbits = 0u;
            PCB_UNROLL
            for (int q = 0; q < (8 * N + 31) / 32; ++q) {
                const int e = lane + 32 * q;
                if (e < 8 * N) {
                    const unsigned mk = __ldg(mrow + e);
                    if ((mk >> c) & 1u) { cplx* pv = myrows + (e / N) * LD + e % N; *pv = cscale(*pv, op.ediag[c]); }
                    actbits |= (abits_t)((mk >> (4 + c)) & 1u) << q;
                }
            }
            // pass 2: the coupled elements, GB at a time -- the gathers of a batch (taps of the other components' planes, L2) are all
            // issued before any is consumed; one element per trip leaves every trip waiting a full L2 round trip (1.27 ms per
            // 16 columns at N = 120 against 0.60 + 0.59 ms for the separate stencil kernel + half)
            constexpr int GB = 4;      // (8 per batch: 1.00 ms instead of 0.94 ms -- registers)
            while (__any_sync(0xffffffffu, actbits != 0u)) {
                int eq[GB];
                bool ok[GB];
                cplx add[GB];
                PCB_UNROLL
                for (int u = 0; u < GB; ++u) {
                    ok[u] = actbits != 0u;
                    const int q = ok[u] ? (sizeof(abits_t) == 8 ? __ffsll((long long)actbits) : __ffs((int)actbits)) - 1 : 0;
                    actbits &= actbits - (abits_t)1;
                    eq[u] = lane + 32 * q;
                }
                PCB_UNROLL
                for (int u = 0; u < GB; ++u) {
                    const int rl = eq[u] / N, cl = eq[u] % N;
                    const int ii[3] = {i0, __ldg(ctab + cl), __ldg(ctab + 2 * N + prow + rl)};
                    const unsigned mk = ok[u] ? (unsigned)__ldg(mrow + eq[u]) : 0u;
                    add[u] = pcb_crossdof_couple<N, (STEN - 1) / 2>(op, c, ii, mk, Xcol, ok[u]);
                }
                PCB_UNROLL
                for (int u = 0; u < GB; ++u)
                    if (ok[u]) { cplx* pv = myrows + (eq[u] / N) * LD + eq[u] % N; *pv = cadd(*pv, add[u]); }
            }
            __syncwarp();
        }
        if (FWD) {
            // ---- forward y on own rows: lanes = (row fastest, digit) ----
            for (int it = lane; it < 8 * R2; it += 32) {
                cplx* __restrict__ row = myrows + (it % 8) * LD;
                const int n2 = it / 8, b2 = P::lin2(n2);
                cplx v[R1];
                PCB_UNROLL
                for (int n1 = 0; n1 < R1; ++n1) v[n1] = row[P::wrap(P::lin1(n1) + b2)];
                Dft<R1, -1>::run(v);
                PCB_UNROLL
                for (int k1 = 0; k1 < R1; ++k1) {
                    cplx val = v[k1];
                    if (!P::PFA && k1 > 0) val = cmul(val, __ldg(tw + k1 * R2 + n2));
                    row[P::wrap(P::lin1(k1) + b2)] = val;
                }
            }
            __syncwarp();
            for (int it = lane; it < 8 * R1; it += 32) {
                cplx* __restrict__ row = myrows + (it % 8) * LD;
                const int k1 = it / 8, b1 = P::lin1(k1);
                cplx v[R2];
                PCB_UNROLL
                for (int n2 = 0; n2 < R2; ++n2) v[n2] = row[P::wrap(b1 + P::lin2(n2))];
                Dft<R2, -1>::run(v);
                PCB_UNROLL
                for (int k2 = 0; k2 < R2; ++k2) row[P::wrap(b1 + P::lin2(k2))] = v[k2];
            }
        }
        __syncthreads();
        // ---- z on own slots (columns CW w .. CW w + CW - 1): lanes = (slot fastest, digit) ----
        cplx* __restrict__ mycols = pl + CW * warp;
        if (FWD) {
            for (int it = lane; it < CW * ZR2; it += 32) {
                cplx* __restrict__ cp = mycols + it % CW;
                const int n2 = it / CW, b2 = PZ::lin2(n2);
                cplx v[ZR1];
                PCB_UNROLL
                for (int n1 = 0; n1 < ZR1; ++n1) v[n1] = cp[PZ::wrap(PZ::lin1(n1) + b2) * LD];
                Dft<ZR1, -1>::run(v);
                PCB_UNROLL
                for (int k1 = 0; k1 < ZR1; ++k1) {
                    cplx val = v[k1];
                    if (!PZ::PFA && k1 > 0) val = cmul(val, __ldg(twz + k1 * ZR2 + n2));
                    cp[PZ::wrap(PZ::lin1(k1) + b2) * LD] = val;
                }
            }
            __syncwarp();
        }
        if (HALF == 0 && DIEL != 2) {
            // forward radix R2 (-> real space), M, inverse radix R2: the values stay in registers
            PCB_UNROLL
            for (int q = 0; q < ZI; ++q) {
                const int it = lane + 32 * q;
                if (it >= CW * ZR1) break;
                cplx* __restrict__ cp = mycols + it % CW;
                const int k1 = it / CW, b1 = PZ::lin1(k1);
                // materials: the item's index bytes (k_mat_bytes, same item order as mbits), one vector load issued ahead of the
                // column loads and the radix step.  (Fetched with the row loads as mbits is, the ZI x 4 words stay live through
                // the y steps: 68 bytes of spills at N = 120.)
                constexpr int MW = (DIEL == 4) ? pcb_mat_pad(ZR2) / 4 : 1;
                unsigned mw[MW];
                if (DIEL == 4) pcb_ldg_words<MW>(mw, op.matp + (((((long long)c * N + i0) * N + CW * warp + it % CW) * ZS + hz) * ZR1 + k1) * (4 * MW));
                cplx v[ZR2];
                PCB_UNROLL
                for (int n2 = 0; n2 < ZR2; ++n2) v[n2] = cp[PZ::wrap(b1 + PZ::lin2(n2)) * LD];
                Dft<ZR2, -1>::run(v);
                if (DIEL == 1) {
                    const double scl = op.ediag[c];
                    const unsigned w = mbits[q];
                    PCB_UNROLL
                    for (int k2 = 0; k2 < ZR2; ++k2) v[k2] = cscale(v[k2], ((w >> k2) & 1u) ? scl : 1.0);   // branch-free: no divergence
                }
                if (DIEL == 4) pcb_mat_scale<ZR2>(op, mw, v);
                Dft<ZR2, +1>::run(v);
                PCB_UNROLL
                for (int n2 = 0; n2 < ZR2; ++n2) {
                    cplx val = v[n2];
                    if (!PZ::PFA && k1 > 0) { const cplx t = __ldg(twz + k1 * ZR2 + n2); val = cmul(val, cmake(t.x, -t.y)); }
                    cp[PZ::wrap(b1 + PZ::lin2(n2)) * LD] = val;
                }
            }
        } else {
            if (FWD) {       // (A) forward radix R2 (-> real space) and the diagonal of M
                PCB_UNROLL
                for (int q = 0; q < ZI; ++q) {
                    const int it = lane + 32 * q;
                    if (it >= CW * ZR1) break;
                    cplx* __restrict__ cp = mycols + it % CW;
                    const int b1 = PZ::lin1(it / CW);
                    cplx v[ZR2];
                    PCB_UNROLL
                    for (int n2 = 0; n2 < ZR2; ++n2) v[n2] = cp[PZ::wrap(b1 + PZ::lin2(n2)) * LD];
                    Dft<ZR2, -1>::run(v);
                    if (DIEL == 2) {
                        const double scl = op.ediag[c];
                        const unsigned w = mbits[q];
                        PCB_UNROLL
                        for (int k2 = 0; k2 < ZR2; ++k2) v[k2] = cscale(v[k2], ((w >> k2) & 1u) ? scl : 1.0);
                    }
                    PCB_UNROLL
                    for (int k2 = 0; k2 < ZR2; ++k2) cp[PZ::wrap(b1 + PZ::lin2(k2)) * LD] = v[k2];
                }
            }
#ifndef PCB_EMU
            if (DIEL == 2) {   // (B) off-diagonal terms at the coupled points of this CTA's third of the rows
                pcb_cluster_sync();
                PCB_UNROLL
                for (int q = 0; q < PBQ; ++q) {
                    const int e = threadIdx.x + q * NTHR;
                    const unsigned mk = (pmask[q / 4] >> (8 * (q % 4))) & 0xffu;      // 0 beyond pcnt
                    if (mk & 8u) {
                        const unsigned off = (unsigned)(((prow0 + e / N) * LD + e % N) * (int)sizeof(cplx));
                        const cplx u0 = pcb_ld_cluster(pbase[0] + off), u1 = pcb_ld_cluster(pbase[1] + off), u2 = pcb_ld_cluster(pbase[2] + off);
                        const cplx v0 = cscale(u0, (mk & 1u) ? inv_d[0] : 1.0), v1 = cscale(u1, (mk & 2u) ? inv_d[1] : 1.0),
                                   v2 = cscale(u2, (mk & 4u) ? inv_d[2] : 1.0);
                        pcb_st_cluster(pbase[0] + off, cfma(op.eoff[0], v1, cfma(op.eoff[1], v2, u0)));
                        pcb_st_cluster(pbase[1] + off, cfmac(op.eoff[0], v0, cfma(op.eoff[2], v2, u1)));
                        pcb_st_cluster(pbase[2] + off, cfmac(op.eoff[1], v0, cfmac(op.eoff[2], v1, u2)));
                    }
                }
                pcb_cluster_sync();
            }
#endif
            if (INV) {       // (C) inverse radix R2
                PCB_UNROLL
                for (int q = 0; q < ZI; ++q) {
                    const int it = lane + 32 * q;
                    if (it >= CW * ZR1) break;
                    cplx* __restrict__ cp = mycols + it % CW;
                    const int k1 = it / CW, b1 = PZ::lin1(k1);
                    cplx v[ZR2];
                    PCB_UNROLL
                    for (int k2 = 0; k2 < ZR2; ++k2) v[k2] = cp[PZ::wrap(b1 + PZ::lin2(k2)) * LD];
                    Dft<ZR2, +1>::run(v);
                    PCB_UNROLL
                    for (int n2 = 0; n2 < ZR2; ++n2) {
                        cplx val = v[n2];
                        if (!PZ::PFA && k1 > 0) { const cplx t = __ldg(twz + k1 * ZR2 + n2); val = cmul(val, cmake(t.x, -t.y)); }
                        cp[PZ::wrap(b1 + PZ::lin2(n2)) * LD] = val;
                    }
                }
            }
        }
        if (INV) {
            __syncwarp();
            for (int it = lane; it < CW * ZR2; it += 32) {
                cplx* __restrict__ cp = mycols + it % CW;
                const int n2 = it / CW, b2 = PZ::lin2(n2);
                cplx v[ZR1];
                PCB_UNROLL
                for (int k1 = 0; k1 < ZR1; ++k1) v[k1] = cp[PZ::wrap(PZ::lin1(k1) + b2) * LD];
                Dft<ZR1, +1>::run(v);
                PCB_UNROLL
                for (int n1 = 0; n1 < ZR1; ++n1) cp[PZ::wrap(PZ::lin1(n1) + b2) * LD] = v[n1];
            }
        }
        __syncthreads();
        if (INV) {
            // ---- inverse y on own rows ----
            for (int it = lane; it < 8 * R1; it += 32) {
                cplx* __restrict__ row = myrows + (it % 8) * LD;
                const int k1 = it / 8, b1 = P::lin1(k1);
                cplx v[R2];
                PCB_UNROLL
                for (int k2 = 0; k2 < R2; ++k2) v[k2] = row[P::wrap(b1 + P::lin2(k2))];
                Dft<R2, +1>::run(v);
                PCB_UNROLL
                for (int n2 = 0; n2 < R2; ++n2) {
                    cplx val = v[n2];
                    if (!P::PFA && k1 > 0) { const cplx t = __ldg(tw + k1 * R2 + n2); val = cmul(val, cmake(t.x, -t.y)); }
                    row[P::wrap(b1 + P::lin2(n2))] = val;
                }
            }
            __syncwarp();
            for (int it = lane; it < 8 * R2; it += 32) {
                cplx* __restrict__ row = myrows + (it % 8) * LD;
                const int n2 = it / 8, b2 = P::lin2(n2);
                cplx v[R1];
                PCB_UNROLL
                for (int k1 = 0; k1 < R1; ++k1) v[k1] = row[P::wrap(P::lin1(k1) + b2)];
                Dft<R1, +1>::run(v);
                PCB_UNROLL
                for (int n1 = 0; n1 < R1; ++n1) row[P::wrap(P::lin1(n1) + b2)] = v[n1];
            }
            __syncwarp();
        }
        // ---- store own rows ----
#ifndef PCB_EMU
        if (TMA) {
            pcb_fence_async_smem();                         // the rows were written through the generic proxy
            __syncwarp();
            if (lane == 0) {
                PCB_UNROLL
                for (int r = 0; r < 8; ++r) pcb_bulk_store(base + r * N, myrows + r * LD, N * (unsigned)sizeof(cplx));
                pcb_bulk_commit();
            }
        } else
#endif
        for (int e = lane; e < 8 * N; e += 32) base[e] = myrows[(e / N) * LD + e % N];
        __syncwarp();      // own rows are free again for the next plane's loads
    }
#ifndef PCB_EMU
    if (TMA && lane == 0) asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory");      // stores done before the CTA exits
#endif
}

// ---------------------------------------------------------------------------------------
// Plane mode, pass 2 of 3, FIVE shared-memory sweeps instead of seven (plans N = 8 R2 with odd R2: 24, 72, 120).
// The seven sweeps of k_mid are y8, y15 | z8, z15 M z15, z8 | y15, y8 (N = 120); the plane pass is bound by shared-memory
// wavefronts, so the transforms of the two axes are interleaved on 2-D register tiles:
//     A : y radix-8  x  z radix-4      (32 values per item)        z:  8 = 4 x 2 (Cooley-Tukey inside the Good-Thomas step)
//     B : y radix-R2 x  z radix-2      (2 R2 values per item)      y:  Cooley-Tukey (unit-stride digits, twiddles in A)
//     C : z radix-R2, M, z radix-R2 inverse                        (as in k_mid; the z digits sit in slot order d = 2k' + k'')
//     B', A' : the inverses of B and A.
// 32 complex values per thread need 128+ registers, so the CTA has 8 warps of up to 255 registers instead of 15 of 128: a
// HALF-WARP h owns the eight rows rho(n1, h) = lin(n1, h) of one z digit n2 = h -- exactly the rows its items of A, B, B', A'
// touch -- so those four sweeps, the TMA row loads before them and the TMA row stores after them need no CTA-wide barrier; only
// C (columns) is bracketed by the two barriers the seven-sweep kernel has as well.  Lane maps: in A the 16 lanes of a half-warp
// are the y digit n2 (consecutive columns), in B the 8 digits k1 (column stride R2, odd -> distinct banks), in C consecutive
// columns: every LDS.128 / STS.128 is conflict-free with the row stride N + 1.
// ---------------------------------------------------------------------------------------
template <class P>
struct Mid2 {
    static constexpr int N = P::N, R2 = P::R2;
    static constexpr bool OK = (P::R1 == 8) && (R2 % 2 == 1) && (R2 <= 15);
    static constexpr int NW = (R2 + 1) / 2, NTHR = 32 * NW;      // one half-warp per z digit
    static constexpr int CI = (8 * N + NTHR - 1) / NTHR;         // items of sweep C per thread
    PCB_HD static int rho(int n1, int n2) { const int s = R2 * n1 + 8 * n2; return s >= N ? s - N : s; }   // z slot (row) of digits (n1, n2)
    PCB_HD static int k1z(int d) { return (d >> 1) + 4 * (d & 1); }                                       // z digit held by slot digit d = 2k' + k''
    PCB_HD static int coordy(int col) { return col / R2 + 8 * (col % R2); }                                // y index held by column col after the forward steps
    // z index held by row `row` after the forward steps: row = rho(d, k2) -> d = row R2^-1 mod 8, k2 = row 8^-1 mod R2
    PCB_HD static int coordz(int row) {
        const int d = ((row % 8) * P::U) % 8, k2 = ((row % R2) * P::V) % R2;
        return P::wrap(P::lout1(k1z(d)) + P::lout2(k2));
    }
};

// the byte mask in the slot order of k_mid2 (coupled dielectric on clusters): maskp2[i0][row][col] = mask(i0, coordy(col), coordz(row))
template <class P>
__global__ void k_mask_plane2(PcbOp op, unsigned char* __restrict__ out) {
    typedef Mid2<P> M2;
    constexpr int N = P::N;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)N * N * N) return;
    const int col = (int)(t % N), row = (int)((t / N) % N), i0 = (int)(t / ((long long)N * N));
    out[t] = op.mask[((long long)M2::coordz(row) * N + M2::coordy(col)) * N + i0];
}

// mbits2[c][i0][d][col], bit k2 = "component c of grid point (i0, i1 = coordy(col), i2 = lout(k1z(d), k2)) lies in Omega_1"
template <class P>
__global__ void k_mask_bits2(PcbOp op, unsigned* __restrict__ out) {
    typedef Mid2<P> M2;
    constexpr int N = P::N, R2 = P::R2;
    const long long total = 3LL * N * 8 * N;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const int col = (int)(t % N), d = (int)((t / N) % 8), i0 = (int)((t / (8LL * N)) % N), c = (int)(t / (8LL * N * N));
    const int i1 = M2::coordy(col), o1 = P::lout1(M2::k1z(d));
    unsigned w = 0u;
    for (int k2 = 0; k2 < R2; ++k2) {
        const int i2 = P::wrap(o1 + P::lout2(k2));
        w |= ((unsigned)(op.mask[((long long)i2 * N + i1) * N + i0] >> c) & 1u) << k2;
    }
    out[t] = w;
}

// DIEL = 2: the coupled 3x3 dielectric on clusters of three CTAs, exactly as in k_mid<2>: sweep C is split at real space --
// forward radix-R2 + diagonal -> plane, cluster barrier, off-diagonal terms at the coupled points of this CTA's third of the rows
// through distributed shared memory (byte mask in this kernel's slot order, op.maskp2), cluster barrier, inverse radix-R2.
template <class P, int DIEL, int TMA = 0>
__global__ void __launch_bounds__(Mid2<P>::NTHR, 1) k_mid2(PcbOp op, PcbCols cols, const cplx* __restrict__ tw, int ncols) {
    typedef Mid2<P> M2;
    constexpr int N = P::N, R2 = P::R2, LD = N + 1, NTHR = M2::NTHR, CI = M2::CI;
    static_assert(M2::OK, "k_mid2 needs N = 8 * R2 with odd R2 <= 15");
    int first = blockIdx.x, stride = gridDim.x, total = 3 * N * ncols, crank = 0;
#ifndef PCB_EMU
    unsigned pbase[3] = {0u, 0u, 0u};
    double inv_d[3] = {1.0, 1.0, 1.0};
#endif
    PCB_DYN_SMEM(cplx, pl);   // [N rows][LD] (+ one mbarrier per warp behind it when TMA)
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int h = tid >> 4, l = tid & 15;             // half-warp = z digit n2, lane within it
    const bool hact = h < R2;
    const int nrw = (2 * warp + 1 < R2) ? 16 : 8;     // rows this warp moves (both half-warps, or one in the last warp)
    const long long nn = op.nn;
    const double RH = 0.70710678118654752440;
#ifndef PCB_EMU
    unsigned long long* mybar = reinterpret_cast<unsigned long long*>(pl + (size_t)N * LD) + warp;
    unsigned phase = 0;
    if (TMA) {
        if (lane == 0) { pcb_mbar_init(mybar, 1); pcb_fence_mbar_init(); }
        __syncthreads();
    }
#endif
    int rr[8];                // rows of this half-warp: rr[n1] = rho(n1, h) * LD
    PCB_UNROLL
    for (int n1 = 0; n1 < 8; ++n1) rr[n1] = M2::rho(n1, hact ? h : 0) * LD;
#ifndef PCB_EMU
    if (DIEL == 2) {
        crank = (int)pcb_cluster_ctarank(); first = (int)pcb_cluster_id(); stride = (int)pcb_cluster_count(); total = N * ncols;
        PCB_UNROLL
        for (int r = 0; r < 3; ++r) { pbase[r] = pcb_mapa(pcb_smem_u32(pl), (unsigned)r); inv_d[r] = 1.0 / op.ediag[r]; }
    }
#endif

    for (int pid = first; pid < total; pid += stride) {
        const int col = (DIEL == 2) ? pid / N : pid / (3 * N), c = (DIEL == 2) ? crank : (pid / N) % 3, i0 = pid % N;
        cplx* __restrict__ base = cols.wrk[col] + c * nn + (long long)i0 * N * N;
        // ---- load the warp's rows ----
#ifndef PCB_EMU
        if (TMA) {
            if (lane == 0) {
                pcb_bulk_wait_read();                       // the previous plane's bulk stores have read these rows
                pcb_mbar_expect_tx(mybar, (unsigned)nrw * N * (unsigned)sizeof(cplx));
                for (int r = 0; r < nrw; ++r) {
                    const int row = M2::rho(r & 7, 2 * warp + (r >> 3));
                    pcb_bulk_load(pl + row * LD, base + (long long)row * N, N * (unsigned)sizeof(cplx), mybar);
                }
            }
        } else
#endif
        {
            for (int e = lane; e < nrw * N; e += 32) {
                const int r = e / N, row = M2::rho(r & 7, 2 * warp + (r >> 3));
                pcb_cp16(pl + row * LD + e % N, base + (long long)row * N + e % N);
            }
            pcb_cp_commit();
        }
        unsigned mb[CI];
        if (DIEL >= 1) {
            PCB_UNROLL
            for (int q = 0; q < CI; ++q) {
                const int it = tid + NTHR * q;
                mb[q] = (it < 8 * N) ? __ldg(op.mbits2 + ((long long)c * N + i0) * (8 * N) + it) : 0u;
            }
        }
        // coupled dielectric: mask bytes of this thread's points of step (B) (point e = tid + q NTHR of the CTA's third of the rows)
        constexpr int PBQ = (DIEL == 2) ? ((N + 2) / 3 * N + NTHR - 1) / NTHR : 1;
        unsigned pmask[(PBQ + 3) / 4];
        int prow0 = 0;
        if (DIEL == 2) {
            prow0 = (crank * N) / 3;
            const int pcnt = (((crank + 1) * N) / 3 - prow0) * N;
            const unsigned char* __restrict__ mp = op.maskp2 + (long long)i0 * N * N + prow0 * N;
            PCB_UNROLL
            for (int w = 0; w < (PBQ + 3) / 4; ++w) pmask[w] = 0u;
            PCB_UNROLL
            for (int q = 0; q < PBQ; ++q) {
                const int e = tid + q * NTHR;
                if (e < pcnt) pmask[q / 4] |= (unsigned)__ldg(mp + e) << (8 * (q % 4));
            }
        }
#ifndef PCB_EMU
        if (TMA) { pcb_mbar_wait(mybar, phase); phase ^= 1u; } else
#endif
        pcb_cp_wait<0>();
        __syncwarp();

        // ---- A: forward y radix-8 (columns n1 R2 + n2y) x forward z radix-4 (rows rho(2p + q, h)) ----
        if (hact && l < R2) {
            PCB_UNROLL
            for (int q = 0; q < 2; ++q) {
                cplx v[4][8];
                PCB_UNROLL
                for (int p = 0; p < 4; ++p) {
                    PCB_UNROLL
                    for (int n1 = 0; n1 < 8; ++n1) v[p][n1] = pl[rr[2 * p + q] + n1 * R2 + l];
                }
                PCB_UNROLL
                for (int p = 0; p < 4; ++p) Dft<8, -1>::run(v[p]);
                PCB_UNROLL
                for (int k1 = 0; k1 < 8; ++k1) {
                    cplx u[4] = {v[0][k1], v[1][k1], v[2][k1], v[3][k1]};
                    if (k1 > 0) {
                        const cplx t = __ldg(tw + k1 * R2 + l);
                        PCB_UNROLL
                        for (int p = 0; p < 4; ++p) u[p] = cmul(u[p], t);
                    }
                    Dft<4, -1>::run(u);
                    if (q == 1) {      // w8^{k'}: exp(-2 pi i k' / 8)
                        u[1] = cmake((u[1].x + u[1].y) * RH, (u[1].y - u[1].x) * RH);
                        u[2] = cmake(u[2].y, -u[2].x);
                        u[3] = cmake((u[3].y - u[3].x) * RH, -(u[3].x + u[3].y) * RH);
                    }
                    PCB_UNROLL
                    for (int kp = 0; kp < 4; ++kp) pl[rr[2 * kp + q] + k1 * R2 + l] = u[kp];
                }
            }
        }
        __syncwarp();
        // ---- B: forward y radix-R2 (columns k1 R2 + n2y) x forward z radix-2 (rows rho(2k', h), rho(2k' + 1, h)) ----
        if (hact) {
            PCB_UNROLL
            for (int b = 0; b < 2; ++b) {
                const int item = l + 16 * b, k1 = item & 7, kp = item >> 3;
                cplx* __restrict__ p0 = pl + M2::rho(2 * kp, h) * LD + k1 * R2;
                cplx* __restrict__ p1 = pl + M2::rho(2 * kp + 1, h) * LD + k1 * R2;
                cplx v0[R2], v1[R2];
                PCB_UNROLL
                for (int n2 = 0; n2 < R2; ++n2) { v0[n2] = p0[n2]; v1[n2] = p1[n2]; }
                Dft<R2, -1>::run(v0);
                Dft<R2, -1>::run(v1);
                PCB_UNROLL
                for (int k2 = 0; k2 < R2; ++k2) { p0[k2] = cadd(v0[k2], v1[k2]); p1[k2] = csub(v0[k2], v1[k2]); }
            }
        }
        __syncthreads();
        if (DIEL == 2) {
#ifndef PCB_EMU
            // ---- C1: z radix-R2 forward (-> real space) and the diagonal of M ----
            PCB_UNROLL
            for (int q = 0; q < CI; ++q) {
                const int it = tid + NTHR * q;
                if (it >= 8 * N) break;
                const int d = it / N;
                cplx* __restrict__ cp = pl + it % N;
                cplx v[R2];
                PCB_UNROLL
                for (int n2 = 0; n2 < R2; ++n2) v[n2] = cp[M2::rho(d, n2) * LD];
                Dft<R2, -1>::run(v);
                const double scl = op.ediag[c];
                const unsigned w = mb[q];
                PCB_UNROLL
                for (int k2 = 0; k2 < R2; ++k2) cp[M2::rho(d, k2) * LD] = cscale(v[k2], ((w >> k2) & 1u) ? scl : 1.0);
            }
            // ---- (B): off-diagonal terms at the coupled points of this CTA's third of the rows, through distributed shared memory ----
            pcb_cluster_sync();
            PCB_UNROLL
            for (int q = 0; q < PBQ; ++q) {
                const int e = tid + q * NTHR;
                const unsigned mk = (pmask[q / 4] >> (8 * (q % 4))) & 0xffu;      // 0 beyond the CTA's share
                if (mk & 8u) {
                    const unsigned off = (unsigned)(((prow0 + e / N) * LD + e % N) * (int)sizeof(cplx));
                    const cplx u0 = pcb_ld_cluster(pbase[0] + off), u1 = pcb_ld_cluster(pbase[1] + off), u2 = pcb_ld_cluster(pbase[2] + off);
                    const cplx v0 = cscale(u0, (mk & 1u) ? inv_d[0] : 1.0), v1 = cscale(u1, (mk & 2u) ? inv_d[1] : 1.0),
                               v2 = cscale(u2, (mk & 4u) ? inv_d[2] : 1.0);
                    pcb_st_cluster(pbase[0] + off, cfma(op.eoff[0], v1, cfma(op.eoff[1], v2, u0)));
                    pcb_st_cluster(pbase[1] + off, cfmac(op.eoff[0], v0, cfma(op.eoff[2], v2, u1)));
                    pcb_st_cluster(pbase[2] + off, cfmac(op.eoff[1], v0, cfmac(op.eoff[2], v1, u2)));
                }
            }
            pcb_cluster_sync();
            // ---- C2: z radix-R2 inverse ----
            PCB_UNROLL
            for (int q = 0; q < CI; ++q) {
                const int it = tid + NTHR * q;
                if (it >= 8 * N) break;
                const int d = it / N;
                cplx* __restrict__ cp = pl + it % N;
                cplx v[R2];
                PCB_UNROLL
                for (int k2 = 0; k2 < R2; ++k2) v[k2] = cp[M2::rho(d, k2) * LD];
                Dft<R2, +1>::run(v);
                PCB_UNROLL
                for (int n2 = 0; n2 < R2; ++n2) cp[M2::rho(d, n2) * LD] = v[n2];
            }
            __syncthreads();
#endif
        } else {
            // ---- C: z radix-R2 over the rows rho(d, n2), M, inverse; lanes = consecutive columns; two items per trip (both items'
            //      loads are issued before either transform: the plane carries no restrict information, so item by item every
            //      load would wait behind the previous item's stores) ----
            PCB_UNROLL
            for (int q = 0; q < CI; q += 2) {
                const int ita = tid + NTHR * q, itb = ita + NTHR;
                if (ita >= 8 * N) break;
                const bool hasb = (q + 1 < CI) && itb < 8 * N;
                const int da = ita / N, db = hasb ? itb / N : 0;
                cplx* __restrict__ ca = pl + ita % N;
                cplx* __restrict__ cb = pl + (hasb ? itb % N : 0);
                cplx va[R2], vb[R2];
                PCB_UNROLL
                for (int n2 = 0; n2 < R2; ++n2) va[n2] = ca[M2::rho(da, n2) * LD];
                if (hasb) {
                    PCB_UNROLL
                    for (int n2 = 0; n2 < R2; ++n2) vb[n2] = cb[M2::rho(db, n2) * LD];
                }
                Dft<R2, -1>::run(va);
                if (DIEL == 1) {
                    const double scl = op.ediag[c];
                    const unsigned w = mb[q];
                    PCB_UNROLL
                    for (int k2 = 0; k2 < R2; ++k2) va[k2] = cscale(va[k2], ((w >> k2) & 1u) ? scl : 1.0);
                }
                Dft<R2, +1>::run(va);
                PCB_UNROLL
                for (int n2 = 0; n2 < R2; ++n2) ca[M2::rho(da, n2) * LD] = va[n2];
                if (hasb) {
                    Dft<R2, -1>::run(vb);
                    if (DIEL == 1) {
                        const double scl = op.ediag[c];
                        const unsigned w = mb[(q + 1 < CI) ? q + 1 : q];
                        PCB_UNROLL
                        for (int k2 = 0; k2 < R2; ++k2) vb[k2] = cscale(vb[k2], ((w >> k2) & 1u) ? scl : 1.0);
                    }
                    Dft<R2, +1>::run(vb);
                    PCB_UNROLL
                    for (int n2 = 0; n2 < R2; ++n2) cb[M2::rho(db, n2) * LD] = vb[n2];
                }
            }
            __syncthreads();
        }
        // ---- B': inverse z radix-2 x inverse y radix-R2 ----
        if (hact) {
            PCB_UNROLL
            for (int b = 0; b < 2; ++b) {
                const int item = l + 16 * b, k1 = item & 7, kp = item >> 3;
                cplx* __restrict__ p0 = pl + M2::rho(2 * kp, h) * LD + k1 * R2;
                cplx* __restrict__ p1 = pl + M2::rho(2 * kp + 1, h) * LD + k1 * R2;
                cplx v0[R2], v1[R2];
                PCB_UNROLL
                for (int k2 = 0; k2 < R2; ++k2) { const cplx a = p0[k2], bb = p1[k2]; v0[k2] = cadd(a, bb); v1[k2] = csub(a, bb); }
                Dft<R2, +1>::run(v0);
                Dft<R2, +1>::run(v1);
                PCB_UNROLL
                for (int n2 = 0; n2 < R2; ++n2) { p0[n2] = v0[n2]; p1[n2] = v1[n2]; }
            }
        }
        __syncwarp();
        // ---- A': conjugate twiddles, inverse z radix-4 x inverse y radix-8 ----
        if (hact && l < R2) {
            PCB_UNROLL
            for (int q = 0; q < 2; ++q) {
                cplx v[4][8];
                PCB_UNROLL
                for (int k1 = 0; k1 < 8; ++k1) {
                    cplx u[4];
                    PCB_UNROLL
                    for (int kp = 0; kp < 4; ++kp) u[kp] = pl[rr[2 * kp + q] + k1 * R2 + l];
                    if (q == 1) {      // conj w8^{k'}
                        u[1] = cmake((u[1].x - u[1].y) * RH, (u[1].x + u[1].y) * RH);
                        u[2] = cmake(-u[2].y, u[2].x);
                        u[3] = cmake(-(u[3].x + u[3].y) * RH, (u[3].x - u[3].y) * RH);
                    }
                    Dft<4, +1>::run(u);
                    if (k1 > 0) {
                        const cplx t = __ldg(tw + k1 * R2 + l);
                        const cplx tc = cmake(t.x, -t.y);
                        PCB_UNROLL
                        for (int p = 0; p < 4; ++p) u[p] = cmul(u[p], tc);
                    }
                    PCB_UNROLL
                    for (int p = 0; p < 4; ++p) v[p][k1] = u[p];
                }
                PCB_UNROLL
                for (int p = 0; p < 4; ++p) Dft<8, +1>::run(v[p]);
                PCB_UNROLL
                for (int p = 0; p < 4; ++p) {
                    PCB_UNROLL
                    for (int n1 = 0; n1 < 8; ++n1) pl[rr[2 * p + q] + n1 * R2 + l] = v[p][n1];
                }
            }
        }
        __syncwarp();
        // ---- store the warp's rows ----
#ifndef PCB_EMU
        if (TMA) {
            pcb_fence_async_smem();                         // the rows were written through the generic proxy
            __syncwarp();
            if (lane == 0) {
                for (int r = 0; r < nrw; ++r) {
                    const int row = M2::rho(r & 7, 2 * warp + (r >> 3));
                    pcb_bulk_store(base + (long long)row * N, pl + row * LD, N * (unsigned)sizeof(cplx));
                }
                pcb_bulk_commit();
            }
        } else
#endif
        for (int e = lane; e < nrw * N; e += 32) {
            const int r = e / N, row = M2::rho(r & 7, 2 * warp + (r >> 3));
            base[(long long)row * N + e % N] = pl[row * LD + e % N];
        }
        __syncwarp();      // own rows are free again for the next plane's loads
    }
#ifndef PCB_EMU
    if (TMA && lane == 0) asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory");      // stores done before the CTA exits
#endif
}

// (Round 2, measured and removed: k_mid3 -- a warp working on its two row sets one after the other with all 32 lanes, each set on
// its own mbarrier, so that the reload of set 0 for the next plane is in flight behind the inverse sweeps of set 1 and that of
// set 1 behind the forward sweeps of set 0: identical results, 0.822 vs 0.807 ms.  Together with the L2-prefetch variant this
// says the plane pass does not wait for its rows; it waits for dependent FP64 issue and the two CTA barriers around sweep C.)
// Plane-mode set-up for the coupled dielectric: the byte mask (bit c: edge DoF of component c, bit 3: volume DoF in Omega_1)
// in the slot order of the plane pass, maskp[i0][row][col] = mask(i0, i1 = coord(col), i2 = coord(row)).
template <class P, int ZS = 1>
__global__ void k_mask_plane(PcbOp op, unsigned char* __restrict__ out) {
    constexpr int N = P::N;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)N * N * N) return;
    const int col = (int)(t % N), row = (int)((t / N) % N), i0 = (int)(t / ((long long)N * N));
    out[t] = op.mask[((long long)ZSplit<P, ZS>::coord_row(row) * N + P::coord(col)) * N + i0];
}
// slot <-> index tables of the plane layout (the real-space stencil on plane-slot order): columns tab[s] = coord(s),
// tab[N + coord(s)] = s; rows tab[2N + rho] = coord_row(rho), tab[3N + coord_row(rho)] = rho (equal to the column tables
// except in the z-split plane mode, where row rho = h N/2 + s holds i2 = 2 coord_z(s) + h)
template <class P, int ZS = 1>
__global__ void k_coord_tables(int* __restrict__ tab) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= P::N) return;
    const int i = P::coord(s), j = ZSplit<P, ZS>::coord_row(s);
    tab[s] = i;
    tab[P::N + i] = s;
    tab[2 * P::N + s] = j;
    tab[3 * P::N + j] = s;
}

// ---------------------------------------------------------------------------------------
// Launch table: one entry per supported grid size, filled by the per-size translation units.
// ---------------------------------------------------------------------------------------
struct PcbOpLaunch {
    int N;
    int r1, r2;
    int plane_mode;   // 1: the fused (i1,i2)-plane pass exists for this size (N % 8 == 0 and the plane fits in shared memory)
    int plane_coupled; // 1: ... also for the coupled 3x3 dielectric (clusters of three CTAs; CUDA build only)
    int plane_five;    // 1: the five-sweep form of the plane pass (k_mid2) exists: N = 8 R2, R2 odd
    int lx;            // rows per tile of the x passes (a tile must lie in one i2 plane for the peer-memory passes: N % lx == 0)
    int plane_split;   // z-split plane mode (half planes): 0 not available, 1 selectable, 2 the plane mode of this size
    int zr1, zr2;      // ... radices of its z plan (the plan of N / 2)
    int plane_split_coupled;   // ... 1: with the cluster form of the coupled 3x3 dielectric (CUDA build only)
    // mode: 0 plain 3-D FFT forward, 1 plain inverse (1/N^3), 2 A = AMA^H, 3 H = AMA^H + gamma B^H B + shift
    int (*apply)(const PcbOp& op, const PcbCols& cols, int ncols, int mode, const cplx* tw, cudaStream_t s, int sms);
    // split passes used by the cross-DoF dielectric and by the tests: pass ids below
    int (*pass)(const PcbOp& op, const PcbCols& cols, int ncols, int pass_id, const cplx* tw, cudaStream_t s, int sms);
};
enum { PCB_PASS_XFWD_SYM = 0, PCB_PASS_XFWD = 1, PCB_PASS_YFWD = 2, PCB_PASS_ZFWD = 3, PCB_PASS_ZINV = 4,
       PCB_PASS_YINV = 5, PCB_PASS_XINV = 6, PCB_PASS_XINV_A = 7, PCB_PASS_XINV_H = 8, PCB_PASS_ZMID = 9,
       // plane mode (three passes, transposed scratch columns in cols.wrk)
       PCB_PASS_XFWD_SYM_T = 10, PCB_PASS_MID = 11, PCB_PASS_XINV_A_T = 12, PCB_PASS_XINV_H_T = 13,
       PCB_PASS_MASKBITS = 14 /* set-up: op.mask -> (unsigned*)op.mbits */,
       PCB_PASS_MID_FWD = 15, PCB_PASS_MID_INV = 16 /* halves of the plane pass around the cross-DoF stencil */,
       PCB_PASS_MASKPLANE = 17 /* set-up: op.mask -> (unsigned char*)op.maskp */, PCB_PASS_COORDTAB = 18 /* set-up: (int*)op.ctab */,
       PCB_PASS_MASKBITS2 = 19 /* set-up: op.mask -> (unsigned*)op.mbits2 (five-sweep plane pass) */,
       // large-grid mode over peer memory: x passes reading / writing the slabs of all ranks (op.dist)
       PCB_PASS_XFWD_SYM_D = 20, PCB_PASS_XINV_A_D = 21, PCB_PASS_XINV_H_D = 22,
       PCB_PASS_XFWD_SYM_TD = 23, PCB_PASS_XINV_A_TD = 24, PCB_PASS_XINV_H_TD = 25,
       // cross-DoF dielectric with the stencil fused into the inverse half of the plane pass (four kernels)
       PCB_PASS_MID_FWD_O = 26 /* forward half, planes -> cols.out */, PCB_PASS_MID_INV_ST = 27 /* stencil on load + inverse half, cols.out -> cols.wrk */,
       PCB_PASS_MASKACTIVE = 28 /* set-up: bits 4-6 of op.maskp */, PCB_PASS_MASKPLANE2 = 29 /* set-up: op.mask -> (unsigned char*)op.maskp2 */,
       PCB_PASS_XINV_T = 30 /* plane mode: plain inverse x pass (1/N^3, no symbol) from the transposed work column */,
       PCB_PASS_MATBYTES = 31 /* set-up: op.mat -> (unsigned char*)op.matp (materials dielectric) */ };

const PcbOpLaunch* pcb_find_plan(int N);
