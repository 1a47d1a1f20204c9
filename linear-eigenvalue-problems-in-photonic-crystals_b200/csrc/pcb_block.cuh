// pcb200 -- LOBPCG block kernels on the planar column layout (see pcb_common.cuh).
//
//   k_resid_precond : W = K_P^-1 (X diag(lambda) - HX) and column 2-norms of the raw residual in one pass
//                     (lobpcg.py:394-397 + numerical_experiments.py:83 / pcfft.py:50-70 / discretization.py:284-295)
//   k_gram2         : G = S^H S, T = S^H HS for a list of columns, Hermitian half only, on the FP64 tensor pipe
//                     (mma.sync m8n8k4 = SASS DMMA; orthogonalization.py:143-144)
//   k_update        : P <- [W P] E_wp, X <- X E_x + P (same for HS) in one pass, also DMMA (lobpcg.py:1248-1270)
//   k_coldots       : diag(A^H B) for column pairs (numerical_experiments.py:105-111, environment.py:131-157)
//   layout helpers  : row-major (R, k) host layout <-> planar columns, index list -> bit mask
// All reductions are two-stage (per-CTA partials, then a fixed-order sum) so results are deterministic.
#pragma once
#include "pcb_operator.cuh"

#define PCB_MAXL 96          // max columns in one Gram / update call (3m, m <= 32)

struct PcbColList {          // device pointers of up to PCB_MAXL columns (nullptr = zero column)
    const cplx* p[PCB_MAXL];
};
struct PcbColListW {
    cplx* p[PCB_MAXL];
};

PCB_D double pcb_warp_sum(double v) {
    PCB_UNROLL
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- layout: (R, k) row-major <-> planar columns -------------------------------------------------
// rm[r*ld + j] <-> col[j][r];  32x32 tiles through shared memory, both sides coalesced.
template <int TO_COLS>
__global__ void __launch_bounds__(256) k_transpose(cplx* __restrict__ rm, long long ld, PcbColListW cols, int k, long long R) {
    __shared__ cplx tile[32][33];
    const long long r0 = (long long)blockIdx.x * 32;
    const int j0 = blockIdx.y * 32;
    const int tx = threadIdx.x % 32, ty = threadIdx.x / 32;   // 32 x 8
    if (TO_COLS) {
        for (int rr = ty; rr < 32; rr += 8) {
            const long long r = r0 + rr;
            const int j = j0 + tx;
            if (r < R && j < k) tile[rr][tx] = rm[r * ld + j];
        }
        __syncthreads();
        for (int jj = ty; jj < 32; jj += 8) {
            const long long r = r0 + tx;
            const int j = j0 + jj;
            if (r < R && j < k) cols.p[j][r] = tile[tx][jj];
        }
    } else {
        for (int jj = ty; jj < 32; jj += 8) {
            const long long r = r0 + tx;
            const int j = j0 + jj;
            if (r < R && j < k) tile[tx][jj] = cols.p[j][r];
        }
        __syncthreads();
        for (int rr = ty; rr < 32; rr += 8) {
            const long long r = r0 + rr;
            const int j = j0 + tx;
            if (r < R && j < k) rm[r * ld + j] = tile[rr][tx];
        }
    }
}

// mask[cell] |= bit for every index in the list (edge list: row index r = c*nn + cell -> bit c)
__global__ void k_mask_from_index(const long long* __restrict__ ind, long long n, long long nn, int volume,
                                  unsigned* __restrict__ mask32) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long r = ind[i];
    if (r < 0 || r >= (volume ? nn : 3 * nn)) return;
    const int c = volume ? 3 : (int)(r / nn);
    const long long cell = volume ? r : r - c * nn;
    atomicOr(mask32 + (cell >> 2), (1u << c) << (8 * (int)(cell & 3)));
}

// ---- preconditioner symbol: inverse of K_P = K_A K_A^H + gamma K_B + shift I at one grid point --------
// (inverse_3_times_3_B -> inverse_3_times_3_block, discretization.py:224-295, cofactor formulas)
struct PcbPinv { double f11, f22, f33; cplx f12, f13, f23; };
PCB_HD PcbPinv pcb_pinv(const cplx k[3], double pnt, double shift) {
    const double b0 = cabs2(k[0]), b1 = cabs2(k[1]), b2 = cabs2(k[2]);
    const double d11 = pnt * b0 + b1 + b2 + shift;
    const double d22 = b0 + pnt * b1 + b2 + shift;
    const double d33 = b0 + b1 + pnt * b2 + shift;
    const double g = pnt - 1.0;
    const cplx d12 = cscale(cmulc(k[0], k[1]), g);
    const cplx d13 = cscale(cmulc(k[0], k[2]), g);
    const cplx d23 = cscale(cmulc(k[1], k[2]), g);
    const cplx t = cmul(cmul(d12, d23), cconj(d13));
    const double det = (d11 * d22 * d33 - (d11 * cabs2(d23) + d22 * cabs2(d13) + d33 * cabs2(d12))) + 2.0 * t.x;
    const double id = 1.0 / det;
    PcbPinv f;
    f.f11 = (d22 * d33 - cabs2(d23)) * id;
    f.f22 = (d11 * d33 - cabs2(d13)) * id;
    f.f33 = (d11 * d22 - cabs2(d12)) * id;
    f.f12 = cscale(csub(cmul(d13, cconj(d23)), cscale(d12, d33)), id);
    f.f13 = cscale(csub(cmul(d12, d23), cscale(d13, d22)), id);
    f.f23 = cscale(csub(cmul(d13, cconj(d12)), cscale(d23, d11)), id);
    return f;
}
PCB_HD void pcb_pinv_apply(const PcbPinv& f, const cplx r[3], cplx w[3]) {   // H_block with inv_fft (pcfft.py:50-70)
    w[0] = cfma(f.f12, r[1], cfma(f.f13, r[2], cscale(r[0], f.f11)));
    w[1] = cfmac(f.f12, r[0], cfma(f.f23, r[2], cscale(r[1], f.f22)));
    w[2] = cfmac(f.f13, r[0], cfmac(f.f23, r[1], cscale(r[2], f.f33)));
}

#define PCB_RP_CH 8     // columns per CTA chunk in k_resid_precond
#define PCB_MAXC_RP 32  // columns per k_resid_precond launch
struct PcbResidArgs {
    const cplx* x[PCB_MAXC_RP];
    const cplx* hx[PCB_MAXC_RP];
    cplx* w[PCB_MAXC_RP];
    double lambda[PCB_MAXC_RP];
};

// MODE 0: W = lambda X - HX (no preconditioner);  1: W = K_P^-1 (lambda X - HX);  2: W = K_P^-1 X (P_func alone)
// partial[(blockIdx.x * ncols) + j] = sum over this CTA's points of |r_j|^2  (raw residual, before K_P^-1)
// RND: the residual is rounded to complex64 and widened again before K_P^-1 -- the `.astype(complex64)` hand-over of
// lobpcg_sep_softlock_mixedprecision (lobpcg.py:574-577); the norms are those of the unrounded residual (:544-545).
template <int MODE, bool RND = false>
__global__ void __launch_bounds__(256) k_resid_precond(PcbOp op, PcbResidArgs a, int ncols, double* __restrict__ partial) {
    __shared__ double red[8][PCB_RP_CH];
    const int N = op.N;
    const long long nn = op.nloc;          // cells of this slab (= N^3 on a full context); also the component stride
    const int j0 = blockIdx.y * PCB_RP_CH;
    double acc[PCB_RP_CH];
    PCB_UNROLL
    for (int j = 0; j < PCB_RP_CH; ++j) acc[j] = 0.0;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < nn; p += (long long)gridDim.x * blockDim.x) {
        PcbPinv f;
        if (MODE) {
            const int i0 = (int)(p % N), i1 = (int)((p / N) % N), i2 = op.z0 + (int)(p / ((long long)N * N));
            const Sym3 s = pcb_symbol(op.T, N, i0, i1, i2);
            f = pcb_pinv(s.k, op.gamma, op.pshift);
        }
        PCB_UNROLL
        for (int j = 0; j < PCB_RP_CH; ++j) {
            const int jj = j0 + j;
            if (jj < ncols) {
                cplx r[3], w[3];
                PCB_UNROLL
                for (int c = 0; c < 3; ++c) {
                    const cplx x = a.x[jj][c * nn + p];
                    if (MODE == 2) r[c] = x;
                    else {
                        const cplx h = a.hx[jj][c * nn + p];
                        r[c] = cmake(fma(x.x, a.lambda[jj], -h.x), fma(x.y, a.lambda[jj], -h.y));
                    }
                }
                acc[j] += cabs2(r[0]) + cabs2(r[1]) + cabs2(r[2]);
                if (RND) {
                    PCB_UNROLL
                    for (int c = 0; c < 3; ++c) r[c] = cmake((double)(float)r[c].x, (double)(float)r[c].y);
                }
                if (MODE) pcb_pinv_apply(f, r, w);
                else { w[0] = r[0]; w[1] = r[1]; w[2] = r[2]; }
                PCB_UNROLL
                for (int c = 0; c < 3; ++c) a.w[jj][c * nn + p] = w[c];
            }
        }
    }
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    PCB_UNROLL
    for (int j = 0; j < PCB_RP_CH; ++j) {
        const double v = pcb_warp_sum(acc[j]);
        if (lane == 0) red[warp][j] = v;
    }
    __syncthreads();
    if (threadIdx.x < PCB_RP_CH) {
        double v = 0.0;
        for (int w = 0; w < 8; ++w) v += red[w][threadIdx.x];
        const int jj = j0 + threadIdx.x;
        if (jj < ncols) partial[(long long)blockIdx.x * ncols + jj] = v;
    }
}

// out[j] = sum_b partial[b*n + j] in fixed order (deterministic)
__global__ void k_sum_partials(const double* __restrict__ partial, int nblocks, int n, double* __restrict__ out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    double v = 0.0;
    for (int b = 0; b < nblocks; ++b) v += partial[(long long)b * n + j];
    out[j] = v;
}

// ---- Gram pair on the FP64 tensor pipe (DMMA m8n8k4) ------------------------------------------------------------
// G = S^H S and T = S^H HS.  An entry conj(a) b = (ar br + ai bi) + i (ar bi - ai br) is formed from THREE real products
// (the 3M scheme: 25 % fewer DMMAs than the four of the real-expanded form),
//   P1 = sum ar br,  P2 = sum ai bi,  P3 = sum (ar - ai)(br + bi)   ->   Re = P1 + P2,  Im = P3 - P1 + P2,
// each a real GEMM over the rows: one DMMA (8 x 8 x 4) covers 4 rows of an 8 x 8 column-tile pair.  The three partial sums
// are all of size |a||b|, the same magnitude the four-product form accumulates, so the rounding error bound is unchanged.
// Columns are grouped in tiles of 8; only tile pairs (ta <= tb) are accumulated (Hermitian completion in k_gram_finish).
// Each warp owns up to PPW tile pairs x {G, T} x {P1, P2, P3} = 6 DMMAs per pair and 4-row step; a lane fetches one complex
// element per operand tile (LDS.128) and derives the third operand with one DADD.
// Row tiles of PCB_GM_TR rows are staged [column][row] (+4 rows pad: conflict-free LDS.128) with double-buffered cp.async.
#define PCB_GM_TR 32
#define PCB_GM_LD (PCB_GM_TR + 4)
#define PCB_GM_PPW 2
#define PCB_GM_MAXW 20

PCB_HD void pcb_pair_from_index(int p, int nb, int& ia, int& ib) {   // row-major upper triangle incl. diagonal
    int a = 0, rem = p;
    while (rem >= nb - a) { rem -= nb - a; ++a; }
    ia = a; ib = a + rem;
}

// TSIDE (leading tile rows only, pcb_gram2_top): T_ab = conj(hs_a) s_b instead of conj(s_a) hs_b -- the same number for a
// Hermitian H -- so that only the first `nh` columns of HS are read at all.
// WMAX: most warps the instantiation is launched with; up to 12 warps two CTAs share an SM (register cap 80), which is what
// keeps the DMMA pipe fed across the per-tile barriers (ncu: 1 CTA of 11 warps reaches 63 % of the DMMA peak).
template <int PPW, bool TSIDE, int WMAX>     // PPW tile pairs per warp (1 or 2): the accumulators are 12 PPW doubles per lane
__global__ void __launch_bounds__(32 * WMAX, WMAX <= 12 ? 2 : 1)
k_gram2(PcbColList S, PcbColList HS, int n, int nh, int nt, int pair0, int npairs, long long R, cplx* __restrict__ partial /* [gridDim.x][2][nc*nc] */) {
    PCB_DYN_SMEM(cplx, sm);                      // [2 stages][2: S, HS][nc][LD]
    const int nc = 8 * nt;
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int warp = tid >> 5, lane = tid & 31, W = nthr >> 5;
    const int g = lane >> 2, tig = lane & 3;
    const size_t matElems = (size_t)nc * PCB_GM_LD;
    // tile pairs of this warp: pairs [pair0, pair0 + npairs) of the row-major upper triangle
    const int base = npairs / W, extra = npairs % W;
    const int cnt = base + (warp < extra ? 1 : 0);
    const int p0 = warp * base + (warp < extra ? warp : extra);
    int ta[PPW], tb[PPW];
    PCB_UNROLL
    for (int i = 0; i < PPW; ++i) {
        ta[i] = tb[i] = 0;
        if (i < cnt) pcb_pair_from_index(pair0 + p0 + i, nt, ta[i], tb[i]);
    }
    double acc[PPW][6][2];      // [pair][G: P1 P2 P3 | T: P1 P2 P3][c0, c1]
    PCB_UNROLL
    for (int i = 0; i < PPW; ++i) {
        PCB_UNROLL
        for (int q = 0; q < 6; ++q) acc[i][q][0] = acc[i][q][1] = 0.0;
    }
    // zero the padding columns (never loaded) of both stages
    for (int idx = tid; idx < 4 * (nc - n) * PCB_GM_LD; idx += nthr) {
        const int buf = idx / ((nc - n) * PCB_GM_LD), rem = idx % ((nc - n) * PCB_GM_LD);
        sm[(size_t)buf * matElems + (size_t)(n + rem / PCB_GM_LD) * PCB_GM_LD + rem % PCB_GM_LD] = cmake(0.0, 0.0);
    }
    const long long ntiles = (R + PCB_GM_TR - 1) / PCB_GM_TR;
    auto load_tile = [&](long long t, int stage) {      // warp per column, lane per row (PCB_GM_TR == 32): no index arithmetic
        const long long r = t * PCB_GM_TR + lane;
        cplx* d0 = sm + (size_t)(stage * 2) * matElems + lane;
        for (int c = warp; c < n; c += W) {
            const cplx* sp = S.p[c];
            const cplx* hp = HS.p[c];
            cplx* ds = d0 + (size_t)c * PCB_GM_LD;
            cplx* dh = ds + matElems;
            if (sp != nullptr && r < R) { pcb_cp16(ds, sp + r); if (!TSIDE || c < nh) pcb_cp16(dh, hp + r); }
            else { *ds = cmake(0.0, 0.0); *dh = cmake(0.0, 0.0); }
        }
        pcb_cp_commit();
    };
    long long t = blockIdx.x;
    int stage = 0;
    if (t < ntiles) load_tile(t, 0);
    for (; t < ntiles; t += gridDim.x) {
        const long long tn = t + gridDim.x;
        if (tn < ntiles) { load_tile(tn, stage ^ 1); pcb_cp_wait<1>(); } else { pcb_cp_wait<0>(); }
        __syncthreads();
        const cplx* s0 = sm + (size_t)(stage * 2) * matElems;
        const cplx* h0 = s0 + matElems;
        PCB_UNROLL
        for (int i = 0; i < PPW; ++i) {
            if (i < cnt) {
                // A fragment: (column ta*8 + g, row 4 step + tig); B fragments: (row 4 step + tig, column tb*8 + g)
                const cplx* pa = s0 + (size_t)(ta[i] * 8 + g) * PCB_GM_LD + tig;
                const cplx* pb = s0 + (size_t)(tb[i] * 8 + g) * PCB_GM_LD + tig;
                const cplx* ph = h0 + (size_t)((TSIDE ? ta[i] : tb[i]) * 8 + g) * PCB_GM_LD + tig;
                PCB_UNROLL
                for (int step = 0; step < PCB_GM_TR / 4; ++step) {
                    const cplx a = pa[4 * step], b = pb[4 * step], h = ph[4 * step];
                    const double am = a.x - a.y, bp = b.x + b.y;
                    pcb_dmma(acc[i][0][0], acc[i][0][1], a.x, b.x);
                    pcb_dmma(acc[i][1][0], acc[i][1][1], a.y, b.y);
                    pcb_dmma(acc[i][2][0], acc[i][2][1], am, bp);
                    if (TSIDE) {          // h is the A operand (column ta of HS)
                        pcb_dmma(acc[i][3][0], acc[i][3][1], h.x, b.x);
                        pcb_dmma(acc[i][4][0], acc[i][4][1], h.y, b.y);
                        pcb_dmma(acc[i][5][0], acc[i][5][1], h.x - h.y, bp);
                    } else {
                        pcb_dmma(acc[i][3][0], acc[i][3][1], a.x, h.x);
                        pcb_dmma(acc[i][4][0], acc[i][4][1], a.y, h.y);
                        pcb_dmma(acc[i][5][0], acc[i][5][1], am, h.x + h.y);
                    }
                }
            }
        }
        __syncthreads();
        stage ^= 1;
    }
    cplx* out = partial + (size_t)blockIdx.x * 2 * nc * nc;
    PCB_UNROLL
    for (int i = 0; i < PPW; ++i) {
        if (i < cnt) {
            const int ra = ta[i] * 8 + g;
            PCB_UNROLL
            for (int j = 0; j < 2; ++j) {
                const int cb = tb[i] * 8 + 2 * tig + j;
                out[ra * nc + cb] = cmake(acc[i][0][j] + acc[i][1][j], (acc[i][2][j] - acc[i][0][j]) + acc[i][1][j]);
                out[nc * nc + ra * nc + cb] = cmake(acc[i][3][j] + acc[i][4][j], (acc[i][5][j] - acc[i][3][j]) + acc[i][4][j]);
            }
        }
    }
}

// Sum the per-CTA partials in fixed order and complete the Hermitian matrices:
// entry (a,b) was accumulated iff tile(a) <= tile(b) and tile(a) < ttop; the others are conj of (b,a) (or zero if neither was).
__global__ void k_gram_finish(const cplx* __restrict__ partial, int nblocks, int nt, int ttop, cplx* __restrict__ out /* [2][nc*nc] */) {
    const int nc = 8 * nt;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= 2 * nc * nc) return;
    const int which = e / (nc * nc), ab = e % (nc * nc);
    const int a = ab / nc, b = ab % nc;
    const bool direct = (a / 8) <= (b / 8);
    const int src = direct ? a * nc + b : b * nc + a;
    if ((direct ? a : b) / 8 >= ttop) { out[e] = cmake(0.0, 0.0); return; }
    cplx v = cmake(0.0, 0.0);
#ifndef PCB_EMU
#pragma unroll 8
#endif
    for (int k = 0; k < nblocks; ++k) v = cadd(v, partial[(size_t)k * 2 * nc * nc + which * nc * nc + src]);   // independent loads, fixed order
    out[e] = direct ? v : cconj(v);
}

// ---- subspace update on the FP64 tensor pipe -----------------------------------------------------------------------
// Y = S E as a real GEMM: per row r, A[r][2k] = Re s_rk, A[r][2k+1] = Im s_rk (memory order of a complex element),
// B[2k][2j] = Re E_kj, B[2k][2j+1] = Im E_kj, B[2k+1][2j] = -Im E_kj, B[2k+1][2j+1] = Re E_kj; the C fragment of a lane is
// (Re, Im) of one output element -> one 16-byte store.  Input columns: kx X-columns then kp active W/P-columns (both
// padded to even with null = zero columns); E' is ((kx+kp) x MPp) complex, rows in the same order.  The accumulator first
// runs over the W/P part (-> Pn, stored to P/HP), then continues over the X part (-> X E_x + Pn, stored in place).
// A CTA stages TR rows of all input columns of S and HS ([column][row], cp.async double buffer); warp (rt, jp) owns the
// 8-row tile rt and the output column tiles {2jp, 2jp+1} (4 complex columns each) of both S and HS.
// Measured alternatives (B200, N = 120, m = 16, n_loc = 48; this form: 2.77 ms = 4.8 TB/s): a third cp.async stage 2.81 ms (the
// loads are not what it waits for); one of S / HS per stage with 64-row tiles 2.93 ms, with 32-row tiles 3.77 ms (E' fragments
// are then fetched twice per row tile); the 3M product scheme of the Gram kernel (6 DMMAs, two LDS.128 and three LDS.64 per
// 4 input columns and 8 output columns instead of 8 DMMAs and 12 LDS.64; 12 warps of 48-row tiles) 3.04 ms, and 28.3 vs 23.1 ms
// at N = 160, m = 32 -- fewer instructions on every pipe, yet slower: with one CTA per SM the 16 warps x 2 short DMMA chains of
// this form overlap the stage barriers better than 12 warps x 6 chains.
template <int TR>
struct PcbUpd {
    static constexpr int LD = TR + 4;      // complex; LD*16 mod 128 == 64: the two k-columns of an A fragment hit disjoint banks
};

template <int TR, int JW, int NST = 2>   // JW = output column tiles (of 4 complex columns) per warp; NST = cp.async stages
__global__ void __launch_bounds__(TR == 48 ? 768 : 512, 1)
k_update(PcbColList Sin, PcbColList HSin, PcbColListW Xout, PcbColListW HXout, PcbColListW Pout, PcbColListW HPout,
         const cplx* __restrict__ E, int m, int kx, int kp, int MPp, long long R) {
    constexpr int LD = PcbUpd<TR>::LD;
    PCB_DYN_SMEM(cplx, sm);
    const int nl = kx + kp;
    const int LDE = 2 * MPp;                         // doubles per row of the real-expanded E (MPp = MP + 2: LDE mod 16 == 4)
    double* sEr = reinterpret_cast<double*>(sm);     // [2 nl][LDE]: row 2k = (Re E_k., Im E_k.), row 2k+1 = (-Im E_k., Re E_k.)
    cplx* sT = sm + (size_t)2 * nl * MPp;            // [2 stages][2: S, HS][nl][LD]
    const size_t matElems = (size_t)nl * LD;
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int warp = tid >> 5, lane = tid & 31, W = nthr >> 5;
    const int g = lane >> 2, tig = lane & 3;
    constexpr int RT = TR / 8;
    const int rt = warp % RT, jp = warp / RT;      // warp (rt, jp): rows rt*8.., column tiles JW*jp ..
    for (int i = tid; i < nl * MPp; i += nthr) {
        const cplx e = E[i];
        const int k = i / MPp, j = i % MPp;
        sEr[(size_t)(2 * k) * LDE + 2 * j] = e.x;       sEr[(size_t)(2 * k) * LDE + 2 * j + 1] = e.y;
        sEr[(size_t)(2 * k + 1) * LDE + 2 * j] = -e.y;  sEr[(size_t)(2 * k + 1) * LDE + 2 * j + 1] = e.x;
    }
    const long long ntiles = (R + TR - 1) / TR;
    auto load_tile = [&](long long t, int stage) {      // TR lanes of a warp per column (two columns per trip when TR == 16,
        constexpr int CPW = TR >= 32 ? 1 : 32 / TR;      // a second, half-filled trip over the rows when TR == 48)
        const int sub = TR >= 32 ? 0 : lane / TR, rr0 = TR >= 32 ? lane : lane % TR;
        cplx* d0 = sT + (size_t)(stage * 2) * matElems;
        for (int c = warp * CPW + sub; c < nl; c += W * CPW) {
            const cplx* sp = c < PCB_MAXL ? Sin.p[c] : nullptr;      // columns past the list are zero padding
            const cplx* hp = c < PCB_MAXL ? HSin.p[c] : nullptr;
            PCB_UNROLL
            for (int q = 0; q < (TR + 31) / 32; ++q) {
                const int rr = rr0 + 32 * q;
                if (TR % 32 != 0 && TR > 32 && rr >= TR) break;
                const long long r = t * TR + rr;
                cplx* ds = d0 + (size_t)c * LD + rr;
                cplx* dh = ds + matElems;
                if (sp != nullptr && r < R) { pcb_cp16(ds, sp + r); pcb_cp16(dh, hp + r); }
                else { *ds = cmake(0.0, 0.0); *dh = cmake(0.0, 0.0); }
            }
        }
        pcb_cp_commit();
    };
    long long t = blockIdx.x;
    int stage = 0;
    if (NST == 2) {
        if (t < ntiles) load_tile(t, 0);
    } else {      // three stages: two tiles in flight, ONE barrier per tile (the buffer refilled below was read two barriers ago)
        PCB_UNROLL
        for (int i = 0; i < NST - 1; ++i) {
            const long long tt = t + (long long)i * gridDim.x;
            if (tt < ntiles) load_tile(tt, i); else pcb_cp_commit();
        }
    }
    const double* bbase = sEr + (size_t)tig * LDE + 8 * (JW * jp) + g;    // B fragment: row 2k + tig, column 8 jt + g
    for (; t < ntiles; t += gridDim.x) {
        if (NST == 2) {
            const long long tn = t + gridDim.x;
            if (tn < ntiles) { load_tile(tn, stage ^ 1); pcb_cp_wait<1>(); } else { pcb_cp_wait<0>(); }
            __syncthreads();
        } else {
            pcb_cp_wait<NST - 2>();
            __syncthreads();
            const long long tn = t + (long long)(NST - 1) * gridDim.x;
            if (tn < ntiles) load_tile(tn, (stage + NST - 1) % NST); else pcb_cp_commit();
        }
        const double* s0 = reinterpret_cast<const double*>(sT + (size_t)(stage * 2) * matElems);
        const double* h0 = reinterpret_cast<const double*>(sT + (size_t)(stage * 2 + 1) * matElems);
        double acc[2][JW][2];     // [S|HS][j-tile][c0,c1]
        PCB_UNROLL
        for (int q = 0; q < 2; ++q) {
            PCB_UNROLL
            for (int j = 0; j < JW; ++j) acc[q][j][0] = acc[q][j][1] = 0.0;
        }
        const long long r = t * TR + rt * 8 + g;
        // A fragment: element (row rt*8 + g, column k + (tig>>1)), component tig&1
        const int aoff = (tig >> 1) * (2 * LD) + (rt * 8 + g) * 2 + (tig & 1);
        PCB_UNROLL
        for (int part = 0; part < 2; ++part) {
            const int k0 = part == 0 ? kx : 0, k1 = part == 0 ? nl : kx;
#ifndef PCB_EMU
#pragma unroll 4
#endif
            for (int k = k0; k < k1; k += 2) {
                const double as = s0[(size_t)k * (2 * LD) + aoff];
                const double ah = h0[(size_t)k * (2 * LD) + aoff];
                PCB_UNROLL
                for (int j = 0; j < JW; ++j) {
                    const double bj = bbase[(size_t)(2 * k) * LDE + 8 * j];
                    pcb_dmma(acc[0][j][0], acc[0][j][1], as, bj);
                    pcb_dmma(acc[1][j][0], acc[1][j][1], ah, bj);
                }
            }
            if (r < R) {
                PCB_UNROLL
                for (int j = 0; j < JW; ++j) {
                    const int jj = (JW * jp + j) * 4 + tig;
                    if (jj < m) {
                        if (part == 0) {
                            Pout.p[jj][r] = cmake(acc[0][j][0], acc[0][j][1]);
                            HPout.p[jj][r] = cmake(acc[1][j][0], acc[1][j][1]);
                        } else {
                            Xout.p[jj][r] = cmake(acc[0][j][0], acc[0][j][1]);
                            HXout.p[jj][r] = cmake(acc[1][j][0], acc[1][j][1]);
                        }
                    }
                }
            }
        }
        if (NST == 2) { __syncthreads(); stage ^= 1; }
        else stage = (stage + 1) % NST;
    }
}

// ---- subspace update FUSED with the next residual, its norms and the preconditioner ------------------------------------
// (lobpcg.py:1248-1270 followed by :394-397 and :442 of the next iteration.)  After the Rayleigh-Ritz step the new Ritz values
// are known, and the new X' = X E_x + P', HX' = HX E_x + HP' sit in the accumulator fragments of k_update -- (Re, Im) of one
// element per lane -- so r = lambda X' - HX' and |r|^2 cost nothing to form there, instead of a separate pass that re-reads the
// 2m columns X', HX' one launch later.  The preconditioner K_P^-1 couples the three components of a grid point, so this form
// of the kernel takes its row tiles as 3 components x 16 cells (48 rows, 24 warps = 6 row tiles x 4 column tiles): the raw
// residual of a tile goes through 12 KB of shared memory, 256 threads apply the 3x3 symbol inverse (one grid point and column
// each) and store W.  m <= 16 (10-band runs); other widths keep pcb_update + pcb_residual.
struct PcbUpdRes { cplx* w[16]; double lambda[16]; };
// On the device the 256 preconditioner threads are EIGHT EXTRA WARPS (warps 24-31 of a 1024-thread CTA) that trail the 24 DMMA
// warps by one tile: the raw residual is double-buffered in shared memory and handed over with named barriers (bar.arrive /
// bar.sync), so the ~1000-cycle dependency chain of the symbol inverse overlaps the next tile's products instead of holding
// all 24 warps at a CTA barrier (measured with that barrier: 7.65 ms per LOBPCG iteration, i.e. no gain over the separate
// residual pass at 7.57 ms).  The host-emulation build runs the same phases back to back with 768 threads.
#ifndef PCB_EMU
PCB_D void pcb_bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;\n" ::"r"(id), "r"(n) : "memory"); }
PCB_D void pcb_bar_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;\n" ::"r"(id), "r"(n) : "memory"); }
#define PCB_UPDRES_THREADS 1024
#else
#define PCB_UPDRES_THREADS 768
#endif

// K_P^-1 on the raw residual of one tile (sR: [48][17]): grid point `cl` of the tile and column `col` per thread
PCB_D void pcb_updres_precond(const PcbOp& op, const PcbUpdRes& rs, const cplx* __restrict__ sR, long long t, int idx, int m) {
    constexpr int TC = 16, RS = 17;
    const int cl = idx % TC, col = idx / TC;
    const long long nloc = op.nloc;
    const long long p = t * TC + cl;
    if (p < nloc && col < m) {
        const int N = op.N;
        const int i0 = (int)(p % N), i1 = (int)((p / N) % N), i2 = op.z0 + (int)(p / ((long long)N * N));
        const Sym3 sy = pcb_symbol(op.T, N, i0, i1, i2);
        const PcbPinv f = pcb_pinv(sy.k, op.gamma, op.pshift);
        const cplx rv[3] = {sR[cl * RS + col], sR[(TC + cl) * RS + col], sR[(2 * TC + cl) * RS + col]};
        cplx wv[3];
        pcb_pinv_apply(f, rv, wv);
        cplx* __restrict__ wp = rs.w[col];
        PCB_UNROLL
        for (int c = 0; c < 3; ++c) wp[c * nloc + p] = wv[c];
    }
}

__global__ void __launch_bounds__(PCB_UPDRES_THREADS, 1)
k_update_res(PcbOp op, PcbColList Sin, PcbColList HSin, PcbColListW Xout, PcbColListW HXout, PcbColListW Pout, PcbColListW HPout, PcbUpdRes rs,
             const cplx* __restrict__ E, int m, int kx, int kp, int MPp, double* __restrict__ partial /* [gridDim.x][16] */) {
    constexpr int TR = 48, TC = 16, LD = PcbUpd<48>::LD, RT = TR / 8, RS = 17, NC = 768;     // NC = threads of the 24 product warps
    PCB_DYN_SMEM(cplx, sm);
    __shared__ double red[24][4];
    const int nl = kx + kp;
    const int LDE = 2 * MPp;
    double* sEr = reinterpret_cast<double*>(sm);     // [2 nl][LDE] real-expanded E (see k_update)
    cplx* sT = sm + (size_t)2 * nl * MPp;            // [2 stages][2: S, HS][nl][LD]
    const size_t matElems = (size_t)nl * LD;
    cplx* sR = sT + 4 * matElems;                    // [2][TR][RS] raw residual of the tile (double-buffered on the device)
    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, tig = lane & 3;
    const long long nloc = op.nloc;
    const long long ntiles = (nloc + TC - 1) / TC;
#ifndef PCB_EMU
    enum { BAR_PROD = 1, BAR_FULL = 2, BAR_EMPTY = 4 };      // named barriers: product warps; sR[b] written (+b); sR[b] consumed (+b)
    if (warp >= 24) {      // ---- preconditioner warps ----
        int it = 0;
        for (long long t = blockIdx.x; t < ntiles; t += gridDim.x, ++it) {
            const int b = it & 1;
            pcb_bar_sync(BAR_FULL + b, PCB_UPDRES_THREADS);
            pcb_updres_precond(op, rs, sR + b * TR * RS, t, tid - NC, m);
            if (t + 2 * (long long)gridDim.x < ntiles) pcb_bar_arrive(BAR_EMPTY + b, PCB_UPDRES_THREADS);
        }
        __syncthreads();      // the final reduction's barrier
        return;
    }
#endif
    const int W = NC >> 5;
    const int rt = warp % RT, jp = warp / RT;
    for (int i = tid; i < nl * MPp; i += NC) {
        const cplx e = E[i];
        const int k = i / MPp, j = i % MPp;
        sEr[(size_t)(2 * k) * LDE + 2 * j] = e.x;       sEr[(size_t)(2 * k) * LDE + 2 * j + 1] = e.y;
        sEr[(size_t)(2 * k + 1) * LDE + 2 * j] = -e.y;  sEr[(size_t)(2 * k + 1) * LDE + 2 * j + 1] = e.x;
    }
    // row rr of tile t: component rr / 16, cell t*16 + rr % 16
    auto load_tile = [&](long long t, int stage) {
        cplx* d0 = sT + (size_t)(stage * 2) * matElems;
        for (int c = warp; c < nl; c += W) {
            const cplx* sp = c < PCB_MAXL ? Sin.p[c] : nullptr;
            const cplx* hp = c < PCB_MAXL ? HSin.p[c] : nullptr;
            PCB_UNROLL
            for (int q = 0; q < 2; ++q) {
                const int rr = lane + 32 * q;
                if (rr >= TR) break;
                const long long cell = t * TC + rr % TC;
                const long long r = (long long)(rr / TC) * nloc + cell;
                cplx* ds = d0 + (size_t)c * LD + rr;
                cplx* dh = ds + matElems;
                if (sp != nullptr && cell < nloc) { pcb_cp16(ds, sp + r); pcb_cp16(dh, hp + r); }
                else { *ds = cmake(0.0, 0.0); *dh = cmake(0.0, 0.0); }
            }
        }
        pcb_cp_commit();
    };
#ifndef PCB_EMU
#define PCB_PROD_SYNC() pcb_bar_sync(BAR_PROD, NC)
#else
#define PCB_PROD_SYNC() __syncthreads()
#endif
    long long t = blockIdx.x;
    int stage = 0, it = 0;
    if (t < ntiles) load_tile(t, 0);
    const double* bbase = sEr + (size_t)tig * LDE + 8 * jp + g;
    const int jj = jp * 4 + tig;                     // this lane's output column
    const double lam = jj < 16 ? rs.lambda[jj] : 0.0;
    double nrm = 0.0;
    for (; t < ntiles; t += gridDim.x, ++it) {
        const long long tn = t + gridDim.x;
        if (tn < ntiles) { load_tile(tn, stage ^ 1); pcb_cp_wait<1>(); } else { pcb_cp_wait<0>(); }
        PCB_PROD_SYNC();
        const double* s0 = reinterpret_cast<const double*>(sT + (size_t)(stage * 2) * matElems);
        const double* h0 = reinterpret_cast<const double*>(sT + (size_t)(stage * 2 + 1) * matElems);
        double acc[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
        const int rr = rt * 8 + g;
        const long long cell = t * TC + rr % TC;
        const long long r = (long long)(rr / TC) * nloc + cell;
        const bool live = cell < nloc && jj < m;
        const int aoff = (tig >> 1) * (2 * LD) + rr * 2 + (tig & 1);
#ifndef PCB_EMU
        const int b = it & 1;
#else
        const int b = 0;
#endif
        cplx* __restrict__ sRb = sR + b * TR * RS;
        PCB_UNROLL
        for (int part = 0; part < 2; ++part) {
            const int k0 = part == 0 ? kx : 0, k1 = part == 0 ? nl : kx;
#ifndef PCB_EMU
#pragma unroll 4
#endif
            for (int k = k0; k < k1; k += 2) {
                const double as = s0[(size_t)k * (2 * LD) + aoff];
                const double ah = h0[(size_t)k * (2 * LD) + aoff];
                const double bj = bbase[(size_t)(2 * k) * LDE];
                pcb_dmma(acc[0][0], acc[0][1], as, bj);
                pcb_dmma(acc[1][0], acc[1][1], ah, bj);
            }
            if (part == 0) {
                if (live) {
                    Pout.p[jj][r] = cmake(acc[0][0], acc[0][1]);
                    HPout.p[jj][r] = cmake(acc[1][0], acc[1][1]);
                }
            } else {
                cplx res = cmake(0.0, 0.0);
                if (live) {
                    Xout.p[jj][r] = cmake(acc[0][0], acc[0][1]);
                    HXout.p[jj][r] = cmake(acc[1][0], acc[1][1]);
                    res = cmake(fma(acc[0][0], lam, -acc[1][0]), fma(acc[0][1], lam, -acc[1][1]));      // lambda x' - hx'
                    nrm += cabs2(res);
                }
#ifndef PCB_EMU
                if (it >= 2) pcb_bar_sync(BAR_EMPTY + b, PCB_UPDRES_THREADS);      // the preconditioner warps are done with this buffer
#endif
                if (jj < 16) sRb[rr * RS + jj] = res;
#ifndef PCB_EMU
                pcb_bar_arrive(BAR_FULL + b, PCB_UPDRES_THREADS);
#endif
            }
        }
        PCB_PROD_SYNC();
        stage ^= 1;
#ifdef PCB_EMU
        if (tid < TC * 16) pcb_updres_precond(op, rs, sRb, t, tid, m);      // (the next tile's sR writes follow its top-of-loop barrier)
#endif
    }
#undef PCB_PROD_SYNC
    // column norms: lanes with the same tig hold the same column
    nrm += __shfl_xor_sync(0xffffffffu, nrm, 4);
    nrm += __shfl_xor_sync(0xffffffffu, nrm, 8);
    nrm += __shfl_xor_sync(0xffffffffu, nrm, 16);
    if (g == 0) red[warp][tig] = nrm;
    __syncthreads();
    if (tid < 16) {
        const int jq = tid / 4, tq = tid % 4;
        double v = 0.0;
        for (int q = 0; q < RT; ++q) v += red[jq * RT + q][tq];
        partial[(long long)blockIdx.x * 16 + tid] = v;
    }
}

// ---- diag(A^H B) for column pairs -------------------------------------------------------------
__global__ void __launch_bounds__(256) k_coldots(PcbColList A, PcbColList B, int ncols, long long R, cplx* __restrict__ partial) {
    __shared__ double red[8][2];
    const int j = blockIdx.y;
    const cplx* __restrict__ a = A.p[j];
    const cplx* __restrict__ b = B.p[j];
    double sr = 0.0, si = 0.0;
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < R; r += (long long)gridDim.x * blockDim.x) {
        const cplx x = a[r], y = b[r];
        sr += x.x * y.x + x.y * y.y;
        si += x.x * y.y - x.y * y.x;
    }
    sr = pcb_warp_sum(sr);
    si = pcb_warp_sum(si);
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    if (lane == 0) { red[warp][0] = sr; red[warp][1] = si; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double vr = 0.0, vi = 0.0;
        for (int w = 0; w < 8; ++w) { vr += red[w][0]; vi += red[w][1]; }
        partial[(long long)blockIdx.x * ncols + j] = cmake(vr, vi);
    }
}

// ---- linear combination helper: Y = a*X + b*Y on columns (used by the drop-in operator wrappers) ------
__global__ void k_axpby(const cplx* __restrict__ x, cplx* __restrict__ y, double a, double b, long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const cplx u = x[i], v = y[i];
        y[i] = cmake(a * u.x + b * v.x, a * u.y + b * v.y);
    }
}

// ---- dielectric multiply as a stand-alone real-space kernel ---------------------------------------
// Point-wise types (none / chiral / trivial): Y = M X in one pass (the drop-in Diels(x) callable).
__global__ void __launch_bounds__(256) k_diel_point(PcbOp op, const cplx* __restrict__ X, cplx* __restrict__ Y) {
    const long long nn = op.nn;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < nn; p += (long long)gridDim.x * blockDim.x) {
        cplx u[3] = {X[p], X[nn + p], X[2 * nn + p]};
        unsigned m = op.diel ? op.mask[p] : 0u;
        if (op.diel == PCB_DIEL_CHIRAL) m &= 7u;
        pcb_diel_point(op, m, u);
        Y[p] = u[0]; Y[nn + p] = u[1]; Y[2 * nn + p] = u[2];
    }
}
// Materials dielectric: Y_r = inv_eps[mat[r]] X_r over the 3 nn rows (in place allowed)
PCB_D cplx pcb_mat_point(const PcbOp& op, long long r, cplx x) { return cscale(x, __ldg(op.inv_eps + __ldg(op.mat + r))); }
__global__ void __launch_bounds__(256) k_diel_mat(PcbOp op, const cplx* X, cplx* Y) {
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < 3 * op.nn; r += (long long)gridDim.x * blockDim.x)
        Y[r] = pcb_mat_point(op, r, X[r]);
}

// Cross-DoF dielectric (discretization.py:403-453): diagonal + eps_ab * S_ab couplings,
// S_ab = (I_a T_ab + T_ab I_b)/2,  T_ab = c (x) c^T on two of the three axes (stencil c with 2k taps).
// One thread per grid point computes all three output components (gather form); out of place.

// K > 0: 2K taps known at compile time (K = 1 is the reference's default, discretization.py:403); K = 0: runtime st.k.
// One thread per grid point and column (blockIdx.y): all three output components (gather form); out of place.
// The gather at one grid point p of the natural layout: y = (M X)(p) from the point's own values d[c] = X[c nn + p] and its
// stencil neighbours; mp = mask byte of p.  Shared by k_diel_crossdof and k_field_energy.
template <int K>
PCB_D void pcb_crossdof_gather(const PcbOp& op, const PcbStencil& st, const cplx* __restrict__ X, long long p, unsigned mp,
                               const cplx d[3], cplx y[3]) {
    const int N = op.N;
    const long long nn = op.nn;
    const int i[3] = {(int)(p % N), (int)((p / N) % N), (int)(p / ((long long)N * N))};
    const long long stride[3] = {1, N, (long long)N * N};
    PCB_UNROLL
    for (int c = 0; c < 3; ++c) y[c] = cscale(d[c], ((mp >> c) & 1u) ? op.ediag[c] : 1.0);
    // pairs (a,b): (0,1) c-axis 2, ct-axis 1;  (0,2) c-axis 2, ct-axis 0;  (1,2) c-axis 1, ct-axis 0
    constexpr int PA[3] = {0, 0, 1}, PB[3] = {1, 2, 2}, CAX[3] = {2, 2, 1}, TAX[3] = {1, 0, 0};
    const int kk = K > 0 ? K : st.k;
    const int taps = 2 * kk;
    PCB_UNROLL
    for (int pr = 0; pr < 3; ++pr) {
        const cplx e = op.eoff[pr];
        if (e.x == 0.0 && e.y == 0.0) continue;
        const int a = PA[pr], b = PB[pr], cax = CAX[pr], tax = TAX[pr];
        const double Ia = (double)((mp >> a) & 1u), Ib_p = (double)((mp >> b) & 1u);
        const cplx* __restrict__ Xa = X + a * nn;
        const cplx* __restrict__ Xb = X + b * nn;
        cplx sa = cmake(0.0, 0.0), sb = cmake(0.0, 0.0);
#ifndef PCB_EMU
#pragma unroll
#endif
        for (int j1 = 0; j1 < (K > 0 ? 2 * K : taps); ++j1) {
            const int oc = 1 - kk + j1;
            // wrapped displacement along the c-axis for +oc and -oc (|oc| <= k < N)
            const int cp = i[cax] + oc, cm = i[cax] - oc;
            const long long dcp = (long long)(cp >= N ? oc - N : (cp < 0 ? oc + N : oc)) * stride[cax];
            const long long dcm = (long long)(cm >= N ? -oc - N : (cm < 0 ? -oc + N : -oc)) * stride[cax];
#ifndef PCB_EMU
#pragma unroll
#endif
            for (int j2 = 0; j2 < (K > 0 ? 2 * K : taps); ++j2) {
                const int ot = 1 - kk + j2;
                const double w = st.w[j1] * st.w[j2] * 0.5;
                const int tm = i[tax] - ot, tp = i[tax] + ot;
                const long long dtm = (long long)(tm >= N ? -ot - N : (tm < 0 ? -ot + N : -ot)) * stride[tax];
                const long long dtp = (long long)(tp >= N ? ot - N : (tp < 0 ? ot + N : ot)) * stride[tax];
                // y_a(p) += e/2 * T(p,q) (I_a(p) + I_b(q)) x_b(q),  q = p + oc on the c-axis, - ot on the ct-axis
                const long long qi = p + dcp + dtm;
                const double Ibq = (double)((__ldg(op.mask + qi) >> b) & 1u);
                sa = cadd(sa, cscale(Xb[qi], w * (Ia + Ibq)));
                // y_b(p) += conj(e)/2 * T(p',p) (I_a(p') + I_b(p)) x_a(p'),  p' = p - oc on the c-axis, + ot on the ct-axis
                const long long pi_ = p + dcm + dtp;
                const double Iap = (double)((__ldg(op.mask + pi_) >> a) & 1u);
                sb = cadd(sb, cscale(Xa[pi_], w * (Iap + Ib_p)));
            }
        }
        y[a] = cfma(e, sa, y[a]);
        y[b] = cfmac(e, sb, y[b]);
    }
}

// K > 0: 2K taps known at compile time (K = 1 is the reference's default, discretization.py:403); K = 0: runtime st.k.
// One thread per grid point and column (blockIdx.y): all three output components (gather form); out of place.
template <int K>
__global__ void __launch_bounds__(256) k_diel_crossdof(PcbOp op, PcbStencil st, PcbCols cols) {
    const long long nn = op.nn;
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= nn) return;
    const cplx* __restrict__ X = cols.in[blockIdx.y];
    cplx* __restrict__ Y = cols.out[blockIdx.y];
    const unsigned mp = __ldg(op.mask + p);
    const cplx d[3] = {X[p], X[nn + p], X[2 * nn + p]};
    cplx y[3];
    pcb_crossdof_gather<K>(op, st, X, p, mp, d, y);
    PCB_UNROLL
    for (int c = 0; c < 3; ++c) Y[c * nn + p] = y[c];
}

// The same operator on the PLANE-SLOT layout of the plane pass (pcb_operator.cuh): columns hold W'[c][i0][row][col] with the
// real-space point (i0, i1 = coord(col), i2 = coord(row)); ctab = slot -> index and index -> slot tables of the plan.  Reads
// cols.wrk (output of the forward half of the plane pass), writes cols.out (input of the inverse half).  For the Good-Thomas
// plans (N = 72, 120) coord is multiplication by a constant mod N, so a +-1 neighbour along i1 is a constant slot shift and the
// gathers of a warp (lanes along col) stay contiguous.
// The gather at slot position pt of the plane-slot layout: y = (M X)(pt), d[c] = X[c nn + pt], mp = maskp[pt] (bits 0-3 are read).
// Shared by k_diel_crossdof_t and k_field_energy_t.
template <int K>
PCB_D void pcb_crossdof_gather_t(const PcbOp& op, const PcbStencil& st, const cplx* __restrict__ X, long long pt, unsigned mp,
                                 const cplx d[3], cplx y[3]) {
    const int N = op.N;
    const long long nn = op.nn;
    const int* __restrict__ ctab = op.ctab;
    const int scol = (int)(pt % N), srow = (int)((pt / N) % N);
    const int i[3] = {(int)(pt / ((long long)N * N)), __ldg(ctab + scol), __ldg(ctab + 2 * N + srow)};
    const unsigned char* __restrict__ maskp = op.maskp;      // the byte mask in the same slot order (k_mask_plane): coalesced
    PCB_UNROLL
    for (int c = 0; c < 3; ++c) y[c] = cscale(d[c], ((mp >> c) & 1u) ? op.ediag[c] : 1.0);
    constexpr int PA[3] = {0, 0, 1}, PB[3] = {1, 2, 2}, CAX[3] = {2, 2, 1}, TAX[3] = {1, 0, 0};
    const int kk = K > 0 ? K : st.k;
    const int taps = 2 * kk;
    PCB_UNROLL
    for (int pr = 0; pr < 3; ++pr) {
        const cplx e = op.eoff[pr];
        if (e.x == 0.0 && e.y == 0.0) continue;
        const int a = PA[pr], b = PB[pr], cax = CAX[pr], tax = TAX[pr];
        const double Ia = (double)((mp >> a) & 1u), Ib_p = (double)((mp >> b) & 1u);
        const cplx* __restrict__ Xa = X + a * nn;
        const cplx* __restrict__ Xb = X + b * nn;
        cplx sa = cmake(0.0, 0.0), sb = cmake(0.0, 0.0);
#ifndef PCB_EMU
#pragma unroll
#endif
        for (int j1 = 0; j1 < (K > 0 ? 2 * K : taps); ++j1) {
            const int oc = 1 - kk + j1;
#ifndef PCB_EMU
#pragma unroll
#endif
            for (int j2 = 0; j2 < (K > 0 ? 2 * K : taps); ++j2) {
                const int ot = 1 - kk + j2;
                const double w = st.w[j1] * st.w[j2] * 0.5;
                // q = p + oc on the c-axis, - ot on the t-axis;  p' = p - oc on the c-axis, + ot on the t-axis
                int q[3] = {i[0], i[1], i[2]}, r[3] = {i[0], i[1], i[2]};
                q[cax] = pcb_wrap(i[cax] + oc, N); q[tax] = pcb_wrap(i[tax] - ot, N);
                r[cax] = pcb_wrap(i[cax] - oc, N); r[tax] = pcb_wrap(i[tax] + ot, N);
                const long long qs = ((long long)q[0] * N + __ldg(ctab + 3 * N + q[2])) * N + __ldg(ctab + N + q[1]);
                const long long rs = ((long long)r[0] * N + __ldg(ctab + 3 * N + r[2])) * N + __ldg(ctab + N + r[1]);
                const double Ibq = (double)((__ldg(maskp + qs) >> b) & 1u);
                sa = cadd(sa, cscale(Xb[qs], w * (Ia + Ibq)));
                const double Iap = (double)((__ldg(maskp + rs) >> a) & 1u);
                sb = cadd(sb, cscale(Xa[rs], w * (Iap + Ib_p)));
            }
        }
        y[a] = cfma(e, sa, y[a]);
        y[b] = cfmac(e, sb, y[b]);
    }
}

template <int K>
__global__ void __launch_bounds__(256) k_diel_crossdof_t(PcbOp op, PcbStencil st, PcbCols cols) {
    const long long nn = op.nn;
    const long long pt = (long long)blockIdx.x * blockDim.x + threadIdx.x;      // position in the slot layout
    if (pt >= nn) return;
    const cplx* __restrict__ X = cols.wrk[blockIdx.y];
    cplx* __restrict__ Y = cols.out[blockIdx.y];
    const unsigned mp = __ldg(op.maskp + pt);
    const cplx d[3] = {X[pt], X[nn + pt], X[2 * nn + pt]};
    cplx y[3];
    pcb_crossdof_gather_t<K>(op, st, X, pt, mp, d, y);
    PCB_UNROLL
    for (int c = 0; c < 3; ++c) Y[c * nn + pt] = y[c];
}

// ---- electric energy of a mode in the dielectric (pcb_field_energy) ------------------------------------------------------
// Input: D = FFT3(K_A^H x) in real space, one column per blockIdx.y.  Per cell, E = M D is formed in registers and
//   e_tot += Re sum_c conj(D_c) E_c,   e_in += the same over the components c whose bit c of the mask is set (edge DoF in Omega_1).
// partial[(blockIdx.x * ncols + j) * 2 + {0: e_in, 1: e_tot}] = this CTA's sums for column j.  The grid-stride loop runs over a
// grid that does not depend on ncols, and both reduction stages have a fixed order: a column gets the same bits at any width.
// DIEL: 0 none (e_in = 0, no mask), 1 chiral, 2 trivial (point-wise, pcb_diel_point), 3 cross-DoF (the stencil gather; K as in
// k_diel_crossdof), 4 materials (e_in: the rows outside the background, index != 0).
PCB_D void pcb_energy_block_store(double ein, double etot, double* __restrict__ partial, int ncols) {
    __shared__ double red[8][2];
    ein = pcb_warp_sum(ein);
    etot = pcb_warp_sum(etot);
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    if (lane == 0) { red[warp][0] = ein; red[warp][1] = etot; }
    __syncthreads();
    if (threadIdx.x < 2) {
        double v = 0.0;
        for (int w = 0; w < 8; ++w) v += red[w][threadIdx.x];
        partial[((long long)blockIdx.x * ncols + blockIdx.y) * 2 + threadIdx.x] = v;
    }
}
// materials: bit c set where row c nn + p is outside the background (index != 0)
PCB_D unsigned pcb_mat_bits(const PcbOp& op, long long p) {
    unsigned m = 0u;
    PCB_UNROLL
    for (int c = 0; c < 3; ++c) m |= (__ldg(op.mat + c * op.nn + p) != 0 ? 1u : 0u) << c;
    return m;
}
// plane-slot position pt = (i0 N + row) N + col -> natural cell (i2 N + i1) N + i0, i1 = coord(col), i2 = coord_row(row)
PCB_D long long pcb_slot_to_cell(const PcbOp& op, long long pt) {
    const int N = op.N;
    const int col = (int)(pt % N), row = (int)((pt / N) % N), i0 = (int)(pt / ((long long)N * N));
    return ((long long)__ldg(op.ctab + 2 * N + row) * N + __ldg(op.ctab + col)) * N + i0;
}
PCB_D void pcb_energy_point(const cplx d[3], const cplx y[3], unsigned m, double& ein, double& etot) {
    PCB_UNROLL
    for (int c = 0; c < 3; ++c) {
        const double t = fma(d[c].x, y[c].x, d[c].y * y[c].y);
        etot += t;
        if ((m >> c) & 1u) ein += t;
    }
}

// natural layout [c][i2][i1][i0] (after the x, y, z forward passes); mask: op.mask
template <int DIEL, int K>
__global__ void __launch_bounds__(256) k_field_energy(PcbOp op, PcbStencil st, PcbCols cols, int ncols, double* __restrict__ partial) {
    const long long nn = op.nn;
    const cplx* __restrict__ X = cols.in[blockIdx.y];
    double ein = 0.0, etot = 0.0;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < nn; p += (long long)gridDim.x * blockDim.x) {
        const cplx d[3] = {X[p], X[nn + p], X[2 * nn + p]};
        const unsigned m = DIEL == 4 ? pcb_mat_bits(op, p) : DIEL ? (unsigned)__ldg(op.mask + p) : 0u;
        cplx y[3];
        if (DIEL == 3) pcb_crossdof_gather<K>(op, st, X, p, m, d, y);
        else if (DIEL == 4) {
            PCB_UNROLL
            for (int c = 0; c < 3; ++c) y[c] = pcb_mat_point(op, c * nn + p, d[c]);
        }
        else {
            y[0] = d[0]; y[1] = d[1]; y[2] = d[2];
            if (DIEL) pcb_diel_point(op, DIEL == 1 ? (m & 7u) : m, y);
        }
        pcb_energy_point(d, y, m, ein, etot);
    }
    pcb_energy_block_store(ein, etot, partial, ncols);
}

// plane-slot layout W'[c][i0][row][col] (after the x-forward pass and the forward half of the plane pass); mask: op.maskp, the
// byte mask in the same slot order (bits 0-3; the cross-DoF activity bits 4-6 are not read)
template <int DIEL, int K>
__global__ void __launch_bounds__(256) k_field_energy_t(PcbOp op, PcbStencil st, PcbCols cols, int ncols, double* __restrict__ partial) {
    const long long nn = op.nn;
    const cplx* __restrict__ X = cols.in[blockIdx.y];
    double ein = 0.0, etot = 0.0;
    for (long long pt = (long long)blockIdx.x * blockDim.x + threadIdx.x; pt < nn; pt += (long long)gridDim.x * blockDim.x) {
        const cplx d[3] = {X[pt], X[nn + pt], X[2 * nn + pt]};
        // materials: the natural-order position of the slot through the coordinate tables (no slot-ordered copy of the map)
        const long long p = DIEL == 4 ? pcb_slot_to_cell(op, pt) : 0;
        const unsigned m = DIEL == 4 ? pcb_mat_bits(op, p) : DIEL ? (unsigned)__ldg(op.maskp + pt) : 0u;
        cplx y[3];
        if (DIEL == 3) pcb_crossdof_gather_t<K>(op, st, X, pt, m, d, y);
        else if (DIEL == 4) {
            PCB_UNROLL
            for (int c = 0; c < 3; ++c) y[c] = pcb_mat_point(op, c * nn + p, d[c]);
        }
        else {
            y[0] = d[0]; y[1] = d[1]; y[2] = d[2];
            if (DIEL) pcb_diel_point(op, DIEL == 1 ? (m & 7u) : (m & 15u), y);
        }
        pcb_energy_point(d, y, m, ein, etot);
    }
    pcb_energy_block_store(ein, etot, partial, ncols);
}

// ---- electric energy per material (pcb_material_energy) ------------------------------------------------------------------
// Materials dielectric only.  Input: D = FFT3(K_A^H x) in real space, one column per blockIdx.y.  Row r = c nn + p adds
// Re conj(D_r) E_r, E_r = inv_eps[mat[r]] D_r (pcb_mat_point), to the bin of its material mat[r].
// partial[(blockIdx.x * ncols + j) * n_mat + m] = this CTA's sum for material m of column j.  No atomics.
//   S > 0 (n_mat <= S): each thread keeps S bins in registers (one select and add per bin and row), summed by the butterfly of
//     pcb_warp_sum once at the end: no vote and no warp barrier per row.
//   S = 0 (any n_mat <= 256): per row component, the lanes of a warp that hold the same material form one group (match_any); a
//     whole-warp group is summed by the butterfly, any other group by its lowest lane in lane order, into the warp's own bins.  On a
//     map that changes material from lane to lane every row then pays a vote, two warp barriers and a serial leader sum.
// Either way the eight warps' bins are added in warp order, and the grid does not depend on ncols: a column gets the same bits at any
// width.  (A given n_mat always takes the same path.)
#define PCB_ME_MAX 256      // materials of one dielectric (pcb_diel_create_materials)
PCB_D unsigned pcb_match_any(unsigned key) {
#ifdef PCB_EMU
    unsigned g = 0u;
    for (int l = 0; l < 32; ++l) g |= (__shfl_sync(0xffffffffu, key, l) == key ? 1u : 0u) << l;
    return g;
#else
    return __match_any_sync(0xffffffffu, key);
#endif
}
// t of every lane into bins[key]; key = PCB_ME_MAX: a lane past the end (nothing added).  All 32 lanes call it.
PCB_D void pcb_bin_add(double* bins, double* tv, unsigned key, double t, int lane) {
    const unsigned g = pcb_match_any(key);
    if (g == 0xffffffffu) {                        // one material across the warp (the usual case: maps are smooth along i0)
        const double s = pcb_warp_sum(t);
        if (lane == 0 && key < PCB_ME_MAX) bins[key] += s;
        return;
    }
    tv[lane] = t;
    __syncwarp();
    if (key < PCB_ME_MAX && __ffs((int)g) - 1 == lane) {
        double s = 0.0;
        for (unsigned q = g; q; q &= q - 1u) s += tv[__ffs((int)q) - 1];
        bins[key] += s;
    }
    __syncwarp();
}
#define PCB_ME_REG 16       // materials whose bins a thread keeps in registers (k_material_energy[_t]<PCB_ME_REG>)
// T = 0: natural layout [c][i2][i1][i0]; T = 1: plane-slot layout W'[c][i0][row][col], the cell found through pcb_slot_to_cell
template <int T, int S>
PCB_D void pcb_material_energy_body(const PcbOp& op, const cplx* __restrict__ X, int ncols, int n_mat, double* __restrict__ partial) {
    __shared__ double bins[8][S ? S : PCB_ME_MAX];
    __shared__ double tv[8][S ? 1 : 32];
    const long long nn = op.nn;
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    double acc[S ? S : 1];
    PCB_UNROLL
    for (int k = 0; k < (S ? S : 1); ++k) acc[k] = 0.0;
    if (!S) {
        for (int i = threadIdx.x; i < 8 * n_mat; i += blockDim.x) bins[i / n_mat][i % n_mat] = 0.0;
        __syncthreads();
    }
    // warp-uniform trip count: the lanes past nn take part in the votes with key PCB_ME_MAX
    for (long long p0 = (long long)blockIdx.x * blockDim.x + 32 * warp; p0 < nn; p0 += (long long)gridDim.x * blockDim.x) {
        const long long pt = p0 + lane;
        const bool in = pt < nn;
        const long long p = !in ? 0 : T ? pcb_slot_to_cell(op, pt) : pt;
        cplx d[3];
        unsigned m[3];
        PCB_UNROLL
        for (int c = 0; c < 3; ++c) {
            d[c] = in ? X[c * nn + pt] : cmake(0.0, 0.0);
            m[c] = in ? (unsigned)__ldg(op.mat + c * nn + p) : (unsigned)PCB_ME_MAX;
        }
        PCB_UNROLL
        for (int c = 0; c < 3; ++c) {
            const cplx y = in ? cscale(d[c], __ldg(op.inv_eps + m[c])) : cmake(0.0, 0.0);
            const double t = fma(d[c].x, y.x, d[c].y * y.y);
            if (S) {
                PCB_UNROLL
                for (int k = 0; k < (S ? S : 1); ++k) acc[k] += m[c] == (unsigned)k ? t : 0.0;      // a select: acc stays in registers
            } else {
                pcb_bin_add(bins[warp], tv[warp], m[c], t, lane);
            }
        }
    }
    if (S) {
        PCB_UNROLL
        for (int k = 0; k < (S ? S : 1); ++k) {
            const double v = pcb_warp_sum(acc[k]);
            if (lane == 0) bins[warp][k] = v;
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n_mat; i += blockDim.x) {
        double v = 0.0;
        for (int w = 0; w < 8; ++w) v += bins[w][i];
        partial[((long long)blockIdx.x * ncols + blockIdx.y) * n_mat + i] = v;
    }
}
template <int S>
__global__ void __launch_bounds__(256) k_material_energy(PcbOp op, PcbCols cols, int ncols, int n_mat, double* __restrict__ partial) {
    pcb_material_energy_body<0, S>(op, cols.in[blockIdx.y], ncols, n_mat, partial);
}
template <int S>
__global__ void __launch_bounds__(256) k_material_energy_t(PcbOp op, PcbCols cols, int ncols, int n_mat, double* __restrict__ partial) {
    pcb_material_energy_body<1, S>(op, cols.in[blockIdx.y], ncols, n_mat, partial);
}

// ---- band velocity matrices (pcb_band_velocity) ---------------------------------------------------------------------------
// Input: X (cols.in) and E^ = IFFT3(M FFT3(K_A^H x)) (cols.out), natural layout; tau = dK_d/dalpha_d, [3][N] complex (device).
// For d, a, b cyclic:  W_d[i][j] = sum_q conj(x_i,b) F_j,d,a - conj(x_i,a) F_j,d,b  with  F_j,d,c = tau_d[q_d] E^_j,c
// (tau folded into E^ while staging), plus xx[j] = sum |x_j|^2 and xax[j] = Re sum conj(x_j) . (K x E^_j) on the diagonal blocks.
// blockIdx.y = (I, J), a pair of blocks of PCB_BV_B columns (X_I against E^_J); blockIdx.x strides over chunks of PCB_BV_P
// points.  A chunk is staged [c or m][column][point] in shared memory (+1 point pad: the staging stores and the broadcast loads
// of the register tiles are conflict-free); slice s of the chunk (points s P/S .. (s+1) P/S - 1) belongs to warps 2s, 2s+1, whose
// 64 lanes hold the 256 entries of the block as 2 x 2 register tiles (rows it + 8 ki, columns jt + 8 kj) for all three d.
// Determinism: an entry (d, i, j) is summed over the CTA's chunks in order, within a chunk over its slice's points in order,
// then over the S slices in order, then over the CTAs in order (k_sum_partials).  None of this depends on ncols or on (I, J):
// a column pair gets the same bits at any width.  partial[blockIdx.x * E + e], E = 6 n^2 + 2 n doubles:
// e = 2 ((d n + i) n + j) + {re, im} for W, 6 n^2 + j for xx, 6 n^2 + n + j for xax.
#define PCB_BV_B 16
#define PCB_BV_P 32
#define PCB_BV_S 4
#define PCB_BV_NT 256
#define PCB_BV_LD (PCB_BV_P + 1)
#define PCB_BV_SMEM ((3 + 6) * PCB_BV_B * PCB_BV_LD * (int)sizeof(cplx))
#ifdef PCB_EMU
#define PCB_BV_ROLLED
#else
#define PCB_BV_ROLLED _Pragma("unroll 1")
#endif
__global__ void __launch_bounds__(PCB_BV_NT, 2) k_band_velocity(PcbOp op, PcbCols cols, const cplx* __restrict__ tau, int ncols,
                                                                int nb, double* __restrict__ partial) {
    static_assert(PCB_BV_B == 16 && PCB_BV_NT == 256 && PCB_BV_S * 2 * 32 == PCB_BV_NT, "tile mapping below assumes these");
    constexpr int B = PCB_BV_B, P = PCB_BV_P, S = PCB_BV_S, LD = PCB_BV_LD, PS = P / S;
    PCB_DYN_SMEM(cplx, sm);
    cplx* __restrict__ Xs = sm;                     // [c][i][p]
    cplx* __restrict__ Fs = sm + 3 * B * LD;        // [m = 2 d + {0: a, 1: b}][j][p]
    __shared__ double red[2][PCB_BV_NT / 32][2];
    const int N = op.N;
    const long long nn = op.nn;
    const int I = blockIdx.y / nb, J = blockIdx.y % nb;
    const bool diag = (I == J);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int s = warp >> 1, t = (warp & 1) * 32 + lane;
    const int it = t >> 3, jt = t & 7;              // a warp reads 4 distinct rows and 8 distinct columns per load: broadcasts
    const long long nchunks = (nn + P - 1) / P;
    cplx acc[3][2][2];
    PCB_UNROLL
    for (int d = 0; d < 3; ++d)
        PCB_UNROLL
        for (int ki = 0; ki < 2; ++ki)
            PCB_UNROLL
            for (int kj = 0; kj < 2; ++kj) acc[d][ki][kj] = cmake(0.0, 0.0);
    double axx0 = 0.0, axx1 = 0.0, axax0 = 0.0, axax1 = 0.0;      // xx, xax of the columns staged as r = 0, 1
    for (long long ch = blockIdx.x; ch < nchunks; ch += gridDim.x) {
        // stage: thread = (point lane, columns warp and warp + 8); zero rows past the last column / point
        const long long q = ch * P + lane;
        const bool qok = q < nn;
        const int i0 = (int)(q % N), i1 = (int)((q / N) % N), i2 = (int)(q / ((long long)N * N));
        cplx tq[3] = {cmake(0.0, 0.0), cmake(0.0, 0.0), cmake(0.0, 0.0)};
        if (qok) { tq[0] = __ldg(tau + i0); tq[1] = __ldg(tau + N + i1); tq[2] = __ldg(tau + 2 * N + i2); }
        Sym3 sy;
        if (diag && qok) sy = pcb_symbol(op.T, N, i0, i1, i2);
        PCB_BV_ROLLED
        for (int r = 0; r < 2; ++r) {
            const int jl = warp + 8 * r;
            const int ci = I * B + jl, cj = J * B + jl;
            cplx xv[3], ev[3];
            PCB_UNROLL
            for (int c = 0; c < 3; ++c) {
                xv[c] = (qok && ci < ncols) ? cols.in[ci][c * nn + q] : cmake(0.0, 0.0);
                ev[c] = (qok && cj < ncols) ? cols.out[cj][c * nn + q] : cmake(0.0, 0.0);
                Xs[(c * B + jl) * LD + lane] = xv[c];
            }
            PCB_UNROLL
            for (int d = 0; d < 3; ++d) {
                const int a = (d + 1) % 3, b = (d + 2) % 3;
                Fs[((2 * d) * B + jl) * LD + lane] = cmul(tq[d], ev[a]);
                Fs[((2 * d + 1) * B + jl) * LD + lane] = cmul(tq[d], ev[b]);
            }
            if (diag && qok) {      // (I == J: xv and ev belong to the same column)
                cplx z[3];
                pcb_cross(sy.k, ev, z);
                double sxx = 0.0, sxax = 0.0;
                PCB_UNROLL
                for (int c = 0; c < 3; ++c) {
                    sxx += cabs2(xv[c]);
                    sxax += fma(xv[c].x, z[c].x, xv[c].y * z[c].y);
                }
                if (r == 0) { axx0 += sxx; axax0 += sxax; } else { axx1 += sxx; axax1 += sxax; }
            }
        }
        __syncthreads();
        // accumulate: this slice's points in order, 2 x 2 tile x 3 directions = 24 complex FMAs per point and lane
        PCB_BV_ROLLED
        for (int u = 0; u < PS; ++u) {
            const int p = s * PS + u;
            cplx xv[3][2];
            PCB_UNROLL
            for (int c = 0; c < 3; ++c)
                PCB_UNROLL
                for (int ki = 0; ki < 2; ++ki) xv[c][ki] = Xs[(c * B + it + 8 * ki) * LD + p];
            PCB_UNROLL
            for (int d = 0; d < 3; ++d) {
                const int a = (d + 1) % 3, b = (d + 2) % 3;
                cplx fa[2], fb[2];
                PCB_UNROLL
                for (int kj = 0; kj < 2; ++kj) {
                    fa[kj] = Fs[((2 * d) * B + jt + 8 * kj) * LD + p];
                    fb[kj] = Fs[((2 * d + 1) * B + jt + 8 * kj) * LD + p];
                }
                PCB_UNROLL
                for (int ki = 0; ki < 2; ++ki)
                    PCB_UNROLL
                    for (int kj = 0; kj < 2; ++kj)
                        acc[d][ki][kj] = cfmac(cneg(xv[a][ki]), fb[kj], cfmac(xv[b][ki], fa[kj], acc[d][ki][kj]));
            }
        }
        __syncthreads();
    }
    // slices -> CTA (fixed order) through shared memory: red_w[s][d][i][j]
    cplx* __restrict__ rw = sm;
    PCB_UNROLL
    for (int d = 0; d < 3; ++d)
        PCB_UNROLL
        for (int ki = 0; ki < 2; ++ki)
            PCB_UNROLL
            for (int kj = 0; kj < 2; ++kj) rw[((s * 3 + d) * B + it + 8 * ki) * B + jt + 8 * kj] = acc[d][ki][kj];
    PCB_UNROLL
    for (int r = 0; r < 2; ++r) {
        const double vx = pcb_warp_sum(r ? axx1 : axx0), va = pcb_warp_sum(r ? axax1 : axax0);
        if (lane == 0) { red[r][warp][0] = vx; red[r][warp][1] = va; }
    }
    __syncthreads();
    const long long E = 6LL * ncols * ncols + 2LL * ncols;
    double* __restrict__ out = partial + (long long)blockIdx.x * E;
    for (int e = tid; e < 3 * B * B; e += PCB_BV_NT) {
        const int d = e / (B * B), i = (e / B) % B, j = e % B;
        const int gi = I * B + i, gj = J * B + j;
        if (gi >= ncols || gj >= ncols) continue;
        cplx v = rw[(d * B + i) * B + j];
        PCB_UNROLL
        for (int sl = 1; sl < S; ++sl) v = cadd(v, rw[((sl * 3 + d) * B + i) * B + j]);
        const long long o = 2LL * (((long long)d * ncols + gi) * ncols + gj);
        out[o] = v.x;
        out[o + 1] = v.y;
    }
    if (diag && tid < 2 * B) {
        const int jl = tid % B, which = tid / B;       // column jl was staged by warp jl % 8, r = jl / 8
        const int gj = I * B + jl;
        if (gj < ncols) out[6LL * ncols * ncols + (long long)which * ncols + gj] = red[jl / 8][jl % 8][which];
    }
}

// Set-up for the fused stencil-on-load: bit 4 + c of the slot-ordered mask byte = "component c at this point has a non-zero
// cross-DoF coupling term" (its own DoF or any tap of a pair with eps_ab != 0 lies in Omega_1) -- elsewhere M is the identity
// for that component and the plane pass touches nothing.  src: k_mask_plane's bytes (bits 0-3), dst: the same plus bits 4-6.
__global__ void __launch_bounds__(256) k_mask_active(PcbOp op, const unsigned char* __restrict__ src, unsigned char* __restrict__ dst) {
    const int N = op.N;
    const long long pt = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (pt >= op.nn) return;
    const int* __restrict__ ctab = op.ctab;
    const int i[3] = {(int)(pt / ((long long)N * N)), ctab[(int)(pt % N)], ctab[2 * N + (int)((pt / N) % N)]};
    const unsigned mp = src[pt];
    constexpr int PA[3] = {0, 0, 1}, PB[3] = {1, 2, 2}, CAX[3] = {2, 2, 1}, TAX[3] = {1, 0, 0};
    const int kk = op.sten.k;
    unsigned act = 0u;
    for (int pr = 0; pr < 3; ++pr) {
        const cplx e = op.eoff[pr];
        if (e.x == 0.0 && e.y == 0.0) continue;
        const int a = PA[pr], b = PB[pr], cax = CAX[pr], tax = TAX[pr];
        act |= (((mp >> a) & 1u) << a) | (((mp >> b) & 1u) << b);
        for (int j1 = 0; j1 < 2 * kk; ++j1)
            for (int j2 = 0; j2 < 2 * kk; ++j2) {
                const int oc = 1 - kk + j1, ot = 1 - kk + j2;
                int q[3] = {i[0], i[1], i[2]}, r[3] = {i[0], i[1], i[2]};
                q[cax] = pcb_wrap(i[cax] + oc, N); q[tax] = pcb_wrap(i[tax] - ot, N);
                r[cax] = pcb_wrap(i[cax] - oc, N); r[tax] = pcb_wrap(i[tax] + ot, N);
                const long long qs = ((long long)q[0] * N + ctab[3 * N + q[2]]) * N + ctab[N + q[1]];
                const long long rs = ((long long)r[0] * N + ctab[3 * N + r[2]]) * N + ctab[N + r[1]];
                act |= ((unsigned)(src[qs] >> b) & 1u) << a;      // y_a(p) sees I_b(q)
                act |= ((unsigned)(src[rs] >> a) & 1u) << b;      // y_b(p) sees I_a(r)
            }
    }
    dst[pt] = (unsigned char)((mp & 15u) | (act << 4));
}

// ---- stand-alone point-wise symbol multiplies (drop-in A_block / H_block kernels) ---------------------
// MODE 0: Y = k x X (K_A, _kernels.py:43-71);  1: Y = (-conj k) x X (K_A^H, pcfft.py:148);
// MODE 2: Y = gamma conj(k) (k . X)  (h_block with D_B = gamma*(|k_c|^2, conj(k_a) k_b), pcfft.py:176)
template <int MODE>
__global__ void __launch_bounds__(256) k_symbol_point(PcbOp op, PcbCols cols) {
    const int N = op.N;
    const long long nn = op.nn;
    const cplx* __restrict__ X = cols.in[blockIdx.y];
    cplx* __restrict__ Y = cols.out[blockIdx.y];
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < nn; p += (long long)gridDim.x * blockDim.x) {
        const int i0 = (int)(p % N), i1 = (int)((p / N) % N), i2 = (int)(p / ((long long)N * N));
        const Sym3 s = pcb_symbol(op.T, N, i0, i1, i2);
        cplx x[3] = {X[p], X[nn + p], X[2 * nn + p]}, z[3];
        if (MODE == 0) {
            pcb_cross(s.k, x, z);
        } else if (MODE == 1) {
            cplx a[3];
            PCB_UNROLL
            for (int c = 0; c < 3; ++c) a[c] = cmake(-s.k[c].x, s.k[c].y);
            pcb_cross(a, x, z);
        } else {
            cplx dot = cadd(cadd(cmul(s.k[0], x[0]), cmul(s.k[1], x[1])), cmul(s.k[2], x[2]));
            dot = cscale(dot, op.gamma);
            PCB_UNROLL
            for (int c = 0; c < 3; ++c) z[c] = cmulc(s.k[c], dot);
        }
        Y[p] = z[0]; Y[nn + p] = z[1]; Y[2 * nn + p] = z[2];
    }
}

// ---- geometry: the dielectric region Omega_1 evaluated on the device straight into the per-cell bit mask ------------------
// (dielectric.py:104-261: mesh3d_edge_dofs / mesh3d_volume_dofs, coo = mesh @ inv(ct^T), FLAG_<lattice>(coo)).  One thread per
// cell classifies its four DoFs -- bit c: edge DoF of component c (half a cell along axis c), bit 3: volume DoF (cell centre).
// A DoF whose decision margin is below a tolerance (|lhs - rhs| of the deciding inequality; exact ties of the flat lattices,
// or last-bit differences between this arithmetic and NumPy's) is reported in `amb` with the same bit layout: the host
// re-evaluates those few points with the reference's own NumPy expression, so the index sets stay bit-identical to the
// reference's while the O(N^3) work runs here (FCC, N = 120: 34 sphere / spheroid tests for each of 6.9 M points).
enum { PCB_GEOM_SC_FLAT1 = 0, PCB_GEOM_SC_FLAT2 = 1, PCB_GEOM_SC_CURV = 2, PCB_GEOM_BCC_SG = 3, PCB_GEOM_BCC_DG = 4, PCB_GEOM_FCC = 5 };
struct PcbGeom { int kind; double minv[9]; };      // minv = inv(ct^T), row-major: coo_j = sum_i mesh_i minv[i][j]

PCB_HD void pcb_geom_point(const PcbGeom& g, double u0, double u1, double u2, bool& inside, bool& amb) {
    const double x = u0 * g.minv[0] + u1 * g.minv[3] + u2 * g.minv[6];
    const double y = u0 * g.minv[1] + u1 * g.minv[4] + u2 * g.minv[7];
    const double z = u0 * g.minv[2] + u1 * g.minv[5] + u2 * g.minv[8];
    double margin = 1.0;
    inside = false;
#define PCB_GEOM_LE(lhs, rhs) ((margin = fmin(margin, fabs((lhs) - (rhs)))), (lhs) <= (rhs))
#define PCB_GEOM_GE(lhs, rhs) ((margin = fmin(margin, fabs((lhs) - (rhs)))), (lhs) >= (rhs))
#define PCB_GEOM_LT(lhs, rhs) ((margin = fmin(margin, fabs((lhs) - (rhs)))), (lhs) < (rhs))
    if (g.kind == PCB_GEOM_SC_FLAT1) {
        const bool a = PCB_GEOM_LE(x, 0.25), b = PCB_GEOM_LE(y, 0.25), c = PCB_GEOM_LE(z, 0.25);
        inside = (a && b) || (a && c) || (b && c);
    } else if (g.kind == PCB_GEOM_SC_FLAT2) {
        const bool xl = PCB_GEOM_LE(x, 0.25), yl = PCB_GEOM_LE(y, 0.25);
        const bool z1 = PCB_GEOM_GE(z, 0.25), z2 = PCB_GEOM_LE(z, 0.5), z3 = PCB_GEOM_GE(z, 0.5), z4 = PCB_GEOM_LE(z, 0.75), z5 = PCB_GEOM_GE(z, 0.75);
        const bool y1 = PCB_GEOM_GE(y, 0.5), y2 = PCB_GEOM_LE(y, 0.75), x1 = PCB_GEOM_GE(x, 0.5), x2 = PCB_GEOM_LE(x, 0.75);
        inside = (xl && yl) || (xl && z1 && z2) || (y1 && y2 && z3 && z4) || (x1 && x2 && z5);
    } else if (g.kind == PCB_GEOM_SC_CURV) {
        const double px = x - 0.5, py = y - 0.5, pz = z - 0.5;
        const double xx = px * px, yy = py * py, zz = pz * pz;
        const double rod2 = 0.11 * 0.11, ball2 = 0.345 * 0.345;
        const bool a = PCB_GEOM_LE(xx + yy + zz, ball2), b = PCB_GEOM_LE(xx + yy, rod2), c = PCB_GEOM_LE(xx + zz, rod2), d = PCB_GEOM_LE(yy + zz, rod2);
        inside = a || b || c || d;
    } else if (g.kind == PCB_GEOM_BCC_SG || g.kind == PCB_GEOM_BCC_DG) {
        const double tp = 2.0 * M_PI;
        double gy = sin(tp * x) * cos(tp * y) + sin(tp * y) * cos(tp * z) + sin(tp * z) * cos(tp * x);
        if (g.kind == PCB_GEOM_BCC_DG) gy = fabs(gy);
        margin = fabs(gy - 1.1);
        inside = gy > 1.1;
    } else {      // FCC diamond network: 18 spheres at the lattice sites, 16 prolate spheroids along the bonds
        const double r2 = 0.12 * 0.12, b_ell = 0.11;
        const double basis[4][3] = {{0, 0, 0}, {0, 0.5, 0.5}, {0.5, 0, 0.5}, {0.5, 0.5, 0}};
        const double sites[14][3] = {{0, 0, 0}, {1, 0, 0}, {0, 1, 0}, {0, 0, 1}, {0, 1, 1}, {1, 0, 1}, {1, 1, 0}, {1, 1, 1},
                                     {0, 0.5, 0.5}, {0.5, 0, 0.5}, {0.5, 0.5, 0}, {1, 0.5, 0.5}, {0.5, 1, 0.5}, {0.5, 0.5, 1}};
        for (int s = 0; s < 18; ++s) {
            const double sx = s < 14 ? sites[s][0] : 0.25 + basis[s - 14][0];
            const double sy = s < 14 ? sites[s][1] : 0.25 + basis[s - 14][1];
            const double sz = s < 14 ? sites[s][2] : 0.25 + basis[s - 14][2];
            const double d2 = (x - sx) * (x - sx) + (y - sy) * (y - sy) + (z - sz) * (z - sz);
            if (PCB_GEOM_LT(d2, r2)) inside = true;
        }
        for (int i = 0; i < 4; ++i) {
            const double hx = (basis[i][0] - 0.25) / 2, hy = (basis[i][1] - 0.25) / 2, hz = (basis[i][2] - 0.25) / 2;
            const double mx = (basis[i][0] + 0.25) / 2, my = (basis[i][1] + 0.25) / 2, mz = (basis[i][2] + 0.25) / 2;
            const double len = sqrt(hx * hx + hy * hy + hz * hz);
            const double dx = hx / len, dy = hy / len, dz = hz / len;
            const double major2 = b_ell * b_ell + len * len;
            for (int j = 0; j < 4; ++j) {
                const double X0 = x - (mx + basis[j][0]), X1 = y - (my + basis[j][1]), X2 = z - (mz + basis[j][2]);
                const double al = dx * X0 + dy * X1 + dz * X2;
                const double along = al * al, across = (X0 * X0 + X1 * X1 + X2 * X2) - along;
                if (PCB_GEOM_LT(along / major2 + across / (b_ell * b_ell), 1.0)) inside = true;
            }
        }
    }
#undef PCB_GEOM_LE
#undef PCB_GEOM_GE
#undef PCB_GEOM_LT
    amb = margin < 1e-10;
}

__global__ void __launch_bounds__(256) k_geom_mask(PcbGeom g, int N, unsigned char* __restrict__ mask, unsigned char* __restrict__ amb) {
    const long long nn = (long long)N * N * N;
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= nn) return;
    const int i[3] = {(int)(p % N), (int)((p / N) % N), (int)(p / ((long long)N * N))};
    unsigned m = 0u, a = 0u;
    PCB_UNROLL
    for (int d = 0; d < 4; ++d) {      // d < 3: edge DoF of component d; d == 3: cell centre
        double u[3];
        PCB_UNROLL
        for (int ax = 0; ax < 3; ++ax) u[ax] = (d == 3 || d == ax) ? ((double)i[ax] + 0.5) / (double)N : (double)i[ax] / (double)N;
        bool in, am;
        pcb_geom_point(g, u[0], u[1], u[2], in, am);
        m |= (in ? 1u : 0u) << d;
        a |= (am ? 1u : 0u) << d;
    }
    mask[p] = (unsigned char)m;
    amb[p] = (unsigned char)a;
}

// ---- x0 = U[0,1) + i U[0,1) on the device: counter-based (splitmix64 of (seed, column, element)) ---------
PCB_HD unsigned long long pcb_mix64(unsigned long long z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
// The value of global row r_g = c*nn + cell depends on (seed, column, r_g) only, so a slab context (rows [c][off .. off+nloc))
// generates exactly its part of the vector a full context would.
__global__ void __launch_bounds__(256) k_fill_uniform(PcbColListW cols, long long nloc, long long nn, long long off, int col0,
                                                      unsigned long long seed) {
    cplx* __restrict__ Y = cols.p[blockIdx.y];
    const unsigned long long base = pcb_mix64(seed ^ (0xD1B54A32D192ED03ull * (unsigned long long)(col0 + blockIdx.y + 1)));
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < 3 * nloc; r += (long long)gridDim.x * blockDim.x) {
        const unsigned long long rg = (unsigned long long)((r / nloc) * nn + off + r % nloc);
        const unsigned long long a = pcb_mix64(base + 2ull * rg);
        const unsigned long long b = pcb_mix64(base + 2ull * rg + 1ull);
        Y[r] = cmake((double)(a >> 11) * (1.0 / 9007199254740992.0), (double)(b >> 11) * (1.0 / 9007199254740992.0));
    }
}
