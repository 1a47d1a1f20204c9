// pcb200 -- common device/host definitions for the sm_100a kernels.
//
// Layout (DESIGN.md "Data layout in HBM"): a *column* is one vector of the block X,
// stored planar: 3 component grids back to back, each N^3 complex128 with i0 fastest:
//     elem(c, i0, i1, i2) = c*nn + i0 + N*i1 + N*N*i2          (nn = N^3)
// which is exactly the reference's row index r (discretization.py:326-328).  A block of
// k columns is k such vectors, each contiguous (column-major), so every kernel streams
// 128-bit vectors; the reference's (3nn, k) row-major layout exists only at the C ABI
// boundary (pcb_block_upload / pcb_block_download).
#pragma once

#ifdef PCB_EMU
#include "emu_cuda.h"   // tests/emu: host emulation of the CUDA execution model (tests only)
#else
#include <cuda_runtime.h>
#endif

#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>

typedef double2 cplx;

#define PCB_HD __host__ __device__ __forceinline__
#define PCB_D __device__ __forceinline__

#ifdef PCB_EMU
#define PCB_LAUNCH(kernel, grid, block, smem, stream, ...) \
    pcbemu::launch((grid), (block), (smem), [=]() { kernel(__VA_ARGS__); })
#define PCB_DYN_SMEM(type, name) type* name = reinterpret_cast<type*>(pcbemu::dyn_smem())
#define PCB_UNROLL
#else
#define PCB_LAUNCH(kernel, grid, block, smem, stream, ...) \
    kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__)
#define PCB_DYN_SMEM(type, name)                                  \
    extern __shared__ __align__(16) unsigned char pcb_dyn_smem_[]; \
    type* name = reinterpret_cast<type*>(pcb_dyn_smem_)
#define PCB_UNROLL _Pragma("unroll")
#endif

// ---- complex helpers ---------------------------------------------------------------
PCB_HD cplx cmake(double re, double im) { cplx r; r.x = re; r.y = im; return r; }
PCB_HD cplx cadd(cplx a, cplx b) { return cmake(a.x + b.x, a.y + b.y); }
PCB_HD cplx csub(cplx a, cplx b) { return cmake(a.x - b.x, a.y - b.y); }
PCB_HD cplx cmul(cplx a, cplx b) { return cmake(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
PCB_HD cplx cmulc(cplx a, cplx b) { /* conj(a) * b */ return cmake(a.x * b.x + a.y * b.y, a.x * b.y - a.y * b.x); }
PCB_HD cplx cconj(cplx a) { return cmake(a.x, -a.y); }
PCB_HD cplx cneg(cplx a) { return cmake(-a.x, -a.y); }
PCB_HD cplx cscale(cplx a, double s) { return cmake(a.x * s, a.y * s); }
PCB_HD double cabs2(cplx a) { return a.x * a.x + a.y * a.y; }
PCB_HD cplx cfma(cplx a, cplx b, cplx c) { /* a*b + c */
    return cmake(fma(a.x, b.x, fma(-a.y, b.y, c.x)), fma(a.x, b.y, fma(a.y, b.x, c.y)));
}
PCB_HD cplx cfmac(cplx a, cplx b, cplx c) { /* conj(a)*b + c */
    return cmake(fma(a.x, b.x, fma(a.y, b.y, c.x)), fma(a.x, b.y, fma(-a.y, b.x, c.y)));
}

// FP64 tensor-core MMA (DMMA): D(8x8) += A(8x4) B(4x8).  Fragment layout (PTX ISA, m8n8k4 .f64):
//   a = A[lane>>2][lane&3],  b = B[lane&3][lane>>2],  (c0, c1) = C[lane>>2][2*(lane&3) + {0,1}].
#ifdef PCB_EMU
PCB_D void pcb_dmma(double& c0, double& c1, double a, double b) { pcbemu::mma884(c0, c1, a, b); }
#else
PCB_D void pcb_dmma(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
#endif

#include "pcb_codelets.cuh"

// ---- error handling -------------------------------------------------------------------
void pcb_set_error(const char* fmt, ...);
#define PCB_CUDA_OK(expr)                                                                 \
    do {                                                                                  \
        cudaError_t e_ = (expr);                                                          \
        if (e_ != cudaSuccess) {                                                          \
            pcb_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
            (void)cudaGetLastError(); /* a recoverable failure (e.g. cudaMalloc) must not poison later launch checks */ \
            return -1;                                                                    \
        }                                                                                 \
    } while (0)
// same, running CLEANUP (a statement) before returning: frees partially built objects on the failure paths
#define PCB_CUDA_OK_OR(expr, CLEANUP)                                                     \
    do {                                                                                  \
        cudaError_t e_ = (expr);                                                          \
        if (e_ != cudaSuccess) {                                                          \
            pcb_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
            (void)cudaGetLastError();                                                     \
            CLEANUP;                                                                      \
            return -1;                                                                    \
        }                                                                                 \
    } while (0)

// ---- operator description shared by all kernels ---------------------------------------
// Fourier symbols are generated on the fly from nine 1-D tables (SURVEY A.2-A.3):
//     K_c(i0,i1,i2) = T[c][0][i0] + T[c][1][i1] + T[c][2][i2],
//     T[c][j][l]    = (CT[c][j]*D1[l] + (j==c) * i*alpha_c*D0[l]) / SCAL
// replacing the reference's 192*N^3-byte symbol arrays (fft_blocks, discretization.py:301-346).
enum { PCB_DIEL_NONE = 0, PCB_DIEL_CHIRAL = 1, PCB_DIEL_TRIVIAL = 2, PCB_DIEL_CROSSDOF = 3, PCB_DIEL_MATERIALS = 4 };

// Large-grid mode over peer memory (NVLink): the columns of one distributed apply live as SLABS on all ranks -- rank g holds the
// i2 planes [zb[g], zb[g+1]) of every column as [c][local cell] -- and the x passes of the operator read / write them in place
// through pointers mapped with CUDA IPC (device-resident table, one per context).
#define PCB_MAXC_DIST 32
#define PCB_MAXW 8
struct PcbDist {
    int world;
    int zb[PCB_MAXW + 1];
    const double2* src[PCB_MAXC_DIST][PCB_MAXW];   // input column j, slab of rank g
    double2* dst[PCB_MAXC_DIST][PCB_MAXW];         // output column j, slab of rank g
};

struct PcbStencil { int k; double w[8]; };   // averaging stencil of the cross-DoF dielectric: taps w[j] at offsets (1-k+j), j < 2k
PCB_HD int pcb_wrap(int i, int N) { i %= N; return i < 0 ? i + N : i; }

struct PcbOp {
    int N;
    long long nn;             // N^3
    long long nloc;           // cells owned by the context: N^3, or (z1 - z0) N^2 on a slab context (large-grid mode)
    int z0;                   // first i2 plane of the slab (0 on a full context)
    const cplx* T;            // [3][3][N] symbol tables (device)
    double gamma;             // penalty gamma (= pnt; the symbols in T are already / SCAL)
    double shift;             // shift added by H
    double pshift;            // shift seen by the preconditioner (= shift / SCAL^2)
    double inv_n3;            // 1 / N^3 (normalisation of the inverse transform)
    int diel;                 // PCB_DIEL_*
    union {
        const unsigned char* mask;  // [nn] bit c: edge DoF of component c in Omega_1; bit 3: volume DoF
        const unsigned char* mat;   // materials: [3 nn] material index of row r = c nn + p (natural order)
    };
    union {
        const unsigned* mbits;      // plane mode: [c][i0][slot][k1] words, bit k2 = component c of (i0, i1 = coord(slot), i2 = lout(k1,k2)) in Omega_1
        const unsigned char* matp;  // materials, plane mode: the index bytes of each z item, in the item order of mbits (k_mat_bytes)
    };
    union {
        const unsigned* mbits2;     // five-sweep plane pass (k_mid2): [c][i0][d][col] words, bit k2 (k_mask_bits2)
        const double* inv_eps;      // materials: [n_mat] 1 / eps of each material (index 0: the background)
    };
    const unsigned char* maskp2; // the same byte mask in the slot order of the five-sweep plane pass (k_mask_plane2), coupled dielectric
    const unsigned char* maskp; // plane mode, coupled dielectric: the byte mask in plane-slot order, [i0][row][col] = mask(i0, coord(col), coord(row))
    PcbStencil sten;            // cross-DoF dielectric: its averaging stencil (the fused stencil-on-load of the plane pass)
    int mid_five;               // plane mode: 1 = the five-sweep plane pass (k_mid2), 0 = the seven-sweep one (k_mid)
    const PcbDist* dist;        // large-grid mode over peer memory: slab pointers of the columns (device memory), else null
    const int* ctab;            // plane mode: [0, N) column slot -> grid index (coord), [N, 2N) grid index -> column slot, [2N, 4N) the same for rows
    int zsplit;                 // plane mode: 1 = z-split form (half planes, ZSplit in pcb_operator.cuh)
    double ediag[3];          // diagonal entries inside Omega_1 (chiral: 1/eps for all three)
    cplx eoff[3];             // eps_12, eps_13, eps_23 (trivial / crossdof)
};

// Fourier symbol k_c at a grid point from the 1-D tables.
struct Sym3 { cplx k[3]; };
PCB_D Sym3 pcb_symbol(const cplx* __restrict__ T, int N, int i0, int i1, int i2) {
    Sym3 s;
    PCB_UNROLL
    for (int c = 0; c < 3; ++c) {
        const cplx a = __ldg(T + (c * 3 + 0) * N + i0);
        const cplx b = __ldg(T + (c * 3 + 1) * N + i1);
        const cplx d = __ldg(T + (c * 3 + 2) * N + i2);
        s.k[c] = cmake(a.x + b.x + d.x, a.y + b.y + d.y);
    }
    return s;
}
