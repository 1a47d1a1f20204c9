/* pcb200 -- C ABI of the B200-native photonic-crystal hot path (libpcb200.so).
 *
 * Drop-in boundary for paper_2's data-parallel path.  The reference is pure Python over
 * CuPy (no FFI of its own), so each entry point below names the reference call it replaces
 * (paths relative to /root/reference/paper_2).  Host code (Python, ctypes) owns the control
 * flow; everything that touches O(N^3) data is behind these functions.
 *
 * Conventions
 *   - complex128 everywhere = two doubles (re, im); "cols" arguments are host arrays of DEVICE
 *     pointers, one per column; a column is one vector of 3*N^3 complex128 stored planar
 *     [component c][i2][i1][i0] (i0 fastest) = the reference's row index r = c*nn + i0 + N*i1 + N^2*i2
 *     (discretization.py:326-328).
 *   - return value: 0 ok; < 0 CUDA / argument error, message via pcb_last_error().
 *   - every call is ordered on the context's stream; calls that write HOST memory return after the
 *     data is visible.  One context per GPU and per host thread.
 *   - there is no CPU fallback: pcb_ctx_create fails when no CUDA device is present.
 */
#ifndef PCB200_H
#define PCB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pcb_ctx pcb_ctx;     /* one GPU + one grid size N: stream, twiddles, workspaces        */
typedef struct pcb_diel pcb_diel;   /* dielectric M: bit mask of Omega_1 + eps entries                 */
typedef struct pcb_op pcb_op;       /* one k-point: symbol tables, gamma, shift, (optional) dielectric */

/* dielectric kinds (discretization.py:352 chiral_handle, :368 pseudochiral_trivial_handle,
 * :403 pseudochiral_crossdof_handle; NONE = `Diels = lambda x: x`, numerical_experiments.py:227; MATERIALS: several isotropic
 * materials, one index per edge DoF, created by pcb_diel_create_materials) */
enum { PCB_DIEL_KIND_NONE = 0, PCB_DIEL_KIND_CHIRAL = 1, PCB_DIEL_KIND_TRIVIAL = 2, PCB_DIEL_KIND_CROSSDOF = 3,
       PCB_DIEL_KIND_MATERIALS = 4 };

/* pcb_apply modes */
enum {
    PCB_APPLY_FFT = 0,   /* unnormalised forward 3-D DFT of every component (cupyx fftn, pcfft.py:149)            */
    PCB_APPLY_IFFT = 1,  /* inverse 3-D DFT with 1/N^3 (ifftn, pcfft.py:151)                                      */
    PCB_APPLY_A = 2,     /* AMA(x, a_fft, Diels)            pcfft.py:130-158                                      */
    PCB_APPLY_H = 3,     /* AMA_BB(x, a_fft, b_fft, Diels, shift)   pcfft.py:160-181                              */
    PCB_APPLY_P = 4,     /* H_block(x, inv_fft)  = K_P^-1 x  pcfft.py:50-70 with discretization.py:284-295        */
    PCB_APPLY_M = 5,     /* Diels(x) in real space          discretization.py:352-453                             */
    PCB_APPLY_KA = 6,    /* A_block_kernel(x, D_A)           pcfft.py:32-43 / _kernels.py:43-71                   */
    PCB_APPLY_KAH = 7,   /* A_block_kernel(x, -conj(D_A))    pcfft.py:148                                         */
    PCB_APPLY_KB = 8,    /* H_block_kernel(x, D_B) = gamma K_B x   pcfft.py:18-30,176 / _kernels.py:13-41         */
    PCB_APPLY_DFIELD = 9, /* D = FFT3(K_A^H x): the real-space field of AMA (pcfft.py:148-149), natural layout        */
    PCB_APPLY_EFIELD = 10, /* E = M D (the dielectric applied to that field), natural layout                         */
    PCB_APPLY_EFOURIER = 11 /* E^ = IFFT3(M FFT3(K_A^H x)): AMA before its last K_A (A x = K_A E^), natural layout   */
};

const char* pcb_last_error(void);
const char* pcb_backend(void);                 /* "cuda-sm_100a" (product) or "host-emu" (tests/emu only) */
int pcb_device_count(int* n);
int pcb_supported_sizes(int* sizes, int cap);  /* returns how many grid sizes N have FFT plans */

int pcb_ctx_create(int device, int N, pcb_ctx** ctx);
void pcb_ctx_destroy(pcb_ctx* ctx);
long long pcb_ctx_trim(pcb_ctx* ctx);               /* frees the context's cached E^ columns of pcb_band_velocity; returns the bytes freed */
int pcb_sync(pcb_ctx* ctx);
int pcb_launch_count(pcb_ctx* ctx, long long* n);   /* kernels launched by this context so far */
/* pass-structure switches (A/B measurements, tests): "plane", "plane_coupled", "plane_cross" (0 / 1 / 2), "mid_five" (-1 auto, 0, 1),
 * "plane_split" (0 / 1: z-split form of the plane mode where a size has both forms; always on for N = 128, 144, 160; dielectrics
 * must be re-created after a change); defaults from the PCB200_* environment variables; seen by operators created or updated
 * afterwards */
int pcb_ctx_option(pcb_ctx* ctx, const char* name, int value);
/* stream ordering between two contexts of one process without a host sync (16 slots per context): pcb_ctx_record marks the work
 * enqueued on ctx so far, pcb_ctx_wait makes later work of `waiter` start after that mark (the reference is single-stream) */
int pcb_ctx_record(pcb_ctx* ctx, int slot);
int pcb_ctx_wait(pcb_ctx* waiter, pcb_ctx* owner, int slot);
int pcb_mem_info(pcb_ctx* ctx, size_t* free_bytes, size_t* total_bytes);
int pcb_timer_start(pcb_ctx* ctx);                  /* CUDA event on the context's stream */
int pcb_timer_stop(pcb_ctx* ctx, float* ms);        /* second event + synchronize + elapsed */

/* memory (replaces cupy.empty / cp.asarray / .get(); environment.py, lobpcg.py:365-369) */
int pcb_malloc(pcb_ctx* ctx, size_t bytes, void** dptr);
int pcb_free(pcb_ctx* ctx, void* dptr);
int pcb_host_alloc(size_t bytes, void** hptr);      /* pinned host memory */
int pcb_host_free(void* hptr);
int pcb_memcpy_h2d(pcb_ctx* ctx, void* dst, const void* src, size_t bytes);
int pcb_memcpy_d2h(pcb_ctx* ctx, void* dst, const void* src, size_t bytes);
int pcb_memcpy_d2d(pcb_ctx* ctx, void* dst, const void* src, size_t bytes);
int pcb_memset_zero(pcb_ctx* ctx, void* dst, size_t bytes);
/* (R, k) row-major host block (the reference's array layout, leading dimension ld elements) <-> planar device columns */
int pcb_block_upload(pcb_ctx* ctx, const void* host_rm, long long ld, int k, void* const* cols);
int pcb_block_download(pcb_ctx* ctx, void* host_rm, long long ld, int k, const void* const* cols);
/* x0 = rand + 1j*rand generated on the device (cp.random.rand, numerical_experiments.py:66,426): counter-based, seeded */
int pcb_fill_uniform(pcb_ctx* ctx, int k, void* const* cols, unsigned long long seed);

/* dielectric (discretization.py:352-453).  ind_e: int64 row indices r in [0, 3nn) of edge DoFs in Omega_1
 * (dielectric.diel_io_index(..., 'edge')); ind_v: int64 cell indices in [0, nn) of volume DoFs (trivial only).
 * ediag[3]: diagonal value inside Omega_1 per component (chiral: 1/eps);  eoff[6] = (re,im) of eps_12, eps_13, eps_23.
 * stencil: the 2k averaging weights mfd_stencil(k, 0) (crossdof only). */
int pcb_diel_create(pcb_ctx* ctx, int kind, const int64_t* ind_e, long long n_e, const int64_t* ind_v, long long n_v,
                    const double* ediag, const double* eoff, int k, const double* stencil, pcb_diel** diel);
/* Several isotropic materials: (M x)_r = inv_eps[mat[r]] x_r.  mat: HOST array of n = 3 N^3 material indices in row order
 * r = c N^3 + p (index 0: the background, whose inv_eps[0] need not be 1); inv_eps: HOST array of n_mat values 1 / eps, 1 <= n_mat
 * <= 256.  inv_eps = {1, 1/eps} with mat = 1 on ind_e is the chiral M.  Fails with -1 (nothing allocated) when n != 3 N^3, n_mat is
 * out of range, some mat[r] >= n_mat or some inv_eps is not finite and > 0; with -2 on a slab context.  A / H run the plane pass
 * where the plane mode applies (seven sweeps: "mid_five" is ignored) and the five-pass operator elsewhere; pcb_field_energy's
 * e_in is the energy in the rows with mat[r] != 0. */
int pcb_diel_create_materials(pcb_ctx* ctx, const uint8_t* mat, long long n, const double* inv_eps, int n_mat, pcb_diel** diel);
/* Replace the 1 / eps table of a materials dielectric in place (dispersive materials: eps at a new frequency).  inv_eps: HOST array
 * of n_mat values.  One copy on the context's stream into the table's own allocation, behind the work already queued: every
 * operator built on diel sees the new values from its next launch; the index map and the plane-pass index bytes are not rebuilt.
 * The call waits for the copy, so inv_eps may be reused on return.  Fails with -1, the old table in force, when diel is not of
 * kind MATERIALS, n_mat differs from the n_mat it was created with, or some value is not finite and > 0. */
int pcb_diel_set_inv_eps(pcb_diel* diel, const double* inv_eps, int n_mat);
void pcb_diel_destroy(pcb_diel* diel);

/* operator for one k-point (numerical_experiments.py:434-448 pc_mfd_handle).  tables: [3][3][N] complex128,
 * K_c(i0,i1,i2) = tables[c][0][i0] + tables[c][1][i1] + tables[c][2][i2]  (= a_fft, fft_blocks discretization.py:301-346);
 * gamma = pnt, shift = relax_opt[0] as used by H, pshift the shift inside K_P^-1 (= shift for SCAL = 1). */
int pcb_op_create(pcb_ctx* ctx, const double* tables, double gamma, double shift, double pshift, pcb_diel* diel,
                  pcb_op** op);
int pcb_op_update(pcb_op* op, const double* tables, double gamma, double shift, double pshift, pcb_diel* diel);
void pcb_op_destroy(pcb_op* op);

/* Y_j = op(X_j), j < ncols.  in[j] == out[j] (in place) is allowed for every mode except PCB_APPLY_H outside the plane mode
 * (which re-reads X in its last pass), PCB_APPLY_A with the cross-DoF dielectric on the plane halves and PCB_APPLY_M with the
 * cross-DoF dielectric (out serves as work space of the plane halves / the stencil gathers); the call fails with -2 in those
 * cases, before anything is enqueued: no output column is written.  Distinct columns must not overlap.
 * PCB_APPLY_DFIELD / PCB_APPLY_EFIELD (forward x, y, z passes; EFIELD then M point-wise in place on out, or the cross-DoF stencil
 * from the context's scratch into out) read X only in their first pass: in place is allowed for every dielectric.
 * PCB_APPLY_EFOURIER runs the passes of PCB_APPLY_A (the last x pass without K_A) and follows its in-place rule. */
int pcb_apply(pcb_op* op, int mode, int ncols, const void* const* in, void* const* out);

/* Y_host = op(X_host): the reference-facing call with host arrays -- x_host, y_host are the reference's row-major (3N^3, k)
 * blocks (leading dimensions in elements; pinned memory from pcb_host_alloc makes the copies asynchronous).  Chunks of 8 columns
 * flow through an H2D / compute / D2H pipeline on three streams so that both PCIe directions overlap.  Replaces
 * `cp.asarray(x)` + H_func / A_func / P_func + `.get()` of a NumPy caller (numerical_experiments.py:73-85). */
int pcb_apply_host(pcb_op* op, int mode, int k, const void* x_host, long long ldx, void* y_host, long long ldy);

/* Same as pcb_apply for PCB_APPLY_A / PCB_APPLY_H, with a CUDA event between the passes: pass_ms[i] = device time of
 * pass i.  Five-pass operator: (x-forward+K_A^H, y-forward, z-forward+M+z-inverse, y-inverse, x-inverse+K_A+gamma K_B+shift),
 * npass <- 5; plane mode (N % 8 == 0, N <= 120 on whole planes; N = 128, 144, 160 on half planes with the radix-2 step of the z
 * transform inside the x passes; identity / isotropic M, and the coupled 3x3 M on clusters of three CTAs -- whole planes when
 * N % 3 == 0): (x-forward, fused y/z/M/z/y plane pass, x-inverse), npass <- 3; cross-DoF M: plane sizes (x-forward, y/z forward on
 * planes, [stencil kernel, or fused into the next pass: npass <- 4,] z/y inverse on planes, x-inverse), npass <- 5, other sizes
 * (x, y, z forward, stencil, z, y, x inverse), npass <- 7.
 * pass_ms must hold 8 floats.  Measurement aid for bench.py's per-pass roofline; not used by the solver. */
int pcb_apply_timed(pcb_op* op, int mode, int ncols, const void* const* in, void* const* out, float* pass_ms, int* npass);

/* Electric energy of modes in the dielectric.  For column x_j let D = FFT3(K_A^H x_j) (unnormalised, = PCB_APPLY_DFIELD) and
 * E = M D, rows r = c N^3 + p:  e_tot[j] = Re sum_r conj(D_r) E_r / N^3 (= x_j^H A x_j, independent of gamma and the shift) and
 * e_in[j] = the same sum over the rows in Omega_1 (bit c of the dielectric mask at cell p: the edge DoFs of ind_e); e_in = 0 without
 * a dielectric.  e_in / e_tot is the fraction f of the mode's electric energy inside the dielectric (0 <= f <= 1 for the chiral M;
 * the pseudochiral M couples rows, so a single row's term may be negative and f may leave [0, 1] slightly).  e_in, e_tot: HOST
 * arrays of ncols doubles; x is read only.  Any ncols (launches of 32 columns); the reduction has a fixed grid and order, so a
 * column gives the same bits at any width and on every call.  Runs the forward passes of A (the plane layout where A runs in plane
 * mode, else the natural layout) into the context's scratch and a reduction kernel over them.  A slab context fails with -2. */
int pcb_field_energy(pcb_op* op, int ncols, const void* const* x, double* e_in, double* e_tot);

/* Electric energy of modes per material (materials dielectric).  With D and E = M D as for pcb_field_energy,
 *     e_mat[j][m] = Re sum_{r: mat[r] = m} conj(D_r) E_r / N^3,   m < n_mat,
 * e_mat a HOST array [ncols][n_mat].  sum_m e_mat[j][m] = e_tot and sum_{m != 0} e_mat[j][m] = e_in of pcb_field_energy (to
 * rounding); since E_r = D_r / eps_m, dlambda/deps_m = -e_m / (eps_m x^H x) (Hellmann-Feynman).  Any ncols, in launches of 32
 * columns; x is read only.  Runs the forward passes of A into the scratch as pcb_field_energy does, then a kernel that bins the
 * rows by material without timing-dependent atomics over a grid fixed by the context, and a fixed-order sum: a column's row of
 * e_mat has the same bits at any width and on every call.  Fails with -1 when op has no dielectric or one of another kind, or
 * n_mat differs from the dielectric's; with -2 on a slab context.  Nothing is written to e_mat in a refusal. */
int pcb_material_energy(pcb_op* op, int ncols, const void* const* x, int n_mat, double* e_mat);

/* Band velocity matrices (Hellmann-Feynman).  The symbols depend on the k-point alpha only through the Bloch term of the diagonal
 * tables, dK_c/dalpha_d = delta_cd tau_d[i_d]; dtables = tau as a HOST array [3][N] complex128 (FourierSymbols.dtables).  With
 * E^ = PCB_APPLY_EFOURIER of x and, for d, a, b cyclic, W_d[i][j] = x_i^H ((tau_d e_d) x E^_j)
 *     = sum_q tau_d[q_d] (conj(x_i,b) E^_j,a - conj(x_i,a) E^_j,b),
 * the call returns V_d = W_d + W_d^H = X^H (dA/dalpha_d) X (Hermitian): V HOST, [3][ncols][ncols] complex128 row-major;
 * xx[j] = x_j^H x_j and xax[j] = Re x_j^H A x_j = Re sum_q conj(x_j) . (K x E^_j) (HOST doubles), so that
 * dlambda_j/dalpha_d = V_d[j][j] / xx[j] for a band that is not degenerate.  1 <= ncols <= 32 (the solver's block width); x is
 * read only.  Runs the passes of A with a plain last x pass into a buffer of ncols columns kept by the context (released by
 * pcb_ctx_trim), then the reduction kernel over a grid that depends on the context only and a fixed-order sum: entry (d, i, j)
 * gets the same bits at any width (V of a subset of columns is the matching sub-block of a wider call) and on every call.
 * ncols > 32 and slab contexts fail with -2, before anything is written to V, xx or xax. */
int pcb_band_velocity(pcb_op* op, int ncols, const void* const* x, const double* dtables, void* V, double* xx, double* xax);

/* LOBPCG block kernels
 * pcb_residual: r_j = lambda_j x_j - hx_j (lobpcg.py:394-395); norms2[j] = ||r_j||^2 (environment.norms :131-143);
 *   precond = 0: w_j = r_j;  1: w_j = K_P^-1 r_j (p_func fused, lobpcg.py:442);  2: w_j = K_P^-1 c64(r_j) and
 *   3: w_j = c64(r_j), the residual rounded to complex64 and widened again -- the single-precision hand-over to the
 *   preconditioner of lobpcg_sep_softlock_mixedprecision (lobpcg.py:574-577).  norms2 (always of the unrounded r_j) is HOST memory. */
int pcb_residual(pcb_op* op, int precond, int ncols, const void* const* x, const void* const* hx, void* const* w,
                 const double* lambda, double* norms2);
/* G = S^H S, T = S^H HS, both hermitized (orthogonalization.py:26-33,143-144); n x n row-major complex128 on the HOST.
 * Only one triangle (of 4x4 column blocks) is accumulated and completed by conjugation: HS must be H S with H Hermitian,
 * so that S^H HS is Hermitian up to rounding -- which is the only way the solver uses it. */
int pcb_gram2(pcb_ctx* ctx, int n, const void* const* s, const void* const* hs, void* G, void* T);
/* Same, accumulating only the rows of the first `ntop` columns (rounded up to a multiple of 8): rows a < ntop of G and T (and,
 * by Hermitian completion, their columns) are valid, the rest is zero.  Used by the solver's incremental Gram update, where
 * only the new block W changes between iterations and the [X P] blocks follow from the previous Rayleigh-Ritz rotation.
 * When ntop (rounded up) < n the rows of T are formed as (hs_a)^H s_b -- equal to s_a^H hs_b for the Hermitian H this
 * is defined for -- so only the first ntop (rounded up to 8) columns of `hs` are read; the other entries of `hs` may be NULL. */
int pcb_gram2_top(pcb_ctx* ctx, int n, int ntop, const void* const* s, const void* const* hs, void* G, void* T);
/* _sep_update_after_rr (lobpcg.py:1248-1270): s/hs list the n_loc input columns [X(m) | W_act | P_act];
 * E is (n_loc x m) row-major complex128 on the host.  Pn = [W_act P_act] E[m:], X <- X E[:m] + Pn (in place), P <- Pn. */
int pcb_update(pcb_ctx* ctx, int m, int n_loc, void* const* s, void* const* hs, void* const* p_out, void* const* hp_out,
               const void* E);
/* pcb_update and, fused into the same pass for m <= 16, the NEXT iteration's residual / norms / preconditioner (lobpcg.py:1248-1270
 * followed by :394-397,442): with the new Ritz values `lambda` (m doubles, host), w_out_j = K_P^-1 (lambda_j x_j - hx_j) on the updated
 * X, HX and norms2[j] = ||lambda_j x_j - hx_j||^2 (HOST).  The residual is formed from the update's accumulators, so X and HX are not
 * re-read; wider blocks run pcb_update + pcb_residual back to back.  w_out may be the W columns that are inputs of the update. */
int pcb_update_resid(pcb_op* op, int m, int nl, void* const* s, void* const* hs, void* const* p_out, void* const* hp_out, const void* E,
                     const double* lambda, void* const* w_out, double* norms2);
/* the same in two halves: _start enqueues the kernels and returns (host bookkeeping overlaps the GPU), _wait delivers norms2 */
int pcb_update_resid_start(pcb_op* op, int m, int nl, void* const* s, void* const* hs, void* const* p_out, void* const* hp_out, const void* E,
                           const double* lambda, void* const* w_out);
int pcb_update_resid_wait(pcb_op* op, int m, double* norms2);
/* the last tiled block kernel pcb_gram2 / pcb_gram2_top / pcb_update / pcb_update_resid planned on this context: its name (e.g.
 * "k_gram2", "k_update<32,1,3>", "k_update_res"), the CTAs it was launched with and the row tiles they share (test and measurement
 * aid: which instantiation and how many tiles per CTA a shape selects) */
int pcb_block_launch_info(pcb_ctx* ctx, char* name, int cap, long long* grid, long long* tiles);
/* out[j] = a_j^H b_j (complex128 on the host) -- diag(x^H y) of numerical_experiments.py:105-111, environment.dots */
int pcb_coldots(pcb_ctx* ctx, int ncols, const void* const* a, const void* const* b, void* out);
/* y_j = alpha x_j + beta y_j */
int pcb_axpby(pcb_ctx* ctx, int ncols, const void* const* x, void* const* y, double alpha, double beta);

/* Geometry (dielectric.py:104-261: mesh3d_edge_dofs / mesh3d_volume_dofs, coo = mesh @ inv(ct^T), FLAG_<lattice>): Omega_1 of a
 * lattice evaluated on the device for all 4 N^3 DoF points.  kind: 0 sc_flat1, 1 sc_flat2, 2 sc_curv, 3 bcc_sg, 4 bcc_dg, 5 fcc;
 * minv = inv(ct^T) (9 doubles, row-major).  host_mask[cell] bit c = edge DoF of component c inside, bit 3 = volume DoF inside;
 * host_amb[cell] marks (same bits) the DoFs whose decision margin is below 1e-10 -- the caller re-evaluates those with the
 * reference's NumPy expression, which keeps the index sets bit-identical.  Both arrays: N^3 bytes of HOST memory. */
int pcb_geometry_mask(pcb_ctx* ctx, int kind, const double* minv, unsigned char* host_mask, unsigned char* host_amb);

/* ---- large-grid mode (BASELINE config 5; SURVEY 8e-ii): dense phase row-sharded, operator on whole columns ------------
 * A SLAB context owns the i2 planes [z0, z1) of every column: its "column" is 3 * (z1-z0) * N^2 complex128 ([c][local cell]),
 * and pcb_residual / pcb_gram2 / pcb_update / pcb_coldots / pcb_axpby / pcb_fill_uniform / block up/download work on it
 * unchanged (pcb_apply: PCB_APPLY_P only).  With a communicator attached, pcb_gram2, pcb_residual and pcb_coldots
 * all-reduce their n_loc x n_loc / per-column results over the ranks with NCCL before returning them -- the only
 * collective of the dense phase.  The reference has no counterpart (single GPU, lobpcg.py / orthogonalization.py:143-144). */
int pcb_ctx_create_slab(int device, int N, int z0, int z1, pcb_ctx** ctx);
int pcb_comm_unique_id(void* id128);                                   /* rank 0: ncclGetUniqueId (128 bytes) */
int pcb_comm_init(pcb_ctx* ctx, const void* id128, int rank, int world); /* every rank: ncclCommInitRank on the slab context */
int pcb_comm_set_host_callbacks(pcb_ctx* ctx, void* allreduce_cb, void* p2p_cb);  /* host-emu test build only */
int pcb_comm_destroy(pcb_ctx* ctx);
/* Large-grid mode over PEER MEMORY (NVLink): instead of gathering whole columns with pcb_slab_exchange, the first and the last
 * FFT pass of the operator read and write the slabs of all ranks in place (CUDA IPC mappings), tile by tile, so the transfer
 * overlaps the transforms and no staging copy of the block exists.
 *   pcb_comm_share   collective: peers[g] <- rank g's allocation `dptr` (base of a pcb_malloc block) mapped into this process
 *   pcb_comm_unshare closes the mappings
 *   pcb_comm_barrier stream-ordered barrier over the ranks (one-element ncclAllReduce on the context's stream)
 *   pcb_apply_dist   PCB_APPLY_A / PCB_APPLY_H on `ncols` columns owned by this rank: src[j*world+g] / dst[j*world+g] are column
 *                    j's input / output slab on rank g, zb[0..world] the slab boundaries, xcopy[j] / work[j] local full columns;
 *                    src == NULL: xcopy[j] already holds the whole input column (gathered with pcb_slab_exchange) and only the
 *                    scatter of the result is fused into the last pass */
int pcb_comm_share(pcb_ctx* ctx, void* dptr, void** peers);
int pcb_comm_unshare(pcb_ctx* ctx, void** peers);
int pcb_comm_barrier(pcb_ctx* ctx);
int pcb_apply_dist(pcb_op* op, int mode, int ncols, const void* const* src, void* const* dst, const int* zb, int world,
                   void* const* xcopy, void* const* work);
/* measurement aid: average device time (ms) of one NCCL all-reduce of `count` doubles over the communicator */
int pcb_comm_allreduce_timed(pcb_ctx* ctx, long long count, int reps, float* ms);
/* slab layout <-> whole columns on their owner rank, one grouped ncclSend/ncclRecv per call (see pcb_capi.cu) */
int pcb_slab_exchange(pcb_ctx* ctx, int to_full, int ncols, const int* owners, const int* zb, void* const* slab_cols,
                      void* const* full_cols);

#ifdef __cplusplus
}
#endif
#endif /* PCB200_H */
