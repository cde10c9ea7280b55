/* xtd_sigma.h -- C-ABI of the B200-native Davidson sigma-vector engine (libxtdsigma.so).
 *
 * Drop-in boundary (SURVEY 8b).  The reference has no FFI: its operator interface is the Python pair
 * `vind, hdiag = obj.gen_vind()` (xtddft/XTDA.py:694-698, xtddft/SF_TDA.py:162-244, xtddft/XSF_TDA.py:1029-1277,
 * xtddft/XSF_TDA_GPU.py:357-729) whose `vind(zs[nvec,dim]) -> [nvec,dim]` is handed to the Davidson solver
 * (xtddft/utils/Davidson.py:21).  This library is what a `vind` implemented on a B200 binds through ctypes:
 * plain pointers and sizes, no torch / numpy types, return code 0 = OK, negative = error
 * (`xtd_last_error()` has the message); nothing throws across the boundary.
 *
 * Conventions
 *   - fp64 everywhere; matrices are row-major with an explicit leading dimension.
 *   - pointers named *_dev are device pointers owned by the caller (kept alive until xtd_destroy);
 *     pointers named *_host are host arrays copied during the call.
 *   - one engine per GPU per process; not thread-safe per engine; all work is enqueued on the stream given to
 *     xtd_set_stream (default: the legacy default stream).
 *   - The engine executes a generic *plan* (channels, exchange block weights, Coulomb blocks, grid kernel,
 *     local terms, layout maps); `xtddft_b200/plan.py` compiles X-TDA / SF-TDA / XSF-TDA into it.
 */
#ifndef XTD_SIGMA_H
#define XTD_SIGMA_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct xtd_engine* xtd_handle;

enum { XTD_FXC_NONE = 0, XTD_FXC_UKS = 1, XTD_FXC_ALDA0 = 2, XTD_FXC_MCOL = 3, XTD_FXC_UKS_TAU = 4, XTD_FXC_MCOL_TAU = 5 };
enum { XTD_SIDE_RIGHT = 0, XTD_SIDE_LEFT = 1, XTD_SIDE_LEFT_T = 2, XTD_SIDE_RIGHT_T = 3 };

typedef struct {
  double flops_gemm;          /* useful FP64 flops issued through the DMMA GEMM since the last reset */
  unsigned long long launches; /* kernels launched by this library since the last reset */
  double ms[12];              /* device time per phase of the last xtd_sigma* call (see XTD_T_* below) */
  double flops[12];           /* DMMA GEMM flops issued inside each phase of the last xtd_sigma* call */
} xtd_stats;
enum { XTD_T_PACK = 0, XTD_T_XC_GEMM = 1, XTD_T_XC_STREAM = 2, XTD_T_K1 = 3, XTD_T_K2 = 4, XTD_T_J = 5,
       XTD_T_LOCAL = 6, XTD_T_UNPACK = 7, XTD_T_TOTAL = 8, XTD_T_K2_SLICE = 9, XTD_T_XC_SLICE = 10 };

const char* xtd_last_error(void);
int xtd_version(void);

/* life cycle -------------------------------------------------------------------------------------------*/
int xtd_create(xtd_handle* out, int nao, long workspace_bytes);
int xtd_destroy(xtd_handle h);
int xtd_set_stream(xtd_handle h, void* cuda_stream);

/* orbitals: C[nao, nmo] of spin 0/1 (replaces the captured mo_coeff of XTDA.py:564-586) */
int xtd_set_mo(xtd_handle h, int spin, const double* c_dev, long ld, int nmo);

/* a trial-vector block z[no, nv]; idx = MO column per internal position, -1 = zero pad orbital.
 * blocks = (start, n) pairs of the 1 or 2 sub-blocks of the occ / vir positions.  Returns the channel id. */
int xtd_add_channel(xtd_handle h, int spin_o, const int* occ_idx_host, int no, int spin_v, const int* vir_idx_host, int nv,
                    const int* o_blocks_host, int nob, const int* v_blocks_host, int nvb);
/* address of channel `ch` inside the internal sigma buffer for `nvec` vectors: element (x,i,a) at
 * base + x*vec_stride + i*ld + a (doubles) */
int xtd_channel_layout(xtd_handle h, int ch, int nvec, long* base, long* vec_stride, long* ld);

/* density fitting (replaces mf.get_jk / get_j / get_k with mf.density_fit(), XTDA.py:520-539, SF_TDA.py:273-276,
 * XSF_TDA.py:857,996).  Declare every exchange term and Coulomb block first, then stream the 3-centre tensor
 * in aux chunks: L[np, nao, nao] (ld_row, stride_p) or lower-triangular packed rows (packed=1, stride_p).
 * The chunk is transformed to the MO blocks each term needs and is not kept. */
int xtd_add_kterm(xtd_handle h, int tensor, int ch, const double* weights_host, int nob, int nvb);
/* Exchange of the TRANSPOSED trial density -- the B-matrix-type term that the hermi = 1 response of the Z-vector / coupled-perturbed
 * operator adds to the direct term above (`vresp(dm + dm.T)`, grad_hb/tdroks_sfu.py:284-298, grad_hb/tduks_sfu.py:249-258):
 *   sigma[i,a] += weight * sum_P sum_jb L^P_ib z_jb L^P_ja
 * on the MO-resident occupied-virtual block of channel `ch` (kept as Lov[P][i][a]); 4 naux no^2 nv flops per vector.  Declare
 * before xtd_df_begin. */
int xtd_add_kterm_t(xtd_handle h, int tensor, int ch, double weight);
int xtd_add_jblock(xtd_handle h, int ch, int r0, int nr, int c0, int nc);
int xtd_set_jmix(xtd_handle h, const double* mix_host, int n);
/* Exchange contraction sigma += U . Lvv of uniform-weight terms: slices = 0 (default) runs it as FP64 DMMA GEMMs; slices = 3..8
 * emulates FP64 on the INT8 tensor cores (tcgen05.mma kind::i8, csrc/ozaki.cuh) with that many 7-bit digits per operand
 * (radix-256 digits: relative truncation 2^(-8 slices) below each row's scale; 6 -> ~1e-12 on sigma) and keeps Lvv as 8-bit
 * planes only.  Call before xtd_df_begin; with it every xtd_df_add chunk but the last must hold a multiple of the scale group
 * (at most 4 aux functions; the Python engine carries ragged remainders over). */
int xtd_set_exchange_emulation(xtd_handle h, int slices);
/* ROHF-form Fock matrices of the spin-adaptation terms (XTDA.py:607-613, XSF_TDA.py:1103-1111: `scf.ROHF(mol).get_veff(dm)`): only
 * their spin difference F_beta - F_alpha = K[D_open] enters the sigma build (h and J cancel).  Declare the open-shell MOs of `spin`
 * before streaming tensor 0; every xtd_df_add then accumulates kopen[p][q] += sum_P sum_u L^P_pu L^P_qu (MO basis, all nmo x nmo,
 * this rank's aux functions; sum over ranks with one all-reduce).  xtd_get_kopen copies it to out_dev[nmo][ld]. */
int xtd_set_open_orbitals(xtd_handle h, int spin, const int* open_idx_host, int n_open);
int xtd_get_kopen(xtd_handle h, double* out_dev, long ld);
int xtd_df_begin(xtd_handle h, int tensor, long naux_local);
int xtd_df_add(xtd_handle h, int tensor, const double* l_dev, long np, long ld_row, long stride_p, int packed);
int xtd_jblock_diag(xtd_handle h, int jb, double* out_dev);   /* out[nr*nc] = sum_P L_ia^2 */

/* grid (replaces ni.block_loop / nr_uks_fxc / nr_uks_fxc_sf_tda(_mc), XTDA.py:514, SF_TDA.py:90-160, 976-1047):
 * ao[nvar, ng, nao] with row stride ld_row and component stride stride_comp, weights[ng], cached kernel:
 *   XTD_FXC_UKS   fxc[2,nvar,2,nvar,ng] unweighted   (numint.cache_xc_kernel)
 *   XTD_FXC_ALDA0 f[ng] weighted                     (SF_TDA.cache_xc_kernel_sf)
 *   XTD_FXC_MCOL  fxc[nvar,nvar,ng] unweighted       (cache_xc_kernel_sf_mc)
 *   XTD_FXC_UKS_TAU / XTD_FXC_MCOL_TAU   meta-GGA: the same layouts with 5 kernel components (rho, grad rho, tau) over the
 *                 4 AO components value + gradient (MGGA_DENSITY_LAPL off, SF_TDA.py:141-152, 1028-1040) */
int xtd_set_grid(xtd_handle h, const double* ao_dev, int nvar, long ng, long ld_row, long stride_comp, const double* w_dev);
int xtd_set_fxc(xtd_handle h, int kind, const double* fxc_dev);
/* Transform the AO values once to the occupied / virtual MO values of every declared channel (phi = ao.Co, phiv = ao.Cv)
 * and build the per-point kernel tables.  Needs the channels, xtd_set_grid and xtd_set_fxc; implied by xtd_finalize.
 * After it returns the ao, weights and (UKS / MCOL) fxc buffers are no longer referenced and may be freed -- call it
 * before streaming the 3-centre tensor when memory is tight.  The ALDA0 kernel f[ng] stays referenced. */
int xtd_grid_commit(xtd_handle h);

/* local terms (Fock blocks, Delta-A couplings; XTDA.py:628-687, XSF_TDA.py:1146-1274):
 *   RIGHT: dst[r,c] += alpha * sum_b src[r,b] M[b,c]   M[mrows=k, mcols=nc]
 *   LEFT : dst[r,c] += alpha * sum_j M[r,j] src[j,c]   M[mrows=nr, mcols=k]
 * and with the source block entering TRANSPOSED (ROHF orbital-Hessian couplings between the open-virtual block of one spin and the
 * closed-open block of the other, grad_hb/tdroks_sfu.py:310,319):
 *   LEFT_T : dst[r,c] += alpha * sum_k M[r,k] src[c,k]   M[mrows=nr, mcols=k]
 *   RIGHT_T: dst[r,c] += alpha * sum_j src[j,r] M[j,c]   M[mrows=k, mcols=nc] */
int xtd_add_local_gemm(xtd_handle h, int side, int dst_ch, int r0, int nr, int c0, int nc, int src_ch, int sr0, int sc0,
                       const double* mat_host, int mrows, int mcols, double alpha);
int xtd_add_rank1(xtd_handle h, int dst_ch, const double* u_host, int src_ch, const double* v_host); /* dense [no,nv] */
int xtd_add_diag(xtd_handle h, int ch, const double* d_host);                                        /* dense [no,nv] */

/* layout maps between the caller's vector (ext_dim) and the internal blocks.
 * gather (per channel): rows = i*nv+a, CSR over external indices.
 * scatter: rows = external index, CSR over (channel, i*ld+a) */
int xtd_set_gather(xtd_handle h, int ch, const long* indptr_host, const long* cols_host, const double* vals_host, long nnz);
int xtd_set_scatter(xtd_handle h, long ext_dim, const long* indptr_host, const long* offs_host, const signed char* chans_host,
                    const double* vals_host, long nnz);

int xtd_finalize(xtd_handle h, int max_nvec);

/* the operator: hz = A z for nvec trial vectors (device pointers, [nvec, ext_dim] contiguous) */
int xtd_sigma(xtd_handle h, int nvec, const double* z_dev, double* hz_dev);
/* multi-GPU: rank-local part (linear in this rank's aux block and grid batch) -> internal buffer; the caller
 * all-reduces xtd_partial_buffer() (NCCL) and calls xtd_sigma_finish, which adds the replicated local terms. */
int xtd_sigma_partial(xtd_handle h, int nvec, const double* z_dev);
int xtd_partial_buffer(xtd_handle h, int nvec, double** ptr, long* nelem);
int xtd_sigma_finish(xtd_handle h, int nvec, double* hz_dev);
/* end-to-end entry with HOST vectors (pinned staging, H2D + sigma + D2H on the engine stream, synchronous) */
int xtd_sigma_host(xtd_handle h, int nvec, const double* z_host, double* hz_host);

int xtd_get_stats(xtd_handle h, xtd_stats* out);
int xtd_reset_stats(xtd_handle h);
/* which GEMM arrangement the grid path uses for nvec vectors: 1 = split-gradient form (value GEMM on either side of the
 * orbital product, gradient halves streamed), 0 = one GEMM per AO component.  Used by the bench to count streamed bytes. */
int xtd_xc_split_form(xtd_handle h, int nvec);
/* how many auxiliary-function chunks (exchange build) and grid chunks the last eager xtd_sigma* call looped over; the
 * environment variables XTD_CHUNK_AUX / XTD_CHUNK_GRID (read by xtd_create) bound the chunk sizes from above */
int xtd_last_chunks(xtd_handle h, long* aux_chunks, long* grid_chunks);

/* Responses of symmetric MO-block densities on the engine's resident blocks (the right-hand side and the W matrix of the Z-vector
 * equation of the gradients, grad_hb/tdroks_sfu.py:241-254,339-351).  Two-channel plans only.  xtd_enable_block_response (before the
 * grid commit and xtd_df_begin) keeps the Coulomb Loo / Lvv of tensor 0 for every channel and the fp64 virtual MO values on the grid.
 * dens_dev, per channel c in order: Doo[no][no] | Dvv[nv][nv] | Dov[no][nv] on the channel's internal positions (Dvo = Dov^T);
 * out_dev, per channel: the occupied-occupied [no][no] and occupied-virtual [no][nv] blocks of
 *     coef[0] J[D_0 + D_1] + coef[3] f_xc[D_c] + coef[1] K_0[D_c] + coef[2] K_1[D_c]
 * (f_xc with the kernel table as uploaded; K_t = exchange with DF tensor t).  x_dev (may be null): X[no_1][nv_0] on (channel-1
 * occupied) x (channel-0 virtual); xout_dev[no_1 + nv_1][no_0 + nv_0] = coef[4] K_0[X] on (channel-1 occupied, virtual) x (channel-0
 * occupied, virtual).  Outputs are this rank's partial sums (aux block, grid batch): all-reduce them over the ranks. */
int xtd_enable_block_response(xtd_handle h);
int xtd_block_response(xtd_handle h, const double* dens_dev, double* out_dev, const double* coef_host, const double* x_dev, double* xout_dev);

/* Davidson subspace algebra on device vectors (Davidson.py:152-271): all row vectors of length n */
int xtd_vec_dots(void* stream, double* g_dev, int ldg, const double* a_dev, long lda, int m, const double* b_dev, long ldb, int k, long n);
int xtd_vec_lincomb(void* stream, double* y_dev, long ldy, const double* x_dev, long ldx, const double* c_dev, int ldc, int m, int k,
                    long n, double beta);
int xtd_vec_residual(void* stream, double* r_dev, const double* ax_dev, const double* x_dev, long ld, const double* e_dev,
                     double* nrm2_dev, int k, long n);
int xtd_vec_precond(void* stream, double* x_dev, long ld, const double* hdiag_dev, const double* shift_dev, double* nrm2_dev, int k,
                    long n);
int xtd_vec_scale(void* stream, double* x_dev, long ld, const double* s_dev, int k, long n);

/* The solver around the operator (replaces `lib.davidson1` / utils/Davidson.py:21-298 as called at XTDA.py:775-777, SF_TDA.py:392-395,
 * XSF_TDA.py:1467-1470): block Davidson with the subspace resident in HBM and the host control flow in C++.  x0_dev [n0, dim] initial
 * vectors, hdiag_dev [dim] the diagonal preconditioner; on return e_host[nroots], conv_host[nroots], x_dev [nroots, dim] (Ritz vectors).
 * Returns the number of roots found (<= nroots) or a negative error code.  Multi-GPU: `allreduce` sums the partial sigma block over the
 * ranks (device buffer of n doubles, on the engine stream; return 0 on success); NULL on a single rank. */
typedef struct {
  double tol, tol_residual /* <= 0: sqrt(tol) */, lindep, level_shift;
  int max_cycle, max_space /* 12: the solver adds 4 (nroots - 1) */, pick_positive /* keep eigenvalues > 1e-3 (X-TDA) */;
  int (*allreduce)(void* ctx, double* dev_buf, long n);
  void* allreduce_ctx;
} xtd_solver_opts;
int xtd_davidson(xtd_handle h, int nroots, const xtd_solver_opts* opts, const double* hdiag_dev, const double* x0_dev, int n0,
                 double* e_host, double* x_dev, int* conv_host, int* ncycle, int* nsigma);

/* host-only pieces of xtd_davidson, exported for the CPU test suite: eigen-decomposition of a symmetric n x n matrix (row-major in,
 * eigenvectors in the columns out, eigenvalues ascending) and Gram-Schmidt coefficients from a Gram matrix (returns the rows kept) */
int xtd_host_sym_eig(double* a, int n, double* w);
int xtd_host_gs_coefficients(const double* g, int n, double lindep, double* t_out);

/* plain GEMM entry (tests / benchmarks of the DMMA kernel): C[M,N] = alpha * A[M,K] * B[N,K]^T */
int xtd_dgemm_tn(void* stream, int m, int n, int k, double alpha, const double* a_dev, long lda, const double* b_dev, long ldb,
                 double* c_dev, long ldc, int accumulate);
/* general form: A is [M,K] row-major when a_kc != 0, else [K,M]; B is [N,K] when b_kc != 0, else [K,N] */
int xtd_dgemm(void* stream, int m, int n, int k, double alpha, const double* a_dev, long lda, int a_kc, const double* b_dev, long ldb,
              int b_kc, double* c_dev, long ldc, int accumulate);
/* FP64 contraction emulated on the INT8 tensor cores (tcgen05.mma kind::i8, Ozaki splitting into `slices` radix-256
 * digit planes per operand; csrc/ozaki.cuh):  C[M,N] (+)= alpha * sum_q A[q][M,K] B[q][N,K]^T  with both operands K-contiguous,
 * row stride ld and q-slice stride sq (even, 16-byte aligned base).  `group` q-slices share one power-of-two row scale and
 * one exact int32 accumulation (0 = choose).  ms_out[3] (may be null) = device time of slicing A, slicing B, the int8 GEMM. */
int xtd_ozaki_gemm(void* stream, int m, int n, int k, int nq, int slices, int group, const double* a_dev, long lda, long sqa,
                   const double* b_dev, long ldb, long sqb, double* c_dev, long ldc, double alpha, int accumulate, double* ms_out);
unsigned long long xtd_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif
