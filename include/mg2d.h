/* mg2d.h -- C ABI of libmg2d_sm100.so: the B200 (sm_100a) hot path of vmos1/2d_multigrid.
 *
 * The reference has no FFI: it is one C++ translation unit (S6/mgrid_ntl.cpp) whose hot path is the member
 * functions of `class Level : Near_null` plus the free functions of modules_main.h.  Each entry point below
 * replaces one of those functions (cited as S6/<file>:<lines>, S6 = code/6_ntl-mg_new_code/
 * 3_combining_laplace_and_wilson/, S2 = code/2_scalar_2d_nontelescoping/telescoping_2d_laplace_Mgrid.cpp).
 *
 * Contract
 *   - plain C: opaque handle, device pointers, ints, doubles, a cudaStream_t passed as void*.
 *   - every call returns 0 on success or a negative MG2D_E* code; mg2d_last_error() gives the text.
 *     No exceptions, no exit().
 *   - the caller owns every field/operator buffer; the library owns only the reduction workspace created by
 *     mg2d_create().  All calls are asynchronous on the given stream and never synchronise.
 *   - one handle per GPU and per stream of work; a handle is not thread-safe.
 *
 * Data layout (device memory, x fastest: site s = x + y*Lx, as S6/level.h:69-75)
 *   dtype MG2D_C128: interleaved (re,im) doubles;  MG2D_C64: interleaved floats.
 *   field      v[s][n]                       n dof per site (level 0 Wilson: n = 2 spin components)
 *   links      U[s][2]                       U_x(s), U_y(s)                     (S6/gauge.h:29-37)
 *   operator   D[s][k][j][i]  k = 0..4       5-point block stencil, slot k: 0 self, 1 x+1, 2 x-1, 3 y+1, 4 y-1
 *                                            (S6/level.h:8).  NOTE: each n x n block is stored COLUMN-major
 *                                            (element (i,j) at j*n+i) so that a warp streams it coalesced.
 *   projector  P[s][ic][jf]                  near-null vectors, nc x nf row-major per fine site
 *                                            (phi_null(s)(ic,jf), S6/near_null.h:12)
 *
 * Strip decomposition (1-D in y): every stencil call works on `Ly` locally owned rows of width `Lx` and takes
 * the two neighbouring rows as separate pointers `lo` (row y-1 of local row 0) and `hi` (row y+1 of the last
 * local row).  On one GPU these are just the last / first owned row (periodic wrap).
 */
#ifndef MG2D_H
#define MG2D_H
#ifdef __cplusplus
extern "C" {
#endif

typedef struct mg2d_ctx mg2d_ctx;
struct mg2d_halo_link;

enum { MG2D_C128 = 0, MG2D_C64 = 1 };
enum { MG2D_OK = 0, MG2D_EINVAL = -1, MG2D_ECUDA = -2, MG2D_EUNSUPPORTED = -3 };
/* stencil modes */
enum { MG2D_MODE_APPLY = 0,   /* out = D in                         Level::f_apply_D   S6/level.h:251-265 */
       MG2D_MODE_RESID = 1 }; /* out = b - D in                     Level::f_residue   S6/level.h:61-77   */
/* reduction slots written by the stencil calls when `dots` != NULL (doubles, device memory, per vector) */
enum { MG2D_DOT_OUT2 = 0,     /* sum |out|^2                        f_get_residue_mag  S6/level.h:79-98   */
       MG2D_DOT_OUTIN_RE = 1, /* Re <out, in> = Re sum conj(out) in (MR smoother)                          */
       MG2D_DOT_OUTIN_IM = 2,
       MG2D_DOT_B2 = 3,       /* sum |b|^2 (MODE_RESID only)                                               */
       MG2D_NDOTS = 4 };

int         mg2d_version(void);
int         mg2d_create(mg2d_ctx** ctx, int device);
int         mg2d_destroy(mg2d_ctx* ctx);
const char* mg2d_last_error(mg2d_ctx* ctx);
int         mg2d_launch_count(mg2d_ctx* ctx);          /* kernels launched through this handle so far */

/* ---- level-0 operators, matrix free ------------------------------------------------------------------ */
/* U(1) Wilson-Dirac: Level::f_compute_lvl0_matrix (wilson branch, S6/level.h:155-172) fused into
 * Level::f_apply_D / f_residue / f_get_residue_mag.  n = 2.  `U_lo` = link row below local row 0. */
int mg2d_wilson_apply(mg2d_ctx*, void* out, const void* in, const void* in_lo, const void* in_hi,
                      const void* U, const void* U_lo, const void* b, double mass, int Lx, int Ly,
                      int mode, int dtype, double* dots, void* stream);
/* materialise the level-0 stencil D[s][5][n][n] (both branches of f_compute_lvl0_matrix, S6/level.h:131-175):
 * stencil 0 = wilson (n=2), 1 = gauged laplace (n=1). */
int mg2d_lvl0_matrix(mg2d_ctx*, void* D, const void* U, const void* U_lo, double mass, int stencil,
                     int Lx, int Ly, int dtype, void* stream);
/* Wilson-clover (Sheikholeslami-Wohlert) level 0: the self block becomes (2+m) 1 + f(s) s3 with the real field
 * f = F[s] of mg2d_clover_field (double for MG2D_C128, float for MG2D_C64; F_lo / F_hi = its rows -1 / Ly).
 *   mg2d_wilson_sw_apply       mg2d_wilson_apply with the clover self term (APPLY, RESID, fused dots)
 *   mg2d_wilson_sw_relax_rb    mg2d_wilson_relax_rb with D0 = diag(2+m+f, 2+m-f)
 *   mg2d_wilson_sw_relax_rb2   mg2d_wilson_relax_rb2 with D0 = diag(2+m+f, 2+m-f); the red stage recomputes rows -1
 *                              and Ly, hence F_lo / F_hi
 *   mg2d_clover_add            stored operator: D[s][0] += diag(F[s], -F[s]) on nsites sites (stencil 0 blocks) */
int mg2d_wilson_sw_apply(mg2d_ctx*, void* out, const void* in, const void* in_lo, const void* in_hi,
                         const void* U, const void* U_lo, const void* F, const void* b, double mass, int Lx, int Ly,
                         int mode, int dtype, double* dots, void* stream);
int mg2d_wilson_sw_relax_rb(mg2d_ctx*, void* phi, const void* phi_lo, const void* phi_hi, const void* U,
                            const void* U_lo, const void* F, const void* r, double mass, int Lx, int Ly, int colour,
                            int yoff, int dtype, void* stream);
int mg2d_wilson_sw_relax_rb2(mg2d_ctx*, void* out, const void* in, const void* in_lo2, const void* in_hi2,
                             const void* U, const void* U_lo2, const void* U_hi, const void* F, const void* F_lo,
                             const void* F_hi, const void* r, const void* r_lo, const void* r_hi, double mass, int Lx,
                             int Ly, int yoff, int dtype, const struct mg2d_halo_link* link, void* stream);
int mg2d_clover_add(mg2d_ctx*, void* D, const void* F, long long nsites, int dtype, void* stream);
/* Twisted mass: + i mu gamma5 = i mu s3 on the level-0 self block, which becomes diag(2+m+f+i mu, 2+m-f-i mu) with f the
 * clover field (F == NULL: no clover, f = 0).  D_tm^dag D_tm = D^dag D + mu^2, and g5 D_tm(mu) g5 = D_tm(-mu)^dag.
 *   mg2d_wilson_tm_apply       mg2d_wilson_sw_apply with the twisted self term (APPLY, RESID, fused dots)
 *   mg2d_wilson_tm_relax_rb    mg2d_wilson_sw_relax_rb with D0 = diag(2+m+f+i mu, 2+m-f-i mu)
 *   mg2d_wilson_tm_relax_rb2   mg2d_wilson_sw_relax_rb2 with the same D0 (F, F_lo, F_hi all NULL or F_lo / F_hi given)
 *   mg2d_twist_add             stored operator: D[s][0] += diag(i mu, -i mu) on nsites sites (stencil 0 blocks)
 * mu must be finite.  The coarse levels need no entry point: on a chirality-split projector the Galerkin product carries
 * the twist as i mu Gamma5_c on the coarse self blocks. */
int mg2d_wilson_tm_apply(mg2d_ctx*, void* out, const void* in, const void* in_lo, const void* in_hi,
                         const void* U, const void* U_lo, const void* F, const void* b, double mass, double mu, int Lx,
                         int Ly, int mode, int dtype, double* dots, void* stream);
int mg2d_wilson_tm_relax_rb(mg2d_ctx*, void* phi, const void* phi_lo, const void* phi_hi, const void* U,
                            const void* U_lo, const void* F, const void* r, double mass, double mu, int Lx, int Ly,
                            int colour, int yoff, int dtype, void* stream);
int mg2d_wilson_tm_relax_rb2(mg2d_ctx*, void* out, const void* in, const void* in_lo2, const void* in_hi2,
                             const void* U, const void* U_lo2, const void* U_hi, const void* F, const void* F_lo,
                             const void* F_hi, const void* r, const void* r_lo, const void* r_hi, double mass, double mu,
                             int Lx, int Ly, int yoff, int dtype, const struct mg2d_halo_link* link, void* stream);
int mg2d_twist_add(mg2d_ctx*, void* D, double mu, long long nsites, int dtype, void* stream);
/* Twist of a built hierarchy changed in place (MG.set_twist): Im D[s][0](i,i) = base[s][i] + delta Gamma5_c(i,i) for a stored
 * operator with n in {2,4,8,16,32} (column-major blocks), Gamma5_c = diag(+1 x n/2, -1 x n/2) (n = 2: sigma3 of level 0).
 * base [nsites][n] fp64 holds the imaginary diagonal at the build twist mu_b and delta = mu - mu_b (finite); the sum is formed
 * in fp64 and rounded once to dtype, so delta = 0 restores the operator bit for bit.  Real parts are not touched. */
int mg2d_twist_set(mg2d_ctx*, void* D, const double* base, double delta, int n, long long nsites, int dtype, void* stream);

/* ---- generic 5-point block stencil (all coarse levels; level 0 in reference-compat mode) -------------- */
/* Level::f_apply_D / f_residue, n in {1,2,4,8,16,32}; nvec vectors `vstride` elements apart. */
int mg2d_stencil_apply(mg2d_ctx*, void* out, const void* in, const void* in_lo, const void* in_hi,
                       const void* D, const void* b, int n, int Lx, int Ly, int mode, int dtype,
                       int nvec, long long vstride, long long hstride, double* dots, void* stream);
/* D0inv[s] = inverse(D[s][0]) (column-major like D): the `D(x+y*L,0).inverse()` of S6/level.h:116, hoisted. */
int mg2d_block_inverse(mg2d_ctx*, void* D0inv, const void* D, int n, long long nsites, int dtype, void* stream);
/* Level::f_relax with gs_flag=0 (Jacobi), one sweep: out = -D0inv (sum_{k>=1} D_k in(s+d_k) - r). */
int mg2d_relax_jacobi(mg2d_ctx*, void* out, const void* in, const void* in_lo, const void* in_hi,
                      const void* D, const void* D0inv, const void* r, int n, int Lx, int Ly, int dtype,
                      int nvec, long long vstride, long long hstride, void* stream);
/* Level::f_relax with gs_flag=1: `num_iter` lexicographic Gauss-Seidel sweeps (x outer, y inner, S6/level.h:
 * 113-123) executed as anti-diagonal wavefronts, which reproduces the sequential order exactly.  Whole
 * periodic lattice on one GPU (Ly == Lx).  r == NULL means r = 0 (near-null relaxation, S6/level.h:196-198). */
int mg2d_relax_gs(mg2d_ctx*, void* phi, const void* D, const void* D0inv, const void* r, int n, int L,
                  int num_iter, int dtype, int nvec, long long vstride, void* stream);
/* One lexicographic Gauss-Seidel sweep (same order: x outer, y inner over the GLOBAL lattice) on the strip of rows [y0, y0+Ly) of an
 * Lx x Lglobal lattice: global anti-diagonal fronts, every rank updates its part of a front once the value it needs from the
 * previous rank (first local row; new) has arrived.  phi_lo / phi_hi: this rank's halo buffers holding the neighbours' OLD
 * boundary rows (mg2d_halo_exchange before every sweep); push_next_lo: the next rank's lo buffer (NULL on the last rank);
 * push_last_hi: the last rank's hi buffer (rank 0 only: its row 0 is the periodic upper neighbour of the last row);
 * slot_*: 64-byte progress slots of this rank, the next and the last one (zeroed, peer-mapped).  Parity mode: 2L-1 dependent
 * fronts and one flag hop per front. */
int mg2d_relax_gs_strip(mg2d_ctx*, void* phi, const void* phi_lo, const void* phi_hi, const void* D, const void* D0inv,
                        const void* r, int n, int Lx, int Ly, int y0, int Lglobal, int dtype, void* slot_mine, void* slot_next,
                        void* slot_last, void* push_next_lo, void* push_last_hi, int first_rank, int last_rank, void* stream);

/* Level::f_relax update rule in red-black (two-colour) ordering, one half sweep IN PLACE: the sites with
 * (x + y + yoff) % 2 == colour are updated from the other colour (parallel stand-in for the sequential
 * lexicographic order of S6/level.h:113-123; mirrored by oracle Level.relax_rb).  Lx even. */
int mg2d_relax_rb(mg2d_ctx*, void* phi, const void* phi_lo, const void* phi_hi, const void* D, const void* D0inv,
                  const void* r, int n, int Lx, int Ly, int colour, int yoff, int dtype, int nvec,
                  long long vstride, long long hstride, void* stream);
/* the same for the matrix-free level-0 Wilson operator (D0 = (2+m) 1) */
int mg2d_wilson_relax_rb(mg2d_ctx*, void* phi, const void* phi_lo, const void* phi_hi, const void* U,
                         const void* U_lo, const void* r, double mass, int Lx, int Ly, int colour, int yoff,
                         int dtype, void* stream);

/* One FULL red-black sweep (colour 0, then colour 1) of the matrix-free Wilson operator in a single pass, OUT OF PLACE
 * (out != in): every phi / r / link element is read once and every result written once (128 B/site in complex128
 * instead of ~224 B moved by two half-sweep launches).  Needs the neighbour data two rows deep: in_lo2 = rows
 * (-2, -1), in_hi2 = rows (Ly, Ly+1) of `in`; U_lo2 = link rows (-2, -1), U_hi = link row Ly; r_lo / r_hi = rows
 * -1 / Ly of r (r == NULL: r = 0).  On one GPU these are the periodic wrap rows of the arrays themselves. */
int mg2d_wilson_relax_rb2(mg2d_ctx*, void* out, const void* in, const void* in_lo2, const void* in_hi2,
                          const void* U, const void* U_lo2, const void* U_hi, const void* r, const void* r_lo,
                          const void* r_hi, double mass, int Lx, int Ly, int yoff, int dtype,
                          const struct mg2d_halo_link* link, void* stream);

/* The same half sweep on pre-multiplied hopping blocks M[s][k-1][j][i] = -D0inv(s) D_k(s), k = 1..4 (built once by
 * mg2d_premultiply): phi(s) <- sum_k M_k(s) phi(s+d_k) + c(s), c = D0inv r.  4 blocks per updated site instead of 5.
 * cmode 0: r = 0; 1: first sweep of a relax call (c computed from D0inv, r and stored in cbuf[nvec][S][n]);
 * 2: c read from cbuf.  link (may be NULL): fused neighbour push / wait on strips, see mg2d_halo_link. */
int mg2d_premultiply(mg2d_ctx*, void* M, const void* D, const void* D0inv, int n, long long nsites, int dtype, void* stream);
int mg2d_relax_rb_pm(mg2d_ctx*, void* phi, const void* phi_lo, const void* phi_hi, const void* M, const void* D0inv,
                     const void* r, void* cbuf, int cmode, int n, int Lx, int Ly, int colour, int yoff, int dtype,
                     int nvec, long long vstride, long long hstride, const struct mg2d_halo_link* link, void* stream);

/* `nsweeps` full red-black sweeps (both colours) of the pre-multiplied update in ONE cooperative launch, the half sweeps
 * separated by grid-wide barriers: for the small levels of the hierarchy (whole periodic L x L lattice on this GPU, one
 * vector) where a half sweep is a latency-bound ~10 us launch.  r == NULL: r = 0. */
int mg2d_relax_rb_pm_sweeps(mg2d_ctx*, void* phi, const void* M, const void* D0inv, const void* r, void* cbuf,
                            int n, int L, int nsweeps, int dtype, void* stream);

/* Low-rank hopping blocks of the FIRST coarse level (no reference counterpart in storage; same update as f_relax,
 * S6/level.h:100-128).  Every fine hopping term has rank one (Wilson spin projector (1 -+ sigma_mu)/2, S6/level.h:155-172;
 * a scalar for the Laplacian) and only `block` fine links cross an aggregate face, so the Galerkin hopping block
 * (S6/modules_main.h:148-155) is D_k(X) = sum_{b<block} A_q B_q^dagger, q = (k-1)*block + b: rank <= block.
 *   mg2d_hop_factors   A, B [Sc][4*block][nc] from the fine operator Df (n_dof 1 or 2) and the projector P (+ halo rows);
 *                      *status |= 4 when a fine hopping block is not rank one to 1e-13 (the caller then keeps dense blocks)
 *   mg2d_lowrank_pack  F[s][2][n*rank/8][32]: conj(B) and -D0inv A in the lane order of the sweep kernel
 *   mg2d_relax_rb_lr   the red-black half sweep of mg2d_relax_rb_pm (same cmode / link / batch meaning) streaming
 *                      2*4*rank*n numbers per site instead of 4*n*n.  (n, rank) in {(16,4), (8,2)}: 8 null vectors over
 *                      4x4 aggregates, 4 over 2x2 (wilson); 16 over 4x4 (laplace). */
int mg2d_lowrank_supported(int n, int rank);
int mg2d_hop_factors(mg2d_ctx*, void* A, void* B, const void* Df, const void* P, const void* P_lo, const void* P_hi,
                     int nf, int nc, int Lxf, int Lyf, int block, int dtype, int* status, void* stream);
int mg2d_lowrank_pack(mg2d_ctx*, void* F, const void* A, const void* B, const void* D0inv, int n, int rank,
                      long long nsites, int dtype, void* stream);
/* mg2d_lowrank_pack_a: only the -D0inv A half of F (after D0inv changed; the conj(B) half does not depend on the self
 * blocks), bit-identical to what mg2d_lowrank_pack writes there. */
int mg2d_lowrank_pack_a(mg2d_ctx*, void* F, const void* A, const void* D0inv, int n, int rank, long long nsites, int dtype,
                        void* stream);
int mg2d_relax_rb_lr(mg2d_ctx*, void* phi, const void* phi_lo, const void* phi_hi, const void* F, const void* D0inv,
                     const void* r, void* cbuf, int cmode, int n, int rank, int Lx, int Ly, int colour, int yoff,
                     int dtype, int nvec, long long vstride, long long hstride, const struct mg2d_halo_link* link, void* stream);

/* The same half sweep for the complex64 preconditioner hierarchy with the operator stored in half precision:
 * Dh / D0invh are __half2 (re,im) arrays in the [s][k][j][i] / [s][j][i] order (built by mg2d_to_half from the complex64
 * operator); fields and arithmetic stay fp32.  n in {8,16,32}.  Mixed-precision option, no reference counterpart. */
int mg2d_relax_rb_half(mg2d_ctx*, void* phi, const void* phi_lo, const void* phi_hi, const void* Dh, const void* D0invh,
                       const void* r, int n, int Lx, int Ly, int colour, int yoff, void* stream);
int mg2d_to_half(mg2d_ctx*, void* dst_half2, const void* src_c64, long long nelem, void* stream);

/* ---- BLAS-1 style fused updates ------------------------------------------------------------------------ */
/* MR smoother update: alpha = omega * <t,res>/<t,t> read from `dots` (as written by a stencil call with
 * in=res, out=t); phi += alpha res; res -= alpha t. */
int mg2d_mr_update(mg2d_ctx*, void* phi, void* res, const void* t, const double* dots, double omega,
                   long long nelem, int dtype, int nvec, long long vstride, void* stream);
/* y += a x, a = (a_re, a_im), or a read from device `a_dev` (2 doubles) when a_dev != NULL. */
int mg2d_axpy(mg2d_ctx*, void* y, const void* x, double a_re, double a_im, const double* a_dev,
              long long nelem, int dtype, void* stream);
/* y += sign*(num/den) x and (if y2) y2 += sign*(num/den) x2; num = 2 doubles (complex), den = 1 double, both on
 * the device: the Gram-Schmidt and step updates of the outer GCR without a host round trip. */
int mg2d_axpy_ratio2(mg2d_ctx*, void* y, const void* x, void* y2, const void* x2, const double* num,
                     const double* den, double sign, long long nelem, int dtype, void* stream);
/* Outer flexible GCR (no reference counterpart; SURVEY 8f N3), classical Gram-Schmidt against nj <= 8 stored
 * directions W_j / Z_j (`stride` elements apart), one pass each:
 *   mg2d_gcr_dots : out[2j..2j+1] = <W_j, w>
 *   mg2d_gcr_ortho: w -= sum_j (dots_j / wn2_j) W_j ; z -= sum_j (...) Z_j ; out = { |w|^2, Re<w,r>, Im<w,r> } of the new w
 *   mg2d_gcr_step : a = <w,r>/|w|^2 (wr = the three doubles above); x += a z ; r -= a w ; out[0] = |r|^2 ;
 *                   *wn2_slot = |w|^2 (kept for the projections of later iterations) */
int mg2d_gcr_dots(mg2d_ctx*, const void* W, long long stride, int nj, const void* w, long long nelem, int dtype,
                  double* out, void* stream);
int mg2d_gcr_ortho(mg2d_ctx*, void* w, void* z, const void* r, const void* W, const void* Z, long long stride, int nj,
                   const double* dots, const double* wn2, long long nelem, int dtype, double* out, void* stream);
int mg2d_gcr_step(mg2d_ctx*, void* x, void* r, const void* z, const void* w, const double* wr, double* wn2_slot,
                  long long nelem, int dtype, double* out, void* stream);   /* wn2_slot (may be NULL) receives |w|^2 */
/* Lazy solution update of the same iteration (identical iterates up to rounding): mg2d_gcr_ortho with z = Z = NULL leaves
 * the preconditioned residuals z_i raw; mg2d_gcr_step_lazy does r -= a w, out[0] = |r|^2, *wn2_slot = |w|^2 and advances
 * the 8 x 8 coefficient recursion in `coef` (144 doubles, device) that expresses the orthogonalised directions in the
 * raw z_i (nj = index of this iteration within the restart cycle; nj = 0 resets); mg2d_gcr_xupdate adds the accumulated
 * combination x += sum_{i<nj} g_i Z_i once per restart cycle (or at convergence). */
int mg2d_gcr_step_lazy(mg2d_ctx*, void* r, const void* w, const double* wr, double* wn2_slot, const double* dots,
                       const double* wn2, int nj, double* coef, long long nelem, int dtype, double* out, void* stream);
int mg2d_gcr_xupdate(mg2d_ctx*, void* x, const void* Z, long long stride, int nj, const double* coef, long long nelem,
                     int dtype, void* stream);
int mg2d_zero(mg2d_ctx*, void* x, long long nelem, int dtype, void* stream);
int mg2d_copy(mg2d_ctx*, void* dst, const void* src, long long nelem, int dtype, void* stream);
/* dst = src converted between MG2D_C128 and MG2D_C64 */
int mg2d_convert(mg2d_ctx*, void* dst, int dst_dtype, const void* src, int src_dtype, long long nelem, void* stream);
/* out[0] = sum |x|^2 (f_g_norm, S6/modules_indiv.h:70-92) */
int mg2d_norm2(mg2d_ctx*, const void* x, long long nelem, int dtype, double* out, void* stream);
/* out[2*(i*ny+j) .. +1] = <x_i, y_j> = sum conj(x_i) y_j  (f_min_res Gram matrix, S6/modules_main.h:324-366) */
int mg2d_cdot_batch(mg2d_ctx*, const void* x, long long xstride, int nx, const void* y, long long ystride,
                    int ny, long long nelem, int dtype, double* out, void* stream);
/* x *= 1/sqrt(norm2[0]) with norm2 on the device (rescale branch of f_g_norm, S6/modules_indiv.h:88-89) */
int mg2d_scale_inv_norm(mg2d_ctx*, void* x, const double* norm2, long long nelem, int dtype, void* stream);

/* ---- block aggregation: restriction / prolongation ------------------------------------------------------ */
/* Near_null::f_restriction (S6/near_null.h:217-240): vc(X) = sum_{s in agg(X,quad)} P(s) vf(s).
 * Lxf x Lyf fine sites (local strip), block x block aggregates, quad 1..4 (f_get_base_site,
 * S6/modules_indiv.h:6-14; quad != 1 requires the whole periodic lattice on one GPU). */
int mg2d_restrict(mg2d_ctx*, void* vc, const void* vf, const void* P, int nf, int nc, int Lxf, int Lyf,
                  int block, int quad, int dtype, void* stream);
/* Near_null::f_prolongation (S6/near_null.h:242-264): vf(s) += P(s)^dagger vc(X(s)); zero_vc != 0 also
 * clears vc afterwards (f_prolongate_phi, S6/modules_main.h:243-252). */
int mg2d_prolong_add(mg2d_ctx*, void* vf, void* vc, const void* P, int nf, int nc, int Lxf, int Lyf,
                     int block, int quad, int zero_vc, int dtype, void* stream);

/* The same two operators on a chirality-compacted projector Pc[s][ic][jf'] (nc x nf/2): Level::f_near_null
 * (S6/level.h:236-245) leaves row ic < nc/2 non-zero only in its first nf/2 columns and row ic >= nc/2 only in its
 * last nf/2; Pc keeps that half.  Half the bytes, identical results.  accumulate = 0 writes vf = P^dagger vc
 * (valid because every fine site belongs to exactly one aggregate) instead of adding. */
int mg2d_restrict_chiral(mg2d_ctx*, void* vc, const void* vf, const void* Pc, int nf, int nc, int Lxf, int Lyf,
                         int block, int quad, int dtype, void* stream);
int mg2d_prolong_chiral(mg2d_ctx*, void* vf, void* vc, const void* Pc, int nf, int nc, int Lxf, int Lyf,
                        int block, int quad, int zero_vc, int accumulate, int dtype, void* stream);

/* ---- setup ---------------------------------------------------------------------------------------------- */
/* Level::f_near_null tail (S6/level.h:217-246): P rows from the relaxed vectors V[v][s][nf]:
 * laplace: P[s][v][:] = conj(V_v(s)); wilson: chirality split, row v gets the upper nf/2 components,
 * row nc/2+v the lower ones, the rest 0. */
int mg2d_pack_null(mg2d_ctx*, void* P, const void* V, int nvec, long long vstride, int nf, int nc,
                   long long nsites, int wilson, int dtype, void* stream);
/* Near_null::f_norm_nn (S6/near_null.h:24-48, f_block_norm S6/modules_indiv.h:94-135): every row of P
 * normalised per aggregate.  `status` (device int, may be NULL) gets bit 1 when a block norm is NaN or below 1e-40
 * (the reference exits there, S6/modules_indiv.h:119-126). */
int mg2d_norm_nn(mg2d_ctx*, void* P, int nf, int nc, int Lxf, int Lyf, int block, int quad, int dtype,
                 int* status, void* stream);
/* Near_null::f_ortho (S6/near_null.h:97-173): per-aggregate modified Gram-Schmidt, t -= (dot/|u|) u, then
 * block-normalise.  `status` (device int, may be NULL) is set non-zero on NaN / tiny norms (:149-159). */
int mg2d_ortho(mg2d_ctx*, void* P, int nf, int nc, int Lxf, int Lyf, int block, int quad, int dtype,
               int* status, void* stream);
/* Near_null::f_check_ortho (S6/near_null.h:175-214): out[0] = max over aggregates and d2<d1 of |<row d1,row d2>| */
int mg2d_check_ortho(mg2d_ctx*, const void* P, int nf, int nc, int Lxf, int Lyf, int block, int quad, int dtype,
                     double* out, void* stream);
/* f_compute_coarse_matrix (S6/modules_main.h:81-185): Dc = P Df P^dagger split into the self block and the
 * four face blocks.  P_lo / P_hi: projector rows below / above the local strip (quad 1 multi-GPU), else the
 * periodic wrap rows. */
int mg2d_coarse_matrix(mg2d_ctx*, void* Dc, const void* Df, const void* P, const void* P_lo, const void* P_hi,
                       int nf, int nc, int Lxf, int Lyf, int block, int quad, int dtype, void* stream);

/* ---- non-telescoping min-res (f_min_res, S6/modules_main.h:283-373) --------------------------------------- */
/* Solve the ncopies x ncopies system A a = src with column-pivoted Householder QR (the
 * `A.colPivHouseholderQr().solve(src)` of :371) on the device.  gram = output of mg2d_cdot_batch
 * (A row-major, complex as 2 doubles), src likewise; a[2*q..] receives the weights. */
int mg2d_minres_solve(mg2d_ctx*, const double* gram, const double* src, int ncopies, double* a, void* stream);
/* f_scale_phi (S6/modules_main.h:375-384): phi += sum_q a_q e_q ; e_q = 0.  e_q are `estride` apart. */
int mg2d_scale_phi(mg2d_ctx*, void* phi, void* e, long long estride, const double* a, int ncopies,
                   long long nelem, int dtype, void* stream);

/* ---- multi-GPU strips: peer-to-peer halo exchange over NVLink (no reference counterpart; SURVEY 8e) ------- */
/* Neighbour push fused into a smoother kernel.  The kernel processes its boundary rows LAST; before it reads the halo
 * rows it waits (wait != 0) until both neighbours' flags in `slot_mine` have reached the local epoch, it stores the
 * boundary rows it produces straight into the neighbours' halo buffers (peer-mapped pointers, NULL = no push) and its
 * last CTA releases the neighbours' flags with epoch + 1: no separate exchange launch, the interior overlaps the
 * transfer.  Slots are the 64-byte records mg2d_halo_exchange uses. */
typedef struct mg2d_halo_link {
    void* slot_mine; void* slot_prev; void* slot_next;
    void* push_next_lo; void* push_prev_hi;
    int wait;
} mg2d_halo_link;
/* Reductions summed over all ranks INSIDE the producing kernel: every rank owns a mailbox (mg2d_comm_mailbox_bytes()
 * bytes of zeroed, peer-mapped memory); mg2d_comm_create builds the descriptor from the `world` mailbox pointers as seen
 * from this rank and attaches it; while mg2d_comm_reduce(ctx, 1) is in force the `dots` / norm outputs of
 * mg2d_wilson_apply, mg2d_stencil_apply (nvec = 1), mg2d_norm2 and mg2d_gcr_* are global sums, bit-identical on every
 * rank (contributions added in rank order).  mg2d_allreduce sums n <= 64 doubles in place (batched reductions). */
int mg2d_comm_mailbox_bytes(void);
int mg2d_comm_create(mg2d_ctx*, int world, int rank, void* const* mailbox_ptrs, void** desc_out);
int mg2d_comm_attach(mg2d_ctx*, void* desc);                   /* share one descriptor between handles of one rank */
int mg2d_comm_reduce(mg2d_ctx*, int on);
int mg2d_comm_error(mg2d_ctx*, void* desc, long long* out);    /* synchronous: non-zero after a peer time-out */
int mg2d_allreduce(mg2d_ctx*, double* buf, int n, void* stream);
int mg2d_halo_errors(mg2d_ctx*, const void* slots, int nslots, long long* out);   /* synchronous */
/* A slab of device memory other ranks can map (CUDA IPC): cudaMalloc + zero + 64-byte handle. */
int mg2d_ipc_alloc(mg2d_ctx*, long long bytes, void** ptr, void* handle64);
int mg2d_ipc_open(mg2d_ctx*, const void* handle64, void** ptr);
/* One kernel = one halo exchange of a field's boundary rows with both strip neighbours: acknowledges the previous
 * rows, waits for the neighbours' acknowledgements, stores `last` into next's lo buffer and `first` into prev's hi
 * buffer through peer mappings, publishes the epoch (st.release.sys) and waits for the neighbours' rows.  Slots are
 * 64-byte records {flag_lo, flag_hi, ack_prev, ack_next, epoch, error} inside the IPC slab. */
int mg2d_halo_exchange(mg2d_ctx*, const void* first, const void* last, long long src_stride_bytes, long long row_bytes,
                       int nvec, void* next_lo, void* prev_hi, void* slot_mine, void* slot_prev, void* slot_next,
                       void* stream);

/* ---- inputs generated on the device (SURVEY 8f N1; the reference draws from std::mt19937 / reads link files) ------ */
/* out[e] = (lo + (hi-lo) u(seed, stream_id, offset+e), 0): counter-based uniform numbers (splitmix64 of the key), so a
 * strip starting at global element `offset` holds what the whole field holds there (f_init_near_null_vector,
 * S6/modules_indiv.h:52-68, for lattices beyond the sequential mt19937 stream; mirrored by oracle counter_uniform). */
int mg2d_fill_uniform(mg2d_ctx*, void* out, long long nelem, long long offset, unsigned long long seed,
                      unsigned long long stream_id, double lo, double hi, int dtype, void* stream);
/* One checkerboard half-update (sites with (x+y)%2 == parity, direction mu) of compact-U(1) Wilson-action Metropolis on
 * the phases theta[s][2] (doubles); proposal theta + (2u1-1) delta, accept if u2 < exp(-dS); u1, u2 = counter numbers of
 * streams 2*tag, 2*tag+1 at index s.  Produces the configurations S6/gauge.h:88-110 reads from files it does not ship. */
int mg2d_gauge_metropolis(mg2d_ctx*, double* theta, int L, double beta, double delta, int mu, int parity,
                          unsigned long long seed, unsigned long long tag, void* stream);
/* Gauge::f_plaquette (S6/gauge.h:50-63): out[0..1] = sum_s U_x(s) U_y(s+x) conj(U_x(s+y)) conj(U_y(s)) (re, im). */
int mg2d_plaquette(mg2d_ctx*, const void* U, int L, int dtype, double* out, void* stream);
/* clover field of rows [0, Ly) of an Lx-wide strip: F[s] = (csw/8) sum over the four plaquettes P with a corner at s of
 * Im U_P, U_P = U_x(b) U_y(b+x) conj(U_x(b+y)) conj(U_y(b)) (the orientation of mg2d_plaquette).  U_lo / U_hi = link rows
 * -1 / Ly (on one GPU the periodic wrap rows of U).  A strip gets its rows of the whole-lattice field bit for bit. */
int mg2d_clover_field(mg2d_ctx*, void* F, const void* U, const void* U_lo, const void* U_hi, double csw, int Lx, int Ly,
                      int dtype, void* stream);
/* U[e] = polar(1, theta[e]) (S6/gauge.h:106) */
int mg2d_phases_to_links(mg2d_ctx*, void* U, const double* theta, long long nelem, int dtype, void* stream);
/* out[e] = N(0, variance) real deviates: Box-Muller (cosine branch) on the counter numbers at indices 2(offset+e) and
 * 2(offset+e)+1 of (seed, stream_id), so a draw is reproducible from its key alone (HMC momenta and pseudofermion sources). */
int mg2d_fill_gaussian(mg2d_ctx*, double* out, long long nelem, long long offset, unsigned long long seed,
                       unsigned long long stream_id, double variance, void* stream);

/* ---- two-flavour Wilson HMC on the links U[s][mu] = e^{i theta[s][mu]} (complex128, whole lattice, L x L) ---------- */
/* P[s][mu] -= eps (F^g_mu(s) + F^f_mu(s)) for both directions: F^g = dS_g/dtheta of S_g = beta sum_P (1 - cos theta_P);
 * F^f = dS_f/dtheta of S_f = phi^dag (D^dag D)^-1 phi from X = (D^dag D)^-1 phi and Y = D X (csrc/hmc.cu).  X = Y = NULL:
 * gauge force only. */
int mg2d_hmc_momentum(mg2d_ctx*, double* P, const void* U, const void* X, const void* Y, double beta, double eps, int L,
                      void* stream);
/* theta[e] += eps P[e]; U[e] = polar(1, theta[e]) (complex128) and, when U32 is not NULL, its complex64 copy. */
int mg2d_hmc_links(mg2d_ctx*, double* theta, const double* P, double eps, void* U, void* U32, long long nelem, void* stream);
/* out = gamma5 in = sigma3 in on nsites two-component complex128 sites (out may equal in). */
int mg2d_gamma5(mg2d_ctx*, void* out, const void* in, long long nsites, void* stream);

/* ---- multi-shift CG for (D^dag D + sigma_k) x_k = phi, all shifts at once (one-flavour RHMC; csrc/rhmc.cu) ------------- */
/* Jegerlehner's recurrences on complex128 two-component fields of nsites sites.  The base system is the smallest shift
 * sigma_0; the host applies the operator with mg2d_wilson_apply (t = D p_0, dots[MG2D_DOT_OUT2] = |t|^2), mg2d_gamma5 and
 * mg2d_wilson_apply again (w = D gamma5 t, so (D^dag D) p_0 = gamma5 w).  `sc` holds the fp64 scalars on the device:
 * the slots below, then from MG2D_MSC_SHIFTS on, for N = nshift shifts sorted ascending, s_k = sigma_k - sigma_0 [N],
 * zeta_k [N], zeta_k of the previous iteration [N], a_k [N], b_k [N], the accumulate-mode weights w_k [N], and the Lanczos
 * history (alpha_i, beta_i) of iteration i at 2i, 2i+1.  Start: r = p_k = phi, x_k = 0, RR = |phi|^2, PP = |phi|^2,
 * ALPHA_PREV = 1, BETA_PREV = 0, zeta = zeta_prev = 1, NACT_NEXT = N, ITER = 0, THRESH = (tol |phi|)^2.
 *   mg2d_msc_pass_a  r -= alpha (gamma5 w + sigma_0 p_0), alpha = RR / (dots[0] + sigma_0 PP); |r|^2 reduced in the kernel,
 *                    whose last CTA runs the scalar recurrences and sets NACT (the shifts pass B updates) and NACT_NEXT
 *                    (1 + the last shift whose residual |zeta_k| |r| is still above THRESH^(1/2); 0 = all converged)
 *   mg2d_msc_pass_b  k < NACT: x_k += a_k p_k, p_k = zeta_k r + b_k p_k, X and P laid out [N][nsites][2]; with X == NULL
 *                    and y != NULL (accumulate mode) y += sum_k w_k a_k p_k instead; PP = |p_0|^2 when sigma_0 != 0 */
enum { MG2D_MSC_RR = 0, MG2D_MSC_ALPHA_PREV = 1, MG2D_MSC_BETA_PREV = 2, MG2D_MSC_PP = 3, MG2D_MSC_NACT = 4,
       MG2D_MSC_NACT_NEXT = 5, MG2D_MSC_ITER = 6, MG2D_MSC_THRESH = 7, MG2D_MSC_SHIFTS = 8, MG2D_MSC_MAX_SHIFTS = 64 };
int mg2d_msc_pass_a(mg2d_ctx*, void* r, const void* w, const void* p0, const double* dots, double* sc, double sigma0,
                    int nshift, long long nsites, void* stream);
int mg2d_msc_pass_b(mg2d_ctx*, void* X, void* P, void* y, const void* r, double* sc, double sigma0, int nshift,
                    long long nsites, void* stream);

/* ---- gauge-ensemble measurements (complex128, whole lattice, L x L; csrc/measure.cu) ------------------------------ */
/* out[y][a][b][re, im] = G_ab(y) = sum_x tr[s_a S(x,y) s_b s3 S(x,y)^dag s3] for every row y (time), a, b = 0..3, with
 * S_{al,be}(s) = psi_be(s)_al from the two point-source propagator columns psi_be = D^-1 e_{s0,be} ([L*L][2] each, 32-byte
 * aligned), s0 = 1 and s1, s2, s3 = gamma_x, gamma_y, gamma5.  -G_ab is the connected correlator of the bilinears s_a, s_b. */
int mg2d_meson_contract(mg2d_ctx*, const void* psi0, const void* psi1, int L, double* out, void* stream);
/* out[0] = sum_P arg U_P, arg in (-pi, pi], U_P oriented as in mg2d_plaquette; the topological charge is out[0] / 2 pi. */
int mg2d_topo_charge(mg2d_ctx*, const void* U, int L, double* out, void* stream);
/* out[2 ((T-1) r_max + R-1) + (0, 1)] = sum_s of the product of the links around the anticlockwise R x T rectangle with base
 * s (R links along x, T along y; W(1,1) is the plaquette sum), 1 <= R <= r_max, 1 <= T <= t_max.  Needs
 * 1 <= r_max, t_max <= 32 and r_max, t_max < L (MG2D_EINVAL otherwise). */
int mg2d_wilson_loops(mg2d_ctx*, const void* U, int L, int r_max, int t_max, double* out, void* stream);

/* ---- real scalar Laplace geometric MG, BASELINE config 1 (S2) -------------------------------------------- */
/* relax (S2:46-72): num_iter lexicographic GS sweeps phi = scale (sum nbrs - b a^2), wavefront order. */
int mg2d_s2_relax(mg2d_ctx*, double* phi, const double* b, int L, double scale, double a, int num_iter,
                  int gs_flag, void* stream);
/* f_projection (S2:74-110): res_c = 1/4 sum_{2x2, quadrant} (b - A phi). */
int mg2d_s2_project(mg2d_ctx*, double* res_c, const double* b, const double* phi, int L, double scale, double a,
                    int quad, void* stream);
/* f_interpolate (S2:112-143): phi_f(4 sites) += phi_c ; phi_c = 0. */
int mg2d_s2_interpolate(mg2d_ctx*, double* phi_f, double* phi_c, int Lc, int quad, void* stream);
/* f_get_residue_mag (S2:23-44): out[0] = sum |b - A phi|. */
int mg2d_s2_residue_mag(mg2d_ctx*, const double* phi, const double* b, int L, double scale, double a,
                        double* out, void* stream);
/* x *= s */
int mg2d_s2_scale(mg2d_ctx*, double* x, double s, long long n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MG2D_H */
