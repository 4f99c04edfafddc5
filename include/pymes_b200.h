/*
 * pymes_b200.h -- C ABI of the B200-native coupled-cluster contraction engine.
 *
 * This is the drop-in boundary for the amplitude-equation hot path of
 * nickirk/pymes (reference commit 734974a).  The reference has no FFI: its
 * backend seam is the per-module alias `einsum = partial(np.einsum, optimize=True)`
 * (pymes/solver/ccsd.py:11, eom_ccsd.py:9, feast_eom_ccsd.py:16, mp2.py:5,
 * model/ueg.py:10) plus bare `np.einsum` in pymes/solver/ccd.py and
 * pymes/mixer/diis.py.  Every entry point below replaces a family of those
 * einsum / elementwise numpy call sites; the reference lines are cited per
 * function.  INTEGRATION.md shows the ctypes stub a pymes maintainer would add.
 *
 * Conventions
 *   - all data pointers are DEVICE pointers to float64 unless stated otherwise;
 *   - strides are in ELEMENTS (not bytes);
 *   - every call is asynchronous on the given CUDA stream (pass 0 for the
 *     legacy default stream) and returns 0 on success, a cudaError_t value
 *     (> 0) for CUDA failures, or a negative PMB_E_* code for bad arguments;
 *   - the library never allocates persistent device memory: scratch space is
 *     handed in by the caller (`ws`, `ws_bytes`); query sizes with the
 *     *_workspace functions.
 */
#ifndef PYMES_B200_H
#define PYMES_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PMB_MAX_DIMS 4   /* indices per index group (M, N or K)            */
#define PMB_MAX_TERMS 8  /* A.B products accumulated into one output       */

#define PMB_E_BADARG (-1)
#define PMB_E_WORKSPACE (-2)
#define PMB_E_UNSUPPORTED (-3)

typedef void *pmb_stream_t; /* cudaStream_t */

/* ------------------------------------------------------------------------ */
/* library / device information                                             */
/* ------------------------------------------------------------------------ */
int pmb_version(void);
/* sm count, compute capability (major*10+minor), total global memory bytes  */
int pmb_device_info(int *sm_count, int *cc, size_t *global_mem);
/* number of kernels this library has launched since load (or last reset)   */
long long pmb_launch_count(void);
void pmb_launch_count_reset(void);
const char *pmb_error_string(int code);

/* ------------------------------------------------------------------------ */
/* generic binary tensor contraction on FP64 tensor cores (DMMA)             */
/*                                                                          */
/*   C[m, n] = beta * C[m, n] + sum_t alpha_t * sum_k A_t[m, k] * B_t[k, n]  */
/*                                                                          */
/* m, n and k are COMPOSITE indices: each is a group of up to PMB_MAX_DIMS   */
/* tensor indices, listed fastest-varying first, with one extent per index   */
/* and one stride per index per operand.  An arbitrary index permutation of  */
/* a 4-index tensor is therefore described by strides only and is fused into */
/* the tile loads -- nothing is transposed in memory.                        */
/*                                                                          */
/* Replaces every two-operand einsum of the hot path, e.g.                   */
/*   pp ladder   "abcd,cdij->abij"  pymes/solver/ccd.py:187, eom_ccsd.py:383  */
/*   hh ladder   "klij,abkl->abij"  ccd.py:186 ; I_klij build ccd.py:180      */
/*   ring terms  ccd.py:190-191,202-204,233-235,238-240                       */
/*   X_ac / X_ki ccd.py:213-221,231-232                                       */
/*   T1 dressing ccsd.py:257-286,322-419 ; singles residual ccsd.py:428-436   */
/*   EOM sigma   eom_ccsd.py:288-308,332-383                                  */
/* ------------------------------------------------------------------------ */
struct pmb_ueg_operand;              /* generated operand, declared below    */

typedef struct {
    const double *A;
    const double *B;
    int32_t nk;                      /* number of contracted indices (>= 0)  */
    int32_t _pad;
    int64_t k_ext[PMB_MAX_DIMS];     /* extents of the contracted indices    */
    int64_t a_kstr[PMB_MAX_DIMS];    /* strides of A along them              */
    int64_t b_kstr[PMB_MAX_DIMS];    /* strides of B along them              */
    int64_t a_mstr[PMB_MAX_DIMS];    /* strides of A along the M indices     */
    int64_t b_nstr[PMB_MAX_DIMS];    /* strides of B along the N indices     */
    double alpha;
    /* NULL: A is read from memory.  Otherwise A is never stored: the tiles of */
    /* this term's A operand are EVALUATED by the producer warps of the kernel */
    /* (UEG integrals, see pmb_ueg_operand_t); `A`, a_kstr and a_mstr are then  */
    /* ignored.  At most one term of a contraction may have a generated A.     */
    const struct pmb_ueg_operand *a_gen;
} pmb_term_t;

typedef struct {
    int32_t nm, nn, nterms, _pad;
    int64_t m_ext[PMB_MAX_DIMS];
    int64_t n_ext[PMB_MAX_DIMS];
    int64_t c_mstr[PMB_MAX_DIMS];
    int64_t c_nstr[PMB_MAX_DIMS];
    double *C;
    double beta;                     /* 0: C is overwritten and never read   */
    pmb_term_t terms[PMB_MAX_TERMS];
} pmb_contract_t;

/* bytes of scratch needed for `d` (split-K partial sums; 0 if not split)    */
size_t pmb_contract_workspace(const pmb_contract_t *d);
int pmb_contract(const pmb_contract_t *d, void *ws, size_t ws_bytes,
                 pmb_stream_t stream);
/* tuning/diagnostic knobs: force a tile configuration (-1 = heuristic; bits   */
/* 0-2 the configuration, +8 flips the copy interleaving, +16 makes generated  */
/* operands use the scanning producer instead of the non-zero walker, +32 keeps */
/* the n-fastest tile order for launches with a generated operand, +256 keeps   */
/* it for stored operands too instead of the banded order) and                 */
/* a split-K factor (0 = heuristic).                                          */
void pmb_contract_set_tuning(int tile_config, int split_k);
/* L2 budget (bytes) for one operand's k window; contractions whose smaller      */
/* operand exceeds it are issued as a fixed-order sequence of k-window launches */
/* accumulating in C.  0 disables the windows, a negative value restores the     */
/* defaults (40 MiB for the single-role tile kernels, off for the               */
/* warp-specialised kernel).                                                    */
void pmb_contract_set_panel_bytes(long long bytes);

/* ------------------------------------------------------------------------ */
/* HBM-bound elementwise / reduction kernels                                 */
/* All 4-index tensors below are addressed as X[a,b,i,j] with explicit       */
/* element strides s[4] so that views of V_pqrs can be passed directly.      */
/* ------------------------------------------------------------------------ */

/* out[a,b,i,j] = alpha * in[a,b,i,j] (+ beta * out[a,b,i,j] if beta != 0).   */
/* `in` may be any permuted / sliced view.  Replaces the `.copy()` and        */
/* `+= V_block` statements of ccd.py:178,185 and ccsd.py:323-415.             */
int pmb_axpby4(const int64_t ext[4], double alpha, const double *in,
               const int64_t in_str[4], double beta, double *out,
               const int64_t out_str[4], pmb_stream_t stream);

/* Row blocks: the three functions below work on the rows a in [a_lo, a_lo+na)  */
/* of an [a,b,i,j] tensor (the (ab)-block a rank owns in a sharded run); the   */
/* amplitude-shaped arguments are the LOCAL contiguous [na,nv,no,no] blocks.   */
/* a_lo = 0, na = nv is the whole tensor.                                     */

/* T2[a,b,i,j] = V_abij[a,b,i,j] / (e_i + e_j - e_a - e_b + shift)            */
/* pymes/solver/mp2.py:16-18.  V_abij points at row a_lo (strided view).      */
int pmb_mp2_amplitudes(int no, int nv, int a_lo, int na, const double *eps_i,
                       const double *eps_a, double shift, const double *V_abij,
                       const int64_t v_str[4], double *T2, pmb_stream_t stream);

/* dT = R * (1 / (e_i + e_j - e_a - e_b + shift)); T += delta * dT;          */
/* scal[0] = sum dT^2.    ccd.py:123-124,138 ; ccsd.py:152-156,177-179,197   */
/* denom_mode = 1 replaces the sum by the PRODUCT e_i e_j (-e_a)(-e_b): that  */
/* is what the reference's Brueckner branch executes (ccd.py:118,             */
/* einsum('i,j,a,b->abij')), reproduced for bug-compatibility.                */
int pmb_update_doubles(int no, int nv, int a_lo, int na, const double *eps_i,
                       const double *eps_a, double shift, double delta, int denom_mode,
                       const double *R, double *dT, double *T2, double *scal, void *ws,
                       size_t ws_bytes, pmb_stream_t stream);
/* same for singles: dT1 = R1 / (e_i - e_a + shift); T1 += delta * dT1       */
int pmb_update_singles(int no, int nv, const double *eps_i, const double *eps_a,
                       double shift, double delta, const double *R1, double *dT1,
                       double *T1, pmb_stream_t stream);

/* scal[0] = 2 sum tau[a,b,i,j] V[i,j,a,b]; scal[1] = - sum tau[a,b,i,j] V[i,j,b,a]; */
/* scal[2] = sum T2^2,   tau = T2 + T1 (x) T1 (T1 may be NULL).               */
/* ccd.py:256-262,137 ; ccsd.py:458-466,196 ; mp2.py:19-20 (exchange written  */
/* there as V[j,i,a,b]: set mp2_form = 1).                                   */
/* V_ijab and T1 are the FULL tensors; T2 is the local row block.              */
int pmb_energy_doubles(int no, int nv, int a_lo, int na, const double *T2, const double *T1,
                       const double *V_ijab, const int64_t v_str[4],
                       int mp2_form, double *scal, void *ws, size_t ws_bytes,
                       pmb_stream_t stream);

/* Tt[a,b,i,j] = 2 T[a,b,i,j] - T[b,a,i,j]          ccd.py:199                */
/* (swap_ij = 1:  2 T[a,b,i,j] - T[a,b,j,i]          ccsd.py:430)             */
int pmb_tilde(int no, int nv, const double *T2, double *Tt, int swap_ij,
              pmb_stream_t stream);

/* R[a,b,i,j] (+)= Ex[a,b,i,j] + Ex[b,a,j,i]                                 */
/* ccd.py:249-252 ; eom_ccsd.py:254,377.  accumulate = 0 overwrites R.        */
int pmb_sym_baji(int no, int nv, const double *Ex, double *R, int accumulate,
                 pmb_stream_t stream);

/* out[k] = sum_x X_k[x] * Y[x], k = 0..nvec-1     diis.py:65-78;             */
/* eom_ccsd.py:103-109 ; feast_eom_ccsd.py:137-146                            */
int pmb_dots(int nvec, const double *const *X, const double *Y, int64_t n,
             double *out, void *ws, size_t ws_bytes, pmb_stream_t stream);

/* out[x] = sum_k c[k] * X_k[x] (+ beta*out)       diis.py:97-103;            */
/* eom_ccsd.py:122-147 ; feast_eom_ccsd.py:151-164                            */
int pmb_lincomb(int nvec, const double *c_host, const double *const *X,
                int64_t n, double beta, double *out, pmb_stream_t stream);

size_t pmb_reduce_workspace(void);

/* Batched strided multiply-reduce (no tensor cores; HBM/L2-bound):             */
/*   out[I] = beta * out[I] + alpha * sum_R A[I,R] * B[I,R]                      */
/* I = up to 4 output indices (an operand that lacks one has stride 0 there),   */
/* R = up to 4 summed indices present in both operands; first listed index is   */
/* the fastest.  Covers the einsums of the reference that are NOT matrix        */
/* products because an index is shared by both operands AND the output:        */
/* the H-bar diagonals eom_ccsd.py:169-266 ("kica,caki->ai", "kiab,abkj->abij", */
/* "ijcd,cdij->ij", ...).  nr = 0 gives an elementwise product.                 */
typedef struct {
    const double *A;
    const double *B;
    double *out;
    int32_t ni, nr;
    int64_t i_ext[PMB_MAX_DIMS], o_istr[PMB_MAX_DIMS], a_istr[PMB_MAX_DIMS], b_istr[PMB_MAX_DIMS];
    int64_t r_ext[PMB_MAX_DIMS], a_rstr[PMB_MAX_DIMS], b_rstr[PMB_MAX_DIMS];
    double alpha, beta;
} pmb_bdot_t;
int pmb_bdot(const pmb_bdot_t *d, pmb_stream_t stream);

/* Matrix-vector form of a contraction (no tensor cores; HBM-bound):               */
/*   out[X] = beta * out[X] + alpha * sum_K vec[K] * B[K, X]                        */
/* for the einsums of the hot path in which one operand carries NO output index   */
/* and the other is o.v^3-sized -- the T1 dressing of the Fock matrix             */
/* "ci,iabc->ab", "ci,iacb->ab", "jacb,bj->ac", "jabc,bj->ac" (ccsd.py:257-286)    */
/* and of the singles residual (ccsd.py:428-436).  As a 128-row DMMA tile they     */
/* use 1/128 of the tensor work and gather 8 bytes at a time (measured 0.7 TB/s);  */
/* here B is streamed once, coalesced along whichever of X / K is its unit-stride  */
/* direction (first listed index of the group).  Deterministic (fixed order).      */
typedef struct {
    const double *vec;
    const double *B;
    double *out;
    int32_t nk, nx;
    int64_t k_ext[PMB_MAX_DIMS], v_kstr[PMB_MAX_DIMS], b_kstr[PMB_MAX_DIMS];
    int64_t x_ext[PMB_MAX_DIMS], b_xstr[PMB_MAX_DIMS], o_xstr[PMB_MAX_DIMS];
    double alpha, beta;
} pmb_gemv_t;
int pmb_gemv(const pmb_gemv_t *d, pmb_stream_t stream);

/* Shifted complex diagonal preconditioner of the FEAST linear solves             */
/* feast_eom_ccsd.py:341-342:  y = x / (z - diag + shift), x = xr + i xi,        */
/* z = zr + i zi, diag real; evaluated on the fly (nothing of size n is stored   */
/* per quadrature node).  yr/yi may alias xr/xi.                                 */
int pmb_cdiv_shifted(int64_t n, const double *diag, double zr, double zi, double shift,
                     const double *xr, const double *xi, double *yr, double *yi,
                     pmb_stream_t stream);

/* ------------------------------------------------------------------------ */
/* UEG momentum-conserving two-electron integrals  pymes/model/ueg.py:265-596 */
/*                                                                          */
/* The reference's triple Python loop (ueg.py:384-507) evaluates, for every  */
/* (p, r, q'), s = map[k_q' - (k_r - k_p)] and a weight that depends only on */
/* the pair (p, r) plus -- for the non-hermitian TC term -- a dot product    */
/* with (k_r - k_s).  The build is therefore split into                      */
/*   1. pmb_ueg_umat        : u_mat(q) for every distinct transfer q          */
/*   2. pmb_ueg_pair_tables : W0[p,r], W1[p,r] for one of the nine branches   */
/*   3. pmb_ueg_build_block : the HBM-bound dense write of any V sub-block    */
/*      V[p,q,r,s] = delta(s, s*) * ( W0a[p,r] + W1a[p,r]*(k_r-k_s).(k_r-k_p) */
/*                                   + 1/2 (W0s[p,r] + W0s[q,s]) )            */
/*      (W0s carries the (pq)(rs)<->(qp)(sr) symmetrised effective two-body   */
/*      term of ueg.py:509-513), so each rank of a sharded run generates      */
/*      only its own rows and V_pqrs never has to exist as one array.         */
/* ------------------------------------------------------------------------ */
typedef struct {
    int32_t n_orb;            /* number of plane waves nP                      */
    int32_t imax;             /* index-map half width (ueg.py:119-125,153)     */
    int32_t n_occ;            /* n_ele / 2                                     */
    int32_t n_ele;
    double omega;             /* cell volume (ueg.py:69)                       */
    const double *u_table;    /* correlator u tabulated over n2 = |k_int|^2:   */
    int32_t u_table_len;      /*   u_table[n2] = u(n2 (2 pi/L)^2); the host    */
    int32_t _pad;             /*   evaluates any of ueg.py:740-956 once        */
    const int32_t *kvec;      /* [nP][3] integer k vectors (device)            */
    const double *kp;         /* [nP][3] (k + shift) 2 pi / L (device)         */
    const int32_t *index_map; /* [(2 imax+1)^3] orbital index or -1 (device)   */
} pmb_ueg_t;

/* branches of eval_2b_integrals, in the order of ueg.py:411-504             */
#define PMB_UEG_COULOMB 0
#define PMB_UEG_RPA 1
#define PMB_UEG_ONLY_2B 2
#define PMB_UEG_ONLY_HERMI_2B 3
#define PMB_UEG_ONLY_NON_HERMI_2B 4
#define PMB_UEG_EFFECT_2B 5
#define PMB_UEG_EXCHANGE_1 6
#define PMB_UEG_EXCHANGE_2 7
#define PMB_UEG_EXCHANGE_3 8

/* out[n] = sum_{k' in [-cutoff,cutoff]^3} (k1.k2) u(k1^2) u(k2^2) / Omega,     */
/* k1 = 2 pi k'/L (L = box_len), k2 = 2 pi q_n/L - k1, for nq integer transfer  */
/* vectors q (device, int32 [nq][3]).                                          */
/* ueg.py:581-596 (cutoff = 30 there).  One CTA per q, fixed-order reduction.  */
int pmb_ueg_umat(const pmb_ueg_t *u, double box_len, int cutoff, int nq,
                 const int32_t *qvec, double *out, pmb_stream_t stream);

/* W0[p*nP+r], W1[p*nP+r] for `mode`; umat_pr[p*nP+r] = u_mat(k_r - k_p) is     */
/* needed by modes 2 and 3 only (may be NULL otherwise).                       */
int pmb_ueg_pair_tables(const pmb_ueg_t *u, int mode, const double *umat_pr,
                        double *W0, double *W1, pmb_stream_t stream);

/* Momentum-compressed block: out[np][nq][nr] = V[p,q,r,s*(p,q,r)] if s* lies in  */
/* [lo[3], lo[3]+ext[3]), else 0 -- the one candidate non-zero of every dense    */
/* row, same formula and rounding as pmb_ueg_build_block (ext[3] / 1 smaller:     */
/* 0.93 GB instead of 454 GB for V_abcd at 515 orbitals).  8 B per element.       */
int pmb_ueg_build_nz(const pmb_ueg_t *u, const double *W0a, const double *W1a,
                     const double *W0s, const int32_t lo[4], const int32_t ext[4],
                     double *out, pmb_stream_t stream);

/* Dense block out[np][nq][nr][ns] of V for p in [lo[0], lo[0]+ext[0]) etc.    */
/* W1a and W0s may be NULL.                                                    */
int pmb_ueg_build_block(const pmb_ueg_t *u, const double *W0a, const double *W1a,
                        const double *W0s, const int32_t lo[4], const int32_t ext[4],
                        double *out, pmb_stream_t stream);

/* ------------------------------------------------------------------------ */
/* Never-materialised UEG integrals (SURVEY 8(f).1).                          */
/*                                                                          */
/* The v^4 block V_abcd of the 54-electron / ~500-orbital UEG is 300-450 GB  */
/* of which one element in v is non-zero.  Instead of being written to HBM    */
/* by pmb_ueg_build_block and read back by the particle-particle ladder       */
/* "abcd,cdij->abij" (ccd.py:187), it can be handed to pmb_contract as a      */
/* GENERATED A operand: the producer warps fill the shared-memory tile with   */
/* exactly the values pmb_ueg_build_block would have stored (same formula,    */
/* same rounding), so results are bit-identical to the materialised path and  */
/* the block costs no memory and no HBM traffic.                              */
/*                                                                          */
/* The operand is the sub-block V[lo[0]+.., lo[1]+.., lo[2]+.., lo[3]+..] of  */
/* the (p,q,r,s) tensor; m_axis[d] / k_axis[d] say which of the four V axes   */
/* (0 = p .. 3 = s) the d-th M index / K index of the contraction runs over   */
/* (extents come from the contraction descriptor).  Every axis must appear    */
/* exactly once.  Limits: n_orb <= 2047, imax <= 27.                          */
/* ------------------------------------------------------------------------ */
typedef struct pmb_ueg_operand {
    pmb_ueg_t ueg;
    const double *W0a;        /* pair tables as for pmb_ueg_build_block        */
    const double *W1a;        /*   (W1a, W0s may be NULL)                      */
    const double *W0s;
    const int32_t *lin;       /* [nP] n^2 kx + n ky + kz, n = 2 imax + 1 (dev) */
    /* optional compressed values from pmb_ueg_build_nz for this very block:     */
    /* nz[(p-lo0, q-lo1, r-lo2)] = V[p,q,r,s*].  With it the producers only LOOK */
    /* UP the non-zero elements (no FP64 arithmetic next to the DMMA stream, one */
    /* load requested tiles ahead); NULL: they evaluate the formula in place.    */
    const double *nz;
    int32_t lo[4];
    int32_t m_axis[PMB_MAX_DIMS];
    int32_t k_axis[PMB_MAX_DIMS];
} pmb_ueg_operand_t;

/* ------------------------------------------------------------------------ */
/* Block-diagonal contraction: the momentum-blocked path of SURVEY 8(f).1.     */
/*                                                                          */
/* As the matrix [(p,q),(r,s)] a UEG integral block is non-zero only where     */
/* k_p + k_q = k_r + k_s (pymes/model/ueg.py:411-513): grouped by total        */
/* momentum it is block diagonal, and a contraction over (r,s) -- the          */
/* particle-particle ladder "abcd,cdij->abij" (ccd.py:187, eom_ccsd.py:383),   */
/* "kbcd,cdij->kbij" / "alcd,cdij->alij" of the T1 dressing (ccsd.py:405-419)  */
/* -- only has to visit the diagonal blocks: 2 o^2 nnz(V) flop instead of      */
/* 2 o^2 v^4 (54e / 515 plane waves: 4.8e10 instead of 8.3e13).                */
/*                                                                          */
/*   C[c_moff[m] + cn(n)] = beta * C[..] + alpha * sum_{k in group(m)}          */
/*                          A[a_moff[m] + a_koff[k]] * B[b_koff[k] + bn(n)]     */
/*   n = n1 * n0_ext + n0,  bn(n) = n1 * b_n1str + n0,  cn(n) = n1 * c_n1str + n0*/
/*                                                                          */
/* Rows and entries are LISTS (element offsets into A, B, C), sorted by group  */
/* by the host; `tiles` cuts every group's rows into pieces of <= 64:           */
/* {first row, rows, first entry, entries} per tile.  Every row belongs to at   */
/* most one tile; rows outside all tiles are not touched.  With the            */
/* compressed integrals of pmb_ueg_build_nz, a_moff = ((p*nq + q)*nr) and       */
/* a_koff = r (the s index is implied by the group).  One CTA per (tile, 128    */
/* columns), DMMA.m8n8k4, fixed summation order, no workspace.                 */
/* ------------------------------------------------------------------------ */
typedef struct {
    const double *A;
    const double *B;
    double *C;
    const int64_t *a_moff;    /* [rows]    device */
    const int64_t *c_moff;    /* [rows]    device */
    const int64_t *a_koff;    /* [entries] device */
    const int64_t *b_koff;    /* [entries] device */
    const int32_t *tiles;     /* [n_tiles][4] device, 16-byte aligned */
    int32_t n_tiles;
    int32_t n0_ext;           /* unit-stride column index (e.g. (i,j) flattened) */
    int32_t n1_ext;           /* outer column index (e.g. the right-hand side), 1 if none */
    int32_t _pad;
    int64_t b_n1str;
    int64_t c_n1str;
    double alpha;
    double beta;              /* 0: C is overwritten (in the tiles' rows) and never read */
} pmb_blocked_t;
int pmb_blocked_contract(const pmb_blocked_t *d, pmb_stream_t stream);

/* A UEG integral block times a ONE-index contraction (T1 dressing products       */
/* "abid,dj->abij", "abcj,ci->abij", "iabc,cj->iabj", "iacb,cj->iajb",           */
/* ccsd.py:322-419):                                                            */
/*   out[..] = beta * out[..] + alpha * val[x] * D[idx[x] * d_ystr + j * d_jstr]  */
/* for every output element (x0,x1,x2,j); x = x0*x_str[0] + x1*x_str[1] +         */
/* x2*x_str[2] addresses the tables val[x] = V[x0,x1,x2 | y*] and idx[x] = y*      */
/* (the one orbital the reference's lookup ueg.py:395-404 finds on the summed     */
/* axis, local index, or -1).  `out` is C-contiguous with extents ext[0..3]       */
/* (slowest first); role[d] in {0,1,2,3} says which of x0, x1, x2, j output       */
/* dimension d is.  HBM-bound: one pass over the output instead of one over the   */
/* o.v^3 block.                                                                  */
typedef struct {
    const double *val;
    const int32_t *idx;
    const double *D;
    double *out;
    int32_t ext[4];
    int32_t role[4];
    int64_t x_str[3];
    int64_t d_ystr;
    int64_t d_jstr;
    double alpha;
    double beta;
} pmb_gather_t;
int pmb_gather_expand(const pmb_gather_t *d, pmb_stream_t stream);

/* ------------------------------------------------------------------------ */
/* Block-diagonal x block-diagonal contraction: two momentum-conserving        */
/* operands, rows and entries from A, entries and columns from B, all three    */
/* sorted by group on the host.  Per tile {r0, rn, e0, en, c0, cn}:            */
/*   C[c_row[r] + c_col[n]] += alpha * sum_{k = e0}^{e0+en-1}                    */
/*                  A[a_row[r] + a_ent[k]] * B[b_ent[k] + b_col[n]]             */
/* for r in [r0, r0+rn), n in [c0, c0+cn).  Elements outside every tile are    */
/* not touched (the caller clears or scales them first).  Every C element      */
/* belongs to at most one tile; one CTA per tile, FP64 FMA from shared memory, */
/* fixed summation order, no atomics, no workspace.                            */
/* ------------------------------------------------------------------------ */
typedef struct {
    const double *A;
    const double *B;
    double *C;
    const int64_t *a_row;     /* [rows]    device */
    const int64_t *a_ent;     /* [entries] device */
    const int64_t *b_ent;     /* [entries] device */
    const int64_t *b_col;     /* [columns] device */
    const int64_t *c_row;     /* [rows]    device */
    const int64_t *c_col;     /* [columns] device */
    const int32_t *tiles;     /* [n_tiles][6] device */
    int32_t n_tiles;
    int32_t _pad;
    double alpha;
} pmb_group_t;
int pmb_group_contract(const pmb_group_t *d, pmb_stream_t stream);

/* The same product for n_batch right-hand sides at once (Davidson / FEAST     */
/* blocks): right-hand side b reads A + b*a_bstr, B + b*b_bstr and writes        */
/* C + b*c_bstr with the one set of lists and tiles in g.  A batch stride of 0  */
/* shares that operand between all right-hand sides (c_bstr only when          */
/* n_batch == 1).  One CTA per (tile, right-hand side); same summation order    */
/* as pmb_group_contract, no atomics.  1 <= n_batch <= 65535.                   */
typedef struct {
    pmb_group_t g;
    int32_t n_batch;
    int32_t _pad;
    int64_t a_bstr;
    int64_t b_bstr;
    int64_t c_bstr;
} pmb_group_batched_t;
int pmb_group_contract_batched(const pmb_group_batched_t *d, pmb_stream_t stream);

/* Momentum residue of a strided tensor of rank 1..4:                          */
/*   out[0] = max |x[i0,..]| over the elements with sum_d key_d[i_d] != 0,       */
/* key_d = keys + (ext[0] + .. + ext[d-1]) (per-axis signed momentum labels,    */
/* device), 0 when there is none.  One pass over the tensor; out is device.    */
int pmb_momentum_residue(int ndim, const int64_t ext[4], const int64_t str[4], const double *x,
                         const int64_t *keys, double *out, pmb_stream_t stream);

/* ------------------------------------------------------------------------ */
/* Synthetic non-hermitian integrals (BASELINE.json configs[2]; SURVEY 8(d) C3   */
/* recipe): out[np][nq][nr][ns] = V[lo[0]+.., lo[1]+.., lo[2]+.., lo[3]+..] with  */
/*   V[p,q,r,s] = eps * table[ h(seed, c) >> 48 ],                                */
/*   c = min(((p n + q) n + r) n + s, ((q n + p) n + s) n + r)                    */
/* -- a counter-based generator keyed on the canonical representative of the      */
/* one symmetry a transcorrelated V keeps, (pq)(rs) <-> (qp)(sr)                  */
/* (pymes/util/fcidump.py:147-149); h = two splitmix64 finaliser rounds of         */
/* c * 0x9E3779B97F4A7C15 + seed * 0xBF58476D1CE4E5B9 + 1; `table` = 65536        */
/* standard-normal quantiles (device, made by the host).  Bit-identical to        */
/* pymes_b200/util/synthetic.py on the host.  HBM-bound, 8 B per element.         */
/* ------------------------------------------------------------------------ */
int pmb_synth_block(int n_orb, unsigned long long seed, double eps, const double *table,
                    const int32_t lo[4], const int32_t ext[4], double *out, pmb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PYMES_B200_H */
