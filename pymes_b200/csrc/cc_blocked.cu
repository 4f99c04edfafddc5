// Block-diagonal contraction on the FP64 tensor cores: pmb_blocked_contract.
//
// A momentum-conserving integral block V[p,q,r,s] (pymes/model/ueg.py:411-513: non-zero only
// where k_p + k_q = k_r + k_s) is, as the matrix [(p,q), (r,s)] that a contraction such as the
// particle-particle ladder "abcd,cdij->abij" (ccd.py:187) multiplies with, block diagonal once
// its rows and columns are grouped by total momentum Q: rows (p,q) with k_p + k_q = Q meet only
// the entries (r,s) with k_r + k_s = Q.  At 54 electrons / 515 plane waves the 5.7e10 elements of
// V_abcd hold 3.3e7 non-zeros in 3809 such groups (SURVEY 8(f).1), so the ladder is 4.8e10 flop
// instead of 8.3e13.  The host sorts the row and entry lists by group and cuts each group's rows
// into tiles of <= 64; one CTA owns (row tile, 128 columns), walks the group's entries 16 at a
// time through a two-stage cp.async pipeline and multiplies with DMMA.m8n8k4.  Every address is
// list-driven (row / entry offset tables), so the same kernel serves the compressed integrals
// (pmb_ueg_build_nz: A[a_moff[m] + a_koff[k]] with a_koff = r) and a dense strided block.
//
// Each C element is written by exactly one CTA in a fixed summation order: deterministic, no
// atomics, no workspace.
#include "common.cuh"

namespace pmb {
namespace {

constexpr int BM = 64, BN = 128, BK = 16, NT = 256, SPAD = 4;
constexpr int LDA = BM + SPAD, LDB = BN + SPAD;   // (LD mod 16) == 4: conflict-free fragment loads
constexpr int WARPS_M = 2, WARPS_N = 4;
constexpr int WM = BM / WARPS_M, WN = BN / WARPS_N;
constexpr int MT = WM / 8, NTL = WN / 8;
constexpr int KCH = 512;                           // entry offsets staged in shared memory at a time
constexpr int PER_A = BM * BK / NT, PER_B = BN * BK / NT;
static_assert(NT % BK == 0 && NT % BN == 0, "thread -> element mappings");
static_assert(WARPS_M * WARPS_N * 32 == NT, "warp grid");

constexpr size_t kSmemBytes = (size_t)2 * BK * (LDA + LDB) * 8 + (size_t)2 * KCH * 8 + (size_t)2 * BM * 8;

__device__ __forceinline__ void dmma(double (&c)[2], double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
        : "+d"(c[0]), "+d"(c[1])
        : "d"(a), "d"(b));
}
// src_bytes = 0 zero-fills the destination (ragged edges need no branches)
__device__ __forceinline__ void cp_async8z(unsigned smem_addr, const double *gsrc, int src_bytes) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(smem_addr), "l"(gsrc), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
}

__global__ void __launch_bounds__(NT, 2) blocked_kernel(const __grid_constant__ pmb_blocked_t p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *As = reinterpret_cast<double *>(smem_raw);          // [2][BK][LDA]
    double *Bs = As + 2 * BK * LDA;                              // [2][BK][LDB]
    long long *s_ak = reinterpret_cast<long long *>(Bs + 2 * BK * LDB);   // [KCH]
    long long *s_bk = s_ak + KCH;                                // [KCH]
    long long *s_am = s_bk + KCH;                                // [BM]
    long long *s_cm = s_am + BM;                                 // [BM]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int warp_m = warp % WARPS_M, warp_n = warp / WARPS_M;
    const int4 tile = *reinterpret_cast<const int4 *>(p.tiles + 4 * (size_t)blockIdx.x);
    const int m0 = tile.x, mn = tile.y, k0 = tile.z, kn = tile.w;
    const int n_base = blockIdx.y * BN;
    const int nrem = p.n0_ext * p.n1_ext - n_base;

    for (int i = tid; i < BM; i += NT) {
        const bool ok = i < mn;
        s_am[i] = ok ? p.a_moff[m0 + i] : 0;
        s_cm[i] = ok ? p.c_moff[m0 + i] : 0;
    }
    __syncthreads();
    // B tile: a thread keeps its column and steps the entry
    const int b_n = tid % BN, b_k0 = tid / BN;
    constexpr int B_KSTEP = NT / BN;
    const bool b_nok = b_n < nrem;
    long long b_noff = 0;
    if (b_nok) {
        const int n = n_base + b_n, q = n / p.n0_ext;
        b_noff = (long long)q * p.b_n1str + (n - q * p.n0_ext);
    }
    // A tile: a thread keeps its entry and steps the row
    const int a_k = tid % BK, a_m0 = tid / BK;
    constexpr int A_MSTEP = NT / BK;
    const unsigned as_base = (unsigned)__cvta_generic_to_shared(As);
    const unsigned bs_base = (unsigned)__cvta_generic_to_shared(Bs);

    double acc[MT][NTL][2];
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < NTL; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    for (int kc = 0; kc < kn; kc += KCH) {
        const int kcn = min(KCH, kn - kc);
        __syncthreads();           // the previous chunk's tables are no longer read
        for (int i = tid; i < kcn; i += NT) {
            s_ak[i] = p.a_koff[k0 + kc + i];
            s_bk[i] = p.b_koff[k0 + kc + i];
        }
        __syncthreads();
        const int nkt = (kcn + BK - 1) / BK;
        auto issue = [&](int kt, int st) {
            const int kb = kt * BK;
            {
                const int k = kb + a_k;
                const bool kok = k < kcn;
                const long long ko = kok ? s_ak[k] : 0;
                const unsigned dst = as_base + (unsigned)(((st * BK + a_k) * LDA + a_m0) * 8);
#pragma unroll
                for (int it = 0; it < PER_A; ++it) {
                    const int m = a_m0 + it * A_MSTEP;
                    const bool ok = kok && m < mn;
                    cp_async8z(dst + (unsigned)(it * A_MSTEP * 8), p.A + (ok ? s_am[m] + ko : 0), ok ? 8 : 0);
                }
            }
            {
                const unsigned dst = bs_base + (unsigned)(((st * BK + b_k0) * LDB + b_n) * 8);
#pragma unroll
                for (int it = 0; it < PER_B; ++it) {
                    const int k = kb + b_k0 + it * B_KSTEP;
                    const bool ok = b_nok && k < kcn;
                    cp_async8z(dst + (unsigned)(it * B_KSTEP * LDB * 8), p.B + (ok ? s_bk[k] + b_noff : 0),
                               ok ? 8 : 0);
                }
            }
            cp_async_commit();
        };
        issue(0, 0);
        for (int kt = 0; kt < nkt; ++kt) {
            const int st = kt & 1;
            if (kt + 1 < nkt) {
                issue(kt + 1, st ^ 1);
                cp_async_wait<1>();
            } else {
                cp_async_wait<0>();
            }
            __syncthreads();       // everyone's copies of tile kt have landed
            const double *a = As + st * BK * LDA + warp_m * WM + (lane >> 2) + (lane & 3) * LDA;
            const double *b = Bs + st * BK * LDB + warp_n * WN + (lane >> 2) + (lane & 3) * LDB;
#pragma unroll
            for (int ks = 0; ks < BK / 4; ++ks) {
                double af[MT], bf[NTL];
#pragma unroll
                for (int i = 0; i < MT; ++i) af[i] = a[ks * 4 * LDA + i * 8];
#pragma unroll
                for (int j = 0; j < NTL; ++j) bf[j] = b[ks * 4 * LDB + j * 8];
#pragma unroll
                for (int i = 0; i < MT; ++i)
#pragma unroll
                    for (int j = 0; j < NTL; ++j) dmma(acc[i][j], af[i], bf[j]);
            }
            __syncthreads();       // stage st may be overwritten by the next iteration's copies
        }
    }

    // ---- epilogue: C = alpha * acc + beta * C, one owner per element ----------------------
    const int row0 = warp_m * WM + (lane >> 2), col0 = warp_n * WN + (lane & 3) * 2;
    long long c_noff[NTL][2];
#pragma unroll
    for (int j = 0; j < NTL; ++j)
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            const int nl = col0 + j * 8 + c;
            long long off = 0;
            if (nl < nrem) {
                const int n = n_base + nl, q = n / p.n0_ext;
                off = (long long)q * p.c_n1str + (n - q * p.n0_ext);
            }
            c_noff[j][c] = off;
        }
    const bool rd = p.beta != 0.0;
#pragma unroll
    for (int i = 0; i < MT; ++i) {
        const int ml = row0 + i * 8;
        if (ml >= mn) continue;
        double *crow = p.C + s_cm[ml];
        double old[NTL][2];
#pragma unroll
        for (int j = 0; j < NTL; ++j)
#pragma unroll
            for (int c = 0; c < 2; ++c)
                old[j][c] = (rd && col0 + j * 8 + c < nrem) ? crow[c_noff[j][c]] : 0.0;
#pragma unroll
        for (int j = 0; j < NTL; ++j)
#pragma unroll
            for (int c = 0; c < 2; ++c)
                if (col0 + j * 8 + c < nrem) crow[c_noff[j][c]] = p.alpha * acc[i][j][c] + p.beta * old[j][c];
    }
}

}  // namespace
}  // namespace pmb

using namespace pmb;

extern "C" int pmb_blocked_contract(const pmb_blocked_t *d, pmb_stream_t stream) {
    if (!d || d->n_tiles < 0 || d->n0_ext < 1 || d->n1_ext < 1) return PMB_E_BADARG;
    if (d->n_tiles == 0) return 0;
    if (!d->A || !d->B || !d->C || !d->a_moff || !d->c_moff || !d->a_koff || !d->b_koff || !d->tiles)
        return PMB_E_BADARG;
    const long long n = (long long)d->n0_ext * d->n1_ext;
    if (n > 0x7fffffffLL) return PMB_E_UNSUPPORTED;
    const long long tiles_n = (n + BN - 1) / BN;
    if (tiles_n > 65535) return PMB_E_UNSUPPORTED;
    // per device, so not cached: a host-side call of a microsecond
    cudaError_t e = cudaFuncSetAttribute(blocked_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)kSmemBytes);
    if (e != cudaSuccess) return (int)e;
    dim3 grid((unsigned)d->n_tiles, (unsigned)tiles_n);
    blocked_kernel<<<grid, NT, kSmemBytes, (cudaStream_t)stream>>>(*d);
    count_launch();
    return cuda_status();
}

// ---------------------------------------------------------------------------
// pmb_gather_expand: a momentum-conserving integral block times a ONE-index contraction.
//
// out[x0,x1,x2,j] (+)= alpha * sum_y V[x0,x1,x2 | y] * D[y, j] has, for a UEG block, exactly one
// candidate y per (x0,x1,x2) -- the orbital the reference's index lookup finds (ueg.py:395-404).  With
// the values val[x] = V[x, y*(x)] and partners idx[x] = y*(x) (or -1) tabulated once per block and
// summed axis, the product is an HBM-bound pass over the OUTPUT: 8 B written (16 with beta != 0)
// per element, 12 B of table per (x0,x1,x2), instead of a pass over the o.v^3 block (25 GB at
// v = 488).  These are the T1 dressing products "abid,dj->abij", "abcj,ci->abij", "iabc,cj->iabj",
// "iacb,cj->iajb" of ccsd.py:322-419.  One thread per output element in output memory order (the
// output is C-contiguous); `role` says which output dimension is x0 / x1 / x2 / j.
// ---------------------------------------------------------------------------
namespace pmb {
namespace {

// I = unsigned when the output has fewer than 2^31 elements (32-bit index arithmetic), else long long
template <typename I>
__global__ void __launch_bounds__(256) gather_expand_kernel(const __grid_constant__ pmb_gather_t p) {
    const I e3 = (I)p.ext[3], e2 = (I)p.ext[2], e1 = (I)p.ext[1];
    const long long total = (long long)p.ext[0] * p.ext[1] * p.ext[2] * p.ext[3];
    const bool rd = p.beta != 0.0;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total;
         e += (long long)gridDim.x * blockDim.x) {
        I c[4];
        I q = (I)e;
        c[3] = q % e3; q /= e3;
        c[2] = q % e2; q /= e2;
        c[1] = q % e1;
        c[0] = q / e1;
        long long xoff = 0, j = 0;
#pragma unroll
        for (int d = 0; d < 4; ++d) {
            if (p.role[d] == 3) j = (long long)c[d];
            else xoff += (long long)c[d] * p.x_str[p.role[d]];
        }
        const int t = __ldg(p.idx + xoff);
        double v = 0.0;
        if (t >= 0) v = p.alpha * __ldg(p.val + xoff) * __ldg(p.D + (long long)t * p.d_ystr + j * p.d_jstr);
        if (rd) v += p.beta * p.out[e];
        p.out[e] = v;
    }
}

}  // namespace
}  // namespace pmb

extern "C" int pmb_gather_expand(const pmb_gather_t *d, pmb_stream_t stream) {
    if (!d || !d->val || !d->idx || !d->D || !d->out) return PMB_E_BADARG;
    long long total = 1;
    int seen = 0;
    for (int k = 0; k < 4; ++k) {
        if (d->ext[k] < 1 || d->role[k] < 0 || d->role[k] > 3) return PMB_E_BADARG;
        seen |= 1 << d->role[k];
        total *= d->ext[k];
    }
    if (seen != 15) return PMB_E_BADARG;
    long long blocks = (total + 255) / 256;
    if (blocks > 32LL * kSmCount) blocks = 32LL * kSmCount;
    if (total < (1LL << 31))
        gather_expand_kernel<unsigned><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(*d);
    else
        gather_expand_kernel<long long><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(*d);
    count_launch();
    return cuda_status();
}

// ---------------------------------------------------------------------------
// pmb_group_contract: both operands momentum-conserving (amplitudes, ring intermediates).
//
// A ring product such as "kaic,cbkj->abij" (ccd.py:233) of two tensors that are each non-zero only
// where their signed momenta sum to zero is block diagonal in ALL three index pairs at once: rows
// (a,i), entries (k,c) and columns (b,j) with the same group key g meet only each other.  At 54
// electrons / 515 plane waves that is 1140 groups of at most 27 x 27 x 27 instead of one
// 13176 x 13176 x 13176 product.  The host sorts the three lists by group and cuts each group into
// tiles of <= 32 rows x 32 columns; one CTA owns a tile, gathers 32-entry slabs of A and B into
// shared memory and accumulates with FP64 FMA (2 x 2 outputs per thread).  The work per product is
// a few 10^7 flop, so the tensor cores would buy nothing here; what matters is that no zero is
// read.  Each C element belongs to one tile: deterministic, no atomics.
//
// A tile of at most GE outputs with more than GK entries (a diagonal build such as "kcdl,cdil->ki":
// 1 x 1 tiles of ~8.8e3 entries at 54 electrons) would walk its slabs on a single thread.  Such a
// tile takes the entry-split form instead: each of the GNT threads sums every GNT-th entry, then a
// fixed-order tree in shared memory combines the partial sums -- still deterministic, no atomics.
// The form is chosen per tile from (rn, en, cn), so the host plan and the C ABI do not know it.
// ---------------------------------------------------------------------------
namespace pmb {
namespace {

constexpr int GT = 32, GK = 32, GNT = 256, GE = 4;
static_assert(GE * GNT <= GK * (GT + 1), "the entry-split partial sums reuse As");
static_assert((GNT & (GNT - 1)) == 0, "tree reduction over GNT threads");

// One tile of a group product.  A, B and C are the operands of one right-hand side: the batched
// entry point offsets the descriptor's pointers by its batch strides.
__device__ __forceinline__ void group_tile(const pmb_group_t &p, const double *A, const double *B,
                                           double *C) {
    __shared__ double As[GK][GT + 1];
    __shared__ double Bs[GK][GT + 1];
    __shared__ long long s_ar[GT], s_cr[GT], s_bc[GT], s_cc[GT];
    const int *tl = p.tiles + 6 * (size_t)blockIdx.x;
    const int r0 = tl[0], rn = tl[1], e0 = tl[2], en = tl[3], c0 = tl[4], cn = tl[5];
    const int tid = threadIdx.x;
    if (tid < GT) {
        const bool ok = tid < rn;
        s_ar[tid] = ok ? p.a_row[r0 + tid] : 0;
        s_cr[tid] = ok ? p.c_row[r0 + tid] : 0;
    } else if (tid < 2 * GT) {
        const int j = tid - GT;
        const bool ok = j < cn;
        s_bc[j] = ok ? p.b_col[c0 + j] : 0;
        s_cc[j] = ok ? p.c_col[c0 + j] : 0;
    }
    const int no = rn * cn;
    if (en > GK && no <= GE) {
        __syncthreads();                          // offsets staged
        double acc[GE];
#pragma unroll
        for (int o = 0; o < GE; ++o) acc[o] = 0.0;
        for (int k = tid; k < en; k += GNT) {
            const long long ae = __ldg(p.a_ent + e0 + k), be = __ldg(p.b_ent + e0 + k);
#pragma unroll
            for (int o = 0; o < GE; ++o)
                if (o < no) acc[o] = fma(__ldg(A + s_ar[o / cn] + ae), __ldg(B + be + s_bc[o % cn]), acc[o]);
        }
        double *red = &As[0][0];                  // [GE][GNT]
#pragma unroll
        for (int o = 0; o < GE; ++o) red[o * GNT + tid] = acc[o];
        for (int w = GNT / 2; w > 0; w >>= 1) {
            __syncthreads();
            if (tid < w) {
#pragma unroll
                for (int o = 0; o < GE; ++o) red[o * GNT + tid] += red[o * GNT + tid + w];
            }
        }
        __syncthreads();
        if (tid < no) C[s_cr[tid / cn] + s_cc[tid % cn]] += p.alpha * red[tid * GNT];
        return;
    }
    const int tx = tid % 16, ty = tid / 16;       // columns tx, tx+16; rows ty, ty+16
    double acc[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
    for (int kc = 0; kc < en; kc += GK) {
        __syncthreads();                          // offsets staged / previous slab consumed
        for (int idx = tid; idx < GK * GT; idx += GNT) {
            const int k = idx / GT, m = idx % GT;
            const bool kok = kc + k < en;
            const long long ae = kok ? __ldg(p.a_ent + e0 + kc + k) : 0;
            const long long be = kok ? __ldg(p.b_ent + e0 + kc + k) : 0;
            As[k][m] = (kok && m < rn) ? __ldg(A + s_ar[m] + ae) : 0.0;
            Bs[k][m] = (kok && m < cn) ? __ldg(B + be + s_bc[m]) : 0.0;
        }
        __syncthreads();
#pragma unroll 8
        for (int k = 0; k < GK; ++k) {
            const double a0 = As[k][ty], a1 = As[k][ty + 16];
            const double b0 = Bs[k][tx], b1 = Bs[k][tx + 16];
            acc[0][0] = fma(a0, b0, acc[0][0]);
            acc[0][1] = fma(a0, b1, acc[0][1]);
            acc[1][0] = fma(a1, b0, acc[1][0]);
            acc[1][1] = fma(a1, b1, acc[1][1]);
        }
    }
    if (en <= 0) __syncthreads();                 // the offsets above are visible
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const int m = ty + 16 * i;
        if (m >= rn) continue;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int n = tx + 16 * j;
            if (n >= cn) continue;
            double *c = C + s_cr[m] + s_cc[n];
            *c += p.alpha * acc[i][j];
        }
    }
}

__global__ void __launch_bounds__(GNT) group_kernel(const __grid_constant__ pmb_group_t p) {
    group_tile(p, p.A, p.B, p.C);
}

// blockIdx.y = right-hand side; a batch stride of 0 shares that operand between all of them
__global__ void __launch_bounds__(GNT) group_batched_kernel(const __grid_constant__ pmb_group_batched_t p) {
    const long long b = blockIdx.y;
    group_tile(p.g, p.g.A + b * p.a_bstr, p.g.B + b * p.b_bstr, p.g.C + b * p.c_bstr);
}

// One pass over a strided tensor: max |x| where the signed momenta of its indices do not cancel.
// Non-negative doubles order like their bit patterns, so the maximum is an integer atomicMax.
struct Residue {
    long long ext[4], str[4], koff[4];   // koff < 0: the axis is absent (extent 1, key 0)
};

__device__ __forceinline__ long long axis_key(const long long *keys, long long koff, long long i) {
    return koff < 0 ? 0 : __ldg(keys + koff + i);
}

__global__ void __launch_bounds__(256) residue_kernel(const __grid_constant__ Residue s, const double *x,
                                                      const long long *keys, unsigned long long *out) {
    __shared__ unsigned long long red[256];
    const long long total = s.ext[0] * s.ext[1] * s.ext[2] * s.ext[3];
    unsigned long long best = 0;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total;
         e += (long long)gridDim.x * blockDim.x) {
        long long q = e;
        const long long i3 = q % s.ext[3]; q /= s.ext[3];
        const long long i2 = q % s.ext[2]; q /= s.ext[2];
        const long long i1 = q % s.ext[1];
        const long long i0 = q / s.ext[1];
        const long long sum = axis_key(keys, s.koff[0], i0) + axis_key(keys, s.koff[1], i1) +
                              axis_key(keys, s.koff[2], i2) + axis_key(keys, s.koff[3], i3);
        if (sum == 0) continue;
        const double v = fabs(x[i0 * s.str[0] + i1 * s.str[1] + i2 * s.str[2] + i3 * s.str[3]]);
        const unsigned long long b = (unsigned long long)__double_as_longlong(v);
        best = b > best ? b : best;
    }
    red[threadIdx.x] = best;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w && red[threadIdx.x + w] > red[threadIdx.x]) red[threadIdx.x] = red[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0 && red[0] != 0) atomicMax(out, red[0]);
}

}  // namespace
}  // namespace pmb

extern "C" int pmb_group_contract(const pmb_group_t *d, pmb_stream_t stream) {
    if (!d || d->n_tiles < 0) return PMB_E_BADARG;
    if (d->n_tiles == 0) return 0;
    if (!d->A || !d->B || !d->C || !d->a_row || !d->a_ent || !d->b_ent || !d->b_col || !d->c_row ||
        !d->c_col || !d->tiles)
        return PMB_E_BADARG;
    group_kernel<<<(unsigned)d->n_tiles, GNT, 0, (cudaStream_t)stream>>>(*d);
    count_launch();
    return cuda_status();
}

extern "C" int pmb_group_contract_batched(const pmb_group_batched_t *d, pmb_stream_t stream) {
    if (!d || d->g.n_tiles < 0 || d->n_batch < 1 || d->n_batch > 65535) return PMB_E_BADARG;
    // each right-hand side owns its outputs: a C shared by several would be summed into twice
    if (d->c_bstr == 0 && d->n_batch > 1) return PMB_E_BADARG;
    if (d->g.n_tiles == 0) return 0;
    const pmb_group_t &g = d->g;
    if (!g.A || !g.B || !g.C || !g.a_row || !g.a_ent || !g.b_ent || !g.b_col || !g.c_row || !g.c_col || !g.tiles)
        return PMB_E_BADARG;
    group_batched_kernel<<<dim3((unsigned)g.n_tiles, (unsigned)d->n_batch), GNT, 0, (cudaStream_t)stream>>>(*d);
    count_launch();
    return cuda_status();
}

extern "C" int pmb_momentum_residue(int ndim, const int64_t ext[4], const int64_t str[4], const double *x,
                                    const int64_t *keys, double *out, pmb_stream_t stream) {
    if (ndim < 1 || ndim > 4 || !ext || !str || !x || !keys || !out) return PMB_E_BADARG;
    // right-align the axes: missing leading axes have extent 1 and no key
    Residue s;
    long long total = 1, koff = 0;
    for (int d = 0; d < 4; ++d) {
        const int src = d - (4 - ndim);
        s.ext[d] = src >= 0 ? ext[src] : 1;
        s.str[d] = src >= 0 ? str[src] : 0;
        s.koff[d] = src >= 0 ? koff : -1;
        if (s.ext[d] < 1) return PMB_E_BADARG;
        if (src >= 0) koff += ext[src];
        total *= s.ext[d];
    }
    cudaError_t e = cudaMemsetAsync(out, 0, sizeof(double), (cudaStream_t)stream);
    if (e != cudaSuccess) return (int)e;
    long long blocks = (total + 255) / 256;
    if (blocks > 8LL * kSmCount) blocks = 8LL * kSmCount;
    residue_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        s, x, (const long long *)keys, (unsigned long long *)out);
    count_launch();
    return cuda_status();
}

namespace pmb {
namespace {

// Compact <-> dense vectors of one momentum sector: right-hand side b copies n_idx doubles through
// the index list idx (shared by every right-hand side).  Batches run over gridDim.y with a stride
// loop, so any n_batch fits; offsets are 64-bit throughout.  Pure copies: values pass bit-exact.
__global__ void __launch_bounds__(256)
    sector_gather_kernel(int64_t n_batch, int64_t n_idx, const int64_t *__restrict__ idx,
                         const double *__restrict__ src, int64_t src_bstr, double *__restrict__ dst,
                         int64_t dst_bstr) {
    for (int64_t b = blockIdx.y; b < n_batch; b += gridDim.y) {
        const double *s = src + b * src_bstr;
        double *d = dst + b * dst_bstr;
        for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n_idx;
             k += (int64_t)gridDim.x * blockDim.x)
            d[k] = s[idx[k]];
    }
}

__global__ void __launch_bounds__(256)
    sector_scatter_kernel(int64_t n_batch, int64_t n_idx, const int64_t *__restrict__ idx,
                          const double *__restrict__ src, int64_t src_bstr, double *__restrict__ dst,
                          int64_t dst_bstr) {
    for (int64_t b = blockIdx.y; b < n_batch; b += gridDim.y) {
        const double *s = src + b * src_bstr;
        double *d = dst + b * dst_bstr;
        for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n_idx;
             k += (int64_t)gridDim.x * blockDim.x)
            d[idx[k]] = s[k];
    }
}

// About 16 CTAs per SM in all: the index range first, the batch fills what it leaves.
static dim3 sector_grid(int64_t n_batch, int64_t n_idx) {
    long long bx = (n_idx + 255) / 256;
    if (bx > 16LL * kSmCount) bx = 16LL * kSmCount;
    long long by = (16LL * kSmCount) / bx;
    if (by < 1) by = 1;
    if (by > n_batch) by = n_batch;
    if (by > 65535) by = 65535;
    return dim3((unsigned)bx, (unsigned)by, 1);
}

}  // namespace
}  // namespace pmb

extern "C" int pmb_sector_gather(int64_t n_batch, int64_t n_idx, const int64_t *idx, const double *src,
                                 int64_t src_bstr, double *dst, int64_t dst_bstr, pmb_stream_t stream) {
    if (n_batch < 1 || n_idx < 1 || !idx || !src || !dst) return PMB_E_BADARG;
    sector_gather_kernel<<<sector_grid(n_batch, n_idx), 256, 0, (cudaStream_t)stream>>>(
        n_batch, n_idx, idx, src, src_bstr, dst, dst_bstr);
    count_launch();
    return cuda_status();
}

extern "C" int pmb_sector_scatter(int64_t n_batch, int64_t n_idx, const int64_t *idx, const double *src,
                                  int64_t src_bstr, double *dst, int64_t dst_bstr, pmb_stream_t stream) {
    if (n_batch < 1 || n_idx < 1 || !idx || !src || !dst) return PMB_E_BADARG;
    sector_scatter_kernel<<<sector_grid(n_batch, n_idx), 256, 0, (cudaStream_t)stream>>>(
        n_batch, n_idx, idx, src, src_bstr, dst, dst_bstr);
    count_launch();
    return cuda_status();
}
