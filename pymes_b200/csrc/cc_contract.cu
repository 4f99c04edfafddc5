// Generic strided binary tensor contraction on the FP64 tensor cores of B200.
//
//   C[m,n] = beta*C[m,n] + sum_t alpha_t * sum_k A_t[m,k] * B_t[k,n]
//
// m, n, k are composite indices (groups of up to 4 tensor indices each, with
// per-operand element strides), so every index permutation that the coupled-
// cluster equations need is expressed by strides and is fused into the tile
// loads: nothing is ever transposed in HBM.
//
// sm_100a has no tcgen05 kind for f64, so FP64 tensor work is issued as
// warp-level mma.sync.m8n8k4.f64 (SASS DMMA.8x8x4).  One DMMA per SM
// sub-partition every 16 cycles is the hardware peak (64 FMA/clk/SM), which
// leaves ample issue slots for everything else; the kernels are organised so
// that the DMMA pipe is the only thing that can be busy.  Two kernels:
//   * contract_ws_kernel (large shapes): one 128x128x16 CTA per SM, four
//     producer warps (offset tables, cp.async gathers -- or, for a generated
//     operand, the expansion of compressed UEG integrals into the tile) and
//     eight consumer warps (fragment LDS + DMMA only) coupled by mbarriers over
//     a 4-stage shared-memory ring; ragged tiles use compile-time widths;
//   * contract_kernel (small / skinny shapes): single-role CTAs, 3-4-stage
//     cp.async pipeline, one __syncthreads per k-tile, split-K when the output
//     has fewer tiles than the machine has CTA slots.
// Common to both: shared tiles stored [k][x] with a +4 pad (stores of either
// thread mapping and the fragment loads are bank-conflict free), and a
// thread->element mapping of the gathers that follows each operand's
// unit-stride direction (x-fast or k-fast) so global accesses stay coalesced
// to full 32 B sectors for any permutation.
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "ueg_device.cuh"

namespace pmb {

constexpr int BK = 16;
constexpr int SPAD = 4;
static_assert(BK == 16, "the main loop is written for four DMMA k sub-steps per tile");

template <int V>
struct IntC {
    static constexpr int value = V;
};

struct TermDev {
    const double *A;
    const double *B;
    int nk, K;
    int k_ext[PMB_MAX_DIMS];
    long long a_kstr[PMB_MAX_DIMS], b_kstr[PMB_MAX_DIMS];
    long long a_mstr[PMB_MAX_DIMS], b_nstr[PMB_MAX_DIMS];
    double alpha;
    int a_kfast, b_kfast;
    int b_vec2;              // B tile copied 16 bytes at a time (see make_gat_vec2)
    int kt_begin, nkt;
};

struct Params {
    int nm, nn, nterms;
    int M, N;
    int m_ext[PMB_MAX_DIMS], n_ext[PMB_MAX_DIMS];
    long long c_mstr[PMB_MAX_DIMS], c_nstr[PMB_MAX_DIMS];
    double *C;
    double beta;
    int tiles_m, tiles_n;
    int raster_m_fast;       // consecutive CTAs walk m inside one column of tiles (see launch_ws)
    int raster_group;        // > 1: consecutive CTAs walk m inside a band of that many tile rows (tile_coords)
    int total_ktiles, ktiles_per_split, nsplit;
    int kt_base, kt_limit;   // k-tile window of this launch (K-panel), [0, total_ktiles) if not panelled
    // Tail launch (see pmb_contract): this launch covers the output tiles [tile_base, tile_base +
    // gridDim.x) only, split over k; partial sums go to ws[split][tile - tile_base][BM x BN].
    int tile_base, tail;
    double *ws;
    TermDev t[PMB_MAX_TERMS];
    // generated A operand (never-materialised UEG integrals): term index or -1
    int gen_term;
    int gen_n3;                       // (2 imax + 1)^3, size of the index map
    int gen_map_smem;                 // index map, plane-wave vectors and lin[] staged in shared memory
    int gen_walk;                     // K = (s fastest, r): producers walk the non-zeros directly
    int gen_l0;                       // imax (n^2 + n + 1)
    int gen_lo[4];
    int gen_m_axis[PMB_MAX_DIMS], gen_k_axis[PMB_MAX_DIMS];
    pmb_ueg_t gen_ueg;
    const double *gen_W0a, *gen_W1a, *gen_W0s;
    const int *gen_lin;
    const double *gen_nz;             // compressed values [ext_p][ext_q][ext_r] or NULL
    int gen_ext[4];                   // block extents along (p, q, r, s)
};

// Generated operand: table entries are not element offsets but packed 64-bit words
//   [63..44] partial sum of the flattened index-map location  +L(p) +L(q) -L(r)  (signed)
//   [43..33] p   [32..22] q   [21..11] r   [10..0] s          (orbital indices, 11 bits each)
// Every V axis belongs to either the M or the K group, so (row word + k word) is the full
// description of one element: the orbital fields are disjoint and the signed location parts
// add in two's complement.  The element is non-zero iff index_map[loc] == s -- exactly the
// reference's test (ueg.py:397-407), flattened bounds check included.
constexpr int kGenLocShift = 44, kGenFieldBits = 11, kGenFieldMask = (1 << kGenFieldBits) - 1;

__device__ __forceinline__ long long gen_decomp(const Params &p, int idx, int nd, const int *ext, const int *axis) {
    long long e = 0;
#pragma unroll
    for (int d = 0; d < PMB_MAX_DIMS; ++d) {
        if (d < nd) {
            const int x = ext[d];
            const int q = idx / x;
            const int ax = axis[d];
            const int orb = p.gen_lo[ax] + (idx - q * x);
            const int sign = ax == 2 ? -1 : (ax == 3 ? 0 : 1);
            e += (long long)(sign * p.gen_lin[orb]) * (1LL << kGenLocShift);
            e += (long long)orb << (kGenFieldBits * (3 - ax));
            idx = q;
        }
    }
    return e;
}

// Is the element described by word e non-zero?  `map` is the index map (shared-memory copy
// when it fits, else global).
__device__ __forceinline__ bool gen_hit(const Params &p, const int *map, long long e) {
    const int loc = (int)(e >> kGenLocShift);
    const int sstar = (unsigned)loc < (unsigned)p.gen_n3 ? map[loc] : -1;
    return sstar == ((int)e & kGenFieldMask);
}
// position of element (p,q,r,.) in the compressed value table
__device__ __forceinline__ long long gen_nz_index(const Params &p, int op, int oq, int orr) {
    return ((long long)(op - p.gen_lo[0]) * p.gen_ext[1] + (oq - p.gen_lo[1])) * p.gen_ext[2] + (orr - p.gen_lo[2]);
}
// value of a non-zero element
__device__ __forceinline__ double gen_value(const Params &p, long long e) {
    if (p.gen_nz)
        return __ldg(p.gen_nz + gen_nz_index(p, (int)(e >> (3 * kGenFieldBits)) & kGenFieldMask,
                                             (int)(e >> (2 * kGenFieldBits)) & kGenFieldMask,
                                             (int)(e >> kGenFieldBits) & kGenFieldMask));
    return ueg_value(p.gen_ueg, p.gen_W0a, p.gen_W1a, p.gen_W0s, (int)(e >> (3 * kGenFieldBits)) & kGenFieldMask,
                     (int)(e >> (2 * kGenFieldBits)) & kGenFieldMask, (int)(e >> kGenFieldBits) & kGenFieldMask,
                     (int)e & kGenFieldMask);
}

// Output tile of the `tile`-th CTA.  Three orders:
//   n fastest (default of the single-role kernels),
//   m fastest (generated A operand: a wave streams one column of B tiles together),
//   banded   (stored operands, warp-specialised kernel): bands of `raster_group` tile rows, m fastest
//            inside a band.  A wave of 148 CTAs then covers ~12 x 12 tiles and shares 12 A row panels
//            and 12 B column panels through L2, instead of one A panel and 103 B panels: the ring-type
//            contraction at v = 488 moved 187 GB of DRAM traffic per launch n-fastest (45 x its
//            algorithmic 4.2 GB; ncu, profiles/r2_ring_ncu.md).
__device__ __forceinline__ void tile_coords(const Params &p, int tile, int &tile_m, int &tile_n) {
    if (p.raster_m_fast) {
        tile_n = tile / p.tiles_m;
        tile_m = tile % p.tiles_m;
    } else if (p.raster_group > 1) {
        const int per = p.raster_group * p.tiles_n;
        const int band = tile / per;
        const int first = band * p.raster_group;
        const int rows = min(p.raster_group, p.tiles_m - first);
        const int in = tile - band * per;
        tile_n = in / rows;
        tile_m = first + in - tile_n * rows;
    } else {
        tile_n = tile % p.tiles_n;
        tile_m = tile / p.tiles_n;
    }
}

__device__ __forceinline__ long long decomp(int idx, int nd, const int *ext,
                                            const long long *str) {
    long long off = 0;
#pragma unroll
    for (int d = 0; d < PMB_MAX_DIMS; ++d) {
        if (d < nd) {
            const int e = ext[d];
            const int q = idx / e;
            off += (long long)(idx - q * e) * str[d];
            idx = q;
        }
    }
    return off;
}

__device__ __forceinline__ void dmma(double (&c)[2], double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
        : "+d"(c[0]), "+d"(c[1])
        : "d"(a), "d"(b));
}

// 8-byte asynchronous global->shared copies (LDGSTS).  Shared addresses are 32-bit
// shared-window byte addresses so that the per-copy offset folds into the instruction.
__device__ __forceinline__ void cp_async8(unsigned smem_addr, const double *gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(smem_addr), "l"(gsrc));
}
// src_bytes = 0 zero-fills the destination: ragged tile edges need no branches
__device__ __forceinline__ void cp_async8z(unsigned smem_addr, const double *gsrc, int src_bytes) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(smem_addr), "l"(gsrc), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
}

// Per-thread description of the asynchronous gather of one [BK][BX] operand tile.
// Two thread->element mappings exist, chosen per operand by its unit-stride direction:
//   x-fast: consecutive threads walk x (the operand is unit-stride along m/n); a thread
//           keeps x and steps k by NT/BX per copy,
//   k-fast: every 4 lanes read 4 consecutive k (one 32 B sector), 8 x per warp; a thread
//           keeps k and steps x per copy.
// Both reduce to the same straight-line code: address = base + tab[it * tstep], shared
// destination = sdst + it * dstep, so the k-tile loop has no mapping- or edge-dependent
// branches and ptxas can place the copies in the issue shadow of the DMMAs.
// Rows/columns outside the tensor have table offset 0: they read valid memory and only feed
// accumulator rows/columns that are never stored.  Only k >= K must be zero-filled
// (src-size 0), which also turns the copies of tiles beyond the k range into no-ops.
struct Gat {
    const double *base;     // operand + fixed part of the offset
    const long long *tab;   // varying part (shared): tab[it * tstep]
    unsigned sdst;          // shared-window byte address of copy 0
    int tstep, dstep;       // per-copy increments (table elements, shared bytes)
    int k0, kinc;           // k index of copy `it` is k0 + it * kinc
};

template <int BX, int NT>
__device__ __forceinline__ Gat make_gat(unsigned S, const double *__restrict__ G, const long long *s_x,
                                        const long long *s_k, bool kfast, int tid) {
    constexpr int LD = BX + SPAD;
    constexpr int KSTEP = NT / BX;
    constexpr int KQ = BK / 4, NW = NT / 32;
    static_assert(NW % KQ == 0, "warps must tile the k quads");
    constexpr int XSTEP = (NW / KQ) * 8;
    const int lane = tid & 31, warp = tid >> 5;
    const int x = kfast ? (warp / KQ) * 8 + (lane >> 2) : tid % BX;
    const int k = kfast ? (warp % KQ) * 4 + (lane & 3) : tid / BX;
    const long long *fixed = kfast ? s_k + k : s_x + x;
    Gat g;
    g.base = G + *fixed;
    g.tab = kfast ? s_x + x : s_k + k;
    g.tstep = kfast ? XSTEP : KSTEP;
    g.sdst = S + (unsigned)((k * LD + x) * 8);
    g.dstep = kfast ? XSTEP * 8 : KSTEP * LD * 8;
    g.k0 = k;
    g.kinc = kfast ? 0 : KSTEP;
    return g;
}

template <int IT0, int IT1>
__device__ __forceinline__ void gat_issue(const Gat &g, int krem) {
#pragma unroll
    for (int it = IT0; it < IT1; ++it) {
        const long long off = g.tab[it * g.tstep];
        cp_async8z(g.sdst + (unsigned)(it * g.dstep), g.base + off, (g.k0 + it * g.kinc < krem) ? 8 : 0);
    }
}
// same, with the table look-ups of CHUNK copies issued back to back before the copies that
// depend on them (the dedicated producer warps have the registers for it)
template <int PER, int CHUNK>
__device__ __forceinline__ void gat_issue_batched(const Gat &g, int krem) {
    static_assert(PER % CHUNK == 0, "copies must split into whole chunks");
#pragma unroll
    for (int c0 = 0; c0 < PER; c0 += CHUNK) {
        long long off[CHUNK];
#pragma unroll
        for (int j = 0; j < CHUNK; ++j) off[j] = g.tab[(c0 + j) * g.tstep];
#pragma unroll
        for (int j = 0; j < CHUNK; ++j) {
            const int it = c0 + j;
            cp_async8z(g.sdst + (unsigned)(it * g.dstep), g.base + off[j], (g.k0 + it * g.kinc < krem) ? 8 : 0);
        }
    }
}

// 16-byte form of the x-fast gather, for operands whose composite x index is DENSE in memory
// (consecutive x are consecutive doubles), whose k strides are even and whose base is 16-byte
// aligned -- tau of the ladder when it lives in a pitch-padded buffer ([v,v,736] for o = 27: a
// 729-double pitch leaves every other row misaligned).  A thread owns a PAIR of columns and steps
// k; half as many LDGSTS as the 8-byte form.
__device__ __forceinline__ void cp_async16z(unsigned smem_addr, const double *gsrc, int src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(smem_addr), "l"(gsrc), "r"(src_bytes));
}
template <int BX, int NT>
__device__ __forceinline__ Gat make_gat_vec2(unsigned S, const double *__restrict__ G, const long long *s_x,
                                             const long long *s_k, int tid) {
    constexpr int LD = BX + SPAD;
    constexpr int HX = BX / 2;
    constexpr int KSTEP = NT / HX;
    static_assert(NT % HX == 0 && BK % KSTEP == 0, "pairs of columns must tile the producer threads");
    const int x = 2 * (tid % HX), k = tid / HX;
    Gat g;
    g.base = G + s_x[x];
    g.tab = s_k + k;
    g.tstep = KSTEP;
    g.sdst = S + (unsigned)((k * LD + x) * 8);
    g.dstep = KSTEP * LD * 8;
    g.k0 = k;
    g.kinc = KSTEP;
    return g;
}
template <int PER, int CHUNK>
__device__ __forceinline__ void gat_issue_vec2(const Gat &g, int krem) {
    static_assert(PER % CHUNK == 0, "copies must split into whole chunks");
#pragma unroll
    for (int c0 = 0; c0 < PER; c0 += CHUNK) {
        long long off[CHUNK];
#pragma unroll
        for (int j = 0; j < CHUNK; ++j) off[j] = g.tab[(c0 + j) * g.tstep];
#pragma unroll
        for (int j = 0; j < CHUNK; ++j) {
            const int it = c0 + j;
            cp_async16z(g.sdst + (unsigned)(it * g.dstep), g.base + off[j], (g.k0 + it * g.kinc < krem) ? 16 : 0);
        }
    }
}

// Epilogue shared by both kernels.  DMMA C fragment: row = lane/4, cols = 2*(lane%4) + {0,1}.
// `row0` / `col0` are this lane's first row / column inside the CTA tile.  With beta != 0 the
// old values of one fragment row (2*NTL elements) are all loaded before anything is stored:
// the loads are independent, so one row costs one memory round trip instead of 2*NTL
// dependent read-modify-write chains (k-window launches pay this once per window).
template <int MT, int NTL>
__device__ __forceinline__ void store_tile(const Params &p, double (&acc)[MT][NTL][2], const long long *s_cm,
                                           const long long *s_cn, int row0, int col0, int mrem, int nrem,
                                           int ncols = NTL) {
    // only the first `ncols` fragment columns of the warp tile are in use (ragged tiles of
    // the warp-specialised kernel): the others never reach memory
    nrem = min(nrem, col0 - (col0 & 7) + ncols * 8);
    const bool rd = p.beta != 0.0;
#pragma unroll
    for (int i = 0; i < MT; ++i) {
        const int ml = row0 + i * 8;
        if (ml >= mrem) continue;
        double *crow = p.C + s_cm[ml];
        if (rd) {
            double old[NTL][2];
#pragma unroll
            for (int j = 0; j < NTL; ++j)
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    const int nl = col0 + j * 8 + c;
                    old[j][c] = nl < nrem ? crow[s_cn[nl]] : 0.0;
                }
#pragma unroll
            for (int j = 0; j < NTL; ++j)
#pragma unroll
                for (int c = 0; c < 2; ++c) acc[i][j][c] += p.beta * old[j][c];
        }
#pragma unroll
        for (int j = 0; j < NTL; ++j)
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const int nl = col0 + j * 8 + c;
                if (nl < nrem) crow[s_cn[nl]] = acc[i][j][c];
            }
    }
}

// split-K partial sums: plain row-major [split][M][N] workspace
template <int MT, int NTL>
__device__ __forceinline__ void store_partial(const Params &p, const double (&acc)[MT][NTL][2], int m0, int n0,
                                              int row0, int col0, int mrem, int nrem, int ncols = NTL) {
    nrem = min(nrem, col0 - (col0 & 7) + ncols * 8);
    constexpr int kTailTile = 128;     // tail launches exist for the 128 x 128 kernels only
    double *ws = p.tail ? p.ws + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * (size_t)(kTailTile * kTailTile)
                        : p.ws + (size_t)blockIdx.y * (size_t)p.M * (size_t)p.N;
    const size_t ld = p.tail ? (size_t)kTailTile : (size_t)p.N;
    if (p.tail) m0 = n0 = 0;
#pragma unroll
    for (int i = 0; i < MT; ++i) {
        const int ml = row0 + i * 8;
        if (ml >= mrem) continue;
        double *row = ws + (size_t)(m0 + ml) * ld + n0;
#pragma unroll
        for (int j = 0; j < NTL; ++j) {
            const int nl = col0 + j * 8;
            if (nl < nrem) row[nl] = acc[i][j][0];
            if (nl + 1 < nrem) row[nl + 1] = acc[i][j][1];
        }
    }
}

template <int BM, int BN, int WARPS_M, int WARPS_N, int STAGES, int MINB, bool INTERLEAVE>
__global__ void __launch_bounds__(WARPS_M *WARPS_N * 32, MINB)
    contract_kernel(const __grid_constant__ Params p) {
    constexpr int NT = WARPS_M * WARPS_N * 32;
    constexpr int WM = BM / WARPS_M, WN = BN / WARPS_N;
    constexpr int MT = WM / 8, NTL = WN / 8;
    constexpr int LDA = BM + SPAD, LDB = BN + SPAD;
    constexpr int TPB = NT / (2 * BK);   // k-offset tiles produced per batch (one warp each)
    constexpr int KRING = 2 * TPB;       // ring of k-offset tiles
    constexpr int PER_A = BM * BK / NT, PER_B = BN * BK / NT;
    constexpr int NPARTS = BK / 4;       // one slice of the next tile's copies per DMMA sub-step
    static_assert(NT % BM == 0 && NT % BN == 0, "x-fast mapping needs NT % BX == 0");
    static_assert(PER_A % NPARTS == 0 && PER_B % NPARTS == 0, "tile copies must split evenly");
    static_assert(TPB >= STAGES && (KRING & (KRING - 1)) == 0, "k-offset ring");

    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *As = reinterpret_cast<double *>(smem_raw);    // [STAGES][BK][LDA]
    double *Bs = As + STAGES * BK * LDA;                   // [STAGES][BK][LDB]
    long long *s_k = reinterpret_cast<long long *>(Bs + STAGES * BK * LDB);  // [KRING][2][BK]
    long long *s_am = s_k + KRING * 2 * BK;                // [nterms][BM]
    long long *s_bn = s_am + p.nterms * BM;                // [nterms][BN]

    const unsigned as_base = (unsigned)__cvta_generic_to_shared(As);
    const unsigned bs_base = (unsigned)__cvta_generic_to_shared(Bs);
    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    const int warp_m = warp % WARPS_M, warp_n = warp / WARPS_M;
    const int tile_n = blockIdx.x % p.tiles_n, tile_m = blockIdx.x / p.tiles_n;
    const int m0 = tile_m * BM, n0 = tile_n * BN;
    const int mrem = p.M - m0, nrem = p.N - n0;
    const int kt_lo = p.kt_base + blockIdx.y * p.ktiles_per_split;
    const int kt_hi = min(kt_lo + p.ktiles_per_split, p.kt_limit);

    // term that owns global k-tile g (terms are laid out back to back along k)
    auto term_of = [&](int g) {
        int ti = 0;
        while (ti + 1 < p.nterms && g >= p.t[ti + 1].kt_begin) ++ti;
        return ti;
    };
    // Element offsets of the BK contracted indices of k-tile g, both operands: one warp per
    // tile (lanes 0-15 operand A, 16-31 operand B).  Every warp of the CTA produces one tile
    // of a batch, so no warp falls behind the others at the k-tile barrier.
    auto koffs = [&](int g) {
        if (g < kt_hi) {
            const TermDev &t = p.t[term_of(g)];
            const int kk = lane & (BK - 1);
            const int k = (g - t.kt_begin) * BK + kk;
            long long off = 0;
            if (k < t.K) off = decomp(k, t.nk, t.k_ext, lane >= BK ? t.b_kstr : t.a_kstr);
            s_k[(g & (KRING - 1)) * 2 * BK + lane] = off;
        }
    };
    struct TileGat {
        Gat a, b;
        int krem;
    };
    // gather descriptors of k-tile g into pipeline stage st; tiles beyond the range become
    // zero-fill no-ops (krem = 0)
    auto tile_gat = [&](int g, int st) {
        const int ti = term_of(g < kt_hi ? g : kt_lo);
        const TermDev &t = p.t[ti];
        const long long *ko = s_k + (g & (KRING - 1)) * 2 * BK;
        TileGat r;
        r.a = make_gat<BM, NT>(as_base + (unsigned)(st * BK * LDA * 8), t.A, s_am + ti * BM, ko,
                               t.a_kfast != 0, tid);
        r.b = make_gat<BN, NT>(bs_base + (unsigned)(st * BK * LDB * 8), t.B, s_bn + ti * BN, ko + BK,
                               t.b_kfast != 0, tid);
        r.krem = g < kt_hi ? t.K - (g - t.kt_begin) * BK : 0;
        return r;
    };

    for (int ti = 0; ti < p.nterms; ++ti) {
        const TermDev &t = p.t[ti];
        for (int i = tid; i < BM; i += NT)
            s_am[ti * BM + i] = (i < mrem) ? decomp(m0 + i, p.nm, p.m_ext, t.a_mstr) : 0;
        for (int i = tid; i < BN; i += NT)
            s_bn[ti * BN + i] = (i < nrem) ? decomp(n0 + i, p.nn, p.n_ext, t.b_nstr) : 0;
    }
    if (warp < STAGES) koffs(kt_lo + warp);
    __syncthreads();
#pragma unroll
    for (int s = 0; s < STAGES - 1; ++s) {
        const TileGat r = tile_gat(kt_lo + s, s);
        gat_issue<0, PER_A>(r.a, r.krem);
        gat_issue<0, PER_B>(r.b, r.krem);
        cp_async_commit();
    }

    double acc[MT][NTL][2];
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < NTL; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    // The accumulators hold (sum so far) / alpha of the current term, so no operand is ever
    // scaled in the inner loop: at a term boundary they are rescaled by alpha_old / alpha_new
    // (terms with alpha == 0 are dropped on the host) and once more by alpha in the epilogue.
    int cur_term = term_of(kt_lo);
    double alpha = p.t[cur_term].alpha;
    int term_end = p.t[cur_term].kt_begin + p.t[cur_term].nkt;
    int st = 0;                    // pipeline stage of tile g
    int st_next = STAGES - 1;      // stage that tile g + STAGES - 1 goes to
    int batch = 0;                 // position of g in the current k-offset batch
    for (int g = kt_lo; g < kt_hi; ++g) {
        cp_async_wait<STAGES - 2>();   // tile g has landed (this thread's copies)
        __syncthreads();               // ... everyone's; stage (g-1) is free again
        if (batch == 0) koffs(g + STAGES + warp);
        batch = batch + 1 == TPB ? 0 : batch + 1;
        const TileGat nxt = tile_gat(g + STAGES - 1, st_next);
        if (!INTERLEAVE) {
            gat_issue<0, PER_A>(nxt.a, nxt.krem);
            gat_issue<0, PER_B>(nxt.b, nxt.krem);
            cp_async_commit();
        }
        if (g >= term_end) {
            cur_term = term_of(g);
            const double ratio = alpha / p.t[cur_term].alpha;
            alpha = p.t[cur_term].alpha;
            term_end = p.t[cur_term].kt_begin + p.t[cur_term].nkt;
            if (ratio != 1.0) {
#pragma unroll
                for (int i = 0; i < MT; ++i)
#pragma unroll
                    for (int j = 0; j < NTL; ++j) {
                        acc[i][j][0] *= ratio;
                        acc[i][j][1] *= ratio;
                    }
            }
        }
        const double *a = As + st * BK * LDA + warp_m * WM + (lane >> 2) + (lane & 3) * LDA;
        const double *b = Bs + st * BK * LDB + warp_n * WN + (lane >> 2) + (lane & 3) * LDB;
        auto substep = [&](auto part) {
            constexpr int ks = decltype(part)::value;
            double af[MT], bf[NTL];
#pragma unroll
            for (int i = 0; i < MT; ++i) af[i] = a[ks * 4 * LDA + i * 8];
#pragma unroll
            for (int j = 0; j < NTL; ++j) bf[j] = b[ks * 4 * LDB + j * 8];
            if (INTERLEAVE) {
                gat_issue<ks *(PER_A / NPARTS), (ks + 1) * (PER_A / NPARTS)>(nxt.a, nxt.krem);
                gat_issue<ks *(PER_B / NPARTS), (ks + 1) * (PER_B / NPARTS)>(nxt.b, nxt.krem);
            }
#pragma unroll
            for (int i = 0; i < MT; ++i)
#pragma unroll
                for (int j = 0; j < NTL; ++j) dmma(acc[i][j], af[i], bf[j]);
        };
        substep(IntC<0>{});
        substep(IntC<1>{});
        substep(IntC<2>{});
        substep(IntC<3>{});
        if (INTERLEAVE) cp_async_commit();
        st = st + 1 == STAGES ? 0 : st + 1;
        st_next = st_next + 1 == STAGES ? 0 : st_next + 1;
    }
    if (alpha != 1.0) {
#pragma unroll
        for (int i = 0; i < MT; ++i)
#pragma unroll
            for (int j = 0; j < NTL; ++j) {
                acc[i][j][0] *= alpha;
                acc[i][j][1] *= alpha;
            }
    }
    cp_async_wait<0>();

    // ---- epilogue -------------------------------------------------------
    const int row0 = warp_m * WM + (lane >> 2), col0 = warp_n * WN + (lane & 3) * 2;
    if (p.nsplit > 1) {
        store_partial<MT, NTL>(p, acc, m0, n0, row0, col0, mrem, nrem);
        return;
    }
    __syncthreads();
    for (int i = tid; i < BM; i += NT)
        s_am[i] = (i < mrem) ? decomp(m0 + i, p.nm, p.m_ext, p.c_mstr) : 0;
    for (int i = tid; i < BN; i += NT)
        s_bn[i] = (i < nrem) ? decomp(n0 + i, p.nn, p.n_ext, p.c_nstr) : 0;
    __syncthreads();
    store_tile<MT, NTL>(p, acc, s_am, s_bn, row0, col0, mrem, nrem);
}

// ---------------------------------------------------------------------------
// Warp-specialised variant (the large-shape path).
//
// tools/micro/dmma_issue.cu shows that 8 warps running nothing but the fragment LDS + DMMA
// sub-steps reach 99 % of the FP64 tensor peak, while contract_kernel above sits at ~70 %:
// its warps spend issue time on offset tables, 64-bit gather addresses and LDGSTS between
// the DMMA bursts, and meet at a CTA-wide barrier every k-tile.  Here the two jobs are
// separate warps that only talk through shared-memory mbarriers:
//   * producer warps (one warpgroup, 128 threads, 72 registers) own the k-offset tables,
//     the gather descriptors and the cp.async copies; a stage is published with
//     cp.async.mbarrier.arrive.noinc on full[stage] (the barrier completes when the copies
//     of all 128 threads have landed);
//   * consumer warps (WARPS_M x WARPS_N, 208 registers) wait on full[stage], run the four
//     LDS + DMMA sub-steps and release the stage with one arrive per warp on empty[stage].
// There is no __syncthreads in the k loop and the consumers' instruction stream is the
// microbenchmark's.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
    unsigned ok;
    do {
        asm volatile(
            "{\n.reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n}\n"
            : "=r"(ok)
            : "r"(bar), "r"(parity)
            : "memory");
    } while (!ok);
}
// one non-blocking test of the phase (no "memory" clobber: the caller orders its loads)
__device__ __forceinline__ unsigned mbar_probe(unsigned bar, unsigned parity) {
    unsigned ok;
    asm volatile(
        "{\n.reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity));
    return ok;
}
__device__ __forceinline__ void mbar_arrive(unsigned bar) {
    asm volatile("{\n.reg .b64 st;\nmbarrier.arrive.shared::cta.b64 st, [%0];\n}\n" ::"r"(bar) : "memory");
}
// arrive on `bar` once every cp.async issued so far by this thread has completed
__device__ __forceinline__ void cp_async_arrive(unsigned bar) {
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void producer_sync() { asm volatile("bar.sync 1, 128;\n" ::: "memory"); }

constexpr int kWsProducerThreads = 128;
constexpr int kWsKRing = 16;     // k-offset tiles kept in shared memory (4 batches of 4)

template <int BM, int BN, int WARPS_M, int WARPS_N, int STAGES>
__global__ void __launch_bounds__(WARPS_M *WARPS_N * 32 + kWsProducerThreads, 1)
    contract_ws_kernel(const __grid_constant__ Params p) {
    constexpr int NC = WARPS_M * WARPS_N * 32;     // consumer threads
    constexpr int NP = kWsProducerThreads;
    constexpr int NCW = NC / 32;
    constexpr int WM = BM / WARPS_M, WN = BN / WARPS_N;
    constexpr int MT = WM / 8, NTL = WN / 8;
    constexpr int LDA = BM + SPAD, LDB = BN + SPAD;
    constexpr int TPB = NP / 32;                   // k-offset tiles per batch, one warp each
    constexpr int KRING = kWsKRing;
    constexpr int PER_A = BM * BK / NP, PER_B = BN * BK / NP;
    static_assert(NC % 128 == 0, "setmaxnreg works on whole warpgroups");
    static_assert(NP % BM == 0 && NP % BN == 0, "x-fast mapping needs NP % BX == 0");
    static_assert(KRING == 4 * TPB, "ring must hold four batches (see the hazard note below)");

    extern __shared__ __align__(16) unsigned char smem_raw[];
    unsigned long long *bars = reinterpret_cast<unsigned long long *>(smem_raw);   // full[S], empty[S]
    double *As = reinterpret_cast<double *>(smem_raw + 128);   // [STAGES][BK][LDA]
    double *Bs = As + STAGES * BK * LDA;                        // [STAGES][BK][LDB]
    long long *s_k = reinterpret_cast<long long *>(Bs + STAGES * BK * LDB);  // [KRING][2][BK]
    long long *s_cm = s_k + KRING * 2 * BK;                     // [BM]  C row offsets
    long long *s_cn = s_cm + BM;                                // [BN]  C column offsets
    long long *s_am = s_cn + BN;                                // [nterms][BM]
    long long *s_bn = s_am + p.nterms * BM;                     // [nterms][BN]
    // generated operand only: plane-wave vectors [3 n_orb] and the index map [gen_n3 + 1]
    double *s_kp = reinterpret_cast<double *>(s_bn + p.nterms * BN);
    int *s_map = reinterpret_cast<int *>(s_kp + 3 * p.gen_ueg.n_orb);
    int *s_lin = s_map + p.gen_n3 + 1;                           // [n_orb]

    const unsigned bar_base = (unsigned)__cvta_generic_to_shared(bars);
    const unsigned as_base = (unsigned)__cvta_generic_to_shared(As);
    const unsigned bs_base = (unsigned)__cvta_generic_to_shared(Bs);
    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    // Tile order.  Default: n fastest -- the CTAs of a wave share A row panels through L2.  With a
    // generated A there is nothing to share on that side; m fastest makes a whole wave work on
    // ONE column of tiles, whose equal-sized CTAs start and finish together and therefore
    // stream the same k range of B at the same time: B is read from HBM once per wave instead
    // of once per CTA (ncu: 2.64 TB -> see profiles/ for the pp ladder at v = 488).
    const int tile = (int)blockIdx.x + p.tile_base;
    int tile_m, tile_n;
    tile_coords(p, tile, tile_m, tile_n);
    const int m0 = tile_m * BM, n0 = tile_n * BN;
    const int mrem = p.M - m0, nrem = p.N - n0;
    const int kt_lo = p.kt_base + blockIdx.y * p.ktiles_per_split;
    const int kt_hi = min(kt_lo + p.ktiles_per_split, p.kt_limit);

    auto term_of = [&](int g) {
        int ti = 0;
        while (ti + 1 < p.nterms && g >= p.t[ti + 1].kt_begin) ++ti;
        return ti;
    };

    // ---- common prologue: offset tables of this output tile, barriers ----
    for (int ti = 0; ti < p.nterms; ++ti) {
        const TermDev &t = p.t[ti];
        if (ti == p.gen_term) {
            // generated operand: packed (location, orbitals) words, L0 enters on the row side
            for (int i = tid; i < BM; i += NC + NP)
                s_am[ti * BM + i] = (i < mrem) ? gen_decomp(p, m0 + i, p.nm, p.m_ext, p.gen_m_axis) +
                                                     (long long)p.gen_l0 * (1LL << kGenLocShift)
                                               : 0;
        } else {
            for (int i = tid; i < BM; i += NC + NP)
                s_am[ti * BM + i] = (i < mrem) ? decomp(m0 + i, p.nm, p.m_ext, t.a_mstr) : 0;
        }
        for (int i = tid; i < BN; i += NC + NP)
            s_bn[ti * BN + i] = (i < nrem) ? decomp(n0 + i, p.nn, p.n_ext, t.b_nstr) : 0;
    }
    if (p.gen_term >= 0 && p.gen_map_smem) {
        for (int i = tid; i <= p.gen_n3; i += NC + NP)
            s_map[i] = i < p.gen_n3 ? __ldg(p.gen_ueg.index_map + i) : -1;   // [n3] = sentinel
        for (int i = tid; i < 3 * p.gen_ueg.n_orb; i += NC + NP) s_kp[i] = __ldg(p.gen_ueg.kp + i);
        for (int i = tid; i < p.gen_ueg.n_orb; i += NC + NP) s_lin[i] = __ldg(p.gen_lin + i);
    }
    for (int i = tid; i < BM; i += NC + NP)
        s_cm[i] = (i < mrem) ? decomp(m0 + i, p.nm, p.m_ext, p.c_mstr) : 0;
    for (int i = tid; i < BN; i += NC + NP)
        s_cn[i] = (i < nrem) ? decomp(n0 + i, p.nn, p.n_ext, p.c_nstr) : 0;
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) {
            // full[s]: every producer thread through its cp.async group and -- when a term has
            // a generated operand -- one plain (release) arrive per producer warp, which orders
            // the warp's st.shared tile writes before the consumers' reads
            mbar_init(bar_base + s * 8, p.gen_term >= 0 ? NP + NP / 32 : NP);
            mbar_init(bar_base + (STAGES + s) * 8, NCW);        // empty[s]: every consumer warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncthreads();

    if (warp >= NCW) {
        // =========================== producers ===========================
        asm volatile("setmaxnreg.dec.sync.aligned.u32 72;\n");
        const int ptid = tid - NC, pwarp = warp - NCW;
        // Element offsets of the BK contracted indices of k-tile g (lanes 0-15 operand A,
        // 16-31 operand B), ring slot (g - kt_lo) mod KRING.  Batch b+1 (four tiles) is
        // written just before the producer barrier that opens batch b and is first read after
        // the barrier that opens batch b+1; the slots it overwrites belonged to batch b-3,
        // which every producer had finished when this warp passed the barrier of batch b-1.
        auto koffs = [&](int g) {
            if (g < kt_hi) {
                const TermDev &t = p.t[term_of(g)];
                const int kk = lane & (BK - 1);
                const int k = (g - t.kt_begin) * BK + kk;
                long long off = 0;
                if (k < t.K) {
                    if (lane < BK && term_of(g) == p.gen_term)
                        off = gen_decomp(p, k, t.nk, t.k_ext, p.gen_k_axis);
                    else
                        off = decomp(k, t.nk, t.k_ext, lane >= BK ? t.b_kstr : t.a_kstr);
                }
                s_k[((g - kt_lo) & (KRING - 1)) * 2 * BK + lane] = off;
            }
        };
        koffs(kt_lo + pwarp);
        // Generated operand, fast path (index map and plane-wave vectors staged in shared
        // memory).  This thread owns row gx of the tile and every GKSTEP-th k (x-fast mapping:
        // conflict-free stores).  One element in n_orb is non-zero, so a tile column is 16
        // zero stores plus, now and then, one evaluated element -- whose four pair-table words
        // sit in L2 behind the queue of this SM's own operand copies (measured: ~3000 cycles
        // per load round trip).  The scan for tile g+1 therefore runs at the end of tile g and
        // issues those loads; they are consumed one tile later, off the critical path.
        constexpr int GKSTEP = NP / BM;
        const bool gen_fast = p.gen_term >= 0 && p.gen_map_smem;
        const int gx = ptid % BM, gk0 = ptid / BM;
        const long long gem = p.gen_term >= 0 ? s_am[p.gen_term * BM + gx] : 0;
        unsigned nx_hits = 0;          // bit `it`: element it of the next tile's column is non-zero
        long long nx_e = 0;            // packed word of its first non-zero element
        UegWords nx_w = {0.0, 0.0, 0.0, 0.0};
        auto gen_scan = [&](int g) {
            nx_hits = 0;
            if (g >= kt_hi || term_of(g) != p.gen_term) return;
            const TermDev &t = p.t[p.gen_term];
            const long long *ko = s_k + ((g - kt_lo) & (KRING - 1)) * 2 * BK;
            const int krem = t.K - (g - t.kt_begin) * BK;
            // branch-free, in batches of 8: table words and map entries are independent loads
            // (out-of-range locations read the -1 sentinel that ends the shared map)
#pragma unroll
            for (int h = 0; h < PER_A; h += 8) {
                long long e[8];
                int ss[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) e[j] = gem + ko[gk0 + (h + j) * GKSTEP];
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    ss[j] = s_map[min((unsigned)(e[j] >> kGenLocShift), (unsigned)p.gen_n3)];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const bool hit = ss[j] == ((int)e[j] & kGenFieldMask) && gk0 + (h + j) * GKSTEP < krem;
                    nx_hits |= (hit ? 1u : 0u) << (h + j);
                }
            }
            if (nx_hits) {
                nx_e = gem + ko[gk0 + (__ffs(nx_hits) - 1) * GKSTEP];
                const int op = (int)(nx_e >> (3 * kGenFieldBits)) & kGenFieldMask,
                          oq = (int)(nx_e >> (2 * kGenFieldBits)) & kGenFieldMask,
                          orr = (int)(nx_e >> kGenFieldBits) & kGenFieldMask;
                if (p.gen_nz)
                    nx_w.w0 = ueg_ld<true>(p.gen_nz + gen_nz_index(p, op, oq, orr));
                else
                    nx_w = ueg_load_words<true>(p.gen_ueg.n_orb, p.gen_W0a, p.gen_W1a, p.gen_W0s, op, oq, orr,
                                                (int)nx_e & kGenFieldMask);
            }
        };
        // Walker (the pp ladder and every other contraction over K = (r, s) with s fastest):
        // for a row (p, q) the non-zeros are one per r, at s = s*(p, q, r), i.e. at the
        // increasing K positions r_l * ext_s + (s* - lo_s).  Instead of testing all 16 elements
        // of every tile column, the thread keeps the position of its NEXT non-zero: a tile costs
        // 16 zero stores and one compare, and the pair-table words of a non-zero are requested
        // when the previous one is placed -- ext_s / 16 tiles before they are needed.
        static_assert(GKSTEP == 1, "the walker owns whole tile columns");
        const bool gen_walk = gen_fast && p.gen_walk;
        const int wk_ext_s = gen_walk ? p.t[p.gen_term].k_ext[0] : 1;
        const int wk_ext_r = gen_walk ? p.t[p.gen_term].k_ext[1] : 0;
        const int wk_loc = (int)(gem >> kGenLocShift);      // L0 + L(p) + L(q) of this row
        const int wk_p = (int)(gem >> (3 * kGenFieldBits)) & kGenFieldMask;
        const int wk_q = (int)(gem >> (2 * kGenFieldBits)) & kGenFieldMask;
        const double *wk_nz = p.gen_nz ? p.gen_nz + gen_nz_index(p, wk_p, wk_q, p.gen_lo[2]) : nullptr;
        int wk_c = 0;                  // next local r to examine
        int wk_k = 0x7fffffff;         // local K position of the pending non-zero (none: INT_MAX)
        int wk_r = 0, wk_s = 0;        // its r and s orbitals
        UegWords wk_w = {0.0, 0.0, 0.0, 0.0};
        auto wk_advance = [&]() {
            wk_k = 0x7fffffff;
            while (wk_c < wk_ext_r) {
                const int c = wk_c++;
                const int r = p.gen_lo[2] + c;
                const int sst = s_map[min((unsigned)(wk_loc - s_lin[r]), (unsigned)p.gen_n3)];
                const int sl = sst - p.gen_lo[3];
                if (sst >= 0 && (unsigned)sl < (unsigned)wk_ext_s) {
                    wk_k = c * wk_ext_s + sl;
                    wk_r = r;
                    wk_s = sst;
                    if (p.gen_nz)
                        wk_w.w0 = ueg_ld<true>(wk_nz + c);
                    else
                        wk_w = ueg_load_words<true>(p.gen_ueg.n_orb, p.gen_W0a, p.gen_W1a, p.gen_W0s, wk_p, wk_q, r,
                                                    sst);
                    break;
                }
            }
        };
        if (gen_walk && gx < mrem) {
            // first K position this CTA covers inside the generated term (split-K / multi-term)
            const int kstart = max(kt_lo - p.t[p.gen_term].kt_begin, 0) * BK;
            wk_c = kstart / wk_ext_s;
            wk_advance();
            while (wk_k < kstart) wk_advance();
        }
        int st = 0, batch = 0;
        static_assert(STAGES <= 8, "one byte of wk_dirty per ring stage");
        constexpr unsigned kClean = 0xfeu, kFull = 0xffu;
        unsigned long long wk_dirty = ~0ULL;   // every stage: content unknown (kFull)
        unsigned empty_parity = 1;     // first pass over the ring: the stages are free
        for (int g = kt_lo; g < kt_hi; ++g) {
            if (batch == 0) {
                koffs(g + TPB + pwarp);
                producer_sync();
            }
            if (gen_fast && !gen_walk && g == kt_lo) gen_scan(g);       // prime the look-ahead
            batch = batch + 1 == TPB ? 0 : batch + 1;
            mbar_wait(bar_base + (STAGES + st) * 8, empty_parity);
            const int ti = term_of(g);
            const TermDev &t = p.t[ti];
            const long long *ko = s_k + ((g - kt_lo) & (KRING - 1)) * 2 * BK;
            const int krem = t.K - (g - t.kt_begin) * BK;
            const Gat gb = t.b_vec2 ? make_gat_vec2<BN, NP>(bs_base + (unsigned)(st * BK * LDB * 8), t.B,
                                                            s_bn + ti * BN, ko + BK, ptid)
                                    : make_gat<BN, NP>(bs_base + (unsigned)(st * BK * LDB * 8), t.B, s_bn + ti * BN,
                                                       ko + BK, t.b_kfast != 0, ptid);
            if (ti == p.gen_term) {
                // B first: its copies are in flight while the A tile is written
                if (t.b_vec2)
                    gat_issue_vec2<PER_B / 2, 8>(gb, krem);
                else
                    gat_issue_batched<PER_B, 8>(gb, krem);
                double *dst = As + st * BK * LDA + gk0 * LDA + gx;
                if (gen_walk) {
                    // The tile column of this row is zero except, once in ~ext_s / 16 tiles, one element.
                    // Instead of 16 zero stores per tile the thread remembers what it wrote into each
                    // ring stage (one byte per stage: kClean, a k position, or kFull = unknown / several)
                    // and, when the stage comes round again, clears exactly that.  (PMB_WS_DEBUG runs
                    // showed the producers' shared-memory traffic costing 2.4 % of the DMMA rate.)
                    const int kbase = (g - t.kt_begin) * BK;
                    const unsigned was = (unsigned)((wk_dirty >> (8 * st)) & 0xffULL);
                    if (was == kFull) {
#pragma unroll
                        for (int it = 0; it < PER_A; ++it) dst[it * LDA] = 0.0;
                    } else if (was != kClean) {
                        dst[was * LDA] = 0.0;
                    }
                    unsigned now = kClean;
                    while (wk_k < kbase + BK) {
                        const unsigned pos = (unsigned)(wk_k - kbase);
                        dst[pos * LDA] =
                            p.gen_nz ? wk_w.w0
                                     : ueg_combine(wk_w, p.gen_W1a != nullptr, p.gen_W0s != nullptr, s_kp, wk_p,
                                                   wk_r, wk_s);
                        now = now == kClean ? pos : kFull;
                        wk_advance();
                    }
                    wk_dirty = (wk_dirty & ~(0xffULL << (8 * st))) | ((unsigned long long)now << (8 * st));
                } else if (gen_fast) {
                    unsigned hits = nx_hits;               // scanned one tile ago
#pragma unroll
                    for (int it = 0; it < PER_A; ++it) dst[it * GKSTEP * LDA] = 0.0;
                    if (hits) {
                        const int it = __ffs(hits) - 1;
                        hits &= hits - 1;
                        dst[it * GKSTEP * LDA] =
                            p.gen_nz ? nx_w.w0
                                     : ueg_combine(nx_w, p.gen_W1a != nullptr, p.gen_W0s != nullptr, s_kp,
                                                   (int)(nx_e >> (3 * kGenFieldBits)) & kGenFieldMask,
                                                   (int)(nx_e >> kGenFieldBits) & kGenFieldMask,
                                                   (int)nx_e & kGenFieldMask);
                    }
                    while (hits) {                         // a second one in the same column: rare
                        const int it = __ffs(hits) - 1;
                        hits &= hits - 1;
                        dst[it * GKSTEP * LDA] = gen_value(p, gem + ko[gk0 + it * GKSTEP]);
                    }
                } else {
                    // fallback (tables too large for shared memory): scan and evaluate in place
                    unsigned hits = 0;
#pragma unroll
                    for (int it = 0; it < PER_A; ++it) {
                        const int k = gk0 + it * GKSTEP;
                        if (k < krem && gen_hit(p, p.gen_ueg.index_map, gem + ko[k])) hits |= 1u << it;
                        dst[it * GKSTEP * LDA] = 0.0;
                    }
                    while (hits) {
                        const int it = __ffs(hits) - 1;
                        hits &= hits - 1;
                        dst[it * GKSTEP * LDA] = gen_value(p, gem + ko[gk0 + it * GKSTEP]);
                    }
                }
            } else {
                const Gat ga = make_gat<BM, NP>(as_base + (unsigned)(st * BK * LDA * 8), t.A, s_am + ti * BM, ko,
                                                t.a_kfast != 0, ptid);
                gat_issue_batched<PER_A, 8>(ga, krem);
                if (t.b_vec2)
                    gat_issue_vec2<PER_B / 2, 8>(gb, krem);
                else
                    gat_issue_batched<PER_B, 8>(gb, krem);
                wk_dirty |= 0xffULL << (8 * st);          // a stored operand's tile now lives in this stage
            }
            if (p.gen_term >= 0) {
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_base + st * 8);
            }
            cp_async_arrive(bar_base + st * 8);
            if (gen_fast && !gen_walk) gen_scan(g + 1);    // tile g is published; look ahead
            if (++st == STAGES) {
                st = 0;
                empty_parity ^= 1;
            }
        }
        cp_async_wait<0>();
        return;
    }

    // ============================= consumers =============================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 208;\n");
    const int warp_m = warp % WARPS_M, warp_n = warp / WARPS_M;
    double acc[MT][NTL][2];
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < NTL; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    // accumulators hold (sum so far) / alpha of the current term (see contract_kernel)
    int cur_term = term_of(kt_lo);
    double alpha = p.t[cur_term].alpha;
    int term_end = p.t[cur_term].kt_begin + p.t[cur_term].nkt;
    int st = 0;
    unsigned full_parity = 0;
    const double *a0 = As + warp_m * WM + (lane >> 2) + (lane & 3) * LDA;
    // Ragged tiles.  The fragment columns that intersect C are dealt out evenly over the
    // WARPS_N warps of a row, in compile-time widths of 2, 4, 6 or 8 fragments: the pp ladder's
    // last tile (89 of 128 columns = 12 fragments) runs 6 + 6 instead of 8 + 4(+4 wasted), so
    // the two warps that share a scheduler finish together and the CTA takes 6/8 of a full one.
    // (Per-fragment predication was measured to cost more than the padding it skips:
    // C[40000,N] = A.B took 75.7 ms at N = 729 against 72.6 ms at N = 768, tools/micro_edge.py.)
    // Fragments that are computed but lie outside C read offset-0 operand data and are never
    // stored.  Rows are not subdivided: a warp row is active or not.
    static_assert(NTL == 8, "column widths 2/4/6/8");
    const int nfrag = max(0, min(WARPS_N * NTL, (nrem + 7) >> 3));
    const int ncw = min(NTL, (((nfrag + WARPS_N - 1) / WARPS_N) + 1) & ~1);    // per warp, even
    const int wn_off = warp_n * ncw * 8;
    const int mact = max(0, min(MT, (mrem - warp_m * WM + 7) >> 3));
    const int wmode = (mact == 0 || nfrag - warp_n * ncw <= 0) ? 0 : ncw;
    const double *b0 = Bs + wn_off + (lane >> 2) + (lane & 3) * LDB;
    auto substep = [&](const double *a, const double *b, auto part, auto ncols) {
        constexpr int ks = decltype(part)::value;
        constexpr int NC_ = decltype(ncols)::value;
        double af[MT], bf[NC_];
#pragma unroll
        for (int i = 0; i < MT; ++i) af[i] = a[ks * 4 * LDA + i * 8];
#pragma unroll
        for (int j = 0; j < NC_; ++j) bf[j] = b[ks * 4 * LDB + j * 8];
#pragma unroll
        for (int i = 0; i < MT; ++i)
#pragma unroll
            for (int j = 0; j < NC_; ++j) dmma(acc[i][j], af[i], bf[j]);
    };
    unsigned ready = 0;
    for (int g = kt_lo; g < kt_hi; ++g) {
        if (g >= term_end) {
            cur_term = term_of(g);
            const double ratio = alpha / p.t[cur_term].alpha;
            alpha = p.t[cur_term].alpha;
            term_end = p.t[cur_term].kt_begin + p.t[cur_term].nkt;
            if (ratio != 1.0) {
#pragma unroll
                for (int i = 0; i < MT; ++i)
#pragma unroll
                    for (int j = 0; j < NTL; ++j) {
                        acc[i][j][0] *= ratio;
                        acc[i][j][1] *= ratio;
                    }
            }
        }
        if (!ready) mbar_wait(bar_base + st * 8, full_parity);
        asm volatile("" ::: "memory");
        const double *a = a0 + st * BK * LDA;
        const double *b = b0 + st * BK * LDB;
        // The barrier of the next stage is probed while the last sub-step still has DMMAs to
        // issue, so the round trip of the try_wait is hidden; a failed probe falls back to the
        // spinning wait at the top of the next iteration.
        const int nst = st + 1 == STAGES ? 0 : st + 1;
        const unsigned npar = nst == 0 ? full_parity ^ 1u : full_parity;
        auto ktile = [&](auto ncols) {
            substep(a, b, IntC<0>{}, ncols);
            substep(a, b, IntC<1>{}, ncols);
            substep(a, b, IntC<2>{}, ncols);
            ready = mbar_probe(bar_base + nst * 8, npar);
            substep(a, b, IntC<3>{}, ncols);
        };
        if (wmode == 8)
            ktile(IntC<8>{});
        else if (wmode == 6)
            ktile(IntC<6>{});
        else if (wmode == 4)
            ktile(IntC<4>{});
        else if (wmode == 2)
            ktile(IntC<2>{});
        else
            ready = mbar_probe(bar_base + nst * 8, npar);
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_base + (STAGES + st) * 8);
        if (++st == STAGES) {
            st = 0;
            full_parity ^= 1;
        }
    }
    if (alpha != 1.0) {
#pragma unroll
        for (int i = 0; i < MT; ++i)
#pragma unroll
            for (int j = 0; j < NTL; ++j) {
                acc[i][j][0] *= alpha;
                acc[i][j][1] *= alpha;
            }
    }

    // ---- epilogue (consumers only) ----
    const int row0 = warp_m * WM + (lane >> 2), col0 = wn_off + (lane & 3) * 2;
    if (wmode == 0) return;
    if (p.nsplit > 1)
        store_partial<MT, NTL>(p, acc, m0, n0, row0, col0, mrem, nrem, ncw);
    else
        store_tile<MT, NTL>(p, acc, s_cm, s_cn, row0, col0, mrem, nrem, ncw);
}

// C[m,n] = beta*C[m,n] + sum_s ws[s][m][n]  (split-K second stage, fixed order)
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const __grid_constant__ Params p) {
    const size_t MN = (size_t)p.M * (size_t)p.N;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < MN;
         idx += (size_t)gridDim.x * blockDim.x) {
        const int m = (int)(idx / (size_t)p.N), n = (int)(idx - (size_t)m * p.N);
        double s = 0.0;
        for (int k = 0; k < p.nsplit; ++k) s += p.ws[(size_t)k * MN + idx];
        double *dst = p.C + decomp(m, p.nm, p.m_ext, p.c_mstr) + decomp(n, p.nn, p.n_ext, p.c_nstr);
        if (p.beta != 0.0) s += p.beta * (*dst);
        *dst = s;
    }
}

// Second stage of a tail launch: C tile = beta*C + sum_s ws[s][tile][.][.], fixed order.  One CTA
// per tail tile, threads walk the tile row-major (n fastest, like the partial sums were stored).
__global__ void __launch_bounds__(256) tail_reduce_kernel(const __grid_constant__ Params p) {
    constexpr int BT = 128;
    const int tile = (int)blockIdx.x + p.tile_base;
    int tile_m, tile_n;
    tile_coords(p, tile, tile_m, tile_n);
    const int m0 = tile_m * BT, n0 = tile_n * BT;
    const int mrem = min(BT, p.M - m0), nrem = min(BT, p.N - n0);
    const size_t stride = (size_t)gridDim.x * BT * BT;
    const double *src = p.ws + (size_t)blockIdx.x * BT * BT;
    for (int e = threadIdx.x; e < BT * BT; e += blockDim.x) {
        const int ml = e / BT, nl = e - ml * BT;
        if (ml >= mrem || nl >= nrem) continue;
        double s = 0.0;
        for (int k = 0; k < p.nsplit; ++k) s += src[(size_t)k * stride + e];
        double *dst = p.C + decomp(m0 + ml, p.nm, p.m_ext, p.c_mstr) + decomp(n0 + nl, p.nn, p.n_ext, p.c_nstr);
        if (p.beta != 0.0) s += p.beta * (*dst);
        *dst = s;
    }
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
struct TileCfg {
    int bm, bn, threads;
    double eff;
};
static const TileCfg kCfg[] = {
    // eff = measured pp-ladder rate relative to the best config (profiles/r1_tile_sweep.md)
    {128, 128, 256, 1.00}, {128, 64, 256, 0.90}, {64, 64, 128, 1.00}, {64, 32, 128, 0.80},
    {128, 64, 128, 0.90},
    // warp-specialised kernels (384 threads: 8 consumer + 4 producer warps, one CTA per SM)
    {128, 128, 384, 1.30}, {128, 128, 384, 1.00}};
constexpr int kNumCfg = 7;

static int g_no_vec2 = 0;          // tuning bit 128: 8-byte copies even where 16-byte ones are possible
static int g_no_tail = 0;          // tuning bit 64: never cut the tail wave off (see tail_plan)
static int g_gen_no_walk = 0;      // tuning bit 16: generated operands use the scanning producer
static int g_gen_no_mraster = 0;   // tuning bit 32: keep the default tile order for generated operands
static int g_no_band_raster = 0;   // tuning bit 256: n-fastest tile order for stored operands (see tile_coords)
constexpr int kRasterBand = 12;    // 12 x 12.3 tiles per wave of 148 CTAs
static int g_force_cfg = -1;
static int g_force_split = 0;
// L2 budget for one operand's k window (0 = no windows).  The warp-specialised kernel runs
// without windows: its producers prefetch four k-tiles deep, DRAM is at 6 % utilisation even
// with the smaller operand re-read per row tile (profiles/pp_ladder_ws_v200_ncu.md), and a
// window costs a read-modify-write of C (measured: ring terms 33.0 vs 30.4 TFLOP/s).
constexpr long long kPanelDefault = 40LL << 20, kPanelDefaultWs = 0;
static long long g_panel_bytes = kPanelDefault, g_panel_bytes_ws = kPanelDefaultWs;

template <int BM, int BN, int STAGES, int NT>
constexpr size_t smem_bytes(int nterms) {
    return sizeof(double) * STAGES * BK * (BM + SPAD + BN + SPAD) +
           sizeof(long long) * ((size_t)nterms * (BM + BN) + 2 * (NT / (2 * BK)) * 2 * BK);
}

template <int BM, int BN, int WMW, int WNW, int STAGES, int MINB, bool IL>
static int launch_one(const Params &p, dim3 grid, cudaStream_t s) {
    auto kern = contract_kernel<BM, BN, WMW, WNW, STAGES, MINB, IL>;
    const size_t sm = smem_bytes<BM, BN, STAGES, WMW * WNW * 32>(p.nterms);
    static bool attr_done = false;
    if (!attr_done) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)smem_bytes<BM, BN, STAGES, WMW * WNW * 32>(PMB_MAX_TERMS));
        if (e != cudaSuccess) return (int)e;
        attr_done = true;
    }
    kern<<<grid, WMW * WNW * 32, sm, s>>>(p);
    count_launch();
    return cuda_status();
}

template <int BM, int BN, int STAGES>
constexpr size_t ws_smem_bytes(int nterms) {
    return 128 + sizeof(double) * STAGES * BK * (BM + SPAD + BN + SPAD) +
           sizeof(long long) * ((size_t)kWsKRing * 2 * BK + (size_t)(nterms + 1) * (BM + BN));
}

constexpr size_t kMaxSmemOptin = 232448;   // 227 KB per CTA on sm_100

// The pair tables of a generated operand are a few MB that every CTA keeps hitting at random
// (W0s[q,s*] once per non-zero element) while GB-sized operands stream through L2 and push them
// out: without help each hit is a DRAM round trip on the producers' critical path.  The launch
// therefore carries an access-policy window that keeps the tables in the persisting part of L2.
// PMB_GEN_L2_PERSIST=0 disables it (A/B measurements).
static bool gen_l2_window(const Params &p, cudaStream_t s, bool on) {
    static int enabled = -1;
    static size_t max_window = 0;
    if (enabled < 0) {
        const char *e = getenv("PMB_GEN_L2_PERSIST");
        enabled = !(e && e[0] == '0');
        int dev = 0, max_persist = 0, max_win = 0;
        if (cudaGetDevice(&dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&max_win, cudaDevAttrMaxAccessPolicyWindowSize, dev) != cudaSuccess ||
            max_persist <= 0 || max_win <= 0)
            enabled = 0;
        if (enabled) {
            size_t want = 32u << 20;
            if (want > (size_t)max_persist) want = (size_t)max_persist;
            if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want) != cudaSuccess) enabled = 0;
            max_window = want < (size_t)max_win ? want : (size_t)max_win;
        }
        cudaGetLastError();
    }
    if (!enabled) return false;
    cudaStreamAttrValue attr;
    memset(&attr, 0, sizeof(attr));
    if (on) {
        const size_t tab = sizeof(double) * (size_t)p.gen_ueg.n_orb * (size_t)p.gen_ueg.n_orb;
        const char *lo = nullptr, *hi = nullptr;
        const double *tabs[3] = {p.gen_W0a, p.gen_W1a, p.gen_W0s};
        for (const double *t : tabs) {
            if (!t) continue;
            const char *b = (const char *)t;
            if (!lo || b < lo) lo = b;
            if (!hi || b + tab > hi) hi = b + tab;
        }
        // one window: all tables when they were allocated side by side, else the randomly
        // accessed one (W0s; W0a / W1a are read at CTA-uniform, slowly advancing addresses)
        if (!lo || (size_t)(hi - lo) > max_window) {
            lo = (const char *)(p.gen_W0s ? p.gen_W0s : p.gen_W0a);
            hi = lo + tab;
            if (tab > max_window) return false;
        }
        attr.accessPolicyWindow.base_ptr = const_cast<char *>(lo);
        attr.accessPolicyWindow.num_bytes = (size_t)(hi - lo);
        attr.accessPolicyWindow.hitRatio = 1.0f;
        attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    }
    const bool ok = cudaStreamSetAttribute(s, cudaStreamAttributeAccessPolicyWindow, &attr) == cudaSuccess;
    cudaGetLastError();
    return ok;
}

template <int BM, int BN, int WMW, int WNW, int STAGES>
static int launch_ws(Params &p, dim3 grid, cudaStream_t s) {
    auto kern = contract_ws_kernel<BM, BN, WMW, WNW, STAGES>;
    static bool attr_done = false;
    if (!attr_done) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)kMaxSmemOptin);
        if (e != cudaSuccess) return (int)e;
        attr_done = true;
    }
    size_t smem = ws_smem_bytes<BM, BN, STAGES>(p.nterms);
    p.gen_map_smem = 0;
    const size_t gen_extra = sizeof(double) * 3 * (size_t)p.gen_ueg.n_orb +
                             sizeof(int) * ((size_t)p.gen_n3 + 1 + (size_t)p.gen_ueg.n_orb);
    if (p.gen_term >= 0 && smem + gen_extra <= kMaxSmemOptin) {
        // generated operand: the plane-wave vectors (12 KB at 515 orbitals) and the index map
        // (8.8 KB at imax = 6) ride in shared memory
        p.gen_map_smem = 1;
        smem += gen_extra;
    }
    if (p.gen_term >= 0) {
        const TermDev &t = p.t[p.gen_term];
        p.gen_walk = t.nk == 2 && p.gen_k_axis[0] == 3 && p.gen_k_axis[1] == 2 && !g_gen_no_walk;
    }
    // (with compressed values the pair tables are not read by the kernel at all)
    const bool window = p.gen_term >= 0 && !p.gen_nz && gen_l2_window(p, s, true);
    kern<<<grid, WMW * WNW * 32 + kWsProducerThreads, smem, s>>>(p);
    count_launch();
    const int rc = cuda_status();
    if (window) gen_l2_window(p, s, false);      // the launch has captured the attribute
    return rc;
}

template <int BM, int BN, int WMW, int WNW, int STAGES, int MINB>
static int launch_cfg(const Params &p, dim3 grid, cudaStream_t s, bool interleave) {
    return interleave ? launch_one<BM, BN, WMW, WNW, STAGES, MINB, true>(p, grid, s)
                      : launch_one<BM, BN, WMW, WNW, STAGES, MINB, false>(p, grid, s);
}

static bool prod_fits(const int64_t *ext, int n, int64_t *out) {
    int64_t v = 1;
    for (int i = 0; i < n; ++i) {
        if (ext[i] <= 0) return false;
        v *= ext[i];
        if (v >= (1LL << 31)) return false;
    }
    *out = v;
    return true;
}

// Split-K factor for `tiles` output tiles on `slots` co-resident CTA slots: skinny outputs
// with a long k (I_klij, Fock-like terms, o.v^3 blocks against T1) get enough CTAs to fill the
// machine; outputs that already fill it are never split (the workspace would be output-sized).
static int split_for(int64_t tiles, int64_t slots, int kt) {
    if (tiles >= slots || kt < 8) return 1;
    int64_t n = slots / tiles;
    if (n > kt / 4) n = kt / 4;
    if (n > 192) n = 192;
    return n < 1 ? 1 : (int)n;
}

// Tile configuration by a cost model: time ~ waves x (CTAs sharing an SM) x tile area / (rate
// of the configuration x split-K factor), i.e. padded work over the part of the machine the
// launch can actually fill.
static int choose_cfg(int64_t M, int64_t N, int kt, int *nsplit) {
    int best = 0;
    double best_cost = 1e300;
    for (int c = 0; c < kNumCfg; ++c) {
        if (g_force_cfg >= 0 && (g_force_cfg & 7) < kNumCfg && c != (g_force_cfg & 7)) continue;
        const int64_t tiles = ((M + kCfg[c].bm - 1) / kCfg[c].bm) * ((N + kCfg[c].bn - 1) / kCfg[c].bn);
        const int per_sm = (kCfg[c].threads == 128) ? 3 : 1;   // co-resident CTAs
        const int64_t slots = (int64_t)kSmCount * per_sm;
        const int split = split_for(tiles, slots, kt);
        double waves = (double)((tiles * split + slots - 1) / slots);
        if (c >= 5 && split == 1 && !g_no_tail && kt >= 64) {
            // the warp-specialised kernel cuts a sparse last wave off and splits it over k
            // (tail_plan): it then costs 1 / floor(148 / rest) of a wave
            const int64_t rest = tiles % slots;
            if (tiles > slots && rest > 0 && rest <= slots / 2) {
                int64_t ts = slots / rest;
                if (ts > kt / 16) ts = kt / 16;
                if (ts >= 2) waves = (double)(tiles / slots) + 1.0 / (double)ts;
            }
        }
        const double cost = waves * per_sm * kCfg[c].bm * kCfg[c].bn / (kCfg[c].eff * split);
        if (cost < best_cost * 0.999) {
            best_cost = cost;
            best = c;
            *nsplit = split;
        }
    }
    return best;
}

static int build_params(const pmb_contract_t *d, Params &p, int &cfg) {
    if (!d || d->nterms < 1 || d->nterms > PMB_MAX_TERMS) return PMB_E_BADARG;
    if (d->nm < 0 || d->nm > PMB_MAX_DIMS || d->nn < 0 || d->nn > PMB_MAX_DIMS) return PMB_E_BADARG;
    if (!d->C) return PMB_E_BADARG;
    int64_t M, N;
    if (!prod_fits(d->m_ext, d->nm, &M) || !prod_fits(d->n_ext, d->nn, &N)) return PMB_E_BADARG;
    p.nm = d->nm;
    p.nn = d->nn;
    p.nterms = d->nterms;
    p.M = (int)M;
    p.N = (int)N;
    for (int i = 0; i < PMB_MAX_DIMS; ++i) {
        p.m_ext[i] = i < d->nm ? (int)d->m_ext[i] : 1;
        p.n_ext[i] = i < d->nn ? (int)d->n_ext[i] : 1;
        p.c_mstr[i] = i < d->nm ? d->c_mstr[i] : 0;
        p.c_nstr[i] = i < d->nn ? d->c_nstr[i] : 0;
    }
    p.C = d->C;
    p.beta = d->beta;
    int kt = 0;
    int nkeep = 0;
    p.gen_term = -1;
    p.gen_n3 = p.gen_l0 = p.gen_map_smem = p.gen_walk = 0;
    memset(&p.gen_ueg, 0, sizeof(p.gen_ueg));
    p.gen_W0a = p.gen_W1a = p.gen_W0s = nullptr;
    p.gen_lin = nullptr;
    p.gen_nz = nullptr;
    for (int ti = 0; ti < d->nterms; ++ti) {
        const pmb_term_t &s = d->terms[ti];
        if ((!s.A && !s.a_gen) || !s.B || s.nk < 0 || s.nk > PMB_MAX_DIMS) return PMB_E_BADARG;
        // a zero coefficient contributes nothing; keep one such term only if nothing else is left
        if (s.alpha == 0.0 && !(ti == d->nterms - 1 && nkeep == 0)) continue;
        TermDev &t = p.t[nkeep++];
        int64_t K;
        if (!prod_fits(s.k_ext, s.nk, &K)) return PMB_E_BADARG;
        t.A = s.A;
        t.B = s.B;
        t.nk = s.nk;
        t.K = (int)K;
        for (int i = 0; i < PMB_MAX_DIMS; ++i) {
            t.k_ext[i] = i < s.nk ? (int)s.k_ext[i] : 1;
            t.a_kstr[i] = i < s.nk ? s.a_kstr[i] : 0;
            t.b_kstr[i] = i < s.nk ? s.b_kstr[i] : 0;
            t.a_mstr[i] = i < d->nm ? s.a_mstr[i] : 0;
            t.b_nstr[i] = i < d->nn ? s.b_nstr[i] : 0;
        }
        t.alpha = s.alpha;
        if (s.a_gen) {
            // generated A operand: validate the axis assignment and the packing limits
            const pmb_ueg_operand_t &g = *s.a_gen;
            if (p.gen_term >= 0) return PMB_E_UNSUPPORTED;         // one per contraction
            if (!g.W0a && !g.W0s && !g.nz) return PMB_E_BADARG;
            if (!g.lin || !g.ueg.index_map || !g.ueg.kp || g.ueg.n_orb <= 0) return PMB_E_BADARG;
            if (g.ueg.n_orb > kGenFieldMask || g.ueg.imax < 0 || g.ueg.imax > 27) return PMB_E_UNSUPPORTED;
            int seen = 0;
            for (int i = 0; i < d->nm; ++i) {
                const int ax = g.m_axis[i];
                if (ax < 0 || ax > 3 || (seen >> ax & 1)) return PMB_E_BADARG;
                if (g.lo[ax] < 0 || g.lo[ax] + d->m_ext[i] > g.ueg.n_orb) return PMB_E_BADARG;
                seen |= 1 << ax;
                p.gen_m_axis[i] = ax;
            }
            for (int i = 0; i < s.nk; ++i) {
                const int ax = g.k_axis[i];
                if (ax < 0 || ax > 3 || (seen >> ax & 1)) return PMB_E_BADARG;
                if (g.lo[ax] < 0 || g.lo[ax] + s.k_ext[i] > g.ueg.n_orb) return PMB_E_BADARG;
                seen |= 1 << ax;
                p.gen_k_axis[i] = ax;
            }
            if (seen != 15) return PMB_E_BADARG;
            const int n = 2 * g.ueg.imax + 1;
            p.gen_term = nkeep - 1;
            p.gen_n3 = n * n * n;
            p.gen_l0 = g.ueg.imax * (n * n + n + 1);
            for (int i = 0; i < 4; ++i) p.gen_lo[i] = g.lo[i];
            for (int i = 0; i < d->nm; ++i) p.gen_ext[g.m_axis[i]] = (int)d->m_ext[i];
            for (int i = 0; i < s.nk; ++i) p.gen_ext[g.k_axis[i]] = (int)s.k_ext[i];
            p.gen_nz = g.nz;
            p.gen_ueg = g.ueg;
            p.gen_W0a = g.W0a;
            p.gen_W1a = g.W1a;
            p.gen_W0s = g.W0s;
            p.gen_lin = g.lin;
        }
        // follow the unit-stride direction of each operand
        auto kfast = [](int nk, const int64_t *kstr, const int64_t *kext, int nx, const int64_t *xstr) {
            if (nk == 0) return 0;
            const int64_t ks = kstr[0] < 0 ? -kstr[0] : kstr[0];
            if (nx == 0) return 1;
            const int64_t xs = xstr[0] < 0 ? -xstr[0] : xstr[0];
            if (ks == 1 && kext[0] > 1) return (xs == 1) ? 0 : 1;
            return ks < xs ? 1 : 0;
        };
        t.a_kfast = kfast(s.nk, s.a_kstr, s.k_ext, d->nm, s.a_mstr);
        t.b_kfast = kfast(s.nk, s.b_kstr, s.k_ext, d->nn, s.b_nstr);
        // 16-byte copies of B: N group dense in memory, even k strides, aligned base, and at least
        // one contracted index (the tile loop then runs over real k offsets)
        t.b_vec2 = 0;
        if (!g_no_vec2 && d->nn >= 1 && s.nk >= 1 && !t.b_kfast && ((uintptr_t)s.B & 15) == 0) {
            bool ok = true;
            int64_t dense = 1;
            for (int i = 0; i < d->nn && ok; ++i) {
                ok = s.b_nstr[i] == dense;
                dense *= d->n_ext[i];
            }
            for (int i = 0; i < s.nk && ok; ++i) ok = (s.b_kstr[i] % 2) == 0;
            t.b_vec2 = ok ? 1 : 0;
        }
        t.kt_begin = kt;
        t.nkt = (t.K + BK - 1) / BK;
        kt += t.nkt;
    }
    p.nterms = nkeep;
    p.total_ktiles = kt;
    int nsplit = 1;
    cfg = choose_cfg(M, N, kt, &nsplit);
    // only the warp-specialised kernel has producer warps that can evaluate an operand
    if (p.gen_term >= 0 && cfg < 5) {
        cfg = 5;
        nsplit = split_for((int64_t)((M + 127) / 128) * ((N + 127) / 128), kSmCount, kt);
    }
    p.tiles_m = (int)((M + kCfg[cfg].bm - 1) / kCfg[cfg].bm);
    p.tiles_n = (int)((N + kCfg[cfg].bn - 1) / kCfg[cfg].bn);
    p.raster_m_fast = p.gen_term >= 0 && !g_gen_no_mraster;
    p.raster_group = (cfg >= 5 && p.gen_term < 0 && !g_no_band_raster && p.tiles_m > kRasterBand &&
                      p.tiles_n > kRasterBand) ? kRasterBand : 0;
    if (g_force_split > 0) nsplit = g_force_split;
    if (nsplit > kt) nsplit = kt;
    if (nsplit < 1) nsplit = 1;
    p.ktiles_per_split = (kt + nsplit - 1) / nsplit;
    p.nsplit = (kt + p.ktiles_per_split - 1) / p.ktiles_per_split;
    p.kt_base = 0;
    p.kt_limit = kt;
    p.tile_base = 0;
    p.tail = 0;
    p.ws = nullptr;
    return 0;
}

// K-panels.  Every CTA streams (BM + BN) x K operand elements; CTAs of one wave share them
// only through L2, and only while they work on the same k range.  When neither operand fits
// in L2 (pp ladder at v >= 250: T2 is 0.6-1.4 GB) CTAs drift apart and the small operand is
// re-read from HBM once per row tile (ncu, profiles/: 1.31 TB for 79 GB algorithmic).  The
// contraction is therefore issued as a sequence of launches over k windows whose slice of the
// smaller operand stays L2-resident; partial sums accumulate in C (beta = 1 after the first
// window, fixed order, deterministic).
static int panel_ktiles(const Params &p, int cfg) {
    const long long g_panel_bytes = cfg >= 5 ? g_panel_bytes_ws : pmb::g_panel_bytes;
    if (p.nsplit > 1 || g_panel_bytes <= 0) return p.total_ktiles;
    const double small_rows = (double)(p.M < p.N ? p.M : p.N);
    const double small_bytes = small_rows * (double)p.total_ktiles * BK * 8.0;
    if (small_bytes <= (double)g_panel_bytes) return p.total_ktiles;
    long long kt = (long long)((double)g_panel_bytes / (small_rows * BK * 8.0));
    if (kt < 64) kt = 64;
    const int npanel = (int)((p.total_ktiles + kt - 1) / kt);
    return (p.total_ktiles + npanel - 1) / npanel;      // equal windows
}

// Tail wave.  The warp-specialised kernel runs one CTA per SM, so a grid of `tiles` CTAs takes
// ceil(tiles / 148) waves and the last one may be nearly empty (ring terms of an 8-way sharded
// 515-orbital sweep: 1339 tiles = 9.05 waves; the pair of o.v^3.tau contractions: 4.18 waves each).
// When the last wave would fill at most half of the machine, the launch is cut in two: the full
// waves as they are, and the R remaining tiles as a second launch split floor(148 / R) ways over k
// (partial sums to the workspace, fixed-order second stage) -- the tail then costs 1/split of a
// wave.  Only for long k loops (a wave >= ~130 us), without k windows.
struct TailPlan {
    int full_tiles, tail_tiles, split;
};
static TailPlan tail_plan(const Params &p, int cfg) {
    TailPlan t = {0, 0, 1};
    if (cfg < 5 || g_no_tail || p.nsplit != 1 || panel_ktiles(p, cfg) < p.total_ktiles) return t;
    const int tiles = p.tiles_m * p.tiles_n;
    const int full = (tiles / kSmCount) * kSmCount, rest = tiles - full;
    if (full == 0 || rest == 0 || rest > kSmCount / 2 || p.total_ktiles < 64) return t;
    int split = kSmCount / rest;
    if (split > p.total_ktiles / 16) split = p.total_ktiles / 16;
    if (split < 2) return t;
    t.full_tiles = full;
    t.tail_tiles = rest;
    t.split = split;
    return t;
}

}  // namespace pmb

using namespace pmb;

extern "C" void pmb_contract_set_tuning(int tile_config, int split_k) {
    g_gen_no_walk = tile_config >= 0 && (tile_config & 16);
    g_gen_no_mraster = tile_config >= 0 && (tile_config & 32);
    g_no_tail = tile_config >= 0 && (tile_config & 64);
    g_no_vec2 = tile_config >= 0 && (tile_config & 128);
    g_no_band_raster = tile_config >= 0 && (tile_config & 256);
    g_force_cfg = tile_config >= 0 ? (tile_config & 15) : tile_config;
    g_force_split = split_k;
}

extern "C" void pmb_contract_set_panel_bytes(long long bytes) {
    g_panel_bytes = bytes < 0 ? kPanelDefault : bytes;
    g_panel_bytes_ws = bytes < 0 ? kPanelDefaultWs : bytes;
}

namespace pmb {

// Coefficient runs.  The kernels keep their accumulators in units of the current term's alpha and
// rescale them by alpha_old / alpha_new at a term boundary, which overflows or underflows when the
// coefficients are far apart (alphas 2^600 and 2^-600: the ratio is inf).  The terms are therefore
// issued in runs of consecutive terms whose non-zero finite |alpha| lie within a factor 2^kCoefSpread
// of each other -- one launch sequence per run, the caller's beta on the first, beta = 1 after it.
// Ordinary coefficients form one run: one launch sequence, as before.
constexpr int kCoefSpread = 64;

// split the terms of `d` into runs: run r is terms [first[r], first[r + 1]); returns the count
static int coef_runs(const pmb_contract_t *d, int *first) {
    int nrun = 1, lo = 0, hi = 0;
    bool open = false;
    first[0] = 0;
    for (int ti = 0; ti < d->nterms; ++ti) {
        const double a = d->terms[ti].alpha;
        if (a == 0.0 || !std::isfinite(a)) continue;      // dropped, or fits any run
        const int e = std::ilogb(a);
        if (!open) {
            lo = hi = e;
            open = true;
        } else if ((e > hi ? e : hi) - (e < lo ? e : lo) > kCoefSpread) {
            first[nrun++] = ti;
            lo = hi = e;
        } else {
            lo = e < lo ? e : lo;
            hi = e > hi ? e : hi;
        }
    }
    first[nrun] = d->nterms;
    return nrun;
}

// descriptor of run r: its terms, beta = 1 after the first run
static pmb_contract_t run_descriptor(const pmb_contract_t *d, const int *first, int r) {
    pmb_contract_t q = *d;
    q.nterms = first[r + 1] - first[r];
    for (int i = 0; i < q.nterms; ++i) q.terms[i] = d->terms[first[r] + i];
    if (r > 0) q.beta = 1.0;
    return q;
}

static size_t workspace_one(const pmb_contract_t *d) {
    Params p;
    int cfg;
    if (build_params(d, p, cfg) != 0) return 0;
    if (p.nsplit <= 1) {
        const TailPlan t = tail_plan(p, cfg);
        return sizeof(double) * (size_t)t.tail_tiles * (size_t)t.split * 128 * 128;
    }
    return sizeof(double) * (size_t)p.nsplit * (size_t)p.M * (size_t)p.N;
}

static int contract_one(const pmb_contract_t *d, void *ws, size_t ws_bytes, cudaStream_t s);

}  // namespace pmb

extern "C" size_t pmb_contract_workspace(const pmb_contract_t *d) {
    if (!d || d->nterms < 1 || d->nterms > PMB_MAX_TERMS) return 0;
    int first[PMB_MAX_TERMS + 1];
    const int nrun = coef_runs(d, first);
    if (nrun == 1) return workspace_one(d);
    Params p;
    int cfg;
    if (build_params(d, p, cfg) != 0) return 0;
    size_t need = 0;
    for (int r = 0; r < nrun; ++r) {
        const pmb_contract_t q = run_descriptor(d, first, r);
        const size_t w = workspace_one(&q);
        need = w > need ? w : need;
    }
    return need;
}

extern "C" int pmb_contract(const pmb_contract_t *d, void *ws, size_t ws_bytes, pmb_stream_t stream) {
    if (!d || d->nterms < 1 || d->nterms > PMB_MAX_TERMS) return PMB_E_BADARG;
    int first[PMB_MAX_TERMS + 1];
    const int nrun = coef_runs(d, first);
    if (nrun == 1) return contract_one(d, ws, ws_bytes, (cudaStream_t)stream);
    Params p;
    int cfg;
    const int rc = build_params(d, p, cfg);     // every argument error before anything launches
    if (rc != 0) return rc;
    const size_t need = pmb_contract_workspace(d);
    if (need && (!ws || ws_bytes < need)) return PMB_E_WORKSPACE;
    for (int r = 0; r < nrun; ++r) {
        const pmb_contract_t q = run_descriptor(d, first, r);
        const int rr = contract_one(&q, ws, ws_bytes, (cudaStream_t)stream);
        if (rr != 0) return rr;
    }
    return 0;
}

int pmb::contract_one(const pmb_contract_t *d, void *ws, size_t ws_bytes, cudaStream_t s) {
    Params p;
    int cfg;
    int rc = build_params(d, p, cfg);
    if (rc != 0) return rc;
    if (p.nsplit > 1) {
        const size_t need = sizeof(double) * (size_t)p.nsplit * (size_t)p.M * (size_t)p.N;
        if (!ws || ws_bytes < need) return PMB_E_WORKSPACE;
        p.ws = (double *)ws;
    }
    const TailPlan tail = tail_plan(p, cfg);
    if (tail.split > 1) {
        const size_t need = sizeof(double) * (size_t)tail.tail_tiles * (size_t)tail.split * 128 * 128;
        if (!ws || ws_bytes < need) return PMB_E_WORKSPACE;
        // full waves, unsplit
        dim3 g1((unsigned)tail.full_tiles, 1, 1);
        rc = cfg == 5 ? launch_ws<128, 128, 4, 2, 4>(p, g1, s) : launch_ws<128, 128, 4, 2, 6>(p, g1, s);
        if (rc != 0) return rc;
        // the rest, split over k
        Params q = p;
        q.tile_base = tail.full_tiles;
        q.tail = 1;
        q.ws = (double *)ws;
        q.ktiles_per_split = (p.total_ktiles + tail.split - 1) / tail.split;
        q.nsplit = (p.total_ktiles + q.ktiles_per_split - 1) / q.ktiles_per_split;
        dim3 g2((unsigned)tail.tail_tiles, (unsigned)q.nsplit, 1);
        rc = cfg == 5 ? launch_ws<128, 128, 4, 2, 4>(q, g2, s) : launch_ws<128, 128, 4, 2, 6>(q, g2, s);
        if (rc != 0) return rc;
        tail_reduce_kernel<<<(unsigned)tail.tail_tiles, 256, 0, s>>>(q);
        count_launch();
        return cuda_status();
    }
    dim3 grid((unsigned)(p.tiles_m * p.tiles_n), (unsigned)p.nsplit, 1);
    // copies of the next tile interleaved with the DMMA sub-steps: pays off when one CTA
    // owns the SM (cfg 0), costs registers/occupancy otherwise.  Tuning bit 8 flips it.
    bool il = (cfg == 0);
    if (g_force_cfg >= 0 && (g_force_cfg & 8)) il = !il;
    const int window = panel_ktiles(p, cfg);
    for (int base = 0; base < p.total_ktiles && rc == 0; base += window) {
        if (window < p.total_ktiles) {
            p.kt_base = base;
            p.kt_limit = base + window < p.total_ktiles ? base + window : p.total_ktiles;
            p.ktiles_per_split = window;
            if (base > 0) p.beta = 1.0;
        }
        switch (cfg) {
            case 0: rc = launch_cfg<128, 128, 4, 2, 4, 1>(p, grid, s, il); break;
            case 1: rc = launch_cfg<128, 64, 4, 2, 4, 1>(p, grid, s, il); break;
            case 2: rc = launch_cfg<64, 64, 2, 2, 3, 3>(p, grid, s, il); break;
            case 4: rc = launch_cfg<128, 64, 2, 2, 3, 2>(p, grid, s, il); break;
            case 5: rc = launch_ws<128, 128, 4, 2, 4>(p, grid, s); break;
            case 6: rc = launch_ws<128, 128, 4, 2, 6>(p, grid, s); break;
            default: rc = launch_cfg<64, 32, 2, 2, 3, 3>(p, grid, s, il); break;
        }
    }
    if (rc != 0) return rc;
    if (p.nsplit > 1) {
        const size_t MN = (size_t)p.M * p.N;
        int blocks = (int)((MN + 255) / 256);
        if (blocks > 4 * kSmCount) blocks = 4 * kSmCount;
        splitk_reduce_kernel<<<blocks, 256, 0, s>>>(p);
        count_launch();
        rc = cuda_status();
    }
    return rc;
}
