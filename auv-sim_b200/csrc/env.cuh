// env.cuh -- the world model in HBM and its shared-memory staging.
//
// Layout in HBM (one blob per precision, built once by auvrrt_env_create):
//   EnvHeader | circles SoA (cx, cy, r, r_eff, r_eff^2) | polygon (px, py) | habitats SoA |
//   time bins (b0, b1) | cell index (breakpoints, piece offsets, candidates) | probs [T][C]
// Everything up to `hot_bytes` is copied into shared memory by ONE TMA bulk copy
// (cp.async.bulk.shared::cluster.global, completion on an mbarrier) at kernel start; the
// probability table follows it into shared memory too when it fits, else it is read from L2.
//
// Semantics preserved from the reference:
//  * r_eff[j] = max_{k >= j} r[k].  RRT.check_collision never resets dList between obstacles
//    (rrt_dubins.py:535-542), so it reports a collision iff  exists k: min_{j<=k} m_j <= r_k
//    <=> exists j: m_j <= max_{k>=j} r_k.  The running-minimum quirk is therefore EXACTLY an
//    inflation of circle j to the suffix maximum of the radii, in obstacle order.
//  * cell index: cost.py:181-184 scans the cell dict in order and takes the first cell with
//    x>=c0 and x<=c2 and y>=c1 and x<=c3 (sic).  The x-conditions say x in [c0, min(c2,c3)].
//    The breakpoints {c0, min(c2,c3)} cut the x axis into points and open intervals ("pieces") on
//    which the set of x-admissible cells is constant; within a piece, a cell can only be the
//    first match if its c1 is strictly below the c1 of every earlier admissible cell, so each
//    piece keeps that strictly decreasing candidate list.  First candidate with c1 <= y wins.
//    Lookup (find_cell): an x-bucket table (buckets no wider than 0.25 m) gives the last breakpoint left of the
//    bucket; a bucket holds at most one breakpoint (else it is flagged and the breakpoints are walked), so one
//    compare settles the piece; brk[NB] = +inf is a sentinel.  pfirst[piece] is the piece's first candidate.
#pragma once
#include "common.cuh"

namespace auv {

struct EnvHeader {
    int K, E, H, T, C, NB, NP, NCAND;
    int convex;        // +1: convex CCW, -1: convex CW, 0: general simple polygon
    int hot_bytes;     // bytes [0, hot_bytes) are staged in shared memory
    int total_bytes;
    int off_cx, off_cy, off_cr, off_creff, off_creff2;
    int off_px, off_py;
    int off_hx, off_hy, off_hr, off_hr2;
    int off_b0, off_b1;
    int off_brk, off_piece, off_c1, off_cell;
    int off_probs;
    int off_xb;        // x-bucket table for the shark-cell pieces (u16 per bucket, see find_cell), staged
    int nxb;           // number of x buckets (0: none)
    int off_pfirst;    // first candidate of every piece (PFirst<R> per piece), staged
    int off_grid;      // classification grid (3 planes of u32, one word per cell each), not staged: read through L1/L2
    int gnx, gny;      // grid dimensions (0: no grid)
    int bins_uniform;  // 1: bins are [s0 + i w, s0 + (i+1) w], contiguous and in order
    int off_one;       // single-candidate tables (One<R> rows, staged): K+1 circles, then max(E,1) boundary edges, then max(H,1) habitats
    int pad_;
    double bbox[4];    // minx, miny, maxx, maxy of the polygon (Polygon.bounds, rrt_dubins.py:334)
    double gx0, gy0, gs;   // grid origin and cell size
    double bin_s0, bin_w;
    double xb0, xbw;       // x-bucket origin and width
    double pad2_[2];
};
static_assert(sizeof(EnvHeader) % 16 == 0, "EnvHeader must keep 16-byte alignment of the arrays");

// Classification grid (built once on the host, see api.cu): three u32 words per cell of a uniform
// grid over the polygon's bounding box (stored as three planes: word 0 of every cell, then word 1, then word 2, so
// the one word most waypoints need is dense in L1), so that most waypoints are classified by ONE load instead
// of the loops over circles / polygon edges / habitats / shark cells, and the rest by a short
// per-cell candidate list.  A code is only definitive when every point of the cell (plus a rounding
// margin) gets the same answer from the exact test; candidate lists hold every object that can
// decide a point of the cell.  Results are therefore identical to the exact tests by construction.
//  word 0  bits 0-1   polygon: 0 ambiguous, 1 strictly inside, 2 outside
//          bit  2     1: clear of every (inflated) obstacle circle
//          bits 3-10  habitat: 0..63 first-match habitat (definitive); 64 + h: habitat h is the only one a point of
//                     the cell can be in and must be tested; 128 none; 192 ambiguous (candidates in word 2)
//                     (the low six bits always index a valid row of the habitat table)
//          bit  11    circles: more than 3 candidates -> full loop
//          bit  12    habitats: more than 3 candidates -> full loop
//          bit  13    polygon: convex fast path not applicable / more than 2 candidate edges -> full test
//          bit  14    circles: exactly ONE candidate, its index in bits 16-25; index K (a row with radius +inf) says
//                     "every point of the cell is inside some circle"
//          bit  15    polygon ambiguous with exactly ONE candidate edge (convex ring), its index in bits 26-30
//          bit  31    the collision test of this cell needs the general path (words 1 / 2 or the full loops); clear:
//                     bits 0-2 and the two single candidates decide it (point_unsafe_one, geom.cuh)
//  word 1  three 10-bit circle indices (0x3FF = none): the only circles a point of the cell can hit
//  word 2  bits 0-17 three 6-bit habitat indices (0x3F = none), in list order; bits 18-27 two 5-bit
//          polygon edge indices (0x1F = none): the only edges whose half-plane is not already decided
// The single-candidate forms keep the common boundary cells (one circle, one habitat or one polygon edge
// nearby) on a short branch-free path: in a kernel that runs one edge per thread a rare slow path taken by one
// lane stalls the other 31.
#define AUV_GRID_HAB_NONE 128u
#define AUV_GRID_HAB_AMBIG 192u
#define AUV_GRID_HAB_ONE 64u
#define AUV_GRID_CIRC_MANY (1u << 11)
#define AUV_GRID_HAB_MANY (1u << 12)
#define AUV_GRID_POLY_FULL (1u << 13)
#define AUV_GRID_CIRC_ONE (1u << 14)
#define AUV_GRID_POLY_ONE (1u << 15)
#define AUV_GRID_SLOW (1u << 31)
#define AUV_GRID_ALL_AMBIG ((AUV_GRID_HAB_AMBIG << 3) | AUV_GRID_CIRC_MANY | AUV_GRID_HAB_MANY | AUV_GRID_POLY_FULL | AUV_GRID_SLOW)

struct Cls { unsigned code; int idx; };   // word 0 and the cell index (-1 outside the grid)

// First candidate of a piece of the cell index (see the top of this file): v >= 0: cell id (bits 0-29), c1 its lower
// y bound, bit 30: more candidates follow in the piece's list; v == -1: the piece has no candidate.
template <typename R> struct alignas(8) PFirst { R c1; int v; };

// One row of the single-candidate tables, fetched with one 16-byte load (fp32):
//   circle   {cx, cy, r_eff^2, r_eff}      (row K: {0, 0, +inf, +inf})
//   edge i   {ax, ay, s (bx - ax), s (by - ay)}, s = +1 for a CCW ring, -1 for CW: strictly inside the half-plane <=> det > 0
//   habitat  {hx, hy, r^2, r}
template <typename R> struct alignas(16) One { R x, y, z, w; };

template <typename R> struct EnvView {
    int K, E, H, T, C, NB, NP, convex;
    int gnx, gny, ncell, bins_uniform, nxb;
    R gx0, gy0, ginv, gxo, gyo, bin_s0, bin_w, bin_winv, bin_off, bin_lo, bin_hi, xb0, xbinv, xbo;
    const unsigned *grid;
    const unsigned *grid0s;        // plane 0 of the grid in shared memory (kernels that stage it), else nullptr
    const PFirst<R> *pfirst;
    const One<R> *cone, *pone, *hone;
    // A copy of this view in shared memory, or nullptr.  Kernels that run one edge per thread publish one so that
    // the rare slow paths (boundary cells, ambiguous habitats, buckets with several breakpoints) can live OUT OF LINE,
    // taking just this pointer: the hot loop stays short and its registers free.
    const EnvView<R> *shared_self;
    const unsigned short *xb;
    R minx, miny, maxx, maxy;
    const R *cx, *cy, *cr, *creff, *creff2;
    const R *px, *py;
    const R *hx, *hy, *hr, *hr2;
    const R *b0, *b1;
    const R *brk;
    const int *piece;
    const R *c1;
    const int *cell;
    const R *probs;

    // every field but bin_lo / bin_hi (they are read from the bound arrays) from a header and the addresses of the staged
    // image and of the probability table; usable on the host
    __host__ __device__ __forceinline__ void bind_header(const EnvHeader &h, const unsigned char *hot, const unsigned char *probs_base) {
        K = h.K; E = h.E; H = h.H; T = h.T; C = h.C; NB = h.NB; NP = h.NP; convex = h.convex;
        shared_self = nullptr;
        minx = (R)h.bbox[0]; miny = (R)h.bbox[1]; maxx = (R)h.bbox[2]; maxy = (R)h.bbox[3];
        cx = (const R *)(hot + h.off_cx); cy = (const R *)(hot + h.off_cy);
        cr = (const R *)(hot + h.off_cr); creff = (const R *)(hot + h.off_creff);
        creff2 = (const R *)(hot + h.off_creff2);
        px = (const R *)(hot + h.off_px); py = (const R *)(hot + h.off_py);
        hx = (const R *)(hot + h.off_hx); hy = (const R *)(hot + h.off_hy);
        hr = (const R *)(hot + h.off_hr); hr2 = (const R *)(hot + h.off_hr2);
        b0 = (const R *)(hot + h.off_b0); b1 = (const R *)(hot + h.off_b1);
        brk = (const R *)(hot + h.off_brk); piece = (const int *)(hot + h.off_piece);
        c1 = (const R *)(hot + h.off_c1); cell = (const int *)(hot + h.off_cell);
        probs = (const R *)(probs_base + h.off_probs);
        pfirst = (const PFirst<R> *)(hot + h.off_pfirst);
        cone = (const One<R> *)(hot + h.off_one); pone = cone + (K + 1); hone = pone + (E > 0 ? E : 1);
    }
    __device__ __forceinline__ void bind(const unsigned char *hot, const unsigned char *probs_base) {
        bind_header(*(const EnvHeader *)hot, hot, probs_base);
        bin_lo = T > 0 ? b0[0] : (R)1; bin_hi = T > 0 ? b1[T - 1] : (R)0;      // [first b0, last b1]; empty when T == 0
    }
    // A view the host bound to the blob in HBM, moved to a copy of the staged image (probability table included) at
    // `to`.  The kernel receives the view as a parameter: its scalars and array offsets then come from the constant
    // bank instead of registers loaded from the staged header, and every array is `to` plus a uniform offset.
    __device__ __forceinline__ void move_staged(const unsigned char *from, const unsigned char *to) {
#define AUV_MOVE(p) p = (decltype(p))(to + ((const unsigned char *)(p) - from))
        AUV_MOVE(cx); AUV_MOVE(cy); AUV_MOVE(cr); AUV_MOVE(creff); AUV_MOVE(creff2); AUV_MOVE(px); AUV_MOVE(py);
        AUV_MOVE(hx); AUV_MOVE(hy); AUV_MOVE(hr); AUV_MOVE(hr2); AUV_MOVE(b0); AUV_MOVE(b1);
        AUV_MOVE(brk); AUV_MOVE(piece); AUV_MOVE(c1); AUV_MOVE(cell); AUV_MOVE(probs); AUV_MOVE(pfirst);
        AUV_MOVE(cone); AUV_MOVE(pone); AUV_MOVE(hone); AUV_MOVE(xb);
#undef AUV_MOVE
    }
    // Tell the compiler that the staged arrays live in shared memory (the pointers are computed from offsets read
    // at run time, so address-space inference cannot see it): loads become LDS with 32-bit addresses instead of
    // generic loads with 64-bit address arithmetic.  Only for kernels that ALWAYS stage the hot part.
    __device__ __forceinline__ void assume_hot_shared(bool probs_too) const {
        __builtin_assume(__isShared(cx)); __builtin_assume(__isShared(cy)); __builtin_assume(__isShared(cr));
        __builtin_assume(__isShared(creff)); __builtin_assume(__isShared(creff2));
        __builtin_assume(__isShared(px)); __builtin_assume(__isShared(py));
        __builtin_assume(__isShared(hx)); __builtin_assume(__isShared(hy)); __builtin_assume(__isShared(hr));
        __builtin_assume(__isShared(hr2)); __builtin_assume(__isShared(b0)); __builtin_assume(__isShared(b1));
        __builtin_assume(__isShared(brk)); __builtin_assume(__isShared(piece)); __builtin_assume(__isShared(c1));
        __builtin_assume(__isShared(cell)); __builtin_assume(__isShared(pfirst)); __builtin_assume(__isShared(xb));
        __builtin_assume(__isShared(cone)); __builtin_assume(__isShared(pone)); __builtin_assume(__isShared(hone));
        if (probs_too) __builtin_assume(__isShared(probs));
    }
    // the grid stays in global memory: bind it from the blob in HBM
    __host__ __device__ __forceinline__ void bind_grid_header(const EnvHeader &h, const unsigned char *blob_global, const unsigned char *hot) {
        gnx = h.gnx; gny = h.gny; bins_uniform = h.bins_uniform; nxb = h.nxb;
        xb0 = (R)h.xb0; xbinv = (R)(1.0 / h.xbw); xbo = (R)(-h.xb0 / h.xbw); xb = (const unsigned short *)(hot + h.off_xb);
        gx0 = (R)h.gx0; gy0 = (R)h.gy0; ginv = (R)(1.0 / h.gs);
        gxo = (R)(-h.gx0 / h.gs); gyo = (R)(-h.gy0 / h.gs);
        bin_s0 = (R)h.bin_s0; bin_w = (R)h.bin_w; bin_winv = (R)(1.0 / h.bin_w); bin_off = (R)(-h.bin_s0 / h.bin_w);
        grid = (const unsigned *)(blob_global + h.off_grid);
        grid0s = nullptr;
        ncell = gnx * gny;
    }
    __device__ __forceinline__ void bind_grid(const unsigned char *blob_global, const unsigned char *hot) {
        bind_grid_header(*(const EnvHeader *)hot, blob_global, hot);
    }
    // classification of the cell containing (x, y); off the grid: outside the polygon, everything else ambiguous
    // GRIDS: plane 0 is read from its shared-memory copy (grid0s)
    template <bool GRIDS = false>
    __device__ __forceinline__ Cls classify(R x, R y) const {
        Cls c;
        int ix, iy;
        if (sizeof(R) == 4) {
            // floor via round-toward-minus-infinity onto 2^23: two full-rate instructions per coordinate instead of
            // F2I on the conversion pipe; anything out of range (negative, huge, NaN) fails the unsigned compares
            const float fx = fmaf((float)x, (float)ginv, (float)gxo), fy = fmaf((float)y, (float)ginv, (float)gyo);
            ix = __float_as_int(__fadd_rd(fx, 8388608.f)) - 0x4B000000;
            iy = __float_as_int(__fadd_rd(fy, 8388608.f)) - 0x4B000000;
        } else {
            const R fx = (x - gx0) * ginv, fy = (y - gy0) * ginv;
            const bool in = fx >= (R)0 && fy >= (R)0 && fx < (R)gnx && fy < (R)gny;
            ix = in ? (int)fx : -1; iy = in ? (int)fy : -1;
        }
        if (!((unsigned)ix < (unsigned)gnx && (unsigned)iy < (unsigned)gny)) {
            // the grid covers the polygon's bounding box plus one cell all round: a point off the grid is outside the
            // polygon (code 2) whatever else is undecided about it
            // (code 2 settles the collision test: no SLOW flag; without a grid everything takes the general path)
            c.code = gnx > 0 ? (((AUV_GRID_HAB_AMBIG << 3) | AUV_GRID_HAB_MANY | AUV_GRID_CIRC_MANY | AUV_GRID_POLY_FULL) | 2u) : AUV_GRID_ALL_AMBIG;
            c.idx = -1; return c;
        }
        c.idx = iy * gnx + ix;
        c.code = GRIDS ? grid0s[c.idx] : __ldg(grid + c.idx);
        return c;
    }
    __device__ __forceinline__ unsigned word1(const Cls &c) const { return __ldg(grid + ncell + c.idx); }
    __device__ __forceinline__ unsigned word2(const Cls &c) const { return __ldg(grid + 2 * ncell + c.idx); }
};

// ---- TMA bulk staging -------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t phase) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(phase)
        : "memory");
}

// Stage `bytes` (multiple of 16) of the blob into shared memory.  One elected thread arms the
// mbarrier with the byte count and issues the bulk copies (<= 64 KiB each); everybody waits.
// Must be called by all threads of the CTA.
__device__ __forceinline__ void stage_env_tma(unsigned char *smem_dst, const unsigned char *blob,
                                              int bytes, uint64_t *bar) {
    if (threadIdx.x == 0) mbar_init(bar, 1);
    __syncthreads();
    if (threadIdx.x == 0) {
        mbar_expect_tx(bar, (uint32_t)bytes);
        for (int o = 0; o < bytes; o += 65536) {
            int n = bytes - o < 65536 ? bytes - o : 65536;
            tma_bulk_g2s(smem_dst + o, blob + o, (uint32_t)n, bar);
        }
    }
    mbar_wait(bar, 0);
}

// bytes of dynamic shared memory a kernel needs for the env given a budget
struct EnvStagePlan { int bytes; int probs_staged; };

}  // namespace auv
