// api.cu -- the C ABI (include/auvrrt.h): world-model flattening and host-buffer entry points.
// No CPU fallback anywhere: every compute entry runs the CUDA kernels or fails with AUVRRT_ERR_CUDA.
#include <algorithm>
#include <deque>
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <vector>
#include "launch.h"

using namespace auv;

extern "C" const char *auvrrt_last_error(void) { return g_err; }
extern "C" int auvrrt_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}
extern "C" int64_t auvrrt_launch_count(void) { return g_launches; }
extern "C" double auvrrt_stream_u(uint64_t seed, int64_t k, int f32) {
    uint64_t z = stream_bits(stream_key(seed), (uint32_t)k);
    return f32 ? (double)(z >> 41) * 0x1.0p-23 : (double)(z >> 11) * 0x1.0p-53;
}

int auv::need_device(int device) {
    int n = auvrrt_device_count();
    if (n <= 0) return set_err(AUVRRT_ERR_CUDA, "no CUDA device: libauvrrt has no CPU fallback");
    if (device < 0 || device >= n) return set_err(AUVRRT_ERR_ARG, "device %d out of range (%d devices)", device, n);
    AUV_CUDA(cudaSetDevice(device));
    return AUVRRT_OK;
}

// ------------------------------------------------------------------ env blob builder (host)
namespace {

template <typename R>
std::vector<unsigned char> build_blob(const double *circles, int K, const double *poly, int E, const double *hab,
                                      int H, const double *bins, int T, const double *cells, int C,
                                      const double *probs, EnvHeader *hout) {
    EnvHeader h;
    memset(&h, 0, sizeof(h));
    h.K = K; h.E = E; h.H = H; h.T = T; h.C = C;
    // --- cell index on R-rounded bounds (see env.cuh)
    std::vector<R> lo(C), hi(C), c1(C);
    std::vector<R> brk;
    for (int c = 0; c < C; c++) {
        R c0 = (R)cells[4 * c], cy1 = (R)cells[4 * c + 1], c2 = (R)cells[4 * c + 2], c3 = (R)cells[4 * c + 3];
        lo[c] = c0; hi[c] = std::min(c2, c3); c1[c] = cy1;
        if (hi[c] >= lo[c]) { brk.push_back(lo[c]); brk.push_back(hi[c]); }
    }
    std::sort(brk.begin(), brk.end());
    brk.erase(std::unique(brk.begin(), brk.end()), brk.end());
    const int NB = (int)brk.size(), NP = NB > 0 ? 2 * NB : 0;
    std::vector<int> piece(NP + 1, 0);
    std::vector<R> cand_c1;
    std::vector<int> cand_cell;
    for (int p = 0; p < NP; p++) {
        piece[p] = (int)cand_c1.size();
        const int i = p >> 1;
        const bool point = (p & 1) == 0;
        if (!point && i + 1 >= NB) continue;         // no interval after the last breakpoint
        bool have = false;
        R cur = 0;
        for (int c = 0; c < C; c++) {
            if (!(hi[c] >= lo[c])) continue;
            bool covers = point ? (lo[c] <= brk[i] && brk[i] <= hi[c]) : (lo[c] <= brk[i] && hi[c] >= brk[i + 1]);
            if (!covers) continue;
            if (!have || c1[c] < cur) { cand_c1.push_back(c1[c]); cand_cell.push_back(c); cur = c1[c]; have = true; }
        }
    }
    if (NP > 0) piece[NP] = (int)cand_c1.size();
    h.NB = NB; h.NP = NP; h.NCAND = (int)cand_c1.size();
    // --- polygon convexity / orientation (fast build uses half-plane tests when convex)
    h.convex = 0;
    if (E >= 3) {
        int pos = 0, neg = 0;
        for (int i = 0; i < E; i++) {
            const double *a = poly + 2 * i, *b = poly + 2 * ((i + 1) % E), *c = poly + 2 * ((i + 2) % E);
            double cr = (b[0] - a[0]) * (c[1] - b[1]) - (b[1] - a[1]) * (c[0] - b[0]);
            if (cr > 0) pos++; else if (cr < 0) neg++; else { pos++; neg++; }
        }
        if (neg == 0) h.convex = 1; else if (pos == 0) h.convex = -1;
    }
    h.bbox[0] = h.bbox[1] = INFINITY; h.bbox[2] = h.bbox[3] = -INFINITY;
    for (int i = 0; i < E; i++) {
        h.bbox[0] = std::min(h.bbox[0], poly[2 * i]); h.bbox[2] = std::max(h.bbox[2], poly[2 * i]);
        h.bbox[1] = std::min(h.bbox[1], poly[2 * i + 1]); h.bbox[3] = std::max(h.bbox[3], poly[2 * i + 1]);
    }
    // --- lay out
    size_t o = sizeof(EnvHeader);
    auto take = [&](size_t bytes) { size_t r = o; o += (bytes + 15) & ~(size_t)15; return (int)r; };
    const size_t sr = sizeof(R);
    // circles: K rows + one "always hit" row (radius +inf) that grid cells wholly inside a circle point at
    h.off_cx = take(sr * (K + 1)); h.off_cy = take(sr * (K + 1)); h.off_cr = take(sr * (K + 1)); h.off_creff = take(sr * (K + 1));
    h.off_creff2 = take(sr * (K + 1));
    h.off_px = take(sr * E); h.off_py = take(sr * E);
    h.off_hx = take(sr * H); h.off_hy = take(sr * H); h.off_hr = take(sr * H); h.off_hr2 = take(sr * H);
    // sentinels in front of / behind three arrays keep the lookups of geom.cuh free of bounds branches:
    // b1[-1] = just below b0[0];  brk[-1] = -inf, brk[NB] = +inf;  pfirst[-2] = pfirst[-1] = "no candidate"
    h.off_b0 = take(sr * T); h.off_b1 = take(sr * (T + 2)) + 2 * (int)sr;
    h.off_brk = take(sr * (NB + 4)) + 2 * (int)sr;
    h.off_piece = take(4 * (size_t)(NP + 1)); h.off_c1 = take(sr * cand_c1.size());
    h.off_cell = take(4 * cand_cell.size());
    h.off_pfirst = take(sizeof(PFirst<R>) * (size_t)(NP + 2)) + 2 * (int)sizeof(PFirst<R>);
    // x-bucket table over the breakpoints (find_cell): buckets of at most 0.25 m (at most 8192 of them), from one
    // bucket left of the first breakpoint to one bucket right of the last
    h.nxb = 0; h.xb0 = 0.0; h.xbw = 1.0;
    if (NB >= 2 && NB < 32760 && (double)brk[NB - 1] > (double)brk[0]) {
        const double span = (double)brk[NB - 1] - (double)brk[0];
        int nin = (int)ceil(span / 0.25);
        nin = std::min(8190, std::max(16, nin));
        h.xbw = span / nin * (1.0 + 1e-12);
        h.xb0 = (double)brk[0] - h.xbw;
        h.nxb = nin + 2;
    }
    h.off_xb = take(2 * (size_t)h.nxb);
    h.off_one = take(sizeof(One<R>) * (size_t)((K + 1) + std::max(E, 1) + std::max(H, 1)));
    h.pad_ = 0;
    h.hot_bytes = (int)o;
    h.off_probs = take(sr * (size_t)T * C);
    h.total_bytes = (int)o;          // what may be staged in shared memory ends here
    // --- classification grid (env.cuh): geometry
    int max_cells = 16384;
    if (const char *ev = getenv("AUVRRT_GRID_CELLS")) max_cells = atoi(ev);
    h.gnx = h.gny = 0; h.gs = 1.0; h.gx0 = h.gy0 = 0.0;
    if (E >= 3 && max_cells >= 16 && h.bbox[2] > h.bbox[0] && h.bbox[3] > h.bbox[1]) {
        double wx = h.bbox[2] - h.bbox[0], wy = h.bbox[3] - h.bbox[1];
        double gs = sqrt(wx * wy / max_cells);
        gs = ceil(gs * 4.0) / 4.0;                       // multiples of 0.25 m
        if (gs < 0.25) gs = 0.25;
        h.gs = gs; h.gx0 = h.bbox[0] - gs; h.gy0 = h.bbox[1] - gs;
        h.gnx = (int)ceil(wx / gs) + 2; h.gny = (int)ceil(wy / gs) + 2;
    }
    h.off_grid = take(12 * (size_t)h.gnx * h.gny);
    // --- uniform time bins?
    h.bins_uniform = 0; h.bin_s0 = 0.0; h.bin_w = 1.0;
    if (T >= 1 && T <= 32) {
        bool ok = true;
        for (int i = 0; i < T && ok; i++) {
            if (!((R)bins[2 * i + 1] > (R)bins[2 * i])) ok = false;
            if (i + 1 < T && (R)bins[2 * i + 1] != (R)bins[2 * i + 2]) ok = false;
        }
        // ... and equally wide (find_bin guesses the bin arithmetically and corrects by at most one)
        const double w = (bins[2 * T - 1] - bins[0]) / T;
        for (int i = 0; i < T && ok; i++)
            if (fabs(bins[2 * i + 1] - (bins[0] + (i + 1) * w)) > 0.25 * w) ok = false;
        if (ok) { h.bins_uniform = 1; h.bin_s0 = bins[0]; h.bin_w = w; }
    }
    std::vector<unsigned char> blob(o, 0);
    auto arr = [&](int off) { return (R *)(blob.data() + off); };
    R suffix = 0;
    for (int k = K - 1; k >= 0; k--) {
        R r = (R)circles[3 * k + 2];
        suffix = (k == K - 1) ? r : std::max(suffix, r);
        arr(h.off_cx)[k] = (R)circles[3 * k]; arr(h.off_cy)[k] = (R)circles[3 * k + 1]; arr(h.off_cr)[k] = r;
        arr(h.off_creff)[k] = suffix; arr(h.off_creff2)[k] = suffix * suffix;
    }
    arr(h.off_cx)[K] = (R)0; arr(h.off_cy)[K] = (R)0; arr(h.off_cr)[K] = (R)INFINITY;
    arr(h.off_creff)[K] = (R)INFINITY; arr(h.off_creff2)[K] = (R)INFINITY;
    for (int i = 0; i < E; i++) { arr(h.off_px)[i] = (R)poly[2 * i]; arr(h.off_py)[i] = (R)poly[2 * i + 1]; }
    {
        // single-candidate tables (env.cuh, One<R>): the same numbers the SoA arrays hold, one row per object; the edge
        // differences are formed in R exactly as the kernels' direct formula forms them
        One<R> *one = (One<R> *)(blob.data() + h.off_one);
        for (int k = 0; k <= K; k++) {
            One<R> r; r.x = arr(h.off_cx)[k]; r.y = arr(h.off_cy)[k]; r.z = arr(h.off_creff2)[k]; r.w = arr(h.off_creff)[k];
            one[k] = r;
        }
        One<R> *pone = one + (K + 1);
        { One<R> z; z.x = z.y = z.z = z.w = (R)0; pone[0] = z; }
        const R sgn = h.convex < 0 ? (R)-1 : (R)1;
        for (int i = 0; i < E; i++) {
            const int j = (i + 1) % E;
            const R ax = (R)poly[2 * i], ay = (R)poly[2 * i + 1], bx = (R)poly[2 * j], by = (R)poly[2 * j + 1];
            volatile R ex = bx - ax, ey = by - ay;
            One<R> r; r.x = ax; r.y = ay; r.z = sgn * ex; r.w = sgn * ey;
            pone[i] = r;
        }
        One<R> *hone = pone + std::max(E, 1);
        { One<R> z; z.x = z.y = (R)0; z.z = z.w = (R)-1; hone[0] = z; }
        for (int i = 0; i < H; i++) {
            const R r0 = (R)hab[3 * i + 2];
            One<R> r; r.x = (R)hab[3 * i]; r.y = (R)hab[3 * i + 1]; r.z = r0 * r0; r.w = r0;
            hone[i] = r;
        }
    }
    for (int i = 0; i < H; i++) {
        R r = (R)hab[3 * i + 2];
        arr(h.off_hx)[i] = (R)hab[3 * i]; arr(h.off_hy)[i] = (R)hab[3 * i + 1]; arr(h.off_hr)[i] = r;
        arr(h.off_hr2)[i] = r * r;
    }
    for (int i = 0; i < T; i++) { arr(h.off_b0)[i] = (R)bins[2 * i]; arr(h.off_b1)[i] = (R)bins[2 * i + 1]; }
    arr(h.off_b1)[-1] = T > 0 ? std::nextafter((R)bins[0], (R)-INFINITY) : (R)0;
    for (int i = 0; i < NB; i++) arr(h.off_brk)[i] = brk[i];
    arr(h.off_brk)[NB] = (R)INFINITY;
    arr(h.off_brk)[-1] = (R)-INFINITY;
    {
        // entry = 1 + (index of the last breakpoint left of the bucket, -1 if none); bit 15: more than one breakpoint
        // lies in the bucket grown by the margin -> walk.  The margin (2e-3 m fp32, 1e-6 m fp64) is far above the
        // rounding error of the device's bucket index, so an x that the device files under bucket b has at most
        // that one undecided breakpoint to its right.
        const double margin = sizeof(R) == 4 ? 2e-3 : 1e-6;
        unsigned short *xb = (unsigned short *)(blob.data() + h.off_xb);
        for (int b = 0; b < h.nxb; b++) {
            const double xa = h.xb0 + b * h.xbw - margin, xe = h.xb0 + (b + 1) * h.xbw + margin;
            int lo_i = -1, inside = 0;
            for (int i = 0; i < NB; i++) {
                if ((double)brk[i] < xa) lo_i = i;
                else if ((double)brk[i] <= xe) inside++;
            }
            xb[b] = (unsigned short)((lo_i + 1) | (inside > 1 ? 0x8000 : 0));
        }
        PFirst<R> *pf = (PFirst<R> *)(blob.data() + h.off_pfirst);
        { PFirst<R> none; none.c1 = (R)0; none.v = -1; pf[-2] = none; pf[-1] = none; }
        for (int p = 0; p < NP; p++) {
            PFirst<R> e; e.c1 = (R)0; e.v = -1;
            const int k0 = piece[p], k1 = piece[p + 1];
            if (k1 > k0) { e.c1 = cand_c1[k0]; e.v = cand_cell[k0] | (k1 - k0 > 1 ? (1 << 30) : 0); }
            pf[p] = e;
        }
    }
    memcpy(blob.data() + h.off_piece, piece.data(), 4 * piece.size());
    for (size_t i = 0; i < cand_c1.size(); i++) arr(h.off_c1)[i] = cand_c1[i];
    if (!cand_cell.empty()) memcpy(blob.data() + h.off_cell, cand_cell.data(), 4 * cand_cell.size());
    for (size_t i = 0; i < (size_t)T * C; i++) arr(h.off_probs)[i] = (R)probs[i];
    // --- classification grid: codes.  A code is definitive only if the whole cell, grown by `margin`
    // (far above the rounding error of the kernels' exact tests near a decision boundary), gets one
    // answer; everything else is "ambiguous" and falls back to the exact test on the device.
    if (h.gnx > 0) {
        const double margin = sizeof(R) == 4 ? 2e-3 : 1e-6;
        const double gs = h.gs, rho = gs * 0.70710678118654757 * (1.0 + 1e-9) + margin;
        unsigned *grid = (unsigned *)(blob.data() + h.off_grid);
        auto seg_dist = [](double px, double py, double ax, double ay, double bx, double by) {
            double vx = bx - ax, vy = by - ay, wx = px - ax, wy = py - ay;
            double L2 = vx * vx + vy * vy, t = L2 > 0 ? (wx * vx + wy * vy) / L2 : 0.0;
            t = t < 0 ? 0 : (t > 1 ? 1 : t);
            double dx = px - (ax + t * vx), dy = py - (ay + t * vy);
            return sqrt(dx * dx + dy * dy);
        };
        auto inside_poly = [&](double px, double py) {
            bool in = false;
            for (int i = 0, j = E - 1; i < E; j = i++) {
                double xi = poly[2 * i], yi = poly[2 * i + 1], xj = poly[2 * j], yj = poly[2 * j + 1];
                if ((yi > py) != (yj > py) && px < (xj - xi) * (py - yi) / (yj - yi) + xi) in = !in;
            }
            return in;
        };
        std::vector<double> reff(K);
        for (int k = K - 1; k >= 0; k--) reff[k] = (k == K - 1) ? circles[3 * k + 2] : std::max(reff[k + 1], circles[3 * k + 2]);
        for (int iy = 0; iy < h.gny; iy++)
            for (int ix = 0; ix < h.gnx; ix++) {
                const double x0 = h.gx0 + ix * gs, y0 = h.gy0 + iy * gs, mx = x0 + 0.5 * gs, my = y0 + 0.5 * gs;
                unsigned code = 0, w1 = 0x3FFFFFFFu, w2 = 0x0FFFFFFFu;
                // polygon: definitive if no edge comes within rho of the centre; else (convex ring) the
                // edges whose supporting line does
                double dmin = INFINITY;
                int ne = 0, ecand[2] = {0x1F, 0x1F};
                bool efull = (h.convex == 0) || E > 31;
                for (int i = 0; i < E; i++) {
                    int j = (i + 1) % E;
                    double d = seg_dist(mx, my, poly[2 * i], poly[2 * i + 1], poly[2 * j], poly[2 * j + 1]);
                    dmin = std::min(dmin, d);
                    // distance to the supporting LINE decides whether the half-plane test is constant on the cell
                    double vx = poly[2 * j] - poly[2 * i], vy = poly[2 * j + 1] - poly[2 * i + 1], L = hypot(vx, vy);
                    double dl = L > 0 ? fabs(vx * (my - poly[2 * i + 1]) - vy * (mx - poly[2 * i])) / L : 0.0;
                    if (dl <= rho) { if (ne < 2) ecand[ne] = i; ne++; }
                }
                if (dmin > rho) code |= inside_poly(mx, my) ? 1u : 2u;
                else {
                    // ambiguous w.r.t. the boundary.  For a convex ring the point is inside iff it is on the
                    // inner side of EVERY edge; edges farther than rho (as lines) have a constant side on the
                    // cell, so if any of those is the outer side the cell is outside, else only the
                    // candidates remain to be tested.
                    bool outer_const = false;
                    if (h.convex != 0)
                        for (int i = 0; i < E; i++) {
                            int j = (i + 1) % E;
                            double vx = poly[2 * j] - poly[2 * i], vy = poly[2 * j + 1] - poly[2 * i + 1], L = hypot(vx, vy);
                            double cr = vx * (my - poly[2 * i + 1]) - vy * (mx - poly[2 * i]);
                            double dl = L > 0 ? fabs(cr) / L : 0.0;
                            if (dl > rho && ((h.convex > 0 && cr < 0) || (h.convex < 0 && cr > 0))) outer_const = true;
                        }
                    if (outer_const) code |= 2u;
                    else if (efull || ne > 2) code |= AUV_GRID_POLY_FULL;
                    else {
                        w2 = (w2 & ~(0x3FFu << 18)) | ((unsigned)ecand[0] << 18) | ((unsigned)ecand[1] << 23);
                        if (ne == 1) code |= AUV_GRID_POLY_ONE | ((unsigned)ecand[0] << 26);
                    }
                }
                // obstacle circles (inflated radii): candidates = circles a point of the cell can hit
                int nc = 0; unsigned cc3[3] = {0x3FF, 0x3FF, 0x3FF};
                bool covered = false;                    // some circle holds the whole cell: every point is a hit
                for (int k = 0; k < K; k++) {
                    const double d = hypot(mx - circles[3 * k], my - circles[3 * k + 1]);
                    if (d - rho <= reff[k]) { if (nc < 3) cc3[nc] = (unsigned)k; nc++; }
                    if (d + rho < reff[k]) covered = true;
                }
                const bool poly_general = (code & 3u) == 0u && !(code & AUV_GRID_POLY_ONE);
                bool circ_general = false;
                if (nc == 0) code |= 4u;
                else if (covered && K <= 1022) code |= AUV_GRID_CIRC_ONE | ((unsigned)K << 16);
                else if (nc > 3 || K > 1022) { code |= AUV_GRID_CIRC_MANY; circ_general = true; }
                else {
                    w1 = cc3[0] | (cc3[1] << 10) | (cc3[2] << 20);
                    if (nc == 1) code |= AUV_GRID_CIRC_ONE | (cc3[0] << 16);
                    else circ_general = true;
                }
                if (poly_general || circ_general) code |= AUV_GRID_SLOW;
                // habitats: first match in list order
                unsigned hc = AUV_GRID_HAB_NONE;
                int nh = 0; unsigned hh3[3] = {0x3F, 0x3F, 0x3F};
                bool hmany = false;
                for (int q = 0; q < H; q++) {
                    double d = hypot(mx - hab[3 * q], my - hab[3 * q + 1]);
                    if (d - rho <= hab[3 * q + 2]) {                       // the cell touches habitat q
                        const bool covers = d + rho < hab[3 * q + 2];
                        if (nh == 0 && covers && q < 64) { hc = (unsigned)q; break; }    // definitive
                        hc = AUV_GRID_HAB_AMBIG;
                        if (nh < 3) hh3[nh] = (unsigned)q; else hmany = true;
                        nh++;
                        if (covers) break;                                 // later habitats can never be first
                    }
                }
                if (hc == AUV_GRID_HAB_AMBIG) {
                    if (hmany || H > 62) code |= AUV_GRID_HAB_MANY;
                    else {
                        w2 = (w2 & ~0x3FFFFu) | hh3[0] | (hh3[1] << 6) | (hh3[2] << 12);
                        if (nh == 1) hc = AUV_GRID_HAB_ONE + hh3[0];      // only this habitat can hold a point of the cell
                    }
                }
                code |= hc << 3;
                const size_t ncell = (size_t)h.gnx * h.gny, ci = (size_t)iy * h.gnx + ix;      // three planes
                grid[ci] = code; grid[ncell + ci] = w1; grid[2 * ncell + ci] = w2;
            }
    }
    memcpy(blob.data(), &h, sizeof(h));
    *hout = h;
    return blob;
}

int check_precision(int precision) {
    if (precision != AUVRRT_F32 && precision != AUVRRT_F64) return set_err(AUVRRT_ERR_ARG, "precision must be AUVRRT_F32 or AUVRRT_F64");
    return AUVRRT_OK;
}

// One host-buffer call on the legacy default stream.  in() copies a host array to the device when it is declared;
// out() allocates a device output that finish(), after the launch, copies back where the host pointer is non-null.
// Real arrays (in_real, out_real) are double on the host and R on the device: for R = float they pass through an fp64
// buffer and k_convert / k_convert_back.  Zero-length arrays get 16 bytes.  Every buffer lives as long as the object.
// The first error sticks in rc: later steps do nothing and hand out NULL, so a caller checks rc once, before its launch.
class Staging {
  public:
    int rc = AUVRRT_OK;

    template <typename T> const T *in(const T *h, int64_t n) {
        T *d = (T *)alloc(sizeof(T), n, false);
        if (d && n > 0) copy(d, h, sizeof(T) * (size_t)n, cudaMemcpyHostToDevice);
        return d;
    }
    template <typename R> const R *in_real(const double *h, int64_t n) {
        if (sizeof(R) == 8) return (const R *)in(h, n);
        R *d = (R *)alloc(sizeof(R), n, false);
        if (d && n > 0) {
            const double *t = in(h, n);
            if (t) keep(launch_convert<R>(t, d, n, 0));
        }
        return d;
    }
    template <typename T> T *out(T *h, int64_t n, bool zero = false) {
        T *d = (T *)alloc(sizeof(T), n, zero);
        if (d && h && n > 0) outs.push_back(Out{h, d, n, false, sizeof(T) * (size_t)n});
        return d;
    }
    template <typename R> R *out_real(double *h, int64_t n, bool zero = false) {
        if (sizeof(R) == 8) return (R *)out(h, n, zero);
        R *d = (R *)alloc(sizeof(R), n, zero);
        if (d && h && n > 0) outs.push_back(Out{h, d, n, true, 8 * (size_t)n});
        return d;
    }
    // every conversion and copy back, then one synchronisation
    int finish() {
        for (const Out &o : outs) {
            const void *src = o.dev;
            if (o.widen) {
                double *t = (double *)alloc(8, o.n, false);
                if (t) keep(launch_convert_back<float>((const float *)o.dev, t, o.n, 0));
                src = t;
            }
            copy(o.host, src, o.bytes, cudaMemcpyDeviceToHost);
        }
        if (!rc) keep_cuda(cudaStreamSynchronize(0), "cudaStreamSynchronize");
        return rc;
    }

  private:
    struct Out { void *host; const void *dev; int64_t n; bool widen; size_t bytes; };   // bytes: on the host
    std::deque<DBuf> bufs;
    std::vector<Out> outs;

    void *alloc(size_t size, int64_t n, bool zero) {
        if (rc) return nullptr;
        bufs.emplace_back();
        DBuf &b = bufs.back();
        if ((rc = b.alloc(n > 0 ? size * (size_t)n : 0))) return nullptr;
        if (zero) keep_cuda(cudaMemsetAsync(b.p, 0, b.bytes, 0), "cudaMemsetAsync");
        return rc ? nullptr : b.p;
    }
    void copy(void *dst, const void *src, size_t bytes, cudaMemcpyKind kind) {
        if (!rc) keep_cuda(cudaMemcpyAsync(dst, src, bytes, kind, 0), "cudaMemcpyAsync");
    }
    void keep(int r) { if (!rc) rc = r; }
    void keep_cuda(cudaError_t e, const char *what) {
        if (e != cudaSuccess) keep(set_err(AUVRRT_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e)));
    }
};

// env-owned buffers of the host plan path, grown on demand and reused across calls: device scratch or pinned host staging
int env_grow(void *&p, size_t &have, size_t bytes, bool pinned, void **out) {
    if (have < bytes) {
        if (p) { if (pinned) cudaFreeHost(p); else cudaFree(p); }
        p = nullptr; have = 0;
        const size_t want = bytes + bytes / 4 + 256;
        cudaError_t er = pinned ? cudaMallocHost(&p, want) : cudaMalloc(&p, want);
        if (er != cudaSuccess)
            return set_err(AUVRRT_ERR_CUDA, "%s(%zu): %s", pinned ? "cudaMallocHost" : "cudaMalloc", want, cudaGetErrorString(er));
        have = want;
    }
    *out = p;
    return AUVRRT_OK;
}
int env_dev_scratch(auvrrt_env *e, int slot, size_t bytes, void **out) {
    return env_grow(e->d_scratch[slot], e->d_scratch_bytes[slot], bytes, false, out);
}
int env_pinned(auvrrt_env *e, int slot, size_t bytes, void **out) {
    return env_grow(e->h_pinned[slot], e->h_pinned_bytes[slot], bytes, true, out);
}

}  // namespace

// ------------------------------------------------------------------ env
extern "C" int auvrrt_env_create(const double *circles, int K, const double *poly, int E, const double *habitats,
                                 int H, const double *bins, int T, const double *cells, int C, const double *probs,
                                 int device, auvrrt_env_t **out) {
    if (!out) return set_err(AUVRRT_ERR_ARG, "env_create: out is NULL");
    *out = nullptr;
    if (K < 0 || E < 0 || H < 0 || T < 0 || C < 0) return set_err(AUVRRT_ERR_ARG, "env_create: negative count");
    if ((K && !circles) || (E && !poly) || (H && !habitats) || (T && !bins) || (C && !cells) || (T && C && !probs))
        return set_err(AUVRRT_ERR_ARG, "env_create: NULL array with non-zero count");
    if (H > 64) return set_err(AUVRRT_ERR_UNSUPPORTED, "env_create: more than 64 habitats");
    AUV_TRY(need_device(device));
    auvrrt_env *e = new auvrrt_env();
    memset(e, 0, sizeof(*e));
    e->device = device; e->K = K; e->E = E; e->H = H; e->T = T; e->C = C;
    e->h_bins = (double *)malloc(16 * (size_t)std::max(T, 1));
    if (!e->h_bins) { delete e; return set_err(AUVRRT_ERR_CUDA, "env_create: out of host memory"); }
    if (T) memcpy(e->h_bins, bins, 16 * (size_t)T);
    std::vector<unsigned char> b32 = build_blob<float>(circles, K, poly, E, habitats, H, bins, T, cells, C, probs, &e->h32);
    std::vector<unsigned char> b64 = build_blob<double>(circles, K, poly, E, habitats, H, bins, T, cells, C, probs, &e->h64);
    cudaError_t er = cudaMalloc((void **)&e->blob32, b32.size());
    if (er == cudaSuccess) er = cudaMalloc((void **)&e->blob64, b64.size());
    if (er == cudaSuccess) er = cudaMemcpy(e->blob32, b32.data(), b32.size(), cudaMemcpyHostToDevice);
    if (er == cudaSuccess) er = cudaMemcpy(e->blob64, b64.data(), b64.size(), cudaMemcpyHostToDevice);
    if (er == cudaSuccess) er = cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking);
    if (er != cudaSuccess) {
        int rc = set_err(AUVRRT_ERR_CUDA, "env_create: %s", cudaGetErrorString(er));
        auvrrt_env_destroy(e);
        return rc;
    }
    *out = e;
    return AUVRRT_OK;
}
// The world-model blob as the kernels see it (EnvHeader + tables, env.cuh), built on the host only: what the
// CPU-only tests validate the classification grid and the cell index against the exact predicates with.
extern "C" int64_t auvrrt_env_host_blob(const double *circles, int K, const double *poly, int E, const double *habitats,
                                        int H, const double *bins, int T, const double *cells, int C, const double *probs,
                                        int precision, unsigned char *out, int64_t cap) {
    if (K < 0 || E < 0 || H < 0 || T < 0 || C < 0 || H > 64 || (precision != AUVRRT_F32 && precision != AUVRRT_F64)) {
        set_err(AUVRRT_ERR_ARG, "env_host_blob: bad argument");
        return -1;
    }
    EnvHeader h;
    std::vector<unsigned char> b = AUV_DISPATCH(precision, build_blob, circles, K, poly, E, habitats, H, bins, T, cells, C, probs, &h);
    if (out && cap >= (int64_t)b.size()) memcpy(out, b.data(), b.size());
    return (int64_t)b.size();
}
extern "C" void auvrrt_env_destroy(auvrrt_env_t *e) {
    if (!e) return;
    cudaSetDevice(e->device);
    if (e->blob32) cudaFree(e->blob32);
    if (e->blob64) cudaFree(e->blob64);
    for (int i = 0; i < 8; i++) if (e->d_scratch[i]) cudaFree(e->d_scratch[i]);
    for (int i = 0; i < 4; i++) if (e->h_pinned[i]) cudaFreeHost(e->h_pinned[i]);
    if (e->stream) cudaStreamDestroy(e->stream);
    free(e->h_bins);
    delete e;
}

// ------------------------------------------------------------------ shark-occupancy table of a live world
extern "C" int auvrrt_env_set_probs_dev(auvrrt_env_t *env, const double *d_probs, void *stream) {
    if (!env || (!d_probs && (int64_t)env->T * env->C > 0)) return set_err(AUVRRT_ERR_ARG, "env_set_probs_dev: NULL argument");
    AUV_CUDA(cudaSetDevice(env->device));
    return launch_probs_to_env(env, d_probs, nullptr, 0, (cudaStream_t)stream);
}
extern "C" int auvrrt_env_set_probs(auvrrt_env_t *env, const double *probs) {
    if (!env || (!probs && (int64_t)env->T * env->C > 0)) return set_err(AUVRRT_ERR_ARG, "env_set_probs: NULL argument");
    const size_t n = (size_t)env->T * env->C;
    if (n == 0) return AUVRRT_OK;
    AUV_CUDA(cudaSetDevice(env->device));
    void *d = nullptr;
    AUV_TRY(env_dev_scratch(env, 7, 8 * n, &d));
    AUV_CUDA(cudaMemcpyAsync(d, probs, 8 * n, cudaMemcpyHostToDevice, env->stream));
    AUV_TRY(launch_probs_to_env(env, (const double *)d, nullptr, 0, env->stream));
    AUV_CUDA(cudaStreamSynchronize(env->stream));
    return AUVRRT_OK;
}
extern "C" int auvrrt_env_get_probs(const auvrrt_env_t *env, int precision, double *out) {
    if (!env || (!out && (int64_t)env->T * env->C > 0)) return set_err(AUVRRT_ERR_ARG, "env_get_probs: NULL argument");
    AUV_TRY(check_precision(precision));
    const size_t n = (size_t)env->T * env->C;
    if (n == 0) return AUVRRT_OK;
    AUV_CUDA(cudaSetDevice(env->device));
    if (precision == AUVRRT_F64) {
        AUV_CUDA(cudaMemcpyAsync(out, env->blob64 + env->h64.off_probs, 8 * n, cudaMemcpyDeviceToHost, env->stream));
        AUV_CUDA(cudaStreamSynchronize(env->stream));
        return AUVRRT_OK;
    }
    std::vector<float> f(n);
    AUV_CUDA(cudaMemcpyAsync(f.data(), env->blob32 + env->h32.off_probs, 4 * n, cudaMemcpyDeviceToHost, env->stream));
    AUV_CUDA(cudaStreamSynchronize(env->stream));
    for (size_t i = 0; i < n; i++) out[i] = (double)f[i];
    return AUVRRT_OK;
}

// ------------------------------------------------------------------ nearest node
extern "C" int64_t auvrrt_nn_scratch_bytes(int nq) { return nn_scratch_bytes(nq); }
extern "C" int auvrrt_nn_dev(const void *tx, const void *ty, int64_t n, const void *qx, const void *qy, int nq,
                             int precision, void *scratch, int64_t scratch_bytes, int32_t *out_idx, void *stream) {
    AUV_TRY(check_precision(precision));
    cudaStream_t s = (cudaStream_t)stream;
    if (precision == AUVRRT_F32)
        return launch_nn<float>((const float *)tx, (const float *)ty, n, (const float *)qx, (const float *)qy, nq, scratch, scratch_bytes, out_idx, s);
    return launch_nn<double>((const double *)tx, (const double *)ty, n, (const double *)qx, (const double *)qy, nq, scratch, scratch_bytes, out_idx, s);
}
template <typename R>
static int nn_host(const double *tx, const double *ty, int64_t n, const double *qx, const double *qy, int nq, int32_t *out) {
    Staging st;
    const R *dtx = st.in_real<R>(tx, n), *dty = st.in_real<R>(ty, n), *dqx = st.in_real<R>(qx, nq), *dqy = st.in_real<R>(qy, nq);
    const int64_t scratch_bytes = nn_scratch_bytes(nq);
    unsigned char *scratch = st.out<unsigned char>(nullptr, scratch_bytes);
    int32_t *didx = st.out(out, nq);
    AUV_TRY(st.rc);
    AUV_TRY(launch_nn<R>(dtx, dty, n, dqx, dqy, nq, scratch, scratch_bytes, didx, 0));
    return st.finish();
}
extern "C" int auvrrt_nn(const double *tx, const double *ty, int64_t n, const double *qx, const double *qy, int nq,
                         int precision, int device, int32_t *out_idx) {
    AUV_TRY(check_precision(precision));
    AUV_TRY(need_device(device));
    if (nq <= 0) return AUVRRT_OK;
    if (n <= 0) return set_err(AUVRRT_ERR_ARG, "nn: empty tree");
    return AUV_DISPATCH(precision, nn_host, tx, ty, n, qx, qy, nq, out_idx);
}

// ------------------------------------------------------------------ steer (arc)
template <typename R>
static int steer_arc_host(const double *parents, int64_t n, const double *u, const int64_t *uoff, const double params[5],
                          double *leaf, int32_t *counts, double *wp, int wp_cap, int32_t *used, int32_t *status) {
    Staging st;
    const R *dp = st.in_real<R>(parents, 5 * n);
    const double *du = st.in(u, uoff[n]);
    const int64_t *doff = st.in(uoff, n + 1);
    R *dleaf = st.out_real<R>(leaf, 5 * n);
    int32_t *dcnt = st.out(counts, n);
    // wp_cap 0: one zeroed row per edge on the device, nothing to copy back
    R *dwp = st.out_real<R>(wp_cap > 0 ? wp : nullptr, 6 * n * std::max(wp_cap, 1), true);
    int32_t *dused = st.out(used, n), *dst = st.out(status, n);
    AUV_TRY(st.rc);
    AUV_TRY(launch_steer_arc<R>(dp, n, du, doff, params, dleaf, dcnt, dwp, wp_cap, dused, dst, 0));
    return st.finish();
}
extern "C" int auvrrt_steer_arc(const double *parents, int64_t n, const double *u, const int64_t *uoff,
                                const double params[5], int precision, int device, double *leaf, int32_t *counts,
                                double *waypoints, int wp_cap, int32_t *used, int32_t *status) {
    AUV_TRY(check_precision(precision));
    AUV_TRY(need_device(device));
    if (n <= 0) return AUVRRT_OK;
    if (!parents || !u || !uoff || !params) return set_err(AUVRRT_ERR_ARG, "steer_arc: NULL input");
    return AUV_DISPATCH(precision, steer_arc_host, parents, n, u, uoff, params, leaf, counts, waypoints, wp_cap, used, status);
}

// ------------------------------------------------------------------ steer (Dubins)
template <typename R>
static int steer_dubins_host(const double *from, const double *to, int64_t n, double rho, int W, uint8_t *word,
                             double *seg, double *length, double *wp) {
    Staging st;
    const R *df = st.in_real<R>(from, 3 * n), *dt = st.in_real<R>(to, 3 * n);
    uint8_t *dword = st.out(word, n);
    R *dseg = st.out_real<R>(seg, 3 * n), *dlen = st.out_real<R>(length, n);
    R *dwp = wp ? st.out_real<R>(wp, 3 * n * W, true) : nullptr;
    AUV_TRY(st.rc);
    AUV_TRY(launch_steer_dubins<R>(df, dt, n, rho, W, dword, dseg, dlen, dwp, 0));
    return st.finish();
}
extern "C" int auvrrt_steer_dubins(const double *from, const double *to, int64_t n, double rho, int W, int precision,
                                   int device, uint8_t *word, double *seg, double *length, double *waypoints) {
    AUV_TRY(check_precision(precision));
    AUV_TRY(need_device(device));
    if (n <= 0) return AUVRRT_OK;
    if (!(rho > 0)) return set_err(AUVRRT_ERR_ARG, "steer_dubins: rho must be > 0");
    if (waypoints && W < 2) return set_err(AUVRRT_ERR_ARG, "steer_dubins: W must be >= 2");
    return AUV_DISPATCH(precision, steer_dubins_host, from, to, n, rho, W, word, seg, length, waypoints);
}

// ------------------------------------------------------------------ collide
template <typename R>
static int collide_host(const auvrrt_env *env, const double *points, const int64_t *off, int64_t n, uint8_t *out) {
    Staging st;
    const R *dp = st.in_real<R>(points, 2 * off[n]);
    const int64_t *doff = st.in(off, n + 1);
    uint8_t *dout = st.out(out, n);
    AUV_TRY(st.rc);
    AUV_TRY(launch_collide<R>(env, dp, doff, n, dout, 0));
    return st.finish();
}
extern "C" int auvrrt_collide(const auvrrt_env_t *env, const double *points, const int64_t *off, int64_t n,
                              int precision, uint8_t *out_safe) {
    AUV_TRY(check_precision(precision));
    if (!env) return set_err(AUVRRT_ERR_ARG, "collide: env is NULL");
    AUV_TRY(need_device(env->device));
    if (n <= 0) return AUVRRT_OK;
    return AUV_DISPATCH(precision, collide_host, env, points, off, n, out_safe);
}
template <typename R>
static int collide_points_host(const auvrrt_env *env, const double *points, int64_t n, uint8_t *out) {
    Staging st;
    const R *dp = st.in_real<R>(points, 2 * n);
    uint8_t *dout = st.out(out, n);
    AUV_TRY(st.rc);
    AUV_TRY(launch_collide_points<R>(env, dp, n, dout, 0));
    return st.finish();
}
extern "C" int auvrrt_collide_points(const auvrrt_env_t *env, const double *points, int64_t n, int precision, uint8_t *out_safe) {
    AUV_TRY(check_precision(precision));
    if (!env) return set_err(AUVRRT_ERR_ARG, "collide_points: env is NULL");
    AUV_TRY(need_device(env->device));
    if (n <= 0) return AUVRRT_OK;
    return AUV_DISPATCH(precision, collide_points_host, env, points, n, out_safe);
}

// ------------------------------------------------------------------ cost
template <typename R>
static int cost_host(const auvrrt_env *env, const double *points, const int64_t *off, int64_t n, const double *t_total,
                     const double weights[3], unsigned mask, int n_hab, double *out) {
    Staging st;
    const R *dp = st.in_real<R>(points, 3 * off[n]);
    const int64_t *doff = st.in(off, n + 1);
    const R *dt = st.in_real<R>(t_total, n);
    R *dout = st.out_real<R>(out, 4 * n);
    AUV_TRY(st.rc);
    AUV_TRY(launch_cost<R>(env, dp, doff, n, dt, weights, mask, n_hab, dout, 0));
    return st.finish();
}
extern "C" int auvrrt_cost(const auvrrt_env_t *env, const double *points, const int64_t *off, int64_t n,
                           const double *t_total, const double weights[3], const uint8_t *bin_mask, int n_habitats,
                           int precision, double *out) {
    AUV_TRY(check_precision(precision));
    if (!env) return set_err(AUVRRT_ERR_ARG, "cost: env is NULL");
    AUV_TRY(need_device(env->device));
    if (n <= 0) return AUVRRT_OK;
    unsigned mask = 0xffffffffu;
    if (bin_mask) {
        if (env->T > 32) return set_err(AUVRRT_ERR_UNSUPPORTED, "cost: bin_mask supports at most 32 time bins");
        mask = 0;
        for (int b = 0; b < env->T; b++) if (bin_mask[b]) mask |= 1u << b;
    }
    int nh = n_habitats < 0 ? env->H : std::min(n_habitats, env->H);
    return AUV_DISPATCH(precision, cost_host, env, points, off, n, t_total, weights, mask, nh, out);
}
template <typename R>
static int cost_point_host(const auvrrt_env *env, const double *points, int64_t n, unsigned long long visited, int tb,
                           const double weights[3], double *out) {
    Staging st;
    const R *dp = st.in_real<R>(points, 2 * n);
    R *dout = st.out_real<R>(out, n);
    AUV_TRY(st.rc);
    AUV_TRY(launch_cost_point<R>(env, dp, n, visited, tb, weights, dout, 0));
    return st.finish();
}
extern "C" int auvrrt_cost_point(const auvrrt_env_t *env, const double *points, int64_t n, const uint8_t *visited,
                                 int tb, const double weights[3], int precision, double *out_sum) {
    AUV_TRY(check_precision(precision));
    if (!env) return set_err(AUVRRT_ERR_ARG, "cost_point: env is NULL");
    AUV_TRY(need_device(env->device));
    if (n <= 0) return AUVRRT_OK;
    unsigned long long vm = 0;
    if (visited) for (int h = 0; h < env->H; h++) if (visited[h]) vm |= 1ull << h;
    return AUV_DISPATCH(precision, cost_point_host, env, points, n, vm, tb, weights, out_sum);
}

// ------------------------------------------------------------------ fused edges
extern "C" int auvrrt_edges_dubins_dev(const auvrrt_env_t *env, const void *from, const void *to, int64_t n, double rho,
                                       int W, int precision, uint8_t *out_safe, uint8_t *out_word, void *out_length,
                                       void *stream) {
    AUV_TRY(check_precision(precision));
    if (!env) return set_err(AUVRRT_ERR_ARG, "edges_dubins: env is NULL");
    cudaStream_t s = (cudaStream_t)stream;
    if (precision == AUVRRT_F32)
        return launch_edges_dubins<float>(env, (const float *)from, (const float *)to, n, rho, W, out_safe, out_word, (float *)out_length, s);
    return launch_edges_dubins<double>(env, (const double *)from, (const double *)to, n, rho, W, out_safe, out_word, (double *)out_length, s);
}
extern "C" int auvrrt_edges_arc_dev(const auvrrt_env_t *env, const void *parents, const uint64_t *seeds, int64_t n,
                                    const double params[5], int precision, uint8_t *out_safe, int32_t *out_counts,
                                    void *out_leaf, void *stream) {
    AUV_TRY(check_precision(precision));
    if (!env) return set_err(AUVRRT_ERR_ARG, "edges_arc: env is NULL");
    cudaStream_t s = (cudaStream_t)stream;
    if (precision == AUVRRT_F32)
        return launch_edges_arc<float>(env, (const float *)parents, seeds, n, params, out_safe, out_counts, (float *)out_leaf, s);
    return launch_edges_arc<double>(env, (const double *)parents, seeds, n, params, out_safe, out_counts, (double *)out_leaf, s);
}
template <typename R>
static int edges_dubins_host(const auvrrt_env *env, const double *from, const double *to, int64_t n, double rho, int W,
                             uint8_t *safe, uint8_t *word, double *length, double vel = 1.0, double w3 = 0.0, double *cost = nullptr) {
    Staging st;
    const R *df = st.in_real<R>(from, 3 * n), *dt = st.in_real<R>(to, 3 * n);
    uint8_t *dsafe = st.out(safe, n), *dword = st.out(word, n);
    R *dlen = st.out_real<R>(length, n);
    R *dcost = cost ? st.out_real<R>(cost, 3 * n) : nullptr;
    AUV_TRY(st.rc);
    AUV_TRY(launch_edges_dubins<R>(env, df, dt, n, rho, W, dsafe, dword, dlen, 0, vel, w3, dcost));
    return st.finish();
}
extern "C" int auvrrt_edges_dubins(const auvrrt_env_t *env, const double *from, const double *to, int64_t n, double rho,
                                   int W, int precision, uint8_t *out_safe, uint8_t *out_word, double *out_length) {
    AUV_TRY(check_precision(precision));
    if (!env) return set_err(AUVRRT_ERR_ARG, "edges_dubins: env is NULL");
    AUV_TRY(need_device(env->device));
    if (n <= 0) return AUVRRT_OK;
    return AUV_DISPATCH(precision, edges_dubins_host, env, from, to, n, rho, W, out_safe, out_word, out_length);
}
extern "C" int auvrrt_edges_dubins_cost_dev(const auvrrt_env_t *env, const void *from, const void *to, int64_t n, double rho,
                                            int W, double velocity, double w3, int precision, uint8_t *out_safe,
                                            uint8_t *out_word, void *out_length, void *out_cost, void *stream) {
    AUV_TRY(check_precision(precision));
    if (!env) return set_err(AUVRRT_ERR_ARG, "edges_dubins_cost: env is NULL");
    if (!out_cost) return set_err(AUVRRT_ERR_ARG, "edges_dubins_cost: out_cost is NULL");
    cudaStream_t s = (cudaStream_t)stream;
    if (precision == AUVRRT_F32)
        return launch_edges_dubins<float>(env, (const float *)from, (const float *)to, n, rho, W, out_safe, out_word, (float *)out_length, s,
                                          velocity, w3, (float *)out_cost);
    return launch_edges_dubins<double>(env, (const double *)from, (const double *)to, n, rho, W, out_safe, out_word, (double *)out_length, s,
                                       velocity, w3, (double *)out_cost);
}
extern "C" int auvrrt_edges_dubins_cost(const auvrrt_env_t *env, const double *from, const double *to, int64_t n, double rho,
                                        int W, double velocity, double w3, int precision, uint8_t *out_safe,
                                        uint8_t *out_word, double *out_length, double *out_cost) {
    AUV_TRY(check_precision(precision));
    if (!env) return set_err(AUVRRT_ERR_ARG, "edges_dubins_cost: env is NULL");
    if (!out_cost) return set_err(AUVRRT_ERR_ARG, "edges_dubins_cost: out_cost is NULL");
    AUV_TRY(need_device(env->device));
    if (n <= 0) return AUVRRT_OK;
    return AUV_DISPATCH(precision, edges_dubins_host, env, from, to, n, rho, W, out_safe, out_word, out_length, velocity, w3, out_cost);
}
template <typename R>
static int edges_arc_host(const auvrrt_env *env, const double *parents, const uint64_t *seeds, int64_t n,
                          const double params[5], uint8_t *safe, int32_t *counts, double *leaf, double w3 = 0.0,
                          double *cost = nullptr) {
    Staging st;
    const R *dp = st.in_real<R>(parents, 5 * n);
    const uint64_t *dseed = st.in(seeds, n);
    uint8_t *dsafe = st.out(safe, n);
    int32_t *dcnt = st.out(counts, n);
    R *dleaf = st.out_real<R>(leaf, 5 * n);
    R *dcost = cost ? st.out_real<R>(cost, 3 * n) : nullptr;
    AUV_TRY(st.rc);
    AUV_TRY(launch_edges_arc<R>(env, dp, dseed, n, params, dsafe, dcnt, dleaf, 0, w3, dcost));
    return st.finish();
}
extern "C" int auvrrt_edges_arc(const auvrrt_env_t *env, const double *parents, const uint64_t *seeds, int64_t n,
                                const double params[5], int precision, uint8_t *out_safe, int32_t *out_counts,
                                double *out_leaf) {
    AUV_TRY(check_precision(precision));
    if (!env) return set_err(AUVRRT_ERR_ARG, "edges_arc: env is NULL");
    AUV_TRY(need_device(env->device));
    if (n <= 0) return AUVRRT_OK;
    return AUV_DISPATCH(precision, edges_arc_host, env, parents, seeds, n, params, out_safe, out_counts, out_leaf);
}

extern "C" int auvrrt_edges_arc_cost_dev(const auvrrt_env_t *env, const void *parents, const uint64_t *seeds, int64_t n,
                                         const double params[5], double w3, int precision, uint8_t *out_safe,
                                         int32_t *out_counts, void *out_leaf, void *out_cost, void *stream) {
    AUV_TRY(check_precision(precision));
    if (!env || !out_cost) return set_err(AUVRRT_ERR_ARG, "edges_arc_cost: env / out_cost is NULL");
    cudaStream_t s = (cudaStream_t)stream;
    if (precision == AUVRRT_F32)
        return launch_edges_arc<float>(env, (const float *)parents, seeds, n, params, out_safe, out_counts, (float *)out_leaf, s, w3,
                                       (float *)out_cost);
    return launch_edges_arc<double>(env, (const double *)parents, seeds, n, params, out_safe, out_counts, (double *)out_leaf, s, w3,
                                    (double *)out_cost);
}
extern "C" int auvrrt_edges_arc_cost(const auvrrt_env_t *env, const double *parents, const uint64_t *seeds, int64_t n,
                                     const double params[5], double w3, int precision, uint8_t *out_safe,
                                     int32_t *out_counts, double *out_leaf, double *out_cost) {
    AUV_TRY(check_precision(precision));
    if (!env || !out_cost || !out_safe || !out_counts || !out_leaf) return set_err(AUVRRT_ERR_ARG, "edges_arc_cost: NULL argument");
    AUV_TRY(need_device(env->device));
    if (n <= 0) return AUVRRT_OK;
    return AUV_DISPATCH(precision, edges_arc_host, env, parents, seeds, n, params, out_safe, out_counts, out_leaf, w3, out_cost);
}

// ------------------------------------------------------------------ planner
extern "C" int64_t auvrrt_plan_workspace_bytes(const auvrrt_env_t *env, const auvrrt_plan_params_t *params, int precision) {
    if (!env || !params || check_precision(precision)) return -1;
    if (need_device(env->device)) return -1;
    return AUV_DISPATCH(precision, plan_workspace_bytes, env, params, 0);
}
extern "C" int64_t auvrrt_plan_workspace_bytes_q(const auvrrt_env_t *env, const auvrrt_plan_params_t *params, int precision, int64_t Q) {
    if (!env || !params || check_precision(precision)) return -1;
    if (need_device(env->device)) return -1;
    return AUV_DISPATCH(precision, plan_workspace_bytes, env, params, Q);
}
extern "C" int auvrrt_plan_batch_dev(const auvrrt_env_t *env, const void *starts, const uint64_t *seeds, int64_t Q,
                                     const auvrrt_plan_params_t *params, int precision, void *workspace,
                                     int64_t workspace_bytes, auvrrt_plan_record_t *out_records, uint32_t *out_chain,
                                     void *out_path, const auvrrt_plan_trace_t *trace, void *stream) {
    AUV_TRY(check_precision(precision));
    if (!env || !params) return set_err(AUVRRT_ERR_ARG, "plan_batch: NULL env or params");
    // the in-kernel path writer walks the chain buffer: without one no path would be written
    if (out_path && params->path_cap > 0 && !out_chain)
        return set_err(AUVRRT_ERR_ARG, "plan_batch: out_path needs out_chain");
    cudaStream_t s = (cudaStream_t)stream;
    if (precision == AUVRRT_F32)
        return launch_plan<float>(env, (const float *)starts, seeds, Q, params, workspace, workspace_bytes, out_records, out_chain, (float *)out_path, trace, s);
    return launch_plan<double>(env, (const double *)starts, seeds, Q, params, workspace, workspace_bytes, out_records, out_chain, (double *)out_path, trace, s);
}

// Host-buffer planner: the call a reference-side binding makes.  Device buffers and pinned staging
// areas are owned by the env handle and reused across calls.
template <typename R>
static int plan_host(auvrrt_env *env, const double *starts, const uint64_t *seeds, int64_t Q,
                     const auvrrt_plan_params_t *p, auvrrt_plan_record_t *rec, uint32_t *chain, double *path,
                     const auvrrt_plan_trace_t *trace) {
    cudaStream_t s = env->stream;
    const int I = p->iterations;
    int64_t wsb = plan_workspace_bytes<R>(env, p, Q);
    if (wsb < 0) return AUVRRT_ERR_CUDA;
    void *ws, *dstart, *dseed, *drec, *dchain = nullptr, *dpath = nullptr, *dtrace = nullptr;
    AUV_TRY(env_dev_scratch(env, 0, (size_t)wsb, &ws));
    AUV_TRY(env_dev_scratch(env, 1, sizeof(R) * 5 * (size_t)Q, &dstart));
    AUV_TRY(env_dev_scratch(env, 2, 8 * (size_t)Q, &dseed));
    AUV_TRY(env_dev_scratch(env, 3, sizeof(auvrrt_plan_record_t) * (size_t)Q, &drec));
    const int ccap = p->chain_cap > 0 ? p->chain_cap : 1;
    if (chain) AUV_TRY(env_dev_scratch(env, 4, 4 * (size_t)Q * ccap, &dchain));
    // in-kernel path materialisation walks the chain, so paths need a chain buffer
    if (path && p->path_cap > 0 && p->group == 1)
        return set_err(AUVRRT_ERR_UNSUPPORTED, "plan_batch: group 1 (thread per tree) writes no paths; use auvrrt_materialize");
    if (path && p->path_cap > 0) {
        AUV_TRY(env_dev_scratch(env, 4, 4 * (size_t)Q * ccap, &dchain));
        AUV_TRY(env_dev_scratch(env, 5, sizeof(R) * 6 * (size_t)Q * p->path_cap, &dpath));
    }
    // inputs: host -> pinned -> device
    void *hp;
    AUV_TRY(env_pinned(env, 0, sizeof(R) * 5 * (size_t)Q + 8 * (size_t)Q, &hp));
    R *hs = (R *)hp;
    for (int64_t i = 0; i < 5 * Q; i++) hs[i] = (R)starts[i];
    uint64_t *hseed = (uint64_t *)((unsigned char *)hp + ((sizeof(R) * 5 * (size_t)Q + 7) & ~(size_t)7));
    memcpy(hseed, seeds, 8 * (size_t)Q);
    AUV_CUDA(cudaMemcpyAsync(dstart, hs, sizeof(R) * 5 * (size_t)Q, cudaMemcpyHostToDevice, s));
    AUV_CUDA(cudaMemcpyAsync(dseed, hseed, 8 * (size_t)Q, cudaMemcpyHostToDevice, s));
    auvrrt_plan_trace_t dtr;
    memset(&dtr, 0, sizeof(dtr));
    size_t n_it = (size_t)Q * I;
    if (p->trace) {
        if (!trace) return set_err(AUVRRT_ERR_ARG, "plan_batch: trace requested without trace buffers");
        size_t bytes = n_it * (4 + 4 + 8 + 5 * sizeof(R)) + n_it + 64;
        AUV_TRY(env_dev_scratch(env, 6, bytes, &dtrace));
        unsigned char *b = (unsigned char *)dtrace;
        dtr.leaf = (double *)b; b += n_it * 5 * sizeof(R);
        dtr.upos = (int64_t *)b; b += n_it * 8;
        dtr.parent = (int32_t *)b; b += n_it * 4;
        dtr.nwp = (int32_t *)b; b += n_it * 4;
        dtr.safe = (uint8_t *)b;
        AUV_CUDA(cudaMemsetAsync(dtrace, 0, bytes, s));
    }
    AUV_TRY(launch_plan<R>(env, (const R *)dstart, (const uint64_t *)dseed, Q, p, ws, wsb, (auvrrt_plan_record_t *)drec,
                           (uint32_t *)dchain, (R *)dpath, p->trace ? &dtr : nullptr, s));
    // outputs: device -> pinned -> caller
    void *hrec;
    AUV_TRY(env_pinned(env, 1, sizeof(auvrrt_plan_record_t) * (size_t)Q, &hrec));
    AUV_CUDA(cudaMemcpyAsync(hrec, drec, sizeof(auvrrt_plan_record_t) * (size_t)Q, cudaMemcpyDeviceToHost, s));
    void *hchain = nullptr, *hpath = nullptr;
    if (chain) {
        AUV_TRY(env_pinned(env, 2, 4 * (size_t)Q * ccap, &hchain));
        AUV_CUDA(cudaMemcpyAsync(hchain, dchain, 4 * (size_t)Q * ccap, cudaMemcpyDeviceToHost, s));
    }
    if (dpath) {
        AUV_TRY(env_pinned(env, 3, sizeof(R) * 6 * (size_t)Q * p->path_cap, &hpath));
        AUV_CUDA(cudaMemcpyAsync(hpath, dpath, sizeof(R) * 6 * (size_t)Q * p->path_cap, cudaMemcpyDeviceToHost, s));
    }
    AUV_CUDA(cudaStreamSynchronize(s));
    memcpy(rec, hrec, sizeof(auvrrt_plan_record_t) * (size_t)Q);
    if (chain) memcpy(chain, hchain, 4 * (size_t)Q * ccap);
    if (dpath) {
        const R *hp2 = (const R *)hpath;
        for (size_t i = 0; i < (size_t)6 * Q * p->path_cap; i++) path[i] = (double)hp2[i];
    }
    if (p->trace) {
        std::vector<R> leaf(n_it * 5);
        AUV_CUDA(cudaMemcpy(leaf.data(), dtr.leaf, n_it * 5 * sizeof(R), cudaMemcpyDeviceToHost));
        if (trace->leaf) for (size_t i = 0; i < n_it * 5; i++) trace->leaf[i] = (double)leaf[i];
        if (trace->upos) AUV_CUDA(cudaMemcpy(trace->upos, dtr.upos, n_it * 8, cudaMemcpyDeviceToHost));
        if (trace->parent) AUV_CUDA(cudaMemcpy(trace->parent, dtr.parent, n_it * 4, cudaMemcpyDeviceToHost));
        if (trace->nwp) AUV_CUDA(cudaMemcpy(trace->nwp, dtr.nwp, n_it * 4, cudaMemcpyDeviceToHost));
        if (trace->safe) AUV_CUDA(cudaMemcpy(trace->safe, dtr.safe, n_it, cudaMemcpyDeviceToHost));
    }
    return AUVRRT_OK;
}
extern "C" int auvrrt_plan_batch(const auvrrt_env_t *env, const double *starts, const uint64_t *seeds, int64_t Q,
                                 const auvrrt_plan_params_t *params, int precision, auvrrt_plan_record_t *out_records,
                                 uint32_t *out_chain, double *out_path, const auvrrt_plan_trace_t *trace) {
    AUV_TRY(check_precision(precision));
    if (!env || !params || !out_records) return set_err(AUVRRT_ERR_ARG, "plan_batch: NULL env, params or out_records");
    AUV_TRY(need_device(env->device));
    if (Q <= 0) return AUVRRT_OK;
    if (!starts || !seeds) return set_err(AUVRRT_ERR_ARG, "plan_batch: NULL starts or seeds");
    auvrrt_env *e = const_cast<auvrrt_env *>(env);
    return AUV_DISPATCH(precision, plan_host, e, starts, seeds, Q, params, out_records, out_chain, out_path, trace);
}

template <typename R>
static int materialize_host(const auvrrt_env *env, const double *starts, const uint64_t *seeds, const uint32_t *chain,
                            const int32_t *depth, int64_t Q, const auvrrt_plan_params_t *p, double *path, int32_t *n_path) {
    const int ccap = p->chain_cap > 0 ? p->chain_cap : 1;
    Staging st;
    const R *ds = st.in_real<R>(starts, 5 * Q);
    const uint64_t *dseed = st.in(seeds, Q);
    const uint32_t *dchain = st.in(chain, Q * ccap);
    const int32_t *ddepth = st.in(depth, Q);
    R *dpath = st.out_real<R>(path, 6 * Q * p->path_cap, true);
    int32_t *dn = st.out(n_path, Q);
    AUV_TRY(st.rc);
    AUV_TRY(launch_materialize<R>(env, ds, dseed, dchain, ddepth, 1, Q, nullptr, Q, p, dpath, dn, 0));
    return st.finish();
}
extern "C" int auvrrt_materialize(const auvrrt_env_t *env, const double *starts, const uint64_t *seeds,
                                  const uint32_t *chain, const int32_t *depth, int64_t Q,
                                  const auvrrt_plan_params_t *params, int precision, double *out_path,
                                  int32_t *out_n_path) {
    AUV_TRY(check_precision(precision));
    if (!env || !params) return set_err(AUVRRT_ERR_ARG, "materialize: NULL env or params");
    AUV_TRY(need_device(env->device));
    if (Q <= 0) return AUVRRT_OK;
    if (params->path_cap < 1) return set_err(AUVRRT_ERR_ARG, "materialize: path_cap must be >= 1");
    if (params->group != 0 && params->group != 32 && params->group != 16 && params->group != 8 && params->group != 1)
        return set_err(AUVRRT_ERR_ARG, "materialize: group must be 32, 16, 8 or 1");
    // a chain holds chain_cap positions: a record of an overflowed plan (depth > chain_cap) cannot be re-created
    if (!starts || !seeds || !chain || !depth || !out_path || !out_n_path) return set_err(AUVRRT_ERR_ARG, "materialize: NULL buffer");
    for (int64_t q = 0; q < Q; q++)
        if (depth[q] < 0 || depth[q] > params->chain_cap)
            return set_err(AUVRRT_ERR_ARG, "materialize: depth[%lld] = %d outside [0, chain_cap = %d]", (long long)q, depth[q],
                           params->chain_cap);
    return AUV_DISPATCH(precision, materialize_host, env, starts, seeds, chain, depth, Q, params, out_path, out_n_path);
}

// ------------------------------------------------------------------ the device end of a planning step
extern "C" int auvrrt_plan_group(const auvrrt_plan_params_t *p, int64_t Q, int with_path) {
    if (!p) { set_err(AUVRRT_ERR_ARG, "plan_group: params is NULL"); return -1; }
    const int G = plan_group(p, Q, with_path != 0);
    return G < 0 ? -1 : G;
}
static int need_a_device() {
    if (auvrrt_device_count() <= 0) return set_err(AUVRRT_ERR_CUDA, "no CUDA device: libauvrrt has no CPU fallback");
    return AUVRRT_OK;
}
extern "C" int auvrrt_plan_best_dev(const auvrrt_plan_record_t *records, int64_t Q, const int64_t *mission_off, int64_t M,
                                    int64_t *out_best, double *out_cost, void *stream) {
    AUV_TRY(need_a_device());
    if (M <= 0) return AUVRRT_OK;
    if (!mission_off || !out_best || !out_cost || (Q > 0 && !records)) return set_err(AUVRRT_ERR_ARG, "plan_best: NULL buffer");
    return launch_plan_best(records, Q, mission_off, M, out_best, out_cost, (cudaStream_t)stream);
}
extern "C" int auvrrt_materialize_dev(const auvrrt_env_t *env, const void *starts, const uint64_t *seeds,
                                      const auvrrt_plan_record_t *records, const uint32_t *chain, int64_t Q,
                                      const int64_t *pick, int64_t M, const auvrrt_plan_params_t *params, int precision,
                                      void *out_path, int32_t *out_n_path, void *stream) {
    AUV_TRY(need_a_device());
    AUV_TRY(check_precision(precision));
    if (!env || !params) return set_err(AUVRRT_ERR_ARG, "materialize_dev: NULL env or params");
    // the evaluator must be the one of the planner that made the chains: group 0 would leave it to a guess
    if (params->group != 32 && params->group != 16 && params->group != 8 && params->group != 1)
        return set_err(AUVRRT_ERR_ARG, "materialize_dev: group must name the planner that ran: 32, 16, 8 or 1 (see auvrrt_plan_group)");
    if (params->path_cap < 1) return set_err(AUVRRT_ERR_ARG, "materialize_dev: path_cap must be >= 1");
    if (M <= 0) return AUVRRT_OK;
    if (!pick || !out_path || !out_n_path || (Q > 0 && (!starts || !seeds || !records || !chain)))
        return set_err(AUVRRT_ERR_ARG, "materialize_dev: NULL buffer");
    const int32_t *depth = records ? &records->depth : nullptr;
    const int stride = (int)(sizeof(auvrrt_plan_record_t) / sizeof(int32_t));
    cudaStream_t s = (cudaStream_t)stream;
    if (precision == AUVRRT_F32)
        return launch_materialize<float>(env, (const float *)starts, seeds, chain, depth, stride, Q, pick, M, params,
                                         (float *)out_path, out_n_path, s);
    return launch_materialize<double>(env, (const double *)starts, seeds, chain, depth, stride, Q, pick, M, params,
                                      (double *)out_path, out_n_path, s);
}

extern "C" int auvrrt_calibrate_fp32(int device, int iters, double *out_flops, double *out_ms) {
    AUV_TRY(need_device(device));
    double f = 0, ms = 0;
    AUV_TRY(launch_calibrate_fp32(iters > 0 ? iters : 4096, &f, &ms));
    if (out_flops) *out_flops = f;
    if (out_ms) *out_ms = ms;
    return AUVRRT_OK;
}
