// c5_exact.cu — per-view kernels whose arithmetic must equal the reference's host code bit for
// bit. This file is compiled with -fmad=false (no FMA contraction), like the reference's plain
// x86-64 -O3 build (CMakeLists.txt:4-7), so that rotated coordinates and the solid (NaN) mask are
// identical to the oracle's, not merely close.
//
//   rotate_vertices  K1: object3d_base::rotate_around_{x,y}_axis (object3d_base.cpp:202-219 ->
//                    tetra.cpp:44-62), once per UNIQUE vertex instead of 12 private points per tet.
//   solid_mask       K5: the solid branch of the face scan conversion (plane.cpp:23-27,57-142,
//                    line.cpp:246-249): union of the inclusive scanline footprints of the faces
//                    of solid tets.
//   bvh_refit        per-view boxes of the boundary-face LBVH (no reference counterpart: it
//                    replaces the full scan conversion plane.cpp:184-192 as the way a ray finds
//                    the tets it crosses).
#include <algorithm>
#include <cstring>

#include "c5_internal.h"

namespace c5 {

namespace {

struct RotSet {
    Rot r[kMaxRot];
    int n;
};

C5_HD void rotate_point(const RotSet& rs, double& x, double& y, double& z) {
    for (int k = 0; k < rs.n; k++) {
        const double c = rs.r[k].c, s = rs.r[k].s;
        if (rs.r[k].axis == 0) { // tetra.cpp:44-48
            const double y0 = y;
            y = y * c - z * s;
            z = y0 * s + z * c;
        } else { // tetra.cpp:51-62
            x -= rs.r[k].x0;
            const double x1 = x;
            x = x * c - z * s;
            z = x1 * s + z * c;
            x += rs.r[k].x0;
        }
    }
}

C5_HD void rotate_vertex_body(int64_t i, const double* px, const double* py, const double* pz, Vtx* out,
                              const RotSet& rs) {
    double x = px[i], y = py[i], z = pz[i];
    rotate_point(rs, x, y, z);
    Vtx v;
    v.x = x;
    v.y = y;
    v.z = z;
    v.w = 0.0;
    out[i] = v;
}

} // namespace

__global__ void __launch_bounds__(256)
rotate_vertices(int64_t n, const double* __restrict__ px, const double* __restrict__ py,
                const double* __restrict__ pz, Vtx* __restrict__ out, RotSet rs) {
    const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
    if (i < n) rotate_vertex_body(i, px, py, pz, out, rs);
}

namespace {

C5_HD void rotate_xyz_body(int64_t i, const double* in, double* out, const RotSet& rs) {
    double x = in[3 * i], y = in[3 * i + 1], z = in[3 * i + 2];
    rotate_point(rs, x, y, z);
    out[3 * i] = x;
    out[3 * i + 1] = y;
    out[3 * i + 2] = z;
}

} // namespace

__global__ void __launch_bounds__(256)
rotate_solid_points(int64_t n, const double* __restrict__ in, double* __restrict__ out, RotSet rs) {
    const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
    if (i < n) rotate_xyz_body(i, in, out, rs);
}

namespace {

// ---- solid mask --------------------------------------------------------------------------------

struct MaskGrid {
    int res_x, res_y;
    double x_min, y_min, step_x, step_y;
    double inv_step_x, inv_step_y; // RN(1 / step), from the host
    const double* ys; // accumulated row coordinates (plane.cpp:304-314)
    uint8_t* mask;
    int row_begin, row_end; // only rows of this band are marked (the walk reads no others)
};

// Correctly rounded n / d from the correctly rounded reciprocal r = RN(1 / d) (Markstein 1990):
//     q0 = RN(n r);  e = n - d q0  (exact in one FMA, q0 being within an ulp of n/d);  q = RN(q0 + e r)
// equals RN(n / d) for normal operands. The scanline loop divides by the same few denominators
// (the pixel pitch, one dy per edge) hundreds of times per face, so one IEEE divide per denominator
// and three FMA-class instructions per quotient replace the ~20-instruction divide sequence — with
// bit-identical results (600 M random and worst-case operand pairs agree with `/`; the masks are
// compared bit for bit with the reference's in tests/).
C5_HD double div_by(double n, double d, double r) {
    const double q0 = n * r;
    const double e = fma(-d, q0, n);
    return fma(e, r, q0);
}

C5_HD double pixel_of_x(const MaskGrid& g, double x) { // plane.cpp:194-202
    const double r = div_by(x - g.x_min, g.step_x, g.inv_step_x);
    const double hi = static_cast<double>(g.res_x) - 1;
    if (r < 0) return 0;
    if (r > hi) return hi;
    return r;
}
C5_HD double pixel_of_y(const MaskGrid& g, double y) { // plane.cpp:204-212
    const double r = div_by(y - g.y_min, g.step_y, g.inv_step_y);
    const double hi = static_cast<double>(g.res_y) - 1;
    if (r < 0) return 0;
    if (r > hi) return hi;
    return r;
}

// x of the edge p1-p2 at height y (plane.cpp:50-55), with dy = p1y - p2y and its reciprocal hoisted
struct EdgeFn {
    double x1, y1, dx, dy, rdy;
    bool flat;
};
C5_HD EdgeFn make_edge(const double* p1, const double* p2) {
    EdgeFn e;
    e.x1 = p1[0];
    e.y1 = p1[1];
    e.dx = p1[0] - p2[0];
    e.dy = p1[1] - p2[1];
    e.flat = fabs(e.dy) < DBL_EPSILON;
    e.rdy = e.flat ? 0.0 : 1.0 / e.dy;
    return e;
}
C5_HD double edge_x(const EdgeFn& e, double y) {
    if (e.flat) return e.x1;
    return div_by(e.dx * (y - e.y1), e.dy, e.rdy) + e.x1;
}

// Sets the bytes [p, e) to 1; the aligned middle of the span goes eight pixels at a time (concurrent
// writers only ever write ones, so a wide store inside the span cannot lose anything). Write-only: a
// test-before-store saved redundant stores while every fan face drew its whole footprint, but it makes
// every pixel a dependent load (ncu, pass 1: 61 long-scoreboard stall cycles per issued instruction);
// since the tile flags the rows that are still drawn are few and stores are fire-and-forget.
C5_HD void mark_span(uint8_t* p, uint8_t* e) {
    while (p < e && (reinterpret_cast<uintptr_t>(p) & 7u)) *p++ = 1;
    for (; p + 8 <= e; p += 8) *reinterpret_cast<unsigned long long*>(p) = 0x0101010101010101ull;
    while (p < e) *p++ = 1;
}

// Everything the scan conversion of one projected triangle derives from its three points before the
// row loop (plane.cpp:57-100): y-sorted vertices, the rows of the band the triangle reaches, which
// side the long edge is on and the three edge functions.
struct FaceScan {
    double p1x, p1y; // the middle vertex
    EdgeFn e_long, e_low, e_up;
    bool long_edge_is_left;
    long long j_lo, j_hi; // empty if j_lo > j_hi
};

// First half of the setup: the vertices in y-descending order and the rows of the band the triangle
// reaches. Faces outside the band, and tall faces in the listing pass, stop here.
struct FaceRows {
    const double *p0, *p1, *p2;
    long long j_lo, j_hi;
};

C5_HD FaceRows scan_rows(const MaskGrid& g, const double* a, const double* b, const double* c) {
    FaceRows R;
    R.p0 = a;
    R.p1 = b;
    R.p2 = c;
    const double* t;
    // y-descending with the tie order of a stable insertion sort (std::sort on 3 items, plane.cpp:61)
    if (R.p1[1] > R.p0[1]) { t = R.p0; R.p0 = R.p1; R.p1 = t; }
    if (R.p2[1] > R.p0[1]) { t = R.p2; R.p2 = R.p1; R.p1 = R.p0; R.p0 = t; }
    else if (R.p2[1] > R.p1[1]) { t = R.p1; R.p1 = R.p2; R.p2 = t; }
    R.j_hi = static_cast<long long>(floor(pixel_of_y(g, R.p0[1])));
    R.j_lo = static_cast<long long>(ceil(pixel_of_y(g, R.p2[1])));
    if (R.j_lo < g.row_begin) R.j_lo = g.row_begin;
    if (R.j_hi > g.row_end - 1) R.j_hi = g.row_end - 1;
    return R;
}

// Second half: which side the long edge is on and the three edge functions (a divide each).
C5_HD FaceScan scan_edges(const FaceRows& R) {
    const double *p0 = R.p0, *p1 = R.p1, *p2 = R.p2;
    // which side of the long edge p0-p2 the middle vertex lies on (plane.cpp:46-48,66-89)
    const double rel = (p2[1] - p0[1]) * p1[0] + (p0[0] - p2[0]) * p1[1] + (p2[0] * p0[1] - p0[0] * p2[1]);
    const bool asc_above = (p0[0] >= p2[0]) && (rel >= 0);
    const bool des_below = (p0[0] < p2[0]) && (rel > 0);
    FaceScan S;
    S.long_edge_is_left = !(asc_above || des_below);
    S.j_lo = R.j_lo;
    S.j_hi = R.j_hi;
    S.p1x = p1[0];
    S.p1y = p1[1];
    S.e_long = make_edge(p0, p2);
    S.e_low = make_edge(p2, p1);
    S.e_up = make_edge(p0, p1);
    return S;
}

// The two ends of the triangle's footprint at height y (plane.cpp:101-137), unrounded.
C5_HD void scan_ends(const FaceScan& S, double y, double& x_lo, double& x_hi) {
    const double x_long = edge_x(S.e_long, y);
    const double x_short = (y < S.p1y) ? edge_x(S.e_low, y) : edge_x(S.e_up, y);
    x_lo = S.long_edge_is_left ? x_long : x_short;
    x_hi = S.long_edge_is_left ? x_short : x_long;
}

C5_HD void scan_row(const MaskGrid& g, const FaceScan& S, long long j) {
    const double y = g.ys[j]; // == ys[j_lo] + (j - j_lo) additions of step_y (plane.cpp:100,138)
    double x_lo, x_hi;
    scan_ends(S, y, x_lo, x_hi);
    const long long i_hi = static_cast<long long>(floor(pixel_of_x(g, x_hi)));
    const long long i_lo = static_cast<long long>(ceil(pixel_of_x(g, x_lo)));
    uint8_t* row = g.mask + static_cast<size_t>(j) * g.res_x;
    if (i_lo <= i_hi) mark_span(row + i_lo, row + i_hi + 1);
}

// ---- tall faces ------------------------------------------------------------------------------------
// The reference's solids are fans of tets around a centre (object3d_base.cpp:156-193): two thirds of
// their faces run from the centre to a surface edge — slivers a pixel or two wide and a hundred rows
// tall, almost all of it under pixels the small surface faces have marked already. Marking is
// idempotent, so a face may skip any stretch of rows whose footprint is PROVEN marked: the mask is cut
// into tiles of kTileW x kTileH pixels with one flag per tile ("every pixel of the tile that lies in
// the band is solid"), built after the small faces have been drawn. A tall face walks its rows one
// tile row at a time; the footprint of a triangle over a range of rows is bounded by its ends at the
// first and the last of those rows and by the middle vertex, so four edge evaluations decide whether
// all tiles under it are full — against two per row plus the stores otherwise. What is skipped is
// only ever marked already, so the mask stays bit-identical to the reference's.
constexpr int kTileW = 16, kTileH = 8; // default tile: 16 x 8 and 16 x 4 measured best, smaller tiles slower (profiles/r02_exp_mask_tile_sizes.jsonl); (c5_debug_set "mask_tile" = 100 w + h overrides, for experiments)
constexpr int kSmallRows = 8; // faces of at most this many rows are drawn at once, by one thread

struct TileGrid {
    uint8_t* full; // [tiles_y][tiles_x]
    int tiles_x, tiles_y;
    int w, h;      // tile size in pixels (w a multiple of 8)
};

// Whether every pixel under face S in tile row c is PROVEN marked; [ja, jb] = the rows of S in that tile row.
C5_HD bool tile_row_covered(const MaskGrid& g, const TileGrid& tg, const FaceScan& S, long long c, long long& ja, long long& jb) {
    ja = c * tg.h > S.j_lo ? c * tg.h : S.j_lo;
    jb = c * tg.h + tg.h - 1 < S.j_hi ? c * tg.h + tg.h - 1 : S.j_hi;
    const double ya = g.ys[ja], yb = g.ys[jb];
    double lo_a, hi_a, lo_b, hi_b;
    scan_ends(S, ya, lo_a, hi_a);
    scan_ends(S, yb, lo_b, hi_b);
    double x_min = fmin(fmin(lo_a, hi_a), fmin(lo_b, hi_b));
    double x_max = fmax(fmax(lo_a, hi_a), fmax(lo_b, hi_b));
    if (S.p1y >= ya && S.p1y <= yb) { // the short edge changes inside the range: its corner may stick out
        x_min = fmin(x_min, S.p1x);
        x_max = fmax(x_max, S.p1x);
    }
    bool covered = x_min == x_min && x_max == x_max; // (never skip on a NaN)
    if (covered) {
        // two pixels of margin each way: edge_x is monotone in y only up to its rounding
        long long i_a = static_cast<long long>(floor(pixel_of_x(g, x_min))) - 2;
        long long i_b = static_cast<long long>(ceil(pixel_of_x(g, x_max))) + 2;
        if (i_a < 0) i_a = 0;
        if (i_b > g.res_x - 1) i_b = g.res_x - 1;
        const uint8_t* flags = tg.full + c * tg.tiles_x;
        for (long long t = i_a / tg.w; t <= i_b / tg.w && covered; t++) covered = flags[t] != 0;
    }
    return covered;
}

// face f of a solid tet: 0 = (v0,v1,v2), 1 = (v0,v1,v3), 2 = (v0,v2,v3), 3 = (v1,v2,v3) (plane.cpp:30-37)
C5_HD void face_corners(int64_t f, const double* pts, const double*& a, const double*& b, const double*& c) {
    const double* p = pts + 12 * (f >> 2);
    const int k = static_cast<int>(f & 3);
    a = p + (k == 3 ? 3 : 0);
    b = p + (k >= 2 ? 6 : 3);
    c = p + (k == 0 ? 6 : 9);
}

// pass 2 for one tile
C5_HD void tile_flag_body(int ty, int tx, const MaskGrid& g, const TileGrid& tg) {
    const int j0 = ty * tg.h > g.row_begin ? ty * tg.h : g.row_begin;
    const int j1 = ty * tg.h + tg.h < g.row_end ? ty * tg.h + tg.h : g.row_end;
    const int i0 = tx * tg.w, i1 = i0 + tg.w < g.res_x ? i0 + tg.w : g.res_x;
    bool all = true;
    for (int j = j0; j < j1 && all; j++) {
        const uint8_t* row = g.mask + static_cast<size_t>(j) * g.res_x;
        if (i1 - i0 == tg.w && (reinterpret_cast<uintptr_t>(row + i0) & 7u) == 0) {
            const unsigned long long* w = reinterpret_cast<const unsigned long long*>(row + i0);
            for (int k = 0; k < tg.w / 8; k++) all = all && w[k] == 0x0101010101010101ull;
        } else {
            for (int i = i0; i < i1; i++) all = all && row[i] != 0;
        }
    }
    tg.full[static_cast<size_t>(ty) * tg.tiles_x + tx] = all ? 1 : 0;
}

// ---- a warp's 32 faces, shared ---------------------------------------------------------------------
// One face per thread leaves most lanes idle: faces differ in height by two orders of magnitude, two
// thirds of a pass-1 warp hold faces that are only listed, and the rare tile row that does have to be
// drawn stalls the other 31 lanes (ncu, per-face kernels: 7.5 of 32 lanes active on the Roche lobe,
// profiles/r02_mask_*). So a warp sets up its 32 faces one per lane, parks the FaceScans in shared
// memory and deals out the ITEMS (rows in pass 1, tile rows in pass 3, rows of uncovered tile rows in
// its drain) lane by lane, whoever the face belongs to. The arithmetic per item is the same
// functions on the same operands whichever lane runs it, so the mask cannot differ.
#define C5_HDN __host__ __device__ // (not force-inlined, unlike C5_HD)
constexpr int kFaceFields = 17; // p1x p1y + 3 x {x1 y1 dx dy rdy}
struct WarpFaces {
    double f[kFaceFields][32];
    int j_lo[32], j_hi[32], bits[32]; // bits: flat (long, low, up), long_edge_is_left
    int first[32];                    // items of the faces of the lower lanes (exclusive prefix sum)
    int c_lo[32];                     // pass 3: first tile row of the face
    int list[64][2];                  // pass 3: (lane of the face, tile row) still to be drawn
};

C5_HDN void wf_store_edge(WarpFaces& w, int at, int lane, const EdgeFn& e) {
    w.f[at][lane] = e.x1;
    w.f[at + 1][lane] = e.y1;
    w.f[at + 2][lane] = e.dx;
    w.f[at + 3][lane] = e.dy;
    w.f[at + 4][lane] = e.rdy;
}
C5_HDN EdgeFn wf_load_edge(const WarpFaces& w, int at, int o, bool flat) {
    EdgeFn e;
    e.x1 = w.f[at][o];
    e.y1 = w.f[at + 1][o];
    e.dx = w.f[at + 2][o];
    e.dy = w.f[at + 3][o];
    e.rdy = w.f[at + 4][o];
    e.flat = flat;
    return e;
}
C5_HDN void wf_store(WarpFaces& w, int lane, const FaceScan& S) {
    w.f[0][lane] = S.p1x;
    w.f[1][lane] = S.p1y;
    wf_store_edge(w, 2, lane, S.e_long);
    wf_store_edge(w, 7, lane, S.e_low);
    wf_store_edge(w, 12, lane, S.e_up);
    w.j_lo[lane] = static_cast<int>(S.j_lo);
    w.j_hi[lane] = static_cast<int>(S.j_hi);
    w.bits[lane] = (S.e_long.flat ? 1 : 0) | (S.e_low.flat ? 2 : 0) | (S.e_up.flat ? 4 : 0) | (S.long_edge_is_left ? 8 : 0);
}
C5_HDN FaceScan wf_load(const WarpFaces& w, int o) {
    FaceScan S;
    const int bits = w.bits[o];
    S.p1x = w.f[0][o];
    S.p1y = w.f[1][o];
    S.e_long = wf_load_edge(w, 2, o, bits & 1);
    S.e_low = wf_load_edge(w, 7, o, bits & 2);
    S.e_up = wf_load_edge(w, 12, o, bits & 4);
    S.long_edge_is_left = bits & 8;
    S.j_lo = w.j_lo[o];
    S.j_hi = w.j_hi[o];
    return S;
}

// Exclusive prefix sum of n over the warp, left in w.first; returns the total.
__device__ int wf_deal(WarpFaces& w, int lane, int n) {
    int incl = n;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int up = __shfl_up_sync(0xFFFFFFFFu, incl, d);
        if (lane >= d) incl += up;
    }
    w.first[lane] = incl - n;
    __syncwarp();
    return __shfl_sync(0xFFFFFFFFu, incl, 31);
}
// The lane whose face item i belongs to: the LAST lane with first <= i (lanes without items share
// their `first` with the next lane that has some, and that one is the later of them).
C5_HDN int wf_owner(const WarpFaces& w, int i) {
    int o = 0;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        if (w.first[o + d] <= i) o += d;
    }
    return o;
}

} // namespace

constexpr int kMaskWarps = 4; // warps per block of the two face passes (5.6 KB of shared memory each)

// Pass 1: faces that do not reach the band cost their row range and nothing else; tall ones are appended
// to `tall` (one atomic per warp); the rows of the small ones are dealt out over the warp and drawn.
__global__ void __launch_bounds__(32 * kMaskWarps)
solid_mask_small(int64_t n_faces, const uint32_t* __restrict__ faces, const double* __restrict__ pts, MaskGrid g,
                 uint32_t* __restrict__ tall, unsigned* n_tall) {
    __shared__ WarpFaces shared[kMaskWarps];
    WarpFaces& w = shared[threadIdx.x >> 5];
    const unsigned full = 0xFFFFFFFFu;
    const int lane = threadIdx.x & 31;
    const int64_t k = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
    uint32_t f = 0;
    bool is_tall = false;
    int rows = 0;
    if (k < n_faces) {
        f = faces[k];
        const double *a, *b, *c;
        face_corners(f, pts, a, b, c);
        const FaceRows R = scan_rows(g, a, b, c);
        if (R.j_lo <= R.j_hi) {
            if (R.j_hi - R.j_lo >= kSmallRows) {
                is_tall = true;
            } else {
                wf_store(w, lane, scan_edges(R));
                rows = static_cast<int>(R.j_hi - R.j_lo) + 1;
            }
        }
    }
    const unsigned m = __ballot_sync(full, is_tall);
    if (m) {
        unsigned base = 0;
        if (lane == 0) base = atomicAdd(n_tall, static_cast<unsigned>(__popc(m)));
        base = __shfl_sync(full, base, 0);
        if (is_tall) tall[base + __popc(m & ((1u << lane) - 1u))] = f;
    }
    const int total = wf_deal(w, lane, rows);
    for (int i = lane; i < total; i += 32) {
        const int o = wf_owner(w, i);
        const FaceScan S = wf_load(w, o);
        scan_row(g, S, S.j_lo + (i - w.first[o]));
    }
}

// Pass 3: the tall faces. The tile rows of a warp's 32 faces are dealt out over its lanes; a tile row that
// is not proven solid goes to a short list, and the list's ROWS are dealt out in turn.
__global__ void __launch_bounds__(32 * kMaskWarps)
solid_mask_tall(const uint32_t* __restrict__ tall, const unsigned* __restrict__ n_tall, const double* __restrict__ pts,
                MaskGrid g, TileGrid tg) {
    __shared__ WarpFaces shared[kMaskWarps];
    WarpFaces& w = shared[threadIdx.x >> 5];
    const unsigned full = 0xFFFFFFFFu;
    const int lane = threadIdx.x & 31;
    const unsigned n = *n_tall;
    auto drain = [&](int n_list) {
        __syncwarp();
        for (int k = lane; k < n_list * tg.h; k += 32) {
            const int e = k / tg.h;
            const int o = w.list[e][0];
            const long long j = static_cast<long long>(w.list[e][1]) * tg.h + k % tg.h;
            if (j >= w.j_lo[o] && j <= w.j_hi[o]) scan_row(g, wf_load(w, o), j);
        }
        __syncwarp();
    };
    for (unsigned base = (blockIdx.x * kMaskWarps + (threadIdx.x >> 5)) * 32u; base < n; base += gridDim.x * kMaskWarps * 32u) {
        int items = 0;
        if (base + lane < n) {
            const double *a, *b, *c;
            face_corners(tall[base + lane], pts, a, b, c);
            const FaceRows R = scan_rows(g, a, b, c);
            if (R.j_lo <= R.j_hi) {
                wf_store(w, lane, scan_edges(R));
                w.c_lo[lane] = static_cast<int>(R.j_lo / tg.h);
                items = static_cast<int>(R.j_hi / tg.h - R.j_lo / tg.h) + 1;
            }
        }
        const int total = wf_deal(w, lane, items);
        int n_list = 0;
        for (int at = 0; at < total; at += 32) {
            const int i = at + lane;
            bool draw = false;
            int o = 0, c = 0;
            if (i < total) {
                o = wf_owner(w, i);
                c = w.c_lo[o] + (i - w.first[o]);
                long long ja, jb;
                draw = !tile_row_covered(g, tg, wf_load(w, o), c, ja, jb);
            }
            const unsigned m = __ballot_sync(full, draw);
            if (m) {
                if (n_list + __popc(m) > 64) {
                    drain(n_list);
                    n_list = 0;
                }
                if (draw) {
                    const int at_list = n_list + __popc(m & ((1u << lane) - 1u));
                    w.list[at_list][0] = o;
                    w.list[at_list][1] = c;
                }
                n_list += __popc(m);
            }
        }
        drain(n_list); // (also fences this batch's FaceScans against the next one's stores)
    }
}

// Pass 2: one thread per tile of the band.
__global__ void __launch_bounds__(256) mask_tile_flags(MaskGrid g, TileGrid tg, int tile_row_begin, int tile_row_end) {
    const int64_t k = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
    const int64_t n = static_cast<int64_t>(tile_row_end - tile_row_begin) * tg.tiles_x;
    if (k >= n) return;
    tile_flag_body(tile_row_begin + static_cast<int>(k / tg.tiles_x), static_cast<int>(k % tg.tiles_x), g, tg);
}

namespace {

// ---- unique solid faces (once per upload) --------------------------------------------------------
// The reference's solids are fans of tets around a centre (object3d_base.cpp:156-193): every fan
// face belongs to two tets and would be scan-converted twice. Faces are compared on the exact bit
// patterns of their three points (order-independent), so dropping a duplicate cannot change the mask.
C5_HD void face_points(const double* pts, uint32_t f, const double*& a, const double*& b, const double*& c) {
    const double* p = pts + 12 * static_cast<size_t>(f >> 2);
    const int k = static_cast<int>(f & 3);
    a = p + (k == 3 ? 3 : 0);
    b = p + (k >= 2 ? 6 : 3);
    c = p + (k == 0 ? 6 : 9);
}
C5_HD bool point_less(const double* u, const double* v) {
    if (u[0] != v[0]) return u[0] < v[0];
    if (u[1] != v[1]) return u[1] < v[1];
    return u[2] < v[2];
}
C5_HD void sorted_face(const double* pts, uint32_t f, const double* out[3]) {
    face_points(pts, f, out[0], out[1], out[2]);
    const double* t;
    if (point_less(out[1], out[0])) { t = out[0]; out[0] = out[1]; out[1] = t; }
    if (point_less(out[2], out[1])) { t = out[1]; out[1] = out[2]; out[2] = t; }
    if (point_less(out[1], out[0])) { t = out[0]; out[0] = out[1]; out[1] = t; }
}
C5_HD uint64_t mix64(uint64_t z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
C5_HD uint64_t double_bits(double v) {
#ifdef __CUDA_ARCH__
    return static_cast<uint64_t>(__double_as_longlong(v));
#else
    uint64_t b;
    memcpy(&b, &v, sizeof(b));
    return b;
#endif
}

struct SolidFaceKeyOp {
    const double* pts;
    uint64_t* keys;
    uint32_t* vals;
    C5_HD void operator()(int64_t f) const {
        const double* p[3];
        sorted_face(pts, static_cast<uint32_t>(f), p);
        uint64_t h = 0;
        for (int i = 0; i < 3; i++) {
            for (int c = 0; c < 3; c++) h = mix64(h ^ double_bits(p[i][c]));
        }
        keys[f] = h;
        vals[f] = static_cast<uint32_t>(f);
    }
};

struct SolidFaceFirstOp {
    const double* pts;
    const uint64_t* keys; // sorted
    const uint32_t* vals;
    uint8_t* first;
    C5_HD void operator()(int64_t i) const {
        bool dup = false;
        if (i > 0 && keys[i] == keys[i - 1]) {
            const double *p[3], *q[3];
            sorted_face(pts, vals[i], p);
            sorted_face(pts, vals[i - 1], q);
            dup = true;
            for (int k = 0; k < 3; k++) {
                for (int c = 0; c < 3; c++) dup = dup && double_bits(p[k][c]) == double_bits(q[k][c]);
            }
        }
        first[i] = dup ? 0 : 1;
    }
};

struct WidenU32Op {
    const uint32_t* src;
    uint64_t* out;
    C5_HD void operator()(int64_t i) const { out[i] = src[i]; }
};
struct GatherU32Op {
    const uint32_t* src;
    const uint32_t* idx;
    uint32_t* out;
    C5_HD void operator()(int64_t i) const { out[i] = src[idx[i]]; }
};

} // namespace

namespace {

// ---- BVH refit ---------------------------------------------------------------------------------

C5_HD void store_child_box(BvhNode* nodes, int32_t link, float xlo, float xhi, float ylo, float yhi, float zlo,
                           float zhi) {
    BvhNode& n = nodes[link >> 1];
    const int w = link & 1;
    n.xlo[w] = xlo;
    n.xhi[w] = xhi;
    n.ylo[w] = ylo;
    n.yhi[w] = yhi;
    n.zlo[w] = zlo;
    n.zhi[w] = zhi;
}

C5_HD float load_f(const float* p) {
#ifdef __CUDA_ARCH__
    return __ldcg(p); // L2: the sibling's box was written by another SM
#else
    return *p;
#endif
}

// One thread per leaf. A boundary face can only be an ENTRY face for rays travelling +z if its
// outward normal has n_z < 0; the others get an empty box, which prunes them (and every subtree
// made only of them) from all queries of this view.
C5_HD void refit_leaf_body(int64_t leaf, const BFace* faces, const Vtx* vrot, BvhNode* nodes,
                           const int32_t* node_parent, const int32_t* leaf_parent, uint32_t* flags) {
    const BFace f = faces[leaf];
    const Vtx a = vrot[f.a], b = vrot[f.b], c = vrot[f.c];
    const double nz = (b.x - a.x) * (c.y - a.y) - (b.y - a.y) * (c.x - a.x);
    float xlo = INFINITY, xhi = -INFINITY, ylo = INFINITY, yhi = -INFINITY, zlo = INFINITY, zhi = -INFINITY;
    if (nz < 0) {
        xlo = f_round_down(fmin(a.x, fmin(b.x, c.x)));
        xhi = f_round_up(fmax(a.x, fmax(b.x, c.x)));
        ylo = f_round_down(fmin(a.y, fmin(b.y, c.y)));
        yhi = f_round_up(fmax(a.y, fmax(b.y, c.y)));
        zlo = f_round_down(fmin(a.z, fmin(b.z, c.z)));
        zhi = f_round_up(fmax(a.z, fmax(b.z, c.z)));
    }
    int32_t link = leaf_parent[leaf];
    while (true) {
        store_child_box(nodes, link, xlo, xhi, ylo, yhi, zlo, zhi);
        const int32_t node = link >> 1;
#ifdef __CUDA_ARCH__
        __threadfence();
        const uint32_t arrived = atomicAdd(&flags[node], 1u);
#else
        const uint32_t arrived = flags[node]++;
#endif
        if (arrived == 0) return; // the sibling subtree is not done yet; its last thread continues
#ifdef __CUDA_ARCH__
        __threadfence();
#endif
        link = node_parent[node];
        if (link < 0) return; // root
        const BvhNode& n = nodes[node];
        xlo = fminf(load_f(&n.xlo[0]), load_f(&n.xlo[1]));
        xhi = fmaxf(load_f(&n.xhi[0]), load_f(&n.xhi[1]));
        ylo = fminf(load_f(&n.ylo[0]), load_f(&n.ylo[1]));
        yhi = fmaxf(load_f(&n.yhi[0]), load_f(&n.yhi[1]));
        zlo = fminf(load_f(&n.zlo[0]), load_f(&n.zlo[1]));
        zhi = fmaxf(load_f(&n.zhi[0]), load_f(&n.zhi[1]));
    }
}

} // namespace

__global__ void __launch_bounds__(256)
bvh_refit(int64_t n_leaves, const BFace* __restrict__ faces, const Vtx* __restrict__ vrot, BvhNode* nodes,
          const int32_t* __restrict__ node_parent, const int32_t* __restrict__ leaf_parent, uint32_t* flags) {
    const int64_t leaf = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
    if (leaf < n_leaves) refit_leaf_body(leaf, faces, vrot, nodes, node_parent, leaf_parent, flags);
}

namespace {

// Source function s = Q / min(alpha, limit) of one cell or channel, Q read from q[k]. Channel renders
// are bitwise equal to plain renders because cells and channels both get s from here.
C5_HD double source_fn(double alpha, const double* q, int64_t k, double limit) {
    if (alpha > limit) alpha = limit;         // line.cpp:216-218
    // alpha^ < DBL_EPSILON leaves I unchanged (line.cpp:221); the walk tests alpha itself, s is unused
    return (alpha < DBL_EPSILON) ? 0.0 : q[k] / alpha;
}

C5_HD void prepare_cell_body(int64_t t, Fields* fields, const double* q0, double limit) {
    fields[t].s = source_fn(fields[t].alpha, q0, t, limit);
}

// Channel c of tet t (k = t * n + c): s_c from ch_q0[c][t] and the alpha_c beside it in the record.
C5_HD void prepare_channel_body(int64_t k, double* rec, const double* q0, int64_t n_tets, int n, double limit) {
    const int64_t t = k / n;
    const int c = static_cast<int>(k - t * n);
    double* r = rec + t * channel_stride(n) + 2 * c;
    r[1] = source_fn(r[0], q0 + c * n_tets, t, limit);
}

} // namespace

// Source function s = Q / min(alpha, limit) per cell; rerun only when --alpha_limit changes.
__global__ void __launch_bounds__(256)
prepare_cells(int64_t n, Fields* __restrict__ fields, const double* __restrict__ q0, double limit) {
    const int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
    if (t < n) prepare_cell_body(t, fields, q0, limit);
}

// The same for the uploaded channels (n_tets * n_channels records).
__global__ void __launch_bounds__(256)
prepare_channels(int64_t n_tets, int n_channels, double* __restrict__ rec, const double* __restrict__ q0, double limit) {
    const int64_t k = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
    if (k < n_tets * n_channels) prepare_channel_body(k, rec, q0, n_tets, n_channels, limit);
}

namespace {

RotSet make_rotset(const Rot* rot, int n_rot) {
    RotSet rs;
    rs.n = n_rot;
    for (int k = 0; k < kMaxRot; k++) rs.r[k] = k < n_rot ? rot[k] : Rot{0, 0, 1.0, 0.0, 0.0};
    return rs;
}

unsigned grid_for(int64_t n, int block) {
    return static_cast<unsigned>((n + block - 1) / block);
}

} // namespace

void launch_rotate_vertices(DeviceState& d, const Rot* rot, int n_rot) {
    const RotSet rs = make_rotset(rot, n_rot);
    count_launch();
    if (kHostSim) {
        for (int64_t i = 0; i < d.n_pts; i++) rotate_vertex_body(i, d.px.p, d.py.p, d.pz.p, d.vrot.p, rs);
        return;
    }
    rotate_vertices<<<grid_for(d.n_pts, 256), 256, 0, d.stream>>>(d.n_pts, d.px.p, d.py.p, d.pz.p, d.vrot.p, rs);
    C5_CUDA(cudaGetLastError());
}

void launch_rotate_solids(DeviceState& d, const Rot* rot, int n_rot) {
    SolidSet& ss = d.solid_follow;
    if (ss.n == 0) return;
    const RotSet rs = make_rotset(rot, n_rot);
    const int64_t n = ss.n * 4;
    count_launch();
    if (kHostSim) {
        for (int64_t i = 0; i < n; i++) rotate_xyz_body(i, ss.pts0.p, ss.pts_view.p, rs);
        return;
    }
    rotate_solid_points<<<grid_for(n, 256), 256, 0, d.stream>>>(n, ss.pts0.p, ss.pts_view.p, rs);
    C5_CUDA(cudaGetLastError());
}

namespace {

// The three passes over the faces of `ss`, into g.mask (which may hold marks already; they only help).
void mask_passes(DeviceState& d, SolidSet& ss, const MaskGrid& g, const TileGrid& tg) {
    if (ss.n == 0) return;
    d.mask_tall.ensure(static_cast<size_t>(std::max(d.solid_follow.n_faces, d.solid_static.n_faces)));
    d.mask_counts.ensure(1);
    dev_zero(d.mask_counts.p, sizeof(unsigned), d.stream);
    const int ty0 = g.row_begin / tg.h, ty1 = (g.row_end + tg.h - 1) / tg.h;
    if (kHostSim) {
        // The same three passes on the host, organised the way the kernels are: 32 faces at a time in a
        // WarpFaces, their items dealt out one by one (wf_owner / wf_load), uncovered tile rows through the
        // 64-entry list and its drain. What the CPU tests cannot reach is only the warp plumbing itself
        // (shuffles, ballots); the item -> (face, row) arithmetic is the kernels' own.
        static WarpFaces w;
        count_launch();
        unsigned& n_tall = d.mask_counts.p[0];
        for (int64_t base = 0; base < ss.n_faces; base += 32) {
            int total = 0;
            for (int lane = 0; lane < 32; lane++) {
                int rows = 0;
                if (base + lane < ss.n_faces) {
                    const uint32_t f = ss.faces.p[base + lane];
                    const double *a, *b, *c;
                    face_corners(f, ss.pts_view.p, a, b, c);
                    const FaceRows R = scan_rows(g, a, b, c);
                    if (R.j_lo <= R.j_hi) {
                        if (R.j_hi - R.j_lo >= kSmallRows) {
                            d.mask_tall.p[n_tall++] = f;
                        } else {
                            wf_store(w, lane, scan_edges(R));
                            rows = static_cast<int>(R.j_hi - R.j_lo) + 1;
                        }
                    }
                }
                w.first[lane] = total;
                total += rows;
            }
            for (int i = 0; i < total; i++) {
                const int o = wf_owner(w, i);
                const FaceScan S = wf_load(w, o);
                scan_row(g, S, S.j_lo + (i - w.first[o]));
            }
        }
        count_launch();
        for (int ty = ty0; ty < ty1; ty++) {
            for (int tx = 0; tx < tg.tiles_x; tx++) tile_flag_body(ty, tx, g, tg);
        }
        count_launch();
        auto drain = [&](int n_list) {
            for (int k = 0; k < n_list * tg.h; k++) {
                const int e = k / tg.h;
                const int o = w.list[e][0];
                const long long j = static_cast<long long>(w.list[e][1]) * tg.h + k % tg.h;
                if (j >= w.j_lo[o] && j <= w.j_hi[o]) scan_row(g, wf_load(w, o), j);
            }
        };
        for (unsigned base = 0; base < n_tall; base += 32) {
            int total = 0;
            for (int lane = 0; lane < 32; lane++) {
                int items = 0;
                if (base + lane < n_tall) {
                    const double *a, *b, *c;
                    face_corners(d.mask_tall.p[base + lane], ss.pts_view.p, a, b, c);
                    const FaceRows R = scan_rows(g, a, b, c);
                    if (R.j_lo <= R.j_hi) {
                        wf_store(w, lane, scan_edges(R));
                        w.c_lo[lane] = static_cast<int>(R.j_lo / tg.h);
                        items = static_cast<int>(R.j_hi / tg.h - R.j_lo / tg.h) + 1;
                    }
                }
                w.first[lane] = total;
                total += items;
            }
            int n_list = 0;
            for (int at = 0; at < total; at += 32) {   // one round of the warp: 32 items, then the list bookkeeping
                int found[32][2], m = 0;
                for (int i = at; i < total && i < at + 32; i++) {
                    const int o = wf_owner(w, i);
                    const int c = w.c_lo[o] + (i - w.first[o]);
                    long long ja, jb;
                    if (!tile_row_covered(g, tg, wf_load(w, o), c, ja, jb)) {
                        found[m][0] = o;
                        found[m][1] = c;
                        m++;
                    }
                }
                if (m) {
                    if (n_list + m > 64) {
                        drain(n_list);
                        n_list = 0;
                    }
                    for (int k = 0; k < m; k++) {
                        w.list[n_list + k][0] = found[k][0];
                        w.list[n_list + k][1] = found[k][1];
                    }
                    n_list += m;
                }
            }
            drain(n_list);
        }
        return;
    }
    if (d.sm_count == 0) C5_CUDA(cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, d.device));
    constexpr int kBlock = 32 * kMaskWarps;
    // pass 1: small faces are drawn, tall ones listed
    count_launch();
    prefer_side_carveout(solid_mask_small, d.device);
    solid_mask_small<<<grid_for(ss.n_faces, kBlock), kBlock, 0, d.stream>>>(ss.n_faces, ss.faces.p, ss.pts_view.p, g,
                                                                             d.mask_tall.p, d.mask_counts.p);
    C5_CUDA(cudaGetLastError());
    // pass 2: which tiles of the band are solid already
    count_launch();
    mask_tile_flags<<<grid_for(static_cast<int64_t>(ty1 - ty0) * tg.tiles_x, 256), 256, 0, d.stream>>>(g, tg, ty0, ty1);
    C5_CUDA(cudaGetLastError());
    // pass 3: tall faces, skipping tile rows that are solid already
    count_launch();
    prefer_side_carveout(solid_mask_tall, d.device);
    solid_mask_tall<<<static_cast<unsigned>(d.sm_count) * 16u, kBlock, 0, d.stream>>>(d.mask_tall.p, d.mask_counts.p,
                                                                                      ss.pts_view.p, g, tg);
    C5_CUDA(cudaGetLastError());
}

} // namespace

// The solid mask of rows [row_begin, row_end) of the view, in d.mask.
//
// Solids that do not follow the view (the reference's accretor sphere is never rotated, main.cpp:116)
// have the same footprint in every view of a sweep: their mask depends on the pixel grid alone. It is
// scan-converted ONCE per (resolution, window, upload) for the whole image into d.mask_static, and a view
// starts from a copy of its band of it instead of from zeros; only the solids that follow the view
// are scan-converted per view. Marks are ones OR-ed together, so the order cannot matter.
void launch_solid_mask(DeviceState& d, int res_x, int res_y, double x_min, double y_min, double step_x,
                       double step_y, int row_begin, int row_end) {
    MaskGrid g{res_x, res_y, x_min, y_min, step_x, step_y, 1.0 / step_x, 1.0 / step_y, d.ys.p, d.mask.p, row_begin, row_end};
    int tile_w = kTileW, tile_h = kTileH;
    if (d.opt_mask_tile > 0) {
        tile_w = std::max(8, (d.opt_mask_tile / 100) & ~7);
        tile_h = std::max(1, d.opt_mask_tile % 100);
    }
    TileGrid tg{nullptr, (res_x + tile_w - 1) / tile_w, (res_y + tile_h - 1) / tile_h, tile_w, tile_h};
    d.mask_tiles.ensure(static_cast<size_t>(tg.tiles_x) * tg.tiles_y);
    tg.full = d.mask_tiles.p;
    const size_t n_pix = static_cast<size_t>(res_x) * res_y;
    uint8_t* band = d.mask.p + static_cast<size_t>(row_begin) * res_x;
    const size_t band_bytes = static_cast<size_t>(row_end - row_begin) * res_x;
    if (d.solid_static.n > 0 && !d.opt_no_static_mask) {
        StaticMaskKey key{res_x, res_y, x_min, y_min, step_x, step_y};
        if (!d.mask_static_valid || std::memcmp(&key, &d.mask_static_key, sizeof(key)) != 0) {
            d.mask_static.ensure(n_pix);
            dev_zero(d.mask_static.p, n_pix, d.stream);
            MaskGrid gs = g;
            gs.mask = d.mask_static.p;
            gs.row_begin = 0;
            gs.row_end = res_y;
            mask_passes(d, d.solid_static, gs, tg);
            d.mask_static_key = key;
            d.mask_static_valid = true;
        }
        d2d(band, d.mask_static.p + static_cast<size_t>(row_begin) * res_x, band_bytes, d.stream);
    } else {
        dev_zero(band, band_bytes, d.stream);
        mask_passes(d, d.solid_static, g, tg);
    }
    mask_passes(d, d.solid_follow, g, tg);
}

namespace {

DeviceState& mesh_owner(DeviceState& dd) {
    return dd.origin ? *dd.origin : dd;
}

// Runs `prepare` on the context that owns the mesh unless its `limit` already holds alpha_limit.
// What it writes belongs to that owner; its siblings read the same array, possibly on other streams
// right now, so a change of --alpha_limit (rare) is fenced by device-wide syncs, unless the caller
// has fenced every stream that reads the array with events (`fenced`).
template <class Prepare>
void prepare_for_limit(DeviceState& dd, double alpha_limit, double DeviceState::*limit, bool DeviceState::*valid,
                       bool fenced, Prepare prepare) {
    DeviceState& d = mesh_owner(dd);
    if (d.*valid && d.*limit == alpha_limit) return;
    const bool shared = !fenced && (dd.origin != nullptr || d.mesh_shared);
    if (shared && !kHostSim) C5_CUDA(cudaDeviceSynchronize());
    struct SyncAfter {
        bool on;
        ~SyncAfter() {
            if (on) cudaDeviceSynchronize();
        }
    } sync_after{shared && !kHostSim};
    count_launch();
    prepare(d);
    d.*limit = alpha_limit;
    d.*valid = true;
}

} // namespace

void launch_prepare_cells(DeviceState& dd, double alpha_limit, bool fenced) {
    prepare_for_limit(dd, alpha_limit, &DeviceState::cells_limit, &DeviceState::cells_limit_valid, fenced, [&](DeviceState& d) {
        if (kHostSim) {
            for (int64_t t = 0; t < d.n_tets; t++) prepare_cell_body(t, d.fields.p, d.q0.p, alpha_limit);
        } else {
            prepare_cells<<<grid_for(d.n_tets, 256), 256, 0, dd.stream>>>(d.n_tets, d.fields.p, d.q0.p, alpha_limit);
            C5_CUDA(cudaGetLastError());
        }
    });
}

void launch_prepare_channels(DeviceState& dd, double alpha_limit, bool fenced) {
    if (mesh_owner(dd).n_channels == 0) return;
    prepare_for_limit(dd, alpha_limit, &DeviceState::ch_limit, &DeviceState::ch_limit_valid, fenced, [&](DeviceState& d) {
        const int64_t n = d.n_tets * d.n_channels;
        if (kHostSim) {
            for (int64_t k = 0; k < n; k++) prepare_channel_body(k, d.ch_rec.p, d.ch_q0.p, d.n_tets, d.n_channels, alpha_limit);
        } else {
            prepare_channels<<<grid_for(n, 256), 256, 0, dd.stream>>>(d.n_tets, d.n_channels, d.ch_rec.p, d.ch_q0.p,
                                                                      alpha_limit);
            C5_CUDA(cudaGetLastError());
        }
    });
}

void dedupe_solid_faces(DeviceState& d, SolidSet& ss) {
    const int64_t n_all = ss.n * 4;
    ss.n_faces = 0;
    ss.faces.release();
    if (n_all == 0) return;
    DevBuf<uint64_t> keys;
    DevBuf<uint32_t> vals, pos;
    DevBuf<uint8_t> first;
    keys.alloc(static_cast<size_t>(n_all));
    vals.alloc(static_cast<size_t>(n_all));
    pos.alloc(static_cast<size_t>(n_all));
    first.alloc(static_cast<size_t>(n_all));
    for_each(d.stream, n_all, SolidFaceKeyOp{ss.pts0.p, keys.p, vals.p});
    sort_pairs_u64(keys.p, vals.p, static_cast<size_t>(n_all), 64, d.stream);
    for_each(d.stream, n_all, SolidFaceFirstOp{ss.pts0.p, keys.p, vals.p, first.p});
    const size_t n_u = select_flagged(first.p, pos.p, static_cast<size_t>(n_all), d.stream);
    ss.faces.alloc(n_u);
    for_each(d.stream, static_cast<int64_t>(n_u), GatherU32Op{vals.p, pos.p, ss.faces.p});
    // ... in face-id order: consecutive threads of the per-view passes then read consecutive tets' points
    // (the hash order left every thread alone in its cache line)
    if (n_u > 1) {
        for_each(d.stream, static_cast<int64_t>(n_u), WidenU32Op{ss.faces.p, keys.p});
        sort_pairs_u64(keys.p, ss.faces.p, n_u, 32, d.stream);
    }
    stream_sync(d.stream);
    ss.n_faces = static_cast<int64_t>(n_u);
}

void launch_bvh_refit(DeviceState& d) {
    dev_zero(d.refit_flags.p, d.refit_flags.bytes(), d.stream);
    count_launch();
    if (kHostSim) {
        for (int64_t i = 0; i < d.n_bfaces; i++) {
            refit_leaf_body(i, d.bfaces.p, d.vrot.p, d.nodes.p, d.node_parent.p, d.leaf_parent.p, d.refit_flags.p);
        }
        return;
    }
    bvh_refit<<<grid_for(d.n_bfaces, 256), 256, 0, d.stream>>>(d.n_bfaces, d.bfaces.p, d.vrot.p, d.nodes.p,
                                                                d.node_parent.p, d.leaf_parent.p,
                                                                d.refit_flags.p);
    C5_CUDA(cudaGetLastError());
}

} // namespace c5
