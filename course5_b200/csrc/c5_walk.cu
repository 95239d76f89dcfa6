// c5_walk.cu — K3 + K4 + K4g: per-pixel ray entry (LBVH over boundary faces), the tet walk, and the
// warp-per-ray kernel for rays that graze the boundary.
//
// Replaces, for one view, the reference's
//   plane::find_intersections   plane.cpp:184-192 (scan-convert every face of every tet, one
//                               mutex-guarded push per tet-step, line.cpp:29-67,229-232)
//   line::calculate_intersections / direct_calculate_ray_value / integrate_ray_value_by_i
//                               line.cpp:84-227 (2 face-plane z's per record, per-pixel sort,
//                               tau = sum dz*alpha, I recurrence with the alpha clamp)
//   plane::trace_rays           plane.cpp:144-172 (driver, float cast)
// by one thread per pixel that (1) finds the lowest boundary face under the pixel whose outward
// normal points to -z, (2) walks tet to tet through the face-neighbour table in +z order — the
// order in which the reference integrates I (line.cpp:206: from the record with the lowest z
// to the highest) — and (3) on leaving the mesh asks the BVH for the next entries above (meshes
// with cavities or a bumpy silhouette are crossed several times). Rays with many crossings, or
// whose searches are expensive, are deferred to grazing_rays_* (one warp per ray, further down).
//
// File map: loads -> entry search (one thread) -> one crossing (FP64 over cell fields or channels,
// FP32) -> field policies -> one ray, in warp-synchronised phases (trace_ray) -> grazing rays:
// composition, serial form, warp-cooperative collection / sort / walk -> kernels (walk_block,
// fill_background, graze_block) -> host loops -> launch_walk. Everything from trace_ray on is one
// body over a field policy: FP64 cell fields, FP32 cell fields, K uploaded channels, or the depth,
// gradient and tangent passes of the derivatives.
//
// Geometry of one step. All rays are parallel to z, so "which face does the ray leave through"
// is a 2-D question about the projected tet. The entry face (a,b,c) is kept counter-clockwise in
// projection, with coordinates relative to the pixel. With d the fourth vertex and
//     s_v = orient2(d, v)   (z-component of (d-p) x (v-p)),  v in {a,b,c},
// the ray leaves through face (d,a,b) iff s_a >= 0 > s_b, through (d,b,c) iff s_b >= 0 > s_c,
// through (d,c,a) iff s_c >= 0 > s_a. orient2 is exactly antisymmetric (c5_types.h), so two tets
// sharing an edge agree on the side the ray passes: the walk is watertight without epsilons.
// Two of the s values are also barycentric weights of the pixel in the exit face (the third is one
// more orient2 of the two vertices that stay), so the exit z costs one divide; it is the entry z
// of the next tet, i.e. each face plane is evaluated once per ray, not twice as in line.cpp:103-122.
//
// Per step the thread reads the tet's 32-byte Conn and 16-byte Fields and ONE new 32-byte vertex; the
// other three vertices stay in registers (the 72 B/step algorithmic figure of SURVEY.md §8d counts
// 16 B of vertex ids the walk does without: it tracks which local slots of the tet hold the entry
// face's vertices, c5_types.h).
#include "c5_internal.h"

#include <algorithm>
#include <utility>

namespace c5 {

namespace {

constexpr int kStack = 64;        // private LBVH traversal stack; a search that would overflow it is an incomplete search
constexpr int kBlock = 128;       // 4 warps of 32 rays

// The pixel kernels' rays are dealt out by region: the walk's rectangle is cut into regions of kRegion x kRegion
// pixels from its origin (i0, j0), and each region into kBlocksPerRegion blocks of kBlock rays. A block keeps its
// slots on the SM until its longest ray ends, and a warp issues until its longest ray does, so rays that take
// about as many steps should share a block and a warp. order_rays sorts each region's pixels by the tet-steps the
// state's previous view took there (DeviceState::ray_cost): stably by (cost_bucket, local Morton index), where that
// saves enough (sort_pays), else in Morton order: warps of 8 x 4 pixels, blocks of 16 x 8. Every thread still
// traces one pixel, fixed when its block starts, so the image and every count do not depend on the order.
// The constants are measured (one B200, profiles/r13_ray_order_constants_one_b200.jsonl, every region sorted,
// against the Morton order of the same build): regions of 16, 32 and 64 pixels all cut C3's time per view by
// 11-14 %, but only 16 x 16 kept the oblique view near the Morton order (32 and 64: 1 % slower); larger regions
// scatter a block's rays over more tets. Of buckets 1, 8 and 32 steps wide, 1 is the best over both views.
constexpr int kRegionLog = 4;
constexpr int kRegion = 1 << kRegionLog;
constexpr int kRegionPix = kRegion * kRegion;
constexpr int kBlocksPerRegion = kRegionPix / kBlock;
constexpr int kBucketShift = 0;   // costs less than 2^kBucketShift steps apart may share a bucket
constexpr int kBuckets = 128;     // bucket 0: cost 0 (a miss, a solid pixel, outside the rectangle, unknown)
static_assert(kRegionPix % kBlock == 0, "a region is whole blocks");

struct WalkParams {
    const Conn* conn;
    const Fields* fields;
    const Vtx* vrot;
    const BFace* bfaces;
    const BvhNode* nodes;
    const double* xs;
    const double* ys;
    const uint8_t* mask;  // may be null
    double* out;          // band buffer: {tau, I} at ((j - row_begin) * res_x + i)
    uint32_t* steps;      // may be null; same indexing
    unsigned long long* counters;
    unsigned long long* row_cost; // [res_y]
    DeferredRay* queue;   // rays handed to the grazing-ray kernel; counters[kDeferred] of them
    int res_x, res_y, row_begin, row_end;
    int i0, i1, j0, j1;   // pixel rectangle [i0,i1) x [j0,j1) of the band that can see the mesh: the regions cover it
    int n_regions_x;      // regions per row of the rectangle
    uint16_t* cost;       // [res_y][res_x] tet-steps of each pixel's ray (saturating), written by the pixel kernel
    uint16_t* order;      // [region][kRegionPix] local Morton indices in walk order, written by order_rays
    int graze_cap;        // entries one cooperative collection may hold (<= kGrazeList)
    int serial_cap;       // same for the serial (host loop) form (<= kSerialList)
    int query_budget;     // BVH nodes one thread of the pixel kernel may visit per search before deferring the ray
    int max_steps;
    int round_float;
    double alpha_limit;
    // channel renders only (null otherwise)
    const double* rec;    // [n_tets][channel_stride(K)]: {alpha_c, s_c} per channel
    double* ch_queue;     // [deferred ray][K] {tau, I}: the channel values DeferredRay::tau/inten hold otherwise
};

// The gradient pass's kernels take these (the walk functions see the WalkParams part; the gradient
// policy below casts back). A separate type keeps WalkParams, and so every other kernel, as it was.
struct GradParams : WalkParams {
    const double* grad_in; // band buffer: {g_tau, g_I} per pixel, indexed like out (the per-view kernels: the
                           // view's one {g_tau, g_I}, c5_render_flux_grad_device)
    const double* depth;   // the depth pass's band buffer: {tau, I, lam, 0} per pixel
    double* grad_alpha;    // [n_tets] Morton order, accumulated with atomics
    double* grad_q;
};

// The forward-mode kernels (c5_render_jvp) take these, for the same reason.
struct JvpParams : WalkParams {
    const double* dir;     // [n_tets][2] Morton order: the direction {v_alpha, v_q} of each tet
};

// ---- loads through the read-only path ----------------------------------------------------------
struct ConnData {
    int4 nbr;
    uint4 apex;
};

// sm_100 has 256-bit global loads (SASS LDG.E.ENL2.256): a 32-byte Conn is one of them, a 32-byte
// vertex one, and the 16-byte Fields one LDG.128: 3 load instructions per tet-step.
C5_HD ConnData load_conn(const Conn* conn, int t) {
    ConnData c;
#ifdef __CUDA_ARCH__
    asm volatile("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(c.nbr.x), "=r"(c.nbr.y), "=r"(c.nbr.z), "=r"(c.nbr.w), "=r"(c.apex.x), "=r"(c.apex.y),
                   "=r"(c.apex.z), "=r"(c.apex.w)
                 : "l"(conn + t));
#else
    const Conn& s = conn[t];
    c.nbr = make_int4(s.nbr[0], s.nbr[1], s.nbr[2], s.nbr[3]);
    c.apex = make_uint4(s.apex[0], s.apex[1], s.apex[2], s.apex[3]);
#endif
    return c;
}

// alpha and s of the tet being crossed, loaded by a field policy's fetch() together with its Conn
struct TetFields {
    double alpha, s;
    C5_HD void load(const Fields* fields, int t) {
#ifdef __CUDA_ARCH__
        asm volatile("ld.global.nc.v2.f64 {%0,%1}, [%2];" : "=d"(alpha), "=d"(s) : "l"(fields + t));
#else
        alpha = fields[t].alpha;
        s = fields[t].s;
#endif
    }
};

// Where the ray goes after leaving tet t through the face opposite local slot k: the next tet, its
// new vertex, and the slots in it of the exit face's vertices. `slots` holds the slots in t of the
// face the walk keeps (a, b, c: 2 bits each); the dropped vertex is the one at bit `sh`, and the new
// vertex d of t, at the slot the three leave free, takes its place.
C5_HD int step_across(const ConnData& c, uint32_t& slots, uint32_t sh, int& id_next) {
    const uint32_t k = (slots >> sh) & 3u;
    // two selects per word on the bits of k, without branches
    const bool k0 = k & 1u, k1 = k & 2u;
    const int t_next = k1 ? (k0 ? c.nbr.w : c.nbr.z) : (k0 ? c.nbr.y : c.nbr.x);
    const uint32_t apex = k1 ? (k0 ? c.apex.w : c.apex.z) : (k0 ? c.apex.y : c.apex.x);
    id_next = static_cast<int>(apex & kApexIdMask);
    const uint32_t sd = (slots ^ (slots >> 2) ^ (slots >> 4)) & 3u; // 0 ^ 1 ^ 2 ^ 3 == 0
    const uint32_t face = (slots & ~(3u << sh)) | (sd << sh);
    // perm: 2-bit field s = the slot in the next tet of slot s of this one (s != k), i.e. the map
    // rotated by k fields
    const uint32_t rot = (apex >> kApexIdBits) << 2;
    const uint32_t perm = ((rot << 8) | rot) >> (8u - 2u * k);
    slots = ((perm >> (2u * (face & 3u))) & 3u) | (((perm >> (2u * ((face >> 2) & 3u))) & 3u) << 2) |
            (((perm >> (2u * (face >> 4))) & 3u) << 4);
    return t_next;
}

// The entry of a crossing through boundary face `leaf`: its vertices (a, c, b of the stored winding,
// counter-clockwise in projection), tet, apex and their slots.
struct Entry {
    int ia, ib, ic, t, id;
    uint32_t slots;
};
C5_HD Entry load_entry(const WalkParams& P, int leaf) {
#ifdef __CUDA_ARCH__
    const int4 f = __ldg(reinterpret_cast<const int4*>(P.bfaces + leaf));
    const int2 e = __ldg(reinterpret_cast<const int2*>(&P.bfaces[leaf].apex));
    return Entry{f.x, f.z, f.y, f.w, e.x, static_cast<uint32_t>(e.y)};
#else
    const BFace& bf = P.bfaces[leaf];
    return Entry{bf.a, bf.c, bf.b, bf.tet, bf.apex, static_cast<uint32_t>(bf.slots)};
#endif
}

C5_HD void load_vtx(const Vtx* vrot, int id, double& x, double& y, double& z) {
#ifdef __CUDA_ARCH__
    [[maybe_unused]] double w;
    asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(x), "=d"(y), "=d"(z), "=d"(w) : "l"(vrot + id));
#else
    x = vrot[id].x;
    y = vrot[id].y;
    z = vrot[id].z;
#endif
}

// ---- entry search --------------------------------------------------------------------------------

// Entry list of one ray: the lowest entry faces above z_after, sorted by (z, leaf). A ray through a
// convex mesh has one entry; cavities add a few; a ray grazing a bumpy boundary (the jittered side
// walls of the synthetic grids, seen edge-on) has ~100. A thread walking such a ray alone is a chain
// of dependent BVH queries and short crossings, and a handful of them set the run time of a whole
// row band (measured: 1.2-1.3 ms for ANY band of the C3 README view, profiles/r01_exp_bands.jsonl).
// So the pixel kernel only ever asks for a short list (kInline entries); a ray whose list comes back
// full is handed to the grazing-ray kernel below, where a whole warp works on it.
template <int kCap>
struct EntryList {
    double z[kCap];
    int leaf[kCap];
    int n;
};

constexpr int kInline = 4;   // re-entry list of the pixel kernel: fewer entries than this are walked in place
constexpr int kSerialList = 64; // list of the serial (host loop) grazing path

// Depth at which the ray through (px, py) enters the mesh through boundary face `leaf`: inclusive
// point-in-triangle test with the same orientation predicate the walk uses, then the barycentric z.
// False if the face is not under the pixel, faces +z, or lies at or below z_after.
C5_HD bool entry_depth(const WalkParams& P, int leaf, double px, double py, double z_after, double& z_out) {
#ifdef __CUDA_ARCH__
    const int4 f = __ldg(reinterpret_cast<const int4*>(P.bfaces + leaf));
#else
    const BFace& bf = P.bfaces[leaf];
    const int4 f = make_int4(bf.a, bf.b, bf.c, bf.tet);
#endif
    double ax, ay, az, bx, by, bz, cx, cy, cz;
    load_vtx(P.vrot, f.x, ax, ay, az);
    load_vtx(P.vrot, f.y, bx, by, bz);
    load_vtx(P.vrot, f.z, cx, cy, cz);
    ax -= px; ay -= py;
    bx -= px; by -= py;
    cx -= px; cy -= py;
    const double o_ab = orient2(ax, ay, bx, by);
    const double o_bc = orient2(bx, by, cx, cy);
    const double o_ca = orient2(cx, cy, ax, ay);
    // outward normal towards -z  <=>  clockwise in projection  <=>  all three <= 0 inside
    if (!(o_ab <= 0 && o_bc <= 0 && o_ca <= 0)) return false;
    const double sum = o_ab + o_bc + o_ca;
    if (!(sum < 0)) return false;
    const double z = (o_bc * az + o_ca * bz + o_ab * cz) / sum;
    if (!(z > z_after)) return false;
    z_out = z;
    return true;
}

C5_HD bool entry_before(double z0, int leaf0, double z1, int leaf1) { // strict (z, leaf) order
    return z0 < z1 || (z0 == z1 && leaf0 < leaf1);
}

// Keeps the `cap` lowest entries, sorted; faces arrive roughly near-to-far, so the insertion from
// the back is close to linear.
template <int kCap>
C5_HD void insert_entry(EntryList<kCap>& L, int cap, double z, int leaf) {
    if (L.n == cap) {
        if (!entry_before(z, leaf, L.z[cap - 1], L.leaf[cap - 1])) return;
        L.n--; // the highest one falls off
    }
    int k = L.n++;
    while (k > 0 && entry_before(z, leaf, L.z[k - 1], L.leaf[k - 1])) {
        L.z[k] = L.z[k - 1];
        L.leaf[k] = L.leaf[k - 1];
        k--;
    }
    L.z[k] = z;
    L.leaf[k] = leaf;
}

// The (up to cap <= kCap) lowest entry faces strictly above z_after under pixel (px, py), by one
// thread with a private stack. cap = 1 is the classic nearest-hit search: once one face is found,
// every node whose box starts above it is pruned. L.n == cap on return means "there may be more
// above L.z[cap - 1]"; L.n < cap means the list is complete.
//
// `budget` bounds the nodes one thread may visit. A ray that runs along a boundary wall (inside or
// outside it) overlaps the boxes of every facet of that wall: proving "no further entry" then costs
// hundreds of dependent loads, and the few blocks holding such rays ran 60 % longer than all others
// (block timeline, profiles/r01_trace_band_c3.txt). A search that exceeds its budget returns false
// and the ray is handed to the grazing-ray kernel, where 32 lanes share the traversal.
template <int kCap>
C5_HD bool bvh_collect_entries(const WalkParams& P, double px, double py, double z_after, EntryList<kCap>& L, int cap,
                               int budget) {
    int stack[kStack];
    int sp = 0;
    L.n = 0;
    int node = 0;
    const float fx_lo = f_round_down(px), fx_hi = f_round_up(px);
    const float fy_lo = f_round_down(py), fy_hi = f_round_up(py);
    // (one exit from the loop: with a `return` in the middle the compiler stopped reconverging the
    // warp after the search and the tet walk ran with half-empty warps — 8.3 instead of 4.7 ms on C3)
    bool complete = true;
    while (true) {
        if (--budget < 0) {
            complete = false;
            break;
        }
        // (staging the top BVH levels in shared memory was measured slower than letting L1 serve them:
        // C3 6.38 ms with 0 nodes, 6.54 with 63, 6.88 with 255; profiles/r01_exp_c3_variants_b.jsonl)
        const BvhNode* n = P.nodes + node;
#ifdef __CUDA_ARCH__
        const float4 bx = *reinterpret_cast<const float4*>(n->xlo); // xlo0 xlo1 xhi0 xhi1
        const float4 by = *reinterpret_cast<const float4*>(n->ylo);
        const float4 bz = *reinterpret_cast<const float4*>(n->zlo);
        const int2 ch = *reinterpret_cast<const int2*>(n->child);
#else
        const float4 bx = make_float4(n->xlo[0], n->xlo[1], n->xhi[0], n->xhi[1]);
        const float4 by = make_float4(n->ylo[0], n->ylo[1], n->yhi[0], n->yhi[1]);
        const float4 bz = make_float4(n->zlo[0], n->zlo[1], n->zhi[0], n->zhi[1]);
        const int2 ch = make_int2(n->child[0], n->child[1]);
#endif
        // once the list is full, nothing above its highest entry can get in
        const double z_cap = (L.n == cap) ? L.z[cap - 1] : INFINITY;
        // boxes are rounded outward and the pixel is widened to floats, so this never misses
        bool h0 = fx_hi >= bx.x && fx_lo <= bx.z && fy_hi >= by.x && fy_lo <= by.z &&
                  static_cast<double>(bz.z) > z_after && static_cast<double>(bz.x) <= z_cap;
        bool h1 = fx_hi >= bx.y && fx_lo <= bx.w && fy_hi >= by.y && fy_lo <= by.w &&
                  static_cast<double>(bz.w) > z_after && static_cast<double>(bz.y) <= z_cap;
        double z;
        if (h0 && ch.x < 0) {
            if (entry_depth(P, ~ch.x, px, py, z_after, z)) insert_entry(L, cap, z, ~ch.x);
            h0 = false;
        }
        if (h1 && ch.y < 0) {
            if (entry_depth(P, ~ch.y, px, py, z_after, z)) insert_entry(L, cap, z, ~ch.y);
            h1 = false;
        }
        if (h0 && h1) {
            const bool first0 = bz.x <= bz.y; // descend into the lower subtree first
            if (sp == kStack) { // a tree deeper than the private stack: never drop a subtree, hand the ray on
                complete = false;
                break;
            }
            stack[sp++] = first0 ? ch.y : ch.x;
            node = first0 ? ch.x : ch.y;
        } else if (h0) {
            node = ch.x;
        } else if (h1) {
            node = ch.y;
        } else {
            if (sp == 0) break;
            node = stack[--sp];
        }
    }
    return complete;
}

// ---- one crossing ----------------------------------------------------------------------------------

// One crossing of the mesh: the ray enters through boundary face `leaf` at depth z_in and goes from
// tet to tet until it leaves through another boundary face; returns that depth. tau, inten and steps
// are updated in place. kAffine: the caller does not know the intensity the ray arrives with (the
// grazing-ray kernel walks the crossings of one ray in parallel); inten then starts at 0 and gain at
// 1, and the crossing maps an arriving I to inten + gain * I (the recurrence of line.cpp:206-225 is
// affine in I: s - (s - I) e = s (1 - e) + e I).
//
// `acc` integrates the fields along the crossing: fetch(P, t) is issued with tet t's Conn load and
// step(P, dz) adds one segment. CellFields below integrates the cells' own alpha and s; ChanFields
// integrates K uploaded field pairs over the same steps.
template <bool kAffine, class Acc>
C5_HD double crossing_walk(const WalkParams& P, double px, double py, int leaf, double z_in, Acc& acc,
                           uint32_t& steps, uint32_t& error) {
    const Entry e = load_entry(P, leaf);
    int id = e.id;
    uint32_t slots = e.slots;
    double ax, ay, az, bx, by, bz, cx, cy, cz;
    load_vtx(P.vrot, e.ia, ax, ay, az);
    load_vtx(P.vrot, e.ib, bx, by, bz);
    load_vtx(P.vrot, e.ic, cx, cy, cz);
    ax -= px; ay -= py;
    bx -= px; by -= py;
    cx -= px; cy -= py;
    int t = e.t;
    double z_cur = z_in;
    while (true) {
        if (steps >= static_cast<uint32_t>(P.max_steps)) {
            error = 1;
            break;
        }
        // id = the vertex of tet t that is not on the entry face. It is known BEFORE t's Conn is
        // read (Conn::apex of the previous tet, BFace::apex at entry), so the Conn, Fields and vertex
        // loads of a step are independent and overlap: one memory latency per step, not two.
        const ConnData c = load_conn(P.conn, t);
        acc.fetch(P, t);
        double dx, dy, dz;
        load_vtx(P.vrot, id, dx, dy, dz);
        dx -= px;
        dy -= py;
        const double sa = orient2(dx, dy, ax, ay);
        const double sb = orient2(dx, dy, bx, by);
        const double sc = orient2(dx, dy, cx, cy);
        // which face the ray leaves through, hence the next tet and its new vertex
        const bool drop_c = sa >= 0 && sb < 0;             // through (d, a, b)
        const bool drop_a = !drop_c && sb >= 0 && sc < 0;  // through (d, b, c)
        int id_next;                                        // else through (d, c, a)
        const int t_next = step_across(c, slots, drop_c ? 4u : drop_a ? 0u : 2u, id_next);
        // Barycentric weights of the pixel in the exit face (weight of a vertex = orient2 of the
        // other two, in cyclic order). Two of them are s values; the third belongs to d and is the
        // orient2 of the two vertices that stay — recomputed here (3 flops) rather than carried
        // from step to step (6 registers): same operands, same operations, so the same bits.
        double wa, wb, wc;
        if (drop_c) { // leaves through (d, a, b): c is replaced by d
            cx = dx; cy = dy; cz = dz;
            wa = -sb;
            wb = sa;
            wc = orient2(ax, ay, bx, by);
        } else if (drop_a) { // through (d, b, c): a is replaced
            ax = dx; ay = dy; az = dz;
            wb = -sc;
            wc = sb;
            wa = orient2(bx, by, cx, cy);
        } else { // through (d, c, a): b is replaced
            bx = dx; by = dy; bz = dz;
            wc = -sa;
            wa = sc;
            wb = orient2(cx, cy, ax, ay);
        }
        const double wsum = wa + wb + wc;
        const double z_exit = (wsum != 0.0) ? (wa * az + wb * bz + wc * cz) / wsum : z_cur;
        const double dzv = fabs(z_exit - z_cur);
        acc.step(P, dzv);
        steps++;
        z_cur = z_exit;
        t = t_next;
        id = id_next;
        if (t < 0) break;
    }
    return z_cur;
}

// One segment of length dz through a medium (alpha, s):
// tau: line.cpp:176-193 (alpha not clamped);
// I: line.cpp:206-225 with s = Q / a^:  (Q - (Q - a^ I) e) / a^  ==  s - (s - I) e  ==  I - (s - I) m,
// m = e - 1 = expm1(-a^ dz). The last form does not cancel: s - (s - I) e subtracts two numbers of
// size s to get an increment of size Q dz, and loses log10(1 / (a^ dz)) digits a step (all of them
// once exp rounds to 1, below a^ dz ~ 1e-16), while -(s - I) m and I are each exact to a few ulps.
template <bool kAffine>
C5_HD void segment(double alpha, double s, double limit, double dzv, double& tau, double& inten, double& gain) {
    tau += dzv * alpha;
    double a_c = alpha;
    if (a_c > limit) a_c = limit;
    if (!(a_c < DBL_EPSILON)) {
        const double m = expm1(-a_c * dzv);
        inten = inten - (s - inten) * m;
        if (kAffine) gain *= 1.0 + m;
    }
}

// K {tau, I} pairs, of one ray or of one crossing. A crossing walked without the I it arrives with
// (kAffine) also yields gain[c], the factor it puts on that I; elsewhere gain stays 1 and is not read.
// Loops over K are unrolled with fixed bounds, so the arrays live in registers.
// The pixel kernel's pairs are value-initialised and stored by fold expressions over c = 0 .. K-1 of
// force-inlined calls. A loop, even of one trip, is unrolled only after the compiler's early passes,
// which then see the arrays in memory: the FP64 pixel kernel came out slower that way (C3 on one
// B200: 4.416 against 4.401 ms per view).
template <int K, int... C>
C5_HD void fill_pairs(double (&a)[K], double v, std::integer_sequence<int, C...>) {
    ((a[C] = v), ...);
}

template <int K>
struct Pairs {
    double tau[K], inten[K], gain[K];
    C5_HD void reset() {
#pragma unroll
        for (int c = 0; c < K; c++) {
            tau[c] = 0.0;
            inten[c] = 0.0;
            gain[c] = 1.0;
        }
    }
};

template <bool kAffine>
struct CellFields {
    Pairs<1>& v;
    TetFields c;
    C5_HD void fetch(const WalkParams& P, int t) { c.load(P.fields, t); }
    C5_HD void step(const WalkParams& P, double dzv) {
        segment<kAffine>(c.alpha, c.s, P.alpha_limit, dzv, v.tau[0], v.inten[0], v.gain[0]);
    }
};

// K uploaded field pairs. A step reads tet t's record of K {alpha_c, s_c} pairs (padded to 32-byte
// sectors) together with t's Conn, since t is known at the top of the step, so a channel adds FP64
// work and a store but no further round trip. The tet's own Fields are not read.
template <int K, bool kAffine>
struct ChanFields {
    const double* rec;
    Pairs<K>& v;
    double f[channel_stride(K)]; // the record of the tet being crossed

    // f stays uninitialised: fetch fills it before every step (zeroing it costs the K = 3 grazing-ray
    // kernel 24 more bytes of spills)
    C5_HD ChanFields(const double* rec_, Pairs<K>& v_) : rec(rec_), v(v_) {}
    C5_HD void fetch(const WalkParams&, int t) {
        const double* p = rec + static_cast<size_t>(t) * channel_stride(K);
#ifdef __CUDA_ARCH__
#pragma unroll
        for (int k = 0; k < channel_stride(K); k += 4) {
            asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];"
                         : "=d"(f[k]), "=d"(f[k + 1]), "=d"(f[k + 2]), "=d"(f[k + 3])
                         : "l"(p + k));
        }
#else
        for (int k = 0; k < channel_stride(K); k++) f[k] = p[k];
#endif
    }
    C5_HD void step(const WalkParams& P, double dzv) {
#pragma unroll
        for (int c = 0; c < K; c++) segment<kAffine>(f[2 * c], f[2 * c + 1], P.alpha_limit, dzv, v.tau[c], v.inten[c], v.gain[c]);
    }
};

// ---- FP32 variant -----------------------------------------------------------------------------------
// Same crossing with the per-step geometry in single precision: FP32 orientation tests (still exactly
// antisymmetric: two rounded products, one rounded difference), FP32 divide and expm1f — about half
// the issue slots and 56 instead of 72 registers. What stays in double: the ENTRY search (so the
// hit/miss set is the FP64 one, bit for bit), the vertex fetch and its subtraction of the pixel
// position / entry depth (rounding a coordinate ~1 to float would cost 1e-7, i.e. 1e-5 of a tet;
// rounding the DIFFERENCE costs 6e-8 of the tet size), and the accumulators tau and I. The walk
// is not bandwidth-bound (DESIGN.md §4), so keeping 32-byte vertices costs nothing measurable.
// Tolerance vs the reference: 1e-4 relative (tests/parity.py).
C5_HD float fmul_rn(float a, float b) {
#ifdef __CUDA_ARCH__
    return __fmul_rn(a, b);
#else
    return a * b;
#endif
}
C5_HD float fsub_rn(float a, float b) {
#ifdef __CUDA_ARCH__
    return __fsub_rn(a, b);
#else
    return a - b;
#endif
}
C5_HD float orient2f(float ux, float uy, float vx, float vy) {
    return fsub_rn(fmul_rn(ux, vy), fmul_rn(uy, vx));
}

template <bool kAffine>
C5_HD double crossing_f32(const WalkParams& P, double px, double py, int leaf, double z_in, double& tau,
                          double& inten, double& gain, uint32_t& steps, uint32_t& error) {
    const float limit = static_cast<float>(P.alpha_limit);
    const double z0 = z_in; // depths are kept relative to the entry point of the crossing
    const Entry e = load_entry(P, leaf);
    int id = e.id;
    uint32_t slots = e.slots;
    float ax, ay, az, bx, by, bz, cx, cy, cz;
    {
        double x, y, z;
        load_vtx(P.vrot, e.ia, x, y, z);
        ax = static_cast<float>(x - px); ay = static_cast<float>(y - py); az = static_cast<float>(z - z0);
        load_vtx(P.vrot, e.ib, x, y, z);
        bx = static_cast<float>(x - px); by = static_cast<float>(y - py); bz = static_cast<float>(z - z0);
        load_vtx(P.vrot, e.ic, x, y, z);
        cx = static_cast<float>(x - px); cy = static_cast<float>(y - py); cz = static_cast<float>(z - z0);
    }
    float wa = orient2f(bx, by, cx, cy);
    float wb = orient2f(cx, cy, ax, ay);
    float wc = orient2f(ax, ay, bx, by);
    int t = e.t;
    float z_cur = 0.f;
    while (true) {
        if (steps >= static_cast<uint32_t>(P.max_steps)) {
            error = 1;
            break;
        }
        const ConnData c = load_conn(P.conn, t);
        TetFields fc;
        fc.load(P.fields, t);
        float dx, dy, dz;
        {
            double x, y, z;
            load_vtx(P.vrot, id, x, y, z);
            dx = static_cast<float>(x - px);
            dy = static_cast<float>(y - py);
            dz = static_cast<float>(z - z0);
        }
        const float sa = orient2f(dx, dy, ax, ay);
        const float sb = orient2f(dx, dy, bx, by);
        const float sc = orient2f(dx, dy, cx, cy);
        const bool drop_c = sa >= 0 && sb < 0;
        const bool drop_a = !drop_c && sb >= 0 && sc < 0;
        int id_next;
        const int t_next = step_across(c, slots, drop_c ? 4u : drop_a ? 0u : 2u, id_next);
        if (drop_c) {
            cx = dx; cy = dy; cz = dz;
            wa = -sb;
            wb = sa;
        } else if (drop_a) {
            ax = dx; ay = dy; az = dz;
            wb = -sc;
            wc = sb;
        } else {
            bx = dx; by = dy; bz = dz;
            wc = -sa;
            wa = sc;
        }
        const float wsum = wa + wb + wc;
        const float z_exit = (wsum != 0.0f) ? (wa * az + wb * bz + wc * cz) / wsum : z_cur;
        const float dzv = fabsf(z_exit - z_cur);
        tau += static_cast<double>(dzv) * fc.alpha;
        float a_c = static_cast<float>(fc.alpha);
        if (a_c > limit) a_c = limit;
        const double a_d = fc.alpha > P.alpha_limit ? P.alpha_limit : fc.alpha;
        if (!(a_d < DBL_EPSILON)) { // the cancellation-free form of segment(), expm1f's error is relative
            const double m = static_cast<double>(expm1f(-a_c * dzv));
            inten = inten - (fc.s - inten) * m;
            if (kAffine) gain *= 1.0 + m;
        }
        steps++;
        z_cur = z_exit;
        t = t_next;
        id = id_next;
        if (t < 0) break;
    }
    // the next crossing must lie above this one's exit (and strictly above its entry)
    const double z_exit_abs = z0 + static_cast<double>(z_cur);
    return z_exit_abs > z0 ? z_exit_abs : z0;
}

// ---- field policies ----------------------------------------------------------------------------------
// What a ray integrates. Everything from trace_ray on is written once over a policy F:
//   F::K                   {tau, I} pairs per pixel, stored at out[((j - row_begin) * res_x + i) * K + c];
//   F::crossing<kAffine>   the crossing that integrates them into a Pairs<K>;
//   F::kChanQueue          a deferred ray's values wait in WalkParams::ch_queue and DeferredRay::tau/inten
//                          stay 0; otherwise they wait in DeferredRay::tau/inten;
//   F::kImage              the pixels are stored and a grazing ray's steps are counted (false: the gradient
//                          pass, whose result is its atomics);
//   F::kTangent            pair 1 is the tangent of pair 0, and a grazing ray's fold composes it as one
//                          (compose_crossing);
//   F::kRewalk             after a grazing ray's fold, each crossing the fold took is walked again with
//                          crossing<false>, from the pairs it was entered with.
// crossing() also gets the ray's pixel (j * res_x + i); only the gradient pass reads it.
struct CellsF64 { // the cells' own fields
    static constexpr int K = 1;
    static constexpr bool kChanQueue = false;
    static constexpr bool kImage = true;
    static constexpr bool kTangent = false;
    static constexpr bool kRewalk = false;
    template <bool kAffine>
    static C5_HD double crossing(const WalkParams& P, double px, double py, uint32_t, int leaf, double z_in, Pairs<1>& v,
                                 uint32_t& steps, uint32_t& error) {
        CellFields<kAffine> acc{v};
        return crossing_walk<kAffine>(P, px, py, leaf, z_in, acc, steps, error);
    }
};

struct CellsF32 { // the cells' own fields, FP32 step geometry
    static constexpr int K = 1;
    static constexpr bool kChanQueue = false;
    static constexpr bool kImage = true;
    static constexpr bool kTangent = false;
    static constexpr bool kRewalk = false;
    template <bool kAffine>
    static C5_HD double crossing(const WalkParams& P, double px, double py, uint32_t, int leaf, double z_in, Pairs<1>& v,
                                 uint32_t& steps, uint32_t& error) {
        return crossing_f32<kAffine>(P, px, py, leaf, z_in, v.tau[0], v.inten[0], v.gain[0], steps, error);
    }
};

// Several field pairs in one walk (c5_render_channels): the rays, their entry searches, deferrals and
// steps are those of CellsF64; only what is integrated differs.
template <int N>
struct Channels {
    static constexpr int K = N;
    static constexpr bool kChanQueue = true;
    static constexpr bool kImage = true;
    static constexpr bool kTangent = false;
    static constexpr bool kRewalk = false;
    template <bool kAffine>
    static C5_HD double crossing(const WalkParams& P, double px, double py, uint32_t, int leaf, double z_in, Pairs<K>& v,
                                 uint32_t& steps, uint32_t& error) {
        ChanFields<K, kAffine> acc{P.rec, v};
        return crossing_walk<kAffine>(P, px, py, leaf, z_in, acc, steps, error);
    }
};

// ---- gradients (c5_render_grad) ------------------------------------------------------------------------
// The vector-Jacobian product of the pre-cast image with respect to every cell's alpha and Q, in two
// passes over the same rays (DESIGN.md §5c). With a^ = min(alpha, limit), x = a^ dz, m = expm1(-x) and
// e = 1 + m, a segment does I_out = I_in - (s - I_in) m, s = Q / a^, so
//   dtau/dalpha  = dz                                       (every segment: tau uses the unclamped alpha)
//   dI_out/dQ    = -m / a^                                   (a^ >= DBL_EPSILON; else the step is skipped)
//   dI_out/dalpha = s a^ dz^2 f(x) - I_in dz e,  f(x) = ((1 + x) e^-x - 1) / x^2   (and alpha <= limit)
// and a change of I_out reaches the viewer times T = exp(-(lam_ray - lam_through)): lam is the clamped
// optical depth, the sum of x over the segments that change I, lam_ray its value for the whole ray and
// lam_through its running value at the segment's exit. The difference of the two sums, unlike a ratio of
// gains, does not underflow on an opaque ray.
//   Depth pass (CellsDepth): the image of CellsF64 plus lam_ray, as a second pair {lam, 0} per pixel.
//   Gradient pass (CellsGrad): the same rays again, carrying {lam_through, I}, adding into grad_alpha /
//   grad_q with FP64 atomics. It defers exactly the rays the depth pass deferred: same search, same budget.

// The clamped depth one segment adds (0 where the step leaves I alone). Both passes add the same rounded
// product, so the last segment of a ray the pixel kernel finishes sees T = exp(0) = 1 exactly (a grazing
// ray's sums are grouped by crossing and may differ in the last bits).
C5_HD double lam_term(double alpha, double limit, double dzv) {
    double a_c = alpha;
    if (a_c > limit) a_c = limit;
    return a_c < DBL_EPSILON ? 0.0 : mul_rn(a_c, dzv);
}

// f(x) = ((1 + x) e^-x - 1) / x^2 for x >= 0, m = expm1(-x). The numerator cancels to O(x^2) near 0, so
// below 1/2 the Taylor series sum_{n>=2} (-1)^(n+1) (n-1)/n! x^(n-2) is summed instead (16 terms: the
// next one is below 3e-18 relative); above, (1 + x)(1 + m) - 1 loses at most one digit.
C5_HD double grad_f(double x, double m) {
    if (x < 0.5) {
        constexpr double c[16] = {-1.0 / 2.0, 1.0 / 3.0, -1.0 / 8.0, 1.0 / 30.0, -1.0 / 144.0, 1.0 / 840.0,
                                  -1.0 / 5760.0, 1.0 / 45360.0, -1.0 / 403200.0, 1.0 / 3991680.0, -1.0 / 43545600.0,
                                  1.0 / 518918400.0, -1.0 / 6706022400.0, 1.0 / 93405312000.0,
                                  -1.0 / 1394852659200.0, 1.0 / 22230464256000.0};
        double r = c[15];
#pragma unroll
        for (int k = 14; k >= 0; k--) r = r * x + c[k];
        return r;
    }
    return ((1.0 + x) * (1.0 + m) - 1.0) / (x * x);
}

C5_HD void add_to(double* p, double v) {
#ifdef __CUDA_ARCH__
    atomicAdd(p, v);
#else
    *p += v;
#endif
}

// What the gradient pass knows about a ray before it walks it: its upstream gradient and lam_ray.
struct GradRay {
    double g_tau, g_I, lam_ray;
};

// kViewG: every pixel of the view has the same upstream, the two doubles at grad_in.
template <bool kViewG>
C5_HD GradRay grad_ray(const GradParams& P, uint32_t pixel) {
    const size_t o = pixel - static_cast<size_t>(P.row_begin) * static_cast<size_t>(P.res_x);
    if (kViewG) return GradRay{P.grad_in[0], P.grad_in[1], P.depth[4 * o + 2]};
    return GradRay{P.grad_in[2 * o], P.grad_in[2 * o + 1], P.depth[4 * o + 2]};
}

// One segment of the gradient pass through tet t; lam and inten are the ray's lam_through and I.
C5_HD void grad_segment(const GradParams& P, int t, double alpha, double s, double dzv, const GradRay& r, double& lam,
                        double& inten) {
    double ga = r.g_tau * dzv;
    double gq = 0.0;
    double a_c = alpha;
    if (a_c > P.alpha_limit) a_c = P.alpha_limit;
    if (!(a_c < DBL_EPSILON)) {
        const double x = mul_rn(a_c, dzv);
        const double m = expm1(-x);
        lam += x;
        const double gt = r.g_I * exp(lam - r.lam_ray); // g_I T
        gq = gt * (-m / a_c);
        if (alpha <= P.alpha_limit) ga += gt * (s * x * dzv * grad_f(x, m) - inten * dzv * (1.0 + m));
        inten = inten - (s - inten) * m;
    }
    if (ga != 0.0) add_to(P.grad_alpha + t, ga);
    if (gq != 0.0) add_to(P.grad_q + t, gq);
}

// Depth pass: pair 0 is CellFields' {tau, I} (the same operations, so the same bits), tau[1] is lam.
template <bool kAffine>
struct DepthFields {
    Pairs<2>& v;
    TetFields c;
    C5_HD void fetch(const WalkParams& P, int t) { c.load(P.fields, t); }
    C5_HD void step(const WalkParams& P, double dzv) {
        segment<kAffine>(c.alpha, c.s, P.alpha_limit, dzv, v.tau[0], v.inten[0], v.gain[0]);
        v.tau[1] += lam_term(c.alpha, P.alpha_limit, dzv);
    }
};

// A crossing of a grazing ray walked without the I it arrives with: tau[0] is its lam, inten[0] + gain[0] I
// its exit I (the gradient kernel's first walk of a crossing).
struct LamFields {
    Pairs<1>& v;
    TetFields c;
    C5_HD void fetch(const WalkParams& P, int t) { c.load(P.fields, t); }
    C5_HD void step(const WalkParams& P, double dzv) {
        double tau = 0.0;
        segment<true>(c.alpha, c.s, P.alpha_limit, dzv, tau, v.inten[0], v.gain[0]);
        v.tau[0] += lam_term(c.alpha, P.alpha_limit, dzv);
    }
};

// Gradient pass: tau[0] is lam_through, inten[0] is I, both from the ray's entry (or the deferred ray's state).
struct GradFields {
    const GradParams& G;
    Pairs<1>& v;
    GradRay r;
    int t;
    TetFields c;
    C5_HD void fetch(const WalkParams& P, int t_) {
        t = t_;
        c.load(P.fields, t_);
    }
    C5_HD void step(const WalkParams&, double dzv) {
        grad_segment(G, t, c.alpha, c.s, dzv, r, v.tau[0], v.inten[0]);
    }
};

struct CellsDepth { // {tau, I} of CellsF64 and {lam, 0}
    static constexpr int K = 2;
    static constexpr bool kChanQueue = true;
    static constexpr bool kImage = true;
    static constexpr bool kTangent = false;
    static constexpr bool kRewalk = false;
    template <bool kAffine>
    static C5_HD double crossing(const WalkParams& P, double px, double py, uint32_t, int leaf, double z_in, Pairs<2>& v,
                                 uint32_t& steps, uint32_t& error) {
        DepthFields<kAffine> acc{v};
        return crossing_walk<kAffine>(P, px, py, leaf, z_in, acc, steps, error);
    }
};

// The gradient pass: nothing is stored but the atomics; P is the WalkParams of a GradParams. kViewG: one
// upstream per view (grad_ray), the light-curve form. A grazing ray's crossing is walked affinely for its
// lam and (A, B), and once the fold has given it the {lam, I} it is entered with, again with the gradient.
template <bool kViewG>
struct CellsGradT {
    static constexpr int K = 1;
    static constexpr bool kChanQueue = false;
    static constexpr bool kImage = false;
    static constexpr bool kTangent = false;
    static constexpr bool kRewalk = true;
    template <bool kAffine>
    static C5_HD double crossing(const WalkParams& P, double px, double py, uint32_t pixel, int leaf, double z_in,
                                 Pairs<1>& v, uint32_t& steps, uint32_t& error) {
        if constexpr (kAffine) {
            LamFields acc{v};
            return crossing_walk<true>(P, px, py, leaf, z_in, acc, steps, error);
        } else {
            const GradParams& G = static_cast<const GradParams&>(P);
            GradFields acc{G, v, grad_ray<kViewG>(G, pixel), 0};
            return crossing_walk<false>(P, px, py, leaf, z_in, acc, steps, error);
        }
    }
};
using CellsGrad = CellsGradT<false>;
using CellsGradView = CellsGradT<true>;

// ---- forward mode (c5_render_jvp) ------------------------------------------------------------------------
// The Jacobian-vector product of the pre-cast image along a field direction (v_alpha, v_Q), carried forward
// along the ray beside {tau, I}, in the walk's +z order (DESIGN.md §5c, "Forward mode"). With the partials of
// the gradient pass above, a segment does
//   dtau  += v_alpha dz                                                   (every segment)
//   dI_out = e dI_in + (-m / a^) v_Q + (s x dz f(x) - I_in dz e) v_a^       (a^ >= DBL_EPSILON; else unchanged)
// with v_a^ = v_alpha where alpha <= limit, else 0: the coefficients grad_segment multiplies by g_I T (except that
// e = exp(-x) past x = 1/2, where 1 + m loses digits), so <g, J v> and <J^T g, v> agree to rounding. A crossing
// walked affinely (I_out = A + B I_in) also carries the tangent of B, held in gain[1]:
// dI_out = dA + dB I_in + B dI_in, and per segment dB_out = e dB_in - B_in dz e v_a^.
// Pair 0 goes through the operations of segment(), so it is c5_render_raw's {tau, I} bit for bit; dtau is
// added like tau, so v_alpha = alpha gives dtau == tau bit for bit.
template <bool kAffine>
C5_HD void jvp_segment(double alpha, double s, double va, double vq, double limit, double dzv, Pairs<2>& v) {
    v.tau[0] += dzv * alpha;
    v.tau[1] += dzv * va;
    double a_c = alpha;
    if (a_c > limit) a_c = limit;
    if (!(a_c < DBL_EPSILON)) {
        const double m = expm1(-a_c * dzv);
        const double x = mul_rn(a_c, dzv);
        // 1 + m has an absolute error of an ulp of 1: past x = 1/2 it would cost the tangent digits in
        // proportion to 1 / e (at x = 16, e ~ 1e-7: seven), so e is taken from exp there
        const double e = x < 0.5 ? 1.0 + m : exp(-x);
        const double i_in = v.inten[0];
        double di = v.inten[1] * e + (-m / a_c) * vq;
        if (alpha <= limit) {
            di += (s * x * dzv * grad_f(x, m) - i_in * dzv * e) * va;
            if (kAffine) v.gain[1] = v.gain[1] * e - (v.gain[0] * dzv * e) * va;
        } else if (kAffine) {
            v.gain[1] = v.gain[1] * e;
        }
        v.inten[1] = di;
        v.inten[0] = i_in - (s - i_in) * m;
        if (kAffine) v.gain[0] *= 1.0 + m;
    }
}

template <bool kAffine>
struct JvpFields {
    const double* dir;
    Pairs<2>& v;
    TetFields c;
    double va, vq;
    C5_HD void fetch(const WalkParams& P, int t) {
        c.load(P.fields, t);
#ifdef __CUDA_ARCH__
        asm volatile("ld.global.nc.v2.f64 {%0,%1}, [%2];" : "=d"(va), "=d"(vq) : "l"(dir + 2 * static_cast<size_t>(t)));
#else
        va = dir[2 * static_cast<size_t>(t)];
        vq = dir[2 * static_cast<size_t>(t) + 1];
#endif
    }
    C5_HD void step(const WalkParams& P, double dzv) {
        jvp_segment<kAffine>(c.alpha, c.s, va, vq, P.alpha_limit, dzv, v);
    }
};

// {tau, I} of CellsF64 and {dtau, dI}; P is the WalkParams of a JvpParams. A deferred ray's two pairs wait in
// ch_queue.
struct CellsJvp {
    static constexpr int K = 2;
    static constexpr bool kChanQueue = true;
    static constexpr bool kImage = true;
    static constexpr bool kTangent = true;
    static constexpr bool kRewalk = false;
    template <bool kAffine>
    static C5_HD double crossing(const WalkParams& P, double px, double py, uint32_t, int leaf, double z_in, Pairs<2>& v,
                                 uint32_t& steps, uint32_t& error) {
        if (kAffine) v.gain[1] = 0.0; // an affine crossing starts from reset pairs: B = 1, and dB = 0
        JvpFields<kAffine> acc{static_cast<const JvpParams&>(P).dir, v};
        return crossing_walk<kAffine>(P, px, py, leaf, z_in, acc, steps, error);
    }
};

C5_HD void store2(double* p, double a, double b) {
#ifdef __CUDA_ARCH__
    *reinterpret_cast<double2*>(p) = make_double2(a, b);
#else
    p[0] = a;
    p[1] = b;
#endif
}

// ---- one ray (pixel kernel) ------------------------------------------------------------------------

template <int K>
struct RayResult {
    Pairs<K> v;
    uint32_t steps;
    uint32_t error;
    uint32_t deferred; // handed to the grazing-ray kernel: the pixel is stored there
};

// A ray's FIRST query is a nearest-hit search (cap 1: most rays enter once and the search stays as
// cheap as it can be). After the first exit ONE more query asks for the next kInline entries above:
// for a convex mesh it finds nothing after visiting a handful of nodes; a cavity gives one or two,
// which are walked here. A full list, or a search that runs out of budget, means a grazing ray: its
// state goes to the deferred queue.
//
// The four phases are written out and separated by __syncwarp over the lanes that trace (`tracing`,
// a ballot taken where the warp is still whole): the searches and the walks must each run with the
// warp CONVERGED — a search is hundreds of dependent loads and a walk hundreds of steps; executed
// lane group by lane group they cost a multiple. Left to the compiler's reconvergence analysis this
// was fragile: an innocent change to the search loop (a second exit) made it stop reconverging
// after the search and the whole kernel ran 1.75 x slower (8.3 vs 4.7 ms on C3).
C5_HD void sync_lanes(unsigned lanes) {
#ifdef __CUDA_ARCH__
    __syncwarp(lanes);
#else
    (void)lanes;
#endif
}

template <class F>
C5_HD RayResult<F::K> trace_ray(const WalkParams& P, double px, double py, uint32_t pixel, unsigned tracing) {
    RayResult<F::K> r{};
    double z_after = -INFINITY;
    EntryList<kInline> L;

    // A: nearest entry
    bool defer = !bvh_collect_entries(P, px, py, z_after, L, 1, P.query_budget);
    sync_lanes(tracing);
    // B: first crossing
    const bool entered = !defer && L.n > 0;
    if (entered) {
        z_after = F::template crossing<false>(P, px, py, pixel, L.leaf[0], L.z[0], r.v, r.steps, r.error);
    }
    sync_lanes(tracing);
    // C: anything above the exit?
    L.n = 0;
    if (entered && !r.error) {
        const bool searched = bvh_collect_entries(P, px, py, z_after, L, kInline, P.query_budget);
        defer = !searched || L.n == kInline; // too many boxes in the way, or too many entries
    }
    sync_lanes(tracing);
    // D: the few re-entries of a cavity or a dent
    for (int e = 0; e < kInline - 1; e++) {
        // an entry at or below the ray's position is already behind it (two boundary faces sharing
        // the edge the ray passes through report the same depth)
        if (!defer && e < L.n && L.z[e] > z_after && !r.error) {
            z_after = F::template crossing<false>(P, px, py, pixel, L.leaf[e], L.z[e], r.v, r.steps, r.error);
        }
        sync_lanes(tracing);
    }
    if (defer) {
#ifdef __CUDA_ARCH__
        const unsigned long long slot = atomicAdd(&P.counters[kDeferred], 1ull);
#else
        const unsigned long long slot = P.counters[kDeferred]++;
#endif
        // read by the grazing-ray kernel, which is launched after this one on the same stream
        DeferredRay& q = P.queue[slot];
        q.tau = F::kChanQueue ? 0.0 : r.v.tau[0];
        q.inten = F::kChanQueue ? 0.0 : r.v.inten[0];
        q.z_after = z_after;
        q.pixel = pixel;
        q.steps = r.steps;
        if (F::kChanQueue) {
#pragma unroll
            for (int c = 0; c < F::K; c++) store2(P.ch_queue + 2 * (slot * F::K + c), r.v.tau[c], r.v.inten[c]);
        }
        r.deferred = 1;
    }
    return r;
}

// ---- grazing rays ----------------------------------------------------------------------------------
// A deferred ray has many crossings (~110 on the C3 README view, each a few tets long). Two facts
// make it parallel: (1) its crossings are independent once their entry faces are known — tau is a
// sum and I an affine recurrence, so crossing k yields (tau_k, A_k, B_k) and the ray's values are
// their composition in z order; (2) collecting the entry faces is a BVH traversal with a wide
// frontier. So one WARP takes one ray: the lanes expand 32 BVH nodes per round from a shared stack,
// rank-sort the entries found, walk 32 crossings at a time and fold the results in order.

template <int K>
struct RayAcc {
    Pairs<K> v; // gain unused
    double z_after;
    uint32_t steps, error;
};

// A deferred ray as trace_ray left it.
template <class F>
C5_HD RayAcc<F::K> load_deferred(const WalkParams& P, unsigned long long slot) {
    const DeferredRay& q = P.queue[slot];
    RayAcc<F::K> a;
    if (F::kChanQueue) {
#pragma unroll
        for (int c = 0; c < F::K; c++) {
            a.v.tau[c] = P.ch_queue[2 * (slot * F::K + c)];
            a.v.inten[c] = P.ch_queue[2 * (slot * F::K + c) + 1];
        }
    } else {
        a.v.tau[0] = q.tau;
        a.v.inten[0] = q.inten;
    }
    a.z_after = q.z_after;
    a.steps = q.steps;
    a.error = 0;
    return a;
}

// Folds crossing (z_in -> z_out) into the ray unless the ray is already past its entry. kTangent (CellsJvp):
// pair 1 is the tangent of pair 0 and its gain the tangent of pair 0's, so the fold is the 2 x 2 lower-triangular
// map dI_out = dA + dB I_in + B dI_in beside I_out = A + B I_in.
template <int K, bool kTangent = false>
C5_HD void compose_crossing(RayAcc<K>& a, double z_in, double z_out, const Pairs<K>& k, uint32_t steps_k,
                            uint32_t error_k) {
    if (!(z_in > a.z_after)) return;
    if constexpr (kTangent) {
        a.v.tau[0] += k.tau[0];
        a.v.tau[1] += k.tau[1];
        a.v.inten[1] = k.inten[1] + k.gain[1] * a.v.inten[0] + k.gain[0] * a.v.inten[1];
        a.v.inten[0] = k.inten[0] + k.gain[0] * a.v.inten[0];
    } else {
#pragma unroll
        for (int c = 0; c < K; c++) {
            a.v.tau[c] += k.tau[c];
            a.v.inten[c] = k.inten[c] + k.gain[c] * a.v.inten[c];
        }
    }
    a.steps += steps_k;
    a.error |= error_k;
    a.z_after = z_out;
}

// Serial form (one thread does everything): the host-loop build, and the reference the warp
// version is tested against. Same crossing function, same composition, same re-walk.
template <class F>
C5_HD RayAcc<F::K> graze_ray_serial(const WalkParams& P, unsigned long long slot, double px, double py) {
    RayAcc<F::K> a = load_deferred<F>(P, slot);
    const uint32_t pixel = P.queue[slot].pixel;
    EntryList<kSerialList> L;
    int crossings = 0;
    while (!a.error) {
        if (!bvh_collect_entries(P, px, py, a.z_after, L, P.serial_cap, 0x7FFFFFFF)) a.error = 1; // stack overflow
        for (int e = 0; e < L.n; e++) {
            if (!(L.z[e] > a.z_after)) continue;
            Pairs<F::K> k;
            k.reset();
            uint32_t steps_k = 0, error_k = 0;
            const double z_out = F::template crossing<true>(P, px, py, pixel, L.leaf[e], L.z[e], k, steps_k, error_k);
            if constexpr (F::kRewalk) {
                Pairs<F::K> entered = a.v;
                uint32_t steps_g = 0, error_g = 0;
                F::template crossing<false>(P, px, py, pixel, L.leaf[e], L.z[e], entered, steps_g, error_g);
            }
            compose_crossing<F::K, F::kTangent>(a, L.z[e], z_out, k, steps_k, error_k);
            if (++crossings > 65536) a.error = 1;
        }
        if (L.n < P.serial_cap) break;
    }
    return a;
}

C5_HD double __longlong_as_double_hd(long long bits) {
#ifdef __CUDA_ARCH__
    return __longlong_as_double(bits);
#else
    double v;
    memcpy(&v, &bits, sizeof(v));
    return v;
#endif
}

// Pair k of the band buffer.
C5_HD void store_pair(const WalkParams& P, size_t k, double t, double v) {
    if (P.round_float) { // plane.cpp:165-166 then object2d.cpp:19-20
        t = static_cast<double>(static_cast<float>(t));
        v = static_cast<double>(static_cast<float>(v));
    }
    store2(P.out + 2 * k, t, v);
}

template <int K, int... C>
C5_HD void store_pairs(const WalkParams& P, size_t o, const double (&tau)[K], const double (&inten)[K],
                       std::integer_sequence<int, C...>) {
    (store_pair(P, o * K + C, tau[C], inten[C]), ...);
}

template <int K>
C5_HD void store_pixel(const WalkParams& P, int i, int j, const double (&tau)[K], const double (&inten)[K],
                       uint32_t steps) {
    const size_t o = static_cast<size_t>(j - P.row_begin) * P.res_x + i;
    store_pairs(P, o, tau, inten, std::make_integer_sequence<int, K>{});
    if (P.steps) P.steps[o] = steps;
}

// Pixels of the band outside the rectangle the walk covers: background (or solid), n pairs wide.
C5_HD bool background_pixel(const WalkParams& P, int n, int i, int j) {
    const bool solid = P.mask && P.mask[static_cast<size_t>(j) * P.res_x + i];
    const double v = solid ? __longlong_as_double_hd(0x7FF8000000000000ll) : 0.0; // quiet NaN (config.hpp:26-27)
    const size_t o = static_cast<size_t>(j - P.row_begin) * P.res_x + i;
    for (int c = 0; c < n; c++) store2(P.out + 2 * (o * n + c), v, v);
    if (P.steps) P.steps[o] = 0;
    return solid;
}

// ---- warp-cooperative form ---------------------------------------------------------------------------
constexpr int kGrazeWarps = 2;    // warps (= rays in flight) per block: small blocks fit into the gaps the pixel kernels leave
constexpr int kGrazeBlocksPerSm = 12; // grid of the grazing-ray kernel (persistent warps drawing tickets). The kernel is
                                      // latency-bound: C3 whole view alone 0.80 ms with 4 blocks per SM, 0.57 with 8, 0.50 with 12,
                                      // 0.51 with 16 (profiles/r02_exp_graze_blocks.jsonl); blocks that find the queue empty leave at once
constexpr int kGrazeList = 256;   // entries per collection; more are fetched by another round
constexpr int kGrazeStack = 512;  // shared traversal stack per warp ...
constexpr int kGrazeSlack = 128;  // ... plus room for one wide round and a depth-first tail
constexpr int kGrazePerLane = kGrazeList / 32;

struct GrazeSmem {
    double z[kGrazeList];
    int leaf[kGrazeList];
    int stack[kGrazeStack + kGrazeSlack];
};

// Sorts S.z / S.leaf [0, n) by (z, leaf): every lane ranks its own <= 8 entries against all n
// (broadcast reads), then scatters them. n <= 256, so this is a few thousand compares per lane.
__device__ __forceinline__ void graze_sort(GrazeSmem& S, int n, int lane) {
    double zr[kGrazePerLane];
    int lr[kGrazePerLane], rank[kGrazePerLane];
#pragma unroll
    for (int q = 0; q < kGrazePerLane; q++) {
        const int k = q * 32 + lane;
        zr[q] = k < n ? S.z[k] : INFINITY;
        lr[q] = k < n ? S.leaf[k] : 0x7FFFFFFF;
        rank[q] = 0;
    }
    for (int m = 0; m < n; m++) {
        const double zm = S.z[m];
        const int lm = S.leaf[m];
#pragma unroll
        for (int q = 0; q < kGrazePerLane; q++) rank[q] += entry_before(zm, lm, zr[q], lr[q]) ? 1 : 0;
    }
    __syncwarp();
#pragma unroll
    for (int q = 0; q < kGrazePerLane; q++) {
        if (q * 32 + lane < n) {
            S.z[rank[q]] = zr[q];
            S.leaf[rank[q]] = lr[q];
        }
    }
    __syncwarp();
}

// All entry faces above z_after under (px, py), collected by the whole warp into S (sorted).
// Returns their number; `truncated` is set if the list overflowed and only the lowest part was kept
// (everything up to the last kept entry is present: the caller walks it and asks again).
__device__ __forceinline__ int graze_collect(const WalkParams& P, GrazeSmem& S, double px, double py, double z_after,
                                             int lane, bool& truncated) {
    const unsigned full = 0xFFFFFFFFu;
    const unsigned lt = (1u << lane) - 1u;
    const float fx_lo = f_round_down(px), fx_hi = f_round_up(px);
    const float fy_lo = f_round_down(py), fy_hi = f_round_up(py);
    int sp = 1, n = 0;
    double z_cap = INFINITY;
    truncated = false;
    if (lane == 0) S.stack[0] = 0;
    __syncwarp();
    while (sp > 0) {
        if (n > P.graze_cap - 64) { // a round appends at most 64: keep the lowest half, forget the rest
            graze_sort(S, n, lane);
            n = P.graze_cap / 2;
            z_cap = S.z[n - 1];
            truncated = true;
            __syncwarp();
        }
        // 32 nodes per round while the stack has room for their 64 children; else depth first
        const int take = sp <= kGrazeStack - 64 ? (sp < 32 ? sp : 32) : 1;
        const int node = lane < take ? S.stack[sp - 1 - lane] : -1;
        sp -= take;
        __syncwarp();
        bool h0 = false, h1 = false;
        int2 ch = make_int2(0, 0);
        if (node >= 0) {
            const BvhNode* nd = P.nodes + node;
            const float4 bx = *reinterpret_cast<const float4*>(nd->xlo);
            const float4 by = *reinterpret_cast<const float4*>(nd->ylo);
            const float4 bz = *reinterpret_cast<const float4*>(nd->zlo);
            ch = *reinterpret_cast<const int2*>(nd->child);
            h0 = fx_hi >= bx.x && fx_lo <= bx.z && fy_hi >= by.x && fy_lo <= by.z &&
                 static_cast<double>(bz.z) > z_after && static_cast<double>(bz.x) <= z_cap;
            h1 = fx_hi >= bx.y && fx_lo <= bx.w && fy_hi >= by.y && fy_lo <= by.w &&
                 static_cast<double>(bz.w) > z_after && static_cast<double>(bz.y) <= z_cap;
        }
        double z0 = 0.0, z1 = 0.0;
        const bool e0 = h0 && ch.x < 0 && entry_depth(P, ~ch.x, px, py, z_after, z0) && z0 <= z_cap;
        const bool e1 = h1 && ch.y < 0 && entry_depth(P, ~ch.y, px, py, z_after, z1) && z1 <= z_cap;
        unsigned m = __ballot_sync(full, e0);
        if (e0) {
            const int pos = n + __popc(m & lt);
            S.z[pos] = z0;
            S.leaf[pos] = ~ch.x;
        }
        n += __popc(m);
        m = __ballot_sync(full, e1);
        if (e1) {
            const int pos = n + __popc(m & lt);
            S.z[pos] = z1;
            S.leaf[pos] = ~ch.y;
        }
        n += __popc(m);
        const bool i0 = h0 && ch.x >= 0, i1 = h1 && ch.y >= 0;
        m = __ballot_sync(full, i0);
        if (i0) S.stack[sp + __popc(m & lt)] = ch.x;
        sp += __popc(m);
        m = __ballot_sync(full, i1);
        if (i1) S.stack[sp + __popc(m & lt)] = ch.y;
        sp += __popc(m);
        __syncwarp();
    }
    graze_sort(S, n, lane);
    return n;
}

template <class F>
__device__ __forceinline__ void graze_block(const WalkParams& P) {
    __shared__ GrazeSmem smem[kGrazeWarps];
    const unsigned full = 0xFFFFFFFFu;
    const int lane = threadIdx.x & 31;
    GrazeSmem& S = smem[threadIdx.x >> 5];
    // Launched after the pixel kernel on the same stream, so the queue and its length are final.
    // The length lives on the device: a fixed grid of persistent warps draws tickets until they run
    // out (an empty queue costs one short launch).
    const unsigned long long n_rays = P.counters[kDeferred];
    while (true) {
        unsigned long long ticket = 0;
        if (lane == 0) ticket = atomicAdd(&P.counters[kTicket], 1ull);
        ticket = __shfl_sync(full, ticket, 0);
        if (ticket >= n_rays) break;
        const uint32_t q_pixel = P.queue[ticket].pixel;
        const int i = static_cast<int>(q_pixel % static_cast<uint32_t>(P.res_x));
        const int j = static_cast<int>(q_pixel / static_cast<uint32_t>(P.res_x));
        const double px = P.xs[i], py = P.ys[j];
        RayAcc<F::K> a = load_deferred<F>(P, ticket);
        const uint32_t q_steps = a.steps;
        int crossings = 0;
        bool truncated = true;
        while (truncated && !a.error) {
            const int n = graze_collect(P, S, px, py, a.z_after, lane, truncated);
            for (int base = 0; base < n; base += 32) {
                const int k = base + lane;
                const bool have = k < n;
                const double z_in = have ? S.z[k] : INFINITY;
                double z_out = z_in;
                Pairs<F::K> f;
                f.reset();
                uint32_t steps_k = 0, error_k = 0;
                if (have && z_in > a.z_after) { // a is the same in every lane
                    z_out = F::template crossing<true>(P, px, py, q_pixel, S.leaf[k], z_in, f, steps_k, error_k);
                }
                const int cnt = n - base < 32 ? n - base : 32;
                Pairs<F::K> entered = a.v; // kRewalk: the pairs this lane's crossing is entered with ...
                bool taken = false;        // ... and whether the fold takes it
                for (int l = 0; l < cnt; l++) {
                    Pairs<F::K> g;
#pragma unroll
                    for (int c = 0; c < F::K; c++) {
                        g.tau[c] = __shfl_sync(full, f.tau[c], l);
                        g.inten[c] = __shfl_sync(full, f.inten[c], l);
                        g.gain[c] = __shfl_sync(full, f.gain[c], l);
                    }
                    const double z_l = __shfl_sync(full, z_in, l);
                    if constexpr (F::kRewalk) {
                        if (lane == l) {
                            entered = a.v;
                            taken = z_l > a.z_after;
                        }
                    }
                    compose_crossing<F::K, F::kTangent>(a, z_l, __shfl_sync(full, z_out, l), g,
                                                        __shfl_sync(full, steps_k, l), __shfl_sync(full, error_k, l));
                }
                if constexpr (F::kRewalk) {
                    if (taken) {
                        uint32_t steps_g = 0, error_g = 0;
                        F::template crossing<false>(P, px, py, q_pixel, S.leaf[k], z_in, entered, steps_g, error_g);
                    }
                }
            }
            crossings += n;
            if (crossings > 65536) a.error = 1;
            __syncwarp();
        }
        if constexpr (F::kImage) {
            if (lane == 0) {
                store_pixel(P, i, j, a.v.tau, a.v.inten, a.steps);
                const unsigned long long more = a.steps - q_steps;
                if (more) {
                    atomicAdd(&P.counters[kSteps], more);
                    atomicAdd(&P.row_cost[j], more);
                    if (q_steps == 0) atomicAdd(&P.counters[kHitPixels], 1ull); // deferred before its first step
                }
                if (a.error) atomicAdd(&P.counters[kWalkErrors], 1ull);
            }
        }
    }
}

// ---- kernel ----------------------------------------------------------------------------------------

// Morton decode: bits 0, 2, 4, ... of v (x of a local Morton index m; y is compact_bits(m >> 1))
C5_HD int compact_bits(uint32_t v) {
    v &= 0x55555555u;
    v = (v | (v >> 1)) & 0x33333333u;
    v = (v | (v >> 2)) & 0x0F0F0F0Fu;
    v = (v | (v >> 4)) & 0x00FF00FFu;
    return static_cast<int>(v & 0xFFFFu);
}

// The sort key of a ray that took `cost` steps in the previous view, in a region whose least nonzero cost is
// `least`: 0 for no steps, then one bucket per 2^kBucketShift steps from the least up, the last one open.
C5_HD int cost_bucket(uint32_t cost, uint32_t least) {
    if (cost == 0) return 0;
    const uint32_t b = (cost >> kBucketShift) - (least >> kBucketShift);
    return 1 + static_cast<int>(b < kBuckets - 2 ? b : kBuckets - 2);
}

// The cost of local Morton index m of region (rx, ry); pixels outside the rectangle cost 0.
C5_HD uint32_t region_cost(const WalkParams& P, int rx, int ry, uint32_t m) {
    const int i = P.i0 + rx * kRegion + compact_bits(m), j = P.j0 + ry * kRegion + compact_bits(m >> 1);
    return i < P.i1 && j < P.j1 ? P.cost[static_cast<size_t>(j) * P.res_x + i] : 0u;
}

// A region keeps the Morton order unless sorting it saves at least kMinSaving percent of its warps' issue time,
// modelled as the sum over its warps of the most steps any of their rays takes ("warp steps"). Where the previous
// view's step counts are even (the oblique view, the 50 M-tet C5t) a sort saves little, and its blocks, spread over
// the region instead of one compact 16 x 8 patch, share fewer tets in L1: those views then walk as they did in
// Morton order. Measured (profiles/r14_ray_order_threshold_one_b200.jsonl): sorting every region (0 %) costs C5t 1.2 %
// against the parent; 10 % keeps C3's gain (4.63 -> 4.14 ms) and C5t within 0.3 %; 20 % loses most of C3's gain.
constexpr uint32_t kMinSaving = 10;

// Warp steps of the sorted order: the last ray of a sorted warp takes the most steps of its warp, up to the width
// of a bucket (one step, kBucketShift = 0) and the last, open bucket.
C5_HD bool sort_pays(uint32_t morton_steps, uint32_t sorted_steps) {
    return static_cast<uint64_t>(sorted_steps) * 100u <= static_cast<uint64_t>(morton_steps) * (100u - kMinSaving);
}

// One region's order, by one thread (the host-loop build): a stable counting sort, kept if sort_pays. cost[m] is
// local Morton index m's.
C5_HD void order_region(const uint16_t* cost, uint16_t* order) {
    uint32_t least = 0xFFFFu;
    for (int m = 0; m < kRegionPix; m++) {
        if (cost[m] && cost[m] < least) least = cost[m];
    }
    int start[kBuckets] = {};
    for (int m = 0; m < kRegionPix; m++) start[cost_bucket(cost[m], least)]++;
    for (int b = 0, sum = 0; b < kBuckets; b++) {
        const int n = start[b];
        start[b] = sum;
        sum += n;
    }
    for (int m = 0; m < kRegionPix; m++) order[start[cost_bucket(cost[m], least)]++] = static_cast<uint16_t>(m);
    uint32_t morton_steps = 0, sorted_steps = 0;
    for (int w = 0; w < kRegionPix; w += 32) {
        uint32_t most = 0;
        for (int l = 0; l < 32; l++) most = cost[w + l] > most ? cost[w + l] : most;
        morton_steps += most;
        sorted_steps += cost[order[w + 31]];
    }
    if (!sort_pays(morton_steps, sorted_steps)) {
        for (int m = 0; m < kRegionPix; m++) order[m] = static_cast<uint16_t>(m);
    }
}

// The same by one block per region, kOrderThreads threads taking kOrderItems local Morton indices each (m = q
// kOrderThreads + thread). The bits of words[b][w] are the indices 32 w .. 32 w + 31 that fall into bucket b (one
// __match_any_sync per warp of indices); an index's place is the start of its bucket plus the members of that
// bucket below it. Shared memory is used here and not in the walk kernels, whose L1 capacity serves the tets.
constexpr int kOrderThreads = kRegionPix < 1024 ? kRegionPix : 1024;
constexpr int kOrderItems = kRegionPix / kOrderThreads;
constexpr int kOrderWords = kRegionPix / 32;
static_assert(sizeof(uint32_t) * kBuckets * (kOrderWords + 1) <= 40 * 1024, "order_rays' bitmaps fit static shared memory");

__global__ void __launch_bounds__(kOrderThreads) order_rays(const WalkParams P) {
    __shared__ uint32_t words[kBuckets][kOrderWords + 1]; // (+1: lanes reading different buckets hit different banks)
    __shared__ uint32_t start[kBuckets];
    __shared__ uint32_t least_all, morton_steps, sorted_steps, nonzero;
    const unsigned full = 0xFFFFFFFFu;
    const int lane = threadIdx.x & 31;
    const int rx = static_cast<int>(blockIdx.x) % P.n_regions_x, ry = static_cast<int>(blockIdx.x) / P.n_regions_x;
    for (int k = threadIdx.x; k < kBuckets * (kOrderWords + 1); k += kOrderThreads) (&words[0][0])[k] = 0u;
    if (threadIdx.x == 0) {
        least_all = 0xFFFFu;
        morton_steps = 0;
        sorted_steps = 0;
        nonzero = 0;
    }
    uint32_t cost[kOrderItems];
    uint32_t least = 0xFFFFu, most = 0, rays = 0;
#pragma unroll
    for (int q = 0; q < kOrderItems; q++) {
        cost[q] = region_cost(P, rx, ry, static_cast<uint32_t>(q * kOrderThreads + threadIdx.x));
        if (cost[q] && cost[q] < least) least = cost[q];
        most += __reduce_max_sync(full, cost[q]); // the warp steps of Morton warp q
        rays += __popc(__ballot_sync(full, cost[q] != 0));
    }
    least = __reduce_min_sync(full, least);
    __syncthreads();
    if (lane == 0) {
        atomicMin(&least_all, least);
        atomicAdd(&morton_steps, most);
        atomicAdd(&nonzero, rays);
    }
    __syncthreads();
    least = least_all;
    // The sort puts the rays with steps last, ceil(nonzero / 32) warps of them, and the last ray of each of those
    // warps takes at least `least` steps: when even that bound saves too little, the region keeps the Morton order
    // without sorting (most regions of evenly costed views: the kernel then takes a fraction of its time).
    if (nonzero == 0 || !sort_pays(morton_steps, (nonzero + 31u) / 32u * least)) {
#pragma unroll
        for (int q = 0; q < kOrderItems; q++) {
            const uint32_t m = static_cast<uint32_t>(q * kOrderThreads + threadIdx.x);
            P.order[static_cast<size_t>(blockIdx.x) * kRegionPix + m] = static_cast<uint16_t>(m);
        }
        return;
    }
    int bucket[kOrderItems];
    unsigned same[kOrderItems];
#pragma unroll
    for (int q = 0; q < kOrderItems; q++) {
        bucket[q] = cost_bucket(cost[q], least);
        same[q] = __match_any_sync(full, bucket[q]);
        if (lane == __ffs(same[q]) - 1) words[bucket[q]][(q * kOrderThreads + threadIdx.x) >> 5] = same[q];
    }
    __syncthreads();
    if (threadIdx.x < 32) { // exclusive scan of the bucket sizes, kBuckets / 32 consecutive buckets per lane
        constexpr int kPer = kBuckets / 32;
        uint32_t n[kPer], sum = 0;
#pragma unroll
        for (int k = 0; k < kPer; k++) {
            n[k] = 0;
            for (int w = 0; w < kOrderWords; w++) n[k] += __popc(words[lane * kPer + k][w]);
            sum += n[k];
        }
        uint32_t below = sum;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t o = __shfl_up_sync(full, below, d);
            if (lane >= d) below += o;
        }
        below -= sum;
#pragma unroll
        for (int k = 0; k < kPer; k++) {
            start[lane * kPer + k] = below;
            below += n[k];
        }
    }
    __syncthreads();
    const unsigned lower = (1u << lane) - 1u;
    uint32_t pos[kOrderItems];
#pragma unroll
    for (int q = 0; q < kOrderItems; q++) {
        const uint32_t m = static_cast<uint32_t>(q * kOrderThreads + threadIdx.x);
        pos[q] = start[bucket[q]] + __popc(same[q] & lower);
        for (uint32_t w = 0; w < (m >> 5); w++) pos[q] += __popc(words[bucket[q]][w]);
        if ((pos[q] & 31u) == 31u) atomicAdd(&sorted_steps, cost[q]);
    }
    __syncthreads();
    const bool sorted = sort_pays(morton_steps, sorted_steps);
#pragma unroll
    for (int q = 0; q < kOrderItems; q++) {
        const uint32_t m = static_cast<uint32_t>(q * kOrderThreads + threadIdx.x);
        P.order[static_cast<size_t>(blockIdx.x) * kRegionPix + (sorted ? pos[q] : m)] = static_cast<uint16_t>(m);
    }
}
static_assert(kBuckets % 32 == 0, "the scan gives each lane the same number of buckets");

template <class F>
__device__ __forceinline__ void walk_block(const WalkParams& P) {
    // block b takes slots kBlock (b % kBlocksPerRegion) .. of region b / kBlocksPerRegion's order; regions are in
    // row-major order, so the blocks resident at one time cover a few rows of regions
    const int region = static_cast<int>(blockIdx.x) / kBlocksPerRegion;
    const int i_lo = P.i0 + (region % P.n_regions_x) * kRegion, j_lo = P.j0 + (region / P.n_regions_x) * kRegion;

    // Regions that cannot see the mesh (outside the root's two boxes) skip the rays.
    const int i_hi = min(i_lo + kRegion, P.i1) - 1, j_hi = min(j_lo + kRegion, P.j1) - 1;
    bool region_sees_mesh;
    {
        const BvhNode* root = P.nodes;
        const float x0 = f_round_down(P.xs[i_lo]), x1 = f_round_up(P.xs[i_hi]);
        const float y0 = f_round_down(P.ys[j_lo]), y1 = f_round_up(P.ys[j_hi]);
        const bool s0 = x1 >= root->xlo[0] && x0 <= root->xhi[0] && y1 >= root->ylo[0] && y0 <= root->yhi[0];
        const bool s1 = x1 >= root->xlo[1] && x0 <= root->xhi[1] && y1 >= root->ylo[1] && y0 <= root->yhi[1];
        region_sees_mesh = s0 || s1;
    }

    const int lane = threadIdx.x & 31;
    const uint32_t m = __ldg(P.order + static_cast<size_t>(blockIdx.x) * kBlock + threadIdx.x);
    const int i = i_lo + compact_bits(m);
    const int j = j_lo + compact_bits(m >> 1);
    const bool live = i < P.i1 && j < P.j1;

    RayResult<F::K> res{};
    bool solid = false;
    if (live) solid = P.mask && P.mask[static_cast<size_t>(j) * P.res_x + i];
    // the lanes that will trace a ray, agreed on while the warp is whole (trace_ray synchronises on it)
    const unsigned tracing = __ballot_sync(0xFFFFFFFFu, live && !solid && region_sees_mesh);
    if (live) {
        if (solid) {
            if (F::kImage) {
                double nan[F::K];
                fill_pairs(nan, __longlong_as_double(0x7FF8000000000000ll), std::make_integer_sequence<int, F::K>{}); // quiet NaN (config.hpp:26-27)
                store_pixel(P, i, j, nan, nan, 0);
            }
        } else {
            if (region_sees_mesh) {
                res = trace_ray<F>(P, P.xs[i], P.ys[j],
                                   static_cast<uint32_t>(j) * static_cast<uint32_t>(P.res_x) + static_cast<uint32_t>(i),
                                   tracing);
            }
            if (F::kImage && !res.deferred) store_pixel(P, i, j, res.v.tau, res.v.inten, res.steps);
        }
        // the next view's order (a deferred ray counts the steps it took here)
        P.cost[static_cast<size_t>(j) * P.res_x + i] = static_cast<uint16_t>(min(res.steps, 0xFFFFu));
    }

    // statistics: one atomic per warp per counter, one per row the warp's rays lie on for the row costs
    const unsigned full = 0xFFFFFFFFu;
    for (unsigned rows = full; rows;) { // the same trips in every lane
        const int first = __ffs(rows) - 1;
        const int jr = __shfl_sync(full, j, first);
        const unsigned on_row = __ballot_sync(full, j == jr);
        const unsigned row_steps = __reduce_add_sync(full, j == jr ? res.steps : 0u);
        if (lane == first && row_steps) atomicAdd(&P.row_cost[jr], static_cast<unsigned long long>(row_steps));
        rows &= ~on_row;
    }
    const unsigned warp_steps = __reduce_add_sync(full, res.steps);
    const unsigned hits = __popc(__ballot_sync(full, live && res.steps > 0));
    const unsigned solids = __popc(__ballot_sync(full, solid));
    const unsigned errors = __popc(__ballot_sync(full, res.error != 0));
    if (lane == 0) {
        if (warp_steps) atomicAdd(&P.counters[kSteps], static_cast<unsigned long long>(warp_steps));
        if (hits) atomicAdd(&P.counters[kHitPixels], static_cast<unsigned long long>(hits));
        if (solids) atomicAdd(&P.counters[kSolidPixels], static_cast<unsigned long long>(solids));
        if (errors) atomicAdd(&P.counters[kWalkErrors], static_cast<unsigned long long>(errors));
    }
}

// Resident blocks of 128 threads per SM for the K-channel pixel kernel. K = 1, 2: the most blocks
// whose register cap (72, 80) leaves the kernel free of spills. K >= 3: the occupancy the registers
// ptxas needs without a cap allow (110..128 registers: 4 blocks, 136..150: 3), so the bound only
// records it (-Xptxas -v; the registers per K are in DESIGN.md).
constexpr int chan_blocks_per_sm(int K) {
    return K <= 1 ? 7 : K <= 2 ? 6 : K <= 5 ? 4 : 3;
}

} // namespace

// The product kernels. 8 blocks of 128 threads per SM = 64 registers. With the 64-byte cell that cap
// spilled in the step loop (8.9 ms on C3) and 7 blocks = 72 registers was the best bound (5.41 ms against
// 5.64 with the compiler's own 80). Tracking face slots instead of vertex ids freed the registers: at 64
// the kernel spills 28 bytes, none of them in the step loop (profiles/r09_ptxas_walk.txt,
// r09_sass_step_loop.txt), and C3 takes 4.35 instead of 4.49 ms per view at 7 blocks (one B200,
// profiles/r09_bench_c3_bounds_one_b200.jsonl).
__global__ void __launch_bounds__(kBlock, 8) tet_walk_fp64(const WalkParams P) { walk_block<CellsF64>(P); }
// optional single-precision step geometry (north-star item (d)); entry search and accumulators stay FP64.
// 9 blocks = 56 registers: oblique view 1.90 against 2.03 ms at 8 blocks (same file). Since the pixel order
// (order_rays) it spills 12 bytes outside the step loop (-Xptxas -v).
__global__ void __launch_bounds__(kBlock, 9) tet_walk_fp32(const WalkParams P) { walk_block<CellsF32>(P); }
template <int K>
__global__ void __launch_bounds__(kBlock, chan_blocks_per_sm(K)) tet_walk_ch(const WalkParams P) { walk_block<Channels<K>>(P); }

// The walk's grid only covers the pixel rectangle that can see the mesh (a one-wave row band whose
// grid is 60 % empty tiles fills the SMs unevenly: measured 1.60 M busy cycles on the fullest SM
// against 1.07 M on average, profiles/r01_walk_band_c3.csv). Everything else in the band is background
// or solid and is written by this streaming kernel, n {tau, I} pairs per pixel.
__global__ void __launch_bounds__(256) fill_background(const WalkParams P, int n) {
    const int n_rows = P.row_end - P.row_begin;
    const int64_t k = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
    bool solid = false;
    if (k < static_cast<int64_t>(n_rows) * P.res_x) {
        const int j = P.row_begin + static_cast<int>(k / P.res_x), i = static_cast<int>(k % P.res_x);
        if (!(i >= P.i0 && i < P.i1 && j >= P.j0 && j < P.j1)) solid = background_pixel(P, n, i, j);
    }
    const unsigned solids = __popc(__ballot_sync(0xFFFFFFFFu, solid));
    if ((threadIdx.x & 31) == 0 && solids) atomicAdd(&P.counters[kSolidPixels], static_cast<unsigned long long>(solids));
}

// Grazing rays (deferred by the pixel kernel): persistent warps, one ray per warp at a time.
__global__ void __launch_bounds__(32 * kGrazeWarps) grazing_rays_fp64(const WalkParams P) { graze_block<CellsF64>(P); }
__global__ void __launch_bounds__(32 * kGrazeWarps) grazing_rays_fp32(const WalkParams P) { graze_block<CellsF32>(P); }
template <int K>
__global__ void __launch_bounds__(32 * kGrazeWarps) grazing_rays_ch(const WalkParams P) { graze_block<Channels<K>>(P); }

// The two passes of c5_render_grad: the depth pass stores {tau, I, lam, 0} per pixel, the gradient pass
// adds into grad_alpha / grad_q. Their register counts are in DESIGN.md §5c (-Xptxas -v).
__global__ void __launch_bounds__(kBlock) tet_walk_depth(const WalkParams P) { walk_block<CellsDepth>(P); }
__global__ void __launch_bounds__(kBlock) tet_walk_grad(const GradParams P) { walk_block<CellsGrad>(P); }
__global__ void __launch_bounds__(32 * kGrazeWarps) grazing_rays_depth(const WalkParams P) { graze_block<CellsDepth>(P); }
__global__ void __launch_bounds__(32 * kGrazeWarps) grazing_rays_grad(const GradParams P) { graze_block<CellsGrad>(P); }
// The gradient pass with one {g_tau, g_I} per view (c5_render_flux_grad_device): registers in DESIGN.md §5c.
__global__ void __launch_bounds__(kBlock) tet_walk_grad_view(const GradParams P) { walk_block<CellsGradView>(P); }
__global__ void __launch_bounds__(32 * kGrazeWarps) grazing_rays_grad_view(const GradParams P) {
    graze_block<CellsGradView>(P);
}
// Forward mode (c5_render_jvp): {tau, I, dtau, dI} per pixel. Registers in DESIGN.md §5c.
__global__ void __launch_bounds__(kBlock) tet_walk_jvp(const JvpParams P) { walk_block<CellsJvp>(P); }
__global__ void __launch_bounds__(32 * kGrazeWarps) grazing_rays_jvp(const JvpParams P) { graze_block<CellsJvp>(P); }

namespace {

// The pixel and grazing-ray kernels of each field policy.
template <class F>
struct Kernels;
template <>
struct Kernels<CellsF64> {
    static constexpr void (*walk)(WalkParams) = tet_walk_fp64;
    static constexpr void (*graze)(WalkParams) = grazing_rays_fp64;
};
template <>
struct Kernels<CellsF32> {
    static constexpr void (*walk)(WalkParams) = tet_walk_fp32;
    static constexpr void (*graze)(WalkParams) = grazing_rays_fp32;
};
template <int K>
struct Kernels<Channels<K>> {
    static constexpr void (*walk)(WalkParams) = tet_walk_ch<K>;
    static constexpr void (*graze)(WalkParams) = grazing_rays_ch<K>;
};
template <>
struct Kernels<CellsDepth> {
    static constexpr void (*walk)(WalkParams) = tet_walk_depth;
    static constexpr void (*graze)(WalkParams) = grazing_rays_depth;
};
template <>
struct Kernels<CellsGrad> {
    static constexpr void (*walk)(GradParams) = tet_walk_grad;
    static constexpr void (*graze)(GradParams) = grazing_rays_grad;
};
template <>
struct Kernels<CellsGradView> {
    static constexpr void (*walk)(GradParams) = tet_walk_grad_view;
    static constexpr void (*graze)(GradParams) = grazing_rays_grad_view;
};
template <>
struct Kernels<CellsJvp> {
    static constexpr void (*walk)(JvpParams) = tet_walk_jvp;
    static constexpr void (*graze)(JvpParams) = grazing_rays_jvp;
};

void background_on_host(const WalkParams& P, int n) {
    for (int j = P.row_begin; j < P.row_end; j++) {
        for (int i = 0; i < P.res_x; i++) {
            if (i >= P.i0 && i < P.i1 && j >= P.j0 && j < P.j1) continue;
            if (background_pixel(P, n, i, j)) P.counters[kSolidPixels]++;
        }
    }
}

void order_on_host(const WalkParams& P, int n_regions) {
    uint16_t cost[kRegionPix];
    for (int r = 0; r < n_regions; r++) {
        for (int m = 0; m < kRegionPix; m++) cost[m] = static_cast<uint16_t>(region_cost(P, r % P.n_regions_x, r / P.n_regions_x, m));
        order_region(cost, P.order + static_cast<size_t>(r) * kRegionPix);
    }
}

template <class F>
void walk_on_host(const WalkParams& P) {
    for (int j = P.j0; j < P.j1; j++) {
        for (int i = P.i0; i < P.i1; i++) {
            if (P.mask && P.mask[static_cast<size_t>(j) * P.res_x + i]) {
                P.cost[static_cast<size_t>(j) * P.res_x + i] = 0;
                if (F::kImage) {
                    double nan[F::K];
                    fill_pairs(nan, NAN, std::make_integer_sequence<int, F::K>{});
                    store_pixel(P, i, j, nan, nan, 0);
                }
                P.counters[kSolidPixels]++;
                continue;
            }
            const uint32_t pixel = static_cast<uint32_t>(j) * static_cast<uint32_t>(P.res_x) + static_cast<uint32_t>(i);
            const RayResult<F::K> r = trace_ray<F>(P, P.xs[i], P.ys[j], pixel, 0);
            if (F::kImage && !r.deferred) store_pixel(P, i, j, r.v.tau, r.v.inten, r.steps);
            P.cost[pixel] = static_cast<uint16_t>(std::min(r.steps, 0xFFFFu));
            P.counters[kSteps] += r.steps;
            P.row_cost[j] += r.steps;
            if (r.steps) P.counters[kHitPixels]++;
            if (r.error) P.counters[kWalkErrors]++;
        }
    }
}

template <class F>
void graze_on_host(const WalkParams& P) {
    const unsigned long long n_rays = P.counters[kDeferred];
    for (unsigned long long k = 0; k < n_rays; k++) {
        const DeferredRay& q = P.queue[k];
        const int i = static_cast<int>(q.pixel % static_cast<uint32_t>(P.res_x));
        const int j = static_cast<int>(q.pixel / static_cast<uint32_t>(P.res_x));
        const RayAcc<F::K> a = graze_ray_serial<F>(P, k, P.xs[i], P.ys[j]);
        if constexpr (F::kImage) {
            store_pixel(P, i, j, a.v.tau, a.v.inten, a.steps);
            P.counters[kSteps] += a.steps - q.steps;
            P.row_cost[j] += a.steps - q.steps;
            if (q.steps == 0 && a.steps > 0) P.counters[kHitPixels]++;
            if (a.error) P.counters[kWalkErrors]++;
        }
    }
    P.counters[kTicket] = n_rays;
}

// Policy F's pixel kernel over `grid` blocks, then its grazing-ray kernel for the rays the pixel
// kernel deferred: a fixed grid of persistent warps that draw tickets. The host-loop build runs both
// as loops.
template <class F, class Params>
void launch_rays(DeviceState& d, const WalkLaunch& w, const Params& P, unsigned grid) {
    if (kHostSim) {
        walk_on_host<F>(P);
        count_launch();
        graze_on_host<F>(P);
        return;
    }
    const cudaStream_t ps = w.pixel_stream ? w.pixel_stream : d.stream;
    if (ps != d.stream) wait_for(ps, d.stream, d.ev_side);
    prefer_side_carveout(Kernels<F>::walk, d.device);
    Kernels<F>::walk<<<grid, kBlock, 0, ps>>>(P);
    C5_CUDA(cudaGetLastError());
    if (w.mark_walk_done) C5_CUDA(cudaEventRecord(w.mark_walk_done, ps));
    if (w.mark_walk_done_tl) C5_CUDA(cudaEventRecord(w.mark_walk_done_tl, ps));
    if (ps != d.stream) wait_for(d.stream, ps, d.ev_side);
    if (d.sm_count == 0) C5_CUDA(cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, d.device));
    const unsigned graze_grid = static_cast<unsigned>(d.sm_count) * static_cast<unsigned>(kGrazeBlocksPerSm);
    count_launch();
    prefer_side_carveout(Kernels<F>::graze, d.device);
    Kernels<F>::graze<<<graze_grid, 32 * kGrazeWarps, 0, d.stream>>>(P);
    C5_CUDA(cudaGetLastError());
}

} // namespace

int order_one_region(const uint16_t* cost_rows, uint16_t* order, int32_t* bucket) {
    uint16_t cost[kRegionPix];
    uint32_t least = 0xFFFFu;
    for (uint32_t m = 0; m < kRegionPix; m++) {
        cost[m] = cost_rows[compact_bits(m >> 1) * kRegion + compact_bits(m)];
        if (cost[m] && cost[m] < least) least = cost[m];
    }
    order_region(cost, order);
    for (int m = 0; m < kRegionPix; m++) bucket[m] = cost_bucket(cost[m], least);
    return kRegion;
}

// One view's rays on d.stream: background fill, the ray order, the pixel kernel (on w.pixel_stream when one is
// given), then the grazing-ray kernel for the rays it deferred — four launches in stream order, no kernel ever
// waits for another one. (Round 1
// ran the grazing-ray kernel BESIDE the pixel kernel, spinning on the queue; CUDA promises no forward
// progress between kernels, and with three or four views in flight the ordered form is also the faster
// one: profiles/r02_exp_lanes_graze_after.jsonl against r02_exp_lanes_graze_beside.jsonl.)
void launch_walk(DeviceState& d, const WalkLaunch& w) {
    if (w.precision != 64 && w.precision != 32) fail(C5_E_INVALID, "render: precision must be 64 or 32");
    const bool f32 = w.precision == 32;
    WalkParams P{};
    P.conn = d.conn.p;
    P.fields = d.fields.p;
    P.vrot = d.vrot.p;
    P.bfaces = d.bfaces.p;
    P.nodes = d.nodes.p;
    P.xs = d.xs.p;
    P.ys = d.ys.p;
    P.mask = w.use_mask ? d.mask.p : nullptr;
    P.out = w.out;
    P.steps = w.write_steps ? d.steps.p : nullptr;
    P.counters = w.counters ? w.counters : d.counters.p;
    P.row_cost = w.row_cost ? w.row_cost : d.row_cost.p;
    P.queue = d.queue.p;
    P.res_x = w.res_x;
    P.res_y = w.res_y;
    P.row_begin = w.row_begin;
    P.row_end = w.row_end;
    // the walk covers [i0,i1) x [j0,j1): the caller's estimate of where the mesh can be, cut to the band
    P.i0 = w.i_begin < 0 ? 0 : w.i_begin;
    P.i1 = w.i_end > w.res_x ? w.res_x : w.i_end;
    P.j0 = w.j_begin < w.row_begin ? w.row_begin : w.j_begin;
    P.j1 = w.j_end > w.row_end ? w.row_end : w.j_end;
    const bool empty_rect = P.i0 >= P.i1 || P.j0 >= P.j1;
    if (empty_rect) P.i0 = P.i1 = P.j0 = P.j1 = 0;
    const bool whole_band = P.i0 == 0 && P.i1 == w.res_x && P.j0 == w.row_begin && P.j1 == w.row_end;
    P.n_regions_x = (P.i1 - P.i0 + kRegion - 1) / kRegion;
    const int n_regions = P.n_regions_x * ((P.j1 - P.j0 + kRegion - 1) / kRegion);
    // (sized for the whole image: the rectangle moves from view to view)
    d.ray_order.ensure(static_cast<size_t>((w.res_x + kRegion - 1) / kRegion) * ((w.res_y + kRegion - 1) / kRegion) * kRegionPix);
    P.cost = d.ray_cost.p;
    P.order = d.ray_order.p;
    if (w.pass != kGradPass) {
        d.ray_order_grid[0] = n_regions;
        d.ray_order_grid[1] = P.n_regions_x;
        d.ray_order_grid[2] = kRegion;
        d.ray_order_origin[0] = P.i0;
        d.ray_order_origin[1] = P.j0;
    }
    // c5_debug_set (tests shrink these to reach the overflow paths on small meshes); defaults otherwise
    P.graze_cap = d.opt_graze_list >= 128 && d.opt_graze_list <= kGrazeList ? (d.opt_graze_list & ~1) : kGrazeList;
    P.query_budget = d.opt_query_budget >= 1 ? d.opt_query_budget : 64;
    P.serial_cap = d.opt_serial_list >= 2 && d.opt_serial_list <= kSerialList ? d.opt_serial_list : kSerialList;
    P.max_steps = static_cast<int>(d.n_tets < (1 << 20) ? d.n_tets : (1 << 20));
    P.round_float = w.round_through_float;
    P.alpha_limit = w.alpha_limit;

    if (w.channels < 0 || w.channels > C5_MAX_CHANNELS || (w.channels && f32)) {
        fail(C5_E_INVALID, "render: channels need precision 64 and 1 .. C5_MAX_CHANNELS channels");
    }
    if (w.channels) {
        P.rec = d.ch_rec.p;
        P.ch_queue = d.ch_queue.p;
    }
    if (w.pass != kImagePass && (w.channels || f32)) fail(C5_E_INVALID, "render_grad: FP64 over the cells' own fields only");
    if (w.pass == kDepthPass || w.pass == kJvpPass) P.ch_queue = d.ch_queue.p;
    const int n_pairs = w.channels ? w.channels : (w.pass == kDepthPass || w.pass == kJvpPass) ? 2 : 1;
    if (!whole_band && w.pass != kGradPass) { // the gradient pass stores no pixel
        count_launch();
        if (kHostSim) {
            background_on_host(P, n_pairs);
        } else {
            const int64_t n = static_cast<int64_t>(w.row_end - w.row_begin) * w.res_x;
            fill_background<<<static_cast<unsigned>((n + 255) / 256), 256, 0, d.stream>>>(P, n_pairs);
            C5_CUDA(cudaGetLastError());
        }
    }
    if (empty_rect) return; // the mesh is not in this band: no rays
    // The order of the view's rays, from the steps the state's last view took at each pixel (c5_debug_set
    // "no_ray_order": from equal costs, the Morton order). The gradient pass walks the rays of the depth pass
    // before it, over the same rectangle, and takes the same order.
    // (Made on a stream of its own beside the view's prologue, the order cost the C4 sweep, three views in flight,
    // 4.5 % against 1.2 % on the view's stream: profiles/r14_ray_order_threshold_one_b200.jsonl.)
    if (w.pass != kGradPass) {
        if (d.opt_no_ray_order) dev_zero(d.ray_cost.p, d.ray_cost.bytes(), d.stream);
        count_launch();
        if (kHostSim) {
            order_on_host(P, n_regions);
        } else {
            prefer_side_carveout(order_rays, d.device);
            order_rays<<<static_cast<unsigned>(n_regions), kOrderThreads, 0, d.stream>>>(P);
            C5_CUDA(cudaGetLastError());
        }
    }
    count_launch();
    const unsigned grid = static_cast<unsigned>(n_regions) * kBlocksPerRegion;
    if (w.pass == kDepthPass) {
        launch_rays<CellsDepth>(d, w, P, grid);
        return;
    }
    if (w.pass == kJvpPass) {
        JvpParams J{};
        static_cast<WalkParams&>(J) = P;
        J.dir = w.dir;
        launch_rays<CellsJvp>(d, w, J, grid);
        return;
    }
    if (w.pass == kGradPass) {
        GradParams G{};
        static_cast<WalkParams&>(G) = P;
        G.grad_in = w.grad_in;
        G.depth = w.depth;
        G.grad_alpha = w.grad_alpha;
        G.grad_q = w.grad_q;
        if (w.grad_per_view) {
            launch_rays<CellsGradView>(d, w, G, grid);
        } else {
            launch_rays<CellsGrad>(d, w, G, grid);
        }
        return;
    }
    switch (w.channels) {
    case 0:
        if (f32) {
            launch_rays<CellsF32>(d, w, P, grid);
        } else {
            launch_rays<CellsF64>(d, w, P, grid);
        }
        break;
    case 1: launch_rays<Channels<1>>(d, w, P, grid); break;
    case 2: launch_rays<Channels<2>>(d, w, P, grid); break;
    case 3: launch_rays<Channels<3>>(d, w, P, grid); break;
    case 4: launch_rays<Channels<4>>(d, w, P, grid); break;
    case 5: launch_rays<Channels<5>>(d, w, P, grid); break;
    case 6: launch_rays<Channels<6>>(d, w, P, grid); break;
    case 7: launch_rays<Channels<7>>(d, w, P, grid); break;
    default: launch_rays<Channels<8>>(d, w, P, grid); break;
    }
}

} // namespace c5
