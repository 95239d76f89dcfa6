// c5_topology.cu — one-off per mesh: flatten points + connectivity into the device-resident
// arrays the per-view kernels read (north-star item (a); SURVEY.md §2.3 K2).
//
// The reference keeps a private copy of the 4 points in every tet and no connectivity
// (object3d_base.cpp:37-51, tetra.hpp:42-45). Here:
//   1. vertices are sorted along a 63-bit Morton curve (file frame) -> px/py/pz SoA;
//   2. tets are sorted along the Morton curve of their centroids -> Fields records and the tets'
//      vertex ids (a buffer of the upload only);
//   3. every tet face gets the key (sorted vertex triple); a radix sort brings the two copies of
//      an interior face together -> Conn::nbr and Conn::apex with the face's slot map; unmatched
//      faces are the domain boundary;
//   4. boundary faces are wound outward, Morton-sorted, and a Karras LBVH hierarchy is built over
//      them (only the boxes are refitted per view, c5_exact.cu);
//   5. the hierarchy is relabelled breadth-first on the host so the top levels are a contiguous
//      prefix the walk kernel stages in shared memory.
#include <algorithm>
#include <queue>
#include <vector>

#include "c5_internal.h"

namespace c5 {

static_assert(C5_MAX_POINTS == (1 << kApexIdBits), "a vertex id must fit the id bits of Conn::apex");

namespace {

C5_HD int clz64(uint64_t v) {
#ifdef __CUDA_ARCH__
    return __clzll(static_cast<long long>(v));
#else
    return v ? __builtin_clzll(v) : 64;
#endif
}
C5_HD int clz32(uint32_t v) {
#ifdef __CUDA_ARCH__
    return __clz(static_cast<int>(v));
#else
    return v ? __builtin_clz(v) : 32;
#endif
}

struct Box3 {
    double lo[3], inv[3];
};

// -- 1. vertex Morton keys --------------------------------------------------------------------
struct VertexKeyOp {
    const double* xyz;
    Box3 box;
    uint64_t* keys;
    uint32_t* vals;
    C5_HD void operator()(int64_t i) const {
        keys[i] = morton3(xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2], box.lo, box.inv);
        vals[i] = static_cast<uint32_t>(i);
    }
};

struct VertexScatterOp {
    const double* xyz;
    const uint32_t* perm; // new -> old
    uint32_t* inv;        // old -> new
    double *px, *py, *pz;
    C5_HD void operator()(int64_t i) const {
        const uint32_t old = perm[i];
        inv[old] = static_cast<uint32_t>(i);
        px[i] = xyz[3 * old];
        py[i] = xyz[3 * old + 1];
        pz[i] = xyz[3 * old + 2];
    }
};

// -- 2. tet Morton keys, validation ------------------------------------------------------------
struct TetKeyOp {
    const double* xyz;
    const int32_t* tets;
    int64_t n_pts;
    Box3 box;
    uint64_t* keys;
    uint32_t* vals;
    int* err;
    C5_HD void operator()(int64_t t) const {
        double c[3] = {0, 0, 0};
        bool ok = true;
        for (int k = 0; k < 4; k++) {
            const int32_t v = tets[4 * t + k];
            if (v < 0 || v >= n_pts) {
                ok = false;
                continue;
            }
            for (int a = 0; a < 3; a++) c[a] += 0.25 * xyz[3 * static_cast<int64_t>(v) + a];
            for (int m = 0; m < k; m++) {
                if (tets[4 * t + m] == v) ok = false;
            }
        }
        if (!ok) *err = 2;
        keys[t] = morton3(c[0], c[1], c[2], box.lo, box.inv);
        vals[t] = static_cast<uint32_t>(t);
    }
};

struct CellFillOp {
    const int32_t* tets;
    const double* alpha;
    const double* q;
    const uint32_t* tperm; // new -> old tet
    const uint32_t* vinv;  // old -> new vertex
    int32_t* tv;           // [n_tets][4] vertex ids
    Fields* fields;
    double* q0;
    C5_HD void operator()(int64_t t) const {
        const uint32_t old = tperm[t];
        for (int k = 0; k < 4; k++) tv[4 * t + k] = static_cast<int32_t>(vinv[tets[4 * static_cast<int64_t>(old) + k]]);
        Fields c;
        c.alpha = alpha[old];
        c.s = 0.0; // set by prepare_cells for the view's alpha_limit
        q0[t] = q[old];
        fields[t] = c;
    }
};

// -- 3. face keys and matching -------------------------------------------------------------------
// Face f = 4 t + k is the face of tet t opposite its local vertex k.
struct FaceKeyOp {
    const int32_t* tv;
    uint64_t* key_lo_mid;
    uint32_t* key_hi;
    uint32_t* hi_sort; // copy that gets sorted
    uint32_t* idx;
    C5_HD void operator()(int64_t f) const {
        const int32_t* v = tv + 4 * (f >> 2);
        const int k = static_cast<int>(f & 3);
        uint32_t a = static_cast<uint32_t>(v[(k + 1) & 3]);
        uint32_t b = static_cast<uint32_t>(v[(k + 2) & 3]);
        uint32_t d = static_cast<uint32_t>(v[(k + 3) & 3]);
        uint32_t t;
        if (a > b) { t = a; a = b; b = t; }
        if (b > d) { t = b; b = d; d = t; }
        if (a > b) { t = a; a = b; b = t; }
        key_lo_mid[f] = (static_cast<uint64_t>(a) << 32) | b;
        key_hi[f] = d;
        hi_sort[f] = d;
        idx[f] = static_cast<uint32_t>(f);
    }
};

struct GatherKeyOp {
    const uint64_t* key_lo_mid;
    const uint32_t* idx;
    uint64_t* out;
    C5_HD void operator()(int64_t i) const { out[i] = key_lo_mid[idx[i]]; }
};

struct FaceMatchOp {
    const uint64_t* key_lo_mid; // by face
    const uint32_t* key_hi;     // by face
    const uint32_t* idx;        // faces sorted by (lo, mid, hi)
    int64_t n_faces;
    const int32_t* tv;    // [n_tets][4] vertex ids
    Conn* conn;
    uint8_t* is_boundary; // by face
    int* err;
    C5_HD bool same(uint32_t f, uint32_t g) const {
        return key_lo_mid[f] == key_lo_mid[g] && key_hi[f] == key_hi[g];
    }
    // Conn::apex of face f, whose twin is face g: g's apex id and the slots in g's tet of f's
    // vertices at slots (k + 1) & 3, (k + 2) & 3, (k + 3) & 3 (the twins share these three vertices)
    C5_HD uint32_t apex_word(uint32_t f, uint32_t g) const {
        const int32_t* vf = tv + 4 * static_cast<int64_t>(f >> 2);
        const int32_t* vg = tv + 4 * static_cast<int64_t>(g >> 2);
        uint32_t map = 0;
        for (uint32_t j = 1; j <= 3; j++) {
            const int32_t x = vf[(f + j) & 3];
            uint32_t slot = 0;
            for (uint32_t m = 1; m < 4; m++) {
                if (vg[m] == x) slot = m;
            }
            map |= slot << (2 * (j - 1));
        }
        return static_cast<uint32_t>(vg[g & 3]) | (map << kApexIdBits);
    }
    C5_HD void operator()(int64_t i) const {
        const uint32_t f = idx[i];
        const bool eq_prev = i > 0 && same(f, idx[i - 1]);
        const bool eq_next = i + 1 < n_faces && same(f, idx[i + 1]);
        if (eq_prev && eq_next) {
            *err = 1; // a face shared by three or more tets
            return;
        }
        if (eq_next) {
            const uint32_t g = idx[i + 1];
            conn[f >> 2].nbr[f & 3] = static_cast<int32_t>(g >> 2);
            conn[g >> 2].nbr[g & 3] = static_cast<int32_t>(f >> 2);
            conn[f >> 2].apex[f & 3] = apex_word(f, g);
            conn[g >> 2].apex[g & 3] = apex_word(g, f);
            is_boundary[f] = 0;
            is_boundary[g] = 0;
        } else if (!eq_prev) {
            conn[f >> 2].nbr[f & 3] = -1;
            conn[f >> 2].apex[f & 3] = 0;
            is_boundary[f] = 1;
        }
    }
};

// -- 4. boundary faces and the LBVH hierarchy --------------------------------------------------
struct BFaceOp {
    const int32_t* tv;
    const double *px, *py, *pz;
    const uint32_t* bface_ids; // face index f of each boundary face
    Box3 box;
    BFace* out;
    uint64_t* keys;
    uint32_t* vals;
    C5_HD void operator()(int64_t i) const {
        const uint32_t f = bface_ids[i];
        const int32_t* v = tv + 4 * static_cast<int64_t>(f >> 2);
        const int k = static_cast<int>(f & 3);
        int32_t a = v[(k + 1) & 3], b = v[(k + 2) & 3], cc = v[(k + 3) & 3];
        int32_t sb = (k + 2) & 3, sc = (k + 3) & 3; // slots of b and cc
        const int32_t d = v[k];
        const double ax = px[a], ay = py[a], az = pz[a];
        const double ux = px[b] - ax, uy = py[b] - ay, uz = pz[b] - az;
        const double vx = px[cc] - ax, vy = py[cc] - ay, vz = pz[cc] - az;
        const double wx = px[d] - ax, wy = py[d] - ay, wz = pz[d] - az;
        const double det = (uy * vz - uz * vy) * wx + (uz * vx - ux * vz) * wy + (ux * vy - uy * vx) * wz;
        if (det > 0) { // normal points at the opposite vertex, i.e. inward: flip
            const int32_t t = b;
            b = cc;
            cc = t;
            const int32_t st = sb;
            sb = sc;
            sc = st;
        }
        BFace bf;
        bf.a = a;
        bf.b = b;
        bf.c = cc;
        bf.tet = static_cast<int32_t>(f >> 2);
        bf.apex = d;
        bf.slots = ((k + 1) & 3) | (sc << 2) | (sb << 4); // a, c, b
        bf.pad[0] = bf.pad[1] = 0;
        out[i] = bf;
        keys[i] = morton3((px[a] + px[b] + px[cc]) / 3.0, (py[a] + py[b] + py[cc]) / 3.0,
                          (pz[a] + pz[b] + pz[cc]) / 3.0, box.lo, box.inv);
        vals[i] = static_cast<uint32_t>(i);
    }
};

struct GatherBFaceOp {
    const BFace* in;
    const uint32_t* perm;
    BFace* out;
    C5_HD void operator()(int64_t i) const { out[i] = in[perm[i]]; }
};

// Karras 2012, "Maximizing parallelism in the construction of BVHs, octrees and k-d trees":
// internal node i covers a contiguous range of the sorted keys; ties are broken by index.
struct KarrasOp {
    const uint64_t* codes;
    int n; // leaves
    int32_t* left;  // per internal node: >= 0 internal, < 0 leaf ~index
    int32_t* right;
    C5_HD int delta(int i, int j) const {
        if (j < 0 || j >= n) return -1;
        const uint64_t a = codes[i], b = codes[j];
        if (a == b) return 64 + clz32(static_cast<uint32_t>(i) ^ static_cast<uint32_t>(j));
        return clz64(a ^ b);
    }
    C5_HD void operator()(int64_t ii) const {
        const int i = static_cast<int>(ii);
        const int d = (delta(i, i + 1) - delta(i, i - 1)) >= 0 ? 1 : -1;
        const int dmin = delta(i, i - d);
        int lmax = 2;
        while (delta(i, i + lmax * d) > dmin) lmax *= 2;
        int l = 0;
        for (int t = lmax / 2; t >= 1; t /= 2) {
            if (delta(i, i + (l + t) * d) > dmin) l += t;
        }
        const int j = i + l * d;
        const int dnode = delta(i, j);
        int s = 0;
        int t = l;
        do {
            t = (t + 1) / 2;
            if (delta(i, i + (s + t) * d) > dnode) s += t;
        } while (t > 1);
        const int gamma = i + s * d + (d < 0 ? d : 0);
        const int lo = i < j ? i : j, hi = i < j ? j : i;
        left[i] = (lo == gamma) ? ~gamma : gamma;
        right[i] = (hi == gamma + 1) ? ~(gamma + 1) : gamma + 1;
    }
};

Box3 bounding_box(const double* pts, int64_t n) {
    double lo[3] = {pts[0], pts[1], pts[2]}, hi[3] = {pts[0], pts[1], pts[2]};
    for (int64_t i = 1; i < n; i++) {
        for (int a = 0; a < 3; a++) {
            const double v = pts[3 * i + a];
            if (v < lo[a]) lo[a] = v;
            if (v > hi[a]) hi[a] = v;
        }
    }
    Box3 b;
    for (int a = 0; a < 3; a++) {
        b.lo[a] = lo[a];
        b.inv[a] = hi[a] > lo[a] ? 1.0 / (hi[a] - lo[a]) : 0.0;
    }
    return b;
}

int bits_for(uint64_t n) {
    int b = 1;
    while (b < 64 && (uint64_t{1} << b) < n) b++;
    return b;
}

// Channel records from channel-major file-order fields: record t holds {alpha_c, 0} (s_c is set by
// prepare_channels) of old tet tperm[t] for every channel c, and zeros in the padding.
struct ChannelGatherOp {
    const double* alpha;   // [n][n_tets], file order
    const double* q;
    const uint32_t* tperm; // new -> old tet
    int64_t n_tets;
    int n;
    double* rec;           // [n_tets][channel_stride(n)]
    double* q0;            // [n][n_tets], Morton order
    C5_HD void operator()(int64_t t) const {
        const int64_t old = tperm[t];
        double* r = rec + t * channel_stride(n);
        for (int k = 2 * n; k < channel_stride(n); k++) r[k] = 0.0;
        for (int c = 0; c < n; c++) {
            r[2 * c] = alpha[c * n_tets + old];
            r[2 * c + 1] = 0.0;
            q0[c * n_tets + t] = q[c * n_tets + old];
        }
    }
};

// The alpha of channel record t (stride channel_stride(1)) into tet t: c5_update_fields gathers the
// tets' new fields as one channel, then moves alpha into Fields.
struct CellAlphaOp {
    const double* rec;
    Fields* fields;
    C5_HD void operator()(int64_t t) const { fields[t].alpha = rec[t * channel_stride(1)]; }
};

// n channel-major arrays of file-order alpha and q: record t of rec gets {alpha_c, 0} of old tet
// tperm[t] for every channel, q0 gets Q in Morton order. Shared by c5_upload_channels and c5_update_fields.
void gather_file_order(DeviceState& d, const double* alpha, const double* q, int n, double* rec, double* q0) {
    cudaStream_t s = d.stream;
    const size_t n_t = static_cast<size_t>(d.n_tets), n_all = n_t * static_cast<size_t>(n);
    DevBuf<double> alpha_in, q_in;
    DevBuf<uint32_t> tperm;
    alpha_in.alloc(n_all);
    q_in.alloc(n_all);
    tperm.alloc(n_t);
    h2d(alpha_in.p, alpha, alpha_in.bytes(), s);
    h2d(q_in.p, q, q_in.bytes(), s);
    h2d(tperm.p, d.tperm.data(), tperm.bytes(), s);
    for_each(s, d.n_tets, ChannelGatherOp{alpha_in.p, q_in.p, tperm.p, d.n_tets, n, rec, q0});
    stream_sync(s); // the staging buffers are freed on return
}

// c5_update_fields_device: file-order device fields straight into Fields (no staging, no allocation).
struct FieldGatherOp {
    const double* alpha;   // [n_tets], file order
    const double* q;
    const uint32_t* tperm; // new -> old tet
    Fields* fields;
    double* q0;            // Morton order
    C5_HD void operator()(int64_t t) const {
        const uint32_t old = tperm[t];
        fields[t].alpha = alpha[old];
        q0[t] = q[old];
    }
};

// c5_render_grad_device: the gradient pass's Morton-order sums into the caller's file-order arrays.
struct GradScatterOp {
    const uint32_t* tperm; // new -> old tet
    const double* in_alpha;
    const double* in_q;
    double* out_alpha;     // either may be null
    double* out_q;
    C5_HD void operator()(int64_t t) const {
        const uint32_t old = tperm[t];
        if (out_alpha) out_alpha[old] = in_alpha[t];
        if (out_q) out_q[old] = in_q[t];
    }
};

} // namespace

void build_mesh(DeviceState& d, const double* pts, int64_t n_pts, const int32_t* tets, int64_t n_tets,
                const double* alpha, const double* q) {
    if (n_pts < 4 || n_tets < 1) fail(C5_E_INVALID, "upload_mesh: need at least 4 points and 1 tet");
    if (n_pts > C5_MAX_POINTS) fail(C5_E_INVALID, "upload_mesh: more than C5_MAX_POINTS (2^26) points");
    if (n_tets >= (int64_t{1} << 29)) fail(C5_E_INVALID, "upload_mesh: more than 2^29 tets");
    cudaStream_t s = d.stream;
    const Box3 box = bounding_box(pts, n_pts);
    for (int a = 0; a < 3; a++) d.mesh_lo[a] = d.mesh_hi[a] = pts[a];
    for (int64_t i = 1; i < n_pts; i++) {
        for (int a = 0; a < 3; a++) {
            const double v = pts[3 * i + a];
            if (v < d.mesh_lo[a]) d.mesh_lo[a] = v;
            if (v > d.mesh_hi[a]) d.mesh_hi[a] = v;
        }
    }

    DevBuf<int> err;
    err.alloc(1);
    dev_zero(err.p, sizeof(int), s);
    auto check = [&](const char* what) {
        int e = 0;
        d2h(&e, err.p, sizeof(int), s);
        stream_sync(s);
        if (e == 1) fail(C5_E_TOPOLOGY, std::string(what) + ": a face is shared by more than two tets");
        if (e == 2) fail(C5_E_INVALID, std::string(what) + ": tet with an out-of-range or repeated vertex id");
    };

    // 1. vertices
    DevBuf<double> xyz;
    xyz.alloc(static_cast<size_t>(3 * n_pts));
    h2d(xyz.p, pts, xyz.bytes(), s);
    DevBuf<uint32_t> vinv;
    vinv.alloc(static_cast<size_t>(n_pts));
    d.px.alloc(static_cast<size_t>(n_pts));
    d.py.alloc(static_cast<size_t>(n_pts));
    d.pz.alloc(static_cast<size_t>(n_pts));
    {
        DevBuf<uint64_t> keys;
        DevBuf<uint32_t> perm;
        keys.alloc(static_cast<size_t>(n_pts));
        perm.alloc(static_cast<size_t>(n_pts));
        for_each(s, n_pts, VertexKeyOp{xyz.p, box, keys.p, perm.p});
        sort_pairs_u64(keys.p, perm.p, static_cast<size_t>(n_pts), 63, s);
        for_each(s, n_pts, VertexScatterOp{xyz.p, perm.p, vinv.p, d.px.p, d.py.p, d.pz.p});
    }

    // 2. tets in Morton order: fields, and the vertex ids faces 3. and 4. are built from
    d.conn.alloc(static_cast<size_t>(n_tets));
    d.fields.alloc(static_cast<size_t>(n_tets));
    DevBuf<int32_t> tv;
    tv.alloc(static_cast<size_t>(4 * n_tets));
    {
        DevBuf<int32_t> tets_in;
        DevBuf<double> alpha_in, q_in;
        DevBuf<uint64_t> keys;
        DevBuf<uint32_t> tperm;
        tets_in.alloc(static_cast<size_t>(4 * n_tets));
        alpha_in.alloc(static_cast<size_t>(n_tets));
        q_in.alloc(static_cast<size_t>(n_tets));
        keys.alloc(static_cast<size_t>(n_tets));
        tperm.alloc(static_cast<size_t>(n_tets));
        h2d(tets_in.p, tets, tets_in.bytes(), s);
        h2d(alpha_in.p, alpha, alpha_in.bytes(), s);
        h2d(q_in.p, q, q_in.bytes(), s);
        for_each(s, n_tets, TetKeyOp{xyz.p, tets_in.p, n_pts, box, keys.p, tperm.p, err.p});
        check("upload_mesh");
        sort_pairs_u64(keys.p, tperm.p, static_cast<size_t>(n_tets), 63, s);
        d.q0.alloc(static_cast<size_t>(n_tets));
        for_each(s, n_tets, CellFillOp{tets_in.p, alpha_in.p, q_in.p, tperm.p, vinv.p, tv.p, d.fields.p, d.q0.p});
        d.tperm.resize(static_cast<size_t>(n_tets));
        d2h(d.tperm.data(), tperm.p, tperm.bytes(), s);
        stream_sync(s);
    }
    xyz.release();
    vinv.release();

    // 3. face matching
    const int64_t n_faces = 4 * n_tets;
    DevBuf<uint32_t> bface_ids;
    size_t n_b = 0;
    {
        DevBuf<uint64_t> key_lm, key_sorted;
        DevBuf<uint32_t> key_hi, hi_sort, idx;
        DevBuf<uint8_t> is_boundary;
        key_lm.alloc(static_cast<size_t>(n_faces));
        key_hi.alloc(static_cast<size_t>(n_faces));
        hi_sort.alloc(static_cast<size_t>(n_faces));
        idx.alloc(static_cast<size_t>(n_faces));
        for_each(s, n_faces, FaceKeyOp{tv.p, key_lm.p, key_hi.p, hi_sort.p, idx.p});
        const int vbits = bits_for(static_cast<uint64_t>(n_pts));
        sort_pairs_u32(hi_sort.p, idx.p, static_cast<size_t>(n_faces), vbits, s); // by hi
        hi_sort.release();
        key_sorted.alloc(static_cast<size_t>(n_faces));
        for_each(s, n_faces, GatherKeyOp{key_lm.p, idx.p, key_sorted.p});
        sort_pairs_u64(key_sorted.p, idx.p, static_cast<size_t>(n_faces), 32 + vbits, s); // stable: by (lo, mid, hi)
        key_sorted.release();
        is_boundary.alloc(static_cast<size_t>(n_faces));
        dev_zero(is_boundary.p, is_boundary.bytes(), s);
        for_each(s, n_faces, FaceMatchOp{key_lm.p, key_hi.p, idx.p, n_faces, tv.p, d.conn.p, is_boundary.p, err.p});
        check("upload_mesh");
        bface_ids.alloc(static_cast<size_t>(n_faces));
        n_b = select_flagged(is_boundary.p, bface_ids.p, static_cast<size_t>(n_faces), s);
    }
    if (n_b < 4) fail(C5_E_TOPOLOGY, "upload_mesh: fewer than 4 boundary faces");

    // 4. boundary faces, Morton-sorted, + Karras hierarchy
    d.bfaces.alloc(n_b);
    DevBuf<int32_t> left, right;
    left.alloc(n_b - 1);
    right.alloc(n_b - 1);
    {
        DevBuf<BFace> unsorted;
        DevBuf<uint64_t> keys;
        DevBuf<uint32_t> perm;
        unsorted.alloc(n_b);
        keys.alloc(n_b);
        perm.alloc(n_b);
        for_each(s, static_cast<int64_t>(n_b),
                 BFaceOp{tv.p, d.px.p, d.py.p, d.pz.p, bface_ids.p, box, unsorted.p, keys.p, perm.p});
        sort_pairs_u64(keys.p, perm.p, n_b, 63, s);
        for_each(s, static_cast<int64_t>(n_b), GatherBFaceOp{unsorted.p, perm.p, d.bfaces.p});
        for_each(s, static_cast<int64_t>(n_b - 1), KarrasOp{keys.p, static_cast<int>(n_b), left.p, right.p});
        stream_sync(s);
    }
    bface_ids.release();
    tv.release();

    // 5. breadth-first relabel on the host (n_b is small: the surface of the mesh)
    std::vector<int32_t> h_left(n_b - 1), h_right(n_b - 1);
    d2h(h_left.data(), left.p, left.bytes(), s);
    d2h(h_right.data(), right.p, right.bytes(), s);
    stream_sync(s);
    left.release();
    right.release();

    const size_t n_int = n_b - 1;
    std::vector<int32_t> order; // new -> old
    std::vector<int32_t> new_id(n_int, -1);
    order.reserve(n_int);
    order.push_back(0);
    new_id[0] = 0;
    for (size_t head = 0; head < order.size(); head++) {
        const int32_t old = order[head];
        const int32_t ch[2] = {h_left[static_cast<size_t>(old)], h_right[static_cast<size_t>(old)]};
        for (int32_t c : ch) {
            if (c >= 0) {
                if (static_cast<size_t>(c) >= n_int || new_id[static_cast<size_t>(c)] != -1) {
                    fail(C5_E_TOPOLOGY, "upload_mesh: LBVH hierarchy is not a tree (internal error)");
                }
                new_id[static_cast<size_t>(c)] = static_cast<int32_t>(order.size());
                order.push_back(c);
            }
        }
    }
    if (order.size() != n_int) fail(C5_E_TOPOLOGY, "upload_mesh: LBVH hierarchy is disconnected (internal error)");

    std::vector<BvhNode> h_nodes(n_int);
    std::vector<int32_t> h_node_parent(n_int, -1), h_leaf_parent(n_b, -1);
    for (size_t nn = 0; nn < n_int; nn++) {
        const int32_t old = order[nn];
        BvhNode& node = h_nodes[nn];
        const int32_t ch[2] = {h_left[static_cast<size_t>(old)], h_right[static_cast<size_t>(old)]};
        for (int w = 0; w < 2; w++) {
            node.xlo[w] = node.ylo[w] = node.zlo[w] = INFINITY;
            node.xhi[w] = node.yhi[w] = node.zhi[w] = -INFINITY;
            const int32_t link = (static_cast<int32_t>(nn) << 1) | w;
            if (ch[w] >= 0) {
                node.child[w] = new_id[static_cast<size_t>(ch[w])];
                h_node_parent[static_cast<size_t>(node.child[w])] = link;
            } else {
                node.child[w] = ch[w];
                const size_t leaf = static_cast<size_t>(~ch[w]);
                if (leaf >= n_b || h_leaf_parent[leaf] != -1) {
                    fail(C5_E_TOPOLOGY, "upload_mesh: LBVH leaf linked twice (internal error)");
                }
                h_leaf_parent[leaf] = link;
            }
        }
        node.pad[0] = node.pad[1] = 0;
    }
    d.nodes.alloc(n_int);
    d.node_parent.alloc(n_int);
    d.leaf_parent.alloc(n_b);
    d.refit_flags.alloc(n_int);
    h2d(d.nodes.p, h_nodes.data(), d.nodes.bytes(), s);
    h2d(d.node_parent.p, h_node_parent.data(), d.node_parent.bytes(), s);
    h2d(d.leaf_parent.p, h_leaf_parent.data(), d.leaf_parent.bytes(), s);
    stream_sync(s);

    d.vrot.alloc(static_cast<size_t>(n_pts));
    d.n_pts = n_pts;
    d.n_tets = n_tets;
    d.n_bfaces = static_cast<int64_t>(n_b);
    d.cells_limit_valid = false;
}

void upload_channels(DeviceState& d, const double* alpha, const double* q, int n) {
    d.ch_rec.release();
    d.ch_q0.release();
    d.n_channels = 0;
    d.ch_limit_valid = false;
    if (n == 0) return;
    const size_t n_t = static_cast<size_t>(d.n_tets);
    d.ch_rec.alloc(n_t * static_cast<size_t>(channel_stride(n)));
    d.ch_q0.alloc(n_t * static_cast<size_t>(n));
    gather_file_order(d, alpha, q, n, d.ch_rec.p, d.ch_q0.p);
    d.n_channels = n;
}

void update_fields(DeviceState& d, const double* alpha, const double* q) {
    DevBuf<double> rec;
    rec.alloc(static_cast<size_t>(d.n_tets) * channel_stride(1));
    gather_file_order(d, alpha, q, 1, rec.p, d.q0.p);
    for_each(d.stream, d.n_tets, CellAlphaOp{rec.p, d.fields.p});
    stream_sync(d.stream);
    d.cells_limit_valid = false; // fields[].s is derived again from the new q0 at the next render
}

void upload_tperm(DeviceState& d) {
    d.tperm_dev.alloc(d.tperm.size());
    h2d(d.tperm_dev.p, d.tperm.data(), d.tperm_dev.bytes(), d.stream);
    stream_sync(d.stream); // the host vector is pageable and may change at the next upload_mesh
}

void gather_fields(DeviceState& d, const uint32_t* tperm, const double* alpha, const double* q, cudaStream_t s) {
    for_each(s, d.n_tets, FieldGatherOp{alpha, q, tperm, d.fields.p, d.q0.p});
    d.cells_limit_valid = false; // fields[].s is derived again from the new q0 at the next render
}

void scatter_grads(int64_t n_tets, const uint32_t* tperm, const double* in_alpha, const double* in_q, double* out_alpha,
                   double* out_q, cudaStream_t s) {
    for_each(s, n_tets, GradScatterOp{tperm, in_alpha, in_q, out_alpha, out_q});
}

} // namespace c5
