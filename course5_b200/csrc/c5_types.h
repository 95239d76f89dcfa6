// c5_types.h — device-resident data layout and the small math helpers shared by the kernels.
#pragma once

#include <cfloat>
#include <cmath>
#include <cstdint>
#include <cstring>

#include "c5_rt.h"

namespace c5 {

// ---- data layout in HBM ----------------------------------------------------------------------
//
// Cell record: everything one tet-step reads about the tet it is in, in ONE 64-byte aligned
// record (two 32-byte sectors of one 128-byte line): connectivity, the face-neighbour table, the
// vertex ids across each face, and the two cell scalars. nbr[k] is the tet across the face
// OPPOSITE local vertex k (the face that omits vertex k; the reference's face f omits vertex
// 3 - f, plane.cpp:30-37), or -1 on the domain boundary; apex[k] is the vertex of THAT tet which
// is not on the shared face. Knowing apex[k] when the ray leaves through face k lets the walk
// issue the next cell load and the next vertex load together instead of one after the other.
// s = Q / min(alpha, limit) (the source function) is refreshed when --alpha_limit changes, so the
// I recurrence needs no divide: I <- I - (s - I) expm1(-a dz). Tets are in Morton order of centroids.
struct alignas(64) Cell {
    int32_t v[4];
    int32_t nbr[4];
    int32_t apex[4];
    double alpha; // "AbsorpCoef"
    double s;     // "radEnLooseRate" / min(alpha, alpha_limit)
};
static_assert(sizeof(Cell) == 64, "Cell must be 64 bytes");

// Rotated vertex: one 32-byte sector per vertex (a 24-byte record would straddle sectors half
// the time). Vertices are stored in Morton order.
struct alignas(32) Vtx {
    double x, y, z, w;
};
static_assert(sizeof(Vtx) == 32, "Vtx must be 32 bytes");

// Boundary face, wound so that (b-a)x(c-a) points OUT of the mesh. tet is the cell behind it and
// apex that cell's fourth vertex.
struct alignas(32) BFace {
    int32_t a, b, c, tet;
    int32_t apex, pad[3];
};
static_assert(sizeof(BFace) == 32, "BFace must be 32 bytes");

// Binary LBVH node over boundary faces, 64 bytes: both children's boxes (floats, rounded
// outward) and child links. child >= 0: internal node index; child < 0: leaf ~child (index into
// the Morton-sorted BFace array). An empty box has lo = +inf, hi = -inf.
// Per view only the boxes change (refit); back-facing leaves get empty boxes.
struct alignas(64) BvhNode {
    float xlo[2], xhi[2]; // [child]
    float ylo[2], yhi[2];
    float zlo[2], zhi[2];
    int32_t child[2];
    int32_t pad[2];
};
static_assert(sizeof(BvhNode) == 64, "BvhNode must be 64 bytes");

// A ray the pixel kernel could not finish cheaply (its re-entry list came back full: it grazes a
// bumpy boundary and has many short crossings — or a BVH search ran out of budget). The
// grazing-ray kernel, launched after the pixel kernel on the same stream, continues it from here.
struct alignas(32) DeferredRay {
    double tau, inten; // accumulated so far
    double z_after;    // the ray has left the mesh at this depth
    uint32_t pixel;    // j * res_x + i
    uint32_t steps;    // tets crossed so far
};
static_assert(sizeof(DeferredRay) == 32, "DeferredRay must be 32 bytes");

struct Rot {       // one rotation with the trig evaluated on the host by libm (so it is the same
    int32_t axis;  // cos/sin the reference's host code multiplies by, tetra.cpp:44-62)
    int32_t pad;
    double c, s, x0;
};

// ---- exact (non-contracted) arithmetic --------------------------------------------------------
// The orientation predicate must be exactly antisymmetric, o(u,v) == -o(v,u), so that two tets
// sharing an edge always agree on which side of it a ray passes. With FMA contraction
// fma(ux,vy,-(uy*vx)) and fma(vx,uy,-(vy*ux)) are not negatives of each other; two rounded
// products and one rounded subtraction are.
C5_HD double mul_rn(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
C5_HD double sub_rn(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}
C5_HD double add_rn(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}

// z-component of u x v for 2-D vectors u, v (both relative to the ray's pixel).
C5_HD double orient2(double ux, double uy, double vx, double vy) {
    return sub_rn(mul_rn(ux, vy), mul_rn(uy, vx));
}

C5_HD float f_round_down(double v) {
#ifdef __CUDA_ARCH__
    return __double2float_rd(v);
#else
    float f = static_cast<float>(v);
    if (static_cast<double>(f) > v) f = nextafterf(f, -INFINITY);
    return f;
#endif
}
C5_HD float f_round_up(double v) {
#ifdef __CUDA_ARCH__
    return __double2float_ru(v);
#else
    float f = static_cast<float>(v);
    if (static_cast<double>(f) < v) f = nextafterf(f, INFINITY);
    return f;
#endif
}

// 21 bits per axis interleaved into a 63-bit Morton code.
C5_HD uint64_t spread21(uint64_t v) {
    v &= 0x1FFFFFull;
    v = (v | (v << 32)) & 0x001F00000000FFFFull;
    v = (v | (v << 16)) & 0x001F0000FF0000FFull;
    v = (v | (v << 8)) & 0x100F00F00F00F00Full;
    v = (v | (v << 4)) & 0x10C30C30C30C30C3ull;
    v = (v | (v << 2)) & 0x1249249249249249ull;
    return v;
}
C5_HD uint64_t morton3(double x, double y, double z, const double lo[3], const double inv[3]) {
    double fx = (x - lo[0]) * inv[0], fy = (y - lo[1]) * inv[1], fz = (z - lo[2]) * inv[2];
    fx = fx < 0 ? 0 : (fx > 1 ? 1 : fx);
    fy = fy < 0 ? 0 : (fy > 1 ? 1 : fy);
    fz = fz < 0 ? 0 : (fz > 1 ? 1 : fz);
    const uint64_t ix = static_cast<uint64_t>(fx * 2097151.0);
    const uint64_t iy = static_cast<uint64_t>(fy * 2097151.0);
    const uint64_t iz = static_cast<uint64_t>(fz * 2097151.0);
    return (spread21(ix) << 2) | (spread21(iy) << 1) | spread21(iz);
}

} // namespace c5
