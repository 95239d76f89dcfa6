/* CPU restatement of course5's per-pixel ray pass. TEST INFRASTRUCTURE ONLY.
 *
 * Nothing in the product (course5_b200/, the `course` CLI, libc5gpu.so) may link or
 * call this. Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference legs use it, as the checker.
 *
 * Parity pin: the reference has no tests or golden vectors (SURVEY.md §4), so this
 * restatement is pinned against the reference itself — oracle/_ref/libc5ref.so, the
 * unmodified reference sources — bit for bit (tests/test_oracle.py) and against
 * fixtures generated from it (tests/golden/, made by tests/golden/make_golden.py).
 */
#ifndef C5_ORACLE_H
#define C5_ORACLE_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct c5o_view {
    int res_x, res_y;
    double window[4];   /* x_max, x_min, y_max, y_min — main.cpp:83 */
    double alpha_limit; /* config.hpp:25, read at line.cpp:204 */
    int threads;
} c5o_view;

/* In-place view rotations of n points (xyz triples): Rx(a0), Ry(Y*pi) about x = x0,
 * Rx(-a0 + X*pi), a0 = -I*pi + pi/2 — main.cpp:96,105-107 with tetra.cpp:44-62. */
void c5o_rotate_points(double* pts, int64_t n_points, double X, double Y, double I, double x0);

/* One rotation, like object3d_base::rotate_around_{x,y}_axis. axis 0 = x, 1 = y. */
void c5o_rotate_axis(double* pts, int64_t n_points, int axis, double angle, double x0);

/* Accumulated pixel coordinates — plane.cpp:298-314. */
void c5o_pixel_coords(const c5o_view* v, double* xs, double* ys);

/* The ray pass over tets ALREADY in the view frame.
 *   tet_pts   [n_tets][4][3]   transparent tets (the grid)
 *   solid_pts [n_solid][4][3]  solid tets (may be NULL / 0)
 *   tau, inten [res_y][res_x]  pre-float-cast doubles, x fastest; NaN under solids, 0 on a miss
 *   steps      [res_y][res_x]  records per pixel (0 under solids); may be NULL
 *   solid      [res_y][res_x]  1 under a solid; may be NULL
 *   anomalies  pixels of a tet that were covered by an odd number of its faces (the reference's
 *              behaviour there is undefined — SURVEY.md §3.3); may be NULL
 * Returns 0, -1 on bad arguments, -2 on allocation failure. */
int c5o_render(const double* tet_pts, const double* alpha, const double* q, int64_t n_tets,
               const double* solid_pts, int64_t n_solid, const c5o_view* v, double* tau, double* inten,
               uint32_t* steps, uint8_t* solid, uint64_t* total_steps, uint64_t* anomalies);

/* The segments c5o_render integrates, per pixel: the same inputs, and seg_start[n_pix + 1], the prefix
 * sum of the steps a c5o_render call returned (pixel j * res_x + i crosses seg_start[pix + 1] -
 * seg_start[pix] tets). Pixel pix's segments go to seg_tet / seg_dz [seg_start[pix] ..] in the order
 * the I recurrence takes them (line.cpp:206-225: the lowest segment first, where the ray enters); the
 * sum of seg_dz * alpha[seg_tet] in reverse order is its tau. Test infrastructure for an integration
 * that does not come from the code under test.
 * Returns 0, -1 on bad arguments, -2 on allocation failure, -3 when a pixel's record count is not
 * its span of seg_start. */
int c5o_render_segments(const double* tet_pts, const double* alpha, const double* q, int64_t n_tets,
                        const double* solid_pts, int64_t n_solid, const c5o_view* v, const int64_t* seg_start,
                        int32_t* seg_tet, double* seg_dz);

#ifdef __cplusplus
}
#endif
#endif
