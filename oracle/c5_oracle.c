/* CPU restatement of course5's per-pixel ray pass — see c5_oracle.h.
 * TEST INFRASTRUCTURE ONLY; never linked into the product.
 *
 * The reference is object-order: every face of every tet is scan-converted onto the pixel
 * grid, each pixel collects (tet, two face bits) records, and per pixel the two face-plane z's
 * are evaluated, the segments sorted by z and integrated. This file restates that algorithm
 * with the same floating-point expressions in the same order (compile with
 * -ffp-contract=off, like the reference's plain x86-64 -O3 build), but with its own data
 * structures: instead of a heap object per pixel with per-thread pairing slots and a mutex
 * (line.hpp:81-90), face hits of one tet are paired locally and records are bucketed into a
 * CSR array by pixel.
 *
 * Reference lines restated (all under /root/reference/project/src):
 *   rotations               tetra.cpp:44-62, main.cpp:96,105-107
 *   pixel coordinates       plane.cpp:298-314
 *   pixel index of x / y    plane.cpp:194-212
 *   edge functions          plane.cpp:46-55
 *   face scan conversion    plane.cpp:57-142   (faces of a tet: plane.cpp:30-37)
 *   record pairing          line.cpp:29-67
 *   face-plane z            line.cpp:150-174, face order line.cpp:103-122
 *   per-record dz, sort     line.cpp:124-147
 *   tau                     line.cpp:176-193
 *   I recurrence            line.cpp:195-227
 *   solid pixels            plane.cpp:23-27,130-131; line.cpp:178-180,197-199,246-249
 */
#include "c5_oracle.h"

#include <float.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#ifdef _OPENMP
#include <omp.h>
#endif

/* ------------------------------------------------------------------ rotations */

void c5o_rotate_axis(double* pts, int64_t n_points, int axis, double angle, double x0) {
    int64_t i;
    if (axis == 0) {
        /* tetra.cpp:44-48 */
        for (i = 0; i < n_points; i++) {
            double* p = pts + 3 * i;
            const double y = p[1];
            p[1] = p[1] * cos(angle) - p[2] * sin(angle);
            p[2] = y * sin(angle) + p[2] * cos(angle);
        }
    } else {
        /* tetra.cpp:51-62: about the axis parallel to y through (x0, 0, 0) */
        for (i = 0; i < n_points; i++) {
            double* p = pts + 3 * i;
            double x;
            p[0] -= x0;
            x = p[0];
            p[0] = p[0] * cos(angle) - p[2] * sin(angle);
            p[2] = x * sin(angle) + p[2] * cos(angle);
            p[0] += x0;
        }
    }
}

void c5o_rotate_points(double* pts, int64_t n_points, double X, double Y, double I, double x0) {
    const double PI = 3.14159265358979323846; /* config.hpp:45 */
    const double a0 = -I * PI + PI / 2.;      /* main.cpp:96 */
    c5o_rotate_axis(pts, n_points, 0, a0, 0.0);
    c5o_rotate_axis(pts, n_points, 1, Y * PI, x0);
    c5o_rotate_axis(pts, n_points, 0, -a0 + X * PI, 0.0);
}

/* ------------------------------------------------------------------ pixel grid */

typedef struct grid {
    int res_x, res_y;
    double x_min, y_min, step_x, step_y;
    double* xs;
    double* ys;
} grid;

void c5o_pixel_coords(const c5o_view* v, double* xs, double* ys) {
    const double step_x = (v->window[0] - v->window[1]) / (v->res_x - 1.);
    const double step_y = (v->window[2] - v->window[3]) / (v->res_y - 1.);
    double c = v->window[1];
    int i;
    for (i = 0; i < v->res_x; i++) {
        xs[i] = c;
        c = c + step_x;
    }
    c = v->window[3];
    for (i = 0; i < v->res_y; i++) {
        ys[i] = c;
        c = c + step_y;
    }
}

static double pix_of_x(const grid* g, double x) {
    const double r = (x - g->x_min) / g->step_x;
    const double hi = (double)g->res_x - 1;
    if (r < 0) return 0;
    if (r > hi) return hi;
    return r;
}

static double pix_of_y(const grid* g, double y) {
    const double r = (y - g->y_min) / g->step_y;
    const double hi = (double)g->res_y - 1;
    if (r < 0) return 0;
    if (r > hi) return hi;
    return r;
}

/* implicit line through p1,p2 evaluated at pos (plane.cpp:46-48) */
static double side_of(const double* p1, const double* p2, const double* pos) {
    return (p2[1] - p1[1]) * pos[0] + (p1[0] - p2[0]) * pos[1] + (p2[0] * p1[1] - p1[0] * p2[1]);
}

/* x of the edge p1-p2 at height y (plane.cpp:50-55) */
static double edge_x_at(const double* p1, const double* p2, double y) {
    if (fabs(p1[1] - p2[1]) < DBL_EPSILON) return p1[0];
    return (p1[0] - p2[0]) * (y - p1[1]) / (p1[1] - p2[1]) + p1[0];
}

/* Scan-converts one triangle; calls emit(ctx, i, j) for every covered pixel. */
typedef void (*emit_fn)(void* ctx, size_t i, size_t j);

static void scan_face(const grid* g, const double* a, const double* b, const double* c, emit_fn emit,
                      void* ctx) {
    const double* p[3];
    const double* t;
    double rel, y_it;
    int asc_above, des_below, position;
    size_t j, j_lo, j_hi;

    /* y-descending, with the tie behaviour of libstdc++'s std::sort on 3 elements
     * (a stable insertion sort with a strict comparator) — plane.cpp:61 */
    p[0] = a;
    p[1] = b;
    p[2] = c;
    if (p[1][1] > p[0][1]) { t = p[0]; p[0] = p[1]; p[1] = t; }
    if (p[2][1] > p[0][1]) { t = p[2]; p[2] = p[1]; p[1] = p[0]; p[0] = t; }
    else if (p[2][1] > p[1][1]) { t = p[1]; p[1] = p[2]; p[2] = t; }

    rel = side_of(p[0], p[2], p[1]);
    asc_above = (p[0][0] >= p[2][0]) && (rel >= 0);
    des_below = (p[0][0] < p[2][0]) && (rel > 0);
    position = !(asc_above || des_below);

    j_hi = (size_t)floor(pix_of_y(g, p[0][1]));
    j_lo = (size_t)ceil(pix_of_y(g, p[2][1]));
    y_it = g->ys[j_lo];

    for (j = j_lo; j <= j_hi; j++) {
        double x_lo, x_hi;
        size_t i, i_lo, i_hi;
        if (position) {
            x_lo = edge_x_at(p[0], p[2], y_it);
            x_hi = (y_it < p[1][1]) ? edge_x_at(p[2], p[1], y_it) : edge_x_at(p[0], p[1], y_it);
        } else {
            x_hi = edge_x_at(p[0], p[2], y_it);
            x_lo = (y_it < p[1][1]) ? edge_x_at(p[2], p[1], y_it) : edge_x_at(p[0], p[1], y_it);
        }
        i_hi = (size_t)floor(pix_of_x(g, x_hi));
        i_lo = (size_t)ceil(pix_of_x(g, x_lo));
        for (i = i_lo; i <= i_hi; i++) emit(ctx, i, j);
        y_it = y_it + g->step_y;
    }
}

/* ------------------------------------------------------------------ record collection */

typedef struct rec {
    uint32_t pixel; /* j * res_x + i */
    uint32_t data;  /* face bits 31..28 | tet id 27..0 — line.hpp:71-79 */
} rec;

typedef struct rec_list {
    rec* v;
    size_t n, cap;
    int failed;
} rec_list;

static void rec_push(rec_list* l, uint32_t pixel, uint32_t data) {
    if (l->n == l->cap) {
        size_t cap = l->cap ? l->cap * 2 : (1u << 16);
        rec* nv = (rec*)realloc(l->v, cap * sizeof(rec));
        if (!nv) {
            l->failed = 1;
            return;
        }
        l->v = nv;
        l->cap = cap;
    }
    l->v[l->n].pixel = pixel;
    l->v[l->n].data = data;
    l->n++;
}

/* hits of the 4 faces of ONE tet: key = pixel * 4 + face */
typedef struct hit_buf {
    uint64_t* v;
    size_t n, cap;
    int res_x;
    unsigned face;
    int failed;
} hit_buf;

static void emit_hit(void* ctx, size_t i, size_t j) {
    hit_buf* h = (hit_buf*)ctx;
    if (h->n == h->cap) {
        size_t cap = h->cap ? h->cap * 2 : 256;
        uint64_t* nv = (uint64_t*)realloc(h->v, cap * sizeof(uint64_t));
        if (!nv) {
            h->failed = 1;
            return;
        }
        h->v = nv;
        h->cap = cap;
    }
    h->v[h->n++] = ((uint64_t)(j * (size_t)h->res_x + i) << 2) | h->face;
}

static int cmp_u64(const void* a, const void* b) {
    const uint64_t x = *(const uint64_t*)a, y = *(const uint64_t*)b;
    return (x > y) - (x < y);
}

typedef struct solid_ctx {
    uint8_t* mask;
    int res_x;
} solid_ctx;

static void emit_solid(void* ctx, size_t i, size_t j) {
    solid_ctx* s = (solid_ctx*)ctx;
    s->mask[j * (size_t)s->res_x + i] = 1;
}

/* ------------------------------------------------------------------ per-pixel integration */

/* z of the plane through p1,p2,p3 at (x, y) — line.cpp:150-174 */
static double face_z(double x, double y, const double* p1, const double* p2, const double* p3) {
    const double x_x1 = (x - p1[0]) * ((p2[1] - p1[1]) * (p3[2] - p1[2]) - (p3[1] - p1[1]) * (p2[2] - p1[2]));
    const double y_y1 = (y - p1[1]) * ((p2[0] - p1[0]) * (p3[2] - p1[2]) - (p3[0] - p1[0]) * (p2[2] - p1[2]));
    const double z_minor = ((p2[0] - p1[0]) * (p3[1] - p1[1]) - (p3[0] - p1[0]) * (p2[1] - p1[1]));
    return (y_y1 - x_x1) / z_minor + p1[2];
}

typedef struct seg {
    double key_z; /* the higher of the two face z's */
    double dz;
    uint32_t tet;
} seg;

static int cmp_seg_desc(const void* a, const void* b) {
    const double x = ((const seg*)a)->key_z, y = ((const seg*)b)->key_z;
    return (x < y) - (x > y);
}

/* The whole pass, shared by c5o_render and c5o_render_segments. tau and inten may be NULL (not
 * stored); with seg_tet, each pixel's segments are also stored at seg_start[pix] .. seg_start[pix + 1]
 * in the order I is integrated (r = n - 1 .. 0), and a pixel whose record count differs from that
 * span makes the pass return -3. */
static int render_pass(const double* tet_pts, const double* alpha, const double* q, int64_t n_tets,
                       const double* solid_pts, int64_t n_solid, const c5o_view* v, double* tau, double* inten,
                       uint32_t* steps, uint8_t* solid, uint64_t* total_steps, uint64_t* anomalies,
                       const int64_t* seg_start, int32_t* seg_tet, double* seg_dz) {
    grid g;
    size_t n_pix;
    uint8_t* mask = NULL;
    rec_list* lists = NULL;
    size_t* start = NULL;
    rec* csr = NULL;
    int n_thr = 1, t, rc = 0;
    uint64_t odd = 0, sum_steps = 0, mismatch = 0;
    int64_t k;

    if (!v || v->res_x < 2 || v->res_y < 2 || n_tets < 0 || n_tets >= (1 << 28)) return -1;
    n_pix = (size_t)v->res_x * (size_t)v->res_y;
    if (n_pix >= 0xFFFFFFFFu) return -1;

    g.res_x = v->res_x;
    g.res_y = v->res_y;
    g.x_min = v->window[1];
    g.y_min = v->window[3];
    g.step_x = (v->window[0] - v->window[1]) / (v->res_x - 1.);
    g.step_y = (v->window[2] - v->window[3]) / (v->res_y - 1.);
    g.xs = (double*)malloc(sizeof(double) * (size_t)v->res_x);
    g.ys = (double*)malloc(sizeof(double) * (size_t)v->res_y);
    mask = (uint8_t*)calloc(n_pix, 1);
    if (!g.xs || !g.ys || !mask) {
        rc = -2;
        goto done;
    }
    c5o_pixel_coords(v, g.xs, g.ys);

#ifdef _OPENMP
    n_thr = v->threads > 0 ? v->threads : omp_get_max_threads();
#endif
    lists = (rec_list*)calloc((size_t)n_thr, sizeof(rec_list));
    if (!lists) {
        rc = -2;
        goto done;
    }

    /* solids first: a solid pixel yields NaN whatever else covers it, so order is immaterial */
#pragma omp parallel for num_threads(n_thr) schedule(dynamic, 64)
    for (k = 0; k < n_solid; k++) {
        const double* p = solid_pts + 12 * k;
        solid_ctx s;
        s.mask = mask;
        s.res_x = v->res_x;
        scan_face(&g, p + 0, p + 3, p + 6, emit_solid, &s);
        scan_face(&g, p + 0, p + 3, p + 9, emit_solid, &s);
        scan_face(&g, p + 0, p + 6, p + 9, emit_solid, &s);
        scan_face(&g, p + 3, p + 6, p + 9, emit_solid, &s);
    }

    /* transparent tets: scan the 4 faces, pair face hits per pixel into records */
#pragma omp parallel num_threads(n_thr) reduction(+ : odd)
    {
        int me = 0;
        hit_buf h;
        int64_t id;
#ifdef _OPENMP
        me = omp_get_thread_num();
#endif
        memset(&h, 0, sizeof(h));
        h.res_x = v->res_x;
#pragma omp for schedule(dynamic, 64)
        for (id = 0; id < n_tets; id++) {
            const double* p = tet_pts + 12 * id;
            size_t a;
            h.n = 0;
            /* face f omits vertex 3 - f (plane.cpp:30-37) */
            h.face = 0; scan_face(&g, p + 0, p + 3, p + 6, emit_hit, &h);
            h.face = 1; scan_face(&g, p + 0, p + 3, p + 9, emit_hit, &h);
            h.face = 2; scan_face(&g, p + 0, p + 6, p + 9, emit_hit, &h);
            h.face = 3; scan_face(&g, p + 3, p + 6, p + 9, emit_hit, &h);
            if (h.n > 1) qsort(h.v, h.n, sizeof(uint64_t), cmp_u64);
            /* consecutive hits of one pixel, in face order, pair up (line.cpp:34-54) */
            for (a = 0; a < h.n;) {
                const uint64_t pixel = h.v[a] >> 2;
                size_t b = a;
                while (b < h.n && (h.v[b] >> 2) == pixel) b++;
                while (a + 1 < b) {
                    const uint32_t bits = (1u << (28 + (h.v[a] & 3))) | (1u << (28 + (h.v[a + 1] & 3)));
                    rec_push(&lists[me], (uint32_t)pixel, bits | (uint32_t)id);
                    a += 2;
                }
                if (a < b) {
                    odd++;
                    a = b;
                }
            }
        }
        free(h.v);
        if (h.failed) lists[me].failed = 1;
    }
    for (t = 0; t < n_thr; t++) {
        if (lists[t].failed) rc = -2;
    }
    if (rc) goto done;

    /* bucket the records by pixel (CSR) */
    start = (size_t*)calloc(n_pix + 1, sizeof(size_t));
    if (!start) {
        rc = -2;
        goto done;
    }
    {
        size_t total = 0, i;
        for (t = 0; t < n_thr; t++) {
            for (i = 0; i < lists[t].n; i++) start[lists[t].v[i].pixel + 1]++;
            total += lists[t].n;
        }
        for (i = 0; i < n_pix; i++) start[i + 1] += start[i];
        csr = (rec*)malloc((total ? total : 1) * sizeof(rec));
        if (!csr) {
            rc = -2;
            goto done;
        }
        {
            size_t* fill = (size_t*)malloc(n_pix * sizeof(size_t));
            if (!fill) {
                rc = -2;
                goto done;
            }
            memcpy(fill, start, n_pix * sizeof(size_t));
            for (t = 0; t < n_thr; t++) {
                for (i = 0; i < lists[t].n; i++) csr[fill[lists[t].v[i].pixel]++] = lists[t].v[i];
                free(lists[t].v);
                lists[t].v = NULL;
            }
            free(fill);
        }
    }

    /* per pixel: face z's, order, integrate */
#pragma omp parallel num_threads(n_thr) reduction(+ : sum_steps, mismatch)
    {
        seg* segs = NULL;
        size_t segs_cap = 0;
        int64_t pix;
#pragma omp for schedule(dynamic, 256)
        for (pix = 0; pix < (int64_t)n_pix; pix++) {
            const size_t b = start[pix], e = start[pix + 1], n = e - b;
            const double x = g.xs[pix % v->res_x], y = g.ys[pix / v->res_x];
            size_t r;
            double sum, I;
            if (mask[pix]) {
                if (tau) tau[pix] = NAN;
                if (inten) inten[pix] = NAN;
                if (steps) steps[pix] = 0;
                if (seg_tet && seg_start[pix + 1] != seg_start[pix]) mismatch++;
                continue;
            }
            if (steps) steps[pix] = (uint32_t)n;
            sum_steps += n;
            if (n > segs_cap) {
                free(segs);
                segs_cap = n * 2;
                segs = (seg*)malloc(segs_cap * sizeof(seg));
            }
            for (r = 0; r < n; r++) {
                const uint32_t d = csr[b + r].data;
                const uint32_t id = d & 0x0FFFFFFFu;
                const double* p = tet_pts + 12 * (size_t)id;
                double z[2] = {0, 0};
                int m = 0;
                /* bit 31 -> (v1,v2,v3), 30 -> (v0,v2,v3), 29 -> (v0,v1,v3), 28 -> (v0,v1,v2) */
                if (d & (1u << 31)) z[m++] = face_z(x, y, p + 3, p + 6, p + 9);
                if (d & (1u << 30)) z[m++] = face_z(x, y, p + 0, p + 6, p + 9);
                if (d & (1u << 29)) z[m++] = face_z(x, y, p + 0, p + 3, p + 9);
                if (d & (1u << 28)) z[m++] = face_z(x, y, p + 0, p + 3, p + 6);
                if (z[0] < z[1]) {
                    const double s = z[0];
                    z[0] = z[1];
                    z[1] = s;
                }
                segs[r].key_z = z[0];
                segs[r].dz = z[0] - z[1];
                segs[r].tet = id;
            }
            if (n > 1) qsort(segs, n, sizeof(seg), cmp_seg_desc);
            if (seg_tet) {
                if (seg_start[pix + 1] - seg_start[pix] != (int64_t)n) {
                    mismatch++;
                } else {
                    int64_t o = seg_start[pix];
                    for (r = n; r-- > 0; o++) {
                        seg_tet[o] = (int32_t)segs[r].tet;
                        seg_dz[o] = segs[r].dz;
                    }
                }
            }

            sum = 0;
            for (r = 0; r < n; r++) sum = sum + segs[r].dz * alpha[segs[r].tet];

            I = 0;
            for (r = n; r-- > 0;) {
                const double Q = q[segs[r].tet];
                double a = alpha[segs[r].tet];
                double Cc;
                if (a > v->alpha_limit) a = v->alpha_limit;
                Cc = Q - a * I;
                if (!(a < DBL_EPSILON)) I = (Q - Cc * exp(-a * segs[r].dz)) / a;
            }
            if (tau) tau[pix] = sum;
            if (inten) inten[pix] = I;
        }
        free(segs);
    }
    if (solid) memcpy(solid, mask, n_pix);
    if (total_steps) *total_steps = sum_steps;
    if (anomalies) *anomalies = odd;
    if (mismatch) rc = -3;

done:
    if (lists) {
        for (t = 0; t < n_thr; t++) free(lists[t].v);
        free(lists);
    }
    free(start);
    free(csr);
    free(mask);
    free(g.xs);
    free(g.ys);
    return rc;
}

int c5o_render(const double* tet_pts, const double* alpha, const double* q, int64_t n_tets,
               const double* solid_pts, int64_t n_solid, const c5o_view* v, double* tau, double* inten,
               uint32_t* steps, uint8_t* solid, uint64_t* total_steps, uint64_t* anomalies) {
    if (!tau || !inten) return -1;
    return render_pass(tet_pts, alpha, q, n_tets, solid_pts, n_solid, v, tau, inten, steps, solid, total_steps,
                       anomalies, NULL, NULL, NULL);
}

int c5o_render_segments(const double* tet_pts, const double* alpha, const double* q, int64_t n_tets,
                        const double* solid_pts, int64_t n_solid, const c5o_view* v, const int64_t* seg_start,
                        int32_t* seg_tet, double* seg_dz) {
    if (!seg_start || !seg_tet || !seg_dz) return -1;
    return render_pass(tet_pts, alpha, q, n_tets, solid_pts, n_solid, v, NULL, NULL, NULL, NULL, NULL, NULL,
                       seg_start, seg_tet, seg_dz);
}
