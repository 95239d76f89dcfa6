/* c5gpu.h — C ABI of the B200 ray pass that replaces course5's OpenMP loops.
 *
 * The reference has no plugin/FFI API; its hot path is reached by three C++ calls in one
 * place (/root/reference/project/src/main.cpp:127-129):
 *
 *     plane base_plane{res_x, res_y, {acc_disk, roche_lobe, acc_sphere}, domain};   // :127
 *     base_plane.find_intersections();                                              // :128
 *     object2d result = base_plane.trace_rays(tetra_value::alpha, tetra_value::Q);  // :129
 *
 * preceded by three rotations per object (main.cpp:104-107,112-114) that the reference
 * charges to its load timer. This header is what a binding for that path links against:
 * plain pointers and sizes, no C++ or torch types, no exceptions. Every call returns C5_OK
 * or a negative C5_E_* code; c5_last_error() gives the text. A context is thread-compatible
 * (one thread at a time), not thread-safe.
 *
 * The library is CUDA-only (sm_100a). There is no CPU path: without a usable device
 * c5_create() fails with C5_E_CUDA.
 */
#ifndef C5GPU_H
#define C5GPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define C5_ABI_VERSION 9
#define C5_MAX_IN_FLIGHT 8
#define C5_MAX_ROT 8
#define C5_MAX_CHANNELS 8
#define C5_MAX_POINTS (1 << 26) /* c5_upload_mesh: points per mesh (vertex ids are packed in 26 bits) */

typedef struct c5_ctx c5_ctx;

enum c5_status {
    C5_OK = 0,
    C5_E_INVALID = -1,  /* bad argument */
    C5_E_CUDA = -2,     /* CUDA runtime error / no device */
    C5_E_NOMEM = -3,
    C5_E_TOPOLOGY = -4, /* mesh is not a conforming manifold partition (a face shared by >2 tets) */
    C5_E_STATE = -5,    /* call order (render before upload_mesh, ...) */
    C5_E_WALK = -6,     /* a ray exceeded the step cap (reported in c5_stats.walk_errors too) */
    C5_E_NCCL = -7      /* no longer returned; the value stays reserved */
};

/* One rigid rotation, the unit of object3d_base::rotate_around_{x,y}_axis
 * (object3d_base.cpp:202-219 -> tetra.cpp:44-62). axis 0: about the x axis through the origin;
 * axis 1: about the axis parallel to y through (x0, 0, 0). angle in radians. */
typedef struct c5_rotation {
    int32_t axis;
    int32_t reserved;
    double angle;
    double x0;
} c5_rotation;

/* One view. Replaces the implicit inputs of the reference's ray pass: the plane constructor
 * arguments (plane.hpp:19), the window literal (main.cpp:83), the rotations applied to the
 * geometry beforehand (main.cpp:96,104-107) and app::instance().config.limit_alpha_value read
 * inside the loop (line.cpp:204). */
typedef struct c5_view {
    int32_t res_x, res_y;       /* plane(res_x, res_y, ...) */
    double window[4];           /* x_max, x_min, y_max, y_min */
    int32_t n_rot;              /* rotations applied in order to the grid and to view-following solids */
    int32_t reserved0;
    c5_rotation rot[C5_MAX_ROT];
    double alpha_limit;         /* --alpha_limit */
    int32_t precision;          /* 64 (default) or 32 */
    int32_t round_through_float;/* 1: (double)(float)v like plane.cpp:165-166 + object2d.cpp:19-20 */
    int32_t use_solids;         /* 1: pixels under uploaded solid tets become NaN (line.cpp:246-249) */
    int32_t row_begin, row_end; /* row band [row_begin, row_end); 0,0 = all rows */
    int32_t reserved1;
} c5_view;

/* Fills *v the way main.cpp:83-107 sets a view up from the CLI flags (angles in units of pi):
 * window {2.2,-0.2,0.9,-0.9}; rotations Rx(a0), Ry(Y*pi) about x0 = 1, Rx(-a0 + X*pi),
 * a0 = -I*pi + pi/2; precision 64; round_through_float 1; use_solids 1; all rows. */
void c5_view_from_flags(c5_view* v, int32_t res_x, int32_t res_y, double X_pi, double Y_pi, double I_pi,
                        double alpha_limit);

typedef struct c5_stats {
    uint64_t pixels;        /* pixels of the rendered band(s) */
    uint64_t tet_steps;     /* sum over pixels of tets crossed == plane::count_all_intersections (plane.cpp:3-12) */
    uint64_t hit_pixels;    /* pixels crossing >= 1 tet */
    uint64_t solid_pixels;  /* pixels under the solid mask */
    uint64_t walk_errors;   /* rays stopped by the step cap (0 on a valid mesh) */
    float ms_rotate;        /* device time per phase (CUDA events), max over devices */
    float ms_bvh;
    float ms_mask;
    float ms_walk;
    float ms_gather;        /* always 0 (nothing is gathered); kept for the struct's layout */
    float ms_d2h;
    float ms_total;         /* whole call on the device timeline, max over devices */
    int32_t n_devices;
    int32_t grazing_rays;   /* rays with so many crossings that the grazing-ray kernel finished them */
    float ms_graze;         /* the grazing-ray kernel's share of ms_walk */
    int32_t reserved;
} c5_stats;

typedef struct c5_mesh_info {
    int64_t n_points, n_tets, n_boundary_faces, n_bvh_nodes, n_solid_tets;
    int64_t device_bytes;   /* per device */
} c5_mesh_info;

/* devices: CUDA ordinals, n_dev >= 1. With n_dev > 1 the mesh is replicated, each device
 * renders a contiguous band of rows (cut by the previous view's cost) and stores it in its rows
 * of the caller's buffers: in place if `out` is page-locked, else by its own device-to-host copy. */
int c5_create(const int32_t* devices, int32_t n_dev, c5_ctx** out);
void c5_destroy(c5_ctx* ctx);
const char* c5_last_error(const c5_ctx* ctx); /* ctx may be NULL: text of the last failed c5_create */
int c5_abi_version(void);

/* Replaces object3d_base::read_vtk_file's output (object3d_base.cpp:13-52: an AoS of private
 * per-tet point copies) by shared points + connectivity, which are flattened once into
 * device-resident arrays: Morton-reordered vertices and tets, a face-neighbour table, the
 * boundary-face list and an LBVH hierarchy over it. Caller keeps ownership of the host arrays;
 * the call blocks. alpha = "AbsorpCoef", q = "radEnLooseRate" (object3d_accretion_disk.cpp:4).
 * At most C5_MAX_POINTS points (67,108,864) and fewer than 2^29 tets; a larger mesh is C5_E_INVALID, refused
 * before any of its arrays is read. */
int c5_upload_mesh(c5_ctx* ctx, const double* points_xyz, int64_t n_points, const int32_t* tet_vertices,
                   int64_t n_tets, const double* alpha, const double* q);

/* Solid tets (the reference's Roche lobe and sphere, tetra_type::solid): [n][4][3] doubles in the
 * frame BEFORE the view rotations. follows_view = 1 for objects main.cpp rotates with the view
 * (the Roche lobe, main.cpp:112-114), 0 for those it does not (the sphere, main.cpp:116). Calls
 * append; c5_clear_solids() empties the set. */
int c5_upload_solids(c5_ctx* ctx, const double* tet_points, int64_t n_tets, int32_t follows_view);
int c5_clear_solids(c5_ctx* ctx);

int c5_mesh_info_get(const c5_ctx* ctx, c5_mesh_info* out);

/* plane ctor + find_intersections + trace_rays for one view (main.cpp:127-129), including the
 * rotations main.cpp:104-107 does beforehand. out: caller-owned HOST buffer of
 * res_y * res_x * 2 doubles, x fastest, {tau, I} per pixel — the vtkImageData layout of
 * object2d.cpp:17-21 (with a row band: only rows [row_begin,row_end) are written, at their
 * final position). stats may be NULL. If `out` is page-locked (cudaHostAlloc, cudaHostRegister or
 * c5_host_register) and 16-byte aligned the walk kernel stores its pixels straight into it over
 * PCIe (the shortest path for one view at a time); any other buffer gets a device-to-host copy. */
int c5_render(c5_ctx* ctx, const c5_view* view, double* out, c5_stats* stats);

/* The same pass, asynchronous: c5_render_submit enqueues the view and returns a ticket at once;
 * c5_render_wait blocks until that view's image is complete in `out` and fills stats (may be NULL).
 * Up to c5_set_views_in_flight() views (default 3, at most C5_MAX_IN_FLIGHT) may be submitted before
 * the first is waited for; each is rendered by a lane of its own — per-view device state plus a
 * stream; the mesh is shared — so that consecutive views overlap on the device: the tail of one
 * view's walk and its grazing-ray kernel run beside the next view's rays, and the copy engine moves
 * one view's image to the host while the SMs walk the next. `out` (page-locked for any overlap: a
 * copy to pageable memory blocks the submitting thread) must stay valid and untouched
 * until the wait returns; *view is copied. One more submit than lanes returns C5_E_STATE. Tickets may
 * be waited for in any order, once each. A sweep is: submit k+1, k+2; wait k; write frame k; ...
 * Single-device contexts that are not siblings. */
int c5_render_submit(c5_ctx* ctx, const c5_view* view, double* out, uint64_t* ticket);
int c5_render_wait(c5_ctx* ctx, uint64_t ticket, c5_stats* stats);
int c5_set_views_in_flight(c5_ctx* ctx, int32_t n);

/* Test/diagnostic variant: same pass, but also returns per-pixel tets crossed and the solid
 * mask (each res_y * res_x, x fastest; either may be NULL). With view->round_through_float = 0
 * the doubles are the pre-cast values the parity gate is defined on. */
int c5_render_raw(c5_ctx* ctx, const c5_view* view, double* out, uint32_t* steps, uint8_t* solid_mask,
                  c5_stats* stats);

/* ---- several field pairs from one view ------------------------------------------------------------
 * c5_upload_channels replaces the context's channels: n_channels (0 .. C5_MAX_CHANNELS) pairs of cell
 * fields, alpha and q each n_channels * n_tets doubles, channel-major (alpha[c * n_tets + k] for tet k
 * in the order given to c5_upload_mesh). n_channels = 0 removes them. Needs a mesh (C5_E_STATE
 * otherwise); goes through the parent like every upload (C5_E_STATE on a sibling) and reaches the
 * parts of a multi-device context; siblings and lanes see it at their next render. C5_E_STATE while
 * the context or one of its lanes has a submitted view. No topology or BVH is rebuilt;
 * c5_upload_mesh drops the channels. While channels are uploaded, c5_mesh_info.device_bytes
 * includes them.
 *
 * c5_render_channels is c5_render_raw over the uploaded channels, in ONE walk: out holds
 * res_y * res_x * n * 2 doubles, x fastest, {tau_0, I_0, ..., tau_{n-1}, I_{n-1}} per pixel (a row
 * band writes only its rows). Channel c is the image c5_render_raw gives for a mesh uploaded with
 * (alpha_c, q_c): the same rays, hit set, solid mask and steps. steps, solid_mask and stats mean what
 * they mean for c5_render_raw (counts are the geometry's, not multiplied by n); steps and solid_mask
 * may be NULL. A page-locked, 16-byte aligned `out` is written in place. FP64 only: precision 32 is
 * C5_E_INVALID; no channels uploaded is C5_E_STATE. Single- and multi-device contexts and siblings. */
int c5_upload_channels(c5_ctx* ctx, const double* alpha, const double* q, int32_t n_channels);
int c5_render_channels(c5_ctx* ctx, const c5_view* view, double* out, uint32_t* steps, uint8_t* solid_mask,
                       c5_stats* stats);

/* ---- flux: per-row sums of a view, reduced on the device (light curves) ---------------------------
 * The image stays in device memory; only its row sums reach the host (16 bytes per pair and row).
 * For a view and its n pairs:
 *   rows[j][c]  = {sum_i tau_c(i,j), sum_i I_c(i,j)} over the pixels of row j NOT under the solid mask,
 *                 of exactly the doubles the image would hold for the same view (round_through_float
 *                 and precision included); background pixels add their 0, and a NaN outside the mask
 *                 makes the sum NaN;
 *   total[c]    = the sum of rows[j][c] in increasing j, accumulated in double on the host.
 * Summation order of a row: one block of 256 threads; thread t adds the pixels x = t, t+256, ... in
 * increasing x, starting from 0; the 256 partials are folded by a halving tree, p[t] += p[t+s] for
 * s = 128, 64, ..., 1. The sums are therefore bit-identical for any row band, any number of devices
 * and any number of views in flight.
 *
 * channels: 0 = the cells' own alpha/Q (one pair; precision 64 or 32), 1 = all uploaded channels
 * (n pairs; FP64 only, like c5_render_channels). rows: res_y * n * 2 doubles, rows outside the
 * view's band are written as 0; total: n * 2 doubles. Either may be NULL, not both.
 * Stats mean what they mean for c5_render_raw (the geometry is counted once), except that ms_d2h
 * is the time from the end of the walk until the row sums are in host memory: the reduction and a
 * copy of a few KB. C5_E_INVALID: both outputs NULL, channels not 0 or 1, or precision 32 with
 * channels = 1. C5_E_STATE: no mesh, or channels = 1 with none uploaded.
 *
 * c5_render_flux works on single-device, multi-device and sibling contexts; a multi-device context
 * reduces each device's band on that device and merges the rows. c5_render_flux_submit is the
 * pipelined form with the scope of c5_render_submit (single-device contexts that are not siblings,
 * C5_E_STATE otherwise): it shares the lanes, the tickets and c5_render_wait with it, which writes
 * rows / total (need not be page-locked; they must stay valid until the wait returns). */
int c5_render_flux(c5_ctx* ctx, const c5_view* view, int32_t channels, double* rows, double* total,
                   c5_stats* stats);
int c5_render_flux_submit(c5_ctx* ctx, const c5_view* view, int32_t channels, double* rows, double* total,
                          uint64_t* ticket);

/* ---- gradients: the derivative of a view with respect to every tet's alpha and Q --------------------
 * c5_update_fields replaces the cells' own alpha and Q (n_tets doubles each, tets in the order given to
 * c5_upload_mesh) without rebuilding topology or BVH; channels and solids stay. It goes through the
 * parent like every upload and reaches the parts of a multi-device context; siblings and lanes see the
 * new fields at their next render. Every render afterwards is bit-identical to one from a context
 * uploaded with these fields. C5_E_INVALID: NULL array. C5_E_STATE: no mesh, a sibling context, or a
 * submitted view in flight on the context or one of its lanes.
 *
 * c5_render_grad computes, for one view, the vector-Jacobian product of the pre-cast image (what
 * c5_render_raw gives with round_through_float = 0) against an upstream gradient g: res_y * res_x * 2
 * doubles, x fastest, {g_tau, g_I} per pixel, of which only the view's row band is read. It writes, in
 * the tet order given to c5_upload_mesh and overwriting,
 *   grad_alpha[t] = sum over pixels of g_tau dtau/dalpha_t + g_I dI/dalpha_t
 *   grad_q[t]     = sum over pixels of g_I dI/dQ_t
 * Pixels under the solid mask and background pixels contribute nothing. The derivative is that of the
 * function the walk computes, segment lengths included: vertex positions and the view are not
 * parameters. dtau/dalpha_t counts every segment (tau uses the unclamped alpha); a segment whose
 * min(alpha, alpha_limit) is below DBL_EPSILON leaves I unchanged and adds nothing to dI; dI/dalpha_t is
 * 0 where alpha_t > alpha_limit (the clamp) and flows where alpha_t == alpha_limit.
 * Either gradient array may be NULL, not both. out (optional, res_y * res_x * 2 doubles) receives the
 * {tau, I} image c5_render_raw gives for the view, bit for bit. stats mean what they mean for
 * c5_render_raw, except that ms_d2h spans the gradient pass and the copies of the gradients.
 * The call runs two walks over the same rays, a depth pass and a gradient pass: two kernel launches
 * more than c5_render_raw of the same view (none more when the mesh is outside the band). Each device
 * adds its band's contributions into its own buffers with FP64 atomics, so the gradients are NOT
 * bit-reproducible from run to run (they agree to rounding, ~1e-15 relative); a multi-device context
 * adds the devices' gradients on the host in device order. g and the gradients are host arrays
 * (copied in and out on every call); c5_render_grad_device below is the same call on device memory.
 * C5_E_INVALID: NULL g, both gradient arrays NULL, precision 32, or
 * round_through_float != 0 (the float cast is piecewise constant: ask for the raw values).
 * C5_E_STATE: no mesh, or a submitted view in flight on this context. Single-device, multi-device and
 * sibling contexts. Not covered: uploaded channels, the FP32 variant. The views of a light curve go through
 * the lanes in one call, c5_render_flux_grad_device below. */
int c5_update_fields(c5_ctx* ctx, const double* alpha, const double* q);
int c5_render_grad(c5_ctx* ctx, const c5_view* view, const double* g, double* grad_alpha, double* grad_q, double* out,
                   c5_stats* stats);

/* ---- gradients on device memory (fit loops whose fields, loss and optimiser live on the GPU) -------------
 * c5_update_fields_device is c5_update_fields with d_alpha and d_q DEVICE pointers on the context's device
 * (n_tets doubles each, tets in the order given to c5_upload_mesh), gathered into the cells on the device
 * by one kernel through a device copy of the tet permutation. That copy (4 bytes per tet, shared with
 * siblings) is made at the first call of either device form and counted in c5_mesh_info.device_bytes from
 * then on; c5_upload_mesh drops it. Same semantics as c5_update_fields: channels and solids stay, and every
 * render afterwards is bit-identical to one from a fresh upload of these fields.
 * Ordering, without synchronising the host: the gather is enqueued on `stream` (a cudaStream_t; NULL = the
 * legacy default stream) after `stream` has waited (events) for everything the library had enqueued on the
 * internal streams of the context, its lanes and its siblings; those internal streams, and those of lanes
 * and siblings made later, then wait for the gather, so the library's later renders (c5_render, c5_render_raw, c5_render_flux, submits, ...) and the
 * caller's later work on `stream` see the new fields. Work the caller put on streams of its own (e.g.
 * c5_render_device with stats == NULL) is the caller's to order, as for c5_render_device. d_alpha and d_q
 * must stay valid until the gather has run on `stream`. C5_E_INVALID: a NULL or not 8-byte aligned pointer,
 * or a multi-device context (single-device contexts only). C5_E_STATE: no mesh, a sibling context, or a
 * submitted view in flight on the context or one of its lanes.
 *
 * c5_render_grad_device is c5_render_grad on device memory, enqueued on `stream`. Band-sized buffers, as
 * for c5_render_device: d_g holds (row_end - row_begin) * res_x * 2 doubles, {g_tau, g_I} per pixel of the
 * view's row band (0,0 = all rows), and the optional d_out the same number, receiving that band of the
 * image c5_render_raw gives, bit for bit. d_grad_alpha and d_grad_q (n_tets doubles each, file order,
 * overwritten; either may be NULL, not both) are scattered from the walk's Morton order on the device.
 * stats == NULL: enqueue only — nothing is read back, the host is not synchronised, and a ray stopped by the
 * step cap is not reported; successive calls and the caller's work on `stream` pipeline on the device.
 * The context's own later renders wait for the call (an event; the host does not wait). Successive
 * device-form calls on one context share its scratch buffers: keep them on one stream, or order them.
 * stats != NULL: `stream` is synchronised and stats are those of c5_render_grad. Three kernel launches more
 * than c5_render_raw of the same view (the gradient pass's two and the scatter). C5_E_INVALID: any cause
 * c5_render_grad has, a pointer not 8-byte aligned, or a multi-device context. C5_E_STATE: no mesh, or a
 * submitted view in flight on this context. Single-device contexts and siblings. */
int c5_update_fields_device(c5_ctx* ctx, const double* d_alpha, const double* d_q, void* stream);
int c5_render_grad_device(c5_ctx* ctx, const c5_view* view, const double* d_g, double* d_grad_alpha, double* d_grad_q,
                          double* d_out, void* stream, c5_stats* stats);

/* c5_render_flux_grad_device is the gradient of a light curve, on device memory: with total_k view k's
 * c5_render_flux total {sum tau, sum I} (round_through_float = 0), it gives the gradient of
 * sum_k g_k . total_k, that is
 *   grad_alpha[t] = sum_k sum_{p not under the solid mask} (g_tau_k dtau_p/dalpha_t + g_I_k dI_p/dalpha_t),
 * and grad_q[t] likewise with g_I_k dI_p/dQ_t. d_g holds n_views * 2 doubles {g_tau_k, g_I_k} on the
 * context's device; the kernels read it, the host does not. d_grad_alpha and d_grad_q (n_tets doubles
 * each, file order, overwritten; either may be NULL, not both) as for c5_render_grad_device. Each view
 * keeps its own resolution, window, rotations and row band; views of different sizes may be mixed.
 * The views are dealt round-robin to the context's lanes (c5_set_views_in_flight, the lanes of
 * c5_render_submit); each runs the depth pass and the gradient pass on its lane's stream, all lanes add
 * into one accumulator, and one scatter to file order runs at the end. Ordering, without synchronising the
 * host: the accumulator is zeroed on `stream` and every lane starts after that, so after the caller's
 * earlier work on `stream` (a c5_update_fields_device, whatever wrote d_g); `stream` then waits for every
 * lane and runs the scatter, and the context's own later renders wait for it. Launches: the sum over the
 * views of what c5_render_grad_device launches for each, less n_views - 1 (one scatter per call).
 * stats == NULL: enqueue only, as for c5_render_grad_device. stats != NULL: `stream` is synchronised; the
 * counts are summed over the views, each counted as c5_render_raw counts it, ms_total is the call's span
 * on `stream` and the other ms_* fields are 0; a ray stopped by the step cap is C5_E_WALK.
 * c5_last_row_cost is not changed. C5_E_INVALID: n_views < 1, NULL views or d_g, a pointer not 8-byte
 * aligned, both gradients NULL, precision 32, round_through_float != 0, or a multi-device context.
 * C5_E_STATE: no mesh, a sibling context, or a submitted view in flight on the context or one of its
 * lanes. */
int c5_render_flux_grad_device(c5_ctx* ctx, const c5_view* views, int32_t n_views, const double* d_g,
                               double* d_grad_alpha, double* d_grad_q, void* stream, c5_stats* stats);

/* ---- forward mode: the Jacobian-vector product of a view along a field direction ------------------------
 * c5_render_jvp gives, for one view, the change of the pre-cast image (what c5_render_raw gives with
 * round_through_float = 0) when the cells' alpha and Q move along the direction (v_alpha, v_q):
 *   tangent[p] = {sum_t dtau_p/dalpha_t v_alpha[t],  sum_t dI_p/dalpha_t v_alpha[t] + dI_p/dQ_t v_q[t]}
 * with the derivatives c5_render_grad uses (the clamp, the DBL_EPSILON skip and the walk's segment lengths
 * alike), so <g, J v> equals <c5_render_grad(g), v> to rounding. v_alpha and v_q are host arrays of n_tets
 * doubles, in the tet order given to c5_upload_mesh; either may be NULL (zero), not both. tangent receives
 * res_y * res_x * 2 doubles {dtau, dI} per pixel, x fastest, in the layout of c5_render_raw's out (a row band
 * writes only its rows); pixels under the solid mask get NaN in both, background pixels 0. out (optional, the
 * same size) receives the {tau, I} image c5_render_raw gives for the view, bit for bit. Only the cells' own
 * fields are differentiated; uploaded channels are not.
 * The tangent is carried forward along each ray beside {tau, I}, in ONE walk: no depth pass and no atomics,
 * since each ray owns its pixel. The result is bit-reproducible from run to run, for any row band, any
 * number of devices and on siblings, and the device form gives the host form's bits. Launches: what
 * c5_render_raw launches for the same view, plus one gather of the direction into the walk's tet order.
 * That tangent field (16 bytes per tet) is made at a context's first call and reused; the context that owns
 * the mesh counts it in c5_mesh_info.device_bytes from then on (a sibling holds its own, not counted), and
 * c5_upload_mesh drops it. stats mean what they mean for c5_render_raw, except that ms_d2h is the copy of
 * both pairs. C5_E_INVALID: NULL tangent, both directions NULL, precision 32, or round_through_float != 0.
 * C5_E_STATE: no mesh, or a submitted view in flight on this context. Single-device, multi-device (each
 * device renders its band of both images) and sibling contexts.
 *
 * c5_render_jvp_device is c5_render_jvp on device memory, enqueued on `stream`, with the ordering contract of
 * c5_render_grad_device: d_v_alpha and d_v_q are n_tets doubles each on the context's device (file order, read
 * by the gather; either may be NULL, not both, 8-byte aligned); d_tangent and the optional d_out hold the view's
 * row band only, (row_end - row_begin) * res_x * 2 doubles, 16-byte aligned as for c5_render_device.
 * stats == NULL: enqueue only. stats != NULL: `stream` is synchronised and stats are those of c5_render_jvp.
 * The context's own later renders wait for the call. C5_E_INVALID: any cause c5_render_jvp has, a misaligned
 * pointer, or a multi-device context. C5_E_STATE as for c5_render_jvp. Single-device contexts and siblings.
 *
 * A Gauss-Newton step needs J^T J v: c5_render_jvp_device along v, then c5_render_grad_device with the
 * tangent as d_g (INTEGRATION.md, section E). */
int c5_render_jvp(c5_ctx* ctx, const c5_view* view, const double* v_alpha, const double* v_q, double* tangent,
                  double* out, c5_stats* stats);
int c5_render_jvp_device(c5_ctx* ctx, const c5_view* view, const double* d_v_alpha, const double* d_v_q,
                         double* d_tangent, double* d_out, void* stream, c5_stats* stats);

/* ---- light curves on device memory: a curve and its J v in one call, the views on the lanes -------------
 * c5_render_flux_device writes, for each view k in view order, the total c5_render_flux gives for it, bit for
 * bit, to d_total: n_views * n * 2 doubles on the context's device, n = 1, or the number of uploaded channels
 * with channels = 1. channels, precision and round_through_float mean what they mean for c5_render_flux.
 *
 * c5_render_flux_jvp_device writes d_tangent[k] = {sum_p dtau_p, sum_p dI_p} (n_views * 2 doubles): view k's
 * c5_render_jvp tangent summed over the pixels outside its solid mask in the flux order above (each row in the
 * order of its 256 threads and halving tree, then the rows in increasing j from 0). The optional d_total
 * (n_views * 2 doubles) receives the views' c5_render_flux totals, bit for bit. d_v_alpha and d_v_q are as
 * for c5_render_jvp_device (file order, either may be NULL, not both, 8-byte aligned). Views must be FP64 with
 * round_through_float = 0; only the cells' own fields are differentiated. d_tangent has exactly the layout
 * c5_render_flux_grad_device reads as d_g, so a light curve's J^T J v is two calls with nothing in between.
 *
 * Both calls deal the views as c5_render_flux_grad_device does: view k goes to lane k % views_in_flight and
 * runs there, on the lane's stream, what c5_render_flux runs for it (the walk, then the row sums; the J v call
 * walks with the tangent beside {tau, I}), then one small kernel that adds the view's rows into its slot of
 * the output. The J v call gathers the direction once, on `stream`, into the context's tangent field (counted
 * in c5_mesh_info.device_bytes as for c5_render_jvp), which every lane reads. Ordering, without synchronising
 * the host: `stream` first waits for the context's own stream, every lane then waits for `stream`, so it sees
 * the caller's earlier work there (a c5_update_fields_device, the writes of the direction), `stream` waits for
 * every lane before the call returns, and the context's own stream waits for `stream`. No atomics: both
 * results are bit-reproducible from run to run, for any number of lanes and any order of the views.
 * Launches: the sum over the views of what c5_render_flux launches for each, plus n_views, plus one gather
 * for the J v call. stats == NULL: enqueue only. stats != NULL: `stream` is synchronised; the counts are
 * summed over the views, ms_total is the call's span on `stream` and the other ms_* fields are 0.
 * C5_E_INVALID: n_views < 1, NULL views, a NULL or not 8-byte aligned output, any argument cause of
 * c5_render_flux (c5_render_flux_device) or c5_render_jvp_device (c5_render_flux_jvp_device), or a multi-device
 * context. C5_E_STATE: no mesh, a sibling context, a submitted view in flight on the context or one of its
 * lanes, or channels = 1 with no channels uploaded. Single-device contexts that are not siblings. */
int c5_render_flux_device(c5_ctx* ctx, const c5_view* views, int32_t n_views, int32_t channels, double* d_total,
                          void* stream, c5_stats* stats);
int c5_render_flux_jvp_device(c5_ctx* ctx, const c5_view* views, int32_t n_views, const double* d_v_alpha,
                              const double* d_v_q, double* d_tangent, double* d_total, void* stream, c5_stats* stats);

/* Device-resident variant for callers that own device memory (e.g. a torch tensor that an NCCL
 * gather will read): d_out is a DEVICE pointer on the context's first device to
 * (row_end - row_begin) * res_x * 2 doubles — the band only. Work is enqueued on `stream`
 * (a cudaStream_t; NULL = the legacy default stream). d_out must be 16-byte aligned (pixels are
 * stored as one 128-bit word; C5_E_INVALID otherwise). With stats != NULL the call returns
 * after the stream has been synchronised, so stats (and c5_last_row_cost) are final. With
 * stats == NULL nothing is read back and the call returns as soon as the work is enqueued: the
 * caller orders later work on the same stream (successive views and an NCCL gather then pipeline
 * on the device without host round trips). Single-device contexts only. */
int c5_render_device(c5_ctx* ctx, const c5_view* view, void* d_out, void* stream, c5_stats* stats);

/* Per-row tet-step totals of the last render on this context (res_y entries; rows outside the
 * rendered band are 0). Callers use it to cut cost-balanced row bands for the next view. */
int c5_last_row_cost(c5_ctx* ctx, uint64_t* rows, int32_t n_rows);

/* A second context on the same device that SHARES parent's uploaded mesh and solids (no copy) and
 * owns only per-view state (rotated vertices, BVH boxes, mask, counters). Two views can then be in
 * flight at once — c5_render_device(parent, ..., stream_a) and c5_render_device(sibling, ...,
 * stream_b) — so that the tail of one view's walk overlaps the start of the next one's: a sweep's
 * throughput is then set by the work, not by the last rays of every view. Uploads go through the
 * parent (a sibling picks them up at its next render); destroy siblings before the parent. */
int c5_create_sibling(c5_ctx* parent, c5_ctx** out);

/* ---- one image, several processes (one process per GPU) -----------------------------------------
 * Row bands are independent (plane.cpp:161-169 has no cross-pixel state), so N processes can
 * render N bands of one view straight into ONE image and nothing has to be gathered afterwards:
 *
 *  - a DEVICE image on one GPU that the other GPUs' walk kernels store into through NVLink peer
 *    mappings (CUDA IPC): the owner calls c5_image_create and passes the 64-byte handle to the
 *    other processes (any byte transport), they call c5_image_open and hand
 *    `(char*)ptr + row_begin * res_x * 16` to c5_render_device as d_out;
 *  - a HOST image in shared memory (shm_open / mmap, the caller's business) that every process
 *    registers with c5_host_register: c5_render() with a row band then writes the band in place
 *    over that GPU's own PCIe link (a registered buffer is device-addressable, so the walk stores
 *    into it directly).
 *
 * Ordering between processes (all bands of view k written before anyone reads view k) is the
 * caller's: one barrier per view on the streams involved. */
#define C5_IPC_HANDLE_BYTES 80 /* a cudaIpcMemHandle_t (64) + the image's offset in its allocation + its size */
int c5_image_create(c5_ctx* ctx, uint64_t bytes, void** d_ptr, uint8_t handle[C5_IPC_HANDLE_BYTES]);
int c5_image_open(c5_ctx* ctx, const uint8_t handle[C5_IPC_HANDLE_BYTES], void** d_ptr);
int c5_image_close(c5_ctx* ctx, void* d_ptr); /* frees (owner) or unmaps (importer) */
int c5_host_register(c5_ctx* ctx, void* ptr, uint64_t bytes);
int c5_host_unregister(c5_ctx* ctx, void* ptr);

/* Number of kernels this library has launched on behalf of ctx (and the lanes c5_render_submit
 * made for it) since creation. */
uint64_t c5_kernel_launches(const c5_ctx* ctx);

/* ---- diagnostics (tests, profiling scripts; no effect on results) ----------------------------------
 * c5_debug_set(ctx, key, value) — applies to ctx, its lanes and its siblings:
 *   "graze_list"    entries one cooperative collection of the grazing-ray kernel holds (128..256, 0 = default):
 *                   tests shrink it to reach the overflow path on small meshes
 *   "query_budget"  BVH nodes a thread of the pixel kernel may visit per search before it hands the
 *                   ray to the grazing-ray kernel (>= 1, 0 = default 64)
 *   "serial_list"   the same for the serial form of the CPU test build (2..64)
 *   "mask_tile"     100 w + h: tile size of the solid mask's "already solid" flags (0 = default)
 *   "no_static_mask" 1: solids that do not follow the view are scan-converted in every view, like the
 *                   others, instead of once per pixel grid (tests compare the two)
 *   "no_zero_copy"  1: page-locked output buffers get a device-to-host copy like pageable ones
 *   "timeline"      n > 0: keep the phase events of the last n views of every lane (0 = off)
 * Unknown keys return C5_E_INVALID.
 * c5_timeline_read: for the last views rendered by ctx itself (not its lanes; oldest first, at most
 * max_views), six times in milliseconds since `origin` (a cudaEvent_t the caller recorded earlier
 * on the same device): view start, vertices rotated, BVH refitted, solid mask done, pixel kernel
 * done, grazing-ray kernel done. Synchronises with the last of them. */
int c5_debug_set(c5_ctx* ctx, const char* key, int64_t value);
int c5_timeline_read(c5_ctx* ctx, void* origin, float* ms_out, int32_t max_views, int32_t* n_views);

#ifdef __cplusplus
}
#endif
#endif /* C5GPU_H */
