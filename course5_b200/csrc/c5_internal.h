// c5_internal.h — context and the entry points shared between the library's translation units.
#pragma once

#include <string>
#include <utility>
#include <vector>

#include "../../include/c5gpu.h"
#include "c5_types.h"

namespace c5 {

constexpr int kMaxRot = C5_MAX_ROT;
constexpr int kTimelinePhases = 6; // start, rotated, refitted, masked, pixel kernel done, grazing-ray kernel done

// Counters the walk kernel accumulates (one 64-bit atomic per warp).
// kDeferred = rays the pixel kernel handed to the grazing-ray kernel, kTicket = how many of those
// the grazing-ray kernel's warps have drawn.
enum Counter { kSteps = 0, kHitPixels = 1, kSolidPixels = 2, kWalkErrors = 3, kDeferred = 4, kTicket = 5,
               kNumCounters = 8 };

struct StaticMaskKey {  // what the footprint of a solid that is never rotated depends on (all of it, bit for bit)
    int res_x, res_y;
    double x_min, y_min, step_x, step_y;
};

struct SolidSet {
    DevBuf<double> pts0;      // [n][4][3] pre-view frame
    DevBuf<double> pts_view;  // [n][4][3] view frame (rotated copy, or == pts0 content for static ones)
    DevBuf<uint32_t> faces;   // unique faces (4 * tet + k): a fan face shared by two tets is scanned once
    int64_t n = 0, n_faces = 0;
    double extent = 0.0;      // largest edge length of any solid tet (rotation invariant)
};

// Everything resident on ONE device.
struct DeviceState {
    int device = 0;
    cudaStream_t stream = nullptr;
    // A view's prologue and grazing-ray kernel run on `side`, of the device's greatest priority, forked from and
    // joined into the stream the view is enqueued on (enqueue_view); its pixel kernel runs on that stream. Their blocks
    // then take the SM slots that another lane's pixel kernel frees, instead of waiting for its last wave.
    cudaStream_t side = nullptr;
    cudaEvent_t ev_side = nullptr;   // the fork and join edges between the view's stream and `side`
    cudaEvent_t ev[8] = {};

    // mesh (uploaded once)
    int64_t n_pts = 0, n_tets = 0, n_bfaces = 0;
    double mesh_lo[3] = {0, 0, 0}, mesh_hi[3] = {0, 0, 0}; // bounding box in the file frame
    DevBuf<double> px, py, pz;       // Morton-ordered file-frame coordinates (SoA: the rotate kernel streams them)
    DevBuf<Conn> conn;               // per tet (Morton order): neighbours and apexes with their slot maps
    DevBuf<Fields> fields;           // per tet (Morton order): alpha and s
    DevBuf<double> q0;               // Q per tet (Morton order); fields[t].s is derived from it
    double cells_limit = 0.0;        // the alpha_limit fields[].s was last prepared for
    bool cells_limit_valid = false;
    DeviceState* origin = nullptr;   // sibling context: the device state that owns the mesh (and these two flags)
    uint64_t mesh_version = 0;       // bumped by every upload; a sibling re-aliases when it falls behind
    bool mesh_shared = false;        // some sibling aliases this state's arrays
    DevBuf<BFace> bfaces;            // Morton-sorted boundary faces (BVH leaves)
    DevBuf<BvhNode> nodes;           // n_bfaces - 1 internal nodes, BFS order (root = 0)
    DevBuf<int32_t> node_parent;     // per internal node: (parent << 1) | which child, -1 for the root
    DevBuf<int32_t> leaf_parent;     // per leaf: (parent << 1) | which child
    DevBuf<uint32_t> refit_flags;    // per internal node arrival counter
    std::vector<uint32_t> tperm;     // new -> old tet (host): places the file-order fields of c5_upload_channels
    DevBuf<uint32_t> tperm_dev;      // the same on the device, made at the first device-form gradient call
                                     // (siblings read their origin's)

    // channels (c5_upload_channels; aliased by siblings like the mesh)
    int n_channels = 0;
    DevBuf<double> ch_rec;           // [n_tets][channel_stride(n)]: {alpha_c, s_c} per channel, Morton order
    DevBuf<double> ch_q0;            // [n][n_tets]: Q per channel and tet (Morton order); s_c is derived from it
    double ch_limit = 0.0;           // the alpha_limit ch_rec's s_c were last prepared for
    bool ch_limit_valid = false;

    // solids
    SolidSet solid_follow, solid_static;

    // per view
    DevBuf<Vtx> vrot;
    DevBuf<double> xs, ys;
    int xs_res = 0, ys_res = 0;
    double xs_win[2] = {0, 0}, ys_win[2] = {0, 0};
    DevBuf<uint8_t> mask;
    DevBuf<uint32_t> mask_tall;      // solid mask: faces taller than a few rows, listed by the first pass
    DevBuf<unsigned> mask_counts;    // their number per solid set
    DevBuf<uint8_t> mask_tiles;      // "every pixel of this 16 x 8 tile is solid already"
    DevBuf<uint8_t> mask_static;     // whole-image mask of the solids that do not follow the view (cached)
    StaticMaskKey mask_static_key{}; // the pixel grid mask_static was scan-converted for
    bool mask_static_valid = false;  // reset by every upload / clear of solids
    DevBuf<double> out;              // band output, {tau, I} per pixel
    DevBuf<uint32_t> steps;
    DevBuf<unsigned long long> counters;
    DevBuf<unsigned long long> row_cost;
    DevBuf<uint16_t> ray_cost;       // [res_y][res_x] tet-steps of each pixel's ray in this state's last view, saturating
                                     // (0: a miss, a solid pixel, or unknown); the walk's pixel order is made from it
    int ray_cost_res[2] = {0, 0};    // the key ray_cost was written under: pixel grid, window and mesh version
    double ray_cost_win[4] = {0, 0, 0, 0};
    uint64_t ray_cost_mesh = 0;
    DevBuf<uint16_t> ray_order;      // per region of the walk's rectangle: its pixels in the order the walk takes them
    int ray_order_grid[3] = {0, 0, 0};    // of the last order: regions, regions per row, region side, and ...
    int ray_order_origin[2] = {0, 0};     // ... the rectangle's first pixel (c5_debug_ray_order_read)
    DevBuf<DeferredRay> queue;       // grazing rays of the current view (capacity: pixels of the band)
    DevBuf<double> ch_queue;         // their channel values {tau, I} (channel renders only)
    DevBuf<double> row_flux;         // flux renders: [res_y][pairs] {sum tau, sum I} of the band's rows
    DevBuf<double> grad_alpha, grad_q; // c5_render_grad: [n_tets] Morton order, this device's band only
    DevBuf<double> grad_in;          // c5_render_grad: the band's {g_tau, g_I} per pixel
    DevBuf<double> jvp_dir;          // c5_render_jvp: [n_tets][2] {v_alpha, v_q}, Morton order; made at this state's
                                     // first call, dropped by c5_upload_mesh (a sibling's when it follows a new mesh)
    int sm_count = 0;
    cudaEvent_t ev_walk = nullptr;   // between the pixel kernel and the grazing-ray kernel (phase times)
    cudaEvent_t ev_done = nullptr;   // after the view's last copy: what c5_render_wait waits for
    cudaEvent_t ev_fields = nullptr; // orders this stream and a caller's stream around the device-form gradient calls
    cudaEvent_t ev_gather = nullptr; // after the last c5_update_fields_device gather: a sibling made later waits on it
    // results of the view in flight, copied by the stream into pinned host memory
    unsigned long long* h_counters = nullptr;   // [kNumCounters]
    uint64_t* h_row_cost = nullptr;             // [h_row_cost_n]
    size_t h_row_cost_n = 0;
    double* h_row_flux = nullptr;               // [h_row_flux_n]: row_flux of a flux view
    size_t h_row_flux_n = 0;
    unsigned long long* h_view_counters = nullptr; // the light-curve device calls with stats: [view][kNumCounters]
    size_t h_view_counters_n = 0;
    // c5_debug_set (tests, diagnostics); 0 = default
    int opt_graze_list = 0, opt_query_budget = 0, opt_serial_list = 0, opt_mask_tile = 0;
    bool opt_no_zero_copy = false, opt_no_static_mask = false, opt_no_ray_order = false;
    // c5_debug_set("timeline", n): phase events of the last n views, read by c5_timeline_read
    std::vector<cudaEvent_t> tl_events;         // [n][kTimelinePhases]
    uint64_t tl_views = 0;                      // views recorded since the timeline was enabled

    uint64_t launches = 0;
};

struct MeshHost;

} // namespace c5

namespace c5 {
struct ViewPlan {      // a validated c5_view: trig evaluated, band and pixel steps resolved
    Rot rot[kMaxRot];
    int n_rot;
    int row_begin, row_end;
    double x_min, y_min, step_x, step_y;
};
struct FluxOut {       // the caller's arrays of a flux render (either may be null)
    double* rows;      // res_y * pairs * 2
    double* total;     // pairs * 2
};
struct PendingView {   // the view a context has in flight between c5_render_submit and c5_render_wait
    bool active = false;
    uint64_t ticket = 0;
    c5_view view{};
    ViewPlan plan{};
    bool d2h_copy = false; // the image went through the device band buffer and a copy (not stored in place)
    int flux_pairs = 0;    // flux view: pairs per row sum (0: an image view)
    FluxOut flux{};
};
} // namespace c5

struct c5_ctx {
    c5::DeviceState dev;             // siblings point DeviceState::origin at it: a context is never moved
    std::string err;
    bool has_mesh = false;
    c5_mesh_info info{};
    int64_t channel_bytes = 0;       // device bytes of the uploaded channels (included in info.device_bytes)
    std::vector<uint64_t> last_row_cost;
    std::vector<c5_ctx*> parts;      // multi-device context: one context per further device (owned)
    c5_ctx* parent = nullptr;        // sibling context (c5_create_sibling): shares parent's mesh and solids
    std::vector<c5_ctx*> siblings;   // contexts created from this one (the caller's, and our own lanes)
    std::vector<c5_ctx*> lanes;      // lanes of c5_render_submit beyond this context itself (owned; also in siblings)
    int views_in_flight = 3;
    uint64_t next_ticket = 1;
    unsigned next_lane = 0;
    c5::PendingView pending;         // this context's own view in flight
    std::vector<std::pair<void*, bool>> images;   // c5_image_create (true) / c5_image_open (false) pointers
    std::vector<std::pair<void*, void*>> image_offsets; // imported images: (pointer handed out, mapping base)
    std::vector<void*> registered;                // c5_host_register pointers
};

namespace c5 {

// c5_topology.cu — builds every mesh-resident array of `d` from host input.
void build_mesh(DeviceState& d, const double* pts, int64_t n_pts, const int32_t* tets, int64_t n_tets,
                const double* alpha, const double* q);

// c5_exact.cu — kernels whose arithmetic must match the reference's host code bit for bit
// (compiled with -fmad=false).
void launch_rotate_vertices(DeviceState& d, const Rot* rot, int n_rot);
void launch_rotate_solids(DeviceState& d, const Rot* rot, int n_rot);
void launch_solid_mask(DeviceState& d, int res_x, int res_y, double x_min, double y_min, double step_x,
                       double step_y, int row_begin, int row_end);
void launch_bvh_refit(DeviceState& d);
void dedupe_solid_faces(DeviceState& d, SolidSet& ss); // fills ss.faces / ss.n_faces from ss.pts0
// fields[t].s = q0[t] / min(alpha, limit), on d.stream, unless fields[] already hold that limit. A mesh shared with
// siblings is fenced by device-wide syncs around the launch, unless `fenced`: the caller has ordered every stream
// that reads the cells around d.stream with events.
void launch_prepare_cells(DeviceState& d, double alpha_limit, bool fenced = false);
void launch_prepare_channels(DeviceState& d, double alpha_limit, bool fenced = false); // the same for every channel of ch_rec

// c5_topology.cu — places n channels of file-order fields (channel-major) in ch_rec / ch_q0.
void upload_channels(DeviceState& d, const double* alpha, const double* q, int n);
// c5_topology.cu — replaces fields[].alpha and q0 by file-order fields (c5_update_fields).
void update_fields(DeviceState& d, const double* alpha, const double* q);
// c5_topology.cu — what the device forms (c5_update_fields_device, c5_render_grad_device) need.
// d.tperm_dev from d.tperm (allocates and blocks: made once, at the first device-form call)
void upload_tperm(DeviceState& d);
// The two ops below allocate nothing and launch one kernel on s.
// fields[t].alpha = alpha[tperm[t]], q0[t] = q[tperm[t]]: file-order device fields into d's tets
void gather_fields(DeviceState& d, const uint32_t* tperm, const double* alpha, const double* q, cudaStream_t s);
// dir[t] = {v_alpha[tperm[t]], v_q[tperm[t]]}, a null direction read as 0: c5_render_jvp's tangent field
void gather_direction(int64_t n_tets, const uint32_t* tperm, const double* v_alpha, const double* v_q, double* dir,
                      cudaStream_t s);
// out[tperm[t]] = in[t] for both gradients (a null output is skipped): Morton order back to file order
void scatter_grads(int64_t n_tets, const uint32_t* tperm, const double* in_alpha, const double* in_q, double* out_alpha,
                   double* out_q, cudaStream_t s);

// c5_walk.cu
struct WalkLaunch {
    int res_x, res_y, row_begin, row_end;
    int i_begin, i_end, j_begin, j_end; // pixel rectangle that can see the mesh (clipped to the band by the launch)
    double alpha_limit;
    int round_through_float;
    int use_mask;
    int write_steps;
    int precision;
    int channels; // 0: the cells' own fields; n: the n uploaded channels, n {tau, I} per pixel
    double* out; // {tau, I} per pixel (per channel) of the band, x fastest
    // the pixel kernel's stream, when it is not d.stream: the launch orders it after the prologue enqueued on
    // d.stream so far and orders d.stream's grazing-ray kernel after it, through d.ev_side (null: d.stream)
    cudaStream_t pixel_stream;
    cudaEvent_t mark_walk_done;    // recorded between the pixel kernel and the grazing-ray kernel (may be null)
    cudaEvent_t mark_walk_done_tl; // the same moment for the timeline ring (may be null)
    // c5_render_grad (channels 0, precision 64): kDepthPass stores {tau, I, lam, 0} per pixel into out;
    // kGradPass reads them (depth) and the band's {g_tau, g_I} (grad_in), adds into grad_alpha / grad_q,
    // stores no pixel and counts into its own counters / row_cost. grad_per_view: grad_in is the view's one
    // {g_tau, g_I}, the upstream of every pixel (c5_render_flux_grad_device)
    int pass;
    int grad_per_view;
    const double* depth;
    const double* grad_in;
    double* grad_alpha;
    double* grad_q;
    unsigned long long* counters;
    unsigned long long* row_cost;
    // c5_render_jvp (channels 0, precision 64): kJvpPass stores {tau, I, dtau, dI} per pixel into out, the
    // tangent along dir ([n_tets][2] {v_alpha, v_q}, Morton order)
    const double* dir;
};
enum WalkPass { kImagePass = 0, kDepthPass = 1, kGradPass = 2, kJvpPass = 3 };
void launch_walk(DeviceState& d, const WalkLaunch& w);
// c5_walk.cu — the pixel order of one region of the walk (c5_debug_ray_order): cost_rows[y][x] in, order[k] = the
// local Morton index of the k-th pixel and bucket[m] = the sort bucket of Morton index m out; returns the region side.
int order_one_region(const uint16_t* cost_rows, uint16_t* order, int32_t* bucket);
// c5_flux.cu — row_flux[j] for the rows [row_begin,row_end) of d.out (pairs {tau, I} per pixel),
// skipping pixels under d.mask when use_mask; the summation order is documented there.
void launch_reduce_rows(DeviceState& d, int res_x, int res_y, int row_begin, int row_end, int pairs, bool use_mask);
// c5_flux.cu — one launch: word c of the total of row_flux's rows [row_begin,row_end) (`words` doubles per row,
// summed in increasing j from 0) into lo[c] for c < split, hi[c - split] otherwise; a null destination is skipped.
void launch_total_rows(DeviceState& d, int row_begin, int row_end, int words, int split, double* lo, double* hi);
// doubles per tet of ch_rec: n {alpha, s} pairs padded to 32 bytes (read with 256-bit loads)
C5_HD constexpr int channel_stride(int n_channels) { return 4 * ((n_channels + 1) / 2); }

} // namespace c5
