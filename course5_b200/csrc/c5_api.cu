// c5_api.cu — the C ABI of include/c5gpu.h: context, mesh/solid upload, the per-view pipeline.
#include <cmath>
#include <cstring>
#include <algorithm>
#include <exception>
#include <mutex>
#include <thread>
#include <utility>
#include <vector>

#include <dlfcn.h>

#include "c5_internal.h"

using namespace c5;

namespace {

std::mutex g_create_err_mu;
std::string g_create_err;

const double kPi = 3.14159265358979323846; // config.hpp:45

template <class Fn>
int guarded(c5_ctx* ctx, Fn&& fn) {
    try {
        if (ctx) g_launch_counter = &ctx->dev.launches;
        fn();
        return C5_OK;
    } catch (const Error& e) {
        if (ctx) ctx->err = e.text;
        return e.code;
    } catch (const std::bad_alloc&) {
        if (ctx) ctx->err = "host allocation failed";
        return C5_E_NOMEM;
    } catch (const std::exception& e) {
        if (ctx) ctx->err = e.what();
        return C5_E_INVALID;
    }
}

void use_device(const DeviceState& d) {
    if (!kHostSim) C5_CUDA(cudaSetDevice(d.device));
}

// The context and, for a multi-device context, its parts: one context per device.
std::vector<c5_ctx*> with_parts(c5_ctx* ctx) {
    std::vector<c5_ctx*> all{ctx};
    all.insert(all.end(), ctx->parts.begin(), ctx->parts.end());
    return all;
}

// Phase events of the view being enqueued: 0 start, 1 rotated, 2 BVH refitted, 3 mask done,
// 4 walk done (pixel + grazing-ray kernel), 5 image copy starts, 6 image on the host;
// ev_walk sits between the two walk kernels.
void record(DeviceState& d, int k) {
    if (!kHostSim) C5_CUDA(cudaEventRecord(d.ev[k], d.stream));
}

// c5_debug_set("timeline", n): the same moments kept for the last n views (c5_timeline_read).
void timeline_mark(DeviceState& d, int phase) {
    if (kHostSim || d.tl_events.empty()) return;
    const size_t n = d.tl_events.size() / kTimelinePhases;
    C5_CUDA(cudaEventRecord(d.tl_events[(d.tl_views % n) * kTimelinePhases + static_cast<size_t>(phase)], d.stream));
}

float elapsed(DeviceState& d, int a, int b) {
    if (kHostSim) return 0.f;
    float ms = 0.f;
    C5_CUDA(cudaEventElapsedTime(&ms, d.ev[a], d.ev[b]));
    return ms;
}

ViewPlan plan_view(const c5_view* v) {
    if (!v) fail(C5_E_INVALID, "render: view is NULL");
    if (v->res_x < 2 || v->res_y < 2) fail(C5_E_INVALID, "render: resolution must be at least 2 x 2");
    if (static_cast<int64_t>(v->res_x) * v->res_y >= (int64_t{1} << 31)) fail(C5_E_INVALID, "render: image too large");
    if (v->n_rot < 0 || v->n_rot > kMaxRot) fail(C5_E_INVALID, "render: n_rot out of range");
    if (!(v->window[0] > v->window[1]) || !(v->window[2] > v->window[3])) {
        fail(C5_E_INVALID, "render: window must be {x_max, x_min, y_max, y_min} with max > min");
    }
    if (v->precision != 64 && v->precision != 32 && v->precision != 0) {
        fail(C5_E_INVALID, "render: precision must be 64 or 32");
    }
    ViewPlan p{};
    p.n_rot = v->n_rot;
    for (int k = 0; k < v->n_rot; k++) {
        if (v->rot[k].axis != 0 && v->rot[k].axis != 1) fail(C5_E_INVALID, "render: rotation axis must be 0 or 1");
        // the trig is evaluated here by the host libm, exactly like the reference's host loop
        p.rot[k] = Rot{v->rot[k].axis, 0, std::cos(v->rot[k].angle), std::sin(v->rot[k].angle), v->rot[k].x0};
    }
    p.row_begin = v->row_begin;
    p.row_end = v->row_end;
    if (p.row_begin == 0 && p.row_end == 0) p.row_end = v->res_y;
    if (p.row_begin < 0 || p.row_end > v->res_y || p.row_begin >= p.row_end) {
        fail(C5_E_INVALID, "render: bad row band");
    }
    p.x_min = v->window[1];
    p.y_min = v->window[3];
    p.step_x = (v->window[0] - v->window[1]) / (v->res_x - 1.); // plane.cpp:298-302
    p.step_y = (v->window[2] - v->window[3]) / (v->res_y - 1.);
    return p;
}

// Pixel coordinates by repeated addition (plane.cpp:304-314) — not x_min + i * step.
void ensure_pixel_tables(DeviceState& d, const c5_view* v, const ViewPlan& p) {
    if (d.xs_res != v->res_x || d.xs_win[0] != v->window[0] || d.xs_win[1] != v->window[1]) {
        std::vector<double> xs(static_cast<size_t>(v->res_x));
        double c = p.x_min;
        for (int i = 0; i < v->res_x; i++) {
            xs[static_cast<size_t>(i)] = c;
            c = c + p.step_x;
        }
        d.xs.alloc(xs.size());
        h2d(d.xs.p, xs.data(), d.xs.bytes(), d.stream);
        stream_sync(d.stream);
        d.xs_res = v->res_x;
        d.xs_win[0] = v->window[0];
        d.xs_win[1] = v->window[1];
    }
    if (d.ys_res != v->res_y || d.ys_win[0] != v->window[2] || d.ys_win[1] != v->window[3]) {
        std::vector<double> ys(static_cast<size_t>(v->res_y));
        double c = p.y_min;
        for (int j = 0; j < v->res_y; j++) {
            ys[static_cast<size_t>(j)] = c;
            c = c + p.step_y;
        }
        d.ys.alloc(ys.size());
        h2d(d.ys.p, ys.data(), d.ys.bytes(), d.stream);
        stream_sync(d.stream);
        d.ys_res = v->res_y;
        d.ys_win[0] = v->window[2];
        d.ys_win[1] = v->window[3];
    }
}

// Where on the screen the mesh can be: the view-frame box of the 8 corners of its file-frame box,
// widened by a pixel. The walk's grid covers only that rectangle (the rest of the band is filled as
// background); a conservative hint — inside it every tile is still tested against the BVH root.
void mesh_pixel_rect(const DeviceState& d, const c5_view* v, const ViewPlan& p, WalkLaunch& w) {
    double lo[2] = {INFINITY, INFINITY}, hi[2] = {-INFINITY, -INFINITY};
    for (int corner = 0; corner < 8; corner++) {
        double x = (corner & 1) ? d.mesh_hi[0] : d.mesh_lo[0];
        double y = (corner & 2) ? d.mesh_hi[1] : d.mesh_lo[1];
        double z = (corner & 4) ? d.mesh_hi[2] : d.mesh_lo[2];
        for (int k = 0; k < p.n_rot; k++) { // tetra.cpp:44-62
            const double c = p.rot[k].c, s = p.rot[k].s;
            if (p.rot[k].axis == 0) {
                const double y0 = y;
                y = y * c - z * s;
                z = y0 * s + z * c;
            } else {
                x -= p.rot[k].x0;
                const double x1 = x;
                x = x * c - z * s;
                z = x1 * s + z * c;
                x += p.rot[k].x0;
            }
        }
        lo[0] = std::min(lo[0], x);
        hi[0] = std::max(hi[0], x);
        lo[1] = std::min(lo[1], y);
        hi[1] = std::max(hi[1], y);
    }
    auto pixel = [](double c, double c_min, double step, int res, bool up) {
        double r = (c - c_min) / step + (up ? 2.0 : -2.0); // one pixel for rounding, one for the repeated-addition tables
        if (!(r > -1.0)) r = -1.0;
        if (!(r < res + 1.0)) r = res + 1.0;
        return static_cast<int>(up ? std::ceil(r) : std::floor(r));
    };
    w.i_begin = pixel(lo[0], p.x_min, p.step_x, v->res_x, false);
    w.i_end = pixel(hi[0], p.x_min, p.step_x, v->res_x, true) + 1;
    w.j_begin = pixel(lo[1], p.y_min, p.step_y, v->res_y, false);
    w.j_end = pixel(hi[1], p.y_min, p.step_y, v->res_y, true) + 1;
}

// The walk of view v's band: what every pass over its rays shares.
WalkLaunch view_walk(const DeviceState& d, const c5_view* v, const ViewPlan& p) {
    WalkLaunch w{};
    w.res_x = v->res_x;
    w.res_y = v->res_y;
    w.row_begin = p.row_begin;
    w.row_end = p.row_end;
    w.alpha_limit = v->alpha_limit;
    w.round_through_float = v->round_through_float;
    w.use_mask = v->use_solids && (d.solid_follow.n + d.solid_static.n) > 0 ? 1 : 0;
    w.precision = v->precision ? v->precision : 64;
    mesh_pixel_rect(d, v, p, w);
    return w;
}

// Enqueues one view's kernels for rows [row_begin,row_end) on device d. Events:
// 0 start, 1 rotated, 2 bvh, 3 mask, 4 walk.
// channels > 0: the walk integrates that many uploaded channels (c5_render_channels).
// pass = kDepthPass: the first pass of c5_render_grad ({tau, I, lam, 0} per pixel into d.out).
// pass = kJvpPass: c5_render_jvp ({tau, I, dtau, dI} per pixel into d.out, the tangent along dir).
void enqueue_view(DeviceState& d, const c5_view* v, const ViewPlan& p, bool want_steps, double* out_override = nullptr,
                  int channels = 0, int pass = kImagePass, const double* dir = nullptr) {
    use_device(d);
    g_launch_counter = &d.launches;
    ensure_pixel_tables(d, v, p);
    // Per-view buffers are sized for the WHOLE image, not the band: cost-balanced bands move from view to
    // view, and a buffer that had to grow in the middle of a sweep would cost a cudaFree (a device-wide
    // synchronisation) and a cudaMalloc on the spot.
    const size_t n_pix = static_cast<size_t>(v->res_y) * v->res_x;
    const bool solids = v->use_solids && (d.solid_follow.n + d.solid_static.n) > 0;
    const bool two_pairs = pass == kDepthPass || pass == kJvpPass;
    const size_t words = 2 * static_cast<size_t>(channels ? channels : two_pairs ? 2 : 1); // doubles per pixel
    if (!out_override) d.out.ensure(words * n_pix);
    if (want_steps) d.steps.ensure(n_pix);
    d.counters.ensure(kNumCounters);
    d.queue.ensure(n_pix); // every ray may be deferred (reserved, hardly ever touched)
    if (channels || two_pairs) d.ch_queue.ensure(words * n_pix);
    d.row_cost.ensure(static_cast<size_t>(v->res_y));
    if (solids) d.mask.ensure(n_pix);

    record(d, 0);
    timeline_mark(d, 0);
    launch_prepare_cells(d, v->alpha_limit); // no-op unless --alpha_limit changed since the last view
    if (channels) launch_prepare_channels(d, v->alpha_limit); // the same for the channels
    launch_rotate_vertices(d, p.rot, p.n_rot);
    if (solids) launch_rotate_solids(d, p.rot, p.n_rot);
    record(d, 1);
    timeline_mark(d, 1);
    launch_bvh_refit(d);
    record(d, 2);
    timeline_mark(d, 2);
    if (solids) {
        launch_solid_mask(d, v->res_x, v->res_y, p.x_min, p.y_min, p.step_x, p.step_y, p.row_begin, p.row_end);
    }
    record(d, 3);
    timeline_mark(d, 3);
    dev_zero(d.counters.p, kNumCounters * sizeof(unsigned long long), d.stream);
    dev_zero(d.row_cost.p, static_cast<size_t>(v->res_y) * sizeof(unsigned long long), d.stream);
    WalkLaunch w = view_walk(d, v, p);
    w.write_steps = want_steps ? 1 : 0;
    w.channels = channels;
    w.pass = pass;
    w.dir = dir;
    w.out = out_override ? out_override : d.out.p;
    w.mark_walk_done = d.ev_walk;
    w.mark_walk_done_tl = nullptr;
    if (!kHostSim && !d.tl_events.empty()) {
        const size_t n = d.tl_events.size() / kTimelinePhases;
        w.mark_walk_done_tl = d.tl_events[(d.tl_views % n) * kTimelinePhases + 4];
    }
    if (!kHostSim) { // a band the mesh does not reach launches no walk kernels: the markers are recorded anyway
        C5_CUDA(cudaEventRecord(d.ev_walk, d.stream));
        if (w.mark_walk_done_tl) C5_CUDA(cudaEventRecord(w.mark_walk_done_tl, d.stream));
    }
    launch_walk(d, w);
    record(d, 4);
    timeline_mark(d, 5);
    if (!d.tl_events.empty()) d.tl_views++;
}

// Contiguous row bands of [row_begin,row_end) with equal estimated cost (previous view's per-row
// tet-steps plus a constant per row), one per device; equal heights when there is no history.
std::vector<std::pair<int, int>> cut_bands(const c5_ctx* ctx, const c5_view* v, const ViewPlan& p, int n) {
    const int rows = p.row_end - p.row_begin;
    std::vector<double> cost(static_cast<size_t>(rows), 1.0);
    if (ctx->last_row_cost.size() == static_cast<size_t>(v->res_y)) {
        double total = 0;
        for (int j = 0; j < rows; j++) total += static_cast<double>(ctx->last_row_cost[static_cast<size_t>(p.row_begin + j)]);
        if (total > 0) {
            const double base = 64.0 + 0.02 * total / rows; // empty rows are not free (BVH miss, stores)
            for (int j = 0; j < rows; j++) {
                cost[static_cast<size_t>(j)] = base + static_cast<double>(ctx->last_row_cost[static_cast<size_t>(p.row_begin + j)]);
            }
        }
    }
    double total = 0;
    for (double c : cost) total += c;
    std::vector<std::pair<int, int>> bands;
    int lo = 0;
    double acc = 0;
    int j = 0;
    for (int b = 0; b < n; b++) {
        const double target = total * (b + 1) / n;
        while (j < rows && (acc + cost[static_cast<size_t>(j)] <= target || j == lo) && rows - (j + 1) >= n - b - 1) {
            acc += cost[static_cast<size_t>(j)];
            j++;
        }
        if (b == n - 1) j = rows;
        bands.emplace_back(p.row_begin + lo, p.row_begin + j);
        lo = j;
    }
    return bands;
}

// ---- one device: submit / wait -----------------------------------------------------------------------
// A view is enqueued on the context's stream together with the copies that bring its results to the
// host (image unless it is stored in place, counters, per-row costs -> page-locked staging), then an
// event; waiting for the view is waiting for that event. Nothing in between touches the host, so
// several contexts that share a mesh (the lanes of c5_render_submit) overlap on the device.

// flux_words: doubles of row sums a flux view copies back (res_y * pairs * 2; 0 for other views)
void ensure_host_staging(DeviceState& d, size_t rows, size_t flux_words = 0) {
    if (!d.h_counters) d.h_counters = static_cast<unsigned long long*>(host_pinned_alloc(kNumCounters * sizeof(unsigned long long)));
    if (rows > d.h_row_cost_n) {
        host_pinned_free(d.h_row_cost);
        d.h_row_cost = nullptr;
        d.h_row_cost_n = 0;
        d.h_row_cost = static_cast<uint64_t*>(host_pinned_alloc(rows * sizeof(uint64_t)));
        d.h_row_cost_n = rows;
    }
    if (flux_words > d.h_row_flux_n) {
        host_pinned_free(d.h_row_flux);
        d.h_row_flux = nullptr;
        d.h_row_flux_n = 0;
        d.h_row_flux = static_cast<double*>(host_pinned_alloc(flux_words * sizeof(double)));
        d.h_row_flux_n = flux_words;
    }
}

void follow_parent(c5_ctx* ctx);

// flux != null: a flux view. No image leaves the device: the band's rows are summed (launch_reduce_rows)
// and the sums are copied into page-locked staging; c5_render_wait / the caller hands them to `flux`.
void submit_view(c5_ctx* ctx, const c5_view* v, double* out, uint32_t* steps, uint8_t* solid_mask, uint64_t ticket,
                 bool in_place_allowed = true, bool channels = false, const FluxOut* flux = nullptr) {
    follow_parent(ctx);
    if (ctx->pending.active) fail(C5_E_STATE, "render: this context still has a view in flight (c5_render_wait it first)");
    if (!ctx->has_mesh) fail(C5_E_STATE, "render: no mesh uploaded");
    if (!out && !flux) fail(C5_E_INVALID, "render: out is NULL");
    const ViewPlan p = plan_view(v);
    DeviceState& d = ctx->dev;
    if (channels && d.n_channels == 0) fail(C5_E_STATE, "render_channels: no channels uploaded");
    const int n_ch = channels ? d.n_channels : 0;
    const size_t words = 2 * static_cast<size_t>(channels ? n_ch : 1); // doubles per pixel of `out`
    use_device(d);
    const size_t n_pix_band = static_cast<size_t>(p.row_end - p.row_begin) * v->res_x;
    const size_t band_off = static_cast<size_t>(p.row_begin) * v->res_x;
    // A PAGE-LOCKED host buffer is device-addressable: the walk can store its pixels straight into it
    // (posted 128-byte writes over PCIe, spread over the kernel's run time) and the separate
    // device-to-host copy of the image disappears. That is the shorter path for ONE view at a time
    // (c5_render). With several views in flight the copy engine is the better one: it moves view k's
    // image while the SMs walk view k+1, and the walk kernels are not held up by PCIe write
    // back-pressure (C3, 4 views in flight: 4.76 ms per view against 5.53 in place and 4.59 with no host
    // image at all; profiles/r02_bench_c3_n1_e2e_*.json) — so c5_render_submit passes
    // in_place_allowed = false. Pixels are stored as one 128-bit word, so an in-place buffer must be
    // 16-byte aligned; pageable or misaligned buffers take the copy.
    double* host_direct = nullptr;
    if (!kHostSim && !flux && in_place_allowed && !d.opt_no_zero_copy && (reinterpret_cast<uintptr_t>(out) & 15u) == 0) {
        cudaPointerAttributes attr{};
        if (cudaPointerGetAttributes(&attr, out) == cudaSuccess && attr.type == cudaMemoryTypeHost && attr.devicePointer) {
            host_direct = static_cast<double*>(attr.devicePointer) + words * band_off;
        } else {
            cudaGetLastError(); // pageable memory reports an error on some drivers: not ours
        }
    }
    ensure_host_staging(d, static_cast<size_t>(v->res_y), flux ? words * static_cast<size_t>(v->res_y) : 0);
    enqueue_view(d, v, p, steps != nullptr, host_direct, n_ch);
    const bool solids = v->use_solids && (d.solid_follow.n + d.solid_static.n) > 0;
    record(d, 5);
    if (flux) { // after the grazing-ray kernel: deferred rays are in the sums
        launch_reduce_rows(d, v->res_x, v->res_y, p.row_begin, p.row_end, static_cast<int>(words / 2), solids);
        const size_t rows_off = words * static_cast<size_t>(p.row_begin);
        d2h(d.h_row_flux + rows_off, d.row_flux.p + rows_off, words * static_cast<size_t>(p.row_end - p.row_begin) * sizeof(double),
            d.stream);
    } else if (!host_direct) {
        d2h(out + words * band_off, d.out.p, words * n_pix_band * sizeof(double), d.stream);
    }
    record(d, 6);
    if (steps) d2h(steps + band_off, d.steps.p, n_pix_band * sizeof(uint32_t), d.stream);
    if (solid_mask) {
        if (solids) d2h(solid_mask + band_off, d.mask.p + band_off, n_pix_band, d.stream);
        else std::memset(solid_mask + band_off, 0, n_pix_band);
    }
    d2h(d.h_counters, d.counters.p, kNumCounters * sizeof(unsigned long long), d.stream);
    d2h(d.h_row_cost, d.row_cost.p, static_cast<size_t>(v->res_y) * sizeof(uint64_t), d.stream);
    if (!kHostSim) C5_CUDA(cudaEventRecord(d.ev_done, d.stream));
    ctx->pending.active = true;
    ctx->pending.ticket = ticket;
    ctx->pending.view = *v;
    ctx->pending.plan = p;
    ctx->pending.d2h_copy = host_direct == nullptr;
    ctx->pending.flux_pairs = flux ? static_cast<int>(words / 2) : 0;
    ctx->pending.flux = flux ? *flux : FluxOut{};
}

// What one device reports for a view: its stats and per-row tet-steps.
struct ViewResult {
    c5_stats st{};
    std::vector<uint64_t> row_cost;
    std::vector<double> flux; // flux views: res_y * pairs * 2 row sums, 0 outside the band
};

// Reads d's last view (planned as p) from the page-locked staging, once the stream has passed the
// copies into it. A submitted view ends with the image on the host (event 6); a view of
// c5_render_device ends with the walk (event 4) and has no ms_d2h. A flux view (flux_pairs > 0) ends
// with its row sums on the host (event 6).
ViewResult read_view(DeviceState& d, const c5_view& v, const ViewPlan& p, bool submitted, int flux_pairs = 0) {
    ViewResult r;
    c5_stats& st = r.st;
    const unsigned long long* c = d.h_counters;
    st.pixels = static_cast<uint64_t>(p.row_end - p.row_begin) * static_cast<uint64_t>(v.res_x);
    st.tet_steps = c[kSteps];
    st.hit_pixels = c[kHitPixels];
    st.solid_pixels = c[kSolidPixels];
    st.walk_errors = c[kWalkErrors];
    st.grazing_rays = static_cast<int32_t>(c[kDeferred]);
    st.ms_rotate = elapsed(d, 0, 1);
    st.ms_bvh = elapsed(d, 1, 2);
    st.ms_mask = elapsed(d, 2, 3);
    st.ms_walk = elapsed(d, 3, 4);
    if (!kHostSim) C5_CUDA(cudaEventElapsedTime(&st.ms_graze, d.ev_walk, d.ev[4]));
    if (submitted) st.ms_d2h = elapsed(d, 5, 6);
    st.ms_total = elapsed(d, 0, submitted ? 6 : 4);
    st.n_devices = 1;
    r.row_cost.assign(d.h_row_cost, d.h_row_cost + v.res_y);
    if (flux_pairs) {
        const size_t words = 2 * static_cast<size_t>(flux_pairs);
        r.flux.assign(words * static_cast<size_t>(v.res_y), 0.0);
        std::copy(d.h_row_flux + words * static_cast<size_t>(p.row_begin), d.h_row_flux + words * static_cast<size_t>(p.row_end),
                  r.flux.begin() + static_cast<std::ptrdiff_t>(words * static_cast<size_t>(p.row_begin)));
    }
    return r;
}

// Hands a flux view's row sums (res_y rows of `words` doubles) to the caller: the rows as they are,
// total[c] = sum of rows[j][c] in increasing j, accumulated in double.
void deliver_flux(const std::vector<double>& rows, size_t words, const FluxOut& f) {
    if (f.rows) std::copy(rows.begin(), rows.end(), f.rows);
    if (!f.total) return;
    for (size_t c = 0; c < words; c++) f.total[c] = 0.0;
    for (size_t j = 0; j < rows.size() / words; j++) {
        for (size_t c = 0; c < words; c++) f.total[c] += rows[j * words + c];
    }
}

// Row costs go to `owner` (the context the caller holds), stats to *st (may be NULL); a ray stopped
// by the step cap is C5_E_WALK.
void report(c5_ctx* owner, ViewResult& r, c5_stats* st) {
    owner->last_row_cost = std::move(r.row_cost);
    if (st) *st = r.st;
    if (r.st.walk_errors) {
        fail(C5_E_WALK, "render: " + std::to_string(r.st.walk_errors) + " ray(s) exceeded the step cap");
    }
}

// Waits for the view `lane` has in flight and reads it.
ViewResult wait_view(c5_ctx* lane) {
    if (!lane->pending.active) fail(C5_E_STATE, "render_wait: no view in flight");
    DeviceState& d = lane->dev;
    use_device(d);
    lane->pending.active = false; // whatever happens below, the lane is free again
    if (!kHostSim) C5_CUDA(cudaEventSynchronize(d.ev_done));
    return read_view(d, lane->pending.view, lane->pending.plan, true, lane->pending.flux_pairs);
}

// The stats of one view rendered as bands by several devices: counters and row costs add up, phase
// times are the slowest device's.
ViewResult merge_results(const std::vector<ViewResult>& results, int res_y) {
    ViewResult total;
    c5_stats& t = total.st;
    total.row_cost.assign(static_cast<size_t>(res_y), 0);
    for (const ViewResult& r : results) {
        const c5_stats& s = r.st;
        t.pixels += s.pixels;
        t.tet_steps += s.tet_steps;
        t.hit_pixels += s.hit_pixels;
        t.solid_pixels += s.solid_pixels;
        t.walk_errors += s.walk_errors;
        t.grazing_rays += s.grazing_rays;
        t.ms_rotate = std::max(t.ms_rotate, s.ms_rotate);
        t.ms_bvh = std::max(t.ms_bvh, s.ms_bvh);
        t.ms_mask = std::max(t.ms_mask, s.ms_mask);
        t.ms_walk = std::max(t.ms_walk, s.ms_walk);
        t.ms_graze = std::max(t.ms_graze, s.ms_graze);
        t.ms_d2h = std::max(t.ms_d2h, s.ms_d2h);
        t.ms_total = std::max(t.ms_total, s.ms_total);
        for (size_t j = 0; j < total.row_cost.size(); j++) total.row_cost[j] += r.row_cost[j];
    }
    t.n_devices = static_cast<int32_t>(results.size());
    return total;
}

// Multi-device contexts (c5_create with several devices): the context and each of its parts render
// one cost-balanced row band, as c5_render does for a row band, straight into its final rows of the
// caller's buffers. One host thread per device submits: a copy into pageable memory blocks the
// submitting thread until its device is done, so one thread would render the bands one after another.
// A flux render (flux != null) merges the parts' row sums and sums the total over all rows in order.
void render_multi_device(c5_ctx* ctx, const c5_view* v, double* out, uint32_t* steps, uint8_t* solid_mask, c5_stats* st,
                         bool channels = false, const FluxOut* flux = nullptr) {
    if (!ctx->has_mesh) fail(C5_E_STATE, "render: no mesh uploaded");
    const ViewPlan p = plan_view(v);
    const std::vector<c5_ctx*> parts = with_parts(ctx);
    const size_t n = parts.size();
    if (static_cast<size_t>(p.row_end - p.row_begin) < n) fail(C5_E_INVALID, "render: fewer rows than devices");
    const auto bands = cut_bands(ctx, v, p, static_cast<int>(n));
    std::vector<c5_view> band_views(n, *v);
    std::vector<std::exception_ptr> errors(n);
    auto submit = [&](size_t r) {
        try {
            band_views[r].row_begin = bands[r].first;
            band_views[r].row_end = bands[r].second;
            const FluxOut part_flux{}; // the merged sums are handed over below
            submit_view(parts[r], &band_views[r], out, steps, solid_mask, 0, true, channels, flux ? &part_flux : nullptr);
        } catch (...) {
            errors[r] = std::current_exception();
        }
    };
    if (kHostSim) {
        for (size_t r = 0; r < n; r++) submit(r);
    } else {
        std::vector<std::thread> workers;
        for (size_t r = 0; r < n; r++) workers.emplace_back(submit, r);
        for (auto& w : workers) w.join();
    }
    // every band that was submitted is waited for, also when another failed: none may still be
    // writing into the caller's buffers once this returns
    std::vector<ViewResult> results(n);
    for (size_t r = 0; r < n; r++) {
        if (!parts[r]->pending.active) continue;
        try {
            results[r] = wait_view(parts[r]);
        } catch (...) {
            if (!errors[r]) errors[r] = std::current_exception();
        }
    }
    for (auto& e : errors) {
        if (e) std::rethrow_exception(e);
    }
    ViewResult total = merge_results(results, v->res_y);
    if (flux) {
        const size_t words = results[0].flux.size() / static_cast<size_t>(v->res_y);
        std::vector<double> rows(words * static_cast<size_t>(v->res_y), 0.0);
        for (size_t r = 0; r < n; r++) {
            const size_t lo = words * static_cast<size_t>(bands[r].first), hi = words * static_cast<size_t>(bands[r].second);
            std::copy(results[r].flux.begin() + static_cast<std::ptrdiff_t>(lo), results[r].flux.begin() + static_cast<std::ptrdiff_t>(hi),
                      rows.begin() + static_cast<std::ptrdiff_t>(lo));
        }
        deliver_flux(rows, words, *flux);
    }
    report(ctx, total, st);
}

// ---- gradients (c5_render_grad) ------------------------------------------------------------------------

// What one device returns for its band of a gradient render: the depth pass's stats and the band's
// gradients, in the file order of the tets.
struct GradResult {
    ViewResult view;
    std::vector<double> grad_alpha, grad_q; // empty unless asked for
};

// The depth pass (with the view prologue, enqueue_view) and the gradient pass of band [row_begin,row_end)
// of v on d.stream, into d.grad_alpha / d.grad_q (Morton order), zeroed first. The band's {g_tau, g_I} per
// pixel are g_host's rows (the whole image, copied to d.grad_in) or d_g (a device band buffer, read in
// place); with g_per_view, d_g is the view's one {g_tau, g_I}. acc != null: the pass adds into acc's
// accumulators instead, which the caller has zeroed (the views of c5_render_flux_grad_device).
// Events: 0..4 as for an image, 5 depth pass done.
void enqueue_grad(DeviceState& d, const c5_view* v, const ViewPlan& p, const double* g_host, const double* d_g,
                  DeviceState* acc = nullptr, bool g_per_view = false) {
    const size_t n_t = static_cast<size_t>(d.n_tets);
    const size_t n_pix_band = static_cast<size_t>(p.row_end - p.row_begin) * v->res_x;
    const size_t band_off = static_cast<size_t>(p.row_begin) * v->res_x;
    // the gradient pass counts into the second half, so that the stats stay the depth pass's
    d.counters.ensure(2 * kNumCounters);
    d.row_cost.ensure(2 * static_cast<size_t>(v->res_y));
    if (!acc) {
        d.grad_alpha.ensure(n_t);
        d.grad_q.ensure(n_t);
    }
    if (g_host) d.grad_in.ensure(2 * static_cast<size_t>(v->res_y) * v->res_x);
    enqueue_view(d, v, p, false, nullptr, 0, kDepthPass);
    record(d, 5);
    if (!acc) {
        dev_zero(d.grad_alpha.p, n_t * sizeof(double), d.stream);
        dev_zero(d.grad_q.p, n_t * sizeof(double), d.stream);
    }
    dev_zero(d.counters.p + kNumCounters, kNumCounters * sizeof(unsigned long long), d.stream);
    dev_zero(d.row_cost.p + v->res_y, static_cast<size_t>(v->res_y) * sizeof(unsigned long long), d.stream);
    if (g_host) h2d(d.grad_in.p, g_host + 2 * band_off, 2 * n_pix_band * sizeof(double), d.stream);
    WalkLaunch w = view_walk(d, v, p);
    w.pass = kGradPass;
    w.depth = d.out.p;
    w.grad_in = g_host ? d.grad_in.p : d_g; // indexed like the band's out, or the view's one pair
    w.grad_per_view = g_per_view ? 1 : 0;
    w.grad_alpha = (acc ? *acc : d).grad_alpha.p;
    w.grad_q = (acc ? *acc : d).grad_q.p;
    w.counters = d.counters.p + kNumCounters;
    w.row_cost = d.row_cost.p + v->res_y;
    launch_walk(d, w);
}

// Band [row_begin,row_end) of v on ctx's device: enqueue_grad, then the copies. Blocks until the results
// are on the host. Events: 0..5 as for enqueue_grad, 6 gradients on the host.
GradResult grad_band(c5_ctx* ctx, const c5_view* v, const double* g, bool want_alpha, bool want_q, double* out) {
    follow_parent(ctx);
    if (ctx->pending.active) fail(C5_E_STATE, "render_grad: this context still has a view in flight (c5_render_wait it first)");
    if (!ctx->has_mesh) fail(C5_E_STATE, "render: no mesh uploaded");
    const ViewPlan p = plan_view(v);
    DeviceState& d = ctx->dev;
    use_device(d);
    const size_t n_t = static_cast<size_t>(d.n_tets);
    const size_t n_pix_band = static_cast<size_t>(p.row_end - p.row_begin) * v->res_x;
    const size_t band_off = static_cast<size_t>(p.row_begin) * v->res_x;
    ensure_host_staging(d, static_cast<size_t>(v->res_y));
    enqueue_grad(d, v, p, g, nullptr);
    std::vector<double> morton[2];
    for (int k = 0; k < 2; k++) {
        if (!(k == 0 ? want_alpha : want_q)) continue;
        morton[k].resize(n_t);
        d2h(morton[k].data(), (k == 0 ? d.grad_alpha : d.grad_q).p, n_t * sizeof(double), d.stream);
    }
    record(d, 6);
    d2h(d.h_counters, d.counters.p, kNumCounters * sizeof(unsigned long long), d.stream);
    d2h(d.h_row_cost, d.row_cost.p, static_cast<size_t>(v->res_y) * sizeof(uint64_t), d.stream);
    std::vector<double> band(out ? 4 * n_pix_band : 0); // the depth pass's {tau, I, lam, 0} per pixel
    if (out) d2h(band.data(), d.out.p, band.size() * sizeof(double), d.stream);
    stream_sync(d.stream);
    for (size_t k = 0; k < band.size() / 4; k++) { // its first pair is the image of c5_render_raw
        out[2 * (band_off + k)] = band[4 * k];
        out[2 * (band_off + k) + 1] = band[4 * k + 1];
    }
    GradResult r;
    const std::vector<uint32_t>& tperm = (d.origin ? *d.origin : d).tperm; // new -> old tet
    for (int k = 0; k < 2; k++) {
        if (morton[k].empty()) continue;
        std::vector<double>& file = k == 0 ? r.grad_alpha : r.grad_q;
        file.resize(n_t);
        for (size_t t = 0; t < n_t; t++) file[tperm[t]] = morton[k][t];
    }
    r.view = read_view(d, *v, p, true);
    return r;
}

// The lanes of c5_render_submit: lane 0 is the context itself, the others are sibling contexts the
// library makes (and owns) on first use.
c5_ctx* lane_of(c5_ctx* ctx, unsigned k) {
    return k == 0 ? ctx : ctx->lanes[k - 1];
}

void ensure_lanes(c5_ctx* ctx) {
    while (static_cast<int>(ctx->lanes.size()) + 1 < ctx->views_in_flight) {
        c5_ctx* lane = nullptr;
        const int rc = c5_create_sibling(ctx, &lane);
        if (rc != C5_OK) fail(rc, "render_submit: cannot create a lane: " + ctx->err);
        ctx->lanes.push_back(lane);
    }
}

// c5_render_submit / c5_render_flux_submit: the view goes to the next lane in turn, or any free one.
void submit_on_lane(c5_ctx* ctx, const c5_view* view, double* out, uint64_t* ticket, bool channels, const FluxOut* flux) {
    ensure_lanes(ctx);
    const unsigned n = static_cast<unsigned>(ctx->lanes.size()) + 1;
    c5_ctx* lane = nullptr;
    for (unsigned k = 0; k < n && !lane; k++) {
        c5_ctx* cand = lane_of(ctx, (ctx->next_lane + k) % n);
        if (!cand->pending.active) {
            lane = cand;
            ctx->next_lane = (ctx->next_lane + k + 1) % n;
        }
    }
    if (!lane) fail(C5_E_STATE, "render_submit: " + std::to_string(n) + " views are in flight already (c5_render_wait one first)");
    const uint64_t t = ctx->next_ticket++;
    try {
        g_launch_counter = &lane->dev.launches;
        submit_view(lane, view, out, nullptr, nullptr, t, /*in_place_allowed=*/ctx->views_in_flight == 1, channels, flux);
    } catch (const Error& e) {
        if (lane != ctx) ctx->err = e.text; // (guarded() reports through ctx)
        throw;
    }
    *ticket = t;
}

// A render over the uploaded channels needs them on the context and, alike, on every part.
void check_channels_ready(c5_ctx* ctx) {
    follow_parent(ctx);
    if (!ctx->has_mesh) fail(C5_E_STATE, "render: no mesh uploaded");
    if (ctx->dev.n_channels == 0) fail(C5_E_STATE, "render_channels: no channels uploaded");
    for (const c5_ctx* part : ctx->parts) { // every band must be as wide as the caller's image
        if (part->dev.n_channels != ctx->dev.n_channels) fail(C5_E_STATE, "render_channels: the devices hold different channels");
    }
}

// Arguments of c5_render_flux / c5_render_flux_submit.
void check_flux_args(const c5_view* view, int32_t channels, const double* rows, const double* total) {
    if (!rows && !total) fail(C5_E_INVALID, "render_flux: rows and total are both NULL");
    if (channels != 0 && channels != 1) fail(C5_E_INVALID, "render_flux: channels must be 0 or 1");
    if (channels && view && view->precision == 32) fail(C5_E_INVALID, "render_flux: channels are FP64 only (precision 64)");
}

// ---- gradients on device memory (c5_update_fields_device, c5_render_grad_device) ------------------------

void check_device_array(const void* p, const char* what) {
    if (!p) fail(C5_E_INVALID, std::string(what) + " is NULL");
    if (reinterpret_cast<uintptr_t>(p) & 7u) fail(C5_E_INVALID, std::string(what) + " must be 8-byte aligned");
}

// The device copy of the tet permutation, on the state that owns the mesh: made by the first device-form
// call (not at upload, so that contexts that never use it do not pay its 4 bytes per tet) and counted in
// device_bytes from then on.
const uint32_t* resident_tperm(c5_ctx* ctx) {
    c5_ctx* owner = ctx->parent ? ctx->parent : ctx;
    DeviceState& o = owner->dev;
    if (!o.tperm_dev.p) {
        use_device(o);
        upload_tperm(o);
        owner->info.device_bytes += static_cast<int64_t>(o.tperm_dev.bytes());
        if (owner != ctx) ctx->info = owner->info;
    }
    return o.tperm_dev.p;
}

// The context's own stream and those of its lanes and siblings: the streams the library renders on.
std::vector<DeviceState*> internal_streams(c5_ctx* ctx) {
    std::vector<DeviceState*> all{&ctx->dev};
    for (c5_ctx* s : ctx->siblings) all.push_back(&s->dev); // the caller's siblings and our lanes
    return all;
}

// c5_render_grad_device on a single-device context or a sibling: enqueue_grad on the caller's stream with
// d_g read in place, then the scatter into file order and the strided copy of the image.
void grad_band_device(c5_ctx* ctx, const c5_view* v, const double* d_g, double* d_grad_alpha, double* d_grad_q,
                      double* d_out, void* stream, c5_stats* stats) {
    follow_parent(ctx);
    if (!ctx->has_mesh) fail(C5_E_STATE, "render: no mesh uploaded");
    if (ctx->pending.active) fail(C5_E_STATE, "render_grad_device: this context has a submitted view in flight");
    const ViewPlan p = plan_view(v);
    DeviceState& d = ctx->dev;
    use_device(d);
    const uint32_t* tperm = resident_tperm(ctx);
    const size_t n_pix_band = static_cast<size_t>(p.row_end - p.row_begin) * v->res_x;
    if (stats) ensure_host_staging(d, static_cast<size_t>(v->res_y));
    // run on the CALLER's stream, like c5_render_device: the scratch arrays are the context's own
    cudaStream_t own = d.stream;
    if (!kHostSim) d.stream = static_cast<cudaStream_t>(stream);
    try {
        enqueue_grad(d, v, p, nullptr, d_g);
        scatter_grads(d.n_tets, tperm, d.grad_alpha.p, d.grad_q.p, d_grad_alpha, d_grad_q, d.stream);
        // the depth pass left {tau, I, lam, 0} per pixel: its first pair is the image of c5_render_raw
        if (d_out) d2d_2d(d_out, 2 * sizeof(double), d.out.p, 4 * sizeof(double), 2 * sizeof(double), n_pix_band, d.stream);
        record(d, 6);
        if (!kHostSim && d.stream != own) { // the context's own later renders reuse these scratch arrays: they wait
            C5_CUDA(cudaEventRecord(d.ev_fields, d.stream));
            C5_CUDA(cudaStreamWaitEvent(own, d.ev_fields, 0));
        }
        if (stats) {
            d2h(d.h_counters, d.counters.p, kNumCounters * sizeof(unsigned long long), d.stream);
            d2h(d.h_row_cost, d.row_cost.p, static_cast<size_t>(v->res_y) * sizeof(uint64_t), d.stream);
            stream_sync(d.stream);
            ViewResult r = read_view(d, *v, p, true);
            report(ctx, r, stats);
        }
    } catch (...) {
        d.stream = own;
        throw;
    }
    d.stream = own;
}

// Two timing events for the span of a call on a caller's stream (created only when stats are asked for).
struct SpanEvents {
    cudaEvent_t e[2] = {};
    ~SpanEvents() {
        for (cudaEvent_t x : e) {
            if (x) cudaEventDestroy(x);
        }
    }
};

// Page-locked room for the counters of n_views views, copied there one view at a time by the calls over the lanes.
void ensure_view_counters(DeviceState& o, int32_t n_views) {
    const size_t n = static_cast<size_t>(n_views) * kNumCounters;
    if (n <= o.h_view_counters_n) return;
    host_pinned_free(o.h_view_counters);
    o.h_view_counters = nullptr;
    o.h_view_counters_n = 0;
    o.h_view_counters = static_cast<unsigned long long*>(host_pinned_alloc(n * sizeof(unsigned long long)));
    o.h_view_counters_n = n;
}

// The stats of a call over the lanes, once `s` has waited for every lane: the views' counters summed (each view's
// in o.h_view_counters), ms_total the call's span on s (span.e[0] recorded at its start), the other times 0.
void report_views(DeviceState& o, const c5_view* views, const std::vector<ViewPlan>& plans, cudaStream_t s,
                  const SpanEvents& span, c5_stats* stats) {
    if (!kHostSim) C5_CUDA(cudaEventRecord(span.e[1], s));
    stream_sync(s);
    c5_stats st{};
    for (size_t k = 0; k < plans.size(); k++) {
        const unsigned long long* c = o.h_view_counters + k * kNumCounters;
        const ViewPlan& p = plans[k];
        st.pixels += static_cast<uint64_t>(p.row_end - p.row_begin) * static_cast<uint64_t>(views[k].res_x);
        st.tet_steps += c[kSteps];
        st.hit_pixels += c[kHitPixels];
        st.solid_pixels += c[kSolidPixels];
        st.walk_errors += c[kWalkErrors];
        st.grazing_rays += static_cast<int32_t>(c[kDeferred]);
    }
    if (!kHostSim) C5_CUDA(cudaEventElapsedTime(&st.ms_total, span.e[0], span.e[1]));
    st.n_devices = 1;
    *stats = st;
    if (st.walk_errors) fail(C5_E_WALK, "render: " + std::to_string(st.walk_errors) + " ray(s) exceeded the step cap");
}

// c5_render_flux_grad_device: view k goes to lane k % views_in_flight, where the depth and the gradient pass
// run on the lane's own stream with the view's one upstream pair d_g[2k..2k+1], all adding into the owner's
// Morton-order accumulators; one scatter into file order on the caller's stream at the end.
void flux_grad_device(c5_ctx* ctx, const c5_view* views, int32_t n_views, const double* d_g, double* d_grad_alpha,
                      double* d_grad_q, void* stream, c5_stats* stats) {
    if (ctx->parent) fail(C5_E_STATE, "render_flux_grad_device: a sibling context; call through its parent");
    if (!ctx->has_mesh) fail(C5_E_STATE, "render: no mesh uploaded");
    for (unsigned k = 0; k <= ctx->lanes.size(); k++) {
        if (lane_of(ctx, k)->pending.active) fail(C5_E_STATE, "render_flux_grad_device: a submitted view is in flight");
    }
    std::vector<ViewPlan> plans;
    for (int32_t k = 0; k < n_views; k++) plans.push_back(plan_view(&views[k]));
    ensure_lanes(ctx);
    const unsigned n_lanes = static_cast<unsigned>(ctx->lanes.size()) + 1;
    for (unsigned k = 0; k < n_lanes; k++) follow_parent(lane_of(ctx, k));
    DeviceState& o = ctx->dev;
    use_device(o);
    const uint32_t* tperm = resident_tperm(ctx);
    const size_t n_t = static_cast<size_t>(o.n_tets);
    o.grad_alpha.ensure(n_t);
    o.grad_q.ensure(n_t);
    if (stats) ensure_view_counters(o, n_views);
    cudaStream_t s = kHostSim ? o.stream : static_cast<cudaStream_t>(stream);
    SpanEvents span;
    if (stats && !kHostSim) {
        for (cudaEvent_t& e : span.e) C5_CUDA(cudaEventCreate(&e));
        C5_CUDA(cudaEventRecord(span.e[0], s));
    }
    // 1. the accumulators are zeroed on `stream` once the context's own stream is done with them (an earlier
    // call's scatter, a host-form gradient), 2. every lane starts after that (and so after the caller's
    // earlier work on `stream`, such as a field update or whatever wrote d_g)
    if (!kHostSim) {
        C5_CUDA(cudaEventRecord(o.ev_fields, o.stream));
        C5_CUDA(cudaStreamWaitEvent(s, o.ev_fields, 0));
    }
    dev_zero(o.grad_alpha.p, n_t * sizeof(double), s);
    dev_zero(o.grad_q.p, n_t * sizeof(double), s);
    if (!kHostSim) {
        C5_CUDA(cudaEventRecord(o.ev_fields, s));
        for (unsigned k = 0; k < n_lanes; k++) C5_CUDA(cudaStreamWaitEvent(lane_of(ctx, k)->dev.stream, o.ev_fields, 0));
    }
    for (int32_t k = 0; k < n_views; k++) {
        DeviceState& d = lane_of(ctx, static_cast<unsigned>(k) % n_lanes)->dev;
        enqueue_grad(d, &views[k], plans[static_cast<size_t>(k)], nullptr, d_g + 2 * static_cast<size_t>(k), &o, true);
        if (stats) d2h(o.h_view_counters + static_cast<size_t>(k) * kNumCounters, d.counters.p,
                       kNumCounters * sizeof(unsigned long long), d.stream);
    }
    // 3. `stream` waits for every lane, then scatters
    if (!kHostSim) {
        for (unsigned k = 0; k < n_lanes; k++) {
            DeviceState& d = lane_of(ctx, k)->dev;
            C5_CUDA(cudaEventRecord(d.ev_fields, d.stream));
            C5_CUDA(cudaStreamWaitEvent(s, d.ev_fields, 0));
        }
    }
    g_launch_counter = &o.launches;
    scatter_grads(o.n_tets, tperm, o.grad_alpha.p, o.grad_q.p, d_grad_alpha, d_grad_q, s);
    // 4. the context's own later renders (and the next call's zeroing) wait for the scatter
    if (!kHostSim) {
        C5_CUDA(cudaEventRecord(o.ev_fields, s));
        C5_CUDA(cudaStreamWaitEvent(o.stream, o.ev_fields, 0));
    }
    if (stats) report_views(o, views, plans, s, span, stats);
}

// ---- forward mode (c5_render_jvp, c5_render_jvp_device) -------------------------------------------------

// The tangent field of ctx's own device state, [n_tets][2] {v_alpha, v_q} in Morton order: made at the state's
// first call and reused by every later one. The context that owns the mesh counts it in device_bytes from then on
// (a sibling's, like its other per-view arrays, is not counted); c5_upload_mesh drops it.
double* resident_dir(c5_ctx* ctx) {
    DeviceState& d = ctx->dev;
    const size_t n = 2 * static_cast<size_t>(d.n_tets);
    if (d.jvp_dir.n != n) { // first call, or a sibling that followed its parent to a mesh of another size
        if (!ctx->parent) ctx->info.device_bytes -= static_cast<int64_t>(d.jvp_dir.bytes());
        d.jvp_dir.alloc(n);
        if (!ctx->parent) ctx->info.device_bytes += static_cast<int64_t>(d.jvp_dir.bytes());
    }
    return d.jvp_dir.p;
}

// One launch gathers the file-order direction (device pointers; a null one is 0) into the tangent field, then the
// view's walk stores {tau, I, dtau, dI} per pixel of the band into d.out. Events: 0..4 as for an image.
void enqueue_jvp(DeviceState& d, const c5_view* v, const ViewPlan& p, const uint32_t* tperm, double* dir,
                 const double* d_v_alpha, const double* d_v_q) {
    g_launch_counter = &d.launches;
    gather_direction(d.n_tets, tperm, d_v_alpha, d_v_q, dir, d.stream);
    enqueue_view(d, v, p, false, nullptr, 0, kJvpPass, dir);
}

// Band [row_begin,row_end) of v on ctx's device from host arrays: the direction goes to the device through the
// gradient's scratch arrays (file order, n_tets each), then enqueue_jvp and the copy of the band. Blocks until the
// results are on the host. Events: 0..4 as for enqueue_jvp, 5..6 around the copy.
ViewResult jvp_band(c5_ctx* ctx, const c5_view* v, const double* v_alpha, const double* v_q, double* tangent,
                    double* out) {
    follow_parent(ctx);
    if (ctx->pending.active) fail(C5_E_STATE, "render_jvp: this context still has a view in flight (c5_render_wait it first)");
    if (!ctx->has_mesh) fail(C5_E_STATE, "render: no mesh uploaded");
    const ViewPlan p = plan_view(v);
    DeviceState& d = ctx->dev;
    use_device(d);
    const uint32_t* tperm = resident_tperm(ctx);
    double* dir = resident_dir(ctx);
    const size_t n_t = static_cast<size_t>(d.n_tets);
    const size_t n_pix_band = static_cast<size_t>(p.row_end - p.row_begin) * v->res_x;
    const size_t band_off = static_cast<size_t>(p.row_begin) * v->res_x;
    ensure_host_staging(d, static_cast<size_t>(v->res_y));
    if (v_alpha) {
        d.grad_alpha.ensure(n_t);
        h2d(d.grad_alpha.p, v_alpha, n_t * sizeof(double), d.stream);
    }
    if (v_q) {
        d.grad_q.ensure(n_t);
        h2d(d.grad_q.p, v_q, n_t * sizeof(double), d.stream);
    }
    enqueue_jvp(d, v, p, tperm, dir, v_alpha ? d.grad_alpha.p : nullptr, v_q ? d.grad_q.p : nullptr);
    record(d, 5);
    std::vector<double> band(4 * n_pix_band); // {tau, I, dtau, dI} per pixel
    d2h(band.data(), d.out.p, band.size() * sizeof(double), d.stream);
    record(d, 6);
    d2h(d.h_counters, d.counters.p, kNumCounters * sizeof(unsigned long long), d.stream);
    d2h(d.h_row_cost, d.row_cost.p, static_cast<size_t>(v->res_y) * sizeof(uint64_t), d.stream);
    stream_sync(d.stream);
    for (size_t k = 0; k < n_pix_band; k++) {
        tangent[2 * (band_off + k)] = band[4 * k + 2];
        tangent[2 * (band_off + k) + 1] = band[4 * k + 3];
        if (out) {
            out[2 * (band_off + k)] = band[4 * k];
            out[2 * (band_off + k) + 1] = band[4 * k + 1];
        }
    }
    return read_view(d, *v, p, true);
}

// c5_render_jvp_device on a single-device context or a sibling: enqueue_jvp on the caller's stream, then the
// strided copies of the two pairs into the caller's band buffers.
void jvp_band_device(c5_ctx* ctx, const c5_view* v, const double* d_v_alpha, const double* d_v_q, double* d_tangent,
                     double* d_out, void* stream, c5_stats* stats) {
    follow_parent(ctx);
    if (!ctx->has_mesh) fail(C5_E_STATE, "render: no mesh uploaded");
    if (ctx->pending.active) fail(C5_E_STATE, "render_jvp_device: this context has a submitted view in flight");
    const ViewPlan p = plan_view(v);
    DeviceState& d = ctx->dev;
    use_device(d);
    const uint32_t* tperm = resident_tperm(ctx);
    double* dir = resident_dir(ctx);
    const size_t n_pix_band = static_cast<size_t>(p.row_end - p.row_begin) * v->res_x;
    if (stats) ensure_host_staging(d, static_cast<size_t>(v->res_y));
    // run on the CALLER's stream, like c5_render_device: the scratch arrays are the context's own
    cudaStream_t own = d.stream;
    if (!kHostSim) d.stream = static_cast<cudaStream_t>(stream);
    try {
        enqueue_jvp(d, v, p, tperm, dir, d_v_alpha, d_v_q);
        record(d, 5);
        d2d_2d(d_tangent, 2 * sizeof(double), d.out.p + 2, 4 * sizeof(double), 2 * sizeof(double), n_pix_band, d.stream);
        if (d_out) d2d_2d(d_out, 2 * sizeof(double), d.out.p, 4 * sizeof(double), 2 * sizeof(double), n_pix_band, d.stream);
        record(d, 6);
        if (!kHostSim && d.stream != own) { // the context's own later renders reuse these scratch arrays: they wait
            C5_CUDA(cudaEventRecord(d.ev_fields, d.stream));
            C5_CUDA(cudaStreamWaitEvent(own, d.ev_fields, 0));
        }
        if (stats) {
            d2h(d.h_counters, d.counters.p, kNumCounters * sizeof(unsigned long long), d.stream);
            d2h(d.h_row_cost, d.row_cost.p, static_cast<size_t>(v->res_y) * sizeof(uint64_t), d.stream);
            stream_sync(d.stream);
            ViewResult r = read_view(d, *v, p, true);
            report(ctx, r, stats);
        }
    } catch (...) {
        d.stream = own;
        throw;
    }
    d.stream = own;
}

// Arguments c5_render_jvp and c5_render_jvp_device share.
void check_jvp_args(const c5_view* view, const double* v_alpha, const double* v_q, const double* tangent, const char* who) {
    if (!tangent) fail(C5_E_INVALID, std::string(who) + ": tangent is NULL");
    if (!v_alpha && !v_q) fail(C5_E_INVALID, std::string(who) + ": v_alpha and v_q are both NULL");
    if (view && view->precision == 32) fail(C5_E_INVALID, std::string(who) + ": FP64 only (precision 64)");
    if (view && view->round_through_float) {
        fail(C5_E_INVALID, std::string(who) + ": the float cast has no useful derivative; set round_through_float = 0");
    }
}

// ---- light curves on device memory (c5_render_flux_device, c5_render_flux_jvp_device) ---------------------

// After a field update the first render derives fields[].s again (launch_prepare_cells), which on a mesh shared
// with lanes is fenced by device-wide syncs: the host would wait for the caller's earlier work. Here the cells
// (and channels) are prepared for alpha_limit on `s` instead, fenced by events: `s` waits for every stream the
// library renders on, and they all wait for `s`. A view with another limit still takes the synced path.
void prepare_fenced(c5_ctx* ctx, double alpha_limit, bool channels, cudaStream_t s) {
    DeviceState& o = ctx->dev;
    const bool cells = !(o.cells_limit_valid && o.cells_limit == alpha_limit);
    const bool chans = channels && !(o.ch_limit_valid && o.ch_limit == alpha_limit);
    if (!cells && !chans) return;
    const std::vector<DeviceState*> internal = internal_streams(ctx);
    if (!kHostSim) {
        for (DeviceState* x : internal) {
            C5_CUDA(cudaEventRecord(x->ev_fields, x->stream));
            C5_CUDA(cudaStreamWaitEvent(s, x->ev_fields, 0));
        }
    }
    cudaStream_t own = o.stream;
    if (!kHostSim) o.stream = s;
    try {
        if (cells) launch_prepare_cells(o, alpha_limit, true);
        if (chans) launch_prepare_channels(o, alpha_limit, true);
    } catch (...) {
        o.stream = own;
        throw;
    }
    o.stream = own;
    if (!kHostSim) {
        C5_CUDA(cudaEventRecord(o.ev_fields, s));
        for (DeviceState* x : internal) C5_CUDA(cudaStreamWaitEvent(x->stream, o.ev_fields, 0));
    }
}

// View k goes to lane k % views_in_flight, where its walk, its row sums and its total run on the lane's own
// stream, the total straight into the caller's array. jvp: the direction is gathered once, on `stream`, into the
// owner's tangent field, which every lane's walk reads (lanes share the owner's tet order); the walk's
// {tau, I, dtau, dI} per pixel is a two-pair band, so the row sums of a K = 2 channel image give the flux and the
// tangent at once. Otherwise each view runs what c5_render_flux runs (n_ch pairs: 0 = the cells' own fields).
void flux_device(c5_ctx* ctx, const c5_view* views, int32_t n_views, int n_ch, bool jvp, const double* d_v_alpha,
                 const double* d_v_q, double* d_tangent, double* d_total, void* stream, c5_stats* stats) {
    const std::string who = jvp ? "render_flux_jvp_device" : "render_flux_device";
    if (ctx->parent) fail(C5_E_STATE, who + ": a sibling context; call through its parent");
    if (!ctx->has_mesh) fail(C5_E_STATE, "render: no mesh uploaded");
    for (unsigned k = 0; k <= ctx->lanes.size(); k++) {
        if (lane_of(ctx, k)->pending.active) fail(C5_E_STATE, who + ": a submitted view is in flight");
    }
    std::vector<ViewPlan> plans;
    for (int32_t k = 0; k < n_views; k++) plans.push_back(plan_view(&views[k]));
    ensure_lanes(ctx);
    const unsigned n_lanes = static_cast<unsigned>(ctx->lanes.size()) + 1;
    for (unsigned k = 0; k < n_lanes; k++) follow_parent(lane_of(ctx, k));
    DeviceState& o = ctx->dev;
    use_device(o);
    const uint32_t* tperm = jvp ? resident_tperm(ctx) : nullptr;
    double* dir = jvp ? resident_dir(ctx) : nullptr;
    if (stats) ensure_view_counters(o, n_views);
    cudaStream_t s = kHostSim ? o.stream : static_cast<cudaStream_t>(stream);
    SpanEvents span;
    if (stats && !kHostSim) {
        for (cudaEvent_t& e : span.e) C5_CUDA(cudaEventCreate(&e));
        C5_CUDA(cudaEventRecord(span.e[0], s));
    }
    // 1. `stream` waits for the context's own stream (an earlier call's lanes may still read the tangent field),
    // 2. the gather, 3. every lane starts after that, and so after the caller's earlier work on `stream` (a
    // c5_update_fields_device, whatever wrote the direction)
    if (!kHostSim) {
        C5_CUDA(cudaEventRecord(o.ev_fields, o.stream));
        C5_CUDA(cudaStreamWaitEvent(s, o.ev_fields, 0));
    }
    g_launch_counter = &o.launches;
    prepare_fenced(ctx, views[0].alpha_limit, n_ch > 0, s);
    if (jvp) gather_direction(o.n_tets, tperm, d_v_alpha, d_v_q, dir, s);
    if (!kHostSim) {
        C5_CUDA(cudaEventRecord(o.ev_fields, s));
        for (unsigned k = 0; k < n_lanes; k++) C5_CUDA(cudaStreamWaitEvent(lane_of(ctx, k)->dev.stream, o.ev_fields, 0));
    }
    const int pairs = jvp ? 2 : n_ch ? n_ch : 1;      // pairs per pixel of the walk's band
    const int total_words = jvp ? 2 : 2 * pairs;      // d_total's doubles per view
    for (int32_t k = 0; k < n_views; k++) {
        DeviceState& d = lane_of(ctx, static_cast<unsigned>(k) % n_lanes)->dev;
        const c5_view* v = &views[k];
        const ViewPlan& p = plans[static_cast<size_t>(k)];
        if (jvp) enqueue_view(d, v, p, false, nullptr, 0, kJvpPass, dir);
        else enqueue_view(d, v, p, false, nullptr, n_ch);
        const bool solids = v->use_solids && (d.solid_follow.n + d.solid_static.n) > 0;
        launch_reduce_rows(d, v->res_x, v->res_y, p.row_begin, p.row_end, pairs, solids);
        launch_total_rows(d, p.row_begin, p.row_end, 2 * pairs, total_words,
                          d_total ? d_total + static_cast<size_t>(k) * total_words : nullptr,
                          jvp ? d_tangent + 2 * static_cast<size_t>(k) : nullptr);
        if (stats) d2h(o.h_view_counters + static_cast<size_t>(k) * kNumCounters, d.counters.p,
                       kNumCounters * sizeof(unsigned long long), d.stream);
    }
    // 4. `stream` waits for every lane, and the context's own later renders (and the next call) wait for `stream`
    if (!kHostSim) {
        for (unsigned k = 0; k < n_lanes; k++) {
            DeviceState& d = lane_of(ctx, k)->dev;
            C5_CUDA(cudaEventRecord(d.ev_fields, d.stream));
            C5_CUDA(cudaStreamWaitEvent(s, d.ev_fields, 0));
        }
        C5_CUDA(cudaEventRecord(o.ev_fields, s));
        C5_CUDA(cudaStreamWaitEvent(o.stream, o.ev_fields, 0));
    }
    if (stats) report_views(o, views, plans, s, span, stats);
}

void upload_solids(c5_ctx* ctx, const double* pts, int64_t n, int follows) {
    if (n < 0 || (n > 0 && !pts)) fail(C5_E_INVALID, "upload_solids: bad arguments");
    if (n == 0) return;
    for (c5_ctx* c : with_parts(ctx)) {
        DeviceState& d = c->dev;
        use_device(d);
        SolidSet& ss = follows ? d.solid_follow : d.solid_static;
        const size_t old_n = static_cast<size_t>(ss.n), add = static_cast<size_t>(n);
        DevBuf<double> merged;
        merged.alloc((old_n + add) * 12);
        if (old_n) d2d(merged.p, ss.pts0.p, old_n * 12 * sizeof(double), d.stream);
        h2d(merged.p + old_n * 12, pts, add * 12 * sizeof(double), d.stream);
        stream_sync(d.stream);
        ss.pts0 = std::move(merged);
        ss.n = static_cast<int64_t>(old_n + add);
        ss.pts_view.alloc(static_cast<size_t>(ss.n) * 12);
        // static solids are never rotated: their view-frame copy is the upload itself
        if (!follows) {
            d2d(ss.pts_view.p, ss.pts0.p, ss.pts0.bytes(), d.stream);
            stream_sync(d.stream);
        }
        // longest tet edge of this upload: bounds how many rows one face can span in any view
        for (size_t t = 0; t < add; t++) {
            const double* q = pts + 12 * t;
            for (int a = 0; a < 4; a++) {
                for (int b = a + 1; b < 4; b++) {
                    const double dx = q[3 * a] - q[3 * b], dy = q[3 * a + 1] - q[3 * b + 1], dz = q[3 * a + 2] - q[3 * b + 2];
                    ss.extent = std::max(ss.extent, std::sqrt(dx * dx + dy * dy + dz * dz));
                }
            }
        }
        g_launch_counter = &d.launches;
        dedupe_solid_faces(d, ss);
        d.mask_static_valid = false;
    }
    ctx->info.n_solid_tets += n;
}

// Points a sibling's device state at the mesh and solids its parent owns; per-view arrays are its own.
void alias_mesh(DeviceState& s, DeviceState& o) {
    use_device(s);
    s.origin = &o;
    o.mesh_shared = true;
    s.n_pts = o.n_pts;
    s.n_tets = o.n_tets;
    s.n_bfaces = o.n_bfaces;
    for (int a = 0; a < 3; a++) {
        s.mesh_lo[a] = o.mesh_lo[a];
        s.mesh_hi[a] = o.mesh_hi[a];
    }
    s.px.alias(o.px);
    s.py.alias(o.py);
    s.pz.alias(o.pz);
    s.conn.alias(o.conn);
    s.fields.alias(o.fields);
    s.q0.alias(o.q0);
    s.n_channels = o.n_channels;
    s.ch_rec.alias(o.ch_rec);
    s.ch_q0.alias(o.ch_q0);
    s.bfaces.alias(o.bfaces);
    s.node_parent.alias(o.node_parent);
    s.leaf_parent.alias(o.leaf_parent);
    s.nodes.alloc(o.nodes.n); // child links are static, the boxes are refitted per view
    if (o.nodes.n) d2d(s.nodes.p, o.nodes.p, o.nodes.bytes(), s.stream);
    s.refit_flags.alloc(o.refit_flags.n);
    s.vrot.alloc(static_cast<size_t>(o.n_pts));
    const SolidSet* from[2] = {&o.solid_follow, &o.solid_static};
    SolidSet* to[2] = {&s.solid_follow, &s.solid_static};
    for (int k = 0; k < 2; k++) {
        to[k]->n = from[k]->n;
        to[k]->n_faces = from[k]->n_faces;
        to[k]->extent = from[k]->extent;
        to[k]->pts0.alias(from[k]->pts0);
        to[k]->faces.alias(from[k]->faces);
        if (k == 0) to[k]->pts_view.alloc(from[k]->pts_view.n); // rotated with the view
        else to[k]->pts_view.alias(from[k]->pts_view);         // static solids are never rotated
    }
    s.mask_static_valid = false;
    stream_sync(s.stream);
    s.mesh_version = o.mesh_version;
}

// A sibling follows its parent's uploads lazily, at its next render.
void follow_parent(c5_ctx* ctx) {
    if (!ctx->parent) return;
    c5_ctx* par = ctx->parent;
    DeviceState& s = ctx->dev;
    DeviceState& o = par->dev;
    if (par->has_mesh && (s.origin != &o || s.mesh_version != o.mesh_version)) alias_mesh(s, o);
    ctx->has_mesh = par->has_mesh;
    ctx->info = par->info;
}

// cudaMalloc may carve an allocation out of a larger block, and a CUDA IPC handle names the BLOCK:
// the importer gets the block's base address. The driver knows the base (cuMemGetAddressRange);
// the offset travels with the handle. libcuda is loaded lazily so that the library still loads on
// machines without a driver (the CPU-only build container).
uint64_t offset_in_allocation(void* p) {
    using Fn = int (*)(unsigned long long*, size_t*, unsigned long long);
    static Fn fn = [] {
        void* h = dlopen("libcuda.so.1", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libcuda.so", RTLD_NOW | RTLD_GLOBAL);
        return h ? reinterpret_cast<Fn>(dlsym(h, "cuMemGetAddressRange_v2")) : nullptr;
    }();
    if (!fn) fail(C5_E_CUDA, "image_create: cuMemGetAddressRange not available (libcuda.so.1)");
    unsigned long long base = 0;
    size_t size = 0;
    const int rc = fn(&base, &size, static_cast<unsigned long long>(reinterpret_cast<uintptr_t>(p)));
    if (rc != 0) fail(C5_E_CUDA, "image_create: cuMemGetAddressRange failed (" + std::to_string(rc) + ")");
    return static_cast<uint64_t>(reinterpret_cast<uintptr_t>(p)) - base;
}

} // namespace

extern "C" {

int c5_abi_version(void) {
    return C5_ABI_VERSION;
}

void c5_view_from_flags(c5_view* v, int32_t res_x, int32_t res_y, double X_pi, double Y_pi, double I_pi,
                        double alpha_limit) {
    if (!v) return;
    std::memset(v, 0, sizeof(*v));
    v->res_x = res_x;
    v->res_y = res_y;
    v->window[0] = 2.2; // main.cpp:83
    v->window[1] = -0.2;
    v->window[2] = 0.9;
    v->window[3] = -0.9;
    const double a0 = -I_pi * kPi + kPi / 2.; // main.cpp:96
    v->n_rot = 3;
    v->rot[0] = c5_rotation{0, 0, a0, 0.0};                 // main.cpp:105
    v->rot[1] = c5_rotation{1, 0, Y_pi * kPi, 1.0};         // main.cpp:106, ACC_X0 = 1 (config.hpp:55)
    v->rot[2] = c5_rotation{0, 0, -a0 + X_pi * kPi, 0.0};   // main.cpp:107
    v->alpha_limit = alpha_limit;
    v->precision = 64;
    v->round_through_float = 1;
    v->use_solids = 1;
}

int c5_create(const int32_t* devices, int32_t n_dev, c5_ctx** out) {
    if (!out) return C5_E_INVALID;
    *out = nullptr;
    c5_ctx* ctx = nullptr;
    auto failed = [&](int code, const std::string& text) {
        {
            std::lock_guard<std::mutex> lock(g_create_err_mu);
            g_create_err = text;
        }
        c5_destroy(ctx); // the same teardown as a finished context: parts, streams, events, device memory
        return code;
    };
    try {
        if (n_dev < 1 || !devices) fail(C5_E_INVALID, "c5_create: need at least one device");
        ctx = new c5_ctx();
        if (!kHostSim) {
            int count = 0;
            cudaError_t e = cudaGetDeviceCount(&count);
            if (e != cudaSuccess || count == 0) {
                fail(C5_E_CUDA, std::string("c5_create: no CUDA device (") + cudaGetErrorString(e) +
                                    "); this library has no CPU path");
            }
            for (int k = 0; k < n_dev; k++) {
                if (devices[k] < 0 || devices[k] >= count) fail(C5_E_INVALID, "c5_create: device ordinal out of range");
            }
        }
        DeviceState& d = ctx->dev;
        d.device = devices[0];
        if (!kHostSim) {
            C5_CUDA(cudaSetDevice(d.device));
            C5_CUDA(cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking));
            for (auto& e : d.ev) C5_CUDA(cudaEventCreate(&e));
            C5_CUDA(cudaEventCreate(&d.ev_walk));
            C5_CUDA(cudaEventCreateWithFlags(&d.ev_done, cudaEventDisableTiming));
            C5_CUDA(cudaEventCreateWithFlags(&d.ev_fields, cudaEventDisableTiming));
            C5_CUDA(cudaEventCreateWithFlags(&d.ev_gather, cudaEventDisableTiming));
        }
        for (int k = 1; k < n_dev; k++) { // every further device: a single-device context of its own
            c5_ctx* part = nullptr;
            const int rc = c5_create(&devices[k], 1, &part);
            if (rc != C5_OK) fail(rc, c5_last_error(nullptr));
            ctx->parts.push_back(part);
        }
        *out = ctx;
        return C5_OK;
    } catch (const Error& e) {
        return failed(e.code, e.text);
    } catch (const std::exception& e) {
        return failed(C5_E_NOMEM, e.what());
    }
}

int c5_create_sibling(c5_ctx* parent, c5_ctx** out) {
    if (!parent || !out) return C5_E_INVALID;
    *out = nullptr;
    if (parent->parent || !parent->parts.empty()) {
        parent->err = "create_sibling: the parent must be a single-device context that is not itself a sibling";
        return C5_E_INVALID;
    }
    const int32_t device = parent->dev.device;
    c5_ctx* ctx = nullptr;
    const int rc = c5_create(&device, 1, &ctx);
    if (rc != C5_OK) return rc;
    // the internal streams made before a c5_update_fields_device wait for its gather; a sibling made after it
    // waits here, so that its renders see the new fields too (an event never recorded is no wait)
    if (!kHostSim) {
        const cudaError_t e = cudaStreamWaitEvent(ctx->dev.stream, parent->dev.ev_gather, 0);
        if (e != cudaSuccess) {
            parent->err = std::string("create_sibling: ") + cudaGetErrorString(e);
            c5_destroy(ctx);
            return C5_E_CUDA;
        }
    }
    ctx->parent = parent;
    parent->siblings.push_back(ctx);
    DeviceState& from = parent->dev;
    DeviceState& to = ctx->dev;
    to.opt_graze_list = from.opt_graze_list;
    to.opt_query_budget = from.opt_query_budget;
    to.opt_serial_list = from.opt_serial_list;
    to.opt_no_static_mask = from.opt_no_static_mask;
    to.opt_mask_tile = from.opt_mask_tile;
    to.opt_no_zero_copy = from.opt_no_zero_copy;
    *out = ctx;
    return C5_OK;
}

void c5_destroy(c5_ctx* ctx) {
    if (!ctx) return;
    for (c5_ctx* lane : ctx->lanes) c5_destroy(lane); // our own lanes go first (each leaves ctx->siblings)
    ctx->lanes.clear();
    for (c5_ctx* part : ctx->parts) c5_destroy(part);
    ctx->parts.clear();
    if (ctx->parent) { // a sibling leaves its parent's list
        auto& sib = ctx->parent->siblings;
        sib.erase(std::remove(sib.begin(), sib.end(), ctx), sib.end());
    }
    for (c5_ctx* s : ctx->siblings) { // a parent going first takes the shared mesh with it
        if (!kHostSim) {
            cudaSetDevice(s->dev.device);
            cudaDeviceSynchronize();
        }
        s->parent = nullptr;
        s->has_mesh = false;
        s->dev.origin = nullptr;
    }
    ctx->siblings.clear();
    DeviceState& d = ctx->dev;
    if (!kHostSim && d.stream) {
        cudaSetDevice(d.device);
        cudaStreamSynchronize(d.stream);
    }
    for (void* p : ctx->registered) {
        if (!kHostSim) cudaHostUnregister(p);
    }
    for (auto& im : ctx->images) {
        if (im.second) dev_free(im.first);
        else if (!kHostSim) cudaIpcCloseMemHandle(im.first);
    }
    host_pinned_free(d.h_counters);
    host_pinned_free(d.h_row_cost);
    host_pinned_free(d.h_row_flux);
    host_pinned_free(d.h_view_counters);
    if (!kHostSim) {
        for (cudaEvent_t e : d.tl_events) cudaEventDestroy(e);
        if (d.ev_walk) cudaEventDestroy(d.ev_walk);
        if (d.ev_done) cudaEventDestroy(d.ev_done);
        if (d.ev_fields) cudaEventDestroy(d.ev_fields);
        if (d.ev_gather) cudaEventDestroy(d.ev_gather);
        for (auto& e : d.ev) {
            if (e) cudaEventDestroy(e);
        }
        if (d.stream) cudaStreamDestroy(d.stream);
    }
    delete ctx; // DevBuf destructors free on the current device, d.device
}

const char* c5_last_error(const c5_ctx* ctx) {
    if (ctx) return ctx->err.c_str();
    std::lock_guard<std::mutex> lock(g_create_err_mu);
    static thread_local std::string copy;
    copy = g_create_err;
    return copy.c_str();
}

int c5_upload_mesh(c5_ctx* ctx, const double* points_xyz, int64_t n_points, const int32_t* tet_vertices,
                   int64_t n_tets, const double* alpha, const double* q) {
    if (!ctx) return C5_E_INVALID;
    return guarded(ctx, [&] {
        if (ctx->parent) fail(C5_E_STATE, "upload_mesh: a sibling context shares its parent's mesh; upload through the parent");
        if (!points_xyz || !tet_vertices || !alpha || !q) fail(C5_E_INVALID, "upload_mesh: NULL array");
        if (!ctx->siblings.empty() && !kHostSim) C5_CUDA(cudaDeviceSynchronize()); // siblings may be rendering from it
        ctx->dev.mesh_version++;
        const std::vector<c5_ctx*> all = with_parts(ctx);
        for (c5_ctx* c : all) {
            c->has_mesh = false;
            use_device(c->dev);
            upload_channels(c->dev, nullptr, nullptr, 0); // a new mesh drops the channels
            c->dev.tperm_dev.release();                   // and the device copy of the old permutation
            c->dev.jvp_dir.release();                     // and the tangent field of c5_render_jvp
        }
        ctx->info.device_bytes -= ctx->channel_bytes;
        ctx->channel_bytes = 0;
        const size_t before = dev_bytes_in_use();
        for (c5_ctx* c : all) {
            use_device(c->dev);
            g_launch_counter = &c->dev.launches;
            build_mesh(c->dev, points_xyz, n_points, tet_vertices, n_tets, alpha, q);
        }
        ctx->info.n_points = n_points;
        ctx->info.n_tets = n_tets;
        ctx->info.n_boundary_faces = ctx->dev.n_bfaces;
        ctx->info.n_bvh_nodes = ctx->dev.n_bfaces - 1;
        ctx->info.device_bytes = static_cast<int64_t>((dev_bytes_in_use() - before) / all.size());
        for (c5_ctx* c : all) c->has_mesh = true;
    });
}

#ifdef C5_HOSTSIM
// Host-loop build only, for the layout tests: the topology as the walk reads it. conn gets 8 int32 per
// tet (Conn), bfaces 8 int32 per boundary face (BFace), tperm the tet permutation (Morton -> file order).
extern "C" int c5_hostsim_topology(c5_ctx* ctx, int32_t* conn, int32_t* bfaces, uint32_t* tperm) {
    if (!ctx || !conn || !bfaces || !tperm) return C5_E_INVALID;
    return guarded(ctx, [&] {
        if (!ctx->has_mesh) fail(C5_E_STATE, "hostsim_topology: no mesh");
        const c5::DeviceState& d = ctx->dev;
        std::memcpy(conn, d.conn.p, d.conn.bytes());
        std::memcpy(bfaces, d.bfaces.p, d.bfaces.bytes());
        std::memcpy(tperm, d.tperm.data(), d.tperm.size() * sizeof(uint32_t));
    });
}
#endif

int c5_upload_solids(c5_ctx* ctx, const double* tet_points, int64_t n_tets, int32_t follows_view) {
    if (!ctx) return C5_E_INVALID;
    return guarded(ctx, [&] {
        if (ctx->parent) fail(C5_E_STATE, "upload_solids: upload through the parent context");
        if (!ctx->siblings.empty() && !kHostSim) C5_CUDA(cudaDeviceSynchronize());
        ctx->dev.mesh_version++;
        upload_solids(ctx, tet_points, n_tets, follows_view);
    });
}

int c5_clear_solids(c5_ctx* ctx) {
    if (!ctx) return C5_E_INVALID;
    return guarded(ctx, [&] {
        if (ctx->parent) fail(C5_E_STATE, "clear_solids: clear through the parent context");
        if (!ctx->siblings.empty() && !kHostSim) C5_CUDA(cudaDeviceSynchronize());
        ctx->dev.mesh_version++;
        for (c5_ctx* c : with_parts(ctx)) {
            DeviceState& d = c->dev;
            use_device(d);
            for (SolidSet* ss : {&d.solid_follow, &d.solid_static}) {
                ss->pts0.release();
                ss->pts_view.release();
                ss->faces.release();
                ss->n = 0;
                ss->n_faces = 0;
                ss->extent = 0.0;
            }
            d.mask_static_valid = false;
        }
        ctx->info.n_solid_tets = 0;
    });
}

int c5_mesh_info_get(const c5_ctx* ctx, c5_mesh_info* out) {
    if (!ctx || !out) return C5_E_INVALID;
    *out = ctx->info;
    return C5_OK;
}

int c5_render(c5_ctx* ctx, const c5_view* view, double* out, c5_stats* stats) {
    return c5_render_raw(ctx, view, out, nullptr, nullptr, stats);
}

int c5_render_raw(c5_ctx* ctx, const c5_view* view, double* out, uint32_t* steps, uint8_t* solid_mask,
                  c5_stats* stats) {
    if (!ctx) return C5_E_INVALID;
    return guarded(ctx, [&] {
        if (!ctx->parts.empty()) {
            render_multi_device(ctx, view, out, steps, solid_mask, stats);
            return;
        }
        submit_view(ctx, view, out, steps, solid_mask, 0);
        ViewResult r = wait_view(ctx);
        report(ctx, r, stats);
    });
}

int c5_upload_channels(c5_ctx* ctx, const double* alpha, const double* q, int32_t n_channels) {
    if (!ctx) return C5_E_INVALID;
    return guarded(ctx, [&] {
        if (ctx->parent) fail(C5_E_STATE, "upload_channels: a sibling context shares its parent's channels; upload through the parent");
        if (!alpha || !q) fail(C5_E_INVALID, "upload_channels: NULL array");
        if (n_channels < 0 || n_channels > C5_MAX_CHANNELS) fail(C5_E_INVALID, "upload_channels: n_channels must be 0 .. C5_MAX_CHANNELS");
        if (!ctx->has_mesh) fail(C5_E_STATE, "upload_channels: no mesh uploaded");
        for (unsigned k = 0; k <= ctx->lanes.size(); k++) {
            if (lane_of(ctx, k)->pending.active) fail(C5_E_STATE, "upload_channels: a submitted view is in flight");
        }
        if (!ctx->siblings.empty() && !kHostSim) C5_CUDA(cudaDeviceSynchronize()); // siblings may be rendering from them
        ctx->dev.mesh_version++; // siblings and lanes re-alias at their next render
        const std::vector<c5_ctx*> all = with_parts(ctx);
        // the old channels go first: a failed upload leaves none anywhere, and the sizes say so
        ctx->info.device_bytes -= ctx->channel_bytes;
        ctx->channel_bytes = 0;
        try {
            for (c5_ctx* c : all) {
                use_device(c->dev);
                g_launch_counter = &c->dev.launches;
                upload_channels(c->dev, alpha, q, n_channels);
            }
        } catch (...) {
            for (c5_ctx* c : all) {
                use_device(c->dev);
                upload_channels(c->dev, nullptr, nullptr, 0);
            }
            throw;
        }
        ctx->channel_bytes = static_cast<int64_t>(ctx->dev.ch_rec.bytes() + ctx->dev.ch_q0.bytes());
        ctx->info.device_bytes += ctx->channel_bytes;
    });
}

int c5_render_channels(c5_ctx* ctx, const c5_view* view, double* out, uint32_t* steps, uint8_t* solid_mask,
                       c5_stats* stats) {
    if (!ctx) return C5_E_INVALID;
    return guarded(ctx, [&] {
        if (view && view->precision == 32) fail(C5_E_INVALID, "render_channels: FP64 only (precision 64)");
        check_channels_ready(ctx);
        if (!ctx->parts.empty()) {
            render_multi_device(ctx, view, out, steps, solid_mask, stats, true);
            return;
        }
        submit_view(ctx, view, out, steps, solid_mask, 0, true, true);
        ViewResult r = wait_view(ctx);
        report(ctx, r, stats);
    });
}

int c5_update_fields(c5_ctx* ctx, const double* alpha, const double* q) {
    if (!ctx) return C5_E_INVALID;
    return guarded(ctx, [&] {
        if (ctx->parent) fail(C5_E_STATE, "update_fields: a sibling context shares its parent's fields; update through the parent");
        if (!alpha || !q) fail(C5_E_INVALID, "update_fields: NULL array");
        if (!ctx->has_mesh) fail(C5_E_STATE, "update_fields: no mesh uploaded");
        for (unsigned k = 0; k <= ctx->lanes.size(); k++) {
            if (lane_of(ctx, k)->pending.active) fail(C5_E_STATE, "update_fields: a submitted view is in flight");
        }
        if (!ctx->siblings.empty() && !kHostSim) C5_CUDA(cudaDeviceSynchronize()); // siblings may be rendering from them
        ctx->dev.mesh_version++; // siblings and lanes re-alias at their next render
        for (c5_ctx* c : with_parts(ctx)) {
            use_device(c->dev);
            g_launch_counter = &c->dev.launches;
            update_fields(c->dev, alpha, q);
        }
    });
}

int c5_render_grad(c5_ctx* ctx, const c5_view* view, const double* g, double* grad_alpha, double* grad_q, double* out,
                   c5_stats* stats) {
    if (!ctx) return C5_E_INVALID;
    return guarded(ctx, [&] {
        if (!g) fail(C5_E_INVALID, "render_grad: g is NULL");
        if (!grad_alpha && !grad_q) fail(C5_E_INVALID, "render_grad: grad_alpha and grad_q are both NULL");
        if (view && view->precision == 32) fail(C5_E_INVALID, "render_grad: FP64 only (precision 64)");
        if (view && view->round_through_float) {
            fail(C5_E_INVALID, "render_grad: the float cast has no useful derivative; set round_through_float = 0");
        }
        follow_parent(ctx);
        if (!ctx->has_mesh) fail(C5_E_STATE, "render: no mesh uploaded");
        const ViewPlan p = plan_view(view);
        const std::vector<c5_ctx*> parts = with_parts(ctx);
        const size_t n = parts.size();
        if (static_cast<size_t>(p.row_end - p.row_begin) < n) fail(C5_E_INVALID, "render: fewer rows than devices");
        const auto bands = cut_bands(ctx, view, p, static_cast<int>(n));
        std::vector<c5_view> band_views(n, *view);
        std::vector<GradResult> results(n);
        std::vector<std::exception_ptr> errors(n);
        auto run = [&](size_t r) {
            try {
                band_views[r].row_begin = bands[r].first;
                band_views[r].row_end = bands[r].second;
                results[r] = grad_band(parts[r], &band_views[r], g, grad_alpha != nullptr, grad_q != nullptr, out);
            } catch (...) {
                errors[r] = std::current_exception();
            }
        };
        if (kHostSim || n == 1) {
            for (size_t r = 0; r < n; r++) run(r);
        } else {
            std::vector<std::thread> workers;
            for (size_t r = 0; r < n; r++) workers.emplace_back(run, r);
            for (auto& w : workers) w.join();
        }
        for (auto& e : errors) {
            if (e) std::rethrow_exception(e);
        }
        // each device summed its own band: add them in device order
        const size_t n_t = static_cast<size_t>(ctx->info.n_tets);
        for (int k = 0; k < 2; k++) {
            double* dst = k == 0 ? grad_alpha : grad_q;
            if (!dst) continue;
            for (size_t r = 0; r < n; r++) {
                const std::vector<double>& src = k == 0 ? results[r].grad_alpha : results[r].grad_q;
                for (size_t t = 0; t < n_t; t++) dst[t] = r == 0 ? src[t] : dst[t] + src[t];
            }
        }
        std::vector<ViewResult> views(n);
        for (size_t r = 0; r < n; r++) views[r] = std::move(results[r].view);
        ViewResult total = n == 1 ? std::move(views[0]) : merge_results(views, view->res_y);
        report(ctx, total, stats);
    });
}

int c5_update_fields_device(c5_ctx* ctx, const double* d_alpha, const double* d_q, void* stream) {
    if (!ctx) return C5_E_INVALID;
    return guarded(ctx, [&] {
        if (ctx->parent) fail(C5_E_STATE, "update_fields_device: a sibling context shares its parent's fields; update through the parent");
        if (!ctx->parts.empty()) fail(C5_E_INVALID, "update_fields_device: single-device contexts only");
        check_device_array(d_alpha, "update_fields_device: d_alpha");
        check_device_array(d_q, "update_fields_device: d_q");
        if (!ctx->has_mesh) fail(C5_E_STATE, "update_fields_device: no mesh uploaded");
        for (unsigned k = 0; k <= ctx->lanes.size(); k++) {
            if (lane_of(ctx, k)->pending.active) fail(C5_E_STATE, "update_fields_device: a submitted view is in flight");
        }
        DeviceState& d = ctx->dev;
        use_device(d);
        const uint32_t* tperm = resident_tperm(ctx);
        cudaStream_t s = kHostSim ? d.stream : static_cast<cudaStream_t>(stream);
        const std::vector<DeviceState*> internal = internal_streams(ctx);
        if (!kHostSim) { // the gather waits for every render the library has enqueued on the old fields ...
            for (DeviceState* x : internal) {
                C5_CUDA(cudaEventRecord(x->ev_fields, x->stream));
                C5_CUDA(cudaStreamWaitEvent(s, x->ev_fields, 0));
            }
        }
        ctx->dev.mesh_version++; // siblings and lanes re-alias at their next render
        gather_fields(d, tperm, d_alpha, d_q, s);
        if (!kHostSim) { // ... and every later one waits for the gather, also those of lanes made later
            C5_CUDA(cudaEventRecord(d.ev_gather, s));
            for (DeviceState* x : internal) C5_CUDA(cudaStreamWaitEvent(x->stream, d.ev_gather, 0));
        }
    });
}

int c5_render_grad_device(c5_ctx* ctx, const c5_view* view, const double* d_g, double* d_grad_alpha, double* d_grad_q,
                          double* d_out, void* stream, c5_stats* stats) {
    if (!ctx) return C5_E_INVALID;
    return guarded(ctx, [&] {
        check_device_array(d_g, "render_grad_device: d_g");
        if (!d_grad_alpha && !d_grad_q) fail(C5_E_INVALID, "render_grad_device: d_grad_alpha and d_grad_q are both NULL");
        if (d_grad_alpha) check_device_array(d_grad_alpha, "render_grad_device: d_grad_alpha");
        if (d_grad_q) check_device_array(d_grad_q, "render_grad_device: d_grad_q");
        if (d_out) check_device_array(d_out, "render_grad_device: d_out");
        if (view && view->precision == 32) fail(C5_E_INVALID, "render_grad_device: FP64 only (precision 64)");
        if (view && view->round_through_float) {
            fail(C5_E_INVALID, "render_grad_device: the float cast has no useful derivative; set round_through_float = 0");
        }
        if (!ctx->parts.empty()) fail(C5_E_INVALID, "render_grad_device: single-device contexts only");
        grad_band_device(ctx, view, d_g, d_grad_alpha, d_grad_q, d_out, stream, stats);
    });
}

int c5_render_flux_grad_device(c5_ctx* ctx, const c5_view* views, int32_t n_views, const double* d_g,
                               double* d_grad_alpha, double* d_grad_q, void* stream, c5_stats* stats) {
    if (!ctx) return C5_E_INVALID;
    return guarded(ctx, [&] {
        if (n_views < 1 || !views) fail(C5_E_INVALID, "render_flux_grad_device: need at least one view");
        check_device_array(d_g, "render_flux_grad_device: d_g");
        if (!d_grad_alpha && !d_grad_q) fail(C5_E_INVALID, "render_flux_grad_device: d_grad_alpha and d_grad_q are both NULL");
        if (d_grad_alpha) check_device_array(d_grad_alpha, "render_flux_grad_device: d_grad_alpha");
        if (d_grad_q) check_device_array(d_grad_q, "render_flux_grad_device: d_grad_q");
        for (int32_t k = 0; k < n_views; k++) {
            if (views[k].precision == 32) fail(C5_E_INVALID, "render_flux_grad_device: FP64 only (precision 64)");
            if (views[k].round_through_float) {
                fail(C5_E_INVALID, "render_flux_grad_device: the float cast has no useful derivative; set round_through_float = 0");
            }
        }
        if (!ctx->parts.empty()) fail(C5_E_INVALID, "render_flux_grad_device: single-device contexts only");
        flux_grad_device(ctx, views, n_views, d_g, d_grad_alpha, d_grad_q, stream, stats);
    });
}

int c5_render_jvp(c5_ctx* ctx, const c5_view* view, const double* v_alpha, const double* v_q, double* tangent,
                  double* out, c5_stats* stats) {
    if (!ctx) return C5_E_INVALID;
    return guarded(ctx, [&] {
        check_jvp_args(view, v_alpha, v_q, tangent, "render_jvp");
        follow_parent(ctx);
        if (!ctx->has_mesh) fail(C5_E_STATE, "render: no mesh uploaded");
        const ViewPlan p = plan_view(view);
        const std::vector<c5_ctx*> parts = with_parts(ctx);
        const size_t n = parts.size();
        if (static_cast<size_t>(p.row_end - p.row_begin) < n) fail(C5_E_INVALID, "render: fewer rows than devices");
        const auto bands = cut_bands(ctx, view, p, static_cast<int>(n));
        std::vector<c5_view> band_views(n, *view);
        std::vector<ViewResult> results(n);
        std::vector<std::exception_ptr> errors(n);
        auto run = [&](size_t r) {
            try {
                band_views[r].row_begin = bands[r].first;
                band_views[r].row_end = bands[r].second;
                results[r] = jvp_band(parts[r], &band_views[r], v_alpha, v_q, tangent, out);
            } catch (...) {
                errors[r] = std::current_exception();
            }
        };
        if (kHostSim || n == 1) {
            for (size_t r = 0; r < n; r++) run(r);
        } else {
            std::vector<std::thread> workers;
            for (size_t r = 0; r < n; r++) workers.emplace_back(run, r);
            for (auto& w : workers) w.join();
        }
        for (auto& e : errors) {
            if (e) std::rethrow_exception(e);
        }
        ViewResult total = n == 1 ? std::move(results[0]) : merge_results(results, view->res_y);
        report(ctx, total, stats);
    });
}

int c5_render_jvp_device(c5_ctx* ctx, const c5_view* view, const double* d_v_alpha, const double* d_v_q,
                         double* d_tangent, double* d_out, void* stream, c5_stats* stats) {
    if (!ctx) return C5_E_INVALID;
    return guarded(ctx, [&] {
        check_jvp_args(view, d_v_alpha, d_v_q, d_tangent, "render_jvp_device");
        if (d_v_alpha) check_device_array(d_v_alpha, "render_jvp_device: d_v_alpha");
        if (d_v_q) check_device_array(d_v_q, "render_jvp_device: d_v_q");
        if (reinterpret_cast<uintptr_t>(d_tangent) & 15u) fail(C5_E_INVALID, "render_jvp_device: d_tangent must be 16-byte aligned");
        if (reinterpret_cast<uintptr_t>(d_out) & 15u) fail(C5_E_INVALID, "render_jvp_device: d_out must be 16-byte aligned");
        if (!ctx->parts.empty()) fail(C5_E_INVALID, "render_jvp_device: single-device contexts only");
        jvp_band_device(ctx, view, d_v_alpha, d_v_q, d_tangent, d_out, stream, stats);
    });
}

int c5_render_flux_device(c5_ctx* ctx, const c5_view* views, int32_t n_views, int32_t channels, double* d_total,
                          void* stream, c5_stats* stats) {
    if (!ctx) return C5_E_INVALID;
    return guarded(ctx, [&] {
        if (n_views < 1 || !views) fail(C5_E_INVALID, "render_flux_device: need at least one view");
        check_device_array(d_total, "render_flux_device: d_total");
        for (int32_t k = 0; k < n_views; k++) check_flux_args(&views[k], channels, nullptr, d_total);
        if (!ctx->parts.empty()) fail(C5_E_INVALID, "render_flux_device: single-device contexts only");
        if (channels) check_channels_ready(ctx);
        flux_device(ctx, views, n_views, channels ? ctx->dev.n_channels : 0, false, nullptr, nullptr, nullptr, d_total,
                    stream, stats);
    });
}

int c5_render_flux_jvp_device(c5_ctx* ctx, const c5_view* views, int32_t n_views, const double* d_v_alpha,
                              const double* d_v_q, double* d_tangent, double* d_total, void* stream, c5_stats* stats) {
    if (!ctx) return C5_E_INVALID;
    return guarded(ctx, [&] {
        if (n_views < 1 || !views) fail(C5_E_INVALID, "render_flux_jvp_device: need at least one view");
        check_device_array(d_tangent, "render_flux_jvp_device: d_tangent");
        if (d_total) check_device_array(d_total, "render_flux_jvp_device: d_total");
        if (d_v_alpha) check_device_array(d_v_alpha, "render_flux_jvp_device: d_v_alpha");
        if (d_v_q) check_device_array(d_v_q, "render_flux_jvp_device: d_v_q");
        for (int32_t k = 0; k < n_views; k++) check_jvp_args(&views[k], d_v_alpha, d_v_q, d_tangent, "render_flux_jvp_device");
        if (!ctx->parts.empty()) fail(C5_E_INVALID, "render_flux_jvp_device: single-device contexts only");
        flux_device(ctx, views, n_views, 0, true, d_v_alpha, d_v_q, d_tangent, d_total, stream, stats);
    });
}

int c5_set_views_in_flight(c5_ctx* ctx, int32_t n) {
    if (!ctx) return C5_E_INVALID;
    return guarded(ctx, [&] {
        if (n < 1 || n > C5_MAX_IN_FLIGHT) fail(C5_E_INVALID, "set_views_in_flight: 1 .. C5_MAX_IN_FLIGHT");
        if (ctx->parent || !ctx->parts.empty()) fail(C5_E_INVALID, "set_views_in_flight: single-device contexts that are not siblings");
        for (unsigned k = 0; k <= ctx->lanes.size(); k++) {
            if (lane_of(ctx, k)->pending.active) fail(C5_E_STATE, "set_views_in_flight: views are in flight");
        }
        while (static_cast<int>(ctx->lanes.size()) + 1 > n) { // lanes that are no longer wanted
            c5_destroy(ctx->lanes.back());
            ctx->lanes.pop_back();
        }
        ctx->views_in_flight = n;
        ctx->next_lane = 0;
    });
}

int c5_render_submit(c5_ctx* ctx, const c5_view* view, double* out, uint64_t* ticket) {
    if (!ctx || !ticket) return C5_E_INVALID;
    return guarded(ctx, [&] {
        if (ctx->parent || !ctx->parts.empty()) fail(C5_E_INVALID, "render_submit: single-device contexts that are not siblings");
        submit_on_lane(ctx, view, out, ticket, false, nullptr);
    });
}

int c5_render_flux(c5_ctx* ctx, const c5_view* view, int32_t channels, double* rows, double* total, c5_stats* stats) {
    if (!ctx) return C5_E_INVALID;
    return guarded(ctx, [&] {
        check_flux_args(view, channels, rows, total);
        if (channels) check_channels_ready(ctx);
        const FluxOut f{rows, total};
        if (!ctx->parts.empty()) {
            render_multi_device(ctx, view, nullptr, nullptr, nullptr, stats, channels != 0, &f);
            return;
        }
        submit_view(ctx, view, nullptr, nullptr, nullptr, 0, false, channels != 0, &f);
        ViewResult r = wait_view(ctx);
        deliver_flux(r.flux, 2 * static_cast<size_t>(ctx->pending.flux_pairs), f);
        report(ctx, r, stats);
    });
}

int c5_render_flux_submit(c5_ctx* ctx, const c5_view* view, int32_t channels, double* rows, double* total,
                          uint64_t* ticket) {
    if (!ctx || !ticket) return C5_E_INVALID;
    return guarded(ctx, [&] {
        check_flux_args(view, channels, rows, total);
        if (ctx->parent || !ctx->parts.empty()) fail(C5_E_STATE, "render_flux_submit: single-device contexts that are not siblings");
        const FluxOut f{rows, total};
        submit_on_lane(ctx, view, nullptr, ticket, channels != 0, &f);
    });
}

int c5_render_wait(c5_ctx* ctx, uint64_t ticket, c5_stats* stats) {
    if (!ctx) return C5_E_INVALID;
    return guarded(ctx, [&] {
        for (unsigned k = 0; k <= ctx->lanes.size(); k++) {
            c5_ctx* lane = lane_of(ctx, k);
            if (lane->pending.active && lane->pending.ticket == ticket && ticket != 0) {
                ViewResult r = wait_view(lane);
                if (lane->pending.flux_pairs) deliver_flux(r.flux, 2 * static_cast<size_t>(lane->pending.flux_pairs), lane->pending.flux);
                report(ctx, r, stats);
                return;
            }
        }
        fail(C5_E_INVALID, "render_wait: no view with this ticket is in flight");
    });
}

int c5_render_device(c5_ctx* ctx, const c5_view* view, void* d_out, void* stream, c5_stats* stats) {
    if (!ctx) return C5_E_INVALID;
    return guarded(ctx, [&] {
        follow_parent(ctx);
        if (!ctx->has_mesh) fail(C5_E_STATE, "render: no mesh uploaded");
        if (!d_out) fail(C5_E_INVALID, "render_device: d_out is NULL");
        if (reinterpret_cast<uintptr_t>(d_out) & 15u) fail(C5_E_INVALID, "render_device: d_out must be 16-byte aligned");
        if (!ctx->parts.empty()) fail(C5_E_INVALID, "render_device: single-device contexts only");
        if (ctx->pending.active) fail(C5_E_STATE, "render_device: this context has a submitted view in flight");
        const ViewPlan p = plan_view(view);
        DeviceState& d = ctx->dev;
        if (stats) ensure_host_staging(d, static_cast<size_t>(view->res_y));
        // run on the CALLER's stream (NULL = the legacy default stream, which is what torch's
        // default "current stream" is) so the result is ordered with the caller's later work
        cudaStream_t own = d.stream;
        if (!kHostSim) d.stream = static_cast<cudaStream_t>(stream);
        try {
            enqueue_view(d, view, p, false, static_cast<double*>(d_out)); // the walk stores into the caller's buffer
            // stats == NULL: fire and forget — nothing is read back and the stream is not synchronised,
            // so successive views (and the caller's gather) pipeline on the device
            if (stats) {
                d2h(d.h_counters, d.counters.p, kNumCounters * sizeof(unsigned long long), d.stream);
                d2h(d.h_row_cost, d.row_cost.p, static_cast<size_t>(view->res_y) * sizeof(uint64_t), d.stream);
                stream_sync(d.stream);
                ViewResult r = read_view(d, *view, p, false);
                report(ctx, r, stats);
            }
        } catch (...) {
            d.stream = own;
            throw;
        }
        d.stream = own;
    });
}

int c5_last_row_cost(c5_ctx* ctx, uint64_t* rows, int32_t n_rows) {
    if (!ctx || !rows || n_rows < 0) return C5_E_INVALID;
    for (int32_t j = 0; j < n_rows; j++) {
        rows[j] = static_cast<size_t>(j) < ctx->last_row_cost.size() ? ctx->last_row_cost[static_cast<size_t>(j)] : 0;
    }
    return C5_OK;
}

int c5_image_create(c5_ctx* ctx, uint64_t bytes, void** d_ptr, uint8_t handle[C5_IPC_HANDLE_BYTES]) {
    if (!ctx || !d_ptr || !handle) return C5_E_INVALID;
    return guarded(ctx, [&] {
        if (bytes == 0) fail(C5_E_INVALID, "image_create: zero bytes");
        use_device(ctx->dev);
        void* p = dev_alloc(bytes);
        std::memset(handle, 0, C5_IPC_HANDLE_BYTES);
        uint64_t offset = 0;
        if (kHostSim) {
            std::memcpy(handle, &p, sizeof(p)); // same-process stand-in (CPU logic tests only)
        } else {
            static_assert(sizeof(cudaIpcMemHandle_t) + 16 <= C5_IPC_HANDLE_BYTES, "IPC handle size");
            cudaIpcMemHandle_t h;
            try {
                offset = offset_in_allocation(p);
                C5_CUDA(cudaIpcGetMemHandle(&h, p));
            } catch (...) {
                dev_free(p);
                throw;
            }
            std::memcpy(handle, &h, sizeof(h));
        }
        std::memcpy(handle + 64, &offset, sizeof(offset));
        std::memcpy(handle + 72, &bytes, sizeof(bytes));
        ctx->images.emplace_back(p, true);
        *d_ptr = p;
    });
}

int c5_image_open(c5_ctx* ctx, const uint8_t handle[C5_IPC_HANDLE_BYTES], void** d_ptr) {
    if (!ctx || !d_ptr || !handle) return C5_E_INVALID;
    return guarded(ctx, [&] {
        use_device(ctx->dev);
        void* p = nullptr;
        if (kHostSim) {
            std::memcpy(&p, handle, sizeof(p));
        } else {
            cudaIpcMemHandle_t h;
            std::memcpy(&h, handle, sizeof(h));
            // maps the owner's allocation into this process and enables peer access to its device
            C5_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
        }
        uint64_t offset = 0;
        std::memcpy(&offset, handle + 64, sizeof(offset));
        ctx->images.emplace_back(p, false); // the mapping's base: what cudaIpcCloseMemHandle wants back
        ctx->image_offsets.emplace_back(static_cast<char*>(p) + offset, p);
        *d_ptr = static_cast<char*>(p) + offset;
    });
}

int c5_image_close(c5_ctx* ctx, void* d_ptr) {
    if (!ctx || !d_ptr) return C5_E_INVALID;
    return guarded(ctx, [&] {
        for (size_t k = 0; k < ctx->image_offsets.size(); k++) { // an imported image is known by its offset pointer
            if (ctx->image_offsets[k].first != d_ptr) continue;
            d_ptr = ctx->image_offsets[k].second;
            ctx->image_offsets.erase(ctx->image_offsets.begin() + static_cast<long>(k));
            break;
        }
        for (size_t k = 0; k < ctx->images.size(); k++) {
            if (ctx->images[k].first != d_ptr) continue;
            const bool owner = ctx->images[k].second;
            ctx->images.erase(ctx->images.begin() + static_cast<long>(k));
            use_device(ctx->dev);
            if (owner) dev_free(d_ptr);
            else if (!kHostSim) C5_CUDA(cudaIpcCloseMemHandle(d_ptr));
            return;
        }
        fail(C5_E_INVALID, "image_close: not an image of this context");
    });
}

int c5_host_register(c5_ctx* ctx, void* ptr, uint64_t bytes) {
    if (!ctx || !ptr || bytes == 0) return C5_E_INVALID;
    return guarded(ctx, [&] {
        use_device(ctx->dev);
        if (!kHostSim) C5_CUDA(cudaHostRegister(ptr, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped));
        ctx->registered.push_back(ptr);
    });
}

int c5_host_unregister(c5_ctx* ctx, void* ptr) {
    if (!ctx || !ptr) return C5_E_INVALID;
    return guarded(ctx, [&] {
        for (size_t k = 0; k < ctx->registered.size(); k++) {
            if (ctx->registered[k] != ptr) continue;
            ctx->registered.erase(ctx->registered.begin() + static_cast<long>(k));
            if (!kHostSim) C5_CUDA(cudaHostUnregister(ptr));
            return;
        }
        fail(C5_E_INVALID, "host_unregister: not registered through this context");
    });
}

uint64_t c5_kernel_launches(const c5_ctx* ctx) {
    uint64_t n = 0;
    if (ctx) {
        n = ctx->dev.launches;
        for (const c5_ctx* lane : ctx->lanes) n += c5_kernel_launches(lane);
        for (const c5_ctx* part : ctx->parts) n += c5_kernel_launches(part);
    }
    return n;
}

int c5_debug_set(c5_ctx* ctx, const char* key, int64_t value) {
    if (!ctx || !key) return C5_E_INVALID;
    return guarded(ctx, [&] {
        const std::string k = key;
        std::vector<c5_ctx*> all = with_parts(ctx);
        all.insert(all.end(), ctx->siblings.begin(), ctx->siblings.end()); // the caller's siblings and our lanes
        for (c5_ctx* c : all) {
            DeviceState& d = c->dev;
            if (k == "graze_list") d.opt_graze_list = static_cast<int>(value);
            else if (k == "query_budget") d.opt_query_budget = static_cast<int>(value);
            else if (k == "serial_list") d.opt_serial_list = static_cast<int>(value);
            else if (k == "mask_tile") d.opt_mask_tile = static_cast<int>(value);
            else if (k == "no_static_mask") {
                d.opt_no_static_mask = value != 0;
                d.mask_static_valid = false;
            }
            else if (k == "no_zero_copy") d.opt_no_zero_copy = value != 0;
            else if (k == "timeline") {
                if (value < 0 || value > 4096) fail(C5_E_INVALID, "debug_set: timeline 0 .. 4096 views");
                if (kHostSim) continue;
                use_device(d);
                C5_CUDA(cudaStreamSynchronize(d.stream));
                for (cudaEvent_t e : d.tl_events) cudaEventDestroy(e);
                d.tl_events.clear();
                d.tl_views = 0;
                for (int64_t i = 0; i < value * kTimelinePhases; i++) {
                    cudaEvent_t e = nullptr;
                    C5_CUDA(cudaEventCreate(&e));
                    d.tl_events.push_back(e);
                }
            } else {
                fail(C5_E_INVALID, "debug_set: unknown key '" + k + "'");
            }
        }
    });
}

int c5_timeline_read(c5_ctx* ctx, void* origin, float* ms_out, int32_t max_views, int32_t* n_views) {
    if (!ctx || !ms_out || !n_views || max_views < 0) return C5_E_INVALID;
    return guarded(ctx, [&] {
        *n_views = 0;
        if (kHostSim) return;
        if (!origin) fail(C5_E_INVALID, "timeline_read: origin event is NULL");
        DeviceState& d = ctx->dev;
        use_device(d);
        const uint64_t cap = d.tl_events.size() / kTimelinePhases;
        if (cap == 0) return;
        const uint64_t have = std::min<uint64_t>({d.tl_views, cap, static_cast<uint64_t>(max_views)});
        for (uint64_t i = 0; i < have; i++) {
            const uint64_t view = d.tl_views - have + i;
            for (int ph = 0; ph < kTimelinePhases; ph++) {
                cudaEvent_t e = d.tl_events[(view % cap) * kTimelinePhases + static_cast<size_t>(ph)];
                C5_CUDA(cudaEventSynchronize(e));
                C5_CUDA(cudaEventElapsedTime(ms_out + i * kTimelinePhases + ph, static_cast<cudaEvent_t>(origin), e));
            }
        }
        *n_views = static_cast<int32_t>(have);
    });
}

} // extern "C"
