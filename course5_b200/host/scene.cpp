// scene.cpp — see scene.hpp.
#include "scene.hpp"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <stdexcept>

#include "vti_writer.hpp"

namespace c5host {

namespace {

void apply(const c5_rotation& r, point& p) {
    if (r.axis == 0) rotate_point_x(p, r.angle);
    else rotate_point_y(p, r.angle, r.x0);
}

bool same_rotations(const std::vector<c5_rotation>& a, const std::vector<c5_rotation>& b) {
    if (a.size() != b.size()) return false;
    for (std::size_t i = 0; i < a.size(); i++) {
        if (a[i].axis != b[i].axis || a[i].angle != b[i].angle || a[i].x0 != b[i].x0) return false;
    }
    return true;
}

void check(c5_ctx* ctx, int rc, const char* what) {
    if (rc != C5_OK) {
        throw std::runtime_error(std::string(what) + ": " + c5_last_error(ctx) + " (code " + std::to_string(rc) + ")");
    }
}

} // namespace

void object3d_base::read_vtk_file(const std::string& filename, const std::vector<std::string>& scalar_labels) {
    _data->type = tetra_type::transparent;
    _data->grid = read_legacy_vtk(filename);
    for (std::size_t i = 0; i < scalar_labels.size() && i < 2; i++) {
        _data->labels[i] = scalar_labels[i];
        if (!_data->grid.cell_scalars.count(scalar_labels[i])) {
            throw std::runtime_error(filename + ": no cell scalar named '" + scalar_labels[i] + "'");
        }
    }
}

void object3d_base::init_polar(const std::function<double(const point&)>& potential_function, double x0, double y0,
                               double z0, double level_value, double step, double angle_step,
                               tetra_type arg_tetra_type, double, double) {
    _data->type = arg_tetra_type;
    _data->solid = c5host::init_polar(potential_function, x0, y0, z0, level_value, step, angle_step);
    _data->pending.clear();
}

void object3d_base::rotate_around_x_axis(double angle) {
    _data->pending.push_back(c5_rotation{0, 0, angle, 0.0});
}

void object3d_base::rotate_around_y_axis(double angle, double x0) {
    _data->pending.push_back(c5_rotation{1, 0, angle, x0});
}

void object3d_base::bake_rotations() {
    if (_data->pending.empty()) return;
    for (const auto& r : _data->pending) {
        for (auto& t : _data->solid) {
            for (auto& p : t) apply(r, p);
        }
        const std::size_t n = _data->grid.n_points();
        for (std::size_t i = 0; i < n; i++) {
            point p{_data->grid.points[3 * i], _data->grid.points[3 * i + 1], _data->grid.points[3 * i + 2]};
            apply(r, p);
            std::copy(p.begin(), p.end(), _data->grid.points.begin() + 3 * static_cast<std::ptrdiff_t>(i));
        }
    }
    _data->pending.clear();
}

std::array<double, 4> object3d_base::get_boundaries() {
    double x_max = -INFINITY, x_min = INFINITY, y_max = -INFINITY, y_min = INFINITY;
    auto visit = [&](point p) {
        for (const auto& r : _data->pending) apply(r, p);
        x_max = std::max(x_max, p[0]);
        x_min = std::min(x_min, p[0]);
        y_max = std::max(y_max, p[1]);
        y_min = std::min(y_min, p[1]);
    };
    for (const auto& t : _data->solid) {
        for (const auto& p : t) visit(p);
    }
    // only points that cells use count (the reference's tets own copies of their points)
    for (int32_t v : _data->grid.tets) {
        visit({_data->grid.points[3 * static_cast<std::size_t>(v)], _data->grid.points[3 * static_cast<std::size_t>(v) + 1],
               _data->grid.points[3 * static_cast<std::size_t>(v) + 2]});
    }
    return {x_max, x_min, y_max, y_min};
}

object3d_accretion_disk::object3d_accretion_disk(const std::string& filename) {
    read_vtk_file(filename, {"AbsorpCoef", "radEnLooseRate"}); // object3d_accretion_disk.cpp:4
}

object3d_roche_lobe::object3d_roche_lobe(const point& pos_accretor, double dist, double donor_angle_around_y,
                                         double m_accretor, double m_donor, double def_omega) {
    _data->type = tetra_type::solid;
    // the donor rotation is part of the object (object3d_roche_lobe.cpp:48), so it is baked here
    _data->solid = make_roche_lobe(pos_accretor, dist, donor_angle_around_y, m_accretor, m_donor, def_omega);
}

object3d_sphere::object3d_sphere(const point& center, double R) {
    _data->type = tetra_type::solid;
    _data->solid = make_sphere(center, R);
}

void object2d::export_to_vti(const std::string& filename, bool compress, const std::vector<vti_array>& extra) const {
    write_vti(filename, _image.data(), _x, _y, compress ? vti_encoding::zlib_raw : vti_encoding::raw, extra);
}

void image_ref::export_to_vti(const std::string& filename, bool compress) const {
    write_vti(filename, data, x, y, compress);
}

plane::plane(std::size_t res_x, std::size_t res_y, std::vector<object3d_base> objects3d,
             std::vector<double> global_boundaries, render_options options)
    : _objects(std::move(objects3d)), _x(res_x), _y(res_y), _options(std::move(options)) {
    const std::size_t gb = global_boundaries.size();
    if (gb > 0 && gb != 4) throw std::runtime_error("plane initializer. wrong manual boundaries"); // plane.cpp:262-264
    if (_objects.empty()) throw std::runtime_error("plane initializer. empty set of objects to render"); // :269-271
    if (gb == 4) {
        std::copy(global_boundaries.begin(), global_boundaries.end(), _global_boundaries.begin());
    } else { // union of the objects' boxes (plane.cpp:273-285)
        _global_boundaries = _objects[0].get_boundaries();
        for (std::size_t i = 1; i < _objects.size(); i++) {
            const auto b = _objects[i].get_boundaries();
            _global_boundaries[0] = std::max(_global_boundaries[0], b[0]);
            _global_boundaries[1] = std::min(_global_boundaries[1], b[1]);
            _global_boundaries[2] = std::max(_global_boundaries[2], b[2]);
            _global_boundaries[3] = std::min(_global_boundaries[3], b[3]);
        }
    }
    if (_objects[0].get_pointer()->type != tetra_type::transparent || _objects[0].get_pointer()->grid.tets.empty()) {
        throw std::runtime_error("plane initializer. the first object must be the tetrahedral grid");
    }
    std::vector<int32_t> devs(_options.devices.begin(), _options.devices.end());
    c5_ctx* ctx = nullptr;
    const int rc = c5_create(devs.data(), static_cast<int32_t>(devs.size()), &ctx);
    if (rc != C5_OK) throw std::runtime_error(std::string("c5_create: ") + c5_last_error(nullptr));
    _ctx = ctx;
}

plane::~plane() {
    // views still in flight write into _buffers: wait for them before the memory goes away
    for (const auto& pv : _pending) c5_render_wait(_ctx, pv.ticket, nullptr);
    for (const auto& pf : _pending_flux) {
        for (int k = 0; k < pf.n; k++) c5_render_wait(_ctx, pf.tickets[k], nullptr);
    }
    for (auto& b : _buffers) c5_host_unregister(_ctx, b.data());
    c5_destroy(_ctx);
}

void plane::set_views_in_flight(int n) {
    if (!_pending.empty()) throw std::runtime_error("set_views_in_flight: views are in flight");
    check(_ctx, c5_set_views_in_flight(_ctx, n), "c5_set_views_in_flight");
    _in_flight_max = n;
}

void plane::submit_rays() {
    if (!_uploaded) find_intersections();
    if (static_cast<int>(_pending.size()) >= _in_flight_max) {
        throw std::runtime_error("submit_rays: collect a view first (" + std::to_string(_in_flight_max) + " are in flight)");
    }
    if (_free_buffers.empty()) { // one more page-locked image, kept for the life of the plane
        _buffers.emplace_back(_x * _y * 2);
        check(_ctx, c5_host_register(_ctx, _buffers.back().data(), _buffers.back().size() * sizeof(double)), "c5_host_register");
        _free_buffers.push_back(_buffers.size() - 1);
    }
    const std::size_t b = _free_buffers.back();
    std::uint64_t ticket = 0;
    check(_ctx, c5_render_submit(_ctx, &_view, _buffers[b].data(), &ticket), "c5_render_submit");
    _free_buffers.pop_back();
    _pending.push_back({ticket, b});
}

void plane::collect_rays(const std::function<void(const image_ref&)>& consume) {
    if (_pending.empty()) throw std::runtime_error("collect_rays: nothing was submitted");
    const pending_view pv = _pending.front();
    _pending.erase(_pending.begin());
    struct give_back { // also when the wait or the consumer throws
        std::vector<std::size_t>& pool;
        std::size_t b;
        ~give_back() { pool.push_back(b); }
    } guard{_free_buffers, pv.buffer};
    check(_ctx, c5_render_wait(_ctx, pv.ticket, &_stats), "c5_render_wait");
    consume(image_ref{_buffers[pv.buffer].data(), _x, _y});
}

object2d plane::collect_rays() {
    std::vector<double> copy;
    collect_rays([&](const image_ref& im) { copy.assign(im.data, im.data + im.x * im.y * 2); });
    return object2d{std::move(copy), _x, _y};
}

void plane::submit_flux() {
    if (!_uploaded) find_intersections();
    if (static_cast<int>(_pending_flux.size()) >= flux_frames_in_flight()) {
        throw std::runtime_error("submit_flux: collect a frame first (" + std::to_string(_pending_flux.size()) + " are in flight)");
    }
    pending_flux pf{{0, 0}, 0, std::vector<double>(2 + 2 * _options.channels.size())};
    check(_ctx, c5_render_flux_submit(_ctx, &_view, 0, nullptr, pf.total.data(), &pf.tickets[0]), "c5_render_flux_submit");
    pf.n = 1;
    if (!_options.channels.empty()) {
        const int rc = c5_render_flux_submit(_ctx, &_view, 1, nullptr, pf.total.data() + 2, &pf.tickets[1]);
        if (rc != C5_OK) {
            const std::string text = c5_last_error(_ctx);
            c5_render_wait(_ctx, pf.tickets[0], nullptr); // the first view writes into pf.total
            throw std::runtime_error("c5_render_flux_submit failed (" + std::to_string(rc) + "): " + text);
        }
        pf.n = 2;
    }
    _pending_flux.push_back(std::move(pf)); // moving the vector keeps its buffer where the views write
}

plane::frame_flux plane::collect_flux() {
    if (_pending_flux.empty()) throw std::runtime_error("collect_flux: nothing was submitted");
    pending_flux pf = std::move(_pending_flux.front());
    _pending_flux.erase(_pending_flux.begin());
    c5_stats st{};
    const int rc = c5_render_wait(_ctx, pf.tickets[0], &st);
    const std::string text = rc == C5_OK ? "" : c5_last_error(_ctx);
    const int rc_ch = pf.n > 1 ? c5_render_wait(_ctx, pf.tickets[1], nullptr) : C5_OK; // waited for also when the first failed
    if (rc != C5_OK) throw std::runtime_error("c5_render_wait failed (" + std::to_string(rc) + "): " + text);
    check(_ctx, rc_ch, "c5_render_wait");
    _stats = st;
    return frame_flux{st, std::move(pf.total)};
}

void plane::find_intersections() {
    object_data& grid = *_objects[0].get_pointer();
    const auto& alpha = grid.grid.cell_scalars.at(grid.labels[0]);
    const auto& q = grid.grid.cell_scalars.at(grid.labels[1]);
    check(_ctx, c5_upload_mesh(_ctx, grid.grid.points.data(), static_cast<int64_t>(grid.grid.n_points()),
                               grid.grid.tets.data(), static_cast<int64_t>(grid.grid.n_tets()), alpha.data(), q.data()),
          "c5_upload_mesh");
    check(_ctx, c5_clear_solids(_ctx), "c5_clear_solids");
    if (!_options.channels.empty()) { // channel-major, in the file's tet order
        const std::size_t n_t = grid.grid.n_tets(), n = _options.channels.size();
        std::vector<double> ch_alpha(n * n_t), ch_q(n * n_t);
        for (std::size_t c = 0; c < n; c++) {
            for (int k = 0; k < 2; k++) {
                const auto it = grid.grid.cell_scalars.find(_options.channels[c][static_cast<std::size_t>(k)]);
                if (it == grid.grid.cell_scalars.end() || it->second.size() != n_t) {
                    throw std::runtime_error("no cell scalar named '" + _options.channels[c][static_cast<std::size_t>(k)] + "'");
                }
                std::copy(it->second.begin(), it->second.end(), (k ? ch_q : ch_alpha).begin() + static_cast<std::ptrdiff_t>(c * n_t));
            }
        }
        check(_ctx, c5_upload_channels(_ctx, ch_alpha.data(), ch_q.data(), static_cast<int32_t>(n)), "c5_upload_channels");
    }

    // the grid's recorded rotations define the view; solids that recorded the same list follow it
    // on the device, the others are baked on the host and uploaded as static
    std::memset(&_view, 0, sizeof(_view));
    _view.res_x = static_cast<int32_t>(_x);
    _view.res_y = static_cast<int32_t>(_y);
    for (int k = 0; k < 4; k++) _view.window[k] = _global_boundaries[static_cast<std::size_t>(k)];
    if (grid.pending.size() > C5_MAX_ROT) throw std::runtime_error("too many recorded rotations");
    _view.n_rot = static_cast<int32_t>(grid.pending.size());
    for (std::size_t k = 0; k < grid.pending.size(); k++) _view.rot[k] = grid.pending[k];
    _view.alpha_limit = _options.alpha_limit;
    _view.precision = _options.precision;
    _view.round_through_float = 1;
    _view.use_solids = 1;

    for (std::size_t i = 1; i < _objects.size(); i++) {
        object_data& obj = *_objects[i].get_pointer();
        if (obj.type != tetra_type::solid) throw std::runtime_error("only the first object may be transparent");
        int follows = 0;
        std::vector<tet_points> baked;
        const std::vector<tet_points>* pts = &obj.solid;
        if (!obj.pending.empty()) {
            if (same_rotations(obj.pending, grid.pending)) {
                follows = 1;
            } else {
                baked = obj.solid;
                for (const auto& r : obj.pending) {
                    for (auto& t : baked) {
                        for (auto& p : t) apply(r, p);
                    }
                }
                pts = &baked;
            }
        }
        check(_ctx, c5_upload_solids(_ctx, &(*pts)[0][0][0], static_cast<int64_t>(pts->size()), follows),
              "c5_upload_solids");
    }
    check(_ctx, c5_mesh_info_get(_ctx, &_info), "c5_mesh_info_get");
    _uploaded = true;
}

void plane::set_view_rotations(const std::vector<c5_rotation>& rotations) {
    if (rotations.size() > C5_MAX_ROT) throw std::runtime_error("too many rotations");
    if (!_uploaded) find_intersections();
    _view.n_rot = static_cast<int32_t>(rotations.size());
    for (std::size_t k = 0; k < rotations.size(); k++) _view.rot[k] = rotations[k];
}

object2d plane::trace_rays(tetra_value value_alpha, tetra_value value_Q) {
    if (value_alpha != tetra_value::alpha || value_Q != tetra_value::Q) {
        throw std::runtime_error("trace_rays: the scalar roles are fixed to (alpha, Q)");
    }
    if (!_uploaded) find_intersections();
    if (_x == 0 || _y == 0) throw std::runtime_error("critical error. empty plane"); // plane.cpp:151-153
    std::vector<double> image(_x * _y * 2);
    check(_ctx, c5_render(_ctx, &_view, image.data(), &_stats), "c5_render");
    return object2d{std::move(image), _x, _y};
}

std::vector<std::vector<double>> plane::trace_channels() {
    if (!_uploaded) find_intersections();
    const std::size_t n = _options.channels.size(), n_pix = _x * _y;
    std::vector<double> all(n_pix * n * 2);
    check(_ctx, c5_render_channels(_ctx, &_view, all.data(), nullptr, nullptr, nullptr), "c5_render_channels");
    std::vector<std::vector<double>> out(n, std::vector<double>(n_pix * 2));
    for (std::size_t p = 0; p < n_pix; p++) {
        for (std::size_t c = 0; c < n; c++) {
            out[c][2 * p] = all[(p * n + c) * 2];
            out[c][2 * p + 1] = all[(p * n + c) * 2 + 1];
        }
    }
    return out;
}

} // namespace c5host
