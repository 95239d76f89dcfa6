// scene.hpp — host-side mirror of the reference's objects for the ray pass, backed by the C ABI.
//
// Same class and method names as the reference so main() reads like main.cpp:96-137:
//   object3d_base / object3d_accretion_disk / object3d_roche_lobe / object3d_sphere
//       (object3d_base.hpp:22-42 and the three derived headers)
//   plane(res_x, res_y, objects, boundaries), find_intersections(), trace_rays(alpha, Q)
//       (plane.hpp:16-68)
//   object2d::export_to_vti (object2d.hpp:13-23)
// What differs is where the work happens: an object keeps shared points + connectivity (not
// per-tet point copies), rotate_around_* only RECORDS the rotation (the device applies the list
// per view, once per unique vertex), find_intersections() uploads the scene and builds the
// device topology, trace_rays() runs the per-view kernels.
#pragma once

#include <array>
#include <cstddef>
#include <cstdint>
#include <functional>
#include <memory>
#include <string>
#include <vector>

#include "../../include/c5gpu.h"
#include "config.hpp"
#include "solids.hpp"
#include "vti_writer.hpp"
#include "vtk_reader.hpp"

namespace c5host {

enum class tetra_value : std::size_t { alpha = 0, solid_color = 0, Q = 1 }; // tetra.hpp:8
enum class tetra_type { transparent = 0, solid = 1 };                       // tetra.hpp:10

struct object_data {
    tetra_type type = tetra_type::transparent;
    tet_grid grid;                        // transparent objects: shared points + connectivity + scalars
    std::array<std::string, 2> labels{};  // scalar names for {alpha, Q}
    std::vector<tet_points> solid;        // solid objects: tet soup
    std::vector<c5_rotation> pending;     // rotations recorded since the geometry was last baked
};

class object3d_base {
public:
    object3d_base() = default;
    virtual ~object3d_base() = default;

    void read_vtk_file(const std::string& filename, const std::vector<std::string>& scalar_labels);
    void init_polar(const std::function<double(const point&)>& potential_function, double x0, double y0, double z0,
                    double level_value, double step, double angle_step,
                    tetra_type arg_tetra_type = tetra_type::transparent, double tetra_v1 = 0, double tetra_v2 = 0);
    std::shared_ptr<object_data> get_pointer() { return _data; }

    virtual void rotate_around_x_axis(double angle);
    virtual void rotate_around_y_axis(double angle, double x0);
    // {x_max, x_min, y_max, y_min} of the geometry with the recorded rotations applied
    virtual std::array<double, 4> get_boundaries();

protected:
    void bake_rotations(); // applies and clears the recorded rotations on the host
    std::shared_ptr<object_data> _data = std::make_shared<object_data>();
};

class object3d_accretion_disk : public object3d_base {
public:
    object3d_accretion_disk() = default;
    explicit object3d_accretion_disk(const std::string& filename);
};

class object3d_roche_lobe : public object3d_base {
public:
    object3d_roche_lobe(const point& pos_accretor, double dist, double donor_angle_around_y, double m_accretor,
                        double m_donor, double def_omega);
};

class object3d_sphere : public object3d_base {
public:
    object3d_sphere(const point& center, double R);
};

class object2d {
public:
    object2d(std::vector<double> image, std::size_t res_x, std::size_t res_y)
        : _image(std::move(image)), _x(res_x), _y(res_y) {}
    // extra: further arrays beside ImageScalars (course --channels)
    void export_to_vti(const std::string& filename, bool compress = false, const std::vector<vti_array>& extra = {}) const;
    const std::vector<double>& data() const { return _image; } // res_y * res_x * {tau, I}, x fastest
    std::size_t get_x() const { return _x; }
    std::size_t get_y() const { return _y; }

private:
    std::vector<double> _image;
    std::size_t _x, _y;
};

// An image that lives in someone else's buffer (a submitted view's page-locked memory).
struct image_ref {
    const double* data; // res_y * res_x * {tau, I}, x fastest
    std::size_t x, y;
    void export_to_vti(const std::string& filename, bool compress = false) const;
};

struct render_options {
    std::vector<int> devices{0};
    double alpha_limit = 2.5; // the reference reads app::instance().config.limit_alpha_value (line.cpp:204)
    int precision = 64;
    std::vector<std::array<std::string, 2>> channels; // (alpha, Q) cell scalar names uploaded as channels
};

class plane {
public:
    plane() = delete;
    plane(std::size_t res_x, std::size_t res_y, std::vector<object3d_base> objects3d,
          std::vector<double> global_boundaries = {}, render_options options = {});
    ~plane();
    plane(const plane&) = delete;
    plane& operator=(const plane&) = delete;

    void find_intersections();
    object2d trace_rays(tetra_value value_alpha, tetra_value value_Q);
    // The pairs of render_options::channels for the same view, in one walk (c5_render_channels):
    // one (res_y, res_x, 2) image per channel.
    std::vector<std::vector<double>> trace_channels();
    // Sweeps: replace the recorded view rotations (grid and view-following solids) without
    // re-uploading anything; the next trace_rays() renders the new view in milliseconds.
    void set_view_rotations(const std::vector<c5_rotation>& rotations);
    // Sweeps, pipelined (c5_render_submit / c5_render_wait): submit_rays() enqueues the view with the
    // current rotations and returns at once; collect_rays() returns the OLDEST submitted view's image.
    // Up to `views_in_flight` (default 3) may be submitted before the first is collected, so the device
    // renders frames k+1, k+2 while the caller writes frame k to disk.
    void set_views_in_flight(int n);
    int views_in_flight() const { return _in_flight_max; }
    void submit_rays();
    // `consume` sees the image in the page-locked buffer the device wrote (no copy); the buffer is
    // handed back to the pool when it returns.
    void collect_rays(const std::function<void(const image_ref&)>& consume);
    object2d collect_rays(); // the same, as a copy
    // Light curves, pipelined (c5_render_flux_submit): submit_flux() enqueues the current view as a flux
    // view of the cells' own fields and, with render_options::channels, one more over the channels; no
    // image leaves the device. collect_flux() returns the OLDEST submitted frame's sums. A frame takes
    // one lane per flux view, so flux_frames_in_flight() frames may be submitted before the first is
    // collected.
    struct frame_flux {
        c5_stats stats;            // of the cells' own view
        std::vector<double> total; // {tau, I} sums of the cells' fields, then of each channel
    };
    void submit_flux();
    frame_flux collect_flux();
    int flux_frames_in_flight() const { return _in_flight_max / (_options.channels.empty() ? 1 : 2); }
    std::size_t pending_views() const { return _pending.size(); }
    std::size_t count_all_intersections() const { return static_cast<std::size_t>(_stats.tet_steps); }
    std::size_t get_x() const { return _x; }
    std::size_t get_y() const { return _y; }
    const c5_stats& stats() const { return _stats; }
    const c5_mesh_info& mesh_info() const { return _info; }

private:
    std::vector<object3d_base> _objects;
    std::array<double, 4> _global_boundaries{};
    std::size_t _x{}, _y{};
    render_options _options;
    c5_ctx* _ctx = nullptr;
    c5_view _view{};
    c5_stats _stats{};
    c5_mesh_info _info{};
    bool _uploaded = false;
    // page-locked image buffers of the submitted views, oldest first
    struct pending_view {
        std::uint64_t ticket;
        std::size_t buffer;
    };
    std::vector<std::vector<double>> _buffers; // registered with the context (c5_host_register)
    std::vector<std::size_t> _free_buffers;
    std::vector<pending_view> _pending;
    struct pending_flux {
        std::uint64_t tickets[2];
        int n; // flux views of the frame
        std::vector<double> total; // written by c5_render_wait
    };
    std::vector<pending_flux> _pending_flux;
    int _in_flight_max = 3;
};

} // namespace c5host
