// host_abi.cpp — C entry points into the HOST-side pieces (solid generators, VTK reader, .vti
// reader/writer, CLI parser) so tests can drive them from Python without a GPU. Built into
// course5_b200/libc5host.so; contains no device code and no ray pass.
#include <cstring>
#include <sstream>
#include <string>
#include <vector>

#include "cli.hpp"
#include "config.hpp"
#include "solids.hpp"
#include "vti_writer.hpp"
#include "vtk_reader.hpp"

using namespace c5host;

namespace {
thread_local std::string g_err;
template <class Fn>
long long guarded(Fn&& fn) {
    try {
        return fn();
    } catch (const std::exception& e) {
        g_err = e.what();
        return -1;
    }
}
std::vector<tet_points> g_solids[2];
tet_grid g_grid;
} // namespace

extern "C" {

const char* c5host_last_error(void) { return g_err.c_str(); }

// which: 0 = Roche lobe (with donor angle, in units of pi), 1 = sphere. Returns the tet count and
// keeps the result for c5host_solids_copy.
long long c5host_solids_make(int which, double donor_angle_pi) {
    return guarded([&]() -> long long {
        g_solids[which ? 1 : 0] = which ? make_sphere({ACC_X0, ACC_Y0, ACC_Z0}, ACC_DISK_R)
                                        : make_roche_lobe({ACC_X0, ACC_Y0, ACC_Z0}, L, donor_angle_pi * PI, M_ACC,
                                                          M_DONOR, OMEGA);
        return static_cast<long long>(g_solids[which ? 1 : 0].size());
    });
}

void c5host_solids_copy(int which, double* out) {
    const auto& v = g_solids[which ? 1 : 0];
    if (!v.empty()) std::memcpy(out, &v[0][0][0], v.size() * sizeof(tet_points));
}

// Reads a legacy VTK file; returns the tet count (points via c5host_grid_sizes / _copy).
long long c5host_read_vtk(const char* filename) {
    return guarded([&]() -> long long {
        g_grid = read_legacy_vtk(filename);
        return static_cast<long long>(g_grid.n_tets());
    });
}
long long c5host_grid_points(void) { return static_cast<long long>(g_grid.n_points()); }
int c5host_grid_has_scalar(const char* name) { return g_grid.cell_scalars.count(name) ? 1 : 0; }
void c5host_grid_copy(double* points, int32_t* tets, const char* alpha_name, double* alpha, const char* q_name,
                      double* q) {
    std::memcpy(points, g_grid.points.data(), g_grid.points.size() * sizeof(double));
    std::memcpy(tets, g_grid.tets.data(), g_grid.tets.size() * sizeof(int32_t));
    if (alpha && g_grid.cell_scalars.count(alpha_name)) {
        const auto& a = g_grid.cell_scalars[alpha_name];
        std::memcpy(alpha, a.data(), a.size() * sizeof(double));
    }
    if (q && g_grid.cell_scalars.count(q_name)) {
        const auto& b = g_grid.cell_scalars[q_name];
        std::memcpy(q, b.data(), b.size() * sizeof(double));
    }
}

long long c5host_write_vti(const char* filename, const double* image, long long res_x, long long res_y, int compress) {
    return guarded([&]() -> long long {
        write_vti(filename, image, static_cast<std::size_t>(res_x), static_cast<std::size_t>(res_y),
                  compress == 2 ? vti_encoding::zlib_base64 : compress == 1 ? vti_encoding::zlib_raw : vti_encoding::raw);
        return 0;
    });
}

// write_vti with n_extra further arrays: names[k] and data[k] (res_y * res_x * 2 doubles each).
long long c5host_write_vti_arrays(const char* filename, const double* image, long long res_x, long long res_y, int compress,
                                  int n_extra, const char* const* names, const double* const* data) {
    return guarded([&]() -> long long {
        std::vector<vti_array> extra;
        for (int k = 0; k < n_extra; k++) extra.push_back(vti_array{names[k], data[k]});
        write_vti(filename, image, static_cast<std::size_t>(res_x), static_cast<std::size_t>(res_y),
                  compress == 2 ? vti_encoding::zlib_base64 : compress == 1 ? vti_encoding::zlib_raw : vti_encoding::raw,
                  extra);
        return 0;
    });
}

// Returns the number of doubles (res_x * res_y * comps), fills dims; call again with `out` to copy.
// `name`: the PointData array (NULL or empty: the first one, ImageScalars).
long long c5host_read_vti_array(const char* filename, const char* name, long long* res_x, long long* res_y,
                                long long* comps, double* out) {
    return guarded([&]() -> long long {
        std::size_t x, y, c;
        double* img = nullptr;
        read_vti(filename, x, y, c, img, name ? name : "");
        *res_x = static_cast<long long>(x);
        *res_y = static_cast<long long>(y);
        *comps = static_cast<long long>(c);
        if (out) std::memcpy(out, img, x * y * c * sizeof(double));
        delete[] img;
        return static_cast<long long>(x * y * c);
    });
}

long long c5host_read_vti(const char* filename, long long* res_x, long long* res_y, long long* comps, double* out) {
    return guarded([&]() -> long long {
        std::size_t x, y, c;
        double* img = nullptr;
        read_vti(filename, x, y, c, img);
        *res_x = static_cast<long long>(x);
        *res_y = static_cast<long long>(y);
        *comps = static_cast<long long>(c);
        if (out) std::memcpy(out, img, x * y * c * sizeof(double));
        delete[] img;
        return static_cast<long long>(x * y * c);
    });
}

// Parses a command line; result: 0 run, 1 exit 0 (help / missing -f -d), 2 error. `text` receives
// what was printed (truncated to cap), `values` = {res_x, res_y, X, Y, D, I, alpha_limit, threads}.
int c5host_parse_cli(int argc, char** argv, char* text, int cap, double* values, char* file, char* dest, int scap) {
    config_str cfg;
    std::ostringstream out;
    const cli_result r = program_options(argc, argv, cfg, out);
    const std::string s = out.str();
    if (text && cap > 0) {
        std::strncpy(text, s.c_str(), static_cast<size_t>(cap) - 1);
        text[cap - 1] = 0;
    }
    if (values) {
        values[0] = static_cast<double>(cfg.resolution_x);
        values[1] = static_cast<double>(cfg.resolution_y);
        values[2] = cfg.angle_around_x;
        values[3] = cfg.angle_around_y;
        values[4] = cfg.donor_angle;
        values[5] = cfg.system_initial_angle_around_y;
        values[6] = cfg.limit_alpha_value;
        values[7] = cfg.threads;
    }
    if (file && scap > 0) {
        std::strncpy(file, cfg.file.c_str(), static_cast<size_t>(scap) - 1);
        file[scap - 1] = 0;
    }
    if (dest && scap > 0) {
        std::strncpy(dest, cfg.destination.c_str(), static_cast<size_t>(scap) - 1);
        dest[scap - 1] = 0;
    }
    return r == cli_result::run ? 0 : (r == cli_result::exit_ok ? 1 : 2);
}

} // extern "C"
