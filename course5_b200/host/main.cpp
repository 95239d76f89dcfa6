// main.cpp — the `course` executable: same flags, same stdout lines, same .vti as the reference's
// main (main.cpp:73-141), with the OpenMP loops replaced by the B200 ray pass behind the C ABI.
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <fstream>
#include <iostream>
#include <sstream>
#include <thread>

#include "cli.hpp"
#include "config.hpp"
#include "scene.hpp"

using namespace c5host;

namespace {

std::vector<int> parse_devices(const std::string& s) {
    std::vector<int> out;
    std::stringstream ss(s);
    std::string item;
    while (std::getline(ss, item, ',')) {
        if (!item.empty()) out.push_back(std::stoi(item));
    }
    if (out.empty()) out.push_back(0);
    return out;
}

std::string g17(double v) { // %.17g: parses back to the same double
    char buf[32];
    std::snprintf(buf, sizeof(buf), "%.17g", v);
    return buf;
}

long long ms_between(std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
    return std::chrono::duration_cast<std::chrono::milliseconds>(b - a).count();
}

} // namespace

int main(int argc, char** argv) {
    config_str config;
    const cli_result parsed = program_options(argc, argv, config, std::cout);
    if (parsed == cli_result::exit_ok) return 0;
    if (parsed == cli_result::exit_error) return 1;

    const std::vector<double> domain(DOMAIN, DOMAIN + 4); // {x_max, x_min, y_max, y_min}, main.cpp:83

    // banner, main.cpp:85-92
    std::cout << "Defined grid resolution: " << config.resolution_x << "x" << config.resolution_y << std::endl;
    std::cout << "Source file: " << config.file << std::endl;
    std::cout << "Number of parallel threads: " << config.threads << std::endl;
    std::cout << "Initial rotate angle of roche lobe: " << config.donor_angle << " Pi" << std::endl;
    std::cout << "Plane angle around x: " << config.angle_around_x << " Pi" << std::endl;
    std::cout << "Plane angle around y: " << config.angle_around_y << " Pi" << std::endl;
    std::cout << "Initial system angle around y: " << config.system_initial_angle_around_y << " Pi" << std::endl;
    std::cout << "Limit alpha value: " << config.limit_alpha_value << std::endl;

    try {
        auto t1 = std::chrono::steady_clock::now();
        const double make_perpendicular_to_y_angle = -config.system_initial_angle_around_y * PI + PI / 2.;
        const double last_angle = -make_perpendicular_to_y_angle + config.angle_around_x * PI;

        // the file is read on its own thread while the solids are generated (main.cpp:98-108,117)
        object3d_accretion_disk acc_disk{};
        std::string load_error;
        std::thread loader([&]() {
            try {
                acc_disk = object3d_accretion_disk{config.file};
                acc_disk.rotate_around_x_axis(make_perpendicular_to_y_angle);
                acc_disk.rotate_around_y_axis(config.angle_around_y * PI, ACC_X0);
                acc_disk.rotate_around_x_axis(last_angle);
            } catch (const std::exception& e) {
                load_error = e.what();
            }
        });

        auto roche_lobe = object3d_roche_lobe{{ACC_X0, ACC_Y0, ACC_Z0}, L, config.donor_angle * PI, M_ACC, M_DONOR, OMEGA};
        roche_lobe.rotate_around_x_axis(make_perpendicular_to_y_angle);
        roche_lobe.rotate_around_y_axis(config.angle_around_y * PI, ACC_X0);
        roche_lobe.rotate_around_x_axis(last_angle);

        auto acc_sphere = object3d_sphere{{ACC_X0, ACC_Y0, ACC_Z0}, ACC_DISK_R}; // not rotated, main.cpp:116
        loader.join();
        if (!load_error.empty()) throw std::runtime_error(load_error);
        for (const auto& pair : config.channels) {
            for (const std::string& name : pair) {
                if (!acc_disk.get_pointer()->grid.cell_scalars.count(name)) {
                    throw std::runtime_error(config.file + ": no cell scalar named '" + name + "' (--channels)");
                }
            }
        }
        auto t2 = std::chrono::steady_clock::now();
        std::cout << "Loading data with VTK lib and other preparations completed in " << ms_between(t1, t2) << " ms. "
                  << std::endl;

        render_options options;
        options.devices = parse_devices(config.devices);
        options.alpha_limit = config.limit_alpha_value;
        options.precision = config.precision;
        options.channels = config.channels;

        t1 = std::chrono::steady_clock::now();
        plane base_plane{config.resolution_x, config.resolution_y, {acc_disk, roche_lobe, acc_sphere}, domain, options};
        base_plane.find_intersections();
        // the view of sweep frame k (frame 0 is the view the flags describe)
        auto y_of = [&](int k) {
            return config.angle_around_y + (config.sweep_y_to - config.angle_around_y) * k / std::max(config.frames, 1);
        };
        auto rotations_of = [&](int k) {
            return std::vector<c5_rotation>{c5_rotation{0, 0, make_perpendicular_to_y_angle, 0.0},
                                            c5_rotation{1, 0, y_of(k) * PI, ACC_X0}, c5_rotation{0, 0, last_angle, 0.0}};
        };

        if (config.light_curve) {
            // --light_curve: every frame through the pipelined flux calls; only its sums leave the device
            std::ofstream csv(config.destination);
            if (!csv) throw std::runtime_error("cannot write " + config.destination);
            csv << "frame,Y_pi,hit_pixels,solid_pixels,tau_sum,I_sum";
            for (const auto& pair : config.channels) csv << "," << pair[0] << ":" << pair[1] << "_tau_sum," << pair[0] << ":" << pair[1] << "_I_sum";
            csv << "\n";
            if (!config.channels.empty()) base_plane.set_views_in_flight(4); // two flux views per frame
            const int frames = config.frames < 1 ? 1 : config.frames;
            const int ahead = base_plane.flux_frames_in_flight();
            for (int k = 0; k < frames + ahead; k++) {
                if (k - ahead >= 0) {
                    const plane::frame_flux f = base_plane.collect_flux();
                    csv << (k - ahead) << "," << g17(y_of(k - ahead)) << "," << f.stats.hit_pixels << "," << f.stats.solid_pixels;
                    for (double v : f.total) csv << "," << g17(v);
                    csv << "\n";
                }
                if (k < frames) {
                    base_plane.set_view_rotations(rotations_of(k));
                    base_plane.submit_flux();
                }
            }
            csv.close();
            if (!csv) throw std::runtime_error("cannot write " + config.destination);
            std::cout << "Light curve of " << frames << " frames completed in "
                      << ms_between(t1, std::chrono::steady_clock::now()) << " ms. " << std::endl;
        } else {
            object2d result = base_plane.trace_rays(tetra_value::alpha, tetra_value::Q);
            // --channels: the named pairs in one further walk, written beside ImageScalars as "A:Q"
            const std::vector<std::vector<double>> channels =
                config.channels.empty() ? std::vector<std::vector<double>>{} : base_plane.trace_channels();
            t2 = std::chrono::steady_clock::now();
            std::cout << "Ray-tracing completed in " << ms_between(t1, t2) << " ms. " << std::endl;

            if (config.frames <= 1) {
                std::vector<vti_array> extra;
                for (std::size_t c = 0; c < channels.size(); c++) {
                    extra.push_back(vti_array{config.channels[c][0] + ":" + config.channels[c][1], channels[c].data()});
                }
                result.export_to_vti(config.destination, false, extra);
            } else {
                // in-process sweep: the scene stays on the device, only the rotations change
                std::string stem = config.destination, ext = ".vti";
                const auto dot = stem.rfind('.');
                if (dot != std::string::npos) {
                    ext = stem.substr(dot);
                    stem = stem.substr(0, dot);
                }
                const auto t3 = std::chrono::steady_clock::now();
                // Frame 0 is the view just rendered. The others go through the pipelined calls: up to three
                // views are in flight on the device while this thread writes the previous frame's file.
                result.export_to_vti(stem + "_0" + ext);
                const int ahead = base_plane.views_in_flight();
                for (int k = 1; k < config.frames + ahead; k++) {
                    if (k - ahead >= 1) {
                        base_plane.collect_rays([&](const image_ref& frame) { frame.export_to_vti(stem + "_" + std::to_string(k - ahead) + ext); });
                    }
                    if (k < config.frames) {
                        base_plane.set_view_rotations(rotations_of(k));
                        base_plane.submit_rays();
                    }
                }
                std::cout << "Sweep of " << config.frames << " frames completed in "
                          << ms_between(t3, std::chrono::steady_clock::now()) << " ms. " << std::endl;
            }
        }
        std::cout << "Result exported. Calculations completed." << std::endl;

        if (config.stats) {
            const c5_stats& s = base_plane.stats();
            const c5_mesh_info& m = base_plane.mesh_info();
            std::cout << "{\"pixels\": " << s.pixels << ", \"tet_steps\": " << s.tet_steps << ", \"hit_pixels\": "
                      << s.hit_pixels << ", \"solid_pixels\": " << s.solid_pixels << ", \"ms_rotate\": " << s.ms_rotate
                      << ", \"ms_bvh\": " << s.ms_bvh << ", \"ms_mask\": " << s.ms_mask << ", \"ms_walk\": " << s.ms_walk
                      << ", \"ms_gather\": " << s.ms_gather << ", \"ms_d2h\": " << s.ms_d2h << ", \"ms_total\": "
                      << s.ms_total << ", \"n_devices\": " << s.n_devices << ", \"n_tets\": " << m.n_tets
                      << ", \"n_boundary_faces\": " << m.n_boundary_faces << ", \"device_bytes\": " << m.device_bytes
                      << "}" << std::endl;
        }
    } catch (const std::exception& e) {
        std::cerr << "course: " << e.what() << std::endl;
        return 2;
    }
    return 0;
}
