// config.hpp — run configuration and the physical constants of the binary system.
// Values are the contract of /root/reference/project/include/config.hpp:7-74 and must stay
// bit-identical (they feed the solid-object generators and the view rotations).
#pragma once

#include <array>
#include <cstddef>
#include <limits>
#include <string>
#include <vector>

namespace c5host {

// What the CLI fills (main.cpp:44-66); passed by value to whoever needs it — there is no global.
struct config_str {
    std::string file;
    std::string destination;
    int threads = 1;                           // -j: accepted for the host baseline, unused by the GPU path
    std::size_t resolution_x = 1200;           // main.cpp:27
    std::size_t resolution_y = 900;            // main.cpp:28
    double angle_around_x = 0;                 // -X, units of pi
    double angle_around_y = 0;                 // -Y
    double donor_angle = 0;                    // -D
    double system_initial_angle_around_y = 0;  // -I
    double limit_alpha_value = 2.5;            // --alpha_limit
    double acc_disk_solid_color = std::numeric_limits<double>::quiet_NaN();
    double roche_lobe_solid_color = std::numeric_limits<double>::quiet_NaN();
    // additions (not in the reference)
    std::string devices = "0";                 // --devices 0,1,...  CUDA ordinals
    bool stats = false;                        // --stats: one JSON line with per-phase timings
    int precision = 64;
    int frames = 1;                            // --frames N: in-process sweep of -Y (replaces utility/rotate_traces.py)
    double sweep_y_to = 2.0;                   // --sweep_y_to: end angle (exclusive), units of pi
    std::vector<std::array<std::string, 2>> channels; // --channels A:Q,...: (alpha, Q) cell array names
    bool light_curve = false;                  // --light_curve: the destination is a CSV of per-frame sums, no .vti
};

constexpr double PI = 3.14159265358979323846;  // config.hpp:45
constexpr double L = 0.945;                    // distance between the stars, R_sol (config.hpp:50)
constexpr double ACC_X0 = 1;                   // accretor position (config.hpp:55-57)
constexpr double ACC_Y0 = 0;
constexpr double ACC_Z0 = 0;
constexpr double ACC_DISK_R = 0.02;            // config.hpp:58
constexpr double M_ACC = 0.73;                 // config.hpp:59
constexpr double M_DONOR = 0.1;                // config.hpp:64
constexpr long double G_SOL = 132700000000000000000.; // config.hpp:69 (long double on purpose)
constexpr double OMEGA = 2 * PI * 10000;       // config.hpp:74

// {x_max, x_min, y_max, y_min}: the hard-coded view window (main.cpp:83)
constexpr double DOMAIN[4] = {2.2, -0.2, 0.9, -0.9};

} // namespace c5host
