// cli.cpp — see cli.hpp.
#include "cli.hpp"

#include <algorithm>
#include <array>
#include <cstdlib>
#include <iostream>
#include <stdexcept>
#include <thread>
#include <vector>

namespace c5host {

namespace {

struct option {
    const char* long_name;
    char short_name; // 0 = none
    bool takes_value;
};

const option kOptions[] = {
    {"help", 'h', false},          {"file", 'f', true},           {"destination", 'd', true},
    {"threads", 'j', true},        {"resolution_x", 'x', true},   {"resolution_y", 'y', true},
    {"angle_around_x", 'X', true}, {"angle_around_y", 'Y', true}, {"donor_angle", 'D', true},
    {"initial_system_angle", 'I', true}, {"alpha_limit", 0, true},
    // additions of this build (absent from the reference)
    {"devices", 0, true},          {"stats", 0, false},           {"precision", 0, true},
    {"frames", 0, true},           {"sweep_y_to", 0, true},       {"channels", 0, true},
    {"light_curve", 0, false},
};

// --channels A:Q[,A:Q...]: pairs of CELL_DATA array names, at most C5_MAX_CHANNELS (8)
std::vector<std::array<std::string, 2>> parse_channels(const std::string& value) {
    std::vector<std::array<std::string, 2>> out;
    std::size_t at = 0;
    while (at <= value.size()) {
        const std::size_t comma = std::min(value.find(',', at), value.size());
        const std::string item = value.substr(at, comma - at);
        const std::size_t colon = item.find(':');
        if (colon == std::string::npos || colon == 0 || colon + 1 == item.size() ||
            item.find(':', colon + 1) != std::string::npos) {
            throw std::runtime_error("--channels: '" + item + "' is not of the form ALPHA:Q");
        }
        out.push_back({item.substr(0, colon), item.substr(colon + 1)});
        at = comma + 1;
    }
    if (out.size() > 8) throw std::runtime_error("--channels: at most 8 channels");
    return out;
}

const option* find_long(const std::string& name, std::string& err) {
    const option* exact = nullptr;
    std::vector<const option*> prefixed;
    for (const auto& o : kOptions) {
        const std::string ln = o.long_name;
        if (ln == name) exact = &o;
        if (ln.rfind(name, 0) == 0) prefixed.push_back(&o);
    }
    if (exact) return exact;
    if (prefixed.size() == 1) return prefixed[0];
    err = prefixed.empty() ? "unrecognised option '--" + name + "'" : "option '--" + name + "' is ambiguous";
    return nullptr;
}

const option* find_short(char c) {
    for (const auto& o : kOptions) {
        if (o.short_name && o.short_name == c) return &o;
    }
    return nullptr;
}

double to_double(const std::string& opt, const std::string& v) {
    char* end = nullptr;
    const double d = std::strtod(v.c_str(), &end);
    if (v.empty() || end != v.c_str() + v.size()) {
        throw std::runtime_error("the argument ('" + v + "') for option '--" + opt + "' is invalid");
    }
    return d;
}

long long to_integer(const std::string& opt, const std::string& v) {
    char* end = nullptr;
    const long long d = std::strtoll(v.c_str(), &end, 10);
    if (v.empty() || end != v.c_str() + v.size()) {
        throw std::runtime_error("the argument ('" + v + "') for option '--" + opt + "' is invalid");
    }
    return d;
}

} // namespace

void print_usage(std::ostream& out) {
    // the text Boost prints for the reference's options_description (readme.md:20-35)
    out << "Allowed options:\n"
           "  -h [ --help ]                          produce help message\n"
           "  -f [ --file ] arg                      source file\n"
           "  -d [ --destination ] arg               destination file\n"
           "  -j [ --threads ] arg                   number of parallel threads\n"
           "  -x [ --resolution_x ] arg (=1200)      set x axis resolution\n"
           "  -y [ --resolution_y ] arg (=900)       set y axis resolution\n"
           "  -X [ --angle_around_x ] arg (=0)       rotate view plane by angle around x \n"
           "                                         axis\n"
           "  -Y [ --angle_around_y ] arg (=0)       rotate view plane by angle around y \n"
           "                                         axis\n"
           "  -D [ --donor_angle ] arg (=0)          initial donor angle around y axis\n"
           "  -I [ --initial_system_angle ] arg (=0) initial angle of system y axis\n"
           "  --alpha_limit arg (=2.5)               limit alpha value\n"
           "\n"
           "B200 build only:\n"
           "  --devices arg (=0)                     CUDA device ordinals, comma separated\n"
           "  --precision arg (=64)                  64 or 32\n"
           "  --stats                                print per-phase timings as one JSON line\n"
           "  --frames arg (=1)                      render a sweep of -Y in this process: frame k\n"
           "                                         uses Y + (sweep_y_to - Y) k / frames and is\n"
           "                                         written to <destination stem>_<k>.vti\n"
           "  --sweep_y_to arg (=2)                  end angle of the sweep (exclusive)\n"
           "  --channels arg                         A:Q[,A:Q...]: also render these pairs of cell\n"
           "                                         arrays of the input file in the same walk, each\n"
           "                                         as a further array named A:Q (with --frames\n"
           "                                         only with --light_curve)\n"
           "  --light_curve                          write the light curve instead of images: -d names\n"
           "                                         a CSV with one line per frame (frame, Y_pi,\n"
           "                                         hit_pixels, solid_pixels, tau_sum, I_sum, then\n"
           "                                         A:Q_tau_sum, A:Q_I_sum per --channels pair), sums\n"
           "                                         over the pixels outside the solids, printed %.17g\n"
        << std::endl;
}

cli_result program_options(int argc, char** argv, config_str& cfg, std::ostream& out) {
    bool help = false, have_file = false, have_dest = false, have_threads = false;
    try {
        for (int i = 1; i < argc; i++) {
            const std::string tok = argv[i];
            const option* opt = nullptr;
            std::string value;
            bool has_value = false;
            if (tok.size() > 2 && tok[0] == '-' && tok[1] == '-') {
                std::string name = tok.substr(2);
                const auto eq = name.find('=');
                if (eq != std::string::npos) {
                    value = name.substr(eq + 1);
                    name = name.substr(0, eq);
                    has_value = true;
                }
                std::string err;
                opt = find_long(name, err);
                if (!opt) throw std::runtime_error(err);
            } else if (tok.size() >= 2 && tok[0] == '-') {
                opt = find_short(tok[1]);
                if (!opt) throw std::runtime_error("unrecognised option '" + tok + "'");
                if (tok.size() > 2) {
                    if (!opt->takes_value) throw std::runtime_error("option '" + tok.substr(0, 2) + "' does not take a value");
                    value = tok.substr(2);
                    has_value = true;
                }
            } else {
                throw std::runtime_error("too many positional options have been specified on the command line");
            }
            if (opt->takes_value && !has_value) {
                if (i + 1 >= argc) {
                    throw std::runtime_error(std::string("the required argument for option '--") + opt->long_name +
                                             "' is missing");
                }
                value = argv[++i];
            }
            const std::string name = opt->long_name;
            if (name == "help") help = true;
            else if (name == "file") { cfg.file = value; have_file = true; }
            else if (name == "destination") { cfg.destination = value; have_dest = true; }
            else if (name == "threads") { cfg.threads = static_cast<int>(to_integer(name, value)); have_threads = true; }
            else if (name == "resolution_x") cfg.resolution_x = static_cast<std::size_t>(to_integer(name, value));
            else if (name == "resolution_y") cfg.resolution_y = static_cast<std::size_t>(to_integer(name, value));
            else if (name == "angle_around_x") cfg.angle_around_x = to_double(name, value);
            else if (name == "angle_around_y") cfg.angle_around_y = to_double(name, value);
            else if (name == "donor_angle") cfg.donor_angle = to_double(name, value);
            else if (name == "initial_system_angle") cfg.system_initial_angle_around_y = to_double(name, value);
            else if (name == "alpha_limit") cfg.limit_alpha_value = to_double(name, value);
            else if (name == "devices") cfg.devices = value;
            else if (name == "stats") cfg.stats = true;
            else if (name == "precision") cfg.precision = static_cast<int>(to_integer(name, value));
            else if (name == "frames") cfg.frames = static_cast<int>(to_integer(name, value));
            else if (name == "sweep_y_to") cfg.sweep_y_to = to_double(name, value);
            else if (name == "channels") cfg.channels = parse_channels(value);
            else if (name == "light_curve") cfg.light_curve = true;
        }
        if (!cfg.channels.empty() && cfg.frames > 1 && !cfg.light_curve) {
            throw std::runtime_error("--channels cannot be combined with --frames > 1");
        }
    } catch (const std::exception& e) {
        out << "Error! " << e.what() << std::endl;
        print_usage(out);
        return cli_result::exit_error;
    }
    if (help) {
        print_usage(out);
        return cli_result::exit_ok;
    }
    if (!(have_file && have_dest)) {
        out << "Error! Source filename and destination filename must be specified" << std::endl;
        print_usage(out);
        return cli_result::exit_ok;
    }
    if (!have_threads) {
        cfg.threads = std::max(static_cast<int>(std::thread::hardware_concurrency()), 1); // main.cpp:57
    }
    return cli_result::run;
}

} // namespace c5host
