// vti_writer.cpp — see vti_writer.hpp.
#include "vti_writer.hpp"

#include <cstdint>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <sstream>
#include <atomic>
#include <cstdlib>
#include <stdexcept>
#include <thread>
#include <vector>

#include <unistd.h>
#include <zlib.h>

namespace c5host {

namespace {

struct file_closer {
    FILE* f;
    ~file_closer() {
        if (f) std::fclose(f);
    }
};

const char kB64[] = "ABCDEFGHIJKLMNOPQRSTUVWXYZabcdefghijklmnopqrstuvwxyz0123456789+/";

// One self-contained base64 stream (padded): VTK encodes the block table and the data separately.
std::string base64(const unsigned char* p, std::size_t n) {
    std::string out((n + 2) / 3 * 4, '=');
    char* o = &out[0];
    std::size_t i = 0;
    for (; i + 2 < n; i += 3, o += 4) {
        const unsigned v = (p[i] << 16) | (p[i + 1] << 8) | p[i + 2];
        o[0] = kB64[v >> 18];
        o[1] = kB64[(v >> 12) & 63];
        o[2] = kB64[(v >> 6) & 63];
        o[3] = kB64[v & 63];
    }
    if (i + 1 == n) {
        const unsigned v = p[i] << 16;
        o[0] = kB64[v >> 18];
        o[1] = kB64[(v >> 12) & 63];
    } else if (i + 2 == n) {
        const unsigned v = (p[i] << 16) | (p[i + 1] << 8);
        o[0] = kB64[v >> 18];
        o[1] = kB64[(v >> 12) & 63];
        o[2] = kB64[(v >> 6) & 63];
    }
    return out;
}

// Threads for the block compressor: the blocks of VTK's compressed layout are independent zlib streams, so a
// 69 MB frame (66 blocks) is deflated by as many cores as there are, and the bytes written do not depend on how
// many took part. C5_VTI_THREADS overrides (1 = the serial path; tests compare the two).
unsigned compressor_threads(std::uint64_t n_blocks) {
    unsigned n = std::thread::hardware_concurrency();
    if (const char* e = std::getenv("C5_VTI_THREADS")) {
        const long v = std::strtol(e, nullptr, 10);
        if (v > 0) n = static_cast<unsigned>(v);
    }
    if (n == 0) n = 1;
    if (n > 32) n = 32;
    if (n > n_blocks) n = static_cast<unsigned>(n_blocks);
    return n == 0 ? 1 : n;
}

// Decodes ONE padded base64 stream starting at p (stops after its padding or at a non-alphabet byte);
// returns the bytes and advances p past the stream.
std::vector<unsigned char> unbase64(const unsigned char*& p, const unsigned char* end, std::size_t want_bytes) {
    static int lut[256];
    static bool init = false;
    if (!init) {
        for (int& v : lut) v = -1;
        for (int i = 0; i < 64; i++) lut[static_cast<unsigned char>(kB64[i])] = i;
        init = true;
    }
    std::vector<unsigned char> out;
    const std::size_t quads = (want_bytes + 2) / 3;
    out.reserve(quads * 3);
    for (std::size_t q = 0; q < quads; q++) {
        int v[4];
        for (int k = 0; k < 4; k++) {
            while (p < end && (*p == '\n' || *p == '\r' || *p == ' ')) ++p;
            if (p >= end) throw std::runtime_error("base64 stream is truncated");
            v[k] = (*p == '=') ? -2 : lut[*p];
            if (v[k] == -1) throw std::runtime_error("bad base64 character");
            ++p;
        }
        out.push_back(static_cast<unsigned char>((v[0] << 2) | (v[1] >> 4)));
        if (v[2] >= 0) out.push_back(static_cast<unsigned char>(((v[1] & 15) << 4) | (v[2] >> 2)));
        if (v[2] >= 0 && v[3] >= 0) out.push_back(static_cast<unsigned char>(((v[2] & 3) << 6) | v[3]));
    }
    if (out.size() < want_bytes) throw std::runtime_error("base64 stream is shorter than its header says");
    out.resize(want_bytes);
    return out;
}

} // namespace

void write_vti(const std::string& filename, const double* image, std::size_t res_x, std::size_t res_y,
               bool compress) {
    write_vti(filename, image, res_x, res_y, compress ? vti_encoding::zlib_raw : vti_encoding::raw);
}

namespace {

// One array's appended data in VTK's compressed block layout: [n_blocks][block_size][last_block_size]
// [compressed sizes...] then the blocks; with b64 the table and the blocks as two base64 streams.
std::string compressed_payload(const double* data, std::uint64_t n_bytes, bool b64, const std::string& filename) {
    const std::uint64_t block = 1u << 20;
    const std::uint64_t n_blocks = (n_bytes + block - 1) / block;
    const std::uint64_t last = n_bytes - (n_blocks - 1) * block;
    std::vector<std::vector<unsigned char>> packed(n_blocks);
    std::vector<std::uint64_t> header(3 + n_blocks);
    header[0] = n_blocks;
    header[1] = block;
    header[2] = (last == block) ? 0 : last;
    const unsigned char* src = reinterpret_cast<const unsigned char*>(data);
    std::atomic<std::uint64_t> next{0};
    std::atomic<bool> failed{false};
    auto deflate_blocks = [&] {   // blocks are handed out one at a time: the last, short one does not unbalance anyone
        for (std::uint64_t b = next.fetch_add(1); b < n_blocks && !failed.load(); b = next.fetch_add(1)) {
            const uLong in_size = static_cast<uLong>(b + 1 == n_blocks ? last : block);
            uLongf out_size = compressBound(in_size);
            packed[b].resize(out_size);
            if (compress2(packed[b].data(), &out_size, src + b * block, in_size, Z_BEST_SPEED) != Z_OK) {
                failed.store(true);
                return;
            }
            packed[b].resize(out_size);
            header[3 + b] = out_size;
        }
    };
    const unsigned n_threads = compressor_threads(n_blocks);
    if (n_threads <= 1) {
        deflate_blocks();
    } else {
        std::vector<std::thread> pool;
        for (unsigned t = 1; t < n_threads; t++) pool.emplace_back(deflate_blocks);
        deflate_blocks();
        for (auto& t : pool) t.join();
    }
    if (failed.load()) throw std::runtime_error("zlib failed while writing " + filename);
    std::vector<unsigned char> all(reinterpret_cast<const unsigned char*>(header.data()),
                                   reinterpret_cast<const unsigned char*>(header.data() + header.size()));
    const std::size_t table = all.size();
    for (const auto& p : packed) all.insert(all.end(), p.begin(), p.end());
    if (!b64) return std::string(all.begin(), all.end());
    // vtkXMLWriter's default (EncodeAppendedData on): the block table is one base64 stream, the
    // concatenated compressed blocks another
    return base64(all.data(), table) + base64(all.data() + table, all.size() - table);
}

} // namespace

void write_vti(const std::string& filename, const double* image, std::size_t res_x, std::size_t res_y,
               vti_encoding encoding, const std::vector<vti_array>& extra) {
    const bool compress = encoding != vti_encoding::raw;
    const bool b64 = encoding == vti_encoding::zlib_base64;
    FILE* fp = std::fopen(filename.c_str(), "wb");
    if (!fp) throw std::runtime_error("cannot write " + filename);
    file_closer closer{fp};
    const std::uint64_t n_bytes = static_cast<std::uint64_t>(res_x) * res_y * 2 * sizeof(double);
    const int ex = static_cast<int>(res_x) - 1, ey = static_cast<int>(res_y) - 1;
    std::vector<vti_array> arrays{{"ImageScalars", image}};
    arrays.insert(arrays.end(), extra.begin(), extra.end());
    // compressed arrays are packed first: their sizes give the offsets the header lists
    std::vector<std::string> payload(compress ? arrays.size() : 0);
    for (std::size_t a = 0; a < payload.size(); a++) payload[a] = compressed_payload(arrays[a].data, n_bytes, b64, filename);
    std::string data_arrays;
    std::uint64_t offset = 0;
    for (std::size_t a = 0; a < arrays.size(); a++) {
        data_arrays += "        <DataArray type=\"Float64\" Name=\"" + arrays[a].name +
                       "\" NumberOfComponents=\"2\" format=\"appended\" offset=\"" + std::to_string(offset) + "\"/>\n";
        offset += compress ? payload[a].size() : sizeof(n_bytes) + n_bytes;
    }
    std::fprintf(fp,
                 "<?xml version=\"1.0\"?>\n"
                 "<VTKFile type=\"ImageData\" version=\"1.0\" byte_order=\"LittleEndian\" header_type=\"UInt64\"%s>\n"
                 "  <ImageData WholeExtent=\"0 %d 0 %d 0 0\" Origin=\"0 0 0\" Spacing=\"1 1 1\">\n"
                 "    <Piece Extent=\"0 %d 0 %d 0 0\">\n"
                 "      <PointData Scalars=\"ImageScalars\">\n"
                 "%s"
                 "      </PointData>\n"
                 "      <CellData/>\n"
                 "    </Piece>\n"
                 "  </ImageData>\n"
                 "  <AppendedData encoding=\"%s\">\n   _",
                 compress ? " compressor=\"vtkZLibDataCompressor\"" : "", ex, ey, ex, ey, data_arrays.c_str(),
                 b64 ? "base64" : "raw");
    for (std::size_t a = 0; a < arrays.size(); a++) {
        if (compress) {
            std::fwrite(payload[a].data(), 1, payload[a].size(), fp);
            continue;
        }
        std::fwrite(&n_bytes, sizeof(n_bytes), 1, fp);
        // the pixels go straight from the caller's buffer to the file descriptor: stdio would copy 69 MB through its
        // own buffer first
        std::fflush(fp);
        const char* at = reinterpret_cast<const char*>(arrays[a].data);
        std::uint64_t left = n_bytes;
        while (left > 0) {
            const ssize_t w = ::write(fileno(fp), at, left > (1u << 30) ? (1u << 30) : left);
            if (w <= 0) throw std::runtime_error("short write to " + filename);
            at += w;
            left -= static_cast<std::uint64_t>(w);
        }
    }
    std::fprintf(fp, "\n  </AppendedData>\n</VTKFile>\n");
}

void read_vti(const std::string& filename, std::size_t& res_x, std::size_t& res_y, std::size_t& comps,
              double*& image_out, const std::string& name) {
    std::ifstream in(filename, std::ios::binary);
    if (!in) throw std::runtime_error("cannot open " + filename);
    std::stringstream ss;
    ss << in.rdbuf();
    const std::string all = ss.str();
    auto attr = [&](const std::string& tag, const std::string& name) -> std::string {
        const std::size_t t = all.find("<" + tag);
        if (t == std::string::npos) throw std::runtime_error(filename + ": no <" + tag + ">");
        const std::size_t e = all.find('>', t);
        const std::size_t a = all.find(name + "=\"", t);
        if (a == std::string::npos || a > e) return "";
        const std::size_t s = a + name.size() + 2;
        return all.substr(s, all.find('"', s) - s);
    };
    int x0, x1, y0, y1, z0, z1;
    if (std::sscanf(attr("ImageData", "WholeExtent").c_str(), "%d %d %d %d %d %d", &x0, &x1, &y0, &y1, &z0, &z1) != 6) {
        throw std::runtime_error(filename + ": bad WholeExtent");
    }
    res_x = static_cast<std::size_t>(x1 - x0 + 1);
    res_y = static_cast<std::size_t>(y1 - y0 + 1);
    // the array: its element (by name, or the first one) and where its data starts in the appended section
    std::size_t array_at = all.find("<DataArray");
    if (!name.empty()) {
        const std::size_t named = all.find("Name=\"" + name + "\"");
        if (named == std::string::npos) throw std::runtime_error(filename + ": no array named '" + name + "'");
        array_at = all.rfind("<DataArray", named);
    }
    if (array_at == std::string::npos) throw std::runtime_error(filename + ": no <DataArray>");
    auto array_attr = [&](const std::string& key) -> std::string {
        const std::size_t e = all.find('>', array_at);
        const std::size_t a = all.find(" " + key + "=\"", array_at);
        if (a == std::string::npos || a > e) return "";
        const std::size_t s = a + key.size() + 3;
        return all.substr(s, all.find('"', s) - s);
    };
    comps = static_cast<std::size_t>(std::stoul(array_attr("NumberOfComponents")));
    const std::string off = array_attr("offset");
    const std::size_t array_offset = off.empty() ? 0 : static_cast<std::size_t>(std::stoull(off));
    const bool compressed = !attr("VTKFile", "compressor").empty();
    const bool b64 = attr("AppendedData", "encoding") == "base64";
    const std::size_t marker = all.find("<AppendedData");
    const std::size_t under = all.find('_', all.find('>', marker));
    const unsigned char* p = reinterpret_cast<const unsigned char*>(all.data()) + under + 1 + array_offset;
    const unsigned char* file_end = reinterpret_cast<const unsigned char*>(all.data()) + all.size();
    const std::size_t n_values = res_x * res_y * comps;
    std::vector<unsigned char> decoded; // base64: the appended section turned back into the raw layout
    if (b64) {
        if (!compressed) {
            std::vector<unsigned char> h = unbase64(p, file_end, 8);
            std::uint64_t n_bytes;
            std::memcpy(&n_bytes, h.data(), 8);
            std::vector<unsigned char> d = unbase64(p, file_end, n_bytes);
            decoded = h;
            decoded.insert(decoded.end(), d.begin(), d.end());
        } else {
            const unsigned char* q = p;
            std::vector<unsigned char> h3 = unbase64(q, file_end, 24); // how many blocks: then the whole table
            std::uint64_t n_blocks;
            std::memcpy(&n_blocks, h3.data(), 8);
            std::vector<unsigned char> h = unbase64(p, file_end, 24 + 8 * n_blocks);
            std::uint64_t total = 0;
            for (std::uint64_t b = 0; b < n_blocks; b++) {
                std::uint64_t sz;
                std::memcpy(&sz, h.data() + 24 + 8 * b, 8);
                total += sz;
            }
            std::vector<unsigned char> d = unbase64(p, file_end, total);
            decoded = h;
            decoded.insert(decoded.end(), d.begin(), d.end());
        }
        p = decoded.data();
    }
    image_out = new double[n_values];
    if (!compressed) {
        std::uint64_t n_bytes;
        std::memcpy(&n_bytes, p, 8);
        if (n_bytes != n_values * sizeof(double)) throw std::runtime_error(filename + ": unexpected data size");
        std::memcpy(image_out, p + 8, n_bytes);
    } else {
        std::uint64_t hdr[3];
        std::memcpy(hdr, p, 24);
        std::vector<std::uint64_t> sizes(hdr[0]);
        std::memcpy(sizes.data(), p + 24, 8 * hdr[0]);
        const unsigned char* src = p + 24 + 8 * hdr[0];
        unsigned char* dst = reinterpret_cast<unsigned char*>(image_out);
        for (std::uint64_t b = 0; b < hdr[0]; b++) {
            uLongf out_size = static_cast<uLongf>((b + 1 == hdr[0] && hdr[2]) ? hdr[2] : hdr[1]);
            if (uncompress(dst, &out_size, src, static_cast<uLong>(sizes[b])) != Z_OK) {
                throw std::runtime_error(filename + ": zlib inflate failed");
            }
            dst += out_size;
            src += sizes[b];
        }
    }
}

} // namespace c5host
