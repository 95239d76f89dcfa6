// vti_writer.hpp — the .vti the reference exports (object2d.cpp:7-29): vtkImageData with
// dimensions (res_x, res_y, 1), one PointData array "ImageScalars" (utility/screen.py:12 colours
// by ('POINTS', 'ImageScalars', 'Y')), Float64, 2 components {tau, I}, x fastest.
#pragma once

#include <cstddef>
#include <string>
#include <vector>

namespace c5host {

// How the appended data section is written; all three are standard VTK XML that vtkXMLImageDataReader
// (and ParaView, utility/screen.py:5) reads.
//   raw          header_type UInt64 byte count + the doubles, encoding="raw" (fastest to write)
//   zlib_raw     vtkZLibDataCompressor blocks (block table of UInt64s + compressed blocks), encoding="raw"
//   zlib_base64  the same blocks with the table and the data as two base64 streams: what
//                vtkXMLImageDataWriter — the reference's writer, object2d.cpp:24-27 — writes with its
//                defaults (appended data mode, EncodeAppendedData on, zlib compressor)
enum class vti_encoding { raw = 0, zlib_raw = 1, zlib_base64 = 2 };

// A further PointData array beside ImageScalars: Float64, 2 components per pixel, x fastest, in the
// same encoding (`course --channels` writes one per channel, named "A:Q" after its fields).
struct vti_array {
    std::string name;
    const double* data;
};

// image: res_y * res_x * 2 doubles, x fastest. Without extra arrays the file is byte for byte what
// it was before they existed.
void write_vti(const std::string& filename, const double* image, std::size_t res_x, std::size_t res_y,
               vti_encoding encoding, const std::vector<vti_array>& extra = {});
void write_vti(const std::string& filename, const double* image, std::size_t res_x, std::size_t res_y,
               bool compress = false); // false: raw, true: zlib_raw

// Reads back what write_vti (or the oracle's shim writer) wrote: raw, zlib or zlib + base64 appended
// Float64 ImageScalars. Used by tests and by `course --compare`.
// `name`: the PointData array to read (empty: the first one, ImageScalars).
void read_vti(const std::string& filename, std::size_t& res_x, std::size_t& res_y, std::size_t& comps,
              double*& image_out, const std::string& name = "");

} // namespace c5host
