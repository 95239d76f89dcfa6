// c5_flux.cu — per-row sums of a rendered band (c5_render_flux, c5_render_flux_submit): the light
// curve of a sweep needs 16 bytes per pair and VIEW, so the image stays on the device and only its
// row sums are copied to the host. The device forms (c5_render_flux_device, c5_render_flux_jvp_device)
// also add the rows into the view's total on the device, in the host's order.
//
// Summation order (the contract of include/c5gpu.h, which makes the sums bit-identical for any band
// cut, device count and number of views in flight): one block of 256 threads per row; thread t adds
// the pixels x = t, t + 256, ... of its row in increasing x, starting from 0, skipping pixels under
// the solid mask; the 256 partials are folded by a halving tree, p[t] += p[t + s] for s = 128, 64,
// ..., 1. The host-loop build runs the same two functions in the same order.
#include "c5_internal.h"

namespace c5 {

namespace {

constexpr int kFluxThreads = 256;

// Thread t's partial sums of one row: 2K sums, {tau_c, I_c} per pair. row: the band buffer's row
// (K pairs per pixel, x fastest); mask_row: the whole-image mask's row, null without solids.
template <int K>
C5_HD void row_partials(const double* row, const uint8_t* mask_row, int res_x, int t, double (&acc)[2 * K]) {
    for (int c = 0; c < 2 * K; c++) acc[c] = 0.0;
    const double2* px = reinterpret_cast<const double2*>(row);
    for (int i = t; i < res_x; i += kFluxThreads) {
        if (mask_row && mask_row[i]) continue;
        for (int c = 0; c < K; c++) {
            const double2 v = px[static_cast<size_t>(i) * K + c];
            acc[2 * c] += v.x;
            acc[2 * c + 1] += v.y;
        }
    }
}

// One level of the tree over partials p[word][256] (word-major, so that the threads of a warp hit
// distinct banks): p[t] += p[t + s].
template <int K>
C5_HD void fold_level(double* p, int t, int s) {
    for (int c = 0; c < 2 * K; c++) p[c * kFluxThreads + t] += p[c * kFluxThreads + t + s];
}

} // namespace

// One block per row of the band. At K = 8 the partials take 256 x 16 doubles = 32 KB of shared memory.
template <int K>
__global__ void __launch_bounds__(kFluxThreads) reduce_rows(const double* out, const uint8_t* mask, int res_x,
                                                            int row_begin, double* row_flux) {
    __shared__ double p[2 * K * kFluxThreads];
    const int j = row_begin + static_cast<int>(blockIdx.x);
    const int t = static_cast<int>(threadIdx.x);
    double acc[2 * K];
    row_partials<K>(out + static_cast<size_t>(blockIdx.x) * res_x * 2 * K, mask ? mask + static_cast<size_t>(j) * res_x : nullptr,
                    res_x, t, acc);
    for (int c = 0; c < 2 * K; c++) p[c * kFluxThreads + t] = acc[c];
    __syncthreads();
    for (int s = kFluxThreads / 2; s > 0; s >>= 1) {
        if (t < s) fold_level<K>(p, t, s);
        __syncthreads();
    }
    if (t < 2 * K) row_flux[static_cast<size_t>(j) * 2 * K + t] = p[t * kFluxThreads];
}

// The view's total on the device (c5_render_flux_device, c5_render_flux_jvp_device): thread c adds word c of the
// band's rows of row_flux (`words` per row) in increasing j, starting from 0 — the host's order for the total,
// where the rows outside the band are +0 and leave the sum's bits alone. Word c < split goes to lo[c], the others
// to hi[c - split]; a null destination is skipped.
C5_HD double band_total(const double* row_flux, int words, int row_begin, int row_end, int c) {
    double s = 0.0;
    for (int j = row_begin; j < row_end; j++) s += row_flux[static_cast<size_t>(j) * words + c];
    return s;
}

__global__ void __launch_bounds__(32) total_rows(const double* row_flux, int words, int row_begin, int row_end, int split,
                                                 double* lo, double* hi) {
    const int c = static_cast<int>(threadIdx.x);
    if (c >= words) return;
    double* dst = c < split ? (lo ? lo + c : nullptr) : (hi ? hi + (c - split) : nullptr);
    if (dst) *dst = band_total(row_flux, words, row_begin, row_end, c);
}

namespace {

template <int K>
void reduce_rows_on_host(const double* out, const uint8_t* mask, int res_x, int row_begin, int row_end, double* row_flux) {
    std::vector<double> p(static_cast<size_t>(2 * K * kFluxThreads));
    for (int j = row_begin; j < row_end; j++) {
        for (int t = 0; t < kFluxThreads; t++) {
            double acc[2 * K];
            row_partials<K>(out + static_cast<size_t>(j - row_begin) * res_x * 2 * K, mask ? mask + static_cast<size_t>(j) * res_x : nullptr,
                            res_x, t, acc);
            for (int c = 0; c < 2 * K; c++) p[static_cast<size_t>(c * kFluxThreads + t)] = acc[c];
        }
        for (int s = kFluxThreads / 2; s > 0; s >>= 1) {
            for (int t = 0; t < s; t++) fold_level<K>(p.data(), t, s);
        }
        for (int c = 0; c < 2 * K; c++) row_flux[static_cast<size_t>(j) * 2 * K + c] = p[static_cast<size_t>(c * kFluxThreads)];
    }
}

template <int K>
void launch_k(DeviceState& d, int res_x, int row_begin, int row_end, const uint8_t* mask) {
    count_launch();
    if (kHostSim) {
        reduce_rows_on_host<K>(d.out.p, mask, res_x, row_begin, row_end, d.row_flux.p);
        return;
    }
    reduce_rows<K><<<static_cast<unsigned>(row_end - row_begin), kFluxThreads, 0, d.stream>>>(d.out.p, mask, res_x, row_begin,
                                                                                              d.row_flux.p);
    C5_CUDA(cudaGetLastError());
}

} // namespace

void launch_reduce_rows(DeviceState& d, int res_x, int res_y, int row_begin, int row_end, int pairs, bool use_mask) {
    d.row_flux.ensure(static_cast<size_t>(res_y) * 2 * static_cast<size_t>(pairs));
    const uint8_t* mask = use_mask ? d.mask.p : nullptr;
    switch (pairs) {
    case 1: launch_k<1>(d, res_x, row_begin, row_end, mask); break;
    case 2: launch_k<2>(d, res_x, row_begin, row_end, mask); break;
    case 3: launch_k<3>(d, res_x, row_begin, row_end, mask); break;
    case 4: launch_k<4>(d, res_x, row_begin, row_end, mask); break;
    case 5: launch_k<5>(d, res_x, row_begin, row_end, mask); break;
    case 6: launch_k<6>(d, res_x, row_begin, row_end, mask); break;
    case 7: launch_k<7>(d, res_x, row_begin, row_end, mask); break;
    case 8: launch_k<8>(d, res_x, row_begin, row_end, mask); break;
    default: fail(C5_E_INVALID, "render_flux: 1 .. C5_MAX_CHANNELS pairs");
    }
}

void launch_total_rows(DeviceState& d, int row_begin, int row_end, int words, int split, double* lo, double* hi) {
    count_launch();
    if (kHostSim) {
        for (int c = 0; c < words; c++) {
            double* dst = c < split ? (lo ? lo + c : nullptr) : (hi ? hi + (c - split) : nullptr);
            if (dst) *dst = band_total(d.row_flux.p, words, row_begin, row_end, c);
        }
        return;
    }
    total_rows<<<1, 32, 0, d.stream>>>(d.row_flux.p, words, row_begin, row_end, split, lo, hi);
    C5_CUDA(cudaGetLastError());
}

} // namespace c5
