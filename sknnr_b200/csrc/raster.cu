// Raster front end (scope row f4): the step either side of the hot path when the caller is a
// map - the "sknnr-spatial"-style loop that feeds every pixel of a band-major image through
// kneighbors / predict and writes band-major result layers back.
//
// A raster block arrives as d bands of `rows` contiguous pixels ([d][rows], what GDAL / rasterio /
// xarray hand out).  On the host that layout costs a strided transpose plus a boolean-mask copy
// before scikit-learn can see [n_valid, d] rows; here both happen on the device, next to the
// search:
//   raster_mask_kernel    valid[p] = every band finite and != nodata; per-group counts
//   raster_scan_kernel    exclusive scan of the group counts (one CTA), total to the host
//   raster_gather_kernel  stable compaction + transpose: Xc[pos[p]][b] = band[b][p]
//   (the usual chunk pipeline runs on Xc)
//   raster_scatter_kernel band-major result layers, `fill` where the pixel was masked
// All four are HBM-bound streaming kernels (8d bytes in, 8d out per pixel at f64).  The mask and
// the gather read the bands in the caller's element type (float64, float32 or an integer type), and
// the gather keeps it: the projection converts the compacted rows to float64 as it loads them.
#include "common.cuh"
#include "kernels.h"

#include <type_traits>

namespace sk {

constexpr int RASTER_THREADS = 256;

template <typename T>
__global__ void __launch_bounds__(RASTER_THREADS)
raster_mask_kernel(const T *__restrict__ bands, long long rows, int d, int use_nodata, double nodata,
                   int *__restrict__ pos, int *__restrict__ counts) {
    const long long g0 = (long long)blockIdx.x * RASTER_GROUP;
    int total = 0;
#pragma unroll
    for (int i = 0; i < RASTER_GROUP / RASTER_THREADS; ++i) {
        const long long p = g0 + threadIdx.x + i * RASTER_THREADS;
        bool ok = p < rows;
        if (ok) {
            for (int b = 0; b < d; ++b) {
                const double v = x_to_f64(bands[(long long)b * rows + p]);
                // isfinite on the value the search will see; nodata compares in float64 (the caller
                // rounds it to a float band's own type first; an integer band is never NaN / inf)
                if constexpr (std::is_floating_point<T>::value)
                    ok = ok && isfinite(v) && !(use_nodata && v == nodata);
                else
                    ok = ok && !(use_nodata && v == nodata);
            }
            pos[p] = ok ? 1 : 0;
        }
        total += __syncthreads_count(ok);
    }
    if (threadIdx.x == 0) counts[blockIdx.x] = total;
}

// counts[0..n) -> exclusive offsets in place; counts[n] = total
__global__ void __launch_bounds__(1024)
raster_scan_kernel(int *__restrict__ counts, int n, int *__restrict__ total_out) {
    __shared__ int wsum[32];
    __shared__ int carry_s;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (int base = 0; base < n; base += 1024) {
        const int i = base + threadIdx.x;
        const int v = i < n ? counts[i] : 0;
        int x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(SK_FULL, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) wsum[warp] = x;
        __syncthreads();
        if (warp == 0) {
            int w = wsum[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(SK_FULL, w, o);
                if (lane >= o) w += y;
            }
            wsum[lane] = w;
        }
        __syncthreads();
        const int carry = carry_s;
        const int incl = x + (warp ? wsum[warp - 1] : 0) + carry;
        if (i < n) counts[i] = incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry_s = incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        counts[n] = carry_s;
        *total_out = carry_s;
    }
}

// One CTA per group of RASTER_GROUP pixels, thread t owns pixels 4t .. 4t+3 (stable order).
// pos[p]: in = valid flag, out = compacted row of the block or -1.
template <typename T>
__global__ void __launch_bounds__(RASTER_THREADS)
raster_gather_kernel(const T *__restrict__ bands, long long rows, int d, const int *__restrict__ offs,
                     int *__restrict__ pos, T *__restrict__ xc) {
    __shared__ int wsum[RASTER_THREADS / 32];
    constexpr int PER = RASTER_GROUP / RASTER_THREADS;
    const long long p0 = (long long)blockIdx.x * RASTER_GROUP + threadIdx.x * PER;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int flag[PER], mine = 0;
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        flag[i] = (p0 + i < rows) ? pos[p0 + i] : 0;
        mine += flag[i];
    }
    int x = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(SK_FULL, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) wsum[warp] = x;
    __syncthreads();
    int before = offs[blockIdx.x] + x - mine;
    for (int w = 0; w < warp; ++w) before += wsum[w];
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        const long long p = p0 + i;
        if (p >= rows) break;
        if (!flag[i]) {
            pos[p] = -1;
            continue;
        }
        pos[p] = before;
        T *dst = xc + (long long)before * d;
        for (int b = 0; b < d; ++b) dst[b] = bands[(long long)b * rows + p];
        ++before;
    }
}

// Band-major result layers of a block: layer j of `out` is out + j * ld_out.
template <typename T>
__global__ void __launch_bounds__(RASTER_THREADS)
raster_scatter_kernel(const int *__restrict__ pos, long long rows, const T *__restrict__ src, int width,
                      T fill, T *__restrict__ out, long long ld_out) {
    const long long p = (long long)blockIdx.x * RASTER_THREADS + threadIdx.x;
    if (p >= rows) return;
    const int r = pos[p];
    for (int j = 0; j < width; ++j) out[(long long)j * ld_out + p] = r >= 0 ? src[(long long)r * width + j] : fill;
}

cudaError_t launch_raster_mask(const void *bands, int x_dtype, long long rows, int d, int use_nodata,
                               double nodata, int *pos, int *counts, int *total_out, cudaStream_t st) {
    if (rows <= 0) return cudaSuccess;
    const int groups = (int)((rows + RASTER_GROUP - 1) / RASTER_GROUP);
    cudaError_t e = with_x_type(x_dtype, [&](auto zero) {
        using T = decltype(zero);
        raster_mask_kernel<T><<<groups, RASTER_THREADS, 0, st>>>((const T *)bands, rows, d, use_nodata, nodata, pos, counts);
        return cudaGetLastError();
    });
    if (e != cudaSuccess) return e;
    raster_scan_kernel<<<1, 1024, 0, st>>>(counts, groups, total_out);
    return cudaGetLastError();
}

cudaError_t launch_raster_gather(const void *bands, int x_dtype, long long rows, int d, const int *offs,
                                 int *pos, void *xc, cudaStream_t st) {
    if (rows <= 0) return cudaSuccess;
    const int groups = (int)((rows + RASTER_GROUP - 1) / RASTER_GROUP);
    return with_x_type(x_dtype, [&](auto zero) {
        using T = decltype(zero);
        raster_gather_kernel<T><<<groups, RASTER_THREADS, 0, st>>>((const T *)bands, rows, d, offs, pos, (T *)xc);
        return cudaGetLastError();
    });
}

cudaError_t launch_raster_scatter_f64(const int *pos, long long rows, const double *src, int width,
                                      double fill, double *out, long long ld_out, cudaStream_t st) {
    if (rows <= 0 || width <= 0) return cudaSuccess;
    const unsigned grid = (unsigned)((rows + RASTER_THREADS - 1) / RASTER_THREADS);
    raster_scatter_kernel<double><<<grid, RASTER_THREADS, 0, st>>>(pos, rows, src, width, fill, out, ld_out);
    return cudaGetLastError();
}

cudaError_t launch_raster_scatter_i64(const int *pos, long long rows, const long long *src, int width,
                                      long long fill, long long *out, long long ld_out, cudaStream_t st) {
    if (rows <= 0 || width <= 0) return cudaSuccess;
    const unsigned grid = (unsigned)((rows + RASTER_THREADS - 1) / RASTER_THREADS);
    raster_scatter_kernel<long long><<<grid, RASTER_THREADS, 0, st>>>(pos, rows, src, width, fill, out, ld_out);
    return cudaGetLastError();
}

}  // namespace sk
