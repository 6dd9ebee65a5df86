// Projection into the estimator's feature space (north_star piece 1; seam S2,
// ref:src/sknnr/_base.py:236-239).  One affine map covers the four float transformers:
//     Z = ((X - center) / scale) @ proj
//   StandardScalerWithDOF   $SP/sklearn/preprocessing/_data.py:1131-1134
//   MahalanobisTransformer  ref:src/sknnr/transformers/_mahalanobis_transformer.py:55
//   CCorATransformer        ref:src/sknnr/transformers/_ccora_transformer.py:70
//   CCATransformer          ref:src/sknnr/transformers/_cca_transformer.py:87
// computed in float64 exactly as written (true division, centre first).  Raw map pixels are
// read from HBM once, in the caller's element type (float64, float32 or an integer type, each
// value converted to float64 on load); the kernel emits both operands the rest of the path needs:
//   z64  [n_q, d_out] float64          - exact re-rank operand
//   qimg [n_qtiles][dpad][256] float32 - search-kernel query tile image, -2 * (Z - mu)
#include "common.cuh"
#include "kernels.h"

#include <type_traits>

namespace sk {

constexpr int PROJ_THREADS = 128;  // one thread per query row; 128 rows per CTA
constexpr int PROJ_KCHUNK = 8;

template <typename TX>
__global__ void __launch_bounds__(PROJ_THREADS)
project_kernel(const TX *__restrict__ X, long long ldx, long long n_q, int d_in, int d_out,
               int dpad, const double *__restrict__ center, const double *__restrict__ scale,
               const double *__restrict__ proj, const double *__restrict__ mu,
               double *__restrict__ z64, float *__restrict__ qimg, __half *__restrict__ qimg_tc,
               int tc_kc, double tc_sigma, const int *__restrict__ n_rows_dev, int *__restrict__ nonfinite,
               int xs_in_smem, int ps_in_smem) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int xs_ld = d_in | 1;  // odd row stride (in doubles): conflict-free row reads
    double *xs = reinterpret_cast<double *>(smem_raw);           // [128][xs_ld]
    double *ps = xs + (size_t)PROJ_THREADS * xs_ld;              // [d_in][d_out] (if proj)
    const long long q0 = (long long)blockIdx.x * PROJ_THREADS;
    if (n_rows_dev) {  // compacted launch: only the first *n_rows_dev rows exist
        const long long n_dev = *n_rows_dev;
        if (q0 >= (n_dev + QTILE - 1) / QTILE * QTILE) return;
        n_q = min(n_q, n_dev);
    }
    const int rows = (int)min((long long)PROJ_THREADS, n_q - q0);

    // coalesced load of the tile's rows, centring and scaling on the way in; (row, column) advance
    // incrementally (no integer division per element).  Without a projector the scaled value already
    // is z: it goes to z64 from here, where consecutive threads write consecutive addresses.
    // (xs_in_smem == 0: more features than a 128-row tile can stage in shared memory - every thread
    // then reads its own row from global memory in the loop below; ps_in_smem == 0: a projector too
    // large for shared memory is read through the read-only cache instead)
    if (xs_in_smem) {
        const int dr = PROJ_THREADS / d_in, dc = PROJ_THREADS - dr * d_in;
        int r = threadIdx.x / d_in, c = threadIdx.x - r * d_in;
        const bool z_here = !proj && z64 && d_out == d_in;
        // (every thread makes exactly d_in passes; the loads of eight passes are issued together, ahead
        // of the divisions, so that eight rows' worth of HBM requests are in flight per thread)
        constexpr int UNR = 8;
        for (int e0 = 0; e0 < d_in; e0 += UNR) {
            double v[UNR];
            int rr[UNR], cc[UNR];
#pragma unroll
            for (int u = 0; u < UNR; ++u) {
                rr[u] = r;
                cc[u] = c;
                const bool have = e0 + u < d_in && r < rows;
                v[u] = have ? x_to_f64(X[(q0 + r) * ldx + c]) : 0.0;
                r += dr;
                c += dc;
                if (c >= d_in) {
                    c -= d_in;
                    ++r;
                }
            }
#pragma unroll
            for (int u = 0; u < UNR; ++u) {
                if (e0 + u >= d_in) break;
                double w = v[u];
                if (rr[u] < rows) {
                    // NaN / inf anywhere in the query block: the caller raises scikit-learn's ValueError
                    // (an integer matrix holds neither)
                    if constexpr (std::is_floating_point<TX>::value)
                        if (nonfinite && !isfinite(w)) *nonfinite = 1;
                    if (center) w -= center[cc[u]];
                    if (scale) w /= scale[cc[u]];
                    if (z_here) z64[(q0 + rr[u]) * d_out + cc[u]] = w;
                }
                xs[rr[u] * xs_ld + cc[u]] = w;
            }
        }
    }
    const bool z_later = z64 && (proj || d_out != d_in || !xs_in_smem);
    if (!xs_in_smem) ps = xs;   // nothing staged in front of the projector
    if (proj && ps_in_smem)
        for (int e = threadIdx.x; e < d_in * d_out; e += PROJ_THREADS) ps[e] = proj[e];
    __syncthreads();
    const double *pmat = ps_in_smem ? ps : proj;

    const int r = threadIdx.x;
    const double *xr = xs + r * xs_ld;
    auto xval = [&](int i) -> double {
        if (xs_in_smem) return xr[i];
        double v = 0.0;
        if (r < rows) {
            v = x_to_f64(X[(q0 + r) * ldx + i]);
            if constexpr (std::is_floating_point<TX>::value)
                if (nonfinite && !isfinite(v)) *nonfinite = 1;
            if (center) v -= center[i];
            if (scale) v /= scale[i];
        }
        return v;
    };
    // row (q0 + r) lives in query tile (q0 + r) / QTILE at column (q0 + r) % QTILE
    const long long qrow = q0 + r;
    float *qt = qimg ? qimg + (size_t)(qrow / QTILE) * dpad * QTILE + (qrow % QTILE) : nullptr;
    // tensor-core image: consecutive 128-row operands [chunk][row][8] FP16 (two of them form one CTA
    // tile of the tensor kernel): element k < d_out = -2 * sigma * (z_k - mu_k) (sigma = the index's
    // power-of-two scale that brings the reference plots into FP16 range), elements d_out .. d_out+2
    // = 1 (they meet the 3-way FP16 split of sigma^2 |r - mu|^2 on the reference side, which folds
    // |r|^2 into the contraction), zero up to the padded depth 8 * tc_kc.
    uint4 *qc = nullptr;
    if (qimg_tc) {
        qc = reinterpret_cast<uint4 *>(qimg_tc) + ((size_t)(qrow / TC_M) * tc_kc) * TC_M + (qrow % TC_M);
    }
    const int k_end = qc ? max(dpad, 8 * tc_kc) : dpad;
    for (int k0 = 0; k0 < k_end; k0 += PROJ_KCHUNK) {
        double z[PROJ_KCHUNK];
#pragma unroll
        for (int kk = 0; kk < PROJ_KCHUNK; ++kk) z[kk] = 0.0;
        if (k0 >= d_out) {
        } else if (proj) {
            for (int i = 0; i < d_in; ++i) {
                const double xv = xval(i);
                const double *pr = pmat + (size_t)i * d_out + k0;
#pragma unroll
                for (int kk = 0; kk < PROJ_KCHUNK; ++kk)
                    if (k0 + kk < d_out) z[kk] += xv * pr[kk];
            }
        } else {
#pragma unroll
            for (int kk = 0; kk < PROJ_KCHUNK; ++kk)
                if (k0 + kk < d_out) z[kk] = xval(k0 + kk);
        }
        float hv[PROJ_KCHUNK];
#pragma unroll
        for (int kk = 0; kk < PROJ_KCHUNK; ++kk) {
            const int k = k0 + kk;
            float sv = 0.0f, h = 0.0f;
            if (k < d_out && r < rows) {
                if (z_later) z64[(q0 + r) * d_out + k] = z[kk];
                const double c2 = -2.0 * (z[kk] - mu[k]);
                sv = (float)c2;
                h = (float)(c2 * tc_sigma);
            } else if (k >= d_out && k < d_out + 3 && r < rows) {
                h = 1.0f;
            }
            hv[kk] = h;
            if (qt && k < dpad) qt[(size_t)k * QTILE] = sv;
        }
        if (qc && k0 < 8 * tc_kc) {
            // round to nearest even; |h| >= 65520 becomes +-inf (such rows fail the certificate, refine.cu)
            const __half2 h01 = __floats2half2_rn(hv[0], hv[1]), h23 = __floats2half2_rn(hv[2], hv[3]);
            const __half2 h45 = __floats2half2_rn(hv[4], hv[5]), h67 = __floats2half2_rn(hv[6], hv[7]);
            uint4 u;
            u.x = *reinterpret_cast<const uint32_t *>(&h01);
            u.y = *reinterpret_cast<const uint32_t *>(&h23);
            u.z = *reinterpret_cast<const uint32_t *>(&h45);
            u.w = *reinterpret_cast<const uint32_t *>(&h67);
            qc[(size_t)(k0 / 8) * TC_M] = u;
        }
    }
}

cudaError_t launch_project(const void *X, int x_dtype, long long ldx, long long n_q, int d_in,
                           int d_out, int dpad, const double *center, const double *scale,
                           const double *proj, const double *mu, double *z64, float *qimg,
                           __half *qimg_tc, int tc_kc, double tc_sigma, const int *n_rows_dev,
                           int *nonfinite, cudaStream_t st) {
    if (n_q <= 0) return cudaSuccess;
    const int xs_ld = d_in | 1;
    // what fits the 227 KB of shared memory is staged there: the 128-row tile first, then the projector
    const size_t cap = 227 * 1024, xs_bytes = (size_t)PROJ_THREADS * xs_ld * 8;
    const size_t ps_bytes = proj ? (size_t)d_in * d_out * 8 : 0;
    const int xs_in_smem = xs_bytes <= cap ? 1 : 0;
    const int ps_in_smem = (xs_in_smem ? xs_bytes : 0) + ps_bytes <= cap ? 1 : 0;
    const size_t smem = (xs_in_smem ? xs_bytes : 0) + (ps_in_smem ? ps_bytes : 0);
    // cover whole query tiles so that padding columns of the last tile are zero-filled (every
    // CTA tile size of the search engines divides padded_rows, a multiple of PROJ_THREADS)
    const long long padded = padded_rows(n_q);
    const long long grid = (padded + PROJ_THREADS - 1) / PROJ_THREADS;
    return with_x_type(x_dtype, [&](auto zero) {
        using TX = decltype(zero);
        cudaError_t e = cudaFuncSetAttribute(project_kernel<TX>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             227 * 1024);
        if (e != cudaSuccess) return e;
        project_kernel<TX><<<(unsigned)grid, PROJ_THREADS, smem, st>>>(
            (const TX *)X, ldx, n_q, d_in, d_out, dpad, center, scale, proj, mu, z64, qimg, qimg_tc,
            tc_kc, tc_sigma, n_rows_dev, nonfinite, xs_in_smem, ps_in_smem);
        return cudaGetLastError();
    });
}

}  // namespace sk
