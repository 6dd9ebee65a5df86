// GPU forest walk for RFNN (SURVEY.md section 8, row f1): the terminal node of every tree of the
// fitted forests for every query row, i.e. RFNodeTransformer.transform
// (ref:src/sknnr/transformers/_tree_node_transformer.py:177-201 -> sklearn est.apply ->
// $SP/sklearn/tree/_tree.pyx:977-994), emitted either as node IDs (transform parity) or directly
// as the 16-bit node codes the Hamming search consumes, so that query rows never return to the
// host between the forest and the neighbour search.
//
// Semantics replicated bit for bit from scikit-learn's Tree._apply_dense:
//   * X is cast to float32 first (DTYPE), so float64 inputs are rounded to nearest even;
//   * at an internal node go left iff (double)x[feature] <= threshold (threshold is float64) - for
//     a float32 x that is x <= (largest float32 <= threshold), which is what the 16-byte nodes hold;
//     NaN follows the node's missing_go_to_left flag;
//   * a node is a leaf when children_left == -1.
//
// One thread walks its query through FOREST_ILP trees at a time (independent pointer chases in
// flight: the walk is load-latency bound); a warp = 32 consecutive queries in the same trees, so the
// top levels are a broadcast and deeper levels gather 16-byte nodes from L1/L2.  The CTA's
// query tile lives in shared memory as float32; results are staged per 32-tree group and written
// as whole rows.
#include "common.cuh"
#include "kernels.h"

namespace sk {

constexpr int FOREST_THREADS = 256;  // queries per CTA
constexpr int FOREST_TG = 32;        // trees per staging group
constexpr int FOREST_ILP = 2;        // trees walked concurrently by one thread

template <typename TX>
__global__ void __launch_bounds__(FOREST_THREADS)
forest_apply_kernel(const TX *__restrict__ X, long long ldx, long long n_q, int d,
                    const ForestNode *__restrict__ nodes, const int *__restrict__ roots, int n_trees,
                    uint16_t *__restrict__ out_codes, int *__restrict__ out_ids, long long ld_out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *xs = reinterpret_cast<float *>(smem_raw);                       // [FOREST_THREADS][d | 1]
    const int xs_ld = d | 1;
    int *stage = reinterpret_cast<int *>(xs + (size_t)FOREST_THREADS * xs_ld);  // [FOREST_THREADS][FOREST_TG + 1]
    const long long q0 = (long long)blockIdx.x * FOREST_THREADS;
    const int rows = (int)min((long long)FOREST_THREADS, n_q - q0);
    for (int e = threadIdx.x; e < FOREST_THREADS * d; e += FOREST_THREADS) {
        const int r = e / d, c = e - r * d;
        xs[r * xs_ld + c] = r < rows ? (float)X[(q0 + r) * ldx + c] : 0.0f;  // round to float32 like DTYPE
    }
    __syncthreads();
    const float *xr = xs + threadIdx.x * xs_ld;
    for (int t0 = 0; t0 < n_trees; t0 += FOREST_TG) {
        const int tn = min(FOREST_TG, n_trees - t0);
        for (int tt = 0; tt < tn; tt += FOREST_ILP) {
            int node[FOREST_ILP], root[FOREST_ILP];
            bool done[FOREST_ILP];
#pragma unroll
            for (int u = 0; u < FOREST_ILP; ++u) {
                done[u] = tt + u >= tn;
                root[u] = done[u] ? 0 : roots[t0 + tt + u];
                node[u] = root[u];
            }
            while (true) {
                bool all = true;
                ForestNode nd[FOREST_ILP];
#pragma unroll
                for (int u = 0; u < FOREST_ILP; ++u)
                    if (!done[u]) nd[u] = nodes[node[u]];
#pragma unroll
                for (int u = 0; u < FOREST_ILP; ++u) {
                    if (done[u]) continue;
                    if (nd[u].left < 0) {
                        stage[threadIdx.x * (FOREST_TG + 1) + tt + u] = out_ids ? node[u] - root[u] : nd[u].right;
                        done[u] = true;
                        continue;
                    }
                    const float x = xr[nd[u].feat & 0x7fffffff];
                    const bool go_left = isnan(x) ? (nd[u].feat < 0) : (x <= nd[u].thr);
                    node[u] = go_left ? nd[u].left : nd[u].right;
                    all = false;
                }
                if (all) break;
            }
        }
        __syncthreads();
        // row-contiguous write of the group: [rows][tn]
        for (int e = threadIdx.x; e < rows * tn; e += FOREST_THREADS) {
            const int r = e / tn, c = e - r * tn;
            const int v = stage[r * (FOREST_TG + 1) + c];
            if (out_ids)
                out_ids[(q0 + r) * ld_out + t0 + c] = v;
            else
                out_codes[(q0 + r) * ld_out + t0 + c] = (uint16_t)v;
        }
        __syncthreads();
    }
}

size_t forest_smem_bytes(int d) {
    return ((size_t)FOREST_THREADS * (d | 1) + (size_t)FOREST_THREADS * (FOREST_TG + 1)) * 4;
}

cudaError_t launch_forest_apply(const void *X, int x_is_f32, long long ldx, long long n_q, int d,
                                const ForestNode *nodes, const int *roots, int n_trees,
                                uint16_t *out_codes, int *out_ids, long long ld_out, cudaStream_t st) {
    if (n_q <= 0) return cudaSuccess;
    const size_t smem = forest_smem_bytes(d);
    if (smem > 227 * 1024) return cudaErrorInvalidValue;
    const long long grid = (n_q + FOREST_THREADS - 1) / FOREST_THREADS;
    cudaError_t e;
    if (x_is_f32) {
        e = cudaFuncSetAttribute(forest_apply_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) return e;
        forest_apply_kernel<float><<<(unsigned)grid, FOREST_THREADS, smem, st>>>(
            (const float *)X, ldx, n_q, d, nodes, roots, n_trees, out_codes, out_ids, ld_out);
    } else {
        e = cudaFuncSetAttribute(forest_apply_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) return e;
        forest_apply_kernel<double><<<(unsigned)grid, FOREST_THREADS, smem, st>>>(
            (const double *)X, ldx, n_q, d, nodes, roots, n_trees, out_codes, out_ids, ld_out);
    }
    return cudaGetLastError();
}

}  // namespace sk
