// Batched all-pairs shortest path lengths of small graphs: replaces util.all_pairs_shortest_paths (src/util.py:101-110,
// networkx all_pairs_dijkstra_path_length; call sites gnn_offloading_agent.py:286-287,304-305, AdHoc_test.py:135-136,
// AdHoc_train.py:134-135) - the largest CPU cost of a rollout step (SURVEY 8f #2).
//
// One CTA per graph, one THREAD per source node: the sources are independent single-source problems, so thread s owns
// column s of the n x n fp64 distance matrix (column-major in shared memory for n <= 167: neighbouring lanes hit
// neighbouring banks; larger graphs work in the output block) and relaxes it to the fixed point
//     d[s][v] = min_u fl(d[s][u] + w(u,v)),   d[s][s] = 0,
// from +inf, sweeping v = 0..n-1 in place until a sweep changes nothing (no data is shared between threads: no races,
// no block barriers; the warp moves in lockstep through the CSR).  It is the system Dijkstra's algorithm solves, with
// the same left-to-right path sums, so the results are bit-identical to the reference's (fl(a + w) is monotone in a;
// weights > 0).  weight == NULL: hop counts.  The graph must be stored with both directions of every edge
// (undirected, like env.graph_c).
#include <cfloat>
#include <cstdint>

#include "mho_common.cuh"
#include "mho_internal.h"

namespace {

constexpr int APSP_THREADS = 128;

struct ApspParams {
    const int32_t* node_off;
    const int32_t* rowptr;
    const int32_t* colidx;
    const double* weight;   // nullable
    const int64_t* out_off;
    double* dist;
    int smem_nodes;         // graphs up to this size run in shared memory
};

__global__ void __launch_bounds__(APSP_THREADS) apsp_kernel(const __grid_constant__ ApspParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int g = blockIdx.x, tid = threadIdx.x;
    const int n0 = p.node_off[g], n = p.node_off[g + 1] - n0;
    if (n <= 0) return;
    double* out = p.dist + p.out_off[g];
    const bool in_smem = n <= p.smem_nodes;
    double* d = in_smem ? reinterpret_cast<double*>(smem_raw) : out;
    // element (source s, node v): shared memory is column-major [v][s]; the output block is row-major [s][v]
    const int sv = in_smem ? 1 : n, vv = in_smem ? n : 1;
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    const int32_t* rp = p.rowptr + n0;
    for (int s = tid; s < n; s += APSP_THREADS) {
        double* col = d + (size_t)s * sv;
        for (int v = 0; v < n; ++v) col[(size_t)v * vv] = (v == s) ? 0.0 : inf;
        for (int sweep = 0; sweep < n; ++sweep) {   // a sweep that changes nothing ends it; at most n - 1 can change anything
            bool changed = false;
            for (int v = 0; v < n; ++v) {
                if (v == s) continue;
                const double cur = col[(size_t)v * vv];
                double best = cur;
                const int e1 = rp[v + 1];
                for (int e = rp[v]; e < e1; ++e) {
                    const int u = p.colidx[e] - n0;
                    const double cand = col[(size_t)u * vv] + (p.weight ? p.weight[e] : 1.0);
                    best = cand < best ? cand : best;
                }
                if (best < cur) { col[(size_t)v * vv] = best; changed = true; }
            }
            if (!changed) break;
        }
    }
    if (in_smem) {
        __syncthreads();
        for (int i = tid; i < n * n; i += APSP_THREADS) {
            const int s = i / n, v = i - s * n;
            out[i] = d[(size_t)v * n + s];
        }
    }
}

}  // namespace

cudaError_t apsp_launch(int n_graphs, const int32_t* node_off, const int32_t* rowptr, const int32_t* colidx, const double* weight,
                        const int64_t* out_off, double* dist, int max_smem_optin, cudaStream_t st) {
    ApspParams p{node_off, rowptr, colidx, weight, out_off, dist, 0};
    int nodes = 0;
    while ((size_t)(nodes + 1) * (nodes + 1) * 8 <= (size_t)max_smem_optin) ++nodes;
    p.smem_nodes = nodes;
    const size_t smem = (size_t)nodes * nodes * 8;
    return mho_launch<apsp_kernel>(dim3((unsigned)n_graphs), dim3(APSP_THREADS), smem, st, false, p);
}
