// VJP of the ChebConv stack for sm_100a: one CTA per graph instance.
//
// Replaces the reference's tape replay
//   gradients = g.gradient(delay_mtx_ts, self.model.trainable_weights, output_gradients=grad_dist_np)
// (src/gnn_offloading_agent.py:448) from the GNN output back to every kernel/bias; the caller has
// already pulled grad_dist through the queue head.  Per layer (SURVEY App. A.4):
//   G    = dOut (.) act'(Out)                      act' from the OUTPUT sign (relu/leaky)
//   db   = sum_i G[i,:]
//   dW_k = T_k^T G                                  T_k recomputed on-chip from the saved input
//   dIn  = sum_k T_k(A^T) (G W_k^T)                 Clenshaw: b_k = U_k + 2 A^T b_{k+1} - b_{k+2},
//                                                   dIn = U_0 + A^T b_1 - b_2
// One gradient vector PER GRAPH is written (the reference memorises one gradient list per
// instance, :142,:450, and replays them one by one, :156-169); a second kernel adds them in a
// fixed order into the buffer a data-parallel all-reduce ships.
//
// Shared memory: three swizzled [rows][32] fp32 tiles - R0/R1 (Chebyshev ring in phase A, Clenshaw
// ring in phase B) and G - plus the staged CSR slice and W^T of the current layer.
#include "mho_common.cuh"
#include "mho_internal.h"

struct BwdParams {
    BatchDev b;
    const int32_t* rowptr_t;  // transpose operator (nullptr => symmetric)
    const int32_t* colidx_t;
    const float* vals_t;
    int n_layers;
    LayerDev layers[MHO_MAX_LAYERS];
    const float* X;
    const float* Y;
    const float* saved;
    const float* dY;
    float* grads;  // [n_graphs, n_params]
    float* dX;     // nullable
    long long n_params;
    int rows_cap;
    int nnz_cap;   // 0 => CSR read from global
    int w_floats_cap;
};

template <bool HAS_VALS, bool STAGED>
__global__ void __launch_bounds__(MHO_THREADS, 4) cheb_backward_kernel(const __grid_constant__ BwdParams p) {
    extern __shared__ __align__(1024) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const size_t tile_bytes = (size_t)p.rows_cap * 128;
    unsigned char* R0 = smem;
    unsigned char* R1 = R0 + tile_bytes;
    unsigned char* Gb = R1 + tile_bytes;
    float* Wt_s = reinterpret_cast<float*>(Gb + tile_bytes);  // [K][fo_pad][32] (f contiguous)
    int* rp_s = reinterpret_cast<int*>(Wt_s + p.w_floats_cap);
    const int rp_words = (p.rows_cap + 1 + 3) & ~3;
    uint32_t* pre_s = reinterpret_cast<uint32_t*>(rp_s + rp_words);
    float* val_s = reinterpret_cast<float*>(pre_s + p.nnz_cap);
    const uint32_t R_a[2] = {smem_u32(R0), smem_u32(R1)};
    const uint32_t G_a = smem_u32(Gb);
    const uint32_t pre_a = smem_u32(pre_s), val_a = smem_u32(val_s);
    const uint32_t key = swz_key((uint32_t)lane);
    const bool symmetric = (p.rowptr_t == nullptr);

    for (int g = blockIdx.x; g < p.b.n_graphs; g += gridDim.x) {
        const int node0 = __ldg(p.b.graph_off + g), node1 = __ldg(p.b.graph_off + g + 1);
        const int rows = node1 - node0;
        const int nz0 = __ldg(p.b.rowptr + node0);
        const int nnz = __ldg(p.b.rowptr + node1) - nz0;
        float* gout = p.grads + (size_t)g * p.n_params;

        __syncthreads();  // previous graph fully done with shared memory
        for (int i = tid; i <= rows; i += MHO_THREADS)
            rp_s[i] = STAGED ? (__ldg(p.b.rowptr + node0 + i) - nz0) : __ldg(p.b.rowptr + node0 + i);
        if (STAGED) {
            for (int e = tid; e < nnz; e += MHO_THREADS) {
                pre_s[e] = swz_row((uint32_t)(__ldg(p.b.colidx + nz0 + e) - node0));
                if (HAS_VALS) val_s[e] = __ldg(p.b.vals + nz0 + e);
            }
        }

        for (int li = p.n_layers - 1; li >= 0; --li) {
            const LayerDev& L = p.layers[li];
            const int fi = L.f_in, fo = L.f_out, K = L.K;
            const bool last = (li == p.n_layers - 1);
            const float* out_g = last ? p.Y : p.saved + p.layers[li + 1].saved_off;   // this layer's output
            const float* in_g = (li == 0) ? p.X : p.saved + L.saved_off;               // this layer's input
            const bool lane_f = lane < fi;

            // ---- G = dOut (.) act'(out); padded columns are zero.  dOut: dY (last) or already in Gb.
            for (int idx = tid; idx < rows * 32; idx += MHO_THREADS) {
                const int r = idx >> 5, c = idx & 31;
                const uint32_t a = G_a + swz_off((uint32_t)r, (uint32_t)c);
                float gval = 0.f;
                if (c < fo) {
                    const float d = last ? __ldg(p.dY + (size_t)(node0 + r) * fo + c) : lds_f32(a);
                    gval = d * act_grad_from_out(__ldg(out_g + (size_t)(node0 + r) * fo + c), L.act, L.slope);
                }
                sts_f32(a, gval);
            }
            // ---- T_0 = layer input
            for (int idx = tid; idx < rows * 32; idx += MHO_THREADS) {
                const int r = idx >> 5, c = idx & 31;
                sts_f32(R_a[0] + swz_off((uint32_t)r, (uint32_t)c), c < fi ? __ldg(in_g + (size_t)(node0 + r) * fi + c) : 0.f);
            }
            __syncthreads();

            // =========================== phase A: db, dW_k ===========================
            // dW_k = T_k^T G as register-blocked rank-1 updates: the rows are dealt to four groups of two warps; inside a
            // group thread j owns the 4 x 4 block (f = 4 (j >> 3).., o = 4 (j & 7)..): two LDS.128 feed 16 FMAs per row.
            // The four partial blocks meet in shared memory (the W^T region, idle until phase B) and are added in a fixed
            // order, one float4 of the result per thread.
            const int rg = warp >> 1, jj = ((warp & 1) << 5) | lane;
            const uint32_t fblk = (uint32_t)(jj >> 3), oblk = (uint32_t)(jj & 7);
            float* red_s = Wt_s;                       // [4 groups][32 f][32 o]
            float* redb_s = Wt_s + 4 * 1024;           // [4 groups][32 o]
            int cur = 0;
            for (int k = 0; k < K; ++k) {
                float acc[4][4], bs[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int a = 0; a < 4; ++a)
#pragma unroll
                    for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
                const uint32_t Tk = R_a[cur];
                for (int i = rg; i < rows; i += 4) {
                    const uint32_t rowa = (uint32_t)i << 7, sw = (uint32_t)i & 7u;
                    const uint4 tq = lds_u128(Tk + rowa + ((fblk ^ sw) << 4));
                    const uint4 gq = lds_u128(G_a + rowa + ((oblk ^ sw) << 4));
                    const float t[4] = {__uint_as_float(tq.x), __uint_as_float(tq.y), __uint_as_float(tq.z), __uint_as_float(tq.w)};
                    const float gg[4] = {__uint_as_float(gq.x), __uint_as_float(gq.y), __uint_as_float(gq.z), __uint_as_float(gq.w)};
#pragma unroll
                    for (int a = 0; a < 4; ++a)
#pragma unroll
                        for (int b = 0; b < 4; ++b) acc[a][b] = fmaf(t[a], gg[b], acc[a][b]);
                    if (k == 0 && fblk == 0u) {
#pragma unroll
                        for (int b = 0; b < 4; ++b) bs[b] += gg[b];
                    }
                }
#pragma unroll
                for (int a = 0; a < 4; ++a)
                    *reinterpret_cast<float4*>(red_s + rg * 1024 + (int)(fblk * 4 + a) * 32 + (int)oblk * 4) =
                        make_float4(acc[a][0], acc[a][1], acc[a][2], acc[a][3]);
                if (k == 0 && fblk == 0u) *reinterpret_cast<float4*>(redb_s + rg * 32 + (int)oblk * 4) = make_float4(bs[0], bs[1], bs[2], bs[3]);
                __syncthreads();
                {
                    const int f = tid >> 3, o4 = (tid & 7) * 4;
                    const float4 p0 = *reinterpret_cast<const float4*>(red_s + f * 32 + o4);
                    const float4 p1 = *reinterpret_cast<const float4*>(red_s + 1024 + f * 32 + o4);
                    const float4 p2 = *reinterpret_cast<const float4*>(red_s + 2048 + f * 32 + o4);
                    const float4 p3 = *reinterpret_cast<const float4*>(red_s + 3072 + f * 32 + o4);
                    const float v[4] = {((p0.x + p1.x) + p2.x) + p3.x, ((p0.y + p1.y) + p2.y) + p3.y,
                                        ((p0.z + p1.z) + p2.z) + p3.z, ((p0.w + p1.w) + p2.w) + p3.w};
                    if (f < fi) {
                        float* dst = gout + L.param_off + ((size_t)k * fi + f) * fo + o4;
#pragma unroll
                        for (int b = 0; b < 4; ++b)
                            if (o4 + b < fo) dst[b] = v[b];
                    }
                    if (k == 0 && tid < 32 && tid < fo)
                        gout[L.param_off + (size_t)K * fi * fo + tid] =
                            ((redb_s[tid] + redb_s[32 + tid]) + redb_s[64 + tid]) + redb_s[96 + tid];
                }
                // T_{k+1} (forward operator A), in place over T_{k-1}
                if (k + 1 < K) {
                    const uint32_t Tsrc = R_a[cur], Tdst = R_a[cur ^ 1];
                    for (int r = warp; r < rows; r += MHO_NWARPS) {
                        if (lane_f) {
                            const float s = gather_row<HAS_VALS, STAGED>(Tsrc, rp_s[r], rp_s[r + 1], pre_a, val_a, p.b.colidx,
                                                                        p.b.vals, node0, key);
                            const uint32_t d = Tdst + (swz_row((uint32_t)r) ^ key);
                            sts_f32(d, k == 0 ? s : 2.f * s - lds_f32(d));
                        }
                    }
                }
                __syncthreads();
                cur ^= 1;
            }

            const bool need_din = (li > 0) || (p.dX != nullptr);
            if (!need_din) continue;

            // =========================== phase B: dIn ===============================
            // W^T of this layer: Wt_s[(k*fo + o)*32 + f] = W[k][f][o]  (lane = f reads conflict-free)
            for (int idx = tid; idx < K * fo * 32; idx += MHO_THREADS) {
                const int f = idx & 31, ko = idx >> 5;
                const int k = ko / fo, o = ko - k * fo;
                Wt_s[idx] = f < fi ? __ldg(L.W + ((size_t)k * fi + f) * fo + o) : 0.f;
            }
            for (int idx = tid; idx < rows * 32; idx += MHO_THREADS) {  // b_{K} = b_{K+1} = 0
                const uint32_t off = swz_off((uint32_t)(idx >> 5), (uint32_t)(idx & 31));
                sts_f32(R_a[0] + off, 0.f);
                sts_f32(R_a[1] + off, 0.f);
            }
            __syncthreads();

            // CSR of A^T: the staged slice when symmetric, else the caller's transpose from global
            const int32_t* tcol = symmetric ? p.b.colidx : p.colidx_t;
            const float* tval = symmetric ? p.b.vals : p.vals_t;
            int bcur = 0;  // R[bcur] holds b_{k+1}, R[bcur^1] holds b_{k+2}
            for (int k = K - 1; k >= 0; --k) {
                const float* Wk = Wt_s + (size_t)k * fo * 32;
                for (int r0 = warp * 4; r0 < rows; r0 += MHO_NWARPS * 4) {
                    float u[4] = {0.f, 0.f, 0.f, 0.f};
                    // U_k[r][f] = sum_o G[r][o] W_k[f][o]
                    for (int oc = 0; oc < fo; oc += 4) {
                        float w[4];
#pragma unroll
                        for (int j = 0; j < 4; ++j) w[j] = (oc + j < fo) ? Wk[(oc + j) * 32 + lane] : 0.f;
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const uint32_t r = (uint32_t)(r0 + q);
                            if ((int)r < rows) {
                                const uint4 gq = lds_u128(G_a + (r << 7) + ((((uint32_t)(oc >> 2)) ^ (r & 7u)) << 4));
                                u[q] = fmaf(__uint_as_float(gq.x), w[0], u[q]);
                                u[q] = fmaf(__uint_as_float(gq.y), w[1], u[q]);
                                u[q] = fmaf(__uint_as_float(gq.z), w[2], u[q]);
                                u[q] = fmaf(__uint_as_float(gq.w), w[3], u[q]);
                            }
                        }
                    }
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int r = r0 + q;
                        if (r < rows && lane_f) {
                            float s = 0.f;
                            if (K > 1) {
                                if (symmetric) {
                                    s = gather_row<HAS_VALS, STAGED>(R_a[bcur], rp_s[r], rp_s[r + 1], pre_a, val_a, tcol, tval,
                                                                    node0, key);
                                } else {
                                    s = gather_row<HAS_VALS, false>(R_a[bcur], __ldg(p.rowptr_t + node0 + r),
                                                                   __ldg(p.rowptr_t + node0 + r + 1), 0, 0, tcol, tval, node0, key);
                                }
                            }
                            const uint32_t d = R_a[bcur ^ 1] + (swz_row((uint32_t)r) ^ key);
                            if (k > 0) {
                                sts_f32(d, u[q] + 2.f * s - lds_f32(d));       // b_k over b_{k+2}
                            } else {
                                u[q] = (K > 1) ? u[q] + s - lds_f32(d) : u[q];  // dIn = U_0 + A^T b_1 - b_2
                            }
                        }
                    }
                    if (k == 0) {
                        // all G reads of these 4 rows are done (u complete): overwrite G rows with dIn
                        __syncwarp();
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const int r = r0 + q;
                            if (r < rows) {
                                sts_f32(G_a + (swz_row((uint32_t)r) ^ key), lane_f ? u[q] : 0.f);
                                if (li == 0 && p.dX != nullptr && lane_f) p.dX[(size_t)(node0 + r) * fi + lane] = u[q];
                            }
                        }
                    }
                }
                __syncthreads();
                bcur ^= 1;
            }
        }
    }
}

// deterministic sum over graphs, out[p] = sum_g grads[g][p], in two fixed-order stages so that enough loads are in
// flight: slice s of MHO_SUM_SLICES sums its run of graphs (4 independent chains), then the slices are added in order.
#define MHO_SUM_SLICES 32
__global__ void grads_sum_stage1(const float* __restrict__ grads, float* __restrict__ part, int n_graphs, long long n_params) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_params) return;
    const int per = (n_graphs + MHO_SUM_SLICES - 1) / MHO_SUM_SLICES;
    const int g0 = blockIdx.y * per, g1 = min(g0 + per, n_graphs);
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    int g = g0;
    for (; g + 4 <= g1; g += 4) {
        s0 += grads[(size_t)(g + 0) * n_params + p];
        s1 += grads[(size_t)(g + 1) * n_params + p];
        s2 += grads[(size_t)(g + 2) * n_params + p];
        s3 += grads[(size_t)(g + 3) * n_params + p];
    }
    for (; g < g1; ++g) s0 += grads[(size_t)g * n_params + p];
    part[(size_t)blockIdx.y * n_params + p] = (s0 + s1) + (s2 + s3);
}
__global__ void grads_sum_stage2(const float* __restrict__ part, float* __restrict__ out, long long n_params) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_params) return;
    float s = 0.f;
#pragma unroll 8
    for (int i = 0; i < MHO_SUM_SLICES; ++i) s += part[(size_t)i * n_params + p];
    out[p] = s;
}

// One-launch variant for parameter counts that are multiples of 4 (every 32-wide layer): float4 columns, 32 slices of
// graphs summed with 8 loads in flight, and the LAST block of each column group (a self re-arming counter) adds the 32
// slice sums in slice order - the result does not depend on which block that is.
#define MHO_SUM_SLICES4 32
__global__ void __launch_bounds__(128) grads_sum_fused(const float4* __restrict__ grads, float4* part, float4* __restrict__ out, unsigned int* counters,
                                                        int n_graphs, int n_params4) {
    const int col = blockIdx.x * 128 + threadIdx.x;
    const int per = (n_graphs + MHO_SUM_SLICES4 - 1) / MHO_SUM_SLICES4;
    const int g0 = blockIdx.y * per, g1 = min(g0 + per, n_graphs);
    if (col < n_params4) {
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
        int g = g0;
        for (; g + 8 <= g1; g += 8) {
            float4 v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = __ldcs(grads + (size_t)(g + i) * n_params4 + col);
#pragma unroll
            for (int i = 0; i < 8; ++i) { s.x += v[i].x; s.y += v[i].y; s.z += v[i].z; s.w += v[i].w; }
        }
        for (; g < g1; ++g) { const float4 v = __ldcs(grads + (size_t)g * n_params4 + col); s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w; }
        __stcg(part + (size_t)blockIdx.y * n_params4 + col, s);
    }
    __threadfence();
    __syncthreads();
    __shared__ int last_s;
    if (threadIdx.x == 0) {
        const unsigned int t = atomicAdd(counters + blockIdx.x, 1u);
        last_s = (t == (unsigned int)(MHO_SUM_SLICES4 - 1));
        if (last_s) counters[blockIdx.x] = 0u;   // re-armed for the next call (stream order)
    }
    __syncthreads();
    if (!last_s) return;
    __threadfence();
    if (col < n_params4) {
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int i0 = 0; i0 < MHO_SUM_SLICES4; i0 += 16) {
            float4 v[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = __ldcg(part + (size_t)(i0 + i) * n_params4 + col);
#pragma unroll
            for (int i = 0; i < 16; ++i) { s.x += v[i].x; s.y += v[i].y; s.z += v[i].z; s.w += v[i].w; }
        }
        out[col] = s;
    }
}

static size_t bwd_smem_bytes(int rows_cap, int nnz_cap, int w_floats, bool has_vals) {
    size_t s = (size_t)rows_cap * 128 * 3 + (size_t)w_floats * 4;
    s += (size_t)((rows_cap + 1 + 3) & ~3) * 4;
    s += (size_t)nnz_cap * 4 * (has_vals ? 2 : 1);
    return s + 16;
}

template <bool HAS_VALS, bool STAGED>
static cudaError_t launch_bwd(const BwdParams& p, int grid, size_t smem, cudaStream_t st) {
    return mho_launch<cheb_backward_kernel<HAS_VALS, STAGED>>(dim3((unsigned)grid), dim3(MHO_THREADS), smem, st, false, p);
}

extern "C" int mho_cheb_backward(mho_ctx_t* c, const mho_batch_t* b, const mho_layer_t* layers, int32_t n_layers,
                                 const float* X, const float* Y, const void* saved, const float* dY,
                                 float* grads_per_graph, float* grads_sum, float* dX, mho_stream_t stream) {
    if (!c || !b) { mho_set_error("mho_cheb_backward: NULL argument"); return MHO_ERR_INVALID; }
    int rc = validate_layers(layers, n_layers, "mho_cheb_backward");
    if (rc) return rc;
    if (b->tile_off != nullptr) { mho_set_error("mho_cheb_backward: needs a one-graph-per-tile batch (tile_off == NULL)"); return MHO_ERR_INVALID; }
    if (!b->graph_off || !b->rowptr) { mho_set_error("mho_cheb_backward: invalid batch"); return MHO_ERR_INVALID; }
    const int64_t P = mho_param_count(layers, n_layers);
    cudaStream_t st = (cudaStream_t)stream;
    if (cudaSetDevice(c->device) != cudaSuccess) { mho_set_error("cudaSetDevice failed"); return MHO_ERR_CUDA; }
    if (b->n_graphs == 0 || b->total_nodes == 0) {
        if (grads_sum) cudaMemsetAsync(grads_sum, 0, (size_t)P * 4, st);
        if (grads_per_graph && b->n_graphs > 0) cudaMemsetAsync(grads_per_graph, 0, (size_t)P * 4 * b->n_graphs, st);
        return MHO_OK;
    }
    if (!X || !Y || !dY || !grads_per_graph || (n_layers > 1 && !saved)) { mho_set_error("mho_cheb_backward: X/Y/dY/grads/saved is NULL"); return MHO_ERR_INVALID; }
    if ((b->rowptr_t == nullptr) != (b->colidx_t == nullptr)) { mho_set_error("mho_cheb_backward: rowptr_t/colidx_t must both be set or both NULL"); return MHO_ERR_INVALID; }
    if (b->max_tile_rows < 1) { mho_set_error("mho_cheb_backward: batch.max_tile_rows must be the largest graph"); return MHO_ERR_INVALID; }

    // the tensor-core VJPs write the per-graph gradient rows; otherwise the CUDA-core kernel below does
    bool rows_written = false;
    if (cheb_backward_f16_eligible(b, layers, n_layers, X, Y, dY, dX, c->max_smem_optin)) {
        cudaError_t e = cheb_backward_f16_launch(b, layers, X, Y, dY, grads_per_graph, (long long)P, c->num_sms, st);
        if (e != cudaSuccess) { mho_set_error("cheb_backward_f16 launch failed: %s", cudaGetErrorString(e)); return MHO_ERR_CUDA; }
        c->launches += 1;
        rows_written = true;
    } else if (cheb_mlp_backward_eligible(b, layers, n_layers, X, saved, dX, c->max_smem_optin)) {
        // K = 1 stack (the shipped model): tensor-core VJP with cached W^T images
        LayerDev ld[MHO_MAX_LAYERS];
        mho_fill_layers(layers, n_layers, b->total_nodes, ld);
        auto& img = c->img[MHO_IMG_MLP_BWD];
        rc = ensure_image(c, img, layers, n_layers, (size_t)cheb_mlp_backward_weight_bytes(n_layers), "prepare_mlp_backward_weights",
                          [&](unsigned char* out) { return prepare_mlp_backward_weights_launch(ld, n_layers, out, st); });
        if (rc) return rc;
        cudaError_t e = cheb_mlp_backward_launch(b, ld, n_layers, X, Y, (const float*)saved, dY, grads_per_graph, (long long)P, img.ptr, c->num_sms, st);
        if (e != cudaSuccess) { mho_set_error("cheb_mlp_backward launch failed: %s", cudaGetErrorString(e)); return MHO_ERR_CUDA; }
        c->launches += 1;
        rows_written = true;
    }
    BwdParams p;
    memset(&p, 0, sizeof(p));
    p.b.graph_off = b->graph_off; p.b.rowptr = b->rowptr; p.b.colidx = b->colidx; p.b.vals = b->vals;
    p.b.tile_off = nullptr; p.b.tile_info = nullptr; p.b.n_graphs = b->n_graphs; p.b.n_tiles = b->n_graphs;
    p.rowptr_t = b->rowptr_t; p.colidx_t = b->colidx_t; p.vals_t = b->vals_t;
    p.n_layers = n_layers;
    mho_fill_layers(layers, n_layers, b->total_nodes, p.layers);
    p.X = X; p.Y = Y; p.saved = (const float*)saved; p.dY = dY; p.grads = grads_per_graph; p.dX = dX;
    p.n_params = P;
    p.rows_cap = pad16(b->max_tile_rows < 16 ? 16 : b->max_tile_rows);
    if (p.rows_cap > MHO_MAX_TILE_ROWS) { mho_set_error("mho_cheb_backward: graph of %d nodes exceeds %d", b->max_tile_rows, MHO_MAX_TILE_ROWS); return MHO_ERR_TOO_LARGE; }
    int wf = 0;
    for (int l = 0; l < n_layers; ++l) { int v = layers[l].K * layers[l].f_out * 32; wf = v > wf ? v : wf; }
    if (wf < 4 * 1024 + 128) wf = 4 * 1024 + 128;   // also the phase-A reduction scratch: 4 partial 32 x 32 blocks + 4 bias rows
    p.w_floats_cap = wf;
    const bool has_vals = b->vals != nullptr;
    if (has_vals && b->rowptr_t && !b->vals_t) { mho_set_error("mho_cheb_backward: vals_t missing for a weighted non-symmetric operator"); return MHO_ERR_INVALID; }
    bool staged = true;
    int nnz_cap = (b->max_tile_nnz + 3) & ~3;
    size_t smem = bwd_smem_bytes(p.rows_cap, nnz_cap, wf, has_vals);
    if (smem > (size_t)c->max_smem_optin) {
        staged = false; nnz_cap = 0;
        smem = bwd_smem_bytes(p.rows_cap, 0, wf, has_vals);
        if (smem > (size_t)c->max_smem_optin) {
            mho_set_error("mho_cheb_backward: graph of %d nodes with K*f_out*32=%d weights needs %zu B of shared memory (> %d)",
                          b->max_tile_rows, wf, smem, c->max_smem_optin);
            return MHO_ERR_TOO_LARGE;
        }
    }
    p.nnz_cap = nnz_cap;
    int per_sm = (int)((size_t)(228 * 1024) / (smem + 1024));
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 4) per_sm = 4;   // 56-64 registers x 256 threads: four CTAs fit the register file
    int grid = c->num_sms * per_sm;
    if (grid > b->n_graphs) grid = b->n_graphs;
    cudaError_t e = cudaSuccess;
    if (!rows_written) {
        if (has_vals) e = staged ? launch_bwd<true, true>(p, grid, smem, st) : launch_bwd<true, false>(p, grid, smem, st);
        else e = staged ? launch_bwd<false, true>(p, grid, smem, st) : launch_bwd<false, false>(p, grid, smem, st);
        if (e != cudaSuccess) { mho_set_error("cheb_backward launch failed: %s", cudaGetErrorString(e)); return MHO_ERR_CUDA; }
        c->launches += 1;
    }
    if (grads_sum) {
        const int threads = 128;
        const bool vec4 = (P % 4 == 0) && ((reinterpret_cast<uintptr_t>(grads_per_graph) | reinterpret_cast<uintptr_t>(grads_sum)) & 15u) == 0;
        if (vec4) {
            const int P4 = (int)(P / 4);
            const int nblk = (P4 + threads - 1) / threads;
            // scratch: one counter per column group (4 KB at a fixed place: zeroed when the slot is (re)allocated, self re-arming
            // after that), then the slice sums
            const size_t cnt_bytes = 4096;
            if ((size_t)nblk * sizeof(unsigned int) > cnt_bytes) { mho_set_error("mho_cheb_backward: %lld parameters exceed the reduction's column groups", (long long)P); return MHO_ERR_TOO_LARGE; }
            const size_t need = cnt_bytes + (size_t)MHO_SUM_SLICES4 * P * sizeof(float);
            const bool fresh = c->scratch.size() <= 2 || c->scratch[2].bytes < need;
            unsigned char* sc = (unsigned char*)mho_scratch(c, 2, need);
            if (!sc) { mho_set_error("mho_cheb_backward: cudaMalloc of the reduction scratch failed"); return MHO_ERR_CUDA; }
            if (fresh && cudaMemsetAsync(sc, 0, cnt_bytes, st) != cudaSuccess) { mho_set_error("mho_cheb_backward: memset failed"); return MHO_ERR_CUDA; }
            grads_sum_fused<<<dim3((unsigned)nblk, MHO_SUM_SLICES4), threads, 0, st>>>((const float4*)grads_per_graph, (float4*)(sc + cnt_bytes), (float4*)grads_sum,
                                                                                     (unsigned int*)sc, b->n_graphs, P4);
            e = cudaGetLastError();
            if (e != cudaSuccess) { mho_set_error("grads_sum launch failed: %s", cudaGetErrorString(e)); return MHO_ERR_CUDA; }
            c->launches += 1;
        } else {
            float* part = (float*)mho_scratch(c, 1, (size_t)MHO_SUM_SLICES * P * sizeof(float));
            if (!part) { mho_set_error("mho_cheb_backward: cudaMalloc of the reduction scratch failed"); return MHO_ERR_CUDA; }
            const dim3 g1((unsigned)((P + threads - 1) / threads), MHO_SUM_SLICES);
            grads_sum_stage1<<<g1, threads, 0, st>>>(grads_per_graph, part, b->n_graphs, P);
            grads_sum_stage2<<<g1.x, threads, 0, st>>>(part, grads_sum, P);
            e = cudaGetLastError();
            if (e != cudaSuccess) { mho_set_error("grads_sum launch failed: %s", cudaGetErrorString(e)); return MHO_ERR_CUDA; }
            c->launches += 2;
        }
    }
    return MHO_OK;
}
