// VJP of a stack of K = 1 ChebConv layers on the tensor cores (sm_100a, tcgen05 + TMEM) - the training step of the model the
// reference ships and trains (ACOAgent._build_model with Spektral's default K = 1, gnn_offloading_agent.py:81-123; the tape replay
//   gradients = g.gradient(delay_mtx_ts, self.model.trainable_weights, output_gradients=grad_dist_np)   (:448) ).
// Shapes: every layer K = 1, hidden widths 32, first f_in a multiple of 4, last f_out <= 4, graphs of <= 128 nodes, no input
// gradient; every other stack stays with cheb_backward.cu.  One gradient vector PER GRAPH (:142 / :450).
//
// With K = 1 a layer is Out = act(In W + b) per node; per graph and layer, from the last layer down:
//   G = dOut (.) act'(Out)      db = sum_i G[i, :]      dW = In^T G      dIn = G W^T   (= dOut of the layer below)
// One graph per CTA pass, two CTAs per SM, thread = one node row x 16 of the 32 columns (8 warps).  Per layer:
//   * the layer's input rows (the activations the forward kept) arrive by cp.async in a rotating set of three staging tiles
//     (16 B chunks XOR-swizzled with the row); a thread reads its 16 fp32 values ONCE: they become two fp16 parts IN PLACE (the
//     staging tile turns into the part tile [node][h 64 B | l' 64 B]), and their signs are kept in a register: act' of the
//     layer below needs nothing else;
//   * max |G| and max |In| of the graph are reduced across the CTA (shared-memory atomics + one barrier): ONE power-of-two scale
//     per graph, layer and operand (the node rows are the reduction dimension of In^T G);
//   * dW^T = G^T In: one UMMA per 16-node slice, A = the part tile of G read MN-major (rows of D: [G_h o | G_l' o]), B = the part
//     tile of In (columns of D: [In_h f | In_l' f]); the four 32 x 32 blocks of D are the four part products;
//     dIn = G W^T: the same part tile of G read K-major (A), B = the prepared W^T image (rows f, K = o): g w ~ gh wh - gh wl' -
//     gl' wh, 3 x (f_out / 16) UMMAs of N = 32.  Both groups are issued together and waited for once;
//   * dIn comes back from tensor memory as the next G (times act' from the kept signs); the dW accumulator is drained by the two
//     lane quadrants that hold it (exchange through shared memory, coalesced rows of the gradient vector); db: exact fp32 column
//     sums by warp butterflies, added in a fixed order.
// Tensor memory: 64 columns dW | 32 columns dIn -> 128 allocated.
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <type_traits>

#include "mho_common.cuh"
#include "mho_internal.h"
#include "f16_common.cuh"

#ifdef MHO_PROBE
#define MPROBE(id) do { if (blockIdx.x == 0 && tid == 0 && mpn < 120) { mprobe_s[mpn] = (clock64() << 8) | (long long)(id); ++mpn; } } while (0)
#else
#define MPROBE(id) do { } while (0)
#endif

namespace {

constexpr int MB_THREADS = 256;
constexpr int MB_MAX_LAYERS = 6;
constexpr uint32_t MB_TCOLS = 128u, MB_DIN_COL = 64u;
constexpr int MB_WT_BYTES = 32 * 128 + 1024;   // W^T rows f: [h over o 64 B | l' over o 64 B] (SWIZZLE_128B), then header [0] = 1 / scale
constexpr int MB_SMALL_FLOATS = 128 * 4;       // Y / dY rows of one graph (f_out_last <= 4)

struct MbParams {
    const int32_t* graph_off;
    int n_graphs;
    const float* X;
    const float* Y;
    const float* dY;
    const float* saved;
    float* grads;
    long long n_params;
    const unsigned char* wT;   // n_layers images of MB_WT_BYTES
    int n_layers;
    int fi[MB_MAX_LAYERS], fo[MB_MAX_LAYERS], act[MB_MAX_LAYERS];
    float slope[MB_MAX_LAYERS];
    long long saved_off[MB_MAX_LAYERS], param_off[MB_MAX_LAYERS];
};

struct MbPrepParams { int n_layers; LayerDev layers[MB_MAX_LAYERS]; unsigned char* out; };

// per layer: W[0][f][o] scaled by a power of two (max |w'| in [2^13, 2^14)) as fp16 h | l' rows f (the N index of dIn = G W^T;
// the K dimension is the output feature o, zero-padded to 32), SWIZZLE_128B; header [0] = 1 / scale
__global__ void __launch_bounds__(256) mlpT_prepare_weights_kernel(const __grid_constant__ MbPrepParams p) {
    __shared__ float red[256];
    __shared__ float s_scale;
    const LayerDev& L = p.layers[blockIdx.x];
    unsigned char* img = p.out + (size_t)blockIdx.x * MB_WT_BYTES;
    const int tid = threadIdx.x, total = L.f_in * L.f_out;
    float m = 0.f;
    for (int i = tid; i < total; i += 256) m = fmaxf(m, fabsf(__ldg(L.W + i)));
    red[tid] = m;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (tid < s) red[tid] = fmaxf(red[tid], red[tid + s]);
        __syncthreads();
    }
    if (tid == 0) {
        const float wmax = red[0];
        int e = (wmax > 0.f && wmax < 3.0e38f) ? expo_above(wmax) : 14;
        e = max(-100, min(100, e));
        s_scale = pow2f(14 - e);
    }
    __syncthreads();
    const float sc = s_scale;
    for (int i = tid; i < 32 * 32; i += 256) {
        const int f = i >> 5, o = i & 31;
        const float w = (f < L.f_in && o < L.f_out) ? __ldg(L.W + (size_t)f * L.f_out + o) * sc : 0.f;
        const __half h = __float2half_rn(w);
        const __half l = __float2half_rn(__half2float(h) - w);
        unsigned char* row = img + (size_t)f * 128;
        const uint32_t ch = (uint32_t)o >> 3, key = (uint32_t)f & 7u;
        *reinterpret_cast<__half*>(row + ((ch ^ key) << 4) + (o & 7) * 2) = h;
        *reinterpret_cast<__half*>(row + (((4u + ch) ^ key) << 4) + (o & 7) * 2) = l;
    }
    if (tid == 0) reinterpret_cast<float*>(img + 32 * 128)[0] = 1.f / sc;
}

__device__ __forceinline__ void mb_bar_drain() { asm volatile("bar.sync 6, 128;" ::: "memory"); }
__device__ __forceinline__ void mb_bar_drain_arrive() { asm volatile("bar.arrive 6, 128;" ::: "memory"); }

__global__ void __launch_bounds__(MB_THREADS, 2) cheb_mlp_backward_f16_kernel(const __grid_constant__ MbParams p) {
    extern __shared__ __align__(1024) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int L = p.n_layers;
    // shared memory (1024-aligned): G part tile | three staging / part tiles | W^T images | Y, dY rows [2 graphs] | drain staging |
    // control block
    const uint32_t smem_a = smem_u32(smem);
    const uint32_t pg_a = smem_a, t_a = smem_a + HF_TILE_BYTES, w_a = smem_a + 4u * HF_TILE_BYTES;
    unsigned char* w_s = smem + 4 * HF_TILE_BYTES;
    unsigned char* small_s = w_s + (size_t)L * MB_WT_BYTES;                 // [2][Y | dY][MB_SMALL_FLOATS]
    float* stg_s = reinterpret_cast<float*>(small_s + 4 * MB_SMALL_FLOATS * 4);   // [32][32]
    unsigned char* ctl_s = reinterpret_cast<unsigned char*>(stg_s + 1024);
    const uint32_t small_a = smem_u32(small_s), ctl_a = smem_u32(ctl_s);
    // control block: tile loads [3] +0, small loads [2] +24, weights +40, mma +48, tmem slot +56, reductions +64 ([2][2]), db
    // partials +128 ([4][32])
    const uint32_t bar_t = ctl_a, bar_small = ctl_a + 24, bar_w = ctl_a + 40, bar_mma = ctl_a + 48, tslot = ctl_a + 56;
    unsigned int* red_s = reinterpret_cast<unsigned int*>(ctl_s + 64);
    float* dbs_s = reinterpret_cast<float*>(ctl_s + 128);

#ifdef MHO_PROBE
    __shared__ long long mprobe_s[128];
    int mpn = 0;
    if (tid < 128) mprobe_s[tid] = 0;
    __syncthreads();
#endif
    const int G = (int)gridDim.x;
    const int n_my = (int)blockIdx.x < p.n_graphs ? (p.n_graphs - (int)blockIdx.x + G - 1) / G : 0;
    const int n_items = n_my * L;   // item s = (graph s / L, layer L - 1 - s % L)

    // input rows of item s -> staging tile s % 3
    auto issue_tile = [&](int s) {   // all threads
        if (s < n_items) {
            const int g = (int)blockIdx.x + (s / L) * G, l = L - 1 - s % L;
            const int node0 = __ldg(p.graph_off + g), rows = __ldg(p.graph_off + g + 1) - node0;
            const int fi = p.fi[l], cpr = fi >> 2;
            const float* src = l == 0 ? p.X + (size_t)node0 * fi : p.saved + p.saved_off[l] + (size_t)node0 * fi;
            const uint32_t dst = t_a + (uint32_t)(s % 3) * HF_TILE_BYTES;
#pragma unroll
            for (int i = 0; i < 4; ++i) {   // 128 rows x 8 chunk slots
                const int row = (tid >> 3) + 32 * i, ch = tid & 7;
                if (row < rows && ch < cpr)
                    cp_async16(dst + (uint32_t)row * 128u + (uint32_t)((ch ^ (row & 7)) << 4), src + (size_t)row * fi + (size_t)ch * 4);
            }
        }
        cp_async_mbar_arrive(bar_t + 8u * (uint32_t)(s % 3));
    };
    auto issue_small = [&](int j) {   // Y and dY rows of graph j
        if (j < n_my) {
            const int g = (int)blockIdx.x + j * G;
            const int node0 = __ldg(p.graph_off + g), rows = __ldg(p.graph_off + g + 1) - node0;
            const int fo = p.fo[L - 1];
            const uint32_t dst = small_a + (uint32_t)(j & 1) * (2u * MB_SMALL_FLOATS * 4u);
            for (int c = tid; c < rows * fo; c += MB_THREADS) {
                cp_async4(dst + (uint32_t)c * 4u, p.Y + (size_t)node0 * fo + c);
                cp_async4(dst + MB_SMALL_FLOATS * 4u + (uint32_t)c * 4u, p.dY + (size_t)node0 * fo + c);
            }
        }
        cp_async_mbar_arrive(bar_small + 8u * (uint32_t)(j & 1));
    };

    if (tid == 0) {
        mbar_init(bar_t, MB_THREADS);
        mbar_init(bar_t + 8, MB_THREADS);
        mbar_init(bar_t + 16, MB_THREADS);
        mbar_init(bar_small, MB_THREADS);
        mbar_init(bar_small + 8, MB_THREADS);
        mbar_init(bar_w, 1);
        mbar_init(bar_mma, 2);   // the dW group (thread 0) and the dIn group (thread 32)
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (tid < 4) red_s[tid] = 0u;
    if (warp == 0) tmem_alloc(tslot, MB_TCOLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(ctl_s + 56);
    if (tid == 0) {
        mbar_expect_tx(bar_w, (uint32_t)(L * MB_WT_BYTES));
        bulk_g2s(w_a, p.wT, (uint32_t)(L * MB_WT_BYTES), bar_w);
    }
    issue_small(0);
    issue_small(1);
    issue_tile(0);
    issue_tile(1);
    issue_tile(2);

    const int q = warp & 3, hh = warp >> 2;
    const uint32_t r = (uint32_t)(q * 32 + lane);
    const uint32_t tmem_lane = tmem_base + ((uint32_t)(q * 32) << 16);
    const uint32_t key = r & 7u;
    uint32_t ph_mma = 0;
    mbar_wait(bar_w, 0u);

    auto split_row = [&](uint32_t tile_a, const float (&v)[16], float scale) {
        const uint64_t S2 = pk2(scale, scale);
        uint32_t h[8], l[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            float y0, y1;
            upk2(mul2(pk2(v[2 * e], v[2 * e + 1]), S2), y0, y1);
            split2(y0, y1, h[e], l[e]);
        }
        const uint32_t prow_a = tile_a + r * 128u;
        sts_u128(prow_a + (((uint32_t)(2 * hh) ^ key) << 4), h[0], h[1], h[2], h[3]);
        sts_u128(prow_a + (((uint32_t)(2 * hh + 1) ^ key) << 4), h[4], h[5], h[6], h[7]);
        sts_u128(prow_a + (((uint32_t)(4 + 2 * hh) ^ key) << 4), l[0], l[1], l[2], l[3]);
        sts_u128(prow_a + (((uint32_t)(5 + 2 * hh) ^ key) << 4), l[4], l[5], l[6], l[7]);
    };

    float g[16];   // this thread's 16 columns of G of the current layer
#pragma unroll
    for (int e = 0; e < 16; ++e) g[e] = 0.f;
    int node0 = 0, rows = 0;
    float* gout = p.grads;

    // one item = one layer of one graph.  FULL: a 32 -> 32 layer (every predicate on the widths folds away)
    auto item = [&](int s, auto full_tag) {
        constexpr bool FULL = decltype(full_tag)::value;
        const int j = s / L, l = L - 1 - s % L;
        const int fi = FULL ? 32 : p.fi[l], fo = FULL ? 32 : p.fo[l];
        const uint32_t tile_a = t_a + (uint32_t)(s % 3) * HF_TILE_BYTES;
        if (l == L - 1) {
            // ---- a new graph: G of the last layer from dY and Y
            const int gi = (int)blockIdx.x + j * G;
            node0 = __ldg(p.graph_off + gi);
            rows = __ldg(p.graph_off + gi + 1) - node0;
            gout = p.grads + (size_t)gi * p.n_params;
            mbar_wait(bar_small + 8u * (uint32_t)(j & 1), (uint32_t)((j >> 1) & 1));
            const float* ys = reinterpret_cast<const float*>(small_s) + (j & 1) * 2 * MB_SMALL_FLOATS;
            const float* ds = ys + MB_SMALL_FLOATS;
#pragma unroll
            for (int e = 0; e < 16; ++e) {
                const int c = 16 * hh + e;
                g[e] = ((int)r < rows && c < fo) ? ds[r * fo + c] * act_grad_from_out(ys[r * fo + c], p.act[l], p.slope[l]) : 0.f;
            }
        }
        const bool live = (int)r < rows;
        const int nks = (rows + 15) >> 4;

        // ---- this layer's input rows: 16 fp32 values of this thread's row, their signs (act' of the layer below), the maxima
        MPROBE(1);
        mbar_wait(bar_t + 8u * (uint32_t)(s % 3), (uint32_t)((s / 3) & 1));
        MPROBE(2);
        float v[16];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int col = 16 * hh + 4 * c;
            float4 x4 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (live && col < fi) x4 = lds_f128(tile_a + r * 128u + (((uint32_t)(4 * hh + c) ^ key) << 4));
            v[4 * c] = x4.x; v[4 * c + 1] = x4.y; v[4 * c + 2] = x4.z; v[4 * c + 3] = x4.w;
        }
        unsigned int pos = 0u;
        float vm = 0.f, gm = 0.f;
#pragma unroll
        for (int e = 0; e < 16; ++e) {
            pos |= (v[e] > 0.f ? 1u : 0u) << e;
            vm = fmaxf(vm, fabsf(v[e]));
            gm = fmaxf(gm, fabsf(g[e]));
        }
        {
            const unsigned int wg = __reduce_max_sync(0xffffffffu, __float_as_uint(gm));
            const unsigned int wv = __reduce_max_sync(0xffffffffu, __float_as_uint(vm));
            unsigned int* red = red_s + (s & 1) * 2;
            if (lane == 0) { atomicMax(red, wg); atomicMax(red + 1, wv); }
        }
        // db: column sums of this warp's 32 rows (butterfly: 16 -> 8 -> 4 -> 2 -> 1 values per lane), fixed order
        {
            float s8[8], s4[4], s2[2], s1;
            const bool b16 = lane & 16, b8 = lane & 8, b4 = lane & 4, b2 = lane & 2;
#pragma unroll
            for (int i = 0; i < 8; ++i) { const float o = __shfl_xor_sync(0xffffffffu, b16 ? g[i] : g[i + 8], 16); s8[i] = (b16 ? g[i + 8] : g[i]) + o; }
#pragma unroll
            for (int i = 0; i < 4; ++i) { const float o = __shfl_xor_sync(0xffffffffu, b8 ? s8[i] : s8[i + 4], 8); s4[i] = (b8 ? s8[i + 4] : s8[i]) + o; }
#pragma unroll
            for (int i = 0; i < 2; ++i) { const float o = __shfl_xor_sync(0xffffffffu, b4 ? s4[i] : s4[i + 2], 4); s2[i] = (b4 ? s4[i + 2] : s4[i]) + o; }
            { const float o = __shfl_xor_sync(0xffffffffu, b2 ? s2[0] : s2[1], 2); s1 = (b2 ? s2[1] : s2[0]) + o; }
            s1 += __shfl_xor_sync(0xffffffffu, s1, 1);
            const int col = (b16 ? 8 : 0) + (b8 ? 4 : 0) + (b4 ? 2 : 0) + (b2 ? 1 : 0);
            if (!(lane & 1)) dbs_s[q * 32 + 16 * hh + col] = s1;
        }
        MPROBE(3);
        bar_compute();   // #1: the maxima are complete; every thread has read its fp32 input values (the tile is rewritten in place)
        const unsigned int* red = red_s + (s & 1) * 2;
        const int eg = max(-100, min(110, expo_above(__uint_as_float(red[0]))));
        const int ei = max(-100, min(110, expo_above(__uint_as_float(red[1]))));
        if (tid == 0) { unsigned int* o = red_s + ((s + 1) & 1) * 2; o[0] = 0u; o[1] = 0u; }
        split_row(pg_a, g, pow2f(15 - eg));
        split_row(tile_a, v, pow2f(15 - ei));
        fence_proxy_async();
        tc_fence_before();
        MPROBE(4);
        bar_compute();   // #2
        MPROBE(5);
        if (tid == 0) {
            tc_fence_after();
            // dW^T = G^T In: A = the G part tile MN-major, B = the In part tile MN-major, one UMMA per 16-node slice
            const uint32_t id_dw = idesc_f16(64u, 1u, 0u) | (1u << 15);
#pragma unroll
            for (int ks = 0; ks < 8; ++ks)
                if (ks == 0 || ks < nks) umma_f16_ss(tmem_base, desc_sw128(pg_a + (uint32_t)ks * 2048u), desc_sw128(tile_a + (uint32_t)ks * 2048u), id_dw, ks > 0 ? 1u : 0u);
            umma_commit(bar_mma);
        } else if (tid == 32) {
            // a second issuing thread: the two groups are independent and an issuing thread stalls until its group is accepted
            tc_fence_after();
            if (l > 0) {
                // dIn = G W^T:  g w ~ gh wh - gh wl' - gl' wh, 16-wide K slices over the output features
                const uint32_t wl_a = w_a + (uint32_t)l * MB_WT_BYTES;
                const uint32_t id_pos = idesc_f16(32u, 0u, 0u), id_neg = idesc_f16(32u, 0u, 1u);
                const uint32_t d = tmem_base + MB_DIN_COL;
                const int nko = fo > 16 ? 2 : 1;
                for (int ks = 0; ks < nko; ++ks) umma_f16_ss(d, desc_sw128(pg_a + 64u + 32u * ks), desc_sw128(wl_a + 32u * ks), id_neg, ks > 0 ? 1u : 0u);
                for (int ks = 0; ks < nko; ++ks) umma_f16_ss(d, desc_sw128(pg_a + 32u * ks), desc_sw128(wl_a + 64u + 32u * ks), id_neg, 1u);
                for (int ks = 0; ks < nko; ++ks) umma_f16_ss(d, desc_sw128(pg_a + 32u * ks), desc_sw128(wl_a + 32u * ks), id_pos, 1u);
                umma_commit(bar_mma);
            } else {
                mbar_arrive(bar_mma);   // (no input gradient for the first layer: the second arrival of this phase)
            }
        }
        if (tid < 32 && tid < fo)
            gout[p.param_off[l] + (long long)fi * fo + tid] = ((dbs_s[tid] + dbs_s[32 + tid]) + dbs_s[64 + tid]) + dbs_s[96 + tid];
        MPROBE(6);
        mbar_wait(bar_mma, ph_mma);
        ph_mma ^= 1u;
        tc_fence_after();
        MPROBE(7);
        issue_tile(s + 3);   // this item's tile is free: the rows of the layer three items ahead (possibly of the next graphs)
        if (l == 0) issue_small(j + 2);   // (buffer j & 1: last read at the top of this graph)

        MPROBE(8);
        // ---- dW accumulator -> gradient rows.  D rows: [G_h o | G_l' o] (lanes 0-31 / 32-63), D columns: [In_h f | In_l' f]
        if (q < 2) {
            uint32_t a[16], b[16];
            tmem_ld16(tmem_lane + (uint32_t)(16 * hh), a);
            tmem_ld16(tmem_lane + 32u + (uint32_t)(16 * hh), b);
            tmem_wait_ld_();
            float w[16];
#pragma unroll
            for (int e = 0; e < 16; ++e) w[e] = __uint_as_float(a[e]) - __uint_as_float(b[e]);
            float* st = stg_s + (16 * hh) * 32 + lane;
            if (q == 1) {
#pragma unroll
                for (int e = 0; e < 16; ++e) st[e * 32] = w[e];
                mb_bar_drain_arrive();
            } else {
                mb_bar_drain();
                const float us = pow2f(eg - 15) * pow2f(ei - 15);
                float* dst = gout + p.param_off[l] + lane;   // W[f][o]: f * fo + o
                if (lane < fo) {
#pragma unroll
                    for (int e = 0; e < 16; ++e)
                        if (16 * hh + e < fi) dst[(size_t)(16 * hh + e) * fo] = (w[e] - st[e * 32]) * us;
                }
            }
        }
        MPROBE(10);
        // ---- dIn = the dOut of the layer below; times act' of that layer (from the signs of its output = this layer's input)
        if (l > 0) {
            uint32_t d16[16];
            tmem_ld16(tmem_lane + MB_DIN_COL + (uint32_t)(16 * hh), d16);
            tmem_wait_ld_();
            const float un = pow2f(eg - 15) * reinterpret_cast<const float*>(w_s + (size_t)l * MB_WT_BYTES + 32 * 128)[0];
            const int a_below = p.act[l - 1];
            const float sl = p.slope[l - 1];
#pragma unroll
            for (int e = 0; e < 16; ++e) {
                const float d = (live && 16 * hh + e < fi) ? __uint_as_float(d16[e]) * un : 0.f;
                const bool on = (pos >> e) & 1u;
                g[e] = a_below == MHO_ACT_RELU ? (on ? d : 0.f) : a_below == MHO_ACT_LEAKY ? (on ? d : sl * d) : d;
            }
        }
        tc_fence_before();   // this thread's tensor-memory reads precede the next item's UMMAs (behind its barriers)
        MPROBE(9);
    };
    for (int s = 0; s < n_items; ++s) {
        const int l = L - 1 - s % L;
        if (p.fi[l] == 32 && p.fo[l] == 32) item(s, std::true_type{}); else item(s, std::false_type{});
    }
#ifdef MHO_PROBE
    __syncthreads();
    if (blockIdx.x == 0 && tid == 0) {
        const long long base = mprobe_s[0] >> 8;
        for (int i = 0; i < 128; ++i) if (mprobe_s[i]) printf("m %2d t %7lld\n", (int)(mprobe_s[i] & 255), (mprobe_s[i] >> 8) - base);
    }
#endif

    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, MB_TCOLS);
}

size_t mb_smem_bytes(int n_layers) {
    return (size_t)4 * HF_TILE_BYTES + (size_t)n_layers * MB_WT_BYTES + 4 * MB_SMALL_FLOATS * 4 + 4096 + 1024;
}

}  // namespace

// -------------------------------------------------------------------------------------------
// host side
// -------------------------------------------------------------------------------------------
bool cheb_mlp_backward_eligible(const mho_batch_t* b, const mho_layer_t* layers, int n_layers, const void* X, const void* saved, const void* dX,
                                int max_smem_optin) {
    if (n_layers < 2 || n_layers > MB_MAX_LAYERS || dX != nullptr || saved == nullptr || b->max_tile_rows > 128) return false;
    for (int l = 0; l < n_layers; ++l) {
        if (layers[l].K != 1) return false;
        if (l > 0 && layers[l].f_in != 32) return false;
        if (l + 1 < n_layers && layers[l].f_out != 32) return false;
    }
    if ((layers[0].f_in & 3) != 0 || layers[0].f_in > 32 || layers[n_layers - 1].f_out > 4) return false;
    if ((reinterpret_cast<uintptr_t>(X) & 15u) != 0 || (reinterpret_cast<uintptr_t>(saved) & 15u) != 0) return false;
    return mb_smem_bytes(n_layers) + 1024 <= (size_t)std::min(max_smem_optin, (228 * 1024) / 2 - 1024);
}

int cheb_mlp_backward_weight_bytes(int n_layers) { return n_layers * MB_WT_BYTES; }

cudaError_t prepare_mlp_backward_weights_launch(const LayerDev* layers, int n_layers, unsigned char* out, cudaStream_t st) {
    MbPrepParams p;
    memset(&p, 0, sizeof(p));
    p.n_layers = n_layers;
    for (int l = 0; l < n_layers; ++l) p.layers[l] = layers[l];
    p.out = out;
    // the kernel writes the W^T rows, not the padding of each layer's block
    const cudaError_t e = cudaMemsetAsync(out, 0, (size_t)n_layers * MB_WT_BYTES, st);
    if (e != cudaSuccess) return e;
    mlpT_prepare_weights_kernel<<<n_layers, 256, 0, st>>>(p);
    return cudaGetLastError();
}

cudaError_t cheb_mlp_backward_launch(const mho_batch_t* b, const LayerDev* layers, int n_layers, const float* X, const float* Y, const float* saved,
                                     const float* dY, float* grads, long long n_params, const unsigned char* wT, int num_sms, cudaStream_t st) {
    MbParams p;
    memset(&p, 0, sizeof(p));
    p.graph_off = b->graph_off;
    p.n_graphs = b->n_graphs;
    p.X = X; p.Y = Y; p.dY = dY; p.saved = saved;
    p.grads = grads;
    p.n_params = n_params;
    p.wT = wT;
    p.n_layers = n_layers;
    for (int l = 0; l < n_layers; ++l) {
        p.fi[l] = layers[l].f_in; p.fo[l] = layers[l].f_out; p.act[l] = layers[l].act; p.slope[l] = layers[l].slope;
        p.saved_off[l] = layers[l].saved_off; p.param_off[l] = layers[l].param_off;
    }
    const size_t smem = mb_smem_bytes(n_layers) + 1024;
    const int grid = std::min(2 * num_sms, std::max(1, p.n_graphs));
    return mho_launch<cheb_mlp_backward_f16_kernel>(dim3((unsigned)grid), dim3(MB_THREADS), smem, st, false, p);
}
