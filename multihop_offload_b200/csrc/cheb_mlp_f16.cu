// Fused forward of a stack of K = 1 ChebConv layers (sm_100a, tcgen05 + TMEM + bulk copies) - the model the reference
// actually ships and runs: ACOAgent._build_model with Spektral's default K = 1 (gnn_offloading_agent.py:81-123, executed at
// :149): 4 -> 32 -> 32 -> 32 -> 32 -> 1, leaky_relu x 4 + relu.  With K = 1 a ChebConv layer never touches the operator:
// Y = act(X W_0 + b) per node, so a batch is just rows, cut into 128-row tiles that ignore graph boundaries.
//
// One CTA (8 warps; thread = one row x 16 of the 32 columns) takes a tile through every layer without leaving the SM:
//   layer input (registers) -> per-row power-of-two scale (row maximum: the two threads of a row meet through shared memory
//   behind a 64-thread barrier) -> two fp16 parts (x = h - l', 22 significand bits) into a SWIZZLE_128B part tile ->
//   hardware barrier, thread 0 issues the 3 part products x 2 K slices as tcgen05.mma (N = 16 or 32; a layer of <= 16 inputs
//   needs one K slice) -> tensor memory (32 columns) -> un-scale, bias, activation in packed fp32 -> next layer.
// Round 1 ran this model through cheb_dense_kernel (bf16 x 3 parts, six part products, 16 warps, ~3.5 k cycles per layer and
// tile); this kernel needs ~0.8 k.  Only 32 tensor-memory columns and ~45 KB of shared memory per CTA: four CTAs per SM.
#include <algorithm>
#include <cstdio>
#include <cstring>

#include "mho_common.cuh"
#include "mho_internal.h"
#include "f16_common.cuh"

namespace {

constexpr int MLP_THREADS = 256;
constexpr int MLP_LAYER_BYTES = 32 * 128 + 1024;  // (1024-aligned: SWIZZLE_128B atoms) weight rows [o][h 64 B | l' 64 B] (K dim = input feature), bias row, header

struct MlpParams {
    BatchDev b;
    const float* X;
    float* Y;
    float* saved;               // nullable: the inputs of layers 1.. (activations kept for the VJP)
    const unsigned char* wimg;  // n_layers x MLP_LAYER_BYTES
    int n_layers;
    int f_in0;                  // multiple of 4
    int f_out_last;
    int fi[MHO_MAX_LAYERS], fo[MHO_MAX_LAYERS], act[MHO_MAX_LAYERS];
    float slope[MHO_MAX_LAYERS];
    long long saved_off[MHO_MAX_LAYERS];   // element offset of layer l's INPUT inside `saved` (l >= 1)
    int total_nodes;
    int stage_bytes;            // 16 KB staging tile for rows that leave as whole 128 B lines (only when some f_out == 32 leaves)
};

struct MlpPrepParams { int n_layers; LayerDev layers[MHO_MAX_LAYERS]; unsigned char* out; };

// per layer: W[0][f][o] scaled by a power of two (max |w'| in [2^13, 2^14)) as fp16 h | l' rows (row = output o, the
// K dimension is the input feature f, zero-padded to 32), SWIZZLE_128B; bias row; header [0] = 1 / scale
__global__ void __launch_bounds__(256) mlp_prepare_weights_kernel(const __grid_constant__ MlpPrepParams p) {
    __shared__ float red[256];
    __shared__ float s_scale;
    const LayerDev& L = p.layers[blockIdx.x];
    unsigned char* img = p.out + (size_t)blockIdx.x * MLP_LAYER_BYTES;
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
        unsigned char* row = img + (size_t)o * 128;
        const uint32_t ch = (uint32_t)f >> 3, key = (uint32_t)o & 7u;
        *reinterpret_cast<__half*>(row + ((ch ^ key) << 4) + (f & 7) * 2) = h;
        *reinterpret_cast<__half*>(row + (((4u + ch) ^ key) << 4) + (f & 7) * 2) = l;
    }
    float* bias = reinterpret_cast<float*>(img + 32 * 128);
    if (tid < 32) bias[tid] = (L.b != nullptr && tid < L.f_out) ? __ldg(L.b + tid) : 0.f;
    if (tid == 32) bias[32] = 1.f / sc;
}

__global__ void __launch_bounds__(MLP_THREADS, 4) cheb_mlp_f16_kernel(const __grid_constant__ MlpParams p) {
    extern __shared__ __align__(1024) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    // shared memory: part tile 16 KB | [staging tile 16 KB: rows that leave through whole 128 B lines] | weights | control
    // block (full[2] +0, w +16, mma +24, tmem slot +32, tile info +48 ([2][4])) | row maxima [2 layer parities][2 halves][128]
    // | two input buffers of 128 rows x f_in0 floats
    unsigned char* stage_s = smem + HF_TILE_BYTES;
    unsigned char* w_s = stage_s + p.stage_bytes;
    unsigned char* ctl_s = w_s + (size_t)p.n_layers * MLP_LAYER_BYTES;
    const uint32_t parts_a = smem_u32(smem), stage_a = smem_u32(stage_s), w_a = smem_u32(w_s), ctl_a = smem_u32(ctl_s);
    const uint32_t bar_full = ctl_a, bar_w = ctl_a + 16, bar_mma = ctl_a + 24, tslot = ctl_a + 32;
    volatile int* tinfo_s = reinterpret_cast<volatile int*>(ctl_s + 48);
    float* rmax_s = reinterpret_cast<float*>(ctl_s + 128);
    unsigned char* xin_s = ctl_s + 128 + 2048;
    const uint32_t xin_a = smem_u32(xin_s);
    const uint32_t xin_bytes = 128u * (uint32_t)p.f_in0 * 4u;

    const int G = (int)gridDim.x;
    const int n_my = (int)blockIdx.x < p.b.n_tiles ? (p.b.n_tiles - (int)blockIdx.x + G - 1) / G : 0;
    const uint32_t w_bytes = (uint32_t)p.n_layers * MLP_LAYER_BYTES;

    auto issue_load = [&](int j) {   // lane 0 of warp 0
        const int buf = j & 1;
        const int4 ti = __ldg(reinterpret_cast<const int4*>(p.b.tile_info) + ((int)blockIdx.x + j * G));
        tinfo_s[buf * 4 + 0] = ti.x; tinfo_s[buf * 4 + 1] = ti.y;
        const uint32_t nb = (uint32_t)ti.y * (uint32_t)p.f_in0 * 4u;
        mbar_expect_tx(bar_full + 8u * buf, nb);
        bulk_g2s(xin_a + (uint32_t)buf * xin_bytes, p.X + (size_t)ti.x * p.f_in0, nb, bar_full + 8u * buf);
    };

    if (tid == 0) {
        mbar_init(bar_full, 1);
        mbar_init(bar_full + 8, 1);
        mbar_init(bar_w, 1);
        mbar_init(bar_mma, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (warp == 0) {
        __syncwarp();
        if (lane == 0) {
            if (n_my > 0) issue_load(0);
            mbar_expect_tx(bar_w, w_bytes);
            bulk_g2s(w_a, p.wimg, w_bytes, bar_w);
        }
        __syncwarp();
        tmem_alloc(tslot, 32u);
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(ctl_s + 32);

    const int q = warp & 3, hh = warp >> 2;
    const uint32_t r = (uint32_t)(q * 32 + lane);
    const uint32_t tmem_row = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(16 * hh);
    const uint32_t key = r & 7u;
    const uint32_t prow_a = parts_a + r * 128u;
    uint32_t ph_mma = 0;
    mbar_wait(bar_w, 0u);   // weights, biases, scales

    for (int j = 0; j < n_my; ++j) {
        const int buf = j & 1;
        if (tid == 0 && j + 1 < n_my) issue_load(j + 1);   // the other input buffer: its last reader was tile j - 1's first layer
        mbar_wait(bar_full + 8u * buf, (uint32_t)((j >> 1) & 1));
        const int node0 = tinfo_s[buf * 4 + 0], rows = tinfo_s[buf * 4 + 1];
        const bool live = (int)r < rows;

        // ---- layer 0 input: this thread's 16 columns of its row
        float y[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) y[e] = 0.f;
        if (live) {
            const uint32_t xa = xin_a + (uint32_t)buf * xin_bytes + r * (uint32_t)p.f_in0 * 4u;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int col = 16 * hh + 4 * c;
                if (col < p.f_in0) {
                    const float4 v = lds_f128(xa + (uint32_t)col * 4u);
                    y[4 * c] = v.x; y[4 * c + 1] = v.y; y[4 * c + 2] = v.z; y[4 * c + 3] = v.w;
                }
            }
        }

        for (int l = 0; l < p.n_layers; ++l) {
            const int fi = p.fi[l], fo = p.fo[l];
            const unsigned char* wl_s = w_s + (size_t)l * MLP_LAYER_BYTES;
            const uint32_t wl_a = w_a + (uint32_t)l * MLP_LAYER_BYTES;
            const float* bias_s = reinterpret_cast<const float*>(wl_s + 32 * 128);
            // ---- row maximum: the two threads of a row (column halves) meet through shared memory
            float rm = fmaxf(fmaxf(fmaxf(fabsf(y[0]), fabsf(y[1])), fmaxf(fabsf(y[2]), fabsf(y[3]))), fmaxf(fmaxf(fabsf(y[4]), fabsf(y[5])), fmaxf(fabsf(y[6]), fabsf(y[7]))));
            rm = fmaxf(rm, fmaxf(fmaxf(fmaxf(fabsf(y[8]), fabsf(y[9])), fmaxf(fabsf(y[10]), fabsf(y[11]))), fmaxf(fmaxf(fabsf(y[12]), fabsf(y[13])), fmaxf(fabsf(y[14]), fabsf(y[15])))));
            {   // (always: the thread that reads the other 16 output columns un-scales with the same row scale)
                rmax_s[(l & 1) * 256 + hh * 128 + (int)r] = rm;
                bar_quadrant(q);
                rm = fmaxf(rm, rmax_s[(l & 1) * 256 + (hh ^ 1) * 128 + (int)r]);
            }
            int ex = expo_above(rm);
            ex = max(-100, min(110, ex));
            const float s_row = pow2f(15 - ex);
            const float unscale = pow2f(ex - 15) * bias_s[32];   // 1 / (row scale x weight scale)
            // ---- two fp16 parts of the scaled row into the part tile (columns past the layer's input width are zero)
            if (hh == 0 || fi > 16) {
                const uint64_t S2 = pk2(s_row, s_row);
                uint32_t h[8], lo[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    float a0, a1;
                    upk2(mul2(pk2(y[2 * e], y[2 * e + 1]), S2), a0, a1);
                    split2(a0, a1, h[e], lo[e]);
                }
                sts_u128(prow_a + (((uint32_t)(2 * hh) ^ key) << 4), h[0], h[1], h[2], h[3]);
                sts_u128(prow_a + (((uint32_t)(2 * hh + 1) ^ key) << 4), h[4], h[5], h[6], h[7]);
                sts_u128(prow_a + (((uint32_t)(4 + 2 * hh) ^ key) << 4), lo[0], lo[1], lo[2], lo[3]);
                sts_u128(prow_a + (((uint32_t)(5 + 2 * hh) ^ key) << 4), lo[4], lo[5], lo[6], lo[7]);
            }
            fence_proxy_async();
            tc_fence_before();
            bar_compute();
            if (tid == 0) {
                tc_fence_after();
                const uint32_t n = (uint32_t)(fo > 16 ? 32 : 16);
                const uint32_t id_pos = idesc_f16(n, 0u, 0u), id_neg = idesc_f16(n, 0u, 1u);
                const int nks = fi > 16 ? 2 : 1;   // 16-wide K slices of the input features
                // x w ~ xh wh - xh wl' - xl' wh
                for (int ks = 0; ks < nks; ++ks) umma_f16_ss(tmem_base, desc_sw128(parts_a + 64u + 32u * ks), desc_sw128(wl_a + 32u * ks), id_neg, ks > 0 ? 1u : 0u);
                for (int ks = 0; ks < nks; ++ks) umma_f16_ss(tmem_base, desc_sw128(parts_a + 32u * ks), desc_sw128(wl_a + 64u + 32u * ks), id_neg, 1u);
                for (int ks = 0; ks < nks; ++ks) umma_f16_ss(tmem_base, desc_sw128(parts_a + 32u * ks), desc_sw128(wl_a + 32u * ks), id_pos, 1u);
                umma_commit(bar_mma);
            }
            mbar_wait(bar_mma, ph_mma);
            ph_mma ^= 1u;
            tc_fence_after();
            // ---- this thread's 16 output columns: un-scale, bias, activation
            const bool has_cols = 16 * hh < fo;
            if (fo > 16 || hh == 0) {   // (the warps of the other column half skip the load: uniform per warp)
                uint32_t v[16];
                tmem_ld16(tmem_row, v);
                tmem_wait_ld_();
                const uint64_t U2 = pk2(unscale, unscale);
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const float4 bv = *reinterpret_cast<const float4*>(bias_s + 16 * hh + 4 * c);
                    upk2(fma2(pk2(__uint_as_float(v[4 * c]), __uint_as_float(v[4 * c + 1])), U2, pk2(bv.x, bv.y)), y[4 * c], y[4 * c + 1]);
                    upk2(fma2(pk2(__uint_as_float(v[4 * c + 2]), __uint_as_float(v[4 * c + 3])), U2, pk2(bv.z, bv.w)), y[4 * c + 2], y[4 * c + 3]);
                }
                const int a = p.act[l];
                if (a == MHO_ACT_RELU) {
#pragma unroll
                    for (int e = 0; e < 16; ++e) y[e] = fmaxf(y[e], 0.f);
                } else if (a == MHO_ACT_LEAKY) {
                    const float sl = p.slope[l];
#pragma unroll
                    for (int e = 0; e < 16; ++e) y[e] = y[e] > 0.f ? y[e] : sl * y[e];
                }
#pragma unroll
                for (int e = 0; e < 16; ++e)
                    if (!live || 16 * hh + e >= fo) y[e] = 0.f;
            } else {
#pragma unroll
                for (int e = 0; e < 16; ++e) y[e] = 0.f;
            }
            (void)has_cols;
            tc_fence_before();   // this thread's TMEM reads are done before the next layer's UMMAs overwrite the columns

            // ---- rows that leave the SM: the activations kept for the VJP (hidden layers), the output (last layer)
            const bool last = l == p.n_layers - 1;
            float* gout = last ? p.Y : (p.saved != nullptr ? p.saved + p.saved_off[l + 1] : nullptr);
            if (gout != nullptr) {
                if (fo == 32 && p.stage_bytes != 0 && (reinterpret_cast<uintptr_t>(gout) & 15u) == 0) {
                    // whole 128 B lines through the staging tile
                    const uint32_t ya = stage_a + r * 128u;
#pragma unroll
                    for (int c = 0; c < 4; ++c) sts_f128(ya + (((uint32_t)(4 * hh + c) ^ key) << 4), make_float4(y[4 * c], y[4 * c + 1], y[4 * c + 2], y[4 * c + 3]));
                    bar_quadrant(q);
                    float* dst = gout + (size_t)node0 * 32;
#pragma unroll
                    for (int pp = 0; pp < 4; ++pp) {
                        const uint32_t row = (uint32_t)(32 * q + 16 * hh + 4 * pp) + ((uint32_t)lane >> 3), ch = (uint32_t)lane & 7u;
                        if ((int)row < rows) *reinterpret_cast<float4*>(dst + (size_t)row * 32 + ch * 4) = lds_f128(stage_a + row * 128u + ((ch ^ (row & 7u)) << 4));
                    }
                    bar_quadrant(q);   // the staging rows are rewritten by the next layer that leaves
                } else if (live) {
                    float* dst = gout + (size_t)(node0 + (int)r) * fo + 16 * hh;
#pragma unroll
                    for (int e = 0; e < 16; ++e)
                        if (16 * hh + e < fo) dst[e] = y[e];
                }
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, 32u);
}

}  // namespace

// -------------------------------------------------------------------------------------------
// host side
// -------------------------------------------------------------------------------------------
static size_t mlp_smem_bytes(int n_layers, int f_in0, bool stage) {
    return (size_t)HF_TILE_BYTES + (stage ? (size_t)HF_TILE_BYTES : 0) + (size_t)n_layers * MLP_LAYER_BYTES + 128 + 2048 + (size_t)2 * 128 * f_in0 * 4 + 1024;
}

bool cheb_mlp_eligible(const mho_layer_t* layers, int n_layers, int max_tile_rows, const void* X, int max_smem_optin) {
    if (max_tile_rows > 128 || n_layers < 1) return false;
    for (int l = 0; l < n_layers; ++l)
        if (layers[l].K != 1 || layers[l].f_in > 32 || layers[l].f_out > 32) return false;
    if ((layers[0].f_in & 3) != 0 || (reinterpret_cast<uintptr_t>(X) & 15u) != 0) return false;   // 16 B input rows (bulk copy)
    return mlp_smem_bytes(n_layers, layers[0].f_in, true) <= (size_t)max_smem_optin;
}

int cheb_mlp_weight_bytes(int n_layers) { return n_layers * MLP_LAYER_BYTES; }

cudaError_t prepare_mlp_weights_launch(const LayerDev* layers, int n_layers, unsigned char* out, cudaStream_t st) {
    MlpPrepParams p;
    memset(&p, 0, sizeof(p));
    p.n_layers = n_layers;
    for (int l = 0; l < n_layers; ++l) p.layers[l] = layers[l];
    p.out = out;
    mlp_prepare_weights_kernel<<<n_layers, 256, 0, st>>>(p);
    return cudaGetLastError();
}

cudaError_t cheb_mlp_launch(const FwdParams& fp, const unsigned char* wimg, int num_sms, cudaStream_t st) {
    MlpParams p;
    memset(&p, 0, sizeof(p));
    p.b = fp.b;
    p.X = fp.X; p.Y = fp.Y; p.saved = fp.saved;
    p.wimg = wimg;
    p.n_layers = fp.n_layers;
    p.f_in0 = fp.layers[0].f_in;
    p.f_out_last = fp.layers[fp.n_layers - 1].f_out;
    p.total_nodes = fp.total_nodes;
    for (int l = 0; l < fp.n_layers; ++l) {
        p.fi[l] = fp.layers[l].f_in; p.fo[l] = fp.layers[l].f_out; p.act[l] = fp.layers[l].act; p.slope[l] = fp.layers[l].slope;
        p.saved_off[l] = fp.layers[l].saved_off;
    }
    bool stage = fp.layers[fp.n_layers - 1].f_out == 32;   // the output rows, or kept activations of a 32-wide hidden layer
    for (int l = 0; l + 1 < fp.n_layers; ++l) stage = stage || (fp.saved != nullptr && fp.layers[l].f_out == 32);
    p.stage_bytes = stage ? HF_TILE_BYTES : 0;
    const size_t smem = mlp_smem_bytes(fp.n_layers, p.f_in0, stage);
    int per_sm = (int)((size_t)(227 * 1024) / (smem + 1024));
    per_sm = std::max(1, std::min(per_sm, 4));
    int grid = std::min(num_sms * per_sm, std::max(1, p.b.n_tiles));
    return mho_launch<cheb_mlp_f16_kernel>(dim3((unsigned)grid), dim3(MLP_THREADS), smem, st, true, p);
}
