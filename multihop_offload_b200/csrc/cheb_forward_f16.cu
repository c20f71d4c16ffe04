// ChebConv layer forward, second-generation tensor-core kernel (sm_100a, tcgen05 + TMEM + bulk async copies) for the
// workload the benchmark and the reference's K > 1 models run: ONE layer, 32 -> 32 features, 2 <= K <= 10, BINARY
// operator (vals == NULL), tiles of <= 128 nodes.  Replaces model([x_in, a_in]) of gnn_offloading_agent.py:149
// (spektral ChebConv of :95-110) for those shapes; everything else stays with cheb_forward_dense.cu / cheb_forward.cu.
//
// Same mathematics as cheb_forward_dense.cu (dense 128 x 128 adjacency block on the tensor core, Clenshaw recurrence
//      P_k = X W_k,   B_K-1 = P_K-1,   B_k = P_k + 2 A B_k+1 - B_k+2,   out = act(P_0 + A B_1 - B_2 + bias) ),
// re-engineered around what the first kernel's profile showed (28 % tensor pipe, 57 % issue slots, 18 k warp
// instructions per tile):
//   * fp32 operands travel as TWO fp16 parts (x = h - l', h = rn16(x), l' = rn16(h - x): 22 significand bits) after a
//     power-of-two scale per GRAPH and per Clenshaw step that keeps every part inside fp16's range.  The scales come
//     from an upper bound of max |B_k| (graph max |X|, per-k weight norms from the prepared image, the graph's max degree;
//     for K > 5 the running maxima of |B_k| themselves), never from the data of the step itself: no extra barrier.
//     X W needs 3 part products instead of 6 (h h, h l, l h; 2^-22), the adjacency UMMA has N = 64 instead of 96, a
//     split costs 2 instructions per element (F2FP + FHADD, mixed-precision subtract) instead of 5.5.
//   * one thread owns 16 accumulator columns of its row (8 compute warps per tile instead of 16): per-thread overheads
//     (addresses, waits, fences, loop control) are paid once per 16 elements.
//   * all warps of the eight-warp kernel meet at a hardware named barrier; thread 0 then issues the UMMA group and commits
//     to one mbarrier every thread waits on; warp 0 also issues the 1-D bulk copies (cp.async.bulk -> mbarrier complete_tx)
//     that bring the NEXT tile's input rows and adjacency bit rows into the other staging buffer.  (A ninth, dedicated issuer
//     warp costs two CTAs per SM their registers; the warp-specialised variant further down - cheb_f16ws_kernel, 12 warps
//     with setmaxnreg - is what K <= 5 batches with bit rows run through.)
//   * the adjacency products are never accumulated onto P_k (the per-step scale differs): the UMMA overwrites two
//     consumed column blocks, so nothing has to be cleared.
// Tensor memory: K * 32 columns P, 32 spare, 64 adjacency (fp16 pairs) = 256 for K <= 5 -> two CTAs per SM; the tensor
// pipe sees two independent issuers (one per CTA).  Measured cost of this UMMA (tools/umma_probe3.cu): 57-63 cycles on an
// idle GPU, 84 with every SM busy.
#include <cuda_fp16.h>
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <type_traits>

#include "mho_common.cuh"
#include "mho_internal.h"
#include "f16_common.cuh"

// -DMHO_PROBE: CTAs 0 and gridDim.x - 1 record clock64 marks (compute thread 0 and the control lane) and print them
#ifdef MHO_PROBE
#define PROBE_C(id) do { if (probe_on && tid == 0 && pn_c < 120) { probe_s[pn_c] = (clock64() << 8) | (long long)(id); ++pn_c; } } while (0)
#define PROBE_M(id) do { if (probe_on && lane == 0 && pn_m < 60) { probe_s[128 + pn_m] = (clock64() << 8) | (long long)(id); ++pn_m; } } while (0)
#else
#define PROBE_C(id) do { } while (0)
#define PROBE_M(id) do { } while (0)
#endif

namespace {

constexpr int HF_COMPUTE_THREADS = 256;
constexpr int HF_THREADS = 256;         // 8 compute warps (no dedicated issuer: the last warp to arrive issues the UMMAs)

struct HfParams {
    BatchDev b;
    const float* X;
    float* Y;
    const unsigned char* wimg;  // [32 K rows x 128 B: W'_k[o][f] as fp16 h | l][bias row 128 B][header 128 B]
    int act;
    float slope;
    int use_bits;     // the batch carries adjacency bit rows
    int nnz_cap;      // CSR staging capacity in ints (multiple of 4), 0 with bit rows
    int stage_bytes;  // bytes of one operator staging set (multiple of 16)
};

__host__ __device__ constexpr int hf_w_bytes(int K) { return ((32 * K * 128 + 256) + 1023) & ~1023; }

// ---- weight image ---------------------------------------------------------------------------------------------------
// rows n = k * 32 + o (K-major operand rows of X W), 128 B each: [h: 32 fp16 over f][l' : 32 fp16 over f], 16 B chunks
// XOR-swizzled with (n & 7) (SWIZZLE_128B).  Weights are scaled by a power of two so that max |w'| is in [2^13, 2^14).
// Then the bias row (32 fp32) and a header: [0] = 1 / scale, [1 + k] = max_o sum_f |w'_k[f][o]| (bound of |x' W'_k| / max |x'|).
struct HfPrepParams { const float* W; const float* b; int K; unsigned char* out; };

__global__ void __launch_bounds__(256) hf_prepare_weights_kernel(const HfPrepParams p) {
    __shared__ float red[256];
    __shared__ float s_scale;
    __shared__ float colsum[MHO_MAX_K * 32];
    const int tid = threadIdx.x;
    const int total = p.K * 32 * 32;
    float m = 0.f;
    for (int i = tid; i < total; i += 256) m = fmaxf(m, fabsf(__ldg(p.W + i)));
    red[tid] = m;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (tid < s) red[tid] = fmaxf(red[tid], red[tid + s]);
        __syncthreads();
    }
    if (tid == 0) {
        const float wmax = red[0];
        int e = (wmax > 0.f && wmax < 3.0e38f) ? expo_above(wmax) : 14;   // wmax < 2^e
        e = max(-100, min(100, e));
        s_scale = pow2f(14 - e);                                           // wmax * scale < 2^14
    }
    __syncthreads();
    const float sc = s_scale;
    for (int i = tid; i < total; i += 256) {
        const int k = i >> 10, f = (i >> 5) & 31, o = i & 31;   // W[k][f][o], o fastest: coalesced
        const float w = __ldg(p.W + i) * sc;
        const __half h = __float2half_rn(w);
        const __half l = __float2half_rn(__half2float(h) - w);   // stored negated like the activations' low part: w = h - l'
        const uint32_t n = (uint32_t)(k * 32 + o);
        unsigned char* row = p.out + (size_t)n * 128;
        const uint32_t ch = (uint32_t)f >> 3, key = n & 7u;
        *reinterpret_cast<__half*>(row + ((ch ^ key) << 4) + (f & 7) * 2) = h;
        *reinterpret_cast<__half*>(row + (((4u + ch) ^ key) << 4) + (f & 7) * 2) = l;
    }
    // column sums of |w'| per (k, o)
    for (int i = tid; i < p.K * 32; i += 256) {
        const int k = i >> 5, o = i & 31;
        float s = 0.f;
        for (int f = 0; f < 32; ++f) s += fabsf(__ldg(p.W + ((size_t)k * 32 + f) * 32 + o) * sc);
        colsum[i] = s;
    }
    __syncthreads();
    float* bias = reinterpret_cast<float*>(p.out + (size_t)p.K * 32 * 128);
    float* hdr = bias + 32;
    if (tid < 32) bias[tid] = p.b ? __ldg(p.b + tid) : 0.f;
    if (tid == 32) hdr[0] = 1.f / sc;
    if (tid >= 64 && tid < 64 + p.K) {
        const int k = tid - 64;
        float mx = 0.f;
        for (int o = 0; o < 32; ++o) mx = fmaxf(mx, colsum[k * 32 + o]);
        hdr[1 + k] = mx * 1.01f + 1e-30f;   // slack for the rounding of the parts
    }
}

// ---- the kernel ---------------------------------------------------------------------------------------------------------
// One tile in flight per CTA, two CTAs per SM (K <= 5; one CTA with 512 tensor-memory columns for K > 5).  Per tile:
//   [end of the previous tile: arrive for this tile's X W group - its part tile was written a tile ago]
//   epilogue of the previous tile and this tile's adjacency expansion run under the X W group;
//   X W done -> scales, B_K-1 = P_K-1 / row scale, split, arrive;   next tile's input rows are split into the OTHER part
//   tile inside the wait window of a Clenshaw step;   steps k = K-2 .. 0: wait, LDTM, recurrence (packed fp32), split, arrive.
template <int K>
__global__ void __launch_bounds__(HF_THREADS, (K <= 5 ? 2 : 1)) cheb_f16_kernel(const __grid_constant__ HfParams p) {
    extern __shared__ __align__(1024) unsigned char smem[];
    constexpr bool TRACK = K > 5;   // Clenshaw step scales from the running maxima of |B_k| (K <= 5: the a-priori bounds suffice)
    constexpr int W_BYTES = hf_w_bytes(K);
    constexpr uint32_t TCOLS = (K <= 5) ? 256u : 512u;
    constexpr uint32_t ADJ_COL = TCOLS - 64u;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#ifdef MHO_PROBE
    __shared__ long long probe_s[192];
    const bool probe_on = blockIdx.x == 0 || blockIdx.x == gridDim.x - 1;
    int pn_c = 0, pn_m = 0;
    if (tid < 192) probe_s[tid] = 0;
    __syncthreads();
    unsigned long long gt0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt0));
#endif
    PROBE_C(1);

    // ---- shared memory carve-up: two part tiles | two staging tiles | weights | control block | LUT | masks | operator staging
    unsigned char* w_s = smem + 4 * HF_TILE_BYTES;
    unsigned char* ctl_s = w_s + W_BYTES;            // 1536 B
    unsigned char* lut_s = ctl_s + 1536;             // 16 x 8 B: four adjacency bits -> four fp16 (0 / 1)
    unsigned char* mask_s = lut_s + 128;             // 2 x 2 KB bit rows built from a CSR slice
    unsigned char* op_s = mask_s + 4096;             // two operator staging sets
    unsigned char* grp_s = op_s + 2 * p.stage_bytes; // per-graph scales: [2][132] graph starts, [3][4] start flags, [3][128] max |x|, [3][128] max degree
    const uint32_t smem_a = smem_u32(smem), xs_a = smem_a + 2u * HF_TILE_BYTES, w_a = smem_u32(w_s), ctl_a = smem_u32(ctl_s), lut_a = smem_u32(lut_s),
                   mask_a = smem_u32(mask_s), op_a = smem_u32(op_s);
    // control block: full[2] +0, empty[2] +16, parts +32, mma +40, tmem slot +48, tile info +64 ([buf][4]), reductions +96 ([3][2]),
    // running maxima +128 ([3][16]), row scales +512 ([2][128] floats)
    const uint32_t bar_full = ctl_a, bar_empty = ctl_a + 16, bar_w = ctl_a + 32, bar_mma = ctl_a + 40, tslot = ctl_a + 48;
    volatile int* tinfo_s = reinterpret_cast<volatile int*>(ctl_s + 64);
    unsigned int* red_s = reinterpret_cast<unsigned int*>(ctl_s + 96);
    unsigned int* track_s = reinterpret_cast<unsigned int*>(ctl_s + 128);
    float* rowscale_s = reinterpret_cast<float*>(ctl_s + 512);
    const uint32_t gb_a = smem_u32(grp_s);                                          // graph starts of the staged tiles
    unsigned int* gmax_s = reinterpret_cast<unsigned int*>(grp_s + 1056 + 64);      // max |x| (float bits) per graph of the tile
    unsigned int* gdeg_s = gmax_s + 3 * 128;                                        // max degree per graph of the tile
    const bool groups = p.b.tile_graph0 != nullptr;

    const int G = (int)gridDim.x;
    const int n_my = (int)blockIdx.x < p.b.n_tiles ? (p.b.n_tiles - (int)blockIdx.x + G - 1) / G : 0;

    // tile descriptors are fetched one tile ahead (registers of warp 0): the loads that depend on them - the bulk copies, the
    // graph starts - are issued without waiting for global memory
    int4 ti_pref = make_int4(0, 0, 0, 0);
    int g0_pref = 0, pref_j = -1;
    auto prefetch_desc = [&](int j) {
        if (j < n_my) {
            ti_pref = __ldg(reinterpret_cast<const int4*>(p.b.tile_info) + ((int)blockIdx.x + j * G));
            if (groups) g0_pref = __ldg(p.b.tile_graph0 + ((int)blockIdx.x + j * G));
            pref_j = j;
        }
    };
    auto issue_load = [&](int j) {   // all of warp 0
        const int buf = j & 1;
        if (pref_j != j) prefetch_desc(j);
        const int4 ti = ti_pref;
        const int g0 = g0_pref;
        prefetch_desc(j + 1);
        const uint32_t fb = bar_full + 8u * buf;
        const uint32_t opb = op_a + (uint32_t)(buf * p.stage_bytes);
        if (lane == 0) {
            tinfo_s[buf * 4 + 0] = ti.x; tinfo_s[buf * 4 + 1] = ti.y; tinfo_s[buf * 4 + 2] = ti.z; tinfo_s[buf * 4 + 3] = ti.w;
            const uint32_t xb = (uint32_t)ti.y * 128u;
            mbar_expect_tx(fb, xb + (p.use_bits ? (uint32_t)ti.y * 16u : 0u));
            bulk_g2s(xs_a + (uint32_t)buf * HF_TILE_BYTES, p.X + (size_t)ti.x * 32, xb, fb);
            if (p.use_bits) bulk_g2s(opb, p.b.adj_bits + (size_t)ti.x * 4, (uint32_t)ti.y * 16u, fb);
        }
        if (!p.use_bits) {
            // CSR slice: row pointers at opb, column ids 132 ints further (4 B alignment only: cp.async, not a bulk copy)
            for (int i = lane; i <= ti.y; i += 32) cp_async4(opb + (uint32_t)i * 4u, p.b.rowptr + ti.x + i);
            for (int e = lane; e < ti.w; e += 32) cp_async4(opb + 528u + (uint32_t)e * 4u, p.b.colidx + ti.z + e);
        }
        if (groups) {
            // node offsets of the graphs that follow the tile's first one (at most 128 start inside a 128-row tile)
            for (int e = lane; e < 128; e += 32) {
                const int gi = min(g0 + 1 + e, p.b.n_graphs);   // graph_off[n_graphs] = total_nodes: beyond every tile
                cp_async4(gb_a + (uint32_t)(buf * 132 + e) * 4u, p.b.graph_off + gi);
            }
        }
        if (!p.use_bits || groups) cp_async_mbar_arrive(fb);
    };

    if (tid == 0) {
        const uint32_t full_count = (p.use_bits && !groups) ? 1u : 33u;   // expect_tx arrive (+ one cp.async arrive per lane of warp 0)
        mbar_init(bar_full, full_count);
        mbar_init(bar_full + 8, full_count);
        mbar_init(bar_empty, 8);
        mbar_init(bar_empty + 8, 8);
        mbar_init(bar_mma, 1);
        mbar_init(bar_w, 1);      // the weight image (one bulk copy)
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (tid < 16) {
        const uint32_t x = ((tid & 1) ? 0x3C00u : 0u) | ((tid & 2) ? 0x3C000000u : 0u), y = ((tid & 4) ? 0x3C00u : 0u) | ((tid & 8) ? 0x3C000000u : 0u);
        asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(lut_a + (uint32_t)tid * 8u), "r"(x), "r"(y) : "memory");
    }
    if (tid < 104) reinterpret_cast<unsigned int*>(ctl_s + 96)[tid] = 0u;   // reductions and running maxima
    for (int i = tid; i < 6 * 128; i += HF_COMPUTE_THREADS) gmax_s[i] = 0u;   // per-graph maxima
    asm volatile("griddepcontrol.wait;" ::: "memory");   // from here on global memory written by earlier launches in the stream is read
    if (warp == 0) {
        __syncwarp();
        if (n_my > 0) issue_load(0);   // the first tile's loads fly during the rest of the set-up
        if (lane == 0) {               // the weight image is first needed by the first X W group / the first scales: one bulk
            mbar_expect_tx(bar_w, (uint32_t)W_BYTES);   // copy, waited for where it is used, not here
            bulk_g2s(w_a, p.wimg, (uint32_t)W_BYTES, bar_w);
        }
        tmem_alloc(tslot, TCOLS);
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(ctl_s + 48);
    PROBE_C(2);
    PROBE_M(2);

    {
        // =========================== compute warps ===========================
        const int q = warp & 3, hh = warp >> 2;                 // TMEM lane quadrant, column half
        const uint32_t r = (uint32_t)(q * 32 + lane);           // tile row = TMEM lane
        const uint32_t tmem_row = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(16 * hh);
        const uint32_t key = r & 7u;
        const float* bias_s = reinterpret_cast<const float*>(w_s + (size_t)K * 32 * 128);
        const float* hdr_s = bias_s + 32;
        const bool leaky_max = p.act == MHO_ACT_LEAKY && p.slope >= 0.f && p.slope <= 1.f;
        uint32_t ph_mma = 0;
        float b1[16], b2[16];

        // ---- input rows of tile j -> part tile j & 1 (row-scaled), the tile's maxima via shared-memory atomics.  No arrive.
        float mx_keep = 0.f;   // tile maximum carried from the first half of a split to the second
        auto x_split = [&](int j, int part) {   // part 0 / 1: the two halves of the rows; part 2: both
            const int buf = j & 1;
            PROBE_C(3);
            if (part != 1) mbar_wait(bar_full + 8u * buf, (uint32_t)((j >> 1) & 1));
            PROBE_C(4);
            const int node0 = tinfo_s[buf * 4 + 0], rows = tinfo_s[buf * 4 + 1], nz0 = tinfo_s[buf * 4 + 2];
            const uint32_t parts_a = smem_a + (uint32_t)buf * HF_TILE_BYTES;
            const uint32_t xb_a = xs_a + (uint32_t)buf * HF_TILE_BYTES;
            const uint32_t opb = op_a + (uint32_t)(buf * p.stage_bytes);
            const uint32_t gb = gb_a + (uint32_t)(buf * 132) * 4u;
            float mx = part == 1 ? mx_keep : 0.f;
#pragma unroll
            for (int pp = 0; pp < 2; ++pp) {
                if (part != 2 && part != pp) continue;
                const int cp = tid + 256 * pp, row = cp >> 2, q4 = cp & 3;
                float x[8];
                float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
                if (row < rows) { a = lds_f128(xb_a + (uint32_t)row * 128u + (uint32_t)q4 * 32u); b = lds_f128(xb_a + (uint32_t)row * 128u + (uint32_t)q4 * 32u + 16u); }
                x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
                float rm = fmaxf(fmaxf(fmaxf(fabsf(x[0]), fabsf(x[1])), fmaxf(fabsf(x[2]), fabsf(x[3]))), fmaxf(fmaxf(fabsf(x[4]), fabsf(x[5])), fmaxf(fabsf(x[6]), fabsf(x[7]))));
                rm = fmaxf(rm, __shfl_xor_sync(0xffffffffu, rm, 1));
                rm = fmaxf(rm, __shfl_xor_sync(0xffffffffu, rm, 2));   // the row's maximum (four lanes share a row)
                mx = fmaxf(mx, rm);
                int ex = expo_above(rm);                               // row max < 2^ex
                ex = max(-100, min(110, ex));
                const float s_row = pow2f(15 - ex);
                if (q4 == 0) {
                    rowscale_s[buf * 128 + row] = pow2f(ex - 15);
                    
                }
                if (groups && q4 == 0 && row < rows)   // (a warp-level pre-reduction of these atomics was measured: no gain)
                    atomicMax(gmax_s + (j % 3) * 128 + group_of(gb, node0 + row, node0 + rows), __float_as_uint(rm));
                const uint64_t S2 = pk2(s_row, s_row);
                uint32_t h[4], l[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    float y0, y1;
                    upk2(mul2(pk2(x[2 * e], x[2 * e + 1]), S2), y0, y1);
                    split2(y0, y1, h[e], l[e]);
                }
                const uint32_t ra = parts_a + (uint32_t)row * 128u, rk = (uint32_t)row & 7u;
                sts_u128(ra + (((uint32_t)q4 ^ rk) << 4), h[0], h[1], h[2], h[3]);
                sts_u128(ra + (((4u + (uint32_t)q4) ^ rk) << 4), l[0], l[1], l[2], l[3]);
            }
            if (part == 0) { mx_keep = mx; fence_proxy_async(); return; }
            // operator: max degree of the tile (and, from a CSR slice, the bit rows)
            unsigned int deg = 0u;
            if (p.use_bits) {
                if (tid < rows) { const uint4 m4 = lds_u128(opb + (uint32_t)tid * 16u); deg = __popc(m4.x) + __popc(m4.y) + __popc(m4.z) + __popc(m4.w); }
            } else {
                const int row = tid >> 1, sub = tid & 1;
                uint32_t m0 = 0u, m1 = 0u, m2 = 0u, m3 = 0u;
                if (row < rows) {
                    const int e0 = (int)lds_u32(opb + (uint32_t)row * 4u) - nz0, e1 = (int)lds_u32(opb + (uint32_t)row * 4u + 4u) - nz0;
                    deg = (unsigned int)(e1 - e0);
                    for (int e = e0 + sub; e < e1; e += 2) {
                        const uint32_t c = lds_u32(opb + 528u + (uint32_t)e * 4u) - (uint32_t)node0;
                        const uint32_t bit = 1u << (c & 31u), w = c >> 5;
                        m0 |= (w == 0u) ? bit : 0u;
                        m1 |= (w == 1u) ? bit : 0u;
                        m2 |= (w == 2u) ? bit : 0u;
                        m3 |= (w == 3u) ? bit : 0u;
                    }
                }
                m0 |= __shfl_xor_sync(0xffffffffu, m0, 1);
                m1 |= __shfl_xor_sync(0xffffffffu, m1, 1);
                m2 |= __shfl_xor_sync(0xffffffffu, m2, 1);
                m3 |= __shfl_xor_sync(0xffffffffu, m3, 1);
                asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(mask_a + (uint32_t)buf * 2048u + (uint32_t)row * 16u + (uint32_t)sub * 8u), "r"(sub ? m2 : m0), "r"(sub ? m3 : m1) : "memory");
            }
            {
                const unsigned int wm = __reduce_max_sync(0xffffffffu, __float_as_uint(mx));
                const unsigned int wd = __reduce_max_sync(0xffffffffu, deg);
                unsigned int* red = red_s + (j % 3) * 2;
                if (lane == 0) { atomicMax(red, wm); atomicMax(red + 1, wd); }
                if (groups && deg > 0u) atomicMax(gdeg_s + (j % 3) * 128 + group_of(gb, node0 + (p.use_bits ? tid : (tid >> 1)), node0 + rows), deg);
            }
            fence_proxy_async();   // the part tile is read by the tensor core
            PROBE_C(7);
        };

        // ---- the tile's adjacency -> tensor memory (fp16 0 / 1 pairs)
        auto adjacency = [&](int j) {
            const int buf = j & 1;
            const int rows = tinfo_s[buf * 4 + 1];
            uint2 m2v = make_uint2(0u, 0u);
            if ((int)r < rows) {
                const uint32_t src = (p.use_bits ? op_a + (uint32_t)(buf * p.stage_bytes) : mask_a + (uint32_t)buf * 2048u) + r * 16u + (uint32_t)hh * 8u;
                asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(m2v.x), "=r"(m2v.y) : "r"(src));
            }
#pragma unroll
            for (int w2 = 0; w2 < 2; ++w2) {
                const uint32_t m = w2 ? m2v.y : m2v.x;
                uint32_t aw[16];
#pragma unroll
                for (int b4 = 0; b4 < 8; ++b4) {
                    uint2 v;
                    const uint32_t idx = b4 == 0 ? ((m << 3) & 0x78u) : ((m >> (4 * b4 - 3)) & 0x78u);
                    asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(lut_a + idx));
                    aw[2 * b4] = v.x; aw[2 * b4 + 1] = v.y;
                }
                tmem_st16(tmem_base + ((uint32_t)(q * 32) << 16) + ADJ_COL + (uint32_t)(32 * hh + 16 * w2), aw);
            }
        };

        // ---- all warps have written their parts -> thread 0 issues the UMMA group.
        // `what`: -1 = X W group of the tile whose parts are in part tile `buf`, k >= 0 = Clenshaw step k.
        auto arrive_issue = [&](int buf, int what, int rows_t) {
            tc_fence_before();
            const uint32_t parts_a = smem_a + (uint32_t)buf * HF_TILE_BYTES;
            if (what < 0) {
                // X W group: the A operand is all 128 rows -> hardware barrier over the 8 warps, then a fixed thread issues (the
                // barrier unit answers within a few tens of cycles; an mbarrier arrive that returns its state, or waking a
                // dedicated issuer warp, costs 150-200)
                bar_compute();
                if (tid == 0) {
                    mbar_wait(bar_w, 0u);   // (returns at once from the second tile on)
                    tc_fence_after();
                    // P' = X' [W'_0 | ... | W'_K-1]:  x w ~ xh wh - xh wl' - xl' wh, two 16-wide K steps each
                    PROBE_M(11);
#pragma unroll
                    for (int g = 0; g < (K + 4) / 5; ++g) {
                        const int nb = (K - 5 * g) < 5 ? (K - 5 * g) : 5;   // column blocks of this group
                        const uint32_t d = tmem_base + (uint32_t)(160 * g);
                        const uint32_t wg = w_a + (uint32_t)(160 * g) * 128u;
                        const uint32_t id_pos = idesc_f16((uint32_t)(32 * nb), 0u, 0u), id_neg = idesc_f16((uint32_t)(32 * nb), 0u, 1u);
#pragma unroll
                        for (int ks = 0; ks < 2; ++ks) umma_f16_ss(d, desc_sw128(parts_a + 64u + 32u * ks), desc_sw128(wg + 32u * ks), id_neg, ks > 0 ? 1u : 0u);
#pragma unroll
                        for (int ks = 0; ks < 2; ++ks) umma_f16_ss(d, desc_sw128(parts_a + 32u * ks), desc_sw128(wg + 64u + 32u * ks), id_neg, 1u);
#pragma unroll
                        for (int ks = 0; ks < 2; ++ks) umma_f16_ss(d, desc_sw128(parts_a + 32u * ks), desc_sw128(wg + 32u * ks), id_pos, 1u);
                    }
                    umma_commit(bar_mma);
                    PROBE_M(12);
                }
            } else {
                // Clenshaw step: D = A parts(B_k+1) into column blocks k+1 (A h) and k+2 (A l').  (Measured and rejected: one issuer
                // per lane quadrant behind 64-thread barriers with an ordering flag - four commits and the flag polls cost more
                // than the parallel issue wins.)
                bar_compute();
                if (tid == 0) {
                    tc_fence_after();
                    PROBE_M(20 + what);
                    const uint32_t id_adj = idesc_f16(64u, 1u, 0u);
                    const uint32_t d = tmem_base + (uint32_t)(32 * (what + 1));
                    const int nks = (rows_t + 15) >> 4;   // 16-node slices beyond the tile's rows are all zero
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks)
                        if (ks == 0 || ks < nks) umma_f16_ts(d, tmem_base + ADJ_COL + (uint32_t)(ks * 8), desc_sw128(parts_a + (uint32_t)ks * 2048u), id_adj, ks > 0 ? 1u : 0u);
                    umma_commit(bar_mma);
                    PROBE_M(30 + what);
                }
            }
        };

        // split B_k (b1) with tau_k = 2^(15 - (e - 127)) into part tile `buf`, then arrive for Clenshaw step k - 1
        auto split_arrive = [&](int buf, int e1, int step, int rows_t) {
            const uint64_t T2 = pk2(__uint_as_float((uint32_t)(269 - e1) << 23), __uint_as_float((uint32_t)(269 - e1) << 23));
            const uint32_t prow_a = smem_a + (uint32_t)buf * HF_TILE_BYTES + r * 128u;
            uint32_t h[8], l[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                float y0, y1;
                upk2(mul2(pk2(b1[2 * e], b1[2 * e + 1]), T2), y0, y1);
                split2(y0, y1, h[e], l[e]);
            }
            PROBE_C(60);
            sts_u128(prow_a + (((uint32_t)(2 * hh) ^ key) << 4), h[0], h[1], h[2], h[3]);
            sts_u128(prow_a + (((uint32_t)(2 * hh + 1) ^ key) << 4), h[4], h[5], h[6], h[7]);
            sts_u128(prow_a + (((uint32_t)(4 + 2 * hh) ^ key) << 4), l[0], l[1], l[2], l[3]);
            sts_u128(prow_a + (((uint32_t)(5 + 2 * hh) ^ key) << 4), l[4], l[5], l[6], l[7]);
            PROBE_C(61);
            fence_proxy_async();
            PROBE_C(62);
            arrive_issue(buf, step, rows_t);
        };

        if (n_my > 0) {
            x_split(0, 2);
            arrive_issue(0, -1, 0);   // (the first tile's bit rows, built by all threads, are read behind the barrier at the top of the tile loop)
        }
        for (int j = 0; j < n_my; ++j) {
            const int buf = j & 1;
            const int node0 = tinfo_s[buf * 4 + 0], rows = tinfo_s[buf * 4 + 1];
            // the tile's maxima are complete: every warp split this tile's rows before it arrived for a later group of the
            // previous tile, whose completion this thread has waited for (first tile: the barrier below)
            if (j == 0) { bar_compute(); mbar_wait(bar_w, 0u); }   // (+ the weight image: header, bias)
            unsigned int* red = red_s + (j % 3) * 2;
            unsigned int* trk = track_s + (j % 3) * 16;
            float xmax = __uint_as_float(red[0]);
            float dmax2 = 2.f * (float)red[1];
            const float xmax_tile = xmax, dmax2_tile = dmax2;
            (void)xmax_tile; (void)dmax2_tile;
            if (groups) {   // the graph of this thread's row: block-diagonal operator => its own scale per step
                const int g = group_of(gb_a + (uint32_t)(buf * 132) * 4u, node0 + min((int)r, rows - 1), node0 + rows);   // (padding rows: the last graph)
                xmax = __uint_as_float(gmax_s[(j % 3) * 128 + g]);
                dmax2 = 2.f * (float)gdeg_s[(j % 3) * 128 + g];
            }
            if (tid == 0) { unsigned int* o = red_s + ((j + 2) % 3) * 2; o[0] = 0u; o[1] = 0u; }   // last read a tile ago, next written a tile ahead
            if (TRACK && tid < 16) track_s[((j + 2) % 3) * 16 + tid] = 0u;
            if (groups) {
                if (tid < 128) { gmax_s[((j + 2) % 3) * 128 + tid] = 0u; gdeg_s[((j + 2) % 3) * 128 + tid] = 0u; }
            }
            const float inv_si = rowscale_s[buf * 128 + r];
            int e_tau[K];   // clamped exponent fields of the bounds of |B_k| (units of the weight scale), k = 1 .. K-1
            {
                float bet1 = 0.f, bet2 = 0.f;
#pragma unroll
                for (int k = K - 1; k >= 1; --k) {
                    const float bet = xmax * hdr_s[1 + k] + dmax2 * bet1 + bet2;
                    const int e = (int)((__float_as_uint(bet) >> 23) & 0xffu) + 1;   // bet < 2^(e - 127)
                    e_tau[k] = max(30, min(240, e));
                    bet2 = bet1;
                    bet1 = bet;
                }
                e_tau[0] = 127;
            }
            adjacency(j);
            if (warp == 0 && j + 1 < n_my) {
                if (j + 1 >= 2) {   // tile j - 1 (same staging buffer) has stored its output rows
                    if (lane == 0) mbar_wait(bar_empty + 8u * ((j + 1) & 1), (uint32_t)((((j + 1) >> 1) + 1) & 1));
                    __syncwarp();
                }
                issue_load(j + 1);
            }

            // ---- X W done -> scales, B_K-1 = P_K-1 / row scale
            PROBE_C(8);
            mbar_wait(bar_mma, ph_mma);
            ph_mma ^= 1u;
            tc_fence_after();
            PROBE_C(9);
            const uint64_t I2 = pk2(inv_si, inv_si);
            {
                uint32_t v[16];
                tmem_ld16(tmem_row + (uint32_t)(32 * (K - 1)), v);
                tmem_wait_ld_();
                float m = 0.f;
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    upk2(mul2(pk2(__uint_as_float(v[2 * e]), __uint_as_float(v[2 * e + 1])), I2), b1[2 * e], b1[2 * e + 1]);
                    b2[2 * e] = 0.f; b2[2 * e + 1] = 0.f;
                    if (TRACK) m = fmaxf(m, fmaxf(fabsf(b1[2 * e]), fabsf(b1[2 * e + 1])));
                }
                if (TRACK) {
                    const unsigned int wm = __reduce_max_sync(0xffffffffu, __float_as_uint(m));
                    if (lane == 0) atomicMax(trk + (K - 1), wm);
                }
            }
            tmem_wait_st_();   // the adjacency stores have completed (first read by the first Clenshaw step's UMMAs)
            split_arrive(buf, e_tau[K - 1], K - 2, rows);
            PROBE_C(20 + K - 2);

            // ---- Clenshaw steps
#pragma unroll
            for (int k = K - 2; k >= 0; --k) {
                // the next tile's input rows are split into the other part tile inside one step's wait window
                if (K >= 4) {   // two wait windows, half of the rows each
                    if (k == K - 3 && j + 1 < n_my) x_split(j + 1, 0);
                    if (k == K - 4 && j + 1 < n_my) x_split(j + 1, 1);
                } else if (k == (K == 3 ? 1 : 0) && j + 1 < n_my) {
                    x_split(j + 1, 2);
                }
                const int e1 = e_tau[k + 1];   // the UMMAs multiplied parts(B_k+1) scaled with tau_k+1
                mbar_wait(bar_mma, ph_mma);
                ph_mma ^= 1u;
                tc_fence_after();
                PROBE_C(30 + k);
                const float cfac = __uint_as_float((uint32_t)(e1 - 15 + (k > 0 ? 1 : 0)) << 23);   // (k > 0 ? 2 : 1) / tau_k+1
                const uint64_t C2 = pk2(cfac, cfac);
                uint32_t vp[16], vh[16], vl[16];
                tmem_ld16(tmem_row + (uint32_t)(32 * k), vp);
                tmem_ld16(tmem_row + (uint32_t)(32 * (k + 1)), vh);
                tmem_ld16(tmem_row + (uint32_t)(32 * (k + 2)), vl);
                tmem_wait_ld_();
                PROBE_C(50 + k);
                float m = 0.f;
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const uint64_t dv = sub2(pk2(__uint_as_float(vh[2 * e]), __uint_as_float(vh[2 * e + 1])), pk2(__uint_as_float(vl[2 * e]), __uint_as_float(vl[2 * e + 1])));
                    const uint64_t bk = fma2(pk2(__uint_as_float(vp[2 * e]), __uint_as_float(vp[2 * e + 1])), I2, fma2(dv, C2, pk2(-b2[2 * e], -b2[2 * e + 1])));
                    b2[2 * e] = b1[2 * e]; b2[2 * e + 1] = b1[2 * e + 1];
                    upk2(bk, b1[2 * e], b1[2 * e + 1]);
                    if (TRACK) m = fmaxf(m, fmaxf(fabsf(b1[2 * e]), fabsf(b1[2 * e + 1])));
                }
                if (k > 0) {
                    int e0 = e_tau[k];
                    if (TRACK) {
                        const unsigned int wm = __reduce_max_sync(0xffffffffu, __float_as_uint(m));
                        if (lane == 0) atomicMax(trk + k, wm);
                        // the maxima of |B_k+1| and |B_k+2| are complete (their atomics preceded the arrive / UMMA / wait round of
                        // this step): tighter bound of |B_k| than the a-priori one
                        const float m1 = __uint_as_float(trk[k + 1]);
                        const float m2 = (k + 2 <= K - 1) ? __uint_as_float(trk[k + 2]) : 0.f;
                        const float bet = xmax_tile * hdr_s[1 + k] + dmax2_tile * m1 + m2;   // tile-wide: bounds every graph of the tile
                        e0 = min(e0, max(30, min(240, (int)((__float_as_uint(bet) >> 23) & 0xffu) + 1)));
                        e_tau[k] = e0;
                    }
                    split_arrive(buf, e0, k - 1, rows);
                    PROBE_C(20 + k - 1);
                }
            }
            // ---- the next tile's X W group may start: its part tile was written inside this tile, P is consumed
            if (j + 1 < n_my) arrive_issue(buf ^ 1, -1, 0);

            // ---- epilogue: unscale, bias, activation; output rows through the staging tile as whole 128 B lines
            PROBE_C(40);
            {
                const uint32_t xb_a = xs_a + (uint32_t)buf * HF_TILE_BYTES;
                const float inv_sw = hdr_s[0];
                const uint64_t W2 = pk2(inv_sw, inv_sw);
                float y[16];
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const float4 bv = *reinterpret_cast<const float4*>(bias_s + 16 * hh + 4 * c);
                    upk2(fma2(pk2(b1[4 * c], b1[4 * c + 1]), W2, pk2(bv.x, bv.y)), y[4 * c], y[4 * c + 1]);
                    upk2(fma2(pk2(b1[4 * c + 2], b1[4 * c + 3]), W2, pk2(bv.z, bv.w)), y[4 * c + 2], y[4 * c + 3]);
                }
                if (p.act == MHO_ACT_RELU) {
#pragma unroll
                    for (int e = 0; e < 16; ++e) y[e] = fmaxf(y[e], 0.f);
                } else if (leaky_max) {
                    const uint64_t SL2 = pk2(p.slope, p.slope);
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        float s0, s1;
                        upk2(mul2(pk2(y[2 * e], y[2 * e + 1]), SL2), s0, s1);
                        y[2 * e] = fmaxf(y[2 * e], s0); y[2 * e + 1] = fmaxf(y[2 * e + 1], s1);
                    }
                } else if (p.act == MHO_ACT_LEAKY) {
                    const float sl = p.slope;
#pragma unroll
                    for (int e = 0; e < 16; ++e) y[e] = y[e] > 0.f ? y[e] : sl * y[e];
                }
                const uint32_t ya = xb_a + r * 128u;
#pragma unroll
                for (int c = 0; c < 4; ++c) sts_f128(ya + (((uint32_t)(4 * hh + c) ^ key) << 4), make_float4(y[4 * c], y[4 * c + 1], y[4 * c + 2], y[4 * c + 3]));
                bar_quadrant(q);   // the two warps of this lane quadrant hold all 32 columns of its rows
                float* dst = p.Y + (size_t)node0 * 32;
#pragma unroll
                for (int pp = 0; pp < 4; ++pp) {
                    const uint32_t row = (uint32_t)(32 * q + 16 * hh + 4 * pp) + ((uint32_t)lane >> 3), ch = (uint32_t)lane & 7u;
                    if ((int)row < rows) *reinterpret_cast<float4*>(dst + (size_t)row * 32 + ch * 4) = lds_f128(xb_a + row * 128u + ((ch ^ (row & 7u)) << 4));
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_empty + 8u * buf);   // the staging buffer may be refilled
            }
            PROBE_C(41);
        }
    }
#ifdef MHO_PROBE
    __syncthreads();
    if (probe_on && tid == 0) {
        unsigned long long gt1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt1));
        printf("cta %d tiles %d globaltimer start %llu end +%llu ns\n", (int)blockIdx.x, n_my, gt0, gt1 - gt0);
        const long long base = probe_s[0] >> 8;
        for (int i = 0; i < 192; ++i) {
            if (probe_s[i] == 0) continue;
            printf("cta %d %s id %2d  t %7lld\n", (int)blockIdx.x, i < 128 ? "C" : "M", (int)(probe_s[i] & 255), (probe_s[i] >> 8) - base);
        }
    }
#endif

    // ---- teardown
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, TCOLS);
}

// ---- warp-specialised variant (K <= 5, bit rows, per-graph scales) ---------------------------------------------------------
// Same arithmetic as cheb_f16_kernel - the two kernels give bit-identical results - with the work that does not belong to the
// dependent chain of a tile moved off the eight compute warps (12 warps per CTA, two CTAs per SM, register budgets re-balanced
// with setmaxnreg):
//   * warps 0-7, COMPUTE (thread = one row x 16 columns): adjacency expansion under the X W group, then per round trip: wait,
//     tensor-memory load, recurrence in packed fp32, split, arrive; the rows of the NEXT tile are split inside the wait
//     windows of two Clenshaw steps (the windows are ~1 k cycles: the UMMA group under load); B_0 goes to the staging tile raw.
//   * warps 8-10, SERVICE (96 threads): bulk loads two tiles ahead; un-scale, bias, activation and the coalesced output store
//     of the CURRENT tile.
//   * warp 11, ISSUE: one thread issues every tcgen05.mma group (an issuing thread stalls until the tensor pipe has accepted the
//     group: 50-130 cycles per UMMA with two CTAs sharing the pipe).
// Hand-offs: named barriers with fixed arrive / sync counts where the two sides alternate strictly (parts ready: 256 + 32, output
// rows staged: 256 + 96).  For K >= 4 (template flag S_SPLIT) the service warps also split the next tile's rows - measured 5 %
// faster on the benchmark layer - with monotonic shared-memory counters for "rows split" / "part tile free" (one side may run
// ahead there); 96 threads need ~7 k cycles for a tile's rows, more than a K <= 3 tile lasts, so those keep the split in the
// compute warps' wait windows.
__device__ __forceinline__ void ws_parts_arrive() { asm volatile("bar.arrive 1, 288;" ::: "memory"); }
__device__ __forceinline__ void ws_parts_wait() { asm volatile("bar.sync 1, 288;" ::: "memory"); }
__device__ __forceinline__ void ws_out_arrive() { asm volatile("bar.arrive 2, 352;" ::: "memory"); }
__device__ __forceinline__ void ws_out_wait() { asm volatile("bar.sync 2, 352;" ::: "memory"); }
__device__ __forceinline__ void ws_service_sync() { asm volatile("bar.sync 3, 96;" ::: "memory"); }
__device__ __forceinline__ void ws_poll(volatile int* c, int target) { while (*c < target) { } }
__device__ __forceinline__ void tmem_ld8_(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
}

template <int K, bool S_SPLIT>
__global__ void __launch_bounds__(384, 2) cheb_f16ws_kernel(const __grid_constant__ HfParams p) {
    extern __shared__ __align__(1024) unsigned char smem[];
    constexpr int W_BYTES = hf_w_bytes(K);
    constexpr uint32_t TCOLS = 256u, ADJ_COL = TCOLS - 64u;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#ifdef MHO_PROBE
    __shared__ long long wprobe_s[256];
    int wpn = 0;
    if (tid < 256) wprobe_s[tid] = 0;
    __syncthreads();
#define WPROBE(id) do { if (blockIdx.x == 0 && (tid == 0 || tid == 256 || tid == 352) && wpn < 80) { wprobe_s[(tid == 0 ? 0 : tid == 256 ? 88 : 176) + wpn] = (clock64() << 8) | (long long)(id); ++wpn; } } while (0)
#else
#define WPROBE(id) do { } while (0)
#endif
    // shared memory: as in cheb_f16_kernel (two part tiles | two staging tiles | weights | control block | LUT | masks (unused) |
    // operator staging | graph starts and per-graph maxima)
    unsigned char* w_s = smem + 4 * HF_TILE_BYTES;
    unsigned char* ctl_s = w_s + W_BYTES;
    unsigned char* lut_s = ctl_s + 1536;
    unsigned char* op_s = lut_s + 128 + 4096;
    unsigned char* grp_s = op_s + 2 * p.stage_bytes;
    const uint32_t smem_a = smem_u32(smem), xs_a = smem_a + 2u * HF_TILE_BYTES, w_a = smem_u32(w_s), ctl_a = smem_u32(ctl_s), lut_a = smem_u32(lut_s),
                   op_a = smem_u32(op_s);
    // control block: full[2] +0, weights +32, mma +40, tmem slot +48, tile info +64
    // ([buf][4]), reductions +96 ([3][2]), row scales +512 ([2][128] floats)
    const uint32_t bar_full = ctl_a, bar_w = ctl_a + 32, bar_mma = ctl_a + 40, tslot = ctl_a + 48;
    volatile int* xs_count = reinterpret_cast<volatile int*>(ctl_s + 56);   // S_SPLIT: + 3 per tile whose rows are split (service warps)
    volatile int* pf_count = reinterpret_cast<volatile int*>(ctl_s + 60);   // S_SPLIT: + 8 per tile whose UMMAs are all complete (compute warps)
    volatile int* tinfo_s = reinterpret_cast<volatile int*>(ctl_s + 64);
    unsigned int* red_s = reinterpret_cast<unsigned int*>(ctl_s + 96);
    float* rowscale_s = reinterpret_cast<float*>(ctl_s + 512);
    const uint32_t gb_a = smem_u32(grp_s);
    unsigned int* gmax_s = reinterpret_cast<unsigned int*>(grp_s + 1056 + 64);
    unsigned int* gdeg_s = gmax_s + 3 * 128;

    const int G = (int)gridDim.x;
    const int n_my = (int)blockIdx.x < p.b.n_tiles ? (p.b.n_tiles - (int)blockIdx.x + G - 1) / G : 0;

    if (tid == 0) {
        mbar_init(bar_full, 33u);        // expect_tx arrive + one cp.async arrive per lane of the loading warp
        mbar_init(bar_full + 8, 33u);
        mbar_init(bar_mma, 1);
        mbar_init(bar_w, 1);
        *xs_count = 3;   // (tile 0 is split by the compute warps)
        *pf_count = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (tid < 16) {
        const uint32_t x = ((tid & 1) ? 0x3C00u : 0u) | ((tid & 2) ? 0x3C000000u : 0u), y = ((tid & 4) ? 0x3C00u : 0u) | ((tid & 8) ? 0x3C000000u : 0u);
        asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(lut_a + (uint32_t)tid * 8u), "r"(x), "r"(y) : "memory");
    }
    if (tid >= 32 && tid < 38) red_s[tid - 32] = 0u;
    for (int i = tid; i < 6 * 128; i += 384) gmax_s[i] = 0u;
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (warp == 0) tmem_alloc(tslot, TCOLS);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(ctl_s + 48);

    if (warp < 8) {
        // ======================================================= compute warps =======================================================
        asm volatile("setmaxnreg.inc.sync.aligned.u32 88;");
        const int q = warp & 3, hh = warp >> 2;
        const uint32_t r = (uint32_t)(q * 32 + lane);
        const uint32_t tmem_row = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(16 * hh);
        const uint32_t key = r & 7u;
        const float* bias_s = reinterpret_cast<const float*>(w_s + (size_t)K * 32 * 128);
        const float* hdr_s = bias_s + 32;
        uint32_t ph_mma = 0;
        float b1[16], b2[16];
        auto split_arrive = [&](int buf, int e1) {
            const uint64_t T2 = pk2(__uint_as_float((uint32_t)(269 - e1) << 23), __uint_as_float((uint32_t)(269 - e1) << 23));
            const uint32_t prow_a = smem_a + (uint32_t)buf * HF_TILE_BYTES + r * 128u;
            uint32_t h[8], l[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                float y0, y1;
                upk2(mul2(pk2(b1[2 * e], b1[2 * e + 1]), T2), y0, y1);
                split2(y0, y1, h[e], l[e]);
            }
            sts_u128(prow_a + (((uint32_t)(2 * hh) ^ key) << 4), h[0], h[1], h[2], h[3]);
            sts_u128(prow_a + (((uint32_t)(2 * hh + 1) ^ key) << 4), h[4], h[5], h[6], h[7]);
            sts_u128(prow_a + (((uint32_t)(4 + 2 * hh) ^ key) << 4), l[0], l[1], l[2], l[3]);
            sts_u128(prow_a + (((uint32_t)(5 + 2 * hh) ^ key) << 4), l[4], l[5], l[6], l[7]);
            fence_proxy_async();
            tc_fence_before();
            ws_parts_arrive();
        };
        // rows of tile j -> part tile j & 1 (row-scaled), per-graph maxima of |x| and of the degree.  part 0 / 1: the two halves of the
        // rows (one wait window of a Clenshaw step each), part 1 also the degrees; part 2: everything
        auto x_split = [&](int j, int part) {
            const int buf = j & 1;
            if (part != 1) mbar_wait(bar_full + 8u * buf, (uint32_t)((j >> 1) & 1));
            const int node0 = tinfo_s[buf * 4 + 0], rows = tinfo_s[buf * 4 + 1];
            const uint32_t parts_a = smem_a + (uint32_t)buf * HF_TILE_BYTES;
            const uint32_t xb_a = xs_a + (uint32_t)buf * HF_TILE_BYTES;
            const uint32_t gb = gb_a + (uint32_t)(buf * 132) * 4u;
#pragma unroll
            for (int pp = 0; pp < 2; ++pp) {
                if (part != 2 && part != pp) continue;
                const int cp = tid + 256 * pp, row = cp >> 2, q4 = cp & 3;
                float x[8];
                float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
                if (row < rows) { a = lds_f128(xb_a + (uint32_t)row * 128u + (uint32_t)q4 * 32u); b = lds_f128(xb_a + (uint32_t)row * 128u + (uint32_t)q4 * 32u + 16u); }
                x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
                float rm = fmaxf(fmaxf(fmaxf(fabsf(x[0]), fabsf(x[1])), fmaxf(fabsf(x[2]), fabsf(x[3]))), fmaxf(fmaxf(fabsf(x[4]), fabsf(x[5])), fmaxf(fabsf(x[6]), fabsf(x[7]))));
                rm = fmaxf(rm, __shfl_xor_sync(0xffffffffu, rm, 1));
                rm = fmaxf(rm, __shfl_xor_sync(0xffffffffu, rm, 2));
                int ex = expo_above(rm);
                ex = max(-100, min(110, ex));
                const float s_row = pow2f(15 - ex);
                if (q4 == 0) rowscale_s[buf * 128 + row] = pow2f(ex - 15);
                if (q4 == 0 && row < rows) atomicMax(gmax_s + (j % 3) * 128 + group_of(gb, node0 + row, node0 + rows), __float_as_uint(rm));
                const uint64_t S2 = pk2(s_row, s_row);
                uint32_t h[4], l[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    float y0, y1;
                    upk2(mul2(pk2(x[2 * e], x[2 * e + 1]), S2), y0, y1);
                    split2(y0, y1, h[e], l[e]);
                }
                const uint32_t ra = parts_a + (uint32_t)row * 128u, rk = (uint32_t)row & 7u;
                sts_u128(ra + (((uint32_t)q4 ^ rk) << 4), h[0], h[1], h[2], h[3]);
                sts_u128(ra + (((4u + (uint32_t)q4) ^ rk) << 4), l[0], l[1], l[2], l[3]);
            }
            if (part != 0 && tid < rows) {
                const uint4 m4 = lds_u128(op_a + (uint32_t)(buf * p.stage_bytes) + (uint32_t)tid * 16u);
                const unsigned int deg = __popc(m4.x) + __popc(m4.y) + __popc(m4.z) + __popc(m4.w);
                if (deg > 0u) atomicMax(gdeg_s + (j % 3) * 128 + group_of(gb, node0 + tid, node0 + rows), deg);
            }
            fence_proxy_async();   // the part tile is read by the tensor core
        };
        if (n_my > 0) {
            x_split(0, 2);
            tc_fence_before();
            ws_parts_arrive();     // -> the issue warp: X W group of tile 0
            mbar_wait(bar_w, 0u);
        }
        for (int j = 0; j < n_my; ++j) {
            const int buf = j & 1;
            const int rows = tinfo_s[buf * 4 + 1];
            const int node0 = tinfo_s[buf * 4 + 0];
            // per-thread scales of tile j: the graph of this thread's row (block-diagonal operator => its own scale per step), the
            // row scale of X, the exponents of the Clenshaw bounds.  Needs every thread's share of the row split of tile j:
            // S_SPLIT: complete since the end of tile j - 1 (counter); otherwise complete once the X W group has been issued
            float inv_si = 0.f;
            int e_tau[K];
            auto tile_scales = [&]() {
                const int g = group_of(gb_a + (uint32_t)(buf * 132) * 4u, node0 + min((int)r, rows - 1), node0 + rows);
                const float xmax = __uint_as_float(gmax_s[(j % 3) * 128 + g]);
                const float dmax2 = 2.f * (float)gdeg_s[(j % 3) * 128 + g];
                inv_si = rowscale_s[buf * 128 + r];
                // the maxima of tile j + 2 go into the slot tile j - 1 used; they are collected after every thread has arrived for
                // the X W group of tile j + 1 (S_SPLIT: after every warp has counted this tile complete), i.e. after these clears
                if (tid < 128) { gmax_s[((j + 2) % 3) * 128 + tid] = 0u; gdeg_s[((j + 2) % 3) * 128 + tid] = 0u; }
                float bet1 = 0.f, bet2 = 0.f;
#pragma unroll
                for (int kk = K - 1; kk >= 1; --kk) {
                    const float bet = xmax * hdr_s[1 + kk] + dmax2 * bet1 + bet2;
                    const int e = (int)((__float_as_uint(bet) >> 23) & 0xffu) + 1;
                    e_tau[kk] = max(30, min(240, e));
                    bet2 = bet1;
                    bet1 = bet;
                }
                e_tau[0] = 127;
            };
            if (S_SPLIT && j > 0) tile_scales();   // (tile 0 is split by the compute warps themselves: see below)
            // ---- the tile's adjacency -> tensor memory (fp16 0 / 1 pairs), under the X W group
            {
                uint2 m2v = make_uint2(0u, 0u);
                if ((int)r < rows) {
                    const uint32_t src = op_a + (uint32_t)(buf * p.stage_bytes) + r * 16u + (uint32_t)hh * 8u;
                    asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(m2v.x), "=r"(m2v.y) : "r"(src));
                }
#pragma unroll
                for (int w2 = 0; w2 < 2; ++w2) {
                    const uint32_t m = w2 ? m2v.y : m2v.x;
                    uint32_t aw[16];
#pragma unroll
                    for (int b4 = 0; b4 < 8; ++b4) {
                        uint2 v;
                        const uint32_t idx = b4 == 0 ? ((m << 3) & 0x78u) : ((m >> (4 * b4 - 3)) & 0x78u);
                        asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(lut_a + idx));
                        aw[2 * b4] = v.x; aw[2 * b4 + 1] = v.y;
                    }
                    tmem_st16(tmem_base + ((uint32_t)(q * 32) << 16) + ADJ_COL + (uint32_t)(32 * hh + 16 * w2), aw);
                }
            }
            // ---- X W done -> B_K-1 = P_K-1 / row scale
            WPROBE(1);
            mbar_wait(bar_mma, ph_mma);
            WPROBE(2);
            ph_mma ^= 1u;
            tc_fence_after();
            if (!S_SPLIT || j == 0) tile_scales();   // every thread's share of the split precedes the X W group's issue
            const uint64_t I2 = pk2(inv_si, inv_si);
            {
                uint32_t v[16];
                tmem_ld16(tmem_row + (uint32_t)(32 * (K - 1)), v);
                tmem_wait_ld_();
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    upk2(mul2(pk2(__uint_as_float(v[2 * e]), __uint_as_float(v[2 * e + 1])), I2), b1[2 * e], b1[2 * e + 1]);
                    b2[2 * e] = 0.f; b2[2 * e + 1] = 0.f;
                }
            }
            tmem_wait_st_();   // the adjacency stores have completed (first read by the first Clenshaw step's UMMAs)
            split_arrive(buf, e_tau[K - 1]);
            // ---- Clenshaw steps (two halves of 8 columns: 24 instead of 48 live accumulator registers)
#pragma unroll
            for (int k = K - 2; k >= 0; --k) {
                // the next tile's input rows are split into the other part tile inside the wait windows
                if (S_SPLIT) {
                } else if (K >= 4) {
                    if (k == K - 3 && j + 1 < n_my) x_split(j + 1, 0);
                    if (k == K - 4 && j + 1 < n_my) x_split(j + 1, 1);
                } else if (k == (K == 3 ? 1 : 0) && j + 1 < n_my) {
                    x_split(j + 1, 2);
                }
                const int e1 = e_tau[k + 1];
                WPROBE(10 + k);
                mbar_wait(bar_mma, ph_mma);
                ph_mma ^= 1u;
                tc_fence_after();
                WPROBE(20 + k);
                const float cfac = __uint_as_float((uint32_t)(e1 - 15 + (k > 0 ? 1 : 0)) << 23);   // (k > 0 ? 2 : 1) / tau_k+1
                const uint64_t C2 = pk2(cfac, cfac);
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    uint32_t vp[8], vh[8], vl[8];
                    tmem_ld8_(tmem_row + (uint32_t)(32 * k + 8 * half), vp);
                    tmem_ld8_(tmem_row + (uint32_t)(32 * (k + 1) + 8 * half), vh);
                    tmem_ld8_(tmem_row + (uint32_t)(32 * (k + 2) + 8 * half), vl);
                    tmem_wait_ld_();
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int c = 8 * half + 2 * e;
                        const uint64_t dv = sub2(pk2(__uint_as_float(vh[2 * e]), __uint_as_float(vh[2 * e + 1])), pk2(__uint_as_float(vl[2 * e]), __uint_as_float(vl[2 * e + 1])));
                        const uint64_t bk = fma2(pk2(__uint_as_float(vp[2 * e]), __uint_as_float(vp[2 * e + 1])), I2, fma2(dv, C2, pk2(-b2[c], -b2[c + 1])));
                        b2[c] = b1[c]; b2[c + 1] = b1[c + 1];
                        upk2(bk, b1[c], b1[c + 1]);
                    }
                }
                if (k > 0) split_arrive(buf, e_tau[k]);
            }
            // ---- every UMMA of this tile has completed and its accumulators are read: the next tile's X W group may be issued (its
            // rows were split a tile ago) and this tile's part tile may be refilled with the rows of tile j + 2
            WPROBE(30);
            tc_fence_before();
            if (S_SPLIT) {
                // the service warps split the next tile's rows: they must be done before its X W group is issued, and they may refill
                // this tile's part tile (rows of tile j + 2) once every warp has counted here
                if (j + 1 < n_my) { if (lane == 0) ws_poll(xs_count, 3 * (j + 2)); __syncwarp(); __threadfence_block(); }
                if (lane == 0) { __threadfence_block(); atomicAdd(const_cast<int*>(pf_count), 1); }
            }
            ws_parts_arrive();
            // ---- B_0 (still in units of the weight scale) -> staging tile; the service warps un-scale, add the bias, apply the
            // activation and store the rows
            {
                const uint32_t ya = xs_a + (uint32_t)buf * HF_TILE_BYTES + r * 128u;
#pragma unroll
                for (int c = 0; c < 4; ++c) sts_f128(ya + (((uint32_t)(4 * hh + c) ^ key) << 4), make_float4(b1[4 * c], b1[4 * c + 1], b1[4 * c + 2], b1[4 * c + 3]));
                ws_out_arrive();   // (st.shared + bar.arrive / bar.sync + ld.shared: the documented producer-consumer pattern)
                WPROBE(31);
            }
        }
    } else if (warp < 11) {
        // ======================================================= service warps =======================================================
        asm volatile("setmaxnreg.dec.sync.aligned.u32 64;");
        const int st = tid - 256;   // 0 .. 95
        int4 ti_pref = make_int4(0, 0, 0, 0);
        int g0_pref = 0, pref_j = -1;
        auto prefetch_desc = [&](int j) {
            if (j < n_my) {
                ti_pref = __ldg(reinterpret_cast<const int4*>(p.b.tile_info) + ((int)blockIdx.x + j * G));
                g0_pref = __ldg(p.b.tile_graph0 + ((int)blockIdx.x + j * G));
                pref_j = j;
            }
        };
        auto issue_load = [&](int j) {   // all of warp 8
            const int buf = j & 1;
            if (pref_j != j) prefetch_desc(j);
            const int4 ti = ti_pref;
            const int g0 = g0_pref;
            prefetch_desc(j + 1);
            const uint32_t fb = bar_full + 8u * buf;
            const uint32_t opb = op_a + (uint32_t)(buf * p.stage_bytes);
            if (lane == 0) {
                tinfo_s[buf * 4 + 0] = ti.x; tinfo_s[buf * 4 + 1] = ti.y; tinfo_s[buf * 4 + 2] = ti.z; tinfo_s[buf * 4 + 3] = ti.w;
                const uint32_t xb = (uint32_t)ti.y * 128u;
                mbar_expect_tx(fb, xb + (uint32_t)ti.y * 16u);
                bulk_g2s(xs_a + (uint32_t)buf * HF_TILE_BYTES, p.X + (size_t)ti.x * 32, xb, fb);
                bulk_g2s(opb, p.b.adj_bits + (size_t)ti.x * 4, (uint32_t)ti.y * 16u, fb);
            }
            for (int e = lane; e < 128; e += 32) {
                const int gi = min(g0 + 1 + e, p.b.n_graphs);
                cp_async4(gb_a + (uint32_t)(buf * 132 + e) * 4u, p.b.graph_off + gi);
            }
            cp_async_mbar_arrive(fb);
        };
        // rows of tile j -> part tile j & 1 (row-scaled), per-graph maxima of |x| and of the degree
        auto x_split_s = [&](int j) {
            const int buf = j & 1;
            WPROBE(70);
            mbar_wait(bar_full + 8u * buf, (uint32_t)((j >> 1) & 1));
            WPROBE(71);
            const int node0 = tinfo_s[buf * 4 + 0], rows = tinfo_s[buf * 4 + 1];
            const uint32_t parts_a = smem_a + (uint32_t)buf * HF_TILE_BYTES;
            const uint32_t xb_a = xs_a + (uint32_t)buf * HF_TILE_BYTES;
            const uint32_t opb = op_a + (uint32_t)(buf * p.stage_bytes);
            const uint32_t gb = gb_a + (uint32_t)(buf * 132) * 4u;
            for (int it = st; it < 512; it += 96) {   // (it >> 2 = row, 4 lanes per row; whole warps drop out together)
                const int row = it >> 2, q4 = it & 3;
                float x[8];
                float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
                if (row < rows) { a = lds_f128(xb_a + (uint32_t)row * 128u + (uint32_t)q4 * 32u); b = lds_f128(xb_a + (uint32_t)row * 128u + (uint32_t)q4 * 32u + 16u); }
                x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
                float rm = fmaxf(fmaxf(fmaxf(fabsf(x[0]), fabsf(x[1])), fmaxf(fabsf(x[2]), fabsf(x[3]))), fmaxf(fmaxf(fabsf(x[4]), fabsf(x[5])), fmaxf(fabsf(x[6]), fabsf(x[7]))));
                rm = fmaxf(rm, __shfl_xor_sync(0xffffffffu, rm, 1));
                rm = fmaxf(rm, __shfl_xor_sync(0xffffffffu, rm, 2));
                int ex = expo_above(rm);
                ex = max(-100, min(110, ex));
                const float s_row = pow2f(15 - ex);
                if (q4 == 0) rowscale_s[buf * 128 + row] = pow2f(ex - 15);
                if (q4 == 0 && row < rows) atomicMax(gmax_s + (j % 3) * 128 + group_of(gb, node0 + row, node0 + rows), __float_as_uint(rm));
                const uint64_t S2 = pk2(s_row, s_row);
                uint32_t h[4], l[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    float y0, y1;
                    upk2(mul2(pk2(x[2 * e], x[2 * e + 1]), S2), y0, y1);
                    split2(y0, y1, h[e], l[e]);
                }
                const uint32_t ra = parts_a + (uint32_t)row * 128u, rk = (uint32_t)row & 7u;
                sts_u128(ra + (((uint32_t)q4 ^ rk) << 4), h[0], h[1], h[2], h[3]);
                sts_u128(ra + (((4u + (uint32_t)q4) ^ rk) << 4), l[0], l[1], l[2], l[3]);
            }
            for (int row = st; row < rows; row += 96) {
                const uint4 m4 = lds_u128(opb + (uint32_t)row * 16u);
                const unsigned int deg = __popc(m4.x) + __popc(m4.y) + __popc(m4.z) + __popc(m4.w);
                if (deg > 0u) atomicMax(gdeg_s + (j % 3) * 128 + group_of(gb, node0 + row, node0 + rows), deg);
            }
            fence_proxy_async();   // the part tile is read by the tensor core
            __syncwarp();
            if (lane == 0) { __threadfence_block(); atomicAdd(const_cast<int*>(xs_count), 1); }
            WPROBE(72);
        };
        if (warp == 8) {
            if (n_my > 0) issue_load(0);
            if (lane == 0) {
                mbar_expect_tx(bar_w, (uint32_t)W_BYTES);
                bulk_g2s(w_a, p.wimg, (uint32_t)W_BYTES, bar_w);
            }
            __syncwarp();
            if (n_my > 1) issue_load(1);
        }
        for (int j = 0; j < n_my; ++j) {
            const int buf = j & 1;
            if (S_SPLIT && j + 1 < n_my) {
                // part tile (j + 1) & 1 was last read by the UMMAs of tile j - 1; its maxima slots were cleared by the compute warps
                if (j >= 1) { if (lane == 0) ws_poll(pf_count, 8 * j); __syncwarp(); __threadfence_block(); }
                x_split_s(j + 1);
            }
            WPROBE(73);
            ws_out_wait();   // the rows of B_0 of tile j are in the staging tile
            WPROBE(74);
            {
                const int node0 = tinfo_s[buf * 4 + 0], rows = tinfo_s[buf * 4 + 1];
                const uint32_t xb_a = xs_a + (uint32_t)buf * HF_TILE_BYTES;
                float* dst = p.Y + (size_t)node0 * 32;
                const float* bias_s = reinterpret_cast<const float*>(w_s + (size_t)K * 32 * 128);
                const float inv_sw = bias_s[32];
                const bool leaky_max = p.act == MHO_ACT_LEAKY && p.slope >= 0.f && p.slope <= 1.f;
                for (int c = st; c < rows * 8; c += 96) {
                    const uint32_t row = (uint32_t)c >> 3, ch = (uint32_t)c & 7u;
                    const float4 v = lds_f128(xb_a + row * 128u + ((ch ^ (row & 7u)) << 4));
                    const float4 bv = *reinterpret_cast<const float4*>(bias_s + 4 * ch);
                    float y[4] = {fmaf(v.x, inv_sw, bv.x), fmaf(v.y, inv_sw, bv.y), fmaf(v.z, inv_sw, bv.z), fmaf(v.w, inv_sw, bv.w)};
                    if (p.act == MHO_ACT_RELU) {
#pragma unroll
                        for (int e = 0; e < 4; ++e) y[e] = fmaxf(y[e], 0.f);
                    } else if (leaky_max) {
#pragma unroll
                        for (int e = 0; e < 4; ++e) y[e] = fmaxf(y[e], y[e] * p.slope);
                    } else if (p.act == MHO_ACT_LEAKY) {
#pragma unroll
                        for (int e = 0; e < 4; ++e) y[e] = y[e] > 0.f ? y[e] : p.slope * y[e];
                    }
                    *reinterpret_cast<float4*>(dst + (size_t)row * 32 + ch * 4) = make_float4(y[0], y[1], y[2], y[3]);
                }
            }
            WPROBE(75);
            ws_service_sync();   // the staging buffer (and its tile descriptor) may be refilled
            if (warp == 8 && j + 2 < n_my) issue_load(j + 2);
        }
    } else {
        // ========================================================= issue warp =========================================================
        asm volatile("setmaxnreg.dec.sync.aligned.u32 64;");
        auto issue_xw = [&](int buf) {
            const uint32_t parts_a = smem_a + (uint32_t)buf * HF_TILE_BYTES;
            // P' = X' [W'_0 | ... | W'_K-1]:  x w ~ xh wh - xh wl' - xl' wh, two 16-wide K steps each
            const uint32_t id_pos = idesc_f16((uint32_t)(32 * K), 0u, 0u), id_neg = idesc_f16((uint32_t)(32 * K), 0u, 1u);
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) umma_f16_ss(tmem_base, desc_sw128(parts_a + 64u + 32u * ks), desc_sw128(w_a + 32u * ks), id_neg, ks > 0 ? 1u : 0u);
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) umma_f16_ss(tmem_base, desc_sw128(parts_a + 32u * ks), desc_sw128(w_a + 64u + 32u * ks), id_neg, 1u);
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) umma_f16_ss(tmem_base, desc_sw128(parts_a + 32u * ks), desc_sw128(w_a + 32u * ks), id_pos, 1u);
            umma_commit(bar_mma);
        };
        if (n_my > 0) {
            ws_parts_wait();   // tile 0's rows are split (compute warps)
            if (lane == 0) { mbar_wait(bar_w, 0u); tc_fence_after(); issue_xw(0); }
            __syncwarp();
        }
        for (int j = 0; j < n_my; ++j) {
            const int buf = j & 1;
            const uint32_t parts_a = smem_a + (uint32_t)buf * HF_TILE_BYTES;
            for (int k = K - 2; k >= 0; --k) {
                WPROBE(40 + k);
                ws_parts_wait();   // the parts of B_k+1 are in place
                WPROBE(50 + k);
                if (lane == 0) {
                    tc_fence_after();
                    const int rows_t = tinfo_s[buf * 4 + 1];
                    const uint32_t id_adj = idesc_f16(64u, 1u, 0u);
                    const uint32_t d = tmem_base + (uint32_t)(32 * (k + 1));
                    const int nks = (rows_t + 15) >> 4;   // 16-node slices beyond the tile's rows are all zero
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks)
                        if (ks == 0 || ks < nks) umma_f16_ts(d, tmem_base + ADJ_COL + (uint32_t)(ks * 8), desc_sw128(parts_a + (uint32_t)ks * 2048u), id_adj, ks > 0 ? 1u : 0u);
                    umma_commit(bar_mma);
                }
                __syncwarp();
                WPROBE(60 + k);
            }
            WPROBE(65);
            ws_parts_wait();       // tile j's accumulators are consumed (and the compute warps have seen the rows of tile j + 1 split)
            WPROBE(66);
            if (j + 1 < n_my && lane == 0) { tc_fence_after(); issue_xw(buf ^ 1); }
            __syncwarp();
            WPROBE(67);
        }
    }
#ifdef MHO_PROBE
    __syncthreads();
    if (blockIdx.x == 0 && tid == 0) {
        const long long base = wprobe_s[0] >> 8;
        for (int i = 0; i < 256; ++i) {
            if (wprobe_s[i] == 0) continue;
            printf("%s id %2d  t %7lld\n", i < 88 ? "t0  " : i < 176 ? "t256" : "t352", (int)(wprobe_s[i] & 255), (wprobe_s[i] >> 8) - base);
        }
    }
#endif

    // ---- teardown
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, TCOLS);
}

template <int K, bool S_SPLIT>
cudaError_t launch_ws(const HfParams& p, size_t smem, int grid, cudaStream_t st) {
    return mho_launch<cheb_f16ws_kernel<K, S_SPLIT>>(dim3((unsigned)grid), dim3(384), smem, st, true, p);
}

template <int K>
cudaError_t launch_k(const HfParams& p, size_t smem, int grid, cudaStream_t st) {
    return mho_launch<cheb_f16_kernel<K>>(dim3((unsigned)grid), dim3(HF_THREADS), smem, st, true, p);
}

}  // namespace

// -------------------------------------------------------------------------------------------
// host side
// -------------------------------------------------------------------------------------------
static size_t hf_smem_bytes(int K, bool has_bits, int max_tile_nnz, int* stage_bytes) {
    const int nnz_cap = has_bits ? 0 : ((max_tile_nnz + 3) & ~3);
    const int stage = has_bits ? 2048 : ((528 + nnz_cap * 4 + 15) & ~15);
    if (stage_bytes) *stage_bytes = stage;
    return (size_t)4 * HF_TILE_BYTES + (size_t)hf_w_bytes(K) + 1536 + 128 + 4096 + (size_t)2 * stage + 1056 + 64 + 6 * 512;
}

bool cheb_f16_eligible(const mho_layer_t* layers, int n_layers, bool has_vals, bool has_bits, bool has_saved, bool has_graph_starts,
                       int max_tile_rows, int max_tile_nnz, const void* X, const void* Y, const void* bits, int max_smem_optin) {
    // one scale per tile is exact to 1e-5 only while tile mates stay within ~2^7 of each other in magnitude at every Clenshaw
    // step: without the graph starts (mho_batch_t.tile_graph0) the batch goes to the bf16 x 3 kernel, which needs no scales
    if (n_layers != 1 || has_vals || has_saved || !has_graph_starts || max_tile_rows > 128) return false;
    const mho_layer_t& L = layers[0];
    if (L.f_in != 32 || L.f_out != 32 || L.K < 2 || L.K > 10) return false;
    if ((reinterpret_cast<uintptr_t>(X) & 15u) || (reinterpret_cast<uintptr_t>(Y) & 15u) || (reinterpret_cast<uintptr_t>(bits) & 15u)) return false;
    const size_t smem = hf_smem_bytes(L.K, has_bits, max_tile_nnz, nullptr);
    const size_t budget = L.K <= 5 ? (size_t)(228 * 1024) / 2 - 1024 : (size_t)max_smem_optin;
    return smem <= std::min(budget, (size_t)max_smem_optin);
}

int cheb_f16_weight_bytes(int K) { return hf_w_bytes(K); }

cudaError_t prepare_f16_weights_launch(const LayerDev& L, unsigned char* out, cudaStream_t st) {
    HfPrepParams p{L.W, L.b, L.K, out};
    // the kernel writes the weight rows, bias and header, not the padding up to hf_w_bytes
    const cudaError_t e = cudaMemsetAsync(out, 0, (size_t)hf_w_bytes(L.K), st);
    if (e != cudaSuccess) return e;
    hf_prepare_weights_kernel<<<1, 256, 0, st>>>(p);
    return cudaGetLastError();
}

cudaError_t cheb_f16_launch(const FwdParams& fp, const unsigned char* wimg, int max_tile_nnz, int num_sms, int max_smem_optin, cudaStream_t st) {
    HfParams p;
    memset(&p, 0, sizeof(p));
    p.b = fp.b;
    p.X = fp.X;
    p.Y = fp.Y;
    p.wimg = wimg;
    p.act = fp.layers[0].act;
    p.slope = fp.layers[0].slope;
    p.use_bits = fp.b.adj_bits != nullptr ? 1 : 0;
    const int K = fp.layers[0].K;
    int stage = 0;
    p.nnz_cap = p.use_bits ? 0 : ((max_tile_nnz + 3) & ~3);
    const size_t smem = hf_smem_bytes(K, p.use_bits != 0, max_tile_nnz, &stage);
    p.stage_bytes = stage;
    int grid = num_sms * (K <= 5 ? 2 : 1);   // (one CTA per SM per launch + more streams was measured: no gain)
    if (grid > p.b.n_tiles) grid = p.b.n_tiles;
    if (grid < 1) grid = 1;
    if (K <= 5 && p.use_bits && p.b.tile_graph0 != nullptr) {
        switch (K) {
            // who splits the next tile's rows: the compute warps inside their wait windows (short tiles: the 96 service threads need
            // ~7 k cycles for a tile's rows), or the service warps (K >= 4: 5 % faster on the benchmark layer)
            case 2: return launch_ws<2, false>(p, smem, grid, st);
            case 3: return launch_ws<3, false>(p, smem, grid, st);
            case 4: return launch_ws<4, true>(p, smem, grid, st);
            default: return launch_ws<5, true>(p, smem, grid, st);
        }
    }
    switch (K) {
        case 2: return launch_k<2>(p, smem, grid, st);
        case 3: return launch_k<3>(p, smem, grid, st);
        case 4: return launch_k<4>(p, smem, grid, st);
        case 5: return launch_k<5>(p, smem, grid, st);
        case 6: return launch_k<6>(p, smem, grid, st);
        case 7: return launch_k<7>(p, smem, grid, st);
        case 8: return launch_k<8>(p, smem, grid, st);
        case 9: return launch_k<9>(p, smem, grid, st);
        case 10: return launch_k<10>(p, smem, grid, st);
        default: return cudaErrorInvalidValue;
    }
}
