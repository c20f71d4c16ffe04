// VJP of ONE ChebConv layer on the tensor cores (sm_100a, tcgen05 + TMEM): the training step of the benchmark
// configuration and of the reference's K > 1 models - 32 -> 32 features, 2 <= K <= 10, BINARY operator (vals == NULL),
// graphs of <= 128 nodes, first layer (no input gradient).  Replaces, for those shapes, the tape replay
//   gradients = g.gradient(delay_mtx_ts, self.model.trainable_weights, output_gradients=grad_dist_np)
// (gnn_offloading_agent.py:448); everything else stays with cheb_backward.cu.  One gradient vector PER GRAPH is written
// (the reference memorises one gradient list per instance, :142/:450, and replays them one by one, :156-169).
//
//   G = dOut (.) act'(Out)        db = sum_i G[i, :]        dW_k = T_k^T G,   T_0 = X, T_1 = A X, T_k = 2 A T_k-1 - T_k-2
//
// One graph per CTA pass, two CTAs per SM, 12 warps per CTA in three roles (register budgets re-balanced with setmaxnreg):
//   * 8 COMPUTE warps (thread = one node row x 16 of the 32 columns) carry the recurrence: they wait for A T_k-1 in tensor
//     memory, form T_k in packed fp32, split it into two fp16 parts (x = h - l', 22 significand bits, ONE power-of-two scale
//     per graph and step - the node rows are the reduction dimension of both products, so a scale may not vary along them)
//     and arrive on a named barrier.  Nothing else sits on their critical path.
//   * 2 ISSUE warps: thread 320 issues the recurrence product (A = the graph's 128 x 128 adjacency block in tensor memory as
//     fp16 0 / 1, B = the part tile [node][h 64 B | l' 64 B] of T_k, MN-major, N = 64), then thread 352 issues
//     dW_k^T = G^T T_k as ONE more UMMA per 16-node slice on the same part tile (A = the part tile of G read MN-major: rows
//     of D = [G_h o | G_l' o], columns = [T_h f | T_l' f]).  An issuing thread stalls until the tensor pipe has accepted its
//     group (~50-100 cycles per UMMA): that is why these are not compute warps.
//   * 2 SERVICE warps (TMEM lanes 0-63): cp.async of the next graph's X, dOut, Out rows (16 B chunks XOR-swizzled with the
//     row) and bit rows; db = exact fp32 column sums of G in a fixed order; and the drain of the dW accumulators (two
//     64-column accumulators alternate): (hh - hl') - (l'h - l'l') through a shared-memory exchange between the two lane
//     quadrants, un-scaled, as coalesced 128 B rows of the gradient vector.
// Scales: max |X|, max |G| and the maximum degree are reduced across the compute warps once per graph; the scales of
// T_1 .. T_K-1 come from the a-priori bound beta_k = 2 dmax beta_k-1 + beta_k-2 (K <= 6) or from the running maxima of
// |T_k-1|, |T_k-2| (K > 6: the a-priori recurrence loses ~3 bits per step).
// Tensor memory: 64 columns recurrence accumulator | 2 x 64 dW accumulators | 64 adjacency = 256 -> two CTAs per SM.
#include <algorithm>
#include <cstdio>
#include <cstring>

#include "mho_common.cuh"
#include "mho_internal.h"
#include "f16_common.cuh"

// -DMHO_PROBE: CTA 0 records clock64 marks of threads 0 (compute), 320 (issuer) and prints them
#ifdef MHO_PROBE
#define BPROBE(id) do { if (blockIdx.x == 0 && (tid == 0 || tid == 256 || tid == 320 || tid == 352) && pn < 64) { probe_s[(tid == 0 ? 0 : tid == 256 ? 64 : tid == 320 ? 128 : 192) + pn] = (clock64() << 8) | (long long)(id); ++pn; } } while (0)
#else
#define BPROBE(id) do { } while (0)
#endif

namespace {

constexpr int BF_THREADS = 384;
constexpr uint32_t BF_TCOLS = 256u, BF_ADJ_COL = 192u, BF_DW_COL = 64u;

struct BfParams {
    const int32_t* graph_off;
    const uint32_t* adj_bits;   // [total_nodes][4], bit j of word w of node i: i ~ graph_node0(i) + 32 w + j
    int n_graphs;
    const float* X;
    const float* Y;
    const float* dY;
    float* grads;               // [n_graphs][n_params]: W[K][32][32] then b[32]
    long long n_params;
    int K;
    int act;
    float slope;
};

// shared memory (1024-aligned): two T part tiles | G part tile | X, dY, Y staging (swizzled 128 B rows) | bit rows | drain
// staging [2][32][32] | control block
constexpr uint32_t BF_PT = 0, BF_PG = 2 * HF_TILE_BYTES, BF_XS = 3 * HF_TILE_BYTES, BF_DS = 4 * HF_TILE_BYTES, BF_YS = 5 * HF_TILE_BYTES,
                   BF_BITS = 6 * HF_TILE_BYTES, BF_STG = BF_BITS + 2048, BF_CTL = BF_STG + 8192, BF_SMEM = BF_CTL + 1024;

// named barriers: 1 = parts ready (256 compute arrive, the recurrence issue warp waits; the dW issue warp, which may lag a
// step behind, polls a monotonic shared-memory counter of warp arrivals instead),
// 3 = the two service warps (db), 4 = staging rows consumed (256 compute arrive, the 2 service warps wait), 5 = compute warps,
// 6 / 7 = drain exchange of the even / odd dW accumulator, 8 / 9 = that accumulator is drained (service warps -> dW warp)
__device__ __forceinline__ void bar_parts_arrive() { asm volatile("bar.arrive 1, 288;" ::: "memory"); }
__device__ __forceinline__ void bar_parts_wait() { asm volatile("bar.sync 1, 288;" ::: "memory"); }
__device__ __forceinline__ void bar_loaders() { asm volatile("bar.sync 3, 64;" ::: "memory"); }
__device__ __forceinline__ void bar_staging_arrive() { asm volatile("bar.arrive 4, 320;" ::: "memory"); }
__device__ __forceinline__ void bar_staging_wait() { asm volatile("bar.sync 4, 320;" ::: "memory"); }
__device__ __forceinline__ void bar_compute_warps() { asm volatile("bar.sync 5, 256;" ::: "memory"); }
__device__ __forceinline__ void bar_drain(int which) {   // the two service warps, blocking on both sides
    if (which == 0) asm volatile("bar.sync 6, 64;" ::: "memory"); else asm volatile("bar.sync 7, 64;" ::: "memory");
}
__device__ __forceinline__ void bar_drained(int which, bool wait) {   // 64 service threads arrive, the dW warp waits
    if (which == 0) { if (wait) asm volatile("bar.sync 8, 96;" ::: "memory"); else asm volatile("bar.arrive 8, 96;" ::: "memory"); }
    else { if (wait) asm volatile("bar.sync 9, 96;" ::: "memory"); else asm volatile("bar.arrive 9, 96;" ::: "memory"); }
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
}

template <bool TRACK>
__global__ void __launch_bounds__(BF_THREADS, 2) cheb_backward_f16_kernel(const __grid_constant__ BfParams p) {
    extern __shared__ __align__(1024) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t smem_a = smem_u32(smem);
    const uint32_t pt_a = smem_a + BF_PT, pg_a = smem_a + BF_PG, xs_a = smem_a + BF_XS, ds_a = smem_a + BF_DS, ys_a = smem_a + BF_YS,
                   bits_a = smem_a + BF_BITS, ctl_a = smem_a + BF_CTL;
    unsigned char* ctl_s = smem + BF_CTL;
    // control block: loads +0, recurrence +8, dW[2] +16, tmem slot +32, reductions +64 ([2][4]), exponent of the G scale +96 ([2]),
    // LUT +128, db halves +256 ([2][32]), scale exponents of T_k +512 ([2][16]), running maxima of |T_k| +768 ([2][16])
    const uint32_t bar_ld = ctl_a, bar_mma = ctl_a + 8, bar_dw = ctl_a + 16, tslot = ctl_a + 32, lut_a = ctl_a + 128;
    unsigned int* red_s = reinterpret_cast<unsigned int*>(ctl_s + 64);
    volatile int* egs_s = reinterpret_cast<volatile int*>(ctl_s + 96);
    volatile int* pcount_s = reinterpret_cast<volatile int*>(ctl_s + 108);  // compute-warp arrivals so far (8 per step)
    volatile int* cstep_s = reinterpret_cast<volatile int*>(ctl_s + 104);   // recurrence groups issued so far (graph * 16 + step + 1)
    float* dbh_s = reinterpret_cast<float*>(ctl_s + 256);
    volatile int* esc_s = reinterpret_cast<volatile int*>(ctl_s + 512);
    unsigned int* trk_s = reinterpret_cast<unsigned int*>(ctl_s + 768);
    float* stg_s = reinterpret_cast<float*>(smem + BF_STG);
#ifdef MHO_PROBE
    __shared__ long long probe_s[256];
    int pn = 0;
    if (tid < 256) probe_s[tid] = 0;
    __syncthreads();
#endif
    const int G = (int)gridDim.x, K = p.K;
    const int n_my = (int)blockIdx.x < p.n_graphs ? (p.n_graphs - (int)blockIdx.x + G - 1) / G : 0;

    if (tid == 0) {
        mbar_init(bar_ld, 64);       // one cp.async arrive per load thread
        mbar_init(bar_mma, 1);
        mbar_init(bar_dw, 1);
        mbar_init(bar_dw + 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (tid < 16) {
        const uint32_t x = ((tid & 1) ? 0x3C00u : 0u) | ((tid & 2) ? 0x3C000000u : 0u), y = ((tid & 4) ? 0x3C00u : 0u) | ((tid & 8) ? 0x3C000000u : 0u);
        asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(lut_a + (uint32_t)tid * 8u), "r"(x), "r"(y) : "memory");
    }
    if (tid < 8) red_s[tid] = 0u;
    if (tid == 0) { *cstep_s = 0; *pcount_s = 0; }
    if (tid < 32) trk_s[tid] = 0u;
    if (warp == 0) tmem_alloc(tslot, BF_TCOLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(ctl_s + 32);

    // graph extents are fetched one graph ahead (every role needs them)
    int nx_node0 = 0, nx_rows = 0;
    auto prefetch_extent = [&](int j) {
        if (j < n_my) {
            const int g = (int)blockIdx.x + j * G;
            nx_node0 = __ldg(p.graph_off + g);
            nx_rows = __ldg(p.graph_off + g + 1) - nx_node0;
        }
    };
    prefetch_extent(0);

    if (warp < 8) {
        // =================================================== compute warps ===================================================
        asm volatile("setmaxnreg.inc.sync.aligned.u32 88;");
        const int q = warp & 3, hh = warp >> 2;                 // TMEM lane quadrant, column half
        const uint32_t r = (uint32_t)(q * 32 + lane);           // graph row = TMEM lane
        const uint32_t tmem_lane = tmem_base + ((uint32_t)(q * 32) << 16);
        const uint32_t key = r & 7u;
        uint32_t ph_mma = 0, ph_dw0 = 0, ph_dw1 = 0;
        auto wait_dw = [&](int k) {
            if (k & 1) { mbar_wait(bar_dw + 8, ph_dw1); ph_dw1 ^= 1u; } else { mbar_wait(bar_dw, ph_dw0); ph_dw0 ^= 1u; }
        };
        // scaled fp32 row -> two fp16 parts into row r of a part tile
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

        for (int j = 0; j < n_my; ++j) {
            const int rows = nx_rows;
            prefetch_extent(j + 1);
            const bool live = (int)r < rows;

            // ---- input rows: T_0 = X, G = dOut (.) act'(Out); the graph's maxima; adjacency -> tensor memory
            BPROBE(1);
            mbar_wait(bar_ld, (uint32_t)(j & 1));
            BPROBE(2);
            float tp[16], tpp[16];
            {
                float gr[16];
                float xm = 0.f, gm = 0.f;
                unsigned int deg = 0u;
                uint2 m2v = make_uint2(0u, 0u);
                if (live) {
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const uint32_t off = r * 128u + (((uint32_t)(4 * hh + c) ^ key) << 4);
                        const float4 x4 = lds_f128(xs_a + off), d4 = lds_f128(ds_a + off), y4 = lds_f128(ys_a + off);
                        tp[4 * c] = x4.x; tp[4 * c + 1] = x4.y; tp[4 * c + 2] = x4.z; tp[4 * c + 3] = x4.w;
                        gr[4 * c] = d4.x * act_grad_from_out(y4.x, p.act, p.slope);
                        gr[4 * c + 1] = d4.y * act_grad_from_out(y4.y, p.act, p.slope);
                        gr[4 * c + 2] = d4.z * act_grad_from_out(y4.z, p.act, p.slope);
                        gr[4 * c + 3] = d4.w * act_grad_from_out(y4.w, p.act, p.slope);
                    }
                    const uint4 m4 = lds_u128(bits_a + r * 16u);
                    deg = __popc(m4.x) + __popc(m4.y) + __popc(m4.z) + __popc(m4.w);
                    m2v = hh ? make_uint2(m4.z, m4.w) : make_uint2(m4.x, m4.y);
                } else {
#pragma unroll
                    for (int e = 0; e < 16; ++e) { tp[e] = 0.f; gr[e] = 0.f; }
                }
                bar_staging_arrive();   // this thread's staging rows are consumed (the load warps refill them once all have arrived)
#pragma unroll
                for (int e = 0; e < 16; ++e) { tpp[e] = 0.f; xm = fmaxf(xm, fabsf(tp[e])); gm = fmaxf(gm, fabsf(gr[e])); }
                {
                    const unsigned int wx = __reduce_max_sync(0xffffffffu, __float_as_uint(xm));
                    const unsigned int wg = __reduce_max_sync(0xffffffffu, __float_as_uint(gm));
                    const unsigned int wd = __reduce_max_sync(0xffffffffu, deg);
                    unsigned int* red = red_s + (j & 1) * 4;
                    if (lane == 0) { atomicMax(red, wx); atomicMax(red + 1, wg); atomicMax(red + 2, wd); }
                }
                // adjacency block -> tensor memory as fp16 0 / 1 pairs (the previous graph's recurrence UMMAs have completed)
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
                    tmem_st16(tmem_lane + BF_ADJ_COL + (uint32_t)(32 * hh + 16 * w2), aw);
                }
                BPROBE(3);
                bar_compute_warps();   // the maxima are complete
                BPROBE(4);
                const unsigned int* red = red_s + (j & 1) * 4;
                const float gmax = __uint_as_float(red[1]);
                const int eg = max(-100, min(110, expo_above(gmax)));   // |G| < 2^eg
                if (tid == 0) egs_s[j & 1] = eg;
                // the previous graph's last two dW products read the part tiles that are rewritten now
                if (j > 0) { wait_dw(K - 2); wait_dw(K - 1); }
                split_row(pg_a, gr, pow2f(15 - eg));
            }
            const unsigned int* red = red_s + (j & 1) * 4;
            const float xmax = __uint_as_float(red[0]);
            const float dmax = (float)red[2];
            if (tid == 0) { unsigned int* o = red_s + ((j + 1) & 1) * 4; o[0] = 0u; o[1] = 0u; o[2] = 0u; }
            unsigned int* trk = trk_s + (j & 1) * 16;
            if (TRACK && tid < 16) trk_s[((j + 1) & 1) * 16 + tid] = 0u;   // last read a graph ago
            volatile int* esc = esc_s + (j & 1) * 16;
            int e_cur = max(-100, min(110, expo_above(xmax)));     // |T_0| < 2^e_cur
            float bet1 = xmax, bet2 = 0.f;                          // bounds of |T_k-1|, |T_k-2|
            if (tid == 0) esc[0] = e_cur;
            split_row(pt_a, tp, pow2f(15 - e_cur));
            fence_proxy_async();
            tmem_wait_st_();
            tc_fence_before();
            __threadfence_block();
            BPROBE(5);
            __syncwarp();
            if (lane == 0) atomicAdd(const_cast<int*>(pcount_s), 1);
            bar_parts_arrive();

            int e_prev = e_cur;
            for (int k = 1; k < K; ++k) {
                // ---- T_k = c (A T_k-1) - T_k-2
                BPROBE(10 + k);
                mbar_wait(bar_mma, ph_mma);
                ph_mma ^= 1u;
                tc_fence_after();
                BPROBE(20 + k);
                uint32_t vh[16], vl[16];
                tmem_ld16(tmem_lane + (uint32_t)(16 * hh), vh);
                tmem_ld16(tmem_lane + 32u + (uint32_t)(16 * hh), vl);
                tmem_wait_ld_();
                const float cfac = pow2f(e_prev - 15 + (k > 1 ? 1 : 0));   // (k > 1 ? 2 : 1) / tau_k-1
                const uint64_t C2 = pk2(cfac, cfac);
                float m = 0.f;
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const uint64_t dv = sub2(pk2(__uint_as_float(vh[2 * e]), __uint_as_float(vh[2 * e + 1])), pk2(__uint_as_float(vl[2 * e]), __uint_as_float(vl[2 * e + 1])));
                    const uint64_t tk = fma2(dv, C2, pk2(-tpp[2 * e], -tpp[2 * e + 1]));
                    tpp[2 * e] = tp[2 * e]; tpp[2 * e + 1] = tp[2 * e + 1];
                    upk2(tk, tp[2 * e], tp[2 * e + 1]);
                    if (TRACK) m = fmaxf(m, fmaxf(fabsf(tp[2 * e]), fabsf(tp[2 * e + 1])));
                }
                if (TRACK) {
                    // the maxima of |T_k-1| and |T_k-2| are complete (their atomics preceded an arrive and an UMMA round): a bound
                    // of |T_k| that overshoots by one step's factor at most
                    if (k >= 2) bet1 = __uint_as_float(trk[k - 1]);
                    if (k >= 3) bet2 = __uint_as_float(trk[k - 2]);
                    const unsigned int wm = __reduce_max_sync(0xffffffffu, __float_as_uint(m));
                    if (lane == 0) atomicMax(trk + k, wm);
                }
                const float bet = (k > 1 ? 2.f : 1.f) * dmax * bet1 + bet2;
                bet2 = bet1;
                bet1 = bet;
                e_cur = max(-100, min(110, expo_above(bet)));
                if (tid == 0) esc[k] = e_cur;
                if (k >= 2) wait_dw(k - 2);   // its UMMAs read the part tile that is rewritten now (complete long ago)
                split_row(pt_a + (uint32_t)(k & 1) * HF_TILE_BYTES, tp, pow2f(15 - e_cur));
                fence_proxy_async();
                tc_fence_before();
                __threadfence_block();
                BPROBE(30 + k);
                __syncwarp();
                if (lane == 0) atomicAdd(const_cast<int*>(pcount_s), 1);
                bar_parts_arrive();
                e_prev = e_cur;
            }
        }
    } else {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
        if (warp >= 10) {
            // ================================================== issue warps ==================================================
            // Thread 320 issues the recurrence product, then thread 352 the dW product of the same part tile.  An issuing thread
            // stalls until the tensor pipe has accepted its group: these warps do nothing else.
            const bool chain_warp = warp == 10;
            const uint32_t id_adj = idesc_f16(64u, 1u, 0u);                 // A from tensor memory, B MN-major
            const uint32_t id_dw = idesc_f16(64u, 1u, 0u) | (1u << 15);     // A (the G part tile) MN-major too
            int issued0 = 0, issued1 = 0;   // dW groups issued into accumulator 0 / 1 so far
            int dstep = 0;                  // steps seen so far
            for (int j = 0; j < n_my; ++j) {
                const int rows = nx_rows;
                prefetch_extent(j + 1);
                const int nks = (rows + 15) >> 4;   // 16-node slices beyond the graph's rows are all zero
                for (int k = 0; k < K; ++k) {
                    BPROBE(40 + k);
                    // the parts of T_k (k = 0: and of G, the adjacency block) are in place
                    ++dstep;
                    if (chain_warp) bar_parts_wait();
                    else { if (lane == 0) { while (*pcount_s < 8 * dstep) { } } __syncwarp(); __threadfence_block(); }
                    BPROBE(50 + k);
                    tc_fence_after();
                    const uint32_t ptk = pt_a + (uint32_t)(k & 1) * HF_TILE_BYTES;
                    if (chain_warp) {
                        if (lane == 0 && k + 1 < K) {
#pragma unroll
                            for (int ks = 0; ks < 8; ++ks)
                                if (ks == 0 || ks < nks) umma_f16_ts(tmem_base, tmem_base + BF_ADJ_COL + (uint32_t)(ks * 8), desc_sw128(ptk + (uint32_t)ks * 2048u), id_adj, ks > 0 ? 1u : 0u);
                            umma_commit(bar_mma);
                        }
                        if (lane == 0) *cstep_s = j * 16 + k + 1;   // (after the group has been accepted)
                        __syncwarp();
                        BPROBE(60 + k);
                    } else {
                        // the accumulator's previous contents have been drained
                        if (k & 1) { if (issued1 > 0) bar_drained(1, true); ++issued1; } else { if (issued0 > 0) bar_drained(0, true); ++issued0; }
                        BPROBE(80 + k);
                        // the recurrence product goes first (the compute warps wait for it); the recurrence warp may be a step ahead
                        if (lane == 0) { while (*cstep_s < j * 16 + k + 1) { } }
                        __syncwarp();
                        BPROBE(90 + k);
                        if (lane == 0) {
                            tc_fence_after();
                            const uint32_t d = tmem_base + BF_DW_COL + 64u * (uint32_t)(k & 1);
#pragma unroll
                            for (int ks = 0; ks < 8; ++ks)
                                if (ks == 0 || ks < nks) umma_f16_ss(d, desc_sw128(pg_a + (uint32_t)ks * 2048u), desc_sw128(ptk + (uint32_t)ks * 2048u), id_dw, ks > 0 ? 1u : 0u);
                            umma_commit(bar_dw + 8u * (uint32_t)(k & 1));
                        }
                        __syncwarp();
                        BPROBE(100 + k);
                    }
                }
            }
        } else {
            // ================================================= service warps =================================================
            // loads of the next graph, db, and the drain of the dW accumulators (warp 8: TMEM lanes 0-31 = rows G_h o, warp 9: lanes
            // 32-63 = rows G_l' o)
            const int lt = tid - 256;   // 0 .. 63
            const bool h_warp = warp == 8;
            const uint32_t tmem_lane = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
            uint32_t ph_dw0 = 0, ph_dw1 = 0;
            // rows of X, dY, Y (16 B chunks XOR-swizzled with the row: the row-per-lane reads of the compute warps are
            // conflict-free) and bit rows
            auto issue_loads = [&](int node0, int rows) {
                for (int c = lt; c < rows * 8; c += 64) {
                    const int row = c >> 3, ch = c & 7;
                    const uint32_t d = (uint32_t)row * 128u + (uint32_t)((ch ^ (row & 7)) << 4);
                    const size_t sidx = (size_t)(node0 + row) * 32 + (size_t)ch * 4;
                    cp_async16(xs_a + d, p.X + sidx);
                    cp_async16(ds_a + d, p.dY + sidx);
                    cp_async16(ys_a + d, p.Y + sidx);
                }
                for (int i = lt; i < rows; i += 64) cp_async16(bits_a + (uint32_t)i * 16u, p.adj_bits + (size_t)(node0 + i) * 4);
                cp_async_mbar_arrive(bar_ld);
            };
            if (n_my > 0) issue_loads(nx_node0, nx_rows);
            for (int j = 0; j < n_my; ++j) {
                const int rows = nx_rows;
                float* gout = p.grads + (size_t)((int)blockIdx.x + j * G) * p.n_params;
                prefetch_extent(j + 1);
                BPROBE(1);
                mbar_wait(bar_ld, (uint32_t)(j & 1));
                BPROBE(2);
                // db[o] = sum_r G[r][o]: thread = (column o, half of the rows), fixed order, exact fp32
                {
                    const int o = lt & 31, half = lt >> 5;
                    const int r0 = half * 64, r1 = min(rows, r0 + 64);
                    float sum = 0.f;
                    const uint32_t ocol = ((uint32_t)o & 3u) * 4u, och = (uint32_t)o >> 2;
                    int rb = r0;
                    for (; rb + 8 <= r1; rb += 8) {   // 8 rows in flight, added in row order (rb is a multiple of 8: row & 7 = i)
                        const uint32_t base = (uint32_t)rb * 128u + ocol;
                        float d[8], y[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const uint32_t off = base + (uint32_t)i * 128u + ((och ^ (uint32_t)i) << 4);
                            d[i] = lds_f32(ds_a + off);
                            y[i] = lds_f32(ys_a + off);
                        }
#pragma unroll
                        for (int i = 0; i < 8; ++i) sum += d[i] * act_grad_from_out(y[i], p.act, p.slope);
                    }
                    for (; rb < r1; ++rb) {
                        const uint32_t off = (uint32_t)rb * 128u + ((och ^ ((uint32_t)rb & 7u)) << 4) + ocol;
                        sum += lds_f32(ds_a + off) * act_grad_from_out(lds_f32(ys_a + off), p.act, p.slope);
                    }
                    dbh_s[half * 32 + o] = sum;
                    bar_loaders();
                    if (half == 0) gout[(size_t)K * 1024 + o] = dbh_s[o] + dbh_s[32 + o];
                }
                BPROBE(3);
                bar_staging_wait();   // every compute thread has read its rows (and this warp pair its own)
                BPROBE(4);
                if (j + 1 < n_my) issue_loads(nx_node0, nx_rows);
                BPROBE(5);
                // dW_k accumulator -> gradient rows.  D rows: [G_h o | G_l' o] (lanes 0-31 / 32-63), D columns: [T_h f | T_l' f]:
                // (hh - hl') - (l'h - l'l'), the second bracket through shared memory, un-scaled, as coalesced 128 B rows
                volatile int* esc = esc_s + (j & 1) * 16;
                for (int k = 0; k < K; ++k) {
                    BPROBE(10 + k);
                    if (k & 1) { mbar_wait(bar_dw + 8, ph_dw1); ph_dw1 ^= 1u; } else { mbar_wait(bar_dw, ph_dw0); ph_dw0 ^= 1u; }
                    BPROBE(20 + k);
                    tc_fence_after();
                    const uint32_t col = BF_DW_COL + 64u * (uint32_t)(k & 1);
                    float* st = stg_s + (k & 1) * 1024 + lane;
                    // each warp finishes 16 of the 32 f columns (warp 8: f < 16, warp 9: f >= 16) and hands the other 16 over
                    const int keep0 = h_warp ? 0 : 16, give0 = h_warp ? 16 : 0;
                    float w[16];
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        uint32_t a[8], b[8];
                        tmem_ld8(tmem_lane + col + (uint32_t)(give0 + 8 * c), a);
                        tmem_ld8(tmem_lane + col + 32u + (uint32_t)(give0 + 8 * c), b);
                        tmem_wait_ld_();
#pragma unroll
                        for (int e = 0; e < 8; ++e) st[(give0 + 8 * c + e) * 32] = __uint_as_float(a[e]) - __uint_as_float(b[e]);
                    }
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        uint32_t a[8], b[8];
                        tmem_ld8(tmem_lane + col + (uint32_t)(keep0 + 8 * c), a);
                        tmem_ld8(tmem_lane + col + 32u + (uint32_t)(keep0 + 8 * c), b);
                        tmem_wait_ld_();
#pragma unroll
                        for (int e = 0; e < 8; ++e) w[8 * c + e] = __uint_as_float(a[e]) - __uint_as_float(b[e]);
                    }
                    tc_fence_before();
                    const float us = (h_warp ? 1.f : -1.f) * pow2f(esc[k] - 15) * pow2f(egs_s[j & 1] - 15);
                    float* dst = gout + (size_t)k * 1024 + keep0 * 32 + lane;
                    bar_drain(k & 1);
#pragma unroll
                    for (int e = 0; e < 16; ++e) dst[e * 32] = (w[e] - st[(keep0 + e) * 32]) * us;   // warp 9: -(l' part - h part)
                    BPROBE(30 + k);
                    bar_drained(k & 1, false);   // both warps have read the accumulator: the dW warp may overwrite it
                }
            }
        }
    }
#ifdef MHO_PROBE
    __syncthreads();
    if (blockIdx.x == 0 && tid == 0) {
        const long long base = probe_s[0] >> 8;
        for (int i = 0; i < 256; ++i) {
            if (probe_s[i] == 0) continue;
            printf("%s id %2d  t %7lld\n", i < 64 ? "t0  " : i < 128 ? "t256" : i < 192 ? "t320" : "t352", (int)(probe_s[i] & 255), (probe_s[i] >> 8) - base);
        }
    }
#endif

    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, BF_TCOLS);
}

}  // namespace

// -------------------------------------------------------------------------------------------
// host side
// -------------------------------------------------------------------------------------------
bool cheb_backward_f16_eligible(const mho_batch_t* b, const mho_layer_t* layers, int n_layers, const void* X, const void* Y, const void* dY,
                                const void* dX, int max_smem_optin) {
    if (n_layers != 1 || dX != nullptr || b->vals != nullptr || b->adj_bits == nullptr || b->max_tile_rows > 128) return false;
    const mho_layer_t& L = layers[0];
    if (L.f_in != 32 || L.f_out != 32 || L.K < 2 || L.K > 10) return false;
    if ((reinterpret_cast<uintptr_t>(X) & 15u) || (reinterpret_cast<uintptr_t>(Y) & 15u) || (reinterpret_cast<uintptr_t>(dY) & 15u) ||
        (reinterpret_cast<uintptr_t>(b->adj_bits) & 15u))
        return false;
    return (size_t)BF_SMEM + 1024 <= (size_t)max_smem_optin;
}

cudaError_t cheb_backward_f16_launch(const mho_batch_t* b, const mho_layer_t* layers, const float* X, const float* Y, const float* dY,
                                     float* grads, long long n_params, int num_sms, cudaStream_t st) {
    BfParams p;
    memset(&p, 0, sizeof(p));
    p.graph_off = b->graph_off;
    p.adj_bits = b->adj_bits;
    p.n_graphs = b->n_graphs;
    p.X = X; p.Y = Y; p.dY = dY;
    p.grads = grads;
    p.n_params = n_params;
    p.K = layers[0].K;
    p.act = layers[0].act;
    p.slope = layers[0].slope;
    const size_t smem = (size_t)BF_SMEM + 1024;
    const dim3 grid((unsigned)std::min(2 * num_sms, std::max(1, p.n_graphs)));
    if (p.K > 6) return mho_launch<cheb_backward_f16_kernel<true>>(grid, dim3(BF_THREADS), smem, st, false, p);   // running-maximum scales
    return mho_launch<cheb_backward_f16_kernel<false>>(grid, dim3(BF_THREADS), smem, st, false, p);
}
