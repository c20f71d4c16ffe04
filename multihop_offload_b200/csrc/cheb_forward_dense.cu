// ChebConv stack forward, all-tensor-core form (sm_100a, tcgen05 + TMEM) for batches of small graphs with a
// BINARY adjacency (vals == NULL): replaces model([x_in, a_in]) of gnn_offloading_agent.py:149 (model of :81-123,
// spektral ChebConv) for tiles of <= 128 nodes.
//
// A tile of packed graphs is at most 128 nodes, so its block of the operator fits one UMMA: the tile's adjacency is
// expanded into a dense 128 x 128 bf16 matrix (0/1 - exact in any format) and the sparse recurrence becomes a
// tensor-core product.  The polynomial is evaluated with Clenshaw's recurrence, which needs
// the input only once:
//      P_k   = X W_k                         one UMMA, N = K * 32 columns of TMEM           (k = 0..K-1)
//      B_K-1 = P_K-1
//      B_k   = P_k + 2 A B_k+1 - B_k+2       UMMA accumulating A (2 B_k+1) straight onto P_k's TMEM columns
//      out   = P_0 + A B_1 - B_2             (then bias, activation)
// fp32 operands are carried through the bf16 tensor core as three bf16 parts (x = h + m + l exactly, 8 + 8 + 8
// mantissa bits); 0/1 times a part is exact and TMEM accumulates in fp32, so the adjacency products are fp32-grade,
// and X W keeps the six part products down to 2^-24 relative.  CUDA cores only move accumulators: per step each
// thread reads its 8 TMEM values (row = TMEM lane, 8 columns), applies the recurrence with B_k+1 / B_k+2 held in
// registers, splits the result into parts and stores three 16 B chunks.  No CSR walk, no row segments, no fixups.
//
// The tile's adjacency lives in TENSOR MEMORY (A operand of the UMMA, 128 lanes x 64 columns of bf16 pairs, written with
// tcgen05.st from 16 B of adjacency bits per node); the three part tiles ([node][32 bf16], 64 B rows, SWIZZLE_64B) are
// at once the K-major A operand of X W and the MN-major B operand of A B (three N-atoms one LBO apart: one N = 96 UMMA
// per 16 nodes covers the three parts).  Shared memory per CTA (2 CTAs / SM, tensor memory is the limit): part tiles
// 24 KB, the bf16 weight parts of every layer, two operator staging sets, a 16 KB input staging tile.
#include <cuda_bf16.h>
#include <algorithm>
#include <cstdio>
#include <cstring>

#include "mho_common.cuh"
#include "mho_internal.h"

// -DMHO_PROBE: CTA 0 records clock64 marks of its first tile (thread 0 = UMMA issuer, thread 479 = a plain worker)
#ifdef MHO_PROBE
#ifndef MHO_PROBE_IT
#define MHO_PROBE_IT 1
#endif
#define PROBE(id) do { if (blockIdx.x == 0 && it == MHO_PROBE_IT && (tid == 0 || tid == 479) && pn < 48) { pt[pn] = clock64(); pid[pn++] = (id); } } while (0)
#else
#define PROBE(id) do { } while (0)
#endif

namespace {

constexpr int DN_THREADS = 512;
constexpr int DN_PART_BYTES = 128 * 64;  // one bf16 part tile: 128 nodes x 32 features

struct DenseParams {
    BatchDev b;
    int n_layers;
    LayerDev layers[MHO_MAX_LAYERS];
    const float* X;
    float* Y;
    float* saved;
    const unsigned char* wimg;         // per layer: [part h][part m][part l] (n_rows x 64 B each) + 128 B bias row
    int w_off[MHO_MAX_LAYERS];         // byte offset of each layer's block (multiples of 1024)
    int w_bytes;                       // bytes of the shared-memory weight region
    int w_resident;                    // 1: every layer's images stay in shared memory; 0: two slots of w_slot bytes, layers stream through
    int w_slot;
    int w_lbytes[MHO_MAX_LAYERS];      // bytes of each layer's block
    int nnz_cap;                       // staged colidx capacity (multiple of 4)
    int stage_words;                   // words per operator staging set: 512 (bit rows) or 132 + nnz_cap (CSR slice)
    int need_adj;                      // some layer has K > 1
    int tmem_cols;                     // power of two >= max_l K_l * nblk_l
    int* sched;
};

__host__ __device__ inline int dn_nblk(int K, int f_out) { return K > 1 ? 32 : pad16(f_out); }
__host__ __device__ inline int dn_layer_rows(int K, int f_out) { return K * dn_nblk(K, f_out); }
__host__ __device__ inline int dn_layer_bytes(int K, int f_out) { return (3 * dn_layer_rows(K, f_out) * 64 + 128 + 1023) & ~1023; }

// [rows][32 bf16] tile with 64 B rows, SWIZZLE_64B: 16 B chunk c of row r lives at chunk c ^ ((r >> 1) & 3)
__device__ __forceinline__ uint32_t sw64_off(uint32_t row, uint32_t chunk) { return (row << 6) | ((chunk ^ ((row >> 1) & 3u)) << 4); }

// x = h + m + l with three bf16 (exact for normal fp32): truncate, subtract, truncate, subtract
__device__ __forceinline__ void split3(float x, uint32_t& h, uint32_t& m, uint32_t& l) {
    const uint32_t xb = __float_as_uint(x);
    h = xb & 0xffff0000u;
    const float r1 = x - __uint_as_float(h);
    m = __float_as_uint(r1) & 0xffff0000u;
    const float r2 = r1 - __uint_as_float(m);
    l = __float_as_uint(r2) & 0xffff0000u;  // r2 has <= 8 significant bits: already a bf16
}

// eight fp32 -> one 16 B chunk per part, stored at (row, chunk) of the three part tiles.  A part is the upper half of
// the fp32 word, so two neighbours pack with one byte permute; the remainders come from exact subtractions.
__device__ __forceinline__ void store_parts(uint32_t parts_a, uint32_t row, uint32_t chunk, const float (&v)[8]) {
    uint32_t ph[4], pm[4], pl[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float x0 = v[2 * j], x1 = v[2 * j + 1];
        ph[j] = __byte_perm(__float_as_uint(x0), __float_as_uint(x1), 0x7632);
        const float r0 = x0 - __uint_as_float(__float_as_uint(x0) & 0xffff0000u);
        const float r1 = x1 - __uint_as_float(__float_as_uint(x1) & 0xffff0000u);
        pm[j] = __byte_perm(__float_as_uint(r0), __float_as_uint(r1), 0x7632);
        const float q0 = r0 - __uint_as_float(__float_as_uint(r0) & 0xffff0000u);
        const float q1 = r1 - __uint_as_float(__float_as_uint(r1) & 0xffff0000u);
        pl[j] = __byte_perm(__float_as_uint(q0), __float_as_uint(q1), 0x7632);  // <= 8 significant bits left: exact
    }
    const uint32_t off = sw64_off(row, chunk);
    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(parts_a + off), "r"(ph[0]), "r"(ph[1]), "r"(ph[2]), "r"(ph[3]) : "memory");
    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(parts_a + DN_PART_BYTES + off), "r"(pm[0]), "r"(pm[1]), "r"(pm[2]), "r"(pm[3]) : "memory");
    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(parts_a + 2 * DN_PART_BYTES + off), "r"(pl[0]), "r"(pl[1]), "r"(pl[2]), "r"(pl[3]) : "memory");
}

// shared-memory operand descriptors (cute::UMMA::SmemDescriptor): start >> 4 | LBO << 16 | SBO << 32 | version 1 << 46 | layout << 61
__device__ __forceinline__ uint64_t desc_sw64(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {  // layout 4 = SWIZZLE_64B
    return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) | (1ull << 46) | (4ull << 61);
}
// kind::f16 instruction descriptor: fp32 accumulate, bf16 x bf16, M = 128
__device__ __forceinline__ uint32_t idesc_bf16_m128(uint32_t n, uint32_t b_mn_major) {
    return (1u << 4) | (1u << 7) | (1u << 10) | (b_mn_major << 16) | ((n >> 3) << 17) | ((128u >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}

struct PrepDenseParams {
    int n_layers;
    LayerDev layers[MHO_MAX_LAYERS];
    int w_off[MHO_MAX_LAYERS];
    unsigned char* out;
};

__global__ void prepare_dense_weights_kernel(const __grid_constant__ PrepDenseParams p) {
    for (int l = blockIdx.y; l < p.n_layers; l += gridDim.y) {
        const LayerDev& L = p.layers[l];
        const int nblk = dn_nblk(L.K, L.f_out);
        const int n_rows = L.K * nblk;
        unsigned char* img = p.out + p.w_off[l];
        const int total = n_rows * 32;
        for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
            const int k = idx / (nblk * 32), rem = idx - k * nblk * 32;
            const int f = rem / nblk, o = rem - f * nblk;  // o fastest: coalesced reads of W[k][f][.]
            float w = 0.f;
            if (f < L.f_in && o < L.f_out) w = __ldg(L.W + ((size_t)k * L.f_in + f) * L.f_out + o);
            uint32_t h, m, lo;
            split3(w, h, m, lo);
            const uint32_t n = (uint32_t)(k * nblk + o);
            const uint32_t off = sw64_off(n, (uint32_t)f >> 3) + ((uint32_t)f & 7u) * 2u;
            *reinterpret_cast<uint16_t*>(img + off) = (uint16_t)(h >> 16);
            *reinterpret_cast<uint16_t*>(img + (size_t)n_rows * 64 + off) = (uint16_t)(m >> 16);
            *reinterpret_cast<uint16_t*>(img + (size_t)n_rows * 128 + off) = (uint16_t)(lo >> 16);
        }
        if (blockIdx.x == 0 && threadIdx.x < 32) {
            float* bias = reinterpret_cast<float*>(img + (size_t)n_rows * 192);
            bias[threadIdx.x] = (L.b != nullptr && (int)threadIdx.x < L.f_out) ? __ldg(L.b + threadIdx.x) : 0.f;
        }
    }
}

struct TileInfoD { int node0, rows, nz0, nnz; };
__device__ __forceinline__ TileInfoD load_tile(const BatchDev& b, int i) {
    const int4 v = __ldg(reinterpret_cast<const int4*>(b.tile_info) + i);
    return TileInfoD{v.x, v.y, v.z, v.w};
}

// operator of one tile -> staging: the precomputed bit rows (16 B per node) when the batch carries them, else the CSR slice
__device__ __forceinline__ void issue_csr_loads(const DenseParams& p, const TileInfoD& t, uint32_t rp_a, uint32_t ci_a, int tid) {
    if (!p.need_adj) return;  // every layer has K = 1: the operator is never touched
    if (p.b.adj_bits != nullptr) {
        if (tid < t.rows) cp_async16(rp_a + tid * 16, p.b.adj_bits + (size_t)(t.node0 + tid) * 4);
        return;
    }
    for (int i = tid; i <= t.rows; i += DN_THREADS) cp_async4(rp_a + i * 4, p.b.rowptr + t.node0 + i);
    for (int e = tid; e < t.nnz; e += DN_THREADS) cp_async4(ci_a + e * 4, p.b.colidx + t.nz0 + e);
}

// A operand straight from tensor memory (".ts" form): lane = row, 32-bit column = two consecutive bf16 of K
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_st_32x32b_x16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
                 "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
                 "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
                 : "memory");
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void tmem_st_32x32b_x8(uint32_t taddr, const uint32_t (&r)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]),
                 "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_32x32b_x8_nowait(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
}

__device__ __forceinline__ void load_x_rows(const DenseParams& p, const TileInfoD& t, uint32_t r, int c0, float (&x)[8]) {
    const int fi0 = p.layers[0].f_in;
#pragma unroll
    for (int j = 0; j < 8; ++j) x[j] = 0.f;
    if ((int)r < t.rows) {
        const float* src = p.X + (size_t)(t.node0 + (int)r) * fi0 + c0;
        if ((fi0 & 3) == 0 && c0 + 8 <= fi0 && (reinterpret_cast<uintptr_t>(p.X) & 15u) == 0) {
            const float4 a = __ldg(reinterpret_cast<const float4*>(src)), b = __ldg(reinterpret_cast<const float4*>(src) + 1);
            x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (c0 + j < fi0) x[j] = __ldg(src + j);
        }
    }
}

// input rows of one tile -> the 16 KB staging tile ([row][32 fp32], 16 B chunks XOR-swizzled with row & 7), coalesced:
// eight neighbouring lanes fetch one row.  Needs f_in % 4 == 0 (16 B chunks); chunks past f_in are never read.
__device__ __forceinline__ void issue_x_loads(const DenseParams& p, const TileInfoD& t, uint32_t xs_a, int tid) {
    const int fi0 = p.layers[0].f_in;
    const int cpr = fi0 >> 2;  // 16 B chunks per row
    const float* src = p.X + (size_t)t.node0 * fi0;
    for (int i = tid; i < t.rows * 8; i += DN_THREADS) {
        const uint32_t row = (uint32_t)i >> 3, ch = (uint32_t)i & 7u;
        if ((int)ch < cpr) cp_async16(xs_a + (row << 7) + ((ch ^ (row & 7u)) << 4), src + (size_t)row * fi0 + ch * 4);
    }
}
__device__ __forceinline__ void read_x_staged(const DenseParams& p, uint32_t xs_a, uint32_t r, int cb, bool live, float (&x)[8]) {
    const int cpr = p.layers[0].f_in >> 2;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const uint32_t ch = (uint32_t)(2 * cb + h);
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (live && (int)ch < cpr) v = lds_f128(xs_a + (r << 7) + ((ch ^ (r & 7u)) << 4));
        x[4 * h] = v.x; x[4 * h + 1] = v.y; x[4 * h + 2] = v.z; x[4 * h + 3] = v.w;
    }
}

__global__ void __launch_bounds__(DN_THREADS, 2) cheb_dense_kernel(const __grid_constant__ DenseParams p) {
    extern __shared__ __align__(1024) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    // ---- shared memory carve-up
    unsigned char* parts_s = smem;
    unsigned char* w_s = parts_s + 3 * DN_PART_BYTES;
    int* csr0 = reinterpret_cast<int*>(w_s + p.w_bytes);
    const int rp_words = (128 + 2 + 3) & ~3;
    const int csr_words = p.stage_words;
    int* s_idx = csr0 + 2 * csr_words;   // [2..3] mbarrier, [4] TMEM base, [8] index and [12..15] bounds of the tile after next
    const uint32_t parts_a = smem_u32(parts_s), w_a = smem_u32(w_s), csr_a0 = smem_u32(csr0);
    const uint32_t mbar = smem_u32(s_idx + 2), tslot = smem_u32(s_idx + 4);
    uint2* lut_s = reinterpret_cast<uint2*>(s_idx + 16);                  // 4 adjacency bits -> two bf16 pairs
    unsigned int* mask_s = reinterpret_cast<unsigned int*>(s_idx + 48);   // [128 rows][4] adjacency bits of the tile
    const uint32_t xs_a = smem_u32(s_idx + 48 + 512 + 208);               // 16 KB input staging tile
    const bool x_staged = (p.layers[0].f_in & 3) == 0 && (reinterpret_cast<uintptr_t>(p.X) & 15u) == 0;  // 16 B cp.async chunks
    if (tid < 16)
        lut_s[tid] = make_uint2(((tid & 1) ? 0x3F80u : 0u) | ((tid & 2) ? 0x3F800000u : 0u), ((tid & 4) ? 0x3F80u : 0u) | ((tid & 8) ? 0x3F800000u : 0u));

    // thread <-> accumulator element: TMEM lane = tile row; warp w may touch lane quadrant (w & 3); column block w >> 2
    const int q = warp & 3, cb = warp >> 2;
    const uint32_t r = (uint32_t)(q * 32 + lane);
    const int c0 = cb * 8;

    if (warp == 0) tmem_alloc(tslot, (uint32_t)p.tmem_cols);
    if (tid == 0) mbar_init(mbar, 1);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(s_idx + 4);
    const uint32_t tmem_row = tmem_base + ((uint32_t)(q * 32) << 16);
    const uint32_t adj_col = (uint32_t)(p.tmem_cols - 64);  // the tile's adjacency: 128 lanes x 64 columns (bf16 pairs)
    uint32_t mma_phase = 0;

    // from here on global memory written by earlier launches in the stream is read
    asm volatile("griddepcontrol.wait;" ::: "memory");
    {   // resident: every layer's images; streaming: the first layer's into slot 0
        const int nb = p.w_resident ? p.w_bytes : p.w_lbytes[0];
        for (int c = tid; c < nb / 16; c += DN_THREADS) cp_async16(w_a + (uint32_t)c * 16u, p.wimg + (size_t)c * 16);
    }
    int wslot = 0;  // streaming mode: the slot holding the current layer's images

    // ---- tile scheduler (dynamic from the third tile of a CTA on; the last CTA out re-arms the counters)
    // the first two tiles of every CTA are static (no round trip to the counter before work starts); the counter
    // hands out tiles 2 * gridDim.x onwards
    const int i_cur = (int)blockIdx.x, i_nxt = (int)(blockIdx.x + gridDim.x);
    auto finish = [&]() {
        cp_async_wait<0>();
        tc_fence_before();
        __syncthreads();
        if (warp == 0) tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
        if (tid == 0) {
            __threadfence();
            if (atomicAdd(p.sched + 1, 1) == (int)gridDim.x - 1) { p.sched[0] = 0; p.sched[1] = 0; }
        }
    };
    if (i_cur >= p.b.n_tiles) { finish(); return; }
    TileInfoD cur = load_tile(p.b, i_cur);
    bool has_nxt = i_nxt < p.b.n_tiles;
    TileInfoD nxt = cur;
    if (has_nxt) nxt = load_tile(p.b, i_nxt);
    issue_csr_loads(p, cur, csr_a0, csr_a0 + rp_words * 4, tid);
    if (x_staged) issue_x_loads(p, cur, xs_a, tid);
    cp_async_commit();
    int cs = 0;
    cp_async_wait<0>();  // the first tile's operator slice and input rows, and the weights, have landed
    __syncthreads();

#ifdef MHO_PROBE
    long long pt[48]; int pid[48]; int pn = 0;
#endif
    for (int it = 0;; ++it) {
        PROBE(0);
        const int* rp_s = csr0 + cs * csr_words;
        const int* ci_s = rp_s + rp_words;
        const int rows = cur.rows, node0 = cur.node0, nz0 = cur.nz0;
        const bool live = (int)r < rows;

        // the scheduler's last thread fetches the index (and bounds) of tile it+2 in the background
        int i_nn = p.b.n_tiles;
        if (tid == DN_THREADS - 1 && has_nxt) i_nn = 2 * (int)gridDim.x + atomicAdd(p.sched, 1);
        PROBE(1);
        {
            float xin[8];
            if (x_staged) read_x_staged(p, xs_a, r, cb, live, xin);
            else load_x_rows(p, cur, r, c0, xin);
            store_parts(parts_a, r, (uint32_t)cb, xin);
        }
        PROBE(2);

        PROBE(3);

        for (int li = 0; li < p.n_layers; ++li) {
            const LayerDev& L = p.layers[li];
            const int K = L.K;
            const int nblk = dn_nblk(K, L.f_out);
            const int n_rows = K * nblk;
            const int w_pos = p.w_resident ? p.w_off[li] : wslot * p.w_slot;
            const uint32_t w_l = w_a + (uint32_t)w_pos;
            const float* bias_s = reinterpret_cast<const float*>(w_s + w_pos + (size_t)n_rows * 192);
            if (!p.w_resident) cp_async_wait<0>();  // this layer's images (issued one layer ago) have landed

            PROBE(4);
            // ---- P = X_l [W_0 | ... | W_K-1]: six part products, two 16-wide K steps each
            fence_proxy_async();  // part tiles / cp.async-written weights -> tensor-core proxy
            tc_fence_before();
            __syncthreads();
            if (tid == 0) {
                tc_fence_after();
                const uint32_t idesc = idesc_bf16_m128((uint32_t)n_rows, 0u);
                const uint64_t a0 = desc_sw64(parts_a, 16, 512);
                const uint64_t b0 = desc_sw64(w_l, 16, 512);
                const uint64_t a_step = (uint64_t)(DN_PART_BYTES >> 4), b_step = (uint64_t)((n_rows * 64) >> 4);
                // smallest terms first: (m,m) (h,l) (l,h) (h,m) (m,h) (h,h)
                const int pa[6] = {1, 0, 2, 0, 1, 0}, pb[6] = {1, 2, 0, 1, 0, 0};
                uint32_t accum = 0u;
#pragma unroll
                for (int t = 0; t < 6; ++t) {
#pragma unroll
                    for (int ks = 0; ks < 2; ++ks) {
                        umma_bf16(tmem_base, a0 + a_step * pa[t] + 2 * ks, b0 + b_step * pb[t] + 2 * ks, idesc, accum);
                        accum = 1u;
                    }
                }
                umma_commit(mbar);
            }
            PROBE(5);
            // the tile's adjacency goes to tensor memory while the first layer's X W group runs (it is first read by the
            // first Clenshaw step, behind that step's fence + barrier)
            if (li == 0 && p.need_adj) {
                    // CSR -> 128 x 128 adjacency bits (four lanes per row), then every thread expands the 32 bits of its (row, 32-column block) to 16 bf16 pairs in tensor memory
                    // (every UMMA that read the previous tile's adjacency has completed: its epilogue waited for them)
                    if (p.b.adj_bits == nullptr) {
                        // four neighbouring lanes share a row: entries dealt round-robin, bits gathered in registers, OR-reduced
                        // across the four lanes with shuffles, lane s publishes word s
                        const int row = tid >> 2;
                        uint32_t m0 = 0u, m1 = 0u, m2 = 0u, m3 = 0u;
                        if (row < rows) {
                            const int e1 = rp_s[row + 1] - nz0;
#pragma unroll 2
                            for (int e = rp_s[row] - nz0 + (tid & 3); e < e1; e += 4) {
                                const uint32_t c = (uint32_t)(ci_s[e] - node0);
                                const uint32_t bit = 1u << (c & 31u), w = c >> 5;
                                m0 |= (w == 0u) ? bit : 0u;
                                m1 |= (w == 1u) ? bit : 0u;
                                m2 |= (w == 2u) ? bit : 0u;
                                m3 |= (w == 3u) ? bit : 0u;
                            }
                        }
#pragma unroll
                        for (int d = 1; d < 4; d <<= 1) {
                            m0 |= __shfl_xor_sync(0xffffffffu, m0, d);
                            m1 |= __shfl_xor_sync(0xffffffffu, m1, d);
                            m2 |= __shfl_xor_sync(0xffffffffu, m2, d);
                            m3 |= __shfl_xor_sync(0xffffffffu, m3, d);
                        }
                        const int sub = tid & 3;
                        mask_s[tid] = sub == 0 ? m0 : (sub == 1 ? m1 : (sub == 2 ? m2 : m3));  // word (row, sub); rows past the tile: 0
                    }
                    PROBE(30);
                    if (p.b.adj_bits == nullptr) __syncthreads();
                    PROBE(31);
                    const uint32_t mask = p.b.adj_bits != nullptr ? (live ? (uint32_t)rp_s[r * 4 + cb] : 0u) : mask_s[r * 4 + cb];
                    uint32_t aw[16];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const uint2 w = lut_s[(mask >> (4 * j)) & 15u];
                        aw[2 * j] = w.x; aw[2 * j + 1] = w.y;
                    }
                    PROBE(32);
                    tmem_st_32x32b_x16(tmem_row + adj_col + (uint32_t)(cb * 16), aw);
                }
            if (!p.w_resident) {
                // the next layer's images (the first layer's, for the next tile, after the last) go to the other slot: its
                // last readers were the previous layer's UMMAs and epilogue, complete before this layer's barrier
                const int ln = (li + 1 == p.n_layers) ? 0 : li + 1;
                if (ln != 0 || has_nxt) {
                    const uint32_t dst = w_a + (uint32_t)((wslot ^ 1) * p.w_slot);
                    const unsigned char* src = p.wimg + p.w_off[ln];
                    for (int c = tid; c < p.w_lbytes[ln] / 16; c += DN_THREADS) cp_async16(dst + (uint32_t)c * 16u, src + (size_t)c * 16);
                }
                cp_async_commit();
                wslot ^= 1;
            }
            // the next tile's operator slice and input rows stream in behind the first layer's UMMAs (every thread
            // has read the input staging tile: the barrier above)
            if (li == 0) {
                if (has_nxt) {
                    const uint32_t rp_n = csr_a0 + (uint32_t)((cs ^ 1) * csr_words) * 4u;
                    issue_csr_loads(p, nxt, rp_n, rp_n + rp_words * 4, tid);
                    if (x_staged) issue_x_loads(p, nxt, xs_a, tid);
                }
                cp_async_commit();
            }
            mbar_wait(mbar, mma_phase);
            mma_phase ^= 1u;
            tc_fence_after();
            PROBE(6);

            float b1[8], b2[8];
            uint32_t v[8];
            tmem_ld_32x32b_x8(tmem_row + (uint32_t)((K - 1) * nblk + c0), v);
#pragma unroll
            for (int j = 0; j < 8; ++j) { b1[j] = __uint_as_float(v[j]); b2[j] = 0.f; }
            if (c0 >= nblk) {
#pragma unroll
                for (int j = 0; j < 8; ++j) b1[j] = 0.f;
            }

            // ---- Clenshaw steps: D_k (+)= A (2 B_k+1)  [k >= 1],  D_0 (+)= A B_1.  One UMMA per 16 nodes covers the three
            // parts at once (N = 96: the part tiles are three N-atoms, LBO apart): columns [32k, 32k+32) (+)= A h, the two
            // blocks behind them - P_k+1 / P_k+2, consumed already and zeroed as soon as they were read - receive A m, A l.
            const uint32_t zero8[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
            if (K > 1) {
                tmem_st_32x32b_x8(tmem_row + (uint32_t)((K - 1) * 32 + c0), zero8);
                tmem_st_32x32b_x8(tmem_row + (uint32_t)(K * 32 + c0), zero8);
            }
            for (int k = K - 2; k >= 0; --k) {
                float s[8];
                const float f = k > 0 ? 2.f : 1.f;
#pragma unroll
                for (int j = 0; j < 8; ++j) s[j] = f * b1[j];
                PROBE(10);
                store_parts(parts_a, r, (uint32_t)cb, s);
                tmem_wait_st();
                fence_proxy_async();
                tc_fence_before();
                PROBE(11);
                __syncthreads();
                PROBE(12);
                if (tid == 0) {
                    tc_fence_after();
                    const uint32_t idesc = idesc_bf16_m128(96u, 1u);
                    const uint64_t b0 = desc_sw64(parts_a, DN_PART_BYTES, 512);   // MN-major: 8 node rows per 512 B group, N-atoms one part apart
                    const uint32_t d = tmem_base + (uint32_t)(k * 32);
                    const uint32_t a0 = tmem_base + adj_col;
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks) umma_bf16_ts(d, a0 + (uint32_t)(ks * 8), b0 + (uint64_t)((ks * 1024) >> 4), idesc, 1u);
                    umma_commit(mbar);
                }
                PROBE(13);
                mbar_wait(mbar, mma_phase);
                mma_phase ^= 1u;
                tc_fence_after();
                PROBE(14);
                uint32_t v1[8], v2[8];
                tmem_ld_32x32b_x8_nowait(tmem_row + (uint32_t)(k * 32 + c0), v);
                tmem_ld_32x32b_x8_nowait(tmem_row + (uint32_t)((k + 1) * 32 + c0), v1);
                tmem_ld_32x32b_x8_nowait(tmem_row + (uint32_t)((k + 2) * 32 + c0), v2);
                tmem_wait_ld();
                if (k > 0) {  // blocks k and k+1 are the next step's scratch: clear them while the recurrence computes
                    tmem_st_32x32b_x8(tmem_row + (uint32_t)(k * 32 + c0), zero8);
                    tmem_st_32x32b_x8(tmem_row + (uint32_t)((k + 1) * 32 + c0), zero8);
                }
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float bk = (__uint_as_float(v[j]) + (__uint_as_float(v1[j]) + __uint_as_float(v2[j]))) - b2[j];
                    b2[j] = b1[j];
                    b1[j] = bk;
                }
            }
            PROBE(15);

            // ---- epilogue: bias + activation; last layer -> Y, hidden layer -> part tiles of the next layer (+ saved)
            const bool last = (li == p.n_layers - 1);
            const int fo = L.f_out;
            float y[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) y[j] = b1[j] + bias_s[(c0 + j) & 31];
            if (L.act == MHO_ACT_RELU) {
#pragma unroll
                for (int j = 0; j < 8; ++j) y[j] = fmaxf(y[j], 0.f);
            } else if (L.act == MHO_ACT_LEAKY) {
                const float sl = L.slope;
#pragma unroll
                for (int j = 0; j < 8; ++j) y[j] = y[j] > 0.f ? y[j] : sl * y[j];
            }
            if (!live || c0 + 8 > fo) {
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    if (!live || c0 + j >= fo) y[j] = 0.f;
            }
            PROBE(16);
            float* gout = last ? p.Y : (p.saved ? p.saved + p.layers[li + 1].saved_off : nullptr);
            const bool out16 = gout != nullptr && (reinterpret_cast<uintptr_t>(gout) & 15u) == 0;  // `saved` blocks start at odd offsets
            if (last && fo == 32 && out16) {
                // through shared memory (the part tiles are free: every UMMA has completed) so that a warp writes four
                // whole 128 B rows per instruction instead of 32 row fragments
                sts_f128(parts_a + (r << 7) + (((uint32_t)(2 * cb) ^ (r & 7u)) << 4), make_float4(y[0], y[1], y[2], y[3]));
                sts_f128(parts_a + (r << 7) + (((uint32_t)(2 * cb + 1) ^ (r & 7u)) << 4), make_float4(y[4], y[5], y[6], y[7]));
                __syncthreads();
                float* dst = gout + (size_t)node0 * 32;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const uint32_t row = (uint32_t)(tid >> 3) + 64u * h, ch = (uint32_t)tid & 7u;
                    if ((int)row < rows)
                        *reinterpret_cast<float4*>(dst + (size_t)row * 32 + ch * 4) = lds_f128(parts_a + (row << 7) + ((ch ^ (row & 7u)) << 4));
                }
            } else if (gout != nullptr && live && c0 < fo) {
                float* dst = gout + (size_t)(node0 + (int)r) * fo + c0;
                if (out16 && (fo & 3) == 0 && c0 + 8 <= fo) {
                    *reinterpret_cast<float4*>(dst) = make_float4(y[0], y[1], y[2], y[3]);
                    *reinterpret_cast<float4*>(dst + 4) = make_float4(y[4], y[5], y[6], y[7]);
                } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        if (c0 + j < fo) dst[j] = y[j];
                }
            }
            if (!last) store_parts(parts_a, r, (uint32_t)cb, y);
            PROBE(20);
        }
#ifdef MHO_PROBE
        if (blockIdx.x == 0 && it == MHO_PROBE_IT && (tid == 0 || tid == 479)) {
            for (int i = 1; i < pn; ++i) printf("t%d id %d +%lld (abs %lld)\n", tid, pid[i], pt[i] - pt[i - 1], pt[i] - pt[0]);
        }
#endif

        if (!has_nxt) break;
        if (tid == DN_THREADS - 1) {
            s_idx[8] = i_nn;
            if (i_nn < p.b.n_tiles) *reinterpret_cast<int4*>(s_idx + 12) = __ldg(reinterpret_cast<const int4*>(p.b.tile_info) + i_nn);
        }
        cp_async_wait<0>();  // the next tile's operator slice and input rows have landed (issued a whole tile ago)
        tc_fence_before();
        __syncthreads();  // ... and every TMEM read of this tile is done before the next tile's UMMAs overwrite the columns
        cs ^= 1;
        cur = nxt;
        has_nxt = s_idx[8] < p.b.n_tiles;
        if (has_nxt) { const int4 v4 = *reinterpret_cast<const int4*>(s_idx + 12); nxt = TileInfoD{v4.x, v4.y, v4.z, v4.w}; }
    }
    finish();
}

}  // namespace

// -------------------------------------------------------------------------------------------
// host side
// -------------------------------------------------------------------------------------------
bool cheb_dense_eligible(const mho_layer_t* layers, int n_layers, bool has_vals, bool has_bits, int max_tile_rows, int max_tile_nnz,
                         int max_smem_optin) {
    if (max_tile_rows > 128) return false;
    int wb = 0;
    bool need_adj = false;
    for (int l = 0; l < n_layers; ++l) {
        if (layers[l].f_in > 32 || layers[l].f_out > 32 || layers[l].K < 1) return false;
        if (dn_layer_rows(layers[l].K, layers[l].f_out) + (layers[l].K > 1 ? 96 : 0) > 256) return false;  // TMEM: P + a spare block + adjacency
        wb += dn_layer_bytes(layers[l].K, layers[l].f_out);
        need_adj |= layers[l].K > 1;
    }
    if (has_vals && need_adj) return false;  // weighted operators go through the CSR-walk kernel (K = 1 stacks never read them)
    int wmax = 0;
    for (int l = 0; l < n_layers; ++l) wmax = std::max(wmax, dn_layer_bytes(layers[l].K, layers[l].f_out));
    const size_t stage = !need_adj ? 16 : (has_bits ? 512 : (size_t)132 + ((max_tile_nnz + 3) & ~3));   // words per operator staging set
    const size_t rest = (size_t)3 * DN_PART_BYTES + 2 * stage * 4 + 192 + 2048 + 832 + 16384;
    const size_t budget = std::min((size_t)(228 * 1024) / 2 - 1024, (size_t)max_smem_optin);
    // all layers' weight images resident, or (multi-layer stacks with K > 1) two slots the layers stream through
    return rest + wb <= budget || (n_layers > 1 && rest + 2 * (size_t)wmax <= budget);
}

int cheb_dense_weight_bytes(const mho_layer_t* layers, int n_layers, int* w_off) {
    int wb = 0;
    for (int l = 0; l < n_layers; ++l) { w_off[l] = wb; wb += dn_layer_bytes(layers[l].K, layers[l].f_out); }
    return wb;
}

cudaError_t prepare_dense_weights_launch(const LayerDev* layers, int n_layers, const int* w_off, unsigned char* out, cudaStream_t st) {
    PrepDenseParams p;
    p.n_layers = n_layers;
    for (int l = 0; l < n_layers; ++l) { p.layers[l] = layers[l]; p.w_off[l] = w_off[l]; }
    p.out = out;
    // the kernel writes the weight parts and bias rows, not the padding of each layer's block
    const int bytes = w_off[n_layers - 1] + dn_layer_bytes(layers[n_layers - 1].K, layers[n_layers - 1].f_out);
    const cudaError_t e = cudaMemsetAsync(out, 0, (size_t)bytes, st);
    if (e != cudaSuccess) return e;
    dim3 grid(8, n_layers);
    prepare_dense_weights_kernel<<<grid, 256, 0, st>>>(p);
    return cudaGetLastError();
}

cudaError_t cheb_dense_launch(const FwdParams& fp, const unsigned char* wimg, const int* w_off, int w_bytes, int max_tile_nnz,
                              int num_sms, cudaStream_t st) {
    DenseParams p;
    memset(&p, 0, sizeof(p));
    p.b = fp.b;
    p.n_layers = fp.n_layers;
    int cols = 32;
    for (int l = 0; l < fp.n_layers; ++l) {
        p.layers[l] = fp.layers[l];
        p.w_off[l] = w_off[l];
        p.need_adj |= fp.layers[l].K > 1 ? 1 : 0;
    }
    for (int l = 0; l < fp.n_layers; ++l) {
        const int n = dn_layer_rows(fp.layers[l].K, fp.layers[l].f_out) + (p.need_adj ? 96 : 0);
        while (cols < n) cols <<= 1;
    }
    p.X = fp.X; p.Y = fp.Y; p.saved = fp.saved;
    p.wimg = wimg;
    int wmax = 0;
    for (int l = 0; l < fp.n_layers; ++l) {
        p.w_lbytes[l] = (l + 1 < fp.n_layers ? w_off[l + 1] : w_bytes) - w_off[l];
        wmax = std::max(wmax, p.w_lbytes[l]);
    }
    p.nnz_cap = (max_tile_nnz + 3) & ~3;
    p.stage_words = !p.need_adj ? 16 : (p.b.adj_bits != nullptr ? 512 : 132 + p.nnz_cap);
    p.tmem_cols = cols;
    p.sched = fp.sched;
    const size_t rest = (size_t)3 * DN_PART_BYTES + (size_t)2 * p.stage_words * 4 + 192 + 2048 + 832 + 16384;
    p.w_resident = (fp.n_layers == 1 || rest + (size_t)w_bytes <= (size_t)(228 * 1024) / 2 - 1024) ? 1 : 0;
    p.w_slot = wmax;
    p.w_bytes = p.w_resident ? w_bytes : 2 * wmax;
    const size_t smem = rest + (size_t)p.w_bytes;
    int grid = num_sms * 2;
    if (grid > p.b.n_tiles) grid = p.b.n_tiles;
    if (grid < 1) grid = 1;
    return mho_launch<cheb_dense_kernel>(dim3((unsigned)grid), dim3(DN_THREADS), smem, st, true, p);
}
