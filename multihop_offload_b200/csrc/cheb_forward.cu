// Batched ChebConv forward (single layer or fused L-layer stack) for sm_100a.
//
// Replaces, for a whole batch of graph instances, the reference's eager per-graph call
//   ACOAgent.predict -> self.model([x_in, a_in])        (src/gnn_offloading_agent.py:144-150)
// of the Keras model built at :81-123 out of spektral.layers.ChebConv:
//   Y = act( sum_k T_k W[k] + b ),  T_0 = X, T_1 = A X, T_k = 2 A T_{k-1} - T_{k-2}.
//
// Design (see DESIGN.md "forward kernel"):
//   * persistent CTAs walk "tiles" = runs of consecutive graphs (block-diagonal operator => a run
//     of graphs is just a bigger graph) of at most rows_cap nodes; the next tile's X rows and CSR
//     slice are fetched with cp.async into a third tile buffer while the current tile computes;
//   * the CSR slice is turned in place into a stream of pre-swizzled shared-memory row offsets
//     whose low bits flag "last entry of its row" - each warp then walks a contiguous, nnz-balanced
//     chunk of that stream 4 entries per LDS.128, one lane per feature: every neighbour gather is a
//     single conflict-free 128 B wavefront and four of them are in flight per warp;
//   * the Chebyshev recurrence runs on-chip on two swizzled [rows][32] fp32 tiles (T_k overwrites
//     T_{k-2} in place);
//   * the dense contraction [T_0|..|T_{K-1}] . W runs on the tensor cores (mma.sync m16n8k8 TF32,
//     3xTF32 split in registers for fp32-grade accuracy) straight out of the same tiles via
//     ldmatrix, interleaved with the sparse step for T_{k+1};
//   * HBM traffic per tile is exactly X in, Y out, CSR once; T_k never leaves the SM.
#include "mho_common.cuh"

// the forward kernel runs 16 warps per CTA: two CTAs per SM then give 32 resident warps, which this
// latency-bound kernel needs; the dense part maps warp w -> m-tile slot (w & 7), n-tile half (w >> 3)
#define FWD_THREADS 512
#define FWD_NWARPS (FWD_THREADS / 32)
#define FWD_MSLOTS (FWD_NWARPS / 2)

struct TileInfo {
    int node0, rows, nz0, nnz;
};

__device__ __forceinline__ TileInfo load_tile_info(const BatchDev& b, int tile) {
    TileInfo t;
    if (b.tile_info != nullptr) {  // one 16 B load instead of three dependent ones
        const int4 v = __ldg(reinterpret_cast<const int4*>(b.tile_info) + tile);
        t.node0 = v.x; t.rows = v.y; t.nz0 = v.z; t.nnz = v.w;
        return t;
    }
    const int g0 = b.tile_off ? __ldg(b.tile_off + tile) : tile;
    const int g1 = b.tile_off ? __ldg(b.tile_off + tile + 1) : tile + 1;
    t.node0 = __ldg(b.graph_off + g0);
    const int node1 = __ldg(b.graph_off + g1);
    t.rows = node1 - t.node0;
    t.nz0 = __ldg(b.rowptr + t.node0);
    t.nnz = __ldg(b.rowptr + node1) - t.nz0;
    return t;
}

// -------------------------------------------------------------------------------------------
// Weight preparation (one tiny launch whenever the weights changed): Keras layout W[k][f][o] ->
// per layer a block of 128 B rows  [hi image: K*fo_img rows][lo image: K*fo_img rows][bias: 8 rows],
// fo_img = pad16(f_out) (the UMMA N extent), every image 1024 B aligned so that it is at once an
// ldmatrix source and a tcgen05 SWIZZLE_128B K-major B operand;
// image row (k*fo_img + o) holds W[k][.][o] over f (transposed, 128B-swizzled on o) split into
// TF32 hi / lo parts (cvt.rna), so that a CTA stages it with straight 16 B cp.async copies and
// ldmatrix yields ready-to-use mma B fragments.
// -------------------------------------------------------------------------------------------
struct PrepParams {
    int n_layers;
    LayerDev layers[MHO_MAX_LAYERS];
    int row_off[MHO_MAX_LAYERS];
    unsigned char* out;
};

__global__ void prepare_weights_kernel(const __grid_constant__ PrepParams p) {
    for (int l = blockIdx.y; l < p.n_layers; l += gridDim.y) {
        const LayerDev& L = p.layers[l];
        const int fo_pad = pad16(L.f_out);
        const int n_rows = L.K * fo_pad;
        unsigned char* hi_img = p.out + (size_t)p.row_off[l] * 128;
        unsigned char* lo_img = hi_img + (size_t)n_rows * 128;
        float* bias = reinterpret_cast<float*>(lo_img + (size_t)n_rows * 128);
        const int total = n_rows * 32;
        for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
            // o fastest: coalesced reads of W[k][f][.]
            const int k = idx / (fo_pad * 32), rem = idx - k * fo_pad * 32;
            const int f = rem / fo_pad, o = rem - f * fo_pad;
            float w = 0.f;
            if (f < L.f_in && o < L.f_out) w = __ldg(L.W + ((size_t)k * L.f_in + f) * L.f_out + o);
            uint32_t hi, lo;
            split_tf32(w, hi, lo);
            const uint32_t off = (uint32_t)(k * fo_pad) * 128u + swz_off((uint32_t)o, (uint32_t)f);
            *reinterpret_cast<uint32_t*>(hi_img + off) = hi;
            *reinterpret_cast<uint32_t*>(lo_img + off) = lo;
        }
        if (blockIdx.x == 0 && threadIdx.x < 32)
            bias[threadIdx.x] = (L.b != nullptr && (int)threadIdx.x < L.f_out) ? __ldg(L.b + threadIdx.x) : 0.f;
    }
}

int wprep_layer_rows(int K, int f_out) { return 2 * K * pad16(f_out) + 8; }

cudaError_t prepare_weights_launch(const LayerDev* layers, int n_layers, const int* row_off, unsigned char* out,
                                   cudaStream_t st) {
    PrepParams p;
    p.n_layers = n_layers;
    for (int l = 0; l < n_layers; ++l) { p.layers[l] = layers[l]; p.row_off[l] = row_off[l]; }
    p.out = out;
    dim3 grid(8, n_layers);
    prepare_weights_kernel<<<grid, 256, 0, st>>>(p);
    return cudaGetLastError();
}

// copy one layer's prepared block (hi, lo, bias) into shared memory with 16 B cp.async
__device__ __forceinline__ void stage_weights_async(const FwdParams& p, int l, uint32_t dst, int tid) {
    const int rows = 2 * p.layers[l].K * pad16(p.layers[l].f_out) + 8;
    const unsigned char* src = p.wprep + (size_t)p.wprep_row_off[l] * 128;
    for (int c = tid; c < rows * 8; c += FWD_THREADS) cp_async16(dst + (uint32_t)c * 16u, src + (size_t)c * 16);
}

// -------------------------------------------------------------------------------------------
// acc[nt][4] += T[row0..row0+15][0..fi_pad) . W_k   (3xTF32: lo*hi + hi*lo + hi*hi, fp32 accumulate)
// A is split in registers (5 integer/float ops per element), W comes pre-split from the images.
// -------------------------------------------------------------------------------------------
__device__ __forceinline__ void mma_tile(float (&acc)[2][4], uint32_t T_addr, int row0, uint32_t whi_k, uint32_t wlo_k,
                                         int nchunks, int nt0, int nnt, int lane) {
    const uint32_t arow = (uint32_t)row0 + (lane & 7) + ((lane >> 3) & 1) * 8;
    const uint32_t a_base = T_addr + (arow << 7);
    const uint32_t a_key = arow & 7u;
    const uint32_t a_sel = (uint32_t)(lane >> 4);        // 0: chunk 2c, 1: chunk 2c+1
    const uint32_t b_r = (uint32_t)(lane & 7);
    const uint32_t b_sel = (uint32_t)((lane >> 3) & 1);  // k half
    uint32_t o_nt = (uint32_t)nt0 + (uint32_t)(lane >> 4);  // which n-tile of this warp's pair
    if ((int)o_nt >= nnt) o_nt = (uint32_t)(nnt - 1);       // odd n-tile count: duplicate, result unused
    const uint32_t boff = ((o_nt * 8u + b_r) << 7);
    const bool two = (nt0 + 1 < nnt);
#pragma unroll 2
    for (int c = 0; c < nchunks; ++c) {
        uint32_t a[4], ah[4], al[4], bh[4], bl[4];
        ldmatrix_x4(a_base + ((((uint32_t)(2 * c) + a_sel) ^ a_key) << 4), a[0], a[1], a[2], a[3]);
        const uint32_t bch = ((((uint32_t)(2 * c) + b_sel) ^ b_r) << 4);  // (o & 7) == b_r
        ldmatrix_x4(whi_k + boff + bch, bh[0], bh[1], bh[2], bh[3]);
        ldmatrix_x4(wlo_k + boff + bch, bl[0], bl[1], bl[2], bl[3]);
#pragma unroll
        for (int i = 0; i < 4; ++i) split_tf32_fast(__uint_as_float(a[i]), ah[i], al[i]);
        mma_tf32(acc[0], al, bh[0], bh[1]);
        mma_tf32(acc[0], ah, bl[0], bl[1]);
        mma_tf32(acc[0], ah, bh[0], bh[1]);
        if (two) {
            mma_tf32(acc[1], al, bh[2], bh[3]);
            mma_tf32(acc[1], ah, bl[2], bl[3]);
            mma_tf32(acc[1], ah, bh[2], bh[3]);
        }
    }
}

// -------------------------------------------------------------------------------------------
// Sparse recurrence step, stream form, perfectly balanced.  The tile's entry stream is cut into
// 4*NWARPS equal SEGMENTS regardless of row boundaries; a warp is 4 groups of 8 lanes, each group
// walks one segment, one entry per step, each lane holding 4 features (one 16 B chunk): one LDS.128
// per lane = one full 128 B row per group = 4 neighbour gathers per warp instruction, each a
// conflict-free quarter-warp wavefront.
//   first step : Tdst[r] = sum_j A[r,j] Tsrc[j]
//   later steps: Tdst[r] = 2 sum_j A[r,j] Tsrc[j] - Tdst[r]      (T_{k+1} overwrites T_{k-1})
// Rows that straddle segments (hub rows!) are finished in spmm_fixup after a barrier: a group
// that starts mid-row keeps the partial sum of its first row ("head"), every group publishes the
// partial sum after its last row end ("leftover") in shared memory.
// stream word = swizzled smem row offset | bit0 (last entry of its row) | bit1 (next row(s) empty).
// rp_s holds the RAW global row pointers of the tile (subtract nz0).
// -------------------------------------------------------------------------------------------
struct SegInfo {
    int sb, n;      // first entry and entry count of this group's segment
    int r0;         // row containing entry sb
    int mid;        // segment starts in the middle of row r0
    int seg_len;    // nominal segment length L (entry e belongs to group e / L)
};

struct HeadState {
    float4 head;
    int head_row;
    int pending;    // 1: the head row's sum is still in `head` and must be completed by spmm_fixup
};

template <bool FIRST>
__device__ __forceinline__ void emit_row(uint32_t Tdst, int row, uint32_t ckey, const float4& acc) {
    const uint32_t d = Tdst + (swz_row((uint32_t)row) ^ ckey);
    if (FIRST) {
        sts_f128(d, acc);
    } else {
        const float4 q = lds_f128(d);
        sts_f128(d, make_float4(fmaf(2.f, acc.x, -q.x), fmaf(2.f, acc.y, -q.y), fmaf(2.f, acc.z, -q.z), fmaf(2.f, acc.w, -q.w)));
    }
}

// (returns the next non-empty row by value: a by-reference row would live in local memory)
template <bool FIRST>
__device__ __noinline__ int emit_empty_rows(uint32_t Tdst, int row, int rows, const int* rp_s, uint32_t ckey) {
    while (row < rows && rp_s[row + 1] == rp_s[row]) {
        emit_row<FIRST>(Tdst, row, ckey, make_float4(0.f, 0.f, 0.f, 0.f));
        ++row;
    }
    return row;
}

// one stream entry: gather, accumulate
template <bool HAS_VALS>
__device__ __forceinline__ void gather_acc(float4& acc, uint32_t Tsrc, uint32_t cur, float cv, uint32_t ckey) {
    const float4 t = lds_f128(Tsrc + ((cur & ~3u) ^ ckey));
    if (HAS_VALS) {
        acc.x = fmaf(cv, t.x, acc.x); acc.y = fmaf(cv, t.y, acc.y);
        acc.z = fmaf(cv, t.z, acc.z); acc.w = fmaf(cv, t.w, acc.w);
    } else {
        acc.x += t.x; acc.y += t.y; acc.z += t.z; acc.w += t.w;
    }
}

template <bool HAS_VALS, bool FIRST, bool WAIT_MMA>
__device__ __forceinline__ void spmm_seg_walk(uint32_t Tsrc, uint32_t Tdst, const SegInfo& sg, int rows,
                                              const int* rp_s, uint32_t pre_a, uint32_t val_a, uint32_t ckey,
                                              uint32_t left_a, bool is_group0, HeadState& hs, uint32_t mbar, uint32_t parity) {
    hs.pending = 0;
    hs.head_row = 0;
    hs.head = make_float4(0.f, 0.f, 0.f, 0.f);
    if (is_group0) {  // empty rows in front of the first stored entry belong to nobody's stream
        emit_empty_rows<FIRST>(Tdst, 0, rows, rp_s, ckey);
    }
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (sg.n > 0) {
        int row = sg.r0;
        uint32_t ea = pre_a + (uint32_t)sg.sb * 4u, va = val_a + (uint32_t)sg.sb * 4u;
        const uint32_t ea_end = ea + (uint32_t)sg.n * 4u;
        uint32_t pw = lds_u32(ea);
        float vv = HAS_VALS ? lds_f32(va) : 1.f;
        // the first row end seen by a segment that starts mid-row closes a row begun in an earlier segment:
        // its partial sum is parked (completed by spmm_fixup), peeled out of the steady-state loop
        if (sg.mid) {
            for (;;) {
                const uint32_t cur = pw;
                const float cv = vv;
                ea += 4; va += 4;
                if (ea < ea_end) { pw = lds_u32(ea); if (HAS_VALS) vv = lds_f32(va); }
                gather_acc<HAS_VALS>(acc, Tsrc, cur, cv, ckey);
                if (cur & 1u) {
                    hs.head = acc; hs.head_row = row; hs.pending = 1;
                    acc = make_float4(0.f, 0.f, 0.f, 0.f);
                    ++row;
                    if (cur & 2u) row = emit_empty_rows<FIRST>(Tdst, row, rows, rp_s, ckey);
                    break;
                }
                if (ea >= ea_end) break;
            }
        }
        while (ea < ea_end) {
            const uint32_t cur = pw;
            const float cv = vv;
            ea += 4; va += 4;
            if (ea < ea_end) {  // next step's stream word is in flight during the gather
                pw = lds_u32(ea);
                if (HAS_VALS) vv = lds_f32(va);
            }
            gather_acc<HAS_VALS>(acc, Tsrc, cur, cv, ckey);
            if (cur & 1u) {
                emit_row<FIRST>(Tdst, row, ckey, acc);
                acc = make_float4(0.f, 0.f, 0.f, 0.f);
                ++row;
                if (cur & 2u) row = emit_empty_rows<FIRST>(Tdst, row, rows, rp_s, ckey);
            }
        }
    }
    if (WAIT_MMA) mbar_wait(mbar, parity);  // the slot aliases a tcgen05 operand tile: the step's MMAs must be done
    sts_f128(left_a, acc);  // partial sum of the row still open at the end of the segment (0 if none)
}

// after a barrier: complete the rows that straddled segment boundaries (deterministic order)
template <bool FIRST>
__device__ __forceinline__ void spmm_fixup(uint32_t Tdst, const SegInfo& sg, int group, const int* rp_s, int nz0,
                                           uint32_t ckey, uint32_t left_base, const HeadState& hs) {
    if (hs.pending) {
        const int e_start = rp_s[hs.head_row] - nz0;  // the row's first entry lives in group j0 <= group - 1
        int j0 = group - 1;
        while (j0 > 0 && j0 * sg.seg_len > e_start) --j0;
        float4 tot = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int j = j0; j < group; ++j) {
            const float4 q = lds_f128(left_base + (uint32_t)j * 128u + ckey);
            tot.x += q.x; tot.y += q.y; tot.z += q.z; tot.w += q.w;
        }
        tot.x += hs.head.x; tot.y += hs.head.y; tot.z += hs.head.z; tot.w += hs.head.w;
        emit_row<FIRST>(Tdst, hs.head_row, ckey, tot);
    }
}

// row-per-warp fallback used when the CSR slice stays in global memory (huge / dense tiles)
template <bool HAS_VALS>
__device__ __forceinline__ void spmm_rows_global(uint32_t Tsrc, uint32_t Tdst, bool first, int rows, const int* rp_s,
                                                 const int32_t* __restrict__ colidx, const float* __restrict__ vals,
                                                 int node0, int warp, uint32_t key) {
    for (int r = warp; r < rows; r += FWD_NWARPS) {
        const float s = gather_row<HAS_VALS, false>(Tsrc, rp_s[r], rp_s[r + 1], 0, 0, colidx, vals, node0, key);
        const uint32_t d = Tdst + (swz_row((uint32_t)r) ^ key);
        sts_f32(d, first ? s : 2.f * s - lds_f32(d));
    }
}

// -------------------------------------------------------------------------------------------
// Issue the loads of one tile: X rows -> swizzled tile buffer, raw rowptr / colidx / vals -> staging.
// Everything that can be is a cp.async (completion: cp_async_wait + __syncthreads by the caller).
// -------------------------------------------------------------------------------------------
template <bool HAS_VALS, bool STAGED>
__device__ __forceinline__ void issue_tile_loads(const FwdParams& p, const TileInfo& t, uint32_t Tbuf, uint32_t rp_a,
                                                 uint32_t pre_a, uint32_t val_a, int tid) {
    const int fi = p.layers[0].f_in;
    if ((fi & 3) == 0 && (reinterpret_cast<uintptr_t>(p.X) & 15u) == 0) {
        const int cpr = fi >> 2;  // 16 B chunks per row
        const float* src = p.X + (size_t)t.node0 * fi;
        const int total = t.rows * cpr;
        if (cpr == 8) {
            for (int c = tid; c < total; c += FWD_THREADS) {
                const uint32_t r = (uint32_t)c >> 3, ch = (uint32_t)c & 7u;
                cp_async16(Tbuf + (r << 7) + ((ch ^ (r & 7u)) << 4), src + (size_t)c * 4);
            }
        } else {
            for (int c = tid; c < total; c += FWD_THREADS) {
                const uint32_t r = (uint32_t)(c / cpr), ch = (uint32_t)(c - (int)r * cpr);
                cp_async16(Tbuf + (r << 7) + ((ch ^ (r & 7u)) << 4), src + (size_t)c * 4);
            }
            if (cpr & 1) {  // f_in = 4 (mod 8): zero the pad chunk so columns [f_in, pad8(f_in)) are defined
                for (int r = tid; r < t.rows; r += FWD_THREADS) {
                    const uint32_t a = Tbuf + ((uint32_t)r << 7) + ((((uint32_t)cpr) ^ ((uint32_t)r & 7u)) << 4);
                    asm volatile("st.shared.v4.u32 [%0], {%1,%1,%1,%1};" ::"r"(a), "r"(0u));
                }
            }
        }
    } else {
        const int fi_pad = pad8(fi);
        for (int idx = tid; idx < t.rows * fi_pad; idx += FWD_THREADS) {
            const int r = idx / fi_pad, c = idx - r * fi_pad;
            sts_f32(Tbuf + swz_off((uint32_t)r, (uint32_t)c), c < fi ? __ldg(p.X + (size_t)(t.node0 + r) * fi + c) : 0.f);
        }
    }
    for (int i = tid; i <= t.rows; i += FWD_THREADS) cp_async4(rp_a + i * 4, p.b.rowptr + t.node0 + i);
    if (STAGED) {
        for (int e = tid; e < t.nnz; e += FWD_THREADS) {
            cp_async4(pre_a + e * 4, p.b.colidx + t.nz0 + e);
            if (HAS_VALS) cp_async4(val_a + e * 4, p.b.vals + t.nz0 + e);
        }
    }
}

// tcgen05 A operands of a [rows_cap][32] fp32 tile: the tile itself serves as the "hi" part - kind::tf32 reads
// fp32 words and ignores the low 13 mantissa bits (verified on B200: tests pass with errors ~1e-6) - and this
// pass writes the matching "lo" tile, lo = rn_tf32(x - trunc_tf32(x)), in the same swizzled layout.
__device__ __forceinline__ void split_tile_lo(uint32_t src, uint32_t alo, int n_rows16, int tid) {
    for (int idx = tid; idx < n_rows16 * 16 * 8; idx += FWD_THREADS) {
        const uint32_t off = (uint32_t)idx << 4;  // (row, physical chunk) -> byte offset; the swizzle is a permutation
        const float4 v = lds_f128(src + off);
        const float x[4] = {v.x, v.y, v.z, v.w};
        uint32_t l[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float hi = __uint_as_float(__float_as_uint(x[i]) & 0xffffe000u);
            l[i] = (__float_as_uint(x[i] - hi) + 0x1000u) & 0xffffe000u;
        }
        asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(alo + off), "r"(l[0]), "r"(l[1]), "r"(l[2]), "r"(l[3]));
    }
}

template <int MT, bool HAS_VALS, bool STAGED, bool TC5>
__global__ void __launch_bounds__(FWD_THREADS, (MT == 1 ? 2 : 1))
cheb_forward_kernel(const __grid_constant__ FwdParams p) {
    extern __shared__ __align__(1024) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // programmatic dependent launch: let the next launch in the stream start filling SM slots as soon as this
    // grid's CTAs drain; it parks at griddepcontrol.wait (below) until this grid has completed
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const uint32_t key = swz_key((uint32_t)lane);        // lane = feature layout (global-CSR fallback)
    const uint32_t ckey = ((uint32_t)lane & 7u) << 4;    // lane = 16 B chunk layout (stream walk)

    // ---- shared memory carve-up
    const uint32_t tile_bytes = (uint32_t)p.rows_cap * 128u;
    const int n_tbuf = p.prefetch ? 3 : 2;
    // TC5: one more tile holds the TF32 "lo" part of T_k (the fp32 tile itself is the "hi" tcgen05 operand); the
    // leftover slots of the walk alias the head of the lo tile (written only after the step's MMAs completed)
    unsigned char* Alo = smem + (size_t)n_tbuf * tile_bytes;
    unsigned char* Wimg = Alo + (TC5 ? tile_bytes : 0u);  // per layer: [hi rows][lo rows][8 bias rows]
    unsigned char* left_s = TC5 ? Alo : Wimg + (size_t)p.w_rows_cap * 128;  // 4*NWARPS leftover slots of 128 B
    int* csr0 = reinterpret_cast<int*>(Wimg + (size_t)p.w_rows_cap * 128 + (TC5 ? 0 : 4 * FWD_NWARPS * 128));
    const int rp_words = (p.rows_cap + 2 + 3) & ~3;
    const int csr_words = rp_words + p.nnz_cap * (HAS_VALS ? 2 : 1);
    const uint32_t smem_a = smem_u32(smem);
    const uint32_t w_a = smem_u32(Wimg);
    const uint32_t csr_a0 = smem_u32(csr0);
    const uint32_t left_base = smem_u32(left_s);
    // TC5: warp 0 feeds the tensor core (MMA issue costs its elected thread a few hundred cycles per step), so it
    // sits out the walk: 4*(NWARPS-1) lane groups over warps 1..; otherwise every warp walks
    constexpr int NGROUPS = TC5 ? 4 * (FWD_NWARPS - 1) : 4 * FWD_NWARPS;
    const bool walker = !TC5 || warp > 0;
    const int group = walker ? (warp - (TC5 ? 1 : 0)) * 4 + (lane >> 3) : NGROUPS;  // NGROUPS = "no segment"
    const uint32_t left_a = left_base + (uint32_t)group * 128u + ckey;

    // rotating tile buffers: bx = T_0 / X of the current tile, bs = scratch, bp = prefetch target
    uint32_t bx = smem_a, bs = smem_a + tile_bytes, bp = smem_a + 2u * tile_bytes;
    int cs = 0;  // CSR staging set of the current tile

    // everything above touched only this CTA's shared / tensor memory; from here on global memory written by
    // earlier launches in the stream is read (weights image, scheduler counters, inputs)
    asm volatile("griddepcontrol.wait;" ::: "memory");
    // resident weights ride in the first cp.async group (waited for before the first tile computes)
    if (p.w_resident)
        for (int l = 0; l < p.n_layers; ++l) stage_weights_async(p, l, w_a + (uint32_t)p.w_row_off[l] * 128u, tid);

    // ---- tile scheduler.  Dynamic (largest tile first, CTAs pull indices from a global counter) when the
    // batch carries tile_info - with only ~2 tiles per CTA a static split leaves 30 % of the SMs idle in
    // the last round - else static round-robin.  The pipeline always knows the next TWO tile indices.
    int* s_idx = csr0 + (p.prefetch ? 2 : 1) * csr_words;  // two ints behind the CSR staging set(s)
    // TC5: completion mbarrier (8 B) and the TMEM base address slot behind them
    const uint32_t mbar = smem_u32(s_idx + 2), tslot = smem_u32(s_idx + 4);
    const uint32_t alo_a = smem_u32(Alo);
    uint32_t tmem_base = 0, mma_phase = 0;
    if (TC5) {
        if (warp == 0) tmem_alloc(tslot, 32);
        if (tid == 0) mbar_init(mbar, 1);
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
        tmem_base = *reinterpret_cast<volatile uint32_t*>(s_idx + 4);
    }
    const bool dyn = (p.sched != nullptr);
    int it = 0;
    int i_cur, i_nxt;
    if (dyn) {
        if (tid == 0) { s_idx[0] = atomicAdd(p.sched, 1); s_idx[1] = atomicAdd(p.sched, 1); }
        __syncthreads();
        i_cur = s_idx[0]; i_nxt = s_idx[1];
        __syncthreads();  // slot 0 is rewritten by thread 0 at the top of the first iteration
    } else {
        i_cur = blockIdx.x; i_nxt = blockIdx.x + gridDim.x;
    }
    auto finish = [&]() {
        cp_async_wait<0>();
        if (TC5) {
            tc_fence_before();
            __syncthreads();
            if (warp == 0) tmem_dealloc(tmem_base, 32);
        }
        if (dyn && tid == 0) {  // the last CTA out re-arms the counters for the next launch
            __threadfence();
            if (atomicAdd(p.sched + 1, 1) == (int)gridDim.x - 1) { p.sched[0] = 0; p.sched[1] = 0; }
        }
    };
    if (i_cur >= p.b.n_tiles) { finish(); return; }
    TileInfo cur = load_tile_info(p.b, i_cur);
    TileInfo nxt = cur;
    bool has_nxt = i_nxt < p.b.n_tiles;
    if (p.prefetch) {
        issue_tile_loads<HAS_VALS, STAGED>(p, cur, bx, csr_a0, csr_a0 + rp_words * 4, csr_a0 + (rp_words + p.nnz_cap) * 4, tid);
        cp_async_commit();
    }
    if (has_nxt) nxt = load_tile_info(p.b, i_nxt);

    for (;; ++it) {
        const uint32_t rp_a = csr_a0 + (uint32_t)(cs * csr_words) * 4u;
        const uint32_t pre_a = rp_a + rp_words * 4, val_a = pre_a + p.nnz_cap * 4;
        const int* rp_s = csr0 + cs * csr_words;
        if (dyn && tid == 0) s_idx[it & 1] = has_nxt ? atomicAdd(p.sched, 1) : p.b.n_tiles;  // index of tile it+2
        if (p.prefetch) {
            // next tile's loads go out now
            if (has_nxt) {
                const uint32_t rp_n = csr_a0 + (uint32_t)((cs ^ 1) * csr_words) * 4u;
                issue_tile_loads<HAS_VALS, STAGED>(p, nxt, bp, rp_n, rp_n + rp_words * 4, rp_n + (rp_words + p.nnz_cap) * 4, tid);
            }
            cp_async_commit();
            cp_async_wait<1>();  // the current tile's group has landed; the next tile's may still fly
        } else {
            issue_tile_loads<HAS_VALS, STAGED>(p, cur, bx, rp_a, pre_a, val_a, tid);
            cp_async_commit();
            cp_async_wait<0>();
        }
        if (TC5) fence_proxy_async();  // cp.async-written weight images -> visible to the tensor-core proxy
        __syncthreads();
        // the tile after next: its index was published by the barrier, its bounds are consumed next iteration
        const int i_nn = dyn ? s_idx[it & 1] : (int)(blockIdx.x + (it + 2) * gridDim.x);
        const bool has_nn = has_nxt && i_nn < p.b.n_tiles;
        TileInfo nn = nxt;
        if (has_nn) nn = load_tile_info(p.b, i_nn);

        const int rows = cur.rows, node0 = cur.node0, nz0 = cur.nz0;
        const int n_mtiles = (rows + 15) >> 4;
        SegInfo sg;
        sg.sb = 0; sg.n = 0; sg.r0 = 0; sg.mid = 0; sg.seg_len = 1;
        if (STAGED) {
            // column ids -> swizzled smem row offsets (one thread per entry) ...
            for (int e = tid; e < cur.nnz; e += FWD_THREADS)
                sts_u32(pre_a + e * 4, swz_row(lds_u32(pre_a + e * 4) - (uint32_t)node0));
            // ... the group's segment of the entry stream and the row it starts in ...
            {
                const int L = (cur.nnz + NGROUPS - 1) / NGROUPS;
                sg.seg_len = L > 0 ? L : 1;
                const int sb = min(group * sg.seg_len, cur.nnz);
                sg.sb = sb;
                sg.n = min(sg.seg_len, cur.nnz - sb);
                int lo = 0, hi = rows;  // largest r with rp[r] - nz0 <= sb  (== row containing sb when n > 0)
                while (lo < hi) {
                    const int mid = (lo + hi + 1) >> 1;
                    if (rp_s[mid] - nz0 <= sb) lo = mid; else hi = mid - 1;
                }
                sg.r0 = lo;
                sg.mid = (sg.n > 0 && (rp_s[lo] - nz0) < sb) ? 1 : 0;
            }
            __syncthreads();
            // ... then the row-end / next-row-empty flags (one thread per row)
            for (int r = tid; r < rows; r += FWD_THREADS) {
                const int e1 = rp_s[r + 1] - nz0;
                if (e1 > rp_s[r] - nz0) {
                    const bool next_empty = (r + 1 < rows) && (rp_s[r + 2] == rp_s[r + 1]);
                    const uint32_t a = pre_a + (uint32_t)(e1 - 1) * 4u;
                    sts_u32(a, lds_u32(a) | 1u | (next_empty ? 2u : 0u));
                }
            }
            __syncthreads();
        }

        for (int li = 0; li < p.n_layers; ++li) {
            const LayerDev& L = p.layers[li];
            const int fi_pad = pad8(L.f_in), fo_pad = pad8(L.f_out), fo_img = pad16(L.f_out);
            const int nchunks = fi_pad >> 3, nnt = fo_pad >> 3;
            const int w_rows_l = L.K * fo_img;
            const int w_row0 = p.w_resident ? p.w_row_off[li] : 0;
            const uint32_t w_l = w_a + (uint32_t)w_row0 * 128u;
            const float* bias_s = reinterpret_cast<const float*>(Wimg + (size_t)(w_row0 + 2 * w_rows_l) * 128);
            if (!p.w_resident) {
                // restage this layer's block (after every warp left the previous layer's epilogue, which
                // reads its bias row); it joins the pending (next-tile) group, so drain everything
                if (li > 0) __syncthreads();
                stage_weights_async(p, li, w_l, tid);
                cp_async_commit();
                cp_async_wait<0>();
                if (TC5) fence_proxy_async();
                __syncthreads();
            } else if (li > 0) {
                __syncthreads();  // H_l written by the previous layer's epilogue
            }
            if (TC5) {  // A operands of T_0 (every MMA that read the split tiles has completed: the epilogue waited)
                split_tile_lo(bx, alo_a, n_mtiles, tid);
                fence_proxy_async();  // also publishes the generic-proxy writes of bx (epilogue / cp.async) to the tensor core
                __syncthreads();
            }

            const int mslot = warp & (FWD_MSLOTS - 1), nt0 = (warp / FWD_MSLOTS) * 2;
            const bool has_n = nt0 < nnt;  // this warp's n-tile half exists for this layer
            const uint32_t idesc = umma_idesc_tf32_m128((uint32_t)fo_img);
            float acc[MT][2][4];
#pragma unroll
            for (int m = 0; m < MT; ++m)
#pragma unroll
                for (int n = 0; n < 2; ++n)
#pragma unroll
                    for (int i = 0; i < 4; ++i) acc[m][n][i] = 0.f;

            uint32_t tk = bx, tprev = bs;  // T_k, and the buffer T_{k+1} is written to (holds T_{k-1})
            for (int k = 0; k < L.K; ++k) {
                const uint32_t whi_k = w_l + (uint32_t)(k * fo_img) * 128u;
                const uint32_t wlo_k = whi_k + (uint32_t)w_rows_l * 128u;
                const bool more = k + 1 < L.K;
                HeadState hs;
                hs.pending = 0;
                if (TC5) {
                    // one thread feeds the tensor core: D[128 x fo_img] (+)= A_lo B_hi + A_hi B_lo + A_hi B_hi per 8-wide
                    // K chunk, straight from the swizzled tiles; completion is signalled on the mbarrier
                    if (tid == 0) {
                        tc_fence_after();
                        // D[128 x fo_img] (+)= A_lo B_lo + A_lo B_hi + A_hi B_lo + A_hi B_hi per 8-wide K chunk; descriptors
                        // advance by 32 B (= +2 in the >>4 address field) per chunk
                        uint64_t a_hi = umma_desc_sw128(tk), a_lo = umma_desc_sw128(alo_a);
                        uint64_t b_hi = umma_desc_sw128(whi_k), b_lo = umma_desc_sw128(wlo_k);
                        uint32_t accum = k > 0 ? 1u : 0u;
                        for (int c = 0; c < nchunks; ++c) {
                            umma_tf32(tmem_base, a_lo, b_lo, idesc, accum);
                            umma_tf32(tmem_base, a_lo, b_hi, idesc, 1u);
                            umma_tf32(tmem_base, a_hi, b_lo, idesc, 1u);
                            umma_tf32(tmem_base, a_hi, b_hi, idesc, 1u);
                            accum = 1u;
                            a_hi += 2; a_lo += 2; b_hi += 2; b_lo += 2;
                        }
                        umma_commit(mbar);
                    }
                    if (more) {
                        // (the walk parks its leftovers in the head of the lo tile: wait for the MMAs first)
                        if (walker) {
                            if (k == 0) spmm_seg_walk<HAS_VALS, true, true>(tk, tprev, sg, rows, rp_s, pre_a, val_a, ckey, left_a, group == 0, hs, mbar, mma_phase);
                            else spmm_seg_walk<HAS_VALS, false, true>(tk, tprev, sg, rows, rp_s, pre_a, val_a, ckey, left_a, group == 0, hs, mbar, mma_phase);
                        }
                        __syncthreads();
                        if (k == 0) spmm_fixup<true>(tprev, sg, group, rp_s, nz0, ckey, left_base, hs);
                        else spmm_fixup<false>(tprev, sg, group, rp_s, nz0, ckey, left_base, hs);
                        __syncthreads();
                        // (walkers waited on this phase inside the walk; the MMA warp checks once here - long complete -
                        //  instead of spinning on the barrier while the others walk)
                        if (!walker) mbar_wait(mbar, mma_phase);
                        mma_phase ^= 1u;
                        split_tile_lo(tprev, alo_a, n_mtiles, tid);
                        fence_proxy_async();  // lo tile AND the walk's generic-proxy writes of T_{k+1} -> tensor-core proxy
                    }
                } else {
                if (more) {
                    if (STAGED) {
                        if (k == 0) spmm_seg_walk<HAS_VALS, true, false>(tk, tprev, sg, rows, rp_s, pre_a, val_a, ckey, left_a, group == 0, hs, 0u, 0u);
                        else spmm_seg_walk<HAS_VALS, false, false>(tk, tprev, sg, rows, rp_s, pre_a, val_a, ckey, left_a, group == 0, hs, 0u, 0u);
                    } else {
                        spmm_rows_global<HAS_VALS>(tk, tprev, k == 0, rows, rp_s, p.b.colidx, p.b.vals, node0, warp, key);
                    }
                }
                // the dense contribution of T_k right behind the walk: warps that finish their segment early
                // start on the tensor cores, so one barrier absorbs the imbalance of both
                if (has_n) {
#pragma unroll
                    for (int m = 0; m < MT; ++m) {
                        const int mt = mslot + m * FWD_MSLOTS;
                        if (mt < n_mtiles) mma_tile(acc[m], tk, mt * 16, whi_k, wlo_k, nchunks, nt0, nnt, lane);
                    }
                }
                if (more && STAGED) {
                    __syncthreads();  // every group's leftover is published
                    if (k == 0) spmm_fixup<true>(tprev, sg, group, rp_s, nz0, ckey, left_base, hs);
                    else spmm_fixup<false>(tprev, sg, group, rp_s, nz0, ckey, left_base, hs);
                }
                }
                if (TC5) {
                    // only the MMA warp needs everybody's lo-tile slice before it feeds the tensor core again; the
                    // walkers just signal and move on (their next gathers need T_{k+1}, final since the last barrier)
                    if (more) {
                        if (warp == 0) asm volatile("bar.sync 1, %0;" ::"n"(FWD_THREADS) : "memory");
                        else asm volatile("bar.arrive 1, %0;" ::"n"(FWD_THREADS) : "memory");
                    }
                } else {
                    __syncthreads();
                }
                const uint32_t tmp = tk; tk = tprev; tprev = tmp;
            }

            // ---- epilogue: bias + activation; last layer -> Y, hidden layer -> tile bx (+ saved)
            const bool last = (li == p.n_layers - 1);
            const int fo = L.f_out;
            float* gout = last ? p.Y : (p.saved ? p.saved + p.layers[li + 1].saved_off : nullptr);
            const int g = lane >> 2, t4 = lane & 3;
            if (TC5) {
                // accumulator: TMEM lane = tile row, column = output feature.  warp w reads lane quadrant (w & 3),
                // 8-column block (w >> 2): thread t holds row 32 q + t, columns 8 cb .. 8 cb + 7
                mbar_wait(mbar, mma_phase);
                mma_phase ^= 1u;
                tc_fence_after();
                const int q = warp & 3, cb = warp >> 2;
                const int r = q * 32 + lane;
                if (cb * 8 < fo_img) {
                    uint32_t v[8];
                    tmem_ld_32x32b_x8(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(cb * 8), v);
                    float y[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) y[j] = apply_act(__uint_as_float(v[j]) + bias_s[cb * 8 + j], L.act, L.slope);
                    if (!last) {
                        // columns >= f_out are exact zeros (zero W rows, zero bias, act(0) = 0)
                        sts_f128(bx + swz_off((uint32_t)r, (uint32_t)(cb * 8)), make_float4(y[0], y[1], y[2], y[3]));
                        sts_f128(bx + swz_off((uint32_t)r, (uint32_t)(cb * 8 + 4)), make_float4(y[4], y[5], y[6], y[7]));
                    }
                    if (gout != nullptr && r < rows) {
                        float* dst = gout + (size_t)(node0 + r) * fo + cb * 8;
                        if ((fo & 3) == 0 && cb * 8 + 8 <= fo && (reinterpret_cast<uintptr_t>(gout) & 15u) == 0) {
                            *reinterpret_cast<float4*>(dst) = make_float4(y[0], y[1], y[2], y[3]);
                            *reinterpret_cast<float4*>(dst + 4) = make_float4(y[4], y[5], y[6], y[7]);
                        } else {
#pragma unroll
                            for (int j = 0; j < 8; ++j)
                                if (cb * 8 + j < fo) dst[j] = y[j];
                        }
                    }
                }
                tc_fence_before();  // TMEM reads ordered before the next layer's / tile's MMAs (which follow a barrier)
            } else {
#pragma unroll
            for (int m = 0; m < MT; ++m) {
                const int mt = mslot + m * FWD_MSLOTS;
                if (has_n && mt < n_mtiles) {
#pragma unroll
                    for (int n = 0; n < 2; ++n) {
                        if (nt0 + n < nnt) {
                            const int col = (nt0 + n) * 8 + 2 * t4;
                            const float b0 = bias_s[col], b1 = bias_s[col + 1];
#pragma unroll
                            for (int h = 0; h < 2; ++h) {
                                const int r = mt * 16 + g + h * 8;
                                const float y0 = apply_act(acc[m][n][2 * h] + b0, L.act, L.slope);
                                const float y1 = apply_act(acc[m][n][2 * h + 1] + b1, L.act, L.slope);
                                if (!last) {
                                    // padded columns are exact zeros (zero W rows, zero bias, act(0)=0)
                                    const uint32_t a = bx + swz_off((uint32_t)r, (uint32_t)col);
                                    asm volatile("st.shared.v2.f32 [%0], {%1,%2};" ::"r"(a), "f"(y0), "f"(y1));
                                }
                                if (gout != nullptr && r < rows) {
                                    float* dst = gout + (size_t)(node0 + r) * fo + col;
                                    if ((fo & 1) == 0 && col + 1 < fo && (reinterpret_cast<uintptr_t>(gout) & 7u) == 0) {
                                        *reinterpret_cast<float2*>(dst) = make_float2(y0, y1);
                                    } else {
                                        if (col < fo) dst[0] = y0;
                                        if (col + 1 < fo) dst[1] = y1;
                                    }
                                }
                            }
                        }
                    }
                }
            }
            }  // !TC5
        }
        // rotate: the prefetched buffer becomes the next tile's X, the old X/scratch become scratch/prefetch
        if (!has_nxt) break;
        if (p.prefetch) {
            const uint32_t o_bx = bx, o_bs = bs;
            bx = bp; bs = o_bx; bp = o_bs;
            cs ^= 1;
        } else {
            __syncthreads();  // staging buffers are rewritten right away by the next tile's loads
        }
        cur = nxt; nxt = nn; has_nxt = has_nn;
    }
    finish();
}

// -------------------------------------------------------------------------------------------
// host launcher
// -------------------------------------------------------------------------------------------
static size_t fwd_smem_bytes(int rows_cap, int nnz_cap, int w_rows, bool has_vals, bool prefetch, bool tc5) {
    size_t s = (size_t)rows_cap * 128 * ((prefetch ? 3 : 2) + (tc5 ? 1 : 0)) + (size_t)w_rows * 128 + (tc5 ? 0 : 4 * FWD_NWARPS * 128);
    const size_t csr_words = (size_t)((rows_cap + 2 + 3) & ~3) + (size_t)nnz_cap * (has_vals ? 2 : 1);
    s += csr_words * 4 * (prefetch ? 2 : 1);
    return s + 32;  // + the scheduler's two index slots, the MMA completion mbarrier and the TMEM address slot
}

template <int MT, bool HAS_VALS, bool STAGED, bool TC5 = false>
static cudaError_t launch_one(const FwdParams& p, int grid, size_t smem, cudaStream_t st) {
    return mho_launch<cheb_forward_kernel<MT, HAS_VALS, STAGED, TC5>>(dim3((unsigned)grid), dim3(FWD_THREADS), smem, st, true, p);
}

template <int MT>
static cudaError_t launch_mt(const FwdParams& p, bool has_vals, bool staged, int grid, size_t smem, cudaStream_t st) {
    if (has_vals) return staged ? launch_one<MT, true, true>(p, grid, smem, st) : launch_one<MT, true, false>(p, grid, smem, st);
    return staged ? launch_one<MT, false, true>(p, grid, smem, st) : launch_one<MT, false, false>(p, grid, smem, st);
}

// Returns cudaSuccess or an error; *too_large set when the tile cannot fit in shared memory.
cudaError_t cheb_forward_launch(FwdParams& p, int max_tile_rows, int max_tile_nnz, int num_sms, int max_smem_optin,
                                cudaStream_t st, bool* too_large) {
    *too_large = false;
    p.rows_cap = pad16(max_tile_rows < 16 ? 16 : max_tile_rows);
    const bool has_vals = p.b.vals != nullptr;
    const int MTn = (p.rows_cap + 16 * FWD_MSLOTS - 1) / (16 * FWD_MSLOTS);
    if (MTn > 4) { *too_large = true; return cudaSuccess; }
    const int mt_sel = MTn <= 1 ? 1 : (MTn <= 2 ? 2 : 4);
    const int reg_limit = mt_sel == 1 ? 2 : 1;

    // weight blocks (hi + lo images + bias row per layer): resident when all of them cost <= 64 KB
    int w_sum = 0, w_max = 0;
    for (int l = 0; l < p.n_layers; ++l) {
        const int r = wprep_layer_rows(p.layers[l].K, p.layers[l].f_out);
        p.w_row_off[l] = w_sum;
        w_sum += r;
        w_max = r > w_max ? r : w_max;
    }
    p.w_resident = (p.n_layers == 1 || w_sum * 128 <= 64 * 1024) ? 1 : 0;
    p.w_rows_cap = p.w_resident ? w_sum : w_max;
    if (!p.w_resident) for (int l = 0; l < p.n_layers; ++l) p.w_row_off[l] = 0;

    // preference order: tcgen05 dense path (one 128-row M tile, no prefetch buffer), then
    // staged+prefetch with >=2 CTAs/SM, staged+prefetch, staged, global CSR
    const int nnz_cap = (max_tile_nnz + 3) & ~3;
    bool staged = true, prefetch = true, tc5 = false;
    auto per_sm_of = [&](size_t s) { int v = (int)((size_t)(228 * 1024) / (s + 1024)); return v > reg_limit ? reg_limit : v; };
    size_t smem = 0;
    if (mt_sel == 1) {
        p.rows_cap = 128;  // the UMMA M extent
        const size_t s5p = fwd_smem_bytes(128, nnz_cap, p.w_rows_cap, has_vals, true, true);
        const size_t s5 = fwd_smem_bytes(128, nnz_cap, p.w_rows_cap, has_vals, false, true);
        if (s5p <= (size_t)max_smem_optin && per_sm_of(s5p) >= 2) { tc5 = true; prefetch = true; smem = s5p; }
        else if (s5 <= (size_t)max_smem_optin) { tc5 = true; prefetch = false; smem = s5; }
    }
    if (!tc5) {
        smem = fwd_smem_bytes(p.rows_cap, nnz_cap, p.w_rows_cap, has_vals, true, false);
        const size_t smem_np = fwd_smem_bytes(p.rows_cap, nnz_cap, p.w_rows_cap, has_vals, false, false);
        if (smem > (size_t)max_smem_optin || (per_sm_of(smem) < 2 && per_sm_of(smem_np) >= 2 && reg_limit >= 2)) {
            prefetch = false;
            smem = smem_np;
        }
        if (smem > (size_t)max_smem_optin) {
            staged = false;
            smem = fwd_smem_bytes(p.rows_cap, 0, p.w_rows_cap, has_vals, false, false);
            if (smem > (size_t)max_smem_optin) { *too_large = true; return cudaSuccess; }
        }
    }
    p.tc5 = tc5 ? 1 : 0;
    p.nnz_cap = staged ? nnz_cap : 0;
    p.prefetch = prefetch ? 1 : 0;
    if (p.b.tile_info == nullptr) p.sched = nullptr;  // static round-robin without a (sorted) tile_info
    int per_sm = per_sm_of(smem);
    if (per_sm < 1) per_sm = 1;
    int grid = num_sms * per_sm;
    if (grid > p.b.n_tiles) grid = p.b.n_tiles;
    if (grid < 1) grid = 1;
    if (p.tc5) return has_vals ? launch_one<1, true, true, true>(p, grid, smem, st) : launch_one<1, false, true, true>(p, grid, smem, st);
    switch (mt_sel) {
        case 1: return launch_mt<1>(p, has_vals, staged, grid, smem, st);
        case 2: return launch_mt<2>(p, has_vals, staged, grid, smem, st);
        default: return launch_mt<4>(p, has_vals, staged, grid, smem, st);
    }
}
