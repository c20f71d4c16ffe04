// Shared device helpers for libmho (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/mho.h"

#define MHO_THREADS 256
#define MHO_NWARPS (MHO_THREADS / 32)

// ---------------------------------------------------------------------------------------------
// Shared-memory tile layout: [rows][32] fp32, one row = 128 B, 16-byte chunks XOR-swizzled with
// (row & 7).  This is the canonical "K-major, SWIZZLE_128B" layout: conflict-free for the
// row gathers of the sparse recurrence (a warp reads one row = 32 distinct banks), conflict-free
// for ldmatrix (8 rows x 16 B land in 8 distinct bank groups), writable by TMA with
// CU_TENSOR_MAP_SWIZZLE_128B and directly describable as a tcgen05 smem operand.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t swz_off(uint32_t row, uint32_t col) {
    return (row << 7) | ((((col >> 2) ^ (row & 7u)) << 4)) | ((col & 3u) << 2);
}
// row part of the offset with the swizzle key folded in: off(row, col) = swz_row(row) ^ lane_key(col)
__device__ __forceinline__ uint32_t swz_row(uint32_t row) { return (row << 7) | ((row & 7u) << 4); }
__device__ __forceinline__ uint32_t swz_key(uint32_t col) { return ((col >> 2) << 4) | ((col & 3u) << 2); }

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ float lds_f32(uint32_t addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_f32(uint32_t addr, float v) {
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v));
}
__device__ __forceinline__ uint4 lds_u128(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src));
}
__device__ __forceinline__ void cp_async4(uint32_t dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src));
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_u32(uint32_t addr, uint32_t v) {
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N)); }

// ---------------------------------------------------------------------------------------------
// 3xTF32: a*b ~= a_lo*b_hi + a_hi*b_lo + a_hi*b_hi with fp32 accumulate (error ~2^-21 per product)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t f2tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
    hi = f2tf32(x);
    lo = f2tf32(x - __uint_as_float(hi));
}
// Cheap round-to-nearest(ties away) TF32 split with integer ops (the PTX cvt.rna.tf32.f32 expands to
// ~5 instructions with its inf/nan handling): hi = rn_tf32(x), lo = rn_tf32(x - hi).  5 instructions.
__device__ __forceinline__ void split_tf32_fast(float x, uint32_t& hi, uint32_t& lo) {
    hi = (__float_as_uint(x) + 0x1000u) & 0xffffe000u;
    lo = (__float_as_uint(x - __uint_as_float(hi)) + 0x1000u) & 0xffffe000u;
}
__device__ __forceinline__ float4 lds_f128(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_f128(uint32_t addr, float4 v) {
    asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w));
}
__device__ __forceinline__ void ldmatrix_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
                 : "r"(addr));
}
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// ---------------------------------------------------------------------------------------------
// s = sum_{e in [e0,e1)} val[e] * T[col[e]][lane]   for one operator row, one lane per feature.
// STAGED: col ids were pre-translated to swizzled smem row offsets (pre_a), 4 per LDS.128;
// otherwise the CSR slice is read from global memory through L1 (e0/e1 are global offsets).
// ---------------------------------------------------------------------------------------------
template <bool HAS_VALS, bool STAGED>
__device__ __forceinline__ float gather_row(uint32_t Tsrc, int e0, int e1, uint32_t pre_a, uint32_t val_a,
                                            const int32_t* __restrict__ colidx, const float* __restrict__ vals,
                                            int node0, uint32_t key) {
    float s0 = 0.f, s1 = 0.f;
    int e = e0;
    if (STAGED) {
        for (; (e & 3) && e < e1; ++e) {  // head (unaligned)
            uint32_t p;
            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(p) : "r"(pre_a + e * 4));
            const float t = lds_f32(Tsrc + (p ^ key));
            s0 = HAS_VALS ? fmaf(lds_f32(val_a + e * 4), t, s0) : s0 + t;
        }
        for (; e + 4 <= e1; e += 4) {  // body: 4 pre-swizzled offsets per LDS.128
            const uint4 p = lds_u128(pre_a + e * 4);
            const float t0 = lds_f32(Tsrc + (p.x ^ key));
            const float t1 = lds_f32(Tsrc + (p.y ^ key));
            const float t2 = lds_f32(Tsrc + (p.z ^ key));
            const float t3 = lds_f32(Tsrc + (p.w ^ key));
            if (HAS_VALS) {
                const uint4 v = lds_u128(val_a + e * 4);
                s0 = fmaf(__uint_as_float(v.x), t0, s0);
                s1 = fmaf(__uint_as_float(v.y), t1, s1);
                s0 = fmaf(__uint_as_float(v.z), t2, s0);
                s1 = fmaf(__uint_as_float(v.w), t3, s1);
            } else {
                s0 += t0 + t2;
                s1 += t1 + t3;
            }
        }
        for (; e < e1; ++e) {  // tail
            uint32_t p;
            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(p) : "r"(pre_a + e * 4));
            const float t = lds_f32(Tsrc + (p ^ key));
            s1 = HAS_VALS ? fmaf(lds_f32(val_a + e * 4), t, s1) : s1 + t;
        }
    } else {
        for (; e < e1; ++e) {
            const uint32_t j = (uint32_t)(__ldg(colidx + e) - node0);
            const float t = lds_f32(Tsrc + (swz_row(j) ^ key));
            s0 = HAS_VALS ? fmaf(__ldg(vals + e), t, s0) : s0 + t;
        }
    }
    return s0 + s1;
}

__device__ __forceinline__ float apply_act(float z, int act, float slope) {
    if (act == MHO_ACT_RELU) return fmaxf(z, 0.f);
    if (act == MHO_ACT_LEAKY) return z > 0.f ? z : slope * z;
    return z;
}
__device__ __forceinline__ float act_grad_from_out(float y, int act, float slope) {
    // act'(z) expressed with the OUTPUT y: for relu and leaky (slope>0) y>0 <=> z>0 (TF uses strict >)
    if (act == MHO_ACT_RELU) return y > 0.f ? 1.f : 0.f;
    if (act == MHO_ACT_LEAKY) return y > 0.f ? 1.f : slope;
    return 1.f;
}

// ---------------------------------------------------------------------------------------------
// tcgen05 (5th-generation tensor core) helpers: TMEM allocation, UMMA descriptors, MMA issue,
// completion barrier, TMEM -> register loads.  cta_group::1 only.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t slot_smem_addr, uint32_t ncols) {  // one full warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_smem_addr), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // the allocating warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "MHO_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra MHO_DONE_%=;\n\t"
        "bra MHO_WAIT_%=;\n\t"
        "MHO_DONE_%=:\n\t"
        "}" ::"r"(bar), "r"(parity) : "memory");
}
// K-major, SWIZZLE_128B shared-memory operand descriptor (cute::UMMA::SmemDescriptor): start address >> 4,
// LBO = 1 (unused for swizzled K-major), SBO = 1024 B between 8-row groups, version 1, layout type 2.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
    return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// kind::tf32, fp32 accumulate, both operands K-major, M = 128 (cute::UMMA::InstrDescriptor bit layout)
__device__ __forceinline__ uint32_t umma_idesc_tf32_m128(uint32_t n) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((n >> 3) << 17) | ((128u >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {  // arrive on `bar` once every MMA issued so far has completed
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__host__ __device__ __forceinline__ int pad8(int x) { return (x + 7) & ~7; }
__host__ __device__ __forceinline__ int pad16(int x) { return (x + 15) & ~15; }

// Device-side view of one layer (pointers are device pointers)
struct LayerDev {
    int K, f_in, f_out, act;
    float slope;
    const float* W;
    const float* b;
    long long param_off;  // offset of this layer's kernel in the flat parameter vector
    long long saved_off;  // element offset of this layer's INPUT inside `saved` (layers >= 1)
};

struct BatchDev {
    const int32_t* graph_off;
    const int32_t* rowptr;
    const int32_t* colidx;
    const float* vals;
    const int32_t* tile_off;
    const int32_t* tile_info;  // optional [n_tiles][4] = {node0, rows, nz0, nnz}
    const uint32_t* adj_bits;  // optional [total_nodes][4] binary operator as bit rows (tile-local columns)
    const int32_t* tile_graph0;  // optional [n_tiles] first graph of each listed tile (per-graph operand scales)
    int n_tiles;
    int n_graphs;
};

struct FwdParams {
    BatchDev b;
    int n_layers;
    LayerDev layers[MHO_MAX_LAYERS];
    const float* X;
    float* Y;
    float* saved;     // nullable
    // prepared weights (mho_prepare kernel): per layer [hi image][lo image][bias(32)] as 128 B rows
    const unsigned char* wprep;
    int wprep_row_off[MHO_MAX_LAYERS];  // first 128 B row of each layer's block inside wprep
    int rows_cap;     // multiple of 16, >= max tile rows
    int nnz_cap;      // staged nnz capacity (multiple of 4); 0 => read CSR from global memory
    int w_rows_cap;   // rows (of 128 B) of the smem weight region (hi+lo images)
    int w_resident;   // 1: every layer's images stay in smem for the CTA's lifetime; 0: restaged per layer per tile
    int w_row_off[MHO_MAX_LAYERS];  // first smem image row of each layer (w_resident) else 0
    int* sched;       // {next tile counter, finished-CTA counter} in device memory (dynamic scheduler) or NULL
    int prefetch;     // 1: third tile buffer + second CSR staging set, next tile fetched with cp.async
    int total_nodes;
    int tc5;          // 1: dense part on tcgen05.mma (TMEM accumulators); needs rows_cap <= 128
};

// ---------------------------------------------------------------------------------------------
// Launch Kernel<<<grid, block, smem, st>>>(args...).  pdl: programmatic dependent launch - the kernel may start
// while the previous one in the stream drains, so it must execute griddepcontrol.wait before it reads that
// kernel's results.  The dynamic shared memory limit is sticky per (kernel, device): it is raised only when a
// launch needs more than the default 48 KB and more than an earlier launch on the same device set.
// ---------------------------------------------------------------------------------------------
template <auto Kernel, typename... Args>
cudaError_t mho_launch(dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, Args... args) {
    static int smem_set[64] = {0};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (smem > 48 * 1024 && (int)smem > smem_set[dev & 63]) {
        e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        smem_set[dev & 63] = (int)smem;
    }
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, Kernel, args...);
}
