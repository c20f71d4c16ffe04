// C-ABI glue of libmho.so: context, argument validation, tile planning, launch wrappers.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <algorithm>
#include <vector>

#include "mho_common.cuh"
#include "mho_internal.h"

static thread_local char g_err[512] = "";

void mho_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

#define CUDA_TRY(expr)                                                                      \
    do {                                                                                    \
        cudaError_t _e = (expr);                                                            \
        if (_e != cudaSuccess) {                                                            \
            mho_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return MHO_ERR_CUDA;                                                            \
        }                                                                                   \
    } while (0)

// MHO_DEBUG & 128: report a pending (non-sticky) CUDA error at API boundaries - a call whose error return was dropped
static void dbg_check(const char* where) {
    static int dbg = -1;
    if (dbg < 0) { const char* e = getenv("MHO_DEBUG"); dbg = e ? atoi(e) : 0; }
    if (!(dbg & 128)) return;
    cudaError_t e = cudaPeekAtLastError();
    if (e != cudaSuccess) { fprintf(stderr, "[mho] pending CUDA error at %s: %s\n", where, cudaGetErrorString(e)); cudaGetLastError(); }
}

extern "C" const char* mho_last_error(void) { return g_err; }
extern "C" int mho_version(void) { return MHO_VERSION; }

extern "C" int mho_create(mho_ctx_t** out, int device) {
    if (!out) { mho_set_error("mho_create: ctx is NULL"); return MHO_ERR_INVALID; }
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
        mho_set_error("mho_create: no CUDA device visible; libmho has no CPU fallback");
        return MHO_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= n) { mho_set_error("mho_create: device %d out of range [0,%d)", device, n); return MHO_ERR_INVALID; }
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        mho_set_error("mho_create: device %d is sm_%d%d; libmho is built for sm_100a only", device, prop.major, prop.minor);
        return MHO_ERR_NO_DEVICE;
    }
    CUDA_TRY(cudaSetDevice(device));
    mho_ctx* c = new mho_ctx();
    c->device = device;
    c->num_sms = prop.multiProcessorCount;
    c->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
    if (cudaMalloc((void**)&c->sched, 2 * sizeof(int)) != cudaSuccess || cudaMemset(c->sched, 0, 2 * sizeof(int)) != cudaSuccess) {
        mho_set_error("mho_create: cudaMalloc for the scheduler state failed");
        delete c;
        return MHO_ERR_CUDA;
    }
    *out = c;
    return MHO_OK;
}

extern "C" int mho_destroy(mho_ctx_t* c) {
    if (!c) return MHO_OK;
    cudaSetDevice(c->device);
    for (auto& s : c->scratch) if (s.ptr) cudaFree(s.ptr);
    for (auto& im : c->img) if (im.ptr) cudaFree(im.ptr);
    if (c->sched) cudaFree(c->sched);
    if (c->h2d_stream) {
        cudaStreamDestroy(c->h2d_stream); cudaStreamDestroy(c->d2h_stream);
        for (int i = 0; i < 2 * MHO_EV_PER_SLOT; ++i) cudaEventDestroy(c->ev[i]);
    }
    delete c;
    return MHO_OK;
}

extern "C" int mho_apsp(mho_ctx_t* c, int32_t n_graphs, const int32_t* node_off, const int32_t* rowptr, const int32_t* colidx,
                        const double* weight, const int64_t* out_off, double* dist, mho_stream_t stream) {
    if (!c || n_graphs < 0 || !node_off || !rowptr || !out_off || !dist) { mho_set_error("mho_apsp: invalid argument"); return MHO_ERR_INVALID; }
    if (n_graphs == 0) return MHO_OK;
    CUDA_TRY(cudaSetDevice(c->device));
    cudaError_t e = apsp_launch(n_graphs, node_off, rowptr, colidx, weight, out_off, dist, c->max_smem_optin, (cudaStream_t)stream);
    if (e != cudaSuccess) { mho_set_error("apsp launch failed: %s", cudaGetErrorString(e)); return MHO_ERR_CUDA; }
    c->launches += 1;
    return MHO_OK;
}

extern "C" int mho_env_step(mho_ctx_t* c, const mho_env_t* nets, const mho_env_items_t* items, const mho_env_out_t* out,
                            mho_stream_t stream) {
    if (!c || !nets || !items || !out) { mho_set_error("mho_env_step: NULL argument"); return MHO_ERR_INVALID; }
    const mho_env_t& E = *nets;
    const mho_env_items_t& I = *items;
    const mho_env_out_t& O = *out;
    if (E.n_nets < 0 || I.n_items < 0 || E.max_nodes < 0 || E.max_links < 0 || I.max_jobs < 0) {
        mho_set_error("mho_env_step: negative count"); return MHO_ERR_INVALID;
    }
    if (I.n_items == 0) return MHO_OK;
    if (E.n_nets == 0 || !E.node_off || !E.link_off || !E.server_off || !E.adj_rowptr || !E.link_rates || !E.cf_degs ||
        !E.proc_bws || !E.cf_rowptr || !E.hop || !E.hop_off || !E.T || !I.net || !I.mode || !I.job_off || !I.sp || !I.sp_off ||
        !O.dst || !O.nhop || !O.delay_est || !O.delay_emp || !O.status) {
        mho_set_error("mho_env_step: a required pointer is NULL"); return MHO_ERR_INVALID;
    }
    if ((O.routes && (!O.routes_off || O.route_stride < E.max_nodes + 1)) || (O.delay_links && !O.links_off) ||
        (O.delay_nodes && !O.nodes_off) || (O.unit && !O.unit_off)) {
        mho_set_error("mho_env_step: an optional output lacks its offsets (or route_stride < max_nodes + 1)"); return MHO_ERR_INVALID;
    }
    if (E.max_nodes > MHO_ENV_MAX_NODES || E.max_links > MHO_ENV_MAX_LINKS || I.max_jobs > MHO_ENV_MAX_JOBS) {
        mho_set_error("mho_env_step: %d nodes / %d links / %d jobs exceed the limits %d / %d / %d", E.max_nodes, E.max_links,
                      I.max_jobs, (int)MHO_ENV_MAX_NODES, (int)MHO_ENV_MAX_LINKS, (int)MHO_ENV_MAX_JOBS);
        return MHO_ERR_TOO_LARGE;
    }
    CUDA_TRY(cudaSetDevice(c->device));
    if (env_step_smem(E.max_nodes, E.max_links, I.max_jobs) > (size_t)c->max_smem_optin) {
        mho_set_error("mho_env_step: shared memory need exceeds the device's limit"); return MHO_ERR_TOO_LARGE;
    }
    cudaError_t e = env_step_launch(E, I, O, (cudaStream_t)stream);
    if (e != cudaSuccess) { mho_set_error("env_step launch failed: %s", cudaGetErrorString(e)); return MHO_ERR_CUDA; }
    c->launches += 1;
    return MHO_OK;
}

extern "C" int mho_host_alloc(void** ptr, size_t bytes) {
    if (!ptr) { mho_set_error("mho_host_alloc: ptr is NULL"); return MHO_ERR_INVALID; }
    *ptr = nullptr;
    CUDA_TRY(cudaHostAlloc(ptr, bytes ? bytes : 1, cudaHostAllocDefault));
    return MHO_OK;
}

extern "C" int mho_host_free(void* ptr) {
    if (ptr) CUDA_TRY(cudaFreeHost(ptr));
    return MHO_OK;
}

extern "C" int64_t mho_launch_count(const mho_ctx_t* c) { return c ? c->launches : 0; }

extern "C" int mho_invalidate_weights(mho_ctx_t* c) {
    if (c) for (auto& im : c->img) im.valid = false;
    return MHO_OK;
}

// grow-only device scratch slots (used by the *_host convenience calls and the backward reducer)
void* mho_scratch(mho_ctx* c, int slot, size_t bytes) {
    if ((int)c->scratch.size() <= slot) c->scratch.resize(slot + 1);
    auto& s = c->scratch[slot];
    if (s.bytes < bytes) {
        if (s.ptr) cudaFree(s.ptr);
        s.ptr = nullptr;
        s.bytes = 0;
        size_t want = bytes + bytes / 4 + 256;
        if (cudaMalloc(&s.ptr, want) != cudaSuccess) { s.ptr = nullptr; return nullptr; }
        s.bytes = want;
    }
    return s.ptr;
}

// ---------------------------------------------------------------------------------------------
extern "C" int mho_plan_tiles(const int32_t* goff, const int32_t* rowptr, int32_t n_graphs, int32_t tile_rows,
                              int32_t* tile_off, int32_t* n_tiles, int32_t* max_rows, int32_t* max_nnz) {
    if (!goff || !rowptr || !tile_off || !n_tiles || !max_rows || !max_nnz || n_graphs < 0 || tile_rows < 1) {
        mho_set_error("mho_plan_tiles: invalid argument");
        return MHO_ERR_INVALID;
    }
    int nt = 0, mr = 0, mz = 0;
    int g = 0;
    tile_off[0] = 0;
    while (g < n_graphs) {
        int start = g;
        int rows = goff[g + 1] - goff[g];
        if (rows > MHO_MAX_TILE_ROWS) {
            mho_set_error("mho_plan_tiles: graph %d has %d nodes; one CTA holds at most %d", g, rows, MHO_MAX_TILE_ROWS);
            return MHO_ERR_TOO_LARGE;
        }
        ++g;
        while (g < n_graphs && (goff[g + 1] - goff[start]) <= tile_rows) ++g;
        rows = goff[g] - goff[start];
        int nnz = rowptr[goff[g]] - rowptr[goff[start]];
        mr = rows > mr ? rows : mr;
        mz = nnz > mz ? nnz : mz;
        tile_off[++nt] = g;
    }
    *n_tiles = nt;
    *max_rows = mr;
    *max_nnz = mz;
    return MHO_OK;
}

extern "C" int mho_fill_tile_info(const int32_t* goff, const int32_t* rowptr, const int32_t* tile_off, int32_t n_tiles,
                                  int32_t* out) {
    if (!goff || !rowptr || !out || n_tiles < 0) { mho_set_error("mho_fill_tile_info: invalid argument"); return MHO_ERR_INVALID; }
    for (int t = 0; t < n_tiles; ++t) {
        const int g0 = tile_off ? tile_off[t] : t, g1 = tile_off ? tile_off[t + 1] : t + 1;
        const int n0 = goff[g0], n1 = goff[g1];
        out[4 * t + 0] = n0; out[4 * t + 1] = n1 - n0; out[4 * t + 2] = rowptr[n0]; out[4 * t + 3] = rowptr[n1] - rowptr[n0];
    }
    return MHO_OK;
}

// ---------------------------------------------------------------------------------------------
int validate_layers(const mho_layer_t* layers, int n_layers, const char* who) {
    if (!layers || n_layers < 1 || n_layers > MHO_MAX_LAYERS) { mho_set_error("%s: n_layers=%d not in [1,%d]", who, n_layers, MHO_MAX_LAYERS); return MHO_ERR_INVALID; }
    for (int l = 0; l < n_layers; ++l) {
        const mho_layer_t& L = layers[l];
        if (L.K < 1 || L.K > MHO_MAX_K || L.f_in < 1 || L.f_in > MHO_MAX_F || L.f_out < 1 || L.f_out > MHO_MAX_F || !L.W ||
            L.act < 0 || L.act > 2) {
            mho_set_error("%s: layer %d invalid (K=%d f_in=%d f_out=%d act=%d W=%p); limits K<=%d F<=%d", who, l, L.K, L.f_in,
                          L.f_out, L.act, (const void*)L.W, MHO_MAX_K, MHO_MAX_F);
            return MHO_ERR_INVALID;
        }
        if (l > 0 && layers[l - 1].f_out != L.f_in) { mho_set_error("%s: layer %d f_in=%d != previous f_out=%d", who, l, L.f_in, layers[l - 1].f_out); return MHO_ERR_INVALID; }
    }
    return MHO_OK;
}

static int validate_batch(const mho_batch_t* b, const char* who) {
    if (!b || b->n_graphs < 0 || !b->graph_off || !b->rowptr || (b->total_nnz > 0 && !b->colidx)) { mho_set_error("%s: invalid batch", who); return MHO_ERR_INVALID; }
    if (b->max_tile_rows < 1 && b->n_graphs > 0) { mho_set_error("%s: batch.max_tile_rows must be set (mho_plan_tiles)", who); return MHO_ERR_INVALID; }
    return MHO_OK;
}

extern "C" int mho_fill_adj_bits(const int32_t* goff, const int32_t* rowptr, const int32_t* colidx, const int32_t* tile_off,
                                 int32_t n_tiles, uint32_t* out) {
    if (!goff || !rowptr || !tile_off || !out || n_tiles < 0) { mho_set_error("mho_fill_adj_bits: invalid argument"); return MHO_ERR_INVALID; }
    for (int t = 0; t < n_tiles; ++t) {
        const int n0 = goff[tile_off[t]], n1 = goff[tile_off[t + 1]];
        if (n1 - n0 > 128) { mho_set_error("mho_fill_adj_bits: tile %d has %d nodes (> 128)", t, n1 - n0); return MHO_ERR_TOO_LARGE; }
        for (int i = n0; i < n1; ++i) {
            uint32_t w[4] = {0u, 0u, 0u, 0u};
            for (int e = rowptr[i]; e < rowptr[i + 1]; ++e) {
                const int c = colidx[e] - n0;
                if (c < 0 || c >= n1 - n0) { mho_set_error("mho_fill_adj_bits: entry (%d,%d) leaves its tile", i, colidx[e]); return MHO_ERR_INVALID; }
                w[c >> 5] |= 1u << (c & 31);
            }
            memcpy(out + (size_t)i * 4, w, sizeof(w));
        }
    }
    return MHO_OK;
}

void mho_fill_layers(const mho_layer_t* layers, int n_layers, int total_nodes, LayerDev* out) {
    long long poff = 0, soff = 0;
    for (int l = 0; l < n_layers; ++l) {
        out[l].K = layers[l].K; out[l].f_in = layers[l].f_in; out[l].f_out = layers[l].f_out;
        out[l].act = layers[l].act; out[l].slope = layers[l].slope;
        out[l].W = layers[l].W; out[l].b = layers[l].b;
        out[l].param_off = poff;
        poff += (long long)layers[l].K * layers[l].f_in * layers[l].f_out + layers[l].f_out;
        out[l].saved_off = 0;
        if (l >= 1) { out[l].saved_off = soff; soff += (long long)total_nodes * layers[l].f_in; }
    }
}

extern "C" int64_t mho_param_count(const mho_layer_t* layers, int32_t n_layers) {
    if (!layers) return 0;
    int64_t p = 0;
    for (int l = 0; l < n_layers; ++l) p += (int64_t)layers[l].K * layers[l].f_in * layers[l].f_out + layers[l].f_out;
    return p;
}

extern "C" size_t mho_saved_bytes(const mho_batch_t* b, const mho_layer_t* layers, int32_t n_layers) {
    if (!b || !layers) return 0;
    size_t s = 0;
    for (int l = 1; l < n_layers; ++l) s += (size_t)b->total_nodes * layers[l].f_in * sizeof(float);
    return s;
}

extern "C" int mho_cheb_forward(mho_ctx_t* c, const mho_batch_t* b, const mho_layer_t* layers, int32_t n_layers,
                                const float* X, float* Y, void* saved, mho_stream_t stream) {
    if (!c) { mho_set_error("mho_cheb_forward: ctx is NULL"); return MHO_ERR_INVALID; }
    dbg_check("mho_cheb_forward entry");
    int rc = validate_batch(b, "mho_cheb_forward");
    if (rc) return rc;
    rc = validate_layers(layers, n_layers, "mho_cheb_forward");
    if (rc) return rc;
    if (b->n_graphs == 0 || b->total_nodes == 0) return MHO_OK;  // empty batch: nothing to do
    if (!X || !Y) { mho_set_error("mho_cheb_forward: X/Y is NULL"); return MHO_ERR_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    FwdParams p;
    memset(&p, 0, sizeof(p));
    p.b.graph_off = b->graph_off; p.b.rowptr = b->rowptr; p.b.colidx = b->colidx; p.b.vals = b->vals;
    p.b.tile_off = b->tile_off; p.b.n_graphs = b->n_graphs;
    p.b.tile_info = b->tile_info;
    p.b.adj_bits = b->adj_bits;
    p.b.tile_graph0 = b->tile_graph0;
    p.b.n_tiles = b->tile_off ? b->n_tiles : b->n_graphs;
    p.n_layers = n_layers;
    mho_fill_layers(layers, n_layers, b->total_nodes, p.layers);
    p.X = X; p.Y = Y; p.saved = (float*)saved; p.total_nodes = b->total_nodes;
    p.sched = c->sched;
    // one 32 -> 32 layer with 2 <= K <= 10 on a binary operator (the benchmark layer): second-generation tensor-core kernel
    if (b->tile_off && b->tile_info &&
        cheb_f16_eligible(layers, n_layers, b->vals != nullptr, b->adj_bits != nullptr, saved != nullptr && n_layers > 1 /* one layer keeps nothing */, b->tile_graph0 != nullptr && b->graph_off != nullptr,
                          b->max_tile_rows, b->max_tile_nnz, X, Y, b->adj_bits, c->max_smem_optin)) {
        auto& img = c->img[MHO_IMG_F16];
        rc = ensure_image(c, img, layers, 1, (size_t)cheb_f16_weight_bytes(layers[0].K), "prepare_f16_weights",
                          [&](unsigned char* out) { return prepare_f16_weights_launch(p.layers[0], out, (cudaStream_t)stream); });
        if (rc) return rc;
        dbg_check("f16 prepared");
        cudaError_t e = cheb_f16_launch(p, img.ptr, b->max_tile_nnz, c->num_sms, c->max_smem_optin, (cudaStream_t)stream);
        dbg_check("f16 launched");
        if (e != cudaSuccess) { mho_set_error("cheb_f16 launch failed: %s", cudaGetErrorString(e)); return MHO_ERR_CUDA; }
        c->launches += 1;
        return MHO_OK;
    }
    // stacks whose layers all have K = 1 (the model the reference ships): fused per-row MLP kernel, fp16 parts
    if (b->tile_off && b->tile_info && cheb_mlp_eligible(layers, n_layers, b->max_tile_rows, X, c->max_smem_optin)) {
        auto& img = c->img[MHO_IMG_MLP];
        rc = ensure_image(c, img, layers, n_layers, (size_t)cheb_mlp_weight_bytes(n_layers), "prepare_mlp_weights",
                          [&](unsigned char* out) { return prepare_mlp_weights_launch(p.layers, n_layers, out, (cudaStream_t)stream); });
        if (rc) return rc;
        cudaError_t e = cheb_mlp_launch(p, img.ptr, c->num_sms, (cudaStream_t)stream);
        if (e != cudaSuccess) { mho_set_error("cheb_mlp launch failed: %s", cudaGetErrorString(e)); return MHO_ERR_CUDA; }
        c->launches += 1;
        return MHO_OK;
    }
    // dense-adjacency tcgen05 path (binary adjacency, tiles <= 128 nodes, <= 32 features per layer, stacks)
    if (b->tile_off && b->tile_info && c->sched &&
        cheb_dense_eligible(layers, n_layers, b->vals != nullptr, b->adj_bits != nullptr, b->max_tile_rows, b->max_tile_nnz, c->max_smem_optin)) {
        auto& img = c->img[MHO_IMG_DENSE];
        int w_off[MHO_MAX_LAYERS];
        const int w_bytes = cheb_dense_weight_bytes(layers, n_layers, w_off);
        rc = ensure_image(c, img, layers, n_layers, (size_t)w_bytes, "prepare_dense_weights",
                          [&](unsigned char* out) { return prepare_dense_weights_launch(p.layers, n_layers, w_off, out, (cudaStream_t)stream); });
        if (rc) return rc;
        cudaError_t e = cheb_dense_launch(p, img.ptr, w_off, w_bytes, b->max_tile_nnz, c->num_sms, (cudaStream_t)stream);
        dbg_check("dense launched");
        if (e != cudaSuccess) { mho_set_error("cheb_dense launch failed: %s", cudaGetErrorString(e)); return MHO_ERR_CUDA; }
        c->launches += 1;
        return MHO_OK;
    }
    int rows = 0;
    for (int l = 0; l < n_layers; ++l) { p.wprep_row_off[l] = rows; rows += wprep_layer_rows(layers[l].K, layers[l].f_out); }
    auto& img = c->img[MHO_IMG_WALK];
    rc = ensure_image(c, img, layers, n_layers, (size_t)rows * 128, "prepare_weights",
                      [&](unsigned char* out) { return prepare_weights_launch(p.layers, n_layers, p.wprep_row_off, out, (cudaStream_t)stream); });
    if (rc) return rc;
    p.wprep = img.ptr;
    bool too_large = false;
    cudaError_t e = cheb_forward_launch(p, b->max_tile_rows, b->max_tile_nnz, c->num_sms, c->max_smem_optin,
                                        (cudaStream_t)stream, &too_large);
    if (too_large) {
        mho_set_error("mho_cheb_forward: tile of %d rows / K up to %d does not fit in %d B of shared memory", b->max_tile_rows,
                      MHO_MAX_K, c->max_smem_optin);
        return MHO_ERR_TOO_LARGE;
    }
    if (e != cudaSuccess) { mho_set_error("cheb_forward launch failed: %s", cudaGetErrorString(e)); return MHO_ERR_CUDA; }
    c->launches += 1;
    return MHO_OK;
}

// ---------------------------------------------------------------------------------------------
// Host-buffer convenience: numpy in / numpy out, like ACOAgent.predict (gnn_offloading_agent.py:144-150)
// ---------------------------------------------------------------------------------------------
// The call is pipelined over chunks of the batch on three streams - uploads, kernels (the caller's stream),
// downloads - so PCIe in, compute and PCIe out overlap; with pinned host buffers the step costs about
// max(H2D, D2H) instead of their sum.  Global node / nnz offsets are kept (tile_info carries them), so a
// chunk is just a slice of every array uploaded to its final place.
// Two calls may be in flight (mho_cheb_forward_host_async): each uses one of two device staging slots, so the upload
// of call i+1 runs while call i computes and downloads - both PCIe directions busy at once.
static int forward_host_impl(mho_ctx_t* c, int32_t n_graphs, const int32_t* goff_h, const int32_t* rowptr_h,
                             const int32_t* colidx_h, const float* vals_h, const mho_layer_t* layers,
                             int32_t n_layers, const float* X_h, float* Y_h, mho_stream_t stream, bool sync, int32_t* ticket) {
    if (!c || !goff_h || !rowptr_h || !X_h || !Y_h || n_graphs < 0) { mho_set_error("mho_cheb_forward_host: invalid argument"); return MHO_ERR_INVALID; }
    if (ticket) *ticket = -1;
    int rc = validate_layers(layers, n_layers, "mho_cheb_forward_host");
    if (rc) return rc;
    if (n_graphs == 0) return MHO_OK;
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int total_nodes = goff_h[n_graphs];
    const int64_t nnz = rowptr_h[total_nodes];
    if (total_nodes == 0) return MHO_OK;
    if (nnz > 0 && !colidx_h) { mho_set_error("mho_cheb_forward_host: colidx is NULL"); return MHO_ERR_INVALID; }
    std::vector<int32_t> tile_off((size_t)n_graphs + 1);
    int32_t n_tiles = 0, mr = 0, mz = 0;
    std::vector<int32_t> tinfo;
    bool all_k1 = true;
    for (int l = 0; l < n_layers; ++l) all_k1 = all_k1 && layers[l].K == 1 && layers[l].f_in <= 32 && layers[l].f_out <= 32;
    if (all_k1) {
        // no layer touches the operator: full 128-node row tiles that ignore graph boundaries, whatever the graph sizes
        n_tiles = (total_nodes + 127) / 128;
        tinfo.resize((size_t)n_tiles * 4 + 4);
        for (int t = 0; t < n_tiles; ++t) {
            const int a = 128 * t, b2 = std::min(a + 128, total_nodes);
            tinfo[4 * t] = a; tinfo[4 * t + 1] = b2 - a; tinfo[4 * t + 2] = rowptr_h[a]; tinfo[4 * t + 3] = rowptr_h[b2] - rowptr_h[a];
            mz = std::max(mz, tinfo[4 * t + 3]);
        }
        mr = std::min(128, total_nodes);
    } else {
        rc = mho_plan_tiles(goff_h, rowptr_h, n_graphs, 128, tile_off.data(), &n_tiles, &mr, &mz);
        if (rc) return rc;
        tinfo.resize((size_t)n_tiles * 4 + 4);
        mho_fill_tile_info(goff_h, rowptr_h, tile_off.data(), n_tiles, tinfo.data());
    }

    // chunks: contiguous runs of tiles of roughly equal bytes, ~300 tiles each (measured: copies of a few MB keep both
    // PCIe directions efficient; 2 chunks beat 1, 3 and 4 for the 594-tile benchmark batch), at most 8 chunks
    int n_chunks = (n_tiles + 150) / 300;
    if (n_chunks > n_tiles) n_chunks = n_tiles;
    if (n_chunks < 1) n_chunks = 1;
    if (n_chunks > 8) n_chunks = 8;
    std::vector<int> cstart((size_t)n_chunks + 1, 0);
    {
        const long long total_cost = 64LL * total_nodes + 2LL * nnz;
        int t = 0;
        for (int k = 1; k < n_chunks; ++k) {
            const long long target = total_cost * k / n_chunks;
            while (t < n_tiles && 64LL * tinfo[4 * t] + 2LL * tinfo[4 * t + 2] < target) ++t;
            cstart[k] = t;
        }
        cstart[n_chunks] = n_tiles;
    }
    // node extent of each chunk (its tiles are a contiguous run of nodes), taken before the tiles are reordered
    std::vector<int> cn0((size_t)n_chunks), cn1((size_t)n_chunks);
    for (int k = 0; k < n_chunks; ++k) {
        cn0[k] = tinfo[4 * (size_t)cstart[k]];
        cn1[k] = cstart[k + 1] > cstart[k] ? tinfo[4 * (size_t)(cstart[k + 1] - 1)] + tinfo[4 * (size_t)(cstart[k + 1] - 1) + 1] : cn0[k];
    }
    // inside every chunk: largest tile first for the kernel's dynamic scheduler (tinfo is consumed in order); the index of
    // each tile's first graph travels with it (per-graph operand scales of the fp16 tensor-core kernel)
    std::vector<int32_t> tgraph0;
    if (!all_k1) {
        struct T5 { int32_t v[4]; int32_t g0; };
        std::vector<T5> tt((size_t)n_tiles);
        for (int t = 0; t < n_tiles; ++t) { memcpy(tt[t].v, &tinfo[4 * (size_t)t], 16); tt[t].g0 = tile_off[t]; }
        for (int k = 0; k < n_chunks; ++k)
            std::stable_sort(tt.begin() + cstart[k], tt.begin() + cstart[k + 1],
                             [](const T5& a, const T5& b) { return 3LL * a.v[1] + a.v[3] > 3LL * b.v[1] + b.v[3]; });
        tgraph0.resize((size_t)n_tiles + 4);
        for (int t = 0; t < n_tiles; ++t) { memcpy(&tinfo[4 * (size_t)t], tt[t].v, 16); tgraph0[t] = tt[t].g0; }
    } else {
        for (int k = 0; k < n_chunks; ++k) {
            struct T4 { int32_t v[4]; };
            T4* beg = reinterpret_cast<T4*>(tinfo.data()) + cstart[k];
            T4* end = reinterpret_cast<T4*>(tinfo.data()) + cstart[k + 1];
            std::stable_sort(beg, end, [](const T4& a, const T4& b) { return 3LL * a.v[1] + a.v[3] > 3LL * b.v[1] + b.v[3]; });
        }
    }

    const int f_in = layers[0].f_in, f_out = layers[n_layers - 1].f_out;
    const size_t b_rp = (size_t)(total_nodes + 1) * 4, b_ci = (size_t)nnz * 4;
    const size_t b_va = vals_h ? (size_t)nnz * 4 : 0, b_ti = (size_t)n_tiles * 16 + 16;
    const size_t b_go = tgraph0.empty() ? 0 : (size_t)(n_graphs + 1) * 4, b_tg = tgraph0.empty() ? 0 : (size_t)n_tiles * 4 + 16;
    const size_t b_x = (size_t)total_nodes * f_in * 4, b_y = (size_t)total_nodes * f_out * 4;
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t total = al(b_rp) + al(b_ci) + al(b_va) + al(b_ti) + al(b_go) + al(b_tg) + al(b_x) + al(b_y);
    const int slot = (int)(c->host_calls & 1);
    c->host_calls += 1;
    // an error return below leaves uploads / kernels of this call in flight on the slot's buffers: drain the three streams
    // before returning so that the next call that recycles the slot cannot overwrite them (the ticket stays -1)
    struct DrainOnError {
        mho_ctx* c; cudaStream_t st; bool armed;
        ~DrainOnError() {
            if (!armed) return;
            if (c->h2d_stream) cudaStreamSynchronize(c->h2d_stream);
            cudaStreamSynchronize(st);
            if (c->d2h_stream) cudaStreamSynchronize(c->d2h_stream);
        }
    } drain{c, st, true};
    if (!c->h2d_stream) {
        CUDA_TRY(cudaStreamCreateWithFlags(&c->h2d_stream, cudaStreamNonBlocking));
        CUDA_TRY(cudaStreamCreateWithFlags(&c->d2h_stream, cudaStreamNonBlocking));
        for (int i = 0; i < 2 * MHO_EV_PER_SLOT; ++i) CUDA_TRY(cudaEventCreateWithFlags(&c->ev[i], cudaEventDisableTiming));
    }
    cudaEvent_t* ev = c->ev + slot * MHO_EV_PER_SLOT;
    cudaEvent_t ev_done = ev[2 * MHO_MAX_CHUNKS + 1];
    // the slot's previous user (two calls ago) must have finished its downloads before the buffers are recycled;
    // growing the slot frees device memory, which waits for the device anyway
    if (c->slot_used[slot]) CUDA_TRY(cudaEventSynchronize(ev_done));
    char* base = (char*)mho_scratch(c, slot == 0 ? 0 : 4, total);
    if (!base) { mho_set_error("mho_cheb_forward_host: cudaMalloc of %zu B failed", total); return MHO_ERR_CUDA; }
    char* q = base;
    int32_t* d_rp = (int32_t*)q; q += al(b_rp);
    int32_t* d_ci = (int32_t*)q; q += al(b_ci);
    float* d_va = vals_h ? (float*)q : nullptr; q += al(b_va);
    int32_t* d_ti = (int32_t*)q; q += al(b_ti);
    int32_t* d_go = b_go ? (int32_t*)q : nullptr; q += al(b_go);
    int32_t* d_tg = b_tg ? (int32_t*)q : nullptr; q += al(b_tg);
    float* d_x = (float*)q; q += al(b_x);
    float* d_y = (float*)q;

    cudaStream_t sh = c->h2d_stream, sd = c->d2h_stream;
    // uploads may start as soon as the slot is free (checked above): they do NOT wait for the caller's stream, whose
    // pending work is the other slot's kernels
    if (d_go) {
        // tile descriptors, graph offsets and first-graph indices are adjacent on the device: ONE staged (pageable) copy
        std::vector<int32_t> meta((al(b_ti) + al(b_go) + al(b_tg)) / 4, 0);
        memcpy(meta.data(), tinfo.data(), (size_t)n_tiles * 16);
        memcpy(meta.data() + al(b_ti) / 4, goff_h, b_go);
        memcpy(meta.data() + (al(b_ti) + al(b_go)) / 4, tgraph0.data(), (size_t)n_tiles * 4);
        CUDA_TRY(cudaMemcpyAsync(d_ti, meta.data(), meta.size() * 4, cudaMemcpyHostToDevice, sh));  // pageable: returns after staging
    } else {
        CUDA_TRY(cudaMemcpyAsync(d_ti, tinfo.data(), (size_t)n_tiles * 16, cudaMemcpyHostToDevice, sh));  // pageable: returns after staging
    }

    // node / nnz extent of each chunk (tiles of a chunk are a contiguous run of graphs)
    auto chunk_nodes = [&](int k, int& n0, int& n1) { n0 = cn0[k]; n1 = cn1[k]; };
    for (int k = 0; k < n_chunks; ++k) {
        int n0, n1;
        chunk_nodes(k, n0, n1);
        const int64_t z0 = rowptr_h[n0], z1 = rowptr_h[n1];
        CUDA_TRY(cudaMemcpyAsync(d_rp + n0, rowptr_h + n0, (size_t)(n1 - n0 + 1) * 4, cudaMemcpyHostToDevice, sh));
        if (z1 > z0) CUDA_TRY(cudaMemcpyAsync(d_ci + z0, colidx_h + z0, (size_t)(z1 - z0) * 4, cudaMemcpyHostToDevice, sh));
        if (vals_h && z1 > z0) CUDA_TRY(cudaMemcpyAsync(d_va + z0, vals_h + z0, (size_t)(z1 - z0) * 4, cudaMemcpyHostToDevice, sh));
        CUDA_TRY(cudaMemcpyAsync(d_x + (size_t)n0 * f_in, X_h + (size_t)n0 * f_in, (size_t)(n1 - n0) * f_in * 4, cudaMemcpyHostToDevice, sh));
        CUDA_TRY(cudaEventRecord(ev[k], sh));

        CUDA_TRY(cudaStreamWaitEvent(st, ev[k], 0));
        mho_batch_t b;
        memset(&b, 0, sizeof(b));
        b.n_graphs = n_graphs; b.total_nodes = total_nodes; b.total_nnz = nnz;
        b.graph_off = d_go ? d_go : (const int32_t*)d_rp;  // dereferenced only together with tile_graph0
        b.tile_graph0 = d_tg ? d_tg + cstart[k] : nullptr;
        b.rowptr = d_rp; b.colidx = d_ci; b.vals = d_va;
        b.tile_off = (const int32_t*)d_ti;   // non-NULL marks "tiled"; bounds again come from tile_info
        b.tile_info = d_ti + 4 * (size_t)cstart[k];
        b.n_tiles = cstart[k + 1] - cstart[k]; b.max_tile_rows = mr; b.max_tile_nnz = mz;
        if (b.n_tiles > 0) {
            rc = mho_cheb_forward(c, &b, layers, n_layers, d_x, d_y, nullptr, stream);
            if (rc) return rc;
        }
        CUDA_TRY(cudaEventRecord(ev[MHO_MAX_CHUNKS + k], st));
        CUDA_TRY(cudaStreamWaitEvent(sd, ev[MHO_MAX_CHUNKS + k], 0));
        CUDA_TRY(cudaMemcpyAsync(Y_h + (size_t)n0 * f_out, d_y + (size_t)n0 * f_out, (size_t)(n1 - n0) * f_out * 4, cudaMemcpyDeviceToHost, sd));
    }
    CUDA_TRY(cudaEventRecord(ev_done, sd));
    drain.armed = false;
    c->slot_used[slot] = true;
    if (ticket) *ticket = slot;
    if (sync) {
        CUDA_TRY(cudaEventSynchronize(ev_done));
        CUDA_TRY(cudaStreamSynchronize(st));
    }
    return MHO_OK;
}

extern "C" int mho_cheb_forward_host(mho_ctx_t* c, int32_t n_graphs, const int32_t* goff_h, const int32_t* rowptr_h,
                                     const int32_t* colidx_h, const float* vals_h, const mho_layer_t* layers,
                                     int32_t n_layers, const float* X_h, float* Y_h, mho_stream_t stream) {
    return forward_host_impl(c, n_graphs, goff_h, rowptr_h, colidx_h, vals_h, layers, n_layers, X_h, Y_h, stream, true, nullptr);
}

extern "C" int mho_cheb_forward_host_async(mho_ctx_t* c, int32_t n_graphs, const int32_t* goff_h, const int32_t* rowptr_h,
                                           const int32_t* colidx_h, const float* vals_h, const mho_layer_t* layers,
                                           int32_t n_layers, const float* X_h, float* Y_h, mho_stream_t stream, int32_t* ticket) {
    if (!ticket) { mho_set_error("mho_cheb_forward_host_async: ticket is NULL"); return MHO_ERR_INVALID; }
    return forward_host_impl(c, n_graphs, goff_h, rowptr_h, colidx_h, vals_h, layers, n_layers, X_h, Y_h, stream, false, ticket);
}

extern "C" int mho_host_wait(mho_ctx_t* c, int32_t ticket) {
    if (!c || ticket < 0 || ticket > 1) { mho_set_error("mho_host_wait: invalid ticket"); return MHO_ERR_INVALID; }
    if (!c->slot_used[ticket]) return MHO_OK;
    CUDA_TRY(cudaSetDevice(c->device));
    CUDA_TRY(cudaEventSynchronize(c->ev[ticket * MHO_EV_PER_SLOT + 2 * MHO_MAX_CHUNKS + 1]));
    return MHO_OK;
}
