// Internal (non-ABI) declarations shared by the libmho translation units.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <vector>

#include "../../include/mho.h"

struct mho_scratch_slot {
    void* ptr = nullptr;
    size_t bytes = 0;
};

struct mho_wkey {
    const void* W; const void* b; int K, f_in, f_out;
    bool operator==(const mho_wkey& o) const { return W == o.W && b == o.b && K == o.K && f_in == o.f_in && f_out == o.f_out; }
};

// A kernel family's device image of the weights of a layer stack (split / transposed / padded parts, bias).
// Cached under the stack's weight pointers and shapes; mho_invalidate_weights drops every image, because the
// optimizer rewrites the weights in place.
struct mho_wimage {
    std::vector<mho_wkey> key;
    bool valid = false;
    unsigned char* ptr = nullptr;
    size_t bytes = 0;
};
enum { MHO_IMG_WALK, MHO_IMG_DENSE, MHO_IMG_F16, MHO_IMG_MLP, MHO_IMG_MLP_BWD, MHO_N_IMAGES };

#define MHO_MAX_CHUNKS 8
#define MHO_EV_PER_SLOT (2 * MHO_MAX_CHUNKS + 2)   // per staging slot: upload / kernel events per chunk, start, done

struct mho_ctx {
    // pipelined host call: upload / download streams and per-chunk events
    cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr;
    cudaEvent_t ev[2 * MHO_EV_PER_SLOT] = {};
    int64_t host_calls = 0;          // host-buffer calls so far: call i uses staging slot i & 1
    bool slot_used[2] = {false, false};
    // prepared weights: TF32 hi/lo images of the CSR-walk kernel (cheb_forward.cu), bf16 parts of the dense-adjacency
    // kernel (cheb_forward_dense.cu), fp16 parts of the one-layer tensor-core kernel (cheb_forward_f16.cu), fp16 images
    // of the fused K = 1 stack kernel (cheb_mlp_f16.cu) and fp16 W^T images of its VJP (cheb_mlp_backward_f16.cu)
    mho_wimage img[MHO_N_IMAGES];
    int* sched = nullptr;  // two zero-initialised ints: dynamic tile scheduler state (self re-arming)
    int device = 0;
    int num_sms = 0;
    int max_smem_optin = 0;
    int64_t launches = 0;
    std::vector<mho_scratch_slot> scratch;
};

void mho_set_error(const char* fmt, ...);
void* mho_scratch(mho_ctx* c, int slot, size_t bytes);
int validate_layers(const mho_layer_t* layers, int n_layers, const char* who);

// Make `img` hold the image of `layers` (n_layers entries), `bytes` long: unless it was built from the same stack,
// (re)allocate it and enqueue prep(img.ptr), which counts as one launch.  `what` names the prep launch in errors.
template <class Prep>
int ensure_image(mho_ctx* c, mho_wimage& img, const mho_layer_t* layers, int n_layers, size_t bytes, const char* what, Prep prep) {
    bool same = img.valid && (int)img.key.size() == n_layers;
    for (int l = 0; same && l < n_layers; ++l)
        same = img.key[l] == mho_wkey{layers[l].W, layers[l].b, layers[l].K, layers[l].f_in, layers[l].f_out};
    if (same) return MHO_OK;
    img.valid = false;
    if (bytes > img.bytes) {
        if (img.ptr) cudaFree(img.ptr);
        img.ptr = nullptr; img.bytes = 0;
        if (cudaMalloc((void**)&img.ptr, bytes) != cudaSuccess) { mho_set_error("cudaMalloc(%zu) for prepared weights failed", bytes); return MHO_ERR_CUDA; }
        img.bytes = bytes;
    }
    const cudaError_t e = prep(img.ptr);
    if (e != cudaSuccess) { mho_set_error("%s launch failed: %s", what, cudaGetErrorString(e)); return MHO_ERR_CUDA; }
    c->launches += 1;
    img.key.clear();
    for (int l = 0; l < n_layers; ++l) img.key.push_back(mho_wkey{layers[l].W, layers[l].b, layers[l].K, layers[l].f_in, layers[l].f_out});
    img.valid = true;
    return MHO_OK;
}

struct LayerDev;
struct FwdParams;
void mho_fill_layers(const mho_layer_t* layers, int n_layers, int total_nodes, LayerDev* out);
int wprep_layer_rows(int K, int f_out);
cudaError_t prepare_weights_launch(const LayerDev* layers, int n_layers, const int* row_off, unsigned char* out,
                                   cudaStream_t st);
bool cheb_dense_eligible(const mho_layer_t* layers, int n_layers, bool has_vals, bool has_bits, int max_tile_rows, int max_tile_nnz,
                         int max_smem_optin);
int cheb_dense_weight_bytes(const mho_layer_t* layers, int n_layers, int* w_off);
cudaError_t prepare_dense_weights_launch(const LayerDev* layers, int n_layers, const int* w_off, unsigned char* out, cudaStream_t st);
cudaError_t cheb_dense_launch(const FwdParams& fp, const unsigned char* wimg, const int* w_off, int w_bytes, int max_tile_nnz,
                              int num_sms, cudaStream_t st);
bool cheb_f16_eligible(const mho_layer_t* layers, int n_layers, bool has_vals, bool has_bits, bool has_saved, bool has_graph_starts,
                       int max_tile_rows, int max_tile_nnz, const void* X, const void* Y, const void* bits, int max_smem_optin);
int cheb_f16_weight_bytes(int K);
cudaError_t prepare_f16_weights_launch(const LayerDev& L, unsigned char* out, cudaStream_t st);
cudaError_t cheb_f16_launch(const FwdParams& fp, const unsigned char* wimg, int max_tile_nnz, int num_sms, int max_smem_optin, cudaStream_t st);
bool cheb_mlp_eligible(const mho_layer_t* layers, int n_layers, int max_tile_rows, const void* X, int max_smem_optin);
int cheb_mlp_weight_bytes(int n_layers);
cudaError_t prepare_mlp_weights_launch(const LayerDev* layers, int n_layers, unsigned char* out, cudaStream_t st);
cudaError_t cheb_mlp_launch(const FwdParams& fp, const unsigned char* wimg, int num_sms, cudaStream_t st);
bool cheb_backward_f16_eligible(const mho_batch_t* b, const mho_layer_t* layers, int n_layers, const void* X, const void* Y, const void* dY,
                                const void* dX, int max_smem_optin);
cudaError_t cheb_backward_f16_launch(const mho_batch_t* b, const mho_layer_t* layers, const float* X, const float* Y, const float* dY,
                                     float* grads, long long n_params, int num_sms, cudaStream_t st);
bool cheb_mlp_backward_eligible(const mho_batch_t* b, const mho_layer_t* layers, int n_layers, const void* X, const void* saved, const void* dX,
                                int max_smem_optin);
int cheb_mlp_backward_weight_bytes(int n_layers);
cudaError_t prepare_mlp_backward_weights_launch(const LayerDev* layers, int n_layers, unsigned char* out, cudaStream_t st);
cudaError_t cheb_mlp_backward_launch(const mho_batch_t* b, const LayerDev* layers, int n_layers, const float* X, const float* Y, const float* saved,
                                     const float* dY, float* grads, long long n_params, const unsigned char* wT, int num_sms, cudaStream_t st);
cudaError_t apsp_launch(int n_graphs, const int32_t* node_off, const int32_t* rowptr, const int32_t* colidx, const double* weight,
                        const int64_t* out_off, double* dist, int max_smem_optin, cudaStream_t st);
size_t env_step_smem(int max_nodes, int max_links, int max_jobs);
cudaError_t env_step_launch(const mho_env_t& nets, const mho_env_items_t& items, const mho_env_out_t& out, cudaStream_t st);
cudaError_t cheb_forward_launch(FwdParams& p, int max_tile_rows, int max_tile_nnz, int num_sms, int max_smem_optin,
                                cudaStream_t st, bool* too_large);
