// Sequential gradient replay with Keras-2 Adam(clipnorm) + max_norm constraints, one launch.
//
// Replaces the Python loop of ACOAgent.replay (src/gnn_offloading_agent.py:156-169):
//     for grad, loss, _ in minibatch: self.optimizer.apply_gradients(zip(grad, weights))
// with optimizer = Adam(lr, clipnorm=1.0) (:114-121) and kernel/bias_constraint=max_norm(1.0)
// (:104-108).  Semantics [upstream Keras-2 optimizer_v2.Adam, keras.constraints.MaxNorm]:
//   per TENSOR: g <- g * clipnorm / max(||g||_2, clipnorm)
//   m <- b1 m + (1-b1) g ; v <- b2 v + (1-b2) g^2 ; w <- w - lr_t m / (sqrt(v) + eps),
//   lr_t = lr(step) * sqrt(1-b2^t) / (1-b1^t), t = step+1 ; lr(step) = lr * decay_rate^(step/decay_steps)
//   then w <- w * clip(||w||_axis0, 0, max_norm) / (1e-7 + ||w||_axis0)   (axis 0 = the K axis of a kernel,
//   the whole vector for a bias).
// The reference runs in fp64; master weights and moments are kept in fp64 here too (updates of
// lr=1e-6 would drown in fp32), and an fp32 copy is emitted for the forward/backward kernels.
// One CTA: the 100 steps are inherently sequential and the model is 3k-16k parameters.
#include "mho_common.cuh"
#include "mho_internal.h"

#define OPT_THREADS 1024

struct OptTensor {
    long long off;   // offset in the flat parameter vector
    int K, fi, fo;   // kernel: [K, fi, fo]; bias: K = 0, fi = 1, fo = length
};

struct OptParams {
    int n_tensors;
    OptTensor t[2 * MHO_MAX_LAYERS];
    double lr, b1, b2, eps, clipnorm, max_norm, decay_rate;
    int decay_steps;
    double* w;
    double* m;
    double* v;
    float* w32;
    const float* grads;
    long long n_params;
    int n_steps;
    long long step0;
};

__device__ __forceinline__ double block_sum(double x, double* red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    __syncthreads();  // protect `red` from the previous use
    if (lane == 0) red[warp] = x;
    __syncthreads();
    double s = 0.0;
#pragma unroll 1
    for (int i = 0; i < OPT_THREADS / 32; ++i) s += red[i];  // same order in every thread: deterministic
    return s;
}

__global__ void __launch_bounds__(OPT_THREADS, 1) adam_replay_kernel(const __grid_constant__ OptParams p) {
    __shared__ double red[OPT_THREADS / 32];
    const int tid = threadIdx.x;
    for (int s = 0; s < p.n_steps; ++s) {
        const float* g = p.grads + (size_t)s * p.n_params;
        const long long step = p.step0 + s;
        const double t = (double)(step + 1);
        const double lr = (p.decay_rate == 1.0) ? p.lr : p.lr * pow(p.decay_rate, (double)step / (double)p.decay_steps);
        const double alpha = lr * sqrt(1.0 - pow(p.b2, t)) / (1.0 - pow(p.b1, t));
        for (int ti = 0; ti < p.n_tensors; ++ti) {
            const OptTensor T = p.t[ti];
            const int n = (T.K > 0 ? T.K : 1) * T.fi * T.fo;
            double ss = 0.0;
            for (int i = tid; i < n; i += OPT_THREADS) { const double gi = (double)g[T.off + i]; ss += gi * gi; }
            double scale = 1.0;
            if (p.clipnorm > 0.0) {
                const double nrm = sqrt(block_sum(ss, red));
                scale = p.clipnorm / fmax(nrm, p.clipnorm);
            }
            for (int i = tid; i < n; i += OPT_THREADS) {
                const double gi = (double)g[T.off + i] * scale;
                const double mi = p.b1 * p.m[T.off + i] + (1.0 - p.b1) * gi;
                const double vi = p.b2 * p.v[T.off + i] + (1.0 - p.b2) * gi * gi;
                p.m[T.off + i] = mi;
                p.v[T.off + i] = vi;
                p.w[T.off + i] -= alpha * mi / (sqrt(vi) + p.eps);
            }
            if (p.max_norm > 0.0) {
                __syncthreads();  // the update above wrote w with a different thread->element mapping
                if (T.K > 0) {  // kernel: norm over the K axis for every (f, o); each thread owns its columns
                    const int cols = T.fi * T.fo;
                    for (int c = tid; c < cols; c += OPT_THREADS) {
                        double q = 0.0;
                        for (int k = 0; k < T.K; ++k) { const double x = p.w[T.off + (size_t)k * cols + c]; q += x * x; }
                        const double nr = sqrt(q);
                        const double f = fmin(fmax(nr, 0.0), p.max_norm) / (1e-7 + nr);
                        for (int k = 0; k < T.K; ++k) p.w[T.off + (size_t)k * cols + c] *= f;
                    }
                } else {  // bias: norm of the whole vector
                    double q = 0.0;
                    for (int i = tid; i < n; i += OPT_THREADS) { const double x = p.w[T.off + i]; q += x * x; }
                    const double nr = sqrt(block_sum(q, red));
                    const double f = fmin(fmax(nr, 0.0), p.max_norm) / (1e-7 + nr);
                    for (int i = tid; i < n; i += OPT_THREADS) p.w[T.off + i] *= f;
                }
            }
        }
        __syncthreads();
    }
    __syncthreads();
    for (long long i = tid; i < p.n_params; i += OPT_THREADS) p.w32[i] = (float)p.w[i];
}

extern "C" int mho_adam_replay(mho_ctx_t* c, const mho_layer_t* layers, int32_t n_layers, const mho_adam_t* cfg,
                               double* params, double* m, double* v, float* params_f32, const float* grads,
                               int32_t n_steps, int64_t step_count, mho_stream_t stream) {
    if (!c || !layers || !cfg || !params || !m || !v || !params_f32 || n_layers < 1 || n_layers > MHO_MAX_LAYERS || n_steps < 0 ||
        (n_steps > 0 && !grads)) {
        mho_set_error("mho_adam_replay: invalid argument");
        return MHO_ERR_INVALID;
    }
    if (cudaSetDevice(c->device) != cudaSuccess) { mho_set_error("cudaSetDevice failed"); return MHO_ERR_CUDA; }
    OptParams p;
    memset(&p, 0, sizeof(p));
    long long off = 0;
    for (int l = 0; l < n_layers; ++l) {
        const mho_layer_t& L = layers[l];
        if (L.K < 1 || L.f_in < 1 || L.f_out < 1) { mho_set_error("mho_adam_replay: layer %d invalid", l); return MHO_ERR_INVALID; }
        p.t[2 * l] = {off, L.K, L.f_in, L.f_out};
        off += (long long)L.K * L.f_in * L.f_out;
        p.t[2 * l + 1] = {off, 0, 1, L.f_out};
        off += L.f_out;
    }
    p.n_tensors = 2 * n_layers;
    p.n_params = off;
    p.lr = cfg->lr; p.b1 = cfg->beta1; p.b2 = cfg->beta2; p.eps = cfg->eps; p.clipnorm = cfg->clipnorm; p.max_norm = cfg->max_norm;
    p.decay_rate = cfg->decay_rate; p.decay_steps = cfg->decay_steps > 0 ? cfg->decay_steps : 1;
    p.w = params; p.m = m; p.v = v; p.w32 = params_f32; p.grads = grads; p.n_steps = n_steps; p.step0 = step_count;
    adam_replay_kernel<<<1, OPT_THREADS, 0, (cudaStream_t)stream>>>(p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { mho_set_error("adam_replay launch failed: %s", cudaGetErrorString(e)); return MHO_ERR_CUDA; }
    c->launches += 1;
    mho_invalidate_weights(c);  // params_f32 changed in place: the packed weight images are stale
    return MHO_OK;
}
