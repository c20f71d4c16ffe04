// Queue-model head that follows the GNN (SURVEY 8f, "next" row 1), fused and batched, fp64 like the reference.
//
// Replaces the TensorFlow op chain of ACOAgent.forward, src/gnn_offloading_agent.py:231-254
//   link_lambda = gather(lambda, maps_ol_el); node_lambda = gather(lambda, maps_on_el)
//   link_mu = rates / (cf_degs + 1);  10x: link_mu = rates / (1 + A_i clip(link_lambda / link_mu, 0, 1))
//   delay = 1 / (mu - lambda);  congested (lambda > mu): T * lambda / (101 mu) links, T * lambda / (100 mu) nodes
// and its VJP (the part of g.gradient(...), :448, between the delay matrix and the GNN output), which
// differentiates through all ten fixed-point iterations like the tape does.
// One CTA per graph instance; everything of a graph (L <= a few hundred links) lives in shared memory.
// A_i (conflict graph of the links, env.adj_i) is symmetric (undirected line graph); the backward relies on it.
#include "mho_common.cuh"
#include "mho_internal.h"

#define QH_THREADS 256
#define QH_ITERS 10

struct HeadDev {
    int n_graphs;
    const int32_t* ext_off;
    const int32_t* link_off;
    const int32_t* comp_off;
    const int32_t* maps_ol_el;
    const int32_t* maps_on_el;
    const double* link_rates;
    const double* cf_degs;
    const double* node_mu;
    const int32_t* adj_rowptr;
    const int32_t* adj_colidx;
    double T;
};

__global__ void __launch_bounds__(QH_THREADS) queue_head_forward_kernel(HeadDev h, const float* __restrict__ lam,
                                                                        double* __restrict__ link_delay,
                                                                        double* __restrict__ node_delay,
                                                                        double* __restrict__ saved_mu, long long total_links) {
    extern __shared__ double sm[];
    for (int g = blockIdx.x; g < h.n_graphs; g += gridDim.x) {
        const int l0 = h.link_off[g], L = h.link_off[g + 1] - l0;
        const int c0 = h.comp_off[g], NC = h.comp_off[g + 1] - c0;
        const int e0 = h.ext_off[g];
        double* ll = sm;          // [L]
        double* mu = sm + L;      // [L]
        double* busy = sm + 2 * L;  // [L]
        __syncthreads();
        for (int i = threadIdx.x; i < L; i += QH_THREADS) {
            ll[i] = (double)lam[e0 + h.maps_ol_el[l0 + i]];
            const double m0 = h.link_rates[l0 + i] / (h.cf_degs[l0 + i] + 1.0);
            mu[i] = m0;
            if (saved_mu) saved_mu[(size_t)l0 + i] = m0;
        }
        __syncthreads();
        for (int it = 0; it < QH_ITERS; ++it) {
            for (int i = threadIdx.x; i < L; i += QH_THREADS) busy[i] = fmin(fmax(ll[i] / mu[i], 0.0), 1.0);
            __syncthreads();
            for (int i = threadIdx.x; i < L; i += QH_THREADS) {
                double s = 0.0;
                const int a = h.adj_rowptr[l0 + i], b = h.adj_rowptr[l0 + i + 1];
                for (int e = a; e < b; ++e) s += busy[h.adj_colidx[e]];
                const double m = h.link_rates[l0 + i] * (1.0 / (1.0 + s));
                mu[i] = m;
                if (saved_mu) saved_mu[(size_t)(it + 1) * total_links + l0 + i] = m;
            }
            __syncthreads();
        }
        for (int i = threadIdx.x; i < L; i += QH_THREADS) {
            const double l = ll[i], m = mu[i];
            link_delay[l0 + i] = (l - m) > 0.0 ? h.T * (l / (101.0 * m)) : 1.0 / (m - l);
        }
        for (int i = threadIdx.x; i < NC; i += QH_THREADS) {
            const double l = (double)lam[e0 + h.maps_on_el[c0 + i]], m = h.node_mu[c0 + i];
            node_delay[c0 + i] = (l - m) > 0.0 ? h.T * (l / (100.0 * m)) : 1.0 / (m - l);
        }
    }
}

__global__ void __launch_bounds__(QH_THREADS) queue_head_backward_kernel(HeadDev h, const float* __restrict__ lam,
                                                                         const double* __restrict__ saved_mu,
                                                                         const double* __restrict__ g_link,
                                                                         const double* __restrict__ g_node,
                                                                         float* __restrict__ g_lam, long long total_links) {
    extern __shared__ double sm[];
    for (int g = blockIdx.x; g < h.n_graphs; g += gridDim.x) {
        const int l0 = h.link_off[g], L = h.link_off[g + 1] - l0;
        const int c0 = h.comp_off[g], NC = h.comp_off[g + 1] - c0;
        const int e0 = h.ext_off[g], NE = h.ext_off[g + 1] - e0;
        double* ll = sm;            // [L]
        double* g_ll = sm + L;      // [L]
        double* g_mu = sm + 2 * L;  // [L] gradient wrt mu_{t+1}
        double* busy = sm + 3 * L;  // [L] busy_t
        double* g_den = sm + 4 * L; // [L]
        __syncthreads();
        for (int i = threadIdx.x; i < NE; i += QH_THREADS) g_lam[e0 + i] = 0.f;
        for (int i = threadIdx.x; i < L; i += QH_THREADS) {
            const double l = (double)lam[e0 + h.maps_ol_el[l0 + i]];
            const double m = saved_mu[(size_t)QH_ITERS * total_links + l0 + i];
            const double gd = g_link[l0 + i];
            ll[i] = l;
            if ((l - m) > 0.0) {
                g_ll[i] = gd * h.T / (101.0 * m);
                g_mu[i] = -gd * h.T * l / (101.0 * m * m);
            } else {
                const double d = m - l;
                g_ll[i] = gd / (d * d);
                g_mu[i] = -gd / (d * d);
            }
        }
        __syncthreads();
        for (int t = QH_ITERS - 1; t >= 0; --t) {
            const double* mu_t = saved_mu + (size_t)t * total_links + l0;
            for (int i = threadIdx.x; i < L; i += QH_THREADS) busy[i] = fmin(fmax(ll[i] / mu_t[i], 0.0), 1.0);
            __syncthreads();
            for (int i = threadIdx.x; i < L; i += QH_THREADS) {
                double s = 0.0;
                const int a = h.adj_rowptr[l0 + i], b = h.adj_rowptr[l0 + i + 1];
                for (int e = a; e < b; ++e) s += busy[h.adj_colidx[e]];
                const double den = 1.0 + s;
                g_den[i] = -g_mu[i] * h.link_rates[l0 + i] / (den * den);
            }
            __syncthreads();
            for (int i = threadIdx.x; i < L; i += QH_THREADS) {
                double gb = 0.0;  // (A_i^T g_den)[i], A_i symmetric
                const int a = h.adj_rowptr[l0 + i], b = h.adj_rowptr[l0 + i + 1];
                for (int e = a; e < b; ++e) gb += g_den[h.adj_colidx[e]];
                const double m = mu_t[i], r = ll[i] / m;
                const double gr = (r >= 0.0 && r <= 1.0) ? gb : 0.0;  // clip_by_value passes the gradient inside [0, 1]
                g_ll[i] += gr / m;
                g_mu[i] = -gr * ll[i] / (m * m);  // wrt mu_t (mu_0 is a constant: the last value is dropped)
            }
            __syncthreads();
        }
        for (int i = threadIdx.x; i < L; i += QH_THREADS) g_lam[e0 + h.maps_ol_el[l0 + i]] = (float)g_ll[i];
        for (int i = threadIdx.x; i < NC; i += QH_THREADS) {
            const double l = (double)lam[e0 + h.maps_on_el[c0 + i]], m = h.node_mu[c0 + i], gd = g_node[c0 + i];
            const double gl = (l - m) > 0.0 ? gd * h.T / (100.0 * m) : gd / ((m - l) * (m - l));
            g_lam[e0 + h.maps_on_el[c0 + i]] = (float)gl;
        }
    }
}

static int fill_head(const mho_head_t* hd, HeadDev& h, const char* who) {
    if (!hd || hd->n_graphs < 0 || !hd->ext_off || !hd->link_off || !hd->comp_off || !hd->maps_ol_el || !hd->maps_on_el ||
        !hd->link_rates || !hd->cf_degs || !hd->node_mu || !hd->adj_rowptr || (hd->total_adj_nnz > 0 && !hd->adj_colidx) ||
        hd->max_links < 0) {
        mho_set_error("%s: invalid head description", who);
        return MHO_ERR_INVALID;
    }
    h.n_graphs = hd->n_graphs; h.ext_off = hd->ext_off; h.link_off = hd->link_off; h.comp_off = hd->comp_off;
    h.maps_ol_el = hd->maps_ol_el; h.maps_on_el = hd->maps_on_el; h.link_rates = hd->link_rates; h.cf_degs = hd->cf_degs;
    h.node_mu = hd->node_mu; h.adj_rowptr = hd->adj_rowptr; h.adj_colidx = hd->adj_colidx; h.T = hd->T;
    return MHO_OK;
}

extern "C" int mho_queue_head_forward(mho_ctx_t* c, const mho_head_t* hd, const float* lam, double* link_delay,
                                      double* node_delay, double* saved_mu, mho_stream_t stream) {
    HeadDev h;
    if (!c) { mho_set_error("mho_queue_head_forward: ctx is NULL"); return MHO_ERR_INVALID; }
    int rc = fill_head(hd, h, "mho_queue_head_forward");
    if (rc) return rc;
    if (hd->n_graphs == 0) return MHO_OK;
    if (!lam || !link_delay || !node_delay) { mho_set_error("mho_queue_head_forward: NULL buffer"); return MHO_ERR_INVALID; }
    if (cudaSetDevice(c->device) != cudaSuccess) { mho_set_error("cudaSetDevice failed"); return MHO_ERR_CUDA; }
    const size_t smem = (size_t)3 * hd->max_links * sizeof(double) + 16;
    if (smem > (size_t)c->max_smem_optin) { mho_set_error("mho_queue_head_forward: %d links per graph exceed shared memory", hd->max_links); return MHO_ERR_TOO_LARGE; }
    int grid = hd->n_graphs < 8 * c->num_sms ? hd->n_graphs : 8 * c->num_sms;
    cudaError_t e = mho_launch<queue_head_forward_kernel>(dim3((unsigned)grid), dim3(QH_THREADS), smem, (cudaStream_t)stream, false, h, lam, link_delay,
                                                           node_delay, saved_mu, hd->total_links);
    if (e != cudaSuccess) { mho_set_error("queue_head_forward launch failed: %s", cudaGetErrorString(e)); return MHO_ERR_CUDA; }
    c->launches += 1;
    return MHO_OK;
}

extern "C" int mho_queue_head_backward(mho_ctx_t* c, const mho_head_t* hd, const float* lam, const double* saved_mu,
                                       const double* g_link, const double* g_node, float* g_lam, mho_stream_t stream) {
    HeadDev h;
    if (!c) { mho_set_error("mho_queue_head_backward: ctx is NULL"); return MHO_ERR_INVALID; }
    int rc = fill_head(hd, h, "mho_queue_head_backward");
    if (rc) return rc;
    if (hd->n_graphs == 0) return MHO_OK;
    if (!lam || !saved_mu || !g_link || !g_node || !g_lam) { mho_set_error("mho_queue_head_backward: NULL buffer"); return MHO_ERR_INVALID; }
    if (cudaSetDevice(c->device) != cudaSuccess) { mho_set_error("cudaSetDevice failed"); return MHO_ERR_CUDA; }
    const size_t smem = (size_t)5 * hd->max_links * sizeof(double) + 16;
    if (smem > (size_t)c->max_smem_optin) { mho_set_error("mho_queue_head_backward: %d links per graph exceed shared memory", hd->max_links); return MHO_ERR_TOO_LARGE; }
    int grid = hd->n_graphs < 8 * c->num_sms ? hd->n_graphs : 8 * c->num_sms;
    cudaError_t e = mho_launch<queue_head_backward_kernel>(dim3((unsigned)grid), dim3(QH_THREADS), smem, (cudaStream_t)stream, false, h, lam, saved_mu,
                                                            g_link, g_node, g_lam, hd->total_links);
    if (e != cudaSuccess) { mho_set_error("queue_head_backward launch failed: %s", cudaGetErrorString(e)); return MHO_ERR_CUDA; }
    c->launches += 1;
    return MHO_OK;
}
