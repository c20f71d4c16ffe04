// Batched environment step: replaces AdhocCloud.offloading(sp, hop) (explore = 0, prob = False; src/offloading_v3.py:388-453)
// or AdhocCloud.local_compute(dproc) (:363-386), then AdhocCloud.run() (:455-550) and the drivers' delay_emp
// (AdHoc_test.py:140-153) - the CPU half of a rollout step.  One CTA per item (network, job set, method):
//   1. thread per job: the cost of every server and of local execution, the first-NaN-else-first-minimum argmin, and the
//      greedy route walk (argmin of sp[nbs, dst] over env.adj_c's stored row), recorded as a per-job link bitmask;
//   2. thread per link: lambda = link_load.sum(axis=1) in numpy's pairwise order over the job axis; thread per node:
//      the server loads in job order;
//   3. thread per link: the ten fixed-point iterations mu <- rates * (1 / (1 + A_i clip(lambda / mu, 0, 1))), one
//      barrier per half step;
//   4. the delays, the last-writer unit-delay matrix and, per job, delay_emp (nansum over links in ascending order,
//      pairwise when the item has one job, plus the node delay).
// Every product that feeds an add is an explicit __dmul_rn so that nothing is contracted into an FMA; fp64 division is
// IEEE.  The results are bit-identical to the reference's numpy arithmetic (oracle/env_oracle.py restates it).
#include <cstdint>

#include "mho_common.cuh"
#include "mho_internal.h"

namespace {

constexpr int ENV_THREADS = 256;

struct EnvParams {
    mho_env_t net;
    mho_env_items_t it;
    mho_env_out_t out;
    int words;   // bitmask words per job: ceil(max_links / 32)
};

__device__ __forceinline__ double nan_d() { return __longlong_as_double(0x7ff8000000000000LL); }

// np.max([a, b]) / np.maximum: NaN-propagating
__device__ __forceinline__ double nanmax(double a, double b) {
    if (isnan(a) || isnan(b)) return nan_d();
    return a > b ? a : b;
}

// np.argmin over a stream of values: the first NaN if there is one, otherwise the first minimum
struct ArgMin {
    int idx = -1;
    double best = 0.0;
    bool nan = false;
    __device__ __forceinline__ void push(int i, double v) {
        if (nan) return;
        if (isnan(v)) { nan = true; idx = i; best = v; return; }
        if (idx < 0 || v < best) { idx = i; best = v; }
    }
};

// numpy's pairwise_sum (numpy/_core/src/umath/loops_utils.h.src) of a(s), ..., a(s + n - 1)
template <class F>
__device__ double pw_leaf(const F& a, int s, int n) {
    if (n < 8) {
        double r = 0.0;
        for (int i = 0; i < n; ++i) r = __dadd_rn(r, a(s + i));
        return r;
    }
    double r[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) r[k] = a(s + k);
    int i = 8;
    for (; i < n - (n % 8); i += 8) {
#pragma unroll
        for (int k = 0; k < 8; ++k) r[k] = __dadd_rn(r[k], a(s + i + k));
    }
    double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                           __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
    for (; i < n; ++i) res = __dadd_rn(res, a(s + i));
    return res;
}

// blocks of more than 128 split at n2 = n/2 - (n/2) % 8; depth 3 covers n <= 1024
template <int D, class F>
__device__ double pairwise_sum(const F& a, int s, int n) {
    if constexpr (D > 0) {
        if (n > 128) {
            int n2 = n / 2;
            n2 -= n2 % 8;
            return __dadd_rn(pairwise_sum<D - 1>(a, s, n2), pairwise_sum<D - 1>(a, s + n2, n - n2));
        }
    }
    return pw_leaf(a, s, n);
}

__global__ void __launch_bounds__(ENV_THREADS) env_step_kernel(const __grid_constant__ EnvParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int s_status;
    const int item = blockIdx.x, tid = threadIdx.x;
    const mho_env_t& E = p.net;
    const mho_env_items_t& I = p.it;
    const mho_env_out_t& O = p.out;
    const int ML = E.max_links, MJ = I.max_jobs, MN = E.max_nodes, W = p.words;
    double* lam = reinterpret_cast<double*>(smem_raw);
    double* mu = lam + ML;
    double* busy = mu + ML;
    double* load = busy + ML;          // [MJ] ul*rate + dl*rate
    double* srv = load + MJ;           // [MN] server_load_array
    uint32_t* mask = reinterpret_cast<uint32_t*>(srv + MN);   // [MJ][W] links on the route of each job
    int* dstv = reinterpret_cast<int*>(mask + (size_t)MJ * W);
    int* nhopv = dstv + MJ;
    int* lastj = nhopv + MJ;           // [ML] last job whose route crosses the link, -1 if none

    if (tid == 0) {
        int st = MHO_ENV_OK;
        const int g = I.net[item], md = I.mode[item];
        const int j0 = I.job_off[item], j1 = I.job_off[item + 1];
        if (g < 0 || g >= E.n_nets || (md != MHO_ENV_GREEDY && md != MHO_ENV_LOCAL) || j1 < j0 || j1 - j0 > MJ) {
            st = MHO_ENV_BAD_ITEM;
        } else {
            const int n = E.node_off[g + 1] - E.node_off[g], L = E.link_off[g + 1] - E.link_off[g];
            if (n <= 0 || n > MN || L < 0 || L > ML) st = MHO_ENV_BAD_ITEM;
        }
        s_status = st;
    }
    __syncthreads();
    if (s_status != MHO_ENV_OK) {
        if (tid == 0) O.status[item] = s_status;
        return;
    }
    const int g = I.net[item], md = I.mode[item];
    const int j0 = I.job_off[item], J = I.job_off[item + 1] - j0;
    const int n0 = E.node_off[g], n = E.node_off[g + 1] - n0;
    const int l0 = E.link_off[g], L = E.link_off[g + 1] - l0;
    const int s0 = E.server_off[g], S = E.server_off[g + 1] - s0;
    const double* sp = I.sp + I.sp_off[item];
    const double* hop = E.hop + E.hop_off[g];
    const int32_t* servers = E.servers + s0;
    const int32_t* arp = E.adj_rowptr + n0;
    const double T = E.T[g];
    for (int j = tid; j < J; j += ENV_THREADS)
        if (I.src[j0 + j] < 0 || I.src[j0 + j] >= n) atomicExch(&s_status, MHO_ENV_BAD_ITEM);
    __syncthreads();
    if (s_status != MHO_ENV_OK) {
        if (tid == 0) O.status[item] = s_status;
        return;
    }

    // ---- 1. decisions and routes (offloading() / local_compute()) ----
    for (int j = tid; j < J; j += ENV_THREADS) {
        uint32_t* mj = mask + (size_t)j * W;
        for (int w = 0; w < W; ++w) mj[w] = 0u;
        const int gj = j0 + j, src = I.src[gj];
        const double ul = I.ul[gj], dl = I.dl[gj], rate = I.rate[gj];
        load[j] = __dadd_rn(__dmul_rn(ul, rate), __dmul_rn(dl, rate));
        int* route = O.routes ? O.routes + O.routes_off[item] + (size_t)j * O.route_stride : nullptr;
        int dst = src, hops = 0, rlen = 0;
        double est;
        if (md == MHO_ENV_LOCAL) {
            est = nanmax(__dmul_rn(sp[(size_t)src * n + src], ul), 1.0);
            if (route) { route[0] = src; route[1] = src; }
            rlen = 2;
        } else {
            const double local = __dmul_rn(sp[(size_t)src * n + src], ul);
            ArgMin am;
            for (int s = 0; s < S; ++s) {
                const int v = servers[s];
                const double up = v == src ? 0.0 : sp[(size_t)src * n + v];     // the diagonal of sp is zeroed
                const double down = v == src ? 0.0 : sp[(size_t)v * n + src];
                const double uld = nanmax(__dmul_rn(up, ul), hop[(size_t)src * n + v]);
                const double dld = nanmax(__dmul_rn(down, dl), hop[(size_t)v * n + src]);
                const double proc = nanmax(__dmul_rn(sp[(size_t)v * n + v], ul), 1.0);
                am.push(s, __dadd_rn(__dadd_rn(uld, dld), proc));
            }
            am.push(S, local);
            if (am.idx < S) {
                est = am.best;
                dst = servers[am.idx];
                int node = src;
                if (route) route[0] = src;
                rlen = 1;
                while (node != dst) {   // routing(): argmin sp[nbs, dst] over the stored adjacency row of the node
                    const int e0 = arp[node], e1 = arp[node + 1];
                    if (hops >= n) { atomicExch(&s_status, MHO_ENV_ROUTE_LOOP); break; }
                    if (e1 <= e0) { atomicExch(&s_status, MHO_ENV_NO_LINK); break; }
                    ArgMin nb;
                    for (int e = e0; e < e1; ++e) {
                        const int u = E.adj_col[e];
                        nb.push(e - e0, u == dst ? 0.0 : sp[(size_t)u * n + dst]);
                    }
                    const int e = e0 + nb.idx, lk = E.adj_link[e];
                    if (lk < 0 || lk >= L) { atomicExch(&s_status, MHO_ENV_NO_LINK); break; }
                    mj[lk >> 5] |= 1u << (lk & 31);
                    node = E.adj_col[e];
                    ++hops;
                    if (route && rlen < O.route_stride) route[rlen] = node;
                    ++rlen;
                }
            } else {
                est = local;
                if (route) { route[0] = src; route[1] = src; }
                rlen = 2;
            }
        }
        if (route) for (int k = rlen; k < O.route_stride; ++k) route[k] = -1;
        dstv[j] = dst;
        nhopv[j] = hops;
        O.dst[gj] = dst;
        O.nhop[gj] = hops;
        O.delay_est[gj] = est;
    }
    __syncthreads();
    const int status = s_status;
    if (tid == 0) O.status[item] = status;
    if (status != MHO_ENV_OK) {   // the reference never returns here: leave a recognisable item
        for (int j = tid; j < J; j += ENV_THREADS) {
            O.dst[j0 + j] = -1; O.nhop[j0 + j] = -1;
            O.delay_est[j0 + j] = nan_d(); O.delay_emp[j0 + j] = nan_d();
            if (O.routes) for (int k = 0; k < O.route_stride; ++k) O.routes[O.routes_off[item] + (size_t)j * O.route_stride + k] = -1;
        }
        if (O.delay_links) for (int i = tid; i < L * J; i += ENV_THREADS) O.delay_links[O.links_off[item] + i] = nan_d();
        if (O.delay_nodes) for (int i = tid; i < n * J; i += ENV_THREADS) O.delay_nodes[O.nodes_off[item] + i] = nan_d();
        if (O.unit) for (int i = tid; i < n * n; i += ENV_THREADS) O.unit[O.unit_off[item] + i] = nan_d();
        return;
    }

    // ---- 2. loads: lambda (pairwise over the job axis), server loads (job order), mu_0 ----
    for (int l = tid; l < L; l += ENV_THREADS) {
        const int w = l >> 5;
        const uint32_t b = 1u << (l & 31);
        auto a = [&](int j) { return (mask[(size_t)j * W + w] & b) ? load[j] : 0.0; };
        lam[l] = J > 0 ? pairwise_sum<4>(a, 0, J) : 0.0;
        int last = -1;
        for (int j = J - 1; j >= 0; --j)
            if (mask[(size_t)j * W + w] & b) { last = j; break; }
        lastj[l] = last;
        mu[l] = E.link_rates[l0 + l] / __dadd_rn(E.cf_degs[l0 + l], 1.0);
    }
    for (int v = tid; v < n; v += ENV_THREADS) {
        double s = 0.0;
        for (int j = 0; j < J; ++j)
            if (dstv[j] == v) s = __dadd_rn(s, __dmul_rn(I.ul[j0 + j], I.rate[j0 + j]));
        srv[v] = s;
    }
    __syncthreads();

    // ---- 3. ten fixed-point iterations of the link service rates ----
    const int32_t* crp = E.cf_rowptr + l0;
    for (int it = 0; it < 10; ++it) {
        for (int l = tid; l < L; l += ENV_THREADS) {
            const double x = lam[l] / mu[l];
            busy[l] = x < 0.0 ? 0.0 : (x > 1.0 ? 1.0 : x);   // np.clip: NaN stays NaN
        }
        __syncthreads();
        for (int l = tid; l < L; l += ENV_THREADS) {
            double nb = 0.0;
            for (int e = crp[l]; e < crp[l + 1]; ++e) nb = __dadd_rn(nb, busy[E.cf_col[e]]);
            mu[l] = __dmul_rn(E.link_rates[l0 + l], 1.0 / __dadd_rn(1.0, nb));
        }
        __syncthreads();
    }

    // ---- 4. delays ----
    auto link_unit = [&](int l, int j) {
        const double m = mu[l], la = lam[l], diff = __dsub_rn(m, la);
        double u = 1.0 / diff;
        if (diff <= 0.0) {
            const int gj = j0 + j;
            u = __dmul_rn(T, la / __dmul_rn(__dadd_rn(I.ul[gj], I.dl[gj]), m));
        }
        return u;
    };
    auto link_delay = [&](int l, int j) {
        const double u = link_unit(l, j), h = (double)nhopv[j];
        return __dadd_rn(nanmax(__dmul_rn(I.ul[j0 + j], u), h), nanmax(__dmul_rn(I.dl[j0 + j], u), h));
    };
    auto node_unit = [&](int j) {
        const int d = dstv[j];
        const double pb = E.proc_bws[n0 + d], ld = srv[d], diff = __dsub_rn(pb, ld);
        double u = 1.0 / diff;
        if (diff <= 0.0) u = __dmul_rn(T, ld / __dmul_rn(I.ul[j0 + j], pb));
        return u;
    };
    auto node_delay = [&](int j) { return nanmax(__dmul_rn(I.ul[j0 + j], node_unit(j)), 1.0); };

    if (O.delay_links) {
        double* dlk = O.delay_links + O.links_off[item];
        for (int i = tid; i < L * J; i += ENV_THREADS) {
            const int l = i / J, j = i - l * J;
            dlk[i] = (mask[(size_t)j * W + (l >> 5)] >> (l & 31)) & 1u ? link_delay(l, j) : nan_d();
        }
    }
    if (O.delay_nodes) {
        double* dnd = O.delay_nodes + O.nodes_off[item];
        for (int i = tid; i < n * J; i += ENV_THREADS) {
            const int v = i / J, j = i - v * J;
            dnd[i] = dstv[j] == v ? node_delay(j) : nan_d();
        }
    }
    if (O.unit) {   // U[n0, n1] = U[n1, n0] of each link on a route and U[dst, dst]: the last job to write wins
        double* U = O.unit + O.unit_off[item];
        for (int i = tid; i < n * n; i += ENV_THREADS) {
            const int a = i / n, b = i - a * n;
            double x = nan_d();
            if (a == b)
                for (int j = J - 1; j >= 0; --j)
                    if (dstv[j] == a) { x = node_unit(j); break; }
            U[i] = x;
        }
        __syncthreads();
        for (int v = tid; v < n; v += ENV_THREADS)
            for (int e = arp[v]; e < arp[v + 1]; ++e) {
                const int lk = E.adj_link[e], u = E.adj_col[e];
                if (lk >= 0 && lk < L && u != v && lastj[lk] >= 0) U[(size_t)v * n + u] = link_unit(lk, lastj[lk]);
            }
    }
    for (int j = tid; j < J; j += ENV_THREADS) {   // nansum(delay_links, 0) + nansum(delay_nodes, 0)
        const uint32_t* mj = mask + (size_t)j * W;
        double s = 0.0;
        if (J == 1) {   // a contiguous column: numpy sums it pairwise
            auto a = [&](int l) {
                if (!((mj[l >> 5] >> (l & 31)) & 1u)) return 0.0;
                const double x = link_delay(l, j);
                return isnan(x) ? 0.0 : x;
            };
            s = L > 0 ? pairwise_sum<4>(a, 0, L) : 0.0;
        } else {
            for (int w = 0; w < W; ++w)
                for (uint32_t bits = mj[w]; bits; bits &= bits - 1) {
                    const int l = (w << 5) + __ffs(bits) - 1;
                    const double x = link_delay(l, j);
                    if (!isnan(x)) s = __dadd_rn(s, x);
                }
        }
        const double nd = node_delay(j);
        O.delay_emp[j0 + j] = __dadd_rn(s, isnan(nd) ? 0.0 : nd);
    }
}

}  // namespace

size_t env_step_smem(int max_nodes, int max_links, int max_jobs) {
    const size_t W = (size_t)(max_links + 31) / 32;
    return (size_t)(3 * max_links + max_jobs + max_nodes) * 8 + (size_t)max_jobs * W * 4 + (size_t)(2 * max_jobs + max_links) * 4;
}

cudaError_t env_step_launch(const mho_env_t& nets, const mho_env_items_t& items, const mho_env_out_t& out, cudaStream_t st) {
    EnvParams p{nets, items, out, (nets.max_links + 31) / 32};
    const size_t smem = env_step_smem(nets.max_nodes, nets.max_links, items.max_jobs);
    return mho_launch<env_step_kernel>(dim3((unsigned)items.n_items), dim3(ENV_THREADS), smem, st, false, p);
}
