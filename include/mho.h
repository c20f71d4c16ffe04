/*
 * mho.h - C-ABI of libmho.so: the B200-native (sm_100a) batched ChebConv hot path of
 * zhongyuanzhao/multihop-offload.
 *
 * The reference has no FFI: its seam is the Python call `self.model([x_in, a_in])`
 * (src/gnn_offloading_agent.py:149, model built at :81-123 from spektral.layers.ChebConv) and
 * the tape VJP `g.gradient(delay_mtx_ts, weights, output_gradients=...)` (:448), plus the
 * optimizer replay (:156-169) that consumes the gradients.  Each entry point below names the
 * reference interface it replaces.  INTEGRATION.md shows the ctypes binding a maintainer adds.
 *
 * Conventions: plain C, int return (0 = ok, <0 = mho_status), message via mho_last_error();
 * all array arguments are caller-owned DEVICE pointers unless the name ends in _host; the
 * callee never frees caller memory; every launch goes to the caller-supplied stream; no hidden
 * synchronisation except in the *_host convenience calls (documented).  One context per
 * (thread, GPU) - and one per stream when several streams launch concurrently (a context holds
 * reduction scratch and staging slots).  fp32 storage, fp32 accumulate; tensor-core operands are exact
 * multi-part splits of the fp32 values (two fp16 parts after power-of-two scales, three bf16 parts,
 * or TF32 hi/lo, depending on the kernel): results agree with an fp32 evaluation to round-off.
 */
#ifndef MHO_H_
#define MHO_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MHO_VERSION 100

typedef struct mho_ctx mho_ctx_t;
typedef void* mho_stream_t; /* a cudaStream_t; NULL = the legacy default stream */

typedef enum {
    MHO_OK = 0,
    MHO_ERR_INVALID = -1,      /* bad argument (NULL pointer, K<1, F>32, ...) */
    MHO_ERR_TOO_LARGE = -2,    /* a graph/tile exceeds what one CTA can hold in shared memory */
    MHO_ERR_CUDA = -3,         /* a CUDA runtime call failed; mho_last_error() has the string */
    MHO_ERR_NO_DEVICE = -4,    /* no sm_100 device: there is NO CPU fallback by design */
    MHO_ERR_NCCL = -5
} mho_status;

enum { MHO_ACT_NONE = 0, MHO_ACT_RELU = 1, MHO_ACT_LEAKY = 2 };
enum { MHO_MAX_F = 32, MHO_MAX_K = 16, MHO_MAX_LAYERS = 16, MHO_MAX_TILE_ROWS = 512 };

/*
 * A batch of independent graphs, concatenated block-diagonally (the reference evaluates one
 * graph per eager call, gnn_offloading_agent.py:144-150; a batch is many such calls at once).
 * Operator = whatever the caller supplies; the reference feeds the raw binary adjacency of
 * the extended line graph (:218), sorted row-major (spektral.utils.sp_matrix_to_sp_tensor,
 * call site :148) - i.e. CSR.
 */
typedef struct {
    int32_t n_graphs;
    int32_t total_nodes;
    int64_t total_nnz;
    const int32_t* graph_off;  /* [n_graphs+1] node offset of each graph */
    const int32_t* rowptr;     /* [total_nodes+1] offsets into colidx/vals (global) */
    const int32_t* colidx;     /* [total_nnz] GLOBAL node ids (block-diagonal CSR) */
    const float*   vals;       /* [total_nnz] or NULL => every stored entry is 1.0 */
    /* transpose operator for the VJP; all three NULL => operator is symmetric (every graph the
       reference produces is: undirected line graph), and the forward arrays are reused */
    const int32_t* rowptr_t;
    const int32_t* colidx_t;
    const float*   vals_t;
    /* tile plan (from mho_plan_tiles): tile t = graphs [tile_off[t], tile_off[t+1]) processed
       by one CTA; NULL => one graph per tile */
    const int32_t* tile_off;   /* [n_tiles+1] graph indices, device */
    const int32_t* tile_info;  /* optional [n_tiles][4] = {node0, rows, nz0, nnz} (device, 16 B aligned), in ANY
                                  order: with it the forward kernel's CTAs pull tiles dynamically in the listed
                                  order (list the largest first) instead of a static round-robin over tile_off;
                                  NULL => bounds derived from tile_off/graph_off/rowptr, static schedule */
    int32_t n_tiles;
    int32_t max_tile_rows;     /* max over tiles of the node count (host-known) */
    int32_t max_tile_nnz;      /* max over tiles of the nnz count (host-known) */
    /* optional (device, 16 B aligned): the BINARY operator as bit rows, [total_nodes][4] words; bit j of word w of
       node i = "i is adjacent to node tile_node0(i) + 32 w + j" (tile of the plan above, <= 128 nodes, from
       mho_fill_adj_bits).  With it the forward's tensor-core path (vals == NULL, tiles <= 128 nodes) reads 16 B per
       node instead of walking the CSR slice; NULL => the kernel derives the bits from rowptr/colidx itself.  In a batch
       with tile_off == NULL (one tile per graph: mho_cheb_backward) the bits are relative to the graph's first node. */
    const uint32_t* adj_bits;
    /* optional (device), [n_tiles] parallel to tile_info: index of the FIRST graph of each listed tile (its graphs are
       consecutive).  With it the fp16-part tensor-core forward scales its operands per GRAPH (graph_off is then read on
       the device): graphs of very different magnitude may share a tile.  NULL => one scale per tile - exact to 1e-5 as
       long as the graphs of a tile are within ~2^10 of each other in magnitude. */
    const int32_t* tile_graph0;
} mho_batch_t;

/* One ChebConv layer: Y = act(sum_k T_k(A) X W[k] + b), T_0=X, T_1=A X, T_k=2 A T_{k-1}-T_{k-2}
 * (spektral.layers.ChebConv.call; K is the Spektral default 1 in the shipped model,
 * gnn_offloading_agent.py:95-110).  W is [K, f_in, f_out] row-major = the Keras kernel layout
 * stored in the checkpoints; b is [f_out] or NULL. */
typedef struct {
    int32_t K, f_in, f_out, act;
    float slope;               /* leaky_relu negative slope (0.2 = tf.nn.leaky_relu default) */
    const float* W;
    const float* b;
} mho_layer_t;

/* ---- context ---------------------------------------------------------------------------- */
/* A context owns the tile-scheduler counters, the packed weight images and the host-call staging slots: use it from ONE
 * stream at a time (launches on one stream are ordered; for concurrent streams create one context per stream). */
int mho_create(mho_ctx_t** ctx, int device);
int mho_destroy(mho_ctx_t* ctx);
const char* mho_last_error(void);
int mho_version(void);
/* number of kernels launched through this context so far (bench.py's gpu_launches claim) */
int64_t mho_launch_count(const mho_ctx_t* ctx);

/* The forward snapshots the weights of a layer set into packed operand images (see DESIGN.md 3.10) the first time it sees
 * a given set of (W, b) pointers and reuses them afterwards.  Call this after modifying weights IN PLACE
 * behind the library's back (mho_adam_replay does it itself). */
int mho_invalidate_weights(mho_ctx_t* ctx);

/* ---- host-side planning helper (pure CPU, no CUDA): greedy packing of consecutive graphs
 * into tiles of at most tile_rows nodes.  graph_off_host/rowptr_host are HOST copies.
 * tile_off_host must have room for n_graphs+1 entries.  Graphs larger than tile_rows get a
 * tile of their own (up to MHO_MAX_TILE_ROWS). */
int mho_plan_tiles(const int32_t* graph_off_host, const int32_t* rowptr_host, int32_t n_graphs,
                   int32_t tile_rows, int32_t* tile_off_host, int32_t* n_tiles,
                   int32_t* max_tile_rows, int32_t* max_tile_nnz);
/* tile_info_host [n_tiles][4] from a plan (tile_off_host NULL => one graph per tile) */
int mho_fill_tile_info(const int32_t* graph_off_host, const int32_t* rowptr_host, const int32_t* tile_off_host,
                       int32_t n_tiles, int32_t* tile_info_host);

/* adj_bits_host [total_nodes][4] from a plan whose tiles have at most 128 nodes (see mho_batch_t.adj_bits);
 * colidx_host holds GLOBAL node ids. */
int mho_fill_adj_bits(const int32_t* graph_off_host, const int32_t* rowptr_host, const int32_t* colidx_host,
                      const int32_t* tile_off_host, int32_t n_tiles, uint32_t* adj_bits_host);

/* ---- forward: replaces ACOAgent.predict -> self.model([x_in, a_in])
 * (gnn_offloading_agent.py:144-150) for a whole batch.  X [total_nodes, layers[0].f_in],
 * Y [total_nodes, layers[n-1].f_out], both row-major fp32.  `saved` (nullable) receives the
 * inputs of layers 1..n-1 (the hidden activations) for the VJP: mho_saved_bytes() bytes.
 * Kernel selection (results agree to fp32 round-off; all tcgen05 / TMEM kernels need tile_off + tile_info and tiles of
 * <= 128 nodes):
 *   - one layer 32 -> 32, 2 <= K <= 10, vals == NULL, tile_graph0 set: csrc/cheb_forward_f16.cu (fp16 two-part operands);
 *   - every layer K = 1, <= 32 features (first f_in a multiple of 4): csrc/cheb_mlp_f16.cu, the whole stack in one launch;
 *     the operator is never read and tile_info may describe ANY runs of <= 128 consecutive nodes (they need not respect
 *     graph boundaries);
 *   - <= 32 features per layer, K <= 5, vals == NULL: csrc/cheb_forward_dense.cu (bf16 three-part operands, fused stacks);
 *   - everything else (weighted operators, tiles of up to 512 nodes, K up to 16): the CSR-walk kernel csrc/cheb_forward.cu.
 * With vals == NULL the CSR must not hold duplicate entries. */
int mho_cheb_forward(mho_ctx_t* ctx, const mho_batch_t* batch, const mho_layer_t* layers,
                     int32_t n_layers, const float* X, float* Y, void* saved, mho_stream_t stream);
size_t mho_saved_bytes(const mho_batch_t* batch, const mho_layer_t* layers, int32_t n_layers);

/* ---- backward: replaces g.gradient(delay_mtx_ts, model.trainable_weights, output_gradients)
 * (gnn_offloading_agent.py:448) from the GNN output back to the weights.  dY is the gradient
 * wrt Y (the caller has already pulled grad_dist through the queue head).  grads_per_graph
 * [n_graphs, n_params] receives one flat gradient per graph instance in variable-creation order
 * (kernel_0, bias_0, kernel_1, ...; the order the reference memorises them, :142,:450);
 * grads_sum [n_params] (nullable) their deterministic sum (the buffer a data-parallel
 * all-reduce ships).  dX nullable.  Requires a one-graph-per-tile batch (tile_off == NULL).
 * One layer 32 -> 32, 2 <= K <= 10, vals == NULL, graphs of <= 128 nodes, dX == NULL and batch->adj_bits set (bit rows
 * relative to each GRAPH's first node: what mho_fill_adj_bits gives for tile_off = 0, 1, 2, ...) runs on the tensor
 * cores (csrc/cheb_backward_f16.cu); stacks whose layers all have K = 1, hidden width 32, first f_in a multiple of 4, last
 * f_out <= 4 (the shipped model) with dX == NULL run on csrc/cheb_mlp_backward_f16.cu; every other shape on
 * csrc/cheb_backward.cu. */
int mho_cheb_backward(mho_ctx_t* ctx, const mho_batch_t* batch, const mho_layer_t* layers,
                      int32_t n_layers, const float* X, const float* Y, const void* saved,
                      const float* dY, float* grads_per_graph, float* grads_sum, float* dX,
                      mho_stream_t stream);
int64_t mho_param_count(const mho_layer_t* layers, int32_t n_layers);

/* ---- optimizer: replaces ACOAgent.replay's loop of optimizer.apply_gradients
 * (gnn_offloading_agent.py:156-169) with Keras Adam(clipnorm=1) (:114-121) and the
 * max_norm(1.0, axis=0) constraints (:104-108): applies n_steps stored gradients
 * SEQUENTIALLY in one launch.  The reference trains in fp64, so the master weights and the
 * moments are fp64 device buffers [n_params] in the flat layout above (lr=1e-6 updates would
 * drown in fp32); params_f32 receives the fp32 copy the forward/backward kernels read.
 * grads [n_steps, n_params] fp32; step_count is the optimizer's iteration counter before the call. */
typedef struct {
    double lr, beta1, beta2, eps, clipnorm, max_norm; /* clipnorm<=0 / max_norm<=0 disable */
    double decay_rate; int32_t decay_steps;           /* ExponentialDecay; decay_rate==1 => constant */
} mho_adam_t;
int mho_adam_replay(mho_ctx_t* ctx, const mho_layer_t* layers, int32_t n_layers,
                    const mho_adam_t* cfg, double* params, double* m, double* v, float* params_f32,
                    const float* grads, int32_t n_steps, int64_t step_count, mho_stream_t stream);

/* ---- queue-model head that follows the GNN: replaces the TensorFlow op chain of ACOAgent.forward,
 * gnn_offloading_agent.py:231-254 (gathers, 10 fixed-point iterations mu <- r / (1 + A_i clip(lambda/mu, 0, 1)),
 * M/M/1 delays with the congestion branch) and its VJP (the head part of :448, through all ten iterations),
 * fused and batched, fp64 like the reference.  All arrays are device pointers; graphs are concatenated:
 * ext_off (= the GNN batch's graph_off), link_off, comp_off [n_graphs+1]; maps_* hold LOCAL extended-edge ids
 * (obj.maps_ol_el / obj.maps_on_el); adj_rowptr [total_links+1] global offsets, adj_colidx LOCAL link ids of the
 * symmetric conflict graph env.adj_i; node_mu = proc_bws[proc_bws > 0]. */
typedef struct {
    int32_t n_graphs, max_links;           /* max_links: largest per-graph link count (shared-memory sizing) */
    int64_t total_links, total_comp, total_adj_nnz;
    const int32_t* ext_off; const int32_t* link_off; const int32_t* comp_off;
    const int32_t* maps_ol_el; const int32_t* maps_on_el;
    const double* link_rates; const double* cf_degs; const double* node_mu;
    const int32_t* adj_rowptr; const int32_t* adj_colidx;
    double T;                              /* env.T, the congestion-penalty constant */
} mho_head_t;
/* lam [total_ext] fp32 (the GNN output) -> link_delay [total_links], node_delay [total_comp] (fp64);
 * saved_mu (nullable) [11 * total_links] keeps mu_0..mu_10 for the backward */
int mho_queue_head_forward(mho_ctx_t* ctx, const mho_head_t* head, const float* lam, double* link_delay,
                           double* node_delay, double* saved_mu, mho_stream_t stream);
/* g_link / g_node: gradients wrt the delays -> g_lam [total_ext] fp32 (the dY of mho_cheb_backward) */
int mho_queue_head_backward(mho_ctx_t* ctx, const mho_head_t* head, const float* lam, const double* saved_mu,
                            const double* g_link, const double* g_node, float* g_lam, mho_stream_t stream);

/* ---- all-pairs shortest path lengths of a batch of small undirected graphs: replaces util.all_pairs_shortest_paths
 * (src/util.py:101-110; call sites gnn_offloading_agent.py:286-287,304-305, AdHoc_test.py:135-136, AdHoc_train.py:134-135).
 * The graphs are concatenated like a mho_batch_t: node_off [n_graphs+1], rowptr [total_nodes+1] (global offsets),
 * colidx [nnz] GLOBAL node ids, both directions of every edge stored; weight [nnz] fp64 edge lengths (> 0, equal
 * for the two directions) or NULL for hop counts.  dist receives one row-major n_g x n_g fp64 block per graph at element
 * offset out_off[g] (out_off [n_graphs], int64); unreachable pairs are +inf (the reference raises KeyError there).
 * Results are bit-identical to Dijkstra's algorithm on the same weights.  All pointers are DEVICE memory. */
int mho_apsp(mho_ctx_t* ctx, int32_t n_graphs, const int32_t* node_off, const int32_t* rowptr, const int32_t* colidx,
             const double* weight, const int64_t* out_off, double* dist, mho_stream_t stream);

/* ---- environment step: replaces AdhocCloud.offloading(sp, hop) with explore = 0, prob = False (src/offloading_v3.py:388-453)
 * or AdhocCloud.local_compute(dproc) (:363-386), followed by AdhocCloud.run() (:455-550) and the drivers'
 * delay_emp = nansum(delay_links, 0) + nansum(delay_nodes, 0) (AdHoc_test.py:140-153), for a batch of ITEMS: one item is
 * one (network, job set, method).  fp64 throughout, bit-identical to the reference (no contracted multiply-adds; the
 * sums follow numpy's summation order).  One CTA per item.
 *
 * Networks are concatenated like mho_head_t; every id stored in the arrays is LOCAL to its network.  Per network g:
 * nodes [node_off[g], node_off[g+1]), links [link_off[g], link_off[g+1]) in env.link_list order, servers
 * [server_off[g], server_off[g+1]) in env.servers order.  adj_rowptr [total_nodes+1] (global offsets) / adj_col /
 * adj_link: env.adj_c row by row in its stored CSR order without explicit zeros (what np.nonzero(adj_c[v]) returns),
 * adj_link = the env.link_list index of (v, u), else of (u, v), else -1.  cf_rowptr [total_links+1] (global offsets) /
 * cf_col: the binary conflict graph env.adj_i, neighbours in ASCENDING order.  hop: one row-major n x n block per network
 * at element offset hop_off[g] (the hop-count shortest paths, instance-invariant). */
enum { MHO_ENV_MAX_NODES = 512, MHO_ENV_MAX_LINKS = 1024, MHO_ENV_MAX_JOBS = 512 };
enum { MHO_ENV_GREEDY = 0, MHO_ENV_LOCAL = 1 };
/* per-item status */
enum {
    MHO_ENV_OK = 0,
    MHO_ENV_ROUTE_LOOP = 1,   /* a route walk did not reach its server within n hops (the reference never returns) */
    MHO_ENV_NO_LINK = 2,      /* a route walk met a node without neighbours or an adjacency entry without a link id
                                 (the reference raises ValueError) */
    MHO_ENV_BAD_ITEM = 3      /* network index, mode, job range, source node or a size beyond the MHO_ENV_MAX_* limits */
};
typedef struct {
    int32_t n_nets;
    int32_t max_nodes, max_links;            /* host-known maxima over the networks (limits and shared-memory sizing) */
    const int32_t* node_off; const int32_t* link_off; const int32_t* server_off;   /* [n_nets+1] */
    const int32_t* servers;                  /* [total_servers] */
    const int32_t* adj_rowptr; const int32_t* adj_col; const int32_t* adj_link;
    const double* link_rates; const double* cf_degs;                             /* [total_links] */
    const double* proc_bws;                  /* [total_nodes] */
    const int32_t* cf_rowptr; const int32_t* cf_col;
    const double* hop; const int64_t* hop_off;
    const double* T;                         /* [n_nets] env.T */
} mho_env_t;
/* Item i: network net[i], mode[i], jobs [job_off[i], job_off[i+1]) in env.jobs order (source node, arrival rate, ul_data,
 * dl_data), and the n x n fp64 shortest-path block at element offset sp_off[i] of sp, row-major as mho_apsp writes it
 * and with the server unit delays on the diagonal (the matrix the reference passes to offloading()).  Items may share
 * a block.  MHO_ENV_LOCAL reads only its diagonal (the dproc of local_compute). */
typedef struct {
    int32_t n_items;
    int32_t max_jobs;                        /* host-known maximum job count of one item */
    const int32_t* net; const int32_t* mode; const int32_t* job_off;   /* [n_items], [n_items], [n_items+1] */
    const double* sp; const int64_t* sp_off;
    const int32_t* src; const double* rate; const double* ul; const double* dl;   /* [total_jobs] */
} mho_env_items_t;
/* Per job (global job index): dst (flow.dst), nhop, delay_est (the delay offloading() / local_compute() returns),
 * delay_emp.  Optional (NULL = not written), each at a per-item ELEMENT offset:
 *   routes [J][route_stride] int32 at routes_off[i]: flow.route, padded with -1 (route_stride >= n + 1);
 *   delay_links [L][J] at links_off[i], delay_nodes [n][J] at nodes_off[i], unit [n][n] at unit_off[i]: run()'s three
 *   matrices, row-major, NaN where run() leaves NaN.
 * status [n_items] (MHO_ENV_*).  An item whose status is ROUTE_LOOP or NO_LINK gets dst = nhop = -1 and NaN delays for
 * all its jobs and NaN/-1 in its optional outputs; a BAD_ITEM writes its status only.  Other items are unaffected. */
typedef struct {
    int32_t* dst; int32_t* nhop; double* delay_est; double* delay_emp;
    int32_t* routes; const int64_t* routes_off; int32_t route_stride;
    double* delay_links; const int64_t* links_off;
    double* delay_nodes; const int64_t* nodes_off;
    double* unit; const int64_t* unit_off;
    int32_t* status;
} mho_env_out_t;
/* MHO_ERR_INVALID on a NULL required pointer, an optional output without its offsets or a negative count;
 * MHO_ERR_TOO_LARGE when max_nodes / max_links / max_jobs exceed the MHO_ENV_MAX_* limits.  All pointers inside the
 * three structs are DEVICE memory; the structs themselves are host memory. */
int mho_env_step(mho_ctx_t* ctx, const mho_env_t* nets, const mho_env_items_t* items, const mho_env_out_t* out,
                 mho_stream_t stream);

/* ---- host-buffer convenience (the reference-facing call: numpy in, numpy out, as
 * ACOAgent.predict takes them).  All pointers are HOST memory (pinned for full speed); the
 * call uploads the batch + X, runs mho_cheb_forward, downloads Y and synchronises `stream`.
 * Weights inside `layers` are still DEVICE pointers (they live on the GPU across steps). */
int mho_cheb_forward_host(mho_ctx_t* ctx, int32_t n_graphs, const int32_t* graph_off_host,
                          const int32_t* rowptr_host, const int32_t* colidx_host,
                          const float* vals_host, const mho_layer_t* layers, int32_t n_layers,
                          const float* X_host, float* Y_host, mho_stream_t stream);

/* Pipelined form: returns once everything is enqueued; *ticket identifies the call for mho_host_wait, which returns
 * when Y_host of that call is complete.  At most two calls may be in flight per context (a third waits for the
 * oldest), each with its own host buffers: the upload of call i+1 then overlaps the download of call i, keeping both
 * PCIe directions busy.  Results of the GNN are identical to the blocking call. */
int mho_cheb_forward_host_async(mho_ctx_t* ctx, int32_t n_graphs, const int32_t* graph_off_host,
                                const int32_t* rowptr_host, const int32_t* colidx_host,
                                const float* vals_host, const mho_layer_t* layers, int32_t n_layers,
                                const float* X_host, float* Y_host, mho_stream_t stream, int32_t* ticket);
int mho_host_wait(mho_ctx_t* ctx, int32_t ticket);

/* Page-locked host staging buffers for the *_host call (cudaHostAlloc): measured on the round-1 box 54 GB/s
 * host->device against 16.5 GB/s from framework-pinned memory that ended up on the wrong NUMA node. */
int mho_host_alloc(void** ptr, size_t bytes);
int mho_host_free(void* ptr);

#ifdef __cplusplus
}
#endif
#endif /* MHO_H_ */
