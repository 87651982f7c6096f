/*
 * gccb200.h -- C ABI of libgccb200.so: the Blackwell (sm_100a) implementation of the
 * THUDM/GCC pretraining hot path (SURVEY.md section 8).
 *
 * The reference has no FFI of its own (it is Python calling DGL / PyTorch), so
 * each entry point cites the reference call site it replaces.  Conventions:
 *   - every pointer is a CALLER-ALLOCATED DEVICE pointer unless marked "host";
 *   - the library never allocates, frees, synchronises or throws; it enqueues
 *     kernels on `stream` (a cudaStream_t passed as void*) and returns
 *     GCCB_OK or a negative gccb_status;  gccb_last_error() gives the text;
 *   - data-dependent failures (capacity overflow, zero-degree vertex, eigen
 *     non-convergence) are reported through a device-side flag word
 *     (gccb_batch_t.flags, GCCB_FLAG_*), so calls stay CUDA-graph capturable;
 *   - stateless, thread-safe per stream.
 * There is no CPU fallback: on a machine without an sm_100 device every compute
 * entry point returns GCCB_ERR_CUDA / GCCB_ERR_ARCH.
 */
#ifndef GCCB200_H_
#define GCCB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GCCB_VERSION 200 /* round 2 */

typedef void* gccb_stream_t; /* cudaStream_t */

typedef enum {
  GCCB_OK = 0,
  GCCB_ERR_BADARG = -1,
  GCCB_ERR_CAPACITY = -2,
  GCCB_ERR_ARCH = -3,
  GCCB_ERR_CUDA = -4
} gccb_status;

/* bits of the device-side flag word */
#define GCCB_FLAG_NODE_OVERFLOW 1   /* batched nodes of a view exceed node_cap          */
#define GCCB_FLAG_EDGE_OVERFLOW 2   /* batched edges of a view exceed edge_cap          */
#define GCCB_FLAG_ZERO_DEGREE 4     /* walk hit a vertex without successors (DGL: FATAL) */
#define GCCB_FLAG_EIG_NOCONV 8      /* eigensolver hit its sweep/iteration limit        */
#define GCCB_FLAG_EIG_TOOBIG 16     /* ego-net larger than the eigensolver supports     */

int gccb_version(void);
/* compute capability (major*10+minor) of the current device, or a negative status */
int gccb_arch(void);
const char* gccb_last_error(void);
/* number of kernels this library has enqueued so far in this process (host counter) */
unsigned long long gccb_launch_count(void);

/* ---- parent graph + sampler constants (host struct, device pointers inside) -------- */
typedef struct {
  const int64_t* indptr;       /* [n_nodes+1] CSR row offsets                                */
  const int32_t* indices;      /* [nnz] neighbour ids, ascending per row                     */
  int64_t n_nodes;
  const int32_t* budget_table; /* [budget_table_len] max_nodes_per_seed by seed degree:
                                  graph_dataset.py:113-124, built on the host               */
  int32_t budget_table_len;
  int32_t max_budget;          /* max over budget_table (sizes shared memory / scratch)      */
  uint32_t restart_thresh;     /* floor(restart_prob * 2^32)                                 */
  uint32_t _pad;
  uint64_t key;                /* Philox key = run seed (train.py:118 --seed)                */
} gccb_graph_t;

/* ---- a batch of ego-subgraphs: B (q,k) pairs = two views of B graphs each ----------
 * Replaces the pair of batched DGLGraphs produced by batcher() (data_util.py:26-32).
 * View v occupies rows [v*node_cap, v*node_cap + N_v) of every per-node array and
 * entries [v*edge_cap, ...) of `indices`; graph g of view v owns rows
 * node_off[v*(B+1)+g] .. node_off[v*(B+1)+g+1).  Row ids inside `indices` are
 * view-local (0..N_v).  The seed of every graph is its first row
 * (data_util.py:226,238).                                                             */
typedef struct {
  int32_t batch;     /* B */
  int32_t node_cap;  /* per view */
  int32_t edge_cap;  /* per view */
  int32_t _pad;
  int32_t* node_off; /* [2][B+1]  node_off[v][B] = N_v                                   */
  int32_t* edge_off; /* [2][B+1]  edge_off[v][B] = E_v                                   */
  int32_t* indptr;   /* [2][node_cap+1] view-local edge offsets                          */
  int32_t* indices;  /* [2][edge_cap]                                                    */
  int32_t* sub_deg;  /* [2][node_cap] in-degree inside the ego-net (graph_encoder.py:154) */
  int32_t* graph_id; /* [2][node_cap] graph index 0..B-1                                  */
  int32_t* orig_id;  /* [2][node_cap] parent vertex id (subv)                             */
  int64_t* counters; /* [2B][4] per ego-net: n, m, recorded walk steps, sum of parent
                        degrees over subv (the induction read volume); slot = v*B+g      */
  int32_t* flags;    /* [1] GCCB_FLAG_* (OR-accumulated; caller clears)                  */
} gccb_batch_t;

/* A2  seed draw.  Replaces LoadBalanceGraphDataset.__iter__ (graph_dataset.py:85-92):
 * np.random.choice(length, p = in_deg^0.75/sum).  cdf = float64 cumulative p (host-built,
 * device-resident); sample i draws 53 Philox bits -> first index with cdf > u.
 * Writes seeds_out[i], sample_ids_out[i] = first_sample + i.                          */
int gccb_draw_seeds(const double* cdf, int64_t n_nodes, uint64_t key, int64_t first_sample,
                    int32_t count, int64_t* seeds_out, int64_t* sample_ids_out,
                    gccb_stream_t stream);

/* A3+A4+A6  random walk with restart, ego-net induction, batching.  Replaces
 * dgl.contrib.sampling.random_walk_with_restart (graph_dataset.py:125-130),
 * _rwr_trace_to_dgl_graph's unique/sort/subgraph (data_util.py:218-239) and
 * dgl.batch (data_util.py:29) for both views of `batch->batch` samples.
 * seeds/sample_ids: [B] (both views start from the same seed: step_dist=[1,0,0]).     */
size_t gccb_sample_batch_workspace(int32_t batch, int32_t max_budget, int32_t edge_cap);
int gccb_sample_batch(const gccb_graph_t* graph, const int64_t* seeds,
                      const int64_t* sample_ids, const gccb_batch_t* batch, void* workspace,
                      size_t workspace_bytes, gccb_stream_t stream);

/* A5  Laplacian positional features.  Replaces
 * _add_undirected_graph_positional_embedding + eigen_decomposision
 * (data_util.py:242-281): top-k (k = min(n-2, pos_dim)) eigenvectors of
 * D^-1/2 A D^-1/2, ascending, row-L2 normalised, zero-padded to pos_dim.
 * pos: [2][node_cap][pos_dim]; eigvals (optional, may be NULL): [2B][pos_dim]
 * ascending top-k eigenvalues (padding = 0).  normalize=0 returns the raw unit
 * eigenvectors (used by the spectral parity tests).
 * Solvers by ego-net size (device-built work lists, csrc/posenc.cu): a dense tridiagonal
 * solver (Householder -> multisection -> inverse iteration; a direct method) for n <= 96,
 * Chebyshev-filtered subspace iteration above.  The environment variable
 * GCCB200_DENSE_MAX (0 .. 228, read on every call) moves that boundary: 0 = subspace
 * iteration / Jacobi for every size, 228 = direct-method accuracy up to 228 vertices.
 * Results are deterministic run to run for a given setting.                              */
size_t gccb_posenc_workspace(int32_t batch, int32_t node_cap);
int gccb_posenc(const gccb_batch_t* batch, int32_t pos_dim, int32_t normalize, float* pos,
                float* eigvals, void* workspace, size_t workspace_bytes,
                gccb_stream_t stream);

/* ---- GIN encoder ----------------------------------------------------------------------
 * Replaces GraphEncoder.forward / UnsupervisedGIN.forward (graph_encoder.py:132-200,
 * gin.py:213-232) incl. DGL GINConv('sum', eps buffer = 0) and SumPooling.
 * Parameters live in ONE flat fp32 buffer; gccb_gin_param_layout gives the layout
 * (the Python module maps the reference's state_dict keys onto slices of it).          */
typedef struct {
  int32_t num_layers;  /* L (GIN layers = L-1, prediction heads = L)  train.py:79 */
  int32_t hidden;      /* node_hidden_dim = output_dim                 train.py:90 */
  int32_t pos_dim;     /* positional_embedding_size (32)                            */
  int32_t deg_dim;     /* degree_embedding_size (16)                                */
  int32_t max_degree;  /* 512                                                       */
  int32_t norm;        /* F.normalize on the output (graph_encoder.py:195-196)     */
  float bn_eps;        /* 1e-5 */
  float bn_momentum;   /* 0.1  */
  float norm_eps;      /* 1e-5 */
  float dropout_p;     /* 0.5 (gin.py:202)                                          */
  int32_t tensor_cores; /* 1: the Linear layers of the MLP (gin.py:107-116) and their input / weight
                           gradients run on tcgen05 tensor cores with bf16 operands and fp32
                           accumulation (hidden >= 128 only; BASELINE config 4); 0: fp32 SIMT  */
  int32_t _pad;
} gccb_gin_cfg_t;

/* offsets (in floats) into the flat parameter buffer; arrays sized for L <= 8 */
typedef struct {
  int64_t w1[8], b1[8], bn1_w[8], bn1_b[8], w2[8], b2[8], bna_w[8], bna_b[8], bnb_w[8], bnb_b[8];
  int64_t wp[8], bp[8];
  int64_t emb;
  int64_t total;     /* number of live floats */
  /* running statistics buffer (separate flat buffer): [layer][bn 0..2][mean|var][hidden] */
  int64_t run_total;
} gccb_gin_layout_t;
int gccb_gin_param_layout(const gccb_gin_cfg_t* cfg, gccb_gin_layout_t* out /* host */);

/* bytes of the activation stash one forward needs for its backward */
size_t gccb_gin_acts_bytes(const gccb_gin_cfg_t* cfg, int32_t batch, int32_t node_cap);

/* forward of ONE view.  bn_running/num_batches_tracked are updated (train-mode BN,
 * train.py:357-365) unless bn_train == 0.  dropout: mask layer ids
 * dropout_layer_base+i, Philox (key, step); dropout_layer_base < 0 = eval dropout.
 * feat: [B][hidden]; pooled_out (optional): [L][B][hidden] (all_outputs).               */
int gccb_gin_forward(const gccb_gin_cfg_t* cfg, const gccb_batch_t* batch, int32_t view,
                     const float* pos, const float* params, float* bn_running,
                     int64_t* num_batches_tracked, int32_t bn_train, uint64_t dropout_key,
                     uint64_t dropout_step, int32_t dropout_layer_base, void* acts,
                     size_t acts_bytes, float* feat, float* pooled_out, gccb_stream_t stream);

/* backward of ONE view (loss.backward(), train.py:408): grads += d loss / d params
 * (flat, same layout; caller zeroes before the first view).  The dropout arguments must
 * repeat the forward's.                                                                 */
size_t gccb_gin_backward_workspace(const gccb_gin_cfg_t* cfg, int32_t batch, int32_t node_cap);
int gccb_gin_backward(const gccb_gin_cfg_t* cfg, const gccb_batch_t* batch, int32_t view,
                      const float* params, const void* acts, const float* dfeat, float* grads,
                      uint64_t dropout_key, uint64_t dropout_step, int32_t dropout_layer_base,
                      void* workspace, size_t workspace_bytes, gccb_stream_t stream);

/* ---- contrastive head ------------------------------------------------------------------ */
/* MemoryMoCo.forward logits (memory_moco.py:33-44): out[B][K+1] = [q.k | q.memory^T] / T */
int gccb_moco_logits(const float* q, const float* k, const float* memory, int32_t B,
                     int32_t d, int32_t K, float T, float* out, gccb_stream_t stream);
/* backward of the above w.r.t. q (k and the queue are detached, memory_moco.py:28,37)    */
int gccb_moco_logits_backward(const float* dout, const float* k, const float* memory,
                              int32_t B, int32_t d, int32_t K, float T, float* dq,
                              gccb_stream_t stream);
/* NCESoftmaxLoss / NCESoftmaxLossNS (criterions.py:12-17, :27-33): mean CE of out[B][C]
 * against label 0 (label_mode 0) or arange(B) (label_mode 1).  dout optional.            */
int gccb_nce_loss(const float* out, int32_t B, int32_t C, int32_t label_mode, float* loss,
                  float* dout, gccb_stream_t stream);
/* fused InfoNCE: loss and dq in one pass over the queue, logits never materialised.
 * stats[0] = loss, stats[1] = mean positive logit ("prob", train.py:394).               */
size_t gccb_infonce_workspace(int32_t B, int32_t d, int32_t K);
int gccb_infonce_fused(const float* q, const float* k, const float* memory, int32_t B,
                       int32_t d, int32_t K, float T, float* stats, float* dq, void* workspace,
                       size_t workspace_bytes, gccb_stream_t stream);
/* FIFO enqueue (memory_moco.py:55-61): memory[(index+i) % K] = k[i]; the write pointer is
 * a device int64 (*index_dev) advanced by parts*B (mod K).  parts > 1: `parts` blocks of B keys,
 * block r at k + r*part_stride floats (every rank's keys inside the gathered exchange buffer, in
 * rank order -> identical queues on all ranks).  skip_word (optional, device): the call is a no-op
 * when (*skip_word & skip_mask) != 0 -- pass gccb_batch_t.flags with
 * GCCB_FLAG_NODE_OVERFLOW|GCCB_FLAG_EDGE_OVERFLOW so that a batch published empty never reaches
 * the queue.                                                                                      */
int gccb_moco_enqueue(float* memory, const float* k, int32_t B, int32_t d, int32_t K,
                      int64_t* index_dev, int32_t parts, int64_t part_stride,
                      const int32_t* skip_word, int32_t skip_mask, gccb_stream_t stream);
/* E2E head (train.py:397-401, criterions.py:27-33): out = k q^T / T, CE vs arange;
 * returns loss, mean diagonal logit, dq and dk.                                          */
int gccb_e2e_nce(const float* q, const float* k, int32_t B, int32_t d, float T, float* stats,
                 float* dq, float* dk, void* workspace /* B*B floats */, size_t workspace_bytes,
                 gccb_stream_t stream);

/* ---- optimiser ------------------------------------------------------------------------- */
/* clip_grad_norm_ (train.py:340-347,409) + Adam with L2 weight decay (train.py:417,667-672)
 * on the first n_live floats, then moment_update (train.py:169-172,430-431) of p_ema over
 * n_all floats (alpha < 0 skips the EMA).  hyper (device, 4 floats): lr, 1-beta1^t,
 * sqrt(1-beta2^t), unused.  grad_norm_out: device float (pre-clip total norm).
 * grad_scale multiplies the gradient first (1/world for data-parallel averaging).
 * skip_word / skip_mask: as for gccb_moco_enqueue -- the whole update (moments, weights, momentum
 * encoder) is a no-op for a step whose batch was published empty.                         */
int gccb_clip_adam_ema(float* p, float* g, float* m, float* v, float* p_ema, int64_t n_live,
                       int64_t n_all, const float* hyper, float beta1, float beta2, float eps,
                       float weight_decay, float clip_norm, float alpha, float grad_scale,
                       float* grad_norm_out, double* workspace /* 1 double */,
                       const int32_t* skip_word, int32_t skip_mask, gccb_stream_t stream);
/* deterministic rank-ordered sum of `world` gathered gradient buffers: out = sum_r in[r].
 * any_flag_out (optional, device int): set to 1 when gathered[r*stride + flag_index] != 0 for any
 * rank r (a rank whose batch overflowed), else 0 -- the skip word of the two calls above when
 * world > 1, so that all replicas skip the same steps and stay identical.                    */
int gccb_sum_ranks(const float* gathered, int32_t world, int64_t stride, int64_t n, float* out,
                   int64_t flag_index, int32_t* any_flag_out, gccb_stream_t stream);

/* ---- tensor-core contraction (tcgen05 + TMEM + TMA; csrc/tc_gemm.cu) ------------------------------
 * The dense products of the path at hidden >= 128 (BASELINE config 4): the GIN MLP's Linear layers
 * (gcc/models/gin.py:107-116) with the BatchNorm column statistics of :115 fused into the epilogue,
 * their input / weight gradients, and the MoCo logits q.queue^T (gcc/contrastive/memory_moco.py:33-44).
 *   out[M x N] = alpha * A[M x K] . B[N x K]^T (+ bias[N])
 * A [M_cap][K] and B [N][K]: bf16, row-major (K contiguous), 16-byte aligned; K % 64 == 0, N % 32 == 0.
 * m_dev (optional): device int with the number of valid rows (<= M_cap), so the row count of a sampled
 * batch never comes back to the host.  out_f32 / out_bf16: [M_cap][ldo] (either may be NULL).
 * colstats (optional): double [2][N], += column sums / sums of squares of the stored values over the
 * valid rows.  splits > 1: split-K over CTAs; the partial products go to `scratch`, which must hold
 * splits * M_cap * N floats (row pitch N), and are added in a fixed order; colstats must be NULL.  A row
 * pitch ldo that is not a multiple of 8 also goes through `scratch` (M_cap * N floats, splits = 1).    */
int gccb_tc_gemm_bf16(const void* A, const void* B, int32_t M_cap, int32_t N, int32_t K,
                      const int32_t* m_dev, const float* bias, float alpha, float* out_f32,
                      void* out_bf16, int32_t ldo, double* colstats, int32_t splits, float* scratch,
                      gccb_stream_t stream);
/* fp32 [rows][lds] -> bf16 [rows_pad][cols_pad] (transpose = 0) or [cols_pad][rows_pad] (transpose = 1),
 * zero padded; rows_dev (optional): device int, rows beyond it are written as zeros.                 */
int gccb_cast_bf16(const float* src, int32_t rows, int32_t cols, int32_t lds, void* dst, int32_t rows_pad,
                   int32_t cols_pad, int32_t transpose, const int32_t* rows_dev, gccb_stream_t stream);

/* ---- frozen-embedding evaluation (csrc/downstream.cu) -----------------------------------------------
 * k-fold scoring of exported embeddings; every (fold, class) or (fold, class pair) problem of a call is
 * solved in ONE launch, one CTA each.  X: float32 [n][d] (the .npy generate.py writes); label: int32 [n]
 * in 0..n_classes-1; fold: int32 [n] in 0..n_folds-1 (row i is a test row of fold fold[i] and a training
 * row of every other fold).  Arithmetic that decides a prediction is fp64.
 * status (per problem): 0 converged, 1 iteration cap reached, 2 (logreg) no further decrease at fp64
 * resolution, 3 / 4 (logreg) class absent from / the only class of the training fold: constant
 * probability 0 / 1 (sklearn's _ConstantPredictor).                                                    */

/* One-vs-rest L2 logistic regression (gcc/tasks/node_classification.py:54-90, TopKRanker(
 * LogisticRegression(C))): problem p = fold*n_classes + class minimises 1/2|w|^2 + C sum log(1 + exp(-s(w.x+b)))
 * over its training rows (intercept unpenalised) by Newton's method with backtracking; stops when
 * lambda^2/2 <= tol * max(1, objective) (Newton decrement) or after max_iter steps.
 * weights: double [n_folds*n_classes][d+1] (w, then b).  prob (optional): double [n][n_classes], the
 * sigmoid probability of every class under the row's own fold model.  pred: int32 [n], the top-1 class
 * (a tie, e.g. probabilities saturated to 1.0, goes to the highest class index).                       */
size_t gccb_logreg_ovr_workspace(int32_t n, int32_t d, int32_t n_classes, int32_t n_folds);
int gccb_logreg_ovr(const float* X, const int32_t* label, const int32_t* fold, int32_t n, int32_t d,
                    int32_t n_classes, int32_t n_folds, double C, int32_t max_iter, double tol,
                    double* weights, double* prob, int32_t* pred, int32_t* status, void* workspace,
                    size_t workspace_bytes, gccb_stream_t stream);

/* RBF C-SVC, one-vs-one (gcc/tasks/graph_classification.py:46-66, SVC(C)): gamma = 1/(d var(X_train))
 * per fold (gamma='scale'), libsvm's SMO with second-order working-set selection, stop when
 * m(alpha) - M(alpha) < eps.  Pairs (ci < cj) in libsvm order, ci is the +1 class; problem
 * p = fold*n_pairs + pair.  gamma: double [n_folds]; coef: double [P][n], y*alpha at the dataset row
 * (0 elsewhere); rho, obj (dual objective): double [P]; dec (optional): double [n][n_pairs], decision
 * values of every row under its own fold; pred: int32 [n], libsvm's vote (f > 0 votes for ci; a tie goes
 * to the lowest class).  n_classes <= 64.  The workspace holds the n x n squared distances (fp32).   */
size_t gccb_svc_ovo_workspace(int32_t n, int32_t n_classes, int32_t n_folds);
int gccb_svc_ovo(const float* X, const int32_t* label, const int32_t* fold, int32_t n, int32_t d,
                 int32_t n_classes, int32_t n_folds, double C, double eps, int64_t max_iter, double* gamma,
                 double* coef, double* rho, double* obj, double* dec, int32_t* pred, int32_t* status,
                 void* workspace, size_t workspace_bytes, gccb_stream_t stream);

/* Similarity-search rank (gcc/tasks/similarity_search.py:40-70): rows E1[idx1[q]] and E2[idx2[q]]
 * (q < m shared keys) are L2-normalised in fp64; rank[q] = number of c < m with
 * score(q, c) > score(q, q), score = e1[q].e2[c].  Recall@k = mean(rank < k).                       */
size_t gccb_sim_rank_workspace(int32_t m, int32_t d);
int gccb_sim_rank(const float* E1, const float* E2, int32_t d, const int32_t* idx1, const int32_t* idx2,
                  int32_t m, int32_t* rank, void* workspace, size_t workspace_bytes, gccb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GCCB200_H_ */
