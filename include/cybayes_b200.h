/*
 * cybayes_b200 -- C ABI of the B200-native Felsenstein-pruning likelihood engine.
 *
 * This is the drop-in boundary for the one hot path of PhyloStar/CyBayes.  The reference
 * has no FFI of its own (it is Cython + NumPy, one process, no device); the functions
 * below are what a reference-side binding for this path binds instead of the bodies of
 *
 *   ML_gamma.matML          (ML_gamma.pyx:7-42)     -> cb_eval (full op list, no input snapshot)
 *   ML_gamma.cache_matML    (ML_gamma.pyx:83-118)   -> cb_eval (dirty-path op list + input snapshot)
 *   ML.matML / cache_matML  (ML.pyx:5-49, 51-83)    -> the same two, context created with n_cats = 1
 *   get_prob_t and friends  (mcmc_gamma.pyx:439-547) -> cb_pmat_build (all edges x categories, one launch)
 *   get_edge_transition_mat (mcmc_gamma.pyx:372-401) -> cb_pmat_build (count = 1..8) or cb_pmat_upload
 *   utils.sites2Mat output  (utils.pyx:94-120)       -> cb_set_tips (state codes instead of 0/1 fp64 matrices)
 *   the final np.sum(np.log(ll)) (ML_gamma.pyx:38,40) -> fused into the root node's kernel
 *   (no reference entry point)                       -> cb_eval_batch: many candidate dirty paths, one launch
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; cb_last_error() gives the
 *     message of the last failure on the calling thread.  There is no CPU fallback: without
 *     a CUDA device cb_create fails.
 *   - all pointers are HOST pointers to caller-owned, C-contiguous buffers that only need to
 *     stay valid for the duration of the call.  Integers are int32_t unless stated, reals are
 *     double.  No torch / numpy types cross this boundary.
 *   - node ids follow the reference: tips 1..n_taxa (file order), internal nodes
 *     n_taxa+1 .. 2*n_taxa-1 (mcmc_gamma.pyx:265-303), the root is whatever the caller names.
 *   - a context is single-threaded (the reference is, utils.pyx:3-7); one context drives one GPU.
 *     Site patterns shard across GPUs as one context (= one process) per GPU with a scalar NCCL
 *     all-reduce per evaluation (cb_comm_init).
 */
#ifndef CYBAYES_B200_H
#define CYBAYES_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CB_MAX_CATS 8

typedef struct cb_ctx cb_ctx;

/* substitution-model kinds for cb_pmat_build */
enum {
  CB_MODEL_JC = 0,         /* ptJC        mcmc_gamma.pyx:507-514 */
  CB_MODEL_F81 = 1,        /* ptF81       mcmc_gamma.pyx:527-547 */
  CB_MODEL_F81_BINARY = 2, /* binaryptF81 mcmc_gamma.pyx:516-525 */
  CB_MODEL_GTR_EIG = 3     /* U exp(lambda d) U^-1; replaces scipy expm at mcmc_gamma.pyx:481 */
};

/* flags for cb_eval */
enum {
  CB_EVAL_WANT_SNAPSHOT = 1, /* keep the recomputed partials and return a new snapshot id      */
  CB_EVAL_STORE_ROOT = 2,    /* also store the root partial (the reference caches it; the fused */
                             /* root kernel does not need it)                                   */
  CB_EVAL_NO_SYNC = 4,       /* enqueue only; the result is read later with cb_result_wait      */
  CB_EVAL_FORCE_LEVELS = 8,  /* never use the single-launch path walk, even for a chain         */
  CB_EVAL_FORCE_WALK = 16,   /* single-launch depth-first walk even on a small alignment (tests)  */
  CB_EVAL_NO_FOLD = 32       /* 2-state family: run cherries as ordinary ops instead of folding them */
};

const char* cb_last_error(void);
int cb_version(void);
int cb_device_count(int* count_out);

/* ---- context ------------------------------------------------------------------------ */
int cb_create(int device, cb_ctx** ctx_out);
int cb_destroy(cb_ctx* ctx);

/* Site-sharded multi-GPU: rank 0 makes a 128-byte NCCL unique id, every rank passes it in.
 * After this, every cb_eval / cb_eval_batch result is the NCCL all-reduced sum over ranks. */
int cb_nccl_unique_id(void* id128_out);
int cb_comm_init(cb_ctx* ctx, const void* id128, int rank, int n_ranks);

/* ---- alignment (leaf data) ------------------------------------------------------------
 * codes[n_taxa][n_sites], uint8 when code_bytes == 1, uint16 when 2: code < n_states is
 * that state (one-hot column of utils.pyx:108-111); code = n_states + k selects row k of
 * amb_sets[n_amb][n_states] (0/1 doubles): k = 0 must be the all-ones set of '?' / '-'
 * (utils.pyx:99-100), further rows are the 'a/b' multi-hot sets (utils.pyx:102-106).
 * weights[n_sites] (NULL = all 1.0) are the site-pattern multiplicities.                */
int cb_set_tips(cb_ctx* ctx, int n_taxa, int64_t n_sites, int n_states, int n_cats,
                const void* codes, int code_bytes, const double* amb_sets, int n_amb,
                const double* weights);

/* Site-pattern compression of a big alignment on the GPU (the reference evaluates every column, utils.pyx:94-120;
 * summing weight * log-likelihood over unique columns is the same number up to summation order): codes as for
 * cb_set_tips.  Outputs: site_to_pattern[n_sites], and for the n_patterns unique columns, in order of first
 * appearance, first_site[] (the column to keep) and weights[] (multiplicities); both sized n_sites by the caller.
 * Exact: equal 128-bit column hashes are verified column by column on the device; a collision is an error.      */
int cb_compress_patterns(int device, const void* codes, int n_taxa, int64_t n_sites, int code_bytes,
                         int64_t* site_to_pattern, int64_t* first_site, double* weights, int64_t* n_patterns_out);

/* ---- transition matrices ---------------------------------------------------------------
 * Device pool of S x S row-major matrices, P[i][j] = Pr(parent i -> child j)
 * (used as P.dot(child) in ML_gamma.pyx:27).  Slot ids are chosen by the caller. */
int cb_pmat_reserve(cb_ctx* ctx, int n_slots);
int cb_pmat_upload(cb_ctx* ctx, int count, const int32_t* slots, const double* mats);
int cb_pmat_download(cb_ctx* ctx, int count, const int32_t* slots, double* mats_out);
/* d[count] = branch length * category rate.  x[count] (may be NULL) = exp(-beta*d) computed by
 * the host libm so JC/F81 matrices equal the reference's bit for bit; NULL = exp on device.
 * gtr = { lambda[S], U[S][S], Uinv[S][S] } for CB_MODEL_GTR_EIG, else NULL.              */
int cb_pmat_build(cb_ctx* ctx, int model, const double* pi, double beta, const double* gtr,
                  int count, const int32_t* slots, const double* d, const double* x);

/* ---- evaluation --------------------------------------------------------------------------
 * An evaluation is a list of node operations in children-before-parents order:
 *   nodes[i]            the internal node recomputed by op i
 *   children[2i..2i+1]  its two children (tip id <= n_taxa, or internal node id)
 *   pslots[(2i+k)*n_cats + c]  P slot of edge (nodes[i], children[2i+k]) for category c
 * An internal child that is not produced by an earlier op of the list is read from
 * snapshot_in (cache_matML's aliasing, ML_gamma.pyx:114).  The last op must be the root.
 * lnL = sum_p w_p * log( sum_c pi . L_root,c[:,p] / n_cats )          (ML_gamma.pyx:38,40)
 * computed with exact power-of-two per-site rescaling (the reference has none).         */
int cb_eval(cb_ctx* ctx, int snapshot_in, int n_ops, const int32_t* nodes,
            const int32_t* children, const int32_t* pslots, const double* pi, int flags,
            int* snapshot_out, double* lnl_out);
/* n_batch independent candidate op lists against the same snapshot, ONE launch (grid.y = candidates).  A
 * candidate is usually a chain (a dirty path: every op after the first consumes the previous op's node); any
 * list whose ops all lie under its last op is accepted (two paths that merge -- an external SPR,
 * mcmc_gamma.pyx:136-185 -- or a whole tree) and walked depth-first.  No snapshot is kept. */
int cb_eval_batch(cb_ctx* ctx, int snapshot_in, int n_batch, const int32_t* op_offsets,
                  const int32_t* nodes, const int32_t* children, const int32_t* pslots,
                  const double* pi, double* lnl_out);
int cb_result_wait(cb_ctx* ctx, double* lnl_out);
/* cb_eval (same op lists, snapshots and flags; CB_EVAL_NO_SYNC is rejected) that also returns the per-site terms of
 * lnL, for site-wise model comparison (WAIC, PSIS-LOO), site-rate estimates and site-wise tree tests.  For pattern p
 * of the context (n_sites = the count given to cb_set_tips: on a sharded context the rank's own slice), with the
 * root partial L_c,p kept as mantissas and one exponent e_p (a power of two, common to the categories):
 *   s_p = sum_c pi . L_c,p / n_cats
 *   site_lnl_out[p]          = log(s_p) + e_p ln 2            (lnL = sum_p w_p site_lnl_out[p], the very terms summed)
 *   cat_post_out[c][p]       = (pi . L_c,p / n_cats) / s_p    (posterior of rate category c, equal priors)
 * cat_post_out may be NULL.  lnl_out equals cb_eval's bit for bit (the same launches and reduction; on a sharded
 * context the all-reduced total).  The root kernel writes l and the category terms, which are copied back once;
 * q is their share of s_p, divided on the host. */
int cb_eval_sites(cb_ctx* ctx, int snapshot_in, int n_ops, const int32_t* nodes, const int32_t* children,
                  const int32_t* pslots, const double* pi, int flags, int* snapshot_out, double* lnl_out,
                  double* site_lnl_out /* [n_sites] */, double* cat_post_out /* [n_cats][n_sites] or NULL */);

/* ---- posterior predictive replicates ------------------------------------------------------
 * Overwrite, in place, every state cell (code < n_states) of the context's alignment with a draw from the model:
 * category uniform over n_cats, root from pi, child from P[slot][parent_state][.]. Ambiguity cells and padding are
 * kept. Edges: parents before children (validated); n_edges = 2 n_taxa - 2, every node but the root the child of one
 * edge. pslots[e * n_cats + c]. Random numbers: Philox4x32-10 with key (seed lo32, seed hi32) and counter
 * (k / 4, column lo32, column hi32, replicate), draw k = output word k % 4; k = 0 the category (x * n_cats) >> 32,
 * k = 1 the root state, k = 1 + child node id the state at that child; a draw is u = (x + 0.5) 2^-32 and picks the
 * first j with u < row[0] + ... + row[j] (fp64, left to right), else n_states - 1.  Column index = column_offset +
 * local column, so the slices of a sharded alignment are slices of one replicate. Fails if the context holds a live
 * snapshot (its partials would describe the old data). codes_out [n_taxa][n_sites] (may be NULL) receives the
 * replicate. */
int cb_simulate(cb_ctx* ctx, int n_edges, const int32_t* parents, const int32_t* children, const int32_t* pslots,
                const double* pi, int root, uint64_t seed, uint32_t replicate, int64_t column_offset,
                void* codes_out);

int cb_snapshot_retain(cb_ctx* ctx, int snapshot);
int cb_snapshot_release(cb_ctx* ctx, int snapshot);
/* out[n_cats][n_states][n_sites] unscaled = stored * 2^scale; scale_out[n_sites] may be NULL,
 * in which case the scaling is folded back into out (may underflow, like the reference). */
int cb_snapshot_read(cb_ctx* ctx, int snapshot, int node, double* out, int32_t* scale_out);

/* ---- native generation loop (SURVEY 8f rank 1) -----------------------------------------------------------
 * The Metropolis-Hastings loop of the reference driver (mat_mcmc_gamma.py:97-221) with its proposal generators
 * (mcmc_gamma.pyx:40-198) run inside the library: cb_chain_run(n) performs n generations -- proposal, P matrices
 * of the touched branches, dirty-path or full evaluation on the GPU, accept test -- without returning to the
 * caller.  For a fixed seed it takes the reference's moves and decisions generation by generation: both random
 * streams (Python `random`, NumPy legacy global generator: MT19937 states handed in and out) and the insertion
 * order of the tree dict are reproduced.  The backend table lets a test replace the CUDA evaluation by callbacks;
 * its three host-maths members are functions whose bits depend on SciPy / BLAS and are therefore always supplied
 * by the caller (discrete-Gamma rates mcmc_gamma.pyx:596-602, beta = 1/(1 - pi.pi) :467, GTR eigensystem).
 * eval_sites (cb_eval_sites without the context) serves cb_chain_site_lnl; NULL = the context's own, which a
 * backend of evaluation callbacks cannot use.                                                                   */
typedef struct cb_chain cb_chain;
typedef struct cb_chain_backend {
  void* user;
  /* NULL = the context's own cb_pmat_build / cb_eval / cb_snapshot_release */
  int (*pmat_build)(void* user, int model, const double* pi, double beta, const double* gtr, int count,
                    const int32_t* slots, const double* d, const double* x);
  int (*eval)(void* user, int snapshot_in, int n_ops, const int32_t* nodes, const int32_t* children,
              const int32_t* pslots, const double* pi, int flags, int* snapshot_out, double* lnl_out);
  int (*snapshot_release)(void* user, int snapshot);
  /* host maths, always required */
  int (*site_rates)(void* user, double alpha, double* rates_out /* n_cats */);
  int (*f81_beta)(void* user, const double* pi, int n_states, double* beta_out);
  int (*gtr_eig)(void* user, const double* pi, const double* exchangeabilities, double* eig_out /* S + 2 S S */);
  int (*eval_sites)(void* user, int snapshot_in, int n_ops, const int32_t* nodes, const int32_t* children,
                    const int32_t* pslots, const double* pi, int flags, int* snapshot_out, double* lnl_out,
                    double* site_lnl_out, double* cat_post_out);
} cb_chain_backend;
/* model: 0 JC, 1 F81, 2 GTR.  param_ids[n_params] in the driver's order (0 pi, 1 rates, 2 tree, 3 bl, 4 srates)
 * with their cumulative normalised weights; tree_cdf[2] = (NNI, eSPR), bl_cdf[2] = (scale_edge, node_slider)
 * (mat_mcmc_gamma.py:65-84).  [slot_base, slot_base + slot_count) is a range of P slots the chain may use as it
 * likes (>= 2 * n_edges * n_cats + 8 * n_cats).                                                                */
int cb_chain_create(cb_ctx* ctx, const cb_chain_backend* backend, int n_taxa, int n_states, int n_cats, int model,
                    int binary, int root, int slot_base, int slot_count, int host_exp_max, int n_params,
                    const int32_t* param_ids, const double* params_cdf, const double* tree_cdf,
                    const double* bl_cdf, cb_chain** chain_out);
/* start state: tree edges in dict insertion order; builds every P matrix and runs the first full evaluation */
int cb_chain_set_state(cb_chain* chain, int n_edges, const int32_t* parents, const int32_t* children,
                       const double* lengths, const double* pi, int n_rates, const double* rates, double alpha,
                       const double* site_rates, double beta, const double* gtr_eig, double* lnl_out);
int cb_chain_set_rng(cb_chain* chain, const uint32_t* py_mt624, int py_pos, const uint32_t* np_mt624, int np_pos);
int cb_chain_get_rng(cb_chain* chain, uint32_t* py_mt624, int* py_pos, uint32_t* np_mt624, int* np_pos);
/* per-generation records (each array n_gens long, any may be NULL): move id (0 scale_edge, 1 node_slider,
 * 2 rooted_NNI, 3 externalSPR, 4 mvDualSlider(pi), 5 scale_alpha, 6 mvDualSlider(rates)), accepted flag, lnL
 * before, proposed lnL, log acceptance ratio, log u */
int cb_chain_run(cb_chain* chain, int64_t n_gens, int8_t* move, int8_t* accepted, double* current_ll,
                 double* proposed_ll, double* ll_ratio, double* log_u);
int cb_chain_get_state(cb_chain* chain, int32_t* parents, int32_t* children, double* lengths, double* pi,
                       double* rates, double* alpha, double* site_rates, double* lnl);
int cb_chain_counters(cb_chain* chain, int64_t* moves7, int64_t* accepts7);
/* Per-site terms of the chain's current state (see cb_eval_sites): one root-only evaluation against the chain's
 * snapshot with its current P matrices and pi.  Between cb_chain_run calls; leaves the chain's random streams,
 * counters, state and snapshot as they are. */
int cb_chain_site_lnl(cb_chain* chain, double* site_lnl_out, double* cat_post_out);
int cb_chain_destroy(cb_chain* chain);

/* ---- introspection / measurement ---------------------------------------------------------- */
int cb_stats(cb_ctx* ctx, int64_t* kernel_launches, int64_t* bytes_h2d, int64_t* bytes_d2h,
             int64_t* device_bytes_in_use);
/* device memory: free / total bytes on the GPU (or under CYBAYES_MAX_DEVICE_BYTES), bytes of partial buffers sitting
 * unused in the context's pool, bytes of one partial buffer -- what the caller needs to decide whether the cache
 * of a full evaluation fits (SURVEY 7: C5's 209 GB cache does not fit one GPU) */
int cb_mem_info(cb_ctx* ctx, int64_t* free_bytes, int64_t* total_bytes, int64_t* pooled_bytes, int64_t* partial_bytes);
/* device time in ms of the kernels of the last synchronous cb_eval / cb_eval_batch
 * (CUDA events on the launching stream) */
int cb_last_eval_ms(cb_ctx* ctx, float* ms_out);
/* ... of its pruning launches alone (without the per-evaluation pre-pass that lays out P matrices / op images) */
int cb_last_eval_main_ms(cb_ctx* ctx, float* ms_out);
/* What the last evaluation had to move, from its op list: bytes of partials (+ exponents) it stored, bytes it
 * read (stored partials read back, tip codes, pattern weights) -- the roofline numerator of bench.py -- and
 * counts8 = { ops run, partials stored, partials read back, children popped from the shared-memory stack,
 * partials stored and re-read inside one launch, cherries folded, pruning launches, small subtrees (children: tips /
 * cherries) kept as records instead of stored partials }. */
int cb_last_eval_info(cb_ctx* ctx, int64_t* bytes_written, int64_t* bytes_read, int32_t* counts8);
/* host microseconds cb_eval / cb_eval_batch have spent since the last reset, by phase: us6 = { plan look-up or build,
 * descriptor fill, upload + launches, wait for the result, snapshot bookkeeping, number of calls } */
int cb_host_profile(cb_ctx* ctx, double* us6, int reset);
/* CUDA events on the engine's stream: cb_mark(ctx, 0) ... work ... cb_mark(ctx, 1); elapsed = device ms */
int cb_mark(cb_ctx* ctx, int which);
int cb_mark_elapsed_ms(cb_ctx* ctx, float* ms_out);
int cb_sync(cb_ctx* ctx);
/* bench helper: FP64 tensor-core (DMMA m8n8k4) peak of this GPU in TFLOP/s, measured from registers */
int cb_fp64_peak(cb_ctx* ctx, double* tflops_out);
/* bench helper: write 256 MB (> the 126 MB L2) to flush it */
int cb_flush_l2(cb_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* CYBAYES_B200_H */
