/* rcmarl.h -- C ABI of librcmarl.so: the sm_100a kernels behind the RPBCAC
 * training hot path (reference: mfigura/Resilient-consensus-based-MARL).
 *
 * The reference has no FFI layer: its boundary is the duck-typed Python Agent
 * API (SURVEY.md 8b).  Each entry point below replaces the TensorFlow/Keras
 * library calls made by one or more reference methods (cited per function);
 * the Python mirror of the reference interface lives in
 * resilient-consensus-based-marl_b200/{agents,training,environments} and binds
 * these symbols with ctypes (INTEGRATION.md shows the stub).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless the name ends in _host;
 *  - no hidden allocation: scratch comes from the caller (`ws`, `ws_bytes`,
 *    see rcmarl_workspace_bytes); all work is stream-ordered on `stream`
 *    (a cudaStream_t passed as void*); no host synchronisation inside;
 *  - return value: 0 on success, negative rcmarl_status otherwise; nothing
 *    throws across the ABI;
 *  - all arithmetic is IEEE fp32 (FFMA on the CUDA cores; no TF32/bf16);
 *  - network parameters are packed in Keras order
 *        [W1(d_in,20) | b1(20) | W2(20,20) | b2(20) | W3(20,n_out) | b3(n_out)]
 *    with y = x @ W + b (main.py:60-82); hidden width is 20, LeakyReLU(0.1);
 *  - the replay buffer is time-major, row = t * n_envs + e (SURVEY App. C):
 *        sa [rows][3*n_agents]  = (x0,y0,a0, x1,y1,a1, ...)   train_agents.py:93
 *        ns [rows][2*n_agents]  = next state                  train_agents.py:90
 *        r  [rows][n_agents]    = scaled local rewards        train_agents.py:91
 */
#ifndef RCMARL_H
#define RCMARL_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RCMARL_HIDDEN 20
#define RCMARL_N_ACTIONS 5
#define RCMARL_MAX_JOBS 32
#define RCMARL_MAX_TERMS 3
#define RCMARL_MAX_NEIGHBOURS 16
#define RCMARL_MAX_H 7
#define RCMARL_MAX_GRID 32

typedef enum {
    RCMARL_OK = 0,
    RCMARL_ERR_ARG = -1,        /* bad argument (null pointer, size, unsupported n_agents/H) */
    RCMARL_ERR_WORKSPACE = -2,  /* workspace too small */
    RCMARL_ERR_CUDA = -3,       /* a CUDA call / launch failed: see rcmarl_last_cuda_error */
    RCMARL_ERR_NO_DEVICE = -4
} rcmarl_status;

/* which part of a buffer row feeds the network (Keras Flatten order) */
typedef enum {
    RCMARL_IN_S = 0,   /* critic / actor on s  : sa without the action column */
    RCMARL_IN_SA = 1,  /* team-reward net on sa                               */
    RCMARL_IN_NS = 2   /* critic on the next state                            */
} rcmarl_input_kind;

/* A set of buffer rows.  Contiguous: time_idx == NULL, rows = [row_begin, row_begin+n_rows).
 * Gathered mini-batch (Appendix C): row(m) = row_begin + time_idx[m / n_envs] * n_envs + m % n_envs. */
typedef struct {
    const float* sa;
    const float* ns;
    const float* r;
    int64_t row_begin;
    int64_t n_rows;
    const int32_t* time_idx;
    int32_t n_envs;
    int32_t n_agents;
} rcmarl_rows;

const char* rcmarl_version(void);
const char* rcmarl_status_string(int status);
int rcmarl_last_cuda_error(void);               /* cudaError_t of the last failure on this thread */
int rcmarl_device_info(int* sm_count, int* cc_major, int* cc_minor);
int64_t rcmarl_param_count(int d_in, int n_out); /* packed length of one network */

/* Scratch needed by the *_grad entry points for `n_jobs` jobs of at most `max_params` parameters. */
int64_t rcmarl_workspace_bytes(int n_jobs, int max_params);

/* How rcmarl_grad / rcmarl_minibatch_sgd would split a one-wave grid of `sm_count` CTAs over `n_jobs` jobs that sweep
 * `n_rows` buffer rows: ctas_host[j] = CTAs of job j (kinds_host[j] = RCMARL_IN_*).  balanced = 0: equal shares (the
 * default of the launchers); 1: shares sized by each job's cost per row (environment switch RCMARL_BALANCED_GRID=1).
 * Host arithmetic only (no device needed); exposed for tests and for sizing experiments. */
int rcmarl_grad_grid_plan(int n_agents, const int32_t* kinds_host, int n_jobs, int loss_mode, int64_t n_rows, int balanced,
                          int sm_count, int32_t* ctas_host);

/* ---------------------------------------------------------------------------
 * K4 / C5.  Coordinate-wise clipped ("winsorised") mean over the neighbour axis,
 * own value = row 0.  Replaces tf.sort/minimum/maximum/clip_by_value/reduce_mean
 * in RPBCAC_agent._resilient_aggregation (agents/resilient_CAC_agents.py:42-58).
 * vals: [n][P] with row stride `row_stride` floats; out: [P].  One streaming read. */
int rcmarl_clip_mean(const float* vals, int n, int64_t P, int64_t row_stride, int H,
                     float* out, void* stream);

/* Hidden-layer parameter consensus for many (agent, net) pairs in one launch:
 * dst[j][0:n_hidden] = clip_mean over k of msgs[in_nodes[j][k]][0:n_hidden]  (own = k 0).
 * Replaces resilient_consensus_critic_hidden / _TR_hidden
 * (agents/resilient_CAC_agents.py:142-166) incl. the neighbour gather at
 * training/train_agents.py:129-130.  The output layer of dst is left untouched (:153). */
typedef struct {
    float* dst;                 /* the agent's own network (packed) */
    const float* msgs;          /* base of the message stack [n_agents][msg_stride] */
    int64_t msg_stride;
    int32_t n_hidden;           /* number of leading parameters to aggregate (W1,b1,W2,b2) */
    int32_t n_in;
    int32_t H;
    int32_t in_nodes[RCMARL_MAX_NEIGHBOURS];
} rcmarl_consensus_job;
int rcmarl_consensus_hidden(const rcmarl_consensus_job* jobs_host, int n_jobs, void* stream);

/* ---------------------------------------------------------------------------
 * K1 / K3.  Batched forward values:  out[row] = add_scale * add[row*add_stride + add_off]
 *                                              + sum_t scale_t * net_t(x_kind_t(row))
 * Replaces critic(ns) / critic(s) / TR(sa) eager calls:
 *   TD target  r + gamma*V(ns)            agents/resilient_CAC_agents.py:114-115, adversarial:131-132,148-149
 *   TD error   TR(sa)+gamma*V(ns)-V(s)    agents/resilient_CAC_agents.py:95-98,  adversarial:113-115
 *   critic(state) logging                 training/train_agents.py:62
 * n_out == RCMARL_N_ACTIONS with `softmax` != 0 gives actor.predict (:215): out[row][5]. */
typedef struct {
    const float* w[RCMARL_MAX_TERMS];
    int32_t kind[RCMARL_MAX_TERMS];
    float scale[RCMARL_MAX_TERMS];
    int32_t n_terms;
    int32_t n_out;              /* 1, or RCMARL_N_ACTIONS (single term only) */
    int32_t softmax;
    int32_t add_off;
    const float* add;           /* optional [rows*add_stride] indexed by absolute buffer row */
    int64_t add_stride;
    float add_scale;
    float* out;                 /* indexed by absolute buffer row */
} rcmarl_value_job;
int rcmarl_values(const rcmarl_rows* rows_host, const rcmarl_value_job* jobs_host, int n_jobs,
                  void* stream);

/* ---------------------------------------------------------------------------
 * K2 / K7 / K9.  Gradient of a summed loss over a row set, for many networks at once.
 *   mode RCMARL_LOSS_MSE:  sum_rows (net(x) - target[row])^2      (Keras MSE * B)
 *   mode RCMARL_LOSS_CE :  sum_rows target[row] * (-log softmax(net(s))[a_row])
 *                          with a_row = sa[row][3*action_agent+2] (Keras weighted sparse CE * B)
 * sums[j] = [ d(loss)/d(theta) (n_params) | loss ]   -- UNSCALED sums, so that a data-parallel
 * all-reduce can be applied before the division by the global batch size.
 * Replaces the forward/backward inside critic.fit / TR.fit / actor.train_on_batch / actor.fit
 * (agents/resilient_CAC_agents.py:99,118,136; adversarial:41,116,133,150,163,224,239,251).
 * max_ctas > 0 plans the grid within that many CTAs (one per SM) instead of the whole GPU (max_ctas = 0), so that other
 * work can run beside it on the remaining SMs (rcmarl_overlap_split). */
typedef enum { RCMARL_LOSS_MSE = 0, RCMARL_LOSS_CE = 1 } rcmarl_loss;
typedef struct {
    const float* w;
    const float* target;        /* regression target / TD-error weight of absolute buffer row `row`:
                                   target[row * target_stride]  (e.g. r + i with stride n_agents) */
    float* sums;                /* [n_params + 1] */
    const int32_t* time_idx;    /* optional per-job override of rows.time_idx (independent fit shuffles) */
    int64_t target_stride;
    int32_t kind;
    int32_t action_agent;       /* CE only */
} rcmarl_grad_job;
int rcmarl_grad(const rcmarl_rows* rows_host, const rcmarl_grad_job* jobs_host, int n_jobs,
                int loss_mode, void* ws, int64_t ws_bytes, int max_ctas, void* stream);

/* theta_dst = theta_src - coef * g   (plain SGD, Keras SGD(lr): coef = lr * 2/B for MSE)
 * loss_out (optional) = loss_coef * g[n]  -- history['loss'][0] bookkeeping. */
typedef struct {
    float* dst;
    const float* src;
    const float* sums;          /* [n - first + 1]: sums for parameters [first, n) then the loss term
                                   (rcmarl_grad: first = 0;  rcmarl_team: first = n - 21) */
    float* loss_out;
    int32_t n;
    int32_t first;              /* only the parameters [first, n) are updated (frozen hidden layers, A.4) */
    float coef;
    float loss_coef;
    int32_t loss_accumulate;    /* 0: *loss_out = loss_coef*g[n];  1: *loss_out += ... (mini-batch epochs) */
    int32_t reserved;
} rcmarl_sgd_job;
int rcmarl_sgd_apply(const rcmarl_sgd_job* jobs_host, int n_jobs, void* stream);

/* K9.  Mini-batch SGD epochs for several networks in lock-step (Keras fit(batch_size=32, epochs=10, shuffle=True),
 * agents/adversarial_CAC_agents.py:133,150,163,239,251): for e < epochs, for each batch b of `mb_times`
 * time rows: rows = { time_idx_j[e*n_times + b*mb_times + i]*n_envs + env }, gradient (rcmarl_grad, MSE), then
 * theta_j -= lr*2/(rows in batch, summed over ranks) * g in place.  Reduction of the CTA partials, the cross-GPU
 * exchange (when an exchange context is bound, see rcmarl_comm_*) and the SGD apply are ONE kernel; the grad kernel
 * of the next step starts its prologue under it (programmatic dependent launch).
 * gjobs[j].time_idx must point at that network's [epochs][n_times] permutation table; sjobs[j].dst == src == gjobs[j].w;
 * sjobs[j].loss_out (optional) accumulates sum(e^2)*loss_coef over epoch 0 only (history['loss'][0]).
 * rows->n_rows / time_idx are ignored.  Without a bound exchange context a data-parallel caller loops over
 * rcmarl_grad / all-reduce / rcmarl_sgd_apply instead. */
int rcmarl_minibatch_sgd(const rcmarl_rows* rows_host, const rcmarl_grad_job* gjobs_host,
                         const rcmarl_sgd_job* sjobs_host, int n_jobs, int epochs, int n_times, int mb_times,
                         float lr, void* ws, int64_t ws_bytes, void* stream);

/* The same fit as ONE persistent kernel (csrc/minibatch_persist.cuh): the CTAs stay resident for all epochs x
 * mini-batches, every chain's parameters live in the shared memory of its CTAs, and the per-step reduction over CTAs
 * (and, with a bound exchange context, over ranks through NVLink peer memory) runs through {value, sequence} cells
 * instead of kernel boundaries -- no launches, no grid barrier, no atomics; results are bitwise reproducible and
 * identical on every rank.  Arguments as rcmarl_minibatch_sgd, except:
 *   sjobs[j].coef > 0 overrides `lr` for chain j (per-agent fast_lr, agents/resilient_CAC_agents.py:36);
 *   cells / cells_bytes: caller-owned scratch of rcmarl_minibatch_cells_bytes() bytes that must be ZERO before the
 *     first call and is otherwise only touched by this entry point;
 *   seq_first >= 1: first of the `rcmarl_minibatch_steps()` consecutive sequence numbers this call consumes; the
 *     caller passes strictly increasing, non-overlapping ranges over the lifetime of `cells`;
 *   max_ctas > 0: the chains share at most that many CTAs (cost-sized shares, as with the whole GPU at max_ctas = 0). */
int64_t rcmarl_minibatch_cells_bytes(int n_jobs, int max_params);
int64_t rcmarl_minibatch_steps(int epochs, int n_times, int mb_times);
int rcmarl_minibatch_fit(const rcmarl_rows* rows_host, const rcmarl_grad_job* gjobs_host,
                         const rcmarl_sgd_job* sjobs_host, int n_jobs, int epochs, int n_times, int mb_times,
                         float lr, void* cells, int64_t cells_bytes, uint32_t seq_first, int max_ctas, void* stream);

/* How an update round may split the GPU between the cooperative agents' full-batch fits (rcmarl_grad: n_fit jobs of kinds
 * fit_kinds_host over fit_rows rows, fit_launches launches per epoch) and the adversaries' mini-batch chains
 * (rcmarl_minibatch_fit: n_chains chains of kinds chain_kinds_host, mb_rows rows per SGD step, mb_steps steps per epoch)
 * when the two run at the same time on two streams of one GPU with sm_count SMs.  budgets_host[0] = max_ctas for the
 * fits, budgets_host[1] = max_ctas for the chains: they sum to at most sm_count, every job and chain gets at least one CTA
 * and the fits' budget is a multiple of n_fit (equal shares).  Both 0: run the phases one after the other on the whole
 * GPU -- when either is empty, world > 1, n_agents != 5 (no measured cost model) or the model predicts too little gain.
 * Host arithmetic only (no device needed). */
int rcmarl_overlap_split(int n_agents, const int32_t* fit_kinds_host, int n_fit, int64_t fit_rows, int fit_launches,
                         const int32_t* chain_kinds_host, int n_chains, int64_t mb_rows, int64_t mb_steps, int world,
                         int sm_count, int32_t* budgets_host);

/* Keras/TF-2 Adam (SURVEY Appendix A.5): m,v updated in place, theta -= lr_t*m/(sqrt(v)+eps);
 * g = grad_scale * sums.  lr_t = lr*sqrt(1-b2^t)/(1-b1^t) is computed by the caller. */
typedef struct {
    float* theta;
    float* m;
    float* v;
    const float* sums;
    float* loss_out;
    int32_t n;
    float grad_scale;
    float lr_t;
    float beta1, beta2, eps;
    float loss_coef;
    int32_t loss_accumulate;
    int32_t reserved;
} rcmarl_adam_job;
int rcmarl_adam_apply(const rcmarl_adam_job* jobs_host, int n_jobs, void* stream);

/* ---------------------------------------------------------------------------
 * K5 + K6 fused.  Per row: phi = features(x) with the agent's (aggregated) hidden layers;
 * est_k = phi . W3_k + b3_k for each neighbour head k (own first); agg = clip_mean_k(est, H);
 * projection step on the agent's own output layer:
 *   sums[0:21] = sum_rows (agg - (phi.W3_own + b3_own)) * [phi;1] / (||phi||^2 + 1)
 * so that theta_out += sums / B reproduces train_on_batch with sample weights
 * 1/(2 lr (||phi||^2+1)).  Replaces resilient_consensus_critic/_TR and
 * critic_update_team/TR_update_team (agents/resilient_CAC_agents.py:60-84,168-206).
 * agg_out (optional) stores agg per absolute row; agg_in (optional) supplies it instead. */
typedef struct {
    const float* w;             /* agent's network: aggregated hidden + current own head */
    const float* msgs;          /* message stack base (heads are read at the W3/b3 offsets) */
    int64_t msg_stride;
    float* sums;                /* [21 + 1] : projection numerators | sum (agg-pred)^2 * weight */
    float* agg_out;
    const float* agg_in;
    int32_t kind;
    int32_t n_in;
    int32_t H;
    int32_t in_nodes[RCMARL_MAX_NEIGHBOURS];
} rcmarl_team_job;
int rcmarl_team(const rcmarl_rows* rows_host, const rcmarl_team_job* jobs_host, int n_jobs,
                void* ws, int64_t ws_bytes, void* stream);

/* out[row] = scale * sum over listed agents of r[row][i] / n_listed, accumulated in list order
 * (r_coop, training/train_agents.py:96-98; scale = -1 gives the Malicious agent's -r_coop, :115-116). */
int rcmarl_reward_mix(const float* r, int64_t n_rows, int n_agents, const int32_t* agents_host,
                      int n_listed, float scale, float* out, void* stream);

/* ---------------------------------------------------------------------------
 * Data parallelism over environment shards (SURVEY 8e): one process per GPU of ONE node.  A bound exchange context
 * makes rcmarl_grad / rcmarl_team / rcmarl_minibatch_sgd return (and apply) sums over ALL ranks: the per-CTA partials
 * are reduced, exchanged through NVLink peer memory (CUDA IPC buffers, one-shot all-reduce, rank-ordered summation =>
 * bitwise identical results on every rank) and, for the mini-batch path, applied -- all inside ONE kernel
 * (csrc/comm.cuh).  Every rank must issue the same sequence of those calls.  Without a bound context the caller
 * all-reduces `sums` itself (e.g. NCCL) between rcmarl_grad and the apply.
 *   create(rank, world <= 8, capacity) -> export a 64-byte IPC handle -> exchange handles out of band (e.g.
 *   torch.distributed.all_gather_object) -> connect(all handles, rank-major) -> bind. */
int rcmarl_comm_create(int rank, int world, int64_t max_floats, void** comm_out);
int rcmarl_comm_handle_bytes(void);
int rcmarl_comm_export(void* comm, void* handle_out_host);
int rcmarl_comm_connect(void* comm, const void* handles_host);
int rcmarl_comm_bind(void* comm);                /* NULL unbinds */
int rcmarl_comm_error(void* comm);               /* 1 if a peer wait timed out (synchronises the device) */
int rcmarl_comm_destroy(void* comm);

/* ---------------------------------------------------------------------------
 * K1 + K8.  A block of episodes under a fixed policy for n_envs environments
 * (training/train_agents.py:46-80 + environments/grid_world.py:37-72 +
 * get_action, agents/resilient_CAC_agents.py:208-219): one thread per (episode, env).
 * Randomness: Philox4x32-10 keyed by (seed, env_offset+env, episode_offset+episode, step, agent)
 * or, for parity tests, injected through `uniforms` / `init_state`. */
typedef struct {
    const float* actor_w;       /* [n_agents][P_actor] */
    const float* critic_w;      /* [n_agents][P_critic] for the est_returns log (train_agents.py:62) */
    const int32_t* desired;     /* [n_agents][2] */
    float* sa; float* ns; float* r;     /* buffer bases */
    int64_t time_begin;         /* first time row written */
    float* est;                 /* [n_episodes][n_envs][n_agents] critic(state_0) */
    float* ret;                 /* [n_episodes][n_envs][n_agents] discounted returns */
    const float* uniforms;      /* optional [n_episodes][max_ep_len][n_envs][n_agents][3] */
    const int32_t* init_state;  /* optional [n_episodes][n_envs][n_agents][2] */
    uint64_t seed;
    int64_t env_offset;         /* global index of local env 0 (data-parallel shards) */
    int64_t episode_offset;
    int32_t n_envs, n_agents, n_episodes, max_ep_len;
    int32_t nrow, ncol;
    float gamma, mu;
    int32_t n_active;           /* agents 0 .. n_active-1 exist (main.py:26 --n_agents); the remaining slots of the
                                   5- / 16-agent instantiation are written as zeros.  0 means n_agents. */
    int32_t reserved;
    float state_tab_x[RCMARL_MAX_GRID];   /* (i-mean)/std, rounded from float64 by the host */
    float state_tab_y[RCMARL_MAX_GRID];
} rcmarl_rollout_args;
int rcmarl_rollout(const rcmarl_rollout_args* args_host, void* stream);

/* Means over the environments of the per-episode logs written by rcmarl_rollout (`est`, `ret`: [n_episodes][n_envs][n_agents])
 * -> out [n_episodes][n_agents]: what training/train_agents.py:168-180 prints and stores per episode, for N environments. */
int rcmarl_episode_means(const float* x, int n_episodes, int n_envs, int n_agents, float* out, void* stream);

/* One transition of Grid_World.step + get_data for n_envs environments
 * (environments/grid_world.py:47-72): state int32 [n_envs][n_agents][2] updated in place. */
int rcmarl_env_step(int32_t* state, const float* action, const int32_t* desired, int n_envs,
                    int n_agents, int nrow, float* reward_scaled, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RCMARL_H */
