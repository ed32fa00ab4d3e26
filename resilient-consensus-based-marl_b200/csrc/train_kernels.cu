// train_kernels.cu -- update-round kernels of the RPBCAC hot path (sm_100a, fp32 FFMA).
//
//   values_kernel   K1/K3  batched forward values / TD targets / TD errors / actor probabilities
//   grad_kernel     K2/K7/K9  fused forward + backward of the 20-wide MLPs over a row set (grad_kernel.cuh):
//                   phase 1: two buffer rows per lane, weights broadcast from shared memory;
//                   phase 2: the per-row activation / delta vectors are staged in a warp-private
//                            shared-memory tile and every lane owns one 8x8 tile of the weight-gradient
//                            outer products, accumulated in registers across ALL rows of the CTA;
//                   deterministic two-level reduction (CTA partials -> reduce_kernel).
//   team_kernel     K5+K6  neighbour-head estimates, clipped mean, projection numerators
//   consensus, sgd/adam apply, reward mix: the small glue kernels.
//
// Reference semantics: agents/resilient_CAC_agents.py, agents/adversarial_CAC_agents.py,
// training/train_agents.py:86-163 (cited per entry point in include/rcmarl.h).
#include <stdlib.h>
#include "common.cuh"
#include "grad_kernel.cuh"
#define RC_GRAD_KERNEL grad_kernel
#define RC_GRAD_WARPS grad_warps
#define RC_GRAD_SMEM grad_smem_floats
// RCMARL_GRAD_WS (default 1): mean-squared-error jobs at n_agents = 5 run on the warp-specialised tensor-core kernel
// (grad_kernel_ws.cuh); -DRCMARL_GRAD_WS=0 (make variant_ffma) keeps them on the FFMA2 kernel of round 1 (grad_kernel.cuh)
#ifndef RCMARL_GRAD_WS
#define RCMARL_GRAD_WS 1
#endif
#if RCMARL_GRAD_WS
#include "grad_kernel_ws.cuh"
#endif
#include "comm.cuh"
#include "minibatch_persist.cuh"

namespace rcmarl {

static thread_local int g_last_cuda = 0;
int last_cuda_error_get() { return g_last_cuda; }
void last_cuda_error_set(int e) { g_last_cuda = e; }

int sm_count_cached() {
    static int n = 0;
    if (n == 0) {
        int dev = 0, v = 0;
        if (cudaGetDevice(&dev) == cudaSuccess &&
            cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && v > 0)
            n = v;
        else
            return 148;  // B200; not cached so that a later call with a device re-queries
    }
    return n;
}

// ============================================================================================
// values
// ============================================================================================
struct ValuesParams {
    rcmarl_rows rows;
    rcmarl_value_job jobs[RCMARL_MAX_JOBS];
};

// value of R = 2 rows per thread: every broadcast weight quad feeds both rows (see grad_kernel.cuh)
template <int NA, int DIN>
__device__ __forceinline__ void value_term2(const rcmarl_rows& R, const float* sw, int kind, const int64_t (&row)[2],
                                            float (&v)[2]) {
    float x[2][DIN], h1[2][HID], h2[2][HID];
    load_x<NA, DIN>(R, kind, row[0], x[0]);
    load_x<NA, DIN>(R, kind, row[1], x[1]);
    features_rows<DIN, 2>(sw, x, h1, h2);
    v[0] = head1<DIN>(sw, h2[0]);
    v[1] = head1<DIN>(sw, h2[1]);
}

template <int NA>
__global__ void __launch_bounds__(256) values_kernel(const __grid_constant__ ValuesParams P) {
    extern __shared__ __align__(16) float smem[];
    const rcmarl_value_job& job = P.jobs[blockIdx.y];
    const rcmarl_rows& R = P.rows;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t n_iter = (R.n_rows + stride - 1) / stride;
    if (job.n_out == NACT) {  // actor.predict: softmax probabilities (single term)
        constexpr int DIN = 2 * NA;
        stage_weights(smem, job.w[0], param_count(DIN, NACT));
        __syncthreads();
        for (int64_t it = 0; it < n_iter; ++it) {
            int64_t m = it * stride + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
            if (m < R.n_rows) {
                int64_t row = row_of(R, m);
                float x[DIN], h1[HID], h2[HID], l[NACT], mx, lse;
                load_x<NA, DIN>(R, job.kind[0], row, x);
                features<DIN>(smem, x, h1, h2);
                head5<DIN>(smem, h2, l);
                if (job.softmax) softmax5(l, mx, lse);
#pragma unroll
                for (int o = 0; o < NACT; ++o) job.out[row * NACT + o] = l[o];
            }
        }
        return;
    }
    for (int t = 0; t < job.n_terms; ++t) {
        const int kind = job.kind[t];
        __syncthreads();
        stage_weights(smem, job.w[t], kind == RCMARL_IN_SA ? param_count(3 * NA, 1) : param_count(2 * NA, 1));
        __syncthreads();
        for (int64_t it = 0; it < n_iter; it += 2) {          // two rows per thread and iteration
            int64_t m[2], row[2];
            bool live[2];
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                m[r] = (it + r) * stride + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
                live[r] = (it + r) < n_iter && m[r] < R.n_rows;
                row[r] = row_of(R, live[r] ? m[r] : 0);
            }
            if (!live[0]) continue;
            float v[2];
            if (kind == RCMARL_IN_SA) value_term2<NA, 3 * NA>(R, smem, kind, row, v);
            else value_term2<NA, 2 * NA>(R, smem, kind, row, v);
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                if (!live[r]) continue;
                float acc;
                if (t == 0)
                    acc = job.add ? job.add_scale * __ldg(job.add + row[r] * job.add_stride + job.add_off) : 0.f;
                else
                    acc = job.out[row[r]];
                job.out[row[r]] = fmaf(job.scale[t], v[r], acc);
            }
        }
    }
}

// Where the CTA partials of job j live: slots first[j] + y * step, y = 0 .. count[j] - 1, each `stride` floats
// (grad_kernel: consecutive slots of the 1-D grid; team_kernel: [y][job] interleaved).
struct PartialSlots {
    int32_t first[RCMARL_MAX_JOBS];
    int32_t count[RCMARL_MAX_JOBS];
    int32_t step, stride;
};

// Deterministic sum over the CTA partials of one parameter, parallel over the 8 warps of a 256-thread block:
// block b of job j owns parameters [32 b, 32 b + 32); warp w adds y = w, w + 8, ... (coalesced 128-byte rows), the
// eight warp sums are combined in warp order.  Returns the total in the threads of warp 0 (others return 0).
__device__ __forceinline__ float block_partial_sum(const float* __restrict__ partial, const PartialSlots& S, int j, int i,
                                                   bool valid, float* sh /* [8][32] */) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int first = S.first[j], count = S.count[j];
    float s = 0.f;
    if (valid)
        for (int y = warp; y < count; y += 8) s += partial[((int64_t)first + (int64_t)y * S.step) * S.stride + i];
    sh[warp * 32 + lane] = s;
    __syncthreads();
    float tot = 0.f;
    if (warp == 0) {
#pragma unroll
        for (int w = 0; w < 8; ++w) tot += sh[w * 32 + lane];
    }
    return tot;
}

// sums[j][i] = sum_y partial[y][j][i], y ascending (deterministic)
struct ReduceParams {
    const float* partial;
    float* sums[RCMARL_MAX_JOBS];
    int32_t n[RCMARL_MAX_JOBS];
    PartialSlots slots;
};
__global__ void __launch_bounds__(256) reduce_kernel(const __grid_constant__ ReduceParams P) {
    __shared__ float sh[256];
    pdl_launch_dependents();     // the next grad kernel may start its prologue; it waits (pdl_wait) before reading
    const int j = blockIdx.y;
    const int i = blockIdx.x * 32 + (threadIdx.x & 31);
    const bool valid = i < P.n[j];
    const float s = block_partial_sum(P.partial, P.slots, j, i, valid, sh);
    if (threadIdx.x < 32 && valid) P.sums[j][i] = s;
}

// fused: sums[j][i] = sum_y partial[y][j][i]; theta = theta - coef * sums (mini-batch SGD step, single GPU)
struct ReduceSgdParams {
    const float* partial;
    rcmarl_sgd_job jobs[RCMARL_MAX_JOBS];
    PartialSlots slots;
};
__global__ void __launch_bounds__(256) reduce_sgd_kernel(const __grid_constant__ ReduceSgdParams P) {
    __shared__ float sh[256];
    pdl_launch_dependents();     // the next grad kernel may start its prologue; it waits (pdl_wait) before reading
#if RCMARL_PDL_REDUCE
    pdl_wait();                  // launched as a programmatic dependent of the grad kernel: its partials must be complete
#endif
    const rcmarl_sgd_job& job = P.jobs[blockIdx.y];
    const int i = blockIdx.x * 32 + (threadIdx.x & 31);
    const bool valid = i <= job.n;
    const float s = block_partial_sum(P.partial, P.slots, blockIdx.y, i, valid, sh);
    if (threadIdx.x >= 32 || !valid) return;
    if (i < job.n) {
        const float v = job.src[i];
        job.dst[i] = i >= job.first ? v - job.coef * s : v;
    } else if (job.loss_out) {
        const float l = job.loss_coef * s;
        *job.loss_out = job.loss_accumulate ? *job.loss_out + l : l;
    }
}

// Multi-GPU variant: reduce the CTA partials, exchange over NVLink peer memory (comm.cuh), write the global sums and
// optionally apply the SGD step -- one kernel, no NCCL call, no host round trip.
struct ReduceCommParams {
    const float* partial;
    float* sums[RCMARL_MAX_JOBS];
    int32_t n[RCMARL_MAX_JOBS];
    rcmarl_sgd_job sgd[RCMARL_MAX_JOBS];
    PartialSlots slots;
    int32_t out_stride, fuse_sgd;     // out_stride: distance between the jobs' blocks in the exchange buffer
    int32_t n_jobs, max_n;            // items = n_jobs x ceil(max_n / 32)
    CommDev comm;
};
__global__ void __launch_bounds__(256) reduce_comm_kernel(const __grid_constant__ ReduceCommParams P) {
    __shared__ float sh[256];
    pdl_launch_dependents();     // the next grad kernel may start its prologue; it waits (pdl_wait) before reading
#if RCMARL_PDL_REDUCE
    pdl_wait();
#endif
    // One item = 32 consecutive elements of one job.  Items are independent (comm.cuh): a CTA walks its items in
    // ascending order on every rank, so any grid size is deadlock-free and nothing has to be co-resident.
    const int blocks_per_job = (P.max_n + 31) / 32;
    const int n_items = blocks_per_job * P.n_jobs;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        const int j = item / blocks_per_job;
        const int i = (item - j * blocks_per_job) * 32 + (threadIdx.x & 31);
        const bool valid = i < P.n[j];
        const int64_t off = (int64_t)j * P.out_stride + i;
        const float s = block_partial_sum(P.partial, P.slots, j, i, valid, sh);
        if (threadIdx.x < 32 && valid) {
            comm_push(P.comm, off, s);
            const float tot = comm_wait_total(P.comm, off);
            if (P.sums[j]) P.sums[j][i] = tot;
            if (P.fuse_sgd) {
                const rcmarl_sgd_job& job = P.sgd[j];
                if (i < job.n) {
                    const float v = job.src[i];
                    job.dst[i] = i >= job.first ? v - job.coef * tot : v;
                } else if (i == job.n && job.loss_out) {
                    const float l = job.loss_coef * tot;
                    *job.loss_out = job.loss_accumulate ? *job.loss_out + l : l;
                }
            }
        }
        __syncthreads();          // sh[] is reused by the next item
    }
}

// grid of reduce_comm_kernel: one CTA per item up to two resident CTAs per SM
static dim3 reduce_comm_grid(int max_n, int n_jobs) {
    const int items = ((max_n + 31) / 32) * n_jobs;
    const int cap = sm_count_cached() * 2;
    return dim3(items < cap ? items : cap);
}

// ============================================================================================
// team: estimates + clipped mean + projection numerators
// ============================================================================================
struct TeamParams {
    rcmarl_rows rows;
    rcmarl_team_job jobs[RCMARL_MAX_JOBS];
    float* partial;
    int32_t n_jobs;
    int32_t stride;
    // jobs of THIS launch (blockIdx.x -> job index).  rcmarl_team launches the team-reward nets (15 inputs) and the critics
    // (10 inputs) separately: the loop body of one instantiation is ~24 KB of SASS, two of them resident on an SM overflow the
    // 32 KB instruction cache (28 % of the stall samples were "no instruction", profiles/r02_ncu_other_kernels.md)
    int32_t job_list[RCMARL_MAX_JOBS];
};
constexpr int TEAM_N = HID + 2;  // 20 weights + bias numerators + diagnostic loss

// MAXN: compile-time bound on the neighbour count (4 / 8 / 16) so that the estimate vector and the rank-counting
// order statistics stay in registers without paying for 16 x 16 predicated compares when n_in = 4
template <int NA, int DIN, int MAXN>
__device__ __forceinline__ void team_body(const TeamParams& P, const rcmarl_team_job& job, float* smem) {
    constexpr int NP = param_count(DIN, 1);
    const rcmarl_rows& R = P.rows;
    float* sw = smem;                       // agent's network
    float* heads = smem + round4(NP);       // [n_in][24]: W3 (20), b3, pad
    stage_weights(sw, job.w, NP);
    for (int i = threadIdx.x; i < job.n_in * 24; i += blockDim.x) {
        const int k = i / 24, j = i % 24;
        const float* m = job.msgs + (int64_t)job.in_nodes[k] * job.msg_stride;
        heads[i] = j < HID ? __ldg(m + off_W3(DIN) + j) : (j == HID ? __ldg(m + off_b3(DIN, 1)) : 0.f);
    }
    __syncthreads();
    float acc[TEAM_N];
#pragma unroll
    for (int j = 0; j < TEAM_N; ++j) acc[j] = 0.f;
    const int64_t stride = (int64_t)gridDim.y * blockDim.x;
    const int64_t n_iter = (R.n_rows + stride - 1) / stride;
    for (int64_t it = 0; it < n_iter; it += 2) {                   // two rows per thread and iteration
        int64_t row[2];
        bool live[2];
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int64_t m = (it + r) * stride + (int64_t)blockIdx.y * blockDim.x + threadIdx.x;
            live[r] = (it + r) < n_iter && m < R.n_rows;
            row[r] = row_of(R, live[r] ? m : 0);
        }
        if (!live[0]) continue;
        float phi[2][HID];
        {
            float x[2][DIN], h1[2][HID];
            load_x<NA, DIN>(R, job.kind, row[0], x[0]);
            load_x<NA, DIN>(R, job.kind, row[1], x[1]);
            features_rows<DIN, 2>(sw, x, h1, phi);
        }
        float agg[2];
        if (job.agg_in) {
            agg[0] = __ldg(job.agg_in + row[0]);
            agg[1] = __ldg(job.agg_in + row[1]);
        } else {
            float est[2][MAXN];
#pragma unroll
            for (int k = 0; k < MAXN; ++k) {
                est[0][k] = 0.f;
                est[1][k] = 0.f;
                if (k < job.n_in) {
                    const float* hk = heads + k * 24;
                    float s0 = hk[HID], s1 = hk[HID];
#pragma unroll
                    for (int j = 0; j < HID; ++j) { s0 = fmaf(phi[0][j], hk[j], s0); s1 = fmaf(phi[1][j], hk[j], s1); }
                    est[0][k] = s0;
                    est[1][k] = s1;
                }
            }
            agg[0] = clip_mean_small<MAXN>(est[0], job.n_in, job.H);
            agg[1] = clip_mean_small<MAXN>(est[1], job.n_in, job.H);
        }
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            if (!live[r]) continue;
            if (job.agg_out) job.agg_out[row[r]] = agg[r];
            if (job.sums) {
                const float pred = head1<DIN>(sw, phi[r]);
                float nrm = 1.f;
#pragma unroll
                for (int j = 0; j < HID; ++j) nrm = fmaf(phi[r][j], phi[r][j], nrm);
                const float err = agg[r] - pred;
                const float c = err / nrm;
#pragma unroll
                for (int j = 0; j < HID; ++j) acc[j] = fmaf(c, phi[r][j], acc[j]);
                acc[HID] += c;
                acc[HID + 1] = fmaf(err, c, acc[HID + 1]);
            }
        }
    }
    if (!job.sums) return;
    __syncthreads();
    float* red = smem;  // [nwarps][TEAM_N]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
#pragma unroll
    for (int j = 0; j < TEAM_N; ++j) {
        float s = warp_sum(acc[j]);
        if (lane == 0) red[warp * TEAM_N + j] = s;
    }
    __syncthreads();
    if (threadIdx.x < TEAM_N) {
        float s = 0.f;
        for (int w = 0; w < nwarps; ++w) s += red[w * TEAM_N + threadIdx.x];
        P.partial[((int64_t)blockIdx.y * P.n_jobs + P.job_list[blockIdx.x]) * P.stride + threadIdx.x] = s;
    }
}

template <int NA>
__global__ void __launch_bounds__(128) team_kernel(const __grid_constant__ TeamParams P) {
    extern __shared__ __align__(16) float smem[];
    const rcmarl_team_job& job = P.jobs[P.job_list[blockIdx.x]];
    const bool sa = job.kind == RCMARL_IN_SA;
    if (job.n_in <= 4) {
        if (sa) team_body<NA, 3 * NA, 4>(P, job, smem); else team_body<NA, 2 * NA, 4>(P, job, smem);
    } else if (job.n_in <= 8) {
        if (sa) team_body<NA, 3 * NA, 8>(P, job, smem); else team_body<NA, 2 * NA, 8>(P, job, smem);
    } else {
        if (sa) team_body<NA, 3 * NA, 16>(P, job, smem); else team_body<NA, 2 * NA, 16>(P, job, smem);
    }
}

// ============================================================================================
// small kernels
// ============================================================================================
struct ConsensusParams { rcmarl_consensus_job jobs[RCMARL_MAX_JOBS]; };
__global__ void __launch_bounds__(256) consensus_hidden_kernel(const __grid_constant__ ConsensusParams P) {
    const rcmarl_consensus_job& job = P.jobs[blockIdx.y];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= job.n_hidden) return;
    float v[RCMARL_MAX_NEIGHBOURS];
#pragma unroll
    for (int k = 0; k < RCMARL_MAX_NEIGHBOURS; ++k)
        v[k] = k < job.n_in ? __ldg(job.msgs + (int64_t)job.in_nodes[k] * job.msg_stride + i) : 0.f;
    job.dst[i] = clip_mean_small<RCMARL_MAX_NEIGHBOURS>(v, job.n_in, job.H);
}

struct SgdParams { rcmarl_sgd_job jobs[RCMARL_MAX_JOBS]; };
__global__ void __launch_bounds__(256) sgd_kernel(const __grid_constant__ SgdParams P) {
    const rcmarl_sgd_job& job = P.jobs[blockIdx.y];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < job.n) {
        const float s = job.src[i];
        job.dst[i] = i >= job.first ? s - job.coef * job.sums[i - job.first] : s;
    }
    if (i == 0 && job.loss_out) {
        const float l = job.loss_coef * job.sums[job.n - job.first];
        *job.loss_out = job.loss_accumulate ? *job.loss_out + l : l;
    }
}

struct AdamParams { rcmarl_adam_job jobs[RCMARL_MAX_JOBS]; };
__global__ void __launch_bounds__(256) adam_kernel(const __grid_constant__ AdamParams P) {
    const rcmarl_adam_job& job = P.jobs[blockIdx.y];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < job.n) {
        const float g = job.grad_scale * job.sums[i];
        const float m = job.beta1 * job.m[i] + (1.f - job.beta1) * g;
        const float v = job.beta2 * job.v[i] + (1.f - job.beta2) * g * g;
        job.m[i] = m;
        job.v[i] = v;
        job.theta[i] = job.theta[i] - job.lr_t * m / (sqrtf(v) + job.eps);
    }
    if (i == 0 && job.loss_out) {
        const float l = job.loss_coef * job.sums[job.n];
        *job.loss_out = job.loss_accumulate ? *job.loss_out + l : l;
    }
}

struct MixParams { int32_t agents[RCMARL_MAX_JOBS]; };
__global__ void __launch_bounds__(256) reward_mix_kernel(const float* __restrict__ r, int64_t n_rows, int n_agents,
                                                         const __grid_constant__ MixParams P, int n_listed,
                                                         float scale, float* __restrict__ out) {
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n_rows) return;
    const float inv = (float)n_listed;
    float s = 0.f;
    for (int k = 0; k < n_listed; ++k) s = s + __ldg(r + row * n_agents + P.agents[k]) / inv;  // train_agents.py:98
    out[row] = scale * s;
}

// ============================================================================================
// host-side launchers
// ============================================================================================
template <typename K>
static int set_smem(K kernel, size_t bytes) {
    if (bytes > 48 * 1024) RC_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return 0;
}

static int check_rows(const rcmarl_rows* r) {
    if (!r || !r->sa || !r->ns || !r->r || r->n_rows < 0 || r->n_envs <= 0) return RCMARL_ERR_ARG;
    if (r->n_agents != 5 && r->n_agents != 16) return RCMARL_ERR_ARG;
    if (r->time_idx && (r->n_rows % r->n_envs) != 0) return RCMARL_ERR_ARG;
    return 0;
}

template <int NA>
static int launch_values(const ValuesParams& P, int n_jobs, cudaStream_t st) {
    const size_t smem = sizeof(float) * round4(param_count(3 * NA, 1) > param_count(2 * NA, NACT)
                                                   ? param_count(3 * NA, 1) : param_count(2 * NA, NACT));
    if (set_smem(values_kernel<NA>, smem)) return RCMARL_ERR_CUDA;
    int64_t gx = (P.rows.n_rows + 255) / 256;
    const int64_t cap = (int64_t)sm_count_cached() * 2;   // 2 resident CTAs per SM (126 registers x 256 threads)
    if (gx > cap) gx = cap;
    if (gx < 1) gx = 1;
    values_kernel<NA><<<dim3((unsigned)gx, n_jobs), 256, smem, st>>>(P);
    RC_CUDA(cudaGetLastError());
    return 0;
}

template <int NA>
static int launch_grad(GradParams& P, int loss_mode, int n_ctas, cudaStream_t st) {
    constexpr int NWM = RC_GRAD_WARPS<NA, RCMARL_LOSS_MSE>(), NWC = RC_GRAD_WARPS<NA, RCMARL_LOSS_CE>();
    constexpr size_t smem_mse = sizeof(float) * (RC_GRAD_SMEM<NA, 3 * NA, 1, NWM>() > RC_GRAD_SMEM<NA, 2 * NA, 1, NWM>()
                                                     ? RC_GRAD_SMEM<NA, 3 * NA, 1, NWM>() : RC_GRAD_SMEM<NA, 2 * NA, 1, NWM>());
    constexpr size_t smem_ce = sizeof(float) * RC_GRAD_SMEM<NA, 2 * NA, NACT, NWC>();
    static_assert(smem_mse <= 227 * 1024 && smem_ce <= 227 * 1024, "grad kernel exceeds the 227 KB shared-memory limit");
    static bool attr_ce = false, attr_mse = false;     // opt-in to > 48 KB dynamic shared memory once per process
    cudaLaunchAttribute pdl;
    pdl.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    pdl.val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(n_ctas);
    cfg.stream = st;
    cfg.attrs = &pdl;
    cfg.numAttrs = 1;
    if (loss_mode == RCMARL_LOSS_CE) {
        if (!attr_ce) {
            if (set_smem(RC_GRAD_KERNEL<NA, RCMARL_LOSS_CE>, smem_ce)) return RCMARL_ERR_CUDA;
            attr_ce = true;
        }
        cfg.blockDim = dim3(32 * NWC);
        cfg.dynamicSmemBytes = smem_ce;
        RC_CUDA(cudaLaunchKernelEx(&cfg, RC_GRAD_KERNEL<NA, RCMARL_LOSS_CE>, P));
#if RCMARL_GRAD_WS
    } else if (NA == 5) {
        constexpr size_t smem_ws = sizeof(float) * ws_smem_floats();
        static_assert(smem_ws <= 227 * 1024, "grad_kernel_ws exceeds the shared-memory limit");
        static bool attr_ws = false;
        if (!attr_ws) {
            if (set_smem(grad_kernel_ws, smem_ws)) return RCMARL_ERR_CUDA;
            attr_ws = true;
        }
        cfg.blockDim = dim3(WS_THREADS);
        cfg.dynamicSmemBytes = smem_ws;
        RC_CUDA(cudaLaunchKernelEx(&cfg, grad_kernel_ws, P));
#endif
    } else {
        if (!attr_mse) {
            if (set_smem(RC_GRAD_KERNEL<NA, RCMARL_LOSS_MSE>, smem_mse)) return RCMARL_ERR_CUDA;
            attr_mse = true;
        }
        cfg.blockDim = dim3(32 * NWM);
        cfg.dynamicSmemBytes = smem_mse;
        RC_CUDA(cudaLaunchKernelEx(&cfg, RC_GRAD_KERNEL<NA, RCMARL_LOSS_MSE>, P));
    }
    RC_CUDA(cudaGetLastError());
    return 0;
}

// chunks (64 rows) one CTA of this configuration consumes per sweep
template <int NA>
static int grad_chunks_per_cta(int loss_mode) {
#if RCMARL_GRAD_WS
    if (NA == 5 && loss_mode == RCMARL_LOSS_MSE) return 2;      // one 128-row tile (= two 64-row chunks) at a time
#endif
    return loss_mode == RCMARL_LOSS_CE ? RC_GRAD_WARPS<NA, RCMARL_LOSS_CE>() : RC_GRAD_WARPS<NA, RCMARL_LOSS_MSE>();
}

template <int NA>
static int launch_team(const TeamParams& P, int n_list, int gy, cudaStream_t st) {
    const size_t smem = sizeof(float) * (round4(param_count(3 * NA, 1)) + RCMARL_MAX_NEIGHBOURS * 24 + 8 * TEAM_N);
    if (set_smem(team_kernel<NA>, smem)) return RCMARL_ERR_CUDA;
    team_kernel<NA><<<dim3(n_list, gy), 128, smem, st>>>(P);
    RC_CUDA(cudaGetLastError());
    return 0;
}

// launch of the fused reduce kernels of the mini-batch loop; with RCMARL_PDL_REDUCE as a programmatic dependent of the
// grad kernel before it (the kernel itself waits for that grid with griddepcontrol.wait)
template <typename K, typename PT>
static int launch_reduce(K kernel, const PT& params, dim3 grid, cudaStream_t st) {
#if RCMARL_PDL_REDUCE
    cudaLaunchAttribute pdl;
    pdl.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    pdl.val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(256);
    cfg.stream = st;
    cfg.attrs = &pdl;
    cfg.numAttrs = 1;
    RC_CUDA(cudaLaunchKernelEx(&cfg, kernel, params));
#else
    kernel<<<grid, 256, 0, st>>>(params);
#endif
    RC_CUDA(cudaGetLastError());
    return 0;
}

static int grid_y_for(int64_t work_items, int n_jobs, int ctas_per_sm) {
    // one resident wave at most: gridDim.x * gridDim.y <= SMs * CTAs-per-SM (a partial second wave would
    // double the kernel time of these persistent, equal-work CTAs)
    int64_t cap = ((int64_t)sm_count_cached() * ctas_per_sm) / n_jobs;
    if (cap < 1) cap = 1;
    int64_t gy = work_items < cap ? work_items : cap;
    return (int)(gy < 1 ? 1 : gy);
}

// Shares of the one-wave, 1-D grid of grad_kernel: job j owns the CTAs [cta_first[j], cta_first[j + 1]).
// Default: equal shares, floor(SMs / n_jobs) CTAs per job (all jobs then sweep the rows in lock-step, which keeps the
// buffer rows they share in L2).  RCMARL_BALANCED_GRID=1 in the environment sizes the shares by cost instead: a job's
// cost per row depends on its network (grad_row_cost) and a CTA works in rounds of `gw` 64-row chunks, so with 148 SMs
// 4 team-reward + 4 critic jobs get 19 + 18 CTAs each instead of 18 + 18, and the 3 chains of a malicious agent
// 48 / 52 / 48 instead of 49 each (the team-reward job then needs 5 rounds instead of 6); greedy: the job that currently
// finishes last gets the next CTA.  Measured on B200 (profiles/r01_late_variants.md, run 3): -1.2 % / -2.2 % on isolated
// full-batch / mini-batch launches but +1.5 % on the C2 update round, so it stays opt-in until that is understood.
#ifndef RCMARL_MB_EQUAL_SHARES
#define RCMARL_MB_EQUAL_SHARES 0
#endif
#ifndef RCMARL_BALANCED_GRID_DEFAULT
#define RCMARL_BALANCED_GRID_DEFAULT 0
#endif
static bool balanced_grid_enabled() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("RCMARL_BALANCED_GRID");
        v = e ? (e[0] != '0') : RCMARL_BALANCED_GRID_DEFAULT;
    }
    return v != 0;
}

// g[j] = CTAs of job j; pure host arithmetic (also behind rcmarl_grad_grid_plan for the CPU tests)
static void plan_shares(int n, const int* cost, int64_t nchunks, int gw, int sms, bool balanced, int* g) {
    int64_t units = (nchunks + gw - 1) / gw;
    if (units < 1) units = 1;
    if (!balanced || n == 1 || n > sms) {
        int64_t gy = sms / n;
        if (gy < 1) gy = 1;
        if (gy > units) gy = units;
        for (int j = 0; j < n; ++j) g[j] = (int)gy;
    } else {
        int used = n;
        for (int j = 0; j < n; ++j) g[j] = 1;
        while (used < sms) {
            int best = -1;
            int64_t best_t = -1;
            for (int j = 0; j < n; ++j) {
                if (g[j] >= units) continue;
                const int64_t per_round = (int64_t)g[j] * gw;
                const int64_t t = ((nchunks + per_round - 1) / per_round) * cost[j];
                if (t > best_t || (t == best_t && g[j] < g[best])) { best_t = t; best = j; }
            }
            if (best < 0) break;
            ++g[best];
            ++used;
        }
    }
}

// CTAs a launcher may plan with: the caller's budget (max_ctas > 0), at most the whole GPU (max_ctas = 0)
static int cta_budget(int max_ctas) {
    const int sms = sm_count_cached();
    return max_ctas > 0 && max_ctas < sms ? max_ctas : sms;
}

static int plan_grad_grid(GradParams& P, PartialSlots& S, const int* cost, int64_t nchunks, int gw, int sms) {
    const int n = P.n_jobs;
    int g[RCMARL_MAX_JOBS];
    plan_shares(n, cost, nchunks, gw, sms, balanced_grid_enabled(), g);
    int first = 0;
    for (int j = 0; j < n; ++j) {
        P.cta_first[j] = (int16_t)first;
        S.first[j] = first;
        S.count[j] = g[j];
        first += g[j];
    }
    P.cta_first[n] = (int16_t)first;
    S.step = 1;
    return first;
}

static int grad_job_cost(int na, int kind, int loss_mode) {
    if (loss_mode == RCMARL_LOSS_CE) return grad_row_cost(2 * na, NACT);
    return grad_row_cost(kind == RCMARL_IN_SA ? 3 * na : 2 * na, 1);
}

#if RCMARL_GRAD_WS
static int launch_mb_persist_ws(const MbParams& P, int n_ctas, cudaStream_t st) {
    constexpr size_t smem = sizeof(float) * ws_smem_floats();
    static int resident = -1;
    if (resident < 0) {
        if (set_smem(mb_persist_ws_kernel, smem)) return RCMARL_ERR_CUDA;
        int per_sm = 0;
        RC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mb_persist_ws_kernel, WS_THREADS, smem));
        resident = per_sm * sm_count_cached();
    }
    if (n_ctas > resident) return RCMARL_ERR_ARG;
    cudaLaunchAttribute pdl;
    pdl.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    pdl.val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(n_ctas);
    cfg.blockDim = dim3(WS_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cfg.attrs = &pdl;
    cfg.numAttrs = 1;
    RC_CUDA(cudaLaunchKernelEx(&cfg, mb_persist_ws_kernel, P));
    RC_CUDA(cudaGetLastError());
    return 0;
}
#endif


template <int NA>
static int launch_mb_persist(const MbParams& P, int n_ctas, cudaStream_t st) {
    constexpr int NW = grad_warps<NA, RCMARL_LOSS_MSE>();
    constexpr size_t smem = sizeof(float) * (grad_smem_floats<NA, 3 * NA, 1, NW>() > grad_smem_floats<NA, 2 * NA, 1, NW>()
                                                 ? grad_smem_floats<NA, 3 * NA, 1, NW>() : grad_smem_floats<NA, 2 * NA, 1, NW>());
    static int resident = -1;                          // CTAs that can be co-resident (the cells protocol needs all of them)
    if (resident < 0) {
        if (set_smem(mb_persist_kernel<NA>, smem)) return RCMARL_ERR_CUDA;
        int per_sm = 0;
        RC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mb_persist_kernel<NA>, 32 * NW, smem));
        resident = per_sm * sm_count_cached();
    }
    if (n_ctas > resident) return RCMARL_ERR_ARG;
    cudaLaunchAttribute pdl;
    pdl.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    pdl.val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(n_ctas);
    cfg.blockDim = dim3(32 * NW);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cfg.attrs = &pdl;
    cfg.numAttrs = 1;
    RC_CUDA(cudaLaunchKernelEx(&cfg, mb_persist_kernel<NA>, P));
    RC_CUDA(cudaGetLastError());
    return 0;
}

// Cost model of rcmarl_overlap_split, per launch of a warp-specialised tensor-core kernel (n_agents = 5):
//   time = fixed + per_tile * max over jobs of (128-row tiles of one CTA of the job * grad_row_cost of the job).
// Constants from the round-2 measurements at the C2 shapes on one B200 (profiles/r02_kernel_experiments.md,
// profiles/r02_bench_c2.json): rcmarl_grad over 12 288 000 rows x 8 jobs, 5.73 ms at 18 CTAs per job; a step of
// rcmarl_minibatch_fit (3 chains x 131 072 rows), 39.2 us at 48 / 52 / 48 CTAs, of which ~11.6 us fixed tail.
// tools/prof_overlap.py measures both at smaller budgets and refits them.  Running at the same time costs the two phases
// some of each other's L2 and HBM bandwidth, which the model leaves out; kOverlapMinGain keeps them serial unless the
// predicted saving clears that.
static constexpr double kFitFixedNs = 30000.0, kFitTileNs = 0.494;     // rcmarl_grad: launch + reduce; ns per tile x cost
static constexpr double kMbFixedNs = 11600.0, kMbTileNs = 0.61;        // one step of rcmarl_minibatch_fit: tail; sweep
static constexpr double kOverlapMinGain = 0.02;

// time of one launch in which job j sweeps `units` tiles with g[j] CTAs
static double shares_time(int n, const int* cost, const int* g, int64_t units, double fixed_ns, double tile_ns) {
    int64_t worst = 0;
    for (int j = 0; j < n; ++j) {
        const int64_t t = (units + g[j] - 1) / g[j] * cost[j];
        if (t > worst) worst = t;
    }
    return fixed_ns + tile_ns * (double)worst;
}

}  // namespace rcmarl

using namespace rcmarl;

extern "C" {

int64_t rcmarl_workspace_bytes(int n_jobs, int max_params) {
    if (n_jobs < 1) n_jobs = 1;
    const int64_t ctas = (int64_t)sm_count_cached() * 2 + 2 * (int64_t)n_jobs;
    return ctas * (int64_t)(max_params + 1) * (int64_t)sizeof(float);
}

int rcmarl_grad_grid_plan(int n_agents, const int32_t* kinds_host, int n_jobs, int loss_mode, int64_t n_rows, int balanced,
                          int sm_count, int32_t* ctas_host) {
    if ((n_agents != 5 && n_agents != 16) || !kinds_host || !ctas_host || n_jobs < 1 || n_jobs > RCMARL_MAX_JOBS ||
        n_rows < 0 || sm_count < 1 || (loss_mode != RCMARL_LOSS_MSE && loss_mode != RCMARL_LOSS_CE))
        return RCMARL_ERR_ARG;
    int cost[RCMARL_MAX_JOBS], g[RCMARL_MAX_JOBS];
    for (int j = 0; j < n_jobs; ++j) {
        if (kinds_host[j] < 0 || kinds_host[j] > 2) return RCMARL_ERR_ARG;
        cost[j] = grad_job_cost(n_agents, kinds_host[j], loss_mode);
    }
    const int cpc = n_agents == 5 ? grad_chunks_per_cta<5>(loss_mode) : grad_chunks_per_cta<16>(loss_mode);
    plan_shares(n_jobs, cost, (n_rows + 63) / 64, cpc, sm_count, balanced != 0, g);
    for (int j = 0; j < n_jobs; ++j) ctas_host[j] = g[j];
    return RCMARL_OK;
}

int rcmarl_overlap_split(int n_agents, const int32_t* fit_kinds_host, int n_fit, int64_t fit_rows, int fit_launches,
                         const int32_t* chain_kinds_host, int n_chains, int64_t mb_rows, int64_t mb_steps, int world,
                         int sm_count, int32_t* budgets_host) {
    if ((n_agents != 5 && n_agents != 16) || !budgets_host || n_fit < 0 || n_fit > RCMARL_MAX_JOBS || n_chains < 0 ||
        n_chains > RCMARL_MAX_JOBS || (n_fit && !fit_kinds_host) || (n_chains && !chain_kinds_host) || fit_rows < 0 ||
        fit_launches < 0 || mb_rows < 0 || mb_steps < 0 || world < 1 || sm_count < 1)
        return RCMARL_ERR_ARG;
    int fit_cost[RCMARL_MAX_JOBS], mb_cost[RCMARL_MAX_JOBS], gf[RCMARL_MAX_JOBS], gm[RCMARL_MAX_JOBS];
    for (int j = 0; j < n_fit; ++j) {
        if (fit_kinds_host[j] < 0 || fit_kinds_host[j] > 2) return RCMARL_ERR_ARG;
        fit_cost[j] = grad_job_cost(n_agents, fit_kinds_host[j], RCMARL_LOSS_MSE);
    }
    for (int j = 0; j < n_chains; ++j) {
        if (chain_kinds_host[j] < 0 || chain_kinds_host[j] > 2) return RCMARL_ERR_ARG;
        mb_cost[j] = grad_job_cost(n_agents, chain_kinds_host[j], RCMARL_LOSS_MSE);
    }
    budgets_host[0] = budgets_host[1] = 0;
    // serial: nothing to overlap; the 16-agent kernels are not covered by the cost model; with world > 1 both phases would
    // draw sequence numbers from the one cell region of the peer-memory exchange, whose call order must match on every rank
    if (n_fit == 0 || n_chains == 0 || fit_rows == 0 || fit_launches == 0 || mb_rows == 0 || mb_steps == 0 ||
        n_agents != 5 || world > 1 || sm_count < n_fit + n_chains)
        return RCMARL_OK;
    const int cpc = grad_chunks_per_cta<5>(RCMARL_LOSS_MSE);
    const int64_t fit_chunks = (fit_rows + 63) / 64, mb_chunks = (mb_rows + 63) / 64;
    const int64_t fit_units = (fit_chunks + cpc - 1) / cpc, mb_units = (mb_chunks + cpc - 1) / cpc;
    auto fit_ns = [&](int ctas) {
        plan_shares(n_fit, fit_cost, fit_chunks, cpc, ctas, false, gf);
        return (double)fit_launches * shares_time(n_fit, fit_cost, gf, fit_units, kFitFixedNs, kFitTileNs);
    };
    auto mb_ns = [&](int ctas) {
        plan_shares(n_chains, mb_cost, mb_chunks, cpc, ctas, true, gm);
        return (double)mb_steps * shares_time(n_chains, mb_cost, gm, mb_units, kMbFixedNs, kMbTileNs);
    };
    const double serial = fit_ns(sm_count) + mb_ns(sm_count);
    double best = serial;
    // equal shares: only multiples of n_fit are worth giving the fits; the chains take every other CTA
    for (int f = n_fit; f <= sm_count - n_chains; f += n_fit) {
        const double t = fit_ns(f) > mb_ns(sm_count - f) ? fit_ns(f) : mb_ns(sm_count - f);
        if (t < best) { best = t; budgets_host[0] = f; budgets_host[1] = sm_count - f; }
    }
    if (best > serial * (1.0 - kOverlapMinGain)) budgets_host[0] = budgets_host[1] = 0;
    return RCMARL_OK;
}

int rcmarl_values(const rcmarl_rows* rows, const rcmarl_value_job* jobs, int n_jobs, void* stream) {
    if (int e = check_rows(rows)) return e;
    if (!jobs || n_jobs < 1 || n_jobs > RCMARL_MAX_JOBS) return RCMARL_ERR_ARG;
    if (rows->n_rows == 0) return RCMARL_OK;
    ValuesParams P;
    P.rows = *rows;
    for (int j = 0; j < n_jobs; ++j) {
        const rcmarl_value_job& q = jobs[j];
        if (!q.out || q.n_terms < 1 || q.n_terms > RCMARL_MAX_TERMS) return RCMARL_ERR_ARG;
        if (q.n_out != 1 && !(q.n_out == NACT && q.n_terms == 1 && q.kind[0] != RCMARL_IN_SA)) return RCMARL_ERR_ARG;
        for (int t = 0; t < q.n_terms; ++t)
            if (!q.w[t] || q.kind[t] < 0 || q.kind[t] > 2) return RCMARL_ERR_ARG;
        P.jobs[j] = q;
    }
    cudaStream_t st = (cudaStream_t)stream;
    return rows->n_agents == 5 ? launch_values<5>(P, n_jobs, st) : launch_values<16>(P, n_jobs, st);
}

int rcmarl_grad(const rcmarl_rows* rows, const rcmarl_grad_job* jobs, int n_jobs, int loss_mode, void* ws,
                int64_t ws_bytes, int max_ctas, void* stream) {
    if (int e = check_rows(rows)) return e;
    if (!jobs || n_jobs < 1 || n_jobs > RCMARL_MAX_JOBS || !ws || max_ctas < 0) return RCMARL_ERR_ARG;
    if (loss_mode != RCMARL_LOSS_MSE && loss_mode != RCMARL_LOSS_CE) return RCMARL_ERR_ARG;
    const int NA = rows->n_agents;
    GradParams P;
    ReduceParams Q;
    P.rows = *rows;
    int maxn = 0;
    int cost[RCMARL_MAX_JOBS];
    for (int j = 0; j < n_jobs; ++j) {
        const rcmarl_grad_job& q = jobs[j];
        if (!q.w || !q.target || !q.sums || q.kind < 0 || q.kind > 2 || q.target_stride < 1) return RCMARL_ERR_ARG;
        if (q.time_idx && !rows->time_idx) return RCMARL_ERR_ARG;   /* overrides need the gathered row mode */
        if (loss_mode == RCMARL_LOSS_CE && (q.kind != RCMARL_IN_S || q.action_agent < 0 || q.action_agent >= NA))
            return RCMARL_ERR_ARG;
        P.jobs[j] = q;
        const int n = loss_mode == RCMARL_LOSS_CE ? param_count(2 * NA, NACT)
                                                   : param_count(q.kind == RCMARL_IN_SA ? 3 * NA : 2 * NA, 1);
        Q.sums[j] = q.sums;
        Q.n[j] = n + 1;
        cost[j] = grad_job_cost(NA, q.kind, loss_mode);
        if (n + 1 > maxn) maxn = n + 1;
    }
    const int64_t nchunks = (rows->n_rows + 63) / 64;
    const int cpc = NA == 5 ? grad_chunks_per_cta<5>(loss_mode) : grad_chunks_per_cta<16>(loss_mode);
    P.partial = (float*)ws;
    P.n_jobs = n_jobs;
    P.stride = maxn;
    Q.slots.stride = maxn;
    const int n_ctas = plan_grad_grid(P, Q.slots, cost, nchunks, cpc, cta_budget(max_ctas));
    if ((int64_t)n_ctas * maxn * (int64_t)sizeof(float) > ws_bytes) return RCMARL_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    int e = NA == 5 ? launch_grad<5>(P, loss_mode, n_ctas, st) : launch_grad<16>(P, loss_mode, n_ctas, st);
    if (e) return e;
    Q.partial = (const float*)ws;
    if (comm_bound()) {
        ReduceCommParams C;
        if (!comm_next(&C.comm, (int64_t)n_jobs * maxn)) return RCMARL_ERR_ARG;
        C.partial = Q.partial; C.slots = Q.slots; C.out_stride = maxn; C.fuse_sgd = 0; C.n_jobs = n_jobs; C.max_n = maxn;
        for (int j = 0; j < n_jobs; ++j) { C.sums[j] = Q.sums[j]; C.n[j] = Q.n[j]; }
        if (launch_reduce(reduce_comm_kernel, C, reduce_comm_grid(maxn, n_jobs), st)) return RCMARL_ERR_CUDA;
    } else {
        reduce_kernel<<<dim3((maxn + 31) / 32, n_jobs), 256, 0, st>>>(Q);
    }
    RC_CUDA(cudaGetLastError());
    return RCMARL_OK;
}

int rcmarl_minibatch_sgd(const rcmarl_rows* rows, const rcmarl_grad_job* gjobs, const rcmarl_sgd_job* sjobs, int n_jobs,
                         int epochs, int n_times, int mb_times, float lr, void* ws, int64_t ws_bytes, void* stream) {
    if (!rows || !rows->sa || !rows->ns || !rows->r || rows->n_envs <= 0) return RCMARL_ERR_ARG;
    if (rows->n_agents != 5 && rows->n_agents != 16) return RCMARL_ERR_ARG;
    if (!gjobs || !sjobs || n_jobs < 1 || n_jobs > RCMARL_MAX_JOBS || !ws || epochs < 1 || n_times < 1 || mb_times < 1)
        return RCMARL_ERR_ARG;
    const int NA = rows->n_agents;
    GradParams P;
    ReduceSgdParams Q;
    P.rows = *rows;
    int maxn = 0;
    int cost[RCMARL_MAX_JOBS];
    for (int j = 0; j < n_jobs; ++j) {
        const rcmarl_grad_job& q = gjobs[j];
        if (!q.w || !q.target || !q.time_idx || q.kind < 0 || q.kind > 2 || q.target_stride < 1) return RCMARL_ERR_ARG;
        if (!sjobs[j].dst || sjobs[j].dst != sjobs[j].src || (const float*)sjobs[j].dst != q.w) return RCMARL_ERR_ARG;
        const int n = param_count(q.kind == RCMARL_IN_SA ? 3 * NA : 2 * NA, 1);
        if (sjobs[j].n != n) return RCMARL_ERR_ARG;
        P.jobs[j] = q;
        Q.jobs[j] = sjobs[j];
        cost[j] = grad_job_cost(NA, q.kind, RCMARL_LOSS_MSE);
        if (n + 1 > maxn) maxn = n + 1;
    }
    P.partial = (float*)ws;
    P.n_jobs = n_jobs;
    P.stride = maxn;
    Q.partial = (const float*)ws;
    Q.slots.stride = maxn;
    int n_ctas = 0, planned_cnt = -1;
    cudaStream_t st = (cudaStream_t)stream;
    const int cpc = NA == 5 ? grad_chunks_per_cta<5>(RCMARL_LOSS_MSE) : grad_chunks_per_cta<16>(RCMARL_LOSS_MSE);
    for (int e = 0; e < epochs; ++e) {
        for (int b = 0; b < n_times; b += mb_times) {
            const int cnt = n_times - b < mb_times ? n_times - b : mb_times;
            const int64_t n_rows = (int64_t)cnt * rows->n_envs;
            P.rows.n_rows = n_rows;
            if (cnt != planned_cnt) {                        // the grid only depends on the mini-batch size
                n_ctas = plan_grad_grid(P, Q.slots, cost, (n_rows + 63) / 64, cpc, sm_count_cached());
                if ((int64_t)n_ctas * maxn * (int64_t)sizeof(float) > ws_bytes) return RCMARL_ERR_WORKSPACE;
                planned_cnt = cnt;
            }
            for (int j = 0; j < n_jobs; ++j) {
                P.jobs[j].time_idx = gjobs[j].time_idx + (int64_t)e * n_times + b;
                Q.jobs[j].coef = lr * 2.0f / (float)n_rows;
                if (e > 0) Q.jobs[j].loss_out = nullptr;
            }
            P.rows.time_idx = P.jobs[0].time_idx;
            int err = NA == 5 ? launch_grad<5>(P, RCMARL_LOSS_MSE, n_ctas, st) : launch_grad<16>(P, RCMARL_LOSS_MSE, n_ctas, st);
            if (err) return err;
            if (comm_bound()) {
                ReduceCommParams C;
                if (!comm_next(&C.comm, (int64_t)n_jobs * maxn)) return RCMARL_ERR_ARG;
                C.partial = Q.partial; C.slots = Q.slots; C.out_stride = maxn; C.fuse_sgd = 1; C.n_jobs = n_jobs; C.max_n = maxn;
                for (int j = 0; j < n_jobs; ++j) {
                    C.sums[j] = nullptr;
                    C.n[j] = Q.jobs[j].n + 1;
                    C.sgd[j] = Q.jobs[j];
                    C.sgd[j].coef = lr * 2.0f / ((float)n_rows * (float)C.comm.world);   // global batch
                }
                if (launch_reduce(reduce_comm_kernel, C, reduce_comm_grid(maxn, n_jobs), st)) return RCMARL_ERR_CUDA;
            } else {
                if (launch_reduce(reduce_sgd_kernel, Q, dim3((maxn + 31) / 32, n_jobs), st)) return RCMARL_ERR_CUDA;
            }
        }
    }
    return RCMARL_OK;
}

int64_t rcmarl_minibatch_cells_bytes(int n_jobs, int max_params) {
    if (n_jobs < 1) n_jobs = 1;
    // level 1: one row of cells per CTA (<= SMs); level 2 (single GPU): 2 slots x n_jobs rows; + the error word
    // (sized generously: a row per CTA AND chain)
    return ((int64_t)sm_count_cached() * (int64_t)n_jobs + 2 * (int64_t)n_jobs) * (int64_t)(max_params + 1) * (int64_t)sizeof(uint2) + 64;
}

int64_t rcmarl_minibatch_steps(int epochs, int n_times, int mb_times) {
    if (epochs < 1 || n_times < 1 || mb_times < 1) return 0;
    return (int64_t)epochs * ((n_times + mb_times - 1) / mb_times);
}

int rcmarl_minibatch_fit(const rcmarl_rows* rows, const rcmarl_grad_job* gjobs, const rcmarl_sgd_job* sjobs, int n_jobs,
                         int epochs, int n_times, int mb_times, float lr, void* cells, int64_t cells_bytes,
                         uint32_t seq_first, int max_ctas, void* stream) {
    if (!rows || !rows->sa || !rows->ns || !rows->r || rows->n_envs <= 0) return RCMARL_ERR_ARG;
    if (rows->n_agents != 5 && rows->n_agents != 16) return RCMARL_ERR_ARG;
    if (!gjobs || !sjobs || n_jobs < 1 || n_jobs > RCMARL_MAX_JOBS || !cells || epochs < 1 || n_times < 1 || mb_times < 1 ||
        seq_first < 1 || max_ctas < 0)
        return RCMARL_ERR_ARG;
    const int NA = rows->n_agents;
    MbParams P;
    P.rows = *rows;
    P.rows.n_rows = 0;
    P.rows.time_idx = nullptr;
    int maxn = 0;
    int cost[RCMARL_MAX_JOBS];
    for (int j = 0; j < n_jobs; ++j) {
        const rcmarl_grad_job& q = gjobs[j];
        if (!q.w || !q.target || !q.time_idx || q.kind < 0 || q.kind > 2 || q.target_stride < 1) return RCMARL_ERR_ARG;
        if (!sjobs[j].dst || sjobs[j].dst != sjobs[j].src || (const float*)sjobs[j].dst != q.w) return RCMARL_ERR_ARG;
        const int n = param_count(q.kind == RCMARL_IN_SA ? 3 * NA : 2 * NA, 1);
        if (sjobs[j].n != n || sjobs[j].first != 0) return RCMARL_ERR_ARG;
        MbChain& c = P.chains[j];
        c.w = sjobs[j].dst; c.target = q.target; c.time_idx = q.time_idx; c.loss_out = sjobs[j].loss_out;
        c.target_stride = q.target_stride; c.lr = sjobs[j].coef > 0.f ? sjobs[j].coef : lr;
        c.loss_coef = sjobs[j].loss_coef; c.kind = q.kind; c.loss_accumulate = sjobs[j].loss_accumulate;
#if RCMARL_GRAD_WS && RCMARL_MB_EQUAL_SHARES
        // experiment (off): equal shares on the tensor-core core (50 / 49 / 49 CTAs at C2 instead of the cost model's 48 / 52 / 48).
        // Measured slower, 41.0 vs 40.1 us per step: the team-reward chain (15 inputs to load per row) is the slower one per tile
        // and wants its 20-tile share (profiles/r02_kernel_experiments.md)
        cost[j] = NA == 5 ? 1 : grad_job_cost(NA, q.kind, RCMARL_LOSS_MSE);
#else
        cost[j] = grad_job_cost(NA, q.kind, RCMARL_LOSS_MSE);
#endif
        if (n + 1 > maxn) maxn = n + 1;
    }
    const int cpc = NA == 5 ? grad_chunks_per_cta<5>(RCMARL_LOSS_MSE) : grad_chunks_per_cta<16>(RCMARL_LOSS_MSE);
    const int64_t n_rows_mb = (int64_t)(n_times < mb_times ? n_times : mb_times) * rows->n_envs;
    // CTA shares by cost (the chains do not share rows in L2 the way the lock-step full-batch jobs do).  A mapping with every
    // CTA serving every chain in turn (reduction of a chain hidden behind the other chains' turns) measured 70 instead of 46 us
    // per step and was removed (profiles/r02_kernel_experiments.md).
    int n_ctas = 0;
    {
        int g[RCMARL_MAX_JOBS];
        plan_shares(n_jobs, cost, (n_rows_mb + 63) / 64, cpc, cta_budget(max_ctas), true, g);
        for (int j = 0; j < n_jobs; ++j) { P.cta_first[j] = (int16_t)n_ctas; n_ctas += g[j]; }
        P.cta_first[n_jobs] = (int16_t)n_ctas;
    }
    P.n_chains = n_jobs; P.epochs = epochs; P.n_times = n_times; P.mb_times = mb_times; P.stride = maxn;
    const int64_t steps = rcmarl_minibatch_steps(epochs, n_times, mb_times);
    if ((uint64_t)seq_first + (uint64_t)steps >= 0xFFFFFFFFull) return RCMARL_ERR_ARG;
    const int64_t l1 = (int64_t)n_ctas * maxn, l2 = 2 * (int64_t)n_jobs * maxn;
    if ((l1 + l2) * (int64_t)sizeof(uint2) + 64 > cells_bytes) return RCMARL_ERR_WORKSPACE;
    if (((uintptr_t)cells & 15) != 0) return RCMARL_ERR_ARG;
    P.cells1 = (uint2*)cells;
    P.seq1 = seq_first;
    if (comm_bound()) {
        if (!comm_reserve(&P.comm, (int64_t)n_jobs * maxn, (uint32_t)steps)) return RCMARL_ERR_ARG;
    } else {
        for (int p = 0; p < COMM_MAX_WORLD; ++p) P.comm.cells[p] = nullptr;
        P.comm.cells[0] = (uint2*)cells + l1;
        P.comm.error = (uint32_t*)((uint2*)cells + l1 + l2);
        P.comm.max_floats = (int64_t)n_jobs * maxn;
        P.comm.rank = 0; P.comm.world = 1; P.comm.seq = seq_first;
    }
    cudaStream_t st = (cudaStream_t)stream;
#if RCMARL_GRAD_WS
    if (NA == 5) return launch_mb_persist_ws(P, n_ctas, st);
#endif
    return NA == 5 ? launch_mb_persist<5>(P, n_ctas, st) : launch_mb_persist<16>(P, n_ctas, st);
}

#if RCMARL_GRAD_WS && RCMARL_WS_TIMELINE
/* debug builds only (csrc/Makefile variant_tl): stage timestamps of the first producer thread, [64 tiles][16 ticks] */
int rcmarl_debug_timeline(long long* out_host, int n) {
    if (!out_host || n < 1 || n > 64 * 16) return RCMARL_ERR_ARG;
    RC_CUDA(cudaMemcpyFromSymbol(out_host, g_ws_timeline, sizeof(long long) * n));
    return RCMARL_OK;
}
/* same for the persistent mini-batch kernel: [64 steps][16 ticks] of CTA 0 / thread 0 */
int rcmarl_debug_timeline_mb(long long* out_host, int n) {
    if (!out_host || n < 1 || n > 64 * 16) return RCMARL_ERR_ARG;
    RC_CUDA(cudaMemcpyFromSymbol(out_host, g_mb_timeline, sizeof(long long) * n));
    return RCMARL_OK;
}
#endif

int rcmarl_team(const rcmarl_rows* rows, const rcmarl_team_job* jobs, int n_jobs, void* ws, int64_t ws_bytes,
                void* stream) {
    if (int e = check_rows(rows)) return e;
    if (!jobs || n_jobs < 1 || n_jobs > RCMARL_MAX_JOBS) return RCMARL_ERR_ARG;
    const int NA = rows->n_agents;
    TeamParams P;
    ReduceParams Q;
    P.rows = *rows;
    bool any_sums = false;
    for (int j = 0; j < n_jobs; ++j) {
        const rcmarl_team_job& q = jobs[j];
        if (!q.w || q.kind < 0 || q.kind > 2) return RCMARL_ERR_ARG;
        if (!q.agg_in) {
            if (!q.msgs || q.n_in < 1 || q.n_in > RCMARL_MAX_NEIGHBOURS || q.H < 0 || q.H >= q.n_in) return RCMARL_ERR_ARG;
        }
        if (!q.sums && !q.agg_out) return RCMARL_ERR_ARG;
        any_sums |= (q.sums != nullptr);
        P.jobs[j] = q;
        Q.sums[j] = q.sums;
        Q.n[j] = q.sums ? TEAM_N : 0;
    }
    // one launch per input kind (see TeamParams::job_list); each fills the GPU on its own: 128 threads x 2 rows, 3 CTAs / SM
    int gy_of[RCMARL_MAX_JOBS], gy_max = 0;
    int lists[2][RCMARL_MAX_JOBS], n_list[2] = {0, 0};
    for (int j = 0; j < n_jobs; ++j) {
        const int g = jobs[j].kind == RCMARL_IN_SA ? 0 : 1;
        lists[g][n_list[g]++] = j;
    }
    for (int g = 0; g < 2; ++g) {
        if (!n_list[g]) continue;
        const int gy = grid_y_for((rows->n_rows + 255) / 256, n_list[g], 3);
        for (int k = 0; k < n_list[g]; ++k) gy_of[lists[g][k]] = gy;
        gy_max = gy > gy_max ? gy : gy_max;
    }
    if (any_sums) {
        if (!ws || (int64_t)gy_max * n_jobs * TEAM_N * (int64_t)sizeof(float) > ws_bytes) return RCMARL_ERR_WORKSPACE;
    }
    P.partial = (float*)ws;
    P.n_jobs = n_jobs;
    P.stride = TEAM_N;
    cudaStream_t st = (cudaStream_t)stream;
    for (int g = 0; g < 2; ++g) {
        if (!n_list[g]) continue;
        for (int k = 0; k < n_list[g]; ++k) P.job_list[k] = lists[g][k];
        const int gy = gy_of[lists[g][0]];
        const int e = NA == 5 ? launch_team<5>(P, n_list[g], gy, st) : launch_team<16>(P, n_list[g], gy, st);
        if (e) return e;
    }
    if (any_sums) {
        Q.partial = (const float*)ws;
        Q.slots.step = n_jobs;                    // team_kernel writes its partials [y][job] interleaved
        Q.slots.stride = TEAM_N;
        for (int j = 0; j < n_jobs; ++j) { Q.slots.first[j] = j; Q.slots.count[j] = gy_of[j]; }
        if (comm_bound()) {
            ReduceCommParams C;
            if (!comm_next(&C.comm, (int64_t)n_jobs * TEAM_N)) return RCMARL_ERR_ARG;
            C.partial = Q.partial; C.slots = Q.slots; C.out_stride = TEAM_N; C.fuse_sgd = 0; C.n_jobs = n_jobs; C.max_n = TEAM_N;
            for (int j = 0; j < n_jobs; ++j) { C.sums[j] = Q.sums[j]; C.n[j] = Q.n[j]; }
            if (launch_reduce(reduce_comm_kernel, C, reduce_comm_grid(TEAM_N, n_jobs), st)) return RCMARL_ERR_CUDA;
        } else {
            reduce_kernel<<<dim3((TEAM_N + 31) / 32, n_jobs), 256, 0, st>>>(Q);
        }
        RC_CUDA(cudaGetLastError());
    }
    return RCMARL_OK;
}

int rcmarl_consensus_hidden(const rcmarl_consensus_job* jobs, int n_jobs, void* stream) {
    if (!jobs || n_jobs < 1 || n_jobs > RCMARL_MAX_JOBS) return RCMARL_ERR_ARG;
    ConsensusParams P;
    int maxn = 0;
    for (int j = 0; j < n_jobs; ++j) {
        const rcmarl_consensus_job& q = jobs[j];
        if (!q.dst || !q.msgs || q.n_in < 1 || q.n_in > RCMARL_MAX_NEIGHBOURS || q.H < 0 || q.H >= q.n_in || q.n_hidden < 1)
            return RCMARL_ERR_ARG;
        P.jobs[j] = q;
        if (q.n_hidden > maxn) maxn = q.n_hidden;
    }
    consensus_hidden_kernel<<<dim3((maxn + 255) / 256, n_jobs), 256, 0, (cudaStream_t)stream>>>(P);
    RC_CUDA(cudaGetLastError());
    return RCMARL_OK;
}

int rcmarl_sgd_apply(const rcmarl_sgd_job* jobs, int n_jobs, void* stream) {
    if (!jobs || n_jobs < 1 || n_jobs > RCMARL_MAX_JOBS) return RCMARL_ERR_ARG;
    SgdParams P;
    int maxn = 0;
    for (int j = 0; j < n_jobs; ++j) {
        if (!jobs[j].dst || !jobs[j].src || !jobs[j].sums || jobs[j].n < 1) return RCMARL_ERR_ARG;
        P.jobs[j] = jobs[j];
        if (jobs[j].n > maxn) maxn = jobs[j].n;
    }
    sgd_kernel<<<dim3((maxn + 255) / 256, n_jobs), 256, 0, (cudaStream_t)stream>>>(P);
    RC_CUDA(cudaGetLastError());
    return RCMARL_OK;
}

int rcmarl_adam_apply(const rcmarl_adam_job* jobs, int n_jobs, void* stream) {
    if (!jobs || n_jobs < 1 || n_jobs > RCMARL_MAX_JOBS) return RCMARL_ERR_ARG;
    AdamParams P;
    int maxn = 0;
    for (int j = 0; j < n_jobs; ++j) {
        if (!jobs[j].theta || !jobs[j].m || !jobs[j].v || !jobs[j].sums || jobs[j].n < 1) return RCMARL_ERR_ARG;
        P.jobs[j] = jobs[j];
        if (jobs[j].n > maxn) maxn = jobs[j].n;
    }
    adam_kernel<<<dim3((maxn + 255) / 256, n_jobs), 256, 0, (cudaStream_t)stream>>>(P);
    RC_CUDA(cudaGetLastError());
    return RCMARL_OK;
}

int rcmarl_reward_mix(const float* r, int64_t n_rows, int n_agents, const int32_t* agents, int n_listed, float scale,
                      float* out, void* stream) {
    if (!r || !out || !agents || n_rows < 0 || n_listed < 1 || n_listed > RCMARL_MAX_JOBS || n_agents < 1)
        return RCMARL_ERR_ARG;
    if (n_rows == 0) return RCMARL_OK;
    MixParams P;
    for (int k = 0; k < n_listed; ++k) {
        if (agents[k] < 0 || agents[k] >= n_agents) return RCMARL_ERR_ARG;
        P.agents[k] = agents[k];
    }
    reward_mix_kernel<<<(unsigned)((n_rows + 255) / 256), 256, 0, (cudaStream_t)stream>>>(r, n_rows, n_agents, P,
                                                                                         n_listed, scale, out);
    RC_CUDA(cudaGetLastError());
    return RCMARL_OK;
}

}  // extern "C"
