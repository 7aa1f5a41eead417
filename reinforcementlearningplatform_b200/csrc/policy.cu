// policy.cu -- K-POLICY: batched Gaussian actor + critic forward for N instances (sm_100a), SURVEY 8(f)-2.
//
// Replaces, for a whole batch of observations, `Proximal_Policy_Optimization2.choose_action`
// (algorithm/policy_base/Proximal_Policy_Optimization2.py:69-76):
//     dist = actor.get_dist(s)            PPOActor_Gaussian.forward, utils/classes.py:563-579:
//                                         tanh(fc1) -> tanh(fc2) -> tanh(fc3) -> relu(mean_layer); Normal(mean, std)
//     a = dist.sample(); a = max(min(a, a_max), a_min); a_logprob = dist.log_prob(a)
// and the critic forward `PPOCritic.forward` (utils/classes.py:610-614: tanh(fc1) -> tanh(fc2) -> fc3) that the
// learner evaluates on s and s' (Proximal_Policy_Optimization2.py:88-90).  Observations come in and actions go out in
// the engine's field-major float32 layout ([dim][N]), i.e. exactly the buffers the step kernels read and write
// (b200env_io with io_dtype = F32): policy_state -> K-POLICY -> action -> step kernel, no host round trip.
//
// Arithmetic: float32 like the reference (torch CPU float32); FMA accumulation in k order, so results differ from
// torch's blocked GEMM only by summation order (tests: <= 2e-6 absolute on mean / value).  tanhf, logf are the
// accurate libdevice versions.  Sampling: a = mean + std * eps with eps either injected ([A][N], parity tests) or
// drawn in-kernel from Philox4x32-10 keyed by (seed, global instance index, step) through Box-Muller, independent of
// launch geometry and sharding.
//
// Mapping: one thread per instance, persistent blocks of 256 threads, 2 blocks per SM.  Every layer's W^T (zero-padded
// to 16 / 32 / 64 outputs) and bias live in shared memory for the whole kernel; the activations of the 256 instances of
// a tile live in ONE [64][256] shared buffer (column = thread, conflict-free) that each layer overwrites in place: a
// thread keeps all (<= 64) outputs of the layer in registers while it walks k, then stores them over its own column.
// Per k: one activation load, CH/4 broadcast LDS.128 of weights, CH independent FFMAs -- bound by the FP32 FMA pipe
// (CUDA cores).  The nets of the reference (6..41 -> 64 -> 64 -> 32 -> A, critic 64 -> 32 -> 1) are far too small for
// a tensor-core tile pipeline to pay unless this kernel dominates a training step; bench.py reports its time next to
// the env step so that decision is made on a measurement.
#include "policy_common.cuh"

namespace {

constexpr int PB = 256;          // threads (= instances) per tile
constexpr int MAX_OUT = 64;      // widest layer (padded) this kernel keeps in registers
constexpr int MAX_LAYERS = 4;

struct NetDev {
    int n_layers;
    int dims[MAX_LAYERS + 1];    // dims[0] = input, dims[l + 1] = outputs of layer l
    int pad[MAX_LAYERS];         // outputs padded to a multiple of 16
    int w_off[MAX_LAYERS];       // float offsets into the shared weight arena: W^T [in][pad]
    int b_off[MAX_LAYERS];
    int out_act;                 // 0 = identity, 1 = relu
    const float *w[MAX_LAYERS];  // global: nn.Linear.weight [out][in] row-major
    const float *b[MAX_LAYERS];  // global: [out]
};

struct PolicyArgs {
    NetDev actor, critic;
    int has_actor, has_critic;
    int act_dim_max;             // rows of one activation buffer
    int arena_floats;
    PolicyIO io;
};

__device__ __forceinline__ void stage_net(const NetDev &nd, float *arena) {
    for (int l = 0; l < nd.n_layers; ++l) {
        const int in = nd.dims[l], out = nd.dims[l + 1], pd = nd.pad[l];
        float *wt = arena + nd.w_off[l], *bs = arena + nd.b_off[l];
        for (int e = threadIdx.x; e < in * pd; e += PB) {
            const int k = e / pd, j = e - k * pd;
            wt[e] = j < out ? __ldg(nd.w[l] + (int64_t)j * in + k) : 0.0f;
        }
        for (int j = threadIdx.x; j < pd; j += PB) bs[j] = j < out ? __ldg(nd.b[l] + j) : 0.0f;
    }
}

// one dense layer for this thread's instance, in place: buf[j] <- act(b[j] + sum_k W[j][k] buf[k]); all CH (= padded
// width) outputs stay in registers until the last input has been read
template <int CH>
__device__ __forceinline__ void dense(const float *__restrict__ wt, const float *__restrict__ bs, int in,
                                      float *__restrict__ buf, int act) {
    const int t = threadIdx.x;
    float acc[CH];
#pragma unroll
    for (int c = 0; c < CH; ++c) acc[c] = bs[c];
#pragma unroll 4
    for (int k = 0; k < in; ++k) {
        const float x = buf[k * PB + t];
        const float4 *w4 = reinterpret_cast<const float4 *>(wt + k * CH);
#pragma unroll
        for (int c = 0; c < CH / 4; ++c) {
            const float4 w = w4[c];
            acc[4 * c + 0] = fmaf(w.x, x, acc[4 * c + 0]);
            acc[4 * c + 1] = fmaf(w.y, x, acc[4 * c + 1]);
            acc[4 * c + 2] = fmaf(w.z, x, acc[4 * c + 2]);
            acc[4 * c + 3] = fmaf(w.w, x, acc[4 * c + 3]);
        }
    }
#pragma unroll
    for (int c = 0; c < CH; ++c) {
        float v = acc[c];
        if (act == 2) v = tanhf(v);
        else if (act == 1) v = policy_fmax_nan(v, 0.0f);
        buf[c * PB + t] = v;
    }
}

__device__ __forceinline__ void run_net(const NetDev &nd, const float *arena, float *buf) {
    for (int l = 0; l < nd.n_layers; ++l) {
        const int act = l + 1 < nd.n_layers ? 2 : nd.out_act;
        const float *wt = arena + nd.w_off[l], *bs = arena + nd.b_off[l];
        if (nd.pad[l] == 64) dense<64>(wt, bs, nd.dims[l], buf, act);
        else if (nd.pad[l] == 32) dense<32>(wt, bs, nd.dims[l], buf, act);
        else dense<16>(wt, bs, nd.dims[l], buf, act);
    }
}

__global__ void __launch_bounds__(PB, 2)
policy_forward_kernel(const __grid_constant__ PolicyArgs a, int64_t n) {
    extern __shared__ __align__(16) float smem[];
    float *arena = smem;
    float *buf = smem + a.arena_floats;                      // activations [act_dim_max][PB], overwritten in place
    if (a.has_actor) stage_net(a.actor, arena);
    if (a.has_critic) stage_net(a.critic, arena);
    __syncthreads();
    const int S = a.has_actor ? a.actor.dims[0] : a.critic.dims[0];
    const int t = threadIdx.x;
    const int64_t tiles = (n + PB - 1) / PB;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const int64_t i = tile * PB + t;
        const bool live = i < n;
        // (each thread only ever touches its own column t of buf: no block synchronisation needed)
        for (int k = 0; k < S; ++k) buf[k * PB + t] = live ? __ldg(a.io.obs + (int64_t)k * n + i) : 0.0f;
        if (a.has_actor) {
            const int A = a.actor.dims[a.actor.n_layers];
            run_net(a.actor, arena, buf);
            if (live) policy_sample_store(a.io, n, i, A, buf + t, PB);
        }
        if (a.has_critic) {
            if (a.has_actor) // the observations again (24..164 B per instance, an L2 hit)
                for (int k = 0; k < S; ++k) buf[k * PB + t] = live ? __ldg(a.io.obs + (int64_t)k * n + i) : 0.0f;
            run_net(a.critic, arena, buf);
            if (live) __stcs(a.io.value + i, buf[t]);
        }
    }
}

int fill_net(const b200_mlp *m, NetDev *nd, int *arena, int *act_rows) {
    if (m->n_layers < 1 || m->n_layers > MAX_LAYERS) return B200ENV_ESIZE;
    nd->n_layers = m->n_layers;
    nd->out_act = m->out_act == 2 ? 0 : m->out_act; // 2 (tanh range map) is applied by policy_sample_store
    for (int l = 0; l <= m->n_layers; ++l) {
        if (m->dims[l] < 1 || m->dims[l] > 1024) return B200ENV_ESIZE;
        nd->dims[l] = m->dims[l];
    }
    for (int l = 0; l < m->n_layers; ++l) {
        if (!m->w[l] || !m->b[l]) return B200ENV_ENULL;
        nd->w[l] = m->w[l];
        nd->b[l] = m->b[l];
        const int o = m->dims[l + 1];
        if (o > MAX_OUT) return B200ENV_ESIZE; // wider layers: not supported by this kernel (no fallback)
        nd->pad[l] = o <= 16 ? 16 : (o <= 32 ? 32 : 64);
        nd->w_off[l] = *arena;
        *arena += nd->dims[l] * nd->pad[l];
        nd->b_off[l] = *arena;
        *arena += nd->pad[l];
        if (nd->pad[l] > *act_rows) *act_rows = nd->pad[l];
    }
    return B200ENV_OK;
}

} // namespace

int policy_launch_fp32(int64_t n, const b200_mlp *actor, const b200_mlp *critic, const PolicyIO &io, cudaStream_t stream) {
    PolicyArgs a = {};
    int arena = 0, rows = 16, rc;
    const int in_dim = actor ? actor->dims[0] : critic->dims[0];
    if (in_dim > rows) rows = in_dim;
    if (actor) {
        if ((rc = fill_net(actor, &a.actor, &arena, &rows))) return rc;
        a.has_actor = 1;
    }
    if (critic) {
        if ((rc = fill_net(critic, &a.critic, &arena, &rows))) return rc;
        a.has_critic = 1;
    }
    a.arena_floats = (arena + 3) / 4 * 4;
    a.act_dim_max = rows;
    a.io = io;
    const size_t smem = ((size_t)a.arena_floats + (size_t)rows * PB) * sizeof(float);
    if (smem > 227 * 1024) return B200ENV_ESIZE; // nets wider than shared memory holds: not supported by this kernel
    static size_t configured[64] = {0}; // per device: the opt-in dynamic shared-memory limit set so far
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) dev = 0;
    if (smem > 48 * 1024 && smem > configured[dev]) {
        if (cudaFuncSetAttribute(policy_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return b200_check_launch();
        configured[dev] = smem;
    }
    int per_sm = (int)((227 * 1024) / (smem + 1024));
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 8) per_sm = 8;
    const unsigned grid = b200_persistent_grid(n, per_sm, PB);
    policy_forward_kernel<<<grid, PB, smem, stream>>>(a, n);
    return b200_check_launch();
}

namespace {
int policy_check(int64_t n, const b200_mlp *actor, const b200_mlp *critic, const float *obs, const float *a_min,
                 const float *a_max, float std_, const float *std_vec, const float *action, const float *value) {
    if (n <= 0) return B200ENV_ESIZE;
    if (!obs || (!actor && !critic)) return B200ENV_ENULL;
    if (actor && (!action || !a_min || !a_max)) return B200ENV_ENULL;
    if (critic && !value) return B200ENV_ENULL;
    if (actor && !std_vec && !(std_ > 0.0f)) return B200ENV_EPARAMS;
    if (actor && (actor->out_act < 0 || actor->out_act > 2)) return B200ENV_EPARAMS;
    if (critic && critic->dims[critic->n_layers > 0 && critic->n_layers <= 4 ? critic->n_layers : 0] != 1) return B200ENV_EPARAMS;
    if (actor && critic && actor->dims[0] != critic->dims[0]) return B200ENV_EPARAMS;
    return B200ENV_OK;
}
} // namespace

extern "C" B200_API int b200_policy_forward(int64_t n, const b200_mlp *actor, const b200_mlp *critic, const float *obs,
                                            const float *a_min, const float *a_max, float std_, const float *noise,
                                            uint64_t seed, uint64_t step, int64_t env_index_offset, int precision,
                                            float *action, float *log_prob, float *mean, float *value,
                                            void *cuda_stream) {
    const int rc = policy_check(n, actor, critic, obs, a_min, a_max, std_, nullptr, action, value);
    if (rc) return rc;
    PolicyIO io = {};
    io.obs = obs; io.a_min = a_min; io.a_max = a_max; io.noise = noise; io.std_ = std_;
    io.out_affine = actor && actor->out_act == 2;
    io.seed = seed; io.step = step; io.off = env_index_offset;
    io.action = action; io.log_prob = log_prob; io.mean = mean; io.value = value;
    if (precision == B200_POLICY_FP32) return policy_launch_fp32(n, actor, critic, io, (cudaStream_t)cuda_stream);
    return B200ENV_EPARAMS;
}

extern "C" B200_API size_t b200_policy_workspace_bytes(const b200_mlp *actor, const b200_mlp *critic) {
    if (!actor && !critic) return 0;
    return policy_umma_workspace_bytes(actor, critic);
}

extern "C" B200_API int b200_policy_pack(const b200_mlp *actor, const b200_mlp *critic, void *workspace,
                                         size_t workspace_bytes, void *cuda_stream) {
    if (!actor && !critic) return B200ENV_ENULL;
    return policy_umma_pack(actor, critic, workspace, workspace_bytes, (cudaStream_t)cuda_stream);
}

extern "C" B200_API int b200_policy_forward_packed(int64_t n, const b200_mlp *actor, const b200_mlp *critic,
                                                   const void *workspace, size_t workspace_bytes, const float *obs,
                                                   const float *a_min, const float *a_max, float std_,
                                                   const float *std_vec, const float *noise, uint64_t seed, uint64_t step,
                                                   int64_t env_index_offset, float *action, float *log_prob, float *mean,
                                                   float *value, void *cuda_stream) {
    const int rc = policy_check(n, actor, critic, obs, a_min, a_max, std_, std_vec, action, value);
    if (rc) return rc;
    PolicyIO io = {};
    io.obs = obs; io.a_min = a_min; io.a_max = a_max; io.noise = noise; io.std_ = std_vec ? 1.0f : std_;
    io.std_vec = std_vec;
    io.out_affine = actor && actor->out_act == 2;
    io.seed = seed; io.step = step; io.off = env_index_offset;
    io.action = action; io.log_prob = log_prob; io.mean = mean; io.value = value;
    return policy_launch_umma(n, actor, critic, workspace, workspace_bytes, io, (cudaStream_t)cuda_stream);
}

extern "C" B200_API int b200_umma_probe(const float *A, const float *W, float *D, int N, int K, int three_pass,
                                        void *cuda_stream) {
    if (!A || !W || !D) return B200ENV_ENULL;
    return policy_umma_probe(A, W, D, N, K, three_pass, (cudaStream_t)cuda_stream);
}
