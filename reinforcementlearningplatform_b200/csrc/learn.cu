// learn.cu -- K-LEARN: the PPO2 / DPPO2 network update on device (SURVEY 8(f)-3).
//
// Replaces the body of the mini-batch loop of Proximal_Policy_Optimization2.learn (algorithm/policy_base/
// Proximal_Policy_Optimization2.py:102-131) -- actor forward, Normal.log_prob, ratio, clipped surrogate, backward,
// clip_grad_norm_, Adam; critic forward, mse_loss, backward, clip, Adam -- which round 1 left to torch autograd (about
// forty library kernels per mini-batch, 0.24 s per learn() of 4096 x 64 samples against 8 ms for collecting them).
//
// ppo2_grad_kernel: one block works on 64-sample tiles of the mini-batch, two blocks per SM; the SMs' blocks are dealt to
// the two nets (actor / critic) in proportion to their measured cost per tile, so both nets' gradients come out of ONE
// launch.  Everything of a tile stays in shared memory:
//     H_l [64][K_l + 4]    input of layer l (H_0 = the gathered observations, H_l = tanh outputs), sample-major;
//     W_l [N_l][K_l + 4]   the layer's weights as nn.Linear stores them (zero-padded), loaded once per block;
// and the three products of a layer are register-tiled fp32 GEMMs whose operands are both read along their contiguous
// index with 16-byte loads (row pitch = width + 4 floats, so that the rows a warp touches fall into distinct banks):
//     forward   Z[s][n]  = sum_k H_l[s][k] W_l[n][k]          thread: 2 samples x (N/8) outputs
//     dW        dW[n][k] = sum_s dZ_l[s][n] H_l[s][k]         thread: RN x RK entries (4 x 4 for 64 x 64 .. 1 x 1 for 8 x 32:
//                                                             all 256 threads share every layer), added to the block's
//                                                             partial gradient (L2) once per tile by the thread that owns them
//     dH        dH[s][k] = sum_n dZ_l[s][n] W_l[n][k]         thread: 2 samples x (K/32) 4-vectors
// dZ_{l-1} = dH * (1 - H_l^2) overwrites H_l in place (its last reader was dW_l), so no separate gradient buffers exist.
// A block adds up its tiles in program order; ppo2_reduce_kernel (a second, wide launch: one thread per parameter) sums
// the per-block partials in block order: the result does not depend on scheduling (no floating-point atomics anywhere).
// History (profiles/r2/learn.md): 128-sample tiles with the weight gradients in 80 persistent registers and one block per
// SM measured the same at large batches and 25 % slower at 4096 samples (half as many tiles to spread over the SMs).
//
// adam_kernel: clip_grad_norm_ + Adam.step over flat parameter / gradient / moment buffers (one segment per net), the
// global norm recomputed in a fixed order by every block so that no grid-wide synchronisation is needed.
//
// Arithmetic is fp32 on the FMA pipe with CUDA's accurate tanhf / expf (the test compares gradients and the updated
// parameters with torch autograd: <= 1e-6).  Tensor cores are not used here on purpose: a 3xTF32 split would need the
// activations in two operand layouts per layer (K-major for forward / dH, sample-major for dW) and the mini-batches of
// the reference's configurations (4096 .. 16384 samples of a 6-64-64-32-8 net = 0.2 .. 0.9 GFLOP) are launch-latency
// bound either way.
#include "common.cuh"

namespace {

constexpr int LT = 256;     // threads per block
constexpr int TM = 64;      // samples per tile
constexpr int TM_LOG2 = 6;
constexpr int MI = TM / 32; // samples per thread in the sample-by-feature products
constexpr int BLOCKS_PER_SM = 2;
constexpr int LMAX = 4;     // layers per net
constexpr int WMAX = 64;    // widest layer / input
constexpr int GRID_CAP = 148 * BLOCKS_PER_SM;

struct LLayer {
    int K, N;            // padded: K to a multiple of 8, N to 8 / 16 / 32 / 64
    int k_real, n_real;
    int w_off, b_off;    // shared-memory float offsets: weights [N][K + 4], bias [N]
    int h_off;           // shared-memory float offset of the layer's input H_l [TM][K + 4]
    int g_w, g_b;        // offsets of weight / bias inside the net's flat gradient
    int rn, rk;          // register tile of the weight-gradient product (dw_layer)
    const float *w, *b;  // global parameters
};

struct LNet {
    int n_layers, P, out_act;
    int gout_off;        // dZ of the output layer [TM][N_out + 4]
    int smem_floats;
    LLayer L[LMAX];
};

// ------------------------------------------------------------------------------------------------ sample permutation
__host__ __device__ __forceinline__ uint32_t feistel_round(uint32_t r, uint32_t k) {
    uint32_t h = (r + k) * 0x9E3779B1u;
    h ^= h >> 15; h *= 0x85EBCA77u;
    h ^= h >> 13; h *= 0xC2B2AE3Du;
    h ^= h >> 16;
    return h;
}
// bijection of [0, 2^(2 * half_bits)) restricted to [0, B) by cycle walking (B > 2^(2 * half_bits - 2): < 4 walks expected)
__host__ __device__ __forceinline__ int64_t perm_index(uint64_t key, int64_t j, int64_t B, int half_bits) {
    const uint32_t mask = (1u << half_bits) - 1u;
    const uint32_t k0 = (uint32_t)key, k1 = (uint32_t)(key >> 32);
    uint64_t x = (uint64_t)j;
    do {
        uint32_t l = (uint32_t)(x >> half_bits) & mask, r = (uint32_t)x & mask;
#pragma unroll
        for (int q = 0; q < 6; ++q) {
            const uint32_t f = feistel_round(r, (q & 1 ? k1 : k0) + 0x632BE5ABu * (uint32_t)q) & mask;
            const uint32_t t = l ^ f;
            l = r;
            r = t;
        }
        x = ((uint64_t)l << half_bits) | r;
    } while ((int64_t)x >= B);
    return (int64_t)x;
}
int half_bits_for(int64_t B) {
    int bits = 1;
    while (((int64_t)1 << bits) < B) ++bits;
    return (bits + 1) / 2 < 1 ? 1 : (bits + 1) / 2;
}

// sample j of a PPO mini-batch: batch position index[first + j] if the caller gave an index, else the keyed permutation
// of [0, T N) at first + j
struct PpoSampler {
    int64_t T, N, first;
    const int64_t *index;
    uint64_t perm_key;
    int half_bits;
    __device__ __forceinline__ int64_t pos(int64_t j) const {
        return index ? index[first + j] : perm_index(perm_key, first + j, T * N, half_bits);
    }
};

struct LearnArgs {
    LNet net[2];                 // 0 actor, 1 critic
    int net_of_y[2];             // slot -> net: blocks 0 .. nblk[0] - 1 work on slot 0, the next nblk[1] on slot 1
    int nblk[2];
    int S, A;
    PpoSampler sp;
    int64_t count;
    const float *s, *a, *a_lp, *adv, *v_target;
    float eps_clip, inv_count, entropy_coef;
    float std_;
    const float *std_vec, *a_min, *a_max;
    float *partial[2];           // [gridDim.x][P + 4]
    float *grad[2];
    float *loss_out;             // [2]
};

// ------------------------------------------------------------------------------------------------ tile GEMMs
// thread coordinates of the sample-by-feature products: sg = 0..31 -> samples sg + 32 i, ng = 0..7 -> features ng + 8 j
template <int NJ>
__device__ __forceinline__ void fwd_layer(const float *__restrict__ H, int ph, const float *__restrict__ W, int pw,
                                          const float *__restrict__ bias, int K, float *__restrict__ out, int po,
                                          bool hidden, int sg, int ng) {
    float acc[MI][NJ];
#pragma unroll
    for (int i = 0; i < MI; ++i)
#pragma unroll
        for (int j = 0; j < NJ; ++j) acc[i][j] = 0.0f;
    // one base pointer per operand row, hoisted: inside the (unrolled) k loop every load is base + immediate -- the
    // address arithmetic was 9 % of the kernel's instructions (LEA per LDS, profiles/r2/learn.md)
    const float *ha[MI], *wa[NJ];
#pragma unroll
    for (int i = 0; i < MI; ++i) ha[i] = H + (sg + 32 * i) * ph;
#pragma unroll
    for (int j = 0; j < NJ; ++j) wa[j] = W + (ng + 8 * j) * pw;
#pragma unroll 4
    for (int k0 = 0; k0 < K; k0 += 4) {
        float4 a[MI];
#pragma unroll
        for (int i = 0; i < MI; ++i) a[i] = *reinterpret_cast<const float4 *>(ha[i] + k0);
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const float4 w = *reinterpret_cast<const float4 *>(wa[j] + k0);
#pragma unroll
            for (int i = 0; i < MI; ++i) {
                acc[i][j] = fmaf(a[i].x, w.x, acc[i][j]);
                acc[i][j] = fmaf(a[i].y, w.y, acc[i][j]);
                acc[i][j] = fmaf(a[i].z, w.z, acc[i][j]);
                acc[i][j] = fmaf(a[i].w, w.w, acc[i][j]);
            }
        }
    }
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
        const float b = bias[ng + 8 * j];
#pragma unroll
        for (int i = 0; i < MI; ++i) {
            const float z = acc[i][j] + b;
            out[(sg + 32 * i) * po + ng + 8 * j] = hidden ? tanhf(z) : z;
        }
    }
}

// dH[s][k] = sum_n G[s][n] W[n][k], then dZ = dH * (1 - H^2) written over H.  k-vectors of 4: v = ng + 8 jv
template <int NV>
__device__ __forceinline__ void bwd_layer(const float *__restrict__ G, int pg, const float *__restrict__ W, int pw, int N,
                                          float *H, int ph, int KG, int sg, int ng) {
    if (ng >= KG) return;
    float4 acc[MI][NV];
#pragma unroll
    for (int i = 0; i < MI; ++i)
#pragma unroll
        for (int jv = 0; jv < NV; ++jv) acc[i][jv] = make_float4(0.f, 0.f, 0.f, 0.f);
    const float *wp = W + 4 * ng;
    const float *ga[MI];
#pragma unroll
    for (int i = 0; i < MI; ++i) ga[i] = G + (sg + 32 * i) * pg;
#pragma unroll 2
    for (int n0 = 0; n0 < N; n0 += 4) {
        float g[MI][4];
#pragma unroll
        for (int i = 0; i < MI; ++i) {
            const float4 t = *reinterpret_cast<const float4 *>(ga[i] + n0);
            g[i][0] = t.x; g[i][1] = t.y; g[i][2] = t.z; g[i][3] = t.w;
        }
#pragma unroll
        for (int q = 0; q < 4; ++q)
#pragma unroll
            for (int jv = 0; jv < NV; ++jv) {
                const float4 w = *reinterpret_cast<const float4 *>(wp + (n0 + q) * pw + 32 * jv);
#pragma unroll
                for (int i = 0; i < MI; ++i) {
                    acc[i][jv].x = fmaf(g[i][q], w.x, acc[i][jv].x);
                    acc[i][jv].y = fmaf(g[i][q], w.y, acc[i][jv].y);
                    acc[i][jv].z = fmaf(g[i][q], w.z, acc[i][jv].z);
                    acc[i][jv].w = fmaf(g[i][q], w.w, acc[i][jv].w);
                }
            }
    }
#pragma unroll
    for (int i = 0; i < MI; ++i)
#pragma unroll
        for (int jv = 0; jv < NV; ++jv) {
            float4 *hp = reinterpret_cast<float4 *>(H + (sg + 32 * i) * ph + 4 * ng + 32 * jv);
            const float4 h = *hp;
            float4 d;
            d.x = acc[i][jv].x * (1.0f - h.x * h.x);
            d.y = acc[i][jv].y * (1.0f - h.y * h.y);
            d.z = acc[i][jv].z * (1.0f - h.z * h.z);
            d.w = acc[i][jv].w * (1.0f - h.w * h.w);
            *hp = d;
        }
}

// dW[RN ng .. ][RK kg .. ] += sum over the tile's samples of dZ[s][n] H[s][k]; db likewise for the kg == 0 threads.
// The RN x RK register tile is chosen per layer (host: fill_net) so that ALL 256 threads share a layer's N x K entries:
// 4 x 4 for 64 x 64, 2 x 4 for 32 x 64, 1 x 2 for 64 x 8, 1 x 1 for 8 x 32 -- with a fixed 4 x 4 tile the small layers
// kept one or two warps busy for 128 iterations while the other warps waited at the barrier (ncu: stall_barrier 1.36 per
// issued instruction, the largest stall of the first version).
template <int RN, int RK>
__device__ __forceinline__ void dw_layer(const float *__restrict__ G, int pg, const float *__restrict__ H, int ph, int ng,
                                         int kg, float (&dw)[16], float (&db)[4]) {
    const float *gp = G + RN * ng, *hp = H + RK * kg;
#pragma unroll 4
    for (int s = 0; s < TM; ++s) {
        float g[RN], h[RK];
        if (RN == 4) { const float4 t = *reinterpret_cast<const float4 *>(gp + s * pg); g[0] = t.x; g[1 % RN] = t.y; g[2 % RN] = t.z; g[3 % RN] = t.w; }
        else if (RN == 2) { const float2 t = *reinterpret_cast<const float2 *>(gp + s * pg); g[0] = t.x; g[1 % RN] = t.y; }
        else g[0] = gp[s * pg];
        if (RK == 4) { const float4 t = *reinterpret_cast<const float4 *>(hp + s * ph); h[0] = t.x; h[1 % RK] = t.y; h[2 % RK] = t.z; h[3 % RK] = t.w; }
        else if (RK == 2) { const float2 t = *reinterpret_cast<const float2 *>(hp + s * ph); h[0] = t.x; h[1 % RK] = t.y; }
        else h[0] = hp[s * ph];
#pragma unroll
        for (int a = 0; a < RN; ++a)
#pragma unroll
            for (int c = 0; c < RK; ++c) dw[a * RK + c] = fmaf(g[a], h[c], dw[a * RK + c]);
        if (kg == 0) {
#pragma unroll
            for (int a = 0; a < RN; ++a) db[a] += g[a];
        }
    }
}

// the thread's RN x RK entries of dW (and RN of db) -> this block's partial gradient, torch parameter layout
// `first`: this is the block's first tile (the partial buffer is not cleared between launches); later tiles add to what
// the SAME thread stored before, in tile order -- no atomics, bit-reproducible.  The accumulators live in the block's
// partial (L2) instead of registers since the tile shrank to 64 samples for two blocks per SM: 80 persistent registers
// per thread did not fit under the 128 of a 2 x 256-thread SM.
template <int RN, int RK>
__device__ __forceinline__ void dw_store(const LLayer &Ly, float *part, int ng, int kg, const float (&dw)[16],
                                         const float (&db)[4], bool first) {
    float old[RN * RK], oldb[RN];
#pragma unroll
    for (int a = 0; a < RN; ++a) {
        const int n = RN * ng + a;
#pragma unroll
        for (int c = 0; c < RK; ++c)
            old[a * RK + c] = (!first && n < Ly.n_real && RK * kg + c < Ly.k_real) ? __ldcg(part + Ly.g_w + n * Ly.k_real + RK * kg + c) : 0.0f;
        oldb[a] = (!first && kg == 0 && n < Ly.n_real) ? __ldcg(part + Ly.g_b + n) : 0.0f;
    }
#pragma unroll
    for (int a = 0; a < RN; ++a) {
        const int n = RN * ng + a;
        if (n < Ly.n_real) {
#pragma unroll
            for (int c = 0; c < RK; ++c)
                if (RK * kg + c < Ly.k_real) __stcg(part + Ly.g_w + n * Ly.k_real + RK * kg + c, old[a * RK + c] + dw[a * RK + c]);
            if (kg == 0) __stcg(part + Ly.g_b + n, oldb[a] + db[a]);
        }
    }
}

// -DLEARN_TRACE (tools/build_variant.sh): thread 0 of block 0 adds up the cycles between the phase barriers of its tiles
// (phase ids: 0 sample indices, 1 gather, 2 + l forward layer l, 6 loss, 7 + 2 l dW_l, 8 + 2 l dH_l + dZ write) ->
// b200_learn_trace_read.  How profiles/r2/learn.md's phase table was measured.  Compiled out of the shipped library.
// The timestamp lives in shared memory so that the tile helpers below can mark their phases too; every kernel that
// runs them starts it with LTRACE_START, and their block 0 adds to the same table (tools/learn_trace.py runs PPO2 alone).
#ifdef LEARN_TRACE
__device__ long long g_learn_trace[16];
__shared__ long long s_lt_prev;
#define LTRACE_START()                                                      \
    do {                                                                    \
        if (blockIdx.x == 0 && threadIdx.x == 0) s_lt_prev = clock64();     \
    } while (0)
#define LTRACE(id)                                                          \
    do {                                                                    \
        if (blockIdx.x == 0 && threadIdx.x == 0) {                          \
            const long long now = clock64();                                \
            g_learn_trace[id] += now - s_lt_prev;                           \
            s_lt_prev = now;                                                \
        }                                                                   \
    } while (0)
#else
#define LTRACE_START() do { } while (0)
#define LTRACE(id) do { } while (0)
#endif

// ------------------------------------------------------------------------------------------------ tile phases
// The phases every tile kernel shares.  One copy each: ppo1_advantage_kernel's V is bit-identical to the critic blocks'
// of ppo2_grad_kernel, and dqn_grad_kernel's backward is ppo2_grad_kernel's, because they run the same code.

// weights and biases of `net` -> w (shared memory, the offsets of fill_net), zero-padded
__device__ __forceinline__ void load_weights(const LNet &net, float *w, int tid) {
    for (int l = 0; l < net.n_layers; ++l) {
        const LLayer &Ly = net.L[l];
        const int pw = Ly.K + 4;
        for (int e = tid; e < Ly.N * pw; e += LT) {
            const int n = e / pw, k = e - n * pw;
            w[Ly.w_off + e] = (n < Ly.n_real && k < Ly.k_real) ? __ldg(Ly.w + n * Ly.k_real + k) : 0.0f;
        }
        for (int n = tid; n < Ly.N; n += LT) w[Ly.b_off + n] = n < Ly.n_real ? __ldg(Ly.b + n) : 0.0f;
    }
}

// layer Ly of the forward: out [TM][po] = act(H [TM][ph] W^T + b), with W and b at Ly's offsets in w
__device__ __forceinline__ void fwd_any(const LLayer &Ly, const float *w, const float *H, int ph, float *out, int po,
                                        bool hidden, int sg, int ng) {
    const float *W = w + Ly.w_off, *bs = w + Ly.b_off;
    const int pw = Ly.K + 4;
    switch (Ly.N >> 3) {
    case 1: fwd_layer<1>(H, ph, W, pw, bs, Ly.K, out, po, hidden, sg, ng); break;
    case 2: fwd_layer<2>(H, ph, W, pw, bs, Ly.K, out, po, hidden, sg, ng); break;
    case 4: fwd_layer<4>(H, ph, W, pw, bs, Ly.K, out, po, hidden, sg, ng); break;
    default: fwd_layer<8>(H, ph, W, pw, bs, Ly.K, out, po, hidden, sg, ng); break;
    }
}

// sample j = tile TM + tid of the mini-batch -> (t, i) in s_t / s_i (t = -1 past `count`); returns its position
// t N + i in the batch (-1 for none)
template <typename Sampler>
__device__ __forceinline__ int64_t tile_samples(const Sampler &sp, int64_t tile, int64_t count, int *s_t, int *s_i,
                                                int tid) {
    int64_t b = -1;
    if (tid < TM) {
        const int64_t j = tile * TM + tid;
        int t = -1, i = 0;
        if (j < count) {
            b = sp.pos(j);
            t = (int)(b / sp.N);
            i = (int)(b - (int64_t)t * sp.N);
        }
        s_t[tid] = t;
        s_i[tid] = i;
    }
    return b;
}

// X [TM][px] = the tile's observations s [T][S][N], zero-padded to K0 fields and for samples t < 0
// (thread = sample s, fields q, q + 4, ...)
__device__ __forceinline__ void gather_obs(const float *s, int S, int64_t N, int K0, const int *s_t, const int *s_i,
                                           float *X, int px, int tid) {
    const int sx = tid & (TM - 1), q = tid >> TM_LOG2;
    const int t = s_t[sx];
    const int64_t i = s_i[sx], tt = t < 0 ? 0 : t;
    for (int k = q; k < K0; k += LT / TM)
        X[sx * px + k] = (t >= 0 && k < S) ? __ldg(s + (tt * S + k) * N + i) : 0.0f;
}

// tile_forward / tile_backward take L = net.n_layers and gout = sm + net.gout_off from the kernel, which reads them once
// before its tile loop.  Read from `net` inside the helpers instead, they made ptxas rebuild the shared-memory base
// (S2UR + ULEA) at every layer: 2.2 % more instructions in ppo1_advantage_kernel and dqn_grad_kernel.

// forward of the tile in H_0 through the net's H_l buffers (fill_net's layout); the output layer's Z goes to gout.
// Ends with a barrier.
__device__ __forceinline__ void tile_forward(const LNet &net, int L, float *sm, float *gout, int sg, int ng) {
#pragma unroll
    for (int l = 0; l < LMAX; ++l) {
        if (l < L) {
            const LLayer &Ly = net.L[l];
            const bool last = l == L - 1;
            float *out = last ? gout : sm + net.L[l + 1 < LMAX ? l + 1 : l].h_off;
            fwd_any(Ly, sm, sm + Ly.h_off, Ly.K + 4, out, Ly.N + 4, !last, sg, ng);
            __syncthreads();
            LTRACE(2 + l);
        }
    }
}

// backward of the tile from dZ of the output layer (in gout): per layer, dW / db added to the block's partial gradient
// `part` (`first`: the block's first tile, see dw_store), then dZ_{l-1} written over H_l.  No barrier after the last dW.
__device__ __forceinline__ void tile_backward(const LNet &net, int L, float *sm, const float *gout, float *part, bool first,
                                              int tid, int sg, int ng) {
#pragma unroll
    for (int l = LMAX - 1; l >= 0; --l) {
        if (l < L) {
            const LLayer &Ly = net.L[l];
            const float *G = (l == L - 1) ? gout : sm + net.L[l + 1 < LMAX ? l + 1 : l].h_off;
            float *H = sm + Ly.h_off;
            const int pg = Ly.N + 4, ph = Ly.K + 4;
            const int kgs = Ly.K >> 2;
            {
                const int kt = Ly.K / Ly.rk, nt = Ly.N / Ly.rn;
                if (tid < nt * kt) {
                    // tn runs fastest: the threads that also sum the bias gradient (tk == 0) are the first nt of the
                    // block, so the other warps skip those adds (they were 5 % of all issued instructions)
                    const int tk = tid / nt, tn = tid - tk * nt;
                    float dw[16], db[4];
#pragma unroll
                    for (int e = 0; e < 16; ++e) dw[e] = 0.0f;
#pragma unroll
                    for (int e = 0; e < 4; ++e) db[e] = 0.0f;
                    switch (Ly.rn * 8 + Ly.rk) {
                    case 4 * 8 + 4: dw_layer<4, 4>(G, pg, H, ph, tn, tk, dw, db); dw_store<4, 4>(Ly, part, tn, tk, dw, db, first); break;
                    case 2 * 8 + 4: dw_layer<2, 4>(G, pg, H, ph, tn, tk, dw, db); dw_store<2, 4>(Ly, part, tn, tk, dw, db, first); break;
                    case 1 * 8 + 4: dw_layer<1, 4>(G, pg, H, ph, tn, tk, dw, db); dw_store<1, 4>(Ly, part, tn, tk, dw, db, first); break;
                    case 1 * 8 + 2: dw_layer<1, 2>(G, pg, H, ph, tn, tk, dw, db); dw_store<1, 2>(Ly, part, tn, tk, dw, db, first); break;
                    default: dw_layer<1, 1>(G, pg, H, ph, tn, tk, dw, db); dw_store<1, 1>(Ly, part, tn, tk, dw, db, first); break;
                    }
                }
            }
            if (l > 0) {
                __syncthreads();
                LTRACE(7 + 2 * l);
                if (kgs == 16) bwd_layer<2>(G, pg, sm + Ly.w_off, ph, Ly.N, H, ph, kgs, sg, ng);
                else bwd_layer<1>(G, pg, sm + Ly.w_off, ph, Ly.N, H, ph, kgs, sg, ng);
                __syncthreads();
                LTRACE(8 + 2 * l);
            }
        }
    }
}

// block sum of every thread's loss_acc in a fixed order -> *out
__device__ __forceinline__ void block_loss_to(float *out, float loss_acc, int tid) {
    __shared__ float s_red[LT / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) loss_acc += __shfl_xor_sync(0xffffffffu, loss_acc, o);
    if ((tid & 31) == 0) s_red[tid >> 5] = loss_acc;
    __syncthreads();
    if (tid == 0) {
        float t = 0.0f;
        for (int w = 0; w < LT / 32; ++w) t += s_red[w];
        *out = t;
    }
}

// ------------------------------------------------------------------------------------------------ the gradient kernel
__global__ void __launch_bounds__(LT, BLOCKS_PER_SM) ppo2_grad_kernel(const __grid_constant__ LearnArgs A) {
    extern __shared__ __align__(16) float sm[];
    __shared__ int s_t[TM], s_i[TM];
    __shared__ float s_act[16 * TM], s_alp[16 * TM], s_tgt[TM];   // the tile's actions, old log-probs [d][s]; adv / v_target
    __shared__ float s_cst[16][4];                                 // per action dimension: var, log std, gain, offset
    const int slot = (int)blockIdx.x >= A.nblk[0] ? 1 : 0;
    const int bx = (int)blockIdx.x - (slot ? A.nblk[0] : 0), nbx = A.nblk[slot];
    const int net_id = A.net_of_y[slot];
    const LNet &net = A.net[net_id];
    const int L = net.n_layers;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int sg = (lane & 3) + 4 * warp, ng = lane >> 2;

    load_weights(net, sm, tid);
    if (net_id == 0 && tid < 16) {
        const int d = tid;
        const float sd = d < A.A ? (A.std_vec ? __ldg(A.std_vec + d) : A.std_) : 1.0f;
        float gain = 1.0f, off2 = 0.0f;
        if (net.out_act == 2 && d < A.A) {
            const float lo = __ldg(A.a_min + d), hi = __ldg(A.a_max + d);
            off2 = (lo + hi) / 2.0f;
            gain = hi - off2;
        }
        s_cst[d][0] = sd * sd; s_cst[d][1] = logf(sd); s_cst[d][2] = gain; s_cst[d][3] = off2;
    }
    float loss_acc = 0.0f;
    float *part = A.partial[net_id] + (size_t)bx * (size_t)(net.P + 4);

    const int64_t tiles = (A.count + TM - 1) / TM;
    const LLayer &L0 = net.L[0];
    const LLayer &LO = net.L[L - 1];
    float *gout = sm + net.gout_off;
    const int pgo = LO.N + 4;
    const int64_t N = A.sp.N;

    LTRACE_START();
    for (int64_t tile = bx; tile < tiles; tile += nbx) {
        __syncthreads();   // the previous tile's last phase has finished with H and s_t / s_i
        LTRACE(15);
        tile_samples(A.sp, tile, A.count, s_t, s_i, tid);
        __syncthreads();
        LTRACE(0);
        {   // gather: H_0[s][k] (observations) and the loss phase's inputs (actions, old log-probs, adv / v_target).
            // Thread = (sample s, field lane q): its fields are q, q + 4, ...; ALL its loads are issued before the first
            // store to shared memory -- the obvious load-store loop (gather_obs) serialised six DRAM round trips per tile
            // (phase trace: 9.5 k of 82 k cycles per tile)
            static_assert(LT % TM == 0 && LT / TM == 4, "4 field lanes per sample");
            float *H0 = sm + L0.h_off;
            const int p0 = L0.K + 4;
            const int s = tid & (TM - 1), q = tid >> TM_LOG2;
            const int t = s_t[s];
            const int64_t i = s_i[s], tt = t < 0 ? 0 : t;
            float vo[WMAX / 4], va[4], vl[4], vt = 0.0f;
#pragma unroll
            for (int j = 0; j < WMAX / 4; ++j) {
                const int k = q + 4 * j;
                vo[j] = (t >= 0 && k < A.S) ? __ldg(A.s + (tt * A.S + k) * N + i) : 0.0f;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int d = q + 4 * j;
                const bool on = net_id == 0 && t >= 0 && d < A.A;
                const int64_t off = (tt * A.A + (on ? d : 0)) * N + i;
                va[j] = on ? __ldg(A.a + off) : 0.0f;
                vl[j] = on ? __ldg(A.a_lp + off) : 0.0f;
            }
            if (q == 0 && t >= 0) vt = __ldg((net_id == 0 ? A.adv : A.v_target) + tt * N + i);
#pragma unroll
            for (int j = 0; j < WMAX / 4; ++j) {
                const int k = q + 4 * j;
                if (k < L0.K) H0[s * p0 + k] = vo[j];
            }
            if (net_id == 0) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int d = q + 4 * j;
                    if (d < A.A) { s_act[d * TM + s] = va[j]; s_alp[d * TM + s] = vl[j]; }
                }
            }
            if (q == 0) s_tgt[s] = vt;
        }
        __syncthreads();
        LTRACE(1);
        tile_forward(net, L, sm, gout, sg, ng);
        // ---------------------------------------------------------------- loss and its gradient at the net's output
        {   // two threads per sample: thread `half` takes the action dimensions half, half + 2, ...
            const int sx = tid >> 1, half = tid & 1;
            float *z = gout + (sx < TM ? sx : 0) * pgo;
            const bool live = sx < TM && s_t[sx < TM ? sx : 0] >= 0;
            if (sx >= TM) {
                // 2 x TM threads work in this phase
            } else if (net_id == 0) {
                // Normal(mean, std).log_prob(a) summed over dimensions, PPO2.py:106-112
                float lp = 0.0f, lp_old = 0.0f;
                float dm[8];   // d lp / d z_d of this thread's dimensions
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const int d = 2 * q + half;
                    dm[q] = 0.0f;
                    if (d < A.A) {
                        const float act = s_act[d * TM + sx], var = s_cst[d][0];
                        lp_old += s_alp[d * TM + sx];
                        float m = z[d], dmdz = 1.0f;
                        if (net.out_act == 1) {
                            dmdz = m > 0.0f ? 1.0f : 0.0f;
                            m = fmaxf(m, 0.0f);
                        } else if (net.out_act == 2) {
                            const float th = tanhf(m), gain = s_cst[d][2];
                            m = th * gain + s_cst[d][3];
                            dmdz = gain * (1.0f - th * th);
                        }
                        const float diff = act - m;
                        lp += -(diff * diff) / (2.0f * var) - s_cst[d][1] - 0.91893853320467274178f;
                        dm[q] = diff / var * dmdz;
                    }
                }
                lp += __shfl_xor_sync(0xffffffffu, lp, 1);
                lp_old += __shfl_xor_sync(0xffffffffu, lp_old, 1);
                const float ratio = expf(lp - lp_old);
                const float adv = s_tgt[sx];
                const float lo = 1.0f - A.eps_clip, hi = 1.0f + A.eps_clip;
                const float surr1 = ratio * adv, surr2 = fminf(fmaxf(ratio, lo), hi) * adv;
                if (live && half == 0) loss_acc += -fminf(surr1, surr2);
                // d(-min(surr1, surr2)) / d ratio: -adv unless the clamp is active and selected
                const bool clamped = ratio < lo || ratio > hi;
                const float dldr = (clamped && !(surr1 < surr2)) ? 0.0f : -adv;
                const float c = live ? dldr * ratio * A.inv_count : 0.0f;
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const int d = 2 * q + half;
                    if (d < LO.N) z[d] = d < A.A ? c * dm[q] : 0.0f;
                }
            } else if (half == 0) {
                const float e = z[0] - s_tgt[sx];
                if (live) loss_acc += e * e;
                z[0] = live ? 2.0f * e * A.inv_count : 0.0f;
                for (int d = 1; d < LO.N; ++d) z[d] = 0.0f;
            }
        }
        __syncthreads();
        LTRACE(6);
        tile_backward(net, L, sm, gout, part, tile == bx, tid, sg, ng);
    }
    block_loss_to(part + net.P, loss_acc, tid);
}

// Sum of the per-block partial gradients in block order: one thread per parameter (consecutive threads read consecutive
// addresses of every partial), the loads of eight partials in flight at a time.  A separate, wide launch: folded into
// the gradient kernel as "the last block to finish reduces" it serialised 64 x 6.9 k dependent L2 reads on one SM and
// cost three times the gradient computation itself (130 of 190 us per 16 k-sample mini-batch).
struct ReduceArgs {
    const float *partial[2];
    float *grad[2];
    float *loss_out;
    int P[2], first_block[2];   // net j owns blocks first_block[j] .. of the launch
    int nets, nblk[2];
    float inv_count;
    // entropy bonus of the fixed-std Gaussian (a constant of the loss value): slot `ent_slot` (-1: none) gets
    // -entropy_coef * sum_d (0.5 + 0.5 log(2 pi) + log std_d), PPO2.py:107,116
    int ent_slot, A;
    float ent_coef, std_;
    const float *std_vec;
    // factor of slot 1's gradient and loss, i.e. of the critic of a two-net launch: value_coef for the v1 critic (c_v mse
    // of the joint loss), 1 for PPO2.  Selected by slot (j == 1) rather than indexed: an indexed per-slot factor moved the
    // kernel's block and address arithmetic off the uniform datapath, and b200_ppo2_grad measured 3.7 % (4096 samples)
    // and 4.1 % (16,384) slower than the parent on a B200 at 1000 W (profiles/ppo1/README.md)
    float scale1;
};
__global__ void __launch_bounds__(256) ppo2_reduce_kernel(const __grid_constant__ ReduceArgs a) {
    const int j = (a.nets > 1 && (int)blockIdx.x >= a.first_block[1]) ? 1 : 0;
    const int p = ((int)blockIdx.x - a.first_block[j]) * 256 + (int)threadIdx.x;
    const int P = a.P[j];
    if (p > P) return;
    const size_t stride = (size_t)(P + 4);
    const float *base = a.partial[j] + p;
    float t = 0.0f;
    int b = 0;
    const int nblk = a.nblk[j];
    for (; b + 8 <= nblk; b += 8) {
        float v[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) v[q] = __ldcg(base + (size_t)(b + q) * stride);
#pragma unroll
        for (int q = 0; q < 8; ++q) t += v[q];
    }
    for (; b < nblk; ++b) t += __ldcg(base + (size_t)b * stride);
    const float scale = j == 1 ? a.scale1 : 1.0f;
    if (p < P) {
        a.grad[j][p] = t * scale;
        return;
    }
    float loss = t * a.inv_count * scale;
    if (j == a.ent_slot) {
        float h = 0.0f;
        for (int d = 0; d < a.A; ++d) h += 0.5f + 0.9189385332046727f + logf(a.std_vec ? a.std_vec[d] : a.std_);
        loss -= a.ent_coef * h;
    }
    a.loss_out[j] = loss;
}

// PPO v1 advantage (the joint loss of b200_ppo1_grad): adv = R_hat - V(s) with the CURRENT critic at the batch's samples,
// before ppo2_grad_kernel reads adv.  The critic blocks of ppo2_grad_kernel run the same tile_samples and tile_forward on
// the same shared-memory layout, and the observations reach H_0 unchanged on both paths, so V is bit-identical to the V
// those blocks compute from the same weights.  A separate launch rather than the critic forward inside the actor's
// blocks: that would put both nets' weights into those blocks and change the shipped gradient kernel; this costs one more
// read of the observations.
struct AdvArgs {
    LNet net;                    // the critic
    int S;
    PpoSampler sp;
    int64_t count;
    const float *s, *ret_hat;
    float *adv, *value;          // value may be NULL
};
__global__ void __launch_bounds__(LT, BLOCKS_PER_SM) ppo1_advantage_kernel(const __grid_constant__ AdvArgs A) {
    extern __shared__ __align__(16) float sm[];
    __shared__ int s_t[TM], s_i[TM];
    const LNet &net = A.net;
    const int L = net.n_layers;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int sg = (lane & 3) + 4 * warp, ng = lane >> 2;
    load_weights(net, sm, tid);
    const int64_t tiles = (A.count + TM - 1) / TM, N = A.sp.N;
    const LLayer &L0 = net.L[0];
    float *gout = sm + net.gout_off;
    const int pgo = net.L[L - 1].N + 4;
    LTRACE_START();
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        __syncthreads();   // the previous tile's last reads of H and s_t / s_i are done
        tile_samples(A.sp, tile, A.count, s_t, s_i, tid);
        __syncthreads();
        gather_obs(A.s, A.S, N, L0.K, s_t, s_i, sm + L0.h_off, L0.K + 4, tid);
        __syncthreads();
        tile_forward(net, L, sm, gout, sg, ng);
        if (tid < TM && s_t[tid] >= 0) {
            const int64_t b = (int64_t)s_t[tid] * N + s_i[tid];
            const float v = gout[tid * pgo];
            A.adv[b] = __fsub_rn(__ldg(A.ret_hat + b), v);
            if (A.value) A.value[b] = v;
        }
    }
}

// ------------------------------------------------------------------------------------------------ DQN / Double DQN
// Three kernels on the same tiles and GEMM helpers as the PPO update (64-sample tiles, 256 threads, weights resident in
// shared memory, fp32 FMA pipe, accurate tanhf; Q-net = tanh hidden layers and an identity head of A <= 64 outputs):
//   dqn_act_kernel     epsilon-greedy action of n instances from field-major observations [S][n]
//   dqn_target_kernel  y = r + gamma (1 - done) Q_next for one mini-batch drawn from the replay ring
//   dqn_grad_kernel    gradient of mse(Q(s)[a], y) into per-block partials, summed by ppo2_reduce_kernel
//
// Greedy index: the first maximum over the A outputs (lowest index on ties); a NaN output counts as larger than every
// number and the first NaN wins, as torch.argmax.
//
// Exploration draw of instance i (global index g = offset + i) at step k: ONE Philox4x32-10 block with
//     key     = (seed lo, seed hi ^ 0x44514E41 "DQNA"),
//     counter = (g lo, g hi, k lo, (k hi) << 8)
// (the counter layout of K-POLICY's noise, in a key domain of its own).  Words r0, r1 of the block:
//     explore  <=>  (r0 >> 8) * 2^-24 < epsilon        (24-bit uniform in [0, 1): epsilon 0 never, 1 always explores)
//     index     =  (r1 * A) >> 32                      (multiply-high: uniform over [0, A) up to 2^-32 / A)
// The draw does not depend on n, on the launch geometry or on the instance's position in the batch.
//
// Replay sampling: sample j of a mini-batch is ring position p = row * N + i with
//     h = splitmix64(sample_key + (j + 1) * 0x9E3779B97F4A7C15),  b = (h * V N) >> 64  (a 64-bit multiply-high),
//     row = (newest_row - b / N) mod R,  i = b mod N
// i.e. uniform WITH replacement over the V = valid_rows newest rows; a caller-given index[j] (ring positions) overrides
// it.  The same function runs on the host (b200_dqn_sample_indices).
#define B200_DQN_KEY_DOMAIN 0x44514E41u

__host__ __device__ __forceinline__ uint64_t dqn_mix(uint64_t key, uint64_t j) {
    uint64_t z = key + (j + 1) * 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
struct DqnSampler {
    int64_t R, N, newest, V;
    const int64_t *index;
    uint64_t key;
    __host__ __device__ __forceinline__ int64_t pos(int64_t j) const {
        if (index) return index[j];
        const uint64_t h = dqn_mix(key, (uint64_t)j), vn = (uint64_t)(V * N);
#ifdef __CUDA_ARCH__
        const uint64_t b = __umul64hi(h, vn);
#else
        const uint64_t b = (uint64_t)(((unsigned __int128)h * vn) >> 64);
#endif
        const int64_t back = (int64_t)(b / (uint64_t)N), i = (int64_t)b - back * N;
        int64_t row = newest - back;
        if (row < 0) row += R;
        return row * N + i;
    }
};

// Forward-only pass of the tile in X: the layers alternate between P and Q (all three [TM][pw]); returns the buffer that
// holds the output [TM][A].  Ends with a barrier.  X is not written, so a second net can run on the same input.
__device__ __forceinline__ const float *dqn_forward(const LNet &net, const float *w, const float *X, float *P, float *Q,
                                                    int pw, int sg, int ng) {
    const float *in = X;
    float *out = P;
#pragma unroll
    for (int l = 0; l < LMAX; ++l) {
        if (l < net.n_layers) {
            fwd_any(net.L[l], w, in, pw, out, pw, l + 1 < net.n_layers, sg, ng);
            __syncthreads();
            in = out;
            out = out == P ? Q : P;
        }
    }
    return in;
}

// first maximum of z[0 .. A - 1], NaN above every number (torch.argmax)
__device__ __forceinline__ int dqn_argmax(const float *z, int A) {
    int best = 0;
    float bv = z[0];
    for (int a = 1; a < A; ++a) {
        const float v = z[a];
        if (bv == bv && (v > bv || v != v)) { bv = v; best = a; }
    }
    return best;
}

struct DqnActArgs {
    LNet net;
    int S, A, pw, wfl;           // wfl: floats of the weights in shared memory; pw: row pitch of X / P / Q
    int64_t n, off;
    const float *obs, *table;
    float epsilon;
    uint64_t seed, step;
    int32_t *index;
    float *value, *q;            // q may be NULL
};
__global__ void __launch_bounds__(LT, BLOCKS_PER_SM) dqn_act_kernel(const __grid_constant__ DqnActArgs A) {
    extern __shared__ __align__(16) float sm[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int sg = (lane & 3) + 4 * warp, ng = lane >> 2;
    float *X = sm + A.wfl, *P = X + TM * A.pw, *Q = P + TM * A.pw;
    load_weights(A.net, sm, tid);
    const int64_t tiles = (A.n + TM - 1) / TM;
    const int K0 = A.net.L[0].K;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        __syncthreads();   // the previous tile's outputs have been read
        {
            const int s = tid & (TM - 1), q = tid >> TM_LOG2;
            const int64_t i = tile * TM + s;
            for (int k = q; k < K0; k += LT / TM)
                X[s * A.pw + k] = (i < A.n && k < A.S) ? __ldg(A.obs + (int64_t)k * A.n + i) : 0.0f;
        }
        __syncthreads();
        const float *Z = dqn_forward(A.net, sm, X, P, Q, A.pw, sg, ng);
        if (tid < TM) {
            const int64_t i = tile * TM + tid;
            if (i < A.n) {
                int idx = dqn_argmax(Z + tid * A.pw, A.A);
                Philox rng(A.seed, (uint64_t)(A.off + i), (uint32_t)A.step);
                rng.k1 ^= B200_DQN_KEY_DOMAIN;
                rng.c3 = (uint32_t)(A.step >> 32) << 8;
                rng.block();
                if ((float)(rng.r[0] >> 8) * (1.0f / 16777216.0f) < A.epsilon)
                    idx = (int)(((uint64_t)rng.r[1] * (uint32_t)A.A) >> 32);
                A.index[i] = idx;
                A.value[i] = __ldg(A.table + idx);
            }
        }
        if (A.q) {
            for (int e = tid; e < A.A * TM; e += LT) {
                const int a = e >> TM_LOG2, s = e & (TM - 1);
                const int64_t i = tile * TM + s;
                if (i < A.n) A.q[(int64_t)a * A.n + i] = Z[s * A.pw + a];
            }
        }
    }
}

// Target of one mini-batch.  Shared memory: the target net's weights, with double_q the online net's after them, then X /
// P / Q [64][W + 4] (W = the widest layer or input).  At the largest nets (64 inputs, four 64-wide layers, 64 actions)
// that is 2 x 70.6 KB + 3 x 17.4 KB = 193.4 KB, under the 227 KB of a block; the demo's 2-64-64-47 nets take 2 x 38.7 KB
// + 3 x 17.4 KB = 129.6 KB (one block per SM).
struct DqnTargetArgs {
    LNet tnet, onet;             // same shapes, hence the same offsets
    int S, A, pw, wfl, double_q;
    DqnSampler sp;
    int64_t count;
    const float *s_, *r;
    const uint8_t *done;
    float gamma;
    float *y;
};
__global__ void __launch_bounds__(LT, BLOCKS_PER_SM) dqn_target_kernel(const __grid_constant__ DqnTargetArgs A) {
    extern __shared__ __align__(16) float sm[];
    __shared__ int s_t[TM], s_i[TM], s_arg[TM];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int sg = (lane & 3) + 4 * warp, ng = lane >> 2;
    float *wo = sm + A.wfl;
    float *X = sm + (A.double_q ? 2 : 1) * A.wfl, *P = X + TM * A.pw, *Q = P + TM * A.pw;
    load_weights(A.tnet, sm, tid);
    if (A.double_q) load_weights(A.onet, wo, tid);
    const int64_t tiles = (A.count + TM - 1) / TM, N = A.sp.N;
    const int K0 = A.tnet.L[0].K;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        __syncthreads();
        tile_samples(A.sp, tile, A.count, s_t, s_i, tid);
        __syncthreads();
        gather_obs(A.s_, A.S, N, K0, s_t, s_i, X, A.pw, tid);
        __syncthreads();
        if (A.double_q) {
            const float *Z = dqn_forward(A.onet, wo, X, P, Q, A.pw, sg, ng);
            if (tid < TM) s_arg[tid] = dqn_argmax(Z + tid * A.pw, A.A);
            __syncthreads();
        }
        const float *Z = dqn_forward(A.tnet, sm, X, P, Q, A.pw, sg, ng);
        if (tid < TM && s_t[tid] >= 0) {
            const float *z = Z + tid * A.pw;
            const float qn = z[A.double_q ? s_arg[tid] : dqn_argmax(z, A.A)];
            const int64_t p = (int64_t)s_t[tid] * N + s_i[tid];
            const float r = __ldg(A.r + p);
            // a done transition (terminal OR time-out) takes y = r: nothing of Q_next, not even a non-finite value
            A.y[tile * TM + tid] = __ldg(A.done + p) ? r : __fadd_rn(r, __fmul_rn(A.gamma, qn));
        }
    }
}

// Gradient of mean_j (Q(s_j)[a_j] - y_j)^2: ppo2_grad_kernel's tile loop for one net with the squared error at the
// selected output as the loss (dZ_out[s][n] = n == a_s ? 2 (Q - y) / M : 0).  An action outside [0, A) reads Q = NaN,
// so the loss shows it.
struct DqnGradArgs {
    LNet net;
    int S, A;
    DqnSampler sp;
    int64_t count;
    const float *s, *y;
    const int32_t *a;
    float inv_count;
    float *partial;              // [gridDim.x][P + 4]
};
__global__ void __launch_bounds__(LT, BLOCKS_PER_SM) dqn_grad_kernel(const __grid_constant__ DqnGradArgs A) {
    extern __shared__ __align__(16) float sm[];
    __shared__ int s_t[TM], s_i[TM], s_a[TM];
    __shared__ float s_y[TM];
    const LNet &net = A.net;
    const int L = net.n_layers;
    const int bx = blockIdx.x, nbx = gridDim.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int sg = (lane & 3) + 4 * warp, ng = lane >> 2;
    load_weights(net, sm, tid);
    float loss_acc = 0.0f;
    float *part = A.partial + (size_t)bx * (size_t)(net.P + 4);
    const int64_t tiles = (A.count + TM - 1) / TM, N = A.sp.N;
    const LLayer &L0 = net.L[0];
    const LLayer &LO = net.L[L - 1];
    float *gout = sm + net.gout_off;
    const int pgo = LO.N + 4;
    LTRACE_START();
    for (int64_t tile = bx; tile < tiles; tile += nbx) {
        __syncthreads();
        const int64_t p = tile_samples(A.sp, tile, A.count, s_t, s_i, tid);
        if (tid < TM) {
            s_a[tid] = p >= 0 ? __ldg(A.a + p) : 0;
            s_y[tid] = p >= 0 ? __ldg(A.y + tile * TM + tid) : 0.0f;
        }
        __syncthreads();
        gather_obs(A.s, A.S, N, L0.K, s_t, s_i, sm + L0.h_off, L0.K + 4, tid);
        __syncthreads();
        tile_forward(net, L, sm, gout, sg, ng);
        {   // four lanes per sample, in one warp: all read Q[a] before any of them writes dZ over the row
            const int sx = tid >> 2, q = tid & 3;
            float *z = gout + sx * pgo;
            const bool live = s_t[sx] >= 0;
            const int act = s_a[sx];
            const float qa = (unsigned)act < (unsigned)A.A ? z[act] : __int_as_float(0x7fc00000);
            const float e = qa - s_y[sx];
            __syncwarp();
            if (live && q == 0) loss_acc += e * e;
            const float c = live ? 2.0f * e * A.inv_count : 0.0f;
            for (int d = q; d < LO.N; d += 4) z[d] = d == act ? c : 0.0f;
        }
        __syncthreads();
        tile_backward(net, L, sm, gout, part, tile == bx, tid, sg, ng);
    }
    block_loss_to(part + net.P, loss_acc, tid);
}

// ------------------------------------------------------------------------------------------------ clip + Adam
struct AdamArgs {
    int64_t off[2], len[2];
    float lr[2];
    float *param, *m, *v;
    const float *grad;
    float one_minus_b1, b2, one_minus_b2, eps, bc1, bc2_sqrt, max_norm, grad_scale;
    float *norm_out;
};
constexpr int AT = 1024;

__global__ void __launch_bounds__(AT) adam_kernel(const __grid_constant__ AdamArgs a) {
    __shared__ float s_red[AT / 32];
    __shared__ float s_total;
    const int seg = blockIdx.y, tid = threadIdx.x;
    const int64_t off = a.off[seg], P = a.len[seg];
    const float *g = a.grad + off;
    // total_norm of clip_grad_norm_, every block in the same order
    float ss = 0.0f;
    for (int64_t p = tid; p < P; p += AT) {
        const float x = __ldcg(g + p) * a.grad_scale;
        ss = fmaf(x, x, ss);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    if ((tid & 31) == 0) s_red[tid >> 5] = ss;
    __syncthreads();
    if (tid == 0) {
        float t = 0.0f;
        for (int w = 0; w < AT / 32; ++w) t += s_red[w];
        s_total = t;
    }
    __syncthreads();
    const float norm = sqrtf(s_total);
    float coef = a.grad_scale;
    if (a.max_norm > 0.0f) coef *= fminf(a.max_norm / (norm + 1e-6f), 1.0f);
    if (blockIdx.x == 0 && tid == 0 && a.norm_out) a.norm_out[seg] = norm;
    const float step_size = a.lr[seg] / a.bc1;
    float *pp = a.param + off, *pm = a.m + off, *pv = a.v + off;
    for (int64_t p = (int64_t)blockIdx.x * AT + tid; p < P; p += (int64_t)gridDim.x * AT) {
        const float gr = __ldcg(g + p) * coef;
        float m = pm[p], v = pv[p];
        m = m + (gr - m) * a.one_minus_b1;                  // exp_avg.lerp_(grad, 1 - beta1)
        v = v * a.b2 + a.one_minus_b2 * gr * gr;            // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1 - beta2)
        const float denom = sqrtf(v) / a.bc2_sqrt + a.eps;
        pp[p] = pp[p] - step_size * (m / denom);            // param.addcdiv_(exp_avg, denom, value=-step_size)
        pm[p] = m;
        pv[p] = v;
    }
}

// ------------------------------------------------------------------------------------------------ host side
int pad_n(int n) { return n <= 8 ? 8 : n <= 16 ? 16 : n <= 32 ? 32 : 64; }

// max_out: the widest output layer the caller's loss handles (16 for the PPO heads, 64 for a Q-net)
int fill_net(const b200_mlp *m, int max_out, LNet *net) {
    *net = LNet{};
    if (m->n_layers < 1 || m->n_layers > LMAX) return B200ENV_ESIZE;
    net->n_layers = m->n_layers;
    net->out_act = m->out_act;
    int off = 0, P = 0;
    for (int l = 0; l < m->n_layers; ++l) {
        const int in = m->dims[l], out = m->dims[l + 1];
        if (in < 1 || out < 1 || in > WMAX || out > WMAX) return B200ENV_ESIZE;
        if (!m->w[l] || !m->b[l]) return B200ENV_ENULL;
        LLayer &Ly = net->L[l];
        const bool last = l + 1 == m->n_layers;
        if (last && out > max_out) return B200ENV_ESIZE;
        Ly.k_real = in;
        Ly.n_real = out;
        Ly.K = l == 0 ? (in + 7) / 8 * 8 : net->L[l - 1].N;
        Ly.N = pad_n(out);
        Ly.w = m->w[l];
        Ly.b = m->b[l];
        Ly.g_w = P;
        Ly.g_b = P + in * out;
        P += in * out + out;
        {   // entries per thread e = N K / 256 (>= 1), as RN x RK with RK the widest vector load that fits
            int e = 1;   // the smallest power of two with N K / e <= 256 threads (N is a power of two, K a multiple of 8)
            while (e < 16 && Ly.N * Ly.K > e * LT) e *= 2;
            Ly.rk = e >= 4 ? 4 : e;
            Ly.rn = e / Ly.rk;
        }
        Ly.w_off = off; off += Ly.N * (Ly.K + 4);
        Ly.b_off = off; off += Ly.N;
    }
    for (int l = 0; l < m->n_layers; ++l) {
        net->L[l].h_off = off;
        off += TM * (net->L[l].K + 4);
    }
    net->gout_off = off;
    off += TM * (net->L[m->n_layers - 1].N + 4);
    net->P = P;
    net->smem_floats = off;
    return B200ENV_OK;
}

int grid_cap() {
    const int v = b200_sm_count() * BLOCKS_PER_SM;
    return v > GRID_CAP ? GRID_CAP : v;
}

// blocks of a launch over `count` samples: one per tile, at most grid_cap()
int grid_for(int64_t count) {
    const int64_t tiles = (count + TM - 1) / TM;
    const int cap = grid_cap();
    return (int)(tiles < cap ? tiles : cap);
}

constexpr size_t SMEM_MAX = 227 * 1024 - 12 * 1024;   // room for the kernels' static shared memory (~10 KB) next to it

size_t partial_floats(const LNet &n) { return (size_t)GRID_CAP * (size_t)(n.P + 4); }

struct Plan {
    LearnArgs a;
    int nets;
    size_t smem;
};

int make_plan(const b200_ppo2_batch *bt, const b200_mlp *actor, const b200_mlp *critic, float std_, const float *std_vec,
              const float *a_min, const float *a_max, float eps_clip, float entropy_coef, float *grad_actor,
              float *grad_critic, float *loss_out, void *workspace, size_t workspace_bytes, Plan *pl) {
    if (!bt || (!actor && !critic) || !loss_out || !workspace) return B200ENV_ENULL;
    if (!bt->s || (actor && !bt->adv) || (critic && !bt->v_target)) return B200ENV_ENULL;
    if (bt->T <= 0 || bt->N <= 0 || bt->N >= ((int64_t)1 << 31) || bt->T >= ((int64_t)1 << 31)) return B200ENV_ESIZE;
    const int64_t B = bt->T * bt->N;
    if (bt->count <= 0 || bt->first < 0 || (!bt->index && bt->first + bt->count > B)) return B200ENV_ESIZE;
    LearnArgs &a = pl->a;
    a = LearnArgs{};
    int rc;
    pl->nets = 0;
    size_t smem_f = 0, ws = 64;   // the partials start after 64 unused bytes, as b200_ppo2_workspace_bytes counts them
    if (actor) {
        if (!grad_actor || !bt->a || !bt->a_lp) return B200ENV_ENULL;
        if (!std_vec && !(std_ > 0.0f)) return B200ENV_EPARAMS;
        if (actor->out_act < 0 || actor->out_act > 2) return B200ENV_EPARAMS;
        if (actor->out_act == 2 && (!a_min || !a_max)) return B200ENV_ENULL;
        if ((rc = fill_net(actor, 16, &a.net[0]))) return rc;
        a.net_of_y[pl->nets++] = 0;
        smem_f = a.net[0].smem_floats;
        a.partial[0] = reinterpret_cast<float *>(static_cast<char *>(workspace) + ws);
        ws += partial_floats(a.net[0]) * 4;
        a.S = actor->dims[0];
        a.A = actor->dims[actor->n_layers];
    }
    if (critic) {
        if (!grad_critic) return B200ENV_ENULL;
        if (critic->dims[critic->n_layers > 0 && critic->n_layers <= 4 ? critic->n_layers : 0] != 1) return B200ENV_EPARAMS;
        if (actor && actor->dims[0] != critic->dims[0]) return B200ENV_EPARAMS;
        if ((rc = fill_net(critic, 16, &a.net[1]))) return rc;
        a.net[1].out_act = 0;
        a.net_of_y[pl->nets++] = 1;
        if ((size_t)a.net[1].smem_floats > smem_f) smem_f = a.net[1].smem_floats;
        a.partial[1] = reinterpret_cast<float *>(static_cast<char *>(workspace) + ws);
        ws += partial_floats(a.net[1]) * 4;
        a.S = critic->dims[0];
    }
    if (ws > workspace_bytes) return B200ENV_ESIZE;
    pl->smem = smem_f * sizeof(float);
    if (pl->smem > SMEM_MAX) return B200ENV_ESIZE;
    a.sp = {bt->T, bt->N, bt->first, bt->index, bt->perm_key, half_bits_for(B)};
    a.count = bt->count;
    a.s = bt->s; a.a = bt->a; a.a_lp = bt->a_lp; a.adv = bt->adv; a.v_target = bt->v_target;
    a.eps_clip = eps_clip;
    a.inv_count = 1.0f / (float)bt->count;
    a.std_ = std_; a.std_vec = std_vec; a.a_min = a_min; a.a_max = a_max;
    a.entropy_coef = entropy_coef;
    a.grad[0] = grad_actor; a.grad[1] = grad_critic;
    a.loss_out = loss_out;
    return B200ENV_OK;
}

// ppo2_reduce_kernel over r.nets slots: r gives everything but the launch's block layout (first_block)
int launch_reduce(ReduceArgs r, cudaStream_t stream) {
    int blocks = 0;
    for (int y = 0; y < r.nets; ++y) {
        r.first_block[y] = blocks;
        blocks += (r.P[y] + 1 + 255) / 256;
    }
    ppo2_reduce_kernel<<<blocks, 256, 0, stream>>>(r);
    return b200_check_launch();
}

int launch_grad(Plan &pl, cudaStream_t stream, float critic_scale = 1.0f) {
    static size_t configured[64] = {0};
    int rc = b200_opt_in_smem(ppo2_grad_kernel, pl.smem, configured);
    if (rc) return rc;
    pl.a.nblk[1] = 0;
    if (pl.nets == 2) {
        // one block per SM; the SMs are dealt to the two nets in proportion to their work per sample (3 x sum K N), so
        // that the actor's and the critic's blocks finish together (an even split left the critic's SMs idle 60 % of the
        // time)
        const int64_t tiles = (pl.a.count + TM - 1) / TM;
        const int cap = grid_cap();
        double work[2] = {0.0, 0.0};
        for (int y = 0; y < 2; ++y) {
            const LNet &n = pl.a.net[pl.a.net_of_y[y]];
            for (int l = 0; l < n.n_layers; ++l) work[y] += (double)n.L[l].K * n.L[l].N;
            work[y] += 2200.0;   // per-tile fixed part (indices, gather, loss, barriers) in units of one K x N product
                                 // term: phase trace, ~20 k of an actor tile's 82 k cycles; with 64 the critic's blocks
                                 // were the tail
        }
        int nb1 = (int)(cap * work[1] / (work[0] + work[1]) + 0.5);
        nb1 = nb1 < 1 ? 1 : (nb1 > cap - 1 ? cap - 1 : nb1);
        pl.a.nblk[0] = (int)(tiles < cap - nb1 ? tiles : cap - nb1);
        pl.a.nblk[1] = (int)(tiles < nb1 ? tiles : nb1);
    } else {
        pl.a.nblk[0] = grid_for(pl.a.count);
    }
    ppo2_grad_kernel<<<pl.a.nblk[0] + pl.a.nblk[1], LT, pl.smem, stream>>>(pl.a);
    ReduceArgs r = {};
    for (int y = 0; y < pl.nets; ++y) {
        const int id = pl.a.net_of_y[y];
        r.partial[y] = pl.a.partial[id];
        r.grad[y] = pl.a.grad[id];
        r.P[y] = pl.a.net[id].P;
    }
    // loss_out is indexed by net id (0 actor, 1 critic): with a single net present its slot is selected here
    r.loss_out = pl.a.loss_out + (pl.nets == 1 ? pl.a.net_of_y[0] : 0);
    r.nets = pl.nets;
    r.nblk[0] = pl.a.nblk[0]; r.nblk[1] = pl.a.nblk[1];
    r.inv_count = pl.a.inv_count;
    r.scale1 = critic_scale;   // slot 1 exists only in two-net launches, and is the critic there
    r.ent_slot = (pl.a.net_of_y[0] == 0 && pl.a.entropy_coef != 0.0f) ? 0 : -1;
    r.A = pl.a.A; r.ent_coef = pl.a.entropy_coef; r.std_ = pl.a.std_; r.std_vec = pl.a.std_vec;
    return launch_reduce(r, stream);
}

int launch_adam(int n_seg, const int64_t *seg_off, const int64_t *seg_len, const float *lr, float *param, const float *grad,
                float *m, float *v, int64_t step, double beta1, double beta2, float eps, float max_norm, float grad_scale,
                float *norm_out, cudaStream_t stream) {
    if (n_seg < 1 || n_seg > 2 || !seg_off || !seg_len || !lr) return B200ENV_EPARAMS;
    if (!param || !grad || !m || !v) return B200ENV_ENULL;
    if (step < 1) return B200ENV_EPARAMS;
    AdamArgs a = {};
    int64_t longest = 0;
    for (int j = 0; j < n_seg; ++j) {
        if (seg_len[j] <= 0 || seg_off[j] < 0) return B200ENV_ESIZE;
        a.off[j] = seg_off[j]; a.len[j] = seg_len[j]; a.lr[j] = lr[j];
        if (seg_len[j] > longest) longest = seg_len[j];
    }
    a.param = param; a.m = m; a.v = v; a.grad = grad;
    // torch.optim.Adam's constants: 1 - beta and the bias corrections in double from the double betas, then rounded
    // (from float betas, 1 - 0.999f = 0.00099998713 instead of 0.001)
    a.one_minus_b1 = (float)(1.0 - beta1);
    a.b2 = (float)beta2;
    a.one_minus_b2 = (float)(1.0 - beta2);
    a.eps = eps;
    a.bc1 = (float)(1.0 - pow(beta1, (double)step));
    a.bc2_sqrt = (float)sqrt(1.0 - pow(beta2, (double)step));
    a.max_norm = max_norm;
    a.grad_scale = grad_scale;
    a.norm_out = norm_out;
    int64_t bx = (longest + (int64_t)AT * 4 - 1) / ((int64_t)AT * 4);
    if (bx < 1) bx = 1;
    if (bx > 64) bx = 64;
    adam_kernel<<<dim3((unsigned)bx, (unsigned)n_seg), AT, 0, stream>>>(a);
    return b200_check_launch();
}

} // namespace

extern "C" B200_API size_t b200_ppo2_workspace_bytes(const b200_mlp *actor, const b200_mlp *critic) {
    size_t ws = 64;
    LNet n;
    if (actor) {
        if (fill_net(actor, 16, &n)) return 0;
        ws += partial_floats(n) * 4;
    }
    if (critic) {
        if (fill_net(critic, 16, &n)) return 0;
        ws += partial_floats(n) * 4;
    }
    return (actor || critic) ? ws : 0;
}

extern "C" B200_API int b200_ppo2_grad(const b200_ppo2_batch *batch, const b200_mlp *actor, const b200_mlp *critic,
                                       float std_, const float *std_vec, const float *a_min, const float *a_max,
                                       float eps_clip, float entropy_coef, float *grad_actor, float *grad_critic,
                                       float *loss_out, void *workspace, size_t workspace_bytes, void *cuda_stream) {
    Plan pl;
    int rc = make_plan(batch, actor, critic, std_, std_vec, a_min, a_max, eps_clip, entropy_coef, grad_actor, grad_critic,
                       loss_out, workspace, workspace_bytes, &pl);
    if (rc) return rc;
    return launch_grad(pl, (cudaStream_t)cuda_stream);
}

namespace {
bool overlaps(const void *a, size_t a_bytes, const void *b, size_t b_bytes) {
    const uintptr_t x = (uintptr_t)a, y = (uintptr_t)b;
    return x < y + b_bytes && y < x + a_bytes;
}
} // namespace

extern "C" B200_API int b200_ppo1_grad(const b200_ppo2_batch *batch, const b200_mlp *actor, const b200_mlp *critic,
                                       float std_, const float *std_vec, const float *a_min, const float *a_max,
                                       float eps_clip, float entropy_coef, float value_coef, float *value,
                                       float *grad_actor, float *grad_critic, float *loss_out, void *workspace,
                                       size_t workspace_bytes, void *cuda_stream) {
    if (!batch || !actor || !critic) return B200ENV_ENULL;
    if (!(value_coef >= 0.0f)) return B200ENV_EPARAMS;
    Plan pl;
    int rc = make_plan(batch, actor, critic, std_, std_vec, a_min, a_max, eps_clip, entropy_coef, grad_actor, grad_critic,
                       loss_out, workspace, workspace_bytes, &pl);
    if (rc) return rc;
    {   // adv and value are written by the advantage launch while R_hat, s, a, a_lp and the index are read by both launches:
        // an output that overlaps an input (e.g. adv == v_target for an in-place call) would be read back as that input
        const size_t tn = (size_t)pl.a.sp.T * (size_t)pl.a.sp.N * sizeof(float);
        const size_t tan_ = tn * (size_t)pl.a.A, tsn = tn * (size_t)pl.a.S;
        const void *in[5] = {batch->v_target, batch->s, batch->a, batch->a_lp, batch->index};
        const size_t in_bytes[5] = {tn, tsn, tan_, tan_, (size_t)(pl.a.sp.first + pl.a.count) * sizeof(int64_t)};
        const void *out[2] = {batch->adv, value};
        for (int o = 0; o < 2; ++o) {
            if (!out[o]) continue;
            for (int k = 0; k < 5; ++k)
                if (in[k] && overlaps(out[o], tn, in[k], in_bytes[k])) return B200ENV_EPARAMS;
        }
        if (value && overlaps(value, tn, batch->adv, tn)) return B200ENV_EPARAMS;
    }
    AdvArgs v = {};
    v.net = pl.a.net[1];
    v.S = pl.a.S;
    v.sp = pl.a.sp;
    v.count = pl.a.count;
    v.s = batch->s; v.ret_hat = batch->v_target;
    v.adv = const_cast<float *>(batch->adv);   // the caller-owned [T][N] buffer this call fills
    v.value = value;
    const size_t smem = (size_t)v.net.smem_floats * sizeof(float);
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    static size_t configured[64] = {0};
    if ((rc = b200_opt_in_smem(ppo1_advantage_kernel, smem, configured))) return rc;
    ppo1_advantage_kernel<<<grid_for(v.count), LT, smem, stream>>>(v);
    if ((rc = b200_check_launch())) return rc;
    return launch_grad(pl, stream, value_coef);
}

extern "C" B200_API int b200_adam_step(int n_seg, const int64_t *seg_off, const int64_t *seg_len, const float *lr,
                                       float *param, const float *grad, float *exp_avg, float *exp_avg_sq, int64_t step,
                                       double beta1, double beta2, float eps, float max_norm, float grad_scale,
                                       float *grad_norm_out, void *cuda_stream) {
    return launch_adam(n_seg, seg_off, seg_len, lr, param, grad, exp_avg, exp_avg_sq, step, beta1, beta2, eps, max_norm,
                       grad_scale, grad_norm_out, (cudaStream_t)cuda_stream);
}

extern "C" B200_API int b200_ppo2_learn(const b200_ppo2_batch *batch, const b200_mlp *actor, const b200_mlp *critic,
                                        float std_, const float *std_vec, const float *a_min, const float *a_max,
                                        float eps_clip, float entropy_coef, int k_epochs, int64_t mini_batch,
                                        float lr_actor, float lr_critic, double beta1, double beta2, float adam_eps,
                                        float max_norm, int64_t step, float *param, float *grad, float *exp_avg,
                                        float *exp_avg_sq, float *loss_out, void *workspace, size_t workspace_bytes,
                                        void *cuda_stream) {
    if (!batch || !actor || !critic || !param || !grad || !exp_avg || !exp_avg_sq) return B200ENV_ENULL;
    if (batch->index) return B200ENV_EPARAMS;   // the loop draws its own permutation per epoch
    if (k_epochs < 1 || mini_batch < 1 || step < 1) return B200ENV_EPARAMS;
    const int64_t B = batch->T * batch->N;
    LNet na, nc;
    int rc;
    if ((rc = fill_net(actor, 16, &na)) || (rc = fill_net(critic, 16, &nc))) return rc;
    const int64_t seg_off[2] = {0, na.P}, seg_len[2] = {na.P, nc.P};
    const float lr[2] = {lr_actor, lr_critic};
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    b200_ppo2_batch bt = *batch;
    Plan pl;
    for (int e = 0; e < k_epochs; ++e) {
        bt.perm_key = batch->perm_key + (uint64_t)e;
        for (int64_t first = 0; first < B; first += mini_batch) {
            bt.first = first;
            bt.count = B - first < mini_batch ? B - first : mini_batch;
            if ((rc = make_plan(&bt, actor, critic, std_, std_vec, a_min, a_max, eps_clip, entropy_coef, grad, grad + na.P,
                                loss_out, workspace, workspace_bytes, &pl))) return rc;
            if ((rc = launch_grad(pl, stream))) return rc;
            if ((rc = launch_adam(2, seg_off, seg_len, lr, param, grad, exp_avg, exp_avg_sq, step, beta1, beta2, adam_eps,
                                  max_norm, 1.0f, nullptr, stream))) return rc;
            ++step;
        }
    }
    return B200ENV_OK;
}

extern "C" B200_API int b200_ppo2_permutation(uint64_t perm_key, int64_t B, int64_t first, int64_t count, int64_t *out_host) {
    if (B <= 0 || first < 0 || count < 0 || first + count > B) return B200ENV_ESIZE;
    if (!out_host && count) return B200ENV_ENULL;
    const int hb = half_bits_for(B);
    for (int64_t j = 0; j < count; ++j) out_host[j] = perm_index(perm_key, first + j, B, hb);
    return B200ENV_OK;
}

// ------------------------------------------------------------------------------------------------ DQN host side
namespace {
// a Q-net: fill_net with heads up to 64 wide, identity head
int dqn_fill(const b200_mlp *m, LNet *n) {
    int rc = fill_net(m, WMAX, n);
    if (rc) return rc;
    return m->out_act == 0 ? B200ENV_OK : B200ENV_EPARAMS;
}
int dqn_weight_floats(const LNet &n) { return n.L[0].h_off; }
// row pitch of the forward-only kernels' X / P / Q buffers: the widest input or output + 4
int dqn_pitch(const LNet &n) {
    int w = n.L[0].K;
    for (int l = 0; l < n.n_layers; ++l) w = n.L[l].N > w ? n.L[l].N : w;
    return w + 4;
}
size_t dqn_y_bytes(int64_t count) { return ((size_t)count * 4 + 63) / 64 * 64; }

bool overlaps_net(const void *x, size_t bytes, const b200_mlp *m) {
    for (int l = 0; l < m->n_layers; ++l)
        if (overlaps(x, bytes, m->w[l], (size_t)m->dims[l] * m->dims[l + 1] * 4) ||
            overlaps(x, bytes, m->b[l], (size_t)m->dims[l + 1] * 4)) return true;
    return false;
}
} // namespace

extern "C" B200_API int b200_dqn_act(int64_t n, const b200_mlp *q, const float *obs, const float *table, float epsilon,
                                     uint64_t seed, uint64_t step, int64_t offset, int32_t *action_index,
                                     float *action_value, float *q_out, void *cuda_stream) {
    if (!q || !obs || !table || !action_index || !action_value) return B200ENV_ENULL;
    if (n <= 0 || n >= ((int64_t)1 << 31)) return B200ENV_ESIZE;
    DqnActArgs a = {};
    int rc = dqn_fill(q, &a.net);
    if (rc) return rc;
    if (!(epsilon >= 0.0f && epsilon <= 1.0f)) return B200ENV_EPARAMS;
    a.S = q->dims[0];
    a.A = q->dims[q->n_layers];
    {   // outputs against inputs and against each other
        const size_t nb = (size_t)n * 4;
        const void *out[3] = {action_index, action_value, q_out};
        const size_t out_b[3] = {nb, nb, nb * (size_t)a.A};
        for (int o = 0; o < 3; ++o) {
            if (!out[o]) continue;
            if (overlaps(out[o], out_b[o], obs, nb * (size_t)a.S) || overlaps(out[o], out_b[o], table, (size_t)a.A * 4) ||
                overlaps_net(out[o], out_b[o], q)) return B200ENV_EPARAMS;
            for (int p = o + 1; p < 3; ++p)
                if (out[p] && overlaps(out[o], out_b[o], out[p], out_b[p])) return B200ENV_EPARAMS;
        }
    }
    a.wfl = dqn_weight_floats(a.net);
    a.pw = dqn_pitch(a.net);
    const size_t smem = ((size_t)a.wfl + 3 * (size_t)TM * a.pw) * sizeof(float);
    if (smem > SMEM_MAX) return B200ENV_ESIZE;
    a.n = n; a.off = offset;
    a.obs = obs; a.table = table;
    a.epsilon = epsilon;
    a.seed = seed; a.step = step;
    a.index = action_index; a.value = action_value; a.q = q_out;
    static size_t configured[64] = {0};
    if ((rc = b200_opt_in_smem(dqn_act_kernel, smem, configured))) return rc;
    dqn_act_kernel<<<grid_for(n), LT, smem, (cudaStream_t)cuda_stream>>>(a);
    return b200_check_launch();
}

extern "C" B200_API size_t b200_dqn_workspace_bytes(const b200_mlp *q, int64_t count) {
    LNet n;
    if (!q || count <= 0 || dqn_fill(q, &n)) return 0;
    return dqn_y_bytes(count) + partial_floats(n) * 4;
}

extern "C" B200_API int b200_dqn_grad(const b200_dqn_batch *bt, const b200_mlp *q, const b200_mlp *q_target, float gamma,
                                      int double_q, float *grad, float *loss_out, void *workspace,
                                      size_t workspace_bytes, void *cuda_stream) {
    if (!bt || !q || !q_target || !grad || !loss_out || !workspace) return B200ENV_ENULL;
    if (!bt->s || !bt->r || !bt->s_ || !bt->a || !bt->done) return B200ENV_ENULL;
    if (bt->R < 2 || bt->N <= 0 || bt->R >= ((int64_t)1 << 31) || bt->N >= ((int64_t)1 << 31) || bt->count <= 0)
        return B200ENV_ESIZE;
    DqnTargetArgs t = {};
    int rc;
    if ((rc = dqn_fill(q, &t.onet)) || (rc = dqn_fill(q_target, &t.tnet))) return rc;
    if (q->n_layers != q_target->n_layers) return B200ENV_EPARAMS;
    for (int l = 0; l <= q->n_layers; ++l)
        if (q->dims[l] != q_target->dims[l]) return B200ENV_EPARAMS;
    if (gamma != gamma) return B200ENV_EPARAMS;
    if (bt->valid_rows < 1 || bt->valid_rows > bt->R - 1 || bt->newest_row < 0 || bt->newest_row >= bt->R)
        return B200ENV_EPARAMS;
    const int S = q->dims[0], A = q->dims[q->n_layers];
    const int64_t count = bt->count;
    if (workspace_bytes < b200_dqn_workspace_bytes(q, count)) return B200ENV_ESIZE;
    {   // grad, loss_out and the workspace are written; the ring, the index and both nets are read
        const size_t rn = (size_t)bt->R * (size_t)bt->N, P = (size_t)t.onet.P;
        const void *in[6] = {bt->s, bt->s_, bt->r, bt->a, bt->done, bt->index};
        const size_t in_b[6] = {rn * S * 4, rn * S * 4, rn * 4, rn * 4, rn, (size_t)count * 8};
        const void *out[3] = {grad, loss_out, workspace};
        const size_t out_b[3] = {P * 4, 4, workspace_bytes};
        for (int o = 0; o < 3; ++o) {
            for (int k = 0; k < 6; ++k)
                if (in[k] && overlaps(out[o], out_b[o], in[k], in_b[k])) return B200ENV_EPARAMS;
            if (overlaps_net(out[o], out_b[o], q) || overlaps_net(out[o], out_b[o], q_target)) return B200ENV_EPARAMS;
            for (int p = o + 1; p < 3; ++p)
                if (overlaps(out[o], out_b[o], out[p], out_b[p])) return B200ENV_EPARAMS;
        }
    }
    DqnSampler sp = {bt->R, bt->N, bt->newest_row, bt->valid_rows, bt->index, bt->sample_key};
    float *y = static_cast<float *>(workspace);
    t.S = S; t.A = A;
    t.wfl = dqn_weight_floats(t.tnet);
    t.pw = dqn_pitch(t.tnet);
    t.double_q = double_q ? 1 : 0;
    t.sp = sp; t.count = count;
    t.s_ = bt->s_; t.r = bt->r; t.done = bt->done;
    t.gamma = gamma;
    t.y = y;
    const size_t smem_t = ((size_t)(1 + t.double_q) * t.wfl + 3 * (size_t)TM * t.pw) * sizeof(float);
    DqnGradArgs g = {};
    g.net = t.onet;
    g.S = S; g.A = A;
    g.sp = sp; g.count = count;
    g.s = bt->s; g.a = bt->a; g.y = y;
    g.inv_count = 1.0f / (float)count;
    g.partial = reinterpret_cast<float *>(static_cast<char *>(workspace) + dqn_y_bytes(count));
    const size_t smem_g = (size_t)g.net.smem_floats * sizeof(float);
    if (smem_t > SMEM_MAX || smem_g > SMEM_MAX) return B200ENV_ESIZE;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    static size_t conf_t[64] = {0}, conf_g[64] = {0};
    if ((rc = b200_opt_in_smem(dqn_target_kernel, smem_t, conf_t)) || (rc = b200_opt_in_smem(dqn_grad_kernel, smem_g, conf_g))) return rc;
    const int blocks = grid_for(count);
    dqn_target_kernel<<<blocks, LT, smem_t, stream>>>(t);
    if ((rc = b200_check_launch())) return rc;
    dqn_grad_kernel<<<blocks, LT, smem_g, stream>>>(g);
    if ((rc = b200_check_launch())) return rc;
    ReduceArgs r = {};
    r.partial[0] = g.partial;
    r.grad[0] = grad;
    r.loss_out = loss_out;
    r.P[0] = g.net.P;
    r.nets = 1;
    r.nblk[0] = blocks;
    r.inv_count = g.inv_count;
    r.scale1 = 1.0f;
    r.ent_slot = -1;
    return launch_reduce(r, stream);
}

extern "C" B200_API int b200_dqn_sample_indices(uint64_t sample_key, int64_t newest_row, int64_t valid_rows, int64_t R,
                                                int64_t N, int64_t first, int64_t count, int64_t *out_host) {
    if (R < 2 || N <= 0 || R >= ((int64_t)1 << 31) || N >= ((int64_t)1 << 31) || first < 0 || count < 0)
        return B200ENV_ESIZE;
    if (valid_rows < 1 || valid_rows > R - 1 || newest_row < 0 || newest_row >= R) return B200ENV_EPARAMS;
    if (!out_host && count) return B200ENV_ENULL;
    const DqnSampler sp = {R, N, newest_row, valid_rows, nullptr, sample_key};
    for (int64_t j = 0; j < count; ++j) out_host[j] = sp.pos(first + j);
    return B200ENV_OK;
}

#ifdef LEARN_TRACE
extern "C" B200_API int b200_learn_trace_read(long long *host) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(host, g_learn_trace, sizeof(long long) * 16);
    long long zero[16] = {0};
    cudaMemcpyToSymbol(g_learn_trace, zero, sizeof(zero));
    return 0;
}
#endif
