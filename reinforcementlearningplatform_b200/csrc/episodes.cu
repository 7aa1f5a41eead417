// episodes.cu -- K-EPISODE: episode returns, lengths and end reasons over a time-major [T, N] rollout (sm_100a).
//
// The reference's train loops sum each episode's reward and count its steps, and test the deterministic policy on whole
// episodes.  Here one thread owns one instance column: it walks t forwards, adds r[t] to the episode in progress and,
// on every done row, emits (return, length, terminal_flag) and starts a new episode.  The carry (acc_return,
// acc_length) persists in caller memory between calls, so an episode that spans two rollouts is counted once with its
// full return.
//
// Every done row ends an episode: the tracker is meant for auto-reset rollouts (B200ENV_AUTO_RESET), where the step
// that reports is_terminal has also started the next episode.
//
// Exactness: acc_return += (double)r[t] is one separately rounded float64 add per row in ascending t, so the per-instance
// carry and records equal a float64 loop over t bit for bit.  The statistics (count, sums of return / return^2 / length /
// length^2, flag histogram) go to per-block partials in caller scratch and are added by a second launch in a fixed
// order, like K-GAE's: repeated runs give the same bits.  9 B of HBM traffic per element for float32 rewards.
#include "common.cuh"

namespace {

constexpr int EP_BLOCK = 128;
constexpr int EP_UNROLL = 8;
constexpr int EP_HIST = 16;                      // flags 0..15 get a bin each, anything else the overflow bin
static_assert(B200_EPISODE_STATS == 6 + EP_HIST, "stats layout: count, 4 sums, 16 flag bins, overflow");

__device__ __forceinline__ double ep_warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}

struct EpisodeSums {
    double r1 = 0.0, r2 = 0.0, l1 = 0.0, l2 = 0.0;
};

template <typename TR>
__global__ void __launch_bounds__(EP_BLOCK)
episode_scan_kernel(int64_t T, int64_t N, const TR *__restrict__ r, const uint8_t *__restrict__ done,
                    const int32_t *__restrict__ flag, double *__restrict__ acc_return, int32_t *__restrict__ acc_length,
                    double *__restrict__ ep_return, int32_t *__restrict__ ep_length, int32_t *__restrict__ ep_flag,
                    int first_only, double *__restrict__ partial) {
    __shared__ unsigned int hist[EP_HIST + 1];
    if (partial && threadIdx.x <= EP_HIST) hist[threadIdx.x] = 0u;
    if (partial) __syncthreads();
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    EpisodeSums s;
    if (n < N) {
        double acc = acc_return[n];
        int32_t len = acc_length[n];
        // open: this instance may still emit; in first_only mode it closes after its first episode
        bool open = !first_only || ep_flag[n] == -1;
        bool emitted = false;
        double rec_ret = 0.0;
        int32_t rec_len = 0, rec_flag = -1;
        auto row = [&](double rv, uint8_t dn, int32_t fl) {
            acc = __dadd_rn(acc, rv);
            ++len;
            if (dn) {
                if (open) {
                    rec_ret = acc; rec_len = len; rec_flag = fl;
                    emitted = true;
                    if (first_only) open = false;
                    if (partial) {
                        s.r1 += acc;
                        s.r2 += acc * acc;
                        s.l1 += (double)len;
                        s.l2 += (double)len * (double)len;
                        atomicAdd(&hist[(fl >= 0 && fl < EP_HIST) ? fl : EP_HIST], 1u);   // integer: order-free
                    }
                }
                acc = 0.0;
                len = 0;
            }
        };
        int64_t t = 0;
        // main loop: EP_UNROLL rows per trip, all loads of a trip issued before the dependent adds
        for (; t + EP_UNROLL <= T; t += EP_UNROLL) {
            TR rr[EP_UNROLL];
            uint8_t dd[EP_UNROLL];
            int32_t ff[EP_UNROLL];
#pragma unroll
            for (int u = 0; u < EP_UNROLL; ++u) {
                const int64_t idx = (t + u) * N + n;
                rr[u] = __ldcs(r + idx);
                dd[u] = __ldcs(done + idx);
                ff[u] = __ldcs(flag + idx);
            }
#pragma unroll
            for (int u = 0; u < EP_UNROLL; ++u) row((double)rr[u], dd[u], ff[u]);
        }
        for (; t < T; ++t) {
            const int64_t idx = t * N + n;
            row((double)__ldcs(r + idx), __ldcs(done + idx), __ldcs(flag + idx));
        }
        acc_return[n] = acc;
        acc_length[n] = len;
        if (emitted) {
            if (ep_return) ep_return[n] = rec_ret;
            if (ep_length) ep_length[n] = rec_len;
            if (ep_flag) ep_flag[n] = rec_flag;
        }
    }
    if (partial) {
        // block b owns partial[j * gridDim.x + b] for every entry j of the stats layout
        __shared__ double sh[4][EP_BLOCK / 32];
        const double v[4] = {ep_warp_sum(s.r1), ep_warp_sum(s.r2), ep_warp_sum(s.l1), ep_warp_sum(s.l2)};
        const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
        if (lane == 0) {
#pragma unroll
            for (int k = 0; k < 4; ++k) sh[k][w] = v[k];
        }
        __syncthreads();
        const int64_t G = gridDim.x, b = blockIdx.x;
        if (threadIdx.x < 4) {
            double a = 0.0;
#pragma unroll
            for (int k = 0; k < EP_BLOCK / 32; ++k) a += sh[threadIdx.x][k];
            partial[(1 + threadIdx.x) * G + b] = a;
        } else if (threadIdx.x >= 32 && threadIdx.x <= 32 + EP_HIST) {
            partial[(5 + threadIdx.x - 32) * G + b] = (double)hist[threadIdx.x - 32];
        } else if (threadIdx.x == 64) {
            unsigned int c = 0;
#pragma unroll
            for (int k = 0; k <= EP_HIST; ++k) c += hist[k];
            partial[b] = (double)c;
        }
    }
}

// fixed-order sum of the per-block partials, one block per stats entry j (the 22 entries are reduced side by side):
// thread k adds blocks k, k + 256, ... sequentially, a fixed shared-memory tree combines the 256 thread sums, thread 0
// increments stats[j]
__global__ void __launch_bounds__(256) episode_stats_reduce_kernel(int64_t blocks, const double *__restrict__ partial,
                                                                   double *stats) {
    __shared__ double sh[256];
    const double *p = partial + blockIdx.x * blocks;
    double a = 0.0;
#pragma unroll 4
    for (int64_t k = threadIdx.x; k < blocks; k += 256) a += p[k];
    sh[threadIdx.x] = a;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) stats[blockIdx.x] += sh[0];
}

int64_t episode_grid(int64_t N) { return (N + EP_BLOCK - 1) / EP_BLOCK; }

} // namespace

extern "C" B200_API size_t b200_episode_scratch_bytes(int64_t N) {
    return N <= 0 ? 0 : (size_t)episode_grid(N) * B200_EPISODE_STATS * sizeof(double);
}

extern "C" B200_API int b200_episode_scan(int r_dtype, int64_t T, int64_t N, const void *r, const uint8_t *done,
                                          const int32_t *flag, double *acc_return, int32_t *acc_length,
                                          double *ep_return, int32_t *ep_length, int32_t *ep_flag, int first_only,
                                          double *stats, void *scratch, size_t scratch_bytes, void *cuda_stream) {
    if (T <= 0 || N <= 0 || N >= ((int64_t)1 << 31)) return B200ENV_ESIZE;
    if (r_dtype != B200ENV_F64 && r_dtype != B200ENV_F32) return B200ENV_EDTYPE;
    if (!r || !done || !flag || !acc_return || !acc_length || (first_only && !ep_flag) || (stats && !scratch))
        return B200ENV_ENULL;
    const int64_t grid = episode_grid(N);
    double *partial = nullptr;
    if (stats) {
        if (scratch_bytes < (size_t)grid * B200_EPISODE_STATS * sizeof(double) || ((uintptr_t)scratch & 7))
            return B200ENV_EPARAMS;
        partial = static_cast<double *>(scratch);
    }
    cudaStream_t s = (cudaStream_t)cuda_stream;
    const int fo = first_only ? 1 : 0;
    if (r_dtype == B200ENV_F64)
        episode_scan_kernel<double><<<(unsigned)grid, EP_BLOCK, 0, s>>>(T, N, (const double *)r, done, flag, acc_return,
                                                                         acc_length, ep_return, ep_length, ep_flag, fo,
                                                                         partial);
    else
        episode_scan_kernel<float><<<(unsigned)grid, EP_BLOCK, 0, s>>>(T, N, (const float *)r, done, flag, acc_return,
                                                                        acc_length, ep_return, ep_length, ep_flag, fo,
                                                                        partial);
    if (partial) episode_stats_reduce_kernel<<<B200_EPISODE_STATS, 256, 0, s>>>(grid, partial, stats);
    return b200_check_launch();
}
