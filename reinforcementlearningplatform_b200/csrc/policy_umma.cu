// policy_umma.cu -- K-POLICY on the 5th-generation tensor cores: tcgen05.mma (UMMA) with TMEM accumulators.
//
// Same contract as policy.cu (Proximal_Policy_Optimization2.choose_action, algorithm/policy_base/
// Proximal_Policy_Optimization2.py:69-76, and the critic forward of learn() :88-90; nets of utils/classes.py:529-615 and
// the 256-wide copies of demonstration/DPPO2/DPPO2-4-UGVForwardObstacleAvoidance/train.py:26-107), rebuilt around the
// Blackwell execution model after round 1's profile showed the legacy HMMA version at 0.50 ms per 1 M instances -- 63 %
// of the device-resident collection step -- and unable to hold a 256-wide layer.
//
// One CTA works on tiles of 128 instances (M = 128 = the TMEM lanes).  Per layer: D[128 x N] (fp32, TMEM) = A[128 x K]
// (activations, shared memory) x W^T (weights [N][K], shared memory), then an epilogue warp-group reads D back with
// tcgen05.ld -- thread r owns instance r -- adds the bias, applies tanh on the SFU, and writes the result straight into
// the next layer's A operand.  fp32-level accuracy comes from the 3xTF32 split kept from round 1: every operand is
// stored as hi = tf32(x) and lo = x - hi and D accumulates A_lo W_hi + A_hi W_lo + A_hi W_hi (tests: <= 5e-6 absolute).
//
// Warp roles (608 threads): warps 0-15 are the epilogue -- two half-groups of four warps per tile slot (a warp may only
// touch the TMEM lane quadrant warp_id % 4, so four warps cover the 128 lanes; the two half-groups of a slot split every
// chunk of accumulator columns); warps 16 and 17 issue the tcgen05.mma of slot 0 / slot 1 from one elected lane each;
// warp 18 feeds the weights with cp.async.bulk (TMA, 1-D) from a pre-packed image in global memory.  Synchronisation is
// mbarrier only:
//   a_full[slot][buf]  (256 arrivals)      epilogue -> MMA: a 32-column K chunk of the next layer's input is in place
//   a_free[slot][buf]  (tcgen05.commit)    MMA -> epilogue: the MMAs that read that chunk have completed
//   d_ready[slot]      (tcgen05.commit)    MMA -> epilogue: the layer's accumulator is complete
//   b_full / b_empty[stage]                weight k-steps streamed through a 4-stage ring (wide nets only)
// Three operating modes, chosen by the host from the layer widths (build_plan):
//   resident, A in TMEM   (the reference's 6-64-64-32-8 actor + 6-64-32-1 critic) the whole weight image (82 KB) stays in
//              shared memory and the ACTIVATIONS never leave tensor memory: the epilogue writes the hi / lo planes of
//              the next layer's input with tcgen05.st and the MMAs are issued in the TS form (A from TMEM, B from shared
//              memory).  Each slot owns 256 TMEM columns (D ping, D pong, A hi, A lo); TWO tiles are in flight per CTA
//              so that the tensor core runs one tile's layer while the other tile's epilogue runs.  Measured reason: in
//              the SS form (A in shared memory) each 128 x 64 x 8 MMA re-reads 4 KB of A, 3 times per k-step -- more
//              than the 128 B/cycle the shared-memory pipe delivers next to the epilogue's own stores;
//   resident, A in shared memory   the same with the activations in a ring of 32 KB chunk buffers (nets whose layer
//              inputs exceed the TMEM budget);
//   streamed   layers up to 256 wide (41-256-256-2): the image does not fit, so every k-step (8 columns of K, hi + lo,
//              N x 64 bytes) is pulled through the ring for each tile; one tile in flight, the layer l+1 MMAs consume
//              32-column chunks of layer l's activations as the epilogue produces them, so the 128 x 256 activation
//              matrix never has to exist in full (only 4 chunk buffers do) and D ping-pongs between the two halves of
//              the 512 TMEM columns.
// Operand layout (both A and W): the canonical K-major, no-swizzle UMMA layout -- 8-row x 16-byte core matrices, rows
// of a core matrix 16 B apart, core matrices 128 B apart along M/N (SBO) and one "slab" (rows x 16 B) apart along K
// (LBO): element (row, k) of an operand with R rows lives at (k / 4) * R * 16 + row * 16 + (k % 4) * 4.  With thread =
// row the epilogue's 16-byte stores of a warp are 512 contiguous bytes: conflict-free without swizzling.
#include "policy_common.cuh"
#include "umma_ptx.cuh"

namespace {
using namespace umma;

constexpr int UM_THREADS = 608;                         // 16 epilogue warps + 2 MMA issuers + weight producer
constexpr int EG_WARPS = 16, MMA_WARP = 16;            // issuer of slot s = warp MMA_WARP + s; producer = warp 18
constexpr int TILE_M = 128;
constexpr int CHUNK_K = 32;                            // activation chunk: 32 columns of K
constexpr uint32_t SLAB = TILE_M * 16;                 // bytes of one 4-column K slab of the A operand
constexpr uint32_t PLANE = (CHUNK_K / 4) * SLAB;       // 16 KB: hi (or lo) plane of a chunk
constexpr uint32_t CHUNK = 2 * PLANE;                  // 32 KB: hi + lo
constexpr int NSTAGE = 4;                              // weight ring (streamed mode)
constexpr uint32_t SMEM_LIMIT = 227 * 1024;
constexpr float TWO_LOG2E = 2.885390081777927f;        // tanh(x) = 1 - 2 / (2^(x * 2 log2 e) + 1)

struct UArgs {
    PolicyPlan p;
    PolicyIO io;
    const unsigned char *image;  // packed weights (global)
    const float *bias;           // packed biases (global)
};

// ------------------------------------------------------------------------------------------------ optional event trace
// -DB200_UMMA_TRACE (tools/build_variant.sh): CTA 0 records (event id, clock64) pairs of one thread per role into a
// global array read back by b200_umma_trace_read -- how the pipeline's per-round latencies were measured
// (profiles/r2/policy_umma.md).  Compiled out of the shipped library.
#ifdef B200_UMMA_TRACE
__device__ long long g_umma_trace[4 * 2048];
__device__ int g_umma_trace_n[4];
// the position is kept in a register of the tracing thread (utrace_pos); one fire-and-forget 16-byte store per event
#define UTRACE_DECL int utrace_pos = 0
#define UTRACE(role, id)                                                                                         \
    do {                                                                                                         \
        if (blockIdx.x == 0 && utrace_pos < 1023) {                                                              \
            *reinterpret_cast<longlong2 *>(&g_umma_trace[(role) * 2048 + 2 * utrace_pos]) =                      \
                make_longlong2((long long)(id), clock64());                                                      \
            g_umma_trace_n[role] = ++utrace_pos;                                                                 \
        }                                                                                                        \
    } while (0)
#else
#define UTRACE_DECL int utrace_pos = 0; (void)utrace_pos
#define UTRACE(role, id) do { } while (0)
#endif

// ------------------------------------------------------------------------------------------------ arithmetic
// tanh of (t / (2 log2 e)) given t: 1 - 2 / (2^t + 1) on the SFU (ex2.approx, rcp.approx), absolute error <= 4e-7;
// 2^t = inf -> 1, 2^t = 0 -> -1
__device__ __forceinline__ float tanh_from_scaled(float t) {
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(t));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
    return fmaf(-2.0f, r, 1.0f);
}

// four activations of row r -> one 16-byte store into the hi plane and one into the lo plane of slab q of a chunk
__device__ __forceinline__ void store_split4(unsigned char *chunk, int q, int r, float y0, float y1, float y2, float y3) {
    uint4 hi, lo;
    hi.x = tf32_hi(y0); hi.y = tf32_hi(y1); hi.z = tf32_hi(y2); hi.w = tf32_hi(y3);
    lo.x = __float_as_uint(y0 - __uint_as_float(hi.x));
    lo.y = __float_as_uint(y1 - __uint_as_float(hi.y));
    lo.z = __float_as_uint(y2 - __uint_as_float(hi.z));
    lo.w = __float_as_uint(y3 - __uint_as_float(hi.w));
    unsigned char *p = chunk + (uint32_t)q * SLAB + (uint32_t)r * 16;
    *reinterpret_cast<uint4 *>(p) = hi;
    *reinterpret_cast<uint4 *>(p + PLANE) = lo;
}

// eight activations of row r -> fp16 hi / lo pairs -> one 16-byte store into each plane of fp16 slab q8 (8 K columns)
__device__ __forceinline__ void store_split8(unsigned char *chunk, int q8, int r, const float *y) {
    uint32_t hi[4], lo[4];
    policy_split_f16x8(y, hi, lo);
    unsigned char *p = chunk + (uint32_t)q8 * SLAB + (uint32_t)r * 16;
    *reinterpret_cast<uint4 *>(p) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4 *>(p + PLANE) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
}

// hidden-layer epilogue for W accumulator columns of row r: D -> tanh(D + b) -> next layer's A chunk.  Written in
// stages over all W values (bias loads first, then every FFMA, every ex2, every rcp ...) so that ptxas sees W independent
// chains: the first version interleaved four values per 16-byte store and reloaded the bias between stores, which
// serialised the groups behind possible shared-memory aliasing -- 2000 cycles per 32-column chunk in the event trace
// against 512 cycles of SFU time.  The accumulator load is issued before the wait for the destination buffer.
template <int W, bool A_TMEM>
__device__ __forceinline__ void epi_tanh_chunk(uint32_t taddr, const float *bias_scaled, float zs, bool next_f16,
                                               unsigned char *chunk, int q0, int r,
                                               uint32_t a_hi_t, uint32_t a_lo_t, uint32_t free_bar, uint32_t free_parity,
                                               int trace_role, int &utrace_pos) {
    uint32_t v[W];
    float t[W];
    if (trace_role >= 0) UTRACE(trace_role, 600);
    tmem_ld<W>(taddr, v);
#pragma unroll
    for (int q = 0; q < W / 4; ++q) {
        const float4 b = *reinterpret_cast<const float4 *>(bias_scaled + 4 * q);
        t[4 * q + 0] = b.x; t[4 * q + 1] = b.y; t[4 * q + 2] = b.z; t[4 * q + 3] = b.w;
    }
    mbar_wait(free_bar, free_parity);
    if (trace_role >= 0) UTRACE(trace_role, 700);
    tmem_wait_ld();
    if (trace_role >= 0) UTRACE(trace_role, 800);
    // tanh(x) = 1 - 2 / (2^t + 1), t = 2 log2(e) x: FFMA, ex2, FADD, rcp, FFMA.  With sixteen epilogue warps the kernel is
    // bound by instruction issue, not by the SFU (ncu: issue slots 2x the SFU's busy cycles), so the plain form wins:
    // sharing one rcp between two or four activations saves SFU operations but costs 2.5 / 3.25 extra issue slots per
    // activation (multiplies + an overflow clamp) and measured no faster (profiles/r2/policy_umma.md).
#pragma unroll
    for (int j = 0; j < W; ++j) t[j] = fmaf(__uint_as_float(v[j]), zs, t[j]);   // zs = 2 log2 e / (the layer's weight scale)
#pragma unroll
    for (int j = 0; j < W; ++j) asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t[j]) : "f"(t[j]));
#pragma unroll
    for (int j = 0; j < W; ++j) asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t[j]) : "f"(t[j] + 1.0f));
#pragma unroll
    for (int j = 0; j < W; ++j) t[j] = fmaf(-2.0f, t[j], 1.0f);
    if (trace_role >= 0) UTRACE(trace_role, 900);
    if (A_TMEM) {
        // hi / lo planes straight into the TMEM columns the next layer's MMAs read as their A operand
#pragma unroll
        for (int j = 0; j < W; ++j) {
            v[j] = tf32_hi(t[j]);
            t[j] -= __uint_as_float(v[j]);
        }
        if (W == 8) tmem_st8(a_hi_t, v);
        else {
#pragma unroll
            for (int c = 0; c + 16 <= W; c += 16) tmem_st16(a_hi_t + c, v + c);
        }
#pragma unroll
        for (int j = 0; j < W; ++j) v[j] = __float_as_uint(t[j]);
        if (W == 8) tmem_st8(a_lo_t, v);
        else {
#pragma unroll
            for (int c = 0; c + 16 <= W; c += 16) tmem_st16(a_lo_t + c, v + c);
        }
        tmem_wait_st();
    } else if (next_f16) {
        // the consumer layer multiplies fp16 pairs: slabs of 8 K columns; q0 counts 4-column slabs of this thread's offset
#pragma unroll
        for (int q = 0; q < W / 8; ++q) store_split8(chunk, (q0 >> 1) + q, r, t + 8 * q);
        fence_proxy_async();
    } else {
#pragma unroll
        for (int q = 0; q < W / 4; ++q) store_split4(chunk, q0 + q, r, t[4 * q + 0], t[4 * q + 1], t[4 * q + 2], t[4 * q + 3]);
        fence_proxy_async();
    }
}

// ------------------------------------------------------------------------------------------------ the kernel
struct BarMap {                       // byte offsets inside the barrier block at the start of dynamic shared memory
    static constexpr uint32_t a_full = 0;       // [2 slots][4 bufs]
    static constexpr uint32_t a_free = 64;      // [2][4]
    static constexpr uint32_t d_ready = 128;    // [2]
    static constexpr uint32_t b_full = 144;     // [NSTAGE]
    static constexpr uint32_t b_empty = 176;    // [NSTAGE]
    static constexpr uint32_t w_ready = 208;
    static constexpr uint32_t tmem_slot = 216;  // u32 written by tcgen05.alloc
    static constexpr uint32_t bytes = 256;
};

// The tcgen05.mma issue loop of slot s, run by ONE lane (chosen with elect.sync) of the slot's own issuer warp: inside an elect-guarded region ptxas knows that a
// single lane is active, keeps descriptors and addresses in uniform registers and issues the three UTCHMMA of a k-step
// back to back.  History (profiles/r2/policy_umma.md): with `if (lane == 0)` every operand of every MMA went through an
// ELECT / R2UR.BROADCAST loop (~30 dependent instructions per MMA, 0.91 ms per 1 M instances); with elect.sync but
// descriptors rebuilt from scratch per k-step (~40 instructions, several LDCU / R2UR round trips) the issue lane was
// still busy 80 % of the time at 600 cycles per k-step (0.60 ms) while the tensor pipe sat at 10 %.  Here everything
// that does not change inside a layer is hoisted and the descriptors advance by additions on their low words.  One issuer
// warp per slot (on different schedulers): the issue-rate probe (tools/umma_rate.py) shows a single thread sustaining one
// 128 x N x 8 MMA per ~41 cycles whatever N <= 64 -- a limit of that thread's instruction stream, not of the tensor pipe:
// two issuing warps reach one per ~28 cycles.
template <bool STREAMED, bool A_TMEM>
__device__ __forceinline__ void mma_issue_loop(const PolicyPlan &P, uint32_t s, uint32_t sbase, uint32_t tmem_base,
                                               int64_t groups, int64_t tiles) {
    const uint32_t nbuf_log2 = (uint32_t)P.nbuf_log2, nbuf_mask = (1u << nbuf_log2) - 1u;
    const int n_layers = P.n_layers, slots = P.slots;
    const uint32_t slot_t = tmem_base + s * (uint32_t)P.slot_cols, pong_off = (uint32_t)P.pong_off;
    const uint32_t a_tm = slot_t + (uint32_t)P.a_col, a_lo_off = (uint32_t)CHUNK_K << nbuf_log2;
    const uint32_t desc_hi = (128u >> 4) | (1u << 14);                      // SBO = 128 B, descriptor version 1
    const uint32_t a_lbo16 = (SLAB >> 4) << 16;
    const uint32_t a_ring16 = ((sbase + P.off_a) & 0x3FFFFu) >> 4, b_base16 = ((sbase + P.off_b) & 0x3FFFFu) >> 4;
    const uint32_t stage16 = P.stage_bytes >> 4;
    const uint32_t bar_af = sbase + BarMap::a_full + s * 32, bar_afr = sbase + BarMap::a_free + s * 32;
    const uint32_t bar_dr = sbase + BarMap::d_ready + s * 8;
    if (!STREAMED) mbar_wait(sbase + BarMap::w_ready, 0);
    UTRACE_DECL;
    uint32_t g = 0, ld = 0, h = 0;
    for (int64_t grp = blockIdx.x; grp < groups; grp += gridDim.x) {
        if (grp * slots + (int64_t)s >= tiles) break;
        for (int li = 0; li < n_layers; ++li) {
            const int K = P.L[li].K, N = P.L[li].N;
            const bool f16 = !A_TMEM && P.L[li].f16 != 0;                    // fp16 pairs: k-steps of 16 (2 slabs of 8)
            const uint32_t idesc = f16 ? umma_idesc_f16(TILE_M, N) : umma_idesc_tf32(TILE_M, N);
            const uint32_t b_lbo16 = (uint32_t)N << 16;                      // (N * 16 B >> 4) in the LBO field
            const uint32_t kstep16 = (uint32_t)N * 4, blo16 = (uint32_t)N * 2;   // N * 64 B and N * 32 B, >> 4
            const uint32_t dcol = slot_t + (ld & 1u) * pong_off;
            ++ld;
            uint32_t acc = 0, b_hi = (b_base16 + (P.L[li].w_off >> 4)) | b_lbo16;
            for (int k0 = 0; k0 < K; k0 += CHUNK_K) {
                const uint32_t buf = g & nbuf_mask;
                UTRACE(2 + s, 1000 + li);
                mbar_wait(bar_af + buf * 8, (g >> nbuf_log2) & 1u);
                tc_fence_after();
                UTRACE(2 + s, 2000 + li);
                // A operand of k-step j: TMEM address or shared-memory descriptor (low word) of the hi plane
                uint32_t a_hi = A_TMEM ? a_tm + buf * CHUNK_K
                                       : (a_ring16 + ((s << nbuf_log2) + buf) * (CHUNK >> 4)) | a_lbo16;
                const int ksteps = min(CHUNK_K, K - k0) >> (f16 ? 4 : 3);
                for (int j = 0; j < ksteps; ++j) {
                    uint32_t stage = 0;
                    if (STREAMED) {
                        stage = h & (NSTAGE - 1);
                        mbar_wait(sbase + BarMap::b_full + stage * 8, (h / NSTAGE) & 1u);
                        tc_fence_after();
                        b_hi = (b_base16 + stage * stage16) | b_lbo16;
                    }
                    if (A_TMEM) {
                        umma_tf32_ts(dcol, a_hi + a_lo_off, b_hi, desc_hi, idesc, acc);             // small terms first
                        umma_tf32_ts(dcol, a_hi, b_hi + blo16, desc_hi, idesc, 1u);
                        umma_tf32_ts(dcol, a_hi, b_hi, desc_hi, idesc, 1u);
                        a_hi += 8;                                                                  // 8 columns of K
                    } else if (f16) {
                        umma_f16_lohi(1u, dcol, a_hi + (PLANE >> 4), b_hi, desc_hi, idesc, acc);
                        umma_f16_lohi(1u, dcol, a_hi, b_hi + blo16, desc_hi, idesc, 1u);
                        umma_f16_lohi(1u, dcol, a_hi, b_hi, desc_hi, idesc, 1u);
                        a_hi += (2 * SLAB) >> 4;                                                    // 16 columns of K
                    } else {
                        umma_tf32_lohi(1u, dcol, a_hi + (PLANE >> 4), b_hi, desc_hi, idesc, acc);
                        umma_tf32_lohi(1u, dcol, a_hi, b_hi + blo16, desc_hi, idesc, 1u);
                        umma_tf32_lohi(1u, dcol, a_hi, b_hi, desc_hi, idesc, 1u);
                        a_hi += (2 * SLAB) >> 4;
                    }
                    acc = 1u;
                    if (STREAMED) {
                        umma_commit(sbase + BarMap::b_empty + stage * 8);
                        ++h;
                    } else {
                        b_hi += kstep16;
                    }
                }
                umma_commit(bar_afr + buf * 8);
                ++g;
            }
            umma_commit(bar_dr);
            UTRACE(2 + s, 3000 + li);
        }
    }
}

// Epilogue: slot s = warp / 8 has TWO half-groups h = (warp / 4) % 2 of four warps each; thread (h, r) owns row r
// (= TMEM lane r) of the slot's tile and, of every chunk of accumulator columns, the half h.  Sixteen epilogue warps
// instead of eight: per-chunk latencies (tcgen05.ld / st round trips, SFU chains, barrier hand-offs) overlap four deep
// per scheduler.  Every chunk barrier therefore counts 256 arrivals.
template <bool A_TMEM>
__device__ __forceinline__ void epilogue_loop(const UArgs &a, int64_t n, unsigned char *smem, uint32_t sbase,
                                              uint32_t tmem_base, int warp, int64_t tiles, int64_t groups) {
    const PolicyPlan &P = a.p;
    const int s = warp >> 3, h = (warp >> 2) & 1;
    const int nbuf = 1 << P.nbuf_log2, nbuf_mask = nbuf - 1;
    const float *bias_s = reinterpret_cast<const float *>(smem + P.off_bias);
    const int r = (warp & 3) * 32 + (threadIdx.x & 31);             // row of the tile = TMEM lane
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;   // this warp's TMEM lane quadrant
    const uint32_t slot_t = tmem_base + lane_base + (uint32_t)(s * P.slot_cols);
    const uint32_t a_hi_base = slot_t + (uint32_t)P.a_col, a_lo_off = (uint32_t)(CHUNK_K * nbuf);
    unsigned char *a_ring = smem + P.off_a + (uint32_t)s * (uint32_t)nbuf * CHUNK;
    float *scr = reinterpret_cast<float *>(smem + P.off_scr) + s * (16 * TILE_M) + r;   // means of row r: scr[j * TILE_M]
    const float *dimc = reinterpret_cast<const float *>(smem + P.off_scr) + 2 * 16 * TILE_M;
    const uint32_t af = sbase + BarMap::a_full + s * 32, afr = sbase + BarMap::a_free + s * 32;
    const uint32_t dr = sbase + BarMap::d_ready + s * 8;
    const bool tracer = h == 0 && r == 0;
    UTRACE_DECL;
    uint32_t g = 0;        // chunks written so far by this slot (ring position)
    uint32_t layers_done = 0;
    for (int64_t grp = blockIdx.x; grp < groups; grp += gridDim.x) {
        const int64_t tile = grp * P.slots + s;
        if (tile >= tiles) break;
        const int64_t i = tile * TILE_M + r;
        const bool live = i < n;
        int pending_A = 0;     // > 0: this row's means sit in scr and still have to be sampled (half-group 0 only)
        for (int li = 0; li < P.n_layers; ++li) {
            const PolicyLayer &L = P.L[li];
            if (L.first) {                       // the layer's input is the observation: K columns, zero-padded
                for (int k0 = 0; k0 < L.K; k0 += CHUNK_K) {
                    const int buf = g & nbuf_mask;
                    mbar_wait(afr + buf * 8, ((g >> P.nbuf_log2) & 1) ^ 1);
                    unsigned char *chunk = a_ring + (uint32_t)buf * CHUNK;
                    const int kw = min(CHUNK_K, L.K - k0);
                    for (int q = h; q < kw / 8; q += 2) {           // 8-column groups dealt to the two half-groups
                        float x[8];
#pragma unroll
                        for (int e = 0; e < 8; ++e) {
                            const int k = k0 + 8 * q + e;
                            x[e] = (live && k < P.S) ? __ldg(a.io.obs + (int64_t)k * n + i) : 0.0f;
                        }
                        if (A_TMEM) {
                            uint32_t hi[8], lo[8];
#pragma unroll
                            for (int e = 0; e < 8; ++e) {
                                hi[e] = tf32_hi(x[e]);
                                lo[e] = __float_as_uint(x[e] - __uint_as_float(hi[e]));
                            }
                            const uint32_t t_hi = a_hi_base + (uint32_t)(buf * CHUNK_K + 8 * q);
                            tmem_st8(t_hi, hi);
                            tmem_st8(t_hi + a_lo_off, lo);
                        } else {
                            store_split4(chunk, 2 * q, r, x[0], x[1], x[2], x[3]);
                            store_split4(chunk, 2 * q + 1, r, x[4], x[5], x[6], x[7]);
                        }
                    }
                    if (A_TMEM) {
                        tmem_wait_st();
                        tc_fence_before();
                    } else {
                        fence_proxy_async();
                    }
                    mbar_arrive(af + buf * 8);
                    ++g;
                }
            }
            // the actor's sampling, deferred to here: the next net's first layer is already with the tensor core
            if (pending_A) {
                if (live) policy_sample_store(a.io, n, i, pending_A, scr, TILE_M, dimc);
                pending_A = 0;
                if (tracer) UTRACE(s, 500 + li);
            }
            if (tracer) UTRACE(s, 100 + li);
            mbar_wait(dr, layers_done & 1);
            tc_fence_after();
            if (tracer) UTRACE(s, 200 + li);
            const uint32_t dcol = slot_t + (uint32_t)((layers_done & 1) * P.pong_off);
            ++layers_done;
            const float zs = bias_s[P.zs_off + li];   // accumulator scale: 1 / (weight scale), x 2 log2 e for tanh layers
            if (L.role == 0) {
                const bool nf16 = !A_TMEM && P.L[li + 1 < P.n_layers ? li + 1 : li].f16 != 0;
                for (int c0 = 0; c0 < L.N; c0 += CHUNK_K) {
                    const int buf = g & nbuf_mask;
                    const uint32_t fbar = afr + buf * 8, fpar = ((g >> P.nbuf_log2) & 1) ^ 1;
                    unsigned char *chunk = a_ring + (uint32_t)buf * CHUNK;
                    const uint32_t t_hi = a_hi_base + (uint32_t)(buf * CHUNK_K);
                    if (L.N - c0 >= CHUNK_K) {                      // 32 columns: 16 each
                        const int o = 16 * h;
                        epi_tanh_chunk<16, A_TMEM>(dcol + c0 + o, bias_s + L.b_off + c0 + o, zs, nf16, chunk, o / 4, r, t_hi + o,
                                                   t_hi + a_lo_off + o, fbar, fpar, tracer ? s : -1, utrace_pos);
                    } else {                                        // 16 columns: 8 each
                        const int o = 8 * h;
                        epi_tanh_chunk<8, A_TMEM>(dcol + c0 + o, bias_s + L.b_off + c0 + o, zs, nf16, chunk, o / 4, r, t_hi + o,
                                                  t_hi + a_lo_off + o, fbar, fpar, tracer ? s : -1, utrace_pos);
                    }
                    if (tracer) UTRACE(s, 300 + li);
                    tc_fence_before();
                    mbar_arrive(af + buf * 8);
                    if (tracer) UTRACE(s, 400 + li);
                    ++g;
                }
            } else if (L.role == 1) {
                // actor output: <= 16 means of this row -> private scratch column; sampled after the next input is out
                if (h == 0) {
                    uint32_t v[16];
                    tmem_ld<16>(dcol, v);
                    tmem_wait_ld();
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        float m = fmaf(__uint_as_float(v[j]), zs, bias_s[L.b_off + j]);
                        if (L.out_act == 1) m = policy_fmax_nan(m, 0.0f);
                        scr[j * TILE_M] = m;
                    }
                    pending_A = L.n_real;
                    tc_fence_before();
                }
            } else if (h == 0) {
                uint32_t v[1];
                tmem_ld<1>(dcol, v);
                tmem_wait_ld();
                if (live) __stcs(a.io.value + i, fmaf(__uint_as_float(v[0]), zs, bias_s[L.b_off]));
                tc_fence_before();
            }
        }
        if (pending_A) {
            if (live) policy_sample_store(a.io, n, i, pending_A, scr, TILE_M, dimc);
            if (tracer) UTRACE(s, 500);
        }
    }
}

__global__ void __launch_bounds__(UM_THREADS, 1)
policy_umma_kernel(const __grid_constant__ UArgs a, int64_t n) {
    extern __shared__ __align__(128) unsigned char smem[];
    const PolicyPlan &P = a.p;
    const uint32_t sbase = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float *bias_s = reinterpret_cast<float *>(smem + P.off_bias);

    if (threadIdx.x == 0) {
        for (int s = 0; s < 2; ++s) {
            for (int b = 0; b < 4; ++b) {
                mbar_init(sbase + BarMap::a_full + (s * 4 + b) * 8, 2 * TILE_M);
                mbar_init(sbase + BarMap::a_free + (s * 4 + b) * 8, 1);
            }
            mbar_init(sbase + BarMap::d_ready + s * 8, 1);
        }
        for (int st = 0; st < NSTAGE; ++st) {
            mbar_init(sbase + BarMap::b_full + st * 8, 1);
            mbar_init(sbase + BarMap::b_empty + st * 8, 1);
        }
        mbar_init(sbase + BarMap::w_ready, 1);
        fence_barrier_init();
    }
    if (warp == MMA_WARP) tmem_alloc(sbase + BarMap::tmem_slot, (uint32_t)P.tmem_cols);
    for (int j = threadIdx.x; j < P.bias_floats; j += UM_THREADS) bias_s[j] = __ldg(a.bias + j);
    if (a.io.action)
        policy_dims_fill(a.io, P.A, reinterpret_cast<float *>(smem + P.off_scr) + 2 * 16 * TILE_M, threadIdx.x, UM_THREADS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t *>(smem + BarMap::tmem_slot);

    const int64_t tiles = (n + TILE_M - 1) / TILE_M;
    const int64_t groups = (tiles + P.slots - 1) / P.slots;    // a group = the `slots` tiles a CTA has in flight

    if (warp < EG_WARPS) {
        // ======================================================================== epilogue groups (two per slot)
        if ((warp >> 3) < P.slots) {
            if (P.a_tmem) epilogue_loop<true>(a, n, smem, sbase, tmem_base, warp, tiles, groups);
            else epilogue_loop<false>(a, n, smem, sbase, tmem_base, warp, tiles, groups);
        }
    } else if (warp < MMA_WARP + 2) {
        // ======================================================================== MMA issuers (one per slot)
        const uint32_t s = (uint32_t)(warp - MMA_WARP);
        if ((int)s < P.slots && elect_one_sync()) {
            if (P.streamed) mma_issue_loop<true, false>(P, s, sbase, tmem_base, groups, tiles);
            else if (P.a_tmem) mma_issue_loop<false, true>(P, s, sbase, tmem_base, groups, tiles);
            else mma_issue_loop<false, false>(P, s, sbase, tmem_base, groups, tiles);
        }
        __syncwarp();
    } else {
        // ======================================================================== weight producer (one thread)
        if (elect_one_sync()) {
            if (!P.streamed) {
                const uint32_t bar = sbase + BarMap::w_ready;
                mbar_expect_tx(bar, P.img_bytes);
                for (uint32_t o = 0; o < P.img_bytes; o += 32768u) {
                    const uint32_t bytes = min(32768u, P.img_bytes - o);
                    bulk_g2s(sbase + P.off_b + o, a.image + o, bytes, bar);
                }
            } else {
                uint32_t h = 0;
                for (int64_t grp = blockIdx.x; grp < groups; grp += gridDim.x) {
                    for (int li = 0; li < P.n_layers; ++li) {
                        const PolicyLayer &L = P.L[li];
                        const uint32_t kstep_bytes = (uint32_t)L.N * 64;
                        for (int kk = 0; kk < L.K / (L.f16 ? 16 : 8); ++kk, ++h) {
                            const int stage = h & (NSTAGE - 1);
                            mbar_wait(sbase + BarMap::b_empty + stage * 8, ((h / NSTAGE) & 1) ^ 1);
                            const uint32_t bar = sbase + BarMap::b_full + stage * 8;
                            mbar_expect_tx(bar, kstep_bytes);
                            bulk_g2s(sbase + P.off_b + (uint32_t)stage * P.stage_bytes, a.image + L.w_off + (uint32_t)kk * kstep_bytes,
                                     kstep_bytes, bar);
                        }
                    }
                }
            }
        }
        __syncwarp();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == MMA_WARP) tmem_dealloc(tmem_base, (uint32_t)P.tmem_cols);
}

// ------------------------------------------------------------------------------------------------ weight packing
struct PackArgs {
    PolicyPlan p;
    const float *w[POLICY_MAX_LAYERS];
    const float *b[POLICY_MAX_LAYERS];
    int k_real[POLICY_MAX_LAYERS];   // nn.Linear in features
    unsigned char *image;
    float *bias;
};

// nn.Linear weights [n_real][k_real] -> the UMMA image, zero-padded, and the bias vector (tanh layers: times 2 log2 e).
// TF32 layers: per k-step of 8 a hi and a lo plane, element (n, k) of a plane at (k % 8 / 4) * N * 16 + n * 16 + (k % 4) * 4.
// fp16 layers (L.f16): weights times 2^s, s chosen per layer so that max |w| 2^s lies in [2^13, 2^14); per k-step of 16 a hi
// and a lo plane of fp16, element (n, k) at (k % 16 / 8) * N * 16 + n * 16 + (k % 8) * 2.  zs[l] = 2^-s (x 2 log2 e for tanh
// layers) is what the epilogue multiplies the accumulator by.  Every block computes its layer's max |w| over all elements
// itself, so the image does not depend on the grid.
__global__ void __launch_bounds__(256) policy_pack_kernel(const __grid_constant__ PackArgs a) {
    __shared__ float s_max[8];
    __shared__ int s_exp;
    const int li = blockIdx.y;
    if (li >= a.p.n_layers) return;
    const PolicyLayer &L = a.p.L[li];
    const int k_real = a.k_real[li];
    const int total = L.K * L.N, real = k_real * L.n_real;
    int sexp = 0;
    if (L.f16) {
        float m = 0.0f;
        for (int e = threadIdx.x; e < real; e += blockDim.x) m = fmaxf(m, fabsf(__ldg(a.w[li] + e)));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = m;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < 8; ++w) m = fmaxf(m, s_max[w]);
            int e = 14;
            if (m > 0.0f && m < 3.0e38f) frexpf(m, &e);      // m = f 2^e, f in [0.5, 1)
            int sx = 14 - e;
            s_exp = sx > 100 ? 100 : (sx < -100 ? -100 : sx);
        }
        __syncthreads();
        sexp = s_exp;
    }
    const float scale = ldexpf(1.0f, sexp);
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
        const int k = e / L.N, nn = e - k * L.N;
        const float w = (nn < L.n_real && k < k_real) ? __ldg(a.w[li] + (int64_t)nn * k_real + k) : 0.0f;
        if (L.f16) {
            const float ws = w * scale;
            const __half hi = __float2half_rn(ws);
            const __half lo = __float2half_rn(ws - __half2float(hi));
            unsigned char *ks = a.image + L.w_off + (uint32_t)(k / 16) * (uint32_t)L.N * 64;
            const uint32_t in_plane = (uint32_t)((k & 15) >> 3) * (uint32_t)L.N * 16 + (uint32_t)nn * 16 + (uint32_t)(k & 7) * 2;
            *reinterpret_cast<__half *>(ks + in_plane) = hi;
            *reinterpret_cast<__half *>(ks + (uint32_t)L.N * 32 + in_plane) = lo;
        } else {
            const uint32_t hi = tf32_hi(w);
            const float lo = w - __uint_as_float(hi);
            unsigned char *ks = a.image + L.w_off + (uint32_t)(k / 8) * (uint32_t)L.N * 64;
            const uint32_t in_plane = (uint32_t)((k & 7) >> 2) * (uint32_t)L.N * 16 + (uint32_t)nn * 16 + (uint32_t)(k & 3) * 4;
            *reinterpret_cast<uint32_t *>(ks + in_plane) = hi;
            *reinterpret_cast<float *>(ks + (uint32_t)L.N * 32 + in_plane) = lo;
        }
    }
    if (blockIdx.x == 0) {
        for (int j = threadIdx.x; j < L.N; j += blockDim.x) {
            const float b = j < L.n_real ? __ldg(a.b[li] + j) : 0.0f;
            a.bias[L.b_off + j] = L.role == 0 ? b * TWO_LOG2E : b;
        }
        if (threadIdx.x == 0) a.bias[a.p.zs_off + li] = (L.role == 0 ? TWO_LOG2E : 1.0f) * ldexpf(1.0f, -sexp);
    }
}

// ------------------------------------------------------------------------------------------------ host side
int add_net(const b200_mlp *m, bool is_actor, int max_width, int max_first_in, bool f16_hidden, PolicyRoute *r) {
    PolicyPlan *P = &r->p;
    if (m->n_layers < 1 || m->n_layers > 4) return B200ENV_ESIZE;
    for (int l = 0; l < m->n_layers; ++l) {
        if (P->n_layers >= POLICY_MAX_LAYERS) return B200ENV_ESIZE;
        const int in = m->dims[l], out = m->dims[l + 1];
        const bool last = l + 1 == m->n_layers;
        // hidden inputs are the previous layer's outputs; output heads: <= 16 actions / 1 value
        if (in < 1 || out < 1 || out > max_width || (l == 0 && in > max_first_in) || (last && out > 16)) return B200ENV_ESIZE;
        PolicyLayer &L = P->L[P->n_layers];
        L.first = l == 0;
        L.f16 = f16_hidden && l > 0;
        L.K = l == 0 ? (in + 7) / 8 * 8 : P->L[P->n_layers - 1].N;               // hidden input = previous padded width
        L.N = (out + 15) / 16 * 16;
        L.n_real = out;
        L.role = last ? (is_actor ? 1 : 2) : 0;
        L.out_act = m->out_act == 2 ? 0 : m->out_act;                            // 2: range map in policy_sample_store
        L.w_off = P->img_bytes;
        P->img_bytes += (uint32_t)L.K * (uint32_t)L.N * (L.f16 ? 4u : 8u);
        L.b_off = P->bias_floats;
        P->bias_floats += L.N;
        r->w[P->n_layers] = m->w[l];
        r->k_real[P->n_layers] = in;
        r->b[P->n_layers] = m->b[l];
        ++P->n_layers;
    }
    return B200ENV_OK;
}

int launch(int64_t n, const PolicyPlan &p, const PolicyIO &io, const unsigned char *image, const float *bias,
           cudaStream_t stream) {
    static size_t configured[64] = {0};
    const int rc = b200_opt_in_smem(policy_umma_kernel, p.smem_bytes, configured);
    if (rc) return rc;
    const int64_t tiles = (n + TILE_M - 1) / TILE_M, groups = (tiles + p.slots - 1) / p.slots, cap = b200_sm_count();
    const UArgs a = {p, io, image, bias};
    policy_umma_kernel<<<(unsigned)(groups < cap ? groups : cap), UM_THREADS, p.smem_bytes, stream>>>(a, n);
    return b200_check_launch();
}

// this file's plan: the first of build_plan's candidates that fits
int build_plan(const b200_mlp *actor, const b200_mlp *critic, PolicyRoute *r) {
    int rc = policy_add_nets(actor, critic, 256, 256, false, r);   // UMMA N <= 256; K chunks <= 8 per layer
    if (rc) return rc;
    PolicyPlan *P = &r->p;
    r->launch = launch;
    int nmax = 16, kmax = 8;
    for (int l = 0; l < P->n_layers; ++l) {
        nmax = P->L[l].N > nmax ? P->L[l].N : nmax;
        kmax = P->L[l].K > kmax ? P->L[l].K : kmax;
    }
    const uint32_t bias_bytes = ((uint32_t)P->bias_floats * 4 + 127) / 128 * 128;
    const int chunks = (kmax + CHUNK_K - 1) / CHUNK_K;
    // candidates in order of preference: resident weights + activations in TMEM (two tiles in flight), resident weights +
    // activations in shared memory with two tiles / one tile in flight, streamed weights
    const uint32_t scr_bytes = 2 * 16 * TILE_M * 4 + 512;                 // actor means awaiting sampling (per slot) + dimc
    for (int cand = 0; cand < 4; ++cand) {
        const int slots = cand <= 1 ? 2 : 1, streamed = cand == 3, a_tmem = cand == 0;
        const int nbuf_log2 = streamed ? 2 : (chunks > 2 ? 2 : 1);
        if (a_tmem && chunks > (1 << nbuf_log2)) continue;                 // TMEM A region holds a whole layer input
        const uint32_t a_bytes = a_tmem ? 0u : (uint32_t)slots * (1u << nbuf_log2) * CHUNK;
        const uint32_t stage = (uint32_t)nmax * 64;
        const uint32_t b_bytes = streamed ? NSTAGE * stage : (P->img_bytes + 127) / 128 * 128;
        const uint32_t total = BarMap::bytes + a_bytes + b_bytes + bias_bytes + scr_bytes;
        const int slot_cols = 2 * nmax + (a_tmem ? 2 * CHUNK_K * (1 << nbuf_log2) : 0);
        int cols = slots * slot_cols, pow2 = 32;
        while (pow2 < cols) pow2 *= 2;
        if (total > SMEM_LIMIT || pow2 > 512) continue;
        if (streamed) {
            // streamed mode: every layer after a net's first multiplies fp16 pairs -- half the image bytes pulled through the
            // ring per tile and half the MMAs (kind::f16 covers K = 16); the image offsets are laid out again
            uint32_t off = 0;
            for (int l = 0; l < P->n_layers; ++l) {
                PolicyLayer &L = P->L[l];
                L.f16 = !L.first;
                L.w_off = off;
                off += (uint32_t)L.K * (uint32_t)L.N * (L.f16 ? 4u : 8u);
            }
            P->img_bytes = off;
        }
        P->slots = slots; P->streamed = streamed; P->nbuf_log2 = nbuf_log2; P->a_tmem = a_tmem;
        P->slot_cols = slot_cols; P->pong_off = nmax; P->a_col = 2 * nmax; P->tmem_cols = pow2;
        P->stage_bytes = stage;
        P->off_a = BarMap::bytes; P->off_b = P->off_a + a_bytes; P->off_bias = P->off_b + b_bytes;
        P->off_scr = P->off_bias + bias_bytes;
        P->smem_bytes = total;
        return B200ENV_OK;
    }
    return B200ENV_ESIZE;
}

} // namespace

int policy_add_nets(const b200_mlp *actor, const b200_mlp *critic, int max_width, int max_first_in, bool f16_hidden,
                    PolicyRoute *r) {
    *r = PolicyRoute{};
    PolicyPlan *P = &r->p;
    int rc;
    if (actor && (rc = add_net(actor, true, max_width, max_first_in, f16_hidden, r))) return rc;
    if (critic && (rc = add_net(critic, false, max_width, max_first_in, f16_hidden, r))) return rc;
    P->S = actor ? actor->dims[0] : critic->dims[0];
    P->A = actor ? actor->dims[actor->n_layers] : 0;
    P->zs_off = P->bias_floats;
    P->bias_floats += POLICY_MAX_LAYERS;
    return B200ENV_OK;
}

int policy_route(const b200_mlp *actor, const b200_mlp *critic, PolicyRoute *r) {
    if (policy_umma16_route(actor, critic, r) == B200ENV_OK) return B200ENV_OK;
    return build_plan(actor, critic, r);
}

int policy_pack(const PolicyRoute &r, void *workspace, size_t bytes, cudaStream_t stream) {
    PackArgs pa = {};
    for (int l = 0; l < r.p.n_layers; ++l) {
        if (!r.w[l] || !r.b[l]) return B200ENV_ENULL;
        pa.w[l] = r.w[l];
        pa.b[l] = r.b[l];
        pa.k_real[l] = r.k_real[l];
    }
    const int rc = policy_workspace_split(r.p, workspace, bytes, &pa.image, &pa.bias);
    if (rc) return rc;
    pa.p = r.p;
    policy_pack_kernel<<<dim3(32, r.p.n_layers), 256, 0, stream>>>(pa);
    return b200_check_launch();
}

// ------------------------------------------------------------------------------------------------ building-block probe
// One 128 x N x K product through exactly the descriptors, layouts and instructions the kernel above uses, with the
// accumulator dumped as is: tests/test_umma_gpu.py checks it against a float64 product (and thereby the hand-packed
// smem / instruction descriptors and the TMEM lane mapping) independently of the policy pipeline.
namespace {
__global__ void __launch_bounds__(128, 1)
umma_probe_kernel(const float *A, const float *W, float *D, int N, int K, int three_pass) {
    extern __shared__ __align__(128) unsigned char smem[];
    const uint32_t sbase = smem_u32(smem);
    const int r = threadIdx.x, warp = r >> 5;
    unsigned char *a_img = smem + 128;                                   // K / 4 slabs, hi plane then lo plane
    const uint32_t a_plane = (uint32_t)(K / 4) * SLAB;
    unsigned char *b_img = a_img + 2 * a_plane;                          // per k-step: hi (N * 32 B), lo (N * 32 B)
    if (r == 0) {
        mbar_init(sbase, 1);
        fence_barrier_init();
    }
    if (warp == 0) tmem_alloc(sbase + 64, 256);
    for (int q = 0; q < K / 4; ++q) {
        const float4 x = *reinterpret_cast<const float4 *>(A + (int64_t)r * K + 4 * q);
        uint4 hi, lo;
        hi.x = tf32_hi(x.x); hi.y = tf32_hi(x.y); hi.z = tf32_hi(x.z); hi.w = tf32_hi(x.w);
        lo.x = __float_as_uint(x.x - __uint_as_float(hi.x)); lo.y = __float_as_uint(x.y - __uint_as_float(hi.y));
        lo.z = __float_as_uint(x.z - __uint_as_float(hi.z)); lo.w = __float_as_uint(x.w - __uint_as_float(hi.w));
        *reinterpret_cast<uint4 *>(a_img + (uint32_t)q * SLAB + r * 16) = hi;
        *reinterpret_cast<uint4 *>(a_img + a_plane + (uint32_t)q * SLAB + r * 16) = lo;
    }
    for (int e = r; e < N * K; e += 128) {
        const int k = e / N, nn = e - k * N;
        const float w = W[(int64_t)nn * K + k];
        const uint32_t hi = tf32_hi(w);
        unsigned char *ks = b_img + (uint32_t)(k / 8) * (uint32_t)N * 64;
        const uint32_t in_plane = (uint32_t)((k & 7) >> 2) * (uint32_t)N * 16 + (uint32_t)nn * 16 + (uint32_t)(k & 3) * 4;
        *reinterpret_cast<uint32_t *>(ks + in_plane) = hi;
        *reinterpret_cast<float *>(ks + (uint32_t)N * 32 + in_plane) = w - __uint_as_float(hi);
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t *>(smem + 64);
    if (r == 0) {
        const uint32_t idesc = umma_idesc_tf32(TILE_M, N);
        uint32_t acc = 0;
        for (int kk = 0; kk < K / 8; ++kk) {
            const uint32_t a_hi = smem_u32(a_img) + (uint32_t)kk * 2 * SLAB, a_lo = a_hi + a_plane;
            const uint32_t b_hi = smem_u32(b_img) + (uint32_t)kk * (uint32_t)N * 64, b_lo = b_hi + (uint32_t)N * 32;
            if (three_pass) {
                umma_tf32(tmem_base, umma_desc(a_lo, SLAB, 128), umma_desc(b_hi, (uint32_t)N * 16, 128), idesc, acc);
                umma_tf32(tmem_base, umma_desc(a_hi, SLAB, 128), umma_desc(b_lo, (uint32_t)N * 16, 128), idesc, 1u);
                acc = 1u;
            }
            umma_tf32(tmem_base, umma_desc(a_hi, SLAB, 128), umma_desc(b_hi, (uint32_t)N * 16, 128), idesc, acc);
            acc = 1u;
        }
        umma_commit(sbase);
    }
    mbar_wait(sbase, 0);
    tc_fence_after();
    const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
    for (int c0 = 0; c0 < N; c0 += 16) {
        uint32_t v[16];
        tmem_ld<16>(tmem_base + lane_base + c0, v);
        tmem_wait_ld();
#pragma unroll
        for (int j = 0; j < 16; ++j) D[(int64_t)r * N + c0 + j] = __uint_as_float(v[j]);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, 256);
}
} // namespace

int policy_umma_probe(const float *A, const float *W, float *D, int N, int K, int three_pass, cudaStream_t stream) {
    if (N < 16 || N > 256 || (N & 15) || K < 8 || K > 64 || (K & 7)) return B200ENV_ESIZE;
    const size_t smem = 128 + 2 * (size_t)(K / 4) * SLAB + (size_t)K * N * 8;
    if (smem > SMEM_LIMIT) return B200ENV_ESIZE;
    if (cudaFuncSetAttribute(umma_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_LIMIT) != cudaSuccess)
        return b200_check_launch();
    umma_probe_kernel<<<1, 128, smem, stream>>>(A, W, D, N, K, three_pass);
    return b200_check_launch();
}

// ------------------------------------------------------------------------------------------------ MMA issue-rate probe
// How long does a chain of `count` tcgen05.mma of shape 128 x N x 8 take when they accumulate into `n_acc` different TMEM
// tiles in rotation (n_acc = 1: every MMA depends on the previous one)?  Operands are whatever the shared memory / TMEM
// holds -- only the timing matters.  Answers whether small-N MMAs are bound by the dependent-accumulate latency
// (profiles/r2/policy_umma.md).
namespace {
__global__ void __launch_bounds__(128, 1) umma_rate_kernel(int N, int count, int n_acc, int ts, long long *cycles) {
    extern __shared__ __align__(128) unsigned char smem[];
    const uint32_t sbase = smem_u32(smem);
    const int warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        mbar_init(sbase, 1);
        mbar_init(sbase + 8, 1);
        fence_barrier_init();
    }
    for (int e = threadIdx.x; e < 16384; e += 128) reinterpret_cast<float *>(smem + 128)[e] = 0.0f;
    if (warp == 0) tmem_alloc(sbase + 64, 512);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t *>(smem + 64);
    // n_acc >= 8 selects TWO issuing warps (n_acc - 8 + 1 accumulators each): is the ~41-cycle cadence a property of the
    // tensor pipe or of one thread's issue path?
    const int issuers = n_acc >= 8 ? 2 : 1, nacc = n_acc >= 8 ? n_acc - 7 : n_acc;
    if (warp < issuers && elect_one_sync()) {
        const uint32_t idesc = umma_idesc_tf32(TILE_M, N), desc_hi = (128u >> 4) | (1u << 14);
        const uint32_t a16 = (((sbase + 128) & 0x3FFFFu) >> 4) | ((SLAB >> 4) << 16);
        const uint32_t b16 = (((sbase + 128 + 8192) & 0x3FFFFu) >> 4) | ((uint32_t)N << 16);
        const long long t0 = clock64();
        for (int k = 0; k < count; ++k) {
            const uint32_t d = tmem_base + (uint32_t)(warp * 192 + (k % nacc) * 64);
            if (ts) umma_tf32_ts(d, tmem_base + 448, b16, desc_hi, idesc, 1u);
            else umma_tf32_lohi(1u, d, a16, b16, desc_hi, idesc, 1u);
        }
        umma_commit(sbase + 8 * warp);
        mbar_wait(sbase + 8 * warp, 0);
        cycles[warp] = clock64() - t0;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, 512);
}
} // namespace

extern "C" B200_API int b200_umma_rate(int N, int count, int n_acc, int ts, long long *cycles_dev, void *cuda_stream) {
    if (N < 16 || N > 64 || (N & 15) || n_acc < 1 || n_acc > 10 || count < 1) return B200ENV_ESIZE;
    if (cudaFuncSetAttribute(umma_rate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024) != cudaSuccess)
        return b200_check_launch();
    umma_rate_kernel<<<1, 128, 128 + 65536 + 8192, (cudaStream_t)cuda_stream>>>(N, count, n_acc, ts, cycles_dev);
    return b200_check_launch();
}

#ifdef B200_UMMA_TRACE
extern "C" B200_API int b200_umma_trace_read(long long *host, int *counts) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(host, g_umma_trace, sizeof(long long) * 4 * 2048);
    cudaMemcpyFromSymbol(counts, g_umma_trace_n, sizeof(int) * 4);
    int zero[4] = {0, 0, 0, 0};
    cudaMemcpyToSymbol(g_umma_trace_n, zero, sizeof(zero));   // (positions restart at 0 with every launch anyway)
    return 0;
}
#endif
