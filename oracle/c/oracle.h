/*
 * oracle.h -- CPU restatement of the reference's environment-step hot path.
 *
 * TEST INFRASTRUCTURE.  This library is the checker, never the product: only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load it.
 * Each function restates, in plain C with the reference's own operation order (no FMA
 * contraction: built with -ffp-contract=off), one method of the Python reference and
 * cites the file:line it follows.  It is pinned against fixtures recorded from the
 * unmodified reference (tests/golden/<name>.npz, made by oracle/gen_golden.py).
 *
 * Buffers use the same field-major SoA layout and the same parameter structs as the
 * engine's C ABI (include/b200env.h), all in float64, host memory.
 */
#ifndef RLP_ORACLE_H
#define RLP_ORACLE_H
#include <stdint.h>
#include <stddef.h>
#include "../../include/b200env.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct oracle_io {
    double *state;       /* [F][n] */
    double *time;        /* [n] */
    uint32_t *episode;   /* [n] */
    const double *action;/* [A][n] */
    const double *dis;   /* [D][n] or NULL */
    double *obs;         /* [S][n] or NULL */
    double *next_obs;    /* [S][n] */
    double *reward;      /* [n] */
    uint8_t *done;       /* [n] */
    int32_t *flag;       /* [n] */
    double *reset_obs;   /* [S][n] or NULL */
    int32_t *substeps;   /* [n] or NULL: RK4 sub-steps taken (time-loop envs, note N1) */
} oracle_io;

/* same semantics as b200env_step / b200env_reset / b200env_observe; nthreads > 1 uses OpenMP */
int oracle_step(int env_id, int64_t n, const void *params, const oracle_io *io, uint32_t flags,
                uint64_t seed, int64_t env_index_offset, int nthreads);
int oracle_reset(int env_id, int64_t n, const void *params, const oracle_io *io, const uint8_t *mask,
                 uint64_t seed, int64_t env_index_offset);
int oracle_observe(int env_id, int64_t n, const void *params, const oracle_io *io);

/* Philox4x32-10 block (Random123 known-answer tests are in tests/test_policy_routes_gpu.py) */
void oracle_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);

/* GAE reverse scan, float32 sequential exactly like the Python loop under numpy >= 2
 * (algorithm/policy_base/Proximal_Policy_Optimization2.py:88-98) */
void oracle_gae(int64_t T, int64_t N, const float *r, const float *vs, const float *vs_next, const float *done,
                const float *success, float gamma, float lambda_gamma /* float32(gamma * lmd) */, float *adv,
                float *v_target, double *stats /* += (sum adv, sum adv^2, T*N), may be NULL */);

/* RunningMeanStd.update + Normalization.__call__ (utils/classes.py:626-656), sample by sample; run = [4][dim] =
 * (n, mean, S, std) */
void oracle_norm_seq(int64_t rows, int dim, const double *x, double *y, double *run, int update, double eps);

/* PPO / DPPO (v1) Monte-Carlo returns (Proximal_Policy_Optimization.py:113-119) */
void oracle_mc_returns(int64_t T, int64_t N, const double *r, const uint8_t *done, double gamma, float *ret);

#ifdef __cplusplus
}
#endif
#endif
