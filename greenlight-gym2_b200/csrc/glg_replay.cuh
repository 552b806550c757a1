// glg_replay.cuh -- the off-policy counterpart of glg_rollout.cuh: SB3 2.6.0's ReplayBuffer (common/buffers.py, optimize_memory_usage
// False, handle_timeout_termination True) filled the way OffPolicyAlgorithm._store_transition fills it behind VecNormalize, as
// kernels on the env handle's outputs (glg_replay_* in include/glgym.h).
//
// Storage.  5 Np of a row's floats (240 of 263 in the default stack) are the WeatherForecastObservations block, weather rows
// kw+1 .. kw+Np (columns 0..4, cast to float) of the env's table: a pure function of the bank row index key = table * rows + kw.
// Per slot and env the buffer keeps, for the observation and for the next observation, the row WITHOUT that block (packed like
// the handle's obs_head) plus its key; then action [6], raw reward (f32) and done.  221 B per transition at the default stack
// instead of SB3's 2140 B.  The sample kernel rebuilds the block from the bank with the step kernel's (float) cast, so the raw rows
// it sees are bit for bit the rows the step wrote.
//
// Keys.  The step writes an observation's block from kw = min(k, rows - Np - 1), k = the timestep before the step; reset (kernel
// or in place) writes rows 1..Np of the new table.  So an observation whose env has timestep t right after it was produced has
// kw = min(max(t - 1, 0), rows - Np - 1), and a terminal observation is keyed by the (timestep + 1, table) the env had before the
// step.  The buffer keeps that anchor (timestep, table) per env, taken after every reset and store: the step kernels know nothing
// of the buffer.
//
//   statistics              : glg_roll_moments / finish / apply kernels of glg_rollout.cuh on the buffer's own statistics,
//                             normalised current observation -> the buffer's [B][obs_dim] array (VecNormalize.step_wait / reset)
//   glg_replay_write_kernel : slot pos <- packed heads of the observation (kept from the last store / reset) and of the next
//                             observation (terminal row of a done env under auto-reset), keys, action, reward, done; new anchors.
//                             GLG_ROLL_ROWS envs per CTA, flat over the CTA's packed [rows][n_head] range: coalesced
//   glg_replay_sample_kernel: one warp per sampled transition: Philox draw of (slot, env), heads gathered, forecast block rebuilt
//                             from the bank, normalised + clipped with the current statistics (glg_roll_apply_kernel's arithmetic),
//                             the warp's lanes walking the output row's columns (coalesced stores)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "glg_philox.h"
#include "glg_rollout.cuh"

constexpr int GLG_REPLAY_NT = 256;  // sample kernel: 8 warps = 8 sampled transitions per CTA

struct GlgReplayArgs {
    int B, obs_dim, n_head, nf, fc_off, Np, rows, auto_reset;
    int store;                     // 0: only take anchors and heads (after a reset)
    size_t slot;                   // ring slot written by this store
    const float *obs, *term_obs;   // handle outputs [B][obs_dim]
    const double *reward;          // [B]
    const unsigned char *done;     // [B]
    const int *timestep, *table;   // [B] after the step
    const float *actions;          // [B][6]
    float *last_head;              // [B][n_head]: head of the observation the next transition starts from
    int *anchor_t, *anchor_tbl;    // [B]
    float *head_obs, *head_next;   // [cap][B][n_head]
    int *key_obs, *key_next;       // [cap][B]
    float *act, *rew;              // [cap][B][6], [cap][B]
    unsigned char *dn;             // [cap][B]
};

// bank row kw of an observation produced when its env's timestep became t (see the header comment)
__device__ __forceinline__ int glg_replay_key(int t, int tbl, int rows, int Np) {
    return tbl * rows + min(max(t - 1, 0), rows - Np - 1);
}

__global__ void __launch_bounds__(GLG_ROLL_NT) glg_replay_write_kernel(const GlgReplayArgs A) {
    const int r0 = blockIdx.x * GLG_ROLL_ROWS, r1 = min(r0 + GLG_ROLL_ROWS, A.B);
    const size_t sb = A.slot * (size_t)A.B;
    const int nh = (r1 - r0) * A.n_head;
    for (int i = threadIdx.x; i < nh; i += GLG_ROLL_NT) {
        const int q = i / A.n_head, c = i - q * A.n_head, r = r0 + q;
        const size_t hi = (size_t)r * A.n_head + c;
        const size_t o = (size_t)r * A.obs_dim + (c >= A.fc_off ? c + A.nf : c);  // nf = 0 without a forecast block
        const float cur = __ldg(A.obs + o);
        if (A.store) {
            A.head_obs[sb * A.n_head + hi] = A.last_head[hi];
            A.head_next[sb * A.n_head + hi] = (A.auto_reset && A.done[r]) ? __ldg(A.term_obs + o) : cur;
        }
        A.last_head[hi] = cur;
    }
    if (A.store)
        for (int i = threadIdx.x; i < (r1 - r0) * GLG_NU; i += GLG_ROLL_NT)
            A.act[(sb + r0) * GLG_NU + i] = __ldg(A.actions + (size_t)r0 * GLG_NU + i);
    if (threadIdx.x < r1 - r0) {
        const int r = r0 + threadIdx.x;
        const int t = A.timestep[r], tb = A.table[r];
        if (A.store) {
            const int ta = A.anchor_t[r], tba = A.anchor_tbl[r];
            const unsigned char d = A.done[r];
            A.key_obs[sb + r] = glg_replay_key(ta, tba, A.rows, A.Np);
            A.key_next[sb + r] = (A.auto_reset && d) ? glg_replay_key(ta + 1, tba, A.rows, A.Np) : glg_replay_key(t, tb, A.rows, A.Np);
            A.rew[sb + r] = (float)A.reward[r];
            A.dn[sb + r] = d;
        }
        A.anchor_t[r] = t;
        A.anchor_tbl[r] = tb;
    }
}

struct GlgReplaySampleArgs {
    int n, B, obs_dim, n_head, nf, fc_off, norm_obs, norm_reward;
    uint32_t upper, call;          // slots to draw from; sample-call number (Philox counter word 1)
    unsigned long long seed;
    double clip_obs, clip_reward;
    const double *norm64;          // [obs_dim + 1][2]: mean, 1/sqrt(var + eps) (glg_roll_finish_kernel)
    const double *weather;         // bank [n_tables][rows][10]
    const float *head_obs, *head_next;
    const int *key_obs, *key_next;
    const float *act, *rew;
    const unsigned char *dn;
    float *obs_out, *next_out;     // [n][obs_dim]
    float *act_out, *rew_out, *done_out;  // [n][6], [n], [n]
    int *idx_out;                  // [n][2] (slot, env) or NULL
};

// one observation row of a sampled transition, lanes walking its columns
__device__ __forceinline__ void glg_replay_row(const GlgReplaySampleArgs &S, const float *head, int key, float *out, int lane) {
    const double *w = S.weather + (size_t)key * GLG_ND;
    for (int c = lane; c < S.obs_dim; c += 32) {
        const int f = c - S.fc_off;
        float v;
        if (f >= 0 && f < S.nf) {
            const int i = f / 5;
            v = (float)__ldg(w + (size_t)(1 + i) * GLG_ND + (f - 5 * i));
        } else {
            v = __ldg(head + (f >= S.nf ? c - S.nf : c));
        }
        if (S.norm_obs) v = (float)fmin(fmax(((double)v - S.norm64[2 * c]) * S.norm64[2 * c + 1], -S.clip_obs), S.clip_obs);
        out[c] = v;
    }
}

__global__ void __launch_bounds__(GLG_REPLAY_NT) glg_replay_sample_kernel(const GlgReplaySampleArgs S) {
    const int i = blockIdx.x * (GLG_REPLAY_NT / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= S.n) return;
    uint32_t slot, env;
    glg_replay_draw(S.seed, S.call, (uint32_t)i, S.upper, (uint32_t)S.B, &slot, &env);
    const size_t se = (size_t)slot * S.B + env;
    glg_replay_row(S, S.head_obs + se * S.n_head, S.key_obs[se], S.obs_out + (size_t)i * S.obs_dim, lane);
    glg_replay_row(S, S.head_next + se * S.n_head, S.key_next[se], S.next_out + (size_t)i * S.obs_dim, lane);
    if (lane < GLG_NU) S.act_out[(size_t)i * GLG_NU + lane] = S.act[se * GLG_NU + lane];
    if (lane == 0) {
        double r = S.rew[se];
        if (S.norm_reward) r = fmin(fmax(r * S.norm64[2 * S.obs_dim + 1], -S.clip_reward), S.clip_reward);
        S.rew_out[i] = (float)r;
        S.done_out[i] = S.dn[se] ? 1.0f : 0.0f;
        if (S.idx_out) {
            S.idx_out[2 * (size_t)i] = (int)slot;
            S.idx_out[2 * (size_t)i + 1] = (int)env;
        }
    }
}
