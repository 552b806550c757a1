// glg_philox.h -- stateless counter-based RNG for the per-step parametric uncertainty (hot-path row S2,
// reference: gl_gym/environments/noise.py:3-23 draws 34 uniforms per step from the env's numpy Generator).
// Philox4x32-10 (Salmon et al., SC'11) keyed by the handle seed; the counter is
//   (draw_block, env_step_counter, global_env_id_lo, global_env_id_hi)
// so results do not depend on how the env batch is sharded over GPUs and no RNG state is stored in HBM.
// Doubles are formed like numpy's next_double: (a>>5, b>>6) -> (a*2^26+b)/2^53 in [0,1).
#pragma once
#include <stdint.h>
#include "glg_model.h"

struct GlgPhilox4 {
    uint32_t v[4];
};

GLG_HD uint32_t glg_mulhi32(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32); }

GLG_HD GlgPhilox4 glg_philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = glg_mulhi32(M0, c0), lo0 = M0 * c0;
        const uint32_t hi1 = glg_mulhi32(M1, c2), lo1 = M1 * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += W0; k1 += W1;
    }
    GlgPhilox4 o;
    o.v[0] = c0; o.v[1] = c1; o.v[2] = c2; o.v[3] = c3;
    return o;
}

GLG_HD double glg_u01(uint32_t a, uint32_t b) {
    return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) * (1.0 / 9007199254740992.0);
}

// 34 multiplicative noise terms n_i = -s/2 + s*U_i  (numpy Generator.uniform(low, high) = low + (high-low)*U)
GLG_HD void glg_noise34(uint64_t seed, uint64_t env_id, uint32_t step_ctr, double scale, double *n34) {
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    const uint32_t e0 = (uint32_t)env_id, e1 = (uint32_t)(env_id >> 32);
#pragma unroll 1
    for (int b = 0; b < 17; ++b) {
        GlgPhilox4 r = glg_philox4x32_10((uint32_t)b, step_ctr, e0, e1, k0, k1);
        n34[2 * b] = -0.5 * scale + scale * glg_u01(r.v[0], r.v[1]);
        n34[2 * b + 1] = -0.5 * scale + scale * glg_u01(r.v[2], r.v[3]);
    }
}

// uniform integer in [0, n) for reset-table selection (draw block 64 keeps it disjoint from the noise blocks)
GLG_HD uint32_t glg_rand_below(uint64_t seed, uint64_t env_id, uint32_t step_ctr, uint32_t n) {
    GlgPhilox4 r = glg_philox4x32_10(64u, step_ctr, (uint32_t)env_id, (uint32_t)(env_id >> 32), (uint32_t)seed,
                                     (uint32_t)(seed >> 32));
    return (uint32_t)(((uint64_t)r.v[0] * (uint64_t)n) >> 32);
}

// replay-buffer index of sample i of sample call `call` (draw block 65, counter (65, call, i, 0), key = the buffer's seed):
// slot uniform in [0, upper), env uniform in [0, B)  -- ReplayBuffer.sample's two randint draws
GLG_HD void glg_replay_draw(uint64_t seed, uint32_t call, uint32_t i, uint32_t upper, uint32_t B, uint32_t *slot, uint32_t *env) {
    GlgPhilox4 r = glg_philox4x32_10(65u, call, i, 0u, (uint32_t)seed, (uint32_t)(seed >> 32));
    *slot = (uint32_t)(((uint64_t)r.v[0] * (uint64_t)upper) >> 32);
    *env = (uint32_t)(((uint64_t)r.v[1] * (uint64_t)B) >> 32);
}

// planner sampling noise of candidate c (draw block 66, counter (66, call, draw, c), key = the planner's seed; draw = (it H + t) 3 + p
// for component pair p of step t in CEM iteration it): two standard normals by Box-Muller, u1 = 1 - U in (0, 1], u2 = U'
GLG_HD void glg_plan_normal2(uint64_t seed, uint32_t call, uint32_t draw, uint32_t c, double *z0, double *z1) {
    GlgPhilox4 r = glg_philox4x32_10(66u, call, draw, c, (uint32_t)seed, (uint32_t)(seed >> 32));
    const double u1 = 1.0 - glg_u01(r.v[0], r.v[1]), u2 = glg_u01(r.v[2], r.v[3]);
    const double rad = sqrt(-2.0 * log(u1)), ang = 6.283185307179586 * u2;
    *z0 = rad * cos(ang);
    *z1 = rad * sin(ang);
}
