// glg_plan.cuh -- receding-horizon planner (glg_plan_* in include/glgym.h): cross-entropy method over action sequences, scored by
// the unchanged step kernels on a second, internal handle of B K planning envs (planning env c = b K + k copies source env b).
//
//   glg_plan_fanout_kernel : state of source env b (x, u, timestep, table, clock, step_ctr) -> planning envs b K .. b K + K - 1;
//                            their episode accumulators and done zeroed; return R_c = 0, alive_c = 1.  One thread per c.
//   glg_plan_sample_kernel : candidate c, step t: a = (float) clamp(mean + std z, -1, 1) in fp64, z from glg_plan_normal2 (draw
//                            block 66); candidate k = 0 takes z = 0, i.e. the (clipped) mean.  Written [H][B K][6], so step t is
//                            one contiguous actions array for glg_step.  One thread per c, looping over t (coalesced stores).
//   glg_plan_accum_kernel  : after step t: R_c += d_t reward_c while alive_c, then alive_c = 0 once done_c.  A masked step adds
//                            nothing, even a non-finite reward.  One thread per c.
//   glg_plan_update_kernel : one CTA per source env: rank the K returns (descending, ties to the lower k, non-finite last) by
//                            counting, mark the E elites, list them in ascending k (warp ballots), then per (t, component) the
//                            elites' mean and population standard deviation, summed in fp64 in ascending k, stored as float.
//                            No atomics: the result does not depend on scheduling.
//   glg_plan_shift_kernel  : mean[t] <- mean[t + 1], mean[H - 1] <- 0, std <- init_std.  One thread per (b, component).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "glg_kernels.cuh"
#include "glg_philox.h"

constexpr int GLG_PLAN_NT = 256;    // elementwise kernels and the update CTA
constexpr int GLG_PLAN_MAXK = 4096;  // candidates per env: the update kernel's shared-memory arrays

struct GlgPlanFanArgs {
    int B, K;
    // source handle (read only), SoA [field][B]
    const double *x, *u, *time;
    const int *timestep, *table;
    const unsigned int *step_ctr;
    // planning handle, SoA [field][B K]
    double *px, *pu, *ptime, *pep_return, *pep_info;
    int *ptimestep, *ptable, *pep_len;
    unsigned int *pstep_ctr;
    unsigned char *pdone;
    double *ret;            // [B K]
    unsigned char *alive;   // [B K]
};

__global__ void __launch_bounds__(GLG_PLAN_NT) glg_plan_fanout_kernel(const GlgPlanFanArgs A) {
    const int c = blockIdx.x * GLG_PLAN_NT + threadIdx.x;
    const int BK = A.B * A.K;
    if (c >= BK) return;
    const int b = c / A.K;
    const size_t sB = (size_t)A.B, sP = (size_t)BK;
#pragma unroll 4
    for (int i = 0; i < GLG_NX; ++i) A.px[i * sP + c] = __ldg(A.x + i * sB + b);
#pragma unroll
    for (int i = 0; i < GLG_NU; ++i) A.pu[i * sP + c] = __ldg(A.u + i * sB + b);
#pragma unroll
    for (int i = 0; i < 2; ++i) A.ptime[i * sP + c] = __ldg(A.time + i * sB + b);
    A.ptimestep[c] = __ldg(A.timestep + b);
    A.ptable[c] = __ldg(A.table + b);
    A.pstep_ctr[c] = __ldg(A.step_ctr + b);
    A.pep_return[c] = 0.0;
    A.pep_len[c] = 0;
#pragma unroll
    for (int j = 0; j < GLG_NINFO; ++j) A.pep_info[j * sP + c] = 0.0;
    A.pdone[c] = 0;
    A.ret[c] = 0.0;
    A.alive[c] = 1;
}

struct GlgPlanSampleArgs {
    int B, K, H;
    uint32_t it, call;  // CEM iteration; earlier glg_plan_run calls (host-checked: I H 3 < 2^32)
    unsigned long long seed;
    const float *mean, *std;  // [H][B][6]
    float *cand;              // [H][B K][6]
};

__global__ void __launch_bounds__(GLG_PLAN_NT) glg_plan_sample_kernel(const GlgPlanSampleArgs S) {
    const int c = blockIdx.x * GLG_PLAN_NT + threadIdx.x;
    const int BK = S.B * S.K;
    if (c >= BK) return;
    const int b = c / S.K, k = c - b * S.K;
    for (int t = 0; t < S.H; ++t) {
        const size_t mo = ((size_t)t * S.B + b) * GLG_NU, co = ((size_t)t * BK + c) * GLG_NU;
#pragma unroll
        for (int p = 0; p < 3; ++p) {
            double z0 = 0.0, z1 = 0.0;
            if (k != 0) glg_plan_normal2(S.seed, S.call, ((uint32_t)S.it * S.H + t) * 3u + p, (uint32_t)c, &z0, &z1);
            const int j = 2 * p;  // explicit rounding: mean + std z is a multiply and an add, not one fused DFMA
            S.cand[co + j] = (float)fmin(fmax(__dadd_rn((double)S.mean[mo + j], __dmul_rn((double)S.std[mo + j], z0)), -1.0), 1.0);
            S.cand[co + j + 1] =
                (float)fmin(fmax(__dadd_rn((double)S.mean[mo + j + 1], __dmul_rn((double)S.std[mo + j + 1], z1)), -1.0), 1.0);
        }
    }
}

__global__ void __launch_bounds__(GLG_PLAN_NT) glg_plan_accum_kernel(int BK, double d, const double *reward, const unsigned char *done,
                                                                    double *ret, unsigned char *alive) {
    const int c = blockIdx.x * GLG_PLAN_NT + threadIdx.x;
    if (c >= BK || !alive[c]) return;
    ret[c] = __dadd_rn(ret[c], __dmul_rn(d, reward[c]));  // unfused, so a host sum of the same rewards is bit-equal
    if (done[c]) alive[c] = 0;
}

struct GlgPlanUpdateArgs {
    int B, K, E, H;
    const double *ret;   // [B K]
    const float *cand;   // [H][B K][6]
    float *mean, *std;   // [H][B][6]
    float *actions;      // [B][6] <- new mean[0], or NULL
};

// order key of a return: non-finite ranks last
__device__ __forceinline__ double glg_plan_key(double r) { return isfinite(r) ? r : -INFINITY; }

__global__ void __launch_bounds__(GLG_PLAN_NT) glg_plan_update_kernel(const GlgPlanUpdateArgs U) {
    __shared__ double key[GLG_PLAN_MAXK];
    __shared__ unsigned char elite[GLG_PLAN_MAXK];
    __shared__ unsigned short list[GLG_PLAN_MAXK];  // 44 KB in all, under the 48 KB of static shared memory
    const int b = blockIdx.x, K = U.K, BK = U.B * U.K;
    for (int k = threadIdx.x; k < K; k += GLG_PLAN_NT) key[k] = glg_plan_key(U.ret[(size_t)b * K + k]);
    __syncthreads();
    // rank of k = candidates ahead of it: a strict total order, so ranks 0 .. E - 1 name exactly E candidates
    for (int k = threadIdx.x; k < K; k += GLG_PLAN_NT) {
        const double v = key[k];
        int rank = 0;
        for (int j = 0; j < K; ++j) {
            const double w = key[j];
            rank += (w > v) || (w == v && j < k);
        }
        elite[k] = rank < U.E;
    }
    __syncthreads();
    if (threadIdx.x < 32) {  // elites in ascending k
        const int lane = threadIdx.x;
        int n = 0;
        for (int base = 0; base < K; base += 32) {
            const bool f = base + lane < K && elite[base + lane];
            const unsigned m = __ballot_sync(0xffffffffu, f);
            if (f) list[n + __popc(m & ((1u << lane) - 1u))] = (unsigned short)(base + lane);
            n += __popc(m);
        }
    }
    __syncthreads();
    const double ne = (double)U.E;
    for (int o = threadIdx.x; o < U.H * GLG_NU; o += GLG_PLAN_NT) {
        const int t = o / GLG_NU, j = o - t * GLG_NU;
        const float *col = U.cand + (size_t)t * BK * GLG_NU + (size_t)b * K * GLG_NU + j;
        double s = 0.0;
        for (int e = 0; e < U.E; ++e) s += (double)col[(size_t)list[e] * GLG_NU];
        const double m = s / ne;
        double q = 0.0;
        for (int e = 0; e < U.E; ++e) {
            const double dv = (double)col[(size_t)list[e] * GLG_NU] - m;
            q += dv * dv;
        }
        const size_t mo = ((size_t)t * U.B + b) * GLG_NU + j;
        const float mf = (float)m;
        U.mean[mo] = mf;
        U.std[mo] = (float)sqrt(q / ne);
        if (U.actions && t == 0) U.actions[(size_t)b * GLG_NU + j] = mf;
    }
}

__global__ void __launch_bounds__(GLG_PLAN_NT) glg_plan_shift_kernel(int B, int H, float init_std, float *mean, float *std) {
    const int i = blockIdx.x * GLG_PLAN_NT + threadIdx.x;  // (b, component) column
    const size_t n = (size_t)B * GLG_NU;
    if (i >= (int)n) return;
    for (int t = 0; t + 1 < H; ++t) {
        mean[t * n + i] = mean[(t + 1) * n + i];
        std[t * n + i] = init_std;
    }
    mean[(H - 1) * n + i] = 0.0f;
    std[(H - 1) * n + i] = init_std;
}
