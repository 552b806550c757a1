// glg_capi.cu -- C-ABI (include/glgym.h) over the sm_100a kernels.  Host side: handle, device buffers, launches.
// No CPU fallback anywhere: every entry point either launches CUDA work or fails with GLG_ERR_CUDA.
#include "../../include/glgym.h"

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <memory>
#include <new>
#include <string>
#include <thread>
#include <vector>

#undef GLG_NX
#undef GLG_NU
#undef GLG_ND
#undef GLG_NP
#undef GLG_NINFO
#undef GLG_NSTATS
#include "glg_kernels.cuh"
#include "glg_roles.cuh"
#include "glg_rollout.cuh"
#include "glg_replay.cuh"
#include "glg_plan.cuh"


static thread_local std::string g_error = "";  // glg_last_error(NULL): the last failure of an entry point without a handle

// The CUDA allocations of one object: device memory (zero-filled) and page-locked host memory, freed together by the
// destructor, which runs with the object's device current.  Nothing else in this file frees CUDA memory.
class CudaMem {
  public:
    CudaMem() = default;
    CudaMem(const CudaMem &) = delete;
    CudaMem &operator=(const CudaMem &) = delete;
    ~CudaMem() {
        for (const Block &b : blocks_) b.host ? cudaFreeHost(b.p) : cudaFree(b.p);
    }
    template <typename T>
    cudaError_t dev(T **p, size_t n) {
        cudaError_t e = cudaMalloc((void **)p, n * sizeof(T));
        if (e != cudaSuccess) return e;
        blocks_.push_back({*p, n * sizeof(T), false});
        return cudaMemset(*p, 0, n * sizeof(T));
    }
    template <typename T>
    cudaError_t host(T **p, size_t n) {
        cudaError_t e = cudaMallocHost((void **)p, n * sizeof(T));
        if (e == cudaSuccess) blocks_.push_back({*p, n * sizeof(T), true});
        return e;
    }
    size_t bytes() const {
        size_t n = 0;
        for (const Block &b : blocks_) n += b.bytes;
        return n;
    }
    void swap(CudaMem &o) { blocks_.swap(o.blocks_); }

  private:
    struct Block {
        void *p;
        size_t bytes;
        bool host;
    };
    std::vector<Block> blocks_;
};

struct glg_handle {
    ~glg_handle();
    glg_config cfg;  // as created; what the setters change since lives in `a`
    // The env's launch state, kept current by the setters: sizes, config scalars, observation layout, ctrl, the bank and the
    // state / output buffers.  Its per-call fields (actions, controls, noise, raw_control) stay 0 here; each launch sets them
    // on a copy.
    GlgStepArgs a = {};
    int n_head = 0;  // obs_dim - 5 Np with a forecast block, else obs_dim: the packed row (obs_head) the host paths copy
    int sms = 148;
    bool have_params = false, general = false, is_reset = false;
    GlgUniform uni;
    CudaMem mem;                   // the state / output buffers `a` points into, `actions` and the pinned host staging
    CudaMem bank, reset_list;      // what a.weather, a.start_day (glg_set_weather) and a.reset_tables point into
    std::vector<float> fc_bank;    // [n_tables][rows][5] float32: the weather columns a forecast block shows, as the kernels cast them
    unsigned long long weather_gen = 0;  // bumped by every glg_set_weather: replay buffers hold keys into the bank
    float *actions = nullptr;      // [B][6] device: the host step paths' actions
    // pinned host staging for glg_step_host
    float *h_actions = nullptr, *h_obs = nullptr;
    double *h_reward = nullptr;
    unsigned char *h_done = nullptr;
    // host side of glg_step_host's overlapped observation path (see there)
    float *h_head = nullptr;     // pinned [B][n_head]: staging of the packed columns for a pageable destination
    unsigned char *h_res = nullptr;  // pinned [2 buffers][17 B]: reward | timestep | table | done of every env after a glg_step_host
    int kt_cur = 0;              // buffer the last glg_step_host filled
    bool kt_valid = false;       // h_res[kt_cur] holds this handle's last host step (a prediction source, verified after every step)
    std::vector<int> fc_pred;    // [2][B]: (table, first weather row) the forecast blocks in the caller's buffer were filled from
    int host_obs_mode = 0;       // glg_set_host_obs_mode
    cudaStream_t own_stream = nullptr;
    cudaEvent_t order_event = nullptr;  // glg_host_path_after
    long long launches = 0;
    void *nccl_comm = nullptr;  // ncclComm_t (glg_nccl_init)
    std::string err;
};
// rule-based controller settings: configs/agents/rule_based.yml
static const double kDefaultCtrl[GLG_NCTRL] = {0, 18, -1, 366, 400, 10, 19.5, 16.5, 0, 5, 800, 4, 85, 2, 5, 1, -1, 5, 10, -1, 4, -2,
                                               2, 2, 100, 85, -1, -100, 1};

#define GLG_CUDA(h, call)                                                                            \
    do {                                                                                             \
        cudaError_t e__ = (call);                                                                    \
        if (e__ != cudaSuccess) {                                                                    \
            char buf__[512];                                                                         \
            snprintf(buf__, sizeof buf__, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
            (h)->err = buf__;                                                                        \
            return GLG_ERR_CUDA;                                                                     \
        }                                                                                            \
    } while (0)

static int fail(glg_handle *h, int code, const char *msg) {
    h->err = msg;
    return code;
}

extern "C" void glg_default_config(glg_config *c) {
    memset(c, 0, sizeof *c);
    c->num_envs = 1;
    c->device = 0;
    c->dt = 900.0;
    c->n_sub = 600;
    c->N = 5760;
    c->Np = 48;
    c->precision = 0;
    c->auto_reset = 1;
    for (int i = 0; i < 6; ++i) {
        c->u_min[i] = 0.0;
        c->u_max[i] = 1.0;
    }
    c->delta_u_max = (double)0.1f;
    c->con_low[0] = 300.; c->con_low[1] = 15.; c->con_low[2] = 50.;
    c->con_high[0] = 1600.; c->con_high[1] = 34.; c->con_high[2] = 85.;
    c->elec_price = 0.3; c->heating_price = 0.09; c->co2_price = 0.3; c->fruit_price = 1.6; c->dmfm = 0.065;
    c->fixed_costs = (15. + 0.015 + 0.07 * 116 + 2.) / 365 / (86400 / 900);
    c->uncertainty_scale = 0.0;
    c->seed = 0;
    c->env_id_offset = 0;
    c->role_warps = 0;
    c->role_lanes = 0;
    for (int i = 0; i < 8; ++i) c->obs_modules[i] = 0;  // empty = the default stack of TomatoEnv.yml
}

extern "C" const char *glg_last_error(const glg_handle *h) { return h ? h->err.c_str() : g_error.c_str(); }

static size_t res_block_bytes(size_t B) { return 17 * B; }  // double reward[B] | int32 timestep[B] | int32 table[B] | uint8 done[B]

// ---- episode-statistics all-reduce over NCCL, bound at run time ---------------------------------------------
struct NcclId {  // ncclUniqueId: 128 opaque bytes, passed by value
    char internal[128];
};
namespace {
struct NcclApi {
    void *lib = nullptr;
    int (*GetUniqueId)(void *) = nullptr;
    int (*CommInitRank)(void **, int, NcclId, int) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    int (*CommDestroy)(void *) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
};
}  // namespace
static NcclApi *nccl_api(std::string *err) {
    static NcclApi api;
    if (api.lib) return &api;
    const char *names[] = {"libnccl.so.2", "libnccl.so"};
    void *lib = nullptr;
    for (const char *n : names) {
        lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (lib) break;
    }
    if (!lib) {
        *err = std::string("NCCL not found (dlopen libnccl.so.2): ") + (dlerror() ? dlerror() : "");
        return nullptr;
    }
    api.GetUniqueId = (int (*)(void *))dlsym(lib, "ncclGetUniqueId");
    api.CommInitRank = (int (*)(void **, int, NcclId, int))dlsym(lib, "ncclCommInitRank");
    api.AllReduce = (int (*)(const void *, void *, size_t, int, int, void *, cudaStream_t))dlsym(lib, "ncclAllReduce");
    api.CommDestroy = (int (*)(void *))dlsym(lib, "ncclCommDestroy");
    api.GetErrorString = (const char *(*)(int))dlsym(lib, "ncclGetErrorString");
    if (!api.GetUniqueId || !api.CommInitRank || !api.AllReduce || !api.CommDestroy) {
        *err = "libnccl.so.2 lacks a required symbol";
        return nullptr;
    }
    api.lib = lib;
    return &api;
}

glg_handle::~glg_handle() {  // memory goes with the CudaMem members
    if (order_event) cudaEventDestroy(order_event);
    if (own_stream) cudaStreamDestroy(own_stream);
    if (nccl_comm) {
        std::string e;
        NcclApi *n = nccl_api(&e);
        if (n) n->CommDestroy(nccl_comm);
    }
}

extern "C" void glg_destroy(glg_handle *h) {
    if (!h) return;
    cudaSetDevice(h->cfg.device);
    delete h;
}

extern "C" int glg_create(const glg_config *cfg, glg_handle **out) {
    if (!cfg || !out) {
        g_error = "glg_create: null argument";
        return GLG_ERR_ARG;
    }
    *out = nullptr;
    if (cfg->num_envs < 1 || cfg->n_sub < 1 || cfg->N < 0 || cfg->Np < 0 || !(cfg->dt > 0) ||
        (cfg->precision != 0 && cfg->precision != 1) ||
        (cfg->role_warps < 0 || cfg->role_warps > 3) ||
        (cfg->integrator != 0 && cfg->integrator != 1) || (cfg->precision == 1 && cfg->role_warps == 1)) {
        g_error = (cfg->precision == 1 && cfg->role_warps == 1)
                      ? "glg_create: the fp32 throughput mode runs on kernel C only (role_warps 0, 2 or 3)"
                      : "glg_create: invalid num_envs / n_sub / N / Np / dt / precision / role_warps / integrator";
        return GLG_ERR_ARG;
    }
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0 || cfg->device < 0 || cfg->device >= ndev) {
        g_error = std::string("glg_create: no usable CUDA device (") + cudaGetErrorString(ce) + "); this library has no CPU fallback";
        return GLG_ERR_CUDA;
    }
    glg_handle *h = new (std::nothrow) glg_handle();
    if (!h) return GLG_ERR_ALLOC;
    h->cfg = *cfg;
    GlgStepArgs &a = h->a;
    a.B = cfg->num_envs; a.n_sub = cfg->n_sub; a.N = cfg->N; a.Np = cfg->Np; a.auto_reset = cfg->auto_reset;
    a.integrator = cfg->integrator;
    a.dt = cfg->dt;
    for (int i = 0; i < GLG_NU; ++i) {
        a.u_min[i] = cfg->u_min[i];
        a.u_max[i] = cfg->u_max[i];
    }
    a.delta_u_max_f32 = (float)cfg->delta_u_max;
    for (int i = 0; i < 3; ++i) {
        a.con_low[i] = cfg->con_low[i];
        a.con_high[i] = cfg->con_high[i];
    }
    a.elec_price = cfg->elec_price; a.heating_price = cfg->heating_price; a.co2_price = cfg->co2_price;
    a.fruit_price = cfg->fruit_price; a.dmfm = cfg->dmfm; a.fixed_costs = cfg->fixed_costs;
    a.uncertainty_scale = cfg->uncertainty_scale;
    a.seed = cfg->seed; a.env_id_offset = cfg->env_id_offset;
    for (int i = 0; i < GLG_NCTRL; ++i) a.ctrl[i] = kDefaultCtrl[i];
    {
        // observation row layout from the module list (tomato_env.py:77-96)
        static const int kDefault[6] = {GLG_OBS_CLIMATE, GLG_OBS_CROP, GLG_OBS_CONTROL, GLG_OBS_WEATHER, GLG_OBS_TIME, GLG_OBS_FORECAST};
        const int sizes[8] = {0, GLG_NOBS_STATE, 4, 3, 6, 5, 5, 5 * cfg->Np};
        unsigned seen = 0;
        int off = 0;
        bool ok = true;
        const bool use_default = cfg->obs_modules[0] == 0;
        a.fc_off = -1;
        for (int m = 0; m < GLG_MAXOBSMOD; ++m) {
            const int id = use_default ? (m < 6 ? kDefault[m] : 0) : cfg->obs_modules[m];
            if (id == 0) break;
            if (id < 1 || id > 7 || (seen >> id & 1u)) {
                ok = false;
                break;
            }
            seen |= 1u << id;
            a.obs_mod[a.obs_nmod] = id;
            a.obs_off[a.obs_nmod] = off;
            if (id == GLG_OBS_FORECAST) a.fc_off = off;
            off += sizes[id];
            ++a.obs_nmod;
        }
        if (!ok || off < 3) {
            g_error = "glg_create: obs_modules must list distinct module ids 1..7 with at least 3 observation entries in total";
            delete h;
            return GLG_ERR_ARG;
        }
        a.obs_dim = off;
        h->n_head = off - (a.fc_off >= 0 ? 5 * cfg->Np : 0);
    }
    // kernel B: envs per CTA.  32 (full warps) is fastest at every batch size measured: a CTA's step time grows with the
    // number of co-resident CTAs faster than under-filled warps could win back (profiles/r1_lane_sweep.txt).
    a.role_lanes = (cfg->role_lanes >= 1 && cfg->role_lanes <= 32) ? cfg->role_lanes : 32;
    {
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, cfg->device) == cudaSuccess) h->sms = prop.multiProcessorCount;
    }
    const size_t B = (size_t)a.B, D = (size_t)a.obs_dim;
    CudaMem &m = h->mem;
    unsigned char *res_block = nullptr;
    cudaError_t e = cudaSetDevice(cfg->device);
    if (e == cudaSuccess) e = m.dev(&a.x, GLG_NX * B);
    if (e == cudaSuccess) e = m.dev(&a.u, GLG_NU * B);
    if (e == cudaSuccess) e = m.dev(&a.time, 2 * B);
    if (e == cudaSuccess) e = m.dev(&a.ep_return, B);
    if (e == cudaSuccess) e = m.dev(&a.ep_info, GLG_NINFO * B);
    // reward | timestep | table | done share one allocation: glg_step_host fetches them with one device->host copy
    if (e == cudaSuccess) e = m.dev(&res_block, res_block_bytes(B));
    if (e == cudaSuccess) {
        a.reward = reinterpret_cast<double *>(res_block);
        a.timestep = reinterpret_cast<int *>(res_block + 8 * B);
        a.table = a.timestep + B;
        a.done = res_block + 16 * B;
    }
    if (e == cudaSuccess) e = m.dev(&a.ep_len, B);
    if (e == cudaSuccess) e = m.dev(&a.step_ctr, B);
    if (e == cudaSuccess) e = m.dev(&a.obs, D * B);
    if (e == cudaSuccess) e = m.dev(&a.term_obs, D * B);
    if (e == cudaSuccess) e = m.dev(&a.obs_head, (size_t)h->n_head * B);
    if (e == cudaSuccess) e = m.dev(&h->actions, GLG_NU * B);
    if (e == cudaSuccess) e = m.dev(&a.info, GLG_NINFO * B);
    if (e == cudaSuccess) e = m.dev(&a.stats, (size_t)GLG_NSTATS);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        g_error = std::string("glg_create: ") + cudaGetErrorString(e);
        glg_destroy(h);
        return GLG_ERR_CUDA;
    }
    *out = h;
    return GLG_OK;
}

extern "C" int glg_set_seed(glg_handle *h, uint64_t seed) {
    if (!h) return GLG_ERR_ARG;
    h->a.seed = seed;
    return GLG_OK;
}

extern "C" int glg_set_params(glg_handle *h, const double *p_host) {
    if (!h || !p_host) return GLG_ERR_ARG;
    for (int i = 0; i < GLG_NP; ++i) h->uni.P[i] = p_host[i];
    glg_make_k(p_host, h->uni.K);
    glg_make_c(p_host, h->uni.C);
    for (int i = 0; i < K_COUNT; ++i) h->uni.Kf[i] = (float)h->uni.K[i];
    for (int i = 0; i < C_COUNT; ++i) h->uni.Cf[i] = (float)h->uni.C[i];
    h->general = !glg_params_nominal_structure(p_host);
    h->have_params = true;
    return GLG_OK;
}

extern "C" int glg_set_weather(glg_handle *h, const double *tables_host, int32_t n_tables, int32_t rows,
                               const double *start_day_host) {
    if (!h || !tables_host || n_tables < 1) return GLG_ERR_ARG;
    if (rows < h->a.N + h->a.Np + 1) return fail(h, GLG_ERR_ARG, "glg_set_weather: rows < N + Np + 1");
    GLG_CUDA(h, cudaSetDevice(h->cfg.device));
    // The new bank and its identity reset-table list are complete before the old ones are released (when `bank` and
    // `reset_list` go out of scope after the swap): a failure leaves the handle as it was.
    CudaMem bank, reset_list;
    double *weather = nullptr, *start_day = nullptr;
    int *reset_tables = nullptr;
    const size_t n = (size_t)n_tables * rows * GLG_ND;
    GLG_CUDA(h, bank.dev(&weather, n));
    GLG_CUDA(h, cudaMemcpy(weather, tables_host, n * sizeof(double), cudaMemcpyHostToDevice));
    std::vector<double> sd(n_tables, 0.0);
    if (start_day_host) sd.assign(start_day_host, start_day_host + n_tables);
    GLG_CUDA(h, bank.dev(&start_day, n_tables));
    GLG_CUDA(h, cudaMemcpy(start_day, sd.data(), n_tables * sizeof(double), cudaMemcpyHostToDevice));
    std::vector<int> ids(n_tables);
    for (int i = 0; i < n_tables; ++i) ids[i] = i;
    GLG_CUDA(h, reset_list.dev(&reset_tables, n_tables));
    GLG_CUDA(h, cudaMemcpy(reset_tables, ids.data(), n_tables * sizeof(int), cudaMemcpyHostToDevice));
    // host copy of what glg_write_forecast shows of the bank (columns 0..4, double -> float), for glg_step_host
    std::vector<float> fc_bank((size_t)n_tables * rows * 5);
    for (size_t r = 0; r < (size_t)n_tables * rows; ++r)
        for (int c = 0; c < 5; ++c) fc_bank[r * 5 + c] = (float)tables_host[r * GLG_ND + c];
    h->bank.swap(bank);
    h->reset_list.swap(reset_list);
    h->fc_bank.swap(fc_bank);
    h->a.weather = weather; h->a.start_day = start_day; h->a.reset_tables = reset_tables;
    h->a.n_tables = n_tables; h->a.rows = rows; h->a.n_reset_tables = n_tables;
    ++h->weather_gen;
    h->kt_valid = false;
    return GLG_OK;
}

extern "C" int glg_set_reset_tables(glg_handle *h, const int32_t *ids, int32_t n) {
    if (!h || !ids || n < 1) return GLG_ERR_ARG;
    if (!h->a.weather) return fail(h, GLG_ERR_STATE, "glg_set_reset_tables: set the weather bank first");
    for (int i = 0; i < n; ++i)
        if (ids[i] < 0 || ids[i] >= h->a.n_tables) return fail(h, GLG_ERR_ARG, "glg_set_reset_tables: id out of range");
    GLG_CUDA(h, cudaSetDevice(h->cfg.device));
    CudaMem list;  // complete before the old list is released, as in glg_set_weather
    int *reset_tables = nullptr;
    GLG_CUDA(h, list.dev(&reset_tables, n));
    GLG_CUDA(h, cudaMemcpy(reset_tables, ids, n * sizeof(int), cudaMemcpyHostToDevice));
    h->reset_list.swap(list);
    h->a.reset_tables = reset_tables;
    h->a.n_reset_tables = n;
    return GLG_OK;
}

static int check_ready(glg_handle *h) {
    if (!h) return GLG_ERR_ARG;
    if (!h->have_params) return fail(h, GLG_ERR_STATE, "parameters not set (glg_set_params)");
    if (!h->a.weather) return fail(h, GLG_ERR_STATE, "weather bank not set (glg_set_weather)");
    return GLG_OK;
}

extern "C" int glg_reset(glg_handle *h, const uint8_t *mask_dev, const int32_t *table_ids_dev, void *stream) {
    int rc = check_ready(h);
    if (rc) return rc;
    GLG_CUDA(h, cudaSetDevice(h->cfg.device));
    const int NT = 128;
    glg_reset_kernel<NT><<<(h->a.B + NT - 1) / NT, NT, 0, (cudaStream_t)stream>>>(h->a, mask_dev, table_ids_dev);
    h->launches += 1;
    GLG_CUDA(h, cudaGetLastError());
    h->is_reset = true;
    h->kt_valid = false;
    return GLG_OK;
}

// Opts kernel F into `smem` bytes of dynamic shared memory on `device` when a launch needs more than F has been allowed there
// so far (the attribute is per kernel and per context).
template <auto F>
static cudaError_t opt_in_smem(int device, size_t smem) {
    static size_t attr_smem_dev[64] = {};  // largest size opted into so far, per device
    size_t &attr_smem = attr_smem_dev[device & 63];
    if (smem > attr_smem) {
        cudaError_t e = cudaFuncSetAttribute(F, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        attr_smem = smem;
    }
    return cudaSuccess;
}

template <bool GENERAL, bool NOISY>
static cudaError_t launch_step(glg_handle *h, const GlgStepArgs &a, cudaStream_t s) {
    constexpr int NT = 64;
    const size_t smem = GlgStepSmem<NT, NOISY>::bytes(a.Np);
    cudaError_t e = opt_in_smem<glg_step_kernel<GENERAL, NOISY, NT>>(h->cfg.device, smem);
    if (e != cudaSuccess) return e;
    glg_step_kernel<GENERAL, NOISY, NT><<<(a.B + NT - 1) / NT, NT, smem, s>>>(h->uni, a);
    return cudaGetLastError();
}

// precision 0: fp64 parity mode ; 1: flux units in fp32, RK4 state / stage sums / epilogue in fp64
template <bool FUSED, bool GENERAL, bool NOISY>
static cudaError_t launch_step_units(glg_handle *h, const GlgStepArgs &a, cudaStream_t s) {
    const auto launch = [&](auto t) {
        using T = decltype(t);
        const size_t smem = GlgRoleSmem<T, GlgLayout<FUSED>::NG, GENERAL, NOISY>::bytes(a.Np);
        cudaError_t e = opt_in_smem<glg_step_units_kernel<T, GENERAL, NOISY, FUSED>>(h->cfg.device, smem);
        if (e != cudaSuccess) return e;
        glg_step_units_kernel<T, GENERAL, NOISY, FUSED><<<(a.B + a.role_lanes - 1) / a.role_lanes, GlgLayout<FUSED>::NT, smem, s>>>(h->uni, a);
        return cudaGetLastError();
    };
    return h->cfg.precision == 1 ? launch(0.0f) : launch(0.0);
}

// Kernel variant: 1 = kernel A (one thread per env), 2 = kernel C latency layout (4 owner + 12 group warps per 32 envs, one CTA
// per SM: the step time of a batch that leaves SMs under-filled is the latency of one CTA), 3 = kernel C throughput layout
// (4 fused warps per 32 envs, 4 CTAs per SM).  Auto-pick: measured with tools/layout_sweep.py the latency layout wins up to two
// waves of CTAs (B = 9472 on 148 SMs: 1.735 vs 1.814 ms), the throughput layout beyond (B = 12 288: 2.60 vs 2.18 ms).
static int pick_role_warps(const glg_handle *h) {
    if (h->cfg.role_warps != 0) return h->cfg.role_warps;
    return h->a.B <= 2 * h->sms * GLG_ROLE_LANES ? 2 : 3;
}
typedef cudaError_t (*StepLauncher)(glg_handle *, const GlgStepArgs &, cudaStream_t);
static const StepLauncher kStepLaunchers[3][2][2] = {  // [kernel variant - 1][general][noisy]
    {{launch_step<false, false>, launch_step<false, true>}, {launch_step<true, false>, launch_step<true, true>}},
    {{launch_step_units<false, false, false>, launch_step_units<false, false, true>},
     {launch_step_units<false, true, false>, launch_step_units<false, true, true>}},
    {{launch_step_units<true, false, false>, launch_step_units<true, false, true>},
     {launch_step_units<true, true, false>, launch_step_units<true, true, true>}}};

static int step_common(glg_handle *h, const float *actions_dev, const double *controls_dev, const double *noise_dev,
                       void *stream, bool rule_based = false) {
    int rc = check_ready(h);
    if (rc) return rc;
    if (!h->is_reset) return fail(h, GLG_ERR_STATE, "step before reset");
    GLG_CUDA(h, cudaSetDevice(h->cfg.device));
    h->kt_valid = false;
    GlgStepArgs a = h->a;
    a.actions = actions_dev;
    a.controls = controls_dev;
    a.raw_control = rule_based ? 2 : (controls_dev ? 1 : 0);
    a.noise = noise_dev;
    const bool noisy = (a.uncertainty_scale != 0.0) || (noise_dev != nullptr);
    const cudaError_t e = kStepLaunchers[pick_role_warps(h) - 1][h->general][noisy](h, a, (cudaStream_t)stream);
    h->launches += 1;
    GLG_CUDA(h, e);
    return GLG_OK;
}

extern "C" int glg_step(glg_handle *h, const float *actions_dev, const double *noise_dev, void *stream) {
    if (!h || !actions_dev) return GLG_ERR_ARG;
    return step_common(h, actions_dev, nullptr, noise_dev, stream);
}

extern "C" int glg_step_raw_control(glg_handle *h, const double *controls_dev, const double *noise_dev, void *stream) {
    if (!h || !controls_dev) return GLG_ERR_ARG;
    return step_common(h, nullptr, controls_dev, noise_dev, stream);
}

extern "C" int glg_set_rule_controller(glg_handle *h, const double *settings29) {
    if (!h) return GLG_ERR_ARG;
    for (int i = 0; i < GLG_NCTRL; ++i) h->a.ctrl[i] = settings29 ? settings29[i] : kDefaultCtrl[i];
    return GLG_OK;
}

extern "C" int glg_step_rule_based(glg_handle *h, const double *noise_dev, void *stream) {
    if (!h) return GLG_ERR_ARG;
    return step_common(h, nullptr, nullptr, noise_dev, stream, true);
}

// known-answer entry for the controller alone: one thread per point
__global__ void glg_rule_control_kernel(GlgStepArgs A, const double *x, const double *d, const double *hod, const double *doy,
                                        double *u, int n) {
    glg_exp_tbl_fill();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double xl[GLG_NX], dl[GLG_ND], ul[GLG_NU];
    for (int j = 0; j < GLG_NX; ++j) xl[j] = x[(size_t)i * GLG_NX + j];
    for (int j = 0; j < GLG_ND; ++j) dl[j] = d[(size_t)i * GLG_ND + j];
    glg_rule_control(A.ctrl, xl, dl, hod[i], doy[i], ul);
    for (int j = 0; j < GLG_NU; ++j) u[(size_t)i * GLG_NU + j] = ul[j];
}
extern "C" int glg_rule_control_batch(const double *settings29, const double *x_dev, const double *d_dev, const double *hod_dev,
                                      const double *doy_dev, double *u_dev, int32_t n, int32_t device, void *stream) {
    if (!x_dev || !d_dev || !hod_dev || !doy_dev || !u_dev || n < 1) {
        g_error = "glg_rule_control_batch: invalid argument";
        return GLG_ERR_ARG;
    }
    GlgStepArgs a;
    memset(&a, 0, sizeof a);
    for (int i = 0; i < GLG_NCTRL; ++i) a.ctrl[i] = settings29 ? settings29[i] : kDefaultCtrl[i];
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) {
        glg_rule_control_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(a, x_dev, d_dev, hod_dev, doy_dev, u_dev, n);
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) {
        g_error = std::string("glg_rule_control_batch: ") + cudaGetErrorString(e);
        return GLG_ERR_CUDA;
    }
    return GLG_OK;
}

static bool is_pinned(const void *p) {
    // small per-thread cache: the callers pass the same few buffers every step, and a stale answer is harmless (a pageable
    // buffer taken for page-locked makes cudaMemcpyAsync stage it itself; the reverse costs one staging copy)
    static thread_local struct { const void *p; bool pinned; } cache[8] = {};
    static thread_local int next = 0;
    for (auto &c : cache)
        if (c.p == p) return c.pinned;
    cudaPointerAttributes at;
    bool pinned = false;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) cudaGetLastError();
    else pinned = at.type == cudaMemoryTypeHost;
    cache[next] = {p, pinned};
    next = (next + 1) % 8;
    return pinned;
}

// Rows [lo, hi) of a per-env host loop on up to 8 threads; small batches run inline (a thread costs ~20 us to start).  A chunk
// whose thread cannot be started (no exception may cross the C boundary) is done by the caller.
template <class F>
static void host_rows(size_t n_rows, size_t bytes_per_row, const F &f) {
    const size_t total = n_rows * bytes_per_row;
    unsigned hw = std::thread::hardware_concurrency();
    size_t nt = total / ((size_t)6 << 20);  // one thread per 6 MB moved
    const size_t cap = hw >= 4 ? (hw / 2 < 8 ? hw / 2 : 8) : 1;
    nt = nt > cap ? cap : nt;
    if (nt <= 1) {
        f((size_t)0, n_rows);
        return;
    }
    std::vector<std::thread> th;
    const size_t chunk = (n_rows + nt - 1) / nt;
    for (size_t t = 1; t < nt; ++t) {
        const size_t lo = t * chunk, hi = lo + chunk < n_rows ? lo + chunk : n_rows;
        if (lo >= hi) continue;
        try {
            th.emplace_back([&f, lo, hi] { f(lo, hi); });
        } catch (...) {
            f(lo, hi);
        }
    }
    f((size_t)0, chunk < n_rows ? chunk : n_rows);
    for (auto &t : th) t.join();
}

extern "C" int glg_host_path_after(glg_handle *h, void *stream) {
    if (!h) return GLG_ERR_ARG;
    GLG_CUDA(h, cudaSetDevice(h->cfg.device));
    if (!h->order_event) GLG_CUDA(h, cudaEventCreateWithFlags(&h->order_event, cudaEventDisableTiming));
    GLG_CUDA(h, cudaEventRecord(h->order_event, (cudaStream_t)stream));
    GLG_CUDA(h, cudaStreamWaitEvent(h->own_stream, h->order_event, 0));
    return GLG_OK;
}

extern "C" int glg_set_host_obs_mode(glg_handle *h, int32_t mode) {
    if (!h || (mode != 0 && mode != 1)) return GLG_ERR_ARG;
    h->host_obs_mode = mode;
    return GLG_OK;
}

// Every host step path: the actions into the handle's device buffer, then the step, both on the handle's own stream.  The
// caller's actions may be pageable (the runtime stages them); page-locked ones make the copy asynchronous.
static int step_from_host(glg_handle *h, const float *actions_host) {
    GLG_CUDA(h, cudaMemcpyAsync(h->actions, actions_host, GLG_NU * (size_t)h->a.B * sizeof(float), cudaMemcpyHostToDevice, h->own_stream));
    return step_common(h, h->actions, nullptr, nullptr, h->own_stream);
}

// Overlapped observation path (host_obs_mode 0, the default, for stacks with a WeatherForecastObservations block): 5 Np of the
// row's floats (240 of 263 in the default stack) are weather rows kw+1 .. kw+Np of the env's table, kw = min(timestep before the
// step, rows - Np - 1) -- known before the kernel runs.  So only the rest of the row (glg_write_obs_row's packed copy, obs_head)
// crosses PCIe, and WHILE THE KERNEL RUNS the host writes the forecast blocks into the caller's buffer from its float32 copy of
// the bank, predicted from the (timestep, table) of the previous host step.  After the synchronise the packed columns are
// scattered into the rows and every prediction is checked against the (timestep, table) the step left behind: rows that reset
// in place (auto-reset draws a new table on the device), and all rows when something other than glg_step_host moved the envs in
// between (reset, tensor steps, set_state), are filled again from the verified values.  The result is the same [B][obs_dim]
// array the full device->host copy (mode 1) delivers, bit for bit (tests/test_gpu_features.py).
static int step_host_overlapped(glg_handle *h, const float *a_src, float *obs_host, double *reward_host, uint8_t *done_host, bool o_pin) {
    const size_t B = (size_t)h->a.B;
    const int Np = h->a.Np, nf = 5 * Np, D = h->a.obs_dim, n_head = h->n_head, fc = h->a.fc_off, rows = h->a.rows;
    if (!h->h_res) {
        GLG_CUDA(h, h->mem.host(&h->h_res, 2 * res_block_bytes(B)));
        h->fc_pred.assign(2 * B, -1);
        h->kt_valid = false;
    }
    if (!o_pin && !h->h_head) GLG_CUDA(h, h->mem.host(&h->h_head, (size_t)n_head * B));
    cudaStream_t s = h->own_stream;
    // result block of the previous host step (prediction source) / of this one
    const unsigned char *res_cur = h->h_res + (size_t)h->kt_cur * res_block_bytes(B);
    unsigned char *res_nxt = h->h_res + (size_t)(h->kt_cur ^ 1) * res_block_bytes(B);
    const int *cur = reinterpret_cast<const int *>(res_cur + 8 * B);
    const int *nxt = reinterpret_cast<const int *>(res_nxt + 8 * B);
    const bool valid = h->kt_valid;  // every entry that moves the envs clears it (step_common included: set again below)
    int rc = step_from_host(h, a_src);
    if (rc) return rc;
    const float *obs_head = h->a.obs_head;
    if (o_pin) {
        // page-locked destination: the copy engine puts the packed columns straight into the rows (strided 2-D copy)
        if (fc > 0)
            GLG_CUDA(h, cudaMemcpy2DAsync(obs_host, (size_t)D * sizeof(float), obs_head, (size_t)n_head * sizeof(float), (size_t)fc * sizeof(float), B,
                                          cudaMemcpyDeviceToHost, s));
        if (n_head > fc)
            GLG_CUDA(h, cudaMemcpy2DAsync(obs_host + fc + nf, (size_t)D * sizeof(float), obs_head + fc, (size_t)n_head * sizeof(float),
                                          (size_t)(n_head - fc) * sizeof(float), B, cudaMemcpyDeviceToHost, s));
    } else {
        GLG_CUDA(h, cudaMemcpyAsync(h->h_head, obs_head, (size_t)n_head * B * sizeof(float), cudaMemcpyDeviceToHost, s));
    }
    // reward | timestep | table | done: one block that starts at a.reward
    GLG_CUDA(h, cudaMemcpyAsync(res_nxt, h->a.reward, res_block_bytes(B), cudaMemcpyDeviceToHost, s));
    // ---- while the GPU works: forecast blocks from the predicted (table, row)
    const float *bank = h->fc_bank.data();
    int *pred_t = h->fc_pred.data(), *pred_r = pred_t + B;
    const int n_tables = h->a.n_tables, kmax = rows - Np - 1;
    host_rows(B, (size_t)nf * sizeof(float), [=](size_t lo, size_t hi) {
        for (size_t i = lo; i < hi; ++i) {
            const int k = valid ? cur[i] : -1, t = valid ? cur[B + i] : -1;
            if (k < 0 || t < 0 || t >= n_tables) {
                pred_t[i] = -1;
                continue;
            }
            const int r0 = (k < kmax ? k : kmax) + 1;
            memcpy(obs_host + i * D + fc, bank + ((size_t)t * rows + r0) * 5, (size_t)nf * sizeof(float));
            pred_t[i] = t;
            pred_r[i] = r0;
        }
    });
    GLG_CUDA(h, cudaStreamSynchronize(s));
    // ---- verify every prediction against what the step left behind (and, for a pageable destination, scatter the packed columns)
    const float *head = h->h_head;
    host_rows(B, o_pin ? 16 : (size_t)D * sizeof(float) / 4, [=](size_t lo, size_t hi) {
        for (size_t i = lo; i < hi; ++i) {
            float *row = obs_host + i * D;
            if (!o_pin) {
                const float *hd = head + i * n_head;
                if (fc > 0) memcpy(row, hd, (size_t)fc * sizeof(float));
                if (n_head > fc) memcpy(row + fc + nf, hd + fc, (size_t)(n_head - fc) * sizeof(float));
            }
            // timestep after the step: 0 = reset in place (row 1 of the new table), else the pre-step timestep + 1
            const int kp = nxt[i], t = nxt[B + i];
            const int r0 = kp <= 0 ? 1 : ((kp - 1 < kmax ? kp - 1 : kmax) + 1);
            if (t != pred_t[i] || r0 != pred_r[i])
                memcpy(row + fc, bank + ((size_t)t * rows + r0) * 5, (size_t)nf * sizeof(float));
        }
    });
    if (reward_host) memcpy(reward_host, res_nxt, B * sizeof(double));
    if (done_host) memcpy(done_host, res_nxt + 16 * B, B);
    h->kt_cur ^= 1;
    h->kt_valid = true;
    return GLG_OK;
}

extern "C" int glg_step_host(glg_handle *h, const float *actions_host, float *obs_host, double *reward_host,
                             uint8_t *done_host) {
    if (!h || !actions_host) return GLG_ERR_ARG;
    GLG_CUDA(h, cudaSetDevice(h->cfg.device));
    const size_t B = (size_t)h->a.B, D = (size_t)h->a.obs_dim;
    if (!h->h_actions) {
        GLG_CUDA(h, h->mem.host(&h->h_actions, GLG_NU * B));
        GLG_CUDA(h, h->mem.host(&h->h_reward, B));
        GLG_CUDA(h, h->mem.host(&h->h_done, B));
    }
    cudaStream_t s = h->own_stream;
    // caller buffers that are page-locked are used directly; pageable ones are staged through the handle's pinned buffers
    const bool a_pin = is_pinned(actions_host);
    const bool o_pin = obs_host && is_pinned(obs_host), r_pin = reward_host && is_pinned(reward_host),
               d_pin = done_host && is_pinned(done_host);
    const float *a_src = actions_host;
    if (!a_pin) {
        memcpy(h->h_actions, actions_host, GLG_NU * B * sizeof(float));
        a_src = h->h_actions;
    }
    if (obs_host && h->host_obs_mode == 0 && h->a.fc_off >= 0 && !h->fc_bank.empty()) {
        return step_host_overlapped(h, a_src, obs_host, reward_host, done_host, o_pin);
    } else {
        h->kt_valid = false;
        if (obs_host && !o_pin && !h->h_obs) GLG_CUDA(h, h->mem.host(&h->h_obs, D * B));
        int rc = step_from_host(h, a_src);
        if (rc) return rc;
        if (obs_host) GLG_CUDA(h, cudaMemcpyAsync(o_pin ? obs_host : h->h_obs, h->a.obs, D * B * sizeof(float), cudaMemcpyDeviceToHost, s));
        if (reward_host) GLG_CUDA(h, cudaMemcpyAsync(r_pin ? reward_host : h->h_reward, h->a.reward, B * sizeof(double), cudaMemcpyDeviceToHost, s));
        if (done_host) GLG_CUDA(h, cudaMemcpyAsync(d_pin ? done_host : h->h_done, h->a.done, B, cudaMemcpyDeviceToHost, s));
        GLG_CUDA(h, cudaStreamSynchronize(s));
        if (obs_host && !o_pin) memcpy(obs_host, h->h_obs, D * B * sizeof(float));
    }
    if (reward_host && !r_pin) memcpy(reward_host, h->h_reward, B * sizeof(double));
    if (done_host && !d_pin) memcpy(done_host, h->h_done, B);
    return GLG_OK;
}

extern "C" int glg_step_host_split(glg_handle *h, const float *actions_host, float *head_host, int32_t *timestep_host,
                                   int32_t *table_host, double *reward_host, uint8_t *done_host) {
    if (!h || !actions_host) return GLG_ERR_ARG;
    GLG_CUDA(h, cudaSetDevice(h->cfg.device));
    const size_t B = (size_t)h->a.B;
    cudaStream_t s = h->own_stream;
    // pageable buffers work too (the runtime stages them); page-locked ones (the Python wrapper's) make the copies asynchronous
    int rc = step_from_host(h, actions_host);
    if (rc) return rc;
    // the kernels write the row without its forecast block a second time, packed: one contiguous copy
    if (head_host) GLG_CUDA(h, cudaMemcpyAsync(head_host, h->a.obs_head, (size_t)h->n_head * B * sizeof(float), cudaMemcpyDeviceToHost, s));
    if (timestep_host) GLG_CUDA(h, cudaMemcpyAsync(timestep_host, h->a.timestep, B * sizeof(int), cudaMemcpyDeviceToHost, s));
    if (table_host) GLG_CUDA(h, cudaMemcpyAsync(table_host, h->a.table, B * sizeof(int), cudaMemcpyDeviceToHost, s));
    if (reward_host) GLG_CUDA(h, cudaMemcpyAsync(reward_host, h->a.reward, B * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (done_host) GLG_CUDA(h, cudaMemcpyAsync(done_host, h->a.done, B, cudaMemcpyDeviceToHost, s));
    GLG_CUDA(h, cudaStreamSynchronize(s));
    return GLG_OK;
}

extern "C" int32_t glg_obs_dim(const glg_handle *h) { return h ? h->a.obs_dim : 0; }
extern "C" float *glg_obs_dev(glg_handle *h) { return h ? h->a.obs : nullptr; }
extern "C" float *glg_terminal_obs_dev(glg_handle *h) { return h ? h->a.term_obs : nullptr; }
extern "C" double *glg_reward_dev(glg_handle *h) { return h ? h->a.reward : nullptr; }
extern "C" uint8_t *glg_done_dev(glg_handle *h) { return h ? h->a.done : nullptr; }
extern "C" double *glg_info_dev(glg_handle *h) { return h ? h->a.info : nullptr; }
extern "C" double *glg_state_dev(glg_handle *h) { return h ? h->a.x : nullptr; }
extern "C" double *glg_controls_dev(glg_handle *h) { return h ? h->a.u : nullptr; }
extern "C" int32_t *glg_timestep_dev(glg_handle *h) { return h ? h->a.timestep : nullptr; }
extern "C" int32_t *glg_table_dev(glg_handle *h) { return h ? h->a.table : nullptr; }
extern "C" double *glg_time_dev(glg_handle *h) { return h ? h->a.time : nullptr; }
extern "C" double *glg_stats_dev(glg_handle *h) { return h ? h->a.stats : nullptr; }
extern "C" int64_t glg_launch_count(const glg_handle *h) { return h ? h->launches : 0; }

extern "C" int glg_clear_stats(glg_handle *h, void *stream) {
    if (!h) return GLG_ERR_ARG;
    GLG_CUDA(h, cudaSetDevice(h->cfg.device));
    GLG_CUDA(h, cudaMemsetAsync(h->a.stats, 0, GLG_NSTATS * sizeof(double), (cudaStream_t)stream));
    return GLG_OK;
}

// full per-env state (checkpoint / restore): [B][n] row-major host <-> [n][B] device SoA when `soa`
template <class T>
static cudaError_t copy_field(bool to_dev, T *dev, T *host, size_t n_per_env, int B, bool soa) {
    if (!host) return cudaSuccess;
    const size_t n = n_per_env * (size_t)B;
    if (!soa || n_per_env == 1) return to_dev ? cudaMemcpy(dev, host, n * sizeof(T), cudaMemcpyHostToDevice) : cudaMemcpy(host, dev, n * sizeof(T), cudaMemcpyDeviceToHost);
    std::vector<T> tmp(n);
    if (to_dev) {
        for (int b = 0; b < B; ++b)
            for (size_t i = 0; i < n_per_env; ++i) tmp[i * B + b] = host[(size_t)b * n_per_env + i];
        return cudaMemcpy(dev, tmp.data(), n * sizeof(T), cudaMemcpyHostToDevice);
    }
    cudaError_t e = cudaMemcpy(tmp.data(), dev, n * sizeof(T), cudaMemcpyDeviceToHost);
    for (int b = 0; b < B; ++b)
        for (size_t i = 0; i < n_per_env; ++i) host[(size_t)b * n_per_env + i] = tmp[i * B + b];
    return e;
}

extern "C" int glg_set_state(glg_handle *h, const double *x_host, const double *u_host, const int32_t *timestep_host) {
    if (!h) return GLG_ERR_ARG;
    h->kt_valid = false;
    GLG_CUDA(h, cudaSetDevice(h->cfg.device));
    GLG_CUDA(h, cudaDeviceSynchronize());
    const int B = h->a.B;
    // copy_field only reads the host side on its way to the device
    GLG_CUDA(h, copy_field(true, h->a.x, const_cast<double *>(x_host), GLG_NX, B, true));
    GLG_CUDA(h, copy_field(true, h->a.u, const_cast<double *>(u_host), GLG_NU, B, true));
    if (timestep_host) {
        // the env clock follows the timestep (tomato_env.py:126-128, :246-247): doy = start_day(table) + k dt/86400 (summed the way
        // the step does, one increment per step), hod = (k dt/3600) mod 24
        if (!h->a.weather) return fail(h, GLG_ERR_STATE, "glg_set_state: set the weather bank first");
        for (int b = 0; b < B; ++b)
            if (timestep_host[b] < 0 || timestep_host[b] > h->a.N) return fail(h, GLG_ERR_ARG, "glg_set_state: timestep outside [0, N]");
        std::vector<int> tb(B);
        std::vector<double> sd(h->a.n_tables), tm((size_t)2 * B);
        GLG_CUDA(h, cudaMemcpy(tb.data(), h->a.table, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost));
        GLG_CUDA(h, cudaMemcpy(sd.data(), h->a.start_day, (size_t)h->a.n_tables * sizeof(double), cudaMemcpyDeviceToHost));
        const double ddoy = fmod(h->a.dt / 86400.0, 365.0), dhod = h->a.dt / 3600.0;
        for (int b = 0; b < B; ++b) {
            double doy = sd[tb[b]], hod = 0.0;
            for (int k = 0; k < timestep_host[b]; ++k) {
                doy += ddoy;
                hod = fmod(hod + dhod, 24.0);
            }
            tm[b] = doy;
            tm[(size_t)B + b] = hod;
        }
        GLG_CUDA(h, cudaMemcpy(h->a.time, tm.data(), tm.size() * sizeof(double), cudaMemcpyHostToDevice));
        GLG_CUDA(h, cudaMemcpy(h->a.timestep, timestep_host, (size_t)B * sizeof(int), cudaMemcpyHostToDevice));
    }
    return GLG_OK;
}

static int state_ex(glg_handle *h, const glg_env_state *s, bool to_dev) {
    if (!h || !s) return GLG_ERR_ARG;
    GLG_CUDA(h, cudaSetDevice(h->cfg.device));
    GLG_CUDA(h, cudaDeviceSynchronize());
    const GlgStepArgs &a = h->a;
    const int B = a.B;
    if (to_dev) h->kt_valid = false;
    if (to_dev) {
        if (s->table) {
            if (!a.weather) return fail(h, GLG_ERR_STATE, "glg_set_state_ex: set the weather bank first");
            for (int b = 0; b < B; ++b)
                if (s->table[b] < 0 || s->table[b] >= a.n_tables) return fail(h, GLG_ERR_ARG, "glg_set_state_ex: table id out of range");
        }
        if (s->timestep)
            for (int b = 0; b < B; ++b)
                if (s->timestep[b] < 0 || s->timestep[b] > a.N + 1) return fail(h, GLG_ERR_ARG, "glg_set_state_ex: timestep outside [0, N + 1]");
    }
    GLG_CUDA(h, copy_field(to_dev, a.x, s->x, GLG_NX, B, true));
    GLG_CUDA(h, copy_field(to_dev, a.u, s->u, GLG_NU, B, true));
    GLG_CUDA(h, copy_field(to_dev, a.timestep, s->timestep, 1, B, false));
    GLG_CUDA(h, copy_field(to_dev, a.table, s->table, 1, B, false));
    GLG_CUDA(h, copy_field(to_dev, a.time, s->time, 2, B, true));
    GLG_CUDA(h, copy_field(to_dev, a.step_ctr, s->step_ctr, 1, B, false));
    GLG_CUDA(h, copy_field(to_dev, a.ep_return, s->ep_return, 1, B, false));
    GLG_CUDA(h, copy_field(to_dev, a.ep_len, s->ep_len, 1, B, false));
    GLG_CUDA(h, copy_field(to_dev, a.ep_info, s->ep_info, GLG_NINFO, B, true));
    if (to_dev) h->is_reset = true;
    return GLG_OK;
}
extern "C" int glg_get_state_ex(glg_handle *h, const glg_env_state *out_host) { return state_ex(h, out_host, false); }
extern "C" int glg_set_state_ex(glg_handle *h, const glg_env_state *in_host) { return state_ex(h, in_host, true); }

extern "C" int glg_get_state(glg_handle *h, double *x_host, double *u_host, int32_t *timestep_host) {
    glg_env_state s = {};
    s.x = x_host; s.u = u_host; s.timestep = timestep_host;
    return state_ex(h, &s, false);
}

// ---- VecNormalize state of a rollout or replay buffer, updated by the glg_roll_* kernels (glg_rollout.cuh) ----
struct GlgNorm {
    int training = 0, norm_obs = 0, norm_reward = 0, blocks = 0;
    double gamma = 0.0, clip_obs = 0.0, clip_reward = 0.0, epsilon = 0.0;
    double *ret = nullptr, *stat = nullptr, *partial = nullptr, *norm64 = nullptr;
};

// c: glg_rollout_config or glg_replay_config, which share the VecNormalize fields.  Arrays for the handle's batch, owned by `mem`
// (the rollout's or replay buffer's).
template <class Cfg>
static cudaError_t norm_create(GlgNorm *n, CudaMem &mem, const glg_handle *h, const Cfg &c) {
    n->training = c.training; n->norm_obs = c.norm_obs; n->norm_reward = c.norm_reward;
    n->gamma = c.gamma; n->clip_obs = c.clip_obs; n->clip_reward = c.clip_reward; n->epsilon = c.epsilon;
    const size_t B = (size_t)h->a.B, D = (size_t)h->a.obs_dim;
    n->blocks = (int)((B + GLG_ROLL_ROWS - 1) / GLG_ROLL_ROWS);
    cudaError_t e = mem.dev(&n->ret, B);
    if (e == cudaSuccess) e = mem.dev(&n->stat, (D + 1) * 3);
    if (e == cudaSuccess) e = mem.dev(&n->partial, (size_t)n->blocks * (D + 1) * 2);
    if (e == cudaSuccess) e = mem.dev(&n->norm64, (D + 1) * 2);
    if (e != cudaSuccess) return e;
    std::vector<double> st;
    for (size_t c = 0; c <= D; ++c) st.insert(st.end(), {0.0, 1.0, 1e-4});  // RunningMeanStd: mean 0, var 1, count 1e-4
    return cudaMemcpy(n->stat, st.data(), st.size() * sizeof(double), cudaMemcpyHostToDevice);
}

// VecNormalize.step_wait (after_step) or .reset on the handle's current outputs: statistics updated, normalised observations into
// obs_out, normalised rewards into reward_out and episode starts into starts_out (either may be NULL).  Three launches on s.
static void norm_update(const GlgNorm &n, glg_handle *h, bool after_step, float *obs_out, float *reward_out, float *starts_out,
                        cudaStream_t s) {
    const GlgStepArgs &e = h->a;
    GlgRollArgs a;
    memset(&a, 0, sizeof a);
    a.B = e.B; a.obs_dim = e.obs_dim; a.n_blocks = n.blocks;
    a.training = n.training; a.norm_obs = n.norm_obs; a.norm_reward = n.norm_reward;
    a.gamma = n.gamma; a.clip_obs = n.clip_obs; a.clip_reward = n.clip_reward; a.epsilon = n.epsilon;
    a.obs = e.obs;
    a.reward = after_step ? e.reward : nullptr;
    a.done = after_step ? e.done : nullptr;
    a.ret = n.ret; a.stat = n.stat; a.partial = n.partial; a.norm64 = n.norm64;
    a.obs_out = obs_out; a.reward_out = reward_out; a.starts_out = starts_out;
    glg_roll_moments_kernel<<<n.blocks, GLG_ROLL_NT, 0, s>>>(a);
    glg_roll_finish_kernel<<<(e.obs_dim + 1 + GLG_ROLL_NT / 32 - 1) / (GLG_ROLL_NT / 32), GLG_ROLL_NT, 0, s>>>(a);
    glg_roll_apply_kernel<<<n.blocks, GLG_ROLL_NT, 0, s>>>(a);
    h->launches += 3;
}

// ---- device rollout: VecNormalize + rollout buffer + GAE (glg_rollout.cuh); its own object, like the replay buffer ----------
struct glg_rollout {
    glg_handle *h = nullptr;  // not read on destruction: the env may already be gone
    int device = 0, n_steps = 0;
    double gae_lambda = 0.0;
    CudaMem mem;
    GlgNorm norm;
    float *obs = nullptr, *rew = nullptr, *starts = nullptr, *adv = nullptr, *ret = nullptr;
};

extern "C" void glg_rollout_destroy(glg_rollout *r) {
    if (!r) return;
    cudaSetDevice(r->device);
    delete r;
}

extern "C" int glg_rollout_create(glg_handle *h, const glg_rollout_config *cfg, glg_rollout **out) {
    if (!h || !cfg || !out) return GLG_ERR_ARG;
    *out = nullptr;
    if (cfg->n_steps < 1 || !(cfg->gamma >= 0.0 && cfg->gamma <= 1.0) || !(cfg->gae_lambda >= 0.0 && cfg->gae_lambda <= 1.0) ||
        !(cfg->clip_obs > 0) || !(cfg->clip_reward > 0) || !(cfg->epsilon > 0))
        return fail(h, GLG_ERR_ARG, "glg_rollout_create: invalid n_steps / gamma / gae_lambda / clip / epsilon");
    GLG_CUDA(h, cudaSetDevice(h->cfg.device));
    glg_rollout *r = new (std::nothrow) glg_rollout();
    if (!r) return fail(h, GLG_ERR_ALLOC, "glg_rollout_create: out of host memory");
    r->h = h; r->device = h->cfg.device; r->n_steps = cfg->n_steps; r->gae_lambda = cfg->gae_lambda;
    const size_t B = (size_t)h->a.B, T = (size_t)cfg->n_steps, D = (size_t)h->a.obs_dim;
    cudaError_t e = r->mem.dev(&r->obs, (T + 1) * B * D);
    if (e == cudaSuccess) e = r->mem.dev(&r->rew, T * B);
    if (e == cudaSuccess) e = r->mem.dev(&r->starts, (T + 1) * B);
    if (e == cudaSuccess) e = r->mem.dev(&r->adv, T * B);
    if (e == cudaSuccess) e = r->mem.dev(&r->ret, T * B);
    if (e == cudaSuccess) e = norm_create(&r->norm, r->mem, h, *cfg);
    if (e != cudaSuccess) {
        glg_rollout_destroy(r);
        return fail(h, GLG_ERR_CUDA, (std::string("glg_rollout_create: ") + cudaGetErrorString(e)).c_str());
    }
    *out = r;
    return GLG_OK;
}
extern "C" int glg_rollout_store(glg_rollout *r, int32_t t, void *stream) {
    if (!r) return GLG_ERR_ARG;
    glg_handle *h = r->h;
    if (t < -1 || t >= r->n_steps) return fail(h, GLG_ERR_ARG, "glg_rollout_store: t outside [-1, n_steps)");
    GLG_CUDA(h, cudaSetDevice(r->device));
    const size_t B = (size_t)h->a.B, D = (size_t)h->a.obs_dim;
    norm_update(r->norm, h, t >= 0, r->obs + (size_t)(t + 1) * B * D, t >= 0 ? r->rew + (size_t)t * B : nullptr,
                r->starts + (size_t)(t + 1) * B, (cudaStream_t)stream);
    GLG_CUDA(h, cudaGetLastError());
    return GLG_OK;
}
extern "C" int glg_rollout_carry(glg_rollout *r, void *stream) {
    if (!r) return GLG_ERR_ARG;
    glg_handle *h = r->h;
    GLG_CUDA(h, cudaSetDevice(r->device));
    const size_t B = (size_t)h->a.B, D = (size_t)h->a.obs_dim, T = (size_t)r->n_steps;
    GLG_CUDA(h, cudaMemcpyAsync(r->obs, r->obs + T * B * D, B * D * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    GLG_CUDA(h, cudaMemcpyAsync(r->starts, r->starts + T * B, B * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return GLG_OK;
}
extern "C" int glg_rollout_gae(glg_rollout *r, const float *values_dev, void *stream) {
    if (!r || !values_dev) return GLG_ERR_ARG;
    glg_handle *h = r->h;
    GLG_CUDA(h, cudaSetDevice(r->device));
    glg_roll_gae_kernel<<<(h->a.B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(r->n_steps, h->a.B, r->norm.gamma, r->gae_lambda,
                                                                                r->rew, values_dev, r->starts, r->adv, r->ret);
    h->launches += 1;
    GLG_CUDA(h, cudaGetLastError());
    return GLG_OK;
}
extern "C" float *glg_rollout_obs_dev(glg_rollout *r) { return r ? r->obs : nullptr; }
extern "C" float *glg_rollout_rewards_dev(glg_rollout *r) { return r ? r->rew : nullptr; }
extern "C" float *glg_rollout_starts_dev(glg_rollout *r) { return r ? r->starts : nullptr; }
extern "C" float *glg_rollout_advantages_dev(glg_rollout *r) { return r ? r->adv : nullptr; }
extern "C" float *glg_rollout_returns_dev(glg_rollout *r) { return r ? r->ret : nullptr; }
extern "C" double *glg_rollout_stats_dev(glg_rollout *r) { return r ? r->norm.stat : nullptr; }

// ---- device replay buffer (glg_replay.cuh): its own object, so several can share an env and none dangles from the handle ----
struct glg_replay {
    glg_handle *h = nullptr;  // not read on destruction: the env may already be gone
    int device = 0;
    uint64_t seed = 0;                   // Philox key of the sample indices
    unsigned long long weather_gen = 0;  // bank generation the keys refer to
    long long cap = 0, pos = 0;
    bool full = false, is_reset = false;
    uint32_t calls = 0;  // sample calls so far (Philox counter)
    CudaMem mem;         // every device array below and the normaliser's: glg_replay_bytes
    GlgNorm norm;
    float *obs_norm = nullptr, *last_head = nullptr, *head_obs = nullptr, *head_next = nullptr, *act = nullptr, *rew = nullptr;
    int *key_obs = nullptr, *key_next = nullptr, *anchor_t = nullptr, *anchor_tbl = nullptr;
    unsigned char *dn = nullptr;
};

extern "C" void glg_replay_destroy(glg_replay *r) {
    if (!r) return;
    cudaSetDevice(r->device);
    delete r;
}

extern "C" int glg_replay_create(glg_handle *h, const glg_replay_config *cfg, glg_replay **out) {
    if (!h || !cfg || !out) {
        g_error = "glg_replay_create: null argument";
        return GLG_ERR_ARG;
    }
    *out = nullptr;
    if (cfg->buffer_size < 1 || !(cfg->gamma >= 0.0 && cfg->gamma <= 1.0) || !(cfg->clip_obs > 0) || !(cfg->clip_reward > 0) ||
        !(cfg->epsilon > 0))
        return fail(h, GLG_ERR_ARG, "glg_replay_create: invalid buffer_size / gamma / clip / epsilon");
    if (!h->a.weather) return fail(h, GLG_ERR_STATE, "glg_replay_create: weather bank not set (glg_set_weather)");
    const size_t B = (size_t)h->a.B, D = (size_t)h->a.obs_dim;
    const long long cap = cfg->buffer_size / h->a.B > 1 ? cfg->buffer_size / h->a.B : 1;  // ReplayBuffer: max(buffer_size // n_envs, 1)
    if (cap > INT32_MAX) return fail(h, GLG_ERR_ARG, "glg_replay_create: more than 2^31 - 1 slots per env");
    GLG_CUDA(h, cudaSetDevice(h->cfg.device));
    glg_replay *r = new (std::nothrow) glg_replay();
    if (!r) return fail(h, GLG_ERR_ALLOC, "glg_replay_create: out of host memory");
    r->h = h;
    r->device = h->cfg.device;
    r->seed = cfg->seed;
    r->weather_gen = h->weather_gen;
    r->cap = cap;
    const size_t CB = (size_t)cap * B, H = (size_t)h->n_head;
    CudaMem &m = r->mem;
    cudaError_t e = m.dev(&r->head_obs, CB * H);
    if (e == cudaSuccess) e = m.dev(&r->head_next, CB * H);
    if (e == cudaSuccess) e = m.dev(&r->key_obs, CB);
    if (e == cudaSuccess) e = m.dev(&r->key_next, CB);
    if (e == cudaSuccess) e = m.dev(&r->act, CB * GLG_NU);
    if (e == cudaSuccess) e = m.dev(&r->rew, CB);
    if (e == cudaSuccess) e = m.dev(&r->dn, CB);
    if (e == cudaSuccess) e = m.dev(&r->obs_norm, B * D);
    if (e == cudaSuccess) e = m.dev(&r->last_head, B * H);
    if (e == cudaSuccess) e = m.dev(&r->anchor_t, B);
    if (e == cudaSuccess) e = m.dev(&r->anchor_tbl, B);
    if (e == cudaSuccess) e = norm_create(&r->norm, m, h, *cfg);
    if (e != cudaSuccess) {
        glg_replay_destroy(r);
        return fail(h, GLG_ERR_CUDA, (std::string("glg_replay_create: ") + cudaGetErrorString(e)).c_str());
    }
    *out = r;
    return GLG_OK;
}

static int replay_check(glg_replay *r, const char *what) {
    glg_handle *h = r->h;
    if (r->weather_gen != h->weather_gen) {
        h->err = std::string(what) + ": the weather bank was replaced (glg_set_weather) after this replay buffer was created; "
                                     "its stored forecast keys no longer refer to it";
        return GLG_ERR_STATE;
    }
    return GLG_OK;
}

static void replay_write_args(const glg_replay *r, GlgReplayArgs *w) {
    const GlgStepArgs &a = r->h->a;
    memset(w, 0, sizeof *w);
    w->B = a.B; w->obs_dim = a.obs_dim; w->n_head = r->h->n_head; w->nf = a.obs_dim - r->h->n_head; w->fc_off = a.fc_off; w->Np = a.Np;
    w->rows = a.rows; w->auto_reset = a.auto_reset;
    w->obs = a.obs; w->term_obs = a.term_obs; w->reward = a.reward; w->done = a.done; w->timestep = a.timestep; w->table = a.table;
    w->last_head = r->last_head; w->anchor_t = r->anchor_t; w->anchor_tbl = r->anchor_tbl;
    w->head_obs = r->head_obs; w->head_next = r->head_next; w->key_obs = r->key_obs; w->key_next = r->key_next;
    w->act = r->act; w->rew = r->rew; w->dn = r->dn;
}

extern "C" int glg_replay_reset(glg_replay *r, void *stream) {
    if (!r) return GLG_ERR_ARG;
    glg_handle *h = r->h;
    int rc = replay_check(r, "glg_replay_reset");
    if (rc) return rc;
    if (!h->is_reset) return fail(h, GLG_ERR_STATE, "glg_replay_reset: the env has not been reset (glg_reset)");
    GLG_CUDA(h, cudaSetDevice(r->device));
    cudaStream_t s = (cudaStream_t)stream;
    norm_update(r->norm, h, false, r->obs_norm, nullptr, nullptr, s);
    GlgReplayArgs w;
    replay_write_args(r, &w);
    w.store = 0;
    glg_replay_write_kernel<<<r->norm.blocks, GLG_ROLL_NT, 0, s>>>(w);
    h->launches += 1;
    GLG_CUDA(h, cudaGetLastError());
    r->is_reset = true;
    return GLG_OK;
}

extern "C" int glg_replay_store(glg_replay *r, const float *actions_dev, void *stream) {
    if (!r) return GLG_ERR_ARG;
    glg_handle *h = r->h;
    if (!actions_dev) return fail(h, GLG_ERR_ARG, "glg_replay_store: actions_dev is NULL");
    int rc = replay_check(r, "glg_replay_store");
    if (rc) return rc;
    if (!r->is_reset) return fail(h, GLG_ERR_STATE, "glg_replay_store: store before glg_replay_reset");
    GLG_CUDA(h, cudaSetDevice(r->device));
    cudaStream_t s = (cudaStream_t)stream;
    norm_update(r->norm, h, true, r->obs_norm, nullptr, nullptr, s);
    GlgReplayArgs w;
    replay_write_args(r, &w);
    w.store = 1;
    w.slot = (size_t)r->pos;
    w.actions = actions_dev;
    glg_replay_write_kernel<<<r->norm.blocks, GLG_ROLL_NT, 0, s>>>(w);
    h->launches += 1;
    GLG_CUDA(h, cudaGetLastError());
    if (++r->pos == r->cap) {
        r->full = true;
        r->pos = 0;
    }
    return GLG_OK;
}

extern "C" int glg_replay_sample(glg_replay *r, int32_t n, float *obs_dev, float *next_obs_dev, float *actions_dev,
                                 float *rewards_dev, float *dones_dev, int32_t *index_dev, void *stream) {
    if (!r) return GLG_ERR_ARG;
    glg_handle *h = r->h;
    if (n < 1 || !obs_dev || !next_obs_dev || !actions_dev || !rewards_dev || !dones_dev)
        return fail(h, GLG_ERR_ARG, "glg_replay_sample: n < 1 or a NULL output");
    int rc = replay_check(r, "glg_replay_sample");
    if (rc) return rc;
    const long long upper = r->full ? r->cap : r->pos;
    if (upper == 0) return fail(h, GLG_ERR_STATE, "glg_replay_sample: the replay buffer is empty (no glg_replay_store yet)");
    GLG_CUDA(h, cudaSetDevice(r->device));
    GlgReplaySampleArgs S;
    memset(&S, 0, sizeof S);
    S.n = n; S.B = h->a.B; S.obs_dim = h->a.obs_dim; S.n_head = h->n_head; S.nf = h->a.obs_dim - h->n_head; S.fc_off = h->a.fc_off;
    S.norm_obs = r->norm.norm_obs; S.norm_reward = r->norm.norm_reward;
    S.upper = (uint32_t)upper; S.call = r->calls; S.seed = r->seed;
    S.clip_obs = r->norm.clip_obs; S.clip_reward = r->norm.clip_reward;
    S.norm64 = r->norm.norm64;
    S.weather = h->a.weather;  // read on every call: glg_set_weather reallocates the bank
    S.head_obs = r->head_obs; S.head_next = r->head_next; S.key_obs = r->key_obs; S.key_next = r->key_next;
    S.act = r->act; S.rew = r->rew; S.dn = r->dn;
    S.obs_out = obs_dev; S.next_out = next_obs_dev; S.act_out = actions_dev; S.rew_out = rewards_dev; S.done_out = dones_dev;
    S.idx_out = index_dev;
    constexpr int per_cta = GLG_REPLAY_NT / 32;
    glg_replay_sample_kernel<<<(n + per_cta - 1) / per_cta, GLG_REPLAY_NT, 0, (cudaStream_t)stream>>>(S);
    h->launches += 1;
    GLG_CUDA(h, cudaGetLastError());
    ++r->calls;
    return GLG_OK;
}

extern "C" int64_t glg_replay_size(const glg_replay *r) { return r ? (r->full ? r->cap : r->pos) : 0; }
extern "C" int64_t glg_replay_bytes(const glg_replay *r) { return r ? (int64_t)r->mem.bytes() : 0; }
extern "C" float *glg_replay_obs_dev(glg_replay *r) { return r ? r->obs_norm : nullptr; }
extern "C" double *glg_replay_stats_dev(glg_replay *r) { return r ? r->norm.stat : nullptr; }

// ---- receding-horizon planner (glg_plan.cuh): its own object holding a second, internal handle of B K planning envs that the
// unchanged step kernels advance; the env handle is only read ----
struct glg_plan {
    glg_handle *h = nullptr;  // the env whose states are planned from (read only; not on destruction: it may already be gone)
    // planning envs: B K, no auto-reset, nominal model; points at h's weather bank and owns none (see plan_sync)
    std::unique_ptr<glg_handle> hp;
    int device = 0, B = 0, BK = 0;
    glg_plan_config cfg = {};
    unsigned long long weather_gen = 0;  // bank generation hp's pointers refer to
    uint32_t calls = 0;                  // glg_plan_run calls so far (Philox counter word 1)
    CudaMem mem;
    float *mean = nullptr, *std = nullptr, *cand = nullptr;
    double *ret = nullptr;
    unsigned char *alive = nullptr;
};

static constexpr long long kPlanMaxBatch = 4194304;  // B K: the largest batch the step kernels were run at (profiles/r2_config_sweep.txt)

extern "C" void glg_plan_destroy(glg_plan *p) {
    if (!p) return;
    cudaSetDevice(p->device);
    delete p;
}

extern "C" int glg_plan_create(glg_handle *h, const glg_plan_config *cfg, glg_plan **out) {
    if (!h || !cfg || !out) {
        g_error = "glg_plan_create: null argument";
        return GLG_ERR_ARG;
    }
    *out = nullptr;
    const glg_plan_config &c = *cfg;
    if (c.horizon < 1 || c.n_candidates < 1 || c.n_elites < 1 || c.n_elites > c.n_candidates || c.n_candidates > GLG_PLAN_MAXK ||
        c.n_iterations < 1)
        return fail(h, GLG_ERR_ARG, "glg_plan_create: need horizon >= 1, 1 <= n_elites <= n_candidates <= 4096, n_iterations >= 1");
    if (!(c.gamma > 0.0 && c.gamma <= 1.0) || !(c.init_std > 0.0 && c.init_std < 3.4e38))  // std is stored as float
        return fail(h, GLG_ERR_ARG, "glg_plan_create: need 0 < gamma <= 1 and a finite init_std > 0");
    if ((long long)h->a.B * c.n_candidates > kPlanMaxBatch)
        return fail(h, GLG_ERR_ARG, "glg_plan_create: num_envs * n_candidates > 4194304 planning envs");
    if ((uint64_t)c.n_iterations * (uint64_t)c.horizon * 3u > UINT32_MAX)
        return fail(h, GLG_ERR_ARG, "glg_plan_create: n_iterations * horizon * 3 must fit the 32-bit Philox counter word");
    if (!h->have_params || !h->a.weather)
        return fail(h, GLG_ERR_STATE, "glg_plan_create: set the env's parameters and weather bank first");
    GLG_CUDA(h, cudaSetDevice(h->cfg.device));
    glg_plan *p = new (std::nothrow) glg_plan();
    if (!p) return fail(h, GLG_ERR_ALLOC, "glg_plan_create: out of host memory");
    p->h = h;
    p->device = h->cfg.device;
    p->cfg = c;
    p->B = h->a.B;
    p->BK = h->a.B * c.n_candidates;
    glg_config pc = h->cfg;  // precision, integrator, n_sub, N, Np, prices, constraints and the observation stack stay the env's
    pc.num_envs = p->BK;
    pc.auto_reset = 0;
    pc.uncertainty_scale = 0.0;
    pc.seed = h->a.seed;  // the env's current seed (glg_set_seed): StateObservations entries are keyed by it
    pc.env_id_offset = 0;
    pc.role_warps = 0;
    pc.role_lanes = 0;
    glg_handle *hp = nullptr;
    int rc = glg_create(&pc, &hp);
    p->hp.reset(hp);
    if (rc != GLG_OK) {
        h->err = std::string("glg_plan_create: planning handle: ") + g_error;
        glg_plan_destroy(p);
        return rc;
    }
    hp->is_reset = true;  // every run / evaluate loads its states (fan-out) before stepping
    const size_t HB6 = (size_t)c.horizon * p->B * GLG_NU, HBK6 = (size_t)c.horizon * p->BK * GLG_NU;
    cudaError_t e = p->mem.dev(&p->mean, HB6);
    if (e == cudaSuccess) e = p->mem.dev(&p->std, HB6);
    if (e == cudaSuccess) e = p->mem.dev(&p->cand, HBK6);
    if (e == cudaSuccess) e = p->mem.dev(&p->ret, (size_t)p->BK);
    if (e == cudaSuccess) e = p->mem.dev(&p->alive, (size_t)p->BK);
    if (e == cudaSuccess) {
        std::vector<float> s0(HB6, (float)c.init_std);
        e = cudaMemcpy(p->std, s0.data(), HB6 * sizeof(float), cudaMemcpyHostToDevice);
    }
    if (e != cudaSuccess) {
        glg_plan_destroy(p);
        return fail(h, GLG_ERR_CUDA, (std::string("glg_plan_create: ") + cudaGetErrorString(e)).c_str());
    }
    p->weather_gen = h->weather_gen;
    *out = p;
    return GLG_OK;
}

// Before every run / evaluate: the env must be reset and still hold the bank the planner was created under; its parameters
// (glg_set_params may have been called since) and bank pointers are copied into the planning handle.  Host fields only.
static int plan_sync(glg_plan *p, const char *what) {
    glg_handle *h = p->h, *hp = p->hp.get();
    if (p->weather_gen != h->weather_gen) {
        h->err = std::string(what) + ": the weather bank was replaced (glg_set_weather) after this planner was created";
        return GLG_ERR_STATE;
    }
    if (!h->is_reset) {
        h->err = std::string(what) + ": the env has not been reset (glg_reset)";
        return GLG_ERR_STATE;
    }
    hp->uni = h->uni;
    hp->general = h->general;
    hp->have_params = true;
    hp->a.weather = h->a.weather; hp->a.start_day = h->a.start_day; hp->a.reset_tables = h->a.reset_tables;
    hp->a.n_tables = h->a.n_tables; hp->a.rows = h->a.rows; hp->a.n_reset_tables = h->a.n_reset_tables;
    return GLG_OK;
}

static int plan_fanout(glg_plan *p, cudaStream_t s) {
    const GlgStepArgs &e = p->h->a, &pe = p->hp->a;
    GlgPlanFanArgs A;
    memset(&A, 0, sizeof A);
    A.B = p->B; A.K = p->cfg.n_candidates;
    A.x = e.x; A.u = e.u; A.time = e.time; A.timestep = e.timestep; A.table = e.table; A.step_ctr = e.step_ctr;
    A.px = pe.x; A.pu = pe.u; A.ptime = pe.time; A.pep_return = pe.ep_return; A.pep_info = pe.ep_info;
    A.ptimestep = pe.timestep; A.ptable = pe.table; A.pep_len = pe.ep_len; A.pstep_ctr = pe.step_ctr; A.pdone = pe.done;
    A.ret = p->ret; A.alive = p->alive;
    glg_plan_fanout_kernel<<<(p->BK + GLG_PLAN_NT - 1) / GLG_PLAN_NT, GLG_PLAN_NT, 0, s>>>(A);
    GLG_CUDA(p->h, cudaGetLastError());
    return GLG_OK;
}

// H steps of the planning envs with the actions seq[t] ([B K][6] each), discounted returns accumulated into p->ret
static int plan_rollout(glg_plan *p, const float *seq, cudaStream_t s) {
    glg_handle *h = p->h, *hp = p->hp.get();
    const size_t step_stride = (size_t)p->BK * GLG_NU;
    double d = 1.0;
    for (int t = 0; t < p->cfg.horizon; ++t) {
        const int rc = glg_step(hp, seq + (size_t)t * step_stride, nullptr, s);
        if (rc != GLG_OK) {
            h->err = "planning step: " + hp->err;
            return rc;
        }
        glg_plan_accum_kernel<<<(p->BK + GLG_PLAN_NT - 1) / GLG_PLAN_NT, GLG_PLAN_NT, 0, s>>>(p->BK, d, hp->a.reward, hp->a.done,
                                                                                            p->ret, p->alive);
        GLG_CUDA(h, cudaGetLastError());
        d *= p->cfg.gamma;
    }
    return GLG_OK;
}

extern "C" int glg_plan_run(glg_plan *p, float *actions_dev, void *stream) {
    if (!p) return GLG_ERR_ARG;
    glg_handle *h = p->h;
    if (!actions_dev) return fail(h, GLG_ERR_ARG, "glg_plan_run: actions_dev is NULL");
    int rc = plan_sync(p, "glg_plan_run");
    if (rc) return rc;
    GLG_CUDA(h, cudaSetDevice(p->device));
    cudaStream_t s = (cudaStream_t)stream;
    const glg_plan_config &c = p->cfg;
    for (int it = 0; it < c.n_iterations; ++it) {
        if ((rc = plan_fanout(p, s))) return rc;
        GlgPlanSampleArgs S;
        memset(&S, 0, sizeof S);
        S.B = p->B; S.K = c.n_candidates; S.H = c.horizon; S.it = (uint32_t)it; S.call = p->calls; S.seed = c.seed;
        S.mean = p->mean; S.std = p->std; S.cand = p->cand;
        glg_plan_sample_kernel<<<(p->BK + GLG_PLAN_NT - 1) / GLG_PLAN_NT, GLG_PLAN_NT, 0, s>>>(S);
        GLG_CUDA(h, cudaGetLastError());
        if ((rc = plan_rollout(p, p->cand, s))) return rc;
        GlgPlanUpdateArgs U;
        memset(&U, 0, sizeof U);
        U.B = p->B; U.K = c.n_candidates; U.E = c.n_elites; U.H = c.horizon;
        U.ret = p->ret; U.cand = p->cand; U.mean = p->mean; U.std = p->std;
        U.actions = it + 1 == c.n_iterations ? actions_dev : nullptr;
        glg_plan_update_kernel<<<p->B, GLG_PLAN_NT, 0, s>>>(U);
        GLG_CUDA(h, cudaGetLastError());
    }
    ++p->calls;
    return GLG_OK;
}

extern "C" int glg_plan_evaluate(glg_plan *p, const float *seq_dev, double *returns_dev, void *stream) {
    if (!p) return GLG_ERR_ARG;
    glg_handle *h = p->h;
    if (!seq_dev || !returns_dev) return fail(h, GLG_ERR_ARG, "glg_plan_evaluate: seq_dev or returns_dev is NULL");
    int rc = plan_sync(p, "glg_plan_evaluate");
    if (rc) return rc;
    GLG_CUDA(h, cudaSetDevice(p->device));
    cudaStream_t s = (cudaStream_t)stream;
    if ((rc = plan_fanout(p, s))) return rc;
    if ((rc = plan_rollout(p, seq_dev, s))) return rc;
    if (returns_dev != p->ret)
        GLG_CUDA(h, cudaMemcpyAsync(returns_dev, p->ret, (size_t)p->BK * sizeof(double), cudaMemcpyDeviceToDevice, s));
    return GLG_OK;
}

extern "C" int glg_plan_shift(glg_plan *p, void *stream) {
    if (!p) return GLG_ERR_ARG;
    glg_handle *h = p->h;
    GLG_CUDA(h, cudaSetDevice(p->device));
    glg_plan_shift_kernel<<<(p->B * GLG_NU + GLG_PLAN_NT - 1) / GLG_PLAN_NT, GLG_PLAN_NT, 0, (cudaStream_t)stream>>>(
        p->B, p->cfg.horizon, (float)p->cfg.init_std, p->mean, p->std);
    GLG_CUDA(h, cudaGetLastError());
    return GLG_OK;
}

extern "C" float *glg_plan_mean_dev(glg_plan *p) { return p ? p->mean : nullptr; }
extern "C" float *glg_plan_std_dev(glg_plan *p) { return p ? p->std : nullptr; }
extern "C" float *glg_plan_candidates_dev(glg_plan *p) { return p ? p->cand : nullptr; }
extern "C" double *glg_plan_returns_dev(glg_plan *p) { return p ? p->ret : nullptr; }

// ---- episode-statistics all-reduce over NCCL (run-time binding: nccl_api above)
extern "C" int glg_nccl_unique_id(uint8_t id_out[128]) {
    if (!id_out) return GLG_ERR_ARG;
    std::string err;
    NcclApi *n = nccl_api(&err);
    if (!n) {
        g_error = err;
        return GLG_ERR_STATE;
    }
    NcclId id;
    const int rc = n->GetUniqueId(&id);
    if (rc != 0) {
        g_error = std::string("ncclGetUniqueId: ") + (n->GetErrorString ? n->GetErrorString(rc) : "error");
        return GLG_ERR_CUDA;
    }
    memcpy(id_out, id.internal, 128);
    return GLG_OK;
}
extern "C" int glg_nccl_init(glg_handle *h, const uint8_t id[128], int32_t rank, int32_t world_size) {
    if (!h || !id || world_size < 1 || rank < 0 || rank >= world_size) return GLG_ERR_ARG;
    NcclApi *n = nccl_api(&h->err);
    if (!n) return GLG_ERR_STATE;
    GLG_CUDA(h, cudaSetDevice(h->cfg.device));
    if (h->nccl_comm) {
        n->CommDestroy(h->nccl_comm);
        h->nccl_comm = nullptr;
    }
    NcclId nid;
    memcpy(nid.internal, id, 128);
    const int rc = n->CommInitRank(&h->nccl_comm, world_size, nid, rank);
    if (rc != 0) {
        h->nccl_comm = nullptr;
        return fail(h, GLG_ERR_CUDA, (std::string("ncclCommInitRank: ") + (n->GetErrorString ? n->GetErrorString(rc) : "error")).c_str());
    }
    return GLG_OK;
}
extern "C" int glg_allreduce_stats(glg_handle *h, void *stream) {
    if (!h) return GLG_ERR_ARG;
    if (!h->nccl_comm) return fail(h, GLG_ERR_STATE, "glg_allreduce_stats: no communicator (glg_nccl_init)");
    NcclApi *n = nccl_api(&h->err);
    if (!n) return GLG_ERR_STATE;
    GLG_CUDA(h, cudaSetDevice(h->cfg.device));
    const int rc = n->AllReduce(h->a.stats, h->a.stats, GLG_NSTATS, /*ncclDouble*/ 8, /*ncclSum*/ 0, h->nccl_comm, (cudaStream_t)stream);
    if (rc != 0) return fail(h, GLG_ERR_CUDA, (std::string("ncclAllReduce: ") + (n->GetErrorString ? n->GetErrorString(rc) : "error")).c_str());
    return GLG_OK;
}

// ---- batched evalF (handle-free) ------------------------------------------------------------------------

template <bool GENERAL, bool PER_ENV_P>
static cudaError_t launch_evalf(const GlgUniform &uni, const double *x, const double *u, const double *d, const double *p,
                                double *xn, unsigned char *bad, int B, double dt, int n_sub, int integrator, cudaStream_t s) {
    constexpr int NT = 64;
    const size_t smem = sizeof(double) * (size_t)(2 * GLG_NX + H_COUNT) * NT;
    cudaError_t e = cudaFuncSetAttribute(glg_evalf_kernel<GENERAL, PER_ENV_P, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    glg_evalf_kernel<GENERAL, PER_ENV_P, NT><<<(B + NT - 1) / NT, NT, smem, s>>>(uni, x, u, d, p, xn, bad, B, dt, n_sub, integrator);
    return cudaGetLastError();
}

extern "C" int glg_evalf_batch(const double *x_dev, const double *u_dev, const double *d_dev, const double *p_dev,
                               int32_t p_stride, double *x_next_dev, uint8_t *bad_dev, int32_t B, double dt, int32_t n_sub,
                               int32_t device, void *stream) {
    return glg_evalf_batch_ex(x_dev, u_dev, d_dev, p_dev, p_stride, x_next_dev, bad_dev, B, dt, n_sub, 0, device, stream);
}

extern "C" int glg_evalf_batch_ex(const double *x_dev, const double *u_dev, const double *d_dev, const double *p_dev,
                                  int32_t p_stride, double *x_next_dev, uint8_t *bad_dev, int32_t B, double dt, int32_t n_sub,
                                  int32_t integrator, int32_t device, void *stream) {
    if (!x_dev || !u_dev || !d_dev || !p_dev || !x_next_dev || B < 1 || n_sub < 1 || (p_stride != 0 && p_stride != GLG_NP) ||
        (integrator != 0 && integrator != 1)) {
        g_error = "glg_evalf_batch: invalid argument";
        return GLG_ERR_ARG;
    }
    cudaError_t e = cudaSetDevice(device);
    cudaStream_t s = (cudaStream_t)stream;
    GlgUniform uni{};  // only read by the shared-p variants (passed to the kernel by value)
    if (e == cudaSuccess) {
        if (p_stride == 0) {
            double ph[GLG_NP];
            e = cudaMemcpyAsync(ph, p_dev, sizeof ph, cudaMemcpyDeviceToHost, s);
            if (e == cudaSuccess) e = cudaStreamSynchronize(s);
            if (e == cudaSuccess) {
                for (int i = 0; i < GLG_NP; ++i) uni.P[i] = ph[i];
                glg_make_k(ph, uni.K);
                glg_make_c(ph, uni.C);
                e = glg_params_nominal_structure(ph)
                        ? launch_evalf<false, false>(uni, x_dev, u_dev, d_dev, p_dev, x_next_dev, bad_dev, B, dt, n_sub, integrator, s)
                        : launch_evalf<true, false>(uni, x_dev, u_dev, d_dev, p_dev, x_next_dev, bad_dev, B, dt, n_sub, integrator, s);
            }
        } else {
            e = launch_evalf<true, true>(uni, x_dev, u_dev, d_dev, p_dev, x_next_dev, bad_dev, B, dt, n_sub, integrator, s);
        }
    }
    if (e != cudaSuccess) {
        g_error = std::string("glg_evalf_batch: ") + cudaGetErrorString(e);
        return GLG_ERR_CUDA;
    }
    return GLG_OK;
}

// ---- roofline denominators ------------------------------------------------------------------------------
template <typename T>
static int measure_peak(int device, double *out) {
    if (!out) return GLG_ERR_ARG;
    cudaError_t e = cudaSetDevice(device);
    cudaDeviceProp prop;
    if (e == cudaSuccess) e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) {
        g_error = std::string("glg_measure_peak: ") + cudaGetErrorString(e);
        return GLG_ERR_CUDA;
    }
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
    CudaMem mem;
    T *buf = nullptr;
    mem.dev(&buf, (size_t)blocks * threads);
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        cudaEventRecord(a);
        glg_fma_peak_kernel<T><<<blocks, threads>>>(buf, iters, (T)0.999999, (T)1e-7);
        cudaEventRecord(b);
        cudaEventSynchronize(b);
        float ms = 0;
        cudaEventElapsedTime(&ms, a, b);
        const double flops = 2.0 * 64.0 * iters * (double)blocks * threads / (ms * 1e-3);
        if (rep > 0 && flops > best) best = flops;
    }
    e = cudaGetLastError();
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    if (e != cudaSuccess) {
        g_error = std::string("glg_measure_peak: ") + cudaGetErrorString(e);
        return GLG_ERR_CUDA;
    }
    *out = best;
    return GLG_OK;
}
extern "C" int glg_measure_fp64_peak(int32_t device, double *flops) { return measure_peak<double>(device, flops); }
extern "C" int glg_measure_fp32_peak(int32_t device, double *flops) { return measure_peak<float>(device, flops); }

#ifdef GLG_TRACE
extern "C" int glg_debug_trace(long long *out_host) {  // [32 evaluations][16 warps][wake, arrive] clock64 stamps of CTA 0
    return cudaMemcpyFromSymbol(out_host, glg_trace, sizeof(long long) * 32 * 16 * 2) == cudaSuccess ? GLG_OK : GLG_ERR_CUDA;
}
#endif

extern "C" int glg_debug_math(int32_t op, const double *in_dev, double *out_dev, int32_t n, void *stream) {
    if (!in_dev || !out_dev || n < 1) return GLG_ERR_ARG;
    glg_math_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(op, in_dev, out_dev, n);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        g_error = std::string("glg_debug_math: ") + cudaGetErrorString(e);
        return GLG_ERR_CUDA;
    }
    return GLG_OK;
}
