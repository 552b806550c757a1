// glg_roles.cuh -- step kernel C: warp-specialised evaluation of the GreenLight RHS with dedicated owner warps.
//
// One CTA = 32 envs x (NO owner warps + NG group warps); lane l of every warp works on env (32*blockIdx.x + l).
//   group warp g : evaluates its flux units (glg_units.h) for the 32 envs from the stage state in shared memory and stores
//                  one partial balance sum per (warp, state) it touches -- nothing else lives in its registers, so ptxas has
//                  the whole register budget for interleaving the transcendental chains of the units (the round-1 kernel
//                  carried the RK4 state of a quarter of the states in every warp: ~75 registers across the group code made
//                  ptxas serialise the chains: photosynthesis 1007 cycles in the kernel vs 570 compiled alone);
//   owner warp o : owns 28/NO states: classical RK4 stage update from the partial sums, state and stage sum in fp64
//                  registers, next stage value back to shared memory.  Also decides the micro-step count of every nominal
//                  substep (harvest guard, graded integrator) and tells the group warps when to stop.
// Synchronisation per RHS evaluation: two named barriers used producer/consumer style (PTX bar.arrive / bar.sync):
//   BAR_PARTS : group warps arrive (do not wait), owner warps wait -- "partial sums are in shared memory"
//   BAR_XS    : owner warps arrive (do not wait), group warps wait -- "stage state of the next evaluation is in shared memory"
// so a group warp blocks once per evaluation, on the data it needs.
// Every role has its own loop (no per-evaluation dispatch).  The loop bodies together must stay below the SM's 32 KB
// instruction cache (tools/ubench/icache2.cu), which is why the three "condensing surface" warps (thermal screen, blackout
// screen, cover) share ONE copy of their code with all addresses in registers (glg_surface_loop).
//
// Shared-memory layout of the exchange, chosen so that every owner-side address is base(owner) + immediate:
//   plan entry n = j * NO + o  : row j of owner o; states sorted by their number of contributing warps (descending), dealt
//                                round-robin, so row j loads as many slots as its hungriest state (its first entry)
//   xs  [n][32]                : stage state of plan entry n (units read state i at row rank(i), a compile-time constant)
//   part[(rowbase_j + c) * NO + o][32] : c-th partial sum of plan entry (j, o); unused (padding) slots stay 0.0
// The env-level work (S1 control update, S2 noise, hoisting, S3-S8 epilogue) is done by warp 0 (lane = env) with the
// same device functions as kernel A, so both kernels share one definition of the step semantics.
#pragma once
#include "glg_kernels.cuh"
#include "glg_units.h"

#define GLG_ROLE_LANES 32
constexpr int GLG_NO = 4;  // owner warps: warps 0..3, one per SM sub-partition
constexpr int GLG_BAR_PARTS = 1, GLG_BAR_XS = 2;
// The role loops of the latency layout together span ~32 KB of code, the SM's instruction-cache capacity
// (tools/ubench/icache2.cu): a variant whose loops span more is 3-20 % slower at B = 4096 whatever it was meant to gain, so every
// change to them is judged with tools/sass_loop_size.py beside the timer (DESIGN.md "Round-2 kernel experiments").
constexpr int GLG_MAXCONTRIB = 8;
constexpr int GLG_MAXROWS = 8;

// -DGLG_TRACE: per-warp clock64() stamps of CTA 0 (wake-up after the barrier wait, arrival at the next barrier) for evaluations
// 64..95 of a step, read back with glg_debug_trace (tools/trace_timeline.py).  Development builds only.
#ifdef GLG_TRACE
__device__ long long glg_trace[32][16][2];
#define GLG_TRACE_MARK(warp_, slot_, ev_)                                                          \
    do {                                                                                             \
        if (blockIdx.x == 0 && (threadIdx.x & 31) == 0 && (ev_) >= 64 && (ev_) < 96) glg_trace[(ev_) - 64][warp_][slot_] = clock64(); \
    } while (0)
#else
#define GLG_TRACE_MARK(warp_, slot_, ev_) do {} while (0)
#endif
// The barrier id is an immediate: with a register id the whole kernel reserves all 16 named barriers.
template <int ID>
__device__ __forceinline__ void glg_bar_sync(int nthreads) { asm volatile("bar.sync %1, %0;" ::"r"(nthreads), "n"(ID) : "memory"); }
// Scheduling fences: the value must be in a register at this point of the instruction stream (ptxas otherwise sinks work that
// was meant to overlap a barrier wait behind the barrier, and re-reads kernel parameters from the constant bank inside loops).
__device__ __forceinline__ void glg_pin(double &v) { asm volatile("" : "+d"(v)); }
__device__ __forceinline__ void glg_pin(int &v) { asm volatile("" : "+r"(v)); }
__device__ __forceinline__ void glg_bar_arrive(int id, int nthreads) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

// ---- owner plan and slot layout (see the header comment)
struct GlgOwnerPlan {
    int n_active;                         // states with at least one contribution
    int nj;                               // rows per owner warp
    int order[GLG_MAXROWS * GLG_NO];      // state of plan entry n, -1 pads
    int rank[GLG_NX];                     // plan entry of state i (states without contribution come after the active ones)
    int row_slots[GLG_MAXROWS];           // slots row j loads
    int row_base[GLG_MAXROWS + 1];        // prefix sum of row_slots
    int slot[16][GLG_NX];                 // part slot of (group warp, state), -1 if none
    int scale_k[GLG_MAXROWS * GLG_NO];    // glg_state_scale_index of the entry's state (-1: 1.0, -2: canopy scale slot)
    int n_slots;                          // NO * row_base[nj]
};
constexpr GlgOwnerPlan glg_make_plan(const GlgWarpTable &wt, int ng) {
    GlgOwnerPlan t{};
    // states sorted by their contribution counts, descending, and dealt round-robin to the owners: a row loads as many slots as
    // its hungriest state
    int n = 0;
    for (int key = GLG_MAXCONTRIB; key >= 0; --key)
        for (int i = 0; i < GLG_NX; ++i)
            if (wt.contribs[i] == key) {
                t.order[n] = i;
                t.rank[i] = n;
                t.scale_k[n] = glg_state_scale_index(i);
                if (key > 0) t.n_active = n + 1;
                ++n;
            }
    t.nj = (GLG_NX + GLG_NO - 1) / GLG_NO;
    for (; n < GLG_MAXROWS * GLG_NO; ++n) {
        t.order[n] = -1;
        t.scale_k[n] = -1;
    }
    t.row_base[0] = 0;
    for (int j = 0; j < GLG_MAXROWS; ++j) {
        int e = 0;
        for (int o = 0; o < GLG_NO; ++o) {
            const int st = j * GLG_NO + o < GLG_NX ? t.order[j * GLG_NO + o] : -1;
            if (st >= 0) e = wt.contribs[st] > e ? wt.contribs[st] : e;
        }
        t.row_slots[j] = e;
        t.row_base[j + 1] = t.row_base[j] + e;
    }
    t.n_slots = GLG_NO * t.row_base[t.nj];
    for (int w = 0; w < 16; ++w)
        for (int i = 0; i < GLG_NX; ++i) {
            t.slot[w][i] = -1;
            if (w < ng && (wt.states[w] >> i & 1u)) {
                int c = 0;  // contributing warps in front of w
                for (int ww = 0; ww < w; ++ww) c += (int)(wt.states[ww] >> i & 1u);
                const int r = t.rank[i], j = r / GLG_NO;
                t.slot[w][i] = (t.row_base[j] + c) * GLG_NO + r % GLG_NO;
            }
        }
    return t;
}
template <int NG, bool GENERAL>
struct GlgPlan {
    static constexpr GlgOwnerPlan plan = glg_make_plan(GlgWT<NG, GENERAL>::t, NG);
    static constexpr int NJ = plan.nj;
    static constexpr int NPART = plan.n_slots;
    static constexpr int CANSCALE = NPART;  // GlgSpecial fields
    static constexpr int LAMBDA = NPART + 1;
    static constexpr int AVENT = NPART + 2;
    static constexpr int ASCR = NPART + 3;
    static constexpr int DUMMY = NPART + 4;  // write-only slot (the cover's "far side" output in the shared surface role)
    static constexpr int NSLOTS = NPART + 5;
    static constexpr int XS_ROWS = NJ * GLG_NO;
    static constexpr int canopy_entry = plan.rank[4];  // its capacity scale changes with the stage LAI
};

template <int I>
struct GlgInt {
    static constexpr int value = I;
};
template <int I, int N, class F>
__device__ __forceinline__ void glg_static_for(F &&f) {
    if constexpr (I < N) {
        f(GlgInt<I>{});
        glg_static_for<I + 1, N>(f);
    }
}

template <class T, int NG, bool GENERAL>
struct GlgXsCol {  // stage-state column of this lane, rows in plan order
    const T *b;
    template <int I>
    __device__ __forceinline__ T at() const {
        constexpr int r = GlgPlan<NG, GENERAL>::plan.rank[I];
        return b[r * GLG_ROLE_LANES];
    }
};

// per-env-step constants of this lane copied to registers in front of a role's loop (indices are compile-time constants after
// inlining, so the array is scalarised and the entries the role never reads cost nothing)
template <class T, int N>
struct GlgRegCol {
    T v[N];
    __device__ __forceinline__ void load(const T *col) {
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = col[i * GLG_ROLE_LANES];
    }
    __device__ __forceinline__ T operator[](int i) const { return v[i]; }
};

template <class T, int NG, bool GENERAL, bool NOISY>
struct GlgRoleSmem {
    using PL = GlgPlan<NG, GENERAL>;
    static constexpr int kColRows = PL::XS_ROWS + PL::NSLOTS + H_COUNT + (NOISY ? C_COUNT : 0);
    // fp32 units: the step's start / end state crosses between warp 0 and the owners in fp64 through its own [28][32] block;
    // fp64 units: the stage-state block itself holds it (the last evaluation leaves the final state there)
    static constexpr int kXfinRows = sizeof(T) == sizeof(double) ? 0 : GLG_NX;
    // weather tile (f64) | fruit row, scale row, [state block] (f64) | T columns | mbarrier | ints
    __host__ __device__ static size_t col_bytes() { return (sizeof(T) * (size_t)kColRows * GLG_ROLE_LANES + 15) / 16 * 16; }
    __host__ __device__ static size_t bytes(int Np) {
        return sizeof(double) * ((size_t)(Np + 1) * GLG_ND + (size_t)(kXfinRows + 2) * GLG_ROLE_LANES) + col_bytes() + 16 +
               sizeof(int) * (5 * GLG_ROLE_LANES + 4 + 16);
    }
};

template <class T>
struct GlgKView;
template <>
struct GlgKView<double> {
    typedef GlgConstView type;
    __device__ __forceinline__ static type k(const GlgUniform &U) { return type{U.K}; }
    __device__ __forceinline__ static type c(const GlgUniform &U) { return type{U.C}; }
};
template <>
struct GlgKView<float> {
    typedef GlgConstViewF type;
    __device__ __forceinline__ static type k(const GlgUniform &U) { return type{U.Kf}; }
    __device__ __forceinline__ static type c(const GlgUniform &U) { return type{U.Cf}; }
};

// ---- one evaluation of the units of group warp W: stage state -> partial sums and specials in shared memory
// HV / CV: views of the per-env-step constants H and (NOISY) the per-env crop constants C: shared-memory columns or registers
template <int NG, int W, bool GENERAL, bool NOISY, class T, class HV, class CV>
__device__ __forceinline__ void glg_group_eval_v(const GlgUniform &U, const T *xs_col, T *part_col, const HV &Hc, const CV &Cc, const double *u) {
    using PL = GlgPlan<NG, GENERAL>;
    const typename GlgKView<T>::type Kv = GlgKView<T>::k(U);
    const GlgConstView Pv{U.P};
    const GlgXsCol<T, NG, GENERAL> X{xs_col};
    constexpr unsigned mask = GlgWT<NG, GENERAL>::t.states[W];
    T v[GLG_NX];
    GlgSpecial<T> sp;
    if constexpr (NOISY) glg_run_warp_units<NG, W, 0, GENERAL>(Kv, Cc, Hc, Pv, u, X, v, sp);
    else glg_run_warp_units<NG, W, 0, GENERAL>(Kv, GlgKView<T>::c(U), Hc, Pv, u, X, v, sp);
    glg_static_for<0, GLG_NX>([&](auto ic) {
        constexpr int i = decltype(ic)::value;
        if constexpr (mask >> i & 1u) {
            constexpr int sl = PL::plan.slot[W][i];
            part_col[sl * GLG_ROLE_LANES] = v[i];
        }
    });
    if constexpr (GlgWT<NG, GENERAL>::has_unit(W, U_PIPES)) part_col[PL::CANSCALE * GLG_ROLE_LANES] = sp.canscale;
    if constexpr (GlgWT<NG, GENERAL>::has_unit(W, U_MAINT)) part_col[PL::LAMBDA * GLG_ROLE_LANES] = sp.lambda;
    if constexpr (GlgWT<NG, GENERAL>::has_unit(W, U_VENT)) part_col[PL::AVENT * GLG_ROLE_LANES] = sp.avent;
    if constexpr (GlgWT<NG, GENERAL>::has_unit(W, U_SCR)) part_col[PL::ASCR * GLG_ROLE_LANES] = sp.ascr;
}
template <int NG, int W, bool GENERAL, bool NOISY, class T>
__device__ __forceinline__ void glg_group_eval(const GlgUniform &U, const T *xs_col, T *part_col, T *h_col, T *c_col, const double *u) {
    glg_group_eval_v<NG, W, GENERAL, NOISY, T>(U, xs_col, part_col, GlgColT<T, GLG_ROLE_LANES>{h_col}, GlgColT<T, GLG_ROLE_LANES>{c_col}, u);
}
// per-evaluation dispatch on the warp index (fused layout: one loop for all warps)
template <int NG, int W, bool GENERAL, bool NOISY, class T>
__device__ __forceinline__ void glg_group_eval_dispatch(int gw, const GlgUniform &U, const T *xs_col, T *part_col, T *h_col, T *c_col,
                                                        const double *u) {
    if constexpr (W + 1 < NG) {
        if (gw == W) glg_group_eval<NG, W, GENERAL, NOISY, T>(U, xs_col, part_col, h_col, c_col, u);
        else glg_group_eval_dispatch<NG, W + 1, GENERAL, NOISY, T>(gw, U, xs_col, part_col, h_col, c_col, u);
    } else {
        glg_group_eval<NG, W, GENERAL, NOISY, T>(U, xs_col, part_col, h_col, c_col, u);
    }
}

// ---- group role: the evaluation loop of group warp W (generic: any unit list).  The per-env-step constants are loop
// invariants: they are read from shared memory once, in front of the loop (the barriers' memory clobber would otherwise force a
// reload per evaluation: ~60 of the group warps' 139 shared-memory loads per evaluation, tools/sasssim).
template <int NG, int W, bool GENERAL, bool NOISY, class T>
__device__ __forceinline__ void glg_group_loop(const GlgUniform &U, const T *xs_col, T *part_col, T *h_col, T *c_col, const double *u,
                                               const volatile int *s_stop, int nthreads) {
    GlgRegCol<T, H_COUNT> Hr;
    Hr.load(h_col);
    GlgRegCol<T, NOISY ? C_COUNT : 1> Cr;
    if (NOISY) Cr.load(c_col);
    int last_eval;
    [[maybe_unused]] int ev = 0;
#pragma unroll 1
    do {
        glg_bar_sync<GLG_BAR_XS>(nthreads);
        GLG_TRACE_MARK(GLG_NO + W, 0, ev);
        // one flag per group warp (the load's immediate offset identifies the role in the SASS, tools/sasssim); read with the
        // stage state, consumed after the arrive: off the critical path
        last_eval = s_stop[W];
        glg_group_eval_v<NG, W, GENERAL, NOISY, T>(U, xs_col, part_col, Hr, Cr, u);
        GLG_TRACE_MARK(GLG_NO + W, 1, ev);
        ++ev;
        glg_bar_arrive(GLG_BAR_PARTS, nthreads);
    } while (!last_eval);
}

// ---- surface role: U_THSCR / U_BLSCR / U_COVER when each is alone in its warp.  One copy of glg_surface_core for the three
// warps; what differs (state rows, coefficient rows, output slots, vapour capacity scale) sits in registers.
template <int NG, bool GENERAL>
struct GlgSurfaceWarps {
    using WT = GlgWT<NG, GENERAL>;
    static constexpr int th = WT::unit_warp(U_THSCR), bl = WT::unit_warp(U_BLSCR), cv = WT::unit_warp(U_COVER);
    static constexpr bool alone(int w, int u) { return w >= 0 && WT::t.units[w] == (1u << u); }
    static constexpr bool shared = alone(th, U_THSCR) && alone(bl, U_BLSCR) && alone(cv, U_COVER);
};
template <int NG, bool GENERAL, int W>
struct GlgIsSurface {
    using SW = GlgSurfaceWarps<NG, GENERAL>;
    static constexpr bool value = SW::shared && (W == SW::th || W == SW::bl || W == SW::cv);
};
template <int NG, bool GENERAL, class T>
__device__ __forceinline__ void glg_surface_loop(int gw, const GlgUniform &U, const T *xs_col, T *part_col, const T *h_col,
                                                 const volatile int *s_stop, int nthreads) {
    using PL = GlgPlan<NG, GENERAL>;
    using SW = GlgSurfaceWarps<NG, GENERAL>;
    constexpr int NL = GLG_ROLE_LANES;
    const bool is_th = gw == SW::th, is_cv = gw == SW::cv;
    constexpr int w_th = SW::th >= 0 ? SW::th : 0, w_bl = SW::bl >= 0 ? SW::bl : 0, w_cv = SW::cv >= 0 ? SW::cv : 0;
    // A = air side (main air for the screens, top compartment for the cover), S = surface, B = far side, V = vapour pressure of A
    constexpr int r2 = PL::plan.rank[2], r3 = PL::plan.rank[3], r5 = PL::plan.rank[5], r7 = PL::plan.rank[7], r15 = PL::plan.rank[15],
                  r16 = PL::plan.rank[16], r20 = PL::plan.rank[20];
    constexpr int s_th7 = PL::plan.slot[w_th][7], s_th2 = PL::plan.slot[w_th][2], s_th3 = PL::plan.slot[w_th][3], s_th15 = PL::plan.slot[w_th][15];
    constexpr int s_bl20 = PL::plan.slot[w_bl][20], s_bl2 = PL::plan.slot[w_bl][2], s_bl3 = PL::plan.slot[w_bl][3], s_bl15 = PL::plan.slot[w_bl][15];
    constexpr int s_cv5 = PL::plan.slot[w_cv][5], s_cv3 = PL::plan.slot[w_cv][3], s_cv16 = PL::plan.slot[w_cv][16];
    const int xa = (is_cv ? r3 : r2) * NL;
    const int xsf = (is_cv ? r5 : is_th ? r7 : r20) * NL;
    const int xb = r3 * NL;  // the cover has no far side: its far coefficient is 0
    const int xv = (is_cv ? r16 : r15) * NL;
    const int ps = (is_cv ? s_cv5 : is_th ? s_th7 : s_bl20) * NL;
    const int pa = (is_cv ? s_cv3 : is_th ? s_th2 : s_bl2) * NL;
    const int pb = (is_cv ? PL::DUMMY : is_th ? s_th3 : s_bl3) * NL;
    const int pv = (is_cv ? s_cv16 : is_th ? s_th15 : s_bl15) * NL;
    const int ha = (is_cv ? (int)H_HECIN : is_th ? (int)H_17TH : (int)H_17BL) * NL;
    const int hb = (is_cv ? (int)H_ZERO : is_th ? (int)H_17TH : (int)H_17BL) * NL;
    const typename GlgKView<T>::type Kv = GlgKView<T>::k(U);
    const T invvp = is_cv ? Kv[K_INVVPTOP] : Kv[K_INVVPAIR];
    const T L = Kv[K_L];
    const volatile int *stop = s_stop + gw;
    const T coef_a = h_col[ha], coef_b = h_col[hb];  // loop invariants
    int last_eval;
    [[maybe_unused]] int ev = 0;
#pragma unroll 1
    do {
        glg_bar_sync<GLG_BAR_XS>(nthreads);
        GLG_TRACE_MARK(GLG_NO + gw, 0, ev);
        T surf, air, far, vp;
        last_eval = *stop;
        glg_surface_core<true, T>(xs_col[xa], xs_col[xsf], xs_col[xb], xs_col[xv], coef_a, coef_b, invvp, L, surf, air, far, vp);
        part_col[ps] = surf;
        part_col[pa] = air;
        part_col[pb] = far;
        part_col[pv] = vp;
        GLG_TRACE_MARK(GLG_NO + gw, 1, ev);
        ++ev;
        glg_bar_arrive(GLG_BAR_PARTS, nthreads);
    } while (!last_eval);
}

template <int NG, int W, bool GENERAL, bool NOISY, class T>
__device__ __forceinline__ void glg_group_dispatch(int gw, const GlgUniform &U, const T *xs_col, T *part_col, T *h_col, T *c_col,
                                                   const double *u, const volatile int *s_stop, int nthreads) {
    if constexpr (W < NG) {
        if constexpr (GlgIsSurface<NG, GENERAL, W>::value) {
            glg_group_dispatch<NG, W + 1, GENERAL, NOISY, T>(gw, U, xs_col, part_col, h_col, c_col, u, s_stop, nthreads);
        } else {
            if (gw == W) glg_group_loop<NG, W, GENERAL, NOISY, T>(U, xs_col, part_col, h_col, c_col, u, s_stop, nthreads);
            else glg_group_dispatch<NG, W + 1, GENERAL, NOISY, T>(gw, U, xs_col, part_col, h_col, c_col, u, s_stop, nthreads);
        }
    }
}

__constant__ double glg_kStageC[4] = {0.5, 0.5, 1.0, 1.0 / 6.0};
__constant__ double glg_kStageW[4] = {1.0, 2.0, 2.0, 1.0};

// ---- owner: RK4 state of the NJ plan rows of owner index o for this lane's env, and the micro-step bookkeeping.
// One nominal RK4 substep = m micro-steps of h_nom/m, m per env = max of the harvest-stiffness guard (glg_model.h; 1 unless an
// organ sits inside its harvest window) and, with integrator = 1, the graded start of the interval and the transient-stiffness
// rule.  Lanes with a smaller m idle with h = 0 for the remaining micro-steps of the CTA, so an env's result never depends on
// its CTA mates.
// Stage update in unscaled units: s = sum of the partial sums, k = scale * s.
//   stage 0..2: acc = (stage ? acc : 0) + w s ; xs = x + (c h scale) s        stage 3: x += (h/6 scale) (acc + s) ; xs = x
// One evaluation, in program order (the order matters: everything in front of the barrier wait is off the critical path,
// what follows it is the CTA's serial section behind its slowest group warp):
//   book()   : stage-sum / state / counter updates of the PREVIOUS evaluation
//   pre()    : (c h scale), the acc term of stage 3, the end-of-interval tests
//   reduce() : partial sums of the group warps -> pairwise tree per row, harvest guard
//   update() : micro-step count of a first evaluation, next stage state to shared memory
template <class T, int NG, bool GENERAL>
struct GlgOwner {
    using PL = GlgPlan<NG, GENERAL>;
    static constexpr int NJ = PL::NJ, NL = GLG_ROLE_LANES;
    static constexpr int can_row = PL::canopy_entry / GLG_NO;
    double xo[NJ], acc[NJ], scale[NJ];  // the RK4 state and stage sum stay fp64 in both precisions
    double hc[NJ], base[NJ], sum[NJ], xn[NJ];
    double h_nom, h_lane, cs, w, can_cs;
    int o, n_sub, graded, sub, q, stage, m_lane, m_cta, n_micro;
    bool can_owner, first, last, split_h;
    int final_eval, flag_next;

    // state index of row j of this owner (compile-time tables, runtime owner index)
    template <int J>
    __device__ __forceinline__ int row_state() const {
        constexpr int st0 = PL::plan.order[J * GLG_NO], st1 = PL::plan.order[J * GLG_NO + 1], st2 = PL::plan.order[J * GLG_NO + 2],
                      st3 = PL::plan.order[J * GLG_NO + 3];
        return o == 0 ? st0 : o == 1 ? st1 : o == 2 ? st2 : st3;
    }
    static constexpr bool kStateInXs = sizeof(T) == sizeof(double);  // see GlgRoleSmem::kXfinRows
    // book_first: the caller's loop runs book() at its top (of the previous evaluation), so the first call has nothing to book
    __device__ __forceinline__ void init(int owner, const GlgStepArgs &A, const double *s_xfin, const double *s_scale, const T *xs_col,
                                         int lane, bool book_first) {
        o = owner;
        glg_static_for<0, NJ>([&](auto jc) {
            constexpr int j = decltype(jc)::value;
            const int st = row_state<j>();
            scale[j] = s_scale[j * GLG_NO + o];
            if (kStateInXs) xo[j] = (double)xs_col[(j * GLG_NO + o) * NL];
            else xo[j] = st >= 0 ? s_xfin[st * NL + lane] : 0.0;
            acc[j] = 0.0;
            sum[j] = 0.0;
            xn[j] = xo[j];
        });
        can_owner = o == PL::canopy_entry % GLG_NO;
        h_nom = A.dt / (double)A.n_sub;
        n_sub = A.n_sub;
        graded = A.integrator == 1;
        glg_pin(h_nom);  // kept in registers: ptxas otherwise re-reads the kernel parameters inside the loop
        glg_pin(n_sub);
        glg_pin(graded);
        sub = q = n_micro = 0;
        stage = book_first ? -1 : 0;  // a leading book() has nothing to book: w = 0, sum = 0
        w = 0.0;
        last = false;
        m_lane = m_cta = 1;
        h_lane = h_nom;
    }
    __device__ __forceinline__ void book() {
#pragma unroll
        for (int j = 0; j < NJ; ++j) acc[j] = glg_fma(w, sum[j], acc[j]);
        if (last) {
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                xo[j] = xn[j];
                acc[j] = 0.0;
            }
        }
        if (++stage == 4) {
            stage = 0;
            if (++q >= m_cta) {
                q = 0;
                ++sub;
            }
        }
    }
    __device__ __forceinline__ void pre(int lane) {
        first = stage == 0 && q == 0;  // first evaluation of a nominal substep: the micro-step count is decided in update()
        last = stage == 3;
        cs = glg_kStageC[stage];  // 1/2, 1/2, 1, 1/6 : constant-bank lookups instead of select chains (loop code size)
        w = glg_kStageW[stage];   // 1, 2, 2, 1
        // is this the last evaluation of the interval?  (m_cta of the last substep is known by its stage 3)
        const bool last_micro = q + 1 >= m_cta && sub + 1 >= n_sub;
        final_eval = last && last_micro;
        flag_next = stage == 2 && last_micro && o == 0 && lane < 16;  // the group warps' next evaluation is the last one
        // speculate m = 1 for a first evaluation (true except at the graded start of an interval and in stiff transients)
        const double hcs = cs * (first ? h_nom : (q < m_lane ? h_lane : 0.0));
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            hc[j] = hcs * scale[j];
            base[j] = xo[j];
        }
        if (last) {
#pragma unroll
            for (int j = 0; j < NJ; ++j) base[j] = glg_fma(hc[j], acc[j], xo[j]);
        }
    }
    // pairwise tree over n slots of row J starting at slot index s0 (in units of NO * NL elements)
    template <int N>
    __device__ __forceinline__ static double tree(const T *p0) {
        double v[N];
#pragma unroll
        for (int c = 0; c < N; ++c) v[c] = (double)p0[c * GLG_NO * NL];
#pragma unroll
        for (int s = 1; s < N; s *= 2)
#pragma unroll
            for (int c = 0; c + s < N; c += 2 * s) v[c] += v[c + s];
        return v[0];
    }
    __device__ __forceinline__ void reduce(const T *part_col) {
        const T *pbase = part_col + o * NL;  // row j, contribution c at pbase[(row_base[j] + c) * NO * NL]
        glg_static_for<0, NJ>([&](auto jc) {
            constexpr int j = decltype(jc)::value;
            constexpr int n = PL::plan.row_slots[j];
            constexpr int rb = PL::plan.row_base[j];
            if constexpr (n == 0) sum[j] = 0.0;
            else sum[j] = tree<n>(pbase + rb * GLG_NO * NL);
        });
        // the canopy's capacity scale K_INVCAPLEAF / LAI changes with the stage (its scale[] entry is 1)
        can_cs = can_owner ? (double)part_col[PL::CANSCALE * NL] : 1.0;
        sum[can_row] *= can_cs;
        // harvest guard: m = 1 unless an organ is inside its harvest window (2 h lambda >= 1)
        split_h = first && (2.0 * h_nom * (double)part_col[PL::LAMBDA * NL] >= 1.0);
    }
    __device__ __forceinline__ void update(const GlgUniform &U, const T *part_col, T *xs_col) {
        T *xbase = xs_col + o * NL;  // row j at xbase[j * NO * NL]
        if (first) {
            // m = 1 for every env of the CTA unless a harvest window is active, the graded integrator is at the start of the
            // interval or its stiffness rule asks for a split: one vote on the common path
            double lam_s = 0.0;
            if (graded) lam_s = glg_stiffness(GlgConstView{U.K}, (double)part_col[PL::ASCR * NL], (double)part_col[PL::AVENT * NL]);
            const bool split = split_h || (graded && (sub < GLG_GRADED_SUBSTEPS || h_nom * lam_s * GLG_STIFF_INV_CFL >= 1.0));
            m_lane = 1;
            m_cta = 1;
            h_lane = h_nom;
            if (__any_sync(0xffffffffu, split)) {
                m_lane = glg_micro_steps_from_lambda((double)part_col[PL::LAMBDA * NL], h_nom);
                if (graded) {
                    int ms = 1 + (int)floor(h_nom * lam_s * GLG_STIFF_INV_CFL);
                    ms = ms > GLG_MAX_MICRO ? GLG_MAX_MICRO : (ms < 1 ? 1 : ms);  // ms < 1 only for a NaN estimate
                    if (ms < glg_graded_m(sub)) ms = glg_graded_m(sub);
                    m_lane = max(m_lane, ms);
                }
                m_cta = __reduce_max_sync(0xffffffffu, m_lane);  // every owner warp sees the same 32 envs
                // reciprocal + multiply instead of an IEEE division; the step size differs from h_nom/m by at most 1 ulp
                h_lane = m_lane == 1 ? h_nom : h_nom * glg_rcp((double)m_lane);
                // redo the stage update with the right step (first evaluation: stage 0, base = x)
                const double hcs = cs * h_lane;
#pragma unroll
                for (int j = 0; j < NJ; ++j) hc[j] = hcs * scale[j];
            }
            n_micro += m_lane;
        }
        // one copy of the stage update for all paths (the loop code must stay below the instruction cache)
#pragma unroll
        for (int j = 0; j < NJ; ++j) xn[j] = glg_fma(hc[j], sum[j], base[j]);
#pragma unroll
        for (int j = 0; j < NJ; ++j) xbase[j * GLG_NO * NL] = (T)xn[j];
    }
    // final state (xn of the last evaluation: the caller leaves its loop right behind that update()) -> s_xfin; returns 1 if
    // any of this owner's states is not finite
    __device__ __forceinline__ int finish(double *s_xfin, int lane) const {
        int bad = 0;
        glg_static_for<0, NJ>([&](auto jc) {
            constexpr int j = decltype(jc)::value;
            const int st = row_state<j>();
            bad |= !(fabs(xn[j]) <= 1.79769313486231570e308);
            if (!kStateInXs && st >= 0) s_xfin[st * NL + lane] = xn[j];  // fp64 units: update() left it in the stage-state block
        });
        return bad;
    }
};


// Two layouts of the same machinery:
//   FUSED = false (latency layout, small batches): NG group warps + GLG_NO dedicated owner warps per 32 envs, every role in its
//           own loop, producer/consumer named barriers.  The step time of a batch that leaves SMs under-filled is the latency of
//           one CTA, so the RHS is spread over as many warps as balance allows (NG = 12).
//   FUSED = true (throughput layout, large batches): NG = GLG_NO = 4 warps per 32 envs; warp w evaluates the units of group
//           warp w AND owns the plan rows of owner w (dedicated owner warps would idle most of the time and hold a quarter of the
//           registers); one loop, two CTA barriers per evaluation, 4 CTAs per SM so that every SM sub-partition runs ONE role's
//           code for four CTAs.  Compared with the round-1 kernel the owner side keeps only the RK4 state in registers (all
//           addresses are immediates of the rank-ordered layout), so the unit code has ~95 registers for interleaving.
template <bool FUSED>
struct GlgLayout {
    static constexpr int NG = FUSED ? GLG_NO : 12;           // group warps per 32 envs
    static constexpr int MINB = FUSED ? 4 : 1;               // CTAs per SM the register budget is sized for
    static constexpr int NT = 32 * (NG + (FUSED ? 0 : GLG_NO));  // threads per CTA
};
template <class T, bool GENERAL, bool NOISY, bool FUSED>
__global__ void __launch_bounds__(GlgLayout<FUSED>::NT, GlgLayout<FUSED>::MINB) glg_step_units_kernel(const __grid_constant__ GlgUniform U,
                                                                                                       const __grid_constant__ GlgStepArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    glg_exp_tbl_fill();
    constexpr int NL = GLG_ROLE_LANES;
    constexpr int NG = GlgLayout<FUSED>::NG, NT = GlgLayout<FUSED>::NT;
    using PL = GlgPlan<NG, GENERAL>;
    using SW = GlgSurfaceWarps<NG, GENERAL>;
    constexpr int NJ = PL::NJ;
    double *s_wtile = reinterpret_cast<double *>(smem_raw);  // [(Np+1)][10] f64
    constexpr int kXfinRows = GlgRoleSmem<T, NG, GENERAL, NOISY>::kXfinRows;
    constexpr bool kStateInXs = kXfinRows == 0;
    double *s_fruit = s_wtile + (size_t)(A.Np + 1) * GLG_ND;  // [32] fruit mass before the step (reward)
    double *s_scale = s_fruit + NL;                            // [XS_ROWS] capacity scale of plan entry n
    double *s_xfin = s_scale + NL;                             // fp32 units only: [28][32] f64, state order: state in / final state out
    T *s_xs = reinterpret_cast<T *>(s_xfin + kXfinRows * NL);  // [XS_ROWS][32] stage state in the units' precision, plan order
    T *s_part = s_xs + PL::XS_ROWS * NL;                      // [NSLOTS][32]: partial sums, specials
    T *s_H = s_part + PL::NSLOTS * NL;                        // [H_COUNT][32]
    T *s_C = s_H + H_COUNT * NL;                              // [C_COUNT][32] (NOISY)
    uint64_t *s_bar = reinterpret_cast<uint64_t *>(reinterpret_cast<unsigned char *>(s_xs) + GlgRoleSmem<T, NG, GENERAL, NOISY>::col_bytes());
    int *s_tbl = reinterpret_cast<int *>(s_bar + 2);
    int *s_k = s_tbl + NL;
    int *s_tbl_t = s_k + NL;
    int *s_k_t = s_tbl_t + NL;
    int *s_bad = s_k_t + NL;
    int *s_misc = s_bad + NL;            // [0..1] weather staging, [2] uniform weather, [3] 0
    volatile int *s_stop = s_misc + 4;   // [16] stop flag, one copy per group warp

    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    // a CTA owns A.role_lanes (<= 32) consecutive envs; lanes beyond that are padding
    const int e = blockIdx.x * A.role_lanes + lane;
    const bool active = lane < A.role_lanes && e < A.B;
    int k = 0, tbl = 0;
    if (active) {
        k = A.timestep[e];
        tbl = A.table[e];
    }
    const int kw = min(k, A.rows - A.Np - 1);
    int bk, bt;
    const int uniform = glg_stage_weather(A, s_wtile, s_bar, s_misc, active, kw, tbl, bk, bt);
    const double *wrow = uniform ? s_wtile : (A.weather + ((size_t)tbl * A.rows + (size_t)kw) * GLG_ND);

    // ---- prologue: warp 0, lane = env; the other warps clear the exchange slots (padding slots must read 0.0)
    double u[GLG_NU], d[GLG_ND];
#pragma unroll
    for (int i = 0; i < GLG_NU; ++i) u[i] = 0.0;
    double fruit_prev = 0.0;
    unsigned int ctr = 0;
    GlgColT<T, NL> Hc{s_H + lane};
    GlgColT<T, NL> Cc{s_C + lane};
    if (warp == 0) {
        double x[GLG_NX];
        if (active) {
            ctr = A.step_ctr[e];
            glg_env_prologue<NOISY>(U, A, e, wrow, ctr, Hc, Cc, x, u, d);
            fruit_prev = x[25];
        } else {
            // padding lanes integrate a copy of a benign state so every warp runs the same loop
            double d0[GLG_ND];
#pragma unroll
            for (int i = 0; i < 7; ++i) d0[i] = A.weather[i];
            glg_init_state(d0, x);
            if (NOISY) {
#pragma unroll
                for (int i = 0; i < C_COUNT; ++i) Cc[i] = (T)U.C[i];
            }
            glg_hoist(GlgConstView{U.P}, u, d0, Hc);
        }
        glg_static_for<0, GLG_NX>([&](auto ic) {
            constexpr int i = decltype(ic)::value;
            constexpr int r = PL::plan.rank[i];
            s_xs[r * NL + lane] = (T)x[i];
            if (!kStateInXs) s_xfin[i * NL + lane] = x[i];
        });
        // what the epilogue needs goes through shared memory, so that nothing of it stays in registers across the loops
        s_fruit[lane] = fruit_prev;
        s_k[lane] = k;
        s_tbl[lane] = tbl;
        s_bad[lane] = 0;
        if (lane < 16) s_stop[lane] = 0;
        if (lane < PL::XS_ROWS) {
            int sk = -1;
            glg_static_for<0, PL::XS_ROWS>([&](auto nc) {
                constexpr int n = decltype(nc)::value;
                constexpr int v = PL::plan.scale_k[n];
                sk = lane == n ? v : sk;
            });
            s_scale[lane] = sk >= 0 ? U.K[sk] : 1.0;  // -1: the units wrote a derivative; -2 (canopy): scaled per stage in the loop
        }
        if (lane == 0) {
            s_misc[2] = uniform;
            s_misc[3] = 0;  // read by nothing; without this store ptxas allocates the registers of every variant differently
        }
    } else {
        for (int i = tid - 32; i < PL::NSLOTS * NL; i += NT - 32) s_part[i] = (T)0;
    }
    __syncthreads();

    T *xs_col = s_xs + lane;
    T *part_col = s_part + lane;
    int n_micro = 0;  // RK4 micro-steps this env executed (owner warp 0 counts)
    if (FUSED) {
        // ---- fused layout: every warp is group warp `warp` and owner `warp`
        if (GENERAL && active && warp == GlgWT<NG, GENERAL>::unit_warp(U_FIR)) {
#pragma unroll
            for (int i = 0; i < GLG_NU; ++i) u[i] = A.u[(size_t)i * A.B + e];
        }
        GlgOwner<T, NG, GENERAL> own;
        own.init(warp, A, s_xfin, s_scale, xs_col, lane, false);
#pragma unroll 1
        for (;;) {
            glg_group_eval_dispatch<NG, 0, GENERAL, NOISY, T>(warp, U, xs_col, part_col, s_H + lane, s_C + lane, u);
            own.pre(lane);
            __syncthreads();
            own.reduce(part_col);
            own.update(U, part_col, xs_col);
            if (own.final_eval) break;
            own.book();  // in front of the barrier: measured 13 % faster at B = 262 144 than at the top of the loop (more spills there)
            __syncthreads();
        }
        n_micro = own.n_micro;
        if (own.finish(s_xfin, lane)) s_bad[lane] = 1;  // benign race: every writer stores 1
    } else if (warp >= GLG_NO) {
        // ---- group warps
        const int gw = warp - GLG_NO;
        if (GENERAL && active && gw == GlgWT<NG, GENERAL>::unit_warp(U_FIR)) {
            // U_FIR's general terms read the raw screen controls; warp 0's prologue stored the updated controls before the barrier
#pragma unroll
            for (int i = 0; i < GLG_NU; ++i) u[i] = A.u[(size_t)i * A.B + e];
        }
        if (SW::shared && (gw == SW::th || gw == SW::bl || gw == SW::cv)) glg_surface_loop<NG, GENERAL, T>(gw, U, xs_col, part_col, s_H + lane, s_stop, NT);
        else glg_group_dispatch<NG, 0, GENERAL, NOISY, T>(gw, U, xs_col, part_col, s_H + lane, s_C + lane, u, s_stop, NT);
    } else {
        // ---- owner warps (GlgOwner)
        GlgOwner<T, NG, GENERAL> own;
        own.init(warp, A, s_xfin, s_scale, xs_col, lane, true);
        glg_bar_arrive(GLG_BAR_XS, NT);  // the prologue's stage state is in shared memory: release the group warps' first evaluation
        [[maybe_unused]] int ev = 0;
#pragma unroll 1
        for (;;) {
            own.book();
            own.pre(lane);
            glg_bar_sync<GLG_BAR_PARTS>(NT);
            own.reduce(part_col);
            GLG_TRACE_MARK(warp, 0, ev);
            own.update(U, part_col, xs_col);
            if (own.final_eval) break;
            if (own.flag_next) s_stop[lane] = 1;
            GLG_TRACE_MARK(warp, 1, ev);
            ++ev;
            glg_bar_arrive(GLG_BAR_XS, NT);
        }
        n_micro = own.n_micro;
        const int bad = own.finish(s_xfin, lane);
        if (bad) s_bad[lane] = 1;  // benign race: every writer stores 1
    }
    __syncthreads();

    // ---- epilogue: warp 0, lane = env
    const int uniform2 = s_misc[2], bk2 = s_misc[0], bt2 = s_misc[1];
    if (warp == 0) {
        const int e = blockIdx.x * A.role_lanes + lane;
        const bool active = lane < A.role_lanes && e < A.B;
        const int k = s_k[lane], tbl = s_tbl[lane];
        const int kw = min(k, A.rows - A.Np - 1);
        const double *wrow = uniform2 ? s_wtile : (A.weather + ((size_t)tbl * A.rows + (size_t)kw) * GLG_ND);
        GlgEnvOut o;
        o.done = 0; o.k_obs = -1; o.tbl_obs = 0; o.k_term = -1; o.tbl_term = 0; o.fin_ret = 0.0; o.fin_len = 0.0;
#pragma unroll
        for (int j = 0; j < GLG_NINFO; ++j) o.fin_info[j] = 0.0;
        const int bad = s_bad[lane];
        if (active) {
            double x[GLG_NX];
            glg_static_for<0, GLG_NX>([&](auto ic) {
                constexpr int i = decltype(ic)::value;
                constexpr int r = PL::plan.rank[i];
                x[i] = kStateInXs ? (double)s_xs[r * NL + lane] : s_xfin[i * NL + lane];
            });
            glg_env_epilogue(U, A, e, k, kw, tbl, wrow, x, s_fruit[lane], bad, A.step_ctr[e], o);
        }
        s_tbl[lane] = o.tbl_obs;
        s_k[lane] = o.k_obs;
        s_tbl_t[lane] = o.tbl_term;
        s_k_t[lane] = o.k_term;
        glg_stats_reduce(A, active, bad, o);
        const int tot = __reduce_add_sync(0xffffffffu, active ? n_micro : 0);
        if (lane == 0 && tot > 0) atomicAdd(&A.stats[15], (double)tot);
    }
    __syncthreads();
    glg_write_forecast(A, A.role_lanes, s_tbl, s_k, s_tbl_t, s_k_t, s_wtile, uniform2, bk2, bt2);
}
