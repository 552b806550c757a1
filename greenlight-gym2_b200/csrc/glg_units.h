// glg_units.h -- the GreenLight right-hand side cut into 13 flux UNITS for the warp-specialised step kernel (glg_roles.cuh).
//
// Same physics as glg_rhs (glg_model.h; reference update() aux_states.hpp:96-1271 and ODE() ode.hpp:6-124), different shape:
// a unit is a set of fluxes that shares its expensive intermediates (a cube root, a saturation pressure, an air flux ...)
// with no other unit, so units can be evaluated by different warps for the same 32 envs without exchanging anything inside
// one evaluation.  Every unit adds its contribution to the balance of each state it touches through `pt.put<i>(v)`; a warp
// that runs several units sums them in registers (GlgAccum) and stores ONE partial sum per (warp, state); the state's owner
// adds the partial sums of the contributing warps and applies the capacity scale.  The unit -> warp assignment is a
// compile-time table (glg_assign), so the same code gives an 8-, 12- or 13-warp split.
//
//   U_OPT    canopy PAR / NIR extinction and multilayer absorption (:299-470)
//   U_PIPES  pipe and grow-pipe convection (two x^0.32 powers, :906-930), slow linear states 21, 26, 27, canopy capacity scale
//   U_FIR    all FIR exchange (:493-632), cover conduction, cover-outside convection, boiler / lamp net input, soil chain
//   U_VENT   roof ventilation (:733-771): CO2 / heat / vapour exchange with outside through the roof and by leakage
//   U_SCR    air flux through the screens (:787-814): CO2 / heat / vapour exchange main air <-> top compartment
//   U_FLOOR  lamp, canopy and floor convection with the main air (:824-935)
//   U_THSCR  thermal screen: convection on both sides + condensation (:835-848, :999-1002)
//   U_BLSCR  blackout screen: convection on both sides + condensation (:852-861, :1003-1005)
//   U_COVER  top compartment -> cover convection + condensation (:866, :1011)
//   U_TRANSP canopy transpiration (:959-981)
//   U_PHOTO  canopy photosynthesis -> buffer inflow (:1041-1097)
//   U_FLOWS  carbohydrate flows buffer -> organs and growth respiration (:1103-1155)
//   U_MAINT  maintenance respiration and harvest (:1161-1188); returns the harvest speed for the micro-step guard
//
// Valid C++ for g++ too: tests/hostmath assembles the RHS from the units on the host and checks it against the oracle.
#pragma once
#include "glg_model.h"

// Scalar type of the units: the stage state's type when it is a tangent type (GlgDual: K, C and p stay plain doubles, so
// constants cost no tangent arithmetic), else the constant sets' type (double in parity mode, float in throughput mode).
template <class XV>
using glg_x_scalar_t = typename std::decay<decltype(std::declval<const XV &>().template at<0>())>::type;
template <class KV, class XV>
using glg_unit_t = typename std::conditional<glg_is_dual<glg_x_scalar_t<XV>>::value, glg_x_scalar_t<XV>, glg_scalar_t<KV>>::type;

enum GlgUnitId { U_OPT, U_PIPES, U_FIR, U_VENT, U_SCR, U_FLOOR, U_THSCR, U_BLSCR, U_COVER, U_TRANSP, U_PHOTO, U_FLOWS, U_MAINT, U_COUNT };

// states unit u contributes to (bit i = state i).  GENERAL adds the interlight node 18 and the grow-pipe FIR term.
GLG_HD constexpr unsigned glg_unit_states(int u, bool general) {
    return u == U_OPT    ? (1u << 4 | 1u << 8 | 1u << 2)
         : u == U_PIPES  ? (1u << 9 | 1u << 19 | 1u << 2 | 1u << 21 | 1u << 26 | 1u << 27)
         : u == U_FIR    ? (1u << 4 | 1u << 5 | 1u << 6 | 1u << 7 | 1u << 8 | 1u << 9 | 0x7C00u /*10..14*/ | 1u << 17 | 1u << 20 |
                            (general ? (1u << 18 | 1u << 19) : 0u))
         : u == U_VENT   ? (1u << 0 | 1u << 1 | 1u << 2 | 1u << 3 | 1u << 15 | 1u << 16)
         : u == U_SCR    ? (1u << 0 | 1u << 1 | 1u << 2 | 1u << 3 | 1u << 15 | 1u << 16)
         : u == U_FLOOR  ? (1u << 2 | 1u << 4 | 1u << 8 | 1u << 17 | (general ? 1u << 18 : 0u))
         : u == U_THSCR  ? (1u << 7 | 1u << 2 | 1u << 3 | 1u << 15)
         : u == U_BLSCR  ? (1u << 20 | 1u << 2 | 1u << 3 | 1u << 15)
         : u == U_COVER  ? (1u << 5 | 1u << 3 | 1u << 16)
         : u == U_TRANSP ? (1u << 4 | 1u << 15)
         : u == U_PHOTO  ? (1u << 22 | 1u << 0)
         : u == U_FLOWS  ? (1u << 22 | 1u << 23 | 1u << 24 | 1u << 25 | 1u << 0)
         : u == U_MAINT  ? (1u << 23 | 1u << 24 | 1u << 25 | 1u << 0)
                         : 0u;
}

// values that are not balance contributions: written to dedicated slots by the unit that has them
template <class T>
struct GlgSpecial {
    T canscale;  // U_PIPES: K_INVCAPLEAF / LAI, the capacity scale of the canopy state 4 at this stage
    T lambda;    // U_MAINT: harvest speed in sigmoid window-widths per second (micro-step guard)
    T avent;     // U_VENT : |roof ventilation flux|        } transient-stiffness estimate of the graded integrator
    T ascr;      // U_SCR  : |air flux through the screens| }
};

// accumulate-in-registers contribution sink: PRIOR = states already written by earlier units of the same warp
template <class T, unsigned PRIOR>
struct GlgAccum {
    T *v;
    template <int I>
    GLG_HD void put(T val) const {
        if (PRIOR >> I & 1u) v[I] += val;
        else v[I] = val;
    }
};

// two x^e powers with their log / exp chains interleaved in source order
template <class T>
GLG_HD void glg_pow2(T b0, T b1, T e, T &y0, T &y1) {
    y0 = glg_pow(b0, e);
    y1 = glg_pow(b1, e);
}

// ---------------------------------------------------------------------------------------------------------
// stage-state access with a compile-time index: the kernel keeps the stage state in owner-plan order in shared memory
#define GLG_X(x, I) ((x).template at<(I)>())
struct GlgArrayX {  // plain array in state order (host tests, kernel A style callers)
    const double *p;
    template <int I>
    GLG_HD double at() const { return p[I]; }
};

template <bool GENERAL, class KV, class CV, class HV, class XV, class PT>
GLG_HD void glg_unit_opt(const KV &K, const CV &C, const HV &H, const XV &x, const PT &pt) {
    typedef glg_unit_t<KV, XV> T;
    const T lai = C[C_SLA] * GLG_X(x, 23);
    const T ea[3] = {-K[K_K1PAR] * lai, -K[K_KNIR] * lai, -K[K_K2PAR] * lai};
    T ey[3];
    if (GENERAL) {
        glg_exp_n<3>(ea, ey);
    } else {  // k1Par == k2Par in the nominal structure
        const T ea2[2] = {ea[0], ea[1]};
        T ey2[2];
        glg_exp_n<2>(ea2, ey2);
        ey[0] = ey2[0]; ey[1] = ey2[1]; ey[2] = ey2[0];
    }
    const T e32 = ey[0], e34 = ey[1], e33 = ey[2];
    const T gPar = (1 - e32) + e32 * K[K_RHOFLRPAR] * (1 - e33);
    const T parLampCanW = H[H_PARLAMP_W] * gPar;
    const T parLampFlrW = H[H_PARLAMPFLR_W] * e32;
    const T rhoCovNir = H[H_RHOCOVNIR];
    const T rhoHat = K[K_RHOCANNIR] * (1 - e34);
    const T den1 = glg_rcp(T(1.) - rhoCovNir * rhoHat);
    const T tCC = H[H_TAUHATCOVNIR] * e34 * den1;
    const T rUp = rhoCovNir + H[H_TAUHAT2] * rhoHat * den1;
    const T rDn = rhoHat + e34 * e34 * rhoCovNir * den1;
    const T den2 = glg_rcp(T(1.) - rDn * K[K_RHOFLRNIR]);
    const T aFlrNir = tCC * K[K_TAUHATFLRNIR] * den2;
    const T rCCF = rUp + tCC * tCC * K[K_RHOFLRNIR] * den2;
    const T aCanNir = 1 - aFlrNir - rCCF;
    const T nirLampCan = H[H_NIRLAMPCAN] * (1 - e34), nirLampFlr = H[H_NIRLAMPFLR] * e34;
    pt.template put<4>(H[H_PARCAN_W] * gPar + H[H_NIRSUN] * aCanNir + nirLampCan);
    pt.template put<8>(H[H_PARFLR_W] * e32 + H[H_NIRSUN] * aFlrNir + nirLampFlr);
    pt.template put<2>((H[H_LAMPRAD] - parLampCanW - nirLampCan - parLampFlrW - nirLampFlr) +
                       (H[H_GLOBAIR_A] + H[H_GLOBAIR_B] * (aCanNir + aFlrNir)));
}

template <class KV, class CV, class XV, class PT>
GLG_HD void glg_unit_pipes(const KV &K, const CV &C, const XV &x, const PT &pt, GlgSpecial<glg_unit_t<KV, XV>> &sp) {
    typedef glg_unit_t<KV, XV> T;
    const T tAir = GLG_X(x, 2), tCan = GLG_X(x, 4), tPipe = GLG_X(x, 9), tGroPipe = GLG_X(x, 19);
    pt.template put<21>((T(1.) / T(86400.)) * (tCan - GLG_X(x, 21)));
    pt.template put<26>((T(1.) / T(86400.)) * tCan);
    pt.template put<27>(T(1.) / T(86400.));
    T pwP, pwG;
    glg_pow2(fabs(tPipe - tAir + T(1e-10)), fabs(tGroPipe - tAir + T(1e-10)), T(0.32), pwP, pwG);
    const T hPipeAir = fabs(K[K_PIPEAIR]) * pwP * (tPipe - tAir);
    const T hGroPipeAir = fabs(K[K_GROPIPEAIR]) * pwG * (tGroPipe - tAir);
    pt.template put<9>(-hPipeAir);
    pt.template put<19>(-hGroPipeAir);
    pt.template put<2>(hPipeAir + hGroPipeAir);
    sp.canscale = K[K_INVCAPLEAF] * glg_rcp(C[C_SLA] * GLG_X(x, 23));
}

template <bool GENERAL, class KV, class CV, class HV, class P, class UT, class XV, class PT>
GLG_HD void glg_unit_fir(const KV &K, const CV &C, const HV &H, const P &p, const UT *u, const XV &x, const PT &pt) {
    typedef glg_unit_t<KV, XV> T;
    const T tCan = GLG_X(x, 4), tCovIn = GLG_X(x, 5), tCovE = GLG_X(x, 6), tThScr = GLG_X(x, 7), tFlr = GLG_X(x, 8), tPipe = GLG_X(x, 9);
    const T tLamp = GLG_X(x, 17), tBlScr = GLG_X(x, 20);
    const T lai = C[C_SLA] * GLG_X(x, 23);
    const T e35 = glg_exp(-K[K_KFIR] * lai);
    const T aCan = 1 - e35;
    T sCan, sFlr, sCovIn, sThScr, sBlScr, sPipe, sLamp, sCovE;
    const T q4Can = glg_sq(glg_sq(tCan + T(GLG_C2K))), q4CovIn = glg_sq(glg_sq(tCovIn + T(GLG_C2K)));
    const T q4ThScr = glg_sq(glg_sq(tThScr + T(GLG_C2K))), q4Flr = glg_sq(glg_sq(tFlr + T(GLG_C2K)));
    const T q4Pipe = glg_sq(glg_sq(tPipe + T(GLG_C2K))), q4Lamp = glg_sq(glg_sq(tLamp + T(GLG_C2K)));
    const T q4BlScr = glg_sq(glg_sq(tBlScr + T(GLG_C2K)));
    T f;
    f = aCan * H[H_C84] * (q4Can - q4CovIn);   sCan = -f; sCovIn = f;
    f = aCan * H[H_C86] * (q4Can - q4ThScr);   sCan -= f; sThScr = f;
    f = aCan * K[K_C87] * (q4Can - q4Flr);     sCan -= f; sFlr = f;
    f = aCan * H[H_C108] * (q4Can - q4BlScr);  sCan -= f; sBlScr = f;
    f = aCan * K[K_C92] * (q4Pipe - q4Can);    sCan += f; sPipe = H[H_HBOIL] - f;
    f = aCan * K[K_C101] * (q4Lamp - q4Can);   sCan += f; sLamp = H[H_LAMPNET] - f;
    f = e35 * H[H_C88] * (q4Pipe - q4CovIn);   sPipe -= f; sCovIn += f;
    f = e35 * H[H_C90] * (q4Pipe - q4ThScr);   sPipe -= f; sThScr += f;
    f = e35 * H[H_C93] * (q4Flr - q4CovIn);    sFlr -= f; sCovIn += f;
    f = e35 * H[H_C95] * (q4Flr - q4ThScr);    sFlr -= f; sThScr += f;
    f = e35 * K[K_C99] * (q4Lamp - q4Flr);     sLamp -= f; sFlr += f;
    f = e35 * K[K_C100] * (q4Lamp - q4Pipe);   sLamp -= f; sPipe += f;
    f = e35 * H[H_C106] * (q4Flr - q4BlScr);   sFlr -= f; sBlScr += f;
    f = e35 * H[H_C107] * (q4Pipe - q4BlScr);  sPipe -= f; sBlScr += f;
    f = K[K_C91] * (q4Pipe - q4Flr);           sPipe -= f; sFlr += f;
    f = H[H_C96] * (q4ThScr - q4CovIn);        sThScr -= f; sCovIn += f;
    f = H[H_C102] * (q4Lamp - q4ThScr);        sLamp -= f; sThScr += f;
    f = H[H_C103] * (q4Lamp - q4CovIn);        sLamp -= f; sCovIn += f;
    f = H[H_C109] * (q4BlScr - q4ThScr);       sBlScr -= f; sThScr += f;
    f = H[H_C110] * (q4BlScr - q4CovIn);       sBlScr -= f; sCovIn += f;
    f = H[H_C112] * (q4Lamp - q4BlScr);        sLamp -= f; sBlScr += f;
    sCovE = H[H_GLOBCOV] - K[K_C98] * (glg_sq(glg_sq(tCovE + T(GLG_C2K))) - H[H_TSKY4]);
    if (GENERAL) {
        // Terms that are identically zero for the default table: sky FIR through the roof (tauRfFir p70),
        // grow-pipe FIR (epsGroPipe p165), interlight FIR (p194,p195).  Written plainly.
        const T sigma = p[2];
        const T pi = T(3.14159265358979323846);
        const T thScr = u[2], blScr = u[5];
        const T tauCovFir = p[70];
        const T tauThFir = 1 - thScr * (1 - p[81]), tauBlFir = 1 - blScr * (1 - p[91]);
        const T fPipe = T(0.49) * pi * p[107] * p[105];
        const T q4Sky = H[H_TSKY4];
        const T q4Int = glg_sq(glg_sq(GLG_X(x, 18) + T(GLG_C2K))), q4Gro = glg_sq(glg_sq(GLG_X(x, 19) + T(GLG_C2K)));
        const T f85 = aCan * p[3] * p[4] * (p[178] * tauCovFir * tauThFir * tauBlFir) * sigma * (q4Can - q4Sky);
        const T f89 = p[124] * p[104] * p[4] * (p[199] * p[178] * tauCovFir * tauThFir * T(0.49) * e35) * sigma * (q4Pipe - q4Sky);
        const T f94 = p[95] * p[4] * (p[199] * p[178] * tauCovFir * tauThFir * tauBlFir * (1 - fPipe) * e35) * sigma * (q4Flr - q4Sky);
        const T f97 = p[74] * p[4] * (tauCovFir * thScr) * sigma * (q4ThScr - q4Sky);
        const T f104 = p[181] * p[182] * p[4] * (tauCovFir * tauThFir * tauBlFir) * sigma * (q4Lamp - q4Sky);
        const T f111 = blScr * p[85] * p[4] * (tauCovFir * tauThFir) * sigma * (q4BlScr - q4Sky);
        const T f105 = p[169] * p[165] * p[3] * sigma * (q4Gro - q4Can);
        const T upF = 1 - glg_exp(-p[203] * (1 - p[189]) * lai);
        const T dnF = 1 - glg_exp(-p[203] * p[189] * lai);
        const T ci = p[194] * p[195] * sigma;
        const T f115 = ci * p[95] * ((1 - fPipe) * (1 - dnF)) * (q4Int - q4Flr);
        const T f116 = ci * p[104] * (fPipe * (1 - dnF)) * (q4Int - q4Pipe);
        const T f117 = ci * p[3] * (dnF + upF) * (q4Int - q4Can);
        const T f118 = ci * p[183] * ((1 - upF) * p[181]) * (q4Int - q4Lamp);
        const T f119 = ci * p[85] * (blScr * p[178] * (1 - upF)) * (q4Int - q4BlScr);
        const T f120 = ci * p[74] * (thScr * tauBlFir * p[178] * (1 - upF)) * (q4Int - q4ThScr);
        const T f121 = ci * (1 - p[70] - p[67]) * (tauThFir * tauBlFir * p[178] * (1 - upF)) * (q4Int - q4CovIn);
        const T f122 = ci * p[4] * (tauCovFir * tauThFir * tauBlFir * p[178] * (1 - upF)) * (q4Int - q4Sky);
        sCan += -f85 + f105 + f117;
        sCovIn += f121;
        sThScr += -f97 + f120;
        sFlr += -f94 + f115;
        sPipe += -f89 + f116;
        sLamp += -f104 + f118;
        sBlScr += -f111 + f119;
        pt.template put<18>(-f122 - f121 - f120 - f116 - f119 - f115 - f117 - f118);
        pt.template put<19>(-f105);
    }
    const T hCovInCovE = K[K_HCOV] * (tCovIn - tCovE);
    // soil chain (:888-910)
    const T hFlrSo1 = K[K_HFLRSO1] * (tFlr - GLG_X(x, 10));
    {
        const T hSo12 = K[K_HSO12] * (GLG_X(x, 10) - GLG_X(x, 11));
        const T hSo23 = K[K_HSO23] * (GLG_X(x, 11) - GLG_X(x, 12));
        const T hSo34 = K[K_HSO34] * (GLG_X(x, 12) - GLG_X(x, 13));
        const T hSo45 = K[K_HSO45] * (GLG_X(x, 13) - GLG_X(x, 14));
        const T hSo5Out = K[K_HSO5OUT] * (GLG_X(x, 14) - H[H_TSOOUT]);
        pt.template put<10>(K[K_INVCAPSO1] * (hFlrSo1 - hSo12));
        pt.template put<11>(K[K_INVCAPSO2] * (hSo12 - hSo23));
        pt.template put<12>(K[K_INVCAPSO3] * (hSo23 - hSo34));
        pt.template put<13>(K[K_INVCAPSO4] * (hSo34 - hSo45));
        pt.template put<14>(K[K_INVCAPSO5] * (hSo45 - hSo5Out));
    }
    pt.template put<4>(sCan);
    pt.template put<5>(sCovIn - hCovInCovE);
    pt.template put<6>(sCovE + hCovInCovE - H[H_HEC_COVEOUT] * (tCovE - H[H_TOUT]));
    pt.template put<7>(sThScr);
    pt.template put<8>(sFlr - hFlrSo1);
    pt.template put<9>(sPipe);
    pt.template put<17>(sLamp);
    pt.template put<20>(sBlScr);
}

// roof ventilation and leakage: exchange with the outside air
template <class KV, class HV, class XV, class PT>
GLG_HD void glg_unit_vent(const KV &K, const HV &H, const XV &x, const PT &pt, GlgSpecial<glg_unit_t<KV, XV>> &sp) {
    typedef glg_unit_t<KV, XV> T;
    const T co2Air = GLG_X(x, 0), co2Top = GLG_X(x, 1), tAir = GLG_X(x, 2), tTop = GLG_X(x, 3), vpAir = GLG_X(x, 15), vpTop = GLG_X(x, 16);
    const T tOut = H[H_TOUT];
    const T tkAir = tAir + T(GLG_C2K), tkTop = tTop + T(GLG_C2K);
    const T ra[3] = {tkAir, tkTop, tAir + H[H_TOUT_2K]};
    T ry[3];
    glg_rcp_n<3>(ra, ry);
    const T rAir = ry[0], rTop = ry[1];
    const T sVent = glg_sqrt(fabs(K[K_GHVENT] * (tAir - tOut) * ry[2] + H[H_CW_WIND2]) + T(1e-300));
    const T aVentRoof = fabs(H[H_VR_A] * sVent + H[H_VR_B]);  // |a136|
    const T rAirF = rAir - T(GLG_C2K_F32_DELTA) * (rAir * rAir);  // 1/(tAir + 273.15f), aux_states.hpp:84
    const T rTopF = rTop - T(GLG_C2K_F32_DELTA) * (rTop * rTop);
    const T vAirT = vpAir * rAirF, vTopT = vpTop * rTopF;
    pt.template put<1>(-(aVentRoof * (co2Top - H[H_CO2OUT])));
    pt.template put<0>(H[H_MCEXT] - H[H_FVENTSIDE_ABS] * (co2Air - H[H_CO2OUT]));
    pt.template put<2>(-(H[H_HEC_AIROUT] * (tAir - tOut)));
    pt.template put<3>(-(fabs(K[K_RHOCP]) * aVentRoof * (tTop - tOut)));
    pt.template put<16>(-(K[K_INVVPTOP] * tkTop) * (T(0.002165) * aVentRoof * (vTopT - H[H_VPOUT_T])));
    pt.template put<15>(-(K[K_INVVPAIR] * tkAir) * (H[H_MVAIROUT_C] * (vAirT - H[H_VPOUT_T])));
    sp.avent = aVentRoof;
}

// air flux through the screens: exchange main air <-> top compartment
template <class KV, class HV, class XV, class PT>
GLG_HD void glg_unit_scr(const KV &K, const HV &H, const XV &x, const PT &pt, GlgSpecial<glg_unit_t<KV, XV>> &sp) {
    typedef glg_unit_t<KV, XV> T;
    const T co2Air = GLG_X(x, 0), co2Top = GLG_X(x, 1), tAir = GLG_X(x, 2), tTop = GLG_X(x, 3), vpAir = GLG_X(x, 15), vpTop = GLG_X(x, 16);
    const T tkAir = tAir + T(GLG_C2K), tkTop = tTop + T(GLG_C2K);
    const T ra[2] = {tkAir, tkTop};
    T ry[2];
    glg_rcp_n<2>(ra, ry);
    const T rAir = ry[0], rTop = ry[1];
    const T rhoTop = K[K_RHOC] * rTop, rhoAir = K[K_RHOC] * rAir;
    const T rhoMean = T(0.5) * (rhoTop + rhoAir);
    const T rMean = glg_rcp(rhoMean);
    const T buoy = K[K_HALFG] * rhoMean * fabs(rhoAir - rhoTop);
    const T pw66 = glg_pow(fabs(tAir - tTop + T(1e-10)), T(0.66));
    const T oneMTh = H[H_1MTH], oneMBl = H[H_1MBL];
    const T sa[2] = {buoy * oneMTh + T(1e-10), buoy * oneMBl + T(1e-10)};
    T sy[2];
    glg_sqrt_n<2>(sa, sy);
    const T fThScr = H[H_THK] * pw66 + (oneMTh * rMean) * sy[0];
    const T fBlScr = H[H_BLK] * pw66 + (oneMBl * rMean) * sy[1];
    const T aScr = fabs(fmin(fThScr, fBlScr));  // |a144|
    const T mcAirTop = aScr * (co2Air - co2Top);
    pt.template put<1>(mcAirTop);
    pt.template put<0>(-mcAirTop);
    const T hAirTop = fabs(K[K_RHOCP]) * aScr * (tAir - tTop);
    pt.template put<2>(-hAirTop);
    pt.template put<3>(hAirTop);
    const T rAirF = rAir - T(GLG_C2K_F32_DELTA) * (rAir * rAir);
    const T rTopF = rTop - T(GLG_C2K_F32_DELTA) * (rTop * rTop);
    const T mvAirTop = T(0.002165) * aScr * (vpAir * rAirF - vpTop * rTopF);
    pt.template put<16>((K[K_INVVPTOP] * tkTop) * mvAirTop);
    pt.template put<15>(-(K[K_INVVPAIR] * tkAir) * mvAirTop);
    sp.ascr = aScr;
}

// transient-stiffness estimate of the graded integrator from the two air fluxes (same rule as glg_rhs / glgo_stiffness)
template <class KV>
GLG_HD double glg_stiffness(const KV &K, double aScr, double aVentRoof) {
    const double lamCov = 2.0 * K[K_HCOV] * K[K_INVCAPCOV];
    const double lamTop = fabs(K[K_RHOCP]) * K[K_INVCAPTOP] * (1.5 * aScr + aVentRoof);
    const double lamGas = (aScr + aVentRoof) * K[K_INVCAPCO2TOP];
    return 1.07 * fmax(lamCov, fmax(lamTop, lamGas));
}

template <bool GENERAL, class KV, class CV, class P, class XV, class PT>
GLG_HD void glg_unit_floor(const KV &K, const CV &C, const P &p, const XV &x, const PT &pt) {
    typedef glg_unit_t<KV, XV> T;
    const T tAir = GLG_X(x, 2), tCan = GLG_X(x, 4), tFlr = GLG_X(x, 8), tLamp = GLG_X(x, 17);
    const T hLampAir = K[K_HLAMPAIR] * (tLamp - tAir);
    const T hCanAir = fabs(K[K_2ALFA] * (C[C_SLA] * GLG_X(x, 23))) * (tCan - tAir);
    // 1.7 |dT|^(1/3) upward, 1.3 |dT|^(1/4) downward (:876): one branch-free root with a per-lane exponent
    const bool up = tFlr > tAir;
    const T dAbs = up ? fabs(tFlr - tAir + T(1e-10)) : fabs(tAir - tFlr + T(1e-10)) + T(1e-300);
    const T hecFlr = (up ? T(1.7) : T(1.3)) * glg_root34(dAbs, up);
    const T hAirFlr = hecFlr * (tAir - tFlr);
    T sAir = hLampAir + hCanAir - hAirFlr;
    if (GENERAL) {
        const T hIntLampAir = fabs(p[198]) * (GLG_X(x, 18) - tAir);  // a167
        sAir += hIntLampAir;
        pt.template put<18>(-hIntLampAir);
    }
    pt.template put<2>(sAir);
    pt.template put<4>(-hCanAir);
    pt.template put<8>(hAirFlr);
    pt.template put<17>(-hLampAir);
}

// A condensing surface S between the air compartment A (whose vapour condenses on it) and, for the screens, a far
// compartment B: free convection A -> S (and S -> B) with cube-root heat exchange coefficients, condensation cond()
// (aux_states.hpp:60-63).  Thermal screen, blackout screen and cover are this one computation on different data, so the
// kernel lets their three warps share ONE copy of the code (glg_roles.cuh: surface role, all addresses in registers).
//   surf = hA - hB + L mv ; air = -hA ; far = +hB ; vp = -(invvp (tA + 273.15)) mv
template <bool HAS_FAR, class T>
GLG_HD void glg_surface_core(T tA, T tS, T tB, T vpA, T coefA, T coefB, T invvp, T L, T &surf, T &air, T &far, T &vp) {
    T cy[2];
    if (HAS_FAR) {
        const T ca[2] = {fabs(tA - tS + T(1e-10)), fabs(tS - tB + T(1e-10))};
        glg_cbrt_n<2>(ca, cy);
    } else {
        cy[0] = glg_cbrt(fabs(tA - tS + T(1e-10)));
        cy[1] = T(0);
    }
    const T dv = vpA - glg_satvp_f(tS);
    const T hecA = coefA * cy[0];
    const T hA = fabs(hecA) * (tA - tS);
    const T hB = HAS_FAR ? fabs(coefB * cy[1]) * (tS - tB) : T(0);
    const T mv = T(6.4e-9) * hecA * dv * glg_inv1pexp(-T(0.1) * dv);
    surf = HAS_FAR ? hA - hB + L * mv : hA + L * mv;
    air = -hA;
    far = hB;
    vp = -(invvp * (tA + T(GLG_C2K))) * mv;
}

// one screen (thermal: I_SCR = 7, blackout: I_SCR = 20): convection main air -> screen -> top compartment, condensation
template <int I_SCR, class KV, class HV, class XV, class PT>
GLG_HD void glg_unit_screen(const KV &K, const HV &H, const XV &x, const PT &pt) {
    typedef glg_unit_t<KV, XV> T;
    T surf, air, far, vp;
    glg_surface_core<true, T>(GLG_X(x, 2), GLG_X(x, I_SCR), GLG_X(x, 3), GLG_X(x, 15), I_SCR == 7 ? H[H_17TH] : H[H_17BL],
                              I_SCR == 7 ? H[H_17TH] : H[H_17BL], K[K_INVVPAIR], K[K_L], surf, air, far, vp);
    pt.template put<I_SCR>(surf);
    pt.template put<2>(air);
    pt.template put<3>(far);
    pt.template put<15>(vp);
}

template <class KV, class HV, class XV, class PT>
GLG_HD void glg_unit_cover(const KV &K, const HV &H, const XV &x, const PT &pt) {
    typedef glg_unit_t<KV, XV> T;
    T surf, air, far, vp;
    glg_surface_core<false, T>(GLG_X(x, 3), GLG_X(x, 5), T(0), GLG_X(x, 16), H[H_HECIN], T(0), K[K_INVVPTOP], K[K_L], surf, air, far, vp);
    pt.template put<5>(surf);
    pt.template put<3>(air);
    pt.template put<16>(vp);
}

template <class KV, class CV, class HV, class XV, class PT>
GLG_HD void glg_unit_transp(const KV &K, const CV &C, const HV &H, const XV &x, const PT &pt) {
    typedef glg_unit_t<KV, XV> T;
    const T co2Air = GLG_X(x, 0), tAir = GLG_X(x, 2), tCan = GLG_X(x, 4), vpAir = GLG_X(x, 15);
    const T vpd = glg_satvp_f(tCan) - vpAir;
    const T lai = C[C_SLA] * GLG_X(x, 23);
    const T rfCo2 = fmin(T(1.5), T(1.) + H[H_CEVAP3] * glg_sq(K[K_ETAMGPPM] * co2Air - 200));
    const T rfVp = fmin(T(5.8), T(1.) + H[H_CEVAP4] * (vpd * vpd));
    const T rS = H[H_RS] * rfCo2 * rfVp;
    const T mvCanAir = vpd * (K[K_VEC] * lai * glg_rcp(K[K_RB] + rS));
    pt.template put<4>(-(K[K_L] * mvCanAir));
    pt.template put<15>((K[K_INVVPAIR] * (tAir + T(GLG_C2K))) * mvCanAir);
}

template <bool GENERAL, class KV, class CV, class HV, class XV, class PT>
GLG_HD void glg_unit_photo(const KV &K, const CV &C, const HV &H, const XV &x, const PT &pt) {
    typedef glg_unit_t<KV, XV> T;
    const T co2Air = GLG_X(x, 0), tAir = GLG_X(x, 2), tCan = GLG_X(x, 4), cBuf = GLG_X(x, 22);
    const T lai = C[C_SLA] * GLG_X(x, 23);
    const T j25 = lai * C[C_J25];
    const T co2Stom = C[C_ETASTOM] * (K[K_PPMC] * (tAir + T(GLG_C2K)) * co2Air);
    const T ra[3] = {j25, tCan + T(GLG_C2K), co2Stom};
    T ry[3];
    glg_rcp_n<3>(ra, ry);
    const T rj = C[C_J25] * ry[0], rCanK = ry[1], rStom = ry[2];
    // PAR absorbed by the canopy in umol (a191): the extinction factor is recomputed (U_OPT has it too); the four
    // exponentials of this unit are independent and evaluated interleaved
    const T ea[5] = {-K[K_K1PAR] * lai, C[C_ARR1] * (1 - C[C_T25K] * rCanK), C[C_ARR2A] - C[C_ARR2B] * rCanK,
                     T(5e-4) * (cBuf - C[C_CBUFMAX]), -K[K_K2PAR] * lai};
    T ey[5];
    if (GENERAL) {
        glg_exp_n<5>(ea, ey);
    } else {
        const T ea4[4] = {ea[0], ea[1], ea[2], ea[3]};
        T ey4[4];
        glg_exp_n<4>(ea4, ey4);
        ey[0] = ey4[0]; ey[1] = ey4[1]; ey[2] = ey4[2]; ey[3] = ey4[3]; ey[4] = ey4[0];
    }
    const T e32 = ey[0], e33 = ey[4];
    const T parCan = H[H_PARUMOL] * ((1 - e32) + e32 * K[K_RHOFLRPAR] * (1 - e33));
    const T gamma = rj * C[C_CGAMMA] * tCan + C[C_20CGAMMA] * (1 - rj);
    const T rb[3] = {T(1.0) + ey[2], T(1.0) + ey[3], 4 * (co2Stom + 2 * gamma)};
    T rz[3];
    glg_rcp_n<3>(rb, rz);
    const T jPot = j25 * ey[1] * C[C_JPOTNUM] * rz[0];
    const T jb = jPot + C[C_ALPHA] * parCan;
    // smaller root of theta J^2 - jb J + jPot alpha par = 0 (:1076-1077); fp32 uses the cancellation-free form
    //   (jb - sqrt(D)) / (2 theta) = (jb^2 - D) / (2 theta (jb + sqrt(D))),  D = jb^2 - 4 theta alpha jPot par + 1e-10
    // (the reference's form loses all fp32 digits when a perturbed t25k makes jPot >> alpha*par); in fp64 the reference's own
    // form is accurate to ~1e-12 and keeps a reciprocal off this unit's critical path.
    const T fourTc = C[C_4THETAALPHA] * jPot * parCan;
    const T sqD = glg_sqrt(jb * jb - fourTc + T(1e-10));
    const T jE = std::is_same<T, float>::value ? C[C_INV2THETA] * (fourTc - T(1e-10)) * glg_rcp(jb + sqD)
                                               : C[C_INV2THETA] * (jb - sqD);
    const T phot = jE * (co2Stom - gamma) * rz[2];
    const T photNet = phot - phot * gamma * rStom;
    const T mcAirBuf = C[C_MCH2O] * rz[1] * photNet;
    pt.template put<22>(mcAirBuf);
    pt.template put<0>(-(C[C_CO2RATIO] * mcAirBuf));
}

template <class KV, class CV, class XV, class PT>
GLG_HD void glg_unit_flows(const KV &K, const CV &C, const XV &x, const PT &pt) {
    typedef glg_unit_t<KV, XV> T;
    const T tCan = GLG_X(x, 4), tCan24 = GLG_X(x, 21), cBuf = GLG_X(x, 22);
    const T gT24 = T(0.047) * tCan24 + T(0.06);
    const T ea[5] = {-T(1.1587) * (tCan24 - C[C_T24MIN]), T(1.3904) * (tCan24 - C[C_T24MAX]), -T(0.869) * (tCan - C[C_TCANMIN]),
                     T(0.5793) * (tCan - C[C_TCANMAX]), -T(5e-3) * (cBuf - C[C_CBUFMIN])};
    T ey[5];
    glg_exp_n<5>(ea, ey);
    const T ra[3] = {(T(1.) + ey[0]) * (T(1.) + ey[1]), (T(1.) + ey[2]) * (T(1.) + ey[3]), T(1.0) + ey[4]};
    T ry[3];
    glg_rcp_n<3>(ra, ry);
    const T hT24 = ry[0], hTCan = ry[1];
    const T sSum = GLG_X(x, 26) * K[K_INVTENDSUM];
    const T sSum1 = sSum - T(1.0);
    const T sa[2] = {sSum * sSum + T(1e-4), sSum1 * sSum1 + T(1e-4)};
    T sy[2];
    glg_sqrt_n<2>(sa, sy);
    const T hTSum = T(0.5) * (sSum + sy[0]) - T(0.5) * (sSum1 + sy[1]);
    const T flow = ry[2] * hT24 * gT24;
    const T mcBufLeaf = flow * C[C_RGLEAF];
    const T mcBufStem = flow * C[C_RGSTEM];
    const T mcBufFruit = flow * hTCan * hTSum * C[C_RGFRUIT];
    const T mcBufAir = C[C_GLEAF] * mcBufLeaf + C[C_GSTEM] * mcBufStem + C[C_GFRUIT] * mcBufFruit;
    pt.template put<22>(-mcBufFruit - mcBufLeaf - mcBufStem - mcBufAir);
    pt.template put<23>(mcBufLeaf);
    pt.template put<24>(mcBufStem);
    pt.template put<25>(mcBufFruit);
    pt.template put<0>(C[C_CO2RATIO] * mcBufAir);
}

template <class KV, class CV, class XV, class PT>
GLG_HD void glg_unit_maint(const KV &K, const CV &C, const XV &x, const PT &pt, GlgSpecial<glg_unit_t<KV, XV>> &sp) {
    typedef glg_unit_t<KV, XV> T;
    const T tCan24 = GLG_X(x, 21), cLeaf = GLG_X(x, 23), cStem = GLG_X(x, 24), cFruit = GLG_X(x, 25);
    const T kHar = T(2.0) * T(4.6052) / T(1e4);  // smoothHar(v, cutoff, 1e4, 5e4) = 5e4/(1+exp(-kHar (v-cutoff)))  (:75-79)
    const T ea[3] = {C[C_LNQ10X] * (tCan24 - 25), -kHar * (cLeaf - C[C_CLEAFMAX]), -kHar * (cFruit - C[C_CFRUITMAX])};
    T ey[3];
    glg_exp_n<3>(ea, ey);
    const T ra[2] = {T(1.0) + ey[1], T(1.0) + ey[2]};
    T ry[2];
    glg_rcp_n<2>(ra, ry);
    const T maint = C[C_MAINT] * ey[0];
    const T mcLeafAir = maint * cLeaf * C[C_MLEAF];
    const T mcStemAir = maint * cStem * C[C_MSTEM];
    const T mcFruitAir = maint * cFruit * C[C_MFRUIT];
    pt.template put<23>(-mcLeafAir - T(5e4) * ry[0]);
    pt.template put<24>(-mcStemAir);
    pt.template put<25>(-mcFruitAir - T(5e4) * ry[1]);
    pt.template put<0>(C[C_CO2RATIO] * (mcLeafAir + mcStemAir + mcFruitAir));
    sp.lambda = glg_harvest_lambda(ry[0], ry[1]);
}

// dispatcher: unit U with the argument set every unit can pick from
template <int U, bool GENERAL, class KV, class CV, class HV, class P, class UT, class XV, class PT>
GLG_HD void glg_unit(const KV &K, const CV &C, const HV &H, const P &p, const UT *u, const XV &x, const PT &pt,
                     GlgSpecial<glg_unit_t<KV, XV>> &sp) {
    if (U == U_OPT) glg_unit_opt<GENERAL>(K, C, H, x, pt);
    else if (U == U_PIPES) glg_unit_pipes(K, C, x, pt, sp);
    else if (U == U_FIR) glg_unit_fir<GENERAL>(K, C, H, p, u, x, pt);
    else if (U == U_VENT) glg_unit_vent(K, H, x, pt, sp);
    else if (U == U_SCR) glg_unit_scr(K, H, x, pt, sp);
    else if (U == U_FLOOR) glg_unit_floor<GENERAL>(K, C, p, x, pt);
    else if (U == U_THSCR) glg_unit_screen<7>(K, H, x, pt);
    else if (U == U_BLSCR) glg_unit_screen<20>(K, H, x, pt);
    else if (U == U_COVER) glg_unit_cover(K, H, x, pt);
    else if (U == U_TRANSP) glg_unit_transp(K, C, H, x, pt);
    else if (U == U_PHOTO) glg_unit_photo<GENERAL>(K, C, H, x, pt);
    else if (U == U_FLOWS) glg_unit_flows(K, C, x, pt);
    else glg_unit_maint(K, C, x, pt, sp);
}

// ---------------------------------------------------------------------------------------------------------
// unit -> group-warp assignment.  Row w lists the units group warp w evaluates (-1 pads).  NG = number of group warps.
// Balanced on FP64 instruction counts (tools/sasssim): each sub-partition (warp id mod 4) gets about a quarter of the work.
// ---------------------------------------------------------------------------------------------------------
constexpr int GLG_MAXUNITS_PER_WARP = 5;
struct GlgAssign {
    int n_warps;
    int unit[16][GLG_MAXUNITS_PER_WARP];
};
GLG_HD constexpr GlgAssign glg_assign(int ng) {
    GlgAssign a{};
    a.n_warps = ng;
    for (int w = 0; w < 16; ++w)
        for (int k = 0; k < GLG_MAXUNITS_PER_WARP; ++k) a.unit[w][k] = -1;
    if (ng == 12) {
        // sub-partition of group warp w is (w + NO) % 4 with NO = 4 owner warps in front => w % 4
        // the heaviest unit of each sub-partition sits on the LOWEST warp id (measured: 1.73 ms vs 1.91 ms per step at B = 4096 with
        // the order reversed); moving floor convection to the maintenance unit's warp was measured and dropped (DESIGN.md item 4)
        const int t[12][2] = {{U_FIR, -1},    {U_PHOTO, -1}, {U_FLOWS, -1}, {U_SCR, -1},
                              {U_TRANSP, -1}, {U_OPT, -1},   {U_PIPES, -1}, {U_VENT, U_FLOOR},
                              {U_COVER, -1},  {U_THSCR, -1}, {U_MAINT, -1}, {U_BLSCR, -1}};
        for (int w = 0; w < 12; ++w)
            for (int k = 0; k < 2; ++k) a.unit[w][k] = t[w][k];
    } else if (ng == 4) {  // one fat warp per sub-partition (throughput layouts: all warps of a sub-partition run the same code)
        const int t[4][5] = {{U_FIR, U_TRANSP, U_COVER, -1, -1}, {U_PHOTO, U_OPT, U_THSCR, -1, -1}, {U_FLOWS, U_PIPES, U_MAINT, -1, -1},
                             {U_SCR, U_VENT, U_FLOOR, U_BLSCR, -1}};
        // measured at B = 262 144 (graded, 300 RK4 steps): this table 30.46 ms per step; three re-deals 33.31 (FP64 instructions
        // per warp 225 / 234 / 227 / 232 instead of 255 / 234 / 232 / 197), 33.98 and 30.48 -- equal FP64 instruction counts per
        // warp do not balance the roles, the dependency chains inside the units do
        for (int w = 0; w < 4; ++w)
            for (int k = 0; k < 5; ++k) a.unit[w][k] = t[w][k];
    } else if (ng == 8) {  // the kernels do not use these two: the host build of the unit split checks them against the oracle
        const int t[8][3] = {{U_FIR, -1, -1},          {U_PHOTO, U_FLOOR, -1}, {U_FLOWS, U_MAINT, -1}, {U_SCR, U_VENT, -1},
                             {U_THSCR, U_TRANSP, -1},  {U_OPT, U_COVER, -1},   {U_PIPES, -1, -1},      {U_BLSCR, -1, -1}};
        for (int w = 0; w < 8; ++w)
            for (int k = 0; k < 3; ++k) a.unit[w][k] = t[w][k];
    } else {  // one unit per warp (13 group warps), in unit order
        for (int w = 0; w < U_COUNT; ++w) a.unit[w][0] = w;
    }
    return a;
}
// everything the kernel needs to know about the assignment, computed in one pass (cheap for the constexpr evaluator)
struct GlgWarpTable {
    unsigned states[16];                         // states warp w contributes to
    unsigned prior[16][GLG_MAXUNITS_PER_WARP];   // states touched by the units before unit k of warp w (accumulator PRIOR mask)
    unsigned units[16];                          // bit u set = warp w evaluates unit u
    int contribs[GLG_NX];                        // number of warps contributing to state i
    int slot[16][GLG_NX];                        // slot of (warp, state) in warp-major order, -1 if none
    int n_part;                                  // number of (warp, state) pairs
};
GLG_HD constexpr GlgWarpTable glg_make_warp_table(int ng, bool general) {
    const GlgAssign a = glg_assign(ng);
    GlgWarpTable t{};
    int n = 0;
    for (int w = 0; w < 16; ++w) {
        unsigned m = 0, um = 0;
        for (int k = 0; k < GLG_MAXUNITS_PER_WARP; ++k) {
            t.prior[w][k] = m;
            if (w < ng && a.unit[w][k] >= 0) {
                m |= glg_unit_states(a.unit[w][k], general);
                um |= 1u << a.unit[w][k];
            }
        }
        t.states[w] = m;
        t.units[w] = um;
        for (int i = 0; i < GLG_NX; ++i) {
            t.slot[w][i] = (m >> i & 1u) ? n : -1;
            n += (int)(m >> i & 1u);
        }
    }
    t.n_part = n;
    for (int i = 0; i < GLG_NX; ++i) {
        int c = 0;
        for (int w = 0; w < ng; ++w) c += (int)(t.states[w] >> i & 1u);
        t.contribs[i] = c;
    }
    return t;
}
template <int NG, bool GENERAL>
struct GlgWT {
    static constexpr GlgWarpTable t = glg_make_warp_table(NG, GENERAL);
    GLG_HD static constexpr bool has_unit(int w, int u) { return (t.units[w] >> u & 1u) != 0; }
    GLG_HD static constexpr int unit_warp(int u) {
        for (int w = 0; w < NG; ++w)
            if (t.units[w] >> u & 1u) return w;
        return -1;
    }
};

// evaluates the units of group warp W in order, accumulating into v[28]; specials into sp
template <int NG, int W, int Kk, bool GENERAL, class KV, class CV, class HV, class P, class UT, class XV, class T>
GLG_HD void glg_run_warp_units(const KV &K, const CV &C, const HV &H, const P &p, const UT *u, const XV &x, T *v,
                               GlgSpecial<T> &sp) {
    constexpr int U = glg_assign(NG).unit[W][Kk < GLG_MAXUNITS_PER_WARP ? Kk : 0];
    if constexpr (Kk < GLG_MAXUNITS_PER_WARP && U >= 0) {
        constexpr unsigned prior = GlgWT<NG, GENERAL>::t.prior[W][Kk];
        const GlgAccum<T, prior> pt{v};
        glg_unit<U, GENERAL>(K, C, H, p, u, x, pt, sp);
        glg_run_warp_units<NG, W, Kk + 1, GENERAL>(K, C, H, p, u, x, v, sp);
    }
}

// ---------------------------------------------------------------------------------------------------------
// One-lane RHS assembled from the units: S[i] = dx_i/dt for one env, generic in the scalar type (double, float, GlgDual).  The
// units of each group warp of the NG-warp assignment are accumulated into that warp's partial sums, the partial sums are added in
// warp order and the owners' capacity scales (glg_state_scale_index) are applied -- the data flow of the warp-specialised kernel,
// in one thread (the sum order of tests/hostmath's hm_rhs_units).  Returns the transient-stiffness estimate of the graded
// integrator, from value parts: it only feeds step-count decisions.
template <class T>
struct GlgArrayXT {  // plain array of scalar type T in state order
    const T *p;
    template <int I>
    GLG_HD T at() const { return p[I]; }
};
template <int NG, int W, bool GENERAL, class KV, class CV, class HV, class P, class UT, class XV, class ST, class T>
GLG_HD void glg_rhs_units_warps(const KV &K, const CV &C, const HV &H, const P &p, const UT *u, const XV &x, ST *sum, GlgSpecial<T> &sp) {
    if constexpr (W < NG) {
        T v[GLG_NX] = {};
        glg_run_warp_units<NG, W, 0, GENERAL>(K, C, H, p, u, x, v, sp);
        constexpr unsigned mask = GlgWT<NG, GENERAL>::t.states[W];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (int i = 0; i < GLG_NX; ++i)
            if (mask >> i & 1u) sum[i] += static_cast<ST>(v[i]);
        glg_rhs_units_warps<NG, W + 1, GENERAL>(K, C, H, p, u, x, sum, sp);
    }
}
template <bool GENERAL, int NG = U_COUNT, class KV, class CV, class HV, class P, class UT, class XV, class ST>
GLG_HD double glg_rhs_units(const KV &K, const CV &C, const HV &H, const P &p, const UT *u, const XV &x, ST *S) {
    typedef glg_unit_t<KV, XV> T;
    ST sum[GLG_NX];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int i = 0; i < GLG_NX; ++i) sum[i] = ST(0.0);
    GlgSpecial<T> sp{};
    glg_rhs_units_warps<NG, 0, GENERAL>(K, C, H, p, u, x, sum, sp);
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int i = 0; i < GLG_NX; ++i) {
        const int sk = glg_state_scale_index(i);
        if (sk >= 0) S[i] = K[sk] * sum[i];
        else if (sk == -1) S[i] = sum[i];
        else S[i] = static_cast<ST>(sp.canscale) * sum[i];
    }
    return glg_stiffness(K, (double)glg_value(sp.ascr), (double)glg_value(sp.avent));
}
