// glg_model.h -- GreenLight right-hand side, restructured for one-thread-per-env evaluation on sm_100a.
//
// What it computes: the 28 state derivatives of the reference model
//   update()  gl_gym/environments/models/aux_states.hpp:96-1271
//   ODE()     gl_gym/environments/models/ode.hpp:6-124
// but NOT in the reference's shape.  The 239-entry auxiliary vector is never materialised.  Work is split by
// how often its inputs change:
//   K  (glg_make_k)  : depends on the nominal parameters only      -> once per handle, lives in __constant__
//   C  (glg_make_c)  : depends on the crop parameters p[128..163]  -> once per handle (nominal) or once per
//                      env-step (parametric-uncertainty mode, noise.py:3-23)
//   H  (glg_hoist)   : depends on (u, d, p) of this env-step       -> once per env-step (zero-order hold,
//                      greenlight_model.cpp:59-63), kept in a shared-memory column per thread
//   glg_rhs          : the state-dependent remainder, evaluated 4*n_sub times per env-step with the stage state
//                      in registers.
// Algebraic rewrites used (all exact in real arithmetic, ~1e-16 relative in fp64; parity gate is 1e-9):
//   pow(T,4) -> (T*T)^2 ; pow(x,1/3) -> cbrt ; pow(x,1/4) -> sqrt(sqrt) ; pow(x,y) -> exp(y*log(x));
//   smoothHar's (tanh(z)+1)/2 -> 1/(1+exp(-2z)) ; FIR coefficient products hoisted ; a77's five-term lamp
//   balance folded into one hoisted constant for the lamp node ; 1/(T+273.15f) from 1/(T+273.15) by one
//   Newton-like correction (the reference's airMv uses a *float* Kelvin offset, aux_states.hpp:84).
// Structural zeros of the reference that hold for ANY parameter values (a[38]=0 => interlight radiation terms,
// a[126]=0 => side vents, a[177..180], a[221], a[223..232], a[234..238]) are dropped.  Terms that vanish only
// for the default parameter values (tauRfFir p70, interlight FIR p194/p195/p198, grow-pipe FIR p165) are
// compiled in when GENERAL=true; the host picks the variant by inspecting the parameter table.
//
// The header is valid C++ for g++ as well: tests build a host copy of exactly this math
// (tests/hostmath) to check the restructuring against the oracle without a GPU.  The product never runs it.
#pragma once
#include <math.h>

#include <type_traits>
#include <utility>

#include "glg_math.h"

#define GLG_NX 28
#define GLG_NU 6
#define GLG_ND 10
#define GLG_NP 208

// ---------------------------------------------------------------------------------------------------------
// field indices
// ---------------------------------------------------------------------------------------------------------
enum GlgK {  // parameter-only constants (non-crop)
    K_K1PAR, K_K2PAR, K_KNIR, K_KFIR,         // canopy extinction coefficients p32..p35
    K_RHOFLRPAR, K_RHOCANNIR, K_RHOFLRNIR, K_TAUHATFLRNIR,
    K_C87, K_C91, K_C92, K_C98, K_C99, K_C100, K_C101,  // FIR pair coefficients that do not depend on u
    K_GHVENT,                                  // g*hVent
    K_RHOC,                                    // mAir*pressure/R
    K_HALFG,                                   // 0.5*g
    K_RHOCP,                                   // rhoAir*cPAir
    K_HECIN,                                   // cHecIn*aCov/aFlr
    K_PIPEAIR, K_GROPIPEAIR,                   // 1.99*pi*phi*l
    K_2ALFA,                                   // 2*alfaLeafAir
    K_HFLRSO1, K_HSO12, K_HSO23, K_HSO34, K_HSO45, K_HSO5OUT, K_HCOV, K_HLAMPAIR,
    K_ETAMGPPM, K_VEC, K_RB, K_L,
    K_INVCAPCO2AIR, K_INVCAPCO2TOP, K_INVCAPAIR, K_INVCAPTOP, K_INVCAPLEAF, K_INVCAPCOV, K_INVCAPTHSCR,
    K_INVCAPFLR, K_INVCAPPIPE, K_INVCAPSO1, K_INVCAPSO2, K_INVCAPSO3, K_INVCAPSO4, K_INVCAPSO5,
    K_INVVPAIR, K_INVVPTOP, K_INVCAPLAMP, K_INVCAPINTLAMP, K_INVCAPGROPIPE, K_INVCAPBLSCR,
    K_PPMC,                                    // co2 density[mg m-3] * T[K] -> ppm
    K_INVTENDSUM,
    K_COUNT
};

enum GlgC {  // crop constants (functions of p[128..163]); uniform, or per-env under parametric uncertainty
    C_SLA, C_J25, C_CGAMMA, C_20CGAMMA, C_ETASTOM,
    C_ARR1, C_T25K, C_ARR2A, C_ARR2B, C_JPOTNUM,  // jPot Arrhenius pieces
    C_INV2THETA, C_ALPHA, C_4THETAALPHA,
    C_MCH2O, C_CO2RATIO, C_CBUFMAX, C_CBUFMIN, C_T24MIN, C_T24MAX, C_TCANMIN, C_TCANMAX,
    C_RGLEAF, C_RGSTEM, C_RGFRUIT, C_GLEAF, C_GSTEM, C_GFRUIT,
    C_MAINT, C_LNQ10X, C_MLEAF, C_MSTEM, C_MFRUIT, C_CLEAFMAX, C_CFRUITMAX,
    C_COUNT
};

enum GlgH {  // per-env-step constants (depend on u, d and p)
    H_PARCAN_W, H_PARLAMP_W, H_PARFLR_W, H_PARLAMPFLR_W, H_PARUMOL,
    H_RHOCOVNIR, H_TAUHATCOVNIR, H_TAUHAT2,
    H_NIRSUN, H_NIRLAMPCAN, H_NIRLAMPFLR, H_LAMPRAD, H_GLOBAIR_A, H_GLOBAIR_B, H_GLOBCOV,
    H_C84, H_C86, H_C108, H_C88, H_C90, H_C93, H_C95, H_C106, H_C107, H_C96, H_C102, H_C103, H_C109, H_C110,
    H_C112,
    H_TSKY4,
    H_TOUT, H_TOUT_2K, H_CW_WIND2, H_VR_A, H_VR_B,
    H_THK, H_BLK, H_1MTH, H_1MBL,
    H_17TH, H_17BL, H_HEC_AIROUT, H_HEC_COVEOUT,
    H_TSOOUT,
    H_CEVAP3, H_CEVAP4, H_RS,
    H_VPOUT_T, H_MVAIROUT_C,
    H_MCEXT, H_CO2OUT, H_FVENTSIDE_ABS,
    H_HBOIL, H_LAMPNET,
    H_HECIN, H_ZERO,  // copies of K_HECIN and 0.0 in the per-env column: the kernel's shared surface role reads all its coefficients from H
    H_COUNT
};

// ---------------------------------------------------------------------------------------------------------
// small math helpers
// ---------------------------------------------------------------------------------------------------------
#define GLG_C2K 273.15
// (double)273.15f - 273.15 : the reference's airMv adds a float Kelvin offset (aux_states.hpp:84)
#define GLG_C2K_F32_DELTA (273.149993896484375 - 273.15)

template <class T>
GLG_HD T glg_sq(T v) { return v * v; }
// exact-libm versions: used outside the substep loop (hoisting, observations), once per env-step
GLG_HD double glg_satvp(double t) { return 610.78 * exp(17.2694 * t / (t + 238.3)); }  // aux_states.hpp:5-12
// fast versions for the RHS (glg_math.h)
template <class T>
GLG_HD T glg_satvp_f(T t) { return T(610.78) * glg_exp(T(17.2694) * (t * glg_rcp(t + T(238.3)))); }
// cond(): aux_states.hpp:60-63.  exp overflow -> 1/(1+huge) = 0, as with IEEE inf in the reference.
template <class T>
GLG_HD T glg_cond(T hec, T vp1, T vp2) {
    const T dv = vp1 - vp2;
    return T(6.4e-9) * hec * dv * glg_inv1pexp(T(-0.1) * dv);
}

// two-layer optics (aux_states.hpp:25-41)
template <class T>
GLG_HD T glg_tau12(T t1, T t2, T r1d, T r2u) { return t1 * t2 / (1. - r1d * r2u); }
template <class T>
GLG_HD T glg_rhoup(T t1, T r1u, T r1d, T r2u) { return r1u + (t1 * t1 * r2u) / (1. - r1d * r2u); }
template <class T>
GLG_HD T glg_rhodn(T t2, T r1d, T r2u, T r2d) { return r2d + (t2 * t2 * r1d) / (1. - r1d * r2u); }

// ---------------------------------------------------------------------------------------------------------
// K: parameter-only constants.  P is anything indexable as p[i] -> double.
// ---------------------------------------------------------------------------------------------------------
template <class P>
GLG_HD void glg_make_k(const P &p, double *K) {
    const double pi = 3.14159265358979323846;
    const double sigma = p[2];
    const double epsCovFir = 1 - p[70] - p[67];  // a28=a29 (:216-220)
    const double fPipe = 0.49 * pi * p[107] * p[105];
    K[K_K1PAR] = p[32]; K[K_K2PAR] = p[33]; K[K_KNIR] = p[34]; K[K_KFIR] = p[35];
    K[K_RHOFLRPAR] = p[98]; K[K_RHOCANNIR] = p[11]; K[K_RHOFLRNIR] = p[97]; K[K_TAUHATFLRNIR] = 1 - p[97];
    K[K_C87] = p[3] * p[95] * p[125] * sigma;           // rCanFlr   (:509)   x aCan
    K[K_C91] = p[124] * p[104] * p[95] * 0.49 * sigma;  // rPipeFlr  (:529)
    K[K_C92] = p[124] * p[104] * p[3] * 0.49 * sigma;   // rPipeCan  (:533)   x aCan
    K[K_C98] = epsCovFir * p[4] * sigma;                // rCovESky  (:563)
    K[K_C99] = p[181] * p[183] * p[95] * p[199] * (1 - fPipe) * sigma;  // rFirLampFlr (:568) x e35
    K[K_C100] = p[181] * p[183] * p[104] * p[199] * fPipe * sigma;      // rLampPipe   (:573) x e35
    K[K_C101] = p[181] * p[183] * p[3] * sigma;                         // rFirLampCan (:577) x aCan
    K[K_GHVENT] = p[26] * p[56];
    K[K_RHOC] = p[36] * p[126] / p[39];
    K[K_HALFG] = 0.5 * p[26];
    K[K_RHOCP] = p[111] * p[23];
    K[K_HECIN] = p[50] * p[47] / p[46];
    K[K_PIPEAIR] = 1.99 * pi * p[105] * p[107];
    K[K_GROPIPEAIR] = 1.99 * pi * p[167] * p[166];
    K[K_2ALFA] = 2 * p[0];
    K[K_HFLRSO1] = fabs(2. / (p[101] / p[99] + p[27] / p[103]));
    K[K_HSO12] = fabs(2. * p[103] / (p[27] + p[28]));
    K[K_HSO23] = fabs(2. * p[103] / (p[28] + p[29]));
    K[K_HSO34] = fabs(2. * p[103] / (p[29] + p[30]));
    K[K_HSO45] = fabs(2. * p[103] / (p[30] + p[31]));
    K[K_HSO5OUT] = fabs(2. * p[103] / (p[31] + p[37]));
    K[K_HCOV] = fabs(1. / (p[73] / p[71]));
    K[K_HLAMPAIR] = fabs(p[185]);
    K[K_ETAMGPPM] = p[7];
    K[K_VEC] = 2. * p[111] * p[23] / (p[1] * p[14]);
    K[K_RB] = p[41];
    K[K_L] = p[1];
    const double capCov01 = 0.1 * (cos(p[45] * pi / 180.) * p[73] * p[64] * p[72]);  // a33=a34 (:227,241-242)
    K[K_INVCAPCO2AIR] = 1. / p[122]; K[K_INVCAPCO2TOP] = 1. / p[123];
    K[K_INVCAPAIR] = 1. / p[112]; K[K_INVCAPTOP] = 1. / p[120];
    K[K_INVCAPLEAF] = 1. / p[16];
    K[K_INVCAPCOV] = 1. / capCov01;
    K[K_INVCAPTHSCR] = 1. / p[119]; K[K_INVCAPFLR] = 1. / p[113]; K[K_INVCAPPIPE] = 1. / p[110];
    K[K_INVCAPSO1] = 1. / p[114]; K[K_INVCAPSO2] = 1. / p[115]; K[K_INVCAPSO3] = 1. / p[116];
    K[K_INVCAPSO4] = 1. / p[117]; K[K_INVCAPSO5] = 1. / p[118];
    K[K_INVVPAIR] = p[39] / (p[38] * p[48]);             // 1/a35 = K*(tAir+273.15)  (:246)
    K[K_INVVPTOP] = p[39] / (p[38] * (p[49] - p[48]));   // 1/a36                     (:249)
    K[K_INVCAPLAMP] = 1. / p[184]; K[K_INVCAPINTLAMP] = 1. / p[191]; K[K_INVCAPGROPIPE] = 1. / p[171];
    K[K_INVCAPBLSCR] = 1. / p[121];
    K[K_PPMC] = 1e6 * 8.3144598 * 1e-6 / (101325 * 44.01e-3);  // co2dens2ppm(T, 1e-6*x0) (:14-23,782)
    K[K_INVTENDSUM] = 1. / p[163];
}

// ---------------------------------------------------------------------------------------------------------
// C: crop constants.
// ---------------------------------------------------------------------------------------------------------
template <class P>
GLG_HD void glg_make_c(const P &p, double *C) {
    C[C_SLA] = p[142];
    C[C_J25] = p[129];
    C[C_CGAMMA] = p[130];
    C[C_20CGAMMA] = 20 * p[130];
    C[C_ETASTOM] = p[131];
    // jPot (:1066-1068): exp(eJ*(Tk-t25k)/(1e-3 R Tk t25k)) = exp(ARR1*(1 - t25k/Tk))
    const double r3 = 1e-3 * p[39];
    C[C_ARR1] = p[132] / (r3 * p[133]);
    C[C_T25K] = p[133];
    // exp((S*Tk - H)/(1e-3 R Tk)) = exp(ARR2A - ARR2B/Tk)
    C[C_ARR2A] = p[134] / r3;
    C[C_ARR2B] = p[135] / r3;
    C[C_JPOTNUM] = 1 + exp((p[134] * p[133] - p[135]) / (r3 * p[133]));
    C[C_INV2THETA] = 1. / (2. * p[136]);
    C[C_ALPHA] = p[137];
    C[C_4THETAALPHA] = 4 * p[136] * p[137];
    C[C_MCH2O] = p[138];
    C[C_CO2RATIO] = p[139] / p[138];
    C[C_CBUFMAX] = p[157]; C[C_CBUFMIN] = p[158];
    C[C_T24MIN] = p[160]; C[C_T24MAX] = p[159]; C[C_TCANMIN] = p[162]; C[C_TCANMAX] = p[161];
    C[C_RGLEAF] = p[155]; C[C_RGSTEM] = p[156]; C[C_RGFRUIT] = p[154];
    C[C_GLEAF] = p[147]; C[C_GSTEM] = p[148]; C[C_GFRUIT] = p[146];
    C[C_MAINT] = 1. - exp(-p[149] * p[143]);
    C[C_LNQ10X] = 0.1 * log(p[150]);  // pow(q10, 0.1*(t-25)) = exp(LNQ10X*(t-25))
    C[C_MLEAF] = p[152]; C[C_MSTEM] = p[153]; C[C_MFRUIT] = p[151];
    C[C_CLEAFMAX] = p[144]; C[C_CFRUITMAX] = p[145];
}

// ---------------------------------------------------------------------------------------------------------
// H: everything that depends on (u, d, p) but not on the state.  Executed once per env-step.
//   u[6]: boil, co2, thScr, vent, lamp, blScr (aux_states.hpp:97-105)   d[>=7]: iGlob,tOut,vpOut,co2Out,wind,tSky,tSoOut
// ---------------------------------------------------------------------------------------------------------
// Generic in u's scalar type T (double in the step kernels; GlgDual for the derivative with respect to the controls).
template <class P, class T, class HOUT>
GLG_HD void glg_hoist(const P &p, const T *u, const double *d, HOUT &H) {
    const double pi = 3.14159265358979323846;
    const T thScr = u[2], blScr = u[5];
    // cover optics: roof+thermal screen -> +blackout screen -> +lamp layer, PAR and NIR (:111-194)
    const T tauThPar = 1 - thScr * (1 - p[80]), rhoThPar = thScr * p[77];
    const T tauA = glg_tau12<T>(p[69], tauThPar, p[66], rhoThPar);
    const T rupA = glg_rhoup<T>(p[69], p[66], p[66], rhoThPar);
    const T rdnA = glg_rhodn<T>(tauThPar, p[66], rhoThPar, rhoThPar);
    const T tauThNir = 1 - thScr * (1 - p[79]), rhoThNir = thScr * p[76];
    const T tauB = glg_tau12<T>(p[68], tauThNir, p[65], rhoThNir);
    const T rupB = glg_rhoup<T>(p[68], p[65], p[65], rhoThNir);
    const T rdnB = glg_rhodn<T>(tauThNir, p[65], rhoThNir, rhoThNir);
    const T tauBlPar = 1 - blScr * (1 - p[90]), rhoBlPar = blScr * p[88];
    const T tauA2 = glg_tau12<T>(tauA, tauBlPar, rdnA, rhoBlPar);
    const T rupA2 = glg_rhoup<T>(tauA, rupA, rdnA, rhoBlPar);
    const T rdnA2 = glg_rhodn<T>(tauBlPar, rdnA, rhoBlPar, rhoBlPar);
    const T tauBlNir = 1 - blScr * (1 - p[89]), rhoBlNir = blScr * p[87];
    const T tauB2 = glg_tau12<T>(tauB, tauBlNir, rdnB, rhoBlNir);
    const T rupB2 = glg_rhoup<T>(tauB, rupB, rdnB, rhoBlNir);
    const T rdnB2 = glg_rhodn<T>(tauBlNir, rdnB, rhoBlNir, rhoBlNir);
    const T tauCovPar = glg_tau12<T>(tauA2, p[176], rdnA2, p[179]);
    const T rhoCovPar = glg_rhoup<T>(tauA2, rupA2, rdnA2, p[179]);
    const T tauCovNir = glg_tau12<T>(tauB2, p[177], rdnB2, p[180]);
    const T rhoCovNir = glg_rhoup<T>(tauB2, rupB2, rdnB2, p[180]);
    const T aCovPar = 1 - tauCovPar - rhoCovPar, aCovNir = 1 - tauCovNir - rhoCovNir;
    const double epsCovFir = 1 - p[70] - p[67];

    // radiation above the canopy (:256-295)
    const double iGlob = d[0];
    const T qLamp = p[172] * u[4];                          // a37
    const T parSun = (1 - p[44]) * tauCovPar * p[6] * iGlob;  // a39
    const T parLamp = p[174] * qLamp;                        // a40
    const T rCan = (1 - p[44]) * iGlob * (p[6] * tauCovPar + p[5] * tauCovNir) + (p[174] + p[175]) * qLamp;  // a45
    H[H_PARCAN_W] = (parSun + parLamp) * (1 - p[10]);
    H[H_PARLAMP_W] = parLamp * (1 - p[10]);
    H[H_PARFLR_W] = (1 - p[98]) * (parSun + parLamp);
    H[H_PARLAMPFLR_W] = (1 - p[98]) * parLamp;
    H[H_PARUMOL] = (p[187] * parLamp + p[140] * parSun) * (1 - p[10]);  // a191 per unit of the LAI factor
    H[H_RHOCOVNIR] = rhoCovNir;
    H[H_TAUHATCOVNIR] = 1 - rhoCovNir;
    H[H_TAUHAT2] = (1 - rhoCovNir) * (1 - rhoCovNir);
    H[H_NIRSUN] = (1 - p[44]) * p[5] * iGlob;
    H[H_NIRLAMPCAN] = p[175] * qLamp * (1 - p[11]);
    H[H_NIRLAMPFLR] = (1 - p[97]) * p[175] * qLamp;
    H[H_LAMPRAD] = (p[174] + p[175]) * qLamp;
    H[H_GLOBAIR_A] = p[44] * iGlob * tauCovPar * p[6];
    H[H_GLOBAIR_B] = p[44] * iGlob * p[5];
    H[H_GLOBCOV] = (aCovPar * p[6] + aCovNir * p[5]) * iGlob;  // a80

    // FIR pair coefficients area*eps1*eps2*F12*sigma that depend on the screens (:476-632)
    const double sigma = p[2];
    const T tauThFir = 1 - thScr * (1 - p[81]);  // a81
    const T tauBlFir = 1 - blScr * (1 - p[91]);  // a82
    const double fPipe = 0.49 * pi * p[107] * p[105];
    const double t178 = p[178], t199 = p[199];
    H[H_C84] = p[3] * epsCovFir * (t178 * tauThFir * tauBlFir) * sigma;                          // can-covIn  x aCan
    H[H_C86] = p[3] * p[74] * (t178 * thScr * tauBlFir) * sigma;                                 // can-thScr  x aCan
    H[H_C108] = p[3] * p[85] * (t178 * blScr) * sigma;                                           // can-blScr  x aCan
    H[H_C88] = p[124] * p[104] * epsCovFir * (t199 * t178 * tauThFir * tauBlFir * 0.49) * sigma; // pipe-covIn x e35
    H[H_C90] = p[124] * p[104] * p[74] * (t199 * t178 * thScr * tauBlFir * 0.49) * sigma;        // pipe-thScr x e35
    H[H_C93] = p[95] * epsCovFir * (t199 * t178 * tauThFir * tauBlFir * (1 - fPipe)) * sigma;    // flr-covIn  x e35
    H[H_C95] = p[95] * p[74] * (t199 * t178 * thScr * tauBlFir * (1 - fPipe)) * sigma;           // flr-thScr  x e35
    H[H_C106] = p[95] * p[85] * (t199 * t178 * blScr * (1 - fPipe)) * sigma;                     // flr-blScr  x e35
    H[H_C107] = p[124] * p[104] * p[85] * (t199 * t178 * blScr * 0.49) * sigma;                  // pipe-blScr x e35
    H[H_C96] = p[74] * epsCovFir * thScr * sigma;                                                // thScr-covIn
    H[H_C102] = p[181] * p[182] * p[74] * (thScr * tauBlFir) * sigma;                            // lamp-thScr
    H[H_C103] = p[181] * p[182] * epsCovFir * (tauThFir * tauBlFir) * sigma;                     // lamp-covIn
    H[H_C109] = blScr * p[85] * p[74] * thScr * sigma;                                           // blScr-thScr
    H[H_C110] = blScr * p[85] * epsCovFir * tauThFir * sigma;                                    // blScr-covIn
    H[H_C112] = p[181] * p[182] * p[85] * blScr * sigma;                                         // lamp-blScr
    H[H_TSKY4] = glg_sq(glg_sq(d[5] + GLG_C2K));

    // ventilation (:698-779).  a126 (side vents) is hard-wired to 0 in the reference, so a134=0 and
    // a137=(1-cLeakTop)*fLeakage for both if_else branches; a133 reduces to its wind term.
    const double tOut = d[1], wind = d[4];
    const T aRoofU = u[3] * p[55];
    const double cD = p[59], cW = p[61];
    const T v132a = u[3] * p[55] * cD / (2. * p[46]);
    const T a133 = cD / p[46] * sqrt(1e-8 + (glg_sq(aRoofU) * cW * (wind * wind)));
    const double fLeak = (wind < p[205]) ? p[205] * p[60] : p[60] * wind;
    const T scrMax = fmax(thScr, blScr);
    const bool roofOnly = (1.0 >= p[8]);  // a127 = 1
    H[H_TOUT] = tOut;
    H[H_TOUT_2K] = tOut + 2 * GLG_C2K;
    H[H_CW_WIND2] = cW * (wind * wind);
    H[H_VR_A] = roofOnly ? p[57] * v132a : p[57] * scrMax * v132a;
    H[H_VR_B] = roofOnly ? p[204] * fLeak : p[57] * (1 - scrMax) * a133 + p[204] * fLeak;
    const double fVentSide = (1 - p[204]) * fLeak;  // a137 (+p57*0)
    H[H_FVENTSIDE_ABS] = fabs(fVentSide);

    // screen air flux factors (:801-809)
    H[H_THK] = thScr * p[84];
    H[H_BLK] = blScr * p[94];
    H[H_1MTH] = 1. - thScr;
    H[H_1MBL] = 1. - blScr;

    // convection coefficients (:835-876)
    H[H_17TH] = 1.7 * thScr;
    H[H_17BL] = 1.7 * blScr;
    H[H_HEC_AIROUT] = fabs(p[111] * p[23] * fVentSide);
    H[H_HEC_COVEOUT] = fabs(p[47] / p[46] * (p[51] + p[52] * pow(wind, p[53])));
    H[H_TSOOUT] = d[6];

    // stomata (:940-954)
    const T sRs = 1. / (1. + exp(p[43] * (rCan - p[40])));
    H[H_CEVAP3] = p[20] * (1. - sRs) + p[19] * sRs;
    H[H_CEVAP4] = p[22] * (1. - sRs) + p[21] * sRs;
    H[H_RS] = p[42] * ((rCan + p[17]) / (rCan + p[18]));

    // vapour / CO2 exchange with outside (:1019-1024,1205-1209)
    H[H_VPOUT_T] = d[2] / (tOut + (GLG_C2K + GLG_C2K_F32_DELTA));
    H[H_MVAIROUT_C] = 0.002165 * fabs(fVentSide);
    H[H_MCEXT] = u[1] * p[109] / p[46];
    H[H_CO2OUT] = d[3];

    // actuators (:1216,1255) ; lamp node: a37 - (a77+a75+a72+a55+a69) - a233 with a77's definition folded in
    H[H_HBOIL] = u[0] * p[108] / p[46];
    H[H_LAMPNET] = qLamp - (p[174] + p[175]) * qLamp - p[186] * qLamp;
    H[H_HECIN] = p[50] * p[47] / p[46];  // = K_HECIN
    H[H_ZERO] = 0.0;
}

// ---------------------------------------------------------------------------------------------------------
// glg_rhs: S[i] = dx_i/dt.  x: 28 stage-state values (x[27] unused).  KV/CV/HV: indexable constant sets.
// GENERAL adds the terms that are zero for the default parameter table; they need raw p,u,d.
//
// Written as a stream: every flux is added to the balance sums of its two nodes as soon as it exists, so only
// the 15 node sums and the current flux are live (the reference's ODE() sums ~10 aux values per state at the
// end, which would keep ~60 fluxes = 120 registers alive across the whole evaluation).
// ---------------------------------------------------------------------------------------------------------
// Returns the transient-stiffness estimate of the graded integrator (same rule as glg_grp_airflow / glgo_stiffness); unused
// by fixed-step callers.
template <bool GENERAL, class KV, class CV, class HV, class P>
GLG_HD double glg_rhs(const KV &K, const CV &C, const HV &H, const P &p, const double *u, const double *d,
                      const double *x, double *S) {
    const double tAir = x[2], tTop = x[3], tCan = x[4], tCovIn = x[5], tCovE = x[6];
    const double tThScr = x[7], tFlr = x[8], tPipe = x[9], tLamp = x[17], tBlScr = x[20];

    // ---- soil chain and the trivial states first (their inputs die early)
    {
        const double hFlrSo1 = K[K_HFLRSO1] * (tFlr - x[10]);
        const double hSo12 = K[K_HSO12] * (x[10] - x[11]);
        const double hSo23 = K[K_HSO23] * (x[11] - x[12]);
        const double hSo34 = K[K_HSO34] * (x[12] - x[13]);
        const double hSo45 = K[K_HSO45] * (x[13] - x[14]);
        const double hSo5Out = K[K_HSO5OUT] * (x[14] - H[H_TSOOUT]);
        S[10] = K[K_INVCAPSO1] * (hFlrSo1 - hSo12);
        S[11] = K[K_INVCAPSO2] * (hSo12 - hSo23);
        S[12] = K[K_INVCAPSO3] * (hSo23 - hSo34);
        S[13] = K[K_INVCAPSO4] * (hSo34 - hSo45);
        S[14] = K[K_INVCAPSO5] * (hSo45 - hSo5Out);
        S[21] = (1. / 86400.) * (tCan - x[21]);
        S[26] = (1. / 86400.) * tCan;
        S[27] = 1. / 86400.;
    }
    // node balance sums [W m-2] / [kg m-2 s-1] / [mg m-2 s-1]
    double sFlr = -(K[K_HFLRSO1] * (tFlr - x[10]));
    double sAir, sTop, sCan, sCovIn, sCovE, sThScr, sPipe, sLamp, sBlScr, sGroPipe, sIntLamp = 0.0;

    // ---- canopy extinction, PAR and NIR absorption (:299-470)
    const double lai = C[C_SLA] * x[23];
    const double e35 = glg_exp(-K[K_KFIR] * lai);
    const double aCan = 1 - e35;
    double parCan;  // a191 [umol m-2 s-1], consumed by photosynthesis
    {
        const double e32 = glg_exp(-K[K_K1PAR] * lai);
        const double e33 = GENERAL ? glg_exp(-K[K_K2PAR] * lai) : e32;  // k1Par == k2Par in the nominal structure
        const double e34 = glg_exp(-K[K_KNIR] * lai);
        const double gPar = (1 - e32) + e32 * K[K_RHOFLRPAR] * (1 - e33);
        parCan = H[H_PARUMOL] * gPar;
        const double parLampCanW = H[H_PARLAMP_W] * gPar;    // a55
        const double parLampFlrW = H[H_PARLAMPFLR_W] * e32;  // a75
        const double rhoCovNir = H[H_RHOCOVNIR];
        const double rhoHat = K[K_RHOCANNIR] * (1 - e34);
        const double den1 = glg_rcp(1. - rhoCovNir * rhoHat);
        const double tCC = H[H_TAUHATCOVNIR] * e34 * den1;
        const double rUp = rhoCovNir + H[H_TAUHAT2] * rhoHat * den1;
        const double rDn = rhoHat + e34 * e34 * rhoCovNir * den1;
        const double den2 = glg_rcp(1. - rDn * K[K_RHOFLRNIR]);
        const double aFlrNir = tCC * K[K_TAUHATFLRNIR] * den2;
        const double rCCF = rUp + tCC * tCC * K[K_RHOFLRNIR] * den2;
        const double aCanNir = 1 - aFlrNir - rCCF;
        const double nirLampCan = H[H_NIRLAMPCAN] * (1 - e34), nirLampFlr = H[H_NIRLAMPFLR] * e34;
        sCan = H[H_PARCAN_W] * gPar + H[H_NIRSUN] * aCanNir + nirLampCan;               // a54+a55+a68+a69
        sFlr += H[H_PARFLR_W] * e32 + H[H_NIRSUN] * aFlrNir + nirLampFlr;               // a74+a75+a71+a72
        sAir = (H[H_LAMPRAD] - parLampCanW - nirLampCan - parLampFlrW - nirLampFlr)     // a77
               + (H[H_GLOBAIR_A] + H[H_GLOBAIR_B] * (aCanNir + aFlrNir));               // a79
    }

    // ---- FIR exchange (:493-632): coefficient * (T1^4 - T2^4), added to both nodes at once
    {
        const double q4Can = glg_sq(glg_sq(tCan + GLG_C2K)), q4CovIn = glg_sq(glg_sq(tCovIn + GLG_C2K));
        const double q4ThScr = glg_sq(glg_sq(tThScr + GLG_C2K)), q4Flr = glg_sq(glg_sq(tFlr + GLG_C2K));
        const double q4Pipe = glg_sq(glg_sq(tPipe + GLG_C2K)), q4Lamp = glg_sq(glg_sq(tLamp + GLG_C2K));
        const double q4BlScr = glg_sq(glg_sq(tBlScr + GLG_C2K));
        double f;
        f = aCan * H[H_C84] * (q4Can - q4CovIn);   sCan -= f; sCovIn = f;
        f = aCan * H[H_C86] * (q4Can - q4ThScr);   sCan -= f; sThScr = f;
        f = aCan * K[K_C87] * (q4Can - q4Flr);     sCan -= f; sFlr += f;
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
        sCovE = H[H_GLOBCOV] - K[K_C98] * (glg_sq(glg_sq(tCovE + GLG_C2K)) - H[H_TSKY4]);  // a80 - a98
        if (GENERAL) {
            // Terms that are identically zero for the default table: sky FIR through the roof (tauRfFir p70),
            // grow-pipe FIR (epsGroPipe p165), interlight FIR/convection (p194,p195,p198).  Written plainly.
            const double sigma = p[2];
            const double pi = 3.14159265358979323846;
            const double thScr = u[2], blScr = u[5];
            const double tauCovFir = p[70];
            const double tauThFir = 1 - thScr * (1 - p[81]), tauBlFir = 1 - blScr * (1 - p[91]);
            const double fPipe = 0.49 * pi * p[107] * p[105];
            const double q4Sky = H[H_TSKY4];
            const double tIntLamp = x[18];
            const double q4Int = glg_sq(glg_sq(tIntLamp + GLG_C2K)), q4Gro = glg_sq(glg_sq(x[19] + GLG_C2K));
            const double f85 = aCan * p[3] * p[4] * (p[178] * tauCovFir * tauThFir * tauBlFir) * sigma * (q4Can - q4Sky);
            const double f89 = p[124] * p[104] * p[4] * (p[199] * p[178] * tauCovFir * tauThFir * 0.49 * e35) * sigma * (q4Pipe - q4Sky);
            const double f94 = p[95] * p[4] * (p[199] * p[178] * tauCovFir * tauThFir * tauBlFir * (1 - fPipe) * e35) * sigma * (q4Flr - q4Sky);
            const double f97 = p[74] * p[4] * (tauCovFir * thScr) * sigma * (q4ThScr - q4Sky);
            const double f104 = p[181] * p[182] * p[4] * (tauCovFir * tauThFir * tauBlFir) * sigma * (q4Lamp - q4Sky);
            const double f111 = blScr * p[85] * p[4] * (tauCovFir * tauThFir) * sigma * (q4BlScr - q4Sky);
            const double f105 = p[169] * p[165] * p[3] * sigma * (q4Gro - q4Can);
            const double upF = 1 - glg_exp(-p[203] * (1 - p[189]) * lai);  // a113
            const double dnF = 1 - glg_exp(-p[203] * p[189] * lai);        // a114
            const double ci = p[194] * p[195] * sigma;
            const double f115 = ci * p[95] * ((1 - fPipe) * (1 - dnF)) * (q4Int - q4Flr);
            const double f116 = ci * p[104] * (fPipe * (1 - dnF)) * (q4Int - q4Pipe);
            const double f117 = ci * p[3] * (dnF + upF) * (q4Int - q4Can);
            const double f118 = ci * p[183] * ((1 - upF) * p[181]) * (q4Int - q4Lamp);
            const double f119 = ci * p[85] * (blScr * p[178] * (1 - upF)) * (q4Int - q4BlScr);
            const double f120 = ci * p[74] * (thScr * tauBlFir * p[178] * (1 - upF)) * (q4Int - q4ThScr);
            const double f121 = ci * (1 - p[70] - p[67]) * (tauThFir * tauBlFir * p[178] * (1 - upF)) * (q4Int - q4CovIn);
            const double f122 = ci * p[4] * (tauCovFir * tauThFir * tauBlFir * p[178] * (1 - upF)) * (q4Int - q4Sky);
            const double hIntLampAir = fabs(p[198]) * (tIntLamp - tAir);
            sAir += hIntLampAir;
            sCan += -f85 + f105 + f117;
            sCovIn += f121;
            sThScr += -f97 + f120;
            sFlr += -f94 + f115;
            sPipe += -f89 + f116;
            sLamp += -f104 + f118;
            sIntLamp = -hIntLampAir - f122 - f121 - f120 - f116 - f119 - f115 - f117 - f118;
            sGroPipe = -f105;
            sBlScr += -f111 + f119;
        } else {
            sGroPipe = 0.0;
        }
    }
    S[18] = K[K_INVCAPINTLAMP] * sIntLamp;
    {   // conduction through the cover, lamp and pipe convection, cover-outside convection
        const double hCovInCovE = K[K_HCOV] * (tCovIn - tCovE);
        sCovIn -= hCovInCovE;
        sCovE += hCovInCovE - H[H_HEC_COVEOUT] * (tCovE - H[H_TOUT]);
        S[6] = K[K_INVCAPCOV] * sCovE;
        const double hLampAir = K[K_HLAMPAIR] * (tLamp - tAir);
        sLamp -= hLampAir;
        sAir += hLampAir;
        S[17] = K[K_INVCAPLAMP] * sLamp;
        const double hPipeAir = fabs(K[K_PIPEAIR]) * glg_pow(fabs(tPipe - tAir + 1e-10), 0.32) * (tPipe - tAir);
        sPipe -= hPipeAir;
        sAir += hPipeAir;
        S[9] = K[K_INVCAPPIPE] * sPipe;
        const double tGroPipe = x[19];
        const double hGroPipeAir = fabs(K[K_GROPIPEAIR]) * glg_pow(fabs(tGroPipe - tAir + 1e-10), 0.32) * (tGroPipe - tAir);
        sAir += hGroPipeAir;
        S[19] = K[K_INVCAPGROPIPE] * (sGroPipe - hGroPipeAir);
        const double hCanAir = fabs(K[K_2ALFA] * lai) * (tCan - tAir);
        sCan -= hCanAir;
        sAir += hCanAir;
        const double hecFlr = (tFlr > tAir) ? 1.7 * glg_cbrt(fabs(tFlr - tAir + 1e-10))
                                            : 1.3 * glg_sqrt(glg_sqrt(fabs(tAir - tFlr + 1e-10) + 1e-300));
        const double hAirFlr = hecFlr * (tAir - tFlr);
        sAir -= hAirFlr;
        S[8] = K[K_INVCAPFLR] * (sFlr + hAirFlr);
    }

    // ---- ventilation through the roof (:733-771) and air flux through the screens (:787-814)
    const double tOut = H[H_TOUT];
    const double vpAir = x[15], vpTop = x[16];
    const double tkAir = tAir + GLG_C2K, tkTop = tTop + GLG_C2K;
    const double rAir = glg_rcp(tkAir), rTop = glg_rcp(tkTop);
    double aVentRoof, aScr;
    {
        const double sVent = glg_sqrt(fabs(K[K_GHVENT] * (tAir - tOut) * glg_rcp(tAir + H[H_TOUT_2K]) + H[H_CW_WIND2]) + 1e-300);
        aVentRoof = fabs(H[H_VR_A] * sVent + H[H_VR_B]);  // |a136|
        const double rhoTop = K[K_RHOC] * rTop, rhoAir = K[K_RHOC] * rAir;
        const double rhoMean = 0.5 * (rhoTop + rhoAir);
        const double rMean = glg_rcp(rhoMean);
        const double buoy = K[K_HALFG] * rhoMean * fabs(rhoAir - rhoTop);
        const double pw66 = glg_pow(fabs(tAir - tTop + 1e-10), 0.66);
        const double oneMTh = H[H_1MTH], oneMBl = H[H_1MBL];
        const double fThScr = H[H_THK] * pw66 + (oneMTh * rMean) * glg_sqrt(buoy * oneMTh + 1e-10);
        const double fBlScr = H[H_BLK] * pw66 + (oneMBl * rMean) * glg_sqrt(buoy * oneMBl + 1e-10);
        aScr = fabs(fmin(fThScr, fBlScr));  // |a144|
    }
    // CO2 of the two air compartments (:1201-1209); the canopy uptake a216 is added after the crop block
    const double co2Air = x[0], co2Top = x[1];
    double sCo2Air;
    {
        const double mcAirTop = aScr * (co2Air - co2Top);
        S[1] = K[K_INVCAPCO2TOP] * (mcAirTop - aVentRoof * (co2Top - H[H_CO2OUT]));
        sCo2Air = H[H_MCEXT] - mcAirTop - H[H_FVENTSIDE_ABS] * (co2Air - H[H_CO2OUT]);
    }
    // sensible exchange air <-> top <-> outside
    {
        const double hAirOut = H[H_HEC_AIROUT] * (tAir - tOut);
        const double hAirTop = fabs(K[K_RHOCP]) * aScr * (tAir - tTop);
        const double hTopOut = fabs(K[K_RHOCP]) * aVentRoof * (tTop - tOut);
        sAir -= hAirOut + hAirTop;
        sTop = hAirTop - hTopOut;
    }
    // ---- screens and cover: convection + condensation share the cube-root HECs (:835-866, :999-1011)
    const double L = K[K_L];
    double sVpAir, sVpTop;
    {
        const double hec17Th = H[H_17TH], hec17Bl = H[H_17BL];
        const double c27 = glg_cbrt(fabs(tAir - tThScr + 1e-10));
        const double hecAirTh = hec17Th * c27;
        const double hAirThScr = fabs(hecAirTh) * (tAir - tThScr);
        const double mvAirThScr = glg_cond(hecAirTh, vpAir, glg_satvp_f(tThScr));
        const double hThScrTop = fabs(hec17Th * glg_cbrt(fabs(tThScr - tTop + 1e-10))) * (tThScr - tTop);
        sAir -= hAirThScr;
        sTop += hThScrTop;
        S[7] = K[K_INVCAPTHSCR] * (sThScr + hAirThScr + L * mvAirThScr - hThScrTop);
        const double c220 = glg_cbrt(fabs(tAir - tBlScr + 1e-10));
        const double hecAirBl = hec17Bl * c220;
        const double hAirBlScr = fabs(hecAirBl) * (tAir - tBlScr);
        const double mvAirBlScr = glg_cond(hecAirBl, vpAir, glg_satvp_f(tBlScr));
        const double hBlScrTop = fabs(hec17Bl * glg_cbrt(fabs(tBlScr - tTop + 1e-10))) * (tBlScr - tTop);
        sAir -= hAirBlScr;
        sTop += hBlScrTop;
        S[20] = K[K_INVCAPBLSCR] * (sBlScr + hAirBlScr + L * mvAirBlScr - hBlScrTop);
        const double hecTopCov = K[K_HECIN] * glg_cbrt(fabs(tTop - tCovIn + 1e-10));
        const double hTopCovIn = fabs(hecTopCov) * (tTop - tCovIn);
        const double mvTopCovIn = glg_cond(hecTopCov, vpTop, glg_satvp_f(tCovIn));
        sTop -= hTopCovIn;
        S[3] = K[K_INVCAPTOP] * sTop;
        S[5] = K[K_INVCAPCOV] * (sCovIn + hTopCovIn + L * mvTopCovIn);
        S[2] = K[K_INVCAPAIR] * sAir;
        sVpAir = -mvAirThScr - mvAirBlScr;
        sVpTop = -mvTopCovIn;
    }
    // ---- air-borne vapour exchange (:1015-1024); airMv's float Kelvin offset handled by a first-order fix
    {
        const double rAirF = rAir - GLG_C2K_F32_DELTA * (rAir * rAir);  // 1/(tAir + 273.15f)
        const double rTopF = rTop - GLG_C2K_F32_DELTA * (rTop * rTop);
        const double vAirT = vpAir * rAirF, vTopT = vpTop * rTopF;
        const double mvAirTop = 0.002165 * aScr * (vAirT - vTopT);
        sVpTop += mvAirTop - 0.002165 * aVentRoof * (vTopT - H[H_VPOUT_T]);
        sVpAir -= mvAirTop + H[H_MVAIROUT_C] * (vAirT - H[H_VPOUT_T]);
        S[16] = (K[K_INVVPTOP] * tkTop) * sVpTop;
    }
    // ---- transpiration (:959-981)
    {
        const double vpd = glg_satvp_f(tCan) - vpAir;
        const double rfCo2 = fmin(1.5, 1. + H[H_CEVAP3] * glg_sq(K[K_ETAMGPPM] * co2Air - 200));
        const double rfVp = fmin(5.8, 1. + H[H_CEVAP4] * (vpd * vpd));
        const double rS = H[H_RS] * rfCo2 * rfVp;
        const double mvCanAir = vpd * (K[K_VEC] * lai * glg_rcp(K[K_RB] + rS));
        S[15] = (K[K_INVVPAIR] * tkAir) * (sVpAir + mvCanAir);
        S[4] = (K[K_INVCAPLEAF] * glg_rcp(lai)) * (sCan - L * mvCanAir);
    }

    // ---- photosynthesis (:1041-1097)
    const double cBuf = x[22], cLeaf = x[23], cStem = x[24], cFruit = x[25], tCan24 = x[21];
    double mcAirBuf;
    {
        const double j25 = lai * C[C_J25];                               // a192
        const double rj = C[C_J25] * glg_rcp(j25);
        const double gamma = rj * C[C_CGAMMA] * tCan + C[C_20CGAMMA] * (1 - rj);  // a193
        const double co2Stom = C[C_ETASTOM] * (K[K_PPMC] * tkAir * co2Air);       // a194 = eta * a138
        const double rCanK = glg_rcp(tCan + GLG_C2K);
        const double jPot = j25 * glg_exp(C[C_ARR1] * (1 - C[C_T25K] * rCanK)) * C[C_JPOTNUM] *
                            glg_inv1pexp(C[C_ARR2A] - C[C_ARR2B] * rCanK);  // a195
        const double jb = jPot + C[C_ALPHA] * parCan;
        const double jE = C[C_INV2THETA] * (jb - glg_sqrt(jb * jb - C[C_4THETAALPHA] * jPot * parCan + 1e-10));  // a196
        const double phot = jE * (co2Stom - gamma) * glg_rcp(4 * (co2Stom + 2 * gamma));                         // a197
        const double photNet = phot - phot * gamma * glg_rcp(co2Stom);                                           // a197-a198
        mcAirBuf = C[C_MCH2O] * glg_inv1pexp(5e-4 * (cBuf - C[C_CBUFMAX])) * photNet;                             // a200
    }
    // ---- carbohydrate flows (:1103-1188)
    {
        const double gT24 = 0.047 * tCan24 + 0.06;
        const double hT24 = glg_rcp((1. + glg_exp(-1.1587 * (tCan24 - C[C_T24MIN]))) * (1. + glg_exp(1.3904 * (tCan24 - C[C_T24MAX]))));
        const double hTCan = glg_rcp((1. + glg_exp(-0.869 * (tCan - C[C_TCANMIN]))) * (1. + glg_exp(0.5793 * (tCan - C[C_TCANMAX]))));
        const double sSum = x[26] * K[K_INVTENDSUM];
        const double sSum1 = sSum - 1.0;
        const double hTSum = 0.5 * (sSum + glg_sqrt(sSum * sSum + 1e-4)) - 0.5 * (sSum1 + glg_sqrt(sSum1 * sSum1 + 1e-4));
        const double flow = glg_inv1pexp(-5e-3 * (cBuf - C[C_CBUFMIN])) * hT24 * gT24;
        const double mcBufLeaf = flow * C[C_RGLEAF];
        const double mcBufStem = flow * C[C_RGSTEM];
        const double mcBufFruit = flow * hTCan * hTSum * C[C_RGFRUIT];
        const double mcBufAir = C[C_GLEAF] * mcBufLeaf + C[C_GSTEM] * mcBufStem + C[C_GFRUIT] * mcBufFruit;
        const double maint = C[C_MAINT] * glg_exp(C[C_LNQ10X] * (tCan24 - 25));
        const double mcLeafAir = maint * cLeaf * C[C_MLEAF];
        const double mcStemAir = maint * cStem * C[C_MSTEM];
        const double mcFruitAir = maint * cFruit * C[C_MFRUIT];
        // smoothHar(v, cutoff, 1e4, 5e4) = 5e4*(tanh(z)+1)/2, z = (2*4.6052/1e4)*(v-cutoff)/2  (:75-79,1184,1188)
        const double kHar = 2.0 * 4.6052 / 1e4;
        const double mcLeafHar = 5e4 * glg_inv1pexp(-kHar * (cLeaf - C[C_CLEAFMAX]));
        const double mcFruitHar = 5e4 * glg_inv1pexp(-kHar * (cFruit - C[C_CFRUITMAX]));
        S[22] = mcAirBuf - mcBufFruit - mcBufLeaf - mcBufStem - mcBufAir;
        S[23] = mcBufLeaf - mcLeafAir - mcLeafHar;
        S[24] = mcBufStem - mcStemAir;
        S[25] = mcBufFruit - mcFruitAir - mcFruitHar;
        const double mcAirCan = C[C_CO2RATIO] * (mcAirBuf - mcBufAir - (mcLeafAir + mcStemAir + mcFruitAir));  // a216
        S[0] = K[K_INVCAPCO2AIR] * (sCo2Air - mcAirCan);
    }
    const double lamCov = 2.0 * K[K_HCOV] * K[K_INVCAPCOV];
    const double lamTop = fabs(K[K_RHOCP]) * K[K_INVCAPTOP] * (1.5 * aScr + aVentRoof);
    const double lamGas = (aScr + aVentRoof) * K[K_INVCAPCO2TOP];
    return 1.07 * fmax(lamCov, fmax(lamTop, lamGas));
}

// Harvest-stiffness guard (same rule as the oracle's glgo_micro_steps): number of equal micro-steps a nominal RK4 substep
// of length h is split into, so that harvest moves an organ at most half a sigmoid window-width per micro-step.
#define GLG_MAX_MICRO 512
// graded integrator (integrator = 1): nominal substep s of a control interval is split in glg_graded_m(s) = 16, 8, 4 x4,
// 2 x6, then 1 (the controls jump at t = 0 and the fast modes relax within seconds: that is where an equal-substep grid commits
// its error; oracle: glgo_graded_m); any nominal substep is split in 1 + floor(h lambda_est / GLG_STIFF_CFL) (RK4's real-axis
// limit is 2.785).  Meant for n_sub = 260 (h = 3.46 s: the largest nominal step the cover pair's 0.653 1/s mode leaves unsplit
// with 3 % to spare is 3.58 s): 300 RK4 steps per interval.
#define GLG_GRADED_SUBSTEPS 12
GLG_HD int glg_graded_m(int s) { return s < 1 ? 16 : s < 2 ? 8 : s < 6 ? 4 : s < GLG_GRADED_SUBSTEPS ? 2 : 1; }
#define GLG_STIFF_CFL 2.5
#define GLG_STIFF_INV_CFL 0.4  // the rule multiplies by this constant (oracle and kernels alike)
template <class T>
GLG_HD T glg_harvest_lambda(T sigLeaf, T sigFruit) {  // sig = 1/(1+exp(-k (c - cMax)))
    return T(5e4 * (2.0 * 4.6052 / 1e4)) * fmax(sigLeaf, sigFruit);  // harvest speed in window-widths per second
}
GLG_HD int glg_micro_steps_from_lambda(double lam, double h) {
    const int m = 1 + (int)floor(2.0 * h * lam);
    return m > GLG_MAX_MICRO ? GLG_MAX_MICRO : (m < 1 ? 1 : m);  // m < 1 only for a NaN lambda (diverged env)
}
template <class CV>
GLG_HD int glg_micro_steps(const CV &C, double cLeaf, double cFruit, double h) {
    const double k = 2.0 * 4.6052 / 1e4;
    const double sL = glg_inv1pexp(-k * (cLeaf - (double)C[C_CLEAFMAX])), sF = glg_inv1pexp(-k * (cFruit - (double)C[C_CFRUITMAX]));
    return glg_micro_steps_from_lambda(glg_harvest_lambda(sL, sF), h);
}

// True when the default-structure (GENERAL=false) variant is exact for this parameter table.
template <class P>
GLG_HD bool glg_params_nominal_structure(const P &p) {
    const bool sky = (p[70] != 0.0);
    const bool gro = (p[169] * p[165] != 0.0);
    const bool intl = (p[194] * p[195] != 0.0) || (p[198] != 0.0);
    const bool kpar = (p[32] != p[33]);  // the fast variant evaluates exp(-k1Par*LAI) once
    return !(sky || gro || intl || kpar);
}

// scalar type of a constant set (double in parity mode, float in throughput mode); all sets passed to one unit
// function (glg_units.h) use the same type
template <class V>
using glg_scalar_t = typename std::remove_cv<typename std::remove_reference<decltype(std::declval<const V &>()[0])>::type>::type;

// index into K of the capacity scale the owner applies to state i's summed contributions; -1: 1.0 (the units
// already wrote a derivative), -2: the per-lane canopy scale written by U_PIPES
GLG_HD constexpr int glg_state_scale_index(int i) {
    return i == 0 ? (int)K_INVCAPCO2AIR : i == 1 ? (int)K_INVCAPCO2TOP : i == 2 ? (int)K_INVCAPAIR : i == 3 ? (int)K_INVCAPTOP
         : i == 4 ? -2 : (i == 5 || i == 6) ? (int)K_INVCAPCOV : i == 7 ? (int)K_INVCAPTHSCR : i == 8 ? (int)K_INVCAPFLR
         : i == 9 ? (int)K_INVCAPPIPE : i == 17 ? (int)K_INVCAPLAMP : i == 18 ? (int)K_INVCAPINTLAMP
         : i == 19 ? (int)K_INVCAPGROPIPE : i == 20 ? (int)K_INVCAPBLSCR : -1;
}
