// magprop_core.cuh -- per-walker arithmetic of the magprop likelihood hot path.
//
// One walker = one thread.  Everything here is straight-line FP64 code on
// registers plus a small per-thread node buffer; the kernels in
// magprop_kernels.cu wrap it.  (tests/hostsim compiles this same header with
// g++ to debug the algorithm in the GPU-less build container; that build is
// test infrastructure and is never loaded by the package.)
//
// Reference behaviour reproduced (file:line are relative to the reference):
//   init_conds            code/synthetic_datasets/funcs.py:51-71, magnetar/funcs.py:17-29
//   ODEs / odes           funcs.py:75-142, magnetar/funcs.py:33-101
//   luminosity stage      funcs.py:175-229, magnetar/funcs.py:157-210
//   interp1d + /1e50      funcs.py:233-236, magnetar/funcs.py:213-217
//   lnlike/lnprior/lnprob mcmc_eqns.py:5-81, magnetar/mcmc_eqns.py:6-119
//
// How the ODE system is solved (DESIGN.md section 3):
//   * eta1 + eta2 = 1, so dMdisc/dt = Mdot_fb(t) - Mdisc/tvisc is linear and
//     independent of omega.  It is evaluated in closed form,
//         Mdisc(t) = K S(u) + C exp(-(u-u0)),  u = (t+tfb)/tvisc,
//     with S tabulated to 7e-16 (disc_table.inc).  This removes the
//     -Mdisc/tvisc stiffness that makes explicit RK need 1e4..1e5 steps.
//   * the remaining scalar spin equation is integrated by Dormand-Prince 5(4)
//     with the Hairer-Norsett-Wanner PI step controller and 4th-order dense
//     output, evaluated at the grid nodes the data need.
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define MP_HD __host__ __device__ __forceinline__
#define MP_TABLE_QUALIFIER __device__ const __align__(128)
// NOT const on the device: a const __constant__ array with a visible initialiser is folded into
// immediates, and every FP64 immediate costs two extra MOVs; a mutable one stays a c[3][..] operand.
#define MP_CONST_QUALIFIER __constant__
#else
#define MP_CONST_QUALIFIER static const
#define MP_HD inline
#define MP_TABLE_QUALIFIER alignas(128) static const
#endif

#include "disc_table.inc"
#include "magprop_constants.hpp"

namespace mp {

constexpr int kWalkerOk = 0;
constexpr int kWalkerPriorReject = 1;
constexpr int kWalkerIntegratorFail = 2;
constexpr int kWalkerNonfiniteState = 4;
constexpr int kWalkerNonfiniteLnlike = 8;
constexpr int kWalkerDeferred = 16;   // internal: handed to the stiff-capable launch

// Device-side copy of mp_model_spec plus derived walker-independent constants.
struct Spec {
  double inertia;        // I
  double inv_inertia;
  double mdot_factor;
  double rhs_n, rhs_tv_per_R, rhs_k;       // tvisc = RdiscI * rhs_tv_per_R
  double lum_n, lum_tv_per_R, lum_k;
  double dipeff, propeff, f_beam;
  double omega2_breakup_rhs;   // omega^2 above which rot_param > breakup_rhs
  double omega2_breakup_lum;
  double sqrt_GMR;             // sqrt(GM*R): lever arm when Rm < R
  double kc;                   // rhs_k * c : capped when Rm*omega >= kc
  double Ccap;                 // kc^(3/2)/sqrt(GM): capped fastness = Ccap / sqrt(omega)
  double sGMkc;                // sqrt(GM*kc): capped lever = sGMkc / sqrt(omega)
  double sqrtGM, inv_sqrtGM;
  // explicit step, which integrates y = omega^-2 (see spin_g): doubled lever arms, 2n, and the
  // break-up boundary in y
  double sqrtGM2, sqrt_GMR2, sGMkc2, rhs_n2, y_breakup_rhs;
  // spin_g's scaling (see there): qa and ni factors, k c and R over GM^(1/3), lever-arm constants
  double g_qa, g_ni, g_kc, g_R, g_floor, g_cap;
  int lprop_binding_term;
  int bucciantini;             // RHS dipole torque of Bucciantini et al. 2006 (figure_3.py:142-143): classical x 4 (Rlc/Rm)^3
  double bucc_cap;             // 4/k^3: that factor where Rm is capped at k*Rlc
  int lum_dipole_only;         // the luminosity stage's Lprop is identically 0 (see make_spec): only Ldip is evaluated
  int unlog_mask;
  double rtol;
  double rtol_stiff;           // tolerance of the Radau error estimate
  double rtol_y;               // explicit variant: tolerance on y = omega^-2 (see make_spec)
  int max_steps;
};

// Grid nodes and data laid out for the kernel (device pointers).
struct DataView {
  int n_nodes;             // nodes the evaluation needs, ascending in time
  int n_data;
  const double* node_t;    // [n_nodes]
  // data sorted by time, pre-divided on the host so the chi-square loop has no division:
  //   residual (y - mod/1e50)/yerr = dat_ys - mod * dat_c
  const double* dat_ys;    // [n_data] y / yerr
  const double* dat_c;     // [n_data] 1e-50 / yerr
  const double* dat_dx;    // [n_data] x - t_lo            (0 when x is a grid node)
  const double* dat_w;     // [n_data] (x - t_lo)/(t_hi - t_lo): interpolation weight of the upper node
  const int* dat_lo;       // [n_data] index into node_t of the lower bracketing node
  double t_start;          // grid[0]: where the initial conditions hold
};

// ---- the disc-mass kernel function S(u) ----------------------------------
// Loads of the dataset / node program.  The kernels stage them in shared memory when they fit (then these are
// LDS through a generic pointer) and leave them in global memory otherwise, so a plain generic load is used
// rather than ld.global.nc.
MP_HD double ldd(const double* p) { return *p; }

MP_HD double ldg(const double* p) {
#if defined(__CUDA_ARCH__)
  return __ldg(p);
#else
  return *p;
#endif
}

MP_HD int64_t dbits(double x) {
#if defined(__CUDA_ARCH__)
  return __double_as_longlong(x);
#else
  union { double d; int64_t i; } v; v.d = x; return v.i;
#endif
}
MP_HD double bitsd(int64_t i) {
#if defined(__CUDA_ARCH__)
  return __longlong_as_double(i);
#else
  union { double d; int64_t i; } v; v.i = i; return v.d;
#endif
}

// Locate u in the table: row pointer and local coordinate s in [-1,1).
struct TableAt {
  const double* row;
  double s;
};

MP_HD int dhi(double x) { return (int)(dbits(x) >> 32); }

// 1 + f, where f in [0,1) is the part of u's mantissa below its top K bits (the position of u inside the K-bit
// sub-interval of its binade): the mantissa shifted up by K bits under a zero exponent.
template <int K>
MP_HD double mantissa_below(double u) {
#if defined(__CUDA_ARCH__)
  const unsigned uh = (unsigned)__double2hiint(u), ul = (unsigned)__double2loint(u);
  return __hiloint2double((int)((__funnelshift_l(ul, uh, K) & 0x000fffffu) | 0x3ff00000u), (int)(ul << K));
#else
  const uint64_t ub = (uint64_t)dbits(u);
  return bitsd((int64_t)(((ub << K) & 0x000fffffffffffffULL) | 0x3ff0000000000000ULL));
#endif
}

// Rows are laid out by (binade, sub-interval), i.e. by the top 11 + MP_DISC_NSUB_LOG2 bits of u, so
// the row index is one shift and one subtraction of the high word.  The local coordinate is
// (u - centre) * 2^(NSUB_LOG2 + 1 - e) with the centre of the sub-interval, read off the mantissa.  Always yields a loadable row (row 0 when u is outside the
// table -- u <= 0, subnormal, NaN/inf included) so callers can evaluate unconditionally and patch
// the rare outside case afterwards.
MP_HD bool table_locate_safe(double u, TableAt& ta) {
  const int hi = dhi(u);
  const int sh = 20 - MP_DISC_NSUB_LOG2;
  const unsigned idx = (unsigned)((hi >> sh) - ((1023 + MP_DISC_EMIN) << MP_DISC_NSUB_LOG2));
  const bool in = idx < (unsigned)((MP_DISC_EMAX - MP_DISC_EMIN + 1) << MP_DISC_NSUB_LOG2);
  ta.row = &mp_disc_table[in ? idx : 0u][0];
  // (the local coordinate from the mantissa bits: see table_locate_fast)
  ta.s = fma(mantissa_below<MP_DISC_NSUB_LOG2>(u), 2.0, -3.0);
  return in;
}
MP_HD bool table_locate(double u, TableAt& ta) { return table_locate_safe(u, ta); }

// The same for the explicit integrator's table (mp_disc_fast: S alone, lower degree on more sub-intervals per binade).
MP_HD bool table_locate_fast(double u, TableAt& ta) {
  const int hi = dhi(u);
  const int sh = 20 - MP_DISC_FAST_NSUB_LOG2;
  const unsigned idx = (unsigned)((hi >> sh) - ((1023 + MP_DISC_EMIN) << MP_DISC_FAST_NSUB_LOG2));
  const bool in = idx < (unsigned)((MP_DISC_EMAX - MP_DISC_EMIN + 1) << MP_DISC_FAST_NSUB_LOG2);
  ta.row = &mp_disc_fast[in ? idx : 0u][0];
  // The local coordinate straight from the mantissa: with u = 2^e (1 + (j + f)/NSUB), f in [0,1) is the mantissa
  // below its top NSUB_LOG2 bits; shifted up by that many bits under a zero exponent it reads m = 1 + f, and
  // s = 2f - 1 = 2m - 3 -- exactly the (u - centre) * 2^(NSUB_LOG2 + 1 - e) of the generic form (both are exact),
  // in four instructions instead of eight.
  ta.s = fma(mantissa_below<MP_DISC_FAST_NSUB_LOG2>(u), 2.0, -3.0);
  return in;
}

// degree-10 polynomial, split into even/odd halves for ILP
MP_HD double poly10(const double* c, double s) {
  const double s2 = s * s;
  double ev = ldg(c + 10);
  double od = ldg(c + 9);
  ev = fma(ev, s2, ldg(c + 8));
  od = fma(od, s2, ldg(c + 7));
  ev = fma(ev, s2, ldg(c + 6));
  od = fma(od, s2, ldg(c + 5));
  ev = fma(ev, s2, ldg(c + 4));
  od = fma(od, s2, ldg(c + 3));
  ev = fma(ev, s2, ldg(c + 2));
  od = fma(od, s2, ldg(c + 1));
  ev = fma(ev, s2, ldg(c + 0));
  return fma(od, s, ev);
}

// Two adjacent table coefficients in one 16-byte load (rows are 16-byte aligned).
struct alignas(16) Pair { double x, y; };
MP_HD Pair ld2(const double* p) {
#if defined(__CUDA_ARCH__)
  const double2 v = __ldg(reinterpret_cast<const double2*>(p));
  Pair r; r.x = v.x; r.y = v.y; return r;
#else
  Pair r; r.x = p[0]; r.y = p[1]; return r;
#endif
}

// poly10 with paired loads: (c0,c1) (c2,c3) ... (c10,pad) feed the even and the odd chain.
MP_HD double poly10p(const double* c, double s, double s2) {
  const Pair p5 = ld2(c + 10), p4 = ld2(c + 8), p3 = ld2(c + 6), p2 = ld2(c + 4), p1 = ld2(c + 2), p0 = ld2(c);
  double ev = p5.x, od = p4.y;
  ev = fma(ev, s2, p4.x);
  od = fma(od, s2, p3.y);
  ev = fma(ev, s2, p3.x);
  od = fma(od, s2, p2.y);
  ev = fma(ev, s2, p2.x);
  od = fma(od, s2, p1.y);
  ev = fma(ev, s2, p1.x);
  od = fma(od, s2, p0.y);
  ev = fma(ev, s2, p0.x);
  return fma(od, s, ev);
}

// A row of mp_disc_fast (degree MP_DISC_FAST_DEG, see tools/gen_disc_table.py).
MP_HD double polyfast(const double* c, double s, double s2) {
#if MP_DISC_FAST_DEG == 6
  const Pair p3 = ld2(c + 6), p2 = ld2(c + 4), p1 = ld2(c + 2), p0 = ld2(c);
  double ev = p3.x, od = p2.y;
  ev = fma(ev, s2, p2.x);
  od = fma(od, s2, p1.y);
  ev = fma(ev, s2, p1.x);
  od = fma(od, s2, p0.y);
  ev = fma(ev, s2, p0.x);
  return fma(od, s, ev);
#elif MP_DISC_FAST_DEG == 5      // (c0,c1) (c2,c3) (c4,c5): 48-byte rows
  const Pair p2 = ld2(c + 4), p1 = ld2(c + 2), p0 = ld2(c);
  double ev = p2.x, od = p2.y;
  ev = fma(ev, s2, p1.x);
  od = fma(od, s2, p1.y);
  ev = fma(ev, s2, p0.x);
  od = fma(od, s2, p0.y);
  return fma(od, s, ev);
#else
#error "mp_disc_fast: degree 5 or 6"
#endif
}

// S outside the table (rare): convergent series below 2^-10, asymptotic above 2^22.
// Kept out of line so the hot stage loop stays small.
#if defined(__CUDACC__)
__device__ __host__ __noinline__
#endif
static double disc_S_outside(double u) {
  if (!(u > 0.0) || !(u < 1.0e300)) return NAN;
  const int e = ((dhi(u) >> 20) & 0x7ff) - 1023;
  if (e > MP_DISC_EMAX) {  // next term 16/u^3 < 3e-19
    const double iu = 1.0 / u;
    const double c = cbrt(iu);
    const double p = iu * c * c;  // u^(-5/3)
    return p * fma(fma(40.0 / 9.0, iu, 5.0 / 3.0), iu, 1.0);
  }
  // e^-u u^(-2/3) sum_k u^k / (k! (k-2/3))
  const double c = cbrt(u);
  double sum = -1.5, term = 1.0;
  for (int k = 1; k <= 6; ++k) {
    term *= u / k;
    sum += term / (k - 2.0 / 3.0);
  }
  return exp(-u) * sum / (c * c);
}

MP_HD double disc_S(double u) {
  TableAt ta;
  if (table_locate(u, ta)) return poly10(ta.row, ta.s);
  return disc_S_outside(u);
}

// ---- per-walker constants ---------------------------------------------------
struct Walker {
  // disc mass: M(t) = K*S(u) + C*exp(-(u-u0)), u = t*inv_tv + eps
  double inv_tv, eps, u0, K, C, M_init;
  double u_late;   // for u >= u_late the transient C*exp(u0-u) is below 1e-18 of K*S(u): M = K*S(u)
  double Kq;       // K^(-1/7): late-phase M^(-1/7) = Kq * Q(u)
  // right-hand side
  double A_rm;     // Rm(uncapped) = A_rm * M^(-2/7)
  double Cw;       // w(uncapped)  = Cw * M^(-3/7) * omega
  double Ccap;     // w(capped)    = Ccap / sqrt(omega)
  double kc;       // k*c : capped when Rm*omega >= k*c
  double sGMA;     // sqrt(GM*A_rm): lever(uncapped) = sGMA * M^(-1/7)
  double sGMkc;    // sqrt(GM*k*c):  lever(capped)   = sGMkc / sqrt(omega)
  double Cdip_I;   // mu^2/(6c^3)/I
  double Cdip_I2;  // 2 mu^2/(6c^3)/I : d(omega^-2)/dt of pure dipole spin-down
  // folded forms used by the explicit step (spin_f): with qa = sqrtA * M^(-1/7),
  //   Rm = qa^2,  w/omega = qa^3/sqrt(GM),  lever = sqrt(GM) qa,  N_acc/I = -lever * ni * tanh
  double sqrtA;    // sqrt(A_rm)
  double KqA;      // Kq * sqrtA : late-phase qa = KqA * Q(u)
  double tvI;      // 1/(tvisc I) : ni = Mdisc * tvI
  double g_sqrtA, g_tvI;   // sqrtA and tvI in spin_g's scaling (explicit variant)
  double KtvI;     // K/(tvisc I) : late-phase ni = KtvI * S(u)
  // luminosity stage (its own alpha/cs7/k/n may differ from the RHS's)
  double l_inv_tv, l_A_rm, l_Cw, l_Ccap, l_kc;
  double l_sqrtA;     // sqrt(l_A_rm): with qa = l_sqrtA M^(-1/7): Rm = qa^2, w = qa^3 omega / sqrt(GM)
  double l_sGMkc;     // sqrt(GM l_kc)
  double l_GM_kc;     // GM / l_kc
  double Ldip_coef;   // mu^2/(6 c^3)
  double dipeff, propeff, f_beam;
  double omega0;
  int bad;         // non-finite / unphysical constants
};

// Accurate-but-slow x^(-1/7) (set-up code only).
MP_HD double pow_m17(double x) { return exp(log(x) * (-1.0 / 7.0)); }

// ---- hot-loop elementary functions -------------------------------------------------
// Hand-rolled so that every polynomial coefficient is a constant-bank operand of
// its DFMA (libdevice's exp/log materialise ~40 immediates per call, which showed
// up as a quarter of all issued instructions in the first ncu profile).
MP_CONST_QUALIFIER double kExpC[13] = {   // 1/n!, n = 0..12
    1.0, 1.0, 1.0 / 2, 1.0 / 6, 1.0 / 24, 1.0 / 120, 1.0 / 720, 1.0 / 5040, 1.0 / 40320, 1.0 / 362880,
    1.0 / 3628800, 1.0 / 39916800, 1.0 / 479001600};
MP_CONST_QUALIFIER double kExpR[4] = {1.4426950408889634074,      // log2(e)
                                      6755399441055744.0,         // 2^52 + 2^51: round-to-nearest-integer shifter
                                      -6.93147180369123816490e-01,  // -ln2 (high part)
                                      -1.90821492927058770002e-10}; // -ln2 (low part)

// exp(x) to ~2e-16 relative for x in [-708, 709]; below -708 returns ~1e-308 (callers
// only ever multiply it by O(1e30) quantities that are already negligible there).
MP_HD double exp_c(double x) {
  double xc = (x < -708.0) ? -708.0 : x;
  xc = (xc > 709.0) ? 709.0 : xc;
  const double kd = fma(xc, kExpR[0], kExpR[1]);
  const int k = (int)(dbits(kd) & 0xffffffffLL);
  const double kf = kd - kExpR[1];
  double r = fma(kf, kExpR[2], xc);
  r = fma(kf, kExpR[3], r);
  const double r2 = r * r;
  double ev = kExpC[12], od = kExpC[11];
  ev = fma(ev, r2, kExpC[10]);
  od = fma(od, r2, kExpC[9]);
  ev = fma(ev, r2, kExpC[8]);
  od = fma(od, r2, kExpC[7]);
  ev = fma(ev, r2, kExpC[6]);
  od = fma(od, r2, kExpC[5]);
  ev = fma(ev, r2, kExpC[4]);
  od = fma(od, r2, kExpC[3]);
  ev = fma(ev, r2, kExpC[2]);
  od = fma(od, r2, kExpC[1]);
  ev = fma(ev, r2, kExpC[0]);
  const double p = fma(od, r, ev);
  const double res = bitsd(dbits(p) + ((int64_t)k << 52));
  return (x == x) ? res : x;
}

MP_CONST_QUALIFIER double kP17[9] = {   // m^(-1/7) on [1,2) in z = 2m - 3, 7.8e-9 relative
    0x1.e32f899a660a5p-1, -0x1.70241e1493922p-5, 0x1.187cfebc0ad9ap-7, -0x1.0b37570227f94p-9,
    0x1.17f49b665ef64p-11, -0x1.306c347674bdbp-13, 0x1.5b8846fafc617p-15, -0x1.fe4427ec39f39p-17,
    0x1.314098ac46cb2p-18};
MP_CONST_QUALIFIER double kP2b7[7] = {  // 2^(-b/7), b = 0..6
    0x1.0000000000000p+0, 0x1.cfbb031a741a5p-1, 0x1.a402feeb9c533p-1, 0x1.7c6a1f29e2ce6p-1,
    0x1.588cea3f093bep-1, 0x1.381147622f886p-1, 0x1.1aa59c4115e7ep-1};

// x^(-1/7) for normal positive x to ~4e-16: exponent split e = 7a + b, polynomial
// seed for the mantissa, one Newton step y += y (1 - m y^7) / 7.  NaN for x <= 0.
MP_HD double pow_m17_fast(double x) {
  const int64_t b = dbits(x);
  const int e = (int)((b >> 52) & 0x7ff) - 1023;
  const double m = bitsd((b & 0x000fffffffffffffLL) | 0x3ff0000000000000LL);
  const int ee = e + 1400;                 // positive for every normal exponent
  const int a = ee / 7;
  const int rem = ee - 7 * a;
  const double z = fma(2.0, m, -3.0);
  const double z2 = z * z;
  double ev = kP17[8], od = kP17[7];
  ev = fma(ev, z2, kP17[6]);
  od = fma(od, z2, kP17[5]);
  ev = fma(ev, z2, kP17[4]);
  od = fma(od, z2, kP17[3]);
  ev = fma(ev, z2, kP17[2]);
  od = fma(od, z2, kP17[1]);
  ev = fma(ev, z2, kP17[0]);
  double y = fma(od, z, ev);
  const double y2 = y * y, y4 = y2 * y2;
  const double y7 = y4 * y2 * y;
  y = fma(y * (1.0 / 7.0), fma(-m, y7, 1.0), y);
  // scale by 2^(-(a-200)) * 2^(-rem/7)
  const double sc = bitsd((int64_t)(1023 - (a - 200)) << 52);
  const double res = y * kP2b7[rem] * sc;
  const bool ok = (b > 0) && (((b >> 52) & 0x7ff) - 1 < 0x7fe);   // positive, normal, finite
  return ok ? res : NAN;
}

// pow_m17_fast out of line, for the rare arguments the seeded form below hands over.
#if defined(__CUDACC__)
__device__ __host__ __noinline__
#endif
static double pow_m17_cold(double x) { return pow_m17_fast(x); }

// x^(-1/7) from a single-precision seed (two MUFU operations, ~3e-7) and one third-order
// correction y (1 + e/7 + 4 e^2/49), e = 1 - x y^7: remainder 0.06 e^3 ~ 3e-19.  A third of the
// FP64 work of pow_m17_fast and none of its integer exponent arithmetic.  Arguments outside the
// single-precision range (and x <= 0, NaN) take pow_m17_fast.
MP_HD double pow_m17_seeded(double x) {
#if defined(__CUDA_ARCH__) && !defined(MP_POW_CVT)
  // double <-> float through the bit patterns (the F2F conversions have ~19 cycles of latency each,
  // measured; the seed only needs the leading 24 bits, truncated) and the bare MUFU operations.
  const long long xb = __double_as_longlong(x);
  const unsigned hi = (unsigned)(xb >> 32), lo = (unsigned)xb;
  if (!(hi - (897u << 20) < (253u << 20))) return pow_m17_cold(x);   // outside float range, x <= 0, NaN
  // ((hi - (896 << 20)) << 3) | (lo >> 29): one funnel shift and one add (896 << 23 = -0x40000000 mod 2^32)
  const float xf = __uint_as_float(__funnelshift_l(lo, hi, 3) + 0x40000000u);
  float lg, sf;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(xf));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(sf) : "f"(lg * (-1.0f / 7.0f)));
  const unsigned fb = __float_as_uint(sf);
  const double y = __hiloint2double((int)((fb >> 3) + (896u << 20)), (int)(fb << 29));
#else
  const float xf = (float)x;
  const float sf = exp2f(log2f(xf) * (-1.0f / 7.0f));
  if (!(xf > 1.0e-36f && xf < 1.0e37f)) return pow_m17_cold(x);
  const double y = (double)sf;
#endif
  const double y2 = y * y, y4 = y2 * y2;
  const double e = fma(-x, (y4 * y2) * y, 1.0);
  return fma(y * e, fma(e, 4.0 / 49.0, 1.0 / 7.0), y);
}

// The same with the first-order correction only, y (1 + e/7): remainder (4/49) e^2 ~ 4e-13 with the seed's
// e ~ 2e-6 -- three orders below the step's tolerance, which is all the integrator's disc block needs.
MP_HD double pow_m17_seeded1(double x) {
#if defined(__CUDA_ARCH__) && !defined(MP_POW_CVT)
  const long long xb = __double_as_longlong(x);
  const unsigned hi = (unsigned)(xb >> 32), lo = (unsigned)xb;
  if (!(hi - (897u << 20) < (253u << 20))) return pow_m17_cold(x);   // outside float range, x <= 0, NaN
  // ((hi - (896 << 20)) << 3) | (lo >> 29): one funnel shift and one add (896 << 23 = -0x40000000 mod 2^32)
  const float xf = __uint_as_float(__funnelshift_l(lo, hi, 3) + 0x40000000u);
  float lg, sf;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(xf));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(sf) : "f"(lg * (-1.0f / 7.0f)));
  const unsigned fb = __float_as_uint(sf);
  const double y = __hiloint2double((int)((fb >> 3) + (896u << 20)), (int)(fb << 29));
#else
  const float xf = (float)x;
  const float sf = exp2f(log2f(xf) * (-1.0f / 7.0f));
  if (!(xf > 1.0e-36f && xf < 1.0e37f)) return pow_m17_cold(x);
  const double y = (double)sf;
#endif
  const double y2 = y * y, y4 = y2 * y2;
  const double e = fma(-x, (y4 * y2) * y, 1.0);
  return fma(y * (1.0 / 7.0), e, y);
}

// The two halves of pow_m17_seeded1 for a block of independent evaluations: the range test of every
// argument first, then the straight-line seeded power -- no branch between the chains, so the compiler
// can interleave them.
MP_HD bool pow_m17_seedable(double x) {
  const unsigned hi = (unsigned)(dbits(x) >> 32);
  return hi - (897u << 20) < (253u << 20);
}
MP_HD double pow_m17_seeded1_inrange(double x) {
#if defined(__CUDA_ARCH__) && !defined(MP_POW_CVT)
  const long long xb = __double_as_longlong(x);
  const unsigned hi = (unsigned)(xb >> 32), lo = (unsigned)xb;
  // ((hi - (896 << 20)) << 3) | (lo >> 29): one funnel shift and one add (896 << 23 = -0x40000000 mod 2^32)
  const float xf = __uint_as_float(__funnelshift_l(lo, hi, 3) + 0x40000000u);
  float lg, sf;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(xf));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(sf) : "f"(lg * (-1.0f / 7.0f)));
  const unsigned fb = __float_as_uint(sf);
  const double y = __hiloint2double((int)((fb >> 3) + (896u << 20)), (int)(fb << 29));
  const double y2 = y * y, y4 = y2 * y2;
  const double e = fma(-x, (y4 * y2) * y, 1.0);
  return fma(y * (1.0 / 7.0), e, y);
#else
  return pow_m17_seeded1(x);
#endif
}

MP_HD double rcp_fast(double x) {
#if defined(__CUDA_ARCH__)
  return __drcp_rn(x);
#else
  return 1.0 / x;
#endif
}
MP_HD double rsqrt_fast(double x) {
#if defined(__CUDA_ARCH__)
  return rsqrt(x);
#else
  return 1.0 / sqrt(x);
#endif
}

// pars = physical (B, P, MdiscI, RdiscI, epsilon, delta)
MP_HD void walker_setup(const Spec& sp, const double* pars, double dipeff, double propeff,
                        double f_beam, double t_start, Walker& w) {
  const double B = pars[0], P = pars[1], MdiscI = pars[2], RdiscI = pars[3];
  const double epsilon = pars[4], delta = pars[5];
  // init_conds: funcs.py:68-69
  w.M_init = MdiscI * kMsol;
  w.omega0 = kTwoPi / (1.0e-3 * P);
  const double mu = 1.0e15 * B * (kR * kR * kR);
  const double tv = RdiscI * sp.rhs_tv_per_R;
  const double M0 = delta * MdiscI * kMsol;
  w.inv_tv = 1.0 / tv;
  w.eps = epsilon;
  w.u0 = fma(t_start, w.inv_tv, epsilon);
  const double ce = cbrt(epsilon);
  w.K = M0 * ce * ce;
  w.C = w.M_init - w.K * disc_S(w.u0);
  // late phase: transient negligible (and u >= 1 so that S > 0 and Q is tabulated)
  w.u_late = INFINITY;
  w.Kq = 0.0;
  if (w.K > 0.0) {
    const double ua = fmax(w.u0 + 45.0, 1.0);
    const double ratio = fabs(w.C) * exp(w.u0 - ua) / (w.K * disc_S(ua));
    w.u_late = (ratio <= 1.0e-19) ? ua : ua + log(ratio * 1.0e19);
    w.u_late -= 6.9;                         // transient <= 1e-16 of K*S (S falls only as a power law)
    w.Kq = pow_m17(w.K);
  }
  const double mu47 = exp(log(mu) * (4.0 / 7.0));
  const double gm17 = exp(log(kGM) * (-1.0 / 7.0));
  const double base = mu47 * gm17;
  w.A_rm = base * exp(log(sp.mdot_factor * w.inv_tv) * (-2.0 / 7.0));
  w.Cw = w.A_rm * sqrt(w.A_rm) / sqrt(kGM);
  w.kc = sp.rhs_k * kC;
  w.Ccap = w.kc * sqrt(w.kc) / sqrt(kGM);
  w.sGMA = sqrt(kGM * w.A_rm);
  w.sqrtA = sqrt(w.A_rm);
  w.KqA = w.Kq * w.sqrtA;
  w.tvI = w.inv_tv * sp.inv_inertia;
  w.KtvI = w.K * w.tvI;
  w.g_sqrtA = w.sqrtA * sp.g_qa;
  w.g_tvI = w.tvI * sp.g_ni;
  w.sGMkc = sqrt(kGM * w.kc);
  w.Ldip_coef = (mu * mu) / (6.0 * (kC * kC * kC));
  w.Cdip_I = w.Ldip_coef * sp.inv_inertia;
  w.Cdip_I2 = 2.0 * w.Cdip_I;
  const double ltv = RdiscI * sp.lum_tv_per_R;
  w.l_inv_tv = 1.0 / ltv;
  w.l_A_rm = base * exp(log(sp.mdot_factor * w.l_inv_tv) * (-2.0 / 7.0));
  w.l_Cw = w.l_A_rm * sqrt(w.l_A_rm) / sqrt(kGM);
  w.l_kc = sp.lum_k * kC;
  w.l_Ccap = w.l_kc * sqrt(w.l_kc) / sqrt(kGM);
  w.l_sqrtA = sqrt(w.l_A_rm);
  w.l_sGMkc = sqrt(kGM * w.l_kc);
  w.l_GM_kc = kGM / w.l_kc;
  w.dipeff = dipeff;
  w.propeff = propeff;
  w.f_beam = f_beam;
  const double probe = w.K + w.C + w.A_rm + w.Cw + w.omega0 + w.l_A_rm + w.inv_tv;
  w.bad = !(isfinite(probe) && w.M_init > 0.0 && tv > 0.0 && ltv > 0.0 && epsilon > 0.0 &&
            delta >= 0.0 && w.omega0 > 0.0 && mu > 0.0);
}

// Disc mass at time t (closed form of funcs.py:126-129).
MP_HD double disc_mass(const Walker& w, double t) {
  const double u = fma(t, w.inv_tv, w.eps);
  TableAt ta;
  const double S = table_locate(u, ta) ? poly10p(ta.row, ta.s, ta.s * ta.s) : disc_S_outside(u);
  if (u >= w.u_late) return w.K * S;            // transient below 1e-16 of K S
  return fma(w.K, S, w.C * exp_c(w.u0 - u));
}

// Quantities of the RHS that depend on time only (through the disc mass).
struct DiscAt {
  double mdot;   // Mdisc/tvisc
  double q;      // Mdisc^(-1/7)
  double rm;     // uncapped Alfven radius  A_rm q^2
  double wq;     // uncapped fastness / omega  Cw q^3
};

MP_HD DiscAt disc_at(const Walker& w, double t) {
  const double u = fma(t, w.inv_tv, w.eps);
  TableAt ta;
  const bool in = table_locate(u, ta);
  double M, q;
  if (in && u >= w.u_late) {
    // late phase: both S and Q = S^(-1/7) from the same table row -- no exp, no log
    const double S = poly10(ta.row, ta.s);
    const double Q = poly10(ta.row + MP_DISC_ROW, ta.s);
    M = w.K * S;
    q = w.Kq * Q;
  } else {
    const double S = in ? poly10(ta.row, ta.s) : disc_S_outside(u);
    const double E = exp_c(w.u0 - u);
    M = fma(w.K, S, w.C * E);
    q = pow_m17_fast(M);
  }
  const double q2 = q * q;
  DiscAt d;
  d.mdot = M * w.inv_tv;
  d.q = q;
  d.rm = w.A_rm * q2;
  d.wq = w.Cw * q2 * q;
  return d;
}

// tanh to 4e-16 absolute (the torque needs absolute, not relative, accuracy).
MP_HD double tanh_abs(double x) {
  if (x > 19.1) return 1.0;
  const double e2 = exp_c(2.0 * x);
  return fma(-2.0, rcp_fast(e2 + 1.0), 1.0);
}

// d(omega)/dt: funcs.py:105-140 with the time-only factors hoisted into DiscAt.
//   Rm/Rc = Rm * omega^(2/3) / GM^(1/3)  =>  w = (Rm/Rc)^(3/2) = Rm^(3/2) omega / sqrt(GM)
//   capped (Rm >= k c/omega):  Rm = k c/omega,  w = (k c)^(3/2) / sqrt(GM omega)
//   lever arm sqrt(GM Rm):     uncapped sqrt(GM A_rm) q ;  capped sqrt(GM k c) / sqrt(omega)
//   Mdotacc - Mdotprop = (eta1 - eta2) Mdot = -tanh(n (w-1)) Mdot
MP_HD double spin_rhs(const Spec& sp, const Walker& w, const DiscAt& d, double omega) {
  double fast, lever;
  if (d.rm * omega >= w.kc) {
    const double r = rsqrt_fast(omega);
    fast = w.Ccap * r;
    lever = (w.kc >= kR * omega) ? w.sGMkc * r : sp.sqrt_GMR;
  } else {
    fast = d.wq * omega;
    lever = (d.rm >= kR) ? w.sGMA * d.q : sp.sqrt_GMR;
  }
  const double om2 = omega * omega;
  double nacc = 0.0;
  if (!(om2 > sp.omega2_breakup_rhs)) {
    const double th = tanh_abs(sp.rhs_n * (fast - 1.0));
    nacc = -lever * d.mdot * th;
  }
  double cdip = w.Cdip_I;
  if (sp.bucciantini) {
    const double q = kC / (omega * d.rm);                       // Rlc / Rm (uncapped)
    cdip *= (d.rm * omega >= w.kc) ? sp.bucc_cap : 4.0 * q * q * q;
  }
  return fma(-cdip * om2, omega, nacc * sp.inv_inertia);
}

// Luminosity stage at one node (erg/s, not yet /1e50): funcs.py:175-229.
struct Lum { double tot, prop, dip; };

MP_HD double rsqrt_pos(double x);
MP_HD double rcp_pos(double x);
MP_HD double exp_small(double x);

// Same mathematics as funcs.py:179-229 at one node, with the hot-loop elementary functions
// (x^(-1/7) to 4e-16, tanh to 4e-16 absolute, Newton reciprocal / reciprocal square root).
MP_HD Lum luminosity(const Spec& sp, const Walker& w, double M, double omega) {
  if (sp.lum_dipole_only) {
    // packaged variant (magnetar/funcs.py:193,206): rot_param > 0.0 switches N_acc off at every node and
    // Lprop = propeff*(-N_acc*omega) has no other term, so Lprop = 0 whatever the disc does (a NaN falls
    // to the isfinite clamp, :207-208) and the light curve is the dipole term alone
    const double o2 = omega * omega;
    double ld = w.dipeff * (w.Ldip_coef * (o2 * o2));
    if (ld <= 0.0 || !isfinite(ld)) ld = 0.0;
    Lum L0;
    L0.dip = ld;
    L0.prop = 0.0;
    L0.tot = w.f_beam * (ld + 0.0);
    return L0;
  }
  const double qa = w.l_sqrtA * pow_m17_seeded(M);             // NaN for M <= 0, as the reference's power
  const double mdot = M * w.l_inv_tv;
  const double rm_u = qa * qa;                                 // funcs.py:186-187
  const double r = rsqrt_pos(omega);
  const bool capped = rm_u * omega >= w.l_kc;                  // Rm >= k*Rlc  (funcs.py:189-190)
  const double rm = capped ? w.l_kc * (r * r) : rm_u;
  const double fast = capped ? w.l_Ccap * r : (rm_u * qa) * (sp.inv_sqrtGM * omega);
  const double om2 = omega * omega;
  const double x = sp.lum_n * (fast - 1.0);
  double th;                                                   // tanh(n (w - 1)), funcs.py:200
  if (x > 19.1) th = 1.0;
  else if (x < -19.1) th = -1.0;
  else th = fma(-2.0, rcp_pos(exp_small(x + x) + 1.0), 1.0);
  if (!(x == x)) th = x;
  const double eta2 = 0.5 * (1.0 + th);
  const double eta1 = 1.0 - eta2;
  const double mprop = eta2 * mdot, macc = eta1 * mdot;
  double nacc;
  if (om2 > sp.omega2_breakup_lum) {
    nacc = 0.0;
  } else {
    const double lev = capped ? w.l_sGMkc * r : sp.sqrtGM * qa;   // sqrt(GM Rm)
    const double lever = (rm < kR) ? sp.sqrt_GMR : lev;
    nacc = lever * (macc - mprop);
  }
  double ldip = w.dipeff * (w.Ldip_coef * (om2 * om2));
  if (ldip <= 0.0 || !isfinite(ldip)) ldip = 0.0;                      // funcs.py:216-219
  double lprop = -1.0 * nacc * omega;
  if (sp.lprop_binding_term) {                                         // funcs.py:222-223
    const double gm_rm = capped ? w.l_GM_kc * omega : kGM * rcp_pos(rm_u);
    lprop -= gm_rm * eta2 * mdot;
  }
  lprop *= w.propeff;
  if (lprop <= 0.0 || !isfinite(lprop)) lprop = 0.0;                   // funcs.py:224-227
  Lum L;
  L.dip = ldip;
  L.prop = lprop;
  L.tot = w.f_beam * (ldip + lprop);                                   // funcs.py:229
  return L;
}

// ---- branch-free forms for the explicit step ------------------------------------------
// The step below evaluates the five disc-mass stages of a step as one block and then the six
// spin-equation stages as one serial chain; both blocks are straight-line code (selects, no
// branches) so the compiler can overlap the independent chains.  CUDA's rsqrt()/division carry a
// special-case branch each; the arguments here are positive and normal, so the Newton forms are
// used bare.
MP_HD double rsqrt_pos(double x) {      // x > 0, normal
#if defined(__CUDA_ARCH__)
  double r;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));     // ~2^-22
  const double e = fma(x, -(r * r), 1.0);
  return fma(fma(e, 0.375, 0.5), r * e, r);                    // third order: ~2^-64
#else
  return 1.0 / sqrt(x);
#endif
}
// One Newton step on the MUFU seed: ~(3/8) 2^-44 = 2e-14 relative.  Ample inside the integrator's right-hand side
// (its local tolerance is 4e-10; the luminosity stage keeps the third-order form).
MP_HD double rsqrt_pos2(double x) {     // x > 0, normal
#if defined(__CUDA_ARCH__)
  double r;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  const double e = fma(x, -(r * r), 1.0);
  return fma(0.5 * r, e, r);
#else
  return 1.0 / sqrt(x);
#endif
}
MP_HD double rcp_pos(double x) {        // 1 <= x (0 for x = inf or beyond 2^1022)
#if defined(__CUDA_ARCH__)
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));       // ~2^-22
  double e = fma(-x, r, 1.0);
  e = fma(e, e, e);
  return fma(r, e, r);                                         // e^3: ~2^-64
#else
  return 1.0 / x;
#endif
}

// exp(x) for |x| <= 40 (no clamping, no NaN handling: the caller guards both).
MP_HD double exp_small(double x) {
  const double kd = fma(x, kExpR[0], kExpR[1]);
  const int k = (int)(dbits(kd) & 0xffffffffLL);
  const double kf = kd - kExpR[1];
  double r = fma(kf, kExpR[2], x);
  r = fma(kf, kExpR[3], r);
  const double r2 = r * r;
  double ev = kExpC[12], od = kExpC[11];
  ev = fma(ev, r2, kExpC[10]);
  od = fma(od, r2, kExpC[9]);
  ev = fma(ev, r2, kExpC[8]);
  od = fma(od, r2, kExpC[7]);
  ev = fma(ev, r2, kExpC[6]);
  od = fma(od, r2, kExpC[5]);
  ev = fma(ev, r2, kExpC[4]);
  od = fma(od, r2, kExpC[3]);
  ev = fma(ev, r2, kExpC[2]);
  od = fma(od, r2, kExpC[1]);
  ev = fma(ev, r2, kExpC[0]);
  const double p = fma(od, r, ev);
  return bitsd(dbits(p) + ((int64_t)k << 52));
}

// exp(x) for |x| <= 40 to ~2e-13 relative (degree 10): the spin chain's tanh needs no more.
MP_HD double exp_small10(double x) {
  const double kd = fma(x, kExpR[0], kExpR[1]);
  const int k = (int)(dbits(kd) & 0xffffffffLL);
  const double kf = kd - kExpR[1];
  double r = fma(kf, kExpR[2], x);
  r = fma(kf, kExpR[3], r);
  const double r2 = r * r;
  double ev = kExpC[10], od = kExpC[9];
  ev = fma(ev, r2, kExpC[8]);
  od = fma(od, r2, kExpC[7]);
  ev = fma(ev, r2, kExpC[6]);
  od = fma(od, r2, kExpC[5]);
  ev = fma(ev, r2, kExpC[4]);
  od = fma(od, r2, kExpC[3]);
  ev = fma(ev, r2, kExpC[2]);
  od = fma(od, r2, kExpC[1]);
  ev = fma(ev, r2, kExpC[0]);
  const double p = fma(od, r, ev);
  return bitsd(dbits(p) + ((int64_t)k << 52));
}
MP_HD double rcp_pos2(double x) {       // 1/x for 1 <= x, ~2^-44 (one Newton step on the MUFU seed)
#if defined(__CUDA_ARCH__)
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  return fma(r, fma(-x, r, 1.0), r);
#else
  return 1.0 / x;
#endif
}

// Disc quantities of one Runge-Kutta stage, in the folded form spin_f wants.
struct StageDisc {
  double qa;   // sqrt(A_rm) * Mdisc^(-1/7)
  double ni;   // Mdisc / (tvisc I)
};

// d(omega)/dt, same mathematics as spin_rhs (funcs.py:105-140), branch-free.
// `side` collects on which side of the break-up boundary the evaluations of a step fell
// (bit 0: below, bit 1: above).
MP_HD double spin_f(const Spec& sp, const Walker& w, const StageDisc& d, double omega, unsigned& side) {
  const double rm = d.qa * d.qa;                               // uncapped Alfven radius
  const double r = rsqrt_pos(omega);
  const bool capped = rm * omega >= sp.kc;                     // Rm >= k*Rlc (funcs.py:109-110)
  const double fast_u = (rm * d.qa) * (sp.inv_sqrtGM * omega);
  const double fast = capped ? sp.Ccap * r : fast_u;
  // (a NaN qa must reach the result: the selects below keep the NaN operand when a comparison fails)
  const double lev_u = (rm < kR) ? sp.sqrt_GMR : sp.sqrtGM * d.qa;            // funcs.py:135-138
  const double lev_c = (sp.kc >= kR * omega) ? sp.sGMkc * r : sp.sqrt_GMR;
  const double lever = capped ? lev_c : lev_u;
  const double om2 = omega * omega;
  // tanh(n (w - 1)) to 4e-16 absolute; beyond |x| = 19.1 it is +-1 to the last bit (most stages of a
  // propeller-phase walker), so the exponential is skipped there
  const double x = sp.rhs_n * (fast - 1.0);
  double th;
  if (x > 19.1) th = 1.0;
  else if (x < -19.1) th = -1.0;
  else th = fma(-2.0, rcp_pos(exp_small(x + x) + 1.0), 1.0);
  const bool above = om2 > sp.omega2_breakup_rhs;
  side |= above ? 2u : 1u;
  th = above ? 0.0 : th;                                       // funcs.py:131-132
  double cdip = w.Cdip_I;
  if (sp.bucciantini) {
    const double q = kC / (omega * rm);
    cdip *= capped ? sp.bucc_cap : 4.0 * q * q * q;
  }
  return fma(-cdip * om2, omega, -(lever * d.ni) * th);
}

// The explicit integrator does not integrate omega but y = omega^-2.  Pure dipole spin-down,
// d(omega)/dt = -C omega^3, is dy/dt = 2C: y is then LINEAR in t and any Runge-Kutta step is exact,
// whereas omega ~ t^(-1/2) costs a power-law solution's ~65 steps per decade at rtol 1e-10.  The
// late-time spin evolution is dipole-dominated, so in y the step count of the four synthetic truths
// drops by 35-50 % at the same accuracy in omega (measured; DESIGN.md section 3).
//   dy/dt = -2 omega^-3 d(omega)/dt = 2 C + 2 omega^-3 sqrt(GM Rm) (Mdisc/(tvisc I)) tanh(n (w - 1))
// with omega = y^(-1/2) (one reciprocal square root -- the omega form needs one as well, for the
// capped branch).  Same mathematics as spin_f / funcs.py:105-140.  The capped branch is a real
// branch: it costs a second reciprocal square root, and the lanes of a warp mostly agree on it.
// `regime` (out): bit 0 = Alfven radius capped at k*Rlc, bit 1 = lever arm at its floor sqrt(GM R).  The
// right-hand side is continuous but kinked where either bit flips; the step uses the bits of its two
// end points to land on such a kink instead of stepping across it (see locate_kink).
// (Classical dipole torque only: a spec with the Bucciantini torque is integrated by the implicit variant,
// whose right-hand side carries the option -- the kernels route every walker there, so this hot function
// pays nothing for a figure-script variant.)
MP_HD double spin_g(const Spec& sp, const Walker& w, const StageDisc& d, double y, unsigned& side, unsigned& regime) {
  // d is in the explicit variant's scaling (disc_stages_dp5 / scale_for_g):
  //   d.qa = GM^(-1/6) sqrt(A_rm) Mdisc^(-1/7)   so that  Rm = GM^(1/3) qa^2,  w = qa^3 omega (uncapped)
  //   d.ni = 2 GM^(2/3) Mdisc/(tvisc I)          so that  2 sqrt(GM Rm) Mdisc/(tvisc I) = qa d.ni
  // which removes three multiplications by constants from every evaluation.
  const double om = rsqrt_pos2(y);                             // omega
  const double iom = y * om;                                   // 1/omega
  const double rm = d.qa * d.qa;                               // uncapped Alfven radius / GM^(1/3)
  const double rcap = sp.g_kc * iom;                           // k*Rlc / GM^(1/3)
  double fast, lev;                                            // fastness w; 2 sqrt(GM Rm) Mdisc/(tvisc I) = lev * d.ni
  if (rm >= rcap) {                                            // Rm >= k*Rlc (funcs.py:109-110)
    const double r = rsqrt_pos2(om);
    fast = sp.Ccap * r;
    const bool floor_ = !(rcap >= sp.g_R);
    lev = floor_ ? sp.g_floor : sp.g_cap * r;
    regime = floor_ ? 3u : 1u;
  } else {                                                     // (also taken by a NaN qa, which then reaches the result)
    fast = (rm * d.qa) * om;
    const bool floor_ = rm < sp.g_R;
    lev = floor_ ? sp.g_floor : d.qa;                          // funcs.py:135-138
    regime = floor_ ? 2u : 0u;
  }
  // tanh(n (w - 1)); beyond |2x| = 38.2 it is +-1 to the last bit.  Inside, 1e-13 absolute is ample for the
  // integrator (the luminosity stage has its own, full-precision evaluation): degree-10 exp, second-order
  // reciprocal.  (Folding the constant factors of 2x into one fused multiply-add on omega, and the cap test into
  // a comparison with 1/omega -- two multiplications fewer on the serial chain -- measured 0.6 % SLOWER.)
  const double x2 = fma(sp.rhs_n2, fast, -sp.rhs_n2);
  double th;
  if (fabs(x2) > 38.2) th = copysign(1.0, x2);
  else th = fma(-2.0, rcp_pos2(exp_small10(x2) + 1.0), 1.0);
  const bool above = y < sp.y_breakup_rhs;                     // rot_param > 0.27 (funcs.py:131-132)
  side |= above ? 2u : 1u;
  th = above ? 0.0 : th;
  return fma((lev * d.ni) * (y * iom), th, w.Cdip_I2);
}

// Generic disc quantities (disc_stages<N>) -> the scaling spin_g wants.
MP_HD void scale_for_g(const Spec& sp, StageDisc& d) {
  d.qa *= sp.g_qa;
  d.ni *= sp.g_ni;
}

MP_HD double spin_g(const Spec& sp, const Walker& w, const StageDisc& d, double y, unsigned& side) {
  unsigned regime;
  return spin_g(sp, w, d, y, side, regime);
}

// Step-size control: Hairer's dopri5 PI controller (beta = 0.04, safety 0.9; h may shrink 5x, grow 10x),
//   accepted:  h_new = h / clamp(err^(0.2 - 0.75 beta) / facold^beta / safety, 0.1, 5),  facold <- max(err, 1e-4)
//   rejected:  h_new = h / min(err^(0.2 - 0.75 beta) / safety, 5)
// evaluated in the log2 domain, in single precision (it steers the step size only): err = aerr/sk becomes a
// difference of two logarithms, the divisions become subtractions, the clamps stay clamps, and one exp2 gives
// 1/fac -- no IEEE division, none of the range checks and fix-up branches of logf/exp2f/"/" on the step's
// serial tail (measured: +2 % with approximate reciprocals alone).  `lfacold` is log2(facold).
struct StepControl {
  static constexpr float beta = 0.04f, expo1 = 0.2f - 0.04f * 0.75f;
  static constexpr float l_safe = -0.15200309f;      // log2(0.9)
  static constexpr float l_shrink = 2.3219281f;      // log2(5)
  static constexpr float l_grow = -3.3219281f;       // log2(0.1)
  static constexpr float l_err_min = -99.657843f;    // log2(1e-30)
  static constexpr float l_err_nan = 33.219281f;     // log2(1e10): NaN => shrink hard
  static constexpr float l_facold_min = -13.287712f; // log2(1e-4)
};
MP_HD float log2_error_ratio(double aerr, double sk) {
  float l;
#if defined(__CUDA_ARCH__)
  float la, ls;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(la) : "f"((float)aerr));
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(ls) : "f"((float)sk));
  l = la - ls;
#else
  l = log2f((float)aerr) - log2f((float)sk);
#endif
  if (!(l == l)) l = StepControl::l_err_nan;
  return fmaxf(l, StepControl::l_err_min);
}
MP_HD double step_scale(float minus_log2_fac) {     // 1/fac
#if defined(__CUDA_ARCH__)
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(minus_log2_fac));
  return (double)r;
#else
  return (double)exp2f(minus_log2_fac);
#endif
}

// ---- Dormand-Prince 5(4) with dense output --------------------------------
// Coefficients: Dormand & Prince 1980; dense output: Hairer, Norsett & Wanner II.6.
// State of the spin integration of one walker.
// The state variable `omega` holds omega in the implicit variant and y = omega^-2 in the explicit one.
struct Integrator {
  double t, omega, h, k1;        // k1 = f(t, state) (FSAL)
  float lfacold;                 // log2 of the controller's previous error ratio (see StepControl)
  int rejected;                  // previous attempt was rejected
  // dense output of the last accepted step: omega(t0 + theta*hs)
  double t0, hs, r1, r2, r3, r4, r5;   // covers [t0, t]
  int n_rhs, n_steps, status;
  int stiff;                     // explicit variant: stiffness detected (the walker is deferred)
  int stiff_votes;               // consecutive steps voting stiff
  // implicit variant only: f, df/domega and the disc quantities at (t, omega), carried from step to step
  double J0, d0_qa, d0_ni;
  int have0;
  // explicit variant only: the disc-mass transient C exp(u0 - u(t)) at the current time, carried from
  // step to step (see disc_stages_dp5)
  double E;
  unsigned regime;               // bits 0-1: spin_g's regime bits at (t, state); bits 2-3: the regime beyond the
                                 // kink the current attempt is aimed at; bits 4..: kinks landed on so far
  double h_resume;               // step size in use when that kink was met (> 0: the attempt is a landing)
};

MP_HD double dense_eval(const Integrator& in, double tq) {
  const double th = (tq - in.t0) / in.hs;
  const double th1 = 1.0 - th;
  return fma(th, fma(th1, fma(th, fma(th1, in.r5, in.r4), in.r3), in.r2), in.r1);
}
// The same with 1/hs supplied: a run of nodes inside one step shares the division.
// 1/hs for the dense output's local coordinate (hs > 0, normal): Newton on the MUFU seed, no IEEE-division fix-up.
MP_HD double rcp_step(double x) {
#if defined(__CUDA_ARCH__)
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));       // ~2^-22
  double e = fma(-x, r, 1.0);
  e = fma(e, e, e);
  return fma(r, e, r);                                         // e^3: ~2^-64
#else
  return 1.0 / x;
#endif
}
MP_HD double dense_eval_r(const Integrator& in, double tq, double ihs) {
  const double th = (tq - in.t0) * ihs;
  const double th1 = 1.0 - th;
  return fma(th, fma(th1, fma(th, fma(th1, in.r5, in.r4), in.r3), in.r2), in.r1);
}

// f(t, omega) out of line: used by the (cold) initialisation only, so the hot
// step loop below holds the single inlined copy of disc_at + spin_rhs.
#if defined(__CUDACC__)
__device__ __host__ __noinline__
#endif
static double spin_f_cold(const Spec& sp, const Walker& w, double t, double omega) {
  const DiscAt d = disc_at(w, t);
  return spin_rhs(sp, w, d, omega);
}

template <int N>
MP_HD void disc_stages(const Walker& w, const double* ts, StageDisc* d);

#if defined(__CUDACC__)
__device__ __host__ __noinline__
#endif
static double spin_g_cold(const Spec& sp, const Walker& w, double t, double y, unsigned* regime) {
  StageDisc d;
  disc_stages<1>(w, &t, &d);
  scale_for_g(sp, d);
  unsigned side = 0u, rg = 0u;
  const double g = spin_g(sp, w, d, y, side, rg);
  if (regime) *regime = rg;
  return g;
}

// INVSQ: the state is y = omega^-2 (explicit variant), tolerance 2 rtol (d(omega)/omega = dy/(2y)).
template <bool INVSQ>
MP_HD void integrator_init(const Spec& sp, const Walker& w, double t_start, double t_end,
                           Integrator& in) {
  in.t = t_start;
  in.omega = INVSQ ? 1.0 / (w.omega0 * w.omega0) : w.omega0;
  in.lfacold = StepControl::l_facold_min;
  in.rejected = 0;
  in.n_steps = 0;
  in.stiff = 0;
  in.stiff_votes = 0;
  in.have0 = 0;
  in.E = w.C;                        // u(t_start) = u0
  in.regime = 0u;
  in.h_resume = 0.0;
  in.J0 = in.d0_qa = in.d0_ni = 0.0;
  in.status = kWalkerOk;
  in.t0 = t_start; in.hs = 1.0;
  in.r1 = in.omega; in.r2 = in.r3 = in.r4 = in.r5 = 0.0;
  unsigned rg0 = 0u;
  in.k1 = INVSQ ? spin_g_cold(sp, w, t_start, in.omega, &rg0) : spin_f_cold(sp, w, t_start, in.omega);
  in.regime = rg0;
  // initial step (Hairer's hinit, order 5)
  const double sk = (INVSQ ? sp.rtol_y : sp.rtol) * fabs(in.omega);
  const double dnf = fabs(in.k1) / sk, dny = fabs(in.omega) / sk;
  double h = (dnf <= 1e-10 || dny <= 1e-10) ? 1.0e-6 : 0.01 * (dny / dnf);
  const double span = t_end - t_start;
  h = fmin(h, span);
  const double y1 = fma(h, in.k1, in.omega);
  const double f1 = INVSQ ? spin_g_cold(sp, w, t_start + h, y1, nullptr) : spin_f_cold(sp, w, t_start + h, y1);
  const double der2 = fabs(f1 - in.k1) / sk / h;
  const double der12 = fmax(der2, dnf);
  const double h1 = (der12 <= 1e-15) ? fmax(1.0e-6, fabs(h) * 1.0e-3)
                                     : exp(log(0.01 / der12) * 0.2);
  in.h = fmin(fmin(100.0 * h, h1), span);
  in.n_rhs = 2;
  if (!(isfinite(in.k1) && isfinite(in.h) && in.h > 0.0)) in.status = kWalkerIntegratorFail;
}

// The implicit variant taking over at (t, omega) with the explicit variant's last step size.
MP_HD void integrator_resume(double t, double omega, double h, Integrator& in) {
  in.t = t;
  in.omega = omega;
  in.h = h;
  in.k1 = 0.0;
  in.lfacold = StepControl::l_facold_min;
  in.rejected = 0;
  in.n_rhs = 0; in.n_steps = 0;
  in.stiff = 0; in.stiff_votes = 0;
  in.have0 = 0;
  in.E = 1.0; in.regime = 0u; in.h_resume = 0.0;
  in.J0 = in.d0_qa = in.d0_ni = 0.0;
  in.status = (omega == omega && h > 0.0) ? kWalkerOk : kWalkerIntegratorFail;
  in.t0 = t; in.hs = 1.0;
  in.r1 = omega; in.r2 = in.r3 = in.r4 = in.r5 = 0.0;
}

// Dormand-Prince tableau (classic form) for the block step, as constant-bank operands.
MP_CONST_QUALIFIER double kDP[36] = {
    1.0 / 5, 3.0 / 10, 4.0 / 5, 8.0 / 9,                                                   // 0: c2..c5
    1.0 / 5,                                                                               // 4: a21
    3.0 / 40, 9.0 / 40,                                                                    // 5: a31 a32
    44.0 / 45, -56.0 / 15, 32.0 / 9,                                                       // 7: a41..a43
    19372.0 / 6561, -25360.0 / 2187, 64448.0 / 6561, -212.0 / 729,                         // 10: a51..a54
    9017.0 / 3168, -355.0 / 33, 46732.0 / 5247, 49.0 / 176, -5103.0 / 18656,               // 14: a61..a65
    35.0 / 384, 500.0 / 1113, 125.0 / 192, -2187.0 / 6784, 11.0 / 84,                      // 19: b1 b3 b4 b5 b6
    71.0 / 57600, -71.0 / 16695, 71.0 / 1920, -17253.0 / 339200, 22.0 / 525, -1.0 / 40,    // 24: e1 e3 e4 e5 e6 e7
    -12715105075.0 / 11282082432.0, 87487479700.0 / 32700410799.0, -10690763975.0 / 1880347072.0,
    701980252875.0 / 199316789632.0, -1453857185.0 / 822651844.0, 69997945.0 / 29380423.0};  // 30: d1 d3 d4 d5 d6 d7
#define MP_DPK(name, idx) static MP_HD double name() { return kDP[idx]; }
struct DP {
  MP_DPK(c2, 0) MP_DPK(c3, 1) MP_DPK(c4, 2) MP_DPK(c5, 3)
  MP_DPK(a21, 4) MP_DPK(a31, 5) MP_DPK(a32, 6) MP_DPK(a41, 7) MP_DPK(a42, 8) MP_DPK(a43, 9)
  MP_DPK(a51, 10) MP_DPK(a52, 11) MP_DPK(a53, 12) MP_DPK(a54, 13)
  MP_DPK(a61, 14) MP_DPK(a62, 15) MP_DPK(a63, 16) MP_DPK(a64, 17) MP_DPK(a65, 18)
  MP_DPK(b1, 19) MP_DPK(b3, 20) MP_DPK(b4, 21) MP_DPK(b5, 22) MP_DPK(b6, 23)
  MP_DPK(e1, 24) MP_DPK(e3, 25) MP_DPK(e4, 26) MP_DPK(e5, 27) MP_DPK(e6, 28) MP_DPK(e7, 29)
  MP_DPK(d1, 30) MP_DPK(d3, 31) MP_DPK(d4, 32) MP_DPK(d5, 33) MP_DPK(d6, 34) MP_DPK(d7, 35)
};

// Block form of the step (the default).  A step's five new stage times depend on (t, h) only, so
// the disc-mass work of all five stages -- ten degree-10 polynomials in the late phase; five
// polynomials, exponentials and x^(-1/7) before it -- is evaluated first as one block of
// independent chains (that is where the FP64 pipe gets saturated); the six evaluations of the
// scalar spin equation, which are inherently serial, follow as one straight-line chain.
// Break-up sliding mode.  N_acc is switched off above rot_param = breakup_rhs (funcs.py:131-132).
// If the spin reaches that boundary while, just inside it, the accretion torque still outweighs the
// dipole torque, the state can neither cross nor leave: the solution chatters along the
// discontinuity (a Filippov sliding mode).  LSODA burns its step budget there and the reference
// returns 'flag' -> -inf (funcs.py:172-173); we detect the situation and fail at once.  Called when
// the evaluations of a step straddled the boundary.  An accepted step that crossed is judged at once; a
// step that only sampled the far side with its stages is judged once the state sits within 1e-6
// of the boundary -- the integrator otherwise realises the sliding mode numerically, hovering
// rtol below the boundary with steps of 1e-8 t (measured: 78 000 steps for one such walker).
#if defined(__CUDACC__)
__device__ __host__ __noinline__
#endif
static bool breakup_sliding_block(const Spec& sp, const Walker& w, const StageDisc d, double y_old, double y_new,
                                  bool accepted) {
  const double om_b = sqrt(sp.omega2_breakup_rhs);
  const bool crossed = (y_old * y_old > sp.omega2_breakup_rhs) != (y_new * y_new > sp.omega2_breakup_rhs);
  const bool near = fabs(y_old - om_b) <= 1.0e-6 * om_b;
  if (!((accepted && crossed) || near)) return false;
  unsigned side = 0u;
  return spin_f(sp, w, d, om_b * (1.0 - 1.0e-12), side) > 0.0;
}
// The same test for the explicit variant, whose state is y = omega^-2 (spinning up = y falling).
#if defined(__CUDACC__)
__device__ __host__ __noinline__
#endif
static bool breakup_sliding_block_y(const Spec& sp, const Walker& w, const StageDisc d, double y_old, double y_new,
                                    bool accepted) {
  const double yb = sp.y_breakup_rhs;
  const bool crossed = (y_old < yb) != (y_new < yb);
  const bool near = fabs(y_old - yb) <= 2.0e-6 * yb;
  if (!((accepted && crossed) || near)) return false;
  unsigned side = 0u;
  return spin_g(sp, w, d, yb * (1.0 + 2.0e-12), side) < 0.0;
}

// Kinks.  The right-hand side is C0 but not C1 where the Alfven radius reaches the light-cylinder cap
// (funcs.py:109-110) and where the lever arm reaches its floor (funcs.py:135-138).  A step across such a
// kink loses its order: the controller answers with a burst of rejections and tiny steps (4-6 rejections
// per kink on the synthetic truths), and what error it lets through is the LARGEST contribution to the
// global error (measured: landing on the kinks lowers the error in omega 5-40x at equal rtol).  So when
// the regime bits of a trial step's two end points differ, the crossing is located -- the margin of the
// bit that flipped at the two ends, one regula-falsi refinement and a final secant estimate, with the
// state interpolated linearly (omega moves by < 1e-3 over a step here; the margin is dominated by the
// disc mass and is close to linear over a step, so this lands within ~1e-3 of the step) -- and the step
// is retried to END on the kink.  Two disc-mass evaluations, no right-hand-side evaluations; kept this
// small because in an ensemble that is spread out the lanes of a warp meet their kinks on different
// trips and each call runs with one active lane.
// Returns the fraction of the step at which the kink sits, or -1.
#if defined(__CUDACC__)
__device__ __host__ __noinline__
#endif
static double locate_kink(const Spec& sp, const Walker& w, double t, double h, double y, double ynew, double qa_end,
                          unsigned r0, unsigned r1) {
  const bool cap_event = ((r0 ^ r1) & 1u) != 0u;
  const bool capped = (r0 & 1u) != 0u;            // used by the floor event only (cap bit equal at both ends)
  // margin(theta): changes sign where the bit flips
  auto margin = [&](double th, double qa) {          // qa in spin_g's scaling
    const double yy = fma(th, ynew - y, y);
    const double rm = qa * qa;
    const double rcap = sp.g_kc * (yy * rsqrt_pos(yy));
    return cap_event ? rm - rcap : (capped ? sp.g_R - rcap : sp.g_R - rm);
  };
  StageDisc d;
  disc_stages<1>(w, &t, &d);
  double a = 0.0, b = 1.0, fa = margin(0.0, d.qa * sp.g_qa), fb = margin(1.0, qa_end);
  if (!(fa * fb < 0.0)) return -1.0;              // also NaN
  {   // one regula-falsi refinement (a second one: +0 accuracy at the landing tolerance, -3..5 % on spread ensembles)
    const double th = (a * fb - b * fa) / (fb - fa);
    const double tt = fma(th, h, t);
    disc_stages<1>(w, &tt, &d);
    const double m = margin(th, d.qa * sp.g_qa);
    if (!(m == m)) return -1.0;
    if ((m < 0.0) == (fa < 0.0)) { a = th; fa = m; }
    else { b = th; fb = m; }
  }
  return (a * fb - b * fa) / (fb - fa);
}

// Second half of the block step: the six serial spin-equation stages, error control, dense output.
// Returns 1 accepted, 0 rejected, 2 a kink lies inside the trial (y_trial / regime_trial describe its end).
MP_HD int step_spin_chain(const Spec& sp, const Walker& w, Integrator& in, const double t, const double y,
                          const double h, const double tn, const StageDisc* d, double& y_trial, unsigned& regime_trial) {
  // ---- spin chain
  const double k1 = in.k1;
  unsigned side = (y < sp.y_breakup_rhs) ? 2u : 1u;
  const double y2 = fma(h, DP::a21() * k1, y);
  const double k2 = spin_g(sp, w, d[0], y2, side);
  const double y3 = fma(h, fma(DP::a32(), k2, DP::a31() * k1), y);
  const double k3 = spin_g(sp, w, d[1], y3, side);
  const double y4 = fma(h, fma(DP::a43(), k3, fma(DP::a42(), k2, DP::a41() * k1)), y);
  const double k4 = spin_g(sp, w, d[2], y4, side);
  const double y5 = fma(h, fma(DP::a54(), k4, fma(DP::a53(), k3, fma(DP::a52(), k2, DP::a51() * k1))), y);
  const double k5 = spin_g(sp, w, d[3], y5, side);
  const double y6 = fma(h, fma(DP::a65(), k5, fma(DP::a64(), k4, fma(DP::a63(), k3, fma(DP::a62(), k2, DP::a61() * k1)))), y);
  const double k6 = spin_g(sp, w, d[4], y6, side);
  const double ynew = fma(h, fma(DP::b6(), k6, fma(DP::b5(), k5, fma(DP::b4(), k4, fma(DP::b3(), k3, DP::b1() * k1)))), y);
  unsigned regime_end;
  const double k7 = spin_g(sp, w, d[4], ynew, side, regime_end);
  in.n_rhs += 6;
#ifndef MP_NO_EVENTS
  if (regime_end != (in.regime & 3u) && in.regime < (8u << 4) && !(in.h_resume > 0.0)) {
    // a kink lies inside this trial step: the caller locates it (none of the stage values are live
    // there) and the trial is dropped
    y_trial = ynew;
    regime_trial = regime_end;
    in.n_steps++;
    return 2;
  }
#endif
  const double esum = fma(DP::e7(), k7, fma(DP::e6(), k6, fma(DP::e5(), k5, fma(DP::e4(), k4, fma(DP::e3(), k3, DP::e1() * k1)))));
  const double errv = h * esum;
  const double sk = sp.rtol_y * ((ynew > y) ? ynew : y);   // (y = omega^-2 > 0; a NaN or negative ynew comes with a NaN error)
  const double aerr = fabs(errv);
  const bool accept = aerr <= sk;                 // false for NaN
  const float lerr = log2_error_ratio(aerr, sk);
  if (accept) {
    const float g = StepControl::expo1 * lerr - StepControl::beta * in.lfacold - StepControl::l_safe;   // log2(fac)
    const double hnew = h * step_scale(-fmaxf(StepControl::l_grow, fminf(StepControl::l_shrink, g)));
    in.lfacold = fmaxf(lerr, StepControl::l_facold_min);
    // dense output (Hairer's contd5)
    const double dsum = fma(DP::d7(), k7, fma(DP::d6(), k6, fma(DP::d5(), k5, fma(DP::d4(), k4, fma(DP::d3(), k3, DP::d1() * k1)))));
    const double ydiff = ynew - y;
    const double bspl = fma(h, k1, -ydiff);
    in.r1 = y;
    in.r2 = ydiff;
    in.r3 = bspl;
    in.r4 = ydiff - h * k7 - bspl;
    in.r5 = h * dsum;
    in.t0 = t; in.hs = h;
    in.t = tn;
    in.omega = ynew;
    in.k1 = k7;
    // (a step that was aimed at a kink ends on it: from here on the far side's regime holds, whichever
    // side of the kink rounding put the end point on)
    const bool landing = in.h_resume > 0.0;
    in.regime = (in.regime & ~3u) | (landing ? ((in.regime >> 2) & 3u) : regime_end);
#ifndef MP_NO_SLIDING
    if (side == 3u && breakup_sliding_block_y(sp, w, d[4], y, ynew, true)) in.status = kWalkerIntegratorFail;
#endif
    // (plain comparisons: fmin/fmax carry NaN handling the finite step sizes here do not need)
    double hn = (in.rejected && h < hnew) ? h : hnew;   // no growth right after a rejection
    if (landing) {                                // this was the (short) step that landed on a kink:
      hn = (in.h_resume > hn) ? in.h_resume : hn;  // carry on with the step size in use before it
      in.h_resume = 0.0;
    }
    in.h = hn;
    in.rejected = 0;
    in.n_steps++;
    // stiffness detection: |lambda| t > 10 (lambda from the last two stages, which share their time)
    // while h < t/20, six accepted steps in a row -> the walker is handed to the implicit variant.  (The
    // thresholds decide only WHERE the hand-over happens -- the same 29 % of prior-uniform walkers end up
    // there whatever they are -- and an early one is what keeps the explicit launch's longest walker short:
    // measured against |lambda| t > 30, h < t/50, twelve steps: longest explicit walker 781 -> 405 steps,
    // total right-hand-side evaluations -8 %, same accuracy on the golden walkers.)
#ifndef MP_NO_VOTES
    const double dy = fabs(ynew - y6);
#ifndef MP_STIFF_LAMT
#define MP_STIFF_LAMT 10.0
#define MP_STIFF_HT 0.05
#define MP_STIFF_NVOTES 6
#endif
    if (fabs(k7 - k6) * tn > MP_STIFF_LAMT * dy && h < MP_STIFF_HT * tn) {   // |lambda| t > 10 while h << t
      if (++in.stiff_votes >= MP_STIFF_NVOTES) { in.stiff = 1; in.stiff_votes = 0; }
    } else {
      in.stiff_votes = 0;
    }
#endif
    return 1;
  }
  // rejected
  const double hnew = h * step_scale(-fminf(StepControl::l_shrink, StepControl::expo1 * lerr - StepControl::l_safe));
  in.h = hnew;
  in.h_resume = 0.0;                  // (a rejected landing attempt: the shorter retry no longer reaches the kink)
  in.rejected = 1;
  in.n_steps++;
#ifndef MP_NO_SLIDING
  if (side == 3u && breakup_sliding_block_y(sp, w, d[4], y, ynew, false)) in.status = kWalkerIntegratorFail;
#endif
  if (!(fabs(hnew) > 1.0e-14 * fabs(t)) || in.n_steps >= sp.max_steps) in.status = kWalkerIntegratorFail;
  return 0;
}

// Disc quantities at N stage times, evaluated as one block of independent chains.
template <int N>
MP_HD void disc_stages(const Walker& w, const double* ts, StageDisc* d) {
  double u[N];
  TableAt ta[N];
  bool in_all = true;
#pragma unroll
  for (int s = 0; s < N; ++s) {
    u[s] = fma(ts[s], w.inv_tv, w.eps);
    in_all = table_locate_safe(u[s], ta[s]) && in_all;
  }
  if (in_all && u[0] >= w.u_late) {
    // late phase: S and Q = S^(-1/7) from the same table row -- no exp, no log
#pragma unroll
    for (int s = 0; s < N; ++s) {
      const double s2 = ta[s].s * ta[s].s;
      const double S = poly10p(ta[s].row, ta[s].s, s2);
      const double Q = poly10p(ta[s].row + MP_DISC_ROW, ta[s].s, s2);
      d[s].ni = (w.K * S) * w.tvI;
      d[s].qa = w.KqA * Q;
    }
  } else {
    double S[N];
#pragma unroll
    for (int s = 0; s < N; ++s) S[s] = poly10p(ta[s].row, ta[s].s, ta[s].s * ta[s].s);
    if (!in_all) {                                      // parameters far outside the prior box
#pragma unroll
      for (int s = 0; s < N; ++s) {
        TableAt tb;
        if (!table_locate(u[s], tb)) S[s] = disc_S_outside(u[s]);
      }
    }
#pragma unroll
    for (int s = 0; s < N; ++s) {
      const double E = exp_c(w.u0 - u[s]);
      const double M = fma(w.K, S[s], w.C * E);
      d[s].ni = M * w.tvI;
      d[s].qa = w.sqrtA * pow_m17_seeded(M);
    }
  }
}

// The same for the five stage times of a Dormand-Prince step, t + (1/5, 3/10, 4/5, 8/9, 1) h, in ONE form for
// every phase: M = K S(u) + E with the transient E = C exp(u0 - u) carried from step to step.  The stage
// fractions are multiples of 1/90, so with a = exp(-h/(90 tvisc)) the five factors are a^18, a^27, a^72,
// a^80, a^90: ONE exponential and ten multiplications per step instead of five exponentials, applied to the
// carried value (E_t -> E_end = E_t a^90; it drifts by ~1e-14 per step relative to itself, <= 2e-12 before
// it stops mattering -- two orders below the step tolerance; the luminosity stage does not use it).  Once
// the transient has died out (u >= u_late) the table's Q = S^(-1/7) would serve as well as the seeded
// x^(-1/7) at the same cost; keeping a single form means the lanes of a warp never split over the phase
// (measured: +11 % on ensembles spread around the posterior, +5 % on a 1e-4 ball).
MP_HD void disc_stages_dp5(const Spec& sp, const Walker& w, const double* ts, double Et, double dl, StageDisc* d, double& Eend) {
  double u[5];
  TableAt ta[5];
  bool in_all = true;
#pragma unroll
  for (int s = 0; s < 5; ++s) {
    u[s] = fma(ts[s], w.inv_tv, w.eps);
    in_all = table_locate_fast(u[s], ta[s]) && in_all;
  }
  if (!in_all) {                                        // parameters far outside the prior box
    disc_stages<5>(w, ts, d);
#pragma unroll
    for (int s = 0; s < 5; ++s) scale_for_g(sp, d[s]);
    Eend = w.C * exp_c(w.u0 - u[4]);
    return;
  }
  const double xa = dl * (-1.0 / 90.0);
  const double a = exp_small(xa < -40.0 ? -40.0 : xa);
  const double a2 = a * a, a4 = a2 * a2, a8 = a4 * a4, a9 = a8 * a;
  const double a18 = a9 * a9, a27 = a18 * a9, a36 = a18 * a18, a72 = a36 * a36;
  const double E[5] = {Et * a18, Et * a27, Et * a72, Et * (a72 * a8), Et * (a72 * a18)};
  // The seeded power's range test is taken once for the five arguments (not once per stage: a branch between
  // the stages keeps the compiler from interleaving their chains -- measured +4 % on the headline workload).
  double M[5];
  bool seedable = true;
#pragma unroll
  for (int s = 0; s < 5; ++s) {
    const double S = polyfast(ta[s].row, ta[s].s, ta[s].s * ta[s].s);
    M[s] = fma(w.K, S, E[s]);
    seedable = pow_m17_seedable(M[s]) && seedable;
  }
  if (seedable) {
#pragma unroll
    for (int s = 0; s < 5; ++s) {
      d[s].ni = M[s] * w.g_tvI;
      d[s].qa = w.g_sqrtA * pow_m17_seeded1_inrange(M[s]);
    }
  } else {
#pragma unroll
    for (int s = 0; s < 5; ++s) {
      d[s].ni = M[s] * w.g_tvI;
      d[s].qa = w.g_sqrtA * pow_m17_cold(M[s]);
    }
  }
  Eend = E[4];
}

MP_HD bool integrator_step(const Spec& sp, const Walker& w, double t_end, Integrator& in) {
  // step budget (accepted steps count too): a walker that has used it up and is asked for another step fails.
  // (Tested on the count alone, before the step -- a step is only asked for while nodes are outstanding; after
  // the step the test needed t_end, which lives in local memory, and a second comparison: -1.5 %.)
  if (in.n_steps >= sp.max_steps) { in.status = kWalkerIntegratorFail; return false; }
  const double t = in.t, y = in.omega;
  double h = in.h;
  bool last = false;
  if (t + 1.01 * h >= t_end) { h = t_end - t; last = true; }
  const double tn = last ? t_end : t + h;
  // The previous step's dense output is dead from here on (every node it covers was drained before
  // this step was attempted); overwriting it frees its registers for the step.
  in.r1 = in.r2 = in.r3 = in.r4 = in.r5 = 0.0;
  in.t0 = t;
  const double ts[5] = {fma(DP::c2(), h, t), fma(DP::c3(), h, t), fma(DP::c4(), h, t), fma(DP::c5(), h, t), tn};
  StageDisc d[5];
  double Eend;
  disc_stages_dp5(sp, w, ts, in.E, (tn - t) * w.inv_tv, d, Eend);
  // (One shared copy of the chain: inlining it after each disc block lets the compiler overlap the
  // two, but lanes of a warp that sit in different phases then run the chain twice -- measured
  // 4 % slower on uniform ensembles, 11 % on spread ones.)
  double y_trial;
  unsigned regime_trial;
  const int code = step_spin_chain(sp, w, in, t, y, h, tn, d, y_trial, regime_trial);
  if (code == 1) in.E = Eend;
  if (code == 2) {
    // locate the kink and aim the next attempt at it; one within 1e-3 of either end of the trial is
    // left alone (its effect is O(1e-6) of a full crossing): the attempt is repeated as one-sided
    const double th = locate_kink(sp, w, t, h, y, y_trial, d[4].qa, in.regime & 3u, regime_trial);
    if (th > 1.0e-3 && th < 1.0 - 1.0e-3) {
      in.h = th * h;
      in.h_resume = h;
      in.regime = ((in.regime & ~(3u << 2)) | (regime_trial << 2)) + (1u << 4);
    } else {
      in.h = h;
      in.regime = (in.regime & ~3u) | regime_trial;
    }
  }
  return code == 1;
}

// ---- Radau IIA (order 5) for the stiff phases -------------------------------------
// When much mass flows, the spin is pinned to the propeller/accretion equilibrium
// w = 1 by the steep tanh(n(w-1)) (relaxation rate 0.1..1 /s against t up to 1e6 s;
// SURVEY.md fact 4) and DP5 becomes stability-bound.  The equation is scalar, so a
// fully implicit 3-stage Radau IIA step is a 3x3 Newton solve with an analytic
// Jacobian -- no linear algebra library, no Jacobian storage.
//   stages  Z_i = h sum_j a_ij f(t + c_j h, y + Z_j),   y_{n+1} = y_n + Z_3
//   error   (f0 + (dd . Z)/h) / (u1/h - J0)            (Hairer & Wanner IV.8)
//   dense   the cubic collocation polynomial, stored in the DP5 dense form (r5 = 0)
struct RadauC {
  static constexpr double s6 = 2.449489742783178098197284;
  static constexpr double c1 = (4.0 - s6) / 10.0, c2 = (4.0 + s6) / 10.0;
  static constexpr double a11 = (88.0 - 7.0 * s6) / 360.0, a12 = (296.0 - 169.0 * s6) / 1800.0, a13 = (-2.0 + 3.0 * s6) / 225.0;
  static constexpr double a21 = (296.0 + 169.0 * s6) / 1800.0, a22 = (88.0 + 7.0 * s6) / 360.0, a23 = (-2.0 - 3.0 * s6) / 225.0;
  static constexpr double a31 = (16.0 - s6) / 36.0, a32 = (16.0 + s6) / 36.0, a33 = 1.0 / 9.0;
  static constexpr double u1 = 3.6378342527444957322;     // 30 / (6 + 81^(1/3) - 9^(1/3))
  static constexpr double dd1 = -(13.0 + 7.0 * s6) / 3.0, dd2 = (-13.0 + 7.0 * s6) / 3.0, dd3 = -1.0 / 3.0;
};

// f and J = df/d(omega) in the folded, branch-free form of spin_f.
MP_HD void spin_fJ(const Spec& sp, const Walker& w, const StageDisc& d, double omega, double& f, double& J,
                   unsigned& side) {
  const double rm = d.qa * d.qa;
  const double r = rsqrt_pos2(omega);                         // (integrator-grade: 2e-14, as in spin_g)
  const double hio = -0.5 * (r * r);                           // -1/(2 omega)
  const bool capped = rm * omega >= sp.kc;
  const double wq = (rm * d.qa) * sp.inv_sqrtGM;
  const double fast_c = sp.Ccap * r;
  const double fast = capped ? fast_c : wq * omega;
  const double dfast = capped ? fast_c * hio : wq;
  const double lev_u = (rm < kR) ? sp.sqrt_GMR : sp.sqrtGM * d.qa;
  const bool lc_var = sp.kc >= kR * omega;
  const double lev_c = lc_var ? sp.sGMkc * r : sp.sqrt_GMR;
  const double lever = capped ? lev_c : lev_u;
  const double dlever = (capped && lc_var) ? lev_c * hio : 0.0;
  const double om2 = omega * omega;
  const double x = sp.rhs_n * (fast - 1.0);
  double th, sech2;
  if (x > 19.1) { th = 1.0; sech2 = 0.0; }
  else if (x < -19.1) { th = -1.0; sech2 = 0.0; }
  else {
    const double rr = rcp_pos2(exp_small10(x + x) + 1.0);
    th = fma(-2.0, rr, 1.0);
    sech2 = 4.0 * rr * (1.0 - rr);
  }
  const bool above = om2 > sp.omega2_breakup_rhs;
  side |= above ? 2u : 1u;
  if (above) { th = 0.0; sech2 = 0.0; }
  double cdip = w.Cdip_I, cdipJ = 3.0 * w.Cdip_I;
  if (sp.bucciantini) {
    const double q = kC / (omega * rm);
    cdip *= capped ? sp.bucc_cap : 4.0 * q * q * q;             // uncapped: -4 C c^3 / Rm^3, no omega left
    cdipJ = capped ? cdipJ * sp.bucc_cap : 0.0;
  }
  f = fma(-cdip * om2, omega, -(lever * d.ni) * th);
  J = fma(-cdipJ, om2, -d.ni * fma(dlever, th, lever * sp.rhs_n * sech2 * dfast));
}

// One Radau IIA step.  The implicit variant of the kernel runs every step through here (walkers
// are bucketed: one that turns stiff under DP5 is re-run implicitly from the start, so the lanes of
// a warp all execute this function).  f, J and the disc quantities at (t, omega) are carried over
// from the previous step's end point.
MP_HD void radau_step(const Spec& sp, const Walker& w, double t_end, Integrator& in) {
  using R = RadauC;
  const double t = in.t, y = in.omega;
  double h = in.h;
  bool last = false;
  if (t + 1.01 * h >= t_end) { h = t_end - t; last = true; }
  const double tn = last ? t_end : t + h;
  const double ts[3] = {fma(R::c1, h, t), fma(R::c2, h, t), tn};
  StageDisc d[3];
  disc_stages<3>(w, ts, d);
  unsigned side = (y * y > sp.omega2_breakup_rhs) ? 2u : 1u;
  if (!in.have0) {
    StageDisc d0;
    disc_stages<1>(w, &t, &d0);
    in.d0_qa = d0.qa; in.d0_ni = d0.ni;
    spin_fJ(sp, w, d0, y, in.k1, in.J0, side);
    in.n_rhs += 1;
    in.have0 = 1;
  }
  const double f0 = in.k1, J0 = in.J0;
  const double sk = sp.rtol * fabs(y);
  // starting values: extrapolate the previous step's collocation polynomial
  double z1 = dense_eval(in, ts[0]) - y;
  double z2 = dense_eval(in, ts[1]) - y;
  double z3 = dense_eval(in, tn) - y;
  if (!(fabs(z3) < 0.5 * fabs(y)) || in.rejected || in.n_steps == 0) { z1 = z2 = z3 = 0.0; }
  bool converged = false;
  double dz_prev = INFINITY;
  int it = 0;
  for (; it < 8; ++it) {
    double f1, f2, f3, J1, J2, J3;
    spin_fJ(sp, w, d[0], y + z1, f1, J1, side);
    spin_fJ(sp, w, d[1], y + z2, f2, J2, side);
    spin_fJ(sp, w, d[2], y + z3, f3, J3, side);
    in.n_rhs += 3;
    // residual G = Z - h A f
    const double g1 = z1 - h * (R::a11 * f1 + R::a12 * f2 + R::a13 * f3);
    const double g2 = z2 - h * (R::a21 * f1 + R::a22 * f2 + R::a23 * f3);
    const double g3 = z3 - h * (R::a31 * f1 + R::a32 * f2 + R::a33 * f3);
    // Newton matrix M = I - h A diag(J)
    const double h1 = h * J1, h2 = h * J2, h3 = h * J3;
    const double m11 = 1.0 - R::a11 * h1, m12 = -R::a12 * h2, m13 = -R::a13 * h3;
    const double m21 = -R::a21 * h1, m22 = 1.0 - R::a22 * h2, m23 = -R::a23 * h3;
    const double m31 = -R::a31 * h1, m32 = -R::a32 * h2, m33 = 1.0 - R::a33 * h3;
    // solve M d = -G by Cramer's rule
    const double c11 = m22 * m33 - m23 * m32, c12 = m23 * m31 - m21 * m33, c13 = m21 * m32 - m22 * m31;
    const double det = m11 * c11 + m12 * c12 + m13 * c13;
    if (!(fabs(det) > 1.0e-300)) break;
    const double idet = -1.0 / det;
    const double d1 = idet * (g1 * c11 + g2 * (m13 * m32 - m12 * m33) + g3 * (m12 * m23 - m13 * m22));
    const double d2 = idet * (g1 * c12 + g2 * (m11 * m33 - m13 * m31) + g3 * (m13 * m21 - m11 * m23));
    const double d3 = idet * (g1 * c13 + g2 * (m12 * m31 - m11 * m32) + g3 * (m11 * m22 - m12 * m21));
    z1 += d1; z2 += d2; z3 += d3;
    const double dz = fmax(fabs(d1), fmax(fabs(d2), fabs(d3)));
    if (!(dz == dz)) break;
    if (dz <= 1.0e-3 * sk + 4.0e-16 * fabs(z3)) { converged = true; ++it; break; }
#ifndef MP_NEWTON_KAPPA
#define MP_NEWTON_KAPPA 0.03
#endif
    // (radau5's stopping rule: with the contraction rate theta = |dZ_k| / |dZ_k-1| the error left after this update
    // is about theta/(1-theta) |dZ_k|; the Newton iteration is quadratic here -- the Jacobians are fresh -- so that is
    // usually met one iteration before the update itself is below the tolerance: 2 instead of 3 iterations per step)
    if (it >= 1 && dz < 0.5 * dz_prev && (dz / (dz_prev - dz)) * dz <= MP_NEWTON_KAPPA * sk) { converged = true; ++it; break; }
    if (it >= 2 && dz > 2.0 * dz_prev) break;      // diverging
    dz_prev = dz;
  }
  in.n_steps++;
  const double ynew = y + z3;
#ifndef MP_NO_SLIDING
  // stages on both sides of the break-up boundary: see breakup_sliding_block
  if (side == 3u && breakup_sliding_block(sp, w, d[2], y, ynew, converged)) in.status = kWalkerIntegratorFail;
#endif
  if (!converged) {
    in.h = 0.5 * h;
    in.rejected = 1;
    if (!(in.h > 1.0e-14 * fabs(t)) || in.n_steps >= sp.max_steps) in.status = kWalkerIntegratorFail;
    return;
  }
  // The embedded estimate is O(h^4) for an O(h^6) local error, so it is held to rtol_stiff
  // (~ rtol^(2/3)), not rtol; the parity tests bound the resulting error.
  const double skn = sp.rtol_stiff * fmax(fabs(y), fabs(ynew));
  const double ih = 1.0 / h;
  const double comb = (R::dd1 * z1 + R::dd2 * z2 + R::dd3 * z3) * ih;
  const double den = R::u1 * ih - J0;
  double errv = (f0 + comb) / den;
  double err = fabs(errv) / skn;
  if (err >= 1.0 && (in.rejected || in.n_steps <= 1)) {
    double fe, Je;
    StageDisc d0; d0.qa = in.d0_qa; d0.ni = in.d0_ni;
    unsigned s2 = 0u;
    spin_fJ(sp, w, d0, y + errv, fe, Je, s2);
    in.n_rhs += 1;
    errv = (fe + comb) / den;
    err = fabs(errv) / skn;
  }
  if (!(err == err)) err = 1.0e10;
  // step-size selection (radau5): order-3 estimate, safety tied to the Newton effort
  const double safe = 0.9, fac = fmin(safe, safe * 15.0 / (double)(7 + 2 * it));
#if defined(__CUDA_ARCH__)
  const double e4 = (double)exp2f(0.25f * __log2f(fmaxf((float)err, 1.0e-30f)));   // steers the step size only
#else
  const double e4 = (double)exp2f(0.25f * log2f(fmaxf((float)err, 1.0e-30f)));
#endif
  const double quot = fmax(0.125, fmin(5.0, e4 / fac));
  const double hnew = h / quot;
  if (err < 1.0) {
    // collocation cubic through (0,0), (c1,z1), (c2,z2), (1,z3) in the DP5 dense form
    const double g1 = (z1 / R::c1 - z3) / (1.0 - R::c1);
    const double g2 = (z2 / R::c2 - z3) / (1.0 - R::c2);
    const double r4 = (g2 - g1) / (R::c2 - R::c1);
    in.r1 = y; in.r2 = z3; in.r3 = g1 - R::c1 * r4; in.r4 = r4; in.r5 = 0.0;
    in.t0 = t; in.hs = h;
    in.t = tn;
    in.omega = ynew;
    unsigned s2 = 0u;
    spin_fJ(sp, w, d[2], ynew, in.k1, in.J0, s2);   // next step's f0, J0
    in.d0_qa = d[2].qa; in.d0_ni = d[2].ni;
    in.n_rhs += 1;
    in.h = in.rejected ? fmin(hnew, h) : hnew;
    in.rejected = 0;
    return;
  }
  in.h = hnew;
  in.rejected = 1;
  if (!(fabs(hnew) > 1.0e-14 * fabs(t)) || in.n_steps >= sp.max_steps) in.status = kWalkerIntegratorFail;
}

// ---- parameter handling -------------------------------------------------------
// theta (as the sampler holds it) -> prior test + physical parameters.
// Returns false when the prior rejects (mcmc_eqns.py:43-49: inclusive, NaN rejects).
MP_HD bool prior_accepts(const double* theta, int ndim, const double* lower, const double* upper) {
  bool ok = true;
  for (int i = 0; i < ndim; ++i) ok = ok && (theta[i] <= upper[i]) && (theta[i] >= lower[i]);
  return ok;
}

MP_HD double exp10_ref(double x) {
  // 10.0 ** x as NumPy computes it (libm pow); CUDA's pow is <= 2 ulp
  return pow(10.0, x);
}

// theta -> (physical parameters, efficiencies) per the reference's lnlike:
//   script   mcmc_eqns.py:16-17   arr[2:] = 10 ** arr[2:]   (unlog_mask bits 2..5)
//   packaged magnetar/mcmc_eqns.py:22-34   7: f_beam; 8: dipeff, propeff; 9: all three
MP_HD void unpack_theta(const Spec& sp, const double* theta, int ndim, double* pars, double& dipeff,
                        double& propeff, double& f_beam) {
  for (int i = 0; i < 6; ++i) pars[i] = ((sp.unlog_mask >> i) & 1) ? exp10_ref(theta[i]) : theta[i];
  dipeff = sp.dipeff;
  propeff = sp.propeff;
  f_beam = sp.f_beam;
  if (ndim == 7) {
    f_beam = theta[6];
  } else if (ndim == 8) {
    dipeff = theta[6];
    propeff = theta[7];
  } else if (ndim == 9) {
    dipeff = theta[6];
    propeff = theta[7];
    f_beam = theta[8];
  }
}


// ---- one walker, in three stages ------------------------------------------------------------------
// A likelihood evaluation is cut where its work changes character (DESIGN.md section 3):
//   1 setup      prior test, theta -> physical parameters, per-walker constants, initial step size.  Same
//                work for every walker: one thread each, no divergence.                   (prepare_walker)
//   2 advance    the spin integration.  The ONLY stage whose cost differs between walkers (40 .. 10^3 steps
//                over the prior box, and an implicit integrator for the stiff ones): the kernels run it with
//                every lane pulling its next walker off a work queue the moment its current one is done, so a
//                warp's lanes all step on every trip whatever the spread of the ensemble.  Its product is the
//                state at the grid nodes the data need, dropped from the dense output into ybuf[walker][node].
//                                                        (integrator_load / integrator_step / drain_nodes)
//   3 reduce     luminosity at those nodes, interpolation onto the data, chi-square (or the model / light-curve
//                output).  Again the same work for every walker.                              (reduce_rows)
// The host simulator of the tests runs the three stages back to back for one walker at a time.
enum EvalMode { kModeLnprob = 0, kModeModelAtData = 1, kModeCurves = 2 };

struct WalkerRec {
  Walker w;
  double y0, h0, k1;     // explicit integrator at t_start: y = omega^-2, first step size, dy/dt
  unsigned regime0;      // spin_g's regime bits there
  int status;            // kWalkerPriorReject | kWalkerNonfiniteState | kWalkerIntegratorFail, or 0: to be integrated
  int n_rhs;             // right-hand-side evaluations spent so far
  int pad_;
};

// A walker on its way from the explicit to the implicit integrator (or, for a spec the explicit step does
// not implement, from setup straight to the implicit one).
struct StiffRec {
  double t, y, h;        // time, y = omega^-2 there, the step size in use
  int wid, jn;           // walker, node cursor
  int n_rhs, n_steps;
};

MP_HD void prepare_walker(const Spec& sp, const double* theta, int ndim, bool use_prior, const double* lower,
                          const double* upper, double t_start, double t_end, WalkerRec& r) {
  r.status = kWalkerOk;
  r.n_rhs = 0;
  r.y0 = r.h0 = r.k1 = 0.0;
  r.regime0 = 0u;
  r.pad_ = 0;
  if (use_prior && !prior_accepts(theta, ndim, lower, upper)) {   // mcmc_eqns.py:66-69: the model is skipped
    r.status = kWalkerPriorReject;
    return;
  }
  double pars[6], dipeff, propeff, f_beam;
  unpack_theta(sp, theta, ndim, pars, dipeff, propeff, f_beam);
  walker_setup(sp, pars, dipeff, propeff, f_beam, t_start, r.w);
  if (r.w.bad) {
    r.status = kWalkerNonfiniteState;
    return;
  }
  Integrator in;
  in.n_rhs = 0;
  if (sp.bucciantini) {
    // the explicit step does not carry this torque: the walker starts in the implicit integrator
    integrator_init<false>(sp, r.w, t_start, t_end, in);
    r.y0 = 1.0 / (in.omega * in.omega);
  } else {
    integrator_init<true>(sp, r.w, t_start, t_end, in);
    r.y0 = in.omega;
  }
  r.h0 = in.h;
  r.k1 = in.k1;
  r.regime0 = in.regime;
  r.n_rhs = in.n_rhs;
  // (t_end == t_start -- a handle without data, or one whose data all sit at the first grid time: the initial state
  // is the whole solution, and the zero step integrator_init leaves for an empty span is not a failure)
  if (in.status != kWalkerOk && t_end > t_start) r.status = kWalkerIntegratorFail;
}

// The explicit integrator as prepare_walker left it (C: the walker's disc-mass transient amplitude, Walker::C).
MP_HD void integrator_load(const WalkerRec& r, double C, double t_start, Integrator& in) {
  in.t = t_start;
  in.omega = r.y0;
  in.h = r.h0;
  in.k1 = r.k1;
  in.lfacold = StepControl::l_facold_min;
  in.rejected = 0;
  in.n_rhs = r.n_rhs;
  in.n_steps = 0;
  in.status = kWalkerOk;
  in.stiff = 0;
  in.stiff_votes = 0;
  in.have0 = 0;
  in.J0 = in.d0_qa = in.d0_ni = 0.0;
  in.E = C;
  in.regime = r.regime0;
  in.h_resume = 0.0;
  in.t0 = t_start; in.hs = 1.0;
  in.r1 = r.y0; in.r2 = in.r3 = in.r4 = in.r5 = 0.0;
}

// The implicit integrator taking a walker over at a StiffRec.
MP_HD void integrator_load_stiff(const StiffRec& q, Integrator& in) {
  integrator_resume(q.t, rsqrt_fast(q.y), q.h, in);
  in.n_rhs = q.n_rhs;
  in.n_steps = q.n_steps;
}

// Drop the state at every node the last accepted step covers into row[] (as y = omega^-2 whichever
// integrator produced it); returns the new node cursor.
// (row[j * rstride] is node j: the kernels lay ybuf out per dataset size, see Work in magprop_kernels.cu)
template <bool STIFF>
MP_HD int drain_nodes(const Integrator& in, int jn, int Nn, const double* node_t, double* row, size_t rstride = 1) {
  if (jn >= Nn) return jn;
  double tn = ldd(node_t + jn);
  if (!(tn <= in.t)) return jn;
  const double ihs = rcp_step(in.hs);
  do {
    const double v = dense_eval_r(in, tn, ihs);
    row[jn * rstride] = STIFF ? 1.0 / (v * v) : v;
    if (++jn >= Nn) break;
    tn = ldd(node_t + jn);
  } while (tn <= in.t);
  return jn;
}

// Luminosity stage at one node of one walker (state y = omega^-2 from ybuf): what stage 3 evaluates per node.
MP_HD Lum node_luminosity(const Spec& sp, const Walker& w, double tn, double t_start, double v, bool need_mass,
                          double& M, double& om) {
  if (w.bad) {                                   // unphysical constants: no solution beyond the initial node
    M = (tn == t_start) ? w.M_init : NAN;
    om = (tn == t_start) ? w.omega0 : NAN;
  } else {
    M = (sp.lum_dipole_only && !need_mass) ? 0.0 : disc_mass(w, tn);
    om = rsqrt_pos(v);                           // ~1 ulp; NaN for a failed walker's NaN
  }
  return luminosity(sp, w, M, om);
}

// Stage 3 for one walker, one node after the other (the form a thread runs when every thread of the warp has
// a walker of its own -- all lanes walk the same node and datum indices, so the loop is converged).
//   kModeLnprob      returns chi-square
//   kModeModelAtData out[dat_orig[i]*ostride] = model at sorted datum i (/1e50)
//   kModeCurves      out[(c*Nn + j)*ostride] = Ltot, Lprop, Ldip (c = 0,1,2), state_out likewise Mdisc, omega
template <int MODE>
MP_HD double reduce_rows(const Spec& sp, const DataView& dv, const Walker& w, const double* row, double* out,
                         double* state_out, int ostride, const int* dat_orig, size_t rstride = 1) {
  const int Nn = dv.n_nodes;
  double chi2 = 0.0, Lprev = 0.0;
  int idat = 0;
  // (the node values come from HBM, one per walker and node: the next node's is requested before this node's
  // luminosity is worked out, so its latency hides behind that arithmetic)
  double y_next = Nn > 0 ? row[0] : 0.0;
  for (int j = 0; j < Nn; ++j) {
    const double tn = ldd(dv.node_t + j);
    const double y_node = y_next;
    if (j + 1 < Nn) y_next = row[(size_t)(j + 1) * rstride];
    double M, om;
    const Lum L = node_luminosity(sp, w, tn, dv.t_start, y_node, MODE == kModeCurves && state_out, M, om);
    if (MODE == kModeCurves) {
      out[(0 * Nn + j) * ostride] = L.tot * 1.0e-50;            // (/1e50, funcs.py:231,236, as one multiplication: <= 1 ulp)
      out[(1 * Nn + j) * ostride] = L.prop * 1.0e-50;
      out[(2 * Nn + j) * ostride] = L.dip * 1.0e-50;
      if (state_out) {
        state_out[(0 * Nn + j) * ostride] = M;
        state_out[(1 * Nn + j) * ostride] = om;
      }
    } else {
      while (idat < dv.n_data) {
        const int lo = dv.dat_lo[idat];
        const double dx = ldd(dv.dat_dx + idat);
        const int hi = lo + (dx != 0.0 ? 1 : 0);
        if (hi > j) break;
        double mod;
        if (dx == 0.0) {
          mod = L.tot;                                   // datum sits on a grid node
        } else {
          mod = fma(L.tot - Lprev, ldd(dv.dat_w + idat), Lprev);   // np.interp: slope*(x-x_lo)+y_lo
        }
        if (MODE == kModeLnprob) {
          const double r = fma(-mod, ldd(dv.dat_c + idat), ldd(dv.dat_ys + idat));   // (y - mod/1e50)/yerr
          chi2 = fma(r, r, chi2);
        } else {
          out[(dat_orig ? dat_orig[idat] : idat) * ostride] = mod * 1.0e-50;
        }
        ++idat;
      }
      Lprev = L.tot;
    }
  }
  return chi2;
}

// lnlike from chi-square and the status so far (mcmc_eqns.py:22-25, 72-79); never NaN.
MP_HD double lnlike_of(double chi2, int& status) {
  double ll = -0.5 * chi2;                           // mcmc_eqns.py:25
  if (status & kWalkerIntegratorFail) {
    ll = -INFINITY;                                  // 'flag' -> -inf (mcmc_eqns.py:22-23)
  } else if (!isfinite(ll)) {
    status |= kWalkerNonfiniteLnlike;                // mcmc_eqns.py:72-79
    ll = -INFINITY;
  }
  return ll;
}

}  // namespace mp
