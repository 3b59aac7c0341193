// magprop_models.cu -- restatements of the reference's model code outside the likelihood pipeline: the coupled
// right-hand side as ODEs()/odes() return it (mp_rhs_batch), and the comparison model of figure 5
// (mp_gompertz_curves).  One thread per walker or parameter set, the reference's operation order kept.
#include <cuda_runtime.h>

#include "magprop_abi.hpp"
#include "magprop_constants.hpp"

namespace mp {

// ---- the coupled right-hand side, as ODEs()/odes() return it -----------------------
// funcs.py:75-142 / magnetar/funcs.py:33-101, operation order kept.
__global__ void rhs_kernel(double inertia_factor, double mdot_factor, double breakup, int dipole_torque,
                           const double* __restrict__ y, const double* __restrict__ t,
                           const double* __restrict__ pars, double n, double alpha, double cs7, double k,
                           int W, double* __restrict__ dydt) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= W) return;
  const double Mdisc = y[2 * i], omega = y[2 * i + 1], tt = t[i];
  const double B = pars[5 * i], MdiscI = pars[5 * i + 1], RdiscI = pars[5 * i + 2];
  const double epsilon = pars[5 * i + 3], delta = pars[5 * i + 4];
  const double inertia = inertia_factor * kM * (kR * kR);
  const double Rdisc = RdiscI * 1.0e5;
  const double tvisc = Rdisc / (alpha * cs7 * 1.0e7);
  const double mu = 1.0e15 * B * (kR * kR * kR);
  const double M0 = delta * MdiscI * kMsol;
  const double tfb = epsilon * tvisc;
  double Rm = pow(mu, 4.0 / 7.0) * pow(kGM, -1.0 / 7.0) * pow((mdot_factor * Mdisc) / tvisc, -2.0 / 7.0);
  const double Rc = pow(kGM / (omega * omega), 1.0 / 3.0);
  const double Rlc = kC / omega;
  if (Rm >= k * Rlc) Rm = k * Rlc;
  const double w = pow(Rm / Rc, 1.5);
  const double x = kGM / (kR * (kC * kC));
  const double modW = 0.6 * kM * (kC * kC) * (x / (1.0 - 0.5 * x));
  const double rot_param = (0.5 * inertia * (omega * omega)) / modW;
  double Ndip = (-1.0 * (mu * mu) * (omega * omega * omega)) / (6.0 * (kC * kC * kC));
  if (dipole_torque) {                                  // figure_3.py:142-143
    const double q = Rlc / Rm;
    Ndip = (-2.0 / 3.0) * (((mu * mu) * (omega * omega * omega)) / (kC * kC * kC)) * (q * q * q);
  }
  const double eta2 = 0.5 * (1.0 + tanh(n * (w - 1.0)));
  const double eta1 = 1.0 - eta2;
  const double Mdotprop = eta2 * (Mdisc / tvisc);
  const double Mdotacc = eta1 * (Mdisc / tvisc);
  const double Mdotfb = (M0 / tfb) * pow((tt + tfb) / tfb, -5.0 / 3.0);
  double Nacc;
  if (rot_param > breakup) Nacc = 0.0;
  else if (Rm >= kR) Nacc = sqrt(kGM * Rm) * (Mdotacc - Mdotprop);
  else Nacc = sqrt(kGM * kR) * (Mdotacc - Mdotprop);
  dydt[2 * i] = Mdotfb - Mdotacc - Mdotprop;
  dydt[2 * i + 1] = (Nacc + Ndip) / inertia;
}

// ---- the comparison model of code/figure_5.py:222-363 ("Ben's model") --------------------------------------
// An accreting-mass magnetar with an exponentially draining disc, advanced by explicit Euler steps of 1 s (the
// reference: a Python loop over 1e6 array elements per parameter set).  One parameter set per thread, the script's
// operation order kept (fractional powers through pow, as NumPy's **); every `stride`-th step is stored.
// out [W][3][n_out] = Ltot, Lprop, Ldip in units of 1e50 erg/s (figure_5.py:354-368).
__global__ void gompertz_kernel(const double* __restrict__ pars, int W, double alpha, double cs7, double k, double omass,
                                double dipeff, double propeff, long long n_steps, int stride, long long n_out,
                                double* __restrict__ out) {
  const int wi = blockIdx.x * blockDim.x + threadIdx.x;
  if (wi >= W) return;
  const double B = pars[6 * wi], P = pars[6 * wi + 1], MdiscI = pars[6 * wi + 2], RdiscI = pars[6 * wi + 3];
  const double spin = P * 1.0e-3;                               // :224
  const double Rdisc = RdiscI * 1.0e5;
  const double visc = alpha * cs7 * 1.0e7 * Rdisc;
  const double mu = 1.0e15 * B * (kR * kR * kR);
  double omega = (2.0 * 3.141592653589793) / spin;             // :229
  const double Mdisc0 = MdiscI * kMsol;
  double M_bg = omass * kMsol;
  const double Mdot0 = (3.0 * Mdisc0 * visc) / (Rdisc * Rdisc);  // :258
  double Mdot = Mdot0, Msum = 0.0, tt = 1.0, omegadot = 0.0;
  const double mu47 = pow(mu, 4.0 / 7.0), mu2 = mu * mu, c3 = kC * kC * kC, c2 = kC * kC, R2 = kR * kR, R3 = kR * kR * kR;
  double* o = out + (size_t)wi * 3 * n_out;
  for (long long i = 0; i < n_steps; ++i) {
    if (i > 0) {                                                // :302-309
      tt = tt + 1.0;
      omega = omega + omegadot;
      M_bg = M_bg + Msum;
      Mdot = Mdot0 * exp((-3.0 * visc * tt) / (Rdisc * Rdisc));
    }
    const double GMb = kG * M_bg;
    double Rm = mu47 * pow(GMb, -1.0 / 7.0) * pow(Mdot, -2.0 / 7.0);
    const double Rc = pow(GMb / (omega * omega), 1.0 / 3.0);
    const double light = kC / omega;
    if (Rm >= (k * light)) Rm = k * light;
    const double lr = light / Rm;
    const double Ndip = (-2.0 / 3.0) * ((mu2 * (omega * omega * omega)) / c3) * (lr * lr * lr);
    const double w = pow(Rm / Rc, 1.5);
    const double nn = 1.0 - w;
    const double inertia = 0.35 * M_bg * R2;
    const double bigT = 0.5 * inertia * (omega * omega);
    const double x = GMb / (kR * c2);
    const double modW = 0.6 * M_bg * c2 * (x / (1.0 - 0.5 * x));
    const double beta = bigT / modW;
    double Nacc;
    if (beta > 0.27) {
      Nacc = 0.0;
    } else if (Rm >= kR) {
      Nacc = nn * sqrt(GMb * Rm) * Mdot;
      if (!isfinite(Nacc)) Nacc = 0.0;
    } else {
      const double f = 1.0 - (omega / sqrt(GMb / R3));
      Nacc = (i == 0) ? f / sqrt(GMb * kR) * Mdot : f * sqrt(GMb * kR) * Mdot;   // (:283-285 divides, :335-337 multiplies)
      if (!isfinite(Nacc)) Nacc = 0.0;
    }
    if (Rc >= Rm) Msum = Mdot;                                  // :293-296, :341-344
    else if (i == 0) Msum = 0.0;
    omegadot = (Ndip + Nacc) / inertia;
    if (i % stride == 0) {
      double lp = (-1.0 * Nacc * omega) - ((GMb * Mdot) / Rm);
      double ld = (mu2 * ((omega * omega) * (omega * omega))) / (6.0 * c3);
      if (!isfinite(lp) || lp <= 0.0) lp = 0.0;                 // :354-361
      if (!isfinite(ld) || ld <= 0.0) ld = 0.0;
      const long long jo = i / stride;
      o[jo] = ((propeff * lp) + (dipeff * ld)) * 1.0e-50;
      o[n_out + jo] = lp * 1.0e-50;
      o[2 * n_out + jo] = ld * 1.0e-50;
    }
  }
}

}  // namespace mp

using namespace mp;

extern "C" int mp_rhs_batch(const mp_model_spec* spec, const double* y, const double* t, const double* pars,
                            const double* knobs, int32_t W, double* dydt, int32_t device) {
  if (!spec || !y || !t || !pars || !knobs || !dydt || W < 0) return fail(MP_ERR_BAD_ARG, "mp_rhs_batch: null pointer");
  if (W == 0) return MP_OK;
  int rc = select_device(device, "mp_rhs_batch");
  if (rc) return rc;
  DevBuf<double> d_all;   // one allocation for the four arrays: y[2W] t[W] pars[5W] dydt[2W]
  MP_CUDA(d_all.ensure((size_t)W * 10));
  double *d_y = d_all.get(), *d_t = d_y + (size_t)2 * W, *d_p = d_y + (size_t)3 * W, *d_o = d_y + (size_t)8 * W;
  MP_CUDA(cudaMemcpy(d_y, y, (size_t)W * 2 * sizeof(double), cudaMemcpyHostToDevice));
  MP_CUDA(cudaMemcpy(d_t, t, (size_t)W * sizeof(double), cudaMemcpyHostToDevice));
  MP_CUDA(cudaMemcpy(d_p, pars, (size_t)W * 5 * sizeof(double), cudaMemcpyHostToDevice));
  rhs_kernel<<<(W + 127) / 128, 128>>>(spec->inertia_factor, spec->mdot_factor, spec->breakup_rhs, spec->dipole_torque, d_y, d_t, d_p,
                                       knobs[0], knobs[1], knobs[2], knobs[3], W, d_o);
  MP_CUDA(cudaGetLastError());
  MP_CUDA(cudaMemcpy(dydt, d_o, (size_t)W * 2 * sizeof(double), cudaMemcpyDeviceToHost));
  return MP_OK;
}

extern "C" int mp_gompertz_curves(const double* pars, int32_t W, const double* knobs, int64_t n_steps, int32_t stride,
                                  double* out, int32_t device) {
  if (!pars || !knobs || !out || W < 0 || n_steps < 1 || stride < 1) return fail(MP_ERR_BAD_ARG, "mp_gompertz_curves: bad argument");
  if (W == 0) return MP_OK;
  int rc = select_device(device, "mp_gompertz_curves");
  if (rc) return rc;
  const long long n_out = (n_steps + stride - 1) / stride;
  DevBuf<double> d_p, d_o;
  MP_CUDA(d_p.ensure((size_t)W * 6));
  MP_CUDA(d_o.ensure((size_t)W * 3 * n_out));
  MP_CUDA(cudaMemcpy(d_p.get(), pars, (size_t)W * 6 * sizeof(double), cudaMemcpyHostToDevice));
  gompertz_kernel<<<(W + 31) / 32, 32>>>(d_p.get(), W, knobs[0], knobs[1], knobs[2], knobs[3], knobs[4], knobs[5], n_steps, stride,
                                         n_out, d_o.get());
  MP_CUDA(cudaGetLastError());
  MP_CUDA(cudaMemcpy(out, d_o.get(), (size_t)W * 3 * n_out * sizeof(double), cudaMemcpyDeviceToHost));
  return MP_OK;
}
