// The boundary source of every wave model, one definition for the host (wfx_wave.cu: the amplitudes of an
// unprofiled step) and the device (wfx_boundary.cu: per-dof delayed sources of a source profile).
#pragma once

#include <cmath>

#ifdef __CUDACC__
#define WFX_HD __host__ __device__
#else
#define WFX_HD
#endif

namespace wfx
{
// g(t) of LinearGLL.hpp:155-162, a Hann ramp over the first alpha = 4 periods (:96-99),
//   g = W(t) p0 w0 / c0 cos(w0 t),
// and its time derivative g'(t) = p0 w0 / c0 (W'(t) cos(w0 t) - W(t) w0 sin(w0 t)), W' = 0 after the ramp
WFX_HD inline void source_eval(double f0, double p0, double c0, double tn, double* g, double* gdot)
{
  const double w0 = 2.0 * M_PI * f0, T = 1.0 / f0, alpha = 4.0;
  const bool ramp = tn < T * alpha;
  const double window = ramp ? 0.5 * (1.0 - cos(f0 * M_PI * tn / alpha)) : 1.0;
  const double rate = ramp ? f0 * M_PI / (2.0 * alpha) * sin(f0 * M_PI * tn / alpha) : 0.0;
  *g = window * p0 * w0 / c0 * cos(w0 * tn);
  *gdot = p0 * w0 / c0 * (rate * cos(w0 * tn) - window * w0 * sin(w0 * tn));
}
} // namespace wfx
