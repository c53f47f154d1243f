// WGS 84 coordinate transformations of the device warp: EPSG:4326 (degrees, x = lon),
// EPSG:3857 and the UTM zones (transverse Mercator, Krueger series to sixth order in n;
// Karney, J. Geodesy 85, 2011).  Same formulas and constants as dask_geomodeling_b200/crs.py;
// the series are summed by Clenshaw's recurrence on complex arguments, the host sums them
// term by term, so the two agree to a few ulps.  Host + device so that the maths can be
// checked on the CPU.
#pragma once
#include <math.h>
#include "../../include/geokernels.h"

namespace gm {
namespace crs {

constexpr double kPi = 3.141592653589793;
constexpr double kDeg = kPi / 180.0;      // numpy.radians
constexpr double kRad2Deg = 180.0 / kPi;  // numpy.degrees
constexpr double kRMerc = 6378137.0;
constexpr double kE = 0.08181919084262149;
constexpr double kE2 = 0.0066943799901413165;
constexpr double kK0A = 0.9996 * 6367449.145823415;   // k0 * rectifying radius
constexpr double kFE = 500000.0, kFNSouth = 10000000.0;
// Karney 2011 eqs. 35 (alpha, forward) and 36 (beta, inverse), WGS 84 values
__host__ __device__ constexpr double alpha(int j) {
  return j == 1 ? 0.0008377318206244698 : j == 2 ? 7.608527773572307e-07
       : j == 3 ? 1.1976455033294527e-09 : j == 4 ? 2.4291706072013587e-12
       : j == 5 ? 5.711757677865804e-15 : 1.4911177312583895e-17;
}
__host__ __device__ constexpr double beta(int j) {
  return j == 1 ? 0.0008377321640579486 : j == 2 ? 5.905870152220203e-08
       : j == 3 ? 1.6734826652839968e-10 : j == 4 ? 2.1647980400627059e-13
       : j == 5 ? 3.7879780461686053e-16 : 7.2487488906941545e-19;
}

// (xi, eta) += sign * sum_j c_j sin(2 j (xi + i eta)), Clenshaw on the complex sine series
template <bool Forward>
__host__ __device__ inline void krueger(double& xi, double& eta) {
  double s2, c2;
  sincos(2.0 * xi, &s2, &c2);
  const double sh = sinh(2.0 * eta), ch = cosh(2.0 * eta);
  // w = 2 cos(2z) = 2 (c2 ch - i s2 sh)
  const double wr = 2.0 * c2 * ch, wi = -2.0 * s2 * sh;
  double br = 0.0, bi = 0.0, b2r = 0.0, b2i = 0.0;   // b_{k+1}, b_{k+2}
#pragma unroll
  for (int k = 6; k >= 1; --k) {
    const double c = Forward ? alpha(k) : beta(k);
    const double nr = c + (wr * br - wi * bi) - b2r;
    const double ni = (wr * bi + wi * br) - b2i;
    b2r = br; b2i = bi; br = nr; bi = ni;
  }
  // sum = b_1 * sin(2z), sin(2z) = s2 ch + i c2 sh
  const double sr = s2 * ch, si = c2 * sh;
  const double sum_r = br * sr - bi * si, sum_i = br * si + bi * sr;
  if (Forward) { xi += sum_r; eta += sum_i; } else { xi -= sum_r; eta -= sum_i; }
}

__host__ __device__ inline double central_meridian(int zone) {
  return 6.0 * (double)(zone < 0 ? -zone : zone) - 183.0;
}

// UTM (x, y) of zone `zone` (+north / -south) -> degrees
__host__ __device__ inline void utm_inverse(double& x, double& y, int zone) {
  double xi = (y - (zone < 0 ? kFNSouth : 0.0)) / kK0A;
  double eta = (x - kFE) / kK0A;
  krueger<false>(xi, eta);
  double sx, cx;
  sincos(xi, &sx, &cx);
  const double she = sinh(eta);
  const double tau_c = sx / hypot(she, cx);
  const double lam = atan2(she, cx);
  double tau = tau_c;
#pragma unroll
  for (int it = 0; it < 3; ++it) {   // conformal -> geographic latitude (Karney 2011, eqs. 19-21)
    const double st = sqrt(1.0 + tau * tau);
    const double sigma = sinh(kE * atanh(kE * tau / st));
    const double tc = tau * sqrt(1.0 + sigma * sigma) - sigma * st;
    tau += (tau_c - tc) / sqrt(1.0 + tc * tc) * (1.0 + (1.0 - kE2) * (tau * tau)) / ((1.0 - kE2) * st);
  }
  x = lam * kRad2Deg + central_meridian(zone);
  y = atan(tau) * kRad2Deg;
}

// degrees -> UTM (x, y) of zone `zone`; |lat| > 90 gives NaN
__host__ __device__ inline void utm_forward(double& x, double& y, int zone) {
  if (fabs(y) > 90.0) { x = y = NAN; return; }
  const double phi = y * kDeg, lam = (x - central_meridian(zone)) * kDeg;
  const double tau = tan(phi);
  const double sigma = sinh(kE * atanh(kE * sin(phi)));
  const double tau_c = tau * sqrt(1.0 + sigma * sigma) - sigma * sqrt(1.0 + tau * tau);
  double sl, cl;
  sincos(lam, &sl, &cl);
  double xi = atan2(tau_c, cl);
  double eta = asinh(sl / hypot(tau_c, cl));
  krueger<true>(xi, eta);
  x = kFE + kK0A * eta;
  y = kK0A * xi + (zone < 0 ? kFNSouth : 0.0);
}

// EPSG:4326 <-> EPSG:3857: x depends on x only and y on y only
__host__ __device__ inline bool is_separable(int a, int b) {
  return (a == GM_CRS_GEOGRAPHIC && b == GM_CRS_MERCATOR) || (a == GM_CRS_MERCATOR && b == GM_CRS_GEOGRAPHIC);
}

// (x, y) in CRS (kind, zone) -> degrees, in place
__host__ __device__ inline void to_degrees(double& x, double& y, int kind, int zone) {
  if (kind == GM_CRS_MERCATOR) {
    x = (x / kRMerc) * kRad2Deg;
    y = (2.0 * atan(exp(y / kRMerc)) - kPi / 2) * kRad2Deg;
  } else if (kind == GM_CRS_UTM) {
    utm_inverse(x, y, zone);
  }
}

// degrees -> (x, y) in CRS (kind, zone), in place; a pole in EPSG:3857 gives +-inf
__host__ __device__ inline void from_degrees(double& x, double& y, int kind, int zone) {
  if (kind == GM_CRS_GEOGRAPHIC) {
    if (fabs(y) > 90.0) y = NAN;
  } else if (kind == GM_CRS_MERCATOR) {
    if (fabs(y) > 90.0) { x = y = NAN; return; }
    x = kRMerc * (x * kDeg);
    y = kRMerc * atanh(sin(y * kDeg));
  } else {
    utm_forward(x, y, zone);
  }
}

}  // namespace crs
}  // namespace gm
