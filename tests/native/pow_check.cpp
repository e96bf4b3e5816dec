// TEST INFRASTRUCTURE - every literal-power helper the generator can emit (inflx_device.cuh:
// inflx_powi<3..64>, inflx_powi_neg<2..64>, inflx_powh<1..63>, inflx_powh_neg<0..63>) under both
// policies, and a libquadmath reference (tests/test_power_helpers.py, tests/test_gpu_power_helpers.py).
//
// Host build: g++ -std=c++17 -ffp-contract=off -fopenmp -DINFLX_DEVICE_HEADER="..." -lquadmath;
// the hardware seeds are then IEEE values (cuda_host_shim.h).  Device build: the GPU test prepends
// the device header and defines INFLX_POW_CHECK_DEVICE; the dispatch below is shared.
//
// kind 0: x^N, 1: x^-N, 2: x^(N+1/2), 3: x^-(N+1/2)
#ifndef INFLX_POW_CHECK_DEVICE
#include "cuda_host_shim.h"
#include INFLX_DEVICE_HEADER
#include <float.h>
#include <quadmath.h>
#endif

template <int K, int N, class OPS>
__device__ __forceinline__ double pw_one(double x, OPS ops) {
  if constexpr (K == 0) return inflx_powi<(N >= 1 ? N : 1)>(x, ops);
  else if constexpr (K == 1) return inflx_powi_neg<(N >= 1 ? N : 1)>(x, ops);
  else if constexpr (K == 2) return inflx_powh<N>(x, ops);
  else return inflx_powh_neg<N>(x, ops);
}

#define PW_C1(K, n) \
  case n:           \
    return pw_one<K, n>(x, ops);
#define PW_C8(K, n) \
  PW_C1(K, n) PW_C1(K, n + 1) PW_C1(K, n + 2) PW_C1(K, n + 3) PW_C1(K, n + 4) PW_C1(K, n + 5) \
  PW_C1(K, n + 6) PW_C1(K, n + 7)
#define PW_C64(K) \
  PW_C8(K, 0) PW_C8(K, 8) PW_C8(K, 16) PW_C8(K, 24) PW_C8(K, 32) PW_C8(K, 40) PW_C8(K, 48) \
  PW_C8(K, 56) PW_C1(K, 64)

template <int K, class OPS>
__device__ double pw_kind(int n, double x, OPS ops) {
  switch (n) { PW_C64(K) }
  return __longlong_as_double(0x7ff4000000000000ll);  // no such instance
}

template <class OPS>
__device__ __forceinline__ double pw(int kind, int n, double x, OPS ops) {
  switch (kind) {
    case 0: return pw_kind<0>(n, x, ops);
    case 1: return pw_kind<1>(n, x, ops);
    case 2: return pw_kind<2>(n, x, ops);
    default: return pw_kind<3>(n, x, ops);
  }
}

#ifdef INFLX_POW_CHECK_DEVICE
// sel = {kind, n}; exact policy, and the speculative policy's value and flag
extern "C" __global__ void pow_eval(const double* x, const int* sel, double* exact, double* spec,
                                    unsigned char* flag, int m) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  exact[i] = pw(sel[0], sel[1], x[i], inflx_exact());
  inflx_chk bad;
  spec[i] = pw(sel[0], sel[1], x[i], inflx_spec(bad));
  flag[i] = bad.any();
}
#else
extern "C" void pow_eval(int kind, int n, const double* x, long m, double* exact, double* spec,
                         unsigned char* flag) {
#pragma omp parallel for schedule(static)
  for (long i = 0; i < m; i++) {
    exact[i] = pw(kind, n, x[i], inflx_exact());
    inflx_chk bad;
    spec[i] = pw(kind, n, x[i], inflx_spec(bad));
    flag[i] = bad.any();
  }
}

// powq(x, y) rounded to double, the distance of the quad value from the nearest rounding boundary
// of that rounding (in ulps of the result; 0.5 means halfway between two boundaries), and glibc's
// pow(x, y)
extern "C" void pow_ref(double y, const double* x, long m, double* ref, double* dist, double* libm) {
#pragma omp parallel for schedule(dynamic, 256)
  for (long i = 0; i < m; i++) {
    const __float128 q = powq((__float128)x[i], (__float128)y);
    const double r = (double)q;
    ref[i] = r;
    libm[i] = pow(x[i], y);
    dist[i] = 0.5;
    if (isnanq(q) || isinfq(q) || q == 0) continue;
    const double rr = isinf(r) ? copysign(DBL_MAX, r) : r;
    const double dn = nextafter(rr, -INFINITY), up = nextafter(rr, INFINITY);
    // spacing below and above rr (beyond +-DBL_MAX: the spacing of the last binade)
    const __float128 sp_dn = isinf(dn) ? (__float128)up - rr : (__float128)rr - dn;
    const __float128 sp_up = isinf(up) ? (__float128)rr - dn : (__float128)up - rr;
    const __float128 d_dn = fabsq(q - (rr - sp_dn / 2)) / sp_dn, d_up = fabsq(q - (rr + sp_up / 2)) / sp_up;
    dist[i] = (double)fminq(d_dn, d_up);
  }
}
#endif
