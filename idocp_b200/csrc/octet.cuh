// octet.cuh -- "octet" execution model helpers (sm_100a) and the CANONICAL ARITHMETIC.
//
// One OCTET = 8 consecutive lanes of a warp works on one (instance, stage) pair or one
// instance; lane l < 7 owns joint l / matrix column l of the 7-dof iiwa14, lane 7 is padding.
// A warp therefore carries 4 independent problems; all cross-lane traffic stays inside the
// octet (width-8 shuffles, per-octet shared-memory tiles).
//
// HBM layout ("slots"): every per-joint vector is one 64-byte slot [8 doubles]; arrays are
// [slot][instance][8] so the 4 octets of a warp (4 consecutive instances) touch 256 contiguous
// bytes per load/store.
//
// Canonical arithmetic: the library is compiled with -fmad=false, so the compiler never
// contracts a*b+c on its own; every fused multiply-add is written explicitly with fma().
// The CPU oracle (oracle/idocp_oracle.c, gcc -ffp-contract=off) performs the SAME sequence of
// IEEE-754 operations (same fma placement, same tree order in the prefix/suffix scans, same
// polynomial sin/cos), which makes the GPU results bit-identical to the oracle's.
#pragma once
#ifndef IDOCP_B200_EMU
#include <cuda_runtime.h>
#endif

namespace idocp_b200 {

constexpr int NV = 7;        // iiwa14 nq = nv = nu
constexpr int OCT = 8;       // lanes per octet
constexpr unsigned FULL = 0xffffffffu;

struct V3 {
  double x, y, z;
};

__device__ __forceinline__ V3 v3(double x, double y, double z) { return V3{x, y, z}; }
__device__ __forceinline__ V3 operator+(V3 a, V3 b) { return V3{a.x + b.x, a.y + b.y, a.z + b.z}; }
__device__ __forceinline__ V3 operator-(V3 a, V3 b) { return V3{a.x - b.x, a.y - b.y, a.z - b.z}; }
__device__ __forceinline__ V3 operator*(double s, V3 a) { return V3{s * a.x, s * a.y, s * a.z}; }
// s * a + b, fused
__device__ __forceinline__ V3 fmav(double s, V3 a, V3 b) { return V3{fma(s, a.x, b.x), fma(s, a.y, b.y), fma(s, a.z, b.z)}; }
__device__ __forceinline__ V3 cross(V3 a, V3 b) {
  return V3{fma(a.y, b.z, -(a.z * b.y)), fma(a.z, b.x, -(a.x * b.z)), fma(a.x, b.y, -(a.y * b.x))};
}
__device__ __forceinline__ double dot(V3 a, V3 b) { return fma(a.z, b.z, fma(a.y, b.y, a.x * b.x)); }

// symmetric 3x3 (xx,xy,xz,yy,yz,zz)
struct S3 {
  double xx, xy, xz, yy, yz, zz;
};
__device__ __forceinline__ V3 mul(const S3& A, V3 b) {
  return V3{fma(A.xz, b.z, fma(A.xy, b.y, A.xx * b.x)), fma(A.yz, b.z, fma(A.yy, b.y, A.xy * b.x)),
            fma(A.zz, b.z, fma(A.yz, b.y, A.xz * b.x))};
}

// sin / cos: Cody-Waite reduction by pi/2 + the classic degree-13/14
// minimax kernels, written with explicit fma so that the oracle can repeat it bit for bit.
__device__ __forceinline__ void canon_sincos(double x, double* sn, double* cs) {
  const double k = rint(x * 6.36619772367581382433e-01);            // x * 2/pi
  double r = fma(-k, 1.57079632673412561417e+00, x);                // pi/2, first 33 bits
  r = fma(-k, 6.07710050650619224932e-11, r);                       // pi/2 tail
  const double z = r * r;
  double ps = fma(z, 1.58969099521155010221e-10, -2.50507602534068634195e-08);
  ps = fma(z, ps, 2.75573137070700676789e-06);
  ps = fma(z, ps, -1.98412698298579493134e-04);
  ps = fma(z, ps, 8.33333333332248946124e-03);
  ps = fma(z, ps, -1.66666666666666324348e-01);
  const double s = fma(r * z, ps, r);
  double pc = fma(z, -1.13596475577881948265e-11, 2.08757232129817482790e-09);
  pc = fma(z, pc, -2.75573143513906633035e-07);
  pc = fma(z, pc, 2.48015872894767294178e-05);
  pc = fma(z, pc, -1.38888888888741095749e-03);
  pc = fma(z, pc, 4.16666666666666019037e-02);
  const double c = fma(z * z, pc, fma(-0.5, z, 1.0));
  const int q = static_cast<int>(static_cast<long long>(k) & 3);   // exact for every |k| < 2^53 (an int overflows past 2^31)
  *sn = (q == 0) ? s : (q == 1) ? c : (q == 2) ? -s : -c;
  *cs = (q == 0) ? c : (q == 1) ? -s : (q == 2) ? -c : s;
}

// Reciprocal square root of a Cholesky pivot: r ~ 1 / sqrt(x) within about one ulp.  A Cholesky column needs only
// r (L_ik = A_ik r; L_kk = x r where somebody reads it), and IEEE sqrt followed by an IEEE division is the longest
// dependent chain of every factorisation here (two library sequences of ~10 dependent FP64 operations each, on the
// critical path of 7 / 18 / 21 sequential pivots).  Canonical definition, repeated operation by operation by the
// oracle (oracle/canon_pivot.h): the seed is the single-precision 1 / sqrt(float(x)) formed with two correctly
// rounded IEEE operations (identical on every IEEE machine), refined by two Newton steps in explicit FP64 fma form
// (relative error 2e-7 -> 5e-14 -> rounding).  Pivots outside (1e-36, 1e36) are reported as failed factorisations
// (canon_pivot_ok): beyond that range the single-precision seed would overflow or vanish.
__device__ __forceinline__ bool canon_pivot_ok(double x) { return x > 1e-36 && x < 1e36; }
__device__ __forceinline__ double canon_rsqrt(double x) {
#ifdef IDOCP_B200_EMU
  const float xf = static_cast<float>(x);
  const float yf = 1.0f / sqrtf(xf);
#else
  const float yf = __fdiv_rn(1.0f, __fsqrt_rn(__double2float_rn(x)));
#endif
  double y = static_cast<double>(yf);
  const double h = 0.5 * x;
  double e = fma(-(h * y), y, 0.5);
  y = fma(y, e, y);
  e = fma(-(h * y), y, 0.5);
  y = fma(y, e, y);
  return y;
}

// natural logarithm (barrier cost of the line search): the classic fdlibm k*ln2 + log(1+f) reduction with the
// degree-14 minimax polynomial in s = f/(2+f), written with plain IEEE operations so that the oracle repeats it bit for
// bit.  Subnormals are scaled by 2^54 first; 0, negatives, NaN and +inf give std::log's results.
__device__ __forceinline__ double canon_log(double x) {
  int k = 0;
  if (!(x >= 2.2250738585072014e-308)) {   // not a positive normal: 0, subnormal, negative or NaN
    if (x == 0.0) return -1.0 / 0.0;
    if (!(x > 0.0)) return (x != x) ? x : 0.0 / 0.0;
    x *= 18014398509481984.0;              // 2^54
    k = -54;
  } else if (!(x < 1.0 / 0.0)) {
    return x;                              // log(+inf) = +inf
  }
  long long bits;
#ifdef IDOCP_B200_EMU
  memcpy(&bits, &x, sizeof(bits));
#else
  bits = __double_as_longlong(x);
#endif
  int hx = static_cast<int>(bits >> 32);
  k += (hx >> 20) - 1023;
  hx &= 0x000fffff;
  const int i = (hx + 0x95f64) & 0x100000;       // mantissa >= sqrt(2): use x/2, k+1
  k += (i >> 20);
  const long long nb = (static_cast<long long>(hx | (i ^ 0x3ff00000)) << 32) | (bits & 0xffffffffLL);
  double m;
#ifdef IDOCP_B200_EMU
  memcpy(&m, &nb, sizeof(m));
#else
  m = __longlong_as_double(nb);
#endif
  const double f = m - 1.0;
  const double s = f / (2.0 + f);
  const double dk = static_cast<double>(k);
  const double z = s * s;
  const double w = z * z;
  const double t1 = w * (3.999999999940941908e-01 + w * (2.222219843214978396e-01 + w * 1.531383769920937332e-01));
  const double t2 = z * (6.666666666666735130e-01 +
                         w * (2.857142874366239149e-01 + w * (1.818357216161805012e-01 + w * 1.479819860511658591e-01)));
  const double R = t2 + t1;
  const double hfsq = 0.5 * f * f;
  return dk * 6.93147180369123816490e-01 - ((hfsq - (s * (hfsq + R) + dk * 1.90821492927058770002e-10)) - f);
}

// acos on [-1, 1]: the fdlibm e_acos.c algorithm with plain IEEE operations (task-space cost: log3 of
// the end-effector rotation error); the oracle repeats it bit for bit.  Arguments below -1 give pi, above 1 give 0,
// NaN gives NaN.
__device__ __forceinline__ double canon_acos_poly(double z) {
  const double pS0 = 1.66666666666666657415e-01, pS1 = -3.25565818622400915405e-01, pS2 = 2.01212532134862925881e-01,
               pS3 = -4.00555345006794114027e-02, pS4 = 7.91534994289814532176e-04, pS5 = 3.47933107596021167570e-05;
  const double qS1 = -2.40339491173441421878e+00, qS2 = 2.02094576023350569471e+00, qS3 = -6.88283971605453293030e-01,
               qS4 = 7.70381505559019352791e-02;
  const double pp = z * (pS0 + z * (pS1 + z * (pS2 + z * (pS3 + z * (pS4 + z * pS5)))));
  const double qq = 1.0 + z * (qS1 + z * (qS2 + z * (qS3 + z * qS4)));
  return pp / qq;
}
__device__ __forceinline__ double canon_acos(double x) {
  const double pio2_hi = 1.57079632679489655800e+00, pio2_lo = 6.12323399573676603587e-17;
  const double pi = 3.14159265358979311600e+00;
  if (!(x > -1.0)) return (x != x) ? x : pi;
  if (!(x < 1.0)) return 0.0;
  if (fabs(x) < 0.5) {
    const double r = canon_acos_poly(x * x);
    return pio2_hi - (x - (pio2_lo - x * r));
  }
  if (x < 0.0) {
    const double z = (1.0 + x) * 0.5;
    const double sq = sqrt(z);
    const double r = canon_acos_poly(z);
    const double w = r * sq - pio2_lo;
    return pi - 2.0 * (sq + w);
  }
  const double z = (1.0 - x) * 0.5;
  const double sq = sqrt(z);
  long long bits;
#ifdef IDOCP_B200_EMU
  memcpy(&bits, &sq, sizeof(bits));
#else
  bits = __double_as_longlong(sq);
#endif
  bits &= static_cast<long long>(0xffffffff00000000ULL);   // df = sq with the low word cleared
  double df;
#ifdef IDOCP_B200_EMU
  memcpy(&df, &bits, sizeof(df));
#else
  df = __longlong_as_double(bits);
#endif
  const double c = (z - df * df) / (sq + df);
  const double r = canon_acos_poly(z);
  const double w = r * sq + c;
  return 2.0 * (df + w);
}

__device__ __forceinline__ int lane_in_octet() { return threadIdx.x & 7; }

// width-8 shuffles on doubles / V3
__device__ __forceinline__ double oct_up(double x, int d) { return __shfl_up_sync(FULL, x, d, OCT); }
__device__ __forceinline__ double oct_down(double x, int d) { return __shfl_down_sync(FULL, x, d, OCT); }
__device__ __forceinline__ double oct_bcast(double x, int src) { return __shfl_sync(FULL, x, src, OCT); }
__device__ __forceinline__ V3 oct_up(V3 a, int d) { return V3{oct_up(a.x, d), oct_up(a.y, d), oct_up(a.z, d)}; }
__device__ __forceinline__ V3 oct_down(V3 a, int d) {
  return V3{oct_down(a.x, d), oct_down(a.y, d), oct_down(a.z, d)};
}

// Hillis-Steele inclusive scans over the octet.  The "add only where the source lane exists"
// predicate is applied as x = fma(y, flag, x) with flag in {0.0, 1.0}: fma(y, 1, x) == x + y and
// fma(y, 0, x) == x exactly, i.e. bit-identical to a predicated add, in one FP64 instruction.
struct ScanFlags {
  double p1, p2, p4;  // prefix: lane >= d
  double s1, s2, s4;  // suffix: lane + d < 8
};
__device__ __forceinline__ ScanFlags scan_flags(int lane) {
  ScanFlags f;
  f.p1 = lane >= 1 ? 1.0 : 0.0; f.p2 = lane >= 2 ? 1.0 : 0.0; f.p4 = lane >= 4 ? 1.0 : 0.0;
  f.s1 = lane + 1 < OCT ? 1.0 : 0.0; f.s2 = lane + 2 < OCT ? 1.0 : 0.0; f.s4 = lane + 4 < OCT ? 1.0 : 0.0;
  return f;
}
// inclusive prefix sum (lane order 0..7)
__device__ __forceinline__ double oct_prefix_sum(double x, const ScanFlags& f) {
  x = fma(oct_up(x, 1), f.p1, x);
  x = fma(oct_up(x, 2), f.p2, x);
  x = fma(oct_up(x, 4), f.p4, x);
  return x;
}
__device__ __forceinline__ V3 oct_prefix_sum(V3 a, const ScanFlags& f) {
  return V3{oct_prefix_sum(a.x, f), oct_prefix_sum(a.y, f), oct_prefix_sum(a.z, f)};
}
// inclusive suffix sum: x_l <- sum_{k >= l} x_k   (lane 7 must hold 0)
__device__ __forceinline__ double oct_suffix_sum(double x, const ScanFlags& f) {
  x = fma(oct_down(x, 1), f.s1, x);
  x = fma(oct_down(x, 2), f.s2, x);
  x = fma(oct_down(x, 4), f.s4, x);
  return x;
}
__device__ __forceinline__ V3 oct_suffix_sum(V3 a, const ScanFlags& f) {
  return V3{oct_suffix_sum(a.x, f), oct_suffix_sum(a.y, f), oct_suffix_sum(a.z, f)};
}
__device__ __forceinline__ double oct_min(double x) {
#pragma unroll
  for (int d = 1; d < OCT; d <<= 1) x = fmin(x, __shfl_xor_sync(FULL, x, d, OCT));
  return x;
}
// sum over lanes 0..6 in ASCENDING lane order (canonical reduction order of the oracle);
// every lane of the octet receives the result.
__device__ __forceinline__ double oct_sum_ordered(double x) {
  double s = oct_bcast(x, 0);
#pragma unroll
  for (int l = 1; l < NV; ++l) s += oct_bcast(x, l);
  return s;
}

}  // namespace idocp_b200
