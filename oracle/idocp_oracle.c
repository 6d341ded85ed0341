/*
 * idocp_oracle.c -- CPU ORACLE (TEST INFRASTRUCTURE, NOT THE PRODUCT).  See idocp_oracle.h.
 *
 * Restates, in plain C and in the reference's own operation order, the per-iteration Newton
 * step of idocp's UnOCPSolver for the iiwa14 (SURVEY.md Appendix A).  File:line citations point
 * into the reference tree.  PARITY UNPINNED at the pinocchio boundary (see header).
 *
 * Canonical reduction order (SURVEY.md A.7): every sum / dot product runs over ascending index,
 * left to right; Eigen's vectorised reductions are not reproducible elsewhere, so this file
 * DEFINES the order and the CUDA kernels follow it.
 */
#include "idocp_oracle.h"
#include "model_iiwa14.h"
#include "canon_pivot.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define NV ORACLE_NV
#define NC 8               /* six components of JointConstraintsFactory + the two acceleration limits */
#define NN (NV * NV)

/* ------------------------------------------------------------------------------------------ */
/* small helpers                                                                               */
/* ------------------------------------------------------------------------------------------ */
/* CANONICAL ARITHMETIC (shared convention with idocp_b200/csrc/octet.cuh): this file is compiled
 * with -ffp-contract=off, every fused multiply-add is an explicit fma(), and the helpers below use
 * the same operation trees as their CUDA twins, so that the GPU results can be compared bit for bit. */
typedef struct { double x, y, z; } v3_t;
typedef struct { double xx, xy, xz, yy, yz, zz; } s3_t;
static inline v3_t V3(double x, double y, double z) { v3_t r = {x, y, z}; return r; }
static inline v3_t vadd(v3_t a, v3_t b) { return V3(a.x + b.x, a.y + b.y, a.z + b.z); }
static inline v3_t vsub(v3_t a, v3_t b) { return V3(a.x - b.x, a.y - b.y, a.z - b.z); }
static inline v3_t vscale(double s, v3_t a) { return V3(s * a.x, s * a.y, s * a.z); }
static inline v3_t vfma(double s, v3_t a, v3_t b) { return V3(fma(s, a.x, b.x), fma(s, a.y, b.y), fma(s, a.z, b.z)); }
static inline v3_t vcross(v3_t a, v3_t b) {
  return V3(fma(a.y, b.z, -(a.z * b.y)), fma(a.z, b.x, -(a.x * b.z)), fma(a.x, b.y, -(a.y * b.x)));
}
static inline double vdot(v3_t a, v3_t b) { return fma(a.z, b.z, fma(a.y, b.y, a.x * b.x)); }
static inline v3_t smul(s3_t A, v3_t b) {
  return V3(fma(A.xz, b.z, fma(A.xy, b.y, A.xx * b.x)), fma(A.yz, b.z, fma(A.yy, b.y, A.xy * b.x)),
            fma(A.zz, b.z, fma(A.yz, b.y, A.xz * b.x)));
}
/* sin / cos: Cody-Waite reduction by pi/2 + degree-13/14 minimax kernels (twin of canon_sincos) */
static inline void canon_sincos(double x, double* sn, double* cs) {
  const double k = rint(x * 6.36619772367581382433e-01);
  double r = fma(-k, 1.57079632673412561417e+00, x);
  r = fma(-k, 6.07710050650619224932e-11, r);
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
  const int q = (int)((long long)k & 3);   /* exact for every |k| < 2^53 (an int overflows past 2^31) */
  *sn = (q == 0) ? s : (q == 1) ? c : (q == 2) ? -s : -c;
  *cs = (q == 0) ? c : (q == 1) ? -s : (q == 2) ? -c : s;
}
void oracle_canon_sincos(double x, double* sn, double* cs) { canon_sincos(x, sn, cs); }
/* natural logarithm (twin of canon_log in octet.cuh): subnormals scaled by 2^54 first; 0, negatives, NaN and +inf
 * as std::log */
static inline double canon_log(double x) {
  int k = 0;
  if (!(x >= 2.2250738585072014e-308)) {   /* not a positive normal: 0, subnormal, negative or NaN */
    if (x == 0.0) return -INFINITY;
    if (!(x > 0.0)) return (x != x) ? x : NAN;
    x *= 18014398509481984.0;              /* 2^54 */
    k = -54;
  } else if (!(x < INFINITY)) {
    return x;                              /* log(+inf) = +inf */
  }
  long long bits;
  memcpy(&bits, &x, sizeof(bits));
  int hx = (int)(bits >> 32);
  k += (hx >> 20) - 1023;
  hx &= 0x000fffff;
  const int i = (hx + 0x95f64) & 0x100000;
  k += (i >> 20);
  const long long nb = ((long long)(hx | (i ^ 0x3ff00000)) << 32) | (bits & 0xffffffffLL);
  double m;
  memcpy(&m, &nb, sizeof(m));
  const double f = m - 1.0;
  const double s = f / (2.0 + f);
  const double dk = (double)k;
  const double z = s * s;
  const double w = z * z;
  const double t1 = w * (3.999999999940941908e-01 + w * (2.222219843214978396e-01 + w * 1.531383769920937332e-01));
  const double t2 = z * (6.666666666666735130e-01 +
                         w * (2.857142874366239149e-01 + w * (1.818357216161805012e-01 + w * 1.479819860511658591e-01)));
  const double R = t2 + t1;
  const double hfsq = 0.5 * f * f;
  return dk * 6.93147180369123816490e-01 - ((hfsq - (s * (hfsq + R) + dk * 1.90821492927058770002e-10)) - f);
}
double oracle_canon_log(double x) { return canon_log(x); }

/* plain (non-canonical) helpers of the independent body-frame RNEA below */
static inline void cross3(const double* a, const double* b, double* c) {
  c[0] = a[1] * b[2] - a[2] * b[1];
  c[1] = a[2] * b[0] - a[0] * b[2];
  c[2] = a[0] * b[1] - a[1] * b[0];
}
/* y = A x for a symmetric 3x3 stored (xx,xy,xz,yy,yz,zz) */
static inline void sym3_mul(const double* A, const double* x, double* y) {
  y[0] = A[0] * x[0] + A[1] * x[1] + A[2] * x[2];
  y[1] = A[1] * x[0] + A[3] * x[1] + A[4] * x[2];
  y[2] = A[2] * x[0] + A[4] * x[1] + A[5] * x[2];
}

double oracle_splitmix_uniform(unsigned long long seed, unsigned long long index) {
  unsigned long long z = seed + (index + 1ULL) * 0x9E3779B97F4A7C15ULL;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  z = z ^ (z >> 31);
  return (double)(z >> 11) * (1.0 / 9007199254740992.0); /* [0,1) */
}

/* ------------------------------------------------------------------------------------------ */
/* robot/: RNEA and its analytical derivatives                                                 */
/* ------------------------------------------------------------------------------------------ */

/* Robot::RNEA -> pinocchio::rnea (include/idocp/robot/robot.hxx:444-460).
 * Featherstone's recursive Newton-Euler in body frames, [linear; angular] spatial vectors,
 * gravity folded into the base acceleration a_0 = (0,0,+9.81). */
void oracle_rnea(const double* q, const double* v, const double* a, double* tau) {
  double vl[NV][3], vw[NV][3], fl[NV][3], fw[NV][3], R[NV][9];
  double al_p[3] = {0.0, 0.0, IIWA14_GRAVITY}, aw_p[3] = {0, 0, 0}, vl_p[3] = {0, 0, 0}, vw_p[3] = {0, 0, 0};
  for (int i = 0; i < NV; ++i) {
    const double c = cos(q[i]), s = sin(q[i]);
    const double* P = IIWA14_PLACEMENT_R[i];
    const double* pp = IIWA14_PLACEMENT_P[i];
    /* liMi rotation = placement * Rz(q) (row-major, child -> parent) */
    double* Ri = R[i];
    for (int r = 0; r < 3; ++r) {
      Ri[3 * r + 0] = c * P[3 * r + 0] + s * P[3 * r + 1];
      Ri[3 * r + 1] = -s * P[3 * r + 0] + c * P[3 * r + 1];
      Ri[3 * r + 2] = P[3 * r + 2];
    }
    /* actInv of the parent's motion: lin = R^T (v - p x w), ang = R^T w */
    double t[3], u[3], vli[3], vwi[3], ali[3], awi[3];
    cross3(pp, vw_p, t);
    for (int k = 0; k < 3; ++k) u[k] = vl_p[k] - t[k];
    for (int k = 0; k < 3; ++k) {
      vli[k] = Ri[k] * u[0] + Ri[3 + k] * u[1] + Ri[6 + k] * u[2];
      vwi[k] = Ri[k] * vw_p[0] + Ri[3 + k] * vw_p[1] + Ri[6 + k] * vw_p[2];
    }
    cross3(pp, aw_p, t);
    for (int k = 0; k < 3; ++k) u[k] = al_p[k] - t[k];
    for (int k = 0; k < 3; ++k) {
      ali[k] = Ri[k] * u[0] + Ri[3 + k] * u[1] + Ri[6 + k] * u[2];
      awi[k] = Ri[k] * aw_p[0] + Ri[3 + k] * aw_p[1] + Ri[6 + k] * aw_p[2];
    }
    /* v_i = S qd + ..., a_i = S qdd + v_i x (S qd) + ...   with S = (0,0,0, 0,0,1) */
    vwi[2] += v[i];
    /* v x (S qd): lin = v_l x (z qd), ang = w x (z qd) */
    ali[0] += vli[1] * v[i];
    ali[1] += -vli[0] * v[i];
    awi[0] += vwi[1] * v[i];
    awi[1] += -vwi[0] * v[i];
    awi[2] += a[i];
    /* f = Y a + v x* (Y v), Y = (m, c, Ic):  Y x = ( m (xl + xw x c) ; Ic xw + c x lin ) */
    const double m = IIWA14_MASS[i];
    const double* cm = IIWA14_COM[i];
    const double* Ic = IIWA14_INERTIA[i];
    double hl[3], hw[3], gl[3], gw[3], tmp[3];
    cross3(vwi, cm, tmp);
    for (int k = 0; k < 3; ++k) hl[k] = m * (vli[k] + tmp[k]);
    sym3_mul(Ic, vwi, hw);
    cross3(cm, hl, tmp);
    for (int k = 0; k < 3; ++k) hw[k] += tmp[k];
    cross3(awi, cm, tmp);
    for (int k = 0; k < 3; ++k) gl[k] = m * (ali[k] + tmp[k]);
    sym3_mul(Ic, awi, gw);
    cross3(cm, gl, tmp);
    for (int k = 0; k < 3; ++k) gw[k] += tmp[k];
    /* v x* h = (w x hl ; w x hw + vl x hl) */
    double c1[3], c2[3], c3[3];
    cross3(vwi, hl, c1);
    cross3(vwi, hw, c2);
    cross3(vli, hl, c3);
    for (int k = 0; k < 3; ++k) {
      fl[i][k] = gl[k] + c1[k];
      fw[i][k] = gw[k] + c2[k] + c3[k];
      vl[i][k] = vli[k]; vw[i][k] = vwi[k];
      vl_p[k] = vli[k]; vw_p[k] = vwi[k]; al_p[k] = ali[k]; aw_p[k] = awi[k];
    }
  }
  for (int i = NV - 1; i >= 0; --i) {
    tau[i] = fw[i][2];
    if (i > 0) {
      /* f_parent += liMi.act(f): lin = R f, ang = R n + p x (R f) */
      const double* Ri = R[i];
      const double* pp = IIWA14_PLACEMENT_P[i];
      double l[3], n[3], t[3];
      for (int r = 0; r < 3; ++r) {
        l[r] = Ri[3 * r] * fl[i][0] + Ri[3 * r + 1] * fl[i][1] + Ri[3 * r + 2] * fl[i][2];
        n[r] = Ri[3 * r] * fw[i][0] + Ri[3 * r + 1] * fw[i][1] + Ri[3 * r + 2] * fw[i][2];
      }
      cross3(pp, l, t);
      for (int k = 0; k < 3; ++k) { fl[i - 1][k] += l[k]; fw[i - 1][k] += n[k] + t[k]; }
    }
  }
  (void)vl; (void)vw;
}

/* per-joint world-frame quantities of the derivative algorithm */
typedef struct {
  v3_t Sl, Sw, dSl, dSw, Bl, Bw;
  v3_t Ul, Uw, Ww, Gl, Gw, Hl, Hw;
  double tau;
} joint_world_t;

#define LANES 8 /* the GPU works on octets: 7 joints + one zero-mass padding lane */

/* Hillis-Steele inclusive scans over the 8 lanes, in the exact tree order of the GPU shuffles
 * (octet.cuh: oct_prefix_sum / oct_suffix_sum) */
static void prefix_sum8(double* x) {
  for (int d = 1; d < LANES; d <<= 1) {
    double y[LANES];
    for (int l = 0; l < LANES; ++l) y[l] = x[l >= d ? l - d : l];
    for (int l = 0; l < LANES; ++l) if (l >= d) x[l] += y[l];
  }
}
static void suffix_sum8(double* x) {
  for (int d = 1; d < LANES; d <<= 1) {
    double y[LANES];
    for (int l = 0; l < LANES; ++l) y[l] = x[l + d < LANES ? l + d : l];
    for (int l = 0; l < LANES; ++l) if (l + d < LANES) x[l] += y[l];
  }
}
static void prefix_sum8_v(v3_t* v) {
  double a[LANES], b[LANES], c[LANES];
  for (int l = 0; l < LANES; ++l) { a[l] = v[l].x; b[l] = v[l].y; c[l] = v[l].z; }
  prefix_sum8(a); prefix_sum8(b); prefix_sum8(c);
  for (int l = 0; l < LANES; ++l) v[l] = V3(a[l], b[l], c[l]);
}
static void suffix_sum8_v(v3_t* v) {
  double a[LANES], b[LANES], c[LANES];
  for (int l = 0; l < LANES; ++l) { a[l] = v[l].x; b[l] = v[l].y; c[l] = v[l].z; }
  suffix_sum8(a); suffix_sum8(b); suffix_sum8(c);
  for (int l = 0; l < LANES; ++l) v[l] = V3(a[l], b[l], c[l]);
}

/* world placements of the 7 joint frames (+ the zero-mass pad lane): local transform placement * Rz(q),
 * then the inclusive prefix product X_l <- X_0 ... X_l in the GPU's Hillis-Steele tree order
 * (chain_dynamics.cuh: chain_fk).  R row-major (joint -> world), p = origin of the joint frame. */
static void chain_fk(const double* q, double R[LANES][9], v3_t* p) {
  /* local transforms: placement * Rz(q) */
  for (int l = 0; l < LANES; ++l) {
    if (l < NV) {
      double sn, cs;
      canon_sincos(q[l], &sn, &cs);
      const double* P = IIWA14_PLACEMENT_R[l];
      for (int r = 0; r < 3; ++r) {
        const double a0 = P[3 * r], a1 = P[3 * r + 1];
        R[l][3 * r + 0] = fma(sn, a1, cs * a0);
        R[l][3 * r + 1] = fma(cs, a1, -(sn * a0));
        R[l][3 * r + 2] = P[3 * r + 2];
      }
      p[l] = V3(IIWA14_PLACEMENT_P[l][0], IIWA14_PLACEMENT_P[l][1], IIWA14_PLACEMENT_P[l][2]);
    } else {
      for (int k = 0; k < 9; ++k) R[l][k] = (k % 4 == 0) ? 1.0 : 0.0;
      p[l] = V3(0, 0, 0);
    }
  }
  /* inclusive prefix product X_l <- X_0 ... X_l */
  for (int d = 1; d < LANES; d <<= 1) {
    double Rs[LANES][9];
    v3_t ps[LANES];
    for (int l = 0; l < LANES; ++l) {
      const int src = l >= d ? l - d : l;
      memcpy(Rs[l], R[src], sizeof(Rs[l]));
      ps[l] = p[src];
    }
    for (int l = d; l < LANES; ++l) {
      const double* S = Rs[l];
      const v3_t pl = p[l];
      p[l] = V3(fma(S[2], pl.z, fma(S[1], pl.y, fma(S[0], pl.x, ps[l].x))),
                fma(S[5], pl.z, fma(S[4], pl.y, fma(S[3], pl.x, ps[l].y))),
                fma(S[8], pl.z, fma(S[7], pl.y, fma(S[6], pl.x, ps[l].z))));
      double Rn[9];
      for (int r = 0; r < 3; ++r)
        for (int k = 0; k < 3; ++k)
          Rn[3 * r + k] = fma(S[3 * r + 2], R[l][6 + k], fma(S[3 * r + 1], R[l][3 + k], S[3 * r] * R[l][k]));
      memcpy(R[l], Rn, sizeof(Rn));
    }
  }
}

/* Robot::RNEADerivatives -> pinocchio::computeRNEADerivatives + lower-triangle mirror of dtau/da
 * (include/idocp/robot/robot.hxx:466-500).  Analytical derivatives of Carpentier & Mansard
 * (RSS 2018) in the WORLD frame; the composite matrices are kept in their structured form
 *   I^C = (m, mc, Ibar)   [10 numbers],   D^C m = (-2 hl x m_w ; Sym m_w - ha x m_w)   [12 numbers]
 * (derivation: DESIGN.md "RNEA derivatives"; mirrored in oracle/np_mirror.py).
 * The chain recursions are evaluated as tree-ordered scans over 8 "lanes" (7 joints + a zero-mass
 * pad) so that the operation order equals the GPU kernel's (chain_dynamics.cuh).
 * Also returns tau = rnea(q,v,a) when tau != NULL. */
static void rnea_derivatives_impl(const double* q, const double* v, const double* a, double* tau,
                                  double* dq, double* dv, double* da) {
  joint_world_t J[LANES];
  double R[LANES][9];
  v3_t p[LANES];
  chain_fk(q, R, p);
  v3_t vw[LANES], vl[LANES], aw[LANES], al[LANES];
  double qd[LANES], qdd[LANES];
  for (int l = 0; l < LANES; ++l) {
    qd[l] = l < NV ? v[l] : 0.0;
    qdd[l] = l < NV ? a[l] : 0.0;
    J[l].Sw = V3(R[l][2], R[l][5], R[l][8]);
    J[l].Sl = vcross(p[l], J[l].Sw);
    vw[l] = vscale(qd[l], J[l].Sw);
    vl[l] = vscale(qd[l], J[l].Sl);
  }
  prefix_sum8_v(vw); prefix_sum8_v(vl);
  for (int l = 0; l < LANES; ++l) {
    J[l].dSl = vadd(vcross(vw[l], J[l].Sl), vcross(vl[l], J[l].Sw));
    J[l].dSw = vcross(vw[l], J[l].Sw);
    aw[l] = vfma(qd[l], J[l].dSw, vscale(qdd[l], J[l].Sw));
    al[l] = vfma(qd[l], J[l].dSl, vscale(qdd[l], J[l].Sl));
  }
  prefix_sum8_v(aw); prefix_sum8_v(al);
  double mS[LANES];
  v3_t mc[LANES], hl[LANES], ha[LANES], fl[LANES], fa[LANES];
  s3_t Ib[LANES], Sym[LANES];
  for (int l = 0; l < LANES; ++l) {
    joint_world_t* j = &J[l];
    al[l].z += IIWA14_GRAVITY;
    j->Bl = vadd(vadd(vadd(vcross(aw[l], j->Sl), vcross(al[l], j->Sw)), vcross(vw[l], j->dSl)), vcross(vl[l], j->dSw));
    j->Bw = vadd(vcross(aw[l], j->Sw), vcross(vw[l], j->dSw));
    const double m = l < NV ? IIWA14_MASS[l] : 0.0;
    const v3_t cm = l < NV ? V3(IIWA14_COM[l][0], IIWA14_COM[l][1], IIWA14_COM[l][2]) : V3(0, 0, 0);
    const double* Rl = R[l];
    const v3_t cw = V3(fma(Rl[2], cm.z, fma(Rl[1], cm.y, fma(Rl[0], cm.x, p[l].x))),
                       fma(Rl[5], cm.z, fma(Rl[4], cm.y, fma(Rl[3], cm.x, p[l].y))),
                       fma(Rl[8], cm.z, fma(Rl[7], cm.y, fma(Rl[6], cm.x, p[l].z))));
    mS[l] = m;
    mc[l] = vscale(m, cw);
    double i0 = 0, i1 = 0, i2 = 0, i3 = 0, i4 = 0, i5 = 0;
    if (l < NV) {
      i0 = IIWA14_INERTIA[l][0]; i1 = IIWA14_INERTIA[l][1]; i2 = IIWA14_INERTIA[l][2];
      i3 = IIWA14_INERTIA[l][3]; i4 = IIWA14_INERTIA[l][4]; i5 = IIWA14_INERTIA[l][5];
    }
    double RI[9];
    for (int r = 0; r < 3; ++r) {
      const double r0 = Rl[3 * r], r1 = Rl[3 * r + 1], r2 = Rl[3 * r + 2];
      RI[3 * r + 0] = fma(r2, i2, fma(r1, i1, r0 * i0));
      RI[3 * r + 1] = fma(r2, i4, fma(r1, i3, r0 * i1));
      RI[3 * r + 2] = fma(r2, i5, fma(r1, i4, r0 * i2));
    }
    const double cc = vdot(cw, cw);
    Ib[l].xx = fma(m, cc - cw.x * cw.x, fma(RI[2], Rl[2], fma(RI[1], Rl[1], RI[0] * Rl[0])));
    Ib[l].xy = fma(m, -(cw.x * cw.y), fma(RI[2], Rl[5], fma(RI[1], Rl[4], RI[0] * Rl[3])));
    Ib[l].xz = fma(m, -(cw.x * cw.z), fma(RI[2], Rl[8], fma(RI[1], Rl[7], RI[0] * Rl[6])));
    Ib[l].yy = fma(m, cc - cw.y * cw.y, fma(RI[5], Rl[5], fma(RI[4], Rl[4], RI[3] * Rl[3])));
    Ib[l].yz = fma(m, -(cw.y * cw.z), fma(RI[5], Rl[8], fma(RI[4], Rl[7], RI[3] * Rl[6])));
    Ib[l].zz = fma(m, cc - cw.z * cw.z, fma(RI[8], Rl[8], fma(RI[7], Rl[7], RI[6] * Rl[6])));
    hl[l] = vfma(m, vl[l], vcross(vw[l], mc[l]));
    ha[l] = vadd(vcross(mc[l], vl[l]), smul(Ib[l], vw[l]));
    fl[l] = vadd(vfma(m, al[l], vcross(aw[l], mc[l])), vcross(vw[l], hl[l]));
    fa[l] = vadd(vadd(vadd(vcross(mc[l], al[l]), smul(Ib[l], aw[l])), vcross(vw[l], ha[l])), vcross(vl[l], hl[l]));
    const v3_t c0 = vcross(vw[l], V3(Ib[l].xx, Ib[l].xy, Ib[l].xz));
    const v3_t c1 = vcross(vw[l], V3(Ib[l].xy, Ib[l].yy, Ib[l].yz));
    const v3_t c2 = vcross(vw[l], V3(Ib[l].xz, Ib[l].yz, Ib[l].zz));
    const double mcv = vdot(mc[l], vl[l]);
    const v3_t vL = vl[l], mC_ = mc[l];
    Sym[l].xx = 2.0 * (c0.x + (mcv - vL.x * mC_.x));
    Sym[l].xy = (c1.x + c0.y) - fma(vL.x, mC_.y, mC_.x * vL.y);
    Sym[l].xz = (c2.x + c0.z) - fma(vL.x, mC_.z, mC_.x * vL.z);
    Sym[l].yy = 2.0 * (c1.y + (mcv - vL.y * mC_.y));
    Sym[l].yz = (c2.y + c1.z) - fma(vL.y, mC_.z, mC_.y * vL.z);
    Sym[l].zz = 2.0 * (c2.z + (mcv - vL.z * mC_.z));
  }
  /* composite (suffix) sums */
  suffix_sum8(mS);
  suffix_sum8_v(mc); suffix_sum8_v(hl); suffix_sum8_v(ha); suffix_sum8_v(fl); suffix_sum8_v(fa);
  {
    double t[6][LANES], u[6][LANES];
    for (int l = 0; l < LANES; ++l) {
      t[0][l] = Ib[l].xx; t[1][l] = Ib[l].xy; t[2][l] = Ib[l].xz; t[3][l] = Ib[l].yy; t[4][l] = Ib[l].yz; t[5][l] = Ib[l].zz;
      u[0][l] = Sym[l].xx; u[1][l] = Sym[l].xy; u[2][l] = Sym[l].xz; u[3][l] = Sym[l].yy; u[4][l] = Sym[l].yz; u[5][l] = Sym[l].zz;
    }
    for (int k = 0; k < 6; ++k) { suffix_sum8(t[k]); suffix_sum8(u[k]); }
    for (int l = 0; l < LANES; ++l) {
      Ib[l].xx = t[0][l]; Ib[l].xy = t[1][l]; Ib[l].xz = t[2][l]; Ib[l].yy = t[3][l]; Ib[l].yz = t[4][l]; Ib[l].zz = t[5][l];
      Sym[l].xx = u[0][l]; Sym[l].xy = u[1][l]; Sym[l].xz = u[2][l]; Sym[l].yy = u[3][l]; Sym[l].yz = u[4][l]; Sym[l].zz = u[5][l];
    }
  }
  for (int l = 0; l < NV; ++l) {
    joint_world_t* j = &J[l];
    const double mC = mS[l];
    j->tau = vdot(j->Sl, fl[l]) + vdot(j->Sw, fa[l]);
    if (tau) tau[l] = j->tau;
    j->Ul = vfma(mC, j->Sl, vcross(j->Sw, mc[l]));
    j->Uw = vadd(vcross(mc[l], j->Sl), smul(Ib[l], j->Sw));
    j->Ww = vadd(vfma(2.0, vcross(hl[l], j->Sl), smul(Sym[l], j->Sw)), vcross(ha[l], j->Sw));
    j->Gl = vfma(-2.0, vcross(hl[l], j->dSw), vadd(vfma(mC, j->Bl, vcross(j->Sw, fl[l])), vcross(j->Bw, mc[l])));
    j->Gw = vsub(vadd(vadd(vadd(vadd(vcross(j->Sw, fa[l]), vcross(j->Sl, fl[l])), vcross(mc[l], j->Bl)), smul(Ib[l], j->Bw)),
                      smul(Sym[l], j->dSw)),
                 vcross(ha[l], j->dSw));
    j->Hl = vscale(2.0, vsub(vfma(mC, j->dSl, vcross(j->dSw, mc[l])), vcross(hl[l], j->Sw)));
    j->Hw = vfma(2.0, vadd(vcross(mc[l], j->dSl), smul(Ib[l], j->dSw)), vsub(smul(Sym[l], j->Sw), vcross(ha[l], j->Sw)));
  }
  if (!dq) return;
  for (int c = 0; c < NV; ++c) {
    const joint_world_t* b = &J[c];
    for (int r = 0; r < NV; ++r) {
      const joint_world_t* x = &J[r];
      if (r <= c) {
        dq[c * NV + r] = vdot(x->Sl, b->Gl) + vdot(x->Sw, b->Gw);
        dv[c * NV + r] = vdot(x->Sl, b->Hl) + vdot(x->Sw, b->Hw);
        da[c * NV + r] = vdot(x->Sl, b->Ul) + vdot(x->Sw, b->Uw);
      } else {
        dq[c * NV + r] = (vdot(x->Ul, b->Bl) + vdot(x->Uw, b->Bw)) + vdot(x->Ww, b->dSw);
        dv[c * NV + r] = fma(2.0, vdot(x->Ul, b->dSl) + vdot(x->Uw, b->dSw), vdot(x->Ww, b->Sw));
        /* robot.hxx:496-499: strictly-lower triangle of dtau/da mirrored from the upper one:
         * M[r][c] = M[c][r] = S_c . U_r */
        da[c * NV + r] = vdot(b->Sl, x->Ul) + vdot(b->Sw, x->Uw);
      }
    }
  }
}

void oracle_rnea_derivatives(const double* q, const double* v, const double* a,
                             double* dq, double* dv, double* da) {
  rnea_derivatives_impl(q, v, a, NULL, dq, dv, da);
}


/* ------------------------------------------------------------------------------------------ */
/* cost/ : TimeVaryingTaskSpace6DCost (src/cost/time_varying_task_space_6d_cost.cpp:68-195)    */
/* on the end-effector frame.  pinocchio pieces restated from their published algorithms       */
/* (pinocchio is absent): framePlacement / getFrameJacobian(LOCAL) (robot.hxx:186,193-203),    */
/* log6 / Jlog6 / log3 / Jlog3 (pinocchio/spatial/log.hxx).  PARITY UNPINNED like the rest.    */
/* ------------------------------------------------------------------------------------------ */
/* acos on [-1, 1]: the fdlibm e_acos.c algorithm with plain IEEE operations (twin of canon_acos in
 * octet.cuh) */
static inline double canon_acos(double x) {
  const double pio2_hi = 1.57079632679489655800e+00, pio2_lo = 6.12323399573676603587e-17;
  const double pi = 3.14159265358979311600e+00;
  const double pS0 = 1.66666666666666657415e-01, pS1 = -3.25565818622400915405e-01, pS2 = 2.01212532134862925881e-01,
               pS3 = -4.00555345006794114027e-02, pS4 = 7.91534994289814532176e-04, pS5 = 3.47933107596021167570e-05;
  const double qS1 = -2.40339491173441421878e+00, qS2 = 2.02094576023350569471e+00, qS3 = -6.88283971605453293030e-01,
               qS4 = 7.70381505559019352791e-02;
  if (!(x > -1.0)) return (x != x) ? x : pi;   /* x <= -1 gives pi, NaN gives NaN */
  if (!(x < 1.0)) return 0.0;
  const double ax = fabs(x);
  if (ax < 0.5) {
    const double z = x * x;
    const double pp = z * (pS0 + z * (pS1 + z * (pS2 + z * (pS3 + z * (pS4 + z * pS5)))));
    const double qq = 1.0 + z * (qS1 + z * (qS2 + z * (qS3 + z * qS4)));
    const double r = pp / qq;
    return pio2_hi - (x - (pio2_lo - x * r));
  }
  if (x < 0.0) {
    const double z = (1.0 + x) * 0.5;
    const double pp = z * (pS0 + z * (pS1 + z * (pS2 + z * (pS3 + z * (pS4 + z * pS5)))));
    const double qq = 1.0 + z * (qS1 + z * (qS2 + z * (qS3 + z * qS4)));
    const double sq = sqrt(z);
    const double r = pp / qq;
    const double w = r * sq - pio2_lo;
    return pi - 2.0 * (sq + w);
  }
  {
    const double z = (1.0 - x) * 0.5;
    const double sq = sqrt(z);
    long long bits;
    memcpy(&bits, &sq, sizeof(bits));
    bits &= (long long)0xffffffff00000000ULL;   /* df = sq with the low word cleared */
    double df;
    memcpy(&df, &bits, sizeof(df));
    const double c = (z - df * df) / (sq + df);
    const double pp = z * (pS0 + z * (pS1 + z * (pS2 + z * (pS3 + z * (pS4 + z * pS5)))));
    const double qq = 1.0 + z * (qS1 + z * (qS2 + z * (qS3 + z * qS4)));
    const double r = pp / qq;
    const double w = r * sq + c;
    return 2.0 * (df + w);
  }
}
double oracle_canon_acos(double x) { return canon_acos(x); }

#define TASK_TAYLOR 1.220703125e-04   /* TaylorSeriesExpansion<double>::precision<3>() = eps^(1/4) = 2^-13 */
#define TASK_PI 3.14159265358979311600e+00

static inline double dot3r(const double* row, v3_t x) { return fma(row[2], x.z, fma(row[1], x.y, row[0] * x.x)); }
/* y = M^T x for a row-major 3x3 */
static inline v3_t mulT3(const double* M, v3_t x) {
  return V3(fma(M[6], x.z, fma(M[3], x.y, M[0] * x.x)), fma(M[7], x.z, fma(M[4], x.y, M[1] * x.x)),
            fma(M[8], x.z, fma(M[5], x.y, M[2] * x.x)));
}
/* M += skew(v) */
static inline void add_skew(v3_t v, double* M) {
  M[1] -= v.z; M[2] += v.y; M[3] += v.z; M[5] -= v.x; M[6] -= v.y; M[7] += v.x;
}

/* pinocchio::log3(R, theta) */
static v3_t log3_canon(const double* R, double* theta_out) {
  const double tr = (R[0] + R[4]) + R[8];
  double theta;
  if (tr > 3.0) theta = 0.0;
  else if (tr < -1.0) theta = TASK_PI;
  else theta = canon_acos((tr - 1.0) * 0.5);
  *theta_out = theta;
  if (theta >= TASK_PI - 1e-2) {
    double sn, cphi;
    canon_sincos(theta - TASK_PI, &sn, &cphi);
    const double beta = (theta * theta) / (1.0 + cphi);
    const double t0 = (R[0] + cphi) * beta, t1 = (R[4] + cphi) * beta, t2 = (R[8] + cphi) * beta;
    return V3((R[7] > R[5] ? 1.0 : -1.0) * (t0 > 0.0 ? sqrt(t0) : 0.0),
              (R[2] > R[6] ? 1.0 : -1.0) * (t1 > 0.0 ? sqrt(t1) : 0.0),
              (R[3] > R[1] ? 1.0 : -1.0) * (t2 > 0.0 ? sqrt(t2) : 0.0));
  }
  double t = 1.0;
  if (theta > TASK_TAYLOR) {
    double sn, cs;
    canon_sincos(theta, &sn, &cs);
    t = theta / sn;
  }
  t *= 0.5;
  return V3(t * (R[7] - R[5]), t * (R[2] - R[6]), t * (R[3] - R[1]));
}

/* pinocchio::Jlog3(theta, log, Jlog) */
static void jlog3_canon(double theta, v3_t w, double* A) {
  double alpha, diag;
  if (theta < TASK_TAYLOR) {
    alpha = 1.0 / 12.0 + (theta * theta) / 720.0;
    diag = 0.5 * (2.0 - (theta * theta) / 6.0);
  } else {
    double st, ct;
    canon_sincos(theta, &st, &ct);
    const double st_1mct = st / (1.0 - ct);
    alpha = 1.0 / (theta * theta) - st_1mct / (2.0 * theta);
    diag = 0.5 * (theta * st_1mct);
  }
  const v3_t aw = vscale(alpha, w);
  const double wv[3] = {w.x, w.y, w.z}, av[3] = {aw.x, aw.y, aw.z};
  for (int r = 0; r < 3; ++r)
    for (int k = 0; k < 3; ++k) A[3 * r + k] = av[r] * wv[k];
  A[0] += diag; A[4] += diag; A[8] += diag;
  add_skew(vscale(0.5, w), A);
}

typedef struct {
  double diff[6];        /* log6(SE3_ref^-1 * oMf) = [linear; angular] */
  double JJ[6 * NV];     /* Jlog6 * frame Jacobian (LOCAL), JJ[c * 6 + k] = row k of column c */
  int kind;              /* 1: 6D cost; 2: TaskSpace3DCost (diff_3d / J_3d in the first three entries, the rest zero) */
} task_eval_t;

/* diff_6d and JJ_6d of computeStageCostDerivatives (:105-119).  ref12 = [R_ref row-major (9), p_ref (3)]
 * as produced by the user's TimeVaryingTaskSpace6DRefBase::compute_q_6d_ref(t) (sampled on the host). */
static void task_evaluate(const double* q, const double* ref12, task_eval_t* te, int with_jacobian, int kind) {
  te->kind = kind;
  double R[LANES][9];
  v3_t p[LANES];
  chain_fk(q, R, p);
  /* robot.framePlacement(frame_id): oMf = oMi[parent joint] * frame placement */
  const double* R6 = R[IIWA14_EE_PARENT_JOINT];
  const double* E = IIWA14_EE_PLACEMENT_R;
  double Rf[9];
  for (int r = 0; r < 3; ++r)
    for (int k = 0; k < 3; ++k)
      Rf[3 * r + k] = fma(R6[3 * r + 2], E[6 + k], fma(R6[3 * r + 1], E[3 + k], R6[3 * r] * E[k]));
  const v3_t ep = V3(IIWA14_EE_PLACEMENT_P[0], IIWA14_EE_PLACEMENT_P[1], IIWA14_EE_PLACEMENT_P[2]);
  const v3_t p6 = p[IIWA14_EE_PARENT_JOINT];
  const v3_t pf = V3(fma(R6[2], ep.z, fma(R6[1], ep.y, fma(R6[0], ep.x, p6.x))),
                     fma(R6[5], ep.z, fma(R6[4], ep.y, fma(R6[3], ep.x, p6.y))),
                     fma(R6[8], ep.z, fma(R6[7], ep.y, fma(R6[6], ep.x, p6.z))));
  if (kind == 2) {
    /* TaskSpace3DCost / TimeVaryingTaskSpace3DCost (src/cost/task_space_3d_cost.cpp:56-140): diff_3d = framePosition -
     * q_3d_ref; J_3d = frameRotation * getFrameJacobian(LOCAL).topRows<3>() */
    te->diff[0] = pf.x - ref12[9]; te->diff[1] = pf.y - ref12[10]; te->diff[2] = pf.z - ref12[11];
    te->diff[3] = te->diff[4] = te->diff[5] = 0.0;
    if (!with_jacobian) return;
    for (int c = 0; c < NV; ++c) {
      const v3_t Sw = V3(R[c][2], R[c][5], R[c][8]);
      const v3_t Jl = mulT3(Rf, vadd(vcross(p[c], Sw), vcross(Sw, pf)));
      for (int r = 0; r < 3; ++r) {
        te->JJ[c * 6 + r] = dot3r(Rf + 3 * r, Jl);
        te->JJ[c * 6 + 3 + r] = 0.0;
      }
    }
    return;
  }
  /* diff_SE3 = SE3_ref^-1 * oMf */
  double Rd[9];
  for (int r = 0; r < 3; ++r)
    for (int k = 0; k < 3; ++k)
      Rd[3 * r + k] = fma(ref12[6 + r], Rf[6 + k], fma(ref12[3 + r], Rf[3 + k], ref12[r] * Rf[k]));
  const v3_t pd = mulT3(ref12, vsub(pf, V3(ref12[9], ref12[10], ref12[11])));
  /* pinocchio::log6 */
  double theta;
  const v3_t w = log3_canon(Rd, &theta);
  const double t2 = theta * theta;
  double st = 0.0, ct = 1.0;
  if (!(theta < TASK_TAYLOR)) canon_sincos(theta, &st, &ct);
  {
    double alpha, beta;
    if (theta < TASK_TAYLOR) {
      alpha = (1.0 - t2 / 12.0) - (t2 * t2) / 720.0;
      beta = 1.0 / 12.0 + t2 / 720.0;
    } else {
      alpha = (theta * st) / (2.0 * (1.0 - ct));
      beta = 1.0 / t2 - st / ((2.0 * theta) * (1.0 - ct));
    }
    const v3_t v = vfma(beta * vdot(w, pd), w, vfma(-0.5, vcross(w, pd), vscale(alpha, pd)));
    te->diff[0] = v.x; te->diff[1] = v.y; te->diff[2] = v.z;
    te->diff[3] = w.x; te->diff[4] = w.y; te->diff[5] = w.z;
  }
  if (!with_jacobian) return;
  /* pinocchio::Jlog6: [[A, B], [0, A]] */
  double A[9], B[9], C[9];
  jlog3_canon(theta, w, A);
  {
    double beta, bdot;
    if (theta < TASK_TAYLOR) {
      beta = 1.0 / 12.0 + t2 / 720.0;
      bdot = 1.0 / 360.0;
    } else {
      const double tinv = 1.0 / theta, t2inv = tinv * tinv;
      const double inv_2_2ct = 1.0 / (2.0 * (1.0 - ct));
      beta = t2inv - (st * tinv) * inv_2_2ct;
      bdot = -2.0 * (t2inv * t2inv) + ((1.0 + st * tinv) * t2inv) * inv_2_2ct;
    }
    const double wTp = vdot(w, pd);
    const v3_t v3 = vsub(vscale(bdot * wTp, w), vscale(fma(t2, bdot, 2.0 * beta), pd));
    const v3_t bw = vscale(beta, w);
    const double v3v[3] = {v3.x, v3.y, v3.z}, bwv[3] = {bw.x, bw.y, bw.z}, wv[3] = {w.x, w.y, w.z},
                 pv[3] = {pd.x, pd.y, pd.z};
    for (int r = 0; r < 3; ++r)
      for (int k = 0; k < 3; ++k) C[3 * r + k] = fma(bwv[r], pv[k], v3v[r] * wv[k]);
    const double dg = wTp * beta;
    C[0] += dg; C[4] += dg; C[8] += dg;
    add_skew(vscale(0.5, pd), C);
    for (int r = 0; r < 3; ++r)
      for (int k = 0; k < 3; ++k) B[3 * r + k] = fma(C[3 * r + 2], A[6 + k], fma(C[3 * r + 1], A[3 + k], C[3 * r] * A[k]));
  }
  /* getFrameJacobian(frame, LOCAL) column c = [Rf^T (S_l + S_w x pf); Rf^T S_w] with the world-frame joint
   * axes S_w = z_c, S_l = p_c x z_c; JJ = Jlog6 * J */
  for (int c = 0; c < NV; ++c) {
    const v3_t Sw = V3(R[c][2], R[c][5], R[c][8]);
    const v3_t Sl = vcross(p[c], Sw);
    const v3_t Jl = mulT3(Rf, vadd(Sl, vcross(Sw, pf)));
    const v3_t Ja = mulT3(Rf, Sw);
    for (int r = 0; r < 3; ++r) {
      te->JJ[c * 6 + r] = dot3r(A + 3 * r, Jl) + dot3r(B + 3 * r, Ja);
      te->JJ[c * 6 + 3 + r] = dot3r(A + 3 * r, Ja);
    }
  }
}

/* set_q_6d_weight(position_weight, rotation_weight) stores head<3> = rotation_weight, tail<3> =
 * position_weight (time_varying_task_space_6d_cost.cpp:45-50) while diff_6d = [linear; angular]: the
 * rotation weight multiplies the linear part.  Restated as is.  wpr = [position(3), rotation(3)]. */
static inline double task_w6k(int kind, const double* wpr, int k) {
  if (kind == 2) return k < 3 ? wpr[k] : 0.0;   /* TaskSpace3DCost: q_3d_weight applies to diff_3d as given */
  return k < 3 ? wpr[3 + k] : wpr[k - 3];
}
#define task_w6(wpr, k) task_w6k(te->kind, wpr, k)

/* lq += scale * JJ^T diag(w6) diff (:116-118, :132-133) */
static void task_add_gradient(const task_eval_t* te, const double* wpr, double scale, int use_scale, double* lq) {
  for (int c = 0; c < NV; ++c) {
    double acc = 0;
    for (int k = 0; k < 6; ++k) acc = fma(te->JJ[c * 6 + k], task_w6(wpr, k) * te->diff[k], acc);
    lq[c] += use_scale ? scale * acc : acc;
  }
}
/* Qqq += scale * JJ^T diag(w6) JJ (:161-162, :175-176) */
static void task_add_hessian(const task_eval_t* te, const double* wpr, double scale, int use_scale, double* Qqq) {
  for (int c = 0; c < NV; ++c)
    for (int r = 0; r < NV; ++r) {
      double acc = 0;
      for (int k = 0; k < 6; ++k) acc = fma(te->JJ[r * 6 + k], task_w6(wpr, k) * te->JJ[c * 6 + k], acc);
      Qqq[c * NV + r] += use_scale ? scale * acc : acc;
    }
}
/* sum(w6 * diff^2) (:74, :87) */
static double task_weighted_sqnorm(const task_eval_t* te, const double* wpr) {
  double l = 0;
  for (int k = 0; k < 6; ++k) l += (task_w6(wpr, k) * te->diff[k]) * te->diff[k];
  return l;
}

/* parity / test getter: diff_6d (6) and JJ_6d (6 x 7, column-major) for a configuration and a reference */
void oracle_task_evaluate_kind(const double* q, const double* ref12, int kind, double* diff6, double* JJ) {
  task_eval_t te;
  task_evaluate(q, ref12, &te, 1, kind);
  memcpy(diff6, te.diff, sizeof(te.diff));
  memcpy(JJ, te.JJ, sizeof(te.JJ));
}
void oracle_task_evaluate(const double* q, const double* ref12, double* diff6, double* JJ) {
  task_eval_t te;
  task_evaluate(q, ref12, &te, 1, 1);
  memcpy(diff6, te.diff, sizeof(te.diff));
  memcpy(JJ, te.JJ, sizeof(te.JJ));
}
/* end-effector placement oMf (R row-major 9, p 3) and LOCAL frame Jacobian (6 x 7 column-major, [lin; ang]) */
void oracle_frame_kinematics(const double* q, double* oMf12, double* J) {
  double R[LANES][9];
  v3_t p[LANES];
  chain_fk(q, R, p);
  const double* R6 = R[IIWA14_EE_PARENT_JOINT];
  const double* E = IIWA14_EE_PLACEMENT_R;
  double Rf[9];
  for (int r = 0; r < 3; ++r)
    for (int k = 0; k < 3; ++k)
      Rf[3 * r + k] = fma(R6[3 * r + 2], E[6 + k], fma(R6[3 * r + 1], E[3 + k], R6[3 * r] * E[k]));
  const v3_t ep = V3(IIWA14_EE_PLACEMENT_P[0], IIWA14_EE_PLACEMENT_P[1], IIWA14_EE_PLACEMENT_P[2]);
  const v3_t p6 = p[IIWA14_EE_PARENT_JOINT];
  const v3_t pf = V3(fma(R6[2], ep.z, fma(R6[1], ep.y, fma(R6[0], ep.x, p6.x))),
                     fma(R6[5], ep.z, fma(R6[4], ep.y, fma(R6[3], ep.x, p6.y))),
                     fma(R6[8], ep.z, fma(R6[7], ep.y, fma(R6[6], ep.x, p6.z))));
  memcpy(oMf12, Rf, sizeof(Rf));
  oMf12[9] = pf.x; oMf12[10] = pf.y; oMf12[11] = pf.z;
  for (int c = 0; c < NV; ++c) {
    const v3_t Sw = V3(R[c][2], R[c][5], R[c][8]);
    const v3_t Sl = vcross(p[c], Sw);
    const v3_t Jl = mulT3(Rf, vadd(Sl, vcross(Sw, pf)));
    const v3_t Ja = mulT3(Rf, Sw);
    J[c * 6 + 0] = Jl.x; J[c * 6 + 1] = Jl.y; J[c * 6 + 2] = Jl.z;
    J[c * 6 + 3] = Ja.x; J[c * 6 + 4] = Ja.y; J[c * 6 + 5] = Ja.z;
  }
}

/* ------------------------------------------------------------------------------------------ */
/* problem                                                                                     */
/* ------------------------------------------------------------------------------------------ */
void oracle_problem_default(oracle_problem_t* p) {
  memset(p, 0, sizeof(*p));
  p->N = 20;
  p->T = 1.0;
  for (int i = 0; i < NV; ++i) {
    p->q_min[i] = IIWA14_Q_MIN[i];
    p->q_max[i] = IIWA14_Q_MAX[i];
    p->v_max[i] = IIWA14_V_MAX[i];
    p->u_max[i] = IIWA14_EFFORT_MAX[i];
  }
  p->barrier = 1.0e-04;
  p->fraction_rate = 0.995;
}

/* ------------------------------------------------------------------------------------------ */
/* data types                                                                                  */
/* ------------------------------------------------------------------------------------------ */
typedef struct { double lmd[NV], gmm[NV], q[NV], v[NV], a[NV], u[NV], beta[NV]; } split_solution_t;
typedef struct { double dlmd[NV], dgmm[NV], dq[NV], dv[NV], da[NV], du[NV], dbeta[NV]; } split_direction_t;
/* ConstraintComponentData (constraints/constraint_component_data.hxx:12-21) */
typedef struct { double slack[NV], dual[NV], residual[NV], duality[NV], dslack[NV], ddual[NV]; } cdata_t;

/* component order = JointConstraintsFactory push_back order regrouped by kinematics level
 * (src/utils/joint_constraints_factory.cpp:30-35, constraints/constraints.hxx:23-34):
 * 0 pos-lower 1 pos-upper | 2 vel-lower 3 vel-upper | 4 torque-lower 5 torque-upper */
enum { C_POS_LO = 0, C_POS_UP, C_VEL_LO, C_VEL_UP, C_TRQ_LO, C_TRQ_UP, C_ACC_LO, C_ACC_UP };

typedef struct {
  /* SplitKKTResidual / SplitKKTMatrix pieces the unconstrained path touches */
  double lq[NV], lv[NV], la[NV], lu[NV], Fq[NV], Fv[NV];
  double Qqq[NN];                 /* full (task-space cost fills it densely) */
  double Qvv[NV], Qaa[NV], Quu[NV]; /* diagonals */
  /* UnconstrainedDynamics members (unocp/unconstrained_dynamics.hxx) */
  double ID[NV], dIDdq[NN], dIDdv[NN], dIDda[NN], lu_condensed[NV];
  /* SplitUnKKTMatrix blocks (order a,q,v; split_unkkt_matrix.hxx:31-118) and SplitUnKKTResidual */
  double uQaa[NN], uQaq[NN], uQav[NN], uQqq[NN], uQqv[NN], uQvq[NN], uQvv[NN];
  double ula[NV], ulq[NV], ulv[NV], uFq[NV], uFv[NV];
  /* LQR policy + Riccati factorisation */
  double K[NV * 2 * NV], k[NV];
  cdata_t c[NC];
  int active[NC];
  task_eval_t te;                 /* CostFunctionData of the task-space cost (diff_6d, JJ_6d) */
} stage_t;

typedef struct { double Pqq[NN], Pqv[NN], Pvq[NN], Pvv[NN], sq[NV], sv[NV]; } riccati_t;

#define FILTER_MAX 256
typedef struct { int n; double cost[FILTER_MAX], viol[FILTER_MAX]; } filter_t;

struct oracle_unocp {
  oracle_problem_t p;
  int N;
  double dt;
  split_solution_t* s;      /* N+1 */
  split_direction_t* d;     /* N+1 */
  stage_t* st;              /* N */
  riccati_t* ric;           /* N+1 */
  /* terminal stage */
  double t_lq[NV], t_lv[NV], t_Qqq[NN], t_Qvv[NN];
  double primal_step, dual_step, max_primal_step;
  filter_t filter;
  split_solution_t* s_try;  /* N+1 */
  int stage_threads;
  double* task_ref;         /* (N+1) x 12: SE3 reference of every stage's time (R row-major, p) */
};

/* ------------------------------------------------------------------------------------------ */
/* constraints/ : pdipm + the six joint-limit components                                       */
/* ------------------------------------------------------------------------------------------ */
/* constraints_data.hpp:18-43: which kinematics levels are live at a time stage */
static void set_active(const oracle_problem_t* p, int time_stage, int* active) {
  const int pos = time_stage >= 2, vel = time_stage >= 1, acc = time_stage >= 0;
  active[C_POS_LO] = active[C_POS_UP] = pos;
  active[C_VEL_LO] = active[C_VEL_UP] = vel;
  active[C_TRQ_LO] = active[C_TRQ_UP] = acc;
  active[C_ACC_LO] = acc && p->enable_acc[0];   /* KinematicsLevel::AccelerationLevel (joint_acceleration_lower_limit.cpp:24-26) */
  active[C_ACC_UP] = acc && p->enable_acc[1];
}

/* g such that slack = g at initialisation and residual = -g + slack  (e.g.
 * joint_position_lower_limit.cpp:50-55,84-89; siblings differ by sign/variable only) */
static inline double con_margin(const oracle_problem_t* p, int comp, const split_solution_t* s, int j) {
  switch (comp) {
    case C_POS_LO: return s->q[j] - p->q_min[j];
    case C_POS_UP: return p->q_max[j] - s->q[j];
    case C_VEL_LO: return s->v[j] - (-p->v_max[j]);
    case C_VEL_UP: return p->v_max[j] - s->v[j];
    case C_TRQ_LO: return s->u[j] - (-p->u_max[j]);
    case C_ACC_LO: return s->a[j] - p->a_min[j];
    case C_ACC_UP: return p->a_max[j] - s->a[j];
    default:       return p->u_max[j] - s->u[j];
  }
}

/* pdipm::SetSlackAndDualPositive (constraints/pdipm.hxx:13-23) */
static void set_slack_and_dual(const oracle_problem_t* p, stage_t* st, const split_solution_t* s) {
  for (int c = 0; c < NC; ++c) {
    cdata_t* d = &st->c[c];
    memset(d, 0, sizeof(*d));
    if (!st->active[c]) continue;
    for (int j = 0; j < NV; ++j) {
      double sl = con_margin(p, c, s, j);
      for (int guard = 0; sl < p->barrier && guard < (1 << 20); ++guard) sl += p->barrier;   /* bound: see k_init_constraints */
      d->slack[j] = sl;
      d->dual[j] = p->barrier / sl;
    }
  }
}

/* computePrimalAndDualResidual of every live component (e.g. joint_position_lower_limit.cpp:84-89)
 * + pdipm::ComputeDuality (pdipm.hxx:26-31).  Written exactly as the reference: residual =
 * (limit - x + slack) for lower limits, (x - limit + slack) for upper limits. */
static void compute_primal_dual_residual(const oracle_problem_t* p, stage_t* st, const split_solution_t* s) {
  for (int c = 0; c < NC; ++c) {
    if (!st->active[c]) continue;
    cdata_t* d = &st->c[c];
    for (int j = 0; j < NV; ++j) {
      double r;
      switch (c) {
        case C_POS_LO: r = p->q_min[j] - s->q[j] + d->slack[j]; break;
        case C_POS_UP: r = s->q[j] - p->q_max[j] + d->slack[j]; break;
        case C_VEL_LO: r = (-p->v_max[j]) - s->v[j] + d->slack[j]; break;
        case C_VEL_UP: r = s->v[j] - p->v_max[j] + d->slack[j]; break;
        case C_TRQ_LO: r = (-p->u_max[j]) - s->u[j] + d->slack[j]; break;
        case C_ACC_LO: r = p->a_min[j] - s->a[j] + d->slack[j]; break;
        case C_ACC_UP: r = s->a[j] - p->a_max[j] + d->slack[j]; break;
        default:       r = s->u[j] - p->u_max[j] + d->slack[j]; break;
      }
      d->residual[j] = r;
      d->duality[j] = d->slack[j] * d->dual[j] - p->barrier;
    }
  }
}

static inline double* con_grad(stage_t* st, int comp) {
  return comp <= C_POS_UP ? st->lq : (comp <= C_VEL_UP ? st->lv : (comp >= C_ACC_LO ? st->la : st->lu));
}
static inline double con_sign(int comp) { return (comp & 1) ? 1.0 : -1.0; } /* lower: -, upper: + */

/* Constraints::augmentDualResidual (constraints.hxx:153-172; joint_*_limit.cpp augmentDualResidual) */
static void augment_dual_residual(stage_t* st, double dt) {
  for (int c = 0; c < NC; ++c) {
    if (!st->active[c]) continue;
    double* l = con_grad(st, c);
    const double sg = con_sign(c);
    for (int j = 0; j < NV; ++j) l[j] += sg * (dt * st->c[c].dual[j]);
  }
}

/* Constraints::condenseSlackAndDual (e.g. joint_position_lower_limit.cpp:64-74) */
static void condense_slack_and_dual(const oracle_problem_t* p, stage_t* st, const split_solution_t* s, double dt) {
  compute_primal_dual_residual(p, st, s);
  for (int c = 0; c < NC; ++c) {
    if (!st->active[c]) continue;
    cdata_t* d = &st->c[c];
    double* l = con_grad(st, c);
    const double sg = con_sign(c);
    for (int j = 0; j < NV; ++j) {
      /* canonical arithmetic: the two divisions by the slack share one reciprocal */
      const double rs = 1.0 / d->slack[j];
      const double h = (dt * d->dual[j]) * rs;
      if (c <= C_POS_UP) st->Qqq[j * NV + j] += h;
      else if (c <= C_VEL_UP) st->Qvv[j] += h;
      else if (c >= C_ACC_LO) st->Qaa[j] += h;
      else st->Quu[j] += h;
      l[j] += sg * ((dt * fma(d->dual[j], d->residual[j], -d->duality[j])) * rs);
    }
  }
}

/* computeSlackAndDualDirection (e.g. joint_torques_upper_limit.cpp:75-80) + pdipm::ComputeDualDirection
 * (pdipm.hxx:76-81) */
static void compute_slack_dual_direction(stage_t* st, const split_direction_t* d) {
  for (int c = 0; c < NC; ++c) {
    if (!st->active[c]) continue;
    cdata_t* cd = &st->c[c];
    const double* dx = c <= C_POS_UP ? d->dq : (c <= C_VEL_UP ? d->dv : (c >= C_ACC_LO ? d->da : d->du));
    for (int j = 0; j < NV; ++j) {
      cd->dslack[j] = ((c & 1) ? -dx[j] : dx[j]) - cd->residual[j];
      cd->ddual[j] = -fma(cd->dual[j], cd->dslack[j], cd->duality[j]) / cd->slack[j];
    }
  }
}

/* pdipm::FractionToBoundary (pdipm.hxx:52-73), literal: only fractions strictly inside (0,1) count */
static double fraction_to_boundary(double rate, const double* vec, const double* dvec) {
  double mn = 1.0;
  for (int i = 0; i < NV; ++i) {
    const double f = -rate * (vec[i] / dvec[i]);
    if (f > 0 && f < 1) {
      if (f < mn) mn = f;
    }
  }
  return mn;
}

static double max_slack_step(const oracle_problem_t* p, const stage_t* st) {
  double mn = 1.0;
  for (int c = 0; c < NC; ++c) {
    if (!st->active[c]) continue;
    const double f = fraction_to_boundary(p->fraction_rate, st->c[c].slack, st->c[c].dslack);
    if (f < mn) mn = f;
  }
  return mn;
}
static double max_dual_step(const oracle_problem_t* p, const stage_t* st) {
  double mn = 1.0;
  for (int c = 0; c < NC; ++c) {
    if (!st->active[c]) continue;
    const double f = fraction_to_boundary(p->fraction_rate, st->c[c].dual, st->c[c].ddual);
    if (f < mn) mn = f;
  }
  return mn;
}

/* ------------------------------------------------------------------------------------------ */
/* cost/ : ConfigurationSpaceCost (src/cost/configuration_space_cost.cpp:241-396)              */
/* ------------------------------------------------------------------------------------------ */
/* CostFunction::computeStageCostDerivatives (cost/cost_function.hxx:78-85): components in push_back
 * order, ConfigurationSpaceCost then (when enabled) TimeVaryingTaskSpace6DCost with the reference
 * SE3 `ref` of this stage's time */
static void stage_cost_derivatives(const oracle_problem_t* p, double dt, const split_solution_t* s, stage_t* st,
                                   const double* ref) {
  for (int j = 0; j < NV; ++j) {
    st->lq[j] += dt * p->q_weight[j] * (s->q[j] - p->q_ref[j]);
    st->lv[j] += dt * p->v_weight[j] * (s->v[j] - p->v_ref[j]);
    st->la[j] += dt * p->a_weight[j] * s->a[j];
    st->lu[j] += dt * p->u_weight[j] * (s->u[j] - p->u_ref[j]);
  }
  if (p->task_enabled) {
    task_evaluate(s->q, ref, &st->te, 1, p->task_enabled);
    task_add_gradient(&st->te, p->task_q_weight, dt, 1, st->lq);
  }
}
/* CostFunction::computeStageCostHessian (:107-114) */
static void stage_cost_hessian(const oracle_problem_t* p, double dt, stage_t* st) {
  for (int j = 0; j < NV; ++j) {
    st->Qqq[j * NV + j] += dt * p->q_weight[j];
    st->Qvv[j] += dt * p->v_weight[j];
    st->Qaa[j] += dt * p->a_weight[j];
    st->Quu[j] += dt * p->u_weight[j];
  }
  if (p->task_enabled) task_add_hessian(&st->te, p->task_q_weight, dt, 1, st->Qqq);
}
/* CostFunction::computeStageCost / computeTerminalCost: sum of the components' values */
static double task_stage_cost(const oracle_problem_t* p, double dt, const double* q, const double* ref) {
  task_eval_t te;
  task_evaluate(q, ref, &te, 0, p->task_enabled);
  return 0.5 * dt * task_weighted_sqnorm(&te, p->task_q_weight);
}
static double task_terminal_cost(const oracle_problem_t* p, const double* q, const double* ref) {
  task_eval_t te;
  task_evaluate(q, ref, &te, 0, p->task_enabled);
  return 0.5 * task_weighted_sqnorm(&te, p->task_qf_weight);
}
static double stage_cost(const oracle_problem_t* p, double dt, const split_solution_t* s) {
  double l = 0, part;
  part = 0; for (int j = 0; j < NV; ++j) part += p->q_weight[j] * (s->q[j] - p->q_ref[j]) * (s->q[j] - p->q_ref[j]);
  l += part;
  part = 0; for (int j = 0; j < NV; ++j) part += p->v_weight[j] * (s->v[j] - p->v_ref[j]) * (s->v[j] - p->v_ref[j]);
  l += part;
  part = 0; for (int j = 0; j < NV; ++j) part += p->a_weight[j] * s->a[j] * s->a[j];
  l += part;
  part = 0; for (int j = 0; j < NV; ++j) part += p->u_weight[j] * (s->u[j] - p->u_ref[j]) * (s->u[j] - p->u_ref[j]);
  l += part;
  return 0.5 * dt * l;
}
static double terminal_cost(const oracle_problem_t* p, const split_solution_t* s) {
  double l = 0, part;
  part = 0; for (int j = 0; j < NV; ++j) part += p->qf_weight[j] * (s->q[j] - p->q_ref[j]) * (s->q[j] - p->q_ref[j]);
  l += part;
  part = 0; for (int j = 0; j < NV; ++j) part += p->vf_weight[j] * (s->v[j] - p->v_ref[j]) * (s->v[j] - p->v_ref[j]);
  l += part;
  return 0.5 * l;
}

/* ------------------------------------------------------------------------------------------ */
/* SplitUnOCP (unocp/split_unocp.hxx)                                                          */
/* ------------------------------------------------------------------------------------------ */
/* steps 1-4 of SURVEY A.2, shared by linearizeOCP (:69-99) and computeKKTResidual (:141-161) */
static void stage_residual_common(const oracle_problem_t* p, double dt, const split_solution_t* s,
                                  const split_solution_t* sn, stage_t* st, int with_derivatives, const double* ref) {
  memset(st->lq, 0, sizeof(double) * NV); memset(st->lv, 0, sizeof(double) * NV);
  memset(st->la, 0, sizeof(double) * NV); memset(st->lu, 0, sizeof(double) * NV);
  stage_cost_derivatives(p, dt, s, st, ref);
  augment_dual_residual(st, dt);
  /* stateequation::linearizeForwardEuler (ocp/state_equation.hxx:11-37,210-221) */
  for (int j = 0; j < NV; ++j) {
    st->Fq[j] = fma(dt, s->v[j], s->q[j] - sn->q[j]);
    st->Fv[j] = fma(dt, s->a[j], s->v[j]) - sn->v[j];
  }
  for (int j = 0; j < NV; ++j) {
    st->lq[j] += sn->lmd[j] - s->lmd[j];
    st->lv[j] += fma(dt, sn->lmd[j], sn->gmm[j]) - s->gmm[j];
    st->la[j] = fma(dt, sn->gmm[j], st->la[j]);
  }
  /* UnconstrainedDynamics::linearizeUnconstrainedDynamics (unocp/unconstrained_dynamics.hxx:55-65,166-177) */
  (void)with_derivatives;
  rnea_derivatives_impl(s->q, s->v, s->a, st->ID, st->dIDdq, st->dIDdv, st->dIDda);
  for (int j = 0; j < NV; ++j) st->ID[j] -= s->u[j];
  for (int j = 0; j < NV; ++j) {
    double tq = 0, tv = 0, ta = 0;
    for (int k = 0; k < NV; ++k) {
      tq = fma(st->dIDdq[j * NV + k], s->beta[k], tq);
      tv = fma(st->dIDdv[j * NV + k], s->beta[k], tv);
      ta = fma(st->dIDda[j * NV + k], s->beta[k], ta);
    }
    st->lq[j] = fma(dt, tq, st->lq[j]);
    st->lv[j] = fma(dt, tv, st->lv[j]);
    st->la[j] = fma(dt, ta, st->la[j]);
    st->lu[j] = fma(-dt, s->beta[j], st->lu[j]);
  }
}

/* SplitUnOCP::linearizeOCP (unocp/split_unocp.hxx:69-99) */
static void split_unocp_linearize(const oracle_problem_t* p, double dt, const split_solution_t* s,
                                  const split_solution_t* sn, stage_t* st, const double* ref) {
  memset(st->Qqq, 0, sizeof(st->Qqq));
  memset(st->Qvv, 0, sizeof(st->Qvv)); memset(st->Qaa, 0, sizeof(st->Qaa)); memset(st->Quu, 0, sizeof(st->Quu));
  stage_residual_common(p, dt, s, sn, st, 1, ref);
  stage_cost_hessian(p, dt, st);
  condense_slack_and_dual(p, st, s, dt);
  /* UnconstrainedDynamics::condenseUnconstrainedDynamics (unconstrained_dynamics.hxx:68-94) */
  for (int j = 0; j < NV; ++j) st->lu_condensed[j] = fma(st->Quu[j], st->ID[j], st->lu[j]);
  for (int j = 0; j < NV; ++j) {
    double tq = 0, tv = 0, ta = 0;
    for (int k = 0; k < NV; ++k) {
      tq = fma(st->dIDdq[j * NV + k], st->lu_condensed[k], tq);
      tv = fma(st->dIDdv[j * NV + k], st->lu_condensed[k], tv);
      ta = fma(st->dIDda[j * NV + k], st->lu_condensed[k], ta);
    }
    st->ulq[j] = st->lq[j] + tq;
    st->ulv[j] = st->lv[j] + tv;
    st->ula[j] = st->la[j] + ta;
    st->uFq[j] = st->Fq[j];
    st->uFv[j] = st->Fv[j];
  }
  /* Q_xy = (dID_dx)^T diag(Quu) (dID_dy) */
  for (int c = 0; c < NV; ++c)
    for (int r = 0; r < NV; ++r) {
      double qq = 0, qv = 0, vv = 0, aq = 0, av = 0, aa = 0;
      for (int k = 0; k < NV; ++k) {
        const double Dq = st->Quu[k] * st->dIDdq[c * NV + k];
        const double Dv = st->Quu[k] * st->dIDdv[c * NV + k];
        const double Da = st->Quu[k] * st->dIDda[c * NV + k];
        qq = fma(st->dIDdq[r * NV + k], Dq, qq);
        qv = fma(st->dIDdq[r * NV + k], Dv, qv);
        vv = fma(st->dIDdv[r * NV + k], Dv, vv);
        aq = fma(st->dIDda[r * NV + k], Dq, aq);
        av = fma(st->dIDda[r * NV + k], Dv, av);
        aa = fma(st->dIDda[r * NV + k], Da, aa);
      }
      st->uQqq[c * NV + r] = qq + st->Qqq[c * NV + r];
      st->uQqv[c * NV + r] = qv;
      st->uQvv[c * NV + r] = vv + (r == c ? st->Qvv[r] : 0.0);
      st->uQaq[c * NV + r] = aq;
      st->uQav[c * NV + r] = av;
      st->uQaa[c * NV + r] = aa + (r == c ? st->Qaa[r] : 0.0);
    }
}

/* SplitUnOCP::computeKKTResidual (split_unocp.hxx:141-161) */
static void split_unocp_kkt_residual(const oracle_problem_t* p, double dt, const split_solution_t* s,
                                     const split_solution_t* sn, stage_t* st, const double* ref) {
  compute_primal_dual_residual(p, st, s);
  stage_residual_common(p, dt, s, sn, st, 0, ref);
}

static double sqnorm(const double* x) {
  double r = 0;
  for (int j = 0; j < NV; ++j) r += x[j] * x[j];
  return r;
}
static double l1norm(const double* x) {
  double r = 0;
  for (int j = 0; j < NV; ++j) r += fabs(x[j]);
  return r;
}

/* SplitUnOCP::squaredNormKKTResidual (split_unocp.hxx:164-174) */
static double split_unocp_sqnorm(const stage_t* st, double dt) {
  double e = 0;
  e += sqnorm(st->lq) + sqnorm(st->lv);   /* lx */
  e += sqnorm(st->la);
  e += sqnorm(st->lu);
  e += sqnorm(st->Fq) + sqnorm(st->Fv);   /* Fx */
  e += dt * dt * sqnorm(st->ID);
  double c2 = 0;
  for (int c = 0; c < NC; ++c)
    if (st->active[c]) c2 += sqnorm(st->c[c].residual) + sqnorm(st->c[c].duality);
  e += dt * dt * c2;
  return e;
}

/* UnconstrainedDynamics::computeCondensedDirection (unconstrained_dynamics.hxx:97-106) +
 * Constraints::computeSlackAndDualDirection */
static void split_unocp_condensed_direction(stage_t* st, double dt, split_direction_t* d) {
  for (int r = 0; r < NV; ++r) {
    double acc = st->ID[r];
    double t = 0;
    for (int c = 0; c < NV; ++c) t = fma(st->dIDdq[c * NV + r], d->dq[c], t);
    acc += t;
    t = 0;
    for (int c = 0; c < NV; ++c) t = fma(st->dIDdv[c * NV + r], d->dv[c], t);
    acc += t;
    t = 0;
    for (int c = 0; c < NV; ++c) t = fma(st->dIDda[c * NV + r], d->da[c], t);
    acc += t;
    d->du[r] = acc;
  }
  for (int r = 0; r < NV; ++r) d->dbeta[r] = fma(st->Quu[r], d->du[r], st->lu[r]) / dt;
  compute_slack_dual_direction(st, d);
}

/* ------------------------------------------------------------------------------------------ */
/* Riccati recursion (unocp/backward_unriccati_recursion_factorizer.hxx,                        */
/* unocp/split_unriccati_factorizer.hxx, src/unocp/unriccati_recursion.cpp)                    */
/* ------------------------------------------------------------------------------------------ */
/* Eigen::LLT<MatrixXd, Lower>: unblocked left-looking Cholesky reading the lower triangle only
 * (SURVEY A.7); returns 0 on success, k+1 when pivot k is not positive (or outside the range of
 * canon_pivot_ok).  Canonical arithmetic: rd[k] = canon_rsqrt(pivot) ~ 1 / L_kk (canon_pivot.h) and the
 * divisions by the diagonal are multiplications by it (rounding-level deviation from Eigen's
 * sqrt + division, far inside the unpinned Eigen boundary). */
static int llt_lower(const double* A, int n, double* L, double* rd) {
  int info = 0;
  for (int i = 0; i < n * n; ++i) L[i] = 0.0;
  for (int k = 0; k < n; ++k) {
    double x = A[k * n + k];
    for (int j = 0; j < k; ++j) x = fma(-L[j * n + k], L[j * n + k], x);
    if (!canon_pivot_ok(x) && !info) info = k + 1;
    rd[k] = canon_rsqrt(x);
    L[k * n + k] = x * rd[k];
    for (int i = k + 1; i < n; ++i) {
      double y = A[k * n + i];
      for (int j = 0; j < k; ++j) y = fma(-L[j * n + i], L[j * n + k], y);
      L[k * n + i] = y * rd[k];
    }
  }
  return info;
}
/* x = (L L^T)^-1 b : forward then backward substitution, one right-hand side */
static void llt_solve(const double* L, const double* rd, int n, const double* b, double* x) {
  for (int i = 0; i < n; ++i) {
    double y = b[i];
    for (int j = 0; j < i; ++j) y = fma(-L[j * n + i], x[j], y);
    x[i] = y * rd[i];
  }
  for (int i = n - 1; i >= 0; --i) {
    double y = x[i];
    for (int j = i + 1; j < n; ++j) y = fma(-L[i * n + j], x[j], y);
    x[i] = y * rd[i];
  }
}

/* the same with the terms of the backward substitution subtracted from the last column backwards (the order in
 * which a column-oriented sweep delivers them: row i is complete but for one term when x[i+1] becomes final, so the
 * rows do not form one long dependent chain).  Used by the 21 + 14 unit right-hand sides of invert_unkkt. */
static void llt_solve_desc(const double* L, const double* rd, int n, const double* b, double* x) {
  for (int i = 0; i < n; ++i) {
    double y = b[i];
    for (int j = 0; j < i; ++j) y = fma(-L[j * n + i], x[j], y);
    x[i] = y * rd[i];
  }
  for (int i = n - 1; i >= 0; --i) {
    double y = x[i];
    for (int j = n - 1; j > i; --j) y = fma(-L[i * n + j], x[j], y);
    x[i] = y * rd[i];
  }
}

/* SplitUnRiccatiFactorizer::backwardRiccatiRecursion (split_unriccati_factorizer.hxx:30-46) */
static int riccati_backward_stage(const riccati_t* rn, double dt, stage_t* st, riccati_t* r) {
  /* BackwardUnRiccatiRecursionFactorizer::factorizeKKTMatrix (:29-54) */
  const double dt2 = dt * dt;
  for (int c = 0; c < NV; ++c)
    for (int rr = 0; rr < NV; ++rr) {
      const int i = c * NV + rr, it = rr * NV + c;
      st->uQqq[i] += rn->Pqq[i];
      st->uQqv[i] = fma(dt, rn->Pqq[i], st->uQqv[i]);
      st->uQqv[i] += rn->Pqv[i];
      st->uQvv[i] = fma(dt2, rn->Pqq[i], st->uQvv[i]);
      st->uQvv[i] = fma(dt, rn->Pqv[i], st->uQvv[i]);
      st->uQvv[i] = fma(dt, rn->Pqv[it], st->uQvv[i]);
      st->uQvv[i] += rn->Pvv[i];
      st->uQaq[i] = fma(dt, rn->Pqv[it], st->uQaq[i]);            /* Qaq^T += dt Pqv */
      st->uQav[i] = fma(dt2, rn->Pqv[it], st->uQav[i]);           /* Qav^T += dt^2 Pqv + dt Pvv */
      st->uQav[i] = fma(dt, rn->Pvv[it], st->uQav[i]);
      st->uQaa[i] = fma(dt2, rn->Pvv[i], st->uQaa[i]);
    }
  for (int c = 0; c < NV; ++c)
    for (int rr = 0; rr < NV; ++rr) st->uQvq[c * NV + rr] = st->uQqv[rr * NV + c];
  for (int j = 0; j < NV; ++j) {
    double t1 = 0, t2 = 0;
    for (int k = 0; k < NV; ++k) {
      t1 = fma(rn->Pqv[j * NV + k], st->uFq[k], t1);     /* (Pqv^T Fq)_j */
      t2 = fma(rn->Pvv[k * NV + j], st->uFv[k], t2);     /* (Pvv Fv)_j   */
    }
    st->ula[j] = fma(dt, t1, st->ula[j]);
    st->ula[j] = fma(dt, t2, st->ula[j]);
    st->ula[j] = fma(-dt, rn->sv[j], st->ula[j]);
  }
  /* llt_.compute(Qaa); K = -llt_.solve(Qax); k = -llt_.solve(la) (:37-40) */
  double L[NN], rd[NV], x[NV];
  const int info = llt_lower(st->uQaa, NV, L, rd);
  for (int c = 0; c < NV; ++c) {
    llt_solve(L, rd, NV, &st->uQaq[c * NV], x);
    for (int j = 0; j < NV; ++j) st->K[c * NV + j] = -x[j];
    llt_solve(L, rd, NV, &st->uQav[c * NV], x);
    for (int j = 0; j < NV; ++j) st->K[(NV + c) * NV + j] = -x[j];
  }
  llt_solve(L, rd, NV, st->ula, x);
  for (int j = 0; j < NV; ++j) st->k[j] = -x[j];
  /* factorizeRiccatiFactorization (:57-89) */
  double GK[NV * 2 * NV];
  for (int c = 0; c < 2 * NV; ++c)
    for (int rr = 0; rr < NV; ++rr) {
      double t = 0;
      for (int k = 0; k < NV; ++k) t = fma(st->uQaa[k * NV + rr], st->K[c * NV + k], t);
      GK[c * NV + rr] = t;
    }
  const double* Kq = st->K;
  const double* Kv = st->K + NN;
  const double* GKq = GK;
  const double* GKv = GK + NN;
  for (int c = 0; c < NV; ++c)
    for (int rr = 0; rr < NV; ++rr) {
      double tqq = 0, tqv = 0, tvv = 0;
      for (int k = 0; k < NV; ++k) {
        tqq = fma(Kq[rr * NV + k], GKq[c * NV + k], tqq);
        tqv = fma(Kq[rr * NV + k], GKv[c * NV + k], tqv);
        tvv = fma(Kv[rr * NV + k], GKv[c * NV + k], tvv);
      }
      r->Pqq[c * NV + rr] = st->uQqq[c * NV + rr] - tqq;
      r->Pqv[c * NV + rr] = st->uQqv[c * NV + rr] - tqv;
      r->Pvv[c * NV + rr] = st->uQvv[c * NV + rr] - tvv;
    }
  for (int c = 0; c < NV; ++c)
    for (int rr = 0; rr < NV; ++rr) r->Pvq[c * NV + rr] = r->Pqv[rr * NV + c];
  /* preserve the symmetry */
  for (int c = 0; c < NV; ++c)
    for (int rr = c; rr < NV; ++rr) {
      const double a = 0.5 * (r->Pqq[c * NV + rr] + r->Pqq[rr * NV + c]);
      r->Pqq[c * NV + rr] = a; r->Pqq[rr * NV + c] = a;
      const double b = 0.5 * (r->Pvv[c * NV + rr] + r->Pvv[rr * NV + c]);
      r->Pvv[c * NV + rr] = b; r->Pvv[rr * NV + c] = b;
    }
  for (int j = 0; j < NV; ++j) {
    double t1 = 0, t2 = 0;
    for (int k = 0; k < NV; ++k) {
      t1 = fma(rn->Pqq[k * NV + j], st->uFq[k], t1);
      t2 = fma(rn->Pqv[k * NV + j], st->uFv[k], t2);
    }
    r->sq[j] = rn->sq[j];
    r->sq[j] -= t1;
    r->sq[j] -= t2;
  }
  for (int j = 0; j < NV; ++j) {
    double t1 = 0, t2 = 0;
    for (int k = 0; k < NV; ++k) {
      t1 = fma(rn->Pqv[j * NV + k], st->uFq[k], t1);     /* Pqv^T Fq */
      t2 = fma(rn->Pvv[k * NV + j], st->uFv[k], t2);
    }
    r->sv[j] = fma(dt, r->sq[j], rn->sv[j]);
    r->sv[j] -= t1;
    r->sv[j] -= t2;
  }
  for (int j = 0; j < NV; ++j) {
    r->sq[j] -= st->ulq[j];
    r->sv[j] -= st->ulv[j];
  }
  for (int j = 0; j < NV; ++j) {
    double t1 = 0, t2 = 0;
    for (int k = 0; k < NV; ++k) {
      t1 = fma(st->uQaq[j * NV + k], st->k[k], t1);      /* Qaq^T k */
      t2 = fma(st->uQav[j * NV + k], st->k[k], t2);
    }
    r->sq[j] -= t1;
    r->sv[j] -= t2;
  }
  return info;
}

/* ------------------------------------------------------------------------------------------ */
/* UnLineSearch + LineSearchFilter (line_search/unline_search.hpp:62-133,                      */
/* src/line_search/unline_search.cpp:56-135, src/line_search/line_search_filter.cpp:34-80)     */
/* ------------------------------------------------------------------------------------------ */
static int filter_is_accepted(const filter_t* f, double cost, double viol) {
  for (int i = 0; i < f->n; ++i)
    if (cost >= f->cost[i] && viol >= f->viol[i]) return 0;
  return 1;
}
static void filter_augment(filter_t* f, double cost, double viol) {
  int w = 0;
  for (int i = 0; i < f->n; ++i) {
    if (cost <= f->cost[i] && viol <= f->viol[i]) continue; /* erased */
    f->cost[w] = f->cost[i]; f->viol[w] = f->viol[i]; ++w;
  }
  f->n = w;
  if (f->n < FILTER_MAX) {
    f->cost[f->n] = cost - 0.005 * viol;       /* line_search_filter.hpp:16-17 */
    f->viol[f->n] = (1 - 0.005) * viol;
    ++f->n;
  }
}

/* SplitUnOCP::stageCost (split_unocp.hxx:177-196): cost + dt * barrier(slack + alpha dslack) */
static double split_unocp_stage_cost(const oracle_problem_t* p, double dt, const stage_t* st,
                                     const split_solution_t* s, double alpha, const double* ref) {
  double cost = stage_cost(p, dt, s);
  if (p->task_enabled) cost += task_stage_cost(p, dt, s->q, ref);
  double bar = 0;
  for (int c = 0; c < NC; ++c) {
    if (!st->active[c]) continue;
    double lg = 0;
    for (int j = 0; j < NV; ++j) {
      const double sl = alpha > 0 ? fma(alpha, st->c[c].dslack[j], st->c[c].slack[j]) : st->c[c].slack[j];
      lg += canon_log(sl);
    }
    bar += -p->barrier * lg;
  }
  cost += dt * bar;
  return cost;
}

/* SplitUnOCP::constraintViolation (split_unocp.hxx:199-217); note it overwrites residual/duality,
 * Fx and ID of the stage exactly as the reference does (the solver re-linearises afterwards). */
static double split_unocp_violation(const oracle_problem_t* p, double dt, stage_t* st,
                                    const split_solution_t* s, const double* qn, const double* vn) {
  compute_primal_dual_residual(p, st, s);
  for (int j = 0; j < NV; ++j) {
    st->Fq[j] = fma(dt, s->v[j], s->q[j] - qn[j]);
    st->Fv[j] = fma(dt, s->a[j], s->v[j]) - vn[j];
  }
  rnea_derivatives_impl(s->q, s->v, s->a, st->ID, NULL, NULL, NULL);
  for (int j = 0; j < NV; ++j) st->ID[j] -= s->u[j];
  double viol = 0;
  viol += l1norm(st->Fq) + l1norm(st->Fv);
  viol += dt * l1norm(st->ID);
  double c1 = 0;
  for (int c = 0; c < NC; ++c)
    if (st->active[c]) c1 += l1norm(st->c[c].residual);
  viol += dt * c1;
  return viol;
}

static void cost_and_violation(oracle_unocp_t* o, const split_solution_t* s, double alpha,
                               double* cost, double* viol) {
  double cs = 0, vs = 0;
  for (int i = 0; i <= o->N; ++i) {
    if (i < o->N) {
      cs += split_unocp_stage_cost(&o->p, o->dt, &o->st[i], &s[i], alpha, o->task_ref + (size_t)i * 12);
      vs += split_unocp_violation(&o->p, o->dt, &o->st[i], &s[i], s[i + 1].q, s[i + 1].v);
    } else {
      double tc = terminal_cost(&o->p, &s[i]);
      if (o->p.task_enabled) tc += task_terminal_cost(&o->p, s[i].q, o->task_ref + (size_t)i * 12);
      cs += tc;
    }
  }
  *cost = cs; *viol = vs;
}

static double line_search_step(oracle_unocp_t* o, double max_primal) {
  double cost, viol;
  if (o->filter.n == 0) {
    cost_and_violation(o, o->s, 0.0, &cost, &viol);
    filter_augment(&o->filter, cost, viol);
  }
  const double min_step = 0.05, rate = 0.75;       /* unline_search.hpp:25-26 */
  double alpha = max_primal;
  while (alpha > min_step) {
    for (int i = 0; i <= o->N; ++i) {
      split_solution_t* t = &o->s_try[i];
      for (int j = 0; j < NV; ++j) {
        t->q[j] = fma(alpha, o->d[i].dq[j], o->s[i].q[j]);
        t->v[j] = fma(alpha, o->d[i].dv[j], o->s[i].v[j]);
        t->a[j] = fma(alpha, o->d[i].da[j], o->s[i].a[j]);
        t->u[j] = fma(alpha, o->d[i].du[j], o->s[i].u[j]);
      }
    }
    cost_and_violation(o, o->s_try, alpha, &cost, &viol);
    if (filter_is_accepted(&o->filter, cost, viol)) {
      filter_augment(&o->filter, cost, viol);
      break;
    }
    alpha *= rate;
  }
  return alpha > min_step ? alpha : min_step;
}

/* ------------------------------------------------------------------------------------------ */
/* UnOCPSolver (src/unocp/unocp_solver.cpp)                                                    */
/* ------------------------------------------------------------------------------------------ */
oracle_unocp_t* oracle_unocp_create(const oracle_problem_t* p) {
  if (p->N <= 0 || !(p->T > 0)) return NULL;
  oracle_unocp_t* o = (oracle_unocp_t*)calloc(1, sizeof(*o));
  o->p = *p;
  o->N = p->N;
  o->dt = p->T / p->N;
  o->s = (split_solution_t*)calloc(o->N + 1, sizeof(split_solution_t));
  o->s_try = (split_solution_t*)calloc(o->N + 1, sizeof(split_solution_t));
  o->d = (split_direction_t*)calloc(o->N + 1, sizeof(split_direction_t));
  o->st = (stage_t*)calloc(o->N, sizeof(stage_t));
  o->ric = (riccati_t*)calloc(o->N + 1, sizeof(riccati_t));
  o->task_ref = (double*)calloc((size_t)(o->N + 1) * 12, sizeof(double));
  for (int i = 0; i <= o->N; ++i) o->task_ref[i * 12] = o->task_ref[i * 12 + 4] = o->task_ref[i * 12 + 8] = 1.0;
  o->stage_threads = 1;
  oracle_unocp_init_constraints(o);  /* the reference ctor ends with initConstraints() (:48) */
  return o;
}

void oracle_unocp_destroy(oracle_unocp_t* o) {
  if (!o) return;
  free(o->s); free(o->s_try); free(o->d); free(o->st); free(o->ric); free(o->task_ref); free(o);
}

void oracle_unocp_set_stage_threads(oracle_unocp_t* o, int nthreads) { o->stage_threads = nthreads > 0 ? nthreads : 1; }

/* UnOCPSolver::initConstraints (:59-70) */
void oracle_unocp_init_constraints(oracle_unocp_t* o) {
  for (int i = 0; i < o->N; ++i) {
    set_active(&o->p, i, o->st[i].active);
    set_slack_and_dual(&o->p, &o->st[i], &o->s[i]);
  }
}

/* UnOCPSolver::setSolution (:157-181) */
int oracle_unocp_set_solution(oracle_unocp_t* o, const char* name, const double* value) {
  for (int i = 0; i <= o->N; ++i) {
    double* dst;
    if (!strcmp(name, "q")) dst = o->s[i].q;
    else if (!strcmp(name, "v")) dst = o->s[i].v;
    else if (!strcmp(name, "a")) dst = o->s[i].a;
    else if (!strcmp(name, "u")) dst = o->s[i].u;
    else return -1;
    memcpy(dst, value, sizeof(double) * NV);
  }
  oracle_unocp_init_constraints(o);
  return 0;
}

/* TerminalOCP::linearizeOCP / computeKKTResidual (ocp/terminal_ocp.hxx:50-66,120-136) */
static void terminal_linearize(oracle_unocp_t* o, int with_hessian) {
  const oracle_problem_t* p = &o->p;
  const split_solution_t* s = &o->s[o->N];
  for (int j = 0; j < NV; ++j) {
    o->t_lq[j] = 0; o->t_lv[j] = 0;
    o->t_lq[j] += p->qf_weight[j] * (s->q[j] - p->q_ref[j]);
    o->t_lv[j] += p->vf_weight[j] * (s->v[j] - p->v_ref[j]);
  }
  task_eval_t te;
  if (p->task_enabled) {   /* TimeVaryingTaskSpace6DCost::computeTerminalCostDerivatives at t + T */
    task_evaluate(s->q, o->task_ref + (size_t)o->N * 12, &te, 1, p->task_enabled);
    task_add_gradient(&te, p->task_qf_weight, 1.0, 0, o->t_lq);
  }
  for (int j = 0; j < NV; ++j) {
    o->t_lq[j] -= s->lmd[j];
    o->t_lv[j] -= s->gmm[j];
  }
  if (with_hessian) {
    memset(o->t_Qqq, 0, sizeof(o->t_Qqq));
    memset(o->t_Qvv, 0, sizeof(o->t_Qvv));
    for (int j = 0; j < NV; ++j) {
      o->t_Qqq[j * NV + j] += p->qf_weight[j];
      o->t_Qvv[j * NV + j] += p->vf_weight[j];
    }
    if (p->task_enabled) task_add_hessian(&te, p->task_qf_weight, 1.0, 0, o->t_Qqq);
  }
}

/* UnOCPSolver::updateSolution (:73-134) */
void oracle_unocp_update_solution(oracle_unocp_t* o, double t, const double* q, const double* v,
                                  int line_search) {
  (void)t; /* ConfigurationSpaceCost is time-invariant */
  const int N = o->N;
  const double dt = o->dt;
#pragma omp parallel for num_threads(o->stage_threads) if (o->stage_threads > 1)
  for (int i = 0; i <= N; ++i) {
    if (i < N) split_unocp_linearize(&o->p, dt, &o->s[i], &o->s[i + 1], &o->st[i], o->task_ref + (size_t)i * 12);
    else terminal_linearize(o, 1);
  }
  /* UnRiccatiRecursion::backwardRiccatiRecursionTerminal (src/unocp/unriccati_recursion.cpp:39-47):
   * Pqv of the terminal stage stays zero as allocated */
  riccati_t* rN = &o->ric[N];
  memcpy(rN->Pqq, o->t_Qqq, sizeof(rN->Pqq));
  memcpy(rN->Pvv, o->t_Qvv, sizeof(rN->Pvv));
  memset(rN->Pqv, 0, sizeof(rN->Pqv)); memset(rN->Pvq, 0, sizeof(rN->Pvq));
  for (int j = 0; j < NV; ++j) { rN->sq[j] = -o->t_lq[j]; rN->sv[j] = -o->t_lv[j]; }
  for (int i = N - 1; i >= 0; --i) riccati_backward_stage(&o->ric[i + 1], dt, &o->st[i], &o->ric[i]);
  for (int j = 0; j < NV; ++j) {
    o->d[0].dq[j] = q[j] - o->s[0].q[j];
    o->d[0].dv[j] = v[j] - o->s[0].v[j];
  }
  /* forwardRiccatiRecursion (split_unriccati_factorizer.hxx:49-57) */
  for (int i = 0; i < N; ++i) {
    split_direction_t* d = &o->d[i];
    split_direction_t* dn = &o->d[i + 1];
    const stage_t* st = &o->st[i];
    for (int r = 0; r < NV; ++r) {
      double acc = 0;
      for (int c = 0; c < NV; ++c) acc = fma(st->K[c * NV + r], d->dq[c], acc);
      for (int c = 0; c < NV; ++c) acc = fma(st->K[(NV + c) * NV + r], d->dv[c], acc);
      d->da[r] = acc + st->k[r];
    }
    for (int j = 0; j < NV; ++j) {
      dn->dq[j] = st->uFq[j] + d->dq[j];
      dn->dv[j] = st->uFv[j] + d->dv[j];
      dn->dq[j] = fma(dt, d->dv[j], dn->dq[j]);
      dn->dv[j] = fma(dt, d->da[j], dn->dv[j]);
    }
  }
  double primal = 1.0, dual = 1.0;
#pragma omp parallel for num_threads(o->stage_threads) if (o->stage_threads > 1)
  for (int i = 0; i <= N; ++i) {
    /* computeCostateDirection (:60-68) */
    const riccati_t* r = &o->ric[i];
    split_direction_t* d = &o->d[i];
    for (int j = 0; j < NV; ++j) {
      double t1 = 0, t2 = 0, t3 = 0, t4 = 0;
      for (int k = 0; k < NV; ++k) {
        t1 = fma(r->Pqq[k * NV + j], d->dq[k], t1);
        t2 = fma(r->Pqv[k * NV + j], d->dv[k], t2);
        t3 = fma(r->Pqv[j * NV + k], d->dq[k], t3);   /* Pqv^T dq */
        t4 = fma(r->Pvv[k * NV + j], d->dv[k], t4);
      }
      d->dlmd[j] = t1; d->dlmd[j] += t2; d->dlmd[j] -= r->sq[j];
      d->dgmm[j] = t3; d->dgmm[j] += t4; d->dgmm[j] -= r->sv[j];
    }
    if (i < N) split_unocp_condensed_direction(&o->st[i], dt, d);
  }
  for (int i = 0; i < N; ++i) {
    const double ps = max_slack_step(&o->p, &o->st[i]);
    const double ds = max_dual_step(&o->p, &o->st[i]);
    if (ps < primal) primal = ps;
    if (ds < dual) dual = ds;
  }
  o->max_primal_step = primal;
  if (line_search) primal = line_search_step(o, primal);
  o->primal_step = primal;
  o->dual_step = dual;
#pragma omp parallel for num_threads(o->stage_threads) if (o->stage_threads > 1)
  for (int i = 0; i <= N; ++i) {
    split_solution_t* s = &o->s[i];
    const split_direction_t* d = &o->d[i];
    for (int j = 0; j < NV; ++j) {
      s->lmd[j] = fma(primal, d->dlmd[j], s->lmd[j]);
      s->gmm[j] = fma(primal, d->dgmm[j], s->gmm[j]);
      s->q[j] = fma(primal, d->dq[j], s->q[j]);
      s->v[j] = fma(primal, d->dv[j], s->v[j]);
    }
    if (i < N) {
      for (int j = 0; j < NV; ++j) {
        s->a[j] = fma(primal, d->da[j], s->a[j]);
        s->u[j] = fma(primal, d->du[j], s->u[j]);
        s->beta[j] = fma(primal, d->dbeta[j], s->beta[j]);
      }
      stage_t* st = &o->st[i];
      for (int c = 0; c < NC; ++c) {
        if (!st->active[c]) continue;
        for (int j = 0; j < NV; ++j) {
          st->c[c].slack[j] = fma(primal, st->c[c].dslack[j], st->c[c].slack[j]);
          st->c[c].dual[j] = fma(dual, st->c[c].ddual[j], st->c[c].dual[j]);
        }
      }
    }
  }
}

/* UnOCPSolver::computeKKTResidual (:205-225) */
void oracle_unocp_compute_kkt_residual(oracle_unocp_t* o, double t, const double* q, const double* v) {
  (void)t; (void)q; (void)v; /* q_prev only matters for a floating base; x0 does not enter the residual */
#pragma omp parallel for num_threads(o->stage_threads) if (o->stage_threads > 1)
  for (int i = 0; i <= o->N; ++i) {
    if (i < o->N) split_unocp_kkt_residual(&o->p, o->dt, &o->s[i], &o->s[i + 1], &o->st[i], o->task_ref + (size_t)i * 12);
    else terminal_linearize(o, 0);
  }
}

/* UnOCPSolver::KKTError (:190-202) */
double oracle_unocp_kkt_error(oracle_unocp_t* o) {
  double e = 0;
  for (int i = 0; i < o->N; ++i) e += split_unocp_sqnorm(&o->st[i], o->dt);
  e += sqnorm(o->t_lq) + sqnorm(o->t_lv);  /* TerminalOCP::squaredNormKKTResidual (terminal_ocp.hxx:139-144) */
  return sqrt(e);
}

void oracle_unocp_clear_line_search_filter(oracle_unocp_t* o) { o->filter.n = 0; }

/* UnOCPSolver::isCurrentSolutionFeasible (:228-237) */
int oracle_unocp_is_feasible(oracle_unocp_t* o) {
  for (int i = 0; i < o->N; ++i)
    for (int c = 0; c < NC; ++c) {
      if (!o->st[i].active[c]) continue;
      for (int j = 0; j < NV; ++j)
        if (con_margin(&o->p, c, &o->s[i], j) < 0) return 0;
    }
  return 1;
}

int oracle_unocp_get_solution(const oracle_unocp_t* o, const char* name, double* out) {
  const int full = !strcmp(name, "lmd") || !strcmp(name, "gmm") || !strcmp(name, "q") || !strcmp(name, "v");
  const int n = full ? o->N + 1 : o->N;
  for (int i = 0; i < n; ++i) {
    const double* src;
    if (!strcmp(name, "lmd")) src = o->s[i].lmd;
    else if (!strcmp(name, "gmm")) src = o->s[i].gmm;
    else if (!strcmp(name, "q")) src = o->s[i].q;
    else if (!strcmp(name, "v")) src = o->s[i].v;
    else if (!strcmp(name, "a")) src = o->s[i].a;
    else if (!strcmp(name, "u")) src = o->s[i].u;
    else if (!strcmp(name, "beta")) src = o->s[i].beta;
    else return -1;
    memcpy(out + i * NV, src, sizeof(double) * NV);
  }
  return n;
}

int oracle_unocp_get_direction(const oracle_unocp_t* o, const char* name, double* out) {
  const int full = !strcmp(name, "dlmd") || !strcmp(name, "dgmm") || !strcmp(name, "dq") || !strcmp(name, "dv");
  const int n = full ? o->N + 1 : o->N;
  for (int i = 0; i < n; ++i) {
    const double* src;
    if (!strcmp(name, "dlmd")) src = o->d[i].dlmd;
    else if (!strcmp(name, "dgmm")) src = o->d[i].dgmm;
    else if (!strcmp(name, "dq")) src = o->d[i].dq;
    else if (!strcmp(name, "dv")) src = o->d[i].dv;
    else if (!strcmp(name, "da")) src = o->d[i].da;
    else if (!strcmp(name, "du")) src = o->d[i].du;
    else if (!strcmp(name, "dbeta")) src = o->d[i].dbeta;
    else return -1;
    memcpy(out + i * NV, src, sizeof(double) * NV);
  }
  return n;
}

int oracle_unocp_get_constraint_data(const oracle_unocp_t* o, const char* name, double* out) {
  const int acc = !strncmp(name, "acc_", 4);
  const int c0 = acc ? C_ACC_LO : 0, nc = acc ? 2 : ORACLE_NC;
  if (acc) name += 4;
  for (int i = 0; i < o->N; ++i)
    for (int c = c0; c < c0 + nc; ++c) {
      const cdata_t* d = &o->st[i].c[c];
      const double* src;
      if (!strcmp(name, "slack")) src = d->slack;
      else if (!strcmp(name, "dual")) src = d->dual;
      else if (!strcmp(name, "residual")) src = d->residual;
      else if (!strcmp(name, "duality")) src = d->duality;
      else if (!strcmp(name, "dslack")) src = d->dslack;
      else if (!strcmp(name, "ddual")) src = d->ddual;
      else return -1;
      double* dst = out + (i * nc + c - c0) * NV;
      if (o->st[i].active[c]) memcpy(dst, src, sizeof(double) * NV);
      else memset(dst, 0, sizeof(double) * NV);
    }
  return o->N;
}

void oracle_unocp_get_step_sizes(const oracle_unocp_t* o, double* out) {
  out[0] = o->primal_step; out[1] = o->dual_step; out[2] = o->max_primal_step;
}

void oracle_unocp_get_unkkt(const oracle_unocp_t* o, int stage, double* Q, double* res) {
  const stage_t* st = &o->st[stage];
  const int D = 3 * NV;
  memset(Q, 0, sizeof(double) * D * D);
  const double* blk[3][3] = {{st->uQaa, st->uQaq, st->uQav}, {NULL, st->uQqq, st->uQqv}, {NULL, st->uQvq, st->uQvv}};
  for (int br = 0; br < 3; ++br)
    for (int bc = 0; bc < 3; ++bc) {
      if (!blk[br][bc]) continue;
      for (int c = 0; c < NV; ++c)
        for (int r = 0; r < NV; ++r) Q[(bc * NV + c) * D + br * NV + r] = blk[br][bc][c * NV + r];
    }
  memcpy(res, st->uFq, sizeof(double) * NV);
  memcpy(res + NV, st->uFv, sizeof(double) * NV);
  memcpy(res + 2 * NV, st->ula, sizeof(double) * NV);
  memcpy(res + 3 * NV, st->ulq, sizeof(double) * NV);
  memcpy(res + 4 * NV, st->ulv, sizeof(double) * NV);
}

void oracle_unocp_get_riccati(const oracle_unocp_t* o, int stage, double* Pqq, double* Pqv, double* Pvv,
                              double* sq, double* sv, double* K, double* k) {
  const riccati_t* r = &o->ric[stage];
  memcpy(Pqq, r->Pqq, sizeof(r->Pqq)); memcpy(Pqv, r->Pqv, sizeof(r->Pqv)); memcpy(Pvv, r->Pvv, sizeof(r->Pvv));
  memcpy(sq, r->sq, sizeof(r->sq)); memcpy(sv, r->sv, sizeof(r->sv));
  if (stage < o->N && K && k) {
    memcpy(K, o->st[stage].K, sizeof(o->st[stage].K));
    memcpy(k, o->st[stage].k, sizeof(o->st[stage].k));
  }
}

/* batch drivers: OpenMP over instances, each instance single-threaded (BASELINE.md mode B) */
void oracle_unocp_batch_update_solution(oracle_unocp_t** os, int batch, double t, const double* q0,
                                        const double* v0, int line_search, int nthreads) {
#pragma omp parallel for num_threads(nthreads) schedule(static)
  for (int b = 0; b < batch; ++b)
    oracle_unocp_update_solution(os[b], t, q0 + (size_t)b * NV, v0 + (size_t)b * NV, line_search);
}

void oracle_unocp_batch_kkt(oracle_unocp_t** os, int batch, double t, const double* q0,
                            const double* v0, double* kkt_out, int nthreads) {
#pragma omp parallel for num_threads(nthreads) schedule(static)
  for (int b = 0; b < batch; ++b) {
    oracle_unocp_compute_kkt_residual(os[b], t, q0 + (size_t)b * NV, v0 + (size_t)b * NV);
    kkt_out[b] = oracle_unocp_kkt_error(os[b]);
  }
}

/* batch getter of the test harness: which = 0 solution, 1 direction; out[batch][(N+1)*NV] (rows beyond the field's
 * stage count are left untouched); returns the number of stages of the field */
int oracle_unocp_batch_get(oracle_unocp_t** os, int batch, int which, const char* name, double* out) {
  int n = 0;
  for (int b = 0; b < batch; ++b) {
    double* dst = out + (size_t)b * (os[b]->N + 1) * NV;
    n = which ? oracle_unocp_get_direction(os[b], name, dst) : oracle_unocp_get_solution(os[b], name, dst);
    if (n < 0) return n;
  }
  return n;
}
void oracle_unocp_batch_step_sizes(oracle_unocp_t** os, int batch, double* out) {
  for (int b = 0; b < batch; ++b) oracle_unocp_get_step_sizes(os[b], out + 3 * (size_t)b);
}

/* ========================================================================================== */
/* UnParNMPCSolver (src/unocp/unparnmpc_solver.cpp, src/unocp/unbackward_correction.cpp,       */
/* unocp/split_unparnmpc.hxx, terminal_unparnmpc.hxx, split_unbackward_correction.hxx,         */
/* split_unkkt_matrix_inverter.hxx).  Stages 1..N are stored at index 0..N-1 (SURVEY A.6).     */
/* ========================================================================================== */
#define NX (2 * NV)        /* 14 */
#define NQ3 (3 * NV)       /* 21 */
#define NK (5 * NV)        /* 35 */

struct oracle_unparnmpc {
  oracle_problem_t p;
  int N;
  double dt;
  split_solution_t* s;       /* N */
  split_solution_t* s_new;   /* N */
  split_direction_t* d;      /* N: du doubles as "da" during the corrections, like the reference */
  stage_t* st;               /* N */
  double* KKTinv;            /* N x 35 x 35, column-major; order [lmd,gmm | a,q,v] */
  double* aux;               /* N x 14 x 14, column-major */
  double* xres;              /* N x 14 */
  double primal_step, dual_step, max_primal_step;
  filter_t filter;
  split_solution_t* s_try;
  double* task_ref;          /* (N+1) x 12: rows 0..N-1 = stage times, row N = line-search time of the last stage */
  int chol_info;             /* first non-zero LLT info of the last updateSolution (0 = all factorizations succeeded) */
};

oracle_unparnmpc_t* oracle_unparnmpc_create(const oracle_problem_t* p) {
  if (p->N <= 0 || !(p->T > 0)) return NULL;
  oracle_unparnmpc_t* o = (oracle_unparnmpc_t*)calloc(1, sizeof(*o));
  o->p = *p;
  o->N = p->N;
  o->dt = p->T / p->N;
  o->s = (split_solution_t*)calloc(o->N, sizeof(split_solution_t));
  o->s_new = (split_solution_t*)calloc(o->N, sizeof(split_solution_t));
  o->s_try = (split_solution_t*)calloc(o->N, sizeof(split_solution_t));
  o->d = (split_direction_t*)calloc(o->N, sizeof(split_direction_t));
  o->st = (stage_t*)calloc(o->N, sizeof(stage_t));
  o->KKTinv = (double*)calloc((size_t)o->N * NK * NK, sizeof(double));
  o->aux = (double*)calloc((size_t)o->N * NX * NX, sizeof(double));
  o->xres = (double*)calloc((size_t)o->N * NX, sizeof(double));
  o->task_ref = (double*)calloc((size_t)(o->N + 1) * 12, sizeof(double));
  for (int i = 0; i <= o->N; ++i) o->task_ref[i * 12] = o->task_ref[i * 12 + 4] = o->task_ref[i * 12 + 8] = 1.0;
  oracle_unparnmpc_init_constraints(o);
  return o;
}

void oracle_unparnmpc_destroy(oracle_unparnmpc_t* o) {
  if (!o) return;
  free(o->s); free(o->s_new); free(o->s_try); free(o->d); free(o->st); free(o->KKTinv); free(o->aux); free(o->xres);
  free(o->task_ref);
  free(o);
}

/* UnParNMPCSolver::initConstraints (:54-66): stage index i uses time step i+1 */
void oracle_unparnmpc_init_constraints(oracle_unparnmpc_t* o) {
  for (int i = 0; i < o->N; ++i) {
    set_active(&o->p, i + 1, o->st[i].active);
    set_slack_and_dual(&o->p, &o->st[i], &o->s[i]);
  }
}

int oracle_unparnmpc_set_solution(oracle_unparnmpc_t* o, const char* name, const double* value) {
  for (int i = 0; i < o->N; ++i) {
    double* dst;
    if (!strcmp(name, "q")) dst = o->s[i].q;
    else if (!strcmp(name, "v")) dst = o->s[i].v;
    else if (!strcmp(name, "a")) dst = o->s[i].a;
    else if (!strcmp(name, "u")) dst = o->s[i].u;
    else return -1;
    memcpy(dst, value, sizeof(double) * NV);
  }
  oracle_unparnmpc_init_constraints(o);
  return 0;
}

/* UnBackwardCorrection::initAuxMat (:55-64): every aux_mat = terminal cost Hessian (Qxx) */
void oracle_unparnmpc_init_backward_correction(oracle_unparnmpc_t* o, double t) {
  (void)t;
  /* TerminalUnParNMPC::computeTerminalCostHessian (terminal_unparnmpc.hxx:230-241) at s[N-1], time t + T */
  double Qqq[NN];
  memset(Qqq, 0, sizeof(Qqq));
  for (int j = 0; j < NV; ++j) Qqq[j * NV + j] += o->p.qf_weight[j];
  if (o->p.task_enabled) {
    task_eval_t te;
    task_evaluate(o->s[o->N - 1].q, o->task_ref + (size_t)(o->N - 1) * 12, &te, 1, o->p.task_enabled);
    task_add_hessian(&te, o->p.task_qf_weight, 1.0, 0, Qqq);
  }
  for (int i = 0; i < o->N; ++i) {
    double* A = o->aux + (size_t)i * NX * NX;
    memset(A, 0, sizeof(double) * NX * NX);
    for (int c = 0; c < NV; ++c)
      for (int r = 0; r < NV; ++r) A[c * NX + r] = Qqq[c * NV + r];
    for (int j = 0; j < NV; ++j) A[(NV + j) * NX + NV + j] = o->p.vf_weight[j];
  }
}

/* gradient part shared by SplitUnParNMPC::linearizeOCP (split_unparnmpc.hxx:69-101) /
 * computeKKTResidual (:141-163) and the TerminalUnParNMPC twins (terminal_unparnmpc.hxx:70-102);
 * backward Euler: stateequation::linearizeBackwardEuler[Terminal] (state_equation.hxx:111-167,224-236) */
static void parnmpc_residual_common(const oracle_problem_t* p, double dt, const double* q_prev, const double* v_prev,
                                    const split_solution_t* s, const split_solution_t* sn, stage_t* st,
                                    const double* ref) {
  const int terminal = (sn == NULL);
  memset(st->lq, 0, sizeof(double) * NV); memset(st->lv, 0, sizeof(double) * NV);
  memset(st->la, 0, sizeof(double) * NV); memset(st->lu, 0, sizeof(double) * NV);
  stage_cost_derivatives(p, dt, s, st, ref);
  if (terminal) {   /* + computeTerminalCostDerivatives at the same time t + T */
    for (int j = 0; j < NV; ++j) {
      st->lq[j] += p->qf_weight[j] * (s->q[j] - p->q_ref[j]);
      st->lv[j] += p->vf_weight[j] * (s->v[j] - p->v_ref[j]);
    }
    if (p->task_enabled) task_add_gradient(&st->te, p->task_qf_weight, 1.0, 0, st->lq);
  }
  augment_dual_residual(st, dt);
  for (int j = 0; j < NV; ++j) {
    st->Fq[j] = fma(dt, s->v[j], q_prev[j] - s->q[j]);
    st->Fv[j] = fma(dt, s->a[j], v_prev[j] - s->v[j]);
  }
  for (int j = 0; j < NV; ++j) {
    if (terminal) {
      st->lq[j] -= s->lmd[j];
      st->lv[j] += fma(dt, s->lmd[j], -s->gmm[j]);
    } else {
      st->lq[j] += sn->lmd[j] - s->lmd[j];
      st->lv[j] += fma(dt, s->lmd[j], -s->gmm[j]) + sn->gmm[j];
    }
    st->la[j] = fma(dt, s->gmm[j], st->la[j]);
  }
  rnea_derivatives_impl(s->q, s->v, s->a, st->ID, st->dIDdq, st->dIDdv, st->dIDda);
  for (int j = 0; j < NV; ++j) st->ID[j] -= s->u[j];
  for (int j = 0; j < NV; ++j) {
    double tq = 0, tv = 0, ta = 0;
    for (int k = 0; k < NV; ++k) {
      tq = fma(st->dIDdq[j * NV + k], s->beta[k], tq);
      tv = fma(st->dIDdv[j * NV + k], s->beta[k], tv);
      ta = fma(st->dIDda[j * NV + k], s->beta[k], ta);
    }
    st->lq[j] = fma(dt, tq, st->lq[j]);
    st->lv[j] = fma(dt, tv, st->lv[j]);
    st->la[j] = fma(dt, ta, st->la[j]);
    st->lu[j] = fma(-dt, s->beta[j], st->lu[j]);
  }
}

/* condensing shared with the UnOCP path (unconstrained_dynamics.hxx:68-94) */
static void condense_unconstrained_dynamics(stage_t* st) {
  for (int j = 0; j < NV; ++j) st->lu_condensed[j] = fma(st->Quu[j], st->ID[j], st->lu[j]);
  for (int j = 0; j < NV; ++j) {
    double tq = 0, tv = 0, ta = 0;
    for (int k = 0; k < NV; ++k) {
      tq = fma(st->dIDdq[j * NV + k], st->lu_condensed[k], tq);
      tv = fma(st->dIDdv[j * NV + k], st->lu_condensed[k], tv);
      ta = fma(st->dIDda[j * NV + k], st->lu_condensed[k], ta);
    }
    st->ulq[j] = st->lq[j] + tq;
    st->ulv[j] = st->lv[j] + tv;
    st->ula[j] = st->la[j] + ta;
    st->uFq[j] = st->Fq[j];
    st->uFv[j] = st->Fv[j];
  }
  for (int c = 0; c < NV; ++c)
    for (int r = 0; r < NV; ++r) {
      double qq = 0, qv = 0, vv = 0, aq = 0, av = 0, aa = 0;
      for (int k = 0; k < NV; ++k) {
        const double Dq = st->Quu[k] * st->dIDdq[c * NV + k];
        const double Dv = st->Quu[k] * st->dIDdv[c * NV + k];
        const double Da = st->Quu[k] * st->dIDda[c * NV + k];
        qq = fma(st->dIDdq[r * NV + k], Dq, qq);
        qv = fma(st->dIDdq[r * NV + k], Dv, qv);
        vv = fma(st->dIDdv[r * NV + k], Dv, vv);
        aq = fma(st->dIDda[r * NV + k], Dq, aq);
        av = fma(st->dIDda[r * NV + k], Dv, av);
        aa = fma(st->dIDda[r * NV + k], Da, aa);
      }
      st->uQqq[c * NV + r] = qq + st->Qqq[c * NV + r];
      st->uQqv[c * NV + r] = qv;
      st->uQvv[c * NV + r] = vv + (r == c ? st->Qvv[r] : 0.0);
      st->uQaq[c * NV + r] = aq;
      st->uQav[c * NV + r] = av;
      st->uQaa[c * NV + r] = aa + (r == c ? st->Qaa[r] : 0.0);
    }
}

static void parnmpc_linearize(const oracle_problem_t* p, double dt, const double* q_prev, const double* v_prev,
                              const split_solution_t* s, const split_solution_t* sn, stage_t* st, const double* ref) {
  const int terminal = (sn == NULL);
  memset(st->Qqq, 0, sizeof(st->Qqq));
  memset(st->Qvv, 0, sizeof(st->Qvv)); memset(st->Qaa, 0, sizeof(st->Qaa)); memset(st->Quu, 0, sizeof(st->Quu));
  parnmpc_residual_common(p, dt, q_prev, v_prev, s, sn, st, ref);
  stage_cost_hessian(p, dt, st);
  if (terminal) {
    for (int j = 0; j < NV; ++j) {
      st->Qqq[j * NV + j] += p->qf_weight[j];
      st->Qvv[j] += p->vf_weight[j];
    }
    if (p->task_enabled) task_add_hessian(&st->te, p->task_qf_weight, 1.0, 0, st->Qqq);
  }
  condense_slack_and_dual(p, st, s, dt);
  condense_unconstrained_dynamics(st);
}

/* SplitUnKKTMatrixInverter::invert (split_unkkt_matrix_inverter.hxx:40-79) on the 21x21 Q (block
 * order a,q,v) -> 35x35 inverse of [[0 F],[F^T Q]], order [lmd,gmm | a,q,v]; all column-major */
static int invert_unkkt(double dt, const double* Q, double* Kinv) {
  double L[NQ3 * NQ3], rd[NQ3], Qinv[NQ3 * NQ3], e[NQ3], x[NQ3];
  int info = llt_lower(Q, NQ3, L, rd);
  for (int c = 0; c < NQ3; ++c) {
    for (int k = 0; k < NQ3; ++k) e[k] = (k == c) ? 1.0 : 0.0;
    llt_solve_desc(L, rd, NQ3, e, x);
    for (int r = 0; r < NQ3; ++r) Qinv[c * NQ3 + r] = x[r];
  }
  /* FQinv (14 x 21): rows Fq: -Qinv[q rows] + dt Qinv[v rows]; rows Fv: dt Qinv[a rows] - Qinv[v rows] */
  double FQ[NX * NQ3];
  for (int c = 0; c < NQ3; ++c)
    for (int r = 0; r < NV; ++r) {
      FQ[c * NX + r] = fma(dt, Qinv[c * NQ3 + 2 * NV + r], -Qinv[c * NQ3 + NV + r]);
      FQ[c * NX + NV + r] = fma(dt, Qinv[c * NQ3 + r], -Qinv[c * NQ3 + 2 * NV + r]);
    }
  /* S = FQinv F^T (14 x 14): S[:, q-part] = -FQ[:, q cols] + dt FQ[:, v cols]; S[:, v-part] = dt FQ[:, a cols] - FQ[:, v cols] */
  double S[NX * NX];
  for (int c = 0; c < NV; ++c)
    for (int r = 0; r < NX; ++r) {
      S[c * NX + r] = fma(dt, FQ[(2 * NV + c) * NX + r], -FQ[(NV + c) * NX + r]);
      S[(NV + c) * NX + r] = fma(dt, FQ[c * NX + r], -FQ[(2 * NV + c) * NX + r]);
    }
  double LS[NX * NX], rdS[NX], Sinv[NX * NX];
  const int info2 = llt_lower(S, NX, LS, rdS);
  if (!info && info2) info = 100 + info2;
  for (int c = 0; c < NX; ++c) {
    for (int k = 0; k < NX; ++k) e[k] = (k == c) ? 1.0 : 0.0;
    llt_solve_desc(LS, rdS, NX, e, x);
    for (int r = 0; r < NX; ++r) Sinv[c * NX + r] = x[r];
  }
  /* top-left = -Sinv */
  for (int c = 0; c < NX; ++c)
    for (int r = 0; r < NX; ++r) Kinv[c * NK + r] = -Sinv[c * NX + r];
  /* top-right = -(top-left * FQinv)  (14 x 21) */
  double TR[NX * NQ3];
  for (int c = 0; c < NQ3; ++c)
    for (int r = 0; r < NX; ++r) {
      double t = 0;
      for (int k = 0; k < NX; ++k) t = fma(Kinv[k * NK + r], FQ[c * NX + k], t);
      TR[c * NX + r] = -t;
      Kinv[(NX + c) * NK + r] = -t;
      Kinv[r * NK + NX + c] = -t;        /* bottom-left = top-right^T */
    }
  /* bottom-right = Qinv - TR^T S TR */
  double STR[NX * NQ3];
  for (int c = 0; c < NQ3; ++c)
    for (int r = 0; r < NX; ++r) {
      double t = 0;
      for (int k = 0; k < NX; ++k) t = fma(S[k * NX + r], TR[c * NX + k], t);
      STR[c * NX + r] = t;
    }
  for (int c = 0; c < NQ3; ++c)
    for (int r = 0; r < NQ3; ++r) {
      double t = 0;
      for (int k = 0; k < NX; ++k) t = fma(TR[r * NX + k], STR[c * NX + k], t);
      Kinv[(NX + c) * NK + NX + r] = Qinv[c * NQ3 + r] - t;
    }
  return info;
}

/* assemble the 21x21 Q (order a,q,v) of a stage as SplitUnBackwardCorrection::coarseUpdate sees it
 * (split_unbackward_correction.hxx:37-53): Qxx += aux_next, then Qvq = Qqv^T, Qxa = Qax^T */
static void assemble_parnmpc_Q(const stage_t* st, const double* aux_next, double* Q) {
  for (int c = 0; c < NV; ++c)
    for (int r = 0; r < NV; ++r) {
      double qq = st->uQqq[c * NV + r], qv = st->uQqv[c * NV + r], vv = st->uQvv[c * NV + r];
      if (aux_next) {
        qq += aux_next[c * NX + r];
        qv += aux_next[(NV + c) * NX + r];
        vv += aux_next[(NV + c) * NX + NV + r];
      }
      Q[c * NQ3 + r] = st->uQaa[c * NV + r];                       /* aa */
      Q[(NV + c) * NQ3 + r] = st->uQaq[c * NV + r];                /* aq */
      Q[(2 * NV + c) * NQ3 + r] = st->uQav[c * NV + r];            /* av */
      Q[r * NQ3 + NV + c] = st->uQaq[c * NV + r];                  /* qa = aq^T */
      Q[r * NQ3 + 2 * NV + c] = st->uQav[c * NV + r];              /* va = av^T */
      Q[(NV + c) * NQ3 + NV + r] = qq;                             /* qq */
      Q[(2 * NV + c) * NQ3 + NV + r] = qv;                         /* qv */
      Q[(NV + r) * NQ3 + 2 * NV + c] = qv;                         /* vq = qv^T */
      Q[(2 * NV + c) * NQ3 + 2 * NV + r] = vv;                     /* vv */
    }
}


/* UnLineSearch::computeCostAndViolation(UnParNMPC&, ...) (src/line_search/unline_search.cpp:87-122):
 * SplitUnParNMPC::stageCost / constraintViolation (unocp/split_unparnmpc.hxx:177-224), TerminalUnParNMPC twins
 * (terminal_unparnmpc.hxx:196-227).  `s` is the current or the trial solution; the previous state of stage i
 * is s[i-1] of THAT solution (x0 for i = 0).  The last stage is evaluated at t + N dt (:113-119), row N of the
 * task reference table. */
static void parnmpc_cost_and_violation(oracle_unparnmpc_t* o, const double* q, const double* v,
                                       const split_solution_t* s, double alpha, double* cost, double* viol) {
  const oracle_problem_t* p = &o->p;
  const int N = o->N;
  const double dt = o->dt;
  double cs = 0, vs = 0;
  for (int i = 0; i < N; ++i) {
    stage_t* st = &o->st[i];
    const int last = (i == N - 1);
    const double* ref = o->task_ref + (size_t)(last ? N : i) * 12;
    double c = stage_cost(p, dt, &s[i]);
    if (p->task_enabled) c += task_stage_cost(p, dt, s[i].q, ref);
    if (last) {
      double tc = terminal_cost(p, &s[i]);
      if (p->task_enabled) tc += task_terminal_cost(p, s[i].q, ref);
      c += tc;
    }
    double bar = 0;
    for (int k = 0; k < NC; ++k) {
      if (!st->active[k]) continue;
      double lg = 0;
      for (int j = 0; j < NV; ++j) {
        const double sl = alpha > 0 ? fma(alpha, st->c[k].dslack[j], st->c[k].slack[j]) : st->c[k].slack[j];
        lg += canon_log(sl);
      }
      bar += -p->barrier * lg;
    }
    c += dt * bar;
    cs += c;
    /* constraintViolation: overwrites residual, Fx and ID of the stage, as the reference does */
    const double* qp = i == 0 ? q : s[i - 1].q;
    const double* vp = i == 0 ? v : s[i - 1].v;
    compute_primal_dual_residual(p, st, &s[i]);
    for (int j = 0; j < NV; ++j) {
      st->Fq[j] = fma(dt, s[i].v[j], qp[j] - s[i].q[j]);
      st->Fv[j] = fma(dt, s[i].a[j], vp[j] - s[i].v[j]);
    }
    rnea_derivatives_impl(s[i].q, s[i].v, s[i].a, st->ID, NULL, NULL, NULL);
    for (int j = 0; j < NV; ++j) st->ID[j] -= s[i].u[j];
    double vi = 0;
    vi += l1norm(st->Fq) + l1norm(st->Fv);
    vi += dt * l1norm(st->ID);
    double c1 = 0;
    for (int k = 0; k < NC; ++k)
      if (st->active[k]) c1 += l1norm(st->c[k].residual);
    vi += dt * c1;
    vs += vi;
  }
  *cost = cs; *viol = vs;
}

/* UnLineSearch::computeStepSize<UnParNMPC> (line_search/unline_search.hpp:62-91) */
static double parnmpc_line_search_step(oracle_unparnmpc_t* o, const double* q, const double* v, double max_primal) {
  double cost, viol;
  if (o->filter.n == 0) {
    parnmpc_cost_and_violation(o, q, v, o->s, 0.0, &cost, &viol);
    filter_augment(&o->filter, cost, viol);
  }
  const double min_step = 0.05, rate = 0.75;
  double alpha = max_primal;
  while (alpha > min_step) {
    for (int i = 0; i < o->N; ++i) {
      split_solution_t* t = &o->s_try[i];
      for (int j = 0; j < NV; ++j) {
        t->q[j] = fma(alpha, o->d[i].dq[j], o->s[i].q[j]);
        t->v[j] = fma(alpha, o->d[i].dv[j], o->s[i].v[j]);
        t->a[j] = fma(alpha, o->d[i].da[j], o->s[i].a[j]);
        t->u[j] = fma(alpha, o->d[i].du[j], o->s[i].u[j]);
      }
    }
    parnmpc_cost_and_violation(o, q, v, o->s_try, alpha, &cost, &viol);
    if (filter_is_accepted(&o->filter, cost, viol)) {
      filter_augment(&o->filter, cost, viol);
      break;
    }
    alpha *= rate;
  }
  return alpha > min_step ? alpha : min_step;
}

/* UnParNMPCSolver::updateSolution (:74-102) */
void oracle_unparnmpc_update_solution(oracle_unparnmpc_t* o, double t, const double* q, const double* v,
                                      int line_search) {
  (void)t;
  const int N = o->N;
  const double dt = o->dt;
  const oracle_problem_t* p = &o->p;
  o->chol_info = 0;
  /* UnBackwardCorrection::coarseUpdate (:67-97) */
  for (int i = 0; i < N; ++i) {
    const double* qp = i == 0 ? q : o->s[i - 1].q;
    const double* vp = i == 0 ? v : o->s[i - 1].v;
    stage_t* st = &o->st[i];
    parnmpc_linearize(p, dt, qp, vp, &o->s[i], i < N - 1 ? &o->s[i + 1] : NULL, st, o->task_ref + (size_t)i * 12);
    double Q[NQ3 * NQ3];
    assemble_parnmpc_Q(st, i < N - 1 ? o->aux + (size_t)(i + 1) * NX * NX : NULL, Q);
    double* Kinv = o->KKTinv + (size_t)i * NK * NK;
    const int info = invert_unkkt(dt, Q, Kinv);
    if (info && !o->chol_info) o->chol_info = 1000 * (i + 1) + info;
    /* d = KKT^-1 residual, residual order [Fq,Fv,la,lq,lv]; d order [dlmd,dgmm,du(=da),dq,dv] */
    double res[NK], dd[NK];
    memcpy(res, st->uFq, sizeof(double) * NV); memcpy(res + NV, st->uFv, sizeof(double) * NV);
    memcpy(res + 2 * NV, st->ula, sizeof(double) * NV); memcpy(res + 3 * NV, st->ulq, sizeof(double) * NV);
    memcpy(res + 4 * NV, st->ulv, sizeof(double) * NV);
    for (int r = 0; r < NK; ++r) {
      double acc = 0;
      for (int c = 0; c < NK; ++c) acc = fma(Kinv[c * NK + r], res[c], acc);
      dd[r] = acc;
    }
    split_direction_t* d = &o->d[i];
    split_solution_t* sn = &o->s_new[i];
    const split_solution_t* s = &o->s[i];
    for (int j = 0; j < NV; ++j) {
      d->dlmd[j] = dd[j]; d->dgmm[j] = dd[NV + j]; d->du[j] = dd[2 * NV + j];
      d->dq[j] = dd[3 * NV + j]; d->dv[j] = dd[4 * NV + j];
      sn->lmd[j] = s->lmd[j] - d->dlmd[j];
      sn->gmm[j] = s->gmm[j] - d->dgmm[j];
      sn->a[j] = s->a[j] - d->du[j];
      sn->q[j] = s->q[j] - d->dq[j];
      sn->v[j] = s->v[j] - d->dv[j];
    }
  }
  /* UnBackwardCorrection::backwardCorrection (:100-134) */
  for (int i = N - 2; i >= 0; --i) {          /* backwardCorrectionSerial */
    const double* Kinv = o->KKTinv + (size_t)i * NK * NK;
    double* xr = o->xres + (size_t)i * NX;
    for (int j = 0; j < NV; ++j) {
      xr[j] = o->s_new[i + 1].lmd[j] - o->s[i + 1].lmd[j];
      xr[NV + j] = o->s_new[i + 1].gmm[j] - o->s[i + 1].gmm[j];
    }
    for (int r = 0; r < NX; ++r) {
      double acc = 0;
      for (int c = 0; c < NX; ++c) acc = fma(Kinv[(NK - NX + c) * NK + r], xr[c], acc);
      if (r < NV) o->s_new[i].lmd[r] -= acc; else o->s_new[i].gmm[r - NV] -= acc;
    }
  }
  for (int i = N - 2; i >= 0; --i) {          /* backwardCorrectionParallel */
    const double* Kinv = o->KKTinv + (size_t)i * NK * NK;
    const double* xr = o->xres + (size_t)i * NX;
    for (int r = 0; r < NQ3; ++r) {
      double acc = 0;
      for (int c = 0; c < NX; ++c) acc = fma(Kinv[(NK - NX + c) * NK + NX + r], xr[c], acc);
      if (r < NV) { o->d[i].du[r] = acc; o->s_new[i].a[r] -= acc; }
      else if (r < 2 * NV) { o->d[i].dq[r - NV] = acc; o->s_new[i].q[r - NV] -= acc; }
      else { o->d[i].dv[r - 2 * NV] = acc; o->s_new[i].v[r - 2 * NV] -= acc; }
    }
  }
  for (int i = 1; i < N; ++i) {               /* forwardCorrectionSerial */
    const double* Kinv = o->KKTinv + (size_t)i * NK * NK;
    double* xr = o->xres + (size_t)i * NX;
    for (int j = 0; j < NV; ++j) {
      xr[j] = o->s_new[i - 1].q[j] - o->s[i - 1].q[j];
      xr[NV + j] = o->s_new[i - 1].v[j] - o->s[i - 1].v[j];
    }
    for (int r = 0; r < NX; ++r) {
      double acc = 0;
      for (int c = 0; c < NX; ++c) acc = fma(Kinv[c * NK + NK - NX + r], xr[c], acc);
      if (r < NV) o->s_new[i].q[r] -= acc; else o->s_new[i].v[r - NV] -= acc;
    }
  }
  double primal = 1.0, dual = 1.0;
  for (int i = 0; i < N; ++i) {               /* forwardCorrectionParallel + directions */
    const double* Kinv = o->KKTinv + (size_t)i * NK * NK;
    split_direction_t* d = &o->d[i];
    split_solution_t* sn = &o->s_new[i];
    const split_solution_t* s = &o->s[i];
    if (i > 0) {
      const double* xr = o->xres + (size_t)i * NX;
      for (int r = 0; r < NQ3; ++r) {
        double acc = 0;
        for (int c = 0; c < NX; ++c) acc = fma(Kinv[c * NK + r], xr[c], acc);
        if (r < NV) { d->dlmd[r] = acc; sn->lmd[r] -= acc; }
        else if (r < 2 * NV) { d->dgmm[r - NV] = acc; sn->gmm[r - NV] -= acc; }
        else { d->du[r - 2 * NV] = acc; sn->a[r - 2 * NV] -= acc; }
      }
      double* A = o->aux + (size_t)i * NX * NX;   /* aux_mat = -KKT^-1[0:14, 0:14] */
      for (int c = 0; c < NX; ++c)
        for (int r = 0; r < NX; ++r) A[c * NX + r] = -Kinv[c * NK + r];
    }
    /* SplitUnBackwardCorrection::computeDirection (:113-121) */
    for (int j = 0; j < NV; ++j) {
      d->dlmd[j] = sn->lmd[j] - s->lmd[j];
      d->dgmm[j] = sn->gmm[j] - s->gmm[j];
      d->da[j] = sn->a[j] - s->a[j];
      d->dq[j] = sn->q[j] - s->q[j];
      d->dv[j] = sn->v[j] - s->v[j];
    }
    split_unocp_condensed_direction(&o->st[i], dt, d);
    const double ps = max_slack_step(p, &o->st[i]);
    const double ds = max_dual_step(p, &o->st[i]);
    if (ps < primal) primal = ps;
    if (ds < dual) dual = ds;
  }
  o->max_primal_step = primal;
  if (line_search) primal = parnmpc_line_search_step(o, q, v, primal);
  o->primal_step = primal;
  o->dual_step = dual;
  for (int i = 0; i < N; ++i) {
    split_solution_t* s = &o->s[i];
    const split_direction_t* d = &o->d[i];
    for (int j = 0; j < NV; ++j) {
      s->lmd[j] = fma(primal, d->dlmd[j], s->lmd[j]);
      s->gmm[j] = fma(primal, d->dgmm[j], s->gmm[j]);
      s->q[j] = fma(primal, d->dq[j], s->q[j]);
      s->v[j] = fma(primal, d->dv[j], s->v[j]);
      s->a[j] = fma(primal, d->da[j], s->a[j]);
      s->u[j] = fma(primal, d->du[j], s->u[j]);
      s->beta[j] = fma(primal, d->dbeta[j], s->beta[j]);
    }
    stage_t* st = &o->st[i];
    for (int c = 0; c < NC; ++c) {
      if (!st->active[c]) continue;
      for (int j = 0; j < NV; ++j) {
        st->c[c].slack[j] = fma(primal, st->c[c].dslack[j], st->c[c].slack[j]);
        st->c[c].dual[j] = fma(dual, st->c[c].ddual[j], st->c[c].dual[j]);
      }
    }
  }
}

/* UnParNMPCSolver::computeKKTResidual (:171-192) and KKTError (:157-168) */
void oracle_unparnmpc_compute_kkt_residual(oracle_unparnmpc_t* o, double t, const double* q, const double* v) {
  (void)t;
  for (int i = 0; i < o->N; ++i) {
    const double* qp = i == 0 ? q : o->s[i - 1].q;
    const double* vp = i == 0 ? v : o->s[i - 1].v;
    compute_primal_dual_residual(&o->p, &o->st[i], &o->s[i]);
    parnmpc_residual_common(&o->p, o->dt, qp, vp, &o->s[i], i < o->N - 1 ? &o->s[i + 1] : NULL, &o->st[i],
                            o->task_ref + (size_t)i * 12);
  }
}

double oracle_unparnmpc_kkt_error(oracle_unparnmpc_t* o) {
  double e = 0;
  for (int i = 0; i < o->N; ++i) e += split_unocp_sqnorm(&o->st[i], o->dt);
  return sqrt(e);
}

int oracle_unparnmpc_get_solution(const oracle_unparnmpc_t* o, const char* name, double* out) {
  for (int i = 0; i < o->N; ++i) {
    const double* src;
    if (!strcmp(name, "lmd")) src = o->s[i].lmd;
    else if (!strcmp(name, "gmm")) src = o->s[i].gmm;
    else if (!strcmp(name, "q")) src = o->s[i].q;
    else if (!strcmp(name, "v")) src = o->s[i].v;
    else if (!strcmp(name, "a")) src = o->s[i].a;
    else if (!strcmp(name, "u")) src = o->s[i].u;
    else if (!strcmp(name, "beta")) src = o->s[i].beta;
    else return -1;
    memcpy(out + i * NV, src, sizeof(double) * NV);
  }
  return o->N;
}

int oracle_unparnmpc_get_direction(const oracle_unparnmpc_t* o, const char* name, double* out) {
  for (int i = 0; i < o->N; ++i) {
    const double* src;
    if (!strcmp(name, "dlmd")) src = o->d[i].dlmd;
    else if (!strcmp(name, "dgmm")) src = o->d[i].dgmm;
    else if (!strcmp(name, "dq")) src = o->d[i].dq;
    else if (!strcmp(name, "dv")) src = o->d[i].dv;
    else if (!strcmp(name, "da")) src = o->d[i].da;
    else if (!strcmp(name, "du")) src = o->d[i].du;
    else if (!strcmp(name, "dbeta")) src = o->d[i].dbeta;
    else return -1;
    memcpy(out + i * NV, src, sizeof(double) * NV);
  }
  return o->N;
}

void oracle_unparnmpc_get_step_sizes(const oracle_unparnmpc_t* o, double* out) {
  out[0] = o->primal_step; out[1] = o->dual_step; out[2] = o->max_primal_step;
}

/* parity getter: 35x35 KKT inverse of a stage (column-major) */
void oracle_unparnmpc_get_kkt_inverse(const oracle_unparnmpc_t* o, int stage, double* out) {
  memcpy(out, o->KKTinv + (size_t)stage * NK * NK, sizeof(double) * NK * NK);
}

void oracle_unparnmpc_batch_update_solution(oracle_unparnmpc_t** os, int batch, double t, const double* q0,
                                            const double* v0, int line_search, int nthreads) {
#pragma omp parallel for num_threads(nthreads) schedule(static)
  for (int b = 0; b < batch; ++b)
    oracle_unparnmpc_update_solution(os[b], t, q0 + (size_t)b * NV, v0 + (size_t)b * NV, line_search);
}

void oracle_unparnmpc_batch_kkt(oracle_unparnmpc_t** os, int batch, double t, const double* q0,
                                const double* v0, double* kkt_out, int nthreads) {
#pragma omp parallel for num_threads(nthreads) schedule(static)
  for (int b = 0; b < batch; ++b) {
    oracle_unparnmpc_compute_kkt_residual(os[b], t, q0 + (size_t)b * NV, v0 + (size_t)b * NV);
    kkt_out[b] = oracle_unparnmpc_kkt_error(os[b]);
  }
}

/* parity getter: the 21x21 Q a stage's coarse update inverted is not stored; re-assemble it from
 * the stage data of the last linearisation (aux of the NEXT iteration is already in place, so this
 * is only exact before the first update) -- used by tests through oracle_invert_unkkt instead */
int oracle_invert_unkkt(double dt, const double* Q, double* Kinv) { return invert_unkkt(dt, Q, Kinv); }

int oracle_unparnmpc_chol_info(const oracle_unparnmpc_t* o) { return o->chol_info; }

/* host-sampled reference of the task-space cost: table[(N+1)][12], row i = compute_q_6d_ref at the time of
 * stage index i (UnOCPSolver: t + i dt, row N = t + T; UnParNMPCSolver: t + (i+1) dt, row N-1 = t + T,
 * row N = t + N dt used only by the line search) */
void oracle_unocp_set_task_ref(oracle_unocp_t* o, const double* table) {
  memcpy(o->task_ref, table, sizeof(double) * (size_t)(o->N + 1) * 12);
}
void oracle_unparnmpc_set_task_ref(oracle_unparnmpc_t* o, const double* table) {
  memcpy(o->task_ref, table, sizeof(double) * (size_t)(o->N + 1) * 12);
}

void oracle_unparnmpc_clear_line_search_filter(oracle_unparnmpc_t* o) { o->filter.n = 0; }
