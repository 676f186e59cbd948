// pamg_unstr.cuh -- fully unstructured P1 DG front-ends as sm_100a kernels: the explicit step (unstr_explicit,
// transport_tri_unstr.F90:588-795), the implicit operator in block-CSR (unstr_implicit :214-387 /
// Semi_implicit_direct transport_tri_semi.F90:1607-1764), its Krylov solve, the Petrov-Galerkin stabilisation, trans_rec
// and the batched element-local inverse (FINDInv, matrix_inversion.F90:50-148 == matrices.F90:1618-1716).
//
// One thread per element.  Everything the library owns per element or per face lies in HBM as structure-of-arrays planes
// (vertex coordinates [6][E], neighbour ids / sides [3][E], penalty lengths [3][E], matrix blocks [36][E], block columns
// [4][E] ...), so every load and store of a warp is one contiguous 256-byte span.  The FIELDS keep the reference's
// (nloc, E) layout - it is the ABI and it keeps the two face values of a neighbour inside one 32-byte sector; a warp
// moves its own 32 records (768 contiguous bytes) through shared memory with fully coalesced accesses (warp_load3 /
// warp_store3).  Geometry (tri_det_nlx ShapFun.F90:1414-1454, det_snlx_all :1554-1590) is recomputed in registers from the
// 6 vertex coordinates - cheaper than streaming 19 stored doubles.  The 3x3 / 4x4 / 6x6 local systems live entirely
// in registers (fully unrolled Gauss-Jordan); tensor cores are pointless for blocks this small.
#pragma once
#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>
#include <string>
#include <vector>

#include "pamg.h"
#include "pamg_kernels.cuh"

namespace pamg {

struct UnstrDev {
  int E = 0;
  size_t ld = 0;              // plane stride in elements: 32 x odd >= E.  A power-of-two E (the synthetic meshes) would put the
                              // same element of all 36 matrix planes into one L2 set: ncu showed 1.32 x the stored bytes going
                              // to DRAM in k_assemble_bsr (lines evicted half written); with an odd number of lines between
                              // planes the streams spread over the sets
  double* X = nullptr;        // [6][ld] planes x1, y1, x2, y2, x3, y3
  double* U = nullptr;        // [6][ld] planes u1x, u1y, u2x, u2y, u3x, u3y of the nodal velocity field u_ele(2,3,E)
                              //         (transport_tri_unstr.F90:504-511); null = the uniform velocity of the call
  int32_t* neig = nullptr;    // [3][ld] 1-based, 0 = boundary
  int32_t* nside = nullptr;   // [3][ld] fNeig | swap<<2 (swap: geometric pairing differs from get_unstr_sn2)
  double* pen = nullptr;      // [3][ld] (L/2) / dx of the diffusion face term: half the face length over the centroid distance
                              //         to the neighbour, or over centroid -> edge midpoint on the domain boundary
                              //         (matrices.F90:84-110); times k it is the penalty coefficient of the face
  double* T[2] = {nullptr, nullptr};   // (3, E) like tnew
  double* told = nullptr;
  int cur = 0;
  // implicit operator in block-CSR: 4 blocks of 3x3 per element row (own, face 1, face 2, face 3)
  double* bsr_val = nullptr;   // [36][ld]: plane (block * 9 + row * 3 + col)
  int32_t* bsr_col = nullptr;  // [4][ld] 0-based element of the block column, -1 = no block
  double* dinv = nullptr;      // [9][ld] inverse of the diagonal block (block-Jacobi preconditioner)
  double* mdt = nullptr;       // [E] A/(12 dt): M/dt = mdt (I + J) per element
  double* work = nullptr;      // 9 vectors of 3E doubles for BiCGStab
  double* dots = nullptr;      // device scalars and partial sums of the Krylov solve
  double* dots_host = nullptr; // pinned mirror
  bool assembled = false;
  double* diag0 = nullptr;     // [9][ld] diagonal blocks without stabilisation: copied out of bsr_val when the stabilisation is
                               //         switched on (pamg_implicit_set_stab), not written by every assembly
  double* stab = nullptr;      // [E][9] Petrov-Galerkin element matrices ; [E][3] diff_coe behind them (ABI order)
  bool with_stab = false;
  double dt = 0.0, ux = 0.0, uy = 0.0, kdiff = 0.0;
  double* xfer = nullptr; size_t xfer_bytes = 0;   // staging for the [E][..] <-> [..][E] conversions at the ABI
  int occ_explicit = 0, occ_assemble = 0, occ_spmv = 0, occ_apply = 0, occ_stab = 0, occ_kry[6] = {0, 0, 0, 0, 0, 0};   // resident CTAs
                              // per SM of the streaming kernels (this device)
  int occ_explicit_f = 0, occ_assemble_f = 0, occ_stab_f = 0;   // the same for the velocity-field instantiations
};

inline size_t plane_stride(int E) {
  size_t q = ((size_t)E + 31) / 32;
  if ((q & 1) == 0) ++q;
  return q * 32;
}

// ---- a warp's 32 consecutive (3, E) records through shared memory: every global access is a full line ----------------
// base = field + 3 * (first element of the warp), nvalid = elements of this warp inside the array, sm = 96 doubles
__device__ __forceinline__ void warp_load3(const double* __restrict__ base, int nvalid, double* sm, int lane, double& a,
                                           double& b, double& c) {
  const int n = nvalid * 3;
  for (int i = lane; i < n; i += 32) sm[i] = __ldg(base + i);
  __syncwarp();
  if (lane < nvalid) { a = sm[lane * 3]; b = sm[lane * 3 + 1]; c = sm[lane * 3 + 2]; }
  __syncwarp();
}
__device__ __forceinline__ void warp_store3(double* __restrict__ base, int nvalid, double* sm, int lane, double a, double b,
                                            double c) {
  if (lane < nvalid) { sm[lane * 3] = a; sm[lane * 3 + 1] = b; sm[lane * 3 + 2] = c; }
  __syncwarp();
  const int n = nvalid * 3;
  for (int i = lane; i < n; i += 32) base[i] = sm[i];
  __syncwarp();
}

// Geometry of one P1 triangle WITHOUT divisions or square roots.  Everything the explicit step and the implicit operator need
// from tri_det_nlx (ShapFun.F90:1414-1454) and det_snlx_all / NORMGI (:1554-1590, 2012-2037) comes as a product in which the
// normalisations cancel:
//   area * grad(phi_i)          = sign(detj)/2 * (D, -C), (-B, A), -(sum)        [A = x1-x3, B = y1-y3, C = x2-x3, D = y2-y3]
//   sdetwei * (n . u) on a face = 1/2 * s * (ey ux - ex uy),  (ex, ey) = the edge vector, s = +-1 makes (ey, -ex) point away
//                                 from the opposite vertex (the reference's test against centroid -> edge midpoint)
// so the kernels spend a few FMAs where the literal formulas need six quotients, three rsqrt and a handful of x/3 (fp64
// division and rsqrt expand to 20-40 instructions each on sm_100a; with them these kernels were issue-bound at a third of the
// HBM rate).  The results differ from the literal order of operations in the last bit only (tests: <= 1e-12 relative).
struct TriEdges {
  double px[3], py[3];
  double A, B, C, D, detj, sgn;    // sgn = sign(detj)
};
__device__ __forceinline__ void tri_edges(const double* __restrict__ X, size_t ld, size_t e, TriEdges& g) {
  const double x1 = __ldg(X + e), y1 = __ldg(X + ld + e), x2 = __ldg(X + 2 * ld + e), y2 = __ldg(X + 3 * ld + e),
               x3 = __ldg(X + 4 * ld + e), y3 = __ldg(X + 5 * ld + e);
  g.px[0] = x1; g.px[1] = x2; g.px[2] = x3; g.py[0] = y1; g.py[1] = y2; g.py[2] = y3;
  g.A = x1 - x3; g.B = y1 - y3; g.C = x2 - x3; g.D = y2 - y3;
  g.detj = g.A * g.D - g.B * g.C;
  g.sgn = g.detj < 0.0 ? -1.0 : 1.0;
}
// face f (0..2) of the gmsh numbering: nodes (l1, l2) = (1,3), (2,1), (3,2) (ShapFun_unstruc.F90:160-188), l3 = the opposite
// vertex.  Returns c = sdetwei * (n . u) (n = outward unit normal, sdetwei = L/2).
__device__ __forceinline__ double face_flux(const TriEdges& g, int l1, int l2, int l3, double ux, double uy) {
  const double ex = g.px[l2] - g.px[l1], ey = g.py[l2] - g.py[l1];
  // (ey, -ex) against (midpoint - centroid) = ((p_l1 - p_l3) + (p_l2 - p_l3)) / 6
  const double mx = (g.px[l1] - g.px[l3]) + (g.px[l2] - g.px[l3]), my = (g.py[l1] - g.py[l3]) + (g.py[l2] - g.py[l3]);
  const double c = 0.5 * (ey * ux - ex * uy);
  return (ey * mx - ex * my < 0.0) ? -c : c;
}

// ---- nodal velocity field u_ele(2,3,E) ------------------------------------------------------------------------------
// Own velocity: six coalesced plane loads.  The neighbour's velocity at its two face nodes (m1, m2) is a gather through L2
// like its T.  Gauss point s of a face weighs (l1, l2) with sn(s, :) = (al, be) at s = 0 and (be, al) at s = 1.
__device__ __forceinline__ void load_vel(const double* __restrict__ U, size_t ld, size_t e, double ux[3], double uy[3]) {
#pragma unroll
  for (int l = 0; l < 3; ++l) { ux[l] = __ldg(U + (size_t)(2 * l) * ld + e); uy[l] = __ldg(U + (size_t)(2 * l + 1) * ld + e); }
}
// Neighbour trace velocity at the face nodes, as the (m1, m2) pair of its T: (x, y) of node m1, then of node m2.  Nside = 0
// (sn2 = 0): zero.  npos = 0 with Nside >= 1: flagged by own = true - the trace is the element's own (sum2 u in the
// uniform form, u_bc = u_ele in trans_rec).
struct FaceVel2 { double ax, ay, bx, by; bool own; };
__device__ __forceinline__ FaceVel2 neighbour_vel(const double* __restrict__ U, size_t ld, int q, int ns, int m1, int m2) {
  FaceVel2 v = {0.0, 0.0, 0.0, 0.0, false};
  if (ns >= 1 && q != 0) {
    const size_t n = (size_t)(q - 1);
    v.ax = __ldg(U + (size_t)(2 * m1) * ld + n); v.ay = __ldg(U + (size_t)(2 * m1 + 1) * ld + n);
    v.bx = __ldg(U + (size_t)(2 * m2) * ld + n); v.by = __ldg(U + (size_t)(2 * m2 + 1) * ld + n);
  } else if (ns >= 1) {
    v.own = true;
  }
  return v;
}
// sdetwei n.u of both traces at Gauss point s and the upwind choice income(s) = 1/2 + 1/2 sign(1, -n.(us + us2)/2), the
// sign taken from the element's own trace alone where sn2 = 0
struct GaussFlux { double c, c2; bool in; };
__device__ __forceinline__ GaussFlux gauss_flux(const TriEdges& g, int l1, int l2, int l3, double a1, double a2,
                                                const double ux[3], const double uy[3], const FaceVel2& v, int ns) {
  GaussFlux r;
  r.c = face_flux(g, l1, l2, l3, a1 * ux[l1] + a2 * ux[l2], a1 * uy[l1] + a2 * uy[l2]);
  r.c2 = v.own ? r.c : face_flux(g, l1, l2, l3, a1 * v.ax + a2 * v.bx, a1 * v.ay + a2 * v.by);
  r.in = signbit(-(ns >= 1 ? r.c + r.c2 : r.c)) == 0;
  return r;
}

struct UnstrArgs {
  const double* X; const int32_t* neig; const int32_t* nside;
  const double* Tin; const double* told; double* Tout;
  double dt, ux, uy, t_bc;
  size_t ld;
  int E, njac, exact, use_dir;
  const double* U;   // velocity planes (FIELD instantiation only); last, so the uniform kernel's parameter offsets stay put
};

// unstr_explicit element loop (transport_tri_unstr.F90:600-791).  One warp = 32 consecutive elements per trip: all the
// streaming loads of a trip (own and told records as 768 contiguous bytes each, six coordinate planes, neighbour ids and
// sides) are issued before anything is used, the six neighbour values are gathered (L2: a locality-ordered mesh keeps
// them a few lines away) and the new record leaves through shared memory as full lines again.
#ifndef PAMG_OCC_EXPLICIT
#define PAMG_OCC_EXPLICIT 4
#endif
#ifndef PAMG_OCC_ASSEMBLE
#define PAMG_OCC_ASSEMBLE 3
#endif
#ifdef PAMG_ASM_STCS
#define ASM_ST(p, v) __stcs((p), (v))
#else
#define ASM_ST(p, v) (*(p) = (v))
#endif
// FIELD: the velocity is the nodal field a.U (u_ele); the volume term takes ugi(g) = sum_i n(g,i) u(:,i) at the three
// Gauss points and every face Gauss point its own upwind choice from the two traces.  The uniform instantiation is the
// kernel as it was before the field existed.
#ifndef PAMG_OCC_EXPLICIT_FIELD
#define PAMG_OCC_EXPLICIT_FIELD 2
#endif
template <bool FIELD>
__global__ void __launch_bounds__(TPB, FIELD ? PAMG_OCC_EXPLICIT_FIELD : PAMG_OCC_EXPLICIT) k_unstr_explicit(UnstrArgs a) {
  __shared__ double smw[TPB / 32][2][96];
  const double al = 0.78867513459481288, be = 0.21132486540518712;  // sn_orig, ShapFun.F90:1100-1111
  // weights of int sn_c * trace over the face: (2/3, 1/3) -- exact products of the 2-point Gauss rule
  const double w2 = al * al + be * be, w1 = 2.0 * al * be;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  double* smT = smw[wib][0];
  double* smO = smw[wib][1];
  const size_t ld = a.ld;
  const double sixth = 1.0 / 6.0;
  for (int e0 = (blockIdx.x * (TPB / 32) + wib) * 32; e0 < a.E; e0 += gridDim.x * TPB) {
    const int nvalid = min(32, a.E - e0);
    const int e = min(e0 + lane, a.E - 1);          // lanes past the end redo the last element and store nothing
    const int n3 = nvalid * 3;
    // ---- every streaming load of the trip
    const double* tin = a.Tin + (size_t)e0 * 3;
    const double* tol = a.told + (size_t)e0 * 3;
    double ra[3], rb[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const int i = lane + 32 * k;
      ra[k] = i < n3 ? __ldg(tin + i) : 0.0;
      rb[k] = i < n3 ? __ldg(tol + i) : 0.0;
    }
    TriEdges g;
    tri_edges(a.X, ld, (size_t)e, g);
    int q[3], enc[3];
#pragma unroll
    for (int f = 0; f < 3; ++f) { q[f] = __ldg(a.neig + (size_t)f * ld + e); enc[f] = __ldg(a.nside + (size_t)f * ld + e); }
    // ---- neighbour values paired with sn_orig(:,1), sn_orig(:,2): get_unstr_sn2 (ShapFun_unstruc.F90:205-222),
    // Nside 1 -> nodes (3,1), 2 -> (1,2), 3 -> (2,3); use_dir: the geometric pairing
    double T2a[3], T2b[3];
    double ux[3], uy[3];
    FaceVel2 v2[3];
    if constexpr (FIELD) load_vel(a.U, ld, (size_t)e, ux, uy);
#pragma unroll
    for (int f = 0; f < 3; ++f) {
      const int ns = enc[f] & 3;
      int m1 = (ns == 1) ? 2 : (ns == 2 ? 0 : 1), m2 = (ns == 1) ? 0 : (ns == 2 ? 1 : 2);
      if (a.use_dir && (enc[f] >> 2)) { const int t = m1; m1 = m2; m2 = t; }
      T2a[f] = a.t_bc; T2b[f] = a.t_bc;
      if (ns >= 1 && q[f] != 0) { const double* nb = a.Tin + (size_t)(q[f] - 1) * 3; T2a[f] = __ldg(nb + m1); T2b[f] = __ldg(nb + m2); }
      // with the neighbour's T, before anything is used: gathered face by face inside the flux loop instead they cost 14 %
      // more time on a B200 (the gathers then wait one after the other)
      if constexpr (FIELD) v2[f] = neighbour_vel(a.U, ld, q[f], ns, m1, m2);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) { smT[lane + 32 * k] = ra[k]; smO[lane + 32 * k] = rb[k]; }
    __syncwarp();
    const double T[3] = {smT[lane * 3], smT[lane * 3 + 1], smT[lane * 3 + 2]};
    const double To[3] = {smO[lane * 3], smO[lane * 3 + 1], smO[lane * 3 + 2]};
    __syncwarp();
    const double sumT = T[0] + T[1] + T[2];
    double rhs[3];
    const int L1[3] = {0, 1, 2}, L2[3] = {2, 0, 1}, L3[3] = {1, 2, 0};
    if constexpr (FIELD) {
      // sum_g (grad(phi_i) . ugi(g)) T(g) detwei(g), ugi and T(g) at the edge midpoints n(g,:) = (1/2,1/2,0), (0,1/2,1/2), (1/2,0,1/2)
      double px = 0.0, py = 0.0;
#pragma unroll
      for (int gq = 0; gq < 3; ++gq) {
        const int i0 = gq == 2 ? 0 : gq, i1 = gq == 2 ? 2 : gq + 1;
        const double tg = 0.5 * (T[i0] + T[i1]);
        px += 0.5 * (ux[i0] + ux[i1]) * tg; py += 0.5 * (uy[i0] + uy[i1]) * tg;
      }
      rhs[0] = g.sgn * (g.D * px - g.C * py) * sixth;
      rhs[1] = g.sgn * (g.A * py - g.B * px) * sixth;
      rhs[2] = -(rhs[0] + rhs[1]);
#pragma unroll
      for (int f = 0; f < 3; ++f) {
        const int l1 = L1[f], l2 = L2[f], ns = enc[f] & 3;
#pragma unroll
        for (int s = 0; s < 2; ++s) {
          const double a1 = s == 0 ? al : be, a2 = s == 0 ? be : al;
          const GaussFlux r = gauss_flux(g, l1, l2, L3[f], a1, a2, ux, uy, v2[f], ns);
          // Nside = 0: c2 = 0, the inflow trace carries nothing (sn2 = 0)
          const double fl = r.in ? r.c2 * (a1 * T2a[f] + a2 * T2b[f]) : r.c * (a1 * T[l1] + a2 * T[l2]);
          rhs[l1] -= a1 * fl; rhs[l2] -= a2 * fl;
        }
      }
    } else {
    // (grad(phi_i) . u) (A/3) sum(T)  (:668-672)
    rhs[0] = g.sgn * (g.D * a.ux - g.C * a.uy) * sixth * sumT;
    rhs[1] = g.sgn * (g.A * a.uy - g.B * a.ux) * sixth * sumT;
    rhs[2] = -(rhs[0] + rhs[1]);
#pragma unroll
    for (int f = 0; f < 3; ++f) {
      const int l1 = L1[f], l2 = L2[f];
      const double c = face_flux(g, l1, l2, L3[f], a.ux, a.uy);   // sdetwei * n . u
      const bool has2 = (enc[f] & 3) >= 1;
      // income = 0.5 + 0.5 sign(1, -n.(u + u2)/2) (:731); u2 = 0 when sn2 = 0 (Nside = 0) does not change the sign
      const bool in = signbit(-c) == 0;
      double ca, cb;
      if (in) { const double f2 = has2 ? c : 0.0; ca = f2 * (w2 * T2a[f] + w1 * T2b[f]); cb = f2 * (w1 * T2a[f] + w2 * T2b[f]); }
      else { ca = c * (w2 * T[l1] + w1 * T[l2]); cb = c * (w1 * T[l1] + w2 * T[l2]); }
      rhs[l1] -= ca; rhs[l2] -= cb;                     // :742-746
    }
    }
    const double area = 0.5 * fabs(g.detj);
    const double m12 = area * (1.0 / 12.0);
    const double iarea = 1.0 / area;
    const double so = To[0] + To[1] + To[2];
    double out[3];
    if (a.exact) {
      // T = M^-1 (M told + dt rhs), M^-1 = (12/A)(I - J/4)  (transport_rect.F90:277-291 semantics)
      double v[3];
#pragma unroll
      for (int i = 0; i < 3; ++i) v[i] = m12 * (To[i] + so) + a.dt * rhs[i];
      const double sv = v[0] + v[1] + v[2];
      const double i12 = 12.0 * iarea;
#pragma unroll
      for (int i = 0; i < 3; ++i) out[i] = i12 * (v[i] - 0.25 * sv);
    } else {
      // Jacobi on the lumped mass ml = A/3 (:774-787): t <- (ml t - M t + rj) / ml = t - (t + sum t)/4 + rj / ml
      double rj[3], tl[3] = {T[0], T[1], T[2]};           // tnew_nonlin(:,ele) == tnew(:,ele) here (:598,783)
      const double iml = 3.0 * iarea;
#pragma unroll
      for (int i = 0; i < 3; ++i) rj[i] = (m12 * (To[i] + so) + a.dt * rhs[i]) * iml;
      for (int it = 0; it < a.njac; ++it) {
        const double st = tl[0] + tl[1] + tl[2];
#pragma unroll
        for (int i = 0; i < 3; ++i) tl[i] = tl[i] - 0.25 * (tl[i] + st) + rj[i];
      }
      out[0] = tl[0]; out[1] = tl[1]; out[2] = tl[2];
    }
    smT[lane * 3] = out[0]; smT[lane * 3 + 1] = out[1]; smT[lane * 3 + 2] = out[2];
    __syncwarp();
    double* to = a.Tout + (size_t)e0 * 3;
#pragma unroll
    for (int k = 0; k < 3; ++k) { const int i = lane + 32 * k; if (i < n3) to[i] = smT[i]; }
    __syncwarp();
  }
}

// [E][K] (ABI order) <-> [K][ld] planes; one thread per element (set-up and read-back only)
template <typename Tp>
__global__ void __launch_bounds__(TPB) k_to_planes(const Tp* __restrict__ aos, Tp* __restrict__ soa, int K, int E, size_t ld) {
  for (int e = blockIdx.x * TPB + threadIdx.x; e < E; e += gridDim.x * TPB)
    for (int k = 0; k < K; ++k) soa[(size_t)k * ld + e] = aos[(size_t)e * K + k];
}
template <typename Tp>
__global__ void __launch_bounds__(TPB) k_from_planes(const Tp* __restrict__ soa, Tp* __restrict__ aos, int K, int E, size_t ld) {
  for (int e = blockIdx.x * TPB + threadIdx.x; e < E; e += gridDim.x * TPB)
    for (int k = 0; k < K; ++k) aos[(size_t)e * K + k] = soa[(size_t)k * ld + e];
}

inline void unstr_free(UnstrDev& u) {
  cudaFree(u.X); cudaFree(u.U); cudaFree(u.neig); cudaFree(u.nside); cudaFree(u.pen); cudaFree(u.T[0]); cudaFree(u.T[1]); cudaFree(u.told);
  cudaFree(u.bsr_val); cudaFree(u.bsr_col); cudaFree(u.dinv); cudaFree(u.mdt); cudaFree(u.work); cudaFree(u.dots); cudaFree(u.diag0); cudaFree(u.stab);
  cudaFree(u.xfer);
  if (u.dots_host) cudaFreeHost(u.dots_host);
  u = UnstrDev();
}

#define UCK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { err = std::string(#call) + ": " + cudaGetErrorString(e_); return PAMG_ERR_CUDA; } } while (0)

inline int unstr_xfer(UnstrDev& u, size_t bytes, std::string& err) {
  if (u.xfer_bytes >= bytes) return PAMG_OK;
  cudaFree(u.xfer); u.xfer = nullptr; u.xfer_bytes = 0;
  UCK(cudaMalloc(&u.xfer, bytes));
  u.xfer_bytes = bytes;
  return PAMG_OK;
}

// grid of a streaming kernel: every resident CTA slot of the device exactly once (a partial last wave of a grid-stride loop
// costs a whole trip), or fewer CTAs for a small mesh
template <typename K>
inline int stream_grid(K kernel, int& occ_cache, int E, int nsm) {
  if (occ_cache <= 0) {
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, TPB, 0) != cudaSuccess || occ < 1) occ = 2;
    occ_cache = occ;
  }
  return std::max(1, std::min((E + TPB - 1) / TPB, nsm * std::min(occ_cache, 8)));   // (8: the Krylov partial sums are sized for it)
}

inline int unstr_setup(UnstrDev& u, int E, const double* X, const int32_t* neig, const int32_t* fneig,
                       cudaStream_t st, std::string& err) {
  unstr_free(u);
  // geometric pairing flag per face: does the neighbour node that get_unstr_sn2 pairs with my first face
  // node actually coincide with it?  (SURVEY B-9: the reference ignores Dir here)
  // penalty length of the diffusion face term (get_d_center Msh2Tri.F90:349-385, add_diffusion_surf matrices.F90:84-110)
  const size_t ld = plane_stride(E);
  std::vector<int32_t> enc(ld * 3, 0), ng(ld * 3, 0);
  std::vector<double> xs(ld * 6, 0.0), pn(ld * 3, 0.0);
  const int L1[3] = {0, 1, 2}, L2[3] = {2, 0, 1};
  for (int e = 0; e < E; ++e) {
    const double* P = X + (size_t)e * 6;
    const double cx = (P[0] + P[2] + P[4]) / 3.0, cy = (P[1] + P[3] + P[5]) / 3.0;
    for (int k = 0; k < 6; ++k) xs[(size_t)k * ld + e] = P[k];
    for (int f = 0; f < 3; ++f) {
      const int q = neig[(size_t)e * 3 + f], ns = fneig[(size_t)e * 3 + f];
      int sw = 0;
      double d;
      if (q != 0 && ns >= 1 && ns <= 3) {
        const int m1 = (ns == 1) ? 2 : (ns == 2 ? 0 : 1);
        const double* a = X + (size_t)e * 6 + 2 * L1[f];
        const double* Q = X + (size_t)(q - 1) * 6;
        const double* b = Q + 2 * m1;
        sw = !(a[0] == b[0] && a[1] == b[1]);
        const double qx = (Q[0] + Q[2] + Q[4]) / 3.0, qy = (Q[1] + Q[3] + Q[5]) / 3.0;
        d = std::sqrt((cx - qx) * (cx - qx) + (cy - qy) * (cy - qy));
      } else if (q != 0) { err = "fNeig must be 1..3 where Neig != 0"; return PAMG_ERR_ARG; }
      else {
        const double mx = 0.5 * (P[2 * L1[f]] + P[2 * L2[f]]), my = 0.5 * (P[2 * L1[f] + 1] + P[2 * L2[f] + 1]);
        d = std::sqrt((cx - mx) * (cx - mx) + (cy - my) * (cy - my));
      }
      const double ex = P[2 * L2[f]] - P[2 * L1[f]], ey = P[2 * L2[f] + 1] - P[2 * L1[f] + 1];
      enc[(size_t)f * ld + e] = (ns & 3) | (sw << 2);
      ng[(size_t)f * ld + e] = q;
      pn[(size_t)f * ld + e] = 0.5 * std::sqrt(ex * ex + ey * ey) / d;
    }
  }
  u.E = E; u.ld = ld;
  UCK(cudaMalloc(&u.X, ld * 6 * sizeof(double)));
  UCK(cudaMalloc(&u.neig, ld * 3 * sizeof(int32_t)));
  UCK(cudaMalloc(&u.nside, ld * 3 * sizeof(int32_t)));
  UCK(cudaMalloc(&u.pen, ld * 3 * sizeof(double)));
  for (int i = 0; i < 2; ++i) UCK(cudaMalloc(&u.T[i], (size_t)E * 3 * sizeof(double)));
  UCK(cudaMalloc(&u.told, (size_t)E * 3 * sizeof(double)));
  UCK(cudaMemcpyAsync(u.X, xs.data(), ld * 6 * sizeof(double), cudaMemcpyHostToDevice, st));
  UCK(cudaMemcpyAsync(u.neig, ng.data(), ld * 3 * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  UCK(cudaMemcpyAsync(u.nside, enc.data(), ld * 3 * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  UCK(cudaMemcpyAsync(u.pen, pn.data(), ld * 3 * sizeof(double), cudaMemcpyHostToDevice, st));
  UCK(cudaMemsetAsync(u.T[0], 0, (size_t)E * 3 * sizeof(double), st));
  UCK(cudaMemsetAsync(u.T[1], 0, (size_t)E * 3 * sizeof(double), st));
  UCK(cudaStreamSynchronize(st));
  u.cur = 0;
  return PAMG_OK;
}

// u_ele(2,3,E) in the reference's layout ([E][6] doubles, host) -> 6 planes; null clears the field.  The operator assembled
// with the previous velocity is stale either way: the implicit entries refuse to run until the next assembly.
inline int unstr_set_velocity(UnstrDev& u, const double* u_ele, int nsm, cudaStream_t st, std::string& err) {
  u.assembled = false;
  u.with_stab = false;
  if (!u_ele) { cudaFree(u.U); u.U = nullptr; return PAMG_OK; }
  const size_t E = (size_t)u.E;
  if (!u.U) UCK(cudaMalloc(&u.U, u.ld * 6 * sizeof(double)));
  // on any failure below the planes hold no valid field: drop them, so that later calls run the uniform path, not garbage
  int rc = unstr_xfer(u, E * 6 * sizeof(double), err);
  if (rc == PAMG_OK) {
    cudaError_t e1 = cudaMemcpyAsync(u.xfer, u_ele, E * 6 * sizeof(double), cudaMemcpyHostToDevice, st);
    if (e1 == cudaSuccess) {
      k_to_planes<double><<<std::max(1, std::min((u.E + TPB - 1) / TPB, nsm * 8)), TPB, 0, st>>>(u.xfer, u.U, 6, u.E, u.ld);
      e1 = cudaGetLastError();
    }
    if (e1 == cudaSuccess) e1 = cudaStreamSynchronize(st);
    if (e1 != cudaSuccess) { err = std::string("pamg_unstr_set_velocity: ") + cudaGetErrorString(e1); rc = PAMG_ERR_CUDA; }
  }
  if (rc != PAMG_OK) { cudaFree(u.U); u.U = nullptr; }
  return rc;
}

// time loop of unstr_explicit (:588-795): told = tnew ; nits x { tnew = tnew_nonlin ; element loop }
inline int unstr_step(UnstrDev& u, double dt, double ux, double uy, double t_bc, int ntime, int nits, int njac,
                      int exact, int use_dir, int nsm, cudaStream_t st, long long& nlaunch, std::string& err) {
  const int grid = u.U ? stream_grid(k_unstr_explicit<true>, u.occ_explicit_f, u.E, nsm)
                       : stream_grid(k_unstr_explicit<false>, u.occ_explicit, u.E, nsm);
  for (int it = 0; it < ntime; ++it) {
    UCK(cudaMemcpyAsync(u.told, u.T[u.cur], (size_t)u.E * 3 * sizeof(double), cudaMemcpyDeviceToDevice, st));
    for (int k = 0; k < nits; ++k) {
      UnstrArgs a;
      a.X = u.X; a.neig = u.neig; a.nside = u.nside; a.Tin = u.T[u.cur]; a.told = u.told; a.Tout = u.T[u.cur ^ 1];
      a.dt = dt; a.ux = ux; a.uy = uy; a.t_bc = t_bc; a.ld = u.ld; a.E = u.E; a.njac = njac; a.exact = exact; a.use_dir = use_dir;
      a.U = u.U;
      if (u.U) k_unstr_explicit<true><<<grid, TPB, 0, st>>>(a);
      else k_unstr_explicit<false><<<grid, TPB, 0, st>>>(a);
      nlaunch++;
      UCK(cudaGetLastError());
      u.cur ^= 1;
    }
  }
  return PAMG_OK;
}

// ------------------------------------------------------------------------------------------------
// Implicit "Jacobian" of unstr_implicit (transport_tri_unstr.F90:270-364) assembled straight into block-CSR on the
// device (SURVEY 8(f1)): one thread per element writes its diagonal block mass/dt - stiff (+ the outflow part of the
// upwind flux, :344-360 with income = 0) and one 3x3 block per inflow face in the neighbour's columns
// (`target_ele`, :339-342).  With kdiff > 0 the diffusion operator of the iterative path is added (the reference's
// implicit drivers compute add_diffusion_vol and drop it, transport_tri_semi.F90:1627; this is the intended use): the
// volume block k A grad(phi_i).grad(phi_j) (ShapFun_unstruc.F90:324-335) on the diagonal and the face penalty
// (k/dx) int sn_i (T - T2) (matrices.F90:113-115, get_diff_surf_stencl transport_tri_semi.F90:468-477) on the own and
// the neighbour's columns.  The reference builds three scalar CSR matrices, converts them to dense and inverts
// the dense (3E)^2 matrix with FINDInv (:366-378); here the operator never leaves its 4-blocks-per-row form, stored as
// 36 + 4 planes so that every store of a warp is one full line.  A face block has four non-zero entries (rows = my two face
// nodes, columns = the neighbour's two); it leaves the registers as soon as its face is done, so only the diagonal block is
// live across the face loop (48 registers instead of 74: 5 resident CTAs per SM keep enough stores in flight for HBM).
struct BsrArgs {
  const double* X; const int32_t* neig; const int32_t* nside; const double* pen;
  double* val; int32_t* col; double* dinv; double* mdt;
  double inv24dt, ux, uy, kdiff;
  size_t ld;
  int E, use_dir;
  const double* U;   // velocity planes (FIELD only)
};

// FIELD: stiff(i,j) = sum_g (grad(phi_i) . ugi(g)) n(g,j) detwei(g) (no longer the same for every j) and the face flux split per
// Gauss point: the sn(s,j) part of an outflow point into the own columns, the sn2(s,j) part of an inflow point into the
// neighbour's.  (HEAD, :339, sends the whole face to one block chosen by income(1); for a uniform velocity both Gauss points
// agree and the two rules coincide.)
#ifndef PAMG_OCC_ASSEMBLE_FIELD
#define PAMG_OCC_ASSEMBLE_FIELD 2
#endif
template <bool FIELD>
__global__ void __launch_bounds__(TPB, FIELD ? PAMG_OCC_ASSEMBLE_FIELD : PAMG_OCC_ASSEMBLE) k_assemble_bsr(BsrArgs a) {
  const double al = 0.78867513459481288, be = 0.21132486540518712;
  const double w2 = al * al + be * be, w1 = 2.0 * al * be;
  const size_t ld = a.ld;
  const double sixth = 1.0 / 6.0;
  for (int e = blockIdx.x * TPB + threadIdx.x; e < a.E; e += gridDim.x * TPB) {
    TriEdges g;
    tri_edges(a.X, ld, (size_t)e, g);
    int q[3], enc[3];
#pragma unroll
    for (int f = 0; f < 3; ++f) { q[f] = __ldg(a.neig + (size_t)f * ld + e); enc[f] = __ldg(a.nside + (size_t)f * ld + e); }
    double pn[3] = {0.0, 0.0, 0.0};
    if (a.kdiff != 0.0) {
#pragma unroll
      for (int f = 0; f < 3; ++f) pn[f] = a.kdiff * __ldg(a.pen + (size_t)f * ld + e);
    }
    const double adet = fabs(g.detj);
    const double m12 = adet * a.inv24dt;                    // A / (12 dt)
    double d[9];
    double ux[3], uy[3];
    if constexpr (FIELD) {
      load_vel(a.U, ld, (size_t)e, ux, uy);
      // a(i,g) = (grad(phi_i) . ugi(g)) A/3 ; stiff(i,j) = sum_g a(i,g) n(g,j): g = 0 holds nodes (0,1), 1 (1,2), 2 (0,2)
      double gx[3], gy[3];
#pragma unroll
      for (int gq = 0; gq < 3; ++gq) {
        const int i0 = gq == 2 ? 0 : gq, i1 = gq == 2 ? 2 : gq + 1;
        gx[gq] = 0.5 * (ux[i0] + ux[i1]); gy[gq] = 0.5 * (uy[i0] + uy[i1]);
      }
      const double Gx[3] = {g.D, -g.B, g.B - g.D}, Gy[3] = {-g.C, g.A, g.C - g.A};
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        double ag[3];
#pragma unroll
        for (int gq = 0; gq < 3; ++gq) ag[gq] = g.sgn * (Gx[i] * gx[gq] + Gy[i] * gy[gq]) * sixth;
        const double st[3] = {0.5 * (ag[0] + ag[2]), 0.5 * (ag[0] + ag[1]), 0.5 * (ag[1] + ag[2])};
#pragma unroll
        for (int j = 0; j < 3; ++j) d[i * 3 + j] = m12 * (i == j ? 2.0 : 1.0) - st[j];
      }
    } else {
      // stiff(i,j) = (grad(phi_i) . u) A/3: the same for every j (:281-283)
      double st[3];
      st[0] = g.sgn * (g.D * a.ux - g.C * a.uy) * sixth;
      st[1] = g.sgn * (g.A * a.uy - g.B * a.ux) * sixth;
      st[2] = -(st[0] + st[1]);
#pragma unroll
      for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) d[i * 3 + j] = m12 * (i == j ? 2.0 : 1.0) - st[i];
    }
    {
      if (a.kdiff != 0.0) {
        // k A grad(phi_i) . grad(phi_j) = k / (2 |detj|) G_i . G_j with the unnormalised gradients G = (D,-C), (-B,A), -(sum)
        const double kk = a.kdiff * 0.5 / adet;
        const double Gx[3] = {g.D, -g.B, g.B - g.D}, Gy[3] = {-g.C, g.A, g.C - g.A};
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
          for (int j = 0; j < 3; ++j) d[i * 3 + j] += kk * (Gx[i] * Gx[j] + Gy[i] * Gy[j]);
      }
    }
    const int L1[3] = {0, 1, 2}, L2[3] = {2, 0, 1}, L3[3] = {1, 2, 0};
    ASM_ST(a.col + e, e);
#pragma unroll
    for (int f = 0; f < 3; ++f) {
      const int l1 = L1[f], l2 = L2[f];
      const double c = face_flux(g, l1, l2, L3[f], a.ux, a.uy);   // sdetwei * n . u
      const int ns = enc[f] & 3;
      const bool in = signbit(-c) == 0;
      // neighbour nodes coincident with (l1, l2): as in get_unstr_sn2, or the geometric pairing with use_dir
      int m1 = (ns == 1) ? 2 : (ns == 2 ? 0 : 1), m2 = (ns == 1) ? 0 : (ns == 2 ? 1 : 2);
      if (a.use_dir && (enc[f] >> 2)) { const int t = m1; m1 = m2; m2 = t; }
      double o11 = 0.0, o12 = 0.0;     // the face block: rows (l1, l2) x columns (m1, m2) = [[o11, o12], [o12, o11]]
      double o21 = 0.0, o22 = 0.0;     // FIELD: [[o11, o12], [o21, o22]]
      int colf = -1;
      if constexpr (FIELD) {
        const FaceVel2 v2 = neighbour_vel(a.U, ld, q[f], ns, m1, m2);
        // the own face-node velocities again (L1 hits): not holding all six across the face loop keeps the kernel in 128
        // registers without spilling
        double fx[3] = {0.0, 0.0, 0.0}, fy[3] = {0.0, 0.0, 0.0};
        fx[l1] = __ldg(a.U + (size_t)(2 * l1) * ld + e); fy[l1] = __ldg(a.U + (size_t)(2 * l1 + 1) * ld + e);
        fx[l2] = __ldg(a.U + (size_t)(2 * l2) * ld + e); fy[l2] = __ldg(a.U + (size_t)(2 * l2 + 1) * ld + e);
#pragma unroll
        for (int s = 0; s < 2; ++s) {
          const double a1 = s == 0 ? al : be, a2 = s == 0 ? be : al;
          const GaussFlux r = gauss_flux(g, l1, l2, L3[f], a1, a2, fx, fy, v2, ns);
          if (!r.in) {
            d[l1 * 3 + l1] += r.c * a1 * a1; d[l1 * 3 + l2] += r.c * a1 * a2;
            d[l2 * 3 + l1] += r.c * a2 * a1; d[l2 * 3 + l2] += r.c * a2 * a2;
          } else if (ns >= 1) {
            const double p11 = r.c2 * a1 * a1, p12 = r.c2 * a1 * a2, p21 = r.c2 * a2 * a1, p22 = r.c2 * a2 * a2;
            if (q[f] != 0) { o11 += p11; o12 += p12; o21 += p21; o22 += p22; colf = q[f] - 1; }
            else {                     // target_ele == 0: the element's own columns at (m1, m2) (:340-342)
#pragma unroll
              for (int j = 0; j < 3; ++j) {
                d[l1 * 3 + j] += (j == m1) ? p11 : ((j == m2) ? p12 : 0.0);
                d[l2 * 3 + j] += (j == m1) ? p21 : ((j == m2) ? p22 : 0.0);
              }
            }
          }
        }
      } else if (!in) {                // outflow: own columns
        d[l1 * 3 + l1] += c * w2; d[l1 * 3 + l2] += c * w1;
        d[l2 * 3 + l1] += c * w1; d[l2 * 3 + l2] += c * w2;
      } else if (ns >= 1) {            // inflow: the neighbour's columns, its nodes paired as in get_unstr_sn2
        if (q[f] != 0) { o11 = c * w2; o12 = c * w1; colf = q[f] - 1; }
        else {                         // target_ele == 0 falls back to the element itself (:340-342)
#pragma unroll
          for (int j = 0; j < 3; ++j) {
            d[l1 * 3 + j] += (j == m1) ? c * w2 : ((j == m2) ? c * w1 : 0.0);
            d[l2 * 3 + j] += (j == m1) ? c * w1 : ((j == m2) ? c * w2 : 0.0);
          }
        }
      }                                // inflow through the domain boundary (Nside = 0): sn2 = 0 -> no block
      if (a.kdiff != 0.0) {
        // penalty diffusion: own block += (k/dx) F, neighbour block -= (k/dx) F, F = (L/2) [[w2, w1], [w1, w2]]; on the
        // domain boundary the exterior trace is Dirichlet data (right-hand side), only the own part stays
        const double kd = pn[f];
        d[l1 * 3 + l1] += kd * w2; d[l1 * 3 + l2] += kd * w1;
        d[l2 * 3 + l1] += kd * w1; d[l2 * 3 + l2] += kd * w2;
        if (q[f] != 0 && ns >= 1) {
          o11 -= kd * w2; o12 -= kd * w1; colf = q[f] - 1;
          if constexpr (FIELD) { o21 -= kd * w1; o22 -= kd * w2; }
        }
      }
      ASM_ST(a.col + (size_t)(1 + f) * ld + e, colf);
      double* v = a.val + (size_t)((1 + f) * 9) * ld + e;
#pragma unroll
      for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
          double x = 0.0;
          if (i == l1) x = (j == m1) ? o11 : ((j == m2) ? o12 : 0.0);
          if constexpr (FIELD) { if (i == l2) x = (j == m1) ? o21 : ((j == m2) ? o22 : 0.0); }
          else { if (i == l2) x = (j == m1) ? o12 : ((j == m2) ? o11 : 0.0); }
          ASM_ST(v + (size_t)(i * 3 + j) * ld, x);
        }
    }
#pragma unroll
    for (int k = 0; k < 9; ++k) ASM_ST(a.val + (size_t)k * ld + e, d[k]);
    // inverse of the diagonal block by its adjugate
    const double c00 = d[4] * d[8] - d[5] * d[7], c01 = d[5] * d[6] - d[3] * d[8], c02 = d[3] * d[7] - d[4] * d[6];
    const double det = d[0] * c00 + d[1] * c01 + d[2] * c02, id = 1.0 / det;
    ASM_ST(a.dinv + e, c00 * id);
    ASM_ST(a.dinv + ld + e, (d[2] * d[7] - d[1] * d[8]) * id);
    ASM_ST(a.dinv + 2 * ld + e, (d[1] * d[5] - d[2] * d[4]) * id);
    ASM_ST(a.dinv + 3 * ld + e, c01 * id);
    ASM_ST(a.dinv + 4 * ld + e, (d[0] * d[8] - d[2] * d[6]) * id);
    ASM_ST(a.dinv + 5 * ld + e, (d[2] * d[3] - d[0] * d[5]) * id);
    ASM_ST(a.dinv + 6 * ld + e, c02 * id);
    ASM_ST(a.dinv + 7 * ld + e, (d[1] * d[6] - d[0] * d[7]) * id);
    ASM_ST(a.dinv + 8 * ld + e, (d[0] * d[4] - d[1] * d[3]) * id);
    ASM_ST(a.mdt + e, m12);
  }
}

// y = A x (block-CSR planes) ; mode 1: y = b - A x.  x, b, y are (3, E) vectors.
__global__ void __launch_bounds__(TPB) k_bsr_spmv(const double* __restrict__ val, const int32_t* __restrict__ col,
                                                  const double* __restrict__ x, const double* __restrict__ b,
                                                  double* __restrict__ y, int En, size_t ld, int mode) {
  __shared__ double smw[TPB / 32][96];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  double* sm = smw[wib];
  const size_t E = ld;   // plane stride
  for (int e0 = (blockIdx.x * (TPB / 32) + wib) * 32; e0 < En; e0 += gridDim.x * TPB) {
    const int nvalid = min(32, En - e0);
    const int e = e0 + lane;
    double s0 = 0, s1 = 0, s2 = 0;
    double b0 = 0, b1 = 0, b2 = 0;
    if (mode == 1) warp_load3(b + (size_t)e0 * 3, nvalid, sm, lane, b0, b1, b2);
    if (lane < nvalid) {
#pragma unroll
      for (int bq = 0; bq < 4; ++bq) {
        const int c = __ldg(col + (size_t)bq * E + e);
        if (c < 0) continue;
        const double* v = val + (size_t)(bq * 9) * E + e;
        const double x0 = __ldg(x + (size_t)c * 3), x1 = __ldg(x + (size_t)c * 3 + 1), x2 = __ldg(x + (size_t)c * 3 + 2);
        s0 += __ldg(v) * x0 + __ldg(v + E) * x1 + __ldg(v + 2 * E) * x2;
        s1 += __ldg(v + 3 * E) * x0 + __ldg(v + 4 * E) * x1 + __ldg(v + 5 * E) * x2;
        s2 += __ldg(v + 6 * E) * x0 + __ldg(v + 7 * E) * x1 + __ldg(v + 8 * E) * x2;
      }
      if (mode == 1) { s0 = b0 - s0; s1 = b1 - s1; s2 = b2 - s2; }
    }
    warp_store3(y + (size_t)e0 * 3, nvalid, sm, lane, s0, s1, s2);
  }
}

// y = Dinv x (block-Jacobi preconditioner) ; mode 1: y = (M/dt) x with M/dt = mdt (I + J) per element (:366-369)
__global__ void __launch_bounds__(TPB) k_block_apply(const double* __restrict__ dinv, const double* __restrict__ mdt,
                                                     const double* __restrict__ x, double* __restrict__ y, int En, size_t ld, int mode) {
  __shared__ double smw[TPB / 32][96];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  double* sm = smw[wib];
  const size_t E = ld;   // plane stride
  for (int e0 = (blockIdx.x * (TPB / 32) + wib) * 32; e0 < En; e0 += gridDim.x * TPB) {
    const int nvalid = min(32, En - e0);
    const int e = e0 + lane;
    double x0 = 0, x1 = 0, x2 = 0, y0 = 0, y1 = 0, y2 = 0;
    warp_load3(x + (size_t)e0 * 3, nvalid, sm, lane, x0, x1, x2);
    if (lane < nvalid) {
      if (mode == 1) {
        const double m = mdt[e], sx = x0 + x1 + x2;
        y0 = m * (x0 + sx); y1 = m * (x1 + sx); y2 = m * (x2 + sx);
      } else {
        const double* d = dinv + e;
        y0 = __ldg(d) * x0 + __ldg(d + E) * x1 + __ldg(d + 2 * E) * x2;
        y1 = __ldg(d + 3 * E) * x0 + __ldg(d + 4 * E) * x1 + __ldg(d + 5 * E) * x2;
        y2 = __ldg(d + 6 * E) * x0 + __ldg(d + 7 * E) * x1 + __ldg(d + 8 * E) * x2;
      }
    }
    warp_store3(y + (size_t)e0 * 3, nvalid, sm, lane, y0, y1, y2);
  }
}

// z = a x + b y + c w   (w may be null; z may alias any input)
__global__ void __launch_bounds__(TPB) k_lincomb(double* z, double a, const double* x, double b, const double* y, double c,
                                                 const double* w, long long n) {
  for (long long i = (long long)blockIdx.x * TPB + threadIdx.x; i < n; i += (long long)gridDim.x * TPB)
    z[i] = a * x[i] + b * y[i] + (w ? c * w[i] : 0.0);
}

// ---- BiCGStab with device-resident scalars -----------------------------------------------------------------------------
// The reference inverts the dense (3E)^2 matrix (FINDInv, transport_tri_unstr.F90:366-378).  Here: BiCGStab, right-
// preconditioned with the inverse diagonal blocks.  Every scalar of the recurrence (rho, alpha, omega, the norms, the
// convergence flag) lives in device memory: a kernel that ends with a dot product leaves its partial sums per CTA and the
// LAST CTA to finish adds them up in a fixed order (deterministic) and derives the scalars the next kernel needs.  One
// iteration is 5 kernels and no host round trip; the host looks at the flag once per batch of iterations.
enum { KS_RHO = 0, KS_ALPHA, KS_OMEGA, KS_RHONEW, KS_RR, KS_BB, KS_STOP2, KS_DONE, KS_ITER, KS_MAXIT, KS_COUNTER = 16, KS_PARTIAL = 32 };

// sum of two per-thread values over the grid: returns true in every thread of the last CTA, with the totals in t0, t1
__device__ __forceinline__ bool grid_sum2(double s0, double s1, double* ks, double& t0, double& t1) {
  __shared__ double sh[2][TPB];
  __shared__ int s_last;
  for (int o = 16; o > 0; o >>= 1) { s0 += __shfl_xor_sync(0xffffffffu, s0, o); s1 += __shfl_xor_sync(0xffffffffu, s1, o); }
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { sh[0][w] = s0; sh[1][w] = s1; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0, b = 0;
    for (int i = 0; i < TPB / 32; ++i) { a += sh[0][i]; b += sh[1][i]; }
    ks[KS_PARTIAL + 2 * blockIdx.x] = a; ks[KS_PARTIAL + 2 * blockIdx.x + 1] = b;
    __threadfence();
    s_last = atomicAdd(reinterpret_cast<unsigned long long*>(ks + KS_COUNTER), 1ull) == (unsigned long long)gridDim.x - 1;
  }
  __syncthreads();
  if (!s_last) return false;
  __threadfence();
  double a = 0, b = 0;
  for (int i = threadIdx.x; i < (int)gridDim.x; i += TPB) {
    a += *(volatile double*)(ks + KS_PARTIAL + 2 * i); b += *(volatile double*)(ks + KS_PARTIAL + 2 * i + 1);
  }
  __syncthreads();
  sh[0][threadIdx.x] = a; sh[1][threadIdx.x] = b;
  __syncthreads();
  for (int s = TPB / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) { sh[0][threadIdx.x] += sh[0][threadIdx.x + s]; sh[1][threadIdx.x] += sh[1][threadIdx.x + s]; }
    __syncthreads();
  }
  t0 = sh[0][0]; t1 = sh[1][0];
  if (threadIdx.x == 0) *reinterpret_cast<unsigned long long*>(ks + KS_COUNTER) = 0ull;
  return true;
}

struct KryArgs {
  const double* val; const int32_t* col; const double* dinv;
  double *x, *b, *r, *rh, *p, *v, *s, *t, *y, *z;
  double* ks;
  size_t ld;
  int E;
};

// start of a solve: r = b - A x ; rh = r ; p = v = 0 ; bb = (b, b) ; rr = (r, r) ; rho_new = (rh, r) = rr
__global__ void __launch_bounds__(TPB) k_kry_init(KryArgs a, double tol) {
  __shared__ double smw[TPB / 32][96];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  double* sm = smw[wib];
  const size_t E = a.ld;   // plane stride
  double sbb = 0, srr = 0;
  for (int e0 = (blockIdx.x * (TPB / 32) + wib) * 32; e0 < a.E; e0 += gridDim.x * TPB) {
    const int nvalid = min(32, a.E - e0);
    const int e = e0 + lane;
    double b0 = 0, b1 = 0, b2 = 0, s0 = 0, s1 = 0, s2 = 0;
    warp_load3(a.b + (size_t)e0 * 3, nvalid, sm, lane, b0, b1, b2);
    if (lane < nvalid) {
#pragma unroll
      for (int bq = 0; bq < 4; ++bq) {
        const int c = __ldg(a.col + (size_t)bq * E + e);
        if (c < 0) continue;
        const double* v = a.val + (size_t)(bq * 9) * E + e;
        const double x0 = a.x[(size_t)c * 3], x1 = a.x[(size_t)c * 3 + 1], x2 = a.x[(size_t)c * 3 + 2];
        s0 += __ldg(v) * x0 + __ldg(v + E) * x1 + __ldg(v + 2 * E) * x2;
        s1 += __ldg(v + 3 * E) * x0 + __ldg(v + 4 * E) * x1 + __ldg(v + 5 * E) * x2;
        s2 += __ldg(v + 6 * E) * x0 + __ldg(v + 7 * E) * x1 + __ldg(v + 8 * E) * x2;
      }
      s0 = b0 - s0; s1 = b1 - s1; s2 = b2 - s2;
      sbb += b0 * b0 + b1 * b1 + b2 * b2; srr += s0 * s0 + s1 * s1 + s2 * s2;
    }
    warp_store3(a.r + (size_t)e0 * 3, nvalid, sm, lane, s0, s1, s2);
    warp_store3(a.rh + (size_t)e0 * 3, nvalid, sm, lane, s0, s1, s2);
    warp_store3(a.p + (size_t)e0 * 3, nvalid, sm, lane, 0.0, 0.0, 0.0);
    warp_store3(a.v + (size_t)e0 * 3, nvalid, sm, lane, 0.0, 0.0, 0.0);
  }
  double bb, rr;
  if (grid_sum2(sbb, srr, a.ks, bb, rr) && threadIdx.x == 0) {
    a.ks[KS_BB] = bb; a.ks[KS_RR] = rr; a.ks[KS_STOP2] = tol * tol * bb;
    a.ks[KS_RHO] = 1.0; a.ks[KS_ALPHA] = 1.0; a.ks[KS_OMEGA] = 1.0; a.ks[KS_RHONEW] = rr;
    a.ks[KS_ITER] = 0.0;
    a.ks[KS_DONE] = (rr <= tol * tol * bb) ? 1.0 : 0.0;
  }
}

// p = r + beta (p - omega v) ; y = Dinv p      (beta from the scalars; breakdown -> done = 2)
__global__ void __launch_bounds__(TPB) k_kry_p(KryArgs a) {
  if (a.ks[KS_DONE] != 0.0) return;
  __shared__ double smw[TPB / 32][96];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  double* sm = smw[wib];
  const size_t E = a.ld;   // plane stride
  const double rho_new = a.ks[KS_RHONEW], rho = a.ks[KS_RHO], alpha = a.ks[KS_ALPHA], omega = a.ks[KS_OMEGA];
  const double beta = (rho_new / rho) * (alpha / omega);
  for (int e0 = (blockIdx.x * (TPB / 32) + wib) * 32; e0 < a.E; e0 += gridDim.x * TPB) {
    const int nvalid = min(32, a.E - e0);
    const int e = e0 + lane;
    double r0 = 0, r1 = 0, r2 = 0, p0 = 0, p1 = 0, p2 = 0, v0 = 0, v1 = 0, v2 = 0, y0 = 0, y1 = 0, y2 = 0;
    warp_load3(a.r + (size_t)e0 * 3, nvalid, sm, lane, r0, r1, r2);
    warp_load3(a.p + (size_t)e0 * 3, nvalid, sm, lane, p0, p1, p2);
    warp_load3(a.v + (size_t)e0 * 3, nvalid, sm, lane, v0, v1, v2);
    p0 = r0 + beta * p0 + (-beta * omega) * v0; p1 = r1 + beta * p1 + (-beta * omega) * v1; p2 = r2 + beta * p2 + (-beta * omega) * v2;
    if (lane < nvalid) {
      const double* d = a.dinv + e;
      y0 = __ldg(d) * p0 + __ldg(d + E) * p1 + __ldg(d + 2 * E) * p2;
      y1 = __ldg(d + 3 * E) * p0 + __ldg(d + 4 * E) * p1 + __ldg(d + 5 * E) * p2;
      y2 = __ldg(d + 6 * E) * p0 + __ldg(d + 7 * E) * p1 + __ldg(d + 8 * E) * p2;
    }
    warp_store3(a.p + (size_t)e0 * 3, nvalid, sm, lane, p0, p1, p2);
    warp_store3(a.y + (size_t)e0 * 3, nvalid, sm, lane, y0, y1, y2);
  }
}

// out = A in, with up to two dot products of the result; WHICH = 0: v = A y, alpha = rho_new / (rh, v)
//                                                         WHICH = 1: t = A z, omega = (t, s) / (t, t)
template <int WHICH>
__global__ void __launch_bounds__(TPB) k_kry_spmv(KryArgs a) {
  if (a.ks[KS_DONE] != 0.0) return;
  __shared__ double smw[TPB / 32][96];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  double* sm = smw[wib];
  const size_t E = a.ld;   // plane stride
  const double* in = WHICH == 0 ? a.y : a.z;
  double* out = WHICH == 0 ? a.v : a.t;
  const double* other = WHICH == 0 ? a.rh : a.s;
  double d0 = 0, d1 = 0;
  for (int e0 = (blockIdx.x * (TPB / 32) + wib) * 32; e0 < a.E; e0 += gridDim.x * TPB) {
    const int nvalid = min(32, a.E - e0);
    const int e = e0 + lane;
    double s0 = 0, s1 = 0, s2 = 0, o0 = 0, o1 = 0, o2 = 0;
    warp_load3(other + (size_t)e0 * 3, nvalid, sm, lane, o0, o1, o2);
    if (lane < nvalid) {
#pragma unroll
      for (int bq = 0; bq < 4; ++bq) {
        const int c = __ldg(a.col + (size_t)bq * E + e);
        if (c < 0) continue;
        const double* v = a.val + (size_t)(bq * 9) * E + e;
        const double x0 = in[(size_t)c * 3], x1 = in[(size_t)c * 3 + 1], x2 = in[(size_t)c * 3 + 2];
        s0 += __ldg(v) * x0 + __ldg(v + E) * x1 + __ldg(v + 2 * E) * x2;
        s1 += __ldg(v + 3 * E) * x0 + __ldg(v + 4 * E) * x1 + __ldg(v + 5 * E) * x2;
        s2 += __ldg(v + 6 * E) * x0 + __ldg(v + 7 * E) * x1 + __ldg(v + 8 * E) * x2;
      }
      d0 += o0 * s0 + o1 * s1 + o2 * s2;
      if (WHICH == 1) d1 += s0 * s0 + s1 * s1 + s2 * s2;
    }
    warp_store3(out + (size_t)e0 * 3, nvalid, sm, lane, s0, s1, s2);
  }
  double t0, t1;
  if (grid_sum2(d0, d1, a.ks, t0, t1) && threadIdx.x == 0) {
    if (WHICH == 0) {
      if (t0 == 0.0) a.ks[KS_DONE] = 2.0; else a.ks[KS_ALPHA] = a.ks[KS_RHONEW] / t0;
    } else {
      a.ks[KS_OMEGA] = (t1 > 0.0) ? t0 / t1 : 0.0;
    }
  }
}

// s = r - alpha v ; z = Dinv s
__global__ void __launch_bounds__(TPB) k_kry_s(KryArgs a) {
  if (a.ks[KS_DONE] != 0.0) return;
  __shared__ double smw[TPB / 32][96];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  double* sm = smw[wib];
  const size_t E = a.ld;   // plane stride
  const double alpha = a.ks[KS_ALPHA];
  for (int e0 = (blockIdx.x * (TPB / 32) + wib) * 32; e0 < a.E; e0 += gridDim.x * TPB) {
    const int nvalid = min(32, a.E - e0);
    const int e = e0 + lane;
    double r0 = 0, r1 = 0, r2 = 0, v0 = 0, v1 = 0, v2 = 0, z0 = 0, z1 = 0, z2 = 0;
    warp_load3(a.r + (size_t)e0 * 3, nvalid, sm, lane, r0, r1, r2);
    warp_load3(a.v + (size_t)e0 * 3, nvalid, sm, lane, v0, v1, v2);
    const double s0 = r0 - alpha * v0, s1 = r1 - alpha * v1, s2 = r2 - alpha * v2;
    if (lane < nvalid) {
      const double* d = a.dinv + e;
      z0 = __ldg(d) * s0 + __ldg(d + E) * s1 + __ldg(d + 2 * E) * s2;
      z1 = __ldg(d + 3 * E) * s0 + __ldg(d + 4 * E) * s1 + __ldg(d + 5 * E) * s2;
      z2 = __ldg(d + 6 * E) * s0 + __ldg(d + 7 * E) * s1 + __ldg(d + 8 * E) * s2;
    }
    warp_store3(a.s + (size_t)e0 * 3, nvalid, sm, lane, s0, s1, s2);
    warp_store3(a.z + (size_t)e0 * 3, nvalid, sm, lane, z0, z1, z2);
  }
}

// x += alpha y + omega z ; r = s - omega t ; rr = (r, r) ; rho <- rho_new ; rho_new = (rh, r) ; convergence / breakdown
__global__ void __launch_bounds__(TPB, 6) k_kry_x(KryArgs a) {   // (unbounded the unroller took 110 registers: 2 CTAs per SM)
  if (a.ks[KS_DONE] != 0.0) return;
  const double alpha = a.ks[KS_ALPHA], omega = a.ks[KS_OMEGA];
  const long long n = 3LL * a.E;
  double d0 = 0, d1 = 0;
  for (long long i = (long long)blockIdx.x * TPB + threadIdx.x; i < n; i += (long long)gridDim.x * TPB) {
    a.x[i] = a.x[i] + alpha * a.y[i] + omega * a.z[i];
    const double r = a.s[i] + (-omega) * a.t[i];
    a.r[i] = r;
    d0 += r * r; d1 += a.rh[i] * r;
  }
  double rr, rho_new;
  if (grid_sum2(d0, d1, a.ks, rr, rho_new) && threadIdx.x == 0) {
    a.ks[KS_RR] = rr; a.ks[KS_RHO] = a.ks[KS_RHONEW]; a.ks[KS_RHONEW] = rho_new;
    const double it = a.ks[KS_ITER] + 1.0;
    a.ks[KS_ITER] = it;
    if (rr <= a.ks[KS_STOP2] || it >= a.ks[KS_MAXIT]) a.ks[KS_DONE] = 1.0;
    else if (rho_new == 0.0 || omega == 0.0) a.ks[KS_DONE] = 2.0;      // breakdown: report what was reached
  }
}

// Petrov-Galerkin residual-based stabilisation (transport_tri_unstr.F90:239-267,278): one thread per element.
// For P1 the gradient of T and inv_jac are constant over the element; rgi differs per Gauss point through T(gi).
// mode 0: write diff_coe (3 per element) and stab (9 per element), both in ABI order [E][..].
// mode 1: additionally write diagonal block = diag0 + stab into the block-CSR planes and refresh its inverse.
struct StabArgs {
  const double* X; const double* tnew; const double* told;
  double* diff_coe; double* stab; const double* diag0; double* val; double* dinv;
  double dt, ux, uy;
  size_t ld;
  int E, mode;
  const double* U;   // velocity planes (FIELD only): ugi(g) = sum_l n(g,l) u(:,l)
};

template <bool FIELD>
__global__ void __launch_bounds__(TPB) k_unstr_stab(StabArgs a) {
  const double toler = 0.00000000001;
  const size_t E = a.ld;   // plane stride
  for (int e = blockIdx.x * TPB + threadIdx.x; e < a.E; e += gridDim.x * TPB) {
    const double x1 = __ldg(a.X + e), y1 = __ldg(a.X + E + e), x2 = __ldg(a.X + 2 * E + e), y2 = __ldg(a.X + 3 * E + e),
                 x3 = __ldg(a.X + 4 * E + e), y3 = __ldg(a.X + 5 * E + e);
    const double A = x1 - x3, B = y1 - y3, C = x2 - x3, D = y2 - y3;
    const double detj = A * D - B * C;
    const double dw = 0.5 * fabs(detj) * (1.0 / 3.0);
    const double a11 = D / detj, a21 = -C / detj, a12 = -B / detj, a22 = A / detj;
    // nx(g,1,l) = a11 nlx1 + a12 nlx2 ; nx(g,2,l) = a21 nlx1 + a22 nlx2 with nlx1 = (1,0,-1), nlx2 = (0,1,-1)
    const double gx[3] = {a11 * 1.0 + a12 * 0.0, a11 * 0.0 + a12 * 1.0, a11 * -1.0 + a12 * -1.0};
    const double gy[3] = {a21 * 1.0 + a22 * 0.0, a21 * 0.0 + a22 * 1.0, a21 * -1.0 + a22 * -1.0};
    const double tn[3] = {a.tnew[(size_t)e * 3], a.tnew[(size_t)e * 3 + 1], a.tnew[(size_t)e * 3 + 2]};
    const double to[3] = {a.told[(size_t)e * 3], a.told[(size_t)e * 3 + 1], a.told[(size_t)e * 3 + 2]};
    double tx = 0.0, ty = 0.0;
#pragma unroll
    for (int l = 0; l < 3; ++l) { tx += gx[l] * tn[l]; ty += gy[l] * tn[l]; }
    const double g2 = tx * tx + ty * ty;
    const double N[3][3] = {{0.5, 0.5, 0.0}, {0.0, 0.5, 0.5}, {0.5, 0.0, 0.5}};   // n(gi, iloc), ShapFun.F90:1038-1040
    double ux[3], uy[3];
    if constexpr (FIELD) load_vel(a.U, E, (size_t)e, ux, uy);
    double dc[3];
#pragma unroll
    for (int g = 0; g < 3; ++g) {
      double ugx = 0.0, ugy = 0.0, tgi = 0.0, togi = 0.0;
#pragma unroll
      for (int l = 0; l < 3; ++l) {
        if constexpr (FIELD) { ugx += N[g][l] * ux[l]; ugy += N[g][l] * uy[l]; }
        else { ugx += N[g][l] * a.ux; ugy += N[g][l] * a.uy; }
        tgi += N[g][l] * tn[l]; togi += N[g][l] * to[l];
      }
      const double rgi = (tgi - togi) / a.dt + (ugx * tx + ugy * ty);
      const double ac = rgi / fmax(toler, g2);
      const double as1 = ac * tx, as2 = ac * ty;
      double ps = fmax(fabs(as1 * a11 + as2 * a12), fabs(as1 * a21 + as2 * a22));
      ps = fmin(1.0 / toler, 0.25 / ps);
      dc[g] = 0.25 * rgi * rgi * ps / fmax(toler, g2);
    }
    double st[9];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        double v = 0.0;
#pragma unroll
        for (int g = 0; g < 3; ++g) v += dc[g] * (gx[j] * gx[i] + gy[j] * gy[i]) * dw;
        st[i * 3 + j] = v;
      }
    if (a.diff_coe) { a.diff_coe[(size_t)e * 3] = dc[0]; a.diff_coe[(size_t)e * 3 + 1] = dc[1]; a.diff_coe[(size_t)e * 3 + 2] = dc[2]; }
    if (a.stab)
#pragma unroll
      for (int q = 0; q < 9; ++q) a.stab[(size_t)e * 9 + q] = st[q];
    if (a.mode == 1) {
      double d[9];
#pragma unroll
      for (int q = 0; q < 9; ++q) { d[q] = a.diag0[(size_t)q * E + e] + st[q]; a.val[(size_t)q * E + e] = d[q]; }
      const double c00 = d[4] * d[8] - d[5] * d[7], c01 = d[5] * d[6] - d[3] * d[8], c02 = d[3] * d[7] - d[4] * d[6];
      const double id = 1.0 / (d[0] * c00 + d[1] * c01 + d[2] * c02);
      double o[9];
      o[0] = c00 * id; o[1] = (d[2] * d[7] - d[1] * d[8]) * id; o[2] = (d[1] * d[5] - d[2] * d[4]) * id;
      o[3] = c01 * id; o[4] = (d[0] * d[8] - d[2] * d[6]) * id; o[5] = (d[2] * d[3] - d[0] * d[5]) * id;
      o[6] = c02 * id; o[7] = (d[1] * d[6] - d[0] * d[7]) * id; o[8] = (d[0] * d[4] - d[1] * d[3]) * id;
#pragma unroll
      for (int q = 0; q < 9; ++q) a.dinv[(size_t)q * E + e] = o[q];
    }
  }
}

inline int implicit_assemble(UnstrDev& u, double dt, double ux, double uy, double kdiff, int use_dir, int nsm, cudaStream_t st,
                             long long& nlaunch, std::string& err) {
  const size_t E = (size_t)u.E, ld = u.ld;
  if (!u.bsr_val) {
    UCK(cudaMalloc(&u.bsr_val, ld * 36 * sizeof(double)));
    UCK(cudaMalloc(&u.bsr_col, ld * 4 * sizeof(int32_t)));
    UCK(cudaMalloc(&u.dinv, ld * 9 * sizeof(double)));
    UCK(cudaMalloc(&u.mdt, E * sizeof(double)));
    UCK(cudaMalloc(&u.work, E * 3 * 9 * sizeof(double)));
    UCK(cudaMalloc(&u.dots, (size_t)(KS_PARTIAL + 2 * nsm * 8 + 2) * sizeof(double)));
    UCK(cudaMemsetAsync(u.dots, 0, (size_t)(KS_PARTIAL + 2 * nsm * 8 + 2) * sizeof(double), st));
    UCK(cudaMallocHost(&u.dots_host, KS_PARTIAL * sizeof(double)));
    UCK(cudaMalloc(&u.stab, E * 12 * sizeof(double)));
  }
  BsrArgs a;
  a.X = u.X; a.neig = u.neig; a.nside = u.nside; a.pen = u.pen; a.val = u.bsr_val; a.col = u.bsr_col; a.dinv = u.dinv;
  a.mdt = u.mdt;
  a.inv24dt = 1.0 / (24.0 * dt); a.ux = ux; a.uy = uy; a.kdiff = kdiff; a.ld = ld; a.E = u.E; a.use_dir = use_dir; a.U = u.U;
  if (u.U) k_assemble_bsr<true><<<stream_grid(k_assemble_bsr<true>, u.occ_assemble_f, u.E, nsm), TPB, 0, st>>>(a);
  else k_assemble_bsr<false><<<stream_grid(k_assemble_bsr<false>, u.occ_assemble, u.E, nsm), TPB, 0, st>>>(a);
  nlaunch++;
  UCK(cudaGetLastError());
  u.assembled = true; u.dt = dt; u.ux = ux; u.uy = uy; u.kdiff = kdiff;
  return PAMG_OK;
}

// time loop of unstr_implicit (:214-387): told = tnew ; rhs = (M/dt) told ; solve (lhs + flux) tnew = rhs, started
// from told, stopped at ||r|| <= tol ||rhs|| (or after max_iters iterations / on a breakdown of the recurrence).
// The host reads the convergence flag once per batch of KRY_BATCH iterations (kernels of a finished solve return at once).
constexpr int KRY_BATCH = 16;
inline int implicit_step(UnstrDev& u, int ntime, int nits, double tol, int max_iters, int* iters_total, double* relres,
                         int nsm, cudaStream_t st, long long& nlaunch, std::string& err, long long* host_syncs = nullptr) {
  const int E = u.E;
  const long long n = 3LL * E;
  const int g_apply = stream_grid(k_block_apply, u.occ_apply, E, nsm);
  const int g_stab = u.U ? stream_grid(k_unstr_stab<true>, u.occ_stab_f, E, nsm) : stream_grid(k_unstr_stab<false>, u.occ_stab, E, nsm);
  const int g_init = stream_grid(k_kry_init, u.occ_kry[0], E, nsm), g_p = stream_grid(k_kry_p, u.occ_kry[1], E, nsm);
  const int g_v = stream_grid(k_kry_spmv<0>, u.occ_kry[2], E, nsm), g_s = stream_grid(k_kry_s, u.occ_kry[3], E, nsm);
  const int g_t = stream_grid(k_kry_spmv<1>, u.occ_kry[4], E, nsm), g_x = stream_grid(k_kry_x, u.occ_kry[5], E, nsm);
  double* W = u.work;
  KryArgs a;
  a.val = u.bsr_val; a.col = u.bsr_col; a.dinv = u.dinv; a.ks = u.dots; a.E = E; a.ld = u.ld;
  a.b = W; a.r = W + n; a.rh = W + 2 * n; a.p = W + 3 * n; a.v = W + 4 * n; a.s = W + 5 * n; a.t = W + 6 * n; a.y = W + 7 * n;
  a.z = W + 8 * n;
  int total = 0;
  double worst = 0.0;
  const double maxit = (double)max_iters;
  for (int it = 0; it < ntime; ++it) {
    for (int k = 0; k < nits; ++k) {
      a.x = u.T[u.cur];
      // the scheme is linear and rhs depends on told only: passes k > 0 of the reference's nonlinear loop re-solve
      // the same system, which here starts converged and costs one residual evaluation
      if (k == 0) {
        UCK(cudaMemcpyAsync(u.told, a.x, (size_t)n * sizeof(double), cudaMemcpyDeviceToDevice, st));
        k_block_apply<<<g_apply, TPB, 0, st>>>(u.dinv, u.mdt, u.told, a.b, E, u.ld, 1); nlaunch++;
      }
      if (u.with_stab) {   // INTENDED use (:367-368 commented at HEAD): diagonal blocks += stab(tnew_nonlin, told)
        StabArgs sa;
        sa.X = u.X; sa.tnew = a.x; sa.told = u.told; sa.diff_coe = u.stab + (size_t)E * 9; sa.stab = u.stab; sa.diag0 = u.diag0;
        sa.val = u.bsr_val; sa.dinv = u.dinv; sa.dt = u.dt; sa.ux = u.ux; sa.uy = u.uy; sa.ld = u.ld; sa.E = E; sa.mode = 1;
        sa.U = u.U;
        if (u.U) k_unstr_stab<true><<<g_stab, TPB, 0, st>>>(sa);
        else k_unstr_stab<false><<<g_stab, TPB, 0, st>>>(sa);
        nlaunch++;
      }
      UCK(cudaMemcpyAsync(u.dots + KS_MAXIT, &maxit, sizeof(double), cudaMemcpyHostToDevice, st));
      k_kry_init<<<g_init, TPB, 0, st>>>(a, tol); nlaunch++;
      for (;;) {
        for (int j = 0; j < KRY_BATCH; ++j) {
          k_kry_p<<<g_p, TPB, 0, st>>>(a);
          k_kry_spmv<0><<<g_v, TPB, 0, st>>>(a);
          k_kry_s<<<g_s, TPB, 0, st>>>(a);
          k_kry_spmv<1><<<g_t, TPB, 0, st>>>(a);
          k_kry_x<<<g_x, TPB, 0, st>>>(a);
          nlaunch += 5;
        }
        UCK(cudaMemcpyAsync(u.dots_host, u.dots, KS_PARTIAL * sizeof(double), cudaMemcpyDeviceToHost, st));
        UCK(cudaStreamSynchronize(st));
        if (host_syncs) ++*host_syncs;
        if (u.dots_host[KS_DONE] != 0.0) break;
      }
      UCK(cudaGetLastError());
      total += (int)u.dots_host[KS_ITER];
      const double bb = u.dots_host[KS_BB], rr = u.dots_host[KS_RR];
      const double rel = bb > 0.0 ? sqrt(rr / bb) : 0.0;
      worst = std::max(worst, rel);
    }
  }
  if (iters_total) *iters_total = total;
  if (relres) *relres = worst;
  return PAMG_OK;
}

// ------------------------------------------------------------------------------------------------
// trans_rec (transport_rect.F90:122-316): explicit DG on bilinear quadrilaterals of a structured rectangular grid,
// one thread per element.  Shape functions of RE2DN4 (ShapFun.F90:72-215, 2x2 Gauss points), face tables of
// surface_pointers_sn (:305-357), neighbours of ele_info (structured_meshgen.F90:19-67) by index arithmetic, det_nlx
// (:1245-1300) and det_snlx_all / NORMGI (:1554-1590, :2012-2054).  volume_term = 0 is HEAD (tnew_gi is never set, :157).
struct RectArgs {
  const double* tin; const double* told; double* tout;
  double dx, dy, dt, ux, uy;
  int ner, nec, njac, direct, volume_term;
};

__global__ void __launch_bounds__(128) k_rect_explicit(RectArgs a) {
  const int totele = a.ner * a.nec;
  const double posi = 0.57735026918962584;     // 1 / sqrt(3)
  const double lxp[4] = {-1, 1, -1, 1}, lyp[4] = {-1, -1, 1, 1}, lx[2] = {-posi, posi};
  const int FN[4][2] = {{1, 0}, {0, 2}, {3, 1}, {2, 3}}, FN2[4][2] = {{3, 2}, {1, 3}, {2, 0}, {0, 1}};   // 0-based
  for (int e = blockIdx.x * 128 + threadIdx.x; e < totele; e += gridDim.x * 128) {
    const int ele = e + 1;
    const int row = (ele + a.ner - 1) / a.ner, col = ele - a.ner * (row - 1);
    const double xl[4][2] = {{a.dx * (col - 1), a.dy * (row - 1)}, {a.dx * col, a.dy * (row - 1)},
                             {a.dx * (col - 1), a.dy * row}, {a.dx * col, a.dy * row}};
    double n[4][4], nx[4][2][4], detwei[4];
#pragma unroll
    for (int q = 0; q < 2; ++q)
#pragma unroll
      for (int pq = 0; pq < 2; ++pq) {
        const int g = q * 2 + pq;
        double nlx[2][4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          n[g][c] = 0.25 * (1.0 + lxp[c] * lx[pq]) * (1.0 + lyp[c] * lx[q]);
          nlx[0][c] = 0.25 * lxp[c] * (1.0 + lyp[c] * lx[q]);
          nlx[1][c] = 0.25 * lyp[c] * (1.0 + lxp[c] * lx[pq]);
        }
        double A = 0, B = 0, Cc = 0, D = 0;
#pragma unroll
        for (int l = 0; l < 4; ++l) { A += nlx[0][l] * xl[l][0]; B += nlx[0][l] * xl[l][1]; Cc += nlx[1][l] * xl[l][0]; D += nlx[1][l] * xl[l][1]; }
        const double detj = A * D - B * Cc;
        detwei[g] = fabs(detj);
        const double a11 = D / detj, a21 = -B / detj, a12 = -Cc / detj, a22 = A / detj;
#pragma unroll
        for (int l = 0; l < 4; ++l) { nx[g][0][l] = a11 * nlx[0][l] + a12 * nlx[1][l]; nx[g][1][l] = a21 * nlx[0][l] + a22 * nlx[1][l]; }
      }
    double tl[4], to[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) { tl[i] = a.tin[(size_t)e * 4 + i]; to[i] = a.told[(size_t)e * 4 + i]; }
    double mass[4][4], ml[4], rhs[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        double m = 0;
#pragma unroll
        for (int g = 0; g < 4; ++g) m += n[g][i] * n[g][j] * detwei[g];
        mass[i][j] = m;
      }
      double l = 0, r = 0;
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        l += n[g][i] * detwei[g];
        double ugx = 0, ugy = 0, tt = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) { ugx += n[g][k] * a.ux; ugy += n[g][k] * a.uy; tt += n[g][k] * tl[k]; }
        const double tg = a.volume_term ? tt : 0.0;
        r += nx[g][0][i] * ugx * tg * detwei[g];
        r += nx[g][1][i] * ugy * tg * detwei[g];
      }
      ml[i] = l; rhs[i] = r;
    }
#pragma unroll
    for (int f = 0; f < 4; ++f) {
      int e22;
      if (f == 0) e22 = ele - a.ner;
      else if (f == 1) { e22 = ele - 1; if ((e22 + a.ner - 1) / a.ner != row || e22 < 1) e22 = 0; }
      else if (f == 2) { e22 = ele + 1; if ((e22 + a.ner - 1) / a.ner != row) e22 = 0; }
      else { e22 = ele + a.ner; if (e22 > totele) e22 = 0; }
      const bool bnd = e22 <= 0;
      const int l1 = FN[f][0], l2 = FN[f][1], m1 = FN2[f][0], m2 = FN2[f][1];
      const double t2a = bnd ? 0.0 : a.tin[(size_t)(e22 - 1) * 4 + m1], t2b = bnd ? 0.0 : a.tin[(size_t)(e22 - 1) * 4 + m2];
      double norm[2], xs[2][2];
#pragma unroll
      for (int d = 0; d < 2; ++d) {
        xs[0][d] = 0; xs[1][d] = 0;
      }
      double sdet[2], snorm[2][2], tsg[2], tsg2[2], us[2][2], us2[2][2];
#pragma unroll
      for (int sg = 0; sg < 2; ++sg) {
        const double s1 = 0.5 * (1.0 - lx[sg]), s2 = 0.5 * (1.0 + lx[sg]);     // sn_orig(sg, 1:2)
        // sums over all four nodes in node order, like the reference (zeros for the nodes off the face)
        double ux_ = 0, uy_ = 0, ux2 = 0, uy2 = 0, xx = 0, xy = 0, tt = 0, tt2 = 0, dxl = 0, dyl = 0;
#pragma unroll
        for (int l = 0; l < 4; ++l) {
          const double fs = (l == l1) ? s1 : ((l == l2) ? s2 : 0.0);
          const double fs2 = (l == m1) ? s1 : ((l == m2) ? s2 : 0.0);
          const double fl = (l == l1) ? -0.5 : ((l == l2) ? 0.5 : 0.0);
          ux_ += fs * a.ux; uy_ += fs * a.uy; ux2 += fs2 * a.ux; uy2 += fs2 * a.uy;
          xx += fs * xl[l][0]; xy += fs * xl[l][1];
          tt += fs * tl[l];
          tt2 += fs2 * ((l == m1) ? t2a : ((l == m2) ? t2b : 0.0));
          dxl += fl * xl[l][0]; dyl += fl * xl[l][1];
        }
        us[sg][0] = ux_; us[sg][1] = uy_; us2[sg][0] = ux2; us2[sg][1] = uy2; xs[sg][0] = xx; xs[sg][1] = xy;
        tsg[sg] = tt; tsg2[sg] = tt2;
        sdet[sg] = sqrt(dyl * dyl + dxl * dxl);
        snorm[sg][0] = dyl; snorm[sg][1] = -dxl;
      }
#pragma unroll
      for (int d = 0; d < 2; ++d) norm[d] = (xs[0][d] + xs[1][d]) / 2.0 - (xl[0][d] + xl[1][d] + xl[2][d] + xl[3][d]) / 4.0;
#pragma unroll
      for (int sg = 0; sg < 2; ++sg) {
        const double ax = snorm[sg][0], ay = snorm[sg][1];
        const double rn = sqrt(ax * ax + ay * ay);
        const double sirn = copysign(1.0 / rn, ax * norm[0] + ay * norm[1]);
        const double nxs = sirn * ax, nys = sirn * ay;
        const double un = nxs * 0.5 * (us[sg][0] + us2[sg][0]) + nys * 0.5 * (us[sg][1] + us2[sg][1]);
        const double income = 0.5 + 0.5 * copysign(1.0, -un);
        const double s1 = 0.5 * (1.0 - lx[sg]), s2 = 0.5 * (1.0 + lx[sg]);
        const double scx = nxs * sdet[sg] * ((1.0 - income) * us[sg][0] * tsg[sg] + income * us2[sg][0] * tsg2[sg]);
        const double scy = nys * sdet[sg] * ((1.0 - income) * us[sg][1] * tsg[sg] + income * us2[sg][1] * tsg2[sg]);
        rhs[l1] -= s1 * scx; rhs[l2] -= s2 * scx;
        rhs[l1] -= s1 * scy; rhs[l2] -= s2 * scy;
      }
    }
    double out[4];
    double v[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) { double sm = 0;
#pragma unroll
      for (int j = 0; j < 4; ++j) sm += mass[i][j] * to[j];
      v[i] = sm + a.dt * rhs[i]; }
    if (a.direct) {
      // FINDInv on the 4x4 mass matrix (no zero pivots for a positive definite matrix), then M^-1 v
      double m[4][8];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) m[i][j] = (j < 4) ? mass[i][j] : ((i + 4) == j ? 1.0 : 0.0);
#pragma unroll
      for (int k = 0; k < 3; ++k)
#pragma unroll
        for (int j = k + 1; j < 4; ++j) {
          const double mm = m[j][k] / m[k][k];
#pragma unroll
          for (int i = 0; i < 8; ++i) if (i >= k) m[j][i] -= mm * m[k][i];
        }
#pragma unroll
      for (int i = 0; i < 4; ++i) { const double mm = m[i][i];
#pragma unroll
        for (int j = 0; j < 8; ++j) if (j >= i) m[i][j] /= mm; }
#pragma unroll
      for (int k = 2; k >= 0; --k)
#pragma unroll
        for (int i = 0; i <= k; ++i) { const double mm = m[i][k + 1];
#pragma unroll
          for (int j = 0; j < 8; ++j) if (j >= k) m[i][j] -= m[k + 1][j] * mm; }
#pragma unroll
      for (int i = 0; i < 4; ++i) { double sm = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) sm += m[i][4 + j] * v[j];
        out[i] = sm; }
    } else {
      double x4[4] = {tl[0], tl[1], tl[2], tl[3]};      // tnew_nonlin(:,ele) == tnew(:,ele) at this point (:126,297)
      for (int k = 0; k < a.njac; ++k) {
        double mt[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) { double sm = 0;
#pragma unroll
          for (int j = 0; j < 4; ++j) sm += mass[i][j] * x4[j];
          mt[i] = sm; }
#pragma unroll
        for (int i = 0; i < 4; ++i) x4[i] = (ml[i] * x4[i] - mt[i] + v[i]) / ml[i];
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) out[i] = x4[i];
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) a.tout[(size_t)e * 4 + i] = out[i];
  }
}

// time loop of trans_rec (:122-316): told = tnew ; nits x { tnew = tnew_nonlin ; element loop } ; returns ntime
inline int rect_run(double CFL, int ner, int nec, double x_length, double y_length, double ux, double uy, double time, int nits,
                    int njac, int direct, int volume_term, double* x_all, double* tnew_host, int* ntime_out, int nsm,
                    cudaStream_t st, long long& nlaunch, std::string& err) {
  const int totele = ner * nec;
  const double dx = x_length / ner, dy = y_length / nec, dt = CFL * dx;
  const int ntime = (int)(time / dt);
  std::vector<double> t0((size_t)totele * 4, 0.0);
  for (int ele = ner / 5; ele <= ner / 2; ++ele)                 // tnew(:, no_ele_row/5 : no_ele_row/2) = 1 (:83)
    if (ele >= 1 && ele <= totele) for (int i = 0; i < 4; ++i) t0[(size_t)(ele - 1) * 4 + i] = 1.0;
  if (x_all)
    for (int ele = 1; ele <= totele; ++ele) {
      const int row = (ele + ner - 1) / ner, col = ele - ner * (row - 1);
      double* x = x_all + (size_t)(ele - 1) * 8;
      x[0] = dx * (col - 1); x[1] = dy * (row - 1); x[2] = dx * col; x[3] = dy * (row - 1);
      x[4] = dx * (col - 1); x[5] = dy * row;       x[6] = dx * col; x[7] = dy * row;
    }
  double *T[2] = {nullptr, nullptr}, *told = nullptr;
  const size_t bytes = (size_t)totele * 4 * sizeof(double);
  auto done = [&]() { cudaFree(T[0]); cudaFree(T[1]); cudaFree(told); };
#define RCK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { err = std::string(#call) + ": " + cudaGetErrorString(e_); done(); return PAMG_ERR_CUDA; } } while (0)
  RCK(cudaMalloc(&T[0], bytes)); RCK(cudaMalloc(&T[1], bytes)); RCK(cudaMalloc(&told, bytes));
  RCK(cudaMemcpyAsync(T[0], t0.data(), bytes, cudaMemcpyHostToDevice, st));
  int cur = 0;
  const int grid = std::max(1, std::min((totele + 127) / 128, nsm * 8));
  for (int it = 0; it < ntime; ++it) {
    RCK(cudaMemcpyAsync(told, T[cur], bytes, cudaMemcpyDeviceToDevice, st));
    for (int k = 0; k < nits; ++k) {
      RectArgs a;
      a.tin = T[cur]; a.told = told; a.tout = T[cur ^ 1]; a.dx = dx; a.dy = dy; a.dt = dt; a.ux = ux; a.uy = uy;
      a.ner = ner; a.nec = nec; a.njac = njac; a.direct = direct; a.volume_term = volume_term;
      k_rect_explicit<<<grid, 128, 0, st>>>(a);
      nlaunch++;
      cur ^= 1;
    }
  }
  RCK(cudaGetLastError());
  RCK(cudaMemcpyAsync(tnew_host, T[cur], bytes, cudaMemcpyDeviceToHost, st));
  RCK(cudaStreamSynchronize(st));
  done();
  if (ntime_out) *ntime_out = ntime;
  return PAMG_OK;
}

// ------------------------------------------------------------------------------------------------
// FINDInv: Gauss-Jordan on [M I], NO partial pivoting; a zero pivot is repaired by ADDING the first lower
// row with a non-zero entry (matrices.F90:1661-1676); errorflag -1 when singular.
template <int N>
__global__ void __launch_bounds__(128) k_local_minv(const double* __restrict__ M, const double* __restrict__ rhs,
                                                     double* __restrict__ x, double* __restrict__ Minv,
                                                     int32_t* __restrict__ status, int batch) {
  for (int bi = blockIdx.x * 128 + threadIdx.x; bi < batch; bi += gridDim.x * 128) {
    double a[N][2 * N];
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
      for (int j = 0; j < 2 * N; ++j) a[i][j] = (j < N) ? M[((size_t)bi * N + i) * N + j] : ((i + N) == j ? 1.0 : 0.0);
    bool ok = true;
#pragma unroll
    for (int k = 0; k < N - 1; ++k) {
      if (ok && a[k][k] == 0.0) {
        // as written the reference only ever tries row k+1: a zero there returns "non-invertible" at once
        if (a[k + 1][k] != 0.0) {
#pragma unroll
          for (int j = 0; j < 2 * N; ++j) a[k][j] += a[k + 1][j];
        } else {
          ok = false;
        }
      }
      if (ok) {
#pragma unroll
        for (int j = k + 1; j < N; ++j) {
          const double m = a[j][k] / a[k][k];
#pragma unroll
          for (int i = 0; i < 2 * N; ++i) if (i >= k) a[j][i] -= m * a[k][i];
        }
      }
    }
#pragma unroll
    for (int i = 0; i < N; ++i) if (a[i][i] == 0.0) ok = false;
    if (ok) {
#pragma unroll
      for (int i = 0; i < N; ++i) {
        const double m = a[i][i];
#pragma unroll
        for (int j = 0; j < 2 * N; ++j) if (j >= i) a[i][j] /= m;
      }
#pragma unroll
      for (int k = N - 2; k >= 0; --k)
#pragma unroll
        for (int i = 0; i <= k; ++i) {
          const double m = a[i][k + 1];
#pragma unroll
          for (int j = 0; j < 2 * N; ++j) if (j >= k) a[i][j] -= a[k + 1][j] * m;
        }
    }
    if (status) status[bi] = ok ? 0 : -1;
    if (Minv)
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) Minv[((size_t)bi * N + i) * N + j] = ok ? a[i][N + j] : 0.0;
    if (x) {
#pragma unroll
      for (int i = 0; i < N; ++i) {
        double s = 0.0;
#pragma unroll
        for (int j = 0; j < N; ++j) s += a[i][N + j] * rhs[(size_t)bi * N + j];
        x[(size_t)bi * N + i] = ok ? s : 0.0;
      }
    }
  }
}

inline int local_minv(int n, int batch, const double* M, const double* rhs, double* x, double* Minv, int32_t* status,
                      int nsm, cudaStream_t st, long long& nlaunch, std::string& err) {
  double *dM = nullptr, *dr = nullptr, *dx = nullptr, *dI = nullptr;
  int32_t* ds = nullptr;
  const size_t nm = (size_t)batch * n * n, nv = (size_t)batch * n;
  int rc = PAMG_OK;
  auto done = [&]() { cudaFree(dM); cudaFree(dr); cudaFree(dx); cudaFree(dI); cudaFree(ds); };
#define MCK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { err = std::string(#call) + ": " + cudaGetErrorString(e_); done(); return PAMG_ERR_CUDA; } } while (0)
  MCK(cudaMalloc(&dM, nm * sizeof(double)));
  MCK(cudaMalloc(&ds, (size_t)batch * sizeof(int32_t)));
  MCK(cudaMemcpyAsync(dM, M, nm * sizeof(double), cudaMemcpyHostToDevice, st));
  if (rhs) {
    MCK(cudaMalloc(&dr, nv * sizeof(double))); MCK(cudaMalloc(&dx, nv * sizeof(double)));
    MCK(cudaMemcpyAsync(dr, rhs, nv * sizeof(double), cudaMemcpyHostToDevice, st));
  }
  if (Minv) MCK(cudaMalloc(&dI, nm * sizeof(double)));
  const int grid = std::max(1, std::min((batch + 127) / 128, nsm * 8));
  if (n == 3) k_local_minv<3><<<grid, 128, 0, st>>>(dM, dr, dx, dI, ds, batch);
  else if (n == 4) k_local_minv<4><<<grid, 128, 0, st>>>(dM, dr, dx, dI, ds, batch);
  else k_local_minv<6><<<grid, 128, 0, st>>>(dM, dr, dx, dI, ds, batch);
  nlaunch++;
  MCK(cudaGetLastError());
  if (x) MCK(cudaMemcpyAsync(x, dx, nv * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (Minv) MCK(cudaMemcpyAsync(Minv, dI, nm * sizeof(double), cudaMemcpyDeviceToHost, st));
  std::vector<int32_t> hs(batch);
  MCK(cudaMemcpyAsync(hs.data(), ds, (size_t)batch * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  MCK(cudaStreamSynchronize(st));
  for (int i = 0; i < batch; ++i) {
    if (status) status[i] = hs[i];
    if (hs[i] != 0) rc = PAMG_ERR_SINGULAR;
  }
  done();
  if (rc) err = "singular block (errorflag = -1)";
  return rc;
}

}  // namespace pamg
