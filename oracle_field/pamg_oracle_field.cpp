// pamg_oracle_field.cpp -- the CPU oracle's unstructured entries with a nodal velocity field u_ele(2,3,E)
// (transport_tri_unstr.F90:105,131-134,227,303; the array crosses the unstructured boundary at :504-511).  Test
// infrastructure only, like the oracle.
//
// The oracle (oracle/pamg_oracle.cpp) is the fixed yardstick of the suite and stays as it is; this translation unit
// includes it, so the geometry (tri_det_nlx, face_geometry), the shape-function tables, FINDInv and the node pairing are
// the oracle's own code, and restates the bodies of orc_unstr_explicit, orc_unstr_implicit_assemble_diff, stab_element,
// orc_unstr_implicit and orc_unstr_implicit_stab line by line with the velocity read from the field:
//   ugi(g,d) = sum_i n(g,i) u(d,i,e)                                   (volume Gauss points)
//   us(s,d)  = sum_q sn(s,q) u(d,q,e),  us2(s,d) = sum_q sn2(s,q) u(d,q,npos)
//              us2 = 0 where sn2 = 0 (Nside = 0); us2 = us where npos = 0 and Nside >= 1 (sum2 * u for a constant field,
//              u_bc = u_ele in trans_rec)
//   income(s) = 1/2 + 1/2 sign(1, -n.(us + us2)/2) per face Gauss point.
// u_ele is in the reference's layout: flat index (e*3 + iloc)*2 + d.
#include "../oracle/pamg_oracle.cpp"

namespace {

inline double uel(const double* u_ele, int e, int iloc, int d) { return u_ele[((size_t)e * 3 + iloc) * 2 + d]; }

// sn, sn2 (rows: face Gauss points, columns: local nodes of the element / of the neighbour) of gmsh face f (1..3) of e
void face_tables(const double* X, int e, int f, int npos, int nside, int use_dir, double sn[2][3], double sn2[2][3]) {
  const double (*x)[2] = reinterpret_cast<const double (*)[2]>(&X[(size_t)e * 6]);
  for (int s = 0; s < 2; ++s)
    for (int q = 0; q < 3; ++q) { sn[s][q] = 0.0; sn2[s][q] = 0.0; }
  const int l1 = UN_FACE_NODES[f - 1][0] - 1, l2 = UN_FACE_NODES[f - 1][1] - 1;
  for (int s = 0; s < 2; ++s) { sn[s][l1] = TB.sn[s][0]; sn[s][l2] = TB.sn[s][1]; }
  const int N2[3][2] = {{3, 1}, {1, 2}, {2, 3}};
  if (nside >= 1) {
    int m1 = N2[nside - 1][0] - 1, m2 = N2[nside - 1][1] - 1;
    if (use_dir && npos != 0) {
      const double (*xn)[2] = reinterpret_cast<const double (*)[2]>(&X[(size_t)(npos - 1) * 6]);
      if (!are_equal2(xn[m1], x[l1])) std::swap(m1, m2);
    }
    for (int s = 0; s < 2; ++s) { sn2[s][m1] = TB.sn[s][0]; sn2[s][m2] = TB.sn[s][1]; }
  }
}

// both traces of the velocity at face Gauss point s
void face_velocity(const double* u_ele, int e, int npos, const double sn[2][3], const double sn2[2][3], int s, double us[2],
                   double us2[2]) {
  double sum2 = 0.0;
  for (int q = 0; q < 3; ++q) sum2 += sn2[s][q];
  for (int d = 0; d < 2; ++d) {
    us[d] = 0.0; us2[d] = 0.0;
    for (int q = 0; q < 3; ++q) us[d] += sn[s][q] * uel(u_ele, e, q, d);
    if (npos != 0)
      for (int q = 0; q < 3; ++q) us2[d] += sn2[s][q] * uel(u_ele, npos - 1, q, d);
  }
  if (npos == 0 && sum2 != 0.0) { us2[0] = us[0]; us2[1] = us[1]; }
}

void stab_element_field(const double x[3][2], const double* tn, const double* to, const double* u_ele, int e, double dt,
                        double diff_coe[3], double stab[9]) {
  const double toler = 0.00000000001;   // :93
  double nx[3][2][3], detwei[3];
  tri_det_nlx(x, nx, detwei);
  double A = 0, B = 0, C = 0, D = 0;
  for (int l = 0; l < 3; ++l) {
    A += TB.nlx[0][0][l] * x[l][0]; B += TB.nlx[0][0][l] * x[l][1];
    C += TB.nlx[0][1][l] * x[l][0]; D += TB.nlx[0][1][l] * x[l][1];
  }
  const double detj = A * D - B * C;
  const double ij[2][2] = {{D / detj, -C / detj}, {-B / detj, A / detj}};
  for (int g = 0; g < 3; ++g) {
    double ugi[2] = {0, 0}, txgi[2] = {0, 0}, tgi = 0, togi = 0;
    for (int l = 0; l < 3; ++l) {
      ugi[0] += TB.n[g][l] * uel(u_ele, e, l, 0); ugi[1] += TB.n[g][l] * uel(u_ele, e, l, 1);
      txgi[0] += nx[g][0][l] * tn[l]; txgi[1] += nx[g][1][l] * tn[l];
      tgi += TB.n[g][l] * tn[l]; togi += TB.n[g][l] * to[l];
    }
    const double rgi = (tgi - togi) / dt + (ugi[0] * txgi[0] + ugi[1] * txgi[1]);
    const double g2 = txgi[0] * txgi[0] + txgi[1] * txgi[1];
    const double a_coef = rgi / std::max(toler, g2);
    const double as[2] = {a_coef * txgi[0], a_coef * txgi[1]};
    double ps = 0.0;
    for (int d = 0; d < 2; ++d) ps = std::max(ps, std::fabs(as[0] * ij[0][d] + as[1] * ij[1][d]));
    ps = std::min(1.0 / toler, 0.25 / ps);
    diff_coe[g] = 0.25 * rgi * rgi * ps / std::max(toler, g2);
  }
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      double v = 0;
      for (int g = 0; g < 3; ++g) v += diff_coe[g] * (nx[g][0][j] * nx[g][0][i] + nx[g][1][j] * nx[g][1][i]) * detwei[g];
      stab[i * 3 + j] = v;
    }
}

}  // namespace

extern "C" {

// orc_unstr_explicit with the field
void orc_unstr_explicit_field(int E, const double* X, const int32_t* neig, const int32_t* fneig, const int32_t* /*dir*/,
                              const double* u_ele, double dt, int ntime, int nits, int njac_its, int exact_minv, int use_dir,
                              double t_bc, double* tnew) {
  std::vector<double> told((size_t)3 * E), tnl((size_t)3 * E);
  for (int it = 0; it < ntime; ++it) {
    std::copy(tnew, tnew + (size_t)3 * E, told.begin());
    std::copy(tnew, tnew + (size_t)3 * E, tnl.begin());
    for (int its = 0; its < nits; ++its) {
      std::copy(tnl.begin(), tnl.end(), tnew);
      for (int e = 0; e < E; ++e) {
        const double (*x)[2] = reinterpret_cast<const double (*)[2]>(&X[(size_t)e * 6]);
        double nx[3][2][3], detwei[3];
        tri_det_nlx(x, nx, detwei);
        const double* Tl = &tnew[(size_t)e * 3];
        const double* To = &told[(size_t)e * 3];
        double ugi[3][2], tgi[3];
        for (int g = 0; g < 3; ++g) {
          for (int d = 0; d < 2; ++d)
            ugi[g][d] = TB.n[g][0] * uel(u_ele, e, 0, d) + TB.n[g][1] * uel(u_ele, e, 1, d) + TB.n[g][2] * uel(u_ele, e, 2, d);
          tgi[g] = TB.n[g][0] * Tl[0] + TB.n[g][1] * Tl[1] + TB.n[g][2] * Tl[2];
        }
        double rhs[3] = {0, 0, 0}, mass[3][3], ml[3];
        for (int i = 0; i < 3; ++i) {
          for (int j = 0; j < 3; ++j) {
            double m = 0;
            for (int g = 0; g < 3; ++g) m += TB.n[g][i] * TB.n[g][j] * detwei[g];
            mass[i][j] = m;
          }
          ml[i] = 0;
          for (int g = 0; g < 3; ++g) ml[i] += TB.n[g][i] * detwei[g];
          for (int g = 0; g < 3; ++g)
            for (int d = 0; d < 2; ++d) rhs[i] += nx[g][d][i] * ugi[g][d] * tgi[g] * detwei[g];
        }
        for (int f = 1; f <= 3; ++f) {
          const int npos = neig[e * 3 + f - 1], nside = fneig[e * 3 + f - 1];
          double T2[3];
          if (npos != 0) for (int q = 0; q < 3; ++q) T2[q] = tnew[(size_t)(npos - 1) * 3 + q];
          else for (int q = 0; q < 3; ++q) T2[q] = t_bc;
          double sn[2][3], sn2[2][3];
          face_tables(X, e, f, npos, nside, use_dir, sn, sn2);
          double sdet[2], snorm[2][2];
          face_geometry(x, f, sdet, snorm);
          for (int s = 0; s < 2; ++s) {
            double ts = 0, t2s = 0;
            for (int q = 0; q < 3; ++q) { ts += sn[s][q] * Tl[q]; t2s += sn2[s][q] * T2[q]; }
            double us[2], us2[2];
            face_velocity(u_ele, e, npos, sn, sn2, s, us, us2);
            const double un = snorm[s][0] * 0.5 * (us[0] + us2[0]) + snorm[s][1] * 0.5 * (us[1] + us2[1]);
            const double income = 0.5 + 0.5 * std::copysign(1.0, -un);
            for (int d = 0; d < 2; ++d) {
              const double sc = snorm[s][d] * sdet[s] * ((1.0 - income) * us[d] * ts + income * us2[d] * t2s);
              for (int i = 0; i < 3; ++i) rhs[i] -= sn[s][i] * sc;
            }
          }
        }
        double* out = &tnl[(size_t)e * 3];
        if (exact_minv) {
          double inv[9], mt[3];
          findinv(&mass[0][0], inv, 3);
          for (int i = 0; i < 3; ++i) mt[i] = mass[i][0] * To[0] + mass[i][1] * To[1] + mass[i][2] * To[2];
          for (int i = 0; i < 3; ++i) {
            double o = 0;
            for (int j = 0; j < 3; ++j) o += inv[i * 3 + j] * (mt[j] + dt * rhs[j]);
            out[i] = o;
          }
        } else {
          double rj[3], tl[3] = {out[0], out[1], out[2]};
          for (int i = 0; i < 3; ++i) rj[i] = mass[i][0] * To[0] + mass[i][1] * To[1] + mass[i][2] * To[2] + dt * rhs[i];
          for (int jit = 0; jit < njac_its; ++jit) {
            double mt[3];
            for (int i = 0; i < 3; ++i) mt[i] = mass[i][0] * tl[0] + mass[i][1] * tl[1] + mass[i][2] * tl[2];
            for (int i = 0; i < 3; ++i) tl[i] = (ml[i] * tl[i] - mt[i] + rj[i]) / ml[i];
          }
          for (int i = 0; i < 3; ++i) out[i] = tl[i];
        }
      }
      std::copy(tnl.begin(), tnl.end(), tnew);
    }
  }
}

// orc_unstr_implicit_assemble_diff with the field.  literal_target = 1: HEAD's rule (:339-342), the whole face block into the
// columns of ONE target element chosen by income(1); literal_target = 0: per face Gauss point, the sn(s,j) part of an outflow
// point into the element's own columns and the sn2(s,j) part of an inflow point into the neighbour's (own columns when
// npos = 0) - what the device assembles.  For a uniform velocity both Gauss points agree and the two rules coincide.
void orc_unstr_implicit_assemble_diff_field(int E, const double* X, const int32_t* neig, const int32_t* fneig,
                                            const double* u_ele, double k, double dt, int use_dir, int literal_target,
                                            double* A, double* Mdt) {
  const size_t N = (size_t)3 * E;
  std::fill(A, A + N * N, 0.0);
  std::fill(Mdt, Mdt + N * N, 0.0);
  for (int e = 0; e < E; ++e) {
    const double (*x)[2] = reinterpret_cast<const double (*)[2]>(&X[(size_t)e * 6]);
    double nx[3][2][3], detwei[3];
    tri_det_nlx(x, nx, detwei);
    double ugi[3][2];
    for (int g = 0; g < 3; ++g)
      for (int d = 0; d < 2; ++d)
        ugi[g][d] = TB.n[g][0] * uel(u_ele, e, 0, d) + TB.n[g][1] * uel(u_ele, e, 1, d) + TB.n[g][2] * uel(u_ele, e, 2, d);
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) {
        double mass = 0, stiff = 0;
        for (int g = 0; g < 3; ++g) {
          mass += TB.n[g][i] * TB.n[g][j] * detwei[g] / dt;
          for (int d = 0; d < 2; ++d) stiff += nx[g][d][i] * ugi[g][d] * detwei[g] * TB.n[g][j];
        }
        double dvol = 0;
        for (int g = 0; g < 3; ++g)
          for (int d = 0; d < 2; ++d) dvol += k * nx[g][d][i] * detwei[g] * nx[g][d][j];
        Mdt[(size_t)(3 * e + i) * N + 3 * e + j] += mass;
        A[(size_t)(3 * e + i) * N + 3 * e + j] += mass - stiff + dvol;
      }
    for (int f = 1; f <= 3; ++f) {
      const int npos = neig[e * 3 + f - 1], nside = fneig[e * 3 + f - 1];
      const int l1 = UN_FACE_NODES[f - 1][0] - 1, l2 = UN_FACE_NODES[f - 1][1] - 1;
      double sn[2][3], sn2[2][3];
      face_tables(X, e, f, npos, nside, use_dir, sn, sn2);
      double sdet[2], snorm[2][2], income[2], us[2][2], us2[2][2];
      face_geometry(x, f, sdet, snorm);
      for (int s = 0; s < 2; ++s) {
        face_velocity(u_ele, e, npos, sn, sn2, s, us[s], us2[s]);
        const double un = snorm[s][0] * 0.5 * (us[s][0] + us2[s][0]) + snorm[s][1] * 0.5 * (us[s][1] + us2[s][1]);
        income[s] = 0.5 + 0.5 * std::copysign(1.0, -un);
      }
      const int nbr = (npos != 0) ? npos : e + 1;
      int target = (int)((1.0 - income[0]) * (e + 1) + income[0] * npos);   // :339
      if (target == 0) target = e + 1;                                      // :340-342
      for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
          double fo = 0, fn = 0;
          for (int d = 0; d < 2; ++d)
            for (int s = 0; s < 2; ++s) {
              fo += snorm[s][d] * sdet[s] * sn[s][i] * (1.0 - income[s]) * sn[s][j] * us[s][d];
              fn += snorm[s][d] * sdet[s] * sn[s][i] * income[s] * sn2[s][j] * us2[s][d];
            }
          if (literal_target) {
            A[(size_t)(3 * e + i) * N + 3 * (target - 1) + j] += fo + fn;
          } else {
            A[(size_t)(3 * e + i) * N + 3 * e + j] += fo;
            A[(size_t)(3 * e + i) * N + 3 * (nbr - 1) + j] += fn;
          }
        }
      if (k != 0.0) {
        const double cx = (x[0][0] + x[1][0] + x[2][0]) / 3, cy = (x[0][1] + x[1][1] + x[2][1]) / 3;
        double dx;
        if (npos != 0) {
          const double (*xn)[2] = reinterpret_cast<const double (*)[2]>(&X[(size_t)(npos - 1) * 6]);
          const double qx = (xn[0][0] + xn[1][0] + xn[2][0]) / 3, qy = (xn[0][1] + xn[1][1] + xn[2][1]) / 3;
          dx = std::sqrt((cx - qx) * (cx - qx) + (cy - qy) * (cy - qy));
        } else {
          const double mx = (x[l1][0] + x[l2][0]) / 2, my = (x[l1][1] + x[l2][1]) / 2;
          dx = std::sqrt((cx - mx) * (cx - mx) + (cy - my) * (cy - my));
        }
        for (int i = 0; i < 3; ++i)
          for (int j = 0; j < 3; ++j) {
            double my_d = 0, ng_d = 0;
            for (int s = 0; s < 2; ++s) {
              my_d += (k / dx) * sn[s][i] * sn[s][j] * sdet[s];
              ng_d += (k / dx) * sn[s][i] * sn2[s][j] * sdet[s];
            }
            A[(size_t)(3 * e + i) * N + 3 * e + j] += my_d;
            if (npos != 0) A[(size_t)(3 * e + i) * N + 3 * (npos - 1) + j] -= ng_d;
          }
      }
    }
  }
}

void orc_unstr_stab_field(int E, const double* X, const double* tnew, const double* told, const double* u_ele, double dt,
                          double* diff_coe, double* stab) {
  for (int e = 0; e < E; ++e)
    stab_element_field(reinterpret_cast<const double (*)[2]>(&X[(size_t)e * 6]), tnew + (size_t)e * 3, told + (size_t)e * 3,
                       u_ele, e, dt, diff_coe + (size_t)e * 3, stab + (size_t)e * 9);
}

// orc_unstr_implicit with the field (split face blocks, no diffusion)
int orc_unstr_implicit_field(int E, const double* X, const int32_t* neig, const int32_t* fneig, const double* u_ele, double dt,
                             int ntime, int nits, int use_dir, double* tnew) {
  const size_t N = (size_t)3 * E;
  std::vector<double> A(N * N), M(N * N), inv(N * N), rhs(N), told(N);
  orc_unstr_implicit_assemble_diff_field(E, X, neig, fneig, u_ele, 0.0, dt, use_dir, 0, A.data(), M.data());
  if (findinv(A.data(), inv.data(), (int)N) != 0) return -1;
  for (int it = 0; it < ntime; ++it) {
    std::copy(tnew, tnew + N, told.begin());
    for (int kk = 0; kk < nits; ++kk) {
      for (size_t i = 0; i < N; ++i) { double s = 0; for (size_t j = 0; j < N; ++j) s += M[i * N + j] * told[j]; rhs[i] = s; }
      for (size_t i = 0; i < N; ++i) { double s = 0; for (size_t j = 0; j < N; ++j) s += inv[i * N + j] * rhs[j]; tnew[i] = s; }
    }
  }
  return 0;
}

// orc_unstr_implicit_stab with the field
int orc_unstr_implicit_stab_field(int E, const double* X, const int32_t* neig, const int32_t* fneig, const double* u_ele,
                                  double dt, int ntime, int nits, int use_dir, double* tnew) {
  const size_t N = (size_t)3 * E;
  std::vector<double> A(N * N), As(N * N), M(N * N), inv(N * N), rhs(N), told(N), dc(N), st((size_t)9 * E);
  orc_unstr_implicit_assemble_diff_field(E, X, neig, fneig, u_ele, 0.0, dt, use_dir, 0, A.data(), M.data());
  for (int it = 0; it < ntime; ++it) {
    std::copy(tnew, tnew + N, told.begin());
    for (size_t i = 0; i < N; ++i) { double s = 0; for (size_t j = 0; j < N; ++j) s += M[i * N + j] * told[j]; rhs[i] = s; }
    for (int kk = 0; kk < nits; ++kk) {
      orc_unstr_stab_field(E, X, tnew, told.data(), u_ele, dt, dc.data(), st.data());
      As = A;
      for (int e = 0; e < E; ++e)
        for (int i = 0; i < 3; ++i)
          for (int j = 0; j < 3; ++j) As[(size_t)(3 * e + i) * N + 3 * e + j] += st[(size_t)e * 9 + i * 3 + j];
      if (findinv(As.data(), inv.data(), (int)N) != 0) return -1;
      for (size_t i = 0; i < N; ++i) { double s = 0; for (size_t j = 0; j < N; ++j) s += inv[i * N + j] * rhs[j]; tnew[i] = s; }
    }
  }
  return 0;
}

}  // extern "C"
