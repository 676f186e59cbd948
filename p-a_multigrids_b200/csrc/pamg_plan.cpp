// pamg_plan.cpp -- host logic of the halo ("overlaps") exchange: strip placement, slot reversal,
// face-node pairing and the per-peer ordering used by the multi-GPU path.  No CUDA in this file.
//
// Reference: update_overlaps (splitting.F90:1210-1397) writes the 3 nodal values of every boundary
// child of parent face f into the NEIGHBOUR parent's strip t_overlap(:, Nside), at slot p or S-p+1
// depending on (f, Nside==2, Dir(f)); the reader side is transport_tri_semi.F90:629-655.
#include <algorithm>
#include <cstring>

#include "pamg_internal.h"

namespace pamg {

namespace {
// nodes of an up child lying on parent side 1,2,3 (0-based node ids): Msh2Tri.F90:877-901
const int SIDE[3][2] = {{0, 2}, {0, 1}, {1, 2}};
// my two face nodes (a,b) in child-face order for parent side mf: child face 1:(1,3) 3:(2,1) 2:(3,2)
// (transport_tri_semi.F90:142-147 with the face map 1->1, 2->3, 3->2 of :629-638)
const int FACE_AB[3][2] = {{0, 2}, {1, 0}, {2, 1}};
// first vertex of the run of strip positions on each parent side: side 1 runs X3->X1, side 2 X1->X2,
// side 3 X3->X2 (splitting.F90:434-449)
const int RUN_START[3] = {2, 0, 2};

inline bool same_pt(const double* p, const double* q) { return p[0] == q[0] && p[1] == q[1]; }

// the 12-case table of splitting.F90:1256-1276 (face 1), :1297-1333 (face 3), :1354-1391 (face 2)
inline int literal_reversed(int mf /*0-based*/, int nside /*1-based*/, int dir) {
  if (mf == 1) return (nside == 2) ? (dir ? 0 : 1) : (dir ? 1 : 0);
  return (nside == 2) ? (dir ? 1 : 0) : (dir ? 0 : 1);
}
}  // namespace

int build_halo_plan(int U_global, const double* X, const int32_t* neig, const int32_t* fneig, const int32_t* dir,
                    int halo_rule, int nparts, const int32_t* part_first, int my_part, HaloPlan& plan) {
  if (U_global < 1 || !X || !neig || !fneig || !dir || nparts < 1 || my_part < 0 || my_part >= nparts)
    return PAMG_ERR_ARG;
  std::vector<int32_t> pf(nparts + 1);
  if (part_first) { for (int i = 0; i <= nparts; ++i) pf[i] = part_first[i]; }
  else { pf[0] = 0; pf[1] = U_global; if (nparts != 1) return PAMG_ERR_ARG; }
  if (pf[0] != 0 || pf[nparts] != U_global) return PAMG_ERR_ARG;
  for (int i = 0; i < nparts; ++i) if (pf[i + 1] < pf[i]) return PAMG_ERR_ARG;
  auto owner = [&](int g) { return (int)(std::upper_bound(pf.begin(), pf.end(), g) - pf.begin()) - 1; };

  plan = HaloPlan();
  plan.nparts = nparts; plan.my_part = my_part;
  plan.first = pf[my_part]; plan.U_local = pf[my_part + 1] - pf[my_part];
  const int UL = plan.U_local, first = plan.first;
  plan.strip_of.assign((size_t)UL * 3, -1);
  plan.dst_strip.assign((size_t)UL * 3, -1);
  plan.rev.assign((size_t)UL * 3, 0);
  plan.hmap.assign((size_t)UL * 3, 0);

  // cut faces, keyed by the (parent, face) of the lower-numbered side: both ranks sort identically
  struct Cut { int peer; int64_t key; int lf; };
  std::vector<Cut> cuts;
  for (int u = 0; u < UL; ++u)
    for (int mf = 0; mf < 3; ++mf) {
      const int g = first + u, lf = u * 3 + mf;
      const int q = neig[(size_t)g * 3 + mf];            // 1-based global, 0 = boundary
      const int a = FACE_AB[mf][0], b = FACE_AB[mf][1];
      if (q == 0) { plan.hmap[lf] = a | (b << 2); continue; }  // Dirichlet entries sit at my own node ids (:1246-1249)
      const int ns = fneig[(size_t)g * 3 + mf];
      if (ns < 1 || ns > 3 || q < 1 || q > U_global) return PAMG_ERR_ARG;
      const double* Xm = &X[(size_t)g * 6];
      const double* Xn = &X[(size_t)(q - 1) * 6];
      int na = -1, nb = -1;
      for (int c = 0; c < 2; ++c) {
        const int nn = SIDE[ns - 1][c];
        if (same_pt(Xn + 2 * nn, Xm + 2 * a)) na = nn;
        if (same_pt(Xn + 2 * nn, Xm + 2 * b)) nb = nn;
      }
      if (na < 0 || nb < 0) return PAMG_ERR_ARG;        // Neig/fNeig do not describe a shared edge
      plan.hmap[lf] = na | (nb << 2);
      const int geo = same_pt(Xm + 2 * RUN_START[mf], Xn + 2 * RUN_START[ns - 1]) ? 0 : 1;
      plan.rev[lf] = halo_rule == 0 ? literal_reversed(mf, ns, dir[(size_t)g * 3 + mf]) : geo;
      const int own = owner(q - 1);
      if (own != my_part) {
        const int64_t kmine = (int64_t)g * 3 + mf, ktheirs = (int64_t)(q - 1) * 3 + (ns - 1);
        cuts.push_back(Cut{own, std::min(kmine, ktheirs), lf});
      }
    }
  std::sort(cuts.begin(), cuts.end(), [](const Cut& x, const Cut& y) {
    return x.peer != y.peer ? x.peer < y.peer : x.key < y.key;
  });
  // strips of cut faces first (receive buffers), then everything else
  int next = 0;
  for (size_t i = 0; i < cuts.size(); ++i) {
    if (i == 0 || cuts[i].peer != cuts[i - 1].peer)
      plan.peers.push_back(HaloPlan::Peer{cuts[i].peer, 0, next, next});
    plan.peers.back().nfaces++;
    plan.strip_of[cuts[i].lf] = next++;
  }
  plan.nsend = next;
  plan.cut_lf.resize(cuts.size());
  for (size_t i = 0; i < cuts.size(); ++i) plan.cut_lf[i] = cuts[i].lf;
  for (int lf = 0; lf < UL * 3; ++lf)
    if (plan.strip_of[lf] < 0) plan.strip_of[lf] = next++;
  plan.nstrips = next;
  // destinations: the neighbour's strip (local) or my send slot in the same order as its receive range
  for (int u = 0; u < UL; ++u)
    for (int mf = 0; mf < 3; ++mf) {
      const int g = first + u, lf = u * 3 + mf;
      const int q = neig[(size_t)g * 3 + mf];
      if (q == 0) continue;
      const int ns = fneig[(size_t)g * 3 + mf];
      if (owner(q - 1) == my_part) plan.dst_strip[lf] = plan.strip_of[(q - 1 - first) * 3 + (ns - 1)];
      else plan.dst_strip[lf] = plan.nstrips + plan.strip_of[lf];  // send slot i <-> my cut strip i
    }
  // strip-free read of a local neighbour: slot p of my strip is written by the neighbour's child at position p or S-1-p
  // according to the NEIGHBOUR's reversal flag (splitting.F90:1256-1391), entries in its local node order
  plan.nsrc.assign((size_t)UL * 3, -1);
  for (int u = 0; u < UL; ++u)
    for (int mf = 0; mf < 3; ++mf) {
      const int g = first + u, lf = u * 3 + mf;
      const int q = neig[(size_t)g * 3 + mf];
      if (q == 0 || owner(q - 1) != my_part) continue;
      const int ns = fneig[(size_t)g * 3 + mf];
      const int ql = q - 1 - first;
      if (ql >= (1 << 24)) continue;                       // does not fit the descriptor: keep the strip
      plan.nsrc[lf] = plan.hmap[lf] | (plan.rev[ql * 3 + (ns - 1)] << 4) | ((ns - 1) << 5) | (ql << 7);
    }
  return PAMG_OK;
}

}  // namespace pamg

extern "C" int pamg_halo_plan(int U_global, const double* X, const int32_t* neig, const int32_t* fneig,
                              const int32_t* dir, int halo_rule, int nparts, const int32_t* part_first,
                              int my_part, int32_t* strip_of, int32_t* dst_strip, int32_t* rev, int32_t* hmap,
                              int32_t* peers, int32_t* counts) {
  pamg::HaloPlan p;
  int rc = pamg::build_halo_plan(U_global, X, neig, fneig, dir, halo_rule, nparts, part_first, my_part, p);
  if (rc != PAMG_OK) return rc;
  const size_t n = (size_t)p.U_local * 3;
  if (strip_of) std::memcpy(strip_of, p.strip_of.data(), n * 4);
  if (dst_strip) std::memcpy(dst_strip, p.dst_strip.data(), n * 4);
  if (rev) std::memcpy(rev, p.rev.data(), n * 4);
  if (hmap) std::memcpy(hmap, p.hmap.data(), n * 4);
  if (peers)
    for (size_t i = 0; i < p.peers.size(); ++i) {
      peers[i * 4 + 0] = p.peers[i].part; peers[i * 4 + 1] = p.peers[i].nfaces;
      peers[i * 4 + 2] = p.peers[i].strip_begin; peers[i * 4 + 3] = p.peers[i].send_begin;
    }
  if (counts) { counts[0] = (int32_t)p.peers.size(); counts[1] = p.nstrips; counts[2] = p.nsend; counts[3] = p.U_local; counts[4] = p.first; }
  return PAMG_OK;
}

// ---- flow levels of the upwind graph (the order of the flow-ordered block Gauss-Seidel preconditioner) -----------------
// Edge c -> e for every face f of e with bit f of inflow_mask[e] set and a neighbour c = neig[e][f] - 1.  level[e] = the
// longest upwind path ending at e (Kahn's algorithm, O(E)).  When the queue runs dry before every element has a level, the
// graph has a cycle: the lowest-index element left gets 1 + the largest level of its already levelled upstream neighbours (0
// if it has none) and enters the queue.  lagged = the edges whose source level is not below their target's: the sweep
// treats those blocks as zero.  order = the elements sorted by (level, index).
int pamg::flow_levels(int E, const int32_t* neig, const int32_t* inflow_mask, int32_t* level, int32_t* order,
                      int32_t* nlevels, int64_t* lagged) {
  if (E < 1 || !neig || !inflow_mask || !level || !order) return PAMG_ERR_ARG;
  std::vector<int32_t> indeg((size_t)E, 0), first((size_t)E + 1, 0), succ;
  for (int e = 0; e < E; ++e)
    for (int f = 0; f < 3; ++f) {
      const int q = neig[(size_t)e * 3 + f];
      if (q < 0 || q > E) return PAMG_ERR_ARG;
      if (q != 0 && ((inflow_mask[e] >> f) & 1)) { ++indeg[e]; ++first[q]; }
    }
  for (int e = 0; e < E; ++e) first[e + 1] += first[e];
  succ.resize((size_t)first[E]);
  {
    std::vector<int32_t> fill(first.begin(), first.end() - 1);
    for (int e = 0; e < E; ++e)
      for (int f = 0; f < 3; ++f) {
        const int q = neig[(size_t)e * 3 + f];
        if (q != 0 && ((inflow_mask[e] >> f) & 1)) succ[(size_t)fill[q - 1]++] = e;
      }
  }
  std::vector<int32_t> queue;
  queue.reserve((size_t)E);
  std::vector<char> placed((size_t)E, 0);
  for (int e = 0; e < E; ++e) {
    level[e] = 0;
    if (indeg[e] == 0) { queue.push_back(e); placed[e] = 1; }
  }
  size_t head = 0;
  int next_free = 0;                       // every element below it is placed
  while (queue.size() < (size_t)E || head < queue.size()) {
    if (head == queue.size()) {            // cycle: the lowest-index element left; level[] already holds 1 + max upstream
      while (placed[next_free]) ++next_free;
      queue.push_back(next_free); placed[next_free] = 1;
    }
    const int c = queue[head++];
    for (int32_t i = first[c]; i < first[c + 1]; ++i) {
      const int e = succ[(size_t)i];
      if (placed[e]) continue;             // an edge into an element placed earlier by the cycle rule
      level[e] = std::max(level[e], level[c] + 1);
      if (--indeg[e] == 0) { queue.push_back(e); placed[e] = 1; }
    }
  }
  int32_t nl = 0;
  int64_t lag = 0;
  for (int e = 0; e < E; ++e) {
    nl = std::max(nl, level[e] + 1);
    for (int f = 0; f < 3; ++f) {
      const int q = neig[(size_t)e * 3 + f];
      if (q != 0 && ((inflow_mask[e] >> f) & 1) && level[q - 1] >= level[e]) ++lag;
    }
  }
  std::vector<int32_t> start((size_t)nl + 1, 0);
  for (int e = 0; e < E; ++e) ++start[(size_t)level[e] + 1];
  for (int l = 0; l < nl; ++l) start[(size_t)l + 1] += start[(size_t)l];
  for (int e = 0; e < E; ++e) order[start[(size_t)level[e]]++] = e;
  if (nlevels) *nlevels = nl;
  if (lagged) *lagged = lag;
  return PAMG_OK;
}

extern "C" int pamg_flow_levels(int E, const int32_t* neig, const int32_t* inflow_mask, int32_t* level, int32_t* order,
                                int32_t* nlevels, int64_t* lagged) {
  return pamg::flow_levels(E, neig, inflow_mask, level, order, nlevels, lagged);
}
