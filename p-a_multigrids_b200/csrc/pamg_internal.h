// pamg_internal.h -- declarations shared by the host-side pieces of libpamg_cuda.so
#ifndef PAMG_INTERNAL_H
#define PAMG_INTERNAL_H
#include <cstdint>
#include <vector>

#include "pamg.h"

namespace pamg {

// parent triangles with the reference's Mesh%X / Neig / fNeig / Dir / region_id (Structures.F90:143-170)
struct Mesh {
  std::vector<double> X;  // [U][3][2]
  std::vector<int32_t> neig, fneig, dir, region;
  void build_neighbours();
  static int read_msh(const char* path, Mesh& out);
  static int synthetic(int kp, int G, Mesh& out);
};

// ---- distributed plan: which halo strips live where (host logic, no CUDA) ----------------------
// A rank owns parents [first, first+U_local).  Every (local parent, gmsh face) owns one halo strip.
// Strips of faces cut by the partition are stored first, grouped by peer and sorted by the canonical
// key of the face pair, so that the receive buffer of a peer IS a contiguous range of the strip array
// and both sides enumerate the shared faces in the same order.
struct HaloPlan {
  int U_local = 0, first = 0, nparts = 1, my_part = 0;
  std::vector<int32_t> strip_of;   // [U_local*3] strip index of (u,mf)
  std::vector<int32_t> dst_strip;  // [U_local*3] where my boundary children of (u,mf) are written:
                                   //   < nstrips : local strip ; >= nstrips : send slot ; -1 : domain boundary
  std::vector<int32_t> rev;        // [U_local*3] 1: slot S-p+1, 0: slot p  (splitting.F90:1256-1391)
  std::vector<int32_t> hmap;       // [U_local*3] strip entry coincident with my face nodes: a | b<<2
  std::vector<int32_t> nsrc;       // [U_local*3] where a sweep reads the exterior values of (u,mf) WITHOUT a strip: the neighbour
                                   //   parent's boundary children in the start-of-sweep field.  -1: strip (domain boundary or a
                                   //   face cut by the GPU partition); else hmap | rev_of_neighbour<<4 | (Nside-1)<<5 | q_local<<7
  std::vector<int32_t> cut_lf;     // (u*3+mf) of the faces cut by the partition, in strip order
  struct Peer { int part; int nfaces; int strip_begin; int send_begin; };
  std::vector<Peer> peers;
  int nstrips = 0, nsend = 0;
};
int build_halo_plan(int U_global, const double* X, const int32_t* neig, const int32_t* fneig, const int32_t* dir,
                    int halo_rule, int nparts, const int32_t* part_first, int my_part, HaloPlan& plan);

// flow levels of the upwind graph (pamg_flow_levels, pamg_plan.cpp)
int flow_levels(int E, const int32_t* neig, const int32_t* inflow_mask, int32_t* level, int32_t* order, int32_t* nlevels,
                int64_t* lagged);

}  // namespace pamg
#endif
