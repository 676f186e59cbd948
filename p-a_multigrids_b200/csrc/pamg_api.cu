// pamg_api.cu -- handle, device memory and the C ABI of libpamg_cuda.so (see include/pamg.h).
// Host orchestration mirrors the contained procedures of Semi_implicit_iterative
// (transport_tri_semi.F90:407-889) and its V-cycle loop (:319-379).  No CPU fallback: every compute
// entry fails with PAMG_ERR_CUDA when no device is present.
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "pamg_internal.h"
#include "pamg_kernels.cuh"
#include "pamg_unstr.cuh"

using namespace pamg;

// ------------------------------------------------------------------ NCCL, bound lazily with dlopen
// (libnccl.so.2; the few entry points used for the halo exchange and the norm all-reduce)
namespace {
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
enum { ncclUint8 = 1, ncclInt32 = 2, ncclFloat64 = 8, ncclSum = 0, ncclMax = 2, ncclMin = 3, ncclSuccess = 0 };
struct NcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(ncclUniqueId*) = nullptr;
  int (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  int (*CommDestroy)(ncclComm_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  int (*Send)(const void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*Recv)(void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  bool load() {
    if (lib) return true;
    lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) return false;
    GetUniqueId = (decltype(GetUniqueId))dlsym(lib, "ncclGetUniqueId");
    CommInitRank = (decltype(CommInitRank))dlsym(lib, "ncclCommInitRank");
    CommDestroy = (decltype(CommDestroy))dlsym(lib, "ncclCommDestroy");
    GroupStart = (decltype(GroupStart))dlsym(lib, "ncclGroupStart");
    GroupEnd = (decltype(GroupEnd))dlsym(lib, "ncclGroupEnd");
    Send = (decltype(Send))dlsym(lib, "ncclSend");
    Recv = (decltype(Recv))dlsym(lib, "ncclRecv");
    AllReduce = (decltype(AllReduce))dlsym(lib, "ncclAllReduce");
    return GetUniqueId && CommInitRank && CommDestroy && GroupStart && GroupEnd && Send && Recv && AllReduce;
  }
};
NcclApi g_nccl;
}  // namespace

// Kernels of different GPUs (or of two parts on one GPU) wait for each other's stores inside the halo exchange.  With lazy
// module loading the FIRST launch of a function can block until running kernels have finished - a deadlock if the running
// kernel is the one that waits.  Ask for eager loading unless the application has chosen a mode itself (this runs when the
// library is loaded, normally before the CUDA context exists); configure_kernels additionally touches every kernel.
__attribute__((constructor)) static void pamg_request_eager_loading() { setenv("CUDA_MODULE_LOADING", "EAGER", 0); }

struct pamg_handle;
namespace { void p2p_close(pamg_handle* h); }
// words of pamg_handle::agg_words (device memory): block counter, per-destination transfer numbers, per-sender flags
// and the number of transfers already consumed per sender
enum { AGG_COUNTER = 0, AGG_EPOCH = 8, AGG_FLAGS = 40, AGG_EXPECT = 72, AGG_WORDS = 104 };

// ------------------------------------------------------------------ handle
// what the strips of the faces cut by the GPU partition hold.  CUT_STAGED: the values of the current iterate, sent by a
// sweep's producer warps, wait in the level's flagged staging buffer under the current exchange number; an unpack is due.
// The letters of the exchange-protocol model (tests/test_exchange_protocol_model.py) are the transitions next to
// ensure_strips: H halo_exchanged, W sweep_done after a sweep that sent, U unpacked, X field_changed.
enum CutState { CUT_STALE, CUT_STAGED, CUT_VALID };

struct LevelDev {
  int s = 0, S = 0;
  long long C = 0, nelem = 0, ndof = 0;
  double* T[2] = {nullptr, nullptr};  // T[cur] = TNONLIN (the iterate); T[cur^1] = TNEW unless aliased
  int cur = 0;
  bool tnew_alias = true;             // TNEW == TNONLIN logically (no separate copy materialised)
  double *told = nullptr, *rhs = nullptr, *res = nullptr;
  double* ovlb[2] = {nullptr, nullptr};       // halo strips, double-buffered: (nstrips + nsend) * 3S doubles each
  int ovl_cur = 0;                            // ovlb[ovl_cur] holds the strips of the current iterate when strips_valid
  bool strips_valid = false;                  // strips of the faces between local parents hold the current iterate
  CutState cut = CUT_STALE;                   // strips of the faces cut by the GPU partition
  // (strips_valid and cut are written only by the transitions next to ensure_strips)
  ulonglong2* xsend = nullptr;                // [U*3] where a sweep's producer warp sends the values of a cut side (ElemArgs::xsend)
  double* ovl_old = nullptr;                  // told strips (update_overlaps as written only)
  double* pc = nullptr;               // [U][NPC]
  double* pc_old = nullptr;           // level 1, theta != 1: [U][NPC] of the old-time operator (1 - theta)(-stiff + flux + diff), no mass (get_RHS :459-460)
  bool rhs_valid = false;             // level 1: RHS matches TOLD
  double* spare = nullptr;            // third field buffer of pamg_smooth_host (level 1, allocated on first use)
};

struct pamg_handle {
  pamg_params p;
  int device = 0, nsm = 148;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[16] = {};
  long long launches = 0;
  std::string err;
  HaloPlan plan;
  int U = 0;  // local parents
  double* xg = nullptr;
  int32_t *strip_of = nullptr, *dst_strip = nullptr, *rev = nullptr, *hmap = nullptr, *nsrc = nullptr, *cut_lf = nullptr;
  // Dirichlet data of domain-boundary faces (pamg_set_boundary_data): global [U_global][3] on the host, local copy on the device
  std::vector<int32_t> bc_kind_h; std::vector<double> bc_val_h;
  int32_t* bc_kind = nullptr; double* bc_val = nullptr;
  // both halo-strip buffers of every level in ONE allocation, kept resident in L2 (access-policy window on the stream): the
  // strips are written by one sweep and read by the next, a whole field of streaming traffic later
  double* strip_arena = nullptr; size_t strip_arena_bytes = 0;
  std::vector<LevelDev> lev;
  double* partial = nullptr; int npartial = 0; int last_partials = 0;
  double* out3 = nullptr;         // device
  double* out3_host = nullptr;    // pinned
  double* scratch = nullptr; size_t scratch_bytes = 0;  // L2 flush
  // resident CTAs per SM of the shared-memory kernels on THIS device ([face_terms]); set once per handle in configure_kernels
  struct KernelCfg { int win2[2] = {0, 0}, win2x = 0, win[2] = {0, 0}, tma[2] = {0, 0}, gs2 = 0, gs2x = 0, gs = 0, halo = 0; bool done = false; } kc;
  bool capturing = false;   // stream capture in progress: no synchronisation, no per-launch error polling
  struct VcGraph { long long key; std::vector<cudaGraphExec_t> exec; std::vector<long long> launches; };   // one graph per GPU of the group
  std::vector<VcGraph> vc_graphs;   // a few cached V-cycle graphs (solver / sweep counts / buffer parity)
  bool graph_nccl = true;       // try to capture NCCL calls into the V-cycle graph (cleared when the library refuses)
  // per-kernel timing (element kernels only)
  bool profiling = false;
  std::vector<cudaEvent_t> pev;  // pairs
  int pev_used = 0;
  // distributed
  ncclComm_t comm = nullptr; int nranks = 1, rank = 0;
  // coarse-level agglomeration: levels >= agg_level are solved on part 0 for the whole mesh (SURVEY 8(e))
  pamg_handle* agg = nullptr;       // part 0 only: handle over ALL parents whose level 1 is my level agg_level
  int agg_level = 0;                // 0 = none
  int level_offset = 0;             // agg handle: its level l is level l + level_offset of the owner
  bool shared_stream = false;
  std::vector<int32_t> part_first;  // copy of the partition table
  int U_global = 0;
  // single-process multi-GPU (pamg_create_multi): the root owns one sub-handle per device and fans every entry out
  std::vector<pamg_handle*> parts;  // root only
  bool is_root = false;
  bool in_group = false;            // sub-handle of such a root: its peers are driven by the same host thread
  unsigned long long* agg_words = nullptr;   // sub-handle: counters / flags of the device-initiated block transfers
  // unstructured
  UnstrDev un;
  int un_use_dir = 0;
  long long un_host_syncs = 0;
  // pamg_smooth_host: copies on their own streams so that the upload of call k+1 overlaps the download of call k
  cudaStream_t up_stream = nullptr, down_stream = nullptr;
  cudaEvent_t ev_up = nullptr, ev_comp = nullptr, ev_down[2] = {nullptr, nullptr};
  unsigned pipe_calls = 0;             // calls since the last pamg_sync
  const double* last_out = nullptr;    // host buffer the most recent call downloads into
  // halo exchange by direct stores into peer memory (CUDA IPC over NVLink); PAMG_P2P=0 keeps ncclSend/ncclRecv
  bool p2p_enabled = true, p2p_ready = false, p2p_failed = false;
  unsigned long long* p2p_sync = nullptr;   // exchange number, block counter (device)
  unsigned long long* p2p_err_host = nullptr;   // error word raised by a halo kernel that timed out: mapped pinned memory, so
  unsigned long long* p2p_err_dev = nullptr;    // every host synchronisation point can check it without a copy
  uint4* p2p_stage = nullptr;               // flagged receive staging of ALL levels (IPC-exported): per level P2P_SLOTS slots x
  long long p2p_strips = 0;                 //   p2p_strips * 3 * S(level) words, levels one after the other
  struct P2PPeer { int slot_at_peer = -1, strip_begin_at_peer = 0; long long recv_strips_at_peer = 0; uint4* stage = nullptr; };
  std::vector<P2PPeer> p2p_peers;      // same order as plan.peers
  std::vector<void*> p2p_opened;       // IPC mappings to close
  unsigned long long p2p_timeout_ns = 60000000000ull;   // PAMG_P2P_TIMEOUT_S: how long a halo kernel polls for a peer before it gives up
};

namespace {

int fail(pamg_handle* h, int code, const std::string& msg) {
  if (h) h->err = msg;
  return code;
}
 #define CK_(hh, call)                                                                            \
  do {                                                                                           \
    cudaError_t e_ = (call);                                                                     \
    if (e_ != cudaSuccess)                                                                       \
      return fail(hh, PAMG_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));        \
  } while (0)
#define CK(call)                                                                                 \
  do {                                                                                           \
    cudaError_t e_ = (call);                                                                     \
    if (e_ != cudaSuccess)                                                                       \
      return fail(h, PAMG_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));         \
  } while (0)

inline int grid_for(const pamg_handle* h, long long n) {
  long long need = (n + TPB - 1) / TPB;
  long long cap = (long long)h->nsm * 8;  // 8 resident CTAs of 256 threads per SM
  return (int)std::max(1ll, std::min(need, cap));
}

bool valid_level(const pamg_handle* h, int level) { return h && level >= 1 && level <= (int)h->lev.size(); }

double* tnew_ptr(LevelDev& L) { return L.tnew_alias ? L.T[L.cur] : L.T[L.cur ^ 1]; }

// make TNEW a real, separate copy of what it logically holds
int materialise_tnew(pamg_handle* h, LevelDev& L) {
  if (!L.tnew_alias) return PAMG_OK;
  CK(cudaMemcpyAsync(L.T[L.cur ^ 1], L.T[L.cur], L.ndof * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  L.tnew_alias = false;
  return PAMG_OK;
}

// ---- transitions of a level's strip state (LevelDev::strips_valid, LevelDev::cut)
// X: something other than a sweep wrote the iterate (upload, fill, copy, prolongation, a coarse correction)
void field_changed(LevelDev& L) { L.strips_valid = false; L.cut = CUT_STALE; }

// H: a k_halo launch exchanged the cut faces of a field under a new exchange number, and copied the strips of every face
// between parents unless it ran HALO_CUT.  Of the iterate: those strips are current.  Of TOLD: the staging buffer no
// longer holds what a sweep's producer warps sent.
void halo_exchanged(LevelDev& L, HaloMode mode, bool of_iterate) {
  if (!of_iterate) { if (L.cut == CUT_STAGED) L.cut = CUT_STALE; return; }
  if (mode != HALO_CUT) L.strips_valid = true;
  L.cut = CUT_VALID;
}

// U: the staged cut-face values are in the strips
void unpacked(LevelDev& L) { L.cut = CUT_VALID; }

// W: the end of a sweep.  The producer warps of a fused sweep wrote the strips of the new iterate, except those of the
// cut faces, whose values they sent to the peers when `sent`; any other sweep leaves no current strips.
void sweep_done(const pamg_handle* h, LevelDev& L, bool fused, bool sent) {
  if (!fused) { field_changed(L); return; }
  L.strips_valid = true;
  L.cut = h->plan.peers.empty() ? CUT_VALID : sent ? CUT_STAGED : CUT_STALE;
}

// undo_norm_sweep: the strips a fused sweep read are current again; what it sent to the peers belongs to the discarded
// iterate
void sweep_undone(LevelDev& L, bool fused) {
  if (!fused) { field_changed(L); return; }
  L.strips_valid = true; L.cut = CUT_VALID;
}

int launch_halo(pamg_handle* h, int level, HaloMode mode);

// halo data of the current iterate, refreshed only if something touched the field since: `all` = the strips of every
// face between parents (in-place sweeps and the kernels that do not read their neighbours' field), otherwise only the
// strips of the faces cut by the GPU partition
int ensure_strips(pamg_handle* h, int level, bool all = true) {
  LevelDev& L = h->lev[level - 1];
  if (!h->p.face_terms) return PAMG_OK;
  if (all && !L.strips_valid) return launch_halo(h, level, HALO_SHARED);
  if (L.cut == CUT_VALID) return PAMG_OK;
  // the values a sweep's producer warps sent are waiting in the staging buffer: unpack them; else a full exchange
  return launch_halo(h, level, (L.cut == CUT_STAGED && h->p2p_ready) ? HALO_UNPACK : HALO_CUT);
}

double* field_ptr(pamg_handle* h, int field, int level, bool for_write, int* rc) {
  *rc = PAMG_OK;
  LevelDev& L = h->lev[level - 1];
  switch (field) {
    case PAMG_TNEW:
      if (for_write) { *rc = materialise_tnew(h, L); field_changed(L); return L.T[L.cur ^ 1]; }
      return tnew_ptr(L);
    case PAMG_TNONLIN:
      if (for_write) { *rc = materialise_tnew(h, L); field_changed(L); }
      return L.T[L.cur];
    case PAMG_TOLD: if (for_write) L.rhs_valid = false; return L.told;
    case PAMG_RHS: if (for_write) L.rhs_valid = true; return L.rhs;
    case PAMG_RES: return L.res;
  }
  *rc = PAMG_ERR_ARG;
  return nullptr;
}

// ---- per-parent geometry in closed form (tri_det_nlx ShapFun.F90:1414-1454; det_snlx_all :1554-1590;
//      level scaling :1678-1683,1751-1780; get_d_center Msh2Tri.F90:358-383; add_diffusion_surf
//      matrices.F90:84-110).  One row of NPC coefficients per parent per level.
// bc_kind: [U_global][3] kinds of the domain-boundary faces (nullptr = Dirichlet everywhere); an open face (kind 2) has no
// penalty term.  Returns false for an open face with inflow (n.u < 0): the exterior trace would have to follow the interior
// one inside the kernels, which is not supported.
// th weights every spatial term (get_A_x :444-446: theta (-stiff + flux + diff_vol + diff_surf) + mass; the diagonal follows
// the operator, ml/dt + theta (K_ii + sum_f my_ii) - the reference's mat_diag_approx leaves theta out, :483, the same thing at
// its only literal theta = 1); with_mass = false drops the mass term: th = 1 - theta without mass is the old-time operator of
// get_RHS (:459-460).
bool parent_coefficients(const pamg_params& p, const double* Xall, const int32_t* neig, const int32_t* bc_kind,
                         int g /*global parent*/, int s, double* pc, double th, bool with_mass = true) {
  bool supported = true;
  const double* X = Xall + (size_t)g * 6;
  const double x1 = X[0], y1 = X[1], x2 = X[2], y2 = X[3], x3 = X[4], y3 = X[5];
  const double A = x1 - x3, B = y1 - y3, Cc = x2 - x3, D = y2 - y3;
  const double detj = A * D - B * Cc;
  const double area = 0.5 * std::fabs(detj);
  const double g1[2] = {D / detj, -Cc / detj}, g2[2] = {-B / detj, A / detj};
  const double g3[2] = {-(g1[0] + g2[0]), -(g1[1] + g2[1])};
  const double* G[3] = {g1, g2, g3};
  const double two_s = std::ldexp(1.0, s), four_s = std::ldexp(1.0, 2 * s);
  pc[PC_CM] = with_mass ? area / (12.0 * four_s * p.dt) : 0.0;
  auto dot = [](const double* a, const double* b) { return a[0] * b[0] + a[1] * b[1]; };
  const double kth = th * p.k;      // (th = 1: bit-identical to the unweighted tables)
  pc[PC_K11] = kth * area * dot(g1, g1); pc[PC_K12] = kth * area * dot(g1, g2); pc[PC_K13] = kth * area * dot(g1, g3);
  pc[PC_K22] = kth * area * dot(g2, g2); pc[PC_K23] = kth * area * dot(g2, g3); pc[PC_K33] = kth * area * dot(g3, g3);
  const double uu[2] = {th * p.u_x, th * p.u_y};
  for (int i = 0; i < 3; ++i) pc[PC_ADV + i] = area * dot(G[i], uu) / (3.0 * two_s);
  const double cx = (x1 + x2 + x3) / 3.0, cy = (y1 + y2 + y3) / 3.0;
  // child faces: f1 = nodes (1,3) on side 1, f2 = (3,2) on side 3, f3 = (2,1) on side 2
  const int fa[3] = {0, 2, 1}, fb[3] = {2, 1, 0}, mface[3] = {0, 2, 1};
  const double V1[2] = {A, B}, V2[2] = {Cc, D};
  const double ci[3][2] = {{1.0 / 3, -2.0 / 3}, {-2.0 / 3, 1.0 / 3}, {1.0 / 3, 1.0 / 3}};  // centroid offsets of child 2's neighbours
  for (int f = 0; f < 3; ++f) {
    const double ax = X[2 * fa[f]], ay = X[2 * fa[f] + 1], bx = X[2 * fb[f]], by = X[2 * fb[f] + 1];
    const double ex = bx - ax, ey = by - ay, L = std::sqrt(ex * ex + ey * ey);
    double nx = ey / L, ny = -ex / L;
    const double mx = 0.5 * (ax + bx), my = 0.5 * (ay + by);
    if (nx * (mx - cx) + ny * (my - cy) < 0) { nx = -nx; ny = -ny; }
    const double lhalf = 0.5 * L;
    pc[PC_FL + f] = (uu[0] * nx + uu[1] * ny) * lhalf / (3.0 * two_s);
    const double dix = ci[f][0] * V1[0] + ci[f][1] * V2[0], diy = ci[f][0] * V1[1] + ci[f][1] * V2[1];
    const double dcI = std::sqrt(dix * dix + diy * diy);
    pc[PC_PENI + f] = kth * lhalf / (3.0 * dcI);
    const int q = neig[(size_t)g * 3 + mface[f]];
    double dcX;
    if (q != 0) {
      const double* Y = Xall + (size_t)(q - 1) * 6;
      const double qx = (Y[0] + Y[2] + Y[4]) / 3.0, qy = (Y[1] + Y[3] + Y[5]) / 3.0;
      dcX = std::sqrt((cx - qx) * (cx - qx) + (cy - qy) * (cy - qy));
    } else {
      dcX = std::sqrt((cx - mx) * (cx - mx) + (cy - my) * (cy - my));
    }
    pc[PC_PENX + f] = kth * lhalf / (3.0 * dcX);
    if (q == 0 && bc_kind && bc_kind[(size_t)g * 3 + mface[f]] == 2) {
      pc[PC_PENX + f] = 0.0;                                 // open face: no data, no penalty
      if (p.face_terms && pc[PC_FL + f] < 0.0) supported = false;
    }
  }
  // omega / D of children with all three faces inside the parent (get_diagonal :481-486): node 1 sits on
  // faces 1,3; node 2 on faces 2,3; node 3 on faces 1,2.  The penalty diagonal exists only with the face block.
  const double f2 = p.face_terms ? 2.0 : 0.0;
  pc[PC_W + 0] = p.omega / (4.0 * pc[PC_CM] + pc[PC_K11] + f2 * (pc[PC_PENI + 0] + pc[PC_PENI + 2]));
  pc[PC_W + 1] = p.omega / (4.0 * pc[PC_CM] + pc[PC_K22] + f2 * (pc[PC_PENI + 1] + pc[PC_PENI + 2]));
  pc[PC_W + 2] = p.omega / (4.0 * pc[PC_CM] + pc[PC_K33] + f2 * (pc[PC_PENI + 0] + pc[PC_PENI + 1]));
  pc[22] = 0.0; pc[23] = 0.0;
  // folded operator of interior children, one set per orientation (struct Folded in pamg_kernels.cuh)
  for (int o = 0; o < 2; ++o) {
    const double sg = o == 0 ? 1.0 : -1.0;
    double* F = pc + PC_FOLD + 16 * o;
    double A[3][3];
    const double K[3][3] = {{pc[PC_K11], pc[PC_K12], pc[PC_K13]}, {pc[PC_K12], pc[PC_K22], pc[PC_K23]},
                            {pc[PC_K13], pc[PC_K23], pc[PC_K33]}};
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j)
        A[i][j] = pc[PC_CM] * ((i == j ? 1.0 : 0.0) + 1.0) - sg * pc[PC_ADV + i] + K[i][j];
    const int fa2[3] = {0, 2, 1}, fb2[3] = {2, 1, 0};   // face nodes (a,b): f1 (1,3), f2 (3,2), f3 (2,1)
    double c[3];
    for (int f = 0; f < 3; ++f) {
      const double pen = p.face_terms ? pc[PC_PENI + f] : 0.0;
      const double fl = p.face_terms ? sg * pc[PC_FL + f] : 0.0;
      const bool in = fl < 0.0;
      const double own = pen + (in ? 0.0 : fl);
      c[f] = -pen + (in ? fl : 0.0);
      const int ia = fa2[f], ib = fb2[f];
      A[ia][ia] += 2.0 * own; A[ia][ib] += own; A[ib][ia] += own; A[ib][ib] += 2.0 * own;
    }
    F[0] = A[0][0]; F[1] = A[0][1]; F[2] = A[0][2]; F[3] = A[1][0]; F[4] = A[1][1]; F[5] = A[1][2];
    F[6] = A[2][0]; F[7] = A[2][1]; F[8] = A[2][2]; F[9] = c[0]; F[10] = c[1]; F[11] = c[2];
    F[12] = pc[PC_W + 0]; F[13] = pc[PC_W + 1]; F[14] = pc[PC_W + 2]; F[15] = 0.0;
  }
  // children with faces on the parent boundary: penalty change per face and omega / D per face mask
  for (int f = 0; f < 3; ++f) pc[PC_DPEN + f] = p.face_terms ? pc[PC_PENX + f] - pc[PC_PENI + f] : 0.0;
  pc[PC_DPEN + 3] = 0.0;
  for (int mask = 0; mask < 8; ++mask) {
    double pen[3];
    for (int f = 0; f < 3; ++f) pen[f] = p.face_terms ? ((mask >> f) & 1 ? pc[PC_PENX + f] : pc[PC_PENI + f]) : 0.0;
    pc[PC_WB + mask * 3 + 0] = p.omega / (4.0 * pc[PC_CM] + pc[PC_K11] + 2.0 * (pen[0] + pen[2]));
    pc[PC_WB + mask * 3 + 1] = p.omega / (4.0 * pc[PC_CM] + pc[PC_K22] + 2.0 * (pen[1] + pen[2]));
    pc[PC_WB + mask * 3 + 2] = p.omega / (4.0 * pc[PC_CM] + pc[PC_K33] + 2.0 * (pen[0] + pen[1]));
  }
  for (int i = PC_WB + 24; i < NPC; ++i) pc[i] = 0.0;
  if (!with_mass) {
    // operator-only table (residual mode reads no omega / D): the diagonal without the mass term may vanish
    for (int i = 0; i < 3; ++i) { pc[PC_W + i] = 0.0; pc[PC_FOLD + 12 + i] = 0.0; pc[PC_FOLD + 16 + 12 + i] = 0.0; }
    for (int i = 0; i < 24; ++i) pc[PC_WB + i] = 0.0;
  }
  return supported;
}

int p2p_upload_args(pamg_handle* h);

void p2p_close(pamg_handle* h) {
  for (void* p : h->p2p_opened) cudaIpcCloseMemHandle(p);
  h->p2p_opened.clear();
  if (h->p2p_sync) { cudaFree(h->p2p_sync); h->p2p_sync = nullptr; }
  if (h->p2p_stage) { cudaFree(h->p2p_stage); h->p2p_stage = nullptr; }
  if (h->p2p_err_host) { cudaFreeHost(h->p2p_err_host); h->p2p_err_host = nullptr; h->p2p_err_dev = nullptr; }
  h->p2p_ready = false; h->p2p_failed = false;
  for (auto& pp : h->p2p_peers) pp.stage = nullptr;
}

// a halo kernel that gave up waiting for a peer GPU raised the error word; every host synchronisation point of the
// partitioned path (residual norms, V-cycle control, downloads, pamg_sync) reports it instead of returning stale numbers
int p2p_check(pamg_handle* h) {
  if (h->p2p_err_host && *(volatile unsigned long long*)h->p2p_err_host)
    return fail(h, PAMG_ERR_CUDA, "halo exchange timed out waiting for a peer GPU");
  return PAMG_OK;
}

// first word of level il (0-based) inside a staging buffer that holds `strips` cut strips per level and slot
long long stage_offset(long long strips, const std::vector<LevelDev>& lev, int il) {
  long long off = 0;
  for (int l = 0; l < il; ++l) off += (long long)P2P_SLOTS * strips * 3 * lev[l].S;
  return off;
}

// local part of the set-up: exchange counters, the flagged receive staging buffers (per level, P2P_SLOTS slots) and the error word
int p2p_alloc_local(pamg_handle* h) {
  long long strips = 0;
  for (const auto& pr : h->plan.peers) strips = std::max(strips, (long long)pr.strip_begin + pr.nfaces);
  h->p2p_strips = strips;
  const size_t nlev = h->lev.size();
  const size_t stage_bytes = (size_t)std::max(1ll, stage_offset(h->p2p_strips, h->lev, (int)nlev)) * sizeof(uint4);
  CK(cudaMalloc(&h->p2p_sync, nlev * P2P_WORDS * sizeof(unsigned long long)));
  CK(cudaMemset(h->p2p_sync, 0, nlev * P2P_WORDS * sizeof(unsigned long long)));
  CK(cudaMalloc(&h->p2p_stage, stage_bytes));
  CK(cudaMemset(h->p2p_stage, 0, stage_bytes));
  CK(cudaHostAlloc(&h->p2p_err_host, sizeof(unsigned long long), cudaHostAllocMapped | cudaHostAllocPortable));
  *h->p2p_err_host = 0;
  CK(cudaHostGetDevicePointer((void**)&h->p2p_err_dev, h->p2p_err_host, 0));
  return PAMG_OK;
}

// collective over all ranks (one process per GPU; called at the first exchange, never during stream capture): allocate
// the staging buffer, exchange its CUDA IPC handle, map the peers' buffers, agree on the outcome.  A local failure is
// folded into the agreement (ok = 0 everywhere -> NCCL send/recv path) instead of leaving the other ranks in a collective.
int p2p_setup(pamg_handle* h) {
  const int R = h->nranks;
  int ok = 1;
  if ((int)h->plan.peers.size() > P2P_MAXP) ok = 0;
  for (const auto& pp : h->p2p_peers) if (pp.slot_at_peer < 0) ok = 0;
  if (p2p_alloc_local(h) != PAMG_OK) { ok = 0; (void)cudaGetLastError(); }
  // what travels: the IPC handle of my staging buffer
  struct Card { cudaIpcMemHandle_t handle; };
  Card mine;
  std::memset(&mine, 0, sizeof(mine));
  if (ok && cudaIpcGetMemHandle(&mine.handle, h->p2p_stage) != cudaSuccess) { ok = 0; (void)cudaGetLastError(); }
  // all-gather of the cards with grouped send / recv (R <= 8)
  const size_t hb = sizeof(Card);
  std::vector<Card> all(R);
  unsigned char* d_buf = nullptr;      // [mine][all R][ok]
  const bool have_buf = cudaMalloc(&d_buf, hb * (R + 1) + sizeof(int)) == cudaSuccess;
  int rc = PAMG_OK;
  if (!have_buf) {
    // without device memory this rank cannot even take part in the agreement
    return fail(h, PAMG_ERR_CUDA, "cudaMalloc failed in the halo-exchange set-up");
  }
  unsigned char* d_mine = d_buf; unsigned char* d_all = d_buf + hb; int* d_ok = (int*)(d_buf + hb * (R + 1));
  if (cudaMemcpy(d_mine, &mine, hb, cudaMemcpyHostToDevice) != cudaSuccess) ok = 0;
  g_nccl.GroupStart();
  for (int r = 0; r < R; ++r) {
    g_nccl.Send(d_mine, hb, ncclUint8, r, h->comm, h->stream);
    g_nccl.Recv(d_all + hb * r, hb, ncclUint8, r, h->comm, h->stream);
  }
  if (g_nccl.GroupEnd() != ncclSuccess) rc = fail(h, PAMG_ERR_CUDA, "handle exchange failed");
  if (!rc && cudaStreamSynchronize(h->stream) != cudaSuccess) ok = 0;
  if (!rc && cudaMemcpy(all.data(), d_all, hb * R, cudaMemcpyDeviceToHost) != cudaSuccess) ok = 0;
  if (!rc && ok) {
    for (size_t i = 0; i < h->plan.peers.size(); ++i) {
      void* ptr = nullptr;
      if (cudaIpcOpenMemHandle(&ptr, all[h->plan.peers[i].part].handle, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { ok = 0; (void)cudaGetLastError(); break; }
      h->p2p_opened.push_back(ptr);
      h->p2p_peers[i].stage = (uint4*)ptr;
    }
  }
  // every rank must take the same path
  if (!rc) {
    if (cudaMemcpy(d_ok, &ok, sizeof(int), cudaMemcpyHostToDevice) != cudaSuccess) ok = 0;
    if (g_nccl.AllReduce(d_ok, d_ok, 1, ncclInt32, ncclMin, h->comm, h->stream) != ncclSuccess) rc = fail(h, PAMG_ERR_CUDA, "ncclAllReduce failed");
    else if (cudaStreamSynchronize(h->stream) != cudaSuccess || cudaMemcpy(&ok, d_ok, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess)
      rc = fail(h, PAMG_ERR_CUDA, "halo-exchange set-up: reading the agreement failed");
  }
  cudaFree(d_buf);
  if (rc) return rc;
  if (ok) {
    if ((rc = p2p_upload_args(h))) return rc;
    h->p2p_ready = true;
  } else h->p2p_failed = true;
  return PAMG_OK;
}

int p2p_args(pamg_handle* h, LevelDev& L, double* ovl, P2PArgs& a) {
  const long long S3 = 3ll * L.S;
  const int il = (int)(&L - h->lev.data());
  const int base = h->plan.peers[0].send_begin;
  a.send = ovl + ((size_t)h->plan.nstrips + base) * S3;
  a.strips = ovl; a.stage = h->p2p_stage + stage_offset(h->p2p_strips, h->lev, il); a.stage_words = h->p2p_strips * S3;
  a.sync = h->p2p_sync + (size_t)il * P2P_WORDS; a.err = h->p2p_err_dev; a.npeers = (int)h->plan.peers.size();
  a.timeout_ns = h->p2p_timeout_ns;
  long long so = 0, ro = 0;
  for (int i = 0; i < a.npeers; ++i) {
    const auto& pr = h->plan.peers[i];
    if ((long long)(pr.send_begin - base) * S3 != so) return fail(h, PAMG_ERR_STATE, "send slots are not contiguous per peer");
    a.remote[i] = h->p2p_peers[i].stage + stage_offset(h->p2p_peers[i].recv_strips_at_peer, h->lev, il) +
                  (long long)h->p2p_peers[i].strip_begin_at_peer * S3;
    a.rstride[i] = h->p2p_peers[i].recv_strips_at_peer * S3;   // the peer's own words per slot on this level
    a.soff[i] = so; a.roff[i] = ro; a.rbeg[i] = (long long)pr.strip_begin * S3;
    so += pr.nfaces * S3; ro += pr.nfaces * S3;
  }
  a.soff[a.npeers] = so; a.roff[a.npeers] = ro;
  a.send_base = base;
  return PAMG_OK;
}

// per level and (parent, side): where the producer warp of a sweep sends the boundary values of a side cut by the GPU
// partition (ElemArgs::xsend) - a host-built table, so that the producer warp has no dependent look-ups to do
int p2p_upload_args(pamg_handle* h) {
  if (h->plan.peers.empty()) return PAMG_OK;
  std::vector<ulonglong2> t((size_t)h->U * 3);
  for (size_t l = 0; l < h->lev.size(); ++l) {
    P2PArgs v;
    std::memset(&v, 0, sizeof(v));
    int rc = p2p_args(h, h->lev[l], h->lev[l].ovlb[0], v);
    if (rc) return rc;
    const long long S3 = 3ll * h->lev[l].S;
    for (int lf = 0; lf < h->U * 3; ++lf) {
      const int d = h->plan.dst_strip[lf];
      t[lf] = make_ulonglong2(0ull, 0ull);
      if (d < h->plan.nstrips) continue;
      const long long q0 = (long long)(d - h->plan.nstrips - v.send_base) * S3;
      int p = 0;
      while (q0 >= v.soff[p + 1]) ++p;
      t[lf] = make_ulonglong2((unsigned long long)(v.remote[p] + (q0 - v.soff[p])), (unsigned long long)v.rstride[p]);
    }
    if (!h->lev[l].xsend) CK(cudaMalloc(&h->lev[l].xsend, t.size() * sizeof(ulonglong2)));
    CK(cudaMemcpy(h->lev[l].xsend, t.data(), t.size() * sizeof(ulonglong2), cudaMemcpyHostToDevice));
  }
  return PAMG_OK;
}

// library exchange of the cut-face strips (one process per GPU, when peer memory is not available): the send slots
// follow the local strips in the strip space; the receive range of a peer is a contiguous range of my own strips
int exchange_halo_nccl(pamg_handle* h, LevelDev& L, double* ovl) {
  if (!h->comm) return fail(h, PAMG_ERR_STATE, "partitioned mesh but pamg_comm_init was not called");
  const size_t S3 = (size_t)3 * L.S;
  g_nccl.GroupStart();
  for (const auto& pr : h->plan.peers) {
    const size_t n = (size_t)pr.nfaces * S3;
    g_nccl.Send(ovl + ((size_t)h->plan.nstrips + pr.send_begin) * S3, n, ncclFloat64, pr.part, h->comm, h->stream);
    g_nccl.Recv(ovl + (size_t)pr.strip_begin * S3, n, ncclFloat64, pr.part, h->comm, h->stream);
  }
  if (g_nccl.GroupEnd() != ncclSuccess) return fail(h, PAMG_ERR_CUDA, "ncclGroupEnd failed in halo exchange");
  return PAMG_OK;
}

// one k_halo launch on level L: `mode` applied to the strips of `src` in `ovl` (HALO_ALL: and to the told strips).  With
// peers the cut faces are exchanged: inside the kernel through peer memory (set up at the first exchange), else by NCCL
// after it.  Without peers there are no cut faces to exchange or unpack.
int launch_halo_kernel(pamg_handle* h, LevelDev& L, HaloMode mode, const double* src, double* ovl) {
  const bool cut = mode != HALO_DIRICHLET && !h->plan.peers.empty();
  if ((mode == HALO_CUT || mode == HALO_UNPACK) && !cut) return PAMG_OK;
  const int level = (int)(&L - h->lev.data()) + 1;
  HaloArgs a;
  a.tnew = src; a.told = L.told; a.ovl = ovl; a.ovl_old = L.ovl_old; a.xg = h->xg;
  a.dst_strip = h->dst_strip; a.rev = h->rev; a.strip_of = h->strip_of;
  a.bc_scale = (h->p.coarse_bc_zero && level + h->level_offset > 1) ? 0.0 : 1.0;
  a.U = h->U; a.s = L.s; a.with_old = (mode == HALO_ALL) ? 1 : 0; a.what = mode; a.nstrips = h->plan.nstrips;
  a.cut_lf = h->cut_lf; a.ncut = (int)h->plan.cut_lf.size();
  a.bc_kind = h->bc_kind; a.bc_val = h->bc_val;
  a.x.npeers = 0;
  if (cut && h->comm && h->p2p_enabled && !h->p2p_ready && !h->p2p_failed && !h->capturing && h->level_offset == 0) {
    int rc = p2p_setup(h);      // collective, first exchange only
    if (rc) return rc;
  }
  const bool fused_x = cut && h->p2p_ready;
  if (fused_x) { int rc = p2p_args(h, L, ovl, a.x); if (rc) return rc; }
  const long long n = (mode == HALO_CUT ? (long long)a.ncut : mode == HALO_UNPACK ? (long long)a.ncut * 3 : (long long)h->U * 3) * L.S;
  // with the exchange fused in, blocks poll for remote data after their own work: keep the grid within one wave
  int grid = grid_for(h, n);
  if (fused_x) grid = std::min(grid, h->nsm * std::min(std::max(h->kc.halo, 1), 4));
  k_halo<<<grid, TPB, 0, h->stream>>>(a);
  h->launches++;
  CK(cudaGetLastError());
  if (cut && !fused_x) return exchange_halo_nccl(h, L, ovl);
  return PAMG_OK;
}

// told values of the cut faces into the neighbours' told strips: the exchange update_overlaps as written makes for
// t_overlap_old (splitting.F90:1259-1262).  The sweeps never read them; the old-time terms (theta != 1) and the entry
// point do.
int exchange_told(pamg_handle* h, LevelDev& L) {
  int rc = launch_halo_kernel(h, L, HALO_CUT, L.told, L.ovl_old);
  if (!rc) halo_exchanged(L, HALO_CUT, false);
  return rc;
}

// the strips of the current iterate: HALO_ALL (pamg_update_overlaps) or what ensure_strips asks for
int launch_halo(pamg_handle* h, int level, HaloMode mode) {
  LevelDev& L = h->lev[level - 1];
  if (mode == HALO_UNPACK && !(h->p2p_ready && L.cut == CUT_STAGED)) return fail(h, PAMG_ERR_STATE, "nothing staged to unpack");
  int rc;
  // the told exchange goes FIRST, so that the staging buffers end up holding the tnew values under the current exchange number
  if (mode == HALO_ALL && (rc = exchange_told(h, L))) return rc;
  if ((rc = launch_halo_kernel(h, L, mode, tnew_ptr(L), L.ovlb[L.ovl_cur]))) return rc;
  if (mode == HALO_UNPACK) unpacked(L);
  else halo_exchanged(L, mode, true);
  return PAMG_OK;
}

// the sweeps of this level run the window kernels with a producer warp (k_element_win2, k_gs_win2; with face terms the
// producer warp also writes the next sweep's strips and sends the cut-face values).  Below s = 6 a parent has fewer than
// 8 tiles, too few for k_element_win2's double-buffered per-parent coefficients; above s = 8 a row (up to 2^(s+1) - 1
// children, the reach of a vertical neighbour) no longer fits the 8-tile ring.
bool producer_level(const LevelDev& L) { return L.s >= 6 && L.s <= 8; }

int add_old_time_terms(pamg_handle* h);

int launch_build_rhs(pamg_handle* h) {
  LevelDev& L = h->lev[0];
  RhsArgs a;
  a.told = L.told; a.rhs = L.rhs; a.pc = L.pc; a.xg = h->xg; a.dt = h->p.dt; a.source_coef = h->p.source_coef;
  a.nelem = L.nelem; a.s = L.s; a.literal_source = h->p.literal_source;
  k_build_rhs<<<grid_for(h, L.nelem), TPB, 0, h->stream>>>(a);
  h->launches++;
  CK(cudaGetLastError());
  if (L.pc_old) { int rc = add_old_time_terms(h); if (rc) return rc; }
  L.rhs_valid = true;
  return PAMG_OK;
}

// opt-in shared memory and resident CTAs per SM of every shared-memory kernel, once per handle (the attribute is per
// device and must not be set during stream capture)
template <typename K>
int configure_one(pamg_handle* h, K kern, int threads, size_t smem, int& resident) {
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, kern, threads, smem));
  if (resident < 1) resident = 1;
  return PAMG_OK;
}
template <bool FACE>
int configure_face(pamg_handle* h) {
  int rc, dummy = 0;
  const int f = FACE ? 1 : 0;
  if ((rc = configure_one(h, k_element_win2<MODE_JACOBI, FACE>, WIN2_THREADS, WIN_SMEM_BYTES, h->kc.win2[f]))) return rc;
  if ((rc = configure_one(h, k_element_win2<MODE_RESID, FACE>, WIN2_THREADS, WIN_SMEM_BYTES, dummy))) return rc;
  if ((rc = configure_one(h, k_element_win2<MODE_RICH, FACE>, WIN2_THREADS, WIN_SMEM_BYTES, dummy))) return rc;
  if constexpr (FACE) {   // (launch_element selects the XCHG and NORM kernels with face terms only)
    if ((rc = configure_one(h, k_element_win2<MODE_JACOBI, FACE, true>, WIN2_THREADS, WIN_SMEM_BYTES, h->kc.win2x))) return rc;
    if ((rc = configure_one(h, k_element_win2<MODE_JACOBI, FACE, false, true>, WIN2_THREADS, WIN_SMEM_BYTES, dummy))) return rc;
    if ((rc = configure_one(h, k_element_win2<MODE_JACOBI, FACE, true, true>, WIN2_THREADS, WIN_SMEM_BYTES, dummy))) return rc;
    if ((rc = configure_one(h, k_element_win2<MODE_RICH, FACE, true>, WIN2_THREADS, WIN_SMEM_BYTES, dummy))) return rc;
  }
  if ((rc = configure_one(h, k_element_win<MODE_JACOBI, FACE>, TPB, WIN_SMEM_BYTES, h->kc.win[f]))) return rc;
  if ((rc = configure_one(h, k_element_win<MODE_RESID, FACE>, TPB, WIN_SMEM_BYTES, dummy))) return rc;
  if ((rc = configure_one(h, k_element_win<MODE_RICH, FACE>, TPB, WIN_SMEM_BYTES, dummy))) return rc;
  // (the in-place GS pass runs with face terms only on s >= 9, in k_element_tma)
  if (!FACE && (rc = configure_one(h, k_element_win<MODE_GS, false>, TPB, WIN_SMEM_BYTES, dummy))) return rc;
  if ((rc = configure_one(h, k_element_tma<MODE_JACOBI, FACE>, TPB, TMA_SMEM_BYTES, h->kc.tma[f]))) return rc;
  if ((rc = configure_one(h, k_element_tma<MODE_RESID, FACE>, TPB, TMA_SMEM_BYTES, dummy))) return rc;
  if ((rc = configure_one(h, k_element_tma<MODE_RICH, FACE>, TPB, TMA_SMEM_BYTES, dummy))) return rc;
  if ((rc = configure_one(h, k_element_tma<MODE_GS, FACE>, TPB, TMA_SMEM_BYTES, dummy))) return rc;
  return PAMG_OK;
}
int configure_kernels(pamg_handle* h) {
  if (h->kc.done) return PAMG_OK;
  int rc;
  if ((rc = configure_face<true>(h))) return rc;
  if ((rc = configure_face<false>(h))) return rc;
  if ((rc = configure_one(h, k_gs_win2<false>, WIN2_THREADS, GSW_SMEM_BYTES, h->kc.gs2))) return rc;
  if ((rc = configure_one(h, k_gs_win2<true>, WIN2_THREADS, GSW_SMEM_BYTES, h->kc.gs2x))) return rc;
  if ((rc = configure_one(h, k_gs_win, TPB, GSW_SMEM_BYTES, h->kc.gs))) return rc;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&h->kc.halo, k_halo, TPB, 0));
  if (h->kc.halo < 1) h->kc.halo = 1;
  // Load every other kernel of the partitioned path NOW.  With lazy module loading (the CUDA 12 default) the first launch
  // of a function may have to wait for running kernels to finish; a halo kernel of one part that is polling for a peer
  // whose next kernel has never been launched in this process would then wait for ever (seen with two parts on one device).
  cudaFuncAttributes fa;
  CK(cudaFuncGetAttributes(&fa, k_halo));
  CK(cudaFuncGetAttributes(&fa, k_gs_small));
  CK(cudaFuncGetAttributes(&fa, k_build_rhs));
  CK(cudaFuncGetAttributes(&fa, k_restrict));
  CK(cudaFuncGetAttributes(&fa, k_prolong_literal));
  CK(cudaFuncGetAttributes(&fa, k_prolong_p1));
  CK(cudaFuncGetAttributes(&fa, k_reduce_partials));
  CK(cudaFuncGetAttributes(&fa, k_fill));
  CK(cudaFuncGetAttributes(&fa, k_push));
  CK(cudaFuncGetAttributes(&fa, k_wait_flags));
  CK(cudaFuncGetAttributes(&fa, k_output_fields));
  CK(cudaFuncGetAttributes(&fa, k_element_direct2<MODE_JACOBI, true>));
  CK(cudaFuncGetAttributes(&fa, k_element_direct2<MODE_JACOBI, false>));
  CK(cudaFuncGetAttributes(&fa, k_element_direct2<MODE_RESID, true>));
  CK(cudaFuncGetAttributes(&fa, k_element_direct2<MODE_RESID, false>));
  CK(cudaFuncGetAttributes(&fa, k_element_direct2<MODE_RICH, true>));
  CK(cudaFuncGetAttributes(&fa, k_element_direct2<MODE_RICH, false>));
  CK(cudaFuncGetAttributes(&fa, k_element_direct2<MODE_GS, false>));
  h->kc.done = true;
  return PAMG_OK;
}

// the arguments of a sweep-kernel launch.  use_strips: every strip of the level holds the start-of-sweep values (else:
// neighbour-field reads where possible); write_next: the kernel's producer warp writes the strips of the next sweep into
// the other strip buffer
ElemArgs elem_args(const pamg_handle* h, const LevelDev& L, const double* Tin, double* Tout, int colour, bool use_strips,
                   bool write_next) {
  ElemArgs a;
  a.xsend = L.xsend; a.xsync = h->p2p_sync ? h->p2p_sync + (size_t)(&L - h->lev.data()) * P2P_WORDS : nullptr;
  a.Tin = Tin; a.Tout = Tout; a.rhs = L.rhs; a.ovl = L.ovlb[L.ovl_cur]; a.pc = L.pc; a.strip_of = h->strip_of; a.hmap = h->hmap;
  // (an in-place pass - the two-pass coloured GS - must see start-of-sweep values across parent faces: strips only)
  a.nsrc = (use_strips || Tin == Tout) ? nullptr : h->nsrc;
  a.ovl_next = write_next ? L.ovlb[L.ovl_cur ^ 1] : nullptr; a.dst_strip = h->dst_strip; a.rev = h->rev; a.nstrips = h->plan.nstrips;
  a.partial = h->partial; a.omega = h->p.omega; a.rsign = (double)h->p.residual_sign; a.nelem = L.nelem; a.s = L.s;
  a.colour = colour; a.partial_off = 0;
  return a;
}

// what a launch takes from somewhere else than the level's current state (the old-time pass of get_RHS, theta != 1)
struct ElemOverride { const double* ovl; const double* pc; double rsign; };

template <int MODE>
int launch_element(pamg_handle* h, LevelDev& L, const double* Tin, double* Tout, int colour, int grid, bool use_strips,
                   bool write_next = false, bool xchg = false, bool norm = false, const ElemOverride* ov = nullptr) {
  ElemArgs a = elem_args(h, L, Tin, Tout, colour, use_strips, write_next);
  if (ov) { a.ovl = ov->ovl; a.pc = ov->pc; a.rsign = ov->rsign; }
  const int f = h->p.face_terms ? 1 : 0;
  const bool prof = !ov && h->profiling && h->pev_used + 2 <= (int)h->pev.size();
  if (prof) CK(cudaEventRecord(h->pev[h->pev_used], h->stream));
  // (the in-place GS pass never runs on a producer level, and with face terms only on s >= 9 (do_smooth): the branches
  // below instantiate no GS kernel it cannot launch)
  if (MODE != MODE_GS && producer_level(L)) {
    if constexpr (MODE != MODE_GS) {
      // window kernel with a producer warp (no CTA-wide barrier between tiles)
      const bool send = MODE != MODE_RESID && xchg;     // a residual evaluation sends nothing
      void (*kern)(ElemArgs) = h->p.face_terms ? k_element_win2<MODE, true> : k_element_win2<MODE, false>;
      if constexpr (MODE != MODE_RESID) if (send) kern = k_element_win2<MODE, true, true>;
      // a Jacobi sweep that also reduces the residual norms of the iterate it starts from (norm_fusable)
      if constexpr (MODE == MODE_JACOBI) if (norm) kern = send ? k_element_win2<MODE, true, true, true> : k_element_win2<MODE, true, false, true>;
      const int tgrid = (int)std::max(1ll, std::min(L.nelem / TPB, (long long)h->nsm * (send ? h->kc.win2x : h->kc.win2[f])));
      kern<<<tgrid, WIN2_THREADS, WIN_SMEM_BYTES, h->stream>>>(a);
      if (MODE == MODE_RESID || norm) h->last_partials = tgrid;
    }
  } else if (L.C >= TPB && L.s <= 8) {
    // (a vertical neighbour is up to 2^(s+1) children away: the 8-tile ring covers s <= 8)
    // window kernel: ring of 8 field tiles in shared memory, every neighbour value read from it
    void (*kern)(ElemArgs) = k_element_win<MODE, false>;
    if constexpr (MODE != MODE_GS) if (h->p.face_terms) kern = k_element_win<MODE, true>;
    const int tgrid = (int)std::max(1ll, std::min(L.nelem / TPB, (long long)h->nsm * h->kc.win[f]));
    kern<<<tgrid, TPB, WIN_SMEM_BYTES, h->stream>>>(a);
    if (MODE == MODE_RESID) h->last_partials = tgrid;
  } else if (L.C >= TPB) {
    // 1-D TMA tiles: contiguous 6 KB spans through shared memory; contiguous tile ranges per CTA, one wave of resident CTAs
    auto kern = h->p.face_terms ? k_element_tma<MODE, true> : k_element_tma<MODE, false>;
    const int tgrid = (int)std::max(1ll, std::min((L.nelem + TPB - 1) / TPB, (long long)h->nsm * h->kc.tma[f]));
    kern<<<tgrid, TPB, TMA_SMEM_BYTES, h->stream>>>(a);
    if (MODE == MODE_RESID) h->last_partials = tgrid;
  } else {
    // branch-free direct kernel (all loads of a child in flight at once): levels with fewer than 256 children per parent
    if (MODE == MODE_RESID) h->last_partials = grid;
    void (*kern)(ElemArgs) = k_element_direct2<MODE, false>;
    if constexpr (MODE != MODE_GS) if (h->p.face_terms) kern = k_element_direct2<MODE, true>;
    kern<<<grid, TPB, 0, h->stream>>>(a);
  }
  if (prof) { CK(cudaEventRecord(h->pev[h->pev_used + 1], h->stream)); h->pev_used += 2; }
  h->launches++;
  CK(cudaGetLastError());
  return PAMG_OK;
}

// theta != 1: RHS -= (1 - theta)(-stiff + flux + diff_vol + diff_surf) told  (get_RHS :459-460).  One residual-mode pass of the
// level-1 sweep kernel over TOLD with the old-time coefficient table: exterior values of faces between local parents straight
// from TOLD, Dirichlet data and cut-face values from the told strips.  RES is the scratch field of the pass.
int add_old_time_terms(pamg_handle* h) {
  LevelDev& L = h->lev[0];
  int rc;
  if (h->p.face_terms && (rc = exchange_told(h, L))) return rc;
  const int grid = grid_for(h, L.nelem);
  if (2 * grid > h->npartial) return fail(h, PAMG_ERR_STATE, "partial buffer too small");
  const ElemOverride ov = {L.ovl_old, L.pc_old, -1.0};     // r = b - A_old told with b = the theta = 1 right-hand side
  if ((rc = launch_element<MODE_RESID>(h, L, L.told, L.res, 0, grid, false, false, false, false, &ov))) return rc;
  CK(cudaMemcpyAsync(L.rhs, L.res, (size_t)L.ndof * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  return PAMG_OK;
}

// coloured Gauss-Seidel sweep in one pass (k_gs_win / k_gs_win2), out of place
// small levels (a CTA holds whole parents): both colours in one launch of k_gs_small
bool gs_small_ok(const pamg_handle* h, const LevelDev& L) { return h->p.face_terms && L.C <= TPB; }

int launch_gs_one_pass(pamg_handle* h, LevelDev& L, const double* Tin, double* Tout, bool use_strips, bool write_next, bool xchg) {
  const ElemArgs a = elem_args(h, L, Tin, Tout, 1, use_strips, write_next);
  if (gs_small_ok(h, L)) {
    const long long ppc = TPB / L.C, nparents = L.nelem / L.C;
    const int sgrid = (int)std::max(1ll, std::min((nparents + ppc - 1) / ppc, (long long)h->nsm * 8));
    k_gs_small<<<sgrid, TPB, 0, h->stream>>>(a);
    h->launches++;
    CK(cudaGetLastError());
    return PAMG_OK;
  }
  const bool producer = producer_level(L);
  const int resident = producer ? (xchg ? h->kc.gs2x : h->kc.gs2) : h->kc.gs;
  const bool prof = h->profiling && h->pev_used + 2 <= (int)h->pev.size();
  if (prof) CK(cudaEventRecord(h->pev[h->pev_used], h->stream));
  const int tgrid = (int)std::max(1ll, std::min(L.nelem / TPB, (long long)h->nsm * resident));
  if (producer && xchg) k_gs_win2<true><<<tgrid, WIN2_THREADS, GSW_SMEM_BYTES, h->stream>>>(a);
  else if (producer) k_gs_win2<false><<<tgrid, WIN2_THREADS, GSW_SMEM_BYTES, h->stream>>>(a);
  else k_gs_win<<<tgrid, TPB, GSW_SMEM_BYTES, h->stream>>>(a);
  if (prof) { CK(cudaEventRecord(h->pev[h->pev_used + 1], h->stream)); h->pev_used += 2; }
  h->launches++;
  CK(cudaGetLastError());
  return PAMG_OK;
}

// a Jacobi sweep of this level can hand out the residual norms of the iterate it starts from (k_element_win2<.., NORM>)
bool norm_fusable(const pamg_handle* h, const LevelDev& L) { return h->p.face_terms && producer_level(L); }

// norm_first: the first sweep (Jacobi on a norm_fusable level) also leaves the partial sums of the residual norms
int do_smooth(pamg_handle* h, int level, int solver, int nsweeps, bool norm_first = false) {
  LevelDev& L = h->lev[level - 1];
  if (level == 1 && !L.rhs_valid) { int rc = launch_build_rhs(h); if (rc) return rc; }
  const int grid = grid_for(h, L.nelem);
  if (solver < 1 || solver > 4) return fail(h, PAMG_ERR_ARG, "solver must be 1 (Jacobi), 2 (Richardson) or 3 (Gauss-Seidel)");
  for (int sw = 0; sw < nsweeps; ++sw) {
    // tnew <- tnew_nonlin (:550) is the buffer swap below; halo from it (:555): either the strips hold it (written by
    // the previous sweep's producer warps or by k_halo), or the sweep reads its neighbours' field directly.  Faces cut
    // by the GPU partition always go through their strips (the exchange step).
    L.tnew_alias = true;
    const bool gs = solver == 3 || solver == 4;
    // GS without face terms (the literal head) or on a level too deep for the window ring: two in-place passes
    const bool in_place = gs && !(h->p.face_terms && L.s <= 8);
    const bool fusedk = h->p.face_terms && producer_level(L);
    const bool use_strips = in_place || fusedk;
    // the producer warps of the sweep send the new cut-face values to the peers themselves (the strips it reads were
    // exchanged by k_halo or unpacked out of the staging buffer just before)
    const bool xs = fusedk && h->p2p_ready && L.xsend && !h->plan.peers.empty();
    int rc = ensure_strips(h, level, use_strips);
    if (rc) return rc;
    if (solver == 1 || solver == 2) {
      rc = (solver == 1) ? launch_element<MODE_JACOBI>(h, L, L.T[L.cur], L.T[L.cur ^ 1], 0, grid, use_strips, fusedk, xs,
                                                       norm_first && sw == 0)
                         : launch_element<MODE_RICH>(h, L, L.T[L.cur], L.T[L.cur ^ 1], 0, grid, use_strips, fusedk, xs);
      if (rc) return rc;
      L.cur ^= 1;
      L.tnew_alias = false;  // the old buffer now holds the start-of-sweep field = tracer%tnew
    } else if (!in_place) {
      // two-colour ordering of the reference's Gauss-Seidel sweep (all down children, then all up children; values across
      // parent faces stay lagged exactly as at :647-655), both colours in one pass over memory, written to the other
      // buffer (which then holds tracer%tnew, as for Jacobi)
      rc = launch_gs_one_pass(h, L, L.T[L.cur], L.T[L.cur ^ 1], use_strips, fusedk, xs);
      if (rc) return rc;
      L.cur ^= 1;
      L.tnew_alias = false;
    } else {
      if (sw == nsweeps - 1 && h->p.keep_tnew_gs) { rc = materialise_tnew(h, L); if (rc) return rc; }  // keep tracer%tnew observable
      rc = launch_element<MODE_GS>(h, L, L.T[L.cur], L.T[L.cur], 0, grid, true);
      if (rc) return rc;
      rc = launch_element<MODE_GS>(h, L, L.T[L.cur], L.T[L.cur], 1, grid, true);   // all children on parent faces are "up"
      if (rc) return rc;
    }
    if (fusedk) L.ovl_cur ^= 1;              // the producer warps wrote the strips of the new iterate
    sweep_done(h, L, fusedk, xs);
  }
  return PAMG_OK;
}

// second stage of the norm reduction, the all-reduce over the ranks and the copy to pinned host memory (queued, not awaited)
int queue_norms(pamg_handle* h) {
  k_reduce_partials<<<1, 1024, 0, h->stream>>>(h->partial, h->last_partials, h->out3);
  h->launches++;
  CK(cudaGetLastError());
  if (h->comm && h->nranks > 1) {
    // global norms: sum of squares, max |r|, max r
    g_nccl.GroupStart();
    g_nccl.AllReduce(h->out3, h->out3, 1, ncclFloat64, ncclSum, h->comm, h->stream);
    g_nccl.AllReduce(h->out3 + 1, h->out3 + 1, 2, ncclFloat64, ncclMax, h->comm, h->stream);
    if (g_nccl.GroupEnd() != ncclSuccess) return fail(h, PAMG_ERR_CUDA, "ncclAllReduce failed");
  }
  CK(cudaMemcpyAsync(h->out3_host, h->out3, 3 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  return PAMG_OK;
}

int do_residual(pamg_handle* h, int level, double* l2, double* linf, double* smax, bool queue_only = false) {
  LevelDev& L = h->lev[level - 1];
  if (level == 1 && !L.rhs_valid) { int rc = launch_build_rhs(h); if (rc) return rc; }
  const int grid = grid_for(h, L.nelem);
  if (2 * grid > h->npartial) return fail(h, PAMG_ERR_STATE, "partial buffer too small");
  // exterior values of faces between local parents come straight from TNEW (what update_overlaps copies); the strips of
  // faces cut by the GPU partition are refreshed here if something touched the field since the last exchange
  const bool use_strips = L.strips_valid;
  int rc = ensure_strips(h, level, use_strips);
  if (rc) return rc;
  rc = launch_element<MODE_RESID>(h, L, tnew_ptr(L), L.res, 0, grid, use_strips);
  if (rc) return rc;
  if (l2 || linf || smax) {
    if ((rc = queue_norms(h))) return rc;
    if (queue_only || h->capturing) return PAMG_OK;      // the caller synchronises (after the graph launch / for the whole group)
    CK(cudaStreamSynchronize(h->stream));
    if ((rc = p2p_check(h))) return rc;
    if (l2) *l2 = std::sqrt(h->out3_host[0]);
    if (linf) *linf = h->out3_host[1];
    if (smax) *smax = h->out3_host[2];
  }
  return PAMG_OK;
}

int do_restrict(pamg_handle* h, int fine_level) {
  if (fine_level >= (int)h->lev.size()) return PAMG_OK;  // splitting.F90:18
  LevelDev& F = h->lev[fine_level - 1];
  LevelDev& Cc = h->lev[fine_level];
  XferArgs a;
  a.src = F.res; a.dst = Cc.rhs; a.ncoarse = Cc.nelem; a.sc = Cc.s; a.mode = h->p.transfer;
  k_restrict<<<grid_for(h, Cc.nelem), TPB, 0, h->stream>>>(a);
  h->launches++;
  CK(cudaGetLastError());
  Cc.rhs_valid = true;
  return PAMG_OK;
}

int do_prolong(pamg_handle* h, int fine_level, bool keep_tnew = true) {
  if (fine_level >= (int)h->lev.size()) return fail(h, PAMG_ERR_ARG, "no coarser level to prolong from");
  LevelDev& F = h->lev[fine_level - 1];
  LevelDev& Cc = h->lev[fine_level];
  XferArgs a;
  a.ncoarse = Cc.nelem; a.sc = Cc.s; a.mode = h->p.transfer;
  if (h->p.transfer == 0) {
    // as written: tracer(ilevel)%tnew += f(tracer(ilevel+1)%tnew), splitting.F90:59-88
    int rc = materialise_tnew(h, F);
    if (rc) return rc;
    a.src = tnew_ptr(Cc); a.dst = F.T[F.cur ^ 1];
    k_prolong_literal<<<grid_for(h, Cc.nelem), TPB, 0, h->stream>>>(a);
  } else {
    if (keep_tnew) {                  // the correction goes to the iterate only: keep tracer%tnew as it was
      int rc = materialise_tnew(h, F);
      if (rc) return rc;
    } else {
      F.tnew_alias = true;            // inside the V-cycle nothing reads the pre-correction field
    }
    a.src = Cc.T[Cc.cur]; a.dst = F.T[F.cur];
    field_changed(F);
    k_prolong_p1<<<grid_for(h, F.nelem), TPB, 0, h->stream>>>(a);
  }
  h->launches++;
  CK(cudaGetLastError());
  return PAMG_OK;
}

int do_fill(pamg_handle* h, double* p, long long n, double v) {
  if (v == 0.0) { CK(cudaMemsetAsync(p, 0, n * sizeof(double), h->stream)); return PAMG_OK; }
  k_fill<<<grid_for(h, n), TPB, 0, h->stream>>>(p, n, v);
  h->launches++;
  CK(cudaGetLastError());
  return PAMG_OK;
}

// ---- groups -------------------------------------------------------------------------------------------------------
// Everything from here on works on a GROUP of handles that advance in lockstep: a plain handle is a group of one (its
// peers, if any, live in other processes and meet it inside the exchange kernels / NCCL calls); the root of a
// single-process multi-GPU handle (pamg_create_multi) is the group of its parts.  The host thread queues each step for
// every part before it moves on, never blocks in between, and all cross-GPU ordering happens on the devices (flagged
// NVLink stores polled by the receiving kernel), so part 0's stream may run ahead of the others without deadlock.
typedef std::vector<pamg_handle*> Group;
Group group_of(pamg_handle* h) { return h->parts.empty() ? Group{h} : h->parts; }
int gfail(pamg_handle* owner, pamg_handle* q, int rc) { if (owner != q) owner->err = q->err; return rc; }
#define GALL(G, owner, q, expr)                                            \
  do {                                                                     \
    for (pamg_handle* q : G) {                                             \
      if (q->in_group) cudaSetDevice(q->device);                           \
      int rc_ = (expr);                                                    \
      if (rc_) return gfail(owner, q, rc_);                                \
    }                                                                      \
  } while (0)

int vcycle_rec(const Group& G, pamg_handle* owner, int level, int solver, int nu1, int nu2, int ncoarse, int skip_pre = 0);

int launch_push(pamg_handle* q, const double* src, double* dst, long long n, int channel, unsigned long long* peer_flag) {
  PushArgs a;
  a.src = src; a.dst = dst; a.n = n; a.counter = q->agg_words + AGG_COUNTER; a.epoch = q->agg_words + AGG_EPOCH + channel;
  a.flag = peer_flag;
  const int grid = (int)std::max(1ll, std::min((n + TPB - 1) / TPB, (long long)q->nsm * 2));
  k_push<<<grid, TPB, 0, q->stream>>>(a);
  q->launches++;
  CK_(q, cudaGetLastError());
  return PAMG_OK;
}

int launch_wait(pamg_handle* q, unsigned senders) {
  WaitArgs a;
  a.flags = q->agg_words + AGG_FLAGS; a.expect = q->agg_words + AGG_EXPECT; a.err = q->p2p_err_dev;
  a.timeout_ns = q->p2p_timeout_ns; a.senders = senders;
  k_wait_flags<<<1, 32, 0, q->stream>>>(a);
  q->launches++;
  CK_(q, cudaGetLastError());
  return PAMG_OK;
}

// Coarse-level agglomeration (SURVEY 8(e)): below agg_level every kernel is launch-latency bound and every sweep
// would pay an exchange, so the restricted right-hand side of all parts is gathered on part 0, the remaining
// levels of the V-cycle run there on the whole mesh (no exchange at all), and the correction is scattered back.
int agg_coarse_solve(const Group& G, pamg_handle* owner, int solver, int nu1, int nu2, int ncoarse) {
  pamg_handle* h0 = G[0];
  const int lvl = h0->agg_level;
  const size_t per_parent = (size_t)3 * h0->lev[lvl - 1].C;
  if (G.size() == 1) {
    // one process per GPU: gather / scatter with grouped ncclSend / ncclRecv
    pamg_handle* h = h0;
    LevelDev& Lc = h->lev[lvl - 1];
    if (!h->comm) return fail(h, PAMG_ERR_STATE, "agglomeration needs pamg_comm_init");
    g_nccl.GroupStart();
    if (h->rank == 0) {
      LevelDev& A = h->agg->lev[0];
      for (int p = 1; p < h->nranks; ++p)
        g_nccl.Recv(A.rhs + per_parent * h->part_first[p], per_parent * (h->part_first[p + 1] - h->part_first[p]), ncclFloat64, p,
                    h->comm, h->stream);
    } else {
      g_nccl.Send(Lc.rhs, per_parent * h->U, ncclFloat64, 0, h->comm, h->stream);
    }
    if (g_nccl.GroupEnd() != ncclSuccess) return fail(h, PAMG_ERR_CUDA, "ncclGroupEnd failed in coarse gather");
    if (h->rank == 0) {
      pamg_handle* g = h->agg;
      LevelDev& A = g->lev[0];
      CK(cudaMemcpyAsync(A.rhs, Lc.rhs, per_parent * h->U * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
      CK(cudaMemsetAsync(A.T[A.cur], 0, A.ndof * sizeof(double), h->stream));
      A.tnew_alias = true; field_changed(A); A.rhs_valid = true;
      const long long l0 = g->launches;
      int rc = vcycle_rec(Group{g}, g, 1, solver, nu1, nu2, ncoarse);
      h->launches += g->launches - l0;
      if (rc) return fail(h, rc, g->err);
      CK(cudaMemcpyAsync(Lc.T[Lc.cur], A.T[A.cur], per_parent * h->U * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    }
    g_nccl.GroupStart();
    if (h->rank == 0) {
      LevelDev& A = h->agg->lev[0];
      for (int p = 1; p < h->nranks; ++p)
        g_nccl.Send(A.T[A.cur] + per_parent * h->part_first[p], per_parent * (h->part_first[p + 1] - h->part_first[p]), ncclFloat64,
                    p, h->comm, h->stream);
    } else {
      g_nccl.Recv(Lc.T[Lc.cur], per_parent * h->U, ncclFloat64, 0, h->comm, h->stream);
    }
    if (g_nccl.GroupEnd() != ncclSuccess) return fail(h, PAMG_ERR_CUDA, "ncclGroupEnd failed in coarse scatter");
    Lc.tnew_alias = true; field_changed(Lc);
    return PAMG_OK;
  }
  // single process, several GPUs: the parts push their slices into part 0's memory (k_push), part 0 waits for the
  // flags, solves, and pushes the corrections back
  pamg_handle* g = h0->agg;
  LevelDev& A = g->lev[0];
  unsigned all = 0;
  for (size_t p = 1; p < G.size(); ++p) {
    pamg_handle* q = G[p];
    cudaSetDevice(q->device);
    LevelDev& Lc = q->lev[lvl - 1];
    int rc = launch_push(q, Lc.rhs, A.rhs + per_parent * q->part_first[p], (long long)(per_parent * q->U), 0,
                         h0->agg_words + AGG_FLAGS + p);
    if (rc) return gfail(owner, q, rc);
    all |= 1u << p;
  }
  {
    pamg_handle* h = h0;
    cudaSetDevice(h->device);
    LevelDev& Lc = h->lev[lvl - 1];
    CK(cudaMemcpyAsync(A.rhs, Lc.rhs, per_parent * h->U * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    CK(cudaMemsetAsync(A.T[A.cur], 0, A.ndof * sizeof(double), h->stream));
    int rc = launch_wait(h, all);
    if (rc) return gfail(owner, h, rc);
    A.tnew_alias = true; field_changed(A); A.rhs_valid = true;
    const long long l0 = g->launches;
    rc = vcycle_rec(Group{g}, g, 1, solver, nu1, nu2, ncoarse);
    h->launches += g->launches - l0;
    if (rc) { h->err = g->err; return gfail(owner, h, rc); }
    CK(cudaMemcpyAsync(Lc.T[Lc.cur], A.T[A.cur], per_parent * h->U * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    Lc.tnew_alias = true; field_changed(Lc);
    for (size_t p = 1; p < G.size(); ++p) {
      pamg_handle* q = G[p];
      LevelDev& Lq = q->lev[lvl - 1];
      rc = launch_push(h, A.T[A.cur] + per_parent * q->part_first[p], Lq.T[Lq.cur], (long long)(per_parent * q->U), (int)p,
                       q->agg_words + AGG_FLAGS + 0);
      if (rc) return gfail(owner, h, rc);
    }
  }
  for (size_t p = 1; p < G.size(); ++p) {
    pamg_handle* q = G[p];
    cudaSetDevice(q->device);
    int rc = launch_wait(q, 1u);
    if (rc) return gfail(owner, q, rc);
    LevelDev& Lq = q->lev[lvl - 1];
    Lq.tnew_alias = true; field_changed(Lq);
  }
  return PAMG_OK;
}

// Jacobi / Richardson sweeps ping-pong between the two T buffers; a cycle that ends on the other buffer would not
// be replayable as a CUDA graph (pointers are baked in), so the iterate is moved back when the sweep count is odd.
int normalise_parity(pamg_handle* h, LevelDev& L, int cur0) {
  if (L.cur == cur0) return PAMG_OK;
  CK(cudaMemcpyAsync(L.T[L.cur ^ 1], L.T[L.cur], L.ndof * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  L.cur ^= 1;
  L.tnew_alias = true;
  return PAMG_OK;
}

// skip_pre (top level of a solve with the fused convergence norm): the first pre-smoothing sweep of this cycle has already
// been run - it was the sweep that reduced the norm of the previous iterate - and the buffer parity is left to the caller
int vcycle_rec(const Group& G, pamg_handle* owner, int level, int solver, int nu1, int nu2, int ncoarse, int skip_pre) {
  const int Lmax = (int)G[0]->lev.size();
  std::vector<int> cur0(G.size());
  for (size_t i = 0; i < G.size(); ++i) cur0[i] = G[i]->lev[level - 1].cur;
  auto restore = [&]() -> int {
    for (size_t i = 0; i < G.size(); ++i) {
      if (G[i]->in_group) cudaSetDevice(G[i]->device);
      int rc = normalise_parity(G[i], G[i]->lev[level - 1], cur0[i]);
      if (rc) return gfail(owner, G[i], rc);
    }
    return PAMG_OK;
  };
  if (level == Lmax) {
    GALL(G, owner, q, do_smooth(q, level, solver, ncoarse));
    return restore();
  }
  GALL(G, owner, q, do_smooth(q, level, solver, nu1 - skip_pre));
  for (pamg_handle* q : G) q->lev[level - 1].tnew_alias = true;   // tnew = tnew_nonlin
  GALL(G, owner, q, do_residual(q, level, nullptr, nullptr, nullptr));
  GALL(G, owner, q, do_restrict(q, level));
  for (pamg_handle* q : G) {
    if (q->in_group) cudaSetDevice(q->device);
    LevelDev& Cc = q->lev[level];
    int rc = do_fill(q, Cc.T[Cc.cur], Cc.ndof, 0.0);
    if (rc) return gfail(owner, q, rc);
    Cc.tnew_alias = true;
    field_changed(Cc);
  }
  int rc;
  if (G[0]->agg_level && level + 1 == G[0]->agg_level) {
    if ((rc = agg_coarse_solve(G, owner, solver, nu1, nu2, ncoarse))) return rc;
  } else {
    if ((rc = vcycle_rec(G, owner, level + 1, solver, nu1, nu2, ncoarse))) return rc;
  }
  GALL(G, owner, q, do_prolong(q, level, false));
  GALL(G, owner, q, do_smooth(q, level, solver, nu2));
  return skip_pre ? PAMG_OK : restore();
}

// one V-cycle followed by the residual norms of level 1 (the copy to pinned memory is queued, not awaited).
// fuse (Jacobi): no residual evaluation of its own - the FIRST pre-smoothing sweep of the next cycle runs here and reduces
// the norms of the iterate it starts from (k_element_win2<.., NORM>); `first` = this is cycle 1, whose own first
// pre-sweep has not been run yet.  The sweep is undone (it wrote the other buffer) when the solve stops at this cycle.
int vcycle_body(const Group& G, pamg_handle* owner, int solver, int nu1, int nu2, int ncoarse, bool fuse = false, bool first = true) {
  int rc;
  if ((rc = vcycle_rec(G, owner, 1, solver, nu1, nu2, ncoarse, (fuse && !first) ? 1 : 0))) return rc;
  for (pamg_handle* q : G) q->lev[0].tnew_alias = true;
  if (fuse) {
    GALL(G, owner, q, do_smooth(q, 1, solver, 1, /*norm_first=*/true));
    GALL(G, owner, q, queue_norms(q));
    return PAMG_OK;
  }
  double dummy;
  GALL(G, owner, q, do_residual(q, 1, &dummy, nullptr, nullptr, /*queue_only=*/true));
  return PAMG_OK;
}

// take back the norm sweep at the end of a fused body: the iterate it started from still sits in the other T buffer, and
// the strips it read (local, unpacked cut faces) in the other strip buffer
int undo_norm_sweep(pamg_handle* h) {
  LevelDev& L = h->lev[0];
  const bool fusedk = h->p.face_terms && producer_level(L);
  L.cur ^= 1;
  L.tnew_alias = true;
  if (fusedk) L.ovl_cur ^= 1;
  sweep_undone(L, fusedk);
  return PAMG_OK;
}

// wait for every part, surface a failed exchange, combine the norms (the parts of one process hold partial sums;
// ranks of a multi-process run have already all-reduced theirs)
int group_norms(const Group& G, pamg_handle* owner, double* l2, double* linf, double* smax) {
  double s0 = 0.0, s1 = 0.0, s2 = 0.0;
  for (pamg_handle* q : G) {
    if (q->in_group) cudaSetDevice(q->device);
    CK_(q, cudaStreamSynchronize(q->stream));
    int rc = p2p_check(q);
    if (rc) return gfail(owner, q, rc);
    s0 += q->out3_host[0]; s1 = std::max(s1, q->out3_host[1]); s2 = std::max(s2, q->out3_host[2]);
  }
  for (pamg_handle* q : G) if (q != owner && !q->err.empty()) { owner->err = q->err; }
  if (l2) *l2 = std::sqrt(s0);
  if (linf) *linf = s1;
  if (smax) *smax = s2;
  return PAMG_OK;
}

void free_levels(pamg_handle* h) {
  for (auto& g : h->vc_graphs) for (auto e : g.exec) cudaGraphExecDestroy(e);
  h->vc_graphs.clear();
  for (auto& L : h->lev) {
    cudaFree(L.T[0]); cudaFree(L.T[1]); cudaFree(L.spare); cudaFree(L.told); cudaFree(L.rhs); cudaFree(L.res);
    cudaFree(L.ovl_old); cudaFree(L.pc); cudaFree(L.pc_old); cudaFree(L.xsend);
  }
  h->lev.clear();
  cudaFree(h->strip_arena); h->strip_arena = nullptr; h->strip_arena_bytes = 0;
  cudaFree(h->xg); cudaFree(h->strip_of); cudaFree(h->dst_strip); cudaFree(h->rev); cudaFree(h->hmap);
  cudaFree(h->nsrc); cudaFree(h->cut_lf); cudaFree(h->bc_kind); cudaFree(h->bc_val);
  cudaFree(h->partial);
  h->xg = nullptr; h->strip_of = h->dst_strip = h->rev = h->hmap = h->nsrc = h->cut_lf = h->bc_kind = nullptr;
  h->bc_val = nullptr; h->partial = nullptr;
}

}  // namespace

// ================================================================== C ABI
// root of a single-process multi-GPU handle: run the entry on every part
#define FANOUT(h, q, expr)                                                              \
  if ((h) && !(h)->parts.empty()) {                                                     \
    for (pamg_handle* q : (h)->parts) { int rc_ = (expr); if (rc_) return gfail((h), q, rc_); } \
    return PAMG_OK;                                                                     \
  }
// entries that only exist on a single device (unstructured front-ends, local inverse ...) run on part 0
#define ON_PART0(h) if ((h) && !(h)->parts.empty()) (h) = (h)->parts[0]

extern "C" {

const char* pamg_version(void) { return "pamg-b200 0.1 (sm_100a)"; }

int pamg_device_count(int* n) {
  if (!n) return PAMG_ERR_ARG;
  int c = 0;
  cudaError_t e = cudaGetDeviceCount(&c);
  if (e != cudaSuccess || c < 1) { *n = 0; return PAMG_ERR_CUDA; }
  *n = c;
  return PAMG_OK;
}

void pamg_default_params(pamg_params* p, int literal_head) {
  if (!p) return;
  std::memset(p, 0, sizeof(*p));
  p->n_split = 1; p->multi_levels = 1; p->n_smooth = 4; p->n_multigrid = 2; p->n_coarse_smooth = 15; p->solver = 3;
  p->theta = 1.0; p->k = 1.0; p->omega = 0.8; p->u_x = 0.0; p->u_y = 0.0;
  if (literal_head) {  // main.F90:46-47, transport_tri_semi.F90:117-140 as checked in
    p->dt = 1.25e-5; p->face_terms = 0; p->literal_source = 1; p->transfer = 0; p->residual_sign = 1;
    p->halo_rule = 0; p->coarse_bc_zero = 0; p->source_coef = -2.0; p->keep_tnew_gs = 1;
  } else {
    p->dt = 1e-3; p->face_terms = 1; p->literal_source = 0; p->transfer = 1; p->residual_sign = -1;
    p->halo_rule = 1; p->coarse_bc_zero = 1; p->source_coef = 2.0; p->keep_tnew_gs = 0;
  }
}

int pamg_create(const pamg_params* p, int device, pamg_handle** out) {
  if (!p || !out) return PAMG_ERR_ARG;
  *out = nullptr;
  if (p->n_split < 1 || p->n_split > 13 || p->multi_levels < 1 || p->multi_levels > p->n_split) return PAMG_ERR_ARG;  // :120-123
  if (!(p->theta >= 0.0 && p->theta <= 1.0)) return PAMG_ERR_ARG;
  if (!(p->dt > 0.0)) return PAMG_ERR_ARG;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) return PAMG_ERR_CUDA;  // no CPU fallback
  if (device < 0 || device >= ndev) return PAMG_ERR_ARG;
  pamg_handle* h = new pamg_handle();
  h->p = *p; h->device = device;
  const char* pp = getenv("PAMG_P2P");
  if (pp && pp[0] == '0') h->p2p_enabled = false;
  const char* pt = getenv("PAMG_P2P_TIMEOUT_S");
  if (pt && atof(pt) > 0.0) h->p2p_timeout_ns = (unsigned long long)(atof(pt) * 1e9);
  if (cudaSetDevice(device) != cudaSuccess) { delete h; return PAMG_ERR_CUDA; }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) h->nsm = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) { delete h; return PAMG_ERR_CUDA; }
  bool ok = true;
  for (auto& e : h->ev) ok = ok && cudaEventCreate(&e) == cudaSuccess;
  ok = ok && cudaMalloc(&h->out3, 3 * sizeof(double)) == cudaSuccess;
  ok = ok && cudaMallocHost(&h->out3_host, 3 * sizeof(double)) == cudaSuccess;
  ok = ok && configure_kernels(h) == PAMG_OK;
  if (!ok) { pamg_destroy(h); return PAMG_ERR_CUDA; }
  *out = h;
  return PAMG_OK;
}

// ---- single process, several GPUs (SURVEY 8(b): one host thread drives 1-8 devices; main.F90:16-51 is serial) ----------
namespace {
// peer pointers are plain device pointers here: enable peer access between the devices of the group, give every part its
// staging buffer / counters, and point the peers at each other
int group_p2p_setup(pamg_handle* root) {
  const Group& G = root->parts;
  for (pamg_handle* a : G)
    for (pamg_handle* b : G) {
      if (a->device == b->device) continue;
      int can = 0;
      CK_(root, cudaDeviceCanAccessPeer(&can, a->device, b->device));
      if (!can) return fail(root, PAMG_ERR_UNSUPPORTED, "the GPUs of the group cannot access each other's memory (no NVLink / PCIe peer access)");
      CK_(root, cudaSetDevice(a->device));
      cudaError_t e = cudaDeviceEnablePeerAccess(b->device, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail(root, PAMG_ERR_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
      (void)cudaGetLastError();
    }
  for (pamg_handle* q : G) {
    CK_(root, cudaSetDevice(q->device));
    if ((int)q->plan.peers.size() > P2P_MAXP) return fail(root, PAMG_ERR_UNSUPPORTED, "too many neighbour parts");
    int rc = p2p_alloc_local(q);
    if (rc) return gfail(root, q, rc);
    CK_(root, cudaMalloc(&q->agg_words, AGG_WORDS * sizeof(unsigned long long)));
    CK_(root, cudaMemset(q->agg_words, 0, AGG_WORDS * sizeof(unsigned long long)));
  }
  for (pamg_handle* q : G) {
    for (size_t i = 0; i < q->plan.peers.size(); ++i) {
      if (q->p2p_peers[i].slot_at_peer < 0) return fail(root, PAMG_ERR_STATE, "inconsistent halo plans between parts");
      q->p2p_peers[i].stage = G[q->plan.peers[i].part]->p2p_stage;
    }
  }
  // (parts that share one GPU use the same protocol: only the small halo / unpack kernels ever poll, never a sweep that
  // fills the device, so a kernel waiting for a peer cannot keep the peer's sweep from running)
  for (pamg_handle* q : G) {
    CK_(root, cudaSetDevice(q->device));
    int rc = p2p_upload_args(q);
    if (rc) return gfail(root, q, rc);
    q->p2p_ready = true;
  }
  return PAMG_OK;
}
}  // namespace

int pamg_create_multi(const pamg_params* p, int ngpus, const int* devices, pamg_handle** out) {
  if (!p || !out || ngpus < 1 || ngpus > 16) return PAMG_ERR_ARG;
  *out = nullptr;
  pamg_handle* root = new pamg_handle();
  root->p = *p; root->is_root = true;
  for (int i = 0; i < ngpus; ++i) {
    pamg_handle* q = nullptr;
    int rc = pamg_create(p, devices ? devices[i] : i, &q);
    if (rc) { pamg_destroy(root); return rc; }
    q->in_group = true; q->nranks = ngpus; q->rank = i;
    root->parts.push_back(q);
  }
  root->device = root->parts[0]->device; root->nsm = root->parts[0]->nsm;
  *out = root;
  return PAMG_OK;
}

void pamg_destroy(pamg_handle* h) {
  if (!h) return;
  if (h->is_root) {
    // root of a group (owns no device memory of its own besides cached graphs)
    for (pamg_handle* q : h->parts) { cudaSetDevice(q->device); if (q->stream) cudaStreamSynchronize(q->stream); }
    for (auto& g : h->vc_graphs) for (auto e : g.exec) cudaGraphExecDestroy(e);
    h->vc_graphs.clear();
    for (pamg_handle* q : h->parts) pamg_destroy(q);
    delete h;
    return;
  }
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  // graphs that contain NCCL nodes must go before the communicator
  for (auto& g : h->vc_graphs) for (auto e : g.exec) cudaGraphExecDestroy(e);
  h->vc_graphs.clear();
  if (h->stream) cudaStreamSynchronize(h->stream);
  if (h->agg) { pamg_destroy(h->agg); h->agg = nullptr; }
  if (h->comm) g_nccl.CommDestroy(h->comm);
  p2p_close(h);
  if (h->agg_words) { cudaFree(h->agg_words); h->agg_words = nullptr; }
  free_levels(h);
  unstr_free(h->un);
  cudaFree(h->out3); cudaFreeHost(h->out3_host); cudaFree(h->scratch);
  for (auto& e : h->ev) if (e) cudaEventDestroy(e);
  for (auto& e : h->pev) if (e) cudaEventDestroy(e);
  if (h->up_stream) { cudaStreamSynchronize(h->up_stream); cudaStreamSynchronize(h->down_stream); cudaStreamDestroy(h->up_stream); cudaStreamDestroy(h->down_stream); cudaEventDestroy(h->ev_up); cudaEventDestroy(h->ev_comp); cudaEventDestroy(h->ev_down[0]); cudaEventDestroy(h->ev_down[1]); }
  if (h->stream && !h->shared_stream) cudaStreamDestroy(h->stream);
  delete h;
}

const char* pamg_last_error(const pamg_handle* h) { return h ? h->err.c_str() : "null handle"; }

int pamg_set_parents_partition(pamg_handle* h, int U_global, const double* X, const int32_t* neig,
                               const int32_t* fneig, const int32_t* dir, int nparts, const int32_t* part_first,
                               int my_part) {
  if (!h) return PAMG_ERR_ARG;
  if (h->is_root) return fail(h, PAMG_ERR_ARG, "a multi-GPU handle partitions the mesh itself: call pamg_set_parents");
  CK(cudaSetDevice(h->device));
  int rc = build_halo_plan(U_global, X, neig, fneig, dir, h->p.halo_rule, nparts, part_first, my_part, h->plan);
  if (rc) return fail(h, rc, "inconsistent parent arrays (X / Neig / fNeig)");
  free_levels(h);
  if (h->agg) { pamg_destroy(h->agg); h->agg = nullptr; }
  h->agg_level = 0;
  // where my cut-face strips live in every peer's strip space (the peer's own plan, rebuilt here on the host)
  p2p_close(h);
  h->p2p_peers.assign(h->plan.peers.size(), pamg_handle::P2PPeer());
  for (size_t i = 0; i < h->plan.peers.size(); ++i) {
    HaloPlan theirs;
    if (build_halo_plan(U_global, X, neig, fneig, dir, h->p.halo_rule, nparts, part_first, h->plan.peers[i].part, theirs)) continue;
    for (size_t j = 0; j < theirs.peers.size(); ++j)
      h->p2p_peers[i].recv_strips_at_peer = std::max(h->p2p_peers[i].recv_strips_at_peer, (long long)theirs.peers[j].strip_begin + theirs.peers[j].nfaces);
    for (size_t j = 0; j < theirs.peers.size(); ++j)
      if (theirs.peers[j].part == my_part && theirs.peers[j].nfaces == h->plan.peers[i].nfaces) {
        h->p2p_peers[i].slot_at_peer = (int)j;
        h->p2p_peers[i].strip_begin_at_peer = theirs.peers[j].strip_begin;
      }
  }
  const int U = h->plan.U_local, first = h->plan.first;
  if (U < 1) return fail(h, PAMG_ERR_ARG, "empty partition");
  h->U = U; h->U_global = U_global;
  h->part_first.assign(nparts + 1, 0);
  if (part_first) for (int i = 0; i <= nparts; ++i) h->part_first[i] = part_first[i]; else h->part_first[1] = U_global;
  std::vector<double> xg((size_t)U * 6);
  for (int u = 0; u < U; ++u) {
    const double* P = X + (size_t)(first + u) * 6;
    double* o = &xg[(size_t)u * 6];
    o[0] = P[4]; o[1] = P[5]; o[2] = P[0] - P[4]; o[3] = P[1] - P[5]; o[4] = P[2] - P[4]; o[5] = P[3] - P[5];
  }
  CK(cudaMalloc(&h->xg, xg.size() * sizeof(double)));
  CK(cudaMemcpy(h->xg, xg.data(), xg.size() * sizeof(double), cudaMemcpyHostToDevice));
  const size_t n3 = (size_t)U * 3 * sizeof(int32_t);
  CK(cudaMalloc(&h->strip_of, n3)); CK(cudaMalloc(&h->dst_strip, n3)); CK(cudaMalloc(&h->rev, n3)); CK(cudaMalloc(&h->hmap, n3));
  CK(cudaMemcpy(h->strip_of, h->plan.strip_of.data(), n3, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(h->dst_strip, h->plan.dst_strip.data(), n3, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(h->rev, h->plan.rev.data(), n3, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(h->hmap, h->plan.hmap.data(), n3, cudaMemcpyHostToDevice));
  CK(cudaMalloc(&h->nsrc, n3));
  CK(cudaMemcpy(h->nsrc, h->plan.nsrc.data(), n3, cudaMemcpyHostToDevice));
  if (!h->plan.cut_lf.empty()) {
    CK(cudaMalloc(&h->cut_lf, h->plan.cut_lf.size() * sizeof(int32_t)));
    CK(cudaMemcpy(h->cut_lf, h->plan.cut_lf.data(), h->plan.cut_lf.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
  }
  // Dirichlet data of the domain-boundary faces (pamg_set_boundary_data), local slice on the device
  const int32_t* bc_glob = nullptr;
  if (!h->bc_kind_h.empty()) {
    if ((int)h->bc_kind_h.size() != U_global * 3) return fail(h, PAMG_ERR_ARG, "pamg_set_boundary_data was given a different number of parents");
    bc_glob = h->bc_kind_h.data();
    CK(cudaMalloc(&h->bc_kind, n3)); CK(cudaMalloc(&h->bc_val, (size_t)U * 3 * sizeof(double)));
    CK(cudaMemcpy(h->bc_kind, h->bc_kind_h.data() + (size_t)first * 3, n3, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->bc_val, h->bc_val_h.data() + (size_t)first * 3, (size_t)U * 3 * sizeof(double), cudaMemcpyHostToDevice));
  }
  h->lev.resize(h->p.multi_levels);
  {
    size_t tot = 0;
    for (int il = 0; il < h->p.multi_levels; ++il) {
      const size_t S = (size_t)1 << (h->p.n_split - il);
      tot += 2 * (((size_t)(h->plan.nstrips + h->plan.nsend) * 3 * S * sizeof(double) + 255) / 256 * 256);
    }
    CK(cudaMalloc(&h->strip_arena, tot));
    CK(cudaMemsetAsync(h->strip_arena, 0, tot, h->stream));
    h->strip_arena_bytes = tot;
    if (!h->shared_stream) {
      // best effort: devices / driver modes without persisting L2 simply run without the window
      cudaDeviceProp prop;
      if (cudaGetDeviceProperties(&prop, h->device) == cudaSuccess && prop.persistingL2CacheMaxSize > 0) {
        const size_t want = std::min((size_t)prop.persistingL2CacheMaxSize, std::max(tot, (size_t)1 << 20));
        cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want);
        cudaStreamAttrValue av;
        std::memset(&av, 0, sizeof(av));
        av.accessPolicyWindow.base_ptr = h->strip_arena;
        av.accessPolicyWindow.num_bytes = std::min(tot, (size_t)prop.accessPolicyMaxWindowSize);
        av.accessPolicyWindow.hitRatio = (float)std::min(1.0, (double)want / (double)std::max(tot, (size_t)1));
        av.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        av.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
        cudaStreamSetAttribute(h->stream, cudaStreamAttributeAccessPolicyWindow, &av);
        (void)cudaGetLastError();
      }
    }
  }
  size_t arena_off = 0;
  std::vector<double> pc((size_t)U * NPC);
  for (int il = 0; il < h->p.multi_levels; ++il) {
    LevelDev& L = h->lev[il];
    L.s = h->p.n_split - il; L.S = 1 << L.s; L.C = 1ll << (2 * L.s);
    L.nelem = L.C * U; L.ndof = 3 * L.nelem;
    const size_t fb = (size_t)L.ndof * sizeof(double);
    CK(cudaMalloc(&L.T[0], fb)); CK(cudaMalloc(&L.T[1], fb)); CK(cudaMalloc(&L.told, fb));
    CK(cudaMalloc(&L.rhs, fb)); CK(cudaMalloc(&L.res, fb));
    CK(cudaMemsetAsync(L.T[0], 0, fb, h->stream)); CK(cudaMemsetAsync(L.T[1], 0, fb, h->stream));
    CK(cudaMemsetAsync(L.told, 0, fb, h->stream)); CK(cudaMemsetAsync(L.rhs, 0, fb, h->stream));
    CK(cudaMemsetAsync(L.res, 0, fb, h->stream));
    const size_t ob = (size_t)(h->plan.nstrips + h->plan.nsend) * 3 * L.S * sizeof(double);
    const size_t obp = (ob + 255) / 256 * 256;
    L.ovlb[0] = reinterpret_cast<double*>(reinterpret_cast<char*>(h->strip_arena) + arena_off);
    L.ovlb[1] = reinterpret_cast<double*>(reinterpret_cast<char*>(h->strip_arena) + arena_off + obp);
    arena_off += 2 * obp;
    CK(cudaMalloc(&L.ovl_old, ob));
    CK(cudaMemsetAsync(L.ovl_old, 0, ob, h->stream));  // :207
    for (int u = 0; u < U; ++u)
      if (!parent_coefficients(h->p, X, neig, bc_glob, first + u, L.s, &pc[(size_t)u * NPC], h->p.theta))
        return fail(h, PAMG_ERR_UNSUPPORTED, "open boundary face (kind 2) with inflow: give it Dirichlet data instead");
    CK(cudaMalloc(&L.pc, pc.size() * sizeof(double)));
    CK(cudaMemcpy(L.pc, pc.data(), pc.size() * sizeof(double), cudaMemcpyHostToDevice));
    if (il == 0 && h->p.theta != 1.0 && h->level_offset == 0) {
      // old-time operator of get_RHS (:459-460), applied to TOLD when the level-1 right-hand side is built
      for (int u = 0; u < U; ++u)
        if (!parent_coefficients(h->p, X, neig, bc_glob, first + u, L.s, &pc[(size_t)u * NPC], 1.0 - h->p.theta, false))
          return fail(h, PAMG_ERR_UNSUPPORTED, "open boundary face (kind 2) with inflow: give it Dirichlet data instead");
      CK(cudaMalloc(&L.pc_old, pc.size() * sizeof(double)));
      CK(cudaMemcpy(L.pc_old, pc.data(), pc.size() * sizeof(double), cudaMemcpyHostToDevice));
    }
    L.cur = 0; L.tnew_alias = true; L.rhs_valid = (il != 0);
  }
  // Dirichlet data sin(x+y) on domain-boundary faces never changes: fill those strips once per level, in both strip
  // buffers, and in the told strips of level 1, which the old-time face terms read (theta != 1)
  for (auto& Lv : h->lev)
    for (double* ovl : {Lv.ovlb[0], Lv.ovlb[1]})
      if ((rc = launch_halo_kernel(h, Lv, HALO_DIRICHLET, nullptr, ovl))) return rc;
  LevelDev& L1 = h->lev[0];
  if (L1.pc_old && (rc = launch_halo_kernel(h, L1, HALO_DIRICHLET, nullptr, L1.ovl_old))) return rc;
  // coarse-level agglomeration on part 0: first level whose GLOBAL size is small enough to be launch-bound
  if (nparts > 1 && h->level_offset == 0) {
    const char* e = getenv("PAMG_AGG_ELEMS");
    // elements of the whole mesh on that level; 0 disables.  With the halo exchange at ~1.5 us per sweep the break-even
    // moved down: 2^21 cost 2.6 ms per solve at 4 GPUs against 2^17 (profiles/README.md)
    const long long limit = e ? atoll(e) : (1ll << 17);
    int lvl = 0;
    for (int il = 2; il <= h->p.multi_levels; ++il)
      if (limit > 0 && (long long)U_global * h->lev[il - 1].C <= limit) { lvl = il; break; }
    if (lvl) {
      h->agg_level = lvl;
      if (my_part == 0) {
        pamg_params ap = h->p;
        ap.n_split = h->lev[lvl - 1].s;
        ap.multi_levels = h->p.multi_levels - lvl + 1;
        pamg_handle* g = new pamg_handle();
        g->p = ap; g->device = h->device; g->nsm = h->nsm;
        g->stream = h->stream; g->shared_stream = true; g->level_offset = lvl - 1;
        g->bc_kind_h = h->bc_kind_h; g->bc_val_h = h->bc_val_h;
        h->agg = g;
        for (auto& ev : g->ev) CK(cudaEventCreate(&ev));
        CK(cudaMalloc(&g->out3, 3 * sizeof(double)));
        CK(cudaMallocHost(&g->out3_host, 3 * sizeof(double)));
        if (configure_kernels(g)) return fail(h, PAMG_ERR_CUDA, g->err);
        int rc3 = pamg_set_parents_partition(g, U_global, X, neig, fneig, dir, 1, nullptr, 0);
        if (rc3) return fail(h, rc3, std::string("agglomerated coarse problem: ") + g->err);
      }
    }
  }
  h->npartial = h->nsm * 16;
  CK(cudaMalloc(&h->partial, (size_t)h->npartial * 3 * sizeof(double)));
  CK(cudaStreamSynchronize(h->stream));
  return PAMG_OK;
}

int pamg_halo_sources(int U_global, const double* X, const int32_t* neig, const int32_t* fneig, const int32_t* dir,
                      int halo_rule, int nparts, const int32_t* part_first, int my_part, int s, int64_t* src) {
  if (!src || s < 1 || s > 13) return PAMG_ERR_ARG;
  HaloPlan plan;
  int rc = build_halo_plan(U_global, X, neig, fneig, dir, halo_rule, nparts, part_first, my_part, plan);
  if (rc != PAMG_OK) return rc;
  const int S = 1 << s;
  for (int lf = 0; lf < plan.U_local * 3; ++lf) {
    const int d = plan.nsrc[lf];
    for (int p = 0; p < S; ++p) {
      int64_t* o = src + ((size_t)lf * S + p) * 2;
      if (d < 0) { o[0] = o[1] = -1; continue; }
      const size_t base = nbr_child_offset(d, p, s);
      o[0] = (int64_t)(base + (d & 3)); o[1] = (int64_t)(base + ((d >> 2) & 3));
    }
  }
  return PAMG_OK;
}

int pamg_numbering(int what, int s, int64_t first, int64_t count, int32_t* out) {
  if (!out || s < 1 || s > 13 || what < 0 || what > 3 || first < 0 || count < 0) return PAMG_ERR_ARG;
  const int64_t C = (int64_t)1 << (2 * s);
  if (first + count > C) return PAMG_ERR_ARG;
  const int b = 2 << s;
  for (int64_t i = 0; i < count; ++i) {
    const int k = (int)(first + i);
    int32_t* o = out + 4 * i;
    int r = 0, ipos = 0, ele = 0, len = 0;
    if (what == 0) { child_from_ele0(k, s, r, ipos, len); o[0] = r; o[1] = ipos; o[2] = len; o[3] = 0; }
    else if (what == 1) { child_from_flat(k, s, r, ipos, ele, len); o[0] = r; o[1] = ipos; o[2] = ele; o[3] = len; }
    else if (what == 2) { int fin[4]; child_from_ele0(k, s, r, ipos, len); fine_children(s, r, ipos, fin); for (int q = 0; q < 4; ++q) o[q] = fin[q]; }
    else {
      if (k + TPB >= C) { o[0] = o[1] = o[2] = o[3] = 0; continue; }
      child_from_ele0(k, s, r, ipos, len);
      child_advance(s, b, k + TPB, r, ipos);
      o[0] = r; o[1] = ipos; o[2] = b + 1 - 2 * r; o[3] = 0;
    }
  }
  return PAMG_OK;
}

int pamg_parent_table(const pamg_params* p, int U, const double* X, const int32_t* neig, const int32_t* bc_kind, int parent,
                      int s, double theta_weight, int with_mass, double* table) {
  if (!p || !X || !neig || !table || U < 1 || parent < 0 || parent >= U || s < 0 || s > 13 || !(p->dt > 0.0)) return PAMG_ERR_ARG;
  for (int f = 0; f < 3; ++f) { const int q = neig[(size_t)parent * 3 + f]; if (q < 0 || q > U) return PAMG_ERR_ARG; }
  return parent_coefficients(*p, X, neig, bc_kind, parent, s, table, theta_weight, with_mass != 0) ? PAMG_OK : PAMG_ERR_UNSUPPORTED;
}

int pamg_set_boundary_data(pamg_handle* h, int U_global, const int32_t* kind, const double* value) {
  if (!h || U_global < 1 || !kind) return PAMG_ERR_ARG;
  for (size_t i = 0; i < (size_t)U_global * 3; ++i)
    if (kind[i] < 0 || kind[i] > 2) return fail(h, PAMG_ERR_ARG, "boundary kind must be 0 (sin(x+y)), 1 (constant) or 2 (open)");
  h->bc_kind_h.assign(kind, kind + (size_t)U_global * 3);
  if (value) h->bc_val_h.assign(value, value + (size_t)U_global * 3);
  else h->bc_val_h.assign((size_t)U_global * 3, 0.0);
  FANOUT(h, q, pamg_set_boundary_data(q, U_global, kind, value));
  if (!h->lev.empty()) return fail(h, PAMG_ERR_STATE, "pamg_set_boundary_data must precede pamg_set_parents (the coefficient tables depend on it)");
  return PAMG_OK;
}

int pamg_set_parents(pamg_handle* h, int U, const double* X, const int32_t* neig, const int32_t* fneig,
                     const int32_t* dir) {
  if (h && h->is_root) {
    // contiguous blocks of parents per GPU (the scheme Generic.F90:387-401 sketches); one part per device
    const int n = (int)h->parts.size();
    if (U < n) return fail(h, PAMG_ERR_ARG, "fewer parents than GPUs");
    std::vector<int32_t> pf(n + 1);
    for (int i = 0; i <= n; ++i) pf[i] = (int32_t)((long long)U * i / n);
    for (auto& g : h->vc_graphs) for (auto e : g.exec) cudaGraphExecDestroy(e);
    h->vc_graphs.clear();
    for (int i = 0; i < n; ++i) {
      pamg_handle* q = h->parts[i];
      if (q->agg_words) { cudaSetDevice(q->device); cudaFree(q->agg_words); q->agg_words = nullptr; }
      int rc = pamg_set_parents_partition(q, U, X, neig, fneig, dir, n, pf.data(), i);
      if (rc) return gfail(h, q, rc);
    }
    h->U = U; h->U_global = U;
    return n > 1 ? group_p2p_setup(h) : PAMG_OK;
  }
  return pamg_set_parents_partition(h, U, X, neig, fneig, dir, 1, nullptr, 0);
}

int pamg_ndof(const pamg_handle* h, int level, int64_t* ndof) {
  if (h && h->is_root && ndof) {
    *ndof = 0;
    for (const pamg_handle* q : h->parts) { if (!valid_level(q, level)) return PAMG_ERR_ARG; *ndof += q->lev[level - 1].ndof; }
    return PAMG_OK;
  }
  if (!valid_level(h, level) || !ndof) return PAMG_ERR_ARG;
  *ndof = h->lev[level - 1].ndof;
  return PAMG_OK;
}

int pamg_upload_field(pamg_handle* h, int field, int level, const double* host) {
  if (h && h->is_root && host) {    // parts own contiguous blocks of parents = contiguous ranges of the field
    size_t off = 0;
    for (pamg_handle* q : h->parts) {
      int rc = pamg_upload_field(q, field, level, host + off);
      if (rc) return gfail(h, q, rc);
      off += (size_t)q->lev[level - 1].ndof;
    }
    return PAMG_OK;
  }
  if (!valid_level(h, level) || !host) return PAMG_ERR_ARG;
  CK(cudaSetDevice(h->device));
  int rc;
  double* d = field_ptr(h, field, level, true, &rc);
  if (rc) return rc;
  CK(cudaMemcpyAsync(d, host, h->lev[level - 1].ndof * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return PAMG_OK;
}

int pamg_download_field(pamg_handle* h, int field, int level, double* host) {
  if (h && h->is_root && host) {
    size_t off = 0;
    for (pamg_handle* q : h->parts) {
      int rc = pamg_download_field(q, field, level, host + off);
      if (rc) return gfail(h, q, rc);
      off += (size_t)q->lev[level - 1].ndof;
    }
    return PAMG_OK;
  }
  if (!valid_level(h, level) || !host) return PAMG_ERR_ARG;
  CK(cudaSetDevice(h->device));
  int rc;
  double* d = field_ptr(h, field, level, false, &rc);
  if (rc) return rc;
  CK(cudaMemcpyAsync(host, d, h->lev[level - 1].ndof * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return p2p_check(h);
}

int pamg_fill_field(pamg_handle* h, int field, int level, double value) {
  FANOUT(h, q, pamg_fill_field(q, field, level, value));
  if (!valid_level(h, level)) return PAMG_ERR_ARG;
  CK(cudaSetDevice(h->device));
  int rc;
  double* d = field_ptr(h, field, level, true, &rc);
  if (rc) return rc;
  return do_fill(h, d, h->lev[level - 1].ndof, value);
}

int pamg_copy_field(pamg_handle* h, int level, int dst_field, int src_field) {
  FANOUT(h, q, pamg_copy_field(q, level, dst_field, src_field));
  if (!valid_level(h, level)) return PAMG_ERR_ARG;
  CK(cudaSetDevice(h->device));
  LevelDev& L = h->lev[level - 1];
  if (dst_field == src_field) return PAMG_OK;
  if (dst_field == PAMG_TNEW && src_field == PAMG_TNONLIN) { L.tnew_alias = true; return PAMG_OK; }      // :550
  if (dst_field == PAMG_TNONLIN && src_field == PAMG_TNEW) {                                             // :327
    if (!L.tnew_alias) { L.cur ^= 1; L.tnew_alias = true; field_changed(L); }
    return PAMG_OK;
  }
  int rc;
  const double* s = field_ptr(h, src_field, level, false, &rc);
  if (rc) return rc;
  double* d = field_ptr(h, dst_field, level, true, &rc);
  if (rc) return rc;
  CK(cudaMemcpyAsync(d, s, L.ndof * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  return PAMG_OK;
}

int pamg_download_overlap(pamg_handle* h, int level, int old, double* host) {
  if (h && h->is_root && host) {
    size_t off = 0;
    for (pamg_handle* q : h->parts) {
      int rc = pamg_download_overlap(q, level, old, host + off);
      if (rc) return gfail(h, q, rc);
      off += (size_t)q->U * 9 * q->lev[level - 1].S;
    }
    return PAMG_OK;
  }
  if (!valid_level(h, level) || !host) return PAMG_ERR_ARG;
  CK(cudaSetDevice(h->device));
  LevelDev& L = h->lev[level - 1];
  const size_t S3 = (size_t)3 * L.S;
  std::vector<double> tmp((size_t)h->plan.nstrips * S3);
  CK(cudaMemcpyAsync(tmp.data(), old ? L.ovl_old : L.ovlb[L.ovl_cur], tmp.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  for (int lf = 0; lf < h->U * 3; ++lf)
    std::memcpy(host + (size_t)lf * S3, &tmp[(size_t)h->plan.strip_of[lf] * S3], S3 * sizeof(double));
  return PAMG_OK;
}

int pamg_device_ptr(pamg_handle* h, int field, int level, void** dptr) {
  if (h && h->is_root) return fail(h, PAMG_ERR_UNSUPPORTED, "a multi-GPU handle has no single device pointer per field");
  if (!valid_level(h, level) || !dptr) return PAMG_ERR_ARG;
  int rc;
  *dptr = field_ptr(h, field, level, false, &rc);
  return rc;
}

int pamg_update_overlaps(pamg_handle* h, int level) {
  FANOUT(h, q, pamg_update_overlaps(q, level));
  if (!valid_level(h, level)) return PAMG_ERR_ARG;
  CK(cudaSetDevice(h->device));
  return launch_halo(h, level, HALO_ALL);
}

int pamg_build_rhs(pamg_handle* h) {
  FANOUT(h, q, pamg_build_rhs(q));
  if (!valid_level(h, 1)) return PAMG_ERR_STATE;
  CK(cudaSetDevice(h->device));
  return launch_build_rhs(h);
}

int pamg_smooth(pamg_handle* h, int level, int solver, int nsweeps) {
  if (h && h->is_root) {
    // lockstep in small batches: a part whose exchange kernel waits for a peer must never have so many launches queued
    // behind it that the host blocks before it has queued the peer's work
    for (int done = 0; done < nsweeps; done += 4)
      for (pamg_handle* q : h->parts) { int rc = pamg_smooth(q, level, solver, std::min(4, nsweeps - done)); if (rc) return gfail(h, q, rc); }
    return PAMG_OK;
  }
  if (!valid_level(h, level) || nsweeps < 0) return PAMG_ERR_ARG;
  CK(cudaSetDevice(h->device));
  return do_smooth(h, level, solver, nsweeps);
}

int pamg_residual(pamg_handle* h, int level, double* l2, double* linf) {
  if (h && h->is_root) {
    const Group& G = h->parts;
    if (!valid_level(G[0], level)) return PAMG_ERR_ARG;
    double dummy;
    GALL(G, h, q, do_residual(q, level, &dummy, nullptr, nullptr, true));
    return group_norms(G, h, l2, linf, nullptr);
  }
  if (!valid_level(h, level)) return PAMG_ERR_ARG;
  CK(cudaSetDevice(h->device));
  return do_residual(h, level, l2, linf, nullptr);
}

int pamg_convergence(pamg_handle* h, int level, double* conv) {
  if (h && h->is_root && conv) {
    const Group& G = h->parts;
    if (!valid_level(G[0], level)) return PAMG_ERR_ARG;
    double dummy;
    GALL(G, h, q, do_residual(q, level, &dummy, nullptr, nullptr, true));
    return group_norms(G, h, nullptr, nullptr, conv);
  }
  if (!valid_level(h, level) || !conv) return PAMG_ERR_ARG;
  CK(cudaSetDevice(h->device));
  double l2, li;
  return do_residual(h, level, &l2, &li, conv);
}

int pamg_restrict(pamg_handle* h, int fine_level) {
  FANOUT(h, q, pamg_restrict(q, fine_level));
  if (!valid_level(h, fine_level)) return PAMG_ERR_ARG;
  CK(cudaSetDevice(h->device));
  return do_restrict(h, fine_level);
}

int pamg_prolong(pamg_handle* h, int fine_level) {
  FANOUT(h, q, pamg_prolong(q, fine_level));
  if (!valid_level(h, fine_level)) return PAMG_ERR_ARG;
  CK(cudaSetDevice(h->device));
  return do_prolong(h, fine_level);
}

int pamg_vcycle_solve(pamg_handle* h, int solver, int nu1, int nu2, int ncoarse, int max_cycles, double tol,
                      int* cycles, double* hist) {
  if (!h || max_cycles < 0) return PAMG_ERR_ARG;
  const Group G = group_of(h);
  if (!valid_level(G[0], 1)) return PAMG_ERR_ARG;
  CK(cudaSetDevice(G[0]->device));
  int rc;
  for (pamg_handle* q : G) { LevelDev& L = q->lev[0]; L.tnew_alias = true; field_changed(L); }
  double r0 = 0, r = 0, dummy;
  GALL(G, h, q, do_residual(q, 1, &dummy, nullptr, nullptr, true));
  if ((rc = group_norms(G, h, &r0, nullptr, nullptr))) return rc;
  if (hist) hist[0] = r0;
  if (cycles) *cycles = 0;
  if (r0 == 0.0) return PAMG_OK;
  // cycle 1 runs eagerly; from cycle 2 on the identical launch sequence (most of it on launch-bound coarse levels) is
  // replayed as one CUDA graph per GPU
  // Jacobi: no residual evaluation per cycle - the first pre-smoothing sweep of the next cycle reduces the norms of the iterate
  // it starts from (same numbers as get_residual's), and is taken back when the solve stops
  bool fuse = solver == 1 && nu1 >= 1;
  for (pamg_handle* q : G) fuse = fuse && norm_fusable(q, q->lev[0]);
  bool swept = false;                       // a fused body has run: its trailing norm sweep is pending
  auto finish = [&]() -> int {
    if (!fuse || !swept) return PAMG_OK;
    for (pamg_handle* q : G) { if (q->in_group) cudaSetDevice(q->device); int rc2 = undo_norm_sweep(q); if (rc2) return gfail(h, q, rc2); }
    GALL(G, h, q, do_residual(q, 1, nullptr, nullptr, nullptr));      // leaves tracer%residuale of the final iterate, as before
    return PAMG_OK;
  };
  const long long key0 = (((((long long)solver * 64 + nu1) * 64 + nu2) * 64 + ncoarse) * 2 + (fuse ? 1 : 0));
  // with NCCL in the cycle (halo exchange fallback, coarse gather/scatter) the capture is attempted once; if the library
  // refuses, the handle falls back to eager launches for good
  bool graph_ok = true;
  for (pamg_handle* q : G) graph_ok = graph_ok && !q->profiling && (!q->comm || q->graph_nccl);
  for (int c = 1; c <= max_cycles; ++c) {
    if (c >= 2 && graph_ok) {
      // the graph bakes in which of the two T buffers holds the iterate and which strip buffer is current, on every level of
      // every part (a hash: the product of the factors does not fit 64 bits for a group of GPUs)
      unsigned long long hk = (unsigned long long)key0;
      for (pamg_handle* q : G) for (auto& Lv : q->lev) hk = hk * 1000003ull + (unsigned long long)(Lv.cur * 2 + Lv.ovl_cur + 1);
      const long long key = (long long)hk;
      pamg_handle::VcGraph* vg = nullptr;
      for (auto& g : h->vc_graphs) if (g.key == key) vg = &g;
      if (!vg) {
        if (h->vc_graphs.size() >= 8) { for (auto e : h->vc_graphs.front().exec) cudaGraphExecDestroy(e); h->vc_graphs.erase(h->vc_graphs.begin()); }
        std::vector<long long> l0(G.size());
        size_t begun = 0;
        cudaError_t ce = cudaSuccess;
        for (; begun < G.size(); ++begun) {
          pamg_handle* q = G[begun];
          if (q->in_group) cudaSetDevice(q->device);
          l0[begun] = q->launches;
          ce = cudaStreamBeginCapture(q->stream, G.size() > 1 ? cudaStreamCaptureModeRelaxed : cudaStreamCaptureModeThreadLocal);
          if (ce != cudaSuccess) break;
          q->capturing = true;
        }
        rc = (ce == cudaSuccess) ? vcycle_body(G, h, solver, nu1, nu2, ncoarse, fuse, false) : PAMG_ERR_CUDA;
        pamg_handle::VcGraph ng;
        ng.key = key;
        for (size_t i = 0; i < begun; ++i) {
          pamg_handle* q = G[i];
          if (q->in_group) cudaSetDevice(q->device);
          q->capturing = false;
          cudaGraph_t graph = nullptr;
          cudaError_t e2 = cudaStreamEndCapture(q->stream, &graph);
          ng.launches.push_back(q->launches - l0[i]);
          q->launches = l0[i];
          cudaGraphExec_t ex = nullptr;
          if (!rc && ce == cudaSuccess && e2 == cudaSuccess) e2 = cudaGraphInstantiate(&ex, graph, 0);
          if (graph) cudaGraphDestroy(graph);
          if (e2 != cudaSuccess && ce == cudaSuccess) ce = e2;
          if (ex) ng.exec.push_back(ex);
        }
        if (rc || ce != cudaSuccess) {
          for (auto e : ng.exec) cudaGraphExecDestroy(e);
          (void)cudaGetLastError();
          bool nccl = false;
          for (pamg_handle* q : G) nccl = nccl || q->comm;
          if (!nccl) {
            if (rc && rc != PAMG_ERR_CUDA) return rc;
            return fail(h, PAMG_ERR_CUDA, std::string("CUDA graph capture of the V-cycle: ") + cudaGetErrorString(ce));
          }
          // NCCL inside the capture was refused: run eagerly from now on (host-side state is periodic per cycle)
          for (pamg_handle* q : G) q->graph_nccl = false;
          graph_ok = false;
          if ((rc = vcycle_body(G, h, solver, nu1, nu2, ncoarse, fuse, false))) return rc;
          goto cycle_done;
        }
        h->vc_graphs.push_back(ng);
        vg = &h->vc_graphs.back();
      }
      for (size_t i = 0; i < G.size(); ++i) {
        if (G[i]->in_group) cudaSetDevice(G[i]->device);
        CK(cudaGraphLaunch(vg->exec[i], G[i]->stream));
        G[i]->launches += vg->launches[i];
      }
    } else {
      if ((rc = vcycle_body(G, h, solver, nu1, nu2, ncoarse, fuse, c == 1))) return rc;
    }
  cycle_done:
    swept = true;
    if ((rc = group_norms(G, h, &r, nullptr, nullptr))) return rc;
    if (hist) hist[c] = r;
    if (cycles) *cycles = c;
    if (r / r0 <= tol) return finish();
  }
  if (cycles) *cycles = max_cycles + 1;
  return finish();
}

int pamg_literal_timestep(pamg_handle* h, int solver, int n_multigrid, int n_smooth) {
  if (!h) return PAMG_ERR_ARG;
  const Group G = group_of(h);
  if (!valid_level(G[0], 1)) return PAMG_ERR_STATE;
  CK(cudaSetDevice(G[0]->device));
  const int ML = (int)G[0]->lev.size();
  GALL(G, h, q, pamg_copy_field(q, 1, PAMG_TOLD, PAMG_TNEW));      // :316
  GALL(G, h, q, pamg_copy_field(q, 1, PAMG_TNONLIN, PAMG_TNEW));   // :317
  for (int mg = 0; mg < n_multigrid; ++mg) {
    for (int il = 1; il <= ML; ++il) {
      GALL(G, h, q, pamg_copy_field(q, il, PAMG_TNONLIN, PAMG_TNEW));   // :327
      GALL(G, h, q, do_smooth(q, il, solver, n_smooth));                // :331
      GALL(G, h, q, do_restrict(q, il));                                // :336
      GALL(G, h, q, do_residual(q, il, nullptr, nullptr, nullptr));     // :338
    }
    GALL(G, h, q, pamg_copy_field(q, ML, PAMG_TNONLIN, PAMG_TNEW));     // :348
    for (int i = 0; i < G[0]->p.n_coarse_smooth; ++i)
      GALL(G, h, q, do_smooth(q, ML, solver, n_smooth));                // :351-352
    for (int il = ML - 1; il >= 1; --il) {
      GALL(G, h, q, pamg_copy_field(q, il, PAMG_TNONLIN, PAMG_TNEW));   // :367
      GALL(G, h, q, do_prolong(q, il));                                 // :370
      GALL(G, h, q, do_smooth(q, il, solver, n_smooth));                // :376
    }
  }
  return PAMG_OK;
}

int pamg_timestep_host(pamg_handle* h, const double* tnew_in, double* tnew_out, int max_cycles, double tol,
                       int* cycles, double* relres) {
  if (!h || !tnew_in || !tnew_out) return PAMG_ERR_ARG;
  const Group G = group_of(h);
  if (!valid_level(G[0], 1)) return PAMG_ERR_ARG;
  // told = tnew ; tnew_nonlin = tnew (transport_tri_semi.F90:316-317)
  size_t off = 0;
  for (pamg_handle* q : G) {
    CK_(q, cudaSetDevice(q->device));
    LevelDev& L = q->lev[0];
    const size_t bytes = (size_t)L.ndof * sizeof(double);
    CK_(q, cudaMemcpyAsync(L.T[L.cur], tnew_in + off, bytes, cudaMemcpyHostToDevice, q->stream));
    L.tnew_alias = true;
    field_changed(L);
    CK_(q, cudaMemcpyAsync(L.told, L.T[L.cur], bytes, cudaMemcpyDeviceToDevice, q->stream));
    L.rhs_valid = false;
    off += (size_t)L.ndof;
  }
  std::vector<double> hist((size_t)max_cycles + 2, 0.0);
  int cyc = 0;
  const pamg_params& P = G[0]->p;
  int rc = pamg_vcycle_solve(h, P.solver, P.n_smooth, P.n_smooth, P.n_coarse_smooth, max_cycles, tol, &cyc, hist.data());
  if (rc) return rc;
  if (cycles) *cycles = cyc;
  if (relres) *relres = hist[0] > 0 ? hist[std::min(cyc, max_cycles)] / hist[0] : 0.0;
  off = 0;
  for (pamg_handle* q : G) {
    CK_(q, cudaSetDevice(q->device));
    LevelDev& L = q->lev[0];
    CK_(q, cudaMemcpyAsync(tnew_out + off, L.T[L.cur], (size_t)L.ndof * sizeof(double), cudaMemcpyDeviceToHost, q->stream));
    off += (size_t)L.ndof;
  }
  for (pamg_handle* q : G) {
    CK_(q, cudaSetDevice(q->device));
    CK_(q, cudaStreamSynchronize(q->stream));
    if ((rc = p2p_check(q))) return gfail(h, q, rc);
  }
  return PAMG_OK;
}

// smoother with HOST buffers, pipelined across calls: upload(k+1) runs while download(k) is still in flight (PCIe is full
// duplex); tnew_out of call k is complete after the next call that reuses it has returned, or after pamg_sync
int pamg_smooth_host(pamg_handle* h, int solver, int nsweeps, const double* tnew_in, double* tnew_out) {
  if (h && h->is_root && tnew_in && tnew_out) {
    // (the parts rotate their field buffers: V-cycle graphs cached on the root have the old addresses baked in)
    if (!h->vc_graphs.empty()) {
      for (pamg_handle* q : h->parts) { cudaSetDevice(q->device); cudaStreamSynchronize(q->stream); }
      for (auto& g : h->vc_graphs) for (auto e : g.exec) cudaGraphExecDestroy(e);
      h->vc_graphs.clear();
    }
    size_t off = 0;
    for (pamg_handle* q : h->parts) {
      int rc = pamg_smooth_host(q, solver, nsweeps, tnew_in + off, tnew_out + off);
      if (rc) return gfail(h, q, rc);
      off += (size_t)q->lev[0].ndof;
    }
    return PAMG_OK;
  }
  if (!valid_level(h, 1) || !tnew_in || !tnew_out || nsweeps < 1) return PAMG_ERR_ARG;
  CK(cudaSetDevice(h->device));
  LevelDev& L = h->lev[0];
  const size_t bytes = (size_t)L.ndof * sizeof(double);
  if (!h->up_stream) {
    CK(cudaStreamCreateWithFlags(&h->up_stream, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&h->down_stream, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&h->ev_up, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->ev_comp, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->ev_down[0], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->ev_down[1], cudaEventDisableTiming));
  }
  if (!L.spare) CK(cudaMalloc(&L.spare, bytes));
  // Three field buffers rotate: the result of call k is downloaded out of one while call k+1 sweeps between the
  // other two and call k+2 uploads into the first again - so the upload only waits for the download issued two calls ago.
  if (h->pipe_calls >= 2) CK(cudaStreamWaitEvent(h->up_stream, h->ev_down[h->pipe_calls & 1], 0));
  else { CK(cudaEventRecord(h->ev_comp, h->stream)); CK(cudaStreamWaitEvent(h->up_stream, h->ev_comp, 0)); }
  // a dependent loop feeds the result of call k back as the input of call k+1 (or passes one buffer for both): then
  // the upload must also wait for the download that is still writing that host range
  if (h->pipe_calls >= 1 && h->last_out) {
    const char *a0 = (const char*)tnew_in, *a1 = a0 + bytes, *b0 = (const char*)h->last_out, *b1 = b0 + bytes;
    if (a0 < b1 && b0 < a1) CK(cudaStreamWaitEvent(h->up_stream, h->ev_down[(h->pipe_calls - 1) & 1], 0));
  }
  h->last_out = tnew_out;
  CK(cudaMemcpyAsync(L.spare, tnew_in, bytes, cudaMemcpyHostToDevice, h->up_stream));
  CK(cudaEventRecord(h->ev_up, h->up_stream));
  CK(cudaStreamWaitEvent(h->stream, h->ev_up, 0));
  // cached V-cycle graphs have the old buffer addresses baked in
  if (!h->vc_graphs.empty()) { CK(cudaStreamSynchronize(h->stream)); for (auto& g : h->vc_graphs) for (auto e : g.exec) cudaGraphExecDestroy(e); h->vc_graphs.clear(); }
  std::swap(L.T[L.cur], L.spare);   // the uploaded field becomes the iterate; the previous result stays in `spare` for its download
  L.tnew_alias = true;              // tnew_nonlin = tnew = the uploaded field (transport_tri_semi.F90:317)
  field_changed(L);
  int rc = do_smooth(h, 1, solver, nsweeps);
  if (rc) return rc;
  CK(cudaEventRecord(h->ev_comp, h->stream));
  CK(cudaStreamWaitEvent(h->down_stream, h->ev_comp, 0));
  CK(cudaMemcpyAsync(tnew_out, L.T[L.cur], bytes, cudaMemcpyDeviceToHost, h->down_stream));
  CK(cudaEventRecord(h->ev_down[h->pipe_calls & 1], h->down_stream));
  h->pipe_calls++;
  return PAMG_OK;
}

// the reference-facing blocking form: when it returns, tnew_out holds the result and tnew_in may be reused
int pamg_smoother_host(pamg_handle* h, int solver, int nsweeps, const double* tnew_in, double* tnew_out) {
  int rc = pamg_smooth_host(h, solver, nsweeps, tnew_in, tnew_out);
  if (rc) return rc;
  return pamg_sync(h);
}

// ---- distributed ------------------------------------------------------------------------------
int pamg_comm_unique_id(char* id128) {
  if (!id128) return PAMG_ERR_ARG;
  if (!g_nccl.load()) return PAMG_ERR_STATE;
  ncclUniqueId id;
  if (g_nccl.GetUniqueId(&id) != ncclSuccess) return PAMG_ERR_CUDA;
  std::memcpy(id128, id.internal, 128);
  return PAMG_OK;
}

int pamg_comm_init(pamg_handle* h, const char* id128, int nranks, int rank) {
  if (!h || !id128 || nranks < 1 || rank < 0 || rank >= nranks) return PAMG_ERR_ARG;
  if (h->is_root || h->in_group) return fail(h, PAMG_ERR_ARG, "a multi-GPU handle of one process needs no communicator");
  if (!g_nccl.load()) return fail(h, PAMG_ERR_STATE, "libnccl.so.2 could not be loaded");
  CK(cudaSetDevice(h->device));
  // the halo plan uses part numbers as ranks and the coarse levels are agglomerated on part 0 = rank 0
  if (h->lev.empty()) return fail(h, PAMG_ERR_STATE, "pamg_comm_init needs pamg_set_parents_partition first");
  if (nranks != h->plan.nparts || rank != h->plan.my_part)
    return fail(h, PAMG_ERR_ARG, "pamg_comm_init: (nranks, rank) must equal (nparts, my_part) of pamg_set_parents_partition");
  if (h->comm) {     // re-initialisation: graphs with NCCL nodes and the peer mappings go with the old communicator
    CK(cudaStreamSynchronize(h->stream));
    for (auto& g : h->vc_graphs) for (auto e : g.exec) cudaGraphExecDestroy(e);
    h->vc_graphs.clear();
    g_nccl.CommDestroy(h->comm); h->comm = nullptr;
    p2p_close(h);
  }
  ncclUniqueId id;
  std::memcpy(id.internal, id128, 128);
  if (g_nccl.CommInitRank(&h->comm, nranks, id, rank) != ncclSuccess) { h->comm = nullptr; return fail(h, PAMG_ERR_CUDA, "ncclCommInitRank failed"); }
  h->nranks = nranks; h->rank = rank;
  return PAMG_OK;
}

int pamg_halo_peer_count(const pamg_handle* h, int* npeers) {
  if (!h || !npeers) return PAMG_ERR_ARG;
  *npeers = (int)h->plan.peers.size();
  return PAMG_OK;
}

int pamg_halo_peer_info(const pamg_handle* h, int idx, int* peer_part, int* nfaces) {
  if (!h || idx < 0 || idx >= (int)h->plan.peers.size()) return PAMG_ERR_ARG;
  if (peer_part) *peer_part = h->plan.peers[idx].part;
  if (nfaces) *nfaces = h->plan.peers[idx].nfaces;
  return PAMG_OK;
}

// ---- unstructured explicit step ------------------------------------------------------------------
int pamg_set_unstructured(pamg_handle* h, int E, const double* X, const int32_t* neig, const int32_t* fneig) {
  ON_PART0(h);
  if (!h || E < 1 || !X || !neig || !fneig) return PAMG_ERR_ARG;
  CK(cudaSetDevice(h->device));
  std::string e;
  int rc = unstr_setup(h->un, E, X, neig, fneig, h->stream, e);
  if (rc) return fail(h, rc, e);
  return PAMG_OK;
}

int pamg_unstr_set_velocity(pamg_handle* h, const double* u_ele) {
  ON_PART0(h);
  if (!h) return PAMG_ERR_ARG;
  if (h->un.E < 1) return fail(h, PAMG_ERR_STATE, "pamg_set_unstructured has not been called");
  CK(cudaSetDevice(h->device));
  std::string e;
  int rc = unstr_set_velocity(h->un, u_ele, h->nsm, h->stream, e);
  h->launches += u_ele ? 1 : 0;
  if (rc) return fail(h, rc, e);
  return PAMG_OK;
}

int pamg_unstr_upload(pamg_handle* h, const double* tnew) {
  ON_PART0(h);
  if (!h || !tnew || h->un.E < 1) return PAMG_ERR_ARG;
  CK(cudaSetDevice(h->device));
  CK(cudaMemcpyAsync(h->un.T[h->un.cur], tnew, (size_t)h->un.E * 3 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return PAMG_OK;
}

int pamg_unstr_download(pamg_handle* h, double* tnew) {
  ON_PART0(h);
  if (!h || !tnew || h->un.E < 1) return PAMG_ERR_ARG;
  CK(cudaSetDevice(h->device));
  CK(cudaMemcpyAsync(tnew, h->un.T[h->un.cur], (size_t)h->un.E * 3 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return PAMG_OK;
}

int pamg_explicit_step(pamg_handle* h, double dt, double u_x, double u_y, double t_bc, int ntime, int nits,
                       int njac_its, int use_exact_minv, int use_dir) {
  ON_PART0(h);
  if (!h || h->un.E < 1 || ntime < 0 || nits < 1 || njac_its < 0) return PAMG_ERR_ARG;
  CK(cudaSetDevice(h->device));
  std::string e;
  long long nl = 0;
  int rc = unstr_step(h->un, dt, u_x, u_y, t_bc, ntime, nits, njac_its, use_exact_minv, use_dir, h->nsm, h->stream, nl, e);
  h->launches += nl;
  if (rc) return fail(h, rc, e);
  return PAMG_OK;
}

// ---- unstructured implicit operator in block-CSR (unstr_implicit, transport_tri_unstr.F90:214-387) --------
int pamg_implicit_assemble_diffusion(pamg_handle* h, double dt, double u_x, double u_y, double k, int use_dir) {
  ON_PART0(h);
  if (!h || h->un.E < 1 || !(dt > 0.0) || k < 0.0) return PAMG_ERR_ARG;
  if (use_dir < 0) use_dir = h->un_use_dir;   // internal: re-assemble with the previous pairing rule
  h->un_use_dir = use_dir; h->un.with_stab = false;
  CK(cudaSetDevice(h->device));
  std::string e;
  long long nl = 0;
  int rc = implicit_assemble(h->un, dt, u_x, u_y, k, use_dir, h->nsm, h->stream, nl, e);
  h->launches += nl;
  if (rc) return fail(h, rc, e);
  return PAMG_OK;
}

int pamg_implicit_assemble(pamg_handle* h, double dt, double u_x, double u_y, int use_dir) {
  return pamg_implicit_assemble_diffusion(h, dt, u_x, u_y, 0.0, use_dir);
}

int pamg_implicit_get_bsr(pamg_handle* h, double* val, int32_t* col) {
  ON_PART0(h);
  if (!h || h->un.E < 1 || (!val && !col)) return PAMG_ERR_ARG;
  if (!h->un.assembled) return fail(h, PAMG_ERR_STATE, "pamg_implicit_assemble has not been called");
  CK(cudaSetDevice(h->device));
  // the blocks live as 36 + 4 planes on the device: back to the [E][4][9] / [E][4] order of the ABI
  const size_t E = (size_t)h->un.E;
  std::string e;
  int rc = unstr_xfer(h->un, E * 36 * sizeof(double), e);
  if (rc) return fail(h, rc, e);
  const int grid = std::max(1, std::min((h->un.E + TPB - 1) / TPB, h->nsm * 8));
  if (val) {
    k_from_planes<double><<<grid, TPB, 0, h->stream>>>(h->un.bsr_val, h->un.xfer, 36, h->un.E, h->un.ld);
    h->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(val, h->un.xfer, E * 36 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  }
  if (col) {
    int32_t* tmp = reinterpret_cast<int32_t*>(h->un.xfer);
    CK(cudaStreamSynchronize(h->stream));
    k_from_planes<int32_t><<<grid, TPB, 0, h->stream>>>(h->un.bsr_col, tmp, 4, h->un.E, h->un.ld);
    h->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(col, tmp, E * 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
  }
  CK(cudaStreamSynchronize(h->stream));
  return PAMG_OK;
}

int pamg_implicit_apply(pamg_handle* h, const double* x, double* y) {
  ON_PART0(h);
  if (!h || h->un.E < 1 || !x || !y) return PAMG_ERR_ARG;
  if (!h->un.assembled) return fail(h, PAMG_ERR_STATE, "pamg_implicit_assemble has not been called");
  CK(cudaSetDevice(h->device));
  const size_t nb = (size_t)h->un.E * 3 * sizeof(double);
  double* W = h->un.work;
  CK(cudaMemcpyAsync(W, x, nb, cudaMemcpyHostToDevice, h->stream));
  const int grid = stream_grid(k_bsr_spmv, h->un.occ_spmv, h->un.E, h->nsm);
  k_bsr_spmv<<<grid, TPB, 0, h->stream>>>(h->un.bsr_val, h->un.bsr_col, W, nullptr, W + (size_t)h->un.E * 3, h->un.E, h->un.ld, 0);
  h->launches++;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(y, W + (size_t)h->un.E * 3, nb, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return PAMG_OK;
}

int pamg_implicit_set_stab(pamg_handle* h, int with_stab) {
  ON_PART0(h);
  if (!h || h->un.E < 1) return PAMG_ERR_ARG;
  if (!h->un.assembled) return fail(h, PAMG_ERR_STATE, "pamg_implicit_assemble has not been called");
  CK(cudaSetDevice(h->device));
  if (h->un.with_stab && !with_stab)   // back to the plain operator: restore the diagonal blocks and their inverses
    return pamg_implicit_assemble_diffusion(h, h->un.dt, h->un.ux, h->un.uy, h->un.kdiff, -1);
  if (with_stab && !h->un.with_stab) {
    // keep the unstabilised diagonal blocks (the first 9 planes of the matrix): every nonlinear pass adds its own stab to them
    const size_t bytes = h->un.ld * 9 * sizeof(double);
    if (!h->un.diag0) CK(cudaMalloc(&h->un.diag0, bytes));
    CK(cudaMemcpyAsync(h->un.diag0, h->un.bsr_val, bytes, cudaMemcpyDeviceToDevice, h->stream));
  }
  h->un.with_stab = with_stab != 0;
  return PAMG_OK;
}

int pamg_unstr_stab(pamg_handle* h, const double* told, double dt, double u_x, double u_y, double* diff_coe, double* stab) {
  ON_PART0(h);
  if (!h || h->un.E < 1 || !told || !(dt > 0.0) || (!diff_coe && !stab)) return PAMG_ERR_ARG;
  CK(cudaSetDevice(h->device));
  const size_t E = (size_t)h->un.E;
  double *d_old = nullptr, *d_out = nullptr;
  CK(cudaMalloc(&d_old, E * 3 * sizeof(double)));
  if (cudaMalloc(&d_out, E * 12 * sizeof(double)) != cudaSuccess) { cudaFree(d_old); return fail(h, PAMG_ERR_CUDA, "cudaMalloc"); }
  cudaMemcpyAsync(d_old, told, E * 3 * sizeof(double), cudaMemcpyHostToDevice, h->stream);
  StabArgs sa;
  sa.X = h->un.X; sa.tnew = h->un.T[h->un.cur]; sa.told = d_old; sa.diff_coe = d_out + E * 9; sa.stab = d_out; sa.diag0 = nullptr;
  sa.val = nullptr; sa.dinv = nullptr; sa.dt = dt; sa.ux = u_x; sa.uy = u_y; sa.ld = h->un.ld; sa.E = h->un.E; sa.mode = 0;
  sa.U = h->un.U;
  const int grid = std::max(1, std::min((h->un.E + TPB - 1) / TPB, h->nsm * 8));
  if (h->un.U) k_unstr_stab<true><<<grid, TPB, 0, h->stream>>>(sa);
  else k_unstr_stab<false><<<grid, TPB, 0, h->stream>>>(sa);
  h->launches++;
  cudaError_t e1 = cudaGetLastError();
  if (stab) cudaMemcpyAsync(stab, d_out, E * 9 * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
  if (diff_coe) cudaMemcpyAsync(diff_coe, d_out + E * 9, E * 3 * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
  cudaError_t e2 = cudaStreamSynchronize(h->stream);
  cudaFree(d_old); cudaFree(d_out);
  if (e1 != cudaSuccess || e2 != cudaSuccess) return fail(h, PAMG_ERR_CUDA, cudaGetErrorString(e1 != cudaSuccess ? e1 : e2));
  return PAMG_OK;
}

int pamg_implicit_step(pamg_handle* h, int ntime, int nits, double tol, int max_iters, int* iters_total, double* relres) {
  ON_PART0(h);
  if (!h || h->un.E < 1 || ntime < 0 || nits < 1 || !(tol > 0.0) || max_iters < 1) return PAMG_ERR_ARG;
  if (!h->un.assembled) return fail(h, PAMG_ERR_STATE, "pamg_implicit_assemble has not been called");
  CK(cudaSetDevice(h->device));
  std::string e;
  long long nl = 0;
  int rc = implicit_step(h->un, ntime, nits, tol, max_iters, iters_total, relres, h->nsm, h->stream, nl, e, &h->un_host_syncs);
  h->launches += nl;
  if (rc) return fail(h, rc, e);
  return PAMG_OK;
}

// measurement aids for the unstructured kernels: average device time of `reps` block-CSR products y = A x on the work
// vectors, and the number of host synchronisations the Krylov solves have made so far
int pamg_implicit_spmv_time(pamg_handle* h, int reps, float* ms) {
  ON_PART0(h);
  if (!h || h->un.E < 1 || reps < 1 || !ms) return PAMG_ERR_ARG;
  if (!h->un.assembled) return fail(h, PAMG_ERR_STATE, "pamg_implicit_assemble has not been called");
  CK(cudaSetDevice(h->device));
  double* W = h->un.work;
  const size_t n = (size_t)h->un.E * 3;
  const int grid = stream_grid(k_bsr_spmv, h->un.occ_spmv, h->un.E, h->nsm);
  CK(cudaMemcpyAsync(W, h->un.T[h->un.cur], n * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  k_bsr_spmv<<<grid, TPB, 0, h->stream>>>(h->un.bsr_val, h->un.bsr_col, W, nullptr, W + n, h->un.E, h->un.ld, 0);
  CK(cudaEventRecord(h->ev[14], h->stream));
  for (int i = 0; i < reps; ++i) k_bsr_spmv<<<grid, TPB, 0, h->stream>>>(h->un.bsr_val, h->un.bsr_col, W, nullptr, W + n, h->un.E, h->un.ld, 0);
  CK(cudaEventRecord(h->ev[15], h->stream));
  h->launches += reps + 1;
  CK(cudaGetLastError());
  CK(cudaEventSynchronize(h->ev[15]));
  CK(cudaEventElapsedTime(ms, h->ev[14], h->ev[15]));
  *ms /= (float)reps;
  return PAMG_OK;
}

int pamg_implicit_host_syncs(pamg_handle* h, int64_t* n) {
  ON_PART0(h);
  if (!h || !n) return PAMG_ERR_ARG;
  *n = h->un_host_syncs;
  return PAMG_OK;
}

// ---- trans_rec front-end (transport_rect.F90:7) -------------------------------------------------------------
int pamg_trans_rec(pamg_handle* h, double CFL, int no_ele_row, int no_ele_col, double x_length, double y_length, double u_x,
                   double u_y, double time, int nits, int njac_its, int direct_solver, int volume_term, double* x_all,
                   double* tnew, int* ntime) {
  ON_PART0(h);
  if (!h || !tnew || no_ele_row < 1 || no_ele_col < 1 || !(CFL > 0.0) || !(x_length > 0.0) || !(y_length > 0.0) || time < 0.0 ||
      nits < 1 || njac_its < 0)
    return PAMG_ERR_ARG;
  CK(cudaSetDevice(h->device));
  std::string e;
  long long nl = 0;
  int rc = rect_run(CFL, no_ele_row, no_ele_col, x_length, y_length, u_x, u_y, time, nits, njac_its, direct_solver, volume_term,
                    x_all, tnew, ntime, h->nsm, h->stream, nl, e);
  h->launches += nl;
  if (rc) return fail(h, rc, e);
  return PAMG_OK;
}

int pamg_apply_local_minv(pamg_handle* h, int n, int batch, const double* M, const double* rhs, double* x,
                          double* Minv, int32_t* status) {
  ON_PART0(h);
  if (!h || batch < 1 || !M || !(n == 3 || n == 4 || n == 6)) return PAMG_ERR_ARG;
  if (!rhs != !x) return PAMG_ERR_ARG;
  CK(cudaSetDevice(h->device));
  std::string e;
  long long nl = 0;
  int rc = local_minv(n, batch, M, rhs, x, Minv, status, h->nsm, h->stream, nl, e);
  h->launches += nl;
  if (rc) return fail(h, rc, e);
  return PAMG_OK;
}

// ---- output (get_vtu, get_vtk_files.F90:10-140; get_error transport_tri_semi.F90:531-540) ---------------------
namespace {
int output_fields(pamg_handle* h, double* x_all, double* analytical, double* error) {
  LevelDev& L = h->lev[0];
  const size_t n = (size_t)L.nelem;
  double* d = nullptr;
  CK(cudaMalloc(&d, n * 12 * sizeof(double)));
  OutArgs a;
  a.xg = h->xg; a.T = tnew_ptr(L); a.x_all = x_all ? d : nullptr; a.analytical = analytical ? d + n * 6 : nullptr;
  a.error = error ? d + n * 9 : nullptr; a.nelem = L.nelem; a.s = L.s;
  k_output_fields<<<grid_for(h, L.nelem), TPB, 0, h->stream>>>(a);
  h->launches++;
  cudaError_t e = cudaGetLastError();
  if (x_all) cudaMemcpyAsync(x_all, d, n * 6 * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
  if (analytical) cudaMemcpyAsync(analytical, d + n * 6, n * 3 * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
  if (error) cudaMemcpyAsync(error, d + n * 9, n * 3 * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
  cudaError_t e2 = cudaStreamSynchronize(h->stream);
  cudaFree(d);
  if (e != cudaSuccess || e2 != cudaSuccess) return fail(h, PAMG_ERR_CUDA, cudaGetErrorString(e != cudaSuccess ? e : e2));
  return PAMG_OK;
}
}  // namespace

int pamg_output_fields(pamg_handle* h, double* x_all, double* analytical, double* error) {
  if (h && h->is_root) {
    size_t off = 0;
    for (pamg_handle* q : h->parts) {
      int rc = pamg_output_fields(q, x_all ? x_all + off * 6 : nullptr, analytical ? analytical + off * 3 : nullptr,
                                  error ? error + off * 3 : nullptr);
      if (rc) return gfail(h, q, rc);
      off += (size_t)q->lev[0].nelem;
    }
    return PAMG_OK;
  }
  if (!h || h->lev.empty() || (!x_all && !analytical && !error)) return PAMG_ERR_ARG;
  CK(cudaSetDevice(h->device));
  return output_fields(h, x_all, analytical, error);
}

int pamg_write_vtu(pamg_handle* h, const char* path, const char* solve_for, int binary) {
  if (!h || !path || !solve_for) return PAMG_ERR_ARG;
  int64_t nd = 0;
  int rc = pamg_ndof(h, 1, &nd);
  if (rc) return rc;
  const size_t n = (size_t)nd / 3;
  std::vector<double> X(n * 6), T(n * 3), An(n * 3), Er(n * 3);
  if ((rc = pamg_output_fields(h, X.data(), An.data(), Er.data()))) return rc;
  if ((rc = pamg_download_field(h, PAMG_TNEW, 1, T.data()))) return rc;
  FILE* f = fopen(path, binary ? "wb" : "w");
  if (!f) return fail(h, PAMG_ERR_IO, std::string("cannot open ") + path);
  const unsigned long long npts = 3ull * n;
  fprintf(f, "<VTKFile type=\"UnstructuredGrid\" version=\"0.1\" byte_order=\"LittleEndian\"%s>\n", binary ? " header_type=\"UInt64\"" : "");
  fprintf(f, "  <UnstructuredGrid>\n    <Piece NumberOfPoints=\"%llu\" NumberOfCells=\"%llu\">\n", npts, (unsigned long long)n);
  fprintf(f, "      <PointData Scalars=\"scalars\">\n");
  if (!binary) {
    // the reference's layout: one value per line, F12.10 for the unknown, F10.7 for error / analytical, F10.3 coordinates
    const double* arr[3] = {T.data(), Er.data(), An.data()};
    const char* names[3] = {solve_for, "error", "analytical"};
    for (int k = 0; k < 3; ++k) {
      fprintf(f, "        <DataArray type=\"Float32\" Name=\"%s\" Format=\"ascii\">\n", names[k]);
      for (size_t i = 0; i < n * 3; ++i) fprintf(f, k == 0 ? "          %12.10f  \n" : "          %10.7f  \n", arr[k][i]);
      fprintf(f, "        </DataArray>\n");
    }
    fprintf(f, "      </PointData>\n      <Points>\n        <DataArray type=\"Float32\" NumberOfComponents=\"3\" Format=\"ascii\">\n");
    for (size_t i = 0; i < n * 3; ++i) fprintf(f, "          %.3f %.3f %.3f   \n", X[2 * i], X[2 * i + 1], 0.0);
    fprintf(f, "        </DataArray>\n      </Points>\n      <Cells>\n        <DataArray type=\"Int32\" Name=\"connectivity\" Format=\"ascii\">\n");
    for (size_t e = 0; e < n; ++e) fprintf(f, "          %zu %zu %zu\n", 3 * e, 3 * e + 1, 3 * e + 2);
    fprintf(f, "        </DataArray>\n        <DataArray type=\"Int32\" Name=\"offsets\" Format=\"ascii\">\n          ");
    for (size_t e = 1; e <= n; ++e) fprintf(f, e == 1 ? "%zu" : "  %zu", 3 * e);
    fprintf(f, "\n        </DataArray>\n        <DataArray type=\"Int32\" Name=\"types\" Format=\"ascii\">\n          ");
    for (size_t e = 0; e < n; ++e) fprintf(f, e == 0 ? "5" : " 5");                  // cell_type 5 = VTK_TRIANGLE (main.F90)
    fprintf(f, "\n        </DataArray>\n      </Cells>\n    </Piece>\n  </UnstructuredGrid>\n</VTKFile>\n");
  } else {
    // raw appended data, Float64 fields: [UInt64 byte count][payload] per array, offsets relative to the '_' marker
    unsigned long long off = 0;
    const char* names[3] = {solve_for, "error", "analytical"};
    for (int k = 0; k < 3; ++k) {
      fprintf(f, "        <DataArray type=\"Float64\" Name=\"%s\" format=\"appended\" offset=\"%llu\"/>\n", names[k], off);
      off += 8 + npts * 8;
    }
    fprintf(f, "      </PointData>\n      <Points>\n        <DataArray type=\"Float64\" NumberOfComponents=\"3\" format=\"appended\" offset=\"%llu\"/>\n      </Points>\n", off);
    off += 8 + npts * 24;
    fprintf(f, "      <Cells>\n        <DataArray type=\"Int64\" Name=\"connectivity\" format=\"appended\" offset=\"%llu\"/>\n", off);
    off += 8 + npts * 8;
    fprintf(f, "        <DataArray type=\"Int64\" Name=\"offsets\" format=\"appended\" offset=\"%llu\"/>\n", off);
    off += 8 + n * 8;
    fprintf(f, "        <DataArray type=\"UInt8\" Name=\"types\" format=\"appended\" offset=\"%llu\"/>\n", off);
    fprintf(f, "      </Cells>\n    </Piece>\n  </UnstructuredGrid>\n  <AppendedData encoding=\"raw\">\n   _");
    auto block = [&](const void* p, unsigned long long bytes) { fwrite(&bytes, 8, 1, f); fwrite(p, 1, bytes, f); };
    block(T.data(), npts * 8); block(Er.data(), npts * 8); block(An.data(), npts * 8);
    std::vector<double> P3(npts * 3);
    for (size_t i = 0; i < npts; ++i) { P3[3 * i] = X[2 * i]; P3[3 * i + 1] = X[2 * i + 1]; P3[3 * i + 2] = 0.0; }
    block(P3.data(), npts * 24);
    std::vector<long long> conn(npts), offs(n);
    for (size_t i = 0; i < npts; ++i) conn[i] = (long long)i;
    for (size_t e = 0; e < n; ++e) offs[e] = 3ll * (long long)(e + 1);
    block(conn.data(), npts * 8); block(offs.data(), n * 8);
    std::vector<unsigned char> types(n, 5);
    block(types.data(), n);
    fprintf(f, "\n  </AppendedData>\n</VTKFile>\n");
  }
  if (fclose(f) != 0) return fail(h, PAMG_ERR_IO, std::string("write failed: ") + path);
  return PAMG_OK;
}

// ---- timing helpers --------------------------------------------------------------------------------
int pamg_sync(pamg_handle* h) {
  if (!h) return PAMG_ERR_ARG;
  FANOUT(h, q, pamg_sync(q));
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize(h->stream));
  if (h->up_stream) { CK(cudaStreamSynchronize(h->up_stream)); CK(cudaStreamSynchronize(h->down_stream)); h->pipe_calls = 0; h->last_out = nullptr; }
  return p2p_check(h);   // a halo exchange that gave up waiting for a peer raised the error word instead of hanging
}

int pamg_event_record(pamg_handle* h, int slot) {
  if (!h || slot < 0 || slot >= 16) return PAMG_ERR_ARG;
  FANOUT(h, q, pamg_event_record(q, slot));
  CK(cudaSetDevice(h->device));
  CK(cudaEventRecord(h->ev[slot], h->stream));
  return PAMG_OK;
}

int pamg_event_elapsed_ms(pamg_handle* h, int a, int b, float* ms) {
  if (!h || !ms || a < 0 || a >= 16 || b < 0 || b >= 16) return PAMG_ERR_ARG;
  if (h->is_root) {      // the slowest GPU of the group
    *ms = 0.f;
    for (pamg_handle* q : h->parts) { float m = 0.f; int rc = pamg_event_elapsed_ms(q, a, b, &m); if (rc) return gfail(h, q, rc); *ms = std::max(*ms, m); }
    return PAMG_OK;
  }
  CK(cudaSetDevice(h->device));
  CK(cudaEventSynchronize(h->ev[b]));
  CK(cudaEventElapsedTime(ms, h->ev[a], h->ev[b]));
  return PAMG_OK;
}

int pamg_launch_count(const pamg_handle* h, int64_t* n) {
  if (!h || !n) return PAMG_ERR_ARG;
  *n = h->launches;
  for (const pamg_handle* q : h->parts) *n += q->launches;
  return PAMG_OK;
}

int pamg_profile(pamg_handle* h, int on) {
  if (!h) return PAMG_ERR_ARG;
  FANOUT(h, q, pamg_profile(q, on));
  CK(cudaSetDevice(h->device));
  if (on && h->pev.empty()) {
    h->pev.resize(2048);
    for (auto& e : h->pev) CK(cudaEventCreate(&e));
  }
  h->profiling = on != 0;
  h->pev_used = 0;
  return PAMG_OK;
}

int pamg_profile_read(pamg_handle* h, double* total_ms, int* launches) {
  if (!h || !total_ms || !launches) return PAMG_ERR_ARG;
  if (h->is_root) {
    *total_ms = 0.0; *launches = 0;
    for (pamg_handle* q : h->parts) { double t = 0; int l = 0; int rc = pamg_profile_read(q, &t, &l); if (rc) return gfail(h, q, rc); *total_ms += t; *launches += l; }
    return PAMG_OK;
  }
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize(h->stream));
  double tot = 0.0;
  for (int i = 0; i + 1 < h->pev_used; i += 2) {
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, h->pev[i], h->pev[i + 1]));
    tot += ms;
  }
  *total_ms = tot;
  *launches = h->pev_used / 2;
  return PAMG_OK;
}

int pamg_host_alloc(void** p, int64_t bytes) {
  if (!p || bytes <= 0) return PAMG_ERR_ARG;
  return cudaMallocHost(p, (size_t)bytes) == cudaSuccess ? PAMG_OK : PAMG_ERR_CUDA;
}

int pamg_host_free(void* p) { return cudaFreeHost(p) == cudaSuccess ? PAMG_OK : PAMG_ERR_CUDA; }

int pamg_flush_l2(pamg_handle* h) {
  if (!h) return PAMG_ERR_ARG;
  FANOUT(h, q, pamg_flush_l2(q));
  CK(cudaSetDevice(h->device));
  if (!h->scratch) {
    h->scratch_bytes = (size_t)256 << 20;
    CK(cudaMalloc(&h->scratch, h->scratch_bytes));
  }
  k_fill<<<grid_for(h, (long long)(h->scratch_bytes / 8)), TPB, 0, h->stream>>>(h->scratch, (long long)(h->scratch_bytes / 8), 1.0);
  CK(cudaGetLastError());
  return PAMG_OK;
}

}  // extern "C"
