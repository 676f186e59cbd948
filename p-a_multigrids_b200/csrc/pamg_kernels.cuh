// pamg_kernels.cuh -- sm_100a kernels of the semi-structured P1 DG hot path.
//
// All kernels are HBM-bandwidth bound fp64 streaming stencils (SURVEY.md 8(d): 24 B per DOF update for a
// Jacobi sweep / residual evaluation); there is no dense contraction, so no tensor-core work.  Design:
//   * one thread per child triangle, 256 threads per CTA, grid-stride over tiles with the grid sized as a
//     multiple of the SM count;
//   * children of a parent are numbered row by row (Msh2Tri.F90:42-58); rows r and 2^s+1-r together hold
//     exactly 2^(s+1) children, so a flat index maps to (row, position) with shifts only - no integer sqrt
//     and no ragged tiles.  Consecutive threads touch consecutive 24-byte records => coalesced streams;
//   * neighbour values are re-reads of the same stream (adjacent rows) served by L1/L2, halo strips and the
//     20 per-parent coefficients come through the read-only path;
//   * geometry is per parent (ShapFun.F90:1661-1684,1737-1783) and folded on the host into closed-form
//     coefficients, so the kernels carry ~100 flops per child.
#pragma once
#include <cstdint>

namespace pamg {

constexpr int NPC = 88;  // doubles per parent per level: ParentRegs (22, padded to 24) + Folded up (16) + Folded down (16)
                         // + boundary corrections: dpen (3, padded to 4) + omega/D for the 8 face masks (24) + pad (4)
constexpr int PC_FOLD = 24;
constexpr int PC_DPEN = 56;   // penX_f - penI_f : what changes when child face f lies on the parent boundary
constexpr int PC_WB = 60;     // [mask][3] omega / D with mask bit f set when face f+1 is on the parent boundary
// per-parent per-level coefficient slots
enum { PC_CM = 0, PC_K11 = 1, PC_K12, PC_K13, PC_K22, PC_K23, PC_K33, PC_ADV = 7, PC_FL = 10, PC_PENI = 13, PC_W = 16, PC_PENX = 19 };

constexpr int TPB = 256;

enum { MODE_JACOBI = 0, MODE_RESID = 1, MODE_GS = 2, MODE_RICH = 3 };

// ------------------------------------------------------------------------------------------------
// update_overlaps across GPUs without a library collective.  Every GPU STORES its cut-face strips straight into
// a staging buffer of its peers over NVLink (peer pointers from CUDA IPC) in a flagged format: a double travels as
// two 8-byte words {low 32 bits, exchange number} {high 32 bits, exchange number}; an aligned 8-byte store is
// atomic, so the receiver simply polls every word of its own staging buffer until it carries the number of this
// exchange and unpacks it into the strip buffer.  No fence, no separate flag, no credit: the latency is one
// NVLink one-way trip.  The staging buffer has several slots indexed by the exchange number (below), and the
// exchange number lives in device memory so that a captured CUDA graph replays correctly.  Polling has a time-out
// that raises the error word (host-mapped memory, checked at every host synchronisation point) instead of hanging the GPU.
//
// Two kinds of kernels take part.  k_halo sends AND receives exchange n in one launch (after something other than a sweep
// changed the field).  The sweep kernels with a producer warp (XCHG) SEND: as a tile is finished the producer warp stores the
// new values of its children on cut faces straight into the peers' staging buffers as exchange n+1 (the NVLink trip hides
// under the rest of the sweep) and the last CTA advances the exchange number; a small unpack launch (k_halo, HALO_UNPACK) before
// the next sweep moves the values - long arrived - from the staging buffer into the strips.  The staging buffer has FOUR
// slots indexed by the exchange number mod 4: a sending sweep that nobody unpacks (a prolongation came next; the level's
// next visit starts with a k_halo exchange) lets a rank run two exchanges ahead of a peer that still has to unpack - two
// slots would be overwritten, four are safe for every launch sequence the host issues (tests/test_exchange_protocol_model.py).
constexpr int P2P_SLOTS = 4;
constexpr int P2P_MAXP = 16;
enum { P2P_EPOCH = 0, P2P_COUNT = 1, P2P_WORDS = 8 };
struct P2PArgs {
  const double* send;                 // my send slots of this level (contiguous, grouped per peer)
  int send_base;                      // first send slot (in strips) of peer 0, relative to the send-slot space
  double* strips;                     // my strip buffer of this level (receive side)
  uint4* remote[P2P_MAXP];            // each peer's staging buffer (slot 0), already offset to my range there
  long long rstride[P2P_MAXP];        // words per slot of each peer's staging buffer
  long long soff[P2P_MAXP + 1];       // prefix offsets (doubles) of the per-peer send ranges
  long long rbeg[P2P_MAXP];           // first double of the strips I receive from each peer
  long long roff[P2P_MAXP + 1];       // prefix offsets (doubles) of the per-peer receive ranges
  uint4* stage;                       // my staging buffer (slot 0)
  long long stage_words;              // words per slot
  unsigned long long* sync;           // exchange number, block counter
  unsigned long long* err;            // error word (mapped host memory): a poll that timed out raises it instead of hanging
  int npeers;
  unsigned long long timeout_ns;
};

__device__ __forceinline__ unsigned long long p2p_now() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// one double into the staging buffer of peer p (idx = offset in doubles inside my range there)
__device__ __forceinline__ void p2p_put(const P2PArgs& a, unsigned e, int p, long long idx, double val) {
  const unsigned long long v = (unsigned long long)__double_as_longlong(val);
  asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(a.remote[p] + (long long)(e & (P2P_SLOTS - 1)) * a.rstride[p] + idx), "r"((unsigned)v), "r"(e),
               "r"((unsigned)(v >> 32)), "r"(e) : "memory");
}


struct ElemArgs {
  const double* Tin;      // field the sweep reads (may alias Tout for the in-place coloured pass)
  double* Tout;           // Jacobi/GS/Richardson: new iterate; residual: RES
  const double* rhs;
  const double* ovl;      // halo strips [strip][S][3]
  const double* pc;       // [U][NPC]
  const int32_t* strip_of;  // [U*3]
  const int32_t* hmap;      // [U*3]
  const int32_t* nsrc;      // [U*3] strip-free source of the exterior values of (u, side), or nullptr: strips only (HaloPlan::nsrc)
  double* ovl_next;         // strips of the NEXT sweep, written by the producer warp of the window kernels (nullptr: not written)
  const int32_t* dst_strip; // [U*3] strip my boundary children of (u, side) are copied to; -1 = domain boundary
  const int32_t* rev;       // [U*3] slot reversal flag
  int nstrips;              // dst_strip >= nstrips: send slot of a face cut by the GPU partition
  const ulonglong2* xsend;  // (XCHG kernels) [U*3] for a side cut by the GPU partition: .x = start of its range in the peer's staging buffer (slot 0),
                            // .y = words per slot there; .x = 0 otherwise (host table: no dependent look-ups in the producer warp)
  unsigned long long* xsync;  // the level's exchange number / block counter (P2PArgs::sync)
  double* partial;        // residual: [nblocks][3] = sum r^2, max |r|, max r
  double omega;
  double rsign;
  long long nelem;        // U * C
  int s;                  // split of this level
  int colour;             // GS: 0 = down children, 1 = up children
  int partial_off;        // first partial slot this launch writes (residual norms)
};

// flat child index t in [0, 4^s) -> row r (1-based), position ipos (1-based), element id ele (1-based)
__host__ __device__ __forceinline__ void child_from_flat(int t, int s, int& r, int& ipos, int& ele, int& len) {
  const int b = 2 << s;            // 2^(s+1)
  const int S = 1 << s;
  const int p = t >> (s + 1);
  const int q = t & (b - 1);
  const int lenA = b - 1 - 2 * p;  // length of row p+1
  if (q < lenA) { r = p + 1; ipos = q + 1; len = lenA; }
  else { r = S - p; ipos = q - lenA + 1; len = 2 * p + 1; }
  ele = 1 + (r - 1) * (b + 1 - r) + ipos - 1;
}

// neighbour values at the nodes coincident with my face nodes (a,b) of child faces
//   f1:(1,3)  f2:(3,2)  f3:(2,1)      (transport_tri_semi.F90:142-147), and the penalty coefficient of each face
struct FaceIn { double n1a, n1b, n2a, n2b, n3a, n3b, pen1, pen2, pen3; };

// The in-parent neighbours of child c in row r (splitting.F90:749-769): across face 1 the child of the adjacent row (below
// an up child, above a down child), whose index nbr1 returns; across face 2 the left child of an up child and the right
// child of a down child (c -+ 1); across face 3 the other one of the two.
__host__ __device__ __forceinline__ int nbr1(int c, bool up, int r, int b) { return up ? c - b - 2 + 2 * r : c + b - 2 * r; }

// Which of that neighbour's nodes meet mine: across face F = 1, 2, 3 my face nodes (a, b) = (1,3), (3,2), (2,1) meet its
// nodes (3,1), (2,3), (1,2).  ld(n) loads node n (0-based) of the neighbour's record.
template <int F, class Ld>
__device__ __forceinline__ void pair_face(Ld ld, double& va, double& vb) {
  va = ld(F == 1 ? 2 : F == 2 ? 1 : 0);
  vb = ld(F == 1 ? 0 : F == 2 ? 2 : 1);
}
// all three faces, the neighbours' records at v1, v2, v3
__device__ __forceinline__ void pair_nodes(const double* v1, const double* v2, const double* v3, FaceIn& fi) {
  pair_face<1>([&](int n) { return v1[n]; }, fi.n1a, fi.n1b);
  pair_face<2>([&](int n) { return v2[n]; }, fi.n2a, fi.n2b);
  pair_face<3>([&](int n) { return v3[n]; }, fi.n3a, fi.n3b);
}

// Up children on the parent boundary (surf_ele, splitting.F90:434-449): face 1 of a row-1 child lies on parent side 0 at
// strip position ipos/2, face 2 of the first child of a row on side 2 and face 3 of the last child on side 1, both at
// position r-1.  The apex child (len = 1) lies on both sides.
__host__ __device__ __forceinline__ void face_on_side(int f, int r, int ipos, int& side, int& pos) {
  side = f == 1 ? 0 : f == 2 ? 2 : 1;
  pos = f == 1 ? ipos >> 1 : r - 1;
}

// Exterior values of a parent face WITHOUT a halo strip.  update_overlaps (splitting.F90:1255-1391) copies the nodal values
// of the neighbour parent's boundary children from the start-of-sweep field into my strip; a sweep that writes to another
// buffer (Jacobi, Richardson, residual, the one-pass coloured GS) can read those same values straight from that field.
// d = HaloPlan::nsrc (>= 0): nodes | reversal << 4 | (Nside-1) << 5 | neighbour parent << 7; p = my 0-based strip position.
// offset (in doubles, inside the level's field) of the neighbour parent's boundary child that faces my strip position p
__host__ __device__ __forceinline__ size_t nbr_child_offset(int d, int p, int s) {
  const int S = 1 << s, b = 2 << s;
  const int m = (d & 16) ? (S - 1 - p) : p;              // the neighbour's own position along the shared edge
  const int ns = (d >> 5) & 3;
  // its boundary child there (surf_ele, splitting.F90:434-449), 0-based in memory order: side 1 = odd children of row 1,
  // side 3 = first child of row m+1, side 2 = last child of row m+1; row m+1 starts at m (b - m)
  const int e0 = (ns == 0) ? 2 * m : (m * (b - m) + (ns == 1 ? b - 2 - 2 * m : 0));
  return ((((size_t)(d >> 7)) << (2 * s)) + (size_t)e0) * 3;
}
__device__ __forceinline__ void nbr_pair(const double* __restrict__ T, int d, int p, int s, double& va, double& vb) {
  const size_t o = nbr_child_offset(d, p, s);
  va = __ldg(T + o + (d & 3)); vb = __ldg(T + o + ((d >> 2) & 3));
}

// exterior values of parent side mf at 0-based position p: neighbour field (d >= 0) or halo strip (Dirichlet data, faces cut by
// the GPU partition, in-place sweeps)
__device__ __forceinline__ void ext_pair(const ElemArgs& a, int d, int strip, int hm, int p, int S, double& va, double& vb) {
  if (d >= 0) { nbr_pair(a.Tin, d, p, a.s, va, vb); return; }
  const double* e = a.ovl + ((size_t)strip * S + p) * 3;
  va = __ldg(e + (hm & 3)); vb = __ldg(e + (hm >> 2));
}

// same with the per-parent tables still in global memory: mf = gmsh side (0..2), slot0 = 0-based strip position
__device__ __forceinline__ void halo_pair(const ElemArgs& a, int u, int mf, int slot0, int S, double& va, double& vb) {
  const int d = a.nsrc ? __ldg(a.nsrc + u * 3 + mf) : -1;
  ext_pair(a, d, __ldg(a.strip_of + u * 3 + mf), __ldg(a.hmap + u * 3 + mf), slot0, S, va, vb);
}

// exterior values across face f of an up child on the parent boundary; ix(j): entry j of the parent's index table
template <class Ix>
__device__ __forceinline__ void ext_face(const ElemArgs& a, int f, int r, int ipos, int S, Ix ix, double& va, double& vb) {
  int side, pos;
  face_on_side(f, r, ipos, side, pos);
  ext_pair(a, ix(8 + side), ix(side), ix(4 + side), pos, S, va, vb);
}

// a sweep that sent exchange e64 + 1 from its producer warps: the last CTA to finish advances the level's exchange number
__device__ __forceinline__ void p2p_advance(unsigned long long* sync, unsigned long long e64) {
  // (no fence: whoever reads the number next is a later kernel on this stream)
  if (atomicAdd(sync + P2P_COUNT, 1ull) == (unsigned long long)gridDim.x - 1) {
    sync[P2P_COUNT] = 0;
    *(volatile unsigned long long*)(sync + P2P_EPOCH) = e64 + 1;
  }
}

// deterministic two-stage norm reduction: warp shuffle, then one partial per CTA
__device__ __forceinline__ void block_partial(double acc_sum, double acc_abs, double acc_max, double* partial) {
  for (int o = 16; o > 0; o >>= 1) {
    acc_sum += __shfl_xor_sync(0xffffffffu, acc_sum, o);
    acc_abs = fmax(acc_abs, __shfl_xor_sync(0xffffffffu, acc_abs, o));
    acc_max = fmax(acc_max, __shfl_xor_sync(0xffffffffu, acc_max, o));
  }
  __shared__ double sh[3][TPB / 32];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { sh[0][w] = acc_sum; sh[1][w] = acc_abs; sh[2][w] = acc_max; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double s0 = 0, s1 = 0, s2 = 0;
    for (int i = 0; i < TPB / 32; ++i) { s0 += sh[0][i]; s1 = fmax(s1, sh[1][i]); s2 = fmax(s2, sh[2][i]); }
    partial[(size_t)blockIdx.x * 3 + 0] = s0;
    partial[(size_t)blockIdx.x * 3 + 1] = s1;
    partial[(size_t)blockIdx.x * 3 + 2] = s2;
  }
}

// ------------------------------------------------------------------------------------------------
// TMA-tiled kernel (Jacobi / Richardson / residual): the CTA owns TPB children that are CONTIGUOUS IN
// MEMORY, i.e. one 6144-byte span of T, of b and of the output.  One elected thread moves the spans with
// 1-D bulk copies (cp.async.bulk -> UBLKCP) that complete on an mbarrier; every thread then works out of
// shared memory (stride-3 doubles is bank-conflict free) and the result leaves through a bulk store.
// This removes the 24-byte-stride LDG/STG traffic that saturated the L1 wavefront pipe in the direct kernel
// (profiles/r1a_jacobi_simple_ncu_full.txt).  Left/right neighbours come from the tile (+1 child of halo on
// each side); only the vertical neighbour (other row) is a global load.
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "LAB_WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra LAB_DONE_%=;\n"
      "bra LAB_WAIT_%=;\n"
      "LAB_DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_store_1d(void* gdst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(smem_src)),
               "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }

// the contiguous range of tiles [tbeg, tend) this CTA owns
__device__ __forceinline__ void cta_tiles(long long ntiles, long long& tbeg, long long& tend) {
  const long long per = (ntiles + gridDim.x - 1) / gridDim.x;
  tbeg = (long long)blockIdx.x * per;
  tend = min(ntiles, tbeg + per);
}

// one tile (TPB children, 6 KB) of src into slot sl of a shared-memory ring, completing on bar[sl]
constexpr uint32_t TILE_BYTES = 3 * TPB * sizeof(double);
__device__ __forceinline__ void load_tile(double* ring, uint64_t* bar, int sl, const double* src, long long tile) {
  mbar_expect_tx(&bar[sl], TILE_BYTES);
  tma_load_1d(ring + sl * 3 * TPB, src + tile * 3 * TPB, TILE_BYTES, &bar[sl]);
}

// memory-order child index k (0-based) -> row, position.  Row r starts at m(b-m), m = r-1; the float sqrt
// guess is off by at most one, fixed with two predicated corrections (no loops, no divergence).
__host__ __device__ __forceinline__ void child_from_ele0(int k, int s, int& r, int& ipos, int& len) {
  const int b = 2 << s, S = 1 << s;
  int m = (int)(((float)b - sqrtf((float)(b * b - 4 * k))) * 0.5f);
  m = max(0, min(m, S - 1));
  m -= (m * (b - m) > k);
  m += (m + 1 < S) && ((m + 1) * (b - m - 1) <= k);
  m -= (m * (b - m) > k);
  r = m + 1;
  ipos = k - m * (b - m) + 1;
  len = b + 1 - 2 * r;
}

// numbering of "my child of the next tile" from that of the current one: TPB positions further along the rows of the
// parent.  Rows are at least TPB long except near the apex, so the loop usually runs zero or one time; the closed form
// (with its square root) is only needed when the walk enters the next parent.
__host__ __device__ __forceinline__ void child_advance(int s, int b, int k_next, int& r, int& ipos) {
  if (k_next < TPB) { int len; child_from_ele0(k_next, s, r, ipos, len); return; }   // first tile of a parent (uniform)
  ipos += TPB;
  int len = b + 1 - 2 * r;
  while (ipos > len) { ipos -= len; len -= 2; ++r; }
}

constexpr int TMA_T_DOUBLES = 3 * TPB + 8;   // tile + one child of halo on each side, padded to 16-byte spans
constexpr int NSTAGE = 3;                    // tiles in flight per CTA
constexpr size_t TMA_SMEM_BYTES = sizeof(double) * (NSTAGE * (TMA_T_DOUBLES + 3 * TPB) + 2 * 3 * TPB) + 16 * NSTAGE + 64;

// per-parent coefficients held in registers while a CTA walks through the tiles of one parent
struct ParentRegs {
  double cm, k11, k12, k13, k22, k23, k33, adv1, adv2, adv3, fl1, fl2, fl3, pi1, pi2, pi3;
  double w1, w2, w3;   // omega / D for children whose three faces are all inside the parent
  double px1, px2, px3;   // penalty coefficients of faces on the parent boundary
};
static_assert(sizeof(ParentRegs) == 22 * sizeof(double), "ParentRegs must mirror the pc table");

// parent u's coefficients (NPC doubles) and, with sIdx, its index table (strip_of at 0..2, hmap at 4..6, nsrc at 8..10)
// into shared memory, one entry per thread of the CTA
__device__ __forceinline__ void load_parent_cta(const ElemArgs& a, int u, int tid, double* sPC, int* sIdx = nullptr) {
  if (tid < NPC) sPC[tid] = __ldg(a.pc + (size_t)u * NPC + tid);
  else if (sIdx) {
    if (tid < NPC + 3) sIdx[tid - NPC] = __ldg(a.strip_of + u * 3 + (tid - NPC));
    else if (tid < NPC + 6) sIdx[4 + tid - NPC - 3] = __ldg(a.hmap + u * 3 + (tid - NPC - 3));
    else if (tid < NPC + 9) sIdx[8 + tid - NPC - 6] = a.nsrc ? __ldg(a.nsrc + u * 3 + (tid - NPC - 6)) : -1;
  }
}

// An up child on parent faces (face_on_side) takes the exterior values of each such face, ext(f, side, pos, va, vb), and
// its boundary penalty px instead of the in-parent neighbour's values and pi.  Returns the mask of those faces (bit f-1).
template <class Ext>
__device__ __forceinline__ int parent_faces(int r, int ipos, int len, const ParentRegs& P, Ext ext, FaceIn& fi) {
  int bmask = 0, side, pos;
  if (r == 1) { face_on_side(1, r, ipos, side, pos); ext(1, side, pos, fi.n1a, fi.n1b); fi.pen1 = P.px1; bmask |= 1; }
  if (ipos == 1) { face_on_side(2, r, ipos, side, pos); ext(2, side, pos, fi.n2a, fi.n2b); fi.pen2 = P.px2; bmask |= 2; }
  if (ipos == len) { face_on_side(3, r, ipos, side, pos); ext(3, side, pos, fi.n3a, fi.n3b); fi.pen3 = P.px3; bmask |= 4; }
  return bmask;
}
// the same in a window kernel, which fetched the values a tile ahead (h1 across face 1, h2 across the side face); the apex
// child lies on both sides and fetches side 1 now
__device__ __forceinline__ int parent_faces_fetched(const ElemArgs& a, int u, int r, int ipos, int len, int S,
                                                    const ParentRegs& P, double h1a, double h1b, double h2a, double h2b,
                                                    FaceIn& fi) {
  return parent_faces(r, ipos, len, P, [&](int f, int side, int pos, double& va, double& vb) {
    if (f == 1) { va = h1a; vb = h1b; }
    else if (f == 3 && len == 1) halo_pair(a, u, side, pos, S, va, vb);
    else { va = h2a; vb = h2b; }
  }, fi);
}

// Folded operator of a child whose three faces are inside the parent, one set per orientation (up / down).
// Everything elem_apply_regs adds up term by term is linear in (T, neighbour values), so for such children
//   (A x)_i = sum_j a_ij T_j + sum_f c_f [[2,1],[1,2]] (n_fa, n_fb)
// with a_ij = mass + advection + diffusion + penalty + outflow flux and c_f = -pen_f (+ inflow flux).
// The host folds the coefficients once per parent and level (fold_coefficients in pamg_api.cu); the kernels
// spend 27 fp64 operations per child instead of ~70 and need no upwind selects.
struct Folded { double a11, a12, a13, a21, a22, a23, a31, a32, a33, c1, c2, c3, w1, w2, w3, pad; };
static_assert(sizeof(Folded) == 16 * sizeof(double), "Folded layout");

// `mask` has bit f-1 set when child face f lies on the parent boundary (only up children, rare); `ext` points
// at the PC_DPEN / PC_WB part of the parent's table.  The correction is the penalty formula with
// dpen = penX - penI (the neighbour values already come from the halo strip), and omega / D is tabulated
// per mask, so a boundary child costs a handful of extra FMAs instead of the generic path with 3 divisions.
// WITH_R: a sweep also hands out the residual rsign (A x - b) of the iterate it STARTS from (rr[0..2]) - the numbers
// get_residual would compute on the same field, for free
template <int MODE, bool WITH_R = false>
__device__ __forceinline__ void elem_apply_folded(const Folded& F, const double* ext, int mask, double T1, double T2,
                                                  double T3, const FaceIn& fi, double b1, double b2, double b3,
                                                  double rsign, double& o1, double& o2, double& o3, double* rr = nullptr) {
  double ax1 = F.a11 * T1 + F.a12 * T2 + F.a13 * T3;
  double ax2 = F.a21 * T1 + F.a22 * T2 + F.a23 * T3;
  double ax3 = F.a31 * T1 + F.a32 * T2 + F.a33 * T3;
  ax1 += F.c1 * (2.0 * fi.n1a + fi.n1b); ax3 += F.c1 * (fi.n1a + 2.0 * fi.n1b);   // face 1: nodes (1,3)
  ax3 += F.c2 * (2.0 * fi.n2a + fi.n2b); ax2 += F.c2 * (fi.n2a + 2.0 * fi.n2b);   // face 2: nodes (3,2)
  ax2 += F.c3 * (2.0 * fi.n3a + fi.n3b); ax1 += F.c3 * (fi.n3a + 2.0 * fi.n3b);   // face 3: nodes (2,1)
  double w1 = F.w1, w2 = F.w2, w3 = F.w3;
  if (mask) {
    if (mask & 1) { const double dp = ext[0], da = T1 - fi.n1a, db = T3 - fi.n1b; ax1 += dp * (2.0 * da + db); ax3 += dp * (da + 2.0 * db); }
    if (mask & 2) { const double dp = ext[1], da = T3 - fi.n2a, db = T2 - fi.n2b; ax3 += dp * (2.0 * da + db); ax2 += dp * (da + 2.0 * db); }
    if (mask & 4) { const double dp = ext[2], da = T2 - fi.n3a, db = T1 - fi.n3b; ax2 += dp * (2.0 * da + db); ax1 += dp * (da + 2.0 * db); }
    const double* wb = ext + 4 + mask * 3;
    w1 = wb[0]; w2 = wb[1]; w3 = wb[2];
  }
  if (WITH_R) { rr[0] = rsign * (ax1 - b1); rr[1] = rsign * (ax2 - b2); rr[2] = rsign * (ax3 - b3); }
  if (MODE == MODE_RESID) {
    o1 = rsign * (ax1 - b1); o2 = rsign * (ax2 - b2); o3 = rsign * (ax3 - b3);
  } else {
    o1 = T1 + w1 * (b1 - ax1); o2 = T2 + w2 * (b2 - ax2); o3 = T3 + w3 * (b3 - ax3);
  }
}

// One child: A x (get_A_x, transport_tri_semi.F90:412-448, theta = 1), the diagonal (get_diagonal :481-486) and the
// update of the chosen solver, term by term with the parent's coefficients; `interior` children (no face on the parent
// boundary) use the precomputed omega / D.
template <int MODE, bool FACE>
__device__ __forceinline__ void elem_apply_regs(const ParentRegs& P, bool up, bool interior, double T1, double T2,
                                                double T3, const FaceIn& fi, double b1, double b2, double b3,
                                                double omega, double rsign, double& o1, double& o2, double& o3) {
  const double sg = up ? 1.0 : -1.0;
  const double sumT = T1 + T2 + T3;
  const double adv = sg * sumT;
  const double mass1 = P.cm * (T1 + sumT), mass2 = P.cm * (T2 + sumT), mass3 = P.cm * (T3 + sumT);
  const double st1 = P.adv1 * adv, st2 = P.adv2 * adv, st3 = P.adv3 * adv;
  double ax1 = mass1 - st1 + (P.k11 * T1 + P.k12 * T2 + P.k13 * T3);
  double ax2 = mass2 - st2 + (P.k12 * T1 + P.k22 * T2 + P.k23 * T3);
  double ax3 = mass3 - st3 + (P.k13 * T1 + P.k23 * T2 + P.k33 * T3);
  double fx1 = 0.0, fx2 = 0.0, fx3 = 0.0;
  if (FACE) {
    {
      const double da = T1 - fi.n1a, db = T3 - fi.n1b;
      ax1 += fi.pen1 * (2.0 * da + db); ax3 += fi.pen1 * (da + 2.0 * db);
    }
    {
      const double da = T3 - fi.n2a, db = T2 - fi.n2b;
      ax3 += fi.pen2 * (2.0 * da + db); ax2 += fi.pen2 * (da + 2.0 * db);
    }
    {
      const double da = T2 - fi.n3a, db = T1 - fi.n3b;
      ax2 += fi.pen3 * (2.0 * da + db); ax1 += fi.pen3 * (da + 2.0 * db);
    }
    {
      const double fl = sg * P.fl1;
      const bool in = fl < 0.0;
      const double wa = in ? fi.n1a : T1, wb = in ? fi.n1b : T3;
      fx1 += fl * (2.0 * wa + wb); fx3 += fl * (wa + 2.0 * wb);
    }
    {
      const double fl = sg * P.fl2;
      const bool in = fl < 0.0;
      const double wa = in ? fi.n2a : T3, wb = in ? fi.n2b : T2;
      fx3 += fl * (2.0 * wa + wb); fx2 += fl * (wa + 2.0 * wb);
    }
    {
      const double fl = sg * P.fl3;
      const bool in = fl < 0.0;
      const double wa = in ? fi.n3a : T2, wb = in ? fi.n3b : T1;
      fx2 += fl * (2.0 * wa + wb); fx1 += fl * (wa + 2.0 * wb);
    }
    ax1 += fx1; ax2 += fx2; ax3 += fx3;
  }
  if (MODE == MODE_RESID) {
    o1 = rsign * (ax1 - b1); o2 = rsign * (ax2 - b2); o3 = rsign * (ax3 - b3);
  } else if (MODE == MODE_RICH) {
    o1 = T1 + omega * (b1 - (mass1 - st1 + fx1));
    o2 = T2 + omega * (b2 - (mass2 - st2 + fx2));
    o3 = T3 + omega * (b3 - (mass3 - st3 + fx3));
  } else {
    double w1 = P.w1, w2 = P.w2, w3 = P.w3;
    if (!interior) {
      double d1 = 4.0 * P.cm + P.k11, d2 = 4.0 * P.cm + P.k22, d3 = 4.0 * P.cm + P.k33;
      if (FACE) { d1 += 2.0 * (fi.pen1 + fi.pen3); d2 += 2.0 * (fi.pen2 + fi.pen3); d3 += 2.0 * (fi.pen1 + fi.pen2); }
      w1 = omega / d1; w2 = omega / d2; w3 = omega / d3;
    }
    o1 = T1 + w1 * (b1 - ax1);
    o2 = T2 + w2 * (b2 - ax2);
    o3 = T3 + w3 * (b3 - ax3);
  }
}

// Pipelined 1-D TMA tile kernel.  Every CTA owns a CONTIGUOUS range of tiles (so it stays inside one parent
// for hundreds of tiles and the vertical neighbours it needs were touched by itself a moment ago); NSTAGE
// tiles are in flight through a ring of shared-memory stages, each filled by two bulk copies that complete
// on the stage's mbarrier.  The vertical neighbour values of the NEXT tile are fetched one iteration ahead,
// the per-parent coefficients live in shared memory, and results leave through one 6 KB bulk store per tile.
// (A warp-decoupled variant with full/empty mbarriers and per-warp stores measured slower: profiles/README.)
template <int MODE, bool FACE>
__global__ void __launch_bounds__(TPB, 3) k_element_tma(ElemArgs a) {
  extern __shared__ __align__(128) unsigned char dsm[];   // TMA_SMEM_BYTES, carved below
  double (*sT)[TMA_T_DOUBLES] = reinterpret_cast<double (*)[TMA_T_DOUBLES]>(dsm);
  double (*sB)[3 * TPB] = reinterpret_cast<double (*)[3 * TPB]>(dsm + sizeof(double) * NSTAGE * TMA_T_DOUBLES);
  double (*sO)[3 * TPB] = reinterpret_cast<double (*)[3 * TPB]>(dsm + sizeof(double) * NSTAGE * (TMA_T_DOUBLES + 3 * TPB));
  uint64_t* bar = reinterpret_cast<uint64_t*>(dsm + sizeof(double) * (NSTAGE * (TMA_T_DOUBLES + 3 * TPB) + 2 * 3 * TPB));
  __shared__ __align__(16) double sPC[NPC];
  const ParentRegs& P = *reinterpret_cast<const ParentRegs*>(sPC);
  const int s = a.s, twos = 2 * s, b = 2 << s, S = 1 << s;
  const long long Cmask = (1ll << twos) - 1;
  const long long ndof = a.nelem * 3;
  const int tid = threadIdx.x;
  double acc_sum = 0.0, acc_abs = 0.0, acc_max = 0.0;
  if (tid == 0) {
    for (int i = 0; i < NSTAGE; ++i) mbar_init(&bar[i], 1);
    fence_mbar_init();
  }
  __syncthreads();
  const long long ntiles = (a.nelem + TPB - 1) / TPB;
  const long long per = (ntiles + gridDim.x - 1) / gridDim.x;
  const long long tbeg = (long long)blockIdx.x * per, tend = min(ntiles, tbeg + per);

  auto issue = [&](long long tile) {   // tid 0 only
    const int st = (int)((tile - tbeg) % NSTAGE);
    const long long g0 = tile * TPB;
    const int count = (int)min((long long)TPB, a.nelem - g0);
    const long long dlo = (g0 == 0) ? 0 : g0 * 3 - 4;          // even offsets => 16-byte aligned spans
    const long long dhi = min(ndof, (g0 + count) * 3 + 4);
    const uint32_t bt = (uint32_t)((dhi - dlo) * 8), bb = (uint32_t)(count * 24);
    mbar_expect_tx(&bar[st], bt + bb);
    tma_load_1d(sT[st], a.Tin + dlo, bt, &bar[st]);
    tma_load_1d(sB[st], a.rhs + g0 * 3, bb, &bar[st]);
  };
  if (tid == 0)
    for (long long t = tbeg; t < min(tend, tbeg + NSTAGE - 1); ++t) issue(t);

  // per-thread state of the tile being prepared (indices, vertical neighbour values)
  struct Prep { int u, r, ipos, len; bool active, up; double va, vb; };
  auto prepare = [&](long long tile, Prep& p) {
    const long long g = tile * TPB + tid;
    p.active = (tile < tend) && (g < a.nelem);
    p.u = 0; p.r = 1; p.ipos = 1; p.len = 1; p.up = true; p.va = 0.0; p.vb = 0.0;
    if (!p.active) return;
    p.u = (int)(g >> twos);
    const int k = (int)(g & Cmask);
    child_from_ele0(k, s, p.r, p.ipos, p.len);
    p.up = p.ipos & 1;
    if (FACE && !(MODE == MODE_GS && (int)p.up != a.colour)) {
      // the neighbour across face 1 is a global load: fetched a tile ahead; up children of row 1 sit on parent side 0
      // and read the halo strip instead
      const int nb = nbr1(k, p.up, p.r, b);                          // 0-based child index
      if (p.up && p.r == 1) {
        int side, pos;
        face_on_side(1, p.r, p.ipos, side, pos);
        halo_pair(a, p.u, side, pos, S, p.va, p.vb);
      } else {
        const unsigned o1 = ((unsigned)(g - k) + (unsigned)nb) * 3u;         // offsets in doubles fit 32 bits
        pair_face<1>([&](int n) { return __ldg(a.Tin + o1 + n); }, p.va, p.vb);
      }
    }
  };
  Prep cur, nxt;
  prepare(tbeg, cur);
  int u_loaded = -1;
  int obuf = 0;
  for (long long tile = tbeg; tile < tend; ++tile) {
    const int it = (int)(tile - tbeg);
    const int st = it % NSTAGE;
    if (tid == 0 && tile + NSTAGE - 1 < tend) issue(tile + NSTAGE - 1);   // its stage was drained last iteration
    prepare(tile + 1, nxt);
    const long long g0 = tile * TPB;
    const int off0 = (g0 == 0) ? 0 : 4;
    {
      const int u_tile = (int)(g0 >> twos);          // uniform over the CTA (a tile never spans two parents)
      if (u_tile != u_loaded) {
        __syncthreads();
        load_parent_cta(a, u_tile, tid, sPC);
        __syncthreads();
        u_loaded = u_tile;
      }
    }
    mbar_wait(&bar[st], (uint32_t)((it / NSTAGE) & 1));
    double* so = sO[obuf];
    if (cur.active) {
      const double* t = sT[st] + off0 + tid * 3;
      const double T1 = t[0], T2 = t[1], T3 = t[2];
      FaceIn fi;
      bool interior = true, bnd = false;
      int bmask = 0;
      if (FACE) {
        fi.n1a = cur.va; fi.n1b = cur.vb;
        fi.pen1 = P.pi1; fi.pen2 = P.pi2; fi.pen3 = P.pi3;
        // face 2 looks left for an up child and right for a down child, face 3 the other way (splitting.F90:749-769)
        bnd = cur.up && (cur.r == 1 || cur.ipos == 1 || cur.ipos == cur.len);   // child on a parent face (rare)
        const int d = cur.up ? -3 : 3;
        fi.n2a = t[d + 1]; fi.n2b = t[d + 2];
        fi.n3a = t[-d]; fi.n3b = t[-d + 1];
        if (bnd) {
          interior = false;
          if (cur.r == 1) { fi.pen1 = P.px1; bmask |= 1; }
          if (cur.ipos == 1) { halo_pair(a, cur.u, 2, cur.r - 1, S, fi.n2a, fi.n2b); fi.pen2 = P.px2; bmask |= 2; }
          if (cur.ipos == cur.len) { halo_pair(a, cur.u, 1, cur.r - 1, S, fi.n3a, fi.n3b); fi.pen3 = P.px3; bmask |= 4; }
        }
      }
      const double* bb = sB[st] + tid * 3;
      double o1, o2, o3;
      if (MODE == MODE_GS && (int)cur.up != a.colour) {
        o1 = T1; o2 = T2; o3 = T3;      // other colour: written back unchanged (in-place pass)
        bmask = 0;
      } else if (FACE && MODE != MODE_RICH) {
        const Folded& F = *reinterpret_cast<const Folded*>(sPC + PC_FOLD + (cur.up ? 0 : 16));
        elem_apply_folded<MODE>(F, sPC + PC_DPEN, bmask, T1, T2, T3, fi, bb[0], bb[1], bb[2], a.rsign, o1, o2, o3);
      } else {
        elem_apply_regs<MODE, FACE>(P, cur.up, interior, T1, T2, T3, fi, bb[0], bb[1], bb[2], a.omega, a.rsign, o1, o2, o3);
      }
      so[tid * 3] = o1; so[tid * 3 + 1] = o2; so[tid * 3 + 2] = o3;
      if (MODE == MODE_RESID) {
        acc_sum += o1 * o1 + o2 * o2 + o3 * o3;
        acc_abs = fmax(acc_abs, fmax(fabs(o1), fmax(fabs(o2), fabs(o3))));
        acc_max = fmax(acc_max, fmax(o1, fmax(o2, o3)));
      }
    }
    if (tid == 0) tma_store_wait_read();   // the previous tile's store has drained the other staging buffer
    fence_async_smem();
    __syncthreads();                       // sO complete; stage `st` fully consumed
    if (tid == 0) {
      const int count = (int)min((long long)TPB, a.nelem - g0);
      tma_store_1d(a.Tout + g0 * 3, so, (uint32_t)(count * 24));
      tma_store_commit();
    }
    obuf ^= 1;
    cur = nxt;
  }
  if (tid == 0) tma_store_wait_all();
  if (MODE == MODE_RESID) block_partial(acc_sum, acc_abs, acc_max, a.partial + (size_t)3 * a.partial_off);
}

// ------------------------------------------------------------------------------------------------
// Window kernel: like k_element_tma, but the field tiles live in a RING of WIN_NT tiles addressed by the global
// child index (child c sits at sT[(c mod 2048) * 3]), and tile t is only computed once tiles t-2 .. t+2 have
// landed.  A vertical neighbour is at most one row (< 512 children = 2 tiles) away, so ALL six neighbour values
// of a child come from shared memory: no global load on the critical path of an interior child.  The strip
// entries of the few children on parent faces are fetched one tile ahead into registers.  The rhs tile ring is
// also the output staging area: a thread overwrites its own three rhs values with its result and the tile
// leaves through one bulk store from that slot.
constexpr int WIN_NT = 8;                    // field tiles resident (power of two)
constexpr int WIN_NB = 4;                    // rhs / output tiles (power of two)
constexpr int WIN_CH = WIN_NT * TPB;
constexpr size_t WIN_SMEM_BYTES = sizeof(double) * 3 * TPB * (WIN_NT + WIN_NB) + 8 * (WIN_NT + WIN_NB) + 64;
__device__ __forceinline__ void tma_store_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read2() { asm volatile("cp.async.bulk.wait_group.read 2;" ::: "memory"); }

// the in-parent neighbours (nbr1) of the child at ring index cw
__device__ __forceinline__ void ring_nbrs(const double* sT, int cw, bool up, int r, int b, FaceIn& fi) {
  const double* tv = sT + (nbr1(cw, up, r, b) & (WIN_CH - 1)) * 3;
  const double* tl = sT + ((cw - 1) & (WIN_CH - 1)) * 3;
  const double* tr = sT + ((cw + 1) & (WIN_CH - 1)) * 3;
  pair_nodes(tv, up ? tl : tr, up ? tr : tl, fi);
}

template <int MODE, bool FACE>
__global__ void __launch_bounds__(TPB, 3) k_element_win(ElemArgs a) {
  extern __shared__ __align__(128) unsigned char dsm[];   // WIN_SMEM_BYTES
  double* sT = reinterpret_cast<double*>(dsm);
  double* sB = sT + 3 * WIN_CH;
  uint64_t* barT = reinterpret_cast<uint64_t*>(sB + 3 * TPB * WIN_NB);
  uint64_t* barB = barT + WIN_NT;
  __shared__ __align__(16) double sPC[NPC];
  __shared__ int sIdx[12];                                // strip_of[0..2], hmap[4..6], nsrc[8..10] of the loaded parent
  const int s = a.s, twos = 2 * s, b = 2 << s, S = 1 << s;
  const long long Cmask = (1ll << twos) - 1;
  const int tid = threadIdx.x;
  double acc_sum = 0.0, acc_abs = 0.0, acc_max = 0.0;
  if (tid == 0) {
    for (int i = 0; i < WIN_NT + WIN_NB; ++i) mbar_init(&barT[i], 1);
    fence_mbar_init();
  }
  __syncthreads();
  const long long ntiles = a.nelem / TPB;                 // the host only launches this kernel when TPB | 4^s
  long long tbeg, tend;
  cta_tiles(ntiles, tbeg, tend);
  const long long tlo = max(0ll, tbeg - 2), thi = min(ntiles, tend + 2);

  auto issueT = [&](long long tile) { load_tile(sT, barT, (int)(tile & (WIN_NT - 1)), a.Tin, tile); };   // tid 0 only
  auto issueB = [&](long long tile) { load_tile(sB, barB, (int)((tile - tbeg) & (WIN_NB - 1)), a.rhs, tile); };
  if (tid == 0 && tbeg < tend) {
    for (long long t = tlo; t < min(thi, tbeg + 5); ++t) issueT(t);
    for (long long t = tbeg; t < min(tend, tbeg + 2); ++t) issueB(t);
  }

  int u_loaded = -1;
  // numbering of a tile's child and, for children on parent faces, their strip entries
  struct Prep { int r, ipos, len; double h1a, h1b, h2a, h2b; };
  auto prepare = [&](long long tile, Prep& p) {
    p.r = 2; p.ipos = 2; p.len = 3; p.h1a = 0.0; p.h1b = 0.0; p.h2a = 0.0; p.h2b = 0.0;
    if (tile >= tend) return;
    const long long g = tile * TPB + tid;
    child_from_ele0((int)(g & Cmask), s, p.r, p.ipos, p.len);
    if (!FACE || !(p.ipos & 1) || (MODE == MODE_GS && a.colour != 1)) return;
    const bool f1 = p.r == 1, side = p.ipos == 1 || p.ipos == p.len;
    if (f1 | side) {
      const int u = (int)(g >> twos);
      const bool same = u == u_loaded;
      if (f1) {       // child face 1 on parent side 1, position ipos/2
        const int strip = same ? sIdx[0] : __ldg(a.strip_of + u * 3), hm = same ? sIdx[4] : __ldg(a.hmap + u * 3);
        const int d = same ? sIdx[8] : (a.nsrc ? __ldg(a.nsrc + u * 3) : -1);
        ext_pair(a, d, strip, hm, p.ipos >> 1, S, p.h1a, p.h1b);
      }
      if (side) {     // first child of a row: face 2 on parent side 3; last child: face 3 on parent side 2
        const int mf = (p.ipos == 1) ? 2 : 1;
        const int strip = same ? sIdx[mf] : __ldg(a.strip_of + u * 3 + mf), hm = same ? sIdx[4 + mf] : __ldg(a.hmap + u * 3 + mf);
        const int d = same ? sIdx[8 + mf] : (a.nsrc ? __ldg(a.nsrc + u * 3 + mf) : -1);
        ext_pair(a, d, strip, hm, p.r - 1, S, p.h2a, p.h2b);
      }
    }
  };
  Prep cur, nxt;
  prepare(tbeg, cur);
  for (long long tile = tbeg; tile < tend; ++tile) {
    const int it = (int)(tile - tbeg);
    const long long g0 = tile * TPB;
    if (tid == 0) {
      if (tile + 5 < thi) issueT(tile + 5);          // slot of tile-3: last read while tile-1 was computed
      if (tile + 2 < tend) { tma_store_wait_read1(); issueB(tile + 2); }   // slot of tile-2: its store has been read
    }
    {
      const int u_tile = (int)(g0 >> twos);          // uniform over the CTA (a tile never spans two parents)
      if (u_tile != u_loaded) {
        __syncthreads();
        if (tid < NPC) sPC[tid] = __ldg(a.pc + (size_t)u_tile * NPC + tid);
        else if (tid < NPC + 3) sIdx[tid - NPC] = __ldg(a.strip_of + u_tile * 3 + (tid - NPC));
        else if (tid < NPC + 6) sIdx[4 + tid - NPC - 3] = __ldg(a.hmap + u_tile * 3 + (tid - NPC - 3));
        else if (tid < NPC + 9) sIdx[8 + tid - NPC - 6] = a.nsrc ? __ldg(a.nsrc + u_tile * 3 + (tid - NPC - 6)) : -1;
        __syncthreads();
        u_loaded = u_tile;
      }
    }
    prepare(tile + 1, nxt);
    if (it == 0) {
      for (long long tw = tlo; tw <= min(tile + 2, thi - 1); ++tw) mbar_wait(&barT[tw & (WIN_NT - 1)], (uint32_t)(((tw - tlo) >> 3) & 1));
    } else if (tile + 2 < thi) {
      mbar_wait(&barT[(tile + 2) & (WIN_NT - 1)], (uint32_t)(((tile + 2 - tlo) >> 3) & 1));
    }
    mbar_wait(&barB[it & (WIN_NB - 1)], (uint32_t)((it / WIN_NB) & 1));
    double* bb = sB + (it & (WIN_NB - 1)) * 3 * TPB + tid * 3;
    {
      const int cw = (int)(g0 & (WIN_CH - 1)) + tid;           // my slot in the ring (g0 is a multiple of TPB)
      const double* t = sT + cw * 3;
      const double T1 = t[0], T2 = t[1], T3 = t[2];
      const bool up = cur.ipos & 1;
      double o1, o2, o3;
      if (MODE == MODE_GS && (int)up != a.colour) {
        o1 = T1; o2 = T2; o3 = T3;      // other colour: written back unchanged (in-place pass)
      } else {
        FaceIn fi;
        int bmask = 0;
        bool interior = true;
        const ParentRegs& P = *reinterpret_cast<const ParentRegs*>(sPC);
        if (FACE) {
          fi.pen1 = P.pi1; fi.pen2 = P.pi2; fi.pen3 = P.pi3;
          ring_nbrs(sT, cw, up, cur.r, b, fi);
          if (up && (cur.r == 1 || cur.ipos == 1 || cur.ipos == cur.len)) {   // child on a parent face (rare)
            interior = false;
            if (cur.r == 1) { fi.n1a = cur.h1a; fi.n1b = cur.h1b; fi.pen1 = P.px1; bmask |= 1; }
            if (cur.ipos == 1) { fi.n2a = cur.h2a; fi.n2b = cur.h2b; fi.pen2 = P.px2; bmask |= 2; }
            if (cur.ipos == cur.len) {
              if (cur.len == 1) halo_pair(a, (int)(g0 >> twos), 1, cur.r - 1, S, fi.n3a, fi.n3b);   // apex child: both sides
              else { fi.n3a = cur.h2a; fi.n3b = cur.h2b; }
              fi.pen3 = P.px3; bmask |= 4;
            }
          }
        }
        if (FACE && MODE != MODE_RICH) {
          const Folded& F = *reinterpret_cast<const Folded*>(sPC + PC_FOLD + (up ? 0 : 16));
          elem_apply_folded<MODE>(F, sPC + PC_DPEN, bmask, T1, T2, T3, fi, bb[0], bb[1], bb[2], a.rsign, o1, o2, o3);
        } else {
          elem_apply_regs<MODE, FACE>(P, up, interior, T1, T2, T3, fi, bb[0], bb[1], bb[2], a.omega, a.rsign, o1, o2, o3);
        }
      }
      bb[0] = o1; bb[1] = o2; bb[2] = o3;
      if (MODE == MODE_RESID) {
        acc_sum += o1 * o1 + o2 * o2 + o3 * o3;
        acc_abs = fmax(acc_abs, fmax(fabs(o1), fmax(fabs(o2), fabs(o3))));
        acc_max = fmax(acc_max, fmax(o1, fmax(o2, o3)));
      }
    }
    fence_async_smem();
    __syncthreads();                       // result tile complete; every read of the window for this tile is done
    if (tid == 0) {
      tma_store_1d(a.Tout + g0 * 3, sB + (it & (WIN_NB - 1)) * 3 * TPB, TILE_BYTES);
      tma_store_commit();
    }
    cur = nxt;
  }
  if (tid == 0) tma_store_wait_all();
  if (MODE == MODE_RESID) block_partial(acc_sum, acc_abs, acc_max, a.partial + (size_t)3 * a.partial_off);
}

// update_overlaps (splitting.F90:1238-1394) folded into the sweep: once a tile of results sits in shared memory, the
// PRODUCER warp copies the values of its children on parent faces into the neighbour parents' strips of the next sweep
// (double-buffered), so in steady state no halo kernel runs between sweeps and the consumer warps never see the extra
// work.  `tile`: 256 results in shared memory, first child k0 (0-based inside parent u); m0: row of k0 (kept across
// tiles of a parent).  Children on parent side 1 are the odd-ipos children of row 1, on side 3 the first and on side 2 the
// last child of every row (surf_ele, splitting.F90:434-449); the slot is the position or its mirror image (:1256-1391).
struct StripDst { int d0, d1, d2, rv; uint4 *r0, *r1, *r2; };   // destination strips of the parent's three sides (-1: none), reversal
                                                                // bits, and for a side cut by the GPU partition the start of its
                                                                // range in the peer's staging buffer (slot of exchange xe)
__device__ __forceinline__ StripDst strip_dst_load(const ElemArgs& a, int u, int lane, unsigned long long xe = 0) {
  int d = 0, rv = 0;
  unsigned long long r = 0;
  if (lane < 3) {
    d = __ldg(a.dst_strip + u * 3 + lane); rv = __ldg(a.rev + u * 3 + lane) << lane;
    if (xe != 0) {
      const ulonglong2 t = __ldg(a.xsend + u * 3 + lane);
      if (t.x) r = t.x + (xe & (P2P_SLOTS - 1)) * t.y * sizeof(uint4);
    }
  }
  StripDst o;
  o.d0 = __shfl_sync(0xffffffffu, d, 0); o.d1 = __shfl_sync(0xffffffffu, d, 1); o.d2 = __shfl_sync(0xffffffffu, d, 2);
  o.rv = __shfl_sync(0xffffffffu, rv, 0) | __shfl_sync(0xffffffffu, rv, 1) | __shfl_sync(0xffffffffu, rv, 2);
  o.r0 = (uint4*)__shfl_sync(0xffffffffu, r, 0); o.r1 = (uint4*)__shfl_sync(0xffffffffu, r, 1); o.r2 = (uint4*)__shfl_sync(0xffffffffu, r, 2);
  return o;
}

// values for a side cut by the GPU partition (remote base set) go straight into the peer's staging buffer, flagged with the
// exchange number xe
__device__ __forceinline__ void strips_from_tile(const ElemArgs& a, const double* __restrict__ tile, const StripDst& sd, int k0,
                                                 int s, int& m0, int lane, unsigned long long xe = 0) {
  const int S = 1 << s, b = 2 << s;
  const int kend = k0 + TPB;
  auto put = [&](int dst, uint4* rbase, int rvf, int pos, int k) {
    const int slot = rvf ? (S - 1 - pos) : pos;
    const double* t = tile + (k - k0) * 3;
    if (rbase != nullptr) {
      const unsigned e = (unsigned)xe;
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        const unsigned long long v = (unsigned long long)__double_as_longlong(t[i]);
        // (volatile: a weak store may sit in the SM until the kernel ends - measured: the peer's unpack launch times out)
        asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(rbase + slot * 3 + i), "r"((unsigned)v), "r"(e), "r"((unsigned)(v >> 32)), "r"(e) : "memory");
      }
      return;
    }
    double* e = a.ovl_next + ((size_t)dst * S + slot) * 3;
    e[0] = t[0]; e[1] = t[1]; e[2] = t[2];
  };
  if (sd.d0 >= 0 && k0 < b - 1) {                    // row 1: children k = 0, 2, 4, .. b-2 at positions k/2
    const int e1 = min(kend, b - 1);
    for (int k = k0 + 2 * lane; k < e1; k += 64) put(sd.d0, sd.r0, sd.rv & 1, k >> 1, k);
  }
  while ((m0 + 1) * (b - m0 - 1) <= k0) ++m0;        // row (0-based) that holds child k0
  if (sd.d1 >= 0 || sd.d2 >= 0) {
    for (int m = m0 + lane; m < S; m += 32) {
      const int first = m * (b - m);
      if (first >= kend) break;
      const int last = (m + 1) * (b - m - 1) - 1;
      if (sd.d2 >= 0 && first >= k0) put(sd.d2, sd.r2, sd.rv & 4, m, first);
      if (sd.d1 >= 0 && last < kend) put(sd.d1, sd.r1, sd.rv & 2, m, last);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Window kernel with a PRODUCER WARP.  Same ring and arithmetic as k_element_win, but the ninth warp of the CTA does
// all the copy-engine work (bulk loads, bulk stores, per-parent coefficient reloads) and the eight consumer warps
// never wait for each other: after writing its results a consumer only ARRIVES on a named barrier (bar.arrive) and
// goes on to the next tile as soon as that tile's data has landed; the producer is the one that waits (bar.sync)
// before it stores the tile and refills the freed ring slots.  Per-parent coefficients are double-buffered by the
// parity of the parent and published through the mbarrier of the first rhs tile of the parent, so the kernel needs
// at least 8 tiles per parent (n_split >= 6 on the level); smaller levels use k_element_win.
constexpr int WIN2_THREADS = TPB + 32;
__device__ __forceinline__ void named_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void named_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }

// XCHG: the producer warp sends the new values of the children on cut faces to the peer GPUs (see P2PArgs).
// NORM (Jacobi with face terms): the sweep also reduces the norms of the residual of the iterate it starts from, exactly as
// the residual kernel would (same tiles per CTA, same order: the same partial sums) - the V-cycle takes its convergence
// norm out of the first pre-smoothing sweep of the next cycle instead of a residual evaluation of its own.
template <int MODE, bool FACE, bool XCHG = false, bool NORM = false>
__global__ void __launch_bounds__(WIN2_THREADS, 3) k_element_win2(ElemArgs a) {
  extern __shared__ __align__(128) unsigned char dsm[];   // WIN_SMEM_BYTES
  double* sT = reinterpret_cast<double*>(dsm);
  double* sB = sT + 3 * WIN_CH;
  uint64_t* barT = reinterpret_cast<uint64_t*>(sB + 3 * TPB * WIN_NB);
  uint64_t* barB = barT + WIN_NT;
  __shared__ __align__(16) double sPC2[2][NPC];
  __shared__ int sIdx2[2][12];
  __shared__ double shp[3][TPB / 32];
  const int s = a.s, twos = 2 * s, b = 2 << s, S = 1 << s;
  const long long Cmask = (1ll << twos) - 1;
  const int tid = threadIdx.x;
  double acc_sum = 0.0, acc_abs = 0.0, acc_max = 0.0;
  if (tid == 0) {
    for (int i = 0; i < WIN_NT + WIN_NB; ++i) mbar_init(&barT[i], 1);
    fence_mbar_init();
  }
  __syncthreads();
  const long long ntiles = a.nelem / TPB;
  long long tbeg, tend;
  cta_tiles(ntiles, tbeg, tend);
  const long long tlo = max(0ll, tbeg - 2), thi = min(ntiles, tend + 2);

  if (tid >= TPB) {
    // ------------------------------------------------------------------ producer warp
    const int lane = tid - TPB;
    int u_loaded = -1;
    // exchange number of the cut-face values this sweep READS (the sweep or k_halo before it sent them); it sends e64 + 1
    unsigned long long e64 = 0;
    if (XCHG) e64 = *(volatile unsigned long long*)(a.xsync + P2P_EPOCH);
    auto issueT = [&](long long tile) { load_tile(sT, barT, (int)(tile & (WIN_NT - 1)), a.Tin, tile); };   // lane 0
    auto issueB = [&](long long tile) {   // whole warp: a new parent's coefficients go out with its first rhs tile
      const int u = (int)((tile * TPB) >> twos);
      if (u != u_loaded) {
        for (int i = lane; i < NPC; i += 32) sPC2[u & 1][i] = __ldg(a.pc + (size_t)u * NPC + i);
        if (lane < 3) {
          sIdx2[u & 1][lane] = __ldg(a.strip_of + u * 3 + lane); sIdx2[u & 1][4 + lane] = __ldg(a.hmap + u * 3 + lane);
          sIdx2[u & 1][8 + lane] = a.nsrc ? __ldg(a.nsrc + u * 3 + lane) : -1;
        }
        u_loaded = u;
        __syncwarp();
      }
      // (the expect_tx releases the coefficient writes above to whoever waits on the tile)
      if (lane == 0) load_tile(sB, barB, (int)((tile - tbeg) & (WIN_NB - 1)), a.rhs, tile);
    };
    if (tbeg < tend) {
      if (lane == 0) for (long long t = tlo; t < min(thi, tbeg + 6); ++t) issueT(t);
      for (long long t = tbeg; t < min(tend, tbeg + 3); ++t) issueB(t);
    }
    int m0 = 0, u_m0 = -1;
    StripDst sd = {-1, -1, -1, 0, nullptr, nullptr, nullptr};
    for (long long p = tbeg; p < tend; ++p) {
      const int it = (int)(p - tbeg);
      named_sync(1 + (it & 3), WIN2_THREADS);            // every consumer warp has written tile p
      if (lane == 0) {
        tma_store_1d(a.Tout + p * 3 * TPB, sB + (it & (WIN_NB - 1)) * 3 * TPB, TILE_BYTES);
        tma_store_commit();
        if (p + 6 < thi) issueT(p + 6);                  // ring slot of tile p-2: no consumer is behind tile p+1
        if (p + 3 < tend) tma_store_wait_read1();        // rhs slot of tile p-1: its store has been read
      }
      __syncwarp();
      if (p + 3 < tend) issueB(p + 3);
      if (MODE != MODE_RESID && a.ovl_next) {            // halo strips of the next sweep from the finished tile
        const int u = (int)((p * TPB) >> twos);
        if (u != u_m0) { m0 = 0; u_m0 = u; sd = strip_dst_load(a, u, lane, XCHG ? e64 + 1 : 0); }      // once per parent
        strips_from_tile(a, sB + (it & (WIN_NB - 1)) * 3 * TPB, sd, (int)((p * TPB) & Cmask), s, m0, lane, XCHG ? e64 + 1 : 0);
      }
    }
    if (XCHG && MODE != MODE_RESID && lane == 0) p2p_advance(a.xsync, e64);
    if (lane == 0) tma_store_wait_all();
  } else {
    // ------------------------------------------------------------------ consumer warps
    // (per-tile index arithmetic in 32-bit: this branch cannot use the uniform datapath)
    const int tbegi = (int)tbeg, tendi = (int)tend, tloi = (int)tlo, thii = (int)thi;
    const int pshift = twos - 8;                          // tiles per parent = 2^pshift (TPB = 2^8)
    const unsigned kmask = (unsigned)Cmask;
    struct Prep { int r, ipos, len; double h1a, h1b, h2a, h2b; };
    // p.r / p.ipos come in as the numbering of my child of the PREVIOUS tile and leave as that of `tile`
    auto prepare = [&](int tile, int u_cur, bool first, Prep& p) {
      p.h1a = 0.0; p.h1b = 0.0; p.h2a = 0.0; p.h2b = 0.0;
      if (tile >= tendi) return;
      const int kk = (int)((((unsigned)tile << 8) + (unsigned)tid) & kmask);
      if (first) child_from_ele0(kk, s, p.r, p.ipos, p.len);
      else child_advance(s, b, kk, p.r, p.ipos);
      p.len = b + 1 - 2 * p.r;
      if (!FACE || !(p.ipos & 1)) return;
      const bool f1 = p.r == 1, side = p.ipos == 1 || p.ipos == p.len;
      if (f1 | side) {
        const int u = tile >> pshift;
        const bool same = u == u_cur;                    // the coefficients of u_cur have been acquired by this thread
        const int* ix = sIdx2[u & 1];
        if (f1) {
          const int strip = same ? ix[0] : __ldg(a.strip_of + u * 3), hm = same ? ix[4] : __ldg(a.hmap + u * 3);
          const int d = same ? ix[8] : (a.nsrc ? __ldg(a.nsrc + u * 3) : -1);
          ext_pair(a, d, strip, hm, p.ipos >> 1, S, p.h1a, p.h1b);
        }
        if (side) {
          const int mf = (p.ipos == 1) ? 2 : 1;
          const int strip = same ? ix[mf] : __ldg(a.strip_of + u * 3 + mf), hm = same ? ix[4 + mf] : __ldg(a.hmap + u * 3 + mf);
          const int d = same ? ix[8 + mf] : (a.nsrc ? __ldg(a.nsrc + u * 3 + mf) : -1);
          ext_pair(a, d, strip, hm, p.r - 1, S, p.h2a, p.h2b);
        }
      }
    };
    Prep cur, nxt;
    cur.r = 2; cur.ipos = 2; cur.len = 3;
    prepare(tbegi, -1, true, cur);
    for (int tile = tbegi; tile < tendi; ++tile) {
      const int it = tile - tbegi;
      const int u_tile = tile >> pshift;
      if (it == 0) {
        for (int tw = tloi; tw <= min(tile + 2, thii - 1); ++tw) mbar_wait(&barT[tw & (WIN_NT - 1)], (uint32_t)(((tw - tloi) >> 3) & 1));
      } else if (tile + 2 < thii) {
        mbar_wait(&barT[(tile + 2) & (WIN_NT - 1)], (uint32_t)(((tile + 2 - tloi) >> 3) & 1));
      }
      mbar_wait(&barB[it & (WIN_NB - 1)], (uint32_t)((it / WIN_NB) & 1));     // also acquires the coefficients of u_tile
      nxt.r = cur.r; nxt.ipos = cur.ipos;
      prepare(tile + 1, u_tile, false, nxt);
      const double* sPC = sPC2[u_tile & 1];
      double* bb = sB + (it & (WIN_NB - 1)) * (3 * TPB) + tid * 3;
      {
        const int cw = ((tile & (WIN_NT - 1)) << 8) + tid;
        const double* t = sT + cw * 3;
        const double T1 = t[0], T2 = t[1], T3 = t[2];
        const bool up = cur.ipos & 1;
        double o1, o2, o3;
        FaceIn fi;
        int bmask = 0;
        bool interior = true;
        const ParentRegs& P = *reinterpret_cast<const ParentRegs*>(sPC);
        if (FACE) {
          fi.pen1 = P.pi1; fi.pen2 = P.pi2; fi.pen3 = P.pi3;
          ring_nbrs(sT, cw, up, cur.r, b, fi);
          if (up && (cur.r == 1 || cur.ipos == 1 || cur.ipos == cur.len)) {
            interior = false;
            if (cur.r == 1) { fi.n1a = cur.h1a; fi.n1b = cur.h1b; fi.pen1 = P.px1; bmask |= 1; }
            if (cur.ipos == 1) { fi.n2a = cur.h2a; fi.n2b = cur.h2b; fi.pen2 = P.px2; bmask |= 2; }
            if (cur.ipos == cur.len) {
              if (cur.len == 1) halo_pair(a, u_tile, 1, cur.r - 1, S, fi.n3a, fi.n3b);
              else { fi.n3a = cur.h2a; fi.n3b = cur.h2b; }
              fi.pen3 = P.px3; bmask |= 4;
            }
          }
        }
        if (FACE && MODE != MODE_RICH) {
          const Folded& F = *reinterpret_cast<const Folded*>(sPC + PC_FOLD + (up ? 0 : 16));
          if (NORM) {
            double rr[3];
            elem_apply_folded<MODE, true>(F, sPC + PC_DPEN, bmask, T1, T2, T3, fi, bb[0], bb[1], bb[2], a.rsign, o1, o2, o3, rr);
            acc_sum += rr[0] * rr[0] + rr[1] * rr[1] + rr[2] * rr[2];
            acc_abs = fmax(acc_abs, fmax(fabs(rr[0]), fmax(fabs(rr[1]), fabs(rr[2]))));
            acc_max = fmax(acc_max, fmax(rr[0], fmax(rr[1], rr[2])));
          } else {
            elem_apply_folded<MODE>(F, sPC + PC_DPEN, bmask, T1, T2, T3, fi, bb[0], bb[1], bb[2], a.rsign, o1, o2, o3);
          }
        } else {
          elem_apply_regs<MODE, FACE>(P, up, interior, T1, T2, T3, fi, bb[0], bb[1], bb[2], a.omega, a.rsign, o1, o2, o3);
        }
        bb[0] = o1; bb[1] = o2; bb[2] = o3;
        if (MODE == MODE_RESID) {
          acc_sum += o1 * o1 + o2 * o2 + o3 * o3;
          acc_abs = fmax(acc_abs, fmax(fabs(o1), fmax(fabs(o2), fabs(o3))));
          acc_max = fmax(acc_max, fmax(o1, fmax(o2, o3)));
        }
      }
      fence_async_smem();
      named_arrive(1 + (it & 3), WIN2_THREADS);          // no waiting: on to the next tile
      cur = nxt;
    }
  }
  if (MODE == MODE_RESID || NORM) {
    if (tid < TPB) {
      for (int o = 16; o > 0; o >>= 1) {
        acc_sum += __shfl_xor_sync(0xffffffffu, acc_sum, o);
        acc_abs = fmax(acc_abs, __shfl_xor_sync(0xffffffffu, acc_abs, o));
        acc_max = fmax(acc_max, __shfl_xor_sync(0xffffffffu, acc_max, o));
      }
      if ((tid & 31) == 0) { shp[0][tid >> 5] = acc_sum; shp[1][tid >> 5] = acc_abs; shp[2][tid >> 5] = acc_max; }
    }
    __syncthreads();
    if (tid == 0) {
      double s0 = 0, s1 = 0, s2 = 0;
      for (int i = 0; i < TPB / 32; ++i) { s0 += shp[0][i]; s1 = fmax(s1, shp[1][i]); s2 = fmax(s2, shp[2][i]); }
      double* partial = a.partial + (size_t)3 * a.partial_off;
      partial[(size_t)blockIdx.x * 3 + 0] = s0; partial[(size_t)blockIdx.x * 3 + 1] = s1; partial[(size_t)blockIdx.x * 3 + 2] = s2;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Coloured Gauss-Seidel sweep in ONE pass over memory (out of place: Tin -> Tout).  Same ring as k_element_win.
// In iteration t every thread first relaxes its child of tile t+2 if that is a DOWN child (reads the old up
// values in tiles t+1 .. t+4, writes the new down values into the ring), then its child of tile t if that is an
// UP child (reads the new down values in tiles t-2 .. t+1, which earlier iterations produced, writes the new up
// values into the ring); the two updates touch disjoint data, so one CTA barrier per tile suffices.  Tile t is
// then final and leaves through a bulk store straight from the ring.  This is the reference's sweep in
// two-colour order (all down children, then all up children, values across parent faces lagged through the
// halo strips) with 24 B/DOF of traffic instead of 48.  A CTA relaxes the down children of the two tiles before
// and the one tile after its own range redundantly (in shared memory only) so that CTAs stay independent.
constexpr size_t GSW_SMEM_BYTES = WIN_SMEM_BYTES;

__global__ void __launch_bounds__(TPB, 3) k_gs_win(ElemArgs a) {
  extern __shared__ __align__(128) unsigned char dsm[];
  double* sT = reinterpret_cast<double*>(dsm);
  double* sB = sT + 3 * WIN_CH;
  uint64_t* barT = reinterpret_cast<uint64_t*>(sB + 3 * TPB * WIN_NB);
  uint64_t* barB = barT + WIN_NT;
  __shared__ __align__(16) double sPC[NPC];       // parent of the tile whose up children are relaxed
  __shared__ __align__(16) double sPD[16];        // folded "down" operator of the parent of tile t+2
  __shared__ int sIdx[12];
  const int s = a.s, twos = 2 * s, b = 2 << s, S = 1 << s;
  const long long Cmask = (1ll << twos) - 1;
  const int tid = threadIdx.x;
  if (tid == 0) {
    for (int i = 0; i < WIN_NT + WIN_NB; ++i) mbar_init(&barT[i], 1);
    fence_mbar_init();
  }
  __syncthreads();
  const long long ntiles = a.nelem / TPB;
  long long tbeg, tend;
  cta_tiles(ntiles, tbeg, tend);
  if (tbeg >= tend) return;
  const long long dlo = max(0ll, tbeg - 2), dhi = min(ntiles - 1, tend);       // tiles whose down children I relax
  const long long tlo = max(0ll, dlo - 1), thi = min(ntiles, dhi + 3);         // field tiles I load: [tlo, thi)
  const long long t0 = dlo - 2;                                                // first iteration

  auto issueT = [&](long long tile) { load_tile(sT, barT, (int)(tile & (WIN_NT - 1)), a.Tin, tile); };
  auto issueB = [&](long long tile) { load_tile(sB, barB, (int)((tile - dlo) & (WIN_NB - 1)), a.rhs, tile); };
  auto waitT = [&](long long tile) { mbar_wait(&barT[tile & (WIN_NT - 1)], (uint32_t)(((tile - tlo) >> 3) & 1)); };
  auto waitB = [&](long long tile) { mbar_wait(&barB[(tile - dlo) & (WIN_NB - 1)], (uint32_t)(((tile - dlo) >> 2) & 1)); };
  if (tid == 0) {
    for (long long t = tlo; t < min(thi, t0 + 6); ++t) issueT(t);        // iteration t0 needs tiles <= t0 + 4; one ahead
    for (long long t = dlo; t <= min(dhi, dlo + 3); ++t) issueB(t);      // all four rhs slots
  }

  int u_up = -1, u_dn = -1;
  struct Prep { int r, ipos, len; double h1a, h1b, h2a, h2b; };
  auto prepare = [&](long long tile, Prep& p) {    // my child of `tile` as an up child: numbering + strip entries
    p.r = 2; p.ipos = 2; p.len = 3; p.h1a = 0.0; p.h1b = 0.0; p.h2a = 0.0; p.h2b = 0.0;
    if (tile < tbeg || tile >= tend) return;
    const long long g = tile * TPB + tid;
    child_from_ele0((int)(g & Cmask), s, p.r, p.ipos, p.len);
    if (!(p.ipos & 1)) return;
    const bool f1 = p.r == 1, side = p.ipos == 1 || p.ipos == p.len;
    if (f1 | side) {
      const int u = (int)(g >> twos);
      const bool same = u == u_up;
      if (f1) {
        const int strip = same ? sIdx[0] : __ldg(a.strip_of + u * 3), hm = same ? sIdx[4] : __ldg(a.hmap + u * 3);
        const int d = same ? sIdx[8] : (a.nsrc ? __ldg(a.nsrc + u * 3) : -1);
        ext_pair(a, d, strip, hm, p.ipos >> 1, S, p.h1a, p.h1b);
      }
      if (side) {
        const int mf = (p.ipos == 1) ? 2 : 1;
        const int strip = same ? sIdx[mf] : __ldg(a.strip_of + u * 3 + mf), hm = same ? sIdx[4 + mf] : __ldg(a.hmap + u * 3 + mf);
        const int d = same ? sIdx[8 + mf] : (a.nsrc ? __ldg(a.nsrc + u * 3 + mf) : -1);
        ext_pair(a, d, strip, hm, p.r - 1, S, p.h2a, p.h2b);
      }
    }
  };
  Prep cur, nxt;
  prepare(t0, cur);
  for (long long tile = t0; tile < tend; ++tile) {
    const long long td = tile + 2;                       // tile whose down children are relaxed now
    const bool doD = td >= dlo && td <= dhi, doU = tile >= tbeg;
    if (tid == 0 && tile > t0) {
      // field slot of tile-3: last read while tile-1 was relaxed; its store (three groups ago) has been read
      if (tile + 5 < thi) { tma_store_wait_read2(); issueT(tile + 5); }
      // rhs slot of tile-1 (= td-3): consumed by the up children of tile-1
      if (td + 1 >= dlo + 4 && td + 1 <= dhi) issueB(td + 1);
    }
    {
      const int ud = doD ? (int)((td * TPB) >> twos) : u_dn;
      const int uu = doU ? (int)((tile * TPB) >> twos) : u_up;
      if (ud != u_dn || uu != u_up) {                    // uniform over the CTA
        __syncthreads();
        if (uu != u_up) load_parent_cta(a, uu, tid, sPC, sIdx);
        if (ud != u_dn && tid >= 128 && tid < 144) sPD[tid - 128] = __ldg(a.pc + (size_t)ud * NPC + PC_FOLD + 16 + (tid - 128));
        __syncthreads();
        u_dn = ud; u_up = uu;
      }
    }
    prepare(tile + 1, nxt);
    if (tile == t0) {
      for (long long tw = tlo; tw < min(thi, tile + 5); ++tw) waitT(tw);
    } else if (tile + 4 < thi) {
      waitT(tile + 4);
    }
    if (doD) {
      waitB(td);
      const long long g = td * TPB + tid;
      int r, ipos, len;
      child_from_ele0((int)(g & Cmask), s, r, ipos, len);
      if (!(ipos & 1)) {                                  // down child: all three faces inside the parent
        const int cw = (int)((td * TPB) & (WIN_CH - 1)) + tid;
        double* t = sT + cw * 3;
        const double T1 = t[0], T2 = t[1], T3 = t[2];
        FaceIn fi;
        ring_nbrs(sT, cw, false, r, b, fi);
        const double* bb = sB + ((td - dlo) & (WIN_NB - 1)) * 3 * TPB + tid * 3;
        const Folded& F = *reinterpret_cast<const Folded*>(sPD);
        double o1, o2, o3;
        elem_apply_folded<MODE_GS>(F, sPD, 0, T1, T2, T3, fi, bb[0], bb[1], bb[2], a.rsign, o1, o2, o3);
        t[0] = o1; t[1] = o2; t[2] = o3;
      }
    }
    if (doU) {
      // rhs of `tile` landed when its down children were relaxed two iterations ago
      if (cur.ipos & 1) {
        const int cw = (int)((tile * TPB) & (WIN_CH - 1)) + tid;
        double* t = sT + cw * 3;
        const double T1 = t[0], T2 = t[1], T3 = t[2];
        FaceIn fi;
        int bmask = 0;
        ring_nbrs(sT, cw, true, cur.r, b, fi);
        if (cur.r == 1 || cur.ipos == 1 || cur.ipos == cur.len)               // child on a parent face (rare)
          bmask = parent_faces_fetched(a, (int)((tile * TPB) >> twos), cur.r, cur.ipos, cur.len, S,
                                       *reinterpret_cast<const ParentRegs*>(sPC), cur.h1a, cur.h1b, cur.h2a, cur.h2b, fi);
        const double* bb = sB + ((tile - dlo) & (WIN_NB - 1)) * 3 * TPB + tid * 3;
        const Folded& F = *reinterpret_cast<const Folded*>(sPC + PC_FOLD);
        double o1, o2, o3;
        elem_apply_folded<MODE_GS>(F, sPC + PC_DPEN, bmask, T1, T2, T3, fi, bb[0], bb[1], bb[2], a.rsign, o1, o2, o3);
        t[0] = o1; t[1] = o2; t[2] = o3;
      }
    }
    fence_async_smem();
    __syncthreads();
    if (tid == 0 && doU) {
      tma_store_1d(a.Tout + tile * 3 * TPB, sT + (tile & (WIN_NT - 1)) * 3 * TPB, TILE_BYTES);
      tma_store_commit();
    }
    cur = nxt;
  }
  if (tid == 0) tma_store_wait_all();
}

// ------------------------------------------------------------------------------------------------
// One-pass coloured Gauss-Seidel with a producer warp (see k_gs_win for the algorithm, k_element_win2 for the roles).
// The two colours depend on each other - the up children of tile t read the down value at the first child of tile t+1, and
// the down phase of tile t+1 reads up values of tile t that the up phase overwrites - so four consumer warps relax the down
// children of tile t+1 and arrive on an mbarrier; the other four wait on it before they relax the up children of tile t.
// The down warps never wait for the up warps (only for data), so they run ahead by up to the depth of the ring.
__device__ __forceinline__ void mbar_arrive_cta(uint64_t* bar) {
  asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

template <bool XCHG>
__global__ void __launch_bounds__(WIN2_THREADS, 3) k_gs_win2(ElemArgs a) {
  extern __shared__ __align__(128) unsigned char dsm[];
  double* sT = reinterpret_cast<double*>(dsm);
  double* sB = sT + 3 * WIN_CH;
  uint64_t* barT = reinterpret_cast<uint64_t*>(sB + 3 * TPB * WIN_NB);
  uint64_t* barB = barT + WIN_NT;
  __shared__ __align__(16) double sPC2[2][NPC];
  __shared__ int sIdx2[2][12];
  __shared__ __align__(8) uint64_t doneD[4];
  const int s = a.s, twos = 2 * s, b = 2 << s, S = 1 << s;
  const long long Cmask = (1ll << twos) - 1;
  const int tid = threadIdx.x;
  if (tid == 0) {
    for (int i = 0; i < WIN_NT + WIN_NB; ++i) mbar_init(&barT[i], 1);
    for (int i = 0; i < 4; ++i) mbar_init(&doneD[i], TPB / 64);   // the four down warps
    fence_mbar_init();
  }
  __syncthreads();
  const long long ntiles = a.nelem / TPB;
  long long tbeg, tend;
  cta_tiles(ntiles, tbeg, tend);
  if (tbeg >= tend) {
    if (XCHG && tid == TPB) p2p_advance(a.xsync, *(volatile unsigned long long*)(a.xsync + P2P_EPOCH));
    return;
  }
  const long long dlo = max(0ll, tbeg - 2), dhi = min(ntiles - 1, tend);       // tiles whose down children I relax
  const long long tlo = max(0ll, dlo - 1), thi = min(ntiles, dhi + 3);         // field tiles I load: [tlo, thi)
  const long long t0 = dlo - 1;                                                // first iteration (down phase one tile ahead)

  if (tid >= TPB) {
    // ------------------------------------------------------------------ producer warp
    const int lane = tid - TPB;
    int u_loaded = -1;
    unsigned long long e64 = 0;                          // exchange number this sweep reads (see k_element_win2)
    if (XCHG) e64 = *(volatile unsigned long long*)(a.xsync + P2P_EPOCH);
    auto issueT = [&](long long tile) { load_tile(sT, barT, (int)(tile & (WIN_NT - 1)), a.Tin, tile); };
    auto issueB = [&](long long tile) {   // whole warp
      const int u = (int)((tile * TPB) >> twos);
      if (u != u_loaded) {
        for (int i = lane; i < NPC; i += 32) sPC2[u & 1][i] = __ldg(a.pc + (size_t)u * NPC + i);
        if (lane < 3) {
          sIdx2[u & 1][lane] = __ldg(a.strip_of + u * 3 + lane); sIdx2[u & 1][4 + lane] = __ldg(a.hmap + u * 3 + lane);
          sIdx2[u & 1][8 + lane] = a.nsrc ? __ldg(a.nsrc + u * 3 + lane) : -1;
        }
        u_loaded = u;
        __syncwarp();
      }
      if (lane == 0) load_tile(sB, barB, (int)((tile - dlo) & (WIN_NB - 1)), a.rhs, tile);
    };
    if (lane == 0) for (long long t = tlo; t < min(thi, t0 + 6); ++t) issueT(t);
    for (long long t = dlo; t <= min(dhi, dlo + 3); ++t) issueB(t);
    int m0 = 0, u_m0 = -1;
    StripDst sd = {-1, -1, -1, 0, nullptr, nullptr, nullptr};
    for (long long tile = t0; tile < tend; ++tile) {
      const int it = (int)(tile - t0);
      named_sync(1 + (it & 3), WIN2_THREADS);            // every consumer warp has finished iteration `tile`
      if (lane == 0) {
        if (tile >= tbeg) {
          tma_store_1d(a.Tout + tile * 3 * TPB, sT + (tile & (WIN_NT - 1)) * 3 * TPB, TILE_BYTES);
          tma_store_commit();
        }
        // ring slot of tile-2: nobody is behind iteration tile+1; its store (two groups ago) has been read
        if (tile + 6 < thi) { tma_store_wait_read2(); issueT(tile + 6); }
      }
      __syncwarp();
      if (tile + 4 >= dlo + 4 && tile + 4 <= dhi) issueB(tile + 4);   // rhs slot of tile: consumed by its up children
      if (a.ovl_next && tile >= tbeg) {                  // halo strips of the next sweep from the finished tile
        const int u = (int)((tile * TPB) >> twos);
        if (u != u_m0) { m0 = 0; u_m0 = u; sd = strip_dst_load(a, u, lane, XCHG ? e64 + 1 : 0); }      // once per parent
        strips_from_tile(a, sT + (tile & (WIN_NT - 1)) * 3 * TPB, sd, (int)((tile * TPB) & Cmask), s, m0, lane, XCHG ? e64 + 1 : 0);
      }
    }
    if (XCHG && lane == 0) p2p_advance(a.xsync, e64);
    if (lane == 0) tma_store_wait_all();
  } else {
    // ------------------------------------------------------------------ consumer warps, split by colour
    // Inside a row up and down children alternate, so a thread per child leaves every other lane idle in each colour phase
    // (ncu: issue-bound at half the lanes).  Here a thread owns a PAIR of adjacent children (2j, 2j+1) of a tile: warps 0-3
    // relax the down child of their pair in tile t+2, warps 4-7 the up child of theirs in tile t - every lane busy, and a warp
    // runs one colour per iteration instead of two.  The one pair per row that straddles a row end holds two up children
    // (last child of row r, first child of row r+1: both on parent faces) and no down child; the down-warp lane that had
    // nothing to do for it relaxes its second child.  (all per-tile index arithmetic in 32-bit: this branch cannot use the
    // uniform datapath)
    const int t0i = (int)t0, tbegi = (int)tbeg, tendi = (int)tend, dloi = (int)dlo, dhii = (int)dhi, tloi = (int)tlo, thii = (int)thi;
    const int pshift = twos - 8;                          // tiles per parent = 2^pshift (TPB = 2^8)
    const unsigned kmask = (unsigned)Cmask;
    auto waitT = [&](int tile) { mbar_wait(&barT[tile & (WIN_NT - 1)], (uint32_t)(((tile - tloi) >> 3) & 1)); };
    auto waitB = [&](int tile) { mbar_wait(&barB[(tile - dloi) & (WIN_NB - 1)], (uint32_t)(((tile - dloi) >> 2) & 1)); };
    const int j2 = (tid & (TPB / 2 - 1)) * 2;             // first child of my pair inside a tile
    int r = 2, ipos = 2;                                  // numbering of child 2j of the tile this thread handled last
    // one up child: row rr, position ip of a row of length ln, at ring index cw; h1 = values across parent face 1,
    // h2 = across the side face the child lies on (side 3 for ip == 1, else side 2)
    auto relax_up = [&](int tile, int cw, int rr, int ip, int ln, double h1a, double h1b, double h2a, double h2b) {
      const int u_tile = tile >> pshift;
      double* t = sT + cw * 3;
      const double T1 = t[0], T2 = t[1], T3 = t[2];
      FaceIn fi;
      int bmask = 0;
      ring_nbrs(sT, cw, true, rr, b, fi);
      if (rr == 1 || ip == 1 || ip == ln) {
        if (rr == 1) { fi.n1a = h1a; fi.n1b = h1b; bmask |= 1; }
        if (ip == 1) { fi.n2a = h2a; fi.n2b = h2b; bmask |= 2; }
        if (ip == ln) {
          if (ln == 1) halo_pair(a, u_tile, 1, rr - 1, S, fi.n3a, fi.n3b);
          else { fi.n3a = h2a; fi.n3b = h2b; }
          bmask |= 4;
        }
      }
      const double* bb = sB + ((tile - dloi) & (WIN_NB - 1)) * (3 * TPB) + (cw & (TPB - 1)) * 3;
      const double* pu = sPC2[u_tile & 1];
      const Folded& F = *reinterpret_cast<const Folded*>(pu + PC_FOLD);
      double o1, o2, o3;
      elem_apply_folded<MODE_GS>(F, pu + PC_DPEN, bmask, T1, T2, T3, fi, bb[0], bb[1], bb[2], a.rsign, o1, o2, o3);
      t[0] = o1; t[1] = o2; t[2] = o3;
    };
    if (tid < TPB / 2) {
      // ---- down warps: tile t+1 (reads the old up values of tiles t .. t+3; the up warps touch tile t only after this phase).
      // A pair whose first child ends its row has no down child: its second child opens the next row - an up child on parent
      // side 3.  The lane that found it idle in the down phase relaxes it one iteration later, when the pair's tile is the up
      // tile (exterior values fetched in between), so that no up warp makes a second trip through the up code.
      bool sec = false;                                    // my pair of tile `tile` holds such a second up child, in row sec_r + 1
      int sec_r = 0;
      double sec_a = 0.0, sec_b = 0.0;
      for (int tile = t0i; tile < tendi; ++tile) {
        const int it = tile - t0i;
        const int td = tile + 1;
        bool nsec = false;
        double nsec_a = 0.0, nsec_b = 0.0;
        if (tile == t0i) {
          for (int tw = tloi; tw < min(thii, tile + 4); ++tw) waitT(tw);
        } else if (tile + 3 < thii) {
          waitT(tile + 3);
        }
        if (td >= dloi && td <= dhii) {
          waitB(td);                                       // also acquires the coefficients of the parent of td
          const int k = (int)((((unsigned)td << 8) + (unsigned)j2) & kmask);
          if (td == dloi) { int len; child_from_ele0(k, s, r, ipos, len); }
          else child_advance(s, b, k, r, ipos);
          // the down child of the pair: child 2j when its position is even, else 2j+1 - unless 2j ends its row
          const int off = ipos & 1;
          if (!off || ipos < b + 1 - 2 * r) {
            const int cw = ((td & (WIN_NT - 1)) << 8) + j2 + off;
            double* t = sT + cw * 3;
            const double T1 = t[0], T2 = t[1], T3 = t[2];
            FaceIn fi;
            ring_nbrs(sT, cw, false, r, b, fi);
            const double* bb = sB + ((td - dloi) & (WIN_NB - 1)) * (3 * TPB) + (j2 + off) * 3;
            const double* pd = sPC2[(td >> pshift) & 1] + PC_FOLD + 16;
            const Folded& F = *reinterpret_cast<const Folded*>(pd);
            double o1, o2, o3;
            elem_apply_folded<MODE_GS>(F, pd, 0, T1, T2, T3, fi, bb[0], bb[1], bb[2], a.rsign, o1, o2, o3);
            t[0] = o1; t[1] = o2; t[2] = o3;
          } else if (td >= tbegi && td < tendi) {
            const int* ix = sIdx2[(td >> pshift) & 1];
            ext_face(a, 2, r + 1, 1, S, [&](int j) { return ix[j]; }, nsec_a, nsec_b);   // first child of row r+1
            nsec = true;
          }
        }
        // down phase of this iteration done (also when there was nothing to do): tell the up warps
        __syncwarp();
        if ((tid & 31) == 0) mbar_arrive_cta(&doneD[it & 3]);
        if (sec) {
          // (its right neighbour may be the first down child of tile+1: every down warp must be through this iteration)
          mbar_wait(&doneD[it & 3], (uint32_t)((it >> 2) & 1));
          relax_up(tile, ((tile & (WIN_NT - 1)) << 8) + j2 + 1, sec_r + 1, 1, b - 1 - 2 * sec_r, 0.0, 0.0, sec_a, sec_b);
        }
        sec = nsec; sec_r = r; sec_a = nsec_a; sec_b = nsec_b;
        fence_async_smem();
        named_arrive(1 + (it & 3), WIN2_THREADS);
      }
    } else {
      // ---- up warps: tile t (reads the new down values of tiles t-2 .. t+1)
      struct Prep { int r, ipos, len, off; double h1a, h1b, h2a, h2b; };   // my first up child of a tile, its halo values
      auto prepare = [&](int tile, Prep& p) {
        p.r = 2; p.ipos = 2; p.len = 3; p.off = 0; p.h1a = 0.0; p.h1b = 0.0; p.h2a = 0.0; p.h2b = 0.0;
        if (tile < tbegi || tile >= tendi) return;
        waitB(tile);                                       // landed long ago; acquires the tables of the tile's parent
        const int k = (int)((((unsigned)tile << 8) + (unsigned)j2) & kmask);
        if (tile == tbegi) { int len; child_from_ele0(k, s, r, ipos, len); }
        else child_advance(s, b, k, r, ipos);
        p.off = (ipos & 1) ^ 1;                            // child 2j when its position is odd, else 2j+1 (same row: rows are odd)
        p.r = r; p.ipos = ipos + p.off; p.len = b + 1 - 2 * r;
        const bool f1 = p.r == 1, side = p.ipos == 1 || p.ipos == p.len;
        if (f1 | side) {
          const int* ix = sIdx2[(tile >> pshift) & 1];
          if (f1) { ext_pair(a, ix[8], ix[0], ix[4], p.ipos >> 1, S, p.h1a, p.h1b); }
          if (side) {
            const int mf = (p.ipos == 1) ? 2 : 1;
            ext_pair(a, ix[8 + mf], ix[mf], ix[4 + mf], p.r - 1, S, p.h2a, p.h2b);
          }
        }
      };
      Prep cur, nxt;
      prepare(t0i, cur);                                   // t0 < tbeg: defaults
      for (int tile = t0i; tile < tendi; ++tile) {
        const int it = tile - t0i;
        if (tile == t0i) {
          for (int tw = tloi; tw < min(thii, tile + 2); ++tw) waitT(tw);
        } else if (tile + 1 < thii) {
          waitT(tile + 1);
        }
        prepare(tile + 1, nxt);
        if (tile >= tbegi) {
          // every down warp has finished THIS iteration: the down children of tile+1 are new (those of tile-2 .. tile are
          // older) and nobody reads the old up values of this tile any more
          mbar_wait(&doneD[it & 3], (uint32_t)((it >> 2) & 1));
          const int cw = ((tile & (WIN_NT - 1)) << 8) + j2 + cur.off;
          relax_up(tile, cw, cur.r, cur.ipos, cur.len, cur.h1a, cur.h1b, cur.h2a, cur.h2b);   // (a second up child of the pair: the down warps)
        }
        fence_async_smem();
        named_arrive(1 + (it & 3), WIN2_THREADS);
        cur = nxt;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Branch-free direct kernel: thread per child, every load of the child (own values, rhs, the three
// neighbours) is issued before the first use so that one memory latency is exposed per child instead of a
// chain of two or three; children on a parent face patch their neighbour values from the halo strips in a
// rare branch.  Coefficients come straight from the per-parent table (L1-resident).  Used on levels with fewer
// than 256 children per parent (n_split <= 3) in every mode but the one-pass GS with face terms (k_gs_small).
// one child, everything from global memory: used by the direct kernel and by the boundary fix-up kernel
template <int MODE, bool FACE>
__device__ __forceinline__ void child_update(const ElemArgs& a, int u, int r, int ipos, int ele, int len, double& acc_sum,
                                             double& acc_abs, double& acc_max) {
  const int s = a.s, twos = 2 * s, b = 2 << s, S = 1 << s;
  const bool up = ipos & 1;
  const unsigned pbase = (unsigned)u << twos;
  const unsigned e0 = pbase + (unsigned)(ele - 1);
  // neighbour children; a missing neighbour (parent face) falls back to the child itself (valid address)
  const int nb1 = up ? (r > 1 ? ele - b - 2 + 2 * r : ele) : ele + b - 2 * r;
  const int nb2 = up ? (ipos > 1 ? ele - 1 : ele) : ele + 1;
  const int nb3 = up ? (ipos < len ? ele + 1 : ele) : ele - 1;
  const unsigned base = e0 * 3u;
  auto ldT = [&](unsigned i) -> double { return MODE == MODE_GS ? a.Tin[i] : __ldg(a.Tin + i); };
  const double T1 = ldT(base), T2 = ldT(base + 1), T3 = ldT(base + 2);
  const double b1 = __ldg(a.rhs + base), b2 = __ldg(a.rhs + base + 1), b3 = __ldg(a.rhs + base + 2);
  FaceIn fi;
  const ParentRegs& P = *reinterpret_cast<const ParentRegs*>(a.pc + (size_t)u * NPC);
  bool interior = true;
  int bmask = 0;
  if (FACE) {
    const unsigned o1 = (pbase + (unsigned)(nb1 - 1)) * 3u, o2 = (pbase + (unsigned)(nb2 - 1)) * 3u,
                   o3 = (pbase + (unsigned)(nb3 - 1)) * 3u;
    pair_face<1>([&](int n) { return ldT(o1 + n); }, fi.n1a, fi.n1b);
    pair_face<2>([&](int n) { return ldT(o2 + n); }, fi.n2a, fi.n2b);
    pair_face<3>([&](int n) { return ldT(o3 + n); }, fi.n3a, fi.n3b);
    fi.pen1 = P.pi1; fi.pen2 = P.pi2; fi.pen3 = P.pi3;
    if (up && (r == 1 || ipos == 1 || ipos == len)) {   // child on a parent face (rare): halo strips
      interior = false;
      bmask = parent_faces(r, ipos, len, P, [&](int, int side, int pos, double& va, double& vb) {
        halo_pair(a, u, side, pos, S, va, vb);
      }, fi);
    }
  }
  double o1v, o2v, o3v;
  if (FACE && MODE != MODE_RICH) {
    const double* pcu = a.pc + (size_t)u * NPC;
    const Folded& F = *reinterpret_cast<const Folded*>(pcu + PC_FOLD + (up ? 0 : 16));
    elem_apply_folded<MODE>(F, pcu + PC_DPEN, bmask, T1, T2, T3, fi, b1, b2, b3, a.rsign, o1v, o2v, o3v);
  } else {
    elem_apply_regs<MODE, FACE>(P, up, interior, T1, T2, T3, fi, b1, b2, b3, a.omega, a.rsign, o1v, o2v, o3v);
  }
  a.Tout[base] = o1v; a.Tout[base + 1] = o2v; a.Tout[base + 2] = o3v;
  if (MODE == MODE_RESID) {
    acc_sum += o1v * o1v + o2v * o2v + o3v * o3v;
    acc_abs = fmax(acc_abs, fmax(fabs(o1v), fmax(fabs(o2v), fabs(o3v))));
    acc_max = fmax(acc_max, fmax(o1v, fmax(o2v, o3v)));
  }
}

template <int MODE, bool FACE>
__global__ void __launch_bounds__(TPB) k_element_direct2(ElemArgs a) {
  const int s = a.s, twos = 2 * s;
  const unsigned Cmask = (1u << twos) - 1u;
  double acc_sum = 0.0, acc_abs = 0.0, acc_max = 0.0;
  const unsigned nelem = (unsigned)a.nelem;
  for (unsigned gid = blockIdx.x * TPB + threadIdx.x; gid < nelem; gid += gridDim.x * TPB) {
    const int u = (int)(gid >> twos);
    int r, ipos, ele, len;
    child_from_flat((int)(gid & Cmask), s, r, ipos, ele, len);
    if (MODE == MODE_GS && (ipos & 1) != a.colour) continue;
    child_update<MODE, FACE>(a, u, r, ipos, ele, len, acc_sum, acc_abs, acc_max);
  }
  if (MODE == MODE_RESID) block_partial(acc_sum, acc_abs, acc_max, a.partial + (size_t)3 * a.partial_off);
}

// ------------------------------------------------------------------------------------------------
// Coloured Gauss-Seidel sweep on a SMALL level (at most TPB children per parent, n_split <= 4) in one launch, out of place.
// Inside a parent the two colours couple only children of that parent, and values across parent faces are lagged by one
// sweep anyway (transport_tri_semi.F90:647-655): a CTA that owns whole parents keeps them in shared memory, relaxes the down
// children, synchronises, relaxes the up children (exterior values straight from the neighbour parents' boundary children in
// the start-of-sweep field, or from the strips of cut / Dirichlet faces) and writes the parents out.  Same arithmetic as the
// two in-place passes over global memory it replaces (three launches per sweep with their halo kernel): these levels are
// launch-bound.
__global__ void __launch_bounds__(TPB) k_gs_small(ElemArgs a) {
  __shared__ double sT[3 * TPB];
  const int s = a.s, twos = 2 * s, C = 1 << twos, b = 2 << s, S = 1 << s;
  const int tid = threadIdx.x;
  const int ppc = TPB >> twos;                          // parents per CTA
  const int nparents = (int)(a.nelem >> twos);
  const int lu = tid >> twos, k = tid & (C - 1);        // my parent inside the CTA, my child (memory order)
  int r, ipos, len;
  child_from_ele0(k, s, r, ipos, len);
  const bool up = ipos & 1;
  double* t = sT + tid * 3;
  for (int pbase = blockIdx.x * ppc; pbase < nparents; pbase += gridDim.x * ppc) {
    const int u = pbase + lu;
    const bool active = u < nparents;
    double b1 = 0.0, b2 = 0.0, b3 = 0.0;
    const size_t g3 = ((size_t)(active ? u : 0) * C + k) * 3;
    if (active) {
      t[0] = __ldg(a.Tin + g3); t[1] = __ldg(a.Tin + g3 + 1); t[2] = __ldg(a.Tin + g3 + 2);
      b1 = __ldg(a.rhs + g3); b2 = __ldg(a.rhs + g3 + 1); b3 = __ldg(a.rhs + g3 + 2);
    }
    const double* pcu = a.pc + (size_t)(active ? u : 0) * NPC;
    FaceIn fi;
    int bmask = 0;
    if (active && up && (r == 1 || ipos == 1 || ipos == len)) {   // exterior values first: their latency hides under the down phase
      if (r == 1) { halo_pair(a, u, 0, ipos >> 1, S, fi.n1a, fi.n1b); bmask |= 1; }
      if (ipos == 1) { halo_pair(a, u, 2, r - 1, S, fi.n2a, fi.n2b); bmask |= 2; }
      if (ipos == len) { halo_pair(a, u, 1, r - 1, S, fi.n3a, fi.n3b); bmask |= 4; }
    }
    __syncthreads();
    const double* P0 = sT + (lu << twos) * 3;           // my parent's children
    if (active && !up) {
      const double T1 = t[0], T2 = t[1], T3 = t[2];
      pair_nodes(P0 + nbr1(k, false, r, b) * 3, P0 + (k + 1) * 3, P0 + (k - 1) * 3, fi);
      const Folded& F = *reinterpret_cast<const Folded*>(pcu + PC_FOLD + 16);
      double o1, o2, o3;
      elem_apply_folded<MODE_GS>(F, pcu + PC_DPEN, 0, T1, T2, T3, fi, b1, b2, b3, a.rsign, o1, o2, o3);
      t[0] = o1; t[1] = o2; t[2] = o3;
    }
    __syncthreads();
    if (active && up) {
      const double T1 = t[0], T2 = t[1], T3 = t[2];
      if (!(bmask & 1)) { const double* tv = P0 + (k + 2 * r - b - 2) * 3; fi.n1a = tv[2]; fi.n1b = tv[0]; }
      if (!(bmask & 2)) { const double* tl = P0 + (k - 1) * 3; fi.n2a = tl[1]; fi.n2b = tl[2]; }
      if (!(bmask & 4)) { const double* tr = P0 + (k + 1) * 3; fi.n3a = tr[0]; fi.n3b = tr[1]; }
      const Folded& F = *reinterpret_cast<const Folded*>(pcu + PC_FOLD);
      double o1, o2, o3;
      elem_apply_folded<MODE_GS>(F, pcu + PC_DPEN, bmask, T1, T2, T3, fi, b1, b2, b3, a.rsign, o1, o2, o3);
      t[0] = o1; t[1] = o2; t[2] = o3;
    }
    if (active) { a.Tout[g3] = t[0]; a.Tout[g3 + 1] = t[1]; a.Tout[g3 + 2] = t[2]; }   // (my own child: no barrier needed)
    __syncthreads();
  }
}

// second stage of the norm reduction: one CTA
__global__ void __launch_bounds__(1024) k_reduce_partials(const double* partial, int n, double* out3) {
  double s0 = 0, s1 = 0, s2 = 0;
  for (int i = threadIdx.x; i < n; i += 1024) {
    s0 += partial[(size_t)i * 3]; s1 = fmax(s1, partial[(size_t)i * 3 + 1]); s2 = fmax(s2, partial[(size_t)i * 3 + 2]);
  }
  for (int o = 16; o > 0; o >>= 1) {
    s0 += __shfl_xor_sync(0xffffffffu, s0, o);
    s1 = fmax(s1, __shfl_xor_sync(0xffffffffu, s1, o));
    s2 = fmax(s2, __shfl_xor_sync(0xffffffffu, s2, o));
  }
  __shared__ double sh[3][32];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { sh[0][w] = s0; sh[1][w] = s1; sh[2][w] = s2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    s0 = 0; s1 = 0; s2 = 0;
    for (int i = 0; i < 32; ++i) { s0 += sh[0][i]; s1 = fmax(s1, sh[1][i]); s2 = fmax(s2, sh[2][i]); }
    out3[0] = s0; out3[1] = s1; out3[2] = s2;
  }
}

// ------------------------------------------------------------------------------------------------
// update_overlaps (splitting.F90:1210-1397): one thread per (parent, side, position)
// ------------------------------------------------------------------------------------------------
// poll my staging buffer, unpack into the strips, and let the last block advance the exchange number
__device__ __forceinline__ void p2p_receive(const P2PArgs& a, unsigned long long e64, bool advance) {
  __shared__ int s_last;
  const int tid = threadIdx.x;
  const unsigned e = (unsigned)e64;
  const long long par = (long long)(e64 & (P2P_SLOTS - 1)) * a.stage_words;
  const long long nr = a.roff[a.npeers];
  volatile unsigned long long* err = a.err;
  for (long long i = (long long)blockIdx.x * TPB + tid; i < nr; i += (long long)gridDim.x * TPB) {
    int p = 0;
    while (i >= a.roff[p + 1]) ++p;
    const long long j = a.rbeg[p] + (i - a.roff[p]);
    const uint4* src = a.stage + par + j;
    uint4 w;
    unsigned long long t0 = 0;
    bool ok = true;
    for (unsigned spins = 0;; ++spins) {
      asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(w.x), "=r"(w.y), "=r"(w.z), "=r"(w.w) : "l"(src) : "memory");
      if (w.y == e && w.w == e) break;
      if ((spins & 1023u) == 1023u) {
        if (*err) { ok = false; break; }
        const unsigned long long t = p2p_now();
        if (t0 == 0) t0 = t;
        else if (t - t0 > a.timeout_ns) { *err = 1; ok = false; break; }
      }
    }
    if (ok) a.strips[j] = __longlong_as_double((long long)(((unsigned long long)w.z << 32) | w.x));
  }
  if (!advance) return;
  __syncthreads();
  if (tid == 0) { __threadfence(); s_last = (atomicAdd(a.sync + P2P_COUNT, 1ull) == (unsigned long long)gridDim.x - 1); }
  __syncthreads();
  if (s_last && tid == 0) { a.sync[P2P_COUNT] = 0; *(volatile unsigned long long*)(a.sync + P2P_EPOCH) = e64; __threadfence(); }
}

// ------------------------------------------------------------------------------------------------
// Device-initiated block transfer between the GPUs of one process (coarse-level agglomeration, SURVEY 8(e)): the sender
// stores a contiguous range straight into the receiver's memory over NVLink, fences at system scope, and the last block
// publishes the transfer number in a flag word on the receiver; the receiver's stream runs k_wait_flags before it touches
// the data.  Both counters live in device memory, so captured CUDA graphs replay correctly, and there is no host
// synchronisation, event or library call between the GPUs.
struct PushArgs {
  const double* src; double* dst;          // dst: peer memory
  long long n;
  unsigned long long* counter;             // local: blocks done
  unsigned long long* epoch;               // local: transfers sent on this channel so far
  unsigned long long* flag;                // peer: transfer number of the last complete transfer
};

__global__ void __launch_bounds__(TPB) k_push(PushArgs a) {
  for (long long i = (long long)blockIdx.x * TPB + threadIdx.x; i < a.n; i += (long long)gridDim.x * TPB) a.dst[i] = a.src[i];
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    if (atomicAdd(a.counter, 1ull) == (unsigned long long)gridDim.x - 1) {
      __threadfence_system();
      const unsigned long long e = *a.epoch + 1;
      *a.epoch = e; *a.counter = 0;
      __threadfence_system();
      *(volatile unsigned long long*)a.flag = e;
    }
  }
}

struct WaitArgs {
  unsigned long long* flags;               // local: one word per sender
  unsigned long long* expect;              // local: transfers received per sender so far
  unsigned long long* err;                 // mapped host memory
  unsigned long long timeout_ns;
  unsigned senders;                        // bit p set: wait for sender p
};

__global__ void k_wait_flags(WaitArgs a) {
  const int p = threadIdx.x;
  if (p < 32 && ((a.senders >> p) & 1u)) {
    const unsigned long long want = a.expect[p] + 1;
    a.expect[p] = want;
    unsigned long long t0 = 0;
    for (unsigned spins = 0;; ++spins) {
      if (*(volatile unsigned long long*)(a.flags + p) >= want) break;
      if ((spins & 1023u) == 1023u) {
        if (*(volatile unsigned long long*)a.err) break;
        const unsigned long long t = p2p_now();
        if (t0 == 0) t0 = t;
        else if (t - t0 > a.timeout_ns) { *(volatile unsigned long long*)a.err = 2; break; }
      }
    }
  }
  __threadfence_system();
}

// what a k_halo launch writes (HaloArgs::what)
enum HaloMode {
  HALO_ALL = 0,        // everything: update_overlaps as written, tnew and told strips
  HALO_DIRICHLET = 1,  // Dirichlet faces only
  HALO_CUT = 2,        // faces cut by the GPU partition only (one thread per position of the faces listed in cut_lf)
  HALO_SHARED = 3,     // every face shared by two parents (no Dirichlet data)
  HALO_UNPACK = 4      // unpack the cut-face values a sweep's producer warps sent into my staging buffer
};

struct HaloArgs {
  P2PArgs x;                               // x.npeers > 0: cut-face strips go straight to the peers (fused exchange)
  const double* tnew; const double* told;
  double* ovl; double* ovl_old;           // strip space: local strips then send slots
  const double* xg;                        // [U][6] X3, X1-X3, X2-X3
  const int32_t* dst_strip; const int32_t* rev; const int32_t* strip_of;
  double bc_scale;
  int U, s, with_old;
  int what;                                // a HaloMode
  int nstrips;
  const int32_t* cut_lf; int ncut;         // HALO_CUT: (u*3+mf) of the cut faces
  // Dirichlet data of domain-boundary faces per (u, side): kind 0 = sin(x+y) (splitting.F90:1246-1252), 1 = the constant
  // bc_val (update_overlaps' t_bc argument, :1210), 2 = open face, no data; nullptr = kind 0 everywhere
  const int32_t* bc_kind; const double* bc_val;
};

__device__ __forceinline__ void child_nodes(const double* __restrict__ xg, int s, int r, int ipos, double x[3][2]) {
  // get_splitting, Msh2Tri.F90:79-106 (same operation order as the reference: divide first)
  const double inv = (double)(1 << s);
  for (int d = 0; d < 2; ++d) {
    const double o = __ldg(xg + d), v1 = __ldg(xg + 2 + d) / inv, v2 = __ldg(xg + 4 + d) / inv;
    if (ipos & 1) {
      x[2][d] = o + (r - 1) * v2 + (ipos / 2) * v1;
      x[1][d] = o + r * v2 + (ipos / 2) * v1;
      x[0][d] = o + (r - 1) * v2 + v1 * (ipos / 2 + 1);
    } else {
      x[0][d] = o + r * v2 + v1 * (ipos / 2 - 1);
      x[1][d] = o + (r - 1) * v2 + v1 * (ipos / 2);
      x[2][d] = o + r * v2 + v1 * (ipos / 2);
    }
  }
}

__global__ void __launch_bounds__(TPB) k_halo(HaloArgs a) {
  const int S = 1 << a.s, b = 2 << a.s;
  const long long n = (a.what == HALO_CUT ? (long long)a.ncut : (long long)a.U * 3) * S;
  unsigned long long e64 = 0;
  if (a.x.npeers > 0) e64 = *(volatile unsigned long long*)(a.x.sync + P2P_EPOCH) + 1;
  if (a.what == HALO_UNPACK) {             // the values of the current exchange sit in my staging buffer (a sweep's producer
    p2p_receive(a.x, e64 - 1, false);      // warps sent them): unpack them into the strips, nothing to send
    return;
  }
  for (long long tid = (long long)blockIdx.x * TPB + threadIdx.x; tid < n; tid += (long long)gridDim.x * TPB) {
    const int i = (int)(tid & (S - 1));           // position - 1
    const int lf = (a.what == HALO_CUT) ? __ldg(a.cut_lf + (tid >> a.s)) : (int)(tid >> a.s);   // u*3 + mf
    const int u = lf / 3, mf = lf - 3 * u;
    const int pos = i + 1;
    int r, ipos;
    if (mf == 0) { r = 1; ipos = 2 * pos - 1; }                  // surf_ele(:,1): odd children of row 1
    else if (mf == 2) { r = pos; ipos = 1; }                     // surf_ele(:,3): first child of each row
    else { r = pos; ipos = b + 1 - 2 * pos; }                    // surf_ele(:,2): last child of each row
    const int ele = 1 + (r - 1) * (b + 1 - r) + ipos - 1;
    const int dst = __ldg(a.dst_strip + lf);
    const size_t S3 = (size_t)3 * S;
    if (a.what == HALO_DIRICHLET && dst >= 0) continue;
    if (a.what == HALO_CUT && dst < a.nstrips) continue;
    if (a.what == HALO_SHARED && dst < 0) continue;
    if (dst < 0) {
      // Dirichlet data at the two face nodes (:1246-1252,1287-1293,1344-1350): sin(x+y), or the constant t_bc of the face
      const int kind = a.bc_kind ? __ldg(a.bc_kind + lf) : 0;
      if (kind == 2) continue;                    // open face: no data (its penalty coefficient is zero)
      double x[3][2];
      child_nodes(a.xg + (size_t)u * 6, a.s, r, ipos, x);
      const int na = (mf == 2) ? 1 : 0, nb = (mf == 0) ? 2 : (mf == 1 ? 1 : 2);
      double ta = a.bc_scale * sin(x[na][0] + x[na][1]);
      double tb = a.bc_scale * sin(x[nb][0] + x[nb][1]);
      if (kind == 1) ta = tb = a.bc_scale * __ldg(a.bc_val + lf);
      const size_t o = (size_t)__ldg(a.strip_of + lf) * S3 + (size_t)i * 3;
      a.ovl[o + na] = ta; a.ovl[o + nb] = tb;
      if (a.with_old) { a.ovl_old[o + na] = ta; a.ovl_old[o + nb] = tb; }
    } else {
      const int slot = __ldg(a.rev + lf) ? (S - pos) : (pos - 1);
      const size_t o = (size_t)dst * S3 + (size_t)slot * 3;
      const size_t src = (((size_t)u << (2 * a.s)) + ele - 1) * 3;
      const double v0 = a.tnew[src], v1 = a.tnew[src + 1], v2 = a.tnew[src + 2];
      a.ovl[o] = v0; a.ovl[o + 1] = v1; a.ovl[o + 2] = v2;
      if (a.with_old) { a.ovl_old[o] = a.told[src]; a.ovl_old[o + 1] = a.told[src + 1]; a.ovl_old[o + 2] = a.told[src + 2]; }
      if (a.x.npeers > 0 && dst >= a.nstrips) {
        // face cut by the GPU partition: the same three values also go straight into the neighbour GPU's staging buffer
        const long long q = (long long)(dst - a.nstrips - a.x.send_base) * (long long)S3 + (long long)slot * 3;
        int p = 0;
        while (q >= a.x.soff[p + 1]) ++p;
        p2p_put(a.x, (unsigned)e64, p, q - a.x.soff[p], v0);
        p2p_put(a.x, (unsigned)e64, p, q - a.x.soff[p] + 1, v1);
        p2p_put(a.x, (unsigned)e64, p, q - a.x.soff[p] + 2, v2);
      }
    }
  }
  if (a.x.npeers > 0) p2p_receive(a.x, e64, true);
}

// ------------------------------------------------------------------------------------------------
// level-1 RHS: source reset (:593) + get_RHS (:452-464), theta = 1
struct RhsArgs {
  const double* told; double* rhs; const double* pc; const double* xg;
  double dt, source_coef;
  long long nelem;
  int s, literal_source;
};

__global__ void __launch_bounds__(TPB) k_build_rhs(RhsArgs a) {
  const int s = a.s, twos = 2 * s;
  const long long Cmask = (1ll << twos) - 1;
  for (long long gid = (long long)blockIdx.x * TPB + threadIdx.x; gid < a.nelem; gid += (long long)gridDim.x * TPB) {
    const int u = (int)(gid >> twos);
    int r, ipos, ele, len;
    child_from_flat((int)(gid & Cmask), s, r, ipos, ele, len);
    const long long base = (((long long)u << twos) + ele - 1) * 3;
    double x[3][2];
    child_nodes(a.xg + (size_t)u * 6, s, r, ipos, x);
    const double cm = __ldg(a.pc + (size_t)u * NPC + PC_CM);
    const double m12 = cm * a.dt;   // A_child / 12
    double s1 = a.source_coef * sin(x[0][0] + x[0][1]);
    double s2 = a.source_coef * sin(x[1][0] + x[1][1]);
    double s3 = a.source_coef * sin(x[2][0] + x[2][1]);
    double q1, q2, q3;
    if (a.literal_source) {  // in-place: src(i) = M(i,:) . src with src already partly overwritten
      q1 = m12 * (2.0 * s1 + s2 + s3);
      q2 = m12 * (q1 + 2.0 * s2 + s3);
      q3 = m12 * (q1 + q2 + 2.0 * s3);
    } else {
      const double ss = s1 + s2 + s3;
      q1 = m12 * (s1 + ss); q2 = m12 * (s2 + ss); q3 = m12 * (s3 + ss);
    }
    const double o1 = a.told[base], o2 = a.told[base + 1], o3 = a.told[base + 2];
    const double so = o1 + o2 + o3;
    a.rhs[base] = cm * (o1 + so) + q1;
    a.rhs[base + 1] = cm * (o2 + so) + q2;
    a.rhs[base + 2] = cm * (o3 + so) + q3;
  }
}

// ------------------------------------------------------------------------------------------------
// restrictor (splitting.F90:10-32) / its INTENDED form (transpose of P1 interpolation).
// One thread per COARSE child; fine ids from the closed form of element_conversion (:105-139).
__host__ __device__ __forceinline__ void fine_children(int sc, int r, int ipos, int fin[4]) {
  const int bf = 4 << sc;  // 2^(sf+1), sf = sc+1
  auto start_f = [&](int rf) { return 1 + (rf - 1) * (bf + 1 - rf); };
  if (ipos & 1) {
    fin[0] = start_f(2 * r - 1) + 2 * ipos - 2;
    fin[1] = fin[0] + 1; fin[2] = fin[0] + 2;
    fin[3] = start_f(2 * r) + 2 * ipos - 2;
  } else {
    fin[2] = start_f(2 * r) + 2 * ipos - 3;
    fin[1] = fin[2] + 1; fin[0] = fin[2] + 2;
    fin[3] = start_f(2 * r - 1) + 2 * ipos - 1;
  }
}

struct XferArgs {
  const double* src; double* dst;
  long long ncoarse;   // U * 4^sc
  int sc;              // coarse split
  int mode;            // 0 literal, 1 intended
};

__global__ void __launch_bounds__(TPB) k_restrict(XferArgs a) {
  const int sc = a.sc, twoc = 2 * sc, twof = twoc + 2;
  const long long Cmask = (1ll << twoc) - 1;
  for (long long gid = (long long)blockIdx.x * TPB + threadIdx.x; gid < a.ncoarse; gid += (long long)gridDim.x * TPB) {
    const int u = (int)(gid >> twoc);
    int r, ipos, ele, len;
    child_from_flat((int)(gid & Cmask), sc, r, ipos, ele, len);
    int fin[4];
    fine_children(sc, r, ipos, fin);
    const long long fb = ((long long)u << twof);
    double R[4][3];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const long long o = (fb + fin[k] - 1) * 3;
      R[k][0] = __ldg(a.src + o); R[k][1] = __ldg(a.src + o + 1); R[k][2] = __ldg(a.src + o + 2);
    }
    const long long oc = (((long long)u << twoc) + ele - 1) * 3;
    if (a.mode == 0) {
      a.dst[oc + 0] = (R[2][0] + R[2][1] + R[2][2]) / 3.0;   // splitting.F90:26
      a.dst[oc + 1] = (R[3][0] + R[3][1] + R[3][2]) / 3.0;   // :27
      a.dst[oc + 2] = (R[0][0] + R[0][1] + R[0][2]) / 3.0;   // :28
    } else {
      // P^T with P from splitting.F90:59-88: fin1 holds coarse node 3, fin3 node 1, fin4 node 2,
      // fin2 is the inverted centre child with nodes mid(2,3), mid(1,3), mid(1,2)
      a.dst[oc + 0] = R[2][0] + 0.5 * (R[0][0] + R[1][1] + R[1][2] + R[2][1] + R[2][2] + R[3][0]);
      a.dst[oc + 1] = R[3][1] + 0.5 * (R[0][1] + R[1][0] + R[1][2] + R[2][1] + R[3][0] + R[3][2]);
      a.dst[oc + 2] = R[0][2] + 0.5 * (R[0][0] + R[0][1] + R[1][0] + R[1][1] + R[2][2] + R[3][2]);
    }
  }
}

// prolongator (splitting.F90:38-91) as written: one thread per coarse child (the mixing of totals and
// corrections for the centre child, SURVEY B-8, only touches that child's own four fine children)
__global__ void __launch_bounds__(TPB) k_prolong_literal(XferArgs a) {
  const int sc = a.sc, twoc = 2 * sc, twof = twoc + 2;
  const long long Cmask = (1ll << twoc) - 1;
  for (long long gid = (long long)blockIdx.x * TPB + threadIdx.x; gid < a.ncoarse; gid += (long long)gridDim.x * TPB) {
    const int u = (int)(gid >> twoc);
    int r, ipos, ele, len;
    child_from_flat((int)(gid & Cmask), sc, r, ipos, ele, len);
    int fin[4];
    fine_children(sc, r, ipos, fin);
    const long long oc = (((long long)u << twoc) + ele - 1) * 3;
    const double c1 = a.src[oc], c2 = a.src[oc + 1], c3 = a.src[oc + 2];
    const long long fb = ((long long)u << twof);
    double* f1 = a.dst + (fb + fin[0] - 1) * 3;
    double* f2 = a.dst + (fb + fin[1] - 1) * 3;
    double* f3 = a.dst + (fb + fin[2] - 1) * 3;
    double* f4 = a.dst + (fb + fin[3] - 1) * 3;
    f1[0] += 0.5 * c3 + 0.5 * c1; f1[1] += 0.5 * c2 + 0.5 * c3; f1[2] += c3;
    f2[0] += f1[1]; f2[1] += f1[0]; f2[2] += 0.5 * c1 + 0.5 * c2;
    f3[0] += c1; f3[1] += f2[2]; f3[2] += f2[1];
    f4[0] += f2[2]; f4[1] += c2; f4[2] += f2[0];
  }
}

// INTENDED prolongation: P1 interpolation of the coarse correction, one thread per FINE child so that
// the read-modify-write of the fine field is a coalesced stream.
__global__ void __launch_bounds__(TPB) k_prolong_p1(XferArgs a) {
  const int sf = a.sc + 1, twof = 2 * sf, twoc = twof - 2;
  const long long nfine = a.ncoarse * 4;
  const long long Fmask = (1ll << twof) - 1;
  const int bc = 2 << a.sc;
  for (long long gid = (long long)blockIdx.x * TPB + threadIdx.x; gid < nfine; gid += (long long)gridDim.x * TPB) {
    const int u = (int)(gid >> twof);
    int rf, ipf, elef, len;
    child_from_flat((int)(gid & Fmask), sf, rf, ipf, elef, len);
    const int rc = (rf + 1) >> 1;
    const int m = ipf & 3;
    int k, ipc;
    if (rf & 1) {
      if (m == 1) { k = 0; ipc = (ipf + 1) >> 1; }
      else if (m == 2) { k = 1; ipc = ipf >> 1; }
      else if (m == 3) { k = 2; ipc = (ipf - 1) >> 1; }
      else { k = 3; ipc = ipf >> 1; }
    } else {
      if (m == 1) { k = 3; ipc = (ipf + 1) >> 1; }
      else if (m == 2) { k = 2; ipc = (ipf + 2) >> 1; }
      else if (m == 3) { k = 1; ipc = (ipf + 1) >> 1; }
      else { k = 0; ipc = ipf >> 1; }
    }
    const int elec = 1 + (rc - 1) * (bc + 1 - rc) + ipc - 1;
    const long long oc = (((long long)u << twoc) + elec - 1) * 3;
    const double c1 = __ldg(a.src + oc), c2 = __ldg(a.src + oc + 1), c3 = __ldg(a.src + oc + 2);
    double e1, e2, e3;
    if (k == 0) { e1 = 0.5 * (c1 + c3); e2 = 0.5 * (c2 + c3); e3 = c3; }
    else if (k == 1) { e1 = 0.5 * (c2 + c3); e2 = 0.5 * (c1 + c3); e3 = 0.5 * (c1 + c2); }
    else if (k == 2) { e1 = c1; e2 = 0.5 * (c1 + c2); e3 = 0.5 * (c1 + c3); }
    else { e1 = 0.5 * (c1 + c2); e2 = c2; e3 = 0.5 * (c2 + c3); }
    const long long of = (((long long)u << twof) + elef - 1) * 3;
    a.dst[of] += e1; a.dst[of + 1] += e2; a.dst[of + 2] += e3;
  }
}

// ------------------------------------------------------------------------------------------------
// output side (get_vtu call site transport_tri_semi.F90:299-312): child coordinates x_all_str (:274), the
// analytical field boundary(x,y) = sin(x+y) (:278, splitting.F90:1401-1405) and get_error (:531-540).
struct OutArgs {
  const double* xg; const double* T;
  double* x_all;     // [nelem][3][2] or nullptr
  double* analytical;  // [nelem][3] or nullptr
  double* error;       // [nelem][3] or nullptr
  long long nelem; int s;
};

__global__ void __launch_bounds__(TPB) k_output_fields(OutArgs a) {
  const int twos = 2 * a.s;
  const long long Cmask = (1ll << twos) - 1;
  for (long long g = (long long)blockIdx.x * TPB + threadIdx.x; g < a.nelem; g += (long long)gridDim.x * TPB) {
    const int u = (int)(g >> twos);
    int r, ipos, len;
    child_from_ele0((int)(g & Cmask), a.s, r, ipos, len);
    double x[3][2];
    child_nodes(a.xg + (size_t)u * 6, a.s, r, ipos, x);
    if (a.x_all)
#pragma unroll
      for (int i = 0; i < 3; ++i) { a.x_all[g * 6 + 2 * i] = x[i][0]; a.x_all[g * 6 + 2 * i + 1] = x[i][1]; }
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const double an = sin(x[i][0] + x[i][1]);
      if (a.analytical) a.analytical[g * 3 + i] = an;
      if (a.error) a.error[g * 3 + i] = fabs(a.T[g * 3 + i] - an);
    }
  }
}

__global__ void __launch_bounds__(TPB) k_fill(double* p, long long n, double v) {
  for (long long i = (long long)blockIdx.x * TPB + threadIdx.x; i < n; i += (long long)gridDim.x * TPB) p[i] = v;
}

}  // namespace pamg
