/*
 * pamg.h -- C ABI of libpamg_cuda.so: the B200 (sm_100a) implementation of the P1 DG
 * transport/diffusion smoother / residual / multigrid hot path of P-A_multigrids.
 *
 * The reference (serial Fortran 90) has no operator / plugin / FFI boundary: smoother,
 * get_residual, restrictor, prolongator and update_overlaps are procedures contained in or called
 * from Semi_implicit_iterative (transport_tri_semi.F90:319-379, :407-889).  This header IS the
 * boundary a Fortran host binds through ISO_C_BINDING (see INTEGRATION.md and
 * p-a_multigrids_b200/host/pamg_iface.F90).  Conventions:
 *   - plain pointers and sizes only; every entry returns int: 0 ok, <0 error
 *     (mirrors ierr / errorflag out-arguments, Msh2Tri.F90:137, matrices.F90:1631);
 *   - field layout at the boundary is the reference's column-major T(nloc=3, C, U), i.e. flat
 *     0-based index ((un-1)*C + (str-1))*3 + (iloc-1)  ==  glob_no_semi-1 (matrices.F90:1496-1500);
 *   - levels are 1-based like ilevel; level l has split s = n_split-l+1 and C = 4**s children
 *     per parent (transport_tri_semi.F90:180,324);
 *   - element / parent ids inside Neig are 1-based, 0 = domain boundary (Structures.F90:151);
 *   - the library owns all device memory; fields stay resident in HBM between calls;
 *   - one host thread per handle; there is NO CPU fallback: every compute entry needs a CUDA device.
 */
#ifndef PAMG_H
#define PAMG_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define PAMG_OK 0
#define PAMG_ERR_ARG (-1)
#define PAMG_ERR_CUDA (-2)
#define PAMG_ERR_STATE (-3)
#define PAMG_ERR_IO (-4)
#define PAMG_ERR_SINGULAR (-5) /* FINDInv errorflag = -1, matrices.F90:1665-1688 */
#define PAMG_ERR_UNSUPPORTED (-6)

/* Everything the reference hard-codes or passes as literal arguments (main.F90:46-47,
 * transport_tri_semi.F90:117-140).  Switches select LITERAL (HEAD) or INTENDED behaviour where the
 * reference is work in progress (SURVEY.md appendix B); nothing is "fixed" silently. */
typedef struct pamg_params {
  int32_t n_split;        /* transport_tri_semi.F90:118 */
  int32_t multi_levels;   /* main.F90:46; must be <= n_split (:120-123) */
  int32_t n_smooth;       /* main.F90:47 */
  int32_t n_multigrid;    /* main.F90:46 */
  int32_t n_coarse_smooth;/* 15 smoother calls on the coarsest level (:351) */
  int32_t solver;         /* 1 Jacobi, 2 Richardson, 3 Gauss-Seidel (two-colour ordering on the GPU) */
  int32_t face_terms;     /* 0: face loop body commented out as at HEAD (:619-688); 1: face block on */
  int32_t literal_source; /* 1: get_RHS sums M*src while overwriting src (:456); 0: plain M*src */
  int32_t transfer;       /* 0: restrictor/prolongator as written (splitting.F90:10-91); 1: P1 interpolation + transpose */
  int32_t residual_sign;  /* +1: r = A x - b (:869);  -1: r = b - A x */
  int32_t halo_rule;      /* 0: Dir/Nside reversal table (splitting.F90:1256-1391); 1: geometric pairing */
  int32_t coarse_bc_zero; /* 1: homogeneous Dirichlet data on levels > 1; 0: sin(x+y) on every level (HEAD) */
  int32_t keep_tnew_gs;   /* 1: the in-place GS sweep keeps tracer%tnew = start-of-last-sweep field (:550) by a device copy;
                             0: TNEW aliases the iterate after a GS smoother call (saves 16 B/DOF per call) */
  int32_t reserved;       /* keeps the doubles 8-byte aligned */
  double theta;           /* :117 (the reference's literal is 1.; 0 <= theta <= 1: get_A_x :444-446 and the old-time branch of get_RHS :459-460) */
  double dt;              /* :133  dt = CFL*dx */
  double k;               /* :136 */
  double omega;           /* :140 */
  double u_x, u_y;        /* :208-212 uniform velocity */
  double source_coef;     /* source = source_coef*sin(x+y); HEAD: -2k (:593) */
} pamg_params;

typedef struct pamg_handle pamg_handle;
typedef struct pamg_mesh pamg_mesh;

/* field ids: tracer(ilevel)%tnew/told/RHS/residuale (Structures.F90:185-188) and tnew_nonlin */
enum { PAMG_TNEW = 0, PAMG_TOLD = 1, PAMG_RHS = 2, PAMG_RES = 3, PAMG_TNONLIN = 5 };

const char* pamg_version(void);
int pamg_device_count(int* n);               /* PAMG_ERR_CUDA when no CUDA driver/device is present */
void pamg_default_params(pamg_params* p, int literal_head);

/* ---- host mesh pipeline (replaces ReadMSH + CheckNeig all-pairs search + getNeigDataMesh,
 *      Msh2Tri.F90:132-334,454-548,780-963, with an O(N) edge hash) ------------------------------ */
int pamg_mesh_read_msh(const char* path, pamg_mesh** out);
/* G right super-triangles (G/2 unit squares in a strip), each split kp times with the reference's own
 * get_splitting numbering (Msh2Tri.F90:69-107) into 4**kp parents: SURVEY 8(d) synthetic input */
int pamg_mesh_synthetic(int kp, int G, pamg_mesh** out);
int pamg_mesh_from_arrays(int U, const double* X /* [U][3][2] */, const int32_t* region, pamg_mesh** out);
/* structured triangles of str_explicit (transport_tri.F90:354; structured_meshgen.F90:190-298: tri_ele_info2,
 * str_tri_X_nodes): no_ele_row triangles per row (even), no_ele_col rows; feed it to pamg_set_unstructured */
int pamg_mesh_structured_tri(int no_ele_row, int no_ele_col, double dx, double dy, pamg_mesh** out);
int pamg_mesh_size(const pamg_mesh* m, int* U);
/* any output pointer may be NULL.  X [U][3][2]; neig/fneig/dir [U][3]; region [U] */
int pamg_mesh_get(const pamg_mesh* m, double* X, int32_t* neig, int32_t* fneig, int32_t* dir, int32_t* region);
void pamg_mesh_free(pamg_mesh* m);

/* ---- handle ------------------------------------------------------------------------------------ */
int pamg_create(const pamg_params* p, int device, pamg_handle** out);
/* One host thread driving ngpus devices (the reference's driver is one serial process, main.F90:16-51): devices[i] is the CUDA
 * device of part i (NULL = 0..ngpus-1; a device may appear more than once).  pamg_set_parents cuts the mesh into ngpus contiguous
 * blocks of parents (the scheme Generic.F90:387-401 sketches); every other entry takes and returns WHOLE-mesh arrays and fans out
 * inside the library.  The halo strips of cut faces travel by direct stores into the neighbour GPU's memory (peer access, no
 * library collective), norms are combined on the host, small coarse levels are agglomerated on part 0.  Entries that exist on a
 * single device only (unstructured front-ends, trans_rec, local inverse) run on part 0. */
int pamg_create_multi(const pamg_params* p, int ngpus, const int* devices, pamg_handle** out);
void pamg_destroy(pamg_handle* h);
const char* pamg_last_error(const pamg_handle* h);
/* Mesh%X, Neig, fNeig, Dir (Structures.F90:143-170).  Builds per-parent geometry for every level
 * (semi_tri_det_nlx_multigrid / semi_det_snlx_multigrid / get_d_center) and allocates the fields. */
int pamg_set_parents(pamg_handle* h, int U, const double* X, const int32_t* neig, const int32_t* fneig,
                     const int32_t* dir);
/* distributed run (one process per GPU): the mesh is cut into nparts contiguous blocks of parents,
 * part i owning [part_first[i], part_first[i+1]); this handle owns block my_part.  Faces cut by the
 * partition exchange their halo strips inside pamg_update_overlaps / pamg_smooth: direct stores into the
 * neighbour GPU's memory over NVLink (CUDA IPC, set up collectively at the first exchange), NCCL send/recv
 * where peer memory is not available. */
int pamg_set_parents_partition(pamg_handle* h, int U_global, const double* X, const int32_t* neig,
                               const int32_t* fneig, const int32_t* dir, int nparts, const int32_t* part_first,
                               int my_part);
/* Dirichlet data of the domain-boundary parent faces (Neig == 0), [U_global][3] in gmsh face order.  update_overlaps carries
 * a t_bc argument (splitting.F90:1210) that HEAD overwrites with boundary(x,y) = sin(x+y) (:1246-1252); this entry makes it
 * data: bc_kind 0 = sin(x+y) (the default everywhere), 1 = the constant bc_value[], 2 = open face (no data and no penalty term; only
 * for faces with n.u >= 0, else pamg_set_parents returns PAMG_ERR_UNSUPPORTED).  bc_value may be NULL (zeros).  Must precede
 * pamg_set_parents / pamg_set_parents_partition. */
int pamg_set_boundary_data(pamg_handle* h, int U_global, const int32_t* bc_kind, const double* bc_value);
int pamg_ndof(const pamg_handle* h, int level, int64_t* ndof);

int pamg_upload_field(pamg_handle* h, int field, int level, const double* host);
int pamg_download_field(pamg_handle* h, int field, int level, double* host);
int pamg_fill_field(pamg_handle* h, int field, int level, double fill_value);
int pamg_copy_field(pamg_handle* h, int level, int dst_field, int src_field);
int pamg_download_overlap(pamg_handle* h, int level, int old, double* host /* [U][3][2**s][3] */);
int pamg_device_ptr(pamg_handle* h, int field, int level, void** dptr); /* for zero-copy interop */

/* ---- the hot path ------------------------------------------------------------------------------ */
/* update_overlaps (splitting.F90:1210-1397): halo strips from TNEW/TOLD of the level */
int pamg_update_overlaps(pamg_handle* h, int level);
/* level-1 RHS = (1/dt) M told + M src - (1 - theta)(-stiff + flux + diff_vol + diff_surf) told (get_RHS,
 * transport_tri_semi.F90:452-464); with theta != 1 the RES field is the scratch of the old-time pass */
int pamg_build_rhs(pamg_handle* h);
/* smoother (:543-722): nsweeps sweeps on TNONLIN; each sweep does TNEW <- TNONLIN (:550), halo (:555),
 * then one Jacobi / Richardson / two-colour GS update of every child */
int pamg_smooth(pamg_handle* h, int level, int solver, int nsweeps);
/* get_residual (:725-873) on TNEW with the current halo strips; norms of RES by warp-shuffle reduction */
int pamg_residual(pamg_handle* h, int level, double* l2, double* linf);
int pamg_convergence(pamg_handle* h, int level, double* conv);   /* get_convergence (:876-889), signed max */
int pamg_restrict(pamg_handle* h, int fine_level);               /* restrictor, splitting.F90:10-32 */
int pamg_prolong(pamg_handle* h, int fine_level);                /* prolongator, splitting.F90:38-91 */
/* V-cycles of the INTENDED composition until ||r||2/||r0||2 <= tol; hist gets max_cycles+1 norms */
int pamg_vcycle_solve(pamg_handle* h, int solver, int nu1, int nu2, int ncoarse, int max_cycles, double tol,
                      int* cycles, double* hist);
/* one itime of the HEAD loop (:316-379), every quirk included */
int pamg_literal_timestep(pamg_handle* h, int solver, int n_multigrid, int n_smooth);
/* whole reference-facing time step with HOST buffers: upload tnew, told=tnew, solve, download tnew */
int pamg_timestep_host(pamg_handle* h, const double* tnew_in, double* tnew_out, int max_cycles, double tol,
                       int* cycles, double* relres);

/* smoother with HOST buffers, blocking like the reference's call (transport_tri_semi.F90:331): upload tnew_in, nsweeps sweeps,
 * download into tnew_out; both buffers are free again when it returns. */
int pamg_smoother_host(pamg_handle* h, int solver, int nsweeps, const double* tnew_in, double* tnew_out);
/* the same, ASYNCHRONOUS and pipelined across calls (pinned memory required for any overlap): the call returns once the
 * work is queued.  tnew_in must stay untouched and tnew_out is not valid until pamg_sync has returned.  The upload of
 * call k+1 overlaps the sweeps and the download of call k - unless tnew_in overlaps the tnew_out of the previous call (a
 * dependent loop, or one buffer for both), in which case the library orders the upload after that download.  Any other
 * entry that reads or writes level-1 fields must be preceded by pamg_sync. */
int pamg_smooth_host(pamg_handle* h, int solver, int nsweeps, const double* tnew_in, double* tnew_out);

/* host-only (no CUDA needed): the folded operator of ONE parent on the level with split s - the table the sweep kernels read.
 * It replaces the per-sweep stencil set-up of get_un_ele_mass_stiff_diffvol / get_diff_surf_stencl / get_diagonal
 * (ShapFun_unstruc.F90:304-335, transport_tri_semi.F90:468-486,575-609) with closed forms evaluated once per parent and level.
 * table[88]: [0] A/(12 dt); [1..6] K11 K12 K13 K22 K23 K33; [7..9] advection; [10..12] upwind flux per child face;
 * [13..15] / [19..21] penalty of faces inside / on the boundary of the parent; [16..18] omega/D of interior children;
 * [24..39], [40..55] folded 3x3 operator + 3 neighbour couplings + omega/D of up / down children; [56..58] penalty change and
 * [60..83] omega/D per face mask for children on parent faces.  parent is 0-based; bc_kind may be NULL (pamg_set_boundary_data);
 * theta_weight multiplies every spatial term (p->theta for the operator of the sweeps, 1 - p->theta with with_mass = 0 for the
 * old-time branch of get_RHS).  Returns PAMG_ERR_UNSUPPORTED for an open boundary face with inflow. */
int pamg_parent_table(const pamg_params* p, int U, const double* X, const int32_t* neig, const int32_t* bc_kind, int parent,
                      int s, double theta_weight, int with_mass, double* table);

/* host-only (no CUDA needed): the closed-form child numbering of the kernels, which replaces the tables of get_str_info,
 * get_str_neig_multigrid and element_conversion (Msh2Tri.F90:32-60, splitting.F90:97-140,732-776).  The SAME functions are
 * compiled for the device; this entry evaluates them on the host for indices first .. first+count-1, out is [count][4]:
 *   what 0: child k (0-based, memory order = element id - 1) at split s -> row, position, row length, 0   (child_from_ele0)
 *   what 1: paired-row index t (rows r and 2^s+1-r share 2^(s+1) slots) -> row, position, element id (1-based), row length
 *   what 2: coarse child k (0-based) at split s -> element ids (1-based) of its four fine children fin(1..4) at split s+1
 *   what 3: row, position of child k + 256 obtained by WALKING from those of child k (child_advance), row length, 0 */
int pamg_numbering(int what, int s, int64_t first, int64_t count, int32_t* out);

/* ---- distributed halo (update_overlaps across GPUs; Generic.F90:387-401 sketches the block partition) -- */
/* host-only: where every halo strip lives and how cut faces are ordered per peer (no CUDA needed).
 * arrays are [U_local*3]; peers is [npeers][4] = part, nfaces, strip_begin, send_begin;
 * counts = npeers, nstrips, nsend, U_local, first */
int pamg_halo_plan(int U_global, const double* X, const int32_t* neig, const int32_t* fneig, const int32_t* dir,
                   int halo_rule, int nparts, const int32_t* part_first, int my_part, int32_t* strip_of,
                   int32_t* dst_strip, int32_t* rev, int32_t* hmap, int32_t* peers, int32_t* counts);
/* host-only: where a sweep reads the exterior values of the parent faces of part my_part WITHOUT a halo strip, on the level with
 * split s.  src is [U_local*3][2**s][2]: for (parent, gmsh side, strip position) the offsets (in doubles, inside the part's
 * field T(3, C, U_local)) of the neighbour's values at the nodes coincident with my face nodes (a, b) - what update_overlaps
 * (splitting.F90:1255-1391) would have copied into my strip and the face block would pick out of it - or -1, -1 where the values
 * come from a strip (Dirichlet data, faces cut by the partition).  The decoding is the function the kernels use. */
int pamg_halo_sources(int U_global, const double* X, const int32_t* neig, const int32_t* fneig, const int32_t* dir,
                      int halo_rule, int nparts, const int32_t* part_first, int my_part, int s, int64_t* src);
int pamg_comm_unique_id(char* id128);                        /* rank 0: ncclGetUniqueId */
int pamg_comm_init(pamg_handle* h, const char* id128, int nranks, int rank);
int pamg_halo_peer_count(const pamg_handle* h, int* npeers);
int pamg_halo_peer_info(const pamg_handle* h, int idx, int* peer_part, int* nfaces);

/* host-only: flow levels of an upwind graph (the function pamg_implicit_set_precond's sweep uses).  Edge c -> e for every face
 * f of e with bit f of inflow_mask[e] set and a neighbour c = neig[e][f] - 1 (neig [E][3], 1-based, 0 = boundary).  level[e] =
 * the longest upwind path ending at e (Kahn's algorithm, O(E)); order [E] = the elements sorted by (level, index).  A cycle:
 * when no element is left whose upstream neighbours all have a level, the lowest-index element left gets 1 + the largest
 * level of its upstream neighbours that have one (0 if none), and its other upstream edges are lagged.  lagged = the number
 * of edges (c, e) with level[c] >= level[e]: 0 for an acyclic graph.  nlevels = 1 + the largest level; nlevels and lagged
 * may be NULL. */
int pamg_flow_levels(int E, const int32_t* neig, const int32_t* inflow_mask, int32_t* level, int32_t* order,
                     int32_t* nlevels, int64_t* lagged);

/* ---- unstructured explicit DG step (unstr_explicit, transport_tri_unstr.F90:588-795) ------------ */
int pamg_set_unstructured(pamg_handle* h, int E, const double* X, const int32_t* neig, const int32_t* fneig);
int pamg_unstr_upload(pamg_handle* h, const double* tnew /* (3,E) */);
int pamg_unstr_download(pamg_handle* h, double* tnew);
/* u_ele(2,3,E) of transport_tri_unstr.F90 in the reference's layout: flat index (e*3 + iloc)*2 + d, HOST array.
 * NULL returns to the uniform velocity.  While a field is set, the u_x, u_y arguments of pamg_explicit_step,
 * pamg_implicit_assemble(_diffusion) and pamg_unstr_stab are not used: in the reference they only fill u_ele.
 * Needs pamg_set_unstructured first (else PAMG_ERR_STATE); pamg_set_unstructured clears the field.  Setting or clearing it
 * makes the assembled operator stale: pamg_implicit_step, _apply, _get_bsr and _set_stab return PAMG_ERR_STATE until the
 * next pamg_implicit_assemble*.  The face flux takes its upwind choice per Gauss point from the two traces
 * (income(s) = 1/2 + 1/2 sign(1, -n.(u + u2)/2)); where n.u changes sign along a face, the inflow point's part goes into the
 * neighbour's columns and the outflow point's into the element's own (HEAD picks one block per face from income(1)). */
int pamg_unstr_set_velocity(pamg_handle* h, const double* u_ele);
/* Boundary data of the domain-boundary faces (neig == 0) of the unstructured mesh, [E][3] in gmsh face order.  The codes are
 * those of pamg_set_boundary_data: bc_kind 0 = sin(x+y) at the face's two nodes, 1 = the values bc_value[e][f][0..1] at the
 * face nodes (l1, l2) = (1,3), (2,1), (3,2), linear along the face (NULL = zeros), 2 = open (no data, no penalty term; refused
 * where a Gauss point of the face has inflow with a non-zero flux).  Entries of interior faces are ignored.  bc_kind = NULL
 * returns to HEAD (no exterior trace on boundary faces: sn2 = 0).  With data, the face term of pamg_explicit_step and of the
 * implicit operator takes its exterior trace g_s = sn(s,1) g1 + sn(s,2) g2 from the data and its exterior velocity from the
 * element (u_bc = u_ele): an inflow Gauss point (the assembly's upwind rule) adds -c_s sn(s,.) g_s, c_s = sdetwei n.u_s, and
 * with k > 0 the penalty adds k (L/2)/dx sum_s sn(s,.) g_s, both to the right-hand side of the implicit solve (computed by
 * the assembly, added to (M/dt) told every time step) or to rhs of the explicit step.  An open face has no penalty term in
 * the operator either.  t_bc of pamg_explicit_step stays the exterior value of the faces without data (a boundary face given
 * fNeig >= 1 keeps HEAD's treatment too).
 * Needs pamg_set_unstructured first (else PAMG_ERR_STATE), which clears the data.  E must be the mesh's E and every kind
 * on a boundary face 0..2 (else PAMG_ERR_ARG, nothing changed).  Setting or clearing the data makes the assembled operator
 * stale like pamg_unstr_set_velocity: pamg_implicit_step, _apply, _get_bsr, _set_stab, _precond_apply and _flow_levels
 * return PAMG_ERR_STATE until the next pamg_implicit_assemble*.  An open face with inflow is refused with
 * PAMG_ERR_UNSUPPORTED by the next assembly (the operator stays unassembled) or explicit step; pamg_last_error names the
 * element and face.  The data adds no upwind edges: the flow levels of pamg_implicit_set_precond do not change.  On a
 * multi-GPU handle it acts on part 0 like every unstructured entry. */
int pamg_unstr_set_boundary(pamg_handle* h, int E, const int32_t* bc_kind, const double* bc_value);
/* ntime x nits nonlinear iterations; njac_its Jacobi iterations on M x = M told + dt rhs, or the exact
 * register-resident local inverse when use_exact_minv != 0 (transport_rect.F90:277-291) */
int pamg_explicit_step(pamg_handle* h, double dt, double u_x, double u_y, double t_bc, int ntime, int nits,
                       int njac_its, int use_exact_minv, int use_dir);

/* ---- unstructured implicit operator in block-CSR (unstr_implicit, transport_tri_unstr.F90:214-387) --
 * Replaces add_to_CSR / add_to_CSR_flux / make_sparse_matrix_flux (matrices.F90:12-161), csr_to_dense and the dense
 * FINDInv of the whole (3E)^2 matrix (:366-378).  Row e holds 4 blocks of 3x3 (row-major): block 0 = own columns
 * (mass/dt - stiffness + outflow flux), block 1+f = inflow flux of gmsh face f+1 in the neighbour's columns.
 * Needs pamg_set_unstructured first.  The time loop works on the field of pamg_unstr_upload / _download. */
int pamg_implicit_assemble(pamg_handle* h, double dt, double u_x, double u_y, int use_dir);
/* the same with the diffusion operator of the iterative path (get_A_x, transport_tri_semi.F90:412-448, face block on): the
 * volume block k A grad(phi_i).grad(phi_j) (ShapFun_unstruc.F90:324-335) on the diagonal and the penalty term
 * (k/dx) int sn_i (T - T2) (matrices.F90:84-115) on the own and the neighbour's columns, dx = centroid distance (centre ->
 * edge midpoint on the domain boundary, where the exterior trace is right-hand-side data).  The reference's implicit drivers
 * compute add_diffusion_vol and drop it (transport_tri_semi.F90:1627); this is the intended operator. */
int pamg_implicit_assemble_diffusion(pamg_handle* h, double dt, double u_x, double u_y, double k, int use_dir);
int pamg_implicit_get_bsr(pamg_handle* h, double* val /* [E][4][9] or NULL */, int32_t* col /* [E][4], 0-based, -1 = none, or NULL */);
int pamg_implicit_apply(pamg_handle* h, const double* x /* host (3,E) */, double* y /* host: (lhs + flux) x */);
/* ntime x nits passes of: told = tnew ; solve (lhs + flux) tnew = (M/dt) told by BiCGStab, right-preconditioned with the
 * preconditioner of pamg_implicit_set_precond (block Jacobi by default), to ||r|| <= tol ||rhs|| (at most max_iters
 * iterations per solve).  iters_total / relres (worst solve) may be NULL. */
int pamg_implicit_step(pamg_handle* h, int ntime, int nits, double tol, int max_iters, int* iters_total, double* relres);
/* measurement aids: average device time (ms) of `reps` block-CSR products; host synchronisations of the Krylov solves so far
 * (the scalars of the recurrence live on the device: one look at the convergence flag per 16 iterations) */
int pamg_implicit_spmv_time(pamg_handle* h, int reps, float* ms);
int pamg_implicit_host_syncs(pamg_handle* h, int64_t* n);

/* ---- preconditioner of the implicit solve ------------------------------------------------------------------------------
 * PAMG_PREC_BLOCK_JACOBI (default): the inverse diagonal 3x3 blocks.  PAMG_PREC_FLOW_GS: one block Gauss-Seidel pass in flow
 * order (a transport sweep), M = D + L with L = every stored off-diagonal block (e, c) whose column element c has a lower
 * flow level than e.  Levels come from the upwind graph of the assembled velocity: e depends on its neighbour c across face
 * f when a Gauss point of f is inflow for e (the assembly's upwind rule) with a non-zero flux; level[e] = the longest upwind
 * path ending at e.  With pure advection and an acyclic graph M is the operator itself and BiCGStab stops after one
 * iteration; diffusion blocks to neighbours of the same or a higher level, and the edges that close a cycle of a nodal
 * field, are lagged (left out of M).  One sweep is one kernel launch whose cost grows with the number of levels.
 * Needs pamg_set_unstructured first (else PAMG_ERR_STATE); an unknown kind is PAMG_ERR_ARG.  May be called before or after
 * assembly; the choice survives pamg_set_unstructured.  The levels are built when first needed (the next
 * pamg_implicit_step, _precond_apply or _flow_levels) and rebuilt after pamg_set_unstructured, pamg_unstr_set_velocity, an
 * assembly with a different u_x / u_y (uniform velocity) or, with a field, a different use_dir; dt, k and the
 * stabilisation keep them.  On a multi-GPU handle it acts on part 0 like every unstructured entry. */
#define PAMG_PREC_BLOCK_JACOBI 0
#define PAMG_PREC_FLOW_GS 1
int pamg_implicit_set_precond(pamg_handle* h, int kind);
/* y = M^-1 x with the selected preconditioner, once (x, y host (3,E)); a timed-out sweep returns PAMG_ERR_CUDA and
 * pamg_last_error names k_flow_sweep.  Needs an assembled operator (else PAMG_ERR_STATE). */
int pamg_implicit_precond_apply(pamg_handle* h, const double* x, double* y);
/* the flow levels of the assembled velocity (built here if stale): level [E] (may be NULL), the number of levels and the
 * number of lagged upwind edges.  Needs an assembled operator (else PAMG_ERR_STATE). */
int pamg_implicit_flow_levels(pamg_handle* h, int32_t* level, int32_t* nlevels, int64_t* lagged);
/* measurement aid: average device time (ms) of `reps` flow sweeps on the work vectors, and the host time (ms) of the last
 * level build: setup_ms[0] mask kernel + download, [1] pamg_flow_levels, [2] upload (setup_ms may be NULL) */
int pamg_implicit_flow_time(pamg_handle* h, int reps, float* ms, double* setup_ms);

/* ---- Petrov-Galerkin residual-based stabilisation (transport_tri_unstr.F90:239-267,278; semi_str_implicit.F90:290-318) --
 * diff_coe(gi) and stab(iloc,jloc) of every element from tnew = the field of pamg_unstr_upload and the given told.
 * HEAD computes stab and never applies it (:367-368 are commented out); pamg_implicit_set_stab(h, 1) applies it the
 * intended way: every nonlinear pass of pamg_implicit_step adds stab(tnew_nonlin, told) to the diagonal blocks. */
int pamg_unstr_stab(pamg_handle* h, const double* told /* host (3,E) */, double dt, double u_x, double u_y,
                    double* diff_coe /* host (3,E) or NULL */, double* stab /* host [E][3][3] or NULL */);
int pamg_implicit_set_stab(pamg_handle* h, int with_stab);

/* ---- trans_rec front-end (transport_rect.F90:7-380): explicit DG on bilinear quadrilaterals of a structured
 * no_ele_row x no_ele_col grid over x_length x y_length, dt = CFL dx, ntime = int(time / dt) steps of nits passes; initial
 * box pulse of :83, t_bc = 0.  direct_solver != 0: FINDInv of the 4x4 mass matrix, else njac_its Jacobi iterations on the
 * lumped mass.  volume_term = 0 reproduces HEAD (tnew_gi is never set, :157: no advection volume integral - the version
 * that wrote the shipped DG-rectangular_structured), 1 is the intended scheme.  x_all [totele][4][2] (may be NULL) and
 * tnew [totele][4] are HOST arrays in the order of the reference's dump (:320-330). */
int pamg_trans_rec(pamg_handle* h, double CFL, int no_ele_row, int no_ele_col, double x_length, double y_length, double u_x,
                   double u_y, double time, int nits, int njac_its, int direct_solver, int volume_term, double* x_all,
                   double* tnew, int* ntime);

/* ---- batched element-local inverse (FINDInv, matrix_inversion.F90:50-148) ----------------------- */
/* M, x, rhs on the HOST; n in {3,4,6}; M row-major [batch][n][n].  x = M^-1 rhs (Minv optional out).
 * status[b] = 0 or -1 (singular) like errorflag. */
int pamg_apply_local_minv(pamg_handle* h, int n, int batch, const double* M, const double* rhs, double* x,
                          double* Minv, int32_t* status);

/* ---- output (get_vtu, get_vtk_files.F90:10-140; call site transport_tri_semi.F90:299-312) ---------------------
 * level-1 child coordinates x_all_str (2,3,C*U) (:274), analytical = sin(x+y) (:278) and get_error = |tnew - analytical|
 * (:531-540), computed on the device; any pointer may be NULL. */
int pamg_output_fields(pamg_handle* h, double* x_all, double* analytical, double* error);
/* one .vtu piece of level 1 with the reference's arrays (<solve_for>, error, analytical; points; triangles).
 * binary = 0: ASCII in the reference's layout and number formats (F12.10 / F10.7 / F10.3, one value per line);
 * binary = 1: raw appended Float64 (SURVEY 8(f4)). */
int pamg_write_vtu(pamg_handle* h, const char* path, const char* solve_for, int binary);

/* ---- timing helpers (CUDA events on the handle's stream) ---------------------------------------- */
int pamg_sync(pamg_handle* h);
int pamg_event_record(pamg_handle* h, int slot);       /* slot 0..15 */
int pamg_event_elapsed_ms(pamg_handle* h, int slot_a, int slot_b, float* ms);
int pamg_launch_count(const pamg_handle* h, int64_t* n); /* kernels launched by this handle so far */
int pamg_flush_l2(pamg_handle* h);                     /* writes a 256 MiB scratch buffer */
/* per-kernel device time of the element kernels (Jacobi / GS / residual): CUDA events recorded on the
 * launching stream around each launch while profiling is on (at most 1024 launches are kept) */
int pamg_profile(pamg_handle* h, int on);
int pamg_profile_read(pamg_handle* h, double* total_ms, int* launches);
/* pinned host memory for the HOST-buffer entry points */
int pamg_host_alloc(void** p, int64_t bytes);
int pamg_host_free(void* p);

#ifdef __cplusplus
}
#endif
#endif
