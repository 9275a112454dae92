/*
 * parelag_b200_api.h -- C facade over the C++ mirror of ParElag's solver API
 * (the headers under parelag_b200/src: ParameterList-driven SolverLibrary / SolverFactory,
 * mfem::Solver::Mult, DeRhamSequence coarse-operator interface).  It exists so that
 * non-C++ hosts (the ctypes tests, bench.py, a C driver) can drive exactly the code
 * path a C++ ParElag driver drives:
 *
 *     lib   = SolverLibrary::CreateLibrary(master_list.Sublist("Preconditioner Library"))
 *     fact  = lib->GetSolverFactory(name)              examples/MultigridTest2Form.cpp:519-523
 *     state->SetDeRhamSequence / SetBoundaryLabels / SetForms
 *     solver = fact->BuildSolver(A, *state)            :537
 *     solver->Mult(B, X)                               :578
 *
 * Return codes and pe_last_error() as in parelag_b200.h; C++ exceptions are caught
 * at this boundary and turned into error codes.
 */
#ifndef PARELAG_B200_API_H
#define PARELAG_B200_API_H
#include "parelag_b200.h"
#include "parelag_b200_par.h"
#ifdef __cplusplus
extern "C" {
#endif

typedef struct pe_sequence pe_sequence; /* a chain of DeRhamSequence levels (fine -> coarse) */
typedef struct pe_solver pe_solver;     /* an mfem::Solver built by a SolverFactory          */

/* process-wide session (parelag::mpi_session): one rank <-> one GPU */
int pe_api_session_create(int rank, int nranks, int device, const void *nccl_unique_id);
int pe_api_session_destroy(void);
pe_ctx *pe_api_session_ctx(void);

/* DeRhamSequence levels with externally supplied operators (the role
 * DeRhamSequenceAlg plays for levels produced by Coarsen()).  P(level, form) maps
 * level+1 -> level; D(level, form) maps form -> form+1 on that level; bdr_mask bit a
 * marks dofs lying on facets with boundary attribute a+1 (DofHandler::MarkDofsOnSelectedBndr). */
int pe_api_sequence_create(int nforms, int nlevels, pe_sequence **out);
int pe_api_sequence_set_P(pe_sequence *s, int level, int form, int nrows, int ncols,
                          const int32_t *I, const int32_t *J, const double *A);
int pe_api_sequence_set_D(pe_sequence *s, int level, int form, int nrows, int ncols,
                          const int32_t *I, const int32_t *J, const double *A);
int pe_api_sequence_set_bdr_mask(pe_sequence *s, int level, int form, int ndofs, const uint32_t *mask);
int pe_api_sequence_free(pe_sequence *s);

/* The full coarsening path on a structured hexahedral mesh (synthetic input of the named
 * shape): AgglomeratedTopology + MFEMRefinedMeshPartitioner + CoarsenLocalPartitioning,
 * DeRhamSequence3D_FE at lowest order with the upscaling targets, then
 * sequence[i+1] = sequence[i]->Coarsen() (examples/MultigridTest2Form.cpp:248-375).
 * alpha/beta: optional per-element weights of the L2 / H(div) element mass matrices.
 * svd_tol < 0: build the topology hierarchy and the fine sequence only (host integer work,
 * no GPU needed). */
int pe_api_hexsequence_create(int nx, int ny, int nz, double Lx, double Ly, double Lz,
                              const double *alpha, const double *beta, int jform_start, int nlevels,
                              double svd_tol, pe_sequence **out);
/* The same on trilinear hexahedra: vertex_xyz[nv x 3] (index-grid numbering, x fastest) replaces the axis-aligned
 * vertices -- the geometry of examples/3DHdivWeakScaling.cpp:148-158 and 3DHcurlWeakScaling.cpp.  The mass matrices of
 * all four forms are built by quadrature (mfem's rules: DeRhamSequenceFE.cpp:633-684, bilinIntegrators.cpp:64-157). */
int pe_api_hexsequence_create_deformed(int nx, int ny, int nz, const double *vertex_xyz, const double *alpha,
                                       const double *beta, int jform_start, int nlevels, double svd_tol, pe_sequence **out);
/* Diagonal tensor coefficient in the H(div) element mass matrices (a VectorFunctionCoefficient in VectorFEMassIntegrator,
 * examples/MultigridTestSPE10.cpp:377-395): beta_xyz[3 * element + axis]; axis-aligned cells. */
int pe_api_hexsequence_create_tensor(int nx, int ny, int nz, double Lx, double Ly, double Lz, const double *alpha, const double *beta_xyz,
                                     int jform_start, int nlevels, double svd_tol, pe_sequence **out);
/* The SPE10 permeability data set as the reference reads and evaluates it (src/SPE10/InversePermeabilityFunction.cpp;
 * class InversePermeabilityFunction in parelag_b200/src/spe10.hpp, process-wide state like the reference's statics):
 * pe_api_spe10_read = SetNumberCells + SetMeshSizes + ReadPermeabilityFile (the Nx x Ny x Nz corner of the 60 x 220 x 85
 *   file with the three blocks K_x, K_y, K_z; reciprocals are stored; with a host communicator rank 0 reads and all receive);
 * pe_api_spe10_set_constant = SetConstantInversePermeability; pe_api_spe10_set_slice = Set2DSlice (0 none, 1 XY, 2 XZ, 3 YZ);
 * pe_api_spe10_inverse_permeability = InversePermeability at npoints points (out: npoints x 3; the data set's x and z
 *   axes run against the mesh axes, :141-178); pe_api_spe10_data = the stored array (3 Nx Ny Nz numbers);
 * pe_api_hexsequence_create_spe10 = the driver's mesh (nx x ny x nz cells of size hx x hy x hz) with the loaded inverse
 *   permeability as the tensor coefficient of the H(div) mass matrix, then the coarsening path as above. */
int pe_api_spe10_read(const char *perm_file, int Nx, int Ny, int Nz, double hx, double hy, double hz);
int pe_api_spe10_set_constant(int Nx, int Ny, int Nz, double hx, double hy, double hz, double ipx, double ipy, double ipz);
int pe_api_spe10_set_slice(int orientation, int npos);
int pe_api_spe10_inverse_permeability(const double *xyz, int npoints, double *out);
int pe_api_spe10_data(double *out, int64_t *count);
int pe_api_hexsequence_create_spe10(int nx, int ny, int nz, double hx, double hy, double hz, int jform_start, int nlevels, double svd_tol,
                                    pe_sequence **out);
/* Options of the topology coarsening inside the sequence builders below and above (process-wide; what the reference's
 * drivers take from their command lines):
 *   partitioner 0 = derefinement by parent element (MFEMRefinedMeshPartitioner.cpp:48-90; logical Cartesian blocks on
 *     grids that are not a multiple of two, LogicalPartitioner.hpp:46-103) -- the default;
 *   1 = GeometricBoxPartitioner::doPartition (src/partitioning/GeometricBoxPartitioner.cpp:20-79; two levels,
 *     num_partitions = elements / 16 as in testsuite/UpscalingGeneralForm.cpp:249-256,367-385 --geometric);
 *   2 = element_partitioning[n] as given (two levels; testsuite/twentyseven.cpp:262-288);
 *   3 = LogicalPartitioner with LogicalCartesianMaterialId (src/partitioning/LogicalPartitioner.hpp:46-128,
 *     CartesianPartitioner.hpp:133-150; examples/LogicalPartitionerDemo.cpp:203-226): element_partitioning[n] holds the
 *     material id (element attribute) of every fine hexahedron; agglomeration by 2 x 2 x 2 logical blocks that keeps the
 *     material ids apart, on every level.
 *   check_topology = second argument of AgglomeratedTopology::CoarsenLocalPartitioning (Topology.cpp:685-739, 421-434):
 *     report, mark and de-agglomerate agglomerated elements / facets / ridges that are disconnected, have holes or
 *     tunnels or a pinched boundary (src/topology/AgglomeratedTopologyCheck.cpp).  Disconnected element partitions are
 *     always split and empty ones removed (connectedComponents.cpp:23-87), as in the reference.
 * pe_api_topology_log: the lines the reference prints during the topology coarsening (same text), collected since the
 *   options were last set, newline separated; *needed = bytes including the terminator (call with buf = NULL first).
 * pe_api_sequence_show_topology: AgglomeratedTopology::ShowMe of one level (Topology.cpp:310-352: entity counts and
 *   Euler characteristic). */
int pe_api_set_topology_options(int partitioner, int check_topology, const int32_t *element_partitioning, int n);
int pe_api_topology_log(char *buf, int64_t capacity, int64_t *needed);
int pe_api_sequence_show_topology(pe_sequence *s, int level, char *buf, int64_t capacity, int64_t *needed);
/* Unstructured tetrahedral meshes (BASELINE configs[0], examples/MultigridTest0Form.cpp:147-375 on meshes/cube456.mesh):
 * the given mesh (0-based vertex numbers; boundary triangles with 1-based attributes) is refined nref times (red
 * refinement, children of element e = 8e .. 8e+7), the finest mesh is level 0 of the sequence and the nlevels - 1 <= nref
 * coarser levels are built by derefinement agglomeration (MFEMRefinedMeshPartitioner.cpp:48-66) and Coarsen().
 * Lowest-order Whitney forms with MFEM's dof meaning; mass matrices in closed form (parelag_b200/src/amge_tet.hpp).
 * pe_api_tetsequence_create_from_file reads the NETGEN neutral format of meshes/cube456.mesh or MFEM's own "MFEM mesh v1.0"
 * format (straight-sided tetrahedra), recognised from the first line like mfem::Mesh(imesh, 1, 1). */
int pe_api_tetsequence_create(int nv, const double *vertex_xyz, int nel, const int32_t *tets, int nbdr, const int32_t *bdr_triangles,
                              const int32_t *bdr_attributes, int nref, int nlevels, int jform_start, double svd_tol, pe_sequence **out);
int pe_api_tetsequence_create_from_file(const char *mesh_file, int nref, int nlevels, int jform_start, double svd_tol, pe_sequence **out);
/* ---- multi-rank (one rank <-> one box of a P0 x P1 x P2 box decomposition <-> one GPU).
 * pe_api_session_set_host_comm: the setup-time host communicator (MPI_Comm in the reference).
 * pe_api_hexsequence_create_par: as pe_api_hexsequence_create for THIS rank's box (nx,ny,nz hexahedra
 *   of extent Lx,Ly,Lz); builds the dof <-> true-dof SharingMaps of every level.
 * pe_api_sequence_get_dofmap: DofHandler::GetDofTrueDof -- global true id / owner / global key of
 *   every local dof (arrays may be NULL).
 * pe_api_sequence_true_operator: DeRhamSequence::ComputeTrueP / ComputeTrueD as a device ParCSR. */
int pe_api_session_set_host_comm(const pe_host_comm *comm);
int pe_api_hexsequence_create_par(const int32_t *procs, int nx, int ny, int nz, double Lx, double Ly, double Lz,
                                  const double *alpha, const double *beta, int jform_start, int nlevels,
                                  double svd_tol, pe_sequence **out);
/* The box decomposition on trilinear hexahedra (examples/3DHdivWeakScaling.cpp:113-158: one box per rank, vertices moved
 * after the refinement): vertex_xyz[nv x 3] are the vertices of THIS rank's box; copies of an interface vertex must be
 * bitwise equal on all ranks that hold it. */
int pe_api_hexsequence_create_par_deformed(const int32_t *procs, int nx, int ny, int nz, const double *vertex_xyz,
                                           const double *alpha, const double *beta, int jform_start, int nlevels,
                                           double svd_tol, pe_sequence **out);
int pe_api_sequence_get_dofmap(pe_sequence *s, int level, int form, int32_t *ndofs, int64_t *gid, int32_t *owner,
                               int64_t *key, int64_t *true_start, int64_t *true_count, int64_t *global_count);
/* SharingMap::Assemble (direction 0: local dof vector -> true dof vector, copies of a shared dof summed on its
 * owner, SharingMap.cpp:768-780) / SharingMap::Distribute (direction 1: true -> local, :664-677), host vectors */
int pe_api_sequence_dofmap_apply(pe_sequence *s, int level, int form, int direction, const double *in, double *out);
int pe_api_sequence_true_operator(pe_sequence *s, int level, const char *what, int form, const int32_t *ess_attr,
                                  int nattr, pe_mat **out);

/* Introspection for parity tests.  what = "P" (a=form), "D" (a=form), "M" (a=form: assembled
 * mass operator), "Me" (a=form, b=codim: block-diagonal entity mass matrices), "B" (a=codim),
 * "AE" (a=codim: agglomerated entity -> entity), "ED" (a=form, b=codim: entity -> dof),
 * "FB" (facet -> boundary attribute).  Call with I=J=A=NULL to get the sizes. */
int pe_api_sequence_get_csr(pe_sequence *s, int level, const char *what, int a, int b,
                            int32_t *nrows, int32_t *ncols, int64_t *nnz, int32_t *I, int32_t *J, double *A);
int pe_api_sequence_get_targets(pe_sequence *s, int level, int form, int32_t *ndofs, int32_t *ntargets, double *out);
int pe_api_sequence_get_bdr_mask(pe_sequence *s, int level, int form, int32_t *ndofs, uint32_t *mask);
/* DeRhamSequence::CheckInvariants (DeRhamSequence.cpp:694-970) of one level against the next coarser one: D non-zero,
 * D_{j+1} D_j = 0, D_f P_j = P_{j+1} D_c, M_c = P^T M_f P (levels that hold their mass matrices).  Non-zero return with the
 * violated identity in pe_last_error(); *worst = the largest residual met.  Host work. */
int pe_api_sequence_check_invariants(pe_sequence *s, int level, double *worst);
int pe_api_sequence_get_stat(pe_sequence *s, int level, const char *name, int64_t *value);
/* System assembly as in the drivers (examples/MultigridTest{0,1,2}Form.cpp:443-475), on the
 * device: A = [M_form +] D^T M_{form+1} D  (the mass term is skipped for form 0), essential
 * rows/cols eliminated with unit diagonal.  Returns a device matrix owned by the caller. */
int pe_api_sequence_assemble_system(pe_sequence *s, int level, int form, const int32_t *ess_attr, int nattr,
                                    pe_mat **out);

/* Mixed (Darcy) system [[M Bt][B 0]] (examples/MultigridTestDarcy.cpp): M = mass of H(div), B = W D_2 with
 * W = mass of L2, Bt = B^T, as device matrices owned by the caller (single rank). */
int pe_api_sequence_assemble_darcy(pe_sequence *s, int level, pe_mat **M, pe_mat **B, pe_mat **Bt);
/* BuildSolver on an MfemBlockOperator: blocks[nblocks*nblocks] row-major, NULL = zero block; ownership of the
 * device matrices passes to the solver (the array entries are set to NULL).  forms[nblocks];
 * ess_attr[nblocks*nattr] (one marker row per block) or NULL. */
int pe_api_solver_build_block(const char *xml_library, const char *solver_name, int nblocks, pe_mat **blocks,
                              pe_sequence *seq, int start_level, const int32_t *forms, const int32_t *ess_attr,
                              int nattr, pe_solver **out);

/* Introspection of the ParameterList machinery (SimpleXMLParameterListReader::GetParameterList,
 * src/utilities/ParELAG_SimpleXMLParameterListReader.cpp:55-297; SolverLibrary::GetSolverFactory):
 * pe_api_parameterlist_dump: every parameter of the parsed document as "path/name<TAB>type<TAB>value", one per line, sorted;
 * pe_api_library_factories: every entry of the "Preconditioner Library" sublist (or of the document itself) as
 *   "name<TAB>Type<TAB>ok" when its factory can be created and initialised (nested factories included), else
 *   "name<TAB>Type<TAB>error: ..." -- e.g. the hypre / direct black-box types that are outside the GPU path.
 * *needed = bytes including the terminator (call with buf = NULL first).  No device needed. */
int pe_api_parameterlist_dump(const char *xml, char *buf, int64_t capacity, int64_t *needed);
int pe_api_library_factories(const char *xml, char *buf, int64_t capacity, int64_t *needed);
/* SolverLibrary::CreateLibrary(xml) -> GetSolverFactory(name) -> BuildSolver(A, state).
 * xml: a <ParameterList name="Preconditioner Library"> document.  seq may be NULL for
 * solvers that need no sequence.  ess_attr[nattr]: essential boundary attribute marker
 * (SolverState::SetBoundaryLabels), may be NULL. */
int pe_api_solver_build(const char *xml_library, const char *solver_name, const pe_parcsr_host *A,
                        pe_sequence *seq, int start_level, int form, const int32_t *ess_attr, int nattr,
                        pe_solver **out);
/* same, for an operator that already lives on the device (ownership of A passes to the solver) */
int pe_api_solver_build_device(const char *xml_library, const char *solver_name, pe_mat *A,
                               pe_sequence *seq, int start_level, int form, const int32_t *ess_attr, int nattr,
                               pe_solver **out);
/* solver->Mult(B, X) with HOST buffers (H2D of b, D2H of x inside the call);
 * iterative_mode != 0 uses x as initial guess */
int pe_api_solver_mult(pe_solver *s, const double *b_host, double *x_host, int n, int iterative_mode);
/* solver->MultTranspose(B, X) with host buffers (HiptmairSmoother::MultTranspose, ParELAG_HiptmairSmoother.cpp:79-109;
 * solvers without a transpose throw not_implemented_error like the reference) */
int pe_api_solver_mult_transpose(pe_solver *s, const double *b_host, double *x_host, int n, int iterative_mode);
/* solver->Mult on device-resident vectors (no copies) */
int pe_api_solver_mult_device(pe_solver *s, const pe_vec *b, pe_vec *x, int iterative_mode);
/* Krylov solvers: apply the preconditioner alone (e.g. one AMGe V-cycle) on device vectors */
int pe_api_solver_prec_mult_device(pe_solver *s, const pe_vec *b, pe_vec *x);
/* the same with HOST buffers: mfem::Solver::Mult(B, X) of the preconditioner object (the AMGe Hierarchy,
 * ParELAG_Hierarchy.cpp:109-136) as a host-side driver calls it; H2D of b and D2H of x inside the call */
int pe_api_solver_prec_mult(pe_solver *s, const double *b_host, double *x_host, int n);
/* Krylov solvers: "(B r, r)" history (what MFEM prints), iteration count, convergence flag; StationarySolver
 * (ParELAG_StationarySolver.cpp:41-147): ||r_k|| per iteration */
int pe_api_solver_get_history(const pe_solver *s, double *hist, int capacity, int *count,
                              int *iterations, int *converged);
/* Hierarchy solvers: number of levels, and size / nnz of A on a level */
int pe_api_solver_num_levels(const pe_solver *s, int *nlevels);
/* Hierarchy solvers: the persistent program the V-cycle was recorded into (NULL until the third
 * preconditioner application with the same buffers, or when recording was not possible) */
int pe_api_solver_program(const pe_solver *s, pe_program **out);
/* Hierarchy solvers: how the last preconditioner-mode V-cycle (Mult with iterative_mode off, e.g.
 * pe_api_solver_prec_mult_device) ran: 0 directly, 1 as a replayed or just-recorded CUDA graph, 2 as the
 * persistent program.  A host-side value: no device work, no synchronisation. */
enum { PE_REPLAY_DIRECT = 0, PE_REPLAY_GRAPH = 1, PE_REPLAY_PROGRAM = 2 };
int pe_api_solver_replay_mode(const pe_solver *s, int *mode);
int pe_api_solver_level_info(const pe_solver *s, int level, int64_t *nrows, int64_t *nnz, int64_t *nnz_P);
/* download A (diag block) of a hierarchy level for parity tests; arrays sized from level_info */
int pe_api_solver_level_matrix(const pe_solver *s, int level, int32_t *I, int32_t *J, double *A);
int pe_api_solver_free(pe_solver *s);

/* TimeManager: seconds accumulated under a timer name; clear all timers */
int pe_api_timer_get(const char *name, double *seconds);
int pe_api_timer_clear(void);

#ifdef __cplusplus
}
#endif
#endif
