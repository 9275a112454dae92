// pe_api.cpp -- C facade over the C++ solver API (see include/parelag_b200_api.h).
#include "parelag_b200_api.h"
#include "parelag_solvers.hpp"
#include "amge_coarsen.hpp"
#include "spe10.hpp"
#include <cstring>

void pe_set_error(const std::string &msg);   // csrc/pe_core.cu

using namespace parelag;

struct pe_sequence { std::vector<std::shared_ptr<DeRhamSequence>> levels; };
struct pe_solver
{
    std::shared_ptr<SolverLibrary> lib;
    std::shared_ptr<mfem::Operator> A;
    std::unique_ptr<mfem::Solver> solver;
    mfem::Vector b, x;
};

static std::unique_ptr<mpi_session> g_session;
static pe_host_comm g_host_comm{};       // copy of the caller's table (function pointers + user)
static bool g_have_host_comm = false;

#define API_TRY try {
#define API_CATCH                                                      \
    }                                                                  \
    catch (const std::exception &e) { pe_set_error(e.what()); return 10; } \
    catch (...) { pe_set_error("unknown C++ exception"); return 11; }  \
    return 0;

extern "C" int pe_api_session_create(int rank, int nranks, int device, const void *id)
{
    API_TRY
    if (!g_session) g_session = make_unique<mpi_session>(rank, nranks, device, id);
    API_CATCH
}
extern "C" int pe_api_session_destroy(void)
{
    API_TRY
    g_session.reset();
    API_CATCH
}
extern "C" pe_ctx *pe_api_session_ctx(void) { return Device::Ctx(); }

extern "C" int pe_api_session_set_host_comm(const pe_host_comm *comm)
{
    API_TRY
    PARELAG_TEST_FOR_EXCEPTION(!comm || !comm->allgather || !comm->alltoallv, std::runtime_error, "pe_api_session_set_host_comm: incomplete callback table");
    g_host_comm = *comm;
    g_have_host_comm = true;
    if (Device::Ctx()) PE_CALL(pe_ctx_set_host_comm(Device::Ctx(), &g_host_comm));
    API_CATCH
}
extern "C" int pe_api_hexsequence_create_par(const int32_t *procs, int nx, int ny, int nz, double Lx, double Ly, double Lz,
                                             const double *alpha, const double *beta, int jstart, int nlevels, double svd_tol,
                                             pe_sequence **out)
{
    API_TRY
    PARELAG_TEST_FOR_EXCEPTION(!g_have_host_comm, std::runtime_error, "pe_api_hexsequence_create_par: call pe_api_session_set_host_comm first");
    auto s = std::make_unique<pe_sequence>();      // released only when the build succeeded
    const int P[3] = {procs[0], procs[1], procs[2]};
    s->levels = BuildHexSequenceHierarchyPar(&g_host_comm, P, nx, ny, nz, Lx, Ly, Lz, alpha, beta, jstart, nlevels, svd_tol);
    *out = s.release();
    API_CATCH
}
extern "C" int pe_api_hexsequence_create_par_deformed(const int32_t *procs, int nx, int ny, int nz, const double *vertex_xyz,
                                                      const double *alpha, const double *beta, int jstart, int nlevels, double svd_tol,
                                                      pe_sequence **out)
{
    API_TRY
    PARELAG_TEST_FOR_EXCEPTION(!g_have_host_comm, std::runtime_error, "pe_api_hexsequence_create_par_deformed: call pe_api_session_set_host_comm first");
    PARELAG_TEST_FOR_EXCEPTION(!vertex_xyz, std::runtime_error, "pe_api_hexsequence_create_par_deformed: vertex coordinates missing");
    auto s = std::make_unique<pe_sequence>();      // released only when the build succeeded
    const int P[3] = {procs[0], procs[1], procs[2]};
    s->levels = BuildHexSequenceHierarchyPar(&g_host_comm, P, nx, ny, nz, 1.0, 1.0, 1.0, alpha, beta, jstart, nlevels, svd_tol, vertex_xyz);
    *out = s.release();
    API_CATCH
}
extern "C" int pe_api_sequence_get_dofmap(pe_sequence *s, int level, int form, int32_t *ndofs, int64_t *gid, int32_t *owner,
                                          int64_t *key, int64_t *true_start, int64_t *true_count, int64_t *global_count)
{
    API_TRY
    auto &seq = *s->levels.at(level);
    const par::SharingMap *m = seq.GetDofTrueDof(form);
    PARELAG_TEST_FOR_EXCEPTION(!m, std::runtime_error, "pe_api_sequence_get_dofmap: no dof <-> true dof map on level " << level << ", form " << form);
    if (ndofs) *ndofs = m->GetLocalSize();
    if (gid) std::copy(m->gid.begin(), m->gid.end(), gid);
    if (owner) std::copy(m->owner.begin(), m->owner.end(), owner);
    if (key) std::copy(m->key.begin(), m->key.end(), key);
    if (true_start) *true_start = m->start;
    if (true_count) *true_count = m->ntrue;
    if (global_count) *global_count = m->global;
    API_CATCH
}
/// SharingMap::Assemble (direction 0: local dof vector -> true dof vector, copies summed) and
/// SharingMap::Distribute (direction 1: true -> local) on host vectors
extern "C" int pe_api_sequence_dofmap_apply(pe_sequence *s, int level, int form, int direction, const double *in, double *out)
{
    API_TRY
    auto &seq = *s->levels.at(level);
    const par::SharingMap *m = seq.GetDofTrueDof(form);
    PARELAG_TEST_FOR_EXCEPTION(!m || !seq.GetComm(), std::runtime_error, "pe_api_sequence_dofmap_apply: no dof <-> true dof map");
    if (direction == 0) m->Assemble(seq.GetComm(), in, out);
    else m->Distribute(seq.GetComm(), in, out);
    API_CATCH
}
/// ComputeTrueP / ComputeTrueD as device ParCSR matrices (what = "P" or "D")
extern "C" int pe_api_sequence_true_operator(pe_sequence *s, int level, const char *what, int form, const int32_t *ess_attr, int nattr,
                                             pe_mat **out)
{
    API_TRY
    auto &seq = *s->levels.at(level);
    std::unique_ptr<mfem::HypreParMatrix> M;
    if (ess_attr)
    {
        mfem::Array<int> ess(ess_attr, nattr);
        M = std::string(what) == "P" ? seq.ComputeTrueP(form, ess) : seq.ComputeTrueD(form, ess);
    }
    else M = std::string(what) == "P" ? seq.ComputeTrueP(form) : seq.ComputeTrueD(form);
    *out = M->Release();
    API_CATCH
}
extern "C" int pe_api_sequence_create(int nforms, int nlevels, pe_sequence **out)
{
    API_TRY
    auto s = std::make_unique<pe_sequence>();      // released only when the build succeeded
    for (int l = 0; l < nlevels; ++l) s->levels.push_back(std::make_shared<DeRhamSequence>(nforms));
    for (int l = 0; l + 1 < nlevels; ++l) s->levels[l]->SetCoarserSequence(s->levels[l + 1]);
    *out = s.release();
    API_CATCH
}
extern "C" int pe_api_sequence_set_P(pe_sequence *s, int level, int form, int nrows, int ncols,
                                     const int32_t *I, const int32_t *J, const double *A)
{
    API_TRY
    s->levels.at(level)->SetP(form, HostCSR(nrows, ncols, I, J, A));
    API_CATCH
}
extern "C" int pe_api_sequence_set_D(pe_sequence *s, int level, int form, int nrows, int ncols,
                                     const int32_t *I, const int32_t *J, const double *A)
{
    API_TRY
    s->levels.at(level)->SetD(form, HostCSR(nrows, ncols, I, J, A));
    API_CATCH
}
extern "C" int pe_api_sequence_set_bdr_mask(pe_sequence *s, int level, int form, int ndofs, const uint32_t *mask)
{
    API_TRY
    auto d = make_unique<DofHandler>();
    d->SetBoundaryMask(std::vector<uint32_t>(mask, mask + ndofs));
    s->levels.at(level)->SetDofHandler(form, std::move(d));
    API_CATCH
}
extern "C" int pe_api_sequence_free(pe_sequence *s) { delete s; return 0; }

extern "C" int pe_api_hexsequence_create(int nx, int ny, int nz, double Lx, double Ly, double Lz, const double *alpha, const double *beta,
                                         int jstart, int nlevels, double svd_tol, pe_sequence **out)
{
    API_TRY
    auto s = std::make_unique<pe_sequence>();      // released only when the build succeeded
    s->levels = BuildHexSequenceHierarchy(nx, ny, nz, Lx, Ly, Lz, alpha, beta, jstart, nlevels, svd_tol);
    *out = s.release();
    API_CATCH
}
extern "C" int pe_api_hexsequence_create_deformed(int nx, int ny, int nz, const double *vertex_xyz, const double *alpha,
                                                  const double *beta, int jstart, int nlevels, double svd_tol, pe_sequence **out)
{
    API_TRY
    PARELAG_TEST_FOR_EXCEPTION(!vertex_xyz, std::runtime_error, "pe_api_hexsequence_create_deformed: vertex coordinates missing");
    auto s = std::make_unique<pe_sequence>();      // released only when the build succeeded
    s->levels = BuildHexSequenceHierarchy(nx, ny, nz, 1.0, 1.0, 1.0, alpha, beta, jstart, nlevels, svd_tol, vertex_xyz);
    *out = s.release();
    API_CATCH
}
extern "C" int pe_api_hexsequence_create_tensor(int nx, int ny, int nz, double Lx, double Ly, double Lz, const double *alpha, const double *beta_xyz,
                                                int jstart, int nlevels, double svd_tol, pe_sequence **out)
{
    API_TRY
    auto s = std::make_unique<pe_sequence>();
    s->levels = BuildHexSequenceHierarchy(nx, ny, nz, Lx, Ly, Lz, alpha, beta_xyz, jstart, nlevels, svd_tol, nullptr, 3);
    *out = s.release();
    API_CATCH
}
// ---- SPE10 data set (src/SPE10/InversePermeabilityFunction.cpp)
extern "C" int pe_api_spe10_read(const char *perm_file, int Nx, int Ny, int Nz, double hx, double hy, double hz)
{
    API_TRY
    InversePermeabilityFunction::SetNumberCells(Nx, Ny, Nz);
    InversePermeabilityFunction::SetMeshSizes(hx, hy, hz);
    InversePermeabilityFunction::Set2DSlice(InversePermeabilityFunction::NONE, -1);
    InversePermeabilityFunction::ReadPermeabilityFile(perm_file, g_host_comm.size > 1 ? &g_host_comm : nullptr);
    API_CATCH
}
extern "C" int pe_api_spe10_set_constant(int Nx, int Ny, int Nz, double hx, double hy, double hz, double ipx, double ipy, double ipz)
{
    API_TRY
    InversePermeabilityFunction::SetNumberCells(Nx, Ny, Nz);
    InversePermeabilityFunction::SetMeshSizes(hx, hy, hz);
    InversePermeabilityFunction::Set2DSlice(InversePermeabilityFunction::NONE, -1);
    InversePermeabilityFunction::SetConstantInversePermeability(ipx, ipy, ipz);
    API_CATCH
}
extern "C" int pe_api_spe10_set_slice(int orientation, int npos)
{
    API_TRY
    PARELAG_TEST_FOR_EXCEPTION(orientation < 0 || orientation > 3, std::runtime_error, "pe_api_spe10_set_slice: orientation 0 = none, 1 = XY, 2 = XZ, 3 = YZ");
    InversePermeabilityFunction::Set2DSlice((InversePermeabilityFunction::SliceOrientation)orientation, npos);
    API_CATCH
}
extern "C" int pe_api_spe10_inverse_permeability(const double *xyz, int npoints, double *out)
{
    API_TRY
    for (int p = 0; p < npoints; ++p)
    {
        out[3 * (size_t)p + 2] = 0.0;
        InversePermeabilityFunction::InversePermeability(xyz + 3 * (size_t)p, out + 3 * (size_t)p);
    }
    API_CATCH
}
extern "C" int pe_api_spe10_data(double *out, int64_t *count)
{
    API_TRY
    const std::vector<double> &d = InversePermeabilityFunction::Data();
    if (count) *count = (int64_t)d.size();
    if (out) std::copy(d.begin(), d.end(), out);
    API_CATCH
}
extern "C" int pe_api_hexsequence_create_spe10(int nx, int ny, int nz, double hx, double hy, double hz, int jstart, int nlevels, double svd_tol,
                                               pe_sequence **out)
{
    API_TRY
    PARELAG_TEST_FOR_EXCEPTION(!InversePermeabilityFunction::Loaded(), std::runtime_error, "pe_api_hexsequence_create_spe10: read the permeability data first");
    // the coefficient of the element mass matrices is evaluated inside the cells (quadrature points of VectorFEMassIntegrator):
    // one value of the piecewise constant data per cell, taken at the cell centre
    std::vector<double> kinv((size_t)3 * nx * ny * nz);
    for (int k = 0; k < nz; ++k)
        for (int j = 0; j < ny; ++j)
            for (int i = 0; i < nx; ++i)
            {
                const double c[3] = {(i + 0.5) * hx, (j + 0.5) * hy, (k + 0.5) * hz};
                InversePermeabilityFunction::InversePermeability(c, &kinv[3 * ((size_t)i + (size_t)nx * (j + (size_t)ny * k))]);
            }
    auto s = std::make_unique<pe_sequence>();
    s->levels = BuildHexSequenceHierarchy(nx, ny, nz, nx * hx, ny * hy, nz * hz, nullptr, kinv.data(), jstart, nlevels, svd_tol, nullptr, 3);
    *out = s.release();
    API_CATCH
}
static int copy_lines(const std::vector<std::string> &lines, char *buf, int64_t capacity, int64_t *needed)
{
    std::string all;
    for (const std::string &l : lines) { all += l; all += '\n'; }
    if (needed) *needed = (int64_t)all.size() + 1;
    if (buf && capacity > 0)
    {
        const size_t n = std::min((size_t)capacity - 1, all.size());
        std::memcpy(buf, all.data(), n);
        buf[n] = 0;
    }
    return 0;
}
extern "C" int pe_api_set_topology_options(int partitioner, int check_topology, const int32_t *element_partitioning, int n)
{
    API_TRY
    PARELAG_TEST_FOR_EXCEPTION(partitioner < 0 || partitioner > 3, std::runtime_error,
                               "pe_api_set_topology_options: partitioner 0 = derefinement / logical Cartesian, 1 = geometric boxes, 2 = given partitioning, "
                               "3 = logical Cartesian with material ids");
    PARELAG_TEST_FOR_EXCEPTION(partitioner >= 2 && (!element_partitioning || n <= 0), std::runtime_error,
                               "pe_api_set_topology_options: partitioners 2 and 3 need the element partitioning / material ids");
    TopologyOptions &o = GlobalTopologyOptions();
    o.partitioner = partitioner;
    o.check_topology = check_topology != 0;
    o.user_partitioning.clear();
    if (partitioner >= 2) o.user_partitioning.assign(element_partitioning, element_partitioning + n);
    o.log.clear();
    API_CATCH
}
extern "C" int pe_api_topology_log(char *buf, int64_t capacity, int64_t *needed)
{
    API_TRY
    copy_lines(GlobalTopologyOptions().log, buf, capacity, needed);
    API_CATCH
}
extern "C" int pe_api_tetsequence_create(int nv, const double *vertex_xyz, int nel, const int32_t *tets, int nbdr, const int32_t *bdr_triangles,
                                         const int32_t *bdr_attributes, int nref, int nlevels, int jstart, double svd_tol, pe_sequence **out)
{
    API_TRY
    PARELAG_TEST_FOR_EXCEPTION(!vertex_xyz || !tets || nv < 4 || nel < 1, std::runtime_error, "pe_api_tetsequence_create: empty mesh");
    auto s = std::make_unique<pe_sequence>();      // released only when the build succeeded
    const TetMesh mesh = TetMesh::FromArrays(nv, vertex_xyz, nel, tets, nbdr, bdr_triangles, bdr_attributes);
    s->levels = BuildTetSequenceHierarchy(mesh, nref, nlevels, nullptr, nullptr, jstart, svd_tol);
    *out = s.release();
    API_CATCH
}
extern "C" int pe_api_tetsequence_create_from_file(const char *mesh_file, int nref, int nlevels, int jstart, double svd_tol, pe_sequence **out)
{
    API_TRY
    auto s = std::make_unique<pe_sequence>();      // released only when the build succeeded
    const TetMesh mesh = TetMesh::Read(mesh_file);        // NETGEN neutral or MFEM mesh v1.0, by the first line
    s->levels = BuildTetSequenceHierarchy(mesh, nref, nlevels, nullptr, nullptr, jstart, svd_tol);
    *out = s.release();
    API_CATCH
}
static HostCSR pool_as_csr(const BlockPool &P)
{
    HostCSR M;
    auto rd = P.rdof_offsets();
    M.nrows = M.ncols = rd.back();
    M.I.assign(1, 0);
    for (int e = 0; e < P.n(); ++e)
        for (int x = 0; x < P.size[e]; ++x)
        {
            for (int y = 0; y < P.size[e]; ++y) { M.J.push_back(rd[e] + y); M.A.push_back(P.block(e)[x * P.size[e] + y]); }
            M.I.push_back((int)M.J.size());
        }
    return M;
}
extern "C" int pe_api_sequence_get_csr(pe_sequence *s, int level, const char *what, int a, int b, int32_t *nrows, int32_t *ncols,
                                       int64_t *nnz, int32_t *I, int32_t *J, double *A)
{
    API_TRY
    auto &seq = *s->levels.at(level);
    const std::string w(what);
    HostCSR tmp;
    const HostCSR *M = nullptr;
    if (w == "P") M = seq.GetP(a);
    else if (w == "D") M = seq.GetDerivativeOperator(a);
    else
    {
        PARELAG_TEST_FOR_EXCEPTION(!seq.data, std::runtime_error, "pe_api_sequence_get_csr: sequence has no coarsening data");
        if (w == "M") { tmp = seq.ComputeMassOperator(a); M = &tmp; }
        else if (w == "Me") { tmp = pool_as_csr(seq.data->M.at({a, b})); M = &tmp; }
        else if (w == "B") M = &seq.data->topo->GetB(a);
        else if (w == "AE") M = &seq.data->topo->AEntityEntity(a);
        else if (w == "ED") M = &seq.data->dof.at(a)->entity_dof.at(b);
        else if (w == "FB") M = &seq.data->topo->FacetBdrAttribute();
    }
    PARELAG_TEST_FOR_EXCEPTION(!M, std::runtime_error, "pe_api_sequence_get_csr: \"" << w << "\" is not available on level " << level);
    if (nrows) *nrows = M->nrows;
    if (ncols) *ncols = M->ncols;
    if (nnz) *nnz = (int64_t)M->J.size();
    if (I) std::copy(M->I.begin(), M->I.end(), I);
    if (J) std::copy(M->J.begin(), M->J.end(), J);
    if (A) std::copy(M->A.begin(), M->A.end(), A);
    API_CATCH
}
extern "C" int pe_api_sequence_get_targets(pe_sequence *s, int level, int form, int32_t *ndofs, int32_t *ntargets, double *out)
{
    API_TRY
    auto &seq = *s->levels.at(level);
    PARELAG_ASSERT(seq.data);
    if (ndofs) *ndofs = seq.data->dof.at(form)->ndofs;
    if (ntargets) *ntargets = seq.data->ntargets.at(form);
    if (out) std::copy(seq.data->targets.at(form).begin(), seq.data->targets.at(form).end(), out);
    API_CATCH
}
extern "C" int pe_api_sequence_get_bdr_mask(pe_sequence *s, int level, int form, int32_t *ndofs, uint32_t *mask)
{
    API_TRY
    auto d = s->levels.at(level)->GetDofHandler(form);
    PARELAG_ASSERT(d);
    if (ndofs) *ndofs = d->GetNDofs();
    if (mask) std::copy(d->GetBoundaryMask().begin(), d->GetBoundaryMask().end(), mask);
    API_CATCH
}
extern "C" int pe_api_sequence_show_topology(pe_sequence *s, int level, char *buf, int64_t capacity, int64_t *needed)
{
    API_TRY
    auto &seq = *s->levels.at(level);
    PARELAG_ASSERT(seq.data && seq.data->topo);
    copy_lines(seq.data->topo->ShowMe(), buf, capacity, needed);
    API_CATCH
}
extern "C" int pe_api_sequence_check_invariants(pe_sequence *s, int level, double *worst)
{
    API_TRY
    const double w = s->levels.at(level)->CheckInvariants();
    if (worst) *worst = w;
    API_CATCH
}
extern "C" int pe_api_sequence_get_stat(pe_sequence *s, int level, const char *name, int64_t *value)
{
    API_TRY
    auto &seq = *s->levels.at(level);
    PARELAG_ASSERT(seq.data);
    auto it = seq.data->stats.find(name);
    *value = it == seq.data->stats.end() ? -1 : it->second;
    API_CATCH
}

extern "C" int pe_api_parameterlist_dump(const char *xml, char *buf, int64_t capacity, int64_t *needed)
{
    API_TRY
    SimpleXMLParameterListReader reader;
    auto pl = reader.Parse(xml);
    std::vector<std::string> lines;
    pl->Dump(lines);
    copy_lines(lines, buf, capacity, needed);
    API_CATCH
}
extern "C" int pe_api_library_factories(const char *xml, char *buf, int64_t capacity, int64_t *needed)
{
    API_TRY
    SimpleXMLParameterListReader reader;
    auto pl = reader.Parse(xml);
    const ParameterList &libpl = pl->IsSublist("Preconditioner Library") ? pl->Sublist("Preconditioner Library") : *pl;
    auto lib = SolverLibrary::CreateLibrary(libpl);
    std::vector<std::string> names = libpl.SublistNames(), lines;
    std::sort(names.begin(), names.end());
    for (const std::string &name : names)
    {
        const std::string type = libpl.Sublist(name).Get<std::string>("Type");
        std::string status = "ok";
        try { (void)lib->GetSolverFactory(name); }
        catch (const std::exception &e)
        {
            status = std::string("error: ") + e.what();
            std::replace(status.begin(), status.end(), '\n', ' ');
        }
        lines.push_back(name + "\t" + type + "\t" + status);
    }
    copy_lines(lines, buf, capacity, needed);
    API_CATCH
}
extern "C" int pe_api_solver_build(const char *xml, const char *name, const pe_parcsr_host *A, pe_sequence *seq,
                                   int start_level, int form, const int32_t *ess_attr, int nattr, pe_solver **out)
{
    API_TRY
    auto s = make_unique<pe_solver>();
    SimpleXMLParameterListReader reader;
    auto pl = reader.Parse(xml);
    s->lib = SolverLibrary::CreateLibrary(*pl);
    auto fact = s->lib->GetSolverFactory(name);
    auto state = fact->GetDefaultState();
    if (seq) state->SetDeRhamSequence(seq->levels.at(start_level));
    std::vector<std::vector<int>> labels(1);
    if (ess_attr) labels[0].assign(ess_attr, ess_attr + nattr);
    state->SetBoundaryLabels(labels);
    state->SetForms({form});
    s->A = std::make_shared<mfem::HypreParMatrix>(*A);
    {
        Timer t = TimeManager::AddTimer(std::string("Build Solver ") + name);
        s->solver = fact->BuildSolver(s->A, *state);
    }
    *out = s.release();
    API_CATCH
}
extern "C" int pe_api_solver_build_device(const char *xml, const char *name, pe_mat *A, pe_sequence *seq,
                                          int start_level, int form, const int32_t *ess_attr, int nattr, pe_solver **out)
{
    API_TRY
    auto s = make_unique<pe_solver>();
    SimpleXMLParameterListReader reader;
    auto pl = reader.Parse(xml);
    s->lib = SolverLibrary::CreateLibrary(*pl);
    auto fact = s->lib->GetSolverFactory(name);
    auto state = fact->GetDefaultState();
    if (seq) state->SetDeRhamSequence(seq->levels.at(start_level));
    std::vector<std::vector<int>> labels(1);
    if (ess_attr) labels[0].assign(ess_attr, ess_attr + nattr);
    state->SetBoundaryLabels(labels);
    state->SetForms({form});
    s->A = std::make_shared<mfem::HypreParMatrix>(A);
    {
        Timer t = TimeManager::AddTimer(std::string("Build Solver ") + name);
        s->solver = fact->BuildSolver(s->A, *state);
    }
    *out = s.release();
    API_CATCH
}
/// SetOperator on a built solver (new values, same pattern); ownership of A passes to the solver, and A is released
/// when the call is refused.  A Krylov solver's preconditioner takes the operator first, then the Krylov solver.
extern "C" int pe_api_solver_set_operator(pe_solver *s, pe_mat *A)
{
    API_TRY
    PARELAG_TEST_FOR_EXCEPTION(!A, std::runtime_error, "pe_api_solver_set_operator: bad arguments");
    auto op = std::make_shared<mfem::HypreParMatrix>(A);      // A is released with op when the call is refused
    PARELAG_TEST_FOR_EXCEPTION(!s, std::runtime_error, "pe_api_solver_set_operator: bad arguments");
    PARELAG_TEST_FOR_EXCEPTION(std::dynamic_pointer_cast<MfemBlockOperator>(s->A), std::runtime_error,
                               "pe_api_solver_set_operator: blocked operators (MfemBlockOperator) are not supported; build a new solver");
    auto held = std::dynamic_pointer_cast<mfem::HypreParMatrix>(s->A);
    PARELAG_TEST_FOR_EXCEPTION(!held, std::runtime_error, "pe_api_solver_set_operator: the solver's operator is not a HypreParMatrix");
    PARELAG_TEST_FOR_EXCEPTION(pe_ctx_nranks(Device::Get()) != 1, std::runtime_error,
                               "pe_api_solver_set_operator: more than one rank is not supported; build a new solver");
    CheckSamePattern(*held, *op, "pe_api_solver_set_operator");
    SetNestedOperator(*s->solver, op);
    s->A = op;
    API_CATCH
}
/// SetOperator on a solver built on an MfemBlockOperator: blocks[nblocks*nblocks] row-major, NULL = zero block, with
/// the held operator's block structure and patterns; ownership of every block passes to the solver, and they are
/// released when the call is refused
extern "C" int pe_api_solver_set_operator_block(pe_solver *s, int nblocks, pe_mat **blocks)
{
    API_TRY
    PARELAG_TEST_FOR_EXCEPTION(nblocks < 1 || !blocks, std::runtime_error, "pe_api_solver_set_operator_block: bad arguments");
    std::vector<std::shared_ptr<mfem::HypreParMatrix>> mats((size_t)nblocks * nblocks);   // released when the call is refused
    for (int k = 0; k < nblocks * nblocks; ++k)
        if (blocks[k]) { mats[k] = std::make_shared<mfem::HypreParMatrix>(blocks[k]); blocks[k] = nullptr; }
    PARELAG_TEST_FOR_EXCEPTION(!s, std::runtime_error, "pe_api_solver_set_operator_block: bad arguments");
    auto held = std::dynamic_pointer_cast<MfemBlockOperator>(s->A);
    PARELAG_TEST_FOR_EXCEPTION(!held, std::runtime_error,
                               "pe_api_solver_set_operator_block: the solver's operator is not an MfemBlockOperator");
    PARELAG_TEST_FOR_EXCEPTION(pe_ctx_nranks(Device::Get()) != 1, std::runtime_error,
                               "pe_api_solver_set_operator_block: more than one rank is not supported; build a new solver");
    PARELAG_TEST_FOR_EXCEPTION((size_t)nblocks != held->GetNumBlockRows() || (size_t)nblocks != held->GetNumBlockCols(),
                               std::runtime_error, "pe_api_solver_set_operator_block: the solver's operator has "
                               << held->GetNumBlockRows() << "x" << held->GetNumBlockCols() << " blocks, not " << nblocks << "x" << nblocks);
    auto op = std::make_shared<MfemBlockOperator>(held->CopyRowOffsets(), held->CopyColumnOffsets());
    for (int i = 0; i < nblocks; ++i)
        for (int j = 0; j < nblocks; ++j)
            if (mats[i * nblocks + j]) op->SetBlock(i, j, mats[i * nblocks + j]);     // refuses a block of the wrong size
    SameBlockStructure(*held, op, "pe_api_solver_set_operator_block");
    SetNestedOperator(*s->solver, op);
    s->A = op;
    API_CATCH
}
/// mixed (Darcy) system blocks as in examples/MultigridTestDarcy.cpp: M = mass(H(div)) (weights folded into
/// the element matrices), B = W D with W = mass(L2), Bt = B^T; the driver solves [[M Bt][B 0]]
extern "C" int pe_api_sequence_assemble_darcy(pe_sequence *s, int level, pe_mat **M_out, pe_mat **B_out, pe_mat **Bt_out)
{
    API_TRY
    auto &seq = *s->levels.at(level);
    PARELAG_TEST_FOR_EXCEPTION(!seq.data, std::runtime_error, "assemble_darcy: sequence has no mass matrices");
    pe_ctx *ctx = Device::Get();
    Timer t = TimeManager::AddTimer("Assemble linear system");
    const int nf = seq.GetNumberOfForms(), uform = nf - 2, pform = nf - 1;
    auto upload = [&](const HostCSR &M) { pe_mat *d = nullptr; auto v = M.View(); PE_CALL(pe_mat_upload(ctx, &v, &d)); return d; };
    auto mass = [&](int j)
    {
        const HostCSR &ED = seq.data->dof.at(j)->entity_dof.at(0);
        HostCSR R;
        R.nrows = (int)ED.J.size(); R.ncols = seq.data->dof[j]->ndofs;
        R.I.resize(R.nrows + 1); std::iota(R.I.begin(), R.I.end(), 0);
        R.J = ED.J; R.A = ED.A;
        pe_mat *Rd = upload(R), *Med = upload(pool_as_csr(seq.data->M.at({j, 0}))), *Md = nullptr;
        PE_CALL(pe_rap(ctx, nullptr, Med, Rd, &Md));
        pe_mat_free(Rd); pe_mat_free(Med);
        return Md;
    };
    pe_mat *M = mass(uform), *W = mass(pform), *D = upload(*seq.GetDerivativeOperator(uform)), *B = nullptr, *Bt = nullptr;
    PE_CALL(pe_spgemm(ctx, W, D, &B));
    pe_mat_free(W); pe_mat_free(D);
    if (seq.IsParallel())
    {
        // the rank-local blocks become ParCSR matrices on true dofs: Assemble(dofTrueDof, ., dofTrueDof)
        // (examples/MultigridTestDarcy.cpp: pM, pB; SharingMap.cpp:975-1011); B^T by the distributed transpose
        auto download = [&](pe_mat *m)
        {
            int32_t nr = 0, nc = 0; int64_t nnz = 0;
            PE_CALL(pe_mat_info(m, &nr, &nc, nullptr, &nnz, nullptr));
            HostCSR L;
            L.nrows = nr; L.ncols = nc; L.I.resize(nr + 1); L.J.resize(nnz); L.A.resize(nnz);
            PE_CALL(pe_mat_download(m, L.I.data(), L.J.data(), L.A.data(), nullptr, nullptr, nullptr, nullptr));
            pe_mat_free(m);
            return L;
        };
        const HostCSR Ml = download(M), Bl = download(B);
        M = seq.AssembleTrue(uform, Ml, uform)->Release();
        B = seq.AssembleTrue(pform, Bl, uform)->Release();
    }
    PE_CALL(pe_mat_transpose(ctx, B, &Bt));
    *M_out = M; *B_out = B; *Bt_out = Bt;
    API_CATCH
}
/// BuildSolver on an MfemBlockOperator: blocks[nblocks*nblocks] row-major, NULL = zero block (ownership of
/// the device matrices passes to the solver); forms[nblocks]; ess_attr[nblocks*nattr] or NULL
extern "C" int pe_api_solver_build_block(const char *xml, const char *name, int nblocks, pe_mat **blocks, pe_sequence *seq,
                                         int start_level, const int32_t *forms, const int32_t *ess_attr, int nattr, pe_solver **out)
{
    API_TRY
    auto s = make_unique<pe_solver>();
    SimpleXMLParameterListReader reader;
    auto pl = reader.Parse(xml);
    s->lib = SolverLibrary::CreateLibrary(*pl);
    auto fact = s->lib->GetSolverFactory(name);
    auto state = fact->GetDefaultState();
    if (seq) state->SetDeRhamSequence(seq->levels.at(start_level));
    std::vector<std::vector<int>> labels(nblocks);
    if (ess_attr) for (int b = 0; b < nblocks; ++b) labels[b].assign(ess_attr + (size_t)b * nattr, ess_attr + (size_t)(b + 1) * nattr);
    state->SetBoundaryLabels(labels);
    state->SetForms(std::vector<int>(forms, forms + nblocks));
    std::vector<std::shared_ptr<mfem::HypreParMatrix>> mats((size_t)nblocks * nblocks);
    std::vector<int> offsets(nblocks + 1, 0);
    for (int i = 0; i < nblocks; ++i)
        for (int j = 0; j < nblocks; ++j)
            if (blocks[i * nblocks + j])
            {
                mats[i * nblocks + j] = std::make_shared<mfem::HypreParMatrix>(blocks[i * nblocks + j]);
                blocks[i * nblocks + j] = nullptr;
            }
    for (int i = 0; i < nblocks; ++i)
    {
        int h = -1;
        for (int j = 0; j < nblocks; ++j) if (mats[i * nblocks + j]) h = mats[i * nblocks + j]->Height();
        for (int j = 0; j < nblocks && h < 0; ++j) if (mats[j * nblocks + i]) h = mats[j * nblocks + i]->Width();
        PARELAG_TEST_FOR_EXCEPTION(h < 0, std::runtime_error, "pe_api_solver_build_block: block row " << i << " is empty");
        offsets[i + 1] = offsets[i] + h;
    }
    auto blop = std::make_shared<MfemBlockOperator>(offsets);
    for (int i = 0; i < nblocks; ++i)
        for (int j = 0; j < nblocks; ++j)
            if (mats[i * nblocks + j]) blop->SetBlock(i, j, mats[i * nblocks + j]);
    s->A = blop;
    {
        Timer t = TimeManager::AddTimer(std::string("Build Solver ") + name);
        s->solver = fact->BuildSolver(s->A, *state);
    }
    *out = s.release();
    API_CATCH
}
extern "C" int pe_api_sequence_assemble_system(pe_sequence *s, int level, int form, const int32_t *ess_attr, int nattr, pe_mat **out)
{
    API_TRY
    auto &seq = *s->levels.at(level);
    PARELAG_TEST_FOR_EXCEPTION(!seq.data, std::runtime_error, "assemble_system: sequence has no mass matrices");
    pe_ctx *ctx = Device::Get();
    Timer t = TimeManager::AddTimer("Assemble linear system");
    auto upload = [&](const HostCSR &M) { pe_mat *d = nullptr; auto v = M.View(); PE_CALL(pe_mat_upload(ctx, &v, &d)); return d; };
    // assembled mass operators: R^T M_e R with R = rDof -> dof (one +-1 per row)
    auto mass = [&](int j)
    {
        const HostCSR &ED = seq.data->dof.at(j)->entity_dof.at(0);
        HostCSR R;
        R.nrows = (int)ED.J.size(); R.ncols = seq.data->dof[j]->ndofs;
        R.I.resize(R.nrows + 1); std::iota(R.I.begin(), R.I.end(), 0);
        R.J = ED.J; R.A = ED.A;
        pe_mat *Rd = upload(R), *Med = upload(pool_as_csr(seq.data->M.at({j, 0}))), *Md = nullptr;
        PE_CALL(pe_rap(ctx, nullptr, Med, Rd, &Md));
        pe_mat_free(Rd); pe_mat_free(Med);
        return Md;
    };
    pe_mat *W = mass(form + 1), *D = upload(*seq.GetDerivativeOperator(form)), *A = nullptr;
    PE_CALL(pe_rap(ctx, nullptr, W, D, &A));
    pe_mat_free(W); pe_mat_free(D);
    if (form > 0)
    {
        pe_mat *M = mass(form), *S = nullptr;
        PE_CALL(pe_spadd(ctx, 1.0, M, 1.0, A, &S));
        pe_mat_free(M); pe_mat_free(A);
        A = S;
    }
    if (ess_attr)
    {
        mfem::Array<int> ess(ess_attr, nattr), marker(seq.GetNumberOfDofs(form));
        seq.GetDofHandler(form)->MarkDofsOnSelectedBndr(ess, marker);
        PE_CALL(pe_mat_eliminate_rowcol(ctx, A, marker.GetData()));
    }
    if (seq.IsParallel())
    {
        // A = Assemble(dofTrueDof, spA, dofTrueDof) (examples/MultigridTest2Form.cpp:560): the local
        // contributions of all holders of a shared dof are summed on its owner
        const par::SharingMap &map = *seq.GetDofTrueDof(form);
        int32_t nr = 0, nc = 0; int64_t nnz = 0;
        PE_CALL(pe_mat_info(A, &nr, &nc, nullptr, &nnz, nullptr));
        HostCSR L;
        L.nrows = nr; L.ncols = nc; L.I.resize(nr + 1); L.J.resize(nnz); L.A.resize(nnz);
        PE_CALL(pe_mat_download(A, L.I.data(), L.J.data(), L.A.data(), nullptr, nullptr, nullptr, nullptr));
        pe_mat_free(A); A = nullptr;
        pe_parcsr_owned *M = nullptr;
        PE_CALL(pe_par_assemble(seq.GetComm(), 0, L.nrows, L.ncols, L.I.data(), L.J.data(), L.A.data(), map.gid.data(), map.owner.data(),
                                map.gid.data(), map.owner.data(), map.start, map.start + map.ntrue, map.global,
                                map.start, map.start + map.ntrue, map.global, &M));
        const int rc = pe_mat_upload(ctx, pe_parcsr_owned_view(M), &A);
        pe_parcsr_owned_free(M);
        PE_CALL(rc);
    }
    *out = A;
    API_CATCH
}
extern "C" int pe_api_solver_mult(pe_solver *s, const double *b, double *x, int n, int iterative_mode)
{
    API_TRY
    PARELAG_TEST_FOR_EXCEPTION(n != s->solver->Height(), std::runtime_error, "pe_api_solver_mult: wrong vector length");
    s->b.SetSize(n); s->x.SetSize(n);
    // H2D straight from the caller's buffer (pinned or pageable), D2H straight into it
    PE_CALL(pe_vec_upload(s->b.Write(), b));
    if (iterative_mode) PE_CALL(pe_vec_upload(s->x.Write(), x));
    const bool saved = s->solver->iterative_mode;
    s->solver->iterative_mode = iterative_mode != 0;
    s->solver->Mult(s->b, s->x);
    s->solver->iterative_mode = saved;
    PE_CALL(pe_vec_download(s->x.Read(), x));
    API_CATCH
}
/// solver->MultTranspose(B, X) with host buffers (e.g. HiptmairSmoother::MultTranspose, HiptmairSmoother.cpp:79-109)
extern "C" int pe_api_solver_mult_transpose(pe_solver *s, const double *b, double *x, int n, int iterative_mode)
{
    API_TRY
    PARELAG_TEST_FOR_EXCEPTION(n != s->solver->Height(), std::runtime_error, "pe_api_solver_mult_transpose: wrong vector length");
    s->b.SetSize(n); s->x.SetSize(n);
    PE_CALL(pe_vec_upload(s->b.Write(), b));
    if (iterative_mode) PE_CALL(pe_vec_upload(s->x.Write(), x));
    const bool saved = s->solver->iterative_mode;
    s->solver->iterative_mode = iterative_mode != 0;
    s->solver->MultTranspose(s->b, s->x);
    s->solver->iterative_mode = saved;
    PE_CALL(pe_vec_download(s->x.Read(), x));
    API_CATCH
}
namespace
{
// a non-owning mfem::Vector over an existing pe_vec
struct VecAlias : mfem::Vector { };
}
extern "C" int pe_api_solver_mult_device(pe_solver *s, const pe_vec *b, pe_vec *x, int iterative_mode)
{
    API_TRY
    const int n = s->solver->Height();
    PARELAG_TEST_FOR_EXCEPTION(pe_vec_size(b) != n || pe_vec_size(x) != n, std::runtime_error, "pe_api_solver_mult_device: wrong vector length");
    s->b.SetSize(n); s->x.SetSize(n);
    PE_CALL(pe_vec_copy(b, s->b.Write()));
    if (iterative_mode) PE_CALL(pe_vec_copy(x, s->x.Write()));
    const bool saved = s->solver->iterative_mode;
    s->solver->iterative_mode = iterative_mode != 0;
    s->solver->Mult(s->b, s->x);
    s->solver->iterative_mode = saved;
    PE_CALL(pe_vec_copy(s->x.Read(), x));
    API_CATCH
}
extern "C" int pe_api_solver_prec_mult_device(pe_solver *s, const pe_vec *b, pe_vec *x)
{
    API_TRY
    auto k = dynamic_cast<const KrylovSolver *>(s->solver.get());
    PARELAG_TEST_FOR_EXCEPTION(!k || !k->GetPreconditioner(), std::runtime_error, "pe_api_solver_prec_mult_device: not a preconditioned Krylov solver");
    const int n = s->solver->Height();
    s->b.SetSize(n); s->x.SetSize(n);
    PE_CALL(pe_vec_copy(b, s->b.Write()));
    k->GetPreconditioner()->Mult(s->b, s->x);
    PE_CALL(pe_vec_copy(s->x.Read(), x));
    API_CATCH
}
/// mfem::Solver::Mult of the PRECONDITIONER held by a Krylov solver (the AMGe Hierarchy: one V-cycle,
/// Hierarchy.cpp:109-136) with HOST vectors: H2D of b, V-cycle, D2H of x inside the call -- what a driver that keeps its
/// vectors on the host pays per preconditioner application.
extern "C" int pe_api_solver_prec_mult(pe_solver *s, const double *b, double *x, int n)
{
    API_TRY
    auto k = dynamic_cast<const KrylovSolver *>(s->solver.get());
    PARELAG_TEST_FOR_EXCEPTION(!k || !k->GetPreconditioner(), std::runtime_error, "pe_api_solver_prec_mult: not a preconditioned Krylov solver");
    PARELAG_TEST_FOR_EXCEPTION(n != s->solver->Height(), std::runtime_error, "pe_api_solver_prec_mult: wrong vector length");
    s->b.SetSize(n); s->x.SetSize(n);
    PE_CALL(pe_vec_upload(s->b.Write(), b));
    k->GetPreconditioner()->Mult(s->b, s->x);
    PE_CALL(pe_vec_download(s->x.Read(), x));
    API_CATCH
}
extern "C" int pe_api_solver_get_history(const pe_solver *s, double *hist, int capacity, int *count, int *iterations, int *converged)
{
    API_TRY
    if (auto st = dynamic_cast<const StationarySolver *>(s->solver.get()))
    {
        // StationarySolver: ||r_k|| per iteration (what "Print Iterations" prints)
        const auto &h = st->GetResidualHistory();
        if (count) *count = (int)h.size();
        for (int i = 0; i < capacity && i < (int)h.size(); ++i) hist[i] = h[i];
        if (iterations) *iterations = st->GetNumIterations();
        if (converged) *converged = st->GetConverged() ? 1 : 0;
        return 0;
    }
    auto k = dynamic_cast<const KrylovSolver *>(s->solver.get());
    PARELAG_TEST_FOR_EXCEPTION(!k, std::runtime_error, "pe_api_solver_get_history: not a Krylov or stationary solver");
    const auto &h = k->GetResidualHistory();
    if (count) *count = (int)h.size();
    for (int i = 0; i < capacity && i < (int)h.size(); ++i) hist[i] = h[i];
    if (iterations) *iterations = k->GetNumIterations();
    if (converged) *converged = k->GetConverged() ? 1 : 0;
    API_CATCH
}
static const Hierarchy *as_hierarchy(const pe_solver *s)
{
    auto h = dynamic_cast<const Hierarchy *>(s->solver.get());
    if (!h)
        if (auto k = dynamic_cast<const KrylovSolver *>(s->solver.get()))
            h = dynamic_cast<const Hierarchy *>(k->GetPreconditioner().get());
    PARELAG_TEST_FOR_EXCEPTION(!h, std::runtime_error, "solver is not a Hierarchy (AMGe) solver");
    return h;
}
extern "C" int pe_api_solver_num_levels(const pe_solver *s, int *nlevels)
{
    API_TRY
    *nlevels = as_hierarchy(s)->GetNumLevels();
    API_CATCH
}
extern "C" int pe_api_solver_program(const pe_solver *s, pe_program **out)
{
    API_TRY
    *out = as_hierarchy(s)->GetProgram();
    API_CATCH
}
extern "C" int pe_api_solver_replay_mode(const pe_solver *s, int *mode)
{
    API_TRY
    *mode = as_hierarchy(s)->LastReplayMode();
    API_CATCH
}
extern "C" int pe_api_solver_level_info(const pe_solver *s, int level, int64_t *nrows, int64_t *nnz, int64_t *nnz_P)
{
    API_TRY
    auto h = const_cast<Hierarchy *>(as_hierarchy(s));
    // a level operator is a ParCSR matrix or (blocked hierarchy) an MfemBlockOperator of ParCSR blocks: sum over blocks
    auto count = [](const Op_Ptr &op, int64_t *rows, int64_t *entries)
    {
        if (auto A = std::dynamic_pointer_cast<mfem::HypreParMatrix>(op)) { *rows = A->M(); *entries = A->NNZ(); return; }
        auto B = std::dynamic_pointer_cast<MfemBlockOperator>(op);
        PARELAG_TEST_FOR_EXCEPTION(!B, std::runtime_error, "pe_api_solver_level_info: level operator is neither ParCSR nor a block operator");
        *rows = B->Height(); *entries = 0;
        for (size_t i = 0; i < B->GetNumBlockRows(); ++i)
            for (size_t j = 0; j < B->GetNumBlockCols(); ++j)
                if (!B->IsZeroBlock(i, j))
                    if (auto blk = dynamic_cast<mfem::HypreParMatrix *>(&B->GetBlock(i, j))) *entries += blk->NNZ();
    };
    int64_t r = 0, e = 0;
    count(h->GetLevel(level).Get<Op_Ptr>("A"), &r, &e);
    if (nrows) *nrows = r;
    if (nnz) *nnz = e;
    if (nnz_P)
    {
        *nnz_P = 0;
        if (h->GetLevel(level).IsKey("P")) { int64_t pr = 0; count(h->GetLevel(level).Get<Op_Ptr>("P"), &pr, nnz_P); }
    }
    API_CATCH
}
extern "C" int pe_api_solver_level_matrix(const pe_solver *s, int level, int32_t *I, int32_t *J, double *A)
{
    API_TRY
    auto h = const_cast<Hierarchy *>(as_hierarchy(s));
    auto M = std::dynamic_pointer_cast<mfem::HypreParMatrix>(h->GetLevel(level).Get<Op_Ptr>("A"));
    PARELAG_TEST_FOR_EXCEPTION(!M, std::runtime_error, "pe_api_solver_level_matrix: the level operator is not a ParCSR matrix");
    PE_CALL(pe_mat_download(M->Handle(), I, J, A, nullptr, nullptr, nullptr, nullptr));
    API_CATCH
}
extern "C" int pe_api_solver_level_block(const pe_solver *s, int level, int i, int j, pe_mat **out)
{
    API_TRY
    *out = nullptr;
    auto op = const_cast<Hierarchy *>(as_hierarchy(s))->GetLevel(level).Get<Op_Ptr>("A");
    const mfem::Operator *blk = op.get();
    if (auto B = std::dynamic_pointer_cast<MfemBlockOperator>(op))
    {
        PARELAG_TEST_FOR_EXCEPTION(i < 0 || j < 0 || (size_t)i >= B->GetNumBlockRows() || (size_t)j >= B->GetNumBlockCols(),
                                   std::runtime_error, "pe_api_solver_level_block: no block (" << i << "," << j << ")");
        if (B->IsZeroBlock(i, j)) return 0;
        blk = &B->GetBlock(i, j);
    }
    else PARELAG_TEST_FOR_EXCEPTION(i != 0 || j != 0, std::runtime_error, "pe_api_solver_level_block: the level operator is not blocked");
    auto M = dynamic_cast<const mfem::HypreParMatrix *>(blk);
    PARELAG_TEST_FOR_EXCEPTION(!M, std::runtime_error, "pe_api_solver_level_block: the block is not a ParCSR matrix");
    PE_CALL(pe_mat_clone(Device::Get(), M->Handle(), out));
    API_CATCH
}
extern "C" int pe_api_solver_free(pe_solver *s) { delete s; return 0; }

extern "C" int pe_api_timer_get(const char *name, double *seconds)
{
    API_TRY
    *seconds = TimeManager::Seconds(name);
    API_CATCH
}
extern "C" int pe_api_timer_clear(void) { TimeManager::ClearAllData(); return 0; }
