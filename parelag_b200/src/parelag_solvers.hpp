// parelag_solvers.hpp -- solver operators and factories of the AMGe solve path, with
// the reference's class names and parameter names; every Mult() runs on the GPU
// through the C ABI (include/parelag_b200.h).
//   HypreSmootherWrapper    src/linalg/solver_ops/ParELAG_HypreSmootherWrapper.{hpp:69-83,cpp:20-35}
//   HypreSmootherFactory    src/linalg/factories/ParELAG_HypreSmootherFactory.cpp:21-43,92-109
//   HiptmairSmoother        src/linalg/solver_ops/ParELAG_HiptmairSmoother.cpp:48-109
//   HiptmairSmootherFactory src/linalg/factories/ParELAG_HiptmairSmootherFactory.cpp:52-179
//   KrylovSolver            src/linalg/solver_ops/ParELAG_KrylovSolver.{cpp:23-96,hpp:68-110} (mfem::CGSolver::Mult)
//   KrylovSolverFactory     src/linalg/factories/ParELAG_KrylovSolverFactory.cpp:25-118
//   Hierarchy               src/linalg/solver_ops/ParELAG_Hierarchy.cpp:109-267,282-383
//   AMGeSolverFactory       src/linalg/factories/ParELAG_AMGeSolverFactory.cpp:26-209
//   StationarySolver        src/linalg/solver_ops/ParELAG_StationarySolver.cpp:41-147
#pragma once
#include <algorithm>
#include <cctype>
#include <cmath>
#include <cstdio>
#include "parelag_core.hpp"
#include "parelag_sequence.hpp"
#include "parelag_block.hpp"

namespace parelag
{

namespace mg_utils
{
/// -(A x - b), bitwise equal to b - A x (src/linalg/utilities/ParELAG_MG_Utils.hpp:405-467)
inline void ComputeResidual(const mfem::Operator &A, const mfem::Vector &x, const mfem::Vector &b, mfem::Vector &r)
{
    auto A_hyp = dynamic_cast<const mfem::HypreParMatrix *>(&A);
    if (!A_hyp) { ComputeResidualGeneric(A, x, b, r); return; }     // block operators
    r.SetSize(b.Size());
    PE_CALL(pe_residual(Device::Get(), A_hyp->Handle(), x.Read(), b.Read(), r.Write()));
}
} // namespace mg_utils

/// the colour numbering of a multicolour SELL level (pe_smoother_colour_numbering): padded length and the device
/// array row -> position; npad == 0: natural numbering
struct ColourNumbering
{
    int32_t npad = 0;
    const int32_t *pos = nullptr;
};
using MatHandle = std::shared_ptr<pe_mat>;
/// copy of A (or of A^T) whose products read columns at cols.pos and write rows at rows.pos (natural where npad == 0)
inline MatHandle RenumberedCopy(const mfem::HypreParMatrix &A, bool transpose, const ColourNumbering &rows,
                                const ColourNumbering &cols)
{
    pe_mat *m = nullptr;
    PE_CALL(pe_mat_renumbered(Device::Get(), A.Handle(), transpose ? 1 : 0, rows.pos, rows.npad, cols.pos, cols.npad, &m));
    return MatHandle(m, [](pe_mat *p) { pe_mat_free(p); });
}

inline bool SolverCaptureSafe(const mfem::Solver *s)
{
    auto p = dynamic_cast<const Solver *>(s);
    return p && p->CaptureSafe();
}

// ------------------------------------------------------------------ Hypre smoother
class HypreSmootherWrapper : public Solver
{
public:
    HypreSmootherWrapper(const Op_Ptr &A, int type, ParameterList &params)
        : Solver(A->Height(), A->Width(), true), A_(std::dynamic_pointer_cast<mfem::HypreParMatrix>(A))
    {
        PARELAG_TEST_FOR_EXCEPTION(!A_, std::runtime_error, "HypreSmootherWrapper: operator must be a HypreParMatrix");
        const int sweeps = params.Get("Sweeps", 1);
        const double damping = params.Get("Damping Factor", 1.0);
        const double omega = params.Get("Omega", 1.0);
        const int cheby_order = params.Get("Cheby Poly Order", 2);
        const double cheby_frac = params.Get("Cheby Poly Fraction", 0.3);
        // how hypre's sequential row order is realised on the GPU (DESIGN.md):
        // "natural" reproduces hypre exactly (level scheduling), "multicolor" is the fast mode
        const std::string ordering = params.Get("GS ordering", "natural");
        PARELAG_TEST_FOR_EXCEPTION(ordering != "natural" && ordering != "multicolor", std::runtime_error,
                                   "HypreSmootherWrapper: \"GS ordering\" must be \"natural\" or \"multicolor\"");
        PE_CALL(pe_smoother_create(Device::Get(), A_->Handle(), type, sweeps, damping, omega, cheby_order, cheby_frac,
                                   ordering == "natural" ? PE_GS_ORDER_NATURAL : PE_GS_ORDER_MULTICOLOR, &smoo_));
    }
    ~HypreSmootherWrapper() override { pe_smoother_free(smoo_); }
    void Mult(const mfem::Vector &rhs, mfem::Vector &sol) const override
    {
        PE_CALL(pe_smoother_apply(smoo_, rhs.Read(), this->iterative_mode ? sol.ReadWrite() : sol.Write(),
                                  this->iterative_mode ? 1 : 0));
    }
    /// all supported relaxations are symmetric operators
    void MultTranspose(const mfem::Vector &rhs, mfem::Vector &sol) const override { Mult(rhs, sol); }
    bool CaptureSafe() const override { return true; }
    pe_smoother *Handle() const noexcept { return smoo_; }
    /// colour numbering of a multicolour SELL Gauss-Seidel smoother on one rank (npad == 0: none)
    ColourNumbering Numbering() const
    {
        ColourNumbering c;
        PE_CALL(pe_smoother_colour_numbering(smoo_, &c.npad, &c.pos));
        return c;
    }
    /// Mult on colour-numbered vectors (Numbering().npad entries); mode 0: sol is the initial guess, 1: zero initial
    /// guess, 2: sol is what pe_smoother_colour_in left
    void MultColour(const mfem::Vector &rhs, mfem::Vector &sol, int mode) const
    {
        PE_CALL(pe_smoother_apply_colour(smoo_, rhs.Read(), mode == 1 ? sol.Write() : sol.ReadWrite(), mode));
    }
private:
    /// the smoother takes op's values (pe_smoother_update); op must have the size and pattern of the held matrix
    void _do_set_operator(const Op_Ptr &op) override
    {
        auto A = std::dynamic_pointer_cast<mfem::HypreParMatrix>(op);
        PARELAG_TEST_FOR_EXCEPTION(!A, std::runtime_error, "HypreSmootherWrapper::SetOperator(): operator must be a HypreParMatrix");
        PE_CALL(pe_smoother_update(smoo_, A->Handle()));
        A_ = std::move(A);
    }
    std::shared_ptr<mfem::HypreParMatrix> A_;
    pe_smoother *smoo_ = nullptr;
};

/// mfem::HypreDiagScale ("Hypre Jacobi", type 413 of ParELAG_HypreSmootherFactory.cpp:27-31): x = diag(A)^{-1} b
/// (HYPRE_ParCSRDiagScale); the initial guess is ignored whatever iterative_mode says.  One Jacobi sweep with unit weight
/// from a zero guess is exactly that.
class HypreDiagScale : public Solver
{
public:
    explicit HypreDiagScale(const Op_Ptr &A) : Solver(A->Height(), A->Width(), true)
    {
        ParameterList p("Hypre Jacobi");
        p.Set("Sweeps", 1); p.Set("Damping Factor", 1.0); p.Set("Omega", 1.0);
        jacobi_ = make_unique<HypreSmootherWrapper>(A, 0, p);
        jacobi_->iterative_mode = false;
    }
    void Mult(const mfem::Vector &rhs, mfem::Vector &sol) const override { jacobi_->Mult(rhs, sol); }
    void MultTranspose(const mfem::Vector &rhs, mfem::Vector &sol) const override { jacobi_->Mult(rhs, sol); }
    bool CaptureSafe() const override { return true; }
private:
    void _do_set_operator(const Op_Ptr &op) override { jacobi_->SetOperator(op); }
    std::unique_ptr<HypreSmootherWrapper> jacobi_;
};

class HypreSmootherFactory : public SolverFactory
{
    std::unique_ptr<mfem::Solver> _do_build_solver(const Op_Ptr &op, SolverState &) const override
    {
        auto &params = GetParameters();
        const std::string name = params.Get("Type", "L1 Gauss-Seidel");
        const int type = TypeFromName(name);
        if (type == 413) return make_unique<HypreDiagScale>(op);
        return make_unique<HypreSmootherWrapper>(op, type, params);
    }
    void _do_set_default_parameters() override
    {
        auto &p = GetParameters();
        p.Get("Type", "L1 Gauss-Seidel"); p.Get("Sweeps", 1); p.Get("Damping Factor", 1.0); p.Get("Omega", 1.0);
        p.Get("Cheby Poly Order", 2); p.Get("Cheby Poly Fraction", 0.3);
    }
    void _do_initialize(const ParameterList &) override {}
public:
    static int TypeFromName(const std::string &n)
    {
        if (n == "Jacobi") return 0;
        if (n == "L1 Jacobi") return 1;
        if (n == "L1 Gauss-Seidel") return 2;
        if (n == "L1 Gauss-Seidel Truncated") return 4;
        if (n == "Lumped Jacobi") return 5;
        if (n == "Gauss-Seidel") return 6;
        if (n == "Chebyshev") return 16;
        if (n == "Hypre Jacobi") return 413;
        PARELAG_TEST_FOR_EXCEPTION(true, std::runtime_error,
                                   "HypreSmootherFactory: smoother type \"" << n << "\" is not supported on the GPU path "
                                   "(supported: Jacobi, L1 Jacobi, L1 Gauss-Seidel, L1 Gauss-Seidel Truncated, Lumped Jacobi, Gauss-Seidel, Chebyshev, "
                                   "Hypre Jacobi)");
        return -1;
    }
};

// ------------------------------------------------------------------ Hiptmair
class HiptmairSmoother : public Solver
{
public:
    HiptmairSmoother(Op_Ptr A, Op_Ptr A_Aux, Op_Ptr D_Op, std::shared_ptr<mfem::Solver> PrimarySolver,
                     std::shared_ptr<mfem::Solver> AuxiliarySolver)
        : Solver(A->Height(), A->Width(), true), A_(std::move(A)), A_aux_(std::move(A_Aux)), D_op_(std::move(D_Op)),
          PrimarySolver_(std::move(PrimarySolver)), AuxiliarySolver_(std::move(AuxiliarySolver))
    {
        PARELAG_ASSERT(A_); PARELAG_ASSERT(D_op_); PARELAG_ASSERT(PrimarySolver_); PARELAG_ASSERT(AuxiliarySolver_);
        AuxB_.SetSize(D_op_->Width());
        AuxX_.SetSize(D_op_->Width());
        PrimaryVec_.SetSize(A_->Height());
    }
    void Mult(const mfem::Vector &B, mfem::Vector &X) const override
    {
        if (this->IsPreconditioner()) X = 0.0;
        PARELAG_ASSERT(PrimarySolver_->iterative_mode);
        PrimarySolver_->Mult(B, X);
        mg_utils::ComputeResidual(*A_, X, B, PrimaryVec_);
        D_op_->MultTranspose(PrimaryVec_, AuxB_);
        PARELAG_ASSERT(!AuxiliarySolver_->iterative_mode);
        AuxiliarySolver_->Mult(AuxB_, AuxX_);
        AddAuxiliaryCorrection(X);
    }
    void MultTranspose(const mfem::Vector &B, mfem::Vector &X) const override
    {
        if (this->IsPreconditioner()) { X = 0.0; D_op_->MultTranspose(B, AuxB_); }
        else { mg_utils::ComputeResidual(*A_, X, B, PrimaryVec_); D_op_->MultTranspose(PrimaryVec_, AuxB_); }
        AuxiliarySolver_->Mult(AuxB_, AuxX_);
        AddAuxiliaryCorrection(X);
        PrimarySolver_->Mult(B, X);
    }
    Op_Ptr GetAuxiliaryOperator() const { return A_aux_; }
    /// the auxiliary operator was computed as D^T A D and FixZeroRows rewrote zero_rows (ZeroRows): SetOperator
    /// recomputes it.  Without this call the auxiliary operator came from the state and SetOperator keeps it.
    void SetComputedAuxiliary(mfem::Vector zero_rows) { aux_zero_rows_ = std::move(zero_rows); aux_computed_ = true; }
    /// The first half of SetOperator(op): the auxiliary operator for op, computed and checked without changing this
    /// smoother (throws on a refusal).  CommitOperator(op, PrepareOperator(op)) is SetOperator(op).
    Op_Ptr PrepareOperator(const Op_Ptr &op) const
    {
        auto A = std::dynamic_pointer_cast<mfem::HypreParMatrix>(op);
        PARELAG_TEST_FOR_EXCEPTION(!A, std::runtime_error, "HiptmairSmoother::SetOperator(): operator must be a HypreParMatrix");
        if (auto held = std::dynamic_pointer_cast<mfem::HypreParMatrix>(A_)) CheckSamePattern(*held, *A, "HiptmairSmoother");
        if (!aux_computed_) return A_aux_;
        auto aux = CopyOf(dynamic_cast<const mfem::HypreParMatrix &>(*A_aux_));
        PE_CALL(pe_rap_numeric(Device::Get(), nullptr, A->Handle(), dynamic_cast<const mfem::HypreParMatrix &>(*D_op_).Handle(), aux->Handle()));
        FixSameZeroRows(*aux, aux_zero_rows_, "the Hiptmair auxiliary operator D^T A D");
        return aux;
    }
    /// the second half: both smoothers and the residual take the new operators (the colour-numbered residual copy is
    /// the enclosing Hierarchy's and refreshed there)
    void CommitOperator(const Op_Ptr &op, const Op_Ptr &aux)
    {
        SetNestedOperator(*PrimarySolver_, op);
        if (aux != A_aux_) SetNestedOperator(*AuxiliarySolver_, aux);
        A_ = op;
        A_aux_ = aux;
    }
    bool CaptureSafe() const override
    { return SolverCaptureSafe(PrimarySolver_.get()) && SolverCaptureSafe(AuxiliarySolver_.get()); }
    pe_smoother *PrimaryHandle() const { return dynamic_cast<const HypreSmootherWrapper &>(*PrimarySolver_).Handle(); }
    /// colour numbering of the primary smoother when both smoothers have one (npad == 0: none)
    ColourNumbering Numbering() const
    {
        auto pri = dynamic_cast<const HypreSmootherWrapper *>(PrimarySolver_.get());
        auto aux = dynamic_cast<const HypreSmootherWrapper *>(AuxiliarySolver_.get());
        if (!pri || !aux || !dynamic_cast<const mfem::HypreParMatrix *>(D_op_.get()) || aux->Numbering().npad == 0) return {};
        return pri->Numbering();
    }
    /// Build the renumbered D (primary <- auxiliary numbering) and D^T; residual: A in the primary numbering (borrowed).
    void SetupColour(const MatHandle &residual)
    {
        auto pri = dynamic_cast<const HypreSmootherWrapper *>(PrimarySolver_.get());
        auto aux = dynamic_cast<const HypreSmootherWrapper *>(AuxiliarySolver_.get());
        auto &D = dynamic_cast<const mfem::HypreParMatrix &>(*D_op_);
        const ColourNumbering p = pri->Numbering(), a = aux->Numbering();
        cres_ = residual;
        cDt_ = RenumberedCopy(D, true, a, p);
        cD_ = RenumberedCopy(D, false, p, a);
        cPrimaryVec_.SetSize(p.npad); cAuxB_.SetSize(a.npad); cAuxX_.SetSize(a.npad);
    }
    /// Mult on vectors in the primary colour numbering (after SetupColour): the same products as Mult, on renumbered
    /// copies, and no renumbering passes; mode as HypreSmootherWrapper::MultColour
    void MultColour(const mfem::Vector &B, mfem::Vector &X, int mode) const
    {
        pe_ctx *ctx = Device::Get();
        dynamic_cast<const HypreSmootherWrapper &>(*PrimarySolver_).MultColour(B, X, mode);
        PE_CALL(pe_residual(ctx, cres_.get(), X.Read(), B.Read(), cPrimaryVec_.Write()));
        PE_CALL(pe_spmv(ctx, 1.0, cDt_.get(), cPrimaryVec_.Read(), 0.0, cAuxB_.Write()));
        dynamic_cast<const HypreSmootherWrapper &>(*AuxiliarySolver_).MultColour(cAuxB_, cAuxX_, 1);
        PE_CALL(pe_spmv(ctx, 1.0, cD_.get(), cAuxX_.Read(), 1.0, X.ReadWrite()));
    }
private:
    /// X += D AuxX_.  On one rank the add rides in the product (beta = 1): acc + X rounds like X + (D AuxX_), so the
    /// bits are those of the separate pass.  With a halo, D's diagonal and off-diagonal blocks are two passes, and
    /// adding X before the second would change the order of the sum, so the separate add stays.
    void AddAuxiliaryCorrection(mfem::Vector &X) const
    {
        auto D_hyp = dynamic_cast<const mfem::HypreParMatrix *>(D_op_.get());
        if (D_hyp && pe_ctx_nranks(Device::Get()) == 1) { D_hyp->Mult(1.0, AuxX_, 1.0, X); return; }
        D_op_->Mult(AuxX_, PrimaryVec_);
        X += PrimaryVec_;
    }
    void _do_set_operator(const Op_Ptr &op) override { CommitOperator(op, PrepareOperator(op)); }
    Op_Ptr A_, A_aux_, D_op_;
    std::shared_ptr<mfem::Solver> PrimarySolver_, AuxiliarySolver_;
    mutable mfem::Vector AuxB_, AuxX_, PrimaryVec_;
    MatHandle cres_, cDt_, cD_;                             // colour-numbered products (SetupColour)
    mutable mfem::Vector cPrimaryVec_, cAuxB_, cAuxX_;
    bool aux_computed_ = false;                              // SetComputedAuxiliary
    mfem::Vector aux_zero_rows_;
};

class HiptmairSmootherFactory : public SolverFactory
{
public:
    /// constructors, setters and getters of ParELAG_HiptmairSmootherFactory.hpp:40-111: the smoother factories may be
    /// handed over directly instead of being looked up in the library by name
    explicit HiptmairSmootherFactory(const ParameterList &params = ParameterList()) { SetParameters(params); }
    explicit HiptmairSmootherFactory(std::shared_ptr<SolverFactory> SmootherFact, const ParameterList &params = ParameterList())
        : PrimaryFact_(std::move(SmootherFact)), AuxiliaryFact_(PrimaryFact_) { SetParameters(params); }
    HiptmairSmootherFactory(std::shared_ptr<SolverFactory> PrimarySolverFactory, std::shared_ptr<SolverFactory> AuxiliarySolverFactory,
                            const ParameterList &params = ParameterList())
        : PrimaryFact_(std::move(PrimarySolverFactory)), AuxiliaryFact_(std::move(AuxiliarySolverFactory)) { SetParameters(params); }
    void SetPrimaryFactory(std::shared_ptr<SolverFactory> PrimaryFact) noexcept { PrimaryFact_ = std::move(PrimaryFact); }
    void SetAuxiliaryFactory(std::shared_ptr<SolverFactory> AuxFact) noexcept { AuxiliaryFact_ = std::move(AuxFact); }
    void SetFactories(std::shared_ptr<SolverFactory> PrimaryFact, std::shared_ptr<SolverFactory> AuxFact) noexcept
    { SetPrimaryFactory(std::move(PrimaryFact)); SetAuxiliaryFactory(std::move(AuxFact)); }
    std::shared_ptr<SolverFactory> GetPrimarySmootherFactory() const noexcept { return PrimaryFact_; }
    std::shared_ptr<SolverFactory> GetAuxiliarySmootherFactory() const noexcept { return AuxiliaryFact_; }

private:
    std::unique_ptr<mfem::Solver> _do_build_solver(const Op_Ptr &op, SolverState &state) const override
    {
        auto my_state = dynamic_cast<NestedSolverState *>(&state);
        PARELAG_ASSERT(my_state);
        auto primary_state = std::shared_ptr<SolverState>{PrimaryFact_->GetDefaultState()};
        auto aux_state = std::shared_ptr<SolverState>{AuxiliaryFact_->GetDefaultState()};
        if (my_state->IsSubState("Primary")) primary_state->MergeState(*my_state->GetSubState("Primary"));
        if (my_state->IsSubState("Auxiliary")) aux_state->MergeState(*my_state->GetSubState("Auxiliary"));
        primary_state->MergeState(*my_state);
        std::vector<int> aux_forms;
        for (int f : primary_state->GetForms()) aux_forms.push_back(f - 1);
        aux_state->SetForms(std::move(aux_forms));      // aux space is one form lower
        aux_state->MergeState(*my_state);

        auto d_op = my_state->GetOperator("D");
        if (!d_op)
        {
            Timer d_timer = TimeManager::AddTimer("Hiptmair: Build D");
            auto &sequence = state.GetDeRhamSequence();
            auto form = state.GetForms().front();
            PARELAG_ASSERT(form > 0);
            auto ess_attr = state.GetBoundaryLabels(0);
            if (ess_attr.size() > 0)
            {
                mfem::Array<int> label_ess(ess_attr.data(), (int)ess_attr.size());
                d_op = sequence.ComputeTrueD(form - 1, label_ess);
            }
            else
                d_op = sequence.ComputeTrueD(form - 1);
        }
        PARELAG_ASSERT(d_op);
        Timer pri_timer = TimeManager::AddTimer("Hiptmair: Build primary smoother");
        auto PrimarySmoo = std::shared_ptr<mfem::Solver>{PrimaryFact_->BuildSolver(op, *primary_state)};
        PrimarySmoo->iterative_mode = true;
        pri_timer.Stop();
        Timer aux_op_timer = TimeManager::AddTimer("Hiptmair: Build auxiliary operator");
        auto aux_op = my_state->GetOperator("Auxiliary A");
        const bool computed = !aux_op;
        mfem::Vector aux_zero_rows;
        if (computed) aux_op = _do_compute_aux_operator(*op, *d_op, aux_zero_rows);
        aux_op_timer.Stop();
        PARELAG_ASSERT(aux_op);
        Timer aux_timer = TimeManager::AddTimer("Hiptmair: Build auxiliary smoother");
        auto AuxiliarySmoo = std::shared_ptr<mfem::Solver>{AuxiliaryFact_->BuildSolver(aux_op, *aux_state)};
        AuxiliarySmoo->iterative_mode = false;
        aux_timer.Stop();
        auto H = make_unique<HiptmairSmoother>(op, aux_op, d_op, PrimarySmoo, AuxiliarySmoo);
        if (computed) H->SetComputedAuxiliary(std::move(aux_zero_rows));
        return H;
    }
    /// D^T A D followed by FixZeroRows (HiptmairSmootherFactory.cpp:143-165); zero_rows: the rows FixZeroRows rewrote
    Op_Ptr _do_compute_aux_operator(mfem::Operator &A, mfem::Operator &D, mfem::Vector &zero_rows) const
    {
        PARELAG_TEST_FOR_EXCEPTION(A.Width() != D.Height(), std::runtime_error,
                                   "A and D do not have compatible sizes to compute D^T*A*D!\nA = " << A.Height() << "x" << A.Width()
                                   << "\nD = " << D.Height() << "x" << D.Width());
        auto A_hyp = dynamic_cast<mfem::HypreParMatrix *>(&A);
        auto D_hyp = dynamic_cast<mfem::HypreParMatrix *>(&D);
        PARELAG_TEST_FOR_EXCEPTION(!A_hyp || !D_hyp, std::runtime_error, "Hiptmair: A and D must be HypreParMatrix");
        std::shared_ptr<mfem::HypreParMatrix> ret{mfem::RAP(A_hyp, D_hyp)};
        zero_rows = ZeroRows(*ret);
        hypre_ParCSRMatrixFixZeroRows(*ret);
        return ret;
    }
    void _do_set_default_parameters() override
    {
        auto &params = GetParameters();
        params.Get("Primary Smoother", "Default Hypre");       // ParELAG_HiptmairSmootherFactory.cpp:26-31
        params.Get("Auxiliary Smoother", "Default Hypre");
    }
    void _do_initialize(const ParameterList &) override
    {
        PARELAG_ASSERT(HasValidSolverLibrary());
        PrimaryFact_ = GetSolverLibrary().GetSolverFactory(GetParameters().Get<std::string>("Primary Smoother"));
        AuxiliaryFact_ = GetSolverLibrary().GetSolverFactory(GetParameters().Get<std::string>("Auxiliary Smoother"));
    }
    std::shared_ptr<SolverFactory> PrimaryFact_, AuxiliaryFact_;
};

// ------------------------------------------------------------------ Krylov (PCG)
/// mfem::CGSolver::Mult restated (preconditioned CG with MFEM's stopping rule and
/// its "(B r, r)" monitor); dots are device reductions + ncclAllReduce.
class KrylovSolver : public Solver
{
public:
    KrylovSolver(Op_Ptr A, std::shared_ptr<mfem::Solver> Prec, ParameterList &params)
        : Solver(A->Height(), A->Width(), false), A_(std::move(A)), Prec_(std::move(Prec))
    {
        std::string name = params.Get("Solver name", "PCG");
        std::transform(name.begin(), name.end(), name.begin(), ::toupper);      // ParELAG_KrylovSolver.cpp:38-40
        PARELAG_TEST_FOR_EXCEPTION(name != "PCG" && name != "CG" && name != "GMRES" && name != "FGMRES" && name != "MINRES" && name != "BICGSTAB",
                                   std::runtime_error, "KrylovSolver::KrylovSolver(...): Bad solver type (\"" << name << "\").\n\n"
                                   "Valid choices are \"CG\", \"GMRES\", \"FGMRES\", \"BiCGSTAB\", \"MINRES\".");
        gmres_ = name == "GMRES";
        method_ = name == "FGMRES" ? 1 : (name == "MINRES" ? 2 : (name == "BICGSTAB" ? 3 : 0));
        restart_ = params.Get("Restart size", 50);
        print_level_ = params.Get("Print level", -1);
        rel_tol_ = params.Get("Relative tolerance", 0.0);
        abs_tol_ = params.Get("Absolute tolerance", 0.0);
        max_iter_ = params.Get("Maximum iterations", 10);
        final_paragraph_ = params.Get("Print final paragraph", false);
    }
    ~KrylovSolver() override { pe_scalars_free(slots_); }
    /// Short inner solves (the AMGe coarse solver: "Maximum iterations" <= 10, no printing) run
    /// "device resident": a fixed number of iterations whose scalars (alpha, beta, the stopping
    /// tests of mfem::CGSolver::Mult) live in HBM.  Once the stopping test fires the step lengths
    /// become 0, so x equals the result of the early exit; there is no host synchronisation and
    /// the enclosing V-cycle can be captured in a CUDA graph.
    bool DeviceResident() const { return !gmres_ && method_ == 0 && max_iter_ >= 1 && max_iter_ <= 10 && print_level_ < 0 && !final_paragraph_; }
    bool CaptureSafe() const override
    {
        return DeviceResident() && (!Prec_ || SolverCaptureSafe(Prec_.get())) &&
               dynamic_cast<const mfem::HypreParMatrix *>(A_.get()) != nullptr;
    }
    void Mult(const mfem::Vector &b, mfem::Vector &x) const override
    {
        if (gmres_) { MultGMRES(b, x); return; }
        if (method_ == 1) { MultFGMRES(b, x); return; }
        if (method_ == 2) { MultMINRES(b, x); return; }
        if (method_ == 3) { MultBiCGSTAB(b, x); return; }
        if (DeviceResident()) { MultDeviceResident(b, x); return; }
        const int n = Height();
        r_.SetSize(n); d_.SetSize(n); z_.SetSize(n);
        history_.clear();
        stats_on_device_ = false;
        converged_ = false; final_iter_ = 0;
        if (this->iterative_mode) { A_->Mult(x, r_); mfem::add(b, -1.0, r_, r_); }
        else { r_ = b; x = 0.0; }
        if (Prec_) { Prec_->Mult(r_, z_); d_ = z_; }
        else d_ = r_;
        double nom0, nom, betanom, alpha, beta, den;
        nom0 = nom = d_ * r_;
        history_.push_back(nom);
        if (print_level_ == 1) std::printf("   Iteration : %3d  (B r, r) = %g\n", 0, nom);
        if (nom < 0.0) { final_norm_ = nom; return; }
        const double r0 = std::max(nom * rel_tol_ * rel_tol_, abs_tol_ * abs_tol_);
        if (nom <= r0) { converged_ = true; final_norm_ = std::sqrt(nom); return; }
        A_->Mult(d_, z_);
        den = z_ * d_;
        if (den <= 0.0)
        {
            // mfem::CGSolver::Mult: a non-positive (Ad, d) is reported, only an exact zero stops the iteration
            if (print_level_ >= 0 && d_ * d_ > 0.0) std::printf("PCG: The operator is not positive definite. (Ad, d) = %g\n", den);
            if (den == 0.0) { final_norm_ = std::sqrt(nom); return; }
        }
        int i = 1;
        bool stopped_early = false;
        while (true)
        {
            alpha = nom / den;
            x.Add(alpha, d_);
            r_.Add(-alpha, z_);
            if (Prec_) { Prec_->Mult(r_, z_); betanom = r_ * z_; }
            else betanom = r_ * r_;
            history_.push_back(betanom);
            if (print_level_ == 1) std::printf("   Iteration : %3d  (B r, r) = %g\n", i, betanom);
            if (betanom < r0) { converged_ = true; final_iter_ = i; break; }
            if (++i > max_iter_) break;
            beta = betanom / nom;
            if (Prec_) { d_ *= beta; d_ += z_; }        // d = z + beta d
            else { d_ *= beta; d_ += r_; }
            A_->Mult(d_, z_);
            den = d_ * z_;
            if (den <= 0.0)
            {
                if (print_level_ >= 0 && d_ * d_ > 0.0) std::printf("PCG: The operator is not positive definite. (Ad, d) = %g\n", den);
                if (den == 0.0) { final_iter_ = i; converged_ = false; stopped_early = true; break; }
            }
            nom = betanom;
        }
        if (!converged_ && !stopped_early) final_iter_ = max_iter_;
        final_norm_ = std::sqrt(std::fabs(betanom));
        if (final_paragraph_ || print_level_ >= 0)
            std::printf("PCG: %s after %d iterations, (B r, r) = %g, (B r_0, r_0) = %g\n",
                        converged_ ? "converged" : "NOT converged", final_iter_, betanom, nom0);
    }
    const std::shared_ptr<mfem::Solver> &GetPreconditioner() const { return Prec_; }
    int GetNumIterations() const { FetchStats(); return final_iter_; }
    bool GetConverged() const { FetchStats(); return converged_; }
    double GetFinalNorm() const { FetchStats(); return final_norm_; }
    /// history[i] = (B r, r) after iteration i (history[0]: initial) -- what MFEM prints
    const std::vector<double> &GetResidualHistory() const { FetchStats(); return history_; }
private:
    /// mfem::GMRESSolver::Mult restated: left-preconditioned restarted GMRES with Givens rotations
    /// ("Generalized Minimum Residual method following the algorithm on p. 20 of the SIAM Templates
    /// book"); monitor ||B r||; history[i] = that norm after iteration i
    void MultGMRES(const mfem::Vector &b, mfem::Vector &x) const
    {
        const int n = Height(), m = restart_;
        r_.SetSize(n); z_.SetSize(n);
        mfem::Vector &r = r_, &w = z_;
        history_.clear(); stats_on_device_ = false; converged_ = false; final_iter_ = 0;
        std::vector<double> H((size_t)(m + 1) * m, 0.0), s(m + 1), cs(m + 1), sn(m + 1);
        auto h = [&](int i, int j) -> double & { return H[(size_t)j * (m + 1) + i]; };
        auto norm = [](const mfem::Vector &v) { return std::sqrt(v * v); };
        if (this->iterative_mode) A_->Mult(x, r); else x = 0.0;
        if (Prec_)
        {
            if (this->iterative_mode) { mfem::add(b, -1.0, r, w); Prec_->Mult(w, r); }
            else Prec_->Mult(b, r);
        }
        else
        {
            if (this->iterative_mode) mfem::add(b, -1.0, r, r); else r = b;
        }
        double beta = norm(r), resid = beta;
        history_.push_back(beta);
        double final_norm = std::max(rel_tol_ * beta, abs_tol_);
        if (print_level_ == 1) std::printf("   Pass : %2d   Iteration : %3d  ||B r|| = %g\n", 1, 0, beta);
        if (beta <= final_norm) { final_norm_ = beta; final_iter_ = 0; converged_ = true; return; }
        if ((int)v_.size() < m + 1) v_.resize(m + 1);
        auto update = [&](int k)
        {
            std::vector<double> y(s.begin(), s.begin() + k + 1);
            for (int i = k; i >= 0; --i)
            {
                y[i] /= h(i, i);
                for (int j = i - 1; j >= 0; --j) y[j] -= h(j, i) * y[i];
            }
            for (int j = 0; j <= k; ++j) x.Add(y[j], v_[j]);
        };
        for (int j = 1; j <= max_iter_;)
        {
            v_[0].Set(1.0 / beta, r);
            std::fill(s.begin(), s.end(), 0.0);
            s[0] = beta;
            int i;
            for (i = 0; i < m && j <= max_iter_; ++i, ++j)
            {
                if (Prec_) { A_->Mult(v_[i], r); Prec_->Mult(r, w); }
                else A_->Mult(v_[i], w);
                for (int k = 0; k <= i; ++k) { h(k, i) = w * v_[k]; w.Add(-h(k, i), v_[k]); }
                h(i + 1, i) = norm(w);
                v_[i + 1].Set(1.0 / h(i + 1, i), w);
                for (int k = 0; k < i; ++k) ApplyPlaneRotation(h(k, i), h(k + 1, i), cs[k], sn[k]);
                GeneratePlaneRotation(h(i, i), h(i + 1, i), cs[i], sn[i]);
                ApplyPlaneRotation(h(i, i), h(i + 1, i), cs[i], sn[i]);
                ApplyPlaneRotation(s[i], s[i + 1], cs[i], sn[i]);
                resid = std::fabs(s[i + 1]);
                history_.push_back(resid);
                if (print_level_ == 1) std::printf("   Pass : %2d   Iteration : %3d  ||B r|| = %g\n", (j - 1) / m + 1, j, resid);
                if (resid <= final_norm) { update(i); final_norm_ = resid; final_iter_ = j; converged_ = true; return; }
            }
            if (print_level_ == 1 && j <= max_iter_) std::printf("Restarting...\n");
            update(i - 1);
            A_->Mult(x, r);
            if (Prec_) { mfem::add(b, -1.0, r, w); Prec_->Mult(w, r); }
            else mfem::add(b, -1.0, r, r);
            beta = norm(r);
            if (beta <= final_norm) { final_norm_ = beta; final_iter_ = j; converged_ = true; return; }
        }
        final_norm_ = beta; final_iter_ = max_iter_; converged_ = false;
    }
    /// mfem::FGMRESSolver::Mult restated (flexible, right-preconditioned; monitor || r ||)
    void MultFGMRES(const mfem::Vector &b, mfem::Vector &x) const
    {
        const int n = Height(), m = restart_;
        r_.SetSize(n);
        mfem::Vector &r = r_;
        history_.clear(); stats_on_device_ = false; converged_ = false; final_iter_ = 0;
        std::vector<double> H((size_t)(m + 1) * m, 0.0), s(m + 1), cs(m + 1), sn(m + 1);
        auto h = [&](int i, int j) -> double & { return H[(size_t)j * (m + 1) + i]; };
        auto norm = [](const mfem::Vector &v) { return std::sqrt(v * v); };
        if (this->iterative_mode) { A_->Mult(x, r); mfem::add(b, -1.0, r, r); }
        else { x = 0.0; r = b; }
        double beta = norm(r), resid = beta;
        history_.push_back(beta);
        const double final_norm = std::max(rel_tol_ * beta, abs_tol_);
        if (beta <= final_norm) { final_norm_ = beta; converged_ = true; return; }
        if ((int)v_.size() < m + 1) v_.resize(m + 1);
        if ((int)zz_.size() < m + 1) zz_.resize(m + 1);
        auto update = [&](int k)
        {
            std::vector<double> y(s.begin(), s.begin() + k + 1);
            for (int i = k; i >= 0; --i)
            {
                y[i] /= h(i, i);
                for (int j = i - 1; j >= 0; --j) y[j] -= h(j, i) * y[i];
            }
            for (int j = 0; j <= k; ++j) x.Add(y[j], zz_[j]);
        };
        for (int j = 1; j <= max_iter_;)
        {
            v_[0].Set(1.0 / beta, r);
            std::fill(s.begin(), s.end(), 0.0);
            s[0] = beta;
            int i;
            for (i = 0; i < m && j <= max_iter_; ++i, ++j)
            {
                zz_[i].SetSize(n);
                if (Prec_) Prec_->Mult(v_[i], zz_[i]); else zz_[i] = v_[i];
                A_->Mult(zz_[i], r);
                for (int k = 0; k <= i; ++k) { h(k, i) = r * v_[k]; r.Add(-h(k, i), v_[k]); }
                h(i + 1, i) = norm(r);
                v_[i + 1].Set(1.0 / h(i + 1, i), r);
                for (int k = 0; k < i; ++k) ApplyPlaneRotation(h(k, i), h(k + 1, i), cs[k], sn[k]);
                GeneratePlaneRotation(h(i, i), h(i + 1, i), cs[i], sn[i]);
                ApplyPlaneRotation(h(i, i), h(i + 1, i), cs[i], sn[i]);
                ApplyPlaneRotation(s[i], s[i + 1], cs[i], sn[i]);
                resid = std::fabs(s[i + 1]);
                history_.push_back(resid);
                if (print_level_ == 1) std::printf("   Pass : %2d   Iteration : %3d  || r || = %g\n", (j - 1) / m + 1, j, resid);
                if (resid <= final_norm) { update(i); final_norm_ = resid; final_iter_ = j; converged_ = true; return; }
            }
            update(i - 1);
            A_->Mult(x, r);
            mfem::add(b, -1.0, r, r);
            beta = norm(r);
            if (beta <= final_norm) { final_norm_ = beta; final_iter_ = j; converged_ = true; return; }
        }
        final_norm_ = beta; final_iter_ = max_iter_; converged_ = false;
    }
    /// mfem::BiCGSTABSolver::Mult restated; history[i] = ||r|| after iteration i
    void MultBiCGSTAB(const mfem::Vector &b, mfem::Vector &x) const
    {
        const int n = Height();
        mfem::Vector &r = r_, &p = d_, &v = z_;
        r.SetSize(n); p.SetSize(n); v.SetSize(n);
        if ((int)v_.size() < 5) v_.resize(5);
        mfem::Vector &rtilde = v_[0], &phat = v_[1], &sv = v_[2], &shat = v_[3], &t = v_[4];
        for (int q = 0; q < 5; ++q) v_[q].SetSize(n);
        history_.clear(); stats_on_device_ = false; converged_ = false; final_iter_ = 0;
        auto norm = [](const mfem::Vector &w) { return std::sqrt(w * w); };
        if (this->iterative_mode) { A_->Mult(x, r); mfem::add(b, -1.0, r, r); }
        else { x = 0.0; r = b; }
        rtilde = r;
        double resid = norm(r), rho_1 = 0, rho_2 = 1, alpha = 1, beta, omega = 1;
        history_.push_back(resid);
        const double tol_goal = std::max(resid * rel_tol_, abs_tol_);
        if (resid <= tol_goal) { final_norm_ = resid; converged_ = true; return; }
        for (int i = 1; i <= max_iter_; ++i)
        {
            rho_1 = rtilde * r;
            if (rho_1 == 0.0) { final_norm_ = resid; final_iter_ = i; return; }
            if (i == 1) p = r;
            else
            {
                beta = (rho_1 / rho_2) * (alpha / omega);
                mfem::add(p, -omega, v, p);
                mfem::add(r, beta, p, p);
            }
            if (Prec_) Prec_->Mult(p, phat); else phat = p;
            A_->Mult(phat, v);
            alpha = rho_1 / (rtilde * v);
            mfem::add(r, -alpha, v, sv);
            resid = norm(sv);
            if (resid < tol_goal)
            {
                x.Add(alpha, phat);
                history_.push_back(resid);
                final_norm_ = resid; final_iter_ = i; converged_ = true; return;
            }
            if (Prec_) Prec_->Mult(sv, shat); else shat = sv;
            A_->Mult(shat, t);
            omega = (t * sv) / (t * t);
            x.Add(alpha, phat);
            x.Add(omega, shat);
            mfem::add(sv, -omega, t, r);
            rho_2 = rho_1;
            resid = norm(r);
            history_.push_back(resid);
            if (print_level_ == 1) std::printf("   Iteration : %3d   ||r|| = %g\n", i, resid);
            if (resid < tol_goal) { final_norm_ = resid; final_iter_ = i; converged_ = true; return; }
            if (omega == 0.0) { final_norm_ = resid; final_iter_ = i; return; }
        }
        final_norm_ = resid; final_iter_ = max_iter_;
    }
    /// mfem::MINRESSolver::Mult restated (van der Vorst, Fig. 6.9, with an SPD preconditioner); history = |eta|
    void MultMINRES(const mfem::Vector &b, mfem::Vector &x) const
    {
        const int n = Height();
        if ((int)v_.size() < 6) v_.resize(6);
        for (int q = 0; q < 6; ++q) v_[q].SetSize(n);
        mfem::Vector *v0 = &v_[0], *v1 = &v_[1], *w0 = &v_[2], *w1 = &v_[3], *q = &v_[4], *u1 = &v_[5];
        history_.clear(); stats_on_device_ = false; converged_ = true; final_iter_ = 0;
        if (!this->iterative_mode) { *v1 = b; x = 0.0; }
        else { A_->Mult(x, *v1); mfem::add(b, -1.0, *v1, *v1); }
        if (Prec_) Prec_->Mult(*v1, *u1);
        mfem::Vector *z = Prec_ ? u1 : v1;
        double beta, eta, gamma0 = 1.0, gamma1 = 1.0, sigma0 = 0.0, sigma1 = 0.0, alpha, delta, rho1, rho2, rho3;
        eta = beta = std::sqrt((*z) * (*v1));
        history_.push_back(eta);
        const double norm_goal = std::max(rel_tol_ * eta, abs_tol_);
        int it = 0;
        if (eta > norm_goal)
        {
            bool done = false;
            for (it = 1; it <= max_iter_; ++it)
            {
                *v1 *= 1.0 / beta;
                if (Prec_) *u1 *= 1.0 / beta;
                z = Prec_ ? u1 : v1;
                A_->Mult(*z, *q);
                alpha = (*z) * (*q);
                if (it > 1) q->Add(-beta, *v0);
                mfem::add(*q, -alpha, *v1, *v0);
                delta = gamma1 * alpha - gamma0 * sigma1 * beta;
                rho3 = sigma0 * beta;
                rho2 = sigma1 * alpha + gamma0 * gamma1 * beta;
                if (!Prec_) beta = std::sqrt((*v0) * (*v0));
                else { Prec_->Mult(*v0, *q); beta = std::sqrt((*v0) * (*q)); }
                rho1 = std::hypot(delta, beta);
                if (it == 1) w0->Set(1.0 / rho1, *z);
                else if (it == 2) mfem::add(1.0 / rho1, *z, -rho2 / rho1, *w1, *w0);
                else { mfem::add(-rho3 / rho1, *w0, -rho2 / rho1, *w1, *w0); w0->Add(1.0 / rho1, *z); }
                gamma0 = gamma1; gamma1 = delta / rho1;
                x.Add(gamma1 * eta, *w0);
                sigma0 = sigma1; sigma1 = beta / rho1;
                eta = -sigma1 * eta;
                history_.push_back(std::fabs(eta));
                if (print_level_ == 1) std::printf("MINRES: iteration %3d: ||r||_B = %g\n", it, std::fabs(eta));
                if (std::fabs(eta) <= norm_goal) { done = true; break; }
                if (Prec_) std::swap(u1, q);
                std::swap(v0, v1);
                std::swap(w0, w1);
            }
            if (!done) { converged_ = false; --it; }
        }
        final_iter_ = it; final_norm_ = std::fabs(eta);
    }
    static void GeneratePlaneRotation(double &dx, double &dy, double &cs, double &sn)
    {
        if (dy == 0.0) { cs = 1.0; sn = 0.0; }
        else if (std::fabs(dy) > std::fabs(dx)) { const double t = dx / dy; sn = 1.0 / std::sqrt(1.0 + t * t); cs = t * sn; }
        else { const double t = dy / dx; cs = 1.0 / std::sqrt(1.0 + t * t); sn = t * cs; }
    }
    static void ApplyPlaneRotation(double &dx, double &dy, double cs, double sn)
    {
        const double t = cs * dx + sn * dy;
        dy = -sn * dx + cs * dy;
        dx = t;
    }
    void MultDeviceResident(const mfem::Vector &b, mfem::Vector &x) const
    {
        pe_ctx *ctx = Device::Get();
        const int n = Height();
        r_.SetSize(n); d_.SetSize(n); z_.SetSize(n);
        if (!slots_) PE_CALL(pe_scalars_create(ctx, PE_PCG_HIST + max_iter_ + 2, &slots_));
        stats_on_device_ = true;
        if (this->iterative_mode) { A_->Mult(x, r_); mfem::add(b, -1.0, r_, r_); }
        else { r_ = b; x = 0.0; }
        if (Prec_) { Prec_->Mult(r_, z_); d_ = z_; }
        else d_ = r_;
        PE_CALL(pe_vec_dot_dev(d_.Read(), r_.Read(), slots_, PE_PCG_DOT));
        PE_CALL(pe_pcg_scalar_step(ctx, slots_, 0, 0, max_iter_, rel_tol_, abs_tol_));
        A_->Mult(d_, z_);
        PE_CALL(pe_vec_dot_dev(z_.Read(), d_.Read(), slots_, PE_PCG_DOT));
        PE_CALL(pe_pcg_scalar_step(ctx, slots_, 1, 0, max_iter_, rel_tol_, abs_tol_));
        for (int i = 1; i <= max_iter_; ++i)
        {
            PE_CALL(pe_vec_axpy_dev(slots_, PE_PCG_ALPHA, 1.0, d_.Read(), x.ReadWrite()));
            PE_CALL(pe_vec_axpy_dev(slots_, PE_PCG_ALPHA, -1.0, z_.Read(), r_.ReadWrite()));
            if (Prec_) { Prec_->Mult(r_, z_); PE_CALL(pe_vec_dot_dev(r_.Read(), z_.Read(), slots_, PE_PCG_DOT)); }
            else PE_CALL(pe_vec_dot_dev(r_.Read(), r_.Read(), slots_, PE_PCG_DOT));
            PE_CALL(pe_pcg_scalar_step(ctx, slots_, 2, i, max_iter_, rel_tol_, abs_tol_));
            if (i == max_iter_) break;
            PE_CALL(pe_vec_xpby_dev(Prec_ ? z_.Read() : r_.Read(), slots_, PE_PCG_BETA, d_.ReadWrite()));   // d = z + beta d
            A_->Mult(d_, z_);
            PE_CALL(pe_vec_dot_dev(d_.Read(), z_.Read(), slots_, PE_PCG_DOT));
            PE_CALL(pe_pcg_scalar_step(ctx, slots_, 3, i, max_iter_, rel_tol_, abs_tol_));
        }
    }
    /// statistics of a device-resident solve are downloaded on demand only
    void FetchStats() const
    {
        if (!stats_on_device_ || !slots_) return;
        std::vector<double> h(PE_PCG_HIST + max_iter_ + 2);
        PE_CALL(pe_scalars_download(Device::Get(), slots_, (int)h.size(), h.data()));
        const int nh = (int)h[PE_PCG_NHIST];
        history_.assign(h.begin() + PE_PCG_HIST, h.begin() + PE_PCG_HIST + nh);
        converged_ = h[PE_PCG_CONVERGED] != 0.0;
        final_iter_ = (int)h[PE_PCG_FINAL_ITER];
        // a negative initial (B r, r) stops at once and is reported as it is, as Mult does
        final_norm_ = h[PE_PCG_NOM0] < 0.0 ? h[PE_PCG_NOM0] : std::sqrt(std::fabs(h[PE_PCG_BETANOM]));
        stats_on_device_ = false;
    }
    void _do_set_operator(const Op_Ptr &op) override { A_ = op; }
    Op_Ptr A_;
    std::shared_ptr<mfem::Solver> Prec_;
    int print_level_ = -1, max_iter_ = 10;
    double rel_tol_ = 0.0, abs_tol_ = 0.0;
    bool final_paragraph_ = false, gmres_ = false;
    int restart_ = 50;
    int method_ = 0;                            // 0 PCG/GMRES, 1 FGMRES, 2 MINRES, 3 BiCGStab
    mutable std::vector<mfem::Vector> v_, zz_;  // Krylov bases of (F)GMRES / work vectors
    mutable mfem::Vector r_, d_, z_;
    mutable std::vector<double> history_;
    mutable bool converged_ = false;
    mutable int final_iter_ = 0;
    mutable double final_norm_ = 0.0;
    mutable double *slots_ = nullptr;          // device scalars of the device-resident mode
    mutable bool stats_on_device_ = false;
};

class KrylovSolverFactory : public SolverFactory
{
    std::unique_ptr<mfem::Solver> _do_build_solver(const Op_Ptr &op, SolverState &state) const override
    {
        auto my_state = dynamic_cast<NestedSolverState *>(&state);
        PARELAG_ASSERT(my_state);
        std::shared_ptr<mfem::Solver> prec;
        if (Prec_Factory_)
        {
            auto prec_state = std::shared_ptr<SolverState>{Prec_Factory_->GetDefaultState()};
            if (my_state->IsSubState("Preconditioner")) prec_state->MergeState(*my_state->GetSubState("Preconditioner"));
            prec_state->MergeState(*my_state);
            prec = Prec_Factory_->BuildSolver(op, *prec_state);
            prec->iterative_mode = false;
        }
        return make_unique<KrylovSolver>(op, prec, GetParameters());
    }
    void _do_set_default_parameters() override
    {
        auto &p = GetParameters();
        p.Get<int>("Print level", -1); p.Get<double>("Relative tolerance", 0.0); p.Get<double>("Absolute tolerance", 0.0);
        p.Get<int>("Maximum iterations", 10); p.Get<int>("Restart size", 50); p.Get<bool>("Print final paragraph", false);
        p.Get<bool>("Time preconditioner setup", false); p.Get<std::string>("Timer name suffix", "");
    }
    void _do_initialize(const ParameterList &) override
    {
        PARELAG_ASSERT(HasValidSolverLibrary());
        std::string prec_name = GetParameters().Get("Preconditioner", "None");
        if (prec_name != "None") Prec_Factory_ = GetSolverLibrary().GetSolverFactory(prec_name);
    }
    std::shared_ptr<SolverFactory> Prec_Factory_;
};

// ------------------------------------------------------------------ Hierarchy
class Hierarchy : public Solver
{
public:
    Hierarchy(const Op_Ptr &A, int NumLevels)
        : Solver(A->Height(), A->Width(), false), CoarseResids_(NumLevels), CoarseSols_(NumLevels), CycleMu_(NumLevels, 0)
    {
        for (int l = 0; l < NumLevels; ++l) Levels_.push_back(std::make_shared<Level>(l));
        Levels_.front()->Set<Op_Ptr>("A", A);
    }
    int GetNumLevels() const noexcept { return (int)Levels_.size(); }
    /// the rows FixZeroRows rewrote in the operator of level l (ZeroRows), in its diagonal block `block` on a blocked
    /// hierarchy, checked again by SetOperator
    void SetZeroRows(int l, mfem::Vector rows, int block = 0)
    {
        if ((int)ZeroRows_.size() <= l) ZeroRows_.resize(l + 1);
        if ((int)ZeroRows_[l].size() <= block) ZeroRows_[l].resize(block + 1);
        ZeroRows_[l][block] = std::move(rows);
    }
    Level &GetLevel(int l) { return *Levels_.at(l); }
    std::vector<std::shared_ptr<Level>>::const_iterator begin() const { return Levels_.begin(); }
    std::vector<std::shared_ptr<Level>>::const_iterator end() const { return Levels_.end(); }
    void SetImplicitTranspose(bool v) noexcept { ImplicitTranspose_ = v; }
    /// Hierarchy::SetCycle (ParELAG_Hierarchy.cpp:57-106): how often a level recurses into the next coarser one (Mu = -1 skips
    /// a level); a recorded cycle is dropped and re-recorded by the next Mult.  (The reference's one-argument form tests
    /// `Mu >= 0` where its message says "Cannot set Mu<0 on every level"; the intended check is applied here.)
    void SetCycle(int Mu)
    {
        PARELAG_TEST_FOR_EXCEPTION(Mu < 0, std::runtime_error, "Hierarchy::SetCycle(): Cannot set Mu<0 on every level.");
        CycleMu_.assign(1, Mu);
        DropRecordedCycle();
    }
    void SetCycle(int Mu, int LevelID)
    {
        PARELAG_TEST_FOR_EXCEPTION(LevelID < 0 || LevelID >= (int)Levels_.size(), std::runtime_error,
                                   "Hierarchy::SetCycle(): LevelID=" << LevelID << " greater than current number of levels (" << Levels_.size() << ").");
        if (CycleMu_.size() != Levels_.size()) CycleMu_ = std::vector<int>(Levels_.size(), CycleMu_.empty() ? 0 : CycleMu_[0]);
        CycleMu_[LevelID] = Mu;
        DropRecordedCycle();
    }
    void SetCycle(std::vector<int> Mus)
    {
        PARELAG_TEST_FOR_EXCEPTION(Mus.size() != Levels_.size(), std::runtime_error,
                                   "Hierarchy::SetCycle(): Input vector has wrong size (" << Mus.size() << "). Correct size is " << Levels_.size() << ".");
        CycleMu_.swap(Mus);
        DropRecordedCycle();
    }
    ~Hierarchy() override { pe_graph_free(graph_); pe_program_free(program_); }
    /// replay the V-cycle as one persistent program kernel (preferred) or one CUDA graph when
    /// every level solver is capture-safe (both default on)
    void SetUseGraph(bool v) noexcept { use_graph_ = v; }
    void SetUseProgram(bool v) noexcept { use_program_ = v; }
    bool UsesGraph() const noexcept { return graph_ != nullptr; }
    bool UsesProgram() const noexcept { return program_ != nullptr; }
    pe_program *GetProgram() const noexcept { return program_; }
    /// how the last preconditioner-mode Mult ran: 0 directly, 1 as a CUDA graph, 2 as the persistent program
    int LastReplayMode() const noexcept { return last_mode_; }
    bool CaptureSafe() const override
    {
        for (auto &lev : Levels_)
            for (const char *key : {"PreSmoother", "PostSmoother", "CoarseSolver"})
                if (lev->IsValidKey(key))
                    if (!SolverCaptureSafe(dynamic_cast<const mfem::Solver *>(lev->Get<Op_Ptr>(key).get()))) return false;
        return true;
    }

    /// one V-cycle (the "Cycle type" parameter is never read by the reference, SURVEY fact 4)
    void Mult(const mfem::Vector &rhs, mfem::Vector &sol) const override
    {
        SetupColour();
        if (this->IsPreconditioner())
        {
            if (ReplayGraph(rhs, sol)) return;
            Cycle(rhs, sol);
        }
        else
        {
            mfem::Vector rhs_view(rhs.Size()), sol_view(sol.Size());
            Levels_.front()->Get<Op_Ptr>("A")->Mult(sol, rhs_view);
            rhs_view *= -1.0;
            rhs_view += rhs;
            Cycle(rhs_view, sol_view);
            sol += sol_view;
        }
    }
    /// Levels are visited as in the reference.  On a colour-numbered level (SetupColour) RHS and SOL are in the level's
    /// colour numbering and SolMode tells the pre-smoother what SOL holds (HypreSmootherWrapper::MultColour).
    void Iterate(const mfem::Vector &RHS, mfem::Vector &SOL, int StartLevel, int NumIterations, bool CycleThisLevel,
                 int SolMode = 0) const
    {
        for (int iteration = 1; iteration <= NumIterations; ++iteration)
        {
            if (StartLevel == (int)Levels_.size() - 1)
            {
                Level &Coarse = *Levels_[StartLevel];
                if (Coarse.IsValidKey("CoarseSolver")) Coarse.Get<Op_Ptr>("CoarseSolver")->Mult(RHS, SOL);
                else
                {
                    if (Coarse.IsValidKey("PreSmoother")) Coarse.Get<Op_Ptr>("PreSmoother")->Mult(RHS, SOL);
                    if (Coarse.IsValidKey("PostSmoother")) Coarse.Get<Op_Ptr>("PostSmoother")->Mult(RHS, SOL);
                }
                continue;
            }
            Level &Fine = *Levels_[StartLevel];
            Level &Coarse = *Levels_[StartLevel + 1];
            const int l = StartLevel;
            const bool fine_c = IsColourLevel(l), coarse_c = IsColourLevel(l + 1);
            pe_ctx *ctx = Device::Get();
            if (fine_c) SmoothColour(*Fine.Get<Op_Ptr>("PreSmoother"), RHS, SOL, iteration == 1 ? SolMode : 0);
            else if (Fine.IsValidKey("PreSmoother")) Fine.Get<Op_Ptr>("PreSmoother")->Mult(RHS, SOL);
            // residual (K1+K7 fused: r = b - A x in one pass)
            tmp_resid_[StartLevel].SetSize(RHS.Size());
            if (fine_c) PE_CALL(pe_residual(ctx, cres_[l].get(), SOL.Read(), RHS.Read(), tmp_resid_[l].Write()));
            else mg_utils::ComputeResidual(*Fine.Get<Op_Ptr>("A"), SOL, RHS, tmp_resid_[StartLevel]);
            auto &P = Coarse.Get<Op_Ptr>("P");
            if (fine_c || coarse_c) PE_CALL(pe_spmv(ctx, 1.0, crestrict_[l].get(), tmp_resid_[l].Read(), 0.0, CoarseResids_[l + 1].Write()));
            else if (ImplicitTranspose_ || !Fine.IsKey("R")) P->MultTranspose(tmp_resid_[StartLevel], CoarseResids_[StartLevel + 1]);
            else Fine.Get<Op_Ptr>("R")->Mult(tmp_resid_[StartLevel], CoarseResids_[StartLevel + 1]);
            // a colour-numbered coarse level starts from a zero guess without the fill (SolMode 1)
            if (!coarse_c) CoarseSols_[StartLevel + 1] = 0.0;
            int cycle_times = 0;
            if (CycleThisLevel && CycleMu_.size() > 1) cycle_times = CycleMu_[StartLevel];
            for (int cycle = 0; cycle <= cycle_times; ++cycle)
                Iterate(CoarseResids_[StartLevel + 1], CoarseSols_[StartLevel + 1], StartLevel + 1, 1, false,
                        coarse_c && cycle == 0 ? 1 : 0);
            // SOL += P * e  (K1 with beta = 1: prolongation and correction in one pass)
            auto P_hyp = std::dynamic_pointer_cast<mfem::HypreParMatrix>(P);
            if (fine_c || coarse_c) PE_CALL(pe_spmv(ctx, 1.0, cprolong_[l].get(), CoarseSols_[l + 1].Read(), 1.0, SOL.ReadWrite()));
            else if (P_hyp) P_hyp->Mult(1.0, CoarseSols_[StartLevel + 1], 1.0, SOL);
            else
            {
                tmp_correct_[StartLevel].SetSize(P->Height());
                P->Mult(CoarseSols_[StartLevel + 1], tmp_correct_[StartLevel]);
                SOL += tmp_correct_[StartLevel];
            }
            if (fine_c) SmoothColour(*Fine.Get<Op_Ptr>("PostSmoother"), RHS, SOL, 0);
            else if (Fine.IsValidKey("PostSmoother")) Fine.Get<Op_Ptr>("PostSmoother")->Mult(RHS, SOL);
        }
    }
    void Finalize()
    {
        tmp_resid_.resize(Levels_.size());
        tmp_correct_.resize(Levels_.size());
        for (size_t l = 0; l < Levels_.size(); ++l)
        {
            const int n = Levels_[l]->Get<Op_Ptr>("A")->Height();
            CoarseResids_[l].SetSize(n);
            CoarseSols_[l].SetSize(n);
        }
    }
private:
    bool IsColourLevel(int l) const { return colour_state_ > 0 && l < (int)colour_.size() && colour_[l].npad > 0; }
    static void SmoothColour(const mfem::Operator &S, const mfem::Vector &B, mfem::Vector &X, int mode)
    {
        if (auto h = dynamic_cast<const HiptmairSmoother *>(&S)) h->MultColour(B, X, mode);
        else dynamic_cast<const HypreSmootherWrapper &>(S).MultColour(B, X, mode);
    }
    static ColourNumbering SmootherNumbering(const mfem::Operator &S)
    {
        if (auto h = dynamic_cast<const HiptmairSmoother *>(&S)) return h->Numbering();
        if (auto w = dynamic_cast<const HypreSmootherWrapper *>(&S)) return w->Numbering();
        return {};
    }
    /// sol = one V-cycle from a zero guess.  With a colour-numbered fine level the right-hand side is renumbered on
    /// entry, in the same pass as the first colour of the pre-smoother's first sweep, and the solution on exit.
    void Cycle(const mfem::Vector &rhs, mfem::Vector &sol) const
    {
        if (!IsColourLevel(0))
        {
            sol = 0.0;
            Iterate(rhs, sol, 0, 1, false);
            return;
        }
        pe_smoother *s = PrimaryHandle(*Levels_[0]->Get<Op_Ptr>("PreSmoother"));
        PE_CALL(pe_smoother_colour_in(s, rhs.Read(), CoarseResids_[0].Write(), CoarseSols_[0].Write()));
        Iterate(CoarseResids_[0], CoarseSols_[0], 0, 1, false, 2);
        PE_CALL(pe_smoother_colour_out(s, CoarseSols_[0].Read(), sol.Write()));
    }
    static pe_smoother *PrimaryHandle(const mfem::Operator &S)
    {
        if (auto h = dynamic_cast<const HiptmairSmoother *>(&S)) return h->PrimaryHandle();
        return dynamic_cast<const HypreSmootherWrapper &>(S).Handle();
    }
    /// Colour-numbered levels (one rank): a level whose pre- and post-smoother are one multicolour SELL Gauss-Seidel
    /// smoother, or one Hiptmair smoother of two, keeps its vectors in that smoother's colour numbering for the whole
    /// cycle.  Its residual, restriction, prolongation (and Hiptmair's D, D^T) run on renumbered copies built here, so
    /// the smoothers need no renumbering passes.  Every other level keeps the natural numbering.
    void SetupColour() const
    {
        if (colour_state_ != 0) return;
        colour_state_ = -1;
        pe_ctx *ctx = Device::Get();
        if (pe_ctx_nranks(ctx) != 1 || pe_ctx_is_capturing(ctx) || pe_ctx_is_recording(ctx)) return;
        const int L = (int)Levels_.size();
        colour_.assign(L, ColourNumbering());
        cres_.assign(L, nullptr); crestrict_.assign(L, nullptr); cprolong_.assign(L, nullptr);
        bool any = false;
        for (int l = 0; l + 1 < L; ++l)
        {
            Level &lev = *Levels_[l];
            if (!lev.IsValidKey("PreSmoother") || !lev.IsValidKey("PostSmoother")) continue;
            auto pre = lev.Get<Op_Ptr>("PreSmoother");
            if (pre != lev.Get<Op_Ptr>("PostSmoother")) continue;
            auto A = std::dynamic_pointer_cast<mfem::HypreParMatrix>(lev.Get<Op_Ptr>("A"));
            auto P = std::dynamic_pointer_cast<mfem::HypreParMatrix>(Levels_[l + 1]->Get<Op_Ptr>("P"));
            if (!A || !P || !(ImplicitTranspose_ || !lev.IsKey("R"))) continue;
            const ColourNumbering c = SmootherNumbering(*pre);
            if (c.npad == 0) continue;
            colour_[l] = c;
            cres_[l] = RenumberedCopy(*A, false, c, c);
            if (auto h = dynamic_cast<HiptmairSmoother *>(pre.get())) h->SetupColour(cres_[l]);
            any = true;
        }
        if (!any) return;
        for (int l = 0; l + 1 < L; ++l)
        {
            if (colour_[l].npad == 0 && colour_[l + 1].npad == 0) continue;
            auto &P = dynamic_cast<const mfem::HypreParMatrix &>(*Levels_[l + 1]->Get<Op_Ptr>("P"));
            crestrict_[l] = RenumberedCopy(P, true, colour_[l + 1], colour_[l]);
            cprolong_[l] = RenumberedCopy(P, false, colour_[l], colour_[l + 1]);
        }
        for (int l = 0; l < L; ++l)
            if (colour_[l].npad > 0)
            {
                // padding entries are allocated zeroed and never written
                CoarseResids_[l] = mfem::Vector(); CoarseResids_[l].SetSize(colour_[l].npad);
                CoarseSols_[l] = mfem::Vector(); CoarseSols_[l].SetSize(colour_[l].npad);
                tmp_resid_[l] = mfem::Vector(); tmp_resid_[l].SetSize(colour_[l].npad);
            }
        colour_state_ = 1;
    }
    /// Preconditioner-mode V-cycle through a CUDA graph: the first call with a given (rhs, sol)
    /// buffer pair runs directly (it allocates work vectors and builds lazy matrix formats), the
    /// second call records the cycle, later calls replay it.  Returns false when the cycle has to
    /// be run directly.
    bool ReplayGraph(const mfem::Vector &rhs, mfem::Vector &sol) const
    {
        pe_ctx *ctx = Device::Get();
        last_mode_ = 0;
        if ((!use_graph_ || graph_failed_) && (!use_program_ || program_failed_)) return false;
        if (pe_ctx_is_capturing(ctx) || pe_ctx_is_recording(ctx) || pe_ctx_is_profiling(ctx)) return false;
        // multi-rank: the NCCL halo exchanges and all-reduces are captured with the kernels (every
        // rank captures and replays the same sequence); the persistent program is single-rank only
        const bool multi = pe_ctx_nranks(ctx) > 1;
        if (capture_safe_ < 0) capture_safe_ = CaptureSafe() ? 1 : 0;
        if (!capture_safe_) return false;
        const void *rp = pe_vec_device_ptr(const_cast<pe_vec *>(rhs.Read()));
        const void *sp = pe_vec_device_ptr(sol.Write());
        if (program_ && graph_rhs_ == rp && graph_sol_ == sp)
        {
            PE_CALL(pe_program_launch(ctx, program_));
            last_mode_ = 2;
            return true;
        }
        if (graph_ && graph_rhs_ == rp && graph_sol_ == sp)
        {
            PE_CALL(pe_graph_launch(ctx, graph_));
            last_mode_ = 1;
            return true;
        }
        if (warm_rhs_ != rp || warm_sol_ != sp) { warm_rhs_ = rp; warm_sol_ = sp; return false; }
        pe_graph_free(graph_);
        graph_ = nullptr;
        pe_program_free(program_);
        program_ = nullptr;
        if (!multi && use_program_ && !program_failed_ && pe_program_begin(ctx) == 0)
        {
            // record the cycle: every C-ABI call below appends an op instead of launching
            bool rec_ok = true;
            try { Cycle(rhs, sol); }
            catch (...) { rec_ok = false; }
            pe_program *p = nullptr;
            if (pe_program_end(ctx, &p) == 0 && rec_ok)
            {
                program_ = p; graph_rhs_ = rp; graph_sol_ = sp;
                PE_CALL(pe_program_launch(ctx, program_));
                last_mode_ = 2;
                return true;
            }
            pe_program_free(p);
            program_failed_ = true;
        }
        if (!use_graph_ || graph_failed_) return false;
        if (pe_graph_begin(ctx) != 0) { graph_failed_ = true; return false; }
        bool ok = true;
        try { Cycle(rhs, sol); }
        catch (...) { ok = false; }
        pe_graph *g = nullptr;
        if (pe_graph_end(ctx, &g) != 0 || !ok)
        {
            pe_graph_free(g);
            graph_failed_ = true;
            return false;           // the caller runs the cycle directly
        }
        graph_ = g; graph_rhs_ = rp; graph_sol_ = sp;
        PE_CALL(pe_graph_launch(ctx, graph_));
        last_mode_ = 1;
        return true;
    }
    void DropRecordedCycle() const
    {
        pe_graph_free(graph_); graph_ = nullptr;
        pe_program_free(program_); program_ = nullptr;
        graph_rhs_ = graph_sol_ = warm_rhs_ = warm_sol_ = nullptr;
    }
    /// the FixZeroRows step of level l (block b) of an update, when the build applied it there
    void FixRecordedZeroRows(mfem::HypreParMatrix &A, int l, int b, const std::string &where) const
    {
        if (l < (int)ZeroRows_.size() && b < (int)ZeroRows_[l].size() && ZeroRows_[l][b].Size() > 0)
            FixSameZeroRows(A, ZeroRows_[l][b], where);
    }
    /// single-form levels: A_l = P_l^T A_{l-1} P_l into a copy of the held A_l's pattern, then FixZeroRows
    std::vector<Op_Ptr> GalerkinProducts(const Op_Ptr &op) const
    {
        auto A = std::dynamic_pointer_cast<mfem::HypreParMatrix>(op);
        auto A0 = std::dynamic_pointer_cast<mfem::HypreParMatrix>(Levels_.front()->Get<Op_Ptr>("A"));
        PARELAG_TEST_FOR_EXCEPTION(!A || !A0, std::runtime_error, "Hierarchy::SetOperator(): operator must be a HypreParMatrix");
        CheckSamePattern(*A0, *A, "Hierarchy");
        std::vector<Op_Ptr> newA(Levels_.size());
        newA[0] = A;
        for (size_t l = 1; l < Levels_.size(); ++l)
        {
            auto &P = dynamic_cast<const mfem::HypreParMatrix &>(*Levels_[l]->Get<Op_Ptr>("P"));
            auto Ac = CopyOf(dynamic_cast<const mfem::HypreParMatrix &>(*Levels_[l]->Get<Op_Ptr>("A")));
            PE_CALL(pe_rap_numeric(Device::Get(), nullptr, dynamic_cast<const mfem::HypreParMatrix &>(*newA[l - 1]).Handle(),
                                   P.Handle(), Ac->Handle()));
            FixRecordedZeroRows(*Ac, (int)l, 0, "the operator of level " + std::to_string(l));
            newA[l] = Ac;
        }
        return newA;
    }
    /// blocked levels (buildBlockedHierarchyFromDeRhamSequence): block (i,j) of A_l = P_i^T A_{l-1}(i,j) P_j into a copy
    /// of the held block's pattern, then FixZeroRows on the diagonal blocks where the build applied it
    std::vector<Op_Ptr> BlockGalerkinProducts(const MfemBlockOperator &held, const Op_Ptr &op) const
    {
        std::vector<Op_Ptr> newA(Levels_.size());
        newA[0] = SameBlockStructure(held, op, "Hierarchy");
        auto hyp = [](const mfem::Operator &M) -> const mfem::HypreParMatrix & { return dynamic_cast<const mfem::HypreParMatrix &>(M); };
        for (size_t l = 1; l < Levels_.size(); ++l)
        {
            auto &Af = dynamic_cast<const MfemBlockOperator &>(*newA[l - 1]);
            auto &Ac = dynamic_cast<const MfemBlockOperator &>(*Levels_[l]->Get<Op_Ptr>("A"));
            auto &P = dynamic_cast<const MfemBlockOperator &>(*Levels_[l]->Get<Op_Ptr>("P"));
            auto next = std::make_shared<MfemBlockOperator>(Ac.CopyRowOffsets());
            for (size_t i = 0; i < Ac.GetNumBlockRows(); ++i)
                for (size_t j = 0; j < Ac.GetNumBlockCols(); ++j)
                {
                    if (Ac.IsZeroBlock(i, j)) continue;
                    auto blk = CopyOf(hyp(Ac.GetBlock(i, j)));
                    PE_CALL(pe_rap_numeric(Device::Get(), hyp(P.GetBlock(i, i)).Handle(), hyp(Af.GetBlock(i, j)).Handle(),
                                           hyp(P.GetBlock(j, j)).Handle(), blk->Handle()));
                    if (i == j)
                        FixRecordedZeroRows(*blk, (int)l, (int)i, "block (" + std::to_string(i) + "," + std::to_string(i) +
                                                                  ") of the operator of level " + std::to_string(l));
                    next->SetBlock(i, j, blk);
                }
            newA[l] = next;
        }
        return newA;
    }
    /// New values on the same pattern (one rank): the state BuildSolver(op) would produce with the same sequence,
    /// parameters and boundary labels.  Level 0 adopts op; A_l = P_l^T A_{l-1} P_l is recomputed by the numeric product
    /// into a copy of the held A_l's pattern (on a blocked hierarchy block by block, P_i^T A_{l-1}(i,j) P_j), then
    /// FixZeroRows; Hiptmair's D^T A D likewise.  Every check (rank count, operator type, block structure, patterns, the
    /// recorded FixZeroRows rows) runs before anything is changed, so a refused call leaves the hierarchy as it was.
    /// Then the smoothers, the coarse solver (a Krylov solver's preconditioner first) and the colour-numbered residual
    /// copies take the new operators, and the recorded cycle is dropped: the next two preconditioner calls run directly
    /// and record again.
    void _do_set_operator(const Op_Ptr &op) override
    {
        pe_ctx *ctx = Device::Get();
        PARELAG_TEST_FOR_EXCEPTION(pe_ctx_nranks(ctx) != 1, std::runtime_error,
                                   "Hierarchy::SetOperator(): more than one rank is not supported; build a new solver");
        const int L = (int)Levels_.size();
        Timer galerkin = TimeManager::AddTimer("SetOperator: Galerkin products");
        auto blocked = std::dynamic_pointer_cast<MfemBlockOperator>(Levels_.front()->Get<Op_Ptr>("A"));
        const std::vector<Op_Ptr> newA = blocked ? BlockGalerkinProducts(*blocked, op) : GalerkinProducts(op);
        galerkin.Stop();
        // the auxiliary operator of every Hiptmair smoother, once per object (pre- and post-smoother are often one)
        Timer aux_timer = TimeManager::AddTimer("SetOperator: Hiptmair auxiliary operators");
        std::vector<std::pair<HiptmairSmoother *, Op_Ptr>> aux;
        for (int l = 0; l + 1 < L; ++l)
            for (const char *key : {"PreSmoother", "PostSmoother"})
                if (Levels_[l]->IsValidKey(key))
                    if (auto h = dynamic_cast<HiptmairSmoother *>(Levels_[l]->Get<Op_Ptr>(key).get()))
                        if (std::none_of(aux.begin(), aux.end(), [h](const std::pair<HiptmairSmoother *, Op_Ptr> &e) { return e.first == h; }))
                            aux.emplace_back(h, h->PrepareOperator(newA[l]));
        aux_timer.Stop();
        // nothing has changed so far; from here on the hierarchy takes the new operators
        Timer smoothers = TimeManager::AddTimer("SetOperator: smoothers and coarse solver");
        for (int l = 0; l < L; ++l)
        {
            Level &lev = *Levels_[l];
            lev.Reset<Op_Ptr>("A", newA[l]);
            Op_Ptr done;
            for (const char *key : {"PreSmoother", "PostSmoother"})
            {
                if (!lev.IsValidKey(key)) continue;
                auto S = lev.Get<Op_Ptr>(key);
                if (S == done) continue;      // pre- and post-smoother are often one object
                if (auto h = dynamic_cast<HiptmairSmoother *>(S.get()))
                    h->CommitOperator(newA[l], std::find_if(aux.begin(), aux.end(),
                                                            [h](const std::pair<HiptmairSmoother *, Op_Ptr> &e) { return e.first == h; })->second);
                else SetNestedOperator(*S, newA[l]);
                done = S;
            }
            if (lev.IsValidKey("CoarseSolver")) SetNestedOperator(*lev.Get<Op_Ptr>("CoarseSolver"), newA[l]);
        }
        smoothers.Stop();
        Timer colour = TimeManager::AddTimer("SetOperator: colour-numbered copies");
        for (int l = 0; l < L; ++l)
            if (colour_state_ > 0 && l < (int)cres_.size() && cres_[l])
                PE_CALL(pe_mat_renumbered_values(ctx, dynamic_cast<const mfem::HypreParMatrix &>(*newA[l]).Handle(),
                                                 colour_[l].pos, cres_[l].get()));
        colour.Stop();
        DropRecordedCycle();
    }
    std::vector<std::vector<mfem::Vector>> ZeroRows_;   // [level][block]: the rows FixZeroRows rewrote at build time (SetZeroRows)
    std::vector<std::shared_ptr<Level>> Levels_;
    mutable std::vector<mfem::Vector> CoarseResids_, CoarseSols_, tmp_resid_, tmp_correct_;
    std::vector<int> CycleMu_;
    bool ImplicitTranspose_ = true;
    bool use_graph_ = true, use_program_ = false;
    mutable bool graph_failed_ = false, program_failed_ = false;
    mutable pe_program *program_ = nullptr;
    mutable int capture_safe_ = -1;
    mutable int last_mode_ = 0;                 // LastReplayMode()
    mutable pe_graph *graph_ = nullptr;
    mutable const void *graph_rhs_ = nullptr, *graph_sol_ = nullptr, *warm_rhs_ = nullptr, *warm_sol_ = nullptr;
    mutable int colour_state_ = 0;              // SetupColour: 0 not yet, 1 some level colour-numbered, -1 none
    mutable std::vector<ColourNumbering> colour_;
    mutable std::vector<MatHandle> cres_, crestrict_, cprolong_;   // per level: A_l, P_{l+1}^T, P_{l+1} renumbered
};

/// Hierarchy.cpp:282-383: per coarse level P = ComputeTrueP(form, ess); A <- P^T A P; FixZeroRows
inline std::unique_ptr<Hierarchy> buildHierarchyFromDeRhamSequence(const Op_Ptr &A_in, const DeRhamSequence &Sequence,
                                                                   std::vector<int> &label_ess, int form, int MaxLevels)
{
    int NumLevels = 1;
    {
        auto seq = Sequence.ViewCoarserSequence();
        while (seq && (MaxLevels < 0 || NumLevels < MaxLevels)) { ++NumLevels; seq = seq->ViewCoarserSequence(); }
    }
    auto H = make_unique<Hierarchy>(A_in, NumLevels);
    H->SetImplicitTranspose(true);
    auto A = std::dynamic_pointer_cast<mfem::HypreParMatrix>(A_in);
    PARELAG_TEST_FOR_EXCEPTION(!A, std::runtime_error, "buildHierarchyFromDeRhamSequence(): operator must be a HypreParMatrix");
    const DeRhamSequence *seq = &Sequence;
    std::shared_ptr<DeRhamSequence> hold;
    const bool have_ess = !label_ess.empty();
    for (int l = 1; l < NumLevels; ++l)
    {
        Level &Coarse = H->GetLevel(l);
        std::shared_ptr<mfem::HypreParMatrix> P;
        if (have_ess)
        {
            mfem::Array<int> ess(label_ess.data(), (int)label_ess.size());
            P = seq->ComputeTrueP(form, ess);
        }
        else P = seq->ComputeTrueP(form);
        std::shared_ptr<mfem::HypreParMatrix> Ac{mfem::RAP(A.get(), P.get())};
        if (have_ess)
        {
            H->SetZeroRows(l, ZeroRows(*Ac));
            hypre_ParCSRMatrixFixZeroRows(*Ac);
        }
        Coarse.Set<Op_Ptr>("P", P);
        Coarse.Set<Op_Ptr>("A", Ac);
        A = Ac;
        hold = seq->CoarserSequence();
        seq = hold.get();
    }
    H->Finalize();
    return H;
}

/// Hierarchy.cpp:400-544: per block P_i = ComputeTrueP(forms[i], ess_i); A_c(i,j) = P_i^T A(i,j) P_j;
/// FixZeroRows on the diagonal blocks with essential conditions
inline std::unique_ptr<Hierarchy> buildBlockedHierarchyFromDeRhamSequence(const Op_Ptr &A_in, const DeRhamSequence &Sequence,
                                                                          std::vector<std::vector<int>> &label_ess,
                                                                          const std::vector<int> &forms, int MaxNumLevels)
{
    auto A = A_in;
    auto A_blocked = std::dynamic_pointer_cast<MfemBlockOperator>(A);
    PARELAG_TEST_FOR_EXCEPTION(!A_blocked, std::runtime_error, "buildBlockedHierarchyFromDeRhamSequence(...): A is not a MfemBlockOperator.");
    const int NumBlockRows = (int)A_blocked->GetNumBlockRows(), NumBlockCols = (int)A_blocked->GetNumBlockCols();
    PARELAG_TEST_FOR_EXCEPTION(NumBlockRows != NumBlockCols, std::runtime_error, "buildBlockedHierarchyFromDeRhamSequence(...): A is not block-square!");
    PARELAG_TEST_FOR_EXCEPTION((int)forms.size() != NumBlockRows, std::runtime_error,
                               "buildBlockedHierarchyFromDeRhamSequence(...): The forms vector has the wrong size (" << forms.size()
                               << "). Should be " << NumBlockRows << ".");
    PARELAG_TEST_FOR_EXCEPTION(forms.size() != label_ess.size(), std::runtime_error,
                               "buildBlockedHierarchyFromDeRhamSequence(...): Forms vector and boundary condition information are inconsistent.");
    int NumLevels = MaxNumLevels;
    {
        int actual = 0;
        std::shared_ptr<DeRhamSequence> tmp;
        const DeRhamSequence *p = &Sequence;
        while (p) { tmp = p->ViewCoarserSequence(); p = tmp.get(); ++actual; }
        if (MaxNumLevels < 1 || MaxNumLevels > actual) NumLevels = actual;
    }
    auto H = make_unique<Hierarchy>(A, NumLevels);
    H->SetImplicitTranspose(true);
    const DeRhamSequence *seq = &Sequence;
    std::shared_ptr<DeRhamSequence> hold;
    for (int l = 1; l < NumLevels; ++l)
    {
        Level &Coarse = H->GetLevel(l);
        auto cseq = seq->CoarserSequence();
        std::vector<int> CoarseOffSets(NumBlockRows + 1, 0);
        for (int ii = 0; ii < NumBlockRows; ++ii) CoarseOffSets[ii + 1] = CoarseOffSets[ii] + cseq->GetNumberOfTrueDofs(forms[ii]);
        auto Ac = std::make_shared<MfemBlockOperator>(CoarseOffSets);
        auto P = std::make_shared<MfemBlockOperator>(A_blocked->CopyRowOffsets(), Ac->CopyRowOffsets());
        std::vector<std::shared_ptr<mfem::HypreParMatrix>> P_blocks(NumBlockRows);
        for (int ii = 0; ii < NumBlockRows; ++ii)
        {
            if (label_ess[ii].size() > 0)
            {
                mfem::Array<int> tmp(label_ess[ii].data(), (int)label_ess[ii].size());
                P_blocks[ii] = seq->ComputeTrueP(forms[ii], tmp);
            }
            else P_blocks[ii] = seq->ComputeTrueP(forms[ii]);
        }
        for (int row = 0; row < NumBlockRows; ++row)
            for (int col = 0; col < NumBlockCols; ++col)
                if (!A_blocked->IsZeroBlock(row, col))
                {
                    auto &Aij = dynamic_cast<mfem::HypreParMatrix &>(A_blocked->GetBlock(row, col));
                    auto tmp = std::shared_ptr<mfem::HypreParMatrix>{mfem::RAP(P_blocks[row].get(), &Aij, P_blocks[col].get())};
                    if (row == col && label_ess[row].size() > 0)
                    {
                        H->SetZeroRows(l, ZeroRows(*tmp), row);
                        hypre_ParCSRMatrixFixZeroRows(*tmp);
                    }
                    Ac->SetBlock(row, col, std::move(tmp));
                }
        for (int row = 0; row < NumBlockRows; ++row) P->SetBlock(row, row, P_blocks[row]);
        A = Ac;
        A_blocked = Ac;
        Coarse.Set<Op_Ptr>("P", P);
        Coarse.Set<Op_Ptr>("A", Ac);
        hold = cseq;
        seq = hold.get();
    }
    H->Finalize();
    return H;
}

class AMGeSolverFactory : public SolverFactory
{
    std::unique_ptr<mfem::Solver> _do_build_solver(const Op_Ptr &op, SolverState &state) const override
    {
        auto my_state = dynamic_cast<NestedSolverState *>(&state);
        PARELAG_ASSERT(my_state);
        auto sequence = state.GetDeRhamSequencePtr();
        PARELAG_TEST_FOR_EXCEPTION(!sequence, std::runtime_error, "AMGeSolverFactory: the state has no DeRhamSequence");
        if (Forms_.size() == 0) Forms_ = state.GetForms();
        PARELAG_ASSERT(Forms_.size() > 0);
        std::unique_ptr<Hierarchy> H;
        {
            Timer t = TimeManager::AddTimer("Build Hierarchy: build from deRham Sequence");
            if (Forms_.size() == 1)
            {
                auto &ess_attr = state.GetBoundaryLabels(0);
                H = buildHierarchyFromDeRhamSequence(op, *sequence, ess_attr, Forms_.front(), MaxLevels_);
            }
            else H = buildBlockedHierarchyFromDeRhamSequence(op, *sequence, state.GetBoundaryLabels(), Forms_, MaxLevels_);
        }
        const int CoarsestLevelID = H->GetNumLevels() - 1;
        for (const auto &level : *H)
        {
            Level &lev = *level;
            const int LevelID = lev.GetLevelID();
            Timer fill = TimeManager::AddTimer("Build Hierarchy: fill level " + std::to_string(LevelID));
            auto A_ptr = lev.Get<Op_Ptr>("A");
            if (print_levels_)
                if (auto A_hyp = std::dynamic_pointer_cast<mfem::HypreParMatrix>(A_ptr))
                    std::cout << "Level " << LevelID << ": A = " << A_hyp->M() << "x" << A_hyp->N() << ", nnz = " << A_hyp->NNZ() << "\n";
            if (LevelID < CoarsestLevelID)
            {
                auto pre_state = std::shared_ptr<SolverState>{PreSmootherFact_->GetDefaultState()};
                auto post_state = std::shared_ptr<SolverState>{PostSmootherFact_->GetDefaultState()};
                if (my_state->IsSubState("PreSmoother")) pre_state->MergeState(*my_state->GetSubState("PreSmoother"));
                if (my_state->IsSubState("PostSmoother")) post_state->MergeState(*my_state->GetSubState("PostSmoother"));
                pre_state->MergeState(state); post_state->MergeState(state);
                pre_state->SetDeRhamSequence(sequence); post_state->SetDeRhamSequence(sequence);
                Timer st = TimeManager::AddTimer("Build smoother: level " + std::to_string(LevelID));
                std::shared_ptr<mfem::Solver> pre = PreSmootherFact_->BuildSolver(A_ptr, *pre_state);
                // the reference builds the post-smoother separately even when the factories
                // coincide; the operator is identical, so it is shared here
                std::shared_ptr<mfem::Solver> post = (PreSmootherFact_ == PostSmootherFact_) ? pre
                                                     : std::shared_ptr<mfem::Solver>(PostSmootherFact_->BuildSolver(A_ptr, *post_state));
                st.Stop();
                pre->iterative_mode = true; post->iterative_mode = true;
                lev.Set<Op_Ptr>("PreSmoother", pre);
                lev.Set<Op_Ptr>("PostSmoother", post);
            }
            else
            {
                auto coarse_state = std::shared_ptr<SolverState>{CoarseSolverFact_->GetDefaultState()};
                if (my_state->IsSubState("Coarse solver")) coarse_state->MergeState(*my_state->GetSubState("Coarse solver"));
                coarse_state->MergeState(state);
                coarse_state->SetDeRhamSequence(sequence);
                Timer ct = TimeManager::AddTimer("Build coarse solver: level " + std::to_string(LevelID));
                lev.Set<Op_Ptr>("CoarseSolver", Op_Ptr(CoarseSolverFact_->BuildSolver(A_ptr, *coarse_state)));
            }
            sequence = sequence->CoarserSequence();
        }
        H->SetUseGraph(use_graph_);
        H->SetUseProgram(use_program_);
        return H;
    }
    void _do_set_default_parameters() override {}
    void _do_initialize(const ParameterList &) override
    {
        auto &params = GetParameters();
        if (params.IsParameter("Smoother"))
        {
            PreSmootherFact_ = GetSolverLibrary().GetSolverFactory(params.Get<std::string>("Smoother"));
            PostSmootherFact_ = PreSmootherFact_;
        }
        else
        {
            if (params.IsParameter("PreSmoother")) PreSmootherFact_ = GetSolverLibrary().GetSolverFactory(params.Get<std::string>("PreSmoother"));
            if (params.IsParameter("PostSmoother")) PostSmootherFact_ = GetSolverLibrary().GetSolverFactory(params.Get<std::string>("PostSmoother"));
        }
        if (params.IsParameter("Coarse solver")) CoarseSolverFact_ = GetSolverLibrary().GetSolverFactory(params.Get<std::string>("Coarse solver"));
        MaxLevels_ = params.Get("Maximum levels", -1);
        Forms_ = params.Get("Forms", std::vector<int>());
        print_levels_ = params.Get("Print level summary", false);
        use_graph_ = params.Get("Use CUDA graph", true);   // extension: replay the V-cycle as one graph
        use_program_ = params.Get("Use persistent program", false);  // extension: the V-cycle as one persistent kernel (experimental, see DESIGN.md)
    }
    std::shared_ptr<SolverFactory> PreSmootherFact_, PostSmootherFact_, CoarseSolverFact_;
    int MaxLevels_ = -1;
    mutable std::vector<int> Forms_;
    bool print_levels_ = false, use_graph_ = true, use_program_ = false;
};

// ------------------------------------------------------------------ Stationary iteration
/// ParELAG_StationarySolver.cpp:41-147: Richardson iteration x += S r with any Solver S as corrector.  The residual is
/// UPDATED (r -= A c), not recomputed; at least one correction is applied; stops when ||r_k|| < atol, when the
/// accumulated ratio ||r_k|| / ||r_0|| < rtol, on a zero correction (||r_k|| / ||r_{k-1}|| == 1), or after MaxIts.
class StationarySolver : public Solver
{
public:
    StationarySolver(Op_Ptr A, std::shared_ptr<mfem::Solver> S, double rtol, double atol, size_t maxit, bool print)
        : Solver(A->Height(), A->Width(), true), A_(std::move(A)), Solver_(std::move(S)), RelTol_(rtol), AbsTol_(atol), MaxIts_(maxit), Print_(print) {}
    void Mult(const mfem::Vector &rhs, mfem::Vector &sol) const override
    {
        Solver_->iterative_mode = false;
        Resid_.SetSize(A_->Height()); Corr_.SetSize(A_->Width()); Tmp_.SetSize(A_->Height());
        if (this->IsPreconditioner()) { Resid_ = rhs; sol = 0.0; }
        else { A_->Mult(sol, Resid_); Resid_ *= -1.0; Resid_ += rhs; }
        double norm_k_1 = std::sqrt(Resid_ * Resid_), norm_k = norm_k_1, norm_ratio = 1.0;      // Vector dot = global sum
        History_.assign(1, norm_k_1);
        if (Print_) std::cout << "    Iteration 0: ||r|| = " << norm_k_1 << std::endl;
        size_t its = 0;
        Converged_ = false;
        while (its < MaxIts_)
        {
            ++its;
            Corr_ = 0.0; Tmp_ = 0.0;
            Solver_->Mult(Resid_, Corr_);
            sol += Corr_;
            A_->Mult(Corr_, Tmp_);
            Resid_ -= Tmp_;
            norm_k = std::sqrt(Resid_ * Resid_);
            History_.push_back(norm_k);
            norm_ratio *= norm_k / norm_k_1;
            if (Print_) std::cout << "    Iteration " << its << ": ||r|| = " << norm_k << "  (" << norm_ratio << ")" << std::endl;
            if (norm_k < AbsTol_ || norm_ratio < RelTol_) { Converged_ = true; break; }
            if (norm_k / norm_k_1 == 1.0) { std::cout << "WARNING: Computed a zero correction! Stopping..." << std::endl; break; }
            norm_k_1 = norm_k;
        }
        NumIts_ = (int)its; FinalNorm_ = norm_k;
        if (Print_)
            std::cout << '\n' << std::string(50, '*') << '\n' << "*  Solver Status: " << (Converged_ ? "Converged" : "Not converged") << '\n'
                      << "*  Solver Iterations: " << its << '\n' << "*  Final norm: " << norm_k << '\n' << std::string(50, '*') << std::endl;
    }
    void MultTranspose(const mfem::Vector &, mfem::Vector &) const override { PARELAG_NOT_IMPLEMENTED(); }
    int GetNumIterations() const { return NumIts_; }
    double GetFinalNorm() const { return FinalNorm_; }
    bool GetConverged() const { return Converged_; }
    /// ||r_k||, k = 0, 1, ... (what "Print Iterations" prints)
    const std::vector<double> &GetResidualHistory() const { return History_; }
    const std::shared_ptr<mfem::Solver> &GetSolver() const { return Solver_; }
private:
    void _do_set_operator(const Op_Ptr &op) override { A_ = op; }
    Op_Ptr A_;
    std::shared_ptr<mfem::Solver> Solver_;
    double RelTol_, AbsTol_;
    size_t MaxIts_;
    bool Print_;
    mutable mfem::Vector Resid_, Corr_, Tmp_;
    mutable std::vector<double> History_;
    mutable int NumIts_ = 0;
    mutable double FinalNorm_ = 0.0;
    mutable bool Converged_ = false;
};

inline void SetNestedOperator(mfem::Operator &S, const Op_Ptr &op)
{
    if (auto k = dynamic_cast<KrylovSolver *>(&S)) { if (k->GetPreconditioner()) SetNestedOperator(*k->GetPreconditioner(), op); }
    else if (auto st = dynamic_cast<StationarySolver *>(&S))
    {
        PARELAG_ASSERT(st->GetSolver());
        SetNestedOperator(*st->GetSolver(), op);
    }
    auto p = dynamic_cast<Solver *>(&S);
    PARELAG_TEST_FOR_EXCEPTION(!p, std::runtime_error, "SetOperator(): the solver is not a parelag::Solver");
    p->SetOperator(op);
}

/// ParELAG_StationarySolverFactory.hpp:27-107 (parameters "Solver", "Maximum Iterations" (size_t, default 1),
/// "Absolute Tolerance", "Relative Tolerance", "Print Iterations")
class StationarySolverFactory : public SolverFactory
{
    std::unique_ptr<mfem::Solver> _do_build_solver(const Op_Ptr &op, SolverState &state) const override
    {
        PARELAG_ASSERT(Fact_);
        auto my_state = dynamic_cast<NestedSolverState *>(&state);
        PARELAG_ASSERT(my_state);
        auto s_state = std::shared_ptr<SolverState>{Fact_->GetDefaultState()};
        if (my_state->IsSubState("Solver")) s_state->MergeState(*my_state->GetSubState("Solver"));
        s_state->MergeState(*my_state);
        std::shared_ptr<mfem::Solver> s = Fact_->BuildSolver(op, *s_state);
        s->iterative_mode = false;
        auto &p = GetParameters();
        return make_unique<StationarySolver>(op, s, p.Get<double>("Relative Tolerance"), p.Get<double>("Absolute Tolerance"),
                                             MaxIterations(p), p.Get<bool>("Print Iterations"));
    }
    /// "Maximum Iterations" is a size_t in the reference; an XML file may also carry it as "int"
    static size_t MaxIterations(ParameterList &p)
    {
        try { return p.Get<size_t>("Maximum Iterations"); }
        catch (const std::exception &) { return (size_t)std::max(p.Get<int>("Maximum Iterations"), 0); }
    }
    void _do_set_default_parameters() override
    {
        auto &p = GetParameters();
        if (!p.IsParameter("Maximum Iterations")) p.Set("Maximum Iterations", (size_t)1);
        p.Get("Absolute Tolerance", 0.0);
        p.Get("Relative Tolerance", 0.0);
        p.Get("Print Iterations", false);
    }
    void _do_initialize(const ParameterList &) override
    {
        PARELAG_ASSERT(HasValidSolverLibrary());
        Fact_ = GetSolverLibrary().GetSolverFactory(GetParameters().Get("Solver", "INVALID"));
    }
    std::shared_ptr<SolverFactory> Fact_;
};

inline void SolverLibrary::RegisterBuiltins()
{
    RegisterFactoryType("AMGe", [] { return std::make_shared<AMGeSolverFactory>(); });
    RegisterFactoryType("Hypre", [] { return std::make_shared<HypreSmootherFactory>(); });
    RegisterFactoryType("Hiptmair", [] { return std::make_shared<HiptmairSmootherFactory>(); });
    RegisterFactoryType("Krylov", [] { return std::make_shared<KrylovSolverFactory>(); });
    RegisterFactoryType("Stationary Iteration", [] { return std::make_shared<StationarySolverFactory>(); });
    RegisterFactoryType("Block GS", [] { return std::make_shared<Block2x2GaussSeidelSolverFactory>(); });
    RegisterFactoryType("Block Jacobi", [] { return std::make_shared<Block2x2JacobiSolverFactory>(); });
    RegisterFactoryType("Block LDU", [] { return std::make_shared<Block2x2LDUSolverFactory>(); });
}
} // namespace parelag
