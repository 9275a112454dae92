// parelag_block.hpp -- block operators and block preconditioners of the mixed (Darcy) path,
// with the reference's class and parameter names; all arithmetic on the GPU through the C ABI.
//   MfemBlockOperator            src/linalg/utilities/ParELAG_MfemBlockOperator.cpp:23-165
//   BlockDiagonalSolver          src/linalg/solver_ops/ParELAG_BlockDiagonalSolver.cpp:66-110
//   BlockTriangularSolver        src/linalg/solver_ops/ParELAG_BlockTriangularSolver.cpp:74-300
//   Block2x2LDUInverseOperator   src/linalg/solver_ops/ParELAG_Block2x2LDUInverseOperator.cpp:73-135
//   SchurComplementFactory       src/linalg/factories/ParELAG_SchurComplementFactory.cpp:36-177
//   Block2x2{Jacobi,GaussSeidel,LDU}SolverFactory   src/linalg/factories/ParELAG_Block2x2*SolverFactory.cpp
#pragma once
#include <algorithm>
#include <tuple>
#include "parelag_core.hpp"
#include "parelag_sequence.hpp"

namespace parelag
{
using Op_Ptr = std::shared_ptr<mfem::Operator>;

/// mfem::BlockVector over an existing vector: non-owning views of its blocks
class BlockVectorView
{
public:
    BlockVectorView(const mfem::Vector &v, const std::vector<int> &offsets)
    {
        for (size_t i = 0; i + 1 < offsets.size(); ++i)
        {
            blk_.push_back(make_unique<mfem::Vector>());
            blk_.back()->MakeRef(v, offsets[i], offsets[i + 1] - offsets[i]);
        }
    }
    mfem::Vector &GetBlock(int i) { return *blk_.at(i); }
    const mfem::Vector &GetBlock(int i) const { return *blk_.at(i); }
private:
    std::vector<std::unique_ptr<mfem::Vector>> blk_;
};

class MfemBlockOperator : public mfem::Operator
{
public:
    using offset_type = int;
    using size_type = size_t;
    explicit MfemBlockOperator(std::vector<offset_type> block_offsets)
        : mfem::Operator(block_offsets.back()), RowOffsets_(block_offsets), ColOffsets_(std::move(block_offsets)) { Init(); }
    MfemBlockOperator(std::vector<offset_type> row_offsets, std::vector<offset_type> col_offsets)
        : mfem::Operator(row_offsets.back(), col_offsets.back()), RowOffsets_(std::move(row_offsets)), ColOffsets_(std::move(col_offsets)) { Init(); }

    void Mult(const mfem::Vector &x, mfem::Vector &y) const override
    {
        BlockVectorView xv(x, ColOffsets_), yv(y, RowOffsets_);
        for (size_type i = 0; i < GetNumBlockRows(); ++i)
        {
            bool first = true;
            for (size_type j = 0; j < GetNumBlockCols(); ++j)
            {
                if (IsZeroBlock(i, j)) continue;
                Accumulate(*Blocks_[i * GetNumBlockCols() + j], false, xv.GetBlock((int)j), yv.GetBlock((int)i), first);
                first = false;
            }
            if (first) yv.GetBlock((int)i) = 0.0;
        }
    }
    void MultTranspose(const mfem::Vector &x, mfem::Vector &y) const override
    {
        BlockVectorView xv(x, RowOffsets_), yv(y, ColOffsets_);
        for (size_type j = 0; j < GetNumBlockCols(); ++j)
        {
            bool first = true;
            for (size_type i = 0; i < GetNumBlockRows(); ++i)
            {
                if (IsZeroBlock(i, j)) continue;
                Accumulate(*Blocks_[i * GetNumBlockCols() + j], true, xv.GetBlock((int)i), yv.GetBlock((int)j), first);
                first = false;
            }
            if (first) yv.GetBlock((int)j) = 0.0;
        }
    }
    void SetBlock(size_type block_row, size_type block_col, std::shared_ptr<mfem::Operator> op)
    {
        PARELAG_TEST_FOR_EXCEPTION(block_row >= GetNumBlockRows() || block_col >= GetNumBlockCols(), std::runtime_error,
                                   "MfemBlockOperator::SetBlock(...):\nInvalid block (" << block_row << "," << block_col << ")");
        PARELAG_TEST_FOR_EXCEPTION(op && (op->Height() != RowOffsets_[block_row + 1] - RowOffsets_[block_row] ||
                                          op->Width() != ColOffsets_[block_col + 1] - ColOffsets_[block_col]), std::runtime_error,
                                   "MfemBlockOperator::SetBlock(...):\nBlock (" << block_row << "," << block_col << ") has the wrong size "
                                   << op->Height() << "x" << op->Width());
        Blocks_[block_row * GetNumBlockCols() + block_col] = std::move(op);
    }
    mfem::Operator &GetBlock(size_type i, size_type j)
    {
        PARELAG_TEST_FOR_EXCEPTION(IsZeroBlock(i, j), std::runtime_error, "MfemBlockOperator::GetBlock(): block (" << i << "," << j << ") is zero");
        return *Blocks_[i * GetNumBlockCols() + j];
    }
    const mfem::Operator &GetBlock(size_type i, size_type j) const { return const_cast<MfemBlockOperator *>(this)->GetBlock(i, j); }
    std::shared_ptr<mfem::Operator> GetBlockPtr(size_type i, size_type j) const { return Blocks_.at(i * GetNumBlockCols() + j); }
    bool IsZeroBlock(size_type i, size_type j) const { return !Blocks_.at(i * GetNumBlockCols() + j); }
    size_type GetNumBlockRows() const noexcept { return RowOffsets_.size() - 1; }
    size_type GetNumBlockCols() const noexcept { return ColOffsets_.size() - 1; }
    const std::vector<offset_type> &ViewRowOffsets() const noexcept { return RowOffsets_; }
    const std::vector<offset_type> &ViewColumnOffsets() const noexcept { return ColOffsets_; }
    std::vector<offset_type> CopyRowOffsets() const { return RowOffsets_; }
    /// CopyRowOffsetsAsMfemArray / CopyColumnOffsetsAsMfemArray (ParELAG_MfemBlockOperator.hpp:198-206)
    void CopyRowOffsetsAsMfemArray(mfem::Array<offset_type> &row_offsets) const
    { row_offsets.SetSize((int)RowOffsets_.size()); for (size_t i = 0; i < RowOffsets_.size(); ++i) row_offsets[(int)i] = RowOffsets_[i]; }
    void CopyColumnOffsetsAsMfemArray(mfem::Array<offset_type> &col_offsets) const
    { col_offsets.SetSize((int)ColOffsets_.size()); for (size_t i = 0; i < ColOffsets_.size(); ++i) col_offsets[(int)i] = ColOffsets_[i]; }
    std::vector<offset_type> CopyColumnOffsets() const { return ColOffsets_; }

private:
    void Init() { Blocks_.assign(GetNumBlockRows() * GetNumBlockCols(), nullptr); }
    /// y = op(x) (first) or y += op(x)
    void Accumulate(const mfem::Operator &op, bool transpose, const mfem::Vector &x, mfem::Vector &y, bool first) const
    {
        auto hyp = dynamic_cast<const mfem::HypreParMatrix *>(&op);
        if (hyp && !transpose) { hyp->Mult(1.0, x, first ? 0.0 : 1.0, y); return; }
        if (first) { if (transpose) op.MultTranspose(x, y); else op.Mult(x, y); return; }
        tmp_.SetSize(y.Size());
        if (transpose) op.MultTranspose(x, tmp_); else op.Mult(x, tmp_);
        y += tmp_;
    }
    std::vector<offset_type> RowOffsets_, ColOffsets_;
    std::vector<std::shared_ptr<mfem::Operator>> Blocks_;
    mutable mfem::Vector tmp_;
};

namespace mg_utils
{
/// r = b - A x for any operator (block operators included)
inline void ComputeResidualGeneric(const mfem::Operator &A, const mfem::Vector &x, const mfem::Vector &b, mfem::Vector &r)
{
    r.SetSize(b.Size());
    A.Mult(x, r);
    mfem::add(b, -1.0, r, r);
}
} // namespace mg_utils

/// a copy of A (pattern and values), to take new values in place of A's
inline std::shared_ptr<mfem::HypreParMatrix> CopyOf(const mfem::HypreParMatrix &A)
{
    pe_mat *m = nullptr;
    PE_CALL(pe_mat_clone(Device::Get(), A.Handle(), &m));
    return std::make_shared<mfem::HypreParMatrix>(m);
}
/// the rows hypre_ParCSRMatrixFixZeroRows rewrites in A: 1.0 on those rows, 0.0 elsewhere
inline mfem::Vector ZeroRows(const mfem::HypreParMatrix &A)
{
    mfem::Vector mask((int)A.Height());
    PE_CALL(pe_mat_zero_rows(Device::Get(), A.Handle(), mask.Write(), nullptr));
    return mask;
}
/// SetOperator on a built solver: the new operator must have the held one's size and sparsity pattern
inline void CheckSamePattern(const mfem::HypreParMatrix &held, const mfem::HypreParMatrix &A, const char *who)
{
    int32_t same = 0;
    PE_CALL(pe_mat_same_pattern(Device::Get(), held.Handle(), A.Handle(), &same));
    PARELAG_TEST_FOR_EXCEPTION(!same, std::runtime_error,
                               who << "::SetOperator(): the new operator has a different size or sparsity pattern; "
                               "build a new solver for it");
}
/// the FixZeroRows step of an update: A (new values) must have the zero rows recorded at build time, then they are fixed
inline void FixSameZeroRows(mfem::HypreParMatrix &A, const mfem::Vector &recorded, const std::string &where)
{
    int32_t changed = 0;
    PE_CALL(pe_mat_zero_rows(Device::Get(), A.Handle(), const_cast<pe_vec *>(recorded.Read()), &changed));
    PARELAG_TEST_FOR_EXCEPTION(changed, std::runtime_error,
                               "SetOperator(): the set of zero rows FixZeroRows rewrites in " << where
                               << " differs from the built solver's; build a new solver for this operator");
    hypre_ParCSRMatrixFixZeroRows(A);
}

/// SetOperator on a solver and the solvers it holds: the preconditioner of a Krylov solver and the corrector of a
/// stationary iteration first (their own SetOperator only swaps the operator), as an mfem driver orders it
void SetNestedOperator(mfem::Operator &S, const Op_Ptr &op);

/// SetOperator on a block solver: op must be an MfemBlockOperator with the held one's block sizes, zero blocks and
/// the sparsity pattern of every block (one rank)
inline std::shared_ptr<MfemBlockOperator> SameBlockStructure(const MfemBlockOperator &held, const Op_Ptr &op, const char *who)
{
    PARELAG_TEST_FOR_EXCEPTION(pe_ctx_nranks(Device::Get()) != 1, std::runtime_error,
                               who << "::SetOperator(): more than one rank is not supported; build a new solver");
    auto A = std::dynamic_pointer_cast<MfemBlockOperator>(op);
    PARELAG_TEST_FOR_EXCEPTION(!A, std::runtime_error, who << "::SetOperator(...): Operator must be an MfemBlockOperator!");
    PARELAG_TEST_FOR_EXCEPTION(A->ViewRowOffsets() != held.ViewRowOffsets() || A->ViewColumnOffsets() != held.ViewColumnOffsets(),
                               std::runtime_error, who << "::SetOperator(): the new operator has different block sizes; build a new solver for it");
    for (size_t i = 0; i < held.GetNumBlockRows(); ++i)
        for (size_t j = 0; j < held.GetNumBlockCols(); ++j)
        {
            PARELAG_TEST_FOR_EXCEPTION(A->IsZeroBlock(i, j) != held.IsZeroBlock(i, j), std::runtime_error,
                                       who << "::SetOperator(): block (" << i << "," << j << ") is " << (held.IsZeroBlock(i, j) ? "" : "not ")
                                       << "zero in the built solver's operator and " << (A->IsZeroBlock(i, j) ? "" : "not ")
                                       << "zero in the new one; build a new solver for it");
            if (held.IsZeroBlock(i, j)) continue;
            auto h = dynamic_cast<const mfem::HypreParMatrix *>(&held.GetBlock(i, j));
            auto a = dynamic_cast<const mfem::HypreParMatrix *>(&A->GetBlock(i, j));
            PARELAG_TEST_FOR_EXCEPTION(!h || !a, std::runtime_error, who << "::SetOperator(): the blocks must be HypreParMatrix");
            CheckSamePattern(*h, *a, who);
        }
    return A;
}

/// one inverse of a block preconditioner, the operator it takes and the one it holds
struct InverseUpdate
{
    mfem::Solver *inv;
    Op_Ptr next, held;
};
/// every inverse takes its new operator, each object once; when one refuses, those already updated take their held
/// operators back (SetOperator with the held operators restores a solver bit for bit) and the refusal is passed on
inline void SetInverseOperators(const std::vector<InverseUpdate> &u)
{
    auto first = [&](size_t i) { for (size_t k = 0; k < i; ++k) if (u[k].inv == u[i].inv) return false; return true; };
    size_t i = 0;
    try
    {
        for (; i < u.size(); ++i)
            if (u[i].next != u[i].held && first(i)) SetNestedOperator(*u[i].inv, u[i].next);
    }
    catch (...)
    {
        for (size_t k = 0; k < i; ++k)
            if (u[k].next != u[k].held && first(k)) SetNestedOperator(*u[k].inv, u[k].held);
        throw;
    }
}

class SchurComplementFactory;
/// How a block preconditioner's second diagonal operator was made (BlockSolverFactory::SecondDiagonalOperator), so
/// that SetOperator can make it again for new blocks
struct SecondDiagonal
{
    std::shared_ptr<const SchurComplementFactory> fact;   // "S Type", "Alpha"; null: the (1,1) block itself
    bool negative = true;                                 // "Use Negative S"
    Op_Ptr S;                                             // the operator the A11 / S inverse was built on
    std::shared_ptr<mfem::HypreParMatrix> product;        // A10 D^-1 A01 when S = A11 - alpha A10 D^-1 A01
    /// the second diagonal operator of the new blocks A (same patterns as the held ones): S computed numerically
    /// into copies of the held patterns, the held S for "MASS", A's (1,1) block without a factory
    SecondDiagonal For(MfemBlockOperator &A) const;
};

inline bool BlockCaptureSafe(const std::vector<std::shared_ptr<mfem::Solver>> &ops)
{
    for (auto &s : ops)
    {
        auto p = dynamic_cast<const Solver *>(s.get());
        if (!p || !p->CaptureSafe()) return false;
    }
    return true;
}

/// SetOperator of BlockDiagonalSolver and BlockTriangularSolver: inverse b takes block (b, b) of op, inverse 1 the
/// second diagonal operator made again for op
inline void SetDiagonalInverses(std::shared_ptr<MfemBlockOperator> &A, SecondDiagonal &second,
                                const std::vector<std::shared_ptr<mfem::Solver>> &inv_ops, const Op_Ptr &op, const char *who)
{
    auto next = SameBlockStructure(*A, op, who);
    SecondDiagonal next_second = second.For(*next);
    std::vector<InverseUpdate> u;
    for (size_t b = 0; b < inv_ops.size(); ++b)
        u.push_back({inv_ops[b].get(), b == 1 ? next_second.S : next->GetBlockPtr(b, b), b == 1 ? second.S : A->GetBlockPtr(b, b)});
    Timer t = TimeManager::AddTimer("SetOperator: block inverses");
    SetInverseOperators(u);
    A = std::move(next);
    second = std::move(next_second);
}

// ------------------------------------------------------------------ block Jacobi
class BlockDiagonalSolver : public Solver
{
public:
    /// second: how the operator of inv_ops[1] was made (its S keeps the Schur complement alive)
    BlockDiagonalSolver(std::shared_ptr<MfemBlockOperator> op, std::vector<std::shared_ptr<mfem::Solver>> inv_ops, SecondDiagonal second)
        : Solver(op->Width(), op->Height(), false), A_(std::move(op)), inv_ops_(std::move(inv_ops)), second_(std::move(second)) {}
    void Mult(const mfem::Vector &rhs, mfem::Vector &sol) const override { Apply(rhs, sol, false); }
    void MultTranspose(const mfem::Vector &rhs, mfem::Vector &sol) const override { Apply(rhs, sol, true); }
    bool CaptureSafe() const override { return BlockCaptureSafe(inv_ops_); }
private:
    void Apply(const mfem::Vector &rhs, mfem::Vector &sol, bool transpose) const
    {
        const auto &off = A_->ViewRowOffsets();
        if (this->IsPreconditioner())
        {
            // Resid = rhs; sol = 0.0
            BlockVectorView r(rhs, off), s(sol, off);
            sol = 0.0;
            for (size_t b = 0; b < inv_ops_.size(); ++b) Inv(b, transpose, r.GetBlock((int)b), s.GetBlock((int)b));
            return;
        }
        // Resid = rhs - A*sol; correction added at the end
        resid_.SetSize(rhs.Size()); corr_.SetSize(sol.Size());
        if (transpose) A_->MultTranspose(sol, resid_); else A_->Mult(sol, resid_);
        resid_ *= -1.0;
        resid_ += rhs;
        corr_ = 0.0;
        BlockVectorView r(resid_, off), s(corr_, off);
        for (size_t b = 0; b < inv_ops_.size(); ++b) Inv(b, transpose, r.GetBlock((int)b), s.GetBlock((int)b));
        sol += corr_;
    }
    void Inv(size_t b, bool transpose, const mfem::Vector &r, mfem::Vector &x) const
    {
        PARELAG_ASSERT(!inv_ops_[b]->iterative_mode);
        if (transpose) inv_ops_[b]->MultTranspose(r, x); else inv_ops_[b]->Mult(r, x);
    }
    /// new block values on the held structure and patterns: the inverses take the new diagonal operators
    void _do_set_operator(const Op_Ptr &op) override { SetDiagonalInverses(A_, second_, inv_ops_, op, "BlockDiagonalSolver"); }
    std::shared_ptr<MfemBlockOperator> A_;
    std::vector<std::shared_ptr<mfem::Solver>> inv_ops_;
    SecondDiagonal second_;
    mutable mfem::Vector resid_, corr_;
};

// ------------------------------------------------------------------ block Gauss-Seidel
class BlockTriangularSolver : public Solver
{
public:
    enum class Triangle { UPPER_TRIANGLE, LOWER_TRIANGLE };
    BlockTriangularSolver(std::shared_ptr<MfemBlockOperator> op, std::vector<std::shared_ptr<mfem::Solver>> inv_ops,
                          SecondDiagonal second, Triangle tri = Triangle::LOWER_TRIANGLE)
        : Solver(op->Width(), op->Height(), false), A_(std::move(op)), inv_ops_(std::move(inv_ops)), second_(std::move(second)), tri_(tri) {}
    void Mult(const mfem::Vector &rhs, mfem::Vector &sol) const override { Apply(rhs, sol, false); }
    void MultTranspose(const mfem::Vector &rhs, mfem::Vector &sol) const override { Apply(rhs, sol, true); }
    bool CaptureSafe() const override { return BlockCaptureSafe(inv_ops_); }
private:
    void Apply(const mfem::Vector &rhs, mfem::Vector &sol, bool transpose) const
    {
        const auto &off = A_->ViewRowOffsets();
        const bool up = (tri_ == Triangle::UPPER_TRIANGLE) != transpose;     // traversal counts DOWN
        if (this->IsPreconditioner())
        {
            BlockVectorView r(rhs, off), s(sol, off);
            sol = 0.0;
            Sweep(r, s, up, transpose);
            return;
        }
        resid_.SetSize(rhs.Size()); corr_.SetSize(sol.Size());
        if (transpose) A_->MultTranspose(sol, resid_); else A_->Mult(sol, resid_);
        resid_ *= -1.0;
        resid_ += rhs;
        corr_ = 0.0;
        BlockVectorView r(resid_, off), s(corr_, off);
        Sweep(r, s, up, transpose);
        sol += corr_;
    }
    /// _do_{lower,upper}_mult[_transp] (BlockTriangularSolver.cpp:183-300)
    void Sweep(const BlockVectorView &rhs, BlockVectorView &sol, bool count_down, bool transpose) const
    {
        const int nb = (int)inv_ops_.size();
        for (int q = 0; q < nb; ++q)
        {
            const int i = count_down ? nb - 1 - q : q;
            const bool first = q == 0;
            if (!first) { tmp_rhs_ = rhs.GetBlock(i); tmp_.SetSize(tmp_rhs_.Size()); }
            for (int p = 0; p < q; ++p)
            {
                const int j = count_down ? nb - 1 - p : p;
                // forward sweeps use A(i,j); transposed sweeps A(j,i)^T
                if (transpose) { if (A_->IsZeroBlock(j, i)) continue; A_->GetBlock(j, i).MultTranspose(sol.GetBlock(j), tmp_); }
                else { if (A_->IsZeroBlock(i, j)) continue; A_->GetBlock(i, j).Mult(sol.GetBlock(j), tmp_); }
                tmp_rhs_ -= tmp_;
            }
            PARELAG_ASSERT(!inv_ops_[i]->iterative_mode);
            const mfem::Vector &r = first ? rhs.GetBlock(i) : tmp_rhs_;
            if (transpose) inv_ops_[i]->MultTranspose(r, sol.GetBlock(i)); else inv_ops_[i]->Mult(r, sol.GetBlock(i));
        }
    }
    void _do_set_operator(const Op_Ptr &op) override { SetDiagonalInverses(A_, second_, inv_ops_, op, "BlockTriangularSolver"); }
    std::shared_ptr<MfemBlockOperator> A_;
    std::vector<std::shared_ptr<mfem::Solver>> inv_ops_;
    SecondDiagonal second_;
    Triangle tri_;
    mutable mfem::Vector resid_, corr_, tmp_rhs_, tmp_;
};

// ------------------------------------------------------------------ block LDU
class Block2x2LDUInverseOperator : public Solver
{
public:
    Block2x2LDUInverseOperator(std::shared_ptr<MfemBlockOperator> A, std::shared_ptr<mfem::Solver> invA00_1, std::shared_ptr<mfem::Solver> invA00_2,
                               std::shared_ptr<mfem::Solver> invA00_3, std::shared_ptr<mfem::Solver> invS, SecondDiagonal S, double DampingFactor)
        : Solver(A->Width(), A->Height(), false), A_(std::move(A)), invA00_1_(std::move(invA00_1)), invA00_2_(std::move(invA00_2)),
          invA00_3_(std::move(invA00_3)), invS_(std::move(invS)), S_(std::move(S)), DampingFactor_(DampingFactor) {}
    void Mult(const mfem::Vector &rhs, mfem::Vector &sol) const override
    {
        const auto &off = A_->ViewRowOffsets();
        Residual_.SetSize(rhs.Size()); Tmp_.SetSize(rhs.Size()); Correction_.SetSize(rhs.Size());
        if (this->IsPreconditioner()) Residual_ = rhs;
        else mg_utils::ComputeResidualGeneric(*A_, sol, rhs, Residual_);
        BlockVectorView R(Residual_, off), T(Tmp_, off), C(Correction_, off);
        // dp = S^{-1}(r_g - A10 A_2^{-1} r_f)
        if (invA00_1_->iterative_mode) T.GetBlock(0) = 0.0;
        invA00_2_->Mult(R.GetBlock(0), T.GetBlock(0));
        A_->GetBlock(1, 0).Mult(T.GetBlock(0), T.GetBlock(1));
        R.GetBlock(1) -= T.GetBlock(1);
        if (invS_->iterative_mode) C.GetBlock(1) = 0.0;
        invS_->Mult(R.GetBlock(1), C.GetBlock(1));
        // du = A_1^{-1} r_f - A_3^{-1} A01 dp
        A_->GetBlock(0, 1).Mult(C.GetBlock(1), C.GetBlock(0));
        if (invA00_3_->iterative_mode) T.GetBlock(0) = 0.0;
        invA00_3_->Mult(C.GetBlock(0), T.GetBlock(0));
        if (invA00_1_->iterative_mode) C.GetBlock(0) = 0.0;
        invA00_1_->Mult(R.GetBlock(0), C.GetBlock(0));
        C.GetBlock(0) -= T.GetBlock(0);
        if (DampingFactor_ != 1.0) Correction_ *= DampingFactor_;
        if (this->IsPreconditioner()) sol = Correction_;
        else sol += Correction_;
    }
    void MultTranspose(const mfem::Vector &, mfem::Vector &) const override { PARELAG_NOT_IMPLEMENTED(); }
private:
    /// new block values on the held structure and patterns: the three A00 inverses take the new (0,0) block, the S
    /// inverse the second diagonal operator made again for op
    void _do_set_operator(const Op_Ptr &op) override
    {
        auto A = SameBlockStructure(*A_, op, "Block2x2LDUInverseOperator");
        SecondDiagonal S = S_.For(*A);
        const Op_Ptr A00 = A->GetBlockPtr(0, 0), held00 = A_->GetBlockPtr(0, 0);
        Timer t = TimeManager::AddTimer("SetOperator: block inverses");
        SetInverseOperators({{invA00_1_.get(), A00, held00}, {invA00_2_.get(), A00, held00}, {invA00_3_.get(), A00, held00},
                             {invS_.get(), S.S, S_.S}});
        A_ = std::move(A);
        S_ = std::move(S);
    }
    std::shared_ptr<MfemBlockOperator> A_;
    std::shared_ptr<mfem::Solver> invA00_1_, invA00_2_, invA00_3_, invS_;
    SecondDiagonal S_;
    double DampingFactor_;
    mutable mfem::Vector Residual_, Tmp_, Correction_;
};

// ------------------------------------------------------------------ Schur complement
class SchurComplementFactory
{
public:
    explicit SchurComplementFactory(std::string type = "MASS", double scaling = 1.0) : Type_(std::move(type)), Alpha_(scaling)
    {
        std::transform(Type_.begin(), Type_.end(), Type_.begin(), ::toupper);
    }
    /// "MASS": sequence.ComputeTrueM(forms.front()); "DIAGONAL": A11 - alpha A10 diag(A00)^{-1} A01; "ABSROWSUM": the
    /// same with absolute row sums (ParELAG_SchurComplementFactory.cpp:36-177)
    /// product (may be null): receives A10 diag^{-1} A01 when A11 is non-zero (the pattern SecondDiagonal::For refills)
    std::unique_ptr<mfem::Operator> BuildOperator(MfemBlockOperator &op, SolverState &state,
                                                  std::shared_ptr<mfem::HypreParMatrix> *product_out = nullptr) const
    {
        PARELAG_ASSERT(op.GetNumBlockRows() == 2);
        PARELAG_ASSERT(op.GetNumBlockCols() == 2);
        if (Type_ == "MASS")
        {
            // "Assume the state has just the important form up front" (SchurComplementFactory.cpp:43-50)
            auto form = state.GetForms().front();
            auto &sequence = state.GetDeRhamSequence();
            return sequence.ComputeTrueM(form);
        }
        PARELAG_TEST_FOR_EXCEPTION(Type_ != "DIAGONAL" && Type_ != "ABSROWSUM", std::runtime_error,
                                   "Schur complement type = \"" << Type_ << "\" is invalid.\nValid types are \"MASS\" and \"DIAGONAL\"");
        auto blk = [&](int i, int j) { return op.IsZeroBlock(i, j) ? nullptr : dynamic_cast<mfem::HypreParMatrix *>(&op.GetBlock(i, j)); };
        auto A00 = blk(0, 0), A01 = blk(0, 1), A10 = blk(1, 0), A11 = blk(1, 1);
        PARELAG_ASSERT(A00 && A01 && A10);
        pe_ctx *ctx = Device::Get();
        mfem::Vector diag(A00->Height());
        if (Type_ == "DIAGONAL") PE_CALL(pe_mat_get_diag(A00->Handle(), diag.Write()));
        else PE_CALL(pe_mat_abs_row_sums(A00->Handle(), diag.Write()));
        // tmp = diag^{-1} A01; product = A10 tmp
        pe_mat *tmp = nullptr, *product = nullptr, *out = nullptr;
        PE_CALL(pe_spadd(ctx, 1.0, A01->Handle(), 0.0, A01->Handle(), &tmp));
        PE_CALL(pe_mat_scale_rows(tmp, diag.Read(), 1));
        const int rc = pe_spgemm(ctx, A10->Handle(), tmp, &product);
        pe_mat_free(tmp);
        PE_CALL(rc);
        if (A11)
        {
            const int rc2 = pe_spadd(ctx, 1.0, A11->Handle(), -1.0 * Alpha_, product, &out);
            if (product_out) *product_out = std::make_shared<mfem::HypreParMatrix>(product);
            else pe_mat_free(product);
            PE_CALL(rc2);
            return make_unique<mfem::HypreParMatrix>(out);
        }
        PE_CALL(pe_mat_scale(product, -1.0 * Alpha_));
        return make_unique<mfem::HypreParMatrix>(product);
    }
    /// BuildOperator for new blocks of op's patterns, numerically into copies of S (BuildOperator's result, as held,
    /// negated or not) and of product: the same values, bit for bit.  "MASS" does not depend on the blocks: S is kept.
    std::pair<Op_Ptr, std::shared_ptr<mfem::HypreParMatrix>> UpdateOperator(MfemBlockOperator &op, const Op_Ptr &S,
                                                                            const std::shared_ptr<mfem::HypreParMatrix> &product) const
    {
        if (Type_ == "MASS") return {S, product};
        auto blk = [&](int i, int j) { return op.IsZeroBlock(i, j) ? nullptr : dynamic_cast<mfem::HypreParMatrix *>(&op.GetBlock(i, j)); };
        auto A00 = blk(0, 0), A01 = blk(0, 1), A10 = blk(1, 0), A11 = blk(1, 1);
        PARELAG_ASSERT(A00 && A01 && A10 && (!A11 || product));
        pe_ctx *ctx = Device::Get();
        mfem::Vector diag(A00->Height());
        if (Type_ == "DIAGONAL") PE_CALL(pe_mat_get_diag(A00->Handle(), diag.Write()));
        else PE_CALL(pe_mat_abs_row_sums(A00->Handle(), diag.Write()));
        auto out = CopyOf(dynamic_cast<const mfem::HypreParMatrix &>(*S));
        if (!A11)
        {
            PE_CALL(pe_spgemm_numeric_scaled(ctx, A10->Handle(), diag.Read(), A01->Handle(), out->Handle()));
            PE_CALL(pe_mat_scale(out->Handle(), -1.0 * Alpha_));
            return {out, nullptr};
        }
        auto prod = CopyOf(*product);
        PE_CALL(pe_spgemm_numeric_scaled(ctx, A10->Handle(), diag.Read(), A01->Handle(), prod->Handle()));
        PE_CALL(pe_spadd_numeric(ctx, 1.0, A11->Handle(), -1.0 * Alpha_, prod->Handle(), out->Handle()));
        return {out, prod};
    }
private:
    std::string Type_;
    double Alpha_;
};

inline SecondDiagonal SecondDiagonal::For(MfemBlockOperator &A) const
{
    SecondDiagonal out = *this;
    if (!fact) { out.S = A.GetBlockPtr(1, 1); return out; }
    Timer t = TimeManager::AddTimer("SetOperator: Schur complements");
    std::tie(out.S, out.product) = fact->UpdateOperator(A, S, product);
    if (negative && out.S != S) PE_CALL(pe_mat_scale(dynamic_cast<mfem::HypreParMatrix &>(*out.S).Handle(), -1.0));
    return out;
}

// ------------------------------------------------------------------ factories
/// BlockSolverFactory: the operator must be an MfemBlockOperator
class BlockSolverFactory : public SolverFactory
{
protected:
    std::unique_ptr<mfem::Solver> _do_build_solver(const Op_Ptr &op, SolverState &state) const override
    {
        auto blop = std::dynamic_pointer_cast<MfemBlockOperator>(op);
        PARELAG_TEST_FOR_EXCEPTION(!blop, std::runtime_error, "BlockSolverFactory::BuildSolver(): the operator is not an MfemBlockOperator");
        return _do_build_block_solver(blop, state);
    }
    virtual std::unique_ptr<mfem::Solver> _do_build_block_solver(const std::shared_ptr<MfemBlockOperator> &blop, SolverState &state) const = 0;
    /// S (negated when "Use Negative S") or A11, with how it was made
    SecondDiagonal SecondDiagonalOperator(MfemBlockOperator &blop, SolverState &state) const
    {
        SecondDiagonal out;
        if (!S_Fact_) { out.S = blop.GetBlockPtr(1, 1); return out; }
        out.fact = S_Fact_;
        out.negative = UseNegativeS_;
        out.S = Op_Ptr(S_Fact_->BuildOperator(blop, state, &out.product));
        if (UseNegativeS_)
            if (auto s_mat = dynamic_cast<mfem::HypreParMatrix *>(out.S.get())) PE_CALL(pe_mat_scale(s_mat->Handle(), -1.0));
        return out;
    }
    void InitSchur()
    {
        auto &params = GetParameters();
        UseNegativeS_ = params.Get<bool>("Use Negative S", true);
        const std::string S_name = params.Get("S Type", "NONE");
        const double alpha = params.Get("Alpha", 1.0);
        std::string up = S_name;
        std::transform(up.begin(), up.end(), up.begin(), ::toupper);
        S_Fact_ = up != "NONE" ? std::make_shared<SchurComplementFactory>(S_name, alpha) : nullptr;
    }
    static std::shared_ptr<SolverState> SubState(const SolverFactory &f, NestedSolverState &mine, const char *name, int form)
    {
        auto s = std::shared_ptr<SolverState>{f.GetDefaultState()};
        if (mine.IsSubState(name)) s->MergeState(*mine.GetSubState(name));
        s->MergeState(mine);
        s->SetForms({form});
        return s;
    }
    std::shared_ptr<SchurComplementFactory> S_Fact_;
    bool UseNegativeS_ = true;
};

class Block2x2JacobiSolverFactory : public BlockSolverFactory
{
    std::unique_ptr<mfem::Solver> _do_build_block_solver(const std::shared_ptr<MfemBlockOperator> &blop, SolverState &state) const override
    {
        PARELAG_ASSERT(blop->GetNumBlockRows() == 2 && blop->GetNumBlockCols() == 2);
        auto my_state = dynamic_cast<NestedSolverState *>(&state);
        PARELAG_ASSERT(my_state);
        const std::vector<int> forms = my_state->GetForms();
        PARELAG_TEST_FOR_EXCEPTION(forms.size() < 2, std::runtime_error, "Block Jacobi: the state must carry two forms");
        auto A00_state = SubState(*InvA00_Fact_, *my_state, "A00", forms[0]);
        auto A11_state = SubState(*InvA11_Fact_, *my_state, "A11", forms[1]);
        std::vector<std::shared_ptr<mfem::Solver>> inv_ops(2);
        inv_ops[0] = std::shared_ptr<mfem::Solver>{InvA00_Fact_->BuildSolver(blop->GetBlockPtr(0, 0), *A00_state)};
        inv_ops[0]->iterative_mode = false;
        SecondDiagonal A11 = SecondDiagonalOperator(*blop, *A11_state);
        inv_ops[1] = std::shared_ptr<mfem::Solver>{InvA11_Fact_->BuildSolver(A11.S, *A11_state)};
        inv_ops[1]->iterative_mode = false;
        return make_unique<BlockDiagonalSolver>(blop, inv_ops, std::move(A11));
    }
    void _do_set_default_parameters() override
    {
        auto &p = GetParameters();
        p.Get<bool>("Use Negative S", true); p.Get<double>("Alpha", 1.0); p.Get("S Type", "NONE");
    }
    void _do_initialize(const ParameterList &) override
    {
        PARELAG_ASSERT(HasValidSolverLibrary());
        auto &params = GetParameters();
        InvA00_Fact_ = GetSolverLibrary().GetSolverFactory(params.Get("A00 Inverse", "Default Hypre"));
        InvA11_Fact_ = GetSolverLibrary().GetSolverFactory(params.Get("A11 Inverse", "Default Hypre"));
        InitSchur();
    }
    std::shared_ptr<SolverFactory> InvA00_Fact_, InvA11_Fact_;
};

class Block2x2GaussSeidelSolverFactory : public BlockSolverFactory
{
    std::unique_ptr<mfem::Solver> _do_build_block_solver(const std::shared_ptr<MfemBlockOperator> &blop, SolverState &state) const override
    {
        PARELAG_ASSERT(blop->GetNumBlockRows() == 2 && blop->GetNumBlockCols() == 2);
        auto my_state = dynamic_cast<NestedSolverState *>(&state);
        PARELAG_ASSERT(my_state);
        const std::vector<int> forms = my_state->GetForms();
        PARELAG_TEST_FOR_EXCEPTION(forms.size() < 2, std::runtime_error, "Block GS: the state must carry two forms");
        auto A00_state = SubState(*InvA00_Fact_, *my_state, "A00", forms[0]);
        auto A11_state = SubState(*InvA11_Fact_, *my_state, "A11", forms[1]);
        std::vector<std::shared_ptr<mfem::Solver>> inv_ops(2);
        inv_ops[0] = std::shared_ptr<mfem::Solver>{InvA00_Fact_->BuildSolver(blop->GetBlockPtr(0, 0), *A00_state)};
        inv_ops[0]->iterative_mode = false;
        SecondDiagonal A11 = SecondDiagonalOperator(*blop, *A11_state);
        inv_ops[1] = std::shared_ptr<mfem::Solver>{InvA11_Fact_->BuildSolver(A11.S, *A11_state)};
        inv_ops[1]->iterative_mode = false;
        return make_unique<BlockTriangularSolver>(blop, inv_ops, std::move(A11), tri_);
    }
    void _do_set_default_parameters() override
    {
        auto &p = GetParameters();
        p.Get<bool>("Use Negative S", true); p.Get<double>("Alpha", 1.0); p.Get("S Type", "NONE"); p.Get("Use triangle", "Lower");
    }
    void _do_initialize(const ParameterList &) override
    {
        PARELAG_ASSERT(HasValidSolverLibrary());
        auto &params = GetParameters();
        InvA00_Fact_ = GetSolverLibrary().GetSolverFactory(params.Get("A00 Inverse", "Default Hypre"));
        InvA11_Fact_ = GetSolverLibrary().GetSolverFactory(params.Get("A11 Inverse", "Default Hypre"));
        InitSchur();
        // "Use triangle": Lower (default) or Upper, any letter case (ParELAG_Block2x2GaussSeidelSolverFactory.cpp:147-165)
        std::string tri = params.Get("Use triangle", "Lower");
        std::transform(tri.begin(), tri.end(), tri.begin(), ::toupper);
        PARELAG_TEST_FOR_EXCEPTION(tri != "LOWER" && tri != "UPPER", std::runtime_error,
                                   "Block2x2GaussSeidelSolverFactory: \"Use triangle\" = \"" << tri << "\" is invalid; valid options are \"Lower\" and \"Upper\"");
        tri_ = tri == "LOWER" ? BlockTriangularSolver::Triangle::LOWER_TRIANGLE : BlockTriangularSolver::Triangle::UPPER_TRIANGLE;
    }
    std::shared_ptr<SolverFactory> InvA00_Fact_, InvA11_Fact_;
    BlockTriangularSolver::Triangle tri_ = BlockTriangularSolver::Triangle::LOWER_TRIANGLE;
};

class Block2x2LDUSolverFactory : public BlockSolverFactory
{
    std::unique_ptr<mfem::Solver> _do_build_block_solver(const std::shared_ptr<MfemBlockOperator> &blop, SolverState &state) const override
    {
        PARELAG_ASSERT(blop->GetNumBlockRows() == 2 && blop->GetNumBlockCols() == 2);
        auto my_state = dynamic_cast<NestedSolverState *>(&state);
        PARELAG_ASSERT(my_state);
        const std::vector<int> forms = my_state->GetForms();
        PARELAG_TEST_FOR_EXCEPTION(forms.size() < 2, std::runtime_error, "Block LDU: the state must carry two forms");
        auto s1 = SubState(*InvA00_1_Fact_, *my_state, "A00_1", forms[0]);
        auto s2 = SubState(*InvA00_2_Fact_, *my_state, "A00_2", forms[0]);
        auto s3 = SubState(*InvA00_3_Fact_, *my_state, "A00_3", forms[0]);
        auto sS = SubState(*InvS_Fact_, *my_state, "InvS", forms[1]);
        auto A00 = blop->GetBlockPtr(0, 0);
        auto inv1 = std::shared_ptr<mfem::Solver>{InvA00_1_Fact_->BuildSolver(A00, *s1)};
        auto inv2 = std::shared_ptr<mfem::Solver>{InvA00_2_Fact_->BuildSolver(A00, *s2)};
        auto inv3 = std::shared_ptr<mfem::Solver>{InvA00_3_Fact_->BuildSolver(A00, *s3)};
        SecondDiagonal A11 = SecondDiagonalOperator(*blop, *sS);
        auto invS = std::shared_ptr<mfem::Solver>{InvS_Fact_->BuildSolver(A11.S, *sS)};
        return make_unique<Block2x2LDUInverseOperator>(blop, inv1, inv2, inv3, invS, std::move(A11), Damping_Factor_);
    }
    void _do_set_default_parameters() override
    {
        auto &p = GetParameters();
        p.Get<bool>("Use Negative S", true); p.Get<double>("Damping Factor", 1.0); p.Get<double>("Alpha", 1.0); p.Get<std::string>("S Type", "NONE");
    }
    void _do_initialize(const ParameterList &) override
    {
        PARELAG_ASSERT(HasValidSolverLibrary());
        auto &params = GetParameters();
        Damping_Factor_ = params.Get<double>("Damping Factor", 1.0);
        InvA00_1_Fact_ = GetSolverLibrary().GetSolverFactory(params.Get("A00_1 Inverse", "Default Hypre"));
        InvA00_2_Fact_ = GetSolverLibrary().GetSolverFactory(params.Get("A00_2 Inverse", "Default Hypre"));
        InvA00_3_Fact_ = GetSolverLibrary().GetSolverFactory(params.Get("A00_3 Inverse", "Default Hypre"));
        InvS_Fact_ = GetSolverLibrary().GetSolverFactory(params.Get("S Inverse", "Default Hypre"));
        InitSchur();
    }
    std::shared_ptr<SolverFactory> InvA00_1_Fact_, InvA00_2_Fact_, InvA00_3_Fact_, InvS_Fact_;
    double Damping_Factor_ = 1.0;
};
} // namespace parelag
