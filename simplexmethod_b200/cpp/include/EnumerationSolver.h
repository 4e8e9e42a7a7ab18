// EnumerationSolver.h — the class the reference declares but never implements
// (reference: src/EnumerationSolver.h:3-10), with the call shape of its sibling
// Solver (reference: src/SimplexSolover.h:285-288):
//
//     EnumerationSolver solver(canonical);
//     Eigen::VectorXd x = solver.solve();        // first n_orig components, as
//                                                // SimplexSolover.h:435-439
//
// Header-only adapter over the C ABI of libenumgpu (include/enumgpu.h): every
// basis is evaluated on the GPU(s); nothing is computed here.  A is handed over
// as GetConstraintsMatrix().data() — Eigen's (and the shim's) column-major
// storage is the ABI's layout, so there is no copy or transposition.
// Errors: std::invalid_argument for bad dimensions (cf. Canonical.cpp:27-46),
// std::runtime_error when no basis is feasible (cf. SimplexSolover.h:371) or
// the CUDA side fails.
// Like Solver, which keeps its working state in the object (SimplexSolover.h:12),
// the solver keeps an enumgpu_handle per device from its first solve() on:
// stream, events, pinned staging and device buffers are created once, so a
// solve is one H2D copy, one kernel launch and one D2H copy.
#pragma once

#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "ProblemTypes/Canonical.h"
#include "enumgpu.h"

class EnumerationSolver {
public:
    explicit EnumerationSolver(const Canonical& problem) : problem_(problem)   // copied, like Solver (SimplexSolover.h:12,285)
    {
        const auto m = problem_.GetConstraintsMatrix().rows(), n = problem_.GetConstraintsMatrix().cols();
        if (m > n) throw std::invalid_argument("EnumerationSolver: more rows than columns, no basis exists");
        if (m < 1 || m > ENUMGPU_MAX_M || n > ENUMGPU_MAX_N)
            throw std::invalid_argument("EnumerationSolver: (m, n) outside the limits of libenumgpu");
    }

    ~EnumerationSolver() { release(); }
    EnumerationSolver(const EnumerationSolver& o)
        : problem_(o.problem_), devices_(o.devices_), algo_(o.algo_), rule_(o.rule_), eps_feas_(o.eps_feas_), eps_piv_(o.eps_piv_),
          rank_begin_(o.rank_begin_), rank_end_(o.rank_end_), check_unbounded_(o.check_unbounded_), optimal_duals_(o.optimal_duals_),
          res_(o.res_), cert_(o.cert_), cert_basis_(o.cert_basis_), solved_(o.solved_), certified_(o.certified_) {}   // handles are not shared
    EnumerationSolver& operator=(const EnumerationSolver&) = delete;

    // optional knobs (not in the reference)
    void setDevices(const std::vector<int>& cuda_ordinals) { release(); devices_.assign(cuda_ordinals.begin(), cuda_ordinals.end()); }
    void setPivotRule(int enumgpu_pivot_rule) { rule_ = enumgpu_pivot_rule; }    // ENUMGPU_PIVOT_ABSOLUTE (default) / _RELATIVE
    void setAlgorithm(int enumgpu_algo) { algo_ = enumgpu_algo; }
    void setTolerances(double eps_feas, double eps_piv) { eps_feas_ = eps_feas; eps_piv_ = eps_piv; }
    void setRankRange(uint64_t begin, uint64_t end) { rank_begin_ = begin; rank_end_ = end; }
    // solve() then certifies its optimum and throws std::runtime_error("objective is unbounded") on an unbounded
    // LP, as the reference's Solver does (SimplexSolover.h:443); needs the whole rank range.  The entry point is
    // held as a pointer so that a program which never turns the check on links only the entries it uses.
    void setCheckUnbounded(bool on) { check_unbounded_ = on ? &enumgpu_certify : nullptr; }
    // certify() (and the unboundedness check) searches all optimal bases for a dual-feasible one when the winner's
    // certificate is undecided (enumgpu_certify_optimum); certificateBasis() then names the basis the certificate
    // belongs to, which may differ from optimalBasis().  Off by default: it costs one more enumeration on a
    // degenerate optimum.  Held as a pointer for the same reason as above.
    void setOptimalDuals(bool on) { optimal_duals_ = on ? &enumgpu_certify_optimum : nullptr; }

    Eigen::VectorXd solve()
    {
        const Eigen::MatrixXd& A = problem_.GetConstraintsMatrix();
        const enumgpu_problem p = problemStruct();
        enumgpu_options o = options();
        o.rank_begin = rank_begin_; o.rank_end = rank_end_;
        o.n_devices = 0; o.devices = nullptr;                     // the handles name the devices
        if (check_unbounded_ && (rank_begin_ | rank_end_) && !(rank_begin_ == 0 && rank_end_ == binomial(p.n, p.m)))
            throw std::invalid_argument("EnumerationSolver: setCheckUnbounded needs the whole rank range");
        int rc = acquire();
        if (rc == ENUMGPU_OK) rc = enumgpu_solve_hv(handles_.data(), static_cast<int32_t>(handles_.size()), &p, &o, &res_);
        else res_.status = rc;
        solved_ = true;
        certified_ = false;
        if (rc == ENUMGPU_ERR_CUDA) throw std::runtime_error(std::string("libenumgpu: ") + enumgpu_last_error());
        if (rc < 0) throw std::invalid_argument(std::string("libenumgpu: ") + enumgpu_last_error());
        if (rc == ENUMGPU_NO_FEASIBLE) throw std::runtime_error("the problem has no feasible basic solution");
        if (check_unbounded_ && certifyWith(check_unbounded_, -1.0).status == ENUMGPU_CERT_UNBOUNDED)
            throw std::runtime_error("objective is unbounded");
        Eigen::VectorXd x = Eigen::VectorXd::Zero(A.cols());
        for (int i = 0; i < res_.m; ++i) x[res_.basis[i]] = res_.x_B[i];
        const int n_orig = problem_.GetOriginalVariablesCount();
        Eigen::VectorXd head(n_orig);
        for (int j = 0; j < n_orig; ++j) head[j] = x[j];
        return head;
    }

    // what the parity metric needs; valid after solve() (also after a "no feasible basis" throw)
    std::vector<int> optimalBasis() const { need(); return std::vector<int>(res_.basis, res_.basis + res_.m); }
    double   objective() const { need(); return res_.objective; }
    uint64_t bestRank() const { need(); return res_.best_rank; }
    uint64_t basesEvaluated() const { need(); return res_.n_bases; }
    uint64_t singularCount() const { need(); return res_.n_singular; }
    uint64_t infeasibleCount() const { need(); return res_.n_infeasible; }
    uint64_t feasibleCount() const { need(); return res_.n_feasible; }
    double   kernelMilliseconds() const { need(); return res_.kernel_ms; }

    // Certificate of the optimal basis of the last solve() (enumgpu_certify): dual values y, reduced costs, and the
    // verdict ENUMGPU_CERT_OPTIMAL / _BOUNDED / _UNBOUNDED (with a ray) / _UNDECIDED.  eps_opt < 0: 1e-9.
    const enumgpu_certificate& certify(double eps_opt = -1.0) { return certifyWith(&enumgpu_certify, eps_opt); }
    const enumgpu_certificate& certificate() const
    {
        if (!certified_) throw std::logic_error("EnumerationSolver: certify() has not been called");
        return cert_;
    }
    // the columns (ascending) of the basis the certificate belongs to; with setOptimalDuals(true) also the window
    // search's source (ENUMGPU_OPT_*), else ENUMGPU_OPT_WINNER
    const std::vector<int>& certificateBasis() const { certificate(); return cert_basis_; }
    int certificateSource() const { certificate(); return cert_source_; }

private:
    void need() const { if (!solved_) throw std::logic_error("EnumerationSolver: solve() has not been called"); }
    using CertifyFn = int (*)(const enumgpu_problem*, const enumgpu_options*, const int32_t*, double, enumgpu_certificate*);
    const enumgpu_certificate& certifyWith(CertifyFn fn, double eps_opt)
    {
        need();
        if (res_.status != ENUMGPU_OK) throw std::runtime_error("the problem has no feasible basic solution");
        const enumgpu_problem p = problemStruct();
        const enumgpu_options o = options();
        int rc;
        if (optimal_duals_) {
            enumgpu_optimum opt{};
            rc = optimal_duals_(&p, &o, &res_, eps_opt, 0, &opt);
            cert_ = opt.cert;
            cert_basis_.assign(opt.basis, opt.basis + res_.m);
            cert_source_ = opt.source;
        } else {
            rc = fn(&p, &o, res_.basis, eps_opt, &cert_);
            cert_basis_.assign(res_.basis, res_.basis + res_.m);
            cert_source_ = ENUMGPU_OPT_WINNER;
        }
        if (rc == ENUMGPU_ERR_CUDA) throw std::runtime_error(std::string("libenumgpu: ") + enumgpu_last_error());
        if (rc < 0) throw std::invalid_argument(std::string("libenumgpu: ") + enumgpu_last_error());
        certified_ = true;
        return cert_;
    }
    static uint64_t binomial(int n, int k)          // C(n, k) for n <= 64, k <= 16: exact in 64 bits
    {
        uint64_t r = 1;
        for (int i = 1; i <= k; ++i) r = r * static_cast<uint64_t>(n - k + i) / static_cast<uint64_t>(i);
        return r;
    }
    enumgpu_problem problemStruct() const
    {
        const Eigen::MatrixXd& A = problem_.GetConstraintsMatrix();
        enumgpu_problem p{};
        p.m = static_cast<int32_t>(A.rows());
        p.n = static_cast<int32_t>(A.cols());
        p.lda = p.m;
        p.maximize = problem_.IsMaximization() ? 1 : 0;
        p.A_colmajor = A.data();
        p.b = problem_.GetRightHandSide().data();
        p.c = problem_.GetObjectiveCoefficients().data();
        return p;
    }
    enumgpu_options options() const
    {
        enumgpu_options o{};
        o.eps_feas = eps_feas_; o.eps_piv = eps_piv_;
        o.algo = algo_;
        o.pivot_rule = rule_;
        o.n_devices = static_cast<int32_t>(devices_.size());
        o.devices = devices_.empty() ? nullptr : devices_.data();
        return o;
    }
    int acquire()
    {
        if (!handles_.empty()) return ENUMGPU_OK;
        const size_t nd = devices_.empty() ? 1 : devices_.size();
        for (size_t i = 0; i < nd; ++i) {
            enumgpu_handle* h = nullptr;
            const int rc = enumgpu_create(devices_.empty() ? -1 : devices_[i], &h);
            if (rc != ENUMGPU_OK) { release(); return rc; }
            handles_.push_back(h);
        }
        return ENUMGPU_OK;
    }
    void release()
    {
        for (enumgpu_handle* h : handles_) enumgpu_destroy(h);
        handles_.clear();
    }

    Canonical problem_;
    std::vector<int32_t> devices_;
    std::vector<enumgpu_handle*> handles_;
    int algo_ = ENUMGPU_ALGO_AUTO, rule_ = ENUMGPU_PIVOT_ABSOLUTE;
    double eps_feas_ = -1.0, eps_piv_ = -1.0;
    uint64_t rank_begin_ = 0, rank_end_ = 0;
    CertifyFn check_unbounded_ = nullptr;      // &enumgpu_certify when setCheckUnbounded(true)
    using OptimumFn = int (*)(const enumgpu_problem*, const enumgpu_options*, const enumgpu_result*, double, uint64_t,
                              enumgpu_optimum*);
    OptimumFn optimal_duals_ = nullptr;        // &enumgpu_certify_optimum when setOptimalDuals(true)
    enumgpu_result res_{};
    enumgpu_certificate cert_{};
    std::vector<int> cert_basis_;
    int cert_source_ = ENUMGPU_OPT_WINNER;
    bool solved_ = false, certified_ = false;
};
