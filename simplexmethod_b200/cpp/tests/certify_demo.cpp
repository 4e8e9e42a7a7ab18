// certify_demo.cpp — the certificate of the enumerated optimum through the C++ adapter:
//   SymmetricalParser::ParseFromFile -> Symmetrical::ToCanonical -> EnumerationSolver::solve() -> certify()
// usage: certify_demo <symmetric LP file> [--optimal-duals]   prints one machine-readable line per fact: the optimum,
//        the verdict (ENUMGPU_CERT_*), the entering column of an edge ray, the duals, the reduced costs, the ray, the
//        counters of the auxiliary enumeration, and whether a solver with setCheckUnbounded(true) reports "objective is
//        unbounded".  --optimal-duals: both solvers use setOptimalDuals(true), and two more lines give the basis the
//        certificate belongs to (cert_basis) and where it came from (source, ENUMGPU_OPT_*).
#include <cstdio>
#include <cstring>
#include <exception>
#include <stdexcept>

#include "EnumerationSolver.h"
#include "SymmetricalParser.h"

int main(int argc, char** argv)
{
    const bool optimal_duals = argc == 3 && !std::strcmp(argv[2], "--optimal-duals");
    if (argc < 2 || (argc > 2 && !optimal_duals)) {
        std::fprintf(stderr, "usage: %s <symmetric LP file> [--optimal-duals]\n", argv[0]);
        return 2;
    }
    SymmetricalParser parser;
    auto sym = parser.ParseFromFile(argv[1]);
    if (!sym) { std::fprintf(stderr, "parse error: %s\n", parser.GetLastError().c_str()); return 3; }
    auto can = sym->ToCanonical();
    try {
        EnumerationSolver solver(*can);
        solver.setOptimalDuals(optimal_duals);
        solver.solve();
        const enumgpu_certificate& cert = solver.certify();
        std::printf("objective %.17g\nbasis", solver.objective());
        for (int j : solver.optimalBasis()) std::printf(" %d", j);
        std::printf("\ncert_status %d\nentering %d\ny", cert.status, cert.entering);
        for (int i = 0; i < cert.m; ++i) std::printf(" %.17g", cert.y[i]);
        std::printf("\nreduced_cost");
        for (int j = 0; j < cert.n; ++j) std::printf(" %.17g", cert.reduced_cost[j]);
        std::printf("\nray");
        for (int j = 0; j < cert.n; ++j) std::printf(" %.17g", cert.ray[j]);
        std::printf("\naux_counts %llu %llu\n", (unsigned long long)cert.n_aux_bases, (unsigned long long)cert.n_rays);
        if (optimal_duals) {
            std::printf("cert_basis");
            for (int j : solver.certificateBasis()) std::printf(" %d", j);
            std::printf("\nsource %d\n", solver.certificateSource());
        }
        EnumerationSolver checked(*can);
        checked.setOptimalDuals(optimal_duals);
        checked.setCheckUnbounded(true);
        try {
            checked.solve();
            std::printf("check_unbounded 0\n");
        } catch (const std::runtime_error& e) {
            if (std::strcmp(e.what(), "objective is unbounded")) throw;
            std::printf("check_unbounded 1\n");
        }
    } catch (const std::exception& e) {
        std::fprintf(stderr, "error: %s\n", e.what());
        return 1;
    }
    return 0;
}
