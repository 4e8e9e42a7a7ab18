// certify_demo.cpp — the certificate of the enumerated optimum through the C++ adapter:
//   SymmetricalParser::ParseFromFile -> Symmetrical::ToCanonical -> EnumerationSolver::solve() -> certify()
// usage: certify_demo [--ranges | --rhs-ranges] <symmetric LP file> [--optimal-duals]   prints one machine-readable line per fact: the optimum,
//        the verdict (ENUMGPU_CERT_*), the entering column of an edge ray, the duals, the reduced costs, the ray, the
//        counters of the auxiliary enumeration, and whether a solver with setCheckUnbounded(true) reports "objective is
//        unbounded".  --optimal-duals: both solvers use setOptimalDuals(true), and two more lines give the basis the
//        certificate belongs to (cert_basis) and where it came from (source, ENUMGPU_OPT_*).
//        --ranges: the cost ranging table instead (costRanges()): "ranging <status> <vertex bases> <ray bases>", then
//        one line per canonical column, "range j decrease increase decrease_rank increase_rank decrease_ray increase_ray".
//        --rhs-ranges: the right-hand-side ranging table instead (rhsRanges()): "rhs_ranging <status> <tight columns>
//        <bases> <singular>", "tight j0 j1 ...", then one line per row, "rhs i shadow_price decrease increase
//        decrease_rank increase_rank".
#include <cstdio>
#include <cstring>
#include <exception>
#include <stdexcept>

#include "EnumerationSolver.h"
#include "SymmetricalParser.h"

static int print_ranges(const Canonical& can)
{
    EnumerationSolver solver(can);
    solver.solve();
    const enumgpu_ranging& r = solver.costRanges();
    std::printf("ranging %d %llu %llu\n", r.status, (unsigned long long)r.n_vertex_bases, (unsigned long long)r.n_ray_bases);
    for (int j = 0; j < r.n; ++j) {
        const enumgpu_cost_range& v = r.range[j];
        std::printf("range %d %.17g %.17g %llu %llu %d %d\n", j, v.decrease, v.increase, (unsigned long long)v.decrease_rank,
                    (unsigned long long)v.increase_rank, v.decrease_ray, v.increase_ray);
    }
    return 0;
}

static int print_rhs_ranges(const Canonical& can)
{
    EnumerationSolver solver(can);
    solver.solve();
    const enumgpu_rhs_ranging& r = solver.rhsRanges();
    std::printf("rhs_ranging %d %d %llu %llu\n", r.status, r.n_tight, (unsigned long long)r.n_bases,
                (unsigned long long)r.n_singular);
    std::printf("tight");
    for (int k = 0; k < r.n_tight; ++k) std::printf(" %d", r.tight[k]);
    std::printf("\n");
    for (int i = 0; i < r.m; ++i) {
        const enumgpu_rhs_range& v = r.range[i];
        std::printf("rhs %d %.17g %.17g %.17g %llu %llu\n", i, v.shadow_price, v.decrease, v.increase,
                    (unsigned long long)v.decrease_rank, (unsigned long long)v.increase_rank);
    }
    return 0;
}

int main(int argc, char** argv)
{
    if (argc == 3 && (!std::strcmp(argv[1], "--ranges") || !std::strcmp(argv[1], "--rhs-ranges"))) {
        SymmetricalParser parser;
        auto sym = parser.ParseFromFile(argv[2]);
        if (!sym) { std::fprintf(stderr, "parse error: %s\n", parser.GetLastError().c_str()); return 3; }
        try {
            const bool rhs = !std::strcmp(argv[1], "--rhs-ranges");
            return rhs ? print_rhs_ranges(*sym->ToCanonical()) : print_ranges(*sym->ToCanonical());
        } catch (const std::exception& e) {
            std::fprintf(stderr, "error: %s\n", e.what());
            return 1;
        }
    }
    const bool optimal_duals = argc == 3 && !std::strcmp(argv[2], "--optimal-duals");
    if (argc < 2 || (argc > 2 && !optimal_duals)) {
        std::fprintf(stderr, "usage: %s [--ranges | --rhs-ranges] <symmetric LP file> [--optimal-duals]\n", argv[0]);
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
