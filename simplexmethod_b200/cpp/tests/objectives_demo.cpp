// objectives_demo.cpp — many cost vectors over one LP through the C++ adapter:
//   SymmetricalParser::ParseFromFile -> Symmetrical::ToCanonical -> EnumerationSolver::solveObjectives()
// usage: objectives_demo <symmetric LP file> <cost file>
//        The cost file holds one cost vector per line, one value per original variable of the LP; the columns that
//        ToCanonical adds get cost 0, as they do for the file's own objective.  All vectors use the file's sense.
//        Prints, for cost vector i (0-based), the lines "status i s", "basis i j ...", "objective i z" and
//        "x i x_1 ... x_n" (x: the original variables).  The whole set is solved by one enumeration.
#include <cstdio>
#include <exception>
#include <fstream>
#include <sstream>
#include <string>
#include <vector>

#include "EnumerationSolver.h"
#include "SymmetricalParser.h"

int main(int argc, char** argv)
{
    if (argc != 3) {
        std::fprintf(stderr, "usage: %s <symmetric LP file> <cost file>\n", argv[0]);
        return 2;
    }
    SymmetricalParser parser;
    auto sym = parser.ParseFromFile(argv[1]);
    if (!sym) { std::fprintf(stderr, "parse error: %s\n", parser.GetLastError().c_str()); return 3; }
    auto can = sym->ToCanonical();
    const int n = static_cast<int>(can->GetConstraintsMatrix().cols()), n_orig = can->GetOriginalVariablesCount();
    std::ifstream in(argv[2]);
    if (!in) { std::fprintf(stderr, "cannot read %s\n", argv[2]); return 3; }
    std::vector<std::vector<double>> rows;
    for (std::string line; std::getline(in, line);) {
        std::istringstream ls(line);
        std::vector<double> row;
        for (double v; ls >> v;) row.push_back(v);
        if (row.empty()) continue;
        if (static_cast<int>(row.size()) != n_orig) {
            std::fprintf(stderr, "cost vector %zu has %zu values, the LP has %d variables\n", rows.size(), row.size(), n_orig);
            return 3;
        }
        rows.push_back(row);
    }
    if (rows.empty()) { std::fprintf(stderr, "no cost vector in %s\n", argv[2]); return 3; }
    Eigen::MatrixXd C = Eigen::MatrixXd::Zero(n, static_cast<Eigen::Index>(rows.size()));
    for (size_t i = 0; i < rows.size(); ++i)
        for (int j = 0; j < n_orig; ++j) C(j, static_cast<Eigen::Index>(i)) = rows[i][static_cast<size_t>(j)];
    try {
        EnumerationSolver solver(*can);
        const std::vector<Eigen::VectorXd> xs = solver.solveObjectives(C);
        const std::vector<enumgpu_result>& res = solver.objectiveResults();
        for (size_t i = 0; i < xs.size(); ++i) {
            std::printf("status %zu %d\nbasis %zu", i, res[i].status, i);
            for (int j = 0; j < res[i].m; ++j) std::printf(" %d", res[i].basis[j]);
            std::printf("\nobjective %zu %.17g\nx %zu", i, res[i].objective, i);
            for (Eigen::Index j = 0; j < xs[i].size(); ++j) std::printf(" %.17g", xs[i][j]);
            std::printf("\n");
        }
    } catch (const std::exception& e) {
        std::fprintf(stderr, "error: %s\n", e.what());
        return 1;
    }
    return 0;
}
