// C++ driver for the satisfiability checks of include/vdf_host.hpp (R1CSShape::is_sat_relaxed / is_sat,
// RunningWitness::check): replays fixtures written by tests/sat_ref.py::sat_check_fixtures and compares the reports
// with the oracle's exactly.
//   usage: sat_check <fixture-dir>      exit 0 = all equal, 2 = mismatch, 3 = library/GPU error
#include <cstdio>
#include <fstream>
#include <iterator>
#include <string>

#include "../../include/vdf_host.hpp"

using namespace vdf_host;

static std::vector<uint8_t> slurp(const std::string& path) {
  std::ifstream f(path, std::ios::binary);
  if (!f) throw std::runtime_error("cannot open " + path);
  return std::vector<uint8_t>((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
}
template <class T>
static std::vector<T> as(const std::vector<uint8_t>& raw) {
  std::vector<T> v(raw.size() / sizeof(T));
  std::memcpy(v.data(), raw.data(), v.size() * sizeof(T));
  return v;
}

static int differs(const char* what, const SatReport& got, const uint64_t* want) {
  const bool same = got.bad_rows == want[0] && got.first_bad_row == want[1] && got.comm_W == want[2] && got.comm_E == want[3];
  std::printf("%s: [%llu %llu %llu %llu]%s\n", what, (unsigned long long)got.bad_rows, (unsigned long long)got.first_bad_row,
              (unsigned long long)got.comm_W, (unsigned long long)got.comm_E, same ? "" : "  MISMATCH");
  return same ? 0 : 1;
}

int main(int argc, char** argv) {
  if (argc != 2) { std::fprintf(stderr, "usage: sat_check <fixture-dir>\n"); return 1; }
  const std::string d = std::string(argv[1]) + "/";
  int bad = 0;
  try {
    init(0);
    auto dims = as<uint64_t>(slurp(d + "dims.bin"));   // cons, vars, io, nnzA, nnzB, nnzC
    CooMatrix M[3];
    const char* names[3] = {"a", "b", "c"};
    for (int m = 0; m < 3; m++) {
      M[m].rows = as<uint64_t>(slurp(d + names[m] + "_rows.bin"));
      M[m].cols = as<uint64_t>(slurp(d + names[m] + "_cols.bin"));
      M[m].vals = as<Fe>(slurp(d + names[m] + "_vals.bin"));
    }
    R1CSShape shape(VDFGPU_FQ, dims[0], dims[1], dims[2], M[0], M[1], M[2]);
    auto W = as<Fe>(slurp(d + "W.bin")), E = as<Fe>(slurp(d + "E.bin")), E_bad = as<Fe>(slurp(d + "E_bad.bin"));
    auto u = as<Fe>(slurp(d + "u.bin")), X = as<Fe>(slurp(d + "X.bin"));
    auto k0d = as<Fe>(slurp(d + "k0_d.bin"));
    auto comm = as<Point>(slurp(d + "comm.bin"));   // comm_W, comm_E
    auto want = as<uint64_t>(slurp(d + "reports.bin"));   // satisfied, then E[cons / 3] corrupted
    Generators g(VDFGPU_PALLAS, k0d[0], k0d[1], dims[0] > dims[1] ? dims[0] : dims[1], true);
    bad += differs("is_sat_relaxed", shape.is_sat_relaxed(&g, W, E, u[0], X, &comm[0], &comm[1]), &want[0]);
    bad += differs("is_sat_relaxed, E corrupted", shape.is_sat_relaxed(&g, W, E_bad, u[0], X, &comm[0], &comm[1]), &want[4]);
    RunningWitness run(shape, g);
    run.set(W, E, u[0], X);
    bad += differs("RunningWitness::check", run.check(&comm[0], &comm[1]), &want[0]);
    run.set(W, E_bad, u[0], X);
    bad += differs("RunningWitness::check, E corrupted", run.check(&comm[0], &comm[1]), &want[4]);
    // nova-snark answers a wrong length with InvalidWitnessLength; the host layer must not let the C ABI read past it
    auto throws = [](auto&& fn) { try { fn(); } catch (const std::invalid_argument&) { return 1; } return 0; };
    std::vector<Fe> shortW(W.begin(), W.end() - 1), shortE(E.begin(), E.end() - 1);
    bad += !throws([&] { shape.is_sat_relaxed(&g, shortW, E, u[0], X, nullptr, nullptr); });
    bad += !throws([&] { shape.is_sat_relaxed(&g, W, shortE, u[0], X, nullptr, nullptr); });
    bad += !throws([&] { shape.is_sat(&g, shortW, X, nullptr); });
  } catch (const std::exception& e) {
    std::fprintf(stderr, "sat_check: %s\n", e.what());
    return 3;
  }
  if (bad) { std::printf("MISMATCH (%d)\n", bad); return 2; }
  std::printf("OK\n");
  return 0;
}
