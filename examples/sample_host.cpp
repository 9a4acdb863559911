// sample_host.cpp -- C++ caller of B200State::sample (include/qipb200.hpp): 10^4 shots of a Bell state drawn from one
// read of the device state.  Exit 0 when only 00 and 11 occur, each with frequency 0.5 +- 0.03.
// Build: see __graft_entry__.build().
#include <cmath>
#include <cstdio>
#include <random>

#include "qipb200.hpp"

int main() {
  using namespace qip;
  typedef std::complex<double> C;
  try {
    Context ctx(0);
    const double s = std::sqrt(0.5);
    B200State<double> st(ctx, 2);
    st.set_basis(0);
    st.apply_all({make_matrix_op<double>({0}, {C(s), C(s), C(s), C(-s)}),                                  // H(0)
                  make_control_op<double>({0}, make_matrix_op<double>({1}, {C(0), C(1), C(1), C(0)}))});  // CNOT(0 -> 1)
    std::mt19937_64 gen(12345);
    std::uniform_real_distribution<double> uni(0.0, 1.0);
    std::vector<double> draws(10000);
    for (double &r : draws) r = uni(gen);
    const std::vector<uint64_t> shots = st.sample({0, 1}, draws);
    size_t counts[4] = {0, 0, 0, 0};
    for (uint64_t m : shots) ++counts[m & 3];
    std::printf("shots=%zu  00:%zu 01:%zu 10:%zu 11:%zu\n", shots.size(), counts[0], counts[1], counts[2], counts[3]);
    const double f0 = counts[0] / (double)shots.size(), f3 = counts[3] / (double)shots.size();
    return (counts[1] == 0 && counts[2] == 0 && std::fabs(f0 - 0.5) < 0.03 && std::fabs(f3 - 0.5) < 0.03) ? 0 : 1;
  } catch (const CircuitError &e) {
    std::fprintf(stderr, "CircuitError(%d): %s\n", e.status, e.what());
    return 2;
  }
}
