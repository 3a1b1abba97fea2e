// Groth16::generate_parameters (include/pairing_b200.hpp) on a circuit read from a file; writes the key's rows for
// tests/test_gpu_groth16_setup.py to compare with the Python binding's.
// in:  u64 num_constraints, num_inputs, num_aux; per matrix u64 nnz, u64 offsets[nv + 1], u32 constraint[nnz], bls_fr coeff[nnz];
//      g1 (13 u64), g2 (25 u64), alpha, beta, gamma, delta, tau (4 u64 each)
// out: alpha_g1, beta_g1, delta_g1, beta_g2, gamma_g2, delta_g2, ic, h, l, a, b_g1, b_g2
#include <stdio.h>

#include "pairing_b200.hpp"

using namespace pairing_b200;

template <class T> static void rd(FILE* f, T* p, size_t n) {
  if (fread(p, sizeof(T), n, f) != n) throw std::runtime_error("short input");
}
template <class T> static void wr(FILE* f, const T* p, size_t n) { fwrite(p, sizeof(T), n, f); }

int main(int argc, char** argv) {
  if (argc != 3) return 1;
  FILE* f = fopen(argv[1], "rb");
  if (!f) return 1;
  uint64_t hdr[3];
  rd(f, hdr, 3);
  const size_t nv = hdr[1] + hdr[2];
  Groth16::Matrix abc[3];
  for (auto& m : abc) {
    uint64_t nnz;
    rd(f, &nnz, 1);
    m.offsets.resize(nv + 1); m.constraint.resize(nnz); m.coeff.resize(nnz);
    rd(f, m.offsets.data(), nv + 1);
    rd(f, m.constraint.data(), nnz);
    rd(f, m.coeff.data(), nnz);
  }
  bls_g1_affine g1;
  bls_g2_affine g2;
  bls_fr sc[5];
  rd(f, &g1, 1); rd(f, &g2, 1); rd(f, sc, 5);
  fclose(f);
  Gpu g(0);
  const Groth16::Parameters p = Groth16::generate_parameters(g, abc, hdr[0], hdr[1], hdr[2], g1, g2, sc[0], sc[1], sc[2], sc[3], sc[4]);
  FILE* o = fopen(argv[2], "wb");
  if (!o) return 1;
  wr(o, &p.alpha_g1, 1); wr(o, &p.beta_g1, 1); wr(o, &p.delta_g1, 1);
  wr(o, &p.beta_g2, 1); wr(o, &p.gamma_g2, 1); wr(o, &p.delta_g2, 1);
  for (const auto* v : {&p.ic, &p.h, &p.l, &p.a, &p.b_g1}) wr(o, v->data(), v->size());
  wr(o, p.b_g2.data(), p.b_g2.size());
  fclose(o);
  printf("cpp groth16 setup ok\n");
  return 0;
}
