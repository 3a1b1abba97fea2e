// pairing_b200.hpp -- C++17 host-side mirror of the `pairing` crate's trait surface for the GPU path, over the C ABI
// of pairing_b200.h.  Header-only.
//
// The reference is Rust; this image has no Rust toolchain, so the host layer above the C ABI that a compiled caller
// uses is C++ (rust/src/lib.rs is the same layer authored in Rust).  Names, argument meaning and error behaviour
// follow the reference:
//   Engine            src/lib.rs:34-110       -> struct Bls12   { miller_loop, final_exponentiation, pairing }
//   CurveProjective   src/lib.rs:114-181      -> struct G1, G2  { double_, add_assign, add_assign_mixed, negate, sub_assign,
//                                                                  mul_assign, into_affine, batch_normalization,
//                                                                  recommended_wnaf_for_scalar / _for_num_scalars }
//   CurveAffine       src/lib.rs:185-234      -> struct G1Affine, G2Affine { prepare, pairing_with, into_projective,
//                                                                  into_compressed, into_uncompressed }
//   EncodedPoint      src/lib.rs:236-263      -> G1Compressed, G1Uncompressed, G2Compressed, G2Uncompressed
//   Wnaf              src/wnaf.rs:75-179      -> class Wnaf<G>  { scalar(k).base(g) | base(g, n).scalar(k) }
//   PrimeField (Fr)   bls12_381/fr.rs:271-572 -> struct FrField { from_repr, into_repr, add/sub/mul_assign, square, inverse, ... }
// Every value is a BATCH (std::vector of the ABI's POD structs): slice-level entry points are what a GPU is for.
// `Option` becomes std::optional, `Result<_, GroupDecodingError>` a per-element status; failures of the device layer
// throw pairing_b200::Error (nothing unwinds across the C ABI itself).  There is no CPU fallback.
#pragma once
#include <cstdint>
#include <cstring>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include "pairing_b200.h"
#include "pairing_b200_mpc.h"

namespace pairing_b200 {

using Fq = bls_fq;
using Fq2 = bls_fq2;
using Fq12 = bls_fq12;
using FrRepr = bls_fr_repr;
using G1Point = bls_g1;            // Jacobian (X, Y, Z), z == 0 <=> infinity (ec.rs:31-36)
using G2Point = bls_g2;
using G1AffinePoint = bls_g1_affine;
using G2AffinePoint = bls_g2_affine;
using G2PreparedPoint = bls_g2_prepared;
using G1PreparedPoint = bls_g1_affine;   // G1Prepared(G1Affine), ec.rs:924-935

struct Error : std::runtime_error {
  int status;
  Error(int s, const std::string& what) : std::runtime_error(what), status(s) {}
};

// One device context (one ordered stream).  Calls on a Gpu must be serialised by the caller.
class Gpu {
 public:
  explicit Gpu(int device = 0) {
    int err = 0;
    ctx_ = bls_ctx_create(device, &err);
    if (!ctx_) throw Error(err, bls_strerror(err));
  }
  ~Gpu() { bls_ctx_destroy(ctx_); }
  Gpu(const Gpu&) = delete;
  Gpu& operator=(const Gpu&) = delete;
  bls_ctx* ctx() const { return ctx_; }
  void check(int rc) const {
    if (rc != BLS_OK) throw Error(rc, std::string(bls_strerror(rc)) + " [" + bls_ctx_last_error(ctx_) + "]");
  }

 private:
  bls_ctx* ctx_;
};

// Several devices of one node behind ONE call (bls_mgpu): an n-pair product or batch is split into contiguous shards inside
// the library; the product's 576-byte partials meet on the first device, which runs the single final exponentiation.
class MultiGpu {
 public:
  explicit MultiGpu(const std::vector<int>& devices) {
    int err = 0;
    m_ = bls_mgpu_create(devices.data(), (int)devices.size(), &err);
    if (!m_) throw Error(err, bls_strerror(err));
  }
  ~MultiGpu() { bls_mgpu_destroy(m_); }
  MultiGpu(const MultiGpu&) = delete;
  MultiGpu& operator=(const MultiGpu&) = delete;
  bls_mgpu* handle() const { return m_; }
  int device_count() const { return bls_mgpu_device_count(m_); }
  void check(int rc) const {
    if (rc == BLS_OK) return;
    std::string msg = bls_strerror(rc);
    for (int i = 0; i < device_count(); i++) {
      const char* e = bls_ctx_last_error(bls_mgpu_ctx(m_, i));
      if (e && *e) msg += std::string(" [device ") + std::to_string(i) + ": " + e + "]";
    }
    throw Error(rc, msg);
  }

 private:
  bls_mgpu* m_;
};

inline bool operator==(const Fq12& a, const Fq12& b) { return std::memcmp(&a, &b, sizeof(Fq12)) == 0; }
inline bool operator!=(const Fq12& a, const Fq12& b) { return !(a == b); }

namespace detail {
inline Fq fq_one() {   // Montgomery R (fq.rs:22-30)
  return Fq{{0x760900000002fffdull, 0xebf4000bc40c0002ull, 0x5f48985753c758baull, 0x77ce585370525745ull, 0x5c071a97a256ec6dull, 0x15f65ec3fa80e493ull}};
}
inline int num_bits(const FrRepr& k) {   // fr.rs:213-225
  for (int i = 3; i >= 0; i--)
    if (k.l[i]) return 64 * i + 64 - __builtin_clzll(k.l[i]);
  return 0;
}
inline int rec_num_scalars(const std::vector<size_t>& table, size_t n) {   // ec.rs:907-921
  int ret = 4;
  for (size_t r : table) {
    if (n > r) ret++; else break;
  }
  return ret;
}
}  // namespace detail

inline Fq12 fq12_one() { Fq12 r; std::memset(&r, 0, sizeof r); r.c0.c0.c0 = detail::fq_one(); return r; }

// ------------------------------------------------------------------------------------------------ Engine
struct G2Affine;
struct Bls12 {
  // ONE Engine::miller_loop over all (G1Prepared, G2Prepared) pairs (mod.rs:40-102); pairs with an infinity member are skipped
  static Fq12 miller_loop(Gpu& g, const std::vector<G1PreparedPoint>& p, const std::vector<G2PreparedPoint>& q) {
    if (p.size() != q.size()) throw Error(BLS_ERR_INVALID_ARGUMENT, "miller_loop: length mismatch");
    Fq12 out;
    g.check(bls_multi_miller_loop_prepared(g.ctx(), p.data(), q.data(), p.size(), &out));
    return out;
  }
  // same, G2 coefficients generated on the fly from affine points (value-identical: the coefficient sequence is consumed in order)
  static Fq12 miller_loop(Gpu& g, const std::vector<G1AffinePoint>& p, const std::vector<G2AffinePoint>& q) {
    if (p.size() != q.size()) throw Error(BLS_ERR_INVALID_ARGUMENT, "miller_loop: length mismatch");
    Fq12 out;
    g.check(bls_multi_miller_loop(g.ctx(), p.data(), q.data(), p.size(), &out));
    return out;
  }
  // Engine::pairing with projective arguments (Into<G1Affine>, Into<G2Affine>), as bench_pairing_full calls it
  static std::vector<Fq12> pairing(Gpu& g, const std::vector<G1Point>& p, const std::vector<G2Point>& q) {
    if (p.size() != q.size()) throw Error(BLS_ERR_INVALID_ARGUMENT, "pairing: length mismatch");
    std::vector<Fq12> out(p.size());
    g.check(bls_pairing_projective_batch(g.ctx(), p.data(), q.data(), out.data(), p.size()));
    return out;
  }
  // the same ONE miller_loop sharded over several devices
  static Fq12 miller_loop(MultiGpu& g, const std::vector<G1AffinePoint>& p, const std::vector<G2AffinePoint>& q) {
    if (p.size() != q.size()) throw Error(BLS_ERR_INVALID_ARGUMENT, "miller_loop: length mismatch");
    Fq12 out;
    g.check(bls_mgpu_multi_miller_loop(g.handle(), p.data(), q.data(), p.size(), &out));
    return out;
  }
  // final_exponentiation(&miller_loop(pairs)) in one call (the batch-verification shape); nullopt is the reference's None
  static std::optional<Fq12> pairing_product(Gpu& g, const std::vector<G1AffinePoint>& p, const std::vector<G2AffinePoint>& q) {
    if (p.size() != q.size()) throw Error(BLS_ERR_INVALID_ARGUMENT, "pairing_product: length mismatch");
    Fq12 out; uint8_t some = 0;
    g.check(bls_pairing_product(g.ctx(), p.data(), q.data(), p.size(), &out, &some));
    return some ? std::optional<Fq12>(out) : std::nullopt;
  }
  static std::optional<Fq12> pairing_product(MultiGpu& g, const std::vector<G1AffinePoint>& p, const std::vector<G2AffinePoint>& q) {
    if (p.size() != q.size()) throw Error(BLS_ERR_INVALID_ARGUMENT, "pairing_product: length mismatch");
    Fq12 out; uint8_t some = 0;
    g.check(bls_mgpu_pairing_product(g.handle(), p.data(), q.data(), p.size(), &out, &some));
    return some ? std::optional<Fq12>(out) : std::nullopt;
  }
  static std::vector<Fq12> pairing(MultiGpu& g, const std::vector<G1AffinePoint>& p, const std::vector<G2AffinePoint>& q) {
    if (p.size() != q.size()) throw Error(BLS_ERR_INVALID_ARGUMENT, "pairing: length mismatch");
    std::vector<Fq12> out(p.size());
    g.check(bls_mgpu_pairing_batch(g.handle(), p.data(), q.data(), out.data(), p.size()));
    return out;
  }
  // n independent single-pair Miller loops
  static std::vector<Fq12> miller_loop_batch(Gpu& g, const std::vector<G1AffinePoint>& p, const std::vector<G2AffinePoint>& q) {
    if (p.size() != q.size()) throw Error(BLS_ERR_INVALID_ARGUMENT, "miller_loop_batch: length mismatch");
    std::vector<Fq12> out(p.size());
    g.check(bls_miller_loop_batch(g.ctx(), p.data(), q.data(), out.data(), p.size()));
    return out;
  }
  // Engine::final_exponentiation (mod.rs:104-160): None for a zero input
  static std::vector<std::optional<Fq12>> final_exponentiation(Gpu& g, const std::vector<Fq12>& f) {
    std::vector<Fq12> out(f.size());
    std::vector<uint8_t> some(f.size());
    g.check(bls_final_exponentiation_batch(g.ctx(), f.data(), out.data(), some.data(), f.size()));
    std::vector<std::optional<Fq12>> r(f.size());
    for (size_t i = 0; i < f.size(); i++)
      if (some[i]) r[i] = out[i];
    return r;
  }
  static std::optional<Fq12> final_exponentiation(Gpu& g, const Fq12& f) { return final_exponentiation(g, std::vector<Fq12>{f})[0]; }
  // Engine::pairing (lib.rs:101-109), per element
  static std::vector<Fq12> pairing(Gpu& g, const std::vector<G1AffinePoint>& p, const std::vector<G2AffinePoint>& q) {
    if (p.size() != q.size()) throw Error(BLS_ERR_INVALID_ARGUMENT, "pairing: length mismatch");
    std::vector<Fq12> out(p.size());
    g.check(bls_pairing_batch(g.ctx(), p.data(), q.data(), out.data(), p.size()));
    return out;
  }
  // e(p_i, q) for every p_i against ONE prepared q: `let q = Q.prepare(); for p in ps { pairing ... }`
  static std::vector<Fq12> pairing_shared_q(Gpu& g, const std::vector<G1AffinePoint>& p, const G2PreparedPoint& q) {
    std::vector<Fq12> out(p.size());
    g.check(bls_pairing_shared_q_batch(g.ctx(), p.data(), &q, out.data(), p.size()));
    return out;
  }
  static std::vector<Fq12> miller_loop_shared_q(Gpu& g, const std::vector<G1PreparedPoint>& p, const G2PreparedPoint& q) {
    std::vector<Fq12> out(p.size());
    g.check(bls_miller_loop_shared_q_batch(g.ctx(), p.data(), &q, out.data(), p.size()));
    return out;
  }
  // Field::pow on Fqk with a scalar-field exponent (lib.rs:306-324)
  static std::vector<Fq12> pow(Gpu& g, const std::vector<Fq12>& a, const std::vector<FrRepr>& k) {
    if (a.size() != k.size()) throw Error(BLS_ERR_INVALID_ARGUMENT, "pow: length mismatch");
    std::vector<Fq12> out(a.size());
    g.check(bls_fq12_pow_batch(g.ctx(), a.data(), k.data(), out.data(), a.size()));
    return out;
  }
  // Fqk::mul_assign over a whole slice (merging partial Miller products)
  static Fq12 product(Gpu& g, const std::vector<Fq12>& f) {
    Fq12 out;
    g.check(bls_fq12_product(g.ctx(), f.data(), f.size(), &out));
    return out;
  }
};

// every binary wrapper takes one n from the first vector: a shorter second vector would be read past its end by the H2D copy
inline void require_same_length(size_t a, size_t b, const char* what) {
  if (a != b) throw Error(BLS_ERR_INVALID_ARGUMENT, std::string(what) + ": length mismatch");
}

// ------------------------------------------------------------------------------------------------ scalar field
// PrimeField / Field for Fr (fr.rs:271-572), batch-shaped.  Values are Montgomery-form `bls_fr`; `from_repr` returns the
// per-element validity the reference reports as Err(NotInField).
struct FrField {
  using Elem = bls_fr;
  static std::vector<Elem> op(Gpu& g, int o, const std::vector<Elem>& a, const std::vector<Elem>* b, std::vector<uint8_t>* ok = nullptr) {
    if (b) require_same_length(a.size(), b->size(), "FrField::op");
    std::vector<Elem> out(a.size());
    std::vector<uint8_t> good(a.size());
    g.check(bls_fr_op_batch(g.ctx(), o, a.data(), b ? b->data() : nullptr, out.data(), good.data(), a.size()));
    if (ok) *ok = good;
    return out;
  }
  static std::vector<Elem> from_repr(Gpu& g, const std::vector<FrRepr>& r, std::vector<uint8_t>* ok = nullptr) {
    std::vector<Elem> a(r.size());
    std::memcpy(a.data(), r.data(), r.size() * sizeof(FrRepr));
    return op(g, BLS_OP_FROM_REPR, a, nullptr, ok);
  }
  static std::vector<FrRepr> into_repr(Gpu& g, const std::vector<Elem>& a) {
    auto o = op(g, BLS_OP_INTO_REPR, a, nullptr);
    std::vector<FrRepr> r(a.size());
    std::memcpy(r.data(), o.data(), a.size() * sizeof(FrRepr));
    return r;
  }
  static std::vector<Elem> add_assign(Gpu& g, const std::vector<Elem>& a, const std::vector<Elem>& b) { return op(g, BLS_OP_ADD, a, &b); }
  static std::vector<Elem> sub_assign(Gpu& g, const std::vector<Elem>& a, const std::vector<Elem>& b) { return op(g, BLS_OP_SUB, a, &b); }
  static std::vector<Elem> mul_assign(Gpu& g, const std::vector<Elem>& a, const std::vector<Elem>& b) { return op(g, BLS_OP_MUL, a, &b); }
  static std::vector<Elem> square(Gpu& g, const std::vector<Elem>& a) { return op(g, BLS_OP_SQR, a, nullptr); }
  static std::vector<Elem> negate(Gpu& g, const std::vector<Elem>& a) { return op(g, BLS_OP_NEG, a, nullptr); }
  static std::vector<Elem> double_(Gpu& g, const std::vector<Elem>& a) { return op(g, BLS_OP_DBL, a, nullptr); }
  // Field::inverse: ok[i] == 0 is the reference's None (zero has no inverse)
  static std::vector<Elem> inverse(Gpu& g, const std::vector<Elem>& a, std::vector<uint8_t>* ok = nullptr) { return op(g, BLS_OP_INV, a, nullptr, ok); }
  // bellman's EvaluationDomain over Fr: a.size() = m * 2^log_n coefficients of m polynomials back to back, natural order
  static std::vector<Elem> transform(Gpu& g, int kind, const std::vector<Elem>& a, int log_n) {
    if (log_n < 0 || log_n > 28 || a.size() % (size_t(1) << log_n)) throw std::invalid_argument("FrField: a.size() is not a multiple of 2^log_n");
    std::vector<Elem> out(a.size());
    g.check(bls_fr_fft_batch(g.ctx(), kind, a.data(), out.data(), log_n, a.size() >> log_n));
    return out;
  }
  static std::vector<Elem> fft(Gpu& g, const std::vector<Elem>& a, int log_n) { return transform(g, BLS_FFT, a, log_n); }
  static std::vector<Elem> ifft(Gpu& g, const std::vector<Elem>& a, int log_n) { return transform(g, BLS_IFFT, a, log_n); }
  static std::vector<Elem> coset_fft(Gpu& g, const std::vector<Elem>& a, int log_n) { return transform(g, BLS_COSET_FFT, a, log_n); }
  static std::vector<Elem> icoset_fft(Gpu& g, const std::vector<Elem>& a, int log_n) { return transform(g, BLS_ICOSET_FFT, a, log_n); }
  // Groth16's quotient polynomial for m proofs (the `h` block of bellman's create_proof): a, b, c hold m * len evaluations,
  // proof after proof; the result holds m * (n - 1) canonical FrRepr, n the smallest power of two >= len (1 for len <= 1)
  static std::vector<FrRepr> groth16_h(Gpu& g, const std::vector<Elem>& a, const std::vector<Elem>& b, const std::vector<Elem>& c, size_t m) {
    require_same_length(a.size(), b.size(), "FrField::groth16_h");
    require_same_length(a.size(), c.size(), "FrField::groth16_h");
    if (m == 0 ? !a.empty() : a.size() % m) throw std::invalid_argument("FrField::groth16_h: a.size() is not a multiple of m");
    const size_t len = m ? a.size() / m : 0;
    size_t n = 1;
    while (n < len) n <<= 1;
    std::vector<FrRepr> h(m * (n - 1));
    g.check(bls_fr_groth16_h_batch(g.ctx(), a.data(), b.data(), c.data(), len, m, h.data()));
    return h;
  }
};

// ------------------------------------------------------------------------------------------------ curves
template <class Proj, class Aff, bool IS_G2> struct Curve {
  using Projective = Proj;
  using Affine = Aff;
  static int op(Gpu& g, int o, const Proj* a, const void* b, Proj* out, size_t n) {
    if constexpr (IS_G2) return bls_g2_op_batch(g.ctx(), o, a, b, out, n);
    else return bls_g1_op_batch(g.ctx(), o, a, b, out, n);
  }
  static std::vector<Proj> unary(Gpu& g, int o, const std::vector<Proj>& a) {
    std::vector<Proj> out(a.size());
    g.check(op(g, o, a.data(), nullptr, out.data(), a.size()));
    return out;
  }
  // CurveProjective::double / negate / add_assign / sub_assign / add_assign_mixed (ec.rs:296-532, lib.rs:156-160)
  static std::vector<Proj> double_(Gpu& g, const std::vector<Proj>& a) { return unary(g, BLS_PT_DOUBLE, a); }
  static std::vector<Proj> negate(Gpu& g, const std::vector<Proj>& a) { return unary(g, BLS_PT_NEGATE, a); }
  static std::vector<Proj> add_assign(Gpu& g, const std::vector<Proj>& a, const std::vector<Proj>& b) {
    require_same_length(a.size(), b.size(), "add_assign");
    std::vector<Proj> out(a.size());
    g.check(op(g, BLS_PT_ADD, a.data(), b.data(), out.data(), a.size()));
    return out;
  }
  static std::vector<Proj> sub_assign(Gpu& g, const std::vector<Proj>& a, const std::vector<Proj>& b) {
    require_same_length(a.size(), b.size(), "sub_assign");
    std::vector<Proj> out(a.size());
    g.check(op(g, BLS_PT_SUB, a.data(), b.data(), out.data(), a.size()));
    return out;
  }
  static std::vector<Proj> add_assign_mixed(Gpu& g, const std::vector<Proj>& a, const std::vector<Aff>& b) {
    require_same_length(a.size(), b.size(), "add_assign_mixed");
    std::vector<Proj> out(a.size());
    g.check(op(g, BLS_PT_ADD_MIXED, a.data(), b.data(), out.data(), a.size()));
    return out;
  }
  // CurveProjective::mul_assign: double-and-add (ec.rs:534-553)
  static std::vector<Proj> mul_assign(Gpu& g, const std::vector<Proj>& a, const std::vector<FrRepr>& k) {
    require_same_length(a.size(), k.size(), "mul_assign");
    std::vector<Proj> out(a.size());
    if constexpr (IS_G2) g.check(bls_g2_mul_batch(g.ctx(), a.data(), k.data(), out.data(), a.size()));
    else g.check(bls_g1_mul_batch(g.ctx(), a.data(), k.data(), out.data(), a.size()));
    return out;
  }
  // CurveProjective::into_affine (ec.rs:586-619)
  static std::vector<Aff> into_affine(Gpu& g, const std::vector<Proj>& a) {
    std::vector<Aff> out(a.size());
    if constexpr (IS_G2) g.check(bls_g2_into_affine_batch(g.ctx(), a.data(), out.data(), a.size()));
    else g.check(bls_g1_into_affine_batch(g.ctx(), a.data(), out.data(), a.size()));
    return out;
  }
  // CurveProjective::batch_normalization (ec.rs:246-294), in place
  static void batch_normalization(Gpu& g, std::vector<Proj>& v) {
    if constexpr (IS_G2) g.check(bls_g2_batch_normalization(g.ctx(), v.data(), v.size()));
    else g.check(bls_g1_batch_normalization(g.ctx(), v.data(), v.size()));
  }
  static bool is_zero(const Proj& p) {   // ec.rs:238-240
    const uint64_t* z = reinterpret_cast<const uint64_t*>(&p.z);
    for (size_t i = 0; i < sizeof(p.z) / 8; i++)
      if (z[i]) return false;
    return true;
  }
  // ec.rs:895-905 / 1586-1596
  static int recommended_wnaf_for_scalar(const FrRepr& k) {
    const int nb = detail::num_bits(k);
    if constexpr (IS_G2) return nb >= 103 ? 4 : (nb >= 37 ? 3 : 2);
    else return nb >= 130 ? 4 : (nb >= 34 ? 3 : 2);
  }
  // ec.rs:907-921 / 1598-1612
  static int recommended_wnaf_for_num_scalars(size_t n) {
    if constexpr (IS_G2) return detail::rec_num_scalars({1, 3, 8, 20, 47, 126, 260, 826, 1501, 4555, 84071}, n);
    else return detail::rec_num_scalars({1, 3, 7, 20, 43, 120, 273, 563, 1630, 3128, 7933, 62569}, n);
  }
  // Wnaf::new().scalar(k_i).base(g_i) for every i (wnaf.rs:111-164)
  static std::vector<Proj> wnaf_mul(Gpu& g, const std::vector<Proj>& bases, const std::vector<FrRepr>& k) {
    if (bases.size() != k.size()) throw Error(BLS_ERR_INVALID_ARGUMENT, "wnaf_mul: length mismatch");
    std::vector<Proj> out(bases.size());
    if constexpr (IS_G2) g.check(bls_g2_wnaf_mul_batch(g.ctx(), bases.data(), k.data(), out.data(), bases.size()));
    else g.check(bls_g1_wnaf_mul_batch(g.ctx(), bases.data(), k.data(), out.data(), bases.size()));
    return out;
  }
  // sum_i k_i * bases_i (bucket method): the normalised representative, (x, y, one) or zero() = (0, one, 0)
  static Proj multiexp(Gpu& g, const std::vector<Aff>& bases, const std::vector<FrRepr>& k) {
    require_same_length(bases.size(), k.size(), "multiexp");
    Proj out;
    if constexpr (IS_G2) g.check(bls_g2_msm(g.ctx(), bases.data(), k.data(), bases.size(), &out));
    else g.check(bls_g1_msm(g.ctx(), bases.data(), k.data(), bases.size(), &out));
    return out;
  }
  // m independent multiexp sums in one call: sum j = sum_i k[j*n + i] * bases[b(j, i)], n = k.size() / m, with
  // b(j, i) = i when bases.size() == n (one set for every sum) and j*n + i when bases.size() == k.size()
  static std::vector<Proj> multiexp_batch(Gpu& g, const std::vector<Aff>& bases, const std::vector<FrRepr>& k, size_t m) {
    if (m == 0 ? !k.empty() : k.size() % m != 0) throw Error(BLS_ERR_INVALID_ARGUMENT, "multiexp_batch: k.size() is not a multiple of m");
    const size_t n = m ? k.size() / m : 0;
    if (bases.size() != n && bases.size() != k.size()) throw Error(BLS_ERR_INVALID_ARGUMENT, "multiexp_batch: bases.size() is neither k.size() / m nor k.size()");
    const int shared = bases.size() == n;
    std::vector<Proj> out(m);
    if constexpr (IS_G2) g.check(bls_g2_msm_batch(g.ctx(), bases.data(), shared, k.data(), n, m, out.data()));
    else g.check(bls_g1_msm_batch(g.ctx(), bases.data(), shared, k.data(), n, m, out.data()));
    return out;
  }
  // From<affine> for projective (ec.rs:570-582)
  static std::vector<Proj> into_projective(const std::vector<Aff>& a) {
    std::vector<Proj> out(a.size());
    for (size_t i = 0; i < a.size(); i++) {
      std::memset(&out[i], 0, sizeof(Proj));
      if (a[i].infinity) {
        reinterpret_cast<Fq*>(&out[i].y)[0] = detail::fq_one();        // zero() = (0, 1, 0)
      } else {
        out[i].x = a[i].x; out[i].y = a[i].y;
        reinterpret_cast<Fq*>(&out[i].z)[0] = detail::fq_one();
      }
    }
    return out;
  }
};
using G1 = Curve<G1Point, G1AffinePoint, false>;
using G2 = Curve<G2Point, G2AffinePoint, true>;

// ------------------------------------------------------------------------------------------------ Groth16 prover
// bellman's groth16::create_proof for m proofs of one circuit (bls_groth16_prove_batch): Params holds the vk points and the
// queries of the proving key; the assignments of the m proofs are back to back (a, b, c: m * len, input: m * num_inputs,
// aux: m * num_aux, r, s: m); the densities are bit-vec's BitVec<u32> words of DensityTracker (shared by the m proofs).
struct Groth16 {
  using Proof = bls_groth16_proof;
  struct Params {
    G1AffinePoint alpha_g1, beta_g1, delta_g1;
    G2AffinePoint beta_g2, delta_g2;
    std::vector<G1AffinePoint> h, l, a, b_g1;
    std::vector<G2AffinePoint> b_g2;
  };
  static std::vector<Proof> create_proof(Gpu& g, const Params& p, const std::vector<bls_fr>& a, const std::vector<bls_fr>& b,
                                         const std::vector<bls_fr>& c, const std::vector<bls_fr>& input, const std::vector<bls_fr>& aux,
                                         const std::vector<uint32_t>& a_aux_density, const std::vector<uint32_t>& b_input_density,
                                         const std::vector<uint32_t>& b_aux_density, const std::vector<bls_fr>& r, const std::vector<bls_fr>& s,
                                         size_t m) {
    if (m == 0 ? !(a.empty() && input.empty() && aux.empty()) : (a.size() % m || input.size() % m || aux.size() % m))
      throw Error(BLS_ERR_INVALID_ARGUMENT, "Groth16::create_proof: a, input or aux is not m rows");
    if (b.size() != a.size() || c.size() != a.size() || r.size() != m || s.size() != m)
      throw Error(BLS_ERR_INVALID_ARGUMENT, "Groth16::create_proof: b, c must match a and r, s hold m values");
    if (p.b_g1.size() != p.b_g2.size()) throw Error(BLS_ERR_INVALID_ARGUMENT, "Groth16::create_proof: b_g1 and b_g2 differ in length");
    const size_t len = m ? a.size() / m : 0, ni = m ? input.size() / m : 0, na = m ? aux.size() / m : 0;
    if (a_aux_density.size() < (na + 31) / 32 || b_aux_density.size() < (na + 31) / 32 || b_input_density.size() < (ni + 31) / 32)
      throw Error(BLS_ERR_INVALID_ARGUMENT, "Groth16::create_proof: a density bitmap is shorter than its variables");
    bls_groth16_params c_params{p.alpha_g1, p.beta_g1, p.delta_g1, p.beta_g2, p.delta_g2, p.h.data(), p.l.data(), p.a.data(),
                                p.b_g1.data(), p.b_g2.data(), p.h.size(), p.l.size(), p.a.size(), p.b_g1.size()};
    std::vector<Proof> out(m);
    g.check(bls_groth16_prove_batch(g.ctx(), &c_params, a.data(), b.data(), c.data(), len, input.data(), ni, aux.data(), na, a_aux_density.data(),
                                    b_input_density.data(), b_aux_density.data(), r.data(), s.data(), m, out.data()));
    return out;
  }

  // bellman's prepare_verifying_key (bls_groth16_prepare_verifying_key); ic stays with the caller
  using PreparedVerifyingKey = bls_groth16_pvk;
  static std::unique_ptr<PreparedVerifyingKey> prepare_verifying_key(Gpu& g, const G1AffinePoint& alpha_g1, const G2AffinePoint& beta_g2,
                                                                     const G2AffinePoint& gamma_g2, const G2AffinePoint& delta_g2) {
    std::unique_ptr<PreparedVerifyingKey> pvk(new PreparedVerifyingKey);
    g.check(bls_groth16_prepare_verifying_key(g.ctx(), &alpha_g1, &beta_g2, &gamma_g2, &delta_g2, pvk.get()));
    return pvk;
  }
  // bellman's verify_proof for m = proofs.size() proofs (bls_groth16_verify_batch): ic holds num_inputs + 1 points, inputs the
  // m rows of num_inputs public inputs (without the leading one) back to back
  static std::vector<bool> verify_proof(Gpu& g, const PreparedVerifyingKey& pvk, const std::vector<G1AffinePoint>& ic,
                                        const std::vector<Proof>& proofs, const std::vector<bls_fr>& inputs) {
    if (ic.empty() || inputs.size() != proofs.size() * (ic.size() - 1))
      throw Error(BLS_ERR_INVALID_ARGUMENT, "Groth16::verify_proof: inputs must hold num_inputs = ic.size() - 1 values per proof");
    std::vector<uint8_t> ok(proofs.size());
    g.check(bls_groth16_verify_batch(g.ctx(), &pvk, ic.data(), ic.size() - 1, proofs.data(), inputs.data(), proofs.size(), ok.data()));
    return std::vector<bool>(ok.begin(), ok.end());
  }
  // the randomized batch check (bls_groth16_verify_rlc_batch) with the caller's randomizers rho (canonical FrRepr, one per proof)
  static bool verify_proofs_batch(Gpu& g, const PreparedVerifyingKey& pvk, const std::vector<G1AffinePoint>& ic, const std::vector<Proof>& proofs,
                                  const std::vector<bls_fr>& inputs, const std::vector<bls_fr_repr>& rho) {
    if (ic.empty() || inputs.size() != proofs.size() * (ic.size() - 1) || rho.size() != proofs.size())
      throw Error(BLS_ERR_INVALID_ARGUMENT, "Groth16::verify_proofs_batch: inputs must hold ic.size() - 1 values and rho one value per proof");
    uint8_t ok = 0;
    g.check(bls_groth16_verify_rlc_batch(g.ctx(), &pvk, ic.data(), ic.size() - 1, proofs.data(), inputs.data(), rho.data(), proofs.size(), &ok));
    return ok != 0;
  }

  // bellman's groth16::generate_parameters (bls_groth16_generate_parameters_batch).  Each matrix is variable-major over
  // num_inputs + num_aux variables (offsets of nv + 1 entries), as KeypairAssembly records A, B and C.  The queries come back
  // trimmed to a_len and b_len, so the Parameters go to create_proof unchanged, with the density bitmaps next to them.
  // Throws on bellman's UnconstrainedVariable (ok = 0).
  struct Matrix {
    std::vector<uint64_t> offsets;
    std::vector<uint32_t> constraint;
    std::vector<bls_fr> coeff;
  };
  struct Parameters : Params {
    G2AffinePoint gamma_g2;
    std::vector<G1AffinePoint> ic;
    std::vector<uint32_t> a_aux_density, b_input_density, b_aux_density;
  };
  static Parameters generate_parameters(Gpu& g, const Matrix abc[3], size_t num_constraints, size_t num_inputs, size_t num_aux,
                                        const G1AffinePoint& g1, const G2AffinePoint& g2, const bls_fr& alpha, const bls_fr& beta,
                                        const bls_fr& gamma, const bls_fr& delta, const bls_fr& tau) {
    return build_key(abc, num_constraints, num_inputs, num_aux, "Groth16::generate_parameters",
                     "UnconstrainedVariable (an l query point is the identity)", [&](const bls_r1cs_matrix* m, const bls_groth16_parameters_out* out) {
      g.check(bls_groth16_generate_parameters_batch(g.ctx(), m, num_constraints, num_inputs, num_aux, &g1, &g2, &alpha, &beta, &gamma, &delta, &tau, out));
    });
  }

  // phase2's MPCParameters::new (bls_groth16_mpc_new_batch): the circuit's key from powersoftau's prepare_phase2 rows for the
  // domain of num_constraints (phase1.n of them; h: n - 1), before any contribution.  Throws on UnconstrainedVariable and on a
  // transcript whose b_g1 and b_g2 disagree on the identity (ok = 0).
  struct Phase1 {
    G1AffinePoint alpha_g1, beta_g1;
    G2AffinePoint beta_g2;
    std::vector<G1AffinePoint> coeffs_g1, alpha_coeffs_g1, beta_coeffs_g1;
    std::vector<G2AffinePoint> coeffs_g2;
    std::vector<G1AffinePoint> h;
  };
  static Parameters mpc_new(Gpu& g, const Matrix abc[3], size_t num_constraints, size_t num_inputs, size_t num_aux, const Phase1& phase1,
                            const G1AffinePoint& g1, const G2AffinePoint& g2) {
    const size_t n = phase1.coeffs_g1.size();
    if (phase1.alpha_coeffs_g1.size() != n || phase1.beta_coeffs_g1.size() != n || phase1.coeffs_g2.size() != n || phase1.h.size() + 1 != n)
      throw Error(BLS_ERR_INVALID_ARGUMENT, "Groth16::mpc_new: the transcript needs n rows per coefficient set and n - 1 h rows");
    const bls_groth16_phase1 ph{phase1.alpha_g1, phase1.beta_g1, phase1.beta_g2, phase1.coeffs_g1.data(), phase1.alpha_coeffs_g1.data(),
                                phase1.beta_coeffs_g1.data(), phase1.coeffs_g2.data(), phase1.h.data(), n};
    return build_key(abc, num_constraints, num_inputs, num_aux, "Groth16::mpc_new",
                     "UnconstrainedVariable (an l query point is the identity) or b_g1 and b_g2 disagreeing on the identity", [&](const bls_r1cs_matrix* m, const bls_groth16_parameters_out* out) {
      g.check(bls_groth16_mpc_new_batch(g.ctx(), m, num_constraints, num_inputs, num_aux, &ph, &g1, &g2, out));
    });
  }

  // phase2's MPCParameters::contribute (bls_groth16_mpc_contribute_batch) for the caller's secret delta, s and r =
  // hash_to_g2(transcript): h and l multiplied by delta^-1, delta_g1 and delta_g2 by delta, in place.  Returns the public key.
  static bls_groth16_mpc_pubkey mpc_contribute(Gpu& g, Parameters& p, const bls_fr& delta, const G1AffinePoint& s, const G2AffinePoint& r) {
    bls_groth16_vk_points vk{p.alpha_g1, p.beta_g1, p.delta_g1, p.beta_g2, p.gamma_g2, p.delta_g2};
    bls_groth16_mpc_pubkey pk;
    g.check(bls_groth16_mpc_contribute_batch(g.ctx(), &delta, &s, &r, &vk, p.h.data(), p.h.size(), p.l.data(), p.l.size(), p.h.data(), p.l.data(), &pk));
    p.delta_g1 = vk.delta_g1;
    p.delta_g2 = vk.delta_g2;
    return pk;
  }

  // phase2's MPCParameters::verify (bls_groth16_mpc_verify_batch): before = the key of mpc_new, after = the contributed key,
  // pks the contributions in order, rho_h / rho_l the caller's randomizers (one per h and l row).
  static bool mpc_verify(Gpu& g, const Parameters& before, const Parameters& after, const std::vector<bls_groth16_mpc_pubkey>& pks,
                         const std::vector<bls_fr_repr>& rho_h, const std::vector<bls_fr_repr>& rho_l) {
    if (rho_h.size() != before.h.size() || rho_l.size() != before.l.size())
      throw Error(BLS_ERR_INVALID_ARGUMENT, "Groth16::mpc_verify: one randomizer per h and l row");
    auto key = [](const Parameters& p) {
      return bls_groth16_key{{p.alpha_g1, p.beta_g1, p.delta_g1, p.beta_g2, p.gamma_g2, p.delta_g2}, p.ic.data(), p.h.data(), p.l.data(), p.a.data(),
                             p.b_g1.data(), p.b_g2.data(), p.ic.size(), p.h.size(), p.l.size(), p.a.size(), p.b_g1.size()};
    };
    const bls_groth16_key kb = key(before), ka = key(after);
    uint8_t ok = 0;
    g.check(bls_groth16_mpc_verify_batch(g.ctx(), &kb, &ka, pks.data(), pks.size(), rho_h.data(), rho_l.data(), &ok));
    return ok != 0;
  }

 private:
  template <class Call>
  static Parameters build_key(const Matrix abc[3], size_t num_constraints, size_t num_inputs, size_t num_aux, const char* who, const char* not_ok,
                              Call call) {
    const size_t nv = num_inputs + num_aux;
    bls_r1cs_matrix m[3];
    for (int i = 0; i < 3; i++) {
      if (abc[i].offsets.size() != nv + 1 || abc[i].constraint.size() != abc[i].coeff.size())
        throw Error(BLS_ERR_INVALID_ARGUMENT, std::string(who) + ": offsets must hold nv + 1 entries and constraint one per coeff");
      m[i] = bls_r1cs_matrix{abc[i].offsets.data(), abc[i].constraint.data(), abc[i].coeff.data(), abc[i].coeff.size()};
    }
    size_t n = 1;
    while (n < num_constraints) n <<= 1;
    Parameters p;
    p.h.resize(n - 1); p.l.resize(num_aux); p.a.resize(nv); p.b_g1.resize(nv); p.b_g2.resize(nv); p.ic.resize(num_inputs);
    p.a_aux_density.resize((num_aux + 31) / 32); p.b_input_density.resize((num_inputs + 31) / 32); p.b_aux_density.resize((num_aux + 31) / 32);
    bls_groth16_vk_points vk;
    uint64_t lens[2] = {0, 0};
    uint8_t ok = 0;
    bls_groth16_parameters_out out{&vk, p.ic.data(), p.h.data(), p.l.data(), p.a.data(), p.b_g1.data(), p.b_g2.data(), p.a_aux_density.data(),
                                   p.b_input_density.data(), p.b_aux_density.data(), lens, &ok};
    call(m, &out);
    if (!ok) throw Error(BLS_ERR_INVALID_ARGUMENT, std::string(who) + ": " + not_ok);
    p.alpha_g1 = vk.alpha_g1; p.beta_g1 = vk.beta_g1; p.delta_g1 = vk.delta_g1;
    p.beta_g2 = vk.beta_g2; p.gamma_g2 = vk.gamma_g2; p.delta_g2 = vk.delta_g2;
    p.a.resize(lens[0]); p.b_g1.resize(lens[1]); p.b_g2.resize(lens[1]);
    return p;
  }
};

// ------------------------------------------------------------------------------------------------ KZG commitments
// m polynomials of n coefficients (Montgomery bls_fr) back to back in p; srs[i] = [tau^i] g.  See pairing_b200.h.
struct Kzg {
  using PreparedVerifyingKey = bls_kzg_pvk;
  static size_t rows(size_t coeffs, size_t n, const char* what) {
    if (n == 0 ? coeffs != 0 : coeffs % n) throw Error(BLS_ERR_INVALID_ARGUMENT, what);
    return n ? coeffs / n : 0;
  }
  // c[j] = sum_i p[j*n + i] srs[i]; with n = 0 the number of polynomials is m
  static std::vector<G1AffinePoint> commit(Gpu& g, const std::vector<G1AffinePoint>& srs, const std::vector<bls_fr>& p, size_t n, size_t m = 0) {
    if (n) m = rows(p.size(), n, "Kzg::commit: p must hold m rows of n coefficients");
    std::vector<G1AffinePoint> c(m);
    g.check(bls_kzg_commit_batch(g.ctx(), srs.data(), srs.size(), p.data(), n, m, c.data()));
    return c;
  }
  struct Opening { std::vector<bls_fr> y; std::vector<G1AffinePoint> proof; };
  // open polynomial j at z[j]: y[j] = p_j(z_j), proof[j] = [q_j(tau)] g
  static Opening open(Gpu& g, const std::vector<G1AffinePoint>& srs, const std::vector<bls_fr>& p, size_t n, const std::vector<bls_fr>& z) {
    if (p.size() != n * z.size()) throw Error(BLS_ERR_INVALID_ARGUMENT, "Kzg::open: p must hold z.size() rows of n coefficients");
    Opening o{std::vector<bls_fr>(z.size()), std::vector<G1AffinePoint>(z.size())};
    g.check(bls_kzg_open_batch(g.ctx(), srs.data(), srs.size(), p.data(), n, z.data(), z.size(), o.y.data(), o.proof.data()));
    return o;
  }
  static std::unique_ptr<PreparedVerifyingKey> prepare_verifying_key(Gpu& g, const G1AffinePoint& g1, const G2AffinePoint& h, const G2AffinePoint& tau_h) {
    std::unique_ptr<PreparedVerifyingKey> pvk(new PreparedVerifyingKey);
    g.check(bls_kzg_prepare_verifying_key(g.ctx(), &g1, &h, &tau_h, pvk.get()));
    return pvk;
  }
  static std::vector<bool> verify(Gpu& g, const PreparedVerifyingKey& pvk, const std::vector<G1AffinePoint>& c, const std::vector<bls_fr>& y,
                                  const std::vector<bls_fr>& z, const std::vector<G1AffinePoint>& proof) {
    if (y.size() != c.size() || z.size() != c.size() || proof.size() != c.size())
      throw Error(BLS_ERR_INVALID_ARGUMENT, "Kzg::verify: c, y, z and proof must have one length");
    std::vector<uint8_t> ok(c.size());
    g.check(bls_kzg_verify_batch(g.ctx(), &pvk, c.data(), y.data(), z.data(), proof.data(), c.size(), ok.data()));
    return std::vector<bool>(ok.begin(), ok.end());
  }
  // the randomized check with the caller's randomizers rho (canonical FrRepr, one per proof)
  static bool verify_batch(Gpu& g, const PreparedVerifyingKey& pvk, const std::vector<G1AffinePoint>& c, const std::vector<bls_fr>& y,
                           const std::vector<bls_fr>& z, const std::vector<G1AffinePoint>& proof, const std::vector<bls_fr_repr>& rho) {
    if (y.size() != c.size() || z.size() != c.size() || proof.size() != c.size() || rho.size() != c.size())
      throw Error(BLS_ERR_INVALID_ARGUMENT, "Kzg::verify_batch: c, y, z, proof and rho must have one length");
    uint8_t ok = 0;
    g.check(bls_kzg_verify_rlc_batch(g.ctx(), &pvk, c.data(), y.data(), z.data(), proof.data(), rho.data(), c.size(), &ok));
    return ok != 0;
  }
  // openings at every omega^k (FK20): the table (2n rows) once per SRS and n = 2^log_n, then y[j*n + k] = p_j(omega^k) and
  // proof[j*n + k] = open(srs, p_j, omega^k).proof for the m = p.size() / n polynomials of p
  static std::vector<G1AffinePoint> open_all_prepare(Gpu& g, const std::vector<G1AffinePoint>& srs, int log_n) {
    if (log_n < 0 || log_n > 24) throw Error(BLS_ERR_INVALID_ARGUMENT, "Kzg::open_all_prepare: log_n must be in 0..24");
    std::vector<G1AffinePoint> table(size_t(2) << log_n);
    g.check(bls_kzg_open_all_prepare(g.ctx(), srs.data(), srs.size(), log_n, table.data()));
    return table;
  }
  static Opening open_all(Gpu& g, const std::vector<G1AffinePoint>& table, const std::vector<bls_fr>& p, int log_n) {
    if (log_n < 0 || log_n > 24 || table.size() != (size_t(2) << log_n))
      throw Error(BLS_ERR_INVALID_ARGUMENT, "Kzg::open_all: the table must hold 2n rows, n = 2^log_n <= 2^24");
    const size_t m = rows(p.size(), size_t(1) << log_n, "Kzg::open_all: p must hold m rows of n coefficients");
    Opening o{std::vector<bls_fr>(p.size()), std::vector<G1AffinePoint>(p.size())};
    g.check(bls_kzg_open_all_batch(g.ctx(), table.data(), p.data(), log_n, m, o.y.data(), o.proof.data()));
    return o;
  }
};

// ------------------------------------------------------------------------------------------------ point FFT
// bellman's EvaluationDomain<Point<G>>: a.size() = m * 2^log_n affine points of m rows back to back, natural order; the
// results are canonical affine rows.  Defined for points of order r (see pairing_b200.h).
struct PointFft {
  template <class Aff, class Fn> static std::vector<Aff> run(Gpu& g, Fn fn, int kind, const std::vector<Aff>& a, int log_n) {
    if (log_n < 0 || log_n > 26 || a.size() % (size_t(1) << log_n)) throw std::invalid_argument("PointFft: a.size() is not a multiple of 2^log_n");
    std::vector<Aff> out(a.size());
    g.check(fn(g.ctx(), kind, a.data(), out.data(), log_n, a.size() >> log_n));
    return out;
  }
  static std::vector<G1AffinePoint> g1(Gpu& g, int kind, const std::vector<G1AffinePoint>& a, int log_n) { return run(g, bls_g1_fft_batch, kind, a, log_n); }
  static std::vector<G2AffinePoint> g2(Gpu& g, int kind, const std::vector<G2AffinePoint>& a, int log_n) { return run(g, bls_g2_fft_batch, kind, a, log_n); }
  // the Lagrange basis [L_i(tau)] g of the powers-of-tau rows [tau^i] g, i < 2^log_n
  static std::vector<G1AffinePoint> g1_lagrange(Gpu& g, const std::vector<G1AffinePoint>& powers, int log_n) { return g1(g, BLS_IFFT, powers, log_n); }
  static std::vector<G2AffinePoint> g2_lagrange(Gpu& g, const std::vector<G2AffinePoint>& powers, int log_n) { return g2(g, BLS_IFFT, powers, log_n); }
};

struct G1Affine {
  static std::vector<G1PreparedPoint> prepare(const std::vector<G1AffinePoint>& p) { return p; }   // ec.rs:924-935
  // CurveAffine::mul (ec.rs:174-177)
  static std::vector<G1Point> mul(Gpu& g, const std::vector<G1AffinePoint>& p, const std::vector<FrRepr>& k) {
    require_same_length(p.size(), k.size(), "G1Affine::mul");
    std::vector<G1Point> out(p.size());
    g.check(bls_g1_affine_mul_batch(g.ctx(), p.data(), k.data(), out.data(), p.size()));
    return out;
  }
  static std::vector<Fq12> pairing_with(Gpu& g, const std::vector<G1AffinePoint>& p, const std::vector<G2AffinePoint>& q) { return Bls12::pairing(g, p, q); }
};
struct G2Affine {
  static std::vector<G2Point> mul(Gpu& g, const std::vector<G2AffinePoint>& q, const std::vector<FrRepr>& k) {
    require_same_length(q.size(), k.size(), "G2Affine::mul");
    std::vector<G2Point> out(q.size());
    g.check(bls_g2_affine_mul_batch(g.ctx(), q.data(), k.data(), out.data(), q.size()));
    return out;
  }
  // G2Affine::prepare -> G2Prepared::from_affine (mod.rs:168-358)
  static std::vector<G2PreparedPoint> prepare(Gpu& g, const std::vector<G2AffinePoint>& q) {
    std::vector<G2PreparedPoint> out(q.size());
    g.check(bls_g2_prepare_batch(g.ctx(), q.data(), out.data(), q.size()));
    return out;
  }
  static std::vector<Fq12> pairing_with(Gpu& g, const std::vector<G2AffinePoint>& q, const std::vector<G1AffinePoint>& p) { return Bls12::pairing(g, p, q); }
};

// Wnaf (wnaf.rs:75-179): `Wnaf<G1>().scalar(k).base(gpu, g)` and `Wnaf<G1>().base(gpu, g, n).scalar(gpu, k)`
template <class G> class Wnaf {
 public:
  using Proj = typename G::Projective;
  class WithScalars {   // Wnaf<usize, &mut Vec<G>, &[i64]>
   public:
    explicit WithScalars(std::vector<FrRepr> k) : k_(std::move(k)) {}
    std::vector<Proj> base(Gpu& g, const std::vector<Proj>& bases) const { return G::wnaf_mul(g, bases, k_); }
   private:
    std::vector<FrRepr> k_;
  };
  class WithBase {      // Wnaf<usize, &[G], &mut Vec<i64>>: one shared window table
   public:
    WithBase(Proj base, int window) : base_(base), window_(window) {}
    int window_size() const { return window_; }
    std::vector<Proj> scalar(Gpu& g, const std::vector<FrRepr>& k) const {
      std::vector<Proj> out(k.size());
      if constexpr (std::is_same<Proj, G2Point>::value) g.check(bls_g2_wnaf_fixed_base_batch(g.ctx(), &base_, window_, k.data(), out.data(), k.size()));
      else g.check(bls_g1_wnaf_fixed_base_batch(g.ctx(), &base_, window_, k.data(), out.data(), k.size()));
      return out;
    }
    WithBase shared() const { return *this; }
   private:
    Proj base_;
    int window_;
  };
  WithScalars scalar(std::vector<FrRepr> k) const { return WithScalars(std::move(k)); }
  WithBase base(const Proj& b, size_t num_scalars) const { return WithBase(b, G::recommended_wnaf_for_num_scalars(num_scalars)); }
};

// EncodedPoint (lib.rs:236-263).  status[i] == BLS_DEC_OK or the code of the reference's GroupDecodingError.
template <bool IS_G2, bool COMPRESSED> struct Encoded {
  using Aff = typename std::conditional<IS_G2, G2AffinePoint, G1AffinePoint>::type;
  static constexpr size_t size() { return (IS_G2 ? 96 : 48) * (COMPRESSED ? 1 : 2); }
  struct Decoded { std::vector<Aff> points; std::vector<uint8_t> status; };
  static Decoded decode(Gpu& g, const std::vector<uint8_t>& bytes, bool checked) {
    if (bytes.size() % size()) throw Error(BLS_ERR_INVALID_ARGUMENT, "encoded data has the wrong length");
    const size_t n = bytes.size() / size();
    Decoded d{std::vector<Aff>(n), std::vector<uint8_t>(n)};
    if constexpr (IS_G2) g.check(bls_g2_decode_batch(g.ctx(), bytes.data(), COMPRESSED, checked, d.points.data(), d.status.data(), n));
    else g.check(bls_g1_decode_batch(g.ctx(), bytes.data(), COMPRESSED, checked, d.points.data(), d.status.data(), n));
    return d;
  }
  static Decoded into_affine(Gpu& g, const std::vector<uint8_t>& bytes) { return decode(g, bytes, true); }
  static Decoded into_affine_unchecked(Gpu& g, const std::vector<uint8_t>& bytes) { return decode(g, bytes, false); }
  static std::vector<uint8_t> from_affine(Gpu& g, const std::vector<Aff>& a) {
    std::vector<uint8_t> out(a.size() * size());
    if constexpr (IS_G2) g.check(bls_g2_encode_batch(g.ctx(), a.data(), COMPRESSED, out.data(), a.size()));
    else g.check(bls_g1_encode_batch(g.ctx(), a.data(), COMPRESSED, out.data(), a.size()));
    return out;
  }
};
using G1Uncompressed = Encoded<false, false>;
using G1Compressed = Encoded<false, true>;
using G2Uncompressed = Encoded<true, false>;
using G2Compressed = Encoded<true, true>;

}  // namespace pairing_b200
