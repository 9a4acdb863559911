// qipb200.hpp -- header-only C++ host mirror of the reference's operator interface for the
// gate-application path, on top of the C ABI (include/qipb200.h).
//
// The reference is Rust; this image has no Rust toolchain, so the host side above the C ABI
// is C++ (the reference is compiled code).  Names, argument order and error behaviour follow
// the reference so that call sites read the same:
//
//   qip::MatrixOp<P>                       <- enum MatrixOp<P>            (qip-iterators/src/iterators/ops.rs:11-91)
//   qip::make_matrix_op / make_swap_op /   <- qip::state_ops::matrix_ops  (qip/src/state_ops/matrix_ops.rs:12-122)
//        make_control_op / make_sparse_matrix_op
//   qip::apply_op / apply_op_overwrite /   <- qip_iterators::matrix_ops   (qip-iterators/src/matrix_ops.rs:98-219)
//        apply_ops                            (host slices in, host slices out; executed on the B200)
//   qip::B200State<P>                      <- the two Vec<Complex<P>> of LocalBuilder::calculate_state_with_init
//                                             (qip/src/builder.rs:406-407,423-514): amplitudes stay in HBM between gates
//   qip::CircuitError                      <- qip::errors::CircuitError   (qip/src/errors.rs:6-22)
//
// P is float or double (trait Precision, qip/src/types.rs:6-13).
#pragma once

#include <complex>
#include <cstdint>
#include <memory>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "qipb200.h"

namespace qip {

struct CircuitError : std::runtime_error {
  int status;
  explicit CircuitError(const std::string &msg, int status_ = 0) : std::runtime_error(msg), status(status_) {}
};

template <typename P>
struct Prec;
template <>
struct Prec<float> {
  static constexpr qip_prec value = QIP_F32;
};
template <>
struct Prec<double> {
  static constexpr qip_prec value = QIP_F64;
};

// enum MatrixOp<P> { Matrix(indices, data), SparseMatrix(indices, rows), Swap(n, indices), Control(nc, indices, Box<op>) }
template <typename P>
class MatrixOp {
 public:
  typedef std::complex<P> C;
  enum Kind { Matrix = QIP_OP_MATRIX, SparseMatrix = QIP_OP_SPARSE, Swap = QIP_OP_SWAP, Control = QIP_OP_CONTROL };

  static MatrixOp new_matrix(std::vector<uint64_t> indices, std::vector<C> data) {  // ops.rs:49-55
    MatrixOp op(Matrix);
    op.indices_ = std::move(indices);
    op.data_ = std::move(data);
    return op;
  }
  static MatrixOp new_sparse(std::vector<uint64_t> indices, const std::vector<std::vector<std::pair<uint64_t, C>>> &rows) {
    MatrixOp op(SparseMatrix);  // ops.rs:58-64
    op.indices_ = std::move(indices);
    op.rowptr_.push_back(0);
    for (const auto &row : rows) {
      for (const auto &e : row) {
        op.cols_.push_back(e.first);
        op.vals_.push_back(e.second);
      }
      op.rowptr_.push_back(op.cols_.size());
    }
    return op;
  }
  static MatrixOp new_swap(std::vector<uint64_t> a, const std::vector<uint64_t> &b) {  // ops.rs:67-78
    MatrixOp op(Swap);
    op.swap_n_ = a.size();
    a.insert(a.end(), b.begin(), b.end());
    op.indices_ = std::move(a);
    return op;
  }
  static MatrixOp new_control(std::vector<uint64_t> c, const std::vector<uint64_t> &r, MatrixOp inner) {  // ops.rs:81-91
    MatrixOp op(Control);
    op.n_control_ = (uint32_t)c.size();
    c.insert(c.end(), r.begin(), r.end());
    op.indices_ = std::move(c);
    op.inner_ = std::make_shared<MatrixOp>(std::move(inner));
    return op;
  }

  size_t num_indices() const { return kind_ == Swap ? 2 * swap_n_ : indices_.size(); }  // ops.rs:24-36
  const std::vector<uint64_t> &indices() const { return indices_; }                     // ops.rs:39-46
  Kind kind() const { return kind_; }
  uint32_t n_control() const { return n_control_; }
  const MatrixOp *inner() const { return inner_.get(); }

  // Borrowed C view; valid while *this lives and is not modified.
  const qip_op *c_op() const {
    c_.kind = kind_;
    c_.n_indices = (uint32_t)indices_.size();
    c_.n_control = n_control_;
    c_.reserved = 0;
    c_.n_entries = kind_ == Matrix ? data_.size() : (kind_ == SparseMatrix ? rowptr_.size() - 1 : 0);
    c_.indices = indices_.data();
    c_.dense = data_.empty() ? nullptr : data_.data();
    c_.sp_rowptr = rowptr_.empty() ? nullptr : rowptr_.data();
    c_.sp_col = cols_.empty() ? nullptr : cols_.data();
    c_.sp_val = vals_.empty() ? nullptr : vals_.data();
    c_.inner = inner_ ? inner_->c_op() : nullptr;
    return &c_;
  }

 private:
  explicit MatrixOp(Kind k) : kind_(k) {}
  Kind kind_;
  std::vector<uint64_t> indices_;
  std::vector<C> data_;
  std::vector<uint64_t> rowptr_, cols_;
  std::vector<C> vals_;
  size_t swap_n_ = 0;
  uint32_t n_control_ = 0;
  std::shared_ptr<MatrixOp> inner_;
  mutable qip_op c_{};
};

// ---- qip/src/state_ops/matrix_ops.rs:12-122 (validating constructors) ------------------------
template <typename P>
MatrixOp<P> make_matrix_op(std::vector<uint64_t> indices, std::vector<std::complex<P>> dat) {
  const size_t n = indices.size();
  if (n == 0) throw CircuitError("Must supply at least one op index");
  if (dat.size() != (size_t(1) << (2 * n)))
    throw CircuitError("Matrix data has " + std::to_string(dat.size()) + " entries versus expected 2^2*" + std::to_string(n));
  return MatrixOp<P>::new_matrix(std::move(indices), std::move(dat));
}
template <typename P>
MatrixOp<P> make_swap_op(std::vector<uint64_t> a, std::vector<uint64_t> b) {
  if (a.empty() || b.empty()) throw CircuitError("Need at least 1 swap index for a and b");
  if (a.size() != b.size())
    throw CircuitError("Swap must be performed on two sets of indices of equal length, found " +
                       std::to_string(a.size()) + " vs " + std::to_string(b.size()));
  return MatrixOp<P>::new_swap(std::move(a), b);
}
template <typename P>
MatrixOp<P> make_control_op(std::vector<uint64_t> c, MatrixOp<P> op) {
  if (c.empty()) throw CircuitError("Must supply at least one control index");
  if (op.kind() == MatrixOp<P>::Control) {  // nested controls are flattened (:112-115)
    std::vector<uint64_t> rest(op.indices().begin() + op.n_control(), op.indices().end());
    c.insert(c.end(), op.indices().begin(), op.indices().begin() + op.n_control());
    return MatrixOp<P>::new_control(std::move(c), rest, *op.inner());
  }
  std::vector<uint64_t> r = op.indices();
  return MatrixOp<P>::new_control(std::move(c), r, std::move(op));
}

// ---- context -----------------------------------------------------------------------------------
class Context {
 public:
  explicit Context(int device = 0) {
    int st = qipb200_init(&ctx_, device);
    if (st != QIPB200_OK) throw CircuitError(qipb200_last_error(nullptr), st);  // no CPU fallback
  }
  // ONE context over several devices of this process (a power-of-two count): states created on it are sharded
  // over the devices inside the library -- what a single-process host like LocalBuilder needs to use a whole box
  explicit Context(const std::vector<int> &devices) {
    int st = qipb200_init_multi(&ctx_, (int)devices.size(), devices.data());
    if (st != QIPB200_OK) throw CircuitError(qipb200_last_error(nullptr), st);
  }
  ~Context() { qipb200_shutdown(ctx_); }
  Context(const Context &) = delete;
  Context &operator=(const Context &) = delete;
  qipb200_ctx *get() const { return ctx_; }
  void check(int st) const {
    if (st != QIPB200_OK) throw CircuitError(qipb200_last_error(ctx_), st);
  }

 private:
  qipb200_ctx *ctx_ = nullptr;
};

// ---- qip_iterators::matrix_ops drop-ins (host slices) -------------------------------------------
template <typename P>
void apply_op(Context &ctx, size_t n, const MatrixOp<P> &op, const std::vector<std::complex<P>> &input,
              std::vector<std::complex<P>> &output, size_t input_offset, size_t output_offset) {  // matrix_ops.rs:98-123
  ctx.check(qipb200_apply_op(ctx.get(), Prec<P>::value, (uint32_t)n, op.c_op(), input.data(), input.size(),
                             output.data(), output.size(), input_offset, output_offset));
}
template <typename P>
void apply_op_overwrite(Context &ctx, size_t n, const MatrixOp<P> &op, const std::vector<std::complex<P>> &input,
                        std::vector<std::complex<P>> &output, size_t input_offset, size_t output_offset) {  // :127-152
  ctx.check(qipb200_apply_op_overwrite(ctx.get(), Prec<P>::value, (uint32_t)n, op.c_op(), input.data(), input.size(),
                                       output.data(), output.size(), input_offset, output_offset));
}

// ---- device-resident state: the body of LocalBuilder::calculate_state_with_init -------------------
template <typename P>
class B200State {
 public:
  B200State(Context &ctx, size_t n) : ctx_(ctx), n_(n) { ctx_.check(qipb200_state_new(ctx.get(), Prec<P>::value, (uint32_t)n, &st_)); }
  ~B200State() { qipb200_state_free(st_); }
  B200State(const B200State &) = delete;
  B200State &operator=(const B200State &) = delete;

  void set_basis(uint64_t index) { ctx_.check(qipb200_state_set_basis(st_, index)); }  // builder.rs:421
  void apply(const MatrixOp<P> &op) { ctx_.check(qipb200_state_apply_op(st_, op.c_op())); }  // builder.rs:499,514
  void apply_all(const std::vector<MatrixOp<P>> &ops, bool fusion = true) {              // builder.rs:423-514
    std::vector<qip_op> c(ops.size());
    for (size_t i = 0; i < ops.size(); ++i) c[i] = *ops[i].c_op();
    ctx_.check(qipb200_state_apply_schedule(st_, c.data(), c.size(), fusion ? QIPB200_SCHED_DEFAULT : QIPB200_SCHED_NO_FUSION));
  }
  std::vector<std::complex<P>> into_state() {  // builder.rs:518
    std::vector<std::complex<P>> out(size_t(1) << n_);
    ctx_.check(qipb200_state_download(st_, out.data(), 0, out.size()));
    return out;
  }
  double prob_magnitude() {  // measurement_ops.rs:11-13
    double v = 0;
    ctx_.check(qipb200_state_norm2(st_, &v));
    return v;
  }
  uint64_t soft_measure(const std::vector<uint64_t> &indices, double r) {  // measurement_ops.rs:153-176, draw supplied
    uint64_t m = 0;
    ctx_.check(qipb200_state_soft_measure(st_, indices.data(), (uint32_t)indices.size(), r, &m));
    return m;
  }
  // soft_measure for every draw in `draws`, from one read of the state (qipb200_state_sample); the state is unchanged
  std::vector<uint64_t> sample(const std::vector<uint64_t> &indices, const std::vector<double> &draws) {
    std::vector<uint64_t> out(draws.size());
    ctx_.check(qipb200_state_sample(st_, indices.data(), (uint32_t)indices.size(), draws.data(), draws.size(), out.data()));
    return out;
  }
  void collapse(const std::vector<uint64_t> &indices, uint64_t measured, double prob) {  // measure_state, :220-269
    ctx_.check(qipb200_state_collapse(st_, indices.data(), (uint32_t)indices.size(), measured, prob));
  }
  std::vector<double> measure_probs(const std::vector<uint64_t> &indices) {  // measurement_ops.rs:115-127
    std::vector<double> out(size_t(1) << indices.size());
    ctx_.check(qipb200_state_measure_probs(st_, indices.data(), (uint32_t)indices.size(), out.data()));
    return out;
  }
  // a schedule parsed from the QIPS wire format (owned by the library): builder.rs:423-514 on foreign circuits
  void apply_parsed(const qip_op *ops, size_t n_ops, bool fusion = true) {
    ctx_.check(qipb200_state_apply_schedule(st_, ops, n_ops, fusion ? QIPB200_SCHED_DEFAULT : QIPB200_SCHED_NO_FUSION));
  }
  qipb200_state *get() const { return st_; }

 private:
  Context &ctx_;
  size_t n_;
  qipb200_state *st_ = nullptr;
};

// ---- QIPS schedule wire format (SURVEY section 8f, N3): RAII over qipb200_schedule_parse ------------
class ParsedSchedule {
 public:
  ParsedSchedule(const void *bytes, size_t len) {
    char err[256];
    if (qipb200_schedule_parse(bytes, len, &s_, err, sizeof(err)) != QIPB200_OK) throw CircuitError(err);
    ops_ = qipb200_schedule_ops(s_, &n_ops_, &n_qubits_, &prec_);
  }
  ~ParsedSchedule() { qipb200_schedule_free(s_); }
  ParsedSchedule(const ParsedSchedule &) = delete;
  ParsedSchedule &operator=(const ParsedSchedule &) = delete;
  const qip_op *ops() const { return ops_; }
  size_t size() const { return n_ops_; }
  uint32_t n_qubits() const { return n_qubits_; }
  qip_prec prec() const { return prec_; }

 private:
  qipb200_schedule *s_ = nullptr;
  const qip_op *ops_ = nullptr;
  size_t n_ops_ = 0;
  uint32_t n_qubits_ = 0;
  qip_prec prec_ = QIP_F64;
};

}  // namespace qip
