#include "planner.h"

#include <ATen/Context.h>
#include <ATen/Functions.h>
#include <ATen/core/Generator.h>
#include <ATen/cuda/EmptyTensor.h>
#include <c10/core/DeviceGuard.h>
#include <c10/core/impl/LocalDispatchKeySet.h>
#include <c10/cuda/CUDACachingAllocator.h>
#include <c10/cuda/CUDAStream.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <atomic>
#include <condition_variable>
#include <deque>
#include <functional>
#include <mutex>
#include <thread>

#include <unistd.h>

#include <ATen/ThreadLocalState.h>
#include <ATen/detail/CUDAHooksInterface.h>
#include <c10/cuda/CUDAFunctions.h>
#include <cuda_runtime_api.h>
#include <torch/csrc/utils/device_lazy_init.h>

#include "fake_tensor.h"
#include "stack_walk.h"
#include "tape.h"
#include "tdx_init.h"

namespace tdx {

using c10::IValue;
using c10::ScalarType;
using torch::jit::Stack;

namespace {

thread_local MaterializeStats g_stats;

// TDX_PROFILE=1: where the per-tensor host time of a materialize call goes (TSC ticks per phase,
// printed on stderr when the session finishes).  Diagnostics only.
struct Prof {
  static bool on() {
    static const bool v = getenv("TDX_PROFILE") != nullptr;
    return v;
  }
  static uint64_t tick() {
#if defined(__x86_64__)
    return __builtin_ia32_rdtsc();
#else
    return 0;
#endif
  }
  uint64_t acc[12] = {};
  const char* names[12] = {"add:record", "add:materialize_value", "add:finish", "emit:geometry+output", "emit:rng",
                           "emit:descs", "fused:note", "real_of", "process:total", "emit:total", "", ""};
};
thread_local Prof g_prof;
struct ProfScope {
  int k;
  uint64_t t0;
  explicit ProfScope(int k_) : k(k_), t0(Prof::on() ? Prof::tick() : 0) {}
  ~ProfScope() {
    if (Prof::on()) g_prof.acc[k] += Prof::tick() - t0;
  }
};
thread_local double g_pending_traverse_us = 0;  // see add_traverse_time
// Where constant chains are folded.  ATen's CPU and CUDA kernels differ in the last bit for 16-bit
// dtypes (the CPU kernels round a Python scalar to the tensor dtype first, the CUDA kernels keep it
// in fp32), and a tensor recorded for CUDA must hold what the program computes on CUDA: so while
// materialising onto a CUDA device the 1-element stand-in lives there.  (plan_info, which may run
// on a machine without a GPU, folds on the CPU.)
thread_local c10::Device g_fold_device = c10::Device(c10::kCPU);
thread_local std::vector<TdxInitDesc> g_last_descs;  // what the last materialize call launched

// Never record / fake anything we do while materialising.
struct NoInterception {
  c10::impl::ExcludeDispatchKeyGuard a{c10::DispatchKey::DeferredInit};
  c10::impl::ExcludeDispatchKeyGuard b{c10::DispatchKey::Fake};
};

// ---------------------------------------------------------------------------------------------
// symbolic state of a storage: what its elements are, as a function of the element index
// ---------------------------------------------------------------------------------------------
// A storage is a list of disjoint SEGMENTS [begin, end) (element indices of the storage, in the
// dtype it currently holds), each with one simple content description.  A tensor initialised as a
// whole is one segment; `weight.normal_(); weight[padding_idx].zero_()` (nn.Embedding, BERT, Gemma,
// OPT, Phi-3) is three; an in-place op through a contiguous view splits the segments it crosses.
struct Sym {
  // Iota: element i = p0 + (i - origin) * p1 (integers): `arange`, and -- with epilogue steps -- the
  // index programs built on it (rotary inv_freq: arange -> float -> / dim -> base ** x -> 1/x -> * s)
  enum Src { Uninit, Const, Uniform, Normal, Iota } src = Uninit;
  at::Tensor cval;                           // Const: a 1-element tensor of the state's dtype (built lazily)
  c10::Scalar cscalar;                       // Const: the value, while no folding has needed a tensor
  bool has_scalar = false;
  double p0 = 0, p1 = 1;                     // Uniform: from,to   Normal: mean,std   Iota: start,step
  uint32_t rng_op = kNoValue;                // the live RNG op
  c10::SmallVector<TdxEpiStep, TDX_MAX_EPI> epi;
  // The RNG source ran on an fp32 tensor that was later cast to a 16-bit dtype: keep the fp32
  // stream and arithmetic (TDX_ALGO_WIDE32) so that the result IS `fp32_tensor.to(dtype)`.
  bool wide = false;
  bool src_noround = false;  // the generated value feeds fp32 epilogue steps before the cast
  // `wide` exists to keep the 16-bit tensor equal to `fp32_source.to(dtype)` when BOTH get
  // materialised.  If nothing can ever ask for the fp32 source (`module.to(torch.bfloat16)` rebinds
  // every parameter to its cast and drops the fp32 tensor), the equality is unobservable and the
  // tensor takes the native 16-bit stream -- same distribution, the fast kernel (wide_observable()).
  uint32_t wide_src_storage = kNoValue;  // the storage the RNG op wrote (and the cast read), if that simple
  uint32_t wide_cast_op = kNoValue;
  bool rng() const { return src == Uniform || src == Normal; }
};

struct Seg {
  int64_t begin = 0, end = 0;
  // Storage index of element 0 of the tensor the segment's source op ran on: an RNG op on a view
  // numbers its elements from the view's first element (global Philox index = index - origin).
  int64_t origin = 0;
  Sym st;
};

struct RngPass {
  uint32_t op;     // tape op
  int64_t numel;   // of the tensor it ran on: what it consumes of the generator's offset
  uint32_t slot;   // Tape::rng entry of the op
};

size_t find_arg(const TapeOp& op, const char* name);

// The Tape::rng entry of an RNG op (made on first sight).
uint32_t rng_slot_of(Tape& tape, uint32_t op_idx) {
  TapeOp& op = tape.ops[op_idx];
  if (op.rng_slot == kNoValue) {
    RngSlot s;
    s.op = op_idx;
    if (op.handle) {
      const size_t pos = find_arg(op, "generator");
      s.explicit_generator = pos != static_cast<size_t>(-1) && pos < op.args.size() && op.args[pos].isGenerator();
    }
    op.rng_slot = static_cast<uint32_t>(tape.rng.size());
    tape.rng.push_back(s);
  }
  return op.rng_slot;
}

// (inline storage: a recording holds one State per storage, and every heap block of a recording is
// one somebody has to free when it dies)
using SegList = c10::SmallVector<Seg, 1>;
using RngChain = c10::SmallVector<RngPass, 2>;

struct State {
  bool opaque = true;
  ScalarType dtype = ScalarType::Undefined;  // dtype of the tensor currently holding the state
  SegList segs;        // sorted, disjoint, covering [0, numel)
  RngChain rng_chain;  // every RNG pass met, live or dead, chronological
};

State make_opaque() { return State{}; }

// Element bits of `v` converted to `dtype` (the conversion at::full performs), without building a
// tensor.  Returns false for dtypes that are not handled here.
bool scalar_bits(const c10::Scalar& v, ScalarType dtype, unsigned char* out, size_t* isz) {
  auto put = [&](auto x) { std::memcpy(out, &x, sizeof(x)); *isz = sizeof(x); return true; };
  switch (dtype) {
    case ScalarType::Float: return put(v.to<float>());
    case ScalarType::Double: return put(v.to<double>());
    case ScalarType::BFloat16: return put(v.to<c10::BFloat16>());
    case ScalarType::Half: return put(v.to<c10::Half>());
    case ScalarType::Long: return put(v.to<int64_t>());
    case ScalarType::Int: return put(v.to<int32_t>());
    case ScalarType::Short: return put(v.to<int16_t>());
    case ScalarType::Char: return put(v.to<int8_t>());
    case ScalarType::Byte: return put(v.to<uint8_t>());
    case ScalarType::Bool: return put(v.to<bool>());
    default: return false;
  }
}

// The value `v` holds once it has been stored in a tensor of `dtype` (what `full(v, dtype=...)` /
// `fill_` keep of it: ATen converts with Scalar::to<scalar_t>()), as a Scalar again.  Lets a dtype
// cast of a constant be folded on the host, exactly: full(v, A).to(B) == B(A(v)).  false: a dtype
// or a value (out-of-range float -> integer) this does not model.
bool stored_value(const c10::Scalar& v, ScalarType dtype, c10::Scalar& out) {
  try {
    switch (dtype) {
      case ScalarType::Float: out = static_cast<double>(v.to<float>()); return true;
      case ScalarType::Double: out = v.to<double>(); return true;
      case ScalarType::BFloat16: out = static_cast<double>(static_cast<float>(v.to<c10::BFloat16>())); return true;
      case ScalarType::Half: out = static_cast<double>(static_cast<float>(v.to<c10::Half>())); return true;
      case ScalarType::Long: out = v.to<int64_t>(); return true;
      case ScalarType::Int: out = static_cast<int64_t>(v.to<int32_t>()); return true;
      case ScalarType::Short: out = static_cast<int64_t>(v.to<int16_t>()); return true;
      case ScalarType::Char: out = static_cast<int64_t>(v.to<int8_t>()); return true;
      case ScalarType::Byte: out = static_cast<int64_t>(v.to<uint8_t>()); return true;
      case ScalarType::Bool: out = v.to<bool>(); return true;
      default: return false;
    }
  } catch (...) {
    return false;
  }
}

// While a tape is analysed at the end of its recording (analyze_tape) the target device is not
// known yet, and a constant chain must be folded with the target device's arithmetic: such
// storages are evaluated when they are materialised instead.  The same holds for programs that
// read a real tensor's value (it may be mutated before the materialisation: the version check
// must see that).
thread_local bool g_analysis_only = false;
thread_local bool g_analysis_deferred = false;  // the last evaluation met one of those

// The 1-element tensor form of a constant state (needed to fold further ops through ATen).
void ensure_cval(Sym& st, ScalarType dtype) {
  if (st.cval.defined() || !st.has_scalar) return;
  c10::impl::ExcludeDispatchKeyGuard a{c10::DispatchKey::DeferredInit};
  c10::impl::ExcludeDispatchKeyGuard b{c10::DispatchKey::Fake};
  st.cval = at::full({1}, st.cscalar, at::TensorOptions().dtype(dtype).device(g_fold_device));
}

bool is_fused_float(ScalarType t) {
  return t == ScalarType::Float || t == ScalarType::BFloat16 || t == ScalarType::Half;
}

// Value of argument `pos` of a recorded op as a double, if it is a number or a real 1-element
// tensor (the form Python scalars take in mul_.Tensor / add_.Tensor).
std::optional<double> scalar_arg(const TapeOp& op, size_t pos) {
  if (pos >= op.args.size()) return std::nullopt;
  const IValue& v = op.args[pos];
  if (v.isDouble()) return v.toDouble();
  if (v.isInt()) return static_cast<double>(v.toInt());
  if (v.isBool()) return v.toBool() ? 1.0 : 0.0;
  if (v.isTensor()) {
    size_t slot = 0;  // which tensor slot of the frame is this argument?
    for (size_t i = 0; i < pos; ++i) {
      if (op.args[i].isTensor()) ++slot;
      else if (op.args[i].isList())
        for (const IValue& e : op.args[i].toListRef()) slot += e.isTensor();
    }
    if (slot >= op.inputs.size()) return std::nullopt;
    const at::Tensor& t = op.inputs[slot].real;
    if (!t.defined() || t.numel() != 1 || !t.is_cpu() || t.is_complex()) return std::nullopt;
    // A Python number the argument parser wrapped into a 0-dim tensor is nobody else's to mutate:
    // its value can be read when the tape is analysed.  Any other real tensor is read when the
    // storage is materialised (it may change until then: the version check must see that).
    if (g_analysis_only && !t.unsafeGetTensorImpl()->is_wrapped_number()) {
      g_analysis_deferred = true;
      return std::nullopt;
    }
    if (!t.is_inference() && static_cast<int64_t>(t._version()) != op.inputs[slot].real_version)
      return std::nullopt;  // mutated since recording: let generic replay raise the error
    return t.item<double>();
  }
  return std::nullopt;
}

// ATen casts uniform_'s bounds to the tensor dtype before use
// ($TORCH/include/ATen/native/cuda/DistributionTemplates.h uniform_kernel, and the CPU twin).
double round_to_dtype(double x, ScalarType t) {
  switch (t) {
    case ScalarType::Float: return static_cast<double>(static_cast<float>(x));
    case ScalarType::BFloat16: return static_cast<double>(static_cast<float>(c10::BFloat16(static_cast<float>(x))));
    case ScalarType::Half: return static_cast<double>(static_cast<float>(c10::Half(static_cast<float>(x))));
    default: return x;
  }
}

size_t find_arg(const TapeOp& op, const char* name) {
  const auto& args = op.handle->schema().arguments();
  for (size_t i = 0; i < args.size(); ++i)
    if (args[i].name() == name) return i;
  return static_cast<size_t>(-1);
}

// Runs the recorded operator on `self` (a 1-element tensor standing for a constant segment), with
// the recorded scalar arguments: exact ATen semantics for constant folding.  `dtype` is the
// segment's dtype before the op; on success it is the result's.
bool fold_const(const TapeOp& op, Sym& st, ScalarType& dtype, bool inplace) {
  if (g_analysis_only) {
    g_analysis_deferred = true;
    return false;
  }
  ensure_cval(st, dtype);
  st.has_scalar = false;
  if (!op.handle || !st.cval.defined()) return false;
  if (inplace) {
    // Segments are split by copying (`w[i].zero_()` makes three of one): their constants are handles
    // to ONE 1-element tensor until somebody writes.  An in-place op replayed on a shared constant
    // would reach every segment that holds it (`full(c); w[i].zero_(); w.add_(1)` added 1 twice to
    // the two outer segments; `w[a:b].mul_(2)` doubled the whole tensor): write to a private copy.
    NoInterception guard;
    st.cval = st.cval.clone();
  }
  Stack stack;
  size_t slot = 0;
  bool ok = true, first_tensor = true;
  for (const IValue& a : op.args) {
    if (a.isTensor()) {
      if (slot >= op.inputs.size()) return false;
      const InputRef& in = op.inputs[slot++];
      if (first_tensor) {
        if (st.cval.device() != g_fold_device) {
          NoInterception guard;
          st.cval = st.cval.to(g_fold_device);
        }
        stack.emplace_back(st.cval);
        first_tensor = false;
      } else if (in.real.defined() && in.real.numel() == 1 && in.real.is_cpu()) {
        stack.emplace_back(in.real);
      } else if (!in.real.defined() && in.value == kNoValue && !in.foreign) {
        stack.emplace_back(at::Tensor());
      } else {
        ok = false;
      }
    } else if (a.isList()) {
      for (const IValue& e : a.toListRef()) ok &= !e.isTensor();
      stack.push_back(a);
    } else if (a.isDevice()) {
      stack.emplace_back(g_fold_device);
    } else {
      stack.push_back(a);
    }
  }
  if (!ok) return false;
  NoInterception guard;
  op.handle->callBoxed(stack);
  if (stack.empty() || !stack.back().isTensor()) return false;
  at::Tensor out = stack.back().toTensor();
  if (out.numel() != 1) return false;
  st.cval = inplace ? st.cval : out;
  dtype = st.cval.scalar_type();
  return true;
}

// ---- segment bookkeeping ------------------------------------------------------------------------
// The elements of the storage a value names, if they are one contiguous run.
bool range_of(const ValueInfo& v, int64_t& begin, int64_t& end) {
  int64_t expect = 1;
  for (int64_t d = static_cast<int64_t>(v.sizes.size()) - 1; d >= 0; --d) {
    if (v.sizes[d] == 1) continue;
    if (v.strides[d] != expect) return false;
    expect *= v.sizes[d];
  }
  begin = v.storage_offset;
  end = v.storage_offset + v.numel;
  return true;
}

// Cuts the segments at `at` so that none straddles it.
void split_at(SegList& segs, int64_t at) {
  for (size_t i = 0; i < segs.size(); ++i) {
    if (segs[i].begin < at && at < segs[i].end) {
      Seg right = segs[i];
      right.begin = at;
      segs[i].end = at;
      segs.insert(segs.begin() + static_cast<std::ptrdiff_t>(i) + 1, std::move(right));
      return;
    }
  }
}

// [b, e) now holds `st` (an op that overwrites what was there).
void overwrite(State& s, int64_t b, int64_t e, Sym st, int64_t origin) {
  if (b >= e) return;
  split_at(s.segs, b);
  split_at(s.segs, e);
  SegList out;
  out.reserve(s.segs.size() + 1);
  bool placed = false;
  for (Seg& g : s.segs) {
    if (g.begin >= b && g.end <= e) {
      if (!placed) {
        Seg n;
        n.begin = b;
        n.end = e;
        n.origin = origin;
        n.st = std::move(st);
        out.push_back(std::move(n));
        placed = true;
      }
      continue;
    }
    out.push_back(std::move(g));
  }
  s.segs = std::move(out);
}

State eval_storage(Tape& tape, uint32_t S, uint32_t upto);

// Applies one recorded op whose output lives on the storage being evaluated.
void transition(Tape& tape, uint32_t op_idx, uint32_t S, State& st) {
  TapeOp& op = tape.ops[op_idx];
  // the output of this op on S
  uint32_t out_v = kNoValue;
  for (uint32_t v : op.outputs)
    if (v != kNoValue && tape.values[v].storage == S) out_v = v;
  const ValueInfo& out = tape.values[out_v];
  auto push_epi = [&](Sym& sy, uint32_t code, double a, double b = 0) {
    if (sy.epi.size() >= TDX_MAX_EPI) return false;
    TdxEpiStep s;
    s.op = code;  // every step rounds to the tensor dtype, like the in-place ATen op it stands for
    s.a = static_cast<float>(a);
    s.b = static_cast<float>(b);
    sy.epi.push_back(s);
    return true;
  };
  auto fresh = [&](Sym sy) {  // a factory: one segment over the whole (new) storage
    RngChain chain = std::move(st.rng_chain);
    st = State{};
    st.opaque = false;
    st.dtype = out.dtype;
    st.rng_chain = std::move(chain);
    Seg g;
    g.begin = 0;
    g.end = out.numel;
    g.st = std::move(sy);
    st.segs.push_back(std::move(g));
  };

  switch (op.kind) {
    case OpKind::Empty:
      if (!out.covers_storage) { st = make_opaque(); return; }
      st.rng_chain.clear();
      fresh(Sym{});
      return;
    case OpKind::Zeros:
    case OpKind::Ones:
    case OpKind::Full: {
      if (!out.covers_storage) { st = make_opaque(); return; }
      Sym sy;
      sy.src = Sym::Const;
      sy.has_scalar = true;
      if (op.kind == OpKind::Zeros) sy.cscalar = 0;
      else if (op.kind == OpKind::Ones) sy.cscalar = 1;
      else {
        const size_t pos = find_arg(op, "fill_value");
        if (pos == static_cast<size_t>(-1) || !op.args[pos].isScalar()) { st = make_opaque(); return; }
        sy.cscalar = op.args[pos].toScalar();
      }
      st.rng_chain.clear();
      fresh(std::move(sy));
      return;
    }
    case OpKind::Randn:
    case OpKind::Rand: {
      if (!out.covers_storage || !is_fused_float(out.dtype)) { st = make_opaque(); return; }
      Sym sy;
      sy.src = op.kind == OpKind::Randn ? Sym::Normal : Sym::Uniform;
      sy.p0 = 0.0;
      sy.p1 = 1.0;
      sy.rng_op = op_idx;
      st.rng_chain.clear();
      fresh(std::move(sy));
      st.rng_chain.push_back(RngPass{op_idx, out.numel, rng_slot_of(tape, op_idx)});
      return;
    }
    case OpKind::Arange: {
      // arange([start,] end[, step]) with integer start / step: exact in int64, and in fp32 as long as
      // every value stays below 2^24 (then no question of how the kernel rounds start + i * step)
      if (!out.covers_storage || !(out.dtype == ScalarType::Long || out.dtype == ScalarType::Float)) {
        st = make_opaque();
        return;
      }
      const size_t ps = find_arg(op, "start"), pt = find_arg(op, "step");
      const auto start = ps == static_cast<size_t>(-1) ? std::optional<double>(0.0) : scalar_arg(op, ps);
      const auto step = pt == static_cast<size_t>(-1) ? std::optional<double>(1.0) : scalar_arg(op, pt);
      const double kExact = out.dtype == ScalarType::Float ? 16777216.0 : 9007199254740992.0;
      if (!start || !step || *start != std::floor(*start) || *step != std::floor(*step) ||
          std::fabs(*start) + std::fabs(*step) * static_cast<double>(out.numel) >= kExact) {
        st = make_opaque();
        return;
      }
      Sym sy;
      sy.src = Sym::Iota;
      sy.p0 = *start;
      sy.p1 = *step;
      st.rng_chain.clear();
      fresh(std::move(sy));
      return;
    }
    case OpKind::Alias:
    case OpKind::View:
    case OpKind::HookVariableData:
    case OpKind::HookSetData:  // `p.data = t`: p now names t's storage; its elements are t's
      return;  // same elements under another tensor object
    default:
      break;
  }

  // ---- dst.copy_(src): the range `out` names becomes src's elements ------------------------------
  if (op.kind == OpKind::CopyInplace) {
    int64_t b = 0, e = 0;
    if (st.opaque || out.dtype != st.dtype || !range_of(out, b, e) || st.segs.empty() || b < 0 ||
        e > st.segs.back().end || op.inputs.size() < 2 || op.inputs[1].value == kNoValue) {
      st = make_opaque();
      return;
    }
    const ValueInfo& in = tape.values[op.inputs[1].value];
    int64_t sb = 0, se = 0;
    if (in.numel != out.numel || in.dtype != out.dtype || in.storage == S || !range_of(in, sb, se) ||
        in.sizes != out.sizes) {  // (no broadcasting, no dtype conversion)
      st = make_opaque();
      return;
    }
    State src = eval_storage(tape, in.storage, op_idx);
    if (src.opaque || src.dtype != in.dtype || src.segs.empty() || sb < 0 || se > src.segs.back().end) {
      st = make_opaque();
      return;
    }
    for (Seg& g : src.segs) {
      const int64_t gb = std::max(g.begin, sb), ge = std::min(g.end, se);
      if (gb >= ge) continue;
      overwrite(st, b + (gb - sb), b + (ge - sb), g.st, g.origin - sb + b);
    }
    for (const RngPass& r : src.rng_chain) {  // the source's passes must have their streams when dst is built
      bool have = false;
      for (const RngPass& q : st.rng_chain) have |= q.op == r.op;
      if (!have) st.rng_chain.push_back(r);
    }
    return;
  }

  // ---- in-place writers through `out` (the whole tensor or a contiguous view of part of it) ----
  const bool inplace = op.kind == OpKind::UniformInplace || op.kind == OpKind::NormalInplace ||
                       op.kind == OpKind::FillInplace || op.kind == OpKind::ZeroInplace ||
                       op.kind == OpKind::MulInplace || op.kind == OpKind::AddInplace ||
                       op.kind == OpKind::ErfinvInplace || op.kind == OpKind::ClampInplace ||
                       op.kind == OpKind::SubInplace || op.kind == OpKind::NegInplace || op.kind == OpKind::DivInplace;
  if (inplace) {
    int64_t b = 0, e = 0;
    if (st.opaque || out.dtype != st.dtype || !range_of(out, b, e) || st.segs.empty() ||
        b < 0 || e > st.segs.back().end) {
      st = make_opaque();
      return;
    }
    if (op.kind == OpKind::UniformInplace || op.kind == OpKind::NormalInplace) {
      if (!is_fused_float(out.dtype)) { st = make_opaque(); return; }
      const bool uni = op.kind == OpKind::UniformInplace;
      const auto a = scalar_arg(op, 1), c = scalar_arg(op, 2);
      if (!a || !c) { st = make_opaque(); return; }
      Sym sy;
      sy.src = uni ? Sym::Uniform : Sym::Normal;
      if (uni) {
        TORCH_CHECK(*a <= *c, "uniform_ expects to return a [from, to) range, but found from=", fmt_double(*a),
                    " > to=", fmt_double(*c));
        sy.p0 = round_to_dtype(*a, out.dtype);
        sy.p1 = round_to_dtype(*c, out.dtype);
      } else {
        TORCH_CHECK(*c >= 0.0, "normal expects std >= 0.0, but found std ", fmt_double(*c));
        sy.p0 = *a;
        sy.p1 = *c;
      }
      sy.rng_op = op_idx;
      overwrite(st, b, e, std::move(sy), b);
      st.rng_chain.push_back(RngPass{op_idx, out.numel, rng_slot_of(tape, op_idx)});
      return;
    }
    if (op.kind == OpKind::FillInplace || op.kind == OpKind::ZeroInplace) {
      Sym sy;
      sy.src = Sym::Const;
      if (op.kind == OpKind::ZeroInplace) {
        sy.cscalar = 0;
        sy.has_scalar = true;
      } else if (op.args.size() > 1 && op.args[1].isScalar()) {
        sy.cscalar = op.args[1].toScalar();
        sy.has_scalar = true;
      } else if (op.inputs.size() > 1 && op.inputs[1].real.defined() &&
                 op.inputs[1].real.numel() == 1 && op.inputs[1].real.is_cpu()) {
        if (g_analysis_only) {
          g_analysis_deferred = true;
          st = make_opaque();
          return;
        }
        NoInterception guard;
        sy.cval = op.inputs[1].real.detach().to(out.dtype).reshape({1}).clone();
      } else {
        st = make_opaque();
        return;
      }
      overwrite(st, b, e, std::move(sy), b);
      return;
    }
    // elementwise: applies to every segment inside [b, e)
    split_at(st.segs, b);
    split_at(st.segs, e);
    for (Seg& g : st.segs) {
      if (g.begin < b || g.end > e) continue;
      Sym& sy = g.st;
      if (sy.src == Sym::Uninit) { st = make_opaque(); return; }
      if (sy.src == Sym::Const) {
        ScalarType dt = st.dtype;
        if (!fold_const(op, sy, dt, /*inplace=*/true) || dt != st.dtype) { st = make_opaque(); return; }
        continue;
      }
      if (sy.src == Sym::Iota && st.dtype != ScalarType::Float) { st = make_opaque(); return; }
      bool ok = true;
      if (op.kind == OpKind::MulInplace) {
        const auto c = scalar_arg(op, 1);
        ok = c && push_epi(sy, TDX_EPI_MUL, *c);
      } else if (op.kind == OpKind::AddInplace) {
        const auto c = scalar_arg(op, 1), alpha = scalar_arg(op, 2);
        ok = c && alpha && push_epi(sy, TDX_EPI_ADD, *c * *alpha);
      } else if (op.kind == OpKind::SubInplace) {
        // x - alpha * c is computed by ATen as x + (-alpha) * c (sub is add with the sign of alpha flipped)
        const auto c = scalar_arg(op, 1), alpha = scalar_arg(op, 2);
        ok = c && alpha && push_epi(sy, TDX_EPI_ADD, -(*c * *alpha));
      } else if (op.kind == OpKind::NegInplace) {
        ok = push_epi(sy, TDX_EPI_MUL, -1.0);
      } else if (op.kind == OpKind::DivInplace) {
        // fp32 only, like DivOut below: ATen's CUDA kernel multiplies by the fp32 reciprocal of the divisor
        const auto c = scalar_arg(op, 1);
        ok = c && st.dtype == ScalarType::Float && *c != 0.0 &&
             push_epi(sy, TDX_EPI_MUL, static_cast<double>(1.0f / static_cast<float>(*c)));
      } else if (op.kind == OpKind::ErfinvInplace) {
        ok = push_epi(sy, TDX_EPI_ERFINV, 0);
      } else {  // clamp_(min, max), either may be None
        const bool has_min = !op.args[1].isNone(), has_max = !op.args[2].isNone();
        const auto lo = scalar_arg(op, 1), hi = scalar_arg(op, 2);
        ok = !((has_min && !lo) || (has_max && !hi)) &&
             push_epi(sy, TDX_EPI_CLAMP, has_min ? *lo : -std::numeric_limits<double>::infinity(),
                      has_max ? *hi : std::numeric_limits<double>::infinity());
      }
      if (!ok) { st = make_opaque(); return; }
    }
    return;
  }

  // ---- out-of-place unary ops: a new storage whose state derives from the argument's -------------
  if (op.kind == OpKind::MulOut || op.kind == OpKind::AddOut || op.kind == OpKind::CloneOut ||
      op.kind == OpKind::CastOut || op.kind == OpKind::DivOut || op.kind == OpKind::PowScalarOut ||
      op.kind == OpKind::ReciprocalOut || op.kind == OpKind::SubOut || op.kind == OpKind::NegOut) {
    if (op.inputs.empty() || op.inputs[0].value == kNoValue || !out.covers_storage) { st = make_opaque(); return; }
    const ValueInfo& in = tape.values[op.inputs[0].value];
    int64_t b = 0, e = 0;
    if (in.numel != out.numel || in.storage == S || !range_of(in, b, e)) { st = make_opaque(); return; }
    State src = eval_storage(tape, in.storage, op_idx);
    if (src.opaque || src.dtype != in.dtype || src.segs.empty() || b < 0 || e > src.segs.back().end) {
      st = make_opaque();
      return;
    }
    // restrict to the argument's elements and renumber from 0
    st = State{};
    st.opaque = false;
    st.dtype = src.dtype;
    st.rng_chain = std::move(src.rng_chain);
    for (Seg& g : src.segs) {
      const int64_t gb = std::max(g.begin, b), ge = std::min(g.end, e);
      if (gb >= ge) continue;
      Seg n = std::move(g);
      n.begin = gb - b;
      n.end = ge - b;
      n.origin -= b;
      st.segs.push_back(std::move(n));
    }
    if (op.kind == OpKind::CloneOut) {
      // a copy: same elements (an RNG segment keeps its op, hence its Philox stream: the clone is
      // bit-identical to its source, as deepcopy semantics require)
      if (out.dtype != st.dtype) st = make_opaque();
      return;
    }
    ScalarType new_dtype = st.dtype;
    for (Seg& g : st.segs) {
      Sym& sy = g.st;
      if (sy.src == Sym::Uninit) {
        if (op.kind != OpKind::CastOut) { st = make_opaque(); return; }
        new_dtype = out.dtype;
        continue;
      }
      if (sy.src == Sym::Const) {
        if (op.kind == OpKind::CastOut && sy.has_scalar && !sy.cval.defined()) {
          // a dtype cast of a plain constant (`ones(n).to(bf16)`, every norm weight of a model
          // converted with Module.to): exact on the host, no 1-element tensor, no device round trip
          c10::Scalar kept, probe;
          if (stored_value(sy.cscalar, st.dtype, kept) && stored_value(kept, out.dtype, probe)) {
            sy.cscalar = kept;
            new_dtype = out.dtype;
            continue;
          }
        }
        ScalarType dt = st.dtype;
        if (!fold_const(op, sy, dt, /*inplace=*/false) || dt != out.dtype) { st = make_opaque(); return; }
        new_dtype = out.dtype;
        continue;
      }
      if (sy.src == Sym::Iota) {
        // index programs: everything after the arange runs in fp32 (the kernel's epilogue)
        if (op.kind == OpKind::CastOut) {
          if (out.dtype == st.dtype) continue;
          if (st.dtype == ScalarType::Float && (out.dtype == ScalarType::BFloat16 || out.dtype == ScalarType::Half)) {
            // `inv_freq.to(torch.bfloat16)` (Module.to(dtype) converts floating buffers too): the fp32
            // program, rounded once at the store.  Terminal: nothing folds onto a 16-bit index program
            // (every later elementwise transition asks for fp32).
            new_dtype = out.dtype;
            continue;
          }
          if (!(st.dtype == ScalarType::Long && out.dtype == ScalarType::Float && sy.epi.empty()) ||
              std::fabs(sy.p0) + std::fabs(sy.p1) * static_cast<double>(out.numel) >= 16777216.0) {
            st = make_opaque();
            return;
          }
          new_dtype = out.dtype;  // int64 -> fp32 of values below 2^24: exact
          continue;
        }
        if (out.dtype != ScalarType::Float ||
            !(st.dtype == ScalarType::Float || (st.dtype == ScalarType::Long && op.kind == OpKind::DivOut && sy.epi.empty())) ||
            std::fabs(sy.p0) + std::fabs(sy.p1) * static_cast<double>(out.numel) >= 16777216.0) {
          st = make_opaque();
          return;
        }
        new_dtype = out.dtype;  // (an int64 arange divided by a number is promoted to fp32 first, like ATen does)
      }
      if (op.kind == OpKind::DivOut || op.kind == OpKind::PowScalarOut || op.kind == OpKind::ReciprocalOut) {
        // fp32 only, with the arithmetic of ATen's CUDA kernels: `t / c` multiplies by the fp32
        // reciprocal of c (BinaryDivTrueKernel.cu), `c ** t` is powf(c, t) (PowKernel.cu), reciprocal
        // is 1.0f / t
        if (out.dtype != ScalarType::Float || (sy.src != Sym::Iota && st.dtype != ScalarType::Float)) {
          st = make_opaque();
          return;
        }
        bool ok = false;
        if (op.kind == OpKind::DivOut) {
          const auto c = scalar_arg(op, 1);
          const size_t pm = find_arg(op, "rounding_mode");
          ok = c && pm == static_cast<size_t>(-1) &&
               push_epi(sy, TDX_EPI_MUL, static_cast<double>(1.0f / static_cast<float>(*c)));
        } else if (op.kind == OpKind::PowScalarOut) {
          const auto base = scalar_arg(op, 0);
          ok = base && *base != 1.0 && push_epi(sy, TDX_EPI_RPOW, *base);
        } else {
          ok = push_epi(sy, TDX_EPI_RECIP, 0);
        }
        if (!ok) { st = make_opaque(); return; }
        continue;
      }
      if (sy.src == Sym::Iota && (op.kind == OpKind::MulOut || op.kind == OpKind::AddOut)) {
        bool ok;
        if (op.kind == OpKind::MulOut) {
          const auto c = scalar_arg(op, 1);
          ok = c && push_epi(sy, TDX_EPI_MUL, *c);
        } else {
          const auto c = scalar_arg(op, 1), alpha = scalar_arg(op, 2);
          ok = c && alpha && push_epi(sy, TDX_EPI_ADD, *c * *alpha);
        }
        if (!ok) { st = make_opaque(); return; }
        continue;
      }
      // RNG source followed by an elementwise op
      if (op.kind == OpKind::CastOut) {
        if (out.dtype == st.dtype) continue;  // a copy
        // fp32 -> bf16/fp16: the values must be exactly `source.to(dtype)` (the fp32 source may be
        // materialised too, e.g. `m.to(torch.bfloat16)` keeps both alive while recording), so the
        // descriptor keeps the fp32 stream/arithmetic and rounds once, at this point of the chain
        if (st.dtype != ScalarType::Float || !(out.dtype == ScalarType::BFloat16 || out.dtype == ScalarType::Half) ||
            sy.wide) {
          st = make_opaque();
          return;
        }
        sy.wide = true;
        {
          bool direct = false;  // did the RNG op write the very storage this cast reads?
          for (uint32_t ov : tape.ops[sy.rng_op].outputs)
            direct |= ov != kNoValue && tape.values[ov].storage == in.storage;
          if (direct) {
            sy.wide_src_storage = in.storage;
            sy.wide_cast_op = op_idx;
          }
        }
        // everything before the cast ran in fp32; the cast itself is the rounding of the last
        // pre-cast step (or of the generated value, if there was none)
        sy.src_noround = !sy.epi.empty();
        for (size_t i = 0; i + 1 < sy.epi.size(); ++i) sy.epi[i].op |= TDX_EPI_NOROUND;
        new_dtype = out.dtype;
        continue;
      }
      if (out.dtype != st.dtype) { st = make_opaque(); return; }  // type promotion: not modelled
      bool ok;
      if (op.kind == OpKind::MulOut) {
        const auto c = scalar_arg(op, 1);
        ok = c && push_epi(sy, TDX_EPI_MUL, *c);
      } else if (op.kind == OpKind::NegOut) {
        ok = push_epi(sy, TDX_EPI_MUL, -1.0);
      } else if (op.kind == OpKind::SubOut) {
        const auto c = scalar_arg(op, 1), alpha = scalar_arg(op, 2);
        ok = c && alpha && push_epi(sy, TDX_EPI_ADD, -(*c * *alpha));
      } else if (op.kind == OpKind::AddOut) {
        const auto c = scalar_arg(op, 1), alpha = scalar_arg(op, 2);
        ok = c && alpha && push_epi(sy, TDX_EPI_ADD, *c * *alpha);
      } else {
        ok = false;  // (every kind admitted above is handled before this point)
      }
      if (!ok) { st = make_opaque(); return; }
    }
    if (new_dtype != out.dtype) { st = make_opaque(); return; }
    st.dtype = new_dtype;
    return;
  }
  st = make_opaque();
}

// Can anything still observe the fp32 tensor a `wide` segment was cast from?  Not if no fake tensor
// names its storage any more, nothing of it has been materialised, and the only ops that ever
// touched it are its own writers and the cast.
bool wide_observable(const Tape& tape, const Sym& sy) {
  if (!sy.wide) return false;
  if (sy.wide_src_storage == kNoValue) return true;
  const StorageInfo& a = tape.storages[sy.wide_src_storage];
  if (a.live > 0 || a.fused_done || a.replayed) return true;
  for (uint32_t oi : a.touching_ops) {
    if (oi == sy.wide_cast_op) continue;
    const TapeOp& op = tape.ops[oi];
    if (op.kind == OpKind::HookSetData) continue;  // `p.data = cast`: names the old storage, never reads it
    bool writes = false;
    for (uint32_t v : op.outputs) writes |= v != kNoValue && tape.values[v].storage == sy.wide_src_storage;
    bool produces = false;  // (metadata queries such as _has_compatible_shallow_copy_type yield no tensor)
    for (uint32_t v : op.outputs) produces |= v != kNoValue;
    if (!writes && produces) return true;  // another reader whose result could be asked for
  }
  return false;
}

bool is_pure_alias(OpKind k) {
  return k == OpKind::Alias || k == OpKind::View || k == OpKind::HookVariableData || k == OpKind::HookSetData;
}

// A reader of an intermediate state does not pin its argument to generic replay if nobody will ever
// have to RUN it: every tensor it produced has a final state the planner can derive symbolically
// (e.g. `original = buf.clone()` followed by `buf.copy_(...)`, `original.copy_(...)`: HF's rotary
// embeddings).  Deriving such a state evaluates the argument as of the reader, never its final state.
thread_local int g_reader_depth = 0;
bool reader_resolves_symbolically(Tape& tape, const TapeOp& op) {
  if (g_reader_depth >= 4) return false;
  struct Depth {
    Depth() { ++g_reader_depth; }
    ~Depth() { --g_reader_depth; }
  } depth;
  for (uint32_t v : op.outputs) {
    if (v == kNoValue) continue;
    const ValueInfo& ov = tape.values[v];
    if (ov.real.defined() || tape.storages[ov.storage].replayed) return false;
    if (eval_storage(tape, ov.storage, static_cast<uint32_t>(tape.ops.size())).opaque) return false;
  }
  return true;
}

// State of storage S after every recorded op with index < upto.
State eval_storage(Tape& tape, uint32_t S, uint32_t upto) {
  const StorageInfo& si = tape.storages[S];
  State st;
  bool any = false;
  // index of the last op (< upto) that changes the CONTENT of S (aliases only re-describe it)
  uint32_t last_writer = kNoValue;
  for (uint32_t oi : si.touching_ops) {
    if (oi >= upto) break;
    const TapeOp& op = tape.ops[oi];
    if (is_pure_alias(op.kind)) continue;
    for (uint32_t v : op.outputs)
      if (v != kNoValue && tape.values[v].storage == S) last_writer = oi;
  }
  for (uint32_t oi : si.touching_ops) {
    if (oi >= upto) break;
    const TapeOp& op = tape.ops[oi];
    bool writes = false;
    for (uint32_t v : op.outputs) writes |= (v != kNoValue && tape.values[v].storage == S);
    if (!writes) {
      // A reader that saw an intermediate state which a later op overwrote must run at its own
      // point in history: only generic replay can do that.  (`p.data = t` names p's old storage
      // as an argument but never reads it.)
      if (op.kind != OpKind::HookSetData && !op.done && last_writer != kNoValue && oi < last_writer &&
          !reader_resolves_symbolically(tape, op))
        return make_opaque();
      continue;
    }
    if (op.done && op.kind == OpKind::Generic) return make_opaque();
    any = true;
    transition(tape, oi, S, st);
    if (st.opaque) return st;
  }
  if (!any) return make_opaque();
  return st;
}

}  // namespace

// What analyze_tape leaves on a storage: the symbolic state, and -- for the states the kernels can
// run -- the same thing laid out for the materialise call, which then touches this block, the
// value's geometry and two RNG slots per tensor and nothing else of the recording (the recording is
// cold in the caches by the time a model is materialised: every line touched is ~100 ns).
struct FastSeg {
  int64_t begin = 0, end = 0, origin = 0;
  uint32_t rng_slot = kNoValue;  // kNoValue: no RNG pass (a constant or an index program)
  bool indexed = false;          // the descriptor's elem_begin matters (RNG and iota sources)
  bool wide = false;
  const Sym* sym = nullptr;      // (into StorageTemplate::st) for the rare questions: wide_observable
  TdxInitDesc proto;             // everything but dst / elem_begin / elem_count / seed / offset
};
struct StorageTemplate {
  State st;
  bool fast = false;
  uint8_t isz = 0;
  int64_t numel = 0;
  c10::SmallVector<FastSeg, 1> segs;  // Uninit segments are left out
};

namespace {

// ---------------------------------------------------------------------------------------------
// batched fused execution
// ---------------------------------------------------------------------------------------------
double now_us();
thread_local double g_call_begin_us = 0;

// Memory of the fused outputs.  A call's tensors are carved out of ONE allocation per submission
// (a "slab"): one trip to the caching allocator -- and, on a cold allocator, one cudaMalloc instead
// of one per tensor (226 of them for Llama-3-8B: ~0.6 s) -- while every tensor still gets a
// StorageImpl of its own (no aliasing is visible through storage identity, `torch.save` writes
// them separately, `untyped_storage().resize_()` works).  The slab goes back to the allocator
// when the last tensor carved from it dies.  TDX_SLAB=0: one allocation per tensor instead
// (memory is then released tensor by tensor).
struct Slab {
  c10::DataPtr block;
};
void slab_ref_delete(void* ctx) { delete static_cast<std::shared_ptr<Slab>*>(ctx); }

bool slab_enabled() {
  static const bool v = [] {
    const char* e = getenv("TDX_SLAB");
    return !(e && e[0] == '0');
  }();
  return v;
}

std::atomic<uint64_t> g_epoch{1};  // process-wide: storages remember the epoch across sessions

struct Batch {
  c10::Device device = c10::Device(c10::kCPU);
  std::vector<TdxInitDesc> descs;
  // Outputs whose memory is assigned at the next submission: the tensor object exists as soon as
  // its program has been planned (the caller can give it its Python identity meanwhile), its
  // storage gets its address when the slab is allocated.
  struct Pending {
    c10::intrusive_ptr<c10::StorageImpl> storage;
    size_t nbytes = 0;
    uint32_t first_desc = 0, n_desc = 0;  // descriptors whose dst is relative to this tensor's base
  };
  std::vector<Pending> pending;
  // Early submission: the first descriptors are launched as soon as a modest amount of work has
  // accumulated, so the GPU starts writing while the host is still planning the rest of the
  // module; the threshold grows after every submission so that the launch count (each launch
  // has a ~10-20 us tail) stays logarithmic.
  int64_t pending_bytes = 0;
  uint64_t epoch = g_epoch.fetch_add(1);  // bumped by every submission: a storage whose fused_epoch == epoch is not on the GPU yet
  int64_t flush_threshold = flush_start();
  static int64_t flush_start() {
    static const int64_t v = [] {
      const char* e = getenv("TDX_FLUSH_BYTES");  // 0 = submit once, at the end
      // measured on Llama-3-8B (profiles/r1_e2e_submission_sweep.txt): 1 GiB start beats 128 MiB and
      // 4 GiB on one GPU; 256 MiB keeps the first launch early when a rank only owns 1/8 of the model
      return e ? static_cast<int64_t>(strtoll(e, nullptr, 10)) : (int64_t{256} << 20);
    }();
    return v;
  }
  // (Submission points depend on bytes only, never on timing: a call then cuts the same slabs every
  // time, which is what lets the caching allocator serve them from its free lists.  A gate on the
  // estimated GPU backlog -- submit only when the GPU is about to run dry -- saved one launch per
  // call at N = 1 and cost a cudaMalloc, i.e. a device synchronisation, whenever the cut moved.)
  // When the call materialises a whole recording the total is known in advance (Tape::fused_bytes,
  // divided by the world size of a sharded call), and so is how fast the host plans relative to the
  // GPU: planning costs ~1.5 us per tensor whatever its size, the kernels write ~4.8 GB/ms.  After
  // the first (256 MiB) submission the rest is cut into at most three more whose sizes grow by the
  // ratio q of the two rates, clamped to [1, 4]: with big tensors (one GPU, q = 4) the GPU is the
  // bottleneck and every chunk hides the planning of the next, larger one -- three launches for
  // 16 GB; when a rank owns an eighth of the model the host is as slow as the GPU (q = 1), the call
  // ends one chunk's GPU time after the last tensor has been planned, and equal chunks make that
  // the smallest.  A function of byte counts only, like the fallback rule (x4 per submission) that
  // applies when there is no estimate or the call outgrows it.
  int64_t expected_total = 0, expected_tensors = 0, submitted_bytes = 0;
  c10::SmallVector<int64_t, 4> schedule;  // thresholds of the submissions after the first
  size_t schedule_pos = 0;
  int64_t last_threshold = 0;
  void expect(int64_t total_bytes, int64_t tensors) {
    if (expected_total == 0 && submitted_bytes == 0) {
      expected_total = total_bytes;
      expected_tensors = tensors;
    }
  }
  int64_t next_threshold() {
    constexpr int64_t kNever = int64_t{1} << 62;
    const int64_t fallback = std::min<int64_t>(last_threshold * 4, int64_t{64} << 30);
    if (expected_total <= 0) return fallback;
    if (submitted_bytes >= expected_total) {  // more than the recording promised (several recordings in one call)
      expected_total = 0;
      return fallback;
    }
    if (schedule.empty()) {
      const double rest = static_cast<double>(expected_total - submitted_bytes);
      const double per_tensor = static_cast<double>(expected_total) / static_cast<double>(std::max<int64_t>(expected_tensors, 1));
      const double q = std::min(4.0, std::max(1.0, per_tensor / 7.2e6));
      int m = 1;
      double sum = q, term = q;
      while (m < 3 && static_cast<double>(submitted_bytes) * sum < rest) {
        ++m;
        term *= q;
        sum += term;
      }
      term = q;
      for (int i = 0; i + 1 < m; ++i) {  // the last chunk is whatever is left when the call ends
        schedule.push_back(std::max<int64_t>(static_cast<int64_t>(rest * term / sum), int64_t{64} << 20));
        term *= q;
      }
      schedule.push_back(kNever);
    }
    const int64_t t = schedule[std::min(schedule_pos, schedule.size() - 1)];
    ++schedule_pos;
    return t;
  }
  void note(int64_t bytes) {
    pending_bytes += bytes;
    if (flush_threshold > 0 && pending_bytes >= flush_threshold) {
      submitted_bytes += pending_bytes;
      if (flush_threshold < (int64_t{1} << 60)) last_threshold = flush_threshold;
      flush();
      flush_threshold = next_threshold();
    }
  }
  void assign_memory();
  void flush();
};

double now_us() {
  return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// An output tensor without memory yet (see Batch::Pending).  Built like at::detail::empty_generic
// does, minus the allocation.
at::Tensor make_output(c10::IntArrayRef sizes, ScalarType dtype, c10::Device dev, size_t nbytes,
                       c10::intrusive_ptr<c10::StorageImpl>& storage_out) {
  c10::Allocator* alloc = c10::cuda::CUDACachingAllocator::get();
  storage_out = c10::make_intrusive<c10::StorageImpl>(c10::StorageImpl::use_byte_size_t(),
                                                      static_cast<int64_t>(nbytes),
                                                      c10::DataPtr(nullptr, dev), alloc, /*resizable=*/true);
  at::Tensor t = at::detail::make_tensor<c10::TensorImpl>(
      c10::Storage(storage_out), c10::DispatchKeySet(c10::DispatchKey::CUDA), c10::scalarTypeToTypeMeta(dtype));
  t.unsafeGetTensorImpl()->generic_set_sizes_contiguous(sizes);
  return t;
}

void Batch::assign_memory() {
  if (pending.empty()) return;
  const double t0 = now_us();
  c10::Allocator* alloc = c10::cuda::CUDACachingAllocator::get();
  constexpr size_t kAlign = 256;  // vector stores need 16; 256 keeps every tensor on its own L2 lines
  if (slab_enabled() && pending.size() > 1) {
    // Slabs hold at most kSlabBytes (a tensor larger than that gets one of its own) and their sizes
    // are rounded to 1/32 of a power of two (<= 3 % over): where a call cuts its submissions depends on
    // timing, and slabs of arbitrary sizes would miss the caching allocator's free lists from one
    // call to the next (a miss is a cudaMalloc -- milliseconds, and a device synchronisation).
    constexpr size_t kSlabBytes = size_t{1} << 30;
    auto rounded = [](size_t n) {
      if (n <= (size_t{2} << 20)) return (n + 511) & ~size_t{511};
      size_t p2 = size_t{1} << 21;
      while (p2 < n) p2 <<= 1;
      const size_t step = p2 >> 5;
      return (n + step - 1) / step * step;
    };
    size_t i = 0;
    while (i < pending.size()) {
      size_t j = i, total = 0;
      while (j < pending.size()) {
        const size_t sz = (pending[j].nbytes + kAlign - 1) & ~(kAlign - 1);
        if (j > i && total + sz > kSlabBytes) break;
        total += sz;
        ++j;
      }
      if (total) {
        auto slab = std::make_shared<Slab>();
        slab->block = alloc->allocate(rounded(total));
        char* base = static_cast<char*>(slab->block.get());
        size_t off = 0;
        for (size_t k = i; k < j; ++k) {
          Pending& p = pending[k];
          if (p.nbytes == 0) continue;
          char* ptr = base + off;
          off += (p.nbytes + kAlign - 1) & ~(kAlign - 1);
          p.storage->set_data_ptr_noswap(
              c10::DataPtr(ptr, new std::shared_ptr<Slab>(slab), &slab_ref_delete, device));
          for (uint32_t q = p.first_desc; q < p.first_desc + p.n_desc; ++q)
            descs[q].dst = ptr + reinterpret_cast<uintptr_t>(descs[q].dst);
        }
      }
      i = j;
    }
  } else {
    for (Pending& p : pending) {
      if (p.nbytes == 0) continue;
      c10::DataPtr d = alloc->allocate(p.nbytes);
      char* ptr = static_cast<char*>(d.get());
      p.storage->set_data_ptr_noswap(std::move(d));
      for (uint32_t k = p.first_desc; k < p.first_desc + p.n_desc; ++k)
        descs[k].dst = ptr + reinterpret_cast<uintptr_t>(descs[k].dst);
    }
  }
  pending.clear();
  g_stats.alloc_us += now_us() - t0;
}

// TDX_TRACE=1: every submission's host time, bytes and GPU start / end (CUDA events, read back when
// the session finishes).
struct SubmissionTrace {
  double host_us = 0, bytes = 0;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
};
thread_local std::vector<SubmissionTrace> g_sub_trace;
thread_local cudaEvent_t g_trace_origin = nullptr;
bool trace_on() {  // TDX_TRACE=2: + the GPU timeline of the submissions (synchronises at the end of the call)
  static const bool v = getenv("TDX_TRACE") != nullptr && getenv("TDX_TRACE")[0] == '2';
  return v;
}

void Batch::flush() {
  NoInterception guard;
  c10::DeviceGuard dg(device.is_cuda() ? device : c10::Device(c10::kCPU));
  assign_memory();
  if (descs.empty()) {
    epoch = g_epoch.fetch_add(1);
    pending_bytes = 0;
    return;
  }
  const double t0 = now_us();
  const int n = static_cast<int>(descs.size());
  // prepare: the plan is laid out on the host and says how much workspace it needs (descriptor table
  // + prefix sums + work lists: tens of KB, not the upper bound of tdx_init_workspace_bytes)
  size_t ws_bytes = 0;
  int rc = tdx_init_prepare(descs.data(), n, &ws_bytes);
  TORCH_CHECK(rc == 0, "libtdx_init: plan failed (", rc, "): ", tdx_last_error());
  // (straight from the caching allocator: freed at the end of this scope, reused in stream order)
  at::Tensor ws = at::detail::empty_cuda({static_cast<int64_t>(std::max<size_t>(ws_bytes, 16))}, at::kByte,
                                         device, std::nullopt);
  auto stream = c10::cuda::getCurrentCUDAStream(device.index());
  SubmissionTrace tr;
  if (trace_on()) {
    if (!g_trace_origin) {
      cudaEventCreate(&g_trace_origin);
      cudaEventRecord(g_trace_origin, stream.stream());
    }
    cudaEventCreate(&tr.e0);
    cudaEventCreate(&tr.e1);
    cudaEventRecord(tr.e0, stream.stream());
  }
  rc = tdx_init_submit(ws.data_ptr(), ws_bytes, stream.stream());
  TORCH_CHECK(rc == 0, "libtdx_init: launch failed (", rc, "): ", tdx_last_error());
  if (trace_on()) {
    cudaEventRecord(tr.e1, stream.stream());
    tr.host_us = now_us() - g_call_begin_us;
    tr.bytes = static_cast<double>(pending_bytes);
    g_sub_trace.push_back(tr);
  }
  g_stats.kernel_launches += tdx_last_launch_count();
  g_stats.descriptors += n;
  g_stats.submissions++;
  g_stats.upload_bytes += static_cast<int64_t>(tdx_last_upload_bytes());
  if (g_stats.first_submit_us == 0) g_stats.first_submit_us = now_us() - g_call_begin_us;
  g_stats.last_submit_us = now_us() - g_call_begin_us;
  g_last_descs.insert(g_last_descs.end(), descs.begin(), descs.end());
  descs.clear();
  pending_bytes = 0;
  epoch = g_epoch.fetch_add(1);
  g_stats.launch_us += now_us() - t0;
}

int tdx_dtype_of(ScalarType t) {
  switch (t) {
    case ScalarType::Float: return TDX_F32;
    case ScalarType::BFloat16: return TDX_BF16;
    case ScalarType::Half: return TDX_F16;
    default: return -1;
  }
}

// Generator state is read once per materialize call and written back once (a CUDA generator's
// set_offset() asks the driver whether the stream is capturing: ~1 us, twice per tensor).
struct GenCache {
  struct Entry {
    at::Generator gen;
    uint64_t seed = 0, offset = 0;
    bool dirty = false;
  };
  std::vector<Entry> entries;
  // the default generator of a device, looked up once per materialize call (the global context's
  // accessor takes a lock and re-validates the device on every call)
  std::vector<std::pair<c10::Device, at::Generator>> defaults;
  const at::Generator& default_generator(c10::Device device) {
    for (const auto& d : defaults)
      if (d.first == device) return d.second;
    defaults.emplace_back(device, at::globalContext().defaultGenerator(device));
    return defaults.back().second;
  }
  Entry& get(const at::Generator& g) {
    for (auto& e : entries)
      if (e.gen.unsafeGetGeneratorImpl() == g.unsafeGetGeneratorImpl()) return e;
    Entry e;
    e.gen = g;
    std::lock_guard<std::mutex> lock(e.gen.mutex());
    e.seed = g.current_seed();
    e.offset = g.get_offset();
    entries.push_back(std::move(e));
    return entries.back();
  }
  // must run before anything else (ATen replay, the user) looks at the generators
  void write_back() {
    for (auto& e : entries) {
      if (!e.dirty) continue;
      std::lock_guard<std::mutex> lock(e.gen.mutex());
      e.gen.set_offset(e.offset);
      e.dirty = false;
    }
    entries.clear();
  }
};

// Gives an RNG op its Philox stream id (once) and advances the generator, so that replaying in
// the same order with the same seed reproduces the same tensors, dead passes included.
void assign_rng(Tape& tape, RngSlot& slot, int64_t numel, c10::Device device, GenCache& cache) {
  if (slot.assigned) return;
  at::Generator gen;
  if (slot.explicit_generator) {
    const TapeOp& op = tape.ops[slot.op];
    const size_t pos = find_arg(op, "generator");
    if (pos != static_cast<size_t>(-1) && op.args[pos].isGenerator()) gen = op.args[pos].toGenerator();
  }
  if (!gen.defined()) gen = cache.default_generator(device);
  TORCH_CHECK(gen.device().type() == device.type(), "Expected a '", device.type(),
              "' device type for generator but found '", gen.device().type(), "'");
  GenCache::Entry& e = cache.get(gen);
  slot.seed = e.seed;
  slot.offset = e.offset;
  // consumption is a function of the GLOBAL element count only: shard-invariant by construction
  const uint64_t blocks = (static_cast<uint64_t>(numel) + 3) / 4;
  e.offset += ((blocks + 3) / 4) * 4 + 4;
  e.dirty = true;
  slot.assigned = true;
}

struct ShardGeom {
  int64_t begin = 0, count = 0;
  c10::SmallVector<int64_t, 4> sizes;
};

ShardGeom shard_of(const ValueInfo& v, const std::optional<ShardSpec>& shard) {
  ShardGeom g;
  g.sizes = v.sizes;
  g.begin = 0;
  g.count = v.numel;
  if (!shard || shard->world <= 1 || v.sizes.empty()) return g;  // 0-dim tensors are replicated
  const int64_t d0 = v.sizes[0];
  const int64_t inner = d0 ? v.numel / d0 : 0;
  const int64_t per = (d0 + shard->world - 1) / shard->world;  // torch.chunk row count
  const int64_t start = std::min(d0, shard->rank * per);
  const int64_t len = std::min(per, d0 - start);
  g.begin = start * inner;
  g.count = len * inner;
  g.sizes[0] = len;
  return g;
}

at::Tensor alias_of(const at::Tensor& base, const ValueInfo& v, bool first) {
  const bool same = base.sizes() == c10::IntArrayRef(v.sizes) &&
                    base.strides() == c10::IntArrayRef(v.strides) &&
                    base.storage_offset() == v.storage_offset;
  if (same && first) return base;  // the common case: the parameter IS the backing tensor
  NoInterception guard;
  at::Tensor t = base.detach();
  if (!same) t.as_strided_(v.sizes, v.strides, v.storage_offset);
  return t;
}

// Lays a state out for emission (StorageTemplate's fast form).  false: some segment is not
// expressible as a descriptor.  `may_sync`: a constant that only exists as a (device) tensor may be
// read back (the materialise path; never the analysis at the end of the recording).
bool build_fast(const Tape& tape, const StorageInfo& si, StorageTemplate& t, bool may_sync) {
  (void)tape;
  t.fast = false;
  t.segs.clear();
  const State& st = t.st;
  if (st.opaque) return false;
  const size_t isz = c10::elementSize(st.dtype);
  if (isz == 0 || si.nbytes % isz) return false;
  const int64_t numel = static_cast<int64_t>(si.nbytes / isz);
  if (numel == 0 || st.segs.empty() || st.segs.back().end != numel) return false;
  for (const Seg& sg : st.segs) {
    const Sym& sy = sg.st;
    if (sy.src == Sym::Uninit) continue;
    FastSeg f;
    f.begin = sg.begin;
    f.end = sg.end;
    f.origin = sg.origin;
    f.sym = &sy;
    TdxInitDesc& d = f.proto;
    std::memset(&d, 0, sizeof(d));
    if (sy.src == Sym::Const) {
      if (!(isz == 1 || isz == 2 || isz == 4 || isz == 8)) return false;
      d.src = TDX_SRC_CONST;
      d.dtype = isz == 1 ? TDX_RAW8 : isz == 2 ? TDX_RAW16 : isz == 4 ? TDX_RAW32 : TDX_RAW64;
      unsigned char pat[16], one[16];
      size_t got = 0;
      if (!(sy.has_scalar && scalar_bits(sy.cscalar, st.dtype, one, &got) && got == isz)) {
        if (!may_sync) return false;
        Sym tmp = sy;
        ensure_cval(tmp, st.dtype);
        if (!tmp.cval.defined()) return false;
        NoInterception guard;
        std::memcpy(one, tmp.cval.cpu().contiguous().data_ptr(), isz);
      }
      for (size_t i = 0; i < 16; i += isz) std::memcpy(pat + i, one, isz);
      std::memcpy(d.fill_bits, pat, 16);
    } else if (sy.src == Sym::Iota) {
      if (!(tdx_dtype_of(st.dtype) >= 0 || (st.dtype == ScalarType::Long && sy.epi.empty()))) return false;
      d.src = TDX_SRC_IOTA;
      d.dtype = st.dtype == ScalarType::Long ? TDX_I64 : static_cast<uint8_t>(tdx_dtype_of(st.dtype));
      d.p0 = sy.p0;
      d.p1 = sy.p1;
      d.n_epi = static_cast<uint8_t>(sy.epi.size());
      for (size_t i = 0; i < sy.epi.size(); ++i) d.epi[i] = sy.epi[i];
      f.indexed = true;
    } else {
      if (tdx_dtype_of(st.dtype) < 0) return false;
      f.indexed = true;
      d.src = sy.src == Sym::Uniform ? TDX_SRC_UNIFORM : TDX_SRC_NORMAL;
      d.dtype = static_cast<uint8_t>(tdx_dtype_of(st.dtype));
      d.p0 = sy.p0;
      d.p1 = sy.p1;
      d.n_epi = static_cast<uint8_t>(sy.epi.size());
      for (size_t i = 0; i < sy.epi.size(); ++i) d.epi[i] = sy.epi[i];
      if (sy.src_noround) d.reserved |= TDX_FLAG_SRC_NOROUND;
      f.wide = sy.wide;
      f.rng_slot = kNoValue;
      for (const RngPass& r : st.rng_chain)
        if (r.op == sy.rng_op) f.rng_slot = r.slot;
      if (f.rng_slot == kNoValue) return false;
    }
    t.segs.push_back(std::move(f));
  }
  t.isz = static_cast<uint8_t>(isz);
  t.numel = numel;
  t.fast = true;
  return true;
}

// ---------------------------------------------------------------------------------------------
// generic replay
// ---------------------------------------------------------------------------------------------
struct Engine {
  MaterializeOptions opts;
  Batch& batch;
  GenCache gens;

  bool sharding(const ValueInfo& vi) const { return opts.shard && opts.shard->world > 1 && !vi.sizes.empty(); }

  at::Tensor real_of(Tape& tape, uint32_t v) {
    ValueInfo& vi = tape.values[v];
    StorageInfo& si = tape.storages[vi.storage];
    if (vi.real.defined() && !(si.fused_done && si.base_is_shard && !sharding(vi))) return vi.real;
    TORCH_INTERNAL_ASSERT(si.fused_done, "value of `", tape.ops[vi.op].name(),
                          "` requested before it was materialised");
    if (si.base_is_shard) {
      if (sharding(vi)) {
        // the backing tensor is this rank's dim-0 chunk; only whole-storage tensors can name it
        TORCH_CHECK(vi.covers_storage,
                    "sharded materialisation only supports tensors that cover their whole storage");
        vi.real = si.base_taken ? [&] { NoInterception guard; return si.base.detach(); }() : si.base;
        si.base_taken = true;
        return vi.real;
      }
      // A reader (a buffer computed from a parameter, say) needs the unsharded tensor of a storage
      // whose backing tensor is one rank's chunk: every element is a function of (seed, offset,
      // index), so the full tensor is generated beside the chunk -- same bits, no communication.
      if (!si.full_base.defined()) {
        int64_t bytes = 0;
        TORCH_INTERNAL_ASSERT(emit_fused(tape, vi.storage, vi, std::nullopt, si.full_base, bytes),
                              "a fused storage stopped being fusible");
        si.fused_epoch = batch.epoch;
      }
      return alias_of(si.full_base, vi, false);  // (not cached in vi.real: that names this rank's view)
    }
    vi.real = alias_of(si.base, vi, !si.base_taken);
    si.base_taken = true;
    return vi.real;
  }

  c10::Device target_device(c10::Device recorded) {
    c10::Device d = opts.device ? *opts.device : recorded;
    if (d.is_cuda() && !d.has_index()) {  // "cuda" = the current device, asked for once per call
      if (current_cuda < 0) current_cuda = c10::cuda::current_device();
      d = c10::Device(c10::kCUDA, current_cuda);
    }
    return d;
  }
  c10::DeviceIndex current_cuda = -1;

  void collect_storage(Tape& tape, uint32_t S, uint32_t upto, std::vector<uint8_t>& mark,
                       std::vector<uint32_t>& visited_upto) {
    if (visited_upto[S] >= upto) return;
    visited_upto[S] = upto;
    if (tape.storages[S].fused_done) return;  // its content comes from the kernels (real_of): nothing to replay
    const auto& touching = tape.storages[S].touching_ops;
    uint32_t last_writer = kNoValue;
    for (uint32_t oi : touching) {
      if (oi >= upto) break;
      for (uint32_t v : tape.ops[oi].outputs)
        if (v != kNoValue && tape.values[v].storage == S) last_writer = oi;
    }
    if (last_writer == kNoValue) return;
    for (size_t k = 0; k < touching.size(); ++k) {
      const uint32_t oi = tape.storages[S].touching_ops[k];
      if (oi > last_writer) break;
      collect_op(tape, oi, mark, visited_upto);
    }
  }

  void collect_op(Tape& tape, uint32_t oi, std::vector<uint8_t>& mark,
                  std::vector<uint32_t>& visited_upto) {
    if (mark[oi] || tape.ops[oi].done) return;
    mark[oi] = 1;
    for (size_t k = 0; k < tape.ops[oi].inputs.size(); ++k) {
      const uint32_t v = tape.ops[oi].inputs[k].value;
      if (v == kNoValue) continue;
      if (tape.values[v].real.defined()) {
        // Built already -- by the op that produced it.  In-place writers recorded on its storage after
        // that op and before this reader may still be waiting: `b = a.clone(); b[2:5].normal_();
        // c = b * 2` with `a` materialised first replays the clone as part of a's history (it reads
        // a), and `b * 2` then found b "real" and never ran the normal_.  Collect what is left of
        // the storage's history up to this op (ops that ran are skipped: TapeOp::done).
        collect_storage(tape, tape.values[v].storage, oi, mark, visited_upto);
        continue;
      }
      // A dependency whose whole program folds is built by the kernels (unsharded: the op reads all
      // of it), not replayed op by op: faster, and its values do not depend on whether it or its
      // reader was asked for first.  (A storage the reader saw in an intermediate state is opaque
      // to the planner -- eval_storage's reader rule -- and is replayed up to `oi` as before.)
      if (!tape.storages[tape.values[v].storage].fused_done) {
        const std::optional<ShardSpec> saved = opts.shard;
        opts.shard = std::nullopt;
        const bool fused = try_fused(tape, v);
        opts.shard = saved;
        if (fused) continue;
      }
      collect_storage(tape, tape.values[v].storage, oi, mark, visited_upto);
    }
  }

  void replay(Tape& tape, uint32_t oi) {
    TapeOp& op = tape.ops[oi];
    if (op.done) return;
    const size_t nargs = op.args.size();
    Stack stack;
    stack.reserve(nargs);
    for (const IValue& a : op.args) {
      if (a.isList()) {  // fresh list: we are about to put tensors into it
        const auto& src = a.toList();
        c10::impl::GenericList l(src.elementType());
        for (const IValue& e : a.toListRef()) l.push_back(e);
        stack.emplace_back(std::move(l));
      } else {
        stack.push_back(a);
      }
    }
    size_t slot = 0;
    for_each_tensor_mut(stack, nargs, [&](at::Tensor& t) {
      InputRef& in = op.inputs[slot++];
      if (in.value != kNoValue) {
        t = real_of(tape, in.value);
        // a fused result that is still sitting in the batch must reach the stream before ATen reads it
        const StorageInfo& isi = tape.storages[tape.values[in.value].storage];
        if (isi.fused_done && isi.fused_epoch == batch.epoch) batch.flush();
      } else if (in.foreign) {
        // (recorded by an earlier deferred_init: same rule -- its descriptor may still be in the batch)
        // It is needed NOW, as an argument: the session's "replay RNG-free programs after the last
        // submission" rule is for tensors the caller asked for, and would hand back nothing here
        // (`b = deferred_init(lambda: a * 2 + 1)` with `a = deferred_init(torch.ones, ...)` raised
        // "Expected a proper Tensor but got None" unless `a` had been materialised first).
        struct NoDeferral {
          bool& flag;
          const bool saved;
          explicit NoDeferral(bool& f) : flag(f), saved(f) { flag = false; }
          ~NoDeferral() { flag = saved; }
        } now(defer_generic);
        t = materialize_value(in.foreign, in.foreign_value);
        const StorageInfo& fsi = in.foreign->storages[in.foreign->values[in.foreign_value].storage];
        if (fsi.fused_done && fsi.fused_epoch == batch.epoch) batch.flush();
      } else if (in.real.defined()) {
        TORCH_CHECK(!in.real.is_inference(), "A `Tensor` argument required for the materialization of `",
                    op.name(), "` was created in inference mode. Materialization cannot be performed "
                    "because in-place updates to inference tensors cannot be tracked.");
        TORCH_CHECK(static_cast<int64_t>(in.real._version()) == in.real_version,
                    "A `Tensor` argument required for the materialization of `", op.name(),
                    "` was updated in-place. Materialization cannot be performed.");
        t = in.real;
        if (opts.device && t.dim() != 0 && t.device() != *opts.device) t = t.to(*opts.device);
      }
    });
    if (opts.device && op.handle) {
      const int di = device_argument_index(*op.handle);
      if (di >= 0 && (stack[di].isDevice() || stack[di].isNone())) stack[di] = *opts.device;
    }
    {
      at::ThreadLocalStateGuard tls(*op.tls);  // (a shared snapshot: see tape.cc)
      NoInterception guard;
      if (op.handle) {
        op.handle->callBoxed(stack);
      } else if (op.kind == OpKind::HookVariableData) {
        at::Tensor self = stack[0].toTensor();
        stack.clear();
        stack.emplace_back(at::Tensor(self.variable_data()));
      } else {  // HookSetData
        at::Tensor self = stack[0].toTensor(), data = stack[1].toTensor();
        self.set_data(data);
        stack.clear();
        stack.emplace_back(self);
      }
    }
    size_t k = 0;
    for_each_tensor(stack, op.num_returns, [&](const at::Tensor& t) {
      if (k < op.outputs.size() && op.outputs[k] != kNoValue) {
        ValueInfo& ov = tape.values[op.outputs[k]];
        ov.real = t;
        tape.storages[ov.storage].replayed = true;  // its content now comes from ATen: never fuse it later
      }
      ++k;
    });
    op.results = std::move(stack);
    op.done = true;
    op.tls.reset();  // (args stay: a later analysis of the tape still reads their scalars)
    g_stats.generic_ops++;
  }

  // Builds the descriptors of storage S (or of one rank's dim-0 chunk of it) and the tensor they
  // write; `vi` is the value whose geometry the tensor takes (the parameter itself, normally).
  // Returns false if the program is not fusible.  `bytes_out`: algorithmic bytes of the descriptors.
  bool emit_fused(Tape& tape, uint32_t S, const ValueInfo& vi, const std::optional<ShardSpec>& shard,
                  at::Tensor& base_out, int64_t& bytes_out, Prebuilt* pre = nullptr) {
    const StorageInfo& si = tape.storages[S];
    const c10::Device dev = target_device(vi.device);
    if (si.tmpl && si.tmpl->fast) {  // analysed when the recording ended: nothing to evaluate
      g_stats.template_hits++;
      return emit_from(tape, *si.tmpl, vi, shard, dev, base_out, bytes_out, pre);
    }
    if (si.tmpl && si.tmpl->st.opaque) return false;
    StorageTemplate tmp;
    if (si.tmpl) {
      tmp.st = si.tmpl->st;  // (a constant whose bits need a tensor: rare)
    } else {
      struct FoldOn {  // constants fold with the target device's arithmetic
        c10::Device prev = g_fold_device;
        explicit FoldOn(c10::Device d) { g_fold_device = d; }
        ~FoldOn() { g_fold_device = prev; }
      } fold_on(dev);
      c10::DeviceGuard fold_guard(dev);
      const double t_eval = now_us();
      tmp.st = eval_storage(tape, S, static_cast<uint32_t>(tape.ops.size()));
      g_stats.eval_us += now_us() - t_eval;
    }
    if (!build_fast(tape, si, tmp, /*may_sync=*/true)) return false;
    return emit_from(tape, tmp, vi, shard, dev, base_out, bytes_out);
  }

  bool emit_from(Tape& tape, const StorageTemplate& t, const ValueInfo& vi, const std::optional<ShardSpec>& shard,
                 c10::Device dev, at::Tensor& base_out, int64_t& bytes_out, Prebuilt* pre = nullptr) {
    ProfScope p_total(9);
    const State& st = t.st;
    const size_t isz = t.isz;
    // geometry of what this rank writes
    const uint64_t pt0 = Prof::on() ? Prof::tick() : 0;
    ShardGeom g;
    if (vi.covers_storage && vi.dtype == st.dtype) {
      g = shard_of(vi, shard);
    } else {
      g.begin = 0;
      g.count = t.numel;
      g.sizes.assign(1, t.numel);
    }
    if (batch.device != dev) {
      batch.flush();
      batch.device = dev;
    }
    Batch::Pending pend;
    pend.nbytes = static_cast<size_t>(g.count) * isz;
    at::Tensor base;
    if (pre && pre->out.defined() && pre->nbytes == pend.nbytes && pre->out.scalar_type() == st.dtype &&
        pre->out.device() == dev && pre->out.sizes() == c10::IntArrayRef(g.sizes)) {
      base = std::move(pre->out);  // the calling thread built the (memory-less) output while it walked the module
      pend.storage = std::move(pre->storage);
      g_stats.prebuilt_outputs++;
    } else {
      base = make_output(g.sizes, st.dtype, dev, pend.nbytes, pend.storage);
    }
    const uint64_t pt1 = Prof::on() ? Prof::tick() : 0;

    // every RNG pass on the chain consumes its slice of the stream, live or dead
    for (const RngPass& r : st.rng_chain) {
      RngSlot& slot = tape.rng[r.slot];
      if (slot.assigned) continue;
      assign_rng(tape, slot, r.numel, dev, gens);
      bool live = false;
      for (const FastSeg& sg : t.segs) live |= sg.rng_slot == r.slot;
      if (!live) g_stats.elided_rng_ops++;
    }
    const uint64_t pt2 = Prof::on() ? Prof::tick() : 0;
    if (Prof::on()) {
      g_prof.acc[3] += pt1 - pt0;
      g_prof.acc[4] += pt2 - pt1;
    }
    ProfScope p_descs(5);

    pend.first_desc = static_cast<uint32_t>(batch.descs.size());
    int64_t bytes = 0;
    for (const FastSeg& sg : t.segs) {
      const int64_t lo = std::max(sg.begin, g.begin), hi = std::min(sg.end, g.begin + g.count);
      if (lo >= hi) continue;
      batch.descs.push_back(sg.proto);
      TdxInitDesc& d = batch.descs.back();
      // byte offset inside the output until the submission gives the output its address
      d.dst = reinterpret_cast<void*>(static_cast<uintptr_t>(lo - g.begin) * isz);
      d.elem_count = static_cast<uint64_t>(hi - lo);
      if (sg.indexed) d.elem_begin = static_cast<uint64_t>(lo - sg.origin);  // index in the tensor the source op ran on
      if (sg.rng_slot != kNoValue) {
        const RngSlot& r = tape.rng[sg.rng_slot];
        d.philox_seed = r.seed;
        d.philox_offset = r.offset;
        if (sg.wide && wide_observable(tape, *sg.sym)) d.algo = TDX_ALGO_WIDE32;
      }
      bytes += (hi - lo) * static_cast<int64_t>(isz);
    }
    pend.n_desc = static_cast<uint32_t>(batch.descs.size()) - pend.first_desc;
    batch.pending.push_back(std::move(pend));
    g_stats.bytes_written += bytes;
    bytes_out = bytes;
    base_out = std::move(base);
    return true;
  }

  // ---- FSDP1 layout ----------------------------------------------------------------------------
  // The parameters of one FlatParameter, flattened and concatenated in order (each start optionally
  // aligned to `align` elements), chunked `world` ways by torch.chunk's rule, the last chunk
  // right-padded with zeros ($TORCH/distributed/fsdp/_flat_param.py:1089-1140 `_get_shard`,
  // :560-640 alignment padding): rank r's chunk is written straight into one 1-D tensor.  Neither a
  // parameter nor the flat parameter ever exists unsharded.  Every parameter's RNG passes are
  // assigned whether or not its elements fall into this rank's chunk, so all ranks agree.
  at::Tensor flat_shard(const std::vector<at::Tensor>& fakes, int64_t rank, int64_t world, int64_t align,
                        const std::optional<at::Tensor>& out_opt, std::vector<int64_t>* offsets_out) {
    TORCH_CHECK_VALUE(world >= 1 && rank >= 0 && rank < world, "flat shard: 0 <= rank < world_size required");
    struct Item {
      std::shared_ptr<Tape> tape;
      uint32_t value = kNoValue;
      int64_t offset = 0, numel = 0;
    };
    std::vector<Item> items;
    items.reserve(fakes.size());
    ScalarType dtype = ScalarType::Undefined;
    std::optional<c10::Device> dev;
    int64_t total = 0;
    for (const at::Tensor& f : fakes) {
      TORCH_CHECK_VALUE(can_materialize(f), "flat shard: every parameter must be a deferred (fake) tensor");
      const auto rec = fake_impl(f)->record();
      const ValueInfo& vi = rec->tape->values[rec->value];
      if (dtype == ScalarType::Undefined) dtype = vi.dtype;
      TORCH_CHECK_VALUE(vi.dtype == dtype, "flat shard: parameters of one flat parameter share one dtype");
      const c10::Device d = target_device(vi.device);
      TORCH_CHECK_VALUE(d.is_cuda(), "flat shard: the target device must be a CUDA device");
      if (!dev) dev = d;
      TORCH_CHECK_VALUE(*dev == d, "flat shard: parameters live on different devices");
      if (align > 1 && total % align) total += align - total % align;
      Item it;
      it.tape = rec->tape;
      it.value = rec->value;
      it.offset = total;
      it.numel = vi.numel;
      total += vi.numel;
      if (offsets_out) offsets_out->push_back(it.offset);
      items.push_back(std::move(it));
    }
    TORCH_CHECK_VALUE(dev.has_value(), "flat shard: no parameters");
    const size_t isz = c10::elementSize(dtype);
    const int64_t chunk = (total + world - 1) / world;
    const int64_t lo = std::min(total, rank * chunk), hi = std::min(total, lo + chunk);
    if (offsets_out) offsets_out->push_back(total);

    if (batch.device != *dev) {
      batch.flush();
      batch.device = *dev;
    }
    at::Tensor out;
    Batch::Pending pend;
    char* abs_base = nullptr;
    if (out_opt && out_opt->defined()) {
      out = *out_opt;
      TORCH_CHECK_VALUE(out.is_cuda() && out.device() == *dev && out.scalar_type() == dtype && out.dim() == 1 &&
                            out.is_contiguous() && out.numel() >= chunk,
                        "flat shard: `out` must be a contiguous 1-D CUDA tensor of the parameters' dtype with at "
                        "least ceil(total / world) elements");
      abs_base = static_cast<char*>(out.data_ptr());
    } else {
      pend.nbytes = static_cast<size_t>(chunk) * isz;
      const int64_t sizes[1] = {chunk};
      out = make_output(sizes, dtype, *dev, pend.nbytes, pend.storage);
    }
    auto place = [&](int64_t flat_index) {  // dst of a flat element of this rank's chunk
      return reinterpret_cast<void*>(abs_base + static_cast<uintptr_t>(flat_index - lo) * isz);
    };
    auto zero_fill = [&](int64_t b, int64_t e) {
      if (b >= e) return;
      TdxInitDesc d;
      std::memset(&d, 0, sizeof(d));
      d.src = TDX_SRC_CONST;
      d.dtype = isz == 1 ? TDX_RAW8 : isz == 2 ? TDX_RAW16 : isz == 4 ? TDX_RAW32 : TDX_RAW64;
      d.dst = place(b);
      d.elem_count = static_cast<uint64_t>(e - b);
      batch.descs.push_back(d);
    };
    struct Deferred {  // parameters the kernels cannot express: replayed whole, then copied (after the flush)
      at::Tensor full;
      int64_t src_begin, dst_begin, count;
    };
    std::vector<Deferred> deferred;
    // Pass 1, in order (it is the order RNG offsets are handed out in): decide per parameter, assign
    // the RNG passes of the fusible ones, replay the others now -- a replay may submit the batch, so
    // none of this chunk's descriptors may be in it yet.
    std::vector<std::unique_ptr<StorageTemplate>> owned;
    std::vector<const StorageTemplate*> plan(items.size(), nullptr);
    for (size_t k = 0; k < items.size(); ++k) {
      const Item& it = items[k];
      Tape& tape = *it.tape;
      const ValueInfo& vi = tape.values[it.value];
      const uint32_t S = vi.storage;
      StorageInfo& si = tape.storages[S];
      const int64_t b = std::max(it.offset, lo), e = std::min(it.offset + it.numel, hi);
      const StorageTemplate* t = nullptr;
      bool fusible = opts.fused && !si.replayed && !si.fused_done && !vi.real.defined() && vi.covers_storage;
      if (fusible) {
        if (si.tmpl && si.tmpl->fast) {
          t = si.tmpl.get();
          g_stats.template_hits++;
        } else if (!(si.tmpl && si.tmpl->st.opaque)) {
          auto tmp = std::make_unique<StorageTemplate>();
          if (si.tmpl) {
            tmp->st = si.tmpl->st;
          } else {
            struct FoldOn {
              c10::Device prev = g_fold_device;
              explicit FoldOn(c10::Device d) { g_fold_device = d; }
              ~FoldOn() { g_fold_device = prev; }
            } fold_on(*dev);
            c10::DeviceGuard fold_guard(*dev);
            tmp->st = eval_storage(tape, S, static_cast<uint32_t>(tape.ops.size()));
          }
          if (build_fast(tape, si, *tmp, /*may_sync=*/true)) {
            t = tmp.get();
            owned.push_back(std::move(tmp));
          }
        }
        fusible = t != nullptr && t->st.dtype == dtype;
      }
      if (!fusible) {
        // generic replay of the whole parameter on the GPU; its slice is copied into the chunk below
        at::Tensor full = materialize_value(it.tape, it.value);
        if (b < e) deferred.push_back(Deferred{full, b - it.offset, b, e - b});
        continue;
      }
      plan[k] = t;
      for (const RngPass& r : t->st.rng_chain) {  // every rank assigns every pass, owner or not
        RngSlot& slot = tape.rng[r.slot];
        if (!slot.assigned) assign_rng(tape, slot, r.numel, *dev, gens);
      }
    }
    if (batch.device != *dev) {
      batch.flush();
      batch.device = *dev;
    }
    pend.first_desc = static_cast<uint32_t>(batch.descs.size());
    // Pass 2: this chunk's descriptors (nothing else touches the batch from here to the flush)
    int64_t bytes = 0, covered = lo;  // [lo, covered) has been written or queued
    for (size_t k = 0; k < items.size(); ++k) {
      const Item& it = items[k];
      Tape& tape = *it.tape;
      const int64_t b = std::max(it.offset, lo), e = std::min(it.offset + it.numel, hi);
      // alignment gap in front of this parameter
      if (it.offset > covered && covered < hi) zero_fill(covered, std::min(it.offset, hi));
      covered = std::max(covered, std::min(it.offset + it.numel, hi));
      const StorageTemplate* t = plan[k];
      if (!t || b >= e) continue;
      const int64_t pb = b - it.offset, pe = e - it.offset;  // the parameter's own elements this rank holds
      for (const FastSeg& sg : t->segs) {
        const int64_t slo = std::max(sg.begin, pb), shi = std::min(sg.end, pe);
        if (slo >= shi) continue;
        batch.descs.push_back(sg.proto);
        TdxInitDesc& d = batch.descs.back();
        d.dst = place(it.offset + slo);
        d.elem_count = static_cast<uint64_t>(shi - slo);
        if (sg.indexed) d.elem_begin = static_cast<uint64_t>(slo - sg.origin);
        if (sg.rng_slot != kNoValue) {
          const RngSlot& r = tape.rng[sg.rng_slot];
          d.philox_seed = r.seed;
          d.philox_offset = r.offset;
          if (sg.wide && wide_observable(tape, *sg.sym)) d.algo = TDX_ALGO_WIDE32;
        }
        bytes += (shi - slo) * static_cast<int64_t>(isz);
      }
    }
    // the right zero-pad of the last rank(s): [hi, lo + chunk)
    if (covered < lo + chunk) {
      const int64_t b = std::max(covered, lo);
      TdxInitDesc d;
      std::memset(&d, 0, sizeof(d));
      d.src = TDX_SRC_CONST;
      d.dtype = isz == 1 ? TDX_RAW8 : isz == 2 ? TDX_RAW16 : isz == 4 ? TDX_RAW32 : TDX_RAW64;
      d.dst = place(b);
      d.elem_count = static_cast<uint64_t>(lo + chunk - b);
      if (d.elem_count) batch.descs.push_back(d);
    }
    if (!abs_base) {
      pend.n_desc = static_cast<uint32_t>(batch.descs.size()) - pend.first_desc;
      batch.pending.push_back(std::move(pend));
    }
    g_stats.bytes_written += bytes;
    g_stats.fused_tensors += static_cast<int64_t>(items.size() - deferred.size());
    batch.flush();
    if (!deferred.empty()) {
      NoInterception guard;
      for (const Deferred& d : deferred)
        out.narrow(0, d.dst_begin - lo, d.count).copy_(d.full.reshape({-1}).narrow(0, d.src_begin, d.count));
    }
    return out;
  }

  // Fused path for the storage of value `v`.  Returns false if the program is not fusible.
  bool try_fused(Tape& tape, uint32_t v, Prebuilt* pre = nullptr) {
    ValueInfo& vi = tape.values[v];
    const uint32_t S = vi.storage;
    StorageInfo& si = tape.storages[S];
    if (!opts.fused || si.replayed) return false;
    if (!target_device(vi.device).is_cuda()) return false;
    const bool sharded = sharding(vi);
    if (sharded && !vi.covers_storage) return false;
    at::Tensor base;
    int64_t bytes = 0;
    if (!emit_fused(tape, S, vi, sharded ? opts.shard : std::nullopt, base, bytes, pre)) return false;
    si.base = std::move(base);
    si.base_is_shard = sharded;
    si.fused_done = true;
    si.fused_epoch = batch.epoch;
    // (the storage's writer ops are not marked done one by one: `fused_done` stops every walk over
    // them -- collect_storage, eval_storage's callers -- and costs no cache line per op)
    g_stats.fused_tensors++;
    {
      ProfScope p(6);
      if (batch.expected_total == 0 && tape.fused_bytes)
        batch.expect(static_cast<int64_t>(tape.fused_bytes / static_cast<uint64_t>(opts.shard ? std::max<int64_t>(opts.shard->world, 1) : 1)),
                     tape.fused_storages);
      batch.note(bytes);  // may submit what has accumulated so far
    }
    return true;
  }

  // Does anything that determines storage S (as of op `upto`) draw random numbers?  A pure walk
  // over the recording (no side effects): programs without RNG can be replayed at any point of the
  // call without changing what anybody gets -- they neither read nor advance a generator.
  static bool is_random_op(const TapeOp& op) {
    switch (op.kind) {
      case OpKind::Randn: case OpKind::Rand: case OpKind::UniformInplace: case OpKind::NormalInplace: return true;
      default: break;
    }
    if (!op.handle) return false;
    const auto& schema = op.handle->schema();
    for (const auto& a : schema.arguments())
      if (a.name() == "generator") return true;
    const std::string& n = schema.name();
    return n.find("dropout") != std::string::npos || n.find("rrelu") != std::string::npos ||
           n.find("rand") != std::string::npos || n.find("bernoulli") != std::string::npos ||
           n.find("multinomial") != std::string::npos || n.find("poisson") != std::string::npos;
  }
  bool deterministic_slice(Tape& tape, uint32_t S, uint32_t upto, std::vector<uint32_t>& seen_upto) {
    if (seen_upto[S] >= upto) return true;
    seen_upto[S] = upto;
    const StorageInfo& si = tape.storages[S];
    if (si.fused_done) return true;
    // The same selection as collect_storage: every op that touches S up to its last writer is
    // replayed with it -- READERS included (they must see S at their point in history), and a reader
    // can draw random numbers through its other arguments: `torch.randn(n).copy_(s)` replays the
    // (dead) randn with s.  Looking at writers only let such a storage be deferred to the end of the
    // call, i.e. moved its reader's draw behind every later tensor's (1 of 3,000 random scripts
    // differed from the reference for that reason).
    uint32_t last_writer = kNoValue;
    for (uint32_t oi : si.touching_ops) {
      if (oi >= upto) break;
      for (uint32_t v : tape.ops[oi].outputs)
        if (v != kNoValue && tape.values[v].storage == S) last_writer = oi;
    }
    if (last_writer == kNoValue) return true;
    for (uint32_t oi : si.touching_ops) {
      if (oi > last_writer) break;
      const TapeOp& op = tape.ops[oi];
      if (op.done) continue;
      if (is_random_op(op)) return false;
      for (const InputRef& in : op.inputs) {
        if (in.foreign) return false;  // (another recording: keep it simple)
        if (in.value == kNoValue || tape.values[in.value].real.defined()) continue;
        if (!deterministic_slice(tape, tape.values[in.value].storage, oi, seen_upto)) return false;
      }
    }
    return true;
  }
  // Set by the session: unfusable programs without RNG are not replayed where the walk meets them but
  // after the call's last fused submission -- their dozen ATen dispatches (Llama's rotary inv_freq:
  // ~0.25 ms of host time) then run while the GPU already works on the whole model.
  bool defer_generic = false;

  // This rank's dim-0 chunk of a fully materialised tensor (generic replay always builds the whole
  // tensor: its ops are recorded on whole tensors).
  at::Tensor chunk_of(const ValueInfo& vi, const at::Tensor& full) {
    NoInterception guard;
    const ShardGeom g = shard_of(vi, opts.shard);
    const int64_t inner = vi.sizes[0] ? vi.numel / vi.sizes[0] : 0;
    const int64_t start = inner ? g.begin / inner : 0;
    return full.narrow(0, start, g.sizes[0]).clone();
  }

  at::Tensor materialize_value(const std::shared_ptr<Tape>& tape_ptr, uint32_t v, Prebuilt* pre = nullptr) {
    Tape& tape = *tape_ptr;
    ValueInfo& vi = tape.values[v];
    StorageInfo& si = tape.storages[vi.storage];
    if (si.fused_done) {
      at::Tensor t = real_of(tape, v);
      // (materialised whole earlier -- as a dependency, or by an unsharded call -- and asked for as a chunk now)
      return (sharding(vi) && !si.base_is_shard) ? chunk_of(vi, t) : t;
    }
    if (vi.real.defined()) return sharding(vi) ? chunk_of(vi, vi.real) : vi.real;
    if (try_fused(tape, v, pre)) {
      ProfScope p(7);
      return real_of(tape, v);
    }
    if (defer_generic) {
      std::vector<uint32_t> seen(tape.storages.size(), 0);
      if (deterministic_slice(tape, vi.storage, static_cast<uint32_t>(tape.ops.size()), seen)) return at::Tensor();
    }

    // generic replay, in recorded order, of everything that determines this storage.  Pending fused
    // descriptors stay in the batch (replay() submits them first if one of its inputs is among them):
    // a module's few unfusable buffers do not split the batch into extra launches.
    gens.write_back();  // ATen's own RNG kernels read the generators
    std::vector<uint8_t> mark(tape.ops.size(), 0);
    std::vector<uint32_t> visited(tape.storages.size(), 0);
    collect_storage(tape, vi.storage, static_cast<uint32_t>(tape.ops.size()), mark, visited);
    for (uint32_t oi = 0; oi < mark.size(); ++oi)
      if (mark[oi]) replay(tape, oi);
    TORCH_INTERNAL_ASSERT(vi.real.defined(), "replay did not produce `", tape.ops[vi.op].name(), "`");
    return sharding(vi) ? chunk_of(vi, vi.real) : vi.real;
  }
};

at::Tensor finish_tensor(const at::Tensor& fake, at::Tensor out) {
  // requires_grad_() is not an operator and cannot be recorded: re-apply it on leaves
  // (same rule as reference deferred_init.cc:722-726)
  if (fake.is_leaf() && fake.requires_grad() && !out.requires_grad() &&
      (out.is_floating_point() || out.is_complex())) {
    out.set_requires_grad(true);
  }
  return out;
}

}  // namespace

// Runs on the thread that walks the module (while the helper plans earlier tensors): builds the
// memory-less output tensor of `fake` -- TensorImpl, StorageImpl, autograd meta: half of what a
// tensor costs the helper -- if the analysis left on the recording says its storage will take the
// fused path.  The helper checks the geometry again and falls back to its own if anything differs.
bool prebuild_output(const at::Tensor& fake, const MaterializeOptions& opts, bool apply_shard, Prebuilt& pre) {
  if (!opts.fused || !can_materialize(fake)) return false;
  const TensorRecord* rec = fake_impl(fake)->record().get();
  if (!rec || !rec->tape || rec->value == kNoValue) return false;
  const Tape& tape = *rec->tape;
  const ValueInfo& vi = tape.values[rec->value];
  const StorageInfo& si = tape.storages[vi.storage];
  const StorageTemplate* t = si.tmpl.get();
  if (!t || !t->fast || si.fused_done || si.replayed || vi.real.defined()) return false;
  c10::Device dev = opts.device ? *opts.device : vi.device;
  if (!dev.is_cuda()) return false;
  if (!dev.has_index()) dev = c10::Device(c10::kCUDA, c10::cuda::current_device());
  const bool sharded = apply_shard && opts.shard && opts.shard->world > 1 && !vi.sizes.empty();
  if (sharded && !vi.covers_storage) return false;
  ShardGeom g;
  if (vi.covers_storage && vi.dtype == t->st.dtype) {
    g = shard_of(vi, sharded ? opts.shard : std::nullopt);
  } else {
    g.count = t->numel;
    g.sizes.assign(1, t->numel);
  }
  pre.nbytes = static_cast<size_t>(g.count) * t->isz;
  pre.out = make_output(g.sizes, t->st.dtype, dev, pre.nbytes, pre.storage);
  return true;
}

struct MaterializeSession::Impl {
  MaterializeOptions opts;
  Batch batch;
  Engine eng;
  double t_begin;
  double add_us = 0;
  bool finished = false;
  struct Deferred {
    at::Tensor fake;
    bool apply_shard;
    size_t ticket;
  };
  std::vector<Deferred> deferred;
  std::function<void(size_t, at::Tensor)> sink;
  explicit Impl(const MaterializeOptions& o) : opts(o), eng{o, batch}, t_begin(now_us()) {}
};

void MaterializeSession::defer_generic_programs(std::function<void(size_t, at::Tensor)> sink) {
  impl_->sink = std::move(sink);
  impl_->eng.defer_generic = static_cast<bool>(impl_->sink);
}

MaterializeSession::MaterializeSession(const MaterializeOptions& opts) {
  g_stats = MaterializeStats{};
  g_stats.traverse_us = g_pending_traverse_us;
  g_pending_traverse_us = 0;
  g_last_descs.clear();
  impl_ = std::make_unique<Impl>(opts);
  g_call_begin_us = impl_->t_begin;
}

MaterializeSession::~MaterializeSession() {
  // also on error paths: tensors planned so far are part of the recording's state (a later call
  // returns them), so their descriptors must run; offsets already handed out must stay consumed
  if (impl_ && !impl_->finished) {
    try { impl_->batch.flush(); } catch (...) {}
    try { impl_->eng.gens.write_back(); } catch (...) {}
  }
}

at::Tensor MaterializeSession::add(const at::Tensor& t, bool apply_shard, size_t ticket, Prebuilt* pre) {
  g_stats.tensors++;
  if (!can_materialize(t)) return t;
  const double t0 = now_us();
  impl_->eng.opts.shard = apply_shard ? impl_->opts.shard : std::nullopt;
  const TensorRecord* rec;
  {
    ProfScope p(0);
    rec = fake_impl(t)->record().get();  // (`t` keeps its record, and the record the tape, alive while we work)
  }
  at::Tensor value;
  {
    ProfScope p(1);
    value = impl_->eng.materialize_value(rec->tape, rec->value, pre);
  }
  if (!value.defined()) {  // an unfusable program without RNG: replayed after the last submission (finish)
    impl_->deferred.push_back(Impl::Deferred{t, apply_shard, ticket});
    impl_->add_us += now_us() - t0;
    return at::Tensor();
  }
  at::Tensor out;
  {
    ProfScope p(2);
    out = finish_tensor(t, std::move(value));
  }
  impl_->add_us += now_us() - t0;
  return out;
}

void MaterializeSession::finish() {
  struct TraceDump {
    ~TraceDump() {
      if (!trace_on() || g_sub_trace.empty()) return;
      cudaEventSynchronize(g_sub_trace.back().e1);
      fprintf(stderr, "[tdx] submissions (host us since call | MB | GPU start..end us since the first submission's enqueue):");
      for (SubmissionTrace& t : g_sub_trace) {
        float a = 0, b = 0;
        cudaEventElapsedTime(&a, g_trace_origin, t.e0);
        cudaEventElapsedTime(&b, g_trace_origin, t.e1);
        fprintf(stderr, "  [%.0f | %.0f | %.0f..%.0f]", t.host_us, t.bytes / 1e6, a * 1e3, b * 1e3);
        cudaEventDestroy(t.e0);
        cudaEventDestroy(t.e1);
      }
      fprintf(stderr, "\n");
      g_sub_trace.clear();
      cudaEventDestroy(g_trace_origin);
      g_trace_origin = nullptr;
    }
  } trace_dump;
  if (Prof::on()) {
    const uint64_t c0 = Prof::tick();
    const double u0 = now_us();
    while (now_us() - u0 < 200.0) {}
    const double ticks_per_us = static_cast<double>(Prof::tick() - c0) / (now_us() - u0);
    fprintf(stderr, "[tdx-prof] %lld tensors:", static_cast<long long>(g_stats.tensors));
    for (int k = 0; k < 10; ++k) fprintf(stderr, " %s=%.0fus", g_prof.names[k], g_prof.acc[k] / ticks_per_us);
    fprintf(stderr, "\n");
    g_prof = Prof{};
  }
  const double t0 = now_us();
  impl_->batch.flush();
  impl_->eng.gens.write_back();
  // the deferred programs: the kernels of every fused tensor are on the stream by now
  const double t_deferred = now_us();
  impl_->eng.defer_generic = false;
  for (Impl::Deferred& d : impl_->deferred) {
    impl_->eng.opts.shard = d.apply_shard ? impl_->opts.shard : std::nullopt;
    const auto rec = fake_impl(d.fake)->record();
    at::Tensor out = finish_tensor(d.fake, impl_->eng.materialize_value(rec->tape, rec->value));
    impl_->sink(d.ticket, std::move(out));
  }
  if (!impl_->deferred.empty()) {
    impl_->deferred.clear();
    impl_->batch.flush();  // (dependencies of the deferred programs that took the fused path)
    impl_->eng.gens.write_back();
  }
  g_stats.deferred_us = now_us() - t_deferred;
  impl_->finished = true;
  impl_->add_us += now_us() - t0;
  g_stats.plan_us = impl_->add_us - g_stats.launch_us;
  // whatever else happened between the first add() and now was the caller walking its modules
  g_stats.traverse_us += (now_us() - impl_->t_begin) - impl_->add_us;
}

std::vector<at::Tensor> materialize_many(const std::vector<at::Tensor>& fakes,
                                         const MaterializeOptions& opts,
                                         const std::vector<uint8_t>* shard_mask) {
  MaterializeSession session(opts);
  std::vector<at::Tensor> out(fakes.size());
  session.defer_generic_programs([&out](size_t i, at::Tensor t) { out[i] = std::move(t); });
  for (size_t i = 0; i < fakes.size(); ++i) {
    at::Tensor t = session.add(fakes[i], !(shard_mask && !(*shard_mask)[i]), i);
    if (t.defined()) out[i] = std::move(t);
  }
  session.finish();
  return out;
}

// ---------------------------------------------------------------------------------------------
// the session on a helper thread
// ---------------------------------------------------------------------------------------------
namespace {

// One helper thread per process, started on first use (and again in a forked child).
class HelperThread {
 public:
  // the planner of materialize_module calls
  static HelperThread& get() { return instance(0); }
  // Cleans up after them (recordings, replaced fake tensors).  A thread of its own: a call that
  // follows another one closely must not find the planner busy with the previous call's teardown.
  static HelperThread& reaper() { return instance(1); }
  static HelperThread& instance(int which) {
    static std::mutex m;
    static std::unique_ptr<HelperThread> inst[2];
    std::lock_guard<std::mutex> lock(m);
    if (!inst[which] || inst[which]->pid_ != getpid()) {
      if (inst[which] && inst[which]->pid_ != getpid()) inst[which].release();  // forked child: the parent's thread is not ours to join
      inst[which].reset(new HelperThread());
    }
    return *inst[which];
  }
  void post(std::function<void()> fn) {
    {
      std::lock_guard<std::mutex> lock(m_);
      q_.push_back(std::move(fn));
      posted_.fetch_add(1, std::memory_order_release);
    }
    cv_.notify_one();
  }
  // Calls come in trains (FSDP materialises one wrapped module after the other; a benchmark loops):
  // after a job the thread polls for the next one this long before it sleeps -- waking a parked
  // thread costs the next call 70-150 us (measured on the B200 hosts: `helper_start_us`).
  void linger(int64_t us) { linger_us_ = us; }
  ~HelperThread() {
    {
      std::lock_guard<std::mutex> lock(m_);
      stop_ = true;
    }
    cv_.notify_one();
    if (th_.joinable()) th_.join();
  }

 private:
  HelperThread() : pid_(getpid()), th_([this] { run(); }) {}
  void run() {
    for (;;) {
      std::function<void()> fn;
      if (linger_us_ > 0 && served_ > 0) {
        const auto until = std::chrono::steady_clock::now() + std::chrono::microseconds(linger_us_);
        while (posted_.load(std::memory_order_acquire) == served_) {
          for (int i = 0; i < 64; ++i) __builtin_ia32_pause();
          if (std::chrono::steady_clock::now() >= until) break;
        }
      }
      {
        std::unique_lock<std::mutex> lock(m_);
        cv_.wait(lock, [this] { return stop_ || !q_.empty(); });
        if (q_.empty()) return;  // stop requested and nothing left
        fn = std::move(q_.front());
        q_.pop_front();
        ++served_;
      }
      fn();
    }
  }
  pid_t pid_;
  std::mutex m_;
  std::condition_variable cv_;
  std::deque<std::function<void()>> q_;
  std::atomic<uint64_t> posted_{0};
  uint64_t served_ = 0;     // (helper thread only)
  std::atomic<int64_t> linger_us_{0};
  bool stop_ = false;
  std::thread th_;
};

bool host_threads_enabled() {
  static const bool v = [] {
    const char* e = getenv("TDX_HOST_THREADS");
    return !(e && e[0] == '0');
  }();
  return v;
}

}  // namespace

// The recording of a model is cold in the caches when it is materialised, and planning one tensor is
// a chain of dependent loads (tensor -> its record -> value -> storage -> analysis block -> RNG
// slots): ~100 ns each, more than the arithmetic.  The helper walks that chain a few queued tensors
// ahead, one link per tensor per step, with prefetches -- by the time a tensor is planned its lines
// have arrived.
class ChainPrefetcher {
 public:
  static constexpr int kDepth = 6;
  void advance(const at::Tensor& fake, int stage) {
    if (!is_fake(fake)) return;
    const FakeTensorImpl* impl = fake_impl(fake);
    switch (stage) {
      case 0:
        __builtin_prefetch(impl);
        __builtin_prefetch(reinterpret_cast<const char*>(impl) + sizeof(c10::TensorImpl));  // (record_ lives past the base)
        return;
      case 1: {
        const TensorRecord* r = impl->record().get();
        if (r) __builtin_prefetch(r);
        return;
      }
      default: break;
    }
    const TensorRecord* r = impl->record().get();
    if (!r || !r->tape || r->value == kNoValue) return;
    const Tape& tape = *r->tape;
    if (r->value >= tape.values.size()) return;
    const ValueInfo* vi = &tape.values[r->value];
    if (stage == 2) {
      __builtin_prefetch(vi);
      __builtin_prefetch(reinterpret_cast<const char*>(vi) + 64);
      __builtin_prefetch(reinterpret_cast<const char*>(vi) + 128);
      return;
    }
    const StorageInfo* si = &tape.storages[vi->storage];
    if (stage == 3) {
      __builtin_prefetch(si);
      __builtin_prefetch(reinterpret_cast<const char*>(si) + 64);
      return;
    }
    const StorageTemplate* t = si->tmpl.get();
    if (!t) return;
    if (stage == 4) {
      for (int k = 0; k < 6; ++k) __builtin_prefetch(reinterpret_cast<const char*>(t) + 64 * k);
      return;
    }
    if (stage == 5) {
      if (!t->st.rng_chain.empty()) {
        __builtin_prefetch(t->st.rng_chain.data());
        // (the slot index is in the chain entry; the first entry's slot is the earliest of the tensor)
      }
      if (!t->segs.empty() && t->segs[0].rng_slot != kNoValue && t->segs[0].rng_slot < tape.rng.size())
        __builtin_prefetch(&tape.rng[t->segs[0].rng_slot]);
      if (t->segs.size() > 0) __builtin_prefetch(reinterpret_cast<const char*>(&t->segs[0]) + 128);
    }
  }
};

struct PipelinedMaterialize::State {
  struct Item {
    at::Tensor fake;
    bool apply_shard = true;
    at::Tensor out;
    Prebuilt pre;  // built by the calling thread (PipelinedMaterialize::add), consumed by the helper
    std::atomic<uint8_t> done{0};
  };
  MaterializeOptions opts;
  bool threaded = false;
  double t_api_begin = now_us();               // (diagnostics: when the helper got going / was done, on the call's clock)
  at::ThreadLocalState tls;                    // the caller's, applied around the whole session
  std::vector<c10::cuda::CUDAStream> streams;  // the caller's current streams (its device, the target device)
  c10::DeviceIndex caller_device = -1;         // the caller's current CUDA device
  std::unique_ptr<MaterializeSession> session;  // inline mode only (the helper keeps its own on its stack)
  std::mutex m;
  std::condition_variable cv_work, cv_done;
  std::vector<std::unique_ptr<Item>> items;  // pushed by the caller, consumed in order by the helper
  bool finish_requested = false;
  bool helper_waiting = false;
  // Mirrors of items.size() / finish_requested the helper polls without the mutex: it plans faster
  // than the caller walks, and a helper that went to sleep after every tensor cost the CALLER a futex
  // wake-up per tensor (the walk of Llama-3-8B went from 0.2 to 0.6 ms when the planner got fast).
  std::atomic<size_t> n_items{0};
  std::atomic<bool> finish_flag{false};
  std::atomic<bool> caller_waiting{false};
  bool finished = false;
  std::exception_ptr error;
  size_t error_ticket = static_cast<size_t>(-1);  // the tensor whose materialisation raised `error`
  MaterializeStats stats;
  std::vector<TdxInitDesc> descs;

  void record_error(size_t ticket = static_cast<size_t>(-1)) {
    std::lock_guard<std::mutex> lock(m);
    if (!error) {
      error = std::current_exception();
      error_ticket = ticket;
      has_error.store(true, std::memory_order_release);
    }
  }
  std::atomic<bool> has_error{false};
  bool failed() { return has_error.load(std::memory_order_acquire); }  // (asked once per tensor: no lock)
  void process(MaterializeSession& s, Item& it, size_t ticket) {
    ProfScope p_total(8);
    if (!failed()) {
      try {
        it.out = s.add(it.fake, it.apply_shard, ticket, it.pre.out.defined() ? &it.pre : nullptr);
        if (!it.out.defined()) return;  // deferred to the end of the session: deliver() completes it
      } catch (...) {
        record_error(ticket);
      }
    }
    it.done.store(1, std::memory_order_release);
    if (caller_waiting.load(std::memory_order_acquire)) {
      std::lock_guard<std::mutex> lock(m);
      cv_done.notify_all();
    }
  }
  void deliver(size_t ticket, at::Tensor t) {  // a deferred result (MaterializeSession::finish)
    Item& it = *items[ticket];
    it.out = std::move(t);
    it.done.store(1, std::memory_order_release);
    if (caller_waiting.load(std::memory_order_acquire)) {
      std::lock_guard<std::mutex> lock(m);
      cv_done.notify_all();
    }
  }
  // The helper's side of one session: one task, one ThreadLocalStateGuard, items in batches.
  void run_on_helper() {
    try {
      at::ThreadLocalStateGuard g(tls);
      // The helper must sit on the caller's device: with another current device every DeviceGuard of
      // the planner would switch devices twice per tensor (and create a context on device 0 in every
      // rank of a multi-GPU job).  Device and streams stay until the next call sets its own.
      if (caller_device >= 0) c10::cuda::set_device(caller_device);
      for (const auto& st : streams) c10::cuda::setCurrentCUDAStream(st);
      const double helper_start = now_us() - t_api_begin;
      MaterializeSession s(opts);
      s.defer_generic_programs([this](size_t ticket, at::Tensor t) { deliver(ticket, std::move(t)); });
      size_t next = 0, first = 0;
      std::vector<Item*> batch;
      for (;;) {
        bool fin;
        // a call lasts a millisecond: poll for that long before sleeping
        for (int spin = 0; spin < 200000 && next == n_items.load(std::memory_order_acquire) &&
                           !finish_flag.load(std::memory_order_acquire); ++spin) {
#if defined(__x86_64__) || defined(__i386__)
          __builtin_ia32_pause();
#endif
        }
        {
          std::unique_lock<std::mutex> lock(m);
          while (next == items.size() && !finish_requested) {
            helper_waiting = true;
            cv_work.wait(lock);
            helper_waiting = false;
          }
          fin = finish_requested;
          batch.clear();
          for (size_t i = next; i < items.size(); ++i) batch.push_back(items[i].get());
          first = next;
          next = items.size();
        }
        ChainPrefetcher pf;
        for (size_t i = 0; i < batch.size(); ++i) {
          // tensor i + d is at link (kDepth - d) of its chain
          for (int d = 1; d <= ChainPrefetcher::kDepth; ++d)
            if (i + d < batch.size()) pf.advance(batch[i + d]->fake, ChainPrefetcher::kDepth - d);
          process(s, *batch[i], first + i);
        }
        if (fin && batch.empty()) break;  // finish() was requested and nothing arrived after it
      }
      if (!failed()) {
        try {
          s.finish();
        } catch (...) {
          record_error();
        }
      }
      g_stats.helper_start_us = helper_start;
      g_stats.helper_done_us = now_us() - t_api_begin;
      stats = g_stats;  // the helper thread's counters of this session
      descs = g_last_descs;
    } catch (...) {  // (session construction / thread-local state)
      record_error();
    }
    std::lock_guard<std::mutex> lock(m);
    for (auto& it : items) it->done.store(1, std::memory_order_release);  // nobody waits for ever
    finished = true;
    cv_done.notify_all();
  }
};

PipelinedMaterialize::PipelinedMaterialize(const MaterializeOptions& opts) : st_(std::make_shared<State>()) {
  st_->opts = opts;
  st_->threaded = host_threads_enabled();
  st_->items.reserve(1024);
  if (st_->threaded) {
    // Counting devices starts the CUDA runtime, which a child forked afterwards cannot use: like
    // torch.cuda, mark such children (is_device_in_bad_fork), where a CPU-only call skips CUDA.
    torch::utils::register_fork_handler_for_device_init(at::kCUDA);
    if (!torch::utils::is_device_in_bad_fork(at::kCUDA) && at::hasCUDA() && c10::cuda::device_count() > 0) {
      // Only devices this call can touch, and only if they are in use already: asking for another
      // device's stream, or sitting on a device the process never used, would create a CUDA context
      // there (a CPU-only materialise on a GPU machine must not start CUDA at all).
      const auto& hooks = at::detail::getCUDAHooks();
      const c10::DeviceIndex cur = c10::cuda::current_device();
      const bool cur_live = hooks.hasPrimaryContext(cur);
      if (cur_live) st_->streams.push_back(c10::cuda::getCurrentCUDAStream(cur));
      if (opts.device && opts.device->is_cuda() && opts.device->has_index()) {
        st_->caller_device = opts.device->index();  // the device every tensor of this call is built on
        if (opts.device->index() != cur && hooks.hasPrimaryContext(opts.device->index()))
          st_->streams.push_back(c10::cuda::getCurrentCUDAStream(opts.device->index()));
      } else if (cur_live) {
        st_->caller_device = cur;
      }
    }
    auto st = st_;
    static const int64_t linger_us = [] {
      const char* e = getenv("TDX_HELPER_LINGER_US");
      return e ? std::max<int64_t>(0, atoll(e)) : int64_t{2000};
    }();
    HelperThread& helper = HelperThread::get();
    helper.linger(linger_us);
    helper.post([st] { st->run_on_helper(); });
  } else {
    st_->session = std::make_unique<MaterializeSession>(opts);
    State* raw = st_.get();
    st_->session->defer_generic_programs([raw](size_t ticket, at::Tensor t) { raw->deliver(ticket, std::move(t)); });
  }
}

PipelinedMaterialize::~PipelinedMaterialize() {
  if (!st_) return;
  if (!st_->threaded) {
    st_->session.reset();  // writes the generators back if finish() was never reached
    return;
  }
  // the helper must be done with the caller's tensors and generators before the caller goes on
  std::unique_lock<std::mutex> lock(st_->m);
  if (!st_->finish_requested) {
    st_->finish_requested = true;
    st_->finish_flag.store(true, std::memory_order_release);
    if (!st_->error) {
      st_->error = std::make_exception_ptr(std::runtime_error("materialize_module was abandoned"));
      st_->has_error.store(true, std::memory_order_release);
    }
    st_->cv_work.notify_one();
  }
  st_->cv_done.wait(lock, [&] { return st_->finished; });
}

size_t PipelinedMaterialize::add(const at::Tensor& fake, bool apply_shard, at::Tensor* speculative) {
  auto item = std::make_unique<State::Item>();
  item->fake = fake;
  item->apply_shard = apply_shard;
  if (st_->threaded && speculative && prebuild_output(fake, st_->opts, apply_shard, item->pre)) {
    // what the helper will (almost certainly) return for this tensor: the caller may give it its
    // Python identity right away and confirm with result() at the end
    *speculative = finish_tensor(fake, item->pre.out);
  }
  State::Item* raw = item.get();
  size_t ticket;
  bool wake;
  {
    std::lock_guard<std::mutex> lock(st_->m);
    ticket = st_->items.size();
    st_->items.push_back(std::move(item));
    st_->n_items.store(st_->items.size(), std::memory_order_release);
    wake = st_->helper_waiting;
  }
  if (!st_->threaded) {
    st_->process(*st_->session, *raw, ticket);
  } else if (wake) {
    st_->cv_work.notify_one();
  }
  return ticket;
}

void PipelinedMaterialize::finish() {
  if (!st_->threaded) {
    if (!st_->failed()) {
      try {
        st_->session->finish();
      } catch (...) {
        st_->record_error();
      }
    }
    st_->session.reset();
    std::lock_guard<std::mutex> lock(st_->m);
    st_->finished = true;
    return;
  }
  std::lock_guard<std::mutex> lock(st_->m);
  st_->finish_requested = true;
  st_->finish_flag.store(true, std::memory_order_release);
  st_->cv_work.notify_one();
}

bool PipelinedMaterialize::ready(size_t ticket) {
  return st_->items[ticket]->done.load(std::memory_order_acquire) != 0;  // (items is only grown by this thread)
}

at::Tensor PipelinedMaterialize::result(size_t ticket) {
  State::Item& it = *st_->items[ticket];
  // The helper finishes a tensor every microsecond or two: spin for a while before paying a futex
  // sleep + wake-up per tensor (and making the helper pay the notify).
  for (int spin = 0; spin < 4096 && it.done.load(std::memory_order_acquire) == 0; ++spin) {
#if defined(__x86_64__) || defined(__i386__)
    __builtin_ia32_pause();
#endif
  }
  if (it.done.load(std::memory_order_acquire) == 0) {
    std::unique_lock<std::mutex> lock(st_->m);
    st_->caller_waiting.store(true, std::memory_order_release);
    st_->cv_done.wait(lock, [&] { return it.done.load(std::memory_order_acquire) != 0; });
    st_->caller_waiting.store(false, std::memory_order_release);
  }
  {
    std::lock_guard<std::mutex> lock(st_->m);
    if (st_->error) std::rethrow_exception(st_->error);
  }
  return it.out;
}

size_t PipelinedMaterialize::failed_ticket() {
  std::lock_guard<std::mutex> lock(st_->m);
  return st_->error ? st_->error_ticket : static_cast<size_t>(-1);
}

void PipelinedMaterialize::join() {
  std::unique_lock<std::mutex> lock(st_->m);
  st_->cv_done.wait(lock, [&] { return st_->finished; });
  if (st_->threaded) {  // inline mode already counted on this thread
    g_stats = st_->stats;
    g_stats.traverse_us = g_pending_traverse_us;  // the caller's own measure of its walk
    g_last_descs = st_->descs;
  }
  g_pending_traverse_us = 0;
  if (st_->error) std::rethrow_exception(st_->error);
}

void release_in_background(std::vector<std::shared_ptr<Tape>> tapes) {
  if (tapes.empty() || !host_threads_enabled()) return;  // (inline mode: they die with the caller's copies)
  auto box = std::make_shared<std::vector<std::shared_ptr<Tape>>>(std::move(tapes));
  HelperThread::reaper().post([box] { box->clear(); });
}

bool post_background(std::function<void()> fn) {
  if (!host_threads_enabled()) return false;
  HelperThread::reaper().post(std::move(fn));
  return true;
}

void drain_background() {
  if (!host_threads_enabled()) return;
  struct Gate {
    std::mutex m;
    std::condition_variable cv;
    int pending = 2;
  };
  auto gate = std::make_shared<Gate>();
  auto arrive = [gate] {
    std::lock_guard<std::mutex> lock(gate->m);
    --gate->pending;
    gate->cv.notify_all();
  };
  HelperThread::get().post(arrive);
  HelperThread::reaper().post(arrive);
  std::unique_lock<std::mutex> lock(gate->m);
  gate->cv.wait(lock, [&] { return gate->pending == 0; });
}

std::vector<int64_t> submission_sizes(int64_t total_bytes, int64_t tensors, bool with_estimate) {
  // (a copy of the bookkeeping in Batch::note with the flush itself left out)
  Batch b;
  std::vector<int64_t> out;
  if (tensors <= 0 || total_bytes <= 0) return out;
  if (with_estimate) b.expect(total_bytes, tensors);
  const int64_t each = total_bytes / tensors;
  int64_t pending = 0;
  for (int64_t i = 0; i < tensors; ++i) {
    pending += each;
    if (b.flush_threshold > 0 && pending >= b.flush_threshold) {
      b.submitted_bytes += pending;
      if (b.flush_threshold < (int64_t{1} << 60)) b.last_threshold = b.flush_threshold;
      out.push_back(pending);
      pending = 0;
      b.flush_threshold = b.next_threshold();
    }
  }
  if (pending) out.push_back(pending);
  return out;
}

void add_wrap_time(double us) { g_stats.wrap_us += us; }
// (materialize_many resets the counters: the traversal that precedes it is reported through a
// pending value that the next reset picks up)
void add_traverse_time(double us) { g_pending_traverse_us += us; }
void add_assign_time(double us) { g_stats.assign_us += us; }

at::Tensor materialize_flat_shard(const std::vector<at::Tensor>& fakes, const MaterializeOptions& opts, int64_t rank,
                                  int64_t world, int64_t align_numel, const std::optional<at::Tensor>& out,
                                  std::vector<int64_t>* offsets) {
  g_stats = MaterializeStats{};
  g_last_descs.clear();
  g_call_begin_us = now_us();
  Batch batch;
  Engine eng{opts, batch};
  at::Tensor result;
  try {
    result = eng.flat_shard(fakes, rank, world, align_numel, out, offsets);
  } catch (...) {
    try { batch.flush(); } catch (...) {}
    try { eng.gens.write_back(); } catch (...) {}
    throw;
  }
  eng.gens.write_back();
  g_stats.tensors = static_cast<int64_t>(fakes.size());
  return result;
}

at::Tensor materialize_one(const at::Tensor& fake, const MaterializeOptions& opts) {
  if (!can_materialize(fake)) return fake;
  return materialize_many({fake}, opts)[0];
}

PlanInfo plan_info(const at::Tensor& fake) {
  PlanInfo info;
  if (!can_materialize(fake)) {
    info.source = "real";
    return info;
  }
  info.deferred = true;
  const auto rec = fake_impl(fake)->record();
  Tape& tape = *rec->tape;
  const ValueInfo& vi = tape.values[rec->value];
  info.dtype = c10::toString(vi.dtype);
  info.numel = vi.numel;
  info.sizes.assign(vi.sizes.begin(), vi.sizes.end());
  info.device = vi.device.str();
  info.requires_grad = fake.is_leaf() && fake.requires_grad();
  const StorageInfo& si = tape.storages[vi.storage];
  if (vi.real.defined() || si.fused_done) {
    info.source = "materialized";
    return info;
  }
  // fold constants where the tensor will live, if that device exists here (a plan built on a
  // machine without a GPU folds 16-bit constant arithmetic with the CPU kernels' rounding)
  struct FoldOn {
    c10::Device prev = g_fold_device;
    explicit FoldOn(c10::Device d) { g_fold_device = d; }
    ~FoldOn() { g_fold_device = prev; }
  } fold_on(vi.device.is_cuda() && at::hasCUDA() ? vi.device : c10::Device(c10::kCPU));
  State fresh;
  if (!si.tmpl) fresh = eval_storage(tape, vi.storage, static_cast<uint32_t>(tape.ops.size()));
  const State& st = si.tmpl ? si.tmpl->st : fresh;
  static const char* names[] = {"uninit", "const", "uniform", "normal", "iota"};
  if (st.opaque || st.segs.empty()) {
    info.source = "opaque";
    // best effort: the first op on the storage the planner does not model
    for (uint32_t oi : si.touching_ops) {
      const TapeOp& op = tape.ops[oi];
      if (op.kind == OpKind::Generic) {
        info.first_unfusable_op = op.name();
        break;
      }
    }
    return info;
  }
  const size_t isz = c10::elementSize(st.dtype);
  // the segment that writes the most elements names the tensor's source
  const Seg* main = &st.segs.front();
  for (const Seg& g : st.segs)
    if (g.end - g.begin > main->end - main->begin) main = &g;
  info.source = names[main->st.src];
  info.fusible = si.replayed ? false : true;
  info.p0 = main->st.p0;
  info.p1 = main->st.p1;
  info.n_epilogue = static_cast<int>(main->st.epi.size());
  info.rng_ops = static_cast<int>(st.rng_chain.size());
  info.wide = wide_observable(tape, main->st);
  info.src_noround = main->st.src_noround;
  for (const TdxEpiStep& e : main->st.epi) info.epilogue.emplace_back(static_cast<int>(e.op), e.a, e.b);
  for (const RngPass& r : st.rng_chain) {
    info.rng_numels.push_back(r.numel);
    info.rng_op_ids.push_back(static_cast<int64_t>((tape.uid << 32) | r.op));
  }
  for (const Seg& g : st.segs) {
    PlanSegment ps;
    ps.begin = g.begin;
    ps.end = g.end;
    ps.origin = g.origin;
    ps.source = names[g.st.src];
    ps.p0 = g.st.p0;
    ps.p1 = g.st.p1;
    ps.wide = wide_observable(tape, g.st);
    ps.src_noround = g.st.src_noround;
    for (const TdxEpiStep& e : g.st.epi) ps.epilogue.emplace_back(static_cast<int>(e.op), e.a, e.b);
    if (g.st.rng()) {
      if (tdx_dtype_of(st.dtype) < 0) info.fusible = false;
      for (size_t i = 0; i < st.rng_chain.size(); ++i)
        if (st.rng_chain[i].op == g.st.rng_op) ps.rng_pass = static_cast<int>(i);
    }
    if (g.st.src == Sym::Const) {
      unsigned char one[16];
      size_t got = 0;
      if (!(g.st.has_scalar && scalar_bits(g.st.cscalar, st.dtype, one, &got) && got == isz)) {
        Sym tmp = g.st;
        ensure_cval(tmp, st.dtype);
        NoInterception guard;
        std::memcpy(one, tmp.cval.cpu().contiguous().data_ptr(), isz);
      }
      ps.const_bytes.assign(reinterpret_cast<const char*>(one), isz);
      if (!(isz == 1 || isz == 2 || isz == 4 || isz == 8)) info.fusible = false;
      if (&g == main) info.const_bytes = ps.const_bytes;
    }
    info.segments.push_back(std::move(ps));
  }
  if (!vi.covers_storage || vi.dtype != st.dtype) info.fusible = false;  // a plan names whole tensors only
  return info;
}

void analyze_tape(Tape& tape) noexcept {
  struct Flag {
    Flag() { g_analysis_only = true; }
    ~Flag() { g_analysis_only = false; }
  } flag;
  const uint32_t n_ops = static_cast<uint32_t>(tape.ops.size());
  for (uint32_t S = 0; S < tape.storages.size(); ++S) {
    StorageInfo& si = tape.storages[S];
    if (si.tmpl || si.fused_done) continue;
    g_analysis_deferred = false;
    try {
      NoInterception guard;
      State st = eval_storage(tape, S, n_ops);
      // constant chains fold with the TARGET device's arithmetic and programs that read a real
      // tensor see its value at materialisation time: both are evaluated then
      if (g_analysis_deferred) continue;
      auto t = std::make_shared<StorageTemplate>();
      t->st = std::move(st);
      build_fast(tape, si, *t, /*may_sync=*/false);
      if (t->fast && si.live > 0) {
        tape.fused_bytes += static_cast<uint64_t>(t->numel) * t->isz;
        tape.fused_storages++;
      }
      si.tmpl = std::move(t);
    } catch (...) {
      // (e.g. uniform_ with from > to: the error is raised when the tensor is materialised)
    }
  }
}

std::vector<std::string> storage_history(const at::Tensor& fake) {
  std::vector<std::string> out;
  if (!can_materialize(fake)) return out;
  const auto rec = fake_impl(fake)->record();
  Tape& tape = *rec->tape;
  const StorageInfo& si = tape.storages[tape.values[rec->value].storage];
  for (uint32_t oi : si.touching_ops) {
    const TapeOp& op = tape.ops[oi];
    std::string line = op.name();
    bool writes = false, covers = true;
    for (uint32_t v : op.outputs)
      if (v != kNoValue && tape.values[v].storage == tape.values[rec->value].storage) {
        writes = true;
        covers = covers && tape.values[v].covers_storage;
      }
    if (is_pure_alias(op.kind)) line += covers ? " [alias]" : " [view]";
    else line += writes ? (covers ? " [writes]" : " [writes part]") : " [reads]";
    out.push_back(line);
  }
  return out;
}

MaterializeStats last_stats() { return g_stats; }

std::string last_descriptors() {
  return std::string(reinterpret_cast<const char*>(g_last_descs.data()),
                     g_last_descs.size() * sizeof(TdxInitDesc));
}

at::Tensor cached_python_tensor(const at::Tensor& fake) {
  if (!can_materialize(fake)) return {};
  const auto& rec = fake_impl(fake)->record();
  return rec->tape->values[rec->value].py_wrapped;
}

void cache_python_tensor(const at::Tensor& fake, const at::Tensor& wrapped) {
  if (!can_materialize(fake)) return;
  const auto& rec = fake_impl(fake)->record();
  rec->tape->values[rec->value].py_wrapped = wrapped;
}

}  // namespace tdx
