// Plans over strided buffers (b200fft_plan_create_strided): the layout rules, checked before any CUDA call, and the passes,
// one plan-time tile kernel per transformed axis in its StrLay form (fast.cuh), reading and writing the user's arrays through
// their strides. No copy pass: the first pass reads the input where it lies and the last one writes the output in place.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>
#include <string>
#include <vector>

#include "tile.hpp"

namespace b200fft {

namespace {

// One buffer over the dimensions (batch, d0, ..., d_{rank-1}) of its own layout: extents and element strides.
struct BufLayout {
  int nd = 0;
  int64_t ext[STR_MAX_OUTER] = {};
  int64_t st[STR_MAX_OUTER] = {};
};

enum Side { REAL_SIDE, COMPLEX_SIDE, FULL };

BufLayout dense_layout(const Problem& p, Side side) {
  BufLayout L;
  L.nd = p.rank + 1;
  L.ext[0] = p.batch;
  for (int a = 0; a < p.rank; ++a) L.ext[a + 1] = p.axes[a].n;
  if (side == COMPLEX_SIDE) L.ext[p.rank] = p.axes[p.rank - 1].n / 2 + 1;
  int64_t s = 1;
  for (int d = L.nd - 1; d >= 0; --d) {
    L.st[d] = s;
    s *= L.ext[d];
  }
  return L;
}
Side in_side(const Problem& p) { return !p.half ? FULL : p.desc.inverse ? COMPLEX_SIDE : REAL_SIDE; }
Side out_side(const Problem& p) { return !p.half ? FULL : p.desc.inverse ? REAL_SIDE : COMPLEX_SIDE; }

BufLayout with_strides(BufLayout L, const std::vector<int64_t>& st) {
  for (int d = 0; d < L.nd; ++d) L.st[d] = st[(size_t)d];
  return L;
}

// largest element offset the layout reaches; false when it does not fit int64
bool max_offset(const BufLayout& L, int64_t* off) {
  int64_t m = 0;
  for (int d = 0; d < L.nd; ++d) {
    int64_t t;
    if (__builtin_mul_overflow(L.ext[d] - 1, L.st[d], &t) || __builtin_add_overflow(m, t, &m)) return false;
  }
  *off = m;
  return true;
}

// One pass of a strided plan, decided on the host alone.
struct StrPassPlan {
  int axis = 0;
  HalfMode half = HALF_NONE;
  BufSel ssel = BUF_INPUT, dsel = BUF_OUTPUT;
  TileSpec spec;
  StrGeo geo{};
  long long count = 0, ncols = 0;
  std::string layout;
};

// Axes right to left like build_passes (api.cu): the first pass reads the input, the others run in place on the output (the
// C2R inverse: on the dense half-spectrum workspace, then the C2R rows into the output). A pass runs as rows when the axis
// has the smallest stride of the buffer it reads, otherwise as column tiles along the dimension that has it.
int plan_passes(const b200fft_plan& plan, std::vector<StrPassPlan>* out) {
  const Problem& p = plan.prob;
  const int last = p.rank - 1;
  const bool inv = p.desc.inverse != 0, f64 = p.desc.out_dtype == B200FFT_F64;
  const bool even = p.axes[last].n % 2 == 0;
  const BufLayout lay[3] = {with_strides(dense_layout(p, in_side(p)), plan.in_strides),
                            with_strides(dense_layout(p, out_side(p)), plan.out_strides), dense_layout(p, COMPLEX_SIDE)};
  const IoSpec in_spec{p.desc.in_dtype, p.desc.in_components};
  const IoSpec work_spec{p.desc.out_dtype, 2};
  auto add = [&](int axis, HalfMode half, BufSel ssel, BufSel dsel, const IoSpec& src) -> int {
    const BufLayout& S = lay[ssel];
    const BufLayout& D = lay[dsel];
    const int k = axis + 1;
    // even half-spectrum rows: the real side is read / written as pairs of scalars, its strides (all even) count pairs
    const int64_t sdiv = half == HALF_R2C && even ? 2 : 1, ddiv = half == HALF_C2R && even ? 2 : 1;
    std::vector<int> cand;
    for (int d = 0; d < S.nd; ++d)
      if (d != k && S.ext[d] > 1) cand.push_back(d);
    int col = -1;
    if (half == HALF_NONE)
      for (int d : cand)
        if (S.st[d] < S.st[k] && (col < 0 || S.st[d] < S.st[col])) col = d;
    std::vector<int> outer;
    for (int d : cand)
      if (d != col) outer.push_back(d);
    std::stable_sort(outer.begin(), outer.end(), [&](int x, int y) { return S.st[x] < S.st[y]; });
    StrPassPlan pp;
    pp.axis = axis;
    pp.half = half;
    pp.ssel = ssel;
    pp.dsel = dsel;
    pp.geo.nouter = (int)outer.size();
    pp.count = 1;
    for (size_t j = 0; j < outer.size(); ++j) {
      pp.geo.ext[j] = S.ext[outer[j]];
      pp.geo.ss[j] = S.st[outer[j]] / sdiv;
      pp.geo.ds[j] = D.st[outer[j]] / ddiv;
      pp.count *= S.ext[outer[j]];
    }
    pp.geo.s_ax = half == HALF_NONE ? S.st[k] : 1;
    pp.geo.d_ax = half == HALF_NONE ? D.st[k] : 1;
    char buf[160];
    if (col >= 0) {
      pp.geo.s_col = S.st[col];
      pp.geo.d_col = D.st[col];
      pp.ncols = S.ext[col];
      snprintf(buf, sizeof buf, "; column tiles along dimension %d (stride %lld -> %lld), axis stride %lld -> %lld", col,
               (long long)S.st[col], (long long)D.st[col], (long long)S.st[k], (long long)D.st[k]);
    } else {
      snprintf(buf, sizeof buf, "; rows, axis stride %lld -> %lld", (long long)S.st[k], (long long)D.st[k]);
    }
    pp.layout = std::string(buf) + (ssel == BUF_INPUT ? " (reads input)" : ssel == BUF_WORK ? " (workspace)" : " (in place)");
    const int64_t n = p.axes[axis].n;
    if (!jit_strided_spec(p.axes[axis], n, pp.ncols, pp.count, src, half == HALF_NONE ? inv : half == HALF_C2R, half, f64, &pp.spec))
      return fail(B200FFT_ERR_UNSUPPORTED, "axis %d: %s", axis, last_error().c_str());
    out->push_back(pp);
    return B200FFT_OK;
  };
  int rc;
  if (!p.half) {
    bool first = true;
    for (int axis = last; axis >= 0; --axis) {
      if (!p.axes[axis].transformed) continue;
      if ((rc = add(axis, HALF_NONE, first ? BUF_INPUT : BUF_OUTPUT, BUF_OUTPUT, first ? in_spec : work_spec))) return rc;
      first = false;
    }
    return B200FFT_OK;
  }
  if (!inv) {
    if ((rc = add(last, HALF_R2C, BUF_INPUT, BUF_OUTPUT, in_spec))) return rc;
    for (int axis = last - 1; axis >= 0; --axis)
      if (p.axes[axis].transformed && (rc = add(axis, HALF_NONE, BUF_OUTPUT, BUF_OUTPUT, work_spec))) return rc;
    return B200FFT_OK;
  }
  bool any = false;
  for (int axis = last - 1; axis >= 0; --axis) {
    if (!p.axes[axis].transformed) continue;
    if ((rc = add(axis, HALF_NONE, any ? BUF_WORK : BUF_INPUT, BUF_WORK, any ? work_spec : in_spec))) return rc;
    any = true;
  }
  return add(last, HALF_C2R, any ? BUF_WORK : BUF_INPUT, BUF_OUTPUT, any ? work_spec : in_spec);
}

}  // namespace

int strided_check(b200fft_plan* plan, const int64_t* in_strides, const int64_t* out_strides, bool* dense) {
  const Problem& p = plan->prob;
  const BufLayout din = dense_layout(p, in_side(p)), dout = dense_layout(p, out_side(p));
  const int nd = p.rank + 1;
  plan->in_strides.assign(din.st, din.st + nd);
  plan->out_strides.assign(dout.st, dout.st + nd);
  if (in_strides) plan->in_strides.assign(in_strides, in_strides + nd);
  if (out_strides) plan->out_strides.assign(out_strides, out_strides + nd);
  // no kernel reads the stride of a dimension of extent 1 (a batch of 1, an axis of one point): any value is the dense one
  for (int d = 0; d < nd; ++d) {
    if (din.ext[d] == 1) plan->in_strides[(size_t)d] = din.st[d];
    if (dout.ext[d] == 1) plan->out_strides[(size_t)d] = dout.st[d];
  }
  *dense = std::equal(plan->in_strides.begin(), plan->in_strides.end(), din.st) &&
           std::equal(plan->out_strides.begin(), plan->out_strides.end(), dout.st);
  if (*dense) return B200FFT_OK;
  const BufLayout in = with_strides(din, plan->in_strides), out = with_strides(dout, plan->out_strides);
  for (int d = 0; d < nd; ++d) {
    if (in.st[d] < 0) return fail(B200FFT_ERR_LAYOUT, "in_strides[%d] = %lld is negative", d, (long long)in.st[d]);
    if (out.st[d] < 1) return fail(B200FFT_ERR_LAYOUT, "out_strides[%d] = %lld: output strides must be at least 1", d, (long long)out.st[d]);
  }
  int64_t in_max = 0, out_max = 0;
  if (!max_offset(in, &in_max) || !max_offset(out, &out_max))
    return fail(B200FFT_ERR_INVALID_ARG, "the %s layout reaches element offsets beyond int64", max_offset(in, &in_max) ? "output" : "input");
  // no two output elements at one offset: in increasing stride order, each stride clears the span of the ones before it
  std::vector<int> order;
  for (int d = 0; d < nd; ++d)
    if (out.ext[d] > 1) order.push_back(d);
  std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return out.st[x] < out.st[y]; });
  for (size_t j = 1; j < order.size(); ++j) {
    const int a = order[j - 1], b = order[j];
    if (out.st[b] < out.st[a] * out.ext[a])  // no overflow: (ext - 1) * stride fits, and so does one stride more here
      return fail(B200FFT_ERR_LAYOUT, "output dimensions %d (stride %lld, extent %lld) and %d (stride %lld) overlap", a,
                  (long long)out.st[a], (long long)out.ext[a], b, (long long)out.st[b]);
  }
  const size_t in_elem = p.in_elem * (in_side(p) == REAL_SIDE || (!p.half && p.desc.in_components == 1) ? 1 : 2);
  const size_t out_elem = p.out_elem * (out_side(p) == REAL_SIDE ? 1 : 2);
  int64_t in_bytes, out_bytes;
  if (__builtin_mul_overflow(in_max + 1, (int64_t)in_elem, &in_bytes) || __builtin_mul_overflow(out_max + 1, (int64_t)out_elem, &out_bytes))
    return fail(B200FFT_ERR_INVALID_ARG, "the strided buffers span more than 2^63 bytes");
  if (p.half) {
    const int last = p.rank;
    if (in.st[last] != 1 || out.st[last] != 1)
      return fail(B200FFT_ERR_UNSUPPORTED, "half-spectrum plans take stride 1 along the last axis on both sides (pitched rows); got "
                  "%lld and %lld", (long long)in.st[last], (long long)out.st[last]);
    const BufLayout& real = p.desc.inverse ? out : in;
    if (p.axes[p.rank - 1].n % 2 == 0)
      for (int d = 0; d < last; ++d)
        if (real.st[d] % 2)
          return fail(B200FFT_ERR_UNSUPPORTED, "real-side stride %lld of dimension %d is odd: the R2C / C2R kernels of an even "
                      "length move real rows as pairs of scalars, so every real-side stride must be even", (long long)real.st[d], d);
  }
  if (p.desc.flags & (B200FFT_FLAG_FORCE_GENERIC | B200FFT_FLAG_FORCE_RT))
    return fail(B200FFT_ERR_UNSUPPORTED, "strided layouts run on the plan-time tier only; %s leaves it out",
                (p.desc.flags & B200FFT_FLAG_FORCE_GENERIC) ? "FORCE_GENERIC" : "FORCE_RT");
  if (const char* e = getenv("B200FFT_JIT"))
    if (atoi(e) == 0) return fail(B200FFT_ERR_UNSUPPORTED, "strided layouts run on the plan-time tier only, which B200FFT_JIT=0 turns off");
  std::vector<StrPassPlan> passes;
  if (int rc = plan_passes(*plan, &passes)) return rc;
  plan->strided = true;
  plan->in_span = (size_t)in_bytes;
  plan->out_span = (size_t)out_bytes;
  if (!p.half) {
    plan->inplace_exact = p.desc.in_components == 2 && p.desc.in_dtype == p.desc.out_dtype && plan->in_strides == plan->out_strides;
  } else {  // the classic padded layout: real strides twice the complex ones on every dimension but the last
    const std::vector<int64_t>& re = p.desc.inverse ? plan->out_strides : plan->in_strides;
    const std::vector<int64_t>& cx = p.desc.inverse ? plan->in_strides : plan->out_strides;
    plan->inplace_exact = p.desc.in_dtype == p.desc.out_dtype;
    // (a dimension of extent 1 holds no second element: its strides, set to each side's dense value above, are not compared)
    for (int d = 0; d + 1 < nd; ++d)
      plan->inplace_exact = plan->inplace_exact && (din.ext[d] == 1 || re[(size_t)d] == 2 * cx[(size_t)d]);
  }
  return B200FFT_OK;
}

int build_strided_passes(b200fft_plan* plan) {
  const Problem& p = plan->prob;
  std::vector<StrPassPlan> v;
  if (int rc = plan_passes(*plan, &v)) return rc;
  for (const StrPassPlan& pp : v)
    if (pp.ssel == BUF_WORK || pp.dsel == BUF_WORK) {
      const BufLayout w = dense_layout(p, COMPLEX_SIDE);
      plan->work_stride = (size_t)w.st[0] * 2 * p.out_elem;
      plan->workspace_bytes = plan->work_stride * (size_t)p.batch;
      if (cudaMalloc(&plan->workspace, plan->workspace_bytes) != cudaSuccess) {
        cudaGetLastError();
        return fail(B200FFT_ERR_ALLOC, "cannot allocate %zu B of C2R workspace", plan->workspace_bytes);
      }
      break;
    }
  for (const StrPassPlan& pp : v) {
    std::unique_ptr<StridedPass> pass = make_jit_strided_pass(*plan, pp.axis, pp.spec, p.axes[pp.axis].n, pp.half, p.desc.inverse != 0);
    if (!pass)
      return fail(B200FFT_ERR_UNSUPPORTED, "axis %d: the plan-time kernel %s of this strided pass could not be built: %s", pp.axis,
                  pp.spec.kind == TILE_COLS ? "(column tiles)" : "(rows)", last_error().c_str());
    pass->geo = pp.geo;
    pass->count = pp.count;
    pass->ncols = pp.ncols;
    pass->dependent = !plan->passes.empty();
    pass->src_sel = pp.ssel;
    pass->dst_sel = pp.dsel;
    pass->axis = pp.axis;
    pass->text += pp.layout;
    plan->passes.push_back(std::move(pass));
  }
  return B200FFT_OK;
}

}  // namespace b200fft
