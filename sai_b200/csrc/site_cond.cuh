// Per-site conditions with the reference's float64 semantics.
//
// Follows compute_matching_loci (sai/stats/stat_utils.py:114-166):
//   freq      = num / (called * ploidy)            IEEE double division (:49-52)
//   valid     = every freq finite and in [0,1]     (:121-130)
//   match_y   = AND_k op_k(src_freq_k, y_k)        (:141-144)
//   match_1my = AND_k op_k(src_freq_k, 1 - y_k)    only without ancestral alleles,
//               with `1 - y_k` evaluated by the host in Python floats (:148-152)
//   inverted  = match_1my & valid -> ref/tgt freq := 1 - freq   (:156-160)
//   cond      = valid & (match_y | match_1my) & ref_freq < w    (:166)
// and UStatistic adds tgt_freq > x (sai/stats/u_statistic.py:92); QStatistic
// keeps tgt_freq of the cond sites (sai/stats/q_statistic.py:92).
// Every arithmetic step uses the explicitly rounded intrinsics so that no FMA
// contraction or fast-math flag can change a decision.
#pragma once
#include "common.cuh"

namespace sai {

struct SiteFlags {
  bool u;
  bool q;
  double q_tgt_freq;
};

// op(f, y) without a jump table: bit 2 = "<", bit 1 = "==", bit 0 = ">" of the relation
// between f and y, tested against the set of relations the operator accepts
// (EQ 010, LT 100, GT 001, LE 110, GE 011).  A NaN satisfies none, like the reference's
// numpy comparisons.
__device__ __forceinline__ bool cmp_op(int op, double f, double y) {
  const int accept = (0x3c62 >> (3 * op)) & 7;  // 011 110 001 100 010
  const int rel = (f < y ? 4 : 0) | (f == y ? 2 : 0) | (f > y ? 1 : 0);
  return (rel & accept) != 0;
}

// One condition block; returns cond and the (possibly inverted) tgt frequency.
__device__ __forceinline__ bool eval_cond(const sai_cond& c, int n_src, bool anc, double fr,
                                          double ft, const double* fs, double& tgt_out) {
  bool my = true, mf = true;
#pragma unroll
  for (int k = 0; k < SAI_MAX_SRC; ++k) {
    if (k < n_src) {
      my = my && cmp_op(c.op[k], fs[k], c.y[k]);
      mf = mf && cmp_op(c.op[k], fs[k], c.one_minus_y[k]);
    }
  }
  const bool inv = !anc && mf;
  const bool match = my || inv;
  const double r = inv ? __dsub_rn(1.0, fr) : fr;
  tgt_out = inv ? __dsub_rn(1.0, ft) : ft;
  return match && (r < c.w);
}

// num / den in IEEE double for den > 0 and 0 <= num <= den (other inputs: result unused).
// 0 / den is exact without dividing, and a zero numerator would send the whole warp
// through __ddiv_rn's slow path (a subroutine call of ~100 instructions): the divider is
// fed den / den on those lanes instead and the quotient replaced by 0.
__device__ __forceinline__ double site_freq(int num, int den) {
  const double q = __ddiv_rn((double)(num > 0 ? num : den), (double)(den > 0 ? den : 1));
  return num > 0 ? q : 0.0;
}

template <typename NumFn, typename CalledFn>
__device__ __forceinline__ SiteFlags eval_site(const sai_job& J, const sai_layout& lay,
                                               NumFn num_of, CalledFn called_of) {
  SiteFlags out{false, false, 0.0};
  const int nr = num_of(J.ref_pop), dr = called_of(J.ref_pop) * lay.pop[J.ref_pop].ploidy;
  const int nt = num_of(J.tgt_pop), dt = called_of(J.tgt_pop) * lay.pop[J.tgt_pop].ploidy;
  // freq in [0,1] and finite  <=>  den > 0 and 0 <= num <= den  (num is never negative)
  bool valid = dr > 0 && nr <= dr && dt > 0 && nt <= dt;
  double fs[SAI_MAX_SRC];
#pragma unroll
  for (int k = 0; k < SAI_MAX_SRC; ++k) {
    if (k < J.n_src) {
      const int sp = J.src_pop[k];
      const int ns = num_of(sp), ds = called_of(sp) * lay.pop[sp].ploidy;
      valid = valid && ds > 0 && ns <= ds;
      fs[k] = site_freq(ns, ds);
    } else {
      fs[k] = 0.0;
    }
  }
  if (!valid) return out;
  const double fr = site_freq(nr, dr);
  const double ft = site_freq(nt, dt);
  const bool anc = J.anc_allele_available != 0;
  // U and Q of one job usually share w and the source conditions (the reference's configs
  // repeat them): evaluate the block once then
  bool shared = J.u.enabled && J.q.enabled && J.u.w == J.q.w;
#pragma unroll
  for (int k = 0; k < SAI_MAX_SRC; ++k)
    if (k < J.n_src)
      shared = shared && J.u.op[k] == J.q.op[k] && J.u.y[k] == J.q.y[k] && J.u.one_minus_y[k] == J.q.one_minus_y[k];
  if (shared) {
    double t;
    const bool c = eval_cond(J.u, J.n_src, anc, fr, ft, fs, t);
    out.u = c && (t > J.x);
    out.q = c;
    out.q_tgt_freq = t;
    return out;
  }
  if (J.u.enabled) {
    double t;
    const bool c = eval_cond(J.u, J.n_src, anc, fr, ft, fs, t);
    out.u = c && (t > J.x);
  }
  if (J.q.enabled) {
    double t;
    const bool c = eval_cond(J.q, J.n_src, anc, fr, ft, fs, t);
    out.q = c;
    out.q_tgt_freq = t;
  }
  return out;
}

// ---------------------------------------------------------------------------
// Integer fast path.  For a FIXED denominator d (= individuals * ploidy: every call of
// the population present), freq(n) = fl(n / d) is non-decreasing in the count n and
// fl(1 - freq(n)) non-increasing, so each float64 decision of compute_matching_loci is
// an interval test on n.  The host finds the interval ends by bisection with the very
// same IEEE operations (build_job_fast), and a site whose populations are all fully
// called is decided with integer compares only -- the divisions are left to the sites
// that fail this test (missing calls) and to the Q-flagged sites, whose target
// frequency is an output.  Decisions are identical by construction; the tests compare
// the masks and Q values of both paths on random data.
// ---------------------------------------------------------------------------
struct CondFast {
  int32_t ref_max;      // not inverted: ref_freq < w      <=>  num_ref <= ref_max
  int32_t ref_inv_min;  // inverted:     1 - ref_freq < w  <=>  num_ref >= ref_inv_min
  int32_t y_lo[SAI_MAX_SRC], y_hi[SAI_MAX_SRC];  // op(src_freq, y)      <=>  y_lo <= num_src <= y_hi
  int32_t f_lo[SAI_MAX_SRC], f_hi[SAI_MAX_SRC];  // op(src_freq, 1 - y)  <=>  f_lo <= num_src <= f_hi
};
struct JobFast {
  int32_t ok;  // thresholds are valid
  int32_t den_ref, den_tgt, den_src[SAI_MAX_SRC];
  int32_t tgt_min;      // not inverted: tgt_freq > x      <=>  num_tgt >= tgt_min
  int32_t tgt_inv_max;  // inverted:     1 - tgt_freq > x  <=>  num_tgt <= tgt_inv_max
  CondFast u, q;
};
struct JobFastBlock {
  JobFast job[SAI_MAX_JOBS];
};

template <typename NumFn, typename CalledFn>
__device__ __forceinline__ SiteFlags eval_site_fast(const JobFast& F, const sai_job& J, const sai_layout& lay,
                                                    NumFn num_of, CalledFn called_of) {
  const int nr = num_of(J.ref_pop), dr = called_of(J.ref_pop) * lay.pop[J.ref_pop].ploidy;
  const int nt = num_of(J.tgt_pop), dt = called_of(J.tgt_pop) * lay.pop[J.tgt_pop].ploidy;
  bool full = F.ok != 0 && dr == F.den_ref && dt == F.den_tgt;
  bool valid = nr <= dr && nt <= dt;
  // one pass over the sources (n_src is warp-uniform: a plain loop, no per-source arrays): the
  // interval tests of both condition blocks against y and against 1 - y
  bool my_u = true, mf_u = true, my_q = true, mf_q = true;
  for (int k = 0; k < J.n_src; ++k) {
    const int sp = J.src_pop[k];
    const int ns = num_of(sp);
    const int ds = called_of(sp) * lay.pop[sp].ploidy;
    full = full && ds == F.den_src[k];
    valid = valid && ns <= ds;
    my_u = my_u && ns >= F.u.y_lo[k] && ns <= F.u.y_hi[k];
    mf_u = mf_u && ns >= F.u.f_lo[k] && ns <= F.u.f_hi[k];
    my_q = my_q && ns >= F.q.y_lo[k] && ns <= F.q.y_hi[k];
    mf_q = mf_q && ns >= F.q.f_lo[k] && ns <= F.q.f_hi[k];
  }
  // warp-uniform choice: a tile with a missing call anywhere takes the division path
  if (!__all_sync(0xffffffffu, full)) return eval_site(J, lay, num_of, called_of);
  SiteFlags out{false, false, 0.0};
  const bool anc = J.anc_allele_available != 0;
  if (J.u.enabled) {
    const bool inv = !anc && mf_u;
    const bool c = valid && (my_u || inv) && (inv ? nr >= F.u.ref_inv_min : nr <= F.u.ref_max);
    out.u = c && (inv ? nt <= F.tgt_inv_max : nt >= F.tgt_min);
  }
  if (J.q.enabled) {
    const bool inv = !anc && mf_q;
    const bool c = valid && (my_q || inv) && (inv ? nr >= F.q.ref_inv_min : nr <= F.q.ref_max);
    out.q = c;
    if (c) {
      const double ft = site_freq(nt, dt);
      out.q_tgt_freq = inv ? __dsub_rn(1.0, ft) : ft;
    }
  }
  return out;
}

// ---------------------------------------------------------------------------
// Gates of the staged genotype pass (k_site_live).  A site is flagged only if its sources
// match (op(src_freq, y), or op(src_freq, 1 - y) without ancestral alleles) and its possibly
// inverted ref_freq < w, so the pass reads the sources first and the reference and target only
// where a job can still hold.  Each factor below is evaluated per lane exactly as eval_site /
// eval_site_fast evaluate it (interval test for a fully called population, the IEEE division
// otherwise), so a gate is a superset of the final decision: it lets through every site that
// will be flagged, and the flags themselves still come from eval_site_fast.
// with_ref == false: sources only (the reference need not have been read yet).
// ---------------------------------------------------------------------------
template <typename NumFn, typename CalledFn>
__device__ __forceinline__ void site_gate(const JobFast& F, const sai_job& J, const sai_layout& lay, bool with_ref,
                                          NumFn num_of, CalledFn called_of, bool& gate_u, bool& gate_q) {
  const bool fast = F.ok != 0;
  bool valid = true, my_u = true, mf_u = true, my_q = true, mf_q = true;
  for (int k = 0; k < J.n_src; ++k) {
    const int sp = J.src_pop[k];
    const int ns = num_of(sp);
    const int ds = called_of(sp) * lay.pop[sp].ploidy;
    valid = valid && ds > 0 && ns <= ds;
    if (fast && ds == F.den_src[k]) {
      my_u = my_u && ns >= F.u.y_lo[k] && ns <= F.u.y_hi[k];
      mf_u = mf_u && ns >= F.u.f_lo[k] && ns <= F.u.f_hi[k];
      my_q = my_q && ns >= F.q.y_lo[k] && ns <= F.q.y_hi[k];
      mf_q = mf_q && ns >= F.q.f_lo[k] && ns <= F.q.f_hi[k];
    } else {
      const double fs = site_freq(ns, ds);
      my_u = my_u && cmp_op(J.u.op[k], fs, J.u.y[k]);
      mf_u = mf_u && cmp_op(J.u.op[k], fs, J.u.one_minus_y[k]);
      my_q = my_q && cmp_op(J.q.op[k], fs, J.q.y[k]);
      mf_q = mf_q && cmp_op(J.q.op[k], fs, J.q.one_minus_y[k]);
    }
  }
  const bool anc = J.anc_allele_available != 0;
  gate_u = valid && J.u.enabled && (my_u || (!anc && mf_u));
  gate_q = valid && J.q.enabled && (my_q || (!anc && mf_q));
  if (!with_ref || !(gate_u || gate_q)) return;
  const int nr = num_of(J.ref_pop), dr = called_of(J.ref_pop) * lay.pop[J.ref_pop].ploidy;
  if (!(dr > 0 && nr <= dr)) {
    gate_u = gate_q = false;
    return;
  }
  const bool full = fast && dr == F.den_ref;
  const double fr = full ? 0.0 : site_freq(nr, dr);
  // ref_freq < w, or 1 - ref_freq < w where the job inverts (as eval_cond)
  auto ref_ok = [&](const CondFast& X, const sai_cond& C, bool inv) {
    if (full) return inv ? nr >= X.ref_inv_min : nr <= X.ref_max;
    return (inv ? __dsub_rn(1.0, fr) : fr) < C.w;
  };
  gate_u = gate_u && ref_ok(F.u, J.u, !anc && mf_u);
  gate_q = gate_q && ref_ok(F.q, J.q, !anc && mf_q);
}

// host: interval ends for one job (plain IEEE double division / subtraction, as on the device)
void build_job_fast(const sai_layout& lay, const sai_job& J, JobFast& F);

}  // namespace sai
