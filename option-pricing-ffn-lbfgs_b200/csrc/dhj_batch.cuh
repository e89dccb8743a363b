// dhj_batch.cuh — throughput kernel for grids / option lists with at most 8 strikes per maturity slice
// (the 15-option grid of C2 / C4 / the generator / the calibrator's market).
//
// Decomposition (DESIGN.md §3): ONE LANE PER COSINE INDEX k, a block of 128 threads walks a batch of
// 32 items (item = one (parameter set, maturity slice)):
//   phase 1  thread t < 32 prepares item t ALONE: parameters (optionally exp/tanh transform), per-set
//            constants, truncation range, pass constants, the slice's strikes (K, log(K/S0), exp(.),
//            binding flags) -> shared memory.  The prologue is therefore executed once per item by one
//            lane instead of redundantly by every lane of a warp (it was ~10 % of the warp-per-item
//            kernel's instructions).
//   phase 2  each WARP takes every fourth item and walks its cosine terms 32 at a time: lane = k within
//            the block of 32 (constants are broadcast reads from shared memory; the KTerm lives in
//            registers and is consumed at once by the <= 8 strikes of the slice); the <= 8 prices
//            accumulate in registers and are written by the warp itself — no block barrier, no
//            partial sums in shared memory.  Walking k in order lets the trigonometric factors that
//            are linear in k advance by rotation (contract_pass).
// A strike whose +-0.1 widening binds (double_heston.py:135-137) is contracted in an extra pass of
// phase 2 with its own (a,b): rare, set up by lane 0 of the warp.
#pragma once
#include "dhj_engine.cuh"

namespace dhj {

constexpr int kBatchThreads = 128;
constexpr int kBatchWarps = kBatchThreads / 32;
// items per block batch: phase 1 fills its warp
#ifndef DHJ_PRICE_ITEMS
#define DHJ_PRICE_ITEMS 32
#endif
constexpr int kPriceItems = DHJ_PRICE_ITEMS;
constexpr int kBatchMaxStrikes = 8;
// resident blocks per SM the kernels are compiled for (register budget = 65 536 / (128 * MINB)).  Measured on C2
// (profiles/README.md): 7 blocks at 72 registers 14.36 ms, 6 at 80 14.40, 5 at 96 14.51, 4 at 122 14.03, 3 at 140
// 14.72 — with room for the temporaries of both Heston factors ptxas overlaps their dependent chains, which is
// worth more than the 12 warps given up.  The fused loss kernel runs the same engine with the same budget (a
// 72-register build that parked its loop state in shared memory was 20 % slower per price and had to evaluate some
// terms differently from the pricing kernel; one arithmetic for both keeps every loss independent of how the
// evaluations are grouped into launches).
#ifndef DHJ_BATCH_MINB
#define DHJ_BATCH_MINB 4
#endif

struct ItemRec {
  SetConsts set;
  PassConsts pass;                 // regular pass: (a0, b0) = (pass.a, pass.b)
  double S0, disc;
  double cmu, smu;                 // cos / sin(32 u_1 mu): the jump term's rotation from one block of 32 k to the next
  double gj2;                      // exp(-2048 alpha), alpha = sj^2 u_1^2 / 2: second ratio of the jump factor's Gaussian
  double K[kBatchMaxStrikes], x[kBatchMaxStrikes], ex[kBatchMaxStrikes];      // strike, log(K/S0), S0 * exp(x)
  double cth[kBatchMaxStrikes], sth[kBatchMaxStrikes];      // cos / sin of theta_j = u_1 (x_j - a0)
  double c32[kBatchMaxStrikes], s32[kBatchMaxStrikes];      // cos / sin of 32 theta_j
  unsigned valid_mask, bind_mask, call_mask;
  int o_lo;                        // first option (slice order) of the slice
  long long out_row;               // p * M
#if defined(DHJ_CHECKED)
  unsigned long long tag;          // batch that prepared the record
#endif
};

// one warp's k-block of strike-independent coefficients P, Q, R.
// Layout: PQ[k] = (P_k, Q_k) and R[k], for 128-bit loads in the contraction (one for P and Q, one for two consecutive
// R); the batch kernel's four 8-term segments are read concurrently by different lanes, so each segment is shifted
// by one 16-byte slot (PQ) / two doubles (R) to land in different banks.
struct CoefStage {
  Pair PQ[36];
  double R[40];
#if defined(DHJ_CHECKED)
  unsigned wtag[32], rtag[32], epoch;      // epoch of the last write per k slot / of the last read per lane / running epoch
#endif
};

// pass of a strike whose +-0.1 widening binds: its own (a, b) and the rotation steps that go with it
struct ExtraPass {
  PassConsts pass;
  double cth, sth, c32, s32, cmu, smu, gj2;      // (cmu, smu, gj2 contiguous: contract_pass reads them as one triple)
};

template <int ITEMS>
struct BatchSmemT {
  ItemRec items[ITEMS];
  ExtraPass extra[kBatchWarps];
  CoefStage stage[kBatchWarps];
  fm::TrigTables ltab;             // fm::log_tab / exp_tab / atan2_tab / sincos_tab tables (per-lane index: shared memory, not the constant bank)
};
using PriceSmem = BatchSmemT<kPriceItems>;

struct PriceArgs;                  // dhj_kernels.cuh

// every block copies the lookup tables into its shared memory once (THREADS: the block size)
template <int THREADS>
__device__ __forceinline__ void load_log_table(fm::Tables* dst, int tid) {
  for (int i = tid; i < 65; i += THREADS) {
    if (i < 64) { dst->log[i] = fm::kTables.log[i]; dst->exp2[i] = fm::kTables.exp2[i]; }
    dst->atan64[i] = fm::kTables.atan64[i];
  }
}
template <int THREADS>
__device__ __forceinline__ void load_log_table(fm::TrigTables* dst, int tid) {
  load_log_table<THREADS>(static_cast<fm::Tables*>(dst), tid);
  for (int i = tid; i < fm::kSinCosTab; i += THREADS) dst->sincos[i] = fm::kTables.sincos[i];
}

// checked build: the stage's epoch bookkeeping starts at zero
__device__ __forceinline__ void stage_check_init(CoefStage& st, int lane) {
#if defined(DHJ_CHECKED)
  st.wtag[lane] = 0u; st.rtag[lane] = 0u;
  if (lane == 0) st.epoch = 0u;
#endif
}

// u_1 = (1*pi)/(b-a), the rotation step's frequency (same correction step as u_of_k)
__device__ __forceinline__ double u_one(const PassConsts& p) {
  const double q0 = kPi * p.rw;
  return fma(fma(-p.w, q0, kPi), p.rw, q0);
}

// rotation steps of one pass: theta = u_1 (x - a) per strike, and the jump term's 32 u_1 mu
__device__ __forceinline__ void strike_rotation(const PassConsts& p, double x, double* cth, double* sth, double* c32,
                                                double* s32) {
  const double th = u_one(p) * (x - p.a);
  fm::sincos_(th, sth, cth);
  fm::sincos_(32.0 * th, s32, c32);
}
__device__ __forceinline__ void jump_rotation(const PassConsts& p, double mu, double* cmu, double* smu) {
  fm::sincos_((32.0 * u_one(p)) * mu, smu, cmu);
}
// The jump factor's magnitude exp(-alpha k^2), alpha = hsj2 u_1^2, is Gaussian in k: from one block of 32 k to the
// next it is multiplied by rho_b = exp(-alpha (64 k + 1024)), and rho itself by the constant exp(-2048 alpha):
// two products per block instead of an exp (exact re-evaluation with the rotations, every kReseed blocks).
__device__ __forceinline__ double jump_alpha(const PassConsts& p, double hsj2) {
  const double u1 = u_one(p);
  return hsj2 * (u1 * u1);
}

// phase 1 for one item, executed by a single thread
__device__ __forceinline__ void prepare_item(ItemRec& rec, const SliceView& v, const Params& m, double S0,
                                             const double* __restrict__ strike_row, int s_idx, long long out_row) {
  rec.set = make_set_consts(m, v.r, v.q);
  const double T = v.slice_T[s_idx];
  double a0, b0;
  truncation_range(m, T, v.r, v.L, &a0, &b0);
  rec.pass = make_pass_consts(rec.set, a0, b0, T);
  rec.S0 = S0;
  rec.disc = fm::exp_(-v.r * T);
  jump_rotation(rec.pass, rec.set.mu, &rec.cmu, &rec.smu);
  rec.gj2 = fm::exp_neg(-2048.0 * jump_alpha(rec.pass, rec.set.hsj2));
  const int o_lo = v.slice_off[s_idx], cnt = v.slice_off[s_idx + 1] - o_lo;
  unsigned bind = 0, call = 0;
#pragma unroll 1
  for (int j = 0; j < cnt; ++j) {
    double K = strike_row[v.pos[o_lo + j]];
    if (v.scale_by_spot) K = K * S0 / 100.0;
    const StrikeConsts sc = make_strike_consts(K, S0);
    rec.K[j] = sc.K; rec.x[j] = sc.x; rec.ex[j] = S0 * sc.ex;
    strike_rotation(rec.pass, sc.x, &rec.cth[j], &rec.sth[j], &rec.c32[j], &rec.s32[j]);
    if (((sc.x - 0.1) < a0) || ((sc.x + 0.1) > b0)) bind |= 1u << j;
    if (v.call[o_lo + j]) call |= 1u << j;
  }
  rec.valid_mask = (1u << cnt) - 1u;
  rec.bind_mask = bind; rec.call_mask = call;
  rec.o_lo = o_lo; rec.out_row = out_row;
}
__device__ __forceinline__ void tag_item(ItemRec& rec, unsigned long long batch_tag) {
#if defined(DHJ_CHECKED)
  rec.tag = batch_tag;
#endif
}

// The quantities that are trigonometric functions of an angle LINEAR in k — the jump term's (cos, sin)(u_k mu)
// and the contraction segments' start (cos, sin)(k theta_j) — are evaluated in full in the first block of 32 k
// (fm::sincos_tab) and then advanced from block to block by one plane rotation (4 FP64 instructions instead of a
// 17-instruction sincos_tab); every kReseed-th block starts from an exact evaluation again (error growth <= kReseed ulp).
constexpr int kReseed = 8;

__device__ __forceinline__ void rotate(double& c, double& s, double cr, double sr) {
  const double c2 = fma(c, cr, -(s * sr)), s2 = fma(s, cr, c * sr);
  c = c2; s = s2;
}

// One pass of ONE WARP over all cosine terms of an item, 32 at a time: CF at this lane's k -> strike-independent
// coefficients in the warp's stage; then the rotation tasks: lane = (strike j, segment s) with 8-term segments,
// reduced over the 4 segments by two shuffles and accumulated in `acc` of the lanes (j, 0).  The sums A1, A2, A3
// (and g0) do not depend on the strike: each lane accumulates its share over the blocks and the warp reduces
// them once at the end of the pass.
__device__ __forceinline__ void contract_pass(const ItemRec& it, const PassConsts& pc, const double* __restrict__ cth,
                                              const double* __restrict__ sth, const double* __restrict__ c32,
                                              const double* __restrict__ s32, const double* __restrict__ cmu_smu,
                                              unsigned mask, int n_cos, int lane, CoefStage& st,
                                              const fm::TrigTables* __restrict__ ltab, double& acc) {
  constexpr int kSeg = 8, kNumSeg = 32 / kSeg;
  const int slot_pq = lane + (lane >> 3), slot_r = lane + 2 * (lane >> 3);      // padded stage slots of this lane's k
  // A1, A2 feed calls, A3 puts (uniform per pass)
  const bool any_call = (it.call_mask & mask) != 0, any_put = (~it.call_mask & mask) != 0;
  double a1 = 0.0, a2 = 0.0, a3 = 0.0, g0_keep = 0.0;
  double cj = 1.0, sj = 0.0, cs = 1.0, sn = 0.0;
  double ej = 1.0, rho = 1.0;                                  // jump Gaussian and its block-to-block ratio
  int blk = 0;
  // two blocks of k per trip (the `exact` test and the loop overhead are shared; four copies overflow the
  // instruction cache: 13.29 / 13.06 / 14.73 ms for 1 / 2 / 4)
#pragma unroll 2
  for (int k0 = 0; k0 < n_cos; k0 += 32, ++blk) {
    const int k = k0 + lane;
    const bool exact = (blk % kReseed) == 0;               // uniform
    const double u = u_of_k(pc, k);
    KTerm t = make_kterm_f(it.set, pc, k, ltab, u, [&](double* cj_out, double* sj_out, double* ej_out) {
      if (exact) {
        fm::sincos_tab(u * it.set.mu, ltab, &sj, &cj);
        ej = jump_gauss(it.set, u, ltab);
        rho = fm::exp_tab_neg(-(jump_alpha(pc, it.set.hsj2) * (double)(64 * k + 1024)), ltab);
      } else {
        ej *= rho; rho *= cmu_smu[2];
        rotate(cj, sj, cmu_smu[0], cmu_smu[1]);
      }
      *cj_out = cj; *sj_out = sj; *ej_out = ej;
    });
    t.G = (k < n_cos) ? t.G : 0.0;                           // ragged last block: every coefficient is a multiple of G
    const KCoef c = make_kcoef(t, pc, k);
    if (any_call) { a1 = fma(c.P, t.t1 + t.t3, a1); a2 = fma(c.R, t.sb, a2); }
    if (any_put) a3 += c.P;
    if (blk == 0) g0_keep = __shfl_sync(kFullMask, c.g0, 0);
    __syncwarp();
#if defined(DHJ_CHECKED)
    const unsigned epoch = st.epoch + 1;                     // (same value in every lane: read between two barriers)
    for (int l = 0; l < 32; ++l) DHJ_CHECK(st.rtag[l] == epoch - 1, kChkWriteBeforeConsumed);
    DHJ_CHECK(slot_pq < 36 && slot_r < 40, kChkSharedIndex);
    __syncwarp();
    st.wtag[lane] = epoch;
    if (lane == 0) st.epoch = epoch;
#endif
    st.PQ[slot_pq] = make_double2(c.P, c.Q); st.R[slot_r] = c.R;
    __syncwarp();
    // task of this lane
    const int j = lane / kNumSeg, s = lane - j * kNumSeg;
    double val = 0.0;
#if defined(DHJ_CHECKED)
    for (int i = 0; i < kSeg; ++i) DHJ_CHECK(st.wtag[s * kSeg + i] == epoch, kChkReadBeforeWrite);
#endif
    if ((mask >> j) & 1u) {
      if (exact) fm::sincos_tab(u_of_k(pc, k0 + s * kSeg) * (it.x[j] - pc.a), ltab, &sn, &cs);
      else rotate(cs, sn, c32[j], s32[j]);
      double spq, sr;
      segment_sums<kSeg>(st.PQ + s * (kSeg + 1), reinterpret_cast<const Pair*>(st.R + s * (kSeg + 2)), cs, sn, cth[j],
                         sth[j], &spq, &sr);
      val = fma(it.K[j], sr, -(it.ex[j] * spq));
    }
    val += __shfl_xor_sync(kFullMask, val, 1);
    val += __shfl_xor_sync(kFullMask, val, 2);
    acc += val;                                              // meaningful in the lanes (j, 0) of active strikes
#if defined(DHJ_CHECKED)
    st.rtag[lane] = epoch;
#endif
  }
  // strike-independent sums of the pass, then the constant part of each strike
  const double A1 = any_call ? warp_sum(a1) : 0.0, A2 = any_call ? warp_sum(a2) : 0.0;
  const double A3 = any_put ? warp_sum(a3) : 0.0;
  __syncwarp();
  const double g0 = g0_keep;
  const int j = lane / kNumSeg;
  if ((mask >> j) & 1u)
    acc += strike_const_part((it.call_mask >> j) & 1u, it.S0, it.K[j], it.x[j], pc, A1, A2, A3, g0);
}

// phase 2 for a batch of `cnt_items` prepared items: warp w prices items w, w + 4, ... on its own — no block
// barrier, no partial sums in shared memory; sink(i, j, item, price) receives each price from lane 4 j.
// Strikes with their own (a, b) get an extra pass each (rare), set up by lane 0 in the warp's ExtraPass.
template <class Smem, class Sink>
__device__ __forceinline__ void run_batch(Smem& sm, const SliceView& v, int cnt_items, int tid,
                                          unsigned long long batch_tag, Sink sink) {
  // the shuffle tells ptxas that the warp index is warp-uniform: the item loop and everything addressed through it
  // then run on the uniform datapath (constants via LDCU into uniform registers, address arithmetic off the
  // vector pipe)
  const int warp = __shfl_sync(kFullMask, tid >> 5, 0), lane = tid & 31;
  ExtraPass& ex = sm.extra[warp];
#pragma unroll 1
  for (int i = warp; i < cnt_items; i += kBatchWarps) {
    const ItemRec& it = sm.items[i];
#if defined(DHJ_CHECKED)
    DHJ_CHECK(it.tag == batch_tag, kChkItemNotPrepared);
#endif
    double acc = 0.0;
    const unsigned reg_mask = it.valid_mask & ~it.bind_mask;
    if (reg_mask)
      contract_pass(it, it.pass, it.cth, it.sth, it.c32, it.s32, &it.cmu, reg_mask, v.n_cos, lane,
                    sm.stage[warp], &sm.ltab, acc);
    unsigned todo = it.valid_mask & it.bind_mask;            // uniform: the masks live in shared memory
    while (todo) {
      const int jb = __ffs(todo) - 1;
      todo &= todo - 1;
      __syncwarp();
      if (lane == 0) {
        ex.pass = make_pass_consts(it.set, py_min(it.pass.a, it.x[jb] - 0.1), py_max(it.pass.b, it.x[jb] + 0.1),
                                   it.pass.T);
        strike_rotation(ex.pass, it.x[jb], &ex.cth, &ex.sth, &ex.c32, &ex.s32);
        jump_rotation(ex.pass, it.set.mu, &ex.cmu, &ex.smu);
        ex.gj2 = fm::exp_neg(-2048.0 * jump_alpha(ex.pass, it.set.hsj2));
      }
      __syncwarp();
      // the task code indexes the rotation steps by strike: point it at the single extra entry
      double acc_b = 0.0;
      contract_pass(it, ex.pass, &ex.cth - jb, &ex.sth - jb, &ex.c32 - jb, &ex.s32 - jb, &ex.cmu, 1u << jb,
                    v.n_cos, lane, sm.stage[warp], &sm.ltab, acc_b);
      if ((lane >> 2) == jb) acc = acc_b;
    }
    const int j = lane >> 2;
    if ((lane & 3) == 0 && ((it.valid_mask >> j) & 1u)) sink(i, j, it, it.disc * acc);
  }
}

}  // namespace dhj
