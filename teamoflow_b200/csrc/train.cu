// Training-step kernels of the matrix-factorization hot path (HBM/L2-bound gather/scatter work).
//
//   user_pass_kernel : fused score + loss + dL/dscore + dE_u for one user per CTA   (tmf_user_pass)
//   spmm_seg_kernel  : deterministic segment-sum of scaled gathered rows            (tmf_spmm_seg)
//   adam1 / reductions / KL statistics / bias, relu, small fp32 GEMM
//
// No float atomics anywhere: every sum has a fixed association order, so results are
// bitwise reproducible run to run (north_star: "deterministic order").
#include <math.h>

#include <algorithm>

#include "common.cuh"

namespace tmf {

// =====================================================================================
// fused user-major pass
// =====================================================================================

struct UserPassParams {
  int ld, n_samples, s_pad;
  long long nnz;
  const int* row_ptr;
  const int* col_idx;
  const float* val;
  const float* Eu;
  const float* Ei;
  const int* samp;
  const int* work_user;   // optional work list: (user, [a, b) slice of its interactions, partial slot or -1)
  const int* work_a;
  const int* work_b;
  const int* work_slot;
  int n_work;
  float* part_G;          // [n_slots][s_pad] partial G of split users
  float* part_E;          // [n_slots][ld]    partial dE_u of split users (without the sample term)
  int* counter;
  float* loss_out;
  float* coef_out;
  const int* coef_pos;    // optional: coefficient slot e (c_k at k, G_uj at nnz + u S + j) is stored at coef_out[coef_pos[e]] -- the
                          // item-major order of the list the item pass streams, so that pass reads its coefficients coalesced
  float* dEu;
  float scale;  // n_items / n_samples (python true division, loss_graphs.py:86)
};

// where coefficient slot e is stored: coef_pos[e] when a slot map is given, e otherwise
__device__ __forceinline__ long long coef_slot(const int* coef_pos, long long e) { return coef_pos ? coef_pos[e] : e; }

// sums over the lane groups whose lane ids differ in bits >= `from` (xor tree: fixed order => deterministic)
__device__ __forceinline__ void xor_reduce(float2& a, int from) {
#pragma unroll
  for (int o = from; o < 32; o <<= 1) {
    a.x += __shfl_xor_sync(0xffffffffu, a.x, o);
    a.y += __shfl_xor_sync(0xffffffffu, a.y, o);
  }
}
__device__ __forceinline__ void xor_reduce(float4& a, int from) {
#pragma unroll
  for (int o = from; o < 32; o <<= 1) {
    a.x += __shfl_xor_sync(0xffffffffu, a.x, o);
    a.y += __shfl_xor_sync(0xffffffffu, a.y, o);
    a.z += __shfl_xor_sync(0xffffffffu, a.z, o);
    a.w += __shfl_xor_sync(0xffffffffu, a.w, o);
  }
}

template <int LPR, int VPL>
__device__ __forceinline__ void load_row(const float* __restrict__ base, long long row, int ld, int nv, int lg,
                                         float4 (&x)[VPL]) {
#pragma unroll
  for (int v = 0; v < VPL; ++v) {
    const int col = lg + LPR * v;
    x[v] = (col < nv) ? ldg4(base + row * ld + 4 * col) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

// Item-row gather for the hot loops: per-lane base pointers with the lane's column CLAMPED into the row (lanes past the
// row's end re-read its last 16 bytes; their user-row entries are zero and their results are never stored), so a row
// address is one 32x32+64-bit multiply-add and the load needs neither a predicate nor a zero fill.
template <int VPL>
__device__ __forceinline__ void load_item(const char* const (&lane_base)[VPL], int row, unsigned ld_bytes, float4 (&x)[VPL]) {
#pragma unroll
  for (int v = 0; v < VPL; ++v)
    x[v] = __ldg(reinterpret_cast<const float4*>(lane_base[v] + (unsigned long long)(unsigned)row * ld_bytes));
}

template <int VPL>
__device__ __forceinline__ float dotv(const float4 (&a)[VPL], const float4 (&b)[VPL]) {
  float s = dot4(a[0], b[0]);
#pragma unroll
  for (int v = 1; v < VPL; ++v) s += dot4(a[v], b[v]);
  return s;
}

constexpr int kUserPassThreads = 32;

// full-warp shuffles (constant mask, sub-warp width): every loop below is warp-uniform so that no variable-mask
// convergence checks (MATCH/REDUX/BRA.DIV, ~6 instructions per shuffle group) are generated
template <int LPR>
__device__ __forceinline__ float gsum(float v) {
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o, LPR);
  return v;
}

// One step of a reduce-scatter over a group of LPR lanes: of the sums lo and hi, the lane keeps lo if its bit o is clear
// and hi if it is set, and adds the partner lane's partial of that sum.  This adds the same two partial sums, in the same
// order, as gsum's step of offset o, so a reduce-scatter whose steps run over gsum's offsets gives every sum gsum's bits.
template <int LPR>
__device__ __forceinline__ float scatter_step(float lo, float hi, int o, bool up) {
  return (up ? hi : lo) + __shfl_xor_sync(0xffffffffu, up ? lo : hi, o, LPR);
}

// One WARP per work item (a CTA is one warp, up to 32 of them resident per SM): the phases of a user are separated by
// warp-level synchronisation only, and many users per SM are in flight in different phases.  (The first version gave a
// user to a 256-thread CTA: 4 CTAs per SM, five block barriers per user and shared-memory reductions over 16 row groups --
// 2.93 ms per C3 epoch against 1.9 ms for this layout.)
// JPL > 0 : each lane keeps JPL sample scores and JPL partial G sums in registers (S <= LPR*JPL)
// JPL == 0: MSE (no samples)
// JPL < 0 : generic WMRB, per-group G partials in shared memory
template <int LPR, int VPL, int JPL, int LOSS>
__global__ void __launch_bounds__(kUserPassThreads, (JPL >= 0 && JPL <= 8 && VPL == 1) ? 32 : 16)
user_pass_kernel(const UserPassParams p) {
  constexpr int NT = kUserPassThreads;
  static_assert(NT == 32, "one warp per work item");
  static_assert(JPL >= 0 || LPR == 32, "the generic WMRB path is only reached with 32 lanes per row");
  constexpr int NG = NT / LPR;
  constexpr int JH = JPL > 0 ? JPL / 2 : 1;
  constexpr int PD = (JPL >= 0 && JPL <= 4 && VPL == 1) ? 4 : 2;   // row buffers of the interaction loop
  constexpr unsigned FULL = 0xffffffffu;
  extern __shared__ __align__(16) float smem[];
  const int tid = threadIdx.x;
  const int g = tid / LPR;
  const int lg = tid % LPR;
  const int ld = p.ld;
  const int nv = ld >> 2;
  const int S = p.n_samples;
  float* sS = smem;                     // [s_pad]  sample scores, later final G_j
  float* sG = sS + p.s_pad;             // [NG][s_pad] per-group partial G (generic path only)
  // [2][NT] d and c of the interactions of the current batch, at their owner lanes' slots (shared memory rather than two
  // registers per lane across the interaction loop, which has none to spare)
  float* sDC = smem + (LOSS == TMF_LOSS_WMRB ? (1 + (JPL < 0 ? NG : 0)) * p.s_pad : 0);
  // [3] user and slot of the work item, then the next work item: warp-uniform values that wait in shared memory (every
  // lane stores the same value) while the sample scores and the interaction loop need the registers
  int* sItem = reinterpret_cast<int*>(sDC + 2 * NT);

  // work items come from an atomic counter; the NEXT item is claimed while the current one is processed, and its id
  // waits in shared memory
  if (tid == 0) sItem[2] = atomicAdd(p.counter, 1);
  for (;;) {
    __syncwarp();  // shared-memory reuse across work items
    const int t_work = sItem[2];
    if (t_work >= p.n_work) break;
    // a work item is a whole user or, for very heavy users, one slice of its interactions (load balance: a user
    // with millions of interactions would otherwise be one CTA's serial tail)
    int u = p.work_user ? p.work_user[t_work] : t_work;
    const int a = p.work_user ? p.work_a[t_work] : p.row_ptr[u];
    const int b = p.work_user ? p.work_b[t_work] : p.row_ptr[u + 1];
    int slot = p.work_user ? p.work_slot[t_work] : -1;

    if (a == b) {  // no interactions: all gradients of this user are zero
      __syncwarp();  // every lane has read this item's id
      if (tid == 0) sItem[2] = atomicAdd(p.counter, 1);
      if (LOSS == TMF_LOSS_WMRB)
        for (int j = tid; j < S; j += NT) p.coef_out[coef_slot(p.coef_pos, p.nnz + (long long)u * S + j)] = 0.f;
      for (int c = tid; c < ld; c += NT) p.dEu[(long long)u * ld + c] = 0.f;
      continue;
    }

    sItem[0] = u;
    sItem[1] = slot;
    float4 eu[VPL];
    load_row<LPR, VPL>(p.Eu, u, ld, nv, lg, eu);  // zero past the row's end
    const char* ei_lane[VPL];
#pragma unroll
    for (int v = 0; v < VPL; ++v) {
      ei_lane[v] = reinterpret_cast<const char*>(p.Ei) + 16 * min(lg + LPR * v, nv - 1);
      // kept in registers (the 64-register variants would rebuild it from p.Ei, four instructions per row gather)
      if constexpr (VPL == 1) asm("" : "+l"(ei_lane[v]));
    }
    const unsigned ld_bytes = 4u * (unsigned)ld;

    // When many samples force the hinge layout's LPR above the row width (S > 16 * row lanes), the two phases that only
    // gather sample rows work in narrower sub-groups of SW lanes (the narrowest power of two >= 4 covering a row), so
    // 32 / SW rows are gathered per load instruction instead of one.
    // (The dispatcher only widens LPR when S / LPR > 16, which lands in the JPL = 16 or generic variants: the others
    // do not carry this path and keep their registers.)
    constexpr bool NARROW_OK = (JPL == 16 || JPL < 0) && VPL == 1 && LPR > 4;
    int SW = LPR;
    if constexpr (NARROW_OK) {
      while (SW > 4 && (SW >> 1) >= nv) SW >>= 1;
    }
    const bool narrow = NARROW_OK && SW < LPR;  // warp-uniform
    const int sl = tid & (SW - 1), sg = tid / SW, NSG = 32 / SW;
    const char* ei_sub = reinterpret_cast<const char*>(p.Ei) + 16 * min(sl, nv - 1);

    float2 sj2[JH];  // this lane's sample scores, two per register pair (FADD2 / FFMA2 operands)
    float2 gj2[JH];  // ... and its partial G sums
    if constexpr (LOSS == TMF_LOSS_WMRB) {
      const int* su = p.samp + (long long)u * S;
      if (NARROW_OK && narrow) {
        const float4 eus = (sl < nv) ? ldg4(p.Eu + (long long)u * ld + 4 * sl) : make_float4(0.f, 0.f, 0.f, 0.f);
        const int n_sit = (S + NSG * 4 - 1) / (NSG * 4);
        for (int it = 0; it < n_sit; ++it) {
          const int j0 = (it * NSG + sg) * 4;
          int idx[4];
          float4 row[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) idx[q] = (j0 + q < S) ? su[j0 + q] : 0;
#pragma unroll
          for (int q = 0; q < 4; ++q)
            row[q] = __ldg(reinterpret_cast<const float4*>(ei_sub + (unsigned long long)(unsigned)idx[q] * ld_bytes));
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            float sc = dot4(eus, row[q]);
            for (int o = SW >> 1; o > 0; o >>= 1) sc += __shfl_xor_sync(FULL, sc, o);
            if (j0 + q < S && sl == 0) sS[j0 + q] = sc;
          }
        }
      } else {
        // 32 samples per round: group g scores samples j0 + g LPR + r, r < LPR.  The round's sample ids are one coalesced
        // load, handed to the group's lanes by shuffle.  The scores are summed by a reduce-scatter over the group (offsets
        // LPR / 2, ..., 1, gsum's order): afterwards lane lg holds the score of sample j0 + g LPR + lg = j0 + tid, and the
        // warp stores the round's 32 scores with one instruction.  The steps down to offset P run as the U rows of samples
        // r, r + P, ... arrive, so P partial sums are live at a time.
        for (int j0 = 0; j0 < S; j0 += 32) {
          constexpr int P = LPR / 2 < 8 ? LPR / 2 : 8;
          constexpr int U = LPR / P;
          const int my_id = (j0 + tid < S) ? su[j0 + tid] : 0;
          float part[P];
#pragma unroll
          for (int r = 0; r < P; ++r) {
            float x[U];
#pragma unroll
            for (int t = 0; t < U; ++t) {
              float4 row[VPL];
              load_item<VPL>(ei_lane, __shfl_sync(FULL, my_id, r + t * P, LPR), ld_bytes, row);
              x[t] = dotv<VPL>(eu, row);
            }
#pragma unroll
            for (int o = LPR / 2, n = U / 2; o >= P; o >>= 1, n >>= 1)
#pragma unroll
              for (int t = 0; t < n; ++t) x[t] = scatter_step<LPR>(x[t], x[t + n], o, lg & o);
            part[r] = x[0];
          }
#pragma unroll
          for (int o = P / 2; o > 0; o >>= 1)
#pragma unroll
            for (int r = 0; r < o; ++r) part[r] = scatter_step<LPR>(part[r], part[r + o], o, lg & o);
          if (j0 + tid < S) sS[j0 + tid] = part[0];
        }
      }
      if constexpr (JPL < 0) {
        for (int j = lg; j < S; j += LPR) sG[g * p.s_pad + j] = 0.f;
      }
      __syncwarp();
      if constexpr (JPL > 0) {
        // padding slots hold a large negative FINITE score: their hinge is negative, so the indicator is 0 and
        // 0 * h stays a (signed) zero in the FFMA2 below (an infinity would turn it into NaN)
#pragma unroll
        for (int t = 0; t < JH; ++t) {
          const int j0 = lg + LPR * (2 * t), j1 = lg + LPR * (2 * t + 1);
          sj2[t] = make_float2((j0 < S) ? sS[j0] : -1e30f, (j1 < S) ? sS[j1] : -1e30f);
          gj2[t] = make_float2(0.f, 0.f);
        }
      }
    }

    float4 acc[VPL];
#pragma unroll
    for (int v = 0; v < VPL; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);

    // ---- interactions of this user, strided over the NG row groups; warp-uniform trip count.  One interaction per
    // row group and iteration: score, S hinge terms (each lane owns JPL of them, evaluated two at a time with packed
    // fp32x2 instructions), dL/dscore, and acc += c * row while the row is still in registers.  Returns d (1 + m for
    // WMRB, the squared error for MSE) and c in every lane of the group.
    auto process = [&](const float4 (&row)[VPL], const float a_k, const bool active, float& d, float& c) {
      const float pk = gsum<LPR>(dotv<VPL>(eu, row));
      c = 0.f;
      d = 0.f;
      if constexpr (LOSS == TMF_LOSS_MSE) {
        const float df = a_k - pk;  // loss_graphs.py:52
        d = df * df;
        c = active ? -2.0f * df : 0.f;
      } else {
        const float base = __fsub_rn(1.0f, pk);
        const bool pos = active && a_k > 0.f;  // loss_graphs.py:74
        float sum, cnt;
        if constexpr (JPL > 0) {
          const float2 base2 = make_float2(base, base);
          float2 ind2[JH];
          float2 sum2 = make_float2(0.f, 0.f), cnt2 = make_float2(0.f, 0.f);
#pragma unroll
          for (int t = 0; t < JH; ++t) {
            const float2 h2 = fadd2(base2, sj2[t]);             // (1 - p) + s, loss_graphs.py:84
            ind2[t] = make_float2(h2.x >= 0.f ? 1.f : 0.f,      // tf.maximum(h, 0): value h and gradient 1 when h >= 0
                                  h2.y >= 0.f ? 1.f : 0.f);
            sum2 = ffma2(ind2[t], h2, sum2);                    // 1 * h + sum rounds once, like the plain add
            cnt2 = fadd2(cnt2, ind2[t]);
          }
          float2 sc = make_float2(sum2.x + sum2.y, cnt2.x + cnt2.y);
#pragma unroll
          for (int o = LPR / 2; o > 0; o >>= 1)
            sc = fadd2(sc, make_float2(__shfl_xor_sync(0xffffffffu, sc.x, o, LPR), __shfl_xor_sync(0xffffffffu, sc.y, o, LPR)));
          sum = sc.x;
          cnt = sc.y;
          const float m = p.scale * sum;                 // :86
          d = __fadd_rn(1.0f, m);                        // >= 1: m is a sum of non-negative terms
          const float w = pos ? p.scale * rcp_approx(d) : 0.f;
          c = -w * cnt;
          const float2 w2 = make_float2(w, w);
#pragma unroll
          for (int t = 0; t < JH; ++t) gj2[t] = ffma2(ind2[t], w2, gj2[t]);
          if (!pos) d = 1.0f;                            // log(1) = 0: no loss for non-positive interactions
        } else {
          sum = 0.f;
          cnt = 0.f;
          for (int j = lg; j < S; j += LPR) {
            const float h = __fadd_rn(base, sS[j]);
            sum += fmaxf(h, 0.f);
            cnt += (h >= 0.f) ? 1.f : 0.f;
          }
          sum = gsum<LPR>(sum);
          cnt = gsum<LPR>(cnt);
          const float m = p.scale * sum;
          d = __fadd_rn(1.0f, m);
          const float w = pos ? __fdividef(p.scale, d) : 0.f;
          c = -w * cnt;
          if (pos) {
            for (int j = lg; j < S; j += LPR) {
              const float h = __fadd_rn(base, sS[j]);
              if (h >= 0.f) sG[g * p.s_pad + j] += w;
            }
          }
          if (!pos) d = 1.0f;
        }
      }
#pragma unroll
      for (int v = 0; v < VPL; ++v) fma4(acc[v], c, row[v]);
    };
    // Iteration it of group g is interaction a + it NG + g.  The iterations run in batches of LPR: in the batch that starts
    // at iteration it0, lane lg of group g owns iteration it0 + lg.  It holds that interaction's value (one coalesced load
    // for the warp's 32 interactions), the group parks the interaction's d and c at the lane's slots of sDC, and once the
    // batch is done the lane stores log(d) (one coalesced store for the warp) and c.  Item ids are held the same way PD - 1
    // iterations ahead (lane lg: iteration it0 + PD - 1 + lg), and the next batch's ids and values are loaded when a batch
    // starts.
    // Software pipeline over PD row buffers: a row is gathered PD - 1 iterations before it is used, so the row's L2 / HBM
    // latency does not sit on the critical path (PD = 4 where the registers allow it: with a 1 GB item table the rows come
    // from HBM and one row in flight per warp would leave the memory system idle).  Iteration i uses buffer i % PD; the
    // loop is unrolled PD times so the buffers are addressed statically (no register copies).  Interactions past the
    // slice are clamped (a tail iteration re-reads the last row and is masked by `active`).
    {
      const int n_it = (b - a + NG - 1) / NG;
      const int n_git = (b - a - g + NG - 1) / NG;  // iterations in which this group has an interaction
      auto clamped = [&](int it) { return min(a + it * NG + g, b - 1); };
      float4 rows[PD][VPL];
#pragma unroll
      for (int q = 0; q < PD - 1; ++q) load_item<VPL>(ei_lane, p.col_idx[clamped(q)], ld_bytes, rows[q]);
      int nxt_id = p.col_idx[clamped(PD - 1 + lg)];
      float nxt_v = p.val[clamped(lg)];
      // shared-memory address of the group's d and c slots, held in a register (rebuilding it costs more than the register)
      unsigned dc_g = (unsigned)__cvta_generic_to_shared(sDC + g * LPR);
      asm("" : "+r"(dc_g));
      for (int it0 = 0; it0 < n_it; it0 += LPR) {
        const int cur_id = nxt_id;
        const float cur_v = nxt_v;
        nxt_id = p.col_idx[clamped(it0 + LPR + PD - 1 + lg)];
        nxt_v = p.val[clamped(it0 + LPR + lg)];
        const int n_in = min(LPR, n_it - it0);
        const int n_act = n_git - it0;  // iterations it0 + i of this group with i < n_act are in the slice
        __syncwarp();  // the previous batch's d and c have been read
        for (int i = 0; i < n_in; i += PD) {
#pragma unroll
          for (int q = 0; q < PD; ++q) {
            if (q == 0 || i + q < n_in) {  // warp-uniform
              load_item<VPL>(ei_lane, __shfl_sync(FULL, cur_id, i + q, LPR), ld_bytes, rows[(q + PD - 1) % PD]);
              float d, c;
              process(rows[q], __shfl_sync(FULL, cur_v, i + q, LPR), i + q < n_act, d, c);
              // every lane of the group holds d and c: all write the same value to the owner's slots
              asm volatile("st.shared.f32 [%0], %1;" ::"r"(dc_g + 4 * (i + q)), "f"(d) : "memory");
              asm volatile("st.shared.f32 [%0], %1;" ::"r"(dc_g + 4 * (NT + i + q)), "f"(c) : "memory");
            }
          }
        }
        __syncwarp();  // the group's stores of d and c are visible to their owner lanes
        if (lg < n_act) {
          // (coef_pos is read here rather than with the batch's values: the loop above has no register to keep it in)
          const int k_own = a + (it0 + lg) * NG + g;
          const float d = sDC[tid];
          p.loss_out[k_own] = LOSS == TMF_LOSS_WMRB ? logf(d) : d;  // log(1 + m), loss_graphs.py:88
          p.coef_out[coef_slot(p.coef_pos, k_own)] = sDC[NT + tid];
        }
      }
    }

    u = sItem[0];
    slot = sItem[1];

    const int* cpos = p.coef_pos;
    if constexpr (LOSS == TMF_LOSS_WMRB) {
      __syncwarp();  // sS (sample scores of the generic path) is no longer read
      // A whole user's G_uj is final and goes to its coefficient slot; a slice's is a partial sum, written to its part_G
      // row and added up by the fix-up kernel.  sS keeps G for the sample term below.  (The JPL > 0 store stays split by
      // destination: a single store through a selected pointer costs the 64-register variants extra spill bytes.)
      if constexpr (JPL > 0) {
        // G_j = sum of the row groups' partial sums
#pragma unroll
        for (int t = 0; t < JH; ++t) {
          xor_reduce(gj2[t], LPR);
          if (g == 0) {
            const int j0 = lg + LPR * (2 * t), j1 = lg + LPR * (2 * t + 1);
            if (slot < 0) {
              const long long e0 = p.nnz + (long long)u * S;
              if (j0 < S) { p.coef_out[coef_slot(cpos, e0 + j0)] = gj2[t].x; sS[j0] = gj2[t].x; }
              if (j1 < S) { p.coef_out[coef_slot(cpos, e0 + j1)] = gj2[t].y; sS[j1] = gj2[t].y; }
            } else {
              float* dst = p.part_G + (long long)slot * p.s_pad;
              if (j0 < S) { dst[j0] = gj2[t].x; sS[j0] = gj2[t].x; }
              if (j1 < S) { dst[j1] = gj2[t].y; sS[j1] = gj2[t].y; }
            }
          }
        }
      } else {
        for (int j = tid; j < S; j += NT) {  // fixed group order => deterministic
          float G = sG[j];
          for (int gg = 1; gg < NG; ++gg) G += sG[gg * p.s_pad + j];
          if (slot < 0) p.coef_out[coef_slot(cpos, p.nnz + (long long)u * S + j)] = G;
          else p.part_G[(long long)slot * p.s_pad + j] = G;
          sS[j] = G;
        }
      }
      __syncwarp();
      const int* su = p.samp + (long long)u * S;
      if (NARROW_OK && narrow) {
        float4 accg = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
        for (int j = (slot < 0 ? sg : S); j < S; j += NSG)
          fma4(accg, sS[j], __ldg(reinterpret_cast<const float4*>(ei_sub + (unsigned long long)(unsigned)su[j] * ld_bytes)));
        xor_reduce(accg, SW);  // over the sub-groups
        if (g == 0 && lg < SW) add4(acc[0], accg);  // lane lg < SW owns column lg in both layouts
      } else {
#pragma unroll 4
        for (int j = (slot < 0 ? g : S); j < S; j += NG) {  // split users: the sample term is added once, in the fix-up
          const float G = sS[j];
          float4 row[VPL];
          load_item<VPL>(ei_lane, su[j], ld_bytes, row);
#pragma unroll
          for (int v = 0; v < VPL; ++v) fma4(acc[v], G, row[v]);
        }
      }
    }

    if (tid == 0) sItem[2] = atomicAdd(p.counter, 1);

    // ---- dE_u[u] = sum over the row groups
#pragma unroll
    for (int v = 0; v < VPL; ++v) {
      xor_reduce(acc[v], LPR);
      const int col = lg + LPR * v;
      if (g == 0 && col < nv) {
        float* dst = slot < 0 ? p.dEu + (long long)u * ld : p.part_E + (long long)slot * ld;
        reinterpret_cast<float4*>(dst)[col] = acc[v];
      }
    }
  }
}

// One CTA per split user: G = sum of the slices' partial G (slice order), dE_u = sum of the slices' partial dE_u
// (slice order) + sum_j G_j * E_i[J_uj].  Fixed association order => deterministic.
__global__ void __launch_bounds__(256) user_fixup_kernel(const UserPassParams p, int loss, int n_split, const int* __restrict__ split_user,
                                                         const int* __restrict__ split_first, const int* __restrict__ split_nseg) {
  extern __shared__ __align__(16) float fsm[];
  float* sG = fsm;            // [s_pad]
  float* sE = sG + p.s_pad;   // [ld]
  float* sP = sE + p.ld;      // [256 / nvp][ld] partial sample terms
  const int tid = threadIdx.x;
  const int nv = p.ld >> 2;
  int nvp = 4;
  while (nvp < nv) nvp <<= 1;  // <= 64 (ld <= 256)
  for (int w = blockIdx.x; w < n_split; w += gridDim.x) {
    const int u = split_user[w], first = split_first[w], nseg = split_nseg[w];
    const int S = p.n_samples;
    __syncthreads();
    if (loss == TMF_LOSS_WMRB) {
      for (int j = tid; j < S; j += 256) {
        float G = 0.f;
        for (int sg = 0; sg < nseg; ++sg) G += p.part_G[(long long)(first + sg) * p.s_pad + j];
        p.coef_out[coef_slot(p.coef_pos, p.nnz + (long long)u * S + j)] = G;
        sG[j] = G;
      }
    }
    for (int c = tid; c < p.ld; c += 256) {
      float s = 0.f;
      for (int sg = 0; sg < nseg; ++sg) s += p.part_E[(long long)(first + sg) * p.ld + c];
      sE[c] = s;
    }
    __syncthreads();
    if (loss == TMF_LOSS_WMRB) {  // sample term: the 256 threads form NP sub-groups of nvp lanes, sub-group jp takes samples jp, jp + NP, ...
      const int* su = p.samp + (long long)u * S;
      const int c4 = tid & (nvp - 1), jp = tid / nvp, NP = 256 / nvp;
      float4 a4 = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c4 < nv) {
#pragma unroll 4
        for (int j = jp; j < S; j += NP) fma4(a4, sG[j], ldg4(p.Ei + (long long)su[j] * p.ld + 4 * c4));
        reinterpret_cast<float4*>(sP + jp * p.ld)[c4] = a4;
      }
      __syncthreads();
      for (int c = tid; c < p.ld; c += 256) {
        float s = sE[c];
        for (int q = 0; q < NP; ++q) s += sP[q * p.ld + c];  // fixed order
        p.dEu[(long long)u * p.ld + c] = s;
      }
    } else {
      for (int c = tid; c < p.ld; c += 256) p.dEu[(long long)u * p.ld + c] = sE[c];
    }
  }
}

template <int LPR, int VPL, int JPL, int LOSS>
static int launch_user_pass(const UserPassParams& p, cudaStream_t st) {
  constexpr int NG = kUserPassThreads / LPR;
  auto kern = user_pass_kernel<LPR, VPL, JPL, LOSS>;
  size_t smem = (2 * kUserPassThreads + 4) * sizeof(float);  // sDC, sItem
  if (LOSS == TMF_LOSS_WMRB) smem += (size_t)(1 + (JPL < 0 ? NG : 0)) * p.s_pad * sizeof(float);
  UserPassParams q = p;
  TMF_REQUIRE(smem <= 200 * 1024, "tmf_user_pass: n_samples=%d too large for shared memory (%zu B)", p.n_samples, smem);
  if (smem > 48 * 1024) TMF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 1;
  TMF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kUserPassThreads, smem));
  if (occ < 1) occ = 1;
  long long grid = (long long)kNumSMs * occ;
  if (grid > p.n_work) grid = p.n_work;
  TMF_CUDA(cudaMemsetAsync(p.counter, 0, sizeof(int), st));
  kern<<<(unsigned)grid, kUserPassThreads, smem, st>>>(q);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

template <int LPR, int VPL>
static int dispatch_user_pass_j(const UserPassParams& p, int loss, cudaStream_t st) {
  if (loss == TMF_LOSS_MSE) return launch_user_pass<LPR, VPL, 0, TMF_LOSS_MSE>(p, st);
  const int jpl = (p.n_samples + LPR - 1) / LPR;
  if (jpl <= 2) return launch_user_pass<LPR, VPL, 2, TMF_LOSS_WMRB>(p, st);
  if (jpl <= 4) return launch_user_pass<LPR, VPL, 4, TMF_LOSS_WMRB>(p, st);
  if (jpl <= 8) return launch_user_pass<LPR, VPL, 8, TMF_LOSS_WMRB>(p, st);
  if (jpl <= 16) return launch_user_pass<LPR, VPL, 16, TMF_LOSS_WMRB>(p, st);
  // tmf_user_pass widens LPR to 32 before ceil(S / LPR) exceeds 16, so only LPR = 32 gets here and only that generic
  // kernel is compiled
  TMF_REQUIRE(LPR == 32, "tmf_user_pass: %d samples at %d lanes per row need a generic kernel that is not compiled",
              p.n_samples, LPR);
  if constexpr (LPR == 32) return launch_user_pass<LPR, VPL, -1, TMF_LOSS_WMRB>(p, st);
  else return TMF_E_INVALID;
}

// =====================================================================================
// deterministic segment-sum of scaled gathered rows
// =====================================================================================

constexpr int kSpmmThreads = 256;

struct SpmmParams {
  int n_seg, ld_src, ld_out, nv, chunk;
  long long n_entries;
  const int* seg_ptr;
  const int* idx;
  const int* cpos;
  const float* coef;
  const float* src;
  float* out;
  float* part_first;  // [n_chunks][ld_out]
  float* part_carry;  // [n_chunks][ld_out]
};

// acc += c * row for the NB entries t .. t + NB - 1 of the batch the group holds (lane t: index my_i, coefficient my_c):
// NB row gathers in flight, summed in entry order
template <int NB, int LPR>
__device__ __forceinline__ void seg_batch(float4& acc, const float* src_lane, unsigned long long ld_src, unsigned gm, int my_i,
                                          float my_c, int t) {
  int i[NB];
  float c[NB];
  float4 r[NB];
#pragma unroll
  for (int q = 0; q < NB; ++q) {
    i[q] = __shfl_sync(gm, my_i, t + q, LPR);
    c[q] = __shfl_sync(gm, my_c, t + q, LPR);
  }
#pragma unroll
  for (int q = 0; q < NB; ++q) r[q] = ldg4(src_lane + (unsigned long long)(unsigned)i[q] * ld_src);
#pragma unroll
  for (int q = 0; q < NB; ++q) fma4(acc, c[q], r[q]);
}

// group `gid` owns entries [gid*chunk, (gid+1)*chunk); walks the segments that intersect it.
template <int LPR>
__global__ void __launch_bounds__(kSpmmThreads) spmm_seg_kernel(const SpmmParams p) {
  const int lg = threadIdx.x % LPR;
  const unsigned gm = group_mask<LPR>();
  const long long gid = ((long long)blockIdx.x * kSpmmThreads + threadIdx.x) / LPR;
  const long long cs = gid * p.chunk;
  if (cs >= p.n_entries) return;
  const long long ce = min(cs + (long long)p.chunk, p.n_entries);
  const int col = blockIdx.y * LPR + lg;  // float4 column
  const bool active = col < p.nv;

  // last segment s with seg_ptr[s] <= cs  (upper_bound - 1)
  int lo = 0, hi = p.n_seg;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if ((long long)p.seg_ptr[mid] <= cs) lo = mid; else hi = mid - 1;
  }
  int s = lo;
  long long sb = p.seg_ptr[s + 1];
  while (sb <= cs) { ++s; sb = p.seg_ptr[s + 1]; }  // skip empty segments
  long long sa = p.seg_ptr[s];
  const float* src_lane = p.src + 4 * min(col, p.nv - 1);  // clamped column: inactive lanes re-read a valid one, never store
  const unsigned long long ld_src = (unsigned long long)p.ld_src;

  // Entries are fetched a batch of LPR ahead (lane t of the group holds entry base + t: index and coefficient), so the
  // index -> coefficient -> row dependency of the NEXT batch resolves while the rows of the current one are gathered;
  // rows are gathered eight at a time.  Sums run in entry order: bitwise deterministic.
  auto fetch = [&](long long base, int& my_i, float& my_c) {
    const long long e = base + lg;
    my_i = 0;
    my_c = 0.f;
    if (e < ce) {
      my_i = p.idx[e];
      my_c = p.coef ? p.coef[coef_slot(p.cpos, e)] : 1.0f;
    }
  };
  int nxt_i;
  float nxt_c;
  fetch(cs, nxt_i, nxt_c);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (long long base = cs; base < ce; base += LPR) {
    const int my_i = nxt_i;
    const float my_c = nxt_c;
    fetch(base + LPR, nxt_i, nxt_c);
    const int nb = (int)min((long long)LPR, ce - base);
    int t = 0;
    while (t < nb) {
      const int te = (int)min((long long)nb, sb - base);  // entries of this batch that belong to segment s
      for (; t + 8 <= te; t += 8) seg_batch<8, LPR>(acc, src_lane, ld_src, gm, my_i, my_c, t);
      if (t + 4 <= te) {
        seg_batch<4, LPR>(acc, src_lane, ld_src, gm, my_i, my_c, t);
        t += 4;
      }
      for (; t < te; ++t) seg_batch<1, LPR>(acc, src_lane, ld_src, gm, my_i, my_c, t);
      if (base + t == sb || base + t == ce) {  // segment (or this chunk's part of it) complete
        if (active) {
          float* dst;
          if (sa >= cs && sb <= ce) dst = p.out + (long long)s * p.ld_out;
          else if (sa < cs) dst = p.part_first + gid * p.ld_out;
          else dst = p.part_carry + gid * p.ld_out;
          reinterpret_cast<float4*>(dst)[col] = acc;
        }
        acc = make_float4(0.f, 0.f, 0.f, 0.f);
        if (base + t < ce) {
          ++s;
          sb = p.seg_ptr[s + 1];
          while (sb <= base + t) { ++s; sb = p.seg_ptr[s + 1]; }  // skip empty segments
          sa = p.seg_ptr[s];
        }
      }
    }
  }
}

// one group per segment: zero-fill empty segments, combine the partials of chunk-spanning ones
template <int LPR>
__global__ void __launch_bounds__(kSpmmThreads) spmm_fixup_kernel(const SpmmParams p) {
  const int lg = threadIdx.x % LPR;
  const long long s = ((long long)blockIdx.x * kSpmmThreads + threadIdx.x) / LPR;
  if (s >= p.n_seg) return;
  const int col = blockIdx.y * LPR + lg;
  if (col >= p.nv) return;
  const long long a = p.seg_ptr[s], b = p.seg_ptr[s + 1];
  float4* dst = reinterpret_cast<float4*>(p.out + s * p.ld_out) + col;
  if (a == b) {
    *dst = make_float4(0.f, 0.f, 0.f, 0.f);
    return;
  }
  const long long c0 = a / p.chunk, c1 = (b - 1) / p.chunk;
  if (c0 == c1) return;
  float4 acc = reinterpret_cast<const float4*>(p.part_carry + c0 * p.ld_out)[col];
  for (long long c = c0 + 1; c <= c1; ++c) add4(acc, reinterpret_cast<const float4*>(p.part_first + c * p.ld_out)[col]);
  *dst = acc;
}

static int spmm_chunk_for(long long n_entries) {
  // enough groups to fill the machine (~148 SMs x 2048 threads / 16 lanes), bounded partial buffers
  long long c = n_entries / 32768;
  int chunk = 32;
  while (chunk < c && chunk < 256) chunk <<= 1;
  return chunk;
}

template <int LPR>
static int launch_spmm(const SpmmParams& p, cudaStream_t st) {
  const long long n_chunks = cdiv(p.n_entries, p.chunk);
  const int gpb = kSpmmThreads / LPR;
  dim3 grid_y((unsigned)1, (unsigned)cdiv(p.nv, LPR));
  if (n_chunks > 0) {
    dim3 grid((unsigned)cdiv(n_chunks, gpb), grid_y.y);
    spmm_seg_kernel<LPR><<<grid, kSpmmThreads, 0, st>>>(p);
    TMF_LAUNCH_CHECK();
  }
  if (p.n_seg > 0) {
    dim3 grid((unsigned)cdiv(p.n_seg, gpb), grid_y.y);
    spmm_fixup_kernel<LPR><<<grid, kSpmmThreads, 0, st>>>(p);
    TMF_LAUNCH_CHECK();
  }
  return TMF_OK;
}

// =====================================================================================
// elementwise / reductions
// =====================================================================================

// 128-bit accesses over the 16-byte aligned body (n4 float4 groups), scalar tail
__global__ void adam1_kernel(float* __restrict__ w, const float* __restrict__ g, long long n, float lr, int vec) {
  const float alpha = adam1_alpha(lr);
  const long long n4 = vec ? (n >> 2) : 0;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  float4* w4 = reinterpret_cast<float4*>(w);
  const float4* g4 = reinterpret_cast<const float4*>(g);
  for (long long q = i; q < n4; q += stride) {
    const float4 gv = __ldcs(g4 + q);  // the gradient is dead after this read
    float4 wv = w4[q];
    wv.x = adam1_apply(wv.x, gv.x, alpha);
    wv.y = adam1_apply(wv.y, gv.y, alpha);
    wv.z = adam1_apply(wv.z, gv.z, alpha);
    wv.w = adam1_apply(wv.w, gv.w, alpha);
    w4[q] = wv;
  }
  for (long long q = 4 * n4 + i; q < n; q += stride) w[q] = adam1_apply(w[q], g[q], alpha);
}

__global__ void adam_kernel(float* __restrict__ w, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                            long long n, float alpha) {
  const float b1 = 0.9f, b2 = 0.999f, eps = 1e-7f;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    const float gi = g[i];
    const float mi = b1 * m[i] + gi * (1.0f - b1);
    const float vi = b2 * v[i] + (gi * gi) * (1.0f - b2);
    m[i] = mi;
    v[i] = vi;
    w[i] = w[i] - __fdiv_rn(alpha * mi, sqrtf(vi) + eps);
  }
}

__global__ void pair_dots_kernel(long long nnz, const int* __restrict__ rows, const int* __restrict__ cols,
                                 const float* __restrict__ Eu, const float* __restrict__ Ei, int ld, float* __restrict__ p) {
  // 8 lanes per pair, float4 strided over the row
  const int lg = threadIdx.x & 7;
  const unsigned gm = group_mask<8>();
  const long long k = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 3;
  if (k >= nnz) return;
  const float* a = Eu + (long long)rows[k] * ld;
  const float* b = Ei + (long long)cols[k] * ld;
  float s = 0.f;
  for (int c = lg; c < (ld >> 2); c += 8) s += dot4(ldg4(a + 4 * c), ldg4(b + 4 * c));
  s = group_sum<8>(s, gm);
  if (lg == 0) p[k] = s;
}

constexpr int kRedBlocks = 1024;
constexpr int kRedThreads = 256;

template <int NV>
__device__ __forceinline__ void block_reduce_store(double (&v)[NV], double* out) {
  __shared__ double sm[NV][kRedThreads / 32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    double x = v[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if (lane == 0) sm[i][w] = x;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      double x = 0.0;
      for (int j = 0; j < kRedThreads / 32; ++j) x += sm[i][j];
      out[i] = x;
    }
  }
}

// Reduction modes and the number of fp64 sums each one produces per block:
//   kRedSum: sum(x)    kRedSumSq: sum(x^2)
//   kRedKLMoments: KL raw moments {cnt+, sum+, sumsq+, cnt-, sum-, sumsq-}, additive over user shards
enum RedMode { kRedSum, kRedSumSq, kRedKLMoments };
template <int MODE>
constexpr int kRedWidth = MODE == kRedKLMoments ? 6 : 1;
constexpr int kRedMaxWidth = std::max({kRedWidth<kRedSum>, kRedWidth<kRedSumSq>, kRedWidth<kRedKLMoments>});
// reduce workspace: kRedStats doubles of statistics, then up to kRedBlocks partial rows of the widest mode
constexpr int kRedStats = 16;

template <int MODE>
__global__ void __launch_bounds__(kRedThreads) reduce_partial_kernel(const float* __restrict__ x, const float* __restrict__ val,
                                                                    long long n, double* __restrict__ partial) {
  constexpr int NV = kRedWidth<MODE>;
  double v[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = 0.0;
  const long long per = (n + gridDim.x - 1) / gridDim.x;
  const long long lo = per * blockIdx.x, hi = min(lo + per, n);
  for (long long i = lo + threadIdx.x; i < hi; i += kRedThreads) {
    const double xi = x[i];
    if (MODE == kRedSum) v[0] += xi;
    if (MODE == kRedSumSq) v[0] += xi * xi;
    if (MODE == kRedKLMoments) {
      if (val[i] > 0.f) { v[0] += 1.0; v[1] += xi; v[2] += xi * xi; } else { v[3] += 1.0; v[4] += xi; v[5] += xi * xi; }
    }
  }
  block_reduce_store<NV>(v, partial + (long long)blockIdx.x * NV);
}

// kRedSum: out_f[0] = sum    kRedSumSq: scale = rsqrt(max(sum, 1e-12)) -> stats[0]
// kRedKLMoments: the six sums -> stats[0..5], nothing derived
template <int MODE>
__global__ void __launch_bounds__(kRedThreads) reduce_final_kernel(const double* __restrict__ partial, int n_blocks,
                                                                  double* __restrict__ stats, float* __restrict__ out_f) {
  constexpr int NV = kRedWidth<MODE>;
  double v[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = 0.0;
  for (int b = threadIdx.x; b < n_blocks; b += kRedThreads)
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] += partial[(long long)b * NV + i];
  __shared__ double res[NV];
  block_reduce_store<NV>(v, res);
  __syncthreads();
  if (threadIdx.x == 0) {
    if (MODE == kRedSum) out_f[0] = (float)res[0];
    if (MODE == kRedSumSq) stats[0] = 1.0 / sqrt(fmax(res[0], 1e-12));
    if (MODE == kRedKLMoments) {
#pragma unroll
      for (int i = 0; i < NV; ++i) stats[i] = res[i];
    }
  }
}

// KL statistics from the six raw moments m = {n+, S+, Q+, n-, S-, Q-} (summed over the ranks under user sharding): means
// rounded to fp32 like tf.nn.moments, population variances about those means (Q - 2 mu S + n mu^2, fp64), s, z, phi and
// the scalar loss.
__global__ void kl_from_moments_kernel(const double* __restrict__ m, double* __restrict__ stats, float* __restrict__ out_f) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const double np_ = m[0], nn_ = m[3];
  const double mp = (double)(float)(m[1] / np_), mn = (double)(float)(m[4] / nn_);
  const float vp = (float)((m[2] - 2.0 * mp * m[1] + np_ * mp * mp) / np_);
  const float vn = (float)((m[5] - 2.0 * mn * m[4] + nn_ * mn * mn) / nn_);
  const float s = sqrtf(vp + vn);
  const float z = ((float)mp - (float)mn) / s;
  const float phi = expf(-0.5f * z * z) * 0.3989422804014327f;
  stats[0] = mp; stats[1] = mn; stats[2] = np_; stats[3] = nn_;
  stats[4] = s; stats[5] = z; stats[6] = phi;
  out_f[0] = 1.0f - 0.5f * erfcf(-z * 0.7071067811865476f);  // 1 - ndtr(z), loss_graphs.py:120-122
}

__global__ void kl_coef_kernel(long long nnz, const float* __restrict__ p, const float* __restrict__ val,
                               const double* __restrict__ stats, float* __restrict__ coef) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= nnz) return;
  const float mp = (float)stats[0], mn = (float)stats[1];
  const float np_ = (float)stats[2], nn_ = (float)stats[3];
  const float s = (float)stats[4], z = (float)stats[5], phi = (float)stats[6];
  if (val[k] > 0.f) coef[k] = -phi / (s * np_) * (1.0f - z * (p[k] - mp) / s);
  else coef[k] = -phi / (s * nn_) * (-1.0f - z * (p[k] - mn) / s);
}

__global__ void scale_kernel(float* __restrict__ w, long long n, const double* __restrict__ stats) {
  const float sc = (float)stats[0];
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) w[i] *= sc;
}

__global__ void bias_add_kernel(float* __restrict__ E, long long n_rows, int n_cols, int ld, const float* __restrict__ bias, int relu) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = n_rows * ld;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < total; i += stride) {
    const int c = (int)(i % ld);
    if (c < n_cols) {
      float v = E[i] + bias[c];
      if (relu) v = v > 0.f ? v : 0.f;  // tf.nn.relu
      E[i] = v;
    }
  }
}

__global__ void relu_mask_kernel(float* __restrict__ dH, const float* __restrict__ H, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride)
    if (!(H[i] > 0.f)) dH[i] = 0.f;  // H > 0 <=> pre-activation > 0 (strict, tf.nn.relu gradient)
}

// column sums in two fixed-order levels
__global__ void col_sum_partial_kernel(const float* __restrict__ dE, long long n_rows, int ld, float* __restrict__ partial) {
  const long long per = (n_rows + gridDim.x - 1) / gridDim.x;
  const long long lo = per * blockIdx.x, hi = min(lo + per, n_rows);
  for (int c = threadIdx.x; c < ld; c += blockDim.x) {
    float s = 0.f;
    for (long long r = lo; r < hi; ++r) s += dE[r * ld + c];
    partial[(long long)blockIdx.x * ld + c] = s;
  }
}
__global__ void col_sum_final_kernel(const float* __restrict__ partial, int n_blocks, int n_cols, int ld, float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_cols) return;
  float s = 0.f;
  for (int b = 0; b < n_blocks; ++b) s += partial[(long long)b * ld + c];
  out[c] = s;
}

// small fp32 GEMM (ReLU embedding second stage and its backward): 64x64 tile, 4x4 per thread
template <int TA, int TB>
__global__ void __launch_bounds__(256) gemm_f32_kernel(int m, int n, int k, const float* __restrict__ A, int lda,
                                                       const float* __restrict__ B, int ldb, float* __restrict__ C, int ldc) {
  __shared__ float sA[16][64 + 1];
  __shared__ float sB[16][64 + 1];
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < k; k0 += 16) {
    for (int i = threadIdx.x; i < 16 * 64; i += 256) {
      const int kk = i / 64, mm = i % 64;
      const int gm_ = m0 + mm, gk = k0 + kk;
      float v = 0.f;
      if (gm_ < m && gk < k) v = TA ? A[(long long)gk * lda + gm_] : A[(long long)gm_ * lda + gk];
      sA[kk][mm] = v;
      const int gn = n0 + mm;
      float w = 0.f;
      if (gn < n && gk < k) w = TB ? B[(long long)gn * ldb + gk] : B[(long long)gk * ldb + gn];
      sB[kk][mm] = w;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = sA[kk][ty * 4 + i]; b[i] = sB[kk][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int gm_ = m0 + ty * 4 + i, gn = n0 + tx * 4 + j;
      if (gm_ < m && gn < n) C[(long long)gm_ * ldc + gn] = acc[i][j];
    }
}

__global__ void gather_rows2d_kernel(const float* __restrict__ in, int n_rows, long long n_cols, const long long* __restrict__ index,
                                     int k, float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)n_rows * k) return;
  const long long r = i / k;
  out[i] = in[r * n_cols + index[i]];
}

__global__ void gather_nd2_kernel(const float* __restrict__ in, long long n_cols, const long long* __restrict__ ind, long long n,
                                  float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = in[ind[2 * i] * n_cols + ind[2 * i + 1]];
}

// one warp per positive interaction: loss_graphs.py:80-88
__global__ void wmrb_forward_kernel(long long n_pos, const int* __restrict__ pos_rows, const float* __restrict__ pos_pred,
                                    const float* __restrict__ sample_pred, int S, float scale, float* __restrict__ loss) {
  const long long k = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (k >= n_pos) return;
  const float base = __fsub_rn(1.0f, pos_pred[k]);
  const float* sp = sample_pred + (long long)pos_rows[k] * S;
  float sum = 0.f;
  for (int j = lane; j < S; j += 32) sum += fmaxf(__fadd_rn(base, sp[j]), 0.f);
  sum = group_sum<32>(sum, 0xffffffffu);
  if (lane == 0) loss[k] = logf(__fadd_rn(1.0f, scale * sum));
}

}  // namespace tmf

// =====================================================================================
// C ABI
// =====================================================================================
using namespace tmf;

extern "C" int tmf_user_pass(int32_t loss, int32_t n_users, int32_t n_items, int64_t nnz, const int32_t* row_ptr, const int32_t* col_idx,
                             const float* val, const float* Eu, const float* Ei, int32_t ld, int32_t n_comp,
                             const int32_t* samp, int32_t n_samples, int32_t n_work, const int32_t* work_user,
                             const int32_t* work_a, const int32_t* work_b, const int32_t* work_slot, float* part_G,
                             float* part_E, int32_t* counter, float* loss_out, float* coef_out, const int32_t* coef_pos, float* dEu,
                             tmf_stream_t stream) {
  TMF_REQUIRE(loss == TMF_LOSS_MSE || loss == TMF_LOSS_WMRB, "tmf_user_pass: unknown loss %d", loss);
  TMF_REQUIRE(n_users >= 0 && n_items > 0 && ld > 0 && ld % 4 == 0 && n_comp <= ld, "tmf_user_pass: bad shape");
  TMF_REQUIRE(ld <= 256, "tmf_user_pass: n_components up to 256 supported (ld=%d)", ld);
  TMF_REQUIRE(aligned16(Eu) && aligned16(Ei) && aligned16(dEu), "tmf_user_pass: embeddings must be 16-byte aligned");
  TMF_REQUIRE(row_ptr && counter && loss_out && coef_out && (nnz == 0 || (col_idx && val)), "tmf_user_pass: null pointer");
  if (loss == TMF_LOSS_WMRB) TMF_REQUIRE(samp && n_samples > 0, "tmf_user_pass: WMRB needs samples (random_ind)");
  if (n_users == 0) return TMF_OK;
  UserPassParams p{};
  p.ld = ld;
  p.n_samples = loss == TMF_LOSS_WMRB ? n_samples : 0;
  p.s_pad = (p.n_samples + 3) & ~3;
  p.row_ptr = row_ptr; p.col_idx = col_idx; p.val = val; p.Eu = Eu; p.Ei = Ei; p.samp = samp;
  p.work_user = work_user; p.work_a = work_a; p.work_b = work_b; p.work_slot = work_slot; p.part_G = part_G; p.part_E = part_E;
  p.n_work = work_user ? n_work : n_users;
  TMF_REQUIRE(!work_user || (work_a && work_b && work_slot), "tmf_user_pass: incomplete work list");
  p.counter = counter; p.loss_out = loss_out; p.coef_out = coef_out; p.coef_pos = coef_pos; p.dEu = dEu;
  p.scale = loss == TMF_LOSS_WMRB ? (float)((double)n_items / (double)n_samples) : 0.f;
  cudaStream_t st = as_stream(stream);
  p.nnz = nnz;  // the G block of coef_out starts at nnz
  const int nv = ld / 4;
  int lpr = 4;
  while (lpr < nv && lpr < 32) lpr <<= 1;
  if (loss == TMF_LOSS_WMRB)
    while (lpr < 32 && (n_samples + lpr - 1) / lpr > 16) lpr <<= 1;
  if (nv > 32) return dispatch_user_pass_j<32, 2>(p, loss, st);
  switch (lpr) {
    case 4: return dispatch_user_pass_j<4, 1>(p, loss, st);
    case 8: return dispatch_user_pass_j<8, 1>(p, loss, st);
    case 16: return dispatch_user_pass_j<16, 1>(p, loss, st);
    default: return dispatch_user_pass_j<32, 1>(p, loss, st);
  }
}

extern "C" size_t tmf_spmm_ws_bytes(int64_t n_entries, int32_t ld_out) {
  const int chunk = spmm_chunk_for(n_entries);
  return (size_t)2 * (size_t)cdiv(n_entries > 0 ? n_entries : 1, chunk) * (size_t)ld_out * sizeof(float) + 256;
}

extern "C" int tmf_spmm_seg(int32_t n_seg, const int32_t* seg_ptr, int64_t n_entries, const int32_t* idx,
                            const int32_t* cpos, const float* coef, const float* src, int32_t ld_src, float* out,
                            int32_t ld_out, int32_t n_cols, void* ws, size_t ws_bytes, tmf_stream_t stream) {
  TMF_REQUIRE(n_seg >= 0 && n_entries >= 0 && n_entries < (1ll << 31), "tmf_spmm_seg: bad sizes");
  TMF_REQUIRE(ld_src % 4 == 0 && ld_out % 4 == 0 && n_cols <= ld_src && n_cols <= ld_out, "tmf_spmm_seg: bad leading dims");
  TMF_REQUIRE(aligned16(src) && aligned16(out) && aligned16(ws), "tmf_spmm_seg: 16-byte alignment required");
  TMF_REQUIRE(ws_bytes >= tmf_spmm_ws_bytes(n_entries, ld_out), "tmf_spmm_seg: workspace too small");
  if (n_seg == 0) return TMF_OK;
  SpmmParams p{};
  p.n_seg = n_seg; p.ld_src = ld_src; p.ld_out = ld_out; p.nv = (n_cols + 3) / 4; p.chunk = spmm_chunk_for(n_entries);
  p.n_entries = n_entries; p.seg_ptr = seg_ptr; p.idx = idx; p.cpos = cpos; p.coef = coef; p.src = src; p.out = out;
  const long long n_chunks = cdiv(n_entries > 0 ? n_entries : 1, p.chunk);
  p.part_first = reinterpret_cast<float*>(ws);
  p.part_carry = p.part_first + n_chunks * ld_out;
  cudaStream_t st = as_stream(stream);
  if (p.nv <= 4) return launch_spmm<4>(p, st);
  if (p.nv <= 8) return launch_spmm<8>(p, st);
  if (p.nv <= 16) return launch_spmm<16>(p, st);
  return launch_spmm<32>(p, st);
}

extern "C" int tmf_pair_dots(int64_t nnz, const int32_t* rows, const int32_t* cols, const float* Eu, const float* Ei,
                             int32_t ld, float* p, tmf_stream_t stream) {
  TMF_REQUIRE(ld % 4 == 0 && aligned16(Eu) && aligned16(Ei), "tmf_pair_dots: alignment");
  if (nnz == 0) return TMF_OK;
  pair_dots_kernel<<<(unsigned)cdiv(nnz * 8, 256), 256, 0, as_stream(stream)>>>(nnz, rows, cols, Eu, Ei, ld, p);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

extern "C" size_t tmf_reduce_ws_bytes(void) { return (size_t)(kRedBlocks * kRedMaxWidth + kRedStats) * sizeof(double); }

static int red_blocks(long long n) { return (int)std::max<long long>(1, std::min<long long>(kRedBlocks, cdiv(n, 4096))); }

extern "C" int tmf_reduce_sum(const float* x, int64_t n, float* out, void* ws, tmf_stream_t stream) {
  TMF_REQUIRE(ws && out, "tmf_reduce_sum: null");
  double* stats = reinterpret_cast<double*>(ws);
  double* partial = stats + kRedStats;
  const int nb = red_blocks(n);
  cudaStream_t st = as_stream(stream);
  reduce_partial_kernel<kRedSum><<<nb, kRedThreads, 0, st>>>(x, nullptr, n, partial);
  reduce_final_kernel<kRedSum><<<1, kRedThreads, 0, st>>>(partial, nb, stats, out);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

extern "C" int tmf_l2_normalize_global(float* w, int64_t n, void* ws, tmf_stream_t stream) {
  TMF_REQUIRE(ws && w, "tmf_l2_normalize_global: null");
  double* stats = reinterpret_cast<double*>(ws);
  double* partial = stats + kRedStats;
  const int nb = red_blocks(n);
  cudaStream_t st = as_stream(stream);
  reduce_partial_kernel<kRedSumSq><<<nb, kRedThreads, 0, st>>>(w, nullptr, n, partial);
  reduce_final_kernel<kRedSumSq><<<1, kRedThreads, 0, st>>>(partial, nb, stats, nullptr);
  scale_kernel<<<grid_stride_blocks(cdiv(n, 256), 16), 256, 0, st>>>(w, n, stats);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

extern "C" int tmf_kl_moments(int64_t nnz, const float* p, const float* val, double* moments_out, void* ws, tmf_stream_t stream) {
  TMF_REQUIRE(ws && moments_out && (nnz == 0 || (p && val)), "tmf_kl_moments: null");
  double* partial = reinterpret_cast<double*>(ws) + kRedStats;
  const int nb = red_blocks(nnz);
  cudaStream_t st = as_stream(stream);
  reduce_partial_kernel<kRedKLMoments><<<nb, kRedThreads, 0, st>>>(p, val, nnz, partial);
  reduce_final_kernel<kRedKLMoments><<<1, kRedThreads, 0, st>>>(partial, nb, moments_out, nullptr);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

extern "C" int tmf_kl_coef_from_moments(int64_t nnz, const float* p, const float* val, const double* moments, float* loss_out,
                                        float* coef_out, void* ws, tmf_stream_t stream) {
  TMF_REQUIRE(ws && moments && loss_out && coef_out && (nnz == 0 || (p && val)), "tmf_kl_coef_from_moments: null");
  double* stats = reinterpret_cast<double*>(ws);
  cudaStream_t st = as_stream(stream);
  kl_from_moments_kernel<<<1, 32, 0, st>>>(moments, stats, loss_out);
  if (nnz > 0) kl_coef_kernel<<<(unsigned)cdiv(nnz, 256), 256, 0, st>>>(nnz, p, val, stats, coef_out);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

extern "C" int tmf_adam1(float* w, const float* g, int64_t n, float lr, tmf_stream_t stream) {
  if (n == 0) return TMF_OK;
  const int vec = aligned16(w) && aligned16(g);  // views at odd offsets take the scalar path
  adam1_kernel<<<grid_stride_blocks(cdiv(cdiv(n, vec ? 4 : 1), 256), 16), 256, 0, as_stream(stream)>>>(w, g, n, lr, vec);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

extern "C" int tmf_adam(float* w, const float* g, float* m, float* v, int64_t n, float lr, int32_t step, tmf_stream_t stream) {
  TMF_REQUIRE(step >= 1, "tmf_adam: step counts from 1");
  if (n == 0) return TMF_OK;
  const float alpha = lr * sqrtf(1.0f - powf(0.999f, (float)step)) / (1.0f - powf(0.9f, (float)step));
  adam_kernel<<<grid_stride_blocks(cdiv(n, 256), 32), 256, 0, as_stream(stream)>>>(w, g, m, v, n, alpha);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

extern "C" int tmf_bias_add(float* E, int64_t n_rows, int32_t n_cols, int32_t ld, const float* bias, int32_t relu,
                            tmf_stream_t stream) {
  if (n_rows == 0) return TMF_OK;
  bias_add_kernel<<<grid_stride_blocks(cdiv(n_rows * ld, 256), 32), 256, 0, as_stream(stream)>>>(
      E, n_rows, n_cols, ld, bias, relu);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

extern "C" int tmf_relu_mask(float* dH, const float* H, int64_t n, tmf_stream_t stream) {
  if (n == 0) return TMF_OK;
  relu_mask_kernel<<<grid_stride_blocks(cdiv(n, 256), 32), 256, 0, as_stream(stream)>>>(dH, H, n);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

extern "C" int tmf_col_sum(const float* dE, int64_t n_rows, int32_t n_cols, int32_t ld, float* out, void* ws,
                           size_t ws_bytes, tmf_stream_t stream) {
  TMF_REQUIRE(ws_bytes >= (size_t)1024 * ld * sizeof(float), "tmf_col_sum: workspace too small");
  const int nb = (int)std::max<long long>(1, std::min<long long>(1024, cdiv(n_rows, 64)));
  cudaStream_t st = as_stream(stream);
  col_sum_partial_kernel<<<nb, 256, 0, st>>>(dE, n_rows, ld, reinterpret_cast<float*>(ws));
  col_sum_final_kernel<<<(unsigned)cdiv(n_cols, 128), 128, 0, st>>>(reinterpret_cast<float*>(ws), nb, n_cols, ld, out);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

extern "C" int tmf_gemm_f32(int32_t ta, int32_t tb, int32_t m, int32_t n, int32_t k, const float* A, int32_t lda,
                            const float* B, int32_t ldb, float* C, int32_t ldc, tmf_stream_t stream) {
  if (m == 0 || n == 0) return TMF_OK;
  dim3 grid((unsigned)cdiv(n, 64), (unsigned)cdiv(m, 64));
  cudaStream_t st = as_stream(stream);
  if (!ta && !tb) gemm_f32_kernel<0, 0><<<grid, 256, 0, st>>>(m, n, k, A, lda, B, ldb, C, ldc);
  else if (ta && !tb) gemm_f32_kernel<1, 0><<<grid, 256, 0, st>>>(m, n, k, A, lda, B, ldb, C, ldc);
  else if (!ta && tb) gemm_f32_kernel<0, 1><<<grid, 256, 0, st>>>(m, n, k, A, lda, B, ldb, C, ldc);
  else gemm_f32_kernel<1, 1><<<grid, 256, 0, st>>>(m, n, k, A, lda, B, ldb, C, ldc);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

extern "C" int tmf_gather_rows2d(const float* in, int32_t n_rows, int64_t n_cols, const int64_t* index, int32_t k,
                                 float* out, tmf_stream_t stream) {
  const long long n = (long long)n_rows * k;
  if (n == 0) return TMF_OK;
  gather_rows2d_kernel<<<(unsigned)cdiv(n, 256), 256, 0, as_stream(stream)>>>(in, n_rows, n_cols,
                                                                           reinterpret_cast<const long long*>(index), k, out);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

extern "C" int tmf_gather_nd2(const float* in, int64_t n_cols, const int64_t* indices2, int64_t n, float* out,
                              tmf_stream_t stream) {
  if (n == 0) return TMF_OK;
  gather_nd2_kernel<<<(unsigned)cdiv(n, 256), 256, 0, as_stream(stream)>>>(in, n_cols, reinterpret_cast<const long long*>(indices2), n, out);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

extern "C" int tmf_wmrb_forward(int64_t n_pos, const int32_t* pos_rows, const float* pos_pred, const float* sample_pred,
                                int32_t n_samples, float scale, float* loss_out, tmf_stream_t stream) {
  if (n_pos == 0) return TMF_OK;
  wmrb_forward_kernel<<<(unsigned)cdiv(n_pos * 32, 256), 256, 0, as_stream(stream)>>>(n_pos, pos_rows, pos_pred, sample_pred,
                                                                                   n_samples, scale, loss_out);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

extern "C" int tmf_user_pass_fixup(int32_t loss, int32_t n_split, const int32_t* split_user, const int32_t* split_first,
                                   const int32_t* split_nseg, const float* Ei, int32_t ld, const int32_t* samp, int32_t n_samples,
                                   int64_t nnz, const float* part_G, const float* part_E, float* coef_out, const int32_t* coef_pos,
                                   float* dEu, tmf_stream_t stream) {
  if (n_split == 0) return TMF_OK;
  TMF_REQUIRE(split_user && split_first && split_nseg && part_E && dEu, "tmf_user_pass_fixup: null pointer");
  UserPassParams p{};
  p.ld = ld; p.n_samples = loss == TMF_LOSS_WMRB ? n_samples : 0; p.s_pad = (p.n_samples + 3) & ~3; p.nnz = nnz;
  p.Ei = Ei; p.samp = samp; p.part_G = const_cast<float*>(part_G); p.part_E = const_cast<float*>(part_E);
  p.coef_out = coef_out; p.coef_pos = coef_pos; p.dEu = dEu;
  const size_t smem = (size_t)(p.s_pad + ld + 1024) * sizeof(float);  // (256 / nvp) partial rows of ld floats <= 1024 floats
  TMF_REQUIRE(smem <= 48 * 1024 && ld <= 256, "tmf_user_pass_fixup: n_samples too large");
  user_fixup_kernel<<<grid_stride_blocks(n_split, 4), 256, smem, as_stream(stream)>>>(p, loss, n_split, split_user, split_first, split_nseg);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}
