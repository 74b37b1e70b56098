// Fused U.V^T + per-row top-k for sm_100a:  tcgen05 bf16 GEMM (TMA-staged operands, fp32 accumulators
// in TMEM) whose epilogue never writes scores to HBM -- it filters each accumulator tile against a
// per-row running threshold and appends the few survivors to a candidate list; an fp64-accumulated
// rerank of the candidates then makes the returned indices exact (ties -> lower item id).
//
// Exactness argument (DESIGN.md "top-k"): with u~, v~ the 16-bit operands (bf16 or fp16, chosen from the data) and du = u - u~,
// dv = v - v~, the tensor-core score s~ of a pair differs from the canonical score s by at most
//   E[row] = |du| max_items|v| + |u~| max_items|dv| + accumulation slack          (Cauchy-Schwarz; norms from pack_bf16_kernel,
// measured on the data, not a format constant -- row_error_kernel).  With t~ the k-th largest s~ seen so far in a row, every item
// of the final top-k satisfies s~ >= t~ - 2E, so the candidate list is a superset of the answer; the rerank sorts it by
// (canonical score desc, item id asc).
//
// Structure (round 2 re-measured the alternatives, profiles/r02_summary.md): two CTAs per SM, each with its own TMA producer,
// MMA-issuing thread, two 128-column TMEM accumulators and FOUR epilogue warps that own their rows outright -- list, queue,
// histogram and threshold of a row are private to one lane, so the filter needs no atomics and no cross-warp hand-shakes.
// Designs with 16 epilogue warps per SM on shared per-row state (one
// CTA per SM, cta_group::2 pairs, two issuing threads) ran the bare MMA pipeline at the sustained tensor peak but spent more
// instructions per score on the shared state and were 10 % slower end to end.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <limits.h>
#include <math.h>
#include <stdlib.h>

#include <algorithm>

#include "common.cuh"
#include "tc_common.cuh"

namespace tmf {

// Development switches (TMF_TOPK_DEBUG / TMF_TOPK_FMT / TMF_TOPK_PROF) exist only in builds compiled with -DTMF_DEVTOOLS
// (scripts/build_variant.sh); the product library reads no environment variable.
#ifdef TMF_DEVTOOLS
#define TMF_DBG(p) ((p).dbg)
#else
#define TMF_DBG(p) 0
#endif
constexpr int BM = 128;        // users per CTA tile (TMEM lanes)
constexpr int BN = 128;        // items per accumulator tile (TMEM columns); two CTAs share an SM
constexpr int BK = 64;         // bf16 elements per 128-byte swizzle row
constexpr int UMMA_K = 16;
constexpr int NSTAGES = 3;     // B-operand ring (16 KB stages)
constexpr int TMEM_COLS = 2 * BN;  // two accumulators per CTA, double-buffered against the epilogue
constexpr int CAP = 2048;      // candidate slots per row (appended, never compacted; saturation -> exact path)
constexpr int INIT_N = 512;    // a row's threshold state is initialised from its first <= INIT_N entries
constexpr int CPL = INIT_N / 32;  // entries per lane in the warp-cooperative initial selection
constexpr int NBINS = 48;      // per-row score histogram bins (16-bit counts, two per word)
constexpr int QCAP = 16;       // per-row survivor queue slots in shared memory (drained warp-wide)
constexpr int HSTRIDE = NBINS / 2 + 1;  // words per row, padded against bank conflicts
constexpr int UB_BATCH = 2048; // user blocks (x128 rows) per main-kernel launch: bounds the candidate workspace to 4 GB
// Wide configuration, 128 < k <= 1024 (DESIGN "top-k", wide k): the same kernel with longer lists.  8192 slots leave ~5k
// appends between saturation rebuilds even in clamp mode, where the k lowest ids stay listed besides >= k entries above the
// threshold; 592 user blocks = exactly two waves of the 2 x 148 persistent CTAs and a 4.96 GB candidate workspace.  The
// first rebuild streams the list through warp_rebuild_selected once it holds k + 2 tiles of entries (warp_rebuild_first keeps
// only INIT_N entries in registers).
constexpr int NARROW_MAX_K = 128;
constexpr int WIDE_MAX_K = 1024;
constexpr int CAP_W = 8192;
constexpr int UB_BATCH_W = 592;
constexpr int TOPK_THREADS = 256;
constexpr int A_SUB_BYTES = BM * BK * 2;   // 16 KB
constexpr int B_STAGE_BYTES = BN * BK * 2; // 16 KB
constexpr int MAX_KB = 4;                  // n_components <= 256
// Error bound of the tensor-core score s~ = fl32(sum u~_c v~_c) against the real score s = sum u_c v_c, with u~ = bf16(u),
// du = u - u~ (both known exactly):  s - sum u~_c v~_c = du.v + u~.dv  =>  |s~ - s| <= |du||v| + |u~||dv| + accumulation.
// The residual norms are computed from the data by pack_bf16_kernel, so the bound is rigorous (unit roundoff of bf16 is
// 2^-8 per operand: worst case 2^-7 |u||v|) AND tight for typical data (about 0.8 * 2^-8 |u||v|).
// ACC_UNIT: slack per accumulated k-step for the fp32 accumulation inside the tensor core, relative to |u~||v~|.
constexpr float ACC_UNIT = 2.4e-7f;
constexpr float NORM_SLACK = 1.0001f;  // rounding of the fp32 norm arithmetic itself

// PTX wrappers (mbarrier, TMA, tcgen05, TMEM loads, descriptors): tc_common.cuh, shared with gemm_tc.cu
// kind::f16 instruction descriptor: D=f32, A=B=bf16, both K-major, M=128, N=256
constexpr uint32_t kIdesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);

// ------------------------------------------------------------------ warp-cooperative selection
__device__ __forceinline__ uint32_t f2key(float x) {
  const uint32_t u = __float_as_uint(x);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key2f(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k);
}

// shared-space reduction (a generic-address atomicAdd compiles to the slow generic ATOM path)
__device__ __forceinline__ void smem_inc(int* p) {
  asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(smem_u32(p)) : "memory");
}

__device__ __forceinline__ bool use_fp16(const float* stats);  // operand format choice, defined with the pack kernels

struct TopkParams {
  long long n_users, n_items;   // real sizes
  int ub0, n_ublocks;           // this launch covers user blocks [ub0, ub0 + n_ublocks)
  int n_tiles, kb;              // item tiles of BN, k-blocks of BK
  int k, clamp, item_offset;
  const float* erow;            // [n_users_pad] error bound E of each user row against this item slab (global row index)
  float2* cand;                 // [batch rows][CAP or CAP_W] (approx score, item id bits), batch-local row index
  int* cnt;                     // [batch rows] candidates per row, -1 = overflow (exact path)
  float* thr_out;               // [batch rows] final keep-threshold of the row
  int* ovf_count;               // [1]
  int* ovf_rows;                // [n_users_pad] global rows handed to the exact path
  float* dump;                  // optional [n_users][dump_ld]: raw bf16-GEMM scores (bring-up / error-bound tests)
  long long dump_ld;
  const float* fmt_stats;       // operand statistics (see use_fp16); NULL with force_fmt >= 0
  int force_fmt;                // -1 = by fmt_stats, 0 = bf16, 1 = fp16
  const float* row_bound;       // optional [n_users]: lower bounds of the rows' k-th best TRUE score (cross-GPU exchange), raw mode only
  unsigned long long* prof;     // optional [8] cycle counters (env TMF_TOPK_PROF=1): where the warps wait
  int dbg;                      // profiling aid (env TMF_TOPK_DEBUG): 1 = no appends, 2 = no filtering, 3 = no TMEM reads
  const int* ex_ptr;            // MASK: [n_users + 1] CSR of the global item ids excluded per row (sorted, distinct)
  const int* ex_idx;
};

// Keep-threshold from a lower bound `kth` of the row's k-th largest approximate score.
//   raw scores   : every top-k member has s~ >= kth - 2E
//   clamped (>0) : every top-k member outside the k lowest item ids has s~ >= max(kth - E, 0) - E
__device__ __forceinline__ float keep_threshold(float kth, float E, int clamp) {
  return clamp ? fmaxf(kth - E, 0.f) - E : kth - 2.f * E;
}

// Whether a list entry (approx score, item id) stays listed under keep-threshold thr.  Clamp mode also keeps the k lowest
// item ids of the slab whatever their score: when fewer than k items score above zero, the answer is filled with zero-score
// items in id order, and those fillers must still be listed.  Every filter of a candidate list goes through here.
__device__ __forceinline__ bool keep_entry(float2 x, float thr, int clamp, int item_offset, int k) {
  return x.x >= thr || (clamp && __float_as_int(x.y) - item_offset < k);
}

// ---- per-row running threshold: a lane-private 48-bin histogram of the appended scores (16-bit counts, two
// bins per shared-memory word).  bthr = the highest bin whose "at or above" count A is still >= k, so the lower
// edge of bin bthr is a valid lower bound of the k-th largest score seen so far; it only ever rises.
//
// ---- SIMD list maintenance.  A lane that finds a survivor only pushes (score, item) onto its own small
// shared-memory queue (3 instructions, no dependent loads).  When a queue is about to fill, the WHOLE warp
// drains: iteration s handles entry s of every lane at once, each lane appending to its own row's list and
// updating its own histogram -- the ~40-instruction append runs once per queue slot for 32 rows instead of
// once per survivor with 1-3 active lanes (measured: 400-600 cycles per survivor in the divergent versions).
struct RowState {
  float thr;      // current keep-threshold (+inf for padded rows)
  float thr_ext;  // externally supplied floor of the threshold (-inf when there is none)
  float lo, w, inv_w, E;
  int cnt;        // list length; > CAP = saturated (-> exact path)
  int cq;         // entries waiting in the lane's queue
  int bthr, A;    // threshold bin and # entries with bin >= bthr
};

__device__ __forceinline__ int hist_get(const uint32_t* hrow, int b) { return (int)((hrow[b >> 1] >> ((b & 1) * 16)) & 0xffffu); }
// explicit shared-space accesses: through generic pointers these compile to the slower ST.E/LD.E with 64-bit addressing
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ void sts_u32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ float2 lds_f2(uint32_t a) { float2 v; asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a)); return v; }
__device__ __forceinline__ int hist_get_s(uint32_t hrow, int b) { return (int)((lds_u32(hrow + 4u * (uint32_t)(b >> 1)) >> ((b & 1) * 16)) & 0xffffu); }

// lower edge of bin bthr, less the rounding of the bin arithmetic: >= k entries are >= it (histogram invariant)
__device__ __forceinline__ float bin_edge(float lo, float w, int bthr) {
  const float slack = 4e-7f * (fabsf(lo) + (float)NBINS * w);
  return lo + (float)bthr * w - slack;
}
__device__ __forceinline__ float edge_threshold(float lo, float w, int bthr, float E, int clamp) {
  return keep_threshold(bin_edge(lo, w, bthr), E, clamp);
}

// ---- masked top-k: each row's cursor into its sorted list of excluded item ids, three words in shared memory
// {position, end, id at the position (INT_MAX past the end)}.  Entries reach a row's list in ascending id order (tiles
// sweep the ids upward, a tile's groups and columns are queued in order, queues drain slot by slot), so the cursor only
// moves forward -- O(row length) over the whole sweep -- and an excluded id is recognised by one compare with the cursor's id.
constexpr int EXCUR_BYTES = 16;  // per row
__device__ __forceinline__ int ex_step(const int* ex_idx, int& pos, int end) {
  ++pos;
  return pos < end ? __ldg(ex_idx + pos) : INT_MAX;
}

// warp-wide drain of the per-lane queues (all lanes must call; st.cq may differ per lane).  Iterations are
// independent of each other -- fire-and-forget histogram increments (red.shared), list stores that nobody waits
// for, threshold fixed for the duration -- so they pipeline; the threshold advances once at the end.
// MASK: excluded ids are dropped here, before the list store and the histogram increment.
struct DrainRet { float thr; int cnt, bthr, A; };
template <int CAP, bool MASK>
__device__ __forceinline__ DrainRet drain_body(float thr, float thr_ext, float lo, float w, float inv_w, float E, int cnt, int cq, int bthr,
                                               int A, uint32_t queue, float2* buf, uint32_t hrow, int k, int clamp, uint32_t excur,
                                               const int* ex_idx) {
  int maxq = cq;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) maxq = max(maxq, __shfl_xor_sync(0xffffffffu, maxq, o));
  int ex_pos = 0, ex_end = 0, ex_next = 0;
  if constexpr (MASK) {
    ex_pos = (int)lds_u32(excur);
    ex_end = (int)lds_u32(excur + 4u);
    ex_next = (int)lds_u32(excur + 8u);
  }
#pragma unroll 4
  for (int s = 0; s < maxq; ++s) {
    const float2 e = lds_f2(queue + 8u * (uint32_t)s);
    bool ok = (s < cq) && (e.x >= thr);
    if constexpr (MASK) {
      if (ok) {
        const int id = __float_as_int(e.y);
        while (ex_next < id) ex_next = ex_step(ex_idx, ex_pos, ex_end);
        ok = ex_next != id;
      }
    }
    const bool okh = ok && (e.x >= lo);
    const int b = (int)fminf(fmaxf((e.x - lo) * inv_w, 0.f), (float)(NBINS - 1));
    const int st_ok = ok && (cnt < CAP);
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.s32 p, %0, 0;\n\t"
        "setp.ne.s32 q, %1, 0;\n\t"
        "@p st.global.cg.v2.f32 [%2], {%3, %4};\n\t"
        "@q red.shared.add.u32 [%5], %6;\n\t"
        "@q red.shared.max.u32 [%7], %8;\n\t}"
        ::"r"(st_ok), "r"((int)okh), "l"(buf + cnt), "f"(e.x), "f"(e.y), "r"(hrow + 4u * (uint32_t)(b >> 1)),
          "r"(1u << ((b & 1) * 16)), "r"(hrow + 4u * (uint32_t)(NBINS / 2)), "r"(f2key(e.x))
        : "memory");
    cnt += ok ? 1 : 0;
    A += (okh && b >= bthr) ? 1 : 0;
  }
  __syncwarp();
  if constexpr (MASK) {
    sts_u32(excur, (uint32_t)ex_pos);
    sts_u32(excur + 8u, (uint32_t)ex_next);
  }
  bool moved = false;
  while (bthr < NBINS - 1) {
    const int hb = hist_get_s(hrow, bthr);
    if (A - hb < k) break;
    A -= hb;
    ++bthr;
    moved = true;
  }
  if (moved) thr = fmaxf(edge_threshold(lo, w, bthr, E, clamp), thr_ext);
  DrainRet r;
  r.thr = thr; r.cnt = cnt; r.bthr = bthr; r.A = A;
  return r;
}
// (out of line, state by value in registers: inlining it at every call site costs registers in the tile loop)
template <int CAP>
__device__ __noinline__ DrainRet drain_queues_nl(float thr, float thr_ext, float lo, float w, float inv_w, float E, int cnt, int cq, int bthr, int A,
                                                 uint32_t queue, float2* buf, uint32_t hrow, int k, int clamp) {
  return drain_body<CAP, false>(thr, thr_ext, lo, w, inv_w, E, cnt, cq, bthr, A, queue, buf, hrow, k, clamp, 0u, nullptr);
}
template <int CAP>
__device__ __noinline__ DrainRet drain_queues_masked_nl(float thr, float thr_ext, float lo, float w, float inv_w, float E, int cnt, int cq,
                                                        int bthr, int A, uint32_t queue, float2* buf, uint32_t hrow, int k, int clamp,
                                                        uint32_t excur, const int* ex_idx) {
  return drain_body<CAP, true>(thr, thr_ext, lo, w, inv_w, E, cnt, cq, bthr, A, queue, buf, hrow, k, clamp, excur, ex_idx);
}
template <int CAP, bool MASK>
__device__ __forceinline__ void drain_queues(RowState& st, uint32_t queue, float2* buf, uint32_t hrow, int k, int clamp, uint32_t excur,
                                             const int* ex_idx) {
  DrainRet r;
  if constexpr (MASK)
    r = drain_queues_masked_nl<CAP>(st.thr, st.thr_ext, st.lo, st.w, st.inv_w, st.E, st.cnt, st.cq, st.bthr, st.A, queue, buf, hrow, k,
                                    clamp, excur, ex_idx);
  else
    r = drain_queues_nl<CAP>(st.thr, st.thr_ext, st.lo, st.w, st.inv_w, st.E, st.cnt, st.cq, st.bthr, st.A, queue, buf, hrow, k, clamp);
  st.thr = r.thr; st.cnt = r.cnt; st.bthr = r.bthr; st.A = r.A;
  st.cq = 0;
}

// One 32-column slice of a row's accumulator BEFORE the row's threshold exists (first 3 tiles; wide k: until the row
// holds k + 2 tiles of entries): every column is appended directly.  (Clamp-mode "filler" items -- the k lowest ids --
// therefore need no special case.)  MASK: except the row's excluded ids.
template <bool DUMP, bool MASK>
__device__ __forceinline__ void epilogue_chunk(uint32_t (&r)[32], int col0, int n_items, bool valid, bool warp_inited,
                                               RowState& st, uint32_t queue, float2* buf, uint32_t hrow, long long row,
                                               const TopkParams& p, uint32_t excur) {
  if (DUMP) {
    if (valid) {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (col0 + j < n_items) p.dump[row * p.dump_ld + col0 + j] = __uint_as_float(r[j]);
    }
    return;
  }
  if (TMF_DBG(p) == 2 || TMF_DBG(p) == 3) return;
  const int id0 = p.item_offset + col0;
  if (!warp_inited) {  // warp-uniform: no threshold yet, keep everything (coalesced per lane, no queue)
    if (valid) {
      uint32_t seen = 0;  // MASK: bit j = id0 + j is excluded
      if constexpr (MASK) {
        int pos = (int)lds_u32(excur), next = (int)lds_u32(excur + 8u);
        const int end = (int)lds_u32(excur + 4u);
        while (next < id0 + 32) {
          if (next >= id0) seen |= 1u << (next - id0);
          next = ex_step(p.ex_idx, pos, end);
        }
        sts_u32(excur, (uint32_t)pos);
        sts_u32(excur + 8u, (uint32_t)next);
      }
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        if (col0 + j < n_items && !((seen >> j) & 1u)) {
          __stcg(buf + st.cnt, make_float2(__uint_as_float(r[j]), __int_as_float(id0 + j)));
          ++st.cnt;
        }
      }
    }
    return;
  }
}

// 8-column group maxima of one 32-column slice (3-input max tree, no branches)
__device__ __forceinline__ void group_max4(const uint32_t (&r)[32], float* m8) {
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    const float a = fmaxf(fmaxf(__uint_as_float(r[8 * g + 0]), __uint_as_float(r[8 * g + 1])), __uint_as_float(r[8 * g + 2]));
    const float b = fmaxf(fmaxf(a, __uint_as_float(r[8 * g + 3])), __uint_as_float(r[8 * g + 4]));
    const float c = fmaxf(fmaxf(b, __uint_as_float(r[8 * g + 5])), __uint_as_float(r[8 * g + 6]));
    m8[g] = fmaxf(c, __uint_as_float(r[8 * g + 7]));
  }
}

// Steady-state filter of one 64-column HALF of an accumulator tile (rows with a threshold).  Pass 1 brings the 64 columns into
// registers (two x32 TMEM loads in flight, one wait) and reduces them to 8 group-maximum hit bits -- no votes, no branches.  One
// REDUX.OR of the per-lane hit masks then names the 8-column groups in which ANY row of the warp has a survivor (about 2 of 8 at
// 1M items); only those are re-read from TMEM (x8) and their survivors queued with predicated stores, all lanes convergent.
// Measured alternatives for pass 2, all slower on the 151,552 x 1M slice (45.9 ms with this version): pushing from the pass-1
// registers through an unrolled chain of warp-uniform blocks (51.0 ms: 16 extra branches per tile) or an indexed jump (register
// arrays spill); issuing the next group's TMEM load under the current group's pushes (48.4 ms); slot indices from a survivor
// mask + popc instead of the running count (47.4 ms).  The epilogue pays per instruction, not per round trip.
template <int CAP, bool MASK>
__device__ __forceinline__ void epilogue_half(uint32_t t_base, int col0, RowState& st, uint32_t queue, float2* buf, uint32_t hrow,
                                              const TopkParams& p, uint32_t excur) {
  uint32_t ra[32], rb[32];
  float m8[4];
  const float thr = st.thr;  // invalid rows carry thr = +inf; NaN-padded columns never win a max or a compare
  unsigned hm = 0;
  tmem_ld32(t_base, ra);
  tmem_ld32(t_base + 32u, rb);
  tmem_ld_wait_for(ra);   // wait::ld covers both loads; the second call pins rb behind a wait as well
  tmem_ld_wait_for(rb);
  group_max4(ra, m8);
#pragma unroll
  for (int g = 0; g < 4; ++g) hm |= (m8[g] >= thr) ? (1u << g) : 0u;
  group_max4(rb, m8);
#pragma unroll
  for (int g = 0; g < 4; ++g) hm |= (m8[g] >= thr) ? (16u << g) : 0u;
  unsigned gmask = __reduce_or_sync(0xffffffffu, hm);
  if (TMF_DBG(p) == 1) gmask = 0;
  if (gmask == 0) return;
  const int id0 = p.item_offset + col0;
  while (gmask) {  // warp-uniform
    const int g = __ffs(gmask) - 1;
    gmask &= gmask - 1;
    uint32_t v[8];
    tmem_ld8(t_base + (uint32_t)(8 * g), v);
    if (__any_sync(0xffffffffu, st.cq > QCAP - 8)) drain_queues<CAP, MASK>(st, queue, buf, hrow, p.k, p.clamp, excur, p.ex_idx);
    tmem_ld_wait_for8(v);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float x = __uint_as_float(v[j]);
      asm volatile("{\n\t.reg .pred p;\n\tsetp.ge.f32 p, %0, %1;\n\t@p st.shared.v2.f32 [%2], {%0, %3};\n\t}"
                   ::"f"(x), "f"(thr), "r"(queue + 8u * (uint32_t)st.cq), "f"(__int_as_float(id0 + 8 * g + j)) : "memory");
      st.cq += (x >= thr) ? 1 : 0;
    }
  }
}
template <int CAP, bool MASK>
__device__ __forceinline__ void epilogue_tile(uint32_t t_base, int col0, RowState& st, uint32_t queue, float2* buf, uint32_t hrow,
                                              const TopkParams& p, uint32_t excur) {
#pragma unroll 1
  for (int h = 0; h < 2; ++h)  // one copy of the code: the unrolled pass 2 is ~4 KB of sparsely executed instructions
    epilogue_half<CAP, MASK>(t_base + (uint32_t)(64 * h), col0 + 64 * h, st, queue, buf, hrow, p, excur);
}

// One step of an 8-bit radix select over 256 shared-memory counters: returns the bin that holds the krem-th largest counted
// entry (bins ranked from 255 down) and sets krem to that entry's rank within the bin.  All lanes; the counted entries
// must number >= krem.
__device__ __forceinline__ int pick_bin(const int* cnt256, int& krem) {
  const int lane = threadIdx.x & 31;
  int c[8];
  int lsum = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) {  // lane L owns bins 255-8L .. 248-8L, visited in descending order
    c[i] = cnt256[255 - 8 * lane - i];
    lsum += c[i];
  }
  int incl = lsum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  const unsigned reach = __ballot_sync(0xffffffffu, incl >= krem);
  const int F = reach ? __ffs(reach) - 1 : 31;
  int bin = 0, knew = 0;
  if (lane == F) {
    int cum = incl - lsum;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (cum + c[i] >= krem) { bin = 255 - 8 * lane - i; knew = krem - cum; break; }
      cum += c[i];
    }
  }
  krem = __shfl_sync(0xffffffffu, knew, F);
  return __shfl_sync(0xffffffffu, bin, F);
}

// Exact k-th largest of a warp's entries by an 8-bit-per-pass radix select.  count(shift, mask, prefix) visits the entries
// and counts each whose key matches prefix under mask into radix[(key >> shift) & 255] (256 ints of shared-memory scratch,
// see count_key).  Needs >= k entries.
template <class Count>
__device__ __forceinline__ float radix_select_kth(int k, int* radix, Count count) {
  const int lane = threadIdx.x & 31;
  uint32_t prefix = 0, mask = 0;
  int krem = k;
#pragma unroll 1
  for (int shift = 24; shift >= 0; shift -= 8) {
#pragma unroll
    for (int i = 0; i < 8; ++i) radix[lane * 8 + i] = 0;
    __syncwarp();
    count(shift, mask, prefix);
    __syncwarp();
    const int bin = pick_bin(radix, krem);
    prefix |= (uint32_t)bin << shift;
    mask |= 255u << shift;
    __syncwarp();
  }
  return key2f(prefix);
}
__device__ __forceinline__ void count_key(int* radix, float x, int shift, uint32_t mask, uint32_t prefix) {
  const uint32_t key = f2key(x);
  if ((key & mask) == prefix) smem_inc(&radix[(key >> shift) & 255u]);
}

// exact k-th largest approximate score of a row's list (n >= k entries in global memory, streamed through L2); also
// returns the list maximum
__device__ __noinline__ float warp_select_kth(const float2* buf, int n, int k, int* radix, float& mx_out) {
  const int lane = threadIdx.x & 31;
  float mx = -INFINITY;
  const float kth = radix_select_kth(k, radix, [&](int shift, uint32_t mask, uint32_t prefix) {
    for (int e0 = 0; e0 < n; e0 += 32 * 8) {  // 8 independent loads in flight per lane (one L2 round trip per 256 entries)
      float sc[8];
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        const int e = e0 + 32 * t + lane;
        sc[t] = (e < n) ? __ldcg(&buf[e].x) : -INFINITY;
      }
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        if (e0 + 32 * t + lane < n) {
          mx = fmaxf(mx, sc[t]);
          count_key(radix, sc[t], shift, mask, prefix);
        }
      }
    }
  });
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  mx_out = mx;
  return kth;
}

// Bin width of a row histogram re-centred on [lo, lo + range (row max - lo)); a degenerate range (all entries equal, or
// not finite) falls back to a narrow one above lo.
__device__ __forceinline__ void hist_range(float lo, float row_max, float range, float& w, float& inv_w) {
  float W = range * (row_max - lo);
  if (!(W > 0.f) || !(W < 3e38f)) W = fmaxf(fabsf(lo), 1.0f) * 1e-3f;
  w = W / (float)NBINS;
  inv_w = (float)NBINS / W;
}

// Empties a row's histogram and records the row maximum (word NBINS/2 holds its key).  All lanes.
__device__ __forceinline__ void hist_reset(uint32_t* hrow, float row_max) {
  const int lane = threadIdx.x & 31;
  for (int i = lane; i < HSTRIDE; i += 32) hrow[i] = 0u;
  __syncwarp();
  if (lane == 0) hrow[NBINS / 2] = f2key(row_max);
}

// One step of the in-place list compaction of a rebuild, an entry per lane: kept entries are written in lane order from
// buf[base] (every read of the step precedes its writes, which land at or below the entries read) and those >= lo are
// counted into the histogram.  All lanes; returns the new base.
__device__ __forceinline__ int compact_step(float2* buf, int base, float2 x, bool keep, uint32_t* hrow, float lo, float inv_w) {
  const int lane = threadIdx.x & 31;
  const unsigned bal = __ballot_sync(0xffffffffu, keep);
  if (keep) {
    __stcg(buf + base + __popc(bal & ((1u << lane) - 1u)), x);
    if (x.x >= lo) {
      const int b = (int)fminf((x.x - lo) * inv_w, (float)(NBINS - 1));
      asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(smem_u32(&hrow[b >> 1])), "r"(1u << ((b & 1) * 16)) : "memory");
    }
  }
  return base + __popc(bal);
}

// all lanes: highest bin with at least k entries at or above it (bin 0 qualifies whenever >= k entries are >= lo).
// Lane L owns histogram word L (bins 2L, 2L+1); a suffix scan over the lanes replaces a 48-step serial walk.
__device__ __forceinline__ void finish_rebuild(const uint32_t* hrow, int k, float lo, float w, float inv_w, int n_new, float* out) {
  const int lane = threadIdx.x & 31;
  const uint32_t word = lane < NBINS / 2 ? hrow[lane] : 0u;
  const int c0 = (int)(word & 0xffffu), c1 = (int)(word >> 16);
  int incl = c0 + c1;  // entries in bins >= 2 * lane after the scan
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_down_sync(0xffffffffu, incl, o);
    if (lane + o < 32) incl += v;
  }
  const int at_hi = incl - c0;  // entries in bins >= 2 * lane + 1
  const unsigned hit_hi = __ballot_sync(0xffffffffu, at_hi >= k);
  const unsigned hit_lo = __ballot_sync(0xffffffffu, incl >= k);
  int bthr = 0, A = __shfl_sync(0xffffffffu, incl, 0);
  const int Lh = hit_hi ? 31 - __clz(hit_hi) : -1, Ll = hit_lo ? 31 - __clz(hit_lo) : -1;
  if (Lh >= 0 && 2 * Lh + 1 >= 2 * Ll) {
    bthr = 2 * Lh + 1;
    A = __shfl_sync(0xffffffffu, at_hi, Lh);
  } else if (Ll >= 0) {
    bthr = 2 * Ll;
    A = __shfl_sync(0xffffffffu, incl, Ll);
  }
  if (lane == 0) {
    out[0] = lo; out[1] = w; out[2] = inv_w; out[3] = __int_as_float(bthr); out[4] = __int_as_float(A);
    out[5] = __int_as_float(n_new);
  }
}

// Warp-cooperative rebuild of one row's threshold state from its list of n (<= CAP) entries, ONE streaming pass through L2:
// given a lower bound lo of the row's k-th largest approximate score and the row maximum, the list is compacted in place
// against max(keep_threshold(lo), thr_floor) (clamp mode also keeps the k lowest item ids) and the kept entries are re-binned
// into a histogram re-centred on [lo, lo + range (row max - lo)).  Two uses:
//  - SATURATION of a row whose histogram is live: lo = the current bin edge (a valid lower bound by the histogram
//    invariant, so no selection is needed), range 2 -- finer bins, hence a tighter running threshold from here on;
//  - the first rebuild at wide k, and a bounded row (idle histogram) that filled up anyway: lo = the exact k-th largest
//    (warp_select_kth), range 4, no floor.
// Results in out[0..5] (shared memory): lo, w, inv_w, bthr, A, n_new.
__device__ __noinline__ void warp_rebuild(float2* buf, int n, int k, int clamp, int item_offset, float E, uint32_t* hrow,
                                          float lo, float row_max, float range, float thr_floor, float* out) {
  const int lane = threadIdx.x & 31;
  const float thr = fmaxf(keep_threshold(lo, E, clamp), thr_floor);
  float w, inv_w;
  hist_range(lo, row_max, range, w, inv_w);
  __syncwarp();
  hist_reset(hrow, row_max);
  int base = 0;
  for (int b0 = 0; b0 < n; b0 += 32 * 8) {
    float2 x[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      const int e = b0 + 32 * t + lane;
      x[t] = (e < n) ? __ldcg(buf + e) : make_float2(-INFINITY, 0.f);
    }
    __syncwarp();  // every read of this batch precedes its writes (writes land at or below b0)
#pragma unroll
    for (int t = 0; t < 8; ++t)
      base = compact_step(buf, base, x[t], b0 + 32 * t + lane < n && keep_entry(x[t], thr, clamp, item_offset, k), hrow, lo, inv_w);
    __syncwarp();
  }
  finish_rebuild(hrow, k, lo, w, inv_w, base, out);
  __syncwarp();
}

// the rebuild from the exact k-th largest entry (no valid lower bound of it is known): selection first, no floor
__device__ __noinline__ void warp_rebuild_selected(float2* buf, int n, int k, int clamp, int item_offset, float E, uint32_t* hrow,
                                                   int* radix, float* out) {
  float mx;
  const float kth = warp_select_kth(buf, n, k, radix, mx);
  warp_rebuild(buf, n, k, clamp, item_offset, E, hrow, kth, mx, 4.0f, -INFINITY, out);
}

// ---- FIRST (re)build of a row (n <= INIT_N entries), entirely in registers.  The entries are loaded once (CPL per lane,
// one L2 round trip) and bucketed linearly over [min, max] into 256 shared-memory counters -- low contention, where the
// radix passes of warp_select_kth pile most keys onto one exponent bucket; the bucket holding the k-th largest is
// re-bucketed once over its own [min, max].  The smallest member of the final bucket is the bound: by construction at
// least k entries are >= it, and it lies within 2^-16 of the score range of the exact k-th.  ~400 instructions per row
// where the four streaming radix passes took ~42 k cycles (25 % of a 125k-item sweep, measured with TMF_TOPK_PROF).
// Outputs as warp_rebuild.
__device__ __noinline__ void warp_rebuild_first(float2* buf, int n, int k, int clamp, int item_offset, float E, uint32_t* hrow,
                                                int* cnt256, float* out) {
  const int lane = threadIdx.x & 31;
  float2 x[CPL];
#pragma unroll
  for (int t = 0; t < CPL; ++t) {
    const int e = lane + 32 * t;
    x[t] = (e < n) ? __ldcg(buf + e) : make_float2(-INFINITY, 0.f);
  }
  unsigned mem = 0;  // bit t: entry t can still be the k-th largest
  float mn = INFINITY, mx = -INFINITY;
#pragma unroll
  for (int t = 0; t < CPL; ++t) {
    if (lane + 32 * t < n) { mem |= 1u << t; mn = fminf(mn, x[t].x); mx = fmaxf(mx, x[t].x); }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  const float row_max = mx;
  float lo_b = mn, hi_b = mx;
  int krem = min(k, n);
#pragma unroll 1
  for (int level = 0; level < 2 && hi_b > lo_b; ++level) {
    const float scale = 256.0f / (hi_b - lo_b);
#pragma unroll
    for (int i = 0; i < 8; ++i) cnt256[lane * 8 + i] = 0;
    __syncwarp();
    int bk[CPL];
#pragma unroll
    for (int t = 0; t < CPL; ++t) {
      bk[t] = (int)fminf(fmaxf((x[t].x - lo_b) * scale, 0.f), 255.f);
      if ((mem >> t) & 1u) smem_inc(&cnt256[bk[t]]);
    }
    __syncwarp();
    const int bin = pick_bin(cnt256, krem);  // the members number >= krem
    float nlo = INFINITY, nhi = -INFINITY;
#pragma unroll
    for (int t = 0; t < CPL; ++t) {
      if (((mem >> t) & 1u) && bk[t] == bin) { nlo = fminf(nlo, x[t].x); nhi = fmaxf(nhi, x[t].x); }
      else mem &= ~(1u << t);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      nlo = fminf(nlo, __shfl_xor_sync(0xffffffffu, nlo, o));
      nhi = fmaxf(nhi, __shfl_xor_sync(0xffffffffu, nhi, o));
    }
    lo_b = nlo; hi_b = nhi;
    __syncwarp();
  }
  const float kth = lo_b;  // >= k entries are >= kth
  const float thr = keep_threshold(kth, E, clamp);
  float w, inv_w;
  hist_range(kth, row_max, 4.0f, w, inv_w);
  hist_reset(hrow, row_max);
  int base = 0;
#pragma unroll
  for (int t = 0; t < CPL; ++t)
    base = compact_step(buf, base, x[t], lane + 32 * t < n && keep_entry(x[t], thr, clamp, item_offset, k), hrow, kth, inv_w);
  __syncwarp();
  finish_rebuild(hrow, k, kth, w, inv_w, base, out);
  __syncwarp();
}

// ------------------------------------------------------------------ the fused kernel
// Byte offsets of the kernel's dynamic shared memory from a 1024-byte aligned base (the swizzled operand tiles need it).
// The kernel carves with it and the host sizes the allocation with it (total + 1024 bytes of room to align the base).
struct TopkSmem { int b, bars, tmem_slot, hist, queues, rebuild_out, total; };
__host__ __device__ __forceinline__ TopkSmem topk_smem(int kb) {
  TopkSmem s;
  s.b = kb * A_SUB_BYTES;                                      // A: kb sub-tiles of [BM][64] bf16
  s.bars = s.b + NSTAGES * B_STAGE_BYTES;                      // B: NSTAGES x [BN][64] bf16
  s.tmem_slot = s.bars + (2 * NSTAGES + 6) * 8;                // mbarriers: full/empty per stage, A full/empty, TMEM full/empty x2
  s.hist = s.tmem_slot + 16;                                   // [BM][HSTRIDE] per-row score histograms
  s.queues = (s.hist + BM * HSTRIDE * 4 + 15) & ~15;           // [BM][QCAP] survivor queues
  s.rebuild_out = s.queues + BM * QCAP * 8;                    // [4 warps][8] rebuild results
  s.total = s.rebuild_out + 4 * 8 * 4;
  return s;
}

// WIDE: the configuration for 128 < k <= 1024 (CAP_W list slots, first rebuild by warp_rebuild_selected)
// MASK: the rows' excluded ids (p.ex_ptr / p.ex_idx) never reach a list or a histogram; the cursors need EXCUR_BYTES per
// row of dynamic shared memory beyond topk_smem(kb).total
template <bool DUMP, bool PROF, bool WIDE, bool MASK = false>
__global__ void __launch_bounds__(TOPK_THREADS, 2)
score_topk_kernel(const __grid_constant__ CUtensorMap tmapU, const __grid_constant__ CUtensorMap tmapV, const TopkParams p) {
  constexpr int cap = WIDE ? CAP_W : CAP;
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const TopkSmem S = topk_smem(p.kb);
  unsigned char* sA = smem;
  unsigned char* sB = smem + S.b;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S.bars);
  uint64_t* full_bar = bars;                  // [NSTAGES]
  uint64_t* empty_bar = bars + NSTAGES;       // [NSTAGES]
  uint64_t* a_full = bars + 2 * NSTAGES;      // [1]
  uint64_t* a_empty = a_full + 1;             // [1]
  uint64_t* tfull = a_empty + 1;              // [2]
  uint64_t* tempty = tfull + 2;               // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + S.tmem_slot);
  uint32_t* hist_rows = reinterpret_cast<uint32_t*>(smem + S.hist);
  float2* queues = reinterpret_cast<float2*>(smem + S.queues);
  float* init_out = reinterpret_cast<float*>(smem + S.rebuild_out);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  auto now = [] () -> long long { return PROF ? clock64() : 0ll; };  // cycle counters only in the profiling build

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmapU) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmapV) : "memory");
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < NSTAGES; ++s) { mbar_init(smem_u32(&full_bar[s]), 1); mbar_init(smem_u32(&empty_bar[s]), 1); }
    mbar_init(smem_u32(a_full), 1);
    mbar_init(smem_u32(a_empty), 1);
    for (int s = 0; s < 2; ++s) { mbar_init(smem_u32(&tfull[s]), 1); mbar_init(smem_u32(&tempty[s]), 128); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {  // TMEM: 256 columns = two 128x128 fp32 accumulators (the SM's other CTA takes the other half)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0, a_phase = 0;
      for (int ub = blockIdx.x; ub < p.n_ublocks; ub += gridDim.x) {
        long long t0 = now();
        mbar_wait(smem_u32(a_empty), a_phase ^ 1);  // previous user block's MMAs retired
        long long w_empty = 0, w_aempty = now() - t0;
        mbar_expect_tx(smem_u32(a_full), p.kb * A_SUB_BYTES);
        for (int kb = 0; kb < p.kb; ++kb)
          tma_load_2d(smem_u32(sA + kb * A_SUB_BYTES), &tmapU, kb * BK, (p.ub0 + ub) * BM, smem_u32(a_full));
        a_phase ^= 1;
        for (int nt = 0; nt < p.n_tiles; ++nt) {
          for (int kb = 0; kb < p.kb; ++kb) {
            t0 = now();
            mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1);
            w_empty += now() - t0;
            mbar_expect_tx(smem_u32(&full_bar[stage]), B_STAGE_BYTES);
            tma_load_2d(smem_u32(sB + stage * B_STAGE_BYTES), &tmapV, kb * BK, nt * BN, smem_u32(&full_bar[stage]));
            if (++stage == NSTAGES) { stage = 0; phase ^= 1; }
          }
        }
        if (PROF) { atomicAdd(p.prof + 0, (unsigned long long)w_empty); atomicAdd(p.prof + 1, (unsigned long long)w_aempty); }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer: the whole warp runs the loop, one elected lane issues =====================
    {
      int stage = 0, acc = 0;
      uint32_t phase = 0, acc_phase = 0, a_phase = 0;
      // operand format bits of the instruction descriptor: a_format (bit 7) / b_format (bit 10): 1 = bf16, 0 = fp16
      const bool f16 = p.force_fmt >= 0 ? p.force_fmt == 1 : use_fp16(p.fmt_stats);
      const uint32_t idesc = f16 ? (kIdesc & ~((1u << 7) | (1u << 10))) : kIdesc;
      const uint64_t a_desc0 = umma_desc_sw128(smem_u32(sA));  // + (byte offset >> 4): sub-tile / k-slice (no carry out of the 14-bit field)
      const uint64_t b_desc0 = umma_desc_sw128(smem_u32(sB));
      for (int ub = blockIdx.x; ub < p.n_ublocks; ub += gridDim.x) {
        mbar_wait(smem_u32(a_full), a_phase);
        a_phase ^= 1;
        long long w_tempty = 0, w_full = 0;
        for (int nt = 0; nt < p.n_tiles; ++nt) {
          long long t0 = now();
          mbar_wait(smem_u32(&tempty[acc]), acc_phase ^ 1);  // epilogue drained this accumulator
          w_tempty += now() - t0;
          __syncwarp();
          tcgen05_fence_after();
          const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
          for (int kb = 0; kb < p.kb; ++kb) {
            t0 = now();
            mbar_wait(smem_u32(&full_bar[stage]), phase);
            w_full += now() - t0;
            __syncwarp();
            tcgen05_fence_after();
            const uint64_t a_desc = a_desc0 + (uint64_t)((kb * A_SUB_BYTES) >> 4);
            const uint64_t b_desc = b_desc0 + (uint64_t)((stage * B_STAGE_BYTES) >> 4);
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k)
              tcgen05_mma_f16_elect(d_tmem, a_desc + (uint64_t)(k * (UMMA_K * 2 / 16)), b_desc + (uint64_t)(k * (UMMA_K * 2 / 16)), idesc,
                                    (uint32_t)((kb | k) != 0));
            tcgen05_commit_elect(smem_u32(&empty_bar[stage]));  // frees the smem slot when these MMAs retire
            if (++stage == NSTAGES) { stage = 0; phase ^= 1; }
          }
          tcgen05_commit_elect(smem_u32(&tfull[acc]));  // accumulator ready for the epilogue
          acc ^= 1;
          if (acc == 0) acc_phase ^= 1;
        }
        tcgen05_commit_elect(smem_u32(a_empty));  // A tile may be overwritten
        if (PROF && lane == 0) { atomicAdd(p.prof + 2, (unsigned long long)w_tempty); atomicAdd(p.prof + 3, (unsigned long long)w_full); }
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue: threshold filter + survivor queues + SIMD list maintenance =====================
    const int q = warp - 4;  // TMEM lane quarter == warp % 4
    int* radix = reinterpret_cast<int*>(queues + q * 32 * QCAP);  // radix-select scratch aliases the warp's (empty) queues
    const uint32_t hrow = smem_u32(hist_rows + (q * 32 + lane) * HSTRIDE);
    const uint32_t queue = smem_u32(queues + (q * 32 + lane) * QCAP);
    const uint32_t excur = smem_u32(smem + S.total + (q * 32 + lane) * EXCUR_BYTES);
    float* iout = init_out + q * 8;
    const int n_items = (int)p.n_items;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int ub = blockIdx.x; ub < p.n_ublocks; ub += gridDim.x) {
      const long long lrow = (long long)ub * BM + q * 32 + lane;       // batch-local row (candidate buffers)
      const long long row = (long long)p.ub0 * BM + lrow;              // global row
      const bool valid = row < p.n_users;
      RowState st;
      st.thr = valid ? -INFINITY : INFINITY;
      st.lo = 0.f; st.w = 0.f; st.inv_w = 0.f;
      st.E = p.erow[row];
      st.cnt = 0; st.cq = 0; st.bthr = 0; st.A = 0;
      bool warp_inited = false;
      if constexpr (MASK) {  // cursor at the row's first excluded id >= item_offset
        int pos = 0, end = 0;
        if (valid) {
          pos = p.ex_ptr[row];
          end = p.ex_ptr[row + 1];
          for (int hi = end; pos < hi;) {
            const int mid = (pos + hi) >> 1;
            if (p.ex_idx[mid] < p.item_offset) pos = mid + 1; else hi = mid;
          }
        }
        sts_u32(excur, (uint32_t)pos);
        sts_u32(excur + 4u, (uint32_t)end);
        sts_u32(excur + 8u, (uint32_t)(pos < end ? p.ex_idx[pos] : INT_MAX));
      }
      // External bound (item-sharded scoring): B = a lower bound of the row's k-th best CANONICAL score over all
      // slabs, so a member of the global top-k has s~ >= B - E.  Clamp mode: only a positive bound says anything
      // (with B <= 0 the zero-score fillers matter).  When every valid row of the warp has such a floor the
      // warm-up (3 unfiltered tiles + radix-select rebuild per row) is skipped: the rows start filtering at the
      // floor with an idle histogram (lo = +inf); a list that still fills up heals through the usual rebuild.
      st.thr_ext = -INFINITY;
      if (!DUMP && p.row_bound != nullptr) {
        if (valid) {
          const float B = p.row_bound[row];
          if (B > -INFINITY && (!p.clamp || B > 0.f)) st.thr_ext = B - st.E;
        }
        if (__all_sync(0xffffffffu, !valid || st.thr_ext > -INFINITY)) {
          warp_inited = true;
          if (valid) st.thr = st.thr_ext;
          st.lo = INFINITY;
        }
      }
      float2* buf = p.cand + lrow * cap;
      long long w_tfull = 0, w_work = 0, w_init = 0;
      for (int nt = 0; nt < p.n_tiles; ++nt) {
        long long t0 = now();
        mbar_wait(smem_u32(&tfull[acc]), acc_phase);
        __syncwarp();  // tcgen05.ld is warp-collective: reconverge after the per-lane spin
        long long t1 = now();
        w_tfull += t1 - t0;
        tcgen05_fence_after();
        const uint32_t t_base = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN);
        if (!DUMP && warp_inited && TMF_DBG(p) < 2) {
          epilogue_tile<cap, MASK>(t_base, nt * BN, st, queue, buf, hrow, p, excur);
        } else if (TMF_DBG(p) < 3) {
          uint32_t ra[32], rb[32];
          tmem_ld32(t_base, ra);
#pragma unroll 1
          for (int ch = 0; ch < BN / 32; ch += 2) {
            // chunk ch is in ra; chunk ch+1 is fetched into rb while ra is filtered (and vice versa)
            tmem_ld_wait_for(ra);
            tmem_ld32(t_base + (uint32_t)((ch + 1) * 32), rb);
            epilogue_chunk<DUMP, MASK>(ra, nt * BN + ch * 32, n_items, valid, warp_inited, st, queue, buf, hrow, row, p, excur);
            tmem_ld_wait_for(rb);
            if (ch + 2 < BN / 32) tmem_ld32(t_base + (uint32_t)((ch + 2) * 32), ra);
            epilogue_chunk<DUMP, MASK>(rb, nt * BN + (ch + 1) * 32, n_items, valid, warp_inited, st, queue, buf, hrow, row, p, excur);
          }
        }
        // accumulator drained: hand it back to the MMA warp before any list maintenance
        tcgen05_fence_before();
        mbar_arrive(smem_u32(&tempty[acc]));
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
        long long t2 = now();
        w_work += t2 - t1;
        if (!DUMP) {
          if (__any_sync(0xffffffffu, st.cq >= QCAP / 2)) {
            const long long td = now();
            drain_queues<cap, MASK>(st, queue, buf, hrow, p.k, p.clamp, excur, p.ex_idx);
            if (PROF && lane == 0) { atomicAdd(p.prof + 10, (unsigned long long)(now() - td)); atomicAdd(p.prof + 11, 1ull); }
          }
          // (re)build: the first time once a row holds INIT_N - BN entries (wide: k + 2 tiles; all valid rows of a warp
          // get there at the same tile because everything is appended until then), later whenever a list is about to saturate.
          // MASK: a row left without a threshold by the first rebuild (lo = +inf, see below) is rebuilt by the full selection
          // as soon as it holds k entries, so it grows at most a tile and a queue beyond k unfiltered and the saturation
          // margin below holds for it as for every other row.
          const int first_n = WIDE ? p.k + 2 * BN : INIT_N - BN;
          const bool first = !warp_inited && __any_sync(0xffffffffu, valid && st.cnt >= first_n);
          auto unbounded = [&]() { return MASK && warp_inited && st.lo == INFINITY && st.cnt >= p.k; };
          unsigned need = __ballot_sync(0xffffffffu, valid && st.cnt <= cap &&
                                                         (first || (warp_inited && st.cnt > cap - 4 * QCAP) || unbounded()));
          if (need) {  // the radix scratch aliases the queues: empty them first (lengths may grow a little)
            const long long tq = now();
            drain_queues<cap, MASK>(st, queue, buf, hrow, p.k, p.clamp, excur, p.ex_idx);
            if (PROF && lane == 0) { atomicAdd(p.prof + 19, (unsigned long long)(now() - tq)); atomicAdd(p.prof + 18, 1ull); }
            need = __ballot_sync(0xffffffffu, valid && st.cnt <= cap &&
                                                  (first || (warp_inited && st.cnt > cap - 4 * QCAP) || unbounded()));
          }
          while (need) {
            const int owner = __ffs(need) - 1;
            need &= need - 1;
            const int n_o = __shfl_sync(0xffffffffu, st.cnt, owner);
            const float E_o = __shfl_sync(0xffffffffu, st.E, owner);
            __syncwarp();
            float2* obuf = p.cand + ((long long)ub * BM + q * 32 + owner) * cap;
            uint32_t* ohist = hist_rows + (q * 32 + owner) * HSTRIDE;
            const float lo_o = __shfl_sync(0xffffffffu, st.lo, owner);
            // MASK: list lengths differ per row (excluded ids are never listed), so the warp's first rebuild can meet a row
            // that holds fewer than k entries.  No lower bound of its k-th best unseen score exists yet: the row keeps no
            // threshold (every entry is listed, so it stays exact) and an idle histogram (lo = +inf) until it holds k
            // entries; then the trigger above gives it the full selection below.
            if (MASK && n_o < p.k) {
              if (lane == owner) {
                st.thr = st.thr_ext;
                st.lo = INFINITY;
                st.bthr = 0;
                st.A = 0;
              }
              __syncwarp();
              continue;
            }
            const long long tr = now();
            int which = 0;
            if (!WIDE && first && n_o <= INIT_N) {
              warp_rebuild_first(obuf, n_o, p.k, p.clamp, p.item_offset, E_o, ohist, radix, iout);
            } else if (lo_o < INFINITY && !first) {  // live histogram: compaction + re-centring in one pass
              which = 1;
              const float w_o = __shfl_sync(0xffffffffu, st.w, owner);
              const int bthr_o = __shfl_sync(0xffffffffu, st.bthr, owner);
              const float ext_o = __shfl_sync(0xffffffffu, st.thr_ext, owner);
              warp_rebuild(obuf, n_o, p.k, p.clamp, p.item_offset, E_o, ohist, bin_edge(lo_o, w_o, bthr_o), key2f(ohist[NBINS / 2]), 2.0f,
                           ext_o, iout);
            } else {  // first rebuild at wide k, or a bounded row (idle histogram) that filled up anyway: full selection
              which = 2;
              warp_rebuild_selected(obuf, n_o, p.k, p.clamp, p.item_offset, E_o, ohist, radix, iout);
            }
            if (PROF && lane == 0) { atomicAdd(p.prof + 13 + 2 * which, (unsigned long long)(now() - tr)); atomicAdd(p.prof + 12 + 2 * which, 1ull); }
            if (lane == owner) {
              st.lo = iout[0]; st.w = iout[1]; st.inv_w = iout[2];
              st.bthr = __float_as_int(iout[3]); st.A = __float_as_int(iout[4]);
              st.cnt = __float_as_int(iout[5]);
              st.thr = fmaxf(edge_threshold(st.lo, st.w, st.bthr, st.E, p.clamp), st.thr_ext);
              if (st.cnt > cap - 8 * QCAP) {  // cannot shrink (massive ties): hand the row to the exact path
                st.cnt = cap + 1;
                st.thr = INFINITY;
              }
            }
            __syncwarp();
          }
          if (first) warp_inited = true;
        }
        w_init += now() - t2;
      }
      if (!DUMP) drain_queues<cap, MASK>(st, queue, buf, hrow, p.k, p.clamp, excur, p.ex_idx);
      if (PROF && lane == 0) {
        atomicAdd(p.prof + 4, (unsigned long long)w_tfull); atomicAdd(p.prof + 5, (unsigned long long)w_work);
        atomicAdd(p.prof + 6, (unsigned long long)w_init); atomicAdd(p.prof + 7, 1ull);
      }
      if (PROF) atomicAdd(p.prof + 20, (unsigned long long)(valid ? min(st.cnt, cap) : 0));
      const bool ovf = st.cnt > cap;
      if (valid && ovf) {
        const int slot = atomicAdd(p.ovf_count, 1);
        p.ovf_rows[slot] = (int)row;
        if (PROF) atomicAdd(p.prof + 8, 1ull);
      }
      p.cnt[lrow] = valid ? (ovf ? -1 : st.cnt) : 0;
      p.thr_out[lrow] = st.thr;
      __syncwarp();
    }
  }

  __syncthreads();
  if (warp == 2) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------ final selection + canonical rerank
constexpr int RR_WARPS = 8;
constexpr int SEL_CAP = 512;   // survivors per row the rerank can rank; more -> exact path
constexpr int RR_CHAINS = 4;   // independent fp64 FMA chains per lane
// wide k: room for the ~k + near-ties survivors of k = 1024 (16 KB of keys per warp), 4 warps so two CTAs share an SM
constexpr int RR_WARPS_W = 4;
constexpr int SEL_CAP_W = 2048;

struct RerankParams {
  long long n_users, n_items, row0;  // rows [row0, row0 + n_rows) are batch-local rows [0, n_rows)
  long long n_rows;
  int k, clamp, item_offset, r, ld;
  const float* U;
  const float* V;
  const float* erow;
  const float2* cand;
  const int* cnt;
  const float* thr;
  int* ovf_count;
  int* ovf_rows;
  unsigned long long* prof;
  int* out_idx;
  float* out_score;
  const int* ex_ptr;  // masked top-k: CSR of the excluded global item ids (exact_rows_kernel only), else NULL
  const int* ex_idx;
};

// Streams a row's list of n entries from global memory (DEPTH loads in flight per lane) and gathers those that pass
// keep_entry into pr[0, SEL_CAP), in list order.  Returns how many passed: beyond SEL_CAP they are counted, not stored.
template <int SEL_CAP, int DEPTH>
__device__ __forceinline__ int gather_kept(const float2* buf, int n, float thr, int clamp, int item_offset, int k, float2* pr) {
  const int lane = threadIdx.x & 31;
  const unsigned lt = (1u << lane) - 1u;
  int m = 0;
  for (int b0 = 0; b0 < n; b0 += 32 * DEPTH) {
    float2 x[DEPTH];
#pragma unroll
    for (int t = 0; t < DEPTH; ++t) {
      const int e = b0 + 32 * t + lane;
      x[t] = (e < n) ? __ldcg(buf + e) : make_float2(-INFINITY, 0.f);
    }
#pragma unroll
    for (int t = 0; t < DEPTH; ++t) {
      const bool keep = b0 + 32 * t + lane < n && keep_entry(x[t], thr, clamp, item_offset, k);
      const unsigned bal = __ballot_sync(0xffffffffu, keep);
      const int pos = m + __popc(bal & lt);
      if (keep && pos < SEL_CAP) pr[pos] = x[t];
      m += __popc(bal);
    }
  }
  return m;
}

constexpr int STG_COLS = 64;              // fp32 components per staged slice of an item row
constexpr int STG_STRIDE = STG_COLS + 4;  // floats; 272-byte rows keep the per-lane float4 reads conflict-free

// One warp per user row.
//  1. the row's candidate list is streamed ONCE from global memory; entries that pass the main kernel's final
//     threshold (a superset of the answer, ~2k of them) land in shared memory;
//  2. the exact k-th largest approximate score of that superset tightens the threshold (k-th - 2E) -> ~1.5k candidates;
//  3. the candidates' fp32 item rows are staged through shared memory by per-lane bulk async copies (one 256-byte
//     copy per candidate and slice: 8 KB in flight per warp, where the per-lane strided loads of the first version
//     exposed a full DRAM latency every 16 bytes), and every lane runs ONE candidate's fp64 FMA chain in
//     component order -- bit-identical to oracle.canonical_scores;
//  4. (score, id) are packed into one 64-bit key and ranked by counting (branch-free, O(m^2)); the wide configuration
//     (m up to SEL_CAP_W) orders the keys by a bitonic sort in shared memory instead (O(m log^2 m)).
template <bool WIDE>
__host__ __device__ __forceinline__ size_t rerank_warp_smem(int ld) {
  return (size_t)ld * sizeof(double) + (WIDE ? SEL_CAP_W : SEL_CAP) * 8 + 32 * STG_STRIDE * 4 + 16;
}
template <bool WIDE>
__global__ void __launch_bounds__((WIDE ? RR_WARPS_W : RR_WARPS) * 32) rerank_kernel(const RerankParams p) {
  constexpr int RR_WARPS = WIDE ? RR_WARPS_W : tmf::RR_WARPS;
  constexpr int SEL_CAP = WIDE ? SEL_CAP_W : tmf::SEL_CAP;
  constexpr int CAP = WIDE ? CAP_W : tmf::CAP;
  extern __shared__ __align__(16) unsigned char rr_smem[];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t per_warp = rerank_warp_smem<WIDE>(p.ld);
  unsigned char* base = rr_smem + (size_t)w * per_warp;
  double* ud = reinterpret_cast<double*>(base);                       // [ld] this user's row, widened once
  float2* pr = reinterpret_cast<float2*>(ud + p.ld);                  // [SEL_CAP] (approx score, id), later 64-bit rank keys
  float* stg = reinterpret_cast<float*>(pr + SEL_CAP);                // [32][STG_STRIDE] staged item-row slices
  int* radix = reinterpret_cast<int*>(stg);                           // radix-select scratch before staging starts
  uint64_t* bar = reinterpret_cast<uint64_t*>(stg + 32 * STG_STRIDE); // this warp's copy-completion barrier
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(pr);

  const long long lrow = (long long)blockIdx.x * RR_WARPS + w;
  if (lrow >= p.n_rows) return;
  const long long row = p.row0 + lrow;
  const int n = p.cnt[lrow];
  if (n < 0) return;  // overflowed in the main kernel: exact_rows_kernel owns it
  const float2* buf = p.cand + lrow * CAP;
  const int k = p.k;
  const unsigned lt = (1u << lane) - 1u;
  if (lane == 0) mbar_init(smem_u32(bar), 1);
  for (int c = lane; c < p.ld; c += 32) ud[c] = (double)p.U[row * p.ld + c];
  float thr = p.thr[lrow];
  // ---- 1. superset by the main kernel's final threshold (or the clamp-mode filler rule)
  int m = gather_kept<SEL_CAP, 8>(buf, n, thr, p.clamp, p.item_offset, k, pr);
  __syncwarp();
  // ---- 2. exact k-th largest approximate score -> final keep-threshold, compact in place
  if (n > k && m > k) {  // (m <= k: an externally bounded row with few local candidates keeps them all)
    float kth;
    if (m <= SEL_CAP) {
      kth = radix_select_kth(k, radix, [&](int shift, uint32_t mask, uint32_t prefix) {
        for (int e = lane; e < m; e += 32) count_key(radix, pr[e].x, shift, mask, prefix);
      });
    } else {  // loose running threshold (badly placed histogram): select over the whole list in global memory
      float mx;
      kth = warp_select_kth(buf, n, k, radix, mx);
    }
    const float E = p.erow[row];
    thr = fmaxf(thr, keep_threshold(kth, E, p.clamp));
    // Clamp mode, wide k: with kth - 2E > 0 at least k listed items score above zero, so no zero-score filler can be in the
    // answer and the k lowest ids are kept only on their own merit (kept unconditionally they would double m past SEL_CAP_W).
    const bool fill = p.clamp && !(WIDE && kth - 2.f * E > 0.f);
    if (m <= SEL_CAP) {
      int m2 = 0;
      for (int e0 = 0; e0 < m; e0 += 32) {
        const int e = e0 + lane;
        const float2 x = e < m ? pr[e] : make_float2(-INFINITY, 0.f);
        const bool keep = e < m && keep_entry(x, thr, fill, p.item_offset, k);
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        __syncwarp();  // all reads of this batch precede its writes (which land at or below e0)
        if (keep) pr[m2 + __popc(bal & lt)] = x;
        m2 += __popc(bal);
      }
      m = m2;
    } else {
      m = gather_kept<SEL_CAP, 4>(buf, n, thr, fill, p.item_offset, k, pr);
    }
  }
  if (m > SEL_CAP) {  // too many near-ties to rank here
    if (lane == 0) {
      if (p.prof) atomicAdd(p.prof + 9, 1ull);
      const int slot = atomicAdd(p.ovf_count, 1);
      p.ovf_rows[slot] = (int)row;
    }
    return;
  }
  __syncwarp();
  // ---- 3. canonical scores: 32 candidates per batch, item rows staged slice by slice
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  uint32_t parity = 0;
  const int n_slices = (p.ld + STG_COLS - 1) / STG_COLS;
  for (int t0 = 0; t0 < m; t0 += 32) {
    const int t = t0 + lane;
    const bool have = t < m;
    const int item = have ? __float_as_int(pr[t].y) : 0;
    const float* vrow = p.V + (long long)(item - p.item_offset) * p.ld;
    const int nb = min(32, m - t0);
    double acc = 0.0;
    for (int sl = 0; sl < n_slices; ++sl) {
      const int c0 = sl * STG_COLS;
      const int ncol = min(STG_COLS, p.ld - c0);  // multiple of 4
      // the previous slice's shared-memory reads (generic proxy) must be ordered before the async-proxy writes
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_expect_tx(smem_u32(bar), (uint32_t)(nb * ncol * 4));
      __syncwarp();
      if (have) {
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(smem_u32(stg + lane * STG_STRIDE)), "l"(vrow + c0), "r"(ncol * 4), "r"(smem_u32(bar))
                     : "memory");
      }
      mbar_wait(smem_u32(bar), parity);
      parity ^= 1;
      const float4* mine = reinterpret_cast<const float4*>(stg + lane * STG_STRIDE);
      const double2* u2 = reinterpret_cast<const double2*>(ud + c0);
#pragma unroll 4
      for (int c4 = 0; c4 < ncol / 4; ++c4) {
        const float4 x = mine[c4];
        const double2 ua = u2[2 * c4], ub = u2[2 * c4 + 1];
        acc = fma(ua.x, (double)x.x, acc);
        acc = fma(ua.y, (double)x.y, acc);
        acc = fma(ub.x, (double)x.z, acc);
        acc = fma(ub.y, (double)x.w, acc);
      }
    }
    if (have) {
      float sc = (float)acc;
      if (p.clamp) sc = sc > 0.f ? sc : 0.f;  // tf.where(p > 0, p, 0.0)
      sc = sc + 0.0f;                         // -0 -> +0 like the oracle
      keys[t] = ((unsigned long long)f2key(sc) << 32) | (unsigned long long)(0xffffffffu - (uint32_t)item);
    }
  }
  __syncwarp();
  if (WIDE) {
    // ---- 4'. bitonic sort, descending: larger key = (higher score, then lower item id); zero keys pad to a power of two
    int np2 = 1;
    while (np2 < m) np2 <<= 1;
    for (int t = m + lane; t < np2; t += 32) keys[t] = 0ull;
    __syncwarp();
    for (int size = 2; size <= np2; size <<= 1) {
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        for (int i = lane; i < np2 / 2; i += 32) {
          const int a = 2 * i - (i & (stride - 1));  // partner pair (a, a + stride), bit `stride` of a clear
          const unsigned long long ka = keys[a], kb = keys[a + stride];
          if ((ka < kb) == ((a & size) == 0)) { keys[a] = kb; keys[a + stride] = ka; }
        }
        __syncwarp();
      }
    }
    for (int t = lane; t < min(m, k); t += 32) {
      const unsigned long long kt = keys[t];
      p.out_idx[row * k + t] = (int)(0xffffffffu - (uint32_t)(kt & 0xffffffffull));
      p.out_score[row * k + t] = key2f((uint32_t)(kt >> 32));
    }
  } else {
    // ---- 4. rank by counting: larger key = (higher score, then lower item id); ids are distinct so ranks are too
    for (int g0 = 0; g0 < m; g0 += 128) {
      unsigned long long mk[4];
      int rank[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int t = g0 + 32 * i + lane;
        mk[i] = t < m ? keys[t] : ~0ull;
        rank[i] = 0;
      }
      for (int o = 0; o < m; ++o) {
        const unsigned long long ko = keys[o];
#pragma unroll
        for (int i = 0; i < 4; ++i) rank[i] += ko > mk[i] ? 1 : 0;
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int t = g0 + 32 * i + lane;
        if (t < m && rank[i] < k) {
          p.out_idx[row * k + rank[i]] = (int)(0xffffffffu - (uint32_t)(mk[i] & 0xffffffffull));
          p.out_score[row * k + rank[i]] = key2f((uint32_t)(mk[i] >> 32));
        }
      }
    }
  }
  // fewer than k local candidates (only with an external bound): pad with entries that lose every comparison
  for (int t = m + lane; t < k; t += 32) {
    p.out_idx[row * k + t] = 0x7fffffff;
    p.out_score[row * k + t] = -INFINITY;
  }
}

// exact path for rows whose candidate list overflowed (huge tie groups, adversarially ordered scores): all
// canonical scores of the row go to scratch; a block-wide radix select finds the k-th largest score T; entries > T
// plus the lowest-indexed entries == T are collected (k in total) and ranked by (score desc, id asc).
// Masked top-k (p.ex_ptr set, raw scores): excluded items score -inf and only the kk = min(k, unseen items) best are
// selected; slots [kk, k) are padded with (-inf, INT32_MAX).
// (At most 32 CTAs run it, so registers matter more than occupancy: minimum 1 block per SM.)
__global__ void __launch_bounds__(256, 1) exact_rows_kernel(const RerankParams p, const int* __restrict__ ovf_count,
                                                         const int* __restrict__ ovf_rows, float* __restrict__ scratch) {
  __shared__ int hist[256];
  __shared__ int s_bin, s_krem, s_cnt_gt, s_cnt_eq, s_warp_tot[8], s_n_ex;
  __shared__ float sel_s[WIDE_MAX_K];
  __shared__ int sel_i[WIDE_MAX_K];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int n_ovf = *ovf_count;
  const int n = (int)p.n_items;
  const int k = p.k;
  float* sc = scratch + (long long)blockIdx.x * p.n_items;
  for (int o = blockIdx.x; o < n_ovf; o += gridDim.x) {
    const long long row = ovf_rows[o];
    const float* u = p.U + row * p.ld;
    if (tid == 0) s_n_ex = 0;
    for (int i = tid; i < n; i += 256) {
      const float* v = p.V + (long long)i * p.ld;
      double acc = 0.0;
      for (int c = 0; c < p.r; ++c) acc = fma((double)u[c], (double)v[c], acc);
      float s = (float)acc;
      if (p.clamp) s = s > 0.f ? s : 0.f;
      sc[i] = s + 0.0f;
    }
    __syncthreads();
    if (p.ex_ptr != nullptr) {
      int n_ex = 0;
      for (int e = p.ex_ptr[row] + tid; e < p.ex_ptr[row + 1]; e += 256) {
        const int i = p.ex_idx[e] - p.item_offset;
        if (i >= 0 && i < n && atomicExch(&sc[i], -INFINITY) != -INFINITY) ++n_ex;  // a repeated id counts once
      }
      atomicAdd(&s_n_ex, n_ex);
      __syncthreads();
    }
    const int kk = min(k, n - s_n_ex);
    for (int t = kk + tid; t < k; t += 256) {
      p.out_idx[row * k + t] = 0x7fffffff;
      p.out_score[row * k + t] = -INFINITY;
    }
    if (kk == 0) {  // block-uniform; every thread has read s_n_ex before the next row resets it
      __syncthreads();
      continue;
    }
    // ---- kk-th largest key, 8 bits per pass
    uint32_t prefix = 0, mask = 0;
    int krem = kk;
    for (int shift = 24; shift >= 0; shift -= 8) {
      hist[tid] = 0;
      __syncthreads();
      for (int i = tid; i < n; i += 256) {
        const uint32_t key = f2key(sc[i]);
        if ((key & mask) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1);
      }
      __syncthreads();
      if (tid == 0) {
        int cum = 0, b = 255;
        for (; b > 0; --b) {
          if (cum + hist[b] >= krem) break;
          cum += hist[b];
        }
        s_bin = b;
        s_krem = krem - cum;
      }
      __syncthreads();
      prefix |= (uint32_t)s_bin << shift;
      mask |= 255u << shift;
      krem = s_krem;
      __syncthreads();
    }
    const float T = key2f(prefix);  // exactly the kk-th largest score; krem of the entries == T are needed
    if (tid == 0) { s_cnt_gt = 0; s_cnt_eq = 0; }
    __syncthreads();
    // ---- collect: every entry > T (kk - krem of them), and the krem lowest-indexed entries == T (ordered scan)
    for (int i0 = 0; i0 < n; i0 += 256) {
      const int i = i0 + tid;
      const float s = i < n ? sc[i] : -INFINITY;
      const bool gt = i < n && s > T;
      const bool eq = i < n && s == T;
      if (gt) {
        const int pos = atomicAdd(&s_cnt_gt, 1);
        sel_s[pos] = s;
        sel_i[pos] = i;
      }
      const unsigned beq = __ballot_sync(0xffffffffu, eq);
      if (lane == 0) s_warp_tot[wid] = __popc(beq);
      __syncthreads();
      int before = s_cnt_eq;
      for (int w2 = 0; w2 < wid; ++w2) before += s_warp_tot[w2];
      const int my = before + __popc(beq & ((1u << lane) - 1u));
      if (eq && my < krem) {  // slots [kk - krem, kk) hold the tied entries in index order
        sel_s[kk - krem + my] = s;
        sel_i[kk - krem + my] = i;
      }
      __syncthreads();
      if (tid == 0) {
        int tot = 0;
        for (int w2 = 0; w2 < 8; ++w2) tot += s_warp_tot[w2];
        s_cnt_eq += tot;
      }
      __syncthreads();
    }
    // ---- rank the kk selected entries
    for (int t = tid; t < kk; t += 256) {
      const float s = sel_s[t];
      const int id = sel_i[t];
      int rank = 0;
      for (int j = 0; j < kk; ++j) rank += (sel_s[j] > s) || (sel_s[j] == s && sel_i[j] < id);
      p.out_idx[row * k + rank] = id + p.item_offset;
      p.out_score[row * k + rank] = s;
    }
    __syncthreads();
  }
}

// Clamp mode of the masked top-k.  The main kernel, the rerank and the exact path rank each row's unseen items by RAW score;
// the clamped ranking (max(s, 0) desc, id asc) differs only where the k-th raw score is <= 0.  Such a row holds all of its
// m < k unseen items with a positive score, in order, and the clamped answer continues with zero-score ties: the lowest
// unseen ids of the slab not among those m (+0.0 each), then padding.  One warp per row.
constexpr int FILL_WARPS = 4;
__device__ __forceinline__ bool sorted_contains(const int* v, int lo, int hi, int x) {
  const int end = hi;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (v[mid] < x) lo = mid + 1; else hi = mid;
  }
  return lo < end && v[lo] == x;
}
__global__ void __launch_bounds__(FILL_WARPS * 32) clamp_fill_kernel(long long n_users, long long n_items, int k, int item_offset,
                                                                   const int* __restrict__ ex_ptr, const int* __restrict__ ex_idx,
                                                                   int* __restrict__ out_idx, float* __restrict__ out_score) {
  __shared__ int pos_ids[FILL_WARPS][WIDE_MAX_K];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * FILL_WARPS + w;
  if (row >= n_users) return;
  int* oi = out_idx + row * k;
  float* os = out_score + row * k;
  if (os[k - 1] > 0.f) return;  // k positive scores: already the clamped answer
  int m = 0;  // the positive entries: a prefix of the sorted row
  for (int t0 = 0; t0 < k; t0 += 32) {
    const unsigned b = __ballot_sync(0xffffffffu, t0 + lane < k && os[t0 + lane] > 0.f);
    m += __popc(b);
    if (b != 0xffffffffu) break;
  }
  // their ids in ascending order (bitonic sort, INT_MAX pads to a power of two)
  int* ids = pos_ids[w];
  int np2 = 1;
  while (np2 < m) np2 <<= 1;
  for (int t = lane; t < np2; t += 32) ids[t] = t < m ? oi[t] : INT_MAX;
  __syncwarp();
  for (int size = 2; size <= np2; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = lane; i < np2 / 2; i += 32) {
        const int a = 2 * i - (i & (stride - 1));
        const int x = ids[a], y = ids[a + stride];
        if ((x > y) == ((a & size) == 0)) { ids[a] = y; ids[a + stride] = x; }
      }
      __syncwarp();
    }
  }
  // the slab's ids upward, 32 at a time: keep those neither excluded nor positive
  const int ea = ex_ptr[row], eb = ex_ptr[row + 1];
  int filled = m;
  for (long long i0 = 0; i0 < n_items && filled < k; i0 += 32) {
    const int id = item_offset + (int)(i0 + lane);
    const bool keep = i0 + lane < n_items && !sorted_contains(ex_idx, ea, eb, id) && !sorted_contains(ids, 0, m, id);
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    const int pos = filled + __popc(bal & ((1u << lane) - 1u));
    if (keep && pos < k) {
      oi[pos] = id;
      os[pos] = 0.0f;
    }
    filled += __popc(bal);
  }
  for (int t = filled + lane; t < k; t += 32) {
    oi[t] = 0x7fffffff;
    os[t] = -INFINITY;
  }
}

// ------------------------------------------------------------------ operand format
// The tensor-core operands are 16-bit: bf16 (8 significant bits, fp32's exponent range) or fp16 (11 significant bits,
// normal range 6e-5 .. 65504).  Where the embeddings fit fp16's range its rounding residuals -- and with them the
// data-derived error bound E, the survivor counts of the epilogue and the rerank's candidate lists -- are ~8x smaller.
// operand_stats_kernel measures both roundings on the actual data; use_fp16() picks the format with the smaller
// relative residual (bf16 whenever a component would overflow fp16).  stats: [0] sum v^2, [1] sum (v - fp16(v))^2,
// [2] sum (v - bf16(v))^2, [3] max|v| (as int bits) for U; [4..7] the same for V.  Either choice is exact (E follows the
// chosen rounding); the float atomics only make a borderline CHOICE run-dependent, never a result.
__device__ __forceinline__ bool use_fp16(const float* stats) {
  if (stats == nullptr) return false;
  const float mx = fmaxf(__int_as_float(__float_as_int(stats[3])), __int_as_float(__float_as_int(stats[7])));
  if (!(mx < 60000.f)) return false;
  const float su = fmaxf(stats[0], 1e-30f), sv = fmaxf(stats[4], 1e-30f);
  const float e16 = sqrtf(stats[1] / su) + sqrtf(stats[5] / sv);
  const float ebf = sqrtf(stats[2] / su) + sqrtf(stats[6] / sv);
  return e16 < ebf;
}

__global__ void __launch_bounds__(256) operand_stats_kernel(const float* __restrict__ src, long long n, int ld, float* __restrict__ stats) {
  float ss = 0.f, s16 = 0.f, sbf = 0.f, mx = 0.f;
  const int lane = threadIdx.x & 31;
  const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < n; row += warps) {  // one warp per row
    const float4* p4 = reinterpret_cast<const float4*>(src + row * ld);
    for (int c4 = lane; c4 < (ld >> 2); c4 += 32) {  // pad columns [r, ld) are zero: they add nothing
      const float4 q = __ldg(p4 + c4);
      const float vv[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float v = vv[j];
        const float d16 = v - __half2float(__float2half_rn(v));
        const float dbf = v - __bfloat162float(__float2bfloat16_rn(v));
        ss = fmaf(v, v, ss);
        s16 = fmaf(d16, d16, s16);
        sbf = fmaf(dbf, dbf, sbf);
        mx = fmaxf(mx, fabsf(v));
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ss += __shfl_xor_sync(0xffffffffu, ss, o);
    s16 += __shfl_xor_sync(0xffffffffu, s16, o);
    sbf += __shfl_xor_sync(0xffffffffu, sbf, o);
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(stats + 0, ss);
    atomicAdd(stats + 1, s16);
    atomicAdd(stats + 2, sbf);
    atomicMax(reinterpret_cast<int*>(stats) + 3, __float_as_int(mx));  // non-negative floats order like ints (inf/NaN sort high)
  }
}

// ------------------------------------------------------------------ operand packing
// one warp per row: fp32 [n, ld] -> bf16 [n_pad, k_pad] (zero padded); per row the l2 norms of the row, of its bf16
// image and of the rounding residual; optional global maxima of the row norm and the residual norm
__global__ void pack_bf16_kernel(const float* __restrict__ src, long long n, int r, int ld, __nv_bfloat16* __restrict__ dst,
                                 long long n_pad, int k_pad, float* __restrict__ norms, float* __restrict__ norms_bf,
                                 float* __restrict__ norms_res, int* __restrict__ max_bits, int nan_pad,
                                 const float* __restrict__ fmt_stats, int force_fmt) {
  const long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n_pad) return;
  const bool f16 = force_fmt >= 0 ? force_fmt == 1 : use_fp16(fmt_stats);
  unsigned short* dst16 = reinterpret_cast<unsigned short*>(dst);
  float ss = 0.f, sb = 0.f, sd = 0.f;
  for (int c = lane; c < k_pad; c += 32) {
    float v = 0.f;
    if (row < n && c < r) v = src[row * ld + c];
    unsigned short bits;
    float vb;
    if (f16) {
      const __half h = __float2half_rn(v);
      bits = __half_as_ushort(h);
      vb = __half2float(h);
    } else {
      const __nv_bfloat16 h = __float2bfloat16_rn(v);
      bits = __bfloat16_as_ushort(h);
      vb = __bfloat162float(h);
    }
    const float d = v - vb;  // exact
    ss = fmaf(v, v, ss);
    sb = fmaf(vb, vb, sb);
    sd = fmaf(d, d, sd);
    // padded ITEM rows are NaN: their scores are NaN in every accumulator row, which fmaxf ignores and every
    // >= test rejects -- the epilogue needs no per-column bounds checks
    dst16[row * k_pad + c] = (nan_pad && row >= n) ? (unsigned short)(f16 ? 0x7E00 : 0x7FC0) : bits;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ss += __shfl_xor_sync(0xffffffffu, ss, o);
    sb += __shfl_xor_sync(0xffffffffu, sb, o);
    sd += __shfl_xor_sync(0xffffffffu, sd, o);
  }
  if (lane == 0) {
    const float nrm = sqrtf(ss) * NORM_SLACK, nb = sqrtf(sb) * NORM_SLACK, nd = sqrtf(sd) * NORM_SLACK;
    if (norms) norms[row] = nrm;
    if (norms_bf) norms_bf[row] = nb;
    if (norms_res) norms_res[row] = nd;
    if (max_bits) {  // non-negative floats order like ints
      atomicMax(max_bits, __float_as_int(nrm));
      atomicMax(max_bits + 1, __float_as_int(nd));
    }
  }
}

// E[row] = |du| max|v| + |u~| max|dv| + accumulation slack (see ACC_UNIT)
__global__ void row_error_kernel(const float* __restrict__ unorm_bf, const float* __restrict__ unorm_res, const int* __restrict__ vmax_bits,
                                 int k_pad, float* __restrict__ erow, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float vmax = __int_as_float(vmax_bits[0]), dvmax = __int_as_float(vmax_bits[1]);
  const float e = unorm_res[i] * vmax + unorm_bf[i] * dvmax + ACC_UNIT * (float)k_pad * unorm_bf[i] * vmax;
  erow[i] = e * NORM_SLACK + 1e-30f;
}

// ------------------------------------------------------------------ host side
// tensor maps: make_tmap_k64 (tc_common.cuh) -- K-major 16-bit [rows, k_pad], 128-byte swizzle, box = 64 x box_rows
static int make_tmap(CUtensorMap* map, void* base, long long rows, int k_pad, int box_rows) {
  static_assert(BK == 64, "make_tmap_k64 boxes are 64 elements wide");
  return make_tmap_k64(map, base, rows, k_pad, box_rows);
}

struct TopkLayout {
  long long nu_pad, ni_pad, batch_rows;
  int k_pad, kb;
  bool wide;                  // k > NARROW_MAX_K: the CAP_W / UB_BATCH_W configuration
  int cap, ub_batch;
  size_t off_ub, off_vb, off_unorm, off_ures, off_erow, off_vnorm, off_vmax, off_cand, off_cnt, off_thr, off_ovfc, off_ovfr, off_scratch, total;
  int scratch_rows;
};

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

static TopkLayout topk_layout(long long n_users, long long n_items, int r, int k) {
  TopkLayout L{};
  L.wide = k > NARROW_MAX_K;
  L.cap = L.wide ? CAP_W : CAP;
  L.ub_batch = L.wide ? UB_BATCH_W : UB_BATCH;
  L.nu_pad = cdiv(n_users, BM) * BM;
  L.ni_pad = cdiv(n_items, BN) * BN;
  L.batch_rows = std::min<long long>(L.nu_pad, (long long)L.ub_batch * BM);
  L.k_pad = (int)(cdiv(r, BK) * BK);
  L.kb = L.k_pad / BK;
  size_t o = 0;
  L.off_ub = o; o = align_up(o + (size_t)L.nu_pad * L.k_pad * 2, 1024);
  L.off_vb = o; o = align_up(o + (size_t)L.ni_pad * L.k_pad * 2, 1024);
  L.off_unorm = o; o = align_up(o + (size_t)L.nu_pad * 4, 256);
  L.off_ures = o; o = align_up(o + (size_t)L.nu_pad * 4, 256);
  L.off_erow = o; o = align_up(o + (size_t)L.nu_pad * 4, 256);
  L.off_vnorm = o; o = align_up(o + (size_t)L.ni_pad * 4, 256);
  L.off_vmax = o; o += 256;
  L.off_cand = o; o = align_up(o + (size_t)L.batch_rows * L.cap * 8, 256);
  L.off_cnt = o; o = align_up(o + (size_t)L.batch_rows * 4, 256);
  L.off_thr = o; o = align_up(o + (size_t)L.batch_rows * 4, 256);
  L.off_ovfc = o; o += 256;
  L.off_ovfr = o; o = align_up(o + (size_t)L.nu_pad * 4, 256);
  L.scratch_rows = (int)std::min<long long>(32, n_users);
  L.off_scratch = o; o = align_up(o + (size_t)L.scratch_rows * n_items * 4, 256);
  L.total = o + 1024;
  return L;
}

}  // namespace tmf

using namespace tmf;

extern "C" size_t tmf_score_topk_ws_bytes(int64_t n_users, int64_t n_items, int32_t n_comp, int32_t k) {
  return topk_layout(n_users, n_items, n_comp, k).total;
}

static int score_topk_impl(const float* U, int64_t n_users, const float* V, int64_t n_items, int32_t n_comp, int32_t ld,
                           int32_t k, int32_t clamp, int32_t item_offset, int32_t* out_idx, float* out_score, void* ws,
                           size_t ws_bytes, tmf_stream_t stream, float* dump, const float* row_bound = nullptr, int force_fmt = -1,
                           const int32_t* ex_ptr = nullptr, const int32_t* ex_idx = nullptr) {
  TMF_REQUIRE(n_users >= 0 && n_items > 0 && n_comp > 0 && n_comp <= ld, "tmf_score_topk: bad shape");
  TMF_REQUIRE(n_comp <= MAX_KB * BK, "tmf_score_topk: n_components up to %d supported", MAX_KB * BK);
  TMF_REQUIRE(k >= 1 && k <= WIDE_MAX_K && k <= n_items, "tmf_score_topk: need 1 <= k <= min(%d, n_items) (k=%d)", WIDE_MAX_K, k);
  TMF_REQUIRE(n_items < (1ll << 31) - BN && n_users < (1ll << 31) - BM, "tmf_score_topk: sizes must fit int32");
  if (n_users == 0) return TMF_OK;
  const TopkLayout L = topk_layout(n_users, n_items, n_comp, k);
  TMF_REQUIRE(ws_bytes >= L.total, "tmf_score_topk: workspace too small");
  unsigned char* w = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(ws) + 1023) & ~(uintptr_t)1023);
  __nv_bfloat16* Ub = reinterpret_cast<__nv_bfloat16*>(w + L.off_ub);
  __nv_bfloat16* Vb = reinterpret_cast<__nv_bfloat16*>(w + L.off_vb);
  float* unorm = reinterpret_cast<float*>(w + L.off_unorm);  // |bf16(u)|
  float* ures = reinterpret_cast<float*>(w + L.off_ures);    // |u - bf16(u)|
  float* erow = reinterpret_cast<float*>(w + L.off_erow);
  float* vnorm = reinterpret_cast<float*>(w + L.off_vnorm);
  int* vmax_bits = reinterpret_cast<int*>(w + L.off_vmax);
  float2* cand = reinterpret_cast<float2*>(w + L.off_cand);
  int* cnt = reinterpret_cast<int*>(w + L.off_cnt);
  float* thr = reinterpret_cast<float*>(w + L.off_thr);
  int* ovfc = reinterpret_cast<int*>(w + L.off_ovfc);
  int* ovfr = reinterpret_cast<int*>(w + L.off_ovfr);
  float* scratch = reinterpret_cast<float*>(w + L.off_scratch);
  cudaStream_t st = as_stream(stream);

  TMF_CUDA(cudaMemsetAsync(vmax_bits, 0, 8, st));
  TMF_CUDA(cudaMemsetAsync(ovfc, 0, 4, st));
#ifdef TMF_DEVTOOLS
  if (force_fmt < 0) {
    const char* e = getenv("TMF_TOPK_FMT");  // A/B aid: "bf16" / "f16"
    if (e) force_fmt = (e[0] == 'f' || e[0] == 'h') ? 1 : 0;
  }
#endif
  float* fmt_stats = reinterpret_cast<float*>(w + L.off_vmax + 16);  // 8 floats inside the 256-byte scalar block
  if (force_fmt < 0) {
    TMF_CUDA(cudaMemsetAsync(fmt_stats, 0, 32, st));
    const int sgrid = 8 * kNumSMs;
    operand_stats_kernel<<<sgrid, 256, 0, st>>>(U, n_users, ld, fmt_stats);
    operand_stats_kernel<<<sgrid, 256, 0, st>>>(V, n_items, ld, fmt_stats + 4);
  }
  pack_bf16_kernel<<<(unsigned)cdiv(L.nu_pad * 32, 256), 256, 0, st>>>(U, n_users, n_comp, ld, Ub, L.nu_pad, L.k_pad, nullptr, unorm, ures,
                                                                       nullptr, 0, fmt_stats, force_fmt);
  pack_bf16_kernel<<<(unsigned)cdiv(L.ni_pad * 32, 256), 256, 0, st>>>(V, n_items, n_comp, ld, Vb, L.ni_pad, L.k_pad, vnorm, nullptr, nullptr,
                                                                       vmax_bits, 1, fmt_stats, force_fmt);
  row_error_kernel<<<(unsigned)cdiv(L.nu_pad, 256), 256, 0, st>>>(unorm, ures, vmax_bits, L.k_pad, erow, L.nu_pad);
  TMF_LAUNCH_CHECK();

  CUtensorMap tmapU, tmapV;
  int rc = make_tmap(&tmapU, Ub, L.nu_pad, L.k_pad, BM);
  if (rc) return rc;
  rc = make_tmap(&tmapV, Vb, L.ni_pad, L.k_pad, BN);
  if (rc) return rc;

  // masked: raw ranking of the unseen items; clamp mode is finished by clamp_fill_kernel
  const bool mask = ex_ptr != nullptr;
  TopkParams p{};
  p.n_users = n_users; p.n_items = n_items;
  p.n_tiles = (int)(L.ni_pad / BN); p.kb = L.kb;
  p.k = k; p.clamp = clamp && !mask ? 1 : 0; p.item_offset = item_offset;
  p.ex_ptr = ex_ptr; p.ex_idx = ex_idx;
  p.erow = erow;
  p.cand = cand; p.cnt = cnt; p.thr_out = thr; p.ovf_count = ovfc; p.ovf_rows = ovfr;
  p.dump = dump; p.dump_ld = n_items;
  p.row_bound = row_bound;
  p.fmt_stats = fmt_stats; p.force_fmt = force_fmt;
  p.dbg = 0;
  p.prof = nullptr;
#ifdef TMF_DEVTOOLS
  { const char* e = getenv("TMF_TOPK_DEBUG"); p.dbg = e ? atoi(e) : 0; }
  if (getenv("TMF_TOPK_PROF")) {
    p.prof = reinterpret_cast<unsigned long long*>(w + L.off_vmax + 64);
    TMF_CUDA(cudaMemsetAsync(p.prof, 0, 192, st));
  }
#endif

  RerankParams q{};
  q.n_users = n_users; q.n_items = n_items; q.k = k; q.clamp = p.clamp; q.item_offset = item_offset; q.r = n_comp; q.ld = ld;
  q.U = U; q.V = V; q.erow = erow; q.prof = p.prof; q.cand = cand; q.cnt = cnt; q.thr = thr; q.ovf_count = ovfc; q.ovf_rows = ovfr;
  q.out_idx = out_idx; q.out_score = out_score;
  q.ex_ptr = ex_ptr; q.ex_idx = ex_idx;

  const size_t smem = 1024 + topk_smem(L.kb).total + (mask ? BM * EXCUR_BYTES : 0);  // + room to align the base
  auto main_kernel = L.wide ? (mask ? score_topk_kernel<false, false, true, true> : score_topk_kernel<false, false, true>)
                   : dump != nullptr ? score_topk_kernel<true, false, false>
                   : mask ? score_topk_kernel<false, false, false, true> : score_topk_kernel<false, false, false>;
#ifdef TMF_DEVTOOLS
  if (p.prof && dump == nullptr && !mask) main_kernel = L.wide ? score_topk_kernel<false, true, true> : score_topk_kernel<false, true, false>;
#endif
  TMF_CUDA(cudaFuncSetAttribute(main_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int rr_warps = L.wide ? RR_WARPS_W : RR_WARPS;
  const size_t rr_smem = (size_t)rr_warps * (L.wide ? rerank_warp_smem<true>(ld) : rerank_warp_smem<false>(ld));
  auto rr_kernel = L.wide ? rerank_kernel<true> : rerank_kernel<false>;
  TMF_CUDA(cudaFuncSetAttribute(rr_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rr_smem));

  // users go through in batches of ub_batch blocks so the candidate workspace stays bounded; V stays packed
  const int total_ublocks = (int)(L.nu_pad / BM);
  for (int ub0 = 0; ub0 < total_ublocks; ub0 += L.ub_batch) {
    p.ub0 = ub0;
    p.n_ublocks = std::min(L.ub_batch, total_ublocks - ub0);
    const int grid = std::min(2 * kNumSMs, p.n_ublocks);  // two CTAs per SM (smem- and TMEM-limited)
    main_kernel<<<grid, TOPK_THREADS, smem, st>>>(tmapU, tmapV, p);
    TMF_LAUNCH_CHECK();
    if (dump != nullptr) continue;
    q.row0 = (long long)ub0 * BM;
    q.n_rows = std::min<long long>((long long)p.n_ublocks * BM, n_users - q.row0);
    rr_kernel<<<(unsigned)cdiv(q.n_rows, rr_warps), rr_warps * 32, rr_smem, st>>>(q);
    TMF_LAUNCH_CHECK();
  }
  if (dump != nullptr) return TMF_OK;
  exact_rows_kernel<<<L.scratch_rows, 256, 0, st>>>(q, ovfc, ovfr, scratch);
  TMF_LAUNCH_CHECK();
  if (mask && clamp) {
    clamp_fill_kernel<<<(unsigned)cdiv(n_users, FILL_WARPS), FILL_WARPS * 32, 0, st>>>(n_users, n_items, k, item_offset, ex_ptr, ex_idx,
                                                                                     out_idx, out_score);
    TMF_LAUNCH_CHECK();
  }
#ifdef TMF_DEVTOOLS
  if (p.prof) {  // profiling aid only: synchronises
    unsigned long long h[24]; int novf = 0;
    TMF_CUDA(cudaStreamSynchronize(st));
    TMF_CUDA(cudaMemcpy(h, p.prof, 192, cudaMemcpyDeviceToHost));
    TMF_CUDA(cudaMemcpy(&novf, ovfc, 4, cudaMemcpyDeviceToHost));
    fprintf(stderr, "[tmf prof] producer wait empty %.3g, a_empty %.3g | mma wait tempty %.3g, full %.3g | epilogue (per warp-sweep, n=%llu) "
                    "wait tfull %.3g, work %.3g, init %.3g cycles | overflow rows %d (main %llu, rerank %llu) | tile-end drains: %llu, %.0f cycles each\n",
            (double)h[0], (double)h[1], (double)h[2], (double)h[3], h[7], (double)h[4] / h[7], (double)h[5] / h[7], (double)h[6] / h[7], novf, h[8], h[9], h[11], h[11] ? (double)h[10] / h[11] : 0.0);
    fprintf(stderr, "[tmf prof] rebuilds: first %llu x %.0f cycles, saturated %llu x %.0f, selected %llu x %.0f | pre-rebuild drains %llu x %.0f | appended entries %.4g (%.1f per row-sweep)\n",
            h[12], h[12] ? (double)h[13] / h[12] : 0.0, h[14], h[14] ? (double)h[15] / h[14] : 0.0, h[16], h[16] ? (double)h[17] / h[16] : 0.0,
            h[18], h[18] ? (double)h[19] / h[18] : 0.0, (double)h[20], h[7] ? (double)h[20] / (32.0 * h[7]) : 0.0);
  }
#endif
  return TMF_OK;
}

extern "C" int tmf_score_topk(const float* U, int64_t n_users, const float* V, int64_t n_items, int32_t n_comp, int32_t ld,
                              int32_t k, int32_t clamp, int32_t item_offset, int32_t* out_idx, float* out_score, void* ws,
                              size_t ws_bytes, tmf_stream_t stream) {
  return score_topk_impl(U, n_users, V, n_items, n_comp, ld, k, clamp, item_offset, out_idx, out_score, ws, ws_bytes, stream, nullptr);
}

extern "C" int tmf_score_topk_bounded(const float* U, int64_t n_users, const float* V, int64_t n_items, int32_t n_comp, int32_t ld,
                                      int32_t k, int32_t clamp, int32_t item_offset, const float* row_bound, int32_t* out_idx,
                                      float* out_score, void* ws, size_t ws_bytes, tmf_stream_t stream) {
  return score_topk_impl(U, n_users, V, n_items, n_comp, ld, k, clamp, item_offset, out_idx, out_score, ws, ws_bytes, stream, nullptr,
                         row_bound);
}

extern "C" int tmf_score_topk_masked(const float* U, int64_t n_users, const float* V, int64_t n_items, int32_t n_comp, int32_t ld,
                                     int32_t k, int32_t clamp, int32_t item_offset, const int32_t* ex_ptr, const int32_t* ex_idx,
                                     int32_t* out_idx, float* out_score, void* ws, size_t ws_bytes, tmf_stream_t stream) {
  TMF_REQUIRE(ex_ptr != nullptr && out_idx != nullptr && out_score != nullptr, "tmf_score_topk_masked: null argument");
  return score_topk_impl(U, n_users, V, n_items, n_comp, ld, k, clamp, item_offset, out_idx, out_score, ws, ws_bytes, stream, nullptr,
                         nullptr, -1, ex_ptr, ex_idx);
}

extern "C" int tmf_score_dense_tc(const float* U, int64_t n_users, const float* V, int64_t n_items, int32_t n_comp, int32_t ld,
                                  int32_t operand_format, float* P, void* ws, size_t ws_bytes, tmf_stream_t stream) {
  TMF_REQUIRE(P != nullptr, "tmf_score_dense_tc: null output");
  TMF_REQUIRE(operand_format >= -1 && operand_format <= 1, "tmf_score_dense_tc: operand_format is -1 (auto), 0 (bf16) or 1 (fp16)");
  return score_topk_impl(U, n_users, V, n_items, n_comp, ld, 1, 0, 0, nullptr, nullptr, ws, ws_bytes, stream, P, nullptr, operand_format);
}
