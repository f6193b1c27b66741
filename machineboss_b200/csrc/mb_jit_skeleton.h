// mb_jit_skeleton.h -- CUDA source of the machine-specialised strip kernels, compiled at run time
// with NVRTC for sm_100a after the generated prelude (defines + the per-machine cell functions,
// see mb_jit.cu) has been placed in front of it.
//
// Mapping (one warp per sequence pair; pairs are pulled from a work counter, longest first):
//   * the DP matrix is cut into vertical strips of 32*MB_C input positions; lane j owns MB_C
//     adjacent columns of the strip and keeps their previous-row cell values (MB_S states each)
//     in registers;
//   * rows are swept in a skew: at step t lane j computes output row t-j, so the cells the warp
//     computes in one step lie on an anti-diagonal (of MB_C-wide blocks); the left neighbour's
//     values arrive with one shuffle per state per step, the diagonal ones are last step's;
//   * the last column of a strip is handed to the next strip through an L2-resident buffer,
//     written by lane 31 and staged back 32 rows at a time through shared memory;
//   * emission log-weights (token-indexed) sit in shared memory, silent log-weights arrive as a
//     __grid_constant__ kernel parameter (constant bank), the transition structure itself is
//     straight-line code in the generated cell function.
// Backward runs the same sweep in reversed coordinates (i' = Li-i, o' = Lo-o) with the machine's
// outgoing transitions.
#ifndef MB_JIT_SKELETON_H
#define MB_JIT_SKELETON_H

static const char* const kJitSkeleton = R"MBSRC(
#define MB_W (32 * MB_C)
#define MB_FULL 0xffffffffu

struct MBArgs {
  const uint8_t* x; const int64_t* xOff;
  const uint8_t* y; const int64_t* yOff;
  const int64_t* order; int64_t nWork; unsigned long long* counter;
  double* bnd; int64_t bndStride;
  double* result;
  const double* emit;
  uint8_t* tb; const int64_t* tbOff;
  double* F; const int64_t* fOff;        // full Forward matrices [outPos][inPos][state] (modes 2, 3)
  const double* ll;                      // Forward log-likelihood per pair (mode 3)
  double* counts;                        // [nTrans] posterior counts (mode 3)
  const int32_t* idTabB;                 // transition id per backward-program table entry (mode 3)
  int32_t* flag;                         // per pair: 1 = the scaled linear sweep saw a dangerous dynamic range
  unsigned* F32; const int64_t* f32Off;  // linear E-step: high words of the Forward values, [outPos][inPos][state]
  int32_t* ef; const int64_t* efOff;     // linear E-step: frame exponent per (strip, block of MB_RESCALE steps)
  // SPLIT mode (few or long pairs: fewer pairs than resident warps).  A work item is ONE STRIP of a pair,
  // items[w] = pair << 16 | strip, the strips of a pair consecutive in w; the warps that claim them run as a
  // pipeline down the strips: strip s writes its last column to the item's own boundary buffer and publishes in
  // prog[w] how many rows of it are complete, strip s + 1 (item w + 1, claimed later, hence never waited for by
  // its predecessor) waits until the rows it is about to stage are there.  items == 0: a warp takes whole pairs.
  const int64_t* items; const int64_t* itemBnd; int* prog;
  const int64_t* rowOf;                  // per pair: its row of counts, [row][MB_NTRANS] (per-pair count kernels, MB_PAIR_ROWS)
};

// Split mode is compiled into a module of its own (MB_SPLIT 1, built the first time a call needs it): in the ordinary
// modules `split` is a compile-time false and none of this costs registers or instructions.
#ifndef MB_SPLIT
#define MB_SPLIT 0
#endif
// rows [0, need) of the previous strip's boundary are complete and visible (split mode)
__device__ __forceinline__ void mb_wait_rows (const int* prog, const int need) {
  while (*(volatile const int*) prog < need) { }
  __threadfence();
}
// lane 31 has written rows [0, rows) of this strip's boundary: make them visible, then say so
__device__ __forceinline__ void mb_publish_rows (int* prog, const int rows) {
  __threadfence();
  *(volatile int*) prog = rows;
}

__device__ __forceinline__ double mb_neg_inf() { return __longlong_as_double (0xfff0000000000000LL); }

// log(exp(a)+exp(b)) = max + softplus(|a-b|).
// The max, the difference and the final add are FP64; softplus(x) = ln(1+e^-x) is evaluated in
// FP32 with the two MUFU operations nothing can remove (ex2, lg2).  The FP64<->FP32 conversions are
// done by exponent re-bias in integer instructions instead of F2F, because F2F shares the XU pipe
// with MUFU (16/clk/SM) and the kernel is XU-bound: this halves the XU work per log-sum-exp.
//   down: |a-b| clamped to [2^-127, 128] (covers 0, inf and the NaN of -inf - -inf), truncated
//         to 24 bits; softplus(128) == 0 in FP32, so no separate cut-off is needed;
//   up:   exact (every FP32 value in [0, ln 2] is a normal double); an exact 0 becomes 2^-127,
//         which cannot change a sum whose other term is a log-weight.
// Unlike the reference's table (src/logsumexp.h:52) this does not truncate at x >= 10, so it is
// the exact function up to FP32 rounding (<= 1.2e-7 absolute); the table differs from it by up to
// 4.5e-5 per operation.
__device__ __forceinline__ double mb_lse (double a, double b) {
  const double t = a - b;
  const int hi = __double2hiint (t);
  const double mx = (hi < 0) ? b : a;
  const int ahi = min (max (hi & 0x7fffffff, 0x38000000), 0x40600000);
  const float x = __uint_as_float (__funnelshift_l ((unsigned) __double2loint (t), (unsigned) (ahi - 0x38000000), 3));
  float e;
  asm ("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-1.4426950408889634f * x));
  const unsigned gb = __float_as_uint (__log2f (1.0f + e) * 0.6931471805599453f);
  return mx + __hiloint2double ((int) ((gb >> 3) + 0x38000000u), (int) (gb << 29));
}

// exp(z) for a posterior log-odds z <= ~0, FP32 on the MUFU pipe
__device__ __forceinline__ float mb_post (double z) {
  return exp2f (1.4426950408889634f * __double2float_rn (z));
}

__device__ __forceinline__ float mb_warp_sum (float v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync (MB_FULL, v, d);
  return v;
}

__device__ __forceinline__ void mb_cp_async16 (void* smem, const void* gmem) {
  asm volatile ("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"((unsigned) __cvta_generic_to_shared (smem)), "l"(gmem));
}
__device__ __forceinline__ void mb_cp_async_commit() { asm volatile ("cp.async.commit_group;"); }
__device__ __forceinline__ void mb_cp_async_wait_all() { asm volatile ("cp.async.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ void mb_prefetch_l2 (const void* p) { asm volatile ("prefetch.global.L2 [%0];" :: "l"(p)); }

__device__ __forceinline__ double mb_warp_sum_d (double v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync (MB_FULL, v, d);
  return v;
}

// lane 0 replaces v by the double at a shared-memory address (the staged boundary row); the other lanes keep theirs:
// one predicated load instead of an unconditional load and two selects
__device__ __forceinline__ void mb_lds_lane0 (double& v, const int lane, const unsigned addr) {
  asm volatile ("{ .reg .pred p; setp.eq.s32 p, %1, 0; @p ld.shared.f64 %0, [%2]; }" : "+d"(v) : "r"(lane), "r"(addr));
}

// log of the scale the result state carries in the normalised linear kernels (0 elsewhere)
template<int DIR> __device__ __forceinline__ double mb_res_log (const MBSil&) { return 0.0; }
#ifdef MB_ROWTAB
template<int DIR> __device__ __forceinline__ double mb_res_log (const MBSilN& P) { return DIR ? P.resLogB : P.resLogF; }
#endif

template<bool B> struct MBBool { static constexpr bool value = B; };

// where a count kernel adds pair k's counts: the summed vector, or (ROWS) the pair's row.  The warps that sweep strips of
// one pair add into the same row, as they add into the same summed vector.
template<bool ROWS> __device__ __forceinline__ double* mb_count_row (const MBArgs& A, const int64_t k) {
#ifdef MB_PAIR_ROWS
  if (ROWS) return A.counts + A.rowOf[k] * (int64_t) MB_NTRANS;
#endif
  return A.counts;
}

template<int DIR> struct MBDir { };
template<> struct MBDir<0> { static const int NE = MB_NEMIT_F; static const int RES = MB_S - 1; };
template<> struct MBDir<1> { static const int NE = MB_NEMIT_B; static const int RES = 0; };

// states whose values are read by later cells (sources of non-silent transition groups); the
// others are temporaries of the cell function and need no shuffle, boundary slot or rescaling
template<int DIR> __device__ __forceinline__ constexpr bool mb_live (int s) { return ((DIR ? MB_LIVE_B : MB_LIVE_F) >> s) & 1ull; }

#define MB_FBLOCK (32 * MB_C * MB_SQ * 4)       // 32-bit words per warp-step block of stored Forward values
#define MB_ROW (MB_S + 1)      // doubles per strip-boundary row: the states + the frame exponent (linear sweeps)

// MODE 0: log-sum-exp score (Forward for DIR 0, Backward for DIR 1); MODE 1: Viterbi + back-pointers;
// MODE 4: Viterbi score only (boss -V without -A: no pointer is formed, packed or stored);
// MODE 2: Forward that also stores every cell (the E-step's ForwardMatrix, counts.cpp:58);
// MODE 3: Backward fused with the posterior-count accumulation of BackwardMatrix::getCounts
//         (backward.cpp:62-87): each transition group's term w + B(dest) is formed once and used
//         both for the Backward log-sum-exp and for exp(F(src) - ll + term).
// ROWS (mode 3): the counts of pair k go to its own row, A.counts + A.rowOf[k] * MB_NTRANS, instead of one summed vector.
template<int MODE, int DIR, bool ROWS = false>
__device__ __forceinline__ void mb_run (const MBSil& P, const MBArgs& A) {
  extern __shared__ double mb_smem[];
  double* E = mb_smem;
  const int NE = MBDir<DIR>::NE;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int q = threadIdx.x; q < NE; q += blockDim.x) E[q] = A.emit[q];
  __syncthreads();
#ifdef MB_ROWTAB
  const unsigned eBase = (unsigned) __cvta_generic_to_shared (E);      // the emission weights in row layout (see the generated prelude)
#endif
  // shared memory: emission table | per warp: 128-byte ring of output-row tokens, published a block
  // ahead so that each lane can fetch its next step's token during the current step | per warp: 32 staged boundary rows | per warp: thread-private count
  // accumulators of the emitting transition groups, acc[ctx * 32 + lane] (count kernels only)
  const int nWarps = blockDim.x >> 5;
  uint8_t* ring = (uint8_t*) (mb_smem + ((NE + 1) & ~1)) + warp * 128;
  double* sIn = mb_smem + ((NE + 1) & ~1) + nWarps * 16 + warp * (32 * MB_ROW);
  float* acc = (float*) (mb_smem + ((NE + 1) & ~1) + nWarps * (16 + 32 * MB_ROW)) + warp * (32 * MB_NCTX) + lane;
  const int64_t wslot = (int64_t) blockIdx.x * nWarps + warp;
  double* bndA = A.bnd + wslot * A.bndStride;
  double* bndB = bndA + (A.bndStride >> 1);
  const double NI = mb_neg_inf();
  const unsigned sInAddr = (unsigned) __cvta_generic_to_shared (sIn);

  for (;;) {
    unsigned long long w = 0;
    if (lane == 0) w = atomicAdd (A.counter, 1ULL);
    w = __shfl_sync (MB_FULL, w, 0);
    if ((int64_t) w >= A.nWork) break;
    const bool split = MB_SPLIT && A.items != 0;
    const int64_t item = split ? A.items[w] : 0;
    const int64_t k = split ? (item >> 16) : A.order[w];
    const int64_t x0 = A.xOff[k], y0 = A.yOff[k];
    const int Li = (int) (A.xOff[k + 1] - x0), Lo = (int) (A.yOff[k + 1] - y0);
    const uint8_t* x = A.x + x0;
    const uint8_t* y = A.y + y0;
    const int nStrips = (Li + MB_W) / MB_W;
    // Back-pointers in SWEEP ORDER: one block per (strip, step) holding the 32 lanes' groups of MB_TBLANE bytes (the lane's
    // MB_C cells of that step; a fitted strip width whose MB_C * MB_TBBYTES is not a power of two pads the group to 16 bytes),
    // so that a step's store is one contiguous run of 32 * MB_TBLANE bytes.  (Row-major rows scattered the skewed lanes over
    // 32 sectors per store.)  Cell (i, o): strip i / MB_W, lane (i % MB_W) / MB_C, step o + lane.
#ifdef MB_TBPAD
#define MB_TBLANE 16
#else
#define MB_TBLANE (MB_C * MB_TBBYTES)
#endif
    uint8_t* tb = MODE == 1 ? A.tb + A.tbOff[k] : (uint8_t*) 0;
    double* Fm = (MODE == 2 || MODE == 3) ? A.F + A.fOff[k] : (double*) 0;
    const double ll = MODE == 3 ? A.ll[k] : 0.0;
    if (MODE == 3 && !(ll > NI)) continue;     // impossible pair: no posterior (the reference would produce NaN)

    const int stripFirst = split ? (int) (item & 0xffff) : 0, stripEnd = split ? stripFirst + 1 : nStrips;
    for (int strip = stripFirst; strip < stripEnd; ++strip) {
      const int col0 = strip * MB_W + lane * MB_C;
      int ta[MB_C];
#ifdef MB_ROWTAB
      unsigned ea[MB_C];      // shared-memory address of each column's input-token row
#endif
#pragma unroll
      for (int c = 0; c < MB_C; ++c) {
        const int i = col0 + c;
        int tok = 1;
        if (i >= 1 && i <= Li) tok = DIR ? x[Li - i] : x[i - 1];
        ta[c] = tok - 1;
#ifdef MB_ROWTAB
        ea[c] = eBase + (unsigned) (tok - 1) * (unsigned) (MB_WA_F * 8);
#endif
      }
      double U[MB_C][MB_S], Lk[MB_S];
#pragma unroll
      for (int s = 0; s < MB_S; ++s) {
        Lk[s] = NI;
#pragma unroll
        for (int c = 0; c < MB_C; ++c) U[c][s] = NI;
      }
      float cs[MB_NSIL_B > 0 ? MB_NSIL_B : 1];
      if (MODE == 3) {
#pragma unroll
        for (int q = 0; q < (MB_NSIL_B > 0 ? MB_NSIL_B : 1); ++q) cs[q] = 0.f;
        for (int q = 0; q < MB_NCTX; ++q) acc[q * 32] = 0.f;
      }
      const bool hasIn = strip > 0, hasOut = strip + 1 < nStrips;
      const double* bin = split ? (hasIn ? A.bnd + A.itemBnd[w - 1] : bndA) : ((strip & 1) ? bndB : bndA);
      double* bout = split ? A.bnd + A.itemBnd[w] : ((strip & 1) ? bndA : bndB);
      const bool waits = split && hasIn, publishes = split && hasOut && lane == 31;
      if (!hasIn) {      // the column left of the matrix: nothing comes from there
        __syncwarp();
        for (int q = lane; q < 32 * MB_ROW; q += 32) sIn[q] = NI;
        __syncwarp();
      }
      if (waits) mb_wait_rows (A.prog + (w - 1), min (32, Lo + 1));
      double stageNext[MB_S];
#pragma unroll
      for (int s = 0; s < MB_S; ++s)
        stageNext[s] = (hasIn && mb_live<DIR> (s) && lane <= Lo) ? __ldcg (bin + (int64_t) lane * MB_ROW + s) : NI;
      // row tokens (0-based): rows 0..31 are published now, rows 32..63 at step 0, and so on one block ahead
      // (the raw 1-based byte is kept until it is published a block later: subtracting 1 at once would make
      // the warp wait for the global load)
      auto rowTok = [&] (const int row) { return (row >= 1 && row <= Lo) ? (int) (DIR ? y[Lo - row] : y[row - 1]) : 1; };
      __syncwarp();
      ring[lane] = (uint8_t) (rowTok (lane) - 1);
      int ynext = rowTok (32 + lane);
      __syncwarp();
      int tokNext = ring[(0 - lane) & 127];          // token of this lane's row at step 0 (only lane 0's is real)
      const int nSteps = Lo + 32;
      // where this lane's row r = t - lane goes: pointers advanced by one row per step instead of recomputed
      uint8_t* tbRow = MODE == 1 ? tb + ((int64_t) strip * (Lo + 32) * 32 + lane) * MB_TBLANE : (uint8_t*) 0;      // this lane's group at step 0
      const int64_t tbStep = 32 * MB_TBLANE;
      double* boutRow = bout + (int64_t) (0 - lane) * MB_ROW;
      // one step of the skewed sweep; STEADY = every lane is inside the matrix (31 <= t < Lo), so the
      // ramp predicates (row in range, origin cell, result cell) fold away
      // every 32 steps (kept out of the step body so that the steady loop carries no block tests)
      auto blockStart = [&] (const int t) {
        if (publishes && t >= 32) mb_publish_rows (A.prog + w, t - 31);      // (steps < t are done: lane 31 has written rows <= t - 32)
        if (waits) mb_wait_rows (A.prog + (w - 1), min (t + 64, Lo + 1));
        if (hasIn) {                        // stage 32 rows of the previous strip's last column: lane q takes row t+q;
          __syncwarp();                     // the values were fetched a block ago, the next block's are fetched now
#pragma unroll
          for (int s = 0; s < MB_S; ++s) if (mb_live<DIR> (s)) sIn[lane * MB_ROW + s] = stageNext[s];
#pragma unroll
          for (int s = 0; s < MB_S; ++s)
            if (mb_live<DIR> (s)) stageNext[s] = (t + 32 + lane <= Lo) ? __ldcg (bin + (int64_t) (t + 32 + lane) * MB_ROW + s) : NI;
          __syncwarp();
        }
        {                                   // publish this block's row tokens, fetch the next block's
          __syncwarp();
          ring[(t + 32 + lane) & 127] = (uint8_t) (ynext - 1);
          ynext = rowTok (t + 64 + lane);
          __syncwarp();
        }
      };
      auto step = [&] (const int t, auto steadyTag) {
        constexpr bool STEADY = decltype (steadyTag)::value;
        const int r = t - lane;
        const int tokb = tokNext;
        tokNext = ring[(t + 1 - lane) & 127];         // next step's token, off the critical path
#ifdef MB_ROWTAB
        const unsigned eb8 = (unsigned) tokb * 8u, ebr = eBase + (unsigned) (MB_NIN * MB_WA_F * 8) + (unsigned) tokb * (unsigned) (MB_WB_F * 8);
#endif
        // left neighbour's last column at this row: a shuffle, or the staged boundary row for lane 0
        double Lc[MB_S];
#pragma unroll
        for (int s = 0; s < MB_S; ++s) {
          if (mb_live<DIR> (s)) {
#ifdef MB_ROWTAB
            Lc[s] = __shfl_up_sync (MB_FULL, U[MB_C - 1][s], 1);
            mb_lds_lane0 (Lc[s], lane, sInAddr + (unsigned) (((t & 31) * MB_ROW + s) * 8));      // a predicated load: no select
#else
            const double fromLane = __shfl_up_sync (MB_FULL, U[MB_C - 1][s], 1);
            const double fromStrip = sIn[(t & 31) * MB_ROW + s];
            Lc[s] = lane ? fromLane : fromStrip;
#endif
          } else Lc[s] = NI;
        }
        if (STEADY || (r >= 0 && r <= Lo)) {
          double Dc[MB_S];
#pragma unroll
          for (int s = 0; s < MB_S; ++s) { Dc[s] = Lk[s]; Lk[s] = Lc[s]; }
          unsigned long long pack0 = 0, pack1 = 0;
          unsigned pack32 = 0;
#ifdef MB_ROWTAB
          unsigned pk[MB_PKW];      // the step's packed back-pointers, filled field by field inside the cells
#pragma unroll
          for (int q = 0; q < MB_PKW; ++q) pk[q] = 0u;
#endif
#pragma unroll
          for (int c = 0; c < MB_C; ++c) {
            double N[MB_S];
            const bool origin = !STEADY && (r == 0) && (col0 + c == 0);
            if (MODE == 0 || MODE == 2) {
              if (DIR == 0) mb_cell_fwd (Dc, Lc, U[c], N, ta[c], tokb, origin, E, P);
              else mb_cell_bwd (Dc, Lc, U[c], N, ta[c], tokb, origin, E, P);
              if (MODE == 2 && col0 + c <= Li) {
                double* fq = Fm + ((int64_t) r * (Li + 1) + (col0 + c)) * MB_S;
                if ((MB_S & 1) == 0) {      // 16-byte aligned rows of states: vector stores
#pragma unroll
                  for (int s = 0; s + 1 < MB_S; s += 2) ((double2*) fq)[s >> 1] = make_double2 (N[s], N[s + 1]);
                } else {
#pragma unroll
                  for (int s = 0; s < MB_S; ++s) fq[s] = N[s];
                }
              }
            } else if (MODE == 3) {
              double Fc[MB_S];
              const int col = col0 + c;
              if (col <= Li) {
                const double* fp = Fm + ((int64_t) (Lo - r) * (Li + 1) + (Li - col)) * MB_S;
#pragma unroll
                for (int s = 0; s < MB_S; ++s) Fc[s] = __ldcs (fp + s) - ll;
              } else {
#pragma unroll
                for (int s = 0; s < MB_S; ++s) Fc[s] = NI;
              }
              mb_cell_cnt (Dc, Lc, U[c], N, ta[c], tokb, origin, E, P, Fc, cs, acc, c);
            } else {
#ifdef MB_ROWTAB
              mb_cell_vitr<MODE == 1> (Dc, Lc, U[c], N, ea[c], ea[c] + eb8, ebr, origin, !STEADY && r == Lo && col0 + c == Li, P, pk, 8 * MB_TBBYTES * c);
#else
              const mb_tbword word = mb_cell_vit (Dc, Lc, U[c], N, ta[c], tokb, origin, !STEADY && r == Lo && col0 + c == Li, E, P);
              if (MODE == 1) {
                const int sh = 8 * MB_TBBYTES * c;
                if (MB_C * MB_TBBYTES <= 4) pack32 |= (unsigned) word << (sh & 31);
                else if (sh < 64) pack0 |= (unsigned long long) word << (sh & 63);
                else pack1 |= (unsigned long long) word << ((sh - 64) & 63);
              }
#endif
            }
#pragma unroll
            for (int s = 0; s < MB_S; ++s) { Dc[s] = U[c][s]; U[c][s] = N[s]; Lc[s] = N[s]; }
          }
          if (MODE == 1) {
            uint8_t* p = tbRow;
#ifdef MB_ROWTAB
            pack32 = pk[0];
            pack0 = MB_PKW > 1 ? (unsigned long long) pk[0] | ((unsigned long long) pk[MB_PKW > 1 ? 1 : 0] << 32) : pk[0];
            pack1 = MB_PKW > 2 ? (unsigned long long) pk[MB_PKW > 2 ? 2 : 0] | (MB_PKW > 3 ? (unsigned long long) pk[MB_PKW > 3 ? 3 : 0] << 32 : 0ull) : 0ull;
#endif
            if (MB_C * MB_TBBYTES == 1) *p = (uint8_t) pack32;
            else if (MB_C * MB_TBBYTES == 2) *(unsigned short*) p = (unsigned short) pack32;
            else if (MB_C * MB_TBBYTES == 4) *(unsigned int*) p = pack32;
            else if (MB_C * MB_TBBYTES == 8) *(unsigned long long*) p = pack0;
            else *(ulonglong2*) p = make_ulonglong2 (pack0, pack1);      // 16 bytes, or a fitted width's padded group (MB_TBPAD)
          }
          if (hasOut && lane == 31) {
#pragma unroll
            for (int s = 0; s < MB_S; ++s) if (mb_live<DIR> (s)) boutRow[s] = U[MB_C - 1][s];
          }
          if (!STEADY && r == Lo) {
#pragma unroll
            for (int c = 0; c < MB_C; ++c)
              if (col0 + c == Li) A.result[k] = U[c][MBDir<DIR>::RES];
          }
        }
        tbRow += tbStep;
        boutRow += MB_ROW;
      };
      {
        int t = 0;
        const int rampUp = min (31, nSteps);
        for (; t < rampUp; ++t) { if ((t & 31) == 0) blockStart (t); step (t, MBBool<false>()); }
        while (t < Lo) {
          if ((t & 31) == 0) blockStart (t);
          const int tend = min (Lo, (t | 31) + 1);
#pragma unroll MB_STEADY_UNROLL
          for (; t < tend; ++t) step (t, MBBool<true>());
        }
        for (; t < nSteps; ++t) { if ((t & 31) == 0) blockStart (t); step (t, MBBool<false>()); }
      }
      if (publishes) mb_publish_rows (A.prog + w, Lo + 1);
      if (MODE == 3) mb_flush_counts (cs, acc, ta, mb_count_row<ROWS> (A, k), A.idTabB, lane);
      __syncwarp();
    }
  }
}

#ifndef MB_PAIR_ROWS
#ifndef MB_SCORE_MODULE
extern "C" __global__ void __launch_bounds__(MB_THREADS, MB_MINBLOCKS) mb_k_forward (const __grid_constant__ MBSil P, const __grid_constant__ MBArgs A) { mb_run<0, 0> (P, A); }
extern "C" __global__ void __launch_bounds__(MB_THREADS, MB_MINBLOCKS) mb_k_backward (const __grid_constant__ MBSil P, const __grid_constant__ MBArgs A) { mb_run<0, 1> (P, A); }
extern "C" __global__ void __launch_bounds__(MB_THREADS, MB_MINBLOCKS_CNT) mb_k_fstore (const __grid_constant__ MBSil P, const __grid_constant__ MBArgs A) { mb_run<2, 0> (P, A); }
extern "C" __global__ void __launch_bounds__(MB_THREADS, MB_MINBLOCKS_CNT) mb_k_bcounts (const __grid_constant__ MBSil P, const __grid_constant__ MBArgs A) { mb_run<3, 1> (P, A); }
#endif
extern "C" __global__ void __launch_bounds__(MB_THREADS, MB_MINBLOCKS) mb_k_viterbi (const __grid_constant__ MBSil P, const __grid_constant__ MBArgs A) { mb_run<1, 0> (P, A); }
extern "C" __global__ void __launch_bounds__(MB_THREADS, MB_MINBLOCKS) mb_k_viterbi_score (const __grid_constant__ MBSil P, const __grid_constant__ MBArgs A) { mb_run<4, 0> (P, A); }
#endif

// ---------------------------------------------------------------------------------------------
// Scaled linear-domain sweep (Forward for DIR 0, Backward for DIR 1).
//
// Same strip / skew mapping as mb_run, but cell values are probabilities in FP64, not log-
// probabilities: a transition group is ONE FMA (value * weight) instead of an add plus a
// log-sum-exp, and the sum it computes is the exact log-sum-exp of the log-domain recurrence.
// All live values of the warp share one power-of-two frame 2^ecur.  Every MB_RESCALE steps the warp
// takes the maximum of its live values (one integer max per value on the high word, one REDUX),
// renormalises everything to [1, 2) with an exact power-of-two multiply and adds the shift to ecur;
// in the same step it stages the next MB_RESCALE rows of the previous strip's boundary, each
// carrying its own frame, already converted to the new frame.  log-likelihood = ln(value) + ecur ln 2.
//
// FP64 spans 2^-1022 .. 2^1023.  At every rescale the warp also takes the minimum non-zero value;
// if the spread max/min exceeds 2^700 (a state that is astronomically unlikely next to its
// neighbours but could still matter later), or a boundary row arrives more than 2^900 away from the
// current frame, the pair is flagged and the host re-runs it with the log-domain kernel (mb_run), as
// it does for every pair whose result is -inf.  The host only selects this kernel when every finite
// log-weight lies in [-24 ln 2, 24 ln 2], which bounds the drift between two rescales by 2^-400.
#define MB_RESCALE 16

// MODE 0: score only.  MODE 2 (DIR 0): also store the Forward values for the E-step -- the HIGH WORD
// of each double (sign, 11-bit exponent, 20-bit mantissa, rounded: relative error 2^-21, full FP64
// range), 4 bytes instead of 8, and only for the states an emitting transition enters (the rest of a
// cell follows from those through its silent transitions, mb_fexpand_lin), plus the frame exponent of
// every rescale block.
// MODE 3 (DIR 1): Backward fused with the posterior counts: for each transition group the product
// term = B(dest) * w feeds the Backward sum and, times F(src) * 2^(eF + eB) / Z, the group's count.
template<int MODE, int DIR, class SIL, bool ROWS = false>
__device__ __forceinline__ void mb_run_lin (const SIL& P, const MBArgs& A) {
#ifdef MB_LANE_FRAMES
  constexpr bool LF = MODE == 0;
#else
  constexpr bool LF = false;
#endif
  extern __shared__ double mb_smem[];
  double* E = mb_smem;
  const int NE = MBDir<DIR>::NE;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int q = threadIdx.x; q < NE; q += blockDim.x) E[q] = A.emit[q];
  __syncthreads();
#ifdef MB_ROWTAB
  // score module: the normalised linear weights in row layout (see the generated prelude)
  constexpr bool ROW = MODE == 0;
  const unsigned eBase = (unsigned) __cvta_generic_to_shared (E);
  constexpr unsigned WA8 = (DIR ? MB_WA_B : MB_WA_F) * 8, WB8 = (DIR ? MB_WB_B : MB_WB_F) * 8;
#else
  constexpr bool ROW = false;
#endif
  // shared memory layout as in mb_run; the count accumulators are FP64 here: accd[ctx * 32 + lane]
  const int nWarps = blockDim.x >> 5;
  uint8_t* ring = (uint8_t*) (mb_smem + ((NE + 1) & ~1)) + warp * 128;
  double* sIn = mb_smem + ((NE + 1) & ~1) + nWarps * 16 + warp * (32 * MB_ROW);
  double* accd = mb_smem + ((NE + 1) & ~1) + nWarps * (16 + 32 * MB_ROW) + warp * (32 * MB_NCTX) + lane;
  // MODE 3: two warp-step blocks of stored Forward words, filled by cp.async one step ahead
  unsigned* fstage = (unsigned*) (mb_smem + ((NE + 1) & ~1) + nWarps * (16 + 32 * MB_ROW + 32 * MB_NCTX)) + warp * (2 * MB_FBLOCK);
  const int64_t wslot = (int64_t) blockIdx.x * nWarps + warp;
  double* bndA = A.bnd + wslot * A.bndStride;
  double* bndB = bndA + (A.bndStride >> 1);
  const unsigned sInAddr = (unsigned) __cvta_generic_to_shared (sIn);

  for (;;) {
    unsigned long long w = 0;
    if (lane == 0) w = atomicAdd (A.counter, 1ULL);
    w = __shfl_sync (MB_FULL, w, 0);
    if ((int64_t) w >= A.nWork) break;
    const bool split = MB_SPLIT && A.items != 0;
    const int64_t item = split ? A.items[w] : 0;
    const int64_t k = split ? (item >> 16) : A.order[w];
    const int64_t x0 = A.xOff[k], y0 = A.yOff[k];
    const int Li = (int) (A.xOff[k + 1] - x0), Lo = (int) (A.yOff[k + 1] - y0);
    const uint8_t* x = A.x + x0;
    const uint8_t* y = A.y + y0;
    const int nStrips = (Li + MB_W) / MB_W;
    int suspect = 0;
    const int nBlk = (Lo + 32 + MB_RESCALE - 1) / MB_RESCALE;
    unsigned* F32 = (MODE == 2 || MODE == 3) ? A.F32 + A.f32Off[k] : (unsigned*) 0;
    int32_t* ef = (MODE == 2 || MODE == 3) ? A.ef + A.efOff[k] : (int32_t*) 0;
    // 1/Z = zf * 2^-lzi with Z = exp(ll) the pair's Forward likelihood (MODE 3)
    int lzi = 0;
    double zf = 1.0;
    if (MODE == 3) {
      const double llk = A.ll[k];
      if (!(llk > mb_neg_inf())) continue;    // impossible pair: no posterior
      const double lz = llk * 1.4426950408889634074;
      const double fl = floor (lz);
      lzi = (int) fl;
      zf = exp2 (fl - lz);
    }

    const int stripFirst = split ? (int) (item & 0xffff) : 0, stripEnd = split ? stripFirst + 1 : nStrips;
    for (int strip = stripFirst; strip < stripEnd; ++strip) {
      // MODE 3 pads the matrix on the LEFT of the reversed sweep (columns < 0: every value there stays
      // exactly 0, a sum of products of zeros), so that its strips and lanes mirror the Forward sweep's:
      // step t of this strip then needs exactly the block the Forward wrote at step Lo+31-t of strip
      // nStrips-1-strip, and both sides stream whole warp-sized blocks (see MB_FBLOCK).
      const int col0 = strip * MB_W + lane * MB_C - (MODE == 3 ? nStrips * MB_W - (Li + 1) : 0);
      int ta[MB_C];
#ifdef MB_ROWTAB
      unsigned ea[MB_C];      // shared-memory address of each column's input-token row
#endif
#pragma unroll
      for (int c = 0; c < MB_C; ++c) {
        const int i = col0 + c;
        int tok = 1;
        if (i >= 1 && i <= Li) tok = DIR ? x[Li - i] : x[i - 1];
        ta[c] = tok - 1;
#ifdef MB_ROWTAB
        ea[c] = eBase + (unsigned) (tok - 1) * WA8;
#endif
      }
      double U[MB_C][MB_S], Lk[MB_S];
#pragma unroll
      for (int s = 0; s < MB_S; ++s) {
        Lk[s] = 0.0;
#pragma unroll
        for (int c = 0; c < MB_C; ++c) U[c][s] = 0.0;
      }
      double csd[MB_NSIL_B > 0 ? MB_NSIL_B : 1];
      if (MODE == 3) {
#pragma unroll
        for (int q = 0; q < (MB_NSIL_B > 0 ? MB_NSIL_B : 1); ++q) csd[q] = 0.0;
        for (int q = 0; q < MB_NCTX; ++q) accd[q * 32] = 0.0;
      }
      const bool hasIn = strip > 0, hasOut = strip + 1 < nStrips;
      const double* bin = split ? (hasIn ? A.bnd + A.itemBnd[w - 1] : bndA) : ((strip & 1) ? bndB : bndA);
      double* bout = split ? A.bnd + A.itemBnd[w] : ((strip & 1) ? bndA : bndB);
      const bool waits = split && hasIn, publishes = split && hasOut && lane == 31;
      if (!hasIn) {
        __syncwarp();
        for (int q = lane; q < MB_RESCALE * MB_ROW; q += 32) sIn[q] = 0.0;
        __syncwarp();
      }
      if (waits) mb_wait_rows (A.prog + (w - 1), min (MB_RESCALE, Lo + 1));
      // row tokens (0-based): rows 0..31 are published now, rows 32..63 at step 0, and so on one block ahead
      // (the raw 1-based byte is kept until it is published a block later: subtracting 1 at once would make
      // the warp wait for the global load)
      auto rowTok = [&] (const int row) { return (row >= 1 && row <= Lo) ? (int) (DIR ? y[Lo - row] : y[row - 1]) : 1; };
      __syncwarp();
      ring[lane] = (uint8_t) (rowTok (lane) - 1);
      int ynext = rowTok (32 + lane);
      __syncwarp();
      int tokNext = ring[(0 - lane) & 127];          // token of this lane's row at step 0 (only lane 0's is real)
      // frame: true value = stored value * 2^ecur; a strip starts in the frame of its first boundary row.
      // LF (score-only sweeps of the wide-lane module): every lane keeps its OWN frame, so that the spread
      // check spans only the lane's columns and the strip can be 256 columns wide; the left neighbour's
      // values then arrive through the exact power-of-two factor gl = 2^(its frame - mine), refreshed
      // whenever the lanes renormalise.
      int ecur = hasIn ? (int) __ldcg (bin + MB_S) : 0;
      double gl = 1.0;
      double stageNext[MB_S];
      double stageNextE = (double) ecur;      // converted when it is used, a block after the load
#pragma unroll
      for (int s = 0; s < MB_S; ++s)
        stageNext[s] = (hasIn && mb_live<DIR> (s) && lane < MB_RESCALE && lane <= Lo) ? __ldcg (bin + (int64_t) lane * MB_ROW + s) : 0.0;
      if (hasIn && lane < MB_RESCALE && lane <= Lo) stageNextE = __ldcg (bin + (int64_t) lane * MB_ROW + MB_S);
      if (MODE == 3) {      // the first step's Forward block
        const unsigned* srcb = F32 + ((int64_t) (nStrips - 1 - strip) * (Lo + 32) + (Lo + 31)) * MB_FBLOCK;
#pragma unroll
        for (int j = 0; j < MB_C * MB_SQ; ++j) mb_cp_async16 (fstage + (j * 32 + lane) * 4, srcb + (j * 32 + (31 - lane)) * 4);
        mb_cp_async_commit();
      }
      const int nSteps = Lo + 32;
      double* boutRow = bout + (int64_t) (0 - lane) * MB_ROW;      // this lane's row r = t - lane of the outgoing boundary, advanced per step
      // one step of the skewed sweep; STEADY = every lane is inside the matrix (31 <= t < Lo), so the
      // ramp predicates (row in range, origin cell, result cell) fold away
      // every MB_RESCALE steps (kept out of the step body so that the steady loop carries no block tests)
      auto blockStart = [&] (const int t) {
        if (publishes && t >= 32) mb_publish_rows (A.prog + w, t - 31);      // (steps < t are done: lane 31 has written rows <= t - 32)
        if (waits) mb_wait_rows (A.prog + (w - 1), min (t + 2 * MB_RESCALE, Lo + 1));
        {
          bool nz = false;      // LF: this lane holds something
          if (t > 0) {
            int mh = 0;
            unsigned ml = 0xffffffffu;
#pragma unroll
            for (int s = 0; s < MB_S; ++s) {
              if (!mb_live<DIR> (s)) continue;
              const int h = __double2hiint (Lk[s]);
              mh = max (mh, h); ml = min (ml, (unsigned) (h - 1));
#pragma unroll
              for (int c = 0; c < MB_C; ++c) { const int g = __double2hiint (U[c][s]); mh = max (mh, g); ml = min (ml, (unsigned) (g - 1)); }
            }
            if (!LF) {
              mh = __reduce_max_sync (MB_FULL, mh);
              ml = __reduce_min_sync (MB_FULL, ml);
            }
            nz = mh >= 0x00100000;
            if (nz) {
              const int ex = mh >> 20;
              const int shift = min (ex - 1023, 1000);
              if (shift != 0) {
                const double f = __hiloint2double ((1023 - shift) << 20, 0);
#pragma unroll
                for (int s = 0; s < MB_S; ++s) {
                  if (!mb_live<DIR> (s)) continue;
                  Lk[s] *= f;
#pragma unroll
                  for (int c = 0; c < MB_C; ++c) U[c][s] *= f;
                }
                ecur += shift;
              }
              if (ml != 0xffffffffu && ex - (int) ((ml + 1u) >> 20) > 700) suspect |= 1;
            }
          }
          if (LF) {
            // A lane that holds nothing yet takes the frame of what is about to reach it: the nearest lane to its left
            // that holds something, or -- for the lanes left of all of those -- the first staged boundary row that is
            // not all zero (a strip starts with every lane empty, and far from the diagonal its first rows have
            // underflowed to zero and carry a meaningless frame).  Then every lane learns its left neighbour's frame.
            bool rowNz = false;
            if (hasIn && lane < MB_RESCALE) {
#pragma unroll
              for (int s = 0; s < MB_S; ++s) if (mb_live<DIR> (s)) rowNz |= stageNext[s] != 0.0;
            }
            const unsigned rowMask = __ballot_sync (MB_FULL, rowNz), nzMask = __ballot_sync (MB_FULL, nz);
            const double eRow = __shfl_sync (MB_FULL, stageNextE, rowMask ? __ffs (rowMask) - 1 : 0);
            if (lane == 0 && !nz && hasIn) ecur = (int) eRow;
            const unsigned below = nzMask & ((1u << lane) - 1u);
            const int eFrom = __shfl_sync (MB_FULL, ecur, below ? 31 - __clz (below) : 0);
            if (!nz && lane > 0) ecur = eFrom;
            const int eL = __shfl_up_sync (MB_FULL, ecur, 1);
            const bool leftNz = __shfl_up_sync (MB_FULL, (int) nz, 1) != 0;
            int d = lane ? eL - ecur : 0;
            if (leftNz && (d < -900 || d > 900)) suspect |= 2;
            d = max (min (d, 1000), -1022);
            gl = __hiloint2double ((1023 + d) << 20, 0);
          }
          if (MODE == 2 && lane == 0) ef[strip * nBlk + t / MB_RESCALE] = ecur;
          if (hasIn) {     // stage rows t .. t+MB_RESCALE-1 of the previous strip's last column, in the current frame;
            const int e0 = LF ? __shfl_sync (MB_FULL, ecur, 0) : ecur;      // (lane 0's frame: it is the one that reads them)
            __syncwarp();  // lane q < MB_RESCALE takes row t+q: fetched a block ago, the next block's are fetched now
            if (lane < MB_RESCALE) {
              double* dst = sIn + lane * MB_ROW;
              int d = (int) stageNextE - e0;
              const bool far = d < -900 || d > 900;
              bool any = false;
              d = max (min (d, 1000), -1023);
              const double f = __hiloint2double ((1023 + d) << 20, 0);
#pragma unroll
              for (int s = 0; s < MB_S; ++s)
                if (mb_live<DIR> (s)) { any |= stageNext[s] != 0.0; dst[s] = stageNext[s] * f; }
              if (far && any) suspect |= 4;
              const int rowN = t + MB_RESCALE + lane;
              const double* src = bin + (int64_t) rowN * MB_ROW;
#pragma unroll
              for (int s = 0; s < MB_S; ++s) if (mb_live<DIR> (s)) stageNext[s] = rowN <= Lo ? __ldcg (src + s) : 0.0;
              stageNextE = rowN <= Lo ? __ldcg (src + MB_S) : (double) e0;
            }
            __syncwarp();
          }
        }
        if ((t & 31) == 0) {                // publish this block's row tokens, fetch the next block's
          __syncwarp();
          ring[(t + 32 + lane) & 127] = (uint8_t) (ynext - 1);
          ynext = rowTok (t + 64 + lane);
          __syncwarp();
        }
      };
      auto step = [&] (const int t, auto steadyTag) {
        constexpr bool STEADY = decltype (steadyTag)::value;
        const int r = t - lane;
        const int tokb = tokNext;
        tokNext = ring[(t + 1 - lane) & 127];         // next step's token, off the critical path
#ifdef MB_ROWTAB
        const unsigned eb8 = (unsigned) tokb * 8u, ebr = eBase + (unsigned) MB_NIN * WA8 + (unsigned) tokb * WB8;
#endif
        double Lc[MB_S];
#pragma unroll
        for (int s = 0; s < MB_S; ++s) {
          if (mb_live<DIR> (s)) {
#ifdef MB_ROWTAB
            double v = __shfl_up_sync (MB_FULL, U[MB_C - 1][s], 1);
            if (LF) v *= gl;
            mb_lds_lane0 (v, lane, sInAddr + (unsigned) (((t & (MB_RESCALE - 1)) * MB_ROW + s) * 8));      // a predicated load: no select
            Lc[s] = v;
#else
            const double fromLane = __shfl_up_sync (MB_FULL, U[MB_C - 1][s], 1);
            const double fromStrip = sIn[(t & (MB_RESCALE - 1)) * MB_ROW + s];
            Lc[s] = lane ? (LF ? fromLane * gl : fromLane) : fromStrip;
#endif
          } else Lc[s] = 0.0;
        }
        // Forward block of this step.  MODE 2 writes it.  MODE 3 reads the mirrored one: it was copied
        // into shared memory by cp.async during the previous step (each lane copies exactly the 16-byte
        // chunks it will read, so no warp barrier is needed), the next one is issued now, and the one
        // after that is pulled into L2.
        unsigned* fblk = (unsigned*) 0;
        const unsigned* fsm = (const unsigned*) 0;
        if (MODE == 2) fblk = F32 + ((int64_t) strip * nSteps + t) * MB_FBLOCK;
        if (MODE == 3) {
          fblk = F32 + ((int64_t) (nStrips - 1 - strip) * nSteps + (Lo + 31 - t)) * MB_FBLOCK;
          mb_cp_async_wait_all();
          fsm = fstage + (t & 1) * MB_FBLOCK;
          if (t + 1 < nSteps) {
            unsigned* dstb = fstage + ((t + 1) & 1) * MB_FBLOCK;
            const unsigned* srcb = fblk - MB_FBLOCK;
#pragma unroll
            for (int j = 0; j < MB_C * MB_SQ; ++j) mb_cp_async16 (dstb + (j * 32 + lane) * 4, srcb + (j * 32 + (31 - lane)) * 4);
            mb_cp_async_commit();
          }
          if (t + 3 < nSteps) {
            mb_prefetch_l2 (fblk - 3 * MB_FBLOCK + lane * 32);
            if (MB_FBLOCK > 1024) mb_prefetch_l2 (fblk - 3 * MB_FBLOCK + 1024 + lane * 32);
          }
        }
        if (STEADY || (r >= 0 && r <= Lo)) {
          double Dc[MB_S];
#pragma unroll
          for (int s = 0; s < MB_S; ++s) { Dc[s] = Lk[s]; Lk[s] = Lc[s]; }
          double kapStep = 0.0;      // MODE 3: stored Forward word -> F * 2^(eF + eB) / Z, one factor for the whole step
          if (MODE == 3) {
            const int eF = __ldg (ef + (nStrips - 1 - strip) * nBlk + (Lo + 31 - t) / MB_RESCALE);      // frame of the Forward block: its strip and step
            const int d = max (min (eF + ecur - lzi, 1000), -1023);
            kapStep = zf * __hiloint2double ((1023 + d) << 20, 0);
          }
#pragma unroll
          for (int c = 0; c < MB_C; ++c) {
            double N[MB_S];
            const bool origin = !STEADY && (r == 0) && (col0 + c == 0);
            if constexpr (MODE == 3) {
              double Fc[MB_S];
              const int col = col0 + c;
              // written by Forward lane 31-lane as its cell MB_C-1-c; the padding columns hold finite values
              // too, so a zero factor replaces a branch around the loads
              const double kap = (col >= 0 && col <= Li) ? kapStep : 0.0;
              unsigned hw[4 * MB_SQ];
#pragma unroll
              for (int g = 0; g < MB_SQ; ++g) {
                const uint4 q = *(const uint4*) (fsm + (((MB_C - 1 - c) * MB_SQ + g) * 32 + lane) * 4);
                hw[4 * g] = q.x; hw[4 * g + 1] = q.y; hw[4 * g + 2] = q.z; hw[4 * g + 3] = q.w;
              }
              mb_fexpand_lin (hw, kap, Fc, P);      // the kept states, and through the silent groups the others
              mb_cell_cnt_lin (Dc, Lc, U[c], N, ta[c], tokb, origin, E, P, Fc, csd, accd, c);
            } else {
#ifdef MB_ROWTAB
              if constexpr (ROW) {
                if (DIR == 0) mb_cell_fwd_linr (Dc, Lc, U[c], N, ea[c], ea[c] + eb8, ebr, origin, P);
                else mb_cell_bwd_linr (Dc, Lc, U[c], N, ea[c], ea[c] + eb8, ebr, origin, P);
              } else
#endif
              {
                if (DIR == 0) mb_cell_fwd_lin (Dc, Lc, U[c], N, ta[c], tokb, origin, E, P);
                else mb_cell_bwd_lin (Dc, Lc, U[c], N, ta[c], tokb, origin, E, P);
              }
              if (MODE == 2) {
                // high words, rounded; 16-byte chunk g of cell c goes to word ((c*MB_SQ + g)*32 + lane)*4 of
                // the block, so every store instruction of the warp writes 512 contiguous bytes
                unsigned hw[4 * MB_SQ];
                mb_fpack_lin (N, hw);
#pragma unroll
                for (int g = 0; g < MB_SQ; ++g)
                  *(uint4*) (fblk + ((c * MB_SQ + g) * 32 + lane) * 4) = make_uint4 (hw[4 * g], hw[4 * g + 1], hw[4 * g + 2], hw[4 * g + 3]);
              }
            }
#pragma unroll
            for (int s = 0; s < MB_S; ++s) { Dc[s] = U[c][s]; U[c][s] = N[s]; Lc[s] = N[s]; }
          }
          if (hasOut && lane == 31) {
#pragma unroll
            for (int s = 0; s < MB_S; ++s) if (mb_live<DIR> (s)) boutRow[s] = U[MB_C - 1][s];
            boutRow[MB_S] = (double) ecur;
          }
          if (!STEADY && r == Lo) {
#pragma unroll
            for (int c = 0; c < MB_C; ++c)
              if (col0 + c == Li) {
                const double v = U[c][MBDir<DIR>::RES];
                A.result[k] = v > 0.0 ? log (v) + (double) ecur * 0.6931471805599453094 + mb_res_log<DIR> (P) : mb_neg_inf();
              }
          }
        }
        boutRow += MB_ROW;
      };
      {
        int t = 0;
        // MODE 3 pads its matrix on the left, so column 0 -- the origin cell, at row 0 -- can sit on any lane, lane 31
        // included, whose row 0 is step 31: the steady loop (which folds the origin test away) starts a step later there
        const int rampUp = min (MODE == 3 ? 32 : 31, nSteps);
        for (; t < rampUp; ++t) { if ((t & (MB_RESCALE - 1)) == 0) blockStart (t); step (t, MBBool<false>()); }
        while (t < Lo) {
          if ((t & (MB_RESCALE - 1)) == 0) blockStart (t);
          const int tend = min (Lo, (t | (MB_RESCALE - 1)) + 1);
#pragma unroll MB_STEADY_UNROLL
          for (; t < tend; ++t) step (t, MBBool<true>());
        }
        for (; t < nSteps; ++t) { if ((t & (MB_RESCALE - 1)) == 0) blockStart (t); step (t, MBBool<false>()); }
      }
      if (publishes) mb_publish_rows (A.prog + w, Lo + 1);
      suspect = (int) __reduce_or_sync (MB_FULL, (unsigned) suspect);      // why: 1 spread, 2 neighbour frame, 4 boundary frame
      if (MODE == 3) mb_flush_counts_lin (csd, accd, ta, mb_count_row<ROWS> (A, k), A.idTabB, lane);
      __syncwarp();
    }
    if (lane == 0) { if (split) { if (suspect) atomicOr (A.flag + k, suspect); } else A.flag[k] = suspect; }
  }
}

#ifndef MB_PAIR_ROWS
#ifdef MB_ROWTAB
extern "C" __global__ void __launch_bounds__(MB_THREADS, MB_MINBLOCKS_LIN) mb_k_forward_lin (const __grid_constant__ MBSilN P, const __grid_constant__ MBArgs A) { mb_run_lin<0, 0> (P, A); }
extern "C" __global__ void __launch_bounds__(MB_THREADS, MB_MINBLOCKS_LIN) mb_k_backward_lin (const __grid_constant__ MBSilN P, const __grid_constant__ MBArgs A) { mb_run_lin<0, 1> (P, A); }
#else
extern "C" __global__ void __launch_bounds__(MB_THREADS, MB_MINBLOCKS_LIN) mb_k_forward_lin (const __grid_constant__ MBSil P, const __grid_constant__ MBArgs A) { mb_run_lin<0, 0> (P, A); }
extern "C" __global__ void __launch_bounds__(MB_THREADS, MB_MINBLOCKS_LIN) mb_k_backward_lin (const __grid_constant__ MBSil P, const __grid_constant__ MBArgs A) { mb_run_lin<0, 1> (P, A); }
#endif
#ifndef MB_SCORE_MODULE
extern "C" __global__ void __launch_bounds__(MB_THREADS, MB_MINBLOCKS_LIN) mb_k_fstore_lin (const __grid_constant__ MBSil P, const __grid_constant__ MBArgs A) { mb_run_lin<2, 0> (P, A); }
extern "C" __global__ void __launch_bounds__(MB_THREADS, MB_MINBLOCKS_CNT) mb_k_bcounts_lin (const __grid_constant__ MBSil P, const __grid_constant__ MBArgs A) { mb_run_lin<3, 1> (P, A); }
#endif
#else
// the per-pair count module (built the first time a call asks for per-pair counts): only the two count kernels, each
// flushing into the row of its pair
extern "C" __global__ void __launch_bounds__(MB_THREADS, MB_MINBLOCKS_CNT) mb_k_bcounts_rows (const __grid_constant__ MBSil P, const __grid_constant__ MBArgs A) { mb_run<3, 1, true> (P, A); }
extern "C" __global__ void __launch_bounds__(MB_THREADS, MB_MINBLOCKS_CNT) mb_k_bcounts_lin_rows (const __grid_constant__ MBSil P, const __grid_constant__ MBArgs A) { mb_run_lin<3, 1, MBSil, true> (P, A); }
#endif
)MBSRC";

#endif
