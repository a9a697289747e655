// viterbiFillBatchKernel: the ViterbiMatrix fill (reference src/viterbi.cpp:62-176) with the READS AS THE
// SIMD LANES.  A group of 32 reads walks the machine together: lane r of every warp works on read r of the
// group and a warp works on one state at a time.  What that buys over one-read-per-cluster
// (viterbi_fill_push.cu, 45 warp-instructions per state-column per read, < 6 % of them fp64):
//   * a transition word, its score and its addresses are decoded ONCE per warp and serve 32 reads;
//   * a gather of S(src), D(src) is one 512-byte row of shared memory, conflict free (one ld.shared.v2.f64);
//   * the closure's control flow (which states are dirty, which transitions to relax) is warp-uniform:
//     no divergence, no per-lane queues; lanes differ only in the fp64 values they add and compare;
//   * records leave as full 32-byte sectors: pred[group][pos][state][cell kind][32 reads].
// The closure is the same least fixed point as the reference's worklist (src/viterbi.cpp:110-159; any fair
// schedule reaches the same bits, SURVEY.md 8a-6), organised as OWNER-COMPUTES edge relaxation: every state
// has a 32-bit work mask, bit j = "in-transition j's source grew (for some read of the group)".  The warp
// that owns a state relaxes exactly the flagged transitions (reading the source's row, writing only its own
// row: no atomics on DP cells, no lost updates), and if any lane grew it flags the corresponding bit of
// each successor's mask.  By default there are no levels and no barriers inside a column: every warp keeps
// relaxing whichever of its states are flagged until the CTA (the team) is quiet; the first version's
// breadth-first levels with one CTA barrier each are still selectable (async_closure = 0).
// tools/union_frontier.py measured what sharing one frontier among 32 reads costs:
// 2.9-7.6 state visits per column instead of 2.0-2.9 per read, i.e. 0.09-0.24 warp-level visits per read.
//
// A TEAM of T CTAs holds the (S,D) columns of one group in shared memory, M = ceil(N/T) states each
// (M*512 bytes); T = 1 for dnastore-l4, the whole GPU for the 46,670-state BASELINE machine.  Nothing
// crosses CTAs through shared memory: a state with successors in other CTAs PUBLISHES its (S,D) row to an
// L2-resident array whenever it grows and then adds 1 to a NOTIFICATION COUNTER of the owner CTA (one counter per
// class of destination states, see the team protocol below); the owner polls its counters when it runs out of
// local work, and the team meets at a counter barrier in L2 once per column.  Nothing is limited by the
// 16-CTA cluster size, so machines that do not fit a cluster (SURVEY 8 f-4) use the same code path.
//
// After the closure one dense pass per column (a) evaluates the predecessor records with the TRACEBACK's
// own association and candidate order (src/viterbi.cpp:251-286), first strict maximum, one byte per DP
// cell; (b) opens duplications (src/viterbi.cpp:161-168); (c) performs the emission step of the NEXT column
// (src/viterbi.cpp:92-106) from the same gathered S(pos)[src] rows.
#include <cuda_runtime.h>

#include <cstdint>

#include "viterbi_batch.h"
#include "viterbi_kernels.h"

namespace dnab {
namespace {

__device__ __forceinline__ uint32_t smemAddr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ double negInf() { return __longlong_as_double(0xFFF0000000000000LL); }
// std::max(a,b) of the reference: keeps a on ties
__device__ __forceinline__ double dmax(double a, double b) { return (a < b) ? b : a; }

// (S,D) of one read of one state: 16 bytes; a warp reads a 512-byte row.  volatile: other warps write rows.
__device__ __forceinline__ double2 ldsRow(uint32_t a) {
  double2 v;
  asm volatile("ld.volatile.shared.v2.f64 {%0,%1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(a));
  return v;
}
__device__ __forceinline__ void stsRow(uint32_t a, double s, double d) {
  asm volatile("st.volatile.shared.v2.f64 [%0], {%1,%2};" ::"r"(a), "d"(s), "d"(d) : "memory");
}
// rows published through L2 for readers on other SMs: never through the reader's L1
__device__ __forceinline__ double2 ldPub2(const double2* p) {
  double2 v;
  asm volatile("ld.relaxed.gpu.global.v2.f64 {%0,%1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void stPub2(double2* p, double s, double d) {
  asm volatile("st.relaxed.gpu.global.v2.f64 [%0], {%1,%2};" ::"l"(p), "d"(s), "d"(d) : "memory");
}
// predecessor records are written once and read by another kernel: streaming stores
__device__ __forceinline__ void stRecord(uint8_t* p, uint32_t v) {
  asm volatile("st.global.cs.u8 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ldVolatileGlobal32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long ldAcquire64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

enum : uint32_t { kCtlFlag = 0, kCtlWake = 4, kCtlDecision = 8, kCtlPending = 16, kCtlPhase = 17, kCtlLock = 18, kCtlSeen = 32 };
constexpr uint32_t kKeepRecord = 0x100u;  // "the S record written by the previous column's pass stands"
constexpr uint32_t kKeepRecordWide = 0x10000u;  // (the same in a kernel for wide states, whose indices reach 0xFFFF)

__device__ __forceinline__ void fenceRelease() { asm volatile("fence.release.gpu;" ::: "memory"); }
__device__ __forceinline__ void stRecordEarly(uint8_t* p, uint32_t v) { asm volatile("st.global.u8 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
// rows carried from one column to the next: rewritten in place every column, so they should stay in L2 (evict-last)
// while the record stream passes through (evict-first)
__device__ __forceinline__ unsigned long long policyEvictLast() {
  unsigned long long pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ double ldCarried(const double* p, unsigned long long pol) {
  double v;
  asm volatile("ld.global.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(pol) : "memory");
  return v;
}
__device__ __forceinline__ void stCarried(double* p, double v, unsigned long long pol) {
  asm volatile("st.global.L2::cache_hint.f64 [%0], %1, %2;" ::"l"(p), "d"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ void redAdd32(uint32_t* p, uint32_t v) {
  asm volatile("red.relaxed.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void stRelaxed32(uint32_t* p, uint32_t v) {
  asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

}  // namespace

// W warps per CTA; KMAX >= k duplication columns unrolled; kTeam: the group's states are spread over T > 1 CTAs;
// kWide: the machine has wide states (viterbi_device.cuh, viterbi_batch.h); only those machines run this instantiation.
template <int W, int KMAX, bool kTeam, bool kDebug, bool kWide>
__global__ void __launch_bounds__(W * 32, 1)
    viterbiFillBatchKernel(const __grid_constant__ BatchTables tb, const __grid_constant__ BatchArgs args) {
  extern __shared__ __align__(16) unsigned char smem[];
  constexpr uint32_t nThreads = W * 32;
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5, lane16 = lane * 16u;
  const uint32_t T = kTeam ? tb.T : 1u, M = tb.M, k = tb.k, Np = T * M, N = tb.nStates, K2 = k + 2;
  const uint32_t team = kTeam ? blockIdx.x / T : blockIdx.x, rank = kTeam ? blockIdx.x - team * T : 0u;
  const uint32_t nSlots = (M + W - 1) / W;
  const double NEG = negInf();
  const BatchLayout lay = makeBatchLayout(M, tb.maxIn, tb.maxOut, tb.nSyms, kTeam);
  // counts of a wide state (header: viterbi_batch.h)
  auto wideCounts = [&](const uint4& h) { return __ldg(tb.wide + bhWideNo(h)); };
  auto nOutLocalOf = [&](const uint4& h) { return (kWide && bhWide(h)) ? (wideCounts(h).w & 0xFFFFu) : bhNOutLocal(h); };
  auto nOutOf = [&](const uint4& h) { return (kWide && bhWide(h)) ? (wideCounts(h).w >> 16) : bhNOut(h); };

  const uint32_t aSD = smemAddr(smem + lay.sd);
  uint32_t* maskCur = reinterpret_cast<uint32_t*>(smem + lay.maskA);
  uint32_t* maskNext = reinterpret_cast<uint32_t*>(smem + lay.maskB);
  uint32_t* remInS = reinterpret_cast<uint32_t*>(smem + lay.remIn);
  uint32_t* clsOffS = reinterpret_cast<uint32_t*>(smem + lay.cls);  // [kNotifyClasses + 1] then the states, by class
  uint32_t* clsStS = clsOffS + kNotifyClasses + 1;
  uint4* hdrS = reinterpret_cast<uint4*>(smem + lay.hdr);
  uint2* hdr2S = reinterpret_cast<uint2*>(smem + lay.hdr2);
  uint2* inS = reinterpret_cast<uint2*>(smem + lay.inE);
  uint2* relS = reinterpret_cast<uint2*>(smem + lay.relE);
  uint32_t* outS = reinterpret_cast<uint32_t*>(smem + lay.outE);
  double* tsE = reinterpret_cast<double*>(smem + lay.tsE);
  double* subS = reinterpret_cast<double*>(smem + lay.sub);
  volatile uint32_t* ctl = reinterpret_cast<volatile uint32_t*>(smem + lay.ctl);

  // ---- the CTA's slice of the tables, resident for the whole launch; local sources become row addresses ----
  {
    for (uint32_t i = tid; i < M; i += nThreads) {
      hdrS[i] = tb.hdr[rank * M + i];
      hdr2S[i] = tb.hdr2[rank * M + i];
      if (kTeam) {
        remInS[i] = tb.remoteIn[rank * M + i];
        clsStS[i] = tb.clsStates[rank * M + i];
      }
      maskCur[i] = 0;
      maskNext[i] = 0;
    }
    const uint32_t inBase = tb.rankInOff[rank], nIn = tb.rankInOff[rank + 1] - inBase;
    for (uint32_t i = tid; i < nIn; i += nThreads) {
      uint2 e = tb.inEdges[inBase + i];
      if (!beRemote(e)) e.x = aSD + (e.x - rank * M) * 512u;
      inS[i] = e;
      uint2 q = tb.relEdges[inBase + i];  // relax entries: local ones come first (hdr2 counts), remote ones keep g
      relS[i] = q;
    }
    __syncthreads();
    for (uint32_t i = tid; i < M; i += nThreads) {
      const uint2 h2 = hdr2S[i];
      uint32_t nLoc = (h2.y & 0xFFu) + ((h2.y >> 8) & 0xFFu);
      if (kWide && bhWide(hdrS[i])) {
        const uint32_t lc = wideCounts(hdrS[i]).y;
        nLoc = (lc & 0xFFFFu) + (lc >> 16);
      }
      for (uint32_t j = 0; j < nLoc; ++j) relS[h2.x + j].x = aSD + (relS[h2.x + j].x - rank * M) * 512u;
    }
    const uint32_t outBase = tb.rankOutOff[rank], nOut = tb.rankOutOff[rank + 1] - outBase;
    for (uint32_t i = tid; i < nOut; i += nThreads) outS[i] = tb.outEdges[outBase + i];
    for (uint32_t i = tid; i < tb.nSyms * 16; i += nThreads) tsE[i] = tb.tsE[i];
    if (tid < 16) subS[tid] = tb.sub[tid];
    if (tid < 64) ctl[tid] = 0;
    if (kTeam && tid <= kNotifyClasses) clsOffS[tid] = tb.clsOff[rank * (kNotifyClasses + 1) + tid];
  }
  __syncthreads();

  // per-state rows private to the owning lane, interleaved: [state][s0 | best emit candidate | k parked T cells][32]
  const uint32_t privKinds = 2 + k;
  double* const privT = args.priv + (size_t)team * Np * privKinds * 32 + lane;
  const unsigned long long polLast = policyEvictLast();
  double2* const sdPubT = args.sdPub + (size_t)team * 2 * Np * 32;  // two parities of the column
  // Team protocol (no returning atomic, no flag to clear).  The states of a CTA that have transitions from other CTAs are
  // dealt into kNotifyClasses classes; notifyT[c * kNotifyClasses + q] counts the notifications ever sent to class q of
  // CTA c ("a source of some state of that class published a new row").  passiveT[parity] = (CTAs of this column that are
  // passive) - (notifications sent and not yet consumed): a sender subtracts its notifications BEFORE the fence that
  // precedes them; the receiver adds what it consumed when it consumes it; so the count can only reach T when every CTA is
  // passive and nothing is undelivered.  Lane q of warp 0 polls class q (one 128-byte line for the warp) and flags only
  // that class's states: a wake-up re-relaxes a 32nd of the transitions that cross CTAs instead of all of them.
  uint32_t* const notifyT = args.teamState + (size_t)team * T * kNotifyClasses;
  uint32_t* const passiveT = args.teamPassive + (size_t)team * 2;
  uint32_t notifySeen = 0;  // (level-synchronous variant, thread 0) notifications consumed so far; the asynchronous closure keeps
                            // one count per class in ctl[kCtlSeen..]; the counters are zeroed before the launch
  unsigned long long* const bar = args.barrier + team;
  unsigned long long barTarget = 0;
  uint32_t col = 0;

  // Team barrier: CTA barrier, one arrival per CTA on a monotonic L2 counter, CTA barrier.
  auto teamBarrier = [&]() {
    __syncthreads();
    if (!kTeam) return;
    barTarget += T;
    if (tid == 0) {
      fenceRelease();
      atomicAdd(bar, 1ull);
      while (ldAcquire64(bar) < barTarget) {
      }
    }
    __syncthreads();
  };

  unsigned long long dbgLevels = 0, dbgVisits = 0, dbgEdges = 0, dbgWakes = 0, dbgClosure = 0, dbgRecord = 0, dbgPassive = 0, dbgInit = 0, dbgBarrier = 0, dbgRelaxCyc = 0, dbgFlushCyc = 0;

  for (int64_t group = team; group < args.nGroups; group += args.nTeams) {
    const int64_t slotIdx = group * 32 + lane;
    int64_t r = -1;
    if (args.order)
      r = args.order[slotIdx];
    else if (args.readBase + slotIdx < args.nReads)
      r = args.readBase + slotIdx;
    const int32_t L = r >= 0 ? args.readLen[r] : -1;
    const uint8_t* seq = r >= 0 ? args.packed + args.byteOff[r] : nullptr;
    int32_t Lmax = L;
    for (int sh = 16; sh > 0; sh >>= 1) Lmax = max(Lmax, __shfl_xor_sync(0xFFFFFFFFu, Lmax, sh));
    uint8_t* const predG = args.pred + (size_t)group * (size_t)(args.maxLen + 1) * N * K2 * 32;
    uint8_t* const predWideG = kWide ? args.predWide + (size_t)group * (size_t)(args.maxLen + 1) * tb.nWide * 64 + lane : nullptr;
    unsigned long long win = 0;
    uint32_t xNext = 0;

    for (int32_t pos = 0; pos <= Lmax; ++pos) {
      const bool act = pos <= L;
      if (pos < L) {  // observed base pos: the next column's emission
        if ((pos & 31) == 0) win = *reinterpret_cast<const unsigned long long*>(seq + (size_t)(pos >> 5) * 8);
        xNext = (uint32_t)(win >> (2 * (pos & 31))) & 3u;
      }
      const uint32_t par = col & 1u;  // columns are numbered across groups: the parity alternates without a break
      ++col;
      unsigned long long stamp = 0;
      if (kDebug) stamp = clock64();
      double2* const sdPubCol = sdPubT + (size_t)par * Np * 32;
      double2* const sdPubNext = sdPubT + (size_t)(par ^ 1u) * Np * 32;
      uint32_t* const passiveCol = passiveT + par;

      // ---- (1) the column starts from the emission step's result (fused into the previous column's
      //          record pass): S = S0, D = -inf (src/viterbi.cpp:66,75-79,92-106) ----
#pragma unroll 4
      for (uint32_t sl = 0; sl < nSlots; ++sl) {
        const uint32_t d = sl * W + warp;
        if (d < M) {
          double s0;
          if (pos == 0) {
            const uint4 h = hdrS[d];
            s0 = (!bhPad(h) && (tb.local || (rank == tb.startRank && d == tb.startLocal))) ? 0.0 : NEG;
            if (kTeam && bhRemoteOut(h)) stPub2(sdPubCol + (size_t)(rank * M + d) * 32 + lane, s0, NEG);
          } else
            s0 = ldCarried(privT + (size_t)(rank * M + d) * privKinds * 32, polLast);
          stsRow(aSD + d * 512u + lane16, s0, NEG);
        }
      }
      if (tid < 8) ctl[tid] = 0;
      if (tid == 0) {
        ctl[kCtlPending] = 0u;  // asynchronous closure: number of warps that found nothing to do
        ctl[kCtlPhase] = 0u;
      }
      if (kDebug) {
        const unsigned long long t = clock64();
        dbgInit += t - stamp;
        stamp = t;
      }
      teamBarrier();
      if (kTeam && rank == 0 && tid == 0) stRelaxed32(passiveT + (par ^ 1u), 0u);  // the other parity's count is dead: reset it for the next column
      if (kDebug) {
        const unsigned long long t = clock64();
        dbgBarrier += t - stamp;
        stamp = t;
      }

      // ---- (2) closure (src/viterbi.cpp:97-99,110-159), owner-computes edge relaxation ----
      const bool asyncClosure = args.asyncClosure != 0;
      uint32_t* const idleS = const_cast<uint32_t*>(reinterpret_cast<volatile uint32_t*>(ctl) + kCtlPending);
      uint32_t* const lockS = const_cast<uint32_t*>(reinterpret_cast<volatile uint32_t*>(ctl) + kCtlLock);
      uint32_t remotePending = 0;  // slots of this warp that grew and have successors in other CTAs
      // relaxes the flagged in-transitions of state d (all of them when `allIn` or when there are few); when a lane
      // grew: stores the row, publishes it if some successor lives in another CTA, flags the local successors' masks.
      auto relax = [&](uint32_t sl, uint32_t m, bool allIn) -> bool {
        const uint32_t d = sl * W + warp;
        const uint4 h = hdrS[d];
        const uint2 h2 = hdr2S[d];
        uint32_t nLE = h2.y & 0xFFu, nLN = (h2.y >> 8) & 0xFFu, nRE = (h2.y >> 16) & 0xFFu, nRN = h2.y >> 24;
        if (kWide && bhWide(h)) {
          const uint4 wc = wideCounts(h);
          nLE = wc.y & 0xFFFFu;
          nLN = wc.y >> 16;
          nRE = wc.z & 0xFFFFu;
          nRN = wc.z >> 16;
        }
        const uint32_t eLN = nLE + nLN, eRE = eLN + nRE, nIn = eRE + nRN;
        const uint2* const rel = relS + h2.x;
        const uint32_t aOwn = aSD + d * 512u + lane16;
        const double2 own = ldsRow(aOwn);
        double s = own.x, dd = own.y;
        const char* const scoreBase = reinterpret_cast<const char*>(tb.symScore);
        auto scoreOf = [&](const uint2& e) { return *reinterpret_cast<const double*>(scoreBase + e.y); };
        auto emitFrom = [&](const double2 v, const uint2& e) {
          dd = dmax(dd, dmax(v.y + tb.delExtend, v.x + tb.delOpen) + scoreOf(e));  // :124-125
          if (kDebug) ++dbgEdges;
        };
        auto nullFrom = [&](const double2 v, const uint2& e) {
          const double sc = scoreOf(e);
          dd = dmax(dd, v.y + sc);  // :140
          s = dmax(s, v.x + sc);    // :147 (:98-99)
          if (kDebug) ++dbgEdges;
        };
        auto one = [&](uint32_t j) {
          const uint2 e = rel[j];
          if (j < eLN) {
            const double2 v = ldsRow(e.x + lane16);
            if (j < nLE)
              emitFrom(v, e);
            else
              nullFrom(v, e);
          } else if (kTeam) {
            const double2 v = ldPub2(sdPubCol + (size_t)e.x * 32 + lane);
            if (j < eRE)
              emitFrom(v, e);
            else
              nullFrom(v, e);
          }
        };
        if (allIn || nIn <= 4u) {  // few transitions: relaxing all of them is cheaper than walking the mask
          // (rolled on purpose: a state has 1-3 in-transitions; the compiler's 8-way unrolling with its remainder
          // scaffolding costs more instructions than the loops execute)
          uint32_t j = 0;
#pragma unroll 1
          for (; j < nLE; ++j) {
            const uint2 e = rel[j];
            emitFrom(ldsRow(e.x + lane16), e);
          }
#pragma unroll 1
          for (; j < eLN; ++j) {
            const uint2 e = rel[j];
            nullFrom(ldsRow(e.x + lane16), e);
          }
          if (kTeam) {
#pragma unroll 1
            for (; j < eRE; ++j) {
              const uint2 e = rel[j];
              emitFrom(ldPub2(sdPubCol + (size_t)e.x * 32 + lane), e);
            }
#pragma unroll 1
            for (; j < nIn; ++j) {
              const uint2 e = rel[j];
              nullFrom(ldPub2(sdPubCol + (size_t)e.x * 32 + lane), e);
            }
          }
        } else {
          while (m) {
            const uint32_t j = (uint32_t)__ffs((int)m) - 1u;
            m &= m - 1u;
            if (j == 31u)
              for (uint32_t jj = 31; jj < nIn; ++jj) one(jj);
            else
              one(j);
          }
        }
        s = dmax(s, dd + tb.delEnd);  // :119-121
        const bool grew = act && ((s > own.x) || (dd > own.y));
        if (!__any_sync(0xFFFFFFFFu, grew)) return false;
        stsRow(aOwn, s, dd);
        if (kTeam && bhRemoteOut(h)) {
          stPub2(sdPubCol + (size_t)(rank * M + d) * 32 + lane, s, dd);
          remotePending |= 1u << sl;
        }
        const uint32_t nLoc = nOutLocalOf(h), outOff = bhOutOff(h);
        uint32_t* const flagTo = asyncClosure ? maskCur : maskNext;
#pragma unroll 1
        for (uint32_t o = lane; o < nLoc; o += 32) {
          const uint32_t w = outS[outOff + o];
          atomicOr(flagTo + boLocal(w), 1u << boBit(w));
        }
        return true;
      };
      // after a level: one release fence per warp orders the rows it published before the notifications it sends
      // now; a notification that finds its target passive takes it out of the passive count on its behalf
      auto flushRemote = [&]() {
        if (!kTeam || !remotePending) return;
        // count the notifications of this flush out of the passive count first, then ONE release fence per warp orders that
        // and the published rows before the notifications themselves (fire-and-forget adds on the targets' counters)
        uint32_t nNotes = 0;
        for (uint32_t rp = remotePending; rp; rp &= rp - 1u) {
          const uint4 h = hdrS[((uint32_t)__ffs((int)rp) - 1u) * W + warp];
          nNotes += nOutOf(h) - nOutLocalOf(h);
        }
        const bool eager = args.eagerNotify != 0;
        if (lane == 0) redAdd32(passiveCol, 0u - (eager ? 2u * nNotes : nNotes));
        if (eager) {
          // Eager notification (option, off): sent at once, WITHOUT waiting for the fence.  The rows were stored a few
          // hundred cycles ago and usually are visible when the target reads them; if not, the target relaxes against the
          // old rows, finds nothing, and the second notification below -- after the fence -- wakes it again.  Both count.
          __syncwarp();
          for (uint32_t rp = remotePending; rp; rp &= rp - 1u) {
            const uint4 h = hdrS[((uint32_t)__ffs((int)rp) - 1u) * W + warp];
            const uint32_t first = bhOutOff(h) + nOutLocalOf(h), last = bhOutOff(h) + nOutOf(h);
            for (uint32_t o = first + lane; o < last; o += 32) redAdd32(notifyT + outS[o], 1u);
          }
        }
        fenceRelease();
        __syncwarp();
        while (remotePending) {
          const uint32_t sl = (uint32_t)__ffs((int)remotePending) - 1u;
          remotePending &= remotePending - 1u;
          const uint4 h = hdrS[sl * W + warp];
          const uint32_t first = bhOutOff(h) + nOutLocalOf(h), last = bhOutOff(h) + nOutOf(h);
          for (uint32_t o = first + lane; o < last; o += 32) redAdd32(notifyT + outS[o], 1u);  // (owner CTA, class) of the successors
        }
      };

      if (asyncClosure) {
        // Asynchronous closure: no level barrier.  Every warp keeps relaxing whichever of its own states are flagged
        // (one mask array; the owner clears the bits it has read, flags are fire-and-forget ORs).  A warp that finds
        // nothing counts itself idle (ctl[kCtlPending]) and backs off; it leaves the count BEFORE it clears a mask, and
        // only after its notifications are out does it return to it.  The CTA is quiet exactly when all W warps are idle
        // and every mask is zero: flags are only set by warps that are not idle, so once that holds nothing can change it.
        const uint32_t iMine = lane * W + warp;
        const bool mineValid = lane < nSlots && iMine < M;
        bool idle = false;
        // first relaxation of every state: all transitions (flags that arrived earlier are covered: cleared first)
        for (uint32_t sl = 0; sl < nSlots; ++sl) {
          const uint32_t d = sl * W + warp;
          if (d >= M) break;
          if (lane == 0) maskCur[d] = 0u;  // (a flag set after this store is kept; one set before it is served by this relaxation)
          __syncwarp();
          unsigned long long tr = 0;
          if (kDebug) tr = clock64();
          relax(sl, 0, true);
          if (kDebug) dbgRelaxCyc += clock64() - tr;
        }
        {
          unsigned long long tr = 0;
          if (kDebug) tr = clock64();
          flushRemote();
          if (kDebug) dbgFlushCyc += clock64() - tr;
        }
        for (;;) {
          uint32_t mym = 0;
          if (mineValid) mym = reinterpret_cast<volatile uint32_t*>(maskCur)[iMine];
          uint32_t work = __ballot_sync(0xFFFFFFFFu, mym != 0);
          if (work) {
            if (idle) {
              if (lane == 0) atomicSub(idleS, 1u);
              idle = false;
              __syncwarp();
            }
            if (mym) atomicAnd(maskCur + iMine, ~mym);  // the bits read; later ones stay for the next round
            while (work) {
              const uint32_t sl = (uint32_t)__ffs((int)work) - 1u;
              work &= work - 1u;
              const uint32_t m = __shfl_sync(0xFFFFFFFFu, mym, sl);
              if (kDebug) ++dbgVisits;
              unsigned long long tr = 0;
              if (kDebug) tr = clock64();
              relax(sl, m, false);
              if (kDebug) dbgRelaxCyc += clock64() - tr;
            }
            {
              unsigned long long tr = 0;
              if (kDebug) tr = clock64();
              flushRemote();
              if (kDebug) dbgFlushCyc += clock64() - tr;
            }
            continue;
          }
          if (!idle) {
            if (lane == 0) atomicAdd(idleS, 1u);
            idle = true;
          }
          if (ctl[kCtlPhase] != 0u) break;
          // ONE idle warp at a time looks after the CTA -- notifications from other CTAs, the quiet check, the team's
          // termination -- whichever gets the lock: a notification does not wait for a particular warp to run out of work
          uint32_t mine = 0;
          if (lane == 0) mine = ctl[kCtlLock] == 0u && atomicCAS(lockS, 0u, 1u) == 0u;  // (peek first: 31 warps may be idle)
          if (!__shfl_sync(0xFFFFFFFFu, mine, 0)) {
            if (args.idleNs) __nanosleep(args.idleNs);
            continue;
          }
          auto unlock = [&]() {
            __syncwarp();
            if (lane == 0) {
              __threadfence_block();
              atomicExch(lockS, 0u);
            }
          };
          if (ctl[kCtlPhase] != 0u) {  // the column ended between the test above and the lock
            unlock();
            break;
          }
          // is the CTA quiet?  (all warps idle, then every mask zero, then still all idle)
          bool quiet = false;
          if (ctl[kCtlPending] == W) {
            bool any = false;
            for (uint32_t i = lane; i < M; i += 32) any |= reinterpret_cast<volatile uint32_t*>(maskCur)[i] != 0u;
            quiet = !__any_sync(0xFFFFFFFFu, any) && ctl[kCtlPending] == W;
          }
          uint32_t action = 0;  // 1: a neighbour CTA published new rows, 2: the column's closure is complete
          uint32_t delta = 0;   // lane q: new notifications of class q
          if (!kTeam) {
            if (quiet) action = 2;
          } else {
            uint32_t seen = ctl[kCtlSeen + lane];  // notifications of class `lane` consumed so far (kept by the lock holder)
            // lane q reads the counter of class q (one line for the warp); returns the warp's total of new notifications
            auto pollClasses = [&]() -> uint32_t {
              const uint32_t c = ldVolatileGlobal32(notifyT + rank * kNotifyClasses + lane);
              delta = c - seen;
              seen = c;
              return __any_sync(0xFFFFFFFFu, delta != 0u) ? __reduce_add_sync(0xFFFFFFFFu, delta) : 0u;
            };
            uint32_t tot = pollClasses();
            if (tot) {  // new rows published by neighbours: consumed (this CTA is not counted passive now)
              if (lane == 0) redAdd32(passiveCol, tot);
              action = 1;
            } else if (quiet) {
              unsigned long long t0 = 0;
              if (kDebug) t0 = clock64();
              if (lane == 0) redAdd32(passiveCol, 1u);  // passive
              for (;;) {
                tot = pollClasses();
                if (tot) {
                  if (lane == 0) redAdd32(passiveCol, tot - 1u);  // active again, and these notifications are consumed
                  action = 1;
                  break;
                }
                uint32_t p = lane == 0 ? ldVolatileGlobal32(passiveCol) : 0u;
                p = __shfl_sync(0xFFFFFFFFu, p, 0);
                if (p == T) {
                  action = 2;
                  break;
                }
              }
              if (kDebug) dbgPassive += clock64() - t0;
            }
            ctl[kCtlSeen + lane] = seen;
          }
          if (action == 2) {
            if (lane == 0) ctl[kCtlPhase] = 1u;
            unlock();
          } else if (action == 1) {
            if (kDebug) ++dbgWakes;
            // the states of the notified classes relax their transitions from other CTAs again; the flagging warp is not
            // idle meanwhile
            if (lane == 0) atomicSub(idleS, 1u);
            idle = false;
            __syncwarp();
            for (uint32_t notified = __ballot_sync(0xFFFFFFFFu, delta != 0u); notified; notified &= notified - 1u) {
              const uint32_t c = (uint32_t)__ffs((int)notified) - 1u;
              for (uint32_t q = clsOffS[c] + lane; q < clsOffS[c + 1]; q += 32) {
                const uint32_t i = clsStS[q];
                atomicOr(maskCur + i, remInS[i]);
              }
            }
            unlock();
          } else {
            unlock();
            if (args.idleNs) __nanosleep(args.idleNs / 2);
          }
        }
        __syncthreads();
      } else
      {
        // (level-synchronous variant, async_closure = 0: thread 0 keeps the TOTAL over the classes in notifySeen and a
        // wake-up flags every transition that crosses CTAs)
        auto notifyTotal = [&]() -> uint32_t {
          uint32_t t = 0;
          for (uint32_t q = 0; q < kNotifyClasses; ++q) t += ldVolatileGlobal32(notifyT + rank * kNotifyClasses + q);
          return t;
        };
        uint32_t lvl = 0;
        bool activated = false;
        // level 0: every transition of every state
        for (uint32_t sl = 0; sl < nSlots; ++sl)
          if (sl * W + warp < M) activated |= relax(sl, 0, true);
        flushRemote();
        for (;;) {
          // four flags in rotation: a slow thread may still be reading the ones of this level while the next are set
          if (activated && lane == 0) ctl[kCtlFlag + ((lvl + 1) & 3u)] = 1u;
          if (tid == 0) {
            ctl[kCtlFlag + ((lvl + 2) & 3u)] = 0u;
            ctl[kCtlWake + ((lvl + 2) & 3u)] = 0u;
          }
          __syncthreads();
          {
            uint32_t* t = maskCur;
            maskCur = maskNext;
            maskNext = t;
          }
          ++lvl;
          const bool haveLocal = ctl[kCtlFlag + (lvl & 3u)] != 0;
          bool wake = kTeam && ctl[kCtlWake + (lvl & 3u)] != 0;
          if (!haveLocal && !wake) {
            if (!kTeam) break;
            // Nothing to do: become passive.  The column's closure is complete when all T CTAs of the team are passive
            // (a CTA that notifies a passive one takes it out of the count before the target knows).
            if (tid == 0) {
              unsigned long long t0 = 0;
              if (kDebug) t0 = clock64();
              uint32_t decision;
              redAdd32(passiveCol, 1u);  // passive
              for (;;) {
                const uint32_t c = notifyTotal();
                if (c != notifySeen) {
                  redAdd32(passiveCol, c - notifySeen - 1u);  // active again, and these notifications are consumed
                  notifySeen = c;
                  decision = 1;
                  break;
                }
                if (ldVolatileGlobal32(passiveCol) == T) {
                  decision = 2;
                  break;
                }
              }
              ctl[kCtlDecision] = decision;
              if (kDebug) dbgPassive += clock64() - t0;
            }
            __syncthreads();
            if (ctl[kCtlDecision] == 2u) break;
            wake = true;
          }
          if (kDebug && haveLocal) ++dbgLevels;
          if (kDebug && wake) ++dbgWakes;
          activated = false;
          uint32_t st = 0;
          if (kTeam && tid == 0) st = notifyTotal();  // consumed after this level's work
          const uint32_t iMine = lane * W + warp;
          uint32_t mym = 0;
          if (lane < nSlots && iMine < M) {
            if (haveLocal) {
              mym = maskCur[iMine];
              if (mym) maskCur[iMine] = 0;
            }
            if (wake) mym |= remInS[iMine];  // a neighbour CTA published new rows
          }
          uint32_t work = __ballot_sync(0xFFFFFFFFu, mym != 0);
          while (work) {
            const uint32_t sl = (uint32_t)__ffs((int)work) - 1u;
            work &= work - 1u;
            const uint32_t m = __shfl_sync(0xFFFFFFFFu, mym, sl);
            if (kDebug) ++dbgVisits;
            activated |= relax(sl, m, false);
          }
          flushRemote();
          if (kTeam && tid == 0 && st != notifySeen) {
            redAdd32(passiveCol, st - notifySeen);  // consumed: the rows are read at the next level
            notifySeen = st;
            ctl[kCtlWake + ((lvl + 1) & 3u)] = 1u;
          }
        }
      }
      if (kDebug) {
        const unsigned long long t = clock64();
        dbgClosure += t - stamp;
        stamp = t;
      }

      // ---- (3) predecessor records with the traceback's arithmetic (src/viterbi.cpp:251-286), (4) duplication
      //      opens (:161-168), (5) emission step of column pos+1 (:92-106) and the emit candidates of its S record ----
      {
        double bv = NEG;  // local mode: first maximum of S(.,L) in reference state order
        uint32_t bo = 0xFFFFFFFFu;
        double pfB = NEG, pfT[KMAX];
        auto fetch = [&](uint32_t sl) {
          const uint32_t d = sl * W + warp;
          if (d < M && pos > 0) {
            const double* row = privT + (size_t)(rank * M + d) * privKinds * 32;
            pfB = ldCarried(row + 32, polLast);
#pragma unroll
            for (uint32_t t = 0; t < (uint32_t)KMAX; ++t)
              if (t < k) pfT[t] = ldCarried(row + 64 + 32 * t, polLast);
          }
        };
#pragma unroll
        for (uint32_t t = 0; t < (uint32_t)KMAX; ++t) pfT[t] = NEG;
        fetch(0);
        for (uint32_t sl = 0; sl < nSlots; ++sl) {
          const uint32_t d = sl * W + warp;
          if (d >= M) break;
          const double curB = pfB;
          double curT[KMAX];
#pragma unroll
          for (uint32_t t = 0; t < (uint32_t)KMAX; ++t) curT[t] = pfT[t];
          if (sl + 1 < nSlots) fetch(sl + 1);
          const uint4 h = hdrS[d];
          if (bhPad(h)) continue;
          const bool wide = kWide && bhWide(h);
          uint32_t nE = bhNEmit(h), nIn = nE + bhNNull(h);
          if (wide) {
            const uint32_t c = wideCounts(h).x;
            nE = c & 0xFFFFu;
            nIn = nE + (c >> 16);
          }
          const uint32_t inOff = bhInOff(h), mdl = bhMdl(h), orig = h.w;
          constexpr uint32_t keep = kWide ? kKeepRecordWide : kKeepRecord;
          const uint32_t none = wide ? kWideNoPred : kNoPred;
          double* const row = privT + (size_t)(rank * M + d) * privKinds * 32;
          const double2 own = ldsRow(aSD + d * 512u + lane16);
          const double sH = own.x, dH = own.y;
          // S record: the emit candidates (:255) were evaluated by the previous column's pass
          double best = pos > 0 ? curB : NEG, bestD = NEG, s0n = NEG, bEn = NEG;
          uint32_t idx = pos > 0 ? keep : none, idxD = none, idxEn = none;
          uint32_t j = 0;
#pragma unroll 1
          for (; j < nE; ++j) {
            const uint2 e = inS[inOff + j];
            const uint32_t sym = beSym(e);
            const double2 v = (kTeam && beRemote(e)) ? ldPub2(sdPubCol + (size_t)e.x * 32 + lane) : ldsRow(e.x + lane16);
            double c = v.y + tb.tsDext[sym];  // :272
            if (c > bestD) {
              bestD = c;
              idxD = 2 * j;
            }
            c = v.x + tb.tsDopen[sym];  // :273
            if (c > bestD) {
              bestD = c;
              idxD = 2 * j + 1;
            }
            const uint32_t b4 = beBase(e) * 4 + xNext;
            s0n = dmax(s0n, ((v.x + tb.symScore[sym]) + tb.noGap) + subS[b4]);  // :94-95 of pos+1
            c = v.x + tsE[sym * 16 + b4];                                       // :255 of pos+1
            if (c > bEn) {
              bEn = c;
              idxEn = j;
            }
          }
#pragma unroll 1
          for (; j < nIn; ++j) {
            const uint2 e = inS[inOff + j];
            const double2 v = (kTeam && beRemote(e)) ? ldPub2(sdPubCol + (size_t)e.x * 32 + lane) : ldsRow(e.x + lane16);
            const double sc = tb.symScore[beSym(e)];
            double c = v.x + sc;  // :257
            if (c > best) {
              best = c;
              idx = j;
            }
            c = v.y + sc;  // :276
            if (c > bestD) {
              bestD = c;
              idxD = nE + j;
            }
          }
          {
            const double c = dH + tb.delEnd;  // :258
            if (c > best) {
              best = c;
              idx = nIn;
            }
          }
          if (mdl > 0 && pos > 0) {
            const double parked = curT[0];  // T(state,pos-1,0)+sub, :261 (slot 0 holds the T -> S candidate)
            if (parked > best) {
              best = parked;
              idx = nIn + 1;
            }
          }
          if (tb.local && pos == 0) {  // :263-264
            const double2 v0 = (kTeam && tb.startRank != rank)
                                   ? ldPub2(sdPubCol + (size_t)(tb.startRank * M + tb.startLocal) * 32 + lane)
                                   : ldsRow(aSD + tb.startLocal * 512u + lane16);
            if (v0.x + 0.0 > best) {
              best = v0.x + 0.0;
              idx = nIn + 2;
            }
          }
          uint8_t* const pr = predG + ((size_t)pos * N + orig) * K2 * 32 + lane;
          uint8_t* const prW = wide ? predWideG + ((size_t)pos * tb.nWide + bhWideNo(h)) * 64 : nullptr;  // the high bytes
          if (act) {
            if (idx != keep) stRecord(pr, idx);
            stRecord(pr + 32, idxD);
            if (wide) {
              if (idx != keep) stRecord(prW, idx >> 8);
              stRecord(prW + 32, idxD >> 8);
            }
          }
          // duplication cells (:161-168) and their records (:281-286).  Parked layout between columns: slot 0 holds
          // T(pos,0)+sub (the T -> S candidate of the next column), slot t >= 1 holds T(pos,t)+sub (the shift into t-1).
          double tNow[KMAX];
#pragma unroll
          for (uint32_t t = 0; t < (uint32_t)KMAX; ++t) {
            tNow[t] = NEG;
            if (t < k) {
              uint32_t idxT = kNoPred;
              if (pos > 0 && t < mdl) {
                double shifted = NEG;
                if (t + 1 < (uint32_t)KMAX && t + 1 < mdl) shifted = curT[t + 1 < (uint32_t)KMAX ? t + 1 : 0];  // T(state,pos-1,t+1)+sub, :285
                if (shifted > NEG) idxT = 0;
                if (sH + tb.tsT[t] > shifted) idxT = 1;                  // :286
                tNow[t] = dmax(shifted, (sH + tb.tanDup) + tb.len[t]);   // :166-167
              }
              if (act) stRecord(pr + (2 + t) * 32, idxT);
            }
          }
          if (kDebug && args.cells && group == 0 && lane == 0 && act) {
            double* cell = args.cells + ((size_t)pos * N + orig) * K2;
            cell[0] = sH;
            cell[1] = dH;
#pragma unroll
            for (uint32_t t = 0; t < (uint32_t)KMAX; ++t)
              if (t < k) cell[2 + t] = tNow[t];
          }
          // column pos+1: T -> S candidate and the T shift (:102-106), parked for the next column
          if (mdl > 0) {
#pragma unroll
            for (uint32_t t = 0; t < (uint32_t)KMAX; ++t)
              if (t < mdl) {
                const double v = tNow[t] + subS[bhCtx(h, t) * 4 + xNext];
                if (t == 0) s0n = dmax(s0n, v);
                stCarried(row + 64 + 32 * t, v, polLast);
              }
          }
          stCarried(row, s0n, polLast);
          stCarried(row + 32, bEn, polLast);
          if (pos < L) {  // the emit part of S(state,pos+1)'s record
            stRecordEarly(pr + (size_t)N * K2 * 32, idxEn);
            if (wide) stRecordEarly(prW + (size_t)tb.nWide * 64, idxEn >> 8);
          }
          if (kTeam && bhRemoteOut(h)) stPub2(sdPubNext + (size_t)(rank * M + d) * 32 + lane, s0n, NEG);
          if (!tb.local) {
            if (rank == tb.endRank && d == tb.endLocal && pos == L && r >= 0) args.loglike[r] = sH;  // viterbi.h:102
          } else if (sH > bv || (sH == bv && orig < bo)) {
            bv = sH;
            bo = orig;
          }
        }
        if (tb.local && pos == L) {  // :171-173, :240-242: this warp's share; the traceback kernel reduces over warps and CTAs
          args.partVal[((size_t)group * T * W + rank * W + warp) * 32 + lane] = bv;
          args.partOrig[((size_t)group * T * W + rank * W + warp) * 32 + lane] = bo;
        }
      }
      __syncthreads();  // rows of this column are dead: the next column's S0 may overwrite them
      if (kDebug) dbgRecord += clock64() - stamp;
    }
  }
  if (kDebug && args.dbg && lane == 0 && rank == 0) {
    // levels and cycles are CTA-uniform: counted by warp 0 of rank 0 of every team; visits and edges by every warp of it
    if (warp == 0) atomicAdd(&args.dbg[1], dbgLevels);
    atomicAdd(&args.dbg[2], dbgVisits);
    atomicAdd(&args.dbg[3], dbgEdges);
    if (warp == 0) atomicAdd(&args.dbg[4], dbgClosure);
    if (warp == 0) atomicAdd(&args.dbg[5], dbgRecord);
    atomicAdd(&args.dbg[6], dbgWakes);    // (asynchronous closure: whichever warp held the CTA's lock)
    atomicAdd(&args.dbg[7], dbgPassive);
    if (warp == 0) atomicAdd(&args.dbg[8], dbgInit);
    if (warp == 0) atomicAdd(&args.dbg[9], dbgBarrier);
    atomicAdd(&args.dbg[10], dbgRelaxCyc);
    atomicAdd(&args.dbg[11], dbgFlushCyc);
  }
}

// ---------------------------------------------------------------------------
// traceback over batch-layout records: one thread per read follows the predecessor records
// (reference src/viterbi.cpp:195-304: loop :247, emitted symbols :299-300), decoding each byte against the
// state's transition lists in REFERENCE order (the records are indexed by reference state)
// ---------------------------------------------------------------------------
__global__ void viterbiTracebackBatchKernel(const BatchTraceTables tb, const BatchTraceArgs args) {
  const int64_t slot = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= args.nSlots) return;
  int64_t read = -1;
  if (args.order)
    read = args.order[slot];
  else if (args.readBase + slot < args.nReads)
    read = args.readBase + slot;
  if (read < 0) return;
  const int64_t group = slot >> 5;
  const uint32_t lane = (uint32_t)(slot & 31);
  const uint32_t N = tb.nStates, k = tb.k, K2 = k + 2;
  const int32_t L = args.readLen[read];
  const double NEG = negInf();

  uint32_t state;
  double ll;
  if (!tb.local) {
    state = N - 1;
    ll = args.loglike[read];
  } else {
    double bv = NEG;
    uint32_t bo = 0xFFFFFFFFu;
    for (uint32_t r = 0; r < tb.T; ++r) {
      const double v = args.partVal[((size_t)group * tb.T + r) * 32 + lane];
      const uint32_t o = args.partOrig[((size_t)group * tb.T + r) * 32 + lane];
      if (o == 0xFFFFFFFFu) continue;
      if (v > bv || (v == bv && o < bo)) {
        bv = v;
        bo = o;
      }
    }
    state = bo == 0xFFFFFFFFu ? 0u : bo;
    ll = bv;
    args.loglike[read] = ll;
  }

  char* out = args.decoded + (size_t)read * args.decodedStride;
  int32_t* path = args.path ? args.path + (size_t)read * 3 * args.pathStride : nullptr;
  int32_t nOut = 0, nPath = 0;
  int32_t status = DNAB_READ_OK_;
  if (!(ll > NEG)) {
    args.decodedLen[read] = 0;
    args.status[read] = DNAB_READ_NO_DECODING_;
    if (args.pathLen) args.pathLen[read] = 0;
    return;
  }
  const uint8_t* predG = args.pred + (size_t)group * (size_t)(args.maxLen + 1) * N * K2 * 32 + lane;
  const uint8_t* predWideG = args.predWide + (size_t)group * (size_t)(args.maxLen + 1) * tb.nWide * 64 + lane;
  int32_t pos = L;
  uint32_t mut = 0;
  const int32_t cap = args.decodedStride;
  while (pos >= 0 && state != 0) {
    if (path) {
      if (nPath < args.pathStride) {
        path[3 * nPath] = (int32_t)state;
        path[3 * nPath + 1] = pos;
        path[3 * nPath + 2] = (int32_t)mut;
      } else
        status = DNAB_READ_OVERFLOW_;
    }
    ++nPath;
    uint32_t p = predG[(((size_t)pos * N + state) * K2 + mut) * 32];
    uint32_t none = kNoPred;
    if (tb.wideOf && mut < 2) {  // a wide state's S and D records: the high byte is in the side plane
      const uint32_t wn = tb.wideOf[state];
      if (wn != 0xFFFFFFFFu) {
        p |= (uint32_t)predWideG[(((size_t)pos * tb.nWide + wn) * 2 + mut) * 32] << 8;
        none = kWideNoPred;
      }
    }
    if (p == none) {
      status = DNAB_READ_TRACEBACK_FAILED_;
      break;
    }
    const uint32_t e0 = tb.emitOff[state], nE = tb.emitOff[state + 1] - e0;
    const uint32_t n0 = tb.nullOff[state], nIn = nE + (tb.nullOff[state + 1] - n0);
    uint32_t sym = 0;
    if (mut == 0) {
      if (p < nE) {
        sym = tb.emitSym[e0 + p];
        state = tb.emitSrc[e0 + p];
        --pos;
      } else if (p < nIn) {
        sym = tb.nullSym[n0 + (p - nE)];
        state = tb.nullSrc[n0 + (p - nE)];
      } else if (p == nIn) {
        mut = 1;
      } else if (p == nIn + 1) {
        mut = 2;
        --pos;
      } else {
        state = 0;  // local mode, pos == 0: jump to (0,0,S)
      }
    } else if (mut == 1) {
      if (p < 2 * nE) {
        sym = tb.emitSym[e0 + (p >> 1)];
        state = tb.emitSrc[e0 + (p >> 1)];
        mut = (p & 1) ? 0 : 1;
      } else {
        sym = tb.nullSym[n0 + (p - 2 * nE)];
        state = tb.nullSrc[n0 + (p - 2 * nE)];
      }
    } else {
      if (p == 0) {
        mut += 1;
        --pos;
      } else
        mut = 0;
    }
    if (sym) {
      if (nOut < cap)
        out[cap - 1 - nOut] = (char)tb.symChar[sym];
      else
        status = DNAB_READ_OVERFLOW_;
      ++nOut;
    }
  }
  const int32_t kept = nOut < cap ? nOut : cap;
  for (int32_t i = 0; i < kept; ++i) out[i] = out[cap - kept + i];
  args.decodedLen[read] = kept;
  args.status[read] = status;
  if (args.pathLen) args.pathLen[read] = nPath;
}

// ---------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------
typedef void (*BatchKernelPtr)(const BatchTables, const BatchArgs);
template <int W, int KMAX, bool kWide>
static BatchKernelPtr pickBatchKernelWK(bool team, bool debug) {
  if (debug) return team ? viterbiFillBatchKernel<W, KMAX, true, true, kWide> : viterbiFillBatchKernel<W, KMAX, false, true, kWide>;
  return team ? viterbiFillBatchKernel<W, KMAX, true, false, kWide> : viterbiFillBatchKernel<W, KMAX, false, false, kWide>;
}
static uint32_t batchWarps(uint32_t warps) { return warps > 24 ? 32u : warps > 16 ? 24u : 16u; }
template <bool kWide>
static BatchKernelPtr pickBatchKernelW(const BatchTables& tb, uint32_t warps, bool debug) {
  const bool team = tb.T > 1;
  const uint32_t w = batchWarps(warps);
  if (w == 32) return tb.k <= 2 ? pickBatchKernelWK<32, 2, kWide>(team, debug) : pickBatchKernelWK<32, kMaxK, kWide>(team, debug);
  if (w == 24) return tb.k <= 2 ? pickBatchKernelWK<24, 2, kWide>(team, debug) : pickBatchKernelWK<24, kMaxK, kWide>(team, debug);
  return tb.k <= 2 ? pickBatchKernelWK<16, 2, kWide>(team, debug) : pickBatchKernelWK<16, kMaxK, kWide>(team, debug);
}
static BatchKernelPtr pickBatchKernel(const BatchTables& tb, uint32_t warps, bool debug) {
  return tb.nWide ? pickBatchKernelW<true>(tb, warps, debug) : pickBatchKernelW<false>(tb, warps, debug);
}

cudaError_t queryBatchTeams(const BatchTables& tb, uint32_t warps, uint32_t smemBytes, int* ctasPerSm) {
  BatchKernelPtr kern = pickBatchKernel(tb, warps, false);
  cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemBytes);
  if (err != cudaSuccess) return err;
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctasPerSm, kern, (int)(batchWarps(warps) * 32), smemBytes);
}

cudaError_t launchFillBatch(const BatchTables& tb, const BatchArgs& args, uint32_t warps, uint32_t smemBytes,
                            cudaStream_t stream, size_t persistBytes) {
  const bool debug = args.dbg != nullptr || args.cells != nullptr;
  BatchKernelPtr kern = pickBatchKernel(tb, warps, debug);
  cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemBytes);
  if (err != cudaSuccess) return err;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(args.nTeams * tb.T);
  cfg.blockDim = dim3(batchWarps(warps) * 32);
  cfg.dynamicSmemBytes = smemBytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  unsigned nAttr = 0;
  if (tb.T > 1) {
    attr[nAttr].id = cudaLaunchAttributeCooperative;  // the CTAs of a team meet at barriers in L2: all must be resident
    attr[nAttr].val.cooperative = 1;
    ++nAttr;
  }
  if (persistBytes) {
    // the rows carried from one column to the next (rewritten in place every column) stay in the persisting part of L2
    // instead of being written back to HBM behind the record stream
    attr[nAttr].id = cudaLaunchAttributeAccessPolicyWindow;
    attr[nAttr].val.accessPolicyWindow.base_ptr = args.priv;
    attr[nAttr].val.accessPolicyWindow.num_bytes = persistBytes;
    attr[nAttr].val.accessPolicyWindow.hitRatio = 1.0f;
    attr[nAttr].val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    attr[nAttr].val.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    ++nAttr;
  }
  cfg.attrs = attr;
  cfg.numAttrs = nAttr;
  return cudaLaunchKernelEx(&cfg, kern, tb, args);
}

cudaError_t launchTracebackBatch(const BatchTraceTables& tb, const BatchTraceArgs& args, cudaStream_t stream) {
  const int threads = 64;
  const int blocks = (int)((args.nSlots + threads - 1) / threads);
  viterbiTracebackBatchKernel<<<blocks, threads, 0, stream>>>(tb, args);
  return cudaGetLastError();
}

}  // namespace dnab
