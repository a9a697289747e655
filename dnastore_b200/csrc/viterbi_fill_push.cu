// viterbiFillPushKernel: the ViterbiMatrix fill (reference src/viterbi.cpp:62-176) for a batch of
// reads, one thread-block cluster per read, with the within-column closure done PUSH style.
//
// Why push.  The project's first fill kernel (round 1, since retired) relaxed dirty states PULL style: a hop
// of a propagation chain cost two transition-table accesses (the state's incoming list, then its
// outgoing list to wake successors) that miss L1 (cluster barriers flush it), plus a bitmap /
// compaction / pending-counter protocol: ~3,000 cycles per hop measured on B200, and a column of the
// BASELINE config-2 machine has chains of 17-46 hops.  Here
//   * the closure is the reference's own phase-2 loop body (src/viterbi.cpp:118-158): a state whose S
//     or D grew pushes max(D+delExtend, S+delOpen)+score into D(dest) over emitting transitions and
//     D+score / S+score over null ones, with a compare-and-swap max on the destination cell (a failed
//     push costs one shared-memory load).  max(a,b)+c == max(a+c,b+c) in IEEE arithmetic and every
//     within-column weight is <= 0, so any schedule reaches the reference's least fixed point bit for
//     bit (SURVEY.md 8a-6); a hop needs one table access: the pusher's outgoing list;
//   * that out-table is compact (one word per transition) and RESIDENT in shared memory;
//   * the incoming lists, needed only by the two dense passes that walk the states in order (first
//     closure pass; predecessor pass, which also performs the emission step of the NEXT column from the
//     same gathered S(pos)[src]), are STREAMED through one shared-memory
//     staging buffer in chunks: every thread fetches its 16-byte pieces of the NEXT chunk into registers
//     (coalesced 128-bit loads) before it works on the current one and stores them after a CTA barrier,
//     so the L2 latency of the table is hidden behind a whole step of the pass; each thread handles
//     kU states per step with their loads interleaved (the passes are latency-, not issue-bound);
//   * the push closure is level-synchronous and breadth first (the order that keeps re-relaxation
//     low): per level the dirty bitmap is compacted into a queue, the queued states push, one CTA
//     barrier; in a cluster, peers are relaxed directly through distributed shared memory (ld /
//     atom.cas / red.or .shared::cluster) and ONE cluster barrier per level makes the flags they set
//     visible; on one-CTA machines a thin frontier (the long tail of a column) is queued by the pushers
//     themselves, which saves the scan and one of the two CTA barriers of a level.
// Everything else -- the emission step, the predecessor records evaluated with the TRACEBACK's own
// floating-point association and candidate order (src/viterbi.cpp:251-286), duplication opens, the
// record layout read by viterbiTracebackKernel (viterbi_traceback.cu) -- follows the reference directly.
#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include <cstdint>
#include <type_traits>

#include "viterbi_kernels.h"

namespace cg = cooperative_groups;

namespace dnab {
namespace {

__device__ __forceinline__ uint32_t smemAddr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ double negInf() { return __longlong_as_double(0xFFF0000000000000LL); }
// std::max(a,b) of the reference: keeps a on ties
__device__ __forceinline__ double dmax(double a, double b) { return (a < b) ? b : a; }

// constant tables / staged table chunks: plain loads
__device__ __forceinline__ double ldsTab(uint32_t a) {
  double v;
  asm("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ uint32_t lds32(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ uint32_t lds16(uint32_t a) {
  uint16_t v;
  asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(a));
  return v;
}
// DP cells: volatile, every relaxation re-reads them
__device__ __forceinline__ double ldsCell(uint32_t a) {
  double v;
  asm volatile("ld.volatile.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ void stsCell(uint32_t a, double v) {
  asm volatile("st.volatile.shared.f64 [%0], %1;" ::"r"(a), "d"(v) : "memory");
}
__device__ __forceinline__ void sts32(uint32_t a, uint32_t v) {
  asm volatile("st.volatile.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ldsVolatile32(uint32_t a) {
  uint32_t v;
  asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ void redOrShared(uint32_t a, uint32_t v) {
  asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t atomExchShared(uint32_t a, uint32_t v) {
  uint32_t old;
  asm volatile("atom.shared.exch.b32 %0, [%1], %2;" : "=r"(old) : "r"(a), "r"(v) : "memory");
  return old;
}
__device__ __forceinline__ uint32_t atomAddShared(uint32_t a, uint32_t v) {
  uint32_t old;
  asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(a), "r"(v) : "memory");
  return old;
}
__device__ __forceinline__ void sts16(uint32_t a, uint32_t v) {
  asm volatile("st.volatile.shared.u16 [%0], %1;" ::"r"(a), "h"((uint16_t)v) : "memory");
}
__device__ __forceinline__ uint32_t mapToRank(uint32_t localAddr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(localAddr), "r"(rank));
  return r;
}
__device__ __forceinline__ double ldPeer(uint32_t clusterAddr) {
  double v;
  asm volatile("ld.relaxed.cluster.shared::cluster.f64 %0, [%1];" : "=d"(v) : "r"(clusterAddr) : "memory");
  return v;
}
__device__ __forceinline__ void stPeerU32(uint32_t localAddr, uint32_t rank, uint32_t v) {
  asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(mapToRank(localAddr, rank)), "r"(v) : "memory");
}

// cell <- max(cell, v) on a cell of THIS CTA; true when the cell grew.  A failed push is one load.
__device__ __forceinline__ bool casMaxLocal(uint32_t a, double v, double old) {
  while (v > old) {
    const unsigned long long assumed = (unsigned long long)__double_as_longlong(old);
    unsigned long long prev;
    asm volatile("atom.shared.cas.b64 %0, [%1], %2, %3;"
                 : "=l"(prev)
                 : "r"(a), "l"(assumed), "l"((unsigned long long)__double_as_longlong(v))
                 : "memory");
    if (prev == assumed) return true;
    old = __longlong_as_double((long long)prev);
  }
  return false;
}
// the same on a cell of a peer CTA, through distributed shared memory
__device__ __forceinline__ bool casMaxPeer(uint32_t clusterAddr, double v, double old) {
  while (v > old) {
    const unsigned long long assumed = (unsigned long long)__double_as_longlong(old);
    unsigned long long prev;
    asm volatile("atom.relaxed.cluster.shared::cluster.cas.b64 %0, [%1], %2, %3;"
                 : "=l"(prev)
                 : "r"(clusterAddr), "l"(assumed), "l"((unsigned long long)__double_as_longlong(v))
                 : "memory");
    if (prev == assumed) return true;
    old = __longlong_as_double((long long)prev);
  }
  return false;
}

__device__ __forceinline__ void sts128(uint32_t a, uint4 v) {
  asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

struct Ctx {
  uint32_t aS, aD, aFlag, aSym, aOutOff, aOutWords;
  const uint4* gOutSlots;    // this CTA's out-slots in global memory (when the table is not in shared memory)
  const uint32_t* gOutOvf;
  uint32_t outInSmem;
  uint32_t aQueueNext;  // thin frontier: this level's pushers queue the states they raise themselves into this small queue
  uint32_t aTailNext;   // ... counted here
  uint32_t capNext;
  double delOpen, delExtend, delEnd;
};

__device__ __forceinline__ uint32_t atomOrShared(uint32_t a, uint32_t v) {
  uint32_t old;
  asm volatile("atom.shared.or.b32 %0, [%1], %2;" : "=r"(old) : "r"(a), "r"(v) : "memory");
  return old;
}
__device__ __forceinline__ void redAndShared(uint32_t a, uint32_t v) {
  asm volatile("red.shared.and.b32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}

// State l of this CTA grew and must push in the next level.  Wide frontier: its bit in the dirty bitmap is set
// and the next level starts with a scan of the bitmap.  Thin frontier (appendMode): the bit doubles as "already
// queued" and the pusher appends the state to the next level's small queue itself, which saves the scan and one
// CTA barrier per level; if that queue is full the bit simply stays set and `deferred` makes the next level scan.
template <bool kAppend>
__device__ __forceinline__ void raise(const Ctx& c, uint32_t l, bool& flagged, bool& deferred) {
  const uint32_t aWord = c.aFlag + 4 * (l >> 5), bit = 1u << (l & 31);
  if (!kAppend) {
    redOrShared(aWord, bit);  // no fence: the flag is consumed only after the next CTA barrier
    flagged = true;
    return;
  }
  if (atomOrShared(aWord, bit) & bit) return;  // queued already (or pending from a peer: the next scan takes it)
  const uint32_t idx = atomAddShared(c.aTailNext, 1u);
  if (idx < c.capNext)
    sts16(c.aQueueNext + 2 * idx, l);
  else
    deferred = true;
}

constexpr uint32_t kNoState = 0xFFFFFFFFu;

// One state's push (reference src/viterbi.cpp:118-158): ssrc = max(S, D+delEnd); over emitting
// transitions max(D+delExtend, ssrc+delOpen)+score -> D(dest); over null ones D+score -> D(dest) and
// ssrc+score -> S(dest).  A destination that grew must push in turn: the first such destination in
// this CTA is RETURNED (the caller flags it or follows it), the others are flagged in the dirty
// bitmap (this CTA's or a peer's) and `flagged` is set.
// Loads that do not depend on each other are issued together: the chain is cells+offsets -> edge word
// -> destination cells -> add/compare -> compare-and-swap (only when the destination grows).
template <bool kCluster, bool kAppend>
__device__ __forceinline__ uint32_t pushState(const Ctx& c, uint32_t s, uint4 slot, bool& flagged, bool& deferred, bool& sent) {
  const uint32_t myS = c.aS + 8 * s, myD = c.aD + 8 * s;
  uint32_t o0, o1;  // shared-memory table: edge range; L2 slots: 0 .. nOut
  if (c.outInSmem) {
    o0 = lds16(c.aOutOff + 2 * s);
    o1 = lds16(c.aOutOff + 2 * s + 2);
  } else {
    o0 = 0;
    o1 = slot.x;
  }
  const double dv = ldsCell(myD);
  double sv = ldsCell(myS);
  {  // ssrc = max(S, D + delEnd) (src/viterbi.cpp:121-122)
    const double viaD = dv + c.delEnd;
    if (viaD > sv) {
      casMaxLocal(myS, viaD, sv);
      sv = viaD;
    }
  }
  const double m = dmax(dv + c.delExtend, sv + c.delOpen);  // src/viterbi.cpp:124
  uint32_t next = kNoState;
  for (uint32_t e = o0; e < o1; ++e) {
    uint32_t w;
    if (c.outInSmem)
      w = lds32(c.aOutWords + 4 * e);
    else if (o1 <= 3)
      w = e == 0 ? slot.y : e == 1 ? slot.z : slot.w;
    else
      w = __ldg(c.gOutOvf + slot.y + e);
    const uint32_t l = peLocal(w);
    const uint32_t dS = c.aS + 8 * l, dD = c.aD + 8 * l;
    const bool emit = peIsEmit(w) != 0;
    const double sc = ldsTab(c.aSym + 8 * peSym(w));
    const double candD = (emit ? m : dv) + sc;  // src/viterbi.cpp:125 / :139
    const double candS = sv + sc;               // src/viterbi.cpp:148 (null transitions only)
    if (!kCluster || !peRemote(w)) {
      const double oldD = ldsCell(dD);
      const double oldS = emit ? candS : ldsCell(dS);
      bool grew = false;
      if (candD > oldD) grew = casMaxLocal(dD, candD, oldD);
      if (candS > oldS) grew |= casMaxLocal(dS, candS, oldS);
      if (grew) {
        if (next == kNoState && !kAppend)
          next = l;
        else
          raise<kAppend>(c, l, flagged, deferred);
      }
    } else {
      const uint32_t r = peRank(w);
      const uint32_t pD = mapToRank(dD, r), pS = mapToRank(dS, r);
      const double oldD = ldPeer(pD);
      const double oldS = emit ? candS : ldPeer(pS);
      bool grew = false;
      if (candD > oldD) grew = casMaxPeer(pD, candD, oldD);
      if (candS > oldS) grew |= casMaxPeer(pS, candS, oldS);
      if (grew) {
        // the compare-and-swap has returned, i.e. it was performed at the peer, before this is issued;
        // the peer consumes the flag after the next cluster barrier
        asm volatile("red.relaxed.cluster.shared::cluster.or.b32 [%0], %1;" ::"r"(mapToRank(c.aFlag + 4 * (l >> 5), r)),
                     "r"(1u << (l & 31))
                     : "memory");
        sent = true;
      }
    }
  }
  return next;
}

}  // namespace

// kWide: the machine has wide states (viterbi_device.cuh); only those machines run this instantiation.
template <int kMaxThreads, int kMinBlocks, bool kCluster, bool kDebug, bool kWide>
__global__ void __launch_bounds__(kMaxThreads, kMinBlocks)
    viterbiFillPushKernel(const __grid_constant__ DevTables tb, const __grid_constant__ FillArgs args) {
  constexpr int kU = kPushStatesPerThread;  // states per thread and step of a dense pass
  constexpr int kV = 2;                     // 16-byte pieces of the next chunk staged in registers per thread
  extern __shared__ __align__(128) unsigned char smem[];
  cg::cluster_group cluster = cg::this_cluster();
  const uint32_t C = kCluster ? tb.C : 1u, M = tb.M, k = tb.k;
  const uint32_t rank = kCluster ? cluster.block_rank() : 0;
  const uint32_t clusterId = blockIdx.x / C;
  const uint32_t tid = threadIdx.x, nThreads = blockDim.x;
  const uint32_t lane = tid & 31;
  const uint32_t Np = C * M;
  const double NEG = negInf();
  const PushLayout& lay = args.play;
  // The shared-window address of the dynamic shared memory.  Taken through an opaque move: left to itself
  // the compiler re-derives it (S2UR SR_CgaCtaId + ULEA + add) at every use -- 10 % of the executed
  // instructions in the profile, and a long-latency S2UR at the head of every dependent address chain.
  uint32_t sm = smemAddr(smem);
  asm volatile("mov.u32 %0, %0;" : "+r"(sm));
  const bool sPrevSmem = tb.sPrevInSmem != 0;
  const bool tRecompute = !sPrevSmem && tb.k <= 2 && args.tRecompute;

  const uint32_t aD = sm + lay.dBuf, aFlag = sm + lay.flag, aSym = sm + lay.symScore, aSub = sm + lay.sub;
  const uint32_t aTsE = sm + lay.tsE, aExt = sm + lay.tsDext, aOpen = sm + lay.tsDopen;
  const uint32_t aBuf = sm + lay.chunk, aChunkOff = sm + lay.chunkOff;
  const double noGap = tb.noGap, delOpen = tb.delOpen, delExtend = tb.delExtend, delEnd = tb.delEnd;

  double* symScore = reinterpret_cast<double*>(smem + lay.symScore);
  double* tsE = reinterpret_cast<double*>(smem + lay.tsE);
  double* tsDext = reinterpret_cast<double*>(smem + lay.tsDext);
  double* tsDopen = reinterpret_cast<double*>(smem + lay.tsDopen);
  double* subS = reinterpret_cast<double*>(smem + lay.sub);
  double* tsT = reinterpret_cast<double*>(smem + lay.tsT);
  double* lenS = reinterpret_cast<double*>(smem + lay.len);
  volatile uint32_t* ctl = reinterpret_cast<volatile uint32_t*>(smem + lay.ctl);
  uint8_t* seqS = smem + lay.seq;
  double* sG = sPrevSmem ? nullptr : args.sScratch + (size_t)clusterId * 2 * Np;
  double* s0G = args.s0Scratch + (size_t)clusterId * Np;  // S0 of the next column, written by the fused emission step
  double* tCol = tb.tInSmem ? reinterpret_cast<double*>(smem + lay.tBuf)
                            : args.tScratch + ((size_t)clusterId * C + rank) * (size_t)k * M;

  // ---- read-independent set-up ----
  for (uint32_t s = tid; s < kMaxSyms; s += nThreads) {
    const double sc = s < tb.nSyms ? tb.symScore[s] : NEG;
    symScore[s] = sc;
    tsDext[s] = sc + tb.delExtend;
    tsDopen[s] = sc + tb.delOpen;
  }
  for (uint32_t j = tid; j < 16; j += nThreads) subS[j] = tb.sub[j];
  for (uint32_t j = tid; j < 8; j += nThreads) {
    lenS[j] = j < k ? tb.len[j] : NEG;
    tsT[j] = j < k ? tb.tanDup + tb.len[j] : NEG;
  }
  auto buildTsE = [&]() {  // [(base*32+sym)*4 + observed] = (score+noGap)+sub[base][observed]
    for (uint32_t j = tid; j < 512; j += nThreads) {
      const uint32_t x = j & 3, sym = (j >> 2) & 31, base = j >> 7;
      tsE[j] = sym < tb.nSyms ? (tb.symScore[sym] + tb.noGap) + tb.sub[base * 4 + x] : NEG;
    }
  };
  buildTsE();
  const uint32_t outOffBytes = (((M + 1) * 2) + 3) & ~3u;
  const uint32_t* gOut = tb.outTable + __ldg(&tb.outSliceOff[rank]);
  if (tb.outInSmem) {
    const uint32_t nW = __ldg(&tb.outSliceOff[rank + 1]) - __ldg(&tb.outSliceOff[rank]);
    uint32_t* dst = reinterpret_cast<uint32_t*>(smem + lay.outTab);
    for (uint32_t j = tid; j < nW; j += nThreads) dst[j] = __ldg(gOut + j);
  }
  const uint32_t nChunks = tb.nChunks;
  {
    uint32_t* co = reinterpret_cast<uint32_t*>(smem + lay.chunkOff);
    for (uint32_t j = tid; j <= nChunks; j += nThreads) co[j] = __ldg(&tb.inChunkOff[rank * (nChunks + 1) + j]);
  }
  for (uint32_t j = tid; j < 64; j += nThreads) ctl[j] = 0;
  {
    uint32_t* fl = reinterpret_cast<uint32_t*>(smem + lay.flag);
    for (uint32_t j = tid; j < (M + 31) / 32; j += nThreads) fl[j] = 0;
  }
  Ctx c;
  c.aD = aD;
  c.aFlag = aFlag;
  c.aSym = aSym;
  c.aOutOff = sm + lay.outTab;
  c.aOutWords = sm + lay.outTab + outOffBytes;
  c.gOutSlots = tb.outSlots + (size_t)rank * M;
  c.gOutOvf = tb.outOvf;
  c.outInSmem = tb.outInSmem;
  c.delOpen = delOpen;
  c.delExtend = delExtend;
  c.delEnd = delEnd;
  __syncthreads();

  // ---- the streamed in-table: chunk `nextChunk` is fetched into registers while the current one is used
  const uint4* gChunks = reinterpret_cast<const uint4*>(tb.inChunks);
  const uint32_t chunkStates = tb.chunkStates;                      // = kU * nThreads
  const uint32_t recBase = ((chunkStates + 1) * 2 + 3) & ~3u;       // records start after the u16 offsets
  uint32_t nextChunk = 0, stageVec0 = 0, stageN = 0;
  uint4 stage[kV];
  auto prefetch = [&]() {
    const uint32_t o0 = lds32(aChunkOff + 4 * nextChunk), o1 = lds32(aChunkOff + 4 * nextChunk + 4);
    stageVec0 = o0 >> 2;
    stageN = (o1 - o0) >> 2;
#pragma unroll
    for (int v = 0; v < kV; ++v) {
      const uint32_t idx = v * nThreads + tid;
      stage[v] = idx < stageN ? __ldg(gChunks + stageVec0 + idx) : make_uint4(0, 0, 0, 0);
    }
  };
  auto commit = [&]() {
    __syncthreads();  // every thread is done with the current chunk (and with this step of the pass)
#pragma unroll
    for (int v = 0; v < kV; ++v) {
      const uint32_t idx = v * nThreads + tid;
      if (idx < stageN) sts128(aBuf + 16 * idx, stage[v]);
    }
    for (uint32_t idx = kV * nThreads + tid; idx < stageN; idx += nThreads)  // oversized chunk: unstaged remainder
      sts128(aBuf + 16 * idx, __ldg(gChunks + stageVec0 + idx));
    __syncthreads();
    nextChunk = nextChunk + 1 == nChunks ? 0 : nextChunk + 1;
  };
  prefetch();
  commit();  // chunk 0 is in the buffer; nextChunk = 1 (or 0 again for a one-chunk slice)

  auto clusterBarrier = [&]() {
    if (kCluster)
      cluster.sync();
    else
      __syncthreads();
  };
  clusterBarrier();  // every CTA's flags exist before a peer can touch them

  // profiling counters (dnab_decoder_debug_counters): added straight to global memory by thread 0 of rank 0, so that
  // they cost no registers when they are off
  // (the counters exist only in the kDebug instantiation, launched when dnab_decoder_set_debug is on: in the
  // production kernel they would cost registers and branches -- 14 counters kept in registers once cost 11 %)
  const bool dbgOn = kDebug && args.dbg != nullptr;  // (the kDebug kernel also serves the cell dump of dnab_viterbi_cells)
  const bool dbgMe = dbgOn && tid == 0 && rank == 0;
  auto dbgAdd = [&](int slot, unsigned long long v) { atomicAdd(&args.dbg[slot], v); };
  // time stamps of the cluster's reporting thread (column phase, closure start, level phase)
  __shared__ unsigned long long dbgStamps[kDebug ? 3 : 1];
  auto dbgStamp = [&](int stamp) {
    if (dbgMe) dbgStamps[stamp] = (unsigned long long)clock64();
  };
  auto dbgLap = [&](int stamp, int slot) {  // adds the time since the stamp to a counter and renews the stamp
    if (dbgMe) {
      const unsigned long long t = (unsigned long long)clock64();
      atomicAdd(&args.dbg[slot], t - dbgStamps[stamp]);
      dbgStamps[stamp] = t;
    }
  };

  // Reads are handed out dynamically (one global counter, fetched by rank 0 and broadcast through
  // distributed shared memory): reads differ in length, and a static stride leaves the clusters that
  // drew short reads idle at the end of the launch.
  auto nextRead = [&]() -> int64_t {
    if (rank == 0 && tid == 0) {
      const unsigned long long r = atomicAdd(args.nextRead, 1ull);
      for (uint32_t p = 0; p < C; ++p) {
        if (kCluster) {
          stPeerU32(sm + lay.ctl + 8 * 4, p, (uint32_t)r);
          stPeerU32(sm + lay.ctl + 9 * 4, p, (uint32_t)(r >> 32));
        } else {
          ctl[8] = (uint32_t)r;
          ctl[9] = (uint32_t)(r >> 32);
        }
      }
    }
    clusterBarrier();
    const int64_t r = (int64_t)(((unsigned long long)ctl[9] << 32) | ctl[8]);
    clusterBarrier();  // everyone has read the slot before rank 0 may overwrite it
    return r;
  };
  for (int64_t read = nextRead(); read < args.nReads; read = nextRead()) {
    const int32_t L = args.readLen[read];
    {  // stage the packed read
      const uint8_t* src = args.packed + args.byteOff[read];
      const uint32_t nVec = ((uint32_t)(L + 3) / 4 + 15) / 16;
      for (uint32_t v = tid; v < nVec; v += nThreads)
        reinterpret_cast<uint4*>(seqS)[v] = __ldg(reinterpret_cast<const uint4*>(src) + v);
    }
    uint8_t* predRead = args.pred + (size_t)read * (size_t)(args.maxLen + 1) * (k + 2) * Np;
    __syncthreads();

    for (int32_t pos = 0; pos <= L; ++pos) {
      const uint32_t cur = pos & 1, prev = cur ^ 1;
      const uint32_t aScur = sm + (sPrevSmem ? (cur ? lay.sBuf[1] : lay.sBuf[0]) : lay.sBuf[0]);
      const uint32_t aSprev = sm + (sPrevSmem ? (prev ? lay.sBuf[1] : lay.sBuf[0]) : lay.sBuf[0]);
      const double* sPrevG = sG + (size_t)prev * Np;  // (only dereferenced when !sPrevSmem)
      double* sCurG = sG + (size_t)cur * Np;
      const uint32_t x = pos > 0 ? (seqS[(pos - 1) >> 2] >> (2 * ((pos - 1) & 3))) & 3u : 0u;
      const uint32_t xNext = pos < L ? (seqS[pos >> 2] >> (2 * (pos & 3))) & 3u : 0u;  // the base column pos+1 reads
      c.aS = aScur;

      // S(pos-1) of the source named by an in-edge word
      auto loadPrev = [&](uint32_t w) -> double {
        if (!sPrevSmem) return sPrevG[peRank(w) * M + peLocal(w)];
        const uint32_t a = aSprev + 8 * peLocal(w);
        return (kCluster && peRemote(w)) ? ldPeer(mapToRank(a, peRank(w))) : ldsCell(a);
      };
      auto loadCell = [&](uint32_t aCol, uint32_t w) -> double {
        const uint32_t a = aCol + 8 * peLocal(w);
        return (kCluster && peRemote(w)) ? ldPeer(mapToRank(a, peRank(w))) : ldsCell(a);
      };
      // record of slot u of this thread in the staged chunk, and its header (padding header when out of range)
      auto recOf = [&](uint32_t u) -> uint32_t { return aBuf + recBase + 4 * lds16(aBuf + 2 * (u * nThreads + tid)); };
      // a wide state's record: its 16-bit counts and wide number follow the header; rec then points one header before
      // its edges, like a narrow record's
      auto wideRecord = [&](uint32_t h, uint32_t& rec, uint32_t& nIn, uint32_t& nE, uint32_t& wn) -> bool {
        if (!kWide || inNIn(h) != kInWide) return false;
        const uint32_t c2 = lds32(rec + 4);
        nE = c2 & 0xFFFFu;
        nIn = c2 >> 16;
        wn = lds32(rec + 8);
        rec += 8;
        return true;
      };

      // Duplication cells without storing them (k <= 2, S columns published in global scratch): T(p,1) =
      // (S(p)+tanDup)+len[1] and T(p,0) = max(T(p-1,1)+sub[ctx1][x_p], (S(p)+tanDup)+len[0]) are functions of
      // the state's own S(p), S(p-1) (src/viterbi.cpp:105-106,161-168), so T(pos-1,0) and T(pos-1,1) are
      // re-derived from S(pos-1), S(pos-2) with the reference's own operations instead of being kept
      // in L2-resident scratch (4 fewer 8-byte global accesses per state in each of the two passes).
      const uint32_t xPrev = pos > 1 ? (seqS[(pos - 2) >> 2] >> (2 * ((pos - 2) & 3))) & 3u : 0u;
      auto dupPrev = [&](uint32_t h, double s1, double s2, double& tPrev0, double& tPrev1) {
        const uint32_t mdl = inMdl(h);
        tPrev0 = NEG;
        tPrev1 = NEG;
        if (pos < 2 || mdl == 0) return;  // T(0,.) = -inf: duplications open from column 1 on
        if (mdl == 1) {
          tPrev0 = (s1 + tb.tanDup) + lenS[0];
          return;
        }
        tPrev1 = (s1 + tb.tanDup) + lenS[1];
        const double shifted = pos >= 3 ? ((s2 + tb.tanDup) + lenS[1]) + subS[inCtx(h, 1) * 4 + xPrev] : NEG;
        tPrev0 = dmax(shifted, (s1 + tb.tanDup) + lenS[0]);
      };

      dbgStamp(0);
      // ---- (1) S0(pos) into shared memory.  The emission step itself (src/viterbi.cpp:92-106) is FUSED into the
      // predecessor pass of the previous column (3b below), which has every S(pos-1)[src] in shared memory
      // anyway; its result travelled through a scratch column in global memory because S(pos-1) was still being
      // read by peers.  Column 0 is initialised here (src/viterbi.cpp:75-79).
      for (uint32_t i = tid; i < M; i += nThreads) {
        const uint32_t g = rank * M + i;
        double s0;
        if (pos == 0) {
          const bool real = __ldg(&tb.origId[g]) != 0xFFFFFFFFu;
          s0 = (real && (tb.local || g == tb.startG)) ? 0.0 : NEG;
          if (!tRecompute)
            for (uint32_t t = 0; t < k; ++t) tCol[t * M + i] = NEG;
        } else
          s0 = s0G[g];
        stsCell(aScur + 8 * i, s0);
        stsCell(aD + 8 * i, NEG);
      }
      clusterBarrier();  // S0 of every CTA is complete before a peer reads it
      dbgLap(0, 3);
      dbgStamp(1);

      // ---- (2a) closure, first pass, PULL over the streamed in-table (src/viterbi.cpp:97-99,110-159).
      // Successors may have read S0(d) / D = -inf or the new values (racy, benign); a state is flagged
      // when its new values can still raise a successor above what S0 / -inf already gave it.
      for (uint32_t j = 0; j < nChunks; ++j) {
        prefetch();
        uint32_t i[kU], rec[kU], h[kU], nIn[kU], nEw[kU], wn[kU];
        double s0[kU], newS[kU], newD[kU];
        uint32_t maxIn = 0;
#pragma unroll
        for (int u = 0; u < kU; ++u) {
          i[u] = j * chunkStates + u * nThreads + tid;
          rec[u] = recOf(u);
          h[u] = i[u] < M ? lds32(rec[u]) : (kInPad << 7);
          nIn[u] = inNIn(h[u]) == kInPad ? 0u : inNIn(h[u]);
          nEw[u] = inNEmit(h[u]);
          wideRecord(h[u], rec[u], nIn[u], nEw[u], wn[u]);
          maxIn = max(maxIn, nIn[u]);
          s0[u] = i[u] < M ? ldsCell(aScur + 8 * i[u]) : NEG;
          newS[u] = s0[u];
          newD[u] = NEG;
        }
        for (uint32_t e = 0; e < maxIn; ++e) {
          uint32_t w[kU];
          double ss[kU], ds[kU];
#pragma unroll
          for (int u = 0; u < kU; ++u) w[u] = e < nIn[u] ? lds32(rec[u] + 4 + 4 * e) : 0u;
#pragma unroll
          for (int u = 0; u < kU; ++u) {
            ss[u] = e < nIn[u] ? loadCell(aScur, w[u]) : NEG;
            ds[u] = e < nIn[u] ? loadCell(aD, w[u]) : NEG;
          }
#pragma unroll
          for (int u = 0; u < kU; ++u) {
            const double sc = ldsTab(aSym + 8 * peSym(w[u]));
            if (e < (kWide ? nEw[u] : inNEmit(h[u])))
              newD[u] = dmax(newD[u], dmax(ds[u] + delExtend, ss[u] + delOpen) + sc);
            else if (e < nIn[u]) {
              newD[u] = dmax(newD[u], ds[u] + sc);
              newS[u] = dmax(newS[u], ss[u] + sc);
            }
          }
        }
#pragma unroll
        for (int u = 0; u < kU; ++u) {
          bool dirty = false;
          if (i[u] < M) {
            newS[u] = dmax(newS[u], newD[u] + delEnd);
            if (newD[u] > NEG) stsCell(aD + 8 * i[u], newD[u]);
            if (newS[u] > s0[u]) stsCell(aScur + 8 * i[u], newS[u]);
            dirty = (newS[u] > s0[u]) || (newD[u] + delExtend > s0[u] + delOpen) || (inHasNullOut(h[u]) && newD[u] > NEG);
          }
          const uint32_t mask = __ballot_sync(0xFFFFFFFFu, dirty);
          if (lane == 0 && i[u] < M) {
            sts32(aFlag + 4 * (i[u] >> 5), mask);
            if (dbgOn && rank == 0) dbgAdd(8, (unsigned long long)__popc(mask));
          }
        }
        commit();
      }
      clusterBarrier();  // no peer pushes into this CTA's cells while its first pass still stores them
      dbgLap(0, 7);

      // ---- (2b) closure, PUSH levels.  Per level: the set bits of the dirty bitmap are taken and
      // compacted into a CTA-wide queue (one lane per bitmap word, one shared-memory atomic per warp);
      // after a CTA barrier every thread pushes the queued states, one state per thread and step, so
      // that all lanes of a warp work whatever the shape of the frontier; a destination that grew is
      // flagged (this CTA's bitmap or a peer's) for the next level.  A level ends with a CTA barrier;
      // when the CTA is quiet it meets the cluster, and the closure ends when nothing crossed CTAs
      // since the last meeting (a per-level cluster barrier measured slower: every level then waits
      // for the slowest CTA).
      {
        const uint32_t nWords = (M + 31) / 32, cap = lay.queueCap;
        const uint32_t aQueue = sm + lay.queue, aTail = sm + lay.ctl;  // ctl[0], ctl[1]: scan-queue tails, by level parity
        // thin frontiers: two small queues (by level parity) the pushers append to themselves, counters ctl[4..6]
        // rotated by level (a counter is zeroed one level before it is appended to)
        const uint32_t capA = lay.appendCap, aA = sm + lay.appendQueue, strideA = (2 * capA + 15u) & ~15u, aTailA = sm + lay.ctl + 16;
        uint32_t round = 0, tA = 0;  // tA = level % 3
        bool sent = false, fromAppend = false;
        // (one-CTA machines only: with peers, their flags would wait for the next scan and cost extra cluster rounds --
        // measured -4 % ... -20 % on config 2, against +23 % / +5 % on configs 4 / 3)
        // every column starts with empty scan-queue tails (a tail is otherwise only zeroed by a scan of the opposite
        // parity, and the level counter restarts at 0: a stale count would replay old queue entries)
        if (tid < 2) sts32(aTail + 4 * tid, 0u);
        if (!kCluster && tid < 3) sts32(aTailA + 4 * tid, 0u);
        __syncthreads();
        for (uint32_t levels = 0;; ++levels) {
          const uint32_t par = levels & 1;
          const bool scanned = kCluster || !fromAppend;
          const uint32_t tANext = tA == 2 ? 0u : tA + 1, tAAfter = tANext == 2 ? 0u : tANext + 1;
          dbgStamp(2);
          bool flagged = false, deferred = false;
          uint32_t n, aList;
          if (kCluster || !fromAppend) {
            // the work list of this level: the set bits of the dirty bitmap, compacted into the big queue
            for (uint32_t base = 0; base < nWords; base += nThreads) {
              if (base + (tid & ~31u) >= nWords) break;  // warp-uniform: this warp has no bitmap word to scan
              const uint32_t wi = base + tid;
              const uint32_t aWord = aFlag + 4 * wi;
              uint32_t taken = (wi < nWords && ldsVolatile32(aWord)) ? atomExchShared(aWord, 0u) : 0u;
              const uint32_t cnt = __popc(taken);
              uint32_t incl = cnt;
#pragma unroll
              for (uint32_t dlt = 1; dlt < 32; dlt <<= 1) {
                const uint32_t up = __shfl_up_sync(0xFFFFFFFFu, incl, dlt);
                if (lane >= dlt) incl += up;
              }
              const uint32_t total = __shfl_sync(0xFFFFFFFFu, incl, 31);
              if (total == 0) continue;  // warp-uniform
              uint32_t wbase = 0;
              if (lane == 31) wbase = atomAddShared(aTail + 4 * par, total);
              wbase = __shfl_sync(0xFFFFFFFFu, wbase, 31);
              uint32_t at = wbase + incl - cnt, putBack = 0;
              while (taken) {
                const uint32_t bit = __ffs(taken) - 1;
                taken &= taken - 1;
                if (at < cap)
                  sts16(aQueue + 2 * at, 32 * wi + bit);
                else
                  putBack |= 1u << bit;  // queue full: the state waits for the next level
                ++at;
              }
              if (putBack) {
                redOrShared(aWord, putBack);
                flagged = true;
              }
            }
            __syncthreads();  // queue complete; every cell stored before the bits were set is visible
            n = ldsVolatile32(aTail + 4 * par);
            if (n > cap) n = cap;
            if (tid == 0) sts32(aTail + 4 * (par ^ 1), 0u);  // the other tail is idle until the next scan
            aList = aQueue;
          } else {
            // the work list was appended by the previous level's pushers (their bits are still set: see below)
            n = ldsVolatile32(aTailA + 4 * tA);
            if (n > capA) n = capA;
            aList = aA + par * strideA;
          }
          dbgLap(2, 9);
          if (dbgMe) dbgAdd(1, 1);
          if (levels > (1u << 22)) __trap();  // never hang the GPU: a closure that does not settle is a bug
          if (!kCluster && tid == 0) sts32(aTailA + 4 * tAAfter, 0u);
          c.aQueueNext = aA + (par ^ 1) * strideA;
          c.aTailNext = aTailA + 4 * tANext;
          c.capNext = capA;
          // one hop per level, breadth first; one state per thread and step
          auto pushList = [&](auto appendTag) {
            constexpr bool kAppend = decltype(appendTag)::value;
            uint32_t sNext = tid < n ? lds16(aList + 2 * tid) : 0u;
            uint4 slNext = (!c.outInSmem && tid < n) ? __ldg(c.gOutSlots + sNext) : make_uint4(0, 0, 0, 0);
            for (uint32_t q = tid; q < n; q += nThreads) {
              const uint32_t sCur = sNext;
              const uint4 slCur = slNext;
              if (q + nThreads < n) {  // the next entry's slot travels while this one is pushed
                sNext = lds16(aList + 2 * (q + nThreads));
                if (!c.outInSmem) slNext = __ldg(c.gOutSlots + sNext);
              }
              // an appended state is "queued" until now: a pusher that raises it after its cells are read queues it again
              if (!kCluster && fromAppend) redAndShared(aFlag + 4 * (sCur >> 5), ~(1u << (sCur & 31)));
              const uint32_t nx = pushState<kCluster, kAppend>(c, sCur, slCur, flagged, deferred, sent);
              if (nx != kNoState) {
                redOrShared(aFlag + 4 * (nx >> 5), 1u << (nx & 31));
                flagged = true;
              }
            }
          };
          if (!kCluster && n <= args.thinN)
            pushList(std::true_type{});
          else
            pushList(std::false_type{});
          if (dbgMe) dbgAdd(2, n);
          dbgLap(2, 10);
          // every push of this level has flagged or queued its successors
          const uint32_t needScan = (uint32_t)__syncthreads_or((flagged || deferred) ? 1 : 0);
          if (scanned && tid == 0) sts32(aTail + 4 * par, 0u);  // consumed: the next scan of this parity starts empty
          tA = tANext;
          dbgLap(2, 12);
          if (needScan) {  // (a scan also takes the bits of whatever was appended meanwhile: that list is dropped)
            fromAppend = false;
            continue;
          }
          if (!kCluster && ldsVolatile32(aTailA + 4 * tA) != 0u) {
            fromAppend = true;
            continue;
          }
          fromAppend = false;
          if (!kCluster) break;
          // locally quiet: meet the cluster; another round if anything crossed CTAs since the last meeting
          dbgStamp(2);
          const uint32_t anySent = (uint32_t)__syncthreads_or(sent ? 1 : 0);
          sent = false;
          if (tid < C) stPeerU32(sm + lay.ctl + (16 + (round & 1) * kMaxCluster + rank) * 4, tid, anySent);
          cluster.sync();
          dbgLap(2, 11);
          uint32_t tot = 0;
          for (uint32_t r = 0; r < C; ++r) tot |= ctl[16 + (round & 1) * kMaxCluster + r];
          ++round;
          if (!tot) break;
          if (dbgMe) dbgAdd(6, 1);
        }
      }
      if (dbgMe) {
        const unsigned long long t = (unsigned long long)clock64();
        atomicAdd(&args.dbg[4], t - dbgStamps[1]);
        dbgStamps[0] = t;
      }

      // ---- (3) predecessor records with the traceback's arithmetic (src/viterbi.cpp:251-286)
      //      (4) duplication opens (src/viterbi.cpp:161-168) ----
      uint8_t* predCol = predRead + (size_t)pos * (k + 2) * Np;
      uint8_t* const predWideCol = kWide ? args.predWide + ((size_t)read * (args.maxLen + 1) + pos) * 2 * tb.nWide : nullptr;
      for (uint32_t j = 0; j < nChunks; ++j) {
        prefetch();
        uint32_t i[kU], rec[kU], h[kU], nIn[kU], idx[kU], idxD[kU], nEw[kU], wn[kU];
        bool wide[kU];
        double sHere[kU], dHere[kU], parked[kU], tPrev1[kU], best[kU], bestD[kU], s0n[kU];
        uint32_t maxIn = 0;
#pragma unroll
        for (int u = 0; u < kU; ++u) {
          i[u] = j * chunkStates + u * nThreads + tid;
          rec[u] = recOf(u);
          h[u] = i[u] < M ? lds32(rec[u]) : (kInPad << 7);
          nIn[u] = inNIn(h[u]) == kInPad ? 0u : inNIn(h[u]);
          nEw[u] = inNEmit(h[u]);
          wide[u] = wideRecord(h[u], rec[u], nIn[u], nEw[u], wn[u]);
          maxIn = max(maxIn, nIn[u]);
          const uint32_t mdl = inMdl(h[u]);
          sHere[u] = i[u] < M ? ldsCell(aScur + 8 * i[u]) : NEG;
          dHere[u] = i[u] < M ? ldsCell(aD + 8 * i[u]) : NEG;
          tPrev1[u] = NEG;
          if (tRecompute) {
            double tPrev0 = NEG;
            if (i[u] < M && mdl > 0 && pos > 0) dupPrev(h[u], sPrevG[rank * M + i[u]], sCurG[rank * M + i[u]], tPrev0, tPrev1[u]);
            parked[u] = (mdl > 0 && pos > 0) ? tPrev0 + subS[inCtx(h[u], 0) * 4 + x] : NEG;
          } else
            parked[u] = (mdl > 0 && pos > 0) ? tCol[(mdl - 1) * M + i[u]] : NEG;  // T(state,pos-1,0)+sub
          best[u] = NEG;
          bestD[u] = NEG;
          idx[u] = wide[u] ? kWideNoPred : kNoPred;
          idxD[u] = idx[u];
          s0n[u] = NEG;
        }
        for (uint32_t e = 0; e < maxIn; ++e) {
          uint32_t w[kU];
          double vs[kU], vd[kU], vp[kU];
#pragma unroll
          for (int u = 0; u < kU; ++u) w[u] = e < nIn[u] ? lds32(rec[u] + 4 + 4 * e) : 0u;
#pragma unroll
          for (int u = 0; u < kU; ++u) {
            vs[u] = e < nIn[u] ? loadCell(aScur, w[u]) : NEG;
            vd[u] = e < nIn[u] ? loadCell(aD, w[u]) : NEG;
            vp[u] = (pos > 0 && e < (kWide ? nEw[u] : inNEmit(h[u]))) ? loadPrev(w[u]) : NEG;
          }
#pragma unroll
          for (int u = 0; u < kU; ++u) {
            const uint32_t nE = kWide ? nEw[u] : inNEmit(h[u]);
            const uint32_t sym8 = 8 * peSym(w[u]);
            if (e < nE) {
              if (pos > 0) {
                const double v = vp[u] + ldsTab(aTsE + 8 * ((((w[u] >> 21) & 0x7Fu) << 2) + x));
                if (v > best[u]) {
                  best[u] = v;
                  idx[u] = e;
                }
              }
              const double ve = vd[u] + ldsTab(aExt + sym8);
              if (ve > bestD[u]) {
                bestD[u] = ve;
                idxD[u] = 2 * e;
              }
              const double vo = vs[u] + ldsTab(aOpen + sym8);
              if (vo > bestD[u]) {
                bestD[u] = vo;
                idxD[u] = 2 * e + 1;
              }
              // (3b) emission step of column pos+1 (src/viterbi.cpp:92-95): the same S(pos)[src], fill association
              if (pos < L)
                s0n[u] = dmax(s0n[u], ((vs[u] + ldsTab(aSym + sym8)) + noGap) + ldsTab(aSub + 8 * (peBase(w[u]) * 4 + xNext)));
            } else if (e < nIn[u]) {
              const double sc = ldsTab(aSym + sym8);
              const double v = vs[u] + sc;
              if (v > best[u]) {
                best[u] = v;
                idx[u] = e;
              }
              const double vn = vd[u] + sc;
              if (vn > bestD[u]) {
                bestD[u] = vn;
                idxD[u] = nE + e;  // = 2*nE + (e - nE)
              }
            }
          }
        }
#pragma unroll
        for (int u = 0; u < kU; ++u)
          if (i[u] < M) {
            const uint32_t g = rank * M + i[u];
            const bool real = inNIn(h[u]) != kInPad;
            const uint32_t mdl = inMdl(h[u]);
            if (!sPrevSmem) sCurG[g] = sHere[u];  // publish the converged column for the next position
            {
              const double v = dHere[u] + delEnd;
              if (v > best[u]) {
                best[u] = v;
                idx[u] = nIn[u];
              }
            }
            if (mdl > 0 && pos > 0 && parked[u] > best[u]) {
              best[u] = parked[u];
              idx[u] = nIn[u] + 1;
            }
            if (tb.local && pos == 0) {
              const uint32_t a = aScur + (tb.startG % M) * 8, r = tb.startG / M;
              const double v = ((!kCluster || r == rank) ? ldsCell(a) : ldPeer(mapToRank(a, r))) + 0.0;
              if (v > best[u]) {
                best[u] = v;
                idx[u] = nIn[u] + 2;
              }
            }
            predCol[g] = (uint8_t)(real ? idx[u] : kNoPred);
            predCol[Np + g] = (uint8_t)(real ? idxD[u] : kNoPred);
            if (wide[u]) {  // the high bytes (a wide state is real)
              predWideCol[wn[u]] = (uint8_t)(idx[u] >> 8);
              predWideCol[tb.nWide + wn[u]] = (uint8_t)(idxD[u] >> 8);
            }
            double* cell = (kDebug && args.cells && read == 0 && real)  // the cell dump exists in the kDebug kernel only
                               ? args.cells + ((size_t)pos * tb.nStates + __ldg(&tb.origId[g])) * (k + 2)
                               : nullptr;
            if (cell) {
              cell[0] = sHere[u];
              cell[1] = dHere[u];
            }
            double tNow0 = NEG;  // T(state,pos,0)
            for (uint32_t t = 0; t < k; ++t) {
              uint32_t idxT = kNoPred;
              double tNow = NEG;
              if (pos > 0 && t < mdl) {
                double shifted = NEG;
                if (t + 1 < mdl) shifted = tRecompute ? tPrev1[u] + subS[inCtx(h[u], 1) * 4 + x] : tCol[t * M + i[u]];
                if (t + 1 < mdl && shifted > NEG) idxT = 0;
                if (sHere[u] + tsT[t] > shifted) idxT = 1;
                tNow = dmax(shifted, (sHere[u] + tb.tanDup) + lenS[t]);  // (4)
                if (!tRecompute) tCol[t * M + i[u]] = tNow;
              }
              predCol[(size_t)(2 + t) * Np + g] = (uint8_t)idxT;
              if (cell) cell[2 + t] = tNow;
              if (t == 0) tNow0 = tNow;
            }
            // (3b) continued: the T -> S candidate and the T shift of column pos+1 (src/viterbi.cpp:102-106)
            if (pos < L) {
              if (mdl > 0) {
                const double t2s = tNow0 + subS[inCtx(h[u], 0) * 4 + xNext];
                s0n[u] = dmax(s0n[u], t2s);
                if (!tRecompute) {
                  for (uint32_t t = 0; t + 1 < mdl; ++t)
                    tCol[t * M + i[u]] = tCol[(t + 1) * M + i[u]] + subS[inCtx(h[u], t + 1) * 4 + xNext];
                  tCol[(mdl - 1) * M + i[u]] = t2s;  // slot mdl-1 is free until (4) of the next column: park the T->S candidate there
                }
              }
              s0G[g] = s0n[u];
            }
          }
        commit();
      }
      clusterBarrier();
      dbgLap(0, 5);
      if (dbgMe) dbgAdd(0, 1);
    }

    // ---- end of read: log-likelihood and traceback start (src/viterbi.cpp:171-173, 239-245) ----
    {
      const double* sLast = reinterpret_cast<const double*>(smem + ((sPrevSmem && (L & 1)) ? lay.sBuf[1] : lay.sBuf[0]));
      if (!tb.local) {
        if (rank == tb.endG / M && tid == 0) {
          args.loglike[read] = sLast[tb.endG % M];
          args.startState[read] = tb.endG;
        }
        __syncthreads();
      } else {
        // first strict maximum in REFERENCE state order: max value, then smallest original index
        double bv = NEG;
        uint32_t bo = 0xFFFFFFFFu, bg = 0;
        for (uint32_t i = tid; i < M; i += nThreads) {
          const uint32_t g = rank * M + i;
          const uint32_t o = __ldg(&tb.origId[g]);
          if (o == 0xFFFFFFFFu) continue;
          const double v = sLast[i];
          if (v > bv || (v == bv && o < bo)) {
            bv = v;
            bo = o;
            bg = g;
          }
        }
        for (int sh = 16; sh > 0; sh >>= 1) {
          const double ov = __shfl_down_sync(0xFFFFFFFFu, bv, sh);
          const uint32_t oo = __shfl_down_sync(0xFFFFFFFFu, bo, sh);
          const uint32_t og = __shfl_down_sync(0xFFFFFFFFu, bg, sh);
          if (ov > bv || (ov == bv && oo < bo)) {
            bv = ov;
            bo = oo;
            bg = og;
          }
        }
        __syncthreads();
        // reduction scratch: the tsE table (rebuilt below) is free between reads
        double* rv = tsE;
        uint32_t* ro = reinterpret_cast<uint32_t*>(tsE + 32);
        if (lane == 0) {
          rv[tid >> 5] = bv;
          ro[2 * (tid >> 5)] = bo;
          ro[2 * (tid >> 5) + 1] = bg;
        }
        __syncthreads();
        if (tid == 0) {
          const uint32_t nw = (nThreads + 31) / 32;
          for (uint32_t w = 1; w < nw; ++w)
            if (rv[w] > bv || (rv[w] == bv && ro[2 * w] < bo)) {
              bv = rv[w];
              bo = ro[2 * w];
              bg = ro[2 * w + 1];
            }
          args.partVal[read * C + rank] = bv;
          args.partOrig[read * C + rank] = bo;
          args.partG[read * C + rank] = bg;
        }
        __syncthreads();
        buildTsE();
        __syncthreads();
      }
    }
  }
  clusterBarrier();  // no CTA may exit while a peer can still touch its shared memory
}

// ---------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------
typedef void (*PushKernelPtr)(const DevTables, const FillArgs);
template <bool kCluster, bool kDebug, bool kWide>
static PushKernelPtr pickPushKernelT(uint32_t threads) {
  if (threads > 800) return viterbiFillPushKernel<1024, 1, kCluster, kDebug, kWide>;  // 64 registers/thread
  if (threads > 640) return viterbiFillPushKernel<800, 1, kCluster, kDebug, kWide>;   // 80
  if (threads > 512) return viterbiFillPushKernel<640, 1, kCluster, kDebug, kWide>;   // 96
  if (threads > 256) return viterbiFillPushKernel<512, 1, kCluster, kDebug, kWide>;   // 128
  // narrow CTAs (small machines, many CTAs per SM): registers are allocated in units of 8, so 81 means 88 and one
  // resident CTA fewer than 80 -- a third block in the launch bounds caps the one-CTA kernel at 80
  if constexpr (!kCluster)
    return viterbiFillPushKernel<256, 3, false, kDebug, kWide>;  // 80
  else
    return viterbiFillPushKernel<256, 2, true, kDebug, kWide>;  // 128
}
template <bool kWide>
static PushKernelPtr pickPushKernelW(const DevTables& tb, uint32_t threads, bool debug) {
  if (debug) return tb.C > 1 ? pickPushKernelT<true, true, kWide>(threads) : pickPushKernelT<false, true, kWide>(threads);
  return tb.C > 1 ? pickPushKernelT<true, false, kWide>(threads) : pickPushKernelT<false, false, kWide>(threads);
}
static PushKernelPtr pickPushKernel(const DevTables& tb, uint32_t threads, bool debug) {
  return tb.nWide ? pickPushKernelW<true>(tb, threads, debug) : pickPushKernelW<false>(tb, threads, debug);
}

static cudaError_t prepPush(PushKernelPtr kern, const DevTables& tb, uint32_t smemBytes) {
  cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemBytes);
  if (err != cudaSuccess) return err;
  if (tb.C > 8) err = cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  return err;
}

static void pushClusterConfig(cudaLaunchConfig_t& cfg, cudaLaunchAttribute* attr, const DevTables& tb, uint32_t nClusters,
                              uint32_t threads, uint32_t smemBytes, cudaStream_t stream) {
  cfg = cudaLaunchConfig_t{};
  cfg.gridDim = dim3(nClusters * tb.C);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smemBytes;
  cfg.stream = stream;
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = tb.C;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
}

cudaError_t launchFillPush(const DevTables& tb, const FillArgs& args, uint32_t nClusters, uint32_t threads,
                           uint32_t smemBytes, cudaStream_t stream) {
  PushKernelPtr kern = pickPushKernel(tb, threads, args.dbg != nullptr || args.cells != nullptr);
  cudaError_t err = prepPush(kern, tb, smemBytes);
  if (err != cudaSuccess) return err;
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute attr[1];
  pushClusterConfig(cfg, attr, tb, nClusters, threads, smemBytes, stream);
  return cudaLaunchKernelEx(&cfg, kern, tb, args);
}

cudaError_t queryMaxClustersPush(const DevTables& tb, uint32_t threads, uint32_t smemBytes, int* nClusters) {
  PushKernelPtr kern = pickPushKernel(tb, threads, false);
  cudaError_t err = prepPush(kern, tb, smemBytes);
  if (err != cudaSuccess) return err;
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute attr[1];
  pushClusterConfig(cfg, attr, tb, 1, threads, smemBytes, nullptr);
  return cudaOccupancyMaxActiveClusters(nClusters, kern, &cfg);
}

}  // namespace dnab
