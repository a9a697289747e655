// Decoder handle: the flat tables resident on one B200 plus the launch logic.
// Implements the decoder half of include/dnastore_b200.h.  There is no CPU
// fallback anywhere in this file: without a CUDA device every entry point fails.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/dnastore_b200.h"
#include "capi_error.h"
#include "viterbi_batch.h"
#include "viterbi_kernels.h"

namespace dnab {

#define CUDA_TRY(expr)                                                                        \
  do {                                                                                        \
    cudaError_t err__ = (expr);                                                               \
    if (err__ != cudaSuccess) {                                                               \
      setLastError(std::string("CUDA error: ") + cudaGetErrorString(err__) + " at " #expr);   \
      return DNAB_ECUDA;                                                                      \
    }                                                                                         \
  } while (0)

template <class T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  ~DevBuf() { release(); }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
  cudaError_t ensure(size_t count) {
    if (count <= n) return cudaSuccess;
    release();
    cudaError_t e = cudaMalloc(&p, count * sizeof(T));
    if (e == cudaSuccess) n = count;
    return e;
  }
  cudaError_t upload(const std::vector<T>& v) {
    cudaError_t e = ensure(std::max<size_t>(v.size(), 1));
    if (e != cudaSuccess || v.empty()) return e;
    return cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
  }
};

// plan of the push kernel (viterbi_fill_push.cu)
struct LaunchPlan {
  uint32_t C = 0, M = 0, threads = 0, tInSmem = 0, sPrevGlobal = 0, smemBytes = 0, nClusters = 0;
  uint32_t outInSmem = 0, outBytes = 0, chunkBytes = 0, queueCap = 0;
  int32_t maxLen = -1;
};

// plan of the read-batched kernel (viterbi_fill_batch.cu)
struct BatchPlan {
  bool ready = false, feasible = false;
  uint32_t T = 0, M = 0, warps = 0, smemBytes = 0, nTeams = 0, ctasPerSm = 0;
  double crossFraction = 0;  // transitions whose ends live in different CTAs
};

}  // namespace dnab

using namespace dnab;

struct dnab_decoder {
  int device = 0;
  int smCount = 0;
  size_t smemOptin = 0;
  // host copy of the tables (owned)
  uint32_t nStates = 0, k = 0, local = 0;
  std::vector<uint32_t> emitOff, emitSrc, nullOff, nullSrc;
  std::vector<uint8_t> emitSym, emitBase, nullSym, ctx, mdl;
  std::vector<uint8_t> symChar;
  std::vector<double> symScore;
  double sub[16], len[kMaxK], noGap, delOpen, delExtend, delEnd, tanDup;
  // user overrides
  uint32_t wantC = 0, wantThreads = 0, wantTMode = 0;  // tMode: 0 auto, 1 smem, 2 global
  uint32_t wantBlockMode = 0;   // transition table: 0 auto, 1 shared memory, 2 global memory
  uint32_t tRecompute = 1;
  uint32_t thinN = 1024;  // push kernel, one-CTA machines: levels of at most this many states queue their successors directly (option "thin_n")
  uint32_t dealChunks = 8;  // push kernel, partition mode 3: DFS chunks dealt per CTA (option "deal_chunks")
  uint32_t queueCap = 0;    // push kernel: cap of the level queue, 0 = automatic (option "queue_cap")
  uint32_t wantSPrevMode = 0;   // S(pos-1): 0 auto, 1 shared memory, 2 global scratch
  uint32_t wantPartition = 0;   // 0/1 index-order runs + in-degree sort (default), 2 DFS runs unsorted, 3 DFS chunks dealt round-robin + sort, 4 DFS runs + sort
  // device-resident structures for the current plan
  LaunchPlan plan;
  DevTables dev{};
  DevBuf<uint32_t> dBlocks, dBlockOff, dOrigId;
  DevBuf<uint32_t> dInChunks, dInChunkOff, dOutTable, dOutSliceOff, dOutOvf;
  DevBuf<uint4> dOutSlots;
  DevBuf<uint8_t> dSymChar;
  // scratch
  DevBuf<uint8_t> dPred, dPredWide;  // predecessor records; high bytes of the wide states' records (viterbi_device.cuh)
  DevBuf<double> dTScratch, dSScratch, dS0Scratch, dPartVal, dCells;
  DevBuf<uint32_t> dStart, dPartOrig, dPartG;
  DevBuf<unsigned long long> dDbg, dNextRead;
  // forward kernel (forward_kernels.cu): CSR tables in reference order, uploaded on first use
  bool fwdReady = false;
  uint32_t fwdThreads = 0;  // options "fwd_threads" (CTA width, 0 = by state count) and "fwd_blocks" (grid cap, 0 = none)
  uint32_t fwdBlocks = 0;
  DevBuf<uint32_t> dFwdEmitOff, dFwdEmitSrc, dFwdNullOff, dFwdNullSrc;
  DevBuf<uint8_t> dFwdEmitMeta, dFwdNullSym, dFwdCtx, dFwdMdl;
  DevBuf<double> dFwdLse, dFwdScratch, dFwdF, dFwdCounts, dFwdLLBack;
  DevBuf<uint32_t> dFwdOutEmitOff, dFwdOutEmitDst, dFwdOutNullOff, dFwdOutNullDst;
  DevBuf<uint8_t> dFwdOutEmitMeta, dFwdOutNullSym;
  DevBuf<long long> dFwdSweepsBack, dFwdPostOff;
  DevBuf<double> dFwdPost;
  DevBuf<long long> dFwdSweeps;
  bool debug = false;
  // read-batched kernel: 32 reads per group are the SIMD lanes (viterbi_fill_batch.cu)
  int32_t wantBatch = -1;       // -1 auto (used when feasible and no push-kernel tuning was requested), 0 off, 1 required
  uint32_t wantTeam = 0;        // CTAs per team (0 = smallest that fits)
  uint32_t wantWarps = 0;       // warps per CTA (0 = 32)
  BatchPlan bplan;
  uint32_t notifyClasses = 32;  // option "notify_classes": notification counters per CTA of a team (1 = a notification wakes every
                                // transition that crosses CTAs; 32 = a 32nd of them, one class per lane of the polling warp)
  uint32_t eagerNotify = 0;     // option "eager_notify"
  uint32_t batchIdleNs = 100;   // option "batch_idle_ns"
  uint32_t asyncClosure = 2;    // read-batched kernel: closure without level barriers: 0 off, 1 on, 2 automatic = on (option "async_closure")
  uint32_t teamSlackPct = 8;    // states per CTA above the balanced share that the partitioner may use (option "team_slack_pct")
  uint32_t wantPersist = 0;     // carried rows in the persisting part of L2 (option "persist_l2")
  size_t persistBytes = 0;
  BatchTables btab{};
  BatchTraceTables btrace{};
  DevBuf<uint4> dbHdr;
  DevBuf<uint2> dbIn, dbRel, dbHdr2;
  DevBuf<uint32_t> dbOut, dbRankInOff, dbRankOutOff, dbRemoteIn, dbEmitOff, dbEmitSrc, dbNullOff, dbNullSrc, dbTeamState, dbTeamPassive, dbClsOff, dbClsStates, dbPartOrig, dbWideOf;
  DevBuf<uint4> dbWide;
  DevBuf<uint8_t> dbEmitSym, dbNullSym;
  DevBuf<double> dbTsE, dbPriv, dbPartVal;
  DevBuf<double2> dbSdPub;
  DevBuf<unsigned long long> dbBarrier;
  DevBuf<int32_t> dbOrder;
  // staging for the host-buffer path
  DevBuf<uint8_t> dPacked;
  DevBuf<int64_t> dByteOff;
  DevBuf<int32_t> dReadLen, dDecodedLen, dStatus, dPath, dPathLen;
  DevBuf<double> dLoglike;
  DevBuf<char> dDecoded;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr;
  // device-path timing: (start, mid, end) event triples per chunk, resolved lazily in get_stats
  bool timing = false;
  std::vector<cudaEvent_t> evPool;
  size_t evUsed = 0;
  dnab_decoder_stats stats{};
  size_t predBudgetBytes = 0;
};

namespace dnab {

// Wide states (viterbi_device.cuh), numbered in reference order: wideOf[s] is the wide number of state s or 0xFFFFFFFF.
// Refuses a state whose records or counts no format holds.  Both planners use this one classification.
static int numberWideStates(const dnab_decoder* d, std::vector<uint32_t>& wideOf, uint32_t& nWide) {
  const uint32_t N = d->nStates;
  std::vector<uint32_t> nOut(N, 0);
  for (uint32_t s : d->emitSrc) ++nOut[s];
  for (uint32_t s : d->nullSrc) ++nOut[s];
  wideOf.assign(N, 0xFFFFFFFFu);
  nWide = 0;
  for (uint32_t s = 0; s < N; ++s) {
    const uint64_t nE = d->emitOff[s + 1] - d->emitOff[s], nN = d->nullOff[s + 1] - d->nullOff[s];
    if (nE + nN + 3 > kMaxWideCandidates || 2 * nE + nN > kMaxWideCandidates) {
      setLastError("state " + std::to_string(s) + " has " + std::to_string(nE) + " emitting and " + std::to_string(nN) +
                   " null incoming transitions: predecessor records hold at most 65535 candidates (nEmit + nNull + 3 and "
                   "2*nEmit + nNull must not exceed 65535)");
      return DNAB_EINVAL;
    }
    if (nOut[s] > kMaxOutDegree) {
      setLastError("state " + std::to_string(s) + " has " + std::to_string(nOut[s]) +
                   " outgoing transitions: at most 65535 are supported");
      return DNAB_EINVAL;
    }
    if (stateIsWide((uint32_t)nE, (uint32_t)nN, nOut[s])) wideOf[s] = nWide++;
  }
  return DNAB_OK;
}

// Alternative order of the states: depth-first preorder over the transition graph.  Cutting it
// into C equal runs keeps more transitions inside one CTA (85% on the BASELINE config 2 machine
// against 56% for index order).  The push kernel deals chunks of it to the CTAs by default
// (partition mode 3); option "partition" selects the others.
static std::vector<uint32_t> dfsOrder(const dnab_decoder* d) {
  const uint32_t N = d->nStates;
  std::vector<uint32_t> outOff(N + 1, 0), outDst;
  auto countEdges = [&](const std::vector<uint32_t>& src) {
    for (uint32_t s : src) ++outOff[s + 1];
  };
  countEdges(d->emitSrc);
  countEdges(d->nullSrc);
  for (uint32_t s = 0; s < N; ++s) outOff[s + 1] += outOff[s];
  outDst.resize(outOff[N]);
  std::vector<uint32_t> fill(outOff.begin(), outOff.end() - 1);
  for (uint32_t g = 0; g < N; ++g) {
    for (uint32_t e = d->emitOff[g]; e < d->emitOff[g + 1]; ++e) outDst[fill[d->emitSrc[e]]++] = g;
    for (uint32_t e = d->nullOff[g]; e < d->nullOff[g + 1]; ++e) outDst[fill[d->nullSrc[e]]++] = g;
  }
  std::vector<uint32_t> order;
  order.reserve(N);
  std::vector<char> seen(N, 0);
  std::vector<uint32_t> stack;
  for (uint32_t root = 0; root < N; ++root) {
    if (seen[root]) continue;
    seen[root] = 1;
    stack.push_back(root);
    while (!stack.empty()) {
      const uint32_t v = stack.back();
      stack.pop_back();
      order.push_back(v);
      for (uint32_t e = outOff[v]; e < outOff[v + 1]; ++e) {
        const uint32_t u = outDst[e];
        if (!seen[u]) {
          seen[u] = 1;
          stack.push_back(u);
        }
      }
    }
  }
  return order;
}

// Assignment of the states to the C CTAs of a cluster, and the state blocks of the traceback.
struct Partition {
  uint32_t C = 0, M = 0;
  std::vector<uint32_t> newOf;   // reference state -> padded index g
  std::vector<uint32_t> origOf;  // padded index g -> reference state (0xFFFFFFFF = padding)
  std::vector<uint32_t> blocks, blockOff;
};

static int buildPartition(const dnab_decoder* d, uint32_t C, const std::vector<uint32_t>& wideOf, Partition& P) {
  const uint32_t N = d->nStates, k = d->k;
  const uint32_t M = (N + C - 1) / C, Np = C * M;
  P.C = C;
  P.M = M;
  // 1. CTA assignment: equal runs of the reference's state order (default) or of a DFS order
  std::vector<uint32_t> order;
  const uint32_t partMode = d->wantPartition ? d->wantPartition : 3u;
  const bool useDfs = partMode >= 2;
  if (C > 1 && useDfs)
    order = dfsOrder(d);
  else {
    order.resize(N);
    for (uint32_t s = 0; s < N; ++s) order[s] = s;
  }
  // 2. inside a CTA: descending in-degree, so that the 32 lanes of a warp walk equally long edge
  //    lists (dense passes) and the few hub states sit together; stable, so runs keep DFS order
  auto inDeg = [&](uint32_t s) { return (d->emitOff[s + 1] - d->emitOff[s]) + (d->nullOff[s + 1] - d->nullOff[s]); };
  P.origOf.assign(Np, 0xFFFFFFFFu);
  P.newOf.assign(N, 0);
  // partition mode 3: the DFS order is cut into 8*C chunks dealt round-robin to the CTAs, trading some
  // locality for CTAs that are busy for equally long inside a closure round
  std::vector<std::vector<uint32_t>> dealt(C);
  if (partMode == 3 && C > 1) {
    const uint32_t deal = std::max<uint32_t>(1, d->dealChunks);  // chunks per CTA (option "deal_chunks")
    const uint32_t chunk = std::max<uint32_t>(32, (N + deal * C - 1) / (deal * C));
    uint32_t r = 0;
    for (uint32_t lo = 0; lo < N;) {
      while (dealt[r].size() >= M) r = (r + 1) % C;  // a CTA never takes more than M states
      const uint32_t hi = std::min<uint32_t>(std::min(N, lo + chunk), lo + (M - (uint32_t)dealt[r].size()));
      dealt[r].insert(dealt[r].end(), order.begin() + lo, order.begin() + hi);
      lo = hi;
      r = (r + 1) % C;
    }
  }
  for (uint32_t r = 0; r < C; ++r) {
    const uint32_t lo = std::min(N, r * M), hi = std::min(N, (r + 1) * M);
    std::vector<uint32_t> mine(order.begin() + lo, order.begin() + hi);
    if (partMode == 3 && C > 1) mine = dealt[r];
    if (partMode != 2)
      std::stable_sort(mine.begin(), mine.end(), [&](uint32_t a, uint32_t b) { return inDeg(a) > inDeg(b); });
    for (uint32_t j = 0; j < mine.size(); ++j) {
      P.origOf[r * M + j] = mine[j];
      P.newOf[mine[j]] = r * M + j;
    }
  }
  // 3. state blocks (viterbi_device.cuh)
  std::vector<std::vector<uint32_t>> outs(N);
  for (uint32_t s = 0; s < N; ++s) {
    for (uint32_t e = d->emitOff[s]; e < d->emitOff[s + 1]; ++e) outs[d->emitSrc[e]].push_back(P.newOf[s]);
    for (uint32_t e = d->nullOff[s]; e < d->nullOff[s + 1]; ++e) outs[d->nullSrc[e]].push_back(P.newOf[s]);
  }
  P.blocks.clear();
  P.blockOff.assign(Np, 0);
  for (uint32_t g = 0; g < Np; ++g) {
    const uint32_t rank = g / M;
    {
      // a block that fits one 32-byte sector must not straddle two (one L1/L2 access per state)
      const uint32_t s0 = P.origOf[g];
      uint32_t words = 2;
      if (s0 != 0xFFFFFFFFu) {
        const uint32_t nIn0 = (d->emitOff[s0 + 1] - d->emitOff[s0]) + (d->nullOff[s0 + 1] - d->nullOff[s0]);
        std::vector<uint32_t> tmp = outs[s0];
        std::sort(tmp.begin(), tmp.end());
        words = 2 + 2 * nIn0 + (uint32_t)(std::unique(tmp.begin(), tmp.end()) - tmp.begin()) + (wideOf[s0] != 0xFFFFFFFFu ? 2 : 0);
      }
      const uint32_t at = (uint32_t)P.blocks.size() % 8;
      if (words <= 8 && at + words > 8)
        while (P.blocks.size() % 8) P.blocks.push_back(0);
    }
    P.blockOff[g] = (uint32_t)P.blocks.size();
    const uint32_t s = P.origOf[g];
    if (s == 0xFFFFFFFFu) {
      P.blocks.push_back(0);
      P.blocks.push_back(0);
    } else {
      const uint32_t nE = d->emitOff[s + 1] - d->emitOff[s], nN = d->nullOff[s + 1] - d->nullOff[s];
      auto& o = outs[s];
      std::sort(o.begin(), o.end());
      o.erase(std::unique(o.begin(), o.end()), o.end());
      uint32_t w1 = 0;
      for (uint32_t i = 0; i < d->mdl[s]; ++i) w1 |= (uint32_t)(d->ctx[(size_t)s * k + i] & 3u) << (2 * i);
      if (wideOf[s] == 0xFFFFFFFFu) {
        P.blocks.push_back(nE | ((nE + nN) << 8) | ((uint32_t)o.size() << 16) | ((uint32_t)d->mdl[s] << 24));
        P.blocks.push_back(w1);
      } else {
        P.blocks.push_back(kHdrWide | ((uint32_t)d->mdl[s] << 24));
        P.blocks.push_back(w1);
        P.blocks.push_back(nE | ((nE + nN) << 16));
        P.blocks.push_back(wideOf[s]);
      }
      auto pushIn = [&](uint32_t src, uint32_t sym, uint32_t base) {
        const uint32_t sg = P.newOf[src], sr = sg / M;
        P.blocks.push_back(((sg % M) * 8) | (sr << 20) | (sr != rank ? kEdgeRemote : 0u));
        P.blocks.push_back((sym * 8) | ((sym * 128 + base * 32) << 8));
      };
      for (uint32_t e = d->emitOff[s]; e < d->emitOff[s + 1]; ++e) pushIn(d->emitSrc[e], d->emitSym[e], d->emitBase[e]);
      for (uint32_t e = d->nullOff[s]; e < d->nullOff[s + 1]; ++e) pushIn(d->nullSrc[e], d->nullSym[e], 0);
      for (uint32_t dg : o) P.blocks.push_back((dg % M) | ((dg / M) << 20) | (dg / M != rank ? kEdgeRemote : 0u));
    }
    if (P.blocks.size() & 1) P.blocks.push_back(0);
  }
  return DNAB_OK;
}

// Tables of the push kernel for a given partition and CTA size (formats: viterbi_device.cuh).
struct PushTables {
  uint32_t chunkStates = 0, nChunks = 0, maxChunkBytes = 0, maxOutBytes = 0;
  std::vector<uint32_t> inChunks, inChunkOff, outTable, outSliceOff, outOvf;
  std::vector<uint4> outSlots;
};

static int buildPushTables(const dnab_decoder* d, const Partition& P, const std::vector<uint32_t>& wideOf, uint32_t chunkStates,
                           PushTables& T) {
  const uint32_t threads = chunkStates;  // (states per chunk = kPushStatesPerThread * threads per CTA)
  const uint32_t N = d->nStates, k = d->k, C = P.C, M = P.M, Np = C * M;
  std::vector<std::vector<uint32_t>> outs(Np);  // out-edge words, "other CTA" bit added below
  std::vector<char> hasNullOut(N, 0);
  for (uint32_t s = 0; s < N; ++s) {
    const uint32_t dg = P.newOf[s];
    for (uint32_t e = d->emitOff[s]; e < d->emitOff[s + 1]; ++e)
      outs[P.newOf[d->emitSrc[e]]].push_back(peMake(dg % M, dg / M, false, d->emitSym[e], 1));
    for (uint32_t e = d->nullOff[s]; e < d->nullOff[s + 1]; ++e) {
      outs[P.newOf[d->nullSrc[e]]].push_back(peMake(dg % M, dg / M, false, d->nullSym[e], 0));
      hasNullOut[d->nullSrc[e]] = 1;
    }
  }
  T.chunkStates = threads;
  T.nChunks = (M + threads - 1) / threads;
  T.inChunks.clear();
  T.inChunkOff.assign((size_t)C * (T.nChunks + 1), 0);
  T.maxChunkBytes = 0;
  const uint32_t offWords = (threads + 1 + 1) / 2;
  for (uint32_t r = 0; r < C; ++r) {
    for (uint32_t j = 0; j < T.nChunks; ++j) {
      const uint32_t start = (uint32_t)T.inChunks.size();  // multiple of 4 words
      T.inChunkOff[(size_t)r * (T.nChunks + 1) + j] = start;
      T.inChunks.resize(start + offWords, 0);
      std::vector<uint16_t> recOff(threads + 1, 0);
      uint32_t at = 0;
      for (uint32_t t = 0; t < threads; ++t) {
        recOff[t] = (uint16_t)at;
        const uint32_t i = j * threads + t;
        if (i >= M) continue;
        const uint32_t s = P.origOf[r * M + i];
        if (s == 0xFFFFFFFFu) {
          T.inChunks.push_back(kInPad << 7);
          at += 1;
          continue;
        }
        const uint32_t nE = d->emitOff[s + 1] - d->emitOff[s], nN = d->nullOff[s + 1] - d->nullOff[s];
        const bool wide = wideOf[s] != 0xFFFFFFFFu;
        uint32_t h = (wide ? kInWide << 7 : nE | ((nE + nN) << 7)) | ((uint32_t)d->mdl[s] << 15) | ((uint32_t)hasNullOut[s] << 30);
        for (uint32_t i2 = 0; i2 < d->mdl[s]; ++i2) h |= (uint32_t)(d->ctx[(size_t)s * k + i2] & 3u) << (18 + 2 * i2);
        T.inChunks.push_back(h);
        if (wide) {
          T.inChunks.push_back(nE | ((nE + nN) << 16));
          T.inChunks.push_back(wideOf[s]);
          at += 2;
        }
        auto pushIn = [&](uint32_t src, uint32_t sym, uint32_t base) {
          const uint32_t sg = P.newOf[src];
          T.inChunks.push_back(peMake(sg % M, sg / M, sg / M != r, sym, base));
        };
        for (uint32_t e = d->emitOff[s]; e < d->emitOff[s + 1]; ++e) pushIn(d->emitSrc[e], d->emitSym[e], d->emitBase[e]);
        for (uint32_t e = d->nullOff[s]; e < d->nullOff[s + 1]; ++e) pushIn(d->nullSrc[e], d->nullSym[e], 0);
        at += 1 + nE + nN;
        if (at > 65535) {
          setLastError("in-table chunk exceeds 16-bit record offsets; use fewer threads per CTA");
          return DNAB_EINVAL;
        }
      }
      recOff[threads] = (uint16_t)at;
      std::memcpy(&T.inChunks[start], recOff.data(), (threads + 1) * sizeof(uint16_t));
      while (T.inChunks.size() % 4) T.inChunks.push_back(0);
      T.maxChunkBytes = std::max<uint32_t>(T.maxChunkBytes, ((uint32_t)T.inChunks.size() - start) * 4);
    }
    T.inChunkOff[(size_t)r * (T.nChunks + 1) + T.nChunks] = (uint32_t)T.inChunks.size();
  }
  T.outTable.clear();
  T.outSliceOff.assign(C + 1, 0);
  T.maxOutBytes = 0;
  const uint32_t outOffWords = (M + 1 + 1) / 2;
  for (uint32_t r = 0; r < C; ++r) {
    const uint32_t start = (uint32_t)T.outTable.size();
    T.outSliceOff[r] = start;
    T.outTable.resize(start + outOffWords, 0);
    std::vector<uint16_t> off(M + 1, 0);
    uint32_t at = 0;
    for (uint32_t i = 0; i < M; ++i) {
      off[i] = (uint16_t)at;
      for (uint32_t w : outs[r * M + i]) {
        T.outTable.push_back(peRank(w) != r ? (w | (1u << 20)) : w);
        ++at;
      }
      if (at > 65535) {
        setLastError("out-table of one CTA exceeds 16-bit offsets; use a larger cluster");
        return DNAB_EINVAL;
      }
    }
    off[M] = (uint16_t)at;
    std::memcpy(&T.outTable[start], off.data(), (M + 1) * sizeof(uint16_t));
    T.maxOutBytes = std::max<uint32_t>(T.maxOutBytes, ((uint32_t)T.outTable.size() - start) * 4);
  }
  T.outSliceOff[C] = (uint32_t)T.outTable.size();
  // the same lists as 16-byte slots for the CTAs that read their out-table from L2
  T.outSlots.assign(Np, make_uint4(0, 0, 0, 0));
  T.outOvf.clear();
  for (uint32_t g = 0; g < Np; ++g) {
    std::vector<uint32_t> words;
    for (uint32_t w : outs[g]) words.push_back(peRank(w) != g / M ? (w | (1u << 20)) : w);
    uint4& slot = T.outSlots[g];
    slot.x = (uint32_t)words.size();
    if (words.size() <= 3) {
      if (words.size() > 0) slot.y = words[0];
      if (words.size() > 1) slot.z = words[1];
      if (words.size() > 2) slot.w = words[2];
    } else {
      slot.y = (uint32_t)T.outOvf.size();
      T.outOvf.insert(T.outOvf.end(), words.begin(), words.end());
    }
  }
  T.outOvf.resize(T.outOvf.size() + 4, 0);
  return DNAB_OK;
}

// Threads per CTA of the push kernel.
static uint32_t pushThreads(const dnab_decoder* d, uint32_t M) {
  // measured on B200 with one state per thread and step: 1024 threads are best for the large slices (configs 2, 3,
  // 5: 10,746-12,361 states per CTA), 640 for 7,066 states (config 4), 128 for 384 states (config 1)
  const uint32_t threads = d->wantThreads ? d->wantThreads
                           : M <= 1024 ? 128 : M <= 2048 ? 256 : M <= 4096 ? 512 : M <= 8192 ? 640 : 1024;
  return std::max<uint32_t>(32, std::min<uint32_t>(1024, (threads + 31) / 32 * 32));
}

// Plan of the push kernel for reads of up to maxLen bases: cluster size, placements, tables, scratch.  The handle
// keeps its current plan until the new one is complete; a failure after the first upload (which replaces buffers the
// current plan points at) leaves no plan, so the next call builds one from scratch.
static int buildPlan(dnab_decoder* d, int32_t maxLen) {
  if (d->plan.maxLen >= maxLen && d->plan.C) return DNAB_OK;
  const int32_t planLen = std::max(maxLen, 1024);
  const uint32_t N = d->nStates, k = d->k;
  LaunchPlan best;
  Partition P;
  PushTables T;
  std::vector<uint32_t> wideOf;
  uint32_t nWide = 0;
  int wrc = numberWideStates(d, wideOf, nWide);
  if (wrc != DNAB_OK) return wrc;
  std::vector<uint32_t> cands = {1, 2, 3, 4, 5, 6, 7, 8, 10, 12, 14, 16};
  if (d->wantC >= 1 && d->wantC <= (uint32_t)kMaxCluster) cands = {d->wantC};
  // Preference: the smallest cluster whose CTAs hold S and D (more reads in flight beats more SMs per
  // read, and fewer transitions cross CTAs); within it the out-table, then S(pos-1), then the T columns
  // join them in shared memory when they fit.  Measured on B200 with the BASELINE config-2 machine:
  // 4 CTAs per read with the out-table in L2 decode 11% more reads per second than 6 CTAs per read
  // with the out-table in shared memory.
  for (uint32_t C : cands) {
    const uint32_t M = (N + C - 1) / C;
    if (M > 65535) continue;
    const uint32_t threads = pushThreads(d, M);
    if (makePushLayout(M, k, 0, 0, 0, 64, 1, (uint32_t)planLen, 1024).total > d->smemOptin) continue;
    int rc = buildPartition(d, C, wideOf, P);
    if (rc != DNAB_OK) return rc;
    rc = buildPushTables(d, P, wideOf, threads * kPushStatesPerThread, T);
    if (rc != DNAB_OK) {
      if (d->wantC) return rc;
      continue;
    }
    // (out-table in smem, S(pos-1) in smem, T in smem, full-size level queue); a short queue defers states to the next level
    const uint32_t opts[8][4] = {{1, 1, 1, 1}, {1, 1, 0, 1}, {1, 0, 1, 1}, {1, 0, 0, 1}, {1, 0, 0, 0}, {0, 0, 1, 1}, {0, 0, 0, 1}, {0, 0, 0, 0}};
    for (const auto& o : opts) {
      const uint32_t needOut = o[0], sIn = o[1], tIn = (k == 0) ? 0 : o[2];
      uint32_t qCap = o[3] ? M : std::max<uint32_t>(1024, M / 4);
      if (d->queueCap) qCap = std::max<uint32_t>(32, std::min<uint32_t>(qCap, d->queueCap));  // option "queue_cap" (test hook)
      if (d->wantBlockMode == 1 && !needOut) continue;
      if (d->wantBlockMode == 2 && needOut) continue;
      if (d->wantSPrevMode == 1 && !sIn) continue;
      if (d->wantSPrevMode == 2 && sIn) continue;
      if (d->wantTMode == 1 && k && !tIn) continue;
      if (d->wantTMode == 2 && tIn) continue;
      const uint32_t smem =
          makePushLayout(M, k, tIn, sIn, needOut ? T.maxOutBytes : 0, T.maxChunkBytes, T.nChunks, (uint32_t)planLen, qCap).total;
      if (smem <= d->smemOptin) {
        best.C = C;
        best.M = M;
        best.threads = threads;
        best.tInSmem = tIn;
        best.sPrevGlobal = sIn ? 0 : 1;
        best.outInSmem = needOut;
        best.outBytes = needOut ? T.maxOutBytes : 0;
        best.chunkBytes = T.maxChunkBytes;
        best.queueCap = qCap;
        best.smemBytes = smem;
        break;
      }
    }
    if (best.C) break;
  }
  if (!best.C) {
    setLastError("machine does not fit: " + std::to_string(N) +
                 " states need more shared memory than a 16-CTA cluster has (or the requested configuration is infeasible)");
    return DNAB_EINVAL;
  }
  best.maxLen = planLen;
  const uint32_t C = best.C, M = best.M;

  DevTables t{};
  t.nStates = N;
  t.M = M;
  t.C = C;
  t.k = k;
  t.local = d->local;
  t.nSyms = (uint32_t)d->symChar.size();
  t.startG = P.newOf[0];
  t.endG = P.newOf[N - 1];
  t.tInSmem = best.tInSmem;
  t.nWide = nWide;
  t.sPrevInSmem = best.sPrevGlobal ? 0 : 1;
  t.outInSmem = best.outInSmem;
  t.chunkStates = T.chunkStates;
  t.nChunks = T.nChunks;
  t.maxChunkBytes = T.maxChunkBytes;
  t.maxOutBytes = T.maxOutBytes;
  for (int i = 0; i < kMaxSyms; ++i) t.symScore[i] = i < (int)d->symScore.size() ? d->symScore[i] : 0.;
  std::memcpy(t.sub, d->sub, sizeof t.sub);
  std::memcpy(t.len, d->len, sizeof t.len);
  t.noGap = d->noGap;
  t.delOpen = d->delOpen;
  t.delExtend = d->delExtend;
  t.delEnd = d->delEnd;
  t.tanDup = d->tanDup;
  int nClusters = 0;
  CUDA_TRY(queryMaxClustersPush(t, best.threads, best.smemBytes, &nClusters));
  if (nClusters < 1) {
    setLastError("no cluster of size " + std::to_string(C) + " can be resident on this device");
    return DNAB_ECUDA;
  }
  best.nClusters = (uint32_t)nClusters;

  // the uploads replace buffers the current plan points at: from here on a failure leaves no plan
  d->plan = LaunchPlan();
  P.blocks.resize(P.blocks.size() + 8, 0);
  T.inChunks.resize(T.inChunks.size() + 4, 0);
  T.outTable.resize(T.outTable.size() + 4, 0);
  CUDA_TRY(d->dBlocks.upload(P.blocks));
  CUDA_TRY(d->dBlockOff.upload(P.blockOff));
  CUDA_TRY(d->dOrigId.upload(P.origOf));
  CUDA_TRY(d->dSymChar.upload(d->symChar));
  CUDA_TRY(d->dInChunks.upload(T.inChunks));
  CUDA_TRY(d->dInChunkOff.upload(T.inChunkOff));
  CUDA_TRY(d->dOutTable.upload(T.outTable));
  CUDA_TRY(d->dOutSliceOff.upload(T.outSliceOff));
  CUDA_TRY(d->dOutSlots.upload(T.outSlots));
  CUDA_TRY(d->dOutOvf.upload(T.outOvf));
  if (!best.tInSmem && k) CUDA_TRY(d->dTScratch.ensure((size_t)nClusters * C * k * M));
  CUDA_TRY(d->dS0Scratch.ensure((size_t)nClusters * C * M));
  if (best.sPrevGlobal) CUDA_TRY(d->dSScratch.ensure((size_t)nClusters * 2 * C * M));
  t.blocks = d->dBlocks.p;
  t.blockOff = d->dBlockOff.p;
  t.origId = d->dOrigId.p;
  t.symChar = d->dSymChar.p;
  t.inChunks = d->dInChunks.p;
  t.inChunkOff = d->dInChunkOff.p;
  t.outTable = d->dOutTable.p;
  t.outSliceOff = d->dOutSliceOff.p;
  t.outSlots = d->dOutSlots.p;
  t.outOvf = d->dOutOvf.p;
  d->dev = t;
  d->plan = best;
  return DNAB_OK;
}


// ---------------------------------------------------------------------------
// read-batched kernel: partition, tables, scratch (formats: viterbi_batch.h)
// ---------------------------------------------------------------------------
// State partition of the read-batched kernel: T parts of at most cap states with few transitions between parts.
// Greedy graph growing (a part grows from a seed by always taking the unassigned state with the most transitions
// into the part, seeds in depth-first order) followed by capacity-bounded label propagation.  On the BASELINE
// machines it leaves 13-22 % of the transitions between CTAs where equal runs of a depth-first order leave 18-53 %.
static std::vector<uint32_t> growPartition(const dnab_decoder* d, uint32_t T, uint32_t cap, const std::vector<uint32_t>& dfs) {
  const uint32_t N = d->nStates;
  std::vector<uint32_t> off(N + 1, 0), nb;
  auto each = [&](auto&& f) {
    for (uint32_t dst = 0; dst < N; ++dst) {
      for (uint32_t e = d->emitOff[dst]; e < d->emitOff[dst + 1]; ++e)
        if (d->emitSrc[e] != dst) f(d->emitSrc[e], dst);
      for (uint32_t e = d->nullOff[dst]; e < d->nullOff[dst + 1]; ++e)
        if (d->nullSrc[e] != dst) f(d->nullSrc[e], dst);
    }
  };
  each([&](uint32_t a, uint32_t b) {
    ++off[a + 1];
    ++off[b + 1];
  });
  for (uint32_t s = 0; s < N; ++s) off[s + 1] += off[s];
  nb.resize(off[N]);
  std::vector<uint32_t> fill(off.begin(), off.end() - 1);
  each([&](uint32_t a, uint32_t b) {
    nb[fill[a]++] = b;
    nb[fill[b]++] = a;
  });
  const uint32_t none = 0xFFFFFFFFu;
  std::vector<uint32_t> part(N, none), conn(N, 0), size(T, 0);
  const uint32_t target = (N + T - 1) / T;
  uint32_t ptr = 0;
  for (uint32_t p = 0; p < T; ++p) {
    const uint32_t quota = p + 1 < T ? target : cap;
    std::vector<std::pair<uint32_t, uint32_t>> heap;  // (connections into the part, state), max-heap
    std::vector<uint32_t> touched;
    while (size[p] < quota) {
      if (heap.empty()) {
        while (ptr < N && part[dfs[ptr]] != none) ++ptr;
        if (ptr >= N) break;
        heap.push_back({0u, dfs[ptr]});
      }
      std::pop_heap(heap.begin(), heap.end());
      const auto top = heap.back();
      heap.pop_back();
      const uint32_t v = top.second;
      if (part[v] != none || top.first != conn[v]) continue;  // stale entry
      part[v] = p;
      ++size[p];
      for (uint32_t e = off[v]; e < off[v + 1]; ++e) {
        const uint32_t u = nb[e];
        if (part[u] != none) continue;
        if (!conn[u]) touched.push_back(u);
        ++conn[u];
        heap.push_back({conn[u], u});
        std::push_heap(heap.begin(), heap.end());
      }
    }
    for (uint32_t u : touched) conn[u] = 0;
  }
  for (uint32_t s = 0; s < N; ++s)
    if (part[s] == none) {  // leftovers (cannot happen with cap >= target): the emptiest part
      const uint32_t p = (uint32_t)(std::min_element(size.begin(), size.end()) - size.begin());
      part[s] = p;
      ++size[p];
    }
  std::vector<uint32_t> cnt(T, 0), seenParts;
  for (int sweep = 0; sweep < 8; ++sweep) {
    uint32_t moved = 0;
    for (uint32_t s = 0; s < N; ++s) {
      seenParts.clear();
      for (uint32_t e = off[s]; e < off[s + 1]; ++e) {
        const uint32_t p = part[nb[e]];
        if (!cnt[p]++) seenParts.push_back(p);
      }
      const uint32_t cur = part[s];
      uint32_t best = cur, bc = cnt[cur];
      for (uint32_t p : seenParts)
        if (cnt[p] > bc && size[p] < cap) {
          best = p;
          bc = cnt[p];
        }
      for (uint32_t p : seenParts) cnt[p] = 0;
      if (best != cur) {
        --size[cur];
        ++size[best];
        part[s] = best;
        ++moved;
      }
    }
    if (moved * 500 < N) break;
  }
  return part;
}

static bool batchWanted(const dnab_decoder* d) {
  if (d->wantBatch == 0) return false;
  if (d->wantBatch == 1) return true;
  // automatic: the batched kernel, unless the caller tuned the one-read-per-cluster push kernel explicitly
  return !(d->wantC || d->wantThreads || d->wantTMode || d->wantBlockMode || d->wantSPrevMode || d->wantPartition);
}

// Plan of the read-batched kernel.  It depends on the options only, so the answer "infeasible" is kept until an option
// changes.  The plan is built in locals and committed at the end; a failure after the first upload leaves no plan.
static int buildBatchPlan(dnab_decoder* d) {
  if (d->bplan.ready) {
    if (!d->bplan.feasible) setLastError("the read-batched kernel cannot take this machine");
    return d->bplan.feasible ? DNAB_OK : DNAB_EINVAL;
  }
  d->bplan.ready = true;  // infeasible until committed below
  BatchPlan bp;
  BatchTables t{};
  const uint32_t N = d->nStates, k = d->k;
  // warps per CTA (measured on B200): 24 when one CTA holds the group (80 registers, no spills: 349k vs 315k reads/s on
  // dnastore-l4), 32 in a team (more states relaxed side by side per level: 1,120 vs 1,060 reads/s on the 46,670-state machine)
  const uint32_t wantW = d->wantWarps ? (d->wantWarps > 24 ? 32u : d->wantWarps > 16 ? 24u : 16u) : 0u;
  uint32_t W = wantW ? wantW : 24u;
  auto nEmitOf = [&](uint32_t s) { return d->emitOff[s + 1] - d->emitOff[s]; };
  auto nNullOf = [&](uint32_t s) { return d->nullOff[s + 1] - d->nullOff[s]; };
  std::vector<uint32_t> wideOf;
  uint32_t nWide = 0;
  {
    const int rc = numberWideStates(d, wideOf, nWide);
    if (rc != DNAB_OK) return rc;
  }
  // successors of every state with the bit they own in the successor's work mask
  std::vector<std::vector<std::pair<uint32_t, uint32_t>>> outs(N);
  for (uint32_t dst = 0; dst < N; ++dst) {
    uint32_t j = 0;
    for (uint32_t e = d->emitOff[dst]; e < d->emitOff[dst + 1]; ++e, ++j) outs[d->emitSrc[e]].push_back({dst, j});
    for (uint32_t e = d->nullOff[dst]; e < d->nullOff[dst + 1]; ++e, ++j) outs[d->nullSrc[e]].push_back({dst, j});
  }
  const std::vector<uint32_t> dfs = dfsOrder(d);
  const uint32_t nSymsB = (uint32_t)d->symChar.size();
  const uint32_t maxTeam = (uint32_t)d->smCount;
  uint32_t T0 = std::max<uint32_t>(1, (uint32_t)(((size_t)N * kBatchReads * 16 + d->smemOptin - 1) / d->smemOptin));
  std::vector<uint4> hdr, wideHdr(nWide);
  std::vector<uint2> inE, relE, hdr2;
  std::vector<uint32_t> outE, rankInOff, rankOutOff, newOf(N), origOf, remoteIn, clsOff, clsStates, clsOf;
  // builds the tables of a team of T CTAs; false when T is infeasible
  auto buildTeam = [&](uint32_t T, uint32_t M) -> bool {
    W = wantW ? wantW : (T > 1 ? 32u : 24u);
    const uint32_t Np = T * M;
    if (M > kBatchMaxSlots * W || M > 65535 || T > 1023) return false;
    if (makeBatchLayout(M, 0, 0, nSymsB, T > 1).total > d->smemOptin) return false;
    // CTA assignment (T > 1): growPartition; inside a CTA descending in-degree, dealt to the warps
    std::vector<uint32_t> part;
    if (T > 1) part = growPartition(d, T, M, dfs);
    std::vector<std::vector<uint32_t>> members(T);
    for (uint32_t s = 0; s < N; ++s) members[T > 1 ? part[s] : 0].push_back(s);
    origOf.assign(Np, 0xFFFFFFFFu);
    for (uint32_t r = 0; r < T; ++r) {
      std::vector<uint32_t>& mine = members[r];
      if (mine.size() > M) return false;
      std::stable_sort(mine.begin(), mine.end(),
                       [&](uint32_t a, uint32_t b) { return nEmitOf(a) + nNullOf(a) > nEmitOf(b) + nNullOf(b); });
      for (uint32_t j = 0; j < mine.size(); ++j) {
        origOf[r * M + j] = mine[j];
        newOf[mine[j]] = r * M + j;
      }
    }
    hdr.assign(Np, make_uint4(0, 0, 1u << 17, 0xFFFFFFFFu));
    hdr2.assign(Np, make_uint2(0, 0));
    remoteIn.assign(Np, 0);
    // position of every in-transition in its destination's relax list: local emit, local null, remote emit, remote null
    std::vector<std::vector<uint32_t>> relPos(N);
    for (uint32_t dst = 0; dst < N; ++dst) {
      const uint32_t nE = nEmitOf(dst), nIn = nE + nNullOf(dst), rD = newOf[dst] / M;
      std::vector<uint32_t> key(nIn), idx(nIn);
      for (uint32_t j = 0; j < nIn; ++j) {
        const uint32_t src = j < nE ? d->emitSrc[d->emitOff[dst] + j] : d->nullSrc[d->nullOff[dst] + (j - nE)];
        key[j] = (newOf[src] / M != rD ? 2u : 0u) + (j < nE ? 0u : 1u);
        idx[j] = j;
      }
      std::stable_sort(idx.begin(), idx.end(), [&](uint32_t a, uint32_t b) { return key[a] < key[b]; });
      relPos[dst].resize(nIn);
      for (uint32_t q = 0; q < nIn; ++q) relPos[dst][idx[q]] = q;
    }
    // notification classes (T > 1): the states of a CTA that have a transition from another CTA are dealt round-robin into
    // `notifyClasses` classes (1 = every notification wakes all of them)
    clsOf.assign(Np, 0);
    clsOff.assign((size_t)T * (kNotifyClasses + 1), 0);
    clsStates.assign(Np, 0);
    for (uint32_t r = 0; r < T; ++r) {
      std::vector<std::vector<uint32_t>> byClass(kNotifyClasses);
      uint32_t ord = 0;
      for (uint32_t i = 0; i < M; ++i) {
        const uint32_t s = origOf[r * M + i];
        if (s == 0xFFFFFFFFu) continue;
        bool remoteIn = false;
        for (uint32_t e = d->emitOff[s]; e < d->emitOff[s + 1]; ++e) remoteIn |= newOf[d->emitSrc[e]] / M != r;
        for (uint32_t e = d->nullOff[s]; e < d->nullOff[s + 1]; ++e) remoteIn |= newOf[d->nullSrc[e]] / M != r;
        if (!remoteIn) continue;
        const uint32_t c = (ord++) % std::max(1u, std::min(d->notifyClasses, kNotifyClasses));
        clsOf[r * M + i] = c;
        byClass[c].push_back(i);
      }
      uint32_t at = 0;
      for (uint32_t c = 0; c < kNotifyClasses; ++c) {
        clsOff[(size_t)r * (kNotifyClasses + 1) + c] = at;
        for (uint32_t i : byClass[c]) clsStates[r * M + at++] = i;
      }
      clsOff[(size_t)r * (kNotifyClasses + 1) + kNotifyClasses] = at;
    }
    inE.clear();
    relE.clear();

    outE.clear();
    rankInOff.assign(T + 1, 0);
    rankOutOff.assign(T + 1, 0);
    uint32_t maxIn = 0, maxOut = 0;
    uint64_t cross = 0, total = 0;
    for (uint32_t r = 0; r < T; ++r) {
      rankInOff[r] = (uint32_t)inE.size();
      rankOutOff[r] = (uint32_t)outE.size();
      for (uint32_t i = 0; i < M; ++i) {
        const uint32_t s = origOf[r * M + i];
        if (s == 0xFFFFFFFFu) continue;
        const uint32_t inOff = (uint32_t)inE.size() - rankInOff[r], outOff = (uint32_t)outE.size() - rankOutOff[r];
        if (inOff > 65535 || outOff > 65535) return false;
        const uint32_t nE = nEmitOf(s), nN = nNullOf(s);
        uint32_t jIn = 0;
        auto pushIn = [&](uint32_t src, uint32_t sym, uint32_t base) {
          const uint32_t sg = newOf[src];
          const bool remote = sg / M != r;
          inE.push_back(make_uint2(sg, sym | (base << 5) | (remote ? 1u << 7 : 0u)));
          ++jIn;
          ++total;
          cross += remote;
        };
        for (uint32_t e = d->emitOff[s]; e < d->emitOff[s + 1]; ++e) pushIn(d->emitSrc[e], d->emitSym[e], d->emitBase[e]);
        for (uint32_t e = d->nullOff[s]; e < d->nullOff[s + 1]; ++e) pushIn(d->nullSrc[e], d->nullSym[e], 0);
        {
          // the closure's copy, in relax order
          const uint32_t nInS = nE + nN, base = (uint32_t)relE.size();
          relE.resize(base + nInS);
          uint32_t cnt[4] = {0, 0, 0, 0};
          remoteIn[r * M + i] = 0;
          for (uint32_t j = 0; j < nInS; ++j) {
            const uint32_t src = j < nE ? d->emitSrc[d->emitOff[s] + j] : d->nullSrc[d->nullOff[s] + (j - nE)];
            const uint32_t sym = j < nE ? d->emitSym[d->emitOff[s] + j] : d->nullSym[d->nullOff[s] + (j - nE)];
            const bool remote = newOf[src] / M != r;
            ++cnt[(remote ? 2 : 0) + (j < nE ? 0 : 1)];
            relE[base + relPos[s][j]] = make_uint2(newOf[src], sym * 8);
            if (remote) remoteIn[r * M + i] |= 1u << std::min(relPos[s][j], 31u);
          }
          if (wideOf[s] == 0xFFFFFFFFu)
            hdr2[r * M + i] = make_uint2(base - rankInOff[r], cnt[0] | (cnt[1] << 8) | (cnt[2] << 16) | (cnt[3] << 24));
          else {
            hdr2[r * M + i] = make_uint2(base - rankInOff[r], 0);
            wideHdr[wideOf[s]] = make_uint4(nE | (nN << 16), cnt[0] | (cnt[1] << 16), cnt[2] | (cnt[3] << 16), 0);
          }
        }
        bool remoteOut = (d->local && s == 0 && T > 1);  // local mode: every CTA reads S(start,0) for the (0,0) escape
        uint32_t nLocal = 0;
        std::vector<uint32_t> remoteNotes;
        for (const auto& o : outs[s]) {  // successors in this CTA first, then the (CTA, class) pairs that own the others
          const uint32_t dg = newOf[o.first];
          const uint32_t bit = std::min(relPos[o.first][o.second], 31u);
          if (dg / M != r) {
            remoteOut = true;
            remoteNotes.push_back((dg / M) * kNotifyClasses + clsOf[dg]);
            continue;
          }
          ++nLocal;
          outE.push_back((dg % M) | (bit << 16));
        }
        std::sort(remoteNotes.begin(), remoteNotes.end());
        remoteNotes.erase(std::unique(remoteNotes.begin(), remoteNotes.end()), remoteNotes.end());
        outE.insert(outE.end(), remoteNotes.begin(), remoteNotes.end());
        const uint32_t nOutEntries = nLocal + (uint32_t)remoteNotes.size();  // (<= outgoing transitions: 255 when narrow)
        uint32_t ctxBits = 0;
        for (uint32_t t = 0; t < d->mdl[s]; ++t) ctxBits |= (uint32_t)(d->ctx[(size_t)s * k + t] & 3u) << (2 * t);
        if (wideOf[s] == 0xFFFFFFFFu)
          hdr[r * M + i] = make_uint4(inOff | (outOff << 16), nE | (nN << 8) | (nOutEntries << 16) | ((uint32_t)d->mdl[s] << 24),
                                      ctxBits | (remoteOut ? 1u << 16 : 0u) | (nLocal << 18), s);
        else {
          hdr[r * M + i] = make_uint4(inOff | (outOff << 16), wideOf[s] | ((uint32_t)d->mdl[s] << 24) | kBhWide,
                                      ctxBits | (remoteOut ? 1u << 16 : 0u), s);
          wideHdr[wideOf[s]].w = nLocal | (nOutEntries << 16);
        }
      }
      maxIn = std::max(maxIn, (uint32_t)inE.size() - rankInOff[r]);
      maxOut = std::max(maxOut, (uint32_t)outE.size() - rankOutOff[r]);
    }
    rankInOff[T] = (uint32_t)inE.size();
    rankOutOff[T] = (uint32_t)outE.size();
    const uint32_t smem = makeBatchLayout(M, maxIn, maxOut, nSymsB, T > 1).total;
    if (smem > d->smemOptin) return false;
    bp.T = T;
    bp.M = M;
    bp.warps = W;
    bp.smemBytes = smem;
    bp.crossFraction = total ? (double)cross / (double)total : 0.;
    t = BatchTables{};
    t.nStates = N;
    t.M = M;
    t.T = T;
    t.k = k;
    t.local = d->local;
    t.nSyms = (uint32_t)d->symChar.size();
    t.startRank = newOf[0] / M;
    t.startLocal = newOf[0] % M;
    t.endRank = newOf[N - 1] / M;
    t.endLocal = newOf[N - 1] % M;
    t.maxIn = maxIn;
    t.maxOut = maxOut;
    return true;
  };
  // states per CTA: the balanced share plus 8 % (then 4 %, then nothing) so that the partitioner can trade balance for
  // fewer transitions between CTAs, as long as columns, tables and the cache of remote rows still fit
  auto tryTeam = [&](uint32_t T) -> bool {
    const uint32_t Mbal = (N + T - 1) / T;
    if (T == 1) return buildTeam(1, Mbal);
    uint32_t last = 0;
    for (uint32_t pct : {d->teamSlackPct, d->teamSlackPct / 2, 0u}) {
      const uint32_t M = std::min<uint32_t>(Mbal + (Mbal * pct + 99) / 100, kBatchMaxSlots * 16u);
      if (M == last) continue;
      last = M;
      if (buildTeam(T, M)) return true;
    }
    return false;
  };
  if (d->wantTeam)
    bp.feasible = tryTeam(d->wantTeam);
  else {
    uint32_t Tmin = 0;
    for (uint32_t T = T0; T <= maxTeam && !Tmin; ++T)
      if (tryTeam(T)) Tmin = T;
    if (Tmin) {
      bp.feasible = true;
      // the teams that fit at once get all the SMs: fewer states per CTA, the same reads in flight
      const uint32_t spread = maxTeam / (maxTeam / Tmin);
      if (spread > Tmin && !tryTeam(spread)) bp.feasible = tryTeam(Tmin);
    }
  }
  if (!bp.feasible) {
    setLastError("the read-batched kernel cannot take this machine: " + std::to_string(N) +
                 " states x 32 reads x 16 bytes exceed the shared memory of " + std::to_string(maxTeam) + " SMs");
    return DNAB_EINVAL;
  }
  for (int i = 0; i < kMaxSyms; ++i) {
    const double sc = i < (int)d->symScore.size() ? d->symScore[i] : 0.;
    t.symScore[i] = sc;
    t.tsDext[i] = sc + d->delExtend;  // src/viterbi.cpp:272
    t.tsDopen[i] = sc + d->delOpen;   // src/viterbi.cpp:273
  }
  for (int i = 0; i < 8; ++i) {
    t.len[i] = i < kMaxK ? d->len[i] : 0.;
    t.tsT[i] = d->tanDup + t.len[i];  // src/viterbi.cpp:286
  }
  std::memcpy(t.sub, d->sub, sizeof t.sub);
  t.noGap = d->noGap;
  t.delOpen = d->delOpen;
  t.delExtend = d->delExtend;
  t.delEnd = d->delEnd;
  t.tanDup = d->tanDup;
  int perSm = 0;
  CUDA_TRY(queryBatchTeams(t, bp.warps, bp.smemBytes, &perSm));
  if (perSm < 1) {
    setLastError("the read-batched kernel does not fit an SM");
    return DNAB_ECUDA;
  }
  bp.ctasPerSm = (uint32_t)perSm;
  bp.nTeams = (uint32_t)d->smCount * bp.ctasPerSm / bp.T;
  if (bp.nTeams < 1) {
    setLastError("a team of " + std::to_string(bp.T) + " CTAs cannot be resident at once");
    return DNAB_EINVAL;
  }

  // a failure from here on says nothing about the machine: it leaves no plan, and the next call tries again
  d->bplan = BatchPlan();
  inE.push_back(make_uint2(0, 0));
  outE.push_back(0);
  relE.push_back(make_uint2(0, 0));
  // score tables with the traceback's association, formed once on the host in IEEE fp64 (-ffp-contract=off)
  std::vector<double> tsE((size_t)kMaxSyms * 16, 0.);
  for (uint32_t sym = 0; sym < d->symScore.size(); ++sym)
    for (uint32_t b = 0; b < 4; ++b)
      for (uint32_t x = 0; x < 4; ++x) {
        volatile double a = d->symScore[sym] + d->noGap;  // (score + noGap) + sub, src/viterbi.cpp:255
        tsE[(sym * 4 + b) * 4 + x] = a + d->sub[b * 4 + x];
      }
  CUDA_TRY(d->dbHdr.upload(hdr));
  CUDA_TRY(d->dbIn.upload(inE));
  CUDA_TRY(d->dbRel.upload(relE));
  CUDA_TRY(d->dbHdr2.upload(hdr2));
  CUDA_TRY(d->dbOut.upload(outE));
  CUDA_TRY(d->dbRankInOff.upload(rankInOff));
  CUDA_TRY(d->dbRankOutOff.upload(rankOutOff));
  CUDA_TRY(d->dbRemoteIn.upload(remoteIn));
  CUDA_TRY(d->dbClsOff.upload(clsOff));
  CUDA_TRY(d->dbClsStates.upload(clsStates));
  CUDA_TRY(d->dbTsE.upload(tsE));
  if (nWide) {
    CUDA_TRY(d->dbWide.upload(wideHdr));
    CUDA_TRY(d->dbWideOf.upload(wideOf));
  }
  // traceback tables in reference order
  CUDA_TRY(d->dbEmitOff.upload(d->emitOff));
  CUDA_TRY(d->dbEmitSrc.upload(d->emitSrc));
  CUDA_TRY(d->dbEmitSym.upload(d->emitSym));
  CUDA_TRY(d->dbNullOff.upload(d->nullOff));
  CUDA_TRY(d->dbNullSrc.upload(d->nullSrc));
  CUDA_TRY(d->dbNullSym.upload(d->nullSym));
  CUDA_TRY(d->dSymChar.upload(d->symChar));
  const size_t Np = (size_t)bp.T * bp.M;
  CUDA_TRY(d->dbPriv.ensure((size_t)bp.nTeams * Np * (2 + k) * 32));
  {
    // L2 set-aside for the carried rows (DESIGN.md 4): as much of them as the device lets a window and the set-aside hold
    cudaDeviceProp prop{};
    d->persistBytes = 0;
    if (d->wantPersist && cudaGetDeviceProperties(&prop, d->device) == cudaSuccess && prop.persistingL2CacheMaxSize > 0) {
      const size_t want = d->dbPriv.n * sizeof(double);
      const size_t setAside = std::min<size_t>(want, (size_t)prop.persistingL2CacheMaxSize);
      if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, setAside) == cudaSuccess)
        d->persistBytes = std::min<size_t>(setAside, (size_t)prop.accessPolicyMaxWindowSize);
      else
        cudaGetLastError();
    }
  }
  CUDA_TRY(d->dbSdPub.ensure(bp.T > 1 ? (size_t)bp.nTeams * 2 * Np * 32 : 1));
  CUDA_TRY(d->dbTeamState.ensure((size_t)bp.nTeams * bp.T * kNotifyClasses));
  CUDA_TRY(d->dbTeamPassive.ensure((size_t)bp.nTeams * 2));
  CUDA_TRY(d->dbBarrier.ensure((size_t)bp.nTeams));
  t.hdr = d->dbHdr.p;
  t.inEdges = d->dbIn.p;
  t.outEdges = d->dbOut.p;
  t.rankInOff = d->dbRankInOff.p;
  t.rankOutOff = d->dbRankOutOff.p;
  t.remoteIn = d->dbRemoteIn.p;
  t.clsOff = d->dbClsOff.p;
  t.clsStates = d->dbClsStates.p;
  t.hdr2 = d->dbHdr2.p;
  t.relEdges = d->dbRel.p;
  t.tsE = d->dbTsE.p;
  t.nWide = nWide;
  t.wide = nWide ? d->dbWide.p : nullptr;
  BatchTraceTables tt{};
  tt.nStates = N;
  tt.k = k;
  tt.local = d->local;
  tt.T = bp.T * bp.warps;
  tt.nWide = nWide;
  tt.wideOf = nWide ? d->dbWideOf.p : nullptr;
  tt.emitOff = d->dbEmitOff.p;
  tt.emitSrc = d->dbEmitSrc.p;
  tt.emitSym = d->dbEmitSym.p;
  tt.nullOff = d->dbNullOff.p;
  tt.nullSrc = d->dbNullSrc.p;
  tt.nullSym = d->dbNullSym.p;
  tt.symChar = d->dSymChar.p;
  d->btab = t;
  d->btrace = tt;
  bp.ready = true;
  d->bplan = bp;
  return DNAB_OK;
}

// The (start, mid, end) events of one fill + traceback launch pair: the handle's own triple when the caller times the
// call itself (host-buffer path), a triple from the pool when device-path timing is on (resolved in get_stats).
static cudaError_t takeEvents(dnab_decoder* d, bool timeIt, cudaEvent_t ev[3], bool* rec) {
  ev[0] = d->ev0;
  ev[1] = d->ev1;
  ev[2] = d->ev2;
  const bool pooled = d->timing && !timeIt;
  if (pooled) {
    while (d->evPool.size() < d->evUsed + 3) {
      cudaEvent_t e;
      const cudaError_t err = cudaEventCreate(&e);
      if (err != cudaSuccess) return err;
      d->evPool.push_back(e);
    }
    for (int i = 0; i < 3; ++i) ev[i] = d->evPool[d->evUsed + i];
    d->evUsed += 3;
  }
  *rec = timeIt || pooled;
  return cudaSuccess;
}

// fill + traceback with the read-batched kernel
static int runDeviceBatch(dnab_decoder* d, int64_t nReads, int32_t maxLen, const uint8_t* dPacked, const int64_t* dByteOff,
                          const int32_t* dReadLen, double* dLoglike, char* dDecoded, int32_t decodedStride,
                          int32_t* dDecodedLen, int32_t* dStatus, int32_t* dPath, int32_t pathStride, int32_t* dPathLen,
                          double* dCells, cudaStream_t stream, bool timeIt) {
  const BatchPlan& bp = d->bplan;
  const uint32_t N = d->nStates, K2 = d->k + 2;
  const int64_t nGroups = (nReads + 31) / 32;
  const size_t perGroupWide = (size_t)(maxLen + 1) * d->btab.nWide * 2 * 32;  // the side plane (wide states only)
  const size_t perGroup = (size_t)(maxLen + 1) * N * K2 * 32;
  int64_t chunk = (int64_t)std::max<size_t>(1, d->predBudgetBytes / (perGroup + perGroupWide));
  chunk = std::min<int64_t>(chunk, nGroups);
  CUDA_TRY(d->dPred.ensure((size_t)chunk * perGroup));
  if (perGroupWide) CUDA_TRY(d->dPredWide.ensure((size_t)chunk * perGroupWide));
  if (d->local) {
    CUDA_TRY(d->dbPartVal.ensure((size_t)chunk * bp.T * bp.warps * 32));
    CUDA_TRY(d->dbPartOrig.ensure((size_t)chunk * bp.T * bp.warps * 32));
  }
  const int32_t* dOrder = nullptr;
  if (!dCells && nReads > 32) {
    // groups of similar length, formed on the device from dReadLen: a group runs for as many columns as its longest read
    const size_t nSlots = (size_t)nGroups * 32;
    CUDA_TRY(d->dbOrder.ensure(nSlots + (size_t)maxLen + 1));  // the order, then the sort's bins
    CUDA_TRY(launchLengthOrder(dReadLen, nReads, maxLen, (int64_t)nSlots, d->dbOrder.p,
                               reinterpret_cast<uint32_t*>(d->dbOrder.p + nSlots), stream));
    d->stats.kernel_launches += 1;
    dOrder = d->dbOrder.p;
  }
  for (int64_t at = 0; at < nGroups; at += chunk) {
    const int64_t n = std::min(chunk, nGroups - at);
    BatchArgs a{};
    a.nReads = nReads;
    a.readBase = at * 32;
    a.nGroups = n;
    a.nTeams = (uint32_t)std::min<int64_t>(bp.nTeams, n);
    a.maxLen = maxLen;
    // automatic (2) = no level barriers, in a team and in a single CTA alike; the numbers of DESIGN.md 6 were measured so
    a.asyncClosure = d->asyncClosure == 2 ? 1u : d->asyncClosure;
    a.idleNs = d->batchIdleNs;
    a.packed = dPacked;
    a.byteOff = dByteOff;
    a.readLen = dReadLen;
    a.order = dOrder ? dOrder + at * 32 : nullptr;
    a.pred = d->dPred.p;
    a.predWide = perGroupWide ? d->dPredWide.p : nullptr;
    a.priv = d->dbPriv.p;
    a.sdPub = d->dbSdPub.p;
    a.teamState = d->dbTeamState.p;
    a.eagerNotify = d->eagerNotify;
    a.teamPassive = d->dbTeamPassive.p;
    a.barrier = d->dbBarrier.p;
    a.loglike = dLoglike;
    a.partVal = d->dbPartVal.p;
    a.partOrig = d->dbPartOrig.p;
    a.cells = at == 0 ? dCells : nullptr;
    a.dbg = d->debug ? d->dDbg.p : nullptr;
    cudaEvent_t ev[3];
    bool rec = false;
    CUDA_TRY(takeEvents(d, timeIt, ev, &rec));
    if (bp.T > 1) {
      CUDA_TRY(cudaMemsetAsync(d->dbTeamState.p, 0, d->dbTeamState.n * sizeof(uint32_t), stream));
      CUDA_TRY(cudaMemsetAsync(d->dbTeamPassive.p, 0, d->dbTeamPassive.n * sizeof(uint32_t), stream));
      CUDA_TRY(cudaMemsetAsync(d->dbBarrier.p, 0, d->dbBarrier.n * sizeof(unsigned long long), stream));
    }
    if (rec) CUDA_TRY(cudaEventRecord(ev[0], stream));
    CUDA_TRY(launchFillBatch(d->btab, a, bp.warps, bp.smemBytes, stream, d->persistBytes));
    if (rec) CUDA_TRY(cudaEventRecord(ev[1], stream));
    BatchTraceArgs ta{};
    ta.nSlots = n * 32;
    ta.maxLen = maxLen;
    ta.readLen = dReadLen;
    ta.order = a.order;
    ta.nReads = nReads;
    ta.readBase = a.readBase;
    ta.pred = d->dPred.p;
    ta.predWide = a.predWide;
    ta.loglike = dLoglike;
    ta.partVal = d->dbPartVal.p;
    ta.partOrig = d->dbPartOrig.p;
    ta.decoded = dDecoded;
    ta.decodedStride = decodedStride;
    ta.decodedLen = dDecodedLen;
    ta.status = dStatus;
    ta.path = dPath;
    ta.pathStride = pathStride;
    ta.pathLen = dPathLen;
    CUDA_TRY(launchTracebackBatch(d->btrace, ta, stream));
    if (rec) CUDA_TRY(cudaEventRecord(ev[2], stream));
    d->stats.kernel_launches += 2;
    d->stats.fill_launches += 1;
    d->stats.traceback_launches += 1;
  }
  d->stats.reads += (uint64_t)nReads;
  return DNAB_OK;
}

static size_t predBytesPerRead(const dnab_decoder* d, int32_t maxLen) {
  return (size_t)(maxLen + 1) * (d->k + 2) * (size_t)d->plan.C * d->plan.M;
}
static size_t predWideBytesPerRead(const dnab_decoder* d, int32_t maxLen) { return (size_t)(maxLen + 1) * 2 * d->dev.nWide; }

// fill + traceback over device-resident inputs/outputs, chunked so that the
// predecessor records of one chunk fit the scratch budget
static int runDevice(dnab_decoder* d, int64_t nReads, int32_t maxLen, const uint8_t* dPacked, const int64_t* dByteOff,
                     const int32_t* dReadLen, double* dLoglike, char* dDecoded, int32_t decodedStride,
                     int32_t* dDecodedLen, int32_t* dStatus, int32_t* dPath, int32_t pathStride, int32_t* dPathLen,
                     double* dCells, cudaStream_t stream, bool timeIt) {
  if (nReads <= 0) return DNAB_OK;
  CUDA_TRY(cudaSetDevice(d->device));
  if (batchWanted(d)) {
    // Automatic choice (measured on B200, DESIGN.md 5.3, 6): the read-batched kernel when the group's columns fit ONE CTA
    // (2x the one-read-per-cluster kernel on dnastore-l4) and when the push kernel would need a cluster of 4 or more CTAs
    // per read (the 46,670-state machine: a 148-CTA team decodes 1,120 reads/s, 33 clusters of 4 decode 1,010); machines in
    // between (7-12k states, one CTA per read in the push kernel) stay on the push kernel -- a team over L2 pays ~3 us per
    // cross-CTA hop of their long, thin deletion chains (3.3k vs 7.1k reads/s on watermark64.1*l4).
    int brc = buildBatchPlan(d);
    bool use = brc == DNAB_OK;
    if (use && d->wantBatch != 1 && d->bplan.T > 1 && buildPlan(d, maxLen) == DNAB_OK && d->plan.C < 4) use = false;
    if (use)
      return runDeviceBatch(d, nReads, maxLen, dPacked, dByteOff, dReadLen, dLoglike, dDecoded, decodedStride, dDecodedLen,
                            dStatus, dPath, pathStride, dPathLen, dCells, stream, timeIt);
    if (d->wantBatch == 1) return brc;
  }
  int rc = buildPlan(d, maxLen);
  if (rc != DNAB_OK) return rc;
  const size_t perRead = predBytesPerRead(d, maxLen), perReadWide = predWideBytesPerRead(d, maxLen);
  int64_t chunk = (int64_t)std::max<size_t>(1, d->predBudgetBytes / (perRead + perReadWide));
  chunk = std::min<int64_t>(chunk, nReads);
  CUDA_TRY(d->dPred.ensure((size_t)chunk * perRead));
  if (perReadWide) CUDA_TRY(d->dPredWide.ensure((size_t)chunk * perReadWide));
  CUDA_TRY(d->dStart.ensure((size_t)chunk));
  if (d->local) {
    CUDA_TRY(d->dPartVal.ensure((size_t)chunk * d->plan.C));
    CUDA_TRY(d->dPartOrig.ensure((size_t)chunk * d->plan.C));
    CUDA_TRY(d->dPartG.ensure((size_t)chunk * d->plan.C));
  }
  for (int64_t at = 0; at < nReads; at += chunk) {
    const int64_t n = std::min(chunk, nReads - at);
    FillArgs fa{};
    fa.play = makePushLayout(d->plan.M, d->k, d->plan.tInSmem, d->plan.sPrevGlobal ? 0 : 1, d->plan.outBytes,
                             d->plan.chunkBytes, d->dev.nChunks, (uint32_t)d->plan.maxLen, d->plan.queueCap);
    fa.nReads = n;
    fa.thinN = d->thinN;
    fa.tRecompute = d->tRecompute;
    fa.maxLen = maxLen;
    fa.packed = dPacked;
    fa.byteOff = dByteOff + at;
    fa.readLen = dReadLen + at;
    fa.pred = d->dPred.p;
    fa.predWide = perReadWide ? d->dPredWide.p : nullptr;
    fa.tScratch = d->dTScratch.p;
    fa.sScratch = d->dSScratch.p;
    fa.s0Scratch = d->dS0Scratch.p;
    fa.loglike = dLoglike + at;
    fa.startState = d->dStart.p;
    fa.partVal = d->dPartVal.p;
    fa.partOrig = d->dPartOrig.p;
    fa.partG = d->dPartG.p;
    fa.cells = at == 0 ? dCells : nullptr;
    fa.dbg = d->debug ? d->dDbg.p : nullptr;
    const uint32_t nClusters = (uint32_t)std::min<int64_t>(d->plan.nClusters, n);
    cudaEvent_t ev[3];
    bool rec = false;
    CUDA_TRY(takeEvents(d, timeIt, ev, &rec));
    if (rec) CUDA_TRY(cudaEventRecord(ev[0], stream));
    CUDA_TRY(d->dNextRead.ensure(1));
    CUDA_TRY(cudaMemsetAsync(d->dNextRead.p, 0, sizeof(unsigned long long), stream));
    fa.nextRead = d->dNextRead.p;
    CUDA_TRY(launchFillPush(d->dev, fa, nClusters, d->plan.threads, d->plan.smemBytes, stream));
    if (rec) CUDA_TRY(cudaEventRecord(ev[1], stream));
    TracebackArgs ta{};
    ta.nReads = n;
    ta.maxLen = maxLen;
    ta.readLen = dReadLen + at;
    ta.pred = d->dPred.p;
    ta.predWide = fa.predWide;
    ta.loglike = dLoglike + at;
    ta.startState = d->dStart.p;
    ta.partVal = d->dPartVal.p;
    ta.partOrig = d->dPartOrig.p;
    ta.partG = d->dPartG.p;
    ta.decoded = dDecoded + (size_t)at * decodedStride;
    ta.decodedStride = decodedStride;
    ta.decodedLen = dDecodedLen + at;
    ta.status = dStatus + at;
    ta.path = dPath ? dPath + (size_t)at * 3 * pathStride : nullptr;
    ta.pathStride = pathStride;
    ta.pathLen = dPathLen ? dPathLen + at : nullptr;
    CUDA_TRY(launchTraceback(d->dev, ta, stream));
    if (rec) CUDA_TRY(cudaEventRecord(ev[2], stream));
    d->stats.kernel_launches += 2;
    d->stats.fill_launches += 1;
    d->stats.traceback_launches += 1;
  }
  d->stats.reads += (uint64_t)nReads;
  return DNAB_OK;
}

}  // namespace dnab

extern "C" {

dnab_decoder* dnab_decoder_create(const dnab_tables* t, int device) {
  if (!t || !t->n_states) {
    setLastError("dnab_decoder_create: empty tables");
    return nullptr;
  }
  int nDev = 0;
  cudaError_t err = cudaGetDeviceCount(&nDev);
  if (err != cudaSuccess || nDev == 0 || device < 0 || device >= nDev) {
    setLastError(std::string("dnab_decoder_create: no usable CUDA device (") +
                 (err != cudaSuccess ? cudaGetErrorString(err) : "device ordinal out of range") +
                 "); this library has no CPU fallback");
    return nullptr;
  }
  if (t->k > (uint32_t)kMaxK) {
    setLastError("duplication depth k=" + std::to_string(t->k) + " exceeds the supported maximum " + std::to_string(kMaxK));
    return nullptr;
  }
  for (uint32_t e = 0; e < t->n_emit; ++e)
    if (t->emit_src[e] >= t->n_states || t->emit_base[e] > 3) {
      setLastError("dnab_decoder_create: emitting transition " + std::to_string(e) + " has a source or base out of range");
      return nullptr;
    }
  for (uint32_t e = 0; e < t->n_null; ++e)
    if (t->null_src[e] >= t->n_states) {
      setLastError("dnab_decoder_create: null transition " + std::to_string(e) + " has a source out of range");
      return nullptr;
    }
  if (t->emit_off[t->n_states] != t->n_emit || t->null_off[t->n_states] != t->n_null) {
    setLastError("dnab_decoder_create: CSR offsets do not end at the transition counts");
    return nullptr;
  }
  auto* d = new dnab_decoder();
  d->device = device;
  cudaSetDevice(device);
  cudaDeviceProp prop{};
  cudaGetDeviceProperties(&prop, device);
  if (prop.major < 10) {
    setLastError(std::string("device ") + prop.name + " is not a Blackwell (sm_100a) GPU");
    delete d;
    return nullptr;
  }
  d->smCount = prop.multiProcessorCount;
  d->smemOptin = prop.sharedMemPerBlockOptin;
  size_t freeB = 0, totalB = 0;
  cudaMemGetInfo(&freeB, &totalB);
  d->predBudgetBytes = std::min<size_t>(freeB / 2, (size_t)48 << 30);
  cudaEventCreate(&d->ev0);
  cudaEventCreate(&d->ev1);
  cudaEventCreate(&d->ev2);

  const uint32_t N = t->n_states, k = t->k;
  d->nStates = N;
  d->k = k;
  d->local = t->local;
  d->emitOff.assign(t->emit_off, t->emit_off + N + 1);
  d->nullOff.assign(t->null_off, t->null_off + N + 1);
  d->emitSrc.assign(t->emit_src, t->emit_src + t->n_emit);
  d->nullSrc.assign(t->null_src, t->null_src + t->n_null);
  d->emitBase.assign(t->emit_base, t->emit_base + t->n_emit);
  d->mdl.assign(t->mdl, t->mdl + N);
  d->ctx.assign(t->ctx, t->ctx + (size_t)N * k);
  // input symbols -> small ids; every transition carrying the same symbol has the same score
  std::map<uint8_t, uint32_t> symId;
  d->symChar.push_back(0);
  d->symScore.push_back(0.);
  symId[0] = 0;
  auto idOf = [&](uint8_t ch, double score, bool& ok) -> uint8_t {
    auto it = symId.find(ch);
    if (it == symId.end()) {
      if (d->symChar.size() >= (size_t)kMaxSyms) {
        ok = false;
        return 0;
      }
      it = symId.emplace(ch, (uint32_t)d->symChar.size()).first;
      d->symChar.push_back(ch);
      d->symScore.push_back(score);
    }
    if (std::memcmp(&d->symScore[it->second], &score, sizeof(double)) != 0) ok = false;
    return (uint8_t)it->second;
  };
  bool ok = true;
  d->emitSym.resize(t->n_emit);
  d->nullSym.resize(t->n_null);
  for (uint32_t e = 0; e < t->n_emit && ok; ++e) d->emitSym[e] = idOf(t->emit_in[e], t->emit_score[e], ok);
  for (uint32_t e = 0; e < t->n_null && ok; ++e) d->nullSym[e] = idOf(t->null_in[e], t->null_score[e], ok);
  if (!ok) {
    setLastError("transition scores are not a function of the input symbol (or more than 31 symbols)");
    dnab_decoder_destroy(d);
    return nullptr;
  }
  std::memcpy(d->sub, t->sub, sizeof d->sub);
  for (int i = 0; i < kMaxK; ++i) d->len[i] = (uint32_t)i < k ? t->len[i] : 0.;
  d->noGap = t->noGap;
  d->delOpen = t->delOpen;
  d->delExtend = t->delExtend;
  d->delEnd = t->delEnd;
  d->tanDup = t->tanDup;
  return d;
}

void dnab_decoder_destroy(dnab_decoder* d) {
  if (!d) return;
  cudaSetDevice(d->device);
  if (d->ev0) cudaEventDestroy(d->ev0);
  if (d->ev1) cudaEventDestroy(d->ev1);
  if (d->ev2) cudaEventDestroy(d->ev2);
  for (cudaEvent_t e : d->evPool) cudaEventDestroy(e);
  delete d;
}

int dnab_decoder_configure(dnab_decoder* d, uint32_t cluster_size, uint32_t threads_per_cta, uint32_t t_in_smem_mode) {
  if (!d) return DNAB_EINVAL;
  d->wantC = cluster_size;
  d->wantThreads = threads_per_cta;
  d->wantTMode = t_in_smem_mode;
  d->plan = LaunchPlan();
  return DNAB_OK;
}

int dnab_decoder_set_option(dnab_decoder* d, const char* key, int64_t value) {
  if (!d || !key || value < 0) {
    setLastError("dnab_decoder_set_option: bad argument");
    return DNAB_EINVAL;
  }
  const std::string k(key);
  const uint32_t v = (uint32_t)value;
  if (k == "kernel") {  // 0 automatic, 1 read-batched, 2 push (one read per cluster)
    if (v > 2) {
      setLastError(v == 3 ? "dnab_decoder_set_option: kernel 3 (the pull-closure fill kernel) was retired; use 0, 1 or 2"
                          : "dnab_decoder_set_option: kernel must be 0, 1 or 2");
      return DNAB_EINVAL;
    }
    d->wantBatch = v == 0 ? -1 : v == 1 ? 1 : 0;
  } else if (k == "team_size")
    d->wantTeam = v;
  else if (k == "warps_per_cta")
    d->wantWarps = v;
  else if (k == "cluster_size")
    d->wantC = v;
  else if (k == "threads_per_cta")
    d->wantThreads = v;
  else if (k == "t_columns")  // 0 auto, 1 shared memory, 2 global scratch
    d->wantTMode = v;
  else if (k == "table")  // 0 auto, 1 shared memory, 2 global memory
    d->wantBlockMode = v;
  else if (k == "s_prev")  // 0 auto, 1 shared memory, 2 global scratch
    d->wantSPrevMode = v;
  else if (k == "partition")  // 0 auto, 1 index runs, 2 DFS runs unsorted, 3 DFS chunks dealt, 4 DFS runs sorted
    d->wantPartition = v;
  else if (k == "thin_n")
    d->thinN = v;
  else if (k == "t_recompute")
    d->tRecompute = v;
  else if (k == "queue_cap")
    d->queueCap = v;
  else if (k == "deal_chunks")
    d->dealChunks = v;
  else if (k == "idle_sleep_ns") {
    // back-off of the retired pull-closure kernel: still accepted so that existing callers keep working; no effect
  } else if (k == "eager_notify")
    d->eagerNotify = v;
  else if (k == "notify_classes")
    d->notifyClasses = v;
  else if (k == "batch_idle_ns")
    d->batchIdleNs = v;
  else if (k == "async_closure")
    d->asyncClosure = v;
  else if (k == "team_slack_pct")
    d->teamSlackPct = v;
  else if (k == "persist_l2")
    d->wantPersist = v;
  else if (k == "pred_budget_mb")
    d->predBudgetBytes = (size_t)value << 20;
  else if (k == "fwd_threads") {
    if (value != 0 && (value > 1024 || value % 32 != 0)) {
      setLastError("dnab_decoder_set_option: fwd_threads must be 0 (automatic) or a multiple of 32 from 32 to 1024");
      return DNAB_EINVAL;
    }
    d->fwdThreads = v;
  } else if (k == "fwd_blocks") {
    if (value > UINT32_MAX) {
      setLastError("dnab_decoder_set_option: fwd_blocks must be below 2^32");
      return DNAB_EINVAL;
    }
    d->fwdBlocks = v;
  } else {
    setLastError("dnab_decoder_set_option: unknown option '" + k + "'");
    return DNAB_EINVAL;
  }
  d->plan = LaunchPlan();
  d->bplan = BatchPlan();
  return DNAB_OK;
}

int dnab_decoder_get_batch_info(const dnab_decoder* dc, dnab_batch_info* info) {
  if (!dc || !info) return DNAB_EINVAL;
  auto* d = const_cast<dnab_decoder*>(dc);
  cudaSetDevice(d->device);
  std::memset(info, 0, sizeof *info);
  if (!batchWanted(d)) return DNAB_OK;
  if (buildBatchPlan(d) != DNAB_OK) return d->wantBatch == 1 ? DNAB_EINVAL : DNAB_OK;
  info->enabled = (d->wantBatch == 1 || d->bplan.T == 1 || buildPlan(d, 1) != DNAB_OK || d->plan.C >= 4) ? 1 : 0;
  info->reads_per_group = kBatchReads;
  info->team_size = d->bplan.T;
  info->states_per_cta = d->bplan.M;
  info->warps_per_cta = d->bplan.warps;
  info->smem_bytes_per_cta = d->bplan.smemBytes;
  info->n_teams = d->bplan.nTeams;
  info->cross_cta_transition_fraction = d->bplan.crossFraction;
  info->wide_states = d->btab.nWide;
  return DNAB_OK;
}

int dnab_decoder_get_info(const dnab_decoder* dc, dnab_decoder_info* info) {
  if (!dc || !info) return DNAB_EINVAL;
  auto* d = const_cast<dnab_decoder*>(dc);
  cudaSetDevice(d->device);
  int rc = buildPlan(d, 1);
  if (rc != DNAB_OK) return rc;
  info->n_states = d->nStates;
  info->k = d->k;
  info->local = d->local;
  info->cluster_size = d->plan.C;
  info->states_per_cta = d->plan.M;
  info->threads_per_cta = d->plan.threads;
  info->smem_bytes_per_cta = d->plan.smemBytes;
  info->t_in_smem = d->plan.tInSmem;
  info->table_in_smem = d->plan.outInSmem;
  info->s_prev_in_smem = d->plan.sPrevGlobal ? 0 : 1;
  info->n_clusters = d->plan.nClusters;
  info->sm_count = (uint32_t)d->smCount;
  return DNAB_OK;
}

/* Profiling aid (not part of the stable ABI): counters accumulated by rank 0 / thread 0 of every
 * cluster: [0] columns, [1] frontier sweeps after the first dense one, [2] worklist entries of
 * rank 0, [3..5] SM cycles in the emission step / closure / predecessor pass. */
int dnab_decoder_set_debug(dnab_decoder* d, int enabled) {
  if (!d) return DNAB_EINVAL;
  cudaSetDevice(d->device);
  if (enabled) {
    if (d->dDbg.ensure(16) != cudaSuccess) return DNAB_ECUDA;
    cudaMemset(d->dDbg.p, 0, 16 * sizeof(unsigned long long));
  }
  d->debug = enabled != 0;
  return DNAB_OK;
}
int dnab_decoder_debug_counters(dnab_decoder* d, unsigned long long* out16) {
  if (!d || !d->dDbg.p) return DNAB_EINVAL;
  cudaSetDevice(d->device);
  return cudaMemcpy(out16, d->dDbg.p, 16 * sizeof(unsigned long long), cudaMemcpyDeviceToHost) == cudaSuccess ? DNAB_OK : DNAB_ECUDA;
}

int dnab_decoder_set_timing(dnab_decoder* d, int enabled) {
  if (!d) return DNAB_EINVAL;
  d->timing = enabled != 0;
  return DNAB_OK;
}

int dnab_decoder_get_stats(const dnab_decoder* dc, dnab_decoder_stats* s) {
  if (!dc || !s) return DNAB_EINVAL;
  auto* d = const_cast<dnab_decoder*>(dc);
  // resolve the pooled event triples of the device path (the caller has synchronised)
  for (size_t i = 0; i + 2 < d->evUsed; i += 3) {
    float a = 0, b = 0;
    if (cudaEventElapsedTime(&a, d->evPool[i], d->evPool[i + 1]) == cudaSuccess &&
        cudaEventElapsedTime(&b, d->evPool[i + 1], d->evPool[i + 2]) == cudaSuccess) {
      d->stats.timed_fill_ms += a;
      d->stats.timed_traceback_ms += b;
      d->stats.timed_fill_launches += 1;
    }
  }
  d->evUsed = 0;
  *s = d->stats;
  return DNAB_OK;
}

int dnab_decoder_reset_timing(dnab_decoder* d) {
  if (!d) return DNAB_EINVAL;
  d->evUsed = 0;
  d->stats.timed_fill_ms = d->stats.timed_traceback_ms = 0;
  d->stats.timed_fill_launches = 0;
  return DNAB_OK;
}

int dnab_viterbi_batch_device(dnab_decoder* d, int64_t n_reads, int32_t max_read_len, const uint8_t* d_packed,
                              const int64_t* d_read_byte_off, const int32_t* d_read_len, double* d_loglike,
                              char* d_decoded, int32_t decoded_stride, int32_t* d_decoded_len, int32_t* d_status,
                              void* cuda_stream) {
  if (!d || n_reads < 0 || max_read_len < 0 || decoded_stride <= 0) {
    setLastError("dnab_viterbi_batch_device: bad argument");
    return DNAB_EINVAL;
  }
  return runDevice(d, n_reads, max_read_len, d_packed, d_read_byte_off, d_read_len, d_loglike, d_decoded, decoded_stride,
                   d_decoded_len, d_status, nullptr, 0, nullptr, nullptr, (cudaStream_t)cuda_stream, false);
}

static int viterbiHost(dnab_decoder* d, int64_t n, const uint8_t* packed, const int64_t* byteOff, const int32_t* readLen,
                       double* loglike, char* decoded, int32_t decodedStride, int32_t* decodedLen, int32_t* status,
                       int32_t* path, int32_t pathStride, int32_t* pathLen, double* cells) {
  if (!d || n < 0 || decodedStride <= 0) {
    setLastError("dnab_viterbi_batch: bad argument");
    return DNAB_EINVAL;
  }
  if (n == 0) return DNAB_OK;
  CUDA_TRY(cudaSetDevice(d->device));
  int32_t maxLen = 0;
  size_t packedBytes = 0;
  uint64_t cellsTotal = 0;
  for (int64_t r = 0; r < n; ++r) {
    if (readLen[r] < 0 || byteOff[r] < 0 || (byteOff[r] & 15)) {
      setLastError("dnab_viterbi_batch: read " + std::to_string(r) + " has a negative length or an offset that is not a multiple of 16");
      return DNAB_EINVAL;
    }
    maxLen = std::max(maxLen, readLen[r]);
    packedBytes = std::max<size_t>(packedBytes, (size_t)byteOff[r] + ((((size_t)readLen[r] + 3) / 4 + 15) & ~(size_t)15));
    cellsTotal += (uint64_t)d->nStates * (uint64_t)(readLen[r] + 1) * (d->k + 2);
  }
  packedBytes = std::max<size_t>(packedBytes, 16);
  CUDA_TRY(d->dPacked.ensure(packedBytes));
  CUDA_TRY(d->dByteOff.ensure((size_t)n));
  CUDA_TRY(d->dReadLen.ensure((size_t)n));
  CUDA_TRY(d->dLoglike.ensure((size_t)n));
  CUDA_TRY(d->dDecoded.ensure((size_t)n * decodedStride));
  CUDA_TRY(d->dDecodedLen.ensure((size_t)n));
  CUDA_TRY(d->dStatus.ensure((size_t)n));
  if (path) {
    CUDA_TRY(d->dPath.ensure((size_t)n * 3 * pathStride));
    CUDA_TRY(d->dPathLen.ensure((size_t)n));
  }
  size_t cellCount = 0;
  if (cells) {
    cellCount = (size_t)(readLen[0] + 1) * d->nStates * (d->k + 2);
    CUDA_TRY(d->dCells.ensure(cellCount));
  }
  cudaStream_t stream = nullptr;
  CUDA_TRY(cudaMemcpyAsync(d->dPacked.p, packed, packedBytes, cudaMemcpyHostToDevice, stream));
  CUDA_TRY(cudaMemcpyAsync(d->dByteOff.p, byteOff, (size_t)n * sizeof(int64_t), cudaMemcpyHostToDevice, stream));
  CUDA_TRY(cudaMemcpyAsync(d->dReadLen.p, readLen, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, stream));
  int rc = runDevice(d, n, maxLen, d->dPacked.p, d->dByteOff.p, d->dReadLen.p, d->dLoglike.p, d->dDecoded.p, decodedStride,
                     d->dDecodedLen.p, d->dStatus.p, path ? d->dPath.p : nullptr, pathStride,
                     path ? d->dPathLen.p : nullptr, cells ? d->dCells.p : nullptr, stream, true);
  if (rc != DNAB_OK) return rc;
  CUDA_TRY(cudaMemcpyAsync(loglike, d->dLoglike.p, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, stream));
  CUDA_TRY(cudaMemcpyAsync(decoded, d->dDecoded.p, (size_t)n * decodedStride, cudaMemcpyDeviceToHost, stream));
  CUDA_TRY(cudaMemcpyAsync(decodedLen, d->dDecodedLen.p, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
  CUDA_TRY(cudaMemcpyAsync(status, d->dStatus.p, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
  if (path) {
    CUDA_TRY(cudaMemcpyAsync(path, d->dPath.p, (size_t)n * 3 * pathStride * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaMemcpyAsync(pathLen, d->dPathLen.p, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
  }
  if (cells) CUDA_TRY(cudaMemcpyAsync(cells, d->dCells.p, cellCount * sizeof(double), cudaMemcpyDeviceToHost, stream));
  CUDA_TRY(cudaStreamSynchronize(stream));
  float ms = 0;
  if (cudaEventElapsedTime(&ms, d->ev0, d->ev1) == cudaSuccess) d->stats.last_fill_ms = ms;
  if (cudaEventElapsedTime(&ms, d->ev1, d->ev2) == cudaSuccess) d->stats.last_traceback_ms = ms;
  d->stats.cells += cellsTotal;
  if (cells && d->local) {
    // the reference overwrites S(end,L) with the column maximum in local mode (src/viterbi.cpp:171-173)
    const size_t endCell = ((size_t)readLen[0] * d->nStates + (d->nStates - 1)) * (d->k + 2);
    cells[endCell] = loglike[0];
  }
  return DNAB_OK;
}

int dnab_viterbi_batch(dnab_decoder* d, int64_t n_reads, const uint8_t* packed, const int64_t* read_byte_off,
                       const int32_t* read_len, double* loglike, char* decoded, int32_t decoded_stride,
                       int32_t* decoded_len, int32_t* status, int32_t* path, int32_t path_stride, int32_t* path_len) {
  return viterbiHost(d, n_reads, packed, read_byte_off, read_len, loglike, decoded, decoded_stride, decoded_len, status,
                     path, path_stride, path_len, nullptr);
}

static int forwardImpl(dnab_decoder* d, int64_t n, const uint8_t* packed, const int64_t* byteOff, const int32_t* readLen,
                       int32_t maxSweeps, double* loglike, int64_t* sweeps, int32_t* status, double* cells,
                       double* loglikeBack, double* counts, double* post = nullptr, const int64_t* postOff = nullptr) {
  if (!d || n < 0 || !loglike) {
    setLastError("dnab_forward_batch: bad argument");
    return DNAB_EINVAL;
  }
  if (n == 0) return DNAB_OK;
  CUDA_TRY(cudaSetDevice(d->device));
  const uint32_t N = d->nStates, k = d->k;
  if (!d->fwdReady) {
    std::vector<uint8_t> meta(d->emitSym.size());
    for (size_t e = 0; e < meta.size(); ++e) meta[e] = (uint8_t)(d->emitSym[e] | (d->emitBase[e] << 5));
    int32_t nLse = 0;
    const double* lseHost = dnab_lse_table(&nLse);
    std::vector<double> lseV(lseHost, lseHost + nLse);
    lseV.push_back(0.);  // lseUnary reads table[n+1]
    CUDA_TRY(d->dFwdEmitOff.upload(d->emitOff));
    CUDA_TRY(d->dFwdEmitSrc.upload(d->emitSrc));
    CUDA_TRY(d->dFwdEmitMeta.upload(meta));
    CUDA_TRY(d->dFwdNullOff.upload(d->nullOff));
    CUDA_TRY(d->dFwdNullSrc.upload(d->nullSrc));
    CUDA_TRY(d->dFwdNullSym.upload(d->nullSym));
    CUDA_TRY(d->dFwdCtx.upload(d->ctx));
    CUDA_TRY(d->dFwdMdl.upload(d->mdl));
    CUDA_TRY(d->dFwdLse.upload(lseV));
    // source-indexed lists for the backward pass: destination ascending, then list order
    auto outLists = [&](const std::vector<uint32_t>& inOff, const std::vector<uint32_t>& inSrc, const std::vector<uint8_t>& inMeta,
                        std::vector<uint32_t>& off, std::vector<uint32_t>& dst, std::vector<uint8_t>& meta) {
      off.assign(N + 2, 0);
      for (uint32_t s : inSrc) off[s + 2]++;
      for (uint32_t s = 0; s < N; ++s) off[s + 2] += off[s + 1];
      dst.assign(std::max<size_t>(inSrc.size(), 1), 0);
      meta.assign(std::max<size_t>(inSrc.size(), 1), 0);
      for (uint32_t dd = 0; dd < N; ++dd)
        for (uint32_t e = inOff[dd]; e < inOff[dd + 1]; ++e) {
          const uint32_t p = off[inSrc[e] + 1]++;
          dst[p] = dd;
          meta[p] = inMeta[e];
        }
      off.pop_back();  // off[s] .. off[s+1] is now the range of source s
    };
    std::vector<uint32_t> oeOff, oeDst, onOff, onDst;
    std::vector<uint8_t> oeMeta, onSym;
    outLists(d->emitOff, d->emitSrc, meta, oeOff, oeDst, oeMeta);
    outLists(d->nullOff, d->nullSrc, d->nullSym, onOff, onDst, onSym);
    CUDA_TRY(d->dFwdOutEmitOff.upload(oeOff));
    CUDA_TRY(d->dFwdOutEmitDst.upload(oeDst));
    CUDA_TRY(d->dFwdOutEmitMeta.upload(oeMeta));
    CUDA_TRY(d->dFwdOutNullOff.upload(onOff));
    CUDA_TRY(d->dFwdOutNullDst.upload(onDst));
    CUDA_TRY(d->dFwdOutNullSym.upload(onSym));
    d->fwdReady = true;
  }
  int32_t maxLen = 0;
  size_t packedBytes = 0;
  for (int64_t r = 0; r < n; ++r) {
    if (readLen[r] < 0 || byteOff[r] < 0 || (byteOff[r] & 15)) {
      setLastError("dnab_forward_batch: read " + std::to_string(r) + " has a negative length or an offset that is not a multiple of 16");
      return DNAB_EINVAL;
    }
    maxLen = std::max(maxLen, readLen[r]);
    packedBytes = std::max<size_t>(packedBytes, (size_t)byteOff[r] + ((((size_t)readLen[r] + 3) / 4 + 15) & ~(size_t)15));
  }
  if (maxLen > 16000) {
    setLastError("dnab_forward_batch: reads longer than 16000 bases are not supported");
    return DNAB_EINVAL;
  }
  packedBytes = std::max<size_t>(packedBytes, 16);
  // one CTA per read in flight; small machines get narrower CTAs and several of them per SM (the kernel is capped
  // at 64 registers, so 1024 threads per SM in total): l4c4 (384 states) 12.1k -> 24.0k reads/s
  const uint32_t fwdThreads = d->fwdThreads ? d->fwdThreads : N >= 4096 ? 1024u : N >= 2048 ? 512u : N >= 1024 ? 256u : 128u;
  const uint32_t fwdPerSm = 1024 / fwdThreads;
  uint32_t nBlocks = (uint32_t)std::min<int64_t>(n, (int64_t)d->smCount * fwdPerSm);
  const uint32_t nc = 5 + k + 16;
  const size_t fPerBlock = counts ? (size_t)(maxLen + 1) * N * (k + 2) : 0;  // forward cells kept for the backward pass
  if (counts) {
    size_t freeB = 0, totalB = 0;
    cudaMemGetInfo(&freeB, &totalB);
    const size_t budget = std::max<size_t>(d->dFwdF.n * sizeof(double), freeB / 2);
    nBlocks = (uint32_t)std::max<size_t>(1, std::min<size_t>(nBlocks, budget / (fPerBlock * sizeof(double))));
  }
  if (d->fwdBlocks) nBlocks = std::min(nBlocks, d->fwdBlocks);
  if (counts) {
    CUDA_TRY(d->dFwdF.ensure((size_t)nBlocks * fPerBlock));
    CUDA_TRY(d->dFwdCounts.ensure((size_t)n * nc));
    CUDA_TRY(d->dFwdLLBack.ensure((size_t)n));
    CUDA_TRY(d->dFwdSweepsBack.ensure((size_t)n));
  }
  CUDA_TRY(d->dPacked.ensure(packedBytes));
  CUDA_TRY(d->dByteOff.ensure((size_t)n));
  CUDA_TRY(d->dReadLen.ensure((size_t)n));
  CUDA_TRY(d->dLoglike.ensure((size_t)n));
  CUDA_TRY(d->dStatus.ensure((size_t)n));
  CUDA_TRY(d->dFwdSweeps.ensure((size_t)n));
  CUDA_TRY(d->dFwdScratch.ensure((size_t)nBlocks * (10 + 2 * k) * N));
  CUDA_TRY(d->dNextRead.ensure(1));
  size_t postRows = 0;
  const uint32_t nClasses = (uint32_t)d->symChar.size() + 1;
  if (post) {
    for (int64_t r = 0; r < n; ++r) postRows = std::max<size_t>(postRows, (size_t)postOff[r] + (size_t)readLen[r]);
    CUDA_TRY(d->dFwdPost.ensure(std::max<size_t>(1, postRows * nClasses)));
    CUDA_TRY(d->dFwdPostOff.ensure((size_t)n));
  }
  size_t cellCount = 0;
  if (cells) {
    cellCount = (size_t)(readLen[0] + 1) * N * (k + 2);
    CUDA_TRY(d->dCells.ensure(cellCount));
  }
  cudaStream_t stream = nullptr;
  CUDA_TRY(cudaMemcpyAsync(d->dPacked.p, packed, packedBytes, cudaMemcpyHostToDevice, stream));
  CUDA_TRY(cudaMemcpyAsync(d->dByteOff.p, byteOff, (size_t)n * sizeof(int64_t), cudaMemcpyHostToDevice, stream));
  CUDA_TRY(cudaMemcpyAsync(d->dReadLen.p, readLen, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, stream));
  CUDA_TRY(cudaMemsetAsync(d->dNextRead.p, 0, sizeof(unsigned long long), stream));
  std::vector<long long> postOffLL;
  if (post) {
    postOffLL.assign(postOff, postOff + n);
    CUDA_TRY(cudaMemcpyAsync(d->dFwdPostOff.p, postOffLL.data(), (size_t)n * sizeof(long long), cudaMemcpyHostToDevice, stream));
    CUDA_TRY(cudaMemsetAsync(d->dFwdPost.p, 0, postRows * nClasses * sizeof(double), stream));
  }
  ForwardTables ft{};
  ft.nStates = N;
  ft.k = k;
  ft.local = d->local;
  ft.nSyms = (uint32_t)d->symChar.size();
  ft.emitOff = d->dFwdEmitOff.p;
  ft.emitSrc = d->dFwdEmitSrc.p;
  ft.emitMeta = d->dFwdEmitMeta.p;
  ft.nullOff = d->dFwdNullOff.p;
  ft.nullSrc = d->dFwdNullSrc.p;
  ft.nullSym = d->dFwdNullSym.p;
  ft.ctx = d->dFwdCtx.p;
  ft.mdl = d->dFwdMdl.p;
  ft.lseTable = d->dFwdLse.p;
  ft.outEmitOff = d->dFwdOutEmitOff.p;
  ft.outEmitDst = d->dFwdOutEmitDst.p;
  ft.outEmitMeta = d->dFwdOutEmitMeta.p;
  ft.outNullOff = d->dFwdOutNullOff.p;
  ft.outNullDst = d->dFwdOutNullDst.p;
  ft.outNullSym = d->dFwdOutNullSym.p;
  for (int i = 0; i < kMaxSyms; ++i) ft.symScore[i] = i < (int)d->symScore.size() ? d->symScore[i] : 0.;
  std::memcpy(ft.sub, d->sub, sizeof ft.sub);
  std::memcpy(ft.len, d->len, sizeof ft.len);
  ft.noGap = d->noGap;
  ft.delOpen = d->delOpen;
  ft.delExtend = d->delExtend;
  ft.delEnd = d->delEnd;
  ft.tanDup = d->tanDup;
  ForwardArgs fa{};
  fa.nReads = n;
  fa.maxSweeps = maxSweeps > 0 ? maxSweeps : 4096;
  fa.packed = d->dPacked.p;
  fa.byteOff = d->dByteOff.p;
  fa.readLen = d->dReadLen.p;
  fa.scratch = d->dFwdScratch.p;
  fa.loglike = d->dLoglike.p;
  fa.sweeps = d->dFwdSweeps.p;
  fa.status = d->dStatus.p;
  fa.nextRead = d->dNextRead.p;
  fa.cells = cells ? d->dCells.p : nullptr;
  fa.maxLen = maxLen;
  fa.F = counts ? d->dFwdF.p : nullptr;
  fa.counts = counts ? d->dFwdCounts.p : nullptr;
  fa.loglikeBack = counts ? d->dFwdLLBack.p : nullptr;
  fa.sweepsBack = counts ? d->dFwdSweepsBack.p : nullptr;
  fa.post = post ? d->dFwdPost.p : nullptr;
  fa.postOff = post ? d->dFwdPostOff.p : nullptr;
  CUDA_TRY(cudaEventRecord(d->ev0, stream));
  CUDA_TRY(launchForward(ft, fa, nBlocks, fwdThreads, stream));
  CUDA_TRY(cudaEventRecord(d->ev1, stream));
  d->stats.kernel_launches += 1;
  d->stats.last_fwd_threads = fwdThreads;
  d->stats.last_fwd_blocks = nBlocks;
  CUDA_TRY(cudaMemcpyAsync(loglike, d->dLoglike.p, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, stream));
  std::vector<long long> sw(sweeps ? (size_t)n : 0);
  if (sweeps) CUDA_TRY(cudaMemcpyAsync(sw.data(), d->dFwdSweeps.p, (size_t)n * sizeof(long long), cudaMemcpyDeviceToHost, stream));
  if (status) CUDA_TRY(cudaMemcpyAsync(status, d->dStatus.p, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
  if (cells) CUDA_TRY(cudaMemcpyAsync(cells, d->dCells.p, cellCount * sizeof(double), cudaMemcpyDeviceToHost, stream));
  if (counts) {
    CUDA_TRY(cudaMemcpyAsync(counts, d->dFwdCounts.p, (size_t)n * nc * sizeof(double), cudaMemcpyDeviceToHost, stream));
    if (loglikeBack) CUDA_TRY(cudaMemcpyAsync(loglikeBack, d->dFwdLLBack.p, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, stream));
  }
  if (post) CUDA_TRY(cudaMemcpyAsync(post, d->dFwdPost.p, postRows * nClasses * sizeof(double), cudaMemcpyDeviceToHost, stream));
  CUDA_TRY(cudaStreamSynchronize(stream));
  for (size_t r = 0; r < sw.size(); ++r) sweeps[r] = (int64_t)sw[r];
  float ms = 0;
  if (cudaEventElapsedTime(&ms, d->ev0, d->ev1) == cudaSuccess) d->stats.last_fill_ms = ms;
  return DNAB_OK;
}

int dnab_forward_batch(dnab_decoder* d, int64_t n, const uint8_t* packed, const int64_t* byteOff, const int32_t* readLen,
                       int32_t maxSweeps, double* loglike, int64_t* sweeps, int32_t* status, double* cells) {
  return forwardImpl(d, n, packed, byteOff, readLen, maxSweeps, loglike, sweeps, status, cells, nullptr, nullptr);
}

int dnab_fwdback_counts_batch(dnab_decoder* d, int64_t n, const uint8_t* packed, const int64_t* byteOff, const int32_t* readLen,
                              int32_t maxSweeps, double* loglike, double* loglikeBack, double* counts, int32_t* status) {
  if (!counts) {
    setLastError("dnab_fwdback_counts_batch: counts must not be null");
    return DNAB_EINVAL;
  }
  return forwardImpl(d, n, packed, byteOff, readLen, maxSweeps, loglike, nullptr, status, nullptr, loglikeBack, counts);
}

int dnab_posterior_classes(const dnab_decoder* d, char* classes, size_t cap) {
  if (!d || !classes) return DNAB_EINVAL;
  const size_t n = d->symChar.size() + 1;
  if (n > (size_t)kPostClasses) {
    // classes: "no input symbol", one per input symbol, "duplication"
    setLastError("posterior decoding tells at most " + std::to_string(kPostClasses - 2) + " input symbols apart; this machine has " +
                 std::to_string(d->symChar.size() - 1));
    return DNAB_EINVAL;
  }
  if (cap < n + 1) {
    setLastError("dnab_posterior_classes: buffer too small");
    return DNAB_EINVAL;
  }
  classes[0] = '-';
  for (size_t i = 1; i < d->symChar.size(); ++i) classes[i] = (char)d->symChar[i];
  classes[n - 1] = '+';
  classes[n] = 0;
  return (int)n;
}

int dnab_posterior_batch(dnab_decoder* d, int64_t n, const uint8_t* packed, const int64_t* byteOff, const int32_t* readLen,
                         int32_t maxSweeps, const int64_t* postOff, double* loglike, double* post, char* decoded, int32_t* status) {
  if (!d || !post || !postOff || !loglike) {
    setLastError("dnab_posterior_batch: null argument");
    return DNAB_EINVAL;
  }
  char classes[kPostClasses + 1];
  const int nc = dnab_posterior_classes(d, classes, sizeof classes);
  if (nc < 0) return nc;
  std::vector<double> counts((size_t)std::max<int64_t>(n, 1) * (5 + d->k + 16)), llBack((size_t)std::max<int64_t>(n, 1));
  const int rc = forwardImpl(d, n, packed, byteOff, readLen, maxSweeps, loglike, nullptr, status, nullptr, llBack.data(), counts.data(),
                             post, postOff);
  if (rc != DNAB_OK) return rc;
  if (decoded)
    for (int64_t r = 0; r < n; ++r)
      for (int32_t p = 0; p < readLen[r]; ++p) {
        const double* row = post + ((size_t)postOff[r] + (size_t)p) * (size_t)nc;
        int best = 0;
        for (int c = 1; c < nc; ++c)
          if (row[c] > row[best]) best = c;
        decoded[(size_t)postOff[r] + (size_t)p] = classes[best];
      }
  return DNAB_OK;
}

int dnab_viterbi_cells(dnab_decoder* d, const uint8_t* packed, int32_t read_len, double* loglike, double* cells) {
  const int64_t off = 0;
  std::vector<char> dec(8 * (size_t)read_len + 1024);
  int32_t decLen = 0, status = 0;
  return viterbiHost(d, 1, packed, &off, &read_len, loglike, dec.data(), (int32_t)dec.size(), &decLen, &status, nullptr,
                     0, nullptr, cells);
}

}  // extern "C"
