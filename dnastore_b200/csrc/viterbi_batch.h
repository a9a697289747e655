// Read-batched Viterbi fill (viterbi_fill_batch.cu): table formats, launch arguments and the
// shared-memory carve-up, shared between the kernel and the host code that plans it (decoder.cu).
//
// The reads are the SIMD lanes.  A GROUP of 32 reads walks the machine together: lane r of every warp
// works on read r of the group, a warp works on ONE state at a time, so a transition is decoded once per
// warp instead of once per read, a gather is one conflict-free 512-byte row of shared memory, and what is
// left per lane is the reference's own fp64 adds and compares (src/viterbi.cpp:92-106,118-158,251-286).
// A TEAM of T CTAs (T = 1 ... the whole GPU) holds the S and D columns of one group in shared memory,
// M = ceil(N/T) states per CTA; everything that crosses CTAs goes through L2 (published rows, inbox
// masks, team barriers), so T is not limited by the cluster size.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "viterbi_device.cuh"

namespace dnab {

constexpr uint32_t kBatchReads = 32;       // reads per group = lanes of a warp
constexpr uint32_t kBatchMaxSlots = 32;    // a warp owns at most this many states (bits of its work mask)
constexpr uint32_t kBatchAllEdges = 0xFFFFFFFFu;

// ---------------------------------------------------------------------------
// Per-CTA tables (resident in shared memory).  Padded state space Np = T*M; state g = rank*M + i lives
// in CTA `rank` at local index i; warp (i % W) owns it as its slot (i / W).
//
//   header  uint4   x: inOff | outOff << 16        (entry offsets inside the rank's edge arrays)
//                   y: nEmit | nNull << 8 | nOut << 16 | mdl << 24
//                   z: ctx (2 bits per duplication index) | hasRemoteOut << 16 | pad << 17 | nOutLocal << 18
//                      (successors in this CTA come first in the out-edge list)
//                   w: reference state index (0xFFFFFFFF for padding)
//   in-edge uint2   x: padded index g of the source
//                   y: symbol id | base << 5 | remote << 7      (emit edges first, reference list order)
//   out-edge u32    successors in this CTA: bits 0..15 destination's local index | 16..20 bit of the destination's
//                   work mask (= index of this transition in the destination's in-edge list, 31 = "31 or later");
//                   then one entry per (OTHER CTA, class) that owns a successor: rank * kNotifyClasses + class, the index
//                   of the notification counter that is incremented when this state publishes a new row
//   remoteIn u32    per state: the bits of its work mask whose transitions come from other CTAs
//   clsOff  u32     [T][kNotifyClasses + 1], clsStates u32 [T*M]: the CTA's states that have transitions from other CTAs,
//                   grouped by notification class (local indices; class q = entries clsOff[q] .. clsOff[q+1])
//   The closure reads its own copy of the in-transitions, grouped so that its loops have no per-edge branch:
//   hdr2    uint2   x: offset of the state's relax entries inside the rank's array
//                   y: local emit | local null << 8 | remote emit << 16 | remote null << 24   (counts, in this order)
//   relax   uint2   x: padded index g of the source, y: symbol id * 8 (byte offset of its score)
//   Bit j of a state's work mask is its j-th relax entry (31 = "31 or later").
//   A WIDE state (viterbi_device.cuh) has bit 27 of header.y set and its wide number in bits 0..23 of header.y
//   (mdl stays in bits 24..26); its counts are in the wide table instead of the 8-bit fields of header.y, header.z
//   and hdr2.y:
//   wide    uint4   x: nEmit | nNull << 16   y: local emit | local null << 16   z: remote emit | remote null << 16
//                   w: nOutLocal | nOut << 16
// ---------------------------------------------------------------------------
__host__ __device__ inline uint32_t bhInOff(const uint4& h) { return h.x & 0xFFFFu; }
__host__ __device__ inline uint32_t bhOutOff(const uint4& h) { return h.x >> 16; }
__host__ __device__ inline uint32_t bhNEmit(const uint4& h) { return h.y & 0xFFu; }
__host__ __device__ inline uint32_t bhNNull(const uint4& h) { return (h.y >> 8) & 0xFFu; }
__host__ __device__ inline uint32_t bhNOut(const uint4& h) { return (h.y >> 16) & 0xFFu; }
__host__ __device__ inline uint32_t bhMdl(const uint4& h) { return (h.y >> 24) & 0x7u; }
__host__ __device__ inline uint32_t bhCtx(const uint4& h, uint32_t i) { return (h.z >> (2 * i)) & 3u; }
__host__ __device__ inline uint32_t bhRemoteOut(const uint4& h) { return (h.z >> 16) & 1u; }
__host__ __device__ inline uint32_t bhPad(const uint4& h) { return (h.z >> 17) & 1u; }
__host__ __device__ inline uint32_t bhNOutLocal(const uint4& h) { return (h.z >> 18) & 0xFFu; }
constexpr uint32_t kBhWide = 1u << 27;
__host__ __device__ inline uint32_t bhWide(const uint4& h) { return (h.y >> 27) & 1u; }
__host__ __device__ inline uint32_t bhWideNo(const uint4& h) { return h.y & 0xFFFFFFu; }
__host__ __device__ inline uint32_t beSym(const uint2& e) { return e.y & 31u; }
__host__ __device__ inline uint32_t beBase(const uint2& e) { return (e.y >> 5) & 3u; }
__host__ __device__ inline uint32_t beRemote(const uint2& e) { return (e.y >> 7) & 1u; }
__host__ __device__ inline uint32_t boLocal(uint32_t w) { return w & 0xFFFFu; }
__host__ __device__ inline uint32_t boBit(uint32_t w) { return (w >> 16) & 31u; }
__host__ __device__ inline uint32_t boRank(uint32_t w) { return (w >> 21) & 0x3FFu; }
__host__ __device__ inline uint32_t boRemote(uint32_t w) { return w >> 31; }

// classes of notification counters per CTA = lanes of the polling warp
constexpr uint32_t kNotifyClasses = 32;

struct BatchTables {
  uint32_t nStates, M, T, k, local, nSyms;
  uint32_t startRank, startLocal, endRank, endLocal;
  uint32_t maxIn, maxOut;        // largest per-rank edge counts (shared-memory sizing)
  const uint4* hdr;              // [T*M]
  const uint2* inEdges;          // all ranks, rank r at rankInOff[r]
  const uint32_t* outEdges;      // all ranks, rank r at rankOutOff[r]
  const uint32_t* rankInOff;     // [T+1]
  const uint32_t* rankOutOff;    // [T+1]
  const uint32_t* remoteIn;      // [T*M]
  const uint32_t* clsOff;        // [T][kNotifyClasses + 1]
  const uint32_t* clsStates;     // [T*M]
  const uint2* hdr2;             // [T*M]
  const uint2* relEdges;         // all ranks, rank r at rankInOff[r] (as many relax entries as in-edges)
  const double* tsE;             // [32 syms][4 bases][4 observed] (score+noGap)+sub: traceback association (src/viterbi.cpp:255)
  const uint4* wide;             // [nWide] counts of the wide states
  uint32_t nWide;
  double symScore[kMaxSyms];     // log(symProb) per symbol id (0 for id 0)
  double tsDext[kMaxSyms];       // score+delExtend (src/viterbi.cpp:272)
  double tsDopen[kMaxSyms];      // score+delOpen   (src/viterbi.cpp:273)
  double tsT[8];                 // tanDup+len[i]   (src/viterbi.cpp:286)
  double len[8];
  double sub[16];
  double noGap, delOpen, delExtend, delEnd, tanDup;
};

struct BatchArgs {
  int64_t nReads;
  int64_t readBase;              // identity order: slot i of this launch is read readBase + i
  int64_t nGroups;
  uint32_t nTeams;
  int32_t maxLen;                // record stride: every group owns (maxLen+1) columns
  uint32_t idleNs;               // asynchronous closure: back-off of a warp that found no work
  uint32_t asyncClosure;         // 1: closure without level barriers (work counter), 0: breadth-first levels
  const uint8_t* packed;         // 2-bit reads
  const int64_t* byteOff;        // [nReads]
  const int32_t* readLen;        // [nReads]
  const int32_t* order;          // optional [nGroups*32]: slot -> read (-1 = empty lane); null = identity
  uint8_t* pred;                 // [nGroups][maxLen+1][nStates][k+2][32] predecessor records, 1 byte per DP cell, reference state order
  uint8_t* predWide;             // [nGroups][maxLen+1][nWide][2][32] high bytes of the wide states' S and D records
  double* priv;                  // [nTeams][Np][2+k][32] rows private to the owning lane, carried from one column to the next:
                                 //   S0 of the next column (emission step fused into the record pass), the best emit candidate of
                                 //   its S record (traceback association), the k parked duplication cells
  double2* sdPub;                // [nTeams][2][Np][32] (S,D) rows of states with successors in other CTAs (T > 1), by column parity
  uint32_t* teamState;           // [nTeams][T][kNotifyClasses] notification counters (T > 1), zeroed before every launch
  uint32_t eagerNotify;          // 1: every notification is also sent once BEFORE the release fence (see flushRemote)
  uint32_t* teamPassive;         // [nTeams][2] passive CTAs of the current column, by column parity, zeroed before every launch
  unsigned long long* barrier;   // [nTeams] team barrier counters (monotonic), zeroed before every launch
  double* loglike;               // [nReads] global mode
  double* partVal;               // [nGroups][T*warps][32] local mode: per-warp best final S ...
  uint32_t* partOrig;            //   ... and its reference state (first maximum in reference order)
  double* cells;                 // optional dump of slot 0 of group 0: [(L+1)][nStates][k+2]
  unsigned long long* dbg;       // optional [16] counters
};

struct BatchLayout {
  uint32_t sd, maskA, maskB, remIn, cls, hdr, hdr2, inE, relE, outE, tsE, sub, ctl, total;
};

__host__ __device__ inline BatchLayout makeBatchLayout(uint32_t M, uint32_t maxIn, uint32_t maxOut, uint32_t nSyms, bool team) {
  BatchLayout L;
  uint32_t at = 0;
  auto take = [&](uint32_t bytes) {
    const uint32_t here = at;
    at += (bytes + 15u) & ~15u;
    return here;
  };
  L.sd = take(M * kBatchReads * 16);
  L.maskA = take(M * 4);
  L.maskB = take(M * 4);
  L.remIn = team ? take(M * 4) : 0;
  L.cls = team ? take((kNotifyClasses + 1 + M) * 4) : 0;
  L.hdr = take(M * 16);
  L.hdr2 = take(M * 8);
  L.inE = take((maxIn + 1) * 8);
  L.relE = take((maxIn + 1) * 8);
  L.outE = take((maxOut + 1) * 4);
  L.tsE = take(nSyms * 16 * 8);
  L.sub = take(16 * 8);
  L.ctl = take(64 * 4);
  L.total = at;
  return L;
}

// reference-order CSR tables for the traceback over batch-layout records
struct BatchTraceTables {
  uint32_t nStates, k, local, T;  // T = per-group partial maxima in local mode (CTAs x warps)
  uint32_t nWide;
  const uint32_t* wideOf;         // [nStates] wide number of every state (0xFFFFFFFF: narrow); null when nWide = 0
  const uint32_t* emitOff;
  const uint32_t* emitSrc;
  const uint8_t* emitSym;
  const uint32_t* nullOff;
  const uint32_t* nullSrc;
  const uint8_t* nullSym;
  const uint8_t* symChar;
};

struct BatchTraceArgs {
  int64_t nSlots;                // nGroups * 32
  int32_t maxLen;
  const int32_t* readLen;
  const int32_t* order;          // slot -> read, or null
  int64_t nReads;
  int64_t readBase;
  const uint8_t* pred;
  const uint8_t* predWide;
  double* loglike;
  const double* partVal;
  const uint32_t* partOrig;
  char* decoded;
  int32_t decodedStride;
  int32_t* decodedLen;
  int32_t* status;
  int32_t* path;
  int32_t pathStride;
  int32_t* pathLen;
};

cudaError_t queryBatchTeams(const BatchTables& tb, uint32_t warps, uint32_t smemBytes, int* ctasPerSm);
// persistBytes > 0: the first persistBytes of args.priv get a persisting L2 access-policy window for this launch
cudaError_t launchFillBatch(const BatchTables& tb, const BatchArgs& args, uint32_t warps, uint32_t smemBytes,
                            cudaStream_t stream, size_t persistBytes);
cudaError_t launchTracebackBatch(const BatchTraceTables& tb, const BatchTraceArgs& args, cudaStream_t stream);

}  // namespace dnab
