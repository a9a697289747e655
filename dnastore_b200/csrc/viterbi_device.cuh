// Device-side table layout of the one-read-per-cluster Viterbi path, shared by its kernels
// (viterbi_fill_push.cu, viterbi_traceback.cu) and the host code that builds it (decoder.cu).
#pragma once
#include <cstdint>

namespace dnab {

constexpr int kMaxSyms = 32;     // distinct input symbols incl. the "no input" symbol 0
constexpr int kMaxK = 6;         // duplication depth supported by the packed state block (-l <= 13)
constexpr int kMaxCluster = 16;
constexpr uint32_t kNoPred = 255;  // predecessor record: "no candidate"

// ---------------------------------------------------------------------------
// Wide states.  A predecessor record is one byte: the index of the winning candidate in the state's
// list (S: nE emit edges, nN null edges, delEnd, T -> S, local start; D: 2*nE emit candidates, nN null
// ones; T: 2), 255 = none.  A state is WIDE when that byte, or one of the 7- and 8-bit count fields of
// the narrow table headers, cannot hold it: nE > 126, nE + nN + 2 > 254 (largest S index), 2*nE + nN
// > 254 (D candidates), or more than 255 outgoing transitions.  Narrow machines (no wide state) use
// exactly the narrow formats.  The wide states of a machine are numbered 0 .. nWide-1 in reference
// order; their S and D records keep the LOW byte in the ordinary record array and store the HIGH byte
// in a side plane, one byte per (wide state, record kind) next to it:
//   read-batched kernel  [group][pos][wide][2][32 reads]
//   push kernel          [read][pos][2][nWide]
// A wide record is the 16-bit index (high << 8 | low), 0xFFFF = none, so a wide state may have at
// most 65,535 candidates in either record (kMaxWideCandidates).  T records stay narrow.
// ---------------------------------------------------------------------------
constexpr uint32_t kWideNoPred = 0xFFFFu;
constexpr uint32_t kMaxWideCandidates = 65535;  // nE + nN + 3 (S) and 2*nE + nN (D)
constexpr uint32_t kMaxOutDegree = 65535;       // outgoing transitions of one state (16-bit counts of the wide headers)
__host__ __device__ inline bool stateIsWide(uint32_t nE, uint32_t nN, uint32_t nOut) {
  return nE > 126 || nE + nN + 2 > 254 || 2 * nE + nN > 254 || nOut > 255;
}

// ---------------------------------------------------------------------------
// State blocks: the traceback kernel decodes a predecessor record of state g against g's
// block (the record is an index into g's incoming edges).  The padded state space (Np = C*M
// states; state g lives in CTA rank g/M at local index g%M) is described by one block of
// 32-bit words per state, 8-byte aligned, found through blockOff[g]:
//
//   word 0   nEmit | nIn<<8 | nOut<<16 | mdl<<24        (nIn = nEmit + nNull)
//   word 1   ctx: 2 bits per duplication index i = tanDupBase(ss,i)
//   then     nIn incoming edges, TWO words each, emit edges first, each group in the
//            reference's list order (source index, transition index):
//              a: bits 0..19  byte offset of the source's cell inside a column (local*8)
//                 bits 20..23 cluster rank of the CTA owning the source
//                 bit  24     set when that CTA is not the block's own CTA
//              b: bits 0..7   sym*8            (byte offset into the per-symbol score tables)
//                 bits 8..20  sym*128+base*32  (byte offset of the (sym,base) row of the
//                                               traceback emit table; bits 13..14 = base)
//   then     nOut outgoing edges, one word each (states to wake when this one grows):
//              bits 0..15 local index, bits 20..23 rank, bit 24 "other CTA"
//   padding to an even number of words.
// Of these the traceback reads nEmit, nIn and the source and symbol of an incoming edge.
// A wide state's block has nEmit = kHdrWide and two more words before its edges:
//   word 2   nEmit | nIn << 16,   word 3   the state's wide number
// (its nOut field is not used).
// ---------------------------------------------------------------------------
constexpr uint32_t kEdgeRemote = 1u << 24;
constexpr uint32_t kHdrWide = 0xFFu;
__host__ __device__ inline uint32_t hdrNEmit(uint32_t w0) { return w0 & 0xFFu; }
__host__ __device__ inline uint32_t hdrNIn(uint32_t w0) { return (w0 >> 8) & 0xFFu; }
__host__ __device__ inline uint32_t edgeOff(uint32_t a) { return a & 0xFFFFFu; }
__host__ __device__ inline uint32_t edgeRank(uint32_t a) { return (a >> 20) & 0xFu; }
__host__ __device__ inline uint32_t edgeSymOff(uint32_t b) { return b & 0xFFu; }

// ---------------------------------------------------------------------------
// Tables of the push kernel (viterbi_fill_push.cu).  Same padded state space and the same
// partition as the state blocks; two compact forms of the transition table:
//
//  * IN-TABLE, streamed.  The dense passes (emission, first closure pass, predecessor
//    pass) visit the states of a CTA in index order, one state per thread and `chunkStates`
//    (= threads per CTA) states per step, so the incoming-edge lists are stored as CHUNKS
//    that a single bulk copy (cp.async.bulk, TMA) brings into shared memory:
//      chunk = [ u16 recOff[chunkStates+1] ] (padded to a word)  [ records ... ]  (padded to 16 B)
//      record = header word, then nIn edge words (emit edges first, reference list order)
//      header: bits 0..6 nEmit | 7..14 nIn (255 = padding state) | 15..17 mdl | 18..29 ctx
//              (2 bits per duplication index) | 30 "has an outgoing null transition"
//      a wide state has nIn = kInWide in its header and two more words before its edges:
//              nEmit | nIn << 16, then its wide number
//      edge:   bits 0..15 source's local index | 16..19 source's rank | 20 source in another
//              CTA | 21..25 input-symbol id | 26..27 emitted base
//  * OUT-TABLE, resident in shared memory when it fits.  The closure after the first pass is
//    PUSH style: a state whose S or D grew relaxes its successors.  Per CTA:
//      [ u16 outOff[M+1] ] (padded to a word)  [ edge words ... ]
//      edge:   bits 0..15 destination's local index | 16..19 rank | 20 other CTA |
//              21..25 input-symbol id | 26 transition emits a base
// ---------------------------------------------------------------------------
constexpr uint32_t kInPad = 255;
constexpr uint32_t kInWide = 254;  // (a narrow state has nIn <= 252)
__host__ __device__ inline uint32_t inNEmit(uint32_t h) { return h & 0x7Fu; }
__host__ __device__ inline uint32_t inNIn(uint32_t h) { return (h >> 7) & 0xFFu; }
__host__ __device__ inline uint32_t inMdl(uint32_t h) { return (h >> 15) & 0x7u; }
__host__ __device__ inline uint32_t inCtx(uint32_t h, uint32_t i) { return (h >> (18 + 2 * i)) & 0x3u; }
__host__ __device__ inline uint32_t inHasNullOut(uint32_t h) { return (h >> 30) & 1u; }
__host__ __device__ inline uint32_t peLocal(uint32_t w) { return w & 0xFFFFu; }
__host__ __device__ inline uint32_t peRank(uint32_t w) { return (w >> 16) & 0xFu; }
__host__ __device__ inline uint32_t peRemote(uint32_t w) { return (w >> 20) & 1u; }
__host__ __device__ inline uint32_t peSym(uint32_t w) { return (w >> 21) & 0x1Fu; }
__host__ __device__ inline uint32_t peBase(uint32_t w) { return (w >> 26) & 0x3u; }
__host__ __device__ inline uint32_t peIsEmit(uint32_t w) { return (w >> 26) & 1u; }
__host__ __device__ inline uint32_t peMake(uint32_t local, uint32_t rank, bool remote, uint32_t sym, uint32_t top) {
  return local | (rank << 16) | (remote ? 1u << 20 : 0u) | (sym << 21) | (top << 26);
}

struct DevTables {
  uint32_t nStates;   // real states
  uint32_t M;         // states per CTA slice
  uint32_t C;         // cluster size; padded state count Np = C*M
  uint32_t k;         // duplication depth
  uint32_t local;     // local-alignment mode
  uint32_t nSyms;
  uint32_t startG;    // padded-space index of reference state 0
  uint32_t endG;      // padded-space index of the reference's last state
  uint32_t tInSmem;   // T columns in shared memory (else in global scratch)
  uint32_t nWide;     // wide states (side plane entries per column and record kind)
  const uint32_t* blocks;    // state blocks (traceback)
  const uint32_t* blockOff;   // [Np] word offset of each state's block
  const uint32_t* origId;     // [Np] reference state index, 0xFFFFFFFF for padding
  const uint8_t* symChar;     // [nSyms] input-symbol character of each id
  uint32_t sPrevInSmem;       // S(pos-1) kept in shared memory (else in global scratch / L2)
  uint32_t outInSmem;         // the CTA's out-table is resident in shared memory
  uint32_t chunkStates;       // states per in-table chunk (= threads per CTA)
  uint32_t nChunks;           // chunks per CTA = ceil(M / chunkStates)
  uint32_t maxChunkBytes;     // largest chunk (shared-memory staging buffer size)
  uint32_t maxOutBytes;       // largest out-table of any rank
  const uint32_t* inChunks;   // all chunks of all ranks (16-byte aligned pieces)
  const uint32_t* inChunkOff; // [C][nChunks+1] word offset of each chunk in inChunks
  const uint4* outSlots;      // [Np] 16-byte out-slots {nOut, e0, e1, e2} (or {nOut, overflow offset} when nOut > 3):
                              // the out-table in the form read straight from L2 when it is not in shared memory
  const uint32_t* outOvf;     // overflow edges of states with more than 3 outgoing transitions
  const uint32_t* outTable;   // all out-tables
  const uint32_t* outSliceOff;// [C+1] word offset of each rank's out-table in outTable
  double symScore[kMaxSyms];  // log(symProb) per id (0 for id 0)
  double sub[16];
  double len[kMaxK > 0 ? kMaxK : 1];
  double noGap, delOpen, delExtend, delEnd, tanDup;
};

}  // namespace dnab
