// Launch interface of the Viterbi fill / traceback and forward kernels used by decoder.cu.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "viterbi_device.cuh"

namespace dnab {

// mirror include/dnastore_b200.h DNAB_READ_* without pulling the C header into device code
constexpr int32_t DNAB_READ_OK_ = 0;
constexpr int32_t DNAB_READ_NO_DECODING_ = 1;
constexpr int32_t DNAB_READ_OVERFLOW_ = 2;
constexpr int32_t DNAB_READ_TRACEBACK_FAILED_ = 3;

// ---------------------------------------------------------------------------
// shared-memory carve-up of the push kernel (viterbi_fill_push.cu); identical in every CTA of
// a cluster.  S and D are the only columns that must be in shared memory; S(pos-1), the T
// columns and the out-table join them when they fit.
// ---------------------------------------------------------------------------
struct PushLayout {
  uint32_t sBuf[2];    // S(pos) / S(pos-1); one buffer only when S(pos-1) lives in global scratch
  uint32_t dBuf;       // D(pos)
  uint32_t tBuf;       // k*M doubles, only if tInSmem
  uint32_t outTab;     // the CTA's out-table, only if outInSmem
  uint32_t chunk;      // staging buffer of the streamed in-table (one chunk)
  uint32_t chunkOff;   // [nChunks+1] u32: word offsets of this CTA's chunks in the global in-table
  uint32_t flag;       // [ceil(M/32)] u32 dirty bitmap: the state must push to its successors
  uint32_t queue;      // [queueCap] u16: the dirty states of the current closure level, compacted
  uint32_t queueCap;
  uint32_t appendQueue;  // 2 x [appendCap] u16: thin frontiers are queued by the pushers themselves
  uint32_t appendCap;
  uint32_t tsE;        // [4 bases][32 syms][4 observed] (score+noGap)+sub, traceback association (src/viterbi.cpp:255)
  uint32_t symScore;   // [kMaxSyms]
  uint32_t tsDext;     // [kMaxSyms] score+delExtend (src/viterbi.cpp:272)
  uint32_t tsDopen;    // [kMaxSyms] score+delOpen   (src/viterbi.cpp:273)
  uint32_t sub;        // [16]
  uint32_t tsT;        // [8] tanDup+len[i]          (src/viterbi.cpp:286)
  uint32_t len;        // [8]
  uint32_t ctl;        // 64 u32 control words: [16..47] sent[2][kMaxCluster]
  uint32_t seq;        // packed read
  uint32_t total;
};

constexpr int kPushStatesPerThread = 1;  // states a thread handles per step of a dense pass (measured on B200: 1 state x 1024
                                         // threads beats 2 x 640, 3 x 512 and 4 x 384 -- more warps hide more latency than interleaved loads)

inline PushLayout makePushLayout(uint32_t M, uint32_t k, uint32_t tInSmem, uint32_t sPrevInSmem, uint32_t outBytes,
                                 uint32_t chunkBytes, uint32_t nChunks, uint32_t maxLen, uint32_t queueCap = 0) {
  PushLayout L;
  uint32_t at = 0;
  auto take = [&](uint32_t bytes) {
    const uint32_t here = at;
    at += (bytes + 15u) & ~15u;
    return here;
  };
  L.sBuf[0] = take(M * 8);
  L.sBuf[1] = sPrevInSmem ? take(M * 8) : L.sBuf[0];
  L.dBuf = take(M * 8);
  L.tBuf = tInSmem ? take(k * M * 8) : 0;
  L.outTab = outBytes ? take(outBytes) : 0;
  L.chunk = take(chunkBytes);
  L.chunkOff = take((nChunks + 1) * 4);
  L.flag = take(((M + 31) / 32) * 4);
  L.queueCap = queueCap ? queueCap : M;  // M entries never overflow; a smaller queue defers states to the next level
  L.queue = take(L.queueCap * 2);
  L.appendCap = 1024;
  L.appendQueue = take(L.appendCap * 2);
  take(L.appendCap * 2);
  L.tsE = take(4 * 32 * 4 * 8);
  L.symScore = take(kMaxSyms * 8);
  L.tsDext = take(kMaxSyms * 8);
  L.tsDopen = take(kMaxSyms * 8);
  L.sub = take(16 * 8);
  L.tsT = take(8 * 8);
  L.len = take(8 * 8);
  L.ctl = take(64 * 4);
  L.seq = take((maxLen + 3) / 4 + 16);
  L.total = at;
  return L;
}

struct FillArgs {
  PushLayout play;
  int64_t nReads;
  int32_t maxLen;            // pred stride: every read owns (maxLen+1) columns of records
  uint32_t thinN;            // a level of at most this many states lets its pushers queue the next level themselves
  uint32_t tRecompute;       // re-derive the duplication cells from S(pos-1), S(pos-2) (k <= 2) instead of storing them
  const uint8_t* packed;     // 2-bit reads
  const int64_t* byteOff;    // [nReads]
  const int32_t* readLen;    // [nReads]
  uint8_t* pred;             // [nReads][maxLen+1][k+2][Np] predecessor records, 1 byte per DP cell
  uint8_t* predWide;         // [nReads][maxLen+1][2][nWide] high bytes of the wide states' S and D records (viterbi_device.cuh)
  double* tScratch;         // [nClusters*C][k][M] T columns when they do not fit in shared memory
  double* sScratch;          // [nClusters][2][Np] S columns of the last two positions when S(pos-1) is not in shared memory
  double* s0Scratch;         // [nClusters][Np] S0 of the next column (the emission step is fused into the predecessor pass)
  double* loglike;           // [nReads] (global mode; local mode: written by the traceback kernel)
  uint32_t* startState;      // [nReads] traceback start (padded index), global mode
  double* partVal;           // [nReads][C] local mode: per-CTA best final S ...
  uint32_t* partOrig;        //             ... its reference state index (tie-break) ...
  uint32_t* partG;           //             ... and padded index
  double* cells;             // optional debug dump of read 0: [(L+1)][nStates][k+2]
  unsigned long long* dbg;   // optional [16] profiling counters (see dnab_decoder_debug_counters)
  unsigned long long* nextRead;  // the next read to hand to a cluster (zeroed before every launch)
};

struct TracebackArgs {
  int64_t nReads;
  int32_t maxLen;
  const int32_t* readLen;
  const uint8_t* pred;
  const uint8_t* predWide;
  double* loglike;
  const uint32_t* startState;
  const double* partVal;
  const uint32_t* partOrig;
  const uint32_t* partG;
  char* decoded;             // [nReads][decodedStride]
  int32_t decodedStride;
  int32_t* decodedLen;
  int32_t* status;
  int32_t* path;             // optional [nReads][pathStride][3]
  int32_t pathStride;
  int32_t* pathLen;
};

// ---------------------------------------------------------------------------
// forward kernel (forward_kernels.cu): the destination-indexed CSR tables in reference order
// ---------------------------------------------------------------------------
struct ForwardTables {
  uint32_t nStates, k, local, nSyms;
  const uint32_t* emitOff;   // [N+1]
  const uint32_t* emitSrc;   // [nEmit]
  const uint8_t* emitMeta;   // [nEmit] symbol id | base << 5
  const uint32_t* nullOff;   // [N+1]
  const uint32_t* nullSrc;   // [nNull]
  const uint8_t* nullSym;    // [nNull]
  const uint8_t* ctx;        // [N*k]
  const uint8_t* mdl;        // [N]
  // source-indexed lists for the backward pass (destination ascending, then list order)
  const uint32_t* outEmitOff;  // [N+1]
  const uint32_t* outEmitDst;  // [nEmit]
  const uint8_t* outEmitMeta;  // [nEmit] symbol id | base << 5
  const uint32_t* outNullOff;  // [N+1]
  const uint32_t* outNullDst;  // [nNull]
  const uint8_t* outNullSym;   // [nNull]
  const double* lseTable;    // the reference's 100,001-entry log(1+exp(-x)) table (logsumexp.cpp:5-15)
  double symScore[kMaxSyms];
  double sub[16];
  double len[kMaxK > 0 ? kMaxK : 1];
  double noGap, delOpen, delExtend, delEnd, tanDup;
};

struct ForwardArgs {
  int64_t nReads;
  int32_t maxSweeps;
  const uint8_t* packed;
  const int64_t* byteOff;
  const int32_t* readLen;
  int32_t maxLen;                // F stride: every block owns (maxLen+1) columns
  double* scratch;               // [nBlocks][(10+2k)*N]: columns + the frontier queue
  double* F;                     // optional [nBlocks][maxLen+1][N][k+2]: forward cells kept for the backward pass
  double* counts;                // optional [nReads][5+k+16] posterior expected counts (needs F)
  double* loglikeBack;           // [nReads] backward log-likelihood (with counts)
  long long* sweepsBack;         // [nReads]
  double* loglike;               // [nReads]
  long long* sweeps;             // [nReads] closure sweeps summed over the columns
  int32_t* status;               // [nReads] 0 ok, 1 a closure did not settle within maxSweeps
  unsigned long long* nextRead;  // zeroed before the launch
  double* cells;                 // optional dump of read 0: [(L+1)][N][k+2]
  double* post;                  // optional [sum of L][nSyms+1]: per read base, posterior of the class of the move that emitted it
  const long long* postOff;      // [nReads] row of read r's first base in post
};

constexpr int kPostClasses = 8;  // input-symbol ids + "duplication" that dnab_posterior_batch can tell apart

cudaError_t launchForward(const ForwardTables& tb, const ForwardArgs& args, uint32_t nBlocks, uint32_t threads,
                          cudaStream_t stream);

// push kernel (viterbi_fill_push.cu) and its traceback (viterbi_traceback.cu)
cudaError_t queryMaxClustersPush(const DevTables& tb, uint32_t threads, uint32_t smemBytes, int* nClusters);
cudaError_t launchFillPush(const DevTables& tb, const FillArgs& args, uint32_t nClusters, uint32_t threads,
                           uint32_t smemBytes, cudaStream_t stream);
cudaError_t launchTraceback(const DevTables& tb, const TracebackArgs& args, cudaStream_t stream);

}  // namespace dnab
