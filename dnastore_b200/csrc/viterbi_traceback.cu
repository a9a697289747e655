// viterbiTracebackKernel: the traceback of the Viterbi fill (reference src/viterbi.cpp:195-304) for the
// one-read-per-cluster push kernel (viterbi_fill_push.cu), on the device, one thread per read.
//
// The fill leaves one predecessor byte per DP cell (two for the S and D cells of wide states, the high
// byte in the side plane), evaluated with the traceback's own floating-point association and candidate
// order; this kernel follows those records from the end cell back to the start state and decodes each
// against the state blocks (viterbi_device.cuh) that the host built for the same partition.  It writes the decoded input-symbol string, the log-likelihood (local mode: the best
// of the per-CTA maxima the fill left) and the status of every read, and optionally the path of cells.
#include <cuda_runtime.h>

#include <cstdint>

#include "viterbi_kernels.h"

namespace dnab {

__device__ __forceinline__ double negInf() { return __longlong_as_double(0xFFF0000000000000LL); }

// reference src/viterbi.cpp:195-304: loop :247, emitted symbols :299-300
__global__ void viterbiTracebackKernel(const DevTables tb, const TracebackArgs args) {
  const int64_t read = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (read >= args.nReads) return;
  const uint32_t C = tb.C, M = tb.M, k = tb.k, Np = C * M;
  const int32_t L = args.readLen[read];
  const double NEG = negInf();

  uint32_t g;
  double ll;
  if (!tb.local) {
    g = args.startState[read];
    ll = args.loglike[read];
  } else {
    double bv = NEG;
    uint32_t bo = 0xFFFFFFFFu, bg = 0;
    for (uint32_t r = 0; r < C; ++r) {
      const double v = args.partVal[read * C + r];
      const uint32_t o = args.partOrig[read * C + r];
      if (o == 0xFFFFFFFFu) continue;
      if (v > bv || (v == bv && o < bo)) {
        bv = v;
        bo = o;
        bg = args.partG[read * C + r];
      }
    }
    g = bg;
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

  const uint8_t* predRead = args.pred + (size_t)read * (size_t)(args.maxLen + 1) * (k + 2) * Np;
  int32_t pos = L;
  uint32_t mut = 0;
  // symbols are produced last-to-first: fill the caller's slot from its END, then shift
  const int32_t cap = args.decodedStride;
  while (pos >= 0 && g != tb.startG) {
    if (path) {
      if (nPath < args.pathStride) {
        path[3 * nPath] = (int32_t)tb.origId[g];
        path[3 * nPath + 1] = pos;
        path[3 * nPath + 2] = (int32_t)mut;
      } else
        status = DNAB_READ_OVERFLOW_;
    }
    ++nPath;
    uint32_t p = predRead[((size_t)pos * (k + 2) + mut) * Np + g];
    const uint32_t* blkp = tb.blocks + tb.blockOff[g];
    uint32_t nE = hdrNEmit(blkp[0]), nIn = hdrNIn(blkp[0]);
    const uint2* edges = reinterpret_cast<const uint2*>(blkp + 2);
    uint32_t none = kNoPred;
    if (nE == kHdrWide) {  // wide state: 16-bit counts, and the S and D records' high bytes in the side plane
      nE = blkp[2] & 0xFFFFu;
      nIn = blkp[2] >> 16;
      edges = reinterpret_cast<const uint2*>(blkp + 4);
      if (mut < 2) {
        p |= (uint32_t)args.predWide[((size_t)read * (args.maxLen + 1) + pos) * 2 * tb.nWide + mut * tb.nWide + blkp[3]] << 8;
        none = kWideNoPred;
      }
    }
    if (p == none) {
      status = DNAB_READ_TRACEBACK_FAILED_;
      break;
    }
    auto srcOf = [&](uint2 e) { return edgeRank(e.x) * M + edgeOff(e.x) / 8; };
    uint32_t sym = 0;
    if (mut == 0) {
      if (p < nIn) {  // incoming emit edge (previous column) or null edge (same column)
        const uint2 e = edges[p];
        sym = edgeSymOff(e.y) / 8;
        g = srcOf(e);
        if (p < nE) --pos;
      } else if (p == nIn) {
        mut = 1;
      } else if (p == nIn + 1) {
        mut = 2;
        --pos;
      } else {
        g = tb.startG;  // local mode, pos == 0: jump to (0,0,S)
      }
    } else if (mut == 1) {
      if (p < 2 * nE) {
        const uint2 e = edges[p >> 1];
        sym = edgeSymOff(e.y) / 8;
        g = srcOf(e);
        mut = (p & 1) ? 0 : 1;
      } else {
        const uint2 e = edges[p - nE];  // null edge number p-2*nE sits after the nE emit edges
        sym = edgeSymOff(e.y) / 8;
        g = srcOf(e);
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

cudaError_t launchTraceback(const DevTables& tb, const TracebackArgs& args, cudaStream_t stream) {
  const int threads = 64;
  const int blocks = (int)((args.nReads + threads - 1) / threads);
  viterbiTracebackKernel<<<blocks, threads, 0, stream>>>(tb, args);
  return cudaGetLastError();
}

}  // namespace dnab
