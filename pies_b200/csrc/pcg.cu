// pcg.cu — global step of Projective Dynamics as a block-Jacobi preconditioned CG.
//
// Replaces the reference's per-substep sparse Cholesky re-factorisation and solve
// (reference Src/Solver.cpp:242-262 SimplicialLLT(S + C_t), :356 solve) with a
// matrix that is never re-assembled: A = S (built once per topology; CSR for the start
// residual, sliced ELLPACK for the iterations) + C_t, the substep's collision terms
// (point-triangle blocks w [3 -1 -1 -1; -1 1 0 0; -1 0 1 0; -1 0 0 1],
// CollisionConstraint.cpp:74-83, and the floor diagonal, :442-445), read from the contact
// lists by the start residual and from their CSR form (detect.cu, k_ccsr_fill) by the mat-vec.
// The three coordinate columns are solved together with separate CG scalars per column,
// warm-started at the current positions.
//
// Determinism: every dot product is reduced in a fixed order (per-CTA partials on a grid that
// is fixed per topology, summed by the last CTA to finish in partial order) — no float atomics.
#include <algorithm>

#include "kernels.h"
#include "common.cuh"

namespace pies {

constexpr int kPartialStride = 20;
// partial / sum slots: per-CTA partials live at partials[cta * kPartialStride + slot]; the last CTA of every
// producing kernel reduces them in a fixed order into scalars[kSums + slot], which the consumers read.
constexpr int kPA = 0;    // p.Ap                      (3)   written by spmv
constexpr int kBB = 3;    // b.b                       (3)   written by residual
constexpr int kSet0 = 6;  // r.z (3) + r.r (3), written by even iterations
constexpr int kSet1 = 12; // r.z (3) + r.r (3), written by odd iterations and by start ("iteration -1")
constexpr int kSums = 16; // offset of the reduced sums inside `scalars`

// Deterministic grid reduction without a second launch: every CTA publishes its partials, takes a ticket, and
// the CTA holding the last ticket sums all partials in a fixed order (independent of which CTA that is).
template <int K>
__device__ __forceinline__ void lastBlockReduce(float* __restrict__ partials, int slot, float* __restrict__ scalars,
                                                int* __restrict__ flag, float* smem /* K * 32 floats */) {
  __shared__ int sLast;
  if (threadIdx.x == 0) {
    __threadfence();
    unsigned t = atomicAdd(reinterpret_cast<unsigned*>(flag + 2), 1u);
    sLast = t == gridDim.x - 1 ? 1 : 0;
  }
  __syncthreads();
  if (!sLast) return;
  __threadfence();
  float v[K];
#pragma unroll
  for (int k = 0; k < K; ++k) v[k] = 0.0f;
  for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) {
    const float* p = partials + b * kPartialStride + slot;
#pragma unroll
    for (int k = 0; k < K; ++k) v[k] += __ldcg(p + k);
  }
  blockSum<K>(v, smem);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int k = 0; k < K; ++k) scalars[kSums + slot + k] = v[k];
    flag[2] = 0;
  }
}

__device__ __forceinline__ void readSums3(const float* __restrict__ scalars, int slot, float (&out)[3]) {
  out[0] = scalars[kSums + slot]; out[1] = scalars[kSums + slot + 1]; out[2] = scalars[kSums + slot + 2];
}

// Programmatic dependent launch (the two kernels of a CG iteration are launched with the stream-serialisation
// attribute): everything before pdlWait() may overlap the tail of the previous kernel, so it must only touch data
// no kernel of the solve writes (matrix, block tables); pdlWait() returns once the previous grid has completed and
// its writes are visible.  pdlLaunchDependents() lets the next kernel start its own independent prologue.
__device__ __forceinline__ void pdlWait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdlLaunchDependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// y_i = (A x)_i for one row (CSR part + collision part from the contact lists), accumulated in fp64 (float
// products are exact in double): used once per
// solve for the start residual, where b and A x agree to ~7 digits and the difference is what
// matters (velocities are position differences divided by h, so sub-ulp position errors count).
__device__ __forceinline__ void applyRowD(uint32_t i, const CsrMatrix& A, const ContactLists& c,
                                          const float4* __restrict__ x, V3 xi, double (&y)[3]) {
  y[0] = y[1] = y[2] = 0.0;
  int beg = A.rowPtr[i], end = A.rowPtr[i + 1];
  for (int k = beg; k < end; ++k) {
    double a = (double)__ldg(A.val + k);
    float4 xv = __ldg(x + __ldg(A.col + k));
    y[0] += a * (double)xv.x; y[1] += a * (double)xv.y; y[2] += a * (double)xv.z;
  }
  if (c.nodeWeights()) {
    double fw = (double)c.floorW[i];
    y[0] += fw * (double)xi.x; y[1] += fw * (double)xi.y; y[2] += fw * (double)xi.z;
  }
  if (c.nTri) {
    int cb = c.incPtr[i], ce = c.incPtr[i + 1];
    for (int k = cb; k < ce; ++k) {
      uint32_t v = c.inc[k];
      uint4 e = __ldg(c.uTri + (v >> 2));
      double wgt = (double)__ldg(c.uW + (v >> 2));
      uint32_t slot = v & 3u;
      double t[3];
      if (slot == 0) {
        float4 xb = __ldg(x + e.y), xc = __ldg(x + e.z), xd = __ldg(x + e.w);
        t[0] = 3.0 * (double)xi.x - (double)xb.x - (double)xc.x - (double)xd.x;
        t[1] = 3.0 * (double)xi.y - (double)xb.y - (double)xc.y - (double)xd.y;
        t[2] = 3.0 * (double)xi.z - (double)xb.z - (double)xc.z - (double)xd.z;
      } else {
        float4 xa = __ldg(x + e.x);
        t[0] = (double)xi.x - (double)xa.x; t[1] = (double)xi.y - (double)xa.y; t[2] = (double)xi.z - (double)xa.z;
      }
      y[0] += wgt * t[0]; y[1] += wgt * t[1]; y[2] += wgt * t[2];
    }
  }
}

// r = b - A x (fp64 accumulation) ; delta = 0 ; partial b.b
__global__ void __launch_bounds__(kThreads) k_pcg_residual(CsrMatrix A, ContactLists c, PcgWork w, const float4* __restrict__ b,
                                                           const float4* __restrict__ x, float4* __restrict__ r,
                                                           float4* __restrict__ delta, float* __restrict__ partials,
                                                           float* __restrict__ scalars, int* __restrict__ flag) {
  __shared__ float smem[128];
  float bb[3] = {0.0f, 0.0f, 0.0f};
  // one 256-row window per CTA step: all of them, or the active ones when the solve is restricted to left-over islands
  const uint32_t nWin = w.actWin ? w.actCounts[0] : (A.n + kThreads - 1) / kThreads;
  for (uint32_t wi = blockIdx.x; wi < nWin; wi += gridDim.x) {
    const uint32_t i = (w.actWin ? w.actWin[wi] : wi) * kThreads + threadIdx.x;
    if (i >= A.n || (w.big && !w.big[i])) continue;
    float4 xi4 = x[i];
    double y[3];
    applyRowD(i, A, c, x, v3(xi4), y);
    float4 bi = b[i];
    r[i] = make_float4((float)((double)bi.x - y[0]), (float)((double)bi.y - y[1]), (float)((double)bi.z - y[2]), 0.0f);
    delta[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    bb[0] += bi.x * bi.x; bb[1] += bi.y * bi.y; bb[2] += bi.z * bi.z;
  }
  blockSum<3>(bb, smem);
  if (threadIdx.x == 0) {
    float* p = partials + blockIdx.x * kPartialStride + kBB;
    p[0] = bb[0]; p[1] = bb[1]; p[2] = bb[2];
    if (blockIdx.x == 0) { flag[0] = 0; flag[1] = 0; }
  }
  lastBlockReduce<3>(partials, kBB, scalars, flag, smem);
}

// x += delta, once per solve (single rounding of the accumulated correction)
__global__ void __launch_bounds__(kThreads) k_pcg_finish(uint32_t n, float4* __restrict__ x, const float4* __restrict__ delta,
                                                         const uint8_t* __restrict__ big) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || (big && !big[i])) return;
  float4 xv = x[i], d = delta[i];
  x[i] = make_float4(xv.x + d.x, xv.y + d.y, xv.z + d.z, xv.w);
}

// Warp-per-block preconditioner application.  The block's symmetric inverse is stored as a packed lower
// triangle (m (m + 1) / 2 floats, <= 2112 B, contiguous: half the HBM stream of a full m x m block): every lane
// issues its up-to-5 independent 16 B loads at once, parks them in shared memory, and the mat-vec
// z_lane = sum_j Minv(j, lane) r_j runs from there.  Triangular numbers are distinct modulo 32, so the packed
// reads of one j are at most two-way bank conflicted.
constexpr int kPcgWarps = kThreads / 32;
constexpr int kInvFloats = 544;                 // >= 32 * 33 / 2 = 528, multiple of 32
constexpr int kInvLoads = (528 / 4 + 31) / 32;  // 16 B loads per lane for the largest block

// Asynchronous global -> shared copy of the block's inverse (cp.async, 16 B per lane per step, no registers held).
__device__ __forceinline__ void issueBlockInv(float* __restrict__ sInv, const float* __restrict__ inv, int m, int lane) {
  const int size4 = (m * (m + 1) / 2 + 3) >> 2;
  __syncwarp();  // the previous block's reads of this buffer are finished
  uint32_t dst = (uint32_t)__cvta_generic_to_shared(sInv) + 16u * lane;
  const float4* src = reinterpret_cast<const float4*>(inv) + lane;
#pragma unroll
  for (int t = 0; t < kInvLoads; ++t) {
    if (lane + 32 * t < size4)
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 512u * t), "l"(src + 32 * t) : "memory");
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
}

// z_lane = sum_j Minv(j, lane) r_j.  r is parked in shared memory (one float4 per member) so every step reads it
// with a single broadcast load instead of three shuffles; tri walks the triangular numbers j (j + 1) / 2.
__device__ __forceinline__ V3 applyBlockInv(const float* __restrict__ sInv, float4* __restrict__ sR, V3 r, int lane, int m) {
  sR[lane] = make_float4(r.x, r.y, r.z, 0.0f);
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncwarp();
  V3 z = v3(0.0f, 0.0f, 0.0f);
  const int col = lane < m ? lane : 0;
  // entry (j, col) of the packed lower triangle: row `col` up to the diagonal (consecutive), then column `col`
  // downwards (stride j + 1)
  int off = col * (col + 1) / 2;
#pragma unroll 4
  for (int j = 0; j < m; ++j) {
    const float mv = sInv[off];
    const float4 rj = sR[j];
    z.x = fmaf(mv, rj.x, z.x); z.y = fmaf(mv, rj.y, z.y); z.z = fmaf(mv, rj.z, z.z);
    off += j < col ? 1 : j + 1;
  }
  __syncwarp();  // sR is rewritten for the warp's next block
  return z;
}

// z = Minv r ; partial r.z (odd parity slot = "iteration -1") and r.r
__global__ void __launch_bounds__(kThreads, 4) k_pcg_start(PcgWork w, float* __restrict__ partials) {
  __shared__ float smem[6 * 32];
  __shared__ __align__(16) float sInv[kPcgWarps][kInvFloats];
  __shared__ float4 sR[kPcgWarps][32];
  int lane = threadIdx.x & 31;
  uint32_t warpsPerGrid = (gridDim.x * blockDim.x) >> 5;
  float acc[6] = {0, 0, 0, 0, 0, 0};
  const uint32_t nBlocks = w.actBlk ? w.actCounts[1] : *w.nBlocksDev;
  for (uint32_t bi = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; bi < nBlocks; bi += warpsPerGrid) {
    const uint32_t blk = w.actBlk ? w.actBlk[bi] : bi;
    int node = w.blockNodes[blk * 32 + lane];
    const uint2 meta = w.blockMeta[blk];
    const int m = (int)meta.y;
    issueBlockInv(sInv[threadIdx.x >> 5], w.blockInv + meta.x, m, lane);
    V3 r = v3(0.0f, 0.0f, 0.0f);
    if (node >= 0) r = v3(w.r[node]);
    V3 z = applyBlockInv(sInv[threadIdx.x >> 5], sR[threadIdx.x >> 5], r, lane, m);
    if (node >= 0) {
      w.z[node] = f4(z, 0.0f);
      acc[0] += r.x * z.x; acc[1] += r.y * z.y; acc[2] += r.z * z.z;
      acc[3] += r.x * r.x; acc[4] += r.y * r.y; acc[5] += r.z * r.z;
    }
  }
  blockSum<6>(acc, smem);
  if (threadIdx.x == 0) {
    float* p = partials + blockIdx.x * kPartialStride + kSet1;
#pragma unroll
    for (int k = 0; k < 6; ++k) p[k] = acc[k];
  }
  lastBlockReduce<6>(partials, kSet1, w.scalars, w.flag, smem);
}

// Convergence test on the latest residual norm (after start, or after the last enqueued iteration).
__global__ void k_pcg_check(float* __restrict__ scalars, int* __restrict__ flag, int set, float tol2) {
  // Already latched by an update kernel in the middle of the burst: the later launches exited early, so `set` holds an
  // older (larger) residual than the one the latch was decided on; scalars[0] is already the right one.
  if (flag[0]) return;
  float bb[3], rr[3];
  readSums3(scalars, kBB, bb);
  readSums3(scalars, set + 3, rr);
  bool conv = rr[0] <= tol2 * bb[0] && rr[1] <= tol2 * bb[1] && rr[2] <= tol2 * bb[2];
  float rel = 0.0f;
  for (int k = 0; k < 3; ++k) if (bb[k] > 0.0f) rel = fmaxf(rel, rr[k] / bb[k]);
  scalars[0] = sqrtf(rel);
  if (conv) flag[0] = 1;
}

// (A) w = A z, then locally beta = rz_new / rz_old ; p = z + beta p ; ap = w + beta ap (A p by recurrence:
// A (z + beta p) = A z + beta A p) ; partial p.ap.  Every CTA first re-evaluates the convergence test of the
// previous iteration from the same partials, so they all agree.  The solve is for the correction delta with an
// fp64 start residual, so only a few digits are asked of this recurrence.
//
// A = S + C_t, processed in windows of 256 consecutive rows (one CTA step, one warp per 32-row slice):
//   * S comes from its sliced-ELLPACK copy (system.h; rows sorted by length inside the window, slices padded and
//     column-major, so lane l finds entry k of its row at 32 k + l: conflict-free, no divergence);
//   * C_t, the substep's collision matrix, is the window's slice of the contact CSR (detect.cu, k_ccsr_fill) plus the
//     per-node diagonal;
//   * z of the window's own rows is staged too: for a body-ordered mesh almost every column of a row lies inside the
//     window, so the gather runs from shared memory; other columns fall back to a global load.
// Everything a window needs ((col, val) of both matrices, z) is copied by cp.async into one of two buffers while the
// previous window is computed, so the only exposed global latency is the first window's.  Per row the sum runs in
// CSR order: S entries, collision entries, collision diagonal.
constexpr int kWinRows = 256;    // == HostSystem::kSellWindow
constexpr int kWinSlices = kWinRows / 32;
// Staged S entries per window, two variants: 2 432 (27-node box bodies: 2 336 entries per window with padding; three CTAs
// per SM) and 4 096 (TetGen meshes: ~15 entries per row, 3 900 per window; two CTAs per SM).  Entries past the tile are
// read straight from global memory by a per-lane serial loop, which is what made the mat-vec of config 5 slow (r02e: 37 %
// of its entries took that path with the small tile).
constexpr int kWinTileSmall = 2432, kWinTileBig = 4096;
constexpr int kWinCTile = 512;   // staged collision entries per window (two per thread)
constexpr int kWinDescs = 64;    // windows of one CTA described per round (more: the pipeline drains and restarts)

// one staging buffer; everything the window's rows need except p / ap
template <int kWinTile>
struct SpmvBufT {
  float4 z[kWinRows];
  int col[kWinTile]; float val[kWinTile];
  int ccol[kWinCTile]; float cval[kWinCTile];
  uint32_t sellRow[kWinRows];
  int cPtr[kWinRows + 4];
  float cDiag[kWinRows];
  uint32_t sellPtr[kWinSlices + 4];
};
static_assert(sizeof(SpmvBufT<kWinTileSmall>) % 16 == 0 && sizeof(SpmvBufT<kWinTileBig>) % 16 == 0, "buffer halves stay 16 B aligned");

struct SpmvWindow { uint32_t base, cnt; int cbase, ccnt; uint32_t win, pad; };  // S entries [base, base + cnt), collision entries [cbase, cbase + ccnt)

__device__ __forceinline__ void cpAsync16(void* smemDst, const void* gmemSrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smemDst)), "l"(gmemSrc) : "memory");
}
__device__ __forceinline__ void cpAsync4(void* smemDst, const void* gmemSrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(smemDst)), "l"(gmemSrc) : "memory");
}

// One commit group with everything of window `wdw`: S entries (16 B granules: slices are 128 B aligned), collision
// entries (4 B: a CSR slice starts anywhere), z / sellRow / cDiag / cPtr of its rows, its slice offsets.  No register
// ever depends on the copied words, so nothing waits before the matching cp.async.wait_group.
template <int kWinTile>
__device__ __forceinline__ void stageWindow(SpmvBufT<kWinTile>& b, const CsrMatrix& A, const ContactLists& c,
                                            const float4* __restrict__ z, const SpmvWindow& m, uint32_t wdw) {
  const uint32_t t = threadIdx.x;
  const uint32_t cnt = min(m.cnt, (uint32_t)kWinTile);
  for (uint32_t i = 4u * t; i < cnt; i += 4u * kThreads) {
    cpAsync16(b.col + i, A.sellCol + m.base + i);
    cpAsync16(b.val + i, A.sellVal + m.base + i);
  }
  const int ccnt = min(m.ccnt, kWinCTile);
  for (int i = (int)t; i < ccnt; i += kThreads) {
    cpAsync4(b.ccol + i, c.cCol + m.cbase + i);
    cpAsync4(b.cval + i, c.cVal + m.cbase + i);
  }
  const uint32_t r0 = wdw * kWinRows, row = r0 + t;
  const uint32_t s0 = wdw * kWinSlices;
  if (row < A.n) cpAsync16(b.z + t, z + row);
  if (r0 + t < A.nSlices * 32u) cpAsync4(b.sellRow + t, A.sellRow + r0 + t);  // sellRow is padded to whole slices; the last window may end early
  if (row < A.n) {
    if (c.cDiag) cpAsync4(b.cDiag + t, c.cDiag + row);
    if (c.cPtr) cpAsync4(b.cPtr + t, c.cPtr + row);
  }
  if (t == 0 && c.cPtr) cpAsync4(b.cPtr + min((uint32_t)kWinRows, A.n - r0), c.cPtr + min(A.n, r0 + kWinRows));
  if (t <= (uint32_t)kWinSlices && s0 + t <= A.nSlices) cpAsync4(b.sellPtr + t, A.sellPtr + s0 + t);
  asm volatile("cp.async.commit_group;" ::: "memory");
}

template <int kWinTile, int kSpmvCtasPerSm>
__global__ void __launch_bounds__(kThreads, kSpmvCtasPerSm) k_pcg_spmv(CsrMatrix A, ContactLists c, PcgWork w,
                                                                       float* __restrict__ partials, int parity, int first,
                                                                       float tol2) {
  using SpmvBuf = SpmvBufT<kWinTile>;
  extern __shared__ __align__(16) unsigned char spmvSmem[];
  __shared__ float smem[128];
  __shared__ float sPz[kWinCTile];  // z-products of the window's collision entries (x- and y-products reuse the staged slots)
  __shared__ float sPzS[kWinTile];  // z-products of the window's S entries
  __shared__ SpmvWindow sDesc[kWinDescs];
  SpmvBuf* bufs = reinterpret_cast<SpmvBuf*>(spmvSmem);
  const float4* __restrict__ z = w.z;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // windows: all of them, or the active ones when the solve is restricted to the left-over islands (islands.cu)
  const uint32_t nWin = w.actWin ? w.actCounts[0] : (A.n + kWinRows - 1) / kWinRows;
  // descriptions of this CTA's first windows: static data, read while the previous kernel drains
  auto describe = [&](uint32_t first_w) {
    const uint32_t mine = min((uint32_t)kWinDescs, (nWin - first_w + gridDim.x - 1) / gridDim.x);
    if (threadIdx.x < mine) {
      const uint32_t wslot = first_w + threadIdx.x * gridDim.x;
      const uint32_t wd = w.actWin ? w.actWin[wslot] : wslot;
      const uint32_t s0 = wd * kWinSlices, s1 = min(A.nSlices, s0 + kWinSlices);
      SpmvWindow m;
      m.base = A.sellPtr[s0]; m.cnt = A.sellPtr[s1] - m.base;
      m.cbase = 0; m.ccnt = 0;
      if (c.cPtr) {
        const uint32_t r0 = wd * kWinRows, r1 = min(A.n, r0 + kWinRows);
        m.cbase = c.cPtr[r0]; m.ccnt = c.cPtr[r1] - m.cbase;
      }
      m.win = wd; m.pad = 0;
      sDesc[threadIdx.x] = m;
    }
    return mine;
  };
  uint32_t mineFirst = 0;
  if (blockIdx.x < nWin) mineFirst = describe(blockIdx.x);
  pdlWait();
  pdlLaunchDependents();
  // convergence state: every thread reads the same words (no barrier, one round trip)
  float rzNew[3], rzOld[3], rr[3], bb[3], beta[3] = {0.0f, 0.0f, 0.0f};
  const int prevSet = parity ? kSet0 : kSet1, olderSet = parity ? kSet1 : kSet0;
  const int done = *(volatile const int*)w.flag;
  readSums3(w.scalars, prevSet, rzNew);  // r.z and r.r written by the previous update (or start)
  readSums3(w.scalars, prevSet + 3, rr);
  readSums3(w.scalars, kBB, bb);
  if (!first) readSums3(w.scalars, olderSet, rzOld);
  if (done || (rr[0] <= tol2 * bb[0] && rr[1] <= tol2 * bb[1] && rr[2] <= tol2 * bb[2])) return;  // the update latches the flag
  if (!first) {
#pragma unroll
    for (int k = 0; k < 3; ++k) beta[k] = rzOld[k] > 0.0f ? rzNew[k] / rzOld[k] : 0.0f;
  }
  float pap[3] = {0.0f, 0.0f, 0.0f};
  // windows of this CTA: blockIdx.x, + gridDim.x, ...; described kWinDescs at a time
  for (uint32_t first_w = blockIdx.x; first_w < nWin; first_w += (uint32_t)kWinDescs * gridDim.x) {
    const uint32_t mine = first_w == blockIdx.x ? mineFirst : describe(first_w);
    __syncthreads();
    stageWindow(bufs[0], A, c, z, sDesc[0], sDesc[0].win);
    for (uint32_t i = 0; i < mine; ++i) {
      const uint32_t wdw = sDesc[i].win;
      const bool pre = i + 1 < mine;
      if (pre) stageWindow(bufs[(i + 1) & 1], A, c, z, sDesc[i + 1], sDesc[i + 1].win);
      SpmvBuf& sb = bufs[i & 1];
      const SpmvWindow cur = sDesc[i];
      if (pre) asm volatile("cp.async.wait_group 1;" ::: "memory");
      else asm volatile("cp.async.wait_group 0;" ::: "memory");
      __syncthreads();
      const int row0 = (int)(wdw * kWinRows);
      const uint32_t sl = wdw * kWinSlices + warp;
      const bool haveSlice = sl < A.nSlices;
      const uint32_t row = haveSlice ? sb.sellRow[warp * 32 + lane] : 0xffffffffu;
      const bool haveRow = row != 0xffffffffu && (!w.big || w.big[row]);
      // p / ap of the row: issued now, consumed after the loops
      float4 po = make_float4(0.0f, 0.0f, 0.0f, 0.0f), apo = po;
      if (haveRow && !first) { po = w.p[row]; apo = w.ap[row]; }
      // Phase 1, balanced over the CTA: every thread turns staged entries into products a * z[col], in place (x over
      // val, y over col, z into sPz / sPzS).  Collision entries first: contacts couple different bodies, so their
      // columns are mostly outside the window and those global gathers should be in flight while the S tile runs.
      const int ccnt = min(cur.ccnt, kWinCTile);
      float ca[2]; float4 cx[2];
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int e = (int)threadIdx.x + j * kThreads;
        ca[j] = 0.0f; cx[j] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if (e < ccnt) {
          const int cc = sb.ccol[e];
          ca[j] = sb.cval[e];
          const uint32_t loc = (uint32_t)(cc - row0);
          cx[j] = loc < (uint32_t)kWinRows ? sb.z[loc] : __ldg(z + cc);
        }
      }
      {
        const int scnt = (int)min(cur.cnt, (uint32_t)kWinTile);
        float* px = sb.val;
        float* py = reinterpret_cast<float*>(sb.col);
#pragma unroll 2
        for (int e = (int)threadIdx.x; e < scnt; e += kThreads) {
          const int cc = sb.col[e];
          const float a = sb.val[e];
          const uint32_t loc = (uint32_t)(cc - row0);
          float4 x;
          if (loc < (uint32_t)kWinRows) x = sb.z[loc]; else x = __ldg(z + cc);
          px[e] = a * x.x; py[e] = a * x.y; sPzS[e] = a * x.z;
        }
      }
      if (ccnt) {
        float* px = sb.cval;
        float* py = reinterpret_cast<float*>(sb.ccol);
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const int e = (int)threadIdx.x + j * kThreads;
          if (e < ccnt) { px[e] = ca[j] * cx[j].x; py[e] = ca[j] * cx[j].y; sPz[e] = ca[j] * cx[j].z; }
        }
      }
      __syncthreads();
      // Phase 2, one warp per slice: the row's products in CSR order; entry k of this lane's row sits at
      // sbase + 32 k + lane of the window's block (conflict-free)
      V3 y = v3(0.0f, 0.0f, 0.0f);
      if (haveSlice) {
        const uint32_t sbase = sb.sellPtr[warp] - cur.base;
        const int len = (int)((sb.sellPtr[warp + 1] - sb.sellPtr[warp]) >> 5);
        const float* px = sb.val;
        const float* py = reinterpret_cast<const float*>(sb.col);
        const int kIn = min(len, (int)(((uint32_t)kWinTile > sbase ? (uint32_t)kWinTile - sbase : 0u) >> 5));  // steps wholly inside the staged tile
#pragma unroll 4
        for (int k = 0; k < kIn; ++k) {
          const uint32_t o = sbase + 32u * k + lane;
          y.x += px[o]; y.y += py[o]; y.z += sPzS[o];
        }
        for (int k = kIn; k < len; ++k) {  // past the staged tile: straight from global memory
          const uint32_t o = sbase + 32u * k + lane;
          const int cc = __ldcs(A.sellCol + cur.base + o);
          const float a = __ldcs(A.sellVal + cur.base + o);
          const float4 x = __ldg(z + cc);
          y.x = fmaf(a, x.x, y.x); y.y = fmaf(a, x.y, y.y); y.z = fmaf(a, x.z, y.z);
        }
      }
      if (haveRow) {
        const uint32_t lr = row - (uint32_t)row0;
        // C_t, per row: its products in CSR order (entries past the staged tile straight from global memory)
        if (c.cPtr) {
          const float* px = sb.cval;
          const float* py = reinterpret_cast<const float*>(sb.ccol);
          const int cb = sb.cPtr[lr] - cur.cbase, cf = sb.cPtr[lr + 1] - cur.cbase;
          for (int e = cb; e < cf; ++e) {
            if (e < kWinCTile) { y.x += px[e]; y.y += py[e]; y.z += sPz[e]; }
            else {
              const float a = c.cVal[cur.cbase + e];
              const float4 x = __ldg(z + c.cCol[cur.cbase + e]);
              y.x = fmaf(a, x.x, y.x); y.y = fmaf(a, x.y, y.y); y.z = fmaf(a, x.z, y.z);
            }
          }
        }
        const float dg = c.cDiag ? sb.cDiag[lr] : 0.0f;
        const float4 zi = sb.z[lr];
        y.x = fmaf(dg, zi.x, y.x); y.y = fmaf(dg, zi.y, y.y); y.z = fmaf(dg, zi.z, y.z);
        V3 pi = v3(zi);
        if (!first) {
          pi = v3(fmaf(beta[0], po.x, zi.x), fmaf(beta[1], po.y, zi.y), fmaf(beta[2], po.z, zi.z));
          y = v3(fmaf(beta[0], apo.x, y.x), fmaf(beta[1], apo.y, y.y), fmaf(beta[2], apo.z, y.z));
        }
        w.p[row] = f4(pi, 0.0f);
        w.ap[row] = f4(y, 0.0f);
        pap[0] += pi.x * y.x; pap[1] += pi.y * y.y; pap[2] += pi.z * y.z;
      }
      __syncthreads();  // this buffer (and sPz) is refilled by the next round
    }
  }
  blockSum<3>(pap, smem);
  if (threadIdx.x == 0) {
    float* p = partials + blockIdx.x * kPartialStride + kPA;
    p[0] = pap[0]; p[1] = pap[1]; p[2] = pap[2];
  }
  lastBlockReduce<3>(partials, kPA, w.scalars, w.flag, smem);
}

// (B) alpha = rz / pAp ; delta += alpha p ; r -= alpha ap ; z = Minv r ; partial r.z (parity slot), r.r.
// Re-evaluates the same convergence test as (A) first: if (A) stopped, this stops too and CTA 0 latches the flag.
__global__ void __launch_bounds__(kThreads, 4) k_pcg_update(PcgWork w, float4* __restrict__ x, float* __restrict__ partials,
                                                         int parity, float tol2) {
  __shared__ float smem[6 * 32];
  __shared__ __align__(16) float sInv[kPcgWarps][kInvFloats];
  __shared__ float4 sR[kPcgWarps][32];
  // block tables are per-substep data no kernel of the solve writes: fetch the first block while the mat-vec drains
  const int lane = threadIdx.x & 31;
  const uint32_t warpsPerGrid = (gridDim.x * blockDim.x) >> 5;
  const uint32_t nBlocks = w.actBlk ? w.actCounts[1] : *w.nBlocksDev;
  uint32_t bi = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int nodeNext = -1;
  uint2 metaNext = make_uint2(0u, 0u);
  if (bi < nBlocks) { const uint32_t blk = w.actBlk ? w.actBlk[bi] : bi; nodeNext = w.blockNodes[blk * 32 + lane]; metaNext = w.blockMeta[blk]; }
  pdlWait();
  pdlLaunchDependents();
  if (*(volatile const int*)w.flag) return;
  float rz[3], pap[3], alpha[3], rr[3], bb[3];
  const int prevSet = parity ? kSet0 : kSet1, mySet = parity ? kSet1 : kSet0;
  readSums3(w.scalars, prevSet + 3, rr);
  readSums3(w.scalars, kBB, bb);
  if (rr[0] <= tol2 * bb[0] && rr[1] <= tol2 * bb[1] && rr[2] <= tol2 * bb[2]) {
    // Late CTAs may already see the flag and leave through ctaConverged: same outcome.
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      float rel = 0.0f;
      for (int k = 0; k < 3; ++k) if (bb[k] > 0.0f) rel = fmaxf(rel, rr[k] / bb[k]);
      w.scalars[0] = sqrtf(rel);
      w.flag[0] = 1;
    }
    return;
  }
  readSums3(w.scalars, prevSet, rz);  // r.z of the previous step
  readSums3(w.scalars, kPA, pap);
#pragma unroll
  for (int k = 0; k < 3; ++k) alpha[k] = pap[k] > 0.0f ? rz[k] / pap[k] : 0.0f;
  float acc[6] = {0, 0, 0, 0, 0, 0};
  // software pipeline: the next block's membership and location are fetched while this block is processed
  for (; bi < nBlocks; bi += warpsPerGrid) {
    const int node = nodeNext;
    const int m = (int)metaNext.y;
    issueBlockInv(sInv[threadIdx.x >> 5], w.blockInv + metaNext.x, m, lane);
    V3 r = v3(0.0f, 0.0f, 0.0f);
    float4 xv, pv4, ap4, r4;
    if (node >= 0) { xv = x[node]; pv4 = w.p[node]; ap4 = w.ap[node]; r4 = w.r[node]; }
    if (bi + warpsPerGrid < nBlocks) {
      const uint32_t nb = w.actBlk ? w.actBlk[bi + warpsPerGrid] : bi + warpsPerGrid;
      nodeNext = w.blockNodes[nb * 32 + lane]; metaNext = w.blockMeta[nb];
    }
    if (node >= 0) {
      V3 pv = v3(pv4), ap = v3(ap4);
      r = v3(r4);
      xv.x += alpha[0] * pv.x; xv.y += alpha[1] * pv.y; xv.z += alpha[2] * pv.z;
      r.x -= alpha[0] * ap.x; r.y -= alpha[1] * ap.y; r.z -= alpha[2] * ap.z;
      x[node] = xv;
      w.r[node] = f4(r, 0.0f);
    }
    V3 z = applyBlockInv(sInv[threadIdx.x >> 5], sR[threadIdx.x >> 5], r, lane, m);
    if (node >= 0) {
      w.z[node] = f4(z, 0.0f);
      acc[0] += r.x * z.x; acc[1] += r.y * z.y; acc[2] += r.z * z.z;
      acc[3] += r.x * r.x; acc[4] += r.y * r.y; acc[5] += r.z * r.z;
    }
  }
  blockSum<6>(acc, smem);
  if (threadIdx.x == 0) {
    float* pp = partials + blockIdx.x * kPartialStride + mySet;
#pragma unroll
    for (int k = 0; k < 6; ++k) pp[k] = acc[k];
    if (blockIdx.x == 0) w.flag[1] += 1;
  }
  lastBlockReduce<6>(partials, mySet, w.scalars, w.flag, smem);
}

int launchPcgInit(cudaStream_t s, const CsrMatrix& A, const ContactLists& c, const PcgWork& w, const float4* b,
                  const float4* x, float tol) {
  k_pcg_residual<<<kReduceBlocks, kThreads, 0, s>>>(A, c, w, b, x, w.r, w.delta, w.partials, w.scalars, w.flag);
  k_pcg_start<<<kReduceBlocks, kThreads, 0, s>>>(w, w.partials);
  k_pcg_check<<<1, 1, 0, s>>>(w.scalars, w.flag, kSet1, tol * tol);
  return 3;
}

// One CG iteration = two kernels.  `it` = iteration index within the solve.
int launchPcgSpmv(cudaStream_t s, const CsrMatrix& A, const ContactLists& c, const PcgWork& w, float tol, int it) {
  const uint32_t nWin = (A.n + kWinRows - 1) / kWinRows;
  if (!nWin) return 0;
  // tile variant by the matrix's average padded entries per window (fixed per topology, like the grid)
  const bool big = A.sellEntries / nWin > (uint64_t)(kWinTileSmall * 9 / 10);
  const size_t smem = big ? 2 * sizeof(SpmvBufT<kWinTileBig>) : 2 * sizeof(SpmvBufT<kWinTileSmall>);
  const int ctas = big ? 2 : 3;
  auto kernel = big ? k_pcg_spmv<kWinTileBig, 2> : k_pcg_spmv<kWinTileSmall, 3>;
  // > 48 KB of dynamic shared memory needs the opt-in (a per-device function attribute: renewed once per solve)
  if (it == 0) cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  const int grid = (int)std::min<uint32_t>(nWin, (uint32_t)(kNumSMs * ctas));  // fixed per topology => fixed-order reduction
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(kThreads); cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kernel, A, c, w, w.partials, it & 1, it == 0 ? 1 : 0, tol * tol);
  return 1;
}

int launchPcgUpdate(cudaStream_t s, const PcgWork& w, float tol, int it) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(kReduceBlocks); cfg.blockDim = dim3(kThreads); cfg.dynamicSmemBytes = 0; cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, k_pcg_update, w, w.delta, w.partials, it & 1, tol * tol);
  return 1;
}

int launchPcgIteration(cudaStream_t s, const CsrMatrix& A, const ContactLists& c, const PcgWork& w, float tol, int it) {
  return launchPcgSpmv(s, A, c, w, tol, it) + launchPcgUpdate(s, w, tol, it);
}

// Latches the convergence flag after the last enqueued iteration (the host reads it next).
int launchPcgCheck(cudaStream_t s, const PcgWork& w, float tol, int lastIt) {
  k_pcg_check<<<1, 1, 0, s>>>(w.scalars, w.flag, (lastIt & 1) ? kSet1 : kSet0, tol * tol);
  return 1;
}

int launchPcgFinish(cudaStream_t s, const PcgWork& w, uint32_t n, float4* x) {
  k_pcg_finish<<<(n + kThreads - 1) / kThreads, kThreads, 0, s>>>(n, x, w.delta, w.big);
  return 1;
}

// Loads this file's kernels now (CUDA loads a kernel lazily at its first launch; for the collision kernels that
// would be the first contact tick of a run, ~1 ms each in the middle of the simulation).
void preloadPcgKernels() {
  cudaFuncAttributes a;
  cudaFuncGetAttributes(&a, k_pcg_residual);
  cudaFuncGetAttributes(&a, k_pcg_finish);
  cudaFuncGetAttributes(&a, k_pcg_start);
  cudaFuncGetAttributes(&a, k_pcg_check);
  cudaFuncGetAttributes(&a, k_pcg_spmv<kWinTileSmall, 3>);
  cudaFuncGetAttributes(&a, k_pcg_spmv<kWinTileBig, 2>);
  cudaFuncGetAttributes(&a, k_pcg_update);
}

}  // namespace pies
