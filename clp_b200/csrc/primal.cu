// primal.cu -- the primal simplex iteration, device resident.
//
// Restates, with the dual engine's factors, FTRAN / BTRAN / PRICE kernels and eta file:
//   ClpPrimalColumnSteepest::pivotColumn     src/ClpPrimalColumnSteepest.cpp (mode 0, exact Devex)
//   ClpPrimalColumnDantzig::pivotColumn      src/ClpPrimalColumnDantzig.cpp:57
//   ClpSimplexPrimal::primalRow              src/ClpSimplexPrimal.cpp:1877 (Harris two-pass ratio test)
//   ClpPrimalColumnSteepest::djsAndDevex2    src/ClpPrimalColumnSteepest.cpp:1470 (d_j and Devex update)
//   ClpSimplexPrimal::updatePrimalsInPrimal  src/ClpSimplexPrimal.cpp:2584 + ClpSimplex::housekeeping
// One iteration (ClpSimplexPrimal::whileIterating :613 order):
//   unpack a_q -> FTRAN -> ratio test (2 kernels) -> BTRAN(e_r) -> PRICE -> d_j / Devex update with the
//   next CHUZC fused in -> x_B update + eta append + housekeeping (tail decodes the next entering column)
// Every kernel reads its scalars from IterState, so the launch sequence does not depend on the data and
// is captured once as a CUDA graph.  All reductions are packed-key atomicMax/Min or fixed-order sums.
#include "kernels_common.cuh"

namespace clpb {

enum : int { TAIL_PRIMAL_RATIO = 8, TAIL_PRIMAL_UPDATE = 9 };

// Pricing key of nonbasic sequence j (0 = not a candidate).  Score d_j^2 / w_j (Devex) or d_j^2
// (Dantzig).  The low 20 bits of the score's bit pattern hold 0xFFFFF - j: among scores that agree in
// their upper 44 bits the smaller sequence wins.
__device__ __forceinline__ unsigned long long pchuzc_key(unsigned char st, double dj, double w, double tol,
                                                         int dantzig, int j)
{
  bool cand;
  if (st == atLowerBound)
    cand = dj < -tol;
  else if (st == atUpperBound)
    cand = dj > tol;
  else if (st == isFree || st == superBasic)
    cand = fabs(dj) > tol;
  else
    cand = false; // basic, fixed
  if (!cand)
    return 0ull;
  const double score = dantzig ? dj * dj : dj * dj / w;
  if (!(score > 0.0))
    return 0ull;
  return ((unsigned long long)__double_as_longlong(score) & ~0xFFFFFull) | (unsigned long long)(0xFFFFF - j);
}

// decode the CHUZC key into seqIn / primalDir / primalDj (single thread)
__device__ __forceinline__ void pchuzc_finish_body(const DeviceModel &d, unsigned long long key)
{
  IterState *st = d.st;
  if (st->numEtas >= d.tmax) {
    st->stop = STOP_ETAS_FULL;
    return;
  }
  if (key == 0ull) {
    st->stop = STOP_NO_COLUMN;
    return;
  }
  const int q = 0xFFFFF - (int)(key & 0xFFFFFull);
  const double dj = __ldcg(d.dj + q);
  st->seqIn = q;
  st->primalDj = dj;
  st->primalDir = dj < 0.0 ? 1 : -1;
  st->primalFlip = 0;
  st->infeasChanged = 0;
  st->ratioBits = 0x7FF0000000000000ull; // +inf
  st->ratioKey = 0ull;
}

// ------------------------------------------------------------------ stand-alone CHUZC
__global__ void __launch_bounds__(256) primal_chuzc_kernel(DeviceModel d)
{
  if (!iter_active(d.st))
    return;
  unsigned long long best = 0ull;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < d.nm; j += gridDim.x * blockDim.x)
    if (!d.colFlagged[j])
      best = max(best, pchuzc_key(d.status[j], d.dj[j], d.devex[j], d.dualTolerance, d.primalDantzig, j));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1)
    best = max(best, __shfl_xor_sync(0xffffffffu, best, o));
  if ((threadIdx.x & 31) == 0 && best != 0ull)
    atomicMax(&d.st->pchuzcKey, best);
}
__global__ void primal_chuzc_finish_kernel(DeviceModel d)
{
  if (!iter_active(d.st))
    return;
  const unsigned long long key = d.st->pchuzcKey;
  d.st->pchuzcKey = 0ull;
  pchuzc_finish_body(d, key);
}
void launch_primal_chuzc(const DeviceModel &d, cudaStream_t s)
{
  int blocks = (d.nm + 255) / 256;
  if (blocks > 148 * 4)
    blocks = 148 * 4;
  primal_chuzc_kernel<<<blocks, 256, 0, s>>>(d);
  primal_chuzc_finish_kernel<<<1, 1, 0, s>>>(d);
}

// ------------------------------------------------------------------ entering column
// rhs3[0..m) = column seqIn of [A | -I]; thread per row, the column's entries staged through shared memory
__global__ void __launch_bounds__(256) primal_unpack_kernel(DeviceModel d)
{
  if (!iter_active(d.st))
    return;
  __shared__ int sRow[256];
  __shared__ double sVal[256];
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  const int q = d.st->seqIn;
  double aq = 0.0;
  if (q >= d.n) {
    aq = row == q - d.n ? -1.0 : 0.0;
  } else {
    const int e0 = d.colStart[q], e1 = d.colStart[q + 1];
    for (int c0 = e0; c0 < e1; c0 += 256) {
      const int e = c0 + threadIdx.x;
      sRow[threadIdx.x] = e < e1 ? d.rowIdx[e] : -1;
      sVal[threadIdx.x] = e < e1 ? d.val[e] : 0.0;
      __syncthreads();
      const int cnt = min(256, e1 - c0);
      for (int t = 0; t < cnt; t++)
        if (sRow[t] == row)
          aq = sVal[t];
      __syncthreads();
    }
  }
  if (row < d.m)
    d.rhs3[row] = aq;
}

// ------------------------------------------------------------------ ratio test
// Step at which basic position p blocks when x_q moves by dir*theta, x_B -= dir*theta*alpha.
// relax = primal tolerance for pass 1 (Harris), 0 for the exact step.  Returns false if p does not block.
// Phase 1: an infeasible basic blocks only at its far bound (it may pass the near bound into
// feasibility); if that bound is infinite it blocks at the near bound.
// toUpper: the bound it blocks at is its upper bound.
__device__ __forceinline__ bool primal_block(double a, double x, double lo, double up, double tol, int phase,
                                             double relax, double &ratio, bool &toUpper)
{
  if (a > 0.0) { // x decreases
    toUpper = false;
    if (phase == 1 && x < lo - tol)
      return false;
    if (phase == 1 && x > up + tol && lo <= -kInf)
      toUpper = true;
    const double bound = toUpper ? up : lo;
    if (bound <= -kInf)
      return false;
    ratio = (x - bound + relax) / a;
  } else { // x increases
    toUpper = true;
    if (phase == 1 && x > up + tol)
      return false;
    if (phase == 1 && x < lo - tol && up >= kInf)
      toUpper = false;
    const double bound = toUpper ? up : lo;
    if (bound >= kInf)
      return false;
    ratio = (bound - x + relax) / -a;
  }
  if (!(ratio > 0.0))
    ratio = 0.0;
  return true;
}

// pass 1: relaxed minimum step over the positions with |alpha| >= acceptablePivot; per-CTA partial sums
// of the entering column's Devex reference weight (sum of alpha_p^2 over reference basics)
__global__ void __launch_bounds__(256) primal_ratio1_kernel(DeviceModel d)
{
  __shared__ double sPart[8];
  IterState *st = d.st;
  if (!iter_active(st))
    return;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  const int dir = st->primalDir, phase = st->primalPhase;
  const double tol = d.primalTolerance;
  unsigned long long best = 0x7FF0000000000000ull;
  double ref = 0.0;
  if (p < d.m) {
    const double alpha = d.rhs3[p];
    const int seq = d.pivotVariable[p];
    if (d.devexRef[seq])
      ref = alpha * alpha;
    const double a = dir * alpha;
    double ratio;
    bool toUpper;
    if (fabs(a) >= st->acceptablePivot && primal_block(a, d.sol[seq], d.lower[seq], d.upper[seq], tol, phase, tol, ratio, toUpper))
      best = (unsigned long long)__double_as_longlong(ratio);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1)
    best = min(best, __shfl_xor_sync(0xffffffffu, best, o));
  ref = warp_sum(ref);
  if ((threadIdx.x & 31) == 0) {
    if (best != 0x7FF0000000000000ull)
      atomicMin(&st->ratioBits, best);
    sPart[threadIdx.x >> 5] = ref;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < 8; w++)
      s += sPart[w];
    d.ratioPart[blockIdx.x] = s;
  }
}

// Tail of the ratio test (single thread): the entering variable's own range competes with the rows
// (bound flip), otherwise the packed key names the pivot row; step length, leaving variable, exact
// Devex reference weight of the entering column.
__device__ __forceinline__ void primal_ratio_tail(const DeviceModel &d)
{
  IterState *st = d.st;
  const int q = st->seqIn, dir = st->primalDir;
  double wq = d.devexRef[q] ? 1.0 : 0.0;
  for (int b = 0; b < (int)gridDim.x; b++)
    wq += __ldcg(d.ratioPart + b);
  st->devexQ = wq < 1.0 ? 1.0 : wq;
  const double range = d.upper[q] - d.lower[q];
  const double thetaMax = __longlong_as_double((long long)atomicAdd(&st->ratioBits, 0ull));
  const unsigned long long key = atomicExch(&st->ratioKey, 0ull);
  if (range < 1.0e29 && range <= thetaMax) {
    st->primalFlip = 1;
    st->pivotRow = 0; // BTRAN / PRICE of this iteration run on a harmless row; nothing reads them
    st->thetaPrimal = dir * range;
    st->alphaCol = 1.0;
    return;
  }
  if (key == 0ull) {
    st->stop = STOP_UNBOUNDED;
    return;
  }
  const int r = 0xFFFFF - (int)(key & 0xFFFFFull);
  const int seq = d.pivotVariable[r];
  const double alpha = __ldcg(d.rhs3 + r);
  const double a = dir * alpha;
  double ratio = 0.0;
  bool toUpper = false;
  primal_block(a, d.sol[seq], d.lower[seq], d.upper[seq], d.primalTolerance, st->primalPhase, 0.0, ratio, toUpper);
  st->pivotRow = r;
  st->seqOut = seq;
  st->alphaCol = alpha;
  st->sigma = toUpper ? 1 : -1; // the bound the leaving variable ends at
  st->thetaPrimal = dir * ratio;
}

// pass 2: among the positions whose exact step is within the relaxed minimum, the largest |alpha|
// (packed key; equal |alpha| in the upper 44 bits: the smaller position wins)
__global__ void __launch_bounds__(256) primal_ratio2_kernel(DeviceModel d)
{
  IterState *st = d.st;
  if (!iter_active(st))
    return;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  const int dir = st->primalDir, phase = st->primalPhase;
  const double thetaMax = __longlong_as_double((long long)st->ratioBits);
  unsigned long long best = 0ull;
  if (p < d.m) {
    const double alpha = d.rhs3[p];
    const double a = dir * alpha;
    const int seq = d.pivotVariable[p];
    double ratio;
    bool toUpper;
    if (fabs(a) >= st->acceptablePivot &&
        primal_block(a, d.sol[seq], d.lower[seq], d.upper[seq], d.primalTolerance, phase, 0.0, ratio, toUpper) &&
        ratio <= thetaMax)
      best = ((unsigned long long)__double_as_longlong(fabs(alpha)) & ~0xFFFFFull) | (unsigned long long)(0xFFFFF - p);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1)
    best = max(best, __shfl_xor_sync(0xffffffffu, best, o));
  if ((threadIdx.x & 31) == 0 && best != 0ull)
    atomicMax(&st->ratioKey, best);
  if (!last_block_done(d.tailCounter + TAIL_PRIMAL_RATIO))
    return;
  if (threadIdx.x == 0)
    primal_ratio_tail(d);
}

void launch_primal_ratio(const DeviceModel &d, cudaStream_t s)
{
  const int blocks = (d.m + 255) / 256;
  primal_ratio1_kernel<<<blocks, 256, 0, s>>>(d);
  primal_ratio2_kernel<<<blocks, 256, 0, s>>>(d);
}

// ------------------------------------------------------------------ d_j / Devex update + next CHUZC
// alpha_rj = rho^T a_j: PRICE wrote the structurals, a slack's column is -e_i
__device__ __forceinline__ double row_entry(const DeviceModel &d, int j)
{
  return j < d.n ? d.alphaRow[j] : -d.rho[j - d.n];
}

__global__ void __launch_bounds__(256) primal_dj_kernel(DeviceModel d)
{
  IterState *st = d.st;
  if (!iter_active(st))
    return;
  const int q = st->seqIn, out = st->seqOut, flip = st->primalFlip;
  const double alphaR = st->alphaCol;
  if (!flip) {
    // pivot accuracy gate (ClpSimplexPrimal::pivotResult :3304): the pivot from the FTRAN column against
    // the same entry from the BTRAN row.  Every thread decides alike; nothing is written on failure.
    const double ar = row_entry(d, q);
    const double err = fabs(ar - alphaR) / (1.0 + fabs(alphaR));
    if (!(fabs(alphaR) >= 1.0e-9) || !(err <= 1.0e-6)) {
      if (blockIdx.x == 0 && threadIdx.x == 0)
        st->stop = STOP_INACCURATE;
      return;
    }
  }
  const double thetaD = flip ? 0.0 : st->primalDj / alphaR;
  const double wq = st->devexQ;
  const double tol = d.dualTolerance;
  unsigned long long best = 0ull;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < d.nm; j += gridDim.x * blockDim.x) {
    unsigned char s = d.status[j];
    double dj = d.dj[j];
    double w = d.devex[j];
    if (flip) {
      if (j == q)
        s = s == atLowerBound ? atUpperBound : atLowerBound;
    } else if (j == q) {
      d.dj[j] = 0.0;
      continue; // becomes basic
    } else if (j == out) {
      dj = -thetaD;
      w = wq / (alphaR * alphaR);
      w = w < 1.0 ? 1.0 : w;
      s = d.lower[j] == d.upper[j] ? isFixed : (st->sigma < 0 ? atLowerBound : atUpperBound);
      d.dj[j] = dj;
      d.devex[j] = w;
    } else if (s != basic && s != isFixed) {
      const double arj = row_entry(d, j);
      if (arj != 0.0) {
        dj -= thetaD * arj;
        d.dj[j] = dj;
        if (!d.primalDantzig) {
          const double ratio = arj / alphaR;
          const double cand = ratio * ratio * wq;
          if (cand > w) {
            w = cand;
            d.devex[j] = w;
          }
        }
      }
    }
    if (!d.colFlagged[j])
      best = max(best, pchuzc_key(s, dj, w, tol, d.primalDantzig, j));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1)
    best = max(best, __shfl_xor_sync(0xffffffffu, best, o));
  if ((threadIdx.x & 31) == 0 && best != 0ull)
    atomicMax(&st->pchuzcKey, best);
}

// ------------------------------------------------------------------ x_B update, eta, housekeeping
__device__ __forceinline__ int infeas_state(double x, double lo, double up, double tol)
{
  return x < lo - tol ? -1 : (x > up + tol ? 1 : 0);
}

__device__ __forceinline__ void primal_fixup_body(const DeviceModel &d)
{
  IterState *st = d.st;
  IterRecord &rec = d.rec[st->iterations % d.recCap];
  const int q = st->seqIn;
  const double delta = st->thetaPrimal;
  if (st->primalFlip) {
    const bool toUpper = d.status[q] == atLowerBound;
    d.status[q] = toUpper ? atUpperBound : atLowerBound;
    d.sol[q] = toUpper ? d.upper[q] : d.lower[q];
  } else {
    const int r = st->pivotRow, out = st->seqOut;
    const double xOut = d.sol[out];
    if (st->primalPhase == 1 && infeas_state(xOut, d.lower[out], d.upper[out], d.primalTolerance) != 0)
      st->infeasChanged = 1; // an infeasible basic left: its phase-1 cost goes
    d.sol[q] += delta;
    d.sol[out] = st->sigma < 0 ? d.lower[out] : d.upper[out];
    d.status[q] = basic;
    d.status[out] = d.lower[out] == d.upper[out] ? isFixed : (st->sigma < 0 ? atLowerBound : atUpperBound);
    d.pivotVariable[r] = q;
    const int t = st->numEtas;
    d.etaPos[t] = r;
    d.etaPrevSame[t] = d.etaLastOfPos[r];
    d.etaLastOfPos[r] = t;
    st->numEtas = t + 1;
  }
  rec.stop = 0;
  rec.pivotRow = st->primalFlip ? -1 : st->pivotRow;
  rec.seqIn = q;
  rec.seqOut = st->primalFlip ? q : st->seqOut;
  rec.sigma = st->sigma;
  rec.numFlips = st->primalFlip;
  rec.thetaDual = st->primalDj;
  rec.thetaPrimal = delta;
  rec.alphaRow = st->devexQ;
  rec.alphaCol = st->alphaCol;
  rec.infeas = 0.0;
  st->iterations += 1;
}

//   CTAs [0, etaBlocks)    : new row of Ginv / column of GinvT (eta_append_row; nu from this iteration's BTRAN)
//   CTAs [etaBlocks, grid) : x_B -= delta * alpha and the new eta column, thread per position
//   tail                   : housekeeping, then decode the entering column of the next iteration
__global__ void __launch_bounds__(256) primal_update_kernel(DeviceModel d, int etaBlocks)
{
  IterState *st = d.st;
  if (!iter_active(st)) {
    if (blockIdx.x == 0 && threadIdx.x == 0)
      d.rec[st->iterations % d.recCap].stop = st->stop;
    return;
  }
  const int flip = st->primalFlip;
  if ((int)blockIdx.x < etaBlocks) {
    if (!flip)
      eta_append_row(d, blockIdx.x * 256 + threadIdx.x, etaBlocks * 256);
  } else {
    const int p = (blockIdx.x - etaBlocks) * 256 + threadIdx.x;
    if (p < d.m) {
      const int r = flip ? -1 : st->pivotRow;
      const double a = d.rhs3[p];
      if (!flip)
        d.W[(size_t)p * d.tmax + st->numEtas] = (p == r) ? a - 1.0 : a;
      if (p != r && a != 0.0) {
        const int seq = d.pivotVariable[p];
        const double x0 = d.sol[seq];
        const double x1 = x0 - st->thetaPrimal * a;
        d.sol[seq] = x1;
        if (st->primalPhase == 1) {
          const double lo = d.lower[seq], up = d.upper[seq], tol = d.primalTolerance;
          if (infeas_state(x0, lo, up, tol) != infeas_state(x1, lo, up, tol))
            atomicOr(&st->infeasChanged, 1);
        }
      }
    }
  }
  if (!last_block_done(d.tailCounter + TAIL_PRIMAL_UPDATE))
    return;
  if (threadIdx.x == 0) {
    primal_fixup_body(d);
    const unsigned long long key = atomicExch(&st->pchuzcKey, 0ull);
    if (st->primalPhase == 1 && atomicAdd(&st->infeasChanged, 0) != 0) {
      st->stop = STOP_PHASE_COSTS;
      return;
    }
    pchuzc_finish_body(d, key);
  }
}

void launch_primal_iteration(const DeviceModel &d, cudaStream_t s)
{
  const int mBlocks = (d.m + 255) / 256;
  primal_unpack_kernel<<<mBlocks, 256, 0, s>>>(d);
  launch_ftran(d, 1, true, s);
  launch_primal_ratio(d, s);
  launch_btran_unit(d, true, s);
  launch_price(d, 0, d.n, false, s);
  int blocks = (d.nm + 255) / 256;
  if (blocks > 148 * 8)
    blocks = 148 * 8;
  primal_dj_kernel<<<blocks, 256, 0, s>>>(d);
  const int etaBlocks = (d.tmax + 1023) / 1024;
  primal_update_kernel<<<etaBlocks + mBlocks, 256, 0, s>>>(d, etaBlocks);
}

// ------------------------------------------------------------------ refresh kernels
// phase 1: cost -1 / +1 for a basic below / above its bounds, 0 otherwise; phase 2: the true costs
__global__ void primal_costs_kernel(DeviceModel d, int phase)
{
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= d.nm)
    return;
  if (phase == 2) {
    d.cost[j] = d.costTrue[j];
    return;
  }
  double c = 0.0;
  if (d.status[j] == basic)
    c = (double)infeas_state(d.sol[j], d.lower[j], d.upper[j], d.primalTolerance);
  d.cost[j] = c;
}
void launch_primal_costs(const DeviceModel &d, int phase, cudaStream_t s)
{
  primal_costs_kernel<<<(d.nm + 255) / 256, 256, 0, s>>>(d, phase);
}

// Devex reset (ClpPrimalColumnSteepest::saveWeights mode 1 in exact Devex): every weight 1, the reference
// framework is the set of nonbasic variables; flagged columns get another chance
__global__ void primal_devex_reset_kernel(DeviceModel d)
{
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= d.nm)
    return;
  d.devex[j] = 1.0;
  d.devexRef[j] = d.status[j] != basic;
  d.colFlagged[j] = 0;
}
void launch_primal_devex_reset(const DeviceModel &d, cudaStream_t s)
{
  primal_devex_reset_kernel<<<(d.nm + 255) / 256, 256, 0, s>>>(d);
}

// the true bounds in force (no dual fake bounds), every nonbasic at the bound its status names
__global__ void primal_bounds_kernel(DeviceModel d)
{
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= d.nm)
    return;
  const double lo = d.lowerTrue[j], up = d.upperTrue[j];
  d.lower[j] = lo;
  d.upper[j] = up;
  d.fake[j] = 0;
  unsigned char st = d.status[j];
  if (st == basic)
    return;
  double x = d.sol[j];
  if (lo == up) {
    st = isFixed;
    x = lo;
  } else if (st == atUpperBound && up < kInf) {
    x = up;
  } else if (lo > -kInf) {
    st = atLowerBound;
    x = lo;
  } else if (up < kInf) {
    st = atUpperBound;
    x = up;
  } else {
    st = isFree;
    x = 0.0;
  }
  d.status[j] = st;
  d.sol[j] = x;
}
void launch_primal_bounds(const DeviceModel &d, cudaStream_t s)
{
  primal_bounds_kernel<<<(d.nm + 255) / 256, 256, 0, s>>>(d);
}

} // namespace clpb
