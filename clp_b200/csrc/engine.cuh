// engine.cuh -- device-resident revised dual simplex iteration engine for B200 (sm_100a).
//
// What Clp does on the host with CoinIndexedVector / CoinFactorization per iteration
// (ClpSimplexDual::whileIterating, /root/reference/src/ClpSimplexDual.cpp:973-2384) is done
// here with all working arrays resident in HBM; the host only sequences kernels, decides
// when to refactorize and keeps the status / pivotVariable bookkeeping.
//
// Basis representation (see DESIGN.md "Basis factors"):
//   positions 0..m-1 are rows; a basic slack of row i always sits at position i (column -e_i),
//   structural basics sit at the remaining ("nucleus") positions.  With rows/positions
//   ordered (C = basic-slack rows, N = nucleus rows):
//        B0 = [ -I   S1 ]      L0 U0 of this block form is trivial except for the k x k
//             [  0   Nuc]      nucleus, which is LU-factorized (partial pivoting) on the GPU
//   and held as the explicit inverse Ninv (both row- and column-major) so that FTRAN / BTRAN
//   through it are HBM-streaming GEMVs instead of latency-bound dense triangular chains.
//   Rank-1 basis changes between refactorizations are kept in product form
//        B_t^-1 = E_t ... E_1 B0^-1,   E_i = I - W_i e_{p_i}^T / d_i
//   with the eta columns W (row-major m x tmax panel) and the small lower-triangular
//   coupling matrix G (G mu = v0[P]) held as an explicit inverse Ginv, so that applying all
//   t etas is ONE panel GEMV plus a t x t GEMV (no sequential eta chain).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace clpb {

// status codes = ClpSimplex::Status (ClpSimplex.hpp:119-126)
enum : unsigned char { isFree = 0, basic = 1, atUpperBound = 2, atLowerBound = 3,
                       superBasic = 4, isFixed = 5 };

constexpr double kInf = 1.0e30;
constexpr double kDevexTryNorm = 1.0e-4; // DEVEX_TRY_NORM ClpSimplex.hpp:2056
constexpr int kHistBuckets = 32768;       // ratio-test histogram level 1: 11 exponent + 4 mantissa bits
constexpr int kHist2Buckets = 4096;       // level 2: the next 12 mantissa bits inside the crossing bucket
constexpr int kMaxFlips = 8192;
constexpr int kPriceTile = 1024;          // entries per TMA-staged tile of the CSC arrays
constexpr int kPriceStages = 2;           // tiles in flight per pipeline
constexpr int kPriceGroups = 4;           // independent 256-thread pipelines per CTA
constexpr int kPriceMaxTilesPerCta = 1024; // descriptors staged in shared memory per CTA
constexpr int kPriceTileAlloc = kPriceTile + 8;
constexpr int kPriceTileCols = 8;         // columns per tile (one warp each)

// stop reasons written by the device into IterState.stop
// (primal simplex: STOP_NO_COLUMN = no entering column, STOP_UNBOUNDED = no blocking row and an
// entering variable without a finite range, STOP_PHASE_COSTS = a basic variable changed its
// infeasibility state in phase 1, so the phase-1 costs and the duals must be recomputed)
enum : int { STOP_NONE = 0, STOP_NO_ROW = 1, STOP_NO_COLUMN = 2, STOP_INACCURATE = 3,
             STOP_ETAS_FULL = 4, STOP_TINY_PIVOT = 5, STOP_FLIPS_OVERFLOW = 6, STOP_UNBOUNDED = 7,
             STOP_PHASE_COSTS = 8 };

// Per-iteration scalars, device resident (one instance).  Every kernel of the iteration reads
// what it needs from here, so the launch sequence is independent of the pivot choices and
// can be replayed (CUDA graph) or enqueued several iterations ahead of the host.
struct IterState {
  int stop;
  int iterations;        // completed iterations since (re)start of the batch
  int numEtas;           // t : etas since last refactorization
  int pivotRow;          // r
  int seqIn, seqOut;
  int sigma;             // +1 leaving variable goes to upper bound, -1 to lower
  int numFlips;
  double infeas;         // primal infeasibility of the leaving variable (>0)
  double thetaDual, thetaPrimal;
  double alphaRow;       // pivot element from the BTRAN row   (rho^T a_q)
  double alphaCol;       // pivot element from the FTRAN column (B^-1 a_q)_r
  double rhoNorm2;       // ||rho||^2 = DSE weight of the pivot row
  double thetaStar;      // ratio at which the BFRT slope is exhausted
  double harrisTheta;    // Harris bound beyond thetaStar
  unsigned long long chuzrKey;   // packed (score,row) argmax
  unsigned long long chuzcKey;   // packed (|alpha|,seq) argmax
  unsigned long long harrisBits; // atomicMin target (double bits, positive)
  double objectiveChange;
  int costShifts;        // number of cost shifts since they were last removed
  int bucket1;           // level-1 ratio bucket in which the BFRT slope is exhausted (-1: none)
  unsigned long long residual; // fixed-point slope still to absorb inside bucket1
  // bound-flip right-hand side in fixed point (order independent => bit-identical on every rank)
  unsigned long long flipMaxBits; // max range (u-l) over this iteration's flips (double bits)
  double flipScale, flipInvScale; // contribution * flipScale is accumulated as int64
  // acceptable pivot of the ratio test (ClpSimplexDual::acceptablePivot_): lives here and not in
  // DeviceModel because the driver relaxes it (ClpSimplexDual.cpp:2072-2074) while the captured
  // iteration graph holds DeviceModel by value
  double acceptablePivot;
  int numFlagged;        // rows currently excluded from CHUZR (ClpSimplex::setFlagged, ClpSimplexDual.cpp:2058-2066)
  // primal simplex (primal.cu)
  int primalDir;         // +1 the entering variable increases, -1 it decreases
  int primalFlip;        // 1: this iteration moves the entering variable to its other bound (no basis change)
  int primalPhase;       // 1 sum of infeasibilities, 2 true costs
  int infeasChanged;     // phase 1: a basic variable changed its infeasibility state in this iteration
  double primalDj;       // d_q of the entering variable
  double devexQ;         // reference weight of the entering column, exact from its FTRAN
  unsigned long long pchuzcKey; // packed (score, sequence) argmax of the primal CHUZC
  unsigned long long ratioBits; // relaxed minimum step of the ratio test (double bits, positive)
  unsigned long long ratioKey;  // packed (|alpha|, position) argmax of the second ratio-test pass
};

struct IterRecord { // what the host reads back per iteration
  int stop, pivotRow, seqIn, seqOut, sigma, numFlips;
  double thetaDual, thetaPrimal, alphaRow, alphaCol, infeas;
};

// Things that change at a refactorization.  Lives in device memory and is read by the kernels,
// so that the kernel arguments (and hence a captured CUDA graph of one iteration) stay valid
// across refactorizations.
struct FactorDesc {
  int k;               // nucleus size
  int ldk;             // row pitch of Ninv / NinvT (multiple of 8)
  const double *Ninv;  // [k x ldk] row-major                 (FTRAN  y = Ninv b)
  const double *NinvT; // [k x ldk] row-major of the transpose (BTRAN  y = Ninv^T b)
  const int *s1Col;    // CSR of S1 = A[C rows, nucleus columns]: nucleus index
  const double *s1Val;
  const int *s1cRow;   // the same S1 by nucleus column (CSC): position (= row) of each entry
  const double *s1cVal;
};

// All device pointers of one model.  Plain struct passed by value to kernels.
struct DeviceModel {
  int m, n, nm;
  long long nnz;
  // column copy (CSC) and row copy (CSR) of A
  const int *colStart;
  const int *rowIdx;
  const unsigned short *rowIdx16; // the same row indices in 16 bits when m <= 65535 (PRICE streams these), else nullptr
  const double *val;
  const int *rowStart;
  const int *colIdx;
  const double *rval;
  const int *priceTileCol; // [numPriceTiles] int4 descriptors {firstCol, nCols, firstEntry, nEntries}
  int numPriceTiles;
  // rim, length n+m (columns then rows, Clp order)
  double *cost, *costTrue, *lower, *upper, *lowerTrue, *upperTrue, *sol, *dj;
  unsigned char *status, *fake;
  int *pivotVariable; // [m] sequence basic at each position
  double *weights;    // [m] dual steepest edge weights (by position)
  // basis factors
  int k;              // nucleus size
  int ldk;            // leading dimension of Ninv / NinvT
  int *posToNuc;      // [m] nucleus index of a position or -1
  int *nucRow;        // [k] position (=row) of nucleus index
  int *nucCol;        // [k] structural sequence of nucleus index
  double *Ninv;       // [k x ldk] row-major : row i contiguous  (FTRAN  y = Ninv b)
  double *NinvT;      // [k x ldk] row-major of the transpose     (BTRAN  y = Ninv^T b)
  FactorDesc *fd;        // device copy of {k, ldk, Ninv, NinvT, s1Col, s1Val} (read by kernels)
  const int *s1RowStart; // CSR of S1 = A[C rows, nucleus columns], rows indexed by position
  const int *s1Col;      // nucleus index
  const double *s1Val;
  const int *s1cStart;   // [k+1] S1 by nucleus column; entries in FactorDesc::s1cRow / s1cVal
  // product-form etas
  int tmax;           // capacity (row pitch of W, pitch of Ginv)
  double *W;          // [m x tmax] row-major, column i = W_i
  int *etaPos;        // [tmax] p_i
  int *etaPrevSame;   // [tmax] previous eta with the same position or -1
  int *etaLastOfPos;  // [m]    last eta index for a position or -1
  double *Ginv;       // [tmax x tmax] row-major lower triangular
  double *GinvT;      // [tmax x tmax] its transpose (row j = column j of Ginv, entries i >= j)
  double *xp;         // [3 x tmax] FTRAN right-hand sides gathered at the eta positions
  // work vectors
  double *rho;        // [m]
  double *alphaRow;   // [n+m] tableau row (dense)
  double *rhs3;       // [3 x m] FTRAN right-hand sides / results: a_q, rho->tau, flip rhs
  double *ywork;      // [3 x k] + scratch
  double *uwork;      // [m] BTRAN input after eta transposes
  double *swork;      // [k]
  long long *flipAcc; // [m] fixed-point accumulator of the bound-flip right-hand side (zero when idle)
  double amax;        // max(1, max |a_ij|): bound for the fixed-point scale of flipAcc
  unsigned int *tailCounter; // [16] last-block-done tickets (one per kernel that has a tail)
  unsigned int *gridBar;     // [2] arrival count / generation of the row-pass grid barrier
  double *aqBuf;      // [m] entering column scattered by the row pass (zero when idle)
  double *candA, *candD; // [n+m] short list of ratio-test candidates near the crossing bucket
  int *candJ, *candCount;
  double *mu;         // [3 x tmax]
  double *nu;         // [tmax]
  // ratio test
  unsigned long long *histWeight; // [kHistBuckets] fixed-point slope per ratio bucket
  unsigned long long *histMin;    // [kHistBuckets] min ratio bits per bucket
  unsigned long long *hist2Weight, *hist2Min; // [kHist2Buckets] second level
  unsigned long long *segTotal;   // [kHistBuckets/1024] per-segment totals of the level-1 scan
  int *segLast;                   // last non-empty bucket per segment
  unsigned int *scanCounter;      // last-block-done ticket
  int *flipList;      // [n+m] flipped sequences of this iteration, ascending
  unsigned int *flipBits; // [(n+m+31)/32] bit mask of the same (cleared by CHUZR)
  IterState *st;
  IterRecord *rec;    // ring of records (device)
  int recCap;
  // tolerances
  double primalTolerance, dualTolerance, zeroTolerance;
  // row-sharded factors (multi-GPU, see DESIGN.md "Multi-GPU"): rank shardRank of shardW streams
  // rows [rank*per_k, (rank+1)*per_k) of Ninv / NinvT (per_k = roundUp8(ceil(k/W)), k from
  // FactorDesc) and positions [rank*shardPerM, ...) of the eta panel W; results go to gather buffers
  // with a fixed per-rank chunk (shardPerK / shardPerM entries per vector) that ONE in-place
  // all-gather per solve completes.  shardW == 1: plain single-GPU layout.
  int shardW, shardRank, shardPerK, shardPerM;
  int dantzig;    // 1: ClpDualRowDantzig (largest infeasibility, weights ignored and left alone); 0: dual steepest edge
  int shardPanel; // 1: the eta panel is row-sharded too (pays only when 8*m*t bytes outweigh one more all-gather)
  double *gatherY; // [W][3][shardPerK]  FTRAN GEMV results
  double *gatherB; // [W][shardPerK]     BTRAN GEMV results
  double *gatherP; // [W][3][shardPerM]  eta-panel results
  unsigned char *flagged; // [m] by position: 1 = row is flagged (skipped by CHUZR until the next refactorization)
  // primal simplex (primal.cu)
  double *devex;             // [n+m] Devex weights by sequence (ClpPrimalColumnSteepest::weights_)
  unsigned char *devexRef;   // [n+m] 1 = in the Devex reference framework (nonbasic at the last reset)
  unsigned char *colFlagged; // [n+m] 1 = excluded from the primal CHUZC until the next refactorization
  double *ratioPart;         // [m/256+1] per-CTA partial sums of the entering column's reference weight
  int primalDantzig;         // primalColumnPivot: 0 Devex, 1 Dantzig
};

// Optional per-kernel CUDA-event brackets (timing mode only): price kernel, FTRAN GEMV, BTRAN GEMV.
struct KernelTimers {
  cudaEvent_t price[2], ftranGemv[2], btranGemv[2];
};
extern KernelTimers *g_kernelTimers; // nullptr outside timing mode (engine.cu)
extern int g_pfiApplyVariant;         // solve.cu
extern int g_priceIdx16;              // price.cu
extern int g_rowPassCtas;             // rowpass.cu
extern int g_gemvVariantF, g_gemvVariantB, g_gemvGridMul; // solve.cu (launch-shape experiments)
// collectives of a sharded run (host side; set by Engine before it enqueues work)
struct ShardCtx {
  int W = 1, rank = 0;
  void *comm = nullptr;
  int (*allGather)(void *comm, void *buf, size_t bytesPerRank, void *stream) = nullptr; // in place
};
extern ShardCtx g_shardCtx;           // solve.cu

// ---- launch wrappers (implemented in the .cu files) ---------------------------------------
// solve.cu
void launch_ftran(const DeviceModel &d, int nrhs, bool applyEtas, cudaStream_t s);
void launch_btran_unit(const DeviceModel &d, bool checkState, cudaStream_t s); // rho = B^-T e_r (r = st->pivotRow)
void launch_ftran_iteration(const DeviceModel &d, bool pregathered, cudaStream_t s); // 3 rhs + etas + pivot scalars (tail)
// rowpass.cu
bool launch_row_pass(const DeviceModel &d, cudaStream_t s);
void launch_eta_rowvec(const DeviceModel &d, int mode, bool checkState, cudaStream_t s);
void launch_ftran_buffer(const DeviceModel &d, double *buf, int nrhs, bool applyEtas, cudaStream_t s);
void launch_btran_dense(const DeviceModel &d, double *vec, bool applyEtas, cudaStream_t s); // vec(m) in/out
// price.cu
void launch_price(const DeviceModel &d, int colBegin, int colEnd, bool fuseHistogram, cudaStream_t s);
void launch_price_slacks(const DeviceModel &d, int colBegin, int colEnd, bool fuseHistogram, cudaStream_t s);
void launch_histogram(const DeviceModel &d, cudaStream_t s);
void launch_transpose_times(const DeviceModel &d, const double *pi, double *z, double scalar,
                            cudaStream_t s);
void launch_times_rows(const DeviceModel &d, const double *x, double *y, double scalar,
                       cudaStream_t s);
void launch_chuzc(const DeviceModel &d, cudaStream_t s);
// update.cu
void launch_chuzr(const DeviceModel &d, cudaStream_t s); // stand-alone CHUZR (start of a batch)
void launch_dual_update_and_flips(const DeviceModel &d, unsigned int *flipBits, cudaStream_t s);
void launch_pivot_updates(const DeviceModel &d, cudaStream_t s);
void launch_make_dual_feasible(const DeviceModel &d, double dualBound, int *counters, cudaStream_t s);
void launch_compute_primals(const DeviceModel &d, double *xn, double *rhs, cudaStream_t s, bool withEtas = false);
void launch_compute_duals(const DeviceModel &d, double *pi, double *z, cudaStream_t s, bool withEtas = false);
void launch_objective(const DeviceModel &d, double *out, cudaStream_t s);
void launch_primal_drift(const DeviceModel &d, const double *xold, unsigned long long *out, cudaStream_t s);
void launch_permute_weights(const double *wOld, double *wNew, const int *srcPos, int m,
                            cudaStream_t s);
void launch_gather_nucleus_matrix(const DeviceModel &d, double *N, int ld, cudaStream_t s);
void launch_count_fake(const DeviceModel &d, int *counter, cudaStream_t s);
void launch_unpack_column(const DeviceModel &d, int seq, double *out, cudaStream_t s);
void launch_eta_append_test(const DeviceModel &d, int pivotRow, int seqIn, cudaStream_t s);
// primal.cu
void launch_primal_chuzc(const DeviceModel &d, cudaStream_t s);  // stand-alone CHUZC (start of a batch)
void launch_primal_ratio(const DeviceModel &d, cudaStream_t s);  // Harris two-pass ratio test over x_B
void launch_primal_iteration(const DeviceModel &d, cudaStream_t s); // one whole primal iteration
void launch_primal_costs(const DeviceModel &d, int phase, cudaStream_t s); // phase-1 or true costs into d.cost
void launch_primal_devex_reset(const DeviceModel &d, cudaStream_t s);
void launch_primal_bounds(const DeviceModel &d, cudaStream_t s); // true bounds in force, nonbasics at them
// factor.cu
int dense_invert(double *A, double *X, int k, int ld, int *dIpiv, int *dPerm, int *dInfo,
                 int *hostIpiv, int *hostPerm, double singularTol, cudaStream_t s, int shardW = 1,
                 int shardRank = 0, int (*allGather)(void *, void *, size_t, void *) = nullptr,
                 void *comm = nullptr, void (*hostOverlap)(void *) = nullptr, void *overlapCtx = nullptr);
void launch_transpose(const double *src, double *dst, int k, int ld, cudaStream_t s);

} // namespace clpb
