// engine.hpp -- host side of the B200 dual simplex engine (C++ interface behind the C ABI).
//
// The host keeps what ClpSimplexDual keeps on the host in the reference: the iteration
// driver (whileIterating / statusOfProblemInDual, src/ClpSimplexDual.cpp:973,4996), the
// refactorization policy (ClpSimplex.cpp:11401 defaultFactorizationFrequency), fake-bound /
// cost-shift clean-up decisions and the problem status.  Everything O(m), O(n) or O(nnz) per
// iteration runs in the CUDA kernels of solve.cu / price.cu / update.cu / factor.cu.
#pragma once
#include "engine.cuh"

#include <algorithm>
#include <string>
#include <vector>

namespace clpb {

struct PhaseTimes { // accumulated device milliseconds per phase (when timing is on)
  double chuzr = 0, btran = 0, price = 0, chuzc = 0, dualUpdate = 0, ftran = 0, update = 0,
         refactor = 0;
  double priceKernel = 0, ftranGemv = 0, btranGemv = 0; // single kernels inside the phases
  double ftranGemvBytes = 0, btranGemvBytes = 0;        // algorithmic bytes of those launches (the nucleus size changes at a refactorization)
  long samples = 0;
};

struct Presolve;

class Engine {
public:
  Engine();
  ~Engine();

  // ---- problem (ClpModel::loadProblem / readMps) ----
  int loadProblem(int numberColumns, int numberRows, const int *columnStart, const int *row,
                  const double *element, const double *columnLower, const double *columnUpper,
                  const double *objective, const double *rowLower, const double *rowUpper);
  int readMps(const char *fileName);

  // ---- parameters ----
  double primalTolerance = 1.0e-7, dualTolerance = 1.0e-7, dualBound = 1.0e10;
  double acceptablePivot = 1.0e-7, zeroTolerance = 1.0e-13;
  int maximumIterations = 2147483647;
  double maximumSeconds = 1.0e30;
  int factorizationFrequency = 0; // 0 = default formula
  int logLevel = 0;
  // ClpSimplex::setDualRowPivotAlgorithm (src/ClpSimplex.cpp:4985): 0 ClpDualRowSteepest (default),
  // 1 ClpDualRowDantzig (src/ClpDualRowDantzig.cpp:56 pivotRow: largest primal infeasibility)
  int dualRowPivot = 0;
  int batch = 16;                 // iterations enqueued per host synchronisation
  int refreshDualsEvery = 0, refreshPrimalsEvery = 0; // experiments: recompute from scratch inside a cycle
  bool timing = false;
  bool useGraph = true;
  // 16-bit row indices for PRICE (m <= 65535): 10 instead of 12 bytes per entry.  Measured at C2: no
  // gain (29.2 vs 29.3 us) -- the kernel is bound by the shared-memory gathers of rho, not by HBM -- so off
  bool priceIdx16 = false;
  bool usePriceTma = false;       // TMA-staged price kernel (default: LDG-direct kernel, 26% faster)
  // 0 = choose per basis (block-banded nucleus when it pays), 1 = always the dense nucleus inverse,
  // 2 = always block-banded (tests)
  int factorMode = 0;
  bool useRowPass = true;         // cooperative row-pass kernel (false / column-sharded: separate kernels)
  int warmupIterations = 0;       // device-timed window starts once this many iterations ran
  double timedMilliseconds = 0.0; // CUDA-event time of the window (iterations + refactorizations)
  int timedIterations = 0;
  double objectiveOffset = 0.0;
  // ClpModel::scaling(mode) (src/ClpModel.hpp): 0 off, 1 equilibrium, 2 geometric, 3 auto, 4 auto
  // (dynamic).  Clp's own default is 3; the benchmark configuration states "scaling off".
  int scalingFlag = 0;
  std::vector<double> rowScale, columnScale; // empty: the problem is solved unscaled
  int computeScaling();                      // ClpPackedMatrix::scale (src/ClpPackedMatrix.cpp:4120)
  // ClpSimplex::setPerturbation (src/ClpSimplex.hpp): 50 perturb the costs before the first
  // iteration, 100 only if few distinct cost values (Clp's default), 102 never (default here: the
  // benchmark configuration states "perturbation off").  ClpSimplexDual::perturb, :6533.
  int perturbation = 102;
  int perturbCosts(std::vector<double> &cost) const; // 0 = perturbed (cost[n] modified in place)
  int previewPerturbation(double *costOut);          // host only (no device): scaled working costs after perturb
  double largestPerturbation = 0.0;
  // column sharding of the pricing pass (multi-GPU): this rank prices [colBegin,colEnd)
  int rank = 0, worldSize = 1;
  void *ncclComm = nullptr; // ncclComm_t when worldSize > 1
  int (*allGatherFn)(void *comm, void *buf, size_t bytesPerRank, void *stream) = nullptr;
  // sharding is used only when a rank's share of the matrix is large enough to amortise the
  // collectives' latency (north_star: "only when n is large enough"); otherwise every rank runs the
  // whole iteration on its own ("replicas only")
  long long shardMinNnzPerRank = 4000000;
  int shardPanelMode = -1; // -1 decide from the panel size, 0 replicate the eta panel, 1 shard it
  int tmaxHint() const { return factorizationFrequency > 0 ? factorizationFrequency : std::min(2048, 2 * defaultFactorizationFrequency()); }
  bool shardActive() const;

  // ---- solve (ClpSimplex::dual) ----
  int dual();
  // Hot start for branch-and-bound style callers (ClpSimplexDual::fastDual, src/ClpSimplexDual.cpp:7241;
  // strongBranching :6965): with hotStart set, a dual() that follows a solve of the SAME model whose
  // bounds were changed through chgColumnLower/Upper / chgRowLower/Upper (Clp_chgColumnLower ...,
  // src/Clp_C_Interface.h:150-156) keeps the device-resident factors, eta file, weights, duals and
  // status: it only re-imposes the bounds, moves nonbasic variables to them, recomputes x_B through
  // the existing factors and iterates -- no upload, no refactorization at the start.
  bool hotStart = false;
  void chgBounds(const double *columnLower, const double *columnUpper, const double *rowLower,
                 const double *rowUpper); // NULL = unchanged
  bool lastSolveWasHot = false;
  // ---- solve (ClpSimplex::primal, src/ClpSimplex.cpp:6145; primal.cu) ----
  // Phase 1 minimises the sum of infeasibilities, phase 2 the true costs; "perturbation" is ignored.
  // With hotStart set, a primal() that follows a solve of the same model keeps the device-resident
  // factors, eta file, x_B and status, recomputes the duals for the (changed) costs and iterates.
  int primal();
  int primalColumnPivot = 0; // ClpSimplex::setPrimalColumnPivotAlgorithm: 0 exact Devex, 1 Dantzig
  // Clp_chgObjCoefficients (src/Clp_C_Interface.h:158): replaces the loaded objective (n entries)
  void chgObjCoefficients(const double *obj);
  // plug-in entries on explicit host vectors (ClpPrimalColumnPivot::pivotColumn, ClpSimplexPrimal::primalRow)
  int primalColumnPivotTest(const double *dj, const unsigned char *stat, const double *weights, int mode);
  int primalRowTest(const double *alpha, const double *xB, const double *lowerB, const double *upperB,
                    int direction, double enteringRange, int phase, double *theta);
  int cycleFor(int k) const; // refactorization interval the default policy uses at nucleus size k (host only)
  int problemStatus = -1;
  int numberIterations = 0, numberRefactorizations = 0;
  double objectiveValue = 0.0, sumPrimalInfeasibilities = 0.0;
  double secondsInLoop = 0.0;
  long kernelLaunches = 0;
  PhaseTimes phase;
  int lastNucleusSize = 0;

  // ---- results (host copies, valid after dual()) ----
  std::vector<double> solution;     // n+m
  std::vector<double> reducedCost;  // n+m
  std::vector<double> rowPrice;     // m
  std::vector<unsigned char> status; // n+m
  std::vector<int> pivotVariable;   // m
  void setStatus(const unsigned char *st);
  // ClpSimplex::writeBasis / readBasis (src/ClpSimplex.cpp:6569,6577 -> ClpSimplexOther.cpp:1018,1136):
  // MPS basis file in the reference's no-names form (C%7.7d / R%7.7d), host only
  int writeBasis(const char *fileName) const;
  int readBasis(const char *fileName);
  const std::vector<unsigned char> &currentStatus() const { return hStatus; }

  // ---- plug-in level entry points (parity tests; host buffers) ----
  int factorize(const int *basicSequence, int *pivotVariableOut);
  int updateColumn(double *vec);            // FTRAN in place, m doubles
  int updateColumnTranspose(double *vec);   // BTRAN in place
  int replaceColumn(int sequenceIn, int pivotRow);
  void transposeTimes(double scalar, const double *pi, double *z);
  void times(double scalar, const double *x, double *y);
  int dualColumnTest(const double *alphaRow, const double *dj, const unsigned char *stat,
                     int sigma, double infeas, double *theta, bool rowPass = false);
  int iterate(int count);                   // run 'count' iterations from the current state
  // ---- the iteration one plug-in call at a time (ClpDualRowPivot / ClpFactorization / ClpMatrixBase
  // methods in the order ClpSimplexDual::whileIterating calls them); device state carries over
  int pivotRowStep(int *sequenceOut, int *direction, double *infeasibility); // ClpDualRowPivot::pivotRow; -1 = none
  int btranPriceStep(double *rho, double *alphaRow);  // updateColumnTranspose(e_r) + transposeTimes; nnz(rho)
  int dualColumnStep(double *theta, double *alpha);   // dualColumn + updateDualsInDual + flips; sequenceIn or -1
  double updateWeightsStep(int *returnCode);          // ClpDualRowPivot::updateWeights (updateTwoColumnsFT); alpha
  int updatePrimalStep(double *changeInObjective);    // updatePrimalSolution + DSE recurrence + replaceColumn + housekeeping
  void saveWeights(int mode);                         // ClpDualRowSteepest::saveWeights modes 1..7
  int unrollWeights();                                // nothing to undo before updatePrimalStep (returns 0)
  int updateColumnFT(double *vec);                    // FTRAN that also keeps the spike for replaceColumn
  int replaceColumnChecked(int sequenceIn, int pivotRow, double pivotCheck, double acceptablePivot);
  std::vector<int> savedWeightSeq;
  std::vector<double> savedWeightVal;
  void getWeights(double *w);
  void getDeviceVector(const char *name, double *out);
  int startup();                            // status -> basis, factorize, compute primals/duals

  int numberRows() const { return m; }
  int numberColumns() const { return n; }
  long long numberElements() const { return (long long)hColStart.empty() ? 0 : hColStart[n]; }
  const std::vector<double> &colLower() const { return hLower; }

  // host copy of the problem
  int m = 0, n = 0, nm = 0;
  std::vector<int> hColStart, hRow;
  std::vector<double> hVal;
  std::vector<double> hLower, hUpper, hCost; // n+m, true bounds/costs (as loaded)
  // what the device works on: the loaded problem, scaled when scalingFlag asks for it
  std::vector<double> wVal, wLower, wUpper, wCost;
  std::string problemName;

private:
  DeviceModel d{};
  cudaStream_t stream = nullptr;
  bool deviceReady = false;
  bool factorsValid = false; // a factorization of the current device basis exists
  void boundsToWorking();    // hLower/hUpper -> wLower/wUpper with the scale factors in force
  int hotPrepare();
  bool costsPending = false; // chgObjCoefficients after the device copy was made: costTrue is stale
  void uploadPendingCosts();
  int primalPhase = 1;
  int primalRefresh();             // refactor + primalRecompute
  int primalRecompute(bool resetDevex); // computePrimals, phase + costs, computeDuals (current factors)
  void primalCosts(bool resetDevex);    // phase from the sum of infeasibilities, its costs, computeDuals
  cudaGraphExec_t primalGraph = nullptr; // one captured primal iteration
  int primalKernelsPerIteration = 0;
  void buildPrimalGraph();
  long long readySignature = -1;
  int trivialSolve(); // m == 0 or n == 0 (a presolved model can be empty): host only
  bool haveUserStatus = false;
  // device allocations (owned)
  std::vector<void *> allocs;
  double *dXn = nullptr, *dRhs = nullptr, *dPi = nullptr, *dZ = nullptr, *dObj = nullptr;
  double *dWeightsTmp = nullptr;
  double *dSolOld = nullptr;             // recurrence-updated solution kept across a refresh (drift measure)
  unsigned long long *dDrift = nullptr;
  double lastPrimalDrift = 0.0;          // relative, of the last refresh
  bool driftMeasured = false;
  int currentCycle = 0;                  // refactorization interval in force (adapted from the drift)
  int *dSrcPos = nullptr, *dCounters = nullptr;
  unsigned char *dFlipFlag = nullptr;
  int *dIpiv = nullptr, *dPerm = nullptr, *dInfo = nullptr;
  int *dS1RowStart = nullptr, *dS1Col = nullptr;
  double *dS1Val = nullptr;
  int *dS1cStart = nullptr, *dS1cRow = nullptr;
  double *dS1cVal = nullptr;
  size_t s1Cap = 0;
  size_t nucCap = 0; // capacity (elements) of Ninv / NinvT
  IterState *hState = nullptr; // pinned
  IterRecord *hRec = nullptr;
  std::vector<cudaEvent_t> events;
  std::vector<KernelTimers> kernelTimers; // one per batch slot (timing mode)
  std::vector<unsigned char> hStatus;
  std::vector<int> hPivot;
  int tmax = 0;
  double currentDualBound = 0.0;
  double currentAcceptablePivot = 1.0e-7;
  void setAcceptablePivot(double value); // device-resident (IterState): no graph re-capture
  cudaGraphExec_t iterGraph = nullptr; // one captured iteration (replayed 'batch' times per sync)
  int kernelsPerIteration = 0;
  void buildIterationGraph();

  template <class T> T *dalloc(size_t count);
  void freeAll();
  int setupDevice();
  int refactor();          // factorize current basis (repairs singular bases)
  int refresh();           // refactor + computeDuals + makeDualFeasible + computePrimals
  void enqueueIteration(bool timed, int slot);
  void enqueueBatchStart();
  void fetchState();
  void downloadSolution();
  int defaultFactorizationFrequency() const;
  void resetStateForRun();
  void buildRowCopy(const std::vector<double> &val, std::vector<int> &rowStart,
                    std::vector<int> &colIdx, std::vector<double> &rval) const;
  void prepareWorkingProblem();
};

// presolve.cpp -- elementary presolve actions and their postsolve (host only)
struct Presolve {
  struct Action {
    char kind;      // 'F' fixed column, 'S' singleton row, 'C' empty column, 'R' empty row, 'D' dominated column, 'g'/'G' column fixed by a forcing row / the row itself
    int col, row;
    double value;   // F/C: the value of the column; S: the coefficient a_ij
    double oldLo, oldUp;         // S: column bounds before the row was folded in
    double impliedLo, impliedUp; // S: bounds the row implies
  };
  int m = 0, n = 0;
  std::vector<Action> actions;
  std::vector<char> colAlive, rowAlive;
  std::vector<int> colMap, rowMap; // original -> reduced index or -1
  std::vector<double> lower, upper, cost; // working bounds (n+m) and costs (n)
  std::vector<int> colStart, rowIdx;
  std::vector<double> val;
  double offset = 0.0;
  // 0 ok (dst loaded with the reduced problem), 1 primal infeasible, 2 dual infeasible (unbounded)
  int presolve(const Engine &src, Engine &dst);
  void postsolve(const std::vector<double> &xr, const std::vector<double> &pir,
                 const std::vector<unsigned char> &statusR, const Engine &orig,
                 std::vector<double> &solution, std::vector<double> &reducedCost,
                 std::vector<double> &rowPrice, std::vector<unsigned char> &status) const;
};

// mps_reader.cpp
int readMpsFile(const char *fileName, int &m, int &n, std::vector<int> &colStart,
                std::vector<int> &row, std::vector<double> &val, std::vector<double> &colLower,
                std::vector<double> &colUpper, std::vector<double> &obj,
                std::vector<double> &rowLower, std::vector<double> &rowUpper, double &objOffset,
                std::string &name);

int writeMpsFile(const char *fileName, int m, int n, const std::vector<int> &colStart,
                 const std::vector<int> &row, const std::vector<double> &val,
                 const std::vector<double> &lower, const std::vector<double> &upper,
                 const std::vector<double> &cost, double objOffset, const std::string &name);

} // namespace clpb
