// capi.cu -- extern "C" surface declared in include/clp_b200.h
#include "../../include/clp_b200.h"
#include "engine.hpp"

#include <cstring>
#include <dlfcn.h>
#include <stdexcept>

struct Clpb_Simplex {
  clpb::Engine e;
  clpb::Presolve pre; // filled by Clpb_presolvedModel on the ORIGINAL model
};

namespace {

// ---- NCCL through dlopen so that single-GPU use has no NCCL dependency -----------------
typedef int (*ncclGetUniqueId_t)(void *);
struct NcclId {
  char internal[128];
};
typedef int (*ncclCommInitRankV_t)(void **, int, NcclId, int);
typedef int (*ncclAllGather_t)(const void *, void *, size_t, int, void *, cudaStream_t);

void *g_nccl = nullptr;
ncclGetUniqueId_t p_getId = nullptr;
ncclCommInitRankV_t p_init = nullptr;
ncclAllGather_t p_allGather = nullptr;

bool loadNccl()
{
  if (g_nccl)
    return true;
  const char *names[] = {"libnccl.so.2", "libnccl.so", nullptr};
  for (int i = 0; names[i] && !g_nccl; i++)
    g_nccl = dlopen(names[i], RTLD_NOW | RTLD_GLOBAL);
  if (!g_nccl)
    return false;
  p_getId = (ncclGetUniqueId_t)dlsym(g_nccl, "ncclGetUniqueId");
  p_init = (ncclCommInitRankV_t)dlsym(g_nccl, "ncclCommInitRank");
  p_allGather = (ncclAllGather_t)dlsym(g_nccl, "ncclAllGather");
  return p_getId && p_init && p_allGather;
}

struct CommWrap {
  void *comm;
  int rank;
};

int allGatherBytes(void *comm, void *buf, size_t bytesPerRank, void *stream)
{
  // in place: rank r's chunk already sits at buf + r*bytesPerRank; ncclChar == 0
  // sendbuff is resolved by NCCL's in-place convention from the rank stored with the comm
  CommWrap *w = static_cast<CommWrap *>(comm);
  const char *send = static_cast<const char *>(buf) + (size_t)w->rank * bytesPerRank;
  return p_allGather(send, buf, bytesPerRank, 0, w->comm, static_cast<cudaStream_t>(stream));
}

template <class F> int guarded(F f)
{
  try {
    return f();
  } catch (const std::exception &ex) {
    if (std::string(ex.what()) == "no CUDA device")
      return CLPB_NO_DEVICE;
    return -99;
  }
}

} // namespace

extern "C" {

Clpb_Simplex *Clpb_newModel(void) { return new Clpb_Simplex(); }
void Clpb_deleteModel(Clpb_Simplex *model) { delete model; }

int Clpb_loadProblem(Clpb_Simplex *model, int numcols, int numrows, const int *start,
                     const int *index, const double *value, const double *collb,
                     const double *colub, const double *obj, const double *rowlb,
                     const double *rowub)
{
  return guarded([&] {
    return model->e.loadProblem(numcols, numrows, start, index, value, collb, colub, obj, rowlb,
                                rowub);
  });
}
int Clpb_readMps(Clpb_Simplex *model, const char *filename, int, int)
{
  return guarded([&] { return model->e.readMps(filename); });
}
Clpb_Simplex *Clpb_presolvedModel(Clpb_Simplex *model, int *status)
{
  Clpb_Simplex *red = new Clpb_Simplex();
  const int rc = model->pre.presolve(model->e, red->e);
  if (status)
    *status = rc;
  if (rc != 0) {
    // presolve itself proved the problem infeasible / unbounded: the ORIGINAL model says so
    model->e.problemStatus = rc;
    model->e.numberIterations = 0;
    delete red;
    return nullptr;
  }
  // parameters travel with the model
  red->e.primalTolerance = model->e.primalTolerance;
  red->e.dualTolerance = model->e.dualTolerance;
  red->e.dualBound = model->e.dualBound;
  red->e.maximumIterations = model->e.maximumIterations;
  red->e.maximumSeconds = model->e.maximumSeconds;
  red->e.scalingFlag = model->e.scalingFlag;
  red->e.perturbation = model->e.perturbation;
  red->e.logLevel = model->e.logLevel;
  red->e.acceptablePivot = model->e.acceptablePivot;
  red->e.zeroTolerance = model->e.zeroTolerance;
  red->e.factorizationFrequency = model->e.factorizationFrequency;
  red->e.batch = model->e.batch;
  red->e.useGraph = model->e.useGraph;
  red->e.useRowPass = model->e.useRowPass;
  red->e.usePriceTma = model->e.usePriceTma;
  red->e.factorMode = model->e.factorMode;
  red->e.dualRowPivot = model->e.dualRowPivot;
  red->e.primalColumnPivot = model->e.primalColumnPivot;
  red->e.rank = model->e.rank;
  red->e.worldSize = model->e.worldSize;
  red->e.ncclComm = model->e.ncclComm;
  red->e.allGatherFn = model->e.allGatherFn;
  return red;
}
int Clpb_postsolve(Clpb_Simplex *model, Clpb_Simplex *reduced)
{
  clpb::Engine &o = model->e, &r = reduced->e;
  if (r.problemStatus != 0) {
    // not optimal: nothing to postsolve, but the original model reports the outcome
    o.problemStatus = r.problemStatus;
    o.numberIterations = r.numberIterations;
    return 0;
  }
  if ((int)r.solution.size() != r.nm || (int)r.rowPrice.size() != r.m || (int)r.status.size() != r.nm)
    return -1; // the reduced model holds no solution
  std::vector<double> xr(r.solution.begin(), r.solution.begin() + r.n);
  model->pre.postsolve(xr, r.rowPrice, r.status, o, o.solution, o.reducedCost, o.rowPrice, o.status);
  o.setStatus(o.status.data());
  double obj = o.objectiveOffset;
  for (int j = 0; j < o.n; j++)
    obj += o.hCost[j] * o.solution[j];
  o.objectiveValue = obj;
  o.problemStatus = r.problemStatus;
  o.numberIterations = r.numberIterations;
  return 0;
}
void Clpb_setSolution(Clpb_Simplex *model, const double *x, const double *rowPrice, const unsigned char *status,
                      int problemStatus)
{
  // hand a solution in from outside (the parity tests solve the presolved model with an independent CPU solver)
  clpb::Engine &e = model->e;
  e.solution.assign(e.nm, 0.0);
  std::copy(x, x + e.n, e.solution.begin());
  e.rowPrice.assign(rowPrice, rowPrice + e.m);
  e.status.assign(status, status + e.nm);
  e.reducedCost.assign(e.nm, 0.0);
  e.problemStatus = problemStatus;
}
int Clpb_writeMps(Clpb_Simplex *model, const char *filename, int, int, double)
{
  clpb::Engine &e = model->e;
  return clpb::writeMpsFile(filename, e.m, e.n, e.hColStart, e.hRow, e.hVal, e.hLower, e.hUpper, e.hCost,
                            e.objectiveOffset, e.problemName);
}
int Clpb_numberRows(Clpb_Simplex *model) { return model->e.numberRows(); }
int Clpb_numberColumns(Clpb_Simplex *model) { return model->e.numberColumns(); }
long long Clpb_getNumElements(Clpb_Simplex *model)
{
  return model->e.hColStart.empty() ? 0 : model->e.hColStart[model->e.n];
}
void Clpb_getProblem(Clpb_Simplex *model, int *start, int *index, double *value, double *collb,
                     double *colub, double *obj, double *rowlb, double *rowub)
{
  clpb::Engine &e = model->e;
  const int n = e.n, m = e.m;
  if (start)
    std::copy(e.hColStart.begin(), e.hColStart.end(), start);
  if (index)
    std::copy(e.hRow.begin(), e.hRow.end(), index);
  if (value)
    std::copy(e.hVal.begin(), e.hVal.end(), value);
  if (collb)
    std::copy(e.hLower.begin(), e.hLower.begin() + n, collb);
  if (colub)
    std::copy(e.hUpper.begin(), e.hUpper.begin() + n, colub);
  if (obj)
    std::copy(e.hCost.begin(), e.hCost.begin() + n, obj);
  if (rowlb)
    std::copy(e.hLower.begin() + n, e.hLower.begin() + n + m, rowlb);
  if (rowub)
    std::copy(e.hUpper.begin() + n, e.hUpper.begin() + n + m, rowub);
}
int Clpb_setParameter(Clpb_Simplex *model, const char *key, double value)
{
  std::string k(key);
  clpb::Engine &e = model->e;
  if (k == "primalTolerance")
    e.primalTolerance = value;
  else if (k == "dualTolerance")
    e.dualTolerance = value;
  else if (k == "dualBound")
    e.dualBound = value;
  else if (k == "maximumIterations")
    e.maximumIterations = (int)value;
  else if (k == "maximumSeconds")
    e.maximumSeconds = value;
  else if (k == "logLevel")
    e.logLevel = (int)value;
  else if (k == "factorizationFrequency")
    e.factorizationFrequency = (int)value;
  else if (k == "batch")
    e.batch = std::max(1, (int)value);
  else if (k == "timing")
    e.timing = value != 0.0;
  else if (k == "warmupIterations")
    e.warmupIterations = (int)value;
  else if (k == "usePriceTma")
    e.usePriceTma = value != 0.0;
  else if (k == "useGraph")
    e.useGraph = value != 0.0;
  else if (k == "useRowPass")
    e.useRowPass = value != 0.0;
  else if (k == "pfiApplyVariant")
    clpb::g_pfiApplyVariant = (int)value;
  else if (k == "rowPassCtas")
    clpb::g_rowPassCtas = (int)value;
  else if (k == "priceIdx16")
    e.priceIdx16 = value != 0.0;
  else if (k == "gemvVariantF")
    clpb::g_gemvVariantF = (int)value;
  else if (k == "gemvVariantB")
    clpb::g_gemvVariantB = (int)value;
  else if (k == "gemvGridMul")
    clpb::g_gemvGridMul = std::max(1, (int)value);
  else if (k == "objectiveOffset")
    e.objectiveOffset = value;
  else if (k == "scaling")
    e.scalingFlag = (int)value;
  else if (k == "perturbation")
    e.perturbation = (int)value;
  else if (k == "refreshDualsEvery")
    e.refreshDualsEvery = (int)value;
  else if (k == "refreshPrimalsEvery")
    e.refreshPrimalsEvery = (int)value;
  else if (k == "hotStart")
    e.hotStart = value != 0.0;
  else if (k == "dualRowPivot")
    e.dualRowPivot = (int)value;
  else if (k == "primalColumnPivot")
    e.primalColumnPivot = (int)value;
  else if (k == "shardPanel")
    e.shardPanelMode = (int)value;
  else if (k == "shardMinNnzPerRank")
    e.shardMinNnzPerRank = (long long)value;
  else if (k == "factorMode")
    e.factorMode = (int)value;
  else if (k == "acceptablePivot")
    e.acceptablePivot = value;
  else
    return -1;
  return 0;
}
void Clpb_scaling(Clpb_Simplex *model, int mode) { model->e.scalingFlag = mode; }
int Clpb_scaleFactors(Clpb_Simplex *model, double *rowScale, double *columnScale)
{
  clpb::Engine &e = model->e;
  const int rc = e.computeScaling(); // host only
  for (int i = 0; i < e.m; i++)
    rowScale[i] = rc == 0 ? e.rowScale[i] : 1.0;
  for (int j = 0; j < e.n; j++)
    columnScale[j] = rc == 0 ? e.columnScale[j] : 1.0;
  return rc;
}
int Clpb_perturbedCosts(Clpb_Simplex *model, double *cost)
{
  // host only: what ClpSimplexDual::perturb would make of the objective for the current status
  clpb::Engine &e = model->e;
  const int rc = e.previewPerturbation(cost);
  return rc;
}
void Clpb_copyinStatus(Clpb_Simplex *model, const unsigned char *statusArray)
{
  model->e.setStatus(statusArray);
}
void Clpb_chgColumnLower(Clpb_Simplex *model, const double *columnLower) { model->e.chgBounds(columnLower, nullptr, nullptr, nullptr); }
void Clpb_chgColumnUpper(Clpb_Simplex *model, const double *columnUpper) { model->e.chgBounds(nullptr, columnUpper, nullptr, nullptr); }
void Clpb_chgRowLower(Clpb_Simplex *model, const double *rowLower) { model->e.chgBounds(nullptr, nullptr, rowLower, nullptr); }
void Clpb_chgRowUpper(Clpb_Simplex *model, const double *rowUpper) { model->e.chgBounds(nullptr, nullptr, nullptr, rowUpper); }
int Clpb_lastSolveWasHot(Clpb_Simplex *model) { return model->e.lastSolveWasHot ? 1 : 0; }
int Clpb_refactorizationInterval(Clpb_Simplex *model, int nucleusSize) { return model->e.cycleFor(nucleusSize); }
int Clpb_dual(Clpb_Simplex *model, int)
{
  return guarded([&] { return model->e.dual(); });
}
int Clpb_primal(Clpb_Simplex *model, int)
{
  return guarded([&] { return model->e.primal(); });
}
void Clpb_chgObjCoefficients(Clpb_Simplex *model, const double *obj) { model->e.chgObjCoefficients(obj); }
int Clpb_primalColumnPivot(Clpb_Simplex *model, const double *dj, const unsigned char *status,
                           const double *weights, int mode)
{
  return guarded([&] { return model->e.primalColumnPivotTest(dj, status, weights, mode); });
}
int Clpb_primalRow(Clpb_Simplex *model, const double *alpha, const double *xB, const double *lowerB,
                   const double *upperB, int direction, double enteringRange, int phase, double *theta)
{
  return guarded([&] {
    return model->e.primalRowTest(alpha, xB, lowerB, upperB, direction, enteringRange, phase, theta);
  });
}
int Clpb_status(Clpb_Simplex *model) { return model->e.problemStatus; }
double Clpb_objectiveValue(Clpb_Simplex *model) { return model->e.objectiveValue; }
int Clpb_numberIterations(Clpb_Simplex *model) { return model->e.numberIterations; }
int Clpb_numberRefactorizations(Clpb_Simplex *model) { return model->e.numberRefactorizations; }
void Clpb_primalColumnSolution(Clpb_Simplex *model, double *x)
{
  if (!model->e.solution.empty())
    std::copy(model->e.solution.begin(), model->e.solution.begin() + model->e.n, x);
}
void Clpb_primalRowSolution(Clpb_Simplex *model, double *y)
{
  if (!model->e.solution.empty())
    std::copy(model->e.solution.begin() + model->e.n, model->e.solution.end(), y);
}
void Clpb_dualColumnSolution(Clpb_Simplex *model, double *dj)
{
  if (!model->e.reducedCost.empty())
    std::copy(model->e.reducedCost.begin(), model->e.reducedCost.begin() + model->e.n, dj);
}
void Clpb_dualRowSolution(Clpb_Simplex *model, double *pi)
{
  if (!model->e.rowPrice.empty())
    std::copy(model->e.rowPrice.begin(), model->e.rowPrice.end(), pi);
}
void Clpb_statusArray(Clpb_Simplex *model, unsigned char *st)
{
  if (!model->e.status.empty())
    std::copy(model->e.status.begin(), model->e.status.end(), st);
  else // before a solve: the status handed in (copyinStatus / readBasis) or the all-slack default
    std::copy(model->e.currentStatus().begin(), model->e.currentStatus().end(), st);
}
int Clpb_writeBasis(Clpb_Simplex *model, const char *filename, int, int)
{
  return model->e.writeBasis(filename);
}
int Clpb_readBasis(Clpb_Simplex *model, const char *filename) { return model->e.readBasis(filename); }
double Clpb_secondsInLoop(Clpb_Simplex *model) { return model->e.secondsInLoop; }
long long Clpb_kernelLaunches(Clpb_Simplex *model) { return model->e.kernelLaunches; }
void Clpb_phaseTimes(Clpb_Simplex *model, double *o /* 14 */)
{
  const clpb::PhaseTimes &p = model->e.phase;
  o[0] = p.chuzr;
  o[1] = p.btran;
  o[2] = p.price;
  o[3] = p.chuzc;
  o[4] = p.dualUpdate;
  o[5] = p.ftran;
  o[6] = p.update;
  o[7] = p.refactor;
  o[8] = (double)p.samples;
  o[9] = p.priceKernel;
  o[10] = p.ftranGemv;
  o[11] = p.btranGemv;
  o[12] = p.ftranGemvBytes;
  o[13] = p.btranGemvBytes;
}
int Clpb_nucleusSize(Clpb_Simplex *model) { return model->e.lastNucleusSize; }
void Clpb_timedWindow(Clpb_Simplex *model, double *milliseconds, int *iterations)
{
  *milliseconds = model->e.timedMilliseconds;
  *iterations = model->e.timedIterations;
}

int Clpb_denseInvert(int k, const double *a, double *x)
{
  return guarded([&] {
    int devCount = 0;
    if (cudaGetDeviceCount(&devCount) != cudaSuccess || devCount == 0)
      throw std::runtime_error("no CUDA device");
    const int ld = (k + 7) / 8 * 8;
    double *dA = nullptr, *dX = nullptr;
    int *dI = nullptr, *dP = nullptr, *dInfo = nullptr;
    cudaMalloc(&dA, sizeof(double) * (size_t)k * ld);
    cudaMalloc(&dX, sizeof(double) * (size_t)k * ld);
    cudaMalloc(&dI, sizeof(int) * k);
    cudaMalloc(&dP, sizeof(int) * k);
    cudaMalloc(&dInfo, sizeof(int));
    cudaMemset(dA, 0, sizeof(double) * (size_t)k * ld);
    // column-major with leading dimension ld
    cudaMemcpy2D(dA, sizeof(double) * ld, a, sizeof(double) * k, sizeof(double) * k, k, cudaMemcpyHostToDevice);
    std::vector<int> hi(k), hp(k);
    cudaStream_t s;
    cudaStreamCreate(&s);
    int info = clpb::dense_invert(dA, dX, k, ld, dI, dP, dInfo, hi.data(), hp.data(), 1.0e-11, s);
    cudaStreamSynchronize(s);
    if (info == 0)
      cudaMemcpy2D(x, sizeof(double) * k, dX, sizeof(double) * ld, sizeof(double) * k, k, cudaMemcpyDeviceToHost);
    cudaStreamDestroy(s);
    cudaFree(dA); cudaFree(dX); cudaFree(dI); cudaFree(dP); cudaFree(dInfo);
    return info;
  });
}

int Clpb_ncclUniqueId(unsigned char *id128)
{
  if (!loadNccl())
    return -1;
  return p_getId(id128);
}
int Clpb_initSharding(Clpb_Simplex *model, int rank, int worldSize, const unsigned char *id128)
{
  if (worldSize <= 1) {
    model->e.rank = 0;
    model->e.worldSize = 1;
    return 0;
  }
  if (!loadNccl())
    return -1;
  NcclId id;
  memcpy(id.internal, id128, 128);
  void *comm = nullptr;
  int rc = p_init(&comm, worldSize, id, rank);
  if (rc != 0)
    return rc;
  CommWrap *w = new CommWrap{comm, rank};
  model->e.rank = rank;
  model->e.worldSize = worldSize;
  model->e.ncclComm = w;
  model->e.allGatherFn = allGatherBytes;
  return 0;
}

int Clpb_factorize(Clpb_Simplex *model, const int *basicSequence, int *pivotVariable)
{
  return guarded([&] { return model->e.factorize(basicSequence, pivotVariable); });
}
int Clpb_updateColumn(Clpb_Simplex *model, double *region)
{
  return guarded([&] { return model->e.updateColumn(region); });
}
int Clpb_updateColumnTranspose(Clpb_Simplex *model, double *region)
{
  return guarded([&] { return model->e.updateColumnTranspose(region); });
}
int Clpb_replaceColumn(Clpb_Simplex *model, int sequenceIn, int pivotRow)
{
  return guarded([&] { return model->e.replaceColumn(sequenceIn, pivotRow); });
}
int Clpb_transposeTimes(Clpb_Simplex *model, double scalar, const double *pi, double *z)
{
  return guarded([&] {
    model->e.transposeTimes(scalar, pi, z);
    return 0;
  });
}
int Clpb_times(Clpb_Simplex *model, double scalar, const double *x, double *y)
{
  return guarded([&] {
    model->e.times(scalar, x, y);
    return 0;
  });
}
int Clpb_dualColumn(Clpb_Simplex *model, const double *alphaRow, const double *dj,
                    const unsigned char *status, int direction, double infeasibility,
                    double *theta)
{
  return guarded(
      [&] { return model->e.dualColumnTest(alphaRow, dj, status, direction, infeasibility, theta); });
}
int Clpb_pivotRow(Clpb_Simplex *model, int *sequenceOut, int *direction, double *infeasibility)
{
  return guarded([&] { return model->e.pivotRowStep(sequenceOut, direction, infeasibility); });
}
int Clpb_updateColumnTransposeAndPrice(Clpb_Simplex *model, double *rho, double *alphaRow)
{
  return guarded([&] { return model->e.btranPriceStep(rho, alphaRow); });
}
int Clpb_dualColumnDevice(Clpb_Simplex *model, double *theta, double *alpha)
{
  return guarded([&] { return model->e.dualColumnStep(theta, alpha); });
}
double Clpb_updateWeights(Clpb_Simplex *model, int *returnCode)
{
  double alpha = 0.0;
  const int rc = guarded([&] {
    alpha = model->e.updateWeightsStep(returnCode);
    return 0;
  });
  if (rc != 0 && returnCode)
    *returnCode = rc;
  return alpha;
}
int Clpb_updatePrimalSolution(Clpb_Simplex *model, double *changeInObjective)
{
  return guarded([&] { return model->e.updatePrimalStep(changeInObjective); });
}
int Clpb_saveWeights(Clpb_Simplex *model, int mode)
{
  return guarded([&] {
    model->e.saveWeights(mode);
    return 0;
  });
}
int Clpb_unrollWeights(Clpb_Simplex *model) { return model->e.unrollWeights(); }
int Clpb_updateColumnFT(Clpb_Simplex *model, double *region)
{
  return guarded([&] { return model->e.updateColumnFT(region); });
}
int Clpb_updateTwoColumnsFT(Clpb_Simplex *model, double *regionFT, double *regionOther)
{
  // ClpFactorization::updateTwoColumnsFT (hpp:125): the FT column keeps its spike, the other is a plain FTRAN
  return guarded([&] {
    int rc = model->e.updateColumn(regionOther);
    if (rc != 0)
      return rc;
    return model->e.updateColumnFT(regionFT);
  });
}
int Clpb_replaceColumnChecked(Clpb_Simplex *model, int sequenceIn, int pivotRow, double pivotCheck,
                              double acceptablePivot)
{
  return guarded([&] { return model->e.replaceColumnChecked(sequenceIn, pivotRow, pivotCheck, acceptablePivot); });
}
// packed (CoinIndexedVector packedMode) forms: number / indices[] / elements[] in and out, the caller's
// arrays have capacity m (n for transposeTimes); entries below the zero tolerance are dropped
static int packDense(const std::vector<double> &v, double zeroTol, int *indices, double *elements)
{
  int nz = 0;
  for (int i = 0; i < (int)v.size(); i++)
    if (std::fabs(v[i]) > zeroTol) {
      indices[nz] = i;
      elements[nz++] = v[i];
    }
  return nz;
}
int Clpb_updateColumnPacked(Clpb_Simplex *model, int *number, int *indices, double *elements)
{
  return guarded([&] {
    std::vector<double> v(model->e.m, 0.0);
    for (int q = 0; q < *number; q++)
      v[indices[q]] = elements[q];
    const int rc = model->e.updateColumn(v.data());
    *number = packDense(v, model->e.zeroTolerance, indices, elements);
    return rc;
  });
}
int Clpb_updateColumnTransposePacked(Clpb_Simplex *model, int *number, int *indices, double *elements)
{
  return guarded([&] {
    std::vector<double> v(model->e.m, 0.0);
    for (int q = 0; q < *number; q++)
      v[indices[q]] = elements[q];
    const int rc = model->e.updateColumnTranspose(v.data());
    *number = packDense(v, model->e.zeroTolerance, indices, elements);
    return rc;
  });
}
int Clpb_transposeTimesPacked(Clpb_Simplex *model, double scalar, int numberPi, const int *indexPi,
                              const double *elementPi, int *numberZ, int *indexZ, double *elementZ)
{
  return guarded([&] {
    std::vector<double> pi(model->e.m, 0.0), z(model->e.n, 0.0);
    for (int q = 0; q < numberPi; q++)
      pi[indexPi[q]] = elementPi[q];
    model->e.transposeTimes(scalar, pi.data(), z.data());
    *numberZ = packDense(z, model->e.zeroTolerance, indexZ, elementZ);
    return 0;
  });
}
int Clpb_dualColumnRowPass(Clpb_Simplex *model, const double *alphaRow, const double *dj,
                           const unsigned char *status, int direction, double infeasibility, double *theta)
{
  return guarded([&] {
    return model->e.dualColumnTest(alphaRow, dj, status, direction, infeasibility, theta, true);
  });
}
int Clpb_startup(Clpb_Simplex *model)
{
  return guarded([&] { return model->e.startup(); });
}
int Clpb_iterate(Clpb_Simplex *model, int count)
{
  return guarded([&] { return model->e.iterate(count); });
}
void Clpb_getWeights(Clpb_Simplex *model, double *weights)
{
  guarded([&] {
    model->e.getWeights(weights);
    return 0;
  });
}
void Clpb_getDeviceVector(Clpb_Simplex *model, const char *name, double *out)
{
  guarded([&] {
    model->e.getDeviceVector(name, out);
    return 0;
  });
}
}
