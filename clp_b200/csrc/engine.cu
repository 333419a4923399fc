// engine.cu -- host driver of the device-resident dual simplex (see engine.hpp).
#include "engine.hpp"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <stdexcept>

namespace clpb {

#define CUDA_OK(call)                                                                             \
  do {                                                                                            \
    cudaError_t e__ = (call);                                                                     \
    if (e__ != cudaSuccess) {                                                                     \
      fprintf(stderr, "clp_b200: CUDA error %s at %s:%d\n", cudaGetErrorString(e__), __FILE__,    \
              __LINE__);                                                                          \
      throw std::runtime_error("CUDA error");                                                     \
    }                                                                                             \
  } while (0)

static inline int roundUp(int v, int a) { return (v + a - 1) / a * a; }

KernelTimers *g_kernelTimers = nullptr;

Engine::Engine() {}
Engine::~Engine()
{
  freeAll();
}

template <class T> T *Engine::dalloc(size_t count)
{
  void *p = nullptr;
  if (count == 0)
    count = 1;
  CUDA_OK(cudaMalloc(&p, count * sizeof(T)));
  allocs.push_back(p);
  return static_cast<T *>(p);
}

void Engine::freeAll()
{
  for (void *p : allocs)
    cudaFree(p);
  allocs.clear();
  for (cudaEvent_t e : events)
    cudaEventDestroy(e);
  events.clear();
  if (iterGraph)
    cudaGraphExecDestroy(iterGraph);
  iterGraph = nullptr;
  if (primalGraph)
    cudaGraphExecDestroy(primalGraph);
  primalGraph = nullptr;
  if (hState)
    cudaFreeHost(hState);
  if (hRec)
    cudaFreeHost(hRec);
  hState = nullptr;
  hRec = nullptr;
  if (stream)
    cudaStreamDestroy(stream);
  stream = nullptr;
  deviceReady = false;
  factorsValid = false;
  nucCap = 0;
  s1Cap = 0;
}

int Engine::defaultFactorizationFrequency() const
{
  // ClpSimplex::defaultFactorizationFrequency, src/ClpSimplex.cpp:11401-11431
  const int cutoff1 = 10000, base = 75, freq0 = 50, freq1 = 150, maximum = 10000;
  int frequency;
  if (m < cutoff1)
    frequency = base + m / freq0;
  else
    frequency = base + cutoff1 / freq0 + (m - cutoff1) / freq1;
  return std::min(maximum, frequency);
}

int Engine::loadProblem(int numberColumns, int numberRows, const int *columnStart, const int *row,
                        const double *element, const double *columnLower,
                        const double *columnUpper, const double *objective, const double *rowLower,
                        const double *rowUpper)
{
  freeAll();
  n = numberColumns;
  m = numberRows;
  nm = n + m;
  if (nm >= (1 << 20) - 1) {
    fprintf(stderr, "clp_b200: n+m must be below 2^20 (packed argmax keys)\n");
    return -1;
  }
  hColStart.assign(columnStart, columnStart + n + 1);
  const long long nnz = hColStart[n];
  hRow.assign(row, row + nnz);
  hVal.assign(element, element + nnz);
  hLower.assign(nm, 0.0);
  hUpper.assign(nm, 0.0);
  hCost.assign(nm, 0.0);
  auto lo = [](double v) { return v < -1.0e29 ? -kInf : v; };
  auto up = [](double v) { return v > 1.0e29 ? kInf : v; };
  for (int j = 0; j < n; j++) {
    hCost[j] = objective ? objective[j] : 0.0;
    hLower[j] = columnLower ? lo(columnLower[j]) : 0.0;
    hUpper[j] = columnUpper ? up(columnUpper[j]) : kInf;
  }
  for (int i = 0; i < m; i++) {
    hLower[n + i] = rowLower ? lo(rowLower[i]) : -kInf;
    hUpper[n + i] = rowUpper ? up(rowUpper[i]) : kInf;
  }
  haveUserStatus = false;
  hStatus.assign(nm, atLowerBound);
  for (int i = 0; i < m; i++)
    hStatus[n + i] = basic;
  problemStatus = -1;
  return 0;
}

int Engine::readMps(const char *fileName)
{
  int mm, nn;
  std::vector<int> cs, ri;
  std::vector<double> va, cl, cu, ob, rl, ru;
  double off = 0.0;
  int rc = readMpsFile(fileName, mm, nn, cs, ri, va, cl, cu, ob, rl, ru, off, problemName);
  if (rc != 0)
    return rc;
  rc = loadProblem(nn, mm, cs.data(), ri.data(), va.data(), cl.data(), cu.data(), ob.data(),
                   rl.data(), ru.data());
  objectiveOffset = off;
  return rc;
}

void Engine::setStatus(const unsigned char *st)
{
  hStatus.assign(st, st + nm);
  haveUserStatus = true;
  factorsValid = false; // a basis handed in from outside is factorized afresh
}

void Engine::buildRowCopy(const std::vector<double> &val, std::vector<int> &rowStart,
                          std::vector<int> &colIdx, std::vector<double> &rval) const
{
  const long long nnz = hColStart[n];
  rowStart.assign(m + 1, 0);
  colIdx.resize(nnz);
  rval.resize(nnz);
  for (long long e = 0; e < nnz; e++)
    rowStart[hRow[e] + 1]++;
  for (int i = 0; i < m; i++)
    rowStart[i + 1] += rowStart[i];
  std::vector<int> fill(rowStart.begin(), rowStart.end() - 1);
  for (int j = 0; j < n; j++)
    for (int e = hColStart[j]; e < hColStart[j + 1]; e++) {
      int at = fill[hRow[e]]++;
      colIdx[at] = j;
      rval[at] = val[e];
    }
}

// computeScaling / prepareWorkingProblem / perturbCosts / previewPerturbation: rim_prep.cpp

// MPS basis file, restating ClpSimplexOther::writeBasis (src/ClpSimplexOther.cpp:1018-1133, the
// branch without names and without values): every basic column is paired with the next nonbasic
// row -- "XU Cj Ri" if that row sits at its upper bound, "XL Cj Ri" otherwise; "UL Cj" marks a
// nonbasic column at its upper bound; everything not mentioned is a column at lower bound / a
// basic row.
int Engine::writeBasis(const char *fileName) const
{
  FILE *fp = fopen(fileName, "w");
  if (!fp)
    return -1;
  fprintf(fp, "NAME          %s       \n", problemName.empty() ? "BLANK" : problemName.c_str());
  int iRow = 0;
  for (int j = 0; j < n; j++) {
    if (hStatus[j] == basic) {
      for (; iRow < m; iRow++)
        if (hStatus[n + iRow] != basic)
          break;
      if (iRow != m) {
        fprintf(fp, " %s C%7.7d     R%7.7d\n", hStatus[n + iRow] == atUpperBound ? "XU" : "XL", j, iRow);
        iRow++;
      } else {
        fprintf(fp, " BS C%7.7d\n", j); // too many basics
      }
    } else if (hStatus[j] == atUpperBound) {
      fprintf(fp, " UL C%7.7d\n", j);
    }
  }
  fprintf(fp, "ENDATA\n");
  fclose(fp);
  return 0;
}

// The reader side lives in CoinMpsIO::readBasis (CoinUtils, not in the reference tree; call site
// src/ClpSimplexOther.cpp:1155).  Standard MPS basis semantics: start from "all columns at lower
// bound, all rows basic"; XU/XL make the column basic and the row nonbasic at upper/lower; UL/LL
// put a column at its upper/lower bound; BS makes a column basic.  Returns 0, -1 (cannot open) or
// the number of records that could not be interpreted.
int Engine::readBasis(const char *fileName)
{
  FILE *fp = fopen(fileName, "r");
  if (!fp)
    return -1;
  std::vector<unsigned char> st(nm, atLowerBound);
  for (int i = 0; i < m; i++)
    st[n + i] = basic;
  auto index = [](const char *name, char kind, int limit) {
    if (name[0] != kind)
      return -1;
    char *end = nullptr;
    long v = strtol(name + 1, &end, 10);
    if (end == name + 1 || v < 0 || v >= limit)
      return -1;
    return (int)v;
  };
  char line[512];
  int bad = 0;
  while (fgets(line, sizeof(line), fp)) {
    char key[16] = "", a[64] = "", b[64] = "";
    const int got = sscanf(line, "%15s %63s %63s", key, a, b);
    if (got < 1 || !strcmp(key, "NAME"))
      continue;
    if (!strcmp(key, "ENDATA"))
      break;
    const int j = got >= 2 ? index(a, 'C', n) : -1;
    if (!strcmp(key, "XU") || !strcmp(key, "XL")) {
      const int i = got >= 3 ? index(b, 'R', m) : -1;
      if (j < 0 || i < 0) {
        bad++;
        continue;
      }
      st[j] = basic;
      st[n + i] = key[1] == 'U' ? atUpperBound : atLowerBound;
    } else if (!strcmp(key, "UL") || !strcmp(key, "LL") || !strcmp(key, "BS")) {
      if (j < 0) {
        bad++;
        continue;
      }
      st[j] = key[0] == 'U' ? atUpperBound : key[0] == 'L' ? atLowerBound : basic;
    } else {
      bad++;
    }
  }
  fclose(fp);
  setStatus(st.data());
  return bad;
}

bool Engine::shardActive() const
{
  if (worldSize <= 1 || allGatherFn == nullptr || hColStart.empty())
    return false;
  const long long per = (n + worldSize - 1) / worldSize;
  if (per * worldSize > nm) // the in-place all-gather of the row shards pads into the slack part
    return false;
  return (long long)hColStart[n] / worldSize >= shardMinNnzPerRank;
}

// Refactorization interval for a nucleus of size k under the default policy: the base interval (2x the
// reference's default), stretched when the modelled cost of a refactorization -- 2k^3 flops at the ~18
// TFLOP/s the rank-32/128 updates reach, plus ~3.5 us per panel column -- exceeds 35 % of the modelled cost
// of the iterations of a cycle (two passes over the explicit inverse, one over A, ~110 us of latency-bound
// kernels, at the ~4.4 TB/s the streams reach).  Capped at 2048 and by a 2 GB eta panel.
int Engine::cycleFor(int k) const
{
  const int base = std::max(8, std::min(2 * defaultFactorizationFrequency(), 2048));
  if (factorizationFrequency > 0)
    return std::max(8, std::min(factorizationFrequency, 2048));
  const double kk = (double)k;
  const double refactorSeconds = 2.0 * kk * kk * kk / 1.8e13 + kk * 3.5e-6 + 5.0e-3;
  const double nnz = hColStart.empty() ? 0.0 : (double)hColStart[n];
  const double iterationSeconds = (16.0 * kk * kk + 12.0 * nnz) / 4.4e12 + 110.0e-6;
  int cycle = (int)(refactorSeconds / (0.35 * iterationSeconds));
  const int memoryCap = (int)std::min(2048.0, 2.0e9 / (8.0 * std::max(1, m)));
  cycle = std::max(base, std::min(cycle, std::max(base, memoryCap)));
  return cycle;
}

int Engine::setupDevice()
{
  // what the device copy was built for: a later scaling() / factorizationFrequency / timing change
  // rebuilds it instead of being silently ignored
  const long long signature = (long long)scalingFlag * 1000003ll + (long long)factorizationFrequency * 101ll +
                              (timing ? 7 : 0) + (long long)worldSize * 13ll + (long long)rank * 17ll +
                              (usePriceTma ? 3 : 0) + (long long)factorMode * 29ll + (shardActive() ? 31 : 0) + (long long)(shardPanelMode + 1) * 37ll + (long long)dualRowPivot * 41ll + (priceIdx16 ? 43 : 0);
  if (deviceReady && signature == readySignature)
    return 0;
  if (deviceReady)
    freeAll();
  readySignature = signature;
  int devCount = 0;
  if (cudaGetDeviceCount(&devCount) != cudaSuccess || devCount == 0) {
    fprintf(stderr, "clp_b200: no CUDA device -- this engine has no CPU fallback\n");
    throw std::runtime_error("no CUDA device");
  }
  CUDA_OK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  const long long nnz = hColStart[n];
  prepareWorkingProblem(); // scaling (if asked for) -> wVal / wLower / wUpper / wCost
  // row copy (CSR) built on the host once
  std::vector<int> rowStart, colIdx;
  std::vector<double> rval;
  buildRowCopy(wVal, rowStart, colIdx, rval);
  d.m = m;
  d.n = n;
  d.nm = nm;
  d.nnz = nnz;
  int *p;
  double *q;
  p = dalloc<int>(n + 1);
  CUDA_OK(cudaMemcpy(p, hColStart.data(), sizeof(int) * (n + 1), cudaMemcpyHostToDevice));
  d.colStart = p;
  p = dalloc<int>(nnz + 16); // padding: TMA tiles are rounded to 16-byte granules
  CUDA_OK(cudaMemset(p, 0, sizeof(int) * (nnz + 16)));
  CUDA_OK(cudaMemcpy(p, hRow.data(), sizeof(int) * nnz, cudaMemcpyHostToDevice));
  d.rowIdx = p;
  d.rowIdx16 = nullptr;
  if (m <= 65535 && priceIdx16) {
    std::vector<unsigned short> r16((size_t)nnz + 32, 0);
    for (long long e = 0; e < nnz; e++)
      r16[e] = (unsigned short)hRow[e];
    unsigned short *p16 = dalloc<unsigned short>(nnz + 32);
    CUDA_OK(cudaMemcpy(p16, r16.data(), sizeof(unsigned short) * (nnz + 32), cudaMemcpyHostToDevice));
    d.rowIdx16 = p16;
  }
  q = dalloc<double>(nnz + 16);
  CUDA_OK(cudaMemset(q, 0, sizeof(double) * (nnz + 16)));
  CUDA_OK(cudaMemcpy(q, wVal.data(), sizeof(double) * nnz, cudaMemcpyHostToDevice));
  d.val = q;
  {
    // cut this rank's column range into tiles of whole columns, <= kPriceTile entries each
    const bool sh = shardActive();
    int per = sh ? (n + worldSize - 1) / worldSize : n;
    int cb = sh ? std::min(n, rank * per) : 0;
    int ce = sh ? std::min(n, cb + per) : n;
    std::vector<int> tiles;
    bool ok = true;
    int c = cb;
    while (c < ce && ok) {
      tiles.push_back(c);
      const int ea = hColStart[c] & ~3;
      int c1 = c;
      while (c1 < ce && c1 - c < kPriceTileCols && ((hColStart[c1 + 1] + 3) & ~3) - ea <= kPriceTile)
        c1++;
      if (c1 == c)
        ok = false; // a single column does not fit a tile: the LDG-direct kernel is used
      c = c1;
    }
    tiles.push_back(ce);
    d.priceTileCol = nullptr;
    d.numPriceTiles = 0;
    const int ntl = (int)tiles.size() - 1;
    if (ok && ce > cb && usePriceTma) {
      std::vector<int> desc((size_t)ntl * 4);
      for (int t = 0; t < ntl; t++) {
        const int t0 = tiles[t], t1 = tiles[t + 1];
        const int ea = hColStart[t0] & ~3;
        desc[4 * t + 0] = t0;
        desc[4 * t + 1] = t1 - t0;
        desc[4 * t + 2] = ea;
        desc[4 * t + 3] = ((hColStart[t1] + 3) & ~3) - ea;
      }
      int *pt = dalloc<int>(desc.size());
      CUDA_OK(cudaMemcpy(pt, desc.data(), sizeof(int) * desc.size(), cudaMemcpyHostToDevice));
      d.priceTileCol = pt;
      d.numPriceTiles = ntl;
    }
  }
  p = dalloc<int>(m + 1);
  CUDA_OK(cudaMemcpy(p, rowStart.data(), sizeof(int) * (m + 1), cudaMemcpyHostToDevice));
  d.rowStart = p;
  p = dalloc<int>(nnz);
  CUDA_OK(cudaMemcpy(p, colIdx.data(), sizeof(int) * nnz, cudaMemcpyHostToDevice));
  d.colIdx = p;
  q = dalloc<double>(nnz);
  CUDA_OK(cudaMemcpy(q, rval.data(), sizeof(double) * nnz, cudaMemcpyHostToDevice));
  d.rval = q;

  d.cost = dalloc<double>(nm);
  d.costTrue = dalloc<double>(nm);
  d.lower = dalloc<double>(nm);
  d.upper = dalloc<double>(nm);
  d.lowerTrue = dalloc<double>(nm);
  d.upperTrue = dalloc<double>(nm);
  d.sol = dalloc<double>(nm);
  d.dj = dalloc<double>(nm);
  d.status = dalloc<unsigned char>(nm);
  d.fake = dalloc<unsigned char>(nm);
  dFlipFlag = dalloc<unsigned char>(nm);
  d.pivotVariable = dalloc<int>(m);
  d.weights = dalloc<double>(m);
  dWeightsTmp = dalloc<double>(m);
  dSolOld = dalloc<double>(nm);
  dDrift = dalloc<unsigned long long>(1);
  dSrcPos = dalloc<int>(m);
  d.posToNuc = dalloc<int>(m);
  d.nucRow = dalloc<int>(m);
  d.nucCol = dalloc<int>(m);
  dS1RowStart = dalloc<int>(m + 1);
  d.s1RowStart = dS1RowStart;
  dS1cStart = dalloc<int>(m + 1);
  d.s1cStart = dS1cStart;
  // Refactorization interval.  The cost model alone (an eta costs one 8m-byte panel column per solve,
  // a refactorization O(k^3) flops) would put it near 2000 at m = 1e4, but measured on the full-size
  // random LP the long cycle costs ~10x more ITERATIONS to reach the same objective: the basic values
  // carried by the update recurrence drift by 1e-4 .. 1 relative inside such a cycle (Engine::refresh
  // measures it) and the row choice degrades.  Twice the reference's own default
  // (ClpSimplex::defaultFactorizationFrequency) keeps the iteration quality of the reference's cadence
  // (profiles/README.md: cycle experiments) at half its refactorization count.
  // ... except where the refactorization itself is the expensive part (staircase-like LPs whose nucleus is
  // nearly all of the basis: 0.5 s per refactorization at k = 17 000): cycleFor(k) stretches the interval so
  // that the modelled refactorization time stays below ~35 % of the modelled iteration time of a cycle.
  // The model depends on the nucleus size only, so the decision is reproducible and identical on all ranks.
  tmax = factorizationFrequency > 0 ? factorizationFrequency : 2 * defaultFactorizationFrequency();
  tmax = std::max(8, std::min(tmax, 2048));
  currentCycle = tmax;
  const int capacity = factorizationFrequency > 0 ? tmax : cycleFor(m);
  d.tmax = roundUp(capacity, 8);
  d.W = dalloc<double>((size_t)m * d.tmax);
  d.etaPos = dalloc<int>(d.tmax);
  d.etaPrevSame = dalloc<int>(d.tmax);
  d.etaLastOfPos = dalloc<int>(m);
  d.Ginv = dalloc<double>((size_t)d.tmax * d.tmax);
  d.GinvT = dalloc<double>((size_t)d.tmax * d.tmax);
  d.xp = dalloc<double>((size_t)3 * d.tmax);
  d.rho = dalloc<double>(m);
  d.alphaRow = dalloc<double>(nm);
  d.rhs3 = dalloc<double>((size_t)3 * m);
  d.uwork = dalloc<double>(m);
  d.ywork = dalloc<double>((size_t)6 * roundUp(m, 8));
  d.swork = dalloc<double>(roundUp(m, 8));
  d.flipAcc = dalloc<long long>(m);
  CUDA_OK(cudaMemset(d.flipAcc, 0, sizeof(long long) * m));
  d.tailCounter = dalloc<unsigned int>(16);
  CUDA_OK(cudaMemset(d.tailCounter, 0, sizeof(unsigned int) * 16));
  d.gridBar = dalloc<unsigned int>(2);
  CUDA_OK(cudaMemset(d.gridBar, 0, sizeof(unsigned int) * 2));
  d.aqBuf = dalloc<double>(m);
  CUDA_OK(cudaMemset(d.aqBuf, 0, sizeof(double) * m));
  d.candA = dalloc<double>(nm);
  d.candD = dalloc<double>(nm);
  d.candJ = dalloc<int>(nm);
  d.candCount = dalloc<int>(1);
  CUDA_OK(cudaMemset(d.candCount, 0, sizeof(int)));
  d.amax = 1.0;
  for (long long e = 0; e < nnz; e++)
    d.amax = std::max(d.amax, std::fabs(wVal[e]));
  d.mu = dalloc<double>((size_t)3 * d.tmax);
  d.nu = dalloc<double>(d.tmax);
  d.histWeight = dalloc<unsigned long long>(kHistBuckets);
  d.histMin = dalloc<unsigned long long>(kHistBuckets);
  d.hist2Weight = dalloc<unsigned long long>(kHist2Buckets);
  d.hist2Min = dalloc<unsigned long long>(kHist2Buckets);
  d.segTotal = dalloc<unsigned long long>(kHistBuckets / 1024);
  d.segLast = dalloc<int>(kHistBuckets / 1024);
  d.scanCounter = dalloc<unsigned int>(1);
  CUDA_OK(cudaMemset(d.scanCounter, 0, sizeof(unsigned int)));
  CUDA_OK(cudaMemset(d.hist2Weight, 0, sizeof(unsigned long long) * kHist2Buckets));
  CUDA_OK(cudaMemset(d.hist2Min, 0xFF, sizeof(unsigned long long) * kHist2Buckets));
  d.flipList = dalloc<int>(nm);
  d.flipBits = dalloc<unsigned int>((nm + 31) / 32 + 4);
  CUDA_OK(cudaMemset(d.flipBits, 0, sizeof(unsigned int) * ((nm + 31) / 32 + 4)));
  d.st = dalloc<IterState>(1);
  d.fd = dalloc<FactorDesc>(1);
  CUDA_OK(cudaMemset(d.fd, 0, sizeof(FactorDesc)));
  d.recCap = 64;
  d.rec = dalloc<IterRecord>(d.recCap);
  dXn = dalloc<double>(n);
  dRhs = dalloc<double>(m);
  dPi = dalloc<double>(m);
  dZ = dalloc<double>(n);
  dObj = dalloc<double>(2);
  dCounters = dalloc<int>(4);
  dIpiv = dalloc<int>(m);
  dPerm = dalloc<int>(m);
  dInfo = dalloc<int>(1);
  CUDA_OK(cudaMallocHost(&hState, sizeof(IterState)));
  CUDA_OK(cudaMallocHost(&hRec, sizeof(IterRecord) * d.recCap));
  d.k = 0;
  d.ldk = 8;
  d.Ninv = nullptr;
  d.NinvT = nullptr;
  d.primalTolerance = primalTolerance;
  d.dualTolerance = dualTolerance;
  d.zeroTolerance = zeroTolerance;
  d.flagged = dalloc<unsigned char>(m);
  d.dantzig = dualRowPivot == 1 ? 1 : 0;
  d.devex = dalloc<double>(nm);
  d.devexRef = dalloc<unsigned char>(nm);
  d.colFlagged = dalloc<unsigned char>(nm);
  CUDA_OK(cudaMemset(d.colFlagged, 0, nm));
  d.ratioPart = dalloc<double>((m + 255) / 256 + 1);
  d.primalDantzig = 0;
  d.shardW = 1;
  d.shardPanel = 0;
  d.shardRank = 0;
  d.shardPerK = d.shardPerM = roundUp(m, 8);
  d.gatherY = d.gatherB = d.gatherP = nullptr;
  if (shardActive()) {
    d.shardW = worldSize;
    // the eta panel streams 8*m*t bytes (t = updates since the last refactorization, on average half
    // the cycle); sharding it costs one more all-gather per iteration (~50 us inside the graph, measured
    // at C3), so it is sharded only when the average replicated pass is slower than that
    d.shardPanel = shardPanelMode >= 0 ? shardPanelMode
                                       : ((8.0 * m * (tmaxHint() / 2.0)) / 2.8e12 * (1.0 - 1.0 / worldSize) > 120e-6 ? 1 : 0);
    d.shardRank = rank;
    d.shardPerK = d.shardPerM = roundUp((m + worldSize - 1) / worldSize, 8);
    d.gatherY = dalloc<double>((size_t)worldSize * 3 * d.shardPerK);
    d.gatherB = dalloc<double>((size_t)worldSize * d.shardPerK);
    d.gatherP = dalloc<double>((size_t)worldSize * 3 * d.shardPerM);
    CUDA_OK(cudaMemset(d.gatherY, 0, sizeof(double) * worldSize * 3 * d.shardPerK));
    CUDA_OK(cudaMemset(d.gatherB, 0, sizeof(double) * worldSize * d.shardPerK));
    CUDA_OK(cudaMemset(d.gatherP, 0, sizeof(double) * worldSize * 3 * d.shardPerM));
    g_shardCtx.W = worldSize;
    g_shardCtx.rank = rank;
    g_shardCtx.comm = ncclComm;
    g_shardCtx.allGather = allGatherFn;
  }
  CUDA_OK(cudaMemset(d.flagged, 0, m));

  CUDA_OK(cudaMemcpy(d.costTrue, wCost.data(), sizeof(double) * nm, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(d.cost, wCost.data(), sizeof(double) * nm, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(d.lowerTrue, wLower.data(), sizeof(double) * nm, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(d.upperTrue, wUpper.data(), sizeof(double) * nm, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(d.lower, wLower.data(), sizeof(double) * nm, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(d.upper, wUpper.data(), sizeof(double) * nm, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemset(d.fake, 0, nm));
  CUDA_OK(cudaMemset(d.dj, 0, sizeof(double) * nm));
  CUDA_OK(cudaMemset(d.histWeight, 0, sizeof(unsigned long long) * kHistBuckets));
  CUDA_OK(cudaMemset(d.histMin, 0xFF, sizeof(unsigned long long) * kHistBuckets));
  CUDA_OK(cudaMemset(d.st, 0, sizeof(IterState)));
  if (timing) {
    events.resize(16 * 8 + 2);
    for (auto &e : events)
      CUDA_OK(cudaEventCreate(&e));
    kernelTimers.resize(16);
    for (auto &kt : kernelTimers)
      for (int q = 0; q < 2; q++) {
        CUDA_OK(cudaEventCreate(&kt.price[q]));
        CUDA_OK(cudaEventCreate(&kt.ftranGemv[q]));
        CUDA_OK(cudaEventCreate(&kt.btranGemv[q]));
      }
  }
  deviceReady = true;
  return 0;
}

void Engine::setAcceptablePivot(double value)
{
  currentAcceptablePivot = value;
  CUDA_OK(cudaMemcpyAsync(&d.st->acceptablePivot, &currentAcceptablePivot, sizeof(double), cudaMemcpyHostToDevice, stream));
  CUDA_OK(cudaStreamSynchronize(stream));
}

void Engine::resetStateForRun()
{
  // nonbasic variables start at a finite bound; weights 1 (ClpDualRowSteepest::saveWeights mode 1)
  std::vector<double> sol0(nm, 0.0);
  int nBasic = 0;
  for (int j = 0; j < nm; j++)
    if (hStatus[j] == basic)
      nBasic++;
  if (nBasic != m) {
    hStatus.assign(nm, atLowerBound);
    for (int i = 0; i < m; i++)
      hStatus[n + i] = basic;
  }
  for (int j = 0; j < nm; j++) {
    if (hStatus[j] == basic)
      continue;
    double lo = wLower[j], up = wUpper[j];
    if (lo > -kInf && up < kInf) {
      if (lo == up) {
        hStatus[j] = isFixed;
        sol0[j] = lo;
      } else if (hStatus[j] == atUpperBound)
        sol0[j] = up;
      else {
        hStatus[j] = atLowerBound;
        sol0[j] = lo;
      }
    } else if (lo > -kInf) {
      hStatus[j] = atLowerBound;
      sol0[j] = lo;
    } else if (up < kInf) {
      hStatus[j] = atUpperBound;
      sol0[j] = up;
    } else {
      hStatus[j] = isFree;
      sol0[j] = 0.0;
    }
  }
  hPivot.clear();
  for (int j = 0; j < nm; j++)
    if (hStatus[j] == basic)
      hPivot.push_back(j);
  CUDA_OK(cudaMemcpy(d.sol, sol0.data(), sizeof(double) * nm, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(d.status, hStatus.data(), nm, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(d.pivotVariable, hPivot.data(), sizeof(int) * m, cudaMemcpyHostToDevice));
  std::vector<double> w(m, 1.0);
  CUDA_OK(cudaMemcpy(d.weights, w.data(), sizeof(double) * m, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(d.cost, wCost.data(), sizeof(double) * nm, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(d.lower, wLower.data(), sizeof(double) * nm, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(d.upper, wUpper.data(), sizeof(double) * nm, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemset(d.fake, 0, nm));
  CUDA_OK(cudaMemset(d.st, 0, sizeof(IterState)));
  CUDA_OK(cudaMemset(d.flipAcc, 0, sizeof(long long) * m));
  CUDA_OK(cudaMemset(d.tailCounter, 0, sizeof(unsigned int) * 16));
  CUDA_OK(cudaMemset(d.gridBar, 0, sizeof(unsigned int) * 2));
  CUDA_OK(cudaMemset(d.aqBuf, 0, sizeof(double) * m));
  CUDA_OK(cudaMemset(d.candCount, 0, sizeof(int)));
  d.primalTolerance = primalTolerance;
  d.dualTolerance = dualTolerance;
  d.zeroTolerance = zeroTolerance;
  CUDA_OK(cudaMemset(d.flagged, 0, m));
  setAcceptablePivot(acceptablePivot);
  currentDualBound = dualBound;
  if (iterGraph) { // DeviceModel (tolerances included) is captured by value: a new run re-captures
    cudaGraphExecDestroy(iterGraph);
    iterGraph = nullptr;
  }
}

// ---------------------------------------------------------------------------------------
// Refactorize the current basis.  Host: canonical positions, nucleus index sets, S1 (symbolic
// part: ClpFactorization::factorize gather of the basis, ClpFactorization.cpp:2212-2244).
// Device: dense nucleus gather, LU, inverse, transpose (numerical part).
int Engine::refactor()
{
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (timing) {
    e0 = events[events.size() - 2];
    e1 = events[events.size() - 1];
    cudaEventRecord(e0, stream);
  }
  CUDA_OK(cudaMemcpyAsync(hStatus.data(), d.status, nm, cudaMemcpyDeviceToHost, stream));
  hPivot.resize(m);
  CUDA_OK(cudaMemcpyAsync(hPivot.data(), d.pivotVariable, sizeof(int) * m, cudaMemcpyDeviceToHost,
                          stream));
  CUDA_OK(cudaStreamSynchronize(stream));
  std::vector<int> hostIpiv(m), hostPerm(m);
  for (int attempt = 0; attempt < 200; attempt++) {
    // ---- canonical positions: basic slack of row i at position i, structurals elsewhere
    std::vector<int> newPivot(m, -1), srcPos(m, -1);
    std::vector<int> queue; // old positions of structurals that must move
    std::vector<int> oldPosOf;
    for (int p = 0; p < m; p++) {
      int seq = hPivot[p];
      if (seq >= n) {
        int i = seq - n;
        newPivot[i] = seq;
        srcPos[i] = p;
      }
    }
    for (int p = 0; p < m; p++) {
      int seq = hPivot[p];
      if (seq < n) {
        if (newPivot[p] < 0 && hStatus[n + p] != basic) {
          newPivot[p] = seq;
          srcPos[p] = p;
        } else
          queue.push_back(p);
      }
    }
    {
      size_t qi = 0;
      for (int p = 0; p < m && qi < queue.size(); p++)
        if (newPivot[p] < 0) {
          newPivot[p] = hPivot[queue[qi]];
          srcPos[p] = queue[qi];
          qi++;
        }
    }
    // ---- nucleus index sets
    std::vector<int> posToNuc(m, -1), nucRow, nucCol;
    for (int p = 0; p < m; p++)
      if (newPivot[p] < n) {
        posToNuc[p] = (int)nucRow.size();
        nucRow.push_back(p);
        nucCol.push_back(newPivot[p]);
      }
    const int k = (int)nucRow.size();
    const int ldk = std::max(8, roundUp(k, 8));
    // ---- nucleus buffers and index sets go to the device first: the LU can start
    if ((size_t)k * ldk > nucCap) {
      int kc = std::min(m, std::max(k + k / 4 + 64, 256));
      int ldc = roundUp(kc, 8);
      nucCap = (size_t)kc * ldc;
      // the old (smaller) pair is released first: at m = 5e4 a factor pair is up to 40 GB
      for (double *old : {d.Ninv, d.NinvT})
        if (old) {
          CUDA_OK(cudaFree(old));
          allocs.erase(std::remove(allocs.begin(), allocs.end(), (void *)old), allocs.end());
        }
      // + worldSize columns: the in-place all-gather of the sharded inverse rounds k up to W*ceil(k/W)
      d.Ninv = dalloc<double>(nucCap + (size_t)(worldSize + 1) * ldc);
      d.NinvT = dalloc<double>(nucCap + (size_t)(worldSize + 1) * ldc);
    }
    d.k = k;
    d.ldk = ldk;
    CUDA_OK(cudaMemcpyAsync(d.posToNuc, posToNuc.data(), sizeof(int) * m, cudaMemcpyHostToDevice, stream));
    if (k > 0) {
      CUDA_OK(cudaMemcpyAsync(d.nucRow, nucRow.data(), sizeof(int) * k, cudaMemcpyHostToDevice, stream));
      CUDA_OK(cudaMemcpyAsync(d.nucCol, nucCol.data(), sizeof(int) * k, cudaMemcpyHostToDevice, stream));
    }
    std::vector<int> s1Start, s1Col, s1cStart, s1cRow;
    std::vector<double> s1Val, s1cVal;
    auto buildS1 = [&]() {
      // ---- S1 = A[C rows, nucleus columns] as CSR over positions (host work, overlapped with the LU)
    s1Start.assign(m + 1, 0);
    for (int j = 0; j < k; j++)
      for (int e = hColStart[nucCol[j]]; e < hColStart[nucCol[j] + 1]; e++)
        if (posToNuc[hRow[e]] < 0)
          s1Start[hRow[e] + 1]++;
    for (int i = 0; i < m; i++)
      s1Start[i + 1] += s1Start[i];
    s1Col.resize(s1Start[m]);
    s1Val.resize(s1Start[m]);
    // the same entries by nucleus column (this loop visits them in that order)
    s1cStart.assign(k + 1, 0);
    s1cRow.resize(s1Start[m]);
    s1cVal.resize(s1Start[m]);
    {
      std::vector<int> fill(s1Start.begin(), s1Start.end() - 1);
      int atc = 0;
      for (int j = 0; j < k; j++) {
        for (int e = hColStart[nucCol[j]]; e < hColStart[nucCol[j] + 1]; e++) {
          int i = hRow[e];
          if (posToNuc[i] < 0) {
            int at = fill[i]++;
            s1Col[at] = j;
            s1Val[at] = wVal[e];
            s1cRow[atc] = i;
            s1cVal[atc] = wVal[e];
            atc++;
          }
        }
        s1cStart[j + 1] = atc;
      }
    }
    };
    int info = 0;
    if (k > 0) {
      // row-major nucleus N in NinvT == column-major N^T ; inverse comes out as row-major N^-1
      CUDA_OK(cudaMemsetAsync(d.NinvT, 0, sizeof(double) * (size_t)k * ldk, stream));
      launch_gather_nucleus_matrix(d, d.NinvT, ldk, stream);
      struct Ctx {
        decltype(buildS1) *fn;
      } ctx{&buildS1};
      info = dense_invert(d.NinvT, d.Ninv, k, ldk, dIpiv, dPerm, dInfo, hostIpiv.data(),
                          hostPerm.data(), 1.0e-11, stream, d.shardW, d.shardRank,
                          d.shardW > 1 ? allGatherFn : nullptr, ncclComm,
                          [](void *c) { (*static_cast<Ctx *>(c)->fn)(); }, &ctx);
      if (info < 0)
        throw std::runtime_error("clp_b200: refactorization failed (allocation or collective)");
      kernelLaunches += 6 * ((k + 31) / 32) * 2;
    } else {
      buildS1();
    }
    if ((size_t)s1Start[m] > s1Cap) {
      s1Cap = (size_t)s1Start[m] * 3 / 2 + 1024;
      dS1Col = dalloc<int>(s1Cap);
      dS1Val = dalloc<double>(s1Cap);
      dS1cRow = dalloc<int>(s1Cap);
      dS1cVal = dalloc<double>(s1Cap);
    }
    d.s1Col = dS1Col;
    d.s1Val = dS1Val;
    {
      FactorDesc hfd;
      hfd.k = k;
      hfd.ldk = ldk;
      hfd.Ninv = d.Ninv;
      hfd.NinvT = d.NinvT;
      hfd.s1Col = dS1Col;
      hfd.s1Val = dS1Val;
      hfd.s1cRow = dS1cRow;
      hfd.s1cVal = dS1cVal;
      // pageable source: the runtime stages the bytes before the call returns, hfd may go out of scope
      CUDA_OK(cudaMemcpyAsync(d.fd, &hfd, sizeof(FactorDesc), cudaMemcpyHostToDevice, stream));
    }
    CUDA_OK(cudaMemcpyAsync(dS1RowStart, s1Start.data(), sizeof(int) * (m + 1), cudaMemcpyHostToDevice, stream));
    CUDA_OK(cudaMemcpyAsync(dS1cStart, s1cStart.data(), sizeof(int) * (k + 1), cudaMemcpyHostToDevice, stream));
    if (s1Start[m] > 0) {
      CUDA_OK(cudaMemcpyAsync(dS1Col, s1Col.data(), sizeof(int) * s1Start[m], cudaMemcpyHostToDevice, stream));
      CUDA_OK(cudaMemcpyAsync(dS1Val, s1Val.data(), sizeof(double) * s1Start[m], cudaMemcpyHostToDevice, stream));
      CUDA_OK(cudaMemcpyAsync(dS1cRow, s1cRow.data(), sizeof(int) * s1Start[m], cudaMemcpyHostToDevice, stream));
      CUDA_OK(cudaMemcpyAsync(dS1cVal, s1cVal.data(), sizeof(double) * s1Start[m], cudaMemcpyHostToDevice, stream));
    }
    if (info == 0) {
      if (k > 0)
        launch_transpose(d.Ninv, d.NinvT, k, ldk, stream);
      // weights follow their variables; pivotVariable takes the canonical order
      CUDA_OK(cudaMemcpyAsync(dSrcPos, srcPos.data(), sizeof(int) * m, cudaMemcpyHostToDevice, stream));
      launch_permute_weights(d.weights, dWeightsTmp, dSrcPos, m, stream);
      CUDA_OK(cudaMemcpyAsync(d.weights, dWeightsTmp, sizeof(double) * m, cudaMemcpyDeviceToDevice, stream));
      CUDA_OK(cudaMemcpyAsync(d.pivotVariable, newPivot.data(), sizeof(int) * m, cudaMemcpyHostToDevice, stream));
      CUDA_OK(cudaMemsetAsync(d.etaLastOfPos, 0xFF, sizeof(int) * m, stream));
      // numEtas = 0 (keep the rest of the state)
      CUDA_OK(cudaMemsetAsync(&d.st->numEtas, 0, sizeof(int), stream));
      // flagged rows get another chance on fresh factors (ClpSimplexDual.cpp:5024ff unflag)
      CUDA_OK(cudaMemsetAsync(d.flagged, 0, m, stream));
      CUDA_OK(cudaMemsetAsync(&d.st->numFlagged, 0, sizeof(int), stream));
      CUDA_OK(cudaStreamSynchronize(stream));
      hPivot = newPivot;
      factorsValid = true;
      numberRefactorizations++;
      lastNucleusSize = k;
      if (timing) {
        cudaEventRecord(e1, stream);
        cudaEventSynchronize(e1);
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        phase.refactor += ms;
      }
      return 0;
    }
    // ---- singular: the LU ran on N^T, so the failing column is nucleus ROW info-1 (a
    // position whose row is dependent); bring its slack in and drop the structural that the
    // permutation had parked there (ClpFactorization.cpp:2382-2532 does the same repair).
    const int jbad = info - 1;
    for (int i = 0; i < k; i++)
      hostPerm[i] = i;
    for (int j = 0; j < jbad; j++) {
      int pp = hostIpiv[j];
      if (pp != j)
        std::swap(hostPerm[j], hostPerm[pp]);
    }
    const int seqLeave = nucCol[hostPerm[jbad]];
    const int rowEnter = nucRow[jbad];
    if (logLevel > 0)
      fprintf(stderr, "clp_b200: singular basis: structural %d out, slack of row %d in\n",
              seqLeave, rowEnter);
    // new basis list (positions are re-canonicalised on the next attempt)
    for (int p = 0; p < m; p++)
      if (newPivot[p] == seqLeave)
        newPivot[p] = n + rowEnter;
    // make srcPos consistent: treat as a fresh basis for weights of the new slack
    hPivot = newPivot;
    hStatus[n + rowEnter] = basic;
    double lo = wLower[seqLeave], up = wUpper[seqLeave];
    unsigned char st;
    double x;
    if (lo > -kInf) {
      st = (lo == up) ? isFixed : atLowerBound;
      x = lo;
    } else if (up < kInf) {
      st = atUpperBound;
      x = up;
    } else {
      st = isFree;
      x = 0.0;
    }
    hStatus[seqLeave] = st;
    CUDA_OK(cudaMemcpy(d.status + seqLeave, &st, 1, cudaMemcpyHostToDevice));
    unsigned char bs = basic;
    CUDA_OK(cudaMemcpy(d.status + n + rowEnter, &bs, 1, cudaMemcpyHostToDevice));
    CUDA_OK(cudaMemcpy(d.sol + seqLeave, &x, sizeof(double), cudaMemcpyHostToDevice));
    // weights: permute to the (old->new) order first so the next attempt starts from newPivot
    CUDA_OK(cudaMemcpy(dSrcPos, srcPos.data(), sizeof(int) * m, cudaMemcpyHostToDevice));
    launch_permute_weights(d.weights, dWeightsTmp, dSrcPos, m, stream);
    CUDA_OK(cudaMemcpyAsync(d.weights, dWeightsTmp, sizeof(double) * m, cudaMemcpyDeviceToDevice, stream));
    CUDA_OK(cudaStreamSynchronize(stream));
  }
  return -1;
}

int Engine::refresh()
{
  struct CycleUpdate {
    // The interval in force follows the nucleus size of the factorization just made (cost model) and
    // the accuracy the last cycle actually had: when the recurrence-updated basic values agree with the
    // recomputed ones to 1e-7 the cycle may run to the capacity of the update buffers (well-conditioned
    // staircase bases: drift 1e-9, and SHORT cycles cost them iterations), when they drift beyond 1e-5 it
    // falls back to the base interval.  Both inputs are device results that are identical on every rank.
    Engine &e;
    ~CycleUpdate()
    {
      int c = e.cycleFor(e.d.k);
      if (e.factorizationFrequency <= 0 && e.driftMeasured) {
        if (e.lastPrimalDrift < 1.0e-7)
          c = e.d.tmax;
        else if (e.lastPrimalDrift > 1.0e-5)
          c = std::max(8, std::min(2 * e.defaultFactorizationFrequency(), 2048));
      }
      e.currentCycle = std::min(c, e.d.tmax);
    }
  } cycleUpdate{*this};
  // keep the recurrence-updated solution: its distance from the recomputed one is the accuracy monitor
  // of the update cycle (ClpSimplexDual::statusOfProblemInDual compares saved and recomputed values the
  // same way, src/ClpSimplexDual.cpp:5170-5195, and shortens the cycle through forceFactorization_)
  const bool measure = numberRefactorizations > 0;
  if (measure) {
    CUDA_OK(cudaMemcpyAsync(dSolOld, d.sol, sizeof(double) * nm, cudaMemcpyDeviceToDevice, stream));
    CUDA_OK(cudaMemsetAsync(dDrift, 0, sizeof(unsigned long long), stream));
  }
  if (refactor() != 0)
    return -1;
  launch_compute_duals(d, dPi, dZ, stream);
  CUDA_OK(cudaMemsetAsync(dCounters, 0, sizeof(int) * 4, stream));
  launch_make_dual_feasible(d, currentDualBound, dCounters, stream);
  launch_compute_primals(d, dXn, dRhs, stream);
  kernelLaunches += 20;
  if (measure) {
    unsigned long long bits = 0ull;
    launch_primal_drift(d, dSolOld, dDrift, stream);
    CUDA_OK(cudaMemcpyAsync(&bits, dDrift, sizeof(bits), cudaMemcpyDeviceToHost, stream));
    CUDA_OK(cudaStreamSynchronize(stream));
    memcpy(&lastPrimalDrift, &bits, sizeof(double));
    driftMeasured = true;
  }
  if (logLevel > 0 && (logLevel > 1 || numberRefactorizations <= 60 || numberRefactorizations % 25 == 0)) {
    // progress line (the reference prints objective / infeasibilities at every refactorization)
    launch_objective(d, dObj, stream);
    double obj2[2];
    CUDA_OK(cudaMemcpyAsync(obj2, dObj, sizeof(double) * 2, cudaMemcpyDeviceToHost, stream));
    CUDA_OK(cudaStreamSynchronize(stream));
    fprintf(stderr, "clp_b200: it %d refactorizations %d nucleus %d objective %.10g sum primal inf %.6g drift %.3g\n",
            numberIterations, numberRefactorizations, d.k, obj2[0] + objectiveOffset, obj2[1], lastPrimalDrift);
  }
  return 0;
}

// ---------------------------------------------------------------------------------------
// One iteration = 17 kernels (18 when column-sharded).  CHUZR is not among them: the row of the
// next iteration is chosen by the update kernel of the previous one, and launch_chuzr() runs once
// at the start of every batch (enqueueBatchStart).
void Engine::enqueueIteration(bool timed, int slot)
{
  cudaEvent_t *ev = timed ? &events[(size_t)slot * 8] : nullptr;
  g_kernelTimers = timed ? &kernelTimers[slot] : nullptr;
  if (timed)
    cudaEventRecord(ev[1], stream);
  launch_btran_unit(d, true, stream);
  if (timed)
    cudaEventRecord(ev[2], stream);
  bool rowPassed = false;
  if (d.shardW > 1) {
    // column-sharded pricing: this rank's block of raw dot products, then ONE exchange per pricing
    // pass -- an in-place all-gather of the row shards (padded to 'per' entries; the padding lands
    // on the slack part of the row, which the row kernels recompute from rho).  Everything after
    // the gather runs replicated on identical data.
    int per = (n + worldSize - 1) / worldSize;
    int c0 = std::min(n, rank * per), c1 = std::min(n, c0 + per);
    launch_price(d, c0, c1, false, stream);
    if (allGatherFn(ncclComm, d.alphaRow, sizeof(double) * per, stream) != 0)
      throw std::runtime_error("clp_b200: all-gather of the row shards failed");
  } else {
    launch_price(d, 0, n, false, stream);
  }
  if (useRowPass)
    rowPassed = true;
  else
    launch_price_slacks(d, 0, n, true, stream); // status mask, slack part, level-1 histogram
  if (timed)
    cudaEventRecord(ev[3], stream);
  if (rowPassed) {
    // row finalize, ratio test, dual update, flips and the FTRAN right-hand sides in one
    // cooperative kernel (rowpass.cu)
    if (!launch_row_pass(d, stream))
      throw std::runtime_error("row pass launch failed");
    if (timed) {
      cudaEventRecord(ev[4], stream);
      cudaEventRecord(ev[5], stream);
    }
  } else {
    launch_chuzc(d, stream);
    if (timed)
      cudaEventRecord(ev[4], stream);
    launch_dual_update_and_flips(d, d.flipBits, stream);
    if (timed)
      cudaEventRecord(ev[5], stream);
  }
  launch_ftran_iteration(d, rowPassed, stream);
  if (timed)
    cudaEventRecord(ev[6], stream);
  launch_pivot_updates(d, stream);
  if (timed)
    cudaEventRecord(ev[7], stream);
  g_kernelTimers = nullptr;
  kernelLaunches += (rowPassed ? 3 + 1 + 1 + 4 + 1 : 3 + 2 + 4 + 3 + 5 + 1) + (d.shardW > 1 ? 2 : 0);
}

// start of a batch: stand-alone CHUZR (2 kernels)
void Engine::enqueueBatchStart()
{
  launch_chuzr(d, stream);
  kernelLaunches += 2;
}

void Engine::buildIterationGraph()
{
  if (iterGraph)
    return;
  // Capture one iteration.  If the cooperative row-pass launch cannot be captured on this driver,
  // capture again with the separate kernels; if that fails too, run without a graph.
  for (int attempt = 0; attempt < 2 && !iterGraph; attempt++) {
    cudaGraph_t graph = nullptr;
    const long before = kernelLaunches;
    bool ok = cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
    if (ok) {
      try {
        enqueueIteration(false, 0);
      } catch (const std::exception &) {
        ok = false;
      }
      if (cudaStreamEndCapture(stream, &graph) != cudaSuccess || graph == nullptr)
        ok = false;
    }
    kernelLaunches = before;
    if (ok) {
      size_t numNodes = 0;
      cudaGraphGetNodes(graph, nullptr, &numNodes);
      kernelsPerIteration = (int)numNodes;
      if (cudaGraphInstantiate(&iterGraph, graph, 0) != cudaSuccess) {
        iterGraph = nullptr;
        ok = false;
      }
    }
    if (graph)
      cudaGraphDestroy(graph);
    if (!ok) {
      cudaGetLastError(); // clear the sticky capture error
      if (useRowPass) {
        fprintf(stderr, "clp_b200: cooperative row pass not capturable, using the separate kernels\n");
        useRowPass = false;
      } else {
        fprintf(stderr, "clp_b200: CUDA graph capture failed, launching kernels directly\n");
        useGraph = false;
        return;
      }
    }
  }
  if (!iterGraph)
    useGraph = false;
}

void Engine::fetchState()
{
  CUDA_OK(cudaMemcpyAsync(hState, d.st, sizeof(IterState), cudaMemcpyDeviceToHost, stream));
  CUDA_OK(cudaStreamSynchronize(stream));
}

void Engine::downloadSolution()
{
  solution.resize(nm);
  reducedCost.resize(nm);
  rowPrice.resize(m);
  status.resize(nm);
  pivotVariable.resize(m);
  launch_objective(d, dObj, stream);
  double obj[2];
  CUDA_OK(cudaMemcpyAsync(solution.data(), d.sol, sizeof(double) * nm, cudaMemcpyDeviceToHost, stream));
  CUDA_OK(cudaMemcpyAsync(reducedCost.data(), d.dj, sizeof(double) * nm, cudaMemcpyDeviceToHost, stream));
  CUDA_OK(cudaMemcpyAsync(rowPrice.data(), dPi, sizeof(double) * m, cudaMemcpyDeviceToHost, stream));
  CUDA_OK(cudaMemcpyAsync(status.data(), d.status, nm, cudaMemcpyDeviceToHost, stream));
  CUDA_OK(cudaMemcpyAsync(pivotVariable.data(), d.pivotVariable, sizeof(int) * m, cudaMemcpyDeviceToHost, stream));
  CUDA_OK(cudaMemcpyAsync(obj, dObj, sizeof(double) * 2, cudaMemcpyDeviceToHost, stream));
  CUDA_OK(cudaStreamSynchronize(stream));
  objectiveValue = obj[0] + objectiveOffset;
  sumPrimalInfeasibilities = obj[1];
  hStatus = status;
  if (!rowScale.empty()) {
    // back to the user's units (ClpSimplex::deleteRim / unscale, src/ClpSimplex.cpp:9430ff)
    for (int j = 0; j < n; j++) {
      solution[j] *= columnScale[j];
      reducedCost[j] /= columnScale[j];
    }
    for (int i = 0; i < m; i++) {
      solution[n + i] /= rowScale[i];
      reducedCost[n + i] *= rowScale[i];
      rowPrice[i] *= rowScale[i];
    }
  }
}

// An LP without rows or without columns (what presolve can leave behind): every column goes to the
// bound its cost prefers; no device work.  0 optimal, 1 primal infeasible, 2 dual infeasible.
int Engine::trivialSolve()
{
  solution.assign(nm, 0.0);
  reducedCost.assign(nm, 0.0);
  rowPrice.assign(m, 0.0);
  status.assign(nm, atLowerBound);
  pivotVariable.resize(m);
  problemStatus = 0;
  objectiveValue = objectiveOffset;
  sumPrimalInfeasibilities = 0.0;
  for (int j = 0; j < n; j++) {
    const double c = hCost[j], lo = hLower[j], up = hUpper[j];
    double x;
    unsigned char st;
    if (lo > up + primalTolerance)
      problemStatus = 1;
    if (c > dualTolerance || (c >= -dualTolerance && lo > -kInf)) {
      x = lo;
      st = atLowerBound;
      if (lo <= -kInf) {
        problemStatus = problemStatus == 1 ? 1 : 2;
        x = up < kInf ? up : 0.0;
      }
    } else if (c < -dualTolerance || up < kInf) {
      x = up;
      st = atUpperBound;
      if (up >= kInf) {
        problemStatus = problemStatus == 1 ? 1 : 2;
        x = lo > -kInf ? lo : 0.0;
      }
    } else {
      x = 0.0;
      st = isFree;
    }
    if (lo == up)
      st = isFixed;
    solution[j] = x;
    status[j] = st;
    reducedCost[j] = c;
    objectiveValue += c * x;
  }
  for (int i = 0; i < m; i++) { // n == 0: every row activity is 0
    status[n + i] = basic;
    pivotVariable[i] = n + i;
    if (hLower[n + i] > primalTolerance || hUpper[n + i] < -primalTolerance)
      problemStatus = 1;
  }
  hStatus = status;
  return problemStatus;
}

void Engine::boundsToWorking()
{
  wLower = hLower;
  wUpper = hUpper;
  if (rowScale.empty())
    return;
  const auto finite = [](double v) { return v > -kInf && v < kInf; };
  for (int j = 0; j < n; j++) {
    if (finite(wLower[j]))
      wLower[j] /= columnScale[j];
    if (finite(wUpper[j]))
      wUpper[j] /= columnScale[j];
  }
  for (int i = 0; i < m; i++) {
    if (finite(wLower[n + i]))
      wLower[n + i] *= rowScale[i];
    if (finite(wUpper[n + i]))
      wUpper[n + i] *= rowScale[i];
  }
}

void Engine::chgBounds(const double *columnLower, const double *columnUpper, const double *rowLower,
                       const double *rowUpper)
{
  auto lo = [](double v) { return v < -1.0e29 ? -kInf : v; };
  auto up = [](double v) { return v > 1.0e29 ? kInf : v; };
  for (int j = 0; j < n; j++) {
    if (columnLower)
      hLower[j] = lo(columnLower[j]);
    if (columnUpper)
      hUpper[j] = up(columnUpper[j]);
  }
  for (int i = 0; i < m; i++) {
    if (rowLower)
      hLower[n + i] = lo(rowLower[i]);
    if (rowUpper)
      hUpper[n + i] = up(rowUpper[i]);
  }
  if (deviceReady)
    boundsToWorking(); // the scale factors of the device copy stay in force
}

// Re-impose the bounds on the device-resident state of the previous solve and recompute x_B through the
// factors + eta file that are already there (no upload of the matrix, no refactorization).
int Engine::hotPrepare()
{
  CUDA_OK(cudaMemcpyAsync(d.lowerTrue, wLower.data(), sizeof(double) * nm, cudaMemcpyHostToDevice, stream));
  CUDA_OK(cudaMemcpyAsync(d.upperTrue, wUpper.data(), sizeof(double) * nm, cudaMemcpyHostToDevice, stream));
  CUDA_OK(cudaMemsetAsync(&d.st->stop, 0, sizeof(int), stream));
  CUDA_OK(cudaMemsetAsync(d.flagged, 0, m, stream));
  CUDA_OK(cudaMemsetAsync(&d.st->numFlagged, 0, sizeof(int), stream));
  setAcceptablePivot(acceptablePivot);
  currentDualBound = dualBound;
  CUDA_OK(cudaMemsetAsync(dCounters, 0, sizeof(int) * 4, stream));
  launch_make_dual_feasible(d, currentDualBound, dCounters, stream);
  launch_compute_primals(d, dXn, dRhs, stream, true);
  kernelLaunches += 12;
  CUDA_OK(cudaStreamSynchronize(stream));
  return 0;
}

int Engine::startup()
{
  setupDevice();
  uploadPendingCosts();
  resetStateForRun();
  largestPerturbation = 0.0;
  if (perturbation <= 100) {
    // perturbed costs go to d.cost (d.costTrue keeps the true ones); costShifts > 0 makes the
    // optimality branch of dual() restore them and carry on
    std::vector<double> pc(wCost.begin(), wCost.begin() + n);
    if (perturbCosts(pc) == 0) {
      for (int j = 0; j < n; j++)
        largestPerturbation = std::max(largestPerturbation, std::fabs(pc[j] - wCost[j]));
      if (largestPerturbation > 0.0) {
        CUDA_OK(cudaMemcpy(d.cost, pc.data(), sizeof(double) * n, cudaMemcpyHostToDevice));
        const int one = 1;
        CUDA_OK(cudaMemcpy(&d.st->costShifts, &one, sizeof(int), cudaMemcpyHostToDevice));
      }
    }
  }
  return refresh();
}

// ClpSimplexDual::dual (src/ClpSimplexDual.cpp:637) : startup, loop, finish.
int Engine::dual()
{
  auto t0 = std::chrono::steady_clock::now();
  problemStatus = -1;
  numberIterations = 0;
  numberRefactorizations = 0;
  kernelLaunches = 0;
  phase = PhaseTimes();
  if (m == 0 || n == 0)
    return trivialSolve();
  driftMeasured = false;
  // a cost change leaves the basis dual infeasible: the bound-change hot start does not apply
  lastSolveWasHot = hotStart && deviceReady && factorsValid && !costsPending;
  if ((lastSolveWasHot ? hotPrepare() : startup()) != 0) {
    problemStatus = 4;
    return problemStatus;
  }
  int dualBoundIncreases = 0;
  int consecutiveTrouble = 0;
  cudaEvent_t evStart = nullptr, evStop = nullptr;
  CUDA_OK(cudaEventCreate(&evStart));
  CUDA_OK(cudaEventCreate(&evStop));
  bool windowOpen = false;
  int windowStartIteration = 0;
  timedMilliseconds = 0.0;
  timedIterations = 0;
  while (problemStatus < 0) {
    if (numberIterations >= maximumIterations) {
      problemStatus = 3;
      break;
    }
    double el = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    if (el > maximumSeconds) {
      problemStatus = 3;
      break;
    }
    if (!windowOpen && numberIterations >= warmupIterations) {
      CUDA_OK(cudaStreamSynchronize(stream));
      CUDA_OK(cudaEventRecord(evStart, stream));
      windowOpen = true;
      windowStartIteration = numberIterations;
    }
    // enqueue a batch of iterations; kernels become no-ops once the device sets a stop reason
    fetchState();
    int room = std::min(currentCycle, d.tmax) - hState->numEtas;
    if (room <= 0) {
      if (refresh() != 0) {
        problemStatus = 4;
        break;
      }
      continue;
    }
    int count = std::min(std::min(batch, room), maximumIterations - numberIterations);
    if (!windowOpen && warmupIterations > numberIterations)
      count = std::min(count, warmupIterations - numberIterations);
    count = std::min(count, d.recCap);
    if (timing)
      count = std::min(count, 16);
    const int before = hState->iterations;
    cudaEvent_t evChuzr0 = timing ? events[0] : nullptr;
    if (timing)
      cudaEventRecord(evChuzr0, stream);
    enqueueBatchStart();
    if (useGraph && !timing)
      buildIterationGraph(); // may clear useGraph
    if (useGraph && !timing) {
      for (int b = 0; b < count; b++)
        CUDA_OK(cudaGraphLaunch(iterGraph, stream));
      kernelLaunches += (long)count * kernelsPerIteration;
    } else {
      for (int b = 0; b < count; b++)
        enqueueIteration(timing, b);
    }
    fetchState();
    const int done = hState->iterations - before;
    numberIterations += done;
    if (timing) {
      for (int b = 0; b < done; b++) {
        float ms[7];
        ms[0] = 0.0f; // CHUZR is fused into the previous iteration's update kernel
        if (b == 0)
          cudaEventElapsedTime(&ms[0], events[0], events[1]); // the batch's stand-alone CHUZR
        for (int q = 1; q < 7; q++)
          cudaEventElapsedTime(&ms[q], events[(size_t)b * 8 + q], events[(size_t)b * 8 + q + 1]);
        phase.chuzr += ms[0];
        phase.btran += ms[1];
        phase.price += ms[2];
        phase.chuzc += ms[3];
        phase.dualUpdate += ms[4];
        phase.ftran += ms[5];
        phase.update += ms[6];
        float k0 = 0, k1 = 0, k2 = 0;
        cudaEventElapsedTime(&k0, kernelTimers[b].price[0], kernelTimers[b].price[1]);
        cudaEventElapsedTime(&k1, kernelTimers[b].ftranGemv[0], kernelTimers[b].ftranGemv[1]);
        cudaEventElapsedTime(&k2, kernelTimers[b].btranGemv[0], kernelTimers[b].btranGemv[1]);
        phase.priceKernel += k0;
        phase.ftranGemv += k1;
        phase.btranGemv += k2;
        phase.ftranGemvBytes += 8.0 * d.k * d.ldk + 48.0 * d.k; // DESIGN.md section 7
        phase.btranGemvBytes += 8.0 * d.k * d.ldk + 16.0 * d.k;
        phase.samples++;
      }
    }
    if (logLevel > 2) {
      CUDA_OK(cudaMemcpy(hRec, d.rec, sizeof(IterRecord) * d.recCap, cudaMemcpyDeviceToHost));
      for (int b = 0; b < done; b++) {
        const IterRecord &r = hRec[(before + b) % d.recCap];
        fprintf(stderr, "TRACE %d out=%d in=%d sigma=%d thetaD=%.12g thetaP=%.12g alpha=%.12g infeas=%.12g flips=%d\n",
                numberIterations - done + b, r.seqOut, r.seqIn, r.sigma, r.thetaDual, r.thetaPrimal,
                r.alphaCol, r.infeas, r.numFlips);
      }
    }
    if (logLevel > 1)
      fprintf(stderr, "clp_b200: it %d etas %d k %d stop %d infeas %.6g theta %.6g\n",
              numberIterations, hState->numEtas, d.k, hState->stop, hState->infeas,
              hState->thetaDual);
    const int stop = hState->stop;
    if (done > 0 && refreshDualsEvery > 0 && hState->stop == STOP_NONE &&
        (numberIterations / refreshDualsEvery) != ((numberIterations - done) / refreshDualsEvery)) {
      launch_compute_duals(d, dPi, dZ, stream, true);
      CUDA_OK(cudaMemsetAsync(dCounters, 0, sizeof(int) * 4, stream));
      launch_make_dual_feasible(d, currentDualBound, dCounters, stream);
      launch_compute_primals(d, dXn, dRhs, stream, true); // the flips moved nonbasic values
    } else if (done > 0 && refreshPrimalsEvery > 0 && hState->stop == STOP_NONE &&
               (numberIterations / refreshPrimalsEvery) != ((numberIterations - done) / refreshPrimalsEvery)) {
      launch_compute_primals(d, dXn, dRhs, stream, true);
    }
    if (done > 0 && currentAcceptablePivot < acceptablePivot && hState->numEtas >= 5)
      setAcceptablePivot(acceptablePivot); // acceptablePivot_ = fabs(...) once pivots() >= 5 (:2070-2074)
    if (stop == STOP_NONE) {
      consecutiveTrouble = 0;
      continue;
    }
    // clear the stop reason for the next batch
    CUDA_OK(cudaMemsetAsync(&d.st->stop, 0, sizeof(int), stream));
    const bool fresh = hState->numEtas == 0;
    switch (stop) {
    case STOP_ETAS_FULL:
    case STOP_INACCURATE:
      if (stop == STOP_INACCURATE && ++consecutiveTrouble > 50) {
        problemStatus = 4;
        break;
      }
      if (refresh() != 0)
        problemStatus = 4;
      break;
    case STOP_TINY_PIVOT:
      if (++consecutiveTrouble > 5)
        problemStatus = 4;
      else if (refresh() != 0)
        problemStatus = 4;
      break;
    case STOP_NO_ROW: {
      if (!fresh) {
        if (refresh() != 0)
          problemStatus = 4;
        break;
      }
      // primal feasible on fresh factors (statusOfProblemInDual :4996 optimality branch)
      if (hState->costShifts > 0) {
        CUDA_OK(cudaMemcpyAsync(d.cost, d.costTrue, sizeof(double) * nm, cudaMemcpyDeviceToDevice, stream));
        CUDA_OK(cudaMemsetAsync(&d.st->costShifts, 0, sizeof(int), stream));
        if (refresh() != 0)
          problemStatus = 4;
        break;
      }
      int atFake = 0;
      CUDA_OK(cudaMemsetAsync(dCounters, 0, sizeof(int) * 4, stream));
      launch_count_fake(d, dCounters, stream);
      CUDA_OK(cudaMemcpyAsync(&atFake, dCounters, sizeof(int), cudaMemcpyDeviceToHost, stream));
      CUDA_OK(cudaStreamSynchronize(stream));
      if (atFake > 0) {
        if (dualBoundIncreases < 2) {
          dualBoundIncreases++;
          currentDualBound *= 1000.0;
          if (refresh() != 0)
            problemStatus = 4;
          break;
        }
        problemStatus = 2;
        break;
      }
      if (hState->numFlagged > 0) {
        // Every row that is still primal infeasible is flagged: its infeasibility is below the
        // reference's 1e-4 test value and no entering column with an acceptable pivot exists on
        // fresh, refined factors.  The reference leaves the dual here with status 10 and lets the
        // primal simplex remove sum-of-infeasibilities < 1e-3 (ClpSimplexDual.cpp:1988-2010,
        // ClpSimplex.cpp:5808-5851).  There is no primal algorithm on this path: the basis is
        // reported optimal when the flagged infeasibilities stay below that 1e-3 threshold
        // (sumPrimalInfeasibilities says how much), primal infeasible otherwise.
        launch_objective(d, dObj, stream);
        double obj2[2];
        CUDA_OK(cudaMemcpyAsync(obj2, dObj, sizeof(double) * 2, cudaMemcpyDeviceToHost, stream));
        CUDA_OK(cudaStreamSynchronize(stream));
        if (logLevel > 0)
          fprintf(stderr, "clp_b200: %d flagged rows left, sum of primal infeasibilities %.3g\n",
                  hState->numFlagged, obj2[1]);
        problemStatus = obj2[1] < 1.0e-3 ? 0 : 1;
        break;
      }
      problemStatus = 0;
      break;
    }
    case STOP_NO_COLUMN: {
      if (logLevel > 0)
        fprintf(stderr, "clp_b200: no entering column: it %d row %d seqOut %d infeas %.6g etas %d acceptable %.1e flagged %d\n",
                numberIterations, hState->pivotRow, hState->seqOut, hState->infeas, hState->numEtas,
                currentAcceptablePivot, hState->numFlagged);
      if (!fresh) {
        if (refresh() != 0)
          problemStatus = 4;
        break;
      }
      int atFake = 0;
      CUDA_OK(cudaMemsetAsync(dCounters, 0, sizeof(int) * 4, stream));
      launch_count_fake(d, dCounters, stream);
      CUDA_OK(cudaMemcpyAsync(&atFake, dCounters, sizeof(int), cudaMemcpyDeviceToHost, stream));
      CUDA_OK(cudaStreamSynchronize(stream));
      if (atFake > 0 && dualBoundIncreases < 2) {
        dualBoundIncreases++;
        currentDualBound *= 1000.0;
        if (refresh() != 0)
          problemStatus = 4;
        break;
      }
      // the reference only believes "no entering column" on fresh factors once the acceptable
      // pivot has been relaxed to 1e-8 (ClpSimplexDual.cpp:1882-1884, :2072-2074): retry the same
      // row with the smaller tolerance before anything else
      if (currentAcceptablePivot > 1.0e-8) {
        setAcceptablePivot(1.0e-8);
        break;
      }
      // a small infeasibility whose row has no usable pivot: flag the row and carry on with the
      // others (setFlagged, ClpSimplexDual.cpp:2058-2066; test value 1e-4 / 1e-6 of :1984-1988)
      if (hState->infeas < 1.0e-4 && hState->numFlagged < m) {
        const unsigned char one = 1;
        const int nf = hState->numFlagged + 1;
        CUDA_OK(cudaMemcpyAsync(d.flagged + hState->pivotRow, &one, 1, cudaMemcpyHostToDevice, stream));
        CUDA_OK(cudaMemcpyAsync(&d.st->numFlagged, &nf, sizeof(int), cudaMemcpyHostToDevice, stream));
        CUDA_OK(cudaStreamSynchronize(stream));
        break;
      }
      // a real infeasibility: the reference calls the problem infeasible only when the best
      // possible pivot of the row is below 1e-11 (:1978); relax step by step down to that
      if (currentAcceptablePivot > 1.0e-11) {
        setAcceptablePivot(std::max(1.0e-11, currentAcceptablePivot * 0.1));
        break;
      }
      problemStatus = 1;
      break;
    }
    default:
      problemStatus = 4;
      break;
    }
  }
  if (windowOpen) {
    CUDA_OK(cudaEventRecord(evStop, stream));
    CUDA_OK(cudaEventSynchronize(evStop));
    float ms = 0.0f;
    cudaEventElapsedTime(&ms, evStart, evStop);
    timedMilliseconds = ms;
    timedIterations = numberIterations - windowStartIteration;
  }
  cudaEventDestroy(evStart);
  cudaEventDestroy(evStop);
  downloadSolution();
  secondsInLoop = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  return problemStatus;
}

// ---------------------------------------------------------------------------------------
// plug-in level entry points (host buffers in, host buffers out)
int Engine::factorize(const int *basicSequence, int *pivotVariableOut)
{
  setupDevice();
  hStatus.assign(nm, atLowerBound);
  for (int p = 0; p < m; p++)
    hStatus[basicSequence[p]] = basic;
  haveUserStatus = true;
  resetStateForRun();
  // keep the caller's order where it is canonical
  std::vector<int> pv(basicSequence, basicSequence + m);
  CUDA_OK(cudaMemcpy(d.pivotVariable, pv.data(), sizeof(int) * m, cudaMemcpyHostToDevice));
  int rc = refactor();
  if (pivotVariableOut)
    std::copy(hPivot.begin(), hPivot.end(), pivotVariableOut);
  return rc;
}

int Engine::updateColumn(double *vec)
{
  CUDA_OK(cudaMemcpyAsync(d.rhs3, vec, sizeof(double) * m, cudaMemcpyHostToDevice, stream));
  launch_ftran_buffer(d, d.rhs3, 1, true, stream);
  CUDA_OK(cudaMemcpyAsync(vec, d.rhs3, sizeof(double) * m, cudaMemcpyDeviceToHost, stream));
  CUDA_OK(cudaStreamSynchronize(stream));
  return 0;
}

int Engine::updateColumnTranspose(double *vec)
{
  CUDA_OK(cudaMemcpyAsync(d.rho, vec, sizeof(double) * m, cudaMemcpyHostToDevice, stream));
  launch_btran_dense(d, d.rho, true, stream);
  CUDA_OK(cudaMemcpyAsync(vec, d.rho, sizeof(double) * m, cudaMemcpyDeviceToHost, stream));
  CUDA_OK(cudaStreamSynchronize(stream));
  return 0;
}

int Engine::replaceColumn(int sequenceIn, int pivotRow)
{
  fetchState();
  if (hState->numEtas >= std::min(currentCycle, d.tmax))
    return 5; // maximum pivots reached (ClpFactorization.hpp:87)
  if (hState->numEtas >= d.tmax)
    return 3; // no room in the update buffers (:86)
  launch_unpack_column(d, sequenceIn, d.rhs3, stream);
  launch_ftran_buffer(d, d.rhs3, 1, true, stream);
  double alpha = 0.0;
  CUDA_OK(cudaMemcpyAsync(&alpha, d.rhs3 + pivotRow, sizeof(double), cudaMemcpyDeviceToHost, stream));
  CUDA_OK(cudaStreamSynchronize(stream));
  if (!(std::fabs(alpha) >= 1.0e-11))
    return 2;
  launch_eta_append_test(d, pivotRow, sequenceIn, stream);
  CUDA_OK(cudaStreamSynchronize(stream));
  hPivot[pivotRow] = sequenceIn;
  return 0;
}

void Engine::transposeTimes(double scalar, const double *pi, double *z)
{
  setupDevice();
  CUDA_OK(cudaMemcpyAsync(dPi, pi, sizeof(double) * m, cudaMemcpyHostToDevice, stream));
  launch_transpose_times(d, dPi, dZ, scalar, stream);
  CUDA_OK(cudaMemcpyAsync(z, dZ, sizeof(double) * n, cudaMemcpyDeviceToHost, stream));
  CUDA_OK(cudaStreamSynchronize(stream));
}

void Engine::times(double scalar, const double *x, double *y)
{
  setupDevice();
  CUDA_OK(cudaMemcpyAsync(dXn, x, sizeof(double) * n, cudaMemcpyHostToDevice, stream));
  launch_times_rows(d, dXn, dRhs, scalar, stream);
  CUDA_OK(cudaMemcpyAsync(y, dRhs, sizeof(double) * m, cudaMemcpyDeviceToHost, stream));
  CUDA_OK(cudaStreamSynchronize(stream));
}

int Engine::dualColumnTest(const double *alphaRow, const double *dj, const unsigned char *stat,
                           int sigma, double infeas, double *theta, bool rowPass)
{
  setupDevice();
  resetStateForRun();
  CUDA_OK(cudaMemcpy(d.alphaRow, alphaRow, sizeof(double) * nm, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(d.dj, dj, sizeof(double) * nm, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(d.status, stat, nm, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemset(d.rho, 0, sizeof(double) * m));
  IterState st;
  memset(&st, 0, sizeof(st));
  st.sigma = sigma;
  st.acceptablePivot = acceptablePivot;
  st.infeas = infeas;
  CUDA_OK(cudaMemcpy(d.st, &st, sizeof(st), cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemsetAsync(d.histWeight, 0, sizeof(unsigned long long) * kHistBuckets, stream));
  CUDA_OK(cudaMemsetAsync(d.histMin, 0xFF, sizeof(unsigned long long) * kHistBuckets, stream));
  CUDA_OK(cudaMemsetAsync(d.hist2Weight, 0, sizeof(unsigned long long) * kHist2Buckets, stream));
  CUDA_OK(cudaMemsetAsync(d.hist2Min, 0xFF, sizeof(unsigned long long) * kHist2Buckets, stream));
  if (rowPass) {
    // the cooperative kernel of the fused iteration: it derives the slack part of the row from rho
    // (alpha_{n+i} = -rho_i) and also runs the dual update / flips / right-hand sides that follow
    std::vector<double> negRho(m);
    for (int i = 0; i < m; i++)
      negRho[i] = -alphaRow[n + i];
    CUDA_OK(cudaMemcpy(d.rho, negRho.data(), sizeof(double) * m, cudaMemcpyHostToDevice));
    CUDA_OK(cudaMemset(d.posToNuc, 0xFF, sizeof(int) * m)); // no factorization in this entry point
    CUDA_OK(cudaMemsetAsync(d.segTotal, 0, sizeof(unsigned long long) * (kHistBuckets / 1024), stream));
    CUDA_OK(cudaMemsetAsync(d.segLast, 0xFF, sizeof(int) * (kHistBuckets / 1024), stream));
    if (!launch_row_pass(d, stream))
      throw std::runtime_error("row pass launch failed");
  } else {
    launch_histogram(d, stream);
    launch_chuzc(d, stream);
  }
  fetchState();
  *theta = hState->thetaDual;
  if (hState->stop != 0)
    return -1;
  return hState->seqIn;
}

int Engine::iterate(int count)
{
  int total = 0;
  while (count > 0) {
    int c = std::min(count, d.recCap);
    fetchState();
    const int before = hState->iterations;
    enqueueBatchStart();
    for (int b = 0; b < c; b++)
      enqueueIteration(false, b);
    fetchState();
    total += hState->iterations - before;
    if (hState->stop != 0)
      break;
    count -= c;
  }
  return total;
}

// ---------------------------------------------------------------------------------------
// One iteration as separate plug-in calls.  The fused kernels decide where the cuts fall:
//   pivotRowStep      = ClpDualRowSteepest::pivotRow (src/ClpDualRowSteepest.cpp:179)
//   btranPriceStep    = ClpFactorization::updateColumnTranspose (:2993) + ClpPackedMatrix::transposeTimes (:706)
//   dualColumnStep    = ClpSimplexDual::dualColumn (:4192) + updateDualsInDual (:2430) + flipBounds (one kernel)
//   updateWeightsStep = ClpDualRowSteepest::updateWeights (:375): the FT-FTRAN pair (+ flip column) and the
//                       BTRAN/FTRAN pivot agreement gate; returns alpha.  The weights themselves are
//                       written by updatePrimalStep, so a rejected pivot leaves them untouched and
//                       unrollWeights (:1022) has nothing to restore
//   updatePrimalStep  = updatePrimalSolution (:630) + the DSE recurrence (:501-538) + replaceColumn (eta
//                       append) + ClpSimplex::housekeeping (src/ClpSimplex.cpp:2065)
int Engine::pivotRowStep(int *sequenceOut, int *direction, double *infeasibility)
{
  CUDA_OK(cudaMemsetAsync(&d.st->stop, 0, sizeof(int), stream));
  launch_chuzr(d, stream);
  kernelLaunches += 2;
  fetchState();
  if (hState->stop == STOP_NO_ROW || hState->stop == STOP_ETAS_FULL) {
    const int why = hState->stop;
    CUDA_OK(cudaMemsetAsync(&d.st->stop, 0, sizeof(int), stream));
    return why == STOP_NO_ROW ? -1 : -2; // -2: the update buffer is full, factorize first
  }
  if (sequenceOut)
    *sequenceOut = hState->seqOut;
  if (direction)
    *direction = hState->sigma;
  if (infeasibility)
    *infeasibility = hState->infeas;
  return hState->pivotRow;
}

int Engine::btranPriceStep(double *rho, double *alphaRow)
{
  launch_btran_unit(d, true, stream);
  launch_price(d, 0, n, false, stream);
  kernelLaunches += 4;
  std::vector<double> r(m);
  CUDA_OK(cudaMemcpyAsync(r.data(), d.rho, sizeof(double) * m, cudaMemcpyDeviceToHost, stream));
  if (alphaRow)
    CUDA_OK(cudaMemcpyAsync(alphaRow, d.alphaRow, sizeof(double) * n, cudaMemcpyDeviceToHost, stream));
  CUDA_OK(cudaStreamSynchronize(stream));
  int nz = 0;
  for (int i = 0; i < m; i++)
    nz += r[i] != 0.0;
  if (rho)
    std::copy(r.begin(), r.end(), rho);
  return nz;
}

int Engine::dualColumnStep(double *theta, double *alpha)
{
  if (!launch_row_pass(d, stream))
    throw std::runtime_error("row pass launch failed");
  kernelLaunches += 1;
  fetchState();
  if (hState->stop == STOP_NO_COLUMN) {
    CUDA_OK(cudaMemsetAsync(&d.st->stop, 0, sizeof(int), stream));
    return -1;
  }
  if (theta)
    *theta = hState->thetaDual;
  if (alpha)
    *alpha = hState->alphaRow;
  return hState->seqIn;
}

double Engine::updateWeightsStep(int *returnCode)
{
  launch_ftran_iteration(d, true, stream);
  kernelLaunches += 4;
  fetchState();
  int rc = 0;
  if (hState->stop == STOP_INACCURATE || hState->stop == STOP_TINY_PIVOT) {
    rc = hState->stop == STOP_INACCURATE ? 1 : 2; // 1: refactorize and retry, 2: no usable pivot
    CUDA_OK(cudaMemsetAsync(&d.st->stop, 0, sizeof(int), stream));
  }
  if (returnCode)
    *returnCode = rc;
  return hState->alphaCol;
}

int Engine::updatePrimalStep(double *changeInObjective)
{
  fetchState();
  const int r = hState->pivotRow, q = hState->seqIn;
  const double gain = hState->thetaDual * hState->infeas; // dual objective gain of the step
  launch_pivot_updates(d, stream);
  kernelLaunches += 1;
  fetchState();
  if (changeInObjective)
    *changeInObjective = gain;
  if (r >= 0 && r < m && q >= 0)
    hPivot[r] = q;
  // the tail of the update kernel already decoded the next pivot row; the stepwise caller asks for it
  // again through pivotRowStep, so a "no row" stop raised here is not an error
  if (hState->stop != 0)
    CUDA_OK(cudaMemsetAsync(&d.st->stop, 0, sizeof(int), stream));
  return hState->numEtas;
}

// ClpDualRowSteepest::saveWeights (src/ClpDualRowSteepest.cpp:773): weights travel with their VARIABLE
// across a refactorization.  1 remember which sequence sits at every position (+ snapshot); 2 re-map the
// snapshot onto the new pivot order (new basics get 1.0, clip at DEVEX_TRY_NORM) and snapshot again;
// 4 restore the snapshot; 5 / 7 initialise to 1.0; 3 / 6 nothing to do here (no infeasibility list is kept:
// CHUZR scans every position).
void Engine::saveWeights(int mode)
{
  if (!deviceReady)
    return;
  std::vector<int> pv(m);
  std::vector<double> w(m);
  CUDA_OK(cudaMemcpy(pv.data(), d.pivotVariable, sizeof(int) * m, cudaMemcpyDeviceToHost));
  CUDA_OK(cudaMemcpy(w.data(), d.weights, sizeof(double) * m, cudaMemcpyDeviceToHost));
  if (mode == 1) {
    savedWeightSeq = pv;
    savedWeightVal = w;
  } else if (mode == 5 || mode == 7 || ((mode == 2 || mode == 4) && savedWeightSeq.empty())) {
    w.assign(m, 1.0);
    CUDA_OK(cudaMemcpy(d.weights, w.data(), sizeof(double) * m, cudaMemcpyHostToDevice));
    savedWeightSeq = pv;
    savedWeightVal = w;
  } else if (mode == 2 || mode == 4) {
    std::vector<int> back(nm, -1);
    for (int i = 0; i < m; i++)
      back[savedWeightSeq[i]] = i;
    for (int i = 0; i < m; i++) {
      const int b = back[pv[i]];
      w[i] = b >= 0 ? std::max(savedWeightVal[b], kDevexTryNorm) : 1.0;
    }
    CUDA_OK(cudaMemcpy(d.weights, w.data(), sizeof(double) * m, cudaMemcpyHostToDevice));
    savedWeightSeq = pv;
    savedWeightVal = w;
  }
}

int Engine::unrollWeights()
{
  return 0;
}

// ClpFactorization::updateColumnFT (src/ClpFactorization.hpp:113): FTRAN in place; the result is also
// what replaceColumn needs (in product form the "spike" is the FTRAN'd column itself), so it stays in
// the first right-hand-side slot on the device.  Returns the number of nonzeros, or -1 when there is
// no room for another update (hpp:120-123: negative = no room).
int Engine::updateColumnFT(double *vec)
{
  fetchState();
  if (hState->numEtas >= d.tmax)
    return -1;
  CUDA_OK(cudaMemcpyAsync(d.rhs3, vec, sizeof(double) * m, cudaMemcpyHostToDevice, stream));
  launch_ftran_buffer(d, d.rhs3, 1, true, stream);
  CUDA_OK(cudaMemcpyAsync(vec, d.rhs3, sizeof(double) * m, cudaMemcpyDeviceToHost, stream));
  CUDA_OK(cudaStreamSynchronize(stream));
  int nz = 0;
  for (int i = 0; i < m; i++) {
    if (std::fabs(vec[i]) < zeroTolerance)
      vec[i] = 0.0;
    nz += vec[i] != 0.0;
  }
  return nz;
}

// ClpFactorization::replaceColumn with its checks (hpp:82-89; CoinAbcTypeFactorization::checkPivot,
// src/CoinAbcBaseFactorization4.cpp:94-131): 0 ok, 1 pivot agrees with pivotCheck only to 1e-8 relative
// ("probably ok", the update is made), 2 singular or inaccurate (nothing changed), 3 no room in the
// update buffers, 5 the maximum number of pivots (factorizationFrequency) is reached.
int Engine::replaceColumnChecked(int sequenceIn, int pivotRow, double pivotCheck, double acceptable)
{
  fetchState();
  const int t = hState->numEtas;
  if (t >= std::min(currentCycle, d.tmax))
    return 5; // maximum pivots reached (the update buffers hold at least that many), so
  if (t >= d.tmax)
    return 3; // "no room" (:86) can only be seen if the two limits are ever decoupled
  launch_unpack_column(d, sequenceIn, d.rhs3, stream);
  launch_ftran_buffer(d, d.rhs3, 1, true, stream);
  double alpha = 0.0;
  CUDA_OK(cudaMemcpyAsync(&alpha, d.rhs3 + pivotRow, sizeof(double), cudaMemcpyDeviceToHost, stream));
  CUDA_OK(cudaStreamSynchronize(stream));
  if (!(std::fabs(alpha) > 1.0e-8) || std::fabs(alpha) < acceptable)
    return 2;
  int rc = 0;
  if (pivotCheck != 0.0) {
    const double checkTolerance = t < 2 ? 1.0e-5 : t < 10 ? 1.0e-6 : t < 50 ? 1.0e-8 : 1.0e-10;
    const double rel = std::fabs(1.0 - std::fabs(alpha / pivotCheck));
    if (rel >= checkTolerance)
      rc = (std::fabs(std::fabs(pivotCheck) - std::fabs(alpha)) < 1.0e-12 || rel < 1.0e-8) ? 1 : 2;
    if (rc == 2)
      return 2;
  }
  launch_eta_append_test(d, pivotRow, sequenceIn, stream);
  CUDA_OK(cudaStreamSynchronize(stream));
  hPivot[pivotRow] = sequenceIn;
  return rc;
}

void Engine::getWeights(double *w)
{
  CUDA_OK(cudaMemcpy(w, d.weights, sizeof(double) * m, cudaMemcpyDeviceToHost));
}

void Engine::getDeviceVector(const char *name, double *out)
{
  std::string s(name);
  CUDA_OK(cudaStreamSynchronize(stream));
  if (s == "sol")
    CUDA_OK(cudaMemcpy(out, d.sol, sizeof(double) * nm, cudaMemcpyDeviceToHost));
  else if (s == "dj")
    CUDA_OK(cudaMemcpy(out, d.dj, sizeof(double) * nm, cudaMemcpyDeviceToHost));
  else if (s == "rho")
    CUDA_OK(cudaMemcpy(out, d.rho, sizeof(double) * m, cudaMemcpyDeviceToHost));
  else if (s == "alphaRow")
    CUDA_OK(cudaMemcpy(out, d.alphaRow, sizeof(double) * nm, cudaMemcpyDeviceToHost));
  else if (s == "pivotVariable") {
    std::vector<int> pv(m);
    CUDA_OK(cudaMemcpy(pv.data(), d.pivotVariable, sizeof(int) * m, cudaMemcpyDeviceToHost));
    for (int i = 0; i < m; i++)
      out[i] = pv[i];
  } else if (s == "status") {
    std::vector<unsigned char> st(nm);
    CUDA_OK(cudaMemcpy(st.data(), d.status, nm, cudaMemcpyDeviceToHost));
    for (int i = 0; i < nm; i++)
      out[i] = st[i];
  }
}

// ---------------------------------------------------------------------------------------
// primal simplex (ClpSimplexPrimal::primal, src/ClpSimplexPrimal.cpp; kernels in primal.cu)

void Engine::chgObjCoefficients(const double *obj)
{
  for (int j = 0; j < n; j++)
    hCost[j] = obj[j];
  if (!deviceReady)
    return; // the device copy is made from hCost at the next solve
  wCost = hCost;
  if (!columnScale.empty())
    for (int j = 0; j < n; j++)
      wCost[j] *= columnScale[j];
  costsPending = true;
}

void Engine::uploadPendingCosts()
{
  if (!costsPending)
    return;
  CUDA_OK(cudaMemcpy(d.costTrue, wCost.data(), sizeof(double) * nm, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(d.cost, wCost.data(), sizeof(double) * nm, cudaMemcpyHostToDevice));
  costsPending = false;
}

// Phase from the sum of infeasibilities of the basics, then that phase's costs and the duals through
// the current factors (eta file included).  Devex is reset on request and whenever the phase changes.
void Engine::primalCosts(bool resetDevex)
{
  launch_objective(d, dObj, stream);
  double obj2[2];
  CUDA_OK(cudaMemcpyAsync(obj2, dObj, sizeof(double) * 2, cudaMemcpyDeviceToHost, stream));
  CUDA_OK(cudaStreamSynchronize(stream));
  sumPrimalInfeasibilities = obj2[1];
  const int phase = obj2[1] > 0.0 ? 1 : 2;
  if (phase != primalPhase)
    resetDevex = true;
  primalPhase = phase;
  CUDA_OK(cudaMemcpyAsync(&d.st->primalPhase, &primalPhase, sizeof(int), cudaMemcpyHostToDevice, stream));
  launch_primal_costs(d, phase, stream);
  launch_compute_duals(d, dPi, dZ, stream, true);
  if (resetDevex)
    launch_primal_devex_reset(d, stream);
  kernelLaunches += 12;
  CUDA_OK(cudaStreamSynchronize(stream));
}

int Engine::primalRecompute(bool resetDevex)
{
  launch_compute_primals(d, dXn, dRhs, stream, true);
  kernelLaunches += 12;
  primalCosts(resetDevex);
  return 0;
}

// refactor -> computePrimals -> phase costs -> computeDuals -> Devex reset (no make_dual_feasible: that
// is the dual's and moves x)
int Engine::primalRefresh()
{
  if (refactor() != 0)
    return -1;
  currentCycle = std::min(cycleFor(d.k), d.tmax);
  return primalRecompute(true);
}

void Engine::buildPrimalGraph()
{
  if (primalGraph)
    return;
  cudaGraph_t graph = nullptr;
  bool ok = cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
  if (ok) {
    try {
      launch_primal_iteration(d, stream);
    } catch (const std::exception &) {
      ok = false;
    }
    if (cudaStreamEndCapture(stream, &graph) != cudaSuccess || graph == nullptr)
      ok = false;
  }
  if (ok) {
    size_t numNodes = 0;
    cudaGraphGetNodes(graph, nullptr, &numNodes);
    primalKernelsPerIteration = (int)numNodes;
    if (cudaGraphInstantiate(&primalGraph, graph, 0) != cudaSuccess) {
      primalGraph = nullptr;
      ok = false;
    }
  }
  if (graph)
    cudaGraphDestroy(graph);
  if (!ok) {
    cudaGetLastError(); // clear the sticky capture error
    fprintf(stderr, "clp_b200: CUDA graph capture of the primal iteration failed, launching kernels directly\n");
    useGraph = false;
  }
}

// ClpSimplex::primal (src/ClpSimplex.cpp:6145) -> ClpSimplexPrimal::primal: startup, loop, finish.
int Engine::primal()
{
  auto t0 = std::chrono::steady_clock::now();
  problemStatus = -1;
  numberIterations = 0;
  numberRefactorizations = 0;
  kernelLaunches = 0;
  phase = PhaseTimes();
  if (worldSize > 1) {
    fprintf(stderr, "clp_b200: primal() does not run on a column-sharded model\n");
    problemStatus = 4;
    return problemStatus;
  }
  if (m == 0 || n == 0)
    return trivialSolve();
  driftMeasured = false;
  lastSolveWasHot = hotStart && deviceReady && factorsValid;
  if (lastSolveWasHot) {
    // keep factors, eta file, x_B and status; new costs (and bounds) in force, duals recomputed
    uploadPendingCosts();
    boundsToWorking();
    CUDA_OK(cudaMemcpyAsync(d.lowerTrue, wLower.data(), sizeof(double) * nm, cudaMemcpyHostToDevice, stream));
    CUDA_OK(cudaMemcpyAsync(d.upperTrue, wUpper.data(), sizeof(double) * nm, cudaMemcpyHostToDevice, stream));
    CUDA_OK(cudaMemsetAsync(&d.st->stop, 0, sizeof(int), stream));
    CUDA_OK(cudaMemsetAsync(&d.st->pchuzcKey, 0, sizeof(unsigned long long), stream));
    launch_primal_bounds(d, stream);
  } else {
    setupDevice();
    uploadPendingCosts();
    resetStateForRun();
  }
  if (primalGraph) { // DeviceModel is captured by value
    cudaGraphExecDestroy(primalGraph);
    primalGraph = nullptr;
  }
  d.primalDantzig = primalColumnPivot == 1 ? 1 : 0;
  setAcceptablePivot(acceptablePivot);
  primalPhase = 0; // decided from the first sum of infeasibilities
  if ((lastSolveWasHot ? primalRecompute(true) : primalRefresh()) != 0) {
    problemStatus = 4;
    return problemStatus;
  }
  int consecutiveTrouble = 0, lastBadColumn = -1, confirmations = 0;
  while (problemStatus < 0) {
    if (numberIterations >= maximumIterations) {
      problemStatus = 3;
      break;
    }
    if (std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() > maximumSeconds) {
      problemStatus = 3;
      break;
    }
    fetchState();
    const int room = std::min(currentCycle, d.tmax) - hState->numEtas;
    if (room <= 0) {
      if (primalRefresh() != 0)
        problemStatus = 4;
      continue;
    }
    int count = std::min(std::min(batch, room), maximumIterations - numberIterations);
    count = std::min(count, d.recCap);
    const int before = hState->iterations;
    launch_primal_chuzc(d, stream);
    kernelLaunches += 2;
    if (useGraph)
      buildPrimalGraph(); // may clear useGraph
    if (useGraph) {
      for (int b = 0; b < count; b++)
        CUDA_OK(cudaGraphLaunch(primalGraph, stream));
      kernelLaunches += (long)count * primalKernelsPerIteration;
    } else {
      for (int b = 0; b < count; b++)
        launch_primal_iteration(d, stream);
    }
    fetchState();
    const int done = hState->iterations - before;
    numberIterations += done;
    if (logLevel > 1)
      fprintf(stderr, "clp_b200: primal it %d etas %d phase %d stop %d\n", numberIterations, hState->numEtas,
              primalPhase, hState->stop);
    const int stop = hState->stop;
    if (stop == STOP_NONE) {
      consecutiveTrouble = 0;
      continue;
    }
    CUDA_OK(cudaMemsetAsync(&d.st->stop, 0, sizeof(int), stream));
    const bool fresh = hState->numEtas == 0;
    switch (stop) {
    case STOP_ETAS_FULL:
      if (primalRefresh() != 0)
        problemStatus = 4;
      break;
    case STOP_PHASE_COSTS: // phase 1: the infeasibility set changed (ClpSimplexPrimal::pivotColumn updates)
      primalCosts(false);
      break;
    case STOP_INACCURATE: {
      if (++consecutiveTrouble > 50) {
        problemStatus = 4;
        break;
      }
      const int q = hState->seqIn;
      if (!fresh && primalRefresh() != 0) {
        problemStatus = 4;
        break;
      }
      if (fresh || q == lastBadColumn) {
        // the same column fails on fresh factors: leave it out until the next refactorization
        const unsigned char one = 1;
        CUDA_OK(cudaMemcpy(d.colFlagged + q, &one, 1, cudaMemcpyHostToDevice));
      }
      lastBadColumn = q;
      break;
    }
    case STOP_NO_COLUMN:
    case STOP_UNBOUNDED:
      // believed only on fresh factors with recomputed primals and duals, and without flagged columns
      if (!fresh || (lastBadColumn >= 0 && confirmations < 3)) {
        confirmations++;
        lastBadColumn = -1;
        if (primalRefresh() != 0)
          problemStatus = 4;
        break;
      }
      if (stop == STOP_NO_COLUMN)
        problemStatus = primalPhase == 2 ? 0 : 1;
      else
        problemStatus = primalPhase == 2 ? 2 : 4;
      break;
    default:
      problemStatus = 4;
      break;
    }
  }
  // leave the device state as a dual hot start expects it: true costs, unit dual weights
  CUDA_OK(cudaMemcpyAsync(d.cost, d.costTrue, sizeof(double) * nm, cudaMemcpyDeviceToDevice, stream));
  if (problemStatus != 0) // optimal: the duals already belong to the true costs
    launch_compute_duals(d, dPi, dZ, stream, true);
  std::vector<double> w(m, 1.0);
  CUDA_OK(cudaMemcpyAsync(d.weights, w.data(), sizeof(double) * m, cudaMemcpyHostToDevice, stream));
  downloadSolution();
  secondsInLoop = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  return problemStatus;
}

int Engine::primalColumnPivotTest(const double *dj, const unsigned char *stat, const double *weights, int mode)
{
  setupDevice();
  resetStateForRun();
  CUDA_OK(cudaMemcpy(d.dj, dj, sizeof(double) * nm, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(d.status, stat, nm, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(d.devex, weights, sizeof(double) * nm, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemset(d.colFlagged, 0, nm));
  DeviceModel dm = d;
  dm.primalDantzig = mode == 1 ? 1 : 0;
  launch_primal_chuzc(dm, stream);
  fetchState();
  return hState->stop != 0 ? -1 : hState->seqIn;
}

// The ratio test on explicit vectors: position p holds a basic slack (sequence n+p) with value xB[p] and
// bounds lowerB[p] / upperB[p]; the entering variable is column 0 with range enteringRange.
int Engine::primalRowTest(const double *alpha, const double *xB, const double *lowerB, const double *upperB,
                          int direction, double enteringRange, int phase, double *theta)
{
  setupDevice();
  resetStateForRun();
  std::vector<double> lo(wLower), up(wUpper), x(nm, 0.0);
  std::vector<int> pv(m);
  std::vector<unsigned char> ref(nm, 0);
  for (int p = 0; p < m; p++) {
    pv[p] = n + p;
    x[n + p] = xB[p];
    lo[n + p] = lowerB[p] < -1.0e29 ? -kInf : lowerB[p];
    up[n + p] = upperB[p] > 1.0e29 ? kInf : upperB[p];
  }
  lo[0] = 0.0;
  up[0] = enteringRange > 1.0e29 ? kInf : enteringRange;
  CUDA_OK(cudaMemcpy(d.lower, lo.data(), sizeof(double) * nm, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(d.upper, up.data(), sizeof(double) * nm, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(d.sol, x.data(), sizeof(double) * nm, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(d.pivotVariable, pv.data(), sizeof(int) * m, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(d.devexRef, ref.data(), nm, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(d.rhs3, alpha, sizeof(double) * m, cudaMemcpyHostToDevice));
  IterState st;
  memset(&st, 0, sizeof(st));
  st.seqIn = 0;
  st.primalDir = direction < 0 ? -1 : 1;
  st.primalPhase = phase == 1 ? 1 : 2;
  st.acceptablePivot = acceptablePivot;
  st.ratioBits = 0x7FF0000000000000ull;
  CUDA_OK(cudaMemcpy(d.st, &st, sizeof(st), cudaMemcpyHostToDevice));
  launch_primal_ratio(d, stream);
  fetchState();
  if (hState->stop == STOP_UNBOUNDED) {
    *theta = kInf;
    return -1;
  }
  *theta = std::fabs(hState->thetaPrimal);
  return hState->primalFlip ? -2 : hState->pivotRow;
}

} // namespace clpb
