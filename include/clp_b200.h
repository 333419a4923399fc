/* clp_b200.h -- C ABI of the B200-native revised dual simplex engine.
 *
 * Drop-in boundary for ONE path of coin-or/Clp: ClpModel::readMps/loadProblem ->
 * ClpSimplex::dual().  Every entry point names the reference interface it replaces
 * (paths relative to the coin-or/Clp source tree).  Conventions follow
 * src/Clp_C_Interface.h: one opaque model pointer, int status returns, caller-owned HOST
 * buffers (plain pointers and sizes), no exceptions across the boundary, single caller thread.
 * Sequence numbering is ClpSimplex's: 0..n-1 columns, n..n+m-1 rows; status bytes are
 * ClpSimplex::Status (src/ClpSimplex.hpp:119-126).
 *
 * The library has NO CPU fallback: every solve/plug-in call needs a CUDA device and returns
 * CLPB_NO_DEVICE (-100) otherwise.
 */
#ifndef CLP_B200_H
#define CLP_B200_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct Clpb_Simplex Clpb_Simplex;

#define CLPB_NO_DEVICE (-100)

/* ---------------- model level: replaces src/Clp_C_Interface.h ---------------- */
/* Clp_newModel :77 / Clp_deleteModel :79 */
Clpb_Simplex *Clpb_newModel(void);
void Clpb_deleteModel(Clpb_Simplex *model);
/* Clp_loadProblem :101 (column-major matrix without gaps; NULL rim arrays take Clp's defaults) */
int Clpb_loadProblem(Clpb_Simplex *model, int numcols, int numrows, const int *start,
                     const int *index, const double *value, const double *collb,
                     const double *colub, const double *obj, const double *rowlb,
                     const double *rowub);
/* Clp_readMps :116 (ClpModel::readMps src/ClpModel.cpp:2884) */
int Clpb_readMps(Clpb_Simplex *model, const char *filename, int keepNames, int ignoreErrors);
/* ClpPresolve::presolvedModel / postsolve (src/ClpPresolve.hpp:40,61) restricted to the elementary
   actions (fixed columns, singleton rows, empty columns, empty rows, dual fixing of dominated columns,
   forcing rows; src/ClpPresolve.cpp:966,1141,1448,1449,1158,1182).  Clpb_presolvedModel returns a NEW model (delete it with Clpb_deleteModel) holding the
   reduced problem, or NULL with *status = 1 (primal infeasible) / 2 (dual infeasible); the original
   model keeps the postsolve information.  After solving the reduced model, Clpb_postsolve writes
   the solution of the original problem (primal, dual, status, objective) into the original model.
   Clpb_setSolution hands a solution of a model in from outside (x[n], rowPrice[m], status[n+m]).
   Host only. */
Clpb_Simplex *Clpb_presolvedModel(Clpb_Simplex *model, int *status);
int Clpb_postsolve(Clpb_Simplex *model, Clpb_Simplex *presolved);
void Clpb_setSolution(Clpb_Simplex *model, const double *x, const double *rowPrice,
                      const unsigned char *status, int problemStatus);
/* Clp_writeMps :123 (ClpModel::writeMps src/ClpModel.cpp:3986): the model as loaded, default names
   R%7.7d / C%7.7d, 17 significant digits; formatType / numberAcross / objSense are accepted for
   signature compatibility.  0 ok, -1 cannot open.  Host only. */
int Clpb_writeMps(Clpb_Simplex *model, const char *filename, int formatType, int numberAcross,
                  double objSense);
/* Clp_numberRows :174, Clp_numberColumns :176, Clp_getNumElements :246 */
int Clpb_numberRows(Clpb_Simplex *model);
int Clpb_numberColumns(Clpb_Simplex *model);
long long Clpb_getNumElements(Clpb_Simplex *model);
/* problem data as loaded (for callers that used readMps): Clp_getRowLower ... Clp_getColUpper :459-475 */
void Clpb_getProblem(Clpb_Simplex *model, int *start, int *index, double *value, double *collb,
                     double *colub, double *obj, double *rowlb, double *rowub);
/* Clp_setPrimalTolerance :179, Clp_setDualTolerance :182, Clp_setDualBound :382,
   Clp_setMaximumIterations :199, Clp_setMaximumSeconds :202, Clp_setLogLevel :314,
   ClpFactorization::maximumPivots (src/ClpFactorization.hpp:149).  Keys: "primalTolerance",
   "dualTolerance", "dualBound", "maximumIterations", "maximumSeconds", "logLevel", "primalColumnPivot",
   "factorizationFrequency", "scaling", "perturbation" (Clp_setPerturbation :395: 50 on,
   100 automatic, 102 off = default here; ClpSimplexDual::perturb src/ClpSimplexDual.cpp:6533), "batch" (iterations enqueued per host sync), "timing" (0/1: per-phase
   CUDA events, no graph replay), "useGraph" (0/1), "warmupIterations", "objectiveOffset". */
int Clpb_setParameter(Clpb_Simplex *model, const char *key, double value);
/* Clp_scaling :354 (ClpModel::scaling(int mode), src/ClpModel.hpp): 0 off (default here; the
   benchmark configuration is unscaled), 1 equilibrium, 2 geometric, 3 automatic (Clp's default),
   4 automatic-dynamic (treated as 3).  The same value can be set with the key "scaling".
   Clpb_scaleFactors runs ClpPackedMatrix::scale (src/ClpPackedMatrix.cpp:4120) on the host and
   copies rowScale[m] / columnScale[n] out (all 1 and return value 1 when the matrix is not
   worth scaling, :4262); dual() applies them to the matrix and the rim and returns the solution
   in the caller's units. */
void Clpb_scaling(Clpb_Simplex *model, int mode);
int Clpb_scaleFactors(Clpb_Simplex *model, double *rowScale, double *columnScale);
/* Host-only preview of ClpSimplexDual::perturb (src/ClpSimplexDual.cpp:6533) for the current
   "perturbation" setting and status: cost[n] = the (scaled) working objective after perturbation.
   Returns 0 if costs were perturbed, 1 if the rule decided not to (copy of the objective). */
int Clpb_perturbedCosts(Clpb_Simplex *model, double *cost);
/* Clp_copyinStatus :280 : status[n+m], columns first */
void Clpb_copyinStatus(Clpb_Simplex *model, const unsigned char *statusArray);
/* ClpSimplex::writeBasis / readBasis (src/ClpSimplex.cpp:6569 / :6577 -> ClpSimplexOther.cpp:1018 /
   :1136): MPS basis file (XU/XL/UL/LL/BS records) in the reference's no-names form C%7.7d / R%7.7d;
   writeValues / formatType are accepted for signature compatibility, values are not written.
   readBasis returns 0, -1 (cannot open) or the number of records it could not interpret; the basis
   becomes the starting basis of the next Clpb_dual (like Clpb_copyinStatus).  Host only. */
int Clpb_writeBasis(Clpb_Simplex *model, const char *filename, int writeValues, int formatType);
int Clpb_readBasis(Clpb_Simplex *model, const char *filename);
/* Clp_chgRowLower :150, Clp_chgRowUpper :152, Clp_chgColumnLower :154, Clp_chgColumnUpper :156: replace a
   whole bound vector of the loaded model.  With the key "hotStart" = 1 (Clpb_setParameter) the next
   Clpb_dual on the same model is the reference's hot start (ClpSimplexDual::fastDual
   src/ClpSimplexDual.cpp:7241, the inner solve of strongBranching :6965): factors, eta file, weights,
   duals and status stay on the device, only the bounds are re-imposed and x_B recomputed -- no upload,
   no refactorization at the start.  Clpb_lastSolveWasHot tells whether the last Clpb_dual took that path. */
void Clpb_chgColumnLower(Clpb_Simplex *model, const double *columnLower);
void Clpb_chgColumnUpper(Clpb_Simplex *model, const double *columnUpper);
void Clpb_chgRowLower(Clpb_Simplex *model, const double *rowLower);
void Clpb_chgRowUpper(Clpb_Simplex *model, const double *rowUpper);
int Clpb_lastSolveWasHot(Clpb_Simplex *model);
/* ClpFactorization::maximumPivots (src/ClpFactorization.hpp:149) as the default policy sets it for a basis
   whose structural part ("nucleus") has nucleusSize columns: twice ClpSimplex::defaultFactorizationFrequency
   (src/ClpSimplex.cpp:11401), stretched when the modelled cost of the dense refactorization outweighs the
   iterations of a cycle; "factorizationFrequency" > 0 overrides it.  Host only. */
int Clpb_refactorizationInterval(Clpb_Simplex *model, int nucleusSize);
/* Clp_dual :346 (ClpSimplex::dual src/ClpSimplex.cpp:5631).  Returns Clp_status :212:
   0 optimal, 1 primal infeasible, 2 dual infeasible, 3 stopped on iterations/time,
   4 stopped due to errors. */
int Clpb_dual(Clpb_Simplex *model, int ifValuesPass);
/* Clp_primal :348 (ClpSimplex::primal src/ClpSimplex.cpp:6145).  Same return codes as Clpb_dual.
   Phase 1 minimises the sum of infeasibilities, phase 2 the loaded costs; pricing by the key
   "primalColumnPivot" (ClpSimplex::setPrimalColumnPivotAlgorithm): 0 exact Devex
   (ClpPrimalColumnSteepest mode 0, the default), 1 Dantzig (ClpPrimalColumnDantzig).  The values pass
   is not built: ifValuesPass != 0 is treated as 0.  "perturbation" is ignored.  A model with
   sharding initialised (Clpb_initSharding, worldSize > 1) is refused with 4.  With "hotStart" = 1 a
   Clpb_primal that follows a solve of the same model keeps the factors, eta file, x_B and status on
   the device, recomputes the duals for the costs now loaded and iterates (Clpb_lastSolveWasHot says
   so): the re-solve after Clpb_chgObjCoefficients. */
int Clpb_primal(Clpb_Simplex *model, int ifValuesPass);
/* Clp_chgObjCoefficients :158: obj[n] replaces the loaded objective (Clpb_getProblem returns it; the
   device copy is updated at the next solve).  A hot Clpb_dual is not taken after a cost change. */
void Clpb_chgObjCoefficients(Clpb_Simplex *model, const double *obj);
int Clpb_status(Clpb_Simplex *model);
/* Clp_objectiveValue :256, Clp_numberIterations :195 */
double Clpb_objectiveValue(Clpb_Simplex *model);
int Clpb_numberIterations(Clpb_Simplex *model);
int Clpb_numberRefactorizations(Clpb_Simplex *model);
/* Clp_primalColumnSolution :230, Clp_primalRowSolution :228, Clp_dualColumnSolution :234,
   Clp_dualRowSolution :232, Clp_statusArray :278 -- copied into caller buffers */
void Clpb_primalColumnSolution(Clpb_Simplex *model, double *x /* n */);
void Clpb_primalRowSolution(Clpb_Simplex *model, double *rowActivity /* m */);
void Clpb_dualColumnSolution(Clpb_Simplex *model, double *reducedCost /* n */);
void Clpb_dualRowSolution(Clpb_Simplex *model, double *rowPrice /* m */);
void Clpb_statusArray(Clpb_Simplex *model, unsigned char *status /* n+m */);
/* measurement: seconds in the iteration loop, kernels launched, per-phase device ms
   (order: chuzr, btran, price, chuzc, dualUpdate, ftran, update, refactor, samples, then the
   single kernels priceKernel, ftranGemv, btranGemv, then the algorithmic bytes summed over the
   timed FTRAN / BTRAN GEMV launches; 14 doubles) */
double Clpb_secondsInLoop(Clpb_Simplex *model);
long long Clpb_kernelLaunches(Clpb_Simplex *model);
void Clpb_phaseTimes(Clpb_Simplex *model, double *out14);
int Clpb_nucleusSize(Clpb_Simplex *model);
/* CUDA-event time (on the engine's stream) and iteration count of the window that starts after
   "warmupIterations" iterations and ends when Clpb_dual returns (refactorizations included) */
void Clpb_timedWindow(Clpb_Simplex *model, double *milliseconds, int *iterations);

/* column-sharded pricing across GPUs (one process per GPU).  ncclUniqueId (128 bytes) is
   created by rank 0 with Clpb_ncclUniqueId and shipped to the other ranks by the caller
   (torch.distributed broadcast); then every rank calls Clpb_initSharding. */
int Clpb_ncclUniqueId(unsigned char *id128);
int Clpb_initSharding(Clpb_Simplex *model, int rank, int worldSize, const unsigned char *id128);

/* ---------------- plug-in level: the three interfaces whileIterating calls ------------- */
/* ClpFactorization::factorize (src/ClpFactorization.hpp:54, .cpp:1649).  basicSequence[m] in,
   pivotVariable[m] out: pivotVariable[i] pivots on row i.  0 ok, -1 singular. */
int Clpb_factorize(Clpb_Simplex *model, const int *basicSequence, int *pivotVariable);
/* ClpFactorization::updateColumn (hpp:117, FTRAN) / updateColumnTranspose (hpp:135, BTRAN);
   region[m] dense, in place */
int Clpb_updateColumn(Clpb_Simplex *model, double *region);
int Clpb_updateColumnTranspose(Clpb_Simplex *model, double *region);
/* ClpFactorization::replaceColumn (hpp:89, return codes hpp:82-88): 0 ok, 1 probably ok (pivot agrees
   with pivotCheck only to 1e-8; the update is made), 2 singular / inaccurate (nothing changed), 3 no room
   in the update buffers, 5 maximum pivots (factorizationFrequency) reached.  Clpb_replaceColumn is the
   unchecked form (codes 0 / 2 / 3 / 5); the checked form restates CoinAbcTypeFactorization::checkPivot
   (src/CoinAbcBaseFactorization4.cpp:94-131) with pivotCheck = the pivot taken from the BTRAN row. */
int Clpb_replaceColumn(Clpb_Simplex *model, int sequenceIn, int pivotRow);
int Clpb_replaceColumnChecked(Clpb_Simplex *model, int sequenceIn, int pivotRow, double pivotCheck,
                              double acceptablePivot);
/* ClpFactorization::updateColumnFT (hpp:113) / updateTwoColumnsFT (hpp:125): FTRAN in place that also
   keeps what replaceColumn needs (in product form the spike is the FTRAN'd column itself).  Returns the
   number of nonzeros, negative when there is no room for another update (hpp:120-123). */
int Clpb_updateColumnFT(Clpb_Simplex *model, double *region);
int Clpb_updateTwoColumnsFT(Clpb_Simplex *model, double *regionFT, double *regionOther);
/* Packed forms (CoinIndexedVector packedMode: number / indices / elements, SURVEY 8b): in place, arrays
   of capacity m (n for the z of transposeTimes), entries <= zeroTolerance dropped as
   ClpPackedMatrix::transposeTimes does (src/ClpPackedMatrix.cpp:931-932). */
int Clpb_updateColumnPacked(Clpb_Simplex *model, int *number, int *indices, double *elements);
int Clpb_updateColumnTransposePacked(Clpb_Simplex *model, int *number, int *indices, double *elements);
int Clpb_transposeTimesPacked(Clpb_Simplex *model, double scalar, int numberPi, const int *indexPi,
                              const double *elementPi, int *numberZ, int *indexZ, double *elementZ);
/* ClpMatrixBase::transposeTimes (src/ClpMatrixBase.hpp:287) z[n] = scalar*A^T pi ;
   ClpMatrixBase::times (hpp:275) y[m] = scalar*A x */
int Clpb_transposeTimes(Clpb_Simplex *model, double scalar, const double *pi, double *z);
int Clpb_times(Clpb_Simplex *model, double scalar, const double *x, double *y);
/* ClpSimplexDual::dualColumn (src/ClpSimplexDual.cpp:4192) on an explicit tableau row:
   alphaRow[n+m], dj[n+m], status[n+m]; direction +1 leaving to upper / -1 to lower.
   Returns sequenceIn or -1; *theta = dual step. */
int Clpb_dualColumn(Clpb_Simplex *model, const double *alphaRow, const double *dj,
                    const unsigned char *status, int direction, double infeasibility,
                    double *theta);
/* The same test run by the cooperative row kernel of the fused iteration (rowpass.cu), which also
   performs the dual update and the bound flips that follow it on the device copy of dj / status. */
int Clpb_dualColumnRowPass(Clpb_Simplex *model, const double *alphaRow, const double *dj,
                           const unsigned char *status, int direction, double infeasibility,
                           double *theta);
/* ClpPrimalColumnPivot::pivotColumn (src/ClpPrimalColumnPivot.hpp) on explicit vectors dj[n+m],
   status[n+m], weights[n+m]; mode 0 Devex (score dj^2/weight), 1 Dantzig (dj^2).  Candidates: at lower
   with dj < -dualTolerance, at upper with dj > dualTolerance, free / superbasic with |dj| > dualTolerance.
   Returns the entering sequence or -1.  Scores that agree in their upper 44 bits: the smaller sequence. */
int Clpb_primalColumnPivot(Clpb_Simplex *model, const double *dj, const unsigned char *status,
                           const double *weights, int mode);
/* ClpSimplexPrimal::primalRow (src/ClpSimplexPrimal.cpp:1877), Harris two-pass ratio test on explicit
   vectors: alpha[m] = B^-1 a_q, basic values xB[m] with bounds lowerB[m] / upperB[m]; the entering
   variable moves up (direction +1) or down (-1) and has range enteringRange (>= 1e30: none).  phase 1:
   infeasible basics block only at their far bound.  Returns the pivot row, -1 no block (unbounded ray), or
   -2 the entering variable reaches its other bound first; *theta = the step (>= 0).  Pivots below
   "acceptablePivot" are ignored; among the rows within the relaxed step the largest |alpha| wins
   (ties: the smaller row). */
int Clpb_primalRow(Clpb_Simplex *model, const double *alpha, const double *xB, const double *lowerB,
                   const double *upperB, int direction, double enteringRange, int phase, double *theta);
/* The dense kernel of the refactorization on its own (CoinAbcDgetrf + inverse,
   src/AbcSimplexParallel.cpp:2491): a[k*k] column-major in, x = a^-1 column-major out.
   Returns 0, or 1 + the index of the first column without an acceptable pivot. */
int Clpb_denseInvert(int k, const double *a, double *x);
/* ---- ClpDualRowPivot (src/ClpDualRowPivot.hpp:23-130) and the calls whileIterating makes around it,
   ONE iteration at a time on the device-resident state (after Clpb_startup).  The fused kernels decide
   where the cuts fall:
     Clpb_pivotRow                       ClpDualRowPivot::pivotRow :30  -> pivot row, -1 none (primal
                                         feasible), -2 update buffers full (factorize first); also the
                                         leaving sequence, its direction (+1 to upper / -1 to lower) and
                                         primal infeasibility
     Clpb_updateColumnTransposeAndPrice  ClpFactorization::updateColumnTranspose(e_r) hpp:135 +
                                         ClpMatrixBase::transposeTimes hpp:308; rho[m] / alphaRow[n]
                                         copied out when not NULL; returns nnz(rho)
     Clpb_dualColumnDevice               ClpSimplexDual::dualColumn + updateDualsInDual + flipBounds
                                         (src/ClpSimplexDual.cpp:4192, :2430, :6345 -- one kernel);
                                         returns sequenceIn or -1, *theta the dual step, *alpha the pivot
                                         element from the row
     Clpb_updateWeights                  ClpDualRowPivot::updateWeights :34 (performs the FT-FTRAN pair
                                         like the reference's, returns alpha from the column); *returnCode
                                         0 ok, 1 pivot disagrees with the row (refactorize), 2 no usable pivot.
                                         The DSE recurrence is applied by the next call, so a rejected
                                         pivot leaves the weights untouched
     Clpb_unrollWeights                  ClpDualRowPivot::unrollWeights :67 -- nothing to undo (see above)
     Clpb_updatePrimalSolution           ClpDualRowPivot::updatePrimalSolution :47 + the weight recurrence +
                                         ClpFactorization::replaceColumn + ClpSimplex::housekeeping (one
                                         kernel); *changeInObjective = dual objective gain; returns the
                                         number of updates since the last factorization
     Clpb_saveWeights                    ClpDualRowPivot::saveWeights :63, modes 1..7 of
                                         ClpDualRowSteepest::saveWeights (src/ClpDualRowSteepest.cpp:773) */
int Clpb_pivotRow(Clpb_Simplex *model, int *sequenceOut, int *direction, double *infeasibility);
int Clpb_updateColumnTransposeAndPrice(Clpb_Simplex *model, double *rho, double *alphaRow);
int Clpb_dualColumnDevice(Clpb_Simplex *model, double *theta, double *alpha);
double Clpb_updateWeights(Clpb_Simplex *model, int *returnCode);
int Clpb_unrollWeights(Clpb_Simplex *model);
int Clpb_updatePrimalSolution(Clpb_Simplex *model, double *changeInObjective);
int Clpb_saveWeights(Clpb_Simplex *model, int mode);
/* run the startup of dual() (basis from status, factorize, computePrimals/Duals) and then
   'count' iterations; DSE weights by pivot row (ClpDualRowSteepest::weights_) */
int Clpb_startup(Clpb_Simplex *model);
int Clpb_iterate(Clpb_Simplex *model, int count);
void Clpb_getWeights(Clpb_Simplex *model, double *weights /* m */);
/* debug reads of device vectors: "sol","dj" (n+m), "rho" (m), "alphaRow" (n+m),
   "pivotVariable" (m, as doubles), "status" (n+m, as doubles) */
void Clpb_getDeviceVector(Clpb_Simplex *model, const char *name, double *out);

#ifdef __cplusplus
}
#endif
#endif
