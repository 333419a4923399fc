// A C++ translation unit compiled against include/clp_b200.h only: how a Clp maintainer binds
// Clp_primal / Clp_chgObjCoefficients.  Host-only calls always run; with a CUDA device (argv[1] == "gpu")
// it also solves a small LP with Clpb_primal, changes the costs and re-solves hot.
#include "clp_b200.h"

#include <cmath>
#include <cstdio>
#include <cstring>
#include <vector>

#define CHECK(cond)                                                                        \
  do {                                                                                     \
    if (!(cond)) {                                                                         \
      std::fprintf(stderr, "primal_consumer.cpp:%d: check failed: %s\n", __LINE__, #cond); \
      return 1;                                                                            \
    }                                                                                      \
  } while (0)

int main(int argc, char **argv)
{
  const bool gpu = argc > 1 && !std::strcmp(argv[1], "gpu");
  // max 3 x0 + 2 x1 (as min of the negation) s.t. x0 + x1 <= 4, x0 + 3 x1 <= 6, 0 <= x0 <= 3, x1 >= 0
  const int start[3] = {0, 2, 4};
  const int index[4] = {0, 1, 0, 1};
  const double value[4] = {1.0, 1.0, 1.0, 3.0};
  const double collb[2] = {0, 0}, colub[2] = {3, 1e30};
  const double obj[2] = {-3.0, -2.0};
  const double rowlb[2] = {-1e30, -1e30}, rowub[2] = {4.0, 6.0};

  Clpb_Simplex *model = Clpb_newModel();
  CHECK(model != nullptr);
  CHECK(Clpb_loadProblem(model, 2, 2, start, index, value, collb, colub, obj, rowlb, rowub) == 0);
  CHECK(Clpb_setParameter(model, "primalColumnPivot", 1) == 0);
  CHECK(Clpb_setParameter(model, "primalColumnPivot", 0) == 0);
  // host only: the new objective is what getProblem returns
  const double obj2[2] = {-1.0, -2.0};
  Clpb_chgObjCoefficients(model, obj2);
  std::vector<double> ob(2);
  Clpb_getProblem(model, nullptr, nullptr, nullptr, nullptr, nullptr, ob.data(), nullptr, nullptr);
  CHECK(ob[0] == -1.0 && ob[1] == -2.0);
  Clpb_chgObjCoefficients(model, obj);

  if (!gpu) {
    CHECK(Clpb_primal(model, 0) == CLPB_NO_DEVICE);
    const double dj[4] = {-1, 0, 0, 0}, w[4] = {1, 1, 1, 1};
    const unsigned char st[4] = {3, 3, 1, 1};
    CHECK(Clpb_primalColumnPivot(model, dj, st, w, 0) == CLPB_NO_DEVICE);
    const double a[2] = {1, 1}, x[2] = {4, 6}, lo[2] = {-1e30, -1e30}, up[2] = {1e30, 1e30};
    double theta = 0.0;
    CHECK(Clpb_primalRow(model, a, x, lo, up, 1, 3.0, 2, &theta) == CLPB_NO_DEVICE);
    Clpb_deleteModel(model);
    std::printf("primal consumer ok (host only)\n");
    return 0;
  }
  CHECK(Clpb_primal(model, 0) == 0);
  // optimum x = (3, 1): -3*3 - 2*1 = -11
  CHECK(std::fabs(Clpb_objectiveValue(model) + 11.0) < 1e-9);
  // new costs: min -x0 - 2 x1 -> x = (3, 1) gives -5, x = (0, 2) gives -4, x = (1.5, 1.5) gives -4.5
  Clpb_chgObjCoefficients(model, obj2);
  CHECK(Clpb_setParameter(model, "hotStart", 1) == 0);
  CHECK(Clpb_primal(model, 0) == 0);
  CHECK(Clpb_lastSolveWasHot(model) == 1);
  CHECK(std::fabs(Clpb_objectiveValue(model) + 5.0) < 1e-9);
  Clpb_deleteModel(model);
  std::printf("primal consumer ok (gpu)\n");
  return 0;
}
