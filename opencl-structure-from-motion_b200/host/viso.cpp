#include "viso.h"

#include <cmath>
#include <cstdlib>
#include <numeric>

VisualOdometry::VisualOdometry(parameters param) : sample_generator(71), param(param) {
  J = 0; p_observe = 0; p_predict = 0;
  matcher = new Matcher(param.match);
  owns_matcher = true;
  Tr_delta = Matrix::eye(4);
  Tr_valid = false;
  srand(0);                  // as the reference does (viso.cpp:35)
  matcher->seedShuffle(0);   // ... and the matcher's own copy of that generator, which bucketFeatures draws from
}

VisualOdometry::~VisualOdometry() { if (owns_matcher) delete matcher; }

void VisualOdometry::adoptMatcher(Matcher* external) {
  if (owns_matcher) delete matcher;
  matcher = external;
  owns_matcher = false;
  matcher->seedShuffle(0);     // same state the own matcher had (viso.cpp:35)
}

bool VisualOdometry::updateMotion() { return setMotion(estimateMotion(p_matched)); }

bool VisualOdometry::setMotion(const std::vector<double>& tr) {
  if (tr.size() != 6) return false;
  Tr_delta = transformationVectorToMatrix(tr);
  Tr_valid = true;
  return true;
}

// rotation Rx(rx) * Ry(ry) * Rz(rz) with translation (viso.cpp:59-84)
Matrix VisualOdometry::transformationVectorToMatrix(std::vector<double> tr) {
  Matrix R = Matrix::rotMatX(tr[0]) * Matrix::rotMatY(tr[1]) * Matrix::rotMatZ(tr[2]);
  Matrix Tr = Matrix::eye(4);
  Tr.setMat(R, 0, 0);
  for (int i = 0; i < 3; i++) Tr.val[i][3] = tr[3 + i];
  return Tr;
}

std::vector<int> VisualOdometry::getRandomSample(unsigned N, unsigned num) {
  // Partial Fisher-Yates over 0..N-1 with a fresh uniform_int_distribution(i, N-1) per draw, exactly the calls of
  // viso.cpp:86-102.  The reference builds the N-element index set anew for every sample (2000 times per frame); here
  // the identity permutation is kept and the few swaps of a sample are undone afterwards: same numbers, no allocation.
  if (sample_pool.size() != N) {
    sample_pool.resize(N);
    std::iota(sample_pool.begin(), sample_pool.end(), 0);
  }
  unsigned picked[16];
  std::vector<int> out(num);
  const unsigned cnt = num < 16 ? num : 16;
  if (num > 16) {                       // not used by the library (8-point and 3-point samples); keep the plain form
    std::vector<int> pool(N);
    std::iota(pool.begin(), pool.end(), 0);
    for (unsigned i = 0; i < num; i++) {
      std::uniform_int_distribution<unsigned> pick(i, N - 1);
      std::swap(pool.at(i), pool.at(pick(sample_generator)));
    }
    pool.resize(num);
    return pool;
  }
  for (unsigned i = 0; i < cnt; i++) {
    std::uniform_int_distribution<unsigned> pick(i, N - 1);
    picked[i] = pick(sample_generator);
    std::swap(sample_pool.at(i), sample_pool.at(picked[i]));
  }
  for (unsigned i = 0; i < cnt; i++) out[i] = sample_pool[i];
  for (unsigned i = cnt; i-- > 0;) std::swap(sample_pool[i], sample_pool[picked[i]]);
  return out;
}
