// oracle_malio.cpp — CPU ORACLE for the MA-LIO measurement hot path.  TEST INFRASTRUCTURE ONLY.
//
// A plain C++ restatement (no Eigen / PCL / ROS / Boost: none exist in this image) of the reference's
// algorithm, function by function, each citing the reference file:line it follows (paths relative to
// /root/reference/MA_LIO).  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
// --impl reference legs may load it; the product (ma-lio_b200/) never does.
//
// PARITY STATUS: the reference ships no tests, golden vectors or fixtures (SURVEY.md §4, §8c), and its
// B/P/U/A code cannot be compiled here (Eigen/PCL/ROS/Boost absent) => "parity unpinned" for those parts:
// this restatement is cross-checked against (a) the real reference ikd_Tree.cpp compiled in place
// (oracle/_ref, K/N parts: pinned by the reference itself), (b) an independent numpy/scipy restatement
// (oracle/np_oracle.py), (c) brute force / finite differences.  Third-party arithmetic restated from
// its published algorithm: Eigen 3.3.7 (unpinned in the repo; Ubuntu 20.04's version per the stale
// build dir) ColPivHouseholderQR::solve, PartialPivLU inverse, JacobiSVD singular values,
// Quaternion::_transformVector / toRotationMatrix.
//
// Build: g++ -O2 -ffp-contract=off -fopenmp (see oracle/Makefile).  -ffp-contract=off: the reference is
// built for baseline x86-64 (CMakeLists.txt:8, no -march), i.e. without FMA.
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <vector>
#include <algorithm>
#include <omp.h>

#include "malio_b200.h"

namespace {

// ------------------------------------------------------------------ small fixed-size algebra
struct Q4 { double w, x, y, z; };

inline Q4 q_from(const double q[4]) { return Q4{q[0], q[1], q[2], q[3]}; }
inline Q4 q_conj(const Q4& q) { return Q4{q.w, -q.x, -q.y, -q.z}; }
// Eigen::Quaternion product (Eigen/src/Geometry/Quaternion.h, quat_product)
inline Q4 q_mul(const Q4& a, const Q4& b) {
  return Q4{a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z,
            a.w * b.x + a.x * b.w + a.y * b.z - a.z * b.y,
            a.w * b.y + a.y * b.w + a.z * b.x - a.x * b.z,
            a.w * b.z + a.z * b.w + a.x * b.y - a.y * b.x};
}
inline void cross3(const double a[3], const double b[3], double o[3]) {
  o[0] = a[1] * b[2] - a[2] * b[1];
  o[1] = a[2] * b[0] - a[0] * b[2];
  o[2] = a[0] * b[1] - a[1] * b[0];
}
// Eigen QuaternionBase::_transformVector: v + w*uv + qv x uv, uv = 2 qv x v
inline void q_rot(const Q4& q, const double v[3], double o[3]) {
  const double qv[3] = {q.x, q.y, q.z};
  double uv[3], c2[3];
  cross3(qv, v, uv);
  uv[0] += uv[0]; uv[1] += uv[1]; uv[2] += uv[2];
  cross3(qv, uv, c2);
  o[0] = v[0] + q.w * uv[0] + c2[0];
  o[1] = v[1] + q.w * uv[1] + c2[1];
  o[2] = v[2] + q.w * uv[2] + c2[2];
}
// Eigen QuaternionBase::toRotationMatrix, row-major 3x3
inline void q_to_R(const Q4& q, double R[9]) {
  const double tx = 2 * q.x, ty = 2 * q.y, tz = 2 * q.z;
  const double twx = tx * q.w, twy = ty * q.w, twz = tz * q.w;
  const double txx = tx * q.x, txy = ty * q.x, txz = tz * q.x;
  const double tyy = ty * q.y, tyz = tz * q.y, tzz = tz * q.z;
  R[0] = 1 - (tyy + tzz); R[1] = txy - twz;       R[2] = txz + twy;
  R[3] = txy + twz;       R[4] = 1 - (txx + tzz); R[5] = tyz - twx;
  R[6] = txz - twy;       R[7] = tyz + twx;       R[8] = 1 - (txx + tyy);
}
inline void skew(const double v[3], double M[9]) {   // SKEW_SYM_MATRX, include/so3_math.h:7
  M[0] = 0; M[1] = -v[2]; M[2] = v[1];
  M[3] = v[2]; M[4] = 0; M[5] = -v[0];
  M[6] = -v[1]; M[7] = v[0]; M[8] = 0;
}
inline void m3v(const double M[9], const double v[3], double o[3]) {
  for (int i = 0; i < 3; ++i) o[i] = M[3 * i] * v[0] + M[3 * i + 1] * v[1] + M[3 * i + 2] * v[2];
}
inline void m3m(const double A[9], const double B[9], double C[9]) {
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) C[3 * i + j] = A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j] + A[3 * i + 2] * B[6 + j];
}

// ------------------------------------------------------------------ K: ikd-Tree search, restated
// PointType_CMP (ikd_Tree.h:93-109)
struct HeapItem {
  float dist = INFINITY;
  float x = 0.f;
  int32_t idx = -1;
  bool operator<(const HeapItem& a) const {
    if (std::fabs(dist - a.dist) < 1e-10) return x < a.x;
    return dist < a.dist;
  }
};
// MANUAL_HEAP (ikd_Tree.h:111-201): max-heap, capacity 2k, same MoveDown / FloatUp
struct ManualHeap {
  HeapItem heap[2 * MALIO_K + 2];
  int heap_size = 0, cap = 2 * MALIO_K;
  void pop() {
    if (heap_size == 0) return;
    heap[0] = heap[heap_size - 1];
    heap_size--;
    MoveDown(0);
  }
  HeapItem top() const { return heap[0]; }
  void push(const HeapItem& p) {
    if (heap_size >= cap) return;
    heap[heap_size] = p;
    FloatUp(heap_size);
    heap_size++;
  }
  int size() const { return heap_size; }
  void MoveDown(int heap_index) {
    int l = heap_index * 2 + 1;
    HeapItem tmp = heap[heap_index];
    while (l < heap_size) {
      if (l + 1 < heap_size && heap[l] < heap[l + 1]) l++;
      if (tmp < heap[l]) {
        heap[heap_index] = heap[l];
        heap_index = l;
        l = heap_index * 2 + 1;
      } else
        break;
    }
    heap[heap_index] = tmp;
  }
  void FloatUp(int heap_index) {
    int ancestor = (heap_index - 1) / 2;
    HeapItem tmp = heap[heap_index];
    while (heap_index > 0) {
      if (heap[ancestor] < tmp) {
        heap[heap_index] = heap[ancestor];
        heap_index = ancestor;
        ancestor = (heap_index - 1) / 2;
      } else
        break;
    }
    heap[heap_index] = tmp;
  }
};

// calc_dist (ikd_Tree.cpp:1694-1699): float, (dx*dx + dy*dy) + dz*dz
inline float calc_dist(const float a[3], const malio_map_node& n) {
  float dist = (a[0] - n.x) * (a[0] - n.x) + (a[1] - n.y) * (a[1] - n.y) + (a[2] - n.z) * (a[2] - n.z);
  return dist;
}
// calc_box_dist (ikd_Tree.cpp:1702-1720); `present` false <=> nullptr or tree_deleted child
inline float calc_box_dist(bool present, const float box[6], const float p[3]) {
  if (!present) return INFINITY;
  float min_dist = 0.0f;
  if (p[0] < box[0]) min_dist += (p[0] - box[0]) * (p[0] - box[0]);
  if (p[0] > box[1]) min_dist += (p[0] - box[1]) * (p[0] - box[1]);
  if (p[1] < box[2]) min_dist += (p[1] - box[2]) * (p[1] - box[2]);
  if (p[1] > box[3]) min_dist += (p[1] - box[3]) * (p[1] - box[3]);
  if (p[2] < box[4]) min_dist += (p[2] - box[4]) * (p[2] - box[4]);
  if (p[2] > box[5]) min_dist += (p[2] - box[5]) * (p[2] - box[5]);
  return min_dist;
}

struct SnapSearch {
  const malio_map_node* nodes;
  int k;
  const float* q;
  ManualHeap heap;
  int64_t visits = 0;
  // KD_TREE::Search (ikd_Tree.cpp:1073-1255) on the snapshot.  `idx < 0` <=> root == nullptr || root->tree_deleted
  // (deleted subtrees are not in the snapshot).  max_dist = INFINITY as called from h_share_model.
  void Search(int64_t idx) {
    if (idx < 0) return;
    visits++;
    const malio_map_node& n = nodes[idx];
    if (!(n.link & MALIO_LINK_POINT_DELETED)) {
      float dist = calc_dist(q, n);
      if (heap.size() < k || dist < heap.top().dist) {
        if (heap.size() >= k) heap.pop();
        HeapItem it; it.dist = dist; it.x = n.x; it.idx = (int32_t)idx;
        heap.push(it);
      }
    }
    const bool hl = n.link & MALIO_LINK_HAS_LEFT, hr = n.link & MALIO_LINK_HAS_RIGHT;
    const int64_t li = hl ? idx + 1 : -1, ri = hr ? (int64_t)(n.link & MALIO_LINK_INDEX_MASK) : -1;
    float dist_left_node = calc_box_dist(hl, n.lbox, q);
    float dist_right_node = calc_box_dist(hr, n.rbox, q);
    if (heap.size() < k || (dist_left_node < heap.top().dist && dist_right_node < heap.top().dist)) {
      if (dist_left_node <= dist_right_node) {
        Search(li);
        if (heap.size() < k || dist_right_node < heap.top().dist) Search(ri);
      } else {
        Search(ri);
        if (heap.size() < k || dist_left_node < heap.top().dist) Search(li);
      }
    } else {
      if (dist_left_node < heap.top().dist) Search(li);
      if (dist_right_node < heap.top().dist) Search(ri);
    }
  }
};

// Nearest_Search (ikd_Tree.cpp:426-461): ascending order by repeated insert(begin) of the heap top
int knn_snapshot(const malio_map_node* nodes, const float* cov, uint32_t n_nodes, const float q[3], int k,
                 float* pts4, float* d2, int32_t* ids, int64_t* visits) {
  SnapSearch s;
  s.nodes = nodes; s.k = k; s.q = q;
  if (n_nodes > 0) s.Search(0);
  int k_found = std::min(k, s.heap.size());
  for (int i = 0; i < k; ++i) {
    if (ids) ids[i] = -1;
    if (d2) d2[i] = INFINITY;
  }
  for (int i = k_found - 1; i >= 0; --i) {
    HeapItem t = s.heap.top();
    if (ids) ids[i] = t.idx;
    if (d2) d2[i] = t.dist;
    if (pts4) {
      pts4[4 * i + 0] = nodes[t.idx].x; pts4[4 * i + 1] = nodes[t.idx].y; pts4[4 * i + 2] = nodes[t.idx].z;
      pts4[4 * i + 3] = cov ? cov[t.idx] : 0.f;
    }
    s.heap.pop();
  }
  if (visits) *visits += s.visits;
  return k_found;
}

// ------------------------------------------------------------------ P: esti_plane<float> (common_lib.h:144-190)
// Eigen::ColPivHouseholderQR<Matrix<float,5,3>>::solve restated (Eigen 3.3 ColPivHouseholderQR.h:
// computeInPlace + _solve_impl; Householder.h: makeHouseholderInPlace / applyHouseholderOnTheLeft).
void colpiv_qr_solve_5x3(const float Ain[5][3], const float bin[5], float xout[3]) {
  const int rows = 5, cols = 3, size = 3;
  float A[5][3];
  for (int i = 0; i < 5; ++i) for (int j = 0; j < 3; ++j) A[i][j] = Ain[i][j];
  float hCoeffs[3] = {0, 0, 0};
  int perm[3] = {0, 1, 2};          // column j of the permuted matrix is original column perm[j]
  float normsUpdated[3], normsDirect[3];
  for (int k = 0; k < cols; ++k) {
    float s = 0.f;
    for (int i = 0; i < rows; ++i) s += A[i][k] * A[i][k];
    normsDirect[k] = std::sqrt(s);
    normsUpdated[k] = normsDirect[k];
  }
  const float eps = std::numeric_limits<float>::epsilon();
  float maxn = std::max(normsUpdated[0], std::max(normsUpdated[1], normsUpdated[2]));
  const float threshold_helper = (maxn * eps) * (maxn * eps) / float(rows);
  const float norm_downdate_threshold = std::sqrt(eps);
  int nonzero_pivots = size;
  float maxpivot = 0.f;
  for (int k = 0; k < size; ++k) {
    int biggest = k;
    for (int j = k + 1; j < cols; ++j) if (normsUpdated[j] > normsUpdated[biggest]) biggest = j;
    float biggest_sq = normsUpdated[biggest] * normsUpdated[biggest];
    if (nonzero_pivots == size && biggest_sq < threshold_helper * float(rows - k)) nonzero_pivots = k;
    if (k != biggest) {
      for (int i = 0; i < rows; ++i) std::swap(A[i][k], A[i][biggest]);
      std::swap(normsUpdated[k], normsUpdated[biggest]);
      std::swap(normsDirect[k], normsDirect[biggest]);
      std::swap(perm[k], perm[biggest]);
    }
    // makeHouseholderInPlace on A[k..rows-1][k]
    float tailSq = 0.f;
    for (int i = k + 1; i < rows; ++i) tailSq += A[i][k] * A[i][k];
    float c0 = A[k][k], beta, tau;
    if (tailSq <= std::numeric_limits<float>::min()) {
      tau = 0.f; beta = c0;
      for (int i = k + 1; i < rows; ++i) A[i][k] = 0.f;
    } else {
      beta = std::sqrt(c0 * c0 + tailSq);
      if (c0 >= 0.f) beta = -beta;
      for (int i = k + 1; i < rows; ++i) A[i][k] = A[i][k] / (c0 - beta);
      tau = (beta - c0) / beta;
    }
    A[k][k] = beta;
    hCoeffs[k] = tau;
    if (std::fabs(beta) > maxpivot) maxpivot = std::fabs(beta);
    // applyHouseholderOnTheLeft to the trailing columns
    if (tau != 0.f) {
      for (int j = k + 1; j < cols; ++j) {
        float tmp = 0.f;
        for (int i = k + 1; i < rows; ++i) tmp += A[i][k] * A[i][j];
        tmp += A[k][j];
        A[k][j] -= tau * tmp;
        for (int i = k + 1; i < rows; ++i) A[i][j] -= tau * A[i][k] * tmp;
      }
    }
    // LAPACK-style norm down-dating
    for (int j = k + 1; j < cols; ++j) {
      if (normsUpdated[j] != 0.f) {
        float temp = std::fabs(A[k][j]) / normsUpdated[j];
        temp = (1.f + temp) * (1.f - temp);
        temp = temp < 0.f ? 0.f : temp;
        float r = normsUpdated[j] / normsDirect[j];
        float temp2 = temp * r * r;
        if (temp2 <= norm_downdate_threshold) {
          float s = 0.f;
          for (int i = k + 1; i < rows; ++i) s += A[i][j] * A[i][j];
          normsDirect[j] = std::sqrt(s);
          normsUpdated[j] = normsDirect[j];
        } else {
          normsUpdated[j] *= std::sqrt(temp);
        }
      }
    }
  }
  // _solve_impl: c = Q^T b ; solve R c = c on the nonzero_pivots block ; un-permute
  float c[5];
  for (int i = 0; i < 5; ++i) c[i] = bin[i];
  xout[0] = xout[1] = xout[2] = 0.f;
  if (nonzero_pivots == 0) return;
  for (int k = 0; k < nonzero_pivots; ++k) {
    float tau = hCoeffs[k];
    if (tau != 0.f) {
      float tmp = 0.f;
      for (int i = k + 1; i < rows; ++i) tmp += A[i][k] * c[i];
      tmp += c[k];
      c[k] -= tau * tmp;
      for (int i = k + 1; i < rows; ++i) c[i] -= tau * A[i][k] * tmp;
    }
  }
  for (int i = nonzero_pivots - 1; i >= 0; --i) {
    float s = c[i];
    for (int j = i + 1; j < nonzero_pivots; ++j) s -= A[i][j] * c[j];
    c[i] = s / A[i][i];
  }
  for (int i = 0; i < nonzero_pivots; ++i) xout[perm[i]] = c[i];
}

// esti_plane<float> (common_lib.h:144-190); near = 5 x {x,y,z,normal_y}
bool esti_plane(float pca_result[4], const float* near4, float threshold, double& plane_cov, double cov_threshold) {
  float A[5][3], b[5], W[5];
  double cov_sum = 0;
  plane_cov = 0;
  for (int j = 0; j < MALIO_K; ++j) {
    A[j][0] = near4[4 * j]; A[j][1] = near4[4 * j + 1]; A[j][2] = near4[4 * j + 2];
    W[j] = near4[4 * j + 3];
    b[j] = -1.0f;
    cov_sum += std::abs(cov_threshold - (double)W[j]);
  }
  if ((double)W[0] > 0.00001) {
    for (int j = 0; j < MALIO_K; ++j)
      plane_cov += ((cov_threshold - (double)W[j]) / cov_sum) * ((cov_threshold - (double)W[j]) / cov_sum) * (double)W[j];
  }
  float normvec[3];
  colpiv_qr_solve_5x3(A, b, normvec);
  float n = std::sqrt(normvec[0] * normvec[0] + normvec[1] * normvec[1] + normvec[2] * normvec[2]);
  pca_result[0] = normvec[0] / n;
  pca_result[1] = normvec[1] / n;
  pca_result[2] = normvec[2] / n;
  pca_result[3] = (float)(1.0 / (double)n);
  for (int j = 0; j < MALIO_K; ++j) {
    if (std::fabs(pca_result[0] * A[j][0] + pca_result[1] * A[j][1] + pca_result[2] * A[j][2] + pca_result[3]) > threshold)
      return false;
  }
  return true;
}

// ------------------------------------------------------------------ U: evalPointUncertainty (associate_uct.hpp:145-175)
// literal: cov_input 9x9, G 4x9, cov = (G cov_input G^T)[0:3,0:3]; returns the full 3x3
void evalPointUncertainty(const float p[3], const malio_pose_entry& pose, double cov_point[9]) {
  double cov_input[9][9];
  for (int i = 0; i < 9; ++i) for (int j = 0; j < 9; ++j) cov_input[i][j] = 0;
  for (int i = 0; i < 6; ++i) for (int j = 0; j < 6; ++j) cov_input[i][j] = pose.cov[6 * i + j] * 10000;
  for (int i = 0; i < 3; ++i) cov_input[6 + i][6 + i] = 0.1;
  const double distance_weight = 0.05;
  const double pc[4] = {p[0] * distance_weight, p[1] * distance_weight, p[2] * distance_weight, 1};
  double Tp[4];
  for (int i = 0; i < 4; ++i) Tp[i] = pose.T[4 * i] * pc[0] + pose.T[4 * i + 1] * pc[1] + pose.T[4 * i + 2] * pc[2] + pose.T[4 * i + 3] * pc[3];
  double G[4][9];
  for (int i = 0; i < 4; ++i) for (int j = 0; j < 9; ++j) G[i][j] = 0;
  // pointToFS: G[0:3,0:3] = point(3) I ; G[0:3,3:6] = -skew(point.xyz)
  for (int i = 0; i < 3; ++i) G[i][i] = Tp[3];
  double sk[9];
  skew(Tp, sk);
  for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) G[i][3 + j] = -sk[3 * i + j];
  // T * D, D = [I3; 0]
  for (int i = 0; i < 4; ++i) for (int j = 0; j < 3; ++j) G[i][6 + j] = pose.T[4 * i + j];
  double GS[4][9];
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 9; ++j) {
      double s = 0;
      for (int k = 0; k < 9; ++k) s += G[i][k] * cov_input[k][j];
      GS[i][j] = s;
    }
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      double s = 0;
      for (int k = 0; k < 9; ++k) s += GS[i][k] * G[j][k];
      cov_point[3 * i + j] = s;
    }
}

// singular values of an N x 3 matrix, descending (JacobiSVD singularValues, laserMapping.cpp:745-747):
// computed as sqrt(eig(A^T A)) with a cyclic Jacobi eigen-solver in double.
void singular_values_Nx3(const double* A, int64_t N, int64_t ld, double sv[3]) {
  double S[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
  for (int64_t i = 0; i < N; ++i)
    for (int a = 0; a < 3; ++a)
      for (int b = 0; b < 3; ++b) S[a][b] += A[i * ld + a] * A[i * ld + b];
  for (int sweep = 0; sweep < 60; ++sweep) {
    double off = std::fabs(S[0][1]) + std::fabs(S[0][2]) + std::fabs(S[1][2]);
    if (off < 1e-300) break;
    for (int p = 0; p < 2; ++p)
      for (int q = p + 1; q < 3; ++q) {
        if (S[p][q] == 0.0) continue;
        double theta = (S[q][q] - S[p][p]) / (2 * S[p][q]);
        double t = (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1));
        double c = 1 / std::sqrt(t * t + 1), s = t * c;
        for (int k = 0; k < 3; ++k) {   // S = S * J
          double skp = S[k][p], skq = S[k][q];
          S[k][p] = c * skp - s * skq;
          S[k][q] = s * skp + c * skq;
        }
        for (int k = 0; k < 3; ++k) {   // S = J^T * S
          double spk = S[p][k], sqk = S[q][k];
          S[p][k] = c * spk - s * sqk;
          S[q][k] = s * spk + c * sqk;
        }
      }
  }
  double e[3] = {S[0][0], S[1][1], S[2][2]};
  std::sort(e, e + 3);
  sv[0] = std::sqrt(std::max(e[2], 0.0));
  sv[1] = std::sqrt(std::max(e[1], 0.0));
  sv[2] = std::sqrt(std::max(e[0], 0.0));
}

// ------------------------------------------------------------------ generic dense helpers (row-major)
// Eigen PartialPivLU-based inverse (Matrix<double,35,35>::inverse(), esekfom.hpp:621,633; dynamic :579)
bool inverse_lu(const double* Ain, int n, double* inv) {
  std::vector<double> A(Ain, Ain + (size_t)n * n);
  std::vector<int> piv(n);
  for (int i = 0; i < n; ++i) piv[i] = i;
  for (int k = 0; k < n; ++k) {
    int p = k;
    double best = std::fabs(A[(size_t)k * n + k]);
    for (int i = k + 1; i < n; ++i) {
      double v = std::fabs(A[(size_t)i * n + k]);
      if (v > best) { best = v; p = i; }
    }
    if (best == 0.0) return false;
    if (p != k) {
      for (int j = 0; j < n; ++j) std::swap(A[(size_t)k * n + j], A[(size_t)p * n + j]);
      std::swap(piv[k], piv[p]);
    }
    for (int i = k + 1; i < n; ++i) {
      A[(size_t)i * n + k] /= A[(size_t)k * n + k];
      double f = A[(size_t)i * n + k];
      for (int j = k + 1; j < n; ++j) A[(size_t)i * n + j] -= f * A[(size_t)k * n + j];
    }
  }
  // solve A X = P  column by column
  std::vector<double> col(n);
  for (int c = 0; c < n; ++c) {
    for (int i = 0; i < n; ++i) col[i] = (piv[i] == c) ? 1.0 : 0.0;
    for (int i = 0; i < n; ++i) {
      double s = col[i];
      for (int j = 0; j < i; ++j) s -= A[(size_t)i * n + j] * col[j];
      col[i] = s;
    }
    for (int i = n - 1; i >= 0; --i) {
      double s = col[i];
      for (int j = i + 1; j < n; ++j) s -= A[(size_t)i * n + j] * col[j];
      col[i] = s / A[(size_t)i * n + i];
    }
    for (int i = 0; i < n; ++i) inv[(size_t)i * n + c] = col[i];
  }
  return true;
}

// ------------------------------------------------------------------ manifold ops (IKFoM_toolkit/mtk)
const double kTol = 1e-11;   // MTK::tolerance<double>(), mtkmath.hpp:122

// cos_sinc_sqrt (mtkmath.hpp:141-171); boost epsilon<double>() = 2^-52
void cos_sinc_sqrt(double x2, double& c, double& sinc) {
  static const double taylor_0_bound = std::numeric_limits<double>::epsilon();
  static const double taylor_2_bound = std::sqrt(taylor_0_bound);
  static const double taylor_n_bound = std::sqrt(taylor_2_bound);
  if (x2 >= taylor_n_bound) {
    double x = std::sqrt(x2);
    c = std::cos(x);
    sinc = std::sin(x) / x;
    return;
  }
  static const double inv[] = {1 / 3., 1 / 4., 1 / 5., 1 / 6., 1 / 7., 1 / 8., 1 / 9.};
  double cosi = 1., s = 1;
  double term = -1 / 2. * x2;
  for (int i = 0; i < 3; ++i) {
    cosi += term;
    term *= inv[2 * i];
    s += term;
    term *= -inv[2 * i + 1] * x2;
  }
  c = cosi;
  sinc = s;
}
// MTK::exp<scalar,3> (mtkmath.hpp:249-256): returns w, writes vec
double mtk_exp3(double res[3], const double vec[3], double scale) {
  double norm2 = vec[0] * vec[0] + vec[1] * vec[1] + vec[2] * vec[2];
  double c, sinc;
  cos_sinc_sqrt(scale * scale * norm2, c, sinc);
  double mult = sinc * scale;
  res[0] = mult * vec[0]; res[1] = mult * vec[1]; res[2] = mult * vec[2];
  return c;
}
// SO3::exp (SOn.hpp:332-336): scale/2 with scale = 1
Q4 so3_exp(const double v[3]) {
  double r[3];
  double w = mtk_exp3(r, v, 0.5);
  return Q4{w, r[0], r[1], r[2]};
}
// SO3::log -> MTK::log (mtkmath.hpp:268-289) with scale 2, plus_minus_periodicity = true
void so3_log(const Q4& q, double res[3]) {
  double nv = std::sqrt(q.x * q.x + q.y * q.y + q.z * q.z);
  if (nv < kTol) nv = kTol;
  double s = 2.0 / nv * std::atan(nv / q.w);
  res[0] = s * q.x; res[1] = s * q.y; res[2] = s * q.z;
}
// MTK::A_matrix (mtkmath.hpp:235-247)
void A_matrix(const double v[3], double res[9]) {
  double squaredNorm = v[0] * v[0] + v[1] * v[1] + v[2] * v[2];
  double norm = std::sqrt(squaredNorm);
  double I[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  if (norm < kTol) {
    for (int i = 0; i < 9; ++i) res[i] = I[i];
    return;
  }
  double h[9], hh[9];
  skew(v, h);
  m3m(h, h, hh);
  double a = (1 - std::cos(norm)) / squaredNorm, b = (1 - std::sin(norm) / norm) / squaredNorm;
  for (int i = 0; i < 9; ++i) res[i] = I[i] + a * h[i] + b * hh[i];
}

const double kGravLen = 98090.0 / 10000.0;   // S2<double,98090,10000,1>, use-ikfom.hpp:8

// S2::S2_Bx, S2_typ == 1 branch (S2.hpp:225-243); res is 3x2 row-major
void S2_Bx(const double vec[3], double res[6]) {
  const double length = kGravLen;
  if (vec[0] + length > kTol) {
    res[0] = -vec[1];                                   res[1] = -vec[2];
    res[2] = length - vec[1] * vec[1] / (length + vec[0]); res[3] = -vec[2] * vec[1] / (length + vec[0]);
    res[4] = -vec[2] * vec[1] / (length + vec[0]);      res[5] = length - vec[2] * vec[2] / (length + vec[0]);
    for (int i = 0; i < 6; ++i) res[i] /= length;
  } else {
    for (int i = 0; i < 6; ++i) res[i] = 0;
    res[3] = -1;   // res(1,1)
    res[4] = 1;    // res(2,0)
  }
}
// S2::boxplus (S2.hpp:136-142)
void S2_boxplus(double vec[3], const double delta[2]) {
  double Bx[6];
  S2_Bx(vec, Bx);
  double Bu[3];
  for (int i = 0; i < 3; ++i) Bu[i] = Bx[2 * i] * delta[0] + Bx[2 * i + 1] * delta[1];
  double r[3];
  double w = mtk_exp3(r, Bu, 0.5);
  double R[9];
  q_to_R(Q4{w, r[0], r[1], r[2]}, R);
  double o[3];
  m3v(R, vec, o);
  vec[0] = o[0]; vec[1] = o[1]; vec[2] = o[2];
}
// S2::boxminus (S2.hpp:144-168): res = this [-] other
void S2_boxminus(const double vec[3], const double other[3], double res[2]) {
  double hv[9], t[3];
  skew(vec, hv);
  m3v(hv, other, t);
  double v_sin = std::sqrt(t[0] * t[0] + t[1] * t[1] + t[2] * t[2]);
  double v_cos = vec[0] * other[0] + vec[1] * other[1] + vec[2] * other[2];
  double theta = std::atan2(v_sin, v_cos);
  if (v_sin < kTol) {
    if (std::fabs(theta) > kTol) { res[0] = 3.1415926; res[1] = 0; }
    else { res[0] = 0; res[1] = 0; }
  } else {
    double Bx[6];
    S2_Bx(other, Bx);
    double ho[9], u[3];
    skew(other, ho);
    m3v(ho, vec, u);
    double f = theta / v_sin;
    res[0] = f * (Bx[0] * u[0] + Bx[2] * u[1] + Bx[4] * u[2]);
    res[1] = f * (Bx[1] * u[0] + Bx[3] * u[1] + Bx[5] * u[2]);
  }
}
// S2::S2_Nx_yy (S2.hpp:269-274): 2x3 row-major
void S2_Nx_yy(const double vec[3], double res[6]) {
  double Bx[6], hv[9];
  S2_Bx(vec, Bx);
  skew(vec, hv);
  const double f = 1 / kGravLen / kGravLen;
  for (int i = 0; i < 2; ++i)
    for (int j = 0; j < 3; ++j)
      res[3 * i + j] = f * (Bx[i] * hv[j] + Bx[2 + i] * hv[3 + j] + Bx[4 + i] * hv[6 + j]);
}
// S2::S2_Mx (S2.hpp:276-291): 3x2 row-major.  NOTE scalar(1/2) == 0 => exp_delta is the identity.
void S2_Mx(const double vec[3], const double delta[2], double res[6]) {
  double Bx[6], hv[9];
  S2_Bx(vec, Bx);
  skew(vec, hv);
  if (std::sqrt(delta[0] * delta[0] + delta[1] * delta[1]) < kTol) {
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 2; ++j)
        res[2 * i + j] = -(hv[3 * i] * Bx[j] + hv[3 * i + 1] * Bx[2 + j] + hv[3 * i + 2] * Bx[4 + j]);
  } else {
    double Bu[3];
    for (int i = 0; i < 3; ++i) Bu[i] = Bx[2 * i] * delta[0] + Bx[2 * i + 1] * delta[1];
    double r[3];
    double w = mtk_exp3(r, Bu, 0.0);   // scalar(1/2): integer division
    double Rm[9];
    q_to_R(Q4{w, r[0], r[1], r[2]}, Rm);
    double A[9], At[9];
    A_matrix(Bu, A);
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) At[3 * i + j] = A[3 * j + i];
    double M1[9], M2[9];
    m3m(Rm, hv, M1);
    m3m(M1, At, M2);
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 2; ++j)
        res[2 * i + j] = -(M2[3 * i] * Bx[j] + M2[3 * i + 1] * Bx[2 + j] + M2[3 * i + 2] * Bx[4 + j]);
  }
}

// state layout (use-ikfom.hpp:14-27 generalised to L LiDARs, SURVEY.md §8a-S)
struct Layout {
  int L, n, c;
  int pos, rot, offR[MALIO_MAX_LIDAR], offT[MALIO_MAX_LIDAR], vel, bg, ba, grav;
  explicit Layout(int L_) : L(L_) {
    n = 17 + 6 * L; c = 6 * (L + 1);
    pos = 0; rot = 3;
    for (int l = 0; l < L; ++l) { offR[l] = 6 + 3 * l; offT[l] = 6 + 3 * L + 3 * l; }
    vel = 6 + 6 * L; bg = vel + 3; ba = bg + 3; grav = ba + 3;
  }
};

// state boxminus: dx = x [-] x0 (MTK_BUILD_MANIFOLD boxminus; vect.hpp:120, SOn.hpp:245-247, S2.hpp:144)
void state_boxminus(const Layout& ly, const malio_state& x, const malio_state& x0, double* dx) {
  for (int i = 0; i < 3; ++i) dx[ly.pos + i] = x.pos[i] - x0.pos[i];
  so3_log(q_mul(q_conj(q_from(x0.rot)), q_from(x.rot)), dx + ly.rot);
  for (int l = 0; l < ly.L; ++l) {
    so3_log(q_mul(q_conj(q_from(x0.ext[l].q)), q_from(x.ext[l].q)), dx + ly.offR[l]);
    for (int i = 0; i < 3; ++i) dx[ly.offT[l] + i] = x.ext[l].t[i] - x0.ext[l].t[i];
  }
  for (int i = 0; i < 3; ++i) {
    dx[ly.vel + i] = x.vel[i] - x0.vel[i];
    dx[ly.bg + i] = x.bg[i] - x0.bg[i];
    dx[ly.ba + i] = x.ba[i] - x0.ba[i];
  }
  S2_boxminus(x.grav, x0.grav, dx + ly.grav);
}
inline void q_store(const Q4& q, double o[4]) { o[0] = q.w; o[1] = q.x; o[2] = q.y; o[3] = q.z; }
// state boxplus (vect.hpp:117, SOn.hpp:241-244, S2.hpp:136)
void state_boxplus(const Layout& ly, malio_state& x, const double* dx) {
  for (int i = 0; i < 3; ++i) x.pos[i] += dx[ly.pos + i];
  q_store(q_mul(q_from(x.rot), so3_exp(dx + ly.rot)), x.rot);
  for (int l = 0; l < ly.L; ++l) {
    q_store(q_mul(q_from(x.ext[l].q), so3_exp(dx + ly.offR[l])), x.ext[l].q);
    for (int i = 0; i < 3; ++i) x.ext[l].t[i] += dx[ly.offT[l] + i];
  }
  for (int i = 0; i < 3; ++i) {
    x.vel[i] += dx[ly.vel + i];
    x.bg[i] += dx[ly.bg + i];
    x.ba[i] += dx[ly.ba + i];
  }
  S2_boxplus(x.grav, dx + ly.grav);
}

}  // namespace

// =================================================================== oracle context
typedef int (*orc_knn_fn)(void* ctx, const float q[3], int k, float* pts4, float* d2, int32_t* ids);

struct orc_ctx {
  malio_params prm;
  // map (snapshot) or hook
  const malio_map_node* nodes = nullptr;
  const float* node_cov = nullptr;
  uint32_t n_nodes = 0;
  orc_knn_fn hook = nullptr;
  void* hook_ctx = nullptr;
  // scan
  std::vector<malio_scan_pt> pts;
  std::vector<malio_pose_entry> table;
  std::vector<uint32_t> table_off;
  std::vector<malio_rigid> tcomp;
  // persistent across passes (file-scope globals in laserMapping.cpp:55-56,61,64)
  std::vector<float> nearest;        // Nearest_Points: N x 5 x {x,y,z,normal_y}
  std::vector<int32_t> nearest_ids;  // N x 5
  std::vector<float> nearest_d2;     // N x 5
  std::vector<int32_t> nearest_cnt;  // N
  std::vector<uint8_t> selected;     // point_selected_surf
  std::vector<float> world;          // feats_down_world xyz
  std::vector<float> normal_y;       // feats_down_body[i].normal_y
  int64_t visits = 0;                // node visits of the restated search (for V-bar, SURVEY.md §8d)
  int64_t searches = 0;
  // last-pass dense outputs (dyn_share_datastruct, esekfom.hpp:80-90)
  std::vector<double> h_x, h, R;
  int n_eff = 0;
  malio_pass_stats st{};
  // multi-rank protocol tests: global min/max injected between the two phases (what the MIN all-reduce delivers)
  bool mm_override = false;
  double ov_umin = 0, ov_umax = 0, ov_tmin = 0, ov_tmax = 0;
  double raw_min_cov = 9999, raw_max_cov = 0;   // local min/max trace of the selected points of the last pass
  // timing split for bench.py's CPU arms (seconds, accumulated since orc_reset_times):
  //   t_K  wall share of Nearest_Search inside S1 (per-thread search time summed / threads)
  //   t_B  rest of h_share_model (S1 without the search, S2-S6)
  //   t_A  update_iterated_dyn_share_modified outside h_share_model (esekfom.hpp:521-718)
  double t_K = 0, t_B = 0, t_A = 0;
  int time_passes = 0;
  bool fast_reduce = false;   // timing arms only: esekfom.hpp:622-635 evaluated by orc_reduce_fast (blocked, vectorised, threaded)
};

extern "C" {

void* orc_create(const malio_params* p) {
  orc_ctx* c = new orc_ctx;
  c->prm = *p;
  return c;
}
void orc_destroy(void* c) { delete (orc_ctx*)c; }

void orc_set_map_snapshot(void* vc, const malio_map_node* nodes, const float* cov, uint32_t n) {
  orc_ctx* c = (orc_ctx*)vc;
  c->nodes = nodes; c->node_cov = cov; c->n_nodes = n;
  c->hook = nullptr;
}
void orc_set_knn_hook(void* vc, orc_knn_fn fn, void* fctx) {
  orc_ctx* c = (orc_ctx*)vc;
  c->hook = fn; c->hook_ctx = fctx;
}
void orc_set_scan(void* vc, const malio_scan_pt* pts, uint32_t n, const malio_pose_entry* table,
                  const uint32_t* table_off, const malio_rigid* tcomp) {
  orc_ctx* c = (orc_ctx*)vc;
  const int L = c->prm.n_lidar;
  c->pts.assign(pts, pts + n);
  c->table_off.assign(table_off, table_off + L + 1);
  c->table.assign(table, table + table_off[L]);
  c->tcomp.clear();
  if (L > 1) c->tcomp.assign(tcomp, tcomp + (L - 1));
  c->nearest.assign((size_t)n * MALIO_K * 4, 0.f);
  c->nearest_ids.assign((size_t)n * MALIO_K, -1);
  c->nearest_d2.assign((size_t)n * MALIO_K, INFINITY);
  c->nearest_cnt.assign(n, 0);
  c->selected.assign(n, 0);
  c->world.assign((size_t)n * 3, 0.f);
  c->normal_y.assign(n, 0.f);
}

// stand-alone restated search over a snapshot (K), batch form
void orc_knn_snapshot_batch(const malio_map_node* nodes, const float* cov, uint32_t n_nodes, const float* q,
                            int64_t nq, int k, int32_t* out_ids, float* out_d2, int32_t* out_found,
                            int64_t* visits_total, int nthreads, int32_t* visits_per_query) {
  int64_t vt = 0;
  if (nthreads < 1) nthreads = 1;
#pragma omp parallel for num_threads(nthreads) schedule(dynamic, 256) reduction(+ : vt)
  for (int64_t i = 0; i < nq; ++i) {
    int64_t v = 0;
    int f = knn_snapshot(nodes, cov, n_nodes, q + 3 * i, k, nullptr, out_d2 ? out_d2 + i * k : nullptr,
                         out_ids ? out_ids + i * k : nullptr, &v);
    if (out_found) out_found[i] = f;
    if (visits_per_query) visits_per_query[i] = (int32_t)v;
    vt += v;
  }
  if (visits_total) *visits_total = vt;
}

// Balanced snapshot over a static point set: median split on the longest extent (KD_TREE::BuildTree,
// ikd_Tree.cpp:696-735), written straight in snapshot form.  The CPU arm of bench.py maps this instead of the
// product's malio_build_static_snapshot when no live reference tree was built; same rule, same nth_element,
// so the same snapshot (tests/test_oracle_cpu.py checks both byte for byte).
static void static_build_rec(const float* xyz, uint32_t* order, int64_t l, int64_t r, uint32_t slot, uint32_t depth,
                             malio_map_node* out, uint32_t* order_out, float box[6], uint32_t& max_depth) {
  max_depth = std::max(max_depth, depth);
  float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int64_t i = l; i <= r; ++i) {
    const float* p = xyz + 3 * (size_t)order[i];
    for (int k = 0; k < 3; ++k) { mn[k] = std::min(mn[k], p[k]); mx[k] = std::max(mx[k], p[k]); }
  }
  int axis = 0;
  for (int k = 1; k < 3; ++k) if (mx[k] - mn[k] > mx[axis] - mn[axis]) axis = k;
  const int64_t mid = (l + r) >> 1;
  std::nth_element(order + l, order + mid, order + r + 1,
                   [&](uint32_t a, uint32_t b) { return xyz[3 * (size_t)a + axis] < xyz[3 * (size_t)b + axis]; });
  malio_map_node& o = out[slot];
  const float* p = xyz + 3 * (size_t)order[mid];
  o.x = p[0]; o.y = p[1]; o.z = p[2];
  order_out[slot] = order[mid];
  const int64_t nl = mid - l, nr = r - mid;
  o.link = (nl > 0 ? MALIO_LINK_HAS_LEFT : 0u) | (nr > 0 ? (MALIO_LINK_HAS_RIGHT | (uint32_t)(slot + 1 + nl)) : 0u);
  for (int k = 0; k < 6; ++k) { o.lbox[k] = 0.f; o.rbox[k] = 0.f; }
  for (int k = 0; k < 3; ++k) { box[2 * k] = mn[k]; box[2 * k + 1] = mx[k]; }
  if (nl > 0) static_build_rec(xyz, order, l, mid - 1, slot + 1, depth + 1, out, order_out, o.lbox, max_depth);
  if (nr > 0) static_build_rec(xyz, order, mid + 1, r, (uint32_t)(slot + 1 + nl), depth + 1, out, order_out, o.rbox, max_depth);
}

int orc_build_static_snapshot(const float* xyz, uint32_t n, malio_map_node* nodes_out, uint32_t* order_out, uint32_t* max_depth_out) {
  uint32_t md = 0;
  if (n > 0) {
    std::vector<uint32_t> order(n);
    for (uint32_t i = 0; i < n; ++i) order[i] = i;
    float box[6];
    static_build_rec(xyz, order.data(), 0, (int64_t)n - 1, 0, 1, nodes_out, order_out, box, md);
  }
  *max_depth_out = md;
  return 0;
}

// per-point pieces exported for unit tests
int orc_esti_plane(const float* near4, float threshold, double cov_threshold, float pabcd[4], double* plane_cov) {
  return esti_plane(pabcd, near4, threshold, *plane_cov, cov_threshold) ? 1 : 0;
}
void orc_eval_point_uncertainty(const float p[3], const malio_pose_entry* pose, double cov[9]) {
  evalPointUncertainty(p, *pose, cov);
}
void orc_qr_solve_5x3(const float* A15, const float* b5, float* x3) {
  float A[5][3];
  for (int i = 0; i < 5; ++i) for (int j = 0; j < 3; ++j) A[i][j] = A15[3 * i + j];
  colpiv_qr_solve_5x3(A, b5, x3);
}
int orc_inverse(const double* A, int n, double* inv) { return inverse_lu(A, n, inv) ? 1 : 0; }
void orc_singular_values_Nx3(const double* A, int64_t N, int64_t ld, double sv[3]) { singular_values_Nx3(A, N, ld, sv); }
void orc_state_boxplus(int L, malio_state* x, const double* dx) { state_boxplus(Layout(L), *x, dx); }
void orc_state_boxminus(int L, const malio_state* x, const malio_state* x0, double* dx) { state_boxminus(Layout(L), *x, *x0, dx); }
void orc_A_matrix(const double v[3], double res[9]) { A_matrix(v, res); }
void orc_S2_Nx_yy(const double vec[3], double res[6]) { S2_Nx_yy(vec, res); }
void orc_S2_Mx(const double vec[3], const double delta[2], double res[6]) { S2_Mx(vec, delta, res); }

// ------------------------------------------------------------------ B: h_share_model (laserMapping.cpp:552-760)
// converge = ekfom_data.converge on entry.  Returns 1 if valid, 0 if "No Effective Points".
static int h_share_model_impl(orc_ctx* c, const malio_pass_state* s, int converge, int nthreads, double* knn_wall_s) {
  const malio_params& P = c->prm;
  const int L = P.n_lidar;
  const int64_t N = (int64_t)c->pts.size();
  const int ncol = 6 * (L + 1);
  // extrinsic_update(): laserMapping.cpp:291-308 — extrinsics come from the (live) state
  Q4 qE[MALIO_MAX_LIDAR];
  double tE[MALIO_MAX_LIDAR][3];
  for (int l = 0; l < L; ++l) { qE[l] = q_from(s->ext[l].q); for (int k = 0; k < 3; ++k) tE[l][k] = s->ext[l].t[k]; }
  Q4 qC[MALIO_MAX_LIDAR];
  double tC[MALIO_MAX_LIDAR][3];
  for (int l = 1; l < L; ++l) { qC[l] = q_from(c->tcomp[l - 1].q); for (int k = 0; k < 3; ++k) tC[l][k] = c->tcomp[l - 1].t[k]; }
  const Q4 srot = q_from(s->rot);

  std::vector<double> cov_plane(N, 0.0);
  std::vector<float> normvec((size_t)N * 4, 0.f);
  if (nthreads < 1) nthreads = 1;
  int64_t visits = 0;
  const double t_enter = omp_get_wtime();
  double knn_thread_s = 0.0;   // per-thread time inside Nearest_Search, summed over threads

  // ---- S1 (:559-612)
#pragma omp parallel for num_threads(nthreads) schedule(dynamic, 256) reduction(+ : visits, knn_thread_s)
  for (int64_t i = 0; i < N; ++i) {
    const malio_scan_pt& pb = c->pts[i];
    double p_body[3] = {pb.x, pb.y, pb.z};
    const int lid = pb.lidar;
    if (lid != 0) {   // :571-572
      double a[3], b[3], d[3];
      q_rot(qE[lid], p_body, a);
      for (int k = 0; k < 3; ++k) a[k] += tE[lid][k];
      q_rot(qC[lid], a, b);
      for (int k = 0; k < 3; ++k) d[k] = (b[k] + tC[lid][k]) - tE[0][k];
      q_rot(q_conj(qE[0]), d, p_body);
    }
    double m[3], g[3];
    q_rot(qE[0], p_body, m);
    for (int k = 0; k < 3; ++k) m[k] += tE[0][k];
    q_rot(srot, m, g);
    float pw[3];
    for (int k = 0; k < 3; ++k) { g[k] += s->pos[k]; pw[k] = (float)g[k]; c->world[3 * i + k] = pw[k]; }   // :574-578

    float* near = &c->nearest[(size_t)i * MALIO_K * 4];
    if (converge) {   // :583-588
      float d2[MALIO_K];
      int32_t ids[MALIO_K];
      int found;
      const double tk0 = omp_get_wtime();
      if (c->hook) found = c->hook(c->hook_ctx, pw, MALIO_K, near, d2, ids);
      else found = knn_snapshot(c->nodes, c->node_cov, c->n_nodes, pw, MALIO_K, near, d2, ids, &visits);
      knn_thread_s += omp_get_wtime() - tk0;
      c->nearest_cnt[i] = found;
      for (int k = 0; k < MALIO_K; ++k) { c->nearest_ids[(size_t)i * MALIO_K + k] = ids[k]; c->nearest_d2[(size_t)i * MALIO_K + k] = d2[k]; }
      c->selected[i] = found < MALIO_K ? 0 : (d2[MALIO_K - 1] > P.knn_max_sqdist ? 0 : 1);
    }
    if (!c->selected[i]) continue;
    float pabcd[4];
    double unit_cov;
    c->selected[i] = 0;
    if (esti_plane(pabcd, near, P.plane_th, unit_cov, P.cov_threshold)) {   // :596
      float pd2 = pabcd[0] * pw[0] + pabcd[1] * pw[1] + pabcd[2] * pw[2] + pabcd[3];
      double nb = std::sqrt(p_body[0] * p_body[0] + p_body[1] * p_body[1] + p_body[2] * p_body[2]);
      float sc = (float)(1 - 0.9 * std::fabs(pd2) / std::sqrt(nb));   // :599
      if (sc > 0.1) {
        c->selected[i] = 1;
        normvec[4 * i] = pabcd[0]; normvec[4 * i + 1] = pabcd[1]; normvec[4 * i + 2] = pabcd[2];
        normvec[4 * i + 3] = pd2;
        cov_plane[i] = unit_cov;
      }
    }
  }
  if (converge) { c->visits += visits; c->searches += N; }
  *knn_wall_s = knn_thread_s / (double)nthreads;
  (void)t_enter;

  // ---- S2 (:614-632) compaction + min/max unit cov
  int effct = 0;
  double max_unit_cov = 0, min_unit_cov = 1000;
  std::vector<int64_t> ori(N);
  for (int64_t i = 0; i < N; ++i) {
    if (c->selected[i]) {
      ori[effct] = i;
      cov_plane[effct] = cov_plane[i];
      if (cov_plane[effct] > max_unit_cov) max_unit_cov = cov_plane[effct];
      if (cov_plane[effct] < min_unit_cov) min_unit_cov = cov_plane[effct];
      effct++;
    }
  }
  c->n_eff = effct;
  c->st = malio_pass_stats{};
  c->st.n_points = (uint32_t)N;
  c->st.n_eff = (uint32_t)effct;
  c->st.searched = converge ? 1 : 0;
  if (c->mm_override) { min_unit_cov = c->ov_umin; max_unit_cov = c->ov_umax; }
  if (effct < 1) {   // :635-639
    c->st.valid = 0;
    return 0;
  }
  c->st.valid = 1;
  c->h_x.assign((size_t)effct * ncol, 0.0);
  c->h.assign(effct, 0.0);
  c->R.assign(effct, 0.0);
  std::vector<float> sel_normal_y(effct, 0.f);   // laserCloudOri[i].normal_y

  double max_cov = 0, min_cov = 9999;
  // ---- S3 (:649-708)
  for (int i = 0; i < effct; ++i) {
    if (cov_plane[i] == 0) cov_plane[i] = 1;
    else if (max_unit_cov == min_unit_cov) cov_plane[i] = (P.plane_cov_max + P.plane_cov_min) / 2;
    else cov_plane[i] = 1 / ((P.plane_cov_max - P.plane_cov_min) * (cov_plane[i] - min_unit_cov) / (max_unit_cov - min_unit_cov) + P.plane_cov_min);

    const malio_scan_pt& lp = c->pts[ori[i]];
    double point_this_be[3] = {lp.x, lp.y, lp.z};
    const int lid = lp.lidar;
    if (lid != 0) {
      double a[3], b[3], d[3];
      q_rot(qE[lid], point_this_be, a);
      for (int k = 0; k < 3; ++k) a[k] += tE[lid][k];
      q_rot(qC[lid], a, b);
      for (int k = 0; k < 3; ++k) d[k] = (b[k] + tC[lid][k]) - tE[0][k];
      q_rot(q_conj(qE[0]), d, point_this_be);
    }
    double point_be_crossmat[9];
    skew(point_this_be, point_be_crossmat);
    double point_this[3];
    q_rot(qE[0], point_this_be, point_this);
    for (int k = 0; k < 3; ++k) point_this[k] += tE[0][k];
    double point_crossmat[9];
    skew(point_this, point_crossmat);

    const float* np_ = &normvec[4 * ori[i]];
    const double norm_vec[3] = {np_[0], np_[1], np_[2]};
    double C[3], A[3], B[3];
    q_rot(q_conj(srot), norm_vec, C);           // :676
    m3v(point_crossmat, C, A);                  // :677
    double* row = &c->h_x[(size_t)i * ncol];
    row[0] = np_[0]; row[1] = np_[1]; row[2] = np_[2]; row[3] = A[0]; row[4] = A[1]; row[5] = A[2];   // :679

    if (P.extrinsic_est_en) {
      if (lid == 0) {   // :684  (M3D * Quaternion) * V3D == (M * R(q)) * C
        double Rq[9], MR[9];
        q_to_R(q_conj(qE[0]), Rq);
        m3m(point_be_crossmat, Rq, MR);
        m3v(MR, C, B);
      } else {          // :687-690
        double point_ori[3] = {lp.x, lp.y, lp.z};
        skew(point_ori, point_be_crossmat);
        double C2[3];
        q_rot(q_conj(qC[lid]), C, C2);
        C[0] = C2[0]; C[1] = C2[1]; C[2] = C2[2];
        double Rq[9], MR[9];
        q_to_R(q_conj(qE[lid]), Rq);
        m3m(point_be_crossmat, Rq, MR);
        m3v(MR, C, B);
      }
      for (int k = 0; k < 3; ++k) { row[6 + 3 * lid + k] = B[k]; row[6 + 3 * (L + lid) + k] = C[k]; }   // :692-693
      int uncertain = (int)lp.table_idx;
      const int tsize = (int)(c->table_off[lid + 1] - c->table_off[lid]);
      if (uncertain >= tsize) uncertain = tsize - 2;   // :695-696
      double cov[9];
      const float pxyz[3] = {lp.x, lp.y, lp.z};
      evalPointUncertainty(pxyz, c->table[c->table_off[lid] + uncertain], cov);
      c->R[i] = cov[0] + cov[4] + cov[8];
      sel_normal_y[i] = (float)(cov[0] + cov[4] + cov[8]);
      if (max_cov < c->R[i]) max_cov = c->R[i];
      if (min_cov > c->R[i]) min_cov = c->R[i];
    }
    c->h[i] = (-1) * np_[3];   // :707
  }
  c->raw_min_cov = min_cov; c->raw_max_cov = max_cov;
  if (c->mm_override) { min_cov = c->ov_tmin; max_cov = c->ov_tmax; }
  c->st.u_min = min_unit_cov; c->st.u_max = max_unit_cov;
  c->st.tau_min = min_cov; c->st.tau_max = max_cov;

  // ---- S4 (:711-722)  FIC.  DEFINED HERE (reference yields 0/0 = NaN, SURVEY.md quirk 8): when every selected
  // point has the same trace and neither clamp fires, R_i = mid-range.
  for (int i = 0; i < effct; ++i) {
    double* row = &c->h_x[(size_t)i * ncol];
    for (int k = 0; k < ncol; ++k) row[k] = row[k] * cov_plane[i];
    c->h[i] = c->h[i] * cov_plane[i];
    if (c->R[i] < min_cov + (max_cov - min_cov) * P.range_min) c->R[i] = P.point_cov_min;
    else if (c->R[i] > min_cov + (max_cov - min_cov) * P.range_max) c->R[i] = P.point_cov_max;
    else {
      double den = (P.range_max - P.range_min) * (max_cov - min_cov);
      if (den == 0.0) c->R[i] = (P.point_cov_max + P.point_cov_min) / 2;
      else c->R[i] = (P.point_cov_max - P.point_cov_min) * (c->R[i] - (min_cov + (max_cov - min_cov) * P.range_min)) / den + P.point_cov_min;
    }
  }
  // ---- S5 (:725-743)
  {
    int k = 0;
    for (int64_t i = 0; i < N; ++i) {
      if (c->selected[i]) {
        if (P.extrinsic_est_en) c->normal_y[i] = sel_normal_y[k];
        k++;
      } else {
        const malio_scan_pt& pb = c->pts[i];
        const int which = pb.lidar;
        int imu_idx = (int)pb.table_idx;
        const int tsize = (int)(c->table_off[which + 1] - c->table_off[which]);
        if (imu_idx >= tsize - 1) imu_idx = tsize - 2;
        double cov[9];
        const float pxyz[3] = {pb.x, pb.y, pb.z};
        evalPointUncertainty(pxyz, c->table[c->table_off[which] + imu_idx], cov);
        c->normal_y[i] = (float)(cov[0] + cov[4] + cov[8]);
      }
    }
  }
  // ---- S6 (:745-759)
  double sv[3];
  singular_values_Nx3(c->h_x.data(), effct, ncol, sv);
  double weight = sv[2] / sv[0];
  if (weight > P.localize_thresh_max) weight = P.localize_cov_max;
  else if (weight < P.localize_thresh_min) weight = P.localize_cov_min;
  else weight = (P.localize_cov_max - P.localize_cov_min) * (weight - P.localize_thresh_min) / (P.localize_thresh_max - P.localize_thresh_min) + P.localize_cov_min;
  for (size_t k = 0; k < c->h_x.size(); ++k) c->h_x[k] *= weight;
  for (int i = 0; i < effct; ++i) c->h[i] *= weight;
  c->st.sigma[0] = sv[0]; c->st.sigma[1] = sv[1]; c->st.sigma[2] = sv[2];
  c->st.loc_weight = weight;
  return 1;
}

int orc_h_share_model(void* vc, const malio_pass_state* s, int converge, int nthreads) {
  orc_ctx* c = (orc_ctx*)vc;
  const double t0 = omp_get_wtime();
  double knn_s = 0.0;
  const int rc = h_share_model_impl(c, s, converge, nthreads < 1 ? 1 : nthreads, &knn_s);
  const double dt = omp_get_wtime() - t0;
  c->t_K += knn_s;
  c->t_B += dt - knn_s;
  c->time_passes += 1;
  return rc;
}
void orc_reset_times(void* vc) { orc_ctx* c = (orc_ctx*)vc; c->t_K = c->t_B = c->t_A = 0; c->time_passes = 0; }
void orc_get_times(void* vc, double out[3], int* passes) {
  orc_ctx* c = (orc_ctx*)vc;
  out[0] = c->t_K; out[1] = c->t_B; out[2] = c->t_A;
  if (passes) *passes = c->time_passes;
}
void orc_set_fast_reduce(void* vc, int enable) { ((orc_ctx*)vc)->fast_reduce = enable != 0; }

// esekfom.hpp:622-635 on the dense outputs of the last pass: HTH = (h_x^T / R) h_x ; HTh = (h_x^T / R) h
// map_incremental's per-point decision (laserMapping.cpp:398-446) with the state after the update
// (pointBodyToWorld, :134-147).  cls: 0 skipped (:406), 1 PointToAdd, 2 PointNoNeedDownsample, 3 dropped (:431)
void orc_map_incremental(void* vc, const malio_pass_state* s, double filter_size_map_min, int flg_EKF_inited,
                         uint8_t* cls, float* world_out) {
  orc_ctx* c = (orc_ctx*)vc;
  const malio_params& P = c->prm;
  const int L = P.n_lidar;
  const int64_t N = (int64_t)c->pts.size();
  Q4 qE[MALIO_MAX_LIDAR], qC[MALIO_MAX_LIDAR];
  double tE[MALIO_MAX_LIDAR][3], tC[MALIO_MAX_LIDAR][3];
  for (int l = 0; l < L; ++l) { qE[l] = q_from(s->ext[l].q); for (int k = 0; k < 3; ++k) tE[l][k] = s->ext[l].t[k]; }
  for (int l = 1; l < L; ++l) { qC[l] = q_from(c->tcomp[l - 1].q); for (int k = 0; k < 3; ++k) tC[l][k] = c->tcomp[l - 1].t[k]; }
  const Q4 srot = q_from(s->rot);
  for (int64_t i = 0; i < N; ++i) {
    cls[i] = 0;
    if (world_out) { world_out[3 * i] = 0.f; world_out[3 * i + 1] = 0.f; world_out[3 * i + 2] = 0.f; }
    if ((double)c->normal_y[i] > P.cov_threshold) continue;                                   // :406
    const malio_scan_pt& pb = c->pts[i];
    const double p_body[3] = {pb.x, pb.y, pb.z};
    const int lid = pb.lidar;
    double a[3], g[3];
    q_rot(qE[lid], p_body, a);
    for (int k = 0; k < 3; ++k) a[k] += tE[lid][k];
    if (lid != 0) {                                                                           // :142
      double b[3];
      q_rot(qC[lid], a, b);
      for (int k = 0; k < 3; ++k) a[k] = b[k] + tC[lid][k];
    }
    q_rot(srot, a, g);
    float w[3];
    for (int k = 0; k < 3; ++k) { g[k] += s->pos[k]; w[k] = (float)g[k]; }
    if (world_out) { world_out[3 * i] = w[0]; world_out[3 * i + 1] = w[1]; world_out[3 * i + 2] = w[2]; }
    const int cnt = c->nearest_cnt[i];
    if (cnt > 0 && flg_EKF_inited) {                                                          // :411
      const float* near = &c->nearest[(size_t)i * MALIO_K * 4];
      const double fs = filter_size_map_min;
      float mid[3];
      for (int k = 0; k < 3; ++k) mid[k] = (float)(std::floor((double)w[k] / fs) * fs + 0.5 * fs);   // :417-419
      const float dist = (w[0] - mid[0]) * (w[0] - mid[0]) + (w[1] - mid[1]) * (w[1] - mid[1]) + (w[2] - mid[2]) * (w[2] - mid[2]);
      if ((double)std::fabs(near[0] - mid[0]) > 0.5 * fs && (double)std::fabs(near[1] - mid[1]) > 0.5 * fs &&
          (double)std::fabs(near[2] - mid[2]) > 0.5 * fs) { cls[i] = 2; continue; }         // :421-425
      bool need_add = true;
      for (int j = 0; j < MALIO_K; ++j) {                                                     // :426-435
        if (cnt < MALIO_K) break;
        const float* q = near + 4 * j;
        const float dj = (q[0] - mid[0]) * (q[0] - mid[0]) + (q[1] - mid[1]) * (q[1] - mid[1]) + (q[2] - mid[2]) * (q[2] - mid[2]);
        if (dj < dist) { need_add = false; break; }
      }
      cls[i] = need_add ? 1 : 3;
    } else {
      cls[i] = 1;                                                                             // :439-440
    }
  }
}

void orc_reduce(void* vc, double* HTH, double* HTh) {
  orc_ctx* c = (orc_ctx*)vc;
  const int ncol = 6 * (c->prm.n_lidar + 1);
  std::vector<double> HT((size_t)ncol * c->n_eff);
  for (int i = 0; i < c->n_eff; ++i) {
    double r = c->R[i];
    if (r < 0.0001) r = 0.001;
    for (int k = 0; k < ncol; ++k) HT[(size_t)k * c->n_eff + i] = c->h_x[(size_t)i * ncol + k] / r;
  }
  for (int a = 0; a < ncol; ++a) {
    for (int b = 0; b < ncol; ++b) {
      double s = 0;
      for (int i = 0; i < c->n_eff; ++i) s += HT[(size_t)a * c->n_eff + i] * c->h_x[(size_t)i * ncol + b];
      HTH[a * ncol + b] = s;
    }
    double s = 0;
    for (int i = 0; i < c->n_eff; ++i) s += HT[(size_t)a * c->n_eff + i] * c->h[i];
    HTh[a] = s;
  }
}

// Timing arms only (bench.py cpu_baseline / --impl reference): the same esekfom.hpp:622-635 quantities, evaluated the way
// an optimised build of the reference evaluates them — Eigen's `HT * h_x_` GEMM (:629) and `P_inv.block * HT * dyn_share.h`
// (:635, which Eigen evaluates left to right: an n x c x N product before the N-vector) — i.e. blocked, vectorised
// (run-time dispatch to AVX2 / AVX-512 clones: MORE generous than the reference's baseline x86-64 build) and spread over
// `nthreads` OpenMP threads with per-thread accumulators.  Summation order differs from orc_reduce, so the parity tests
// never use it.  Kh (n) may be NULL; Pinv_blk is P_inv[:, 0:ncol] TRANSPOSED ([k][q]) with leading dimension ldp.
__attribute__((target_clones("avx512f", "avx2", "default"), optimize("O3")))
static void reduce_rows_fast(const double* hx, const double* h, const double* R, int ncol, int64_t i0, int64_t i1,
                             double* HTH, double* HTh, const double* Pinv_blk, int ldp, int n, double* Kh) {
  double s[MALIO_MAX_COLS], kq[MALIO_MAX_DOF];
  for (int64_t i = i0; i < i1; ++i) {
    double r = R[i];
    if (r < 0.0001) r = 0.001;
    const double* row = hx + (size_t)i * ncol;
    for (int k = 0; k < ncol; ++k) s[k] = row[k] / r;
    for (int a = 0; a < ncol; ++a) {
      double* out = HTH + (size_t)a * ncol;
      const double sa = s[a];
      for (int b = 0; b < ncol; ++b) out[b] += sa * row[b];
    }
    const double hi = h[i];
    for (int a = 0; a < ncol; ++a) HTh[a] += s[a] * hi;
    if (Kh) {   // column i of P_inv.block * HT (Pinv_blk is passed TRANSPOSED: [k][q], unit stride over q), times h_i
      for (int q = 0; q < n; ++q) kq[q] = 0.0;
      for (int k = 0; k < ncol; ++k) {
        const double* pr = Pinv_blk + (size_t)k * ldp;
        const double sk = s[k];
        for (int q = 0; q < n; ++q) kq[q] += pr[q] * sk;
      }
      for (int q = 0; q < n; ++q) Kh[q] += kq[q] * hi;
    }
  }
}
void orc_reduce_fast(void* vc, double* HTH, double* HTh, const double* Pinv_blk, int ldp, int n, double* Kh, int nthreads) {
  orc_ctx* c = (orc_ctx*)vc;
  const int ncol = 6 * (c->prm.n_lidar + 1);
  if (nthreads < 1) nthreads = 1;
  std::vector<double> part((size_t)nthreads * (ncol * ncol + ncol + MALIO_MAX_DOF), 0.0);
  const int64_t N = c->n_eff;
#pragma omp parallel num_threads(nthreads)
  {
    const int t = omp_get_thread_num(), T = omp_get_num_threads();
    double* base = part.data() + (size_t)t * (ncol * ncol + ncol + MALIO_MAX_DOF);
    const int64_t i0 = N * t / T, i1 = N * (t + 1) / T;
    reduce_rows_fast(c->h_x.data(), c->h.data(), c->R.data(), ncol, i0, i1, base, base + ncol * ncol, Pinv_blk, ldp, n,
                     Kh ? base + ncol * ncol + ncol : nullptr);
  }
  std::fill(HTH, HTH + ncol * ncol, 0.0);
  std::fill(HTh, HTh + ncol, 0.0);
  if (Kh) std::fill(Kh, Kh + n, 0.0);
  for (int t = 0; t < nthreads; ++t) {
    const double* base = part.data() + (size_t)t * (ncol * ncol + ncol + MALIO_MAX_DOF);
    for (int k = 0; k < ncol * ncol; ++k) HTH[k] += base[k];
    for (int k = 0; k < ncol; ++k) HTh[k] += base[ncol * ncol + k];
    if (Kh) for (int k = 0; k < n; ++k) Kh[k] += base[ncol * ncol + ncol + k];
  }
}

// ---- helpers for the multi-rank protocol tests (tests/test_multirank_gloo.py)
void orc_set_minmax_override(void* vc, int enable, double umin, double umax, double tmin, double tmax) {
  orc_ctx* c = (orc_ctx*)vc;
  c->mm_override = enable != 0;
  c->ov_umin = umin; c->ov_umax = umax; c->ov_tmin = tmin; c->ov_tmax = tmax;
}
// local min/max as the first phase of a rank sees them: {u_min, u_max, tau_min, tau_max} before any override
void orc_get_local_minmax(void* vc, double out[4]) {
  orc_ctx* c = (orc_ctx*)vc;
  out[0] = c->st.u_min; out[1] = c->st.u_max; out[2] = c->raw_min_cov; out[3] = c->raw_max_cov;
}
// the additive partials of one rank with the (scalar) localization weight divided out:
//   G = sum h_x^T/R h_x / w^2 ; g = sum h_x^T/R h / w^2 ; S = h_x[:,0:3]^T h_x[:,0:3] / w^2 (xx,xy,xz,yy,yz,zz)
void orc_partials(void* vc, double* G, double* g, double* S) {
  orc_ctx* c = (orc_ctx*)vc;
  const int ncol = 6 * (c->prm.n_lidar + 1);
  const double w2 = c->st.loc_weight * c->st.loc_weight;
  orc_reduce(vc, G, g);
  for (int k = 0; k < ncol * ncol; ++k) G[k] /= w2;
  for (int k = 0; k < ncol; ++k) g[k] /= w2;
  double s[6] = {0, 0, 0, 0, 0, 0};
  for (int i = 0; i < c->n_eff; ++i) {
    const double* r = &c->h_x[(size_t)i * ncol];
    s[0] += r[0] * r[0]; s[1] += r[0] * r[1]; s[2] += r[0] * r[2];
    s[3] += r[1] * r[1]; s[4] += r[1] * r[2]; s[5] += r[2] * r[2];
  }
  for (int k = 0; k < 6; ++k) S[k] = s[k] / w2;
}

// accessors
int orc_n_eff(void* vc) { return ((orc_ctx*)vc)->n_eff; }
void orc_get_stats(void* vc, malio_pass_stats* st) { *st = ((orc_ctx*)vc)->st; }
void orc_get_dense(void* vc, double* h_x, double* h, double* R) {
  orc_ctx* c = (orc_ctx*)vc;
  if (h_x) std::memcpy(h_x, c->h_x.data(), c->h_x.size() * 8);
  if (h) std::memcpy(h, c->h.data(), c->h.size() * 8);
  if (R) std::memcpy(R, c->R.data(), c->R.size() * 8);
}
void orc_get_aux(void* vc, float* normal_y, int32_t* nn_ids, float* nn_d2, uint8_t* selected, float* world, int32_t* nn_cnt) {
  orc_ctx* c = (orc_ctx*)vc;
  if (normal_y) std::memcpy(normal_y, c->normal_y.data(), c->normal_y.size() * 4);
  if (nn_ids) std::memcpy(nn_ids, c->nearest_ids.data(), c->nearest_ids.size() * 4);
  if (nn_d2) std::memcpy(nn_d2, c->nearest_d2.data(), c->nearest_d2.size() * 4);
  if (selected) std::memcpy(selected, c->selected.data(), c->selected.size());
  if (world) std::memcpy(world, c->world.data(), c->world.size() * 4);
  if (nn_cnt) std::memcpy(nn_cnt, c->nearest_cnt.data(), c->nearest_cnt.size() * 4);
}
void orc_get_visits(void* vc, int64_t* visits, int64_t* searches) {
  orc_ctx* c = (orc_ctx*)vc;
  *visits = c->visits; *searches = c->searches;
}

// ------------------------------------------------------------------ A: update_iterated_dyn_share_modified (esekfom.hpp:495-721)
// x, P (n x n row-major) updated in place.  dx_log (optional): (max_iter+1) x n, the dx_ of every pass that reached
// :642 (rows of skipped passes are left untouched); pass_flags (optional): per pass bit0 = valid, bit1 = searched.
int orc_update_iterated(void* vc, malio_state* x_, double* P_, int maximum_iter, double R, int nthreads,
                        double* dx_log, int32_t* pass_flags, malio_update_report* rep) {
  orc_ctx* c = (orc_ctx*)vc;
  const Layout ly(c->prm.n_lidar);
  const int n = ly.n, ncol = ly.c;
  bool valid = true, converge = true;
  int t = 0;
  malio_state x_propagated = *x_;
  std::vector<double> P_propagated(P_, P_ + (size_t)n * n);
  std::vector<double> K_h(n), K_x((size_t)n * n), dx_new(n, 0.0), dx(n), L_((size_t)n * n);
  int so3_idx[1 + MALIO_MAX_LIDAR];
  so3_idx[0] = ly.rot;
  for (int l = 0; l < ly.L; ++l) so3_idx[1 + l] = ly.offR[l];
  const int n_so3 = 1 + ly.L;
  int passes = 0, searches = 0;
  if (rep) std::memset(rep, 0, sizeof(*rep));

  auto apply_left3 = [&](std::vector<double>& M, int idx, const double J[9], const std::vector<double>& src) {
    for (int i = 0; i < n; ++i) {   // block<3,1>(idx,i) = J * src.block<3,1>(idx,i)
      double v[3] = {src[(size_t)(idx)*n + i], src[(size_t)(idx + 1) * n + i], src[(size_t)(idx + 2) * n + i]}, o[3];
      m3v(J, v, o);
      for (int k = 0; k < 3; ++k) M[(size_t)(idx + k) * n + i] = o[k];
    }
  };
  auto apply_right3T = [&](std::vector<double>& M, int idx, const double J[9]) {
    for (int i = 0; i < n; ++i) {   // block<1,3>(i,idx) = block<1,3>(i,idx) * J^T
      double v[3] = {M[(size_t)i * n + idx], M[(size_t)i * n + idx + 1], M[(size_t)i * n + idx + 2]}, o[3];
      m3v(J, v, o);
      for (int k = 0; k < 3; ++k) M[(size_t)i * n + idx + k] = o[k];
    }
  };

  std::vector<double> P(P_, P_ + (size_t)n * n);
  double t_seg = omp_get_wtime();   // t_A: everything of this function outside h_share_model
  for (int i = -1; i < maximum_iter; i++) {
    valid = true;
    malio_pass_state ps;
    std::memcpy(ps.rot, x_->rot, sizeof(ps.rot));
    std::memcpy(ps.pos, x_->pos, sizeof(ps.pos));
    std::memcpy(ps.ext, x_->ext, sizeof(ps.ext));
    const bool searched = converge;
    c->t_A += omp_get_wtime() - t_seg;
    valid = orc_h_share_model(c, &ps, converge ? 1 : 0, nthreads) != 0;   // :512
    t_seg = omp_get_wtime();
    passes++;
    if (searched) searches++;
    if (pass_flags) pass_flags[i + 1] = (valid ? 1 : 0) | (searched ? 2 : 0);
    if (!valid) continue;   // :514-517
    const int dof_Measurement = c->n_eff;
    state_boxminus(ly, *x_, x_propagated, dx.data());   // :526
    dx_new = dx;
    P = P_propagated;   // :530
    for (int si = 0; si < n_so3; ++si) {   // :534-549
      const int idx = so3_idx[si];
      double A[9], J[9];
      A_matrix(&dx[idx], A);
      for (int a = 0; a < 3; ++a) for (int b = 0; b < 3; ++b) J[3 * a + b] = A[3 * b + a];
      double o[3];
      m3v(J, &dx_new[idx], o);
      dx_new[idx] = o[0]; dx_new[idx + 1] = o[1]; dx_new[idx + 2] = o[2];
      apply_left3(P, idx, J, P);
      apply_right3T(P, idx, J);
    }
    {   // S2 block (:553-572)
      const int idx = ly.grav;
      double Nx[6], Mx[6], J2[4];
      S2_Nx_yy(x_->grav, Nx);
      S2_Mx(x_propagated.grav, &dx[idx], Mx);
      for (int a = 0; a < 2; ++a) for (int b = 0; b < 2; ++b) J2[2 * a + b] = Nx[3 * a] * Mx[b] + Nx[3 * a + 1] * Mx[2 + b] + Nx[3 * a + 2] * Mx[4 + b];
      double d0 = dx_new[idx], d1 = dx_new[idx + 1];
      dx_new[idx] = J2[0] * d0 + J2[1] * d1;
      dx_new[idx + 1] = J2[2] * d0 + J2[3] * d1;
      for (int k = 0; k < n; ++k) {
        double a0 = P[(size_t)idx * n + k], a1 = P[(size_t)(idx + 1) * n + k];
        P[(size_t)idx * n + k] = J2[0] * a0 + J2[1] * a1;
        P[(size_t)(idx + 1) * n + k] = J2[2] * a0 + J2[3] * a1;
      }
      for (int k = 0; k < n; ++k) {
        double a0 = P[(size_t)k * n + idx], a1 = P[(size_t)k * n + idx + 1];
        P[(size_t)k * n + idx] = a0 * J2[0] + a1 * J2[1];
        P[(size_t)k * n + idx + 1] = a0 * J2[2] + a1 * J2[3];
      }
    }
    if (n > dof_Measurement) {   // :574-582 (scalar R, per-point R ignored)
      const int m = dof_Measurement;
      std::vector<double> Hc((size_t)m * n, 0.0);
      for (int r = 0; r < m; ++r) for (int k = 0; k < ncol; ++k) Hc[(size_t)r * n + k] = c->h_x[(size_t)r * ncol + k];
      std::vector<double> PHt((size_t)n * m), S((size_t)m * m), Sinv((size_t)m * m);
      for (int a = 0; a < n; ++a) for (int r = 0; r < m; ++r) { double s = 0; for (int k = 0; k < n; ++k) s += P[(size_t)a * n + k] * Hc[(size_t)r * n + k]; PHt[(size_t)a * m + r] = s; }
      for (int r = 0; r < m; ++r) for (int q = 0; q < m; ++q) { double s = 0; for (int k = 0; k < n; ++k) s += Hc[(size_t)r * n + k] * PHt[(size_t)k * m + q]; S[(size_t)r * m + q] = s / R + (r == q ? 1.0 : 0.0); }
      inverse_lu(S.data(), m, Sinv.data());
      std::vector<double> K((size_t)n * m);
      for (int a = 0; a < n; ++a) for (int q = 0; q < m; ++q) { double s = 0; for (int r = 0; r < m; ++r) s += PHt[(size_t)a * m + r] * Sinv[(size_t)r * m + q]; K[(size_t)a * m + q] = s / R; }
      for (int a = 0; a < n; ++a) { double s = 0; for (int r = 0; r < m; ++r) s += K[(size_t)a * m + r] * c->h[r]; K_h[a] = s; }
      for (int a = 0; a < n; ++a) for (int b = 0; b < n; ++b) { double s = 0; for (int r = 0; r < m; ++r) s += K[(size_t)a * m + r] * Hc[(size_t)r * n + b]; K_x[(size_t)a * n + b] = s; }
    } else {   // :621-637
      std::vector<double> P_temp((size_t)n * n), P_inv((size_t)n * n), HTH((size_t)ncol * ncol), HTh(ncol);
      inverse_lu(P.data(), n, P_temp.data());
      if (c->fast_reduce) orc_reduce_fast(c, HTH.data(), HTh.data(), nullptr, 0, n, nullptr, nthreads);   // :629 (timing arms)
      else orc_reduce(c, HTH.data(), HTh.data());
      for (int a = 0; a < ncol; ++a) for (int b = 0; b < ncol; ++b) P_temp[(size_t)a * n + b] += HTH[(size_t)a * ncol + b];
      inverse_lu(P_temp.data(), n, P_inv.data());
      if (c->fast_reduce) {   // :635 in the reference's evaluation order: (P_inv.block * HT) * h, a second pass over the rows
        std::vector<double> HTH2((size_t)ncol * ncol), HTh2(ncol), PT((size_t)ncol * n);
        for (int a = 0; a < n; ++a) for (int k = 0; k < ncol; ++k) PT[(size_t)k * n + a] = P_inv[(size_t)a * n + k];
        orc_reduce_fast(c, HTH2.data(), HTh2.data(), PT.data(), n, n, K_h.data(), nthreads);
      } else
      for (int a = 0; a < n; ++a) { double s = 0; for (int k = 0; k < ncol; ++k) s += P_inv[(size_t)a * n + k] * HTh[k]; K_h[a] = s; }
      std::fill(K_x.begin(), K_x.end(), 0.0);
      for (int a = 0; a < n; ++a) for (int b = 0; b < ncol; ++b) { double s = 0; for (int k = 0; k < ncol; ++k) s += P_inv[(size_t)a * n + k] * HTH[(size_t)k * ncol + b]; K_x[(size_t)a * n + b] = s; }
    }
    std::vector<double> dx_(n);   // :642
    for (int a = 0; a < n; ++a) {
      double s = K_h[a];
      for (int b = 0; b < n; ++b) s += (K_x[(size_t)a * n + b] - (a == b ? 1.0 : 0.0)) * dx_new[b];
      dx_[a] = s;
    }
    if (dx_log) std::memcpy(dx_log + (size_t)(i + 1) * n, dx_.data(), n * 8);
    if (rep) { std::memcpy(rep->dx_last, dx_.data(), n * 8); rep->n_eff_last = (uint32_t)dof_Measurement; }
    state_boxplus(ly, *x_, dx_.data());   // :646
    converge = true;   // :649-657
    for (int k = 0; k < n; ++k) if (std::fabs(dx_[k]) > 0.001) { converge = false; break; }
    if (converge) t++;
    if (!t && i == maximum_iter - 2) converge = true;   // :660-663
    if (t > 1 || i == maximum_iter - 1) {   // :665-718
      L_ = P;
      for (int si = 0; si < n_so3; ++si) {
        const int idx = so3_idx[si];
        double A[9], J[9];
        A_matrix(&dx_[idx], A);
        for (int a = 0; a < 3; ++a) for (int b = 0; b < 3; ++b) J[3 * a + b] = A[3 * b + a];
        apply_left3(L_, idx, J, P);   // L_.block<3,1>(idx,i) = J * P_.block<3,1>(idx,i)
        for (int k = 0; k < ncol; ++k) {   // K_x.block<3,1>(idx,k) = J * K_x.block<3,1>(idx,k)
          double v[3] = {K_x[(size_t)idx * n + k], K_x[(size_t)(idx + 1) * n + k], K_x[(size_t)(idx + 2) * n + k]}, o[3];
          m3v(J, v, o);
          for (int q = 0; q < 3; ++q) K_x[(size_t)(idx + q) * n + k] = o[q];
        }
        apply_right3T(L_, idx, J);
        apply_right3T(P, idx, J);
      }
      {
        const int idx = ly.grav;
        double Nx[6], Mx[6], J2[4];
        S2_Nx_yy(x_->grav, Nx);
        S2_Mx(x_propagated.grav, &dx_[idx], Mx);
        for (int a = 0; a < 2; ++a) for (int b = 0; b < 2; ++b) J2[2 * a + b] = Nx[3 * a] * Mx[b] + Nx[3 * a + 1] * Mx[2 + b] + Nx[3 * a + 2] * Mx[4 + b];
        for (int k = 0; k < n; ++k) {
          double a0 = P[(size_t)idx * n + k], a1 = P[(size_t)(idx + 1) * n + k];
          L_[(size_t)idx * n + k] = J2[0] * a0 + J2[1] * a1;
          L_[(size_t)(idx + 1) * n + k] = J2[2] * a0 + J2[3] * a1;
        }
        for (int k = 0; k < ncol; ++k) {
          double a0 = K_x[(size_t)idx * n + k], a1 = K_x[(size_t)(idx + 1) * n + k];
          K_x[(size_t)idx * n + k] = J2[0] * a0 + J2[1] * a1;
          K_x[(size_t)(idx + 1) * n + k] = J2[2] * a0 + J2[3] * a1;
        }
        for (int k = 0; k < n; ++k) {
          double a0 = L_[(size_t)k * n + idx], a1 = L_[(size_t)k * n + idx + 1];
          L_[(size_t)k * n + idx] = a0 * J2[0] + a1 * J2[1];
          L_[(size_t)k * n + idx + 1] = a0 * J2[2] + a1 * J2[3];
          double b0 = P[(size_t)k * n + idx], b1 = P[(size_t)k * n + idx + 1];
          P[(size_t)k * n + idx] = b0 * J2[0] + b1 * J2[1];
          P[(size_t)k * n + idx + 1] = b0 * J2[2] + b1 * J2[3];
        }
      }
      for (int a = 0; a < n; ++a)   // :714
        for (int b = 0; b < n; ++b) {
          double s = 0;
          for (int k = 0; k < ncol; ++k) s += K_x[(size_t)a * n + k] * P[(size_t)k * n + b];
          P_[(size_t)a * n + b] = L_[(size_t)a * n + b] - s;
        }
      if (rep) { rep->passes = passes; rep->searches = searches; rep->converged_count = t; rep->last_status = 0; }
      c->t_A += omp_get_wtime() - t_seg;
      return 0;
    }
  }
  // fell out of the loop (last pass invalid): the reference leaves P_ = P_propagated (or the last :530 value)
  std::memcpy(P_, P.data(), (size_t)n * n * 8);
  c->t_A += omp_get_wtime() - t_seg;
  if (rep) { rep->passes = passes; rep->searches = searches; rep->converged_count = t; rep->last_status = MALIO_ERR_NO_EFFECTIVE_POINTS; }
  return 1;
}

}  // extern "C"
