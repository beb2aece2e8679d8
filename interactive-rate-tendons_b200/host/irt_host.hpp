// irt_host.hpp -- C++ host mirror of the reference's operator interface for the hot path,
// implemented entirely on top of the C ABI (include/irt_b200.h -> libirt_b200.so, CUDA sm_100a).
//
// Same class names, member names, argument meaning and error behaviour as the reference so that
// planner code above the boundary (VoxelCachedLazyPRM's batch loops, apps) reads unchanged:
//
//   tendon::BackboneSpecs / TendonSpecs / TendonResult / TendonRobot
//        tendon/BackboneSpecs.h:15-21, TendonSpecs.h:24-40, TendonResult.h:17-40, TendonRobot.h:52-355
//   collision::VoxelOctree                          collision/VoxelOctree.h:68-330 (value type: block
//        storage + set algebra; voxelisation and collides() run on the GPU)
//   motion_planning::VoxelEnvironment, VoxelBackboneValidityChecker, VoxelBackboneMotionValidator
//        motion-planning/VoxelEnvironment.h:137-167, AbstractVoxelValidityChecker.h:33-52,
//        AbstractVoxelMotionValidator.h:98-135
//   motion_planning::VoxelCachedLazyPRM (batch entry points only)
//        motion-planning/VoxelCachedLazyPRM.h:495-520, .cpp:1563-1782
//
// Status codes are translated back into the reference's exception types:
//   IRT_ERR_INVALID_ARGUMENT -> std::invalid_argument   IRT_ERR_OUT_OF_RANGE -> std::out_of_range
//   IRT_ERR_DOMAIN -> std::domain_error                 everything else -> std::runtime_error
// There is no CPU fallback: without a CUDA device the Context constructor throws.
#pragma once

#include <algorithm>
#include <array>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <functional>
#include <map>
#include <condition_variable>
#include <limits>
#include <memory>
#include <mutex>
#include <optional>
#include <queue>
#include <thread>
#include <random>
#include <set>
#include <stdexcept>
#include <string>
#include <tuple>
#include <utility>
#include <vector>

#include "../../include/irt_b200.h"
#ifdef IRT_TEST_OVER_STANDIN
// built over the test-only stand-in of the C ABI (no GPU): irt_nnset_* come from a sequential host implementation,
// irt_setstore_append from the stand-in's export / import, irt_check_sets_changed from export + host comparison
#include "../../tests/cpp/knn_standin.hpp"
#include "../../tests/cpp/setstore_append_standin.hpp"
#include "../../tests/cpp/env_delta_standin.hpp"
#endif

namespace irt {

inline void check(irt_ctx *ctx, int rc) {
  if (rc == IRT_OK) return;
  std::string msg = std::string(irt_status_string(rc)) + ": " + (ctx ? irt_last_error(ctx) : "");
  switch (rc) {
    case IRT_ERR_INVALID_ARGUMENT: throw std::invalid_argument(msg);
    case IRT_ERR_OUT_OF_RANGE: throw std::out_of_range(msg);
    case IRT_ERR_DOMAIN: throw std::domain_error(msg);
    default: throw std::runtime_error(msg);
  }
}

/// one CUDA device + stream; shared by every mirrored object
class Context {
public:
  explicit Context(int device = 0) {
    int rc = irt_ctx_create(device, &ctx_);
    if (rc != IRT_OK) throw std::runtime_error(std::string("irt_b200: ") + irt_status_string(rc));
  }
  ~Context() { irt_ctx_destroy(ctx_); }
  Context(const Context &) = delete;
  Context &operator=(const Context &) = delete;
  irt_ctx *get() const { return ctx_; }
  static std::shared_ptr<Context> &global() {
    static std::shared_ptr<Context> g;
    if (!g) g = std::make_shared<Context>(0);
    return g;
  }

private:
  irt_ctx *ctx_ = nullptr;
};

}  // namespace irt

namespace collision {
using Point = std::array<double, 3>;
}

namespace tendon {

struct BackboneSpecs {  // tendon/BackboneSpecs.h:15-21
  double L = 0.2, dL = 0.005, ro = 0.01, ri = 0.0, E = 2.1e6, nu = 0.3;
};

struct TendonSpecs {  // tendon/TendonSpecs.h:24-40
  std::vector<double> C, D;
  double max_tension = 20.0, min_length = -0.015, max_length = 0.035;
  static size_t poly_degree(const std::vector<double> &c, double eps) {  // TendonSpecs.cpp:17-25
    if (c.empty()) return 0;
    for (size_t i = c.size() - 1; i > 0; i--)
      if (std::abs(c[i]) > eps) return i;
    return 0;
  }
  size_t r_degree(double eps = 0.0) const { return poly_degree(D, eps); }
  size_t theta_degree(double eps = 0.0) const { return poly_degree(C, eps); }
  bool is_straight(double eps = 0.0) const { return r_degree(eps) == 0 && theta_degree(eps) == 0; }
  bool is_helix(double eps = 0.0) const { return r_degree(eps) == 0 && theta_degree(eps) == 1; }
};

struct TendonResult {  // tendon/TendonResult.h:17-40
  std::vector<double> t;
  std::vector<collision::Point> p;
  std::vector<std::array<double, 9>> R;  // column-major 3x3, like Eigen::Matrix3d storage
  double L = 0.0;
  std::vector<double> L_i;
  std::array<double, 3> u_i{0, 0, 0}, u_f{0, 0, 0}, v_i{0, 0, 1}, v_f{0, 0, 1};
  bool converged = true;
  /// device-computed validity word of this shape (IRT_FLAG_*); not a reference member
  uint32_t flags = 0;

  void rotate_z(double theta) {  // tendon/TendonResult.cpp:13-18
    const double c = std::cos(theta), s = std::sin(theta);
    for (auto &q : p) q = {c * q[0] - s * q[1], s * q[0] + c * q[1], q[2]};
    for (auto &m : R)
      for (int j = 0; j < 3; j++) {
        const double a = m[3 * j], b = m[3 * j + 1];
        m[3 * j] = c * a - s * b;
        m[3 * j + 1] = s * a + c * b;
      }
  }
};

struct TendonRobot {  // tendon/TendonRobot.h:52-355
  double r = 0.015;
  BackboneSpecs specs{};
  std::vector<TendonSpecs> tendons;
  bool enable_rotation = false, enable_retraction = false;
  double residual_threshold = 5e-6;

  size_t state_size() const { return tendons.size() + (enable_rotation ? 1 : 0) + (enable_retraction ? 1 : 0); }

  irt_robot_desc desc() const {
    irt_robot_desc d;
    std::memset(&d, 0, sizeof(d));
    d.r = r; d.L = specs.L; d.dL = specs.dL; d.ro = specs.ro; d.ri = specs.ri; d.E = specs.E; d.nu = specs.nu;
    d.residual_threshold = residual_threshold;
    if (tendons.size() > IRT_MAX_TENDONS) throw std::out_of_range("too many tendons");
    d.n_tendons = (int32_t)tendons.size();
    d.n_c = tendons.empty() ? 0 : (int32_t)tendons[0].C.size();
    d.n_d = tendons.empty() ? 0 : (int32_t)tendons[0].D.size();
    if (d.n_c > IRT_MAX_COEF || d.n_d > IRT_MAX_COEF) throw std::out_of_range("too many coefficients");
    for (size_t j = 0; j < tendons.size(); j++) {
      // get_r_info.h:34-39: every tendon is evaluated with tendon 0's coefficient counts
      for (int i = 0; i < d.n_c && i < (int)tendons[j].C.size(); i++) d.C[j * IRT_MAX_COEF + i] = tendons[j].C[i];
      for (int i = 0; i < d.n_d && i < (int)tendons[j].D.size(); i++) d.D[j * IRT_MAX_COEF + i] = tendons[j].D[i];
      d.max_tension[j] = tendons[j].max_tension;
      d.min_length[j] = tendons[j].min_length;
      d.max_length[j] = tendons[j].max_length;
    }
    d.enable_rotation = enable_rotation ? 1 : 0;
    d.enable_retraction = enable_retraction ? 1 : 0;
    return d;
  }

  /// device handle (robot constants + routing tables), rebuilt when the description changes
  irt_robot *handle() const {
    irt_robot_desc d = desc();
    if (!dev_ || std::memcmp(&d, &cached_, sizeof(d)) != 0) {
      ctx_ = irt::Context::global();
      irt_robot *h = nullptr;
      irt::check(ctx_->get(), irt_robot_create(ctx_->get(), &d, &h));
      dev_ = std::shared_ptr<irt_robot>(h, [](irt_robot *x) { irt_robot_destroy(x); });
      cached_ = d;
    }
    return dev_.get();
  }
  irt_ctx *ctx() const { handle(); return ctx_->get(); }

  /// TendonRobot::shape for a batch (the OpenMP loops of apps/estimate_length_discretization.cpp:62-71)
  std::vector<TendonResult> shape_batch(const std::vector<std::vector<double>> &states) const {
    const size_t S = state_size(), n = states.size(), N = tendons.size();
    for (auto &s : states)
      if (s.size() != S) throw std::invalid_argument("State is not the right size");  // TendonRobot.h:107-109
    irt_robot *h = handle();
    const int cap = irt_robot_max_points(h);
    std::vector<double> flat(n * S), p(n * cap * 3), R(n * cap * 9), t(n * cap), L(n), Li(n * N), uv(n * 12);
    std::vector<int32_t> npts(n);
    std::vector<uint32_t> flags(n);
    for (size_t i = 0; i < n; i++) std::copy(states[i].begin(), states[i].end(), flat.begin() + i * S);
    irt_fk_outputs o;
    std::memset(&o, 0, sizeof(o));
    o.p = p.data(); o.R = R.data(); o.t = t.data(); o.npts = npts.data(); o.L = L.data();
    o.L_i = Li.data(); o.uv = uv.data(); o.flags = flags.data();
    irt::check(ctx_->get(), irt_fk_batch(ctx_->get(), h, flat.data(), (int)S, (int64_t)n, cap, &o));
    std::vector<TendonResult> out(n);
    for (size_t i = 0; i < n; i++) {
      TendonResult &r = out[i];
      const int m = npts[i];
      r.t.assign(t.begin() + i * cap, t.begin() + i * cap + m);
      r.p.resize(m); r.R.resize(m);
      for (int k = 0; k < m; k++) {
        std::memcpy(r.p[k].data(), &p[(i * cap + k) * 3], 24);
        std::memcpy(r.R[k].data(), &R[(i * cap + k) * 9], 72);
      }
      r.L = L[i];
      r.L_i.assign(Li.begin() + i * N, Li.begin() + (i + 1) * N);
      for (int c = 0; c < 3; c++) {
        r.u_i[c] = uv[i * 12 + c]; r.u_f[c] = uv[i * 12 + 3 + c];
        r.v_i[c] = uv[i * 12 + 6 + c]; r.v_f[c] = uv[i * 12 + 9 + c];
      }
      r.flags = flags[i];
      r.converged = !(flags[i] & IRT_FLAG_NONCONVERGED);
    }
    return out;
  }

  TendonResult shape(const std::vector<double> &state) const { return shape_batch({state})[0]; }
  TendonResult shape(const std::vector<double> &tau, double rotation, double retraction) const {
    if (tau.size() != tendons.size()) throw std::out_of_range("tendons and tau are not the same length");
    std::vector<double> st(tau);
    if (enable_rotation) st.push_back(rotation);
    if (enable_retraction) st.push_back(retraction);
    return shape(st);
  }
  std::vector<collision::Point> forward_kinematics(const std::vector<double> &state) const { return shape(state).p; }

  /// random_state (tendon/TendonRobot.cpp:219-247): tensions U[0, max_tension], rotation U[-pi, pi],
  /// retraction U[0, L], in state order.  The generator overload is what a seeded caller uses; the
  /// argument-free form keeps the reference's thread-local std::mt19937 seeded from std::random_device.
  template <class Generator>
  std::vector<double> random_state(Generator &generator) const {
    std::vector<double> state;
    for (auto &tendon : tendons) {
      std::uniform_real_distribution<double> dist(0.0, tendon.max_tension);
      state.push_back(dist(generator));
    }
    if (enable_rotation) {
      std::uniform_real_distribution<double> dist(-M_PI, M_PI);
      state.push_back(dist(generator));
    }
    if (enable_retraction) {
      std::uniform_real_distribution<double> dist(0.0, specs.L);
      state.push_back(dist(generator));
    }
    return state;
  }
  std::vector<double> random_state() const {
    static thread_local std::mt19937 generator{std::random_device{}()};
    return random_state(generator);
  }

  /// home_shape (tendon/TendonRobot.cpp:249-314): straight backbone, closed-form tendon lengths
  TendonResult home_shape(double s_start = 0) const {
    if (s_start < 0.0) s_start = 0.0;
    if (s_start > specs.L) s_start = specs.L;
    std::vector<double> st(state_size(), 0.0);
    const bool had_ret = enable_retraction;
    TendonResult res;
    if (had_ret) {
      st.back() = s_start;
      res = shape(st);  // zero tension == home shape
    } else {
      TendonRobot tmp = *this;
      tmp.enable_retraction = true;
      tmp.dev_.reset();
      st.push_back(s_start);
      res = tmp.shape(st);
    }
    std::vector<double> home(tendons.size());
    std::vector<double> one(state_size(), 0.0);
    if (enable_retraction) one.back() = s_start;
    irt::check(ctx(), irt_home_lengths_batch(ctx(), handle(), one.data(), (int)state_size(), 1, home.data()));
    if (!enable_retraction)
      for (auto &h : home) h *= (s_start == specs.L) ? 0.0 : (specs.L - s_start) / specs.L;
    res.L_i = home;
    return res;
  }
  TendonResult home_shape(const std::vector<double> &state) const {
    return home_shape(enable_retraction ? state.back() : 0.0);
  }

  std::vector<double> calc_dl(const std::vector<double> &home_l, const std::vector<double> &other_l) const {
    if (home_l.size() != other_l.size()) throw std::out_of_range("vector size mismatch");
    std::vector<double> dl(home_l.size());
    for (size_t i = 0; i < dl.size(); i++) dl[i] = home_l[i] - other_l[i];
    return dl;
  }
  bool is_within_length_limits(const std::vector<double> &dl) const {
    if (dl.size() != tendons.size()) throw std::out_of_range("length mismatch");
    for (size_t i = 0; i < dl.size(); i++)
      if (dl[i] < tendons[i].min_length || tendons[i].max_length < dl[i]) return false;
    return true;
  }
  bool is_within_length_limits(const std::vector<double> &home_l, const std::vector<double> &other_l) const {
    return is_within_length_limits(calc_dl(home_l, other_l));
  }
  /// collides_self of a shape computed by this robot (device verdict carried in TendonResult::flags)
  bool collides_self(const TendonResult &shape_) const { return (shape_.flags & IRT_FLAG_SELF_COLLISION) != 0; }
  bool is_valid(const std::vector<double> &state, const TendonResult &, const TendonResult &shape_) const {
    if (shape_.flags & IRT_FLAG_LENGTH_LIMIT) return false;
    for (size_t i = 0; i < tendons.size(); i++)
      if (state[i] < 0.0 || tendons[i].max_tension < state[i]) return false;
    return !collides_self(shape_);
  }

private:
  mutable std::shared_ptr<irt::Context> ctx_;
  mutable std::shared_ptr<irt_robot> dev_;
  mutable irt_robot_desc cached_;
};

}  // namespace tendon

/// Batched forms of the finite-difference Jacobians behind the reference's IK and tip controllers
/// (SURVEY 8(f) row 3).  J of seed k is returned row-major 3 x S (J[i * S + j] = d tip_i / d state_j).
namespace tip_control {

/// tip_control::Jacobian (tip-control/tip_control.cpp:243-265) for many states at once:
/// forward difference with the fixed step `dist` from ps = forward_kinematics(state).back()
inline std::vector<std::vector<double>> Jacobian_batch(const tendon::TendonRobot &robot, double dist,
                                                       const std::vector<std::vector<double>> &states,
                                                       std::vector<collision::Point> *tips = nullptr,
                                                       int mode = IRT_JAC_FORWARD_FIXED) {
  const size_t S = robot.state_size(), n = states.size();
  for (auto &st : states)
    if (st.size() != S) throw std::invalid_argument("State is not the right size");
  std::vector<double> flat(n * S), tip(n * 3), J(n * 3 * S);
  for (size_t i = 0; i < n; i++) std::copy(states[i].begin(), states[i].end(), flat.begin() + i * S);
  irt::check(robot.ctx(), irt_fk_tip_jacobian_batch(robot.ctx(), robot.handle(), flat.data(), (int)S,
                                                    (int64_t)n, mode, dist, tip.data(), J.data()));
  std::vector<std::vector<double>> out(n);
  for (size_t i = 0; i < n; i++) out[i].assign(J.begin() + i * 3 * S, J.begin() + (i + 1) * 3 * S);
  if (tips) {
    tips->resize(n);
    for (size_t i = 0; i < n; i++) (*tips)[i] = {tip[3 * i], tip[3 * i + 1], tip[3 * i + 2]};
  }
  return out;
}

/// tip_control::Jacobian with the reference's own signature (tip_control.cpp:243-265): forward differences
/// from the CALLER'S ps with a step that is a C `float` (tau[i] + dist and the division promote it to
/// double, so the step really taken is double(float(dist))).  One FK batch of S perturbed states; J is
/// returned row-major 3 x S (the reference returns an Eigen::MatrixXd with J(j, i) at the same place).
/// For the batched form above pass double(float(dist)) to take the same step.
inline std::vector<double> Jacobian(const tendon::TendonRobot &robot, const collision::Point &ps, float dist,
                                    const std::vector<double> &tau) {
  const size_t S = tau.size();
  std::vector<std::vector<double>> pert(S, tau);
  for (size_t i = 0; i < S; i++) pert[i][i] = tau[i] + dist;
  auto shapes = robot.shape_batch(pert);
  std::vector<double> J(3 * S);
  for (size_t i = 0; i < S; i++) {
    const collision::Point pos = shapes[i].p.back();
    for (size_t j = 0; j < 3; j++) J[j * S + i] = (pos[j] - ps[j]) / dist;
  }
  return J;
}

/// the Jacobian levmar's dlevmar_bc_dif builds inside tip_control::inverse_kinematics
/// (central differences, d = max(|1e-4 p_j|, delta); tip_control.cpp:85, levmar-2.6 misc_core.c:175-211)
inline std::vector<std::vector<double>> levmar_jacobian_batch(const tendon::TendonRobot &robot, double delta,
                                                              const std::vector<std::vector<double>> &states,
                                                              std::vector<collision::Point> *tips = nullptr) {
  return Jacobian_batch(robot, delta, states, tips, IRT_JAC_LEVMAR_CENTRAL);
}

/// Batching layer under k IK solvers that run side by side (SURVEY 8(f) row 3): every solver asks for the tip and the
/// finite-difference tip Jacobian of ONE state at a time, like the reference's ikController_ does through fk_wrap
/// (tip-control/tip_control.cpp:92-122); the requests of all solvers that are still running are answered by ONE
/// irt_fk_tip_jacobian_batch call.  The solvers stay sequential host code, one thread each.
class LockstepFk {
public:
  struct Eval { collision::Point tip; std::vector<double> J; };   // J row-major 3 x S
  LockstepFk(const tendon::TendonRobot &robot, size_t workers, int mode, double delta)
      : robot_(robot), mode_(mode), delta_(delta), active_(workers), results_(workers), asked_(workers, 0) {}
  Eval evaluate(size_t worker, const std::vector<double> &state) {
    std::unique_lock<std::mutex> lk(mu_);
    pending_.emplace_back(worker, state);
    const size_t gen = generation_;
    if (pending_.size() == active_) flush();
    else cv_.wait(lk, [&] { return generation_ != gen; });
    return results_[worker];
  }
  void finished(size_t) {
    std::unique_lock<std::mutex> lk(mu_);
    active_--;
    if (active_ > 0 && pending_.size() == active_) flush();
  }
  size_t batches() const { return batches_; }
  size_t requests() const { return requests_; }

private:
  void flush() {   // lock held
    std::vector<std::vector<double>> states;
    for (auto &p : pending_) states.push_back(p.second);
    std::vector<collision::Point> tips;
    auto Js = Jacobian_batch(robot_, delta_, states, &tips, mode_);
    for (size_t i = 0; i < pending_.size(); i++) results_[pending_[i].first] = Eval{tips[i], Js[i]};
    requests_ += pending_.size();
    batches_++;
    pending_.clear();
    generation_++;
    cv_.notify_all();
  }
  const tendon::TendonRobot &robot_;
  int mode_;
  double delta_;
  size_t active_;
  std::vector<Eval> results_;
  std::vector<char> asked_;
  std::vector<std::pair<size_t, std::vector<double>>> pending_;
  std::mutex mu_;
  std::condition_variable cv_;
  size_t generation_ = 0, batches_ = 0, requests_ = 0;
};

/// the reference's ikController_: (start state, requested tip, fk) -> final state; fk(state) -> tip + Jacobian
using IkSolver = std::function<std::vector<double>(const std::vector<double> &, const collision::Point &,
                                                   const std::function<LockstepFk::Eval(const std::vector<double> &)> &)>;

/// runs the solver for every start state side by side (one host thread each), FK requests answered in lockstep
inline std::vector<std::vector<double>> solve_ik_lockstep(const tendon::TendonRobot &robot, const IkSolver &solver,
                                                          const std::vector<std::vector<double>> &starts,
                                                          const collision::Point &request, int mode, double delta,
                                                          size_t *batches = nullptr, size_t *requests = nullptr) {
  const size_t k = starts.size();
  LockstepFk fk(robot, k, mode, delta);
  std::vector<std::vector<double>> out(k);
  std::vector<std::exception_ptr> err(k);
  std::vector<std::thread> th;
  for (size_t i = 0; i < k; i++)
    th.emplace_back([&, i] {
      try {
        out[i] = solver(starts[i], request, [&fk, i](const std::vector<double> &st) { return fk.evaluate(i, st); });
      } catch (...) {
        err[i] = std::current_exception();   // a failing solver must not leave the others waiting for it
      }
      fk.finished(i);
    });
  for (auto &t : th) t.join();
  for (auto &e : err)
    if (e) std::rethrow_exception(e);
  if (batches) *batches = fk.batches();
  if (requests) *requests = fk.requests();
  return out;
}

}  // namespace tip_control

namespace collision {

struct Sphere {  // collision/Sphere.h
  Point c;
  double r;
};
struct Capsule {  // collision/Capsule.h
  Point a, b;
  double r;
};

/// Value-type mirror of collision::VoxelOctree: the sparse set of occupied 4x4x4 leaf blocks.
/// Storage is a key-ordered map (Morton key == the reference's visit_leaves order); the heavy
/// operations (voxelising shapes, collides) go through the C ABI.
class VoxelOctree {
public:
  using BlockType = uint64_t;
  using ConstBlockVisitor = std::function<void(size_t, size_t, size_t, uint64_t)>;

  explicit VoxelOctree(size_t Ndim = 4) : N_(Ndim) {
    // collision/VoxelOctree.cpp:83-116
    if (Ndim < 4 || Ndim > 512 || (Ndim & (Ndim - 1)))
      throw std::invalid_argument("unsupported voxel dimension: " + std::to_string(Ndim));
    set_xlim(0.0, 1.0); set_ylim(0.0, 1.0); set_zlim(0.0, 1.0);
  }
  size_t Nx() const { return N_; }
  size_t Ny() const { return N_; }
  size_t Nz() const { return N_; }
  size_t Nbx() const { return N_ / 4; }
  void set_xlim(double a, double b) { lim_check(a, b); lim_[0] = a; lim_[1] = b; }
  void set_ylim(double a, double b) { lim_check(a, b); lim_[2] = a; lim_[3] = b; }
  void set_zlim(double a, double b) { lim_check(a, b); lim_[4] = a; lim_[5] = b; }
  std::pair<double, double> xlim() const { return {lim_[0], lim_[1]}; }
  std::pair<double, double> ylim() const { return {lim_[2], lim_[3]}; }
  std::pair<double, double> zlim() const { return {lim_[4], lim_[5]}; }
  double dx() const { return (lim_[1] - lim_[0]) / N_; }
  double dy() const { return (lim_[3] - lim_[2]) / N_; }
  double dz() const { return (lim_[5] - lim_[4]) / N_; }
  void copy_limits(const VoxelOctree &o) { lim_ = o.lim_; }
  VoxelOctree empty_copy() const { VoxelOctree c(N_); c.lim_ = lim_; return c; }
  bool is_empty() const { return blocks_.empty(); }
  size_t nblocks() const { return blocks_.size(); }
  size_t ncells() const {
    size_t c = 0;
    for (auto &kv : blocks_) c += (size_t)__builtin_popcountll(kv.second);
    return c;
  }
  uint64_t block(size_t bx, size_t by, size_t bz) const {
    auto it = blocks_.find(key(bx, by, bz));
    return it == blocks_.end() ? 0 : it->second;
  }
  void set_block(size_t bx, size_t by, size_t bz, uint64_t v) {
    if (v) blocks_[key(bx, by, bz)] = v; else blocks_.erase(key(bx, by, bz));
  }
  uint64_t union_block(size_t bx, size_t by, size_t bz, uint64_t v) {
    uint64_t old = block(bx, by, bz);
    if (v) blocks_[key(bx, by, bz)] = old | v;
    return old;
  }
  bool cell(size_t ix, size_t iy, size_t iz) const {
    return (block(ix / 4, iy / 4, iz / 4) >> ((ix % 4) * 16 + (iy % 4) * 4 + (iz % 4))) & 1u;
  }
  void add_voxels(const VoxelOctree &o) {
    check_dims(o);
    for (auto &kv : o.blocks_) blocks_[kv.first] |= kv.second;
  }
  void visit_leaves(const ConstBlockVisitor &f) const {
    for (auto &kv : blocks_) {
      int bx, by, bz;
      irt_morton_decode(kv.first, (int)(N_ / 4), &bx, &by, &bz);
      f((size_t)bx, (size_t)by, (size_t)bz, kv.second);
    }
  }
  bool operator==(const VoxelOctree &o) const { return N_ == o.N_ && lim_ == o.lim_ && blocks_ == o.blocks_; }

  // ---- the rest of the reference's value-type surface (collision/VoxelOctree.h:91-290), host side ----
  using ConstOccupiedVoxelVisitor = std::function<void(size_t, size_t, size_t)>;
  using ConstVoxelVisitor = std::function<void(size_t, size_t, size_t, bool)>;
  static size_t largest_supported_size() { return 512; }
  static size_t to_supported_size(size_t Ndim) {  // VoxelOctree.cpp:82-96
    for (size_t n = 4; n <= 512; n *= 2)
      if (Ndim <= n) return n;
    throw std::invalid_argument("too large for supported voxel octree: " + std::to_string(Ndim));
  }
  static uint64_t bitmask(size_t x, size_t y, size_t z) { return uint64_t(1) << (x * 16 + y * 4 + z); }
  size_t N() const { return N_ * N_ * N_; }
  size_t Nby() const { return N_ / 4; }
  size_t Nbz() const { return N_ / 4; }
  void set_xlim(const std::pair<double, double> &l) { set_xlim(l.first, l.second); }
  void set_ylim(const std::pair<double, double> &l) { set_ylim(l.first, l.second); }
  void set_zlim(const std::pair<double, double> &l) { set_zlim(l.first, l.second); }
  Point lower_left() const { return {lim_[0], lim_[2], lim_[4]}; }
  Point upper_right() const { return {lim_[1], lim_[3], lim_[5]}; }
  double dbx() const { return dx() * 4; }
  double dby() const { return dy() * 4; }
  double dbz() const { return dz() * 4; }
  bool is_in_domain(double x, double y, double z) const {  // inclusive on both ends, VoxelOctree.cpp:1505-1509
    return lim_[0] <= x && x <= lim_[1] && lim_[2] <= y && y <= lim_[3] && lim_[4] <= z && z <= lim_[5];
  }
  Point voxel_center(size_t ix, size_t iy, size_t iz) const {
    return {lim_[0] + (ix + 0.5) * dx(), lim_[2] + (iy + 0.5) * dy(), lim_[4] + (iz + 0.5) * dz()};
  }
  Point block_center(size_t bx, size_t by, size_t bz) const {
    return {lim_[0] + (bx + 0.5) * dbx(), lim_[2] + (by + 0.5) * dby(), lim_[4] + (bz + 0.5) * dbz()};
  }
  /// returns the block's value before the operation, like the reference (VoxelOctree.cpp:235-249)
  uint64_t intersect_block(size_t bx, size_t by, size_t bz, uint64_t v) {
    const uint64_t old = block(bx, by, bz);
    set_block(bx, by, bz, old & v);
    return old;
  }
  uint64_t subtract_block(size_t bx, size_t by, size_t bz, uint64_t v) { return intersect_block(bx, by, bz, ~v); }
  /// VoxelOctree.cpp:256-267 as written: the return value is `oldval & mask` when setting and
  /// `oldval & ~mask` when clearing (not "did the cell change", whatever its comment says)
  bool set_cell(size_t ix, size_t iy, size_t iz, bool value = true) {
    const uint64_t mask = bitmask(ix % 4, iy % 4, iz % 4);
    if (value) return union_block(ix / 4, iy / 4, iz / 4, mask) & mask;
    return intersect_block(ix / 4, iy / 4, iz / 4, ~mask) & ~mask;
  }
  std::tuple<size_t, size_t, size_t> nearest_cell(double x, double y, double z) const {  // bounds truncating, :295-307
    const int ix = (int)((x - lim_[0]) / dx()), iy = (int)((y - lim_[2]) / dy()), iz = (int)((z - lim_[4]) / dz());
    return {std::min(N_ - 1, size_t(std::max(0, ix))), std::min(N_ - 1, size_t(std::max(0, iy))),
            std::min(N_ - 1, size_t(std::max(0, iz)))};
  }
  std::tuple<size_t, size_t, size_t> find_cell(double x, double y, double z) const {  // bounds checking, :309-317
    domain_check(x, y, z);
    return {size_t((x - lim_[0]) / dx()), size_t((y - lim_[2]) / dy()), size_t((z - lim_[4]) / dz())};
  }
  std::tuple<size_t, size_t, size_t> nearest_block_idx(double x, double y, double z) const {  // :271-282
    const int ix = (int)((x - lim_[0]) / dx()), iy = (int)((y - lim_[2]) / dy()), iz = (int)((z - lim_[4]) / dz());
    return {std::min(N_ / 4 - 1, size_t(std::max(0, ix / 4))), std::min(N_ / 4 - 1, size_t(std::max(0, iy / 4))),
            std::min(N_ / 4 - 1, size_t(std::max(0, iz / 4)))};
  }
  std::tuple<size_t, size_t, size_t> find_block_idx(double x, double y, double z) const {  // :284-293
    auto [ix, iy, iz] = find_cell(x, y, z);
    return {ix / 4, iy / 4, iz / 4};
  }
  uint64_t find_block(double x, double y, double z) const {
    auto [bx, by, bz] = find_block_idx(x, y, z);
    return block(bx, by, bz);
  }
  std::tuple<size_t, size_t, size_t> nearest_cell(const Point &p) const { return nearest_cell(p[0], p[1], p[2]); }
  std::tuple<size_t, size_t, size_t> find_cell(const Point &p) const { return find_cell(p[0], p[1], p[2]); }
  std::tuple<size_t, size_t, size_t> nearest_block_idx(const Point &p) const { return nearest_block_idx(p[0], p[1], p[2]); }
  std::tuple<size_t, size_t, size_t> find_block_idx(const Point &p) const { return find_block_idx(p[0], p[1], p[2]); }
  uint64_t find_block(const Point &p) const { return find_block(p[0], p[1], p[2]); }
  bool collides(const Point &p) const {  // :967-971
    if (!is_in_domain(p[0], p[1], p[2])) return false;
    auto [ix, iy, iz] = nearest_cell(p);
    return cell(ix, iy, iz);
  }
  void add(const VoxelOctree &o) { add_voxels(o); }
  void remove_point(double x, double y, double z) {  // :980-984
    if (!is_in_domain(x, y, z)) return;
    auto [ix, iy, iz] = nearest_cell(x, y, z);
    set_cell(ix, iy, iz, false);
  }
  void remove_point(const Point &p) { remove_point(p[0], p[1], p[2]); }
  void remove_voxels(const VoxelOctree &o) {  // :986-990
    check_dims(o);
    for (auto &kv : o.blocks_) {
      auto it = blocks_.find(kv.first);
      if (it != blocks_.end() && !(it->second &= ~kv.second)) blocks_.erase(it);
    }
  }
  void remove(const Point &p) { remove_point(p); }
  void remove(const VoxelOctree &o) { remove_voxels(o); }
  void intersect_voxels(const VoxelOctree &o) {  // :992-996
    check_dims(o);
    for (auto it = blocks_.begin(); it != blocks_.end();) {
      auto jt = o.blocks_.find(it->first);
      const uint64_t v = jt == o.blocks_.end() ? 0 : (it->second & jt->second);
      if (v) { it->second = v; ++it; } else { it = blocks_.erase(it); }
    }
  }
  void intersect(const VoxelOctree &o) { intersect_voxels(o); }
  /// TreeNode::visit_blocks (detail/TreeNode.hxx:193-208, :270): octant recursion; an absent child is
  /// reported ONCE, at its origin block, with value 0
  void visit_blocks(const ConstBlockVisitor &f) const {
    if (N_ == 4) { f(0, 0, 0, block(0, 0, 0)); return; }
    visit_blocks_impl(f, 0u, N_ / 4);
  }
  void visit_occupied_voxels(const ConstOccupiedVoxelVisitor &f) const {  // :1013-1033
    visit_leaves([&](size_t bx, size_t by, size_t bz, uint64_t b) {
      for (size_t x = 0; x < 4; x++)
        for (size_t y = 0; y < 4; y++)
          for (size_t z = 0; z < 4; z++)
            if (b & bitmask(x, y, z)) f(4 * bx + x, 4 * by + y, 4 * bz + z);
    });
  }
  void visit_voxels(const ConstVoxelVisitor &f) const {  // :1035-1052
    visit_blocks([&](size_t bx, size_t by, size_t bz, uint64_t b) {
      for (size_t x = 0; x < 4; x++)
        for (size_t y = 0; y < 4; y++)
          for (size_t z = 0; z < 4; z++) f(4 * bx + x, 4 * by + y, 4 * bz + z, (b & bitmask(x, y, z)) != 0);
    });
  }
  void add_line(const Point &a, const Point &b) { add_piecewise_line({a, b}); }  // one segment of :428-432
  void erode_6neighbor() { throw std::runtime_error("erode_6neighbor() unimplemented"); }   // as in the reference,
  void erode_27neighbor() { throw std::runtime_error("erode_27neighbor() unimplemented"); } // :954-965
  void erode(bool use_diagonal = false) { use_diagonal ? erode_27neighbor() : erode_6neighbor(); }
  void erode_sphere(double) { throw std::runtime_error("erode_sphere() unimplemented"); }

  irt_grid grid(const std::array<double, 9> &inv_rot = {1, 0, 0, 0, 1, 0, 0, 0, 1}) const {
    irt_grid g;
    std::memset(&g, 0, sizeof(g));
    g.Ng = (int32_t)N_;
    for (int i = 0; i < 6; i++) g.lim[i] = lim_[i];
    for (int i = 0; i < 9; i++) g.inv_rot[i] = inv_rot[i];
    return g;
  }

  /// voxels of a backbone polyline: add_piecewise_line (collision/VoxelOctree.cpp:428-432), on the GPU
  void add_piecewise_line(const std::vector<Point> &line) {
    auto ctx = irt::Context::global();
    irt_grid g = grid();
    irt_setstore *st = nullptr;
    irt::check(ctx->get(), irt_setstore_create(ctx->get(), &g, &st));
    std::shared_ptr<irt_setstore> guard(st, [](irt_setstore *x) { irt_setstore_destroy(x); });
    int32_t n = (int32_t)line.size();
    std::vector<double> flat(3 * std::max<size_t>(1, line.size()));
    for (size_t i = 0; i < line.size(); i++) std::memcpy(&flat[3 * i], line[i].data(), 24);
    irt::check(ctx->get(), irt_voxelize_shapes(ctx->get(), flat.data(), &n, std::max(1, (int)line.size()), 1, st));
    merge_store(ctx->get(), st, 0);
  }

  /// collides(other): VoxelOctree.cpp:973-978, K3 on the GPU (this = environment, other = set)
  bool collides(const VoxelOctree &other) const {
    check_dims(other);  // std::invalid_argument on mismatch (VoxelOctree.cpp:46-53)
    auto ctx = irt::Context::global();
    irt_grid g = grid();
    irt_env *env = nullptr;
    irt::check(ctx->get(), irt_env_create(ctx->get(), &g, &env));
    std::shared_ptr<irt_env> eg(env, [](irt_env *x) { irt_env_destroy(x); });
    upload_env(ctx->get(), env);
    irt_setstore *st = nullptr;
    irt::check(ctx->get(), irt_setstore_create(ctx->get(), &g, &st));
    std::shared_ptr<irt_setstore> sg(st, [](irt_setstore *x) { irt_setstore_destroy(x); });
    other.to_store(ctx->get(), st);
    uint32_t word = 0;
    irt::check(ctx->get(), irt_check_sets(ctx->get(), st, env, 0, 1, &word));
    return word & 1u;
  }

  /// environment preparation (collision/VoxelOctree.cpp:533-952; VoxelOctree.h:155-201), on the GPU:
  /// upload, morph in place on the device grid, read the dense grid back
  /// add(Point) / add_sphere / add_capsule (collision/VoxelOctree.cpp:319-323, 434-515; VoxelOctree.h:240-242): a
  /// voxel is set when its centre is inside the object; on the GPU, like every other bulk operation here
  void add_point(const Point &p) { add_primitives({p}, {}, {}); }
  void add(const Point &p) { add_point(p); }
  void add_sphere(const Sphere &s) { add_primitives({}, {s}, {}); }
  void add(const Sphere &s) { add_sphere(s); }
  void add_capsule(const Capsule &c) { add_primitives({}, {}, {c}); }
  void add(const Capsule &c) { add_capsule(c); }
  /// all objects of an Environment in ONE device call (Environment::voxelize, Environment.cpp:62-74)
  void add_primitives(const std::vector<Point> &points, const std::vector<Sphere> &spheres,
                      const std::vector<Capsule> &capsules) {
    std::vector<double> p, s, c;
    for (auto &q : points) p.insert(p.end(), q.begin(), q.end());
    for (auto &q : spheres) { s.insert(s.end(), q.c.begin(), q.c.end()); s.push_back(q.r); }
    for (auto &q : capsules) {
      c.insert(c.end(), q.a.begin(), q.a.end()); c.insert(c.end(), q.b.begin(), q.b.end()); c.push_back(q.r);
    }
    on_device([&](irt_ctx *cx, irt_env *e) {
      return irt_env_add_primitives(cx, e, p.data(), (int64_t)points.size(), s.data(), (int64_t)spheres.size(),
                                    c.data(), (int64_t)capsules.size(), 0);
    });
  }

  void dilate_6neighbor(int num = 1) { on_device([&](irt_ctx *c, irt_env *e) { return irt_env_dilate(c, e, num, 0); }); }
  void dilate_27neighbor(int num = 1) { on_device([&](irt_ctx *c, irt_env *e) { return irt_env_dilate(c, e, num, 1); }); }
  void dilate(int num = 1, bool use_diagonal = false) { use_diagonal ? dilate_27neighbor(num) : dilate_6neighbor(num); }
  void dilate_sphere(double r) { on_device([&](irt_ctx *c, irt_env *e) { return irt_env_dilate_sphere(c, e, r); }); }
  void remove_interior_6neighbor() { on_device([&](irt_ctx *c, irt_env *e) { return irt_env_remove_interior(c, e, 0); }); }
  void remove_interior_27neighbor() { on_device([&](irt_ctx *c, irt_env *e) { return irt_env_remove_interior(c, e, 1); }); }
  void remove_interior(bool keep_diagonal = true) { keep_diagonal ? remove_interior_27neighbor() : remove_interior_6neighbor(); }

  // ---- helpers used by the validators ------------------------------------------------------
  template <class F> void on_device(F &&op) {
    auto ctx = irt::Context::global();
    irt_grid g = grid();
    irt_env *env = nullptr;
    irt::check(ctx->get(), irt_env_create(ctx->get(), &g, &env));
    std::shared_ptr<irt_env> eg(env, [](irt_env *x) { irt_env_destroy(x); });
    upload_env(ctx->get(), env);
    irt::check(ctx->get(), op(ctx->get(), env));
    const size_t Nb = N_ / 4;
    std::vector<uint64_t> dense(Nb * Nb * Nb);
    irt::check(ctx->get(), irt_env_download(ctx->get(), env, dense.data()));
    blocks_.clear();
    for (size_t k = 0; k < dense.size(); k++)
      if (dense[k]) blocks_[(uint32_t)k] = dense[k];
  }
  void upload_env(irt_ctx *ctx, irt_env *env) const {
    std::vector<uint8_t> xyz(3 * blocks_.size() + 3);
    std::vector<uint64_t> bits(blocks_.size() + 1);
    size_t i = 0;
    for (auto &kv : blocks_) {
      int bx, by, bz;
      irt_morton_decode(kv.first, (int)(N_ / 4), &bx, &by, &bz);
      xyz[3 * i] = (uint8_t)bx; xyz[3 * i + 1] = (uint8_t)by; xyz[3 * i + 2] = (uint8_t)bz;
      bits[i++] = kv.second;
    }
    irt::check(ctx, irt_env_update_sparse(ctx, env, xyz.data(), bits.data(), (int64_t)blocks_.size()));
  }
  void to_store(irt_ctx *ctx, irt_setstore *st) const {
    std::vector<uint64_t> off{0, (uint64_t)blocks_.size()}, bits;
    std::vector<uint32_t> keys;
    for (auto &kv : blocks_) { keys.push_back(kv.first); bits.push_back(kv.second); }
    keys.push_back(0); bits.push_back(0);
    irt::check(ctx, irt_setstore_import(ctx, st, 1, off.data(), keys.data(), bits.data()));
  }
  /// OR set `i` of a device store into this octree
  void merge_store(irt_ctx *ctx, irt_setstore *st, int64_t i) {
    const int64_t n = irt_setstore_num_sets(st), nb = irt_setstore_num_blocks(st);
    std::vector<uint64_t> off(n + 1), bits(nb + 1);
    std::vector<uint32_t> keys(nb + 1);
    irt::check(ctx, irt_setstore_export(ctx, st, off.data(), keys.data(), bits.data()));
    for (uint64_t j = off[i]; j < off[i + 1]; j++) blocks_[keys[j]] |= bits[j];
  }
  static VoxelOctree from_store(irt_ctx *ctx, irt_setstore *st, int64_t i, const VoxelOctree &like) {
    VoxelOctree v = like.empty_copy();
    v.merge_store(ctx, st, i);
    return v;
  }

private:
  static void lim_check(double a, double b) {
    if (a >= b) throw std::length_error("limits must be positive in size");  // VoxelOctree.cpp:152-177
  }
  void domain_check(double x, double y, double z) const {  // VoxelOctree.cpp:1511-1521
    if (!is_in_domain(x, y, z)) throw std::domain_error("point is out of the voxel dimensions");
  }
  /// node covering nb^3 blocks whose Morton keys start at key_lo (keys are in the reference's child order)
  void visit_blocks_impl(const ConstBlockVisitor &f, uint32_t key_lo, size_t nb) const {
    const size_t c = nb / 2, cc = c * c * c;
    for (uint32_t i = 0; i < 8; i++) {
      const uint32_t lo = key_lo + i * (uint32_t)cc;
      auto it = blocks_.lower_bound(lo);
      const bool present = it != blocks_.end() && it->first < lo + cc;
      int bx, by, bz;
      irt_morton_decode(lo, (int)(N_ / 4), &bx, &by, &bz);
      if (!present) f((size_t)bx, (size_t)by, (size_t)bz, 0);
      else if (c == 1) f((size_t)bx, (size_t)by, (size_t)bz, it->second);
      else visit_blocks_impl(f, lo, c);
    }
  }
  void check_dims(const VoxelOctree &o) const {
    if (N_ != o.N_)
      throw std::invalid_argument("voxel dimension mismatch (" + std::to_string(N_) + " != " + std::to_string(o.N_) + ")");
  }
  uint32_t key(size_t bx, size_t by, size_t bz) const { return irt_morton_key((int)bx, (int)by, (int)bz, (int)(N_ / 4)); }
  size_t N_;
  std::array<double, 6> lim_{};
  std::map<uint32_t, uint64_t> blocks_;
};

}  // namespace collision

namespace motion_planning {

/// the voxelisable part of motion_planning::Environment (motion-planning/Environment.h): points, spheres,
/// capsules and voxelize() (Environment.cpp:62-101).  Meshes are not supported there either (std::logic_error).
struct Environment {
  std::vector<collision::Point> points;
  std::vector<collision::Sphere> spheres;
  std::vector<collision::Capsule> capsules;
  void push_back(const collision::Point &p) { points.push_back(p); }
  void push_back(const collision::Sphere &s) { spheres.push_back(s); }
  void push_back(const collision::Capsule &c) { capsules.push_back(c); }

  std::shared_ptr<collision::VoxelOctree> voxelize(const collision::VoxelOctree &reference) const {
    auto voxels = std::make_shared<collision::VoxelOctree>(reference.empty_copy());
    voxels->add_primitives(points, spheres, capsules);
    return voxels;
  }
  /// every radius grown by `dilate`, points become spheres.  As in the reference, dilate == 0 voxelises an
  /// EMPTY environment (its `dummy` is only filled when dilate > 0, Environment.cpp:86-99).
  std::shared_ptr<collision::VoxelOctree> voxelize(const collision::VoxelOctree &reference, double dilate) const {
    if (dilate < 0.0) throw std::invalid_argument("Negative dilation value given");
    Environment dummy;
    if (dilate > 0.0) {
      for (auto &p : points) dummy.spheres.push_back(collision::Sphere{p, dilate});
      for (auto &s : spheres) dummy.spheres.push_back(collision::Sphere{s.c, s.r + dilate});
      for (auto &c : capsules) dummy.capsules.push_back(collision::Capsule{c.a, c.b, c.r + dilate});
    }
    return dummy.voxelize(reference);
  }
};

/// the part of VoxelEnvironment the hot path uses: inv_rotation + PartialVoxelization
struct VoxelEnvironment {
  std::array<double, 9> inv_rotation{1, 0, 0, 0, 1, 0, 0, 0, 1};  // row-major
  struct PartialVoxelization {  // VoxelEnvironment.h:137-143
    bool is_fully_valid = false;
    double t = 0.0;
    std::vector<double> last_valid;
    std::vector<collision::Point> last_backbone;
    collision::VoxelOctree voxels;
  };
};

/// AbstractVoxelValidityChecker / VoxelBackboneValidityChecker (AbstractVoxelValidityChecker.h:17-65,
/// VoxelBackboneValidityChecker.h:20-57) without the OMPL base class
class VoxelBackboneValidityChecker {
public:
  VoxelBackboneValidityChecker(const tendon::TendonRobot &robot, const VoxelEnvironment &venv,
                               collision::VoxelOctree voxels)
      : robot_(robot), venv_(venv), voxels_(std::move(voxels)) {
    const double mx = std::max({voxels_.dx(), voxels_.dy(), voxels_.dz()});
    if (robot.specs.dL > mx)  // VoxelBackboneValidityChecker.h:37-45
      throw std::invalid_argument("robot.specs.dL is larger than expected by VoxelBackboneValidityChecker");
    home_ = robot.home_shape();
  }
  std::pair<tendon::TendonResult, tendon::TendonResult> fk(const std::vector<double> &state) const {
    return {robot_.shape(state), robot_.enable_retraction ? robot_.home_shape(state) : home_};
  }
  bool is_valid_shape(const tendon::TendonResult &fk_shape, const tendon::TendonResult &home_shape) const {
    if (!fk_shape.converged || !home_shape.converged) return false;  // AbstractValidityChecker.cpp:99-114
    if (!robot_.is_within_length_limits(robot_.calc_dl(home_shape.L_i, fk_shape.L_i))) return false;
    return !robot_.collides_self(fk_shape);
  }
  collision::VoxelOctree voxelize(const tendon::TendonResult &fk_shape) const {
    auto ctx = irt::Context::global();
    irt_grid g = voxels_.grid(venv_.inv_rotation);
    irt_setstore *st = nullptr;
    irt::check(ctx->get(), irt_setstore_create(ctx->get(), &g, &st));
    std::shared_ptr<irt_setstore> guard(st, [](irt_setstore *x) { irt_setstore_destroy(x); });
    int32_t n = (int32_t)fk_shape.p.size();
    std::vector<double> flat(3 * std::max<size_t>(1, fk_shape.p.size()));
    for (size_t i = 0; i < fk_shape.p.size(); i++) std::memcpy(&flat[3 * i], fk_shape.p[i].data(), 24);
    irt::check(ctx->get(), irt_voxelize_shapes(ctx->get(), flat.data(), &n, std::max(1, n), 1, st));
    return collision::VoxelOctree::from_store(ctx->get(), st, 0, voxels_);
  }
  bool collides(const collision::VoxelOctree &v) const { return voxels_.collides(v); }
  const collision::VoxelOctree &voxels() const { return voxels_; }
  const tendon::TendonRobot &robot() const { return robot_; }
  const VoxelEnvironment &venv() const { return venv_; }

private:
  const tendon::TendonRobot &robot_;
  const VoxelEnvironment &venv_;
  collision::VoxelOctree voxels_;
  tendon::TendonResult home_;
};

/// OMPL compound interpolate of the space of Problem.cpp:101-163 restated (RealVector linear, SO2 shortest arc + wrap)
inline std::vector<double> interpolate_states(const tendon::TendonRobot &robot, const std::vector<double> &a,
                                              const std::vector<double> &b, double t) {
  std::vector<double> out(a.size());
  const size_t N = robot.tendons.size();
  for (size_t i = 0; i < a.size(); i++) out[i] = a[i] + (b[i] - a[i]) * t;
  if (robot.enable_rotation) {
    double diff = b[N] - a[N];
    if (std::fabs(diff) > M_PI) {
      diff = (diff > 0.0) ? 2.0 * M_PI - diff : -2.0 * M_PI - diff;
      double v = a[N] - diff * t;
      if (v > M_PI) v -= 2.0 * M_PI; else if (v < -M_PI) v += 2.0 * M_PI;
      out[N] = v;
    }
  }
  return out;
}

/// AbstractVoxelMotionValidator / VoxelBackboneMotionValidator (AbstractVoxelMotionValidator.h:32-193,
/// VoxelBackboneMotionValidator.cpp:19-91); the OMPL space constants come from irt_space
class VoxelBackboneMotionValidator {
public:
  using PartialVoxelization = VoxelEnvironment::PartialVoxelization;
  VoxelBackboneMotionValidator(const tendon::TendonRobot &robot, const VoxelEnvironment &venv,
                               collision::VoxelOctree voxels, irt_space space = {0.02, 0.01, 0.0001})
      : robot_(robot), venv_(venv), voxels_(std::move(voxels)), space_(space) {}

  PartialVoxelization voxelize(const std::vector<double> &a, const std::vector<double> &b) const {
    const size_t S = robot_.state_size();
    if (a.size() != S || b.size() != S) throw std::invalid_argument("start and end are different sizes");
    irt_ctx *ctx = robot_.ctx();
    irt_grid g = voxels_.grid(venv_.inv_rotation);
    irt_setstore *st = nullptr;
    irt::check(ctx, irt_setstore_create(ctx, &g, &st));
    std::shared_ptr<irt_setstore> guard(st, [](irt_setstore *x) { irt_setstore_destroy(x); });
    uint32_t flags = 0;
    double t_last = 0.0;
    int32_t ns = 0;
    irt::check(ctx, irt_voxelize_edges(ctx, robot_.handle(), &space_, a.data(), b.data(), (int)S, 1, st, &flags,
                                       &t_last, &ns));
    if (flags & IRT_FLAG_OUT_OF_DOMAIN) throw std::domain_error("point is out of the voxel dimensions");
    PartialVoxelization pv;
    pv.is_fully_valid = !(flags & IRT_FLAG_PARTIAL);
    if (!pv.is_fully_valid) num_voxelize_errors_++;  // AbstractVoxelMotionValidator.h:105
    pv.t = t_last;
    pv.last_valid = interpolate(a, b, t_last);
    pv.last_backbone = robot_.shape(pv.last_valid).p;
    pv.voxels = collision::VoxelOctree::from_store(ctx, st, 0, voxels_);
    return pv;
  }
  /// voxelize_until_invalid (AbstractVoxelMotionValidator.h:109-127): also stops at the first
  /// configuration whose backbone voxels hit the obstacle voxels of this validator
  PartialVoxelization voxelize_until_invalid(const std::vector<double> &a, const std::vector<double> &b) const {
    const size_t S = robot_.state_size();
    if (a.size() != S || b.size() != S) throw std::invalid_argument("start and end are different sizes");
    irt_ctx *ctx = robot_.ctx();
    irt_grid g = voxels_.grid(venv_.inv_rotation);
    irt_setstore *st = nullptr;
    irt::check(ctx, irt_setstore_create(ctx, &g, &st));
    std::shared_ptr<irt_setstore> guard(st, [](irt_setstore *x) { irt_setstore_destroy(x); });
    irt_env *env = nullptr;
    irt::check(ctx, irt_env_create(ctx, &g, &env));
    std::shared_ptr<irt_env> eg(env, [](irt_env *x) { irt_env_destroy(x); });
    voxels_.upload_env(ctx, env);
    uint32_t flags = 0;
    double t_last = 0.0;
    irt::check(ctx, irt_voxelize_edges_until_invalid(ctx, robot_.handle(), &space_, a.data(), b.data(), (int)S, 1,
                                                     env, st, &flags, &t_last, nullptr));
    if (flags & IRT_FLAG_OUT_OF_DOMAIN) throw std::domain_error("point is out of the voxel dimensions");
    PartialVoxelization pv;
    pv.is_fully_valid = !(flags & IRT_FLAG_PARTIAL);
    pv.t = t_last;
    pv.last_valid = interpolate(a, b, t_last);
    pv.last_backbone = robot_.shape(pv.last_valid).p;
    pv.voxels = collision::VoxelOctree::from_store(ctx, st, 0, voxels_);
    return pv;
  }
  bool collides(const collision::VoxelOctree &swept) const { return voxels_.collides(swept); }
  size_t num_voxelize_errors() const { return num_voxelize_errors_; }
  uint32_t valid_segment_count(const std::vector<double> &a, const std::vector<double> &b) const {
    irt_robot_desc d = robot_.desc();
    return irt_valid_segment_count(&d, &space_, a.data(), b.data());
  }
  std::vector<double> interpolate(const std::vector<double> &a, const std::vector<double> &b, double t) const {
    return interpolate_states(robot_, a, b, t);
  }

private:
  const tendon::TendonRobot &robot_;
  const VoxelEnvironment &venv_;
  collision::VoxelOctree voxels_;
  irt_space space_;
  mutable size_t num_voxelize_errors_ = 0;
};

/// batch entry points of VoxelCachedLazyPRM (VoxelCachedLazyPRM.h:495-520): the graph lives in
/// (states, edges); the voxel caches live on the device; validity words mirror
/// vertexValidityProperty_ / edgeValidityProperty_ (VALIDITY_UNKNOWN = 0, VALIDITY_TRUE = 1).
class VoxelCachedLazyPRM {
public:
  static constexpr unsigned VALIDITY_UNKNOWN = 0, VALIDITY_TRUE = 1;  // VoxelCachedLazyPRM.h:598-601
  VoxelCachedLazyPRM(const tendon::TendonRobot &robot, const VoxelEnvironment &venv,
                     const collision::VoxelOctree &env_voxels, irt_space space = {0.02, 0.01, 0.0001})
      : robot_(robot), venv_(venv), env_voxels_(env_voxels), space_(space) {
    ctx_ = robot.ctx();
    irt_grid g = env_voxels_.grid(venv_.inv_rotation);
    irt::check(ctx_, irt_setstore_create(ctx_, &g, &vstore_));
    irt::check(ctx_, irt_setstore_create(ctx_, &g, &estore_));
    irt::check(ctx_, irt_env_create(ctx_, &g, &env_));
    env_voxels_.upload_env(ctx_, env_);
    // the exact k-NN scans on the device: states under the compound space's distance, tips under plain R^3
    irt_metric sm{(int32_t)robot_.tendons.size(), -1, -1, 0, 0.0, 0.0};
    int col = sm.n_euclid;
    if (robot_.enable_rotation) { sm.so2_col = col++; sm.w_so2 = tensionExtent() / (4.0 * M_PI); }
    if (robot_.enable_retraction) { sm.lin_col = col++; sm.w_lin = 2.0 * tensionExtent() / robot_.specs.L; }
    const irt_metric tm{3, -1, -1, 0, 0.0, 0.0};
    irt::check(ctx_, irt_nnset_create(ctx_, (int)robot_.state_size(), &sm, &nn_states_.set));
    irt::check(ctx_, irt_nnset_create(ctx_, 3, &tm, &nn_tips_.set));
  }
  ~VoxelCachedLazyPRM() {
    irt_setindex_destroy(vindex_); irt_setindex_destroy(eindex_);
    irt_setstore_destroy(vstore_); irt_setstore_destroy(estore_); irt_env_destroy(env_); irt_env_destroy(env_next_);
    irt_nnset_destroy(nn_states_.set); irt_nnset_destroy(nn_tips_.set);
  }
  void setRoadmap(std::vector<std::vector<double>> states, std::vector<std::pair<size_t, size_t>> edges) {
    states_ = std::move(states); edges_ = std::move(edges);
    nn_states_.stale = true;
    vflags_.clear(); eflags_.clear();
    adj_edges_ = (size_t)-1; vertex_removed_.clear(); edge_removed_.clear();
    clearValidity();
  }
  // ---- createRoadmap (VoxelCachedLazyPRM.h:468-495, .cpp:1380-1561) -------------------------------------
  enum CreateRoadmapOption : unsigned {
    LazyRoadmap = 0x0,       // nothing is checked, just sampled configs and connecting edges
    VoxelizeVertices = 0x1,  // voxelize vertices, rejecting invalid shapes
    ValidateVertices = 0x2,  // ... and rejecting vertices that hit the environment
    VoxelizeEdges = 0x4,     // voxelize edges, removing those that are not fully valid
    ValidateEdges = 0x8,     // ... and removing edges that hit the environment
  };
  using Sampler = std::function<std::vector<double>()>;
  /// sampler_->sampleUniform: by default TendonRobot::random_state over a seeded std::mt19937
  /// (the reference's `sample_like_sphere` RetractionSampler is a setSampler() away)
  void setSampler(Sampler s) { sampler_ = std::move(s); }
  void setSeed(uint32_t seed) { gen_.seed(seed); }
  /// KBoundedStrategy(k, range) over nn_ (.cpp:1329-1345): the k nearest milestones of v -- v itself is
  /// one of them, it is in nn_ by then -- no further away than range.  magic::DEFAULT_NEAREST_NEIGHBORS_LAZY
  /// = 5 (.cpp:125); range defaults to SelfConfig::configurePlannerRange's 20 % of the maximum extent.
  void setMaxNearestNeighbors(size_t k) { k_ = k; }
  void setRange(double d) { range_ = d; }
  double getRange() const { return range_ > 0.0 ? range_ : 0.2 * maximumExtent(); }
  /// replaces the default exact (brute-force) neighbour search: v -> candidate neighbours, nearest first
  void setConnectionStrategy(std::function<std::vector<size_t>(size_t)> f) { connection_ = std::move(f); }

  /// weights and extents of the compound space of Problem::create_space_information (Problem.cpp:101-163)
  double tensionExtent() const {
    double e2 = 0.0;
    for (auto &t : robot_.tendons) e2 += t.max_tension * t.max_tension;
    return std::sqrt(e2);
  }
  double maximumExtent() const {  // CompoundStateSpace: sum of weight_i * extent_i
    const double ext = tensionExtent();
    double e = ext;
    if (robot_.enable_rotation) e += (ext / (4.0 * M_PI)) * M_PI;
    if (robot_.enable_retraction) e += (2.0 * ext / robot_.specs.L) * robot_.specs.L;
    return e;
  }
  /// distanceFunction / motionCost: CompoundStateSpace::distance = sum of weight_i * d_i
  double distance(const std::vector<double> &a, const std::vector<double> &b) const {
    const size_t N = robot_.tendons.size();
    const double ext = tensionExtent();
    double d2 = 0.0;
    for (size_t i = 0; i < N; i++) d2 += (a[i] - b[i]) * (a[i] - b[i]);
    double d = std::sqrt(d2);
    size_t k = N;
    if (robot_.enable_rotation) {
      double dr = std::fabs(a[k] - b[k]);  // SO2StateSpace::distance
      if (dr > M_PI) dr = 2.0 * M_PI - dr;
      d += (ext / (4.0 * M_PI)) * dr;
      k++;
    }
    if (robot_.enable_retraction) d += (2.0 * ext / robot_.specs.L) * std::fabs(a[k] - b[k]);
    return d;
  }

  /// Brings the roadmap up to N vertices.  Same order of work as the reference: rejection-sample the new
  /// vertices (here: whole candidate batches through ONE FK / voxelise / check call each round instead of
  /// an OpenMP loop of single shapes), add them all, connect every new vertex to its neighbours
  /// sequentially, then voxelise (and validate) the new edges as one batch and remove the invalid ones.
  /// Options only pertain to what is added.  Duplicate states (addMilestone's was_added == false) cannot
  /// be told apart from a rejected sample here and are not looked for.
  void createRoadmap(size_t N, unsigned opt = LazyRoadmap) {
    const size_t Nv = states_.size();
    if (N <= Nv) return;  // "Graph is already at or bigger than N, skipping roadmap creation"
    adj_edges_ = (size_t)-1; vertex_removed_.clear(); edge_removed_.clear();   // the graph changes: adjacency is rebuilt
    const bool validate_verts = opt & ValidateVertices, validate_edges = opt & ValidateEdges;
    const bool voxelize_verts = validate_verts || (opt & VoxelizeVertices);
    const bool voxelize_edges = validate_edges || (opt & VoxelizeEdges);
    const size_t S = robot_.state_size();
    const bool had_vcache = vflags_.size() == Nv && Nv > 0, had_ecache = eflags_.size() == edges_.size() && !edges_.empty();
    const uint32_t bad_shape = IRT_FLAG_NONCONVERGED | IRT_FLAG_LENGTH_LIMIT | IRT_FLAG_SELF_COLLISION |
                               IRT_FLAG_BAD_STATE | IRT_FLAG_OUT_OF_DOMAIN;

    // ---- rejection sampling, a batch per round (.cpp:1415-1455) ----
    std::vector<std::vector<double>> added;
    irt_setstore *scratch = nullptr;
    irt_grid g = env_voxels_.grid(venv_.inv_rotation);
    irt::check(ctx_, irt_setstore_create(ctx_, &g, &scratch));
    std::shared_ptr<irt_setstore> guard(scratch, [](irt_setstore *x) { irt_setstore_destroy(x); });
    for (int round = 0; added.size() < N - Nv; round++) {
      if (round >= 1000) throw std::runtime_error("createRoadmap: rejection sampling does not terminate");
      const size_t need = N - Nv - added.size(), m = need + need / 4 + 16;
      std::vector<std::vector<double>> cand(m);
      for (auto &c : cand) {
        c = sampler_ ? sampler_() : robot_.random_state(gen_);
        if (c.size() != S) throw std::invalid_argument("State is not the right size");
      }
      std::vector<char> keep(m, 1);
      if (voxelize_verts) {
        std::vector<double> flat(m * S), tips(3 * m);
        std::vector<uint32_t> fl(m), words((m + 31) / 32 + 1, 0);
        for (size_t i = 0; i < m; i++) std::copy(cand[i].begin(), cand[i].end(), flat.begin() + i * S);
        irt::check(ctx_, irt_voxelize_vertices(ctx_, robot_.handle(), flat.data(), (int)S, (int64_t)m, scratch,
                                               fl.data(), tips.data()));
        if (validate_verts) irt::check(ctx_, irt_check_sets(ctx_, scratch, env_, 0, (int64_t)m, words.data()));
        for (size_t i = 0; i < m; i++)
          keep[i] = !(fl[i] & bad_shape) && !((words[i >> 5] >> (i & 31)) & 1u);
      }
      for (size_t i = 0; i < m && added.size() < N - Nv; i++)
        if (keep[i]) added.push_back(std::move(cand[i]));
    }
    states_.insert(states_.end(), added.begin(), added.end());
    vertex_validity_.resize(N, VALIDITY_UNKNOWN);
    if (voxelize_verts || had_vcache) {
      precomputeVertexVoxelCache();  // one batch over all vertices: the old sets are recomputed, not changed
      if (validate_verts) std::fill(vertex_validity_.begin() + Nv, vertex_validity_.end(), VALIDITY_TRUE);
    }

    // ---- empty edges, sequentially, new vertices in index order (.cpp:1486-1500) ----
    std::set<std::pair<size_t, size_t>> have;
    for (auto &e : edges_) have.insert(std::minmax(e.first, e.second));
    std::vector<std::pair<size_t, size_t>> new_edges;
    irt_nnset *nn = connection_ ? nullptr : nearestSet(false, k_);
    std::vector<int64_t> nbr;
    if (nn) {   // every new vertex's KBoundedStrategy neighbours in one device call
      std::vector<double> q((N - Nv) * S);
      for (size_t v = Nv; v < N; v++) std::copy(states_[v].begin(), states_[v].end(), q.begin() + (v - Nv) * S);
      nbr.resize((N - Nv) * k_);
      irt::check(ctx_, irt_nnset_knn(ctx_, nn, q.data(), (int64_t)(N - Nv), (int)k_, getRange(), nullptr, nbr.data(),
                                     nullptr));
    }
    for (size_t v = Nv; v < N; v++) {
      std::vector<size_t> cand;
      if (nn) {
        for (size_t j = 0; j < k_ && nbr[(v - Nv) * k_ + j] >= 0; j++) cand.push_back((size_t)nbr[(v - Nv) * k_ + j]);
      } else {
        cand = connection_ ? connection_(v) : nearestKBounded(v);
      }
      for (size_t n : cand)
        if (n != v && have.insert(std::minmax(v, n)).second) new_edges.emplace_back(v, n);  // connectVertices
    }

    // ---- voxelise / validate the new edges and remove the invalid ones (.cpp:1505-1551) ----
    if (voxelize_edges && !new_edges.empty()) {
      const size_t m = new_edges.size();
      std::vector<double> a(m * S), b(m * S);
      for (size_t i = 0; i < m; i++) {
        std::copy(states_[new_edges[i].first].begin(), states_[new_edges[i].first].end(), a.begin() + i * S);
        std::copy(states_[new_edges[i].second].begin(), states_[new_edges[i].second].end(), b.begin() + i * S);
      }
      std::vector<uint32_t> fl(m), words((m + 31) / 32 + 1, 0);
      irt::check(ctx_, irt_voxelize_edges(ctx_, robot_.handle(), &space_, a.data(), b.data(), (int)S, (int64_t)m,
                                          scratch, fl.data(), nullptr, nullptr));
      if (validate_edges) irt::check(ctx_, irt_check_sets(ctx_, scratch, env_, 0, (int64_t)m, words.data()));
      std::vector<std::pair<size_t, size_t>> kept;
      for (size_t i = 0; i < m; i++)
        if (!(fl[i] & IRT_FLAG_PARTIAL) && !((words[i >> 5] >> (i & 31)) & 1u)) kept.push_back(new_edges[i]);
      new_edges.swap(kept);
    }
    const size_t Ne = edges_.size();
    edges_.insert(edges_.end(), new_edges.begin(), new_edges.end());
    edge_validity_.resize(edges_.size(), VALIDITY_UNKNOWN);
    if (voxelize_edges || had_ecache) {
      precomputeEdgeVoxelCache();
      if (validate_edges) std::fill(edge_validity_.begin() + Ne, edge_validity_.end(), VALIDITY_TRUE);
    } else {
      eflags_.clear();
    }
    if (!(voxelize_verts || had_vcache)) vflags_.clear();
  }
  const std::vector<std::vector<double>> &states() const { return states_; }
  const std::vector<std::pair<size_t, size_t>> &edges() const { return edges_; }
  /// tip position of every vertex with a voxel cache (tipPositionProperty_), xyz per vertex
  const std::vector<double> &tipPositions() const { return tips_; }

  void precomputeVertexVoxelCache() {  // .cpp:1687-1734
    const size_t S = robot_.state_size(), n = states_.size();
    std::vector<double> flat(n * S);
    for (size_t i = 0; i < n; i++) std::copy(states_[i].begin(), states_[i].end(), flat.begin() + i * S);
    vflags_.assign(n, 0); tips_.assign(3 * n, 0.0);
    nn_tips_.stale = true;
    vcache_builds_++;
    irt::check(ctx_, irt_voxelize_vertices(ctx_, robot_.handle(), flat.data(), (int)S, (int64_t)n, vstore_,
                                           vflags_.data(), tips_.data()));
  }
  void precomputeEdgeVoxelCache() {  // .cpp:1736-1782
    const size_t S = robot_.state_size(), n = edges_.size();
    std::vector<double> a(n * S), b(n * S);
    for (size_t i = 0; i < n; i++) {
      std::copy(states_[edges_[i].first].begin(), states_[edges_[i].first].end(), a.begin() + i * S);
      std::copy(states_[edges_[i].second].begin(), states_[edges_[i].second].end(), b.begin() + i * S);
    }
    eflags_.assign(n, 0);
    ecache_builds_++;
    irt::check(ctx_, irt_voxelize_edges(ctx_, robot_.handle(), &space_, a.data(), b.data(), (int)S, (int64_t)n,
                                        estore_, eflags_.data(), nullptr, nullptr));
  }
  void precomputeVoxelCache() { precomputeVertexVoxelCache(); precomputeEdgeVoxelCache(); }
  /// The batch form of the reference's compute-if-absent voxelizeVertex / voxelizeEdge (.cpp:2803-2837, 2879-2902)
  /// over the items the caches lack (vertices and edges that roadmapIk / addMilestone added since the caches were
  /// built): only they are voxelised, into scratch stores, and appended to the cached stores with their flags and
  /// tips.  A cache that does not exist yet is built whole.  Afterwards the next sweep is one K3 launch over every
  /// item.  Validity words are not touched.
  void extendVoxelCache() {
    const size_t S = robot_.state_size(), nv = states_.size(), ne = edges_.size();
    if (vflags_.empty() || vflags_.size() > nv || tips_.size() < 3 * vflags_.size()) {
      precomputeVertexVoxelCache();
    } else if (vflags_.size() < nv) {
      const size_t v0 = vflags_.size(), m = nv - v0;
      std::vector<double> flat(m * S), tips(3 * m);
      for (size_t i = 0; i < m; i++) std::copy(states_[v0 + i].begin(), states_[v0 + i].end(), flat.begin() + i * S);
      std::vector<uint32_t> fl(m);
      std::shared_ptr<irt_setstore> scratch = scratch_store();
      irt::check(ctx_, irt_voxelize_vertices(ctx_, robot_.handle(), flat.data(), (int)S, (int64_t)m, scratch.get(),
                                             fl.data(), tips.data()));
      irt::check(ctx_, irt_setstore_append(ctx_, vstore_, scratch.get(), 0, (int64_t)m, nullptr));
      vflags_.insert(vflags_.end(), fl.begin(), fl.end());
      if (tips_.size() == 3 * v0) {
        tips_.insert(tips_.end(), tips.begin(), tips.end());   // appended rows: the k-NN copy appends them too
      } else if (tips_.size() != 3 * nv || !std::equal(tips.begin(), tips.end(), tips_.begin() + 3 * v0)) {
        tips_.resize(3 * v0);
        tips_.insert(tips_.end(), tips.begin(), tips.end());
        nn_tips_.stale = true;
      }
    }
    if (eflags_.empty() || eflags_.size() > ne) {
      precomputeEdgeVoxelCache();
    } else if (eflags_.size() < ne) {
      const size_t e0 = eflags_.size(), m = ne - e0;
      std::vector<double> a(m * S), b(m * S);
      for (size_t i = 0; i < m; i++) {
        std::copy(states_[edges_[e0 + i].first].begin(), states_[edges_[e0 + i].first].end(), a.begin() + i * S);
        std::copy(states_[edges_[e0 + i].second].begin(), states_[edges_[e0 + i].second].end(), b.begin() + i * S);
      }
      std::vector<uint32_t> fl(m);
      std::shared_ptr<irt_setstore> scratch = scratch_store();
      irt::check(ctx_, irt_voxelize_edges(ctx_, robot_.handle(), &space_, a.data(), b.data(), (int)S, (int64_t)m,
                                          scratch.get(), fl.data(), nullptr, nullptr));
      irt::check(ctx_, irt_setstore_append(ctx_, estore_, scratch.get(), 0, (int64_t)m, nullptr));
      eflags_.insert(eflags_.end(), fl.begin(), fl.end());
    }
  }
  /// clear*VoxelCache (.cpp:1814-1829): drop the cached sets; validity words stay, like the reference's
  void clearVertexVoxelCache() {
    clear_store(vstore_); vflags_.clear(); tips_.clear(); nn_tips_.stale = true;
    irt_setindex_destroy(vindex_); vindex_ = nullptr;
  }
  void clearEdgeVoxelCache() { clear_store(estore_); eflags_.clear(); irt_setindex_destroy(eindex_); eindex_ = nullptr; }
  void clearVoxelCache() { clearVertexVoxelCache(); clearEdgeVoxelCache(); }
  size_t vertexVoxelCacheSize() const { return (size_t)irt_setstore_num_sets(vstore_); }
  size_t edgeVoxelCacheSize() const { return (size_t)irt_setstore_num_sets(estore_); }
  /// Items that joined the roadmap after its voxel cache was built (roadmapIk / addMilestone) have no cached set:
  /// a sweep covers the cached sets with K3 and the few newcomers with one small scratch batch; only when there
  /// are more than maxUncached() of them is the cache rebuilt.
  void setMaxUncached(size_t n) { max_uncached_ = n; }
  void precomputeVertexValidity() {  // .cpp:1563-1598 with warm caches
    if (vflags_.size() != states_.size() &&
        (vflags_.empty() || vflags_.size() > states_.size() || states_.size() - vflags_.size() > max_uncached_))
      precomputeVertexVoxelCache();
    sweep(vstore_, vflags_, kVertexInvalid, vertex_validity_, vwords_, vwords_n_);
    if (vertex_validity_.size() < states_.size()) {
      std::vector<size_t> ids;
      for (size_t v = vertex_validity_.size(); v < states_.size(); v++) ids.push_back(v);
      for (unsigned x : checkVerticesNow(ids)) vertex_validity_.push_back(x);
    }
    vertex_unchecked_.clear();
    vertex_swept_ = true;
    sweeps_++;
  }
  void precomputeEdgeValidity() {  // .cpp:1600-1647
    if (eflags_.size() != edges_.size() &&
        (eflags_.empty() || eflags_.size() > edges_.size() || edges_.size() - eflags_.size() > max_uncached_))
      precomputeEdgeVoxelCache();
    sweep(estore_, eflags_, IRT_FLAG_PARTIAL, edge_validity_, ewords_, ewords_n_);
    if (edge_validity_.size() < edges_.size()) {
      std::vector<size_t> ids;
      for (size_t e = edge_validity_.size(); e < edges_.size(); e++) ids.push_back(e);
      for (unsigned x : checkEdgesNow(ids)) edge_validity_.push_back(x);
    }
    edge_unchecked_.clear();
    edge_swept_ = true;
    sweeps_++;
  }
  void precomputeValidity() { precomputeVertexValidity(); precomputeEdgeValidity(); }
  void clearValidity() {  // .cpp:1656-1663
    vertex_validity_.assign(states_.size(), VALIDITY_UNKNOWN);
    edge_validity_.assign(edges_.size(), VALIDITY_UNKNOWN);
    vertex_swept_ = edge_swept_ = false;
    vertex_unchecked_.clear(); edge_unchecked_.clear();
  }

  // ---- lazy-path consumers: the query side of the planner (SURVEY 8(f) row 2) --------------------------
  /// computeVertexValidity (.cpp:2607-2618).  The reference checks ONE vertex here (voxelise if needed +
  /// collides); with the verdict words of a full sweep on the host it is a table look-up.  The first query
  /// after clearValidity() runs the sweep (one K3 launch over all cached sets), later ones only read.
  bool computeVertexValidity(size_t v) {
    if (!vertex_swept_) precomputeVertexValidity();
    lookups_++;
    if (vertex_unchecked_.erase(v)) {   // joined the roadmap after the sweep, never checked: the reference's lazy check
      vertex_validity_[v] = checkVerticesNow({v})[0];
      single_checks_++;
    }
    return (vertex_validity_[v] & VALIDITY_TRUE) != 0;
  }
  /// computeEdgeValidity (.cpp:2620-2631): is_fully_valid (no IRT_FLAG_PARTIAL) and no hit
  bool computeEdgeValidity(size_t e) {
    if (!edge_swept_) precomputeEdgeValidity();
    lookups_++;
    if (edge_unchecked_.erase(e)) {
      edge_validity_[e] = checkEdgesNow({e})[0];
      single_checks_++;
    }
    return (edge_validity_[e] & VALIDITY_TRUE) != 0;
  }
  size_t sweepCount() const { return sweeps_; }
  size_t lookupCount() const { return lookups_; }
  size_t singleCheckCount() const { return single_checks_; }   // look-ups answered by checking one newcomer
  const std::vector<char> &removedVertices() const { return vertex_removed_; }
  const std::vector<char> &removedEdges() const { return edge_removed_; }
  void restoreRemoved() { vertex_removed_.assign(states_.size(), 0); edge_removed_.assign(edges_.size(), 0); }
  long edgeIndex(size_t a, size_t b) {
    build_adjacency();
    long found = -1;
    for_neighbors(a, [&](size_t nbr, size_t eid) { if (found < 0 && nbr == b) found = (long)eid; });
    return found;
  }
  /// astarSearch (.cpp:2950-2976): A* over the current graph (removed vertices / edges left out), motion cost as
  /// edge weight and heuristic.  Host code in the reference (Boost.Graph) and here.  Empty = no path.
  std::vector<size_t> astarSearch(size_t start, size_t goal) {
    build_adjacency();
    std::vector<size_t> path;
    if (vertex_removed_[start] || vertex_removed_[goal]) return path;
    const size_t n = states_.size();
    std::vector<double> dist(n, std::numeric_limits<double>::infinity());
    std::vector<size_t> prev(n, n);
    std::vector<char> done(n, 0);
    using QE = std::pair<double, size_t>;
    std::priority_queue<QE, std::vector<QE>, std::greater<QE>> heap;
    dist[start] = 0.0; prev[start] = start;
    heap.push({distance(states_[start], states_[goal]), start});
    while (!heap.empty()) {
      const size_t u = heap.top().second;
      heap.pop();
      if (done[u]) continue;
      if (u == goal) {
        for (size_t v = goal; ; v = prev[v]) { path.push_back(v); if (v == start) break; }
        std::reverse(path.begin(), path.end());
        return path;
      }
      done[u] = 1;
      for_neighbors(u, [&](size_t v, size_t eid) {
        if (edge_removed_[eid] || vertex_removed_[v] || done[v]) return;
        const double nd = dist[u] + distance(states_[u], states_[v]);
        if (nd < dist[v]) {
          dist[v] = nd; prev[v] = u;
          heap.push({nd + distance(states_[v], states_[goal]), v});
        }
      });
    }
    return path;
  }
  /// constructSolution (.cpp:2689-2771): A* path, then the lazy checks along it -- every intermediate vertex
  /// first (ALL invalid ones are removed), then the edges from the goal side (the FIRST invalid one is
  /// removed).  Returns the validated path, or an empty one when something was removed / no path exists.
  std::vector<size_t> constructSolution(size_t start, size_t goal) {
    if (start == goal) return {start};
    std::vector<size_t> path = astarSearch(start, goal);
    if (path.empty()) return path;
    bool removed = false;
    for (size_t i = path.size() - 1; i-- > 1;)          // intermediate vertices, goal side first
      if (!computeVertexValidity(path[i])) { vertex_removed_[path[i]] = 1; removed = true; }
    if (removed) return {};
    for (size_t i = path.size() - 1; i >= 1; i--) {     // edges, goal side first
      const long e = edgeIndex(path[i - 1], path[i]);
      if (e < 0 || !computeEdgeValidity((size_t)e)) {
        if (e >= 0) edge_removed_[(size_t)e] = 1;
        return {};
      }
    }
    return path;
  }
  /// the remove-and-retry loop of solveWithRoadmap (.cpp:1977-2096) around constructSolution
  std::vector<size_t> solveWithRoadmap(size_t start, size_t goal, size_t *iterations = nullptr) {
    for (size_t it = 1;; it++) {
      const size_t before = removed_count();
      std::vector<size_t> path = constructSolution(start, goal);
      if (iterations) *iterations = it;
      if (!path.empty() || removed_count() == before) return path;   // solved, or A* found no path
    }
  }
  /// environment replacement (the reference rebuilds its validators, Problem.h:175-216)
  void setEnvironment(const collision::VoxelOctree &env_voxels) {
    env_voxels_ = env_voxels;
    env_voxels_.upload_env(ctx_, env_);
    clearValidity();
  }
  /// the items whose VALIDITY_TRUE bit an updateEnvironment flipped, ascending
  struct EnvironmentChange { std::vector<size_t> vertices, edges; };
  /// Environment replacement that keeps what the change cannot reach.  A validity table that is current (a sweep
  /// ran since the last clearValidity) is patched in place: only the cached sets whose leaves overlap the changed
  /// voxels are re-checked on the device (irt_check_sets_changed over an inverted index of the cache, built on first
  /// use), the items without a cached set in one scratch batch; items still unchecked since the sweep stay unchecked
  /// and their lazy check uses the new grid.  A table that is not current is reset to VALIDITY_UNKNOWN, as
  /// setEnvironment resets it.  Every look-up then answers what it would after setEnvironment(env_voxels); no sweep
  /// is counted.  A chained plan keeps its path when none of the path's items flipped.
  EnvironmentChange updateEnvironment(const collision::VoxelOctree &env_voxels) {
    if (!env_next_) {
      irt_grid g = env_voxels_.grid(venv_.inv_rotation);
      irt::check(ctx_, irt_env_create(ctx_, &g, &env_next_));
    }
    env_voxels_ = env_voxels;
    env_voxels_.upload_env(ctx_, env_next_);
    irt_env *old = env_;
    env_ = env_next_;   // everything that reads env_ sees the new grid
    env_next_ = old;
    EnvironmentChange ch;
    ch.vertices = patchTable(true, old);
    ch.edges = patchTable(false, old);
    return ch;
  }
  const std::vector<unsigned> &vertexValidity() const { return vertex_validity_; }
  const std::vector<unsigned> &edgeValidity() const { return edge_validity_; }
  collision::VoxelOctree vertexVoxels(size_t i) const { return collision::VoxelOctree::from_store(ctx_, vstore_, (int64_t)i, env_voxels_); }
  collision::VoxelOctree edgeVoxels(size_t i) const { return collision::VoxelOctree::from_store(ctx_, estore_, (int64_t)i, env_voxels_); }
  const std::vector<uint32_t> &vertexFlags() const { return vflags_; }
  const std::vector<uint32_t> &edgeFlags() const { return eflags_; }

  // ---- roadmapIk as a batch (.cpp:3095-3420) ---------------------------------------------------------------
  struct IKResult {                 // VoxelCachedLazyPRM.h:356-362
    std::vector<double> controls;   // valid state at or close to the desired tip position
    collision::Point tip_position;  // tip position obtained by controls
    std::vector<double> neighbor;   // where IK started from
    double error = 0.0;             // achieved tip-position error
    size_t index = 0, vertex = 0;   // which of the k neighbours (nearest first) / its roadmap vertex
    size_t lockstep_batches = 0, fk_requests = 0;
    bool accepted = true;           // false: no result within tolerance, the closest valid one is returned
    bool stepped_back = false;      // controls = the last valid state of the edge source -> result
    long source = -1;               // the roadmap vertex that edge starts from (-1: none, or the result itself)
    long added_vertex = -1;         // RMAP_IK_AUTO_ADD: the vertex that joined the roadmap (-1: none)
    bool already_in_roadmap = false;
  };
  /// nnTip_->nearestK: the k vertices whose cached tip positions are nearest to the request (exact)
  std::vector<size_t> nearestTips(const collision::Point &request, size_t k) {
    if (tips_.size() != 3 * states_.size()) precomputeVertexVoxelCache();
    build_adjacency();
    if (irt_nnset *nn = nearestSet(true, k)) {
      const std::vector<uint32_t> words = maskWords(vertex_removed_);
      std::vector<int64_t> idx(k);
      irt::check(ctx_, irt_nnset_knn(ctx_, nn, request.data(), 1, (int)k, INFINITY, words.data(), idx.data(), nullptr));
      std::vector<size_t> out;
      for (int64_t i : idx)
        if (i >= 0) out.push_back((size_t)i);
      return out;
    }
    std::vector<std::pair<double, size_t>> d;
    for (size_t v = 0; v < states_.size(); v++) {
      if (vertex_removed_[v]) continue;
      double s = 0.0;
      for (int c = 0; c < 3; c++) s += (tips_[3 * v + c] - request[c]) * (tips_[3 * v + c] - request[c]);
      d.emplace_back(std::sqrt(s), v);
    }
    k = std::min(k, d.size());
    std::partial_sort(d.begin(), d.begin() + k, d.end());
    std::vector<size_t> out;
    for (size_t i = 0; i < k; i++) out.push_back(d[i].second);
    return out;
  }
  enum RoadmapIkOpts : unsigned {   // VoxelCachedLazyPRM.h:364-381
    RMAP_IK_SIMPLE = 0x0,     // no extra features
    RMAP_IK_AUTO_ADD = 0x1,   // add the IK result to the roadmap, only return one that connects
    RMAP_IK_ACCURATE = 0x2,   // try to connect from the connection-strategy neighbours, not only the IK neighbour
    RMAP_IK_LAZY_ADD = 0x4,   // do not validate the lazily connected edges of the added vertex
  };
  /// CompoundStateSpace::enforceBounds of the space of Problem.cpp:101-163
  std::vector<double> enforceBounds(std::vector<double> x) const {
    const size_t N = robot_.tendons.size();
    for (size_t j = 0; j < N; j++) x[j] = std::min(robot_.tendons[j].max_tension, std::max(0.0, x[j]));
    size_t kk = N;
    if (robot_.enable_rotation) {   // SO2StateSpace::enforceBounds
      double v = std::fmod(x[kk], 2.0 * M_PI);
      if (v < -M_PI) v += 2.0 * M_PI; else if (v >= M_PI) v -= 2.0 * M_PI;
      x[kk++] = v;
    }
    if (robot_.enable_retraction) x[kk] = std::min(robot_.specs.L, std::max(0.0, x[kk]));
    return x;
  }
  /// roadmapIk(request, tolerance, k, opt) of the reference (.cpp:3095-3565) with its per-neighbour loop turned
  /// into batches: the k nearest VALID neighbours in tip space (invalid ones are removed and the query repeated;
  /// validity = table look-ups), the k IK problems solved side by side with their FK requests answered in
  /// lockstep (tip_control::solve_ik_lockstep), ONE FK + is_valid_shape + voxelise + collides call over the k
  /// results, ONE voxelize_until_invalid call over every would-be edge source -> result that the branches below
  /// can ask for, then the reference's order of acceptance walked over those tables:
  ///  * without RMAP_IK_AUTO_ADD the first neighbour (nearest first) whose result is valid and within tolerance;
  ///    failing that the closest valid result; failing that the closest last-valid state of the edges
  ///    source -> result ("stepping them backwards", .cpp:3298-3428);
  ///  * with it the first result within tolerance that a fully valid edge connects to a valid source joins the
  ///    roadmap with that edge (.cpp:3212-3292); failing that the closest last-valid state over the edges of ALL
  ///    results joins it, connected to its source and, lazily, to its connection-strategy neighbours, whose
  ///    edges are validated unless RMAP_IK_LAZY_ADD (.cpp:3430-3565).
  /// Sources per result: the IK neighbour, or with RMAP_IK_ACCURATE connectionStrategy_(vertex) -- the result's
  /// own temporary vertex among them, it is in nn_ by then -- plus the IK neighbour.  Sources found invalid on
  /// the way are removed (removeVertices).  std::nullopt where the reference would index an empty list.
  std::optional<IKResult> roadmapIk(const collision::Point &request, double tolerance, size_t k,
                                    const tip_control::IkSolver &solver, int mode = IRT_JAC_LEVMAR_CENTRAL,
                                    double delta = 1e-6, unsigned opt = RMAP_IK_SIMPLE) {
    const bool auto_add = opt & RMAP_IK_AUTO_ADD, accurate = opt & RMAP_IK_ACCURATE, lazy_add = opt & RMAP_IK_LAZY_ADD;
    std::vector<size_t> nb;
    for (;;) {
      nb = nearestTips(request, k);
      if (nb.empty()) throw std::runtime_error("roadmapIk(): No neighbors were able to be found");
      bool removed = false;
      for (size_t v : nb)
        if (!computeVertexValidity(v)) { vertex_removed_[v] = 1; removed = true; }
      if (!removed) break;
    }
    std::vector<std::vector<double>> starts;
    for (size_t v : nb) starts.push_back(states_[v]);
    size_t batches = 0, requests = 0;
    auto finals = tip_control::solve_ik_lockstep(robot_, solver, starts, request, mode, delta, &batches, &requests);
    // one validity call over the k results
    const size_t S = robot_.state_size(), m = finals.size();
    std::vector<double> flat(m * S), tips(3 * m);
    for (size_t i = 0; i < m; i++) std::copy(finals[i].begin(), finals[i].end(), flat.begin() + i * S);
    std::vector<uint32_t> flags(m), words((m + 31) / 32 + 1, 0);
    irt_setstore *scratch = nullptr;
    irt_grid g = env_voxels_.grid(venv_.inv_rotation);
    irt::check(ctx_, irt_setstore_create(ctx_, &g, &scratch));
    std::shared_ptr<irt_setstore> guard(scratch, [](irt_setstore *x) { irt_setstore_destroy(x); });
    irt::check(ctx_, irt_voxelize_vertices(ctx_, robot_.handle(), flat.data(), (int)S, (int64_t)m, scratch,
                                           flags.data(), tips.data()));
    irt::check(ctx_, irt_check_sets(ctx_, scratch, env_, 0, (int64_t)m, words.data()));
    const uint32_t bad = IRT_FLAG_NONCONVERGED | IRT_FLAG_LENGTH_LIMIT | IRT_FLAG_SELF_COLLISION | IRT_FLAG_BAD_STATE;
    auto tip_error = [&](const double *t) {
      double e2 = 0.0;
      for (int c = 0; c < 3; c++) e2 += (t[c] - request[c]) * (t[c] - request[c]);
      return std::sqrt(e2);
    };
    std::vector<char> valid(m);
    std::vector<double> err(m);
    auto result = [&](size_t i) {
      IKResult r;
      r.controls = finals[i]; r.tip_position = {tips[3 * i], tips[3 * i + 1], tips[3 * i + 2]};
      r.neighbor = starts[i]; r.error = err[i]; r.index = i; r.vertex = nb[i];
      r.lockstep_batches = batches; r.fk_requests = requests;
      return r;
    };
    for (size_t i = 0; i < m; i++) {
      valid[i] = !(flags[i] & bad) && !((words[i >> 5] >> (i & 31)) & 1u);
      err[i] = tip_error(&tips[3 * i]);
    }
    if (!auto_add) {
      std::optional<IKResult> best;
      for (size_t i = 0; i < m; i++) {
        if (!valid[i]) continue;
        if (err[i] < tolerance) return result(i);                // "we've found a good one!"
        if (!best || err[i] < best->error) { best = result(i); best->accepted = false; }
      }
      if (best) return best;                                     // "returning closest valid one"
    }

    // ---- the would-be edges: sources per result in the reference's order; the validity look-ups and removals
    // are replayed on a copy first so that ONE until-invalid batch answers every edge the walk may ask for
    build_adjacency();
    struct Row { long s; bool is_self, ok; };   // s = -1: the result's own temporary vertex
    std::vector<std::vector<double>> bounded(m);
    std::vector<long> own(m);
    for (size_t i = 0; i < m; i++) { bounded[i] = enforceBounds(finals[i]); own[i] = findState(bounded[i]); }
    std::vector<char> removed = vertex_removed_;
    std::vector<char> in_first(m, 0);
    for (size_t i = 0; i < m; i++) in_first[i] = !auto_add || err[i] < tolerance;
    auto plan_result = [&](size_t i) {
      std::vector<Row> rows;
      for (long s : ikNearest(bounded[i], own[i], nb[i], accurate, removed)) {
        const bool is_self = s < 0 || s == own[i];
        const bool ok = s < 0 ? (bool)valid[i] : computeVertexValidity((size_t)s);
        if (!ok && !is_self) removed[(size_t)s] = 1;
        rows.push_back({s, is_self, ok});
      }
      return rows;
    };
    std::vector<std::vector<Row>> plan1(m), plan3(m);
    std::vector<std::pair<size_t, long>> jobs;
    auto add_job = [&](size_t i, long s) {
      if (std::find(jobs.begin(), jobs.end(), std::make_pair(i, s)) == jobs.end()) jobs.emplace_back(i, s);
    };
    for (size_t i = 0; i < m; i++) {
      if (!in_first[i] || (auto_add && own[i] >= 0 && outDegree((size_t)own[i]) > 0)) continue;
      plan1[i] = plan_result(i);
      for (auto &r : plan1[i]) if (r.ok && !(auto_add && r.is_self)) add_job(i, r.s);
    }
    if (auto_add)   // the fallback asks again for the results the loop above left without sources
      for (size_t i = 0; i < m; i++) {
        bool any = false;
        for (auto &r : plan1[i]) any = any || (r.ok && !r.is_self);
        if (own[i] < 0 && !any) {
          plan3[i] = plan_result(i);
          for (auto &r : plan3[i]) if (r.ok) add_job(i, r.s);
        }
      }
    struct Partial { bool fully_valid; std::vector<double> last_valid; collision::Point tip; double error; };
    std::map<std::pair<size_t, long>, Partial> pe_of;
    if (!jobs.empty()) {
      const size_t nj = jobs.size();
      std::vector<double> a(nj * S), b(nj * S), t_last(nj);
      std::vector<uint32_t> fl(nj);
      for (size_t j = 0; j < nj; j++) {
        const std::vector<double> &src = jobs[j].second < 0 ? bounded[jobs[j].first] : states_[(size_t)jobs[j].second];
        std::copy(src.begin(), src.end(), a.begin() + j * S);
        std::copy(finals[jobs[j].first].begin(), finals[jobs[j].first].end(), b.begin() + j * S);
      }
      irt::check(ctx_, irt_voxelize_edges_until_invalid(ctx_, robot_.handle(), &space_, a.data(), b.data(), (int)S,
                                                        (int64_t)nj, env_, scratch, fl.data(), t_last.data(), nullptr));
      std::vector<std::vector<double>> lv(nj);
      for (size_t j = 0; j < nj; j++)
        lv[j] = interpolate_states(robot_, std::vector<double>(a.begin() + j * S, a.begin() + (j + 1) * S),
                                   std::vector<double>(b.begin() + j * S, b.begin() + (j + 1) * S), t_last[j]);
      auto shapes = robot_.shape_batch(lv);                      // last_backbone.back()
      for (size_t j = 0; j < nj; j++) {
        const collision::Point tip = shapes[j].p.back();
        pe_of[jobs[j]] = Partial{!(fl[j] & IRT_FLAG_PARTIAL), lv[j], tip, tip_error(tip.data())};
      }
    }
    // the valid sources of a result in order, with the removals the reference makes on the way; fn returns true
    // where the reference returns (nothing after that point is looked at)
    auto walk = [&](const std::vector<Row> &rows, const std::function<bool(long, bool)> &fn) {
      for (auto &r : rows) {
        if (!r.ok) { if (!r.is_self) vertex_removed_[(size_t)r.s] = 1; continue; }
        if (fn(r.s, r.is_self)) return true;
      }
      return false;
    };
    auto stepped = [&](size_t i, long s, const Partial &e) {
      IKResult r = result(i);
      r.controls = e.last_valid; r.tip_position = e.tip; r.error = e.error;
      r.accepted = false; r.stepped_back = true; r.source = s;
      return r;
    };
    if (!auto_add) {   // "All IKs are in collision, stepping them backwards"
      std::optional<IKResult> best;
      for (size_t i = 0; i < m; i++)
        walk(plan1[i], [&](long s, bool) {
          const Partial &e = pe_of.at({i, s});
          if (!best || e.error < best->error) best = stepped(i, s, e);
          return false;
        });
      return best;
    }
    auto keep_vertex = [&](size_t i) {   // the result's vertex stays in the roadmap with its caches
      if (own[i] >= 0) {
        for (int c = 0; c < 3; c++) tips_[3 * (size_t)own[i] + c] = tips[3 * i + c];
        nn_tips_.stale = true;
        vertex_validity_[(size_t)own[i]] = VALIDITY_TRUE;
        return (size_t)own[i];
      }
      return appendVertex(bounded[i], &tips[3 * i]);
    };
    std::vector<std::vector<long>> nearest(m);
    for (size_t i = 0; i < m; i++) {
      if (!in_first[i]) continue;
      if (own[i] >= 0 && outDegree((size_t)own[i]) > 0) {       // "IK result already part of the roadmap"
        IKResult r = result(i); r.already_in_roadmap = true;
        return r;
      }
      IKResult r = result(i);
      const bool done = walk(plan1[i], [&](long s, bool is_self) {
        if (is_self) {                                           // "State already in the roadmap, returning it."
          const size_t v = keep_vertex(i);
          if (own[i] < 0) r.added_vertex = (long)v; else r.already_in_roadmap = true;
          return true;
        }
        nearest[i].push_back(s);
        if (pe_of.at({i, s}).fully_valid) {                      // connect source -- result vertex
          const size_t v = keep_vertex(i);
          appendEdge((size_t)s, v, VALIDITY_TRUE);
          if (own[i] < 0) r.added_vertex = (long)v;
          r.source = s;
          return true;
        }
        return false;
      });
      if (done) return r;
    }
    // "All IKs rejected, finding closest collision-free connection"
    std::optional<IKResult> best;
    const Partial *best_pe = nullptr;
    for (size_t i = 0; i < m; i++) {
      if (nearest[i].empty()) {
        if (own[i] >= 0) continue;                               // "already part of the roadmap, no need to connect it"
        walk(plan3[i], [&](long s, bool) { nearest[i].push_back(s); return false; });
      }
      for (long s : nearest[i]) {
        const Partial &e = pe_of.at({i, s});
        if (!best || e.error < best->error) { best = stepped(i, s, e); best_pe = &e; }
      }
    }
    if (!best) return best;
    const size_t bi = best->index;
    const long s = best->source;
    best->neighbor = s < 0 ? bounded[bi] : states_[(size_t)s];
    long v = findState(best_pe->last_valid);
    if (v < 0) {
      // addMilestone(state, true): connected lazily to its connection-strategy neighbours (itself not yet in nn_)
      const std::vector<size_t> conn = connectionNeighbors(best_pe->last_valid);
      v = (long)appendVertex(best_pe->last_valid, &tips[3 * bi]);   // the reference caches the IK RESULT's tip here
      for (size_t u : conn) appendEdge((size_t)v, u, VALIDITY_UNKNOWN);
      best->added_vertex = v;
    } else {
      for (int c = 0; c < 3; c++) tips_[3 * (size_t)v + c] = tips[3 * bi + c];
      nn_tips_.stale = true;
      vertex_validity_[(size_t)v] = VALIDITY_TRUE;
    }
    if (s >= 0 && v != s) {
      const long e = edgeIndex((size_t)s, (size_t)v);
      if (e < 0) appendEdge((size_t)s, (size_t)v, VALIDITY_TRUE); else edge_validity_[(size_t)e] = VALIDITY_TRUE;
      if (!lazy_add) {   // every edge of the vertex is validated now, the invalid ones removed
        build_adjacency();
        std::vector<size_t> todo;
        for_neighbors((size_t)v, [&](size_t, size_t eid) {
          if (!edge_removed_[eid] && !(edge_validity_[eid] & VALIDITY_TRUE)) todo.push_back(eid);
        });
        if (!todo.empty()) {
          const std::vector<unsigned> val = checkEdgesNow(todo);
          for (size_t j = 0; j < todo.size(); j++) {
            edge_unchecked_.erase(todo[j]);
            if (val[j] & VALIDITY_TRUE) edge_validity_[todo[j]] = VALIDITY_TRUE;
            else edge_removed_[todo[j]] = 1;
          }
        }
      }
    }
    return best;
  }

  /// addMilestone(state, connect) (.cpp:1854-1885): the vertex of an equal state when the roadmap has one
  /// (tryAddToGraph), else a new vertex with VALIDITY_UNKNOWN, lazily connected -- edges of unknown validity -- to
  /// its connection-strategy neighbours (the vertex itself is not in nn_ yet).  Nothing is voxelised here: queries
  /// check the new items when they first ask for them.  Returns (vertex, was_added).
  std::pair<size_t, bool> addMilestone(const std::vector<double> &state, bool connect = true) {
    if (state.size() != robot_.state_size()) throw std::invalid_argument("State is not the right size");
    build_adjacency();
    const long have = findState(state);
    if (have >= 0) return {(size_t)have, false};
    const std::vector<size_t> conn = connect ? connectionNeighbors(state) : std::vector<size_t>();
    if (tips_.size() != 3 * states_.size()) precomputeVertexVoxelCache();
    const collision::Point tip = robot_.forward_kinematics(state).back();
    const size_t v = appendVertex(state, tip.data(), VALIDITY_UNKNOWN);
    for (size_t u : conn) appendEdge(v, u, VALIDITY_UNKNOWN);
    return {v, true};
  }
  struct ChainedStep {
    IKResult ik;                              // roadmapIk's result for the request
    bool exact = false;                       // false: no path, the plan stays put ("Could not reach goal, no solution")
    std::vector<size_t> path;                 // roadmap vertices start .. goal
    std::vector<std::vector<double>> plan;    // their states
    size_t searches = 0, start_vertex = 0, goal_vertex = 0;
    size_t n_vertices = 0, n_edges = 0;       // size of the roadmap the search ran on
    double tip_error = 0.0;                   // of the plan's last state
  };
  /// The milestone loop of apps/roadmap_chained_plan.cpp:535-679: for every requested tip position roadmapIk gives
  /// the goal configuration, start and goal join the roadmap as milestones (solvePrep, .cpp:2978-3025),
  /// solveWithRoadmap plans between them, and the plan's last state is where the next milestone starts (unless
  /// common_start).  Everything it asks of the device is a batch or a look-up.
  std::vector<ChainedStep> chainedPlan(const std::vector<double> &start_state, const std::vector<collision::Point> &requests,
                                       double tolerance, size_t k, const tip_control::IkSolver &solver,
                                       unsigned opt = RMAP_IK_AUTO_ADD, int mode = IRT_JAC_LEVMAR_CENTRAL,
                                       double delta = 1e-6, bool common_start = false) {
    std::vector<double> current = start_state;
    std::vector<ChainedStep> out;
    for (const collision::Point &request : requests) {
      auto ik = roadmapIk(request, tolerance, k, solver, mode, delta, opt);
      if (!ik) throw std::runtime_error("no IK results returned");
      ChainedStep st;
      st.ik = *ik;
      st.start_vertex = addMilestone(common_start ? start_state : current).first;
      st.goal_vertex = addMilestone(ik->controls).first;
      st.n_vertices = states_.size(); st.n_edges = edges_.size();
      st.path = solveWithRoadmap(st.start_vertex, st.goal_vertex, &st.searches);
      st.exact = !st.path.empty();
      if (st.exact) for (size_t v : st.path) st.plan.push_back(states_[v]);
      else st.plan.push_back(states_[st.start_vertex]);
      const collision::Point tip = robot_.forward_kinematics(st.plan.back()).back();
      double e2 = 0.0;
      for (int c = 0; c < 3; c++) e2 += (tip[c] - request[c]) * (tip[c] - request[c]);
      st.tip_error = std::sqrt(e2);
      if (!common_start) current = st.plan.back();
      out.push_back(std::move(st));
    }
    return out;
  }

private:
  /// tryAddToGraph (.cpp:2777-2801): the vertex whose state equals x (si_->equalStates), else -1
  long findState(const std::vector<double> &x) const {
    const double tol = 2.0 * std::numeric_limits<double>::epsilon();
    for (size_t v = 0; v < states_.size(); v++) {
      if (v < vertex_removed_.size() && vertex_removed_[v]) continue;
      bool same = true;
      for (size_t c = 0; c < x.size() && same; c++) same = std::fabs(states_[v][c] - x[c]) <= tol;
      if (same) return (long)v;
    }
    return -1;
  }
  size_t outDegree(size_t v) {
    build_adjacency();
    size_t c = 0;
    for_neighbors(v, [&](size_t nbr, size_t eid) { c += !edge_removed_[eid] && !vertex_removed_[nbr]; });
    return c;
  }
  /// `nearest` of .cpp:3238-3246, 3340-3349, 3470-3478; -1 stands for the result's own temporary vertex
  std::vector<long> ikNearest(const std::vector<double> &x, long own, size_t ik_neighbor, bool accurate,
                              const std::vector<char> &removed) const {
    if (!accurate) return {(long)ik_neighbor};
    if (irt_nnset *nn = nearestSet(false, k_)) {
      const std::vector<uint32_t> words = maskWords(removed);
      std::vector<int64_t> idx(k_);
      std::vector<double> dist(k_);
      irt::check(ctx_, irt_nnset_knn(ctx_, nn, x.data(), 1, (int)k_, getRange(), words.data(), idx.data(), dist.data()));
      std::vector<long> out;
      size_t zeros = 0;
      for (size_t j = 0; j < k_ && idx[j] >= 0; j++) {
        out.push_back((long)idx[j]);
        zeros += dist[j] <= 0.0;
      }
      if (own < 0 && 0.0 <= getRange()) {   // the temporary vertex: distance 0, after every item at distance 0
        out.insert(out.begin() + (long)zeros, -1L);
        if (out.size() > k_) out.pop_back();
      }
      if (std::find(out.begin(), out.end(), (long)ik_neighbor) == out.end()) out.push_back((long)ik_neighbor);
      return out;
    }
    std::vector<std::pair<double, size_t>> d;
    for (size_t u = 0; u < states_.size(); u++)
      if (!removed[u]) d.emplace_back(distance(x, states_[u]), u);
    if (own < 0) d.emplace_back(0.0, states_.size());            // the temporary vertex: distance 0, the highest index
    const size_t kk = std::min(k_, d.size());
    std::partial_sort(d.begin(), d.begin() + kk, d.end());
    std::vector<long> out;
    for (size_t j = 0; j < kk && d[j].first <= getRange(); j++)
      out.push_back(d[j].second == states_.size() ? -1L : (long)d[j].second);
    if (std::find(out.begin(), out.end(), (long)ik_neighbor) == out.end()) out.push_back((long)ik_neighbor);
    return out;
  }
  size_t appendVertex(const std::vector<double> &state, const double *tip, unsigned validity = VALIDITY_TRUE) {
    build_adjacency();
    states_.push_back(state);
    vertex_validity_.push_back(validity);
    vertex_removed_.push_back(0);
    tips_.insert(tips_.end(), tip, tip + 3);
    if (!(validity & VALIDITY_TRUE)) vertex_unchecked_.insert(states_.size() - 1);
    return states_.size() - 1;                                   // vflags_ is now shorter: the cache lacks the vertex
  }
  void appendEdge(size_t a, size_t b, unsigned validity) {
    build_adjacency();
    edges_.emplace_back(a, b);
    edge_validity_.push_back(validity);
    edge_removed_.push_back(0);
    adj_extra_[a].emplace_back(b, edges_.size() - 1);
    adj_extra_[b].emplace_back(a, edges_.size() - 1);
    adj_extra_count_++;
    if (!(validity & VALIDITY_TRUE)) edge_unchecked_.insert(edges_.size() - 1);
  }
  /// voxelizeVertex + collides for a few vertices (.cpp:2607-2618, 2803-2837)
  std::vector<unsigned> checkVerticesNow(const std::vector<size_t> &ids) {
    const size_t S = robot_.state_size(), m = ids.size();
    std::vector<double> flat(m * S);
    for (size_t i = 0; i < m; i++) std::copy(states_[ids[i]].begin(), states_[ids[i]].end(), flat.begin() + i * S);
    std::vector<uint32_t> fl(m), w((m + 31) / 32 + 1, 0);
    irt_setstore *scratch = nullptr;
    irt_grid g = env_voxels_.grid(venv_.inv_rotation);
    irt::check(ctx_, irt_setstore_create(ctx_, &g, &scratch));
    std::shared_ptr<irt_setstore> guard(scratch, [](irt_setstore *x) { irt_setstore_destroy(x); });
    irt::check(ctx_, irt_voxelize_vertices(ctx_, robot_.handle(), flat.data(), (int)S, (int64_t)m, scratch, fl.data(), nullptr));
    irt::check(ctx_, irt_check_sets(ctx_, scratch, env_, 0, (int64_t)m, w.data()));
    const uint32_t bad = IRT_FLAG_NONCONVERGED | IRT_FLAG_LENGTH_LIMIT | IRT_FLAG_SELF_COLLISION | IRT_FLAG_BAD_STATE;
    std::vector<unsigned> out(m);
    for (size_t i = 0; i < m; i++) out[i] = (!(fl[i] & bad) && !((w[i >> 5] >> (i & 31)) & 1u)) ? VALIDITY_TRUE : VALIDITY_UNKNOWN;
    return out;
  }
  /// voxelizeEdge + collides for a few edges (.cpp:2620-2631, 2879-2902)
  std::vector<unsigned> checkEdgesNow(const std::vector<size_t> &ids) {
    const size_t S = robot_.state_size(), m = ids.size();
    std::vector<double> a(m * S), b(m * S);
    for (size_t i = 0; i < m; i++) {
      std::copy(states_[edges_[ids[i]].first].begin(), states_[edges_[ids[i]].first].end(), a.begin() + i * S);
      std::copy(states_[edges_[ids[i]].second].begin(), states_[edges_[ids[i]].second].end(), b.begin() + i * S);
    }
    std::vector<uint32_t> fl(m), w((m + 31) / 32 + 1, 0);
    irt_setstore *scratch = nullptr;
    irt_grid g = env_voxels_.grid(venv_.inv_rotation);
    irt::check(ctx_, irt_setstore_create(ctx_, &g, &scratch));
    std::shared_ptr<irt_setstore> guard(scratch, [](irt_setstore *x) { irt_setstore_destroy(x); });
    irt::check(ctx_, irt_voxelize_edges(ctx_, robot_.handle(), &space_, a.data(), b.data(), (int)S, (int64_t)m, scratch,
                                        fl.data(), nullptr, nullptr));
    irt::check(ctx_, irt_check_sets(ctx_, scratch, env_, 0, (int64_t)m, w.data()));
    std::vector<unsigned> out(m);
    for (size_t i = 0; i < m; i++)
      out[i] = (!(fl[i] & IRT_FLAG_PARTIAL) && !((w[i >> 5] >> (i & 31)) & 1u)) ? VALIDITY_TRUE : VALIDITY_UNKNOWN;
    return out;
  }
  size_t removed_count() const {
    size_t c = 0;
    for (char x : vertex_removed_) c += x != 0;
    for (char x : edge_removed_) c += x != 0;
    return c;
  }
  void build_adjacency() {
    const size_t n = states_.size(), m = edges_.size();
    // edges appended one query at a time (roadmapIk / addMilestone) live in per-vertex lists next to the CSR
    // (adj_extra_) instead of costing a rebuild each; folded in when their share passes 1/64
    if (adj_edges_ != (size_t)-1 && adj_edges_ <= m && m - adj_edges_ == adj_extra_count_ &&
        m - adj_edges_ <= std::max<size_t>(1024, adj_edges_ / 64))
      return;
    adj_extra_.clear(); adj_extra_count_ = 0;
    adj_ptr_.assign(n + 1, 0);
    for (auto &e : edges_) { adj_ptr_[e.first + 1]++; adj_ptr_[e.second + 1]++; }
    for (size_t i = 0; i < n; i++) adj_ptr_[i + 1] += adj_ptr_[i];
    adj_nbr_.assign(2 * m, 0); adj_eid_.assign(2 * m, 0);
    std::vector<size_t> cur(adj_ptr_.begin(), adj_ptr_.end() - 1);
    for (size_t i = 0; i < m; i++) {
      adj_nbr_[cur[edges_[i].first]] = edges_[i].second; adj_eid_[cur[edges_[i].first]++] = i;
      adj_nbr_[cur[edges_[i].second]] = edges_[i].first; adj_eid_[cur[edges_[i].second]++] = i;
    }
    adj_edges_ = m;
    if (vertex_removed_.size() != n) vertex_removed_.assign(n, 0);
    if (edge_removed_.size() != m) edge_removed_.assign(m, 0);
  }
  /// fn(neighbour, edge id) for every edge at v: its CSR row, then the edges appended since the CSR was built
  template <class F>
  void for_neighbors(size_t v, F &&fn) const {
    if (v + 1 < adj_ptr_.size())
      for (size_t q = adj_ptr_[v]; q < adj_ptr_[v + 1]; q++) fn(adj_nbr_[q], adj_eid_[q]);
    auto it = adj_extra_.find(v);
    if (it != adj_extra_.end())
      for (auto &ne : it->second) fn(ne.first, ne.second);
  }
  /// an empty store on the environment's grid, destroyed with its last owner
  std::shared_ptr<irt_setstore> scratch_store() {
    irt_setstore *st = nullptr;
    irt_grid g = env_voxels_.grid(venv_.inv_rotation);
    irt::check(ctx_, irt_setstore_create(ctx_, &g, &st));
    return std::shared_ptr<irt_setstore>(st, [](irt_setstore *x) { irt_setstore_destroy(x); });
  }
  void clear_store(irt_setstore *st) {
    const uint64_t off = 0;
    const uint32_t key = 0;
    const uint64_t bits = 0;
    irt::check(ctx_, irt_setstore_import(ctx_, st, 0, &off, &key, &bits));
  }
  /// a device copy of states_ or tips_ for the k-NN queries: `rows` of them are on the device; `stale` = the host
  /// array was replaced or written in place since (rebuilt before the next query; appends are appended)
  struct NnMirror { irt_nnset *set = nullptr; size_t rows = 0; bool stale = false; };
  /// the device set mirroring tips_ (tips) or states_, brought up to date, or nullptr where the host scans answer
  /// (k outside [1, IRT_KNN_MAX_K])
  irt_nnset *nearestSet(bool tips, size_t k) const {
    if (k < 1 || k > IRT_KNN_MAX_K) return nullptr;
    NnMirror &m = tips ? nn_tips_ : nn_states_;
    const size_t S = robot_.state_size(), rows = tips ? tips_.size() / 3 : states_.size();
    if (m.stale || m.rows > rows) {
      irt::check(ctx_, irt_nnset_clear(ctx_, m.set));
      m.rows = 0;
      m.stale = false;
    }
    if (rows > m.rows) {
      std::vector<double> flat;
      if (tips) {
        flat.assign(tips_.begin() + 3 * m.rows, tips_.end());
      } else {
        flat.resize((rows - m.rows) * S);
        for (size_t i = m.rows; i < rows; i++) std::copy(states_[i].begin(), states_[i].end(), flat.begin() + (i - m.rows) * S);
      }
      irt::check(ctx_, irt_nnset_append(ctx_, m.set, flat.data(), (int64_t)(rows - m.rows)));
      m.rows = rows;
    }
    return m.set;
  }
  static std::vector<uint32_t> maskWords(const std::vector<char> &flags) {
    std::vector<uint32_t> w(flags.size() / 32 + 1, 0);
    for (size_t i = 0; i < flags.size(); i++)
      if (flags[i]) w[i >> 5] |= 1u << (i & 31);
    return w;
  }
  /// connectionStrategy_ of a state that is not in nn_ yet (addMilestone): the k nearest milestones within the range,
  /// removed ones left out, nearest first
  std::vector<size_t> connectionNeighbors(const std::vector<double> &x) {
    std::vector<size_t> out;
    if (irt_nnset *nn = nearestSet(false, k_)) {
      const std::vector<uint32_t> words = maskWords(vertex_removed_);
      std::vector<int64_t> idx(k_);
      irt::check(ctx_, irt_nnset_knn(ctx_, nn, x.data(), 1, (int)k_, getRange(), words.data(), idx.data(), nullptr));
      for (int64_t i : idx)
        if (i >= 0) out.push_back((size_t)i);
      return out;
    }
    std::vector<std::pair<double, size_t>> d;
    for (size_t u = 0; u < states_.size(); u++)
      if (!vertex_removed_[u]) d.emplace_back(distance(x, states_[u]), u);
    const size_t kk = std::min(k_, d.size());
    std::partial_sort(d.begin(), d.begin() + kk, d.end());
    for (size_t j = 0; j < kk && d[j].first <= getRange(); j++) out.push_back(d[j].second);
    return out;
  }
  /// exact k nearest of v among all milestones (v included, like nn_->nearestK), cut at the range
  std::vector<size_t> nearestKBounded(size_t v) const {
    std::vector<std::pair<double, size_t>> d(states_.size());
    for (size_t i = 0; i < states_.size(); i++) d[i] = {distance(states_[v], states_[i]), i};
    const size_t k = std::min(k_, d.size());
    std::partial_sort(d.begin(), d.begin() + k, d.end());
    std::vector<size_t> out;
    const double bound = getRange();
    for (size_t i = 0; i < k && d[i].first <= bound; i++) out.push_back(d[i].second);
    return out;
  }
  /// updateEnvironment for the vertex (vert) or edge table: the items whose validity bit flipped, ascending
  std::vector<size_t> patchTable(bool vert, irt_env *env_old) {
    std::vector<unsigned> &table = vert ? vertex_validity_ : edge_validity_;
    std::set<size_t> &unchecked = vert ? vertex_unchecked_ : edge_unchecked_;
    const size_t n_items = vert ? states_.size() : edges_.size();
    std::vector<size_t> flipped;
    if (!(vert ? vertex_swept_ : edge_swept_)) {
      table.assign(n_items, VALIDITY_UNKNOWN);
      unchecked.clear();
      return flipped;
    }
    std::vector<uint32_t> &words = vert ? vwords_ : ewords_;
    const size_t n = vert ? vwords_n_ : ewords_n_;
    if (n > 0) {
      irt_setstore *st = vert ? vstore_ : estore_;
      if ((size_t)irt_setstore_num_sets(st) < n) {   // the cache was cleared since the sweep: the same sets again
        if (vert) precomputeVertexVoxelCache(); else precomputeEdgeVoxelCache();
      }
      const std::vector<uint32_t> &flags = vert ? vflags_ : eflags_;
      const uint32_t mask = vert ? kVertexInvalid : IRT_FLAG_PARTIAL;
      irt_setindex *ix = setIndex(vert, n);
      std::vector<int64_t> hits(1024);
      int64_t nh = 0;
      int rc = irt_check_sets_changed(ctx_, st, ix, env_old, env_, 0, (int64_t)n, words.data(), hits.data(),
                                      (int64_t)hits.size(), &nh, nullptr);
      if (rc == IRT_ERR_CAPACITY) {   // more flips than the buffer holds: words are unchanged, try once more
        hits.resize((size_t)nh);
        rc = irt_check_sets_changed(ctx_, st, ix, env_old, env_, 0, (int64_t)n, words.data(), hits.data(),
                                    (int64_t)hits.size(), &nh, nullptr);
      }
      irt::check(ctx_, rc);
      for (int64_t k = 0; k < nh; k++) {
        const size_t i = (size_t)hits[(size_t)k];
        const bool hit = (words[i >> 5] >> (i & 31)) & 1u;
        const unsigned v = (!hit && !(flags[i] & mask)) ? VALIDITY_TRUE : VALIDITY_UNKNOWN;
        if ((table[i] & VALIDITY_TRUE) != v) flipped.push_back(i);
        table[i] = v;
      }
    }
    // items without a cached set when the table was swept, or added since with a known verdict: one scratch batch
    std::vector<size_t> ids;
    for (size_t i = n; i < n_items; i++)
      if (!unchecked.count(i)) ids.push_back(i);
    if (!ids.empty()) {
      const std::vector<unsigned> now = vert ? checkVerticesNow(ids) : checkEdgesNow(ids);
      for (size_t k = 0; k < ids.size(); k++) {
        if ((table[ids[k]] & VALIDITY_TRUE) != (now[k] & VALIDITY_TRUE)) flipped.push_back(ids[k]);
        table[ids[k]] = now[k];
      }
    }
    std::sort(flipped.begin(), flipped.end());
    return flipped;
  }
  /// the inverted index of the vertex or edge cache covering its first n sets, or all but at most maxUncached() of
  /// them: built on first use, rebuilt when the cache was rebuilt since, or when its unindexed tail grew too long
  irt_setindex *setIndex(bool vert, size_t n) {
    irt_setindex *&ix = vert ? vindex_ : eindex_;
    size_t &built = vert ? vindex_build_ : eindex_build_;
    const size_t builds = vert ? vcache_builds_ : ecache_builds_;
    if (!ix || built != builds || (int64_t)n - irt_setindex_num_sets(ix) > (int64_t)max_uncached_) {
      irt_setindex_destroy(ix);
      ix = nullptr;
      irt::check(ctx_, irt_setindex_create(ctx_, vert ? vstore_ : estore_, &ix));
      built = builds;
    }
    return ix;
  }
  /// K3 over every cached set; the verdict words and the number of sets they cover are kept for updateEnvironment
  void sweep(irt_setstore *st, const std::vector<uint32_t> &flags, uint32_t mask, std::vector<unsigned> &validity,
             std::vector<uint32_t> &words, size_t &covered) {
    const int64_t n = irt_setstore_num_sets(st);
    words.assign((n + 31) / 32 + 1, 0);
    covered = (size_t)n;
    if (n > 0) irt::check(ctx_, irt_check_sets(ctx_, st, env_, 0, n, words.data()));
    validity.assign(n, VALIDITY_UNKNOWN);
    for (int64_t i = 0; i < n; i++) {
      const bool hit = (words[i >> 5] >> (i & 31)) & 1u;
      if (!hit && !(flags[i] & mask)) validity[i] = VALIDITY_TRUE;
    }
  }
  const tendon::TendonRobot &robot_;
  const VoxelEnvironment &venv_;
  collision::VoxelOctree env_voxels_;
  irt_space space_;
  irt_ctx *ctx_ = nullptr;
  irt_setstore *vstore_ = nullptr, *estore_ = nullptr;
  irt_env *env_ = nullptr;
  irt_env *env_next_ = nullptr;   // updateEnvironment uploads the next grid here, then swaps it with env_
  static constexpr uint32_t kVertexInvalid =
      IRT_FLAG_NONCONVERGED | IRT_FLAG_LENGTH_LIMIT | IRT_FLAG_SELF_COLLISION | IRT_FLAG_BAD_STATE;
  // the verdict words of the last sweep of each table and the sets they cover; the caches' inverted indices with the
  // cache build they were made from
  std::vector<uint32_t> vwords_, ewords_;
  size_t vwords_n_ = 0, ewords_n_ = 0;
  irt_setindex *vindex_ = nullptr, *eindex_ = nullptr;
  size_t vcache_builds_ = 0, ecache_builds_ = 0, vindex_build_ = 0, eindex_build_ = 0;
  std::vector<std::vector<double>> states_;
  std::vector<std::pair<size_t, size_t>> edges_;
  std::vector<uint32_t> vflags_, eflags_;
  std::vector<double> tips_;
  std::vector<unsigned> vertex_validity_, edge_validity_;
  bool vertex_swept_ = false, edge_swept_ = false;
  size_t sweeps_ = 0, lookups_ = 0, single_checks_ = 0, max_uncached_ = 4096;
  std::set<size_t> vertex_unchecked_, edge_unchecked_;   // joined after the last sweep with VALIDITY_UNKNOWN
  std::vector<char> vertex_removed_, edge_removed_;
  std::vector<size_t> adj_ptr_, adj_nbr_, adj_eid_;
  size_t adj_edges_ = (size_t)-1, adj_extra_count_ = 0;
  std::map<size_t, std::vector<std::pair<size_t, size_t>>> adj_extra_;   // vertex -> (neighbour, edge id) appended since
  Sampler sampler_;
  std::function<std::vector<size_t>(size_t)> connection_;
  std::mt19937 gen_{20220801u};
  size_t k_ = 5;
  double range_ = 0.0;
  mutable NnMirror nn_states_, nn_tips_;   // mutable: ikNearest is const and brings them up to date
};

}  // namespace motion_planning
