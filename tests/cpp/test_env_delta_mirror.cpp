// updateEnvironment of the C++ host mirror (interactive-rate-tendons_b200/host/irt_host.hpp): over consecutive blob
// ticks, every look-up must answer what a twin planner answers after setEnvironment + precomputeValidity with the same
// roadmap and caches, a current table must equal the twin's (items still unchecked since the sweep excepted), the
// returned flips must be exactly the items whose VALIDITY_TRUE bit changed, and no sweep may be counted.  Covered:
// current and non-current tables, tail items (addMilestone), caches extended after the sweep, and the index rebuilt
// after precomputeVoxelCache.  Built and run by tests/test_env_delta_host_logic.py over the test-only stand-in of the
// C ABI (-DIRT_TEST_OVER_STANDIN, with tests/cpp/env_delta_standin.hpp) and by tests/test_gpu_env_delta.py against
// libirt_b200.so.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <random>
#include <vector>

#include "../../interactive-rate-tendons_b200/host/irt_host.hpp"

static int failures = 0;
#define CHECK(cond)                                                         \
  do {                                                                      \
    if (!(cond)) {                                                          \
      std::printf("FAIL %s:%d: %s\n", __FILE__, __LINE__, #cond);           \
      failures++;                                                           \
    }                                                                       \
  } while (0)

using PRM = motion_planning::VoxelCachedLazyPRM;

// XOR a ball of voxels (centres within r of c) into the grid: the replanning tick of bench.py (workloads.toggle_blob)
static void toggle_blob(collision::VoxelOctree &v, const collision::Point &c, double r) {
  const double lo[3] = {v.xlim().first, v.ylim().first, v.zlim().first};
  const double d = v.dx();
  const long N = (long)v.Nx();
  long a[3], b[3];
  for (int k = 0; k < 3; k++) {
    a[k] = std::max(0L, (long)std::floor((c[k] - r - lo[k]) / d));
    b[k] = std::min(N - 1, (long)std::floor((c[k] + r - lo[k]) / d));
  }
  for (long x = a[0]; x <= b[0]; x++)
    for (long y = a[1]; y <= b[1]; y++)
      for (long z = a[2]; z <= b[2]; z++) {
        const double p[3] = {lo[0] + (x + 0.5) * d, lo[1] + (y + 0.5) * d, lo[2] + (z + 0.5) * d};
        const double dd = std::sqrt((p[0] - c[0]) * (p[0] - c[0]) + (p[1] - c[1]) * (p[1] - c[1]) +
                                    (p[2] - c[2]) * (p[2] - c[2]));
        if (dd > r) continue;
        v.set_block(x / 4, y / 4, z / 4,
                    v.block(x / 4, y / 4, z / 4) ^ collision::VoxelOctree::bitmask(x % 4, y % 4, z % 4));
      }
}

static std::vector<size_t> changed(const std::vector<unsigned> &a, const std::vector<unsigned> &b) {
  std::vector<size_t> out;
  for (size_t i = 0; i < a.size() && i < b.size(); i++)
    if ((a[i] & PRM::VALIDITY_TRUE) != (b[i] & PRM::VALIDITY_TRUE)) out.push_back(i);
  return out;
}

// the twin's tables after setEnvironment + precomputeValidity; items in `skip` (unchecked) are not compared
static void check_like_twin(PRM &prm, PRM &twin, const std::vector<char> &vskip, const std::vector<char> &eskip) {
  CHECK(prm.vertexValidity().size() == twin.vertexValidity().size());
  CHECK(prm.edgeValidity().size() == twin.edgeValidity().size());
  for (size_t i = 0; i < prm.vertexValidity().size() && i < twin.vertexValidity().size(); i++)
    if (!vskip[i]) CHECK(prm.vertexValidity()[i] == twin.vertexValidity()[i]);
  for (size_t i = 0; i < prm.edgeValidity().size() && i < twin.edgeValidity().size(); i++)
    if (!eskip[i]) CHECK(prm.edgeValidity()[i] == twin.edgeValidity()[i]);
}

int main(int argc, char **argv) {
  const size_t n_roadmap = argc > 1 ? (size_t)std::atoi(argv[1]) : 60;
  const int ticks = argc > 2 ? std::atoi(argv[2]) : 6;
  tendon::TendonRobot robot;   // Robot B: 6 helical tendons, retraction + rotation
  robot.specs.dL = 0.003;
  robot.enable_retraction = true;
  robot.enable_rotation = true;
  for (int k = 0; k < 6; k++) {
    tendon::TendonSpecs t;
    t.C = {k * M_PI / 3, (k % 2 ? -1.0 : 1.0) * 2 * M_PI / robot.specs.L};
    t.D = {0.01};
    robot.tendons.push_back(t);
  }
  collision::VoxelOctree env(128);
  env.set_xlim(-0.21, 0.21); env.set_ylim(-0.21, 0.21); env.set_zlim(-0.21, 0.21);
  env.add_sphere(collision::Sphere{{0.05, 0.0, 0.12}, 0.03});
  motion_planning::VoxelEnvironment venv;
  PRM prm(robot, venv, env);
  prm.createRoadmap(n_roadmap, PRM::VoxelizeVertices);
  prm.precomputeVoxelCache();
  prm.precomputeValidity();
  PRM twin(robot, venv, env);

  std::mt19937_64 gen(5);
  std::uniform_real_distribution<double> u(-0.1, 0.1), ur(0.005, 0.015);
  size_t flips_seen = 0;
  for (int t = 0; t < ticks; t++) {
    // tick kinds: 0 blob mid-workspace, 1 blob at the robot base, 2 a milestone joins first (unchecked tail),
    // 3 caches extended after the sweep (tail sets), 4 tables not current, 5 caches rebuilt (index rebuilt)
    const int kind = t % 6;
    const size_t nv0 = prm.states().size(), ne0 = prm.edges().size();
    if (kind == 2) {
      std::vector<double> x = prm.states()[(size_t)t % prm.states().size()];
      x[0] += 0.3;
      prm.addMilestone(x);
    } else if (kind == 3) {
      std::vector<double> x = prm.states()[(size_t)(3 * t) % prm.states().size()];
      x[1] += 0.4;
      prm.addMilestone(x);
      prm.extendVoxelCache();
    } else if (kind == 4) {
      prm.clearValidity();
    } else if (kind == 5) {
      prm.precomputeVoxelCache();
    }
    const collision::Point c = kind == 1 ? collision::Point{u(gen) * 0.05, u(gen) * 0.05, 0.0}
                                         : collision::Point{u(gen), u(gen), 0.1 + u(gen)};
    toggle_blob(env, c, ur(gen));
    const std::vector<unsigned> vold = prm.vertexValidity(), eold = prm.edgeValidity();
    const size_t sweeps = prm.sweepCount();
    // the items addMilestone added in this tick are unchecked (VALIDITY_UNKNOWN until a look-up asks); the look-ups
    // at the end of every tick check everything else
    std::vector<char> vskip(prm.states().size(), 0), eskip(prm.edges().size(), 0);
    std::fill(vskip.begin() + nv0, vskip.end(), 1);
    std::fill(eskip.begin() + ne0, eskip.end(), 1);

    const PRM::EnvironmentChange ch = prm.updateEnvironment(env);
    CHECK(prm.sweepCount() == sweeps);
    twin.setRoadmap(prm.states(), prm.edges());
    twin.precomputeVoxelCache();
    twin.setEnvironment(env);
    if (kind == 4) {   // not current: reset, like setEnvironment
      CHECK(ch.vertices.empty() && ch.edges.empty());
      CHECK(prm.vertexValidity() == twin.vertexValidity() && prm.edgeValidity() == twin.edgeValidity());
    }
    twin.precomputeValidity();
    if (kind != 4) {
      check_like_twin(prm, twin, vskip, eskip);
      CHECK(ch.vertices == changed(vold, prm.vertexValidity()));
      CHECK(ch.edges == changed(eold, prm.edgeValidity()));
      flips_seen += ch.vertices.size() + ch.edges.size();
    }
    // look-ups: every item answers what the twin answers
    for (size_t v = 0; v < prm.states().size(); v++) CHECK(prm.computeVertexValidity(v) == twin.computeVertexValidity(v));
    for (size_t e = 0; e < prm.edges().size(); e++) CHECK(prm.computeEdgeValidity(e) == twin.computeEdgeValidity(e));
    if (kind == 4) prm.precomputeValidity();   // current again for the next tick
  }
  // the same grid again: nothing flips
  const PRM::EnvironmentChange none = prm.updateEnvironment(env);
  CHECK(none.vertices.empty() && none.edges.empty());

  if (failures) {
    std::printf("%d failures\n", failures);
    return 1;
  }
  std::printf("env delta mirror ok: %zu vertices, %zu edges, %d ticks, %zu flips\n", prm.states().size(),
              prm.edges().size(), ticks, flips_seen);
  return 0;
}
