// extendVoxelCache of the C++ host mirror (interactive-rate-tendons_b200/host/irt_host.hpp): after addMilestone has
// added vertices and lazy edges that the caches lack, extending the caches must give what precompute*VoxelCache gives
// on a fresh planner with the same states and edges -- the same sets, flags and tips -- without rebuilding the
// cached part, and the next sweep must give the fresh planner's validity tables from the caches alone.  Built and
// run by tests/test_extend_voxel_cache_host_logic.py over the test-only stand-in of the C ABI (-DIRT_TEST_OVER_STANDIN,
// with tests/cpp/setstore_append_standin.hpp) and by tests/test_gpu_setstore_append.py against libirt_b200.so.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstdio>
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

static void check_same_caches(const PRM &a, const PRM &b) {
  CHECK(a.vertexVoxelCacheSize() == b.vertexVoxelCacheSize());
  CHECK(a.edgeVoxelCacheSize() == b.edgeVoxelCacheSize());
  CHECK(a.vertexFlags() == b.vertexFlags());
  CHECK(a.edgeFlags() == b.edgeFlags());
  CHECK(a.tipPositions() == b.tipPositions());
  for (size_t i = 0; i < a.vertexVoxelCacheSize() && i < b.vertexVoxelCacheSize(); i++)
    CHECK(a.vertexVoxels(i) == b.vertexVoxels(i));
  for (size_t i = 0; i < a.edgeVoxelCacheSize() && i < b.edgeVoxelCacheSize(); i++)
    CHECK(a.edgeVoxels(i) == b.edgeVoxels(i));
}

int main(int argc, char **argv) {
  const size_t n_roadmap = argc > 1 ? (size_t)std::atoi(argv[1]) : 60;
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
  collision::VoxelOctree env_vox(128);
  env_vox.set_xlim(-0.21, 0.21); env_vox.set_ylim(-0.21, 0.21); env_vox.set_zlim(-0.21, 0.21);
  env_vox.add_sphere(collision::Sphere{{0.05, 0.0, 0.12}, 0.03});
  motion_planning::VoxelEnvironment venv;
  PRM prm(robot, venv, env_vox);
  prm.createRoadmap(n_roadmap, PRM::VoxelizeVertices);
  prm.precomputeVoxelCache();
  prm.precomputeValidity();
  const size_t nv0 = prm.states().size(), ne0 = prm.edges().size();

  // newcomers: milestones near roadmap states, lazily connected
  std::mt19937_64 gen(11);
  std::normal_distribution<double> noise(0.0, 0.5);
  for (int m = 0; m < 12; m++) {
    std::vector<double> x = prm.states()[(size_t)m * 3 % nv0];
    for (size_t j = 0; j + 2 < x.size(); j++) x[j] = std::max(0.0, x[j] + noise(gen));
    prm.addMilestone(x);
  }
  const size_t nv = prm.states().size(), ne = prm.edges().size();
  CHECK(nv > nv0 && ne > ne0);
  CHECK(prm.vertexFlags().size() == nv0 && prm.edgeFlags().size() == ne0);

  prm.extendVoxelCache();
  CHECK(prm.vertexFlags().size() == nv && prm.edgeFlags().size() == ne);
  CHECK(prm.vertexVoxelCacheSize() == nv && prm.edgeVoxelCacheSize() == ne);

  PRM fresh(robot, venv, env_vox);
  fresh.setRoadmap(prm.states(), prm.edges());
  fresh.precomputeVoxelCache();
  check_same_caches(prm, fresh);

  // the next sweep covers every item from the caches: no scratch batch, the fresh planner's tables
  prm.clearValidity();
  prm.precomputeValidity();
  fresh.precomputeValidity();
  CHECK(prm.vertexValidity() == fresh.vertexValidity());
  CHECK(prm.edgeValidity() == fresh.edgeValidity());
  CHECK(prm.vertexFlags().size() == nv && prm.edgeFlags().size() == ne);

  // nothing to extend: a no-op; a cleared cache is built whole
  prm.extendVoxelCache();
  check_same_caches(prm, fresh);
  prm.clearEdgeVoxelCache();
  prm.extendVoxelCache();
  check_same_caches(prm, fresh);

  if (failures) {
    std::printf("%d failures\n", failures);
    return 1;
  }
  std::printf("extend voxel cache ok: %zu + %zu vertices, %zu + %zu edges\n", nv0, nv - nv0, ne0, ne - ne0);
  return 0;
}
