// The C++ host mirror's nearest-neighbour questions (interactive-rate-tendons_b200/host/irt_host.hpp), answered by
// irt_nnset_knn on the device, against the host scans they replace, restated here over the public distance():
// createRoadmap's KBoundedStrategy connection (the roadmap's edge list, order included) and nearestTips.  Built and
// run by tests/test_gpu_knn.py against libirt_b200.so.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <random>
#include <set>
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

int main() {
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
  motion_planning::VoxelEnvironment venv;
  motion_planning::VoxelCachedLazyPRM prm(robot, venv, env_vox);
  using PRM = motion_planning::VoxelCachedLazyPRM;

  for (size_t N : {2500, 4000}) {   // growing: the device copy of the states is appended to
    const size_t Nv = prm.states().size(), Ne = prm.edges().size();
    prm.createRoadmap(N, PRM::LazyRoadmap);
    const auto &st = prm.states();
    CHECK(st.size() == N);
    std::set<std::pair<size_t, size_t>> have;
    for (size_t e = 0; e < Ne; e++) have.insert(std::minmax(prm.edges()[e].first, prm.edges()[e].second));
    std::vector<std::pair<size_t, size_t>> want;
    for (size_t v = Nv; v < N; v++) {
      std::vector<std::pair<double, size_t>> d(N);
      for (size_t i = 0; i < N; i++) d[i] = {prm.distance(st[v], st[i]), i};
      std::partial_sort(d.begin(), d.begin() + 5, d.end());
      for (size_t j = 0; j < 5 && d[j].first <= prm.getRange(); j++)
        if (d[j].second != v && have.insert(std::minmax(v, d[j].second)).second) want.emplace_back(v, d[j].second);
    }
    CHECK(prm.edges().size() == Ne + want.size());
    CHECK(std::equal(want.begin(), want.end(), prm.edges().begin() + Ne));
    std::printf("createRoadmap(%zu): %zu new edges\n", N, want.size());
  }

  prm.precomputeVertexVoxelCache();
  const std::vector<double> &tips = prm.tipPositions();
  std::mt19937_64 gen(5);
  std::uniform_int_distribution<size_t> pick(0, prm.states().size() - 1);
  std::normal_distribution<double> noise(0.0, 0.003);
  for (int trial = 0; trial < 50; trial++) {
    const size_t v = pick(gen);
    collision::Point req{tips[3 * v] + noise(gen), tips[3 * v + 1] + noise(gen), tips[3 * v + 2] + noise(gen)};
    if (trial % 10 == 0) req = {tips[3 * v], tips[3 * v + 1], tips[3 * v + 2]};
    for (size_t k : {1, 5, 17, 64}) {
      std::vector<std::pair<double, size_t>> d;
      for (size_t u = 0; u < tips.size() / 3; u++) {
        double s = 0.0;
        for (int c = 0; c < 3; c++) s += (tips[3 * u + c] - req[c]) * (tips[3 * u + c] - req[c]);
        d.emplace_back(std::sqrt(s), u);
      }
      std::partial_sort(d.begin(), d.begin() + k, d.end());
      const std::vector<size_t> got = prm.nearestTips(req, k);
      CHECK(got.size() == k);
      for (size_t j = 0; j < k && j < got.size(); j++) CHECK(got[j] == d[j].second);
    }
  }
  if (failures) {
    std::printf("%d failures\n", failures);
    return 1;
  }
  std::printf("knn mirror ok\n");
  return 0;
}
