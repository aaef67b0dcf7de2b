// The calls of the reference's examples/connected_component_extraction.cpp (without the viewer and removeInvalidData)
// through the shims: PointCloud3f from PLY, gridDownsample(0.005f), RadiusNeighborhoodSpecification(0.02^2),
// NormalsProximityEvaluator(normals, 2 deg), ConnectedComponentExtraction3f<>(points).segment(nh, ev, 100, n). Prints
// the labels so that tests/test_gpu_segment.py can compare them with the C ABI; also runs the KDTree3f constructor,
// the seeded overload and extractConnectedComponents once each.
#include <cmath>
#include <cstdio>
#include <cilantro/clustering/connected_component_extraction.hpp>
#include <cilantro/utilities/point_cloud.hpp>
#include <cilantro/utilities/timer.hpp>

int main(int argc, char** argv) {
  if (argc < 2) return 2;
  cilantro::PointCloud3f cloud(argv[1]);
  cloud.gridDownsample(0.005f);
  if (!cloud.hasNormals()) return 3;
  cilantro::Timer timer;
  timer.start();
  cilantro::RadiusNeighborhoodSpecification<float> nh(0.02f * 0.02f);
  cilantro::NormalsProximityEvaluator<float, 3> ev(cloud.normals, (float)(2.0 * M_PI / 180.0));
  cilantro::ConnectedComponentExtraction3f<> cce(cloud.points);
  cce.segment(nh, ev, 100, cloud.size());
  timer.stop();
  std::printf("Segmentation time: %gms\n%zu components found\n", timer.getElapsedTime(), cce.getNumberOfClusters());
  // the same through a KDTree3f and through extractConnectedComponents
  cilantro::KDTree3f<> tree(cloud.points);
  cilantro::ConnectedComponentExtraction3f<> cce2(tree);
  cce2.segment(nh, ev, 100, cloud.size());
  auto segs = cilantro::extractConnectedComponents<size_t>(cloud.points, nh, ev, 100, cloud.size());
  if (cce2.getClusterToPointIndicesMap() != cce.getClusterToPointIndicesMap() || segs != cce.getClusterToPointIndicesMap())
    return 4;
  std::vector<size_t> seeds{0};
  cce2.segment(nh, std::vector<size_t>{0}, cilantro::AlwaysTrueEvaluator<float>());
  std::printf("seeded from point 0: %zu points\n", cce2.getLabeledPointIndices().size());
  std::printf("n %zu\nlabels", cloud.size());
  for (size_t l : cce.getPointToClusterIndexMap()) std::printf(" %zu", l);
  std::printf("\n");
  return 0;
}
