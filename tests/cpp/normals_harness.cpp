// TEST PROGRAM: pcl::NormalEstimation as an application configures it, against PCL's include paths (include/ope_pcl_compat).
//   normals_harness <xyz.f32> <k> <radius> <out.f32>
// sets setKSearch(k) and setRadiusSearch(radius) as given (0 leaves that one unset), computes, and writes nx, ny, nz, curvature of
// every output point to out.f32. Prints the output size and whether every output point still equals a default-constructed one.
#include <pcl/features/normal_3d.h>
#include <pcl/point_types.h>
#include <pcl/search/kdtree.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>

int main(int argc, char** argv) {
  if (argc != 5) { std::fprintf(stderr, "usage: normals_harness xyz.f32 k radius out.f32\n"); return 2; }
  pcl::PointCloud<pcl::PointXYZ>::Ptr cloud(new pcl::PointCloud<pcl::PointXYZ>);
  std::ifstream f(argv[1], std::ios::binary);
  float v[3];
  while (f.read(reinterpret_cast<char*>(v), sizeof(v))) {
    pcl::PointXYZ p;
    p.x = v[0]; p.y = v[1]; p.z = v[2];
    cloud->push_back(p);
  }
  const int k = std::atoi(argv[2]);
  const double radius = std::atof(argv[3]);
  pcl::NormalEstimation<pcl::PointXYZ, pcl::Normal> ne;
  ne.setSearchMethod(pcl::search::KdTree<pcl::PointXYZ>::Ptr(new pcl::search::KdTree<pcl::PointXYZ>));
  if (k) ne.setKSearch(k);
  if (radius != 0) ne.setRadiusSearch(radius);
  ne.setViewPoint(0, 0, 0);
  ne.setInputCloud(cloud);
  pcl::PointCloud<pcl::Normal> out;
  ne.compute(out);
  const pcl::Normal fresh;
  bool untouched = true;
  std::ofstream o(argv[4], std::ios::binary);
  for (const auto& p : out.points) {
    const float w[4] = {p.normal_x, p.normal_y, p.normal_z, p.curvature};
    untouched = untouched && std::memcmp(w, &fresh.normal_x, 3 * sizeof(float)) == 0 && std::memcmp(&w[3], &fresh.curvature, sizeof(float)) == 0;
    o.write(reinterpret_cast<const char*>(w), sizeof(w));
  }
  std::printf("%zu %d\n", out.points.size(), untouched ? 1 : 0);
  return 0;
}
