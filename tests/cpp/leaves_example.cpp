// tests/cpp/leaves_example.cpp — getVoxelCenters / getOccupiedVoxelIndices / isEmpty through the C++ shim, written as a
// reference user would (tsdf_volume_octree.h:278-296).  Built (and, on a GPU box, run) by tests/test_leaves_cpp.py.
#include "../../include/cpu_tsdf_b200/tsdf_volume_octree.h"
#include <cstdio>
using namespace cpu_tsdf_b200;

int main ()
{
  TSDFVolumeOctree::Ptr tsdf (new TSDFVolumeOctree (0, 16));
  if (!tsdf->ok ()) { std::printf ("no device: %d (%s)\n", tsdf->status (), tsdf->lastError ()); return tsdf->status () == B200TSDF_ENODEVICE ? 3 : 1; }
  tsdf->setGridSize (10.f, 10.f, 10.f);
  tsdf->setResolution (2048, 2048, 2048);
  tsdf->setCameraIntrinsics (525., 525., 319.5, 239.5);
  tsdf->reset ();
  if (tsdf->status () != 0) { std::printf ("reset: %s\n", tsdf->lastError ()); return 1; }
  if (!tsdf->isEmpty ()) { std::printf ("isEmpty after reset\n"); return 1; }
  std::vector<Vector3i> indices (2);                  // getOccupiedVoxelIndices appends: these two stay in front
  indices[0] (0) = -7; indices[1] (2) = 11;
  tsdf->getOccupiedVoxelIndices (indices);
  if (tsdf->status () != 0 || indices.size () != 2) { std::printf ("fresh volume: %zu indices (%s)\n", indices.size (), tsdf->lastError ()); return 1; }
  // a fronto-parallel wall 1 m in front of the camera
  PointCloud<PointXYZ> cloud; cloud.width = 640; cloud.height = 480; cloud.points.resize (640 * 480);
  for (int v = 0; v < 480; ++v) for (int u = 0; u < 640; ++u)
  {
    PointXYZ& p = cloud.points[v * 640 + u];
    p.z = 1.0f; p.x = (u - 319.5f) / 525.f; p.y = (v - 239.5f) / 525.f;
  }
  Affine3d pose; pose.m[11] = -1.0;
  for (int i = 0; i < 2; ++i) if (!tsdf->integrateCloud (cloud, PointCloud<PointXYZ> (), pose)) { std::printf ("integrate: %s\n", tsdf->lastError ()); return 1; }
  if (tsdf->isEmpty ()) { std::printf ("isEmpty after integrateCloud\n"); return 1; }
  PointCloud<PointXYZ>::ConstPtr centres = tsdf->getVoxelCenters ();
  std::printf ("getVoxelCenters (): %zu points, width %u height %u\n", centres->size (), centres->width, centres->height);
  if (centres->size () != 4096 || centres->width != 4096 || centres->height != 1) return 1;   // 8^4 level-4 cells at 2048^3 / 10 m
  // the first level-4 cell in the depth-first order is the corner (-x, -y, -z): centre -5 + 10/32
  if (centres->points[0].x != -4.6875f || centres->points[0].y != -4.6875f || centres->points[0].z != -4.6875f) return 1;
  tsdf->getOccupiedVoxelIndices (indices);
  std::printf ("getOccupiedVoxelIndices: %zu indices after the two placeholders\n", indices.size () - 2);
  if (tsdf->status () != 0 || indices.size () < 1000 || indices[0] (0) != -7 || indices[1] (2) != 11) return 1;
  // the wall sits at z = 0, i.e. around finest index 1024
  std::size_t near = 0;
  for (std::size_t i = 2; i < indices.size (); ++i) near += indices[i] (2) >= 1000 && indices[i] (2) <= 1048;
  if (near * 10 < (indices.size () - 2) * 9) { std::printf ("only %zu indices near the wall\n", near); return 1; }
  std::printf ("leaves ok\n");
  return 0;
}
