// oracle/ref_leaves.cpp — the oracle C API of ref_capi.cpp plus the reference's own getVoxelCenters, getOccupiedVoxelIndices
// and isEmpty (tsdf_volume_octree.cpp:576-609, tsdf_volume_octree.h:283-287).  Linked with the reference's src/lib/*.cpp
// compiled verbatim against oracle/compat/ into oracle/_ref/libcpu_tsdf_ref_leaves.so (oracle/leaves.mk).  TEST
// INFRASTRUCTURE: pins the leaf enumeration (tests/test_leaves_ref_pin.py) and is the reference arm of tools/bench_leaves.py.
#include "ref_capi.cpp"

extern "C" {

// getVoxelCenters (nlevels): 3 floats per point, written when xyz is not NULL; returns the point count
int64_t orc_voxel_centers (const orc_volume* v, int nlevels, float* xyz)
{
  pcl::PointCloud<pcl::PointXYZ>::ConstPtr c = v->tsdf->getVoxelCenters (nlevels);
  for (size_t i = 0; xyz && i < c->size (); ++i) { xyz[3 * i] = c->points[i].x; xyz[3 * i + 1] = c->points[i].y; xyz[3 * i + 2] = c->points[i].z; }
  return static_cast<int64_t> (c->size ());
}

// getOccupiedVoxelIndices: 3 int32 per index, written when ijk is not NULL; returns the index count
int64_t orc_occupied_indices (const orc_volume* v, int32_t* ijk)
{
  std::vector<Eigen::Vector3i> idx;
  v->tsdf->getOccupiedVoxelIndices (idx);
  for (size_t i = 0; ijk && i < idx.size (); ++i) for (int k = 0; k < 3; ++k) ijk[3 * i + k] = idx[i] (k);
  return static_cast<int64_t> (idx.size ());
}

int orc_is_empty (const orc_volume* v) { return v->tsdf->isEmpty () ? 1 : 0; }

} // extern "C"
