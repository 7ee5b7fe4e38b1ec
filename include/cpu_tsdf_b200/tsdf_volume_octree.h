// include/cpu_tsdf_b200/tsdf_volume_octree.h — header-only C++ shim over the C ABI (b200tsdf.h)
// with the reference's class surface.
//
// Mirrors cpu_tsdf::TSDFVolumeOctree (include/cpu_tsdf/tsdf_volume_octree.h:51-377) and
// cpu_tsdf::MarchingCubesTSDFOctree (include/cpu_tsdf/marching_cubes_tsdf_octree.h:50-100): same
// method names, argument meaning and return conventions (setters take effect at the next reset();
// integrateCloud returns true; point queries return the in-bounds bool; no exceptions).
//
//   * With PCL + Eigen available define B200TSDF_WITH_PCL before including: integrateCloud takes
//     pcl::PointCloud<PointT> / Eigen::Affine3d, renderView returns pcl::PointCloud<pcl::PointNormal>::Ptr,
//     reconstruct fills a pcl::PolygonMesh — a maintainer can alias `namespace cpu_tsdf = cpu_tsdf_b200`.
//   * Without them (this container) the light-weight stand-ins below are used.
//
// Link with -lb200tsdf (cpu_tsdf_b200/libb200tsdf.so).
#pragma once
#include "../b200tsdf.h"

#include <cstddef>
#include <cstdint>
#include <cstring>
#include <memory>
#include <string>
#include <type_traits>
#include <vector>

#ifdef B200TSDF_WITH_PCL
#include <Eigen/Geometry>
#include <pcl/PolygonMesh.h>
#include <pcl/conversions.h>
#include <pcl/point_cloud.h>
#include <pcl/point_types.h>
#endif

namespace cpu_tsdf_b200
{

#ifndef B200TSDF_WITH_PCL
// stand-ins with the PCL memory layouts the C ABI is told about explicitly (stride / offsets)
struct PointXYZ { float x, y, z, pad = 1.f; };
struct PointXYZRGBA { float x, y, z, pad = 1.f; std::uint8_t b, g, r, a; float pad2[3]; };
struct PointNormal { float x, y, z, pad = 1.f; float normal_x, normal_y, normal_z, npad = 0.f; float curvature, cpad[3]; };
template <typename PointT> struct PointCloud
{
  std::uint32_t width = 0, height = 0;
  bool is_dense = true;
  std::vector<PointT> points;
  typedef std::shared_ptr<PointCloud<PointT>> Ptr;
  typedef std::shared_ptr<const PointCloud<PointT>> ConstPtr;
  const PointT& operator() (std::size_t column, std::size_t row) const { return points[row * width + column]; }
  std::size_t size () const { return points.size (); }
};
struct Affine3d
{
  double m[16] = { 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1 };   // row-major 4x4
  static Affine3d Identity () { return Affine3d (); }
  const double* data () const { return m; }
};
// Eigen::Vector3i as getOccupiedVoxelIndices uses it: idx (0), idx (1), idx (2)
struct Vector3i
{
  int v[3] = { 0, 0, 0 };
  int& operator() (int i) { return v[i]; }
  int operator() (int i) const { return v[i]; }
};
struct TriangleSoup { std::vector<float> xyz; std::vector<std::uint8_t> rgb; std::vector<std::int32_t> polygons; };
struct PointXYZRGBNormal { float x, y, z, pad = 1.f; float normal_x, normal_y, normal_z, npad = 0.f; std::uint8_t b = 0, g = 0, r = 0, a = 255; float curvature = 0.f, cpad[2] = { 0.f, 0.f }; };
#else
using pcl::PointXYZRGBNormal;
using pcl::PointCloud;
using pcl::PointNormal;
using pcl::PointXYZ;
typedef Eigen::Affine3d Affine3d;
typedef Eigen::Vector3i Vector3i;
#endif

namespace detail
{
template <typename T, typename = void> struct has_rgba : std::false_type {};
template <typename T> struct has_rgba<T, decltype ((void) std::declval<T> ().b, (void) std::declval<T> ().r, void ())> : std::true_type {};
template <typename PointT> inline int rgba_offset (std::true_type)
{ PointT p{}; return static_cast<int> (reinterpret_cast<const char*> (&p.b) - reinterpret_cast<const char*> (&p)); }
template <typename PointT> inline int rgba_offset (std::false_type) { return -1; }
template <typename PointT> inline int xyz_offset ()
{ PointT p{}; return static_cast<int> (reinterpret_cast<const char*> (&p.x) - reinterpret_cast<const char*> (&p)); }
inline void pose_rows (const Affine3d& t, double* m)
{
#ifdef B200TSDF_WITH_PCL
  for (int r = 0; r < 4; ++r) for (int c = 0; c < 4; ++c) m[r * 4 + c] = t.matrix () (r, c);
#else
  std::memcpy (m, t.m, sizeof (double) * 16);
#endif
}
}

class TSDFVolumeOctree
{
public:
  typedef std::shared_ptr<TSDFVolumeOctree> Ptr;
  typedef std::shared_ptr<const TSDFVolumeOctree> ConstPtr;

  // cpp:54-85: the same defaults; the CUDA device is chosen at construction
  explicit TSDFVolumeOctree (int device = 0, int pool_log2 = 0)
  {
    b200tsdf_default_config (&cfg_);
    cfg_.device = device;
    if (pool_log2 > 0) cfg_.pool_log2 = pool_log2;
    status_ = b200tsdf_create (&cfg_, &h_);          // B200TSDF_ENODEVICE without a GPU: there is no CPU path
  }
  ~TSDFVolumeOctree () { if (h_) b200tsdf_destroy (h_); }
  TSDFVolumeOctree (const TSDFVolumeOctree&) = delete;
  TSDFVolumeOctree& operator= (const TSDFVolumeOctree&) = delete;

  bool ok () const { return h_ != nullptr && status_ == 0; }
  int status () const { return status_; }
  const char* lastError () const { return h_ ? b200tsdf_last_error (h_) : "no CUDA device"; }
  b200tsdf_t* handle () const { return h_; }

  // ---- setters / getters (cpp:93-198, h:119-198) ----
  void setResolution (int xres, int yres, int zres) { cfg_.xres = xres; cfg_.yres = yres; cfg_.zres = zres; push (); }
  void getResolution (int& xres, int& yres, int& zres) const { xres = cfg_.xres; yres = cfg_.yres; zres = cfg_.zres; }
  void setGridSize (float xsize, float ysize, float zsize) { cfg_.xsize = xsize; cfg_.ysize = ysize; cfg_.zsize = zsize; push (); }
  void getGridSize (float& xsize, float& ysize, float& zsize) const { xsize = cfg_.xsize; ysize = cfg_.ysize; zsize = cfg_.zsize; }
  void setImageSize (int width, int height) { cfg_.image_width = width; cfg_.image_height = height; push (); }
  void getImageSize (int& width, int& height) const { width = cfg_.image_width; height = cfg_.image_height; }
  void setDepthTruncationLimits (float max_dist_pos, float max_dist_neg) { cfg_.max_dist_pos = max_dist_pos; cfg_.max_dist_neg = max_dist_neg; push (); }
  void getDepthTruncationLimits (float& max_dist_pos, float& max_dist_neg) const { max_dist_pos = cfg_.max_dist_pos; max_dist_neg = cfg_.max_dist_neg; }
  void setWeightTruncationLimit (float max_weight) { cfg_.max_weight = max_weight; push (); }
  float getWeightTruncationLimit () const { return cfg_.max_weight; }
  void setGlobalTransform (const Affine3d& trans) { detail::pose_rows (trans, cfg_.global_transform); push (); }
  Affine3d getGlobalTransform () const                                                              // h:135-137 (also what load () read back)
  {
    Affine3d t;
#ifdef B200TSDF_WITH_PCL
    for (int r = 0; r < 4; ++r) for (int c = 0; c < 4; ++c) t.matrix () (r, c) = cfg_.global_transform[r * 4 + c];
#else
    std::memcpy (t.m, cfg_.global_transform, sizeof (double) * 16);
#endif
    return t;
  }
  void setSensorDistanceBounds (float min_sensor_dist, float max_sensor_dist) { cfg_.min_sensor_dist = min_sensor_dist; cfg_.max_sensor_dist = max_sensor_dist; push (); }
  void getSensorDistanceBounds (float& min_sensor_dist, float& max_sensor_dist) const { min_sensor_dist = cfg_.min_sensor_dist; max_sensor_dist = cfg_.max_sensor_dist; }
  void setCameraIntrinsics (double fx, double fy, double cx, double cy) { cfg_.fx = fx; cfg_.fy = fy; cfg_.cx = cx; cfg_.cy = cy; push (); }
  void getCameraIntrinsics (double& fx, double& fy, double& cx, double& cy) const { fx = cfg_.fx; fy = cfg_.fy; cx = cfg_.cx; cy = cfg_.cy; }
  void setMaxVoxelSize (float x, float y, float z) { cfg_.max_cell_x = x; cfg_.max_cell_y = y; cfg_.max_cell_z = z; push (); }
  void setIntegrateColor (bool integrate_color) { cfg_.integrate_color = integrate_color; push (); }
  // h:289-293.  "RGB" and "RGBNormalized" are fused; any other mode (the reference also knows "LAB") makes the next reset () fail
  // with B200TSDF_EINVAL instead of silently fusing something else
  void setColorMode (const std::string& color_mode)
  {
    cfg_.color_mode = color_mode == "RGB" ? B200TSDF_COLOR_RGB : (color_mode == "RGBNormalized" ? B200TSDF_COLOR_RGB_NORMALIZED : B200TSDF_COLOR_LAB);
    push ();
  }
  // h:180-184 (sic).  Values other than 1 draw the extra samples with libc rand () (hpp:69-88), which cannot be reproduced: they are
  // refused — status () becomes B200TSDF_EINVAL and stays so until 1 is set again
  void setNumRandomSplts (int num_random_splits)
  { num_random_splits_ = num_random_splits; status_ = num_random_splits == 1 ? 0 : B200TSDF_EINVAL; }
  int getNumRandomSplits () const { return num_random_splits_; }
  // B200 extension: keep OctreeNode::M_ / nsample_ (octree.cpp:160-161) so that save() writes them as the reference does
  // (they are unused by every default code path; tracking them selects the general, slower update kernel)
  void setTrackVariance (bool track) { cfg_.track_variance = track ? 1 : 0; push (); }

  // ---- the volumetric path ----
  void reset ()                                                                                     // cpp:201-219
  { status_ = !h_ ? B200TSDF_ENODEVICE : (num_random_splits_ != 1 ? B200TSDF_EINVAL : b200tsdf_reset (h_)); }

  // impl/tsdf_volume_octree.hpp:48-103 (normals are unused there as well)
  template <typename PointT, typename NormalT>
  bool integrateCloud (const PointCloud<PointT>& cloud, const PointCloud<NormalT>& /*normals*/, const Affine3d& trans = Affine3d::Identity ())
  {
    if (!h_ || num_random_splits_ != 1) return false;
    double m[16];
    detail::pose_rows (trans, m);
    status_ = b200tsdf_integrate (h_, cloud.points.data (), sizeof (PointT), detail::xyz_offset<PointT> (),
                                  detail::rgba_offset<PointT> (detail::has_rgba<PointT> ()),
                                  static_cast<int> (cloud.width), static_cast<int> (cloud.height), m);
    return status_ == 0;
  }

  // The front end of the reference's `integrate` program for unorganised clouds (src/prog/integrate.cpp:548-635,
  // 673): scale / zero->NaN / world->camera / z-buffer onto the image grid / integrateCloud, all on the device.
  // `points`: n records of `stride` bytes, xyz at xyz_off, colour bytes b,g,r,a at rgba_off (or -1).
  bool integrateUnorganizedCloud (const void* points, std::size_t n, std::size_t stride, int xyz_off, int rgba_off,
                                  const Affine3d& trans = Affine3d::Identity (), float cloud_units = 1.f, bool zero_nans = false,
                                  const Affine3d* world_to_camera = nullptr)
  {
    if (!h_) return false;
    double m[16], w2c[16];
    detail::pose_rows (trans, m);
    b200tsdf_organize_opts opts;
    opts.cloud_units = cloud_units; opts.zero_nans = zero_nans ? 1 : 0; opts.world_to_camera = nullptr;
    if (world_to_camera) { detail::pose_rows (*world_to_camera, w2c); opts.world_to_camera = w2c; }
    status_ = b200tsdf_integrate_unorganized (h_, points, n, stride, xyz_off, rgba_off, &opts, m);
    return status_ == 0;
  }

  bool getFxn (const PointXYZ& pt, float& val) const                                               // cpp:655-672
  { std::uint8_t ok = 0; float p[3] = { pt.x, pt.y, pt.z }; b200tsdf_query (h_, p, 1, 1, 0, &val, nullptr, nullptr, &ok); return ok != 0; }
  bool getGradient (const PointXYZ& pt, float grad[3]) const                                       // cpp:681-700
  { std::uint8_t ok = 0; float p[3] = { pt.x, pt.y, pt.z }; b200tsdf_query (h_, p, 1, 2, 0, nullptr, grad, nullptr, &ok); return ok != 0; }
  bool getHessian (const PointXYZ& pt, float hessian[9]) const                                     // cpp:703-725
  { std::uint8_t ok = 0; float p[3] = { pt.x, pt.y, pt.z }; b200tsdf_query (h_, p, 1, 4, 0, nullptr, nullptr, hessian, &ok); return ok != 0; }
  bool getFxnAndGradient (const PointXYZ& pt, float& val, float grad[3]) const                     // cpp:728-753
  { std::uint8_t ok = 0; float p[3] = { pt.x, pt.y, pt.z }; b200tsdf_query (h_, p, 1, 3, 1, &val, grad, nullptr, &ok); return ok != 0; }
  bool getFxnGradientAndHessian (const PointXYZ& pt, float& val, float grad[3], float hessian[9]) const   // cpp:756-794
  { std::uint8_t ok = 0; float p[3] = { pt.x, pt.y, pt.z }; b200tsdf_query (h_, p, 1, 7, 1, &val, grad, hessian, &ok); return ok != 0; }

  // cpp:278-424: organized cloud in the camera frame, NaN xyz = miss
  typename PointCloud<PointNormal>::Ptr renderView (const Affine3d& trans = Affine3d::Identity (), int downsampleBy = 1) const
  {
    typename PointCloud<PointNormal>::Ptr cloud (new PointCloud<PointNormal>);
    cloud->width = cfg_.image_width / downsampleBy; cloud->height = cfg_.image_height / downsampleBy;
    cloud->is_dense = false;
    cloud->points.resize (static_cast<std::size_t> (cloud->width) * cloud->height);
    double m[16];
    detail::pose_rows (trans, m);
    PointNormal probe{};
    int noff = static_cast<int> (reinterpret_cast<const char*> (&probe.normal_x) - reinterpret_cast<const char*> (&probe));
    b200tsdf_render (h_, m, downsampleBy, cloud->points.data (), sizeof (PointNormal), detail::xyz_offset<PointNormal> (), noff, nullptr);
    return cloud;
  }

  // cpp:427-450: renderView plus the colour of the voxel under every hit (black where the ray misses)
  typename PointCloud<PointXYZRGBNormal>::Ptr renderColoredView (const Affine3d& trans = Affine3d::Identity (), int downsampleBy = 1) const
  {
    typename PointCloud<PointXYZRGBNormal>::Ptr cloud (new PointCloud<PointXYZRGBNormal>);
    cloud->width = cfg_.image_width / downsampleBy; cloud->height = cfg_.image_height / downsampleBy;
    cloud->is_dense = false;
    cloud->points.resize (static_cast<std::size_t> (cloud->width) * cloud->height);
    std::vector<std::uint8_t> rgb (cloud->points.size () * 3);
    double m[16];
    detail::pose_rows (trans, m);
    PointXYZRGBNormal probe{};
    int noff = static_cast<int> (reinterpret_cast<const char*> (&probe.normal_x) - reinterpret_cast<const char*> (&probe));
    if (b200tsdf_render (h_, m, downsampleBy, cloud->points.data (), sizeof (PointXYZRGBNormal), detail::xyz_offset<PointXYZRGBNormal> (), noff, rgb.data ()) != 0) return cloud;
    for (std::size_t i = 0; i < cloud->points.size (); ++i) { auto& p = cloud->points[i]; p.r = rgb[3 * i]; p.g = rgb[3 * i + 1]; p.b = rgb[3 * i + 2]; }
    return cloud;
  }

  // getTSDFValue / interpolateTrilinearly (cpp:454-541; protected in the reference, public here for the callers that subclassed it)
  float getTSDFValue (float x, float y, float z, bool* valid = nullptr) const
  {
    float p[3] = { x, y, z }, v = 0.f; std::uint8_t ok = valid ? (*valid ? 1 : 0) : 1;
    if (b200tsdf_interpolate (h_, p, 1, &v, &ok) != 0) ok = 0;
    if (valid) *valid = ok != 0;
    return v;
  }
  float interpolateTrilinearly (float x, float y, float z, bool* valid = nullptr) const { return getTSDFValue (x, y, z, valid); }

  void save (const std::string& filename) const { if (h_) b200tsdf_save (h_, filename.c_str ()); }   // cpp:222-245
  void load (const std::string& filename)                                                           // cpp:248-275
  { if (h_) { status_ = b200tsdf_load (h_, filename.c_str ()); b200tsdf_get_config (h_, &cfg_); } }

  PointXYZ getVoxelCenter (std::size_t x, std::size_t y, std::size_t z) const                      // cpp:553-560
  { float o[3] = { 0, 0, 0 }; b200tsdf_voxel_center (h_, (std::int64_t) x, (std::int64_t) y, (std::int64_t) z, o); PointXYZ p; p.x = o[0]; p.y = o[1]; p.z = o[2]; return p; }
  bool getVoxelIndex (float x, float y, float z, int& x_i, int& y_i, int& z_i) const               // cpp:562-574
  { std::int32_t o[3] = { 0, 0, 0 }, in = 0; b200tsdf_voxel_index (h_, x, y, z, o, &in); x_i = o[0]; y_i = o[1]; z_i = o[2]; return in != 0; }

  // cpp:576-588: the centres of Octree::getLeaves (leaves, nlevels) in the reference's order, as a cloud of width n and
  // height 1 (nlevels = 0: the root; negative: every leaf).  Empty when the call fails (status () tells why).
  typename PointCloud<PointXYZ>::ConstPtr getVoxelCenters (int nlevels = 4) const
  {
    typename PointCloud<PointXYZ>::Ptr cloud (new PointCloud<PointXYZ>);
    float* xyz = nullptr; std::size_t n = 0;
    status_ = h_ ? b200tsdf_voxel_centers (h_, nlevels, &xyz, &n) : B200TSDF_ENODEVICE;
    if (status_ != 0) n = 0;
    cloud->points.resize (n);
    cloud->width = static_cast<std::uint32_t> (n); cloud->height = 1;
    for (std::size_t i = 0; i < n; ++i) { PointXYZ& p = cloud->points[i]; p.x = xyz[3 * i]; p.y = xyz[3 * i + 1]; p.z = xyz[3 * i + 2]; }
    return cloud;
  }
  // cpp:590-609: appends getVoxelIndex of the centre of every leaf with w > 0 and |d| < 1, as the reference does
  void getOccupiedVoxelIndices (std::vector<Vector3i>& indices) const
  {
    std::int32_t* ijk = nullptr; std::size_t n = 0;
    status_ = h_ ? b200tsdf_occupied_voxel_indices (h_, &ijk, &n) : B200TSDF_ENODEVICE;
    if (status_ != 0) return;
    indices.reserve (indices.size () + n);
    for (std::size_t i = 0; i < n; ++i) { Vector3i idx; idx (0) = ijk[3 * i]; idx (1) = ijk[3 * i + 1]; idx (2) = ijk[3 * i + 2]; indices.push_back (idx); }
  }
  // h:283-287: true from reset () until the first integrateCloud; load () takes the file's flag
  bool isEmpty () const
  {
    std::int32_t e = 1;
    if (h_) b200tsdf_is_empty (h_, &e);
    return e != 0;
  }

  // TSDFInterface::instantiateFromFile (src/lib/tsdf_interface.cpp:44-51): "for now everything is an octree"
  static Ptr instantiateFromFile (const std::string& filename, int device = 0, int pool_log2 = 0)
  {
    Ptr tsdf (new TSDFVolumeOctree (device, pool_log2));
    tsdf->load (filename);
    return tsdf;
  }

private:
  void push () { if (h_) status_ = b200tsdf_set_config (h_, &cfg_); }
  int num_random_splits_ = 1;
  b200tsdf_config cfg_{};
  b200tsdf_t* h_ = nullptr;
  mutable int status_ = 0;
};

// cpu_tsdf::TSDFInterface (include/cpu_tsdf/tsdf_interface.h:64-148): the reference's abstract surface has one implementation, and so
// does this one
typedef TSDFVolumeOctree TSDFInterface;

class MarchingCubesTSDFOctree
{
public:
  MarchingCubesTSDFOctree () = default;                                                            // h:55-60, w_min_ = 2.5
  void setInputTSDF (TSDFVolumeOctree::ConstPtr tsdf_volume) { tsdf_volume_ = tsdf_volume; }       // cpp:43-83
  void setColorByConfidence (bool v) { color_by_confidence_ = v; }
  void setColorByRGB (bool v) { color_by_rgb_ = v; }
  void setMinWeight (float w_min) { w_min_ = w_min; }

#ifndef B200TSDF_WITH_PCL
  // pcl::SurfaceReconstruction::reconstruct -> performReconstruction (cpp:108-143): triangle soup,
  // polygons[i] = {3i, 3i+1, 3i+2}
  bool reconstruct (TriangleSoup& out) const
  {
    if (!tsdf_volume_ || !tsdf_volume_->handle ()) return false;
    float* v = nullptr; std::uint8_t* c = nullptr; std::size_t n = 0;
    int mode = color_by_confidence_ ? 2 : (color_by_rgb_ ? 1 : 0);
    if (b200tsdf_mesh (tsdf_volume_->handle (), w_min_, mode, &v, &c, &n) != 0) return false;
    out.xyz.assign (v, v + 3 * n);
    out.rgb.clear ();
    if (c) out.rgb.assign (c, c + 3 * n);
    out.polygons.resize (n);
    for (std::size_t i = 0; i < n; ++i) out.polygons[i] = static_cast<std::int32_t> (i);
    return true;
  }
#else
  bool reconstruct (pcl::PolygonMesh& output) const
  {
    if (!tsdf_volume_ || !tsdf_volume_->handle ()) return false;
    float* v = nullptr; std::uint8_t* c = nullptr; std::size_t n = 0;
    int mode = color_by_confidence_ ? 2 : (color_by_rgb_ ? 1 : 0);
    if (b200tsdf_mesh (tsdf_volume_->handle (), w_min_, mode, &v, &c, &n) != 0) return false;
    if (mode)
    {
      pcl::PointCloud<pcl::PointXYZRGB> cloud;
      cloud.resize (n);
      for (std::size_t i = 0; i < n; ++i) { auto& p = cloud[i]; p.x = v[3 * i]; p.y = v[3 * i + 1]; p.z = v[3 * i + 2]; if (c) { p.r = c[3 * i]; p.g = c[3 * i + 1]; p.b = c[3 * i + 2]; } }
      pcl::toPCLPointCloud2 (cloud, output.cloud);
    }
    else
    {
      pcl::PointCloud<pcl::PointXYZ> cloud;
      cloud.resize (n);
      for (std::size_t i = 0; i < n; ++i) { auto& p = cloud[i]; p.x = v[3 * i]; p.y = v[3 * i + 1]; p.z = v[3 * i + 2]; }
      pcl::toPCLPointCloud2 (cloud, output.cloud);
    }
    output.polygons.resize (n / 3);
    for (std::size_t i = 0; i < n / 3; ++i) { output.polygons[i].vertices = { (std::uint32_t) (3 * i), (std::uint32_t) (3 * i + 1), (std::uint32_t) (3 * i + 2) }; }
    return true;
  }
#endif

private:
  TSDFVolumeOctree::ConstPtr tsdf_volume_;
  bool color_by_confidence_ = false, color_by_rgb_ = false;
  float w_min_ = 2.5f;
};

#ifndef B200TSDF_WITH_PCL
// The mesh post-processing of the reference's `integrate` program, on the GPU.  Like the reference's versions they
// rebuild the mesh cloud as plain XYZ: vertex colours do not survive (src/prog/integrate.cpp:106, 149, 186, 213).
namespace detail
{
  template <typename Fn> inline bool meshpost (TriangleSoup& mesh, Fn&& call)
  {
    float* v = nullptr; std::int32_t* t = nullptr; std::size_t nv = 0, nt = 0;
    if (call (mesh.xyz.data (), mesh.xyz.size () / 3, mesh.polygons.data (), mesh.polygons.size () / 3, &v, &nv, &t, &nt) != 0) return false;
    mesh.xyz.assign (v, v + 3 * nv); mesh.polygons.assign (t, t + 3 * nt); mesh.rgb.clear ();
    b200tsdf_mesh_free (v); b200tsdf_mesh_free (t);
    return true;
  }
}
// flattenVertices (src/prog/integrate.cpp:103-150)
inline bool flattenVertices (TriangleSoup& mesh, float min_dist = 0.0001f, int device = 0)
{
  return detail::meshpost (mesh, [&] (const float* v, std::size_t nv, const std::int32_t* t, std::size_t nt, float** ov, std::size_t* onv, std::int32_t** ot, std::size_t* ont)
                           { return b200tsdf_mesh_flatten (device, v, nv, t, nt, min_dist, ov, onv, ot, ont); });
}
// cleanupMesh (src/prog/integrate.cpp:152-214)
inline bool cleanupMesh (TriangleSoup& mesh, float face_dist = 0.02f, int min_neighbors = 5, int device = 0)
{
  return detail::meshpost (mesh, [&] (const float* v, std::size_t nv, const std::int32_t* t, std::size_t nt, float** ov, std::size_t* onv, std::int32_t** ot, std::size_t* ont)
                           { return b200tsdf_mesh_cleanup (device, v, nv, t, nt, face_dist, min_neighbors, ov, onv, ot, ont); });
}
#endif

} // namespace cpu_tsdf_b200
