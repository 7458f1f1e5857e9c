// pt_build_dev.h — device-side flattening of a Mesh (SURVEY.md 8f-3): the same three outputs as pt_build.h's host
// builder — dead-triangle mask + DFS leaf order of the reference's BVH, an 8-wide quantised BVH over the live triangles,
// the triangle / normal records — produced by kernels on the current CUDA device (pt_build_dev.cu).
#pragma once
#include "pt_build.h"

namespace pt {

// cudaMalloc'ed arrays on `device`, laid out exactly like the host vectors of MeshBuild; owned by the caller.
struct DevMeshBuffers {
  void *nodes = nullptr, *tris = nullptr, *normals = nullptr;
  int device = -1;
};

struct DevBuildTiming {
  double upload_ms = 0, ref_ms = 0, structure_ms = 0, emit_ms = 0, download_ms = 0, total_ms = 0;
  double sah_ms = 0, plan_ms = 0;  // DevBuildMode::Sah only: binary SAH tree, collapse plan
  int ref_levels = 0, sah_levels = 0;
};

// What build_mesh_device builds after step 1.
enum class DevBuildMode {
  RefOnly,  // step 1 alone — m.dead, m.order and the reference tree's counts are filled, m.ref_done is set, and the host
            // builder (build_mesh) then skips its own restatement and builds the SAH tree from them (the hybrid the commit
            // uses by default for large meshes: the better tree, without the slowest host step)
  Median,   // the reference's median-split tree doubles as the traversal tree (PTC_COMMIT_FAST_BUILD)
  Sah,      // the host builder's tree — binned SAH + collapse plan — built on the device (PTC_COMMIT_DEVICE_SAH)
};

// Builds `m` on the CURRENT device.  Step 1 restates BVHNode::new (src/acceleration/bvh.rs:15-76) level by level: the
// tree's SHAPE depends on the triangle count only (split at n/2, leaf at <= 4), so every level is one pass of vertex
// bounds per node (-> flat nodes, split axis) and ONE stable radix sort of all triangles on (node index, centroid key).
// dead / order come out identical to the host builder's (tested).
// Median: step 2 takes that tree itself — restricted to the live triangles, three binary levels per wide node, leaves of
// <= 3 triangles — as the traversal tree: no SAH, but no second sort either; boxes are computed bottom-up and quantised by
// one kernel per wide level.
// Sah: step 2 makes the decisions of pt_build.cpp's sah_build_view and plan_collapse on the device, and moves triangles
// the way its std::partition does (the two-pointer swap of libstdc++ and libc++), so the wide tree is the host builder's:
// same wide nodes, children, slots, quantised boxes and triangles in every leaf, in the same order — also where all
// centroids of a node coincide and the host splits its current order at count / 2.  Only the numbering of the wide nodes
// below the root's children differs (breadth-first by final parent position, as in Median).
// Fills every output field of MeshBuild (host copies for ptc_scene_mesh_info / ptc_multi_create) and leaves the device
// copies in `out` (RefOnly: none).  Throws std::runtime_error on a CUDA error.
void build_mesh_device(MeshBuild &m, DevMeshBuffers &out, DevBuildTiming *timing = nullptr, DevBuildMode mode = DevBuildMode::Median);

}  // namespace pt
