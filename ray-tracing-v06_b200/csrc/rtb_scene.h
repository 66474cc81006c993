// rtb_scene.h — host scene graph behind the C ABI (include/rtb.h) and its flattener.
#ifndef RTB_SCENE_H
#define RTB_SCENE_H

#include <string>
#include <vector>

#include "../../include/rtb.h"
#include "../../include/rtb_scene_format.h"
#include "rtb_types.h"

struct rtb_scene {
	std::vector<rtbs_texture> textures;
	std::vector<rtbs_material> materials;
	std::vector<rtbs_object> objects;
	std::vector<int32_t> children;
	std::vector<uint8_t> blob;
	int32_t root = -1;
	int32_t background_mode = RTB_BG_SKY_GRADIENT;
	int32_t world_bvh_mode = RTB_WORLD_BVH_QUALITY;
	uint64_t uid = 0;       // unique per rtb_scene_create
	uint64_t version = 0;   // bumped by every mutating call: lets a renderer skip re-flattening an unchanged scene
	float background[3] = {0, 0, 0};
	std::vector<int32_t> sampled_lights;   // rtb_scene_set_sampled_lights: object ids (empty: no light sampling)
	// rtb_scene_set_environment: env_height x env_width x RGB texels already multiplied by env_scale, row 0 = top
	// (env_width = 0: no map, the background applies).
	std::vector<float> env_rgb;
	int32_t env_width = 0, env_height = 0, env_flags = 0;
	float env_scale[3] = {1, 1, 1};
	// rtb_add_mesh_ex: corner attributes of mesh triangles; triangle object k carries tri_attrs[objects[k].aux - 1] when its
	// aux is non-zero (empty: no attributes, the scene serialises as v1 - v3).
	std::vector<rtbs_tri_attr> tri_attrs;
	// GGX width per material (rtb_add_rough_metal / rtb_add_rough_dielectric; 0 for the other kinds).  The scene serialises
	// as v5 and the flatten hash covers the widths only when a rough material exists.
	std::vector<float> mat_alpha;
	bool has_rough() const { for (const rtbs_material& m : materials) if (m.kind == RTB_MAT_ROUGH_METAL || m.kind == RTB_MAT_ROUGH_DIELECTRIC) return true; return false; }

	// Filled by flatten(): the world BVH in the reference's node layout (parity hook).
	std::vector<rtb_bvh_node> world_nodes;
	int32_t world_root = -1;
};

namespace rtb {

void set_error(const std::string& msg);
int fail(int code, const std::string& msg);

struct Box3 { float mn[3], mx[3]; };

// BVH_Handle::Factory restated (BVH.cu:166-383). order[i] = input index at slot i.
int build_bvh(const std::vector<Box3>& boxes, int builder, std::vector<rtb_bvh_node>& nodes,
              std::vector<int>& order, int& root);
// Quality builder used for the world BVH when the scene root is not a reference BVH.
int build_bvh_world_sah(const std::vector<Box3>& boxes, std::vector<rtb_bvh_node>& nodes,
                        std::vector<int>& order, int& root);
int bvh_depth(const std::vector<rtb_bvh_node>& nodes, int root);

// Where RTB_WORLD_BVH_GPU_LBVH builds: the renderer's device and stream, and two grow-only scratch buffers the
// renderer keeps between builds (device memory; pinned host memory for the download), so that a rebuild allocates nothing.
struct GpuScratch { void* device = nullptr; size_t device_bytes = 0; void* pinned = nullptr; size_t pinned_bytes = 0; };
struct GpuBuildContext { int device; void* stream; GpuScratch* scratch; };

// GPU linear BVH (rtb_lbvh.cu): same outputs as build_bvh; inner nodes 0..n-2 (root 0), leaf of sorted position k = n-1+k.
int build_bvh_lbvh_gpu(const std::vector<Box3>& boxes, std::vector<rtb_bvh_node>& nodes, std::vector<int>& order,
                       int& root, const GpuBuildContext& gpu);
void free_gpu_scratch(GpuScratch& scratch);

// Sampling tables of an environment map (DESIGN.md §5d) from its scaled texels: one DevEnvTexel per texel, then the
// marginal CDF over rows (height + 1 floats) and one conditional CDF per row (width + 1 floats each).
void build_env_tables(const float* rgb, int width, int height, std::vector<DevEnvTexel>& texels, std::vector<float>& cdf);
// The sum of the sampling weights (the total build_env_tables divides by, summed in the same order), without the tables:
// 0 means the map cannot be sampled.
double env_weight_sum(const float* rgb, int width, int height);

// Flattens the object graph to world-space primitives + one world BVH.
int flatten(rtb_scene& s, FlatScene& out, const GpuBuildContext* gpu = nullptr);

}  // namespace rtb
#endif
