// rtb_types.h — flattened, aligned device records produced by the host flattener
// (rtb_scene.cpp) and consumed by the wavefront kernels (rtb_kernels.cu).
#ifndef RTB_TYPES_H
#define RTB_TYPES_H

#include <stdint.h>
#include <vector>

namespace rtb {

// Primitive types (4 bits of a leaf reference): a base type, plus PRIM_XF when the primitive is an
// instance (translate / rotate_y chain): its record then holds OBJECT-space geometry followed by
// the world-from-object transform, and the kernels transform the ray exactly like the book's
// translate::hit / rotate_y::hit do (so instanced hits are bit-exact against the oracle too).
enum PrimType : int {
	PRIM_SPHERE = 0, PRIM_MOVING_SPHERE = 1, PRIM_QUAD = 2, PRIM_TRIANGLE = 3,
	PRIM_MEDIUM_SPHERE = 4, PRIM_MEDIUM_BOX = 5,
	PRIM_BOX = 6,   // one BVH leaf for a book box(): (min, max) record followed by its six quad records (hits are reported on those)
	PRIM_XF = 8
};
#define RTB_LEAF_TYPE_BITS 4
// Deepest world BVH the kernels walk: 30 levels on the 32-entry stack (16 entries when <= 17), up to 62 on the
// 64-entry stack that only the GPU linear BVH of a large scene needs.
// Wide-node float layout.  0: (Lmin.xyz, Lext.xyz, Rmin.xyz, Rext.xyz).  1: paired for the packed two-wide FMA of
// sm_100 (FFMA2): (Lmin.xy, Lext.xy | Rmin.xy, Rext.xy | Lmin.z, Rmin.z, Lext.z, Rext.z), so that every operand pair of
// the slab test is an aligned register pair of one 16-byte load.
#ifndef RTB_NODE_PAIRED
#define RTB_NODE_PAIRED 1
#endif
#define RTB_TREE_DEPTH_NORMAL 30
#define RTB_TREE_DEPTH_MAX 62

// Child reference of a wide-layout BVH node: >= 0 inner node index; < 0 leaf,
// ~ref = (prim_index << 4) | PrimType.
inline int make_leaf_ref(int prim, int type) { return ~((prim << RTB_LEAF_TYPE_BITS) | type); }

// 64-byte inner node holding BOTH children's boxes as (min, extent), fetched as 4 x LDG.128:
//   a = (l.min.x, l.min.y, l.min.z, l.ext.x)   b = (l.ext.y, l.ext.z, r.min.x, r.min.y)
//   c = (r.min.z, r.ext.x, r.ext.y, r.ext.z)   d = (left ref, right ref, 0, 0) as int bits
// extents are rounded up so min + ext >= max: the box the kernel tests contains the exact one.
struct alignas(64) DevNode { float f[12]; int32_t left, right, pad0, pad1; };

// 64-byte primitive record (4 x float4):
//   SPHERE         q0 = (c.xyz, r)
//   MOVING_SPHERE  q0 = (c0.xyz, r)       q1 = (c1.xyz, 0)
//   QUAD/TRIANGLE  q0 = (Q.xyz, D)        q1 = (u.xyz, N.x)  q2 = (v.xyz, N.y)  q3 = (w.xyz, N.z)
//   MEDIUM_SPHERE  q0 = (c.xyz, r)        q1 = (-1/density, medium index bits, 0, 0)
//   MEDIUM_BOX     q0 = (bmin.xyz, cos)   q1 = (bmax.xyz, sin)  q2 = (offset.xyz, -1/density)
//                  q3 = (medium index bits, 0, 0, 0)       world = R_y * object + offset
// PRIM_XF variants append the transform T = (cos, sin, off.x, off.y), (off.z, 0, 0, 0):
//   XF SPHERE at q1,q2; XF MOVING_SPHERE at q2,q3; XF QUAD/TRIANGLE in a second record slot (q4,q5).
struct alignas(64) DevPrim { float q[16]; };

struct alignas(8) DevPrimInfo { int32_t material; int32_t object; };

// Light table of a scene with sampled lights (DESIGN.md §5b): one world-space DevPrim per light (SPHERE or QUAD record
// layout), then one DevLightInfo per light.
struct alignas(16) DevLightInfo { int32_t type; float area; float pad0, pad1; };   // PRIM_SPHERE / PRIM_QUAD; quad area

// Environment map (DESIGN.md §5d): per texel its scaled radiance and the numerator of its pdf per solid angle,
// p_ij * W * H / (2 pi^2) (the pdf of a direction is this over sin theta).
struct alignas(16) DevEnvTexel { float r, g, b, pdf; };

// Corner attributes of a mesh triangle (DESIGN.md §5e), in the triangle's own frame, as four float4:
//   (n0.xyz, uv0.x)  (n1.xyz, uv0.y)  (n2.xyz, uv1.x)  (uv1.y, uv2.x, uv2.y, flags bits = RTBS_ATTR_NORMALS | RTBS_ATTR_UVS)
struct alignas(64) DevTriAttr { float q[16]; };

struct alignas(16) DevMaterial { int32_t kind, tex; float param, pad; float albedo[4]; };  // 32 B

struct alignas(16) DevTexture {                                                             // 48 B
	int32_t kind, even, odd; float scale;      // checker: scale holds inv_scale
	float rgb[4];
	int32_t width, height; uint32_t blob_offset; uint32_t pad;
};

// Everything the kernels need about a scene, host-side staging.
struct FlatScene {
	std::vector<DevNode> nodes;          // wide layout actually traversed
	int32_t root_ref = 0;                // inner index or leaf ref
	int32_t bvh_empty = 0;               // every primitive is in pre_list
	std::vector<int32_t> pre_list;       // leaf codes of the media tested before the BVH walk
	std::vector<DevPrim> prims;
	std::vector<DevPrimInfo> prim_info;
	std::vector<int32_t> prim_type;
	std::vector<DevMaterial> materials;
	std::vector<DevTexture> textures;
	std::vector<uint8_t> blob;
	std::vector<DevPrim> lights;         // sampled lights in world space (empty: no light sampling)
	std::vector<DevLightInfo> light_info;
	std::vector<DevEnvTexel> env;        // environment map texels, row 0 = top (empty: no map)
	std::vector<float> env_cdf;          // its marginal CDF (env_height + 1), then env_height conditional CDFs (env_width + 1 each)
	int32_t env_width = 0, env_height = 0, env_sample = 0;
	std::vector<DevTriAttr> tri_attr;    // triangle attribute records (empty: no attributes)
	std::vector<int32_t> attr_slot;      // per record slot: its tri_attr index, or -1 (empty when tri_attr is)
	int32_t n_media = 0;
	int32_t background_mode = 0;
	float background[3] = {0, 0, 0};
	int32_t max_depth_nodes = 0;         // tree depth (stack bound check)
	int32_t builder = 0;                 // rtb_world_bvh_mode that produced the tree (3 = median fallback)
	int32_t n_items = 0;                 // BVH leaves
	float world_min[3] = {0, 0, 0}, world_max[3] = {0, 0, 0};   // bounds of the world BVH
	float bin_min[3] = {0, 0, 0}, bin_max[3] = {0, 0, 0};       // bounds of the primitives' box centres: the ray-binning grid
	float flatten_ms = 0.0f, bvh_build_ms = 0.0f;
};

}  // namespace rtb
#endif
