/*
 * rtb.h — C ABI of the B200-native wavefront path tracer ("rtb" = ray-tracing B200).
 *
 * This is the drop-in boundary for the per-pixel path-tracing hot path of
 * SuperCat908809/Ray-Tracing-v06.  The reference has no FFI: its "API" is the C++
 * object model below, whose device objects are opaque to the host.  Each entry
 * point here cites the reference interface it replaces (paths relative to the
 * reference checkout):
 *
 *   scene assembly   newOnDevice<T>(args...)                main/src/utilities/cuda_utilities/cuda_utils.cuh:16-23
 *                    SphereHandle::MakeSphere/MakeMovingSphere  main/src/rt_engine/geometry/SphereHittable.cuh:134-154
 *                    HittableList(objects, n, bounds)        main/src/rt_engine/geometry/HittableList.cuh:19
 *                    BVH_Handle::Factory / BuildBVH_*        main/src/rt_engine/geometry/BVH.cuh:69-102, BVH.cu:166-210,315-383
 *                    Lambertian/Metal/Dielectric/LambertianTexture  main/src/rt_engine/shaders/cu_materials.cuh:17-144
 *                    solid_texture / checker_texture          main/src/rt_engine/shaders/cu_Textures.cuh:9-40
 *                    Pinhole/DefocusBlur/MotionBlurCamera     main/src/rt_engine/shaders/cu_Cameras.cuh:12-90
 *   rendering        Renderer::MakeRenderer/Render/DownloadRenderbuffer   main/src/Renderer.h:38-46, Renderer.cu:31-137
 *   parity hooks     _sphere_closest_intersection             main/src/rt_engine/geometry/SphereHittable.cuh:15-33
 *                    (google_testing/test.cpp:87-135 recipe)  -> rtb_trace_rays
 *                    BVH_Handle::Factory::_build_bvh_rec1     main/src/rt_engine/geometry/BVH.cu:180-210 -> rtb_bvh_build
 *
 * Conventions: plain pointers and sizes only; every function returns an int status
 * (RTB_OK == 0, negative on error) unless documented otherwise; rtb_last_error()
 * returns a thread-local message for the last failing call; no exceptions cross the
 * ABI.  Host buffers are caller-owned.  One rtb_renderer per CUDA device; objects are
 * thread-compatible, not thread-safe.  All `stream` arguments are a cudaStream_t
 * passed as void* (NULL = the legacy default stream).
 *
 * There is NO CPU fallback: every function that renders or traces fails with
 * RTB_ERR_CUDA when no CUDA device is usable.
 */
#ifndef RTB_H
#define RTB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTB_ABI_VERSION 1

enum rtb_status {
	RTB_OK = 0,
	RTB_ERR_INVALID = -1,     /* bad argument / id */
	RTB_ERR_CUDA = -2,        /* CUDA runtime error or no device */
	RTB_ERR_NOMEM = -3,
	RTB_ERR_STATE = -4,       /* call out of order (e.g. render before set_scene) */
	RTB_ERR_UNSUPPORTED = -5  /* scene construct the flattener cannot express */
};

/* ------------------------------------------------------------------ scene graph */

typedef struct rtb_scene rtb_scene;

enum rtb_texture_kind { RTB_TEX_SOLID = 0, RTB_TEX_CHECKER = 1, RTB_TEX_IMAGE = 2, RTB_TEX_NOISE = 3 };
enum rtb_material_kind {
	RTB_MAT_LAMBERTIAN = 0, RTB_MAT_METAL = 1, RTB_MAT_DIELECTRIC = 2,
	RTB_MAT_DIFFUSE_LIGHT = 3, RTB_MAT_ISOTROPIC = 4,
	RTB_MAT_ROUGH_METAL = 5, RTB_MAT_ROUGH_DIELECTRIC = 6
};
enum rtb_object_kind {
	RTB_OBJ_SPHERE = 0, RTB_OBJ_MOVING_SPHERE = 1, RTB_OBJ_QUAD = 2, RTB_OBJ_TRIANGLE = 3,
	RTB_OBJ_BOX = 4, RTB_OBJ_LIST = 5, RTB_OBJ_BVH = 6, RTB_OBJ_TRANSLATE = 7,
	RTB_OBJ_ROTATE_Y = 8, RTB_OBJ_CONSTANT_MEDIUM = 9
};
/* BVH builders of BVH_Handle::Factory (BVH.cu:166-178 / :212-304 / :315-383). */
enum rtb_bvh_builder { RTB_BVH_TOPDOWN_MEDIAN = 0, RTB_BVH_TOPDOWN_SAH = 1, RTB_BVH_BOTTOMUP = 2 };
/* Miss shader: the reference's hard-coded sky gradient (Renderer.cu:149-154) or a constant colour. */
enum rtb_background_mode { RTB_BG_SKY_GRADIENT = 0, RTB_BG_CONSTANT = 1 };

int  rtb_abi_version(void);
const char* rtb_last_error(void);

int  rtb_scene_create(rtb_scene** out);
void rtb_scene_destroy(rtb_scene* s);

/* Textures: return a texture id >= 0, or a negative rtb_status. */
int rtb_add_solid_texture(rtb_scene* s, const float rgb[3]);
int rtb_add_checker_texture(rtb_scene* s, float scale, int even_tex, int odd_tex);
/* 8-bit image, `channels` in {1,3,4}, row 0 = top row; stored as RGB. */
int rtb_add_image_texture(rtb_scene* s, const uint8_t* pixels, int width, int height, int channels);
/* Perlin marble; gradient/permutation tables are derived from `seed` with Philox4x32-10. */
int rtb_add_noise_texture(rtb_scene* s, float scale, uint32_t seed);

/* Materials: return a material id >= 0, or a negative rtb_status. */
int rtb_add_lambertian(rtb_scene* s, int tex);
int rtb_add_lambertian_color(rtb_scene* s, const float albedo[3]);
int rtb_add_metal(rtb_scene* s, const float albedo[3], float fuzz);
int rtb_add_dielectric(rtb_scene* s, const float albedo[3], float ior);
int rtb_add_diffuse_light(rtb_scene* s, int tex);
int rtb_add_isotropic(rtb_scene* s, int tex);
/* GGX (Trowbridge-Reitz) microfacet materials with isotropic width `alpha` in [RTB_ROUGH_ALPHA_MIN, 1] (DESIGN.md §5f).
 * Directions are drawn from the distribution of visible normals; the throughput weight of a sampled direction is
 * G2 / G1 (height-correlated Smith) times Schlick's Fresnel term (metal, F0 per channel) or the albedo (dielectric).
 * Single scattering only: the energy that multiple scattering between microfacets would return is lost, more of it
 * the larger alpha.  Neither kind is part of the light mixture of rtb_scene_set_sampled_lights.  As alpha -> 0 the
 * metal tends to rtb_add_metal(f0, 0) and the dielectric to rtb_add_dielectric (no 1/ior^2 radiance factor either).
 * RTB_ERR_INVALID (scene unchanged): a null pointer, a non-finite value, alpha outside the range, ior not > 0. */
#define RTB_ROUGH_ALPHA_MIN 0.001f
int rtb_add_rough_metal(rtb_scene* s, const float f0[3], float alpha);
int rtb_add_rough_dielectric(rtb_scene* s, const float albedo[3], float ior, float alpha);

/* Hittables: return an object id >= 0, or a negative rtb_status. */
int rtb_add_sphere(rtb_scene* s, const float center[3], float radius, int mat);
int rtb_add_moving_sphere(rtb_scene* s, const float center0[3], const float center1[3], float radius, int mat);
int rtb_add_quad(rtb_scene* s, const float Q[3], const float u[3], const float v[3], int mat);
int rtb_add_triangle(rtb_scene* s, const float Q[3], const float u[3], const float v[3], int mat);
int rtb_add_box(rtb_scene* s, const float a[3], const float b[3], int mat);
int rtb_add_list(rtb_scene* s, const int* children, int n);
int rtb_add_bvh(rtb_scene* s, const int* children, int n, int builder);
/* A triangle mesh in one call: `vertices` = n_vertices x (x, y, z), `indices` = n_triangles x 3 vertex indices.  Adds one
 * triangle (Q = v0, u = v1 - v0, v = v2 - v0) per face that has an area and returns a BVH group over them - the same
 * objects rtb_add_triangle + rtb_add_bvh would make (the reference has no mesh type; its GL demo loads OBJ files through
 * tiny_obj, main/src/gl_engine/gl_mesh.cpp:124-218). */
int rtb_add_mesh(rtb_scene* s, const float* vertices, int n_vertices, const int* indices, int n_triangles, int mat);
/* rtb_add_mesh with per-vertex attributes (DESIGN.md §5e): `normals` = n_vertices x (x, y, z) shading normals, `uvs` =
 * n_vertices x (u, v) texture coordinates, either or both NULL.  Makes the same triangles under the same BVH group as
 * rtb_add_mesh (the same faces are dropped); each triangle also carries its three corners' attributes.  With normals, a hit
 * is shaded with the normal interpolated from its corners (normalised, put on the face normal's side, facing the ray);
 * front_face and the dielectric's inside / outside test stay with the face normal.  With UVs, textures read the
 * interpolated (u, v) instead of the triangle's own (alpha, beta).  Normals are normalised on the host in double; zero
 * normals are kept (the face normal is used where all three corners interpolate to zero).  No correction for shading-normal
 * artefacts is applied.  With both NULL this is rtb_add_mesh exactly.  RTB_ERR_INVALID (scene unchanged): everything
 * rtb_add_mesh refuses, and a non-finite normal or UV component. */
int rtb_add_mesh_ex(rtb_scene* s, const float* vertices, int n_vertices, const int* indices, int n_triangles,
                    const float* normals, const float* uvs, int mat);
int rtb_add_translate(rtb_scene* s, int child, const float offset[3]);
int rtb_add_rotate_y(rtb_scene* s, int child, float degrees);
int rtb_add_constant_medium(rtb_scene* s, int boundary, float density, int phase_mat);

int rtb_scene_set_root(rtb_scene* s, int object);
int rtb_scene_set_background(rtb_scene* s, int mode, const float rgb[3]);
/* Which tree the renderer walks.  Closest hits do not depend on it (tests/test_gpu_parity.py checks that).
 * RTB_WORLD_BVH_QUALITY (default): a binned-SAH tree over all flattened primitives.
 * RTB_WORLD_BVH_AS_BUILT: when the scene root is a BVH, exactly the tree its BVH_Handle::Factory builder makes
 * (same nodes, same primitive order as the reference), e.g. to inspect it with rtb_scene_world_bvh.
 * RTB_WORLD_BVH_GPU_LBVH: a linear BVH (Morton codes, radix sort, one-pass hierarchy, bottom-up fit) built on the
 * renderer's device inside rtb_renderer_set_scene: a lower-quality tree in a fraction of the build time, for large
 * meshes and scenes that are rebuilt often.  Needs a renderer: rtb_scene_flatten_stats refuses it.  Trees up to 62
 * levels deep are walked (on a 64-entry stack past 30 levels); a deeper one is replaced by the RTB_WORLD_BVH_QUALITY
 * tree (rtb_scene_stats.builder says which builder produced the tree in use). */
enum rtb_world_bvh_mode { RTB_WORLD_BVH_QUALITY = 0, RTB_WORLD_BVH_AS_BUILT = 1, RTB_WORLD_BVH_GPU_LBVH = 2 };
int rtb_scene_set_world_bvh(rtb_scene* s, int mode);

/* Light importance sampling ("Ray Tracing: The Rest of Your Life", mixture pdfs), opt-in per scene.  `objects` names
 * n <= RTB_MAX_SAMPLED_LIGHTS emitters, each a sphere, a quad, or a translate / rotate_y chain ending in one; it is
 * sampled where the chain puts it (the chain from the listed object down, composed as the flattener composes instances).
 * At every Lambertian or isotropic scatter, half of the directions then aim at a point drawn on one of the listed
 * objects (chosen uniformly; quads: uniform in area; spheres: uniform in the cone they subtend) and half are the
 * material's own (cosine-weighted / uniform) directions; the throughput is weighted by scattering pdf / mixture pdf
 * (DESIGN.md §5b).  The expected image does not depend on the list - any list, even one naming objects that do not
 * emit, gives the same converged image - only the noise does.  n = 0 clears the list; a scene without one renders,
 * serialises and hashes exactly as if this had never been called.  Moving spheres, triangles, boxes, lists, BVHs and
 * media return RTB_ERR_UNSUPPORTED; bad ids, n outside [0, 16], a quad without area return RTB_ERR_INVALID (the list
 * is then left unchanged). */
#define RTB_MAX_SAMPLED_LIGHTS 16
int rtb_scene_set_sampled_lights(rtb_scene* s, const int* objects, int n);

/* HDR environment map (DESIGN.md §5d): an equirectangular map of width x height linear RGB float texels, row 0 at the
 * top (+y), each channel multiplied by scale[c] when it is set.  While a map is set, every ray that leaves the scene
 * returns throughput * the nearest texel in its direction instead of the background (which the scene keeps: clearing the
 * map restores it).  RTB_ENV_SAMPLE adds the map, importance-sampled by luminance x sin(theta), as one more strategy of
 * the light-sampling mixture at Lambertian and isotropic scatters (with or without a light list); it changes only the
 * noise, not the expected image.  rgb = NULL with width = height = 0 clears the map.  RTB_ERR_INVALID (scene unchanged):
 * width or height outside [1, 16384], width x height > 2^24, a texel or scale that is negative, NaN or infinite, unknown
 * flags, or RTB_ENV_SAMPLE on a map whose sampling weights are all zero.  A scene without a map renders, serialises and
 * hashes exactly as if this had never been called. */
#define RTB_ENV_SAMPLE 1
#define RTB_ENV_MAX_SIZE 16384
int rtb_scene_set_environment(rtb_scene* s, const float* rgb, int width, int height, const float scale[3], int flags);

int rtb_scene_num_objects(const rtb_scene* s);
/* Children of a list / BVH / mesh group (1 for translate, rotate_y, constant_medium; 0 for primitives). */
int rtb_scene_num_children(const rtb_scene* s, int object);
/* World-space bounds of an object: out6 = {min.xyz, max.xyz} (getSphereBounds & co). */
int rtb_object_bounds(const rtb_scene* s, int object, float out6[6]);

/* Flat binary description of the scene graph (format: include/rtb_scene_format.h).
 * Returns the number of bytes needed; writes only if cap is large enough. */
size_t rtb_scene_serialize(const rtb_scene* s, void* buf, size_t cap);

/* ------------------------------------------------------------------ BVH parity hook (host only) */

/* Same 32-byte layout as BVH::Node (BVH.cuh:16-25). */
typedef struct rtb_bvh_node {
	float bmin[3], bmax[3];
	int32_t left_child_idx;            /* -1 => leaf */
	int32_t right_child_hittable_idx;  /* leaf: index into the (reordered) primitive array */
} rtb_bvh_node;

/* Builds the BVH exactly as BVH_Handle::Factory does over n boxes (aabbs = n x {min.xyz,max.xyz}).
 * nodes_out must hold 2n-1 nodes; order_out[i] = input index of the primitive that ends up at
 * slot i of the reordered array (Factory::hittables, BVH.cu:174-177).  Returns the number of
 * nodes written (root index via root_out) or a negative status. */
int rtb_bvh_build(const float* aabbs, int n, int builder, rtb_bvh_node* nodes_out, int* order_out, int* root_out);

/* The world BVH the renderer traverses after rtb_renderer_set_scene, in the same node layout
 * (leaf payload = flattened primitive index).  Pass NULL to query the node count. */
int rtb_scene_world_bvh(const rtb_scene* s, rtb_bvh_node* nodes_out, int cap, int* root_out);

/* Host-only: runs the flattener (instances -> record slots, world BVH) without touching the GPU and
 * reports its sizes; also fills the world BVH returned by rtb_scene_world_bvh.  out4 = {primitives
 * (BVH leaves), 64-byte record slots, inner nodes of the wide layout, tree depth}. */
int rtb_scene_flatten_stats(rtb_scene* s, int32_t out4[4]);
/* Host-only: FNV-1a hash of what the flattener would upload for traversal and shading (wide nodes, primitive records,
 * per-slot material / object ids, pre-test list).  Two scenes, builds or settings that hash equal render identically. */
int rtb_scene_flatten_hash(rtb_scene* s, uint64_t* hash_out);

/* What rtb_renderer_set_scene last built (declared below with the renderer): sizes as in rtb_scene_flatten_stats,
 * the builder that produced the tree the kernels walk (an rtb_world_bvh_mode value, or RTB_BUILDER_MEDIAN_FALLBACK
 * when both the requested tree and the SAH tree were deeper than the traversal stack), and host wall-clock times. */
enum { RTB_BUILDER_MEDIAN_FALLBACK = 3 };
typedef struct rtb_scene_stats {
	int32_t primitives, record_slots, inner_nodes, depth;
	int32_t builder;
	float flatten_ms;     /* whole flatten: graph walk, BVH build, wide-layout conversion */
	float bvh_build_ms;   /* the BVH build alone (GPU LBVH: upload of boxes, kernels, download of nodes) */
	int32_t reserved;
} rtb_scene_stats;

/* ------------------------------------------------------------------ cameras */

enum rtb_camera_kind { RTB_CAM_PINHOLE = 0, RTB_CAM_DEFOCUS = 1, RTB_CAM_MOTION = 2 };

typedef struct rtb_camera {
	int32_t kind;
	float o[3], u[3], v[3], w[3];
	float viewport_width, viewport_height; /* defocus: unscaled u,v + these (cu_Cameras.cuh:54-64) */
	float lens_radius, focus_dist;
	float t0, t1;                          /* shutter interval; time = mix(t0,t1,rnd) */
} rtb_camera;

int rtb_camera_pinhole(rtb_camera* c, const float lookfrom[3], const float lookat[3], const float up[3],
                       float vfov_deg, float aspect);
int rtb_camera_defocus(rtb_camera* c, const float lookfrom[3], const float lookat[3], const float up[3],
                       float vfov_deg, float aspect, float aperture, float focus_dist, float t0, float t1);
int rtb_camera_motion(rtb_camera* c, const float lookfrom[3], const float lookat[3], const float up[3],
                      float vfov_deg, float aspect, float t0, float t1);

/* ------------------------------------------------------------------ renderer */

typedef struct rtb_renderer rtb_renderer;

enum rtb_render_flags {
	RTB_RENDER_CLEAR = 1,      /* zero the accumulators before rendering */
	RTB_RENDER_VARIANCE = 2    /* also accumulate per-pixel sums of squares */
};

typedef struct rtb_render_params {
	uint32_t width, height;
	uint32_t sample_begin, sample_end; /* samples [begin,end) of every pixel (multi-GPU sample-range partition) */
	uint32_t row_begin, row_end;       /* image rows [begin,end); 0,0 = all rows (tile partition) */
	uint32_t max_depth;                /* path segments, Renderer.cu:146 */
	uint32_t seed;                     /* Philox key word 0 */
	uint32_t flags;
	uint32_t samples_per_batch;        /* 0 = auto */
} rtb_render_params;

typedef struct rtb_counters {
	uint64_t paths;        /* camera paths started */
	uint64_t rays;         /* ray segments submitted to closest-hit traversal */
	uint64_t launches;     /* kernels launched by this library */
	uint64_t batches;
	double   render_ms;    /* CUDA-event time of the last rtb_render call (valid after rtb_synchronize) */
} rtb_counters;

int  rtb_device_count(void);
int  rtb_renderer_create(rtb_renderer** out, int device);
void rtb_renderer_destroy(rtb_renderer* r);
/* Flattens the scene graph into SoA device buffers + one world BVH and uploads them. */
int  rtb_renderer_set_scene(rtb_renderer* r, rtb_scene* s);
int  rtb_renderer_set_camera(rtb_renderer* r, const rtb_camera* cam);
/* Bytes of the scene arena rtb_renderer_set_scene copies host -> device. */
size_t rtb_renderer_scene_bytes(const rtb_renderer* r);
/* Sizes, builder and build times of the scene last flattened by rtb_renderer_set_scene. */
int  rtb_renderer_scene_stats(const rtb_renderer* r, rtb_scene_stats* out);
/* Renders asynchronously on `stream`, ADDING radiance sums into the accumulators. */
int  rtb_render(rtb_renderer* r, const rtb_render_params* p, void* stream);
int  rtb_synchronize(rtb_renderer* r);
/* Device pointer to the float4[w*h] accumulator (rgb = radiance sums, a = sample count). */
void* rtb_renderer_accum_ptr(rtb_renderer* r);
void* rtb_renderer_accum2_ptr(rtb_renderer* r);
/* mean -> clamp[0,1] -> sqrt, alpha 1 (Renderer.cu:206-216); d_out = device float4[w*h] or NULL for the
 * renderer's own output buffer. */
int  rtb_resolve(rtb_renderer* r, void* d_out, void* stream);
/* Renderer::DownloadRenderbuffer: resolve + blocking copy of w*h float4 to host_rgba. */
int  rtb_download(rtb_renderer* r, float* host_rgba);
/* Raw accumulators (rgb sums + count) and sums of squares; either pointer may be NULL. */
int  rtb_download_accum(rtb_renderer* r, float* host_sum, float* host_sum2);
/* Output stage of FirstApp::write_renderbuffer (main/src/FirstApp.cpp:108-122) on the device: the resolved image
 * quantised as uint8 = value * 255.999f, RGB only, rows flipped when flip_rows != 0 (row 0 of the float buffer is the
 * bottom of the picture; stbi_flip_vertically_on_write(true) in the reference); host_rgb holds w*h*3 bytes. */
int  rtb_download_rgb8(rtb_renderer* r, uint8_t* host_rgb, int flip_rows);
/* Uploads to `r` the scene that `src` (a renderer on another device) flattened in its last rtb_renderer_set_scene:
 * one flatten, N uploads (what rtb_multi_set_scene does). */
int  rtb_renderer_share_scene(rtb_renderer* r, const rtb_renderer* src);

/* Progressive rendering across process lifetimes: a checkpoint holds the radiance sums, the sums of squares and the
 * sample cursor (one past the last sample index accumulated since the last RTB_RENDER_CLEAR).  A render continued
 * from a loaded checkpoint - rtb_render with sample_begin = the cursor and without RTB_RENDER_CLEAR - is bit-identical
 * to the uninterrupted one.  (The reference overwrites its output buffer on every Render(), Renderer.cu:216; its RNG
 * state persists instead - with counter-based streams the sample cursor is the whole state.) */
int  rtb_save_accum(rtb_renderer* r, const char* path);
int  rtb_load_accum(rtb_renderer* r, const char* path, uint32_t* width_out, uint32_t* height_out, uint32_t* sample_cursor_out);
uint32_t rtb_renderer_sample_cursor(const rtb_renderer* r);
int  rtb_get_counters(rtb_renderer* r, rtb_counters* out);

/* Adaptive sampling (DESIGN.md §5c): rounds of samples for the pixels whose estimated display-space error is still above
 * `tolerance`, until none is, every remaining one has p->sample_end samples, or max_rounds rounds have run.
 *
 * A pixel's error e is one standard error of its mean, taken through the clamp and square root of rtb_resolve; a pixel is
 * rendered in the next round while the maximum of e over its 3x3 neighbourhood (clipped to the row range) is above the
 * tolerance, and it has taken part in every round so far.  Every pixel first gets min_spp samples.  A stopped pixel never
 * resumes, so an active pixel always holds samples [0, cursor) - the same sums, bit for bit, that a uniform render of
 * `cursor` samples per pixel holds for it.  The decision is a pure function of the accumulators: a render continued in
 * another call, or from a loaded checkpoint, goes on exactly as the uninterrupted one.  tolerance = 10^(-D/20) leaves the
 * image about D dB from its converged value.
 *
 * p->sample_begin must be 0; p->sample_end is the cap (min_spp <= cap <= 2^24).  RTB_RENDER_CLEAR starts from zero; without
 * it the call continues from what the accumulators hold (a render from sample 0 with RTB_RENDER_VARIANCE, an earlier
 * adaptive call, a checkpoint).  Sums of squares are always accumulated.  Rows outside the row range are untouched.
 * The call blocks (it reads the number of active pixels once per round) and is ordered after and before `stream` as
 * rtb_render is; rtb_get_counters reports the device time of the whole call and its paths and rays.  Returns
 * RTB_ERR_INVALID for bad arguments, RTB_ERR_STATE when continuing an accumulator of another size, or one in which a pixel
 * holding the cursor's samples has no sums of squares (a render without RTB_RENDER_VARIANCE), whatever the cursor.  After
 * an error the sample cursor still covers the rounds rendered, and the call is ordered before `stream` as on success. */
typedef struct rtb_adaptive_params {
	float    tolerance;    /* display-space standard error at which a pixel stops (DESIGN.md §5c); >= 0, finite */
	uint32_t min_spp;      /* every pixel gets at least this many samples; >= 2 */
	uint32_t max_rounds;   /* 0 = until no pixel is active or every active pixel has p->sample_end samples */
	uint32_t reserved;
} rtb_adaptive_params;
typedef struct rtb_adaptive_stats {
	uint32_t rounds, cursor;   /* rounds run by this call; sample cursor after it */
	uint32_t active_pixels;    /* pixels the next round would render (0 = done) */
	uint32_t reserved;
	uint64_t samples;          /* camera paths started by this call */
} rtb_adaptive_stats;
int  rtb_render_adaptive(rtb_renderer* r, const rtb_render_params* p, const rtb_adaptive_params* a,
                         rtb_adaptive_stats* out, void* stream);

/* Per-kernel-class device time, measured with CUDA events around every launch on the stream the
 * kernels run on.  Profiling renders run as plain stream launches (no CUDA graph) and are meant for
 * the roofline accounting of bench.py, not for the headline timing. */
typedef struct rtb_profile {
	double   generate_ms, traverse_ms, shade_ms, accumulate_ms;
	uint64_t generate_launches, traverse_launches, shade_launches, accumulate_launches;
	double   tail_ms;          /* fused traverse+shade kernel that finishes short queues */
	uint64_t tail_launches;
	double   bin_ms;           /* ray binning between bounces (bin_scan + bin_permute) */
	uint64_t bin_launches;
} rtb_profile;
int  rtb_renderer_set_profiling(rtb_renderer* r, int on);
int  rtb_get_profile(rtb_renderer* r, rtb_profile* out);   /* synchronizes; totals since the last call */
/* The individual launches behind rtb_get_profile, in launch order (call it BEFORE rtb_get_profile, which resets):
 * ms_out[i] = device time, class_out[i] = 0 generate, 1 traverse, 2 shade (+ texture), 3 accumulate, 4 tail check,
 * 5 ray binning, 6 the select step of an adaptive round (rtb_render_adaptive; not in rtb_get_profile's totals).
 * Returns the number of launches recorded (may exceed cap). */
int  rtb_get_profile_launches(rtb_renderer* r, float* ms_out, int32_t* class_out, int cap);
int  rtb_reset_counters(rtb_renderer* r);
/* Live-queue length at every bounce of the LAST batch rendered (out[b], b < cap); returns max_depth. */
int  rtb_queue_lengths(rtb_renderer* r, uint32_t* out, int cap);

/* ------------------------------------------------------------------ hit-record parity hook */

typedef struct rtb_ray { float o[3]; float time; float d[3]; float pad; } rtb_ray;   /* 32 B */

typedef struct rtb_hit {                                                             /* 64 B */
	float   t;            /* _MISS_DIST (FLT_MAX) on miss */
	int32_t prim;         /* flattened primitive index, -1 on miss */
	int32_t object;       /* scene-graph object id of the primitive */
	int32_t material;
	float   p[3];
	float   n[3];         /* the normal materials see (spheres: outward; quads: facing the ray; triangles with normals:
	                         the interpolated shading normal, facing the ray) */
	int32_t front_face;   /* dot(d, geometric normal) <= 0 */
	float   u, v;         /* texture coordinates (triangles with UVs: the interpolated ones) */
	int32_t nodes_visited;   /* traversal statistics of this ray (rtb_trace_rays only): inner nodes visited, */
	int32_t prims_tested;    /* primitives intersected */
	int32_t pad;
} rtb_hit;

/* Closest hits for n host rays through the traversal code of the wavefront (media are skipped: they are
 * stochastic), with the full hit record materials would see and per-ray traversal statistics. */
int rtb_trace_rays(rtb_renderer* r, const rtb_ray* rays, size_t n, rtb_hit* hits_out);

/* Memory-safety evidence without compute-sanitizer: librtb200_debug.so is this library built with -DRTB_DEBUG_BOUNDS=1,
 * in which every index the kernels form from scene or queue data (traversal stack slot, node, primitive record, material,
 * texture / texel, queue slot, path id, bin) is checked against the size of what it indexes; violations are counted per
 * class - violations_out[0..7] in that order - instead of trapping, checks_out counts the rays that went through checked
 * kernels.  Returns the number of classes, or RTB_ERR_UNSUPPORTED from the release library. */
int rtb_debug_bounds_report(rtb_renderer* r, uint64_t* violations_out, int cap, uint64_t* checks_out);

/* ------------------------------------------------------------------ several GPUs of one box
 *
 * The reference renders on one device (main/src/FirstApp.cpp:39-40,94-101).  An rtb_multi_renderer drives one
 * rtb_renderer per device from a single process: the scene is flattened once and uploaded to every device, a render's
 * sample range [sample_begin, sample_end) is split into contiguous sub-ranges (device i of n renders
 * [begin + spp*i/n, begin + spp*(i+1)/n) of every pixel - perfectly balanced, and with counter-based random streams the
 * very samples one device would have drawn), all devices render concurrently, and the per-device radiance sums are
 * summed onto the first device: one ncclReduce(sum) per render over NVLink (NCCL is loaded at run time, libnccl.so.2),
 * or - RTB_REDUCE_P2P - one kernel on the first device that reads its peers' accumulators through peer memory and adds
 * them in device order (bit-reproducible).  rtb_multi_download then resolves and copies from the first device. */
typedef struct rtb_multi_renderer rtb_multi_renderer;
enum rtb_multi_reduce { RTB_REDUCE_AUTO = 0, RTB_REDUCE_NCCL = 1, RTB_REDUCE_P2P = 2 };

/* devices = n CUDA device indices (NULL: devices 0..n-1). */
int  rtb_multi_renderer_create(rtb_multi_renderer** out, const int* devices, int n, int reduce_mode);
void rtb_multi_renderer_destroy(rtb_multi_renderer* m);
int  rtb_multi_device_count(const rtb_multi_renderer* m);
/* The renderer of device slot i (counters, profiling, scene statistics); owned by m. */
rtb_renderer* rtb_multi_renderer_get(rtb_multi_renderer* m, int i);
/* RTB_REDUCE_NCCL or RTB_REDUCE_P2P: what this object uses (AUTO picks NCCL when it loads, else peer memory). */
int  rtb_multi_reduce_mode(const rtb_multi_renderer* m);
int  rtb_multi_set_scene(rtb_multi_renderer* m, rtb_scene* s);
int  rtb_multi_set_camera(rtb_multi_renderer* m, const rtb_camera* cam);
/* Asynchronous.  Without RTB_RENDER_CLEAR the new samples are added to what every device holds (progressive). */
int  rtb_multi_render(rtb_multi_renderer* m, const rtb_render_params* p);
int  rtb_multi_synchronize(rtb_multi_renderer* m);
/* Resolve of the cross-device total + blocking copy, as rtb_download / rtb_download_accum / rtb_download_rgb8. */
int  rtb_multi_download(rtb_multi_renderer* m, float* host_rgba);
int  rtb_multi_download_accum(rtb_multi_renderer* m, float* host_sum, float* host_sum2);
int  rtb_multi_download_rgb8(rtb_multi_renderer* m, uint8_t* host_rgb, int flip_rows);
/* paths, rays, launches, batches summed over the devices; render_ms = device time of the last rtb_multi_render from the
 * first launch to the end of the reduction, the slowest device (valid after rtb_multi_synchronize). */
int  rtb_multi_get_counters(rtb_multi_renderer* m, rtb_counters* out);
int  rtb_multi_reset_counters(rtb_multi_renderer* m);

#ifdef __cplusplus
}
#endif
#endif /* RTB_H */
