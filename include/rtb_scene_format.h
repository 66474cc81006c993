/*
 * rtb_scene_format.h — the flat binary scene description ("RTBS" v1) written by
 * rtb_scene_serialize().  It is the only thing the product library and the CPU oracle
 * share: the oracle parses this blob and evaluates the *object graph* the way the
 * reference / the book does (recursive lists, BVHs, ray-transforming instances, two
 * boundary queries per medium), while the product flattens the same graph into
 * world-space SoA buffers.  All records are little-endian, 4-byte aligned.
 *
 *   rtbs_header
 *   rtbs_texture  [n_textures]
 *   rtbs_material [n_materials]
 *   rtbs_object   [n_objects]
 *   int32         children[n_children]     (LIST / BVH members)
 *   uint8         blob[n_blob_bytes]       (image texels RGB8; Perlin tables)
 *   int32         n_lights                 (versions 2 and 3: the scene's sampled lights,
 *   int32         lights[n_lights]          rtb_scene_set_sampled_lights; in version 3 n_lights may be 0)
 *   rtbs_env      env                      (versions 3 and 4: the environment map, rtb_scene_set_environment;
 *   float         texels[height][width][3]  in version 4 width = height = 0 when there is none; row 0 = top; already
 *                                            multiplied by env.scale)
 *   uint32        n_tri_attrs              (version 4 only: per-vertex attributes of mesh triangles, rtb_add_mesh_ex)
 *   rtbs_tri_attr tri_attrs[n_tri_attrs]    (a TRIANGLE object whose `aux` is k + 1 carries tri_attrs[k]; aux = 0: none)
 *   uint32        n_materials              (version 5 only: the GGX width of every material, rtb_add_rough_metal /
 *   float         alpha[n_materials]        rtb_add_rough_dielectric; 0 for the other kinds)
 *
 * A scene without attributes is written as version 1 (no sampled lights), 2 or 3 (a map); one with attributes as
 * version 4; one with a rough material as version 5 (the version 4 content, then the widths).
 */
#ifndef RTB_SCENE_FORMAT_H
#define RTB_SCENE_FORMAT_H

#include <stdint.h>

#define RTBS_MAGIC 0x53425452u /* "RTBS" */
#define RTBS_VERSION 1u
#define RTBS_VERSION_LIGHTS 2u
#define RTBS_VERSION_ENV 3u
#define RTBS_VERSION_ATTR 4u
#define RTBS_VERSION_ROUGH 5u

/* Corner attributes of one triangle (DESIGN.md §5e), in the order of its corners v0 (= Q), v1 (= Q + u), v2 (= Q + v).
 * Normals are unit length or zero (normalised on the host); flags say which of the two are present. */
#define RTBS_ATTR_NORMALS 1
#define RTBS_ATTR_UVS 2
typedef struct rtbs_tri_attr {
	float   n[3][3];            /* corner normals (object frame of the triangle) */
	float   uv[3][2];           /* corner texture coordinates */
	int32_t flags;              /* RTBS_ATTR_NORMALS | RTBS_ATTR_UVS */
} rtbs_tri_attr;                /* 64 B */

typedef struct rtbs_env {
	int32_t width, height;
	int32_t flags;              /* RTB_ENV_SAMPLE */
	float   scale[3];           /* the scale the texels were multiplied by (informational) */
} rtbs_env;                     /* 24 B */

typedef struct rtbs_header {
	uint32_t magic, version;
	uint32_t n_textures, n_materials, n_objects, n_children;
	uint32_t n_blob_bytes;
	int32_t  root_object;
	int32_t  background_mode;   /* rtb_background_mode */
	float    background[3];
} rtbs_header;

/* Perlin tables in the blob: 256 x float[3] gradients, then perm_x/y/z: 3 x 256 x int32. */
#define RTBS_PERLIN_POINTS 256
#define RTBS_PERLIN_BYTES (256 * 3 * 4 + 3 * 256 * 4)

typedef struct rtbs_texture {
	int32_t  kind;          /* rtb_texture_kind */
	int32_t  even, odd;     /* checker children (texture ids) */
	float    scale;         /* checker: scale (inv_scale = 1/scale); noise: frequency */
	float    rgb[3];        /* solid colour */
	int32_t  width, height; /* image */
	uint32_t blob_offset;   /* image texels / Perlin tables */
	uint32_t seed;          /* noise */
	uint32_t pad;
} rtbs_texture;             /* 48 B */

typedef struct rtbs_material {
	int32_t kind;           /* rtb_material_kind */
	int32_t tex;            /* albedo / emission / phase texture id, -1 = use `albedo` */
	float   albedo[3];
	float   param;          /* metal: fuzz; dielectric, rough dielectric: ior */
} rtbs_material;            /* 24 B */

/* f[] per kind:
 *   SPHERE           center.xyz, radius
 *   MOVING_SPHERE    center0.xyz, radius, center1.xyz
 *   QUAD / TRIANGLE  Q.xyz, u.xyz, v.xyz
 *   BOX              a.xyz, b.xyz          (six quads, outward normals)
 *   TRANSLATE        offset.xyz            child = children[child_begin]
 *   ROTATE_Y         degrees, sin, cos     child = children[child_begin]
 *   CONSTANT_MEDIUM  density, -1/density   boundary = children[child_begin]; mat = phase material
 *   LIST / BVH       (none)                members = children[child_begin .. +child_count); BVH: builder in `aux`
 */
typedef struct rtbs_object {
	int32_t kind;           /* rtb_object_kind */
	int32_t mat;
	int32_t child_begin, child_count;
	int32_t aux;
	float   f[11];
} rtbs_object;              /* 64 B */

#endif
