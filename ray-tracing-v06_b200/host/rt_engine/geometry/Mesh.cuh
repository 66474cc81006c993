// Triangle meshes in the reference's *Handle idiom.  The reference's RT engine has no mesh type; its GL
// demo loads Wavefront OBJ files through tiny_obj (main/src/gl_engine/gl_mesh.cpp:124-218).  This loader
// reads the same subset that demo uses — `v x y z` and `f a b c ...` records (1-based or negative indices,
// `i/j/k` corner syntax, polygons fanned into triangles) — and registers one Triangle per face under a
// BVH group, so a mesh is an ordinary Hittable that can be listed, instanced or put in a BVH.
// LoadObjShaded also reads `vt` / `vn` records and `v/vt/vn`, `v//vn`, `v/vt` corners for smooth shading and texture
// mapping (rtb_add_mesh_ex, DESIGN.md §5e).
#pragma once
#include <cmath>
#include <map>
#include <tuple>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <glm/glm.hpp>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../rtb_context.h"
#include "../shaders/material.cuh"
#include "Quad.cuh"
#include "aabb.cuh"
#include "hittable.cuh"

class Mesh : public Geometry {
public:
	std::vector<glm::vec3> vertices;
	std::vector<int> indices;   // 3 per triangle, 0-based
	std::vector<glm::vec3> normals;   // per vertex, or empty: flat shading
	std::vector<glm::vec2> uvs;       // per vertex, or empty: textures read the triangles' own (alpha, beta)
};

class MeshHandle {
	aabb bounds;
	Hittable* hittable_ptr{};
	int triangle_count = 0;
	MeshHandle() = default;
	MeshHandle(const MeshHandle&) = delete;
	MeshHandle& operator=(const MeshHandle&) = delete;

public:
	MeshHandle(MeshHandle&& o) noexcept : bounds(o.bounds), hittable_ptr(o.hittable_ptr), triangle_count(o.triangle_count) { o.hittable_ptr = nullptr; }
	~MeshHandle() { delete hittable_ptr; }

	// Reads the `v` / `f` records of a Wavefront OBJ file.
	static Mesh LoadObj(const std::string& path) {
		FILE* f = fopen(path.c_str(), "r");
		if (!f) throw std::runtime_error("MeshHandle::LoadObj: cannot open " + path);
		Mesh m; char line[1024];
		while (fgets(line, sizeof line, f)) {
			if (line[0] == 'v' && (line[1] == ' ' || line[1] == '\t')) {
				float x, y, z;
				if (sscanf(line + 2, "%f %f %f", &x, &y, &z) == 3) m.vertices.push_back(glm::vec3(x, y, z));
			} else if (line[0] == 'f' && (line[1] == ' ' || line[1] == '\t')) {
				std::vector<int> corner;
				for (char* tok = strtok(line + 2, " \t\r\n"); tok; tok = strtok(nullptr, " \t\r\n")) {
					int i = atoi(tok);                                  // "i", "i/j", "i//k", "i/j/k": the vertex index comes first
					if (i < 0) i = (int)m.vertices.size() + i + 1;      // negative: relative to the vertices read so far
					if (i < 1 || i > (int)m.vertices.size()) { fclose(f); throw std::runtime_error("MeshHandle::LoadObj: bad face index in " + path); }
					corner.push_back(i - 1);
				}
				for (size_t k = 2; k < corner.size(); ++k) { m.indices.push_back(corner[0]); m.indices.push_back(corner[k - 1]); m.indices.push_back(corner[k]); }
			}
		}
		fclose(f);
		if (m.indices.empty()) throw std::runtime_error("MeshHandle::LoadObj: no faces in " + path);
		return m;
	}

	// Reads the `v`, `vt`, `vn` and `f` records of a Wavefront OBJ file for smooth shading.  Corners are `v`, `v/vt`, `v//vn`
	// or `v/vt/vn` (1-based or negative indices; polygons fanned into triangles as LoadObj does).
	//  - UVs come from `vt` when every corner names a `vt` record that exists; otherwise the mesh has none.
	//  - Normals come from `vn` when every corner names a `vn` record that exists.  Otherwise they are computed: the normal of
	//    position i is the sum, in double, of cross(p1 - p0, p2 - p0) over the triangles (after fanning) that have i as a
	//    corner - the face normals weighted by twice their area - divided by its length; a zero sum stays zero.
	//  - Every distinct combination of the indices in use - (v), (v, vt), (v, vn) or (v, vt, vn) - becomes one vertex, in
	//    the order of first appearance.
	static Mesh LoadObjShaded(const std::string& path) {
		FILE* f = fopen(path.c_str(), "r");
		if (!f) throw std::runtime_error("MeshHandle::LoadObjShaded: cannot open " + path);
		std::vector<glm::vec3> pos, nrm; std::vector<glm::vec2> tex;
		std::vector<int> corners;   // (v, vt, vn) per corner of the fanned triangles, 0-based, -1 = none
		auto resolve = [](const char* s, int count) {       // 1-based or negative (relative) index -> 0-based, or -1
			if (!*s) return -1;
			int i = atoi(s);
			if (i < 0) i = count + i + 1;
			return i - 1;
		};
		char line[1024]; bool bad = false;
		while (!bad && fgets(line, sizeof line, f)) {
			float x, y, z;
			if (line[0] == 'v' && (line[1] == ' ' || line[1] == '\t')) {
				if (sscanf(line + 2, "%f %f %f", &x, &y, &z) == 3) pos.push_back(glm::vec3(x, y, z));
			} else if (line[0] == 'v' && line[1] == 't' && (line[2] == ' ' || line[2] == '\t')) {
				if (sscanf(line + 3, "%f %f", &x, &y) == 2) tex.push_back(glm::vec2(x, y));
			} else if (line[0] == 'v' && line[1] == 'n' && (line[2] == ' ' || line[2] == '\t')) {
				if (sscanf(line + 3, "%f %f %f", &x, &y, &z) == 3) nrm.push_back(glm::vec3(x, y, z));
			} else if (line[0] == 'f' && (line[1] == ' ' || line[1] == '\t')) {
				std::vector<int> c;
				for (char* tok = strtok(line + 2, " \t\r\n"); tok; tok = strtok(nullptr, " \t\r\n")) {
					char* s1 = strchr(tok, '/'); char* s2 = s1 ? strchr(s1 + 1, '/') : nullptr;
					if (s1) *s1 = 0;
					if (s2) *s2 = 0;
					const int v = resolve(tok, (int)pos.size());
					if (v < 0 || v >= (int)pos.size()) { bad = true; break; }
					const int t = s1 ? resolve(s1 + 1, (int)tex.size()) : -1, n = s2 ? resolve(s2 + 1, (int)nrm.size()) : -1;
					c.push_back(v); c.push_back(t); c.push_back(n);
				}
				for (size_t k = 2; !bad && k < c.size() / 3; ++k)
					for (size_t q : {(size_t)0, k - 1, k}) corners.insert(corners.end(), c.begin() + 3 * q, c.begin() + 3 * q + 3);
			}
		}
		fclose(f);
		if (bad) throw std::runtime_error("MeshHandle::LoadObjShaded: bad face index in " + path);
		if (corners.empty()) throw std::runtime_error("MeshHandle::LoadObjShaded: no faces in " + path);
		bool use_vt = true, use_vn = true;
		for (size_t k = 0; k < corners.size(); k += 3) {
			use_vt = use_vt && corners[k + 1] >= 0 && corners[k + 1] < (int)tex.size();
			use_vn = use_vn && corners[k + 2] >= 0 && corners[k + 2] < (int)nrm.size();
		}
		std::vector<glm::vec3> computed;
		if (!use_vn) {
			std::vector<double> acc(3 * pos.size(), 0.0);
			for (size_t k = 0; k < corners.size(); k += 9) {
				const glm::vec3 &p0 = pos[corners[k]], &p1 = pos[corners[k + 3]], &p2 = pos[corners[k + 6]];
				const double e1[3] = {(double)p1.x - p0.x, (double)p1.y - p0.y, (double)p1.z - p0.z};
				const double e2[3] = {(double)p2.x - p0.x, (double)p2.y - p0.y, (double)p2.z - p0.z};
				const double cr[3] = {e1[1] * e2[2] - e1[2] * e2[1], e1[2] * e2[0] - e1[0] * e2[2], e1[0] * e2[1] - e1[1] * e2[0]};
				for (int j = 0; j < 3; ++j)
					for (int a = 0; a < 3; ++a) acc[3 * (size_t)corners[k + 3 * j] + a] += cr[a];
			}
			computed.resize(pos.size());
			for (size_t i = 0; i < pos.size(); ++i) {
				const double* a = &acc[3 * i];
				const double len = std::sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
				computed[i] = len > 0.0 ? glm::vec3((float)(a[0] / len), (float)(a[1] / len), (float)(a[2] / len)) : glm::vec3(0.0f);
			}
		}
		Mesh m;
		std::map<std::tuple<int, int, int>, int> vertex_of;
		for (size_t k = 0; k < corners.size(); k += 3) {
			const auto key = std::make_tuple(corners[k], use_vt ? corners[k + 1] : -1, use_vn ? corners[k + 2] : -1);
			auto it = vertex_of.find(key);
			if (it == vertex_of.end()) {
				it = vertex_of.emplace(key, (int)m.vertices.size()).first;
				m.vertices.push_back(pos[corners[k]]);
				m.normals.push_back(use_vn ? nrm[corners[k + 2]] : computed[corners[k]]);
				if (use_vt) m.uvs.push_back(tex[corners[k + 1]]);
			}
			m.indices.push_back(it->second);
		}
		return m;
	}

	template <typename MatType> requires GeoAcceptableMat<Triangle, MatType>
	static MeshHandle MakeMesh(const Mesh& mesh, MatType* mat) {
		MeshHandle h{};
		static_assert(sizeof(glm::vec3) == 3 * sizeof(float), "vertices are handed over as packed floats");
		static_assert(sizeof(glm::vec2) == 2 * sizeof(float), "UVs are handed over as packed floats");
		const bool attrs = !mesh.normals.empty() || !mesh.uvs.empty();
		if ((!mesh.normals.empty() && mesh.normals.size() != mesh.vertices.size()) || (!mesh.uvs.empty() && mesh.uvs.size() != mesh.vertices.size()))
			throw std::runtime_error("MakeMesh: normals and UVs must be per vertex");
		const int group = attrs
			? rtb_host::check(rtb_add_mesh_ex(rtb_host::scene(), &mesh.vertices[0].x, (int)mesh.vertices.size(), mesh.indices.data(),
			                                  (int)(mesh.indices.size() / 3), mesh.normals.empty() ? nullptr : &mesh.normals[0].x,
			                                  mesh.uvs.empty() ? nullptr : &mesh.uvs[0].x, mat->rtb_material), "MakeMesh")
			: rtb_host::check(rtb_add_mesh(rtb_host::scene(), &mesh.vertices[0].x, (int)mesh.vertices.size(), mesh.indices.data(),
			                               (int)(mesh.indices.size() / 3), mat->rtb_material), "MakeMesh");
		const int faces = rtb_host::check(rtb_scene_num_children(rtb_host::scene(), group), "MakeMesh");
		float bb[6]; rtb_host::check(rtb_object_bounds(rtb_host::scene(), group, bb), "rtb_object_bounds");
		h.bounds = aabb(glm::vec3(bb[0], bb[1], bb[2]), glm::vec3(bb[3], bb[4], bb[5]));
		h.hittable_ptr = new GeoHittable(group);
		h.triangle_count = faces;
		return h;
	}
	const Hittable* getHittablePtr() const { return hittable_ptr; }
	aabb getBounds() const { return bounds; }
	int triangleCount() const { return triangle_count; }
};
