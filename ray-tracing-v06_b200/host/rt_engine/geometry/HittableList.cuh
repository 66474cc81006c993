// Host mirror of main/src/rt_engine/geometry/HittableList.cuh:10-34.
#pragma once
#include <vector>

#include "../../rtb_context.h"
#include "aabb.cuh"
#include "hittable.cuh"

class HittableList : public Hittable {
	aabb bounds;
	std::vector<int> ids;

public:
	HittableList(const Hittable** objects, int object_count, const aabb& bounds) : bounds(bounds), ids(object_count) {
		for (int i = 0; i < object_count; ++i) ids[i] = objects[i]->rtb_object;
		rtb_object = rtb_host::check(rtb_add_list(rtb_host::scene(), ids.data(), object_count), "HittableList");
	}
	aabb getBounds() const { return bounds; }
	const std::vector<int>& memberIds() const { return ids; }   // object ids of the members, in list order
};
