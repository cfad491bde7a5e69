// TEST INFRASTRUCTURE. Compiles csrc/bepu_shape_bounds_math.cuh (the arithmetic of bepucuda_set_body_collidables' PredictBoundingBoxes kernels) for
// the HOST over the stub cuda_runtime.h and evaluates one body per call, with the reductions of csrc/bepu_shape_bounds.cu replayed in the kernels'
// own combining order: the hull's lanes and the compound's lane runs merged by the same offset-1, 2, 4, ... tree, the mesh's triangles split into
// chunks and strided over 256 "threads" with the keyed combine. tests/test_bounds_all_shapes.py holds it to the reference-derived vectors bit for bit.
//
// Build: g++ -O2 -std=c++17 -ffp-contract=off -fno-fast-math -march=x86-64-v3 -I tests/device_on_host/stubs -I bepuphysics2_b200/csrc -shared -fPIC
#define BEPU_NS bepu_shape_bounds_on_host
#include "bepu_shape_bounds_math.cuh"

#include <climits>
#include <vector>

using namespace BEPU_NS;

// include/bepucuda.h's bepucuda_shape_library
struct HostShapeLibrary {
    const float *spheres, *capsules, *boxes, *triangles, *cylinders, *hull_points;
    const HullRecord* hulls;
    const CompoundChildRecord* compound_children;
    const CompoundRecord *compounds, *big_compounds;
    const float* mesh_triangles;
    const MeshRecord* meshes;
    int64_t counts[13];
};

static const int kLanes = 32;

// The kernels' warp tree: offsets 1, 2, 4, 8, 16, lane l takes lane l + offset when l is a multiple of 2 * offset.
template <class T, class Merge> static T warp_tree(std::vector<T> lanes, Merge merge) {
    for (int offset = 1; offset < kLanes; offset <<= 1)
        for (int l = 0; l + offset < kLanes; l += 2 * offset) merge(lanes[l], lanes[l + offset]);
    return lanes[0];
}

// shape = TypedIndex.Packed; margins {min, max}, allow, orientation, position, linear, angular (AFTER the callback), dt; mesh_chunk: triangles per
// chunk of the mesh pass. out: min.xyz, margin, max.xyz. -1: no built-in bounds.
extern "C" int32_t shape_bounds_on_host(const HostShapeLibrary* library, uint32_t shape, const float* margins, int32_t allow, const float* q, const float* pos, const float* lin,
                                        const float* ang, float dt, int32_t mesh_chunk, float* out) {
    const HostShapeLibrary& h = *library;
    const ShapeLibraryView lib = {h.spheres, h.capsules, h.boxes, h.triangles, h.cylinders, h.hull_points, h.hulls, h.compound_children, h.compounds, h.big_compounds,
                                  h.mesh_triangles, h.meshes, (int32_t)h.counts[5]};
    if (!typed_index_exists(shape) || typed_index_type(shape) > kMesh) return -1;
    const int32_t type = typed_index_type(shape), index = typed_index_index(shape);
    const BodyCollidableRecord c = {shape, margins[0], margins[1], allow};
    const Q4 orientation = {q[0], q[1], q[2], q[3]};
    const V3 position = {pos[0], pos[1], pos[2]};
    const Velocity velocity = {{lin[0], lin[1], lin[2]}, {ang[0], ang[1], ang[2]}};
    V3 mn, mx;
    float margin;
    if (type <= kCylinder) {
        expand_convex_bounds(convex_local_bounds(lib, type, index, orientation), c, position, velocity, dt, mn, mx, margin);
    } else if (type == kConvexHull) {
        const M33 m = matrix_from_quaternion(orientation);
        std::vector<HullLane> lanes(kLanes, HullLane{{3.40282347e+38f, 3.40282347e+38f, 3.40282347e+38f}, {-3.40282347e+38f, -3.40282347e+38f, -3.40282347e+38f}, 0.0f});
        for (int l = 0; l < lib.hull_width; ++l) lanes[l] = hull_lane_fold(lib.hull_points, lib.hull_width, lib.hulls[index], l, m);
        expand_convex_bounds(hull_finish(warp_tree(lanes, [](HullLane& a, const HullLane& b) { hull_lane_merge(a, b); })), c, position, velocity, dt, mn, mx, margin);
    } else if (type == kCompound || type == kBigCompound) {
        const CompoundRecord compound = (type == kCompound ? lib.compounds : lib.big_compounds)[index];
        const int per = (compound.child_count + kLanes - 1) / kLanes;
        std::vector<MergedBounds> lanes(kLanes, merged_bounds_start());
        for (int l = 0; l < kLanes; ++l)
            for (int k = l * per; k < compound.child_count && k < (l + 1) * per; ++k)
                merge_bounds(lanes[l], compound_child_bounds(lib, lib.compound_children[compound.first_child + k], c, orientation, position, velocity, dt));
        const MergedBounds merged = warp_tree(lanes, [](MergedBounds& a, const MergedBounds& b) { merge_bounds(a, b); });
        mn = merged.min, mx = merged.max, margin = merged.speculativeMargin;
    } else {
        const MeshRecord mesh = lib.meshes[index];
        const M33 r = narrow_matrix_from_quaternion(orientation);
        const V3 scale = {mesh.scale[0], mesh.scale[1], mesh.scale[2]};
        V3 runMin = {3.40282347e+38f, 3.40282347e+38f, 3.40282347e+38f}, runMax = {-3.40282347e+38f, -3.40282347e+38f, -3.40282347e+38f};
        for (int32_t first = 0; first < mesh.triangle_count; first += mesh_chunk) {
            const int32_t count = mesh.triangle_count - first < mesh_chunk ? mesh.triangle_count - first : mesh_chunk;
            float best[6];
            int32_t key[6];
            for (int d = 0; d < 6; ++d) best[d] = d < 3 ? 3.40282347e+38f : -3.40282347e+38f, key[d] = INT_MAX;
            for (int thread = 0; thread < 256; ++thread) {
                float v[6];
                int32_t k[6];
                for (int d = 0; d < 6; ++d) v[d] = d < 3 ? 3.40282347e+38f : -3.40282347e+38f, k[d] = INT_MAX;
                for (int32_t t = thread; t < count; t += 256) {
                    V3 a, b, cc;
                    mesh_triangle_vertices(lib.mesh_triangles + 9 * ((size_t)mesh.first_triangle + first + t), scale, r, a, b, cc);
                    mesh_fold_min(a.x, b.x, cc.x, t, v[0], k[0]), mesh_fold_min(a.y, b.y, cc.y, t, v[1], k[1]), mesh_fold_min(a.z, b.z, cc.z, t, v[2], k[2]);
                    mesh_fold_max(a.x, b.x, cc.x, t, v[3], k[3]), mesh_fold_max(a.y, b.y, cc.y, t, v[4], k[4]), mesh_fold_max(a.z, b.z, cc.z, t, v[5], k[5]);
                }
                for (int d = 0; d < 3; ++d) mesh_combine_min(best[d], key[d], v[d], k[d]);
                for (int d = 3; d < 6; ++d) mesh_combine_max(best[d], key[d], v[d], k[d]);
            }
            runMin = vmin3(V3{best[0], best[1], best[2]}, runMin);
            runMax = vmax3(V3{best[3], best[4], best[5]}, runMax);
        }
        mesh_bounds(runMin, runMax, c, position, velocity, dt, mn, mx, margin);
    }
    out[0] = mn.x; out[1] = mn.y; out[2] = mn.z; out[3] = margin; out[4] = mx.x; out[5] = mx.y; out[6] = mx.z;
    return 0;
}
