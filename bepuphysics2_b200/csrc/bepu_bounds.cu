// PredictBoundingBoxes kernel (sm_100a), compiled -fmad=false with IEEE sqrt: the results are bit-identical to a non-contracting CPU evaluation of
// the reference's expressions (tests/test_bounds.py). One thread per body, fully coalesced: reads the 32-B pose / velocity / local inertia records
// the solver keeps resident (96 B), the 32-B shape record and the 8-B activity; writes 32 B of bounds + margin and the activity. HBM-bound
// (168 B per body); the bounding boxes of every body are independent, so there is nothing to order.
#define BEPU_NS bepu_bounds_math
#include "bepu_bounds_math.cuh"
#include "bepu_bounds.h"
#include "bepu_bounds_motion.cuh"

namespace bepucuda {

namespace {

using namespace bepu_bounds_math;

__global__ void predict_bounding_boxes_kernel(BodyBuffers B, const BodyShape* __restrict__ shapes, BodyActivityRecord* __restrict__ activities, float4* __restrict__ bounds,
                                              const __grid_constant__ PredictParams p) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B.count) return;
    const PredictedMotion m = load_predicted_motion(B, i, p);
    BodyActivityRecord activity = activities[i];
    update_sleep_candidacy(activity, m.sleep_energy);
    activities[i] = activity;

    const BodyShape shape = shapes[i];
    if (!(shape.type == 0 || shape.type == 1 || shape.type == 2 || shape.type == 4)) {
        bounds[2 * (size_t)i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        bounds[2 * (size_t)i + 1] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        return;
    }
    const ConvexShape convex = {shape.type, shape.a, shape.b, shape.c, shape.minimum_speculative_margin, shape.maximum_speculative_margin, shape.allow_expansion_beyond_speculative_margin};
    V3 bundleMin, bundleMax;
    float speculativeMargin;
    convex_bounds(convex, m.orientation, m.position, m.velocity, p.dt, bundleMin, bundleMax, speculativeMargin);
    bounds[2 * (size_t)i] = make_float4(bundleMin.x, bundleMin.y, bundleMin.z, speculativeMargin);
    bounds[2 * (size_t)i + 1] = make_float4(bundleMax.x, bundleMax.y, bundleMax.z, 1.0f);
}

}  // namespace

void launch_predict_bounding_boxes(const BodyBuffers& B, const BodyShape* shapes, BodyActivityRecord* activities, float4* bounds, const PredictParams& params, cudaStream_t s) {
    if (B.count <= 0) return;
    predict_bounding_boxes_kernel<<<(unsigned)((B.count + 255) / 256), 256, 0, s>>>(B, shapes, activities, bounds, params);
}

}  // namespace bepucuda
