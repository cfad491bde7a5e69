// The motion state PredictBoundingBoxes bounds one body with (PoseIntegrator.cs:L307-370), read from the body arrays the solver keeps resident.
// Shared by every bounds kernel (bepu_bounds.cu, bepu_shape_bounds.cu) so that the integrated velocity is the same bits in all of them.
// Include after bepu_bounds_math.cuh and bepu_bounds.h.
#pragma once

namespace bepucuda {

struct PredictedMotion {
    BEPU_NS::Q4 orientation;
    BEPU_NS::V3 position;
    BEPU_NS::Velocity velocity;  // after the velocity callback
    float sleep_energy;          // |v|^2 + |w|^2 of the velocity BEFORE the callback (UpdateSleepCandidacy, L286-304)
};

__device__ __forceinline__ PredictedMotion load_predicted_motion(const BodyBuffers& B, int i, const PredictParams& p) {
    using namespace BEPU_NS;
    const float4 q4 = B.pose[2 * (size_t)i], p4 = B.pose[2 * (size_t)i + 1];
    const float4 l4 = B.velocity[2 * (size_t)i], w4 = B.velocity[2 * (size_t)i + 1];
    const float4 i0 = B.inertia_local[2 * (size_t)i], i1 = B.inertia_local[2 * (size_t)i + 1];
    PredictedMotion m;
    m.orientation = {q4.x, q4.y, q4.z, q4.w};
    m.position = {p4.x, p4.y, p4.z};
    const Velocity velocity = {{l4.x, l4.y, l4.z}, {w4.x, w4.y, w4.z}};
    // Bodies.IsKinematic (Bodies.cs:L326-331): every bit of inverse mass and inverse inertia is zero
    const bool kinematic = (__float_as_uint(i1.z) | __float_as_uint(i0.x) | __float_as_uint(i0.y) | __float_as_uint(i0.z) | __float_as_uint(i0.w) | __float_as_uint(i1.x) | __float_as_uint(i1.y)) == 0u;
    m.sleep_energy = length_squared(velocity.lin) + length_squared(velocity.ang);
    m.velocity = predicted_velocity(velocity, p.integrate_velocity_for_kinematics != 0 || !kinematic, p.gravity_dt, p.linear_damping_dt, p.angular_damping_dt);
    return m;
}

// UpdateSleepCandidacy (PoseIntegrator.cs:L286-304)
__device__ __forceinline__ void update_sleep_candidacy(BodyActivityRecord& activity, float sleepEnergy) {
    if (sleepEnergy > activity.sleep_threshold) {
        activity.timesteps_under_threshold_count = 0;
        activity.sleep_candidate = 0;
    } else if (activity.timesteps_under_threshold_count < 255) {
        ++activity.timesteps_under_threshold_count;
        if (activity.timesteps_under_threshold_count >= activity.minimum_timesteps_under_threshold) activity.sleep_candidate = 1;
    }
}

}  // namespace bepucuda
