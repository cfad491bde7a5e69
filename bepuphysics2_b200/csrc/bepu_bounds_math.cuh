// Per-body arithmetic of PredictBoundingBoxes (see bepu_bounds.cu): plain scalar fp32 behind __device__, in its own header so that
// tests/device_on_host can compile it for the host and hold it to the reference-derived vectors without a GPU. Expression shapes follow the reference
// (file:line per function); compiled without FMA contraction.
#pragma once
#include "bepu_device_math.cuh"

namespace BEPU_NS {

struct ConvexShape { int32_t type; float a, b, c, minimum_speculative_margin, maximum_speculative_margin; int32_t allow_expansion_beyond_speculative_margin; };

struct LocalBounds { V3 max; float maximumRadius, maximumAngularExpansion; };

// IConvexShape wide GetBounds, one lane: Sphere.cs:L149-160, Capsule.cs:L226-239, Box.cs:L211-222, Cylinder.cs:L222-235. All four are symmetric (min = -max).
BEPU_DI LocalBounds shape_bounds(const ConvexShape& s, Q4 q) {
    LocalBounds r;
    if (s.type == 0) {
        r.max = {s.a, s.a, s.a};
        r.maximumRadius = 0.0f;
        r.maximumAngularExpansion = 0.0f;
    } else if (s.type == 1) {
        const float radius = s.a, halfLength = s.b;
        V3 segmentOffset = transform_unit_y(q) * halfLength;
        segmentOffset = {fabsf(segmentOffset.x), fabsf(segmentOffset.y), fabsf(segmentOffset.z)};
        r.max = {segmentOffset.x + radius, segmentOffset.y + radius, segmentOffset.z + radius};
        r.maximumRadius = halfLength + radius;
        r.maximumAngularExpansion = halfLength;
    } else if (s.type == 2) {
        const float halfWidth = s.a, halfHeight = s.b, halfLength = s.c;
        const M33 basis = matrix_from_quaternion(q);
        r.max.x = fabsf(halfWidth * basis.x.x) + fabsf(halfHeight * basis.y.x) + fabsf(halfLength * basis.z.x);
        r.max.y = fabsf(halfWidth * basis.x.y) + fabsf(halfHeight * basis.y.y) + fabsf(halfLength * basis.z.y);
        r.max.z = fabsf(halfWidth * basis.x.z) + fabsf(halfHeight * basis.y.z) + fabsf(halfLength * basis.z.z);
        r.maximumRadius = sqrtf(halfWidth * halfWidth + halfHeight * halfHeight + halfLength * halfLength);
        // as written in the reference (Box.cs:L221): HalfLength appears twice, HalfWidth not at all
        r.maximumAngularExpansion = r.maximumRadius - fmin_ps(halfLength, fmin_ps(halfHeight, halfLength));
    } else {
        const float radius = s.a, halfLength = s.b;
        const V3 y = transform_unit_y(q);
        const V3 squared = {1.0f - y.x * y.x, 1.0f - y.y * y.y, 1.0f - y.z * y.z};
        r.max.x = fabsf(halfLength * y.x) + sqrtf(fmax_ps(0.0f, squared.x)) * radius;
        r.max.y = fabsf(halfLength * y.y) + sqrtf(fmax_ps(0.0f, squared.y)) * radius;
        r.max.z = fabsf(halfLength * y.z) + sqrtf(fmax_ps(0.0f, squared.z)) * radius;
        r.maximumRadius = sqrtf(halfLength * halfLength + radius * radius);
        r.maximumAngularExpansion = r.maximumRadius - fmin_ps(halfLength, radius);
    }
    return r;
}

// BoundingBoxHelpers.GetAngularBoundsExpansion (BoundingBoxHelpers.cs:L12-45)
BEPU_DI float angular_bounds_expansion(float angularSpeed, float dt, float maximumRadius, float maximumAngularExpansion) {
    const float a = fmin_ps(angularSpeed * dt, 3.14159274f / 3.0f);
    const float a2 = a * a;
    const float a4 = a2 * a2;
    const float a6 = a4 * a2;
    const float cosAngleMinusOne = a2 * (-1.0f / 2.0f) + a4 * (1.0f / 24.0f) - a6 * (1.0f / 720.0f);
    return fmin_ps(maximumAngularExpansion, sqrtf(-2.0f * maximumRadius * maximumRadius * cosAngleMinusOne));
}

// BoundingBoxBatcher.ExecuteConvexBatch for one body (BoundingBoxBatcher.cs:L176-197), from the shape's local bounds onwards; `velocity` is the
// velocity AFTER the integration callback. The margins are the ones of the body's collidable (also for a compound child: its parent's).
BEPU_DI void expand_convex_bounds(V3 localMin, V3 localMax, float maximumRadius, float maximumAngularExpansion, float minimumSpeculativeMargin, float maximumSpeculativeMargin,
                                  int32_t allowExpansionBeyondSpeculativeMargin, V3 position, const Velocity& velocity, float dt, V3& bundleMin, V3& bundleMax, float& speculativeMargin) {
    const float angularBoundsExpansion = angular_bounds_expansion(length(velocity.ang), dt, maximumRadius, maximumAngularExpansion);
    speculativeMargin = length(velocity.lin) * dt + angularBoundsExpansion;
    speculativeMargin = fmax_ps(minimumSpeculativeMargin, fmin_ps(maximumSpeculativeMargin, speculativeMargin));
    const float maximumBoundsExpansion = allowExpansionBeyondSpeculativeMargin ? 3.40282347e+38f : speculativeMargin;
    // BoundingBoxHelpers.GetBoundsExpansion (BoundingBoxHelpers.cs:L49-58)
    const V3 linearDisplacement = velocity.lin * dt;
    V3 minExpansion = {fmin_ps(0.0f, linearDisplacement.x) - angularBoundsExpansion, fmin_ps(0.0f, linearDisplacement.y) - angularBoundsExpansion, fmin_ps(0.0f, linearDisplacement.z) - angularBoundsExpansion};
    V3 maxExpansion = {fmax_ps(0.0f, linearDisplacement.x) + angularBoundsExpansion, fmax_ps(0.0f, linearDisplacement.y) + angularBoundsExpansion, fmax_ps(0.0f, linearDisplacement.z) + angularBoundsExpansion};
    minExpansion = {fmax_ps(-maximumBoundsExpansion, minExpansion.x), fmax_ps(-maximumBoundsExpansion, minExpansion.y), fmax_ps(-maximumBoundsExpansion, minExpansion.z)};
    maxExpansion = {fmin_ps(maximumBoundsExpansion, maxExpansion.x), fmin_ps(maximumBoundsExpansion, maxExpansion.y), fmin_ps(maximumBoundsExpansion, maxExpansion.z)};
    bundleMin = position + (localMin + minExpansion);
    bundleMax = position + (localMax + maxExpansion);
}

// The symmetric primitives (sphere, capsule, box, cylinder): local min = -max.
BEPU_DI void convex_bounds(const ConvexShape& shape, Q4 orientation, V3 position, const Velocity& velocity, float dt, V3& bundleMin, V3& bundleMax, float& speculativeMargin) {
    const LocalBounds local = shape_bounds(shape, orientation);
    expand_convex_bounds(-local.max, local.max, local.maximumRadius, local.maximumAngularExpansion, shape.minimum_speculative_margin, shape.maximum_speculative_margin,
                         shape.allow_expansion_beyond_speculative_margin, position, velocity, dt, bundleMin, bundleMax, speculativeMargin);
}

// DemoPoseIntegratorCallbacks.IntegrateVelocity (Demos/DemoCallbacks.cs:L99-104) on a copy of the velocity: PredictBoundingBoxes bounds the body
// with the integrated velocity but does not store it (PoseIntegrator.cs:L339). Every bounds kernel goes through this one function.
BEPU_DI Velocity predicted_velocity(Velocity velocity, bool integrate, const float gravityDt[3], float linearDampingDt, float angularDampingDt) {
    if (integrate) {
        velocity.lin = (velocity.lin + V3{gravityDt[0], gravityDt[1], gravityDt[2]}) * linearDampingDt;
        velocity.ang = velocity.ang * angularDampingDt;
    }
    return velocity;
}

}  // namespace BEPU_NS
