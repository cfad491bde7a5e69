// ORACLE PINNING — test infrastructure only. System.Numerics.Vector3 / Quaternion (the narrow types) on top of ref_runtime.h, for the transpiled
// QuaternionEx / Matrix3x3 helpers and the Vector3 overloads of BoundingBoxHelpers (oracle/ref_transpile/shape_bounds_ref.py): component-wise IEEE
// fp32. Vector3.Min / Max lower to minps / maxps like Vector.Min / Max ((a < b) ? a : b); Length = Sqrt(Dot(v, v)) with the dot product summed x, y, z
// in order. Compiled -ffp-contract=off.
#pragma once
#include "ref_runtime.h"

namespace bepu_ref {

struct Vector3 {
    float X, Y, Z;
    Vector3() = default;
    explicit Vector3(float v) : X(v), Y(v), Z(v) {}
    Vector3(float x, float y, float z) : X(x), Y(y), Z(z) {}
    static Vector3 Zero() { return Vector3(0.0f); }
    float LengthSquared() const { return X * X + Y * Y + Z * Z; }
    float Length() const { return std::sqrt(LengthSquared()); }
    static Vector3 Min(Vector3 a, Vector3 b) { return {a.X < b.X ? a.X : b.X, a.Y < b.Y ? a.Y : b.Y, a.Z < b.Z ? a.Z : b.Z}; }
    static Vector3 Max(Vector3 a, Vector3 b) { return {a.X > b.X ? a.X : b.X, a.Y > b.Y ? a.Y : b.Y, a.Z > b.Z ? a.Z : b.Z}; }
    static Vector3 Abs(Vector3 a) { return {std::fabs(a.X), std::fabs(a.Y), std::fabs(a.Z)}; }
    static Vector3 Cross(Vector3 a, Vector3 b) { return {a.Y * b.Z - a.Z * b.Y, a.Z * b.X - a.X * b.Z, a.X * b.Y - a.Y * b.X}; }
};
inline Vector3 operator+(Vector3 a, Vector3 b) { return {a.X + b.X, a.Y + b.Y, a.Z + b.Z}; }
inline Vector3 operator-(Vector3 a, Vector3 b) { return {a.X - b.X, a.Y - b.Y, a.Z - b.Z}; }
inline Vector3 operator*(Vector3 a, Vector3 b) { return {a.X * b.X, a.Y * b.Y, a.Z * b.Z}; }
inline Vector3 operator*(Vector3 a, float s) { return {a.X * s, a.Y * s, a.Z * s}; }
inline Vector3 operator*(float s, Vector3 a) { return {s * a.X, s * a.Y, s * a.Z}; }
inline Vector3 operator-(Vector3 a) { return {-a.X, -a.Y, -a.Z}; }
struct Quaternion { float X, Y, Z, W; };

}  // namespace bepu_ref
