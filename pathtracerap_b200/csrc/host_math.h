// host_math.h - host-side binary32 helpers in the evaluation order of the reference's vendored glm 0.9.6.3
// (paths: /root/reference/PathTracerAP/external/include/glm/...).  Compiled with -ffp-contract=off, so each
// operation rounds exactly as the device's explicit-rounding intrinsics do (exact_math.cuh).
#pragma once
#include <cmath>

#include <cuda_runtime.h>

namespace ptap { namespace hm {

struct V3 { float x, y, z; };
inline V3 v3(float x, float y, float z) { V3 r; r.x = x; r.y = y; r.z = z; return r; }
inline V3 v3(const float* p) { return v3(p[0], p[1], p[2]); }
inline V3 add(V3 a, V3 b) { return v3(a.x + b.x, a.y + b.y, a.z + b.z); }
inline V3 sub(V3 a, V3 b) { return v3(a.x - b.x, a.y - b.y, a.z - b.z); }
inline V3 scale(V3 a, float s) { return v3(a.x * s, a.y * s, a.z * s); }
inline float dot(V3 a, V3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }                 // detail/func_geometric.inl:65-72
inline V3 cross(V3 x, V3 y) { return v3(x.y * y.z - y.y * x.z, x.z * y.x - y.z * x.x, x.x * y.y - y.x * x.y); }   // :134-142
inline V3 normalize(V3 v) { return scale(v, 1.0f / std::sqrt(dot(v, v))); }                    // :154-159
// (m0*x + m1*y) + (m2*z + m3*w), detail/type_mat4x4.inl:617-627; m column-major
inline V3 mat4_mul(const float* m, V3 v, float w)
{
    return v3((m[0] * v.x + m[4] * v.y) + (m[8] * v.z + m[12] * w),
              (m[1] * v.x + m[5] * v.y) + (m[9] * v.z + m[13] * w),
              (m[2] * v.x + m[6] * v.y) + (m[10] * v.z + m[14] * w));
}

// rows of transpose(inverse(mat3(M))) as utility.h:82-88 evaluates it (inverse: detail/type_mat3x3.inl:37-56).
// out[3*r + k] multiplies n[k] in component r.  Also compiled for the device (k_update_instances, -fmad=false): the same bits.
__host__ __device__ inline void normal_matrix(const float* M, float out[9])
{
    auto m = [&](int c, int r) { return M[4 * c + r]; };
    const float ood = 1.0f / (+m(0, 0) * (m(1, 1) * m(2, 2) - m(2, 1) * m(1, 2))
                              - m(1, 0) * (m(0, 1) * m(2, 2) - m(2, 1) * m(0, 2))
                              + m(2, 0) * (m(0, 1) * m(1, 2) - m(1, 1) * m(0, 2)));
    // Inverse[c][r]; component r of transpose(Inverse) * n = sum_k Inverse[r][k] * n[k]
    float inv[3][3];
    inv[0][0] = +(m(1, 1) * m(2, 2) - m(2, 1) * m(1, 2)) * ood;
    inv[1][0] = -(m(1, 0) * m(2, 2) - m(2, 0) * m(1, 2)) * ood;
    inv[2][0] = +(m(1, 0) * m(2, 1) - m(2, 0) * m(1, 1)) * ood;
    inv[0][1] = -(m(0, 1) * m(2, 2) - m(2, 1) * m(0, 2)) * ood;
    inv[1][1] = +(m(0, 0) * m(2, 2) - m(2, 0) * m(0, 2)) * ood;
    inv[2][1] = -(m(0, 0) * m(2, 1) - m(2, 0) * m(0, 1)) * ood;
    inv[0][2] = +(m(0, 1) * m(1, 2) - m(1, 1) * m(0, 2)) * ood;
    inv[1][2] = -(m(0, 0) * m(1, 2) - m(1, 0) * m(0, 2)) * ood;
    inv[2][2] = +(m(0, 0) * m(1, 1) - m(1, 0) * m(0, 1)) * ood;
    for (int r = 0; r < 3; ++r)
        for (int k = 0; k < 3; ++k) out[3 * r + k] = inv[r][k];
}

}}  // namespace ptap::hm
