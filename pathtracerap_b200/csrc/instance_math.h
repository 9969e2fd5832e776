// instance_math.h - what a model's placement contributes to the two-level BVH: its world box (a TLAS leaf) and its terms of the scene
// constants tmin_world / prune / tie / c_pad.  One definition for the host (api.cu: finishBvh, after an upload or a build) and the device
// (bvh_device.cu: k_update_instances, ptap_update_models), so that both derive the same bits: double and binary32 operations that the
// host (-ffp-contract=off) and the device (-fmad=false) round alike, and min / max written as std::min / std::max evaluate them.
#pragma once
#include <math.h>

#include "bvh_build.h"

namespace ptap {

__host__ __device__ inline double maxD(double a, double b) { return a < b ? b : a; }     // std::max
__host__ __device__ inline float minF(float a, float b) { return b < a ? b : a; }        // std::min
__host__ __device__ inline float maxF(float a, float b) { return a < b ? b : a; }        // std::max

// 3x3 inverse in double; false when the matrix is singular
__host__ __device__ inline bool invert3(const double m[9], double out[9])
{
    const double c0 = m[4] * m[8] - m[5] * m[7], c1 = m[5] * m[6] - m[3] * m[8], c2 = m[3] * m[7] - m[4] * m[6];
    const double det = m[0] * c0 + m[1] * c1 + m[2] * c2;
    if (!(fabs(det) > 1e-300)) return false;
    const double id = 1.0 / det;
    out[0] = c0 * id; out[1] = (m[2] * m[7] - m[1] * m[8]) * id; out[2] = (m[1] * m[5] - m[2] * m[4]) * id;
    out[3] = c1 * id; out[4] = (m[0] * m[8] - m[2] * m[6]) * id; out[5] = (m[2] * m[3] - m[0] * m[5]) * id;
    out[6] = c2 * id; out[7] = (m[1] * m[6] - m[0] * m[7]) * id; out[8] = (m[0] * m[4] - m[1] * m[3]) * id;
    return true;
}

// the 3x3 of world_to_model (column-major 4x4) as a row-major double matrix
__host__ __device__ inline void linearPart(const float* W, double w3[9])
{
    const double m[9] = {W[0], W[4], W[8], W[1], W[5], W[9], W[2], W[6], W[10]};
    for (int k = 0; k < 9; ++k) w3[k] = m[k];
}

struct InstanceBox {
    float lo[3], hi[3];     // world box, padded
    double scale;           // Frobenius norm of the inverse of world_to_model's 3x3
    double pad;             // the box's padding
    double trans;           // max(1, |translation of model_to_world|) over the entries the M W = I check visited
    bool consistent;        // M W = I within 2e-5 (relative to the translation in the last column)
};

// World box and scene-constant terms of an instance of the BLAS whose root node is `root`, under world_to_model W and model_to_world M
// (column-major 4x4; row 3 is not read).  False when W is singular.
__host__ __device__ inline bool instanceBox(const float* W, const float* M, const BvhNode& root, InstanceBox& out)
{
    // The kernel maps a world ray into model space with world_to_model (Renderer.cpp:381-382), so the world box of an instance is the image
    // of the BLAS root bounds under the INVERSE of world_to_model (= model_to_world when the two are consistent).
    double w3[9], wi[9];
    linearPart(W, w3);
    if (!invert3(w3, wi)) return false;
    out.trans = 1.0; out.consistent = true;
    for (int r = 0; r < 3 && out.consistent; ++r)
        for (int c = 0; c < 4; ++c) {          // (M * W)[r][c] against the identity; stops at the first entry that fails
            const double scale = c == 3 ? maxD(1.0, fabs((double)M[12 + r])) : 1.0;
            if (c == 3) out.trans = maxD(out.trans, scale);
            const double v = (double)M[0 + r] * W[4 * c + 0] + (double)M[4 + r] * W[4 * c + 1] + (double)M[8 + r] * W[4 * c + 2] + (c == 3 ? (double)M[12 + r] : 0.0);
            if (!(fabs(v - (r == c ? 1.0 : 0.0)) <= 2e-5 * scale)) { out.consistent = false; break; }
        }
    float mlo[3] = {3e38f, 3e38f, 3e38f}, mhi[3] = {-3e38f, -3e38f, -3e38f};
    for (int k = 0; k < 4; ++k) {
        if (!slotUsed(root, k)) continue;
        double lo[3], hi[3];
        decodeChild(root, k, lo, hi);
        for (int a = 0; a < 3; ++a) { mlo[a] = minF(mlo[a], nextafterf((float)lo[a], -3e38f)); mhi[a] = maxF(mhi[a], nextafterf((float)hi[a], 3e38f)); }
    }
    for (int k = 0; k < 3; ++k) { out.lo[k] = 3e38f; out.hi[k] = -3e38f; }
    double ext = 0.0;
    for (int c = 0; c < 8; ++c) {
        const double p[3] = {((c & 1) ? mhi[0] : mlo[0]) - (double)W[12], ((c & 2) ? mhi[1] : mlo[1]) - (double)W[13], ((c & 4) ? mhi[2] : mlo[2]) - (double)W[14]};
        for (int rr = 0; rr < 3; ++rr) {
            const double w = wi[3 * rr] * p[0] + wi[3 * rr + 1] * p[1] + wi[3 * rr + 2] * p[2];
            out.lo[rr] = minF(out.lo[rr], (float)w); out.hi[rr] = maxF(out.hi[rr], (float)w);
            ext = maxD(ext, fabs(w));
        }
    }
    const float pad = (float)(ext * 1e-4 + 1e-3);
    for (int k = 0; k < 3; ++k) { out.lo[k] -= pad; out.hi[k] += pad; }
    double fro = 0.0;
    for (double v : wi) fro += v * v;
    out.scale = sqrt(fro);
    out.pad = (double)pad;
    return true;
}

}  // namespace ptap
