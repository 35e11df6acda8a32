// se3_exact.cuh -- Sophus / Eigen SE3 arithmetic in the reference's operation order, fp64, non-contracted, for the small
// per-entity kernels whose values feed integer decisions (cvRound, cell index, strict comparisons). pose = {qw,qx,qy,qz,t}.
#pragma once

namespace dsdtm {

// Eigen QuaternionBase::_transformVector
__device__ __forceinline__ void qrot_exact(const double* q, double v0, double v1, double v2, double& o0, double& o1, double& o2)
{
    double uv0 = __dsub_rn(__dmul_rn(q[2], v2), __dmul_rn(q[3], v1));
    double uv1 = __dsub_rn(__dmul_rn(q[3], v0), __dmul_rn(q[1], v2));
    double uv2 = __dsub_rn(__dmul_rn(q[1], v1), __dmul_rn(q[2], v0));
    uv0 = __dadd_rn(uv0, uv0); uv1 = __dadd_rn(uv1, uv1); uv2 = __dadd_rn(uv2, uv2);
    const double c0 = __dsub_rn(__dmul_rn(q[2], uv2), __dmul_rn(q[3], uv1));
    const double c1 = __dsub_rn(__dmul_rn(q[3], uv0), __dmul_rn(q[1], uv2));
    const double c2 = __dsub_rn(__dmul_rn(q[1], uv1), __dmul_rn(q[2], uv0));
    o0 = __dadd_rn(__dadd_rn(v0, __dmul_rn(q[0], uv0)), c0);
    o1 = __dadd_rn(__dadd_rn(v1, __dmul_rn(q[0], uv1)), c1);
    o2 = __dadd_rn(__dadd_rn(v2, __dmul_rn(q[0], uv2)), c2);
}

// SE3::inverse(): so3 = conjugate, t = so3 * (t * -1)
__device__ __forceinline__ void se3_inv_exact(const double* p, double* o)
{
    o[0] = p[0]; o[1] = -p[1]; o[2] = -p[2]; o[3] = -p[3];
    qrot_exact(o, __dmul_rn(p[4], -1.0), __dmul_rn(p[5], -1.0), __dmul_rn(p[6], -1.0), o[4], o[5], o[6]);
}

// SE3::operator*: t = t_a + R_a t_b ; q = q_a q_b (Eigen product) ; normalise
__device__ __forceinline__ void se3_mul_exact(const double* A, const double* B, double* o)
{
    double r0, r1, r2;
    qrot_exact(A, B[4], B[5], B[6], r0, r1, r2);
    const double t0 = __dadd_rn(A[4], r0), t1 = __dadd_rn(A[5], r1), t2 = __dadd_rn(A[6], r2);
    const double aw = A[0], ax = A[1], ay = A[2], az = A[3], bw = B[0], bx = B[1], by = B[2], bz = B[3];
    double w = __dsub_rn(__dsub_rn(__dsub_rn(__dmul_rn(aw, bw), __dmul_rn(ax, bx)), __dmul_rn(ay, by)), __dmul_rn(az, bz));
    double x = __dsub_rn(__dadd_rn(__dadd_rn(__dmul_rn(aw, bx), __dmul_rn(ax, bw)), __dmul_rn(ay, bz)), __dmul_rn(az, by));
    double y = __dsub_rn(__dadd_rn(__dadd_rn(__dmul_rn(aw, by), __dmul_rn(ay, bw)), __dmul_rn(az, bx)), __dmul_rn(ax, bz));
    double z = __dsub_rn(__dadd_rn(__dadd_rn(__dmul_rn(aw, bz), __dmul_rn(az, bw)), __dmul_rn(ax, by)), __dmul_rn(ay, bx));
    const double n = sqrt(__dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)), __dmul_rn(z, z)), __dmul_rn(w, w)));
    o[0] = __ddiv_rn(w, n); o[1] = __ddiv_rn(x, n); o[2] = __ddiv_rn(y, n); o[3] = __ddiv_rn(z, n);
    o[4] = t0; o[5] = t1; o[6] = t2;
}

// Feature::mNormal = Pixel2Camera(px, 1.0).normalize(): float evaluation of the camera ray, widened, then normalised in fp64
// (ref: src/Camera.cpp:173-178, src/Frame.cpp:83-92,146-147; Q8)
__device__ __forceinline__ void feature_normal_exact(float ux, float uy, float fx, float fy, float cx, float cy, double* o)
{
    const double n0 = (double)__fdiv_rn(__fmul_rn(1.0f, __fsub_rn(ux, cx)), fx), n1 = (double)__fdiv_rn(__fmul_rn(1.0f, __fsub_rn(uy, cy)), fy), n2 = 1.0;
    const double nn = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(n0, n0), __dmul_rn(n1, n1)), __dmul_rn(n2, n2)));
    o[0] = __ddiv_rn(n0, nn); o[1] = __ddiv_rn(n1, nn); o[2] = __ddiv_rn(n2, nn);
}

}  // namespace dsdtm
