/*
 * antialiasing_oracle.c -- CPU reference of the antialiasing opacity factor and of the preprocess backward of an
 * antialiased forward (test infrastructure only; loaded by tests/antialiasing_oracle.py).
 *
 * With (a0, b, c0) the projected 2D covariance before the 0.3 px^2 dilation and (a, b, c) = (a0 + 0.3, b, c0 + 0.3):
 *     rho = sqrt(max(2.5e-5, (a0 c0 - b^2) / (a c - b^2))),   record opacity = opacity * rho
 *
 * aa_rho: rho on oracle/raster_oracle.c's fp32 projection chain, statement for statement (compiled the same way:
 * -ffp-contract=off, no fast-math), so it is the factor the kernels' pinned-rounding chain must reproduce bit for bit.
 * It also writes the conic, which tests/test_oracle_antialiasing.py holds bitwise to oracle.raster.preprocess's: that
 * pins this chain to the colour oracle's.
 *
 * aa_preprocess_bwd: oracle/raster_oracle.c's per-Gaussian backward (fp64 inside, fp32 in and out), statement for
 * statement, plus the rho term: dL_dopacity_out = dL_dopacity_in * rho, and where det0 / det > 2.5e-5
 * dL/drho = dL_dopacity_in * opacity is added to dL/d(a, b, c) with the exact derivative of det0 / det.  With
 * antialiasing = 0 it must equal oracle.raster.preprocess_bwd byte for byte (and copies dL_dopacity_in).
 *
 * Why a separate file next to the tests rather than new entry points in oracle/raster_oracle.c: the colour oracle is
 * the fixed reference of the plain path, which this feature leaves unchanged, so it is not touched either.
 */
#include <math.h>
#include <stdint.h>
#include <string.h>

/* oracle/raster_oracle.c project_one up to the dilated covariance; returns 0 where it culls before det */
static int cov2d(const float *p, const float *sc, const float *q, float mod, const float *view, float tanfovx,
                 float tanfovy, float focal_x, float focal_y, float *a0_, float *b_, float *c0_) {
    const float x = p[0], y = p[1], z = p[2];
    const float vx = ((view[0] * x + view[4] * y) + view[8] * z) + view[12];
    const float vy = ((view[1] * x + view[5] * y) + view[9] * z) + view[13];
    const float vz = ((view[2] * x + view[6] * y) + view[10] * z) + view[14];
    if (vz <= 0.2f) return 0;
    const float s0 = mod * sc[0], s1 = mod * sc[1], s2 = mod * sc[2];
    const float qr = q[0], qx = q[1], qy = q[2], qz = q[3];
    float R[3][3];
    R[0][0] = 1.0f - 2.0f * (qy * qy + qz * qz);
    R[0][1] = 2.0f * (qx * qy - qr * qz);
    R[0][2] = 2.0f * (qx * qz + qr * qy);
    R[1][0] = 2.0f * (qx * qy + qr * qz);
    R[1][1] = 1.0f - 2.0f * (qx * qx + qz * qz);
    R[1][2] = 2.0f * (qy * qz - qr * qx);
    R[2][0] = 2.0f * (qx * qz - qr * qy);
    R[2][1] = 2.0f * (qy * qz + qr * qx);
    R[2][2] = 1.0f - 2.0f * (qx * qx + qy * qy);
    float M[3][3];
    for (int i = 0; i < 3; ++i) { M[i][0] = R[i][0] * s0; M[i][1] = R[i][1] * s1; M[i][2] = R[i][2] * s2; }
    float S[3][3];
    for (int i = 0; i < 3; ++i)
        for (int j = i; j < 3; ++j) {
            S[i][j] = (M[i][0] * M[j][0] + M[i][1] * M[j][1]) + M[i][2] * M[j][2];
            S[j][i] = S[i][j];
        }
    const float limx = 1.3f * tanfovx, limy = 1.3f * tanfovy;
    const float txtz = vx / vz, tytz = vy / vz;
    const float tx = fminf(limx, fmaxf(-limx, txtz)) * vz;
    const float ty = fminf(limy, fmaxf(-limy, tytz)) * vz;
    const float J00 = focal_x / vz;
    const float J02 = -(focal_x * tx) / (vz * vz);
    const float J11 = focal_y / vz;
    const float J12 = -(focal_y * ty) / (vz * vz);
    float A0[3], A1[3];
    for (int k = 0; k < 3; ++k) {
        const float r0 = view[4 * k + 0], r1 = view[4 * k + 1], r2 = view[4 * k + 2];
        A0[k] = J00 * r0 + J02 * r2;
        A1[k] = J11 * r1 + J12 * r2;
    }
    float B0[3], B1[3];
    for (int l = 0; l < 3; ++l) {
        B0[l] = (A0[0] * S[0][l] + A0[1] * S[1][l]) + A0[2] * S[2][l];
        B1[l] = (A1[0] * S[0][l] + A1[1] * S[1][l]) + A1[2] * S[2][l];
    }
    *a0_ = (B0[0] * A0[0] + B0[1] * A0[1]) + B0[2] * A0[2];
    *b_ = (B0[0] * A1[0] + B0[1] * A1[1]) + B0[2] * A1[2];
    *c0_ = (B1[0] * A1[0] + B1[1] * A1[1]) + B1[2] * A1[2];
    return 1;
}

/* rho[P] and conic[3P] of the Gaussians with radii > 0 (0 elsewhere) */
int aa_rho(int P, const float *means3D, const float *scales, int scale_stride, const float *rots, float scale_mod,
           const float *view, float tanfovx, float tanfovy, int H, int W, const int32_t *radii, float *rho,
           float *conic) {
    const float fx = (float)W / (2.0f * tanfovx), fy = (float)H / (2.0f * tanfovy);
    for (int i = 0; i < P; ++i) {
        rho[i] = 0.0f; conic[3 * (size_t)i] = conic[3 * (size_t)i + 1] = conic[3 * (size_t)i + 2] = 0.0f;
        float a0, b, c0;
        if (!(radii[i] > 0)) continue;
        if (!cov2d(means3D + 3 * (size_t)i, scales + (size_t)scale_stride * i, rots + 4 * (size_t)i, scale_mod, view,
                   tanfovx, tanfovy, fx, fy, &a0, &b, &c0)) return -1;
        const float a = a0 + 0.3f, c = c0 + 0.3f;
        const float det = a * c - b * b;
        if (det == 0.0f) return -1;
        const float det_inv = 1.0f / det;
        conic[3 * (size_t)i] = c * det_inv; conic[3 * (size_t)i + 1] = -b * det_inv; conic[3 * (size_t)i + 2] = a * det_inv;
        rho[i] = sqrtf(fmaxf(2.5e-5f, (a0 * c0 - b * b) / det));
    }
    return 0;
}

int aa_preprocess_bwd(int P, const float *means3D, const float *scales, int scale_stride, const float *rots,
                      float scale_mod, const float *view, const float *proj, float tanfovx, float tanfovy, int H, int W,
                      const int32_t *radii, const float *dL_dmean2D, const float *dL_dconic, float *dL_dmeans3D,
                      float *dL_dscales, float *dL_drots, const float *opacities, const float *dL_dopacity_in,
                      float *dL_dopacity_out, int antialiasing)
{
    const float fx = (float)W / (2.0f * tanfovx), fy = (float)H / (2.0f * tanfovy);
    for (int i = 0; i < P; ++i) {
        float *gm = dL_dmeans3D + 3 * (size_t)i, *gs = dL_dscales + 3 * (size_t)i, *gq = dL_drots + 4 * (size_t)i;
        gm[0] = gm[1] = gm[2] = 0.f; gs[0] = gs[1] = gs[2] = 0.f; gq[0] = gq[1] = gq[2] = gq[3] = 0.f;
        dL_dopacity_out[i] = dL_dopacity_in[i];
        if (!(radii[i] > 0)) continue;
        const float *p = means3D + 3 * (size_t)i, *sc = scales + (size_t)scale_stride * i, *q = rots + 4 * (size_t)i;
        const double x = p[0], y = p[1], z = p[2];
        double Rot[3][3], tr[3];
        for (int r = 0; r < 3; ++r) { for (int k = 0; k < 3; ++k) Rot[r][k] = view[4 * k + r]; tr[r] = view[12 + r]; }
        const double vx = Rot[0][0] * x + Rot[0][1] * y + Rot[0][2] * z + tr[0];
        const double vy = Rot[1][0] * x + Rot[1][1] * y + Rot[1][2] * z + tr[1];
        const double vz = Rot[2][0] * x + Rot[2][1] * y + Rot[2][2] * z + tr[2];
        const double s[3] = { (double)scale_mod * sc[0], (double)scale_mod * sc[1], (double)scale_mod * sc[2] };
        const double qr = q[0], qx = q[1], qy = q[2], qz = q[3];
        double R[3][3] = {
            { 1 - 2 * (qy * qy + qz * qz), 2 * (qx * qy - qr * qz), 2 * (qx * qz + qr * qy) },
            { 2 * (qx * qy + qr * qz), 1 - 2 * (qx * qx + qz * qz), 2 * (qy * qz - qr * qx) },
            { 2 * (qx * qz - qr * qy), 2 * (qy * qz + qr * qx), 1 - 2 * (qx * qx + qy * qy) } };
        double M[3][3], S[3][3];
        for (int a = 0; a < 3; ++a) for (int k = 0; k < 3; ++k) M[a][k] = R[a][k] * s[k];
        for (int a = 0; a < 3; ++a) for (int b = 0; b < 3; ++b) S[a][b] = M[a][0] * M[b][0] + M[a][1] * M[b][1] + M[a][2] * M[b][2];
        const double limx = 1.3 * (double)tanfovx, limy = 1.3 * (double)tanfovy;
        const double txtz = vx / vz, tytz = vy / vz;
        const int clx = (txtz < -limx || txtz > limx), cly = (tytz < -limy || tytz > limy);
        const double tx = fmin(limx, fmax(-limx, txtz)) * vz, ty = fmin(limy, fmax(-limy, tytz)) * vz;
        const double J00 = fx / vz, J02 = -(fx * tx) / (vz * vz), J11 = fy / vz, J12 = -(fy * ty) / (vz * vz);
        double A[2][3];
        for (int k = 0; k < 3; ++k) { A[0][k] = J00 * Rot[0][k] + J02 * Rot[2][k]; A[1][k] = J11 * Rot[1][k] + J12 * Rot[2][k]; }
        double B[2][3];
        for (int r = 0; r < 2; ++r) for (int l = 0; l < 3; ++l) B[r][l] = A[r][0] * S[0][l] + A[r][1] * S[1][l] + A[r][2] * S[2][l];
        const double a = B[0][0] * A[0][0] + B[0][1] * A[0][1] + B[0][2] * A[0][2] + 0.3;
        const double b = B[0][0] * A[1][0] + B[0][1] * A[1][1] + B[0][2] * A[1][2];
        const double c = B[1][0] * A[1][0] + B[1][1] * A[1][1] + B[1][2] * A[1][2] + 0.3;
        const double denom = a * c - b * b;
        const double d2inv = 1.0 / (denom * denom + 0.0000001);
        const double gc0 = dL_dconic[3 * (size_t)i], gc1 = dL_dconic[3 * (size_t)i + 1], gc2 = dL_dconic[3 * (size_t)i + 2];
        double dL_da = d2inv * (-c * c * gc0 + 2 * b * c * gc1 + (denom - a * c) * gc2);
        double dL_dc = d2inv * (-a * a * gc2 + 2 * a * b * gc1 + (denom - a * c) * gc0);
        double dL_db = d2inv * 2 * (b * c * gc0 - (denom + 2 * b * b) * gc1 + a * b * gc2);
        if (antialiasing) {
            /* rho scales the opacity: dL/dopacity = dL/do' rho, and where the clamp is inactive dL/drho = dL/do' opacity
             * reaches (a, b, c) through d(det0 / det) */
            const double a0 = B[0][0] * A[0][0] + B[0][1] * A[0][1] + B[0][2] * A[0][2];
            const double c0 = B[1][0] * A[1][0] + B[1][1] * A[1][1] + B[1][2] * A[1][2];
            const double det0 = a0 * c0 - b * b, ratio = det0 / denom;
            const double rho = sqrt(fmax(2.5e-5, ratio));
            const double g = dL_dopacity_in[i];
            dL_dopacity_out[i] = (float)(g * rho);
            if (ratio > 2.5e-5) {
                const double k = g * (double)opacities[i] / (2 * rho * denom * denom);
                dL_da += k * (c0 * denom - det0 * c);
                dL_dc += k * (a0 * denom - det0 * a);
                dL_db += 2 * k * b * (det0 - denom);
            }
        }
        const double G2[2][2] = { { dL_da, 0.5 * dL_db }, { 0.5 * dL_db, dL_dc } };
        double dS[3][3], dA[2][3];
        for (int k = 0; k < 3; ++k) for (int l = 0; l < 3; ++l) {
            double v = 0; for (int r = 0; r < 2; ++r) for (int t = 0; t < 2; ++t) v += A[r][k] * G2[r][t] * A[t][l];
            dS[k][l] = v;
        }
        for (int r = 0; r < 2; ++r) for (int l = 0; l < 3; ++l) dA[r][l] = 2 * (G2[r][0] * B[0][l] + G2[r][1] * B[1][l]);
        double dJ00 = 0, dJ02 = 0, dJ11 = 0, dJ12 = 0;
        for (int k = 0; k < 3; ++k) { dJ00 += dA[0][k] * Rot[0][k]; dJ02 += dA[0][k] * Rot[2][k]; dJ11 += dA[1][k] * Rot[1][k]; dJ12 += dA[1][k] * Rot[2][k]; }
        const double iz = 1.0 / vz, iz2 = iz * iz, iz3 = iz2 * iz;
        const double dtx = clx ? 0.0 : -fx * iz2 * dJ02;
        const double dty = cly ? 0.0 : -fy * iz2 * dJ12;
        const double dtz = -fx * iz2 * dJ00 - fy * iz2 * dJ11 + 2 * fx * tx * iz3 * dJ02 + 2 * fy * ty * iz3 * dJ12;
        double gmx = Rot[0][0] * dtx + Rot[1][0] * dty + Rot[2][0] * dtz;
        double gmy = Rot[0][1] * dtx + Rot[1][1] * dty + Rot[2][1] * dtz;
        double gmz = Rot[0][2] * dtx + Rot[1][2] * dty + Rot[2][2] * dtz;
        const double hx = proj[0] * x + proj[4] * y + proj[8] * z + proj[12];
        const double hy = proj[1] * x + proj[5] * y + proj[9] * z + proj[13];
        const double hw = proj[3] * x + proj[7] * y + proj[11] * z + proj[15];
        const double mw = 1.0 / (hw + 0.0000001);
        const double mul1 = hx * mw * mw, mul2 = hy * mw * mw;
        const double g2x = dL_dmean2D[3 * (size_t)i], g2y = dL_dmean2D[3 * (size_t)i + 1];
        gmx += (proj[0] * mw - proj[3] * mul1) * g2x + (proj[1] * mw - proj[3] * mul2) * g2y;
        gmy += (proj[4] * mw - proj[7] * mul1) * g2x + (proj[5] * mw - proj[7] * mul2) * g2y;
        gmz += (proj[8] * mw - proj[11] * mul1) * g2x + (proj[9] * mw - proj[11] * mul2) * g2y;
        gm[0] = (float)gmx; gm[1] = (float)gmy; gm[2] = (float)gmz;
        double dM[3][3];
        for (int a2 = 0; a2 < 3; ++a2) for (int k = 0; k < 3; ++k) dM[a2][k] = 2 * (dS[a2][0] * M[0][k] + dS[a2][1] * M[1][k] + dS[a2][2] * M[2][k]);
        double dR[3][3];
        for (int k = 0; k < 3; ++k) {
            double v = 0; for (int a2 = 0; a2 < 3; ++a2) { v += dM[a2][k] * R[a2][k]; dR[a2][k] = dM[a2][k] * s[k]; }
            gs[k] = (float)(v * (double)scale_mod);
        }
        const double dqr = 2 * (-qz * dR[0][1] + qy * dR[0][2] + qz * dR[1][0] - qx * dR[1][2] - qy * dR[2][0] + qx * dR[2][1]);
        const double dqx = 2 * (qy * dR[0][1] + qz * dR[0][2] + qy * dR[1][0] - 2 * qx * dR[1][1] - qr * dR[1][2] + qz * dR[2][0] + qr * dR[2][1] - 2 * qx * dR[2][2]);
        const double dqy = 2 * (-2 * qy * dR[0][0] + qx * dR[0][1] + qr * dR[0][2] + qx * dR[1][0] + qz * dR[1][2] - qr * dR[2][0] + qz * dR[2][1] - 2 * qy * dR[2][2]);
        const double dqz = 2 * (-2 * qz * dR[0][0] - qr * dR[0][1] + qx * dR[0][2] + qr * dR[1][0] - 2 * qz * dR[1][1] + qy * dR[1][2] + qx * dR[2][0] + qy * dR[2][1]);
        gq[0] = (float)dqr; gq[1] = (float)dqx; gq[2] = (float)dqy; gq[3] = (float)dqz;
    }
    return 0;
}
