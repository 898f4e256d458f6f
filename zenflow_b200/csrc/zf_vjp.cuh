// VJP of normalize_spline_params + rational_quadratic_spline_forward (utils.py:37-141) and of the analytic inverse
// (utils.py:144-202) for one (event, dim) row: shared by the stage-style kernel of zf_train.cu (theta from HBM) and the
// fused conditioner-recompute kernel of zf_chain.cu (theta from tensor memory).  Derivation: SURVEY.md Appendix A.
#pragma once
#include "zf_math.cuh"

namespace zf {

__device__ __forceinline__ float squareplus_grad(float a) {  // d/da 0.5*(a + sqrt(a^2+4))
    return 0.5f * (1.0f + a * rsqrtf(a * a + 4.0f));
}

// Adjoints of the gathered bin quantities (Appendix A): x -> (y, log|dy/dx|) inside bin [xk, xk + w) x [yk, yk + h)
// with knot derivatives d0, d1; gy, gld are the cotangents of y and of the log-det.
__device__ __forceinline__ void rqs_scalar_adjoints(float x, float gy, float gld, float xk, float w, float h, float d0, float d1,
                                                    float& g_x, float& g_xk, float& g_w, float& g_yk, float& g_h, float& g_d0,
                                                    float& g_d1) {
    const float s = h / w;
    const float xi_raw = (x - xk) / w;
    const bool clipped = !(xi_raw > kEps && xi_raw < kOneMinusEps);
    const float xi = fminf(fmaxf(xi_raw, kEps), kOneMinusEps);
    const float az = 1.0f - xi;
    const float beta = d1 + d0 - 2.0f * s;
    const float u = s * xi + d0 * az;
    const float num = h * xi * u;
    const float den = s + beta * xi * az;
    const float Dn = den + kEps;
    const float v = d1 * xi + 2.0f * s * az;
    const float num2 = xi * v + d0 * az * az;

    // adjoints (Appendix A)
    g_yk = gy;
    const float g_num = gy / Dn;
    const float g_den = -gy * num / (Dn * Dn) - 2.0f * gld / Dn;
    const float g_num2 = gld / (num2 + kEps);
    float g_s = gld * 2.0f / (s + kEps);
    g_h = g_num * xi * u;
    float g_xi = g_num * h * u;
    const float g_u = g_num * h * xi;
    g_s += g_u * xi;
    g_xi += g_u * s;
    g_d0 = g_u * az;
    float g_az = g_u * d0;
    g_s += g_den;
    const float g_beta = g_den * xi * az;
    g_xi += g_den * beta * az;
    g_az += g_den * beta * xi;
    g_d1 = g_beta;
    g_d0 += g_beta;
    g_s -= 2.0f * g_beta;
    g_xi += g_num2 * v;
    const float g_v = g_num2 * xi;
    g_d0 += g_num2 * az * az;
    g_az += g_num2 * d0 * 2.0f * az;
    g_d1 += g_v * xi;
    g_xi += g_v * d1;
    g_s += g_v * 2.0f * az;
    g_az += g_v * 2.0f * s;
    g_xi -= g_az;
    const float g_xr = clipped ? 0.f : g_xi;
    g_x = g_xr / w;
    g_xk = -g_xr / w;
    g_w = -g_xr * xi_raw / w;
    g_h += g_s / w;
    g_w -= g_s * s / w;
}

// Cotangent of raw theta from the cotangents of what one bin gathers (normalize_spline_params, utils.py:37-62): the
// widths block gets g_xk (knots left of the bin) and g_w (the bin), the heights block g_yk and g_h, the slopes g_d0 and
// g_d1 at the bin's two inner knots.  idx < K is the bin.  row: raw theta (3K-1) in, its cotangent out.
template <int KT>
__device__ __forceinline__ void rqs_theta_adjoints(float* row, int K_rt, int idx, const KnotNorm& kn, float g_xk, float g_w,
                                                   float g_yk, float g_h, float g_d0, float g_d1) {
    const int K = KT > 0 ? KT : K_rt;
    // slopes first (their raw values are needed before the row is overwritten)
    const float c_lo = (idx >= 1) ? row[2 * K + idx - 1] : 0.f;
    const float c_hi = (idx + 1 <= K - 1) ? row[2 * K + idx] : 0.f;

    // widths / heights: W_j = kappa*(s_j/S + c); cotangent of W_j is g_lt (j<idx), g_at (j==idx), 0 otherwise
    const float kappa = kn.rden;
#pragma unroll
    for (int blk = 0; blk < 2; ++blk) {
        float* pr = row + blk * K;
        const float g_lt = blk == 0 ? g_xk : g_yk;
        const float g_at = blk == 0 ? g_w : g_h;
        float S = 0.f, Slt = 0.f, s_at = 0.f;
        constexpr int KS = KT > 0 ? KT : 1;
        if (KT > 0) {
#pragma unroll
            for (int j = 0; j < KS; ++j) {
                const float aj = pr[j];
                const float sj = 0.5f * (aj + sqrtf(fmaf(aj, aj, 4.0f)));   // fp32-tolerance path: plain sqrt
                S += sj;
                Slt += (j < idx) ? sj : 0.f;
                s_at = (j == idx) ? sj : s_at;
            }
        } else {
            for (int j = 0; j < K; ++j) {
                const float sj = squareplus_rn(pr[j]);
                S += sj;
                if (j < idx) Slt += sj;
                if (j == idx) s_at = sj;
            }
        }
        const float A = (g_lt * Slt + g_at * s_at) / S;
        const float ks = kappa / S;
        if (KT > 0) {
#pragma unroll
            for (int j = 0; j < KS; ++j) {
                const float a = pr[j];
                const float gW = (j < idx) ? g_lt : ((j == idx) ? g_at : 0.f);
                // d squareplus/da = 0.5*(1 + a/sqrt(a^2+4)) = s/(2s - a) ... use the rsqrt form
                pr[j] = ks * (gW - A) * squareplus_grad(a);
            }
        } else {
            for (int j = 0; j < K; ++j) {
                const float a = pr[j];
                const float gW = (j < idx) ? g_lt : ((j == idx) ? g_at : 0.f);
                pr[j] = ks * (gW - A) * squareplus_grad(a);
            }
        }
    }
    for (int j = 0; j < K - 1; ++j) row[2 * K + j] = 0.f;
    if (idx >= 1) row[2 * K + idx - 1] = g_d0 * squareplus_grad(c_lo);
    if (idx + 1 <= K - 1) row[2 * K + idx] = g_d1 * squareplus_grad(c_hi);
}

// row: raw theta (3K-1) in shared memory, overwritten by its cotangent.  Returns d/dx.
// KT > 0: K known at compile time (loops unrolled); KT == 0: runtime K.
template <int KT>
__device__ __forceinline__ float rqs_row_backward(float* row, int K_rt, float x, float gy, float gld, const KnotNorm& kn) {
    const int K = KT > 0 ? KT : K_rt;
    RqsBin b;
    rqs_locate<KT>(row, K, true, x, kn, b);
    const int P = 3 * K - 1;
    const bool oob = (x < 0.f) || (x >= 1.f);
    const int idx = b.idx;
    if (oob || idx >= K || !(x == x)) {  // identity branch (or the reference's NaN corner): no parameter gradient
        for (int p = 0; p < P; ++p) row[p] = 0.f;
        return oob ? gy : 0.f;
    }
    const float xk = b.ks, w = b.bs, h = b.bo, d0 = b.dk, d1 = b.dkp1;
    float g_x, g_xk, g_w, g_yk, g_h, g_d0, g_d1;
    rqs_scalar_adjoints(x, gy, gld, xk, w, h, d0, d1, g_x, g_xk, g_w, g_yk, g_h, g_d0, g_d1);
    rqs_theta_adjoints<KT>(row, K, idx, kn, g_xk, g_w, g_yk, g_h, g_d0, g_d1);
    return g_x;
}

// Adjoints of the analytic inverse (utils.py:191-201, rqs_eval_inverse): y -> x inside bin [yk, yk + h) x [xk, xk + w)
// with knot derivatives d0, d1; gx is the cotangent of x.  The formula is differentiated as written (a quadratic root,
// no EPS, no clip), which is what jax.grad of the reference's inverse gives; it is not 1 / (dy/dx) of the forward.
// LD: gld is the cotangent of the inverse's log|dx/dy| = 2 log(den) - 2 log(s) - log(num2) at the root
// (rqs_inverse_log_det), its terms formed only where gld != 0 (no 0 * inf); without LD gld is not read and the code is
// that of the inverse's VJP alone.
template <bool LD = false>
__device__ __forceinline__ void rqs_scalar_inverse_adjoints(float y, float gx, float gld, float yk, float h, float xk, float w,
                                                            float d0, float d1, float& g_y, float& g_yk, float& g_h, float& g_xk,
                                                            float& g_w, float& g_d0, float& g_d1) {
    const float s = h / w;
    const float dy = y - yk;
    const float beta = d1 + d0 - 2.0f * s;
    const float a = h * (s - d0) + dy * beta;
    const float bq = h * d0 - dy * beta;
    const float c = -s * dy;
    const float sq = sqrtf(bq * bq - 4.0f * a * c);
    const float Dq = -bq - sq;
    const float z = 2.0f * c / Dq;
    // x = z w + xk,  z = 2c / Dq,  Dq = -bq - sqrt(bq^2 - 4ac)
    g_xk = gx;
    g_w = gx * z;
    float g_z = gx * w;
    // log-det: den = s + beta z (1 - z), num2 = d1 z^2 + 2 s z (1 - z) + d0 (1 - z)^2, differentiated at fixed z here and
    // through the root (g_z) below
    float gl_s = 0.f, gl_d0 = 0.f, gl_d1 = 0.f;
    const bool with_ld = LD && gld != 0.f;
    if (with_ld) {
        const float az = 1.0f - z, zz = z * az;
        const float den = s + beta * zz;
        const float num2 = z * (d1 * z + 2.0f * s * az) + d0 * (az * az);
        const float g_den = 2.0f * gld / den, g_num2 = -gld / num2;
        const float gl_beta = g_den * zz;
        g_z += g_den * beta * (1.0f - 2.0f * z) + g_num2 * 2.0f * (d1 * z + s * (1.0f - 2.0f * z) - d0 * az);
        gl_s = g_den - 2.0f * gld / s + g_num2 * 2.0f * zz - 2.0f * gl_beta;
        gl_d0 = g_num2 * az * az + gl_beta;
        gl_d1 = g_num2 * z * z + gl_beta;
    }
    float g_c = g_z * 2.0f / Dq;
    const float g_Dq = -g_z * z / Dq;
    const float g_disc = -g_Dq * 0.5f / sq;
    const float g_bq = -g_Dq + g_disc * 2.0f * bq;
    const float g_a = -g_disc * 4.0f * c;
    g_c -= g_disc * 4.0f * a;
    // c = -s dy;  bq = h d0 - dy beta;  a = h (s - d0) + dy beta;  beta = d1 + d0 - 2 s
    float g_s = -g_c * dy;
    float g_dy = -g_c * s;
    g_h = g_bq * d0 + g_a * (s - d0);
    g_d0 = g_bq * h - g_a * h;
    g_dy += (g_a - g_bq) * beta;
    const float g_beta = (g_a - g_bq) * dy;
    g_s += g_a * h;
    g_d1 = g_beta;
    g_d0 += g_beta;
    g_s -= 2.0f * g_beta;
    if (with_ld) {
        g_s += gl_s;
        g_d0 += gl_d0;
        g_d1 += gl_d1;
    }
    // dy = y - yk;  s = h / w
    g_y = g_dy;
    g_yk = -g_dy;
    g_h += g_s / w;
    g_w -= g_s * s / w;
}

// The VJP of normalize_spline_params + rational_quadratic_spline_inverse (utils.py:144-202) on a row: raw theta (3K-1)
// in shared memory, overwritten by its cotangent; gx is the cotangent of x, gld (read only with LD) that of the row's
// log|dx/dy|.  Returns d/dy.  The bin is searched in the heights, as the eval inverse searches it.  Conventions as
// rqs_row_backward: identity branch (y outside [0, 1)): d/dy = gx and no parameter gradient (the log-det is 0 there); the
// reference's NaN corner (past the last knot, NaN input): zero gradients.
template <int KT, bool LD = false>
__device__ __forceinline__ float rqs_row_inverse_backward(float* row, int K_rt, float y, float gx, float gld, const KnotNorm& kn) {
    const int K = KT > 0 ? KT : K_rt;
    RqsBin b;
    rqs_locate<KT>(row, K, false, y, kn, b);
    const int P = 3 * K - 1;
    const bool oob = (y < 0.f) || (y >= 1.f);
    const int idx = b.idx;
    if (oob || idx >= K || !(y == y)) {
        for (int p = 0; p < P; ++p) row[p] = 0.f;
        return oob ? gx : 0.f;
    }
    const float yk = b.ks, h = b.bs, xk = b.ko, w = b.bo, d0 = b.dk, d1 = b.dkp1;
    float g_y, g_yk, g_h, g_xk, g_w, g_d0, g_d1;
    rqs_scalar_inverse_adjoints<LD>(y, gx, gld, yk, h, xk, w, d0, d1, g_y, g_yk, g_h, g_xk, g_w, g_d0, g_d1);
    rqs_theta_adjoints<KT>(row, K, idx, kn, g_xk, g_w, g_yk, g_h, g_d0, g_d1);
    return g_y;
}

// The same VJP with theta in registers (the fused conditioner-recompute kernel reads it from tensor memory) and the
// fast forms: pa = raw widths, pb = raw heights (both overwritten), the finished slope block in row[0, KT-1).
// Valid for |theta| < kThetaFastBound-class inputs (the caller checks and takes rqs_row_backward otherwise).
// The bin search is rqs_block_search_lean's (bit-identical bins); squareplus values are kept doubled
// (s2 = a + sqrt(a^2 + 4)) and d squareplus / d a = s^2 / (s^2 + 1) = s2^2 / (s2^2 + 4) needs no second square root.
// Writes the cotangent of theta to row[0, 3 KT - 1) and returns d/dx.
template <int KT>
__device__ __forceinline__ float rqs_row_vjp_regs(float (&pa)[KT], float (&pb)[KT], float* row, float x, float gy, float gld,
                                                  const KnotNorm& kn) {
    // ---- searched axis (widths): exact, doubled
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < KT; ++j) {
        pa[j] = __fadd_rn(pa[j], sqrt_rn_normal(__fadd_rn(__fmul_rn(pa[j], pa[j]), 4.0f)));
        sum = j == 0 ? pa[0] : __fadd_rn(sum, pa[j]);
    }
    const float rsum = __frcp_rn(sum);
    float acc = 0.f, xk = 0.f, w = 0.f, run = 0.f, slt_w = 0.f, sat_w = 0.f;
    int idx = 0;
#pragma unroll
    for (int j = 0; j < KT; ++j) {
        const float q = div_rn_recip(pa[j], sum, rsum);
        const float wj = div_rn_recip(__fadd_rn(q, kn.c), kn.den, kn.rden);
        const bool in = (j == 0) || (acc <= x);
        xk = in ? acc : xk;
        w = in ? wj : w;
        idx = in ? j : idx;
        slt_w = in ? run : slt_w;       // sum of the doubled squareplus values left of the bin
        sat_w = in ? pa[j] : sat_w;
        run += pa[j];
        acc = __fadd_rn(acc, wj);
    }
    if (acc <= x) idx = KT;
    const bool oob = (x < 0.f) || (x >= 1.f);
    const bool dead = oob || idx >= KT || !(x == x);   // identity branch / the reference's NaN corner: no parameter gradient
    const int ib = dead ? 0 : idx;
    // ---- other axis (heights): SFU square root, doubled
    float sum_h = 0.f, slt_h = 0.f, sat_h = 1.f;
#pragma unroll
    for (int j = 0; j < KT; ++j) {
        pb[j] = squareplus2_sfu(pb[j]);
        slt_h = (j == ib) ? sum_h : slt_h;
        sat_h = (j == ib) ? pb[j] : sat_h;
        sum_h = j == 0 ? pb[0] : sum_h + pb[j];
    }
    const float rsum_h = __frcp_rn(sum_h);
    const float h = (sat_h * rsum_h + kn.c) * kn.rden;
    // ---- knot derivatives
    const float c_lo = (ib >= 1) ? row[ib - 1] : 0.f;
    const float c_hi = (ib + 1 <= KT - 1) ? row[ib] : 0.f;
    const float d0 = (ib >= 1) ? squareplus_rn(c_lo) : 1.0f;
    const float d1 = (ib + 1 <= KT - 1) ? squareplus_rn(c_hi) : 1.0f;
    float g_x, g_xk, g_w, g_yk, g_h, g_d0, g_d1;
    rqs_scalar_adjoints(x, gy, gld, xk, w, h, d0, d1, g_x, g_xk, g_w, g_yk, g_h, g_d0, g_d1);
    if (dead) { g_xk = g_w = g_yk = g_h = g_d0 = g_d1 = 0.f; g_x = oob ? gy : 0.f; }
    // ---- widths / heights: W_j = kappa (s_j / S + c); the cotangent of W_j is g_lt (j < idx), g_at (j == idx), else 0
    {
        const float A = (g_xk * slt_w + g_w * sat_w) * rsum;
        const float ks = 2.0f * kn.rden * rsum;
        const float c1 = ks * (g_xk - A), c2 = ks * (g_w - A), c3 = -ks * A;
#pragma unroll
        for (int j = 0; j < KT; ++j) {
            const float q = pa[j] * pa[j];
            float r;
            asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(q + 4.0f));
            row[j] = ((j < ib) ? c1 : ((j == ib) ? c2 : c3)) * (q * r);
        }
    }
    {
        const float A = (g_yk * slt_h + g_h * sat_h) * rsum_h;
        const float ks = 2.0f * kn.rden * rsum_h;
        const float c1 = ks * (g_yk - A), c2 = ks * (g_h - A), c3 = -ks * A;
#pragma unroll
        for (int j = 0; j < KT; ++j) {
            const float q = pb[j] * pb[j];
            float r;
            asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(q + 4.0f));
            row[KT + j] = ((j < ib) ? c1 : ((j == ib) ? c2 : c3)) * (q * r);
        }
    }
#pragma unroll
    for (int j = 0; j < KT - 1; ++j) row[2 * KT + j] = 0.f;
    if (ib >= 1) row[2 * KT + ib - 1] = g_d0 * squareplus_grad(c_lo);
    if (ib + 1 <= KT - 1) row[2 * KT + ib] = g_d1 * squareplus_grad(c_hi);
    return g_x;
}

}  // namespace zf
