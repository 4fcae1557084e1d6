/*
 * descriptor_oracle.c -- CPU ORACLE for the descriptor stage of processRIFT (src/comparator.cpp:590-684) and the SIFT keypoints
 * of processSift (src/comparator.cpp:435-469).
 *
 * THIS FILE IS TEST INFRASTRUCTURE, a sibling of oracle/pcc_oracle.c: a plain-C restatement of
 *   pcl::IntensityGradientEstimation::computeFeature  (src/comparator.cpp:649-656, r = 0.03)
 *   pcl::RIFTEstimation::computeFeature                (src/comparator.cpp:659-673, r = 0.05, 4 x 8 bins)
 *   pcl::SIFTKeypoint scale space and extrema          (src/comparator.cpp:449-465)
 * over neighbour rows the caller supplies (CSR, sorted by (fp32 d2, original index), as oracle.KdTree.radius
 * returns them).  Nothing under pointcloudcomparator_b200/ may import, link or call it.
 *
 * Every operation is a correctly rounded fp32 + - * / sqrt in the order DESIGN.md section 2 records
 * ("Upstream details that cannot be verified here").  The libm calls are acosf (RIFT) and powf (SIFT's scale table, as PCL
 * calls it); SIFT's expf is restated in fp64 (sift_expf1), bit for bit the device sift_expf.
 * Build: descriptor_oracle/Makefile (gcc -O3 -ffp-contract=off -fno-fast-math).
 */
#include <float.h>
#include <math.h>
#include <stdint.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define ORC_API __attribute__((visibility("default")))

/* Eigen's completely unrolled reduction of a fixed-size 3-vector: a0 + (a1 + a2) */
static inline float sum3(float a0, float a1, float a2) { return a0 + (a1 + a2); }

/* ------------------------------------------------------------------------------------------ */
/* Eigen 3.3 ColPivHouseholderQR<Matrix3f>::compute + solve, real fp32, column-major a[r + 3c]   */
ORC_API void orc_colpiv_qr_solve3(const float *A_in, const float *b, float *x) {
    float a[9];
    memcpy(a, A_in, sizeof a);
    float hc[3], nu[3], nd[3];
    int perm[3] = {0, 1, 2};
    for (int k = 0; k < 3; ++k) {                         /* m_qr.col(k).norm(): fixed size 3 */
        nd[k] = sqrtf(sum3(a[3 * k] * a[3 * k], a[3 * k + 1] * a[3 * k + 1], a[3 * k + 2] * a[3 * k + 2]));
        nu[k] = nd[k];
    }
    float mx = nu[0];
    if (nu[1] > mx) mx = nu[1];
    if (nu[2] > mx) mx = nu[2];
    const float eps = FLT_EPSILON;
    const float te = mx * eps;
    const float threshold_helper = (te * te) / 3.0f;
    const float norm_downdate_threshold = sqrtf(eps);
    int np = 3;
    for (int k = 0; k < 3; ++k) {
        int bi = k;                                       /* maxCoeff: first index of the largest */
        for (int j = k + 1; j < 3; ++j) if (nu[j] > nu[bi]) bi = j;
        const float bsq = nu[bi] * nu[bi];
        if (np == 3 && bsq < threshold_helper * (float)(3 - k)) np = k;
        if (bi != k) {
            for (int r = 0; r < 3; ++r) { float t = a[r + 3 * k]; a[r + 3 * k] = a[r + 3 * bi]; a[r + 3 * bi] = t; }
            float t = nu[k]; nu[k] = nu[bi]; nu[bi] = t;
            t = nd[k]; nd[k] = nd[bi]; nd[bi] = t;
            int ti = perm[k]; perm[k] = perm[bi]; perm[bi] = ti;
        }
        /* makeHouseholderInPlace on col(k).tail(3 - k) */
        const float c0 = a[k + 3 * k];
        float tail_sq = 0.f;
        for (int r = k + 1; r < 3; ++r) tail_sq = (r == k + 1) ? a[r + 3 * k] * a[r + 3 * k] : tail_sq + a[r + 3 * k] * a[r + 3 * k];
        float tau, beta;
        if (tail_sq <= FLT_MIN) {
            tau = 0.f; beta = c0;
            for (int r = k + 1; r < 3; ++r) a[r + 3 * k] = 0.f;
        } else {
            beta = sqrtf(c0 * c0 + tail_sq);
            if (c0 >= 0.f) beta = -beta;
            const float den = c0 - beta;
            for (int r = k + 1; r < 3; ++r) a[r + 3 * k] = a[r + 3 * k] / den;
            tau = (beta - c0) / beta;
        }
        hc[k] = tau;
        a[k + 3 * k] = beta;
        /* applyHouseholderOnTheLeft to the bottom-right (3-k) x (2-k) corner (rows() > 1 here whenever it has columns) */
        if (tau != 0.f) {
            for (int j = k + 1; j < 3; ++j) {
                float t = 0.f;
                for (int r = k + 1; r < 3; ++r) t += a[r + 3 * k] * a[r + 3 * j];
                t = t + a[k + 3 * j];
                a[k + 3 * j] = a[k + 3 * j] - tau * t;
                for (int r = k + 1; r < 3; ++r) a[r + 3 * j] = a[r + 3 * j] - t * (tau * a[r + 3 * k]);
            }
        }
        /* column-norm downdate (LAPACK xGEQPF / Eigen 3.3) */
        for (int j = k + 1; j < 3; ++j) {
            if (nu[j] != 0.f) {
                float t = fabsf(a[k + 3 * j]) / nu[j];
                t = (1.f + t) * (1.f - t);
                t = t < 0.f ? 0.f : t;
                const float q = nu[j] / nd[j];
                const float t2 = t * (q * q);
                if (t2 <= norm_downdate_threshold) {
                    float s = 0.f;
                    for (int r = k + 1; r < 3; ++r) s = (r == k + 1) ? a[r + 3 * j] * a[r + 3 * j] : s + a[r + 3 * j] * a[r + 3 * j];
                    nd[j] = sqrtf(s);
                    nu[j] = nd[j];
                } else {
                    nu[j] *= sqrtf(t);
                }
            }
        }
    }
    if (np == 0) { x[0] = x[1] = x[2] = 0.f; return; }
    float c[3] = {b[0], b[1], b[2]};
    /* c = H_{np-1} ... H_0 b */
    for (int k = 0; k < np; ++k) {
        if (k == 2) { c[2] = c[2] * (1.f - hc[2]); continue; }
        if (hc[k] != 0.f) {
            float t = a[k + 1 + 3 * k] * c[k + 1];
            for (int r = k + 2; r < 3; ++r) t = t + a[r + 3 * k] * c[r];
            t = t + c[k];
            c[k] = c[k] - hc[k] * t;
            for (int r = k + 1; r < 3; ++r) c[r] = c[r] - t * (hc[k] * a[r + 3 * k]);
        }
    }
    /* upper-triangular back substitution over the first np pivots (column oriented, zero right-hand sides skipped) */
    for (int i = np - 1; i >= 0; --i) {
        if (c[i] != 0.f) {
            c[i] = c[i] / a[i + 3 * i];
            for (int s = 0; s < i; ++s) c[s] = c[s] - c[i] * a[s + 3 * i];
        }
    }
    x[0] = x[1] = x[2] = 0.f;
    for (int i = 0; i < np; ++i) x[perm[i]] = c[i];
}

/* ------------------------------------------------------------------------------------------ */
/* IntensityGradientEstimation::computeFeature, is_dense branch (PointCloudXYZRGBtoXYZI leaves is_dense = true).
 * pts[*, stride_f]: the surface; intensity[*]: one float per surface row; normals[nq, 4]; rows nbr[offsets[i] ..
 * offsets[i+1]) in (d2, index) order.  out[nq, 4] = gx, gy, gz, 0. */
ORC_API void orc_intensity_gradient_from_lists(const float *pts, int stride_f, const float *intensity, const float *normals, int64_t nq,
                                               const int64_t *offsets, const int32_t *nbr, float *out) {
#ifdef _OPENMP
#pragma omp parallel for schedule(static)
#endif
    for (int64_t i = 0; i < nq; ++i) {
        float *o = out + 4 * i;
        const int32_t *l = nbr + offsets[i];
        const int64_t m = offsets[i + 1] - offsets[i];
        o[3] = 0.f;
        if (m < 3) { o[0] = o[1] = o[2] = NAN; continue; }     /* |N| == 0: searchForNeighbors fails; < 3: computePointIntensityGradient */
        float cx = 0.f, cy = 0.f, cz = 0.f, mi = 0.f;
        for (int64_t j = 0; j < m; ++j) {
            const float *p = pts + (int64_t)l[j] * stride_f;
            cx += p[0]; cy += p[1]; cz += p[2];
            mi += intensity[l[j]];
        }
        const float fn = (float)m;
        cx = cx / fn; cy = cy / fn; cz = cz / fn; mi = mi / fn;
        float a00 = 0.f, a01 = 0.f, a02 = 0.f, a11 = 0.f, a12 = 0.f, a22 = 0.f, b0 = 0.f, b1 = 0.f, b2 = 0.f;
        for (int64_t j = 0; j < m; ++j) {
            const float *p = pts + (int64_t)l[j] * stride_f;
            const float in = intensity[l[j]];
            if (!isfinite(p[0]) || !isfinite(p[1]) || !isfinite(p[2]) || !isfinite(in)) continue;
            const float x = p[0] - cx, y = p[1] - cy, z = p[2] - cz, v = in - mi;
            a00 += x * x; a01 += x * y; a02 += x * z;
            a11 += y * y; a12 += y * z;
            a22 += z * z;
            b0 += x * v; b1 += y * v; b2 += z * v;
        }
        const float A[9] = {a00, a01, a02, a01, a11, a12, a02, a12, a22};   /* symmetric: column-major == row-major */
        const float b[3] = {b0, b1, b2};
        float x[3];
        orc_colpiv_qr_solve3(A, b, x);
        const float *n = normals + 4 * i;
        /* gradient = (I - n n^T) x: M evaluated first, then one fixed-size-3 reduction per row */
        float M[9];
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c) M[3 * r + c] = (r == c ? 1.f : 0.f) - n[r] * n[c];
        for (int r = 0; r < 3; ++r) o[r] = sum3(M[3 * r] * x[0], M[3 * r + 1] * x[1], M[3 * r + 2] * x[2]);
    }
}

/* ------------------------------------------------------------------------------------------ */
/* Eigen 3.3's SSE reduction of a squared norm over n contiguous floats (packets of 4, two accumulators, predux
 * (l0 + l2) + (l1 + l3), then the scalar tail) -- the order MatrixXf::normalize() uses on an x86-64 build without -march. */
static float sq_norm_sse(const float *h, int n) {
    if (n < 4) {
        float s = h[0] * h[0];
        for (int i = 1; i < n; ++i) s = s + h[i] * h[i];
        return s;
    }
    const int aligned = n & ~3, aligned2 = n & ~7;
    float r0[4], r1[4];
    for (int l = 0; l < 4; ++l) r0[l] = h[l] * h[l];
    if (aligned > 4) {
        for (int l = 0; l < 4; ++l) r1[l] = h[4 + l] * h[4 + l];
        for (int idx = 8; idx < aligned2; idx += 8)
            for (int l = 0; l < 4; ++l) { r0[l] = r0[l] + h[idx + l] * h[idx + l]; r1[l] = r1[l] + h[idx + 4 + l] * h[idx + 4 + l]; }
        for (int l = 0; l < 4; ++l) r0[l] = r0[l] + r1[l];
        if (aligned > aligned2)
            for (int l = 0; l < 4; ++l) r0[l] = r0[l] + h[aligned2 + l] * h[aligned2 + l];
    }
    float s = (r0[0] + r0[2]) + (r0[1] + r0[3]);
    for (int i = aligned; i < n; ++i) s = s + h[i] * h[i];
    return s;
}

/* RIFTEstimation::computeFeature + computeRIFT.  qpts[nq, qstride_f]: the query points (p0); rows nbr / d2 in (d2, index)
 * order over pts; gradient[*, 4] per surface row.  out[nq, nd*ng] in PCL's histogram order (gradient bin outer, distance bin
 * inner); NaN row without neighbours.  Returns -1 when nd*ng is not in 1..32. */
ORC_API int orc_rift_from_lists(const float *pts, int stride_f, const float *qpts, int64_t nq, int qstride_f, const int64_t *offsets,
                                const int32_t *nbr, const float *d2, const float *gradient, float radius, int nd, int ng, float *out) {
    const int nb = nd * ng;
    if (nd < 1 || ng < 1 || nb > 32) return -1;
    const float eps = FLT_EPSILON;
    const float rden = radius + eps, gden = (float)M_PI + eps;
#ifdef _OPENMP
#pragma omp parallel for schedule(static)
#endif
    for (int64_t i = 0; i < nq; ++i) {
        float *o = out + i * nb;
        const int64_t b = offsets[i], m = offsets[i + 1] - b;
        if (m == 0) { for (int k = 0; k < nb; ++k) o[k] = NAN; continue; }
        float h[32];
        for (int k = 0; k < nb; ++k) h[k] = 0.f;
        const float *p0 = qpts + i * qstride_f;
        for (int64_t j = 0; j < m; ++j) {
            const int32_t id = nbr[b + j];
            const float *p = pts + (int64_t)id * stride_f;
            const float *g = gradient + 4 * (int64_t)id;
            const float mag = sqrtf(sum3(g[0] * g[0], g[1] * g[1], g[2] * g[2]));
            float ux = p[0] - p0[0], uy = p[1] - p0[1], uz = p[2] - p0[2];
            const float z = sum3(ux * ux, uy * uy, uz * uz);
            if (z > 0.f) { const float s = sqrtf(z); ux = ux / s; uy = uy / s; uz = uz / s; }     /* normalized(): zero stays zero */
            float ang = acosf(sum3(g[0] * ux, g[1] * uy, g[2] * uz) / mag);
            if (!isfinite(ang)) ang = 0.f;
            const float dist = (float)nd * sqrtf(d2[b + j]) / rden;
            const float grad = (float)ng * ang / gden;
            int dmin = (int)ceilf(dist - 1.f), dmax = (int)floorf(dist + 1.f);
            if (dmin < 0) dmin = 0;
            if (dmax > nd - 1) dmax = nd - 1;
            const int gmin = (int)ceilf(grad - 1.f), gmax = (int)floorf(grad + 1.f);
            for (int gi = gmin; gi <= gmax; ++gi) {
                const int gw = (gi + ng) % ng;
                for (int di = dmin; di <= dmax; ++di) {
                    const float w = (1.0f - fabsf(dist - (float)di)) * (1.0f - fabsf(grad - (float)gi));
                    h[gw * nd + di] += w * mag;
                }
            }
        }
        const float z = sq_norm_sse(h, nb);
        if (z > 0.f) { const float s = sqrtf(z); for (int k = 0; k < nb; ++k) h[k] = h[k] / s; }
        for (int k = 0; k < nb; ++k) o[k] = h[k];
    }
    return 0;
}

/* PCL 1.7 PointXYZRGBtoXYZI: 0.299f r + 0.587f g + 0.114f b, left to right, no contraction.  rgb[n, 3] uint8. */
ORC_API void orc_rgb_to_intensity(const uint8_t *rgb, int64_t n, float *out) {
    for (int64_t i = 0; i < n; ++i) out[i] = 0.299f * (float)rgb[3 * i] + 0.587f * (float)rgb[3 * i + 1] + 0.114f * (float)rgb[3 * i + 2];
}

/* ------------------------------------------------------------------------------------------ */
/* pcl::SIFTKeypoint<PointXYZRGB, PointWithScale> (src/comparator.cpp:449-465) [up]: the per-octave scale table, the field
 * selector, computeScaleSpace and findScaleSpaceExtrema over caller-supplied neighbour rows.                                  */

/* expf restated exactly as pcc_device.cuh sift_expf: fp64, every operation separately rounded (this file is built with
 * -ffp-contract=off), Cody-Waite reduction by fdlibm's split of ln 2, Horner Taylor polynomial to r^11, exact scaling by 2^k,
 * one rounding to fp32.  Valid for x in [-80, 80]. */
static float sift_expf1(float x) {
    const double xd = (double)x;
    const double k = rint(xd * 1.4426950408889634);
    const double r = (xd - k * 0.6931471803691238) - k * 1.9082149292705877e-10;
    double p = 2.505210838544172e-08;
    p = p * r + 2.755731922398589e-07;
    p = p * r + 2.7557319223985893e-06;
    p = p * r + 2.48015873015873e-05;
    p = p * r + 0.0001984126984126984;
    p = p * r + 0.001388888888888889;
    p = p * r + 0.008333333333333333;
    p = p * r + 0.041666666666666664;
    p = p * r + 0.16666666666666666;
    p = p * r + 0.5;
    p = p * r + 1.0;
    p = p * r + 1.0;
    const uint64_t bits = (uint64_t)((int64_t)k + 1023) << 52;
    double two_k;
    memcpy(&two_k, &bits, sizeof two_k);
    return (float)(p * two_k);
}

ORC_API void orc_sift_expf(const float *x, int64_t n, float *out) {
    for (int64_t i = 0; i < n; ++i) out[i] = sift_expf1(x[i]);
}

/* detectKeypointsForOctave: scales[i] = base_scale * powf (2.0f, (1.0f * static_cast<float> (i) - 1.0f) / static_cast<float> (nr_scales_per_octave)) */
ORC_API void orc_sift_scales(float base_scale, int nr_scales_per_octave, float *scales) {
    for (int i = 0; i < nr_scales_per_octave + 3; ++i)
        scales[i] = base_scale * powf(2.0f, (1.0f * (float)i - 1.0f) / (float)nr_scales_per_octave);
}

/* SIFTKeypointFieldSelector<PointXYZRGB>: static_cast<float> (299*p.r + 587*p.g + 114*p.b) / 1000.0f.  rgb[n, 3] uint8. */
ORC_API void orc_sift_field_values(const uint8_t *rgb, int64_t n, float *out) {
    for (int64_t i = 0; i < n; ++i) out[i] = (float)(299 * rgb[3 * i] + 587 * rgb[3 * i + 1] + 114 * rgb[3 * i + 2]) / 1000.0f;
}

/* computeScaleSpace over one sorted radius row per point (rows at max_radius = 3.0f * scales[n_scales-1]), PCL's loop as written:
 * for every scale a walk over the row that breaks at the first neighbour with d2 > 9*sigma_sqr.  values[] by neighbour index,
 * out[nq * (n_scales-1)]; an empty row gives 0/0 = NaN. */
ORC_API void orc_sift_dog_from_lists(const float *values, int64_t nq, const int64_t *offsets, const int32_t *nbr, const float *d2,
                                     const float *scales, int n_scales, float *out) {
#ifdef _OPENMP
#pragma omp parallel for schedule(dynamic, 256)
#endif
    for (int64_t i = 0; i < nq; ++i) {
        float filter_response = 0.0f, previous_filter_response;
        for (int s = 0; s < n_scales; ++s) {
            const float sigma_sqr = powf(scales[s], 2.0f);
            float numerator = 0.0f, denominator = 0.0f;
            for (int64_t j = offsets[i]; j < offsets[i + 1]; ++j) {
                const float value = values[nbr[j]];
                const float dist_sqr = d2[j];
                if (dist_sqr <= 9 * sigma_sqr) {
                    const float w = sift_expf1(-0.5f * dist_sqr / sigma_sqr);
                    numerator += value * w;
                    denominator += w;
                } else break;
            }
            previous_filter_response = filter_response;
            filter_response = numerator / denominator;
            if (s > 0) out[i * (n_scales - 1) + (s - 1)] = filter_response - previous_filter_response;
        }
    }
}

/* findScaleSpaceExtrema over nn[n * k] neighbour rows (entries < 0 are absent): min / max per column with std::min / std::max,
 * then PCL's keypoint test.  Writes at most cap (row, column) pairs in (row, column) order; returns the full count. */
ORC_API int64_t orc_sift_extrema_from_lists(const float *dog, int64_t n, int nc, const int32_t *nn, int k, float min_contrast,
                                            int32_t *out_row, int32_t *out_col, int64_t cap) {
    float min_val[16], max_val[16];
    int64_t found = 0;
    for (int64_t i = 0; i < n; ++i) {
        for (int c = 0; c < nc; ++c) {
            min_val[c] = FLT_MAX;
            max_val[c] = -FLT_MAX;
            for (int j = 0; j < k; ++j) {
                const int32_t id = nn[i * k + j];
                if (id < 0) continue;
                const float d = dog[(int64_t)id * nc + c];
                min_val[c] = (d < min_val[c]) ? d : min_val[c];      /* std::min (min_val, d) */
                max_val[c] = (max_val[c] < d) ? d : max_val[c];      /* std::max (max_val, d) */
            }
        }
        for (int c = 1; c < nc - 1; ++c) {
            const float val = dog[i * nc + c];
            int hit = 0;
            if (fabsf(val) >= min_contrast) {
                if (val == min_val[c] && val < min_val[c - 1] && val < min_val[c + 1]) hit = 1;
                else if (val == max_val[c] && val > max_val[c - 1] && val > max_val[c + 1]) hit = 1;
            }
            if (hit) {
                if (found < cap) { out_row[found] = (int32_t)i; out_col[found] = c; }
                ++found;
            }
        }
    }
    return found;
}

ORC_API int orc_desc_num_threads(void) {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}
