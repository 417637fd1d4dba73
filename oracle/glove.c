/*
 * oracle/glove.c -- TEST INFRASTRUCTURE: CPU restatement of the GloVe objective trained on
 * random-walk co-occurrences, the model behind `Node2VecGloVeEnsmallen` /
 * `DeepWalkGloVeEnsmallen` (/root/reference/embiggen/embedders/ensmallen_embedders/
 * node2vec_glove.py:5-140, deepwalk_glove.py; kwargs `alpha`, `learning_rate`,
 * `learning_rate_decay`, `window_size`, `walk_length`, one walk per node and epoch :104-106).
 * The arithmetic lives in the un-vendored `ensmallen` wheel: PARITY UNPINNED against it; the
 * objective is Pennington et al. 2014 eq. 8 without bias terms, with x_max = the largest
 * count of the epoch.  Floating point is specified operation by operation so that a
 * single-warp GPU launch reproduces the tables bit for bit.  Compile with -ffp-contract=off.
 */
#include "oracle.h"
#include <math.h>
#include <string.h>

/* ln(x) for normal x > 0: x = m * 2^e with m in [sqrt(1/2), sqrt(2)); s = (m-1)/(m+1);
 * ln m = 2 s (1 + s^2/3 + s^4/5 + s^6/7 + s^8/9) */
float orc_log_det(float x) {
    union { float f; uint32_t u; } v;
    v.f = x;
    int32_t e = (int32_t)(v.u >> 23) - 127;
    v.u = (v.u & 0x007FFFFFu) | 0x3F800000u; /* m in [1, 2) */
    float m = v.f;
    if (m > 1.41421356237f) { m = m * 0.5f; e += 1; }
    const float s = (m - 1.0f) / (m + 1.0f);
    const float s2 = s * s;
    float p = 1.0f / 9.0f;
    p = fmaf(p, s2, 1.0f / 7.0f);
    p = fmaf(p, s2, 1.0f / 5.0f);
    p = fmaf(p, s2, 1.0f / 3.0f);
    p = fmaf(p, s2, 1.0f);
    const float lnm = (2.0f * s) * p;
    return fmaf((float)e, 0.693147180559945f, lnm);
}

int orc_glove_train(const uint32_t *centre, const uint32_t *context, const uint32_t *count,
                    uint64_t n_triples, uint32_t max_count, uint32_t embedding_size,
                    uint32_t row_stride, float alpha, float clipping_value, float learning_rate,
                    int tile_semantics, float *t0, float *t1, double *loss_sum, uint64_t *trained) {
    if (!centre || !context || !count || !t0 || !t1 || max_count == 0) return -1;
    if ((row_stride & 3) || row_stride < embedding_size || row_stride > 4096) return -1;
    float h[4096], h0[4096];
    double loss = 0.0;
    uint64_t done = 0;
    uint64_t e = 0;
    while (e < n_triples) {
        const uint32_t c = centre[e];
        float *crow = t0 + (uint64_t)c * row_stride;
        memcpy(h, crow, row_stride * sizeof(float));
        memcpy(h0, crow, row_stride * sizeof(float));
        for (; e < n_triples && centre[e] == c; ++e) {
            float *row = t1 + (uint64_t)context[e] * row_stride;
            const float f = orc_dot(h, row, row_stride);
            if (fabsf(f) > clipping_value) continue;
            const float x = (float)count[e];
            const float weight = orc_exp_det(alpha * orc_log_det(x / (float)max_count));
            const float diff = f - orc_log_det(x);
            const float g = ((2.0f * weight) * diff) * learning_rate;
            loss += (double)weight * (double)diff * (double)diff;
            ++done;
            for (uint32_t k = 0; k < row_stride; ++k) {
                const float old = row[k];
                if (tile_semantics) {
                    const float step = -g * h[k];
                    row[k] = old + step;
                } else {
                    row[k] = fmaf(-g, h[k], old);
                }
                h[k] = fmaf(-g, old, h[k]);
            }
        }
        if (tile_semantics) {
            for (uint32_t k = 0; k < row_stride; ++k) {
                const float change = h[k] - h0[k];
                crow[k] = crow[k] + change;
            }
        } else {
            memcpy(crow, h, row_stride * sizeof(float));
        }
    }
    if (loss_sum) *loss_sum += loss;
    if (trained) *trained += done;
    return 0;
}
