/* dW of gvcnn_view_score_bwd (csrc/paper_mode.cu, view_score_bwd_partial_kernel / _final_kernel), restated for
 * tests/score_grad_oracle.py.  TEST INFRASTRUCTURE ONLY.  Build with -ffp-contract=off: every operation below is one
 * IEEE float32 rounding, fmaf() one rounding of the exact a * b + c.
 *   slice sl of 32 covers shapes [B * sl / 32, B * (sl + 1) / 32)
 *   partial[sl, v, c] = fmaf chain over the slice's shapes in ascending order, from 0
 *   dW[v, c] = 0 + partial[0] + partial[1] + ... (ascending) */
#include <math.h>
#include <stdint.h>

void score_grad_dw(const float *R, const float *dx, int64_t B, int V, int C, float *dW)
{
    const int NS = 32;
    for (int v = 0; v < V; ++v)
        for (int c = 0; c < C; ++c) {
            float s = 0.0f;
            for (int sl = 0; sl < NS; ++sl) {
                const int64_t b0 = B * sl / NS, b1 = B * (sl + 1) / NS;
                float acc = 0.0f;
                for (int64_t b = b0; b < b1; ++b) acc = fmaf(dx[b * V + v], R[(b * V + v) * (int64_t)C + c], acc);
                s = s + acc;
            }
            dW[(int64_t)v * C + c] = s;
        }
}
