/*
 * fuse_oracle.c — TEST INFRASTRUCTURE ONLY.  CPU restatement of the multi-view depth fusion spec (DESIGN.md §3 item 6), the checker of
 * sva_fuse_maps / sva_depth_groups_fused.  No reference counterpart: parity is UNPINNED by the reference; this file is the frozen spec's
 * executable form.  Compiled at test time by tests/fuse_oracle.py (gcc -ffp-contract=off) into a temporary directory.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

#include "../include/sva_c_api.h"

/* Multi-view depth fusion — DESIGN.md §3 item 6 (frozen spec; no reference counterpart, parity UNPINNED by the reference).
 * View g: reference camera view_refs[g], integer map disp[g] and, when subpix != NULL, sub-pixel map subpix[g]; camera i sits at column
 * i % grid_cols, row i / grid_cols.  mask: NULL or width x height, tight (0 = reject).  out_subpix / out_support may be NULL. */
int orc_fuse_views(int32_t width, int32_t height, int32_t grid_cols, const int32_t* view_refs, int32_t n_views, const uint16_t* const* disp,
                   const float* const* subpix, int32_t target, int32_t tol_16, int32_t min_support, const uint8_t* mask, uint16_t* out_disp,
                   float* out_subpix, uint8_t* out_support) {
    const int W = width, H = height, G = n_views;
    const size_t px = (size_t)W * H;
    if (W < 1 || H < 1 || grid_cols < 1 || G < 1 || G > 32) return SVA_ERR_BAD_ARG;
    /* steps 1-3: Z[g][p] = 1 + the largest q of view g landing on target pixel p, 0 where none lands */
    uint32_t* Z = (uint32_t*)calloc(px * G, sizeof(uint32_t));
    if (!Z) return SVA_ERR_NOMEM;
    for (int g = 0; g < G; g++) {
        const long long gx = target % grid_cols - view_refs[g] % grid_cols, gy = target / grid_cols - view_refs[g] / grid_cols;  /* step 2 */
        for (int y = 0; y < H; y++)
            for (int x = 0; x < W; x++) {
                const size_t o = (size_t)y * W + x;
                if (disp[g][o] == SVA_DISP_INVALID) continue;                           /* step 1: used iff valid ... */
                long long q;
                if (subpix) {
                    const float sv = subpix[g][o];
                    if (!(sv >= 0.0f && sv < 4352.0f)) continue;                        /* ... and 0 <= S < 4352 (NaN fails) */
                    q = (long long)nearbyintf(16.0f * sv);                              /* rint, ties to even */
                } else {
                    q = 16LL * disp[g][o];
                }
                const long long xt = x - ((gx * q + 8) >> 4), yt = y - ((gy * q + 8) >> 4);   /* step 2: floor shifts */
                if (xt < 0 || xt >= W || yt < 0 || yt >= H) continue;
                uint32_t* z = &Z[(size_t)g * px + (size_t)yt * W + xt];
                if ((uint32_t)(q + 1) > *z) *z = (uint32_t)(q + 1);                      /* step 3: the nearest surface */
            }
    }
    /* steps 4-5 */
    for (size_t o = 0; o < px; o++) {
        long long best = -1;
        int best_n = 0;
        for (int g = 0; g < G; g++) {
            if (!Z[(size_t)g * px + o]) continue;
            const long long cg = (long long)Z[(size_t)g * px + o] - 1;
            int n = 0;                                                                   /* support(c_g) */
            for (int h = 0; h < G; h++)
                if (Z[(size_t)h * px + o] && llabs((long long)Z[(size_t)h * px + o] - 1 - cg) <= tol_16) n++;
            if (n > best_n || (n == best_n && cg > best)) { best = cg; best_n = n; }      /* largest support, ties: the larger value */
        }
        long long sum = 0;
        for (int h = 0; h < G; h++)
            if (Z[(size_t)h * px + o] && llabs((long long)Z[(size_t)h * px + o] - 1 - best) <= tol_16) sum += (long long)Z[(size_t)h * px + o] - 1;
        const int ok = best_n > 0 && best_n >= min_support && (!mask || mask[o]);
        if (out_support) out_support[o] = (uint8_t)best_n;
        if (!ok) {
            out_disp[o] = SVA_DISP_INVALID;
            if (out_subpix) out_subpix[o] = SVA_SUBPIX_INVALID;
            continue;
        }
        const long long qh = (sum + best_n / 2) / best_n;
        out_disp[o] = (uint16_t)((qh + 8) >> 4);
        if (out_subpix) out_subpix[o] = (float)qh / 16.0f;
    }
    free(Z);
    return SVA_OK;
}


