// k_census.cu — K1a for the census cost mode (sva_params.reserved[0] == SVA_COST_CENSUS): 9 x 7 census signatures of every view, then the
// per-pixel Hamming distance summed over the camera pairs, written in the same planar layout (ApGeom) as the SAD form so that K1b, SGM and K3
// run unchanged.
//
//   T(y,x)   : 62 bits, bit b = [ I(y+dy, x+dx) < I(y,x) ] over dy in [-3,3], dx in [-4,4] without the centre, row-major; outside = 0
//   A(y,x,d) = sum_k popcount(T_R(y,x) ^ T_k(y - gy_k*delta, x - gx_k*delta)),  delta = min_disp + d;  an out-of-image source has T = 0
//
// north_star names a "census/SAD matching cost"; the reference has only SAD (src/functions.cpp:215-218), so this mode has no reference
// counterpart: the spec is frozen in oracle/sva_oracle.c (census_ad_volume) and parity is against that.  Written for correctness first: one
// thread per pixel and 8 disparities, signatures fetched through L1 / L2 (all views' signatures of a c1 frame are 88 MB: L2-resident).
#include "sva_common.cuh"

#define CENSUS_RX 4
#define CENSUS_RY 3

// signature of pixel (x, y): shared by the per-view transform and the batched transform of an array frame's camera stack
__device__ __forceinline__ uint64_t census_signature(const uint8_t* __restrict__ img, size_t pitch, int W, int H, int x, int y) {
    const int c = img[(size_t)y * pitch + x];
    uint64_t t = 0;
    int bit = 0;
#pragma unroll
    for (int dy = -CENSUS_RY; dy <= CENSUS_RY; dy++) {
        const int yy = y + dy;
        const bool row_ok = yy >= 0 && yy < H;
#pragma unroll
        for (int dx = -CENSUS_RX; dx <= CENSUS_RX; dx++) {
            if (dx == 0 && dy == 0) continue;
            const int xx = x + dx;
            const int v = (row_ok && xx >= 0 && xx < W) ? (int)__ldg(img + (size_t)yy * pitch + xx) : 0;
            t |= (uint64_t)(v < c) << bit;
            bit++;
        }
    }
    return t;
}

__global__ void __launch_bounds__(128)
k_census_transform(const uint8_t* __restrict__ img, size_t pitch, int W, int H, uint64_t* __restrict__ out) {
    const int x = blockIdx.x * 128 + threadIdx.x, y = blockIdx.y;
    if (x >= W) return;
    out[(size_t)y * W + x] = census_signature(img, pitch, W, H, x, y);
}

// Cameras of an array frame's stack (tight W x H views, camera i at stack + i * W * H) whose signatures one launch computes.
struct CensusCams {
    int n;
    int cam[SVA_MAX_PAIRS + 1];  // a group reads at most 32 other views and its reference
};

// the signatures of cameras L.cam[blockIdx.z] of the stack into the same slots of the signature stack
__global__ void __launch_bounds__(128)
k_census_transform_stack(const uint8_t* __restrict__ stack, int W, int H, const CensusCams L, uint64_t* __restrict__ sig) {
    const int x = blockIdx.x * 128 + threadIdx.x, y = blockIdx.y;
    if (x >= W) return;
    const size_t off = (size_t)W * H * L.cam[blockIdx.z];
    sig[off + (size_t)y * W + x] = census_signature(stack + off, (size_t)W, W, H, x, y);
}

// one launch for up to SVA_MAX_PAIRS + 1 cameras of the stack, on `stream`
int sva_census_stack(sva_ctx* ctx, const uint8_t* stack, int W, int H, const int* cams, int n, uint64_t* sig, cudaStream_t stream) {
    if (n <= 0) return SVA_OK;
    if (n > SVA_MAX_PAIRS + 1) return ctx->fail(SVA_ERR_BAD_ARG, "census_stack: too many cameras in one launch");
    CensusCams L{};
    L.n = n;
    for (int i = 0; i < n; i++) L.cam[i] = cams[i];
    {
        LaunchScope ls(ctx, "k_census_transform_stack");
        k_census_transform_stack<<<dim3(div_up(W, 128), H, n), 128, 0, stream>>>(stack, W, H, L, sig);
    }
    SVA_CUDA_OK(ctx, cudaGetLastError());
    return SVA_OK;
}

struct CensusPairs {
    int n;
    int gx[SVA_MAX_PAIRS], gy[SVA_MAX_PAIRS];
    int view[SVA_MAX_PAIRS];  // index of the pair's other view
};

__global__ void __launch_bounds__(128)
k_ad_census(const uint64_t* __restrict__ tr, const uint64_t* __restrict__ to, const CensusPairs P, int W, int H, int D, int dmin,
            uint32_t* __restrict__ AP, int wp, int padl, int padt) {
    const int x = blockIdx.x * 128 + threadIdx.x, y = blockIdx.y, d0 = blockIdx.z * 8;
    if (x >= W) return;
    const uint64_t r = tr[(size_t)y * W + x];
    uint32_t acc[8];
#pragma unroll
    for (int i = 0; i < 8; i++) acc[i] = 0;
    const size_t px = (size_t)W * H;
    for (int k = 0; k < P.n; k++) {
        const uint64_t* t = to + px * P.view[k];
        const int gx = P.gx[k], gy = P.gy[k];
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const int delta = dmin + d0 + i, sx = x - gx * delta, sy = y - gy * delta;
            uint64_t v = 0;
            if (sx >= 0 && sx < W && sy >= 0 && sy < H) v = __ldg(t + (size_t)sy * W + sx);
            acc[i] += __popcll(r ^ v);
        }
    }
    uint32_t* out = AP + ((size_t)(y + padt) * (D >> 1) + (d0 >> 1)) * wp + padl + x;
#pragma unroll
    for (int i = 0; i < 4; i++)
        if (d0 + 2 * i < D) out[(size_t)i * wp] = acc[2 * i] | (acc[2 * i + 1] << 16);
}

int sva_ap_prepare(sva_ctx* ctx);

// views as uploaded for this mode: ctx->ref_img / ctx->other_imgs, tight pitch W; or, inside sva_depth_groups, the signatures of the
// array frame's camera stack (ctx->sig_stack), computed once per camera for all groups
int sva_run_ad_census(sva_ctx* ctx) {
    const sva_params& p = ctx->prm;
    const int W = p.width, H = p.height, D = p.num_disp;
    const size_t px = (size_t)W * H;
    SVA_TRY(sva_ap_prepare(ctx));
    if (ctx->sig_stack) {
        CensusPairs P{};
        P.n = ctx->pair_end - ctx->pair_begin;
        for (int i = 0; i < P.n; i++) {
            const int k = ctx->pair_begin + i;
            P.gx[i] = p.pair_gx[k]; P.gy[i] = p.pair_gy[k]; P.view[i] = ctx->sig_view[k];
        }
        {
            LaunchScope ls(ctx, "k_ad_census");
            k_ad_census<<<dim3(div_up(W, 128), H, div_up(D, 8)), 128, 0, ctx->stream>>>(ctx->sig_stack + px * ctx->sig_ref, ctx->sig_stack, P, W, H, D, p.min_disp,
                                                                                        ctx->AP.as<uint32_t>(), ctx->ap.wp, ctx->ap.padl, ctx->ap.padt);
        }
        SVA_CUDA_OK(ctx, cudaGetLastError());
        ctx->have_ad = true;
        return SVA_OK;
    }
    SVA_TRY(ctx->reserve(ctx->census, px * sizeof(uint64_t) * (size_t)(p.n_pairs + 1)));
    uint64_t* tr = ctx->census.as<uint64_t>();
    uint64_t* to = tr + px;
    const dim3 g2(div_up(W, 128), H);
    {
        LaunchScope ls(ctx, "k_census_transform");
        k_census_transform<<<g2, 128, 0, ctx->stream>>>(ctx->ref_img.as<uint8_t>(), (size_t)W, W, H, tr);
        for (int i = ctx->pair_begin; i < ctx->pair_end; i++)
            k_census_transform<<<g2, 128, 0, ctx->stream>>>(ctx->other_imgs.as<uint8_t>() + px * i, (size_t)W, W, H, to + px * i);
        ctx->launches += ctx->pair_end - ctx->pair_begin;
    }
    SVA_CUDA_OK(ctx, cudaGetLastError());
    CensusPairs P{};
    P.n = ctx->pair_end - ctx->pair_begin;
    for (int i = 0; i < P.n; i++) { P.gx[i] = p.pair_gx[ctx->pair_begin + i]; P.gy[i] = p.pair_gy[ctx->pair_begin + i]; P.view[i] = ctx->pair_begin + i; }
    {
        LaunchScope ls(ctx, "k_ad_census");
        k_ad_census<<<dim3(div_up(W, 128), H, div_up(D, 8)), 128, 0, ctx->stream>>>(tr, to, P, W, H, D, p.min_disp, ctx->AP.as<uint32_t>(), ctx->ap.wp, ctx->ap.padl, ctx->ap.padt);
    }
    SVA_CUDA_OK(ctx, cudaGetLastError());
    ctx->have_ad = true;
    return SVA_OK;
}
