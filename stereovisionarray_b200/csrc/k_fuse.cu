// k_fuse.cu — multi-view depth fusion (DESIGN §3 item 6): the disparity maps of several reference views of one array frame merged into
// one camera's view.  No reference counterpart; the spec is orc_fuse_views (tests/fuse_oracle.c), restated in include/sva_c_api.h.
//
// Two launches.  k_fuse_splat forward-warps every used pixel of every view into the target's view and keeps, per view and target pixel,
// the nearest surface: an atomicMax of q + 1 into that view's u32 plane (0 = nothing landed).  k_fuse_consensus reads the G planes of a
// target pixel (coalesced) and votes in registers.  All integer after the fixed-point step, so the order of the atomics and of the views
// cannot change the result.  sva_depth_groups_fused (sva_groups.cu) splats each group's maps straight from its IoSet after its K3; the host
// form below uploads the caller's maps first.
#include "sva_common.cuh"

// grid offsets (col t - col r_g, row t - row r_g) of the views of one splat launch, view v at blockIdx.y = v
struct FuseOffsets {
    int gx[SVA_MAX_PAIRS], gy[SVA_MAX_PAIRS];
};

// §3 item 6 steps 1-3, one thread per source pixel of view v = blockIdx.y.  disp / sub: view v at + v * view_stride; sub == nullptr:
// integer maps.  planes: view v at + v * W * H.
__global__ void __launch_bounds__(256) k_fuse_splat(const uint16_t* __restrict__ disp, const float* __restrict__ sub, size_t view_stride,
                                                    FuseOffsets off, int W, int H, uint32_t* __restrict__ planes) {
    const size_t px = (size_t)W * H, i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    const int v = blockIdx.y;
    if (i >= px) return;
    const uint16_t d = disp[v * view_stride + i];
    if (d == SVA_DISP_INVALID) return;
    int q;
    if (sub) {
        const float s = sub[v * view_stride + i];
        if (!(s >= 0.0f && s < 4352.0f)) return;  // (NaN fails)
        q = __float2int_rn(16.0f * s);             // 16 * s is exact in f32; ties to even
    } else {
        q = 16 * (int)d;
    }
    const int y = (int)(i / W), x = (int)(i - (size_t)y * W);
    // (64-bit: |gx| * q may exceed 2^31 on a wide grid)
    const long long xt = x - ((off.gx[v] * (long long)q + 8) >> 4), yt = y - ((off.gy[v] * (long long)q + 8) >> 4);
    if (xt < 0 || xt >= W || yt < 0 || yt >= H) return;
    atomicMax(planes + v * px + (size_t)yt * W + xt, (uint32_t)q + 1u);
}

// §3 item 6 steps 4-5, one thread per target pixel; MAXG >= G planes are held in registers (empty slots = -1).
template <int MAXG>
__global__ void __launch_bounds__(256) k_fuse_consensus(const uint32_t* __restrict__ planes, int G, int W, size_t px, int tol, int min_support,
                                                        const uint8_t* __restrict__ mask, uint16_t* __restrict__ out_disp,
                                                        float* __restrict__ out_sub, uint8_t* __restrict__ out_support) {
    const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i >= px) return;
    int c[MAXG];
#pragma unroll
    for (int g = 0; g < MAXG; g++) c[g] = g < G ? (int)planes[g * px + i] - 1 : -1;
    int best = -1, best_n = 0;
#pragma unroll
    for (int g = 0; g < MAXG; g++) {
        if (c[g] < 0) continue;
        int n = 0;
#pragma unroll
        for (int h = 0; h < MAXG; h++) n += c[h] >= 0 && abs(c[h] - c[g]) <= tol;
        if (n > best_n || (n == best_n && c[g] > best)) { best = c[g]; best_n = n; }
    }
    int sum = 0;
#pragma unroll
    for (int h = 0; h < MAXG; h++)
        if (c[h] >= 0 && abs(c[h] - best) <= tol) sum += c[h];
    const bool ok = best_n > 0 && best_n >= min_support && (!mask || mask[i] != 0);
    const int qh = ok ? (sum + best_n / 2) / best_n : 0;
    out_disp[i] = ok ? (uint16_t)((qh + 8) >> 4) : (uint16_t)SVA_DISP_INVALID;
    out_sub[i] = ok ? (float)qh / 16.0f : SVA_SUBPIX_INVALID;
    out_support[i] = (uint8_t)best_n;
}

// ---- host side, shared by sva_fuse_maps (below) and sva_depth_groups_fused (sva_groups.cu) ----

static size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

// Every refusal that concerns the fusion itself (SVA_ERR_BAD_ARG; nothing touched).
int sva_fuse_check(sva_ctx* c, int W, int H, int grid_cols, int n_cameras, const int32_t* refs, int n_views, int target, const sva_fuse_params* f,
                   const sva_image_u8* mask) {
    if (!f) return c->fail(SVA_ERR_BAD_ARG, "fuse: null fuse parameters");
    if (n_views < 1 || n_views > SVA_MAX_PAIRS) return c->fail(SVA_ERR_BAD_ARG, "fuse: n_views must be in 1..32");
    if (W < 1 || H < 1) return c->fail(SVA_ERR_BAD_ARG, "fuse: empty image");
    if (grid_cols < 1 || n_cameras < 1 || n_cameras % grid_cols) return c->fail(SVA_ERR_BAD_ARG, "fuse: n_cameras must be a positive multiple of grid_cols");
    if (!refs) return c->fail(SVA_ERR_BAD_ARG, "fuse: null view_refs");
    for (int g = 0; g < n_views; g++)
        if (refs[g] < 0 || refs[g] >= n_cameras) return c->fail(SVA_ERR_BAD_ARG, "fuse: reference of view " + std::to_string(g) + " outside [0, n_cameras)");
    if (target < 0 || target >= n_cameras) return c->fail(SVA_ERR_BAD_ARG, "fuse: target outside [0, n_cameras)");
    if (f->tol_16 < 0 || f->tol_16 > 4095) return c->fail(SVA_ERR_BAD_ARG, "fuse: tol_16 must be in 0..4095");
    if (f->min_support < 1 || f->min_support > n_views) return c->fail(SVA_ERR_BAD_ARG, "fuse: min_support must be in 1..n_views");
    for (int i = 0; i < 6; i++)
        if (f->reserved[i]) return c->fail(SVA_ERR_BAD_ARG, "fuse: non-zero reserved fields");
    if (mask && (!mask->data || mask->cols != W || mask->rows != H || mask->step < (size_t)W))
        return c->fail(SVA_ERR_BAD_ARG, "fuse: target mask is not width x height");
    return SVA_OK;
}

// Workspaces for G views of W x H, and the planes zeroed, on c->stream.
int sva_fuse_begin(sva_ctx* c, int W, int H, int G, bool has_mask) {
    const size_t px = (size_t)W * H;
    SVA_TRY(c->reserve(c->fuse_planes, px * G * sizeof(uint32_t)));
    SVA_TRY(c->reserve(c->fuse_out, align256(px * 2) + px * 5));  // disp u16, then subpix f32 (256-byte aligned), then support u8
    if (has_mask) SVA_TRY(c->reserve(c->fuse_mask, px));
    SVA_CUDA_OK(c, cudaMemsetAsync(c->fuse_planes.p, 0, px * G * sizeof(uint32_t), c->stream));
    return SVA_OK;
}

// Views [v0, v0 + n) of the planes from n maps at disp / sub + k * view_stride (sub == nullptr: integer maps), offsets gx / gy[k].
int sva_fuse_splat(sva_ctx* c, int W, int H, const uint16_t* disp, const float* sub, size_t view_stride, int v0, int n, const int* gx, const int* gy) {
    FuseOffsets off{};
    for (int k = 0; k < n; k++) { off.gx[k] = gx[k]; off.gy[k] = gy[k]; }
    LaunchScope ls(c, "k_fuse_splat");
    const size_t px = (size_t)W * H;
    k_fuse_splat<<<dim3((unsigned)((px + 255) / 256), n), 256, 0, c->stream>>>(disp, sub, view_stride, off, W, H, c->fuse_planes.as<uint32_t>() + v0 * px);
    SVA_CUDA_OK(c, cudaGetLastError());
    return SVA_OK;
}

// The vote over G planes, then the requested outputs into host memory; returns once they are there.
int sva_fuse_finish(sva_ctx* c, int W, int H, int G, const sva_fuse_params* f, const sva_image_u8* mask, uint16_t* out_disp, float* out_sub,
                    uint8_t* out_support) {
    const size_t px = (size_t)W * H;
    if (mask) SVA_CUDA_OK(c, cudaMemcpy2DAsync(c->fuse_mask.p, W, mask->data, mask->step, W, H, cudaMemcpyHostToDevice, c->stream));
    uint8_t* o = c->fuse_out.as<uint8_t>();
    uint16_t* d_disp = (uint16_t*)o;
    float* d_sub = (float*)(o + align256(px * 2));
    uint8_t* d_sup = (uint8_t*)(d_sub + px);
    const uint8_t* d_mask = mask ? c->fuse_mask.as<uint8_t>() : nullptr;
    const unsigned blocks = (unsigned)((px + 255) / 256);
    {
        LaunchScope ls(c, "k_fuse_consensus");
        const uint32_t* pl = c->fuse_planes.as<uint32_t>();
        if (G <= 8) k_fuse_consensus<8><<<blocks, 256, 0, c->stream>>>(pl, G, W, px, f->tol_16, f->min_support, d_mask, d_disp, d_sub, d_sup);
        else if (G <= 16) k_fuse_consensus<16><<<blocks, 256, 0, c->stream>>>(pl, G, W, px, f->tol_16, f->min_support, d_mask, d_disp, d_sub, d_sup);
        else k_fuse_consensus<32><<<blocks, 256, 0, c->stream>>>(pl, G, W, px, f->tol_16, f->min_support, d_mask, d_disp, d_sub, d_sup);
        SVA_CUDA_OK(c, cudaGetLastError());
    }
    SVA_CUDA_OK(c, cudaMemcpyAsync(out_disp, d_disp, px * 2, cudaMemcpyDeviceToHost, c->stream));
    if (out_sub) SVA_CUDA_OK(c, cudaMemcpyAsync(out_sub, d_sub, px * 4, cudaMemcpyDeviceToHost, c->stream));
    if (out_support) SVA_CUDA_OK(c, cudaMemcpyAsync(out_support, d_sup, px, cudaMemcpyDeviceToHost, c->stream));
    SVA_CUDA_OK(c, cudaStreamSynchronize(c->stream));
    return SVA_OK;
}

extern "C" int sva_fuse_maps(sva_ctx* c, int32_t W, int32_t H, int32_t grid_cols, int32_t n_cameras, const int32_t* refs, int32_t G,
                             const uint16_t* const* disp, const float* const* subpix, int32_t target, const sva_fuse_params* f,
                             const sva_image_u8* mask, uint16_t* out_disp, float* out_subpix, uint8_t* out_support) {
    if (!c) return SVA_ERR_BAD_ARG;
    SVA_TRY(sva_fuse_check(c, W, H, grid_cols, n_cameras, refs, G, target, f, mask));
    if (!disp || !out_disp) return c->fail(SVA_ERR_BAD_ARG, "fuse: null disp / out_disp");
    for (int g = 0; g < G; g++)
        if (!disp[g] || (subpix && !subpix[g])) return c->fail(SVA_ERR_BAD_ARG, "fuse: null map of view " + std::to_string(g));
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    const size_t px = (size_t)W * H;
    SVA_TRY(c->reserve(c->fuse_in, align256(px * G * 2) + (subpix ? px * G * 4 : 0)));  // G disp maps, then G subpix maps
    SVA_TRY(sva_fuse_begin(c, W, H, G, mask != nullptr));
    uint16_t* d_disp = c->fuse_in.as<uint16_t>();
    float* d_sub = subpix ? (float*)(c->fuse_in.as<uint8_t>() + align256(px * G * 2)) : nullptr;
    int gx[SVA_MAX_PAIRS], gy[SVA_MAX_PAIRS];
    for (int g = 0; g < G; g++) {
        SVA_CUDA_OK(c, cudaMemcpyAsync(d_disp + px * g, disp[g], px * 2, cudaMemcpyHostToDevice, c->stream));
        if (subpix) SVA_CUDA_OK(c, cudaMemcpyAsync(d_sub + px * g, subpix[g], px * 4, cudaMemcpyHostToDevice, c->stream));
        gx[g] = target % grid_cols - refs[g] % grid_cols;
        gy[g] = target / grid_cols - refs[g] / grid_cols;
    }
    SVA_TRY(sva_fuse_splat(c, W, H, d_disp, d_sub, px, 0, G, gx, gy));
    return sva_fuse_finish(c, W, H, G, f, mask, out_disp, out_subpix, out_support);
}
