// sva_ctx.cu — context lifetime, HBM workspaces, event-based kernel timing.
#include <cerrno>
#include <climits>
#include <cstdio>
#include <cstdlib>

#include "sva_common.cuh"

// Debug guard bands (sva_debug_set_guard): compute-sanitizer is not always available on a GPU box, so the library can check itself.
// A guarded allocation is [GUARD_BYTES canary][payload, poisoned][GUARD_BYTES canary]; sva_debug_check_guards counts canary bytes
// that changed (an out-of-bounds write), and the poison makes a read of never-written memory show up as a parity failure instead of
// passing on the zeros a fresh cudaMalloc usually returns.
void sva_dist_release(sva_ctx* c);  // sva_dist.cu: communicator and row-block link

static constexpr size_t GUARD_BYTES = 256 << 10;
static constexpr int GUARD_CANARY = 0xA5, GUARD_POISON = 0xCD;

__global__ void k_guard_count(const uint8_t* __restrict__ p, size_t n, unsigned long long* bad) {
    unsigned long long local = 0;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) local += p[i] != GUARD_CANARY;
    if (local) atomicAdd(bad, local);
}

void sva_ctx::release(DevBuf& b) {
    if (b.p) cudaFree(b.base ? b.base : b.p);
    b.p = b.base = nullptr;
    b.bytes = 0;
}

void sva_ctx::device_bufs(std::vector<DevBuf*>& out) {
    out = {&ref_img, &other_imgs, &lines, &mask, &A, &AP, &pad_imgs, &pad_ref, &C, &Craw, &S, &disp, &subpix, &other_d, &scratch, &scratch2, &pace_buf, &comm_scratch, &census, &tex_img, &sgm_state, &cam_stack, &cam_sig,
           &fuse_planes, &fuse_in, &fuse_mask, &fuse_out,
           &alt.pad_ref, &alt.pad_imgs, &alt.ref_img, &alt.other_imgs, &alt.lines, &alt.mask, &alt.disp, &alt.subpix};
}

int sva_ctx::reserve(DevBuf& b, size_t bytes) {
    if (b.bytes >= bytes && b.p) return SVA_OK;
    if (b.p) {
        cudaStreamSynchronize(stream);
        release(b);
    }
    size_t want = (bytes + 255) & ~(size_t)255;
    void* raw = nullptr;
    cudaError_t e = cudaMalloc(&raw, want + (guard ? 2 * GUARD_BYTES : 0));
    if (e != cudaSuccess)
        return fail(e == cudaErrorMemoryAllocation ? SVA_ERR_NOMEM : SVA_ERR_CUDA, std::string("cudaMalloc: ") + cudaGetErrorString(e));
    if (guard) {
        cudaMemsetAsync(raw, GUARD_CANARY, want + 2 * GUARD_BYTES, stream);
        cudaMemsetAsync((uint8_t*)raw + GUARD_BYTES, GUARD_POISON, want, stream);
        b.base = raw;
        b.p = (uint8_t*)raw + GUARD_BYTES;
    } else {
        b.base = nullptr;
        b.p = raw;
    }
    b.bytes = want;
    return SVA_OK;
}

int sva_ctx::reserve_pinned(DevBuf& b, size_t bytes) {
    if (b.bytes >= bytes && b.p) return SVA_OK;
    if (b.p) { cudaStreamSynchronize(stream); cudaFreeHost(b.p); b.p = nullptr; b.bytes = 0; }
    cudaError_t e = cudaMallocHost(&b.p, bytes);
    if (e != cudaSuccess) { b.p = nullptr; return fail(SVA_ERR_NOMEM, std::string("cudaMallocHost: ") + cudaGetErrorString(e)); }
    b.bytes = bytes;
    return SVA_OK;
}

void sva_ctx::time_begin(const char* name) {
    while (event_pool.size() < events_used + 2) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        event_pool.push_back(e);
    }
    KernelTime kt{name, event_pool[events_used], event_pool[events_used + 1]};
    events_used += 2;
    cudaEventRecord(kt.beg, stream);
    ktimes.push_back(kt);
}

void sva_ctx::time_end() { cudaEventRecord(ktimes.back().end, stream); }

// why the last sva_create of this thread failed (sva_last_error(NULL))
static thread_local std::string create_err;

// A whole number in [lo, hi] (surrounding blanks allowed), or false: atoi would read a typo as 0 and run another variant without a word.
bool sva_parse_env_int(const char* s, long long lo, long long hi, long long* out) {
    if (!s) return false;
    errno = 0;
    char* end = nullptr;
    const long long v = strtoll(s, &end, 10);
    if (end == s || errno == ERANGE) return false;
    while (*end == ' ' || *end == '\t') end++;
    if (*end != '\0' || v < lo || v > hi) return false;
    *out = v;
    return true;
}

// One A/B switch of DESIGN §8a: unset keeps the default; a value outside [lo, hi], or equal to hole, is refused.
static bool read_switch(const char* name, int& field, int lo, int hi, const char* allowed, int hole = INT_MIN) {
    const char* e = getenv(name);
    if (!e) return true;
    long long v = 0;
    if (!sva_parse_env_int(e, lo, hi, &v) || v == hole) {
        create_err = std::string(name) + "=" + e + " is not valid (allowed: " + allowed + ")";
        return false;
    }
    field = (int)v;
    return true;
}

static bool read_switches(sva_ctx* c) {
    return read_switch("SVA_SGM_PACE", c->tune_sgm_pace, -1, 1, "-1, 0, 1")
           && read_switch("SVA_SGM_PACE_WINDOW", c->tune_sgm_pace_window, 1, 1 << 20, "1 or more")
           && read_switch("SVA_SGM_HSTORE", c->tune_sgm_hstore, 1, 2, "1, 2")
           && read_switch("SVA_STREAM_AD_AHEAD", c->tune_stream_ad_ahead, 0, 2, "0, 1, 2")
           && read_switch("SVA_PREZERO", c->tune_prezero, 0, 1, "0, 1")
           && read_switch("SVA_WTA_SEG", c->tune_wta_seg, -1, 1 << 16, "-1, 0, or a segment length up to 65536")
           && read_switch("SVA_AD_GATHER", c->tune_ad_gather, 0, 1, "0, 1")
           && read_switch("SVA_AD_SET", c->tune_ad_set, 0, 1, "0, 1")
           && read_switch("SVA_AD_TH", c->tune_ad_th, 0, 1 << 16, "0, or rows per tile up to 65536")
           && read_switch("SVA_BOX_SHFL", c->tune_box_shfl, 0, 1, "0, 1")
           && read_switch("SVA_BOX_BANDS", c->tune_box_bands, 0, 1 << 20, "0, or a band count")
           && read_switch("SVA_BOX_OCC", c->tune_box_occ, 0, 3, "0, 2, 3", 1);  // K1b exists for 2 and 3 CTAs per SM
}

extern "C" {

int sva_api_version(void) { return SVA_API_VERSION; }

int sva_create(int device, sva_ctx** out) {
    create_err.clear();
    if (!out) return SVA_ERR_BAD_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) { create_err = "no such CUDA device"; return SVA_ERR_NO_DEVICE; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return SVA_ERR_CUDA;
    if (prop.major != 10) { create_err = "not an sm_100 GPU"; return SVA_ERR_NO_DEVICE; }  // built for sm_100a only; there is no fallback path
    sva_ctx* c = new sva_ctx();
    if (!read_switches(c)) { delete c; return SVA_ERR_BAD_ARG; }
    if (cudaSetDevice(device) != cudaSuccess) { delete c; return SVA_ERR_CUDA; }
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return SVA_ERR_CUDA; }
    c->stream = c->own_stream;
    *out = c;
    return SVA_OK;
}

int sva_destroy(sva_ctx* c) {
    if (!c) return SVA_ERR_BAD_ARG;
    cudaSetDevice(c->device);
    if (c->stream == c->own_stream) cudaStreamSynchronize(c->stream);
    else cudaDeviceSynchronize();  // a borrowed stream (sva_set_stream) may already be gone: never touch its handle here
    sva_dist_release(c);
    if (c->tex) cudaDestroyTextureObject((cudaTextureObject_t)c->tex);
    if (c->aux_stream) cudaStreamSynchronize(c->aux_stream);
    if (c->h2d_stream) { cudaStreamSynchronize(c->h2d_stream); cudaStreamSynchronize(c->d2h_stream); }
    if (c->ad_stream) cudaStreamSynchronize(c->ad_stream);
    if (c->stack_stream) cudaStreamSynchronize(c->stack_stream);
    std::vector<DevBuf*> bufs;
    c->device_bufs(bufs);
    for (DevBuf* b : bufs) c->release(*b);
    if (c->h2d_stream) {
        cudaStreamDestroy(c->h2d_stream); cudaStreamDestroy(c->d2h_stream); cudaEventDestroy(c->ev_mark);
        for (int i = 0; i < 2; i++) { cudaEventDestroy(c->ev_h2d[i]); cudaEventDestroy(c->ev_compute[i]); cudaEventDestroy(c->ev_done[i]); }
    }
    if (c->staging_host.p) cudaFreeHost(c->staging_host.p);
    for (cudaEvent_t e : c->event_pool) cudaEventDestroy(e);
    if (c->aux_stream) { cudaStreamDestroy(c->aux_stream); cudaEventDestroy(c->ev_fork); }
    if (c->ev_zero) cudaEventDestroy(c->ev_zero);
    if (c->ad_stream) { cudaStreamDestroy(c->ad_stream); cudaEventDestroy(c->ev_ad); cudaEventDestroy(c->ev_box); }
    if (c->stack_stream) cudaStreamDestroy(c->stack_stream);
    for (cudaEvent_t e : c->ev_cam) cudaEventDestroy(e);
    cudaStreamDestroy(c->own_stream);
    delete c;
    return SVA_OK;
}

const char* sva_last_error(const sva_ctx* c) { return c ? c->err.c_str() : !create_err.empty() ? create_err.c_str() : "null context"; }

int sva_set_stream(sva_ctx* c, void* s) {  // NULL = the legacy default stream (what torch.cuda.current_stream() usually is)
    if (!c) return SVA_ERR_BAD_ARG;
    cudaStreamSynchronize(c->stream);
    c->stream = (cudaStream_t)s;
    return SVA_OK;
}

int sva_use_own_stream(sva_ctx* c) {
    if (!c) return SVA_ERR_BAD_ARG;
    cudaStreamSynchronize(c->stream);
    c->stream = c->own_stream;
    return SVA_OK;
}

int sva_get_stream(sva_ctx* c, void** out) {
    if (!c || !out) return SVA_ERR_BAD_ARG;
    *out = (void*)c->stream;
    return SVA_OK;
}

int sva_synchronize(sva_ctx* c) {
    if (!c) return SVA_ERR_BAD_ARG;
    SVA_CUDA_OK(c, cudaStreamSynchronize(c->stream));
    return SVA_OK;
}

int sva_debug_set_guard(sva_ctx* c, int on) {  // applies to allocations made from now on
    if (!c) return SVA_ERR_BAD_ARG;
    c->guard = on != 0;
    return SVA_OK;
}

int sva_debug_check_guards(sva_ctx* c, int64_t* guarded_buffers, int64_t* bad_bytes) {
    if (!c || !guarded_buffers || !bad_bytes) return c ? c->fail(SVA_ERR_BAD_ARG, "check_guards: null argument") : SVA_ERR_BAD_ARG;
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    SVA_CUDA_OK(c, cudaDeviceSynchronize());
    unsigned long long* d_bad = nullptr;
    SVA_CUDA_OK(c, cudaMalloc(&d_bad, sizeof *d_bad));
    cudaMemsetAsync(d_bad, 0, sizeof *d_bad, c->stream);
    std::vector<DevBuf*> bufs;
    c->device_bufs(bufs);
    int64_t n = 0;
    for (DevBuf* b : bufs) {
        if (!b->p || !b->base) continue;
        n++;
        k_guard_count<<<64, 256, 0, c->stream>>>((const uint8_t*)b->base, GUARD_BYTES, d_bad);
        k_guard_count<<<64, 256, 0, c->stream>>>((const uint8_t*)b->p + b->bytes, GUARD_BYTES, d_bad);
    }
    unsigned long long bad = 0;
    cudaError_t e = cudaMemcpyAsync(&bad, d_bad, sizeof bad, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cudaFree(d_bad);
    SVA_CUDA_OK(c, e);
    *guarded_buffers = n;
    *bad_bytes = (int64_t)bad;
    return SVA_OK;
}

int sva_kernel_launches(const sva_ctx* c, uint64_t* out) {
    if (!c || !out) return SVA_ERR_BAD_ARG;
    *out = c->launches;
    return SVA_OK;
}

}  // extern "C"
