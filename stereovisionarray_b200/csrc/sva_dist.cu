// sva_dist.cu — multi-GPU entry points of the C ABI (one process per GPU): an NCCL communicator loaded at run time, the packed-u32 reduce of
// the pair-sharded AD volume, and the row-block pipeline whose path-line state crosses GPUs by PEER-DIRECT stores (CUDA IPC over NVLink)
// sequenced by device-side flags instead of host-sequenced NCCL send / recv.
//
// No reference counterpart (the reference is one thread on one CPU, SURVEY §0.1).  Sharding units: the pair loop
// src/CameraStereoVision.cpp:55 and the pixel-row loop src/CameraStereoVision.cpp:49.
#include <dlfcn.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>

#include <nvtx3/nvToolsExt.h>

#include "sva_common.cuh"

// ---- NCCL through dlopen: the few entry points used, declared here so that neither nccl.h nor libnccl is needed to build or load the library ----
namespace {
struct NcclUid { char internal[128]; };
typedef void* NcclComm;
enum { NCCL_UINT8 = 1, NCCL_UINT32 = 3, NCCL_SUM = 0 };  // ncclDataType_t / ncclRedOp_t values of nccl.h (stable since NCCL 2.0)
struct NcclApi {
    void* h = nullptr;
    int (*GetUniqueId)(NcclUid*) = nullptr;
    int (*CommInitRank)(NcclComm*, int, NcclUid, int) = nullptr;
    int (*CommDestroy)(NcclComm) = nullptr;
    int (*Reduce)(const void*, void*, size_t, int, int, int, NcclComm, cudaStream_t) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, NcclComm, cudaStream_t) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, NcclComm, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    std::string err;
};

NcclApi* nccl() {
    static NcclApi api;
    if (api.h || !api.err.empty()) return &api;
    // RTLD_NOLOAD first: a process that already carries an NCCL (torch bundles one) must use THAT copy.  Otherwise SVA_NCCL_LIB names the
    // library, else the system's libnccl.so.2 — loaded RTLD_LOCAL so that it does not satisfy another module's NCCL dependency by accident
    // (a torch imported LATER would bind to it by SONAME all the same: the Python host therefore preloads torch's copy, _lib.py).
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
    if (!h && getenv("SVA_NCCL_LIB")) h = dlopen(getenv("SVA_NCCL_LIB"), RTLD_NOW | RTLD_LOCAL);
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_LOCAL);
    if (!h) { api.err = std::string("dlopen(libnccl.so.2): ") + dlerror(); return &api; }
    bool ok = true;
    auto sym = [&](const char* n) { void* p = dlsym(h, n); if (!p) { ok = false; api.err = std::string("libnccl.so.2 lacks ") + n; } return p; };
    *(void**)&api.GetUniqueId = sym("ncclGetUniqueId");
    *(void**)&api.CommInitRank = sym("ncclCommInitRank");
    *(void**)&api.CommDestroy = sym("ncclCommDestroy");
    *(void**)&api.Reduce = sym("ncclReduce");
    *(void**)&api.AllReduce = sym("ncclAllReduce");
    *(void**)&api.AllGather = sym("ncclAllGather");
    *(void**)&api.GetErrorString = sym("ncclGetErrorString");
    if (ok) api.h = h;
    return &api;
}
}  // namespace

#define SVA_NCCL_OK(ctx, expr)                                                                                            \
    do {                                                                                                                  \
        int r__ = (expr);                                                                                                 \
        if (r__ != 0) return (ctx)->fail(SVA_ERR_COMM, std::string(#expr) + ": " + nccl()->GetErrorString(r__));          \
    } while (0)

// ---- row-block link: the memory a neighbour writes into, and where this rank writes ------------------------------------------------
// layout of the link allocation: [flags: 8 x 128 B][down-state in: 3*W*D u16][up-state in: 3*W*D u16]
enum { F_D_READY = 0, F_U_READY = 1, F_D_ACK = 2, F_U_ACK = 3, F_ERR = 4, F_COUNT = 8 };
constexpr size_t FLAG_STRIDE = 128, FLAGS_BYTES = F_COUNT * FLAG_STRIDE;

struct RowsLink {
    int rank = -1, world = 0, W = 0, H = 0, D = 0;
    int y0 = 0, rows = 0;
    size_t state_bytes = 0;
    uint8_t* mem = nullptr;        // this rank's allocation (cudaMalloc: CUDA IPC exports whole allocations)
    uint8_t* prev = nullptr;       // neighbours' allocations as mapped here (nullptr at the array's ends)
    uint8_t* next = nullptr;
    bool prev_ipc = false, next_ipc = false;
    uint32_t seq = 0;              // frames enqueued so far
    int part_done = 2;             // last part of frame `seq` that was enqueued (2: the frame is complete — see sva_rows_run_part)
    long long timeout_ns = 20000LL * 1000000LL;
    uint32_t* flag(uint8_t* base, int i) const { return (uint32_t*)(base + (size_t)i * FLAG_STRIDE); }
    uint16_t* d_in(uint8_t* base) const { return (uint16_t*)(base + FLAGS_BYTES); }
    uint16_t* u_in(uint8_t* base) const { return (uint16_t*)(base + FLAGS_BYTES + state_bytes); }
};

// Holds the stream until *flag >= want (a neighbour's k_rows_signal), for at most timeout_ns: a neighbour that died must not hang the GPU.
__global__ void k_rows_wait(const uint32_t* flag, uint32_t want, long long timeout_ns, uint32_t* err) {
    unsigned long long t0, t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
        uint32_t v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
        if ((int32_t)(v - want) >= 0) return;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        if ((long long)(t - t0) > timeout_ns) { atomicExch(err, 1u); return; }
        __nanosleep(256);
    }
}

// Publishes `value` in a flag that lives in a neighbour's memory.  Stream order has completed the march that wrote the state before this
// kernel starts; the fence orders those peer writes before the flag for an observer at system scope.
__global__ void k_rows_signal(uint32_t* flag, uint32_t value) {
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(flag), "r"(value) : "memory");
}

static void link_unmap(RowsLink* l) {
    if (l->prev && l->prev_ipc) cudaIpcCloseMemHandle(l->prev);
    if (l->next && l->next_ipc) cudaIpcCloseMemHandle(l->next);
    l->prev = l->next = nullptr;
    l->prev_ipc = l->next_ipc = false;
}

void sva_dist_release(sva_ctx* c) {  // from sva_destroy
    if (c->rows_link) {
        RowsLink* l = (RowsLink*)c->rows_link;
        link_unmap(l);
        if (l->mem) cudaFree(l->mem);
        delete l;
        c->rows_link = nullptr;
    }
    if (c->comm) {
        if (nccl()->h) nccl()->CommDestroy((NcclComm)c->comm);
        c->comm = nullptr;
    }
}

static void pair_range(int n_pairs, int world, int rank, int& b, int& e) {  // balanced contiguous ranges: the first n % world ranks get one more
    const int base = n_pairs / world, extra = n_pairs % world;
    b = rank * base + std::min(rank, extra);
    e = b + base + (rank < extra ? 1 : 0);
}

extern "C" {

int sva_comm_get_unique_id(uint8_t out_id[SVA_COMM_ID_BYTES]) {
    if (!out_id) return SVA_ERR_BAD_ARG;
    NcclApi* n = nccl();
    if (!n->h) return SVA_ERR_COMM;
    NcclUid id;
    if (n->GetUniqueId(&id) != 0) return SVA_ERR_COMM;
    static_assert(sizeof id == SVA_COMM_ID_BYTES, "ncclUniqueId is 128 bytes");
    memcpy(out_id, &id, sizeof id);
    return SVA_OK;
}

int sva_comm_init(sva_ctx* c, const uint8_t id[SVA_COMM_ID_BYTES], int32_t rank, int32_t world) {
    if (!c || !id) return SVA_ERR_BAD_ARG;
    if (world < 1 || rank < 0 || rank >= world) return c->fail(SVA_ERR_BAD_ARG, "comm_init: bad rank / world");
    if (c->comm) return c->fail(SVA_ERR_STATE, "comm_init: the context already has a communicator");
    NcclApi* n = nccl();
    if (!n->h) return c->fail(SVA_ERR_COMM, n->err);
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    NcclUid uid;
    memcpy(&uid, id, sizeof uid);
    NcclComm comm = nullptr;
    SVA_NCCL_OK(c, n->CommInitRank(&comm, world, uid, rank));
    c->comm = comm; c->comm_rank = rank; c->comm_world = world;
    return SVA_OK;
}

int sva_comm_destroy(sva_ctx* c) {
    if (!c) return SVA_ERR_BAD_ARG;
    if (!c->comm) return SVA_OK;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    nccl()->CommDestroy((NcclComm)c->comm);
    c->comm = nullptr;
    return SVA_OK;
}

int sva_comm_barrier(sva_ctx* c) {
    if (!c) return SVA_ERR_BAD_ARG;
    if (!c->comm) return c->fail(SVA_ERR_STATE, "no communicator (sva_comm_init)");
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    SVA_TRY(c->reserve(c->comm_scratch, 256));
    SVA_CUDA_OK(c, cudaMemsetAsync(c->comm_scratch.p, 0, 4, c->stream));
    SVA_NCCL_OK(c, nccl()->AllReduce(c->comm_scratch.p, c->comm_scratch.p, 1, NCCL_UINT32, NCCL_SUM, (NcclComm)c->comm, c->stream));
    SVA_CUDA_OK(c, cudaStreamSynchronize(c->stream));
    return SVA_OK;
}

int sva_frame_ad_device_ptr(sva_ctx* ctx, void** out_ptr, size_t* out_bytes);

int sva_frame_reduce_ad(sva_ctx* c, int32_t root) {
    if (!c) return SVA_ERR_BAD_ARG;
    if (!c->comm) return c->fail(SVA_ERR_STATE, "no communicator (sva_comm_init)");
    if (root < 0 || root >= c->comm_world) return c->fail(SVA_ERR_BAD_ARG, "reduce_ad: bad root");
    if (255 * c->prm.n_pairs >= (1 << 16)) return c->fail(SVA_ERR_BAD_ARG, "reduce_ad: too many pairs for a carry-free packed sum");
    void* ptr = nullptr;
    size_t bytes = 0;
    SVA_TRY(sva_frame_ad_device_ptr(c, &ptr, &bytes));  // planar layout incl. its zero borders: zeros add up to zero
    SVA_NCCL_OK(c, nccl()->Reduce(ptr, ptr, bytes / 4, NCCL_UINT32, NCCL_SUM, root, (NcclComm)c->comm, c->stream));
    if (c->comm_rank == root) SVA_TRY(sva_frame_mark_ad_ready(c));
    return SVA_OK;
}

int sva_depth_pair_sharded(sva_ctx* c, const sva_params* p, const sva_image_u8* ref, const sva_image_u8* others, const sva_image_u8* mask,
                           int32_t root, uint16_t* out_disp, float* out_subpix) {
    if (!c) return SVA_ERR_BAD_ARG;
    if (!c->comm) return c->fail(SVA_ERR_STATE, "no communicator (sva_comm_init)");
    SVA_TRY(sva_frame_upload(c, p, ref, others, mask));
    int b, e;
    pair_range(p->n_pairs, c->comm_world, c->comm_rank, b, e);
    SVA_TRY(sva_frame_set_pair_range(c, b, e));
    SVA_TRY(sva_frame_run(c, SVA_STAGE_AD));  // an empty range zero-fills the partial
    SVA_TRY(sva_frame_reduce_ad(c, root));
    if (c->comm_rank != root) { SVA_CUDA_OK(c, cudaStreamSynchronize(c->stream)); return SVA_OK; }
    if (!out_disp) return c->fail(SVA_ERR_BAD_ARG, "pair_sharded: root needs out_disp");
    SVA_TRY(sva_frame_set_pair_range(c, 0, p->n_pairs));
    SVA_TRY(sva_frame_run(c, SVA_STAGE_BOX));
    SVA_TRY(sva_frame_run(c, SVA_STAGE_SGM));
    return sva_frame_download_disparity(c, out_disp, out_subpix);
}

// ---- row-block pipeline ------------------------------------------------------------------------------------------------------------
int sva_rows_close(sva_ctx* c) {
    if (!c) return SVA_ERR_BAD_ARG;
    if (!c->rows_link) return SVA_OK;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    RowsLink* l = (RowsLink*)c->rows_link;
    link_unmap(l);
    if (l->mem) cudaFree(l->mem);
    delete l;
    c->rows_link = nullptr;
    return SVA_OK;
}

int sva_rows_open(sva_ctx* c, const sva_params* p, int32_t rank, int32_t world) {
    if (!c || !p) return SVA_ERR_BAD_ARG;
    if (world < 1 || rank < 0 || rank >= world) return c->fail(SVA_ERR_BAD_ARG, "rows_open: bad rank / world");
    if (p->n_paths != 8) return c->fail(SVA_ERR_BAD_ARG, "rows_open: the row-block pipeline aggregates 8 paths");
    const int rows_per = (p->height + world - 1) / world;
    if ((long long)rows_per * (world - 1) >= p->height) return c->fail(SVA_ERR_BAD_ARG, "rows_open: fewer image rows than the ranks need (every rank owns at least one row)");
    long long timeout_ms = 0;
    const char* te = getenv("SVA_ROWS_TIMEOUT_MS");
    if (te && !sva_parse_env_int(te, 1, 1LL << 40, &timeout_ms))  // 0 or text would be a time-out that fires at once
        return c->fail(SVA_ERR_BAD_ARG, std::string("rows_open: SVA_ROWS_TIMEOUT_MS=") + te + " is not valid (allowed: milliseconds, 1 or more)");
    SVA_TRY(sva_rows_close(c));
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    RowsLink* l = new RowsLink();
    l->rank = rank; l->world = world; l->W = p->width; l->H = p->height; l->D = p->num_disp;
    l->y0 = rank * rows_per; l->rows = std::min(p->height, (rank + 1) * rows_per) - l->y0;
    l->state_bytes = (((size_t)3 * p->width * p->num_disp * sizeof(uint16_t)) + 255) & ~(size_t)255;
    if (te) l->timeout_ns = timeout_ms * 1000000LL;
    const size_t bytes = FLAGS_BYTES + 2 * l->state_bytes;
    cudaError_t e = cudaMalloc(&l->mem, bytes);
    if (e != cudaSuccess) { delete l; return c->fail(SVA_ERR_NOMEM, std::string("rows_open: cudaMalloc: ") + cudaGetErrorString(e)); }
    e = cudaMemsetAsync(l->mem, 0, FLAGS_BYTES, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) { cudaFree(l->mem); delete l; return c->fail(SVA_ERR_CUDA, std::string("rows_open: ") + cudaGetErrorString(e)); }
    c->rows_link = l;
    return SVA_OK;
}

int sva_rows_export(sva_ctx* c, uint8_t out_handle[SVA_IPC_HANDLE_BYTES]) {
    if (!c || !out_handle) return SVA_ERR_BAD_ARG;
    RowsLink* l = (RowsLink*)c->rows_link;
    if (!l) return c->fail(SVA_ERR_STATE, "rows_export: sva_rows_open first");
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    cudaIpcMemHandle_t h;
    static_assert(sizeof h == SVA_IPC_HANDLE_BYTES, "cudaIpcMemHandle_t is 64 bytes");
    SVA_CUDA_OK(c, cudaIpcGetMemHandle(&h, l->mem));
    memcpy(out_handle, &h, sizeof h);
    return SVA_OK;
}

int sva_rows_connect(sva_ctx* c, const uint8_t* prev_handle, const uint8_t* next_handle) {
    if (!c) return SVA_ERR_BAD_ARG;
    RowsLink* l = (RowsLink*)c->rows_link;
    if (!l) return c->fail(SVA_ERR_STATE, "rows_connect: sva_rows_open first");
    if ((l->rank > 0) != (prev_handle != nullptr) || (l->rank < l->world - 1) != (next_handle != nullptr))
        return c->fail(SVA_ERR_BAD_ARG, "rows_connect: exactly the neighbours that exist must be given (prev for rank > 0, next for rank < world - 1)");
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    link_unmap(l);
    auto open = [&](const uint8_t* hb, uint8_t** out) -> cudaError_t {
        cudaIpcMemHandle_t h;
        memcpy(&h, hb, sizeof h);
        void* p = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
        *out = (uint8_t*)p;
        return e;
    };
    if (prev_handle) {
        cudaError_t e = open(prev_handle, &l->prev);
        if (e != cudaSuccess) { l->prev = nullptr; return c->fail(SVA_ERR_COMM, std::string("rows_connect: cudaIpcOpenMemHandle(prev): ") + cudaGetErrorString(e)); }
        l->prev_ipc = true;
    }
    if (next_handle) {
        cudaError_t e = open(next_handle, &l->next);
        if (e != cudaSuccess) { l->next = nullptr; link_unmap(l); return c->fail(SVA_ERR_COMM, std::string("rows_connect: cudaIpcOpenMemHandle(next): ") + cudaGetErrorString(e)); }
        l->next_ipc = true;
    }
    return SVA_OK;
}

int sva_rows_connect_comm(sva_ctx* c) {
    if (!c) return SVA_ERR_BAD_ARG;
    RowsLink* l = (RowsLink*)c->rows_link;
    if (!l) return c->fail(SVA_ERR_STATE, "rows_connect_comm: sva_rows_open first");
    if (!c->comm) return c->fail(SVA_ERR_STATE, "no communicator (sva_comm_init)");
    if (l->rank != c->comm_rank || l->world != c->comm_world) return c->fail(SVA_ERR_BAD_ARG, "rows_connect_comm: the link was opened for another rank / world");
    const int G = l->world;
    std::vector<uint8_t> all((size_t)G * SVA_IPC_HANDLE_BYTES);
    SVA_TRY(sva_rows_export(c, all.data() + (size_t)l->rank * SVA_IPC_HANDLE_BYTES));
    SVA_TRY(c->reserve(c->comm_scratch, std::max<size_t>(256, all.size())));
    uint8_t* d = c->comm_scratch.as<uint8_t>();
    SVA_CUDA_OK(c, cudaMemcpyAsync(d + (size_t)l->rank * SVA_IPC_HANDLE_BYTES, all.data() + (size_t)l->rank * SVA_IPC_HANDLE_BYTES, SVA_IPC_HANDLE_BYTES, cudaMemcpyHostToDevice, c->stream));
    SVA_NCCL_OK(c, nccl()->AllGather(d + (size_t)l->rank * SVA_IPC_HANDLE_BYTES, d, SVA_IPC_HANDLE_BYTES, NCCL_UINT8, (NcclComm)c->comm, c->stream));
    SVA_CUDA_OK(c, cudaMemcpyAsync(all.data(), d, all.size(), cudaMemcpyDeviceToHost, c->stream));
    SVA_CUDA_OK(c, cudaStreamSynchronize(c->stream));
    return sva_rows_connect(c, l->rank > 0 ? all.data() + (size_t)(l->rank - 1) * SVA_IPC_HANDLE_BYTES : nullptr,
                            l->rank < G - 1 ? all.data() + (size_t)(l->rank + 1) * SVA_IPC_HANDLE_BYTES : nullptr);
}

int sva_rows_connect_local(sva_ctx* c, sva_ctx* prev, sva_ctx* next) {
    if (!c) return SVA_ERR_BAD_ARG;
    RowsLink* l = (RowsLink*)c->rows_link;
    if (!l) return c->fail(SVA_ERR_STATE, "rows_connect_local: sva_rows_open first");
    if ((l->rank > 0) != (prev != nullptr) || (l->rank < l->world - 1) != (next != nullptr))
        return c->fail(SVA_ERR_BAD_ARG, "rows_connect_local: exactly the neighbours that exist must be given");
    link_unmap(l);
    for (sva_ctx* o : {prev, next}) {
        if (!o) continue;
        RowsLink* ol = (RowsLink*)o->rows_link;
        if (!ol || ol->world != l->world || ol->W != l->W || ol->H != l->H || ol->D != l->D || ol->rank != l->rank + (o == prev ? -1 : 1))
            return c->fail(SVA_ERR_BAD_ARG, "rows_connect_local: the neighbour's link is not open for the adjacent rank of the same geometry");
        if (o->device != c->device) {  // one process driving several GPUs: plain peer access
            SVA_CUDA_OK(c, cudaSetDevice(c->device));
            cudaError_t e = cudaDeviceEnablePeerAccess(o->device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return c->fail(SVA_ERR_COMM, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
            cudaGetLastError();
        }
        (o == prev ? l->prev : l->next) = ol->mem;
    }
    return SVA_OK;
}

int sva_rows_run_phase(sva_ctx* c, int32_t phase);
int sva_rows_run_part(sva_ctx* c, int32_t part);

int sva_rows_block(const sva_ctx* c, int32_t* out_y0, int32_t* out_rows) {
    if (!c || !c->rows_link || !out_y0 || !out_rows) return SVA_ERR_BAD_ARG;
    const RowsLink* l = (const RowsLink*)c->rows_link;
    *out_y0 = l->y0; *out_rows = l->rows;
    return SVA_OK;
}

int sva_rows_run(sva_ctx* c) {
    SVA_TRY(sva_rows_run_phase(c, 0));
    return sva_rows_run_phase(c, 1);
}

// One frame in parts, so that a host with several contexts ON ONE STREAM can interleave frames without ever running two of the big
// kernels at once (concurrent launches break the resident, paced waves of the SGM marches: measured 2.5x slower):
//   part 0 = cost volume of the block (+ the horizontal paths on the ranks that do not start a sweep): nothing in it waits for a neighbour;
//   part 1 = the sweep that reaches this rank first (+ the horizontal paths on the two ranks that START a sweep, off the chain);
//   part 2 = the other sweep and K3.
// sva_rows_run_phase keeps the two-phase form (phase 0 = parts 0 + 1, phase 1 = part 2).  Enqueue order for P >= 3 frames in flight:
// part 0 of frame f, part 1 of frame f - 1, part 2 of frame f - P + 1 — every wait for a neighbour's state then sits behind a part 0 of
// a later frame, i.e. behind work that needs no neighbour.
int sva_rows_run_part(sva_ctx* c, int32_t part) {
    if (!c) return SVA_ERR_BAD_ARG;
    RowsLink* l = (RowsLink*)c->rows_link;
    if (!l) return c->fail(SVA_ERR_STATE, "rows_run: sva_rows_open first");
    if (part < 0 || part > 2) return c->fail(SVA_ERR_BAD_ARG, "rows_run_part: part must be 0, 1 or 2");
    if (part != (l->part_done + 1) % 3) return c->fail(SVA_ERR_STATE, "rows_run_part: the parts of a frame run in order 0, 1, 2");
    if (!c->have_frame) return c->fail(SVA_ERR_STATE, "no frame uploaded");
    const sva_params& p = c->prm;
    if (p.width != l->W || p.height != l->H || p.num_disp != l->D || p.n_paths != 8) return c->fail(SVA_ERR_STATE, "rows_run: the uploaded frame does not match the geometry of sva_rows_open");
    const int r = l->rank, G = l->world;
    if ((r > 0 && !l->prev) || (r < G - 1 && !l->next)) return c->fail(SVA_ERR_STATE, "rows_run: neighbours not connected (sva_rows_connect*)");
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    nvtxRangePushA("sva:rows_block");
    struct Pop { ~Pop() { nvtxRangePop(); } } pop;
    const uint32_t seq = part == 0 ? ++l->seq : l->seq;
    l->part_done = part;
    const int y0 = l->y0, n = l->rows;
    uint32_t* err = l->flag(l->mem, F_ERR);
    auto wait = [&](int f, uint32_t want) -> int {
        c->launches++;
        k_rows_wait<<<1, 1, 0, c->stream>>>(l->flag(l->mem, f), want, l->timeout_ns, err);
        SVA_CUDA_OK(c, cudaGetLastError());
        return SVA_OK;
    };
    auto signal = [&](uint8_t* peer, int f) -> int {
        c->launches++;
        k_rows_signal<<<1, 1, 0, c->stream>>>(l->flag(peer, f), seq);
        SVA_CUDA_OK(c, cudaGetLastError());
        return SVA_OK;
    };
    // one sweep on this block: the state arrives in this rank's memory, the state after the block's last row goes straight into the next
    // rank's memory.  The ack keeps a fast producer from overwriting a state its neighbour has not consumed yet (several frames in flight).
    auto sweep = [&](bool down) -> int {
        uint8_t* from = down ? l->prev : l->next;   // rank the sweep comes from
        uint8_t* to = down ? l->next : l->prev;     // rank the sweep goes to
        const int f_ready = down ? F_D_READY : F_U_READY, f_ack = down ? F_D_ACK : F_U_ACK;
        if (from) SVA_TRY(wait(f_ready, seq));
        if (to) SVA_TRY(wait(f_ack, seq - 1));
        const uint16_t* in = from ? (down ? l->d_in(l->mem) : l->u_in(l->mem)) : nullptr;
        uint16_t* out = to ? (down ? l->d_in(to) : l->u_in(to)) : nullptr;
        SVA_TRY(sva_frame_sgm_rows(c, down ? 0 : 1, y0, n, in, out));
        if (from) SVA_TRY(signal(from, f_ack));
        if (to) SVA_TRY(signal(to, f_ready));
        return SVA_OK;
    };
    // The sweeps are serial chains across the ranks (down: 0 -> G-1, up: G-1 -> 0).  Each rank takes first the sweep that reaches it first; the
    // two ranks that START a sweep do so right after their cost volume and run their horizontal paths afterwards, off the chain.
    const bool starts_chain = G > 1 && (r == 0 || r == G - 1);
    const bool down_first = r < (G + 1) / 2;
    if (part == 0) {
        SVA_TRY(sva_frame_rows_begin(c, y0, n));
        SVA_TRY(sva_frame_run(c, SVA_STAGE_AD));
        SVA_TRY(sva_frame_run(c, SVA_STAGE_BOX));
        if (!starts_chain) SVA_TRY(sva_frame_sgm_rows(c, 2, y0, n, nullptr, nullptr));
        return SVA_OK;
    }
    if (part == 1) {
        SVA_TRY(sweep(down_first));
        if (starts_chain) SVA_TRY(sva_frame_sgm_rows(c, 2, y0, n, nullptr, nullptr));
        return SVA_OK;
    }
    SVA_TRY(sweep(!down_first));
    return sva_frame_wta_rows(c, nullptr, y0, n);
}

int sva_rows_run_phase(sva_ctx* c, int32_t phase) {
    if (!c) return SVA_ERR_BAD_ARG;
    if (phase != 0 && phase != 1) return c->fail(SVA_ERR_BAD_ARG, "rows_run_phase: phase must be 0 or 1");
    if (phase == 0) {
        SVA_TRY(sva_rows_run_part(c, 0));
        return sva_rows_run_part(c, 1);
    }
    return sva_rows_run_part(c, 2);
}

int sva_rows_download(sva_ctx* c, uint16_t* out_disp_rows, float* out_subpix_rows) {
    if (!c || !out_disp_rows) return SVA_ERR_BAD_ARG;
    RowsLink* l = (RowsLink*)c->rows_link;
    if (!l) return c->fail(SVA_ERR_STATE, "rows_download: sva_rows_open first");
    SVA_TRY(sva_frame_download_disparity_rows(c, l->rows, out_disp_rows, out_subpix_rows));  // synchronises the stream
    uint32_t err = 0;
    SVA_CUDA_OK(c, cudaMemcpy(&err, l->flag(l->mem, F_ERR), sizeof err, cudaMemcpyDeviceToHost));
    if (err) {
        cudaMemset(l->flag(l->mem, F_ERR), 0, sizeof err);
        return c->fail(SVA_ERR_COMM, "rows: a neighbour's path-line state did not arrive within the time-out (SVA_ROWS_TIMEOUT_MS); the block's maps are not valid");
    }
    return SVA_OK;
}

int sva_depth_rows_sharded(sva_ctx* c, const sva_params* p, const sva_image_u8* ref, const sva_image_u8* others, const sva_image_u8* mask,
                           uint16_t* out_disp_rows, float* out_subpix_rows) {
    if (!c) return SVA_ERR_BAD_ARG;
    SVA_TRY(sva_frame_upload(c, p, ref, others, mask));
    SVA_TRY(sva_rows_run(c));
    return sva_rows_download(c, out_disp_rows, out_subpix_rows);
}

}  // extern "C"
