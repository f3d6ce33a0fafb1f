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

// ---- a stream of frames in the order skewed by chain position (sva_rows_stream_*) ------------------------------------------------------
// Iteration i of rank r enqueues part 0 of frame i, part 1 of frame i - lag1 and part 2 of frame i - lag2 (lag1 = 1 + min(r, G-1-r),
// lag2 = 1 + max(r, G-1-r) <= G), frame f on context f mod (G + 1) — dist.rows_skewed_order.  Every wait for a neighbour then depends on work
// the neighbour enqueued in an EARLIER iteration, so a host that blocks only on work at least two iterations old never blocks on work that is
// not enqueued yet, and the device never runs dry while the host enqueues.
//
// Three streams per rank: the contexts' compute stream, an upload stream and a download stream.  Per context:
//   images of frame f      uploaded after part 0 of the context's previous frame (K1a is their last reader);
//   mask of frame f        uploaded after part 2 of the context's previous frame (K3 is its only reader);
//   part 0 of frame f      waits for the images, part 2 of frame f for the mask.  (Ranks 0 and G-1 run the previous frame's part 2 at the end
//                          of the iteration just before the context is reused: an upload behind it would stall part 0 for the whole copy —
//                          measured at c3 on one B200, 19.6 -> 22.4 ms per frame.)
//   download of frame f    waits for part 2 of frame f, and copies the time-out flag with the rows;
//   part 2 of frame f + P  waits for that download — not part 0 or 1, for the same reason.
int check_frame_args(sva_ctx* c, const sva_params* p, const sva_image_u8* ref, const sva_image_u8* others, const sva_image_u8* mask);

struct sva_rows_stream {
    struct Slot {
        int64_t ticket = -1;
        bool retired = true;
        uint16_t* disp = nullptr;  // the caller's buffers of that ticket
        float* sub = nullptr;
    };
    std::vector<sva_ctx*> ctxs;            // borrowed; context j is link j of the chain
    std::vector<RowsLink*> links;          // the links the stream was created for (a context re-opened since is refused)
    sva_params p{};
    int rank = 0, world = 1, P = 2, lag1 = 1, lag2 = 1;
    size_t disp_bytes = 0, sub_bytes = 0;  // the block's rows of each map (the caller's buffers)
    size_t sub_at = 0, err_at = 0, slot_bytes = 0;  // layout of a staging slot
    cudaStream_t compute = nullptr, h2d = nullptr, d2h = nullptr;
    std::vector<cudaEvent_t> ev_img, ev_mask, ev_p0, ev_p2, ev_out;  // per context: images / mask uploaded, part 0 / part 2 done, download done
    std::vector<cudaEvent_t> ev_slot;               // per slot: the ticket's rows and flag are in the staging
    uint8_t* staging = nullptr;                     // pinned, per slot: [disp rows][subpix rows][time-out flag]
    std::vector<Slot> slots;                        // world + 2: a slot is reused by the ticket world + 2 later, whose part 2 is <= 2 iterations old
    int64_t next = 0;      // next ticket
    int64_t fill = 0;      // first ticket since the last flush
    int64_t finished = 0;  // tickets below this have part 2 and the download enqueued
    std::set<int64_t> failed;  // retired tickets whose context reported a hand-off time-out
    int fail(int code, const std::string& msg) { return ctxs[0]->fail(code, "rows_stream: " + msg); }
    int fwd(int j, int rc) {  // an error of context j, reported through ctxs[0]
        if (rc != SVA_OK && j != 0) ctxs[0]->err = "rows_stream (context " + std::to_string(j) + "): " + ctxs[j]->err;
        return rc;
    }
};

#define SVA_STREAM_CUDA_OK(s, expr)                                                                           \
    do {                                                                                                      \
        cudaError_t e__ = (expr);                                                                             \
        if (e__ != cudaSuccess) return (s)->fail(SVA_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__)); \
    } while (0)

static void rows_stream_release(sva_rows_stream* s) {
    for (cudaStream_t st : {s->h2d, s->d2h})
        if (st) { cudaStreamSynchronize(st); cudaStreamDestroy(st); }
    for (auto* v : {&s->ev_img, &s->ev_mask, &s->ev_p0, &s->ev_p2, &s->ev_out, &s->ev_slot})
        for (cudaEvent_t e : *v) if (e) cudaEventDestroy(e);
    if (s->staging) cudaFreeHost(s->staging);
    delete s;
}

// one context through the local stages of its block, so that every device buffer a frame of this geometry needs exists before the stream
// runs: an allocation inside submit would synchronise the device (a stall, and in a process that plays several ranks a dead-lock)
static int rows_stream_warm_up(sva_rows_stream* s, int j, const std::vector<uint8_t>& zeros) {
    sva_ctx* c = s->ctxs[j];
    RowsLink* l = s->links[j];
    const sva_image_u8 img{zeros.data(), s->p.height, s->p.width, (size_t)s->p.width};
    std::vector<sva_image_u8> others(s->p.n_pairs, img);
    for (const sva_image_u8* mask : {&img, (const sva_image_u8*)nullptr}) {
        SVA_TRY(sva_frame_upload(c, &s->p, &img, others.data(), mask));
        SVA_TRY(sva_frame_rows_begin(c, l->y0, l->rows));
        SVA_TRY(sva_frame_run(c, SVA_STAGE_AD));
        SVA_TRY(sva_frame_run(c, SVA_STAGE_BOX));
        SVA_TRY(sva_frame_sgm_rows(c, 2, l->y0, l->rows, nullptr, nullptr));
        // both sweeps, reading this link's own state buffers and storing nowhere: the paced launches size their pacing buffer here
        SVA_TRY(sva_frame_sgm_rows(c, 0, l->y0, l->rows, l->d_in(l->mem), nullptr));
        SVA_TRY(sva_frame_sgm_rows(c, 1, l->y0, l->rows, l->u_in(l->mem), nullptr));
        SVA_TRY(sva_frame_wta_rows(c, nullptr, l->y0, l->rows));
    }
    SVA_CUDA_OK(c, cudaStreamSynchronize(c->stream));
    return SVA_OK;
}

// copies a ticket's rows from the staging into the caller's buffers once its download is done
static int rows_stream_retire(sva_rows_stream* s, int k) {
    sva_rows_stream::Slot& sl = s->slots[k];
    SVA_STREAM_CUDA_OK(s, cudaEventSynchronize(s->ev_slot[k]));
    const uint8_t* st = s->staging + (size_t)k * s->slot_bytes;
    memcpy(sl.disp, st, s->disp_bytes);
    if (sl.sub) memcpy(sl.sub, st + s->sub_at, s->sub_bytes);
    uint32_t err = 0;
    memcpy(&err, st + s->err_at, sizeof err);
    if (err) s->failed.insert(sl.ticket);
    sl.retired = true;
    return SVA_OK;
}

// one iteration of the skewed order: part 0 of frame i when `with_part0` (its upload already enqueued by the caller), then part 1 / part 2 of
// the frames the lags select among the frames of the current fill, [fill, last)
static int rows_stream_iteration(sva_rows_stream* s, int64_t i, int64_t last, bool with_part0) {
    if (with_part0) {
        const int j = (int)(i % s->P);
        SVA_TRY(s->fwd(j, sva_rows_run_part(s->ctxs[j], 0)));
        SVA_STREAM_CUDA_OK(s, cudaEventRecord(s->ev_p0[j], s->compute));
    }
    const int64_t f1 = i - s->lag1, f2 = i - s->lag2;
    if (f1 >= s->fill && f1 < last) SVA_TRY(s->fwd((int)(f1 % s->P), sva_rows_run_part(s->ctxs[f1 % s->P], 1)));
    if (f2 >= s->fill && f2 < last) {
        const int j = (int)(f2 % s->P), k = (int)(f2 % (int64_t)s->slots.size());
        sva_ctx* c = s->ctxs[j];
        RowsLink* l = s->links[j];
        SVA_STREAM_CUDA_OK(s, cudaStreamWaitEvent(s->compute, s->ev_out[j], 0));   // the context's previous frame is out of disp / subpix
        SVA_STREAM_CUDA_OK(s, cudaStreamWaitEvent(s->compute, s->ev_mask[j], 0));  // this frame's mask is in
        SVA_TRY(s->fwd(j, sva_rows_run_part(c, 2)));
        SVA_STREAM_CUDA_OK(s, cudaEventRecord(s->ev_p2[j], s->compute));
        SVA_STREAM_CUDA_OK(s, cudaStreamWaitEvent(s->d2h, s->ev_p2[j], 0));
        uint8_t* st = s->staging + (size_t)k * s->slot_bytes;
        SVA_STREAM_CUDA_OK(s, cudaMemcpyAsync(st, c->disp.p, s->disp_bytes, cudaMemcpyDeviceToHost, s->d2h));
        if (s->slots[k].sub) SVA_STREAM_CUDA_OK(s, cudaMemcpyAsync(st + s->sub_at, c->subpix.p, s->sub_bytes, cudaMemcpyDeviceToHost, s->d2h));
        SVA_STREAM_CUDA_OK(s, cudaMemcpyAsync(st + s->err_at, l->flag(l->mem, F_ERR), sizeof(uint32_t), cudaMemcpyDeviceToHost, s->d2h));
        SVA_STREAM_CUDA_OK(s, cudaEventRecord(s->ev_out[j], s->d2h));
        SVA_STREAM_CUDA_OK(s, cudaEventRecord(s->ev_slot[k], s->d2h));
        s->finished = f2 + 1;
    }
    return SVA_OK;
}

extern "C" {

int sva_rows_stream_create(sva_ctx* const* ctxs, int32_t n_ctxs, const sva_params* p, sva_rows_stream** out) {
    if (!ctxs || !ctxs[0] || !out) return SVA_ERR_BAD_ARG;
    *out = nullptr;
    sva_ctx* c0 = ctxs[0];
    if (!p) return c0->fail(SVA_ERR_BAD_ARG, "rows_stream_create: null params");
    RowsLink* l0 = (RowsLink*)c0->rows_link;
    if (!l0) return c0->fail(SVA_ERR_STATE, "rows_stream_create: context 0 has no link (sva_rows_open first)");
    const int G = l0->world, P = G + 1;
    if (n_ctxs != P) return c0->fail(SVA_ERR_BAD_ARG, "rows_stream_create: the skewed order keeps world + 1 = " + std::to_string(P) + " frames in flight: pass that many contexts, not " + std::to_string(n_ctxs));
    if (p->width != l0->W || p->height != l0->H || p->num_disp != l0->D || p->n_paths != 8)
        return c0->fail(SVA_ERR_BAD_ARG, "rows_stream_create: the parameters do not match the geometry the links were opened for");
    for (int j = 0; j < P; j++) {
        sva_ctx* c = ctxs[j];
        if (!c) return c0->fail(SVA_ERR_BAD_ARG, "rows_stream_create: null context");
        for (int k = 0; k < j; k++) if (ctxs[k] == c) return c0->fail(SVA_ERR_BAD_ARG, "rows_stream_create: a context is passed twice");
        const RowsLink* l = (const RowsLink*)c->rows_link;
        if (!l) return c0->fail(SVA_ERR_STATE, "rows_stream_create: context " + std::to_string(j) + " has no link (sva_rows_open first)");
        if (l->rank != l0->rank || l->world != G || l->W != l0->W || l->H != l0->H || l->D != l0->D)
            return c0->fail(SVA_ERR_BAD_ARG, "rows_stream_create: the links of the contexts were opened for different ranks, worlds or geometries");
        if (l->part_done != 2) return c0->fail(SVA_ERR_STATE, "rows_stream_create: context " + std::to_string(j) + " is in the middle of a frame (sva_rows_run_part)");
        if (c->device != c0->device || c->stream != c0->stream)
            return c0->fail(SVA_ERR_BAD_ARG, "rows_stream_create: every context must run on the same stream (sva_get_stream / sva_set_stream)");
    }
    SVA_CUDA_OK(c0, cudaSetDevice(c0->device));
    sva_rows_stream* s = new sva_rows_stream();
    s->ctxs.assign(ctxs, ctxs + P);
    for (int j = 0; j < P; j++) s->links.push_back((RowsLink*)ctxs[j]->rows_link);
    s->p = *p;
    s->rank = l0->rank; s->world = G; s->P = P;
    s->lag1 = 1 + std::min(s->rank, G - 1 - s->rank);
    s->lag2 = 1 + std::max(s->rank, G - 1 - s->rank);
    s->compute = c0->stream;
    auto align = [](size_t b) { return (b + 255) & ~(size_t)255; };
    s->disp_bytes = (size_t)p->width * l0->rows * sizeof(uint16_t);
    s->sub_bytes = (size_t)p->width * l0->rows * sizeof(float);
    s->sub_at = align(s->disp_bytes);
    s->err_at = s->sub_at + align(s->sub_bytes);
    s->slot_bytes = s->err_at + 256;
    s->slots.resize(G + 2);
    auto setup = [&]() -> int {
        SVA_STREAM_CUDA_OK(s, cudaStreamCreateWithFlags(&s->h2d, cudaStreamNonBlocking));
        SVA_STREAM_CUDA_OK(s, cudaStreamCreateWithFlags(&s->d2h, cudaStreamNonBlocking));
        for (auto* v : {&s->ev_img, &s->ev_mask, &s->ev_p0, &s->ev_p2, &s->ev_out})
            for (int j = 0; j < P; j++) { v->push_back(nullptr); SVA_STREAM_CUDA_OK(s, cudaEventCreateWithFlags(&v->back(), cudaEventDisableTiming)); }
        for (size_t k = 0; k < s->slots.size(); k++) { s->ev_slot.push_back(nullptr); SVA_STREAM_CUDA_OK(s, cudaEventCreateWithFlags(&s->ev_slot.back(), cudaEventDisableTiming)); }
        cudaError_t e = cudaMallocHost(&s->staging, s->slot_bytes * s->slots.size());
        if (e != cudaSuccess) { s->staging = nullptr; return s->fail(SVA_ERR_NOMEM, std::string("cudaMallocHost: ") + cudaGetErrorString(e)); }
        const std::vector<uint8_t> zeros((size_t)p->width * p->height, 0);
        for (int j = 0; j < P; j++) SVA_TRY(s->fwd(j, rows_stream_warm_up(s, j, zeros)));
        return SVA_OK;
    };
    const int rc = setup();
    if (rc != SVA_OK) { rows_stream_release(s); return rc; }
    *out = s;
    return SVA_OK;
}

int sva_rows_stream_connect_comm(sva_rows_stream* s) {
    if (!s) return SVA_ERR_BAD_ARG;
    if (s->next > s->finished) return s->fail(SVA_ERR_STATE, "connect_comm: frames are in flight (flush first)");
    if (s->world == 1) return SVA_OK;  // no neighbours
    sva_ctx* c0 = s->ctxs[0];
    if (!c0->comm) return s->fail(SVA_ERR_STATE, "connect_comm: context 0 has no communicator (sva_comm_init)");
    if (c0->comm_rank != s->rank || c0->comm_world != s->world) return s->fail(SVA_ERR_BAD_ARG, "connect_comm: the communicator's rank / world differ from the links'");
    for (int j = 0; j < s->P; j++)
        if (s->ctxs[j]->rows_link != s->links[j]) return s->fail(SVA_ERR_STATE, "connect_comm: a link was re-opened or closed since create");
    const int P = s->P, G = s->world;
    const size_t per_rank = (size_t)P * SVA_IPC_HANDLE_BYTES;
    std::vector<uint8_t> all((size_t)G * per_rank);
    for (int j = 0; j < P; j++) SVA_TRY(s->fwd(j, sva_rows_export(s->ctxs[j], all.data() + s->rank * per_rank + (size_t)j * SVA_IPC_HANDLE_BYTES)));
    SVA_CUDA_OK(c0, cudaSetDevice(c0->device));
    SVA_TRY(c0->reserve(c0->comm_scratch, std::max<size_t>(256, all.size())));
    uint8_t* d = c0->comm_scratch.as<uint8_t>();
    SVA_CUDA_OK(c0, cudaMemcpyAsync(d + s->rank * per_rank, all.data() + s->rank * per_rank, per_rank, cudaMemcpyHostToDevice, c0->stream));
    SVA_NCCL_OK(c0, nccl()->AllGather(d + s->rank * per_rank, d, per_rank, NCCL_UINT8, (NcclComm)c0->comm, c0->stream));
    SVA_CUDA_OK(c0, cudaMemcpyAsync(all.data(), d, all.size(), cudaMemcpyDeviceToHost, c0->stream));
    SVA_CUDA_OK(c0, cudaStreamSynchronize(c0->stream));
    for (int j = 0; j < P; j++) {
        auto handle = [&](int r) { return all.data() + (size_t)r * per_rank + (size_t)j * SVA_IPC_HANDLE_BYTES; };
        SVA_TRY(s->fwd(j, sva_rows_connect(s->ctxs[j], s->rank > 0 ? handle(s->rank - 1) : nullptr, s->rank < G - 1 ? handle(s->rank + 1) : nullptr)));
    }
    return sva_comm_barrier(c0);  // nobody runs ahead of a neighbour that has not mapped its side yet
}

int sva_rows_stream_submit(sva_rows_stream* s, const sva_image_u8* ref, const sva_image_u8* others, const sva_image_u8* mask,
                           uint16_t* out_disp_rows, float* out_subpix_rows, int64_t* out_ticket) {
    if (!s) return SVA_ERR_BAD_ARG;
    if (!out_disp_rows || !out_ticket) return s->fail(SVA_ERR_BAD_ARG, "submit: null output");
    const int G = s->world;
    for (int j = 0; j < s->P; j++) {
        const RowsLink* l = s->links[j];
        if (s->ctxs[j]->rows_link != l) return s->fail(SVA_ERR_STATE, "submit: a link was re-opened or closed since create");
        if ((s->rank > 0 && !l->prev) || (s->rank < G - 1 && !l->next))
            return s->fail(SVA_ERR_STATE, "submit: the link of context " + std::to_string(j) + " is not connected (sva_rows_connect*, sva_rows_stream_connect_comm)");
    }
    SVA_TRY(check_frame_args(s->ctxs[0], &s->p, ref, others, mask));
    SVA_CUDA_OK(s->ctxs[0], cudaSetDevice(s->ctxs[0]->device));
    const int64_t i = s->next;
    const int j = (int)(i % s->P), k = (int)(i % (int64_t)s->slots.size());
    sva_rows_stream::Slot& sl = s->slots[k];
    if (!sl.retired) SVA_TRY(rows_stream_retire(s, k));  // ticket i - (G + 2): its download is at least two iterations old
    sl.ticket = i; sl.retired = false; sl.disp = out_disp_rows; sl.sub = out_subpix_rows;
    sva_ctx* c = s->ctxs[j];
    SVA_STREAM_CUDA_OK(s, cudaStreamWaitEvent(s->h2d, s->ev_p0[j], 0));  // K1a of the context's previous frame has read its images
    c->stream = s->h2d;
    const int rc = sva_frame_upload(c, &s->p, ref, others, nullptr);
    c->stream = s->compute;
    if (rc != SVA_OK) { sl.retired = true; sl.ticket = -1; return s->fwd(j, rc); }
    SVA_STREAM_CUDA_OK(s, cudaEventRecord(s->ev_img[j], s->h2d));
    SVA_STREAM_CUDA_OK(s, cudaStreamWaitEvent(s->compute, s->ev_img[j], 0));
    if (mask) {  // K3 of the context's previous frame has read its mask (the buffer exists since create: no allocation here)
        SVA_STREAM_CUDA_OK(s, cudaStreamWaitEvent(s->h2d, s->ev_p2[j], 0));
        SVA_TRY(s->fwd(j, c->reserve(c->mask, (size_t)s->p.width * s->p.height)));
        SVA_STREAM_CUDA_OK(s, cudaMemcpy2DAsync(c->mask.p, s->p.width, mask->data, mask->step, s->p.width, s->p.height, cudaMemcpyHostToDevice, s->h2d));
        c->has_mask = true;
    }
    SVA_STREAM_CUDA_OK(s, cudaEventRecord(s->ev_mask[j], s->h2d));  // (without a mask: right after the images, a wait that costs nothing)
    s->next = i + 1;
    *out_ticket = i;
    return rows_stream_iteration(s, i, i + 1, true);
}

int sva_rows_stream_flush(sva_rows_stream* s) {
    if (!s) return SVA_ERR_BAD_ARG;
    SVA_CUDA_OK(s->ctxs[0], cudaSetDevice(s->ctxs[0]->device));
    for (int64_t i = s->next; s->finished < s->next; i++) SVA_TRY(rows_stream_iteration(s, i, s->next, false));
    s->fill = s->next;
    return SVA_OK;
}

int sva_rows_stream_wait(sva_rows_stream* s, int64_t ticket) {
    if (!s) return SVA_ERR_BAD_ARG;
    if (ticket < 0 || ticket >= s->next) return s->fail(SVA_ERR_BAD_ARG, "wait: unknown ticket " + std::to_string(ticket));
    const int k = (int)(ticket % (int64_t)s->slots.size());
    if (s->slots[k].ticket == ticket && !s->slots[k].retired) {
        if (ticket >= s->finished) return s->fail(SVA_ERR_STATE, "wait: the last part of frame " + std::to_string(ticket) + " is not enqueued yet (submit more frames, or flush)");
        SVA_CUDA_OK(s->ctxs[0], cudaSetDevice(s->ctxs[0]->device));
        SVA_TRY(rows_stream_retire(s, k));
    }
    if (s->failed.count(ticket))
        return s->fail(SVA_ERR_COMM, "frame " + std::to_string(ticket) + ": a neighbour's path-line state did not arrive within the time-out (SVA_ROWS_TIMEOUT_MS); the block's maps are not valid");
    return SVA_OK;
}

int sva_rows_stream_destroy(sva_rows_stream* s) {
    if (!s) return SVA_ERR_BAD_ARG;
    cudaSetDevice(s->ctxs[0]->device);
    cudaStreamSynchronize(s->compute);
    rows_stream_release(s);
    return SVA_OK;
}

}  // extern "C"
