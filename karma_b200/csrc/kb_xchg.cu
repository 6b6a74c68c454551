// kb_xchg.cu -- peer-memory exchange of the kNN stage across the GPUs of one node (sm_100a, NVLink 5 / NVSwitch).
//
// The one exchange step of the path (SURVEY 8e): every rank needs the fp16 operand rows and the 32-byte row
// records of ALL contigs before it can score its own query rows against them, and every rank wants the
// finished k-lists.  Instead of collectives, every rank owns one "arena" (cudaMalloc + CUDA IPC, the same
// layout on every rank) that its peers map:
//   * after K3 a rank pushes its shard of each gathered array into every peer's arena on a side stream (copy engines,
//     three peers at a time), nearest-following rank first, and raises arrive[rank] = epoch there as each shard
//     completes;
//   * K4 (kb_knn_tc.cu) starts on the local shard at once; its TMA producer polls arrive[r] before the first
//     key tile of rank r, so the transfer overlaps the sweep tile by tile;
//   * K5 stores its rows straight into every peer's gathered result arrays (stores over NVLink);
//   * kb_xchg_finish pushes a small per-rank record (validation words), raises lists[rank] = epoch everywhere
//     and waits until every peer has done the same.
// Re-use across passes needs no barrier: a rank announces done[rank] = epoch-1 to its peers when it BEGINS the
// next pass (everything of the previous pass, including the caller's reads of the results, is then behind it in
// stream order) and pushes only after every peer has announced the same.
// All entry points only enqueue (kernels + peer copies): a pass can be captured in a CUDA graph.
#include "kb_common.cuh"
#include <cstdlib>
#include <cstring>

#define KB_XCHG_MAX_WORLD 64

struct KbXchgCtrl {                      // first 1 KB of every arena
    uint32_t epoch;                      // local: number of passes begun
    uint32_t pad[63];
    uint32_t arrive[KB_XCHG_MAX_WORLD];  // written by peers: shard of rank r for pass `value` has landed here
    uint32_t done[KB_XCHG_MAX_WORLD];    // written by peers: rank r no longer reads what I pushed for pass `value`
    uint32_t lists[KB_XCHG_MAX_WORLD];   // written by peers: rank r's results + record for pass `value` are here
};
static_assert(sizeof(KbXchgCtrl) == 1024, "control block is 1 KB");

struct kb_xchg {
    kb_ctx* ctx;
    int world, rank;
    int64_t bytes;
    uint8_t* local;                       // my arena
    uint8_t* peer[KB_XCHG_MAX_WORLD];     // peers' arenas as mapped here (peer[rank] == local)
    uint8_t** d_peer;                     // device copy of peer[]
    bool attached;
    cudaStream_t extra[2];                // two more copy streams: three peer copies in flight at a time
    cudaEvent_t ev_fork, ev_join[2];
};

namespace {

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// bounded spin: a peer that died must surface as a trapped kernel, not as a hung GPU
__device__ __forceinline__ void wait_ge(const uint32_t* p, uint32_t want, int what, int who) {
    const long long t0 = clock64();
    uint32_t it = 0;
    while ((int32_t)(ld_acquire_sys(p) - want) < 0) {
        if ((++it & 0xff) == 0 && clock64() - t0 > 40000000000LL) {
            printf("kb_xchg: timed out waiting for flag %d of rank %d (want %u, have %u)\n", what, who, want, ld_acquire_sys(p));
            __trap();
        }
        __nanosleep(100);
    }
}

// epoch++ and "I am done with pass epoch-1" to every peer
__global__ void kx_begin(uint8_t* local, uint8_t* const* peer, int world, int rank) {
    KbXchgCtrl* c = reinterpret_cast<KbXchgCtrl*>(local);
    __shared__ uint32_t e;
    if (threadIdx.x == 0) { e = c->epoch + 1; c->epoch = e; }
    __syncthreads();
    const int t = threadIdx.x;
    if (t < world && t != rank) {
        __threadfence_system();
        st_release_sys(&reinterpret_cast<KbXchgCtrl*>(peer[t])->done[rank], e - 1);
    }
}
// which: 0 = every peer is done with my previous shard, 2 = every peer's results are here
__global__ void kx_wait(const uint8_t* local, int world, int rank, int which) {
    const KbXchgCtrl* c = reinterpret_cast<const KbXchgCtrl*>(local);
    const uint32_t e = c->epoch;
    const int t = threadIdx.x;
    if (t < world && t != rank) {
        if (which == 0) wait_ge(&c->done[t], e - 1, 0, t);
        else wait_ge(&c->lists[t], e, 2, t);
    }
}
// arrive[rank] = epoch at ONE peer, right behind the copies of that peer's shard on the same stream
__global__ void kx_signal_arrive(const uint8_t* local, uint8_t* peer_arena, int rank) {
    const uint32_t e = reinterpret_cast<const KbXchgCtrl*>(local)->epoch;
    __threadfence_system();
    st_release_sys(&reinterpret_cast<KbXchgCtrl*>(peer_arena)->arrive[rank], e);
}
// my small record (rec_words u32 at rec_off + rank*rec_words*4) to every peer, then lists[rank] = epoch there
__global__ void kx_finish(uint8_t* local, uint8_t* const* peer, int world, int rank, int64_t rec_off, int rec_words) {
    const uint32_t e = reinterpret_cast<const KbXchgCtrl*>(local)->epoch;
    const int64_t off = rec_off + (int64_t)rank * rec_words * 4;
    const uint32_t* src = reinterpret_cast<const uint32_t*>(local + off);
    for (int p = 0; p < world; ++p) {
        if (p == rank) continue;
        uint32_t* dst = reinterpret_cast<uint32_t*>(peer[p] + off);
        for (int i = threadIdx.x; i < rec_words; i += blockDim.x) dst[i] = src[i];
    }
    __threadfence_system();
    __syncthreads();
    const int t = threadIdx.x;
    if (t < world && t != rank) {
        __threadfence_system();
        st_release_sys(&reinterpret_cast<KbXchgCtrl*>(peer[t])->lists[rank], e);
    }
}

}  // namespace

extern "C" int kb_xchg_create(kb_ctx* ctx, int world, int rank, int64_t bytes, kb_xchg** out, void** d_local, uint8_t* handle64) {
    KB_CHECK_ARG(ctx && out && d_local && handle64, "null pointer");
    KB_CHECK_ARG(world >= 1 && world <= KB_XCHG_MAX_WORLD && rank >= 0 && rank < world && bytes >= (int64_t)sizeof(KbXchgCtrl),
                 "world/rank/bytes");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle is 64 bytes");
    KB_CUDA(cudaSetDevice(ctx->device));
    kb_xchg* x = (kb_xchg*)calloc(1, sizeof(kb_xchg));
    if (!x) { kb_set_error("out of host memory"); return KB_EINVAL; }
    x->ctx = ctx; x->world = world; x->rank = rank; x->bytes = bytes;
    cudaError_t e = cudaMalloc((void**)&x->local, (size_t)bytes);
    if (e != cudaSuccess) { free(x); return kb_cuda_fail(e, "cudaMalloc(arena)"); }
    e = cudaMemset(x->local, 0, sizeof(KbXchgCtrl));
    if (e == cudaSuccess) e = cudaMalloc((void**)&x->d_peer, sizeof(uint8_t*) * KB_XCHG_MAX_WORLD);
    cudaIpcMemHandle_t h;
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, x->local);
    if (e != cudaSuccess) { cudaFree(x->local); cudaFree(x->d_peer); free(x); return kb_cuda_fail(e, "arena set-up (cudaIpcGetMemHandle)"); }
    memcpy(handle64, &h, 64);
    for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
        e = cudaStreamCreateWithFlags(&x->extra[i], cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&x->ev_join[i], cudaEventDisableTiming);
    }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&x->ev_fork, cudaEventDisableTiming);
    x->peer[rank] = x->local;
    *out = x; *d_local = x->local;
    return KB_OK;
}

extern "C" int kb_xchg_attach(kb_xchg* x, const uint8_t* handles) {
    KB_CHECK_ARG(x && handles && !x->attached, "null pointer / attached twice");
    KB_CUDA(cudaSetDevice(x->ctx->device));
    for (int p = 0; p < x->world; ++p) {
        if (p == x->rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, handles + 64 * p, 64);
        void* ptr = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) { kb_set_error("cudaIpcOpenMemHandle(rank %d) failed: %s", p, cudaGetErrorString(e)); cudaGetLastError(); return KB_ECUDA; }
        x->peer[p] = reinterpret_cast<uint8_t*>(ptr);
    }
    KB_CUDA(cudaMemcpy(x->d_peer, x->peer, sizeof(uint8_t*) * KB_XCHG_MAX_WORLD, cudaMemcpyHostToDevice));
    x->attached = true;
    return KB_OK;
}

extern "C" int kb_xchg_peer_ptr(kb_xchg* x, int peer, void** d_ptr) {
    KB_CHECK_ARG(x && d_ptr && peer >= 0 && peer < x->world && (x->attached || peer == x->rank), "peer");
    *d_ptr = x->peer[peer];
    return KB_OK;
}

extern "C" int kb_xchg_destroy(kb_xchg* x) {
    if (!x) return KB_OK;
    cudaSetDevice(x->ctx->device);
    cudaDeviceSynchronize();
    for (int p = 0; p < x->world; ++p)
        if (p != x->rank && x->peer[p]) cudaIpcCloseMemHandle(x->peer[p]);
    for (int i = 0; i < 2; ++i) { if (x->extra[i]) cudaStreamDestroy(x->extra[i]); if (x->ev_join[i]) cudaEventDestroy(x->ev_join[i]); }
    if (x->ev_fork) cudaEventDestroy(x->ev_fork);
    cudaFree(x->d_peer);
    cudaFree(x->local);
    free(x);
    return KB_OK;
}

// Touch every peer's copy of this rank's shard regions once (a memset over NVLink) and synchronise: the first access to a
// freshly IPC-mapped multi-gigabyte arena sets up its peer mappings, which must not happen inside the first pass where
// kernels wait (bounded) for the data.
extern "C" int kb_xchg_warm(kb_xchg* x, int n_regions, const int64_t* region_off, const int64_t* shard_bytes) {
    KB_CHECK_ARG(x && x->attached && n_regions >= 0 && (n_regions == 0 || (region_off && shard_bytes)), "arguments");
    KB_CUDA(cudaSetDevice(x->ctx->device));
    for (int p = 0; p < x->world; ++p) {
        if (p == x->rank) continue;
        for (int r = 0; r < n_regions; ++r) {
            const int64_t off = region_off[r] + (int64_t)x->rank * shard_bytes[r];
            KB_CHECK_ARG(off >= (int64_t)sizeof(KbXchgCtrl) && off + shard_bytes[r] <= x->bytes, "region outside the arena");
            if (shard_bytes[r]) KB_CUDA(cudaMemsetAsync(x->peer[p] + off, 0, (size_t)shard_bytes[r], x->ctx->stream));
        }
    }
    KB_CUDA(cudaStreamSynchronize(x->ctx->stream));
    return KB_OK;
}

extern "C" int kb_xchg_begin(kb_xchg* x) {
    KB_CHECK_ARG(x && x->attached, "exchange not attached");
    kx_begin<<<1, KB_XCHG_MAX_WORLD, 0, x->ctx->stream>>>(x->local, x->d_peer, x->world, x->rank);
    x->ctx->launches++;
    KB_CUDA(cudaGetLastError());
    return KB_OK;
}

extern "C" int kb_xchg_push(kb_xchg* x, void* stream, int n_regions, const int64_t* region_off, const int64_t* shard_bytes) {
    KB_CHECK_ARG(x && x->attached && n_regions >= 0 && (n_regions == 0 || (region_off && shard_bytes)), "arguments");
    cudaStream_t st = (cudaStream_t)stream;
    kx_wait<<<1, KB_XCHG_MAX_WORLD, 0, st>>>(x->local, x->world, x->rank, 0);
    x->ctx->launches++;
    KB_CUDA(cudaGetLastError());
    // nearest-following rank first: rank r then receives from r+1, r+2, ... -- the order in which K4 sweeps.  Three
    // peers are served at a time (the caller's stream and two of our own, forked and joined with events, so the
    // whole fan-out is capturable), and every peer's arrival flag is raised right behind ITS copies: one stream
    // of back-to-back peer copies moves ~150 GB/s, and a single flag kernel at the end would hold back the first
    // shard until the last one has gone out
    cudaStream_t sts[3] = {st, x->extra[0], x->extra[1]};
    const int ns = x->world > 2 ? 3 : 1;
    if (ns > 1) {
        KB_CUDA(cudaEventRecord(x->ev_fork, st));
        for (int i = 1; i < ns; ++i) KB_CUDA(cudaStreamWaitEvent(sts[i], x->ev_fork, 0));
    }
    for (int d = 1; d < x->world; ++d) {
        const int p = (x->rank - d + x->world) % x->world;
        cudaStream_t cs = sts[(d - 1) % ns];
        for (int r = 0; r < n_regions; ++r) {
            const int64_t off = region_off[r] + (int64_t)x->rank * shard_bytes[r];
            KB_CHECK_ARG(off >= (int64_t)sizeof(KbXchgCtrl) && off + shard_bytes[r] <= x->bytes, "region outside the arena");
            if (shard_bytes[r] == 0) continue;
            KB_CUDA(cudaMemcpyAsync(x->peer[p] + off, x->local + off, (size_t)shard_bytes[r], cudaMemcpyDeviceToDevice, cs));
        }
        kx_signal_arrive<<<1, 1, 0, cs>>>(x->local, x->peer[p], x->rank);
        x->ctx->launches++;
    }
    KB_CUDA(cudaGetLastError());
    for (int i = 1; i < ns; ++i) {
        KB_CUDA(cudaEventRecord(x->ev_join[i - 1], sts[i]));
        KB_CUDA(cudaStreamWaitEvent(st, x->ev_join[i - 1], 0));
    }
    return KB_OK;
}

extern "C" int kb_xchg_finish(kb_xchg* x, int64_t rec_off, int32_t rec_words) {
    KB_CHECK_ARG(x && x->attached && rec_words >= 0, "arguments");
    KB_CHECK_ARG(rec_words == 0 || (rec_off >= (int64_t)sizeof(KbXchgCtrl) && rec_off + (int64_t)x->world * rec_words * 4 <= x->bytes),
                 "record region outside the arena");
    cudaStream_t st = x->ctx->stream;
    kx_finish<<<1, 256, 0, st>>>(x->local, x->d_peer, x->world, x->rank, rec_off, rec_words);
    kx_wait<<<1, KB_XCHG_MAX_WORLD, 0, st>>>(x->local, x->world, x->rank, 2);
    x->ctx->launches += 2;
    KB_CUDA(cudaGetLastError());
    return KB_OK;
}

// device pointers into the arena's control block that kb_knn needs (arrival flags, epoch word)
extern "C" int kb_xchg_flags(kb_xchg* x, const uint32_t** d_arrive, const uint32_t** d_epoch) {
    KB_CHECK_ARG(x && d_arrive && d_epoch, "null pointer");
    const KbXchgCtrl* c = reinterpret_cast<const KbXchgCtrl*>(x->local);
    *d_arrive = c->arrive; *d_epoch = &c->epoch;
    return KB_OK;
}
