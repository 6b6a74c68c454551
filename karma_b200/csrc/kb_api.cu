// kb_api.cu -- context management and the thin extern "C" layer of libkarma_b200.so.
#include "kb_common.cuh"
#include <cstring>
#include <cstdlib>

static thread_local char g_err[512] = "";

void kb_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int kb_cuda_fail(cudaError_t e, const char* what) {
    kb_set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
    return KB_ECUDA;
}

int kb_mode_describe(int mode, KbMode* m) {
    memset(m, 0, sizeof(*m));
    if (mode == KB_MODE_5P6) {
        m->ka = 5; m->kb = 6; m->pal_b = 1; m->bins_a = 1024; m->bins_b = 64; m->permute = 1;
    } else if (mode == KB_MODE_DENSE_5_6) {
        m->ka = 5; m->kb = 6; m->bins_a = 1024; m->bins_b = 4096;
    } else if (mode == KB_MODE_DENSE_4_5) {
        m->ka = 4; m->kb = 5; m->bins_a = 256; m->bins_b = 1024;
    } else if (mode >= KB_MODE_K(1) && mode <= KB_MODE_K(7)) {
        m->ka = mode - 16; m->bins_a = 1 << (2 * m->ka);
    } else {
        kb_set_error("unknown column mode %d", mode);
        return KB_EINVAL;
    }
    m->cols = m->bins_a + m->bins_b;
    return KB_OK;
}

extern "C" int kb_version(void) { return 105; }
extern "C" const char* kb_last_error(void) { return g_err; }

extern "C" int kb_mode_columns(int mode) {
    KbMode m;
    int rc = kb_mode_describe(mode, &m);
    return rc ? rc : m.cols;
}

extern "C" int kb_create(kb_ctx** out, int device) {
    KB_CHECK_ARG(out, "out");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        kb_set_error("no CUDA device (%s): libkarma_b200 has no CPU fallback", cudaGetErrorString(e));
        return KB_ENOGPU;
    }
    KB_CHECK_ARG(device >= 0 && device < ndev, "device index");
    cudaDeviceProp prop;
    KB_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        kb_set_error("device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
        return KB_ENOGPU;
    }
    KB_CUDA(cudaSetDevice(device));
    kb_ctx* c = (kb_ctx*)calloc(1, sizeof(kb_ctx));
    if (!c) { kb_set_error("out of host memory"); return KB_EINVAL; }
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    c->stream = 0;
    *out = c;
    return KB_OK;
}

static void kb_free_exotic(kb_ctx* c) {
    cudaFree(c->d_ex_keys); cudaFree(c->d_ex_keys_hi); cudaFree(c->d_ex_row); cudaFree(c->d_ex_keyidx); cudaFree(c->d_ex_cnt);
    c->d_ex_keys = nullptr; c->d_ex_keys_hi = nullptr; c->d_ex_row = nullptr; c->d_ex_keyidx = nullptr; c->d_ex_cnt = nullptr;
    c->ex_n_keys = c->ex_n_entries = 0;
}

extern "C" int kb_destroy(kb_ctx* c) {
    if (!c) return KB_OK;
    cudaSetDevice(c->device);
    if (c->ev0) {
        for (int i = 0; i < KB_N_TIMERS; ++i)
            for (int j = 0; j < KB_EV_RING; ++j) { cudaEventDestroy(c->ev0[i][j]); cudaEventDestroy(c->ev1[i][j]); }
        free(c->ev0); free(c->ev1);
    }
    cudaFree(c->d_k1_scratch);
    kb_free_exotic(c);
    cudaFree(c->d_rg_a); cudaFree(c->d_rg_b); cudaFree(c->d_rg_w); cudaFree(c->d_rg_shared);
    kb_links_free(c);
    kb_fuzzy_free(c);
    kb_knn_cache_free(c);
    kb_spectral_free(c);
    kb_mcl_free(c);
    if (c->pool) { cudaDeviceSynchronize(); cudaMemPoolDestroy(c->pool); }
    free(c);
    return KB_OK;
}

// Temporaries of multi-phase builds come from a per-context stream-ordered pool that never gives memory
// back to the driver (release threshold = max), so a repeated build allocates nothing.
int kb_pool_get(kb_ctx* c, cudaMemPool_t* out) {
    if (!c->pool) {
        cudaMemPoolProps props = {};
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = c->device;
        KB_CUDA(cudaMemPoolCreate(&c->pool, &props));
        unsigned long long keep = ~0ull;
        KB_CUDA(cudaMemPoolSetAttribute(c->pool, cudaMemPoolAttrReleaseThreshold, &keep));
    }
    *out = c->pool;
    return KB_OK;
}

extern "C" int kb_set_stream(kb_ctx* c, void* s) {
    KB_CHECK_ARG(c, "ctx");
    c->stream = (cudaStream_t)s;
    return KB_OK;
}

extern "C" int kb_enable_timing(kb_ctx* c, int on) {
    KB_CHECK_ARG(c, "ctx");
    if (on && !c->ev0) {
        KB_CUDA(cudaSetDevice(c->device));
        c->ev0 = (cudaEvent_t(*)[KB_EV_RING])calloc(KB_N_TIMERS, sizeof(*c->ev0));
        c->ev1 = (cudaEvent_t(*)[KB_EV_RING])calloc(KB_N_TIMERS, sizeof(*c->ev1));
        if (!c->ev0 || !c->ev1) { kb_set_error("out of host memory"); return KB_EINVAL; }
        for (int i = 0; i < KB_N_TIMERS; ++i)
            for (int j = 0; j < KB_EV_RING; ++j) {
                KB_CUDA(cudaEventCreate(&c->ev0[i][j]));
                KB_CUDA(cudaEventCreate(&c->ev1[i][j]));
            }
    }
    c->timing = on ? 1 : 0;
    for (int i = 0; i < KB_N_TIMERS; ++i) c->ev_n[i] = 0;
    return KB_OK;
}

extern "C" int kb_stage_ms(kb_ctx* c, int which, float* mean_ms, int* n_launches) {
    KB_CHECK_ARG(c && mean_ms && which >= 0 && which < KB_N_TIMERS, "which");
    const int n = c->ev_n[which] < KB_EV_RING ? c->ev_n[which] : KB_EV_RING;
    if (n_launches) *n_launches = n;
    *mean_ms = 0.f;
    if (!c->ev0) { kb_set_error("timing is not enabled (kb_enable_timing)"); return KB_EINVAL; }
    if (n == 0) return KB_OK;                                   // nothing recorded since the last read
    double sum = 0.0;
    for (int j = 0; j < n; ++j) {
        float ms = 0.f;
        KB_CUDA(cudaEventSynchronize(c->ev1[which][j]));
        KB_CUDA(cudaEventElapsedTime(&ms, c->ev0[which][j], c->ev1[which][j]));
        sum += ms;
    }
    *mean_ms = (float)(sum / n);
    c->ev_n[which] = 0;
    return KB_OK;
}

extern "C" int64_t kb_launch_count(kb_ctx* c) { return c ? c->launches : 0; }

extern "C" int kb_count(kb_ctx* ctx, int mode, const uint8_t* d_bases, const int64_t* d_offsets, int64_t n,
                        uint32_t* d_counts, int64_t ld, uint32_t* d_exotic, uint32_t* d_presence) {
    KB_CHECK_ARG(ctx && d_bases && d_offsets && d_counts, "null pointer");
    KbMode m;
    const int track = (mode & KB_COUNT_NO_COLUMNS) ? 0 : 1;
    int rc = kb_mode_describe(mode & ~KB_COUNT_NO_COLUMNS, &m);
    if (rc) return rc;
    KB_CHECK_ARG(n >= 0 && n < (1LL << 31) - 2, "contig count");
    KB_CHECK_ARG(ld >= m.cols && (ld % 4) == 0, "ld must be >= columns and a multiple of 4");
    KB_CHECK_ARG(((uintptr_t)d_bases % 16) == 0 && ((uintptr_t)d_counts % 16) == 0, "bases/counts must be 16-byte aligned");
    if (n == 0) return KB_OK;
    KB_CUDA(cudaSetDevice(ctx->device));
    return kb_launch_count_kernels(ctx, m, d_bases, d_offsets, n, d_counts, ld, d_exotic, d_presence, track);
}

extern "C" int kb_count_stats(kb_ctx* ctx, int64_t* n_long, int64_t* exotic_total) {
    KB_CHECK_ARG(ctx, "ctx");
    int32_t h[6] = {0, 0, 0, 0, 0, 0};      // K1 scratch: [2..3] exotic total, [4..5] (long contigs << 32) | chunks
    if (ctx->d_k1_scratch) {
        KB_CUDA(cudaSetDevice(ctx->device));
        KB_CUDA(cudaMemcpyAsync(h, ctx->d_k1_scratch, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
        KB_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    if (n_long) *n_long = h[5];
    if (exotic_total) { unsigned long long t; memcpy(&t, &h[2], 8); *exotic_total = (int64_t)t; }
    return KB_OK;
}
