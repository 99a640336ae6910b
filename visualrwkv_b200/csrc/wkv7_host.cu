// wkv7_host.cu — C-ABI entry points for the WKV7 recurrence (see include/vrwkv_b200.h).
// Replaces cuda_forward / cuda_backward of VisualRWKV-v7/v7.00/cuda/wkv7_cuda.cu:132-138.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include <cudaTypedefs.h>

#include "../../include/vrwkv_b200.h"
#include "host_util.h"
#include "wkv7_fwd.cuh"
#include "wkv7_bwd2.cuh"
#include "wkv7_chunk_common.cuh"
#include "wkv7_chunk_fwd.cuh"
#include "wkv7_chunk_dstate.cuh"
#include "wkv7_chunk_bwd.cuh"
#include "wkv7_fwd2.cuh"
#include "wkv7_x6_fwd.cuh"
#include "wkv7_x6_bwd.cuh"

using namespace vrwkv;

static std::atomic<int> g_fwd_variant{0}, g_bwd_variant{0};

extern "C" int vrwkv_wkv7_set_variant(int fwd_variant, int bwd_variant) {
    g_fwd_variant.store(fwd_variant);
    g_bwd_variant.store(bwd_variant);
    return VRWKV_OK;
}

// [B*T, H*64] matrix of `elem_bytes`-wide elements, box = [16 rows x 64 cols].
static int make_stream_map(CUtensorMap* m, const void* base, int B, int T, int H, int elem_bytes) {
    return vrwkv_encode_2d(m, base, elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32,
                           elem_bytes, (uint64_t)H * WKV_N, (uint64_t)B * T, (uint64_t)H * WKV_N * elem_bytes, WKV_N,
                           WKV_TC, CU_TENSOR_MAP_SWIZZLE_NONE);
}

template <int R, int NSTAGE, int UNROLL = 5>
static int launch_fwd2(const CUtensorMap* tm, const Wkv7FwdArgs& a, cudaStream_t st) {
    auto kern = wkv7_fwd2_kernel<R, NSTAGE, UNROLL>;
    const size_t smem = sizeof(Wkv7Fwd2Smem<NSTAGE>) + 128;
    VRWKV_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(a.H, a.B), block((WKV_N / R) * 8 + 32);
    kern<<<grid, block, smem, st>>>(tm[0], tm[1], tm[2], tm[3], tm[4], tm[5], a);
    VRWKV_CUDA(cudaGetLastError());
    vrwkv_count_launch(1);
    return VRWKV_OK;
}

template <int R, int NSTAGE, int UNROLL = 2>
static int launch_bwd2(const CUtensorMap* tm, const Wkv7BwdArgs& a, cudaStream_t st) {
    auto kern = wkv7_bwd2_kernel<R, NSTAGE, UNROLL>;
    const size_t smem = sizeof(Wkv7Bwd2Smem<NSTAGE>) + 128;
    VRWKV_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(a.H, a.B), block((WKV_N / R) * 8 + 32);
    kern<<<grid, block, smem, st>>>(tm[0], tm[1], tm[2], tm[3], tm[4], tm[5], tm[6], tm[7], a);
    VRWKV_CUDA(cudaGetLastError());
    vrwkv_count_launch(1);
    return VRWKV_OK;
}

extern "C" int vrwkv_wkv7_chunk_debug(float* buf) {
    VRWKV_CUDA(cudaMemcpyToSymbol(g_chunk_dbg, &buf, sizeof(buf)));
    return VRWKV_OK;
}

static int launch_chunk_fwd(const void* const* in, const Wkv7FwdArgs& a, bool chunk_ck, cudaStream_t st) {
    CUtensorMap tm[6];
    for (int i = 0; i < 6; i++) {
        int rc = vrwkv_encode_2d(&tm[i], in[i], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (uint64_t)a.H * WKV_N, (uint64_t)a.B * a.T,
                                 (uint64_t)a.H * WKV_N * 2, WKV_N, CK_L, CU_TENSOR_MAP_SWIZZLE_NONE);
        if (rc) return rc;
    }
    const size_t smem = sizeof(Wkv7ChunkSmem) + 1024;
    auto kern = chunk_ck ? wkv7_chunk_fwd_kernel<true> : wkv7_chunk_fwd_kernel<false>;
    VRWKV_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(a.H, a.B), block(CK_THREADS);
    kern<<<grid, block, smem, st>>>(tm[0], tm[1], tm[2], tm[3], tm[4], tm[5], a);
    VRWKV_CUDA(cudaGetLastError());
    vrwkv_count_launch(1);
    return VRWKV_OK;
}

static int make_chunk_map(CUtensorMap* m, const void* base, int B, int T, int H) {
    return vrwkv_encode_2d(m, base, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (uint64_t)H * WKV_N, (uint64_t)B * T,
                           (uint64_t)H * WKV_N * 2, WKV_N, CK_L, CU_TENSOR_MAP_SWIZZLE_NONE);
}

// backward = tensor-core scan of dL/dS over 64-step chunks + the step-by-step kernel on all segments concurrently
template <int R, int NSTAGE>
static int launch_bwd_segmented(const CUtensorMap* tm, const void* w, const void* q, const void* a, const void* b,
                                const void* dy, Wkv7BwdArgs args, cudaStream_t st) {
    const int B = args.B, T = args.T, H = args.H, nseg = T / CK_L;
    float* ds = nullptr;
    if (nseg > 1) {
        // stream-ordered workspace; keep freed blocks in the device's pool instead of returning them to the OS at
        // every synchronisation (the default release threshold of 0 makes each step pay a real cudaMalloc)
        static std::atomic<unsigned> pool_ready{0};
        int dev = 0;
        VRWKV_CUDA(cudaGetDevice(&dev));
        if (!(pool_ready.load() & (1u << dev))) {
            cudaMemPool_t pool;
            VRWKV_CUDA(cudaDeviceGetDefaultMemPool(&pool, dev));
            uint64_t keep = UINT64_MAX;
            VRWKV_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
            pool_ready.fetch_or(1u << dev);
        }
        VRWKV_CUDA(cudaMallocAsync((void**)&ds, (size_t)B * H * nseg * WKV_N * WKV_N * sizeof(float), st));
        CUtensorMap cm[5];
        const void* in[5] = {w, q, a, b, dy};
        for (int i = 0; i < 5; i++) {
            int rc = make_chunk_map(&cm[i], in[i], B, T, H);
            if (rc) return rc;
        }
        const size_t smem = sizeof(Wkv7DstateSmem) + 1024;
        VRWKV_CUDA(cudaFuncSetAttribute(wkv7_chunk_dstate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        Wkv7DstateArgs da{B, T, H, ds};
        wkv7_chunk_dstate_kernel<<<dim3(H, B), CK_THREADS, smem, st>>>(cm[0], cm[1], cm[2], cm[3], cm[4], da);
        VRWKV_CUDA(cudaGetLastError());
        vrwkv_count_launch(1);
    }
    args.ds_in = ds;
    args.span = CK_L / WKV_TC;
    auto kern = wkv7_bwd2_kernel<R, NSTAGE, 2>;
    const size_t smem2 = sizeof(Wkv7Bwd2Smem<NSTAGE>) + 128;
    VRWKV_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
    // two CTAs (2 x ~81 KB) per SM: ask for the largest shared-memory carveout, the default sizes it for one block
    VRWKV_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    dim3 grid(H, B, nseg), block((WKV_N / R) * 8 + 32);
    kern<<<grid, block, smem2, st>>>(tm[0], tm[1], tm[2], tm[3], tm[4], tm[5], tm[6], tm[7], args);
    VRWKV_CUDA(cudaGetLastError());
    vrwkv_count_launch(1);
    if (ds) VRWKV_CUDA(cudaFreeAsync(ds, st));
    return VRWKV_OK;
}

static int ensure_pool_keeps_memory() {
    // stream-ordered workspaces: keep freed blocks in the device's pool instead of returning them to the OS at every
    // synchronisation (the default release threshold of 0 makes each step pay a real cudaMalloc)
    static std::atomic<unsigned> pool_ready{0};
    int dev = 0;
    VRWKV_CUDA(cudaGetDevice(&dev));
    if (!(pool_ready.load() & (1u << dev))) {
        cudaMemPool_t pool;
        VRWKV_CUDA(cudaDeviceGetDefaultMemPool(&pool, dev));
        uint64_t keep = UINT64_MAX;
        VRWKV_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
        pool_ready.fetch_or(1u << dev);
    }
    return VRWKV_OK;
}

static int sm_count() {
    static int n = 0;
    if (!n) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) n = 148;
    }
    return n;
}

static int make_tile_map(CUtensorMap* m, const void* base, int B, int T, int H) {  // [64 steps][64 channels] bf16 boxes, SWIZZLE_128B
    return vrwkv_encode_2d(m, base, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (uint64_t)H * WKV_N, (uint64_t)B * T,
                           (uint64_t)H * WKV_N * 2, WKV_N, X6_L, CU_TENSOR_MAP_SWIZZLE_128B);
}

// round-2 forward: chunk-parallel persistent kernel, x6 products (wkv7_x6_fwd.cuh); `cache` (chunk checkpoints only):
// also write the chunk cache
static int launch_x6_fwd(const void* const* in, const Wkv7FwdArgs& a, bool chunk_ck, cudaStream_t st, void* cache = nullptr) {
    int rc = ensure_pool_keeps_memory();
    if (rc) return rc;
    CUtensorMap tm[6];
    for (int i = 0; i < 6; i++)
        if ((rc = make_tile_map(&tm[i], in[i], a.B, a.T, a.H))) return rc;
    const int BH = a.B * a.H, nitems = BH * (a.T / X6_L);
    const size_t sync_bytes = ((size_t)(BH + 1) * sizeof(int) + 255) & ~(size_t)255;
    const size_t chain_bytes = a.s ? 0 : (size_t)BH * 2 * WKV_N * WKV_N * sizeof(float);
    uint8_t* ws = nullptr;
    VRWKV_CUDA(cudaMallocAsync((void**)&ws, sync_bytes + chain_bytes, st));
    VRWKV_CUDA(cudaMemsetAsync(ws, 0, sync_bytes, st));
    X6FwdArgs xa{a.B, a.T, a.H, a.y, a.s, a.sa, a.state_in, a.state_out, chain_bytes ? (float*)(ws + sync_bytes) : nullptr, (int*)ws,
                 (uint8_t*)cache};
    const size_t smem = sizeof(X6FwdSmem) + 1024;
    // 16-step checkpoints only when a checkpoint tensor in the reference's layout was asked for
    auto kern = cache ? wkv7_x6_fwd_kernel<false, true> : (chunk_ck || !a.s) ? wkv7_x6_fwd_kernel<false> : wkv7_x6_fwd_kernel<true>;
    VRWKV_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int grid = nitems < sm_count() ? nitems : sm_count();
    kern<<<grid, X6_THREADS, smem, st>>>(tm[0], tm[1], tm[2], tm[3], tm[4], tm[5], xa);
    VRWKV_CUDA(cudaGetLastError());
    vrwkv_count_launch(1);
    VRWKV_CUDA(cudaFreeAsync(ws, st));
    return VRWKV_OK;
}

// round-2 backward: one chunk-parallel persistent kernel, x3 products (wkv7_x6_bwd.cuh); `cache`: the forward's chunk cache
static int launch_x3_bwd(const uint16_t* w, const uint16_t* q, const uint16_t* k, const uint16_t* v, const uint16_t* a,
                         const uint16_t* b, const uint16_t* dy, const float* sa, const Wkv7BwdArgs& args, int ck_per_chunk,
                         cudaStream_t st, const void* cache = nullptr) {
    int rc = ensure_pool_keeps_memory();
    if (rc) return rc;
    const int B = args.B, T = args.T, H = args.H;
    CUtensorMap tm[7];
    const void* in[7] = {w, q, k, v, a, b, dy};
    for (int i = 0; i < 7; i++)
        if ((rc = make_tile_map(&tm[i], in[i], B, T, H))) return rc;
    const int BH = B * H, nitems = BH * (T / X6_L);
    const size_t sync_bytes = ((size_t)(BH + 1) * sizeof(int) + 255) & ~(size_t)255;
    const size_t ring_bytes = (size_t)BH * 2 * WKV_N * WKV_N * sizeof(float);
    uint8_t* ws = nullptr;
    VRWKV_CUDA(cudaMallocAsync((void**)&ws, sync_bytes + ring_bytes, st));
    VRWKV_CUDA(cudaMemsetAsync(ws, 0, sync_bytes, st));
    X3BwdArgs xa{B, T, H, w, q, k, a, b, sa, args.s, ck_per_chunk, (float*)(ws + sync_bytes), (int*)ws,
                 args.dw, args.dq, args.dk, args.dv, args.da, args.db, (const uint8_t*)cache};
    const size_t smem = sizeof(X3BwdSmem) + 1024;
    auto kern = cache ? wkv7_x3_bwd_kernel<true> : wkv7_x3_bwd_kernel<false>;
    VRWKV_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int grid = nitems < sm_count() ? nitems : sm_count();
    kern<<<grid, X6_THREADS, smem, st>>>(tm[0], tm[1], tm[2], tm[3], tm[4], tm[5], tm[6], xa);
    VRWKV_CUDA(cudaGetLastError());
    vrwkv_count_launch(1);
    VRWKV_CUDA(cudaFreeAsync(ws, st));
    return VRWKV_OK;
}

// backward entirely on the tensor cores: dS boundary scan, then one CTA per (batch, head, chunk)
static int launch_bwd_chunked(const uint16_t* w, const uint16_t* q, const uint16_t* k, const uint16_t* v, const uint16_t* a,
                              const uint16_t* b, const uint16_t* dy, const float* sa, const Wkv7BwdArgs& args, int ck_per_chunk,
                              cudaStream_t st) {
    const int B = args.B, T = args.T, H = args.H, nch = T / CK_L;
    int rc = ensure_pool_keeps_memory();
    if (rc) return rc;
    const size_t nstate = (size_t)B * H * nch * WKV_N * WKV_N;
    float* ws = nullptr;  // [ds | gws]
    VRWKV_CUDA(cudaMallocAsync((void**)&ws, 2 * nstate * sizeof(float), st));
    CUtensorMap cm[7];
    const void* in[7] = {w, q, k, v, a, b, dy};
    for (int i = 0; i < 7; i++)
        if ((rc = make_chunk_map(&cm[i], in[i], B, T, H))) return rc;
    if (nch > 1) {
        const size_t smem = sizeof(Wkv7DstateSmem) + 1024;
        VRWKV_CUDA(cudaFuncSetAttribute(wkv7_chunk_dstate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        Wkv7DstateArgs da{B, T, H, ws};
        wkv7_chunk_dstate_kernel<<<dim3(H, B), CK_THREADS, smem, st>>>(cm[0], cm[1], cm[4], cm[5], cm[6], da);
        VRWKV_CUDA(cudaGetLastError());
        vrwkv_count_launch(1);
    }
    const size_t smem = sizeof(Wkv7ChunkBwdSmem) + 1024;
    VRWKV_CUDA(cudaFuncSetAttribute(wkv7_chunk_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    Wkv7ChunkBwdArgs ca{B, T, H, w, q, k, v, a, b, dy, sa, args.s, ck_per_chunk, ws, ws + nstate, args.dw, args.dq, args.dk, args.dv, args.da, args.db};
    wkv7_chunk_bwd_kernel<<<dim3(H, B, nch), CK_THREADS, smem, st>>>(cm[0], cm[1], cm[2], cm[3], cm[4], cm[5], cm[6], ca);
    VRWKV_CUDA(cudaGetLastError());
    vrwkv_count_launch(1);
    VRWKV_CUDA(cudaFreeAsync(ws, st));
    return VRWKV_OK;
}

static int check_common(int B, int T, int H, const void* const* ptrs, int nptr) {
    if (B <= 0 || T <= 0 || H <= 0) return vrwkv_fail(VRWKV_EINVAL, "wkv7: B,T,H must be positive (got %d,%d,%d)", B, T, H);
    if ((long long)B * T >= (1ll << 31)) return vrwkv_fail(VRWKV_EUNSUP, "wkv7: B*T too large");
    for (int i = 0; i < nptr; i++) {
        if (!ptrs[i]) return vrwkv_fail(VRWKV_EINVAL, "wkv7: null pointer (arg %d)", i);
        if (((uintptr_t)ptrs[i]) & 15) return vrwkv_fail(VRWKV_EINVAL, "wkv7: pointer %d not 16-byte aligned", i);
    }
    return VRWKV_OK;
}

static unsigned default_flags() {  // VRWKV_WKV7_BOUNDED_DECAY=1 lets the drop-in op use the chunked kernels too
    static const unsigned f = [] {
        const char* e = getenv("VRWKV_WKV7_BOUNDED_DECAY");
        return (e && e[0] == '1') ? (unsigned)VRWKV_WKV7_BOUNDED_DECAY : 0u;
    }();
    return f;
}

extern "C" int vrwkv_wkv7_domain_check(void) {
    int flag = 0, zero = 0;
    VRWKV_CUDA(cudaMemcpyFromSymbol(&flag, g_chunk_domain_err, sizeof(int)));
    if (flag) VRWKV_CUDA(cudaMemcpyToSymbol(g_chunk_domain_err, &zero, sizeof(int)));
    return flag ? vrwkv_fail(VRWKV_EINVAL, "wkv7 chunked kernels: sum over a 64-step chunk of exp(w) exceeded 80 "
                                           "(VRWKV_WKV7_BOUNDED_DECAY promised exp(w) <= 0.607)") : VRWKV_OK;
}

extern "C" int vrwkv_wkv7_forward_ex(int B, int T, int H, const uint16_t* w, const uint16_t* q, const uint16_t* k,
                                     const uint16_t* v, const uint16_t* a, const uint16_t* b, uint16_t* y, float* s,
                                     float* sa, const float* state_in, float* state_out, unsigned flags, void* stream) {
    const void* ptrs[] = {w, q, k, v, a, b, y};
    int rc = check_common(B, T, H, ptrs, 7);
    if (rc) return rc;
    if (s && (T % WKV_TC) != 0)
        return vrwkv_fail(VRWKV_EINVAL, "wkv7 forward: T=%d must be a multiple of %d when checkpoints are requested", T, WKV_TC);
    if ((((uintptr_t)s) | ((uintptr_t)sa) | ((uintptr_t)state_in) | ((uintptr_t)state_out)) & 15)
        return vrwkv_fail(VRWKV_EINVAL, "wkv7 forward: s/sa/state pointers must be 16-byte aligned");
    CUtensorMap tm[6];
    const void* in[6] = {w, q, k, v, a, b};
    for (int i = 0; i < 6; i++)
        if ((rc = make_stream_map(&tm[i], in[i], B, T, H, 2))) return rc;
    Wkv7FwdArgs args{B, T, H, y, s, sa, state_in, state_out};
    cudaStream_t st = (cudaStream_t)stream;
    int var = g_fwd_variant.load();
    if (var == 0) var = ((flags | default_flags()) & VRWKV_WKV7_BOUNDED_DECAY) ? ((flags & VRWKV_WKV7_TF32) ? 3 : 6) : 1;
    if (flags & VRWKV_WKV7_CHUNK_CHECKPOINTS) {
        if (!(flags & VRWKV_WKV7_BOUNDED_DECAY) || (T % CK_L) != 0 || state_in || state_out)
            return vrwkv_fail(VRWKV_EINVAL, "wkv7 forward: CHUNK_CHECKPOINTS needs BOUNDED_DECAY, T %% 64 == 0 and no carried state");
        if (var != 6 && var != 3) var = 6;
    }
    if ((var == 3 || var == 6) && (T % CK_L) != 0) var = 1;  // the chunked kernels walk 64 steps at a time
    switch (var) {
        case 3: return launch_chunk_fwd(in, args, (flags & VRWKV_WKV7_CHUNK_CHECKPOINTS) != 0, st);  // round-1 TF32 tensor-core kernel
        case 6: return launch_x6_fwd(in, args, (flags & VRWKV_WKV7_CHUNK_CHECKPOINTS) != 0, st);     // round-2 x6 chunk-parallel kernel
        case 1: return launch_fwd2<4, 4>(tm, args, st);  // 4 rows x 8 columns per thread, 4 compute warps
        case 2: return launch_fwd2<2, 4>(tm, args, st);  // 2 rows x 8 columns per thread, 8 compute warps
        default: return vrwkv_fail(VRWKV_EINVAL, "wkv7 forward: unknown variant %d", var);
    }
}

extern "C" int vrwkv_wkv7_forward_state(int B, int T, int H, const uint16_t* w, const uint16_t* q, const uint16_t* k,
                                        const uint16_t* v, const uint16_t* a, const uint16_t* b, uint16_t* y, float* s,
                                        float* sa, const float* state_in, float* state_out, void* stream) {
    return vrwkv_wkv7_forward_ex(B, T, H, w, q, k, v, a, b, y, s, sa, state_in, state_out, 0u, stream);
}

extern "C" int vrwkv_wkv7_forward(int B, int T, int H, const uint16_t* w, const uint16_t* q, const uint16_t* k,
                                  const uint16_t* v, const uint16_t* a, const uint16_t* b, uint16_t* y, float* s,
                                  float* sa, void* stream) {
    if (!s || !sa) return vrwkv_fail(VRWKV_EINVAL, "wkv7 forward: s and sa are required (model.py:53-54)");
    if (T % WKV_TC) return vrwkv_fail(VRWKV_EINVAL, "wkv7 forward: T=%d must be a multiple of %d (model.py:49)", T, WKV_TC);
    return vrwkv_wkv7_forward_state(B, T, H, w, q, k, v, a, b, y, s, sa, nullptr, nullptr, stream);
}

extern "C" int vrwkv_wkv7_backward_ex(int B, int T, int H, const uint16_t* w, const uint16_t* q, const uint16_t* k,
                                      const uint16_t* v, const uint16_t* a, const uint16_t* b, const uint16_t* dy,
                                      const float* s, const float* sa, uint16_t* dw, uint16_t* dq, uint16_t* dk,
                                      uint16_t* dv, uint16_t* da, uint16_t* db, unsigned flags, void* stream) {
    const void* ptrs[] = {w, q, k, v, a, b, dy, s, sa, dw, dq, dk, dv, da, db};
    int rc = check_common(B, T, H, ptrs, 15);
    if (rc) return rc;
    if (T % WKV_TC) return vrwkv_fail(VRWKV_EINVAL, "wkv7 backward: T=%d must be a multiple of %d (wkv7_cuda.cu:136)", T, WKV_TC);
    CUtensorMap tm[8];
    const void* in[7] = {w, q, k, v, a, b, dy};
    for (int i = 0; i < 7; i++)
        if ((rc = make_stream_map(&tm[i], in[i], B, T, H, 2))) return rc;
    if ((rc = make_stream_map(&tm[7], sa, B, T, H, 4))) return rc;
    Wkv7BwdArgs args{B, T, H, s, dw, dq, dk, dv, da, db};
    cudaStream_t st = (cudaStream_t)stream;
    int var = g_bwd_variant.load();
    // default with bounded decay: the step-by-step kernel unless the caller kept chunk-granularity checkpoints (then the
    // chunked kernels are the only ones that can read them)
    if (var == 0) {
        if (!((flags | default_flags()) & VRWKV_WKV7_BOUNDED_DECAY)) var = 1;
        else if (flags & VRWKV_WKV7_TF32) var = 5;
        else var = (flags & VRWKV_WKV7_CHUNK_CHECKPOINTS) ? 7 : 1;
    }
    if (flags & VRWKV_WKV7_CHUNK_CHECKPOINTS) {
        if (!(flags & VRWKV_WKV7_BOUNDED_DECAY) || (T % CK_L) != 0 || (var != 5 && var != 7))
            return vrwkv_fail(VRWKV_EINVAL, "wkv7 backward: CHUNK_CHECKPOINTS needs BOUNDED_DECAY, T %% 64 == 0 and a chunked kernel");
    }
    if ((var == 3 || var == 4 || var == 5 || var == 7) && (T % CK_L) != 0) var = 1;
    switch (var) {
        case 7: return launch_x3_bwd(w, q, k, v, a, b, dy, sa, args, (flags & VRWKV_WKV7_CHUNK_CHECKPOINTS) ? 1 : CK_L / WKV_TC, st);
        case 5: return launch_bwd_chunked(w, q, k, v, a, b, dy, sa, args, (flags & VRWKV_WKV7_CHUNK_CHECKPOINTS) ? 1 : CK_L / WKV_TC, st);
        case 3: return launch_bwd_segmented<4, 3>(tm, w, q, a, b, dy, args, st);  // needs sum_chunk exp(w) < ~85
        case 4: return launch_bwd_segmented<2, 3>(tm, w, q, a, b, dy, args, st);  // same, 2 rows per thread (8 compute warps)
        case 1: return launch_bwd2<4, 3>(tm, args, st);
        case 2: return launch_bwd2<2, 3>(tm, args, st);
        default: return vrwkv_fail(VRWKV_EINVAL, "wkv7 backward: unknown variant %d", var);
    }
}

extern "C" int vrwkv_wkv7_backward(int B, int T, int H, const uint16_t* w, const uint16_t* q, const uint16_t* k,
                                   const uint16_t* v, const uint16_t* a, const uint16_t* b, const uint16_t* dy,
                                   const float* s, const float* sa, uint16_t* dw, uint16_t* dq, uint16_t* dk,
                                   uint16_t* dv, uint16_t* da, uint16_t* db, void* stream) {
    return vrwkv_wkv7_backward_ex(B, T, H, w, q, k, v, a, b, dy, s, sa, dw, dq, dk, dv, da, db, 0u, stream);
}

// ---- chunk cache (model path) ----
static const unsigned kCacheFlags = VRWKV_WKV7_BOUNDED_DECAY | VRWKV_WKV7_CHUNK_CHECKPOINTS;

extern "C" size_t vrwkv_wkv7_cache_bytes(int B, int T, int H) {
    if (B <= 0 || T <= 0 || H <= 0 || T % X6_L) return 0;
    return (size_t)B * H * (T / X6_L) * XC_ITEM_BYTES;
}

static int check_cache_call(const char* what, int T, const void* s, const void* sa, const void* cache, unsigned flags) {
    if ((flags & (kCacheFlags | VRWKV_WKV7_TF32)) != kCacheFlags)
        return vrwkv_fail(VRWKV_EINVAL, "%s: needs flags BOUNDED_DECAY | CHUNK_CHECKPOINTS (and not TF32), got 0x%x", what, flags);
    if (T % X6_L) return vrwkv_fail(VRWKV_EINVAL, "%s: T=%d must be a multiple of %d", what, T, X6_L);
    if (!s || !sa || !cache) return vrwkv_fail(VRWKV_EINVAL, "%s: s, sa and cache are required", what);
    if (((uintptr_t)s | (uintptr_t)sa) & 15) return vrwkv_fail(VRWKV_EINVAL, "%s: s and sa must be 16-byte aligned", what);
    if ((uintptr_t)cache & 127) return vrwkv_fail(VRWKV_EINVAL, "%s: cache must be 128-byte aligned", what);
    return VRWKV_OK;
}

extern "C" int vrwkv_wkv7_forward_cache(int B, int T, int H, const uint16_t* w, const uint16_t* q, const uint16_t* k,
                                        const uint16_t* v, const uint16_t* a, const uint16_t* b, uint16_t* y, float* s,
                                        float* sa, void* cache, unsigned flags, void* stream) {
    const void* ptrs[] = {w, q, k, v, a, b, y};
    int rc = check_common(B, T, H, ptrs, 7);
    if (rc || (rc = check_cache_call("wkv7 forward_cache", T, s, sa, cache, flags))) return rc;
    const void* in[6] = {w, q, k, v, a, b};
    Wkv7FwdArgs args{B, T, H, y, s, sa, nullptr, nullptr};
    return launch_x6_fwd(in, args, true, (cudaStream_t)stream, cache);
}

extern "C" int vrwkv_wkv7_backward_cache(int B, int T, int H, const uint16_t* w, const uint16_t* q, const uint16_t* k,
                                         const uint16_t* v, const uint16_t* a, const uint16_t* b, const uint16_t* dy,
                                         const float* s, const float* sa, const void* cache, uint16_t* dw, uint16_t* dq,
                                         uint16_t* dk, uint16_t* dv, uint16_t* da, uint16_t* db, unsigned flags, void* stream) {
    const void* ptrs[] = {w, q, k, v, a, b, dy, s, sa, dw, dq, dk, dv, da, db};
    int rc = check_common(B, T, H, ptrs, 15);
    if (rc || (rc = check_cache_call("wkv7 backward_cache", T, s, sa, cache, flags))) return rc;
    Wkv7BwdArgs args{B, T, H, s, dw, dq, dk, dv, da, db};
    return launch_x3_bwd(w, q, k, v, a, b, dy, sa, args, 1, (cudaStream_t)stream, cache);
}
