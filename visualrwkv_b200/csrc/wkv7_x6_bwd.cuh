// wkv7_x6_bwd.cuh — WKV7 backward, round 2: one chunk-parallel kernel on the tcgen05 tensor cores ("x3" products:
// two bf16 parts per operand, wkv7_x6_common.cuh).  Replaces the reference's serial reverse-time walk
// (VisualRWKV-v7/v7.00/cuda/wkv7_cuda.cu:54-130) for callers that promise bounded decay; the algebra is the hand-derived
// reverse pass of the chunk form (the chunk_backward restatement kept with the tests, checked against the fp64 adjoint of the
// step-by-step oracle):
//     dZ = dS_L E_L                          [dU;dV] = [Bt;Kt] dZ^T + [A_qb|A_qk]^T dY        dR = (I - A_ab)^-T dU
//     dS_0 = dZ + dR^T At + dY^T Qt          (the only quantity the previous chunk waits for)
//     dA = mask([dR;dY] [U;V]^T)             dV += A_ak^T dR
//     [dAt;dQt] = [dR;dY] S_0 + dA [Bt;Kt]   [dBt;dKt] = [U;V] dZ + dA^T [At;Qt]
//     da = dAt E_{t-1}, dq = dQt E_t, dk = dKt / E_t, db = dBt / E_t
//     dG_t = dq q - dk k - db b + (da a)_{t+1}  (+ sum_i dS_L S_L at t = 63);  dw = (reverse cumsum of dG) * (-e^w)
// Work item = one 64-step chunk of one (batch, head); a persistent grid takes items in REVERSE chunk-major order (the last
// chunk of every (b,h) first).  Everything up to dU's local part and the triangular inverse does not depend on dS_L; then
// the item waits (acquire flag) for the chunk after it to publish dL/dS at its start, runs the short dS_0 chain
// (3 products), publishes dS_0 (release flag) and finishes its gradients while the chunk before it proceeds.  dL/dS lives
// in a 2-slot ring per (b,h) (3 MB in all: L2-resident).  Inputs besides the seven bf16 streams: the forward's `sa`
// (rows of U) and its state checkpoints `s` (S at the start / end of the chunk).
#pragma once
#include "wkv7_chunk_common.cuh"
#include "wkv7_x6_common.cuh"

namespace vrwkv {

struct X3BwdArgs {
    int B, T, H;
    const uint16_t *w, *q, *k, *a, *b;   // re-read by the epilogue (L2)
    const float* sa;                     // [B,T,H,64]
    const float* s;                      // transposed state checkpoints, ck_per_chunk per 64-step chunk
    int ck_per_chunk;                    // 4: the reference's [B,H,T/16,64,64]; 1: [B,H,T/64,64,64]
    float* ds;                           // [B*H][2][64*64] ring of dL/dS (row-major [i][j])
    int* sync;                           // [0] item counter, [1 + bh] chunks finished (from the end); zeroed before launch
    uint16_t *dw, *dq, *dk, *dv, *da, *db;
    const uint8_t* cache;                // CACHE: the forward's chunk cache, [B*H*T/64][8 tiles][8 KB] (wkv7_x6_common.cuh)
};

struct alignas(1024) X3BwdSmem {
    uint8_t r1[5 * BT_BYTES];     // raw w,q,k,a,b tiles -> M = A_ab -> Tinv fp32 (+0, 16 KB) | Tinv pair (+16384) | spare 8 KB;
                                  // dU pair at +0 once the inverse is done; S_0 pair at +16384 once dR exists
    uint8_t r2[4 * BT_BYTES];     // [A_qb | A_qk] pairs (part p at p*16384) -> [U_p0][V raw][U_p1][zeros]
    uint8_t aq[4 * BT_BYTES];     // [At;Qt] pairs (part p at p*16384: At tile, Qt tile)
    uint8_t bk[4 * BT_BYTES];     // [Bt;Kt] pairs
    uint8_t drdy[4 * BT_BYTES];   // [dR_p0][dY raw][dR_p1][zeros]
    uint8_t dz[2 * BT_BYTES];     // dZ pair [i][j]
    uint8_t sak[2 * BT_BYTES];    // A_ak pair [t][s]
    uint8_t emat[16384];          // E_t fp32 [t][j] (m64 layout)
    float esc[1024];              // inverse scratch; P1: per row-group decay products; epilogue: partial sums
    float el[WKV_N], gl[WKV_N];
    uint64_t bar_in, bar_dy, bar_v, bar_mma, bar_c3;
    uint32_t tmem_base;
    int next_item;
    uint64_t bar_ca;              // CACHE: the item's chunk-cache tiles
};

// CACHE: [A_qb|A_qk], A_ak and Tinv come from the forward's chunk cache instead of the scores batch, P2 and the inverse.
// They land in r2, sak and the dR slots of drdy (Tinv part p at p*16384), all dead once the item's dA batch has finished,
// so the next item's cache loads are issued there, together with its raw-input loads.
template <bool CACHE = false>
__global__ void __launch_bounds__(X6_THREADS, 1)
wkv7_x3_bwd_kernel(const __grid_constant__ CUtensorMap tm_w, const __grid_constant__ CUtensorMap tm_q,
                   const __grid_constant__ CUtensorMap tm_k, const __grid_constant__ CUtensorMap tm_v,
                   const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                   const __grid_constant__ CUtensorMap tm_dy, const X3BwdArgs p) {
    constexpr int N = WKV_N, L = X6_L;
    extern __shared__ __align__(1024) uint8_t x3_smem_bytes[];
    X3BwdSmem& sm = *reinterpret_cast<X3BwdSmem*>((reinterpret_cast<uintptr_t>(x3_smem_bytes) + 1023) & ~(uintptr_t)1023);
    uint8_t* const mab = sm.r1;              // fp32 A_ab -> Tinv
    uint8_t* const tinv = sm.r1 + 16384;     // Tinv pair [t][s]; diag scratch of the inverse before that
    uint8_t* const du = sm.r1;               // dU pair [t][i]
    uint8_t* const s0p = sm.r1 + 16384;      // S_0 pair [j][i]

    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int qd = warp & 3, cs = warp >> 2;
    const int r = 32 * qd + lane;
    const int T = p.T, H = p.H, BH = p.B * p.H;
    const int nch = T / L, nitems = BH * nch;
    const size_t rstride = (size_t)H * N;

    if (tid == 0) {
        mbar_init(&sm.bar_in, 1);
        mbar_init(&sm.bar_dy, 1);
        mbar_init(&sm.bar_v, 1);
        mbar_init(&sm.bar_mma, 1);
        mbar_init(&sm.bar_c3, 1);
        if constexpr (CACHE) mbar_init(&sm.bar_ca, 1);
        fence_mbar_init();
        tma_prefetch_desc(&tm_w); tma_prefetch_desc(&tm_q); tma_prefetch_desc(&tm_k); tma_prefetch_desc(&tm_v);
        tma_prefetch_desc(&tm_a); tma_prefetch_desc(&tm_b); tma_prefetch_desc(&tm_dy);
        sm.next_item = atomicAdd(&p.sync[0], 1);
    }
    // the zero tile behind dR_p1 stays zero for the whole kernel
    *reinterpret_cast<uint4*>(sm.drdy + 3 * BT_BYTES + tid * 16) = make_uint4(0u, 0u, 0u, 0u);
    __syncwarp();
    if (warp == 0) tmem_alloc<512>(&sm.tmem_base);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = sm.tmem_base;
    const uint32_t tm_row = tmem + ((uint32_t)(32 * qd) << 16);
    // TMEM columns: scores 0-127 (then dA), dA^T 128-255, [dU;dV] 256-319, dR 320-383 (then [dAt;dQt]), dS_0 384-447, [dBt;dKt] 448-511
    constexpr uint32_t C_SC = 0, C_DA = 0, C_DAT = 128, C_UV = 256, C_R = 320, C_AQ = 320, C_DS0 = 384, C_BK = 448;

    const uint32_t b4 = smem_u32(&sm) >> 4;
    const uint32_t O_R1 = (uint32_t)(sm.r1 - (uint8_t*)&sm), O_R2 = (uint32_t)(sm.r2 - (uint8_t*)&sm), O_AQ = (uint32_t)(sm.aq - (uint8_t*)&sm),
                   O_BK = (uint32_t)(sm.bk - (uint8_t*)&sm), O_DRDY = (uint32_t)(sm.drdy - (uint8_t*)&sm), O_DZ = (uint32_t)(sm.dz - (uint8_t*)&sm),
                   O_SAK = (uint32_t)(sm.sak - (uint8_t*)&sm);
    const uint32_t O_TINV = O_R1 + 16384, O_DU = O_R1, O_S0P = O_R1 + 16384;

    auto item_coords = [&](int item, int& c, int& bh, int& bb, int& hh) {
        const int cr = item / BH;
        bh = item - cr * BH;
        c = nch - 1 - cr;
        bb = bh / H;
        hh = bh - bb * H;
    };
    auto load_in5 = [&](int item) {
        int c, bh, bb, hh;
        item_coords(item, c, bh, bb, hh);
        const int x0 = hh * N, y0 = bb * T + c * L;
        mbar_arrive_expect_tx(&sm.bar_in, 5 * BT_BYTES);
        tma_load_2d(sm.r1 + 0 * BT_BYTES, &tm_w, x0, y0, &sm.bar_in);
        tma_load_2d(sm.r1 + 1 * BT_BYTES, &tm_q, x0, y0, &sm.bar_in);
        tma_load_2d(sm.r1 + 2 * BT_BYTES, &tm_k, x0, y0, &sm.bar_in);
        tma_load_2d(sm.r1 + 3 * BT_BYTES, &tm_a, x0, y0, &sm.bar_in);
        tma_load_2d(sm.r1 + 4 * BT_BYTES, &tm_b, x0, y0, &sm.bar_in);
    };
    auto load_dy = [&](int item) {
        int c, bh, bb, hh;
        item_coords(item, c, bh, bb, hh);
        mbar_arrive_expect_tx(&sm.bar_dy, BT_BYTES);
        tma_load_2d(sm.drdy + BT_BYTES, &tm_dy, hh * N, bb * T + c * L, &sm.bar_dy);
    };
    auto load_v = [&](int item) {
        int c, bh, bb, hh;
        item_coords(item, c, bh, bb, hh);
        mbar_arrive_expect_tx(&sm.bar_v, BT_BYTES);
        tma_load_2d(sm.r2 + BT_BYTES, &tm_v, hh * N, bb * T + c * L, &sm.bar_v);
    };
    auto load_cache = [&](int item) {
        int c, bh, bb, hh;
        item_coords(item, c, bh, bb, hh);
        const uint8_t* src = p.cache + (size_t)(c * BH + bh) * XC_ITEM_BYTES;
        mbar_arrive_expect_tx(&sm.bar_ca, XC_ITEM_BYTES);
        bulk_load_1d(sm.r2, src + XC_QB0 * BT_BYTES, 4 * BT_BYTES, &sm.bar_ca);   // [A_qb|A_qk] pairs, part p at p*16384
        bulk_load_1d(sm.sak, src + XC_AK0 * BT_BYTES, 2 * BT_BYTES, &sm.bar_ca);
        bulk_load_1d(sm.drdy, src + XC_TI0 * BT_BYTES, BT_BYTES, &sm.bar_ca);
        bulk_load_1d(sm.drdy + 16384, src + XC_TI1 * BT_BYTES, BT_BYTES, &sm.bar_ca);
    };
    int item = sm.next_item;
    if (tid == 0 && item < nitems) {
        load_in5(item);
        load_dy(item);
        if constexpr (CACHE) load_cache(item);
    }
    __syncwarp();

    uint32_t ph_in = 0, ph_dy = 0, ph_v = 0, ph_mma = 0, ph_c3 = 0, ph_ca = 0;
#ifdef VRWKV_PHASE_STAMPS   // development aid (scripts/dbg_x6_stamps.py, dbg_x3_stamps.py): build with VRWKV_PHASE_STAMPS=1
    float* const dbg = (blockIdx.x == 0 && tid == 0) ? g_chunk_dbg : nullptr;
    int lt = 0, tsi = 0;
    long long tstamp0 = 0;
    auto stamp = [&]() {
        if (dbg && lt == 2) {
            const long long now = clock64();
            if (tsi == 0) tstamp0 = now;
            dbg[3072 + tsi++] = (float)(now - tstamp0);
        }
    };
#else
    int lt = 0;
    auto stamp = [] {};
#endif
    auto mma_wait = [&]() {
        mbar_wait(&sm.bar_mma, ph_mma & 1);
        ph_mma++;
        tc_fence_after();
        __syncwarp();
    };
    auto operands_ready = [&]() {
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();
    };
    auto f8 = [](const uint32_t* v, float (&x)[8]) {
#pragma unroll
        for (int e = 0; e < 8; e++) x[e] = __uint_as_float(v[e]);
    };

    while (item < nitems) {
        int c, bh, bb, hh;
        item_coords(item, c, bh, bb, hh);
        const size_t row0 = ((size_t)bb * T + (size_t)c * L) * rstride + (size_t)hh * N;   // element offset of (t = 0, channel 0)
        const int ckpc = p.ck_per_chunk;
        const float* s_start = c > 0 ? p.s + ((size_t)bh * nch * ckpc + (size_t)c * ckpc - 1) * (N * N) : nullptr;   // S_0, transposed [j][i]
        const float* s_end = p.s + ((size_t)bh * nch * ckpc + (size_t)(c + 1) * ckpc - 1) * (N * N);                  // S_L
        const float* ds_in = p.ds + ((size_t)bh * 2 + (c & 1)) * (N * N);          // dL/dS at the end of this chunk (c < nch-1)
        float* ds_out = p.ds + ((size_t)bh * 2 + ((c + 1) & 1)) * (N * N);         // ... at its start
        const bool last = (c == nch - 1);
        {   // U (= sa rows) and S_0 come from global memory later: start pulling them into L2
            const int t = tid >> 3, i0 = 8 * (tid & 7);
            asm volatile("prefetch.global.L2 [%0];" ::"l"(p.sa + row0 + (size_t)t * rstride + i0));
            if (c > 0) asm volatile("prefetch.global.L2 [%0];" ::"l"(s_start + t * N + i0));
        }
        stamp();  // 0
        // ================= P1: decay products (kept in emat), scaled operands =================
        mbar_wait(&sm.bar_in, ph_in & 1);
        ph_in++;
        {
            const int rg = warp, j0 = 2 * lane;
            float c0[4], c1[4];
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const uint32_t ww = *reinterpret_cast<const uint32_t*>(sm.r1 + bt_off(4 * rg + k, j0));
                const float d0 = __expf(-__expf(bf16lo_to_f32(ww))), d1 = __expf(-__expf(bf16hi_to_f32(ww)));
                c0[k] = k ? c0[k - 1] * d0 : d0;
                c1[k] = k ? c1[k - 1] * d1 : d1;
            }
            *reinterpret_cast<float2*>(&sm.esc[rg * N + j0]) = make_float2(c0[3], c1[3]);
            __syncthreads();
            float pre0 = 1.f, pre1 = 1.f;
#pragma unroll
            for (int g = 0; g < 15; g++) {
                const float2 pp = *reinterpret_cast<const float2*>(&sm.esc[g * N + j0]);
                pre0 *= (g < rg) ? pp.x : 1.f;
                pre1 *= (g < rg) ? pp.y : 1.f;
            }
            float Ep0 = pre0, Ep1 = pre1;
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const int t = 4 * rg + k;
                const float E0 = pre0 * c0[k], E1 = pre1 * c1[k];
                const float F0 = __fdividef(1.f, E0), F1 = __fdividef(1.f, E1);
                const uint32_t off = bt_off(t, j0);
                const uint32_t qq = *reinterpret_cast<const uint32_t*>(sm.r1 + 1 * BT_BYTES + off);
                const uint32_t kk = *reinterpret_cast<const uint32_t*>(sm.r1 + 2 * BT_BYTES + off);
                const uint32_t aa = *reinterpret_cast<const uint32_t*>(sm.r1 + 3 * BT_BYTES + off);
                const uint32_t bb_ = *reinterpret_cast<const uint32_t*>(sm.r1 + 4 * BT_BYTES + off);
                uint32_t s0, s1;
                split2x2(bf16lo_to_f32(aa) * Ep0, bf16hi_to_f32(aa) * Ep1, s0, s1);
                *reinterpret_cast<uint32_t*>(sm.aq + off) = s0;
                *reinterpret_cast<uint32_t*>(sm.aq + 16384 + off) = s1;
                split2x2(bf16lo_to_f32(qq) * E0, bf16hi_to_f32(qq) * E1, s0, s1);
                *reinterpret_cast<uint32_t*>(sm.aq + BT_BYTES + off) = s0;
                *reinterpret_cast<uint32_t*>(sm.aq + 16384 + BT_BYTES + off) = s1;
                split2x2(bf16lo_to_f32(bb_) * F0, bf16hi_to_f32(bb_) * F1, s0, s1);
                *reinterpret_cast<uint32_t*>(sm.bk + off) = s0;
                *reinterpret_cast<uint32_t*>(sm.bk + 16384 + off) = s1;
                split2x2(bf16lo_to_f32(kk) * F0, bf16hi_to_f32(kk) * F1, s0, s1);
                *reinterpret_cast<uint32_t*>(sm.bk + BT_BYTES + off) = s0;
                *reinterpret_cast<uint32_t*>(sm.bk + 16384 + BT_BYTES + off) = s1;
                *reinterpret_cast<float2*>(m64_ptr(sm.emat, t, j0)) = make_float2(E0, E1);
                if (t == L - 1) {
                    *reinterpret_cast<float2*>(&sm.el[j0]) = make_float2(E0, E1);
                    if (E0 < 1e-30f || E1 < 1e-30f) g_chunk_domain_err = 1;
                }
                Ep0 = E0;
                Ep1 = E1;
            }
        }
        operands_ready();
        stamp();  // 1
        if constexpr (CACHE) {
            stamp();  // 2
            stamp();  // 3
            // ================= [dU;dV] = [A_qb|A_qk]^T dY with the forward's tiles =================
            if (warp == 0) {
                mbar_wait(&sm.bar_ca, ph_ca & 1);
                mbar_wait(&sm.bar_dy, ph_dy & 1);
                if (elect_one()) {
                    tc_fence_after();
                    mma_x2b<64, 1, 1>(tmem + C_UV, b4, O_R2, 16384, O_DRDY + BT_BYTES, false);
                    umma_commit(&sm.bar_mma);
                }
                __syncwarp();
            }
            ph_ca++;
            ph_dy++;
            mma_wait();
        } else {
            // ================= scores = [At;Qt] [Bt;Kt]^T =================
            if (warp == 0) {
                if (elect_one()) {
                    tc_fence_after();
                    mma_x3<128, 0, 0>(tmem + C_SC, b4, O_AQ, 16384, O_BK, 16384, false);
                    umma_commit(&sm.bar_mma);
                }
                __syncwarp();
            }
            mma_wait();
            stamp();  // 2
            // ================= P2: masked scores: A_ab fp32 (inverse), [A_qb|A_qk] and A_ak operands =================
            {
                uint32_t v[32];
                tmem_ld32(tm_row + C_SC + 32 * cs, v);
                const int tq = r & 63;
                const bool incl = r >= 64;
                float o[32];
#pragma unroll
                for (int e = 0; e < 32; e++) {
                    const int s = 32 * (cs & 1) + e;
                    const bool keep = incl ? (s <= tq) : (s < tq);
                    o[e] = keep ? __uint_as_float(v[e]) : 0.f;
                }
                if (incl) {   // q rows: A_qb (cs 0,1) -> r2 tile 0, A_qk (cs 2,3) -> r2 tile 1
                    uint8_t* dst = sm.r2 + (cs >> 1) * BT_BYTES;
#pragma unroll
                    for (int cc = 0; cc < 4; cc++) {
                        const float x8[8] = {o[8 * cc], o[8 * cc + 1], o[8 * cc + 2], o[8 * cc + 3], o[8 * cc + 4], o[8 * cc + 5], o[8 * cc + 6], o[8 * cc + 7]};
                        store_pair8(dst + bt_chunk(tq, 4 * (cs & 1) + cc), 16384, x8);
                    }
                } else if (cs < 2) {   // A_ab
#pragma unroll
                    for (int cc = 0; cc < 8; cc++) *m64_chunk(mab, r, 8 * cs + cc) = make_float4(o[4 * cc], o[4 * cc + 1], o[4 * cc + 2], o[4 * cc + 3]);
                } else {               // A_ak
#pragma unroll
                    for (int cc = 0; cc < 4; cc++) {
                        const float x8[8] = {o[8 * cc], o[8 * cc + 1], o[8 * cc + 2], o[8 * cc + 3], o[8 * cc + 4], o[8 * cc + 5], o[8 * cc + 6], o[8 * cc + 7]};
                        store_pair8(sm.sak + bt_chunk(r, 4 * (cs & 1) + cc), BT_BYTES, x8);
                    }
                }
            }
            mbar_wait(&sm.bar_dy, ph_dy & 1);
            ph_dy++;
            operands_ready();
            stamp();  // 3
            // ================= [dU;dV] = [A_qb|A_qk]^T dY   (inverse meanwhile) =================
            if (warp == 0) {
                if (elect_one()) {
                    tc_fence_after();
                    mma_x2b<64, 1, 1>(tmem + C_UV, b4, O_R2, 16384, O_DRDY + BT_BYTES, false);
                    umma_commit(&sm.bar_mma);
                }
                __syncwarp();
            }
            tri_inverse_inplace(mab, sm.esc, reinterpret_cast<float*>(tinv), tid);
            {   // Tinv pair [t][s]
                const int t = tid >> 3, ch = tid & 7;
                const float4 lo = *m64_chunk(mab, t, 2 * ch), hi = *m64_chunk(mab, t, 2 * ch + 1);
                const float x8[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
                store_pair8(tinv + bt_chunk(t, ch), BT_BYTES, x8);
            }
            mma_wait();
        }
        stamp();  // 4
        // r2 is free: v tile, zero tile, next item's raw tiles cannot start yet (r1 holds Tinv)
        if (tid == 0) load_v(item);
        *reinterpret_cast<uint4*>(sm.r2 + 3 * BT_BYTES + tid * 16) = make_uint4(0u, 0u, 0u, 0u);
        // ================= incoming dL/dS: dZ = dS_L E_L (pair [i][j]); d/dG_L = sum_i dS_L S_L =================
        if (!last) {
            if (tid == 0) {
                const int* flag = p.sync + 1 + bh;
                const int need = nch - 1 - c;
                long long t0 = clock64();
                while (ld_acquire(flag) < need) {
                    if (clock64() - t0 > 20000000000LL) __trap();
                }
            }
            __syncthreads();
        }
        stamp();  // 5
        {
            const int i = tid >> 3, j0 = 8 * (tid & 7);
            float x8[8];
            if (!last) {
                const float4 lo = __ldcg(reinterpret_cast<const float4*>(ds_in + i * N + j0)), hi = __ldcg(reinterpret_cast<const float4*>(ds_in + i * N + j0 + 4));
                const float4 e0 = *reinterpret_cast<const float4*>(&sm.el[j0]), e1 = *reinterpret_cast<const float4*>(&sm.el[j0 + 4]);
                x8[0] = lo.x * e0.x; x8[1] = lo.y * e0.y; x8[2] = lo.z * e0.z; x8[3] = lo.w * e0.w;
                x8[4] = hi.x * e1.x; x8[5] = hi.y * e1.y; x8[6] = hi.z * e1.z; x8[7] = hi.w * e1.w;
            } else {
#pragma unroll
                for (int e = 0; e < 8; e++) x8[e] = 0.f;
            }
            store_pair8(sm.dz + bt_chunk(i, tid & 7), BT_BYTES, x8);
        }
        {
            const int j = tid & 63, ig = tid >> 6;
            float acc = 0.f;
            if (!last) {
                const float4 s0 = __ldg(reinterpret_cast<const float4*>(s_end + j * N + 8 * ig)), s1 = __ldg(reinterpret_cast<const float4*>(s_end + j * N + 8 * ig) + 1);
                const float sv[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
#pragma unroll
                for (int e = 0; e < 8; e++) acc = fmaf(__ldcg(ds_in + (size_t)(8 * ig + e) * N + j), sv[e], acc);
            }
            sm.esc[ig * N + j] = acc;
        }
        operands_ready();
        if (tid < N) {
            float x = 0.f;
#pragma unroll
            for (int k = 0; k < 8; k++) x += sm.esc[k * N + tid];
            sm.gl[tid] = x;
        }
        // ================= [dU;dV] += [Bt;Kt] dZ^T =================
        if (warp == 0) {
            if (elect_one()) {
                tc_fence_after();
                mma_x3<64, 0, 0>(tmem + C_UV, b4, O_BK, 16384, O_DZ, BT_BYTES, true);
                umma_commit(&sm.bar_mma);
            }
            __syncwarp();
        }
        mma_wait();
        stamp();  // 6
        // ================= P3: dU pair [t][i] (over the dead fp32 inverse) =================
        if (r < 64) {
            uint32_t v[16];
            tmem_ld16(tm_row + C_UV + 16 * cs, v);
#pragma unroll
            for (int hc = 0; hc < 2; hc++) {
                float x8[8];
                f8(v + 8 * hc, x8);
                store_pair8(du + bt_chunk(r, 2 * cs + hc), BT_BYTES, x8);
            }
        }
        operands_ready();
        // ================= dR = Tinv^T dU =================
        if (warp == 0) {
            if (elect_one()) {
                tc_fence_after();
                if constexpr (CACHE) mma_x3<64, 1, 1>(tmem + C_R, b4, O_DRDY, 16384, O_DU, BT_BYTES, false);
                else mma_x3<64, 1, 1>(tmem + C_R, b4, O_TINV, BT_BYTES, O_DU, BT_BYTES, false);
                umma_commit(&sm.bar_mma);
            }
            __syncwarp();
        }
        // meanwhile: U pair from sa (rows of U) into r2 tiles 0 and 2
        {
            const int t = tid >> 3, i0 = 8 * (tid & 7);
            const float4 lo = __ldg(reinterpret_cast<const float4*>(p.sa + row0 + (size_t)t * rstride + i0)), hi = __ldg(reinterpret_cast<const float4*>(p.sa + row0 + (size_t)t * rstride + i0) + 1);
            const float x8[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
            store_pair8(sm.r2 + bt_chunk(t, tid & 7), 16384, x8);
        }
        mma_wait();
        stamp();  // 7
        // ================= P4: dR pair [t][i]; S_0 pair [j][i] (over the dead Tinv pair) =================
        if (r < 64) {
            uint32_t v[16];
            tmem_ld16(tm_row + C_R + 16 * cs, v);
#pragma unroll
            for (int hc = 0; hc < 2; hc++) {
                float x8[8];
                f8(v + 8 * hc, x8);
                store_pair8(sm.drdy + bt_chunk(r, 2 * cs + hc), 16384, x8);
            }
        }
        {
            const int j = tid >> 3, i0 = 8 * (tid & 7);
            float x8[8];
            if (c > 0) {
                const float4 lo = __ldg(reinterpret_cast<const float4*>(s_start + j * N + i0)), hi = __ldg(reinterpret_cast<const float4*>(s_start + j * N + i0) + 1);
                x8[0] = lo.x; x8[1] = lo.y; x8[2] = lo.z; x8[3] = lo.w; x8[4] = hi.x; x8[5] = hi.y; x8[6] = hi.z; x8[7] = hi.w;
            } else {
#pragma unroll
                for (int e = 0; e < 8; e++) x8[e] = 0.f;
            }
            store_pair8(s0p + bt_chunk(j, tid & 7), BT_BYTES, x8);
        }
        mbar_wait(&sm.bar_v, ph_v & 1);
        ph_v++;
        operands_ready();
        stamp();  // 8
        // ================= dS_0 part (own commit), then everything else that needs dR =================
        if (warp == 0) {
            if (elect_one()) {
                tc_fence_after();
                mma_x3<64, 1, 1>(tmem + C_DS0, b4, O_DRDY, 16384, O_AQ, 16384, false);                        // dR^T At
                mma_x2a<64, 1, 1>(tmem + C_DS0, b4, O_DRDY + BT_BYTES, O_AQ + BT_BYTES, 16384, true);         // dY^T Qt
                umma_commit(&sm.bar_c3);
            }
            __syncwarp();
        }
        // ================= P5: publish dS_0 = dZ + dR^T At + dY^T Qt (the previous chunk is waiting for it) =================
        mbar_wait(&sm.bar_c3, ph_c3 & 1);
        ph_c3++;
        tc_fence_after();
        __syncwarp();
        uint32_t ds0v[16];
        if (c > 0 && r < N) tmem_ld16(tm_row + C_DS0 + 16 * cs, ds0v);
        tc_fence_before();
        __syncthreads();
        if (warp == 0) {
            if (elect_one()) {
                tc_fence_after();
                mma_x3<128, 0, 0>(tmem + C_DA, b4, O_DRDY, 16384, O_R2, 16384, false);                        // dA = [dR;dY][U;V]^T
                mma_x3<128, 0, 0>(tmem + C_DAT, b4, O_R2, 16384, O_DRDY, 16384, false);                       // dA^T
                mma_x3<64, 0, 0>(tmem + C_AQ, b4, O_DRDY, 16384, O_S0P, BT_BYTES, false);                     // [dR;dY] S_0
                mma_x3<64, 0, 1>(tmem + C_BK, b4, O_R2, 16384, O_DZ, BT_BYTES, false);                        // [U;V] dZ
                mma_x3<64, 1, 1>(tmem + C_UV, b4, O_SAK - BT_BYTES, BT_BYTES, O_DRDY, 16384, true);           // dV (rows 64-127) += A_ak^T dR
                umma_commit(&sm.bar_mma);
            }
            __syncwarp();
        }
        if (c > 0) {
            if (r < N) {
                const uint32_t* v = ds0v;
                float4* dst = reinterpret_cast<float4*>(ds_out + (size_t)r * N + 16 * cs);
#pragma unroll
                for (int c4 = 0; c4 < 4; c4++) {
                    float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (!last) {
                        z = __ldcg(reinterpret_cast<const float4*>(ds_in + (size_t)r * N + 16 * cs) + c4);
                        const float4 e = *reinterpret_cast<const float4*>(&sm.el[16 * cs + 4 * c4]);
                        z.x *= e.x; z.y *= e.y; z.z *= e.z; z.w *= e.w;
                    }
                    dst[c4] = make_float4(z.x + __uint_as_float(v[4 * c4]), z.y + __uint_as_float(v[4 * c4 + 1]), z.z + __uint_as_float(v[4 * c4 + 2]),
                                          z.w + __uint_as_float(v[4 * c4 + 3]));
                }
            }
            __syncthreads();
            // release at gpu scope is cumulative: the stores of all threads are ordered before it by the CTA barrier
            if (tid == 0) st_release(p.sync + 1 + bh, nch - c);
        }
        stamp();  // 9
        mma_wait();
        stamp();  // 10
        // the raw-input buffer (now S_0 pair) is dead: fetch the next item and start its loads
        if (tid == 0) {
            const int nxt = atomicAdd(&p.sync[0], 1);
            sm.next_item = nxt;
            if (nxt < nitems) {
                load_in5(nxt);
                if constexpr (CACHE) load_cache(nxt);
            }
        }
        // ================= P6: dA and dA^T masked, packed to bf16 pairs in place in TMEM (A operands) =================
        {
            uint32_t v[32], w2[32];
            const int t = r & 63;
            const bool qrow = r >= 64;
            tmem_ld32_nowait(tm_row + C_DA + 32 * cs, v);    // dA[row r][s'], s' = 32cs + e: columns 0-63 vs U, 64-127 vs V
            tmem_ld32_nowait(tm_row + C_DAT + 32 * cs, w2);  // dA^T[row r = s'][column: a row (0-63) or q row (64-127)]
            tmem_ld_wait();
            uint32_t a0[16], a1[16], t0[16], t1[16];
#pragma unroll
            for (int e = 0; e < 16; e++) {
                const int s0_ = 32 * (cs & 1) + 2 * e, s1_ = s0_ + 1;
                const bool k0 = qrow ? (s0_ <= t) : (s0_ < t), k1 = qrow ? (s1_ <= t) : (s1_ < t);
                split2x2(k0 ? __uint_as_float(v[2 * e]) : 0.f, k1 ? __uint_as_float(v[2 * e + 1]) : 0.f, a0[e], a1[e]);
                const bool m0 = (cs >= 2) ? (t <= s0_) : (t < s0_), m1 = (cs >= 2) ? (t <= s1_) : (t < s1_);
                split2x2(m0 ? __uint_as_float(w2[2 * e]) : 0.f, m1 ? __uint_as_float(w2[2 * e + 1]) : 0.f, t0[e], t1[e]);
            }
            tc_fence_before();
            __syncthreads();   // every warp has read its fp32 columns before anyone overwrites them with packed parts
            tc_fence_after();
            tmem_st16(tm_row + C_DA + 16 * cs, a0);
            tmem_st16(tm_row + C_DA + 64 + 16 * cs, a1);
            tmem_st16(tm_row + C_DAT + 16 * cs, t0);
            tmem_st16(tm_row + C_DAT + 64 + 16 * cs, t1);
            tmem_st_wait();
        }
        tc_fence_before();
        __syncthreads();
        stamp();  // 11
        if (warp == 0) {
            if (elect_one()) {
                tc_fence_after();
                mma_x3_tmemA_k128(tmem + C_AQ, tmem + C_DA, 64, b4, O_BK, 16384);    // [dAt;dQt] += dA [Bt;Kt]
                mma_x3_tmemA_k128(tmem + C_BK, tmem + C_DAT, 64, b4, O_AQ, 16384);   // [dBt;dKt] += dA^T [At;Qt]
                umma_commit(&sm.bar_mma);
            }
            __syncwarp();
        }
        // inputs of the element-wise epilogue: loads issued now, consumed after the products above have finished
        const int et = r & 63, ej0 = 16 * cs;
        const size_t ego = row0 + (size_t)et * rstride + ej0;
        uint4 ein[2][2];
        {   // rows 0-63 finish da, db (need a, b); rows 64-127 finish dq, dk, dv (need q, k)
            const uint16_t* src0 = (r >= 64) ? p.q : p.a;
            const uint16_t* src1 = (r >= 64) ? p.k : p.b;
            ein[0][0] = __ldg(reinterpret_cast<const uint4*>(src0 + ego));
            ein[0][1] = __ldg(reinterpret_cast<const uint4*>(src0 + ego) + 1);
            ein[1][0] = __ldg(reinterpret_cast<const uint4*>(src1 + ego));
            ein[1][1] = __ldg(reinterpret_cast<const uint4*>(src1 + ego) + 1);
        }
        float wpre[8];   // w of this thread's 8 rows in the dw pass (column tid & 63)
#pragma unroll
        for (int k = 0; k < 8; k++) wpre[k] = bf16lo_to_f32((uint32_t)__ldg(p.w + row0 + (size_t)(8 * (tid >> 6) + k) * rstride + (tid & 63)));
        mma_wait();
        stamp();  // 12
        item = sm.next_item;
        if (tid == 0 && item < nitems) load_dy(item);   // the dY tile is dead
        // ================= epilogue =================
        // three [64][64] fp32 scratch arrays with a row pitch of 65 floats (over the dead aq / bk operands): written
        // row-wise by lanes that differ in t, read column-wise by lanes that differ in j
        constexpr int EP = 65;
        float* const kk_s = reinterpret_cast<float*>(sm.aq);              // (db b)[t][j]
        float* const p1_s = reinterpret_cast<float*>(sm.aq) + 64 * EP;    // (dq q - dk k)[t][j]
        float* const p2_s = reinterpret_cast<float*>(sm.aq) + 128 * EP;   // (da a)[t][j]   (runs on into bk)
        {
            const int t = et, j0 = ej0;
            float E[16], Em[16];
#pragma unroll
            for (int c4 = 0; c4 < 4; c4++) {
                const float4 x = *m64_chunk(sm.emat, t, 4 * cs + c4);
                E[4 * c4] = x.x; E[4 * c4 + 1] = x.y; E[4 * c4 + 2] = x.z; E[4 * c4 + 3] = x.w;
                float4 y = make_float4(1.f, 1.f, 1.f, 1.f);
                if (t > 0) y = *m64_chunk(sm.emat, t - 1, 4 * cs + c4);
                Em[4 * c4] = y.x; Em[4 * c4 + 1] = y.y; Em[4 * c4 + 2] = y.z; Em[4 * c4 + 3] = y.w;
            }
            auto un16 = [&](const uint4 (&u)[2], float (&o)[16]) {
                const uint32_t w_[8] = {u[0].x, u[0].y, u[0].z, u[0].w, u[1].x, u[1].y, u[1].z, u[1].w};
#pragma unroll
                for (int e = 0; e < 8; e++) {
                    o[2 * e] = bf16lo_to_f32(w_[e]);
                    o[2 * e + 1] = bf16hi_to_f32(w_[e]);
                }
            };
            auto st16 = [&](uint16_t* ptr, const float (&o)[16]) {
                uint4 u0, u1;
                u0.x = pack_bf16x2(o[0], o[1]); u0.y = pack_bf16x2(o[2], o[3]); u0.z = pack_bf16x2(o[4], o[5]); u0.w = pack_bf16x2(o[6], o[7]);
                u1.x = pack_bf16x2(o[8], o[9]); u1.y = pack_bf16x2(o[10], o[11]); u1.z = pack_bf16x2(o[12], o[13]); u1.w = pack_bf16x2(o[14], o[15]);
                *reinterpret_cast<uint4*>(ptr) = u0;
                *(reinterpret_cast<uint4*>(ptr) + 1) = u1;
            };
            if (r >= 64) {  // dq, dk, dv
                uint32_t vq[16], vk[16], vv[16];
                tmem_ld16_nowait(tm_row + C_AQ + j0, vq);
                tmem_ld16_nowait(tm_row + C_BK + j0, vk);
                tmem_ld16_nowait(tm_row + C_UV + j0, vv);
                tmem_ld_wait();
                float qin[16], kin[16], dq[16], dk[16], dv[16];
                un16(ein[0], qin);
                un16(ein[1], kin);
#pragma unroll
                for (int e = 0; e < 16; e++) {
                    dq[e] = __uint_as_float(vq[e]) * E[e];
                    dk[e] = __fdividef(__uint_as_float(vk[e]), E[e]);
                    dv[e] = __uint_as_float(vv[e]);
                    p1_s[t * EP + j0 + e] = dq[e] * qin[e] - dk[e] * kin[e];
                }
                st16(p.dq + ego, dq);
                st16(p.dk + ego, dk);
                st16(p.dv + ego, dv);
            } else {  // da, db
                uint32_t va[16], vb[16];
                tmem_ld16_nowait(tm_row + C_AQ + j0, va);
                tmem_ld16_nowait(tm_row + C_BK + j0, vb);
                tmem_ld_wait();
                float ain[16], bin[16], da[16], db[16];
                un16(ein[0], ain);
                un16(ein[1], bin);
#pragma unroll
                for (int e = 0; e < 16; e++) {
                    da[e] = __uint_as_float(va[e]) * Em[e];
                    db[e] = __fdividef(__uint_as_float(vb[e]), E[e]);
                    kk_s[t * EP + j0 + e] = db[e] * bin[e];
                    p2_s[t * EP + j0 + e] = da[e] * ain[e];
                }
                st16(p.da + ego, da);
                st16(p.db + ego, db);
            }
        }
        tc_fence_before();
        __syncthreads();
        // dG_t = p1_t - kk_t + p2_{t+1} (+ gl at t = 63); dg = suffix sum over t; dw = dg * (-e^w)
        {
            const int j = tid & 63, rg = tid >> 6;
            float dG[8];
            float run = 0.f;
#pragma unroll
            for (int k = 7; k >= 0; k--) {
                const int t = 8 * rg + k;
                const float nxt = (t == L - 1) ? sm.gl[j] : p2_s[(t + 1) * EP + j];
                run += p1_s[t * EP + j] - kk_s[t * EP + j] + nxt;
                dG[k] = run;  // suffix sum inside the row group
            }
            sm.esc[rg * N + j] = run;
            __syncthreads();
            float off = 0.f;
#pragma unroll
            for (int k = 1; k < 8; k++) off += (k > rg) ? sm.esc[k * N + j] : 0.f;
#pragma unroll
            for (int k = 0; k < 8; k++) {
                const int t = 8 * rg + k;
                const size_t go = row0 + (size_t)t * rstride + j;
                const float g = -__expf(wpre[k]);
                p.dw[go] = f32_to_bf16_bits((dG[k] + off) * g);
            }
        }
        __syncthreads();   // scratch (aq / bk / esc) is rewritten by the next item's P1
        stamp();  // 13
        lt++;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<512>(tmem);
}

}  // namespace vrwkv
