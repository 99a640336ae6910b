// wkv7_x6_fwd.cuh — WKV7 forward, round 2: chunk-parallel on the tcgen05 tensor cores at fp32-level accuracy.
// Same operator contract as the reference forward_kernel (VisualRWKV-v7/v7.00/cuda/wkv7_cuda.cu:10-52): y (bf16),
// sa (fp32, every step), s (fp32 transposed state checkpoints) — the algebra is the chunk-wise restatement kept with the
// tests (wkv7_chunked.py, test infrastructure), checked there against the step-by-step restatement of the reference.
//
// Work item = one 64-step chunk of one (batch, head).  A persistent grid (one 512-thread CTA per SM) takes items from an
// atomic counter in chunk-major order (all (b,h) of chunk 0, then of chunk 1, ...).  Everything that does not depend on
// the incoming state is chunk-local and runs on all SMs at once; the state hand-off between consecutive chunks of a
// (b,h) goes through the checkpoint tensor itself (the next chunk reads what the previous one wrote, L2-resident) behind
// a release/acquire flag.  An item only ever waits for an item with a smaller index, which was fetched earlier by a
// resident CTA, so the scheme cannot deadlock whatever the grid size.
//
// With E_t = prod_{s<=t} exp(-exp(w_s)) inside the chunk (per channel), F = 1/E,
//   At = a E_{t-1}, Qt = q E_t, Kt = k F_t, Bt = b F_t           (fp32, each stored as three bf16 parts)
//   scores = [At;Qt] [Bt;Kt]^T                    -> A_ab, A_ak (strictly lower), A_qb, A_qk (lower triangular)
//   ACC    = [A_ak;A_qk] V                        rows 0-63: AV
//   Tinv   = (I - A_ab)^-1                        fp32 FMAs on the CUDA cores (tri_inverse_inplace)
//   W      = [A_ab;A_qb] Tinv
//   CORR   = W At ;  ACC += W AV                  => [Ah;Qp] = [At;Qt] + CORR,  ACC = [Uh; Y_intra]
//   ---- needs the incoming state S_0 ----
//   ACC   += [Ah;Qp] S_0^T                        => ACC = [U; Y]  (rows of U are the sa_t)
//   Z      = U^T Bt + V^T Kt ;  S_L = (S_0 + Z) diag(E_L)       (per 16-step group when the reference's checkpoints
//                                                                are requested)
// Every product is an "x6" batch (wkv7_x6_common.cuh).  Domain: E_L must stay a normal fp32 number, i.e. the sum over a
// chunk of exp(w) < ~80 — guaranteed by RWKV-7's w = -softplus(.) - 0.5 (model.py:176); the host dispatcher keeps the
// step-by-step kernel for callers that cannot promise that.
#pragma once
#include "wkv7_chunk_common.cuh"
#include "wkv7_x6_common.cuh"

namespace vrwkv {

struct alignas(1024) X6FwdSmem {
    uint8_t v[BT_BYTES];         // raw v tile [t][i] (TMA, SWIZZLE_128B): MN-major operand of two products
    uint8_t in5[5 * BT_BYTES];   // raw w,q,k,a,b tiles; later M = A_ab -> Tinv (fp32, 16 KB) | Tinv parts (24 KB)
    uint8_t aq[X6_TRIPLE128];    // [At;Qt] -> [Ah;Qp]   (part p at p*16384: At tile, Qt tile)
    uint8_t bk[X6_TRIPLE128];    // [Bt;Kt]
    uint8_t avu[X6_TRIPLE64];    // AV parts [s][i] ; then U parts [t][i].  (Read as an M=128 MN-major A operand with 64 real
                                 // rows: the upper half comes from the 8 KB behind each part, so valid memory must follow.)
    uint8_t sca[X6_TRIPLE128];   // A-operand scratch: [A_ak;A_qk] -> [A_ab;A_qb] -> W ; then S_0 parts (first 24 KB)
    float esc[1024];             // coupling scratch of the inverse; P1: per row-group decay products [16][64]
    float el[4][WKV_N];          // E_t at t = 15, 31, 47, 63
    uint64_t bar_in, bar_v, bar_mma;
    uint32_t tmem_base;
    int next_item;
};

struct X6FwdArgs {
    int B, T, H;
    uint16_t* y;
    float* s;                 // checkpoints: [B,H,T/64,64,64] (ck16 == 0) or [B,H,T/16,64,64] (ck16 == 1); may be null
    float* sa;                // may be null
    const float* state_in;    // may be null (zeros); row-major [B,H,64(i),64(j)]
    float* state_out;         // may be null
    float* chain;             // used when s == null: [B*H][2][64*64] hand-off buffer (transposed states)
    int* sync;                // [0] item counter, [1 + b*H + h] number of finished chunks of (b,h); zeroed before launch
    uint8_t* cache;           // CACHE: the chunk cache, [B*H*T/64][8 tiles][8 KB] (wkv7_x6_common.cuh)
};

// CACHE: also write every item's chunk-cache tiles with 1-D bulk copies, each as soon as its tile exists (model path only).
template <bool CK16, bool CACHE = false>
__global__ void __launch_bounds__(X6_THREADS, 1)
wkv7_x6_fwd_kernel(const __grid_constant__ CUtensorMap tm_w, const __grid_constant__ CUtensorMap tm_q,
                   const __grid_constant__ CUtensorMap tm_k, const __grid_constant__ CUtensorMap tm_v,
                   const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b, const X6FwdArgs p) {
    constexpr int N = WKV_N, L = X6_L;
    extern __shared__ __align__(1024) uint8_t x6_smem_bytes[];
    X6FwdSmem& sm = *reinterpret_cast<X6FwdSmem*>((reinterpret_cast<uintptr_t>(x6_smem_bytes) + 1023) & ~(uintptr_t)1023);
    uint8_t* const mab = sm.in5;                   // fp32 A_ab -> Tinv
    uint8_t* const tinv = sm.in5 + 16384;          // Tinv parts (B operand, MN-major); diag scratch of the inverse before that

    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int qd = warp & 3, cs = warp >> 2;
    const int r = 32 * qd + lane;      // accumulator row (TMEM lane) of this thread
    const int T = p.T, H = p.H, BH = p.B * p.H;
    const int nch = T / L, nitems = BH * nch;

    if (tid == 0) {
        mbar_init(&sm.bar_in, 1);
        mbar_init(&sm.bar_v, 1);
        mbar_init(&sm.bar_mma, 1);
        fence_mbar_init();
        tma_prefetch_desc(&tm_w); tma_prefetch_desc(&tm_q); tma_prefetch_desc(&tm_k);
        tma_prefetch_desc(&tm_v); tma_prefetch_desc(&tm_a); tma_prefetch_desc(&tm_b);
        sm.next_item = atomicAdd(&p.sync[0], 1);
    }
    __syncwarp();
    if (warp == 0) tmem_alloc<512>(&sm.tmem_base);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = sm.tmem_base;
    const uint32_t tm_row = tmem + ((uint32_t)(32 * qd) << 16);
    constexpr uint32_t C_SC = 0, C_ACC = 128, C_W = 192, C_CORR = 256;
    constexpr uint32_t C_Z[4] = {320, 384, 448, 0};   // state sums (one per 16-step group with CK16; C_Z[0] otherwise)

    const uint32_t b4 = smem_u32(&sm) >> 4;
    const uint32_t O_V = (uint32_t)(sm.v - (uint8_t*)&sm), O_IN = (uint32_t)(sm.in5 - (uint8_t*)&sm), O_AQ = (uint32_t)(sm.aq - (uint8_t*)&sm),
                   O_BK = (uint32_t)(sm.bk - (uint8_t*)&sm), O_SCA = (uint32_t)(sm.sca - (uint8_t*)&sm), O_AVU = (uint32_t)(sm.avu - (uint8_t*)&sm);
    const uint32_t O_TINV = O_IN + 16384;

    // the cache stores are issued and drained by one thread of warp 2, which idles in the inverse's diagonal blocks
    constexpr int XC_TID = 64;
    auto load_in5 = [&](int item) {   // w,q,k,a,b tiles of an item (one thread)
        const int c = item / BH, bh = item - c * BH, bb = bh / H, hh = bh - bb * H;
        const int x0 = hh * N, y0 = bb * T + c * L;
        mbar_arrive_expect_tx(&sm.bar_in, 5 * BT_BYTES);
        tma_load_2d(sm.in5 + 0 * BT_BYTES, &tm_w, x0, y0, &sm.bar_in);
        tma_load_2d(sm.in5 + 1 * BT_BYTES, &tm_q, x0, y0, &sm.bar_in);
        tma_load_2d(sm.in5 + 2 * BT_BYTES, &tm_k, x0, y0, &sm.bar_in);
        tma_load_2d(sm.in5 + 3 * BT_BYTES, &tm_a, x0, y0, &sm.bar_in);
        tma_load_2d(sm.in5 + 4 * BT_BYTES, &tm_b, x0, y0, &sm.bar_in);
    };
    auto load_v = [&](int item) {
        const int c = item / BH, bh = item - c * BH, bb = bh / H, hh = bh - bb * H;
        mbar_arrive_expect_tx(&sm.bar_v, BT_BYTES);
        tma_load_2d(sm.v, &tm_v, hh * N, bb * T + c * L, &sm.bar_v);
    };
    int item = sm.next_item;
    if (tid == 0 && item < nitems) { load_in5(item); load_v(item); }
    __syncwarp();

    uint32_t ph_in = 0, ph_v = 0, ph_mma = 0;
    // development aid (vrwkv_wkv7_chunk_debug): CTA 0 records the clock at every phase boundary of its third item
#ifdef VRWKV_PHASE_STAMPS   // development aid (scripts/dbg_x6_stamps.py, dbg_x3_stamps.py): build with VRWKV_PHASE_STAMPS=1
    float* const dbg = (blockIdx.x == 0 && tid == 0) ? g_chunk_dbg : nullptr;
    int lt = 0, tsi = 0;
    long long tstamp0 = 0;
    auto stamp = [&]() {
        if (dbg && lt == 2) {
            const long long now = clock64();
            if (tsi == 0) tstamp0 = now;
            dbg[2048 + tsi++] = (float)(now - tstamp0);
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
    auto operands_ready = [&]() {  // generic-proxy writes -> visible to the tensor core, then CTA barrier
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();
    };
    // address of state "after chunk c of (b,h)" in the checkpoint / hand-off storage (transposed [j][i])
    auto state_ptr = [&](int bh, int c) -> float* {
        if (p.s) return p.s + ((size_t)bh * (CK16 ? 4 * nch : nch) + (size_t)(CK16 ? 4 * c + 3 : c)) * (N * N);
        return p.chain + ((size_t)bh * 2 + (c & 1)) * (N * N);
    };

    while (item < nitems) {
        const int c = item / BH, bh = item - c * BH, bb = bh / H, hh = bh - bb * H;
        // ================= P1: decay products and scaled operands (4 rows x 2 channels per thread) =================
        stamp();  // 0
        mbar_wait(&sm.bar_in, ph_in & 1);
        ph_in++;
        stamp();  // 1: inputs landed
        {
            const int rg = warp, j0 = 2 * lane;
            const uint8_t* tw = sm.in5;
            float c0[4], c1[4];
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const uint32_t ww = *reinterpret_cast<const uint32_t*>(tw + bt_off(4 * rg + k, j0));
                const float d0 = __expf(-__expf(bf16lo_to_f32(ww))), d1 = __expf(-__expf(bf16hi_to_f32(ww)));
                c0[k] = k ? c0[k - 1] * d0 : d0;
                c1[k] = k ? c1[k - 1] * d1 : d1;
            }
            *reinterpret_cast<float2*>(&sm.esc[rg * N + j0]) = make_float2(c0[3], c1[3]);
            __syncthreads();
            float pre0 = 1.f, pre1 = 1.f;
#pragma unroll
            for (int g = 0; g < 15; g++) {   // all loads in flight at once; groups >= rg contribute a factor 1
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
                const uint32_t qq = *reinterpret_cast<const uint32_t*>(sm.in5 + 1 * BT_BYTES + off);
                const uint32_t kk = *reinterpret_cast<const uint32_t*>(sm.in5 + 2 * BT_BYTES + off);
                const uint32_t aa = *reinterpret_cast<const uint32_t*>(sm.in5 + 3 * BT_BYTES + off);
                const uint32_t bb_ = *reinterpret_cast<const uint32_t*>(sm.in5 + 4 * BT_BYTES + off);
                uint32_t s0, s1, s2;
                split3x2(bf16lo_to_f32(aa) * Ep0, bf16hi_to_f32(aa) * Ep1, s0, s1, s2);
                *reinterpret_cast<uint32_t*>(sm.aq + off) = s0;
                *reinterpret_cast<uint32_t*>(sm.aq + 16384 + off) = s1;
                *reinterpret_cast<uint32_t*>(sm.aq + 32768 + off) = s2;
                split3x2(bf16lo_to_f32(qq) * E0, bf16hi_to_f32(qq) * E1, s0, s1, s2);
                *reinterpret_cast<uint32_t*>(sm.aq + BT_BYTES + off) = s0;
                *reinterpret_cast<uint32_t*>(sm.aq + 16384 + BT_BYTES + off) = s1;
                *reinterpret_cast<uint32_t*>(sm.aq + 32768 + BT_BYTES + off) = s2;
                split3x2(bf16lo_to_f32(bb_) * F0, bf16hi_to_f32(bb_) * F1, s0, s1, s2);
                *reinterpret_cast<uint32_t*>(sm.bk + off) = s0;
                *reinterpret_cast<uint32_t*>(sm.bk + 16384 + off) = s1;
                *reinterpret_cast<uint32_t*>(sm.bk + 32768 + off) = s2;
                split3x2(bf16lo_to_f32(kk) * F0, bf16hi_to_f32(kk) * F1, s0, s1, s2);
                *reinterpret_cast<uint32_t*>(sm.bk + BT_BYTES + off) = s0;
                *reinterpret_cast<uint32_t*>(sm.bk + 16384 + BT_BYTES + off) = s1;
                *reinterpret_cast<uint32_t*>(sm.bk + 32768 + BT_BYTES + off) = s2;
                if ((t & 15) == 15) *reinterpret_cast<float2*>(&sm.el[t >> 4][j0]) = make_float2(E0, E1);
                if (t == L - 1 && (E0 < 1e-30f || E1 < 1e-30f)) g_chunk_domain_err = 1;
                Ep0 = E0;
                Ep1 = E1;
            }
        }
        operands_ready();
        stamp();  // 2: P1 done
        // ================= scores = [At;Qt] [Bt;Kt]^T =================
        if (warp == 0) {
            if (elect_one()) {
                tc_fence_after();
                mma_x6<128, 0, 0>(tmem + C_SC, b4, O_AQ, 16384, O_BK, 16384, false);
                umma_commit(&sm.bar_mma);
            }
            __syncwarp();
        }
        mma_wait();
        stamp();  // 3: scores done
        // ================= P2: masks; A_ab in fp32 for the inverse; [A_ak;A_qk] operand =================
        float sc0[32];   // warps with cs < 2 keep their slice of [A_ab;A_qb] until the operand buffer is free again
        {
            uint32_t v[32];
            tmem_ld32(tm_row + C_SC + 32 * cs, v);
            const int tq = r & 63;
            const bool incl = r >= 64;   // q rows keep the diagonal
            const int sbase = 32 * (cs & 1);
#pragma unroll
            for (int e = 0; e < 32; e++) {
                const int s = sbase + e;
                const bool keep = incl ? (s <= tq) : (s < tq);
                sc0[e] = keep ? __uint_as_float(v[e]) : 0.f;
            }
            if (cs < 2) {
                if (r < 64) {
#pragma unroll
                    for (int cc = 0; cc < 8; cc++)
                        *m64_chunk(mab, r, 8 * cs + cc) = make_float4(sc0[4 * cc], sc0[4 * cc + 1], sc0[4 * cc + 2], sc0[4 * cc + 3]);
                }
            } else {
                uint8_t* dst = sm.sca + (r >> 6) * BT_BYTES;
#pragma unroll
                for (int cc = 0; cc < 4; cc++) {
                    const float x8[8] = {sc0[8 * cc], sc0[8 * cc + 1], sc0[8 * cc + 2], sc0[8 * cc + 3], sc0[8 * cc + 4], sc0[8 * cc + 5], sc0[8 * cc + 6], sc0[8 * cc + 7]};
                    store_split8(dst + bt_chunk(r & 63, 4 * (cs & 1) + cc), 16384, x8);
                }
            }
        }
        mbar_wait(&sm.bar_v, ph_v & 1);
        ph_v++;
        operands_ready();
        stamp();  // 4: P2 done
        if constexpr (CACHE) {
            if (tid == XC_TID) {   // [A_ak;A_qk] parts 0 and 1: drained before the inverse's first barrier, so before P3 reuses sca
                uint8_t* dst = p.cache + (size_t)item * XC_ITEM_BYTES;
                bulk_store_1d(dst + XC_AK0 * BT_BYTES, sm.sca, BT_BYTES);
                bulk_store_1d(dst + XC_QK0 * BT_BYTES, sm.sca + BT_BYTES, BT_BYTES);
                bulk_store_1d(dst + XC_AK1 * BT_BYTES, sm.sca + 16384, BT_BYTES);
                bulk_store_1d(dst + XC_QK1 * BT_BYTES, sm.sca + 16384 + BT_BYTES, BT_BYTES);
                tma_store_commit();
                tma_store_wait_read<0>();
            }
        }
        // ================= ACC = [A_ak;A_qk] V (runs while the inverse is being computed) =================
        if (warp == 0) {
            if (elect_one()) {
                tc_fence_after();
                mma_x3b<64, 0, 1>(tmem + C_ACC, b4, O_SCA, 16384, O_V, false);
                umma_commit(&sm.bar_mma);
            }
            __syncwarp();
        }
        tri_inverse_inplace(mab, sm.esc, reinterpret_cast<float*>(tinv), tid);
        stamp();  // 5: inverse done
        // ================= P3: Tinv parts; AV parts; [A_ab;A_qb] operand =================
        {
            const int t = tid >> 3, ch = tid & 7;
            const float4 lo = *m64_chunk(mab, t, 2 * ch), hi = *m64_chunk(mab, t, 2 * ch + 1);
            const float x8[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
            store_split8(tinv + bt_chunk(t, ch), BT_BYTES, x8);
        }
        mma_wait();
        if (r < 64) {
            uint32_t v[16];
            tmem_ld16(tm_row + C_ACC + 16 * cs, v);
#pragma unroll
            for (int hc = 0; hc < 2; hc++) {
                float x8[8];
#pragma unroll
                for (int e = 0; e < 8; e++) x8[e] = __uint_as_float(v[8 * hc + e]);
                store_split8(sm.avu + bt_chunk(r, 2 * cs + hc), BT_BYTES, x8);
            }
        }
        if (cs < 2) {
            uint8_t* dst = sm.sca + (r >> 6) * BT_BYTES;
#pragma unroll
            for (int cc = 0; cc < 4; cc++) {
                const float x8[8] = {sc0[8 * cc], sc0[8 * cc + 1], sc0[8 * cc + 2], sc0[8 * cc + 3], sc0[8 * cc + 4], sc0[8 * cc + 5], sc0[8 * cc + 6], sc0[8 * cc + 7]};
                store_split8(dst + bt_chunk(r & 63, 4 * cs + cc), 16384, x8);
            }
        }
        operands_ready();
        stamp();  // 6: P3 done
        if constexpr (CACHE) {
            if (tid == XC_TID) {   // A_qb parts 0 and 1, Tinv parts 0 and 1: read while the W batch runs
                uint8_t* dst = p.cache + (size_t)item * XC_ITEM_BYTES;
                bulk_store_1d(dst + XC_QB0 * BT_BYTES, sm.sca + BT_BYTES, BT_BYTES);
                bulk_store_1d(dst + XC_QB1 * BT_BYTES, sm.sca + 16384 + BT_BYTES, BT_BYTES);
                bulk_store_1d(dst + XC_TI0 * BT_BYTES, tinv, 2 * BT_BYTES);
                tma_store_commit();
            }
        }
        // ================= W = [A_ab;A_qb] Tinv =================
        if (warp == 0) {
            if (elect_one()) {
                tc_fence_after();
                mma_x6<64, 0, 1>(tmem + C_W, b4, O_SCA, 16384, O_TINV, BT_BYTES, false);
                umma_commit(&sm.bar_mma);
            }
            __syncwarp();
        }
        mma_wait();
        stamp();  // 7: W done
        if constexpr (CACHE) {   // P4 overwrites sca and the next item's loads overwrite Tinv
            if (tid == XC_TID) tma_store_wait_read<0>();
            __syncthreads();
        }
        // the raw-input buffer (M / Tinv) is dead: fetch the next item and start its loads
        if (tid == 0) {
            const int nxt = atomicAdd(&p.sync[0], 1);
            sm.next_item = nxt;
            if (nxt < nitems) load_in5(nxt);
        }
        // ================= P4: W parts (A operand) =================
        {
            uint32_t v[16];
            tmem_ld16(tm_row + C_W + 16 * cs, v);
            uint8_t* dst = sm.sca + (r >> 6) * BT_BYTES;
#pragma unroll
            for (int hc = 0; hc < 2; hc++) {
                float x8[8];
#pragma unroll
                for (int e = 0; e < 8; e++) x8[e] = __uint_as_float(v[8 * hc + e]);
                store_split8(dst + bt_chunk(r & 63, 2 * cs + hc), 16384, x8);
            }
        }
        operands_ready();
        stamp();  // 8: P4 done
        // ================= CORR = W At ;  ACC += W AV =================
        if (warp == 0) {
            if (elect_one()) {
                tc_fence_after();
                mma_x6<64, 0, 1>(tmem + C_CORR, b4, O_SCA, 16384, O_AQ, 16384, false);
                mma_x6<64, 0, 1>(tmem + C_ACC, b4, O_SCA, 16384, O_AVU, BT_BYTES, true);
                umma_commit(&sm.bar_mma);
            }
            __syncwarp();
        }
        mma_wait();
        stamp();  // 9: CORR done
        // ================= P5: [At;Qt] += CORR  ->  [Ah;Qp] (in place) =================
        {
            uint32_t v[16];
            tmem_ld16(tm_row + C_CORR + 16 * cs, v);
            uint8_t* base = sm.aq + (r >> 6) * BT_BYTES;
#pragma unroll
            for (int hc = 0; hc < 2; hc++) {
                uint8_t* ptr = base + bt_chunk(r & 63, 2 * cs + hc);
                float x8[8];
                load_split8(ptr, 16384, x8);
#pragma unroll
                for (int e = 0; e < 8; e++) x8[e] += __uint_as_float(v[8 * hc + e]);
                store_split8(ptr, 16384, x8);
            }
        }
        // ================= incoming state: wait for the previous chunk, S_0 parts [j][i] (B operand, MN-major) =================
        const float* s_prev = nullptr;   // transposed [j][i]
        stamp();  // 10: P5 done
        if (c > 0) {
            if (tid == 0) {
                const int* flag = p.sync + 1 + bh;
                long long t0 = clock64();
                while (ld_acquire(flag) < c) {
                    if (clock64() - t0 > 20000000000LL) __trap();
                }
            }
            __syncthreads();
            s_prev = state_ptr(bh, c - 1);
        }
        stamp();  // 11: state arrived
        {
            const int j = tid >> 3, i0 = 8 * (tid & 7);
            float x8[8];
            if (c > 0) {
                const float4 lo = __ldcg(reinterpret_cast<const float4*>(s_prev + j * N + i0)), hi = __ldcg(reinterpret_cast<const float4*>(s_prev + j * N + i0 + 4));
                x8[0] = lo.x; x8[1] = lo.y; x8[2] = lo.z; x8[3] = lo.w; x8[4] = hi.x; x8[5] = hi.y; x8[6] = hi.z; x8[7] = hi.w;
            } else if (p.state_in) {
                const float* src = p.state_in + (size_t)bh * N * N;
#pragma unroll
                for (int e = 0; e < 8; e++) x8[e] = __ldg(src + (i0 + e) * N + j);
            } else {
#pragma unroll
                for (int e = 0; e < 8; e++) x8[e] = 0.f;
            }
            store_split8(sm.sca + bt_chunk(j, tid & 7), BT_BYTES, x8);
        }
        operands_ready();
        stamp();  // 12: S0 parts done
        // ================= ACC += [Ah;Qp] S_0^T  ->  [U;Y] =================
        if (warp == 0) {
            if (elect_one()) {
                tc_fence_after();
                mma_x6<64, 0, 1>(tmem + C_ACC, b4, O_AQ, 16384, O_SCA, BT_BYTES, true);
                umma_commit(&sm.bar_mma);
            }
            __syncwarp();
        }
        mma_wait();
        stamp();  // 13: UY done
        // ================= P7: U parts [t][i]; sa / y to global memory =================
        {
            uint32_t uy[16];
            tmem_ld16(tm_row + C_ACC + 16 * cs, uy);
            const size_t row = (((size_t)bb * T + (size_t)c * L + (r & 63)) * H + hh) * N + 16 * cs;
            if (r < 64) {
#pragma unroll
                for (int hc = 0; hc < 2; hc++) {
                    float x8[8];
#pragma unroll
                    for (int e = 0; e < 8; e++) x8[e] = __uint_as_float(uy[8 * hc + e]);
                    store_split8(sm.avu + bt_chunk(r, 2 * cs + hc), BT_BYTES, x8);
                }
                if (p.sa) {
#pragma unroll
                    for (int c4 = 0; c4 < 4; c4++)
                        *reinterpret_cast<float4*>(p.sa + row + 4 * c4) =
                            make_float4(__uint_as_float(uy[4 * c4]), __uint_as_float(uy[4 * c4 + 1]), __uint_as_float(uy[4 * c4 + 2]),
                                        __uint_as_float(uy[4 * c4 + 3]));
                }
            } else {
                uint4 o0, o1;
                o0.x = pack_bf16x2(__uint_as_float(uy[0]), __uint_as_float(uy[1]));
                o0.y = pack_bf16x2(__uint_as_float(uy[2]), __uint_as_float(uy[3]));
                o0.z = pack_bf16x2(__uint_as_float(uy[4]), __uint_as_float(uy[5]));
                o0.w = pack_bf16x2(__uint_as_float(uy[6]), __uint_as_float(uy[7]));
                o1.x = pack_bf16x2(__uint_as_float(uy[8]), __uint_as_float(uy[9]));
                o1.y = pack_bf16x2(__uint_as_float(uy[10]), __uint_as_float(uy[11]));
                o1.z = pack_bf16x2(__uint_as_float(uy[12]), __uint_as_float(uy[13]));
                o1.w = pack_bf16x2(__uint_as_float(uy[14]), __uint_as_float(uy[15]));
                *reinterpret_cast<uint4*>(p.y + row) = o0;
                *reinterpret_cast<uint4*>(p.y + row + 8) = o1;
            }
        }
        operands_ready();
        stamp();  // 14: P7 done
        // ================= Z = U^T Bt + V^T Kt (rows = i; per 16-step group with CK16) =================
        if (warp == 0) {
            if (elect_one()) {
                tc_fence_after();
                if (CK16) {
#pragma unroll
                    for (int g = 0; g < 4; g++) {
                        mma_x6<64, 1, 1, 1>(tmem + C_Z[g], b4, O_AVU + g * 2048, BT_BYTES, O_BK + g * 2048, 16384, false);
                        mma_x3a<64, 1, 1, 1>(tmem + C_Z[g], b4, O_V + g * 2048, O_BK + BT_BYTES + g * 2048, 16384, true);
                    }
                } else {
                    mma_x6<64, 1, 1>(tmem + C_Z[0], b4, O_AVU, BT_BYTES, O_BK, 16384, false);
                    mma_x3a<64, 1, 1>(tmem + C_Z[0], b4, O_V, O_BK + BT_BYTES, 16384, true);
                }
                umma_commit(&sm.bar_mma);
            }
            __syncwarp();
        }
        mma_wait();
        stamp();  // 15: Z done
        item = sm.next_item;   // written before the barrier in front of the W-times batch
        if (tid == 0 && item < nitems) load_v(item);   // the v tile is dead
        // ================= P8: S_L = (S_0 + Z) diag(E_L)  -> checkpoints (transposed [j][i]) =================
        if (r < N) {
            float acc[16];
            const int i = r;
            if (c > 0) {
#pragma unroll
                for (int e = 0; e < 16; e++) acc[e] = __ldcg(s_prev + (16 * cs + e) * N + i);
            } else if (p.state_in) {
                const float4* src = reinterpret_cast<const float4*>(p.state_in + ((size_t)bh * N + i) * N + 16 * cs);
#pragma unroll
                for (int c4 = 0; c4 < 4; c4++) {
                    const float4 x = __ldg(src + c4);
                    acc[4 * c4] = x.x; acc[4 * c4 + 1] = x.y; acc[4 * c4 + 2] = x.z; acc[4 * c4 + 3] = x.w;
                }
            } else {
#pragma unroll
                for (int e = 0; e < 16; e++) acc[e] = 0.f;
            }
            if (CK16) {
                uint32_t z0[16], z1[16], z2[16], z3[16];
                tmem_ld16_nowait(tm_row + C_Z[0] + 16 * cs, z0);
                tmem_ld16_nowait(tm_row + C_Z[1] + 16 * cs, z1);
                tmem_ld16_nowait(tm_row + C_Z[2] + 16 * cs, z2);
                tmem_ld16_nowait(tm_row + C_Z[3] + 16 * cs, z3);
                tmem_ld_wait();
                float* ck = p.s + (((size_t)bh * 4 * nch + (size_t)4 * c) * N + 16 * cs) * N + i;
#pragma unroll
                for (int e = 0; e < 16; e++) {
                    acc[e] += __uint_as_float(z0[e]);
                    ck[(size_t)e * N] = acc[e] * sm.el[0][16 * cs + e];
                    acc[e] += __uint_as_float(z1[e]);
                    ck[(size_t)(N + e) * N] = acc[e] * sm.el[1][16 * cs + e];
                    acc[e] += __uint_as_float(z2[e]);
                    ck[(size_t)(2 * N + e) * N] = acc[e] * sm.el[2][16 * cs + e];
                    acc[e] += __uint_as_float(z3[e]);
                    acc[e] *= sm.el[3][16 * cs + e];
                    ck[(size_t)(3 * N + e) * N] = acc[e];
                }
            } else {
                uint32_t z0[16];
                tmem_ld16(tm_row + C_Z[0] + 16 * cs, z0);
                float* ck = state_ptr(bh, c) + (size_t)(16 * cs) * N + i;
#pragma unroll
                for (int e = 0; e < 16; e++) {
                    acc[e] = (acc[e] + __uint_as_float(z0[e])) * sm.el[3][16 * cs + e];
                    ck[(size_t)e * N] = acc[e];
                }
            }
            if (p.state_out && c == nch - 1) {
                float4* dst = reinterpret_cast<float4*>(p.state_out + ((size_t)bh * N + i) * N + 16 * cs);
#pragma unroll
                for (int c4 = 0; c4 < 4; c4++) dst[c4] = make_float4(acc[4 * c4], acc[4 * c4 + 1], acc[4 * c4 + 2], acc[4 * c4 + 3]);
            }
        }
        tc_fence_before();
        __syncthreads();
        // release at gpu scope is cumulative: the state stores of all threads are ordered before it by the CTA barrier
        if (tid == 0) st_release(p.sync + 1 + bh, c + 1);
        stamp();  // 16: item done
        lt++;
    }
    if constexpr (CACHE) {
        if (tid == XC_TID) tma_store_wait<0>();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<512>(tmem);
}

}  // namespace vrwkv
