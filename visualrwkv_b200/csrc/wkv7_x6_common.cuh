// wkv7_x6_common.cuh — pieces shared by the round-2 chunked WKV7 kernels (wkv7_x6_fwd.cuh, wkv7_x6_bwd.cuh).
//
// "x6": every fp32 matrix-product operand is split into three bf16 parts (x = x0 + x1 + x2 to 2^-25) and a product is
// the six tcgen05.mma.kind::f16 terms x_i y_j with i + j <= 2 (three terms when one operand is bf16-exact: v, dy),
// accumulated in fp32 in TMEM, smallest terms first.  That restores fp32-level accuracy (the north-star tolerance on the
// fp32 outputs sa / s needs ~1e-6; single TF32 gives 4e-4, a 2-way bf16 split 6e-6 — scripts measured, DESIGN.md 2.2c)
// at the tensor-core time of three TF32 products, and a bf16 tile (64 x 64, 8 KB, SWIZZLE_128B) serves both as a
// K-major and as an MN-major operand, so no operand is stored twice.
//
// The MMAs of a phase are issued by ONE elected lane (elect.sync): with the issuing thread picked by `lane == 0` the
// compiler cannot prove the descriptor / TMEM-address operands warp-uniform and wraps every tcgen05.mma in a
// vote/elect/R2UR "waterfall" loop — ~120 cycles per instruction (scripts/ubench_mma_issue.cu), which was the
// round-1 kernels' single largest cost.
#pragma once
#include "common.cuh"
#include "umma.cuh"
#include "wkv7_fwd.cuh"

namespace vrwkv {

constexpr int X6_L = 64;          // steps per chunk
constexpr int X6_THREADS = 512;   // 16 warps: TMEM lane quadrant = warp & 3, column slice = warp >> 2
constexpr uint32_t X6_TRIPLE64 = 3 * BT_BYTES;       // 3 parts of one 64-row tile
constexpr uint32_t X6_TRIPLE128 = 3 * 2 * BT_BYTES;  // 3 parts of a 128-row operand (two tiles per part)

// Chunk cache (model path): tiles the forward holds anyway and the backward would otherwise rebuild — the masked chunk
// matrices A_qb, A_qk, A_ak and Tinv = (I - A_ab)^-1 — as byte images of the shared-memory tiles ([t][s], SWIZZLE_128B).
// Parts 0 and 1 of the forward's three-way split are exactly the backward's two-way split (split3x2 begins with the
// two cvt.rn steps of split2x2).  Per item (chunk c of (b,h), stored at item c * B*H + b*H + h) 8 tiles of 8 KB:
constexpr uint32_t XC_QB0 = 0, XC_QK0 = 1, XC_QB1 = 2, XC_QK1 = 3, XC_AK0 = 4, XC_AK1 = 5, XC_TI0 = 6, XC_TI1 = 7;
constexpr uint32_t XC_ITEM_BYTES = 8 * BT_BYTES;

__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ int ld_acquire(const int* p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release(int* p, int v) {
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// 8 consecutive fp32 -> the three bf16 parts, one 16-byte store per part.  `p0` is the address in part 0,
// parts are `part_stride` bytes apart.
__device__ __forceinline__ void store_split8(uint8_t* p0, uint32_t part_stride, const float (&x)[8]) {
    uint4 a, b, c;
    split3x2(x[0], x[1], a.x, b.x, c.x);
    split3x2(x[2], x[3], a.y, b.y, c.y);
    split3x2(x[4], x[5], a.z, b.z, c.z);
    split3x2(x[6], x[7], a.w, b.w, c.w);
    *reinterpret_cast<uint4*>(p0) = a;
    *reinterpret_cast<uint4*>(p0 + part_stride) = b;
    *reinterpret_cast<uint4*>(p0 + 2 * part_stride) = c;
}
// the inverse: sum of the three parts (exact to 2^-24)
__device__ __forceinline__ void load_split8(const uint8_t* p0, uint32_t part_stride, float (&x)[8]) {
    const uint4 a = *reinterpret_cast<const uint4*>(p0), b = *reinterpret_cast<const uint4*>(p0 + part_stride),
                c = *reinterpret_cast<const uint4*>(p0 + 2 * part_stride);
    const uint32_t aa[4] = {a.x, a.y, a.z, a.w}, bb[4] = {b.x, b.y, b.z, b.w}, cc[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
    for (int e = 0; e < 4; e++) {
        x[2 * e] = (bf16lo_to_f32(cc[e]) + bf16lo_to_f32(bb[e])) + bf16lo_to_f32(aa[e]);
        x[2 * e + 1] = (bf16hi_to_f32(cc[e]) + bf16hi_to_f32(bb[e])) + bf16hi_to_f32(aa[e]);
    }
}
// byte offset of the 16-byte chunk `ch` (8 bf16) of row `row` inside a tile
__device__ __forceinline__ uint32_t bt_chunk(int row, int ch) { return (uint32_t)row * 128u + (((uint32_t)ch ^ ((uint32_t)row & 7u)) << 4); }

// fp32 64x64 scratch matrix with rows of 256 B whose 16-byte chunks are XOR-swizzled by (row & 7)
__device__ __forceinline__ float* m64_ptr(uint8_t* m, int t, int s) {
    return reinterpret_cast<float*>(m + t * 256 + ((((s >> 2) ^ (t & 7))) << 4) + (s & 3) * 4);
}
__device__ __forceinline__ float4* m64_chunk(uint8_t* m, int t, int chunk) {
    return reinterpret_cast<float4*>(m + t * 256 + ((chunk ^ (t & 7)) << 4));
}

// In place: M <- (I - M)^-1 for a strictly lower triangular 64x64 fp32 M (layout m64_*; the upper triangle must hold
// zeros and stays zero).  All 512 threads; fp32 FMAs on the CUDA cores: the four 16x16 diagonal blocks by forward
// substitution (one column per thread, results staged in `dscr` = 4 KB), then the coupling blocks of the two 32x32
// blocks and of the whole matrix as X_lower = X_b (M_lower X_a), staged through `esc` (4 KB).  Ends with a barrier.
__device__ __forceinline__ void tri_inverse_inplace(uint8_t* m, float* esc, float* dscr, const int tid) {
    if (tid < 64) {
        const int n = tid >> 4, cc = tid & 15;
        float x[16];
#pragma unroll
        for (int t = 0; t < 16; t++) {
            float a0 = (t == cc) ? 1.f : 0.f, a1 = 0.f;
#pragma unroll
            for (int c4 = 0; c4 < (t + 3) / 4; c4++) {
                const float4 q = *m64_chunk(m, 16 * n + t, 4 * n + c4);
                const float mm[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    const int s = 4 * c4 + e;
                    if (s < t) {
                        if (s & 1) a1 = fmaf(mm[e], x[s], a1);
                        else a0 = fmaf(mm[e], x[s], a0);
                    }
                }
            }
            x[t] = a0 + a1;
            dscr[n * 256 + t * 16 + cc] = x[t];
        }
    }
    __syncthreads();
    {   // diagonal blocks into place (1024 values, 2 per thread)
        const int n = tid >> 7, t = (tid >> 3) & 15, c0 = 2 * (tid & 7);
        *reinterpret_cast<float2*>(m64_ptr(m, 16 * n + t, 16 * n + c0)) = *reinterpret_cast<const float2*>(&dscr[n * 256 + t * 16 + c0]);
    }
    __syncthreads();
    // ---- level 1: the (1,0) block of each 32x32 diagonal block: X10 = D1 (M10 D0) ----
    {
        const int b = tid >> 8, t = (tid >> 4) & 15, c = tid & 15, o = 32 * b;
        float e0 = 0.f, e1 = 0.f;
#pragma unroll
        for (int c4 = 0; c4 < 4; c4++) {
            const float4 a = *m64_chunk(m, o + 16 + t, 8 * b + c4);
            e0 = fmaf(a.x, *m64_ptr(m, o + 4 * c4 + 0, o + c), e0);
            e1 = fmaf(a.y, *m64_ptr(m, o + 4 * c4 + 1, o + c), e1);
            e0 = fmaf(a.z, *m64_ptr(m, o + 4 * c4 + 2, o + c), e0);
            e1 = fmaf(a.w, *m64_ptr(m, o + 4 * c4 + 3, o + c), e1);
        }
        esc[b * 256 + t * 16 + c] = e0 + e1;
    }
    __syncthreads();
    {
        const int b = tid >> 8, t = (tid >> 4) & 15, c = tid & 15, o = 32 * b;
        float e0 = 0.f, e1 = 0.f;
#pragma unroll
        for (int c4 = 0; c4 < 4; c4++) {
            const float4 d = *m64_chunk(m, o + 16 + t, 8 * b + 4 + c4);
            e0 = fmaf(d.x, esc[b * 256 + (4 * c4 + 0) * 16 + c], e0);
            e1 = fmaf(d.y, esc[b * 256 + (4 * c4 + 1) * 16 + c], e1);
            e0 = fmaf(d.z, esc[b * 256 + (4 * c4 + 2) * 16 + c], e0);
            e1 = fmaf(d.w, esc[b * 256 + (4 * c4 + 3) * 16 + c], e1);
        }
        *m64_ptr(m, o + 16 + t, o + c) = e0 + e1;
    }
    __syncthreads();
    // ---- level 2: the lower-left 32x32 block: Xc = Xb (Mc Xa) ----
    {
        const int t = tid >> 4, c0 = 2 * (tid & 15);
        float e0 = 0.f, e1 = 0.f;
#pragma unroll
        for (int c4 = 0; c4 < 8; c4++) {
            const float4 q = *m64_chunk(m, 32 + t, c4);
            const float mm[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int e = 0; e < 4; e++) {
                const float2 xa = *reinterpret_cast<const float2*>(m64_ptr(m, 4 * c4 + e, c0));
                e0 = fmaf(mm[e], xa.x, e0);
                e1 = fmaf(mm[e], xa.y, e1);
            }
        }
        *reinterpret_cast<float2*>(&esc[t * 32 + c0]) = make_float2(e0, e1);
    }
    __syncthreads();
    {
        const int t = tid >> 4, c0 = 2 * (tid & 15);
        float e0 = 0.f, e1 = 0.f;
#pragma unroll
        for (int c4 = 0; c4 < 8; c4++) {
            const float4 q = *m64_chunk(m, 32 + t, 8 + c4);
            const float mm[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int e = 0; e < 4; e++) {
                const float2 ev = *reinterpret_cast<const float2*>(&esc[(4 * c4 + e) * 32 + c0]);
                e0 = fmaf(mm[e], ev.x, e0);
                e1 = fmaf(mm[e], ev.y, e1);
            }
        }
        *reinterpret_cast<float2*>(m64_ptr(m, 32 + t, c0)) = make_float2(e0, e1);
    }
    __syncthreads();
}

// ---- MMA batches (called by the one elected issuing lane) ----
// D[128 x N] (+)= A B with both operands split in three parts; part strides in bytes.  `a_mn`/`b_mn` select the
// operand's major-ness; the K-step (16 elements) advances a K-major descriptor by 32 bytes, an MN-major one by 2048.
// Terms are issued smallest first so that the large ones are added last (fewest roundings at full magnitude).
template <int N, int A_MN, int B_MN, int KSTEPS = 4>
__device__ __forceinline__ void mma_x6(uint32_t tmem_d, uint32_t b4, uint32_t a_off, uint32_t a_part, uint32_t b_off, uint32_t b_part,
                                       bool accumulate, uint32_t a_lbo = BT_BYTES, uint32_t b_lbo = BT_BYTES) {
    constexpr uint32_t idesc = umma_idesc_bf16_mj(128, N, A_MN, B_MN);
    constexpr int ta[6] = {2, 0, 1, 1, 0, 0}, tb[6] = {0, 2, 1, 0, 1, 0};
    uint32_t acc = accumulate ? 1u : 0u;
#pragma unroll
    for (int term = 0; term < 6; term++)
#pragma unroll
        for (int ks = 0; ks < KSTEPS; ks++) {
            const uint64_t da = A_MN ? bdesc_mn(b4, a_off + ta[term] * a_part + ks * 2048, a_lbo) : bdesc_k(b4, a_off + ta[term] * a_part + ks * 32);
            const uint64_t db = B_MN ? bdesc_mn(b4, b_off + tb[term] * b_part + ks * 2048, b_lbo) : bdesc_k(b4, b_off + tb[term] * b_part + ks * 32);
            umma_bf16(tmem_d, da, db, idesc, acc);
            acc = 1u;
        }
}
// the same with a bf16-exact (single part) B operand: three terms
template <int N, int A_MN, int B_MN, int KSTEPS = 4>
__device__ __forceinline__ void mma_x3b(uint32_t tmem_d, uint32_t b4, uint32_t a_off, uint32_t a_part, uint32_t b_off, bool accumulate,
                                        uint32_t a_lbo = BT_BYTES, uint32_t b_lbo = BT_BYTES) {
    constexpr uint32_t idesc = umma_idesc_bf16_mj(128, N, A_MN, B_MN);
    uint32_t acc = accumulate ? 1u : 0u;
#pragma unroll
    for (int term = 2; term >= 0; term--)
#pragma unroll
        for (int ks = 0; ks < KSTEPS; ks++) {
            const uint64_t da = A_MN ? bdesc_mn(b4, a_off + term * a_part + ks * 2048, a_lbo) : bdesc_k(b4, a_off + term * a_part + ks * 32);
            const uint64_t db = B_MN ? bdesc_mn(b4, b_off + ks * 2048, b_lbo) : bdesc_k(b4, b_off + ks * 32);
            umma_bf16(tmem_d, da, db, idesc, acc);
            acc = 1u;
        }
}
// ... and with a bf16-exact A operand
template <int N, int A_MN, int B_MN, int KSTEPS = 4>
__device__ __forceinline__ void mma_x3a(uint32_t tmem_d, uint32_t b4, uint32_t a_off, uint32_t b_off, uint32_t b_part, bool accumulate,
                                        uint32_t a_lbo = BT_BYTES, uint32_t b_lbo = BT_BYTES) {
    constexpr uint32_t idesc = umma_idesc_bf16_mj(128, N, A_MN, B_MN);
    uint32_t acc = accumulate ? 1u : 0u;
#pragma unroll
    for (int term = 2; term >= 0; term--)
#pragma unroll
        for (int ks = 0; ks < KSTEPS; ks++) {
            const uint64_t da = A_MN ? bdesc_mn(b4, a_off + ks * 2048, a_lbo) : bdesc_k(b4, a_off + ks * 32);
            const uint64_t db = B_MN ? bdesc_mn(b4, b_off + term * b_part + ks * 2048, b_lbo) : bdesc_k(b4, b_off + term * b_part + ks * 32);
            umma_bf16(tmem_d, da, db, idesc, acc);
            acc = 1u;
        }
}

}  // namespace vrwkv

// =====================================================================================================================
// "x3": two bf16 parts per operand (x = x0 + x1 to 2^-17), three product terms — what the backward uses: its outputs are
// bf16 gradients only (no fp32 side outputs), for which 6e-6 relative product error is 50x below the output rounding.
// =====================================================================================================================
namespace vrwkv {
constexpr uint32_t X3_PAIR64 = 2 * BT_BYTES;   // 2 parts of one 64-row tile (parts 8192 apart)

__device__ __forceinline__ void split2x2(float x, float y, uint32_t& p0, uint32_t& p1) {
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(p0) : "f"(y), "f"(x));
    const float rx = x - __uint_as_float(p0 << 16), ry = y - __uint_as_float(p0 & 0xffff0000u);
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(p1) : "f"(ry), "f"(rx));
}
__device__ __forceinline__ void store_pair8(uint8_t* p0, uint32_t part_stride, const float (&x)[8]) {
    uint4 a, b;
    split2x2(x[0], x[1], a.x, b.x);
    split2x2(x[2], x[3], a.y, b.y);
    split2x2(x[4], x[5], a.z, b.z);
    split2x2(x[6], x[7], a.w, b.w);
    *reinterpret_cast<uint4*>(p0) = a;
    *reinterpret_cast<uint4*>(p0 + part_stride) = b;
}
// D[128 x N] (+)= A B, both operands in two parts: terms (1,0), (0,1), (0,0)
template <int N, int A_MN, int B_MN, int KSTEPS = 4>
__device__ __forceinline__ void mma_x3(uint32_t tmem_d, uint32_t b4, uint32_t a_off, uint32_t a_part, uint32_t b_off, uint32_t b_part,
                                       bool accumulate, uint32_t a_lbo = BT_BYTES, uint32_t b_lbo = BT_BYTES) {
    constexpr uint32_t idesc = umma_idesc_bf16_mj(128, N, A_MN, B_MN);
    constexpr int ta[3] = {1, 0, 0}, tb[3] = {0, 1, 0};
    uint32_t acc = accumulate ? 1u : 0u;
#pragma unroll
    for (int term = 0; term < 3; term++)
#pragma unroll
        for (int ks = 0; ks < KSTEPS; ks++) {
            const uint64_t da = A_MN ? bdesc_mn(b4, a_off + ta[term] * a_part + ks * 2048, a_lbo) : bdesc_k(b4, a_off + ta[term] * a_part + ks * 32);
            const uint64_t db = B_MN ? bdesc_mn(b4, b_off + tb[term] * b_part + ks * 2048, b_lbo) : bdesc_k(b4, b_off + tb[term] * b_part + ks * 32);
            umma_bf16(tmem_d, da, db, idesc, acc);
            acc = 1u;
        }
}
// B bf16-exact (one part): terms a1 b, a0 b
template <int N, int A_MN, int B_MN, int KSTEPS = 4>
__device__ __forceinline__ void mma_x2b(uint32_t tmem_d, uint32_t b4, uint32_t a_off, uint32_t a_part, uint32_t b_off, bool accumulate,
                                        uint32_t a_lbo = BT_BYTES, uint32_t b_lbo = BT_BYTES) {
    constexpr uint32_t idesc = umma_idesc_bf16_mj(128, N, A_MN, B_MN);
    uint32_t acc = accumulate ? 1u : 0u;
#pragma unroll
    for (int term = 1; term >= 0; term--)
#pragma unroll
        for (int ks = 0; ks < KSTEPS; ks++) {
            const uint64_t da = A_MN ? bdesc_mn(b4, a_off + term * a_part + ks * 2048, a_lbo) : bdesc_k(b4, a_off + term * a_part + ks * 32);
            const uint64_t db = B_MN ? bdesc_mn(b4, b_off + ks * 2048, b_lbo) : bdesc_k(b4, b_off + ks * 32);
            umma_bf16(tmem_d, da, db, idesc, acc);
            acc = 1u;
        }
}
// A bf16-exact
template <int N, int A_MN, int B_MN, int KSTEPS = 4>
__device__ __forceinline__ void mma_x2a(uint32_t tmem_d, uint32_t b4, uint32_t a_off, uint32_t b_off, uint32_t b_part, bool accumulate,
                                        uint32_t a_lbo = BT_BYTES, uint32_t b_lbo = BT_BYTES) {
    constexpr uint32_t idesc = umma_idesc_bf16_mj(128, N, A_MN, B_MN);
    uint32_t acc = accumulate ? 1u : 0u;
#pragma unroll
    for (int term = 1; term >= 0; term--)
#pragma unroll
        for (int ks = 0; ks < KSTEPS; ks++) {
            const uint64_t da = A_MN ? bdesc_mn(b4, a_off + ks * 2048, a_lbo) : bdesc_k(b4, a_off + ks * 32);
            const uint64_t db = B_MN ? bdesc_mn(b4, b_off + term * b_part + ks * 2048, b_lbo) : bdesc_k(b4, b_off + term * b_part + ks * 32);
            umma_bf16(tmem_d, da, db, idesc, acc);
            acc = 1u;
        }
}
// A from TMEM: two packed-bf16 parts of 128 K elements each (64 columns per part, `a_part_cols` apart), B MN-major with
// 128 K lines (two tiles back to back inside a part).  D[128 x 64] += A B.
__device__ __forceinline__ void mma_x3_tmemA_k128(uint32_t tmem_d, uint32_t tmem_a, uint32_t a_part_cols, uint32_t b4, uint32_t b_off, uint32_t b_part) {
    constexpr uint32_t idesc = umma_idesc_bf16_mj(128, 64, 0, 1);
    constexpr int ta[3] = {1, 0, 0}, tb[3] = {0, 1, 0};
#pragma unroll
    for (int term = 0; term < 3; term++)
#pragma unroll
        for (int ks = 0; ks < 8; ks++)
            umma_bf16_ts(tmem_d, tmem_a + ta[term] * a_part_cols + 8 * ks, bdesc_mn(b4, b_off + tb[term] * b_part + ks * 2048), idesc, 1u);
}
}  // namespace vrwkv
