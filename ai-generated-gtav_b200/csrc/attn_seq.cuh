// Device body of the fused-rotary non-causal attention on mma.sync tiles (see attn_mma.cu for the op it replaces and for when
// it runs instead of the tcgen05 kernel of attn_tc.cu), shared by attn_seq_kernel and attn_seq144_kernel.
#pragma once
#include "common.cuh"
#include "kernels.h"

namespace gtav {

static constexpr int HD = 64;          // head dim
static constexpr int SROW = HD + 8;    // smem row stride (bf16): 144 B keeps ldmatrix / fragment loads conflict-free

__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], const void* smem_ptr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(smem_u32(smem_ptr)));
}
// rotate the adjacent pair packed in `u` by (cos, sin) and re-round to bf16.  Both products and the sum are rounded
// explicitly: the reference's t * cos + rotate_half(t) * sin rounds each of them (rotary_embedding_torch.py:46-73), and
// an FMA contraction of one product into the sum moves an occasional element by a bf16 ulp.
__device__ __forceinline__ uint32_t rotate_pair(uint32_t u, float2 cs) {
    const float2 x = unpack_bf16x2(u);
    return pack_bf16x2(__fsub_rn(__fmul_rn(x.x, cs.x), __fmul_rn(x.y, cs.y)),
                       __fadd_rn(__fmul_rn(x.y, cs.x), __fmul_rn(x.x, cs.y)));
}


__device__ __forceinline__ void attn_bar(int id, int threads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory"); }
template <bool COHERENT>
__device__ __forceinline__ uint32_t attn_ld32(const bf16* p) {
    if (COHERENT) return __ldcg(reinterpret_cast<const unsigned int*>(p));
    return *reinterpret_cast<const uint32_t*>(p);
}
template <bool COHERENT>
__device__ __forceinline__ uint4 attn_ld128(const bf16* p) {
    if (COHERENT) return __ldcg(reinterpret_cast<const uint4*>(p));
    return *reinterpret_cast<const uint4*>(p);
}

// One work item = (query block qblock of WARPS*16 rows, head, group of SEQ consecutive rows), executed by WARPS warps
// (tid = 0 .. WARPS*32-1) that synchronise on named barrier `bar_id`.  sK / sV: KB*SROW bf16 each.  COHERENT: read
// qkv with ld.global.cg (the buffer was written by other CTAs of the SAME kernel - persistent step kernel).
// PRESTAGED (needs SEQ == KB): the caller has already put the rotated K, V and the rotated WARPS*16 query rows of this
// item (sQ, row stride SROW) into shared memory and synchronised; the body only computes.
// TILED_OUT (SEQ == 144 only): `out` is the pre-tiled activation image [head = 64-column chunk][144 rows][64] with
// the 128-byte swizzle of an UMMA K-major operand (16-byte chunk index ^ (row & 7)) instead of a row-major matrix.
template <int SEQ, int KB, int WARPS, int ROT_PAIRS, bool COHERENT, bool PRESTAGED = false, bool TILED_OUT = false>
__device__ __forceinline__ void attn_seq_body(const bf16* qkv, bf16* out, int heads, const float2* __restrict__ rot, bf16* sK,
                                              bf16* sV, int qblock, int head, int group, int tid, int bar_id,
                                              const bf16* sQ = nullptr) {
    static_assert(SEQ % KB == 0 && KB % 16 == 0 && SEQ % (WARPS * 16) == 0, "tiling");
    static_assert(!PRESTAGED || SEQ == KB, "pre-staged keys must cover the whole sequence");
    const int warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, tig = lane & 3;
    const int ld = 3 * heads * HD;
    const size_t row_base = static_cast<size_t>(group) * SEQ;
    const bf16* qbase = qkv + row_base * ld + head * HD;
    const bf16* kbase = qbase + heads * HD;
    const bf16* vbase = kbase + heads * HD;

    // ---- Q fragments (16 rows x 64 dims per warp): raw loads first, rotary applied once the K/V loads of the
    // first key block are in flight too (one global round trip for everything the block needs) ------------------
    const int q0 = (qblock * WARPS + warp) * 16;        // first query row of this warp (within the group)
    uint32_t qf[4][4];
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
        for (int h = 0; h < 4; ++h) {
            const int r = q0 + g + (h & 1) * 8;
            const int c = ks * 16 + 2 * tig + (h >> 1) * 8;
            if (PRESTAGED) qf[ks][h] = *reinterpret_cast<const uint32_t*>(sQ + (r - qblock * WARPS * 16) * SROW + c);
            else qf[ks][h] = attn_ld32<COHERENT>(qbase + static_cast<size_t>(r) * ld + c);
        }
    }

    float o[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) o[i][j] = 0.f;
    float m_run[2] = {-INFINITY, -INFINITY};
    float l_run[2] = {0.f, 0.f};
    const float sl2 = 0.125f * 1.4426950408889634f;          // 1/sqrt(64) * log2(e)
    constexpr int STAGE_ITERS = (KB * 8) / (WARPS * 32);
    static_assert((KB * 8) % (WARPS * 32) == 0, "staging loop must divide evenly");

    for (int kb0 = 0; kb0 < SEQ; kb0 += KB) {
        if (!PRESTAGED) {
        if (kb0 > 0) attn_bar(bar_id, WARPS * 32);                        // previous block fully consumed
        // ---- stage K (rotated) and V for keys [kb0, kb0+KB): all loads issued before any is consumed ----------
        uint4 kraw[STAGE_ITERS], vraw[STAGE_ITERS];
#pragma unroll
        for (int it = 0; it < STAGE_ITERS; ++it) {
            const int i = tid + it * WARPS * 32;
            const int r = i >> 3, c8 = (i & 7) * 8;
            const size_t goff = static_cast<size_t>(kb0 + r) * ld + c8;
            kraw[it] = attn_ld128<COHERENT>(kbase + goff);
            vraw[it] = attn_ld128<COHERENT>(vbase + goff);
        }
        if (kb0 == 0) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
                for (int h = 0; h < 4; ++h) {
                    const int r = q0 + g + (h & 1) * 8;
                    const int pr = (ks * 16 + 2 * tig + (h >> 1) * 8) >> 1;
                    if (pr < ROT_PAIRS) qf[ks][h] = rotate_pair(qf[ks][h], rot[r * ROT_PAIRS + pr]);
                }
            }
        }
#pragma unroll
        for (int it = 0; it < STAGE_ITERS; ++it) {
            const int i = tid + it * WARPS * 32;
            const int r = i >> 3, c8 = (i & 7) * 8;
            uint32_t kw[4] = {kraw[it].x, kraw[it].y, kraw[it].z, kraw[it].w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int pr = (c8 >> 1) + j;
                if (pr < ROT_PAIRS) kw[j] = rotate_pair(kw[j], rot[(kb0 + r) * ROT_PAIRS + pr]);
            }
            *reinterpret_cast<uint4*>(&sK[r * SROW + c8]) = make_uint4(kw[0], kw[1], kw[2], kw[3]);
            *reinterpret_cast<uint4*>(&sV[r * SROW + c8]) = vraw[it];
        }
        attn_bar(bar_id, WARPS * 32);
        }

        // ---- S = Q K^T for this key block ------------------------------------------------------
        float sc[KB / 8][4];
#pragma unroll
        for (int nt = 0; nt < KB / 8; ++nt) {
#pragma unroll
            for (int j = 0; j < 4; ++j) sc[nt][j] = 0.f;
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
                const bf16* kp = &sK[(nt * 8 + g) * SROW + ks * 16 + 2 * tig];
                mma_bf16_16816(sc[nt], qf[ks], *reinterpret_cast<const uint32_t*>(kp),
                               *reinterpret_cast<const uint32_t*>(kp + 8));
            }
        }
        // ---- online softmax (rows g and g+8 of the warp's 16) ----------------------------------
        float bm[2] = {-INFINITY, -INFINITY};
#pragma unroll
        for (int nt = 0; nt < KB / 8; ++nt) {
            bm[0] = fmaxf(bm[0], fmaxf(sc[nt][0], sc[nt][1]));
            bm[1] = fmaxf(bm[1], fmaxf(sc[nt][2], sc[nt][3]));
        }
        float alpha[2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            bm[h] = fmaxf(bm[h], __shfl_xor_sync(0xffffffffu, bm[h], 1));
            bm[h] = fmaxf(bm[h], __shfl_xor_sync(0xffffffffu, bm[h], 2));
            const float m_new = fmaxf(m_run[h], bm[h]);
            alpha[h] = exp2f((m_run[h] - m_new) * sl2);
            m_run[h] = m_new;
            l_run[h] *= alpha[h];
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            o[i][0] *= alpha[0]; o[i][1] *= alpha[0];
            o[i][2] *= alpha[1]; o[i][3] *= alpha[1];
        }
        const float mo0 = m_run[0] * sl2, mo1 = m_run[1] * sl2;
#pragma unroll
        for (int nt = 0; nt < KB / 8; ++nt) {
            sc[nt][0] = exp2f(sc[nt][0] * sl2 - mo0);
            sc[nt][1] = exp2f(sc[nt][1] * sl2 - mo0);
            sc[nt][2] = exp2f(sc[nt][2] * sl2 - mo1);
            sc[nt][3] = exp2f(sc[nt][3] * sl2 - mo1);
            l_run[0] += sc[nt][0] + sc[nt][1];
            l_run[1] += sc[nt][2] + sc[nt][3];
        }
        // ---- O += P V ---------------------------------------------------------------------------
#pragma unroll
        for (int j = 0; j < KB / 16; ++j) {
            uint32_t pf[4];
            pf[0] = pack_bf16x2(sc[2 * j][0], sc[2 * j][1]);
            pf[1] = pack_bf16x2(sc[2 * j][2], sc[2 * j][3]);
            pf[2] = pack_bf16x2(sc[2 * j + 1][0], sc[2 * j + 1][1]);
            pf[3] = pack_bf16x2(sc[2 * j + 1][2], sc[2 * j + 1][3]);
#pragma unroll
            for (int dn = 0; dn < 8; dn += 2) {
                // four 8x8 blocks of V: keys j*16 + {0..7, 8..15} x dims dn*8 + {0..7, 8..15}
                const int mat = lane >> 3, r = lane & 7;
                uint32_t vf[4];
                ldmatrix_x4_trans(vf, &sV[(j * 16 + (mat & 1) * 8 + r) * SROW + (dn + (mat >> 1)) * 8]);
                mma_bf16_16816(o[dn], pf, vf[0], vf[1]);
                mma_bf16_16816(o[dn + 1], pf, vf[2], vf[3]);
            }
        }
    }
    // ---- normalise and store ----------------------------------------------------------------------
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        l_run[h] += __shfl_xor_sync(0xffffffffu, l_run[h], 1);
        l_run[h] += __shfl_xor_sync(0xffffffffu, l_run[h], 2);
        l_run[h] = 1.0f / l_run[h];
    }
    const int ldo = heads * HD;
    bf16* obase = out + row_base * ldo + head * HD;
#pragma unroll
    for (int dn = 0; dn < 8; ++dn) {
        const int c = dn * 8 + 2 * tig;
        const uint32_t lo = pack_bf16x2(o[dn][0] * l_run[0], o[dn][1] * l_run[0]);
        const uint32_t hi = pack_bf16x2(o[dn][2] * l_run[1], o[dn][3] * l_run[1]);
        if (TILED_OUT) {
            uint8_t* tile = reinterpret_cast<uint8_t*>(out) + static_cast<size_t>(head) * (SEQ * 128);
            const int r0 = q0 + g, r1 = q0 + g + 8;
            *reinterpret_cast<uint32_t*>(tile + r0 * 128 + ((dn ^ (r0 & 7)) << 4) + tig * 4) = lo;
            *reinterpret_cast<uint32_t*>(tile + r1 * 128 + ((dn ^ (r1 & 7)) << 4) + tig * 4) = hi;
        } else {
            *reinterpret_cast<uint32_t*>(obase + static_cast<size_t>(q0 + g) * ldo + c) = lo;
            *reinterpret_cast<uint32_t*>(obase + static_cast<size_t>(q0 + g + 8) * ldo + c) = hi;
        }
    }
}


}  // namespace gtav
