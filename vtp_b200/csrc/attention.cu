// vtp_b200 — fused self-attention forward for short sequences (T = prefix + HW, HW <= 256) on tcgen05.
//
// Replaces layers/attention.py:110-126 (SelfAttention.compute_attention after RoPE: SDPA with scale 1/sqrt(64), no
// mask, no dropout) and nn.MultiheadAttention's causal SDPA in the text tower (layers/block.py:387-412).
//
// One CTA per (query tile of 128 patch rows, head, image); 2 CTAs/SM (112 KB smem, 256 TMEM columns each).
//   S = Q·Kᵀ     one UMMA chain  M=128, N=128|256, K=64      (Q,K tiles by TMA straight out of the packed qkv buffer)
//   softmax      one thread per query row, the whole row lives in TMEM -> exact single-pass softmax (no online rescale)
//   O = P·V      P written as bf16 into a swizzled K-major smem tile in two 128-key halves, V consumed as an MN-major
//                B operand (no transpose); O accumulates in TMEM columns [0,64) that S no longer needs.
// The `prefix` (cls / storage) tokens — 1 in the encoder, 0 in the decoder/text — would cost a third 128-row tile for
// one row, so they are handled on CUDA cores: their key columns are folded into every row's softmax by the row
// threads, and their query rows are computed by a spare warp from the K/V tiles already in smem.
// Sequences with more than 256 non-prefix tokens go to the key-streaming kernel of attention_long.cu.
#include <stdlib.h>

#include <algorithm>

#include "attention.h"
#include "host.h"
#include "ptx.cuh"

namespace vtp {

static constexpr int ATT_THREADS = 192;
static constexpr int MAX_PREFIX = ATT_MAX_PREFIX;
// smem: Q 16K | K 32K | V 32K | P 32K | barriers
static constexpr int SQ = 0, SK = 16384, SV = SK + 32768, SP = SV + 32768, SBAR = SP + 32768;
static constexpr int SPCLS = SBAR + 128;      // bf16 [256]: softmax numerators of the cls query row (warp 5)
static constexpr int ATT_SMEM = SPCLS + 512;  // 115328 B -> 2 CTAs/SM

__device__ __forceinline__ float ex2f(float x) {  // ex2.approx.ftz (ex2f() carries a 4-instruction denormal slow path)
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ uint32_t sw128_off(int row, int col /*bf16 element 0..63*/) {
    return row * 128 + ((((col >> 3) ^ (row & 7)) << 4) | ((col & 7) << 1));
}

__global__ void __launch_bounds__(ATT_THREADS, 2) attn_fwd_kernel(const __grid_constant__ CUtensorMap tm, const AttnDev p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    if (smem_u32(smem) & 1023) __trap();  // SWIZZLE_128B tiles need a 1024B-aligned base
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SBAR);
    uint64_t* bar_qk = bars + 0;   // Q,K landed
    uint64_t* bar_v = bars + 1;    // V landed
    uint64_t* bar_s = bars + 2;    // S complete in TMEM
    uint64_t* bar_p0 = bars + 3;   // P half 0 written (128 arrivals)
    uint64_t* bar_pv0 = bars + 4;  // PV half 0 done (P buffer reusable)
    uint64_t* bar_p1 = bars + 5;   // P half 1 written
    uint64_t* bar_o = bars + 6;    // O complete
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // packed mode (short sequences, e.g. the 37-token local crops): the tile holds `pack` consecutive sequences, every
    // token (cls included) is an ordinary query row / key column and the softmax is masked block-diagonally
    const int qt = blockIdx.x, h = blockIdx.y, b = p.pack ? blockIdx.z * p.pack : blockIdx.z;
    const int D = p.D, T = p.T, prefix = p.prefix, HW = p.HW;
    const long seq_row0 = (long)b * T;
    const int kvrows = 128 * p.nkt;

    if (threadIdx.x == 0) {
        tma_prefetch_desc(&tm);
        mbar_init(bar_qk, 1), mbar_init(bar_v, 1), mbar_init(bar_s, 1), mbar_init(bar_p0, 128);
        mbar_init(bar_pv0, 1), mbar_init(bar_p1, 128), mbar_init(bar_o, 1);
        fence_barrier_init();
    }
    if (warp == 0) {
        tmem_alloc(tmem_slot, 256);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            // ---------------- TMA
            const int row_q = (int)seq_row0 + prefix + 128 * qt;
            const int row_k = (int)seq_row0 + prefix;
            mbar_expect_tx(bar_qk, 16384 + 16384 * p.nkt);
            tma_load_2d(smem + SQ, &tm, bar_qk, h * 64, row_q);
            for (int i = 0; i < p.nkt; ++i) tma_load_2d(smem + SK + i * 16384, &tm, bar_qk, D + h * 64, row_k + 128 * i);
            mbar_expect_tx(bar_v, 16384 * p.nkt);
            for (int i = 0; i < p.nkt; ++i)
                tma_load_2d(smem + SV + i * 16384, &tm, bar_v, 2 * D + h * 64, row_k + 128 * i);
            // ---------------- S = Q Kᵀ
            mbar_wait(bar_qk, 0);
            tc_fence_after();
            const uint32_t idesc_s = umma_idesc_bf16(128, kvrows, 0, 0);
            const uint32_t qa = smem_u32(smem + SQ), ka = smem_u32(smem + SK);
#pragma unroll
            for (int j = 0; j < 4; ++j)
                umma_bf16_ss(tmem, umma_desc_sw128(qa + j * 32, 0, 1024), umma_desc_sw128(ka + j * 32, 0, 1024), idesc_s,
                             j > 0);
            umma_commit(bar_s);
            // ---------------- O = P V  (two 128-key halves through one P buffer)
            const uint32_t idesc_o = umma_idesc_bf16(128, 64, 0, 1);  // B (=V) is MN-major
            const uint32_t pa = smem_u32(smem + SP), va = smem_u32(smem + SV);
            mbar_wait(bar_v, 0);
            for (int half = 0; half < p.nkt; ++half) {
                mbar_wait(half == 0 ? bar_p0 : bar_p1, 0);
                tc_fence_after();
#pragma unroll
                for (int j = 0; j < 8; ++j) {  // 8 k-steps of 16 keys
                    const uint64_t ad = umma_desc_sw128(pa + (j >> 2) * 16384 + (j & 3) * 32, 0, 1024);
                    const uint64_t bd = umma_desc_sw128(va + half * 16384 + j * 2048, 8192, 1024);
                    umma_bf16_ss(tmem, ad, bd, idesc_o, (half > 0 || j > 0) ? 1u : 0u);
                }
                umma_commit(half == 0 && p.nkt == 2 ? bar_pv0 : bar_o);
            }
        }
    } else if (warp <= 4) {
        // ---------------- softmax + epilogue: one thread per query row
        const int q4 = warp & 3;
        const int r = q4 * 32 + lane;             // row within the tile == TMEM lane
        const int qpos = 128 * qt + r;            // patch index of this query
        const int qtok = prefix + qpos;           // token index within the sequence
        const int pseq = p.pack ? r / T : 0;  // packed mode: my sequence within the tile
        const bool row_valid = p.pack ? (pseq < p.pack && b + pseq < p.B) : (qpos < HW);
        const uint32_t trow = tmem + (uint32_t(q4 * 32) << 16);

        // scores against the prefix keys (CUDA cores): q row from smem (swizzled), k rows from global
        float s_pre[MAX_PREFIX];
        mbar_wait(bar_qk, 0);
        if (prefix > 0) {
            float qf[64];
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const uint4 w = *reinterpret_cast<const uint4*>(smem + SQ + sw128_off(r, c * 8));
                qf[c * 8 + 0] = bf16_lo(w.x), qf[c * 8 + 1] = bf16_hi(w.x), qf[c * 8 + 2] = bf16_lo(w.y);
                qf[c * 8 + 3] = bf16_hi(w.y), qf[c * 8 + 4] = bf16_lo(w.z), qf[c * 8 + 5] = bf16_hi(w.z);
                qf[c * 8 + 6] = bf16_lo(w.w), qf[c * 8 + 7] = bf16_hi(w.w);
            }
#pragma unroll
            for (int j = 0; j < MAX_PREFIX; ++j) {
                s_pre[j] = -INFINITY;
                if (j < prefix) {
                    const uint4* kp = reinterpret_cast<const uint4*>(p.qkv + (seq_row0 + j) * 3 * D + D + h * 64);
                    float acc = 0.f;
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        const uint4 w = __ldg(kp + c);
                        acc += qf[c * 8 + 0] * bf16_lo(w.x) + qf[c * 8 + 1] * bf16_hi(w.x) + qf[c * 8 + 2] * bf16_lo(w.y) +
                               qf[c * 8 + 3] * bf16_hi(w.y) + qf[c * 8 + 4] * bf16_lo(w.z) + qf[c * 8 + 5] * bf16_hi(w.z) +
                               qf[c * 8 + 6] * bf16_lo(w.w) + qf[c * 8 + 7] * bf16_hi(w.w);
                    }
                    if (!p.causal || j <= qtok) s_pre[j] = acc;
                }
            }
        } else {
#pragma unroll
            for (int j = 0; j < MAX_PREFIX; ++j) s_pre[j] = -INFINITY;
        }

        mbar_wait(bar_s, 0);
        tc_fence_after();
        // pass 1: row max
        float m = -INFINITY;
#pragma unroll
        for (int j = 0; j < MAX_PREFIX; ++j) m = fmaxf(m, s_pre[j]);
        // keys [kmin,kmax) are visible
        const int kmin = p.pack ? (row_valid ? pseq * T : 0) : 0;
        const int kmax = p.pack ? (row_valid ? kmin + T : 0) : (p.causal ? min(HW, qpos + 1) : HW);
        for (int c = 0; c < kvrows; c += 32) {
            // tcgen05.ld is warp-collective: a chunk is skipped only when no lane of the warp needs it
            if (__all_sync(0xffffffffu, c + 32 <= kmin || c >= kmax)) continue;
            uint32_t rr[32];
            tmem_ld_32x32(trow + c, rr);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i)
                if (c + i >= kmin && c + i < kmax) m = fmaxf(m, __uint_as_float(rr[i]));
        }
        const float msc = (m == -INFINITY) ? 0.f : m * p.scale_log2;
        // pass 2: p = exp2(s*scale*log2e - m*scale*log2e), written as bf16 to the swizzled P tile, half by half
        float l = 0.f;
        float p_pre[MAX_PREFIX];
#pragma unroll
        for (int j = 0; j < MAX_PREFIX; ++j) {
            p_pre[j] = (s_pre[j] == -INFINITY) ? 0.f : ex2f(s_pre[j] * p.scale_log2 - msc);
            l += p_pre[j];
            p_pre[j] = bf16_round(p_pre[j]);
        }
        for (int half = 0; half < p.nkt; ++half) {
            if (half == 1) mbar_wait(bar_pv0, 0);  // P buffer free again
#pragma unroll 1
            for (int c32 = 0; c32 < 4; ++c32) {
                const int c = half * 128 + c32 * 32;
                uint32_t pk[16];
                if (__all_sync(0xffffffffu, c + 32 <= kmin || c >= kmax)) {  // masked for the whole warp: zeros (PV sums over all keys)
#pragma unroll
                    for (int i = 0; i < 16; ++i) pk[i] = 0u;
                } else {
                    uint32_t rr[32];
                    tmem_ld_32x32(trow + c, rr);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 32; i += 2) {
                        const bool v0 = c + i >= kmin && c + i < kmax, v1 = c + i + 1 >= kmin && c + i + 1 < kmax;
                        float e0 = v0 ? ex2f(__uint_as_float(rr[i]) * p.scale_log2 - msc) : 0.f;
                        float e1 = v1 ? ex2f(__uint_as_float(rr[i + 1]) * p.scale_log2 - msc) : 0.f;
                        l += e0 + e1;
                        pk[i >> 1] = pack_bf16x2(e0, e1);
                    }
                }
                // 32 keys = 4 x 16B chunks into chunk-region (c32>>1), columns (c32&1)*32 ..
                uint8_t* pb = smem + SP + (c32 >> 1) * 16384;
#pragma unroll
                for (int v4 = 0; v4 < 4; ++v4) {
                    const int col = (c32 & 1) * 32 + v4 * 8;
                    *reinterpret_cast<uint4*>(pb + sw128_off(r, col)) =
                        make_uint4(pk[v4 * 4], pk[v4 * 4 + 1], pk[v4 * 4 + 2], pk[v4 * 4 + 3]);
                }
            }
            tc_fence_before();
            fence_proxy_async_smem();
            mbar_arrive(half == 0 ? bar_p0 : bar_p1);
        }
        // epilogue
        mbar_wait(bar_o, 0);
        tc_fence_after();
        uint32_t o0[32], o1[32];
        tmem_ld_32x32(trow, o0);
        tmem_ld_32x32(trow + 32, o1);
        tmem_ld_wait();
        float o[64];
#pragma unroll
        for (int i = 0; i < 32; ++i) o[i] = __uint_as_float(o0[i]), o[32 + i] = __uint_as_float(o1[i]);
#pragma unroll
        for (int j = 0; j < MAX_PREFIX; ++j) {
            if (j < prefix && p_pre[j] != 0.f) {
                const uint4* vp = reinterpret_cast<const uint4*>(p.qkv + (seq_row0 + j) * 3 * D + 2 * D + h * 64);
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const uint4 w = __ldg(vp + c);
                    o[c * 8 + 0] += p_pre[j] * bf16_lo(w.x), o[c * 8 + 1] += p_pre[j] * bf16_hi(w.x);
                    o[c * 8 + 2] += p_pre[j] * bf16_lo(w.y), o[c * 8 + 3] += p_pre[j] * bf16_hi(w.y);
                    o[c * 8 + 4] += p_pre[j] * bf16_lo(w.z), o[c * 8 + 5] += p_pre[j] * bf16_hi(w.z);
                    o[c * 8 + 6] += p_pre[j] * bf16_lo(w.w), o[c * 8 + 7] += p_pre[j] * bf16_hi(w.w);
                }
            }
        }
        if (row_valid) {
            const float inv = 1.f / l;
            __nv_bfloat16* op = p.out + (seq_row0 + qtok) * D + h * 64;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                uint4 w;
                w.x = pack_bf16x2(o[c * 8] * inv, o[c * 8 + 1] * inv), w.y = pack_bf16x2(o[c * 8 + 2] * inv, o[c * 8 + 3] * inv);
                w.z = pack_bf16x2(o[c * 8 + 4] * inv, o[c * 8 + 5] * inv), w.w = pack_bf16x2(o[c * 8 + 6] * inv, o[c * 8 + 7] * inv);
                *reinterpret_cast<uint4*>(op + c * 8) = w;
            }
            if (p.lse) {
                if (p.pack) p.lse[((long)(b + pseq) * p.H + h) * T + (r - pseq * T)] = m * p.scale + logf(l);
                else p.lse[((long)b * p.H + h) * T + qtok] = m * p.scale + logf(l);
            }
        }
        tc_fence_before();
    } else {
        // ---------------- warp 5: prefix query rows (only the qt==0 CTA), CUDA cores over the smem K/V tiles
        if (qt == 0 && prefix > 0) {
            mbar_wait(bar_qk, 0);
            mbar_wait(bar_v, 0);
            for (int j = 0; j < prefix; ++j) {
                float qf[64];
                {
                    const uint4* qp = reinterpret_cast<const uint4*>(p.qkv + (seq_row0 + j) * 3 * D + h * 64);
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        const uint4 w = __ldg(qp + c);
                        qf[c * 8 + 0] = bf16_lo(w.x), qf[c * 8 + 1] = bf16_hi(w.x), qf[c * 8 + 2] = bf16_lo(w.y);
                        qf[c * 8 + 3] = bf16_hi(w.y), qf[c * 8 + 4] = bf16_lo(w.z), qf[c * 8 + 5] = bf16_hi(w.z);
                        qf[c * 8 + 6] = bf16_lo(w.w), qf[c * 8 + 7] = bf16_hi(w.w);
                    }
                }
                auto dot_row = [&](const uint4* kp, bool from_smem, int row) {
                    float acc = 0.f;
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        const uint4 w = from_smem ? *reinterpret_cast<const uint4*>(smem + SK + sw128_off(row, c * 8))
                                                  : __ldg(kp + c);
                        acc += qf[c * 8 + 0] * bf16_lo(w.x) + qf[c * 8 + 1] * bf16_hi(w.x) + qf[c * 8 + 2] * bf16_lo(w.y) +
                               qf[c * 8 + 3] * bf16_hi(w.y) + qf[c * 8 + 4] * bf16_lo(w.z) + qf[c * 8 + 5] * bf16_hi(w.z) +
                               qf[c * 8 + 6] * bf16_lo(w.w) + qf[c * 8 + 7] * bf16_hi(w.w);
                    }
                    return acc;
                };
                float sp[MAX_PREFIX], s[8];
                float m = -INFINITY;
#pragma unroll
                for (int t = 0; t < MAX_PREFIX; ++t) {
                    sp[t] = -INFINITY;
                    if (t < prefix && (!p.causal || t <= j))
                        sp[t] = dot_row(reinterpret_cast<const uint4*>(p.qkv + (seq_row0 + t) * 3 * D + D + h * 64), false, 0);
                    m = fmaxf(m, sp[t]);
                }
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int kk = lane + 32 * i;
                    s[i] = -INFINITY;
                    if (kk < HW && kk < kvrows && (!p.causal || prefix + kk <= j)) s[i] = dot_row(nullptr, true, kk);
                    m = fmaxf(m, s[i]);
                }
                m = warp_max(m);
                const float msc = m * p.scale_log2;
                float l = 0.f;
                __nv_bfloat16* pcls = reinterpret_cast<__nv_bfloat16*>(smem + SPCLS);
                __syncwarp();  // previous prefix row has finished reading pcls
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float e = (s[i] == -INFINITY) ? 0.f : ex2f(s[i] * p.scale_log2 - msc);
                    l += e;
                    pcls[lane + 32 * i] = __float2bfloat16_rn(e);  // keys beyond HW / kvrows get 0
                }
                l = warp_sum(l);
                __syncwarp();
                float a0 = 0.f, a1 = 0.f, c0 = 0.f, c1 = 0.f;
#pragma unroll
                for (int t = 0; t < MAX_PREFIX; ++t) {
                    if (t < prefix && sp[t] != -INFINITY) {
                        const float pe = ex2f(sp[t] * p.scale_log2 - msc);
                        l += pe;
                        const uint32_t w = __ldg(reinterpret_cast<const uint32_t*>(p.qkv + (seq_row0 + t) * 3 * D + 2 * D + h * 64) + lane);
                        a0 += bf16_round(pe) * bf16_lo(w), a1 += bf16_round(pe) * bf16_hi(w);
                    }
                }
                // O_cls = P V: the lane owns output dims (2 lane, 2 lane + 1); eight keys per iteration, the numerators come
                // as one broadcast 16-byte read, two independent accumulator pairs (the former per-key shuffle chain cost
                // ~16k cycles and made this warp the straggler of every qt == 0 CTA)
                const int kend = min(HW, kvrows);
                for (int k8 = 0; k8 < kend; k8 += 8) {
                    const uint4 pw = *reinterpret_cast<const uint4*>(pcls + k8);
                    const uint32_t pr[4] = {pw.x, pw.y, pw.z, pw.w};
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const float pk = (u & 1) ? bf16_hi(pr[u >> 1]) : bf16_lo(pr[u >> 1]);
                        const uint32_t w = *reinterpret_cast<const uint32_t*>(smem + SV + sw128_off(k8 + u, 2 * lane));
                        if (u & 1) c0 += pk * bf16_lo(w), c1 += pk * bf16_hi(w);
                        else a0 += pk * bf16_lo(w), a1 += pk * bf16_hi(w);
                    }
                }
                a0 += c0, a1 += c1;
                const float inv = 1.f / l;
                *reinterpret_cast<uint32_t*>(p.out + (seq_row0 + j) * D + h * 64 + 2 * lane) = pack_bf16x2(a0 * inv, a1 * inv);
                if (p.lse && lane == 0) p.lse[((long)b * p.H + h) * T + j] = m * p.scale + logf(l);
            }
        }
    }

    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem, 256);
    }
}


// ------------------------------------------------------------------------------------------------------------
// Variant with TWO row threads per query row (opt-in: VTP_ATTN_FWD8=1).  The one-thread-per-row kernel above is
// latency-bound (profiles/ncu_attn_r1b_before_cls_fix.md: 16 % warps active, 24 % issue slots, 5 % tensor pipe): its 4
// row warps per CTA walk 256 score columns serially.  Here 8 row warps share the 128 TMEM lanes pairwise (warps w and
// w+4 own the same lane quarter, as in attn_bwd_kernel): both compute the full-row max (the cheap pass), then each
// exponentiates HALF of the columns, writes its half of P and later normalises half of the 64 output dims.  With two
// 128-key halves the second P half goes into the Q|K0 region, which is dead once S is complete and the cls warp has
// finished its score pass (bar_kfree) — so both halves are produced concurrently and smem stays at 2 CTAs/SM.  The row
// sums are exchanged once, after the last MMA, through the then-dead P buffer.
static constexpr int ATT8_THREADS = 320;  // warp 0: TMA + MMA; warps 1-8: row warps; warp 9: prefix (cls) query rows

__global__ void __launch_bounds__(ATT8_THREADS, 2) attn_fwd8_kernel(const __grid_constant__ CUtensorMap tm, const AttnDev p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    if (smem_u32(smem) & 1023) __trap();
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SBAR);
    uint64_t* bar_qk = bars + 0;     // Q,K landed
    uint64_t* bar_v = bars + 1;      // V landed
    uint64_t* bar_s = bars + 2;      // S complete in TMEM
    uint64_t* bar_p0 = bars + 3;     // P half 0 written
    uint64_t* bar_p1 = bars + 4;     // P half 1 written (nkt == 2)
    uint64_t* bar_o = bars + 5;      // O complete
    uint64_t* bar_kfree = bars + 6;  // cls warp has finished reading the K tiles
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int qt = blockIdx.x, h = blockIdx.y, b = p.pack ? blockIdx.z * p.pack : blockIdx.z;
    const int D = p.D, T = p.T, prefix = p.prefix, HW = p.HW, nkt = p.nkt;
    const long seq_row0 = (long)b * T;
    const int kvrows = 128 * nkt;

    if (threadIdx.x == 0) {
        tma_prefetch_desc(&tm);
        mbar_init(bar_qk, 1), mbar_init(bar_v, 1), mbar_init(bar_s, 1), mbar_init(bar_p0, nkt == 2 ? 128 : 256);
        mbar_init(bar_p1, 128), mbar_init(bar_o, 1), mbar_init(bar_kfree, 1);
        fence_barrier_init();
    }
    if (warp == 0) {
        tmem_alloc(tmem_slot, 256);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            const int row_q = (int)seq_row0 + prefix + 128 * qt;
            const int row_k = (int)seq_row0 + prefix;
            mbar_expect_tx(bar_qk, 16384 + 16384 * nkt);
            tma_load_2d(smem + SQ, &tm, bar_qk, h * 64, row_q);
            for (int i = 0; i < nkt; ++i) tma_load_2d(smem + SK + i * 16384, &tm, bar_qk, D + h * 64, row_k + 128 * i);
            mbar_expect_tx(bar_v, 16384 * nkt);
            for (int i = 0; i < nkt; ++i) tma_load_2d(smem + SV + i * 16384, &tm, bar_v, 2 * D + h * 64, row_k + 128 * i);
            mbar_wait(bar_qk, 0);
            tc_fence_after();
            const uint32_t idesc_s = umma_idesc_bf16(128, kvrows, 0, 0);
            const uint32_t qa = smem_u32(smem + SQ), ka = smem_u32(smem + SK);
#pragma unroll
            for (int j = 0; j < 4; ++j)
                umma_bf16_ss(tmem, umma_desc_sw128(qa + j * 32, 0, 1024), umma_desc_sw128(ka + j * 32, 0, 1024), idesc_s,
                             j > 0);
            umma_commit(bar_s);
            const uint32_t idesc_o = umma_idesc_bf16(128, 64, 0, 1);  // B (= V) is MN-major
            const uint32_t va = smem_u32(smem + SV);
            mbar_wait(bar_v, 0);
            for (int half = 0; half < nkt; ++half) {
                mbar_wait(half == 0 ? bar_p0 : bar_p1, 0);
                tc_fence_after();
                const uint32_t pa = smem_u32(smem + (half == 0 ? SP : SQ));  // half 1 lives in the dead Q|K0 region
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const uint64_t ad = umma_desc_sw128(pa + (j >> 2) * 16384 + (j & 3) * 32, 0, 1024);
                    const uint64_t bd = umma_desc_sw128(va + half * 16384 + j * 2048, 8192, 1024);
                    umma_bf16_ss(tmem, ad, bd, idesc_o, (half > 0 || j > 0) ? 1u : 0u);
                }
            }
            umma_commit(bar_o);
        }
    } else if (warp <= 8) {
        const int set = (warp - 1) >> 2;  // 0: first half of the columns / output dims, 1: second half
        const int q4 = warp & 3;          // TMEM lane quarter this warp may access (== warp id % 4)
        const int r = q4 * 32 + lane;
        const int qpos = 128 * qt + r;
        const int qtok = prefix + qpos;
        const int pseq = p.pack ? r / T : 0;
        const bool row_valid = p.pack ? (pseq < p.pack && b + pseq < p.B) : (qpos < HW);
        const uint32_t trow = tmem + (uint32_t(q4 * 32) << 16);

        float s_pre[MAX_PREFIX];
        mbar_wait(bar_qk, 0);
        if (prefix > 0) {
            float qf[64];
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const uint4 w = *reinterpret_cast<const uint4*>(smem + SQ + sw128_off(r, c * 8));
                qf[c * 8 + 0] = bf16_lo(w.x), qf[c * 8 + 1] = bf16_hi(w.x), qf[c * 8 + 2] = bf16_lo(w.y);
                qf[c * 8 + 3] = bf16_hi(w.y), qf[c * 8 + 4] = bf16_lo(w.z), qf[c * 8 + 5] = bf16_hi(w.z);
                qf[c * 8 + 6] = bf16_lo(w.w), qf[c * 8 + 7] = bf16_hi(w.w);
            }
#pragma unroll
            for (int j = 0; j < MAX_PREFIX; ++j) {
                s_pre[j] = -INFINITY;
                if (j < prefix) {
                    const uint4* kp = reinterpret_cast<const uint4*>(p.qkv + (seq_row0 + j) * 3 * D + D + h * 64);
                    float acc = 0.f;
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        const uint4 w = __ldg(kp + c);
                        acc += qf[c * 8 + 0] * bf16_lo(w.x) + qf[c * 8 + 1] * bf16_hi(w.x) + qf[c * 8 + 2] * bf16_lo(w.y) +
                               qf[c * 8 + 3] * bf16_hi(w.y) + qf[c * 8 + 4] * bf16_lo(w.z) + qf[c * 8 + 5] * bf16_hi(w.z) +
                               qf[c * 8 + 6] * bf16_lo(w.w) + qf[c * 8 + 7] * bf16_hi(w.w);
                    }
                    if (!p.causal || j <= qtok) s_pre[j] = acc;
                }
            }
        } else {
#pragma unroll
            for (int j = 0; j < MAX_PREFIX; ++j) s_pre[j] = -INFINITY;
        }

        mbar_wait(bar_s, 0);
        tc_fence_after();
        // pass 1 (both threads of a row, redundantly): row max over all visible keys
        float m = -INFINITY;
#pragma unroll
        for (int j = 0; j < MAX_PREFIX; ++j) m = fmaxf(m, s_pre[j]);
        const int kmin = p.pack ? (row_valid ? pseq * T : 0) : 0;
        const int kmax = p.pack ? (row_valid ? kmin + T : 0) : (p.causal ? min(HW, qpos + 1) : HW);
        for (int c = 0; c < kvrows; c += 32) {
            if (__all_sync(0xffffffffu, c + 32 <= kmin || c >= kmax)) continue;
            uint32_t rr[32];
            tmem_ld_32x32(trow + c, rr);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i)
                if (c + i >= kmin && c + i < kmax) m = fmaxf(m, __uint_as_float(rr[i]));
        }
        // Every row thread has now (a) read its Q row for the prefix scores and (b) finished reading ALL score columns.
        // Both matter before anyone moves on: the second P half overwrites the Q tile, and the first P·V MMA overwrites
        // score columns [0,64) with O while a slower partner thread could still be scanning them for its maximum.
        tc_fence_before();
        asm volatile("bar.sync 2, 256;" ::: "memory");
        tc_fence_after();
        const float msc = (m == -INFINITY) ? 0.f : m * p.scale_log2;
        float l = 0.f;
        float p_pre[MAX_PREFIX];
#pragma unroll
        for (int j = 0; j < MAX_PREFIX; ++j) {
            p_pre[j] = (s_pre[j] == -INFINITY) ? 0.f : ex2f(s_pre[j] * p.scale_log2 - msc);
            if (set == 0) l += p_pre[j];        // the prefix key columns are counted once per row
            p_pre[j] = bf16_round(p_pre[j]);
        }
        // pass 2: my half of the columns.  nkt == 2: key half `set` (its own P buffer); nkt == 1: 64 of the 128 keys
        const bool second_buf = (nkt == 2 && set == 1);
        if (second_buf && qt == 0 && prefix > 0) mbar_wait(bar_kfree, 0);  // K0 tile is about to be overwritten
        uint8_t* pbase = smem + (second_buf ? SQ : SP);
        const int nchunk = (nkt == 2) ? 4 : 2;
#pragma unroll 1
        for (int i = 0; i < nchunk; ++i) {
            const int c32 = (nkt == 2) ? i : 2 * set + i;          // 32-key chunk within the 128-key P tile
            const int c = ((nkt == 2) ? set * 128 : 0) + c32 * 32;  // score column
            uint32_t pk[16];
            if (__all_sync(0xffffffffu, c + 32 <= kmin || c >= kmax)) {
#pragma unroll
                for (int k = 0; k < 16; ++k) pk[k] = 0u;
            } else {
                uint32_t rr[32];
                tmem_ld_32x32(trow + c, rr);
                tmem_ld_wait();
#pragma unroll
                for (int k = 0; k < 32; k += 2) {
                    const bool v0 = c + k >= kmin && c + k < kmax, v1 = c + k + 1 >= kmin && c + k + 1 < kmax;
                    const float e0 = v0 ? ex2f(__uint_as_float(rr[k]) * p.scale_log2 - msc) : 0.f;
                    const float e1 = v1 ? ex2f(__uint_as_float(rr[k + 1]) * p.scale_log2 - msc) : 0.f;
                    l += e0 + e1;
                    pk[k >> 1] = pack_bf16x2(e0, e1);
                }
            }
            uint8_t* pb = pbase + (c32 >> 1) * 16384;
#pragma unroll
            for (int v4 = 0; v4 < 4; ++v4) {
                const int col = (c32 & 1) * 32 + v4 * 8;
                *reinterpret_cast<uint4*>(pb + sw128_off(r, col)) =
                    make_uint4(pk[v4 * 4], pk[v4 * 4 + 1], pk[v4 * 4 + 2], pk[v4 * 4 + 3]);
            }
        }
        tc_fence_before();
        fence_proxy_async_smem();
        mbar_arrive(second_buf ? bar_p1 : bar_p0);

        // epilogue: wait for O, exchange the partial row sums through the (now dead) P buffer, normalise 32 dims each
        mbar_wait(bar_o, 0);
        tc_fence_after();
        float* xs = reinterpret_cast<float*>(smem + SP);
        xs[set * 128 + r] = l;
        asm volatile("bar.sync 1, 256;" ::: "memory");
        l = xs[r] + xs[128 + r];
        uint32_t o0[32];
        tmem_ld_32x32(trow + 32 * set, o0);
        tmem_ld_wait();
        float o[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) o[i] = __uint_as_float(o0[i]);
#pragma unroll
        for (int j = 0; j < MAX_PREFIX; ++j) {
            if (j < prefix && p_pre[j] != 0.f) {
                const uint4* vp = reinterpret_cast<const uint4*>(p.qkv + (seq_row0 + j) * 3 * D + 2 * D + h * 64 + 32 * set);
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const uint4 w = __ldg(vp + c);
                    o[c * 8 + 0] += p_pre[j] * bf16_lo(w.x), o[c * 8 + 1] += p_pre[j] * bf16_hi(w.x);
                    o[c * 8 + 2] += p_pre[j] * bf16_lo(w.y), o[c * 8 + 3] += p_pre[j] * bf16_hi(w.y);
                    o[c * 8 + 4] += p_pre[j] * bf16_lo(w.z), o[c * 8 + 5] += p_pre[j] * bf16_hi(w.z);
                    o[c * 8 + 6] += p_pre[j] * bf16_lo(w.w), o[c * 8 + 7] += p_pre[j] * bf16_hi(w.w);
                }
            }
        }
        if (row_valid) {
            const float inv = 1.f / l;
            __nv_bfloat16* op = p.out + (seq_row0 + qtok) * D + h * 64 + 32 * set;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                uint4 w;
                w.x = pack_bf16x2(o[c * 8] * inv, o[c * 8 + 1] * inv), w.y = pack_bf16x2(o[c * 8 + 2] * inv, o[c * 8 + 3] * inv);
                w.z = pack_bf16x2(o[c * 8 + 4] * inv, o[c * 8 + 5] * inv), w.w = pack_bf16x2(o[c * 8 + 6] * inv, o[c * 8 + 7] * inv);
                *reinterpret_cast<uint4*>(op + c * 8) = w;
            }
            if (p.lse && set == 0) {
                if (p.pack) p.lse[((long)(b + pseq) * p.H + h) * T + (r - pseq * T)] = m * p.scale + logf(l);
                else p.lse[((long)b * p.H + h) * T + qtok] = m * p.scale + logf(l);
            }
        }
        tc_fence_before();
    } else {
        // ---------------- warp 9: prefix query rows (only the qt == 0 CTA), CUDA cores over the smem K/V tiles
        if (qt == 0 && prefix > 0) {
            mbar_wait(bar_qk, 0);
            mbar_wait(bar_v, 0);
            for (int j = 0; j < prefix; ++j) {
                float qf[64];
                {
                    const uint4* qp = reinterpret_cast<const uint4*>(p.qkv + (seq_row0 + j) * 3 * D + h * 64);
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        const uint4 w = __ldg(qp + c);
                        qf[c * 8 + 0] = bf16_lo(w.x), qf[c * 8 + 1] = bf16_hi(w.x), qf[c * 8 + 2] = bf16_lo(w.y);
                        qf[c * 8 + 3] = bf16_hi(w.y), qf[c * 8 + 4] = bf16_lo(w.z), qf[c * 8 + 5] = bf16_hi(w.z);
                        qf[c * 8 + 6] = bf16_lo(w.w), qf[c * 8 + 7] = bf16_hi(w.w);
                    }
                }
                auto dot_row = [&](const uint4* kp, bool from_smem, int row) {
                    float acc = 0.f;
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        const uint4 w = from_smem ? *reinterpret_cast<const uint4*>(smem + SK + sw128_off(row, c * 8))
                                                  : __ldg(kp + c);
                        acc += qf[c * 8 + 0] * bf16_lo(w.x) + qf[c * 8 + 1] * bf16_hi(w.x) + qf[c * 8 + 2] * bf16_lo(w.y) +
                               qf[c * 8 + 3] * bf16_hi(w.y) + qf[c * 8 + 4] * bf16_lo(w.z) + qf[c * 8 + 5] * bf16_hi(w.z) +
                               qf[c * 8 + 6] * bf16_lo(w.w) + qf[c * 8 + 7] * bf16_hi(w.w);
                    }
                    return acc;
                };
                float sp[MAX_PREFIX], s[8];
                float m = -INFINITY;
#pragma unroll
                for (int t = 0; t < MAX_PREFIX; ++t) {
                    sp[t] = -INFINITY;
                    if (t < prefix && (!p.causal || t <= j))
                        sp[t] = dot_row(reinterpret_cast<const uint4*>(p.qkv + (seq_row0 + t) * 3 * D + D + h * 64), false, 0);
                    m = fmaxf(m, sp[t]);
                }
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int kk = lane + 32 * i;
                    s[i] = -INFINITY;
                    if (kk < HW && kk < kvrows && (!p.causal || prefix + kk <= j)) s[i] = dot_row(nullptr, true, kk);
                    m = fmaxf(m, s[i]);
                }
                __syncwarp();
                if (j == prefix - 1 && lane == 0) mbar_arrive(bar_kfree);  // last read of the K tiles is behind us
                m = warp_max(m);
                const float msc = m * p.scale_log2;
                float l = 0.f;
                __nv_bfloat16* pcls = reinterpret_cast<__nv_bfloat16*>(smem + SPCLS);
                __syncwarp();
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float e = (s[i] == -INFINITY) ? 0.f : ex2f(s[i] * p.scale_log2 - msc);
                    l += e;
                    pcls[lane + 32 * i] = __float2bfloat16_rn(e);
                }
                l = warp_sum(l);
                __syncwarp();
                float a0 = 0.f, a1 = 0.f, c0 = 0.f, c1 = 0.f;
#pragma unroll
                for (int t = 0; t < MAX_PREFIX; ++t) {
                    if (t < prefix && sp[t] != -INFINITY) {
                        const float pe = ex2f(sp[t] * p.scale_log2 - msc);
                        l += pe;
                        const uint32_t w = __ldg(reinterpret_cast<const uint32_t*>(p.qkv + (seq_row0 + t) * 3 * D + 2 * D + h * 64) + lane);
                        a0 += bf16_round(pe) * bf16_lo(w), a1 += bf16_round(pe) * bf16_hi(w);
                    }
                }
                const int kend = min(HW, kvrows);
                for (int k8 = 0; k8 < kend; k8 += 8) {
                    const uint4 pw = *reinterpret_cast<const uint4*>(pcls + k8);
                    const uint32_t pr[4] = {pw.x, pw.y, pw.z, pw.w};
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const float pk = (u & 1) ? bf16_hi(pr[u >> 1]) : bf16_lo(pr[u >> 1]);
                        const uint32_t w = *reinterpret_cast<const uint32_t*>(smem + SV + sw128_off(k8 + u, 2 * lane));
                        if (u & 1) c0 += pk * bf16_lo(w), c1 += pk * bf16_hi(w);
                        else a0 += pk * bf16_lo(w), a1 += pk * bf16_hi(w);
                    }
                }
                a0 += c0, a1 += c1;
                const float inv = 1.f / l;
                *reinterpret_cast<uint32_t*>(p.out + (seq_row0 + j) * D + h * 64 + 2 * lane) = pack_bf16x2(a0 * inv, a1 * inv);
                if (p.lse && lane == 0) p.lse[((long)b * p.H + h) * T + j] = m * p.scale + logf(l);
            }
        }
    }

    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem, 256);
    }
}

}  // namespace vtp

namespace vtp {

// ------------------------------------------------------------------------------------------------------------
// fp32 attention (accuracy mode): CUDA cores, one CTA per (head, image), K/V in padded smem, one warp per query row.
// Used by the fp32-exact inference mode only (layers/attention.py:124 with fp32 q,k,v).
// K/V go through smem in chunks of C keys (the host picks the largest C that fits, C = T whenever the whole sequence
// does).  Each chunk updates the row's running max / sum / accumulator; with a single chunk the first update is a plain
// assignment, so those shapes run exactly the arithmetic of a one-pass softmax.  With several chunks the query rows go in
// rounds of nw * F32_ROWS rows whose running state stays in registers while the chunks stream past.
static constexpr int F32_ROWS = 8;  // query rows per warp per round
__global__ void attn_fwd_f32_kernel(const float* __restrict__ qkv, float* __restrict__ out, int T, int H, int causal,
                                    float scale, int C) {
    extern __shared__ float sm[];
    const int D = H * 64, h = blockIdx.x, b = blockIdx.y;
    float* Ks = sm;                 // [C][65]
    float* Vs = Ks + (long)C * 65;  // [C][64]
    float* Ps = Vs + (long)C * 64;  // [nwarps][C]
    const float* base = qkv + (long)b * T * 3 * D;
    auto load_chunk = [&](int c0) {
        const int n = min(C, T - c0);
        for (int i = threadIdx.x; i < n * 64; i += blockDim.x) {
            const int t = i >> 6, d = i & 63;
            Ks[t * 65 + d] = base[(long)(c0 + t) * 3 * D + D + h * 64 + d];
            Vs[t * 64 + d] = base[(long)(c0 + t) * 3 * D + 2 * D + h * 64 + d];
        }
    };
    const bool resident = C >= T;
    if (resident) {
        load_chunk(0);
        __syncthreads();
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    float* pw = Ps + (long)warp * C;
    for (int q0 = 0; q0 < T; q0 += nw * F32_ROWS) {
        float m[F32_ROWS], l[F32_ROWS], a0[F32_ROWS], a1[F32_ROWS];
        for (int c0 = 0; c0 < T; c0 += C) {
            if (!resident) {
                __syncthreads();  // every warp is done with the previous chunk
                load_chunk(c0);
                __syncthreads();
            }
#pragma unroll
            for (int i = 0; i < F32_ROWS; ++i) {
                const int q = q0 + warp + nw * i;
                if (q >= T) continue;
                const int kend = min(causal ? q + 1 : T, c0 + C) - c0;  // visible keys of this chunk
                if (kend <= 0) continue;                                // causal: the whole chunk lies ahead of q
                const float* qp = base + (long)q * 3 * D + h * 64;
                float qf[64];
#pragma unroll
                for (int d = 0; d < 64; ++d) qf[d] = qp[d];
                float mc = -INFINITY;
                for (int k = lane; k < kend; k += 32) {
                    float acc = 0.f;
#pragma unroll
                    for (int d = 0; d < 64; ++d) acc += qf[d] * Ks[k * 65 + d];
                    acc *= scale;
                    pw[k] = acc;
                    mc = fmaxf(mc, acc);
                }
                mc = warp_max(mc);
                const float mn = c0 == 0 ? mc : fmaxf(m[i], mc);
                float lc = 0.f;
                for (int k = lane; k < kend; k += 32) {
                    const float e = expf(pw[k] - mn);
                    pw[k] = e;
                    lc += e;
                }
                lc = warp_sum(lc);
                __syncwarp();
                float x0 = 0.f, x1 = 0.f;
                for (int k = 0; k < kend; ++k) {
                    const float pk = pw[k];
                    x0 += pk * Vs[k * 64 + lane], x1 += pk * Vs[k * 64 + 32 + lane];
                }
                if (c0 == 0) {
                    l[i] = lc, a0[i] = x0, a1[i] = x1;
                } else {
                    const float alpha = expf(m[i] - mn);
                    l[i] = l[i] * alpha + lc, a0[i] = a0[i] * alpha + x0, a1[i] = a1[i] * alpha + x1;
                }
                m[i] = mn;
                __syncwarp();
            }
        }
#pragma unroll
        for (int i = 0; i < F32_ROWS; ++i) {
            const int q = q0 + warp + nw * i;
            if (q >= T) continue;
            float* op = out + ((long)b * T + q) * D + h * 64;
            op[lane] = a0[i] / l[i], op[32 + lane] = a1[i] / l[i];
        }
    }
}

}  // namespace vtp

using namespace vtp;

extern "C" int vtp_attention_fwd(const void* qkv, void* out, float* lse, int B, int T, int H, int prefix, int causal,
                                 vtp_stream_t st) {
    VTP_CHECK_ARG(qkv && out && B > 0 && T > 0 && H > 0, "attention_fwd: bad args");
    VTP_CHECK_ARG(prefix >= 0 && prefix <= MAX_PREFIX && prefix < T, "attention_fwd: prefix must be in [0,%d]", MAX_PREFIX);
    const int HW = T - prefix;
    VTP_CHECK_ARG(HW <= 256 || !causal,
                  "attention_fwd: causal attention over %d non-prefix tokens (> 256) is not supported", HW);
    VTP_CHECK_ARG(B <= 65535 && H <= 65535, "attention_fwd: grid too large");
    const int D = H * 64;
    AttnDev p;
    p.qkv = (const __nv_bfloat16*)qkv, p.out = (__nv_bfloat16*)out, p.lse = lse;
    p.B = B, p.T = T, p.H = H, p.D = D, p.prefix = prefix, p.HW = HW, p.causal = causal;
    p.nkt = HW > 128 ? 2 : 1;
    p.scale = 0.125f;
    p.scale_log2 = 0.125f * 1.4426950408889634f;
    p.pack = 0;
    // more than 256 patch tokens: the score row no longer fits TMEM -> key-block streaming kernel (attention_long.cu)
    if (HW > 256) return attn_fwd_long_launch(p, (cudaStream_t)st);
    if (!causal && T <= 64 && B > 1 && getenv("VTP_ATTN_NO_PACK") == nullptr) {
        // several whole sequences per 128-row tile; the prefix tokens become ordinary rows / columns
        p.pack = 128 / T;
        p.prefix = 0, p.HW = T, p.nkt = 1;
    }
    CUtensorMap tm;
    uint64_t dims[2] = {(uint64_t)3 * D, (uint64_t)B * T}, strides[1] = {(uint64_t)3 * D * 2};
    uint32_t box[2] = {64, 128};
    int rc = make_tmap_bf16(&tm, qkv, 2, dims, strides, box);
    if (rc) return rc;
    static bool configured = false;
    if (!configured) {
        VTP_CUDA(cudaFuncSetAttribute(attn_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ATT_SMEM));
        VTP_CUDA(cudaFuncSetAttribute(attn_fwd8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ATT_SMEM));
        configured = true;
    }
    dim3 grid(p.pack ? 1 : ceil_div(HW, 128), H, p.pack ? ceil_div(B, p.pack) : B);
    // persistent ping-pong kernel (attention_pipe.cu) for 128 < HW <= 256: default since its round-2 hardware validation
    // (x1.11 and bit-identical); VTP_ATTN_FWD_PIPE=0 selects the one-tile-per-CTA kernel below
    const char* vp = getenv("VTP_ATTN_FWD_PIPE");
    if (!(vp && vp[0] == '0') && !p.pack && !causal && p.nkt == 2 && HW % 8 == 0) return attn_fwd_pipe_launch(tm, p, (cudaStream_t)st);
    const char* v8 = getenv("VTP_ATTN_FWD8");  // opt-in: two row threads per query row (see attn_fwd8_kernel)
    if (v8 && v8[0] == '1')
        attn_fwd8_kernel<<<grid, ATT8_THREADS, ATT_SMEM, (cudaStream_t)st>>>(tm, p);
    else
        attn_fwd_kernel<<<grid, ATT_THREADS, ATT_SMEM, (cudaStream_t)st>>>(tm, p);
    VTP_LAUNCH_CHECK();
    return VTP_OK;
}

extern "C" int vtp_attention_fwd_f32(const float* qkv, float* out, int B, int T, int H, int causal, vtp_stream_t st) {
    VTP_CHECK_ARG(qkv && out && B > 0 && T > 0 && H > 0 && B <= 65535, "attention_fwd_f32: bad args");
    const int nw = 8;
    // K/V chunk: the whole sequence when it fits in 220 KB of smem, otherwise the largest chunk that does
    const size_t per_key = (65 + 64 + nw) * sizeof(float);
    const int C = (int)std::min<size_t>((size_t)T, 220 * 1024 / per_key);
    const size_t smem = (size_t)C * per_key;
    static size_t configured = 0;
    if (smem > configured) {
        VTP_CUDA(cudaFuncSetAttribute(attn_fwd_f32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = smem;
    }
    attn_fwd_f32_kernel<<<dim3(H, B), nw * 32, smem, (cudaStream_t)st>>>(qkv, out, T, H, causal, 0.125f, C);
    VTP_LAUNCH_CHECK();
    return VTP_OK;
}
