// vtp_b200 — flash-style self-attention forward for long sequences (HW > 256 patch tokens, non-causal) on tcgen05.
//
// Serves images above 256 patches (e.g. 512x512 -> 1024 patches, 272x400 -> 425) where the single-pass kernels of
// attention.cu / attention_pipe.cu cannot hold a whole score row in TMEM.  Same contract as those kernels: packed
// qkv [B*T][3*H*64] read in place, out [B*T][H*64] bf16, scale 1/8, `prefix` (<= 4) leading cls tokens, optional
// lse [B][H][T] written for every row (prefix rows included).
//
// One CTA per (query tile of 128 patch rows, head, image); 2 CTAs/SM (112 KB smem, 256 TMEM columns each).
//   warp 0      TMA producer: Q tile once, then K|V in 128-key blocks through a two-stage ring
//   warps 1-4   softmax: one thread per query row, online softmax over the key blocks; O lives in registers
//   warp 5      MMA issuer:  S = Q·Kᵀ (M=128, N=128, K=64) into TMEM columns [0,128);
//                            PV = P·V  (M=128, N=64,  K=128) into TMEM columns [128,192), read back and added to O
//   warp 6      prefix (cls) query rows (only the qt == 0 CTA): CUDA cores straight from global K/V, online softmax
// Tensor maps are 3-D [B][T][3D]: a block that runs past the end of an image loads zeros instead of the next image's
// rows, and those key columns are masked to -inf (P = 0) in the softmax.  Query rows beyond the image are never stored.
// The prefix keys are folded into every row's running softmax on CUDA cores (as in attention.cu), so no key or query
// tile is padded for them.
#include "attention.h"
#include "host.h"
#include "ptx.cuh"

namespace vtp {

static constexpr int LONG_THREADS = 224;
// smem: Q 16K | P 32K | 2 stages x (K 16K | V 16K) | barriers
static constexpr int L_Q = 0, L_P = 16384, L_KV = L_P + 32768, L_BAR = L_KV + 2 * 32768;
static constexpr int LONG_SMEM = L_BAR + 256;  // 114944 B -> 2 CTAs/SM
static constexpr int L_PV_COL = 128;           // TMEM column of the P·V scratch

__device__ __forceinline__ float ex2l(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ uint32_t swl(int row, int col /* bf16 element 0..63 */) {
    return row * 128 + ((((col >> 3) ^ (row & 7)) << 4) | ((col & 7) << 1));
}
// 32 lanes x 16 columns of fp32 (half of tmem_ld_32x32: O already holds 64 registers of the row thread)
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void unpack8(const uint4 w, float* f) {
    f[0] = bf16_lo(w.x), f[1] = bf16_hi(w.x), f[2] = bf16_lo(w.y), f[3] = bf16_hi(w.y);
    f[4] = bf16_lo(w.z), f[5] = bf16_hi(w.z), f[6] = bf16_lo(w.w), f[7] = bf16_hi(w.w);
}
__device__ __forceinline__ float dot8(const float* q, const uint4 w) {
    return q[0] * bf16_lo(w.x) + q[1] * bf16_hi(w.x) + q[2] * bf16_lo(w.y) + q[3] * bf16_hi(w.y) + q[4] * bf16_lo(w.z) +
           q[5] * bf16_hi(w.z) + q[6] * bf16_lo(w.w) + q[7] * bf16_hi(w.w);
}

__global__ void __launch_bounds__(LONG_THREADS, 2) attn_fwd_long_kernel(const __grid_constant__ CUtensorMap tm, const AttnDev p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    if (smem_u32(smem) & 1023) __trap();  // SWIZZLE_128B tiles need a 1024B-aligned base
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L_BAR);
    uint64_t* q_full = bars + 0;    // Q landed
    uint64_t* kv_full = bars + 1;   // [2] K,V of stage s landed
    uint64_t* kv_empty = bars + 3;  // [2] stage s free again (P·V of its block completed)
    uint64_t* s_full = bars + 5;    // S of the current block complete in TMEM
    uint64_t* p_full = bars + 6;    // P written, S read, previous PV read (128 arrivals)
    uint64_t* pv_done = bars + 7;   // PV of the current block complete (P buffer reusable)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int qt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
    const int D = p.D, T = p.T, prefix = p.prefix, HW = p.HW;
    const int nkb = (HW + 127) >> 7;
    const long seq_row0 = (long)b * T;

    if (threadIdx.x == 0) {
        tma_prefetch_desc(&tm);
        mbar_init(q_full, 1);
        for (int s = 0; s < 2; ++s) mbar_init(&kv_full[s], 1), mbar_init(&kv_empty[s], 1);
        mbar_init(s_full, 1), mbar_init(p_full, 128), mbar_init(pv_done, 1);
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
        // ---------------- TMA producer
        if (lane == 0) {
            mbar_expect_tx(q_full, 16384);
            tma_load_3d(smem + L_Q, &tm, q_full, h * 64, prefix + 128 * qt, b);
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb & 1, u = kb >> 1;
                if (u >= 1) mbar_wait(&kv_empty[s], (u - 1) & 1);
                uint8_t* kv = smem + L_KV + s * 32768;
                mbar_expect_tx(&kv_full[s], 32768);
                tma_load_3d(kv, &tm, &kv_full[s], D + h * 64, prefix + 128 * kb, b);
                tma_load_3d(kv + 16384, &tm, &kv_full[s], 2 * D + h * 64, prefix + 128 * kb, b);
            }
        }
    } else if (warp == 5) {
        // ---------------- MMA issuer.  S_{kb+1} is issued right behind PV_kb: the softmax has finished reading S_kb
        // when it publishes P_kb, so the next score block overlaps the tail of this one's softmax / P·V.
        if (lane == 0) {
            const uint32_t idesc_s = umma_idesc_bf16(128, 128, 0, 0);
            const uint32_t idesc_o = umma_idesc_bf16(128, 64, 0, 1);  // B (= V) is MN-major
            const uint32_t qa = smem_u32(smem + L_Q), pa = smem_u32(smem + L_P);
            auto issue_s = [&](int kb) {
                const int s = kb & 1;
                mbar_wait(&kv_full[s], (kb >> 1) & 1);
                tc_fence_after();
                const uint32_t ka = smem_u32(smem + L_KV + s * 32768);
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    umma_bf16_ss(tmem, umma_desc_sw128(qa + j * 32, 0, 1024), umma_desc_sw128(ka + j * 32, 0, 1024), idesc_s,
                                 j > 0);
                umma_commit(s_full);
            };
            mbar_wait(q_full, 0);
            issue_s(0);
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb & 1;
                mbar_wait(p_full, kb & 1);
                tc_fence_after();
                const uint32_t va = smem_u32(smem + L_KV + s * 32768 + 16384);
#pragma unroll
                for (int j = 0; j < 8; ++j) {  // 8 k-steps of 16 keys
                    const uint64_t ad = umma_desc_sw128(pa + (j >> 2) * 16384 + (j & 3) * 32, 0, 1024);
                    const uint64_t bd = umma_desc_sw128(va + j * 2048, 8192, 1024);
                    umma_bf16_ss(tmem + L_PV_COL, ad, bd, idesc_o, j > 0 ? 1u : 0u);
                }
                umma_commit(pv_done);
                umma_commit(&kv_empty[s]);
                if (kb + 1 < nkb) issue_s(kb + 1);
            }
        }
    } else if (warp <= 4) {
        // ---------------- softmax: one thread per query row
        const int q4 = warp & 3;
        const int r = q4 * 32 + lane;   // row within the tile == TMEM lane
        const int qpos = 128 * qt + r;  // patch index of this query
        const uint32_t trow = tmem + (uint32_t(q4 * 32) << 16);
        const float sl2 = p.scale_log2;

        // the running state starts from the prefix keys (CUDA cores): q row from smem (swizzled), k / v rows from global
        float m = -INFINITY, l = 0.f, o[64];
        mbar_wait(q_full, 0);
        float s_pre[ATT_MAX_PREFIX];
        if (prefix > 0) {
            float qf[64];
#pragma unroll
            for (int c = 0; c < 8; ++c) unpack8(*reinterpret_cast<const uint4*>(smem + L_Q + swl(r, c * 8)), qf + c * 8);
#pragma unroll
            for (int j = 0; j < ATT_MAX_PREFIX; ++j) {
                s_pre[j] = -INFINITY;
                if (j < prefix) {
                    const uint4* kp = reinterpret_cast<const uint4*>(p.qkv + (seq_row0 + j) * 3 * D + D + h * 64);
                    float acc = 0.f;
#pragma unroll
                    for (int c = 0; c < 8; ++c) acc += dot8(qf + c * 8, __ldg(kp + c));
                    s_pre[j] = acc;
                }
                m = fmaxf(m, s_pre[j]);
            }
        }
#pragma unroll
        for (int i = 0; i < 64; ++i) o[i] = 0.f;
        if (prefix > 0) {  // (q is dead by now: q and O are never live together)
            const float msc = m * sl2;
#pragma unroll
            for (int j = 0; j < ATT_MAX_PREFIX; ++j) {
                if (j < prefix) {
                    const float e = ex2l(s_pre[j] * sl2 - msc);
                    l += e;
                    const float pe = bf16_round(e);  // the tensor-core blocks see bf16 P as well
                    const uint4* vp = reinterpret_cast<const uint4*>(p.qkv + (seq_row0 + j) * 3 * D + 2 * D + h * 64);
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        float v[8];
                        unpack8(__ldg(vp + c), v);
#pragma unroll
                        for (int t = 0; t < 8; ++t) o[c * 8 + t] += pe * v[t];
                    }
                }
            }
        }

        for (int kb = 0; kb < nkb; ++kb) {
            const int lim = min(128, HW - 128 * kb);  // valid key columns of this block (warp-uniform)
            mbar_wait(s_full, kb & 1);
            tc_fence_after();
            // pass 1: block row max
            float mb = -INFINITY;
            if (lim == 128) {
                float m0 = -INFINITY, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
#pragma unroll
                for (int c = 0; c < 128; c += 16) {
                    uint32_t rr[16];
                    tmem_ld_32x16(trow + c, rr);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 16; i += 4) {
                        m0 = fmaxf(m0, __uint_as_float(rr[i])), m1 = fmaxf(m1, __uint_as_float(rr[i + 1]));
                        m2 = fmaxf(m2, __uint_as_float(rr[i + 2])), m3 = fmaxf(m3, __uint_as_float(rr[i + 3]));
                    }
                }
                mb = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
            } else {
                for (int c = 0; c < lim; c += 16) {
                    uint32_t rr[16];
                    tmem_ld_32x16(trow + c, rr);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 16; ++i)
                        if (c + i < lim) mb = fmaxf(mb, __uint_as_float(rr[i]));
                }
            }
            const float m_new = fmaxf(m, mb);  // finite: every block holds at least one valid key
            const float alpha = ex2l((m - m_new) * sl2);  // 0 when m = -inf (no prefix, first block)
            const float msc = m_new * sl2;
            m = m_new;
            // fold the previous block's P·V into O (both are in units of the previous max), then rescale
            if (kb > 0) {
                mbar_wait(pv_done, (kb - 1) & 1);  // also: the P buffer is free again
                tc_fence_after();
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    uint32_t v[16];
                    tmem_ld_32x16(trow + L_PV_COL + 16 * q, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 16; ++i) o[16 * q + i] = (o[16 * q + i] + __uint_as_float(v[i])) * alpha;
                }
            } else {
#pragma unroll
                for (int i = 0; i < 64; ++i) o[i] *= alpha;
            }
            l *= alpha;
            // pass 2: p = exp2(s*scale*log2e - m*scale*log2e) as bf16 into the swizzled P tile (two 64-key regions)
            float l0 = 0.f, l1 = 0.f;
#pragma unroll 1
            for (int c16 = 0; c16 < 8; ++c16) {
                const int c = c16 * 16;
                uint8_t* pb = smem + L_P + (c16 >> 2) * 16384;  // keys [64 k, 64 k + 64) form region k
                if (c >= lim) {
#pragma unroll
                    for (int v4 = 0; v4 < 2; ++v4)
                        *reinterpret_cast<uint4*>(pb + swl(r, (c16 & 3) * 16 + v4 * 8)) = make_uint4(0u, 0u, 0u, 0u);
                    continue;
                }
                uint32_t rr[16];
                tmem_ld_32x16(trow + c, rr);
                tmem_ld_wait();
                const int nv = min(16, lim - c);  // valid columns of this chunk; the rest get P = 0
#pragma unroll
                for (int v4 = 0; v4 < 2; ++v4) {
                    uint32_t pk[4];
#pragma unroll
                    for (int i = 0; i < 8; i += 2) {
                        const int k = v4 * 8 + i;
                        float e0 = ex2l(fmaf(__uint_as_float(rr[k]), sl2, -msc));
                        float e1 = ex2l(fmaf(__uint_as_float(rr[k + 1]), sl2, -msc));
                        if (nv < 16) e0 = k < nv ? e0 : 0.f, e1 = k + 1 < nv ? e1 : 0.f;
                        l0 += e0, l1 += e1;
                        pk[i >> 1] = pack_bf16x2(e0, e1);
                    }
                    *reinterpret_cast<uint4*>(pb + swl(r, (c16 & 3) * 16 + v4 * 8)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                }
            }
            l += l0 + l1;
            tc_fence_before();
            fence_proxy_async_smem();
            mbar_arrive(p_full);
        }
        // epilogue: the last block's P·V
        mbar_wait(pv_done, (nkb - 1) & 1);
        tc_fence_after();
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            uint32_t v[16];
            tmem_ld_32x16(trow + L_PV_COL + 16 * q, v);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) o[16 * q + i] += __uint_as_float(v[i]);
        }
        if (qpos < HW) {
            const int qtok = prefix + qpos;
            const float inv = 1.f / l;
            __nv_bfloat16* op = p.out + (seq_row0 + qtok) * D + h * 64;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                uint4 w;
                w.x = pack_bf16x2(o[c * 8] * inv, o[c * 8 + 1] * inv), w.y = pack_bf16x2(o[c * 8 + 2] * inv, o[c * 8 + 3] * inv);
                w.z = pack_bf16x2(o[c * 8 + 4] * inv, o[c * 8 + 5] * inv), w.w = pack_bf16x2(o[c * 8 + 6] * inv, o[c * 8 + 7] * inv);
                *reinterpret_cast<uint4*>(op + c * 8) = w;
            }
            if (p.lse) p.lse[((long)b * p.H + h) * T + qtok] = m * p.scale + logf(l);
        }
        tc_fence_before();
    } else {
        // ---------------- warp 6: prefix query rows of the image (qt == 0 only).  A lane pair takes one key at a time
        // (keys k, k+16, ... for pair k), each lane owning 32 of the 64 dims: half a dot product plus one shuffle gives the
        // score; every pair runs its own online softmax with an fp32 accumulator, and the 16 partial states are merged.
        if (qt == 0 && prefix > 0) {
            const int half = lane & 1, pair = lane >> 1;
            for (int j = 0; j < prefix; ++j) {
                uint4 q4[4];  // my 32 dims of q, packed bf16
                float acc[32];
                const uint4* qp = reinterpret_cast<const uint4*>(p.qkv + (seq_row0 + j) * 3 * D + h * 64 + 32 * half);
#pragma unroll
                for (int c = 0; c < 4; ++c) q4[c] = __ldg(qp + c);
#pragma unroll
                for (int i = 0; i < 32; ++i) acc[i] = 0.f;
                float m = -INFINITY, l = 0.f;
                for (int t0 = 0; t0 < T; t0 += 16) {  // warp-uniform trip count: the shuffle needs every lane
                    const int t = t0 + pair;
                    const bool valid = t < T;
                    const long row = (seq_row0 + (valid ? t : 0)) * 3 * D + h * 64 + 32 * half;
                    const uint4* kp = reinterpret_cast<const uint4*>(p.qkv + row + D);
                    const uint4* vp = reinterpret_cast<const uint4*>(p.qkv + row + 2 * D);
                    float s = 0.f;
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        float qf[8];
                        unpack8(q4[c], qf);
                        s += dot8(qf, __ldg(kp + c));
                    }
                    s += __shfl_xor_sync(0xffffffffu, s, 1);
                    if (!valid) continue;
                    if (s > m) {
                        const float a = ex2l((m - s) * p.scale_log2);  // 0 on the first key
                        l *= a;
#pragma unroll
                        for (int i = 0; i < 32; ++i) acc[i] *= a;
                        m = s;
                    }
                    const float e = ex2l((s - m) * p.scale_log2);
                    l += e;
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        float v[8];
                        unpack8(__ldg(vp + c), v);
#pragma unroll
                        for (int u = 0; u < 8; ++u) acc[c * 8 + u] += e * v[u];
                    }
                }
                // merge the 16 pairs (lanes of equal parity): every pair has seen at least one key, m is finite
                float mw = m;
#pragma unroll
                for (int o = 2; o < 32; o <<= 1) mw = fmaxf(mw, __shfl_xor_sync(0xffffffffu, mw, o));
                const float f = ex2l((m - mw) * p.scale_log2);
                l *= f;
#pragma unroll
                for (int o = 2; o < 32; o <<= 1) l += __shfl_xor_sync(0xffffffffu, l, o);
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    float x = acc[i] * f;
#pragma unroll
                    for (int o = 2; o < 32; o <<= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
                    acc[i] = x;
                }
                if (lane < 2) {  // lane 0: dims [0,32), lane 1: dims [32,64)
                    const float inv = 1.f / l;
                    uint4* op = reinterpret_cast<uint4*>(p.out + (seq_row0 + j) * D + h * 64 + 32 * half);
#pragma unroll
                    for (int c = 0; c < 4; ++c)
                        op[c] = make_uint4(pack_bf16x2(acc[c * 8] * inv, acc[c * 8 + 1] * inv), pack_bf16x2(acc[c * 8 + 2] * inv, acc[c * 8 + 3] * inv),
                                           pack_bf16x2(acc[c * 8 + 4] * inv, acc[c * 8 + 5] * inv), pack_bf16x2(acc[c * 8 + 6] * inv, acc[c * 8 + 7] * inv));
                    if (p.lse && lane == 0) p.lse[((long)b * p.H + h) * T + j] = mw * p.scale + logf(l);
                }
            }
        }
    }

    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem, 256);
    }
}

int attn_fwd_long_launch(const AttnDev& p, cudaStream_t st) {
    VTP_CHECK_ARG(!p.causal && !p.pack && p.HW > 256 && p.prefix <= ATT_MAX_PREFIX,
                  "attention_fwd(long): needs HW > 256 and no causal mask");
    static bool configured = false;
    if (!configured) {
        VTP_CUDA(cudaFuncSetAttribute(attn_fwd_long_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, LONG_SMEM));
        configured = true;
    }
    // [B][T][3D]: boxes of 128 rows x 64 columns that never cross into the next image (zero fill past T)
    CUtensorMap tm;
    uint64_t dims[3] = {(uint64_t)3 * p.D, (uint64_t)p.T, (uint64_t)p.B};
    uint64_t strides[2] = {(uint64_t)3 * p.D * 2, (uint64_t)p.T * 3 * p.D * 2};
    uint32_t box[3] = {64, 128, 1};
    int rc = make_tmap_bf16(&tm, p.qkv, 3, dims, strides, box);
    if (rc) return rc;
    dim3 grid(ceil_div(p.HW, 128), p.H, p.B);
    attn_fwd_long_kernel<<<grid, LONG_THREADS, LONG_SMEM, st>>>(tm, p);
    VTP_LAUNCH_CHECK();
    return VTP_OK;
}

}  // namespace vtp
