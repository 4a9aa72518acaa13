// vtp_b200 — argument block shared by the attention forward kernels (attention.cu, attention_pipe.cu).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

namespace vtp {

static constexpr int ATT_MAX_PREFIX = 4;

struct AttnDev {
    const __nv_bfloat16* qkv;  // [B*T][3D]
    __nv_bfloat16* out;        // [B*T][D]
    float* lse;                // [B][H][T] or null
    int B, T, H, D, prefix, HW, causal, nkt;  // nkt = number of 128-key tiles (1|2)
    int pack;  // > 0: `pack` whole sequences (T <= 64 tokens, prefix tokens included as ordinary rows) share one 128-row tile
    float scale_log2;                         // scale * log2(e)
    float scale;
};

// persistent ping-pong forward for 128 < HW <= 256 (attention_pipe.cu); default for those shapes, VTP_ATTN_FWD_PIPE=0 opts out
int attn_fwd_pipe_launch(const CUtensorMap& tm, const AttnDev& p, cudaStream_t st);
// flash-style forward for HW > 256, non-causal (attention_long.cu); builds its own per-image [B][T][3D] tensor map
int attn_fwd_long_launch(const AttnDev& p, cudaStream_t st);

}  // namespace vtp
