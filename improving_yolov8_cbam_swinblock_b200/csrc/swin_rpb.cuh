// Shared declarations of the relative-position-bias path (SwinBlockRPB): swin_rpb.cu, swin_attn.cu, swin_attn_tc.cu.
#pragma once
#include "common.cuh"

namespace b200 {
// The attention kernels read a dense f32 bias [nh][64][64] (rows / columns >= L zero) and know nothing of ws.  Their
// backward leaves the unscaled dS of each (window, head) or (CTA, warp group, item slot) in its own workspace slot
// [nslots][nh][64][64]; rpb_fold sums the slots in a fixed order and scatters the sum to the table gradient.
constexpr int kRpbMaxWs = 8;
constexpr int kRpbTcCtas = 160;   // grid cap of the tcgen05 backward with bias: its slot count must not depend on the device
int check_rpb(int L, int ws);
size_t rpb_workspace_bytes(long long nslots, int nh);
int rpb_fold(const float* workspace, long long nslots, int nh, int ws, float* gtable, cudaStream_t st);
}  // namespace b200
