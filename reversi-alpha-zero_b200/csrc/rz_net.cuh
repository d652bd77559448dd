// rz_net.cuh -- policy/value network object shared by the inference kernels and the engine.
//
// Architecture = the reference's ReversiModel.build (agent/model.py:28-72): conv3x3(2->F)+BN+ReLU,
// R residual blocks of two conv3x3(F->F)+BN (ReLU after the first, skip-add then ReLU after the
// second), policy head conv1x1(F->2)+BN+ReLU -> Dense(128->64, softmax), value head
// conv1x1(F->1)+BN+ReLU -> Dense(64->V, relu) -> Dense(V->1, tanh).  BN is folded at load time into a
// per-channel fp32 (scale, shift) applied in the conv epilogue:
//   scale = gamma / sqrt(var + 1e-3),  shift = beta + (bias - mean) * scale.
#pragma once
#include <cuda_fp16.h>
#include "rz_common.cuh"

struct rz_net {
    rz_net_cfg cfg;
    int device;
    bool loaded;
    size_t blob_floats;
    float* blob;         // device copy of the fp32 blob (Keras layouts), used by the generic kernel and the heads
    float* scale_shift;  // [n_conv_layers][2][F] folded BN of conv0 + tower convs; then heads: [2][2] policy, [2][1] value
    // offsets (in floats) into blob
    size_t off_conv0, off_res0, res_stride_conv;  // kernel offset of conv0; of res0.conv1; floats per (conv+bn) group
    size_t off_policy_conv, off_policy_fc_k, off_policy_fc_b;
    size_t off_value_conv, off_value_fc1_k, off_value_fc1_b, off_value_fc2_k, off_value_fc2_b;
    // tcgen05 tower (F == 256 only, rz_net_tc.cu): fp16 UMMA K-major no-swizzle images in the order its K / N loops consume them
    __half* tc_w0;       // [cta 2][nh 2][kc 4][n 64][8]: layer-0 weights, K = 18 padded to 32
    __half* tc_w;        // [2R layers][36 stages][cta 2][kbl 2][kc 8][n 64][8]: one 16 KB image per CTA and pipeline stage
    // scratch for the host-buffer predict path
    void* scratch;
    size_t scratch_bytes;
};

namespace rz {

inline int n_conv_layers(const rz_net_cfg& c) { return 1 + 2 * c.res_blocks; }
// per-layer folded BN parameters: scale at [l][0][*], shift at [l][1][*]
inline size_t ss_floats(const rz_net_cfg& c) { return (size_t)n_conv_layers(c) * 2 * c.filters + 4 + 2; }

int net_forward_generic(rz_net* net, const uint64_t* own, const uint64_t* enemy, float* policy, float* value, size_t n,
                        cudaStream_t stream, const uint32_t* n_dev = nullptr);
// batch size known only on the device (count_dev), at most max_n
int net_forward_counted(rz_net* net, const uint64_t* own, const uint64_t* enemy, float* policy, float* value,
                        const uint32_t* count_dev, size_t max_n, int impl, cudaStream_t stream);
// the fused tcgen05 tower on CTA pairs (rz_net_tc.cu)
int net_forward_tc(rz_net* net, const uint64_t* own, const uint64_t* enemy, float* policy, float* value, size_t n,
                   cudaStream_t stream, float* dbg_tower /* nullable: [n][64][256] fp32 tower output */,
                   const uint32_t* n_dev = nullptr /* nullable: actual batch size in device memory (<= n) */,
                   float* dbg_logits = nullptr /* nullable: [n][64] policy logits */, float* dbg_vlogit = nullptr /* nullable: [n] */);
int net_pack_tc(rz_net* net, cudaStream_t stream);
int net_forward(rz_net* net, const uint64_t* own, const uint64_t* enemy, float* policy, float* value, size_t n, int impl,
                cudaStream_t stream);

}  // namespace rz
