// rz_net.cu -- network object: creation, weight loading (BN folding, tcgen05 packing), the generic
// CUDA-core forward kernel (any ModelConfig, e.g. config/mini.yml's 16 filters x 1 block) and the
// predict entry points of the C ABI (agent/api.py:30-45 ReversiModelAPI.predict).
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <new>
#include "rz_bitboard.cuh"
#include "rz_net.cuh"

namespace rz {

constexpr float kBnEps = 1e-3f;  // Keras BatchNormalization default epsilon (agent/model.py:35)

// ---- BN folding --------------------------------------------------------------------------------
// group layout in the blob: kernel[k*k*cin*cout], bias[cout], gamma, beta, mean, var
__global__ void fold_bn_kernel(const float* __restrict__ blob, size_t group_off, size_t kernel_floats, int cout,
                               float* __restrict__ scale, float* __restrict__ shift) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cout) return;
    const float* p = blob + group_off + kernel_floats;
    float bias = p[c], gamma = p[cout + c], beta = p[2 * cout + c], mean = p[3 * cout + c], var = p[4 * cout + c];
    float s = gamma / sqrtf(var + kBnEps);
    scale[c] = s;
    shift[c] = beta + (bias - mean) * s;
}

// ---- generic forward kernel ---------------------------------------------------------------------
// One CTA per position, activations in shared memory as fp32 [C][10][10] (zero border), two buffers.
// Thread t owns output channel oc = t % F and PIX pixels; weights are read from the fp32 blob in the
// Keras layout [kh][kw][Cin][Cout], i.e. coalesced across oc.
constexpr int kGThreads = 256;

template <int PIX>
__device__ __forceinline__ void conv3x3_layer(const float* __restrict__ in, float* __restrict__ out, const float* __restrict__ w,
                                              const float* __restrict__ scale, const float* __restrict__ shift, int cin, int F,
                                              bool add_residual, int oc, int pg, bool active) {
    // pixels handled by this thread: p = pg * PIX + i
    float acc[PIX];
#pragma unroll
    for (int i = 0; i < PIX; ++i) acc[i] = 0.f;
    if (active) {
        for (int ci = 0; ci < cin; ++ci) {
            const float* inc = in + ci * 100;
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
                const float wv = __ldg(w + ((size_t)tap * cin + ci) * F + oc);
                const int dy = tap / 3, dx = tap % 3;  // already +1-shifted into the padded frame
#pragma unroll
                for (int i = 0; i < PIX; ++i) {
                    const int p = pg * PIX + i;
                    acc[i] = fmaf(inc[((p >> 3) + dy) * 10 + (p & 7) + dx], wv, acc[i]);
                }
            }
        }
        const float s = scale[oc], b = shift[oc];
#pragma unroll
        for (int i = 0; i < PIX; ++i) {
            const int p = pg * PIX + i;
            const int o = oc * 100 + ((p >> 3) + 1) * 10 + (p & 7) + 1;
            float y = fmaf(acc[i], s, b);
            if (add_residual) y += out[o];  // in-place residual: out holds the block input
            out[o] = fmaxf(y, 0.f);
        }
    }
}

template <int PIX>
__global__ void __launch_bounds__(kGThreads) net_generic_kernel(const float* __restrict__ blob, const float* __restrict__ ss,
                                                                rz_net net, const u64* __restrict__ own, const u64* __restrict__ enemy,
                                                                float* __restrict__ policy, float* __restrict__ value, size_t n,
                                                                const uint32_t* __restrict__ n_dev) {
    extern __shared__ float smem[];
    if (n_dev) n = *n_dev;
    const int F = net.cfg.filters, R = net.cfg.res_blocks, V = net.cfg.value_fc;
    float* bufA = smem;               // [F][100]
    float* bufB = smem + F * 100;     // [F][100]
    float* hp = bufB + F * 100;       // [128] policy head activations (c*64 + pix)
    float* hv = hp + 128;             // [64]
    float* fc = hv + 64;              // [max(V,64)]
    const int t = threadIdx.x;
    constexpr int NPG = 64 / PIX;
    const int oc = t % F, pg = t / F;
    const bool active = (t < F * NPG) && (pg < NPG);

    for (size_t pos = blockIdx.x; pos < n; pos += gridDim.x) {
        for (int i = t; i < 2 * F * 100; i += kGThreads) smem[i] = 0.f;
        __syncthreads();
        const u64 o = own[pos], e = enemy[pos];
        if (t < 128) {  // input planes into bufB channels 0 (own), 1 (enemy)
            const int c = t >> 6, p = t & 63;
            bufB[c * 100 + ((p >> 3) + 1) * 10 + (p & 7) + 1] = (float)(((c ? e : o) >> p) & 1ULL);
        }
        __syncthreads();
        // conv0: bufB(2 ch) -> bufA
        conv3x3_layer<PIX>(bufB, bufA, blob + net.off_conv0, ss, ss + F, 2, F, false, oc, pg, active);
        __syncthreads();
        for (int r = 0; r < R; ++r) {
            const float* w1 = blob + net.off_res0 + (size_t)(2 * r) * net.res_stride_conv;
            const float* w2 = w1 + net.res_stride_conv;
            const float* ss1 = ss + (size_t)(1 + 2 * r) * 2 * F;
            const float* ss2 = ss1 + 2 * F;
            conv3x3_layer<PIX>(bufA, bufB, w1, ss1, ss1 + F, F, F, false, oc, pg, active);
            __syncthreads();
            conv3x3_layer<PIX>(bufB, bufA, w2, ss2, ss2 + F, F, F, true, oc, pg, active);
            __syncthreads();
        }
        // heads: 1x1 convs (policy 2 ch, value 1 ch) + BN + ReLU
        const float* ssh = ss + (size_t)(1 + 2 * R) * 2 * F;  // policy: scale[2], shift[2]; value: scale, shift
        if (t < 192) {
            const int c = t >> 6, p = t & 63;  // c = 0,1 policy channels; 2 = value
            const float* w = c < 2 ? blob + net.off_policy_conv + c : blob + net.off_value_conv;
            const int wstride = c < 2 ? 2 : 1;
            float acc = 0.f;
            const int o2 = ((p >> 3) + 1) * 10 + (p & 7) + 1;
            for (int ci = 0; ci < F; ++ci) acc = fmaf(bufA[ci * 100 + o2], __ldg(w + (size_t)ci * wstride), acc);
            if (c < 2) hp[c * 64 + p] = fmaxf(fmaf(acc, ssh[c], ssh[2 + c]), 0.f);
            else       hv[p] = fmaxf(fmaf(acc, ssh[4], ssh[5]), 0.f);
        }
        __syncthreads();
        if (t < 64) {  // policy logits
            const float* k = blob + net.off_policy_fc_k;
            float acc = __ldg(blob + net.off_policy_fc_b + t);
            for (int i = 0; i < 128; ++i) acc = fmaf(hp[i], __ldg(k + i * 64 + t), acc);
            fc[t] = acc;
        }
        __syncthreads();
        if (t < 64) {  // softmax over 64 logits
            float m = -INFINITY;
            for (int i = 0; i < 64; ++i) m = fmaxf(m, fc[i]);
            float sum = 0.f;
            for (int i = 0; i < 64; ++i) sum += expf(fc[i] - m);
            policy[pos * 64 + t] = expf(fc[t] - m) / sum;
        }
        __syncthreads();
        for (int j = t; j < V; j += kGThreads) {  // value fc1 + relu
            const float* k = blob + net.off_value_fc1_k;
            float acc = __ldg(blob + net.off_value_fc1_b + j);
            for (int i = 0; i < 64; ++i) acc = fmaf(hv[i], __ldg(k + (size_t)i * V + j), acc);
            fc[j] = fmaxf(acc, 0.f);
        }
        __syncthreads();
        if (t == 0) {
            float acc = __ldg(blob + net.off_value_fc2_b);
            for (int j = 0; j < V; ++j) acc = fmaf(fc[j], __ldg(blob + net.off_value_fc2_k + j), acc);
            value[pos] = tanhf(acc);
        }
        __syncthreads();
    }
}

int net_forward_generic(rz_net* net, const uint64_t* own, const uint64_t* enemy, float* policy, float* value, size_t n,
                        cudaStream_t stream, const uint32_t* n_dev) {
    const int F = net->cfg.filters, V = net->cfg.value_fc;
    RZ_REQUIRE(F >= 2 && F <= 256, "generic kernel supports 2 <= filters <= 256 (got %d)", F);
    const size_t smem = ((size_t)2 * F * 100 + 128 + 64 + (V > 64 ? V : 64)) * sizeof(float);
    int npg = kGThreads / F;  // pixel groups that fit beside the channel dimension
    int pix = 64;
    while (pix > 4 && 64 / (pix / 2) <= npg) pix /= 2;
    size_t blocks = n < (size_t)num_sms() * 2 ? n : (size_t)num_sms() * 2;
    if (smem > 110 * 1024) blocks = n < (size_t)num_sms() ? n : (size_t)num_sms();
#define RZ_LAUNCH_G(P)                                                                                             \
    do {                                                                                                           \
        RZ_CUDA_TRY(cudaFuncSetAttribute(net_generic_kernel<P>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        net_generic_kernel<P><<<(unsigned)blocks, kGThreads, smem, stream>>>(net->blob, net->scale_shift, *net, own, enemy, policy, value, n, n_dev); \
    } while (0)
    switch (pix) {
        case 64: RZ_LAUNCH_G(64); break;
        case 32: RZ_LAUNCH_G(32); break;
        case 16: RZ_LAUNCH_G(16); break;
        case 8: RZ_LAUNCH_G(8); break;
        default: RZ_LAUNCH_G(4); break;
    }
#undef RZ_LAUNCH_G
    RZ_LAUNCH_CHECK();
    return RZ_OK;
}

int net_forward(rz_net* net, const uint64_t* own, const uint64_t* enemy, float* policy, float* value, size_t n, int impl,
                cudaStream_t stream) {
    if (!net->loaded) { set_error("rz_net: weights not loaded"); return RZ_ESTATE; }
    if (n == 0) return RZ_OK;
    if (impl == RZ_NET_IMPL_AUTO) impl = net->cfg.filters == 256 ? RZ_NET_IMPL_TCGEN05 : RZ_NET_IMPL_GENERIC;
    if (impl == RZ_NET_IMPL_TCGEN05) {
        RZ_REQUIRE(net->cfg.filters == 256, "tcgen05 tower requires filters == 256 (got %d)", net->cfg.filters);
        return net_forward_tc(net, own, enemy, policy, value, n, stream, nullptr);
    }
    RZ_REQUIRE(impl == RZ_NET_IMPL_GENERIC, "unknown net impl %d", impl);
    return net_forward_generic(net, own, enemy, policy, value, n, stream);
}

int net_forward_counted(rz_net* net, const uint64_t* own, const uint64_t* enemy, float* policy, float* value,
                        const uint32_t* count_dev, size_t max_n, int impl, cudaStream_t stream) {
    if (!net->loaded) { set_error("rz_net: weights not loaded"); return RZ_ESTATE; }
    if (impl == RZ_NET_IMPL_AUTO) impl = net->cfg.filters == 256 ? RZ_NET_IMPL_TCGEN05 : RZ_NET_IMPL_GENERIC;
    if (impl == RZ_NET_IMPL_TCGEN05)
        return net_forward_tc(net, own, enemy, policy, value, max_n, stream, nullptr, count_dev);
    return net_forward_generic(net, own, enemy, policy, value, max_n, stream, count_dev);
}

static int finish_load(rz_net* net, cudaStream_t stream) {
    const rz_net_cfg& c = net->cfg;
    const int F = c.filters, L = n_conv_layers(c);
    float* ss = net->scale_shift;
    for (int l = 0; l < L; ++l) {
        const size_t off = l == 0 ? net->off_conv0 : net->off_res0 + (size_t)(l - 1) * net->res_stride_conv;
        const size_t kf = l == 0 ? (size_t)9 * 2 * F : (size_t)9 * F * F;
        fold_bn_kernel<<<(F + 127) / 128, 128, 0, stream>>>(net->blob, off, kf, F, ss + (size_t)l * 2 * F, ss + (size_t)l * 2 * F + F);
    }
    float* ssh = ss + (size_t)L * 2 * F;
    fold_bn_kernel<<<1, 32, 0, stream>>>(net->blob, net->off_policy_conv, (size_t)F * 2, 2, ssh, ssh + 2);
    fold_bn_kernel<<<1, 32, 0, stream>>>(net->blob, net->off_value_conv, (size_t)F, 1, ssh + 4, ssh + 5);
    RZ_LAUNCH_CHECK();
    if (F == 256) RZ_TRY(net_pack_tc(net, stream));
    RZ_CUDA_TRY(cudaStreamSynchronize(stream));
    net->loaded = true;
    return RZ_OK;
}

}  // namespace rz

using namespace rz;

extern "C" {

int rz_net_create(const rz_net_cfg* cfg, int device, rz_net** out) {
    RZ_REQUIRE(cfg && out, "rz_net_create: null pointer");
    RZ_REQUIRE(cfg->kernel_size == 3, "only cnn_filter_size == 3 is supported (got %d)", cfg->kernel_size);
    RZ_REQUIRE(cfg->filters >= 2 && cfg->filters <= 256 && cfg->res_blocks >= 0 && cfg->res_blocks <= 64 && cfg->value_fc >= 1 &&
                   cfg->value_fc <= 4096,
               "unsupported model configuration (filters=%d res_blocks=%d value_fc=%d)", cfg->filters, cfg->res_blocks, cfg->value_fc);
    RZ_CUDA_TRY(cudaSetDevice(device));
    rz_net* net = new (std::nothrow) rz_net();
    if (!net) { set_error("out of host memory"); return RZ_ENOMEM; }
    memset(net, 0, sizeof(*net));
    net->cfg = *cfg;
    net->device = device;
    const size_t F = cfg->filters, V = cfg->value_fc, R = cfg->res_blocks;
    size_t off = 0;
    net->off_conv0 = off; off += 9 * 2 * F + 5 * F;
    net->off_res0 = off; net->res_stride_conv = 9 * F * F + 5 * F; off += 2 * R * net->res_stride_conv;
    net->off_policy_conv = off; off += F * 2 + 5 * 2;
    net->off_policy_fc_k = off; off += 128 * 64;
    net->off_policy_fc_b = off; off += 64;
    net->off_value_conv = off; off += F + 5;
    net->off_value_fc1_k = off; off += 64 * V;
    net->off_value_fc1_b = off; off += V;
    net->off_value_fc2_k = off; off += V;
    net->off_value_fc2_b = off; off += 1;
    net->blob_floats = off;
    cudaError_t e = cudaMalloc(&net->blob, off * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(&net->scale_shift, ss_floats(*cfg) * sizeof(float));
    if (e == cudaSuccess && F == 256) {
        e = cudaMalloc(&net->tc_w0, (size_t)2 * 2 * 4 * 64 * 8 * sizeof(__half));
        if (e == cudaSuccess && R > 0) e = cudaMalloc(&net->tc_w, (size_t)2 * R * 36 * 2 * 8192 * sizeof(__half));
    }
    if (e != cudaSuccess) {
        set_error("rz_net_create: cudaMalloc failed: %s", cudaGetErrorString(e));
        cudaGetLastError();
        rz_net_destroy(net);
        return RZ_ENOMEM;
    }
    *out = net;
    return RZ_OK;
}

int rz_net_destroy(rz_net* net) {
    if (!net) return RZ_OK;
    cudaSetDevice(net->device);
    cudaFree(net->blob); cudaFree(net->scale_shift); cudaFree(net->tc_w0); cudaFree(net->tc_w); cudaFree(net->scratch);
    delete net;
    return RZ_OK;
}

int rz_net_blob_size(const rz_net* net, size_t* n_floats) {
    RZ_REQUIRE(net && n_floats, "rz_net_blob_size: null pointer");
    *n_floats = net->blob_floats;
    return RZ_OK;
}

int rz_net_load_weights(rz_net* net, const float* blob_host, size_t n_floats) {
    RZ_REQUIRE(net && blob_host, "rz_net_load_weights: null pointer");
    RZ_REQUIRE(n_floats == net->blob_floats, "weight blob has %zu floats, this configuration needs %zu", n_floats, net->blob_floats);
    RZ_CUDA_TRY(cudaSetDevice(net->device));
    RZ_CUDA_TRY(cudaMemcpy(net->blob, blob_host, n_floats * sizeof(float), cudaMemcpyHostToDevice));
    return finish_load(net, 0);
}

int rz_net_load_weights_dev(rz_net* net, const float* blob_dev, size_t n_floats, void* stream) {
    RZ_REQUIRE(net && blob_dev, "rz_net_load_weights_dev: null pointer");
    RZ_REQUIRE(n_floats == net->blob_floats, "weight blob has %zu floats, this configuration needs %zu", n_floats, net->blob_floats);
    RZ_CUDA_TRY(cudaSetDevice(net->device));
    RZ_CUDA_TRY(cudaMemcpyAsync(net->blob, blob_dev, n_floats * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return finish_load(net, (cudaStream_t)stream);
}

int rz_net_predict_dev(rz_net* net, const uint64_t* own, const uint64_t* enemy, float* policy, float* value, size_t n, int impl,
                       void* stream) {
    RZ_REQUIRE(net && (n == 0 || (own && enemy && policy && value)), "rz_net_predict_dev: null pointer");
    return net_forward(net, own, enemy, policy, value, n, impl, (cudaStream_t)stream);
}

int rz_net_debug_tower_dev(rz_net* net, const uint64_t* own, const uint64_t* enemy, float* policy, float* value, float* tower, size_t n,
                           void* stream) {
    RZ_REQUIRE(net && own && enemy && policy && value && tower, "rz_net_debug_tower_dev: null pointer");
    if (!net->loaded) { set_error("rz_net: weights not loaded"); return RZ_ESTATE; }
    return net_forward_tc(net, own, enemy, policy, value, n, (cudaStream_t)stream, tower);
}

int rz_net_debug_heads_dev(rz_net* net, const uint64_t* own, const uint64_t* enemy, float* policy, float* value, float* tower,
                           float* policy_logits, float* value_logit, size_t n, void* stream) {
    RZ_REQUIRE(net && own && enemy && policy && value && policy_logits && value_logit, "rz_net_debug_heads_dev: null pointer");
    if (!net->loaded) { set_error("rz_net: weights not loaded"); return RZ_ESTATE; }
    return net_forward_tc(net, own, enemy, policy, value, n, (cudaStream_t)stream, tower, nullptr, policy_logits, value_logit);
}

int rz_net_predict(rz_net* net, const uint8_t* planes, float* policy, float* value, size_t n, int impl) {
    RZ_REQUIRE(net && (n == 0 || (planes && policy && value)), "rz_net_predict: null pointer");
    if (n == 0) return RZ_OK;
    RZ_CUDA_TRY(cudaSetDevice(net->device));
    // pack the {0,1} planes [n][2][8][8] into bitboards on the host (128 B -> 16 B per position)
    const size_t need = n * (16 + 65 * 4) + 256;
    if (need > net->scratch_bytes) {
        cudaFree(net->scratch); net->scratch = nullptr; net->scratch_bytes = 0;
        RZ_CUDA_TRY(cudaMalloc(&net->scratch, need));
        net->scratch_bytes = need;
    }
    uint64_t* hb = (uint64_t*)malloc(n * 16);
    if (!hb) { set_error("out of host memory"); return RZ_ENOMEM; }
    for (size_t i = 0; i < n; ++i) {
        uint64_t o = 0, e = 0;
        const uint8_t* p = planes + i * 128;
        for (int b = 0; b < 64; ++b) { o |= (uint64_t)(p[b] != 0) << b; e |= (uint64_t)(p[64 + b] != 0) << b; }
        hb[i] = o; hb[n + i] = e;
    }
    uint64_t* d_own = (uint64_t*)net->scratch;
    uint64_t* d_en = d_own + n;
    float* d_pol = (float*)(d_en + n);
    float* d_val = d_pol + n * 64;
    cudaError_t ce = cudaMemcpyAsync(d_own, hb, n * 16, cudaMemcpyHostToDevice, 0);
    int rc = RZ_OK;
    if (ce == cudaSuccess) rc = net_forward(net, d_own, d_en, d_pol, d_val, n, impl, 0);
    if (ce == cudaSuccess && rc == RZ_OK) ce = cudaMemcpyAsync(policy, d_pol, n * 64 * sizeof(float), cudaMemcpyDeviceToHost, 0);
    if (ce == cudaSuccess && rc == RZ_OK) ce = cudaMemcpyAsync(value, d_val, n * sizeof(float), cudaMemcpyDeviceToHost, 0);
    if (ce == cudaSuccess && rc == RZ_OK) ce = cudaStreamSynchronize(0);
    free(hb);
    if (rc != RZ_OK) return rc;
    if (ce != cudaSuccess) { set_error("rz_net_predict: %s", cudaGetErrorString(ce)); return RZ_ECUDA; }
    return RZ_OK;
}

}  // extern "C"
