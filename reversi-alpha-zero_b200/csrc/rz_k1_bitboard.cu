// rz_k1_bitboard.cu -- K1: stateless batched bitboard operators + their C ABI.
//
// HBM-bound integer work (SURVEY 8(d)): 24 B / position for the legal-move mask, 25 B for the flip
// mask, 42+ B for the fused step.  Layout is structure-of-arrays so every warp access is a fully
// coalesced run.  Two formulations:
//   * bit-sliced (rz_bitsliced.cuh; default for the legal-move and flip operators from 1024 positions on): one thread owns 32
//     positions transposed into one register per square, ~67 integer instructions per position, one CTA of 256 threads per SM
//     (231-240 registers), a warp walks tiles of 1024 positions with 256-byte contiguous loads / stores;
//   * scalar (rz_bitboard.cuh; the tail of a batch, small batches, RZ_K1_IMPL=scalar): two consecutive positions per thread
//     through 128-bit loads / stores, ~180 instructions per position -- integer-issue-bound at a third of the HBM roofline.
// Inputs are streamed with ld.global.nc.L1::no_allocate, outputs with st.global.cs.  Grids are a multiple of the SM count
// (persistent grid-stride loops).
#include <stdlib.h>
#include <string.h>
#include "rz_bitboard.cuh"
#include "rz_bitsliced.cuh"
#include "rz_ptx.cuh"   // mbarrier / bulk-copy wrappers
#include "rz_common.cuh"

namespace rz {

__device__ __forceinline__ ulonglong2 ldg_stream_u64x2(const u64* p) {
    ulonglong2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u64 {%0, %1}, [%2];" : "=l"(r.x), "=l"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ u64 ldg_stream_u64(const u64* p) {
    u64 r;
    asm volatile("ld.global.nc.L1::no_allocate.u64 %0, [%1];" : "=l"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_stream_u64x2(u64* p, u64 a, u64 b) {
    asm volatile("st.global.cs.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(a), "l"(b) : "memory");
}

constexpr int kThreads = 256;

__device__ __forceinline__ void stg_stream_u64(u64* p, u64 a) { asm volatile("st.global.cs.u64 [%0], %1;" ::"l"(p), "l"(a) : "memory"); }

// bit-sliced operators: warp w of the grid handles tiles w, w + n_warps, ...; thread t of the warp owns the 32 positions
// tile * 1024 + i * 32 + t (i = 0..31), so load / store instruction i of the warp covers 256 contiguous bytes
__global__ void __launch_bounds__(kThreads, 1) k1_find_correct_moves_bs(const u64* __restrict__ own, const u64* __restrict__ enemy,
                                                                        u64* __restrict__ out, size_t n_tiles) {
    const int lane = threadIdx.x & 31;
    const size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t t = warp; t < n_tiles; t += n_warps) {
        const size_t base = t * 1024 + lane;
        u64 o[32], e[32], m[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) { o[i] = ldg_stream_u64(own + base + i * 32); e[i] = ldg_stream_u64(enemy + base + i * 32); }
        bs::find_correct_moves32(o, e, m);
#pragma unroll
        for (int i = 0; i < 32; ++i) stg_stream_u64(out + base + i * 32, m[i]);
    }
}

__global__ void __launch_bounds__(kThreads, 1) k1_calc_flip_bs(const uint8_t* __restrict__ pos, const u64* __restrict__ own,
                                                               const u64* __restrict__ enemy, u64* __restrict__ out, size_t n_tiles) {
    const int lane = threadIdx.x & 31;
    const size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t t = warp; t < n_tiles; t += n_warps) {
        const size_t base = t * 1024 + lane;
        u64 o[32], e[32], f[32];
        uint8_t ps[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            o[i] = ldg_stream_u64(own + base + i * 32); e[i] = ldg_stream_u64(enemy + base + i * 32);
            ps[i] = __ldg(pos + base + i * 32);
        }
        if (bs::any_overlap32(o, e)) {      // see k1_bs_staged
            for (int i = 0; i < 32; ++i) out[base + i * 32] = calc_flip(pos[base + i * 32] & 63, own[base + i * 32], enemy[base + i * 32]);
            continue;
        }
        bs::calc_flip32<false>(ps, o, e, f);
#pragma unroll
        for (int i = 0; i < 32; ++i) stg_stream_u64(out + base + i * 32, f[i]);
    }
}

// The same operators with the inputs staged through shared memory: a tile of 1024 positions is 8 KB contiguous in each
// input array, so one lane fetches it with one cp.async.bulk per array (completion on the warp's own mbarrier); as soon as the
// warp has moved a tile from shared memory into registers it starts the copy of its NEXT tile, which lands while the ~2100
// logic instructions of the current one execute.  The register-only kernels above cannot overlap the two phases (their 231-255
// registers leave two warps per scheduler and no room for a second set of inputs) and stop at ~0.5 of the HBM roofline.
constexpr uint32_t kStagePerWarp = 2 * 8192 + 1024;   // own, enemy, pos
constexpr uint32_t kStagedSmem = (kThreads / 32) * kStagePerWarp + 64 + 128;

template <bool FLIP>
__global__ void __launch_bounds__(kThreads, 1) k1_bs_staged(const uint8_t* __restrict__ pos, const u64* __restrict__ own,
                                                            const u64* __restrict__ enemy, u64* __restrict__ out, size_t n_tiles) {
    extern __shared__ uint8_t k1_smem_raw[];
    const uint32_t base = (ptx::smem_u32(k1_smem_raw) + 127u) & ~127u;
    uint8_t* sm = k1_smem_raw + (base - ptx::smem_u32(k1_smem_raw));
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((size_t)gridDim.x * blockDim.x) >> 5;
    const uint32_t bar = base + (kThreads / 32) * kStagePerWarp + w * 8;
    const uint32_t s_own = base + w * kStagePerWarp, s_en = s_own + 8192, s_pos = s_own + 16384;
    const u64* so = reinterpret_cast<const u64*>(sm + w * kStagePerWarp);
    const u64* se = so + 1024;
    const uint8_t* sp = sm + w * kStagePerWarp + 16384;
    if (lane == 0) {
        ptx::mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    auto fetch = [&](size_t t) {   // lane 0 only
        ptx::mbar_expect_tx(bar, FLIP ? 16384u + 1024u : 16384u);
        ptx::bulk_g2s(s_own, own + t * 1024, 8192, bar);
        ptx::bulk_g2s(s_en, enemy + t * 1024, 8192, bar);
        if (FLIP) ptx::bulk_g2s(s_pos, pos + t * 1024, 1024, bar);
    };
    uint32_t phase = 0;
    if (warp < n_tiles && lane == 0) fetch(warp);
    for (size_t t = warp; t < n_tiles; t += n_warps) {
        u64 o[32], e[32], r[32];
        uint8_t ps[32];
        ptx::mbar_wait(bar, phase);
        phase ^= 1;
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            o[i] = so[i * 32 + lane]; e[i] = se[i * 32 + lane];
            if (FLIP) ps[i] = sp[i * 32 + lane];
        }
        const size_t ob = t * 1024 + lane;
        // flips: a thread whose 32 positions include one with a square shared by own and enemy (not a board, but the reference's
        // arithmetic defines the answer) computes them with the scalar code, straight from the staging buffer
        const bool scalar_path = FLIP && bs::any_overlap32(o, e);
        if (scalar_path)
            for (int i = 0; i < 32; ++i) out[ob + i * 32] = calc_flip(sp[i * 32 + lane] & 63, so[i * 32 + lane], se[i * 32 + lane]);
        __syncwarp();                       // every lane is done with the staging buffer: it may be refilled
        if (lane == 0 && t + n_warps < n_tiles) {
            ptx::fence_proxy_async();
            fetch(t + n_warps);
        }
        if (scalar_path) continue;
        if (FLIP) bs::calc_flip32<false>(ps, o, e, r); else bs::find_correct_moves32(o, e, r);
#pragma unroll
        for (int i = 0; i < 32; ++i) stg_stream_u64(out + ob + i * 32, r[i]);
    }
}

// RZ_K1_IMPL: "scalar", "bitsliced" (register-only), "staged" (bit-sliced + shared-memory staging); default per operator below
static int k1_impl() {
    static int v = -1;
    if (v < 0) {
        const char* s = getenv("RZ_K1_IMPL");
        v = !s ? 3 : (strcmp(s, "scalar") == 0 ? 0 : (strcmp(s, "bitsliced") == 0 ? 1 : (strcmp(s, "staged") == 0 ? 2 : 3)));
    }
    return v;
}
static int k1_staged_attr() {
    static bool done = false;
    if (!done) {
        RZ_CUDA_TRY(cudaFuncSetAttribute(k1_bs_staged<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kStagedSmem));
        RZ_CUDA_TRY(cudaFuncSetAttribute(k1_bs_staged<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kStagedSmem));
        done = true;
    }
    return RZ_OK;
}
static int grid_for_tiles(size_t tiles) {
    const size_t per_cta = kThreads / 32;
    size_t blocks = (tiles + per_cta - 1) / per_cta;
    if (blocks > (size_t)num_sms()) blocks = (size_t)num_sms();   // one CTA of 256 threads x ~240 registers per SM
    return (int)(blocks < 1 ? 1 : blocks);
}

__global__ void __launch_bounds__(kThreads) k1_find_correct_moves(const u64* __restrict__ own, const u64* __restrict__ enemy,
                                                                  u64* __restrict__ out, size_t n, int vec_ok) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (vec_ok) {
        const size_t pairs = n >> 1;
        for (size_t i = tid; i < pairs; i += stride) {
            ulonglong2 o = ldg_stream_u64x2(own + 2 * i), e = ldg_stream_u64x2(enemy + 2 * i);
            stg_stream_u64x2(out + 2 * i, find_correct_moves(o.x, e.x), find_correct_moves(o.y, e.y));
        }
        if ((n & 1) && tid == 0) out[n - 1] = find_correct_moves(own[n - 1], enemy[n - 1]);
    } else {
        for (size_t i = tid; i < n; i += stride) out[i] = find_correct_moves(ldg_stream_u64(own + i), ldg_stream_u64(enemy + i));
    }
}

__global__ void __launch_bounds__(kThreads) k1_calc_flip(const uint8_t* __restrict__ pos, const u64* __restrict__ own,
                                                         const u64* __restrict__ enemy, u64* __restrict__ out, size_t n,
                                                         int vec_ok) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (vec_ok) {
        const size_t pairs = n >> 1;
        for (size_t i = tid; i < pairs; i += stride) {
            ulonglong2 o = ldg_stream_u64x2(own + 2 * i), e = ldg_stream_u64x2(enemy + 2 * i);
            const uchar2 p = *reinterpret_cast<const uchar2*>(pos + 2 * i);
            stg_stream_u64x2(out + 2 * i, calc_flip(p.x & 63, o.x, e.x), calc_flip(p.y & 63, o.y, e.y));
        }
        if ((n & 1) && tid == 0) out[n - 1] = calc_flip(pos[n - 1] & 63, own[n - 1], enemy[n - 1]);
    } else {
        for (size_t i = tid; i < n; i += stride) out[i] = calc_flip(pos[i] & 63, own[i], enemy[i]);
    }
}

__global__ void __launch_bounds__(kThreads) k1_step(u64* __restrict__ black, u64* __restrict__ white, uint8_t* __restrict__ next_player,
                                                    uint8_t* __restrict__ turn, uint8_t* __restrict__ done, uint8_t* __restrict__ winner,
                                                    const int8_t* __restrict__ action, u64* __restrict__ legal_out, size_t n) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        EnvState s{black[i], white[i], next_player[i], turn[i], done[i], winner[i]};
        u64 legal = env_step(s, action[i]);
        black[i] = s.black; white[i] = s.white; next_player[i] = s.next_player;
        turn[i] = s.turn; done[i] = s.done; winner[i] = s.winner;
        if (legal_out) legal_out[i] = legal;
    }
}

__global__ void __launch_bounds__(kThreads) k1_dihedral(const u64* __restrict__ x, const uint8_t* __restrict__ t, u64* __restrict__ out, size_t n) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = dihedral(x[i], t[i] & 7);
}

static int grid_for(size_t work_items) {
    const int sms = num_sms();
    size_t blocks = (work_items + kThreads - 1) / kThreads;
    size_t cap = (size_t)sms * 8;  // 8 resident CTAs of 256 threads per SM
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// Scratch device buffers for the host-pointer variants (grown on demand, per thread).
struct Scratch {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return RZ_OK;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        if (cudaMalloc(&p, bytes) != cudaSuccess) { set_error("cudaMalloc(%zu) failed", bytes); cudaGetLastError(); return RZ_ENOMEM; }
        cap = bytes;
        return RZ_OK;
    }
};
static thread_local Scratch g_scratch;

}  // namespace rz

using namespace rz;

extern "C" {

int rz_find_correct_moves_dev(const uint64_t* own, const uint64_t* enemy, uint64_t* out, size_t n, void* stream) {
    RZ_REQUIRE(n == 0 || (own && enemy && out), "rz_find_correct_moves_dev: null pointer");
    if (n == 0) return RZ_OK;
    const int impl = k1_impl() == 3 ? 2 : k1_impl();   // default: bit-sliced with staging
    if (impl != 0 && n >= 1024) {  // whole tiles of 1024 positions bit-sliced, the rest below
        const size_t tiles = n / 1024;
        if (impl == 2 && aligned16(own) && aligned16(enemy)) {
            RZ_TRY(k1_staged_attr());
            k1_bs_staged<false><<<grid_for_tiles(tiles), kThreads, kStagedSmem, (cudaStream_t)stream>>>(nullptr, own, enemy, out, tiles);
        } else {
            k1_find_correct_moves_bs<<<grid_for_tiles(tiles), kThreads, 0, (cudaStream_t)stream>>>(own, enemy, out, tiles);
        }
        RZ_LAUNCH_CHECK();
        own += tiles * 1024; enemy += tiles * 1024; out += tiles * 1024; n -= tiles * 1024;
        if (n == 0) return RZ_OK;
    }
    const int vec = aligned16(own) && aligned16(enemy) && aligned16(out);
    k1_find_correct_moves<<<grid_for(vec ? (n + 1) / 2 : n), kThreads, 0, (cudaStream_t)stream>>>(own, enemy, out, n, vec);
    RZ_LAUNCH_CHECK();
    return RZ_OK;
}

int rz_calc_flip_dev(const uint8_t* pos, const uint64_t* own, const uint64_t* enemy, uint64_t* out, size_t n, void* stream) {
    RZ_REQUIRE(n == 0 || (pos && own && enemy && out), "rz_calc_flip_dev: null pointer");
    if (n == 0) return RZ_OK;
    const int impl = k1_impl() == 3 ? 2 : k1_impl();
    if (impl != 0 && n >= 1024) {
        const size_t tiles = n / 1024;
        if (impl == 2 && aligned16(own) && aligned16(enemy) && aligned16(pos)) {
            RZ_TRY(k1_staged_attr());
            k1_bs_staged<true><<<grid_for_tiles(tiles), kThreads, kStagedSmem, (cudaStream_t)stream>>>(pos, own, enemy, out, tiles);
        } else {
            k1_calc_flip_bs<<<grid_for_tiles(tiles), kThreads, 0, (cudaStream_t)stream>>>(pos, own, enemy, out, tiles);
        }
        RZ_LAUNCH_CHECK();
        pos += tiles * 1024; own += tiles * 1024; enemy += tiles * 1024; out += tiles * 1024; n -= tiles * 1024;
        if (n == 0) return RZ_OK;
    }
    const int vec = aligned16(own) && aligned16(enemy) && aligned16(out) && ((reinterpret_cast<uintptr_t>(pos) & 1) == 0);
    k1_calc_flip<<<grid_for(vec ? (n + 1) / 2 : n), kThreads, 0, (cudaStream_t)stream>>>(pos, own, enemy, out, n, vec);
    RZ_LAUNCH_CHECK();
    return RZ_OK;
}

int rz_step_dev(uint64_t* black, uint64_t* white, uint8_t* next_player, uint8_t* turn, uint8_t* done, uint8_t* winner,
                const int8_t* action, uint64_t* legal_out, size_t n, void* stream) {
    RZ_REQUIRE(n == 0 || (black && white && next_player && turn && done && winner && action), "rz_step_dev: null pointer");
    if (n == 0) return RZ_OK;
    k1_step<<<grid_for(n), kThreads, 0, (cudaStream_t)stream>>>(black, white, next_player, turn, done, winner, action, legal_out, n);
    RZ_LAUNCH_CHECK();
    return RZ_OK;
}

int rz_dihedral_dev(const uint64_t* x, const uint8_t* t, uint64_t* out, size_t n, void* stream) {
    RZ_REQUIRE(n == 0 || (x && t && out), "rz_dihedral_dev: null pointer");
    if (n == 0) return RZ_OK;
    k1_dihedral<<<grid_for(n), kThreads, 0, (cudaStream_t)stream>>>(x, t, out, n);
    RZ_LAUNCH_CHECK();
    return RZ_OK;
}

// ---- host-buffer variants: H2D, kernel, D2H on the default stream --------------------------------
int rz_find_correct_moves(const uint64_t* own, const uint64_t* enemy, uint64_t* out, size_t n) {
    RZ_REQUIRE(n == 0 || (own && enemy && out), "rz_find_correct_moves: null pointer");
    if (n == 0) return RZ_OK;
    const size_t b = ((n * 8 + 255) / 256) * 256;
    RZ_TRY(g_scratch.ensure(3 * b));
    char* d = (char*)g_scratch.p;
    RZ_CUDA_TRY(cudaMemcpyAsync(d, own, n * 8, cudaMemcpyHostToDevice, 0));
    RZ_CUDA_TRY(cudaMemcpyAsync(d + b, enemy, n * 8, cudaMemcpyHostToDevice, 0));
    RZ_TRY(rz_find_correct_moves_dev((u64*)d, (u64*)(d + b), (u64*)(d + 2 * b), n, 0));
    RZ_CUDA_TRY(cudaMemcpyAsync(out, d + 2 * b, n * 8, cudaMemcpyDeviceToHost, 0));
    RZ_CUDA_TRY(cudaStreamSynchronize(0));
    return RZ_OK;
}

int rz_calc_flip(const uint8_t* pos, const uint64_t* own, const uint64_t* enemy, uint64_t* out, size_t n) {
    RZ_REQUIRE(n == 0 || (pos && own && enemy && out), "rz_calc_flip: null pointer");
    if (n == 0) return RZ_OK;
    const size_t b = ((n * 8 + 255) / 256) * 256;
    RZ_TRY(g_scratch.ensure(4 * b));
    char* d = (char*)g_scratch.p;
    RZ_CUDA_TRY(cudaMemcpyAsync(d, own, n * 8, cudaMemcpyHostToDevice, 0));
    RZ_CUDA_TRY(cudaMemcpyAsync(d + b, enemy, n * 8, cudaMemcpyHostToDevice, 0));
    RZ_CUDA_TRY(cudaMemcpyAsync(d + 3 * b, pos, n, cudaMemcpyHostToDevice, 0));
    RZ_TRY(rz_calc_flip_dev((uint8_t*)(d + 3 * b), (u64*)d, (u64*)(d + b), (u64*)(d + 2 * b), n, 0));
    RZ_CUDA_TRY(cudaMemcpyAsync(out, d + 2 * b, n * 8, cudaMemcpyDeviceToHost, 0));
    RZ_CUDA_TRY(cudaStreamSynchronize(0));
    return RZ_OK;
}

int rz_step(uint64_t* black, uint64_t* white, uint8_t* next_player, uint8_t* turn, uint8_t* done, uint8_t* winner,
            const int8_t* action, uint64_t* legal_out, size_t n) {
    RZ_REQUIRE(n == 0 || (black && white && next_player && turn && done && winner && action), "rz_step: null pointer");
    if (n == 0) return RZ_OK;
    const size_t b = ((n * 8 + 255) / 256) * 256;
    RZ_TRY(g_scratch.ensure(8 * b));
    char* d = (char*)g_scratch.p;
    u64 *dB = (u64*)d, *dW = (u64*)(d + b), *dL = (u64*)(d + 2 * b);
    uint8_t *dP = (uint8_t*)(d + 3 * b), *dT = (uint8_t*)(d + 4 * b), *dD = (uint8_t*)(d + 5 * b), *dWn = (uint8_t*)(d + 6 * b);
    int8_t* dA = (int8_t*)(d + 7 * b);
    RZ_CUDA_TRY(cudaMemcpyAsync(dB, black, n * 8, cudaMemcpyHostToDevice, 0));
    RZ_CUDA_TRY(cudaMemcpyAsync(dW, white, n * 8, cudaMemcpyHostToDevice, 0));
    RZ_CUDA_TRY(cudaMemcpyAsync(dP, next_player, n, cudaMemcpyHostToDevice, 0));
    RZ_CUDA_TRY(cudaMemcpyAsync(dT, turn, n, cudaMemcpyHostToDevice, 0));
    RZ_CUDA_TRY(cudaMemcpyAsync(dD, done, n, cudaMemcpyHostToDevice, 0));
    RZ_CUDA_TRY(cudaMemcpyAsync(dWn, winner, n, cudaMemcpyHostToDevice, 0));
    RZ_CUDA_TRY(cudaMemcpyAsync(dA, action, n, cudaMemcpyHostToDevice, 0));
    RZ_TRY(rz_step_dev(dB, dW, dP, dT, dD, dWn, dA, legal_out ? dL : nullptr, n, 0));
    RZ_CUDA_TRY(cudaMemcpyAsync(black, dB, n * 8, cudaMemcpyDeviceToHost, 0));
    RZ_CUDA_TRY(cudaMemcpyAsync(white, dW, n * 8, cudaMemcpyDeviceToHost, 0));
    RZ_CUDA_TRY(cudaMemcpyAsync(next_player, dP, n, cudaMemcpyDeviceToHost, 0));
    RZ_CUDA_TRY(cudaMemcpyAsync(turn, dT, n, cudaMemcpyDeviceToHost, 0));
    RZ_CUDA_TRY(cudaMemcpyAsync(done, dD, n, cudaMemcpyDeviceToHost, 0));
    RZ_CUDA_TRY(cudaMemcpyAsync(winner, dWn, n, cudaMemcpyDeviceToHost, 0));
    if (legal_out) RZ_CUDA_TRY(cudaMemcpyAsync(legal_out, dL, n * 8, cudaMemcpyDeviceToHost, 0));
    RZ_CUDA_TRY(cudaStreamSynchronize(0));
    return RZ_OK;
}

// ---- scalar host twins (single-environment Python objects) ---------------------------------------
uint64_t rz_find_correct_moves_host(uint64_t own, uint64_t enemy) { return find_correct_moves(own, enemy); }
uint64_t rz_calc_flip_host(int pos, uint64_t own, uint64_t enemy) { return calc_flip(pos & 63, own, enemy); }

// host twins of the bit-sliced operators (the same header compiled for the host, groups of 32 consecutive positions): they let
// the CPU test suite hold the formulation the GPU kernels use against the oracle.  pos may be NULL for the legal-move variant.
int rz_bitsliced_host(const uint8_t* pos, const uint64_t* own, const uint64_t* enemy, uint64_t* out, size_t n) {
    RZ_REQUIRE(n == 0 || (own && enemy && out), "rz_bitsliced_host: null pointer");
    for (size_t at = 0; at < n; at += 32) {
        u64 o[32], e[32], r[32];
        uint8_t ps[32];
        const size_t m = n - at < 32 ? n - at : 32;
        for (size_t i = 0; i < 32; ++i) {
            o[i] = i < m ? own[at + i] : 0; e[i] = i < m ? enemy[at + i] : 0; ps[i] = (pos && i < m) ? pos[at + i] : 0;
        }
        if (pos) bs::calc_flip32(ps, o, e, r); else bs::find_correct_moves32(o, e, r);
        for (size_t i = 0; i < m; ++i) out[at + i] = r[i];
    }
    return RZ_OK;
}
uint64_t rz_dihedral_host(uint64_t x, int t) { return dihedral(x, t & 7); }
void rz_env_reset_host(rz_env_state* s) {
    EnvState e; env_reset(e);
    s->black = e.black; s->white = e.white; s->next_player = e.next_player; s->turn = e.turn; s->done = e.done; s->winner = e.winner;
}
void rz_env_update_host(rz_env_state* s, uint64_t black, uint64_t white, int next_player) {
    EnvState e; env_update(e, black, white, next_player);
    s->black = e.black; s->white = e.white; s->next_player = e.next_player; s->turn = e.turn; s->done = e.done; s->winner = e.winner;
}
void rz_env_step_host(rz_env_state* s, int action) {
    EnvState e{s->black, s->white, s->next_player, s->turn, s->done, s->winner};
    env_step(e, action);
    s->black = e.black; s->white = e.white; s->next_player = e.next_player; s->turn = e.turn; s->done = e.done; s->winner = e.winner;
}

}  // extern "C"
