// rz_net_tc.cu -- K4/K5: fused persistent tcgen05 residual tower + heads for the 256-filter network, run on CTA PAIRS
// (cta_group::2) with the epilogue overlapped with the MMA stream.
//
// Every CTA owns a tile of TWO boards (M = 128 pixel rows) and carries it through the WHOLE network without touching HBM
// in between; the two CTAs of a cluster compute their tiles with shared MMAs:
//   * activations live in shared memory as fp16 in the UMMA "K-major, no-swizzle" canonical layout, with a one-pixel zero
//     border, so that each of the nine 3x3 taps is just a different start address of the same buffer (implicit GEMM, no
//     im2col copy):
//         chunk(cg, slot, xp) at cg*2896 + slot*144 + xp*16 bytes   (8 channels = 16 B per chunk)
//         slot = 2*(y+1) + board (the two boards' rows are interleaved so that a dy shift is a uniform 2-slot offset),
//         xp = x+1; xp = 9 of one slot aliases xp = 0 of the next (shared zero chunk).  MMA row m = (2y+board)*8 + x  ->
//         8-row core matrices are board rows.
//   * weights (fp16, 1.18 MB per conv, L2-resident) are streamed by a producer thread with cp.async.bulk in pre-packed
//     16 KB stages per CTA (one tap x 128 input channels x this CTA's 64 of the 128 output channels of an MMA) through a
//     4-deep mbarrier ring;
//   * one thread of the leader CTA issues tcgen05.mma.cta_group::2 with M = 256 (the pair's 2 x 128 rows) and N = 128,
//     each CTA supplying its own A rows and HALF of B, into TMEM accumulators of 2 x 128 columns;
//   * eight epilogue warps per CTA read the accumulator with tcgen05.ld, apply the folded BatchNorm (scale, shift), the
//     skip connection (the fp32 residual stream in the other 256 TMEM columns) and ReLU, and write the next layer's fp16
//     operand straight back into shared memory;
//   * the first conv (2 -> 256 channels, K = 18 padded to 32) is a 2-MMA GEMM per output half on an im2col tile built
//     from the two bitboards; the policy / value heads run on the epilogue warps from the fp32 tower output.
// Why N = 128 halves: with a single 256-column accumulator, MMA(l + 1) cannot start before epilogue(l) has written the
// whole next operand, and the tensor pipe idles for every epilogue (MMA stream alone 28.5 ms of 36.6 ms per 32 768
// positions, profiles/tower_experiments_r02.jsonl).  Here a layer is computed as two output halves (nh = 0, 1: accumulator
// columns 0-127 and 128-255).  While the tensor pipe works on half 1, the epilogue warps drain half 0 and write the first
// 128 channels of the next layer's operand; the next layer's MMAs run their K loop over input channels 0-127 FIRST (all
// nine taps), which only needs what the half-0 epilogue wrote, so they start while the half-1 epilogue is still running,
// and switch to channels 128-255 when that one signals.  The tensor pipe never waits for an epilogue as long as an
// epilogue half takes less than a quarter of a layer's MMAs (it takes about an eighth): 30.9 ms per 32 768 positions
// (profiles/tower_v2_check_r02.log), tensor pipe active 92.7 % of elapsed (profiles/tower_r02_ncu_summary.txt).  Splitting
// B across the pair keeps the shared-memory read rate per MMA cycle at what N = 256 on one CTA needs.
// Operands therefore live in three half-buffers of 128 channels (46 KB each): channels 128-255 are rewritten in place
// (their last reader, this layer's half-1 MMAs, has completed when the half-1 epilogue starts), channels 0-127 alternate
// between two buffers (the half-0 epilogue writes while this layer's half-1 MMAs still read the old ones).
// Barriers that gate the leader's MMA thread (operand halves written, layer-0 operand built, weight stages landed) collect
// the arrivals of BOTH CTAs: the peer's threads arrive remotely (mapa + mbarrier.arrive); tcgen05.commit multicasts
// "stage free" / "accumulator half ready" to both CTAs.
// HBM traffic per position: 16 B in, 260 B out.  Algorithmic work: 2 * 755,343,616 flop (SURVEY 3.2).
#include "rz_bitboard.cuh"
#include "rz_net.cuh"
#include "rz_ptx.cuh"

namespace rz {
namespace tc {

using namespace rz::ptx;

// ---- PTX wrappers only the tower uses --------------------------------------------------------------------------------
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
          "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
          "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
        "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
        "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]),
        "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]),
        "r"(v[31])
        : "memory");
}
// wait::ld that also carries a register dependency on the loaded values, so the compiler cannot schedule a use of
// v[] above the wait (tcgen05.ld completes asynchronously)
__device__ __forceinline__ void tmem_wait_ld_dep(uint32_t (&v)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]), "+r"(v[9]),
                   "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]), "+r"(v[16]), "+r"(v[17]), "+r"(v[18]),
                   "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]), "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]),
                   "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
                 :
                 : "memory");
}
__device__ __forceinline__ void tmem_dep(uint32_t (&v)[32]) {
    asm volatile(""
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]), "+r"(v[9]),
                   "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]), "+r"(v[16]), "+r"(v[17]), "+r"(v[18]),
                   "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]), "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]),
                   "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
                 :
                 : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// two fp32 -> packed fp16x2 (a in the low half), saturating at +-65504; RELU folds max(x, 0) into the convert
template <bool RELU>
__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
    uint32_t d;
    if (RELU) asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(b), "f"(a));
    else      asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(b), "f"(a));
    return d;
}

// tcgen05.mma.cta_group::2 with the descriptors as (low, high) words: the issue loop keeps the high words (LBO / SBO / layout
// bits) constant and only ADDS to the start-address field of the low words -- with N = 128 an MMA lasts 64 cycles, so the
// dozen uniform instructions the compiler spends on rebuilding a descriptor from an address (add, shift, mask, or, twice)
// would make the issuing thread, not the tensor pipe, the bottleneck.
// warp-convergent variants: executed by all 32 lanes of the MMA warp, one elected lane issues.  (Issued from a divergent
// `if (lane == 0)` region the compiler wraps every tcgen05 instruction in an ELECT / branch loop of its own.  Convergent
// issue and the low-word descriptor adds together took a launch from 40.1 to 30.9 ms, DESIGN.md section 5.)
__device__ __forceinline__ void umma2_f16_elect(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                                uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t.reg .b64 da, db;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "mov.b64 da, {%1, %2};\n\t"
        "mov.b64 db, {%3, %4};\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "@q tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %5, p;\n\t}" ::"r"(d_tmem),
        "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma2_commit_elect(uint32_t bar) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n\t}" ::"r"(bar),
        "h"((uint16_t)3)
        : "memory");
}
// shared-memory matrix descriptor, K-major, SWIZZLE_NONE (core matrix = 8 rows x 16 B, rows 16 B apart), as its two words:
// low = start address | LBO (byte distance between the two K-halves of one MMA), high = SBO (between 8-row groups) | version
__device__ __forceinline__ uint32_t desc_lo(uint32_t addr, uint32_t lbo) { return ((addr >> 4) & 0x3FFFu) | (((lbo >> 4) & 0x3FFFu) << 16); }
__device__ __forceinline__ uint32_t desc_hi(uint32_t sbo) { return ((sbo >> 4) & 0x3FFFu) | (1u << 14); }
// non-blocking test of a barrier phase
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
// arrive on the barrier at the same offset in CTA `rank` of the cluster.  Plain (default-semantics) arrive and wait, as the
// 2-SM GEMM pipelines use them: .release.cluster arrives with .acquire.cluster waits are correct too, but the MMA thread
// then spends ~0.5 us per weight stage in the cluster-scope acquire (100 ms per launch,
// profiles/tower_v2_first_version_r02.log).
__device__ __forceinline__ void mbar_arrive_cta(uint32_t bar, uint32_t rank) {
    uint32_t remote;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(bar), "r"(rank));
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}

struct Params {
    const __half* w0;   // layer-0 weight image (16 KB)
    const __half* w;    // tower weight stages
    const float* ss;    // folded BN [L][2][256], then heads
    const float* blob;  // fp32 blob for the head weights
    size_t off_policy_conv, off_policy_fc_k, off_policy_fc_b, off_value_conv, off_value_fc1_k, off_value_fc1_b, off_value_fc2_k,
        off_value_fc2_b;
    const u64* own;
    const u64* enemy;
    float* policy;
    float* value;
    float* dbg_tower;  // nullable
    float* dbg_logits; // nullable: [n][64] policy logits (before the softmax)
    float* dbg_vlogit; // nullable: [n] value before the tanh
    uint32_t n;
    const uint32_t* n_dev;  // nullable: batch size produced on the device (engine waves)
    int n_layers;  // 1 + 2R
    int V;
};

// ---- shared-memory layout ------------------------------------------------------------------------------------------
constexpr int kThreads = 320;  // warp 0 weight producer, warp 1 MMA issuer (leader) / stage relay (peer) + TMEM owner, warps 2..9 epilogue
constexpr int kEpiThreads = 256;
constexpr uint32_t kActCg = 2896, kActSlot = 144;  // byte distance between channel groups of 8 / between board-row slots
constexpr uint32_t kHalfBytes = 16 * kActCg;  // 46,336: 128 channels of the operand
constexpr uint32_t kStageBytes = 16384;               // per CTA: one tap x 128 input channels x 64 of the 128 output channels
constexpr uint32_t kStages = 4;                       // weight ring depth; the ring sits last
// full / empty barrier pairs reserved in the barrier block, kStages of them used: eight is the layout this kernel was
// measured with (profiles/tower_r02_*); a smaller block moves the weight ring and with it the kernel's shared-memory offsets
constexpr uint32_t kBarSlots = 8;
constexpr uint32_t kStagesPerLayer = 36;              // 2 output halves x 2 input halves x 9 taps
// Why 16 KB stages of eight MMAs: with 8 KB stages of four MMAs the issuing thread spends longer on a stage's barrier wait
// + commit than the tensor pipe on its four 64-cycle MMAs (50 ms per launch, 25 ms with the waits removed), and 8 x 8 KB
// ring slots with their own barriers measured 34.5 ms against 31.6 ms for 4 x 16 KB (3 x 16 KB: 33.3 ms;
// profiles/tower_v2_experiments_r02.log).  The next stage's barrier is tested before a stage's MMAs are issued.
constexpr uint32_t kA0Bytes = 8192, kW0Bytes = 8192;
constexpr uint32_t kOffAct = 0;                       // half-buffers A (0), B (1), C (2)
constexpr uint32_t kOffW0 = kOffAct + 3 * kHalfBytes;
constexpr uint32_t kOffSS = kOffW0 + kW0Bytes;           // 2 x [scale 256][shift 256] fp32
// the layer-0 operand (8 KB, live from a tile's first instruction to its layer-0 MMAs) shares its bytes with the head
// scratch (live during a tile's last phase): that buys the fourth weight stage
constexpr uint32_t kOffA0 = kOffSS + 2 * 2048;
constexpr uint32_t kOffPart = kOffA0;                    // [2 column sub-halves][128 rows][4] fp32 head partial sums
constexpr uint32_t kOffHp = kOffPart + 2 * 128 * 4 * 4;  // [2 boards][128]
constexpr uint32_t kOffHv = kOffHp + 2 * 128 * 4;        // [2][64]
constexpr uint32_t kOffLogit = kOffHv + 2 * 64 * 4;      // [2][64]
constexpr uint32_t kMaxV = 512;
constexpr uint32_t kOffFc1 = kOffLogit + 2 * 64 * 4;     // [2][kMaxV]
constexpr uint32_t kOffBar = kOffFc1 + 2 * kMaxV * 4;    // mbarriers
constexpr uint32_t kNumBars = 2 * kBarSlots + 6;         // full, empty, w0, a0, x[2], acc[2]
constexpr uint32_t kOffTmemPtr = kOffBar + kNumBars * 8;
constexpr uint32_t kOffW = (kOffTmemPtr + 16 + 127) & ~127u;   // weight ring
constexpr uint32_t kSmemAlloc = kOffW + kStages * kStageBytes + 128;  // + slack for manual 128 B alignment
static_assert(kSmemAlloc <= 232448, "shared memory budget exceeded");
static_assert(kOffFc1 + 2 * kMaxV * 4 - kOffA0 >= kA0Bytes, "head scratch must cover the layer-0 operand");

// instruction descriptor, kind::f16: D = f32, A = B = f16, K-major both, N = 128, M = 256 (cta_group::2)
constexpr uint32_t kIdesc = (1u << 4) | ((128u >> 3) << 17) | ((256u >> 4) << 24);

// ---- epilogue pieces -----------------------------------------------------------------------------------------------
// layer-0 operand (agent/model.py:30-33 first convolution as a GEMM): im2col of the two bit planes of one board row m =
// (g, x), K index = tap * 2 + plane padded to 32, two of the four 8-wide K chunks (kc0, kc0 + 1) per calling thread;
// a0 = the [4 kc][16 g][8 x][8] fp16 tile in shared memory
__device__ __forceinline__ void build_layer0_operand(uint8_t* a0, u64 o, u64 e, int kc0, int g, int x, int y) {
#pragma unroll
    for (int kk = 0; kk < 2; ++kk) {
        const int kc = kc0 + kk;
        uint32_t w[4];
#pragma unroll
        for (int jp = 0; jp < 4; ++jp) {
            uint32_t packed = 0;
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int k = kc * 8 + jp * 2 + half;
                uint32_t bit = 0;
                if (k < 18) {
                    const int tap = k >> 1, yy = y + tap / 3 - 1, xx = x + tap % 3 - 1;
                    if (yy >= 0 && yy < 8 && xx >= 0 && xx < 8) bit = (uint32_t)((((k & 1) ? e : o) >> (yy * 8 + xx)) & 1ULL);
                }
                packed |= (bit ? 0x3C00u : 0u) << (16 * half);  // fp16 1.0
            }
            w[jp] = packed;
        }
        *reinterpret_cast<uint4*>(a0 + kc * 2048 + g * 128 + x * 16) = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

// folded BatchNorm (+ skip connection + ReLU) on 32 accumulator columns c0 .. c0 + 31 of one row; sc = [scale 256][shift 256].
// conv2: second convolution of a block (adds the fp32 residual r, ReLU); relu_now: block outputs / the last layer (ReLU here);
// otherwise the first convolution of a block, whose ReLU is folded into the fp16 convert of epi_store_operand
__device__ __forceinline__ void epi_math(uint32_t (&v)[32], const uint32_t (&r)[32], const float* sc, int c0, bool conv2, bool relu_now) {
    if (conv2) {
#pragma unroll
        for (int j = 0; j < 32; ++j)
            v[j] = __float_as_uint(fmaxf(fmaf(__uint_as_float(v[j]), sc[c0 + j], sc[256 + c0 + j]) + __uint_as_float(r[j]), 0.f));
    } else if (relu_now) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(fmaxf(fmaf(__uint_as_float(v[j]), sc[c0 + j], sc[256 + c0 + j]), 0.f));
    } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(fmaf(__uint_as_float(v[j]), sc[c0 + j], sc[256 + c0 + j]));
    }
}

// 32 fp32 values of one row -> fp16, four 16-byte chunks (8 channels each) at row_addr + (cg0 + jj) * kActCg
__device__ __forceinline__ void epi_store_operand(const uint32_t (&v)[32], uint32_t row_addr, int cg0, bool already_relu) {
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
        uint4 pk;
        if (already_relu) {
            pk.x = pack_h2<false>(__uint_as_float(v[jj * 8 + 0]), __uint_as_float(v[jj * 8 + 1]));
            pk.y = pack_h2<false>(__uint_as_float(v[jj * 8 + 2]), __uint_as_float(v[jj * 8 + 3]));
            pk.z = pack_h2<false>(__uint_as_float(v[jj * 8 + 4]), __uint_as_float(v[jj * 8 + 5]));
            pk.w = pack_h2<false>(__uint_as_float(v[jj * 8 + 6]), __uint_as_float(v[jj * 8 + 7]));
        } else {
            pk.x = pack_h2<true>(__uint_as_float(v[jj * 8 + 0]), __uint_as_float(v[jj * 8 + 1]));
            pk.y = pack_h2<true>(__uint_as_float(v[jj * 8 + 2]), __uint_as_float(v[jj * 8 + 3]));
            pk.z = pack_h2<true>(__uint_as_float(v[jj * 8 + 4]), __uint_as_float(v[jj * 8 + 5]));
            pk.w = pack_h2<true>(__uint_as_float(v[jj * 8 + 6]), __uint_as_float(v[jj * 8 + 7]));
        }
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(row_addr + (cg0 + jj) * kActCg), "r"(pk.x), "r"(pk.y), "r"(pk.z),
                     "r"(pk.w)
                     : "memory");
    }
}

// tower output columns c0 .. c0 + 31 of one row feed the 1x1 head convolutions from registers (policy: 2 filters, value: 1)
__device__ __forceinline__ void epi_head_partial(const uint32_t (&v)[32], int c0, const Params& p, float& hp0, float& hp1, float& hvv,
                                                 float* dbg_row /* nullable: this row's 256 tower outputs */) {
    const float* wp = p.blob + p.off_policy_conv;
    const float* wv = p.blob + p.off_value_conv;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
        const float a = __uint_as_float(v[j]);
        const float2 w2 = __ldg(reinterpret_cast<const float2*>(wp) + c0 + j);
        hp0 = fmaf(a, w2.x, hp0);
        hp1 = fmaf(a, w2.y, hp1);
        hvv = fmaf(a, __ldg(wv + c0 + j), hvv);
    }
    if (dbg_row) {
#pragma unroll
        for (int j = 0; j < 32; ++j) dbg_row[c0 + j] = __uint_as_float(v[j]);
    }
}

// heads (agent/model.py:43-56) on the 256 epilogue threads of a CTA for its two boards: the per-thread partial sums of the
// two column halves (colhalf 0 / 1 of row m) -> BN + ReLU -> Dense(128 -> 64) + softmax, Dense(64 -> V) + ReLU -> Dense(V -> 1)
// + tanh.  part [2][128][4], hp [2][128], hv [2][64], logit [2][64], fc1 [2][kMaxV]: shared-memory scratch.
__device__ __forceinline__ void heads_phase(const Params& p, float hp0, float hp1, float hvv, int colhalf, int m, int brd, int y, int x,
                                            int et, int ew, int lane, uint32_t pos0, float* part, float* hp, float* hv, float* logit,
                                            float* fc1) {
    const float* ssh = p.ss + (size_t)p.n_layers * 512;
    part[(colhalf * 128 + m) * 4 + 0] = hp0;
    part[(colhalf * 128 + m) * 4 + 1] = hp1;
    part[(colhalf * 128 + m) * 4 + 2] = hvv;
    epi_bar();
    if (colhalf == 0) {
        const float a0 = part[m * 4 + 0] + part[(128 + m) * 4 + 0];
        const float a1 = part[m * 4 + 1] + part[(128 + m) * 4 + 1];
        const float av = part[m * 4 + 2] + part[(128 + m) * 4 + 2];
        const int pix = y * 8 + x;
        hp[brd * 128 + pix] = fmaxf(fmaf(a0, ssh[0], ssh[2]), 0.f);        // Flatten is (C,H,W): index c*64 + pix
        hp[brd * 128 + 64 + pix] = fmaxf(fmaf(a1, ssh[1], ssh[3]), 0.f);
        hv[brd * 64 + pix] = fmaxf(fmaf(av, ssh[4], ssh[5]), 0.f);
    }
    epi_bar();
    if (et < 128) {  // policy logits: Dense(128 -> 64)
        const int b = et >> 6, j = et & 63;
        const float* k = p.blob + p.off_policy_fc_k;
        float acc = __ldg(p.blob + p.off_policy_fc_b + j);
#pragma unroll 8
        for (int i = 0; i < 128; ++i) acc = fmaf(hp[b * 128 + i], __ldg(k + i * 64 + j), acc);
        logit[b * 64 + j] = acc;
    }
    for (int idx = et; idx < 2 * p.V; idx += 256) {  // value Dense(64 -> V) + ReLU
        const int b = idx / p.V, j = idx - b * p.V;
        const float* k = p.blob + p.off_value_fc1_k;
        float acc = __ldg(p.blob + p.off_value_fc1_b + j);
#pragma unroll 8
        for (int i = 0; i < 64; ++i) acc = fmaf(hv[b * 64 + i], __ldg(k + (size_t)i * p.V + j), acc);
        fc1[b * kMaxV + j] = fmaxf(acc, 0.f);
    }
    epi_bar();
    if (ew < 2) {  // softmax over 64 logits, one warp per board
        const int b = ew;
        const float l0 = logit[b * 64 + lane], l1 = logit[b * 64 + 32 + lane];
        float mx = fmaxf(l0, l1);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        const float e0 = expf(l0 - mx), e1 = expf(l1 - mx);
        float s = e0 + e1;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (pos0 + b < p.n) {
            p.policy[(size_t)(pos0 + b) * 64 + lane] = e0 / s;
            p.policy[(size_t)(pos0 + b) * 64 + 32 + lane] = e1 / s;
            if (p.dbg_logits) {
                p.dbg_logits[(size_t)(pos0 + b) * 64 + lane] = l0;
                p.dbg_logits[(size_t)(pos0 + b) * 64 + 32 + lane] = l1;
            }
        }
    } else if (ew < 4) {  // value Dense(V -> 1) + tanh, one warp per board
        const int b = ew - 2;
        float acc = 0.f;
        for (int j = lane; j < p.V; j += 32) acc = fmaf(fc1[b * kMaxV + j], __ldg(p.blob + p.off_value_fc2_k + j), acc);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0 && pos0 + b < p.n) {
            const float pre = acc + __ldg(p.blob + p.off_value_fc2_b);
            p.value[pos0 + b] = tanhf(pre);
            if (p.dbg_vlogit) p.dbg_vlogit[pos0 + b] = pre;
        }
    }
}

// ---- the kernel ----------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads, 1) net_tower_pair_kernel(const Params pp) {
    Params p = pp;
    if (p.n_dev) p.n = *p.n_dev;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 127u) & ~127u;
    uint8_t* sm = smem_raw + (base - smem_u32(smem_raw));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t bar0 = base + kOffBar;
    auto bar_full = [&](uint32_t s) { return bar0 + s * 8; };
    auto bar_empty = [&](uint32_t s) { return bar0 + (kBarSlots + s) * 8; };
    const uint32_t bar_w0 = bar0 + 2 * kBarSlots * 8, bar_a0 = bar_w0 + 8;
    auto bar_x = [&](uint32_t h) { return bar_w0 + 16 + h * 8; };     // operand half h of the next layer written (both CTAs)
    auto bar_acc = [&](uint32_t h) { return bar_w0 + 32 + h * 8; };   // accumulator half h of the current layer complete
    const uint32_t ntiles = (p.n + 1) >> 1;
    const int L = p.n_layers;
    const uint32_t crank = cluster_ctarank();
    const bool leader = crank == 0;
    const uint32_t cbase = blockIdx.x - crank;   // tile of the pair's first CTA in the first iteration
    const uint32_t iters = cbase < ntiles ? (ntiles - cbase + gridDim.x - 1) / gridDim.x : 0u;

    // ---- one-time setup -----------------------------------------------------------------------------
    for (uint32_t i = threadIdx.x * 16; i < 3 * kHalfBytes; i += kThreads * 16) *reinterpret_cast<uint4*>(sm + kOffAct + i) = make_uint4(0, 0, 0, 0);
    fence_proxy_async();
    if (threadIdx.x == 0) {
        // the leader's `full` barriers also collect the peer's "my half of the stage has landed" relay
        for (uint32_t s = 0; s < kStages; ++s) { mbar_init(bar_full(s), leader ? 2 : 1); mbar_init(bar_empty(s), 1); }
        mbar_init(bar_w0, leader ? 2 : 1);
        mbar_init(bar_a0, 2 * kEpiThreads);
        mbar_init(bar_x(0), 2 * kEpiThreads);
        mbar_init(bar_x(1), 2 * kEpiThreads);
        mbar_init(bar_acc(0), 1);
        mbar_init(bar_acc(1), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {  // TMEM: all 512 columns of both SMs of the pair
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(base + kOffTmemPtr) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();  // the peer's barriers are initialised before anyone arrives on them or commits into them
    tc_fence_after();
    const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(sm + kOffTmemPtr);
    const uint32_t tm_res = tmem + 256;  // accumulator halves at tmem + 0 / + 128

    if (warp == 0) {
        // ===== weight producer: this CTA's 64-column slice of every stage =====================================
        if (lane == 0) {
            mbar_expect_tx(bar_w0, kW0Bytes);
            bulk_g2s(base + kOffW0, reinterpret_cast<const uint8_t*>(p.w0) + crank * kW0Bytes, kW0Bytes, bar_w0);
            uint32_t stage = 0, phase = 0;
            for (uint32_t it = 0; it < iters; ++it) {
                for (int l = 1; l < L; ++l) {
                    const uint8_t* src = reinterpret_cast<const uint8_t*>(p.w) + ((size_t)(l - 1) * kStagesPerLayer * 2 + crank) * kStageBytes;
                    for (uint32_t s = 0; s < kStagesPerLayer; ++s) {
                        mbar_wait(bar_empty(stage), phase ^ 1);
                        mbar_expect_tx(bar_full(stage), kStageBytes);
                        bulk_g2s(base + kOffW + stage * kStageBytes, src + (size_t)s * 2 * kStageBytes, kStageBytes, bar_full(stage));
                        if (++stage == kStages) { stage = 0; phase ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (leader) {
            // ===== MMA issuer (leader CTA): the whole warp runs the loop, one elected lane issues ================
            uint32_t stage = 0, phase = 0, a0_par = 0, x_par[2] = {0, 0};
            bool first = true, ready = false;
            for (uint32_t it = 0; it < iters; ++it) {
                // layer 0: [128 rows x 32] im2col tile per CTA x [32 x 128] per output half
                mbar_wait(bar_a0, a0_par);
                a0_par ^= 1;
                tc_fence_after();
                if (first) { mbar_wait(bar_w0, 0); first = false; }
#pragma unroll
                for (uint32_t nh = 0; nh < 2; ++nh) {
#pragma unroll
                    for (uint32_t j = 0; j < 2; ++j)
                        umma2_f16_elect(tmem + nh * 128, desc_lo(base + kOffA0 + j * 2 * 2048, 2048), desc_hi(128),
                                        desc_lo(base + kOffW0 + nh * 4096 + j * 2 * 1024, 1024), desc_hi(128), kIdesc, j);
                    umma2_commit_elect(bar_acc(nh));
                }
                for (int l = 1; l < L; ++l) {
                    const uint32_t x0 = base + kOffAct + ((l & 1) ? 0u : 2u) * kHalfBytes;   // channels 0-127 of this layer's input
                    const uint32_t x1 = base + kOffAct + kHalfBytes;                          // channels 128-255
                    for (uint32_t nh = 0; nh < 2; ++nh) {
                        for (uint32_t kh = 0; kh < 2; ++kh) {
                            if (nh == 0) {  // written by the previous layer's half-kh epilogue of BOTH CTAs (which also drained acc[kh])
                                mbar_wait(bar_x(kh), x_par[kh]);
                                x_par[kh] ^= 1;
                                tc_fence_after();
                            }
                            const uint32_t xb = kh ? x1 : x0;
                            for (uint32_t tap = 0; tap < 9; ++tap) {
                                // tap (kh, kw) reads input pixel (y + kh - 1, x + kw - 1): slot offset 2*kh, chunk offset kw
                                const uint32_t a_tap = xb + (2 * (tap / 3)) * kActSlot + (tap % 3) * 16;
                                const uint32_t a_lo = desc_lo(a_tap, kActCg);
                                if (!ready) mbar_wait(bar_full(stage), phase);
                                tc_fence_after();
                                const uint32_t b_lo = desc_lo(base + kOffW + stage * kStageBytes, 1024);
                                const uint32_t cur = stage;
                                if (++stage == kStages) { stage = 0; phase ^= 1; }
                                ready = mbar_test(bar_full(stage), phase);   // the answer arrives while the MMAs below are issued
#pragma unroll
                                for (uint32_t kbl = 0; kbl < 2; ++kbl) {    // block of 64 input channels within the K half
#pragma unroll
                                    for (uint32_t j = 0; j < 4; ++j)
                                        umma2_f16_elect(tmem + nh * 128, a_lo + ((kbl * 8 + 2 * j) * kActCg >> 4), desc_hi(kActSlot),
                                                        b_lo + ((kbl * 8192 + 2 * j * 1024) >> 4), desc_hi(128), kIdesc, (kh | tap | kbl | j) != 0);
                                }
                                umma2_commit_elect(bar_empty(cur));
                            }
                        }
                        umma2_commit_elect(bar_acc(nh));
                    }
                }
            }
        } else if (lane == 0) {
            // ===== peer CTA: tell the leader when this CTA's half of a weight stage has landed ==================
            uint32_t stage = 0, phase = 0;
            mbar_wait(bar_w0, 0);
            mbar_arrive_cta(bar_w0, 0);
            for (uint32_t it = 0; it < iters; ++it)
                for (int l = 1; l < L; ++l)
                    for (uint32_t s = 0; s < kStagesPerLayer; ++s) {
                        mbar_wait(bar_full(stage), phase);
                        mbar_arrive_cta(bar_full(stage), 0);
                        if (++stage == kStages) { stage = 0; phase ^= 1; }
                    }
        }
    } else {
        // ===== epilogue warps (8) ==================================================================
        const int et = threadIdx.x - 64;        // 0..255
        const int q = warp & 3;                 // TMEM sub-partition this warp may access
        const int sub = (warp - 2) >> 2;        // which 64 of a half's 128 columns this warp handles
        const int m = q * 32 + lane;            // accumulator row == TMEM lane
        const int g = m >> 3, x = m & 7, brd = g & 1, y = g >> 1;
        const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
        float* ss_s = reinterpret_cast<float*>(sm + kOffSS);
        float* part = reinterpret_cast<float*>(sm + kOffPart);
        float* hp = reinterpret_cast<float*>(sm + kOffHp);
        float* hv = reinterpret_cast<float*>(sm + kOffHv);
        float* logit = reinterpret_cast<float*>(sm + kOffLogit);
        float* fc1 = reinterpret_cast<float*>(sm + kOffFc1);
        const uint32_t row_off = (g + 2) * kActSlot + (x + 1) * 16;  // within a half-buffer, + cg * kActCg
        uint32_t acc_par[2] = {0, 0};
        uint32_t ss_buf = 0;

        for (uint32_t it = 0; it < iters; ++it) {
            const uint32_t tile = blockIdx.x + it * gridDim.x;  // may be >= ntiles: dummy tile (no valid board)
            const uint32_t pos0 = tile * 2;
            const bool valid = pos0 + brd < p.n;
            // ---- layer-0 operand: im2col of the two bit planes, K index = tap*2 + plane, padded to 32 ----
            epi_bar();   // the operand shares its bytes with the head scratch the other warps may still be reading (previous tile)
            build_layer0_operand(sm + kOffA0, valid ? p.own[pos0 + brd] : 0, valid ? p.enemy[pos0 + brd] : 0, 2 * sub, g, x, y);
            fence_proxy_async();
            mbar_arrive_cta(bar_a0, 0);   // also says: this thread has finished with the previous tile's accumulators

            float hp0 = 0.f, hp1 = 0.f, hvv = 0.f;
            for (int l = 0; l < L; ++l) {
                // stage this layer's folded BN parameters (double-buffered across layers)
                float* sc = ss_s + ss_buf * 512;
                sc[et] = __ldg(p.ss + (size_t)l * 512 + et);
                sc[256 + et] = __ldg(p.ss + (size_t)l * 512 + 256 + et);
                ss_buf ^= 1;
                epi_bar();
                const bool is_conv2 = l > 0 && (l & 1) == 0;   // second conv of a block: add the skip connection
                const bool keep_res = l == 0 || is_conv2;      // block output: keep fp32 copy in TMEM
                const bool last = l == L - 1;
                // next layer's input: channels 0-127 -> buffer A for odd layers, C for even ones; channels 128-255 -> B
                const uint32_t out0 = base + kOffAct + (((l + 1) & 1) ? 0u : 2u) * kHalfBytes + row_off;
                const uint32_t out1 = base + kOffAct + kHalfBytes + row_off;
#pragma unroll 1
                for (int h = 0; h < 2; ++h) {
                    mbar_wait(bar_acc(h), acc_par[h]);
                    acc_par[h] ^= 1;
                    tc_fence_after();
                    const uint32_t out = h ? out1 : out0;
                    // 2 chunks of 32 accumulator columns per thread; the TMEM load of the second is in flight while the first
                    // is processed
                    uint32_t va[32], vb[32], rr[32];
                    auto prefetch = [&](int c2, uint32_t (&v)[32], uint32_t (&r)[32]) {
                        const int c0 = h * 128 + sub * 64 + c2 * 32;
                        tmem_ld32(tmem + lane_sel + c0, v);
                        if (is_conv2) tmem_ld32(tm_res + lane_sel + c0, r);
                    };
                    auto math = [&](int c2, uint32_t (&v)[32], uint32_t (&r)[32]) {
                        epi_math(v, r, sc, h * 128 + sub * 64 + c2 * 32, is_conv2, keep_res || last);
                    };
                    auto store = [&](int c2, uint32_t (&v)[32]) {
                        const int c0 = h * 128 + sub * 64 + c2 * 32;
                        if (keep_res && !last) tmem_st32(tm_res + lane_sel + c0, v);
                        if (!last) epi_store_operand(v, out, sub * 8 + c2 * 4, keep_res);   // channel group within the half-buffer
                        else epi_head_partial(v, c0, p, hp0, hp1, hvv,
                                              (p.dbg_tower && valid) ? p.dbg_tower + ((size_t)(pos0 + brd) * 64 + y * 8 + x) * 256 : nullptr);
                    };
                    // the residual buffer rr is consumed by math(0) before prefetch(1) refills it
                    prefetch(0, va, rr);
                    tmem_wait_ld_dep(va); if (is_conv2) tmem_dep(rr);
                    math(0, va, rr); prefetch(1, vb, rr); store(0, va);
                    tmem_wait_ld_dep(vb); if (is_conv2) tmem_dep(rr);
                    math(1, vb, rr); store(1, vb);
                    if (!last) {
                        if (keep_res) tmem_wait_st();
                        fence_proxy_async();
                        tc_fence_before();
                        mbar_arrive_cta(bar_x(h), 0);   // operand half h written, accumulator half h drained (this thread's share)
                    }
                }
            }
            // ---- heads (agent/model.py:43-56) on the 256 epilogue threads --------------------------------
            heads_phase(p, hp0, hp1, hvv, sub, m, brd, y, x, et, warp - 2, lane, pos0, part, hp, hv, logit, fc1);
            // the next tile's layer-0 operand build only touches the A0 region, whose last reader (this tile's layer-0 MMAs)
            // completed before the first bar_acc of this tile
        }
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();  // no CTA leaves while the peer may still arrive on its barriers / the pair's MMAs touch its memory
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

// ---- weight packing ------------------------------------------------------------------------------------------------
// layer-0 image: [cta 2][nh 2][kc 4][n 64][8]; K index = (kh*3+kw)*2 + c padded to 32, output channel = nh*128 + cta*64 + n
__global__ void pack_w0_pair_kernel(const float* __restrict__ k0, __half* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 2 * 2 * 4 * 64 * 8) return;
    const int j = i & 7, n = (i >> 3) & 63, kc = (i >> 9) & 3, nh = (i >> 11) & 1, c = i >> 12, k = kc * 8 + j;
    const int co = nh * 128 + c * 64 + n;
    out[i] = __float2half_rn(k < 18 ? k0[(size_t)k * 256 + co] : 0.f);
}
// tower image: [layer][nh 2][kh 2][tap 9][cta 2][kbl 2][kc 8][n 64][8] fp16 (16 KB per CTA and stage);
// input channel = kh*128 + kbl*64 + kc*8 + j, output channel = nh*128 + cta*64 + n
__global__ void pack_w_pair_kernel(const float* __restrict__ blob, size_t off_res0, size_t stride, int n_layers, __half* __restrict__ out) {
    const size_t total = (size_t)n_layers * kStagesPerLayer * 2 * 8192;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int j = i & 7, n = (i >> 3) & 63, kc = (i >> 9) & 7, kbl = (i >> 12) & 1, c = (i >> 13) & 1;
        const size_t ls = i >> 14;                 // layer * 36 + stage
        const int s = (int)(ls % kStagesPerLayer), l = (int)(ls / kStagesPerLayer);
        const int tap = s % 9, kh = (s / 9) & 1, nh = s / 18;
        const int ci = kh * 128 + kbl * 64 + kc * 8 + j, co = nh * 128 + c * 64 + n;
        out[i] = __float2half_rn(blob[off_res0 + (size_t)l * stride + ((size_t)tap * 256 + ci) * 256 + co]);
    }
}

}  // namespace tc

int net_pack_tc(rz_net* net, cudaStream_t stream) {
    tc::pack_w0_pair_kernel<<<(2 * 2 * 4 * 64 * 8 + 255) / 256, 256, 0, stream>>>(net->blob + net->off_conv0, net->tc_w0);
    if (net->cfg.res_blocks > 0)
        tc::pack_w_pair_kernel<<<num_sms() * 8, 256, 0, stream>>>(net->blob, net->off_res0, net->res_stride_conv, 2 * net->cfg.res_blocks, net->tc_w);
    RZ_LAUNCH_CHECK();
    return RZ_OK;
}

int net_forward_tc(rz_net* net, const uint64_t* own, const uint64_t* enemy, float* policy, float* value, size_t n, cudaStream_t stream,
                   float* dbg_tower, const uint32_t* n_dev, float* dbg_logits, float* dbg_vlogit) {
    RZ_REQUIRE(net->cfg.filters == 256, "tcgen05 tower requires 256 filters");
    RZ_REQUIRE(net->cfg.value_fc <= (int)tc::kMaxV, "tcgen05 tower supports value_fc_size <= %u", tc::kMaxV);
    RZ_REQUIRE(n < (1ull << 31), "batch too large");
    static const cudaError_t smem_attr =
        cudaFuncSetAttribute(tc::net_tower_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::kSmemAlloc);
    RZ_CUDA_TRY(smem_attr);
    tc::Params p;
    p.w0 = net->tc_w0; p.w = net->tc_w; p.ss = net->scale_shift; p.blob = net->blob;
    p.off_policy_conv = net->off_policy_conv; p.off_policy_fc_k = net->off_policy_fc_k; p.off_policy_fc_b = net->off_policy_fc_b;
    p.off_value_conv = net->off_value_conv; p.off_value_fc1_k = net->off_value_fc1_k; p.off_value_fc1_b = net->off_value_fc1_b;
    p.off_value_fc2_k = net->off_value_fc2_k; p.off_value_fc2_b = net->off_value_fc2_b;
    p.own = own; p.enemy = enemy; p.policy = policy; p.value = value; p.dbg_tower = dbg_tower;
    p.dbg_logits = dbg_logits; p.dbg_vlogit = dbg_vlogit;
    p.n = (uint32_t)n; p.n_dev = n_dev; p.n_layers = 1 + 2 * net->cfg.res_blocks; p.V = net->cfg.value_fc;
    const uint32_t ntiles = (uint32_t)((n + 1) / 2);
    uint32_t grid = ntiles < (uint32_t)num_sms() ? ntiles : (uint32_t)num_sms();
    grid = (grid + 1) & ~1u;  // whole pairs; a surplus CTA runs dummy tiles
    if (grid > (uint32_t)num_sms()) grid = (uint32_t)num_sms() & ~1u;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(tc::kThreads); cfg.dynamicSmemBytes = tc::kSmemAlloc; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    RZ_CUDA_TRY(cudaLaunchKernelEx(&cfg, tc::net_tower_pair_kernel, p));
    RZ_LAUNCH_CHECK();
    return RZ_OK;
}

}  // namespace rz
