// onb_net.cu -- the policy/value network of the search (ConvResNet, alphazero-training/src/net.rs:118-232) as ONE fused
// kernel on the 5th-generation tensor cores (tcgen05.mma kind::f16 / kind::tf32, accumulators in TMEM, weights streamed by bulk TMA).
//
// What the reference computes per position (net.rs:215-232, restated in onitama_alphazero_b200/net.py):
//   y = relu(bn1(conv3x3(x)))                                  21 -> 64 channels on the 5x5 board
//   y = relu(bn(conv3x3(relu(bn(conv3x3(y))))) + y)            x resnet_block_amnt
//   policy = softmax(linear50x50(flatten(relu(bn(conv1x1 64->2 (y))))))   value = tanh(linear(relu(linear25->64(flatten(relu(bn(conv1x1 64->1 (y))))))))
// BatchNorm runs in eval mode (running statistics) and is folded into the convolution weights and a per-channel bias on the host.
//
// Mapping. A 3x3 convolution over N boards is the GEMM  out[cell][co] = sum_{tap, ci} act[cell + shift(tap)][ci] * W[tap][co][ci].
// Boards are laid out as a continuous sequence of CELLS, 36 per board: one row of 6 zero cells, then 5 rows of (5 squares + 1 zero
// cell). Every out-of-board neighbour of a square is then one of those zero cells (of this board or the next), so a tap is nothing
// but a ROW SHIFT of the activation matrix by dy*6+dx cells. The activations live in shared memory in the tensor core's K-major
// operand layout, one 128-byte swizzled row per cell: a shifted window is just a different start address in the shared-memory
// descriptor -- no im2col copy is ever made.
// One CTA keeps NB boards (two accumulators of 128 cells x 64 channels in TMEM) on chip through ALL layers; only the input planes
// are read from and only policy/value are written to global memory. The residual input of a block is parked in TMEM (pre-loaded
// into the accumulator of the block's second convolution together with that layer's bias), so the skip connection costs nothing.
// Weights (rounded, BN folded, already in the swizzled operand layout) are streamed through a small ring by one producer thread
// with cp.async.bulk + mbarriers; warp 0 runs the MMA issue loop (one elected lane issues); all 8 warps run the epilogues (TMEM ->
// bias/ReLU -> operand format -> shared memory). Arithmetic: f32 accumulation of products of operands rounded to an 11-bit
// significand -- either f16 (default) or tf32 (what libtorch's cuDNN convolutions use by default on this GPU; same significand,
// twice the shared-memory bytes per MMA and half the tensor rate; the kernel is bound by the operand reads). Heads in f32.
// Measurements, the variants that were tried and the phase timings are in DESIGN.md section 5b.
#include <cuda_fp16.h>

#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "onb_internal.h"

namespace onb {
namespace {

constexpr int kHid = 64;             // hidden channels (ConvResNetConfig::hidden_channels) the kernel is built for
constexpr int kInPlanes = 21;        // input planes (common.rs:26-80)
constexpr int kCellsPerBoard = 36;
constexpr int kLead = 8, kTrail = 8;  // zero rows before the first / after the last cell (|shift| <= 7)
constexpr int kMaxBlocks = 16;
// operand format: a 16-byte chunk holds CPC channels; one MMA consumes two chunks of every row (K = 32 bytes)
template <bool F16>
struct Op {
    static constexpr int ELT = F16 ? 2 : 4;
    static constexpr int CPC = 16 / ELT;               // 8 | 4 channels per chunk
    static constexpr int KCH = kHid / CPC;             // 8 | 16 chunks per 64 channels
    static constexpr int IN_PAD = F16 ? 32 : 24;       // input planes padded to a multiple of the MMA's K (16 | 8)
    static constexpr int KCH0 = IN_PAD / CPC;          // 4 | 6
    static constexpr int TAP_BYTES = KCH * 64 * 16;    // one tap of a 64 -> 64 layer: [KB][64 co][128 B], swizzled
    static constexpr int TAP_BYTES0 = 64 * 128;        // first layer: its K (32 | 24 channels) fits the first 128-byte block
    // instruction descriptor (cute::UMMA::InstrDescriptor): f32 accumulate, A/B format, both K-major, N = 64, M = 128
    static constexpr uint32_t idesc(uint32_t n) { return (1u << 4) | ((F16 ? 0u : 2u) << 7) | ((F16 ? 0u : 2u) << 10) | ((n >> 3) << 17) | ((128u >> 4) << 24); }
    static constexpr uint32_t IDESC = idesc(64), IDESC_N128 = idesc(128);
};
// head parameter blob (floats)
constexpr int kHP0 = 0, kHP1 = 64, kHV = 128, kHB = 192, kPhW = 196, kPhB = 2696, kV1W = 2748, kV1B = 4348, kV2W = 4412, kV2B = 4476,
              kHeadFloats = 4480;

// X3 (ONB_NET_F32, f16 operands only): every f32 operand x is split as x = x1 + 2^-11 x2 with x1 = f16(x), x2 = f16((x - x1) 2^11)
// (22+ significand bits; the scaling keeps x2 in f16's normal range however small x is). A product a b is then
// a1 b1 + 2^-11 (a1 b2 + a2 b1) up to 2^-23 relative: three MMAs per step, the first into accumulator D1, the other two into a
// second accumulator D2 that the epilogue adds as D1 + 2^-11 D2. Two activation matrices (a1, a2), weights streamed as (b1, b2)
// pairs per tap, TMEM = {D1, D2} x {plain, residual-preloaded} x 2 x 64 columns = 512: one CTA per SM.
constexpr float kX3Scale = 2048.f, kX3InvScale = 1.f / 2048.f;
template <bool F16, bool X3 = false>
struct Geo {
    static_assert(!X3 || F16, "the split-operand mode is built on the f16 operand path");
    static constexpr int NACC = 2;           // accumulators of 128 cells
    static constexpr int NMAT = X3 ? 2 : 1;  // activation matrices / weight copies per tap
    static constexpr int NB = F16 ? 7 : 6;   // boards per pass (two CTAs per SM)
    static constexpr int CELLS = NB * kCellsPerBoard;
    static constexpr int R = (kLead + CELLS + kTrail + 7) / 8 * 8;  // rows of the activation matrix (whole swizzle periods)
    // weight ring: NSLOT slots of TPS taps, one full/empty barrier round trip and one bulk copy per slot. f16: 3 slots x 3 taps =
    // one whole layer in flight, so the producer runs a layer ahead of the MMAs (with 4 single-tap slots the MMA thread waited for
    // weights, and per-tap slots cost a try_wait + fence + commit for every 8 MMAs); tf32 taps are twice as large: single taps
    static constexpr int NSLOT = 3;
    static constexpr int TPS = F16 ? 3 : 1;
    static constexpr int UPL = 9 / TPS;  // slots per layer
    static constexpr int TAP_STRIDE = NMAT * Op<F16>::TAP_BYTES;  // X3: [b1 tap][b2 tap]
    static constexpr int SLOT_BYTES = TPS * TAP_STRIDE;
    static constexpr int ACT_BYTES = R * Op<F16>::KCH * 16;  // a multiple of 1024: the ring stays aligned to the swizzle period
    static constexpr int OFF_RING = NMAT * ACT_BYTES;
    static constexpr int RING_BYTES = NSLOT * SLOT_BYTES;
    static constexpr int OFF_HEAD = OFF_RING + RING_BYTES;
    static constexpr int HEAD_BYTES = ((NB * 75 * 4 + 15) / 16) * 16;
    static constexpr int OFF_BAR = OFF_HEAD + HEAD_BYTES;
    static constexpr int SMEM_USED = OFF_BAR + (2 * NSLOT + 1) * 8 + 16;
    // TMEM holds two CTAs of 256 columns: ask for enough shared memory that a third CTA can never become resident and block in tcgen05.alloc
    static constexpr int SMEM = SMEM_USED < 78 * 1024 ? 78 * 1024 : SMEM_USED;
    static constexpr int SET_COLS = NMAT * NACC * 64;  // one accumulator set: D1 (and D2) of NACC x 64 columns
    static constexpr int TMEM_COLS = 2 * SET_COLS;     // the plain set + the residual-preloaded set
    static_assert(SMEM_USED <= 227 * 1024, "shared memory");
    static_assert(CELLS <= NACC * 128, "cells must fit the accumulators");
    static_assert(TMEM_COLS == 256 || TMEM_COLS == 512, "power of two");
};

struct NetDev {
    const uint8_t* wconv;  // all conv taps in operand layout
    const uint8_t* wpair;  // ONB_NET_F32 only: the taps as the CTA-pair kernel streams them, [rank][layer][tap][12 KB]
    const float* bias;   // [1 + 2 * n_blocks][64] folded biases
    const float* head;   // kHeadFloats
    int n_blocks;
};

// ---- PTX helpers ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
// bounded wait: a protocol error must end in a trap (the launch fails with an error), never in a hang
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    if (mbar_try(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try(bar, parity)) {
        if (clock64() - t0 > 4000000000ll) __trap();
    }
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes),
                 "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// Operand layout (both A and B): K-major, 128-byte swizzle. A matrix row is KB blocks of 128 bytes (64 f16 | 32 tf32 channels); block
// kb of row r lives at base + kb * rows * 128 + r * 128 and its 16-byte chunk c sits at chunk position c ^ (r & 7) (base 1024-aligned).
// Rows are therefore 128 bytes apart, so a window that starts at ANY row is 128-byte aligned: every 8-row x 32-byte operand fetch of
// the tensor core touches each bank once. (The first version used the no-swizzle layout with rows 16 bytes apart; windows shifted
// by a number of rows that is not a multiple of 8 then straddle two 128-byte lines per core matrix and the MMAs ran at ~80 cycles
// instead of 48.) Descriptor: start address, leading offset 1 (unused for swizzled K-major), 1024 bytes between 8-row groups,
// version 1, base offset = row phase of the start address (start >> 7) & 7, layout type 2 = SWIZZLE_128B.
#ifndef ONB_NET_BASEOFF
#define ONB_NET_BASEOFF 0
#endif
__device__ __forceinline__ uint32_t desc_hi(uint32_t start_addr) {
    return (1024u >> 4) | (1u << 14) | (ONB_NET_BASEOFF ? (((start_addr >> 7) & 7u) << 17) : 0u) | (2u << 29);
}
__device__ __forceinline__ uint32_t desc_lo(uint32_t start_addr) { return ((start_addr & 0x3FFFFu) >> 4) | (1u << 16); }
// one lane of a converged warp (the issue loops run warp-uniformly so that descriptors stay in uniform registers; only the
// tcgen05 instructions themselves are issued by the elected lane)
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}
template <bool F16>
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint32_t a_addr, uint32_t b_addr, uint32_t accumulate, uint32_t idesc = Op<F16>::IDESC) {
    const uint32_t a_lo = desc_lo(a_addr), a_hi = desc_hi(a_addr), b_lo = desc_lo(b_addr), b_hi = desc_hi(b_addr);
    if (F16)
        asm volatile(
            "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
            "setp.ne.b32 p, %6, 0;\n\t"
            "mov.b64 da, {%1, %2};\n\t"
            "mov.b64 db, {%3, %4};\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}" ::"r"(d_tmem),
            "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
            : "memory");
    else
        asm volatile(
            "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
            "setp.ne.b32 p, %6, 0;\n\t"
            "mov.b64 da, {%1, %2};\n\t"
            "mov.b64 db, {%3, %4};\n\t"
            "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %5, p;\n\t}" ::"r"(d_tmem),
            "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
            : "memory");
}
// The same MMAs from precomputed descriptor words. The low word of a shared-memory descriptor -- (address >> 4) in 14 bits | the
// leading-offset field -- is LINEAR in the byte address below 256 KB and the high word is a constant, so an issue loop can keep one
// low word per operand base and add compile-time offsets (>> 4) instead of rebuilding both descriptors for every instruction: the
// MMA warp's own instruction stream (not the tensor pipe) was what paced the pipelined kernels, ~ 100 instructions per tap.
template <bool PAIR, bool F16 = true>
__device__ __forceinline__ void mma_lo(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t accumulate, uint32_t idesc) {
    const uint32_t hi = desc_hi(0u);
    static_assert(ONB_NET_BASEOFF == 0, "the descriptor high word must not depend on the address");
    static_assert(F16 || !PAIR, "the CTA-pair kernels use f16 operands");
    if (!F16)
        asm volatile(
            "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
            "setp.ne.b32 p, %5, 0;\n\t"
            "mov.b64 da, {%1, %3};\n\t"
            "mov.b64 db, {%2, %3};\n\t"
            "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %4, p;\n\t}" ::"r"(d_tmem),
            "r"(a_lo), "r"(b_lo), "r"(hi), "r"(idesc), "r"(accumulate)
            : "memory");
    else if (PAIR)
        asm volatile(
            "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
            "setp.ne.b32 p, %5, 0;\n\t"
            "mov.b64 da, {%1, %3};\n\t"
            "mov.b64 db, {%2, %3};\n\t"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %4, p;\n\t}" ::"r"(d_tmem),
            "r"(a_lo), "r"(b_lo), "r"(hi), "r"(idesc), "r"(accumulate)
            : "memory");
    else
        asm volatile(
            "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
            "setp.ne.b32 p, %5, 0;\n\t"
            "mov.b64 da, {%1, %3};\n\t"
            "mov.b64 db, {%2, %3};\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n\t}" ::"r"(d_tmem),
            "r"(a_lo), "r"(b_lo), "r"(hi), "r"(idesc), "r"(accumulate)
            : "memory");
}
// all MMAs of one tap: K steps of 32 bytes (4 per 128-byte block) x 2 accumulators of 128 rows
// X3: per step TWO instructions instead of three: a1 x [b1 ; b2] as ONE N = 128 MMA (the tap's two weight copies are adjacent in
// the ring, so they are simply 128 consecutive B rows; its 128 result columns are D1 | D2 of the accumulator, which therefore sit
// side by side in TMEM), then a2 x b1 (N = 64) onto D2. a1 is fetched from shared memory once for both of its products: 14 KB of
// operands per step instead of 18 KB -- the operand fetch is what bounds this kernel. a2_off = byte distance of the second
// activation matrix. D2 must hold zeros when D1 was preloaded with the residual (the epilogue that parks the residual writes them).
template <bool F16, bool X3 = false>
__device__ __forceinline__ void issue_tap_mmas(bool elected, uint32_t dcol, uint32_t s_act, int R, int row0, uint32_t b_slot, int ksteps,
                                               bool accumulate_first, uint32_t a2_off = 0) {
    using O = Op<F16>;
    constexpr uint32_t ACC_COLS = X3 ? 128u : 64u;  // TMEM columns per accumulator
    // descriptor low words of the tap's operand bases (whole warp: uniform registers); steps, blocks and accumulators add constants
    const uint32_t a_lo = desc_lo(s_act + (uint32_t)row0 * 128u), b_lo = desc_lo(b_slot), a2_lo = a2_off >> 4;
#ifndef ONB_NET_DBG_NOMMA
    if (elected) {
#pragma unroll
        for (int j = 0; j < O::KCH / 2; ++j) {
            if (j < ksteps) {
                const uint32_t kb = (uint32_t)(j / 4), ks = (uint32_t)(j % 4) * 2u;  // 128-byte block of the row, 32-byte step inside it
                const uint32_t bj = b_lo + kb * (64u * 128u >> 4) + ks;
#pragma unroll
                for (int a = 0; a < 2; ++a) {
                    const uint32_t aj = a_lo + kb * (uint32_t)(R * 8) + (uint32_t)(a * 128 * 8) + ks;
                    if (X3) {
                        mma_lo<false, F16>(dcol + a * ACC_COLS, aj, bj, (accumulate_first || j > 0) ? 1u : 0u, O::IDESC_N128);  // a1 b1 | a1 b2
                        mma_lo<false, F16>(dcol + a * ACC_COLS + 64u, aj + a2_lo, bj, 1u, O::IDESC);                           // a2 b1 -> D2
                    } else {
                        mma_lo<false, F16>(dcol + a * ACC_COLS, aj, bj, (accumulate_first || j > 0) ? 1u : 0u, O::IDESC);
                    }
                }
            }
        }
    }
#endif
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, "
        "%20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
          "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
          "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]),
          "=r"(v[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, "
        "%20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
          "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
          "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]),
          "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, "
        "%20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
        "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]),
        "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]),
        "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
        : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ uint32_t to_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}
// two f32 -> packed f16, round to nearest, SATURATING at +-65504 in the conversion itself (F2FP.SATFINITE: one instruction where a
// clamp + convert was three); activations past f16's range saturate instead of becoming inf
__device__ __forceinline__ uint32_t to_f16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ float2 f16x2_to_float2(uint32_t h) { return __half22float2(*reinterpret_cast<const __half2*>(&h)); }
// store 32 consecutive channels [c0, c0 + 32) of one cell as operand chunks
template <bool F16>
__device__ __forceinline__ void store_channels(uint32_t s_act, int R, int row, int c0, const float (&o)[32]);
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
// byte address of 16-byte chunk `chunk` (0 .. KCH-1) of row `row` (see the operand layout above)
__device__ __forceinline__ uint32_t act_addr(uint32_t s_act, int R, int row, int chunk) {
    return s_act + (uint32_t)(chunk >> 3) * (uint32_t)R * 128u + (uint32_t)row * 128u + (uint32_t)(((chunk & 7) ^ (row & 7)) << 4);
}
template <>
__device__ __forceinline__ void store_channels<true>(uint32_t s_act, int R, int row, int c0, const float (&o)[32]) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
        st_shared_v4(act_addr(s_act, R, row, c0 / 8 + i), to_f16x2(o[8 * i + 0], o[8 * i + 1]), to_f16x2(o[8 * i + 2], o[8 * i + 3]),
                     to_f16x2(o[8 * i + 4], o[8 * i + 5]), to_f16x2(o[8 * i + 6], o[8 * i + 7]));
}
template <>
__device__ __forceinline__ void store_channels<false>(uint32_t s_act, int R, int row, int c0, const float (&o)[32]) {
#pragma unroll
    for (int i = 0; i < 8; ++i)
        st_shared_v4(act_addr(s_act, R, row, c0 / 4 + i), to_tf32(o[4 * i + 0]), to_tf32(o[4 * i + 1]), to_tf32(o[4 * i + 2]),
                     to_tf32(o[4 * i + 3]));
}
// split-operand store: x1 = f16(x) into the first activation matrix, x2 = f16((x - x1) 2^11) into the second (x - x1 is exact in f32)
__device__ __forceinline__ void store_channels_x3(uint32_t s_act, uint32_t a2_off, int R, int row, int c0, const float (&o)[32]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float x0 = o[8 * i + 2 * q], x1 = o[8 * i + 2 * q + 1];
            hi[q] = to_f16x2(x0, x1);  // saturating
            const float2 hf = f16x2_to_float2(hi[q]);
            lo[q] = to_f16x2((x0 - hf.x) * kX3Scale, (x1 - hf.y) * kX3Scale);
        }
        const uint32_t addr = act_addr(s_act, R, row, c0 / 8 + i);
        st_shared_v4(addr, hi[0], hi[1], hi[2], hi[3]);
        st_shared_v4(addr + a2_off, lo[0], lo[1], lo[2], lo[3]);
    }
}
// the same in two steps, for owners that have to hold their chunks back until a reader of the old rows is done
__device__ __forceinline__ void pack_channels_x3(const float (&o)[32], uint32_t (&hi)[16], uint32_t (&lo)[16]) {
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        const float x0 = o[2 * q], x1 = o[2 * q + 1];
        hi[q] = to_f16x2(x0, x1);  // saturating
        const float2 hf = f16x2_to_float2(hi[q]);
        lo[q] = to_f16x2((x0 - hf.x) * kX3Scale, (x1 - hf.y) * kX3Scale);
    }
}
__device__ __forceinline__ void store_packed_x3(uint32_t s_act, uint32_t a2_off, int R, int row, int c0, const uint32_t (&hi)[16], const uint32_t (&lo)[16]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const uint32_t addr = act_addr(s_act, R, row, c0 / 8 + i);
        st_shared_v4(addr, hi[4 * i], hi[4 * i + 1], hi[4 * i + 2], hi[4 * i + 3]);
        st_shared_v4(addr + a2_off, lo[4 * i], lo[4 * i + 1], lo[4 * i + 2], lo[4 * i + 3]);
    }
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xFFFFFFFFu, v, o));
    return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    return v;
}

// cell -> (board in pass, square 0..24) or pad
struct Cell {
    int board, pos;
    bool real;
};
__device__ __forceinline__ Cell decode_cell(int cell, int n_cells) {
    Cell c;
    c.board = cell / kCellsPerBoard;
    const int k = cell - c.board * kCellsPerBoard;  // 0..35: row of 6 zero cells, then 5 x (5 squares + 1 zero cell)
    const int row = k / 6, col = k - row * 6;
    c.real = cell < n_cells && row >= 1 && col < 5;
    c.pos = (row - 1) * 5 + col;
    return c;
}

template <bool F16, bool X3 = false>
__global__ void __launch_bounds__(256, X3 ? 1 : 2)
    k_net_forward(const float* __restrict__ planes, float* __restrict__ policy, float* __restrict__ value, int64_t n, NetDev net) {
    using G = Geo<F16, X3>;
    using O = Op<F16>;
    constexpr int NB = G::NB, CELLS = G::CELLS, R = G::R, NSLOT = G::NSLOT;
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t s_act = smem_u32(smem), s_ring = s_act + G::OFF_RING, s_bar = s_act + G::OFF_BAR;
    float* s_head = reinterpret_cast<float*>(smem + G::OFF_HEAD);
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + G::OFF_BAR + (2 * NSLOT + 1) * 8);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int L = 1 + 2 * net.n_blocks;
    const int64_t n_groups = (n + NB - 1) / NB;
    if ((int64_t)blockIdx.x >= n_groups) return;  // whole CTA, before any allocation
    const int64_t my_groups = (n_groups - blockIdx.x + gridDim.x - 1) / gridDim.x;
    constexpr int TPS = G::TPS, UPL = G::UPL;
    const uint32_t total_units = (uint32_t)my_groups * (uint32_t)(UPL * L);
    auto bar_full = [&](uint32_t s) { return s_bar + s * 8u; };
    auto bar_empty = [&](uint32_t s) { return s_bar + (NSLOT + s) * 8u; };
    const uint32_t bar_acc = s_bar + 2 * NSLOT * 8u;

    if (tid == 0) {
        for (uint32_t s = 0; s < (uint32_t)NSLOT; ++s) {
            mbar_init(bar_full(s), 1);
            mbar_init(bar_empty(s), 1);
        }
        mbar_init(bar_acc, 1);
        fence_barrier_init();
    }
    if (warp == 0) tmem_alloc(smem_u32(s_tmem), G::TMEM_COLS);
    for (int i = tid; i < G::NMAT * G::ACT_BYTES / 16; i += 256) st_shared_v4(s_act + i * 16, 0u, 0u, 0u, 0u);  // pad cells stay zero for good
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *s_tmem;
    constexpr uint32_t A2 = X3 ? (uint32_t)G::ACT_BYTES : 0u;  // second activation matrix
    constexpr uint32_t ACC = X3 ? 128u : 64u;                  // TMEM columns per accumulator (X3: D1 | D2 side by side)
    constexpr uint32_t SET = (uint32_t)G::SET_COLS;  // TMEM columns of one accumulator set (D1 [+ D2])

#ifdef ONB_NET_PROFILE
    long long pf[8] = {0, 0, 0, 0, 0, 0, 0, 0}, pt = clock64();
#define PF(k) do { const long long now__ = clock64(); pf[k] += now__ - pt; pt = now__; } while (0)
#else
#define PF(k) do { } while (0)
#endif
    uint32_t q0 = 0;      // ring position of the current layer's first tap (all threads)
    uint32_t q_prod = 0;  // taps requested so far (producer thread)
    uint32_t acc_par = 0;
    for (int64_t gi = 0; gi < my_groups; ++gi) {
        const int64_t board0 = ((int64_t)blockIdx.x + gi * gridDim.x) * NB;
        // ---- input planes -> channel chunks 0..5 of the activation matrix (create_tensor_from_state layout [21][5][5])
        for (int cell = tid; cell < CELLS; cell += 256) {
            const Cell c = decode_cell(cell, CELLS);
            if (!c.real) continue;
            const int64_t gb = board0 + c.board;
            const float* src = planes + gb * 525 + c.pos;
            float x[32];  // the planes are 0 / 1: exact in either operand format
#pragma unroll
            for (int ch = 0; ch < 32; ++ch) x[ch] = (ch < kInPlanes && gb < n) ? __ldg(src + ch * 25) : 0.f;
            if (X3) store_channels_x3(s_act, A2, R, kLead + cell, 0, x);
            else store_channels<F16>(s_act, R, kLead + cell, 0, x);  // 32 channels: planes 21..31 are zero
        }
        fence_proxy_async();
        PF(0);  // input stage
        for (int l = 0; l < L; ++l) {
            tc_fence_before();
            __syncthreads();
            tc_fence_after();
            PF(1);  // layer-top barrier
            const bool use_s = l >= 2 && (l & 1) == 0;  // second convolution of a block accumulates onto the parked residual
            const bool last = l == L - 1;
            if (warp == 0) {
                // ---- MMA issue: 9 taps x K steps x 2 accumulators (the whole warp runs the loop, one lane issues)
                const bool elected = elect_one();
                const uint32_t dcol = tmem + (use_s ? SET : 0u);
                auto issue_unit = [&](int g, int ksteps) {
                    const uint32_t u = q0 + g, slot = u % NSLOT, use = u / NSLOT;
#ifdef ONB_NET_PROFILE
                    if (!mbar_try(bar_full(slot), use & 1u)) pf[7] += 1;  // weights not there yet
#endif
                    mbar_wait(bar_full(slot), use & 1u);
                    PF(2);  // waiting for weights
                    tc_fence_after();
                    PF(0);  // (profile build: the fence is booked on the input-stage counter)
#pragma unroll
                    for (int tt = 0; tt < TPS; ++tt) {
                        const int t = g * TPS + tt;
                        issue_tap_mmas<F16, X3>(elected, dcol, s_act, R, kLead + (t / 3 - 1) * 6 + (t % 3 - 1),
                                                      s_ring + slot * (uint32_t)G::SLOT_BYTES + (uint32_t)tt * (uint32_t)G::TAP_STRIDE, ksteps,
                                                      use_s || t > 0, A2);
                    }
                    PF(3);  // issuing MMAs
                    if (elected) umma_commit(bar_empty(slot));  // the slot is free again once these MMAs have read it
                    PF(1);  // (profile build: the commit is booked on the barrier counter)
                };
                if (l == 0) {
#pragma unroll 1
                    for (int g = 0; g < UPL; ++g) issue_unit(g, O::KCH0 / 2);
                } else {
#pragma unroll 1
                    for (int g = 0; g < UPL; ++g) issue_unit(g, O::KCH / 2);
                }
                if (elected) umma_commit(bar_acc);
            } else if (tid == 32) {
                // ---- weight producer: keeps the ring NSLOT taps ahead of the MMAs (weights do not depend on the data)
                const uint32_t target = min(q0 + (uint32_t)(UPL + NSLOT), total_units);
                while (q_prod < target) {
                    const uint32_t slot = q_prod % NSLOT, use = q_prod / NSLOT;
                    if (use >= 1) mbar_wait(bar_empty(slot), (use - 1u) & 1u);
                    const uint32_t ul = q_prod % (uint32_t)(UPL * L), layer = ul / UPL, tap = (ul - layer * UPL) * TPS;
                    const uint8_t* src = net.wconv + (size_t)G::NMAT * (layer == 0 ? (size_t)tap * O::TAP_BYTES0
                                                                  : (size_t)9 * O::TAP_BYTES0 + ((size_t)(layer - 1) * 9 + tap) * O::TAP_BYTES);
                    const uint32_t bytes = (uint32_t)(TPS * G::NMAT) * (layer == 0 ? O::TAP_BYTES0 : O::TAP_BYTES);
#ifdef ONB_NET_DBG_NOWEIGHTS
                    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar_full(slot)) : "memory");
                    (void)src; (void)bytes;
#else
                    mbar_expect_tx(bar_full(slot), bytes);
                    bulk_g2s(s_ring + slot * (uint32_t)G::SLOT_BYTES, src, bytes, bar_full(slot));
#endif
                    ++q_prod;
                }
            }
            __syncwarp();
            mbar_wait(bar_acc, acc_par);
            acc_par ^= 1u;
            tc_fence_after();
            PF(4);  // waiting for the accumulators
            // ---- epilogue: this thread owns one cell (TMEM lane) of accumulator warp/4
            const bool preload = (l & 1) == 0 && !last;  // this layer's output is a block input: park it (+ next bias) in TMEM
            const float4* bias_l = reinterpret_cast<const float4*>(net.bias + (size_t)l * 64);
            const float4* bias_n = reinterpret_cast<const float4*>(net.bias + (size_t)(preload ? l + 2 : l) * 64);
            const float4* hw = reinterpret_cast<const float4*>(net.head);
#ifdef ONB_NET_DBG_NOEPI
            if (l >= 0 && !last) { fence_proxy_async(); q0 += (uint32_t)UPL; continue; }
#endif
            const int a = warp >> 2;
            const int cell = a * 128 + (warp & 3) * 32 + lane;
            const Cell c = decode_cell(cell, CELLS);
            const uint32_t tlane = tmem + ((uint32_t)((warp & 3) * 32) << 16);
            const uint32_t tsrc = tlane + (use_s ? SET : 0u) + a * ACC;
            const uint32_t tskip = tlane + SET + a * ACC;
            float hp0 = 0.f, hp1 = 0.f, hv = 0.f;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                uint32_t v[32];
                if (X3) {  // D1 + 2^-11 D2: both loads in flight, one wait
                    uint32_t v2[32];
                    tmem_ld32_nowait(tsrc + h * 32, v);
                    tmem_ld32_nowait(tsrc + 64 + h * 32, v2);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                    for (int i = 0; i < 32; ++i) v[i] = __float_as_uint(fmaf(__uint_as_float(v2[i]), kX3InvScale, __uint_as_float(v[i])));
                } else {
                    tmem_ld32(tsrc + h * 32, v);
                }
                float o[32];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (!use_s) b = __ldg(bias_l + h * 8 + i);
                    o[4 * i + 0] = fmaxf(__uint_as_float(v[4 * i + 0]) + b.x, 0.f);
                    o[4 * i + 1] = fmaxf(__uint_as_float(v[4 * i + 1]) + b.y, 0.f);
                    o[4 * i + 2] = fmaxf(__uint_as_float(v[4 * i + 2]) + b.z, 0.f);
                    o[4 * i + 3] = fmaxf(__uint_as_float(v[4 * i + 3]) + b.w, 0.f);
                }
                if (!last && c.real) {
                    if (X3) store_channels_x3(s_act, A2, R, kLead + cell, h * 32, o);
                    else store_channels<F16>(s_act, R, kLead + cell, h * 32, o);
                }
                if (preload) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float4 b = __ldg(bias_n + h * 8 + i);
                        v[4 * i + 0] = __float_as_uint(o[4 * i + 0] + b.x);
                        v[4 * i + 1] = __float_as_uint(o[4 * i + 1] + b.y);
                        v[4 * i + 2] = __float_as_uint(o[4 * i + 2] + b.z);
                        v[4 * i + 3] = __float_as_uint(o[4 * i + 3] + b.w);
                    }
                    tmem_st32(tskip + h * 32, v);
                    if (X3) {  // the D2 half of the preloaded accumulator starts the next-but-one layer from zero
#pragma unroll
                        for (int i = 0; i < 32; ++i) v[i] = 0u;
                        tmem_st32(tskip + 64 + h * 32, v);
                    }
                }
                if (last) {  // 1x1 convolutions of both heads (net.rs: policy_conv 64 -> 2, vh_conv 64 -> 1)
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float4 w0 = __ldg(hw + (kHP0 / 4) + h * 8 + i), w1 = __ldg(hw + (kHP1 / 4) + h * 8 + i),
                                     w2 = __ldg(hw + (kHV / 4) + h * 8 + i);
                        hp0 = fmaf(o[4 * i + 0], w0.x, fmaf(o[4 * i + 1], w0.y, fmaf(o[4 * i + 2], w0.z, fmaf(o[4 * i + 3], w0.w, hp0))));
                        hp1 = fmaf(o[4 * i + 0], w1.x, fmaf(o[4 * i + 1], w1.y, fmaf(o[4 * i + 2], w1.z, fmaf(o[4 * i + 3], w1.w, hp1))));
                        hv = fmaf(o[4 * i + 0], w2.x, fmaf(o[4 * i + 1], w2.y, fmaf(o[4 * i + 2], w2.z, fmaf(o[4 * i + 3], w2.w, hv))));
                    }
                }
            }
            if (last && c.real) {
                float* hb = s_head + c.board * 75;
                hb[c.pos] = fmaxf(hp0 + __ldg(net.head + kHB + 0), 0.f);
                hb[25 + c.pos] = fmaxf(hp1 + __ldg(net.head + kHB + 1), 0.f);
                hb[50 + c.pos] = fmaxf(hv + __ldg(net.head + kHB + 2), 0.f);
            }
            if (preload) tmem_wait_st();
            fence_proxy_async();
            q0 += (uint32_t)UPL;
            PF(5);  // epilogue
        }
        // ---- heads: one warp per board (ph_linear2 + softmax, vh_linear1 + ReLU + vh_linear2 + tanh)
        __syncthreads();
        for (int b = warp; b < NB; b += 8) {
            const int64_t gb = board0 + b;
            if (gb >= n) continue;
            const float* hb = s_head + b * 75;
            const bool two = lane + 32 < 50;
            float l0 = __ldg(net.head + kPhB + lane), l1 = two ? __ldg(net.head + kPhB + 32 + lane) : 0.f;
            for (int i = 0; i < 50; ++i) {
                const float x = hb[i];
                l0 = fmaf(x, __ldg(net.head + kPhW + i * 50 + lane), l0);
                if (two) l1 = fmaf(x, __ldg(net.head + kPhW + i * 50 + 32 + lane), l1);
            }
            const float m = warp_max(two ? fmaxf(l0, l1) : l0);
            const float e0 = expf(l0 - m), e1 = two ? expf(l1 - m) : 0.f;
            const float s = warp_sum(e0 + e1);
            policy[gb * 50 + lane] = e0 / s;
            if (two) policy[gb * 50 + 32 + lane] = e1 / s;
            float h0 = __ldg(net.head + kV1B + lane), h1 = __ldg(net.head + kV1B + 32 + lane);
            for (int i = 0; i < 25; ++i) {
                const float x = hb[50 + i];
                h0 = fmaf(x, __ldg(net.head + kV1W + i * 64 + lane), h0);
                h1 = fmaf(x, __ldg(net.head + kV1W + i * 64 + 32 + lane), h1);
            }
            float acc = fmaf(fmaxf(h0, 0.f), __ldg(net.head + kV2W + lane), fmaxf(h1, 0.f) * __ldg(net.head + kV2W + 32 + lane));
            acc = warp_sum(acc);
            if (lane == 0) value[gb] = tanhf(acc + __ldg(net.head + kV2B));
        }
        PF(6);  // heads
    }
#ifdef ONB_NET_PROFILE
    if (blockIdx.x == (CL ? 2 : 3) && (tid == 0 || tid == 64))
        printf("net profile tid %d groups %lld: input+fence %lld barrier+commit %lld weights %lld (late %lld) issue %lld acc %lld epilogue %lld heads %lld\n",
               tid, (long long)my_groups, pf[0], pf[1], pf[2], pf[7], pf[3], pf[4], pf[5], pf[6]);
#endif
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, G::TMEM_COLS);
}

// 16-column TMEM access and f16 operand stores of the many-warp epilogues below
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
          "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
        "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]),
        "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
        : "memory");
}
// 16 consecutive channels [c0, c0 + 16) of one cell as f16 operand chunks
__device__ __forceinline__ void store_channels_f16_16(uint32_t s_act, int R, int row, int c0, const float (&o)[16]) {
#pragma unroll
    for (int i = 0; i < 2; ++i)
        st_shared_v4(act_addr(s_act, R, row, c0 / 8 + i), to_f16x2(o[8 * i + 0], o[8 * i + 1]), to_f16x2(o[8 * i + 2], o[8 * i + 3]),
                     to_f16x2(o[8 * i + 4], o[8 * i + 5]), to_f16x2(o[8 * i + 6], o[8 * i + 7]));
}

// ---- CTA-pair (cta_group::2) helpers: cluster-scope barrier traffic and the paired MMA / commit -------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {  // the same shared-memory offset in CTA `rank` of the cluster
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ bool mbar_try_cluster(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {  // arrivals come from the peer CTA as well
    if (mbar_try_cluster(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_cluster(bar, parity)) {
        if (clock64() - t0 > 4000000000ll) __trap();
    }
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t dst_smem, uint32_t cols) {  // the same warp of BOTH CTAs of the pair
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// M = 256 over the CTA pair: each CTA's tensor core takes 128 A rows from its own shared memory and writes 128 lanes of its own
// TMEM; B's N rows are split in halves, the first from the leader's shared memory, the second from the peer's (same offsets)
__device__ __forceinline__ void mma_ss_pair(uint32_t d_tmem, uint32_t a_addr, uint32_t b_addr, uint32_t accumulate, uint32_t idesc) {
    const uint32_t a_lo = desc_lo(a_addr), a_hi = desc_hi(a_addr), b_lo = desc_lo(b_addr), b_hi = desc_hi(b_addr);
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "mov.b64 da, {%1, %2};\n\t"
        "mov.b64 db, {%3, %4};\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %5, p;\n\t}" ::"r"(d_tmem),
        "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {  // arrives on the barrier at this offset in BOTH CTAs
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"((uint16_t)3)
                 : "memory");
}
// one tap of the CTA-pair build: per K step a1 x [b1 ; b2] (N = 128: b1 from the leader, b2 from the peer) and a2 x b1 (N = 64: rows
// 0..31 of b1 from the leader, 32..63 from the peer, both at byte 8192 of the tap)
__device__ __forceinline__ void issue_tap_mmas_pair(bool elected, uint32_t dcol, uint32_t s_act, int row0, uint32_t b_tap, int ksteps, bool accumulate_first,
                                                    uint32_t a2_off) {
    constexpr uint32_t kIdesc128 = (1u << 4) | ((128u >> 3) << 17) | ((256u >> 4) << 24), kIdesc64 = (1u << 4) | ((64u >> 3) << 17) | ((256u >> 4) << 24);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (j < ksteps) {
            const uint32_t a_addr = s_act + (uint32_t)row0 * 128u + (uint32_t)j * 32u, b_addr = b_tap + (uint32_t)j * 32u;
            if (elected) {
                mma_ss_pair(dcol, a_addr, b_addr, (accumulate_first || j > 0) ? 1u : 0u, kIdesc128);
                mma_ss_pair(dcol + 64u, a_addr + a2_off, b_addr + 8192u, 1u, kIdesc64);
            }
        }
    }
}

// ---- the split-operand (f32-faithful) network, warp-specialised and software-pipelined over the two accumulators ------------------
// k_net_forward<f16, X3> issues a layer's MMAs, waits, runs the epilogue with the tensor pipe idle, synchronises the CTA and
// starts over: 63 % of its time is MMA issue (at the operand-fetch / tensor floor), the rest is exposed epilogue, barriers and
// waits, and neither TMEM (512 columns) nor shared memory (219 KB) leaves room for a second CTA to fill the gaps. Here the SAME
// geometry (7 boards, two 128-row accumulators, a1/a2 activation matrices, 3 x 3-tap weight ring) runs as a pipeline of roles:
//   warps 0-3 / 4-7  epilogue of accumulator 0 / 1 (one TMEM lane = one cell per thread, all 64 channels)
//   warp 8           helper of warp 4: channels 32..63 of cells 128..159 (the rows the next layer's accumulator 0 waits for)
//   warp 9           MMA issue (one elected lane): acc 0 of layer l, acc 1 of layer l, acc 0 of layer l + 1, ...
//   warp 10          weight producer (one lane)
// all connected by mbarriers (no CTA-wide barrier inside a board group). While accumulator 1's MMAs run, accumulator 0's epilogue
// runs; accumulator 0's MMAs of the next layer are queued right behind accumulator 1's (the drifting activation window below removes
// the write-after-read hazard of updating the activations in place) and wait for warp 4's rows only in front of their sixth tap.
// The history of the kernel -- what a per-layer timeline (-DONB_X3P_PROFILE) showed at each step and what each change bought, from
// 0.745 ms (plain build) to 0.514 ms -- is in DESIGN.md section 5b. Same products, same accumulation order, same results as
// k_net_forward<f16, X3>.
template <bool CL>
struct GeoX3PT {
    using G = Geo<true, true>;
    static constexpr int THREADS = 11 * 32;  // 8 epilogue warps, warp 8: helper of warp 4 (see the kernel), warp 9: MMA issue, warp 10: weights
    // CL (CTA pair, see below): a tap is [this CTA's 64 B rows of the N = 128 MMA][its 32 B rows of the N = 64 MMA]
    static constexpr int TAP_STRIDE = CL ? 12 * 1024 : G::TAP_STRIDE;
    static constexpr int NSLOT = G::NSLOT;
    static constexpr int SLOT_BYTES = G::TPS * TAP_STRIDE;
    // drifting activation window (see the kernel): layer l's activations start DRIFT_ROWS rows below layer l - 1's, for WRAP
    // layers in a row; the budget is what the weight ring leaves of the 227 KB
    static constexpr int DRIFT_ROWS = 8, WRAP = CL ? 16 : 7;
    static constexpr int R = G::R + DRIFT_ROWS * (WRAP - 1);
    static constexpr int ACT_BYTES = R * 128;  // f16 operands: 64 channels = one 128-byte block per row
    static constexpr int OFF_RING = G::NMAT * ACT_BYTES;
    static constexpr int OFF_HEAD = OFF_RING + NSLOT * SLOT_BYTES;
    static constexpr int OFF_HW = OFF_HEAD + G::HEAD_BYTES;  // CL: the head parameters, copied once (see k_net_forward_f16q)
    static constexpr int HW_BYTES = CL ? kHeadFloats * 4 : 0;
    static constexpr int OFF_BAR = OFF_HW + HW_BYTES;
    // mbarriers: full[3], empty[3], acc_full[2], rows_ready[3] (group 0 | warp 4 | warps 5-7), CL: peer_full[3]
    static constexpr int N_BARS = 2 * NSLOT + 2 + 3 + 2 + (CL ? NSLOT : 0);  // + heads_full, heads_free
    static constexpr int SMEM_USED = OFF_BAR + N_BARS * 8 + 16;
    static constexpr int SMEM = SMEM_USED;
    static_assert(SMEM_USED <= 227 * 1024, "shared memory");
    static_assert(Op<true>::KCH == 8 && ACT_BYTES % 1024 == 0, "one block per row; the ring stays aligned to the swizzle period");
};
using GeoX3P = GeoX3PT<false>;

//
// CL = true: the same pipeline on a PAIR of CTAs (a cluster of two SMs, tcgen05 cta_group::2). The kernel is bound by the tensor
// cores' operand fetch from shared memory (14 KB per K step and SM above); a paired MMA has M = 256 -- each SM contributes its own
// 128 activation rows and accumulates into its own TMEM -- while the weight rows are SPLIT between the two SMs' shared memories,
// so that each SM stores and fetches only half of B: 11 KB per step. Every CTA keeps its own 7 boards, epilogue warps, weight
// producer and weight ring (12 KB per tap: the leader holds b1 and b1[0:32], the peer b2 and b1[32:64]); only the leader's MMA warp
// issues MMAs. Cross-CTA traffic is barrier traffic only: the peer's epilogue threads arrive on the LEADER's rows barriers, the
// peer's warp 9 relays "my share of slot s has landed" to the leader's peer_full[s], and the leader's commits are multicast to the
// accumulator / empty barriers of both CTAs. Same products and accumulation order: results identical to the single-CTA build.
#ifdef ONB_X3P_PROFILE
__device__ long long s_tl[8][12];  // timeline of one board group (the 6th) of one CTA: [layer][event], see the printout at the kernel's end
__device__ long long s_t2[2][8];   // layer 4 of that group, per accumulator: wake, then (weights there, slot issued) x 3, commit issued
#endif
template <bool CL>
__global__ void __launch_bounds__(GeoX3P::THREADS, 1)
    k_net_forward_x3p(const float* __restrict__ planes, float* __restrict__ policy, float* __restrict__ value, int64_t n, NetDev net) {
    using G = Geo<true, true>;
    using GP = GeoX3PT<CL>;
    using O = Op<true>;
    constexpr int NACC = 2;
    constexpr int NB = G::NB, CELLS = G::CELLS, R = GP::R, NSLOT = GP::NSLOT, TPS = G::TPS, UPL = G::UPL;
    constexpr uint32_t A2 = (uint32_t)GP::ACT_BYTES, ACC = 128u, SET = (uint32_t)G::SET_COLS;
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t s_act = smem_u32(smem), s_ring = s_act + GP::OFF_RING, s_bar = s_act + GP::OFF_BAR;
    float* s_head = reinterpret_cast<float*>(smem + GP::OFF_HEAD);
    const float* s_hw = reinterpret_cast<const float*>(smem + GP::OFF_HW);
    auto HW = [&](int i) { return CL ? s_hw[i] : __ldg(net.head + i); };
    auto HW4 = [&](int i) { return CL ? reinterpret_cast<const float4*>(s_hw)[i] : __ldg(reinterpret_cast<const float4*>(net.head) + i); };
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + GP::OFF_BAR + GP::N_BARS * 8);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int L = 1 + 2 * net.n_blocks;
#ifdef ONB_X3P_PROFILE
#define TL(ev) do { if (blockIdx.x == (CL ? 2 : 3) && gi == 5 && l < 8) s_tl[l][ev] = clock64(); } while (0)
#define TL2(ev) do { if (blockIdx.x == (CL ? 2 : 3) && gi == 5 && l == 4 && lane == 0) s_t2[a][ev] = clock64(); } while (0)
#else
#define TL(ev) do { } while (0)
#define TL2(ev) do { } while (0)
#endif
    // CL: the pair works on two consecutive board groups at a time (leader 2 p, peer 2 p + 1; a group past the end computes on zeros
    // and stores nothing), so both CTAs run the same number of rounds
    const uint32_t crank = CL ? cluster_ctarank() : 0u;
    const int64_t n_groups = CL ? ((n + NB - 1) / NB + 1) / 2 : (n + NB - 1) / NB;  // CL: pairs of groups
    const int64_t worker = CL ? (int64_t)(blockIdx.x >> 1) : (int64_t)blockIdx.x, n_workers = CL ? (int64_t)(gridDim.x >> 1) : (int64_t)gridDim.x;
    if (worker >= n_groups) return;  // whole CTA (pair), before any allocation
    const int64_t my_groups = (n_groups - worker + n_workers - 1) / n_workers;
    const uint32_t total_units = (uint32_t)my_groups * (uint32_t)(UPL * L);
    auto bar_full = [&](uint32_t s) { return s_bar + s * 8u; };
    auto bar_empty = [&](uint32_t s) { return s_bar + (NSLOT + s) * 8u; };
    auto bar_acc = [&](uint32_t a) { return s_bar + (2 * NSLOT + a) * 8u; };
    auto bar_rows = [&](uint32_t k) { return s_bar + (2 * NSLOT + 2 + k) * 8u; };  // 0: group 0, 1: warp 4, 2: warps 5-7
    const uint32_t bar_hfull = s_bar + (2 * NSLOT + 5) * 8u, bar_hfree = bar_hfull + 8u;  // s_head written by every cell | read by every head
    auto bar_peer = [&](uint32_t s) { return s_bar + (2 * NSLOT + 7 + s) * 8u; };  // CL, leader's: the peer's share of slot s has landed

    if (tid == 0) {
        for (uint32_t s = 0; s < (uint32_t)NSLOT; ++s) {
            mbar_init(bar_full(s), 1);
            mbar_init(bar_empty(s), 1);
            if (CL) mbar_init(bar_peer(s), 1);
        }
        mbar_init(bar_acc(0), 1);
        mbar_init(bar_acc(1), 1);
        mbar_init(bar_rows(0), CL ? 256 : 128);  // CL: the leader's rows barriers collect the epilogue threads of both CTAs
        mbar_init(bar_rows(1), CL ? 128 : 64);  // warp 4 and its helper
        mbar_init(bar_rows(2), CL ? 192 : 96);
        mbar_init(bar_hfull, 256);
        mbar_init(bar_hfree, 256);
        fence_barrier_init();
    }
    if (warp == 0) {
        if (CL)
            tmem_alloc_pair(smem_u32(s_tmem), G::TMEM_COLS);
        else
            tmem_alloc(smem_u32(s_tmem), G::TMEM_COLS);
    }
    for (int i = tid; i < G::NMAT * GP::ACT_BYTES / 16; i += GeoX3P::THREADS) st_shared_v4(s_act + i * 16, 0u, 0u, 0u, 0u);
    if (CL)
        for (int i = tid; i < kHeadFloats / 4; i += GeoX3P::THREADS)
            reinterpret_cast<float4*>(smem + GP::OFF_HW)[i] = __ldg(reinterpret_cast<const float4*>(net.head) + i);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    if (CL) cluster_sync_all();  // the peer's barriers are initialised before anything arrives on them
    tc_fence_after();
    const uint32_t tmem = *s_tmem;
    // CL: rows barriers live in the leader; every epilogue thread of the pair arrives there with cluster scope
    const uint32_t rows_base = CL ? mapa_shared(bar_rows(0), 0u) : bar_rows(0);
    auto arrive = [&](uint32_t bar) {
        if (CL)
            mbar_arrive_cluster(rows_base + (bar - bar_rows(0)));
        else
            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
    };

    // Drifting activation window. Updating the activations in place has a write-after-read hazard: rows 121..127 of layer l are
    // still read by accumulator 1's MMAs (their windows shift by up to -7 rows) when their owners want to store layer l + 1, and the
    // next layer's accumulator 0 needs exactly those rows, so the tensor pipe drained at every layer boundary while warp 3 waited and
    // stored (a quarter of the layer time in the first pipelined build). Here layer l + 1 is written 8 rows (one swizzle period)
    // BELOW layer l: accumulator 0's owners then write over rows -8..119 of layer l, which accumulator 1 never reads, and the next
    // layer's MMAs are queued behind the current one's with no wait in between. Because the layers slide over each other, zero
    // rows and pad cells no longer keep themselves: pad cells are stored as zeros and the 8 rows before / 8 + 4 rows after the
    // cells are cleared for every layer. After WRAP layers the window jumps back to the top; that one transition does overlap what
    // accumulator 1 reads, and accumulator 0's owners wait for it (as all layer boundaries used to).
    auto base_row = [&](int l) { return kLead + GP::DRIFT_ROWS * (GP::WRAP - 1 - (l % GP::WRAP)); };
    auto zero_rows = [&](int row) {  // 8 rows of both matrices, by one warp
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int idx = lane * 4 + k;  // matrix (1 bit) | row (3 bits) | chunk (3 bits)
            st_shared_v4(s_act + (uint32_t)(idx >> 6) * A2 + (uint32_t)(row + ((idx >> 3) & 7)) * 128u + (uint32_t)(idx & 7) * 16u, 0u, 0u, 0u, 0u);
        }
    };

    if (warp == 10) {
        // ---- weight producer: the ring is filled strictly in tap order, as far ahead as it has free slots
        if (lane == 0) {
            for (uint32_t u = 0; u < total_units; ++u) {
                const uint32_t slot = u % NSLOT, use = u / NSLOT;
                if (use >= 1) mbar_wait(bar_empty(slot), (use - 1u) & 1u);
                const uint32_t ul = u % (uint32_t)(UPL * L), layer = ul / UPL, tap = (ul - layer * UPL) * TPS;
                const uint8_t* src = CL ? net.wpair + ((size_t)crank * (size_t)(9 * L) + (size_t)layer * 9 + tap) * (size_t)GP::TAP_STRIDE
                                        : net.wconv + (size_t)G::NMAT * (layer == 0 ? (size_t)tap * O::TAP_BYTES0
                                                                                    : (size_t)9 * O::TAP_BYTES0 + ((size_t)(layer - 1) * 9 + tap) * O::TAP_BYTES);
                const uint32_t bytes = CL ? (uint32_t)GP::SLOT_BYTES : (uint32_t)(TPS * G::NMAT) * (layer == 0 ? O::TAP_BYTES0 : O::TAP_BYTES);
                mbar_expect_tx(bar_full(slot), bytes);
                bulk_g2s(s_ring + slot * (uint32_t)GP::SLOT_BYTES, src, bytes, bar_full(slot));
            }
        }
    } else if (CL && warp == 9 && crank != 0u) {
        // ---- peer CTA: no MMA issue here; relay "this CTA's share of the slot has landed" to the leader
        if (lane == 0) {
            const uint32_t peer0 = mapa_shared(bar_peer(0), 0u);
            for (uint32_t u = 0; u < total_units; ++u) {
                const uint32_t slot = u % NSLOT, use = u / NSLOT;
                mbar_wait(bar_full(slot), use & 1u);
                mbar_arrive_cluster(peer0 + slot * 8u);
            }
        }
    } else if (warp == 9) {
        // ---- MMA issue (the whole warp runs the loop so that descriptors stay in uniform registers; one elected lane issues)
        const bool elected = elect_one();
        uint32_t q0 = 0, stage = 0;  // stage = number of "rows ready" rounds consumed so far (input stage + epilogues)
        int gl = 0;                  // layers issued so far, over all board groups: the activation window keeps drifting across groups
#ifdef ONB_X3P_PROFILE
        long long t_rows0 = 0, t_rows0b = 0, t_rows1 = 0, t_full = 0, t_issue = 0, t_mark = clock64();
#define XP(var) do { const long long now__ = clock64(); var += now__ - t_mark; t_mark = now__; } while (0)
#else
#define XP(var) do { } while (0)
#endif
        for (int64_t gi = 0; gi < my_groups; ++gi) {
            for (int l = 0; l < L; ++l) {
                const bool use_s = l >= 2 && (l & 1) == 0;
                const uint32_t dcol = tmem + (use_s ? SET : 0u);
                const int ksteps = l == 0 ? O::KCH0 / 2 : O::KCH / 2;
#pragma unroll 1
                for (int a = 0; a < NACC; ++a) {
                    // accumulator 0 needs its own rows and, from its sixth tap on, the first rows of accumulator 1: taps 0..4 shift
                    // the window by -7, -6, -5, -1, 0 rows and stay inside rows 0..127, taps 5..8 (+1, +5, +6, +7) reach up to row
                    // 134 (warp 4's cells). Accumulator 1 needs the rest as well. The MMA queue is shallow: every barrier test that
                    // sits between two taps drains it, so all tests that can be made early are made while MMAs are queued -- the
                    // next slot's weights after the first tap of a slot, accumulator 1's rows during accumulator 0's last slot -- and
                    // accumulator 1 re-tests nothing (the same thread saw the same weights arrive for accumulator 0)
                    XP(t_issue);
                    if (a == 0) {
                        if (CL) mbar_wait_cluster(bar_rows(0), stage & 1u); else mbar_wait(bar_rows(0), stage & 1u);
                        XP(t_rows0);
                        if (lane == 0) TL(0);
                        tc_fence_after();
                    } else {
                        if (lane == 0) TL(2);
                    }
                    TL2(0);
                    auto wait_weights = [&](uint32_t uu) {
                        const uint32_t sl = uu % NSLOT, us = uu / NSLOT;
                        XP(t_issue);
                        mbar_wait(bar_full(sl), us & 1u);
                        if (CL) mbar_wait_cluster(bar_peer(sl), us & 1u);
                        XP(t_full);
                    };
                    if (a == 0) wait_weights(q0);
                    // descriptor low words (see mma_lo): this accumulator's window of the current layer, the second activation matrix,
                    // and per slot the weights; the slot loop is unrolled so that a tap's shift and tests are compile-time constants
                    const uint32_t d_acc = dcol + (uint32_t)a * ACC;
                    const uint32_t a_acc_lo = desc_lo(s_act) + (uint32_t)((base_row(gl) + a * 128) * 8);  // 128-byte rows: 8 per row in the address field
                    constexpr uint32_t kA2Lo = A2 >> 4;
                    constexpr uint32_t kPair128 = (1u << 4) | ((128u >> 3) << 17) | ((256u >> 4) << 24), kPair64 = (1u << 4) | ((64u >> 3) << 17) | ((256u >> 4) << 24);
#pragma unroll
                    for (int g = 0; g < UPL; ++g) {
                        const uint32_t u = q0 + g, slot = u % NSLOT;
                        const uint32_t b_slot_lo = desc_lo(s_ring) + slot * (uint32_t)(GP::SLOT_BYTES >> 4);
                        TL2(1 + 2 * g);
#pragma unroll
                        for (int tt = 0; tt < TPS; ++tt) {
                            const int t = g * TPS + tt;
                            if (a == 0 && t == 5) {  // the first window that reaches into accumulator 1's rows (see above)
                                XP(t_issue);
                                if (CL) mbar_wait_cluster(bar_rows(1), stage & 1u); else mbar_wait(bar_rows(1), stage & 1u);
                                XP(t_rows0b);
                                tc_fence_after();
                            }
                            // per K step: a1 x [b1 ; b2] (N = 128) into D1 | D2, then a2 x b1 (N = 64) onto D2 (issue_tap_mmas / _pair)
                            const uint32_t a_lo = a_acc_lo + (uint32_t)(((t / 3 - 1) * 6 + (t % 3 - 1)) * 8);
                            const uint32_t b_lo = b_slot_lo + (uint32_t)(tt * (GP::TAP_STRIDE >> 4));
                            if (elected) {
#pragma unroll
                                for (int j = 0; j < 4; ++j)
                                    if (j < ksteps) {
                                        const uint32_t accum = (use_s || t > 0 || j > 0) ? 1u : 0u;
                                        if (CL) {
                                            mma_lo<true>(d_acc, a_lo + 2u * j, b_lo + 2u * j, accum, kPair128);
                                            mma_lo<true>(d_acc + 64u, a_lo + kA2Lo + 2u * j, b_lo + (8192u >> 4) + 2u * j, 1u, kPair64);
                                        } else {
                                            mma_lo<false>(d_acc, a_lo + 2u * j, b_lo + 2u * j, accum, O::IDESC_N128);
                                            mma_lo<false>(d_acc + 64u, a_lo + kA2Lo + 2u * j, b_lo + 2u * j, 1u, O::IDESC);
                                        }
                                    }
                            }
                            if (a == 0 && tt == 0) {
                                if (g + 1 < UPL) {
                                    wait_weights(u + 1);
                                } else {  // accumulator 1's turn comes next: its rows (warps 5-7 of the previous stage) are long written
                                    XP(t_issue);
                                    if (CL) mbar_wait_cluster(bar_rows(2), stage & 1u); else mbar_wait(bar_rows(2), stage & 1u);
                                    XP(t_rows1);
                                    tc_fence_after();
                                }
                            }
                        }
                        if (a == NACC - 1 && elected) {  // both accumulators' MMAs have read the slot
                            if (CL) umma_commit_pair(bar_empty(slot)); else umma_commit(bar_empty(slot));
                        }
                        TL2(2 + 2 * g);
                    }
                    if (elected) {
                        if (CL) umma_commit_pair(bar_acc(a)); else umma_commit(bar_acc(a));
                    }
                    if (lane == 0) TL(a == 0 ? 1 : 3);
                    TL2(7);
                }
                q0 += (uint32_t)UPL;
                stage += 1;
                gl = gl + 1 == GP::WRAP ? 0 : gl + 1;
            }
        }
#ifdef ONB_X3P_PROFILE
        XP(t_issue);
        if (blockIdx.x == (CL ? 2 : 3) && lane == 0)
            printf("x3p MMA warp, %lld groups: issue %lld, waiting rows for acc0 %lld (+ %lld before tap 5), for acc1 %lld, waiting weights %lld\n",
                   (long long)my_groups, t_issue, t_rows0, t_rows0b, t_rows1, t_full);
#endif
    } else {
        // ---- epilogue warps: group a = warp >> 2 owns accumulator a; this thread owns one cell (TMEM lane) and its 64 channels
        // Warp 8 is the HELPER of warp 4: the cycle "accumulator 1 done -> warp 4's epilogue -> accumulator 0's taps 5..8 of the next
        // layer -> accumulator 1's MMAs" is what paces a layer once everything else overlaps (timeline: ~ 900 idle tensor cycles per
        // layer in front of tap 5), and a warp's epilogue is a latency chain, not a throughput problem. Warp 8 sits on the same TMEM
        // lane quarter as warp 4 (warp id % 4 == 0) and takes channels 32..63 of cells 128..159, warp 4 keeps channels 0..31: the
        // rows the next accumulator 0 waits for arrive in half the time. The last layer (heads: a sequential sum over all 64
        // channels) stays with warp 4 alone.
        const bool helper = warp == 8;
        const int a = helper ? 1 : warp >> 2;
        const int cell = helper ? 128 + lane : a * 128 + (warp & 3) * 32 + lane;
        const Cell c = decode_cell(cell, CELLS);
        const uint32_t my_rows = a == 0 ? bar_rows(0) : ((warp == 4 || helper) ? bar_rows(1) : bar_rows(2));
        const uint32_t tlane = tmem + ((uint32_t)((warp & 3) * 32) << 16);
        uint32_t acc_par = 0;  // parity of the layer counter (both accumulator barriers complete once per layer)
#ifdef ONB_X3P_PROFILE
        long long e_wait = 0, e_work = 0, e_halo = 0, e_mark = clock64();
#define EP(var) do { const long long now__ = clock64(); var += now__ - e_mark; e_mark = now__; } while (0)
#else
#define EP(var) do { } while (0)
#endif
        auto group_board0 = [&](int64_t g) { return CL ? (2 * (worker + g * n_workers) + (int64_t)crank) * NB : ((int64_t)blockIdx.x + g * gridDim.x) * NB; };
        // input planes -> channel chunks of both activation matrices (create_tensor_from_state layout [21][5][5]); pad cells and
        // planes 21..31 are zero. The loads of the NEXT group are issued before the last layer's accumulator wait and stored from that
        // layer's epilogue (it is simply the next stop of the drifting window), so the next group's MMAs queue up behind this one's
        // while the heads are computed.
        float xin[kInPlanes];
        auto load_input = [&](int64_t g) {
            const int64_t gb = group_board0(g) + c.board;
            const float* src = planes + gb * 525 + c.pos;
#pragma unroll
            for (int ch = 0; ch < kInPlanes; ++ch) xin[ch] = (c.real && g < my_groups && gb < n) ? __ldg(src + ch * 25) : 0.f;
        };
        auto store_input = [&](int row) {
            float x[32];
#pragma unroll
            for (int ch = 0; ch < 32; ++ch) x[ch] = ch < kInPlanes ? xin[ch] : 0.f;
            store_channels_x3(s_act, A2, R, row + cell, 0, x);
        };
        // heads of one board group: one warp per board (ph_linear2 + softmax, vh_linear1 + ReLU + vh_linear2 + tanh) from the 1x1
        // convolution outputs the last layer's epilogue left in s_head. They are computed where the epilogue warps have slack -- after
        // the second layer's epilogue of the NEXT group (its first layer has half the MMAs, its epilogue is already late) -- and right
        // after the last layer only for the last group
        auto local_arrive = [&](uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); };
        auto run_heads = [&](int64_t hb0, uint32_t parity) {
            mbar_wait(bar_hfull, parity);  // every cell's 1x1 outputs of that group are in s_head (no CTA-wide barrier: the two groups are a phase apart)
            for (int b = warp; b < NB; b += 8) {
                const int64_t gb = hb0 + b;
                if (gb >= n) continue;
                const float* hb = s_head + b * 75;
                const bool two = lane + 32 < 50;
                float l0 = HW(kPhB + lane), l1 = two ? HW(kPhB + 32 + lane) : 0.f;
#pragma unroll 10
                for (int i = 0; i < 50; ++i) {
                    const float x = hb[i];
                    l0 = fmaf(x, HW(kPhW + i * 50 + lane), l0);
                    if (two) l1 = fmaf(x, HW(kPhW + i * 50 + 32 + lane), l1);
                }
                const float m = warp_max(two ? fmaxf(l0, l1) : l0);
                const float e0 = expf(l0 - m), e1 = two ? expf(l1 - m) : 0.f;
                const float s = warp_sum(e0 + e1);
                policy[gb * 50 + lane] = e0 / s;
                if (two) policy[gb * 50 + 32 + lane] = e1 / s;
                float h0 = HW(kV1B + lane), h1 = HW(kV1B + 32 + lane);
#pragma unroll 5
                for (int i = 0; i < 25; ++i) {
                    const float x = hb[50 + i];
                    h0 = fmaf(x, HW(kV1W + i * 64 + lane), h0);
                    h1 = fmaf(x, HW(kV1W + i * 64 + 32 + lane), h1);
                }
                float acc = fmaf(fmaxf(h0, 0.f), HW(kV2W + lane), fmaxf(h1, 0.f) * HW(kV2W + 32 + lane));
                acc = warp_sum(acc);
                if (lane == 0) value[gb] = tanhf(acc + HW(kV2B));
            }
            local_arrive(bar_hfree);  // s_head may be overwritten by the next last-layer epilogue once every thread has said so
        };
        int gl = 0;  // layers done so far modulo WRAP, over all board groups (the MMA warp counts the same)
        if (!helper) {
            load_input(0);
            store_input(base_row(0));
        }
        if (warp == 0) zero_rows(base_row(0) - 8);
        if (warp == 7) zero_rows(base_row(0) + 256);
        fence_proxy_async();
        arrive(my_rows);
        for (int64_t gi = 0; gi < my_groups; ++gi) {
            const int64_t board0 = group_board0(gi);
            for (int l = 0; l < L; ++l) {
                const bool use_s = l >= 2 && (l & 1) == 0;  // second convolution of a block accumulates onto the parked residual
                const bool last = l == L - 1;
                const bool feeds = !last || gi + 1 < my_groups;  // this epilogue writes the next stop of the window (layer or input)
                if (last && feeds && !helper) load_input(gi + 1);
                EP(e_work);
                mbar_wait(bar_acc(a), acc_par);
                EP(e_wait);
                if (tid == 0) TL(4);
                if (tid == 128) TL(6);
                if (tid == 224) TL(8);
                tc_fence_after();
                const int rn = base_row(gl + 1);  // where the next layer's activations (or the next group's input) go
                if (feeds) {
                    if (a == 0 && gl + 1 == GP::WRAP) {  // the window jumps back up, over rows accumulator 1's MMAs may still read
                        EP(e_work);
                        mbar_wait(bar_acc(1), acc_par);
                        EP(e_halo);
                    }
                    if (warp == 0) zero_rows(rn - 8);
                    if (warp == 7) zero_rows(rn + 256);
                }
                const bool preload = (l & 1) == 0 && !last;  // this layer's output is a block input: park it (+ next bias) in TMEM
                const float4* bias_l = reinterpret_cast<const float4*>(net.bias + (size_t)l * 64);
                const float4* bias_n = reinterpret_cast<const float4*>(net.bias + (size_t)(preload ? l + 2 : l) * 64);
                const uint32_t tsrc = tlane + (use_s ? SET : 0u) + a * ACC;
                const uint32_t tskip = tlane + SET + a * ACC;
                float hp0 = 0.f, hp1 = 0.f, hv = 0.f;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    // warp 4 and its helper share cells 128..159 by channel halves, except in the last layer (warp 4 alone)
                    if (helper ? (last || h == 0) : (warp == 4 && !last && h == 1)) continue;
                    uint32_t v[32];
                    {
                        uint32_t v2[32];
                        tmem_ld32_nowait(tsrc + h * 32, v);
                        tmem_ld32_nowait(tsrc + 64 + h * 32, v2);
                        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                        for (int i = 0; i < 32; ++i) v[i] = __float_as_uint(fmaf(__uint_as_float(v2[i]), kX3InvScale, __uint_as_float(v[i])));
                    }
                    float o[32];
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (!use_s) b = __ldg(bias_l + h * 8 + i);
                        o[4 * i + 0] = fmaxf(__uint_as_float(v[4 * i + 0]) + b.x, 0.f);
                        o[4 * i + 1] = fmaxf(__uint_as_float(v[4 * i + 1]) + b.y, 0.f);
                        o[4 * i + 2] = fmaxf(__uint_as_float(v[4 * i + 2]) + b.z, 0.f);
                        o[4 * i + 3] = fmaxf(__uint_as_float(v[4 * i + 3]) + b.w, 0.f);
                    }
                    if (!last) {
                        if (!c.real) {  // pad cells are stored too, as zeros (their accumulators hold sums that mean nothing)
#pragma unroll
                            for (int i = 0; i < 32; ++i) o[i] = 0.f;
                        }
                        store_channels_x3(s_act, A2, R, rn + cell, h * 32, o);
                    }
                    if (preload) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const float4 b = __ldg(bias_n + h * 8 + i);
                            v[4 * i + 0] = __float_as_uint(o[4 * i + 0] + b.x);
                            v[4 * i + 1] = __float_as_uint(o[4 * i + 1] + b.y);
                            v[4 * i + 2] = __float_as_uint(o[4 * i + 2] + b.z);
                            v[4 * i + 3] = __float_as_uint(o[4 * i + 3] + b.w);
                        }
                        tmem_st32(tskip + h * 32, v);
#pragma unroll
                        for (int i = 0; i < 32; ++i) v[i] = 0u;  // the D2 half of the preloaded accumulator starts from zero
                        tmem_st32(tskip + 64 + h * 32, v);
                    }
                    if (last) {  // 1x1 convolutions of both heads (net.rs: policy_conv 64 -> 2, vh_conv 64 -> 1)
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const float4 w0 = HW4((kHP0 / 4) + h * 8 + i), w1 = HW4((kHP1 / 4) + h * 8 + i),
                                         w2 = HW4((kHV / 4) + h * 8 + i);
                            hp0 = fmaf(o[4 * i + 0], w0.x, fmaf(o[4 * i + 1], w0.y, fmaf(o[4 * i + 2], w0.z, fmaf(o[4 * i + 3], w0.w, hp0))));
                            hp1 = fmaf(o[4 * i + 0], w1.x, fmaf(o[4 * i + 1], w1.y, fmaf(o[4 * i + 2], w1.z, fmaf(o[4 * i + 3], w1.w, hp1))));
                            hv = fmaf(o[4 * i + 0], w2.x, fmaf(o[4 * i + 1], w2.y, fmaf(o[4 * i + 2], w2.z, fmaf(o[4 * i + 3], w2.w, hv))));
                        }
                    }
                }
                if (last && !helper) {
                    if (gi > 0) mbar_wait(bar_hfree, (uint32_t)(gi - 1) & 1u);  // the previous group's heads are done with s_head
                    if (c.real) {
                        float* hb = s_head + c.board * 75;
                        hb[c.pos] = fmaxf(hp0 + HW(kHB + 0), 0.f);
                        hb[25 + c.pos] = fmaxf(hp1 + HW(kHB + 1), 0.f);
                        hb[50 + c.pos] = fmaxf(hv + HW(kHB + 2), 0.f);
                    }
                    local_arrive(bar_hfull);
                }
                if (preload) tmem_wait_st();
                if (last && feeds && !helper) store_input(rn);
                if (feeds) {
                    fence_proxy_async();
                    tc_fence_before();
                    arrive(my_rows);  // this thread's rows (and its TMEM reads) of the layer are done
                    if (tid == 0) TL(5);
                    if (tid == 128) TL(7);
                    if (tid == 224) TL(9);
                    if (tid == 127) TL(10);
                }
                if (l == 1 && L >= 3 && gi > 0 && !helper) run_heads(group_board0(gi - 1), (uint32_t)(gi - 1) & 1u);
                acc_par ^= 1u;
                gl = gl + 1 == GP::WRAP ? 0 : gl + 1;
            }
            if ((L < 3 || gi + 1 == my_groups) && !helper) run_heads(board0, (uint32_t)gi & 1u);
        }
#ifdef ONB_X3P_PROFILE
        EP(e_work);
        if (blockIdx.x == (CL ? 2 : 3) && (tid == 0 || tid == 127 || tid == 128 || tid == 160))
            printf("x3p epilogue tid %d: waiting for the accumulator %lld, halo wait %lld, work (input, epilogue, heads) %lld\n", tid, e_wait, e_halo, e_work);
#endif
    }
    __syncwarp();
    tc_fence_before();
    __syncthreads();
#ifdef ONB_X3P_PROFILE
    if (blockIdx.x == (CL ? 2 : 3) && tid == 0 && my_groups > 5)
        for (int l = 0; l < L && l < 8; ++l)
            printf("layer %d: MMA wakes for acc0 %6lld, acc0 issued %6lld, wakes for acc1 %6lld, acc1 issued %6lld | acc0 done %6lld, warp 0 arrives %6lld, halo thread arrives %6lld | "
                   "acc1 done %6lld, warp 4 arrives %6lld, warp 7 arrives %6lld\n", l, s_tl[l][0] - s_tl[0][0], s_tl[l][1] - s_tl[0][0], s_tl[l][2] - s_tl[0][0],
                   s_tl[l][3] - s_tl[0][0], s_tl[l][4] - s_tl[0][0], s_tl[l][5] - s_tl[0][0], s_tl[l][10] - s_tl[0][0], s_tl[l][6] - s_tl[0][0],
                   s_tl[l][7] - s_tl[0][0], s_tl[l][9] - s_tl[0][0]);
    if (blockIdx.x == (CL ? 2 : 3) && tid == 0 && my_groups > 5)
        for (int a = 0; a < 2; ++a)
            printf("layer 4 acc %d: wake 0 | slot 0 weights %lld issued %lld | slot 1 weights %lld issued %lld | slot 2 weights %lld issued %lld | commit %lld\n", a,
                   s_t2[a][1] - s_t2[a][0], s_t2[a][2] - s_t2[a][0], s_t2[a][3] - s_t2[a][0], s_t2[a][4] - s_t2[a][0], s_t2[a][5] - s_t2[a][0],
                   s_t2[a][6] - s_t2[a][0], s_t2[a][7] - s_t2[a][0]);
#endif
    if (CL) {
        cluster_sync_all();  // neither CTA leaves (or frees TMEM) while the other may still signal its barriers
        if (warp == 0) tmem_dealloc_pair(tmem, G::TMEM_COLS);
    } else if (warp == 0) {
        tmem_dealloc(tmem, G::TMEM_COLS);
    }
}

// ---- the f16 fast mode as ONE CTA per SM with FOUR accumulators: the pipeline of k_net_forward_x3p with everything it learned ------
// 14 boards (504 cells) per pass in four 128-row accumulators (TMEM: 4 x 64 columns x {plain, residual-preloaded} = 512), sixteen
// epilogue warps (four per accumulator, 16 channels at a time: 576 threads leave 113 registers), one MMA warp, one weight warp.
// The MMAs of a layer are issued accumulator after accumulator; accumulator a's epilogue has the other three accumulators' MMAs to
// hide under. Taken over from k_net_forward_x3p: the drifting activation window (no write-after-read wait at layer boundaries, also
// across board groups), the wait for the next accumulator's first warp only in front of tap 5, barrier tests behind queued MMAs,
// the next group's input stored from the last layer's epilogue, heads computed in the next group's slack, and CL = CTA pairs
// (tcgen05 cta_group::2: each SM keeps rows 32 r .. 32 r + 31 of every tap, 4 KB instead of 8 KB). Twice the boards per weight pass
// of the two-CTAs-per-SM builds (and a quarter of their weight bytes per SM with CL): the L2 -> SM weight stream was 55 % of their
// time. Same products, accumulation order and head sums as k_net_forward<f16>: bit-identical results.
#ifdef ONB_F16Q_PROFILE
__device__ long long q_tl[8][4][4];  // [layer][accumulator][issue start, issue end, accumulator done (first warp of its group), that warp arrives]
#define QTL(l_, a_, e_) do { if (blockIdx.x == 2 && gi == 3 && (l_) < 8) q_tl[l_][a_][e_] = clock64(); } while (0)
#else
#define QTL(l_, a_, e_) do { } while (0)
#endif
template <bool CL>
struct GeoF16Q {
    static constexpr int NACC = 4, NB = 14, CELLS = NB * kCellsPerBoard;  // 504 of 512 rows
    static constexpr int EPI_WARPS = 4 * NACC, THREADS = (EPI_WARPS + 2) * 32;
    static constexpr int DRIFT_ROWS = 8, WRAP = CL ? 12 : 8;
    static constexpr int R = kLead + NACC * 128 + kTrail + DRIFT_ROWS * (WRAP - 1);
    static constexpr int ACT_BYTES = R * 128;
    static constexpr int TAP_STRIDE = CL ? 4096 : 8192;
    // the ring holds TWO layers: a slot is free again only when the LAST accumulator has read it, a third of an accumulator's MMAs
    // before the next layer's first accumulator wants its successor -- with one layer of slots every layer waited for weights
    static constexpr int TPS = 3, UPL = 3, NSLOT = 6;
    static constexpr int SLOT_BYTES = TPS * TAP_STRIDE;
    static constexpr int OFF_RING = ACT_BYTES;
    static constexpr int OFF_HEAD = OFF_RING + NSLOT * SLOT_BYTES;
    static constexpr int HEAD_BYTES = ((NB * 75 * 4 + 15) / 16) * 16;
    static constexpr int OFF_HW = OFF_HEAD + HEAD_BYTES;                 // CL (room to spare): the head parameters, copied once
    static constexpr int HW_BYTES = CL ? kHeadFloats * 4 : 0;
    static constexpr int OFF_BAR = OFF_HW + HW_BYTES;
    // mbarriers: full[6], empty[6], acc[4], rows_first[4] (first warp of a group), rows_rest[4], heads_full, heads_free, CL: peer_full[6]
    static constexpr int N_BARS = 2 * NSLOT + 3 * NACC + 2 + (CL ? NSLOT : 0);
    static constexpr int SMEM = OFF_BAR + N_BARS * 8 + 16;
    static constexpr int SET_COLS = NACC * 64, TMEM_COLS = 2 * SET_COLS;
    static_assert(ACT_BYTES % 1024 == 0 && SMEM <= 227 * 1024 && TMEM_COLS == 512, "geometry");
};

template <bool CL>
__global__ void __launch_bounds__(GeoF16Q<CL>::THREADS, 1)
    k_net_forward_f16q(const float* __restrict__ planes, float* __restrict__ policy, float* __restrict__ value, int64_t n, NetDev net) {
    using GP = GeoF16Q<CL>;
    using O = Op<true>;
    constexpr int NACC = GP::NACC, NB = GP::NB, CELLS = GP::CELLS, R = GP::R, NSLOT = GP::NSLOT, TPS = GP::TPS, UPL = GP::UPL, EW = GP::EPI_WARPS;
    constexpr uint32_t ACC = 64u, SET = (uint32_t)GP::SET_COLS;
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t s_act = smem_u32(smem), s_ring = s_act + GP::OFF_RING, s_bar = s_act + GP::OFF_BAR;
    float* s_head = reinterpret_cast<float*>(smem + GP::OFF_HEAD);
    // head parameters: from shared memory in the pair build (the fully connected heads are latency chains of ~ 150 loads per lane; out
    // of L1 / L2 one board cost a warp ~ 5 000 cycles), from global memory where the weight ring leaves no room
    const float* s_hw = reinterpret_cast<const float*>(smem + GP::OFF_HW);
    auto HW = [&](int i) { return CL ? s_hw[i] : __ldg(net.head + i); };
    auto HW4 = [&](int i) { return CL ? reinterpret_cast<const float4*>(s_hw)[i] : __ldg(reinterpret_cast<const float4*>(net.head) + i); };
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + GP::OFF_BAR + GP::N_BARS * 8);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int L = 1 + 2 * net.n_blocks;
    const uint32_t crank = CL ? cluster_ctarank() : 0u;
    const int64_t n_groups = CL ? ((n + NB - 1) / NB + 1) / 2 : (n + NB - 1) / NB;  // CL: pairs of groups (leader 2 p, peer 2 p + 1)
    const int64_t worker = CL ? (int64_t)(blockIdx.x >> 1) : (int64_t)blockIdx.x, n_workers = CL ? (int64_t)(gridDim.x >> 1) : (int64_t)gridDim.x;
    if (worker >= n_groups) return;  // whole CTA (pair), before any allocation
    const int64_t my_groups = (n_groups - worker + n_workers - 1) / n_workers;
    const uint32_t total_units = (uint32_t)my_groups * (uint32_t)(UPL * L);
    auto bar_full = [&](uint32_t s) { return s_bar + s * 8u; };
    auto bar_empty = [&](uint32_t s) { return s_bar + (NSLOT + s) * 8u; };
    auto bar_acc = [&](uint32_t a) { return s_bar + (2 * NSLOT + a) * 8u; };
    auto bar_first = [&](uint32_t a) { return s_bar + (2 * NSLOT + NACC + a) * 8u; };      // rows of the first warp of group a
    auto bar_rest = [&](uint32_t a) { return s_bar + (2 * NSLOT + 2 * NACC + a) * 8u; };   // rows of its other three warps
    const uint32_t bar_hfull = s_bar + (2 * NSLOT + 3 * NACC) * 8u, bar_hfree = bar_hfull + 8u;  // s_head written by every cell | read by every head
    auto bar_peer = [&](uint32_t s) { return s_bar + (2 * NSLOT + 3 * NACC + 2 + s) * 8u; };   // CL, leader's: the peer's share of slot s landed

    if (tid == 0) {
        for (uint32_t s = 0; s < (uint32_t)NSLOT; ++s) {
            mbar_init(bar_full(s), 1);
            mbar_init(bar_empty(s), 1);
            if (CL) mbar_init(bar_peer(s), 1);
        }
        for (uint32_t a = 0; a < (uint32_t)NACC; ++a) {
            mbar_init(bar_acc(a), 1);
            mbar_init(bar_first(a), CL ? 64 : 32);  // CL: the leader's rows barriers collect the epilogue threads of both CTAs
            mbar_init(bar_rest(a), CL ? 192 : 96);
        }
        mbar_init(bar_hfull, EW * 32);
        mbar_init(bar_hfree, EW * 32);
        fence_barrier_init();
    }
    if (warp == 0) {
        if (CL)
            tmem_alloc_pair(smem_u32(s_tmem), GP::TMEM_COLS);
        else
            tmem_alloc(smem_u32(s_tmem), GP::TMEM_COLS);
    }
    for (int i = tid; i < GP::ACT_BYTES / 16; i += GP::THREADS) st_shared_v4(s_act + i * 16, 0u, 0u, 0u, 0u);
    if (CL)
        for (int i = tid; i < kHeadFloats / 4; i += GP::THREADS)
            reinterpret_cast<float4*>(smem + GP::OFF_HW)[i] = __ldg(reinterpret_cast<const float4*>(net.head) + i);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    if (CL) cluster_sync_all();  // the peer's barriers are initialised before anything arrives on them
    tc_fence_after();
    const uint32_t tmem = *s_tmem;
    const uint32_t rows_base = CL ? mapa_shared(bar_first(0), 0u) : bar_first(0);  // CL: rows barriers live in the leader
    auto arrive = [&](uint32_t bar) {
        if (CL)
            mbar_arrive_cluster(rows_base + (bar - bar_first(0)));
        else
            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
    };
    auto wait_rows = [&](uint32_t bar, uint32_t parity) {
        if (CL) mbar_wait_cluster(bar, parity); else mbar_wait(bar, parity);
    };
    // drifting activation window, see k_net_forward_x3p: layer l + 1 is written 8 rows below layer l
    auto base_row = [&](int l) { return kLead + GP::DRIFT_ROWS * (GP::WRAP - 1 - (l % GP::WRAP)); };
    auto zero_rows = [&](int row) {  // 8 rows, by one warp
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int idx = lane * 2 + k;  // row (3 bits) | chunk (3 bits)
            st_shared_v4(s_act + (uint32_t)(row + (idx >> 3)) * 128u + (uint32_t)(idx & 7) * 16u, 0u, 0u, 0u, 0u);
        }
    };

    if (warp == EW + 1) {
        // ---- weight producer: the ring is filled strictly in tap order, as far ahead as it has free slots
        if (lane == 0) {
            for (uint32_t u = 0; u < total_units; ++u) {
                const uint32_t slot = u % NSLOT, use = u / NSLOT;
                if (use >= 1) mbar_wait(bar_empty(slot), (use - 1u) & 1u);
                const uint32_t ul = u % (uint32_t)(UPL * L), layer = ul / UPL, tap = (ul - layer * UPL) * TPS;
                const uint8_t* src = CL ? net.wpair + ((size_t)crank * (size_t)(9 * L) + (size_t)layer * 9 + tap) * (size_t)GP::TAP_STRIDE
                                        : net.wconv + ((size_t)layer * 9 + tap) * (size_t)O::TAP_BYTES;
                mbar_expect_tx(bar_full(slot), (uint32_t)GP::SLOT_BYTES);
                bulk_g2s(s_ring + slot * (uint32_t)GP::SLOT_BYTES, src, (uint32_t)GP::SLOT_BYTES, bar_full(slot));
            }
        }
    } else if (CL && warp == EW && crank != 0u) {
        // ---- peer CTA: no MMA issue here; relay "this CTA's share of the slot has landed" to the leader
        if (lane == 0) {
            const uint32_t peer0 = mapa_shared(bar_peer(0), 0u);
            for (uint32_t u = 0; u < total_units; ++u) {
                const uint32_t slot = u % NSLOT, use = u / NSLOT;
                mbar_wait(bar_full(slot), use & 1u);
                mbar_arrive_cluster(peer0 + slot * 8u);
            }
        }
    } else if (warp == EW) {
        // ---- MMA issue (the whole warp runs the loop so that descriptors stay in uniform registers; one elected lane issues)
        const bool elected = elect_one();
        constexpr uint32_t kIdescPair = (1u << 4) | ((64u >> 3) << 17) | ((256u >> 4) << 24);
        uint32_t q0 = 0, stage = 0;  // stage = number of "rows ready" rounds consumed so far (input stage + epilogues)
        int gl = 0;                  // layers issued so far modulo WRAP, over all board groups
        auto wait_weights = [&](uint32_t uu) {
            const uint32_t sl = uu % NSLOT, us = uu / NSLOT;
            mbar_wait(bar_full(sl), us & 1u);
            if (CL) mbar_wait_cluster(bar_peer(sl), us & 1u);
        };
        for (int64_t gi = 0; gi < my_groups; ++gi) {
            for (int l = 0; l < L; ++l) {
                const bool use_s = l >= 2 && (l & 1) == 0;
                const uint32_t dcol = tmem + (use_s ? SET : 0u);
                const int ksteps = l == 0 ? O::KCH0 / 2 : O::KCH / 2;
                const int row_l = base_row(gl);
                // accumulator a reads rows 128 a - 7 .. 128 a + 134: group a - 1 (tested when accumulator a - 1 was issued), group a,
                // and from tap 5 on the first warp of group a + 1. Every test that can be made early sits behind queued MMAs.
                wait_rows(bar_first(0), stage & 1u);
                wait_rows(bar_rest(0), stage & 1u);
                tc_fence_after();
                wait_weights(q0);
#pragma unroll 1
                for (int a = 0; a < NACC; ++a) {
                    if (lane == 0) QTL(l, a, 0);
                    const uint32_t d_acc = dcol + (uint32_t)a * ACC;
                    const uint32_t a_acc_lo = desc_lo(s_act) + (uint32_t)((row_l + a * 128) * 8);  // 128-byte rows: 8 per row in the address field
#pragma unroll
                    for (int g = 0; g < UPL; ++g) {  // unrolled: the tap number (window shift, which test sits where) is a compile-time constant
                        const uint32_t u = q0 + g, slot = u % NSLOT;
                        const uint32_t b_slot_lo = desc_lo(s_ring) + slot * (uint32_t)(GP::SLOT_BYTES >> 4);
#pragma unroll
                        for (int tt = 0; tt < TPS; ++tt) {
                            const int t = g * TPS + tt;
                            if (t == 5 && a + 1 < NACC) {  // the first window that reaches into the next accumulator's rows
                                wait_rows(bar_first(a + 1), stage & 1u);
                                tc_fence_after();
                            }
                            // descriptor low words of this tap (whole warp, uniform registers); K step j adds 32 bytes = 2 to both
                            const uint32_t a_lo = a_acc_lo + (uint32_t)(((t / 3 - 1) * 6 + (t % 3 - 1)) * 8);
                            const uint32_t b_lo = b_slot_lo + (uint32_t)(tt * (GP::TAP_STRIDE >> 4));
                            if (elected) {
#pragma unroll
                                for (int j = 0; j < 4; ++j)
                                    if (j < ksteps) mma_lo<CL>(d_acc, a_lo + 2u * j, b_lo + 2u * j, (use_s || t > 0 || j > 0) ? 1u : 0u, CL ? kIdescPair : O::IDESC);
                            }
                            if (tt == 0) {
                                if (a == 0 && g + 1 < UPL) {
                                    wait_weights(u + 1);
                                } else if (g + 1 == UPL && a + 1 < NACC) {  // the next accumulator's other rows: long written
                                    wait_rows(bar_rest(a + 1), stage & 1u);
                                    tc_fence_after();
                                }
                            }
                        }
                        if (a == NACC - 1 && elected) {  // all accumulators' MMAs have read the slot
                            if (CL) umma_commit_pair(bar_empty(slot)); else umma_commit(bar_empty(slot));
                        }
                    }
                    if (elected) {
                        if (CL) umma_commit_pair(bar_acc(a)); else umma_commit(bar_acc(a));
                    }
                    if (lane == 0) QTL(l, a, 1);
                }
                q0 += (uint32_t)UPL;
                stage += 1;
                gl = gl + 1 == GP::WRAP ? 0 : gl + 1;
            }
        }
    } else {
        // ---- epilogue warps: group a = warp >> 2 owns accumulator a; this thread owns one cell (TMEM lane) and its 64 channels
        const int a = warp >> 2;
        const int cell = a * 128 + (warp & 3) * 32 + lane;
        const Cell c = decode_cell(cell, CELLS);
        const uint32_t my_rows = (warp & 3) == 0 ? bar_first(a) : bar_rest(a);
        const uint32_t tlane = tmem + ((uint32_t)((warp & 3) * 32) << 16);
        uint32_t acc_par = 0;  // parity of the layer counter (every accumulator barrier completes once per layer)
        auto group_board0 = [&](int64_t g) { return CL ? (2 * (worker + g * n_workers) + (int64_t)crank) * NB : ((int64_t)blockIdx.x + g * gridDim.x) * NB; };
        float xin[kInPlanes];  // the next input of this cell (create_tensor_from_state layout [21][5][5]); the planes are 0 / 1: exact in f16
        auto load_input = [&](int64_t g) {
            const int64_t gb = group_board0(g) + c.board;
            const float* src = planes + gb * 525 + c.pos;
#pragma unroll
            for (int ch = 0; ch < kInPlanes; ++ch) xin[ch] = (c.real && g < my_groups && gb < n) ? __ldg(src + ch * 25) : 0.f;
        };
        auto store_input = [&](int row) {
#pragma unroll
            for (int part = 0; part < 2; ++part) {
                float x[16];
#pragma unroll
                for (int ch = 0; ch < 16; ++ch) x[ch] = part * 16 + ch < kInPlanes ? xin[part * 16 + ch] : 0.f;
                store_channels_f16_16(s_act, R, row + cell, part * 16, x);  // 32 channels: planes 21..31 and pad cells are zero
            }
        };
        // heads, one warp per board (ph_linear2 + softmax, vh_linear1 + ReLU + vh_linear2 + tanh). Two mbarriers instead of a CTA-wide
        // barrier: the four groups reach this point up to three accumulator phases apart, and nobody should wait for the others
        auto local_arrive = [&](uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); };
        auto run_heads = [&](int64_t hb0, uint32_t parity) {
            mbar_wait(bar_hfull, parity);  // every cell's 1x1 outputs of that group are in s_head
            for (int b = warp; b < NB; b += EW) {
                const int64_t gb = hb0 + b;
                if (gb >= n) continue;
                const float* hb = s_head + b * 75;
                const bool two = lane + 32 < 50;
                float l0 = HW(kPhB + lane), l1 = two ? HW(kPhB + 32 + lane) : 0.f;
#pragma unroll 10
                for (int i = 0; i < 50; ++i) {
                    const float x = hb[i];
                    l0 = fmaf(x, HW(kPhW + i * 50 + lane), l0);
                    if (two) l1 = fmaf(x, HW(kPhW + i * 50 + 32 + lane), l1);
                }
                const float m = warp_max(two ? fmaxf(l0, l1) : l0);
                const float e0 = expf(l0 - m), e1 = two ? expf(l1 - m) : 0.f;
                const float s = warp_sum(e0 + e1);
                policy[gb * 50 + lane] = e0 / s;
                if (two) policy[gb * 50 + 32 + lane] = e1 / s;
                float h0 = HW(kV1B + lane), h1 = HW(kV1B + 32 + lane);
#pragma unroll 5
                for (int i = 0; i < 25; ++i) {
                    const float x = hb[50 + i];
                    h0 = fmaf(x, HW(kV1W + i * 64 + lane), h0);
                    h1 = fmaf(x, HW(kV1W + i * 64 + 32 + lane), h1);
                }
                float acc = fmaf(fmaxf(h0, 0.f), HW(kV2W + lane), fmaxf(h1, 0.f) * HW(kV2W + 32 + lane));
                acc = warp_sum(acc);
                if (lane == 0) value[gb] = tanhf(acc + HW(kV2B));
            }
            local_arrive(bar_hfree);  // s_head may be overwritten by the next last-layer epilogue once every thread has said so
        };
        int gl = 0;  // layers done so far modulo WRAP, over all board groups (the MMA warp counts the same)
        load_input(0);
        store_input(base_row(0));
        if (warp == 0) zero_rows(base_row(0) - 8);
        if (warp == EW - 1) zero_rows(base_row(0) + NACC * 128);
        fence_proxy_async();
        arrive(my_rows);
        for (int64_t gi = 0; gi < my_groups; ++gi) {
            const int64_t board0 = group_board0(gi);
            for (int l = 0; l < L; ++l) {
                const bool use_s = l >= 2 && (l & 1) == 0;  // second convolution of a block accumulates onto the parked residual
                const bool last = l == L - 1;
                const bool feeds = !last || gi + 1 < my_groups;  // this epilogue writes the next stop of the window (layer or input)
                if (last && feeds) load_input(gi + 1);
                mbar_wait(bar_acc(a), acc_par);
                if ((warp & 3) == 0 && lane == 0) QTL(l, a, 2);
                tc_fence_after();
                const int rn = base_row(gl + 1);  // where the next layer's activations (or the next group's input) go
                if (feeds) {
                    // the window jumps back up, over rows the later accumulators' MMAs of this layer may still read
                    if (a + 1 < NACC && gl + 1 == GP::WRAP) mbar_wait(bar_acc(NACC - 1), acc_par);
                    if (warp == 0) zero_rows(rn - 8);
                    if (warp == EW - 1) zero_rows(rn + NACC * 128);
                }
                const bool preload = (l & 1) == 0 && !last;  // this layer's output is a block input: park it (+ next bias) in TMEM
                const float4* bias_l = reinterpret_cast<const float4*>(net.bias + (size_t)l * 64);
                const float4* bias_n = reinterpret_cast<const float4*>(net.bias + (size_t)(preload ? l + 2 : l) * 64);
                const uint32_t tsrc = tlane + (use_s ? SET : 0u) + a * ACC;
                const uint32_t tskip = tlane + SET + a * ACC;
                float hp0 = 0.f, hp1 = 0.f, hv = 0.f;
#pragma unroll
                for (int q = 0; q < 4; ++q) {  // 16 channels at a time
                    const int c0 = q * 16;
                    uint32_t v[16];
                    tmem_ld16_nowait(tsrc + c0, v);
                    tmem_wait_ld();
                    float o[16];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (!use_s) b = __ldg(bias_l + c0 / 4 + i);
                        o[4 * i + 0] = fmaxf(__uint_as_float(v[4 * i + 0]) + b.x, 0.f);
                        o[4 * i + 1] = fmaxf(__uint_as_float(v[4 * i + 1]) + b.y, 0.f);
                        o[4 * i + 2] = fmaxf(__uint_as_float(v[4 * i + 2]) + b.z, 0.f);
                        o[4 * i + 3] = fmaxf(__uint_as_float(v[4 * i + 3]) + b.w, 0.f);
                    }
                    if (!last) {
                        if (!c.real) {  // pad cells are stored too, as zeros (their accumulators hold sums that mean nothing)
#pragma unroll
                            for (int i = 0; i < 16; ++i) o[i] = 0.f;
                        }
                        store_channels_f16_16(s_act, R, rn + cell, c0, o);
                    }
                    if (preload) {
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const float4 b = __ldg(bias_n + c0 / 4 + i);
                            v[4 * i + 0] = __float_as_uint(o[4 * i + 0] + b.x);
                            v[4 * i + 1] = __float_as_uint(o[4 * i + 1] + b.y);
                            v[4 * i + 2] = __float_as_uint(o[4 * i + 2] + b.z);
                            v[4 * i + 3] = __float_as_uint(o[4 * i + 3] + b.w);
                        }
                        tmem_st16(tskip + c0, v);
                    }
                    if (last) {  // 1x1 convolutions of both heads (net.rs: policy_conv 64 -> 2, vh_conv 64 -> 1)
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const float4 w0 = HW4((kHP0 / 4) + c0 / 4 + i), w1 = HW4((kHP1 / 4) + c0 / 4 + i),
                                         w2 = HW4((kHV / 4) + c0 / 4 + i);
                            hp0 = fmaf(o[4 * i + 0], w0.x, fmaf(o[4 * i + 1], w0.y, fmaf(o[4 * i + 2], w0.z, fmaf(o[4 * i + 3], w0.w, hp0))));
                            hp1 = fmaf(o[4 * i + 0], w1.x, fmaf(o[4 * i + 1], w1.y, fmaf(o[4 * i + 2], w1.z, fmaf(o[4 * i + 3], w1.w, hp1))));
                            hv = fmaf(o[4 * i + 0], w2.x, fmaf(o[4 * i + 1], w2.y, fmaf(o[4 * i + 2], w2.z, fmaf(o[4 * i + 3], w2.w, hv))));
                        }
                    }
                }
                if (last) {
                    if (gi > 0) mbar_wait(bar_hfree, (uint32_t)(gi - 1) & 1u);  // the previous group's heads are done with s_head
                    if (c.real) {
                        float* hb = s_head + c.board * 75;
                        hb[c.pos] = fmaxf(hp0 + HW(kHB + 0), 0.f);
                        hb[25 + c.pos] = fmaxf(hp1 + HW(kHB + 1), 0.f);
                        hb[50 + c.pos] = fmaxf(hv + HW(kHB + 2), 0.f);
                    }
                    local_arrive(bar_hfull);
                }
                if (preload) tmem_wait_st();
                if (last && feeds) store_input(rn);
                if (feeds) {
                    fence_proxy_async();
                    tc_fence_before();
                    arrive(my_rows);  // this thread's rows (and its TMEM reads) of the layer are done
                    if ((warp & 3) == 0 && lane == 0) QTL(l, a, 3);
                }
                if (l == 1 && L >= 3 && gi > 0) run_heads(group_board0(gi - 1), (uint32_t)(gi - 1) & 1u);
                acc_par ^= 1u;
                gl = gl + 1 == GP::WRAP ? 0 : gl + 1;
            }
            if (L < 3 || gi + 1 == my_groups) run_heads(board0, (uint32_t)gi & 1u);
        }
    }
    __syncwarp();
    tc_fence_before();
    __syncthreads();
#ifdef ONB_F16Q_PROFILE
    if (blockIdx.x == 2 && tid == 0 && my_groups > 3)
        for (int l = 0; l < L && l < 8; ++l)
            for (int a = 0; a < NACC; ++a)
                printf("f16q layer %d acc %d: issue %6lld .. %6lld | done %6lld, first warp arrives %6lld\n", l, a, q_tl[l][a][0] - q_tl[0][0][0],
                       q_tl[l][a][1] - q_tl[0][0][0], q_tl[l][a][2] - q_tl[0][0][0], q_tl[l][a][3] - q_tl[0][0][0]);
#endif
    if (CL) {
        cluster_sync_all();  // neither CTA leaves (or frees TMEM) while the other may still signal its barriers
        if (warp == 0) tmem_dealloc_pair(tmem, GP::TMEM_COLS);
    } else if (warp == 0) {
        tmem_dealloc(tmem, GP::TMEM_COLS);
    }
}

// ---- 128 hidden channels (ConvResNetConfig{hidden_channels: 128}) ---------------------------------------------------------------
// The structure of k_net_forward, widened: a cell row of the activation matrix is 2 (f16) or 4 (tf32) 128-byte blocks, a weight
// tap is 128 B rows (N = 128) in the same swizzled K-major layout, so one block of a tap is 128 x 128 bytes. Per K step a tap costs
// one N = 128 MMA per accumulator; ONB_NET_F32 issues a1 x [b1 ; b2] as ONE N = 256 MMA (the weight copies of a 128-byte block
// are interleaved per block, [kb][b1 | b2][128 rows]) and a2 x b1 as N = 128, so D1 | D2 sit side by side in 256 TMEM columns.
// Geometry (one CTA per SM in every mode; TMEM and shared memory leave no room for a second):
//   f16:  2 accumulators x 128 cells (7 boards), TMEM 2 sets x 2 x 128 = 512 columns, activations 272 rows x 256 B, 3 slots of 32 KB
//   tf32: 1 accumulator (3 boards), TMEM 2 x 128 = 256, activations 128 rows x 512 B, 2 slots of 64 KB
//   f32:  1 accumulator (3 boards), TMEM 2 x 256 (D1 | D2), a1 + a2 of 128 rows x 256 B, 2 slots of 64 KB (b1, b2)
constexpr int kHidW = 128;
// head parameter blob of the wide network (floats): 1x1 head convolutions [128] each, their biases, ph_linear2 [50 in][50 out] + bias,
// vh_linear1 [25 in][128 out] + bias, vh_linear2 [128] + bias
constexpr int kWP0 = 0, kWP1 = 128, kWV = 256, kWB = 384, kWPhW = 388, kWPhB = 2888, kWV1W = 2940, kWV1B = 6140, kWV2W = 6268,
              kWV2B = 6396, kWHeadFloats = 6400;
template <bool F16, bool X3>
struct GeoW {
    static_assert(!X3 || F16, "the split-operand mode is built on f16 operands");
    static constexpr int CPC = F16 ? 8 : 4;              // channels per 16-byte chunk
    static constexpr int KB = kHidW / CPC / 8;           // 128-byte blocks per activation row / weight row: 2 | 4
    static constexpr int KSTEPS = kHidW / CPC / 2;       // 32-byte K steps per tap: 8 | 16
    static constexpr int KSTEPS0 = (F16 ? 32 : 24) / CPC / 2;  // first layer: 21 planes padded to K = 32 | 24: 2 | 3 steps
    static constexpr int NMAT = X3 ? 2 : 1;
    static constexpr int NACC = F16 && !X3 ? 2 : 1;      // accumulators of 128 cells
    static constexpr int NB = NACC == 2 ? 7 : 3;         // boards per pass
    static constexpr int CELLS = NB * kCellsPerBoard;
    static constexpr int R = (kLead + CELLS + kTrail + 7) / 8 * 8;
    static constexpr int WBLK = kHidW * 128;             // one 128-byte block of all 128 weight rows
    static constexpr int TAP0_BYTES = NMAT * WBLK;       // a first-layer tap (all copies)
    static constexpr int TAP_BYTES = NMAT * KB * WBLK;   // a tap of a 128 -> 128 layer (all copies)
    static constexpr int NSLOT = NACC == 2 ? 3 : 2;      // single-tap ring slots
    static constexpr int SLOT_BYTES = TAP_BYTES;
    static constexpr int ACT_BYTES = R * KB * 128;       // a multiple of 1024
    static constexpr int OFF_RING = NMAT * ACT_BYTES;
    static constexpr int OFF_HEAD = OFF_RING + NSLOT * SLOT_BYTES;
    static constexpr int SPLIT = 2 / NACC;               // threads per cell in the epilogue (each takes 128 / SPLIT channels)
    static constexpr int HEAD_BYTES = ((SPLIT * NB * 75 * 4 + 15) / 16) * 16;
    static constexpr int OFF_BAR = OFF_HEAD + HEAD_BYTES;
    static constexpr int SMEM = OFF_BAR + (2 * NSLOT + 1) * 8 + 16;
    static constexpr int ACC_COLS = X3 ? 256 : 128;      // TMEM columns per accumulator (X3: D1 | D2)
    static constexpr int SET_COLS = NACC * ACC_COLS;
    static constexpr int TMEM_COLS = 2 * SET_COLS;       // the plain set + the residual-preloaded set
    static constexpr uint32_t IDESC = Op<F16>::IDESC_N128, IDESC_X3 = Op<true>::idesc(256);
    // X3: the 9 taps x 128 channels (K = 1152) of a layer are summed in NPH phases of 3 taps: after each phase the epilogue threads
    // add D1 + 2^-11 D2 into f32 registers and the next phase starts from zero. The tensor core's f32 accumulation error grows
    // with the number of products it sums; in one phase the f32-faithful mode missed its 1e-5 bound (max |dv| 1.75e-5 on the
    // 3-block test network, B200), in phases of 3 taps each accumulator sums 384 products, fewer than the 576 of the 64-wide layers
    static constexpr int NPH = X3 ? 3 : 1;
    static_assert(SMEM <= 227 * 1024, "shared memory");
    static_assert(CELLS <= NACC * 128, "cells must fit the accumulators");
    static_assert(TMEM_COLS == 256 || TMEM_COLS == 512, "power of two");
    static_assert(ACT_BYTES % 1024 == 0 && SLOT_BYTES % 1024 == 0, "swizzle period");
};

template <bool F16, bool X3>
__global__ void __launch_bounds__(256, 1)
    k_net_wide(const float* __restrict__ planes, float* __restrict__ policy, float* __restrict__ value, int64_t n, NetDev net) {
    using G = GeoW<F16, X3>;
    constexpr int NB = G::NB, CELLS = G::CELLS, R = G::R, NSLOT = G::NSLOT, NACC = G::NACC, SPLIT = G::SPLIT;
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t s_act = smem_u32(smem), s_ring = s_act + G::OFF_RING, s_bar = s_act + G::OFF_BAR;
    float* s_head = reinterpret_cast<float*>(smem + G::OFF_HEAD);  // [SPLIT][NB][75] partial 1x1 head sums
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + G::OFF_BAR + (2 * NSLOT + 1) * 8);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int L = 1 + 2 * net.n_blocks;
    const int64_t n_groups = (n + NB - 1) / NB;
    if ((int64_t)blockIdx.x >= n_groups) return;
    const int64_t my_groups = (n_groups - blockIdx.x + gridDim.x - 1) / gridDim.x;
    const uint32_t total_units = (uint32_t)my_groups * (uint32_t)(9 * L);
    auto bar_full = [&](uint32_t s) { return s_bar + s * 8u; };
    auto bar_empty = [&](uint32_t s) { return s_bar + (NSLOT + s) * 8u; };
    const uint32_t bar_acc = s_bar + 2 * NSLOT * 8u;

    if (tid == 0) {
        for (uint32_t s = 0; s < (uint32_t)NSLOT; ++s) {
            mbar_init(bar_full(s), 1);
            mbar_init(bar_empty(s), 1);
        }
        mbar_init(bar_acc, 1);
        fence_barrier_init();
    }
    if (warp == 0) tmem_alloc(smem_u32(s_tmem), G::TMEM_COLS);
    for (int i = tid; i < G::NMAT * G::ACT_BYTES / 16; i += 256) st_shared_v4(s_act + i * 16, 0u, 0u, 0u, 0u);  // pad cells stay zero
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *s_tmem;
    constexpr uint32_t A2 = X3 ? (uint32_t)G::ACT_BYTES : 0u;
    constexpr uint32_t ACC = (uint32_t)G::ACC_COLS, SET = (uint32_t)G::SET_COLS;
    // epilogue ownership: TMEM lane quarter warp & 3; with two accumulators warp >> 2 picks the accumulator, with one it picks the
    // half of the channels (both threads of a cell then write partial head sums that the head stage adds in a fixed order)
    const int ep_acc = NACC == 2 ? (warp >> 2) : 0, ep_part = NACC == 2 ? 0 : (warp >> 2);
    constexpr int EP_CH = kHidW / SPLIT;
    static_assert(!X3 || EP_CH == 64, "the phase sums of the split mode are two halves of 32 channels");

    uint32_t q0 = 0, q_prod = 0, acc_par = 0;
    for (int64_t gi = 0; gi < my_groups; ++gi) {
        const int64_t board0 = ((int64_t)blockIdx.x + gi * gridDim.x) * NB;
        for (int cell = tid; cell < CELLS; cell += 256) {
            const Cell c = decode_cell(cell, CELLS);
            if (!c.real) continue;
            const int64_t gb = board0 + c.board;
            const float* src = planes + gb * 525 + c.pos;
            float x[32];
#pragma unroll
            for (int ch = 0; ch < 32; ++ch) x[ch] = (ch < kInPlanes && gb < n) ? __ldg(src + ch * 25) : 0.f;
            if (X3) store_channels_x3(s_act, A2, R, kLead + cell, 0, x);
            else store_channels<F16>(s_act, R, kLead + cell, 0, x);
        }
        fence_proxy_async();
        for (int l = 0; l < L; ++l) {
            tc_fence_before();
            __syncthreads();
            tc_fence_after();
            const bool use_s = l >= 2 && (l & 1) == 0;
            const bool last = l == L - 1;
            const uint32_t tlane = tmem + ((uint32_t)((warp & 3) * 32) << 16);
            const uint32_t tsrc = tlane + (use_s ? SET : 0u) + ep_acc * ACC, tskip = tlane + SET + ep_acc * ACC;
            float part[X3 ? EP_CH : 1];  // X3: the sums of the earlier phases (see GeoW::NPH); X3 has EP_CH = 64
#pragma unroll 1
            for (int ph = 0; ph < G::NPH; ++ph) {
                const int t_begin = ph * 9 / G::NPH, t_end = (ph + 1) * 9 / G::NPH;
                if (warp == 0) {
                    const bool elected = elect_one();
                    const uint32_t dcol = tmem + (use_s ? SET : 0u);
                    const int ksteps = l == 0 ? G::KSTEPS0 : G::KSTEPS;
#pragma unroll 1
                    for (int t = t_begin; t < t_end; ++t) {
                        const uint32_t u = q0 + t, slot = u % NSLOT, use = u / NSLOT;
                        mbar_wait(bar_full(slot), use & 1u);
                        tc_fence_after();
                        const int row0 = kLead + (t / 3 - 1) * 6 + (t % 3 - 1);
                        const uint32_t a_lo = desc_lo(s_act + (uint32_t)row0 * 128u), b_lo = desc_lo(s_ring + slot * (uint32_t)G::SLOT_BYTES);
                        if (elected) {
#pragma unroll 1
                            for (int j = 0; j < ksteps; ++j) {
                                const uint32_t kb = (uint32_t)(j >> 2), ks = (uint32_t)(j & 3) * 2u;  // 128-byte block, 32-byte step in it
                                const uint32_t bj = b_lo + kb * (uint32_t)(G::NMAT * G::WBLK >> 4) + ks;
                                const uint32_t acc = ((use_s && ph == 0) || t > t_begin || j > 0) ? 1u : 0u;
#pragma unroll
                                for (int a = 0; a < NACC; ++a) {
                                    const uint32_t aj = a_lo + kb * (uint32_t)(R * 8) + (uint32_t)(a * 128 * 8) + ks;
                                    if (X3) {
                                        mma_lo<false, true>(dcol, aj, bj, acc, G::IDESC_X3);                 // a1 b1 | a1 b2
                                        mma_lo<false, true>(dcol + 128u, aj + (A2 >> 4), bj, 1u, G::IDESC);  // a2 b1 -> D2
                                    } else {
                                        mma_lo<false, F16>(dcol + a * ACC, aj, bj, acc, G::IDESC);
                                    }
                                }
                            }
                            umma_commit(bar_empty(slot));
                        }
                        __syncwarp();
                    }
                    if (elected) umma_commit(bar_acc);
                } else if (tid == 32) {
                    // weight producer: the ring runs up to NSLOT taps past this phase (weights do not depend on the data)
                    const uint32_t target = min(q0 + (uint32_t)(t_end + NSLOT), total_units);
                    while (q_prod < target) {
                        const uint32_t slot = q_prod % NSLOT, use = q_prod / NSLOT;
                        if (use >= 1) mbar_wait(bar_empty(slot), (use - 1u) & 1u);
                        const uint32_t ul = q_prod % (uint32_t)(9 * L), layer = ul / 9, tap = ul - layer * 9;
                        const uint8_t* src = net.wconv + (layer == 0 ? (size_t)tap * G::TAP0_BYTES
                                                                     : (size_t)9 * G::TAP0_BYTES + ((size_t)(layer - 1) * 9 + tap) * G::TAP_BYTES);
                        const uint32_t bytes = layer == 0 ? (uint32_t)G::TAP0_BYTES : (uint32_t)G::TAP_BYTES;
                        mbar_expect_tx(bar_full(slot), bytes);
                        bulk_g2s(s_ring + slot * (uint32_t)G::SLOT_BYTES, src, bytes, bar_full(slot));
                        ++q_prod;
                    }
                }
                __syncwarp();
                mbar_wait(bar_acc, acc_par);
                acc_par ^= 1u;
                tc_fence_after();
                if constexpr (X3) {
                    if (ph + 1 < G::NPH) {  // fold this phase into registers; the next phase restarts the accumulator from zero
#pragma unroll
                        for (int h = 0; h < EP_CH / 16; ++h) {
                            uint32_t v[16], v2[16];  // 16 columns at a time: the phase sums already hold 64 registers
                            const int ch0 = ep_part * EP_CH + h * 16;
                            tmem_ld16_nowait(tsrc + ch0, v);
                            tmem_ld16_nowait(tsrc + 128 + ch0, v2);
                            tmem_wait_ld();
#pragma unroll
                            for (int i = 0; i < 16; ++i) {
                                const float x = fmaf(__uint_as_float(v2[i]), kX3InvScale, __uint_as_float(v[i]));
                                part[h * 16 + i] = ph == 0 ? x : part[h * 16 + i] + x;
                            }
                        }
                        tc_fence_before();
                        __syncthreads();
                        tc_fence_after();
                    }
                }
            }
            // ---- epilogue: this thread owns one cell (TMEM lane) and EP_CH of its channels
            const bool preload = (l & 1) == 0 && !last;
            const float4* bias_l = reinterpret_cast<const float4*>(net.bias + (size_t)l * kHidW);
            const float4* bias_n = reinterpret_cast<const float4*>(net.bias + (size_t)(preload ? l + 2 : l) * kHidW);
            const float4* hw = reinterpret_cast<const float4*>(net.head);
            const int cell = ep_acc * 128 + (warp & 3) * 32 + lane;
            const Cell c = decode_cell(cell, CELLS);
            float hp0 = 0.f, hp1 = 0.f, hv = 0.f;
#pragma unroll 1
            for (int h = 0; h < EP_CH / 32; ++h) {
                const int ch0 = ep_part * EP_CH + h * 32;
                uint32_t v[32];
                if constexpr (X3) {  // D1 + 2^-11 D2 of the last phase + the earlier phases
                    tmem_ld32(tsrc + ch0, v);
#pragma unroll
                    for (int q = 0; q < 2; ++q) {
                        uint32_t v2[16];
                        tmem_ld16_nowait(tsrc + 128 + ch0 + 16 * q, v2);
                        tmem_wait_ld();
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            const int k = 16 * q + i;
                            v[k] = __float_as_uint(fmaf(__uint_as_float(v2[i]), kX3InvScale, __uint_as_float(v[k])) + (G::NPH > 1 ? (h == 0 ? part[k] : part[32 + k]) : 0.f));
                        }
                    }
                } else {
                    tmem_ld32(tsrc + ch0, v);
                }
                float o[32];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (!use_s) b = __ldg(bias_l + ch0 / 4 + i);
                    o[4 * i + 0] = fmaxf(__uint_as_float(v[4 * i + 0]) + b.x, 0.f);
                    o[4 * i + 1] = fmaxf(__uint_as_float(v[4 * i + 1]) + b.y, 0.f);
                    o[4 * i + 2] = fmaxf(__uint_as_float(v[4 * i + 2]) + b.z, 0.f);
                    o[4 * i + 3] = fmaxf(__uint_as_float(v[4 * i + 3]) + b.w, 0.f);
                }
                if (!last && c.real) {
                    if (X3) store_channels_x3(s_act, A2, R, kLead + cell, ch0, o);
                    else store_channels<F16>(s_act, R, kLead + cell, ch0, o);
                }
                if (preload) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float4 b = __ldg(bias_n + ch0 / 4 + i);
                        v[4 * i + 0] = __float_as_uint(o[4 * i + 0] + b.x);
                        v[4 * i + 1] = __float_as_uint(o[4 * i + 1] + b.y);
                        v[4 * i + 2] = __float_as_uint(o[4 * i + 2] + b.z);
                        v[4 * i + 3] = __float_as_uint(o[4 * i + 3] + b.w);
                    }
                    tmem_st32(tskip + ch0, v);
                    if (X3) {  // the D2 half of the preloaded accumulator starts from zero
#pragma unroll
                        for (int i = 0; i < 32; ++i) v[i] = 0u;
                        tmem_st32(tskip + 128 + ch0, v);
                    }
                }
                if (last) {  // 1x1 convolutions of both heads (policy_conv 128 -> 2, vh_conv 128 -> 1)
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float4 w0 = __ldg(hw + (kWP0 + ch0) / 4 + i), w1 = __ldg(hw + (kWP1 + ch0) / 4 + i), w2 = __ldg(hw + (kWV + ch0) / 4 + i);
                        hp0 = fmaf(o[4 * i + 0], w0.x, fmaf(o[4 * i + 1], w0.y, fmaf(o[4 * i + 2], w0.z, fmaf(o[4 * i + 3], w0.w, hp0))));
                        hp1 = fmaf(o[4 * i + 0], w1.x, fmaf(o[4 * i + 1], w1.y, fmaf(o[4 * i + 2], w1.z, fmaf(o[4 * i + 3], w1.w, hp1))));
                        hv = fmaf(o[4 * i + 0], w2.x, fmaf(o[4 * i + 1], w2.y, fmaf(o[4 * i + 2], w2.z, fmaf(o[4 * i + 3], w2.w, hv))));
                    }
                }
            }
            if (last && c.real) {
                float* hb = s_head + (ep_part * NB + c.board) * 75;
                hb[c.pos] = hp0;
                hb[25 + c.pos] = hp1;
                hb[50 + c.pos] = hv;
            }
            if (preload) tmem_wait_st();
            fence_proxy_async();
            q0 += 9u;
        }
        // ---- heads: the partial 1x1 sums are added in a fixed order (batch invariant), then one warp per board
        __syncthreads();
        for (int i = tid; i < NB * 75; i += 256) {
            float s = s_head[i];
#pragma unroll
            for (int p = 1; p < SPLIT; ++p) s += s_head[p * NB * 75 + i];
            s_head[i] = fmaxf(s + __ldg(net.head + kWB + (i % 75) / 25), 0.f);
        }
        __syncthreads();
        for (int b = warp; b < NB; b += 8) {
            const int64_t gb = board0 + b;
            if (gb >= n) continue;
            const float* hb = s_head + b * 75;
            const bool two = lane + 32 < 50;
            float l0 = __ldg(net.head + kWPhB + lane), l1 = two ? __ldg(net.head + kWPhB + 32 + lane) : 0.f;
            for (int i = 0; i < 50; ++i) {
                const float x = hb[i];
                l0 = fmaf(x, __ldg(net.head + kWPhW + i * 50 + lane), l0);
                if (two) l1 = fmaf(x, __ldg(net.head + kWPhW + i * 50 + 32 + lane), l1);
            }
            const float m = warp_max(two ? fmaxf(l0, l1) : l0);
            const float e0 = expf(l0 - m), e1 = two ? expf(l1 - m) : 0.f;
            const float s = warp_sum(e0 + e1);
            policy[gb * 50 + lane] = e0 / s;
            if (two) policy[gb * 50 + 32 + lane] = e1 / s;
            float hj[4];  // value hidden units lane, lane + 32, lane + 64, lane + 96
#pragma unroll
            for (int k = 0; k < 4; ++k) hj[k] = __ldg(net.head + kWV1B + 32 * k + lane);
            for (int i = 0; i < 25; ++i) {
                const float x = hb[50 + i];
#pragma unroll
                for (int k = 0; k < 4; ++k) hj[k] = fmaf(x, __ldg(net.head + kWV1W + i * kHidW + 32 * k + lane), hj[k]);
            }
            float acc = 0.f;
#pragma unroll
            for (int k = 0; k < 4; ++k) acc = fmaf(fmaxf(hj[k], 0.f), __ldg(net.head + kWV2W + 32 * k + lane), acc);
            acc = warp_sum(acc);
            if (lane == 0) value[gb] = tanhf(acc + __ldg(net.head + kWV2B));
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, G::TMEM_COLS);
}

// ---- host side: fold BatchNorm, round to tf32, lay the weights out as the tensor core reads them ------------------------------
struct Named {
    std::string name;
    const float* data;
    int64_t numel;
};
const Named* find(const std::vector<Named>& ts, const std::string& name, int64_t numel, std::string& err) {
    for (const Named& t : ts)
        if (t.name == name) {
            if (t.numel != numel) {
                err = "tensor " + name + " has " + std::to_string(t.numel) + " elements, expected " + std::to_string(numel);
                return nullptr;
            }
            return &t;
        }
    err = "tensor " + name + " is missing";
    return nullptr;
}
float tf32_round_host(float x) {  // cvt.rna.tf32.f32: nearest, ties away from zero, on the 13 dropped mantissa bits
    uint32_t u;
    memcpy(&u, &x, 4);
    if ((u & 0x7F800000u) != 0x7F800000u) u += 0x1000u;
    u &= 0xFFFFE000u;
    memcpy(&x, &u, 4);
    return x;
}
struct BnFold {
    std::vector<double> scale, shift;  // y = conv_nobias * scale + shift
};
bool fold_bn(const std::vector<Named>& ts, const std::string& conv, const std::string& bn, int c_out, double eps, BnFold& f, std::string& err) {
    const Named *cb = find(ts, conv + ".bias", c_out, err), *w = cb ? find(ts, bn + ".weight", c_out, err) : nullptr,
                *b = w ? find(ts, bn + ".bias", c_out, err) : nullptr, *m = b ? find(ts, bn + ".running_mean", c_out, err) : nullptr,
                *v = m ? find(ts, bn + ".running_var", c_out, err) : nullptr;
    if (!v) return false;
    f.scale.resize(c_out);
    f.shift.resize(c_out);
    for (int i = 0; i < c_out; ++i) {
        const double s = (double)w->data[i] / std::sqrt((double)v->data[i] + eps);
        f.scale[i] = s;
        f.shift[i] = ((double)cb->data[i] - (double)m->data[i]) * s + (double)b->data[i];
    }
    return true;
}

// replaces the current slot's network with the given blobs
int32_t upload_net(Ctx* c, const std::vector<uint8_t>& wconv, const std::vector<float>& bias, const std::vector<float>& head, int n_blocks, int hid,
                   bool f16, bool x3, size_t pair_off, std::string& err) {
    Ctx::NetSlot& ns = c->net[c->net_cur];
    cudaStreamSynchronize(c->stream);  // a forward pass with the old weights may still be running
    for (void** p : {(void**)&ns.w, (void**)&ns.bias, (void**)&ns.head})
        if (*p) {
            cudaFree(*p);
            *p = nullptr;
        }
    ns.loaded = 0;
    cudaError_t e = cudaMalloc(&ns.w, wconv.size());
    if (e == cudaSuccess) e = cudaMalloc(&ns.bias, bias.size() * 4);
    if (e == cudaSuccess) e = cudaMalloc(&ns.head, head.size() * 4);
    if (e == cudaSuccess) e = cudaMemcpyAsync(ns.w, wconv.data(), wconv.size(), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(ns.bias, bias.data(), bias.size() * 4, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(ns.head, head.data(), head.size() * 4, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) {
        err = std::string("CUDA: ") + cudaGetErrorString(e);
        return e == cudaErrorMemoryAllocation ? ONB_E_NOMEM : ONB_E_CUDA;
    }
    ns.blocks = n_blocks;
    ns.hid = hid;
    ns.f16 = f16 ? 1 : 0;
    ns.x3 = x3 ? 1 : 0;
    ns.pair_off = pair_off;
    ns.loaded = 1;
    return ONB_OK;
}

// The 128-wide network (k_net_wide): BatchNorm folded in f64, taps in the swizzled K-major operand layout of GeoW,
// [layer][tap][128-byte block kb][copy][co][128 B]; biases [L][128]; the head blob of the kW* offsets.
int32_t net_load_wide(Ctx* c, const std::vector<Named>& ts, int n_blocks, std::string& err) {
    constexpr int H = kHidW;
    const double eps = 1e-5;
    const int L = 1 + 2 * n_blocks;
    const int mode = c->net_tf32;
    const bool f16 = mode != ONB_NET_TF32, x3 = mode == ONB_NET_F32;
    const int nmat = x3 ? 2 : 1, cpc = f16 ? 8 : 4, kch = H / cpc;
    const size_t blk = (size_t)H * 128, tap0 = nmat * blk, tap = nmat * (size_t)(kch / 8) * blk;
    std::vector<uint8_t> wconv(9 * tap0 + (size_t)(L - 1) * 9 * tap, 0);
    std::vector<float> bias((size_t)(L + 2) * H, 0.f), head(kWHeadFloats, 0.f);
    double w_absmax = 0.0;
    for (int l = 0; l < L; ++l) {
        std::string conv = "conv_init_1", bn = "bn1";
        if (l > 0) {
            const std::string blkname = "resnet_" + std::to_string((l - 1) / 2) + ".resnet_small_block" + std::to_string(((l - 1) & 1) + 1);
            conv = blkname + ".small_block_conv";
            bn = blkname + ".small_block_bn";
        }
        const int c_in = l == 0 ? kInPlanes : H;
        const Named* w = find(ts, conv + ".weight", (int64_t)H * c_in * 9, err);
        if (!w) return ONB_E_INVALID;
        BnFold f;
        if (!fold_bn(ts, conv, bn, H, eps, f, err)) return ONB_E_INVALID;
        const int chunks = l == 0 ? 8 : kch;  // the first layer fills one 128-byte block (channels beyond 21 are zero)
        const size_t tb = l == 0 ? tap0 : tap;
        uint8_t* dst = wconv.data() + (l == 0 ? 0 : 9 * tap0 + (size_t)(l - 1) * 9 * tap);
        for (int t = 0; t < 9; ++t)
            for (int kc = 0; kc < chunks; ++kc)
                for (int co = 0; co < H; ++co)
                    for (int e = 0; e < cpc; ++e) {
                        const int ci = kc * cpc + e;
                        const double xd = ci < c_in ? (double)w->data[((size_t)co * c_in + ci) * 9 + t] * f.scale[co] : 0.0;
                        const float x = (float)xd;
                        if (std::fabs(xd) > w_absmax) w_absmax = std::fabs(xd);
                        uint8_t* q = dst + (size_t)t * tb + (size_t)(kc >> 3) * nmat * blk + (size_t)co * 128 + (size_t)(((kc & 7) ^ (co & 7)) << 4);
                        if (f16) {
                            const __half hv = __float2half_rn(x);
                            memcpy(q + e * 2, &hv, 2);
                            if (x3) {  // w = w1 + 2^-11 w2: b2 follows b1 in the same 128-byte block (one N = 256 MMA reads both)
                                const __half lv = __float2half_rn((float)((xd - (double)__half2float(hv)) * (double)kX3Scale));
                                memcpy(q + blk + e * 2, &lv, 2);
                            }
                        } else {
                            const float r = tf32_round_host(x);
                            memcpy(q + e * 4, &r, 4);
                        }
                    }
        for (int co = 0; co < H; ++co) bias[(size_t)l * H + co] = (float)f.shift[co];
    }
    const Named *pw = find(ts, "policy_conv.weight", 2 * H, err), *vw = pw ? find(ts, "vh_conv.weight", H, err) : nullptr;
    if (!vw) return ONB_E_INVALID;
    BnFold fp, fv;
    if (!fold_bn(ts, "policy_conv", "policy_bn", 2, eps, fp, err) || !fold_bn(ts, "vh_conv", "vh_bn", 1, eps, fv, err)) return ONB_E_INVALID;
    for (int ci = 0; ci < H; ++ci) {
        head[kWP0 + ci] = (float)((double)pw->data[ci] * fp.scale[0]);
        head[kWP1 + ci] = (float)((double)pw->data[H + ci] * fp.scale[1]);
        head[kWV + ci] = (float)((double)vw->data[ci] * fv.scale[0]);
    }
    head[kWB + 0] = (float)fp.shift[0];
    head[kWB + 1] = (float)fp.shift[1];
    head[kWB + 2] = (float)fv.shift[0];
    const Named *p2w = find(ts, "ph_linear2.weight", 2500, err), *p2b = p2w ? find(ts, "ph_linear2.bias", 50, err) : nullptr,
                *v1w = p2b ? find(ts, "vh_linear1.weight", (int64_t)H * 25, err) : nullptr, *v1b = v1w ? find(ts, "vh_linear1.bias", H, err) : nullptr,
                *v2w = v1b ? find(ts, "vh_linear2.weight", H, err) : nullptr, *v2b = v2w ? find(ts, "vh_linear2.bias", 1, err) : nullptr;
    if (!v2b) return ONB_E_INVALID;
    for (int j = 0; j < 50; ++j) {
        for (int i = 0; i < 50; ++i) head[kWPhW + i * 50 + j] = p2w->data[j * 50 + i];
        head[kWPhB + j] = p2b->data[j];
    }
    for (int j = 0; j < H; ++j) {
        for (int i = 0; i < 25; ++i) head[kWV1W + i * H + j] = v1w->data[j * 25 + i];
        head[kWV1B + j] = v1b->data[j];
        head[kWV2W + j] = v2w->data[j];
    }
    head[kWV2B] = v2b->data[0];
    if (f16 && w_absmax > 65504.0) {
        err = "a BatchNorm-folded convolution weight has magnitude " + std::to_string(w_absmax) + " > 65504 (f16 range): load this network with ONB_NET_TF32";
        return ONB_E_INVALID;
    }
    return upload_net(c, wconv, bias, head, n_blocks, H, f16, x3, 0, err);
}

}  // namespace

// Parameters by the reference's VarStore names (net.rs:118-213; '|' or '.' as separator), OIHW / [out][in] f32 as libtorch stores them.
int32_t net_load(Ctx* c, int32_t n_tensors, const char* const* names, const float* const* data, const int64_t* numel, std::string& err) {
    std::vector<Named> ts;
    for (int32_t i = 0; i < n_tensors; ++i) {
        if (!names[i] || !data[i]) {
            err = "null tensor name or data";
            return ONB_E_INVALID;
        }
        std::string s(names[i]);
        for (char& ch : s)
            if (ch == '|') ch = '.';
        ts.push_back(Named{s, data[i], numel[i]});
    }
    int n_blocks = 0;
    for (;; ++n_blocks) {
        bool present = false;
        const std::string key = "resnet_" + std::to_string(n_blocks) + ".resnet_small_block1.small_block_conv.weight";
        for (const Named& t : ts) present |= t.name == key;
        if (!present) break;
    }
    if (n_blocks > kMaxBlocks) {
        err = "more residual blocks than supported";
        return ONB_E_INVALID;
    }
    // the width (ConvResNetConfig::hidden_channels) comes from bn1; every other tensor's size is then checked against it
    int hid = 0;
    for (const Named& t : ts)
        if (t.name == "bn1.weight") hid = (int)t.numel;
    if (hid != 64 && hid != kHidW) {
        err = hid == 0 ? "tensor bn1.weight is missing"
                       : "bn1.weight has " + std::to_string(hid) + " channels: this build supports ConvResNetConfig{hidden_channels: 64 or 128, input_channels: 21}";
        return ONB_E_INVALID;
    }
    if (hid == kHidW) return net_load_wide(c, ts, n_blocks, err);
    const double eps = 1e-5;  // nn::BatchNormConfig default of tch 0.10 / torch
    const int L = 1 + 2 * n_blocks;
    const int mode = c->net_tf32;  // ONB_NET_F16 | ONB_NET_TF32 | ONB_NET_F32 (f16 operands split in two, see Geo)
    const bool f16 = mode != ONB_NET_TF32, x3 = mode == ONB_NET_F32;
    const int nmat = x3 ? 2 : 1;
    const int cpc = f16 ? Op<true>::CPC : Op<false>::CPC, kch = f16 ? Op<true>::KCH : Op<false>::KCH;
    const size_t tap_bytes = f16 ? Op<true>::TAP_BYTES : Op<false>::TAP_BYTES, tap_bytes0 = f16 ? Op<true>::TAP_BYTES0 : Op<false>::TAP_BYTES0;
    std::vector<uint8_t> wconv((size_t)nmat * (9 * tap_bytes0 + (size_t)(L - 1) * 9 * tap_bytes), 0);
    std::vector<float> bias((size_t)(L + 2) * 64, 0.f), head(kHeadFloats, 0.f);
    double w_absmax = 0.0;
    for (int l = 0; l < L; ++l) {
        std::string conv, bn;
        if (l == 0) {
            conv = "conv_init_1";
            bn = "bn1";
        } else {
            const std::string blk = "resnet_" + std::to_string((l - 1) / 2) + ".resnet_small_block" + std::to_string(((l - 1) & 1) + 1);
            conv = blk + ".small_block_conv";
            bn = blk + ".small_block_bn";
        }
        const int c_in = l == 0 ? kInPlanes : kHid;
        const Named* w = find(ts, conv + ".weight", (int64_t)kHid * c_in * 9, err);
        if (!w) {
            if (l == 0) err += " (this build supports ConvResNetConfig{hidden_channels: 64, input_channels: 21})";
            return ONB_E_INVALID;
        }
        BnFold f;
        if (!fold_bn(ts, conv, bn, kHid, eps, f, err)) return ONB_E_INVALID;
        const int chunks = l == 0 ? 8 : kch;  // the first layer fills one whole 128-byte block (channels beyond 21 are zero)
        const size_t tb = l == 0 ? tap_bytes0 : tap_bytes;
        uint8_t* dst = wconv.data() + (size_t)nmat * (l == 0 ? 0 : 9 * tap_bytes0 + (size_t)(l - 1) * 9 * tap_bytes);
        for (int tap = 0; tap < 9; ++tap)
            for (int kc = 0; kc < chunks; ++kc)
                for (int co = 0; co < kHid; ++co)
                    for (int e = 0; e < cpc; ++e) {  // operand layout: [tap][copy][128-byte block][co][chunk ^ (co & 7)][16 bytes of input channels]
                        const int ci = kc * cpc + e;
                        const double xd = ci < c_in ? (double)w->data[((size_t)co * c_in + ci) * 9 + tap] * f.scale[co] : 0.0;
                        const float x = (float)xd;
                        if (std::fabs(xd) > w_absmax) w_absmax = std::fabs(xd);
                        uint8_t* q = dst + (size_t)tap * nmat * tb + (size_t)(kc >> 3) * 64 * 128 + (size_t)co * 128 + (size_t)(((kc & 7) ^ (co & 7)) << 4);
                        if (f16) {
                            const __half hv = __float2half_rn(x);
                            memcpy(q + e * 2, &hv, 2);
                            if (x3) {  // w = w1 + 2^-11 w2 (the remainder is taken from the f64 folded weight)
                                const __half lv = __float2half_rn((float)((xd - (double)__half2float(hv)) * (double)kX3Scale));
                                memcpy(q + tb + e * 2, &lv, 2);
                            }
                        } else {
                            const float r = tf32_round_host(x);
                            memcpy(q + e * 4, &r, 4);
                        }
                    }
        for (int co = 0; co < kHid; ++co) bias[(size_t)l * 64 + co] = (float)f.shift[co];
    }
    {   // heads
        const Named *pw = find(ts, "policy_conv.weight", 2 * kHid, err), *vw = pw ? find(ts, "vh_conv.weight", kHid, err) : nullptr;
        if (!vw) return ONB_E_INVALID;
        BnFold fp, fv;
        if (!fold_bn(ts, "policy_conv", "policy_bn", 2, eps, fp, err) || !fold_bn(ts, "vh_conv", "vh_bn", 1, eps, fv, err)) return ONB_E_INVALID;
        for (int ci = 0; ci < kHid; ++ci) {
            head[kHP0 + ci] = (float)((double)pw->data[ci] * fp.scale[0]);
            head[kHP1 + ci] = (float)((double)pw->data[kHid + ci] * fp.scale[1]);
            head[kHV + ci] = (float)((double)vw->data[ci] * fv.scale[0]);
        }
        head[kHB + 0] = (float)fp.shift[0];
        head[kHB + 1] = (float)fp.shift[1];
        head[kHB + 2] = (float)fv.shift[0];
        const Named *p2w = find(ts, "ph_linear2.weight", 2500, err), *p2b = p2w ? find(ts, "ph_linear2.bias", 50, err) : nullptr,
                    *v1w = p2b ? find(ts, "vh_linear1.weight", (int64_t)kHid * 25, err) : nullptr,
                    *v1b = v1w ? find(ts, "vh_linear1.bias", kHid, err) : nullptr, *v2w = v1b ? find(ts, "vh_linear2.weight", kHid, err) : nullptr,
                    *v2b = v2w ? find(ts, "vh_linear2.bias", 1, err) : nullptr;
        if (!v2b) return ONB_E_INVALID;
        for (int j = 0; j < 50; ++j) {
            for (int i = 0; i < 50; ++i) head[kPhW + i * 50 + j] = p2w->data[j * 50 + i];
            head[kPhB + j] = p2b->data[j];
        }
        for (int j = 0; j < kHid; ++j) {
            for (int i = 0; i < 25; ++i) head[kV1W + i * 64 + j] = v1w->data[j * 25 + i];
            head[kV1B + j] = v1b->data[j];
            head[kV2W + j] = v2w->data[j];
        }
        head[kV2B] = v2b->data[0];
    }
    // f16 operands: a folded weight beyond f16's largest finite value would become inf (the small end is harmless in the split mode and
    // costs significand bits below 6.1e-5 in the plain f16 mode -- see onb.h); such a network has to be loaded with ONB_NET_TF32
    if (f16 && w_absmax > 65504.0) {
        err = "a BatchNorm-folded convolution weight has magnitude " + std::to_string(w_absmax) + " > 65504 (f16 range): load this network with ONB_NET_TF32";
        return ONB_E_INVALID;
    }
    // ONB_NET_F32: a second copy of the taps in the order the CTA-pair kernel streams them (k_net_forward_x3p<true>): per rank of
    // the pair, per layer and tap, 12 KB = [b1 | b2 of the tap: this rank's 64 rows of the N = 128 MMA][rows 32 r .. 32 r + 31 of b1:
    // its 32 rows of the N = 64 MMA]. Moving whole 8-row groups keeps the 128-byte swizzle phase of every row.
    size_t pair_off = 0;
    if (f16 && !x3) {  // the f16 fast mode on CTA pairs (k_net_forward_f16q<true>): per rank, layer and tap the 32 B rows this rank holds
        static_assert(Op<true>::TAP_BYTES == 8192 && Op<true>::TAP_BYTES0 == 8192, "pair layout");
        pair_off = (wconv.size() + 1023) / 1024 * 1024;
        wconv.resize(pair_off + 2 * (size_t)(9 * L) * 4096, 0);
        for (int r = 0; r < 2; ++r)
            for (int t = 0; t < 9 * L; ++t)
                memcpy(wconv.data() + pair_off + ((size_t)r * (size_t)(9 * L) + (size_t)t) * 4096, wconv.data() + (size_t)t * 8192 + (size_t)r * 4096, 4096);
    }
    if (x3) {
        static_assert(Op<true>::TAP_BYTES == 8192 && Op<true>::TAP_BYTES0 == 8192, "pair layout");
        pair_off = (wconv.size() + 1023) / 1024 * 1024;
        const size_t stride = (size_t)GeoX3PT<true>::TAP_STRIDE;
        wconv.resize(pair_off + 2 * (size_t)(9 * L) * stride, 0);
        for (int r = 0; r < 2; ++r)
            for (int t = 0; t < 9 * L; ++t) {
                const uint8_t* b1 = wconv.data() + (size_t)t * 2 * 8192;
                uint8_t* dst = wconv.data() + pair_off + ((size_t)r * (size_t)(9 * L) + (size_t)t) * stride;
                memcpy(dst, b1 + (size_t)r * 8192, 8192);
                memcpy(dst + 8192, b1 + (size_t)r * 32 * 128, 4096);
            }
    }
    return upload_net(c, wconv, bias, head, n_blocks, 64, f16, x3, pair_off, err);
}

template <bool F16, bool X3 = false>
static cudaError_t launch_net_variant(Ctx* c, const float* planes, float* policy, float* value, const NetDev& nd, int sms, int64_t count) {
    using G = Geo<F16, X3>;
    static bool attr[64] = {};  // the opt-in is per device
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !attr[dev]) {
        const cudaError_t e = cudaFuncSetAttribute(k_net_forward<F16, X3>, cudaFuncAttributeMaxDynamicSharedMemorySize, G::SMEM);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) attr[dev] = true;
    }
    const int64_t groups = (count + G::NB - 1) / G::NB, slots = (int64_t)sms * (X3 ? 1 : 2);
    k_net_forward<F16, X3><<<(unsigned)(groups < slots ? groups : slots), 256, G::SMEM, c->stream>>>(planes, policy, value, count, nd);
    return cudaGetLastError();
}

static cudaError_t launch_net_x3p(Ctx* c, const float* planes, float* policy, float* value, const NetDev& nd, int sms, int64_t count) {
    using G = Geo<true, true>;
    static bool attr[64] = {};  // the opt-in is per device
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !attr[dev]) {
        const cudaError_t e = cudaFuncSetAttribute(k_net_forward_x3p<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, GeoX3P::SMEM);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) attr[dev] = true;
    }
    const int64_t groups = (count + G::NB - 1) / G::NB;
    k_net_forward_x3p<false><<<(unsigned)(groups < sms ? groups : sms), GeoX3P::THREADS, GeoX3P::SMEM, c->stream>>>(planes, policy, value, count, nd);
    return cudaGetLastError();
}

// the CTA-pair build: clusters of two CTAs, as many as the device can hold at once (one CTA per SM)
static cudaError_t launch_net_x3pair(Ctx* c, const float* planes, float* policy, float* value, const NetDev& nd, int sms, int64_t count) {
    using G = Geo<true, true>;
    using GP = GeoX3PT<true>;
    static int max_clusters[64] = {};  // per device; 0 = not asked yet
    int dev = 0;
    cudaGetDevice(&dev);
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.blockDim = dim3(GP::THREADS);
    cfg.dynamicSmemBytes = GP::SMEM;
    cfg.stream = c->stream;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    int mc = (dev >= 0 && dev < 64) ? max_clusters[dev] : 0;
    if (mc == 0) {
        cudaError_t e = cudaFuncSetAttribute(k_net_forward_x3p<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, GP::SMEM);
        if (e != cudaSuccess) return e;
        cfg.gridDim = dim3((unsigned)(sms & ~1));
        e = cudaOccupancyMaxActiveClusters(&mc, k_net_forward_x3p<true>, &cfg);
        if (e != cudaSuccess) return e;
        if (mc > sms / 2) mc = sms / 2;
        if (20 * mc < 9 * sms) mc = -1;  // the clusters would leave more than a tenth of the SMs idle
        if (dev >= 0 && dev < 64) max_clusters[dev] = mc;
    }
    if (mc < 0) return cudaErrorLaunchOutOfResources;
    const int64_t pairs = ((count + G::NB - 1) / G::NB + 1) / 2;
    cfg.gridDim = dim3(2u * (unsigned)(pairs < mc ? pairs : mc));
    return cudaLaunchKernelEx(&cfg, k_net_forward_x3p<true>, planes, (float*)policy, (float*)value, (int64_t)count, nd);
}

// the four-accumulator f16 pipeline, on CTA pairs (clusters of two) or single CTAs
template <bool CL>
static cudaError_t launch_net_f16q(Ctx* c, const float* planes, float* policy, float* value, const NetDev& nd, int sms, int64_t count) {
    using GP = GeoF16Q<CL>;
    static int max_workers[64] = {};  // per device; 0 = not asked yet, -1 = the clusters do not fit
    int dev = 0;
    cudaGetDevice(&dev);
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = CL ? 2 : 1;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.blockDim = dim3(GP::THREADS);
    cfg.dynamicSmemBytes = GP::SMEM;
    cfg.stream = c->stream;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    int mw = (dev >= 0 && dev < 64) ? max_workers[dev] : 0;
    if (mw == 0) {
        cudaError_t e = cudaFuncSetAttribute(k_net_forward_f16q<CL>, cudaFuncAttributeMaxDynamicSharedMemorySize, GP::SMEM);
        if (e != cudaSuccess) return e;
        mw = sms;
        if (CL) {
            cfg.gridDim = dim3((unsigned)(sms & ~1));
            e = cudaOccupancyMaxActiveClusters(&mw, k_net_forward_f16q<CL>, &cfg);
            if (e != cudaSuccess) return e;
            if (mw > sms / 2) mw = sms / 2;
            if (20 * mw < 9 * sms) mw = -1;  // the clusters would leave more than a tenth of the SMs idle
        }
        if (dev >= 0 && dev < 64) max_workers[dev] = mw;
    }
    if (mw < 0) return cudaErrorLaunchOutOfResources;
    const int64_t groups = (count + GP::NB - 1) / GP::NB, work = CL ? (groups + 1) / 2 : groups;
    cfg.gridDim = dim3((CL ? 2u : 1u) * (unsigned)(work < mw ? work : mw));
    return cudaLaunchKernelEx(&cfg, k_net_forward_f16q<CL>, planes, (float*)policy, (float*)value, (int64_t)count, nd);
}

// the 128-wide network: one CTA per SM, each working through board groups of GeoW::NB
template <bool F16, bool X3>
static cudaError_t launch_net_wide(Ctx* c, const float* planes, float* policy, float* value, const NetDev& nd, int sms, int64_t count) {
    using G = GeoW<F16, X3>;
    static bool attr[64] = {};  // the opt-in is per device
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !attr[dev]) {
        const cudaError_t e = cudaFuncSetAttribute(k_net_wide<F16, X3>, cudaFuncAttributeMaxDynamicSharedMemorySize, G::SMEM);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) attr[dev] = true;
    }
    const int64_t groups = (count + G::NB - 1) / G::NB;
    k_net_wide<F16, X3><<<(unsigned)(groups < sms ? groups : sms), 256, G::SMEM, c->stream>>>(planes, policy, value, count, nd);
    return cudaGetLastError();
}

cudaError_t launch_net_forward(Ctx* c, const float* planes, float* policy, float* value, int64_t count) {
    if (count <= 0) return cudaSuccess;
    const Ctx::NetSlot& ns = c->net[c->net_cur];
    const NetDev nd{reinterpret_cast<const uint8_t*>(ns.w), reinterpret_cast<const uint8_t*>(ns.w) + ns.pair_off, ns.bias, ns.head, ns.blocks};
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (ns.hid == kHidW) {  // 128 hidden channels: k_net_wide in all three modes (the 64-wide knobs below do not apply)
        if (ns.x3) return launch_net_wide<true, true>(c, planes, policy, value, nd, sms, count);
        return ns.f16 ? launch_net_wide<true, false>(c, planes, policy, value, nd, sms, count)
                      : launch_net_wide<false, false>(c, planes, policy, value, nd, sms, count);
    }
    if (ns.x3) {
        // ONB_NET_F32: split operands, f32-faithful, one CTA per SM. Default: the warp-specialised pipeline on CTA pairs
        // (k_net_forward_x3p<true>, 0.600 ms per 16 384 positions); ONB_NET_X3_PAIR=0: the same pipeline on single CTAs (0.646 ms; also
        // the fallback when the device cannot co-schedule the clusters); ONB_NET_X3_PIPE=0: the plain kernel (0.745 ms).
        const char* pipe = getenv("ONB_NET_X3_PIPE");
        if (pipe && pipe[0] == '0') return launch_net_variant<true, true>(c, planes, policy, value, nd, sms, count);
        const char* pair = getenv("ONB_NET_X3_PAIR");
        if (!(pair && pair[0] == '0')) {
            const cudaError_t e = launch_net_x3pair(c, planes, policy, value, nd, sms, count);
            if (e != cudaErrorLaunchOutOfResources) return e;
            (void)cudaGetLastError();  // no room for the clusters on this device: single CTAs
        }
        return launch_net_x3p(c, planes, policy, value, nd, sms, count);
    }
    if (!ns.f16) return launch_net_variant<false>(c, planes, policy, value, nd, sms, count);  // ONB_NET_TF32: two plain CTAs per SM
    // ONB_NET_F16 default: one CTA per SM with four accumulators (14 boards), the pipeline of k_net_forward_x3p, on CTA pairs
    // (k_net_forward_f16q<true>, 0.226 ms per 16 384 positions); ONB_NET_F16_QUAD=2: on single CTAs (0.269 ms; also the fallback when
    // the clusters cannot be co-scheduled); ONB_NET_F16_QUAD=0: the round-1 build, two plain CTAs per SM (0.322 ms)
    const char* quad = getenv("ONB_NET_F16_QUAD");
    if (quad && quad[0] == '0') return launch_net_variant<true>(c, planes, policy, value, nd, sms, count);
    if (!(quad && quad[0] == '2')) {
        const cudaError_t e = launch_net_f16q<true>(c, planes, policy, value, nd, sms, count);
        if (e != cudaErrorLaunchOutOfResources) return e;
        (void)cudaGetLastError();
    }
    return launch_net_f16q<false>(c, planes, policy, value, nd, sms, count);
}

}  // namespace onb
