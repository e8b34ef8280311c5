// conv_tc.cu -- 3x3x3 (pad 1) and 1x1x1 stride-1 convolutions as an implicit GEMM on the 5th-gen tensor cores.
//
//   D[128 voxels x BN] (TMEM, fp32)  +=  A[128 x 32] (smem, TF32)  x  B[BN x 32]^T (smem, TF32)
//
// * M tile = an 8x2x8 (x,y,z) brick of output voxels, rows ordered z (8 rows = one swizzle atom), y, x.  For every
//   (dy, dz) tap pair (9) and every 32-channel slice of C_in, ONE 4-D TMA box {32 ch, 8 z, 2 y, 10 x} fetches the
//   shifted input slab -- with a one-plane halo in x -- straight from the VC activation tensor; the three x-taps then
//   read rows [16 dx, 16 dx + 128) of that slab, an offset of two whole swizzle atoms, so the descriptor just moves by
//   2 KB: A traffic is 9 x 1.25 instead of 27 bricks per K slice (2.4x less).  Voxels outside the volume are zero-filled
//   by the TMA unit, which *is* the convolution's zero padding -- no halo logic, no im2col buffer.  Rows land 128 B
//   apart in the canonical K-major SWIZZLE_128B layout tcgen05.mma consumes.
// * B tiles = BN rows of the weight matrix W[C_out][27*C_in] (k = tap*C_in + c) for the three x-taps, 2-D TMA, same swizzle.
// * Warp roles (128 threads): thread 0 = TMA producer, thread 32 = MMA issuer (tcgen05.mma
//   kind::tf32, cta_group::1, M=128, N=BN, K=8; 3 x-taps x 4 per stage), all four warps = epilogue
//   (tcgen05.ld 32x32b -> bias / residual / ReLU -> global).  3-stage full/empty mbarrier ring;
//   tcgen05.commit releases smem slots and signals the accumulator.
// * Tiles may be listed explicitly (ragged RoI crops packed on one zero-separated canvas, mask head)
//   or implied by the volume.
//
// Reference call sites: Bottleneck.conv2 (lib/nets/backbones.py:21), geometry2.0 (:216),
// rpn_net_level{1,2} (lib/nets/network.py:40,45), MaskBackbone.geometry.{2,4,6,8} (backbones.py:243-249).
#include <cuda.h>
#include <stdlib.h>
#include <cuda_fp16.h>
#include "common.cuh"

namespace sis3d {

constexpr int TC_BZ = 8;  // brick = (16/BY) x BY x 8 voxels (x,y,z), BY in {2,4}; rows ordered z (8 = one swizzle atom), y, x
constexpr int TC_BM = 128;
constexpr int TC_KC = 32;                      // channels per stage: 32 * 4 B = 128 B = one swizzle row
constexpr int TC_STAGES_MAX = 4;
constexpr int TC_A_BYTES = TC_BM * 128;

struct TcArgs {
    const float *bias, *res;
    float *out;
    const int32_t *tiles;  // [n_tiles][8] = x0,y0,z0,x1,y1,z1,-,- (origin, exclusive valid end) or null
    int X, Y, Z, cin, cout, act, out_ld, out_coff, res_ld, res_coff;
    int tiles_y, tiles_z;
    int gemm_m, gemm_chunks_per_split;  // KS == 0 (plain GEMM y = x W^T, split-K over blockIdx.z)
    __half *out16;                      // optional fp16 twin of the output (same geometry as `out`); `out` may be null
    const float *bias_mid;              // N2 > 0: bias of the 3x3x3 conv (added before the inner ReLU), or null
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t done, spins = 0;
    do {
        if (++spins > (1u << 28)) __trap();  // a broken pipeline becomes a CUDA error, never a hung GPU
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
    } while (!done);
}
__device__ __forceinline__ void tma_load_4d(void *dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
// start>>4 [0,14) | LBO=1 [16,30) | SBO=1024B>>4 [32,46) | version=1 [46,48) | layout=SWIZZLE_128B(2) [61,64)
// ROWB = 128: SWIZZLE_128B (layout 2, 8-row atom = 1024 B);  ROWB = 64: SWIZZLE_64B (layout 4, 8-row atom = 512 B)
template <int ROWB>
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr) {
    constexpr uint64_t sbo = (8 * ROWB) >> 4, layout = ROWB == 128 ? 2 : 4;
    return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (sbo << 32) | (1ull << 46) | (layout << 61);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(0u), "r"(0u), "r"(0u), "r"(0u)
        : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(0u), "r"(0u), "r"(0u), "r"(0u)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float *v) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ void tmem_ld32_add(uint32_t taddr, float *v) {  // v += 32 accumulator columns (round to nearest)
    float t[32];
    tmem_ld32(taddr, t);
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] += t[i];
}
// X3: one logical accumulator = up to three rotating main accumulators (stride `stride` columns) + the cross-term accumulator
template <int X3>
__device__ __forceinline__ void acc_ld32(uint32_t taddr, int n_main, uint32_t stride, uint32_t lo_off, float *v) {
    tmem_ld32(taddr, v);
    if constexpr (X3 != 0) {
        if (n_main > 1) tmem_ld32_add(taddr + stride, v);
        if (n_main > 2) tmem_ld32_add(taddr + 2 * stride, v);
        if constexpr (X3 == 2) {  // fp16 split: the low parts were stored scaled by 2^11, so are the cross terms
            float t[32];
            tmem_ld32(taddr + lo_off, t);
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = fmaf(t[i], 1.0f / 2048.0f, v[i]);
        } else {
            tmem_ld32_add(taddr + lo_off, v);
        }
    }
}

// v = hi + lo with hi = tf32(v) (round to nearest, low 13 bits zero) and lo = tf32(v - hi) (v - hi is exact in fp32)
__device__ __forceinline__ float tf32_rna_bits(float x) {
    uint32_t u;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
    return __uint_as_float(u);
}
__device__ __forceinline__ void split_tf32(float v, float &hi, float &lo) {
    hi = tf32_rna_bits(v);
    lo = tf32_rna_bits(v - hi);
}

// fp16 split (X3 = 2): v = hi + lo / 2048 with hi = fp16(v) (round to nearest) and lo = fp16((v - hi) * 2048): the same
// 11 + 11 significand bits as the TF32 split, but the MMAs run at the fp16 rate (2.5x the measured TF32 rate on B200).
// Scaling the low part keeps it out of fp16's subnormal range; |v| is clamped to the fp16 range first.
__device__ __forceinline__ void split_f16(float v, __half &hi, __half &lo) {
    v = fminf(fmaxf(v, -65504.f), 65504.f);
    hi = __float2half_rn(v);
    lo = __float2half_rn((v - __half2float(hi)) * 2048.0f);
}
// activations, two at a time with packed conversions (4 ALU ops per element); precondition |v| < 65504 (not clamped here: the
// fp16-operand mask stage of the default math mode has the same range requirement)
__device__ __forceinline__ void split_f16x2(float a, float b, uint32_t &hi, uint32_t &lo) {
    const __half2 h = __floats2half2_rn(a, b);
    const float2 hf = __half22float2(h);
    const __half2 l = __floats2half2_rn((a - hf.x) * 2048.0f, (b - hf.y) * 2048.0f);
    hi = *reinterpret_cast<const uint32_t *>(&h);
    lo = *reinterpret_cast<const uint32_t *>(&l);
}
__device__ __forceinline__ void split_f16x8(const float4 a, const float4 b, uint4 &hi, uint4 &lo) {
    split_f16x2(a.x, a.y, hi.x, lo.x);
    split_f16x2(a.z, a.w, hi.y, lo.y);
    split_f16x2(b.x, b.y, hi.z, lo.z);
    split_f16x2(b.z, b.w, hi.w, lo.w);
}

// stages: 4 for BN = 128 (128 KB), 3 for BN <= 64 so that three CTAs fit one SM (the grids of the narrow layers are
// ~1.3-1.5 waves at two CTAs/SM)
template <int BN>
struct TcStages { static constexpr int value = BN >= 128 ? 4 : 3; };
// stage count per kernel flavour: the 3x3x3 stages are 3x bigger (slab + three weight tiles)
// X3 (error-compensated 3xTF32, 64-byte K rows): every stage also holds the low parts of A and B; BN = 32 keeps three
// stages (96 KB, two CTAs per SM), BN = 64 two (88 KB, two CTAs per SM), BN = 128 three (204 KB)
// X3 = 2 (fp16 split, 128-byte fp32 source rows): a stage = the slab (fp32 as it lands, split IN PLACE into fp16 hi / lo tiles of
// half the size each) + fp16 hi/lo weight tiles.  3x3x3: BN = 32: three stages of 32 KB (two CTAs share an SM: one's prologue /
// epilogue runs under the other's main loop), BN = 64: four of 44 KB, BN = 128: three of 68 KB (two stages left the TMA round
// trip exposed: 49 us -> the MMA/feed bound); 1x1 / 2x2x2 / GEMM: four.
template <int BN, int KS, int ROWB, int X3 = 0, int N2 = 0>
struct TcStagesOf {
    static constexpr int value =
        X3 == 2 ? (KS == 3 ? (BN == 64 ? 4 : 3) : 4)
                : (KS == 3 ? (X3 ? (BN == 64 ? 2 : 3) : (BN >= 128 ? 3 : 2)) : TcStages<BN>::value);
};  // narrow 3x3x3 layers: 2 stages so 2-3 CTAs share an SM
template <int BN, int KS, int ROWB, int BY, int N2 = 0, int X3 = 0>
constexpr size_t tc_smem_bytes() {
    // bytes of one weight row in shared memory: ROWB, or 64 (32 fp16 channels) in the fp16-split mode
    return (size_t)TcStagesOf<BN, KS, ROWB, X3, N2>::value *
               ((X3 == 1 ? 2 : 1) * (KS == 3 ? (16 / BY + 2) * BY * TC_BZ : TC_BM) * ROWB +
                (X3 == 1 ? 2 : 1) * (KS == 3 ? 3 : 1) * BN * (X3 == 2 ? 128 : ROWB)) +
           (size_t)(X3 == 1 ? 2 : 1) * N2 * 128 * (BN / 32) + 1024 + 256;
}
constexpr int tc_tmem_cols(int n) { return n <= 32 ? 32 : n <= 64 ? 64 : n <= 128 ? 128 : n <= 256 ? 256 : 512; }

// EB = operand element bytes: 4 -> fp32 storage, kind::tf32;  2 -> fp16 storage, kind::f16 (same 11-bit significand,
// half the operand bytes through L2).  ROWB = bytes of one K slice row in shared memory (128, or 64 for C_in = 32 in fp16).
//
// N2 > 0 (KS = 3, TF32 only) fuses the bottleneck's trailing 1x1 convolution (lib/nets/backbones.py:28-40: conv2 -> relu ->
// conv3 -> +x -> relu): the ReLU'd 128 x BN accumulator is written back to shared memory as a K-major SWIZZLE_128B operand
// (aliasing the drained pipeline stages), multiplied by W3[N2][BN] (its own TMA tile, fetched at kernel start) into a second
// TMEM accumulator, and only that N2-wide result -- plus residual and ReLU -- goes to global memory.  The BN-wide
// intermediate never leaves the SM; operand values and summation order equal the two-kernel path bit for bit.
//
// X3 = 1 (EB = 4 only): error-compensated 3xTF32.  Every fp32 operand is split as v = hi + lo with hi = tf32(v) (round to
// nearest) and lo = tf32(v - hi); the product is accumulated as A_lo.B_hi + A_hi.B_lo + A_hi.B_hi in the same fp32 TMEM
// accumulator (the dropped A_lo.B_lo term is ~2^-22 relative).  Weights are split once at pack time ([2][cout][K]: hi rows,
// then lo rows); the activation slab is split IN SHARED MEMORY by warps 2-3 after the TMA lands (hi overwrites the slab, lo
// goes to a second buffer of the same swizzled layout -- the split is elementwise, so the layout is untouched), published
// to the MMA's async proxy with fence.proxy.async + the conv_done mbarrier.  No extra L2->SM traffic for activations; the
// tensor pipe, which the narrow layers leave mostly idle, does 3x the MMAs.  Result: fp32-class accuracy (the integer
// outputs of the detector -- top-N order, NMS keep lists, class argmax, crop bounds -- match the fp32 path) on tcgen05.
//
// X3 = 2 (EB = 4, ROWB = 128): the same compensation with an fp16 split (split_f16 above): the fp32 slab lands in a staging
// buffer, warps 2-3 write its hi and (scaled) lo parts as two fp16 K-major SWIZZLE_64B tiles, the weights are pre-split fp16
// tiles, and the three products are kind::f16 MMAs -- same 22 significand bits, 2.5x the MMA rate, half as many stages.
template <int BN, int KS, int EB = 4, int ROWB = 128, int BY = 2, int N2 = 0, int X3 = 0>
__global__ void __launch_bounds__(X3 == 2 ? 256 : 128, (X3 == 2 && BN == 32) ? 2 : 1) conv3d_k3_tc_kernel(const __grid_constant__ CUtensorMap tmA,
                                                              const __grid_constant__ CUtensorMap tmB,
                                                              const __grid_constant__ CUtensorMap tmB2, const TcArgs a) {
    static_assert(N2 == 0 || (KS == 3 && EB == 4), "conv3 fusion: TF32 3x3x3 kernels only");
    static_assert(X3 == 0 || EB == 4, "3xTF32 splits fp32-stored operands");
    static_assert(X3 != 2 || ROWB == 128, "the fp16 split reads 128-byte fp32 rows and writes 64-byte fp16 rows");
    constexpr bool XH = X3 == 2;             // fp16 split
    // threads: warp 0 = TMA producer, warp 1 = MMA issuer, warps 2.. = operand splitters (X3), every warp = epilogue.  The fp16
    // split re-lays the slab out (fp32 128-byte rows -> two fp16 64-byte-row tiles), ~4 ALU ops per element: six splitter warps
    // keep it below the MMA time of a stage (two were 2x slower than the tensor pipe)
    constexpr int NT = XH ? 256 : 128;
    constexpr int NSPLIT = NT - 64;          // splitter threads
    constexpr int NHALF = NT / 128;          // epilogue: warps w and w + 4 share TMEM lane quarter w % 4 and alternate column chunks
    constexpr int OPB = XH ? 64 : ROWB;      // bytes of one K-slice row of the MMA operands in shared memory
    constexpr int KC = ROWB / EB;            // channels per pipeline stage
    constexpr int TC_BY = BY, TC_BX = 16 / BY;  // brick: BY = 2 -> 8x2x8 (whole volumes), BY = 4 -> 4x4x8 (small RoI crops)
    // 3x3x3: one stage = one (dy, dz) pair: an x-halo slab of (8+2) x-planes (160 rows) serves the three x-taps --
    // tap dx reads rows [dx*16, dx*16+128), a whole-swizzle-atom offset -- plus the three taps' weight tiles.
    constexpr int XT = KS == 3 ? 3 : 1;      // x-taps per stage
    constexpr int A_ROWS = KS == 3 ? (TC_BX + 2) * TC_BY * TC_BZ : TC_BM;
    constexpr int A_BYTES = A_ROWS * ROWB;
    // weight tiles: X3 = 2 keeps the hi and lo halves of a 32-channel K slice side by side in ONE 128-byte row (one TMA row
    // request instead of two 64-byte ones: the per-SM TMA path moves ~one row per 2.7 cycles whatever its length, and the
    // 64-byte rows made the weight tiles 3/4 of a stage's requests), SWIZZLE_128B; hi = first 64 bytes, lo = last 64
    constexpr int BROW = XH ? 128 : OPB;
    constexpr int NBT = XT * (X3 == 1 ? 2 : 1);  // weight tiles per stage
    constexpr int B_BYTES = BN * BROW;
    // stage layout: X3 = 0: [A | B x XT];  X3 = 1: [A_hi (in place) | A_lo | B_hi x XT | B_lo x XT];
    //               X3 = 2: [A: fp32 as landed -> split in place into A_hi fp16 | A_lo fp16 (half of A_BYTES each) | B_hi x XT | B_lo x XT]
    constexpr int B_OFF = (X3 == 1 ? 2 : 1) * A_BYTES;
    constexpr int STAGE_BYTES = B_OFF + NBT * B_BYTES;
    constexpr int TC_STAGES = TcStagesOf<BN, KS, ROWB, X3, N2>::value;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // SWIZZLE_128B needs 1024 B alignment
    // W3 as BN/32 K slices of [N2 rows][32 ch] (X3: hi slices, then lo slices; fp16 split: 64-byte rows)
    constexpr int B2_SLICE = N2 * 128;  // fp16 split: [hi 64 B | lo 64 B] per row
    constexpr int B2_BYTES = (X3 == 1 ? 2 : 1) * B2_SLICE * (BN / 32);
    // X3 accumulators: the tensor core adds into its fp32 accumulator with truncation, a bias that grows with the length of the
    // accumulation chain -- invisible next to TF32 operand rounding, but the dominant error of the compensated product.  So the
    // hi.hi terms rotate over THREE accumulators (stage it -> it % 3: chains a third as long, summed with round-to-nearest adds in
    // the epilogue) and the two cross terms go to a FOURTH one (2^-11 of the magnitude, its truncation is negligible):
    // columns [0,3BN) main, [3BN,4BN) cross terms; fused tail: [4BN,4BN+N2) main, [4BN+N2,4BN+2N2) cross terms.
    constexpr int TMEM_COLS = tc_tmem_cols(X3 ? 4 * BN + 2 * N2 : BN + N2);
    uint8_t *smem_b2 = smem + TC_STAGES * STAGE_BYTES;
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_b2 + B2_BYTES);
    uint64_t *empty = full + TC_STAGES;
    uint64_t *acc_ready = empty + TC_STAGES;
    uint64_t *b2_full = acc_ready + 1, *acc2_ready = acc_ready + 2;
    uint64_t *conv_done = acc_ready + 3;  // X3: the converter warps finished splitting stage s
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(conv_done + TC_STAGES);

    const int warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        for (int i = 0; i < TC_STAGES; ++i) { mbar_init(full + i, 1); mbar_init(empty + i, 1); mbar_init(conv_done + i, NSPLIT); }
        mbar_init(acc_ready, 1);
        mbar_init(b2_full, 1);
        mbar_init(acc2_ready, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 1) {  // one full warp allocates BN TMEM columns (power of two >= 32)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    // ---- which brick
    int x0 = 0, y0 = 0, z0 = 0, x1 = 0, y1 = 0, z1 = 0;
    if constexpr (KS == 0) {
        // GEMM mode: rows instead of bricks (x0 = first row, set below)
    } else if (a.tiles) {
        const int32_t *t = a.tiles + (size_t)blockIdx.x * 8;
        x0 = t[0]; y0 = t[1]; z0 = t[2]; x1 = t[3]; y1 = t[4]; z1 = t[5];
    } else {
        const int tz = blockIdx.x % a.tiles_z, ty = (blockIdx.x / a.tiles_z) % a.tiles_y, tx = blockIdx.x / (a.tiles_z * a.tiles_y);
        x0 = tx * TC_BX; y0 = ty * TC_BY; z0 = tz * TC_BZ;
        x1 = min(x0 + TC_BX, a.X); y1 = min(y0 + TC_BY, a.Y); z1 = min(z0 + TC_BZ, a.Z);
    }
    const int n0 = blockIdx.y * BN;
    const int kchunks = a.cin / KC;
    constexpr int TAPS = KS == 3 ? 9 : KS == 2 ? 8 : 1;  // pipeline steps per K slice: 9 (dy,dz) pairs (3x3x3), 8 taps (2x2x2/s2), else 1
    int total = TAPS * kchunks, chunk0 = 0;
    if constexpr (KS == 0) {  // split-K GEMM: this CTA owns K chunks [chunk0, chunk0 + total)
        chunk0 = blockIdx.z * a.gemm_chunks_per_split;
        total = max(0, min(a.gemm_chunks_per_split, kchunks - chunk0));
        x0 = blockIdx.x * TC_BM;  // row offset m0
    }

    if (threadIdx.x == 0) {
        // ===== TMA producer =====
        if constexpr (N2 > 0) {
            mbar_expect_tx(b2_full, B2_BYTES);
#pragma unroll
            for (int h = 0; h < (X3 == 1 ? 2 : 1); ++h)  // X3 = 1: rows [N2, 2 N2) of the split W3 are the low parts
#pragma unroll
                for (int kc = 0; kc < BN / 32; ++kc)  // X3 = 2: one 64-half row per K slice = [32 hi | 32 lo]
                    tma_load_2d(smem_b2 + (h * (BN / 32) + kc) * B2_SLICE, &tmB2, b2_full, kc * (XH ? 64 : 32), h * N2);
        }
        for (int it = 0; it < total; ++it) {
            const int s = it % TC_STAGES;
            const uint32_t ph = (it / TC_STAGES) & 1;
            mbar_wait(empty + s, ph ^ 1);
            mbar_expect_tx(full + s, STAGE_BYTES - (X3 == 1 ? A_BYTES : 0));  // X3 = 1: A_lo is written by the splitter warps, not by TMA
            const int tap = it / kchunks, kc = it - tap * kchunks;
            uint8_t *sa = smem + s * STAGE_BYTES;
            if constexpr (KS == 0) {
                tma_load_2d(sa, &tmA, full + s, (chunk0 + it) * KC, x0);
                tma_load_2d(sa + B_OFF, &tmB, full + s, (chunk0 + it) * KC * (XH ? 2 : 1), n0);
                if constexpr (X3 == 1) tma_load_2d(sa + B_OFF + B_BYTES, &tmB, full + s, (chunk0 + it) * KC, a.cout + n0);
            } else if constexpr (KS == 1) {
                tma_load_4d(sa, &tmA, full + s, kc * KC, z0, y0, x0);
                tma_load_2d(sa + B_OFF, &tmB, full + s, kc * KC * (XH ? 2 : 1), n0);
                if constexpr (X3 == 1) tma_load_2d(sa + B_OFF + B_BYTES, &tmB, full + s, kc * KC, a.cout + n0);
            } else if constexpr (KS == 2) {
                // 2x2x2 / stride 2: the tensor map traverses the input with element strides {1,2,2,2}, so the box that starts
                // at input voxel (2 x0 + dx, 2 y0 + dy, 2 z0 + dz) lands as the 128 output rows of this brick for tap (dx,dy,dz)
                const int dx = tap >> 2, dy = (tap >> 1) & 1, dz = tap & 1;
                tma_load_4d(sa, &tmA, full + s, kc * KC, 2 * z0 + dz, 2 * y0 + dy, 2 * x0 + dx);
                tma_load_2d(sa + B_OFF, &tmB, full + s, (tap * a.cin + kc * KC) * (XH ? 2 : 1), n0);
                if constexpr (X3 == 1) tma_load_2d(sa + B_OFF + B_BYTES, &tmB, full + s, tap * a.cin + kc * KC, a.cout + n0);
            } else {
                const int dy = tap / 3, dz = tap % 3;  // tap = (dy, dz) pair; the slab covers x0-1 .. x0+8
                tma_load_4d(sa, &tmA, full + s, kc * KC, z0 + dz - 1, y0 + dy - 1, x0 - 1);
#pragma unroll
                for (int j = 0; j < NBT; ++j) {  // weight tiles: x-taps 0..2 (X3 = 1: hi tiles, then the low parts' tiles)
                    const int dx = j % 3, row0 = (j >= 3 ? a.cout : 0) + n0;
                    // weight columns k = ((dx*3+dy)*3+dz)*C_in + c  (X3 = 2: two halves per k -- [32 hi | 32 lo] per K slice)
                    const int kcol = (((dx * 3 + dy) * 3 + dz) * a.cin + kc * KC) * (XH ? 2 : 1);
                    tma_load_2d(sa + B_OFF + j * B_BYTES, &tmB, full + s, kcol, row0);
                }
            }
        }
    } else if (threadIdx.x == 32) {
        // ===== MMA issuer =====
        // instruction descriptor (cute::UMMA::InstrDescriptor): D=F32 [4,6)=1, A=TF32 [7,10)=2, B=TF32 [10,13)=2,
        // A,B K-major, N>>3 at [17,23), M>>4 at [24,29)
        constexpr uint32_t fmt = (EB == 4 && !XH) ? 2u : 0u;  // F16F32Format: 2 = TF32, 0 = F16
        const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
        for (int it = 0; it < total; ++it) {
            const int s = it % TC_STAGES;
            const uint32_t ph = (it / TC_STAGES) & 1;
            mbar_wait(X3 ? conv_done + s : full + s, ph);  // X3: the split (which itself waited for the TMA) is done
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t sa = smem_u32(smem + s * STAGE_BYTES), sb = sa + B_OFF;
            // operand tiles: X3 = 1: hi at sa (in place), lo at sa + A_BYTES; X3 = 2: fp16 hi at sa (in place), lo half an A_BYTES on
            const uint32_t a_hi = sa, a_lo = sa + (XH ? A_BYTES / 2 : A_BYTES);
#pragma unroll
            for (int dx = 0; dx < XT; ++dx) {
                // x-tap dx: A rows start 16 rows (= two 8-row swizzle atoms) further into the slab
                const uint32_t ax = a_hi + dx * (TC_BY * TC_BZ) * OPB, al_x = a_lo + dx * (TC_BY * TC_BZ) * OPB, bx = sb + dx * B_BYTES;
#pragma unroll
                for (int k = 0; k < OPB / 32; ++k) {  // one MMA consumes 32 B of K (8 tf32 / 16 f16): advance inside the swizzle atom
                    const uint32_t acc = (it | dx | k) ? 1u : 0u;
                    if constexpr (X3) {  // cross terms A_lo.B_hi + A_hi.B_lo -> accumulator 3; A_hi.B_hi -> accumulator it % 3
                        const uint64_t ah = umma_desc<OPB>(ax + k * 32), al = umma_desc<OPB>(al_x + k * 32);
                        const uint64_t bh = umma_desc<BROW>(bx + k * 32);
                        const uint64_t bl = XH ? umma_desc<BROW>(bx + 64 + k * 32) : umma_desc<BROW>(bx + XT * B_BYTES + k * 32);
                        const uint32_t dm = tmem_base + (uint32_t)((it % 3) * BN), acc_m = ((it >= 3) | dx | k) ? 1u : 0u;
                        if constexpr (XH) {
                            umma_f16(tmem_base + 3 * BN, al, bh, idesc, acc);
                            umma_f16(tmem_base + 3 * BN, ah, bl, idesc, 1u);
                            umma_f16(dm, ah, bh, idesc, acc_m);
                        } else {
                            umma_tf32(tmem_base + 3 * BN, al, bh, idesc, acc);
                            umma_tf32(tmem_base + 3 * BN, ah, bl, idesc, 1u);
                            umma_tf32(dm, ah, bh, idesc, acc_m);
                        }
                    } else if constexpr (EB == 4) umma_tf32(tmem_base, umma_desc<ROWB>(ax + k * 32), umma_desc<ROWB>(bx + k * 32), idesc, acc);
                    else umma_f16(tmem_base, umma_desc<ROWB>(ax + k * 32), umma_desc<ROWB>(bx + k * 32), idesc, acc);
                }
            }
            umma_commit(empty + s);  // frees the smem slot once these MMAs retire
        }
        umma_commit(acc_ready);
    } else if (X3 && warp >= 2) {
        // ===== operand splitter (warps 2-3) =====
        const int t = threadIdx.x - 64;
        for (int it = 0; it < total; ++it) {
            const int s = it % TC_STAGES;
            mbar_wait(full + s, (it / TC_STAGES) & 1);
            uint8_t *st = smem + s * STAGE_BYTES;
            if constexpr (XH) {
                // fp32 slab (128-byte rows, SWIZZLE_128B: 16-byte chunk j of row r at r*128 + ((j ^ (r & 7)) << 4)) ->
                // fp16 hi / lo tiles (64-byte rows, SWIZZLE_64B: chunk q of row r at r*64 + ((q ^ ((r >> 1) & 3)) << 4)), IN PLACE:
                // hi takes the first half of the slab's bytes, lo the second.  One work item = 8 channels of one row = source
                // chunks 2q, 2q+1 -> destination chunk q.  Every splitter thread converts its items into registers, the splitter
                // warps meet at a named barrier (all of the fp32 data has been read), then the fp16 tiles are stored.
                constexpr int ITEMS = (A_ROWS * 4 + NSPLIT - 1) / NSPLIT;
                uint4 h[ITEMS], l[ITEMS];
#pragma unroll
                for (int u = 0; u < ITEMS; ++u) {
                    const int i = t + u * NSPLIT;
                    if (i < A_ROWS * 4) {
                        const int r = i >> 2, q = i & 3;
                        const float4 v0 = *reinterpret_cast<const float4 *>(st + r * 128 + (((2 * q) ^ (r & 7)) << 4));
                        const float4 v1 = *reinterpret_cast<const float4 *>(st + r * 128 + (((2 * q + 1) ^ (r & 7)) << 4));
                        split_f16x8(v0, v1, h[u], l[u]);
                    }
                }
                asm volatile("bar.sync 1, %0;" ::"n"(NSPLIT) : "memory");
#pragma unroll
                for (int u = 0; u < ITEMS; ++u) {
                    const int i = t + u * NSPLIT;
                    if (i < A_ROWS * 4) {
                        const int r = i >> 2, q = i & 3;
                        const int d = r * 64 + ((q ^ ((r >> 1) & 3)) << 4);
                        *reinterpret_cast<uint4 *>(st + d) = h[u];
                        *reinterpret_cast<uint4 *>(st + A_BYTES / 2 + d) = l[u];
                    }
                }
            } else {
                // slab -> hi (in place) + lo (second buffer): the split is elementwise, so the swizzled layout is untouched
                float4 *hi = reinterpret_cast<float4 *>(st);
                float4 *lo = reinterpret_cast<float4 *>(st + A_BYTES);
#pragma unroll 2
                for (int i = t; i < A_BYTES / 16; i += NSPLIT) {
                    const float4 v = hi[i];
                    float4 h, l;
                    split_tf32(v.x, h.x, l.x); split_tf32(v.y, h.y, l.y); split_tf32(v.z, h.z, l.z); split_tf32(v.w, h.w, l.w);
                    hi[i] = h;
                    lo[i] = l;
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy stores -> visible to the MMA's async proxy
            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(conv_done + s)) : "memory");
        }
    }
    __syncwarp();
    if constexpr (KS == 0) {
        // ===== GEMM epilogue: raw fp32 partial sums of this K split -> partial[z][m][n] (bias/ReLU in the reduce pass)
        if (total > 0) mbar_wait(acc_ready, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int m = x0 + (int)(threadIdx.x & 127);
        float *prow = a.out + ((int64_t)blockIdx.z * a.gemm_m + m) * a.out_ld + n0;
#pragma unroll 1
        for (int c = (int)(threadIdx.x >> 7); c < BN / 32; c += NHALF) {
            float v[32];
            acc_ld32<X3>(tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(c * 32), min(total, 3), BN, 3 * BN, v);
            if (m < a.gemm_m) {
#pragma unroll
                for (int j = 0; j < 32; j += 4)
                    *reinterpret_cast<float4 *>(prow + c * 32 + j) =
                        total > 0 ? make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
        return;
    }

    // ===== epilogue: TMEM lane r == output row r of the brick =====
    mbar_wait(acc_ready, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const int r = threadIdx.x & 127, half = threadIdx.x >> 7;  // row of the brick / which half of the column chunks
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    uint32_t acc_col = 0;  // first TMEM column of the accumulator the store loop reads
    if constexpr (N2 > 0) {
        // conv2's tile -> ReLU -> shared memory as the A operand of the 1x1 conv: row r, 16-byte chunk j of K slice kc at
        // kc*16 KB + r*128 + ((j ^ (r & 7)) << 4)  (the canonical SWIZZLE_128B K-major layout TMA would have produced)
        uint8_t *a2 = smem;  // aliases the pipeline stages: every TMA write landed and every MMA reading them retired
        // one K slice (32 channels) of the A operand of the 1x1 conv: 128 rows x 128 B (fp32 / TF32 split) or x 64 B (fp16 split);
        // X3: the low parts follow as a second set of slices of the same layout
        constexpr int A2_SLICE = TC_BM * (XH ? 64 : 128);
        constexpr int A2_BYTES = (BN / 32) * A2_SLICE;
#pragma unroll 1
        for (int kc = half; kc < BN / 32; kc += NHALF) {
            float v[32];
            acc_ld32<X3>(tmem_base + lane_base + (uint32_t)(kc * 32), min(total, 3), BN, 3 * BN, v);
            uint8_t *row = a2 + kc * A2_SLICE + r * (XH ? 64 : 128);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float4 o = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                if (a.bias_mid) {
                    const float4 b = __ldg(reinterpret_cast<const float4 *>(a.bias_mid + kc * 32 + 4 * j));
                    o.x += b.x; o.y += b.y; o.z += b.z; o.w += b.w;
                }
                o = make_float4(fmaxf(o.x, 0.f), fmaxf(o.y, 0.f), fmaxf(o.z, 0.f), fmaxf(o.w, 0.f));
                if constexpr (XH) {
                    v[4 * j] = o.x; v[4 * j + 1] = o.y; v[4 * j + 2] = o.z; v[4 * j + 3] = o.w;  // split below, 8 channels per chunk
                } else if constexpr (X3 == 1) {
                    float4 h, l;
                    split_tf32(o.x, h.x, l.x); split_tf32(o.y, h.y, l.y); split_tf32(o.z, h.z, l.z); split_tf32(o.w, h.w, l.w);
                    *reinterpret_cast<float4 *>(row + ((j ^ (r & 7)) << 4)) = h;
                    *reinterpret_cast<float4 *>(row + A2_BYTES + ((j ^ (r & 7)) << 4)) = l;
                } else {
                    *reinterpret_cast<float4 *>(row + ((j ^ (r & 7)) << 4)) = o;
                }
            }
            if constexpr (XH) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {  // 16-byte chunk q = channels 8q..8q+7 of this slice, SWIZZLE_64B position
                    uint4 h, l;
                    split_f16x8(make_float4(v[8 * q], v[8 * q + 1], v[8 * q + 2], v[8 * q + 3]),
                                make_float4(v[8 * q + 4], v[8 * q + 5], v[8 * q + 6], v[8 * q + 7]), h, l);
                    const int d = (q ^ ((r >> 1) & 3)) << 4;
                    *reinterpret_cast<uint4 *>(row + d) = h;
                    *reinterpret_cast<uint4 *>(row + A2_BYTES + d) = l;
                }
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy stores -> visible to the MMA's async proxy
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (threadIdx.x == 32) {
            constexpr uint32_t fmt2 = XH ? 0u : 2u;
            const uint32_t idesc2 = (1u << 4) | (fmt2 << 7) | (fmt2 << 10) | ((uint32_t)(N2 >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
            mbar_wait(b2_full, 0);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t sa2 = smem_u32(a2), sb2 = smem_u32(smem_b2);
            constexpr int OP2 = XH ? 64 : 128;
#pragma unroll
            for (int kc = 0; kc < BN / 32; ++kc)
#pragma unroll
                for (int k = 0; k < OP2 / 32; ++k) {
                    const uint64_t ah = umma_desc<OP2>(sa2 + kc * A2_SLICE + k * 32), bh = umma_desc<128>(sb2 + kc * B2_SLICE + k * 32);
                    if constexpr (X3) {
                        const uint64_t al = umma_desc<OP2>(sa2 + A2_BYTES + kc * A2_SLICE + k * 32);
                        const uint64_t bl = XH ? umma_desc<128>(sb2 + kc * B2_SLICE + 64 + k * 32)
                                               : umma_desc<128>(sb2 + (BN / 32 + kc) * B2_SLICE + k * 32);
                        if constexpr (XH) {
                            umma_f16(tmem_base + 4 * BN + N2, al, bh, idesc2, (kc | k) ? 1u : 0u);
                            umma_f16(tmem_base + 4 * BN + N2, ah, bl, idesc2, 1u);
                            umma_f16(tmem_base + 4 * BN, ah, bh, idesc2, (kc | k) ? 1u : 0u);
                        } else {
                            umma_tf32(tmem_base + 4 * BN + N2, al, bh, idesc2, (kc | k) ? 1u : 0u);
                            umma_tf32(tmem_base + 4 * BN + N2, ah, bl, idesc2, 1u);
                            umma_tf32(tmem_base + 4 * BN, ah, bh, idesc2, (kc | k) ? 1u : 0u);
                        }
                    } else {
                        umma_tf32(tmem_base + BN, ah, bh, idesc2, (kc | k) ? 1u : 0u);
                    }
                }
            umma_commit(acc2_ready);
        }
        __syncwarp();
        mbar_wait(acc2_ready, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        acc_col = X3 ? 4 * BN : BN;
    }
    constexpr int NOUT = N2 > 0 ? N2 : BN;
    const int vz = z0 + (r & (TC_BZ - 1)), vy = y0 + ((r / TC_BZ) % TC_BY), vx = x0 + r / (TC_BZ * TC_BY);
    const bool valid = vx < x1 && vy < y1 && vz < z1;
    const int64_t vox = ((int64_t)vx * a.Y + vy) * a.Z + vz;
    float *orow = a.out ? a.out + vox * a.out_ld + a.out_coff + n0 : nullptr;
    __half *hrow = a.out16 ? a.out16 + vox * a.out_ld + a.out_coff + n0 : nullptr;
    const float *rrow = a.res ? a.res + vox * a.res_ld + a.res_coff + n0 : nullptr;
#pragma unroll 1
    for (int c = half; c < NOUT / 32; c += NHALF) {
        float v[32];
        if constexpr (N2 > 0) acc_ld32<X3>(tmem_base + lane_base + acc_col + (uint32_t)(c * 32), 1, 0, N2, v);
        else acc_ld32<X3>(tmem_base + lane_base + (uint32_t)(c * 32), min(total, 3), BN, 3 * BN, v);
        if (valid) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
                float4 o = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                if (a.bias) {
                    const float4 b = __ldg(reinterpret_cast<const float4 *>(a.bias + n0 + c * 32 + j));
                    o.x += b.x; o.y += b.y; o.z += b.z; o.w += b.w;
                }
                if (rrow) {
                    const float4 q = __ldg(reinterpret_cast<const float4 *>(rrow + c * 32 + j));
                    o.x += q.x; o.y += q.y; o.z += q.z; o.w += q.w;
                }
                if (a.act == 1) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
                if (orow) *reinterpret_cast<float4 *>(orow + c * 32 + j) = o;
                if (hrow) {
                    const __half2 h0 = __floats2half2_rn(o.x, o.y), h1 = __floats2half2_rn(o.z, o.w);
                    uint2 pk;
                    pk.x = *reinterpret_cast<const uint32_t *>(&h0);
                    pk.y = *reinterpret_cast<const uint32_t *>(&h1);
                    *reinterpret_cast<uint2 *>(hrow + c * 32 + j) = pk;
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
}

__global__ void gemm_splitk_reduce_kernel(const float *part, int splits, int64_t split_stride, const float *bias, float *y, int M,
                                          int N, int act) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M * N) return;
    float v = 0.f;
    for (int s = 0; s < splits; ++s) v += part[(int64_t)s * split_stride + i];  // fixed order -> deterministic
    if (bias) v += bias[i % N];
    if (act == 1) v = fmaxf(v, 0.f);
    y[i] = v;
}

// weights [cout][cin][3][3][3] -> [cout][27*cin] with k = tap*cin + c
__global__ void pack_conv_weight_tc_kernel(const float *w, int cout, int cin, int taps, float *out) {
    const int64_t total = (int64_t)cout * taps * cin;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % cin);
        const int tap = (int)((i / cin) % taps);
        const int n = (int)(i / ((int64_t)cin * taps));
        out[i] = w[((int64_t)n * cin + c) * taps + tap];
    }
}

// 3xTF32 weights: rows [0, cout) = tf32(w) (round to nearest), rows [cout, 2 cout) = tf32(w - tf32(w)); same k order
__global__ void pack_conv_weight_tc_x3_kernel(const float *w, int cout, int cin, int taps, float *out) {
    const int64_t total = (int64_t)cout * taps * cin;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % cin);
        const int tap = (int)((i / cin) % taps);
        const int n = (int)(i / ((int64_t)cin * taps));
        float hi, lo;
        split_tf32(w[((int64_t)n * cin + c) * taps + tap], hi, lo);
        out[i] = hi;
        out[total + i] = lo;
    }
}

// fp16-split weights [cout][K/32][64]: per 32-channel K slice (k = tap*cin + c) 32 hi halves = fp16(w), then 32 lo halves =
// fp16((w - fp16(w)) * 2048) -- one 128-byte row per (output channel, K slice), so a TMA box row carries both parts
__global__ void pack_conv_weight_tc_h3_kernel(const float *w, int cout, int cin, int taps, __half *out) {
    const int64_t total = (int64_t)cout * taps * cin;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % cin);
        const int tap = (int)((i / cin) % taps);
        const int n = (int)(i / ((int64_t)cin * taps));
        __half hi, lo;
        split_f16(w[((int64_t)n * cin + c) * taps + tap], hi, lo);
        const int64_t k = (int64_t)tap * cin + c;
        const int64_t o = ((int64_t)n * taps * cin + (k & ~(int64_t)31)) * 2 + (k & 31);
        out[o] = hi;
        out[o + 32] = lo;
    }
}

// fp32 [cout][cin][taps] -> fp16 [cout][taps*cin] (k = tap*cin + c), round to nearest even
__global__ void pack_conv_weight_tc_f16_kernel(const float *w, int cout, int cin, int taps, __half *out) {
    const int64_t total = (int64_t)cout * taps * cin;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % cin);
        const int tap = (int)((i / cin) % taps);
        const int n = (int)(i / ((int64_t)cin * taps));
        out[i] = __float2half_rn(w[((int64_t)n * cin + c) * taps + tap]);
    }
}
// VC fp32 (row stride in_ld, channel offset in_coff) -> dense VC fp16 [rows][C]
__global__ void cast_f16_kernel(const float *in, int in_ld, int in_coff, int64_t rows, int C4, __half *out) {
    const int64_t total = rows * C4;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / C4;
        const int c = (int)(i - r * C4) * 4;
        const float4 v = __ldg(reinterpret_cast<const float4 *>(in + r * in_ld + in_coff + c));
        const __half2 h0 = __floats2half2_rn(v.x, v.y), h1 = __floats2half2_rn(v.z, v.w);
        uint2 pk;
        pk.x = *reinterpret_cast<const uint32_t *>(&h0);
        pk.y = *reinterpret_cast<const uint32_t *>(&h1);
        *reinterpret_cast<uint2 *>(out + r * (int64_t)C4 * 4 + c) = pk;
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {  // resolved through the runtime so libsis3d.so has no link-time dependency on libcuda
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

// ---- operand formats -------------------------------------------------------------------------------------------------------
// One kernel serves four operand formats; a format fixes the kernel's EB / ROWB / X3, the element types of the two tensor maps
// and the shape of the packed weight matrix.  Every box row is one swizzle span (128 or 64 bytes: SWIZZLE_128B / _64B).
enum class TcFormat {
    TF32,    // fp32 storage, kind::tf32
    TF32X3,  // fp32 storage, split 3xTF32 (64-byte K rows so the hi and lo tiles fit the same shared memory)
    F16X3,   // fp32 activations split in shared memory, pre-split fp16 weights, kind::f16
    FP16,    // fp16 storage, kind::f16
};
struct TcFormatInfo {
    int ab;                   // activation element bytes
    int eb, rowb, x3;         // kernel template parameters EB, ROWB, X3
    int wb;                   // weight element bytes (4: fp32, 2: fp16)
    int kmul, nmul;           // packed weights are [cout * nmul][K * kmul]: f16x3 [32 hi | 32 lo] per 32-channel K slice,
                              // tf32x3 hi rows then lo rows
    int kc;                   // channels per pipeline stage (rowb / eb)
    int bn_max;               // widest N tile
};
// fp16 storage: 64 channels per 128-byte row when cin allows it, else 32 per 64-byte row (C_in = 32), with N tiles of at most 64
static TcFormatInfo tc_format(TcFormat f, int cin) {
    switch (f) {
        case TcFormat::TF32: return {4, 4, 128, 0, 4, 1, 1, 32, 128};
        case TcFormat::TF32X3: return {4, 4, 64, 1, 4, 1, 2, 16, 128};
        case TcFormat::F16X3: return {4, 4, 128, 2, 2, 2, 1, 32, 128};
        default: return cin % 64 == 0 ? TcFormatInfo{2, 2, 128, 0, 2, 1, 1, 64, 128} : TcFormatInfo{2, 2, 64, 0, 2, 1, 1, 32, 64};
    }
}

// ---- tensor maps -----------------------------------------------------------------------------------------------------------
static CUtensorMapDataType tc_elem_type(int bytes) { return bytes == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16; }
static CUtensorMapSwizzle tc_row_swizzle(int row_bytes) { return row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B; }

// A operand of the convolutions: the VC activation [X][Y][Z][cin], one box = kc channels of a (16/by) x by x 8 brick, plus a
// one-plane x halo for ks = 3.  ks = 2 (stride 2, pad 0) traverses the input with element strides {1,2,2,2}; a box is given
// in traversed elements, so N loaded voxels = box / stride.
static bool encode_act(CUtensorMap *m, const TcFormatInfo &f, const void *in, int X, int Y, int Z, int cin, int ks, int by) {
    const int sd = ks == 2 ? 2 : 1, bx = 16 / by;
    cuuint64_t dims[4] = {(cuuint64_t)cin, (cuuint64_t)Z, (cuuint64_t)Y, (cuuint64_t)X};
    cuuint64_t strides[3] = {(cuuint64_t)cin * f.ab, (cuuint64_t)Z * cin * f.ab, (cuuint64_t)Y * Z * cin * f.ab};
    cuuint32_t box[4] = {(cuuint32_t)f.kc, (cuuint32_t)(TC_BZ * sd), (cuuint32_t)(by * sd), (cuuint32_t)((ks == 3 ? bx + 2 : bx) * sd)};
    cuuint32_t estr[4] = {1, (cuuint32_t)sd, (cuuint32_t)sd, (cuuint32_t)sd};
    return get_encode()(m, tc_elem_type(f.ab), 4, (void *)in, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        tc_row_swizzle(f.kc * f.ab), CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// a row-major [rows][cols] matrix of eb-byte elements in boxes of box_rows x box_cols: packed weights (L2_256B promotion),
// the fused tail's W3 and the GEMM's activations (L2_128B)
static bool encode_mat(CUtensorMap *m, int eb, const void *p, int64_t cols, int64_t rows, int box_cols, int box_rows,
                       CUtensorMapL2promotion l2) {
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)cols * eb};
    cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    return get_encode()(m, tc_elem_type(eb), 2, (void *)p, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        tc_row_swizzle(box_cols * eb), l2, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
constexpr CUtensorMapL2promotion kWeightL2 = CU_TENSOR_MAP_L2_PROMOTION_L2_256B;

// ---- kernel variants -------------------------------------------------------------------------------------------------------
template <int BN, int KS, int EB, int ROWB, int BY, int N2, int X3>
static int launch_tc(const CUtensorMap &tmA, const CUtensorMap &tmB, const CUtensorMap &tmB2, const TcArgs &a, int n_tiles,
                     int grid_z, cudaStream_t s) {
    const size_t smem = tc_smem_bytes<BN, KS, ROWB, BY, N2, X3>();
    auto kern = conv3d_k3_tc_kernel<BN, KS, EB, ROWB, BY, N2, X3>;
    static bool attr_done = false;
    if (!attr_done) {
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return SIS3D_ELAUNCH;
        attr_done = true;
    }
    kern<<<dim3(n_tiles, N2 > 0 ? 1 : a.cout / BN, grid_z), X3 == 2 ? 256 : 128, smem, s>>>(tmA, tmB, tmB2, a);
    return finish_launch();
}

struct TcVariant {
    int bn, ks, eb, rowb, by, n2, x3;
    int (*launch)(const CUtensorMap &, const CUtensorMap &, const CUtensorMap &, const TcArgs &, int, int, cudaStream_t);
};
#define TC_VARIANT(BN, KS, EB, ROWB, BY, N2, X3) {BN, KS, EB, ROWB, BY, N2, X3, launch_tc<BN, KS, EB, ROWB, BY, N2, X3>}
// Every instantiation of conv3d_k3_tc_kernel.  KS = 0 is the GEMM; N2 > 0 the fused bottleneck tail (BN = cmid, N2 = cout);
// BY = 4 the 4x4x8 bricks of tile lists with cout = 64.
static const TcVariant kTcVariants[] = {
    // tf32
    TC_VARIANT(32, 3, 4, 128, 2, 0, 0), TC_VARIANT(64, 3, 4, 128, 2, 0, 0), TC_VARIANT(128, 3, 4, 128, 2, 0, 0),
    TC_VARIANT(64, 3, 4, 128, 4, 0, 0),
    TC_VARIANT(32, 2, 4, 128, 2, 0, 0), TC_VARIANT(64, 2, 4, 128, 2, 0, 0), TC_VARIANT(128, 2, 4, 128, 2, 0, 0),
    TC_VARIANT(32, 1, 4, 128, 2, 0, 0), TC_VARIANT(64, 1, 4, 128, 2, 0, 0), TC_VARIANT(128, 1, 4, 128, 2, 0, 0),
    TC_VARIANT(32, 0, 4, 128, 2, 0, 0), TC_VARIANT(64, 0, 4, 128, 2, 0, 0), TC_VARIANT(128, 0, 4, 128, 2, 0, 0),
    TC_VARIANT(32, 3, 4, 128, 2, 32, 0), TC_VARIANT(32, 3, 4, 128, 2, 64, 0), TC_VARIANT(64, 3, 4, 128, 2, 128, 0),
    // tf32x3
    TC_VARIANT(32, 3, 4, 64, 2, 0, 1), TC_VARIANT(64, 3, 4, 64, 2, 0, 1), TC_VARIANT(128, 3, 4, 64, 2, 0, 1),
    TC_VARIANT(32, 2, 4, 64, 2, 0, 1), TC_VARIANT(64, 2, 4, 64, 2, 0, 1), TC_VARIANT(128, 2, 4, 64, 2, 0, 1),
    TC_VARIANT(32, 1, 4, 64, 2, 0, 1), TC_VARIANT(64, 1, 4, 64, 2, 0, 1), TC_VARIANT(128, 1, 4, 64, 2, 0, 1),
    TC_VARIANT(32, 0, 4, 64, 2, 0, 1), TC_VARIANT(64, 0, 4, 64, 2, 0, 1), TC_VARIANT(128, 0, 4, 64, 2, 0, 1),
    TC_VARIANT(32, 3, 4, 64, 2, 32, 1), TC_VARIANT(32, 3, 4, 64, 2, 64, 1), TC_VARIANT(64, 3, 4, 64, 2, 128, 1),
    // f16x3
    TC_VARIANT(32, 3, 4, 128, 2, 0, 2), TC_VARIANT(64, 3, 4, 128, 2, 0, 2), TC_VARIANT(128, 3, 4, 128, 2, 0, 2),
    TC_VARIANT(32, 2, 4, 128, 2, 0, 2), TC_VARIANT(64, 2, 4, 128, 2, 0, 2), TC_VARIANT(128, 2, 4, 128, 2, 0, 2),
    TC_VARIANT(32, 1, 4, 128, 2, 0, 2), TC_VARIANT(64, 1, 4, 128, 2, 0, 2), TC_VARIANT(128, 1, 4, 128, 2, 0, 2),
    TC_VARIANT(32, 0, 4, 128, 2, 0, 2), TC_VARIANT(64, 0, 4, 128, 2, 0, 2), TC_VARIANT(128, 0, 4, 128, 2, 0, 2),
    TC_VARIANT(32, 3, 4, 128, 2, 32, 2), TC_VARIANT(32, 3, 4, 128, 2, 64, 2), TC_VARIANT(64, 3, 4, 128, 2, 128, 2),
    // fp16, 128-byte rows
    TC_VARIANT(32, 3, 2, 128, 2, 0, 0), TC_VARIANT(64, 3, 2, 128, 2, 0, 0), TC_VARIANT(128, 3, 2, 128, 2, 0, 0),
    TC_VARIANT(64, 3, 2, 128, 4, 0, 0),
    TC_VARIANT(32, 1, 2, 128, 2, 0, 0), TC_VARIANT(64, 1, 2, 128, 2, 0, 0), TC_VARIANT(128, 1, 2, 128, 2, 0, 0),
    // fp16, 64-byte rows
    TC_VARIANT(32, 3, 2, 64, 2, 0, 0), TC_VARIANT(64, 3, 2, 64, 2, 0, 0),
    TC_VARIANT(32, 1, 2, 64, 2, 0, 0), TC_VARIANT(64, 1, 2, 64, 2, 0, 0),
};
#undef TC_VARIANT
static const TcVariant *tc_variant(const TcFormatInfo &f, int ks, int bn, int by, int n2) {
    for (const TcVariant &v : kTcVariants)
        if (v.eb == f.eb && v.rowb == f.rowb && v.x3 == f.x3 && v.ks == ks && v.bn == bn && v.by == by && v.n2 == n2) return &v;
    return nullptr;
}

// brick height: explicit tile lists (ragged RoI crops) of 64 -> 64 3x3x3 layers use 4x4x8 bricks, everything else 8x2x8
static int tc_brick_y(bool with_tile_list, int ks, int cin, int cout) {
    return (with_tile_list && ks == 3 && cout == 64 && cin % 64 == 0) ? 4 : 2;
}

}  // namespace sis3d
using namespace sis3d;

template <typename T>
static int pack_tc(void (*kern)(const float *, int, int, int, T *), const float *w, int cout, int cin, int ks, T *out, void *stream) {
    if (!w || !out || cout <= 0 || cin <= 0 || (ks != 1 && ks != 2 && ks != 3)) return SIS3D_EINVAL;
    const int taps = ks * ks * ks;
    const int64_t total = (int64_t)cout * taps * cin;
    kern<<<(int)imin64(cdiv64(total, 256), 148 * 8), 256, 0, (cudaStream_t)stream>>>(w, cout, cin, taps, out);
    return finish_launch();
}
extern "C" int sis3d_pack_conv_weight_tc(const float *w, int cout, int cin, int ks, float *w_tc, void *stream) {
    return pack_tc(pack_conv_weight_tc_kernel, w, cout, cin, ks, w_tc, stream);
}
extern "C" int sis3d_pack_conv_weight_tc_x3(const float *w, int cout, int cin, int ks, float *w_x3, void *stream) {
    return pack_tc(pack_conv_weight_tc_x3_kernel, w, cout, cin, ks, w_x3, stream);
}
extern "C" int sis3d_pack_conv_weight_tc_h3(const float *w, int cout, int cin, int ks, uint16_t *w_h3, void *stream) {
    return pack_tc(pack_conv_weight_tc_h3_kernel, w, cout, cin, ks, (__half *)w_h3, stream);
}
extern "C" int sis3d_pack_conv_weight_tc_f16(const float *w, int cout, int cin, int ks, uint16_t *w16, void *stream) {
    if (ks == 2) return SIS3D_EINVAL;  // fp16 storage has no 2x2x2 kernel
    return pack_tc(pack_conv_weight_tc_f16_kernel, w, cout, cin, ks, (__half *)w16, stream);
}

extern "C" int sis3d_conv3d_k3_tc_supported(int cin, int cout) {
    return (cin % TC_KC == 0 && (cout == 32 || cout == 64 || cout % 128 == 0)) ? 1 : 0;
}

// One convolution in any format.  out16 (an fp16 twin of the output, `out` may then be null) exists only with fp16 storage, which
// has no 2x2x2 kernel; the compensated formats take whole volumes only.
static int conv_tc(TcFormat fmt, const void *in, const void *w, const float *bias, const float *residual, int res_ld, int res_coff,
                   float *out, uint16_t *out16, int out_ld, int out_coff, int X, int Y, int Z, int cin, int cout, int ks,
                   const int32_t *tiles, int n_tiles, int act, void *stream) {
    const bool ks_ok = ks == 1 || ks == 3 || (ks == 2 && fmt != TcFormat::FP16);
    if (!in || !w || (!out && !out16) || X <= 0 || Y <= 0 || Z <= 0 || !ks_ok) return SIS3D_EINVAL;
    if (ks == 2 && (tiles || X < 2 || Y < 2 || Z < 2)) return SIS3D_EINVAL;
    const TcFormatInfo f = tc_format(fmt, cin);
    if (f.x3 && tiles) return SIS3D_EUNSUPPORTED;  // the ragged mask stage does not need the compensated product
    if (!sis3d_conv3d_k3_tc_supported(cin, cout)) return SIS3D_EUNSUPPORTED;
    if (((uintptr_t)in | (uintptr_t)w | (uintptr_t)out | (uintptr_t)out16) & 15) return SIS3D_EINVAL;
    if ((out_ld | out_coff | res_ld | res_coff) & 3) return SIS3D_EINVAL;
    if (!get_encode()) return SIS3D_EUNSUPPORTED;
    if (fmt == TcFormat::FP16 && cin % 64 != 0 && cin != 32) return SIS3D_EUNSUPPORTED;
    const int by = tc_brick_y(tiles != nullptr, ks, cin, cout), bx = 16 / by;
    const int BN = min(cout, f.bn_max);
    const int sd = ks == 2 ? 2 : 1;                   // ks == 2 is the stride-2, pad-0 conv: X, Y, Z are the INPUT extents
    const int Xo = X / sd, Yo = Y / sd, Zo = Z / sd;  // output extents (floor, as nn.Conv3d)
    CUtensorMap tmA, tmB;
    if (!encode_act(&tmA, f, in, X, Y, Z, cin, ks, by) ||
        !encode_mat(&tmB, f.wb, w, (int64_t)ks * ks * ks * cin * f.kmul, (int64_t)cout * f.nmul, f.kc * f.kmul, BN, kWeightL2))
        return SIS3D_EINVAL;
    TcArgs a = {};
    a.bias = bias; a.res = residual; a.out = out; a.out16 = (__half *)out16; a.tiles = tiles;
    a.X = Xo; a.Y = Yo; a.Z = Zo; a.cin = cin; a.cout = cout; a.act = act;
    a.out_ld = out_ld; a.out_coff = out_coff; a.res_ld = res_ld; a.res_coff = res_coff;
    a.tiles_y = cdiv(Yo, by); a.tiles_z = cdiv(Zo, TC_BZ);
    if (!tiles) n_tiles = cdiv(Xo, bx) * a.tiles_y * a.tiles_z;
    if (n_tiles <= 0) return SIS3D_OK;
    const TcVariant *v = tc_variant(f, ks, BN, by, 0);
    return v ? v->launch(tmA, tmB, tmB, a, n_tiles, 1, (cudaStream_t)stream) : SIS3D_EUNSUPPORTED;
}
extern "C" int sis3d_conv3d_k3_tc(const float *in, const float *w_tc, const float *bias, const float *residual, int res_ld,
                                  int res_coff, float *out, int out_ld, int out_coff, int X, int Y, int Z, int cin, int cout,
                                  int ks, const int32_t *tiles, int n_tiles, int act, void *stream) {
    return conv_tc(TcFormat::TF32, in, w_tc, bias, residual, res_ld, res_coff, out, nullptr, out_ld, out_coff, X, Y, Z, cin, cout, ks,
                   tiles, n_tiles, act, stream);
}
// error-compensated 3xTF32 (fp32-class accuracy on the tensor cores): w_x3 from sis3d_pack_conv_weight_tc_x3
extern "C" int sis3d_conv3d_k3_tc_x3(const float *in, const float *w_x3, const float *bias, const float *residual, int res_ld,
                                     int res_coff, float *out, int out_ld, int out_coff, int X, int Y, int Z, int cin, int cout,
                                     int ks, int act, void *stream) {
    return conv_tc(TcFormat::TF32X3, in, w_x3, bias, residual, res_ld, res_coff, out, nullptr, out_ld, out_coff, X, Y, Z, cin, cout,
                   ks, nullptr, 0, act, stream);
}
// the same compensation with an fp16 operand split (2.5x the MMA rate): w_h3 from sis3d_pack_conv_weight_tc_h3
extern "C" int sis3d_conv3d_k3_tc_h3(const float *in, const uint16_t *w_h3, const float *bias, const float *residual, int res_ld,
                                     int res_coff, float *out, int out_ld, int out_coff, int X, int Y, int Z, int cin, int cout,
                                     int ks, int act, void *stream) {
    return conv_tc(TcFormat::F16X3, in, w_h3, bias, residual, res_ld, res_coff, out, nullptr, out_ld, out_coff, X, Y, Z, cin, cout,
                   ks, nullptr, 0, act, stream);
}
// fp16-operand variant (kind::f16): activations and weights stored as fp16, fp32 accumulation in TMEM
extern "C" int sis3d_conv3d_tc_f16(const uint16_t *in16, const uint16_t *w16, const float *bias, const float *residual,
                                   int res_ld, int res_coff, float *out32, uint16_t *out16, int out_ld, int out_coff, int X, int Y,
                                   int Z, int cin, int cout, int ks, const int32_t *tiles, int n_tiles, int act, void *stream) {
    return conv_tc(TcFormat::FP16, in16, w16, bias, residual, res_ld, res_coff, out32, out16, out_ld, out_coff, X, Y, Z, cin, cout, ks,
                   tiles, n_tiles, act, stream);
}
extern "C" int sis3d_cast_f16(const float *in, int in_ld, int in_coff, int64_t rows, int C, uint16_t *out, void *stream) {
    if (!in || !out || rows <= 0 || C % 4 != 0 || (in_ld | in_coff) & 3) return SIS3D_EINVAL;
    cast_f16_kernel<<<(int)imin64(cdiv64(rows * (C / 4), 256), 148 * 8), 256, 0, (cudaStream_t)stream>>>(in, in_ld, in_coff, rows, C / 4, (__half *)out);
    return finish_launch();
}

// ---- bottleneck tail: 3x3x3 conv (cin -> cmid) + ReLU + 1x1 conv (cmid -> cout) + residual + act, one kernel ----------------
extern "C" int sis3d_conv3d_k3_tc_fused_supported(int cin, int cmid, int cout) {
    return (cin % TC_KC == 0 && ((cmid == 32 && (cout == 32 || cout == 64)) || (cmid == 64 && cout == 128))) ? 1 : 0;
}
static int conv_tc_fused(TcFormat fmt, const float *in, const void *w2, const float *bias2, const void *w3, const float *bias3,
                         const float *residual, int res_ld, int res_coff, float *out, int out_ld, int out_coff, int X, int Y, int Z,
                         int cin, int cmid, int cout, int act, void *stream) {
    if (!in || !w2 || !w3 || !out || X <= 0 || Y <= 0 || Z <= 0) return SIS3D_EINVAL;
    if (!sis3d_conv3d_k3_tc_fused_supported(cin, cmid, cout)) return SIS3D_EUNSUPPORTED;
    if (((uintptr_t)in | (uintptr_t)w2 | (uintptr_t)w3 | (uintptr_t)out) & 15) return SIS3D_EINVAL;
    if ((out_ld | out_coff | res_ld | res_coff) & 3) return SIS3D_EINVAL;
    if (!get_encode()) return SIS3D_EUNSUPPORTED;
    const TcFormatInfo f = tc_format(fmt, cin);
    CUtensorMap tmA, tmB, tmB2;
    if (!encode_act(&tmA, f, in, X, Y, Z, cin, 3, 2) ||
        !encode_mat(&tmB, f.wb, w2, (int64_t)27 * cin * f.kmul, (int64_t)cmid * f.nmul, f.kc * f.kmul, cmid, kWeightL2) ||
        !encode_mat(&tmB2, f.wb, w3, (int64_t)cmid * f.kmul, (int64_t)cout * f.nmul, TC_KC * f.kmul, cout, kWeightL2))
        return SIS3D_EINVAL;
    TcArgs a = {};
    a.bias = bias3; a.bias_mid = bias2; a.res = residual; a.out = out;
    // the main loop's weight rows (and their lo halves, x3) are indexed with the 3x3x3 conv's width, the epilogue with cout
    a.X = X; a.Y = Y; a.Z = Z; a.cin = cin; a.cout = f.x3 ? cmid : cout; a.act = act;
    a.out_ld = out_ld; a.out_coff = out_coff; a.res_ld = res_ld; a.res_coff = res_coff;
    a.tiles_y = cdiv(Y, 2); a.tiles_z = cdiv(Z, TC_BZ);
    const int n_tiles = cdiv(X, 8) * a.tiles_y * a.tiles_z;
    const TcVariant *v = tc_variant(f, 3, cmid, 2, cout);
    return v ? v->launch(tmA, tmB, tmB2, a, n_tiles, 1, (cudaStream_t)stream) : SIS3D_EUNSUPPORTED;
}
extern "C" int sis3d_conv3d_k3_tc_fused(const float *in, const float *w2_tc, const float *bias2, const float *w3_tc,
                                        const float *bias3, const float *residual, int res_ld, int res_coff, float *out,
                                        int out_ld, int out_coff, int X, int Y, int Z, int cin, int cmid, int cout, int act,
                                        void *stream) {
    return conv_tc_fused(TcFormat::TF32, in, w2_tc, bias2, w3_tc, bias3, residual, res_ld, res_coff, out, out_ld, out_coff, X, Y, Z,
                         cin, cmid, cout, act, stream);
}
extern "C" int sis3d_conv3d_k3_tc_fused_x3(const float *in, const float *w2_x3, const float *bias2, const float *w3_x3,
                                           const float *bias3, const float *residual, int res_ld, int res_coff, float *out,
                                           int out_ld, int out_coff, int X, int Y, int Z, int cin, int cmid, int cout, int act,
                                           void *stream) {
    return conv_tc_fused(TcFormat::TF32X3, in, w2_x3, bias2, w3_x3, bias3, residual, res_ld, res_coff, out, out_ld, out_coff, X, Y,
                         Z, cin, cmid, cout, act, stream);
}
extern "C" int sis3d_conv3d_k3_tc_fused_h3(const float *in, const uint16_t *w2_h3, const float *bias2, const uint16_t *w3_h3,
                                           const float *bias3, const float *residual, int res_ld, int res_coff, float *out,
                                           int out_ld, int out_coff, int X, int Y, int Z, int cin, int cmid, int cout, int act,
                                           void *stream) {
    return conv_tc_fused(TcFormat::F16X3, in, w2_h3, bias2, w3_h3, bias3, residual, res_ld, res_coff, out, out_ld, out_coff, X, Y,
                         Z, cin, cmid, cout, act, stream);
}

// ---- y[M][N] = act(x[M][K] . w[N][K]^T + b): fully connected layer on the tensor cores, split-K ------------------------------
static int gemm_tc_splits(int M, int N, int K, int kc) {
    const int tiles = cdiv(M, TC_BM) * (N / (N >= 128 ? 128 : N));
    const int chunks = K / kc;
    int splits = max(1, min(chunks / (128 / kc), (kNumSMs + tiles - 1) / tiles));
    return splits;
}
extern "C" int sis3d_linear_tc_supported(int K, int N) { return (K % TC_KC == 0 && (N == 32 || N == 64 || N % 128 == 0)) ? 1 : 0; }
extern "C" size_t sis3d_linear_tc_workspace_bytes(int M, int N, int K) {
    return sizeof(float) * (size_t)gemm_tc_splits(M, N, K, 16) * M * N + 16;  // the x3 variant splits K finer: covers both
}
static int linear_tc(TcFormat fmt, const float *x, const void *w_nk, const float *bias, float *y, int M, int K, int N, int act,
                     void *workspace, size_t workspace_bytes, void *stream) {
    if (!x || !w_nk || !y || !workspace || M <= 0) return SIS3D_EINVAL;
    if (!sis3d_linear_tc_supported(K, N)) return SIS3D_EUNSUPPORTED;
    if (((uintptr_t)x | (uintptr_t)w_nk | (uintptr_t)workspace) & 15) return SIS3D_EINVAL;
    if (!get_encode()) return SIS3D_EUNSUPPORTED;
    const TcFormatInfo f = tc_format(fmt, K);
    const int BN = min(N, f.bn_max);
    int splits = gemm_tc_splits(M, N, K, f.kc);
    const int chunks = K / f.kc;
    const int per = cdiv(chunks, splits);
    splits = cdiv(chunks, per);
    if (workspace_bytes < sizeof(float) * (size_t)splits * M * N) return SIS3D_EWORKSPACE;
    CUtensorMap tmA, tmB;
    if (!encode_mat(&tmA, 4, x, K, M, f.kc, TC_BM, CU_TENSOR_MAP_L2_PROMOTION_L2_128B) ||
        !encode_mat(&tmB, f.wb, w_nk, (int64_t)K * f.kmul, (int64_t)N * f.nmul, f.kc * f.kmul, BN, kWeightL2))
        return SIS3D_EINVAL;
    TcArgs a = {};
    a.out = (float *)workspace; a.out_ld = N; a.cin = K; a.cout = N; a.gemm_m = M; a.gemm_chunks_per_split = per;
    cudaStream_t s = (cudaStream_t)stream;
    const TcVariant *v = tc_variant(f, 0, BN, 2, 0);
    const int rc = v ? v->launch(tmA, tmB, tmB, a, cdiv(M, TC_BM), splits, s) : SIS3D_EUNSUPPORTED;
    if (rc) return rc;
    gemm_splitk_reduce_kernel<<<cdiv(M * N, 256), 256, 0, s>>>((const float *)workspace, splits, (int64_t)M * N, bias, y, M, N, act);
    return finish_launch();
}
extern "C" int sis3d_linear_tc(const float *x, const float *w_nk, const float *bias, float *y, int M, int K, int N, int act,
                               void *workspace, size_t workspace_bytes, void *stream) {
    return linear_tc(TcFormat::TF32, x, w_nk, bias, y, M, K, N, act, workspace, workspace_bytes, stream);
}
// w_x3 = sis3d_pack_conv_weight_tc_x3(w[N][K] viewed as a 1x1 conv): [2][N][K]
extern "C" int sis3d_linear_tc_x3(const float *x, const float *w_x3, const float *bias, float *y, int M, int K, int N, int act,
                                  void *workspace, size_t workspace_bytes, void *stream) {
    return linear_tc(TcFormat::TF32X3, x, w_x3, bias, y, M, K, N, act, workspace, workspace_bytes, stream);
}
extern "C" int sis3d_linear_tc_h3(const float *x, const uint16_t *w_h3, const float *bias, float *y, int M, int K, int N, int act,
                                  void *workspace, size_t workspace_bytes, void *stream) {
    return linear_tc(TcFormat::F16X3, x, w_h3, bias, y, M, K, N, act, workspace, workspace_bytes, stream);
}

// brick shape the tensor-core kernel uses for a layer (so callers can build matching tile lists)
extern "C" void sis3d_conv3d_tc_brick(int with_tile_list, int ks, int cin, int cout, int32_t *bx, int32_t *by, int32_t *bz) {
    const int y = tc_brick_y(with_tile_list != 0, ks, cin, cout);
    if (bx) *bx = 16 / y;
    if (by) *by = y;
    if (bz) *bz = TC_BZ;
}
