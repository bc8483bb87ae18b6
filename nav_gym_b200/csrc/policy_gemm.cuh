// policy_gemm.cuh -- part of navgym_b200.cu (included there; one translation unit).
// The pedestrian policy's action mean (human_policy.py:38-55; called from env.py:649-656) as three
// sm_100a launches per forward, every contraction on the 5th-generation tensor cores (the weights
// are laid out for them once, by policy_prepare_kernel):
//
//   policy_features_umma2_kernel  the convolutional front end: scan -> features F [n][4096] as f16 pairs.
//   dense_umma_kernel   <Fc1, 0>: H = relu(F W1^T + b1), F [n][4096], W1 [256][4096]: the big dense contraction of
//                       the system; <Fc2, 1>: act_fc2 + the two heads (N 128, K 256).  tcgen05.mma (kind::f16,
//                       M 128 x N 256 x K 16 per instruction, issued by one thread), operands staged
//                       in shared memory by TMA (cp.async.bulk.tensor, 64-byte swizzle),
//                       accumulators in tensor memory (2 x 256 columns: the epilogue of one tile
//                       overlaps the main loop of the next), read back with tcgen05.ld.
//
// Float32-grade results from the f16 tensor pipe ("f16x3"): every float32 operand x is carried as
// two halves, hi = half(x * s) and lo = half(x * s - hi) with s a power of two chosen from the
// weights so that nothing overflows and the low parts stay out of the subnormal range; hi + lo
// holds 22-24 significant bits of x, products of halves are exact in the float32 accumulator,
// and F W^T = Fh Wh^T + Fl Wh^T + Fh Wl^T up to the dropped Fl Wl^T (2^-22 relative).  Three
// f16 MMAs cost what 1.5 TF32 MMAs would, the operands move as 4 bytes per element (what the
// float32 feature row cost before), and the accuracy is that of a float32 GEMM (tests: means
// within 2e-5 of the reference's float32 CPU forward).
//
// Roofline (DESIGN.md 4.3): 3 x 2 x n x 4096 x 256 flop; at n = 40 960: 258 GFLOP, 0.115 ms at the
// 2.25 PFLOP/s f16 peak.  Per 128-pedestrian tile and 64-wide K block the CTA needs 32 KB of F
// (hi + lo, streamed from HBM once) and 64 KB of W (hi + lo, L2-resident, 4 MB in all) for 1536
// tensor-core cycles: 64 B/clk per SM against ~43 B/clk that L2 sustains per SM with all 148 SMs
// pulling -- the kernel is L2-feed-bound at ~2/3 of the tensor peak.
#include <cuda.h>
#include <cuda_fp16.h>

namespace pg {
// K block of a pipeline stage: 32 f16 = 64-byte rows (64-byte swizzle, 4 stages of 48 KB: the same
// bytes per MMA cycle as 64-wide blocks in 2 stages of 96 KB, but three stages in flight instead of
// one while a stage is being multiplied)
constexpr int BM = 128, BK = 32, UK = 16;
// one dense layer on the tensor cores: BN outputs, KDIM inputs (act_fc1: 256 x 4096; act_fc2: 128 x 256)
template <int BN_, int KDIM_>
struct Dense {
    static constexpr int BN = BN_, KDIM = KDIM_, KB = KDIM_ / BK;
    static constexpr int WBOX = BN_ > 128 ? 64 : BN_;   // weight rows per TMA box (a leftover tile's N parts are multiples of it)
    static constexpr uint32_t A_BYTES = BM * BK * 2;                      // 128 rows x 64 B
    static constexpr uint32_t B_BYTES = BN_ * BK * 2;
    static constexpr uint32_t STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;    // A hi, A lo, W hi, W lo
    static constexpr int STAGES = (192 * 1024) / STAGE_BYTES;
    static constexpr uint32_t SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /* alignment slack */ + 256 /* barriers */;
    // Instruction descriptor, kind::f16: D float32 (bits 4-5 = 1), A and B f16 (0), both K-major,
    // N >> 3 at bit 17, M >> 4 at bit 24.
    static constexpr uint32_t IDESC = (1u << 4) | ((uint32_t)(BN_ >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
    static_assert(2 * BN_ <= 512, "two accumulators in tensor memory");
};
using Fc1 = Dense<256, 4096>;
using Fc2 = Dense<128, 256>;
constexpr int THREADS = 192;                                   // warp 0 TMA, warp 1 MMA, warps 2-5 epilogue
constexpr uint32_t TMEM_COLS = 512;

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    uint32_t ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\t"
                     "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                     "selp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, int c0, int c1, uint32_t bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(bar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// D[tmem] (+)= A[smem] B[smem]^T, both operands K-major; issued by one thread for the CTA
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrive on an mbarrier once every MMA issued so far by this thread has completed
__device__ __forceinline__ void umma_commit(uint32_t bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// Shared-memory matrix descriptor of a K-major tile whose rows are 64 bytes, laid out by TMA
// with the 64-byte swizzle: 8-row groups 512 B apart (stride byte offset), descriptor version
// 1 (sm_100), layout type 4 (SWIZZLE_64B); the leading byte offset is unused for this layout.
__device__ __forceinline__ uint64_t umma_desc_sw64(uint32_t smem_addr)
{
    return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(512 >> 4) << 32) |
           ((uint64_t)1 << 46) | ((uint64_t)4 << 61);
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                   "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                   "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
}  // namespace pg

__device__ __forceinline__ uint32_t pack_half2(float a, float b)
{
    const __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<const uint32_t *>(&h);
}
// (hi, lo) f16 pairs of two floats: hi = half(x), lo = half(x - hi)
__device__ __forceinline__ void split2(float a, float b, uint32_t &hi, uint32_t &lo)
{
    const __half2 h = __floats2half2_rn(a, b);
    const float2 back = __half22float2(h);
    hi = *reinterpret_cast<const uint32_t *>(&h);
    lo = pack_half2(a - back.x, b - back.y);
}

// dense_umma_kernel<L, EPI>: Y = A W^T in the f16x3 scheme, A = (a_hi, a_lo) [n][KDIM] and W = (w_hi, w_lo)
// [BN][KDIM] f16 pairs behind TMA maps; 128-row tiles, persistent over tiles.
//   EPI 0 (act_fc1): h = relu(Y descale + bias), written as f16 hi/lo pairs times s_h2 -- the A operand of the
//          act_fc2 launch; scales[1] = descale, scales[6] = s_h2.
//   EPI 1 (act_fc2 + heads, human_policy.py:51-55): y = relu(Y descale + b2 + [goal, speed] . w2[:, 256:260]),
//          mean = (sigmoid(y . a1 + a1_b), tanh(y . a2 + a2_b)); tab = [7][128] b2, the four extra input columns
//          of fc2's weight, a1_w, a2_w, then a1_b, a2_b; scales[7] = descale.  One thread per pedestrian.
template <class L, int EPI>
__global__ void __launch_bounds__(pg::THREADS, 1)
dense_umma_kernel(const __grid_constant__ CUtensorMap tm_ah, const __grid_constant__ CUtensorMap tm_al,
                  const __grid_constant__ CUtensorMap tm_wh, const __grid_constant__ CUtensorMap tm_wl,
                  const float *__restrict__ bias_or_tab, const float *__restrict__ scales, int n, int num_tiles,
                  __half *__restrict__ h_hi, __half *__restrict__ h_lo,
                  const float *__restrict__ goal, const float *__restrict__ speed, float *__restrict__ mean)
{
    using namespace pg;
    constexpr int BN = L::BN, KB = L::KB, STAGES = L::STAGES;
    constexpr uint32_t A_BYTES = L::A_BYTES, B_BYTES = L::B_BYTES, STAGE_BYTES = L::STAGE_BYTES;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;   // swizzled tiles need 1024-byte alignment
    const uint32_t bars = base + STAGES * STAGE_BYTES;
    const uint32_t full0 = bars, empty0 = bars + 8 * STAGES, tfull0 = bars + 16 * STAGES, tempty0 = tfull0 + 16;
    const uint32_t tmem_slot = tempty0 + 16;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < STAGES; s++) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        for (int b = 0; b < 2; b++) { mbar_init(tfull0 + 8 * b, 1); mbar_init(tempty0 + 8 * b, 128); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {   // one warp allocates the tensor memory (and frees it at the end)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");

    // Work items of this CTA: whole tiles round robin while every CTA gets one; the tiles left over
    // for a last, partly filled round (40 960 pedestrians = 320 tiles on 148 SMs: 24) are split along N
    // into SPLIT parts of BN / SPLIT outputs, so that the round costs a fraction of a tile time instead
    // of a whole one (the launch lasted 3 tile times where the average is 2.16).  All three roles walk
    // the same list.
    const int full_rounds = num_tiles / (int)gridDim.x, full = full_rounds * (int)gridDim.x, rem = num_tiles - full;
    int SPLIT = 1;
    if (L::WBOX < BN && rem > 0) SPLIT = rem * 4 <= (int)gridDim.x ? 4 : (rem * 2 <= (int)gridDim.x ? 2 : 1);
    const int n_items = full_rounds + ((int)blockIdx.x < rem * SPLIT ? 1 : 0);
    auto item = [&](int i, int &tile, int &n0, int &bn) {
        if (i < full_rounds) { tile = (int)blockIdx.x + i * (int)gridDim.x; n0 = 0; bn = BN; }
        else { tile = full + (int)blockIdx.x / SPLIT; bn = BN / SPLIT; n0 = ((int)blockIdx.x % SPLIT) * bn; }
    };
    if (warp == 0) {
        // ---- TMA producer: one thread streams the operand tiles of this CTA's items
        if (lane == 0) {
            uint32_t s = 0, ph = 0;
            for (int i = 0; i < n_items; i++) {
                int tile, n0, bn;
                item(i, tile, n0, bn);
                for (int kb = 0; kb < KB; kb++) {
                    mbar_wait(empty0 + 8 * s, ph ^ 1);
                    const uint32_t st = base + s * STAGE_BYTES, fb = full0 + 8 * s;
                    mbar_expect_tx(fb, 2 * A_BYTES + 2 * (uint32_t)bn * BK * 2);
                    tma_load_2d(st, &tm_ah, kb * BK, tile * BM, fb);
                    tma_load_2d(st + A_BYTES, &tm_al, kb * BK, tile * BM, fb);
                    for (int r = 0; r < bn; r += L::WBOX) {   // weight rows n0 .. n0 + bn, WBOX rows per box
                        tma_load_2d(st + 2 * A_BYTES + (uint32_t)r * BK * 2, &tm_wh, kb * BK, n0 + r, fb);
                        tma_load_2d(st + 2 * A_BYTES + B_BYTES + (uint32_t)r * BK * 2, &tm_wl, kb * BK, n0 + r, fb);
                    }
                    if (++s == STAGES) { s = 0; ph ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ---- MMA issuer: one thread issues every tcgen05.mma of the CTA
        if (lane == 0) {
            uint32_t s = 0, ph = 0;
            for (int it = 0; it < n_items; it++) {
                int tile, n0, bn;
                item(it, tile, n0, bn);
                const uint32_t idesc = (1u << 4) | ((uint32_t)(bn >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
                const uint32_t buf = it & 1;
                mbar_wait(tempty0 + 8 * buf, ((it >> 1) & 1) ^ 1);   // the epilogue has drained this accumulator
                tc_fence_after();
                const uint32_t d = tmem_base + buf * BN;
                for (int kb = 0; kb < KB; kb++) {
                    mbar_wait(full0 + 8 * s, ph);
                    tc_fence_after();
                    const uint32_t st = base + s * STAGE_BYTES;
                    const uint64_t fh = umma_desc_sw64(st), fl = umma_desc_sw64(st + A_BYTES);
                    const uint64_t wh = umma_desc_sw64(st + 2 * A_BYTES), wl = umma_desc_sw64(st + 2 * A_BYTES + B_BYTES);
#pragma unroll
                    for (int k = 0; k < BK / UK; k++) {
                        const uint64_t adv = (uint64_t)((k * UK * 2) >> 4);   // 32 bytes along K inside the swizzle atom
                        umma_f16(d, fl + adv, wh + adv, idesc, (kb | k) != 0);
                        umma_f16(d, fh + adv, wl + adv, idesc, 1);
                        umma_f16(d, fh + adv, wh + adv, idesc, 1);
                    }
                    umma_commit(empty0 + 8 * s);   // the stage is free once these MMAs have read it
                    if (++s == STAGES) { s = 0; ph ^= 1; }
                }
                umma_commit(tfull0 + 8 * buf);     // accumulator complete
            }
        }
    } else {
        // ---- epilogue: warp w reads the TMEM lanes 32 (w % 4) ... + 31 = rows of the tile
        const int q = warp & 3;
        for (int it = 0; it < n_items; it++) {
            int tile, n0, bn;
            item(it, tile, n0, bn);
            const uint32_t buf = it & 1;
            mbar_wait(tfull0 + 8 * buf, (it >> 1) & 1);
            tc_fence_after();
            const int row = tile * BM + q * 32 + lane;
            const uint32_t t0 = tmem_base + ((uint32_t)(q * 32) << 16) + buf * BN;
            if (EPI == 0) {
                const float descale = scales[1], s_h2 = scales[6];
#pragma unroll 1
                for (int c = 0; c < bn / 32; c++) {
                    uint32_t v[32];
                    tmem_ld32(t0 + c * 32, v);
                    if (row < n) {
                        const int col = n0 + c * 32;
                        uint32_t hi[16], lo[16];
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            const float4 b = *reinterpret_cast<const float4 *>(bias_or_tab + col + j);
                            float4 o;
                            o.x = fmaxf(fmaf(__uint_as_float(v[j]), descale, b.x), 0.0f);
                            o.y = fmaxf(fmaf(__uint_as_float(v[j + 1]), descale, b.y), 0.0f);
                            o.z = fmaxf(fmaf(__uint_as_float(v[j + 2]), descale, b.z), 0.0f);
                            o.w = fmaxf(fmaf(__uint_as_float(v[j + 3]), descale, b.w), 0.0f);
                            split2(o.x * s_h2, o.y * s_h2, hi[j >> 1], lo[j >> 1]);
                            split2(o.z * s_h2, o.w * s_h2, hi[(j >> 1) + 1], lo[(j >> 1) + 1]);
                        }
                        uint4 *oh = reinterpret_cast<uint4 *>(h_hi + (size_t)row * BN + col);
                        uint4 *ol = reinterpret_cast<uint4 *>(h_lo + (size_t)row * BN + col);
#pragma unroll
                        for (int i = 0; i < 4; i++) {
                            oh[i] = make_uint4(hi[4 * i], hi[4 * i + 1], hi[4 * i + 2], hi[4 * i + 3]);
                            ol[i] = make_uint4(lo[4 * i], lo[4 * i + 1], lo[4 * i + 2], lo[4 * i + 3]);
                        }
                    }
                }
            } else {
                const float descale = scales[7];
                const float *tab = bias_or_tab;
                float g0 = 0.f, g1 = 0.f, p0 = 0.f, p1 = 0.f;
                if (row < n) {   // torch.cat((a, goal, speed)) (human_policy.py:51)
                    g0 = goal[2 * (size_t)row]; g1 = goal[2 * (size_t)row + 1];
                    p0 = speed[2 * (size_t)row]; p1 = speed[2 * (size_t)row + 1];
                }
                float s1 = 0.f, s2 = 0.f;
#pragma unroll 1
                for (int c = 0; c < BN / 32; c++) {
                    uint32_t v[32];
                    tmem_ld32(t0 + c * 32, v);
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        const int o = c * 32 + j;
                        const float4 b = *reinterpret_cast<const float4 *>(tab + o);
                        const float4 w0 = *reinterpret_cast<const float4 *>(tab + 128 + o), w1 = *reinterpret_cast<const float4 *>(tab + 256 + o);
                        const float4 w2 = *reinterpret_cast<const float4 *>(tab + 384 + o), w3 = *reinterpret_cast<const float4 *>(tab + 512 + o);
                        const float4 a1 = *reinterpret_cast<const float4 *>(tab + 640 + o), a2 = *reinterpret_cast<const float4 *>(tab + 768 + o);
                        const float bb[4] = {b.x, b.y, b.z, b.w}, x0[4] = {w0.x, w0.y, w0.z, w0.w}, x1[4] = {w1.x, w1.y, w1.z, w1.w};
                        const float x2[4] = {w2.x, w2.y, w2.z, w2.w}, x3[4] = {w3.x, w3.y, w3.z, w3.w};
                        const float h1[4] = {a1.x, a1.y, a1.z, a1.w}, h2[4] = {a2.x, a2.y, a2.z, a2.w};
#pragma unroll
                        for (int i = 0; i < 4; i++) {
                            float y = fmaf(__uint_as_float(v[j + i]), descale, bb[i]);
                            y = fmaf(g0, x0[i], y); y = fmaf(g1, x1[i], y); y = fmaf(p0, x2[i], y); y = fmaf(p1, x3[i], y);
                            y = fmaxf(y, 0.0f);
                            s1 = fmaf(y, h1[i], s1);
                            s2 = fmaf(y, h2[i], s2);
                        }
                    }
                }
                if (row < n) {   // human_policy.py:53-55: sigmoid / tanh heads
                    mean[2 * (size_t)row] = 1.0f / (1.0f + expf(-(s1 + tab[896])));
                    mean[2 * (size_t)row + 1] = tanhf(s2 + tab[897]);
                }
            }
            tc_fence_before();
            mbar_arrive(tempty0 + 8 * buf);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        __syncwarp();
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

// ------------------------------------------------------------------ weight preparation
// One CTA, run once per set of weights: folds the first convolution's three identical input
// frames (env.py:647), lays the weights out as the kernels' operands, and chooses the
// power-of-two scales of the f16x3 scheme from bounds on the activations and the weights.
constexpr int FC2_IN = 256 + 2 + 2;   // act_fc2's inputs: act_fc1's output, goal, speed (human_policy.py:51)
struct policy_ws_t {   // device workspace layout (byte offsets from the workspace base)
    size_t fh, fl, wh, wl, w1f, b1, w2, b2, fc1_b, scales, conv1_img, conv2_img, hh, hl, w2h, w2l, fc2_tab, total;
};
static policy_ws_t policy_ws_layout(int max_n)
{
    const size_t np = ((size_t)(max_n > 0 ? max_n : 1) + 127) / 128 * 128;
    policy_ws_t L;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o += (bytes + 1023) / 1024 * 1024; return at; };
    L.fh = take(np * 4096 * 2); L.fl = take(np * 4096 * 2);
    L.wh = take((size_t)256 * 4096 * 2); L.wl = take((size_t)256 * 4096 * 2);
    L.w1f = take(160 * 4); L.b1 = take(32 * 4); L.w2 = take(3072 * 4); L.b2 = take(32 * 4);
    L.fc1_b = take(256 * 4); L.scales = take(64);
    L.conv1_img = take(6144); L.conv2_img = take(12288);
    L.hh = take(np * 256 * 2); L.hl = take(np * 256 * 2);                       // act_fc1's output as f16 pairs
    L.w2h = take(128 * 256 * 2); L.w2l = take(128 * 256 * 2); L.fc2_tab = take(898 * 4);
    L.total = o;
    return L;
}

__global__ void __launch_bounds__(1024) policy_prepare_kernel(const navgym_policy_params_t p, uint8_t *ws, const policy_ws_t L)
{
    __shared__ float red[1024];
    __shared__ float s_bound_h1, s_feat_scale, s_w_scale, s_h_scale, s_w2_scale;
    const int t = threadIdx.x;
    float *w1f = (float *)(ws + L.w1f), *b1 = (float *)(ws + L.b1), *w2 = (float *)(ws + L.w2), *b2 = (float *)(ws + L.b2);
    if (t < 160) {   // act_fea_cv1.weight [32][3][5] summed over the 3 frames
        const int c = t / 5, k = t % 5;
        w1f[t] = (p.cv1_w[(c * 3 + 0) * 5 + k] + p.cv1_w[(c * 3 + 1) * 5 + k]) + p.cv1_w[(c * 3 + 2) * 5 + k];
    }
    if (t < 32) { b1[t] = p.cv1_b[t]; b2[t] = p.cv2_b[t]; }
    for (int i = t; i < 3072; i += 1024) w2[i] = p.cv2_w[i];
    for (int i = t; i < 256; i += 1024) ((float *)(ws + L.fc1_b))[i] = p.fc1_b[i];
    __syncthreads();
    // bound on conv1 outputs (inputs lie in [-0.5, 0.5]: env.py:627-629) and on the features
    if (t == 0) {
        float m = 0.f;
        for (int c = 0; c < 32; c++) {
            float s = fabsf(b1[c]);
            for (int k = 0; k < 5; k++) s += 0.5f * fabsf(w1f[c * 5 + k]);
            m = fmaxf(m, s);
        }
        s_bound_h1 = m;
    }
    __syncthreads();
    if (t < 32) {
        float s = 0.f;
        for (int i = 0; i < 96; i++) s += fabsf(w2[t * 96 + i]);
        red[t] = fabsf(b2[t]) + s_bound_h1 * s;
    }
    __syncthreads();
    if (t == 0) {
        float m = 1e-30f;
        for (int c = 0; c < 32; c++) m = fmaxf(m, red[c]);
        int e;
        frexpf(m, &e);                          // m < 2^e
        s_feat_scale = ldexpf(1.0f, min(max(15 - e, -100), 100));   // features * scale < 2^15
        frexpf(fmaxf(s_bound_h1, 1e-30f), &e);
        s_h_scale = ldexpf(1.0f, min(max(15 - e, -100), 100));      // conv1 outputs * scale < 2^15
        float w2m = 1e-30f;
        for (int i = 0; i < 3072; i++) w2m = fmaxf(w2m, fabsf(w2[i]));
        frexpf(w2m, &e);
        s_w2_scale = ldexpf(1.0f, min(max(14 - e, -100), 100));
    }
    __syncthreads();
    float wm = 0.f;
    for (int i = t; i < 256 * 4096; i += 1024) wm = fmaxf(wm, fabsf(p.fc1_w[i]));
    red[t] = wm;
    __syncthreads();
    for (int o = 512; o > 0; o >>= 1) { if (t < o) red[t] = fmaxf(red[t], red[t + o]); __syncthreads(); }
    if (t == 0) {
        int e;
        frexpf(fmaxf(red[0], 1e-30f), &e);
        s_w_scale = ldexpf(1.0f, min(max(14 - e, -100), 100));      // |w| * scale < 2^14
        float *sc = (float *)(ws + L.scales);
        sc[0] = s_feat_scale;
        sc[1] = 1.0f / (s_feat_scale * s_w_scale);                  // powers of two: exact
        sc[2] = s_h_scale;
        sc[3] = 1.0f / (s_h_scale * s_w2_scale);
    }
    __syncthreads();
    // act_fc2 on the tensor cores: act_fc1's output h >= 0 is handed over as f16 pairs times s_h2, a power
    // of two from a bound on h (|b| + the row's L1 norm x the feature bound 2^15 / s_f: generous, which only
    // costs low-order bits of values far below the bound); fc2's first 256 weight columns are scaled and
    // split like fc1's, the four extra input columns (goal, speed), the bias and the two heads go into a
    // float32 table for the epilogue.
    {
        __shared__ float s_h2, s_w2fc;
        float l1 = 0.f;   // 4 threads per row of fc1_w
        {
            const int row = t >> 2, part = t & 3;
            for (int k = part * 1024; k < part * 1024 + 1024; k++) l1 += fabsf(p.fc1_w[row * 4096 + k]);
        }
        red[t] = l1;
        __syncthreads();
        float rowb = 0.f;
        if (t < 256) rowb = (red[4 * t] + red[4 * t + 1] + red[4 * t + 2] + red[4 * t + 3]) * (32768.0f / s_feat_scale) + fabsf(p.fc1_b[t]);
        __syncthreads();
        if (t < 256) red[t] = rowb;
        __syncthreads();
        if (t == 0) {
            float m = 1e-30f;
            for (int o = 0; o < 256; o++) m = fmaxf(m, red[o]);
            int e;
            frexpf(m, &e);
            s_h2 = ldexpf(1.0f, min(max(15 - e, -100), 100));
            float wm = 1e-30f;
            for (int i = 0; i < 128 * FC2_IN; i++) if (i % FC2_IN < 256) wm = fmaxf(wm, fabsf(p.fc2_w[i]));
            frexpf(wm, &e);
            s_w2fc = ldexpf(1.0f, min(max(14 - e, -100), 100));
            float *sc = (float *)(ws + L.scales);
            sc[6] = s_h2;
            sc[7] = 1.0f / (s_h2 * s_w2fc);
        }
        __syncthreads();
        __half *w2h = (__half *)(ws + L.w2h), *w2l = (__half *)(ws + L.w2l);
        for (int i = t; i < 128 * 256; i += 1024) {
            const int o = i >> 8, k = i & 255;
            const float x = p.fc2_w[o * FC2_IN + k] * s_w2fc;
            const __half hi = __float2half_rn(x);
            w2h[i] = hi;
            w2l[i] = __float2half_rn(x - __half2float(hi));
        }
        float *tab = (float *)(ws + L.fc2_tab);
        if (t < 128) {
            tab[t] = p.fc2_b[t];
            for (int e = 0; e < 4; e++) tab[128 * (1 + e) + t] = p.fc2_w[t * FC2_IN + 256 + e];
            tab[640 + t] = p.a1_w[t];
            tab[768 + t] = p.a2_w[t];
        }
        if (t == 0) { tab[896] = p.a1_b[0]; tab[897] = p.a2_b[0]; }
        __syncthreads();
    }
    // act_fc1's weight, columns permuted from torch's channel-major feature order (c * 128 + pos)
    // to the position-major order the front end writes (pos * 32 + c), scaled and split
    const float sw = s_w_scale;
    __half *wh = (__half *)(ws + L.wh), *wl = (__half *)(ws + L.wl);
    for (int i = t; i < 256 * 4096; i += 1024) {
        const int o = i >> 12, f = i & 4095, pos = f >> 5, c = f & 31;
        const float x = p.fc1_w[o * 4096 + c * 128 + pos] * sw;
        const __half hi = __float2half_rn(x);
        wh[i] = hi;
        wl[i] = __float2half_rn(x - __half2float(hi));
    }
    // Operand images of policy_features_umma2_kernel, byte for byte as they sit in shared memory.
    // conv1 as a GEMM per pedestrian, D1[pos][n = 3 c + tap] = conv1 output 2 pos - 1 + tap of channel c:
    // the A operand row holds the 9 inputs 4 pos - 3 .. 4 pos + 5 (times 2048) at k = 0 .. 8, the constant
    // 2048 at k = 9, and 32768 at k = 10 in row 0 / at k = 11 in row 127 only; so
    //   B1[n][k] = w1f[c][k - 2 tap] s_w1 (0 <= k - 2 tap <= 4), b1[c] s_w1 (k = 9),
    //              -32768 (k = 10 and tap 0, k = 11 and tap 2: the two conv1 outputs that are conv2's own
    //              zero padding, q = -1 and q = 255, are driven far below zero and end as relu = 0), else 0,
    // with s_w1 = s_h / 2048, i.e. the accumulator already carries the scale of conv2's A operand.
    // K-major rows of 32 bytes in 8-row groups, 32-byte swizzle (16-byte piece ^ bit 2 of the row); hi | lo.
    {
        const float s_w1 = s_h_scale * (1.0f / 2048.0f);
        __half *img1 = (__half *)(ws + L.conv1_img);
        for (int i = t; i < 96 * 16; i += 1024) {
            const int n = i >> 4, k = i & 15, c = n / 3, tap = n - 3 * c, kk = k - 2 * tap;
            float x = 0.0f;
            if (kk >= 0 && kk <= 4 && k <= 8) x = w1f[c * 5 + kk] * s_w1;
            else if (k == 9) x = b1[c] * s_w1;
            else if ((k == 10 && tap == 0) || (k == 11 && tap == 2)) x = -32768.0f;
            const __half hi = __float2half_rn(x);
            const uint32_t off = (uint32_t)n * 32u + ((((uint32_t)k >> 3) ^ (((uint32_t)n >> 2) & 1u)) << 4) + ((uint32_t)k & 7u) * 2u;
            img1[off >> 1] = hi;
            img1[(3072u + off) >> 1] = __float2half_rn(x - __half2float(hi));
        }
        // conv2's weight for the same kernel: B2[co][k = 3 ci + tap] (no padded fourth tap), three K
        // blocks of 64 rows -- [32 co][32 k] high parts, then the same rows' low parts, so that one
        // N = 64 MMA multiplies an A tile by both: K-major rows of 64 bytes, 64-byte swizzle (piece ^
        // bits 1-2 of the row)
        __half *img2 = (__half *)(ws + L.conv2_img);
        for (int i = t; i < 32 * 96; i += 1024) {
            const int co = i / 96, k = i - 96 * co, kb = k >> 5, kk = k & 31;
            const float x = w2[co * 96 + k] * s_w2_scale;
            const __half hi = __float2half_rn(x);
            const uint32_t off = (uint32_t)kb * 4096u + (uint32_t)co * 64u + ((((uint32_t)kk >> 3) ^ (((uint32_t)co >> 1) & 3u)) << 4) +
                                 ((uint32_t)kk & 7u) * 2u;
            img2[off >> 1] = hi;
            img2[(2048u + off) >> 1] = __float2half_rn(x - __half2float(hi));
        }
    }
}

struct navgym_policy {
    int max_n, device;
    uint8_t *ws;
    policy_ws_t L;
    CUtensorMap tm_fh, tm_fl, tm_wh, tm_wl;          // act_fc1: features, weight
    CUtensorMap tm_hh, tm_hl, tm_w2h, tm_w2l;        // act_fc2: act_fc1's output, weight
    int sms;
};

typedef CUresult (*navgym_encode_tiled_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                           const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                           CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// [rows][kdim] f16, row-major: boxes of BK columns (one swizzle span) x box_rows rows
static int policy_make_map(CUtensorMap *m, void *base, uint64_t rows, uint32_t box_rows, uint32_t kdim)
{
    static navgym_encode_tiled_fn encode = nullptr;
    if (!encode) {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || !fn) return -1;
        encode = (navgym_encode_tiled_fn)fn;
    }
    const cuuint64_t dims[2] = {(cuuint64_t)kdim, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)kdim * 2};
    const cuuint32_t box[2] = {(cuuint32_t)pg::BK, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : -1;
}

// ------------------------------------------------------------------ front end, both convolutions on the tensor cores
// policy_features_umma2_kernel: conv1 is a GEMM too (M 128 positions x N 96 = 32 channels x 3 taps x
// K 16: the 9 inputs a position's three conv1 outputs need, a bias column, two padding columns; see
// policy_prepare_kernel), so the CUDA cores only convert: scan -> A1 (preprocess, split), D1 -> A2
// (ReLU, split: D1's column order 3 c + tap IS conv2's K order, a thread's accumulator row goes
// straight into its A2 row), D2 -> features.  Per pedestrian 3 + 12 tcgen05.mma (f16x3) and ~1000
// instructions per position instead of ~1750 with conv1 on the CUDA cores.
// GROUPS (3) groups of GWARPS (8) worker warps + one issuing warp each take
// pedestrians round robin and run them start to end.  A warp reaches the TMEM lanes 32 (warp % 4) .. + 31
// = 32 positions; the two worker warps of a group that share a quarter split the columns.
//   P1a the scan, clipped and centred (float64, env.py:627-629), into the group's staging row
//   P1b every thread builds its piece of the A1 rows -> arrive a1full -> 3 MMAs into D1, commit d1full
//   P2  D1 from TMEM, ReLU, hi/lo split, into the A2 rows (K = 96 in three 64-byte-swizzled K blocks;
//       A1 lives in the first bytes of the same buffer: it has been consumed by then)
//       -> arrive a2full -> 12 MMAs (per K step: A hi x (B hi | B lo) as one N = 64 MMA, A lo x B hi)
//       into accumulators that overwrite D1, commit d2full
//   P3a the three accumulators summed into registers; P3b bias, ReLU, feature scale, split, store.
// Order in the steady state: P2(i) | P1a(i + 1) behind conv2's MMAs | P3a(i) | P1b(i + 1) | P3b(i)
// behind the next conv1's MMAs.  What bounds the kernel is the NUMBER of MMAs: a tcgen05.mma of this
// size (N 32 .. 96) costs the tensor pipe ~45-50 cycles whatever N and whichever accumulator it adds
// to, and one thread issues one every ~80 cycles at best (tools/umma_probe.cu) -- so every group has
// its own issuing thread (a single one for all groups kept the kernel at 15 MMAs x ~150 cycles per
// pedestrian: 0.39 ms), with the operand descriptors computed once.
namespace pf {
constexpr int GROUPS = 3, GWARPS = 8;   // 3 x 8 worker warps: 0.32 ms for 40 960 pedestrians; 4 x 4: 0.34 ms
constexpr int SUBS = GWARPS / 4, GTHREADS = 32 * GWARPS;
constexpr int WORKERS = GROUPS * GTHREADS, THREADS = WORKERS + 32 * GROUPS;   // + one issuing warp per group
static_assert(THREADS <= 1024 && GROUPS * 128 <= 512, "threads / TMEM columns");
constexpr uint32_t A2_HALF = 3 * 8192;                 // hi (or lo): 3 K blocks of [128][32] f16
constexpr uint32_t GBUF = 2 * A2_HALF;                 // 48 KB per group; A1 = its first 8 KB (hi | lo, [128][16] f16 each)
constexpr uint32_t A1_HALF = 4096;
constexpr uint32_t B2_BYTES = 3 * 4096, B1_HALF = 3072;
constexpr uint32_t XS_FLOATS = 520;
constexpr uint32_t OFF_B2 = GROUPS * GBUF, OFF_B1 = OFF_B2 + B2_BYTES, OFF_XS = OFF_B1 + 2 * B1_HALF;
constexpr uint32_t OFF_B2S = OFF_XS + GROUPS * XS_FLOATS * 4;   // conv2 bias, 32 floats
constexpr uint32_t OFF_BAR = OFF_B2S + 128;
constexpr uint32_t SMEM_BYTES = OFF_BAR + 256 + 1024;
constexpr uint32_t IDESC1 = (1u << 4) | ((uint32_t)(96 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
constexpr uint32_t IDESC2 = (1u << 4) | ((uint32_t)(32 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);    // N 32: A lo x B hi
constexpr uint32_t IDESC2W = (1u << 4) | ((uint32_t)(64 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);   // N 64: A hi x (B hi | B lo)
static_assert(SMEM_BYTES <= 227 * 1024, "shared memory");
// K-major tile of 32-byte rows, 32-byte swizzle: 8-row groups 256 B apart, layout type 6
__device__ __forceinline__ uint64_t umma_desc_sw32(uint32_t smem_addr)
{
    return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(256 >> 4) << 32) |
           ((uint64_t)1 << 46) | ((uint64_t)6 << 61);
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
}  // namespace pf

#ifdef NAVGYM_PF_PROF
// per-phase cycle sums of the groups' first threads (tools/front_prof.py builds with -DNAVGYM_PF_PROF)
__device__ unsigned long long g_pf_prof[16];
extern "C" void navgym_pf_prof_read(unsigned long long *out, int reset)
{
    cudaMemcpyFromSymbol(out, g_pf_prof, sizeof(g_pf_prof));
    if (reset) { unsigned long long z[16] = {0}; cudaMemcpyToSymbol(g_pf_prof, z, sizeof(z)); }
}
#define PF_T(i) do { if (issuer) { const long long _n = clock64(); atomicAdd(&g_pf_prof[i], (unsigned long long)(_n - _pt)); _pt = _n; } } while (0)
#else
#define PF_T(i)
#endif
__global__ void __launch_bounds__(pf::THREADS, 1)
policy_features_umma2_kernel(const float *__restrict__ scan, int n, const uint4 *__restrict__ conv1_img,
                             const uint4 *__restrict__ conv2_img, const float *__restrict__ b2,
                             const float *__restrict__ scales, __half *__restrict__ out_hi, __half *__restrict__ out_lo)
{
    using namespace pg;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *sm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const uint32_t base = smem_u32(sm);
    const uint32_t bars = base + pf::OFF_BAR;            // group g: a1full, d1full, a2full, d2full at bars + 32 g
    const uint32_t tmem_slot = bars + 32 * pf::GROUPS;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    for (int i = threadIdx.x; i < (int)(pf::B2_BYTES / 16); i += pf::THREADS) reinterpret_cast<uint4 *>(sm + pf::OFF_B2)[i] = conv2_img[i];
    for (int i = threadIdx.x; i < (int)(2 * pf::B1_HALF / 16); i += pf::THREADS) reinterpret_cast<uint4 *>(sm + pf::OFF_B1)[i] = conv1_img[i];
    for (int i = threadIdx.x; i < (int)(pf::GROUPS * pf::XS_FLOATS); i += pf::THREADS) reinterpret_cast<float *>(sm + pf::OFF_XS)[i] = 0.0f;
    if (threadIdx.x < 32) reinterpret_cast<float *>(sm + pf::OFF_B2S)[threadIdx.x] = b2[threadIdx.x];
    if (threadIdx.x == 0) {
        for (int g = 0; g < pf::GROUPS; g++) {
            mbar_init(bars + 32 * g, pf::GTHREADS); mbar_init(bars + 32 * g + 8, 1);
            mbar_init(bars + 32 * g + 16, pf::GTHREADS); mbar_init(bars + 32 * g + 24, 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // the B operands were written with ordinary stores
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");
    const int my_count = blockIdx.x < n ? (n - 1 - blockIdx.x) / gridDim.x + 1 : 0;   // pedestrians of this CTA
    if (warp < pf::GROUPS * pf::GWARPS) {
        const int g = warp / pf::GWARPS, wg = warp % pf::GWARPS, q = wg & 3, sub = wg >> 2, tg = threadIdx.x - g * pf::GTHREADS, pos = q * 32 + lane;
        constexpr int SUBS = pf::SUBS, GT = pf::GTHREADS, PER = 512 / GT, NCOL = 96 / SUBS, NCH = 32 / SUBS;
        float *xs = reinterpret_cast<float *>(sm + pf::OFF_XS) + g * pf::XS_FLOATS;   // xs[3 + i] = input i; the rest stays 0
        uint8_t *gb = sm + g * pf::GBUF;
        const uint32_t a1full = bars + 32 * g, d1full = a1full + 8, a2full = a1full + 16, d2full = a1full + 24;
        const uint32_t taddr = tmem_base + (uint32_t)g * 128u + ((uint32_t)(q * 32) << 16);
        const float descale = scales[3], fscale = scales[0];
        const float *b2s = reinterpret_cast<const float *>(sm + pf::OFF_B2S);
#ifdef NAVGYM_PF_PROF
        const bool issuer = tg == 0;
#endif
        // P1a: a scan (loaded into registers a phase earlier), clipped and centred, into the staging row
        // (barriers on both sides)
        auto load_scan = [&](int p, float (&raw)[PER]) {
#pragma unroll
            for (int i = 0; i < PER; i++) raw[i] = scan[(size_t)p * 512 + tg + GT * i];
        };
        auto stage_scan = [&](const float (&raw)[PER]) {
            asm volatile("bar.sync %0, %1;" ::"r"(1 + g), "n"(GT) : "memory");   // everyone has built its A1 piece from the previous scan
#pragma unroll
            for (int i = 0; i < PER; i++) {
                // env.py:627-629, 648: clip(scan, 0, 6) / 6 - 0.5 in float64, then float32.  One fma
                // instead of the division: within 1.2e-16 of the quotient form, which can move the
                // float32 rounding for about one input in 10^8 (by one float32 ulp)
                const double r = fmin(fmax((double)raw[i], 0.0), 6.0);
                xs[3 + tg + GT * i] = (float)fma(r, 1.0 / 6.0, -0.5);
            }
            asm volatile("bar.sync %0, %1;" ::"r"(1 + g), "n"(GT) : "memory");
        };
        // P1b: this thread's piece of A1 row `pos` (sub 0: k 0-7, sub 1: k 8, the bias and padding
        // columns) -> arrive a1full
        auto build_a1 = [&]() {
            const uint32_t sw = ((uint32_t)pos >> 2) & 1u;
            uint8_t *rowp = gb + pos * 32;
            if (sub == 0) {
                const float4 xa = *reinterpret_cast<const float4 *>(xs + 4 * pos), xb = *reinterpret_cast<const float4 *>(xs + 4 * pos + 4);
                uint32_t h[4], l[4];
                split2(xa.x * 2048.0f, xa.y * 2048.0f, h[0], l[0]);
                split2(xa.z * 2048.0f, xa.w * 2048.0f, h[1], l[1]);
                split2(xb.x * 2048.0f, xb.y * 2048.0f, h[2], l[2]);
                split2(xb.z * 2048.0f, xb.w * 2048.0f, h[3], l[3]);
                *reinterpret_cast<uint4 *>(rowp + ((0u ^ sw) << 4)) = make_uint4(h[0], h[1], h[2], h[3]);
                *reinterpret_cast<uint4 *>(rowp + pf::A1_HALF + ((0u ^ sw) << 4)) = make_uint4(l[0], l[1], l[2], l[3]);
            }
            if (sub == 1) {
                uint32_t h8, l8;
                split2(xs[4 * pos + 8] * 2048.0f, 2048.0f, h8, l8);   // k = 8, and the bias column k = 9
                const uint32_t padw = (pos == 0 ? 0x7800u : 0u) | (pos == 127 ? 0x78000000u : 0u);   // 32768 at k = 10 / k = 11
                *reinterpret_cast<uint4 *>(rowp + ((1u ^ sw) << 4)) = make_uint4(h8, padw, 0u, 0u);
                *reinterpret_cast<uint4 *>(rowp + pf::A1_HALF + ((1u ^ sw) << 4)) = make_uint4(l8, 0u, 0u, 0u);
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // visible to the tensor core's reads
            mbar_arrive(a1full);
        };
        float raw[PER];
        if (g < my_count) {
            load_scan(blockIdx.x + g * gridDim.x, raw);
            stage_scan(raw);
            build_a1();
        }
#ifdef NAVGYM_PF_PROF
        long long _pt = clock64();
#endif
        uint8_t *stg = gb + 2 * pf::A1_HALF;   // feature tile of the pedestrian just finished: hi 8 KB | lo 8 KB, behind A1
        uint32_t par = 0;
        for (int j = g; j < my_count; j += pf::GROUPS, par ^= 1) {
            const int ped = blockIdx.x + j * gridDim.x;
            const bool more = j + pf::GROUPS < my_count;
            PF_T(7);
            if (more) load_scan(blockIdx.x + (j + pf::GROUPS) * gridDim.x, raw);   // lands while P2 runs
            if (j != g) {   // the previous feature tile has left shared memory before P2 writes over it
                if (tg == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                asm volatile("bar.sync %0, %1;" ::"r"(1 + g), "n"(GT) : "memory");
            }
            // ---- P2: columns NCOL sub .. of D1 = K indices of A2
            mbar_wait(d1full, par);
            tc_fence_after();
            PF_T(0);   // wait for conv1's MMAs
            {
                const uint32_t sw = ((uint32_t)pos >> 1) & 3u;
#pragma unroll
                for (int b = 0; b < NCOL / 16; b++) {
                    const int c0 = NCOL * sub + 16 * b;            // first column; K block c0 / 32, pieces (c0 % 32) / 8 and the next
                    uint32_t v[16];
                    pf::tmem_ld16(taddr + c0, v);
                    uint8_t *rowp = gb + (c0 >> 5) * 8192 + pos * 64;
#pragma unroll
                    for (int c = 0; c < 2; c++) {
                        uint32_t h[4], l[4];
#pragma unroll
                        for (int m = 0; m < 4; m++)
                            split2(fmaxf(__uint_as_float(v[8 * c + 2 * m]), 0.0f), fmaxf(__uint_as_float(v[8 * c + 2 * m + 1]), 0.0f), h[m], l[m]);
                        const uint32_t off = ((uint32_t)(((c0 & 31) >> 3) + c) ^ sw) << 4;
                        *reinterpret_cast<uint4 *>(rowp + off) = make_uint4(h[0], h[1], h[2], h[3]);
                        *reinterpret_cast<uint4 *>(rowp + pf::A2_HALF + off) = make_uint4(l[0], l[1], l[2], l[3]);
                    }
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            tc_fence_before();
            mbar_arrive(a2full);
            PF_T(1);   // P2
            // ---- P1a of the next pedestrian, in the shadow of conv2's MMAs
            if (more) stage_scan(raw);
            PF_T(4);   // P1a
            // ---- P3a: channels NCH sub .. of the three accumulators (small products first)
            mbar_wait(d2full, par);
            tc_fence_after();
            PF_T(5);   // rest of the wait for conv2's MMAs
            float acc[NCH];
#pragma unroll
            for (int b = 0; b < NCH / 16; b++) {
                uint32_t v[16];
                pf::tmem_ld16(taddr + 32 + NCH * sub + 16 * b, v);
#pragma unroll
                for (int c = 0; c < 16; c++) acc[16 * b + c] = __uint_as_float(v[c]);
                pf::tmem_ld16(taddr + 64 + NCH * sub + 16 * b, v);
#pragma unroll
                for (int c = 0; c < 16; c++) acc[16 * b + c] += __uint_as_float(v[c]);
                pf::tmem_ld16(taddr + NCH * sub + 16 * b, v);
#pragma unroll
                for (int c = 0; c < 16; c++) acc[16 * b + c] += __uint_as_float(v[c]);
            }
            tc_fence_before();   // ordered before the a1full arrival below: the next MMAs overwrite the accumulators
            PF_T(6);   // P3a
            // ---- P1b of the next pedestrian (conv2's MMAs have read A2: its first bytes take A1)
            if (more) build_a1();
            PF_T(8);   // P1b
            // ---- P3b: bias, ReLU, feature scale, split, position-major store -- in the shadow of conv1's MMAs
            uint32_t hi[NCH / 2], lo[NCH / 2];
#pragma unroll
            for (int c = 0; c < NCH; c += 2) {
                const float a = fmaxf(fmaf(acc[c], descale, b2s[NCH * sub + c]), 0.0f) * fscale;
                const float b = fmaxf(fmaf(acc[c + 1], descale, b2s[NCH * sub + c + 1]), 0.0f) * fscale;
                split2(a, b, hi[c >> 1], lo[c >> 1]);
            }
            // the 128 x 32 tile is contiguous in global memory (position-major): staged in shared memory
            // and written by two bulk copies of 8 KB (a thread's own 64-byte rows as STG.128 reached
            // only a quarter of the store bandwidth: 16 bytes per lane at a 64-byte stride)
            uint4 *sh = reinterpret_cast<uint4 *>(stg + pos * 64 + NCH * sub * 2);
            uint4 *sl = reinterpret_cast<uint4 *>(stg + 8192 + pos * 64 + NCH * sub * 2);
#pragma unroll
            for (int i = 0; i < NCH / 8; i++) {
                sh[i] = make_uint4(hi[4 * i], hi[4 * i + 1], hi[4 * i + 2], hi[4 * i + 3]);
                sl[i] = make_uint4(lo[4 * i], lo[4 * i + 1], lo[4 * i + 2], lo[4 * i + 3]);
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("bar.sync %0, %1;" ::"r"(1 + g), "n"(GT) : "memory");
            if (tg == 0) {
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], 8192;"
                             ::"l"(out_hi + (size_t)ped * 4096), "r"(smem_u32(stg)) : "memory");
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], 8192;"
                             ::"l"(out_lo + (size_t)ped * 4096), "r"(smem_u32(stg + 8192)) : "memory");
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
        }
        if (tg == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // the last tile is on its way out
    } else if (lane == 0) {
        // ---- the group's MMA issuer; every operand descriptor is loop-invariant
        const int g = warp - pf::GROUPS * pf::GWARPS;
        const uint32_t gbuf = base + g * pf::GBUF, dcol = tmem_base + (uint32_t)g * 128u;
        const uint32_t a1full = bars + 32 * g, d1full = a1full + 8, a2full = a1full + 16, d2full = a1full + 24;
        const uint32_t b1h = base + pf::OFF_B1, b2w = base + pf::OFF_B2;
        const uint64_t a1h = pf::umma_desc_sw32(gbuf), a1l = pf::umma_desc_sw32(gbuf + pf::A1_HALF);
        const uint64_t w1h = pf::umma_desc_sw32(b1h), w1l = pf::umma_desc_sw32(b1h + pf::B1_HALF);
        uint64_t ah[6], al[6], w2[6];
#pragma unroll
        for (int ks = 0; ks < 6; ks++) {
            const uint32_t ko = (uint32_t)(ks >> 1) * 8192u + (uint32_t)(ks & 1) * 32u, kw = (uint32_t)(ks >> 1) * 4096u + (uint32_t)(ks & 1) * 32u;
            ah[ks] = umma_desc_sw64(gbuf + ko);
            al[ks] = umma_desc_sw64(gbuf + pf::A2_HALF + ko);
            w2[ks] = umma_desc_sw64(b2w + kw);   // 64 rows: high parts, then low parts
        }
        uint32_t par = 0;
        for (int j = g; j < my_count; j += pf::GROUPS, par ^= 1) {
            mbar_wait(a1full, par);
            tc_fence_after();
            umma_f16(dcol, a1l, w1h, pf::IDESC1, 0);
            umma_f16(dcol, a1h, w1l, pf::IDESC1, 1);
            umma_f16(dcol, a1h, w1h, pf::IDESC1, 1);
            umma_commit(d1full);
            mbar_wait(a2full, par);
            tc_fence_after();
#pragma unroll
            for (int ks = 0; ks < 6; ks++) {
                umma_f16(dcol, ah[ks], w2[ks], pf::IDESC2W, ks != 0);        // columns 0-31 hi x hi, 32-63 hi x lo
                umma_f16(dcol + 64, al[ks], w2[ks], pf::IDESC2, ks != 0);    // columns 64-95 lo x hi
            }
            umma_commit(d2full);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        __syncwarp();
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}
