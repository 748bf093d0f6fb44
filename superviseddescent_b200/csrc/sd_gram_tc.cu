// Tensor-core SYRK / TN-GEMM for sm_100a:  C[i,j] = beta*C[i,j] + alpha * sum_k SA[k,i]*SB[k,j]
//
// This is LinearRegressor::learn's "At * A" (reference verbose_solver.hpp:67, regressors.hpp:208) with
// A^T b folded in as extra columns (SA == SB, upper-triangle tiles only), the trailing update of the blocked
// Cholesky that replaces PartialPivLU (verbose_solver.hpp:89), and -- with two different operands -- the
// block-row solves P = U_jj^-T B of that factorisation.  S is row-major [K x NJ] -- one sample per row, exactly
// as the optimiser stacks the feature rows (superviseddescent.hpp:186-189) -- so BOTH MMA operands are
// "MN-major" (the contraction index K is the slow one).  For 32-bit operands tcgen05 accepts MN-major
// tiles only in the 128B-swizzle / 32B-atom shared-memory layout, which TMA produces directly
// (CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B): no transposition of A anywhere.
//
// Precision: kind::tf32 keeps 10 mantissa bits.  passes == 3 runs the 3xTF32 split
//     a = hi + lo,  lo = rna_tf32(a - hi);   a_i*a_j ~= hi_i*hi_j + hi_i*lo_j + lo_i*hi_j
// (relative error ~2^-21 per product, fp32 accumulation in TMEM); hi is the raw tile as the tensor core
// truncates it, or rna_tf32(a) written back in place (unbiased split).  The split happens in shared memory,
// no hi/lo copies of the operands exist in HBM.  passes == 1 is a single TF32 pass on the raw operand.
//
// Accumulation: the tensor core adds into the fp32 TMEM accumulator with truncation, so a long chain
// drifts low (measured: -1.6e-5 relative after 564 accumulating MMAs).  The chain is therefore cut every
// KC = 128 samples (48 MMAs, ~1e-6): each chunk starts a fresh TMEM accumulator and the epilogue warps
// fold the finished chunk into running sums held in REGISTERS with round-to-nearest adds, while the
// tensor core already works on the next chunk in the other TMEM buffer.
//
// Kernel shape (persistent, one CTA per SM, 512 threads): see syrk_tc2_kernel below.
#include "sd_internal.cuh"

#include <cuda.h>

#include <cstring>
#include <vector>

namespace {

constexpr int BM = 128;          // rows of C per tile   (operand "A": columns i of S)
constexpr int BN = 256;          // cols of C per tile   (operand "B": columns j of S)
constexpr int BK = 16;           // samples (rows of S) per pipeline stage
constexpr int BOX_COLS = 32;     // 32 floats = 128 B = swizzle span
constexpr int BOX_BYTES = BOX_COLS * 4 * BK;              // 2 KB
constexpr int A_BLOCKS = BM / BOX_COLS;                   // 4
constexpr int OPER_BYTES_A = A_BLOCKS * BOX_BYTES;        // 8 KB
constexpr int PIPE_BYTES = 192 * 1024;                    // shared memory of the operand pipeline
constexpr int MAX_STAGES = 8;

// The kernel is compiled for NB = 8 (tiles of 256 columns: the Gram, the trailing updates) and for narrower "B" operands
// (NB * 32 columns, a single tile column): a skinny product C[MI x <=64] = SA^T SB issues MMAs of N = 64 instead of 256 and turns
// the shared memory it does not need for operand B into a deeper pipeline (the product is then bound by the read of SA).
template <int NB>
struct TcCfg {
    static constexpr int B_BLOCKS = NB;
    static constexpr int N_MMA = NB * BOX_COLS;                                    // 64 .. 256
    static constexpr int OPER_BYTES_B = NB * BOX_BYTES;
    static constexpr int RAW_BYTES = OPER_BYTES_A + OPER_BYTES_B;
    static constexpr int STAGE_BYTES = 2 * RAW_BYTES;                              // hi + lo: 48 KB for NB = 8, 24 KB for NB = 2
    static constexpr int STAGES = PIPE_BYTES / STAGE_BYTES < MAX_STAGES ? PIPE_BYTES / STAGE_BYTES : MAX_STAGES;
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align*/ + 1024 /*barriers*/ + 8 /*EPI_WARPS*/ * 4096 /*CBOX_BYTES*/;
    // cute::UMMA::InstrDescriptor: c_format F32 [4,6)=1, a/b_format TF32 [7,10)/[10,13)=2, a/b_major MN [15],[16]=1,
    // n_dim = N>>3 at [17,23), m_dim = M>>4 at [24,29)
    static constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) |
                                      ((uint32_t)(N_MMA >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
};
constexpr int KC_STAGES = 8;      // pipeline stages per accumulation chunk: KC = 8 * BK = 128 samples
constexpr int EPI_WARPS = 8;
constexpr int TMEM_COLS = 512;

// super-tile for L2 reuse: tiles that run concurrently share (GI*128 + GJ*256) operand columns
constexpr int GI = 12, GJ = 12;

// ---- PTX wrappers ----------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// bounded wait: a protocol bug must trap (context error), never hang the GPU
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 8000000000LL) __trap();
    }
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_commit(uint64_t* bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tcgen05_mma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// One lane of a converged warp (cute::elect_one_sync).  Unlike `lane == 0`, the compiler knows the guarded region is
// executed by a single thread, so tcgen05 / TMA instructions inside it take their uniform-register operands directly
// instead of being wrapped in an ELECT / BRA.U.ANY waterfall loop each (measured: the MMA warp was issue-bound).
__device__ __forceinline__ bool elect_one_sync()
{
    uint32_t pred = 0;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// UMMA shared-memory descriptor, MN-major operand in the 128B-swizzle / 32B-atom layout
// (cute::UMMA::SmemDescriptor: start [0,14), LBO [16,30), SBO [32,46), version [46,48) = 1,
//  layout_type [61,64) = 1 = SWIZZLE_128B_BASE32B; all offsets in 16-byte units)
//   LBO = byte distance between consecutive 32-float (128 B) column blocks  = one TMA box  (2 KB)
//   SBO = byte distance between consecutive 4-row swizzle atoms along K    = 512 B
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr)
{
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)(BOX_BYTES >> 4) << 16;
    d |= (uint64_t)(512 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)1 << 61;
    return d;
}

struct TcArgs {
    int K, MI, NJ;
    float* C;
    long long ldc;
    float alpha, beta;
    int passes;          // 1 or 3
    int unbiased;        // round hi in place (slower, unbiased) instead of using the truncated raw tile
    const int2* tiles;   // (ti, tj) per tile
    int num_tiles;       // work items = tiles x ksplit
    int ksplit, kps;     // the K loop of every tile is cut into ksplit ranges of kps pipeline stages (work item t: tile t / ksplit,
                         // range t % ksplit); ksplit > 1 needs the reduce-add write-back onto a zeroed C
    int tma_c;           // 0 = register epilogue, 1 = TMA store (beta == 0), 2 = TMA reduce-add (beta == 1)
    int a_strip;         // > 0: operand A is stored strip-major, [tile row][a_strip contraction rows][128 columns] (sd_cg.cu)
};

// =====================================================================================================
// ONE raw fp32 tile per operand travels L2 -> shared memory; the tensor core truncates it to TF32 by itself
// (that is the "hi" operand), and a transform warpgroup writes lo = a - trunc_tf32(a) next to it in shared
// memory.  (A first version with operands pre-split in HBM was L2-bound at 57 % tensor-pipe activity:
// profiles/r01_summary.md.)
//   warp 0       TMA producer        (raw tiles, 24 KB per stage)
//   warp 1       MMA issuer          (lo*hi, hi*lo, hi*hi; accumulators in TMEM, one fresh accumulator per 128-sample chunk)
//   warps 4..7   transform           (raw -> lo, element-wise in the swizzled layout; fence.proxy.async)
//   warps 8..15  epilogue            (running sums in registers, write-back through the TMA)
// Register budget is rebalanced with setmaxnreg: producer/MMA/transform warpgroups give registers back,
// the two epilogue warpgroups take them (128 running sums + a 32-value TMEM fragment per thread).
// =====================================================================================================
constexpr int T2_THREADS = 512;
constexpr int CBOX_BYTES = 32 * 32 * 4;                     // one 32 x 32 fp32 box of C per epilogue warp (128B-swizzled)
static_assert(EPI_WARPS * CBOX_BYTES == 8 * 4096, "TcCfg::SMEM_BYTES");

// explicit shared-space accesses: the tile pointers come from integer arithmetic on the dynamic shared-memory base, so
// the compiler would otherwise emit generic LD/ST (ncu: 8 wavefronts per 128-bit request instead of 4)
__device__ __forceinline__ float4 lds128(uint32_t addr)
{
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, const float4& v)
{
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

__device__ __forceinline__ float trunc_tf32(float x) { return __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); }
// rna_tf32 of a finite value (what cvt.rna.tf32.f32 returns): round the magnitude to 10 mantissa bits, ties away from zero
__device__ __forceinline__ float rna_tf32_bits(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u); }
// the same value as far as the tensor core is concerned (it ignores the low 13 bits of a TF32 operand)
__device__ __forceinline__ float round_operand(float x) { return __uint_as_float(__float_as_uint(x) + 0x1000u); }

template <int NB>
__global__ void __launch_bounds__(T2_THREADS, 1)
syrk_tc2_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const __grid_constant__ CUtensorMap map_c,
                const TcArgs a)
{
    using Cfg = TcCfg<NB>;
    constexpr int STAGES = Cfg::STAGES, STAGE_BYTES = Cfg::STAGE_BYTES, RAW_BYTES = Cfg::RAW_BYTES, B_BLOCKS = Cfg::B_BLOCKS;
    constexpr uint32_t kInstrDesc = Cfg::IDESC;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
    uint64_t* raw_full = bars;                      // [STAGES] TMA bytes landed
    uint64_t* lo_ready = bars + STAGES;             // [STAGES] transform finished
    uint64_t* empty_bar = bars + 2 * STAGES;        // [STAGES] MMAs retired
    uint64_t* tmem_full = bars + 3 * STAGES;        // [2]
    uint64_t* tmem_empty = bars + 3 * STAGES + 2;   // [2]
    uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(bars + 3 * STAGES + 4);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int num_k = (a.K + BK - 1) / BK;
    const bool split = a.passes == 3;

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&raw_full[s], 1); mbar_init(&lo_ready[s], 128); mbar_init(&empty_bar[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&tmem_full[b], 1); mbar_init(&tmem_empty[b], EPI_WARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
        if (a.tma_c) asm volatile("prefetch.tensormap [%0];" ::"l"(&map_c) : "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_base_slot)), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_base_slot;

    if (warp < 4) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 56;" ::: "memory");
        if (warp == 0) {
            // ===================== TMA producer =====================
            if (elect_one_sync()) {
                uint32_t stage = 0, phase = 0;
                for (int t = blockIdx.x; t < a.num_tiles; t += gridDim.x) {
                    const int2 tile = a.tiles[t / a.ksplit];
                    const int i0 = tile.x * BM, j0 = tile.y * BN;
                    const int kb0 = (t % a.ksplit) * a.kps, kb1 = min(num_k, kb0 + a.kps);
                    for (int kb = kb0; kb < kb1; ++kb) {
                        mbar_wait(&empty_bar[stage], phase ^ 1);
                        mbar_arrive_expect_tx(&raw_full[stage], RAW_BYTES);
                        unsigned char* sa = smem + stage * STAGE_BYTES;
                        unsigned char* sb = sa + OPER_BYTES_A;
                        const int k0 = kb * BK;
#pragma unroll
                        for (int cb = 0; cb < A_BLOCKS; ++cb)
                            tma_load_2d(sa + cb * BOX_BYTES, &map_a, &raw_full[stage], (a.a_strip ? 0 : i0) + cb * BOX_COLS, (a.a_strip ? tile.x * a.a_strip : 0) + k0);
#pragma unroll
                        for (int cb = 0; cb < B_BLOCKS; ++cb) tma_load_2d(sb + cb * BOX_BYTES, &map_b, &raw_full[stage], j0 + cb * BOX_COLS, k0);
                        if (++stage == STAGES) { stage = 0; phase ^= 1; }
                    }
                }
            }
        } else if (warp == 1) {
            // ===================== MMA issuer =====================
            uint32_t stage = 0, phase = 0;
            uint32_t buf = 0, buf_phase = 0;
            for (int t = blockIdx.x; t < a.num_tiles; t += gridDim.x) {
                const int kb0 = (t % a.ksplit) * a.kps, kb1 = min(num_k, kb0 + a.kps);
                for (int kb = kb0; kb < kb1; ++kb) {
                    const bool chunk_first = ((kb - kb0) % KC_STAGES) == 0;
                    const bool chunk_last = ((kb - kb0) % KC_STAGES) == KC_STAGES - 1 || kb == kb1 - 1;
                    if (chunk_first) {
                        mbar_wait(&tmem_empty[buf], buf_phase ^ 1);
                        tcgen05_fence_after();
                    }
                    const uint32_t tmem_d = tmem_base + buf * BN;
                    mbar_wait(split ? &lo_ready[stage] : &raw_full[stage], phase);
                    tcgen05_fence_after();
                    if (elect_one_sync()) {
                        const uint32_t sa_hi = smem_u32(smem + stage * STAGE_BYTES);
                        const uint32_t sb_hi = sa_hi + OPER_BYTES_A;
                        const uint32_t sa_lo = sa_hi + RAW_BYTES;
                        const uint32_t sb_lo = sa_lo + OPER_BYTES_A;
#pragma unroll
                        for (int ks = 0; ks < BK / 8; ++ks) {
                            const uint32_t koff = ks * 8 * 128;
                            const uint32_t first = (chunk_first && ks == 0) ? 0u : 1u;
                            if (split) {
                                tcgen05_mma_tf32(tmem_d, make_desc(sa_lo + koff), make_desc(sb_hi + koff), kInstrDesc, first);
                                tcgen05_mma_tf32(tmem_d, make_desc(sa_hi + koff), make_desc(sb_lo + koff), kInstrDesc, 1u);
                                tcgen05_mma_tf32(tmem_d, make_desc(sa_hi + koff), make_desc(sb_hi + koff), kInstrDesc, 1u);
                            } else {
                                tcgen05_mma_tf32(tmem_d, make_desc(sa_hi + koff), make_desc(sb_hi + koff), kInstrDesc, first);
                            }
                        }
                        tcgen05_commit(&empty_bar[stage]);
                        if (chunk_last) tcgen05_commit(&tmem_full[buf]);
                    }
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                    if (chunk_last) { if (++buf == 2) { buf = 0; buf_phase ^= 1; } }
                }
            }
        }
    } else if (warp < 8) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 72;" ::: "memory");
        // ===================== transform: lo = a - trunc_tf32(a), element-wise on the swizzled bytes =====================
        // All four warps work on the same stage (one warp per stage, four stages in flight, was measured slower on the Gram:
        // 12.4 vs 11.0 ms -- the kernel is bound by shared-memory bandwidth, not by this chain; see DESIGN.md 4.2).
        if (split) {
            const int tt = threadIdx.x - 128;                 // 0..127
            uint32_t stage = 0, phase = 0;
            for (int t = blockIdx.x; t < a.num_tiles; t += gridDim.x) {
                const int kb0 = (t % a.ksplit) * a.kps, kb1 = min(num_k, kb0 + a.kps);
                for (int kb = kb0; kb < kb1; ++kb) {
                    mbar_wait(&raw_full[stage], phase);
                    const uint32_t raw = smem_u32(smem + stage * STAGE_BYTES) + tt * 16;
                    const uint32_t lo = raw + RAW_BYTES;
                    // Round-to-nearest to TF32 of a finite value is "add half an ulp of the 10-bit mantissa to the bit pattern and drop
                    // the low 13 bits"; the tensor core drops those bits by itself, so for an OPERAND the rounding is one integer add
                    // (cvt.rna.tf32.f32 compiles to a compare, a predicated add and a mask per value: with it ncu showed the four
                    // transform warps, not the tensor core, setting the pace).  Loads are batched four deep ahead of the stores.
                    constexpr int NIT = RAW_BYTES / 16 / 128;
                    if (a.unbiased) {
                        // hi = rna_tf32(a) written back in place (the tensor core's truncation is then a no-op and the split is
                        // unbiased), lo = rna_tf32(a - hi).  One more shared-memory write per stage than the variant below.
#pragma unroll
                        for (int i0 = 0; i0 < NIT; i0 += 4) {
                            float4 v[4];
#pragma unroll
                            for (int u = 0; u < 4; ++u) if (i0 + u < NIT) v[u] = lds128(raw + (i0 + u) * 2048);
#pragma unroll
                            for (int u = 0; u < 4; ++u) if (i0 + u < NIT) {
                                float4 h, l;
                                h.x = rna_tf32_bits(v[u].x); h.y = rna_tf32_bits(v[u].y); h.z = rna_tf32_bits(v[u].z); h.w = rna_tf32_bits(v[u].w);
                                l.x = round_operand(v[u].x - h.x); l.y = round_operand(v[u].y - h.y);
                                l.z = round_operand(v[u].z - h.z); l.w = round_operand(v[u].w - h.w);
                                sts128(raw + (i0 + u) * 2048, h);
                                sts128(lo + (i0 + u) * 2048, l);
                            }
                        }
                    } else {
                        // hi is the raw tile as the tensor core sees it (low 13 mantissa bits ignored); the residual is
                        // rounded to TF32 so that the hardware's truncation of the lo operand does not bias it
#pragma unroll
                        for (int i0 = 0; i0 < NIT; i0 += 4) {
                            float4 v[4];
#pragma unroll
                            for (int u = 0; u < 4; ++u) if (i0 + u < NIT) v[u] = lds128(raw + (i0 + u) * 2048);
#pragma unroll
                            for (int u = 0; u < 4; ++u) if (i0 + u < NIT) {
                                float4 l;
                                l.x = round_operand(v[u].x - trunc_tf32(v[u].x)); l.y = round_operand(v[u].y - trunc_tf32(v[u].y));
                                l.z = round_operand(v[u].z - trunc_tf32(v[u].z)); l.w = round_operand(v[u].w - trunc_tf32(v[u].w));
                                sts128(lo + (i0 + u) * 2048, l);
                            }
                        }
                    }
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the tensor core
                    mbar_arrive(&lo_ready[stage]);
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 176;" ::: "memory");
        // ===================== epilogue (warps 8..15) =====================
        const int q = warp & 3;
        const int half = (warp - 8) >> 2;
        uint32_t buf = 0, buf_phase = 0;
        const bool vec_ok = (a.ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(a.C) & 15) == 0);
        for (int t = blockIdx.x; t < a.num_tiles; t += gridDim.x) {
            const int2 tile = a.tiles[t / a.ksplit];
            const int kb0 = (t % a.ksplit) * a.kps, kb1 = min(num_k, kb0 + a.kps);
            const int num_chunks = (kb1 - kb0 + KC_STAGES - 1) / KC_STAGES;
            const int i = tile.x * BM + q * 32 + lane;
            const int j0 = tile.y * BN + half * 128;
            float acc[128];
#pragma unroll
            for (int v = 0; v < 128; ++v) acc[v] = 0.f;
            for (int c = 0; c < num_chunks; ++c) {
                mbar_wait(&tmem_full[buf], buf_phase);
                tcgen05_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + buf * BN + half * 128;
#pragma unroll
                for (int c0 = 0; c0 < 128; c0 += 32) {
                    if (NB < 8 && half * 128 + c0 >= Cfg::N_MMA) continue;     // columns the narrow MMA never writes
                    uint32_t r[32];
                    tmem_ld_32x32b_x32(taddr + c0, r);
                    tmem_ld_wait();
#pragma unroll
                    for (int v = 0; v < 32; ++v) acc[c0 + v] = __fadd_rn(acc[c0 + v], __uint_as_float(r[v]));
                }
                tcgen05_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tmem_empty[buf]);
                if (++buf == 2) { buf = 0; buf_phase ^= 1; }
            }
            if (a.tma_c) {
                // Coalesced write-back through the TMA: the thread-per-row TMEM fragment would touch 32 different
                // lines per store instruction (measured: the epilogue, not the MMAs, set the pace of K = 256 updates).
                // Each warp stages 32 x 32 boxes in 128B-swizzled shared memory and one lane issues a bulk tensor
                // store (beta == 0) or reduce-add (beta == 1, done in L2: C is never read by the SM).  Every element
                // is touched once per launch, so the result is the single rounding of old + alpha * sum; rows and
                // columns outside C are clipped by the tensor map.
                unsigned char* box = smem + STAGES * STAGE_BYTES + 1024 + (warp - 8) * CBOX_BYTES;
                const uint32_t box_u32 = smem_u32(box);
#pragma unroll
                for (int c0 = 0; c0 < 128; c0 += 32) {
                    if (NB < 8 && half * 128 + c0 >= Cfg::N_MMA) continue;
                    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // box buffer free again
                    __syncwarp();
#pragma unroll
                    for (int v = 0; v < 8; ++v) {
                        const float4 o = make_float4(a.alpha * acc[c0 + 4 * v + 0], a.alpha * acc[c0 + 4 * v + 1],
                                                     a.alpha * acc[c0 + 4 * v + 2], a.alpha * acc[c0 + 4 * v + 3]);
                        sts128(box_u32 + lane * 128 + ((v ^ (lane & 7)) << 4), o);
                    }
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) {
                        const int cx = j0 + c0, cy = tile.x * BM + q * 32;
                        if (a.tma_c == 2)
                            asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%1, %2}], [%3];"
                                         ::"l"(&map_c), "r"(cx), "r"(cy), "r"(box_u32) : "memory");
                        else
                            asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%1, %2}], [%3];"
                                         ::"l"(&map_c), "r"(cx), "r"(cy), "r"(box_u32) : "memory");
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    }
                }
            } else if (i < a.MI) {
                float* crow = a.C + (long long)i * a.ldc;
                if (vec_ok && j0 + 128 <= a.NJ && a.beta == 1.f) {
                    // C += alpha * sum as fire-and-forget vector reductions: no load of C, no round trip on the
                    // epilogue's critical path.  Each element is touched once per launch, so the result is the
                    // same single rounding as fmaf(1, old, alpha * sum) and is reproducible.
#pragma unroll
                    for (int v = 0; v < 32; ++v)
                        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(crow + j0 + 4 * v),
                                     "f"(a.alpha * acc[4 * v + 0]), "f"(a.alpha * acc[4 * v + 1]),
                                     "f"(a.alpha * acc[4 * v + 2]), "f"(a.alpha * acc[4 * v + 3]) : "memory");
                } else if (vec_ok && j0 + 128 <= a.NJ) {
#pragma unroll
                    for (int v = 0; v < 32; ++v) {
                        float4 o;
                        o.x = a.alpha * acc[4 * v + 0]; o.y = a.alpha * acc[4 * v + 1];
                        o.z = a.alpha * acc[4 * v + 2]; o.w = a.alpha * acc[4 * v + 3];
                        float4* p = reinterpret_cast<float4*>(crow + j0 + 4 * v);
                        if (a.beta != 0.f) {
                            const float4 old = *p;
                            o.x = fmaf(a.beta, old.x, o.x); o.y = fmaf(a.beta, old.y, o.y);
                            o.z = fmaf(a.beta, old.z, o.z); o.w = fmaf(a.beta, old.w, o.w);
                        }
                        *p = o;
                    }
                } else {
#pragma unroll
                    for (int v = 0; v < 128; ++v) {
                        if (j0 + v < a.NJ) {
                            float o = a.alpha * acc[v];
                            if (a.beta != 0.f) o = fmaf(a.beta, crow[j0 + v], o);
                            crow[j0 + v] = o;
                        }
                    }
                }
            }
        }
    }

    if (warp >= 8 && lane == 0 && a.tma_c) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // writes complete
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 1) {
        tcgen05_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_encodeTiled get_encode_fn()
{
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_encodeTiled>(p);
    }
    return fn;
}

int make_map(sd_ctx* ctx, CUtensorMap* map, const float* base, int64_t ld, int rows, int cols)
{
    PFN_encodeTiled enc = get_encode_fn();
    if (!enc) return sd_fail(ctx, SD_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t gstride[1] = {(cuuint64_t)ld * sizeof(float)};
    cuuint32_t box[2] = {(cuuint32_t)BOX_COLS, (cuuint32_t)BK};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim, gstride, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return sd_fail(ctx, SD_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
    return SD_OK;
}

// C (rows x cols, pitch ld) as 32 x 32 boxes, 128B-swizzled in shared memory
int make_map_c(sd_ctx* ctx, CUtensorMap* map, float* base, int64_t ld, int rows, int cols)
{
    PFN_encodeTiled enc = get_encode_fn();
    if (!enc) return sd_fail(ctx, SD_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t gstride[1] = {(cuuint64_t)ld * sizeof(float)};
    cuuint32_t box[2] = {32, 32};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return sd_fail(ctx, SD_ERR_CUDA, "cuTensorMapEncodeTiled (C) failed (%d)", (int)r);
    return SD_OK;
}

}  // namespace

bool sd_syrk_tc_supported(const float* d_S, int64_t lds, int K, int MI, int NJ, const float* d_C, int64_t ldc)
{
    (void)MI; (void)NJ; (void)d_C; (void)ldc;
    // TMA needs a 16-byte aligned base and row pitch
    return K >= 1 && (reinterpret_cast<uintptr_t>(d_S) & 15) == 0 && (lds % 4) == 0;
}

// A prepared launch of the kernel: tensor maps, tile list (already on the device) and arguments.  Preparing costs three
// cuTensorMapEncodeTiled calls, the tile enumeration and a small host->device copy; iterative callers (sd_cg.cu) prepare once.
struct sd_tc_plan {
    CUtensorMap map_a, map_b, map_c;
    TcArgs args;
    int grid;
    int nb;              // kernel variant: 32-column boxes of operand B per stage (8 = full tiles)
};
static_assert(sizeof(sd_tc_plan) <= SD_TC_PLAN_BYTES, "sd_tc_plan storage");

// C[i,j] = beta*C[i,j] + alpha * sum_{k<K} SA[k,i] * SB[k,j],  i < MI, j < NJ.   SA: K x MI (lda), SB: K x NJ (ldb), both row-major,
// i.e. both operands MN-major.  upper_only keeps the tiles that intersect j >= i (SYRK: SA == SB).  `rows` (optional) keeps the
// tiles whose C rows belong to this rank's block rows (distributed trailing update).  C may alias SB when every CTA's column
// range of SB is read completely before its tile is written: true for MI <= 128 (one tile row; each tile's operand columns are
// its own output columns).  d_tiles: device buffer for the tile list (at least sd_tc_max_tiles(MI, NJ) int2), or NULL to use the
// context's workspace.  *empty is set when no tile survives the filters (nothing to launch).
int sd_gemm_tn_tc_prepare(sd_ctx* ctx, const float* d_SA, int64_t lda, const float* d_SB, int64_t ldb, int K, int MI, int NJ,
                          float* d_C, int64_t ldc, float alpha, float beta, int passes, bool unbiased_split, bool upper_only,
                          const sd_row_filter* rows, int ksplit, void* d_tiles_buf, void* plan_storage, bool* empty, bool narrow, int a_strip_rows)
{
    sd_tc_plan* plan = reinterpret_cast<sd_tc_plan*>(plan_storage);
    *empty = true;
    if (MI <= 0 || NJ <= 0 || K <= 0) return SD_OK;
    SD_REQUIRE(ctx, passes == 1 || passes == 3, "passes must be 1 or 3");
    // operand A either as the row-major K x MI matrix, or strip-major: sd_div_up(MI, 128) strips of a_strip_rows x 128 floats each
    // (rows K .. a_strip_rows - 1 and the columns beyond MI hold zeros): a CTA then streams one contiguous strip
    SD_REQUIRE(ctx, a_strip_rows == 0 || (a_strip_rows % BK == 0 && a_strip_rows >= K), "strip-major operand: rows padded to the pipeline stage");
    int rc = a_strip_rows ? make_map(ctx, &plan->map_a, d_SA, BM, sd_div_up(MI, BM) * a_strip_rows, BM) : make_map(ctx, &plan->map_a, d_SA, lda, K, MI);
    if (rc) return rc;
    rc = make_map(ctx, &plan->map_b, d_SB, ldb, K, NJ);
    if (rc) return rc;

    // tile list, ordered by super-tiles so that concurrently running tiles share operand columns in L2
    const int TI = sd_div_up(MI, BM), TJ = sd_div_up(NJ, BN);
    std::vector<int2>& tiles = ctx->tile_scratch;
    tiles.clear();
    for (int si = 0; si < TI; si += GI)
        for (int sj = 0; sj < TJ; sj += GJ)
            for (int ti = si; ti < si + GI && ti < TI; ++ti) {
                if (rows && rows->nranks > 1 && ((rows->first_row + (int64_t)ti * BM) / rows->block) % rows->nranks != rows->rank) continue;
                for (int tj = sj; tj < sj + GJ && tj < TJ; ++tj)
                    if (!upper_only || tj * BN + BN - 1 >= ti * BM) tiles.push_back(make_int2(ti, tj));
            }
    if (tiles.empty()) return SD_OK;
    int2* d_tiles = (int2*)d_tiles_buf;
    if (!d_tiles) d_tiles = (int2*)sd_workspace(ctx, SD_WS_DIAGINV, tiles.size() * sizeof(int2));
    if (!d_tiles) return SD_ERR_CUDA;
    SD_CUDA(ctx, cudaMemcpyAsync(d_tiles, tiles.data(), tiles.size() * sizeof(int2), cudaMemcpyHostToDevice, ctx->stream));

    TcArgs& a = plan->args;
    a.K = K; a.MI = MI; a.NJ = NJ; a.C = d_C; a.ldc = ldc; a.alpha = alpha; a.beta = beta; a.passes = passes;
    a.unbiased = (ctx->gram_mode == 3 || unbiased_split) ? 1 : 0;
    a.a_strip = a_strip_rows;
    const int num_k = sd_div_up(K, BK);
    if (ksplit < 1) ksplit = 1;
    if (ksplit > num_k) ksplit = num_k;
    a.kps = sd_div_up(num_k, ksplit);
    a.ksplit = sd_div_up(num_k, a.kps);                   // every range non-empty
    a.tiles = d_tiles; a.num_tiles = (int)tiles.size() * a.ksplit;
    const int sms = ctx->sm_count - ctx->syrk_sm_reserve > 0 ? ctx->sm_count - ctx->syrk_sm_reserve : 1;
    plan->grid = a.num_tiles < sms ? a.num_tiles : sms;
    // C goes back through the TMA when it can be described by a tensor map (16-byte aligned base and pitch)
    plan->map_c = plan->map_b;
    a.tma_c = 0;
    if ((beta == 0.f || beta == 1.f) && (ldc % 4) == 0 && (reinterpret_cast<uintptr_t>(d_C) & 15) == 0) {
        rc = make_map_c(ctx, &plan->map_c, d_C, ldc, MI, NJ);
        if (rc) return rc;
        a.tma_c = beta == 1.f ? 2 : 1;
    }
    // split K: the ranges of one tile add into C in any order, which is only reproducible for two of them (a + b == b + a)
    SD_REQUIRE(ctx, a.ksplit == 1 || (a.tma_c == 2 && a.ksplit == 2), "split-K needs beta == 1, the TMA reduce-add write-back and two ranges");
    // a single tile column of at most 192 columns can run the narrow variants
    plan->nb = 8;
    if (narrow && TJ == 1) plan->nb = NJ <= 64 ? 2 : NJ <= 128 ? 4 : NJ <= 192 ? 6 : 8;
    switch (plan->nb) {
    case 2: SD_CUDA(ctx, cudaFuncSetAttribute(syrk_tc2_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<2>::SMEM_BYTES)); break;
    case 4: SD_CUDA(ctx, cudaFuncSetAttribute(syrk_tc2_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<4>::SMEM_BYTES)); break;
    case 6: SD_CUDA(ctx, cudaFuncSetAttribute(syrk_tc2_kernel<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<6>::SMEM_BYTES)); break;
    default: SD_CUDA(ctx, cudaFuncSetAttribute(syrk_tc2_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<8>::SMEM_BYTES)); break;
    }
    *empty = false;
    return SD_OK;
}

int sd_gemm_tn_tc_launch(sd_ctx* ctx, const void* plan_storage)
{
    const sd_tc_plan* plan = reinterpret_cast<const sd_tc_plan*>(plan_storage);
    switch (plan->nb) {
    case 2: syrk_tc2_kernel<2><<<plan->grid, T2_THREADS, TcCfg<2>::SMEM_BYTES, ctx->stream>>>(plan->map_a, plan->map_b, plan->map_c, plan->args); break;
    case 4: syrk_tc2_kernel<4><<<plan->grid, T2_THREADS, TcCfg<4>::SMEM_BYTES, ctx->stream>>>(plan->map_a, plan->map_b, plan->map_c, plan->args); break;
    case 6: syrk_tc2_kernel<6><<<plan->grid, T2_THREADS, TcCfg<6>::SMEM_BYTES, ctx->stream>>>(plan->map_a, plan->map_b, plan->map_c, plan->args); break;
    default: syrk_tc2_kernel<8><<<plan->grid, T2_THREADS, TcCfg<8>::SMEM_BYTES, ctx->stream>>>(plan->map_a, plan->map_b, plan->map_c, plan->args); break;
    }
    SD_LAUNCH_CHECK(ctx, "syrk_tc2_kernel");
    return SD_OK;
}

int sd_gemm_tn_tc(sd_ctx* ctx, const float* d_SA, int64_t lda, const float* d_SB, int64_t ldb, int K, int MI, int NJ,
                  float* d_C, int64_t ldc, float alpha, float beta, int passes, bool unbiased_split, bool upper_only,
                  const sd_row_filter* rows, int ksplit)
{
    alignas(64) unsigned char storage[SD_TC_PLAN_BYTES];
    bool empty = true;
    int rc = sd_gemm_tn_tc_prepare(ctx, d_SA, lda, d_SB, ldb, K, MI, NJ, d_C, ldc, alpha, beta, passes, unbiased_split, upper_only, rows, ksplit,
                                   nullptr, storage, &empty, false, 0);
    if (rc || empty) return rc;
    return sd_gemm_tn_tc_launch(ctx, storage);
}

int sd_syrk_tc(sd_ctx* ctx, const float* d_S, int64_t lds, int K, int MI, int NJ, float* d_C, int64_t ldc,
               float alpha, float beta, int passes, bool unbiased_split, const sd_row_filter* rows)
{
    return sd_gemm_tn_tc(ctx, d_S, lds, d_S, lds, K, MI, NJ, d_C, ldc, alpha, beta, passes, unbiased_split, true, rows);
}
