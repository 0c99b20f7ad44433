// q4_gemv.cu -- decode hot path: fused 4-bit unpack + scale/zero + skinny GEMM (M <= 8) for sm_100a.
//
// Replaces the reference's q4_matmul_kernel + dot_product_8* (exllama_ext/cuda_func/q4_matmul.cu:34-212,
// exllama_ext/matrix.cuh:87-286) and, through the fused prologue/epilogues, rms_norm (rms_norm.cu),
// rope (rope.cu), update_cache_kernel (q4_attn.cu:19-72) and silu_mul (q4_mlp.cu:46-88) on the decode path.
//
// Design (HBM-bound; see DESIGN.md "decode kernel"):
//  * packed qweight [K/8, N] is streamed exactly once: a producer warp moves 16-row x 128-column stages
//    (8 KB = four 2-D TMA boxes of 16 rows x 32 columns, cp.async.bulk.tensor, SWIZZLE_128B) into a GV_NST-deep
//    shared-memory ring guarded by mbarrier full/empty pairs, so ~50 KB per CTA are in flight without holding
//    registers.  Consumer lane (g = lane/4, t = lane%4) reads 4 adjacent columns of k8-row t with one LDS.128;
//    the column chunk a lane owns is pi(g) = (g >> 1) | ((g & 1) << 2), which makes the swizzled pattern
//    bank-conflict free.
//  * group scales / zeros of the CTA's k-range are staged into shared memory with 1-D TMA bulk copies
//    (cp.async.bulk + mbarrier); x is staged by the threads because it is permuted (and gathered through the
//    act-order x_map, and RMS-normalised for the fused decoder ops) on the way in.
//  * the contraction runs on the integer tensor cores (mma.sync m16n8k32 u8 x s8/u8 -> s32, SASS IMMA.16832) with
//    the *nibbles as the A operand straight from registers* (two ops per 8 weights: w & 0x0f0f0f0f, (w >> 4) & ...)
//    and the <= 8 activation rows as the n = 8 operand, so the unpack costs 3/8 instruction per weight and the cost
//    is independent of M for M <= 8.  x is carried per quantisation group as a 16-bit integer with its own scale
//    (two byte planes), the zero point becomes one multiply per group (zp * sum x_q), and everything inside a
//    group is exact integer arithmetic; groups are combined in fp32 with the fp16 group scales.
//    Quantising x to 16 bits per group costs < 1e-4 of the output rms -- below the fp16 rounding of the result
//    (the reference accumulates in fp16, matrix.cuh:87-133).
//  * split-K without global memory: one thread-block CLUSTER owns one 128-column tile; its CS CTAs take contiguous
//    K slices and the leader sums the CS partials out of its own shared memory, where the peers deposited them
//    through DSMEM with st.async (the stores complete transaction bytes on an mbarrier of the leader, so no
//    cluster-scope fence is needed and the peers exit right away).  Fixed summation order => deterministic; no fp16
//    atomics (the reference: q4_matmul.cu:203-211) and no L2 round trips on the critical path.
//  * programmatic dependent launch: weights do not depend on the previous kernel, so the producer warp fills the
//    whole TMA ring BEFORE the consumers' griddepcontrol.wait, and launch_dependents is signalled as soon as the
//    last weight stage has been issued -- back-to-back GEMVs keep HBM busy across the launch boundary.
#include "exl_common.cuh"
#include <cstdlib>
#include <cstring>

#ifndef GV_MINB
#define GV_MINB 2                    // resident CTAs per SM the register allocation is tuned for
#endif
#ifndef GV_GMAXC
#define GV_GMAXC 32
#endif
#ifndef GV_NST
#define GV_NST 6                    // TMA ring depth (stages of 16 k8-rows x 128 columns)
#endif

namespace {

constexpr int CONSUMERS = 256;             // 8 consumer warps: 4 across columns x 2 across k
constexpr int THREADS = CONSUMERS + 32;    // + 1 producer warp
constexpr int WN = 4, WK = 2;
constexpr int STAGE_ROWS = 16;             // k8-rows per ring stage (= 128 k)
constexpr int STAGE_K = STAGE_ROWS * 8;
constexpr int BOX_COLS = 32;                 // TMA box: 32 columns (128 B, SWIZZLE_128B) x 16 k8-rows = 2 KB, one per column-warp
constexpr int BOX_BYTES = STAGE_ROWS * BOX_COLS * 4;
constexpr int STAGE_BYTES = WN * BOX_BYTES;  // 8 KB
constexpr int NST = GV_NST;
static_assert(NST % 2 == 0, "the two k-warp groups alternate ring stages");
constexpr int RED_LD = GV_TILE_N + 4;
constexpr int GMAXC = GV_GMAXC;                  // max quantisation groups staged per chunk
constexpr int SC_ROW = GV_TILE_N * 2;      // bytes of scales per group row in smem
constexpr int ZQ_ROW = GV_TILE_N / 2;      // bytes of packed zeros per group row in smem (raw, as TMA delivers them)
constexpr int SEG_BYTES = GMAXC * GV_MAXM * 16;  // per (segment, token): {sum of x_q over even ring stages, over odd ring stages, x scale, -}
constexpr int XS_BUDGET = 16 * 1024;       // bytes of staged x per chunk
constexpr int SLOT_BUDGET = 16 * 1024;     // bytes of cluster-reduction slots (2 x CS x M x 512 B)
constexpr int MAX_CS = 8;

struct GemvMatDev
{
    const uint32_t* qw; const uint32_t* qz; const half* sc; half* out;
    int N; int tile0;
};

struct alignas(64) GemvArgs
{
    CUtensorMap tmaps[3];              // qweight of each fused matrix ([K/8, N] uint32, box 16 x 32, 128B swizzle)
    const half* x; const uint32_t* x_map;
    int M, K, groups, gs_shift32;      // gs_shift32: log2(groupsize / 32) (30 when there is a single group)
    int spt;                           // ring stages per tile = ceil(K / 128)
    int cs;                            // cluster size == K split factor
    int num_mats;
    GemvMatDev mats[3];
    int no_zero;
    int chunk_stages;                  // staging chunk (ring stages)
    int xs_stride;                     // bytes, == 64 (mod 128)
    // fused prologue / epilogue
    const half* norm_w; float eps; float r_dim;
    const half* sin; const half* cos;
    int head_dim, num_heads, num_kv_heads, past_len, max_seq_len;
    half* key_cache; half* value_cache;
    int debug;                         // EXL_GV_DEBUG bitmask (profiling experiments only)
    // GV_EPI_ALLREDUCE: one-shot all-reduce of the tile over NVLink peer memory
    int tp_rank, tp_world;
    unsigned char* tp_peers[8];
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(void* bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(void* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(void* bar, uint32_t parity)
{
    asm volatile("{\n\t.reg .pred p;\n\tWAIT_LOOP:\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
                 "@p bra DONE;\n\tbra WAIT_LOOP;\n\tDONE:\n\t}" :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
// 1-D TMA bulk copy global -> shared, completion counted on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, void* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// 2-D TMA tile load global -> shared (SASS: UTMALDG); c0 = column (uint32 elements), c1 = k8-row
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* tmap, int c0, int c1, void* bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 :: "r"(smem_u32(dst)), "l"(tmap), "r"(c0), "r"(c1), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

__device__ __forceinline__ void imma_u8s8(int (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1)
{
    asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.u8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void imma_u8u8(int (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1)
{
    asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// first MMA of a segment: C = 0 (no separate clearing of the 16 integer accumulators)
__device__ __forceinline__ void imma_u8s8_z(int (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1)
{
    asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.u8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%10,%10,%10};"
                 : "=r"(c[0]), "=r"(c[1]), "=r"(c[2]), "=r"(c[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1), "r"(0));
}
__device__ __forceinline__ void imma_u8u8_z(int (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1)
{
    asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%10,%10,%10};"
                 : "=r"(c[0]), "=r"(c[1]), "=r"(c[2]), "=r"(c[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1), "r"(0));
}

__device__ __forceinline__ half silu_h(half x)
{
    // same fp16 sequence as the reference (q4_mlp.cu:27-36)
    half one = __float2half(1.0f);
    half e = hexp(__hneg(x));
    half r = hrcp(__hadd(one, e));
    return __hmul(x, r);
}

// Per-thread state of the inner product loop for one tile segment.
// The contraction runs on the integer tensor cores: the 4-bit weights are used as they are (u8 0..15) and each
// x segment (one quantisation group, or its intersection with the staging chunk) is carried as a 16-bit integer
// x_q = 256 * a + b with its own scale sx (a: signed high byte, b: unsigned low byte).  Per segment
//     sum_k x_k (q_k - zp) = sx * ( 256 * sum a_k q_k + sum b_k q_k - zp * sum x_q,k )        (exact in int32)
// and the result is folded into fp32 totals with the group's weight scale.
struct Accum
{
    float acc[8];        // fp32 totals: [col j >> 1][token 2t + (j & 1)]
    int ia[8], ib[8];    // current segment: plane a / plane b integer dot products
    float cs[4];         // segment's weight scales (4 columns)
    uint32_t zp4;        // segment's zero points + 1, one byte per column
    int sxq[2];          // per token (2t, 2t+1): sum of x_q over the part of the segment this k-warp accumulates
    float sxs[2];        // per token: x scale of the segment
    int cur_grp;
    bool fresh;          // integer accumulators are logically zero: the next MMA starts from C = 0
};

__device__ __forceinline__ void seg_flush(Accum& A)
{
    #pragma unroll
    for (int j = 0; j < 8; j++) {
        const int col = j >> 1, tok = j & 1;
        const int zp = (int)((A.zp4 >> (8 * col)) & 0xffu);
        const int val = A.ia[j] * 256 + A.ib[j] - zp * A.sxq[tok];
        A.acc[j] = fmaf(A.cs[col] * A.sxs[tok], (float)val, A.acc[j]);
    }
    A.fresh = true;
}

__device__ __forceinline__ void group_switch(Accum& A, int grp, int g_lo, uint32_t sc_addr, uint32_t zq_addr, uint32_t seg_addr,
                                             int lane_col, int t, int par)
{
    if (A.cur_grp >= 0) seg_flush(A);
    const int gl = grp - g_lo;
    uint2 sc; uint32_t zw; uint4 s0, s1;
    asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(sc.x), "=r"(sc.y) : "r"(sc_addr + gl * SC_ROW + lane_col * 2));
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(zw) : "r"(zq_addr + gl * ZQ_ROW + (lane_col >> 3) * 4));
    const uint32_t ea = seg_addr + (gl * GV_MAXM + 2 * t) * 16;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(s0.x), "=r"(s0.y), "=r"(s0.z), "=r"(s0.w) : "r"(ea));
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(s1.x), "=r"(s1.y), "=r"(s1.z), "=r"(s1.w) : "r"(ea + 16));
    const half2 s01 = *reinterpret_cast<const half2*>(&sc.x);
    const half2 s23 = *reinterpret_cast<const half2*>(&sc.y);
    A.cs[0] = __low2float(s01); A.cs[1] = __high2float(s01);
    A.cs[2] = __low2float(s23); A.cs[3] = __high2float(s23);
    const uint32_t z4 = zw >> ((lane_col & 4) * 4);          // this lane's 4 zero nibbles
    A.zp4 = ((z4 & 0xfu) | ((z4 & 0xf0u) << 4) | ((z4 & 0xf00u) << 8) | ((z4 & 0xf000u) << 12)) + 0x01010101u;
    A.sxq[0] = (int)(par ? s0.y : s0.x); A.sxs[0] = __uint_as_float(s0.z);
    A.sxq[1] = (int)(par ? s1.y : s1.x); A.sxs[1] = __uint_as_float(s1.z);
    A.cur_grp = grp;
}

// Quantise one staged k8-row (8 halves, natural order) with scale 1/inv: returns sum of x_q and the packed byte planes
// {a(0,2,4,6), a(1,3,5,7), b(0,2,4,6), b(1,3,5,7)},  x_q = 256 a + b.
__device__ __forceinline__ int quantise_row(const uint4& hv, float inv, uint4& o)
{
    const half2* h = reinterpret_cast<const half2*>(&hv);
    int sum = 0;
    o = make_uint4(0, 0, 0, 0);
    #pragma unroll
    for (int i = 0; i < 4; i++) {
        const float2 f = __half22float2(h[i]);
        const int q0 = __float2int_rn(f.x * inv), q1 = __float2int_rn(f.y * inv);
        sum += q0 + q1;
        o.x |= (uint32_t)((q0 >> 8) & 0xff) << (8 * i);
        o.y |= (uint32_t)((q1 >> 8) & 0xff) << (8 * i);
        o.z |= (uint32_t)(q0 & 0xff) << (8 * i);
        o.w |= (uint32_t)(q1 & 0xff) << (8 * i);
    }
    return sum;
}
__device__ __forceinline__ float row_absmax(const uint4& hv)
{
    const half2* h = reinterpret_cast<const half2*>(&hv);
    float mx = 0.f;
    #pragma unroll
    for (int i = 0; i < 4; i++) { const float2 f = __half22float2(__habs2(h[i])); mx = fmaxf(mx, fmaxf(f.x, f.y)); }
    return mx;
}

// one unit = this lane's uint4 of weights (4 columns x 8 k) against the two byte planes of x (xb = {a_even, a_odd, b_even, b_odd})
__device__ __forceinline__ void unit_mma(Accum& A, const uint4& w, const uint4& xb)
{
    const uint32_t M4 = 0x0f0f0f0fu;
    const uint32_t lo0 = w.x & M4, hi0 = (w.x >> 4) & M4;      // bytes = nibbles (0,2,4,6) / (1,3,5,7) of column c0
    const uint32_t lo1 = w.y & M4, hi1 = (w.y >> 4) & M4;
    const uint32_t lo2 = w.z & M4, hi2 = (w.z >> 4) & M4;
    const uint32_t lo3 = w.w & M4, hi3 = (w.w >> 4) & M4;
    int (&aA)[4] = *reinterpret_cast<int (*)[4]>(&A.ia[0]);
    int (&aB)[4] = *reinterpret_cast<int (*)[4]>(&A.ia[4]);
    int (&bA)[4] = *reinterpret_cast<int (*)[4]>(&A.ib[0]);
    int (&bB)[4] = *reinterpret_cast<int (*)[4]>(&A.ib[4]);
    // A rows g / g+8 = columns (c0, c1) resp. (c2, c3); logical k 4t+i <-> nibble 2i, 16+4t+i <-> nibble 2i+1 of k8-row t
    if (A.fresh) {                 // warp-uniform
        imma_u8s8_z(aA, lo0, lo1, hi0, hi1, xb.x, xb.y);
        imma_u8u8_z(bA, lo0, lo1, hi0, hi1, xb.z, xb.w);
        imma_u8s8_z(aB, lo2, lo3, hi2, hi3, xb.x, xb.y);
        imma_u8u8_z(bB, lo2, lo3, hi2, hi3, xb.z, xb.w);
        A.fresh = false;
    } else {
        imma_u8s8(aA, lo0, lo1, hi0, hi1, xb.x, xb.y);
        imma_u8u8(bA, lo0, lo1, hi0, hi1, xb.z, xb.w);
        imma_u8s8(aB, lo2, lo3, hi2, hi3, xb.x, xb.y);
        imma_u8u8(bB, lo2, lo3, hi2, hi3, xb.z, xb.w);
    }
}

__device__ __forceinline__ void cluster_arrive_relaxed() { asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank)
{
    uint32_t r; asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank)); return r;
}
// st.async: a DSMEM store that completes tx bytes on an mbarrier of the destination CTA -- the data is visible to whoever
// observes that barrier's phase flip, so no cluster-scope release fence (MEMBAR.GPU) is needed on the sending side
__device__ __forceinline__ void st_async_f32(uint32_t addr, float v, uint32_t mbar)
{
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.f32 [%0], %1, [%2];" :: "r"(addr), "f"(v), "r"(mbar) : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t addr)
{
    uint4 r;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr));
    return r;
}
__device__ __forceinline__ void mbar_wait_a(uint32_t bar_addr, uint32_t parity)
{
    asm volatile("{\n\t.reg .pred p;\n\tWAIT_LOOP:\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
                 "@p bra DONE;\n\tbra WAIT_LOOP;\n\tDONE:\n\t}" :: "r"(bar_addr), "r"(parity) : "memory");
}
__device__ __forceinline__ void mbar_arrive_a(uint32_t bar_addr)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(bar_addr) : "memory");
}
__device__ __forceinline__ void st_release_sys_u32(unsigned* p, unsigned v)
{
    asm volatile("st.release.sys.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_sys_u32(const unsigned* p)
{
    unsigned v; asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v;
}
__device__ __forceinline__ float ld_relaxed_sys_f32(const float* p)
{
    float v; asm volatile("ld.relaxed.sys.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory"); return v;
}
__device__ __forceinline__ void consumer_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

template <int PRO, int EPI>
__global__ void __launch_bounds__(THREADS, GV_MINB) q4_gemv_kernel(const __grid_constant__ GemvArgs a)
{
    extern __shared__ __align__(128) unsigned char smem[];
    const int cs = a.cs, M = a.M, K = a.K, spt = a.spt;
    unsigned char* ring = smem + ((1024u - (smem_u32(smem) & 1023u)) & 1023u);    // NST x STAGE_BYTES, 1 KB aligned (swizzle atom)
    unsigned char* sc_s = ring + NST * STAGE_BYTES;                               // GMAXC x 256
    unsigned char* zq_s = sc_s + GMAXC * SC_ROW;                                  // GMAXC x 64 (raw packed zeros)
    unsigned char* seg_s = zq_s + GMAXC * ZQ_ROW;                                 // GMAXC x 8 tokens x {sum x_q, x scale}
    float* red = reinterpret_cast<float*>(seg_s + SEG_BYTES);                     // WK x 8 x RED_LD
    constexpr int NSUB_ = (EPI == GV_EPI_SILU_MUL) ? 2 : 1;
    float* slots = red + WK * GV_MAXM * RED_LD;                                   // NSUB x cs x M x 128 (cluster reduction)
    unsigned char* xs = reinterpret_cast<unsigned char*>(slots + NSUB_ * cs * M * GV_TILE_N);   // M x xs_stride
    __shared__ __align__(8) unsigned long long full_bar[NST], empty_bar[NST], sc_bar, red_bar[2];
    __shared__ float s_rm[GV_MAXM];
    __shared__ float s_wsum[CONSUMERS / 32];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int rank = cs > 1 ? (int)cluster_ctarank() : 0;
    const int item = blockIdx.x / cs;
    constexpr int NSUB = (EPI == GV_EPI_SILU_MUL) ? 2 : 1;
    const int k8_lim = K >> 3;
    const int sg0 = rank * spt / cs, sg1 = (rank + 1) * spt / cs;       // this CTA's K slice, in ring stages

    if (tid == 0) {
        #pragma unroll
        for (int i = 0; i < NST; i++) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], WN); }
        mbar_init(&sc_bar, 1);
        // split-K partials of the other cs-1 CTAs land in this (leader) CTA's slots through st.async, counted in bytes
        #pragma unroll
        for (int i = 0; i < 2; i++) {
            mbar_init(&red_bar[i], 1);
            if (cs > 1 && rank == 0) mbar_expect_tx(&red_bar[i], (uint32_t)(cs - 1) * (uint32_t)M * GV_TILE_N * 4u);
        }
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();
    if (cs > 1) cluster_arrive_relaxed();  // #0: "this CTA is running" -- waited on before the first DSMEM store

    // resolve (item, sub) -> matrix + column tile
    auto resolve = [&](int sub, int& mi, int& ctile) {
        if (EPI == GV_EPI_SILU_MUL) { mi = sub; ctile = item; }
        else {
            mi = 0;
            if (a.num_mats > 1 && item >= a.mats[1].tile0) mi = 1;
            if (a.num_mats > 2 && item >= a.mats[2].tile0) mi = 2;
            ctile = item - (mi == 0 ? a.mats[0].tile0 : (mi == 1 ? a.mats[1].tile0 : a.mats[2].tile0));
        }
    };

    if (warp == CONSUMERS / 32) {
        // =============================== producer warp: weight stages via TMA bulk copies ===============================
        int j = 0, pslot = 0; uint32_t pphase = 0;     // pphase: parity of the fill the consumers are waiting for
        for (int sub = 0; sub < NSUB; sub++) {
            int mi, ctile; resolve(sub, mi, ctile);
            const CUtensorMap* tm = &a.tmaps[mi];
            const int N = mi == 0 ? a.mats[0].N : (mi == 1 ? a.mats[1].N : a.mats[2].N);
            const int col_tile0 = ctile * GV_TILE_N;
            const int nbox = (min(GV_TILE_N, N - col_tile0) + BOX_COLS - 1) / BOX_COLS;     // column-warps with real columns
            for (int sg = sg0; sg < sg1; sg++, j++) {
                const int slot = pslot;
                if (j >= NST) mbar_wait(&empty_bar[slot], pphase ^ 1u);
                const bool skip = (a.debug & 1) != 0;
                // out-of-range rows / columns of a box are zero-filled by the TMA unit and still count as bytes
                if (lane == 0) mbar_expect_tx(&full_bar[slot], skip ? 0u : (uint32_t)nbox * BOX_BYTES);
                __syncwarp();
                if (lane < nbox && !skip)
                    tma_load_2d(ring + slot * STAGE_BYTES + lane * BOX_BYTES, tm, col_tile0 + lane * BOX_COLS, sg * STAGE_ROWS, &full_bar[slot]);
                if (++pslot == NST) { pslot = 0; pphase ^= 1u; }
            }
            if (sub == NSUB - 1) pdl_launch_dependents();     // every weight byte of this CTA has been requested
        }
        return;
    }

    // =============================================== consumer warps ===============================================
    const int wn = warp & (WN - 1), wk = warp >> 2;
    const int g = lane >> 2, t = lane & 3;
    const int pg = (g >> 1) | ((g & 1) << 2);      // column chunk owned by this lane (bank-conflict-free with the 128B swizzle)
    const int lane_col = wn * 32 + 4 * pg;
    const int xrow = min(g, M - 1);
    const int ecol = tid & (GV_TILE_N - 1);
    const int em0 = tid >> 7;                 // 0 or 1; this thread owns rows em0, em0+2, em0+4, em0+6
    uint32_t sc_parity = 0;
    bool waited_dep = false;
    int jbase = 0;                 // ring position of this sub-tile's first stage
    float v[4] = {0.f, 0.f, 0.f, 0.f}, vprev[4] = {0.f, 0.f, 0.f, 0.f};
    int mi = 0, ctile = 0;

    // o holds the leader's own partial on entry; the other ranks' partials are added in rank order (deterministic)
    auto sum_slots = [&](int buf, float (&o)[4]) {
        for (int r = 1; r < cs; r++) {
            const float* sp = slots + ((size_t)(buf * cs + r) * M) * GV_TILE_N;
            #pragma unroll
            for (int i = 0; i < 4; i++) { const int m = em0 + 2 * i; if (m < M) o[i] += sp[m * GV_TILE_N + ecol]; }
        }
    };

    for (int sub = 0; sub < NSUB; sub++) {
        resolve(sub, mi, ctile);
        const uint32_t* qz = mi == 0 ? a.mats[0].qz : (mi == 1 ? a.mats[1].qz : a.mats[2].qz);
        const half* scp = mi == 0 ? a.mats[0].sc : (mi == 1 ? a.mats[1].sc : a.mats[2].sc);
        const int N = mi == 0 ? a.mats[0].N : (mi == 1 ? a.mats[1].N : a.mats[2].N);
        const int col_tile0 = ctile * GV_TILE_N;
        const int tile_cols = min(GV_TILE_N, N - col_tile0);
        const bool col_ok = (wn * 32) < tile_cols;             // warp-uniform (N % 32 == 0)

        Accum A;
        #pragma unroll
        for (int j = 0; j < 8; j++) { A.acc[j] = 0.f; A.ia[j] = 0; A.ib[j] = 0; }
        #pragma unroll
        for (int j = 0; j < 4; j++) A.cs[j] = 0.f;
        A.zp4 = 0; A.sxq[0] = A.sxq[1] = 0; A.sxs[0] = A.sxs[1] = 0.f;
        A.cur_grp = -1; A.fresh = true;

        for (int c0 = sg0; c0 < sg1; c0 += a.chunk_stages) {
            const int c1 = min(sg1, c0 + a.chunk_stages);
            const int g_lo = a.groups == 1 ? 0 : ((c0 * 4) >> a.gs_shift32);
            const int g_hi = a.groups == 1 ? 0 : min(a.groups - 1, ((c1 * 4 - 1) >> a.gs_shift32));

            consumer_sync();                 // previous chunk / sub-tile finished with sc_s, zq_s, xs, red
            // ---- scales / zeros of groups [g_lo, g_hi] for this tile's columns: TMA bulk copies onto sc_bar ----
            if (warp == 0) {
                const int ng = g_hi - g_lo + 1;
                const uint32_t sc_bytes = (uint32_t)tile_cols * 2, zq_bytes = (uint32_t)tile_cols / 2;
                if (lane == 0) mbar_expect_tx(&sc_bar, (uint32_t)ng * (sc_bytes + zq_bytes));
                __syncwarp();
                for (int gi = lane; gi < ng; gi += 32) {
                    bulk_g2s(sc_s + gi * SC_ROW, scp + (size_t)(g_lo + gi) * N + col_tile0, sc_bytes, &sc_bar);
                    bulk_g2s(zq_s + gi * ZQ_ROW, qz + (size_t)(g_lo + gi) * (N >> 3) + (col_tile0 >> 3), zq_bytes, &sc_bar);
                }
            }

            const bool reuse_x = (NSUB == 2) && sub > 0 && c0 == sg0 && c1 == sg1;   // same x, same quantisation: keep it
            if (!waited_dep) {
                if (PRO == GV_PRO_RMSNORM && !a.x_map) {
                    // the norm weights are constants: pull this thread's rows towards L1 while the previous kernel drains
                    for (int idx = tid; idx < (c1 - c0) * STAGE_ROWS; idx += CONSUMERS) {
                        const int k8 = c0 * STAGE_ROWS + idx;
                        if (k8 < k8_lim) asm volatile("prefetch.global.L1 [%0];" :: "l"(a.norm_w + (size_t)k8 * 8));
                    }
                }
                pdl_wait();                  // everything below may read x / write out
                waited_dep = true;
                if (PRO == GV_PRO_RMSNORM) {
                    // row factor rm = half(rsqrt(mean(x^2) + eps))  (rms_norm.cu:20-79,113-116)
                    for (int m = 0; m < M; m++) {
                        float ss = 0.f;
                        const uint4* xr = reinterpret_cast<const uint4*>(a.x + (size_t)m * K);
                        for (int i = tid; i < K / 8; i += CONSUMERS) {
                            uint4 xv = xr[i];
                            const half2* h = reinterpret_cast<const half2*>(&xv);
                            #pragma unroll
                            for (int j = 0; j < 4; j++) { float2 f = __half22float2(h[j]); ss = fmaf(f.x, f.x, ss); ss = fmaf(f.y, f.y, ss); }
                        }
                        #pragma unroll
                        for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
                        if (lane == 0) s_wsum[warp] = ss;
                        consumer_sync();
                        if (tid == 0) {
                            float tot = 0.f;
                            for (int w = 0; w < CONSUMERS / 32; w++) tot += s_wsum[w];
                            s_rm[m] = __half2float(__float2half_rn(rsqrtf(tot * a.r_dim + a.eps)));
                        }
                        consumer_sync();
                    }
                }
            }

            // ---- stage x[:, c0*128 .. c1*128) into smem: one k8-row (8 values) of one token per thread ----
            // fp16 after the act-order gather / RMS norm, exactly as the reference's separate kernels produce it
            const int k8_0 = c0 * STAGE_ROWS;
            auto stage_row = [&](int m, int j) -> uint4 {
                const int k8 = k8_0 + j;
                uint4 xv = make_uint4(0, 0, 0, 0);
                if (k8 < k8_lim) {
                    const half* xr = a.x + (size_t)m * K;
                    if (a.x_map) {
                        const uint32_t* mp = a.x_map + (size_t)k8 * 8;
                        unsigned short h[8];
                        #pragma unroll
                        for (int i = 0; i < 8; i++) h[i] = __half_as_ushort(xr[mp[i]]);
                        xv.x = h[0] | ((uint32_t)h[1] << 16); xv.y = h[2] | ((uint32_t)h[3] << 16);
                        xv.z = h[4] | ((uint32_t)h[5] << 16); xv.w = h[6] | ((uint32_t)h[7] << 16);
                    } else {
                        xv = *reinterpret_cast<const uint4*>(xr + (size_t)k8 * 8);
                    }
                    if (PRO == GV_PRO_RMSNORM) {
                        // (x * rm) * w with two fp16 multiplies, as rms_norm_kernel (rms_norm.cu:118-131)
                        const half2 rm2 = __float2half2_rn(s_rm[m]);
                        half2* hv = reinterpret_cast<half2*>(&xv);
                        if (a.x_map) {
                            const uint32_t* mp = a.x_map + (size_t)k8 * 8;
                            #pragma unroll
                            for (int i = 0; i < 4; i++) {
                                half2 w2 = __halves2half2(a.norm_w[mp[2 * i]], a.norm_w[mp[2 * i + 1]]);
                                hv[i] = __hmul2(__hmul2(hv[i], rm2), w2);
                            }
                        } else {
                            uint4 wv = *reinterpret_cast<const uint4*>(a.norm_w + (size_t)k8 * 8);
                            const half2* w2 = reinterpret_cast<const half2*>(&wv);
                            #pragma unroll
                            for (int i = 0; i < 4; i++) hv[i] = __hmul2(__hmul2(hv[i], rm2), w2[i]);
                        }
                    }
                }
                return xv;
            };
            // ---- quantise each (token, segment) of x to 16-bit integers with its own scale ----
            if (!reuse_x) {
                const int nseg = g_hi - g_lo + 1;
                const int rows_lo = c0 * STAGE_ROWS, rows_hi = min(c1 * STAGE_ROWS, k8_lim);
                const int nrows = (c1 - c0) * STAGE_ROWS;
                const int rpg = a.groups > 1 ? (4 << a.gs_shift32) : (1 << 30);       // k8-rows per quantisation group
                uint4* table = reinterpret_cast<uint4*>(seg_s);
                for (int idx = tid; idx < nseg * (GV_MAXM - M); idx += CONSUMERS)       // unused tokens: scale 0
                    table[(idx / (GV_MAXM - M)) * GV_MAXM + M + idx % (GV_MAXM - M)] = make_uint4(0, 0, 0, 0);
                if (rpg <= STAGE_ROWS) {
                    // a segment is rpg (4, 8 or 16) consecutive rows inside one ring stage: one thread per row,
                    // max / sum over the segment with width-rpg shuffles (nrows and the thread count are multiples of rpg)
                    for (int base = 0; base < M * nrows; base += CONSUMERS) {
                        const int idx = base + tid;
                        const bool act = idx < M * nrows;
                        const int m = act ? idx / nrows : 0, rr = act ? idx - m * nrows : 0;
                        uint4* rp = reinterpret_cast<uint4*>(xs + (size_t)m * a.xs_stride + (size_t)rr * 16);
                        const uint4 hv = act ? stage_row(m, rr) : make_uint4(0, 0, 0, 0);      // straight from registers: no fp16 round trip
                        float mx = row_absmax(hv);
                        for (int o = rpg >> 1; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
                        uint4 q;
                        int sum = quantise_row(hv, mx > 0.f ? 32767.0f / mx : 0.f, q);
                        for (int o = rpg >> 1; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
                        if (act) {
                            *rp = q;
                            const int r = rows_lo + rr;                       // absolute k8-row
                            if ((r & (rpg - 1)) == 0) {
                                const int gi = r / rpg - g_lo;
                                const int par = (r / STAGE_ROWS - sg0) & 1;             // parity of the stage inside this CTA's slice
                                table[gi * GV_MAXM + m] = make_uint4(par ? 0u : (uint32_t)sum, par ? (uint32_t)sum : 0u,
                                                                     __float_as_uint(mx * (1.0f / 32767.0f)), 0u);
                            }
                        }
                    }
                } else {
                    // large groups (groupsize >= 256 or a single group): stage fp16 first, then one warp per (segment, token)
                    for (int idx = tid; idx < M * nrows; idx += CONSUMERS) {
                        const int m = idx / nrows, j = idx - m * nrows;
                        *reinterpret_cast<uint4*>(xs + (size_t)m * a.xs_stride + (size_t)j * 16) = stage_row(m, j);
                    }
                    consumer_sync();
                    for (int task = warp; task < nseg * M; task += CONSUMERS / 32) {
                        const int gi = task / M, m = task - gi * M;
                        int r_lo = rows_lo, r_hi = rows_hi;
                        if (a.groups > 1) { r_lo = max(rows_lo, (g_lo + gi) * rpg); r_hi = min(rows_hi, (g_lo + gi + 1) * rpg); }
                        unsigned char* xrow_p = xs + (size_t)m * a.xs_stride;
                        float mx = 0.f;
                        for (int r = r_lo + lane; r < r_hi; r += 32)
                            mx = fmaxf(mx, row_absmax(*reinterpret_cast<const uint4*>(xrow_p + (size_t)(r - rows_lo) * 16)));
                        #pragma unroll
                        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
                        const float inv = mx > 0.f ? 32767.0f / mx : 0.f;
                        int sum0 = 0, sum1 = 0;
                        for (int r = r_lo + lane; r < r_hi; r += 32) {
                            uint4* rp = reinterpret_cast<uint4*>(xrow_p + (size_t)(r - rows_lo) * 16);
                            uint4 q;
                            const int sm = quantise_row(*rp, inv, q);
                            *rp = q;
                            if ((r / STAGE_ROWS - sg0) & 1) sum1 += sm; else sum0 += sm;
                        }
                        #pragma unroll
                        for (int o = 16; o > 0; o >>= 1) { sum0 += __shfl_xor_sync(0xffffffffu, sum0, o); sum1 += __shfl_xor_sync(0xffffffffu, sum1, o); }
                        if (lane == 0) table[gi * GV_MAXM + m] = make_uint4((uint32_t)sum0, (uint32_t)sum1, __float_as_uint(mx * (1.0f / 32767.0f)), 0u);
                    }
                }
            }
            mbar_wait(&sc_bar, sc_parity);   // scales / zeros landed
            sc_parity ^= 1;
            consumer_sync();                 // quantised x, segment table, scales and zeros are in place

            // Whole stages alternate between the two k-warps (stage j of this CTA goes to k-warp j & 1), so a warp
            // sees 128 consecutive k per stage and switches quantisation group at most once per 4 units (gs >= 128).
            // rows of this lane inside a stage: r = u*4 + t (u = 0..3); 16-byte chunk pg is stored at pg ^ (r & 7)
            const uint32_t wa_even = smem_u32(ring) + wn * BOX_BYTES + t * 128 + ((pg ^ t) << 4);            // rows t, t+8
            const uint32_t wa_odd = smem_u32(ring) + wn * BOX_BYTES + (t + 4) * 128 + ((pg ^ (t + 4)) << 4); // rows t+4, t+12
            const uint32_t xa0 = smem_u32(xs) + (uint32_t)xrow * (uint32_t)a.xs_stride + (uint32_t)t * 16u;
            const uint32_t full0 = smem_u32(&full_bar[0]), empty0 = smem_u32(&empty_bar[0]);
            const uint32_t sc_a = smem_u32(sc_s), zq_a = smem_u32(zq_s), seg_a = smem_u32(seg_s);
            const bool tail_checks = (K % STAGE_K) != 0;       // only a ragged last stage needs per-unit bounds checks
            const bool skip_math = !col_ok || (a.debug & 5);
            const int rel_par = (wk - jbase) & 1;              // slice-relative parity of the stages this k-warp consumes
            // first stage of this chunk that belongs to this k-warp: global stage counter parity == wk
            int sg = c0 + ((wk - (jbase + (c0 - sg0))) & 1);
            // ring position of that stage; this warp then advances two stages at a time
            int slot = (jbase + (sg - sg0)) % NST;
            uint32_t phase = (uint32_t)((jbase + (sg - sg0)) / NST) & 1u;
            uint32_t xb = xa0 + (uint32_t)(sg - c0) * (STAGE_ROWS * 16);
            #define GV_UNIT_CHECKED(U_, W_, X_)                                                        \
                if (((u0 + U_) * 4 + 4) <= k8_lim) {                                                   \
                    const int grp = (u0 + U_) >> a.gs_shift32;                                         \
                    if (grp != A.cur_grp) group_switch(A, grp, g_lo, sc_a, zq_a, seg_a, lane_col, t, rel_par); \
                    unit_mma(A, W_, X_);                                                               \
                }
            #define GV_UNIT_FAST(U_, W_, X_)                                                           \
                {                                                                                      \
                    const int grp = (u0 + U_) >> gshift;                                               \
                    if (grp != A.cur_grp) group_switch(A, grp, g_lo, sc_a, zq_a, seg_a, lane_col, t, rel_par); \
                    unit_mma(A, W_, X_);                                                               \
                }
            const int gshift = a.gs_shift32;
            for (; sg < c1; sg += 2) {
                mbar_wait_a(full0 + slot * 8, phase);
                if (!skip_math) {
                    const uint32_t wb = slot * STAGE_BYTES;
                    const int u0 = sg * 4;
                    if (!tail_checks) {
                        // two units at a time keeps the live register set small (no spills at 96 registers)
                        {
                            const uint4 w0 = lds128(wa_even + wb), w1 = lds128(wa_odd + wb);
                            const uint4 x0 = lds128(xb), x1 = lds128(xb + 64);
                            GV_UNIT_FAST(0, w0, x0) GV_UNIT_FAST(1, w1, x1)
                        }
                        {
                            const uint4 w2 = lds128(wa_even + wb + 8 * 128), w3 = lds128(wa_odd + wb + 8 * 128);
                            const uint4 x2 = lds128(xb + 128), x3 = lds128(xb + 192);
                            GV_UNIT_FAST(2, w2, x2) GV_UNIT_FAST(3, w3, x3)
                        }
                    } else {
                        #pragma unroll 1
                        for (int u = 0; u < 4; u++) {      // ragged last stage (K % 128 != 0): rare, keep it compact
                            const uint4 wv = lds128(((u & 1) ? wa_odd : wa_even) + wb + (u >> 1) * 8 * 128);
                            const uint4 xv = lds128(xb + u * 64);
                            GV_UNIT_CHECKED(u, wv, xv)
                        }
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive_a(empty0 + slot * 8);
                xb += 2 * STAGE_ROWS * 16;
                slot += 2;
                if (slot >= NST) { slot -= NST; phase ^= 1u; }
            }
            #undef GV_UNIT_CHECKED
            #undef GV_UNIT_FAST
            // x scales are per (segment, chunk): close the open segment before the staging buffers are recycled
            if (A.cur_grp >= 0) { seg_flush(A); A.cur_grp = -1; }
        }
        jbase += sg1 - sg0;
        // ---- reduce the WK k-warps through shared memory: red[wk][m][col] ----
        {
            float* r = red + (size_t)wk * GV_MAXM * RED_LD;
            // acc[0..1]: col lane_col, tokens 2t, 2t+1; acc[2..3]: col +1; acc[4..5]: col +2; acc[6..7]: col +3
            #pragma unroll
            for (int j = 0; j < 4; j++) {
                r[(2 * t) * RED_LD + lane_col + j] = A.acc[2 * j];
                r[(2 * t + 1) * RED_LD + lane_col + j] = A.acc[2 * j + 1];
            }
        }
        consumer_sync();
        #pragma unroll
        for (int i = 0; i < 4; i++) {
            const int m = em0 + 2 * i;
            float sum = 0.f;
            #pragma unroll
            for (int w = 0; w < WK; w++) sum += red[(size_t)w * GV_MAXM * RED_LD + m * RED_LD + ecol];
            v[i] = sum;
        }

        if (cs > 1) {
            // ---- cluster split-K: deposit the partial in the leader's slot [sub][rank] through DSMEM ----
            if (sub == 0) cluster_wait();                     // barrier #0 complete: the leader is running, its mbarriers are initialised
            if (rank != 0) {
                const uint32_t dst = mapa_shared(smem_u32(slots + ((size_t)(sub * cs + rank) * M) * GV_TILE_N), 0);
                const uint32_t bar = mapa_shared(smem_u32(&red_bar[sub]), 0);
                #pragma unroll
                for (int i = 0; i < 4; i++) { const int m = em0 + 2 * i; if (m < M) st_async_f32(dst + (uint32_t)(m * GV_TILE_N + ecol) * 4u, v[i], bar); }
            } else if (NSUB == 2) {
                if (sub == 0) {
                    #pragma unroll
                    for (int i = 0; i < 4; i++) vprev[i] = v[i];
                } else {
                    mbar_wait(&red_bar[0], 0);                // the gate tile's partials arrived while the up tile was computed
                    sum_slots(0, vprev);
                }
            }
        } else if (NSUB == 2 && sub == 0) {
            #pragma unroll
            for (int i = 0; i < 4; i++) vprev[i] = v[i];
        }
    }
    if (cs > 1) {
        if (rank != 0) return;                                // nothing of this CTA is read by anyone: no closing cluster barrier
        mbar_wait(&red_bar[NSUB - 1], 0);
        sum_slots(NSUB - 1, v);
    }

    // ================================== epilogue (leader CTA, consumer warps) ==================================
    {
        half* outp = mi == 0 ? a.mats[0].out : (mi == 1 ? a.mats[1].out : a.mats[2].out);
        const int N = mi == 0 ? a.mats[0].N : (mi == 1 ? a.mats[1].N : a.mats[2].N);
        const int col_tile0 = ctile * GV_TILE_N;
        const int col = col_tile0 + ecol;
        if (EPI == GV_EPI_ALLREDUCE) {
            // Row-parallel projection of a tensor-parallel layer: out += sum over ranks of this rank's partial tile.
            // One-shot "push" all-reduce fused into the epilogue: the tile is stored straight into every peer's receive slot
            // over NVLink (posted writes), a system-scope release flag follows, each rank then sums the W partials out of
            // its OWN memory in rank order (bitwise identical result on every rank) and adds the residual it already holds.
            __shared__ unsigned s_epoch;
            const int W = a.tp_world, R = a.tp_rank;
            unsigned* ctl = reinterpret_cast<unsigned*>(a.tp_peers[R] + TP_DATA_BYTES + TP_FLAG_BYTES);     // {epoch, done}
            if (tid == 0) s_epoch = ld_acquire_sys_u32(ctl);        // after griddepcontrol.wait: the previous launch has bumped it
            consumer_sync();
            const unsigned epoch = s_epoch;
            const int par = (int)(epoch & 1u);
            const int tile_id = item;                                // one matrix: item == column tile
            const size_t slot_me = (((size_t)par * TP_MAX_RANKS + R) * TP_MAX_TILES + tile_id) * 8 * GV_TILE_N;
            for (int p = 0; p < W; p++) {
                if (p == R) continue;
                float* dst = reinterpret_cast<float*>(a.tp_peers[p]) + slot_me;
                #pragma unroll
                for (int i = 0; i < 4; i++) { const int m = em0 + 2 * i; if (m < M) dst[m * GV_TILE_N + ecol] = v[i]; }
            }
            __threadfence_system();
            consumer_sync();
            if (tid < W && tid != R) {
                unsigned* pf = reinterpret_cast<unsigned*>(a.tp_peers[tid] + TP_DATA_BYTES) + ((size_t)par * TP_MAX_RANKS + R) * TP_MAX_TILES + tile_id;
                st_release_sys_u32(pf, epoch + 1u);
                const unsigned* mf = reinterpret_cast<const unsigned*>(a.tp_peers[R] + TP_DATA_BYTES) + ((size_t)par * TP_MAX_RANKS + tid) * TP_MAX_TILES + tile_id;
                // bounded spin: a peer that never shows up (crashed rank, mismatched launch sequence) must not hang the GPU;
                // the miss is counted in ctl[2] (exl_tp_status) and the result of this launch is then undefined
                unsigned spins = 0;
                while (ld_acquire_sys_u32(mf) != epoch + 1u) {
                    if (++spins > TP_SPIN_LIMIT) { atomicAdd(ctl + 2, 1u); break; }
                }
            }
            consumer_sync();
            float tot[4] = {0.f, 0.f, 0.f, 0.f};
            for (int p = 0; p < W; p++) {
                if (p == R) {
                    #pragma unroll
                    for (int i = 0; i < 4; i++) tot[i] += v[i];
                } else {
                    const float* src = reinterpret_cast<const float*>(a.tp_peers[R]) + (((size_t)par * TP_MAX_RANKS + p) * TP_MAX_TILES + tile_id) * 8 * GV_TILE_N;
                    #pragma unroll
                    for (int i = 0; i < 4; i++) { const int m = em0 + 2 * i; if (m < M) tot[i] += ld_relaxed_sys_f32(src + m * GV_TILE_N + ecol); }
                }
            }
            if (col < N) {
                #pragma unroll
                for (int i = 0; i < 4; i++) {
                    const int m = em0 + 2 * i;
                    if (m < M) {
                        half* o = outp + (size_t)m * N + col;
                        *o = __float2half_rn(tot[i] + (a.no_zero ? __half2float(*o) : 0.f));
                    }
                }
            }
            // last tile of this launch bumps the epoch (device-side, so the launch sequence can live in a CUDA graph)
            consumer_sync();
            if (tid == 0) {
                const unsigned done = atomicAdd(ctl + 1, 1u);
                if (done == (unsigned)(gridDim.x / cs) - 1u) { ctl[1] = 0u; __threadfence(); st_release_sys_u32(ctl, epoch + 1u); }
            }
        } else if (EPI == GV_EPI_STORE) {
            if (col < N) {
                #pragma unroll
                for (int i = 0; i < 4; i++) {
                    const int m = em0 + 2 * i;
                    if (m < M) {
                        float r = v[i];
                        half* o = outp + (size_t)m * N + col;
                        if (a.no_zero) r += __half2float(*o);
                        *o = __float2half_rn(r);
                    }
                }
            }
        } else if (EPI == GV_EPI_ROPE_CACHE) {
            // tile == one head (head_dim == 128): rope on q / k (rope.cu:48-67), k/v written to the cache
            // (q4_attn.cu:32-51).  Rows are q_len tokens of one sequence (decode path, model.py:528).
            consumer_sync();
            half* hs = reinterpret_cast<half*>(red);          // [m][128]
            #pragma unroll
            for (int i = 0; i < 4; i++) { const int m = em0 + 2 * i; if (m < M) hs[m * GV_TILE_N + ecol] = __float2half_rn(v[i]); }
            consumer_sync();
            const int head = col_tile0 / GV_TILE_N;
            #pragma unroll
            for (int i = 0; i < 4; i++) {
                const int m = em0 + 2 * i;
                if (m < M && col < N) {
                    half val = hs[m * GV_TILE_N + ecol];
                    if (mi < 2) {
                        const int pos = a.past_len + m;
                        const half* sr = a.sin + (size_t)pos * GV_TILE_N;
                        const half* cr = a.cos + (size_t)pos * GV_TILE_N;
                        const half other = hs[m * GV_TILE_N + (ecol ^ 64)];
                        if (ecol < 64) val = __hfma(val, cr[ecol], __hmul(other, __hneg(sr[ecol])));
                        else           val = __hfma(val, cr[ecol], __hmul(other, sr[ecol]));
                    }
                    outp[(size_t)m * N + col] = val;
                    if (mi >= 1) {
                        half* cache = mi == 1 ? a.key_cache : a.value_cache;
                        cache[((size_t)head * a.max_seq_len + a.past_len + m) * GV_TILE_N + ecol] = val;
                    }
                }
            }
        } else if (EPI == GV_EPI_SILU_MUL) {
            // vprev = gate tile, v = up tile (both fully reduced): silu(gate) * up in fp16 (q4_mlp.cu:27-36,46-88)
            if (col < N) {
                #pragma unroll
                for (int i = 0; i < 4; i++) {
                    const int m = em0 + 2 * i;
                    if (m < M) a.mats[0].out[(size_t)m * N + col] = __hmul(silu_h(__float2half_rn(vprev[i])), __float2half_rn(v[i]));
                }
            }
        }
    }
}

template <int PRO, int EPI>
int launch_cfg(ExlDevice* ds, GemvArgs& a, int items, cudaStream_t stream)
{
    auto kern = q4_gemv_kernel<PRO, EPI>;
    static int attr_device_done[EXL_MAX_DEVICES] = {0};
    static int use_pdl = -1, force_cs = -1;
    if (use_pdl < 0) { const char* e = getenv("EXL_GV_PDL"); use_pdl = e ? atoi(e) : 1; }
    if (force_cs < 0) { const char* e = getenv("EXL_GV_CS"); force_cs = e ? atoi(e) : 0; }
    if (!attr_device_done[ds->device]) {
        EXL_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        attr_device_done[ds->device] = 1;
    }
    // K split factor == cluster size: the largest (<= 8) that keeps every cluster of the launch co-resident.
    static int cap_mult = -1;
    if (cap_mult < 0) { const char* e = getenv("EXL_GV_CAP"); cap_mult = e ? atoi(e) : GV_MINB; }
    const int cap = ds->num_sms * cap_mult;
    const int nsub = (EPI == GV_EPI_SILU_MUL) ? 2 : 1;
    auto smem_for = [&](int c) {
        return (size_t)1024 + (size_t)NST * STAGE_BYTES + (size_t)GMAXC * (SC_ROW + ZQ_ROW) + SEG_BYTES +
               (size_t)WK * GV_MAXM * RED_LD * sizeof(float) + (size_t)nsub * c * a.M * GV_TILE_N * sizeof(float) + (size_t)a.M * a.xs_stride;
    };
    // max co-resident clusters per cluster size, measured once per (device, M) with the occupancy API
    static int max_clusters[EXL_MAX_DEVICES][GV_MAXM + 1][MAX_CS + 1] = {};
    auto clusters_fit = [&](int c) -> int {
        int& cached = max_clusters[ds->device][a.M][c];
        if (cached == 0) {
            cudaLaunchConfig_t q; memset(&q, 0, sizeof(q));
            q.gridDim = dim3((unsigned)(c * 64)); q.blockDim = dim3(THREADS); q.dynamicSmemBytes = smem_for(c);
            cudaLaunchAttribute at[1]; at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = (unsigned)c; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
            q.attrs = at; q.numAttrs = 1;
            int n = 0;
            if (c == 1 || cudaOccupancyMaxActiveClusters(&n, kern, &q) != cudaSuccess) { cudaGetLastError(); n = cap / c; }
            cached = n > 0 ? n : -1;
        }
        return cached;
    };
    int cs = 1;
    for (int c = MAX_CS; c > 1; c--) {
        if ((long long)items * c > cap || c > a.spt) continue;
        if (nsub * c * a.M * GV_TILE_N * (int)sizeof(float) > SLOT_BUDGET) continue;
        if (clusters_fit(c) < items) continue;
        cs = c; break;
    }
    if (force_cs >= 1 && force_cs <= MAX_CS && force_cs <= a.spt && nsub * force_cs * a.M * GV_TILE_N * (int)sizeof(float) <= SLOT_BUDGET) cs = force_cs;
    a.cs = cs;
    const size_t smem = smem_for(cs);
    static const char* const pro_names[2] = {"plain", "rmsnorm"};
    static const char* const epi_names[4] = {"store", "silu_mul", "rope_cache", "allreduce"};
    const size_t used = strlen(g_last_gemv_config);       // one entry per launch of the current exl_q4_* call, in launch order
    snprintf(g_last_gemv_config + used, sizeof(g_last_gemv_config) - used, "%s%s+%s cs=%d chunk=%d items=%d", used ? "; " : "",
             pro_names[PRO], epi_names[EPI], cs, a.chunk_stages, items);

    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned)(items * cs)); cfg.blockDim = dim3(THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    int na = 0;
    if (use_pdl) {
        attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[na].val.programmaticStreamSerializationAllowed = 1;
        na++;
    }
    if (cs > 1) {
        attr[na].id = cudaLaunchAttributeClusterDimension;
        attr[na].val.clusterDim.x = (unsigned)cs; attr[na].val.clusterDim.y = 1; attr[na].val.clusterDim.z = 1;
        na++;
    }
    cfg.attrs = attr; cfg.numAttrs = na;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kern, a);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    if (e != cudaSuccess) return exl_set_err(EXL_ERR_CUDA, "launch of q4_gemv_kernel failed: %s (items %d, cs %d, smem %zu)", cudaGetErrorString(e), items, cs, smem);
    return EXL_OK;
}

} // namespace

int exl_gemv_launch(ExlDevice* ds, const half* x, int M, const exl_q4_matrix* const* mats, half* const* outs,
                    int num_mats, bool no_zero, int prologue, int epilogue, const GemvFused* fused, cudaStream_t stream)
{
    if (M < 1 || M > GV_MAXM) return exl_set_err(EXL_ERR_ARG, "q4_gemv: M=%d out of range [1,%d]", M, GV_MAXM);
    if (num_mats < 1 || num_mats > 3) return exl_set_err(EXL_ERR_ARG, "q4_gemv: num_mats=%d", num_mats);
    const exl_q4_matrix* w0 = mats[0];
    GemvArgs a;
    memset(&a, 0, sizeof(a));
    a.x = x; a.x_map = w0->x_map; a.M = M; a.K = w0->K; a.groups = w0->groups;
    if (w0->K % 32 != 0) return exl_set_err(EXL_ERR_ARG, "q4_gemv: K=%d must be a multiple of 32", w0->K);
    int gs32 = w0->groupsize / 32;
    if (w0->groups > 1 && (w0->groupsize % 32 != 0 || (gs32 & (gs32 - 1)) != 0))
        return exl_set_err(EXL_ERR_ARG, "q4_gemv: groupsize=%d must be 32 * 2^n", w0->groupsize);
    int sh = 0; while ((1 << sh) < gs32) sh++;
    a.gs_shift32 = w0->groups == 1 ? 30 : sh;
    a.spt = (w0->K + STAGE_K - 1) / STAGE_K;
    int tiles = 0;
    for (int i = 0; i < num_mats; i++) {
        const exl_q4_matrix* w = mats[i];
        if (w->K != w0->K || w->groups != w0->groups || w->x_map != w0->x_map)
            return exl_set_err(EXL_ERR_ARG, "q4_gemv: fused matrices must share K, groups and x_map");
        if (w->N % 32 != 0) return exl_set_err(EXL_ERR_ARG, "q4_gemv: N=%d must be a multiple of 32", w->N);
        a.tmaps[i] = w->tmap_w;
        a.mats[i].qw = w->qweight; a.mats[i].qz = w->qzeros; a.mats[i].sc = w->scales; a.mats[i].out = outs[i];
        a.mats[i].N = w->N; a.mats[i].tile0 = tiles;
        tiles += (w->N + GV_TILE_N - 1) / GV_TILE_N;
    }
    int items = tiles;
    if (epilogue == GV_EPI_SILU_MUL) {
        // one cluster computes the gate tile and then the up tile of the same columns and combines them in registers
        if (num_mats != 2 || mats[0]->N != mats[1]->N)
            return exl_set_err(EXL_ERR_ARG, "q4_gemv: SILU_MUL epilogue needs {gate, up} of equal width");
        items = tiles / 2;
    }
    a.num_mats = num_mats;
    a.no_zero = no_zero ? 1 : 0;
    // staging chunk: M * chunk_k * 2 bytes of x <= XS_BUDGET, and at most GMAXC quantisation groups
    int chunk_k = XS_BUDGET / (2 * M);
    if (w0->groups > 1) { int gk = (GMAXC - 1) * w0->groupsize; if (gk < chunk_k) chunk_k = gk; }
    int chunk_stages = chunk_k / STAGE_K;
    if (chunk_stages < 1) return exl_set_err(EXL_ERR_ARG, "q4_gemv: cannot stage a chunk (groupsize %d)", w0->groupsize);
    if (chunk_stages > a.spt) chunk_stages = a.spt;
    a.chunk_stages = chunk_stages;
    a.xs_stride = chunk_stages * STAGE_K * 2 + 64;
    if (const char* e = getenv("EXL_GV_DEBUG")) a.debug = atoi(e);
    a.tp_rank = ds->tp_rank; a.tp_world = ds->tp_world;
    for (int i = 0; i < 8; i++) a.tp_peers[i] = ds->tp_peers[i];
    if (fused) {
        a.norm_w = fused->norm_w; a.eps = fused->eps; a.r_dim = 1.0f / (float)w0->K;
        a.sin = fused->sin; a.cos = fused->cos; a.head_dim = fused->head_dim; a.num_heads = fused->num_heads;
        a.num_kv_heads = fused->num_kv_heads; a.past_len = fused->past_len; a.max_seq_len = fused->max_seq_len;
        a.key_cache = fused->key_cache; a.value_cache = fused->value_cache;
    }

    if (epilogue == GV_EPI_ALLREDUCE) {
        if (ds->tp_world < 2 || !ds->tp_local) return exl_set_err(EXL_ERR_STATE, "q4_gemv: all-reduce epilogue needs exl_tp_init");
        if (num_mats != 1 || items > TP_MAX_TILES) return exl_set_err(EXL_ERR_ARG, "q4_gemv: all-reduce epilogue: one matrix, <= %d tiles", TP_MAX_TILES);
        return launch_cfg<GV_PRO_PLAIN, GV_EPI_ALLREDUCE>(ds, a, items, stream);
    }
    if (prologue == GV_PRO_PLAIN && epilogue == GV_EPI_STORE) return launch_cfg<GV_PRO_PLAIN, GV_EPI_STORE>(ds, a, items, stream);
    if (prologue == GV_PRO_RMSNORM && epilogue == GV_EPI_STORE) return launch_cfg<GV_PRO_RMSNORM, GV_EPI_STORE>(ds, a, items, stream);
    if (prologue == GV_PRO_RMSNORM && epilogue == GV_EPI_ROPE_CACHE) {
        if (!fused || fused->head_dim != GV_TILE_N) return exl_set_err(EXL_ERR_ARG, "q4_gemv: rope epilogue needs head_dim == 128");
        return launch_cfg<GV_PRO_RMSNORM, GV_EPI_ROPE_CACHE>(ds, a, items, stream);
    }
    if (prologue == GV_PRO_RMSNORM && epilogue == GV_EPI_SILU_MUL) return launch_cfg<GV_PRO_RMSNORM, GV_EPI_SILU_MUL>(ds, a, items, stream);
    if (prologue == GV_PRO_PLAIN && epilogue == GV_EPI_SILU_MUL) return launch_cfg<GV_PRO_PLAIN, GV_EPI_SILU_MUL>(ds, a, items, stream);
    return exl_set_err(EXL_ERR_ARG, "q4_gemv: unsupported prologue/epilogue combination %d/%d", prologue, epilogue);
}
