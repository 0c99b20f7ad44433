// q4_gemm_tc.cu -- prefill hot path: GPTQ 4-bit fused-dequant GEMM on the 5th-gen tensor cores (tcgen05 / TMEM).
//
//   out[M, N] (=|+=) x[M, K] . W[K, N],   W[k, n] = scales[g(k), n] * (q[k, n] - (zeros[g(k), n] + 1))
//
// Replaces the reference's prefill path -- column_remap + Q4Matrix::reconstruct (a full fp16 copy of W written to and
// re-read from HBM) + cublasHgemm (exllama_ext/cuda_func/q4_matmul.cu:301-344, q4_matrix.cu:170-223) -- with one
// kernel that never materialises W:
//
//   warp 0     TMA producer: per 64-wide k-block one 128 x 64 fp16 tile of x (SWIZZLE_128B, the UMMA K-major
//              canonical layout) and the matching 8 x 128 tile of packed qweight words into a 4-stage smem ring;
//              the dequantised B operand lives in its own double buffer so the TMA ring can run 4 stages ahead
//   warps 2-17 (two groups of 8 alternating k-blocks) dequantise the packed tile into the B operand: thread = (output column n, half of the k-block), each word is one
//              16-byte k-chunk of row n of the K-major SW128 tile; value = hmul(half(q - zp), scale), bit-identical
//              to the reference's reconstruct_kernel (q4_matrix.cu:196-208); fence.proxy.async, then mbarrier
//   warp 1     one elected thread issues tcgen05.mma.cta_group::1.kind::f16 (M=128, N=128, K=16) x 4 per k-block,
//              fp32 accumulation in 128 TMEM columns; tcgen05.commit frees the smem stage / signals the epilogue
//   warps 2-17 epilogue: tcgen05.ld 32x32b.x32, fp32 -> fp16 (+ the residual already in out for no_zero), global store
//   With MT = 2 a CTA computes a 256 x 128 tile (two 128-row accumulators, 256 TMEM columns) from ONE dequantised B tile,
//   halving the unpack work per MMA.
//
// Act-order matrices gather the columns of x once per call into the library scratch (exl_column_remap) so the TMA
// tile of x is dense; the gather is 2*M*K bytes against 2*M*K*N flops of GEMM.
// fp32 accumulation of exact fp16 products: at least as accurate as the reference's cublasHgemm.
#include "exl_common.cuh"
#include <cstring>
#include <cstdlib>

namespace {

constexpr int BM = 128, BN = 128, BK = 64;    // UMMA tile; a CTA owns MT (1 or 2) M-subtiles that share one dequantised B tile
constexpr int A_BYTES = BM * BK * 2;          // 16 KB per M-subtile, K-major SW128
constexpr int WQ_BYTES = (BK / 8) * BN * 4;   // 4 KB packed words [8][128]
constexpr int B_BYTES = BN * BK * 2;          // 16 KB, K-major SW128
constexpr int DQ_WARPS = 8;                   // dequant warps per k-block
constexpr int DQ_GROUPS = 2;                  // two groups of DQ_WARPS alternate k-blocks (each has two k-block times per tile)
constexpr int TC_THREADS = 64 + DQ_GROUPS * DQ_WARPS * 32; // warp 0 TMA, warp 1 MMA + TMEM alloc, warps 2..17 dequant + epilogue

struct alignas(64) TcArgs
{
    CUtensorMap tmap_x;      // x  [M, K] fp16, box 64 (k) x 128 (m), SWIZZLE_128B
    CUtensorMap tmap_w;      // qw [K/8, N] u32, box 128 (n) x 8 (k8), no swizzle
    const uint32_t* qz; const half* sc; half* out;
    int M, N, K, groups, gs_shift32, no_zero;
};

__device__ __forceinline__ uint32_t s_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void bar_init(void* b, int c) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(s_u32(b)), "r"(c)); }
__device__ __forceinline__ void bar_expect_tx(void* b, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(s_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bar_arrive(void* b) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(s_u32(b)) : "memory"); }
__device__ __forceinline__ void bar_wait(void* b, uint32_t parity)
{
    asm volatile("{\n\t.reg .pred p;\n\tWAIT_LOOP:\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
                 "@p bra DONE;\n\tbra WAIT_LOOP;\n\tDONE:\n\t}" :: "r"(s_u32(b)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_2d(void* dst, const CUtensorMap* tm, int c0, int c1, void* bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 :: "r"(s_u32(dst)), "l"(tm), "r"(c0), "r"(c1), "r"(s_u32(bar)) : "memory");
}
// same, multicast to every CTA of the cluster in cta_mask (lands at the same smem offset, signals the same barrier offset in each)
__device__ __forceinline__ void tma_2d_mc(void* dst, const CUtensorMap* tm, int c0, int c1, void* bar, uint16_t cta_mask)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%2, %3}], [%4], %5;"
                 :: "r"(s_u32(dst)), "l"(tm), "r"(c0), "r"(c1), "r"(s_u32(bar)), "h"(cta_mask) : "memory");
}
__device__ __forceinline__ void umma_commit_mc(void* bar, uint16_t cta_mask)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 :: "r"(s_u32(bar)), "h"(cta_mask) : "memory");
}
__device__ __forceinline__ uint32_t cluster_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all()
{
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// UMMA shared-memory descriptor, K-major, SWIZZLE_128B: start >> 4 | LBO (unused) | SBO = 1024 B (8 rows x 128 B) | version 1 | layout 2
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr)
{
    return (uint64_t)((smem_addr & 0x3ffffu) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// instruction descriptor for kind::f16: D = f32, A = B = f16, both K-major, N = 128, M = 128
template <int N_> __host__ __device__ constexpr uint32_t umma_idesc() { return (1u << 4) | (0u << 7) | (0u << 10) | (0u << 15) | (0u << 16) | ((uint32_t)(N_ >> 3) << 17) | ((uint32_t)(BM >> 4) << 24); }

__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 :: "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(void* bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(s_u32(bar)) : "memory");
}

// one packed word -> 8 halves in natural k order, value = hmul(half(q - zp), scale): bit-exact reconstruct_kernel
__device__ __forceinline__ uint4 dequant8(uint32_t w, uint32_t zs, uint32_t zf, uint32_t s2)
{
    const uint32_t MLO = 0x000f000fu, MHI = 0x00f000f0u, EX = 0x64006400u, R16 = 0x2c002c00u;
    uint32_t p04, p15, p26, p37, t;
    const uint32_t w8 = w >> 8;
    asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(t) : "r"(w), "r"(MLO), "r"(EX));  asm("sub.f16x2 %0, %1, %2;" : "=r"(p04) : "r"(t), "r"(zs));
    asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(t) : "r"(w), "r"(MHI), "r"(EX));  asm("fma.rn.f16x2 %0, %1, %2, %3;" : "=r"(p15) : "r"(t), "r"(R16), "r"(zf));
    asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(t) : "r"(w8), "r"(MLO), "r"(EX)); asm("sub.f16x2 %0, %1, %2;" : "=r"(p26) : "r"(t), "r"(zs));
    asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(t) : "r"(w8), "r"(MHI), "r"(EX)); asm("fma.rn.f16x2 %0, %1, %2, %3;" : "=r"(p37) : "r"(t), "r"(R16), "r"(zf));
    uint4 o;
    o.x = __byte_perm(p04, p15, 0x5410);     // {q0, q1}
    o.y = __byte_perm(p26, p37, 0x5410);     // {q2, q3}
    o.z = __byte_perm(p04, p15, 0x7632);     // {q4, q5}
    o.w = __byte_perm(p26, p37, 0x7632);     // {q6, q7}
    asm("mul.f16x2 %0, %1, %2;" : "=r"(o.x) : "r"(o.x), "r"(s2));
    asm("mul.f16x2 %0, %1, %2;" : "=r"(o.y) : "r"(o.y), "r"(s2));
    asm("mul.f16x2 %0, %1, %2;" : "=r"(o.z) : "r"(o.z), "r"(s2));
    asm("mul.f16x2 %0, %1, %2;" : "=r"(o.w) : "r"(o.w), "r"(s2));
    return o;
}

template <int MT, int NT, int CL>
__global__ void __launch_bounds__(TC_THREADS, 1) q4_gemm_tc_kernel(const __grid_constant__ TcArgs a)
{
    // CL == 2: the two CTAs of a cluster own neighbouring N tiles of the same M rows; each loads ONE of the two x sub-tiles and
    // multicasts it to both, halving the x traffic out of L2 (the operand that dominates it: the weights arrive as 4-bit words).
    static_assert(CL == 1 || MT == 2, "multicast needs two M sub-tiles");
    constexpr int BNT = NT * BN;                                 // columns per CTA (UMMA N)
    constexpr int NSTAGE = 4;                                    // TMA ring: x sub-tiles + packed words
    constexpr int STAGE_B = MT * A_BYTES + NT * WQ_BYTES;
    constexpr int NBBUF = 2;                                     // dequantised B operand: double buffer, decoupled from the TMA ring
    constexpr int BBUF_BYTES = NT * B_BYTES;
    constexpr int TMEM_COLS = MT * BNT;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* smem = smem_raw + ((1024u - (s_u32(smem_raw) & 1023u)) & 1023u);
    __shared__ __align__(8) unsigned long long full_in[NSTAGE], empty[NSTAGE], full_b[NBBUF], empty_b[NBBUF], tmem_full;
    unsigned char* bbuf = smem + (size_t)NSTAGE * STAGE_B;       // 1 KB aligned: STAGE_B is a multiple of 1024
    __shared__ uint32_t tmem_base_s;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n0 = blockIdx.x * BNT, m0 = blockIdx.y * (BM * MT);
    const int nkb = a.K / BK;

    if (tid == 0) {
        for (int i = 0; i < NSTAGE; i++) { bar_init(&full_in[i], 1); bar_init(&empty[i], CL); }
        for (int i = 0; i < NBBUF; i++) { bar_init(&full_b[i], DQ_WARPS); bar_init(&empty_b[i], 1); }
        bar_init(&tmem_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(s_u32(&tmem_base_s)), "n"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (CL > 1) cluster_sync_all();              // peer barriers are initialised before any multicast can signal them
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = tmem_base_s;
    const uint32_t crank = CL > 1 ? cluster_rank() : 0;

    if (warp == 0) {
        // ================================ TMA producer ================================
        if (lane == 0) {
            for (int kb = 0; kb < nkb; kb++) {
                const int s = kb % NSTAGE;
                if (kb >= NSTAGE) bar_wait(&empty[s], (uint32_t)((kb / NSTAGE) - 1) & 1u);
                unsigned char* st = smem + (size_t)s * STAGE_B;
                bar_expect_tx(&full_in[s], MT * A_BYTES + NT * WQ_BYTES);
                if (CL > 1) {
                    // stage s is free only when BOTH CTAs' MMAs have drained it (empty counts CL commits)
                    tma_2d_mc(st + crank * A_BYTES, &a.tmap_x, kb * BK, m0 + (int)crank * BM, &full_in[s], (uint16_t)((1u << CL) - 1));
                } else {
                    #pragma unroll
                    for (int h = 0; h < MT; h++) tma_2d(st + h * A_BYTES, &a.tmap_x, kb * BK, m0 + h * BM, &full_in[s]);   // x tiles: (k, m)
                }
                #pragma unroll
                for (int j = 0; j < NT; j++)                                                                         // packed words: (n, k8)
                    tma_2d(st + MT * A_BYTES + j * WQ_BYTES, &a.tmap_w, n0 + j * BN, kb * (BK / 8), &full_in[s]);
            }
        }
    } else if (warp == 1) {
        // ================================ MMA issuer ================================
        for (int kb = 0; kb < nkb; kb++) {
            const int s = kb % NSTAGE, b = kb % NBBUF;
            bar_wait(&full_b[b], (uint32_t)(kb / NBBUF) & 1u);            // B dequantised (which implies stage s has landed)
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (lane == 0) {
                const uint32_t a_addr = s_u32(smem + (size_t)s * STAGE_B);
                const uint32_t b_addr = s_u32(bbuf + (size_t)b * BBUF_BYTES);
                #pragma unroll
                for (int h = 0; h < MT; h++) {
                    #pragma unroll
                    for (int k = 0; k < BK / 16; k++) {
                        const uint64_t ad = umma_desc_sw128(a_addr + h * A_BYTES + k * 32);
                        const uint64_t bd = umma_desc_sw128(b_addr + k * 32);
                        umma_f16(tmem_base + h * BNT, ad, bd, umma_idesc<BNT>(), (kb > 0 || k > 0) ? 1u : 0u);
                    }
                }
                if (CL > 1) umma_commit_mc(&empty[s], (uint16_t)((1u << CL) - 1));   // tell both producers
                else umma_commit(&empty[s]);                  // TMA stage reusable once these MMAs have read it
                umma_commit(&empty_b[b]);                     // B buffer reusable
                if (kb == nkb - 1) umma_commit(&tmem_full);   // accumulators complete
            }
            __syncwarp();
        }
    } else {
        // ================================ dequant warps ================================
        // 256 threads; NT == 1: thread = (column, half of the k-block) -> 4 words; NT == 2: thread = column -> 8 words
        const int dgrp = (tid - 64) >> 8;              // dequant group: handles k-blocks kb == dgrp (mod DQ_GROUPS)
        const int dt = (tid - 64) & 255;               // 0..255 inside the group
        const int cn = NT == 1 ? (dt & (BN - 1)) : dt; // column inside the CTA tile
        const int hh = NT == 1 ? (dt >> 7) : 0;
        constexpr int WPT = NT == 1 ? 4 : 8;           // words per thread per k-block
        const int col = n0 + cn;
        const int colc = col < a.N ? col : (a.N - 1);
        // group parameters are fetched one k-block ahead (raw words in registers) so their L2 latency never sits on the
        // dequant -> MMA critical path
        int cur_grp[2] = {-1, -1}, nxt_grp[2] = {-1, -1};
        uint32_t zs[2] = {0, 0}, zf[2] = {0, 0}, s2[2] = {0, 0};
        uint32_t nxt_zw[2] = {0, 0}; unsigned short nxt_sh[2] = {0, 0};
        const uint32_t b_off = (uint32_t)((cn >> 3) * 1024 + (cn & 7) * 128);
        const int wq_off = (cn >> 7) * (WQ_BYTES / 4) + (cn & (BN - 1));       // [tile j][row][128]
        auto fetch = [&](int u, int grp) {
            nxt_zw[u] = __ldg(a.qz + (size_t)grp * (a.N >> 3) + (colc >> 3));
            nxt_sh[u] = __half_as_ushort(__ldg(a.sc + (size_t)grp * a.N + colc));
            nxt_grp[u] = grp;
        };
        #pragma unroll
        for (int u = 0; u < WPT / 4; u++) fetch(u, a.groups == 1 ? 0 : ((dgrp * 2 + hh + u) >> a.gs_shift32));
        for (int kb = dgrp; kb < nkb; kb += DQ_GROUPS) {
            const int s = kb % NSTAGE, b = kb % NBBUF;
            unsigned char* st = smem + (size_t)s * STAGE_B;
            const uint32_t* wq = reinterpret_cast<const uint32_t*>(st + MT * A_BYTES) + wq_off + (hh * 4) * BN;
            unsigned char* bt = bbuf + (size_t)b * BBUF_BYTES + b_off;
            #pragma unroll
            for (int u = 0; u < WPT / 4; u++) {        // 32-k units of this thread
                const int grp = a.groups == 1 ? 0 : ((kb * 2 + hh + u) >> a.gs_shift32);
                if (grp != cur_grp[u]) {               // nxt_* holds exactly this group (fetched during the previous k-block)
                    const uint32_t zp = ((nxt_zw[u] >> ((colc & 7) * 4)) & 0xfu) + 1u;
                    zs[u] = (0x6400u + zp) * 0x00010001u;
                    zf[u] = (0xd400u + (zp << 4)) * 0x00010001u;
                    s2[u] = (uint32_t)nxt_sh[u] * 0x00010001u;
                    cur_grp[u] = grp;
                }
                if (kb + DQ_GROUPS < nkb) {
                    const int gn = a.groups == 1 ? 0 : (((kb + DQ_GROUPS) * 2 + hh + u) >> a.gs_shift32);
                    if (gn != nxt_grp[u]) fetch(u, gn);
                }
            }
            bar_wait(&full_in[s], (uint32_t)(kb / NSTAGE) & 1u);
            uint32_t w[WPT];
            #pragma unroll
            for (int i = 0; i < WPT; i++) w[i] = wq[i * BN];
            const int r0 = hh * 4, x7 = cn & 7;
            uint4 v[WPT];
            #pragma unroll
            for (int i = 0; i < WPT; i++) v[i] = dequant8(w[i], zs[i >> 2], zf[i >> 2], s2[i >> 2]);
            if (kb >= NBBUF) bar_wait(&empty_b[b], (uint32_t)((kb / NBBUF) - 1) & 1u);   // the MMAs that read this buffer are done
            #pragma unroll
            for (int i = 0; i < WPT; i++) {
                // row cn of the K-major SW128 tile, 16-byte chunk r stored at r ^ (cn & 7)
                *reinterpret_cast<uint4*>(bt + (((r0 + i) ^ x7) << 4)) = v[i];
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy stores -> visible to the tensor core
            __syncwarp();
            if (lane == 0) bar_arrive(&full_b[b]);
        }

        // ================================ epilogue: warp -> (TMEM lane group, column half) ================================
        bar_wait(&tmem_full, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int lane_grp = warp & 3;                                   // TMEM lanes 32*lane_grp .. +31 belong to this warp
        const int cq = (warp - 2) >> 2;                                  // column quarter of each accumulator (16 warps: 4 lane groups x 4)
        #pragma unroll 1
        for (int h = 0; h < MT; h++) {
            const int m = m0 + h * BM + lane_grp * 32 + lane;
            half* orow = a.out + (size_t)m * a.N + n0;
            #pragma unroll 1
            for (int c0 = cq * (BNT / 4); c0 < (cq + 1) * (BNT / 4); c0 += 32) {
                uint32_t r[32];
                const uint32_t taddr = tmem_base + ((uint32_t)(lane_grp * 32) << 16) + (uint32_t)(h * BNT + c0);
                asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                             "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                             : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                               "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                               "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                               "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                             : "r"(taddr));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (m < a.M) {
                    #pragma unroll
                    for (int j = 0; j < 32; j += 8) {
                        const int nn = n0 + c0 + j;
                        if (nn + 8 <= a.N) {
                            uint4 prev = make_uint4(0, 0, 0, 0);
                            if (a.no_zero) prev = *reinterpret_cast<const uint4*>(orow + c0 + j);
                            const half2* ph = reinterpret_cast<const half2*>(&prev);
                            uint4 o;
                            uint32_t* op = reinterpret_cast<uint32_t*>(&o);
                            #pragma unroll
                            for (int e = 0; e < 4; e++) {
                                float f0 = __uint_as_float(r[j + 2 * e]), f1 = __uint_as_float(r[j + 2 * e + 1]);
                                if (a.no_zero) { const float2 pf = __half22float2(ph[e]); f0 += pf.x; f1 += pf.y; }
                                const half2 hv = __floats2half2_rn(f0, f1);
                                op[e] = *reinterpret_cast<const uint32_t*>(&hv);
                            }
                            *reinterpret_cast<uint4*>(orow + c0 + j) = o;
                        } else {
                            for (int e = 0; e < 8; e++) {
                                if (nn + e < a.N) {
                                    float f = __uint_as_float(r[j + e]);
                                    if (a.no_zero) f += __half2float(orow[c0 + j + e]);
                                    orow[c0 + j + e] = __float2half_rn(f);
                                }
                            }
                        }
                    }
                }
            }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    }

    __syncthreads();
    if (CL > 1) cluster_sync_all();              // no CTA leaves while a peer may still multicast into it / signal its barriers
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "n"(TMEM_COLS) : "memory");
    }
}

typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                             const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                             CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeFn get_encode()
{
    static EncodeFn encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
            encode = (EncodeFn)fn;
    }
    return encode;
}

} // namespace

bool exl_tc_gemm_supported(const exl_q4_matrix* w, int M)
{
    if (M < 1) return false;
    if (w->K % BK != 0 || w->N % 8 != 0) return false;
    if (w->groups > 1) {
        const int gs32 = w->groupsize / 32;
        if (w->groupsize % 32 != 0 || (gs32 & (gs32 - 1)) != 0) return false;
    }
    return true;
}

int exl_tc_gemm_launch(ExlDevice* ds, const half* x, int M, const exl_q4_matrix* w, half* out, bool no_zero, cudaStream_t stream)
{
    if (!exl_tc_gemm_supported(w, M)) return exl_set_err(EXL_ERR_ARG, "tc_gemm: unsupported shape K=%d N=%d groupsize=%d", w->K, w->N, w->groupsize);
    EncodeFn encode = get_encode();
    if (!encode) return exl_set_err(EXL_ERR_CUDA, "tc_gemm: cuTensorMapEncodeTiled unavailable");

    const half* xin = x;
    if (w->x_map) {
        // act-order: gather the columns of x once (column_remap.cu:27-34) so the TMA tile is dense
        const int64_t need = (int64_t)M * w->K;
        half* xm = nullptr;
        if (ds->temp_state && ds->temp_state_numel >= need) xm = ds->temp_state;
        else { int rc = exl_own_scratch(ds, SCR_REMAP, need, &xm); if (rc != EXL_OK) return rc; }
        int rc = exl_column_remap_launch(x, xm, M, w->K, w->x_map, stream);
        if (rc != EXL_OK) return rc;
        xin = xm;
    }

    TcArgs a;
    memset(&a, 0, sizeof(a));
    {
        const cuuint64_t dims[2] = {(cuuint64_t)w->K, (cuuint64_t)M};
        const cuuint64_t strides[1] = {(cuuint64_t)w->K * 2};
        const cuuint32_t box[2] = {BK, BM};
        const cuuint32_t estr[2] = {1, 1};
        CUresult r = encode(&a.tmap_x, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, (void*)xin, dims, strides, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return exl_set_err(EXL_ERR_CUDA, "tc_gemm: tensor map for x failed (%d)", (int)r);
    }
    a.tmap_w = w->tmap_wp;
    a.qz = w->qzeros; a.sc = w->scales; a.out = out;
    a.M = M; a.N = w->N; a.K = w->K; a.groups = w->groups; a.no_zero = no_zero ? 1 : 0;
    int sh = 0; while ((32 << sh) < w->groupsize) sh++;
    a.gs_shift32 = w->groups == 1 ? 30 : sh;

    // tile choice: 256 x 256 (two accumulators x UMMA N = 256, all 512 TMEM columns) when the problem is large enough to fill
    // the machine that way -- x tiles are then reused for 256 columns, which keeps the L2 -> SM operand traffic below the
    // L2 bandwidth; smaller problems use 256 x 128 or 128 x 128 tiles for more CTAs.
    static int force_cfg = -1;
    if (force_cfg < 0) { const char* e = getenv("EXL_TC_CFG"); force_cfg = e ? atoi(e) : 0; }
    int cfg = 0;                                                   // 0: 1x1, 1: 2x1, 2: 2x2
    const long long t22 = (long long)((M + 255) / 256) * ((w->N + 255) / 256);
    const long long t21 = (long long)((M + 255) / 256) * ((w->N + 127) / 128);
    if (M > BM && t22 >= (ds->num_sms * 3) / 4) cfg = 2;
    else if (M > BM && t21 >= ds->num_sms / 2) cfg = 1;
    if (force_cfg >= 1 && force_cfg <= 3) cfg = force_cfg - 1;
    const int MTv = cfg >= 1 ? 2 : 1, NTv = cfg == 2 ? 2 : 1;
    const size_t smem = 1024 + (size_t)4 * (MTv * A_BYTES + NTv * WQ_BYTES) + (size_t)2 * NTv * B_BYTES;
    static int use_mc = -1;
    if (use_mc < 0) { const char* e = getenv("EXL_TC_MC"); use_mc = e ? atoi(e) : 0; }   // x-tile multicast across a 2-CTA cluster: implemented, measured neutral, off by default
    const bool mc = use_mc && MTv == 2;
    static int attr_done[EXL_MAX_DEVICES][3][2] = {};
    void (*kern)(const TcArgs) = nullptr;
    if (cfg == 2)      kern = mc ? q4_gemm_tc_kernel<2, 2, 2> : q4_gemm_tc_kernel<2, 2, 1>;
    else if (cfg == 1) kern = mc ? q4_gemm_tc_kernel<2, 1, 2> : q4_gemm_tc_kernel<2, 1, 1>;
    else               kern = q4_gemm_tc_kernel<1, 1, 1>;
    if (!attr_done[ds->device][cfg][mc]) {
        EXL_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done[ds->device][cfg][mc] = 1;
    }
    unsigned gx = (unsigned)((w->N + BN * NTv - 1) / (BN * NTv));
    if (mc) gx = (gx + 1) & ~1u;                 // clusters of two N tiles; a padding CTA works on out-of-range columns
    cudaLaunchConfig_t lc;
    memset(&lc, 0, sizeof(lc));
    lc.gridDim = dim3(gx, (unsigned)((M + BM * MTv - 1) / (BM * MTv)));
    lc.blockDim = dim3(TC_THREADS); lc.dynamicSmemBytes = smem; lc.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    lc.attrs = at; lc.numAttrs = mc ? 1 : 0;
    static const char* const cfg_names[3][2] = {{"128x128", "128x128"}, {"256x128", "256x128+mc"}, {"256x256", "256x256+mc"}};
    g_last_tc_config = cfg_names[cfg][mc];
    cudaError_t le = cudaLaunchKernelEx(&lc, kern, a);
    if (le != cudaSuccess) return exl_set_err(EXL_ERR_CUDA, "launch of q4_gemm_tc_kernel failed: %s", cudaGetErrorString(le));
    EXL_CHECK_LAUNCH("q4_gemm_tc_kernel");
    return EXL_OK;
}
