// gvd-b200: fp32-faithful NT GEMM on the 5th-generation tensor cores (tcgen05 + TMEM + TMA), sm_100a.
//
//   C[M,N] = act(alpha * A[M,K] . W[N,K]^T + bias)      A, W, C fp32 in HBM, K contiguous
//
// Greedy token ids must be bit-exact against an fp32 oracle, so plain TF32 (10-bit mantissa) is not
// enough (SURVEY.md section 7).  Each operand is split on the fly into tf32 "hi" + tf32 "lo"
// (x = hi + lo to ~21 bits) and three kind::tf32 MMAs accumulate  lo.hi + hi.lo + hi.hi  in the fp32
// TMEM accumulator (the classic 3xTF32 scheme), which reproduces fp32 dot products to ~1e-6 relative.
//
// Per CTA (one 128 x BN output tile, K streamed in 32-element = 128-byte slices):
//   warp 8  : TMA producer   - cp.async.bulk.tensor (SWIZZLE_128B) of the raw fp32 A / W slices into a ring
//   warps 0-7: split warps   - hi = cvt.rna.tf32(x) in place, lo = x - hi into the twin buffer,
//                              fence.proxy.async, arrive "ready"
//   warp 9  : MMA issuer     - one elected thread: 4 K-slices x 3 tcgen05.mma (M=128, N=BN, K=8) per stage,
//                              tcgen05.commit frees the stage / publishes the accumulator
//   warps 0-7: epilogue      - tcgen05.ld TMEM -> registers, bias / activation (or the fused LSTM
//                              pointwise), 128-bit global stores
// Up to three K segments (different A / W tensors) feed one accumulator, so the LSTM gate GEMMs never
// materialise a concatenated input (AttModel.py:138,147-160).
#include <cuda.h>

#include <algorithm>
#include <cstdlib>

#include "gvd_kernels.cuh"

namespace {

constexpr int TC_BM = 128;
constexpr int TC_BK = 32;                 // fp32 elements per K slice = 128 bytes = one swizzle row
constexpr int TC_SPLIT_WARPS = 8;
constexpr int TC_THREADS = (TC_SPLIT_WARPS + 2) * 32;

struct TcSeg {
    int k_len;          // K extent of this segment
    int a_k0, w_k0;     // starting K coordinate inside the A / W tensor maps
};
struct TcParams {
    TcSeg seg[3];
    int nseg;
    int M, N;
    int nh;                               // heads per batch entry: blockIdx.z = b * nh + h
    int a_mul_h, a_mul_b, w_mul_h, w_mul_b; // 0 when the operand is shared across that batch axis (stride 0), else 1
    float* C; long long ldc, sCb, sCh;
    const float* bias; long long sBb;
    const float* scale2; const float* shift2;
    int act;
    float alpha;
    // LSTM mode (mode == 1): columns are gate-major [4][UJ]; row block of W = gate*H + j0
    int mode, H, UJ;
    int cs;                               // thread-block cluster size along N (1, or 8: the A slice is TMA-multicast to the cluster)
    int lag;                              // K slices by which the register drain of a chunk trails the split (env GVD_TC_LAG)
    int dbg;                              // profiling aid (env GVD_TC_DEBUG): 1 skip MMAs, 2 skip split math, 4 skip drain loads
    float sa, sw, oscale;                 // fp16x3 variant: power-of-two operand scales applied before the fp16 split and their inverse product
    int pdl;                              // programmatic dependent launch: bit 0 launched with the attribute, bit 1 / 2: the A / W operand is constant
                                          // data (weights) and may be streamed before the predecessor kernel has finished
    int wpre;                             // fp16x3 variant: the W operand arrives already split (packed hi | lo halves, gvd_pack_f16x3): no W conversion
    const float* pre;                     // [B / pre_div, 4H] additive term or nullptr
    int pre_div;
    const float* bias1; const float* bias2;
    const float* c_prev; float* h_out; float* c_out;
    // greedy-sampler mode (mode == 2): the vocabulary-head GEMM never stores its logits; every CTA reduces its BN columns to
    // (max, sum-exp, top-2) per clip and the last CTA to finish merges them, applies the UNK rule and embeds the next token
    float* pk_part; int* pk_ticket;                         // [gridDim.x][M][8] partials, one zero-initialised counter
    long long* pk_it; long long* pk_seq; float* pk_logp;    // next token [M]; seq / logprob outputs with stride pk_stride (may be null)
    long long pk_stride;
    int pk_unk;
    const float* pk_embed; float* pk_xt; int pk_E;          // xt[M, E] = ReLU(embed[token]) for the next step
};

__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d_mc(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3, uint16_t cta_mask) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4, %5, %6}], [%2], %7;"
        ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "h"(cta_mask)
        : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t cta) {
    uint32_t ra;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(smem_u32(bar)), "r"(cta));
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(ra) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!ok);
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t smem_addr) {
    // K-major, SWIZZLE_128B canonical layout: rows of 128 B, 8-row groups 1024 B apart (SBO), LBO unused
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);            // start address        bits [0,14)
    d |= (uint64_t)1 << 16;                                // leading byte offset  bits [16,30) (ignored for swizzled K-major)
    d |= (uint64_t)(1024 >> 4) << 32;                      // stride byte offset   bits [32,46)
    d |= (uint64_t)1 << 46;                                // descriptor version 1 (Blackwell)
    d |= (uint64_t)2 << 61;                                // layout type SWIZZLE_128B
    return d;
}
__device__ __forceinline__ uint32_t make_idesc_tf32(int M, int N) {
    uint32_t d = 0;
    d |= 1u << 4;                 // c_format = F32
    d |= 2u << 7;                 // a_format = TF32
    d |= 2u << 10;                // b_format = TF32
    d |= (uint32_t)(N >> 3) << 17;
    d |= (uint32_t)(M >> 4) << 24;
    return d;                     // a/b K-major, no negate, dense
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, const float4& v) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
// round-to-nearest (ties away) to tf32 = cvt.rna.tf32.f32 for finite inputs, in two integer ops (the PTX cvt is
// emulated by ptxas with NaN/Inf handling: 5 instructions per element on the split warps' critical path)

constexpr int TC_CHUNK = 2;   // K slices (of 32) accumulated inside TMEM before the fp32 register drain
constexpr int TC_LAG = 1;     // the drain of a chunk trails the split by this many K slices

template <int BN> struct TcCfg {
    static constexpr int STAGES = (BN >= 128) ? 3 : 4;
    static constexpr int A_BYTES = TC_BM * 128;            // one buffer (hi or lo)
    static constexpr int B_BYTES = BN * 128;
    static constexpr int STAGE_BYTES = 2 * (A_BYTES + B_BYTES);
    static constexpr int TMEM_COLS = 2 * BN < 32 ? 32 : 2 * BN;          // two accumulator buffers (ping-pong)
    static constexpr int DRAIN_WARPS = (BN == 32) ? 4 : 8;               // BN=32: one thread keeps all four LSTM gates
    static constexpr int ACC = (BN == 32) ? 32 : BN / 2;                 // fp32 accumulators per drain thread
    static constexpr size_t SMEM = (size_t)STAGES * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;
};

// The tensor core adds each MMA result into the TMEM accumulator with truncation, so a long K
// reduction kept entirely in TMEM drifts (measured: 10x the fp32 CUDA-core error at K=1536).  The
// accumulator therefore only ever holds TC_CHUNK K-slices (small magnitude); the epilogue warps
// drain it into fp32 REGISTER accumulators with round-to-nearest adds while the MMA pipe fills
// the other TMEM buffer.
template <int BN>
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap mapA0, const __grid_constant__ CUtensorMap mapA1,
               const __grid_constant__ CUtensorMap mapA2, const __grid_constant__ CUtensorMap mapW0,
               const __grid_constant__ CUtensorMap mapW1, const __grid_constant__ CUtensorMap mapW2, const TcParams p) {
    using Cfg = TcCfg<BN>;
    constexpr int ST = Cfg::STAGES;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)ST * Cfg::STAGE_BYTES);
    uint64_t* ready = full + ST;
    uint64_t* empty = ready + ST;
    uint64_t* acc_full = empty + ST;          // [2]
    uint64_t* acc_empty = acc_full + 2;       // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int zb = blockIdx.z / p.nh, zh = blockIdx.z % p.nh;
    const int m0 = blockIdx.y * TC_BM;
    const int n0 = p.mode == 0 ? blockIdx.x * BN : blockIdx.x * p.UJ;   // first output column / first hidden unit (LSTM mode)

    int nkb = 0;
#pragma unroll
    for (int s = 0; s < 3; ++s)
        if (s < p.nseg) nkb += (p.seg[s].k_len + TC_BK - 1) / TC_BK;
    const int nchunks = (nkb + TC_CHUNK - 1) / TC_CHUNK;

    if (tid == 0) {
        for (int s = 0; s < ST; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&ready[s], TC_SPLIT_WARPS);
            mbar_init(&empty[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&acc_full[b], 1);
            mbar_init(&acc_empty[b], Cfg::DRAIN_WARPS);
        }
        mbar_fence_init();
    }
    if (warp == TC_SPLIT_WARPS + 1) {          // MMA warp owns the TMEM allocation
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(Cfg::TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    if (warp == TC_SPLIT_WARPS) {
        // ------------------------------------------------------------------ TMA producer
        if (lane == 0) {
            prefetch_tmap(&mapA0); prefetch_tmap(&mapW0);
            int i = 0;
            for (int sg = 0; sg < p.nseg; ++sg) {
                const CUtensorMap* ma = sg == 0 ? &mapA0 : (sg == 1 ? &mapA1 : &mapA2);
                const CUtensorMap* mw = sg == 0 ? &mapW0 : (sg == 1 ? &mapW1 : &mapW2);
                const int nb = (p.seg[sg].k_len + TC_BK - 1) / TC_BK;
                for (int kb = 0; kb < nb; ++kb, ++i) {
                    const int s = i % ST;
                    mbar_wait(&empty[s], ((uint32_t)(i / ST) & 1u) ^ 1u);
                    unsigned char* st = smem + (size_t)s * Cfg::STAGE_BYTES;
                    mbar_expect_tx(&full[s], Cfg::A_BYTES + Cfg::B_BYTES);
                    tma_load_4d(st, ma, &full[s], p.seg[sg].a_k0 + kb * TC_BK, m0, zh * p.a_mul_h, zb * p.a_mul_b);
                    if (p.mode == 0) {
                        tma_load_4d(st + 2 * Cfg::A_BYTES, mw, &full[s], p.seg[sg].w_k0 + kb * TC_BK, n0, zh * p.w_mul_h, zb * p.w_mul_b);
                    } else {
                        // gate-interleaved rows: 4 boxes of UJ rows (UJ*128 B = whole swizzle atoms when UJ == 8)
#pragma unroll
                        for (int g = 0; g < 4; ++g)
                            tma_load_4d(st + 2 * Cfg::A_BYTES + g * (BN / 4) * 128, mw, &full[s], p.seg[sg].w_k0 + kb * TC_BK,
                                        g * p.H + n0, 0, 0);
                    }
                }
            }
        }
    } else if (warp == TC_SPLIT_WARPS + 1) {
        // ------------------------------------------------------------------ MMA issuer
        if (lane == 0) {
            const uint32_t idesc = make_idesc_tf32(TC_BM, BN);
            for (int i = 0; i < nkb; ++i) {
                const int s = i % ST;
                const int c = i / TC_CHUNK, buf = c & 1;
                const bool first = (i % TC_CHUNK) == 0;
                if (first) {                                          // the drain warps have emptied this TMEM buffer
                    mbar_wait(&acc_empty[buf], ((uint32_t)(c >> 1) & 1u) ^ 1u);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                }
                mbar_wait(&ready[s], (uint32_t)(i / ST) & 1u);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t d_tmem = tmem_base + (uint32_t)(buf * BN);
                const uint32_t a_hi = smem_u32(smem + (size_t)s * Cfg::STAGE_BYTES);
                const uint32_t a_lo = a_hi + Cfg::A_BYTES;
                const uint32_t b_hi = a_hi + 2 * Cfg::A_BYTES;
                const uint32_t b_lo = b_hi + Cfg::B_BYTES;
                if (!(p.dbg & 1))
#pragma unroll
                for (int ks = 0; ks < TC_BK / 8; ++ks) {
                    const uint32_t o = ks * 32;                       // 8 tf32 = 32 bytes along K inside the swizzled row
                    const uint64_t dah = make_smem_desc_sw128(a_hi + o), dal = make_smem_desc_sw128(a_lo + o);
                    const uint64_t dbh = make_smem_desc_sw128(b_hi + o), dbl = make_smem_desc_sw128(b_lo + o);
                    umma_tf32(d_tmem, dal, dbh, idesc, (first && ks == 0) ? 0u : 1u);   // small terms first
                    umma_tf32(d_tmem, dah, dbl, idesc, 1u);
                    umma_tf32(d_tmem, dah, dbh, idesc, 1u);
                }
                umma_commit(&empty[s]);                               // stage free once these MMAs have read it
                if ((i % TC_CHUNK) == TC_CHUNK - 1 || i == nkb - 1) umma_commit(&acc_full[buf]);
            }
        }
    } else {
        // ------------------------------------------------------------------ split + drain warps (0..7)
        constexpr int F4_A = Cfg::A_BYTES / 16, F4_B = Cfg::B_BYTES / 16;
        constexpr int ACC = Cfg::ACC;
        const bool drainer = warp < Cfg::DRAIN_WARPS;
        const int q = warp & 3;                                               // TMEM lane quarter this warp may access
        const int cbeg = (Cfg::DRAIN_WARPS == 8) ? (warp >> 2) * ACC : 0;     // first accumulator column of this thread
        float acc[ACC];
#pragma unroll
        for (int j = 0; j < ACC; ++j) acc[j] = 0.f;
        int next_drain = 0;
        auto drain = [&](int c) {
            const int buf = c & 1;
            mbar_wait(&acc_full[buf], (uint32_t)(c >> 1) & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (!(p.dbg & 4))
#pragma unroll
            for (int j0 = 0; j0 < ACC; j0 += 16) {
                uint32_t r[16];
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BN + cbeg + j0);
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                    : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
                      "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                    : "r"(taddr));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int e = 0; e < 16; ++e) acc[j0 + e] += __uint_as_float(r[e]);
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[buf]);
        };
        for (int i = 0; i < nkb; ++i) {
            const int s = i % ST;
            mbar_wait(&full[s], (uint32_t)(i / ST) & 1u);
            // explicit shared-space 128-bit accesses, all loads of the slice issued before the first use
            const uint32_t st_addr = smem_u32(smem + (size_t)s * Cfg::STAGE_BYTES);
            constexpr int NA = F4_A / (TC_SPLIT_WARPS * 32);                 // float4 per thread from the A slice (4)
            constexpr int NB = (F4_B + TC_SPLIT_WARPS * 32 - 1) / (TC_SPLIT_WARPS * 32);   // from the W slice (1..4)
            float4 va[NA], vb[NB];
            if (!(p.dbg & 2)) {
#pragma unroll
            for (int j = 0; j < NA; ++j) va[j] = lds128(st_addr + (uint32_t)(tid + j * TC_SPLIT_WARPS * 32) * 16u);
#pragma unroll
            for (int j = 0; j < NB; ++j) {
                const int f = tid + j * TC_SPLIT_WARPS * 32;
                if (f < F4_B) vb[j] = lds128(st_addr + 2u * Cfg::A_BYTES + (uint32_t)f * 16u);
            }
#pragma unroll
            for (int j = 0; j < NA; ++j) {
                const uint32_t a = st_addr + (uint32_t)(tid + j * TC_SPLIT_WARPS * 32) * 16u;
                float4 h, l;
                h.x = tf32_rna(va[j].x); h.y = tf32_rna(va[j].y); h.z = tf32_rna(va[j].z); h.w = tf32_rna(va[j].w);
                l.x = va[j].x - h.x; l.y = va[j].y - h.y; l.z = va[j].z - h.z; l.w = va[j].w - h.w;
                sts128(a, h);
                sts128(a + Cfg::A_BYTES, l);
            }
#pragma unroll
            for (int j = 0; j < NB; ++j) {
                const int f = tid + j * TC_SPLIT_WARPS * 32;
                if (f < F4_B) {
                    const uint32_t a = st_addr + 2u * Cfg::A_BYTES + (uint32_t)f * 16u;
                    float4 h, l;
                    h.x = tf32_rna(vb[j].x); h.y = tf32_rna(vb[j].y); h.z = tf32_rna(vb[j].z); h.w = tf32_rna(vb[j].w);
                    l.x = vb[j].x - h.x; l.y = vb[j].y - h.y; l.z = vb[j].z - h.z; l.w = vb[j].w - h.w;
                    sts128(a, h);
                    sts128(a + Cfg::B_BYTES, l);
                }
            }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the tensor core
            __syncwarp();
            if (lane == 0) mbar_arrive(&ready[s]);
            if (drainer) {
                // chunk c is complete once K slice min((c+1)*CHUNK, nkb)-1 has been multiplied; trail it by TC_LAG slices
                while (next_drain < nchunks && i >= min((next_drain + 1) * TC_CHUNK, nkb) - 1 + p.lag) drain(next_drain++);
            }
        }
        if (drainer) {
            while (next_drain < nchunks) drain(next_drain++);
            // -------------------------------------------------------------- epilogue (from the register accumulators)
            const int m = m0 + q * 32 + lane;
            (void)m;
            if (p.mode == 0) {
                // bias / activation in registers, then stage the 128 x BN tile through shared memory (the operand ring is idle
                // now) so that every global store instruction writes whole contiguous row segments (128-bit, coalesced)
                const float* bias = p.bias ? p.bias + zb * p.sBb : nullptr;
                float* C = p.C + zb * p.sCb + zh * p.sCh;
                constexpr int LDS_ = BN + 4;
                float* Cs = reinterpret_cast<float*>(smem);
                {
                    const int row = q * 32 + lane;
#pragma unroll
                    for (int j = 0; j < ACC; j += 4) {
                        const int n = n0 + cbeg + j;
                        float v[4];
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            float x = acc[j + e] * p.alpha;
                            const int nn = n + e;
                            if (nn < p.N) {
                                if (bias) x += __ldg(bias + nn);
                                if (p.act >= GVD_ACT_RELU) x = fmaxf(x, 0.f);
                                if (p.act == GVD_ACT_RELU_AFFINE_RELU) x = fmaxf(fmaf(x, __ldg(p.scale2 + nn), __ldg(p.shift2 + nn)), 0.f);
                            }
                            v[e] = x;
                        }
                        *reinterpret_cast<float4*>(Cs + row * LDS_ + cbeg + j) = make_float4(v[0], v[1], v[2], v[3]);
                    }
                }
                asm volatile("bar.sync 2, %0;" ::"n"(Cfg::DRAIN_WARPS * 32) : "memory");
                constexpr int LANES_PER_ROW = BN / 4;                       // float4 per row
                constexpr int ROWS_PER_IT = (Cfg::DRAIN_WARPS * 32) / LANES_PER_ROW;
                const int dt = warp * 32 + lane;                            // index among the drain threads
                const int rsub = dt / LANES_PER_ROW, c4 = (dt % LANES_PER_ROW) * 4;
                const bool vec_ok = (p.ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(C) & 15) == 0);
#pragma unroll 4
                for (int r0 = 0; r0 < TC_BM; r0 += ROWS_PER_IT) {
                    const int row = r0 + rsub, mm = m0 + row, n = n0 + c4;
                    if (mm < p.M && n < p.N) {
                        const float4 v = *reinterpret_cast<const float4*>(Cs + row * LDS_ + c4);
                        float* dst = C + (long long)mm * p.ldc + n;
                        if (vec_ok && n + 3 < p.N) {
                            *reinterpret_cast<float4*>(dst) = v;
                        } else {
                            const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                            for (int e = 0; e < 4; ++e)
                                if (n + e < p.N) dst[e] = vv[e];
                        }
                    }
                }
            } else {
                // fused LSTMCell pointwise: this thread holds i,f,g,o of 8 hidden units of clip row m (AttModel.py:139,160)
                if constexpr (BN == 32) {
                    if (m < p.M) {
                        const int H = p.H;
#pragma unroll
                        for (int jj = 0; jj < 8; ++jj) {
                            const int j = n0 + jj;
                            if (j < H) {
                                float g4[4];
#pragma unroll
                                for (int g = 0; g < 4; ++g) {
                                    float v = acc[g * 8 + jj];
                                    const long long col = (long long)g * H + j;
                                    if (p.pre) v += p.pre[(long long)(p.pre_div > 1 ? m / p.pre_div : m) * 4 * H + col];
                                    if (p.bias1) v += __ldg(p.bias1 + col);
                                    if (p.bias2) v += __ldg(p.bias2 + col);
                                    g4[g] = v;
                                }
                                const float ig = sigmoid_acc(g4[0]), fg = sigmoid_acc(g4[1]), gg = tanhf(g4[2]), og = sigmoid_acc(g4[3]);
                                const float c = fg * p.c_prev[(long long)m * H + j] + ig * gg;
                                p.c_out[(long long)m * H + j] = c;
                                p.h_out[(long long)m * H + j] = og * tanhf(c);
                            }
                        }
                    }
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == TC_SPLIT_WARPS + 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(Cfg::TMEM_COLS) : "memory");
    }
}

// =====================================================================================================
// v2: the A operand's tf32 hi/lo planes live in TENSOR MEMORY (tcgen05.st), not in shared memory.
//
// Ablation of v1 on 100000x1024x2780 (GVD_TC_DEBUG): TMA alone 1.69 ms, MMA alone ~1.4 ms, full 4.1 ms — the
// TMA -> split -> MMA chain is latency-bound because a 64 KB stage (raw + lo copies of A and W) leaves room for
// only 3 stages.  Moving A's hi/lo into TMEM frees the raw A slot as soon as the split warps have read it:
//   shared memory : A raw ring (16 KB/stage, 5-7 stages) + W ring (raw->hi in place + lo, 4-7 stages)
//   tensor memory : 2 accumulator buffers (2 x BN columns) + a ring of A operand slots (64 columns each)
// so 1.5-2x more raw bytes are in flight for the same 227 KB.
// =====================================================================================================
template <int BN, bool F16 = false> struct Tc2Cfg {
    // BN = 256 (opt-in, GVD_TC_BN256): every tf32 MMA with a TMEM A operand costs ~45 cycles + 128.N/256 (profiles/r1_ncu_summary.md),
    // so the widest instruction carries the most work per fixed cost.  512 TMEM columns then hold ONE 256-column accumulator + 4 A
    // slots: no ping-pong, the register drain happens every CHUNK = 16 slices while the MMA warp pauses (~2k of ~34k cycles).
    static constexpr int NG = (BN == 32) ? 4 : 2;                        // split groups of 4 warps (K slice i is split by group i % NG)
    static constexpr int THREADS = (4 * NG + 2) * 32;
    // Every ring length is a multiple of the number of conversion groups: a stage is always converted by the same group, so no group
    // can meet a stage's second fill before its first one (mbarrier parity aliasing, see the score kernel's note).  BN = 128 needs
    // 230.7 KB of the 232.4 KB of shared memory.
    // F16 (fp16x3): the operands are split into fp16 hi + fp16 lo (same 11 significant bits per term as tf32) and multiplied by
    // kind::f16 MMAs (K = 16 per instruction, twice the tf32 rate): 6 instead of 12 MMAs per 32-wide K slice.  The W slice is converted
    // IN PLACE (a 128-byte row of 32 floats becomes 64 B of hi halves | 64 B of lo halves: one buffer per stage instead of two) and an A
    // slot takes 32 instead of 64 TMEM columns, so the rings are deeper for the same shared / tensor memory.
    static constexpr int NRA = F16 ? (BN == 256 ? 6 : 8) : (BN == 256 ? 4 : (BN == 128 ? 6 : (BN == 64 ? 6 : 8)));     // raw A stages (16 KB each)
    static constexpr int NRB = F16 ? (BN == 256 ? 4 : (BN == 128 ? 6 : 8)) : (BN == 256 ? 2 : (BN == 128 ? 4 : (BN == 64 ? 6 : 8)));   // W stages
    static constexpr int TA_COLS = F16 ? 32 : 64;                      // TMEM columns of one A-operand slot (hi | lo)
    static constexpr int NTA = F16 ? 8 : (BN >= 128 ? 4 : (BN == 64 ? 6 : 7));     // TMEM A-operand slots
    static constexpr int A_BYTES = TC_BM * 128;
    static constexpr int B_BYTES = BN * 128;
    static constexpr int B_STAGE = F16 ? B_BYTES : 2 * B_BYTES;        // tf32: hi in place + a lo copy; fp16: hi | lo packed in place
    static constexpr int ACC_BUFS = BN == 256 ? 1 : 2;
    static constexpr int CHUNK = BN == 256 ? 16 : TC_CHUNK;             // K slices accumulated in TMEM between two register drains
    static constexpr int ACC_COLS = ACC_BUFS * BN;
    static constexpr int TMEM_COLS = (ACC_COLS + NTA * TA_COLS) <= 128 ? 128 : ((ACC_COLS + NTA * TA_COLS) <= 256 ? 256 : 512);
    static constexpr int DRAIN_WARPS = (BN == 32) ? 4 : 8;
    static constexpr int ACC = (BN == 32) ? 32 : BN / 2;
    static constexpr int NBAR = 2 * NRA + 3 * NRB + 2 * NTA + 4;
    static constexpr size_t SMEM = (size_t)NRA * A_BYTES + (size_t)NRB * B_STAGE + 1024 + 8 * NBAR + 64;
    static_assert(ACC_COLS + NTA * TA_COLS <= 512, "TMEM budget");
    static_assert(NRA % NG == 0 && NRB % NG == 0, "a stage must always be converted by the same group (no parity aliasing)");
    static_assert(SMEM <= 232448, "shared-memory budget (227 KB per CTA)");
};

__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Warp-converged variants: every lane executes the asm, the hardware elects one lane inside it.  Issuing from a
// C++-level `if (lane == 0)` region makes the compiler wrap EVERY tcgen05 instruction in an ELECT / R2UR.BROADCAST /
// BRA.U.ANY convergence sequence (~7 SASS instructions per MMA), which made the issuer thread the bottleneck.
__device__ __forceinline__ void umma_tf32_ts_elect(uint32_t tmem_d, uint32_t tmem_a, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p, e;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// One K slice of 32 (= 4 tcgen05 K-steps x 3 products) + the two stage-release commits, issued from ONE asm block by
// one elected lane: a single elect.sync instead of one per instruction, operand addresses advanced inside the block.
__device__ __forceinline__ void umma_kslice_elect(uint32_t d_tmem, uint32_t a_hi, uint32_t a_lo, uint64_t b_hi, uint64_t b_lo,
                                                  uint32_t idesc, uint32_t accumulate_first, uint32_t bar_b, uint32_t bar_a) {
    asm volatile(
        "{\n\t"
        ".reg .pred e, p0, pt;\n\t"
        ".reg .b32 ah, al;\n\t"
        ".reg .b64 bh, bl;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "setp.ne.b32 p0, %6, 0;\n\t"
        "setp.eq.b32 pt, 0, 0;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [%2], %3, %5, p0;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %4, %5, pt;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %3, %5, pt;\n\t"
        "add.u32 ah, %1, 8;\n\t add.u32 al, %2, 8;\n\t add.u64 bh, %3, 2;\n\t add.u64 bl, %4, 2;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [al], bh, %5, pt;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah], bl, %5, pt;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah], bh, %5, pt;\n\t"
        "add.u32 ah, %1, 16;\n\t add.u32 al, %2, 16;\n\t add.u64 bh, %3, 4;\n\t add.u64 bl, %4, 4;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [al], bh, %5, pt;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah], bl, %5, pt;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah], bh, %5, pt;\n\t"
        "add.u32 ah, %1, 24;\n\t add.u32 al, %2, 24;\n\t add.u64 bh, %3, 6;\n\t add.u64 bl, %4, 6;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [al], bh, %5, pt;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah], bl, %5, pt;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah], bh, %5, pt;\n\t"
        "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%7];\n\t"
        "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%8];\n\t"
        "}\n" ::"r"(d_tmem), "r"(a_hi), "r"(a_lo), "l"(b_hi), "l"(b_lo), "r"(idesc), "r"(accumulate_first), "r"(bar_b), "r"(bar_a)
        : "memory");
}
// the same 12 MMAs without the stage-release commits (the caller commits once per group of slices)
__device__ __forceinline__ void umma_kslice_nocommit_elect(uint32_t d_tmem, uint32_t a_hi, uint32_t a_lo, uint64_t b_hi, uint64_t b_lo,
                                                           uint32_t idesc, uint32_t accumulate_first) {
    asm volatile(
        "{\n\t"
        ".reg .pred e, p0, pt;\n\t"
        ".reg .b32 ah, al;\n\t"
        ".reg .b64 bh, bl;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "setp.ne.b32 p0, %6, 0;\n\t"
        "setp.eq.b32 pt, 0, 0;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [%2], %3, %5, p0;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %4, %5, pt;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %3, %5, pt;\n\t"
        "add.u32 ah, %1, 8;\n\t add.u32 al, %2, 8;\n\t add.u64 bh, %3, 2;\n\t add.u64 bl, %4, 2;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [al], bh, %5, pt;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah], bl, %5, pt;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah], bh, %5, pt;\n\t"
        "add.u32 ah, %1, 16;\n\t add.u32 al, %2, 16;\n\t add.u64 bh, %3, 4;\n\t add.u64 bl, %4, 4;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [al], bh, %5, pt;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah], bl, %5, pt;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah], bh, %5, pt;\n\t"
        "add.u32 ah, %1, 24;\n\t add.u32 al, %2, 24;\n\t add.u64 bh, %3, 6;\n\t add.u64 bl, %4, 6;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [al], bh, %5, pt;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah], bl, %5, pt;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah], bh, %5, pt;\n\t"
        "}\n" ::"r"(d_tmem), "r"(a_hi), "r"(a_lo), "l"(b_hi), "l"(b_lo), "r"(idesc), "r"(accumulate_first)
        : "memory");
}
__device__ __forceinline__ void umma_commit_elect(uint64_t* bar) {
    asm volatile(
        "{\n\t"
        ".reg .pred e;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t"
        "}\n" ::"r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float* v) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
        "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
        "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
        "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
        "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
        : "memory");
}

__device__ __forceinline__ uint32_t make_idesc_f16(int M, int N) {
    uint32_t d = 0;
    d |= 1u << 4;                 // c_format = F32; a_format = b_format = 0 (F16)
    d |= (uint32_t)(N >> 3) << 17;
    d |= (uint32_t)(M >> 4) << 24;
    return d;
}
__device__ __forceinline__ void tmem_st16u(uint32_t taddr, const uint32_t* v) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
        "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]),
        "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
        : "memory");
}
// two fp32 -> packed half2 (low half = first argument); inputs already carry 11 significant bits or less (exact) or are residuals
__device__ __forceinline__ uint32_t pack_h2(float lo_elem, float hi_elem) {
    uint32_t r;
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi_elem), "f"(lo_elem));
    return r;
}
// x (scaled) -> fp16 hi | fp16 lo of 4 consecutive K values: hi = round-to-11-bits(x) (exact in fp16), lo = fp16(x - hi)
__device__ __forceinline__ void split_h4(const float4& v, float s, uint32_t& h01, uint32_t& h23, uint32_t& l01, uint32_t& l23) {
    const float x0 = v.x * s, x1 = v.y * s, x2 = v.z * s, x3 = v.w * s;
    const float a0 = tf32_rna(x0), a1 = tf32_rna(x1), a2 = tf32_rna(x2), a3 = tf32_rna(x3);
    h01 = pack_h2(a0, a1); h23 = pack_h2(a2, a3);
    l01 = pack_h2(x0 - a0, x1 - a1); l23 = pack_h2(x2 - a2, x3 - a3);
}
// One K slice of 32 in fp16x3: 2 K-steps of 16 x 3 products (lo.hi, hi.lo, hi.hi) + the two stage-release commits.  A slot: hi at
// columns [0,16) (8 per K-step), lo at [16,32); W row: hi halves at bytes [0,64) (32 per K-step), lo halves at [64,128).
__device__ __forceinline__ void umma_kslice_f16_elect(uint32_t d_tmem, uint32_t a_hi, uint64_t b_hi, uint32_t idesc, uint32_t accumulate_first,
                                                      uint32_t bar_b, uint32_t bar_a) {
    asm volatile(
        "{\n\t"
        ".reg .pred e, p0, pt;\n\t"
        ".reg .b32 ah, al;\n\t"
        ".reg .b64 bh, bl;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "setp.ne.b32 p0, %4, 0;\n\t"
        "setp.eq.b32 pt, 0, 0;\n\t"
        "add.u32 al, %1, 16;\n\t add.u64 bl, %2, 4;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], [al], %2, %3, p0;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], bl, %3, pt;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, pt;\n\t"
        "add.u32 ah, %1, 8;\n\t add.u32 al, %1, 24;\n\t add.u64 bh, %2, 2;\n\t add.u64 bl, %2, 6;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], [al], bh, %3, pt;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], [ah], bl, %3, pt;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], [ah], bh, %3, pt;\n\t"
        "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%5];\n\t"
        "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%6];\n\t"
        "}\n" ::"r"(d_tmem), "r"(a_hi), "l"(b_hi), "r"(idesc), "r"(accumulate_first), "r"(bar_b), "r"(bar_a)
        : "memory");
}

template <int BN, bool F16 = false>
__global__ void __launch_bounds__(Tc2Cfg<BN, F16>::THREADS, 1)
tc2_gemm_kernel(const __grid_constant__ CUtensorMap mapA0, const __grid_constant__ CUtensorMap mapA1,
                const __grid_constant__ CUtensorMap mapA2, const __grid_constant__ CUtensorMap mapW0,
                const __grid_constant__ CUtensorMap mapW1, const __grid_constant__ CUtensorMap mapW2, const TcParams p) {
    using Cfg = Tc2Cfg<BN, F16>;
    constexpr int NRA = Cfg::NRA, NRB = Cfg::NRB, NTA = Cfg::NTA, NG = Cfg::NG;
    constexpr int PRODUCER_WARP = 4 * NG, MMA_WARP = 4 * NG + 1;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    unsigned char* smemA = smem;                                         // NRA x 16 KB raw A slices
    unsigned char* smemB = smem + (size_t)NRA * Cfg::A_BYTES;            // NRB x (hi | lo) W slices
    uint64_t* a_full = reinterpret_cast<uint64_t*>(smemB + (size_t)NRB * Cfg::B_STAGE);
    uint64_t* a_empty = a_full + NRA;
    uint64_t* b_full = a_empty + NRA;
    uint64_t* b_ready = b_full + NRB;
    uint64_t* b_empty = b_ready + NRB;
    uint64_t* ta_ready = b_empty + NRB;
    uint64_t* ta_empty = ta_ready + NTA;
    uint64_t* acc_full = ta_empty + NTA;      // [2]
    uint64_t* acc_empty = acc_full + 2;       // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int zb = blockIdx.z / p.nh, zh = blockIdx.z % p.nh;
    const int m0 = blockIdx.y * TC_BM;
    const int n0 = p.mode != 1 ? blockIdx.x * BN : blockIdx.x * p.UJ;   // mode 1 (LSTM): first hidden unit; else first output column

    int nkb = 0;
#pragma unroll
    for (int s = 0; s < 3; ++s)
        if (s < p.nseg) nkb += (p.seg[s].k_len + TC_BK - 1) / TC_BK;
    constexpr int CHUNK = Cfg::CHUNK;
    const int nchunks = (nkb + CHUNK - 1) / CHUNK;

    if (tid == 0) {
        for (int s = 0; s < NRA; ++s) { mbar_init(&a_full[s], 1); mbar_init(&a_empty[s], 4 * p.cs); }
        for (int s = 0; s < NRB; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_ready[s], 4); mbar_init(&b_empty[s], 1); }
        for (int s = 0; s < NTA; ++s) { mbar_init(&ta_ready[s], 4); mbar_init(&ta_empty[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], Cfg::DRAIN_WARPS); }
        mbar_fence_init();
    }
    if (warp == MMA_WARP) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(Cfg::TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (p.cs > 1) cluster_sync_all();          // every CTA's barriers are initialised before any peer multicasts into it
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t tmem_a0 = tmem_base + (uint32_t)Cfg::ACC_COLS;       // first column of the A-operand ring
    const uint32_t crank = p.cs > 1 ? cluster_ctarank() : 0u;

    if (tid == 0) pdl_trigger();                  // the next kernel of the stream may be scheduled (it waits for our completion itself)
    if (warp == PRODUCER_WARP) {
        // ------------------------------------------------------------------ TMA producers: lane 0 streams A, lane 1 streams W
        if (lane == 0) {
            prefetch_tmap(&mapA0);
            if (!(p.pdl & 2)) pdl_wait();         // A produced by the predecessor kernel
            int i = 0;
            for (int sg = 0; sg < p.nseg; ++sg) {
                const CUtensorMap* ma = sg == 0 ? &mapA0 : (sg == 1 ? &mapA1 : &mapA2);
                const int nb = (p.seg[sg].k_len + TC_BK - 1) / TC_BK;
                for (int kb = 0; kb < nb; ++kb, ++i) {
                    const int s = i % NRA;
                    if (p.cs == 1) {
                        mbar_wait(&a_empty[s], ((uint32_t)(i / NRA) & 1u) ^ 1u);
                        mbar_expect_tx(&a_full[s], Cfg::A_BYTES);
                        tma_load_4d(smemA + (size_t)s * Cfg::A_BYTES, ma, &a_full[s], p.seg[sg].a_k0 + kb * TC_BK, m0, zh * p.a_mul_h, zb * p.a_mul_b);
                    } else {
                        // all CTAs of the cluster read the same 128 x 32 activation slice: each loads 1/cs of its rows and multicasts
                        // them into every peer's stage `s` (one L2 read per cluster instead of one per CTA)
                        mbar_wait_cluster(&a_empty[s], ((uint32_t)(i / NRA) & 1u) ^ 1u);       // all peers released stage s
                        mbar_expect_tx(&a_full[s], Cfg::A_BYTES);
                        const int rows = TC_BM / p.cs;
                        tma_load_4d_mc(smemA + (size_t)s * Cfg::A_BYTES + (size_t)crank * rows * 128, ma, &a_full[s], p.seg[sg].a_k0 + kb * TC_BK,
                                       m0 + (int)crank * rows, zh * p.a_mul_h, zb * p.a_mul_b, (uint16_t)((1u << p.cs) - 1u));
                    }
                }
            }
        } else if (lane == 1) {
            prefetch_tmap(&mapW0);
            if (!(p.pdl & 4)) pdl_wait();         // W produced by the predecessor kernel
            int i = 0;
            for (int sg = 0; sg < p.nseg; ++sg) {
                const CUtensorMap* mw = sg == 0 ? &mapW0 : (sg == 1 ? &mapW1 : &mapW2);
                const int nb = (p.seg[sg].k_len + TC_BK - 1) / TC_BK;
                for (int kb = 0; kb < nb; ++kb, ++i) {
                    const int s = i % NRB;
                    mbar_wait(&b_empty[s], ((uint32_t)(i / NRB) & 1u) ^ 1u);
                    unsigned char* st = smemB + (size_t)s * Cfg::B_STAGE;
                    mbar_expect_tx(&b_full[s], Cfg::B_BYTES);
                    if (p.mode != 1) {
                        tma_load_4d(st, mw, &b_full[s], p.seg[sg].w_k0 + kb * TC_BK, n0, zh * p.w_mul_h, zb * p.w_mul_b);
                    } else {
#pragma unroll
                        for (int g = 0; g < 4; ++g)
                            tma_load_4d(st + g * (BN / 4) * 128, mw, &b_full[s], p.seg[sg].w_k0 + kb * TC_BK, g * p.H + n0, 0, 0);
                    }
                }
            }
        }
    } else if (warp == MMA_WARP) {
        // ------------------------------------------------------------------ MMA issuer (A from TMEM, W from shared memory)
        // the whole warp runs this loop converged; one lane is elected inside each asm statement
        {
            const uint32_t idesc = F16 ? make_idesc_f16(TC_BM, BN) : make_idesc_tf32(TC_BM, BN);
            for (int i = 0; i < nkb; ++i) {
                const int sb = i % NRB, sa = i % NTA;
                const int c = i / CHUNK, buf = Cfg::ACC_BUFS == 2 ? (c & 1) : 0;
                const bool first = (i % CHUNK) == 0;
                if (first) mbar_wait(&acc_empty[buf], ((uint32_t)(Cfg::ACC_BUFS == 2 ? (c >> 1) : c) & 1u) ^ 1u);
                mbar_wait((F16 && p.wpre) ? &b_full[sb] : &b_ready[sb], (uint32_t)(i / NRB) & 1u);      // pre-split W: usable as the TMA delivers it
                mbar_wait(&ta_ready[sa], (uint32_t)(i / NTA) & 1u);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t d_tmem = tmem_base + (uint32_t)(buf * BN);
                const uint32_t a_hi = tmem_a0 + (uint32_t)(sa * Cfg::TA_COLS), a_lo = a_hi + 32u;
                const uint32_t b_hi = smem_u32(smemB + (size_t)sb * Cfg::B_STAGE), b_lo = b_hi + Cfg::B_BYTES;
                const uint64_t dbh0 = make_smem_desc_sw128(b_hi), dbl0 = make_smem_desc_sw128(b_lo);
                // products issued small-terms-first: lo.hi, hi.lo, hi.hi per 8-wide K step; +8 TMEM columns / +32 smem bytes per step
                if constexpr (F16) umma_kslice_f16_elect(d_tmem, a_hi, dbh0, idesc, first ? 0u : 1u, smem_u32(&b_empty[sb]), smem_u32(&ta_empty[sa]));
                else umma_kslice_elect(d_tmem, a_hi, a_lo, dbh0, dbl0, idesc, first ? 0u : 1u, smem_u32(&b_empty[sb]), smem_u32(&ta_empty[sa]));
                if ((i % CHUNK) == CHUNK - 1 || i == nkb - 1) umma_commit_elect(&acc_full[buf]);
            }
        }
    } else {
        // ------------------------------------------------------------------ split + drain warps (0..7)
        // The split warps form NG groups of 4 (one warp per TMEM lane quarter); group g splits the K slices i = g (mod NG),
        // so NG independent wait -> load -> convert -> store -> fence chains are in flight.
        constexpr int F4_B = Cfg::B_BYTES / 16;
        constexpr int NBF = F4_B / 128;                                       // float4 of the W slice per thread of a group
        constexpr int ACC = Cfg::ACC;
        const bool drainer = warp < Cfg::DRAIN_WARPS;
        const int q = warp & 3;                                               // TMEM lane quarter of this warp
        const int grp = warp >> 2;                                            // split group (K-slice parity)
        const int gt = q * 32 + lane;                                         // thread index inside the group = A row
        const int row = gt;
        const int cbeg = (Cfg::DRAIN_WARPS == 8) ? (warp >> 2) * ACC : 0;
        float acc[ACC];
#pragma unroll
        for (int j = 0; j < ACC; ++j) acc[j] = 0.f;
        int next_drain = 0;
        auto drain = [&](int c) {
            const int buf = Cfg::ACC_BUFS == 2 ? (c & 1) : 0;
            mbar_wait(&acc_full[buf], (uint32_t)(Cfg::ACC_BUFS == 2 ? (c >> 1) : c) & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (!(p.dbg & 4)) {
                // the tcgen05.ld of (up to) 64 columns are issued back to back and awaited once (a wait per 16 columns serialised the TMEM
                // round trips and paced the whole pipeline)
                constexpr int DB = ACC > 64 ? 64 : ACC;
#pragma unroll
                for (int jb = 0; jb < ACC; jb += DB) {
                    uint32_t r[DB];
#pragma unroll
                    for (int j0 = 0; j0 < DB; j0 += 16) {
                        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BN + cbeg + jb + j0);
                        asm volatile(
                            "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                            : "=r"(r[j0 + 0]), "=r"(r[j0 + 1]), "=r"(r[j0 + 2]), "=r"(r[j0 + 3]), "=r"(r[j0 + 4]), "=r"(r[j0 + 5]), "=r"(r[j0 + 6]),
                              "=r"(r[j0 + 7]), "=r"(r[j0 + 8]), "=r"(r[j0 + 9]), "=r"(r[j0 + 10]), "=r"(r[j0 + 11]), "=r"(r[j0 + 12]), "=r"(r[j0 + 13]),
                              "=r"(r[j0 + 14]), "=r"(r[j0 + 15])
                            : "r"(taddr));
                    }
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                    for (int e = 0; e < DB; ++e) {
                        if constexpr (F16) acc[jb + e] = fmaf(__uint_as_float(r[e]), p.oscale, acc[jb + e]);      // undo the power-of-two operand scales (exact)
                        else acc[jb + e] += __uint_as_float(r[e]);
                    }
                }
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[buf]);
        };
        for (int i = grp; i < nkb; i += NG) {
            const int sa = i % NRA, sb = i % NRB, st = i % NTA;
            if constexpr (F16) {
                // ---------------- fp16x3 split: A row -> TMEM slot (16 hi + 16 lo packed columns), W rows -> hi | lo halves in place
                mbar_wait(&a_full[sa], (uint32_t)(i / NRA) & 1u);
                mbar_wait(&ta_empty[st], ((uint32_t)(i / NTA) & 1u) ^ 1u);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t a_row = smem_u32(smemA + (size_t)sa * Cfg::A_BYTES) + (uint32_t)row * 128u;
                const uint32_t ta = tmem_a0 + ((uint32_t)(q * 32) << 16) + (uint32_t)(st * Cfg::TA_COLS);
                {
                    uint32_t hi[16], lo[16];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float4 v = lds128(a_row + (uint32_t)((j ^ (row & 7)) << 4));                    // undo the 128B swizzle
                        split_h4(v, p.sa, hi[2 * j], hi[2 * j + 1], lo[2 * j], lo[2 * j + 1]);
                    }
                    tmem_st16u(ta, hi);
                    tmem_st16u(ta + 16u, lo);
                }
                if (!p.wpre) {
                mbar_wait(&b_full[sb], (uint32_t)(i / NRB) & 1u);
                const uint32_t b_addr = smem_u32(smemB + (size_t)sb * Cfg::B_STAGE);
                // chunk pairs (2 x 16 B = 8 floats) of the W tile: pair u -> row u / 4, pair-in-row u % 4; a thread owns NP consecutive
                // pairs, so a row is owned by one thread (NP >= 4) or by 4 / NP consecutive lanes of one warp -> read, __syncwarp, write
                constexpr int NP = BN / 32;
                float4 w0[NP], w1[NP];
#pragma unroll
                for (int u0 = 0; u0 < NP; ++u0) {
                    const int u = gt * NP + u0, wr = u >> 2, c2 = u & 3;
                    const uint32_t rb = b_addr + (uint32_t)wr * 128u;
                    w0[u0] = lds128(rb + (uint32_t)(((2 * c2) ^ (wr & 7)) << 4));
                    w1[u0] = lds128(rb + (uint32_t)(((2 * c2 + 1) ^ (wr & 7)) << 4));
                }
                __syncwarp();
#pragma unroll
                for (int u0 = 0; u0 < NP; ++u0) {
                    const int u = gt * NP + u0, wr = u >> 2, c2 = u & 3;
                    const uint32_t rb = b_addr + (uint32_t)wr * 128u;
                    uint32_t h[4], l[4];
                    split_h4(w0[u0], p.sw, h[0], h[1], l[0], l[1]);
                    split_h4(w1[u0], p.sw, h[2], h[3], l[2], l[3]);
                    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(rb + (uint32_t)((c2 ^ (wr & 7)) << 4)), "r"(h[0]), "r"(h[1]), "r"(h[2]), "r"(h[3]) : "memory");
                    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(rb + (uint32_t)(((4 + c2) ^ (wr & 7)) << 4)), "r"(l[0]), "r"(l[1]), "r"(l[2]), "r"(l[3]) : "memory");
                }
                }
            } else if constexpr (BN == 256) {
                // 128 accumulator registers per thread leave ~70 for this loop: convert in pieces of 16 floats
                mbar_wait(&a_full[sa], (uint32_t)(i / NRA) & 1u);
                mbar_wait(&ta_empty[st], ((uint32_t)(i / NTA) & 1u) ^ 1u);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t a_row = smem_u32(smemA + (size_t)sa * Cfg::A_BYTES) + (uint32_t)row * 128u;
                const uint32_t ta = tmem_a0 + ((uint32_t)(q * 32) << 16) + (uint32_t)(st * Cfg::TA_COLS);
#pragma unroll 1
                for (int kh = 0; kh < 2; ++kh) {
                    float hi[16], lo[16];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float4 v = lds128(a_row + (uint32_t)(((kh * 4 + j) ^ (row & 7)) << 4));
                        const float x[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                        for (int e = 0; e < 4; ++e) { hi[j * 4 + e] = tf32_rna(x[e]); lo[j * 4 + e] = x[e] - hi[j * 4 + e]; }
                    }
                    tmem_st16(ta + (uint32_t)(kh * 16), hi);
                    tmem_st16(ta + 32u + (uint32_t)(kh * 16), lo);
                }
                mbar_wait(&b_full[sb], (uint32_t)(i / NRB) & 1u);
                const uint32_t b_addr = smem_u32(smemB + (size_t)sb * Cfg::B_STAGE);
#pragma unroll 1
                for (int j0 = 0; j0 < NBF; j0 += 4) {
                    float4 vb[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) vb[j] = lds128(b_addr + (uint32_t)(gt + (j0 + j) * 128) * 16u);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const uint32_t a = b_addr + (uint32_t)(gt + (j0 + j) * 128) * 16u;
                        float4 h, l;
                        h.x = tf32_rna(vb[j].x); h.y = tf32_rna(vb[j].y); h.z = tf32_rna(vb[j].z); h.w = tf32_rna(vb[j].w);
                        l.x = vb[j].x - h.x; l.y = vb[j].y - h.y; l.z = vb[j].z - h.z; l.w = vb[j].w - h.w;
                        sts128(a, h);
                        sts128(a + Cfg::B_BYTES, l);
                    }
                }
            } else {
            mbar_wait(&a_full[sa], (uint32_t)(i / NRA) & 1u);
            const uint32_t a_row = smem_u32(smemA + (size_t)sa * Cfg::A_BYTES) + (uint32_t)row * 128u;
            float4 va[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) va[j] = lds128(a_row + (uint32_t)((j ^ (row & 7)) << 4));            // undo the 128B swizzle
            mbar_wait(&b_full[sb], (uint32_t)(i / NRB) & 1u);
            const uint32_t b_addr = smem_u32(smemB + (size_t)sb * Cfg::B_STAGE);
            float4 vb[NBF];
#pragma unroll
            for (int j = 0; j < NBF; ++j) vb[j] = lds128(b_addr + (uint32_t)(gt + j * 128) * 16u);
            mbar_wait(&ta_empty[st], ((uint32_t)(i / NTA) & 1u) ^ 1u);          // the MMAs that read this TMEM slot have completed
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            // ---- A: the 32 K values of this thread's row -> tf32 hi / lo -> TMEM operand slot (hi: 32 columns, lo: next 32)
            const uint32_t ta = tmem_a0 + ((uint32_t)(q * 32) << 16) + (uint32_t)(st * Cfg::TA_COLS);
#pragma unroll
            for (int kh = 0; kh < 2; ++kh) {
                float hi[16], lo[16];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 v = va[kh * 4 + j];
                    const float x[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                    for (int e = 0; e < 4; ++e) { hi[j * 4 + e] = tf32_rna(x[e]); lo[j * 4 + e] = x[e] - hi[j * 4 + e]; }
                }
                tmem_st16(ta + (uint32_t)(kh * 16), hi);
                tmem_st16(ta + 32u + (uint32_t)(kh * 16), lo);
            }
            // ---- W: hi in place + lo copy in shared memory
#pragma unroll
            for (int j = 0; j < NBF; ++j) {
                const uint32_t a = b_addr + (uint32_t)(gt + j * 128) * 16u;
                float4 h, l;
                h.x = tf32_rna(vb[j].x); h.y = tf32_rna(vb[j].y); h.z = tf32_rna(vb[j].z); h.w = tf32_rna(vb[j].w);
                l.x = vb[j].x - h.x; l.y = vb[j].y - h.y; l.z = vb[j].z - h.z; l.w = vb[j].w - h.w;
                sts128(a, h);
                sts128(a + Cfg::B_BYTES, l);
            }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) {
                if (p.cs == 1) mbar_arrive(&a_empty[sa]);        // raw A slice consumed (it is in TMEM now)
                else
                    for (int r = 0; r < p.cs; ++r) mbar_arrive_remote(&a_empty[sa], (uint32_t)r);   // every peer refills a part of it
                mbar_arrive(&ta_ready[st]);
                if (!(F16 && p.wpre)) mbar_arrive(&b_ready[sb]);
            }
            if (drainer) {
                while (next_drain < nchunks && i >= min((next_drain + 1) * CHUNK, nkb) - 1 + (Cfg::ACC_BUFS == 2 ? p.lag : 0)) drain(next_drain++);
            }
        }
        if (drainer) {
            while (next_drain < nchunks) drain(next_drain++);
            const int m = m0 + q * 32 + lane;
            (void)m;
            pdl_wait();                           // the epilogue reads / overwrites buffers of the predecessor kernels
            if (p.mode == 3) {
                // transposed store: this thread's row m is a column of C^T; lanes = consecutive m, so every store of a warp is one 128-byte line
                float* C = p.C + zb * p.sCb + zh * p.sCh;
                if (m < p.M) {
#pragma unroll
                    for (int j = 0; j < ACC; ++j) {
                        const int n = n0 + cbeg + j;
                        if (n < p.N) C[(long long)n * p.ldc + m] = acc[j] * p.alpha;
                    }
                }
            } else if (p.mode == 0) {
                const float* bias = p.bias ? p.bias + zb * p.sBb : nullptr;
                float* C = p.C + zb * p.sCb + zh * p.sCh;
                constexpr int LDS_ = BN + 4;
                float* Cs = reinterpret_cast<float*>(smem);
                {
#pragma unroll
                    for (int j = 0; j < ACC; j += 4) {
                        const int n = n0 + cbeg + j;
                        float v[4];
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            float x = acc[j + e] * p.alpha;
                            const int nn = n + e;
                            if (nn < p.N) {
                                if (bias) x += __ldg(bias + nn);
                                if (p.act >= GVD_ACT_RELU) x = fmaxf(x, 0.f);
                                if (p.act == GVD_ACT_RELU_AFFINE_RELU) x = fmaxf(fmaf(x, __ldg(p.scale2 + nn), __ldg(p.shift2 + nn)), 0.f);
                            }
                            v[e] = x;
                        }
                        *reinterpret_cast<float4*>(Cs + row * LDS_ + cbeg + j) = make_float4(v[0], v[1], v[2], v[3]);
                    }
                }
                asm volatile("bar.sync 2, %0;" ::"n"(Cfg::DRAIN_WARPS * 32) : "memory");
                constexpr int LANES_PER_ROW = BN / 4;
                constexpr int ROWS_PER_IT = (Cfg::DRAIN_WARPS * 32) / LANES_PER_ROW;
                const int dt = warp * 32 + lane;
                const int rsub = dt / LANES_PER_ROW, c4 = (dt % LANES_PER_ROW) * 4;
                const bool vec_ok = (p.ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(C) & 15) == 0);
#pragma unroll 4
                for (int r0 = 0; r0 < TC_BM; r0 += ROWS_PER_IT) {
                    const int rr = r0 + rsub, mm = m0 + rr, n = n0 + c4;
                    if (mm < p.M && n < p.N) {
                        const float4 v = *reinterpret_cast<const float4*>(Cs + rr * LDS_ + c4);
                        float* dst = C + (long long)mm * p.ldc + n;
                        if (vec_ok && n + 3 < p.N) {
                            *reinterpret_cast<float4*>(dst) = v;
                        } else {
                            const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                            for (int e = 0; e < 4; ++e)
                                if (n + e < p.N) dst[e] = vv[e];
                        }
                    }
                }
            } else if (p.mode == 2) {
                if constexpr (BN == 32) {
                    // ---- fused greedy sampler (misc/model.py:590-594,615): log_softmax + top-2 + UNK rule without materialising logits
                    const int ncta = gridDim.x;
                    float mloc = -INFINITY, v1 = -INFINITY, v2 = -INFINITY;
                    int i1 = 0x7fffffff, i2 = 0x7fffffff;
                    float xs[32];
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const int n = n0 + j;
                        const float x = n < p.N ? acc[j] + __ldg(p.bias + n) : -INFINITY;
                        xs[j] = x;
                        mloc = fmaxf(mloc, x);
                        if (x > v1 || (x == v1 && n < i1)) { v2 = v1; i2 = i1; v1 = x; i1 = n; }
                        else if (x > v2 || (x == v2 && n < i2)) { v2 = x; i2 = n; }
                    }
                    float sloc = 0.f;
#pragma unroll
                    for (int j = 0; j < 32; ++j) sloc += (n0 + j < p.N) ? expf(xs[j] - mloc) : 0.f;
                    if (m < p.M) {
                        float* pp = p.pk_part + ((long long)blockIdx.x * p.M + m) * 8;
                        *reinterpret_cast<float4*>(pp) = make_float4(mloc, sloc, v1, __int_as_float(i1));
                        *reinterpret_cast<float2*>(pp + 4) = make_float2(v2, __int_as_float(i2));
                    }
                    __threadfence();
                    asm volatile("bar.sync 2, %0;" ::"n"(Cfg::DRAIN_WARPS * 32) : "memory");
                    int* flag = reinterpret_cast<int*>(smem);
                    if (tid == 0) *flag = (atomicAdd(p.pk_ticket, 1) == ncta - 1) ? 1 : 0;
                    asm volatile("bar.sync 2, %0;" ::"n"(Cfg::DRAIN_WARPS * 32) : "memory");
                    if (*flag) {
                        __threadfence();
                        long long* tok_s = reinterpret_cast<long long*>(smem + 64);
                        if (m < p.M) {
                            float M = -INFINITY, S = 0.f, t1 = -INFINITY, t2 = -INFINITY;
                            int j1 = 0x7fffffff, j2 = 0x7fffffff;
                            for (int cta = 0; cta < ncta; ++cta) {          // fixed merge order: independent of which CTA is last
                                const float* pp = p.pk_part + ((long long)cta * p.M + m) * 8;
                                const float4 a4 = __ldcg(reinterpret_cast<const float4*>(pp));
                                const float2 b2 = __ldcg(reinterpret_cast<const float2*>(pp + 4));
                                if (a4.x > M) { S = S * expf(M - a4.x) + a4.y; M = a4.x; } else { S = fmaf(a4.y, expf(a4.x - M), S); }
                                const float cv[2] = {a4.z, b2.x};
                                const int ci[2] = {__float_as_int(a4.w), __float_as_int(b2.y)};
#pragma unroll
                                for (int e = 0; e < 2; ++e) {
                                    if (cv[e] > t1 || (cv[e] == t1 && ci[e] < j1)) { t2 = t1; j2 = j1; t1 = cv[e]; j1 = ci[e]; }
                                    else if (cv[e] > t2 || (cv[e] == t2 && ci[e] < j2)) { t2 = cv[e]; j2 = ci[e]; }
                                }
                            }
                            const float lse = M + logf(S);
                            const bool keep = j1 != p.pk_unk;
                            const long long it = keep ? j1 : j2;
                            p.pk_it[m] = it;
                            if (p.pk_seq) p.pk_seq[(long long)m * p.pk_stride] = it;
                            if (p.pk_logp) p.pk_logp[(long long)m * p.pk_stride] = (keep ? t1 : t2) - lse;
                            tok_s[m] = it;
                        }
                        asm volatile("bar.sync 2, %0;" ::"n"(Cfg::DRAIN_WARPS * 32) : "memory");
                        if (p.pk_xt) {                                       // xt = ReLU(embed[token]) (model.py:79-82,605), coalesced
                            const int E4 = p.pk_E / 4;
                            for (int idx = tid; idx < p.M * E4; idx += Cfg::DRAIN_WARPS * 32) {
                                const int r = idx / E4, e4 = idx % E4;
                                float4 v = __ldg(reinterpret_cast<const float4*>(p.pk_embed + tok_s[r] * p.pk_E) + e4);
                                v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f);
                                reinterpret_cast<float4*>(p.pk_xt + (long long)r * p.pk_E)[e4] = v;
                            }
                        }
                        if (tid == 0) *p.pk_ticket = 0;
                    }
                }
            } else {
                if constexpr (BN == 32) {
                    if (m < p.M) {
                        const int H = p.H;
#pragma unroll
                        for (int jj = 0; jj < 8; ++jj) {
                            const int j = n0 + jj;
                            if (j < H) {
                                float g4[4];
#pragma unroll
                                for (int g = 0; g < 4; ++g) {
                                    float v = acc[g * 8 + jj];
                                    const long long col = (long long)g * H + j;
                                    if (p.pre) v += p.pre[(long long)(p.pre_div > 1 ? m / p.pre_div : m) * 4 * H + col];
                                    if (p.bias1) v += __ldg(p.bias1 + col);
                                    if (p.bias2) v += __ldg(p.bias2 + col);
                                    g4[g] = v;
                                }
                                const float ig = sigmoid_acc(g4[0]), fg = sigmoid_acc(g4[1]), gg = tanhf(g4[2]), og = sigmoid_acc(g4[3]);
                                const float c = fg * p.c_prev[(long long)m * H + j] + ig * gg;
                                p.c_out[(long long)m * H + j] = c;
                                p.h_out[(long long)m * H + j] = og * tanhf(c);
                            }
                        }
                    }
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (p.cs > 1) cluster_sync_all();          // no CTA may exit while a peer can still multicast into it or arrive on its barriers
    if (warp == MMA_WARP) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(Cfg::TMEM_COLS) : "memory");
    }
}

// =====================================================================================================
// Self-attention kernels of the region encoder (transformer.py:84-118):  S = Q_h K_h^T (K = 171 -> 6 slices),
// P = softmax(S / sqrt(d_model)),  O_h = P V_h.
//
// tc_astat_kernel — A-stationary sweep for the short-K score product: one CTA owns a 128-row block of Q for ALL keys.
//   The tf32 hi/lo planes of the whole Q block (<= 6 K slices x 64 TMEM columns) are built once and stay in tensor
//   memory; the CTA then sweeps the key dimension in 64-column tiles, streaming only K.  (The generic kernel spends
//   ~12 us per 128x128 tile of this shape on set-up, pipeline fill and the A split for 2.3 us of MMA work.)
//   PRE : the streamed operand arrives already split into tf32 hi / lo planes (gvd_split_hilo) -> no conversion warps
//         in the loop, the tile loop is bounded by the tensor pipe.
//   SMX : the epilogue is the softmax numerator.  Thread (row, 32-column group g) keeps a running maximum mu_g and
//         stores e = exp((s - mu_g)/sqrt(d)); the per-(row, group) factor F = exp((mu_g - max_row)/sqrt(d)) / sum_row is
//         written at the end of the sweep, and the P.V kernel multiplies it in while it splits its A operand — S is
//         written once and read once, and no separate softmax pass exists.
// tc_pv_kernel — O = (F * E) V: A streamed (row-scaled + split by the conversion warps), V^T pre-split, one N tile of
//   up to 192 columns so that every A slice is split exactly once.
// =====================================================================================================
struct AstatCfg {
    // NRA == NTA: every A slice has its own raw stage.  With fewer stages than slices the two conversion groups alternate on a
    // stage, and a group waiting for the SECOND fill of a stage (parity 1) before the FIRST fill has completed passes the wait on
    // the fresh barrier (parity aliasing): it then converts a half-landed slice and its early release makes the producer re-arm
    // a barrier whose phase is still open.  Seen as rare wrong score blocks / hangs with 3 stages; no reuse, no hazard.
    static constexpr int BN = 64, NRA = 6, NRB = 6, NTA = 6, NG = 2;
    static_assert(NRA == NTA && NRB % NG == 0, "see above");
    static constexpr int THREADS = (4 * NG + 2) * 32;
    static constexpr int A_BYTES = TC_BM * 128, B_BYTES = BN * 128;
    static constexpr int ACC_COLS = 2 * BN, TMEM_COLS = 512;
    static constexpr int NBAR = 2 * NRA + 3 * NRB + NTA + 4 + 1;
    static constexpr size_t SMEM = (size_t)NRA * A_BYTES + (size_t)NRB * 2 * B_BYTES + 1024 + 8 * NBAR + 64;
};
struct AttnParams {
    float* F;            // [batch][ngrp][M] softmax factors (written by SMX scores, read by P.V)
    const float* Fc;
    int ngrp;
    float c;             // log2(e) / sqrt(d_model)
    int f16;             // fp16x3: the streamed operand is an fp16x3 image (one buffer: hi | lo halves), the A slices are split to fp16 planes
    float sa;            // fp16x3: power-of-two scale of the A operand (the image carries its own; both are undone through c / alpha)
    // P.V only: store the output as the fp16x3 operand image of the next GEMM (Wo) instead of fp32 C: row (zb * M + m) of img (pitch img_ld words,
    // zb = clip of the sub-batch), head zh at columns [zh * sCh, zh * sCh + bn) with the pad columns n >= N written as zeros
    uint32_t* img; long long img_ld; float img_scale;
    int direct_store;    // scores: thread-per-row stores instead of the staged coalesced epilogue (GVD_ASTAT_DIRECT: measurement aid)
};

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}
// A slice (128 rows x 32 fp32, SWIZZLE_128B in smem) -> tf32 hi / lo -> TMEM columns [ta, ta+32) / [ta+32, ta+64); thread = row
// fp16x3 variant: 32 K values of this thread's row -> 16 packed hi words (columns [0,16)) + 16 packed lo words ([16,32)) of the slot
__device__ __forceinline__ void split_a_slice_to_tmem_f16(uint32_t a_row, int row, uint32_t ta, float scale) {
    uint32_t hi[16], lo[16];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        const float4 v = lds128(a_row + (uint32_t)((e ^ (row & 7)) << 4));
        split_h4(v, scale, hi[2 * e], hi[2 * e + 1], lo[2 * e], lo[2 * e + 1]);
    }
    tmem_st16u(ta, hi);
    tmem_st16u(ta + 16u, lo);
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
// the 6 fp16x3 MMAs of one K slice without stage-release commits
__device__ __forceinline__ void umma_kslice_f16_nocommit_elect(uint32_t d_tmem, uint32_t a_hi, uint64_t b_hi, uint32_t idesc, uint32_t accumulate_first) {
    asm volatile(
        "{\n\t"
        ".reg .pred e, p0, pt;\n\t"
        ".reg .b32 ah, al;\n\t"
        ".reg .b64 bh, bl;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "setp.ne.b32 p0, %4, 0;\n\t"
        "setp.eq.b32 pt, 0, 0;\n\t"
        "add.u32 al, %1, 16;\n\t add.u64 bl, %2, 4;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], [al], %2, %3, p0;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], bl, %3, pt;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, pt;\n\t"
        "add.u32 ah, %1, 8;\n\t add.u32 al, %1, 24;\n\t add.u64 bh, %2, 2;\n\t add.u64 bl, %2, 6;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], [al], bh, %3, pt;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], [ah], bl, %3, pt;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], [ah], bh, %3, pt;\n\t"
        "}\n" ::"r"(d_tmem), "r"(a_hi), "l"(b_hi), "r"(idesc), "r"(accumulate_first)
        : "memory");
}
__device__ __forceinline__ void split_a_slice_to_tmem(uint32_t a_row, int row, uint32_t ta, float scale) {
    float4 va[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) va[e] = lds128(a_row + (uint32_t)((e ^ (row & 7)) << 4));
#pragma unroll
    for (int kh = 0; kh < 2; ++kh) {
        float hi[16], lo[16];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float4 v = va[kh * 4 + e];
            const float x[4] = {v.x * scale, v.y * scale, v.z * scale, v.w * scale};
#pragma unroll
            for (int c = 0; c < 4; ++c) { hi[e * 4 + c] = tf32_rna(x[c]); lo[e * 4 + c] = x[c] - hi[e * 4 + c]; }
        }
        tmem_st16(ta + (uint32_t)(kh * 16), hi);
        tmem_st16(ta + 32u + (uint32_t)(kh * 16), lo);
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}

template <bool PRE, bool SMX>
__global__ void __launch_bounds__(AstatCfg::THREADS, 1)
tc_astat_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapW, const __grid_constant__ CUtensorMap mapWlo,
                const TcParams p, const AttnParams ap) {
    using Cfg = AstatCfg;
    constexpr int BN = Cfg::BN, NRA = Cfg::NRA, NRB = Cfg::NRB, NTA = Cfg::NTA, NG = Cfg::NG;
    constexpr int PRODUCER_WARP = 4 * NG, MMA_WARP = 4 * NG + 1;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    unsigned char* smemA = smem;
    unsigned char* smemB = smem + (size_t)NRA * Cfg::A_BYTES;
    uint64_t* a_full = reinterpret_cast<uint64_t*>(smemB + (size_t)NRB * 2 * Cfg::B_BYTES);
    uint64_t* a_empty = a_full + NRA;
    uint64_t* b_full = a_empty + NRA;
    uint64_t* b_ready = b_full + NRB;
    uint64_t* b_empty = b_ready + NRB;
    uint64_t* ta_ready = b_empty + NRB;       // [NTA] A slice kb is in TMEM (filled once)
    uint64_t* acc_full = ta_ready + NTA;      // [2]
    uint64_t* acc_empty = acc_full + 2;       // [2]
    uint64_t* dummy = acc_empty + 2;          // sink for the A-slot release commit of umma_kslice_elect (slots are never refilled)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(dummy + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int zb = blockIdx.z / p.nh, zh = blockIdx.z % p.nh;
    const int m0 = blockIdx.y * TC_BM;
    const int nkb = (p.seg[0].k_len + TC_BK - 1) / TC_BK;      // <= NTA (checked on the host)
    const int NT = (p.N + BN - 1) / BN;
    const int nj = NT * nkb;                                     // W slices streamed by this CTA

    if (tid == 0) {
        for (int s = 0; s < NRA; ++s) { mbar_init(&a_full[s], 1); mbar_init(&a_empty[s], 4); }
        for (int s = 0; s < NRB; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_ready[s], 4); mbar_init(&b_empty[s], 1); }
        for (int s = 0; s < NTA; ++s) mbar_init(&ta_ready[s], 4);
        for (int b = 0; b < 2; ++b) { mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], 4 * NG); }
        mbar_init(dummy, 1);
        mbar_fence_init();
    }
    if (warp == MMA_WARP) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(Cfg::TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t tmem_a0 = tmem_base + (uint32_t)Cfg::ACC_COLS;

    if (warp == PRODUCER_WARP) {
        if (lane == 0) {
            prefetch_tmap(&mapA);
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % NRA;
                mbar_wait(&a_empty[s], ((uint32_t)(kb / NRA) & 1u) ^ 1u);
                mbar_expect_tx(&a_full[s], Cfg::A_BYTES);
                tma_load_4d(smemA + (size_t)s * Cfg::A_BYTES, &mapA, &a_full[s], kb * TC_BK, m0, zh * p.a_mul_h, zb * p.a_mul_b);
            }
        } else if (lane == 1) {
            prefetch_tmap(&mapW);
            if (PRE) prefetch_tmap(&mapWlo);
            int s = 0;
            uint32_t ph = 1;
            for (int nt = 0; nt < NT; ++nt) {
                for (int kb = 0; kb < nkb; ++kb) {
                    mbar_wait(&b_empty[s], ph);
                    mbar_expect_tx(&b_full[s], (PRE && !ap.f16) ? 2 * Cfg::B_BYTES : Cfg::B_BYTES);
                    unsigned char* dst = smemB + (size_t)s * 2 * Cfg::B_BYTES;
                    tma_load_4d(dst, &mapW, &b_full[s], kb * TC_BK, nt * BN, zh * p.w_mul_h, zb * p.w_mul_b);
                    if (PRE && !ap.f16) tma_load_4d(dst + Cfg::B_BYTES, &mapWlo, &b_full[s], kb * TC_BK, nt * BN, zh * p.w_mul_h, zb * p.w_mul_b);
                    if (++s == NRB) { s = 0; ph ^= 1u; }
                }
            }
        }
    } else if (warp == MMA_WARP) {
        // The issue path is kept minimal (ncu stall sampling of the first version: the tensor pipe was 39 % active and this warp was
        // found in its own bookkeeping, not on a barrier): ring stage / phase are running counters, the shared-memory descriptors
        // advance by addition, and two K slices are waited for and issued per iteration.
        const uint32_t idesc = ap.f16 ? make_idesc_f16(TC_BM, BN) : make_idesc_tf32(TC_BM, BN);
        const uint64_t desc0 = make_smem_desc_sw128(smem_u32(smemB));                       // stage 0, hi plane
        constexpr uint64_t STAGE_UNITS = (uint64_t)(2 * Cfg::B_BYTES) >> 4, LO_UNITS = (uint64_t)Cfg::B_BYTES >> 4;
        const uint32_t dummy_bar = smem_u32(dummy);
        int s = 0;
        uint32_t ph = 0;
        for (int nt = 0; nt < NT; ++nt) {
            const int buf = nt & 1;
            const uint32_t d_tmem = tmem_base + (uint32_t)(buf * BN);
            mbar_wait(&acc_empty[buf], ((uint32_t)(nt >> 1) & 1u) ^ 1u);
            for (int kb = 0; kb < nkb; kb += 2) {
                const bool two = kb + 1 < nkb;
                int s1 = s + 1;
                uint32_t ph1 = ph;
                if (s1 == NRB) { s1 = 0; ph1 ^= 1u; }
                mbar_wait(PRE ? &b_full[s] : &b_ready[s], ph);
                if (two) mbar_wait(PRE ? &b_full[s1] : &b_ready[s1], ph1);
                if (nt == 0) {
                    mbar_wait(&ta_ready[kb], 0u);
                    if (two) mbar_wait(&ta_ready[kb + 1], 0u);
                }
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t a_hi = tmem_a0 + (uint32_t)(kb * 64);
                const uint64_t dbh = desc0 + (uint64_t)s * STAGE_UNITS;
                if (p.dbg & 8) {            // experiment switch: stage-release commits after every slice (first version)
                    umma_kslice_elect(d_tmem, a_hi, a_hi + 32u, dbh, dbh + LO_UNITS, idesc, kb == 0 ? 0u : 1u, smem_u32(&b_empty[s]), dummy_bar);
                    if (two) {
                        const uint64_t dbh1 = desc0 + (uint64_t)s1 * STAGE_UNITS;
                        umma_kslice_elect(d_tmem, a_hi + 64u, a_hi + 96u, dbh1, dbh1 + LO_UNITS, idesc, 1u, smem_u32(&b_empty[s1]), dummy_bar);
                    }
                } else if (ap.f16) {        // fp16x3: 12 MMAs (the A slot keeps its 64-column pitch, the image is one buffer per stage)
                    umma_kslice_f16_nocommit_elect(d_tmem, a_hi, dbh, idesc, kb == 0 ? 0u : 1u);
                    if (two) umma_kslice_f16_nocommit_elect(d_tmem, a_hi + 64u, desc0 + (uint64_t)s1 * STAGE_UNITS, idesc, 1u);
                    umma_commit_elect(&b_empty[s]);
                    if (two) umma_commit_elect(&b_empty[s1]);
                } else {                    // 24 MMAs, then the two stage releases
                    umma_kslice_nocommit_elect(d_tmem, a_hi, a_hi + 32u, dbh, dbh + LO_UNITS, idesc, kb == 0 ? 0u : 1u);
                    if (two) {
                        const uint64_t dbh1 = desc0 + (uint64_t)s1 * STAGE_UNITS;
                        umma_kslice_nocommit_elect(d_tmem, a_hi + 64u, a_hi + 96u, dbh1, dbh1 + LO_UNITS, idesc, 1u);
                    }
                    umma_commit_elect(&b_empty[s]);
                    if (two) umma_commit_elect(&b_empty[s1]);
                }
                if (two) { s = s1; ph = ph1; }
                if (++s == NRB) { s = 0; ph ^= 1u; }
            }
            umma_commit_elect(&acc_full[buf]);
        }
    } else {
        // ---- split + epilogue warps: two groups of four (one warp per TMEM lane quarter), group g takes slices j = g (mod 2)
        constexpr int NBF = (Cfg::B_BYTES / 16) / 128;
        const int q = warp & 3, grp = warp >> 2, gt = q * 32 + lane, row = gt;
        const int chalf = warp >> 2;                                          // which 32 of the 64 tile columns this thread owns
        float* C = p.C + zb * p.sCb + zh * p.sCh;
        const int m = m0 + row;
        float* Fz = SMX ? ap.F + (long long)blockIdx.z * ap.ngrp * p.M : nullptr;
        float mu = -INFINITY, sigma = 0.f;                                   // SMX: running maximum (raw score units) and sum of this thread's groups
        int next_tile = 0;
        const bool direct_store = ap.direct_store != 0;
        auto epilogue = [&](int nt) {
            const int buf = nt & 1;
            mbar_wait(&acc_full[buf], (uint32_t)(nt >> 1) & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            uint32_t r[32];
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BN + chalf * 32);
            tmem_ld16(taddr, r);
            tmem_ld16(taddr + 16u, r + 16);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[buf]);            // the MMAs of tile nt+2 may overwrite this buffer
            const int n = nt * BN + chalf * 32;
            const int nvalid = p.N - n;                               // columns [0, nvalid) of this group exist
            float v[32];
            if (SMX) {
                float tmax = -INFINITY;
#pragma unroll
                for (int jj = 0; jj < 32; ++jj)
                    if (jj < nvalid) tmax = fmaxf(tmax, __uint_as_float(r[jj]));
                if (tmax > mu) {
                    sigma *= ex2_approx((mu - tmax) * ap.c);
                    mu = tmax;
                }
                const float off = -mu * ap.c;
#pragma unroll
                for (int jj = 0; jj < 32; ++jj) {
                    v[jj] = ex2_approx(fmaf(__uint_as_float(r[jj]), ap.c, off));
                    if (jj < nvalid) sigma += v[jj];
                }
                const int g = 2 * nt + chalf;
                if (m < p.M && g < ap.ngrp) Fz[(long long)g * p.M + m] = mu;
            } else {
#pragma unroll
                for (int jj = 0; jj < 32; ++jj) v[jj] = __uint_as_float(r[jj]) * p.alpha;
            }
            if (nvalid > 0 && !direct_store) {
                // Coalesced store through a warp-private staging tile.  Thread = row: stored directly, every float4 of a warp lands in a different
                // 128-byte line (32 lines per instruction, 8 instructions per line).  Staged: the warp's 32 rows x 32 columns go to ITS 4 KB of the
                // raw-A ring (rows [32 q, 32 q + 32) of stage grp + 2: only this warp ever reads them, its own conversions are done — the epilogue
                // runs after them in program order — and no TMA refills the ring: NRA == NTA), 16-byte chunks XOR-swizzled by the row so that both
                // the row-wise writes and the 4-rows-per-instruction reads are conflict-free; then 8 instructions store 4 whole lines each.
                const uint32_t stg = smem_u32(smemA + (size_t)(grp + 2) * Cfg::A_BYTES) + (uint32_t)(q * 32) * 128u;
#pragma unroll
                for (int c = 0; c < 8; ++c)
                    sts128(stg + (uint32_t)lane * 128u + (uint32_t)((c ^ (lane & 7)) << 4), make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]));
                __syncwarp();
                const int c = lane & 7;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int rr = i * 4 + (lane >> 3);
                    const float4 t = lds128(stg + (uint32_t)rr * 128u + (uint32_t)((c ^ (rr & 7)) << 4));
                    const int mm = m0 + q * 32 + rr, col = 4 * c;
                    if (mm < p.M && col < nvalid) {
                        float* dst = C + (long long)mm * p.ldc + n + col;
                        if (col + 3 < nvalid && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
                            *reinterpret_cast<float4*>(dst) = t;
                        } else {
                            const float tv[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
                            for (int e = 0; e < 4; ++e)
                                if (col + e < nvalid) dst[e] = tv[e];
                        }
                    }
                }
                __syncwarp();                                                       // the next tile's staging overwrites these rows
            } else if (m < p.M && nvalid > 0) {
                float* dst = C + (long long)m * p.ldc + n;
                const bool vec = ((reinterpret_cast<uintptr_t>(dst) & 15) == 0);
#pragma unroll
                for (int jj = 0; jj < 32; jj += 4) {
                    if (vec && jj + 3 < nvalid) {
                        *reinterpret_cast<float4*>(dst + jj) = make_float4(v[jj], v[jj + 1], v[jj + 2], v[jj + 3]);
                    } else {
#pragma unroll
                        for (int e = 0; e < 4; ++e)
                            if (jj + e < nvalid) dst[jj + e] = v[jj + e];
                    }
                }
            }
        };
        for (int j = grp; j < (PRE ? nkb : nj); j += NG) {
            if (j < nkb) {
                // ---- first sweep only: A slice kb = j -> tf32 hi / lo -> its permanent TMEM slot
                const int sa = j % NRA;
                mbar_wait(&a_full[sa], (uint32_t)(j / NRA) & 1u);
                if (ap.f16) split_a_slice_to_tmem_f16(smem_u32(smemA + (size_t)sa * Cfg::A_BYTES) + (uint32_t)row * 128u, row,
                                                      tmem_a0 + ((uint32_t)(q * 32) << 16) + (uint32_t)(j * 64), ap.sa);
                else split_a_slice_to_tmem(smem_u32(smemA + (size_t)sa * Cfg::A_BYTES) + (uint32_t)row * 128u, row,
                                           tmem_a0 + ((uint32_t)(q * 32) << 16) + (uint32_t)(j * 64), 1.f);
                __syncwarp();
                if (lane == 0) { mbar_arrive(&a_empty[sa]); mbar_arrive(&ta_ready[j]); }
            }
            if (!PRE) {
                // ---- W slice: hi in place + lo copy
                const int sb = j % NRB;
                mbar_wait(&b_full[sb], (uint32_t)(j / NRB) & 1u);
                const uint32_t b_addr = smem_u32(smemB + (size_t)sb * 2 * Cfg::B_BYTES);
                float4 vb[NBF];
#pragma unroll
                for (int e = 0; e < NBF; ++e) vb[e] = lds128(b_addr + (uint32_t)(gt + e * 128) * 16u);
#pragma unroll
                for (int e = 0; e < NBF; ++e) {
                    const uint32_t a = b_addr + (uint32_t)(gt + e * 128) * 16u;
                    float4 h, l;
                    h.x = tf32_rna(vb[e].x); h.y = tf32_rna(vb[e].y); h.z = tf32_rna(vb[e].z); h.w = tf32_rna(vb[e].w);
                    l.x = vb[e].x - h.x; l.y = vb[e].y - h.y; l.z = vb[e].z - h.z; l.w = vb[e].w - h.w;
                    sts128(a, h);
                    sts128(a + Cfg::B_BYTES, l);
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(&b_ready[sb]);
                // tile t is complete once W slice (t+1)*nkb - 1 has been multiplied; trail it by one slice
                while (next_tile < NT && j >= (next_tile + 1) * nkb) epilogue(next_tile++);
            }
        }
        while (next_tile < NT) epilogue(next_tile++);
        if (SMX) {
            // ---- merge the two column halves of every row, then turn the stored running maxima into the final factors
            float* xch = reinterpret_cast<float*>(smemA);                     // the raw-A ring is idle after the first sweep
            xch[chalf * 256 + row] = mu;
            xch[chalf * 256 + 128 + row] = sigma;
            asm volatile("bar.sync 1, 256;" ::: "memory");
            const float mu_p = xch[(chalf ^ 1) * 256 + row], sg_p = xch[(chalf ^ 1) * 256 + 128 + row];
            const float mx = fmaxf(mu, mu_p);
            const float l = sigma * ex2_approx((mu - mx) * ap.c) + sg_p * ex2_approx((mu_p - mx) * ap.c);
            const float inv_l = 1.f / l;
            if (m < p.M) {
                for (int g = chalf; g < ap.ngrp; g += 2) {
                    float* f = Fz + (long long)g * p.M + m;
                    *f = ex2_approx((*f - mx) * ap.c) * inv_l;
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == MMA_WARP) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(Cfg::TMEM_COLS) : "memory");
    }
}

// ---- O = (F * E) V  (see the block comment above): one CTA = 128 rows x all (<= 192) columns of one (clip, head)
struct PvCfg {
    static constexpr int BNMAX = 192, NRA = 4, NRB = 3, NTA = 5, NG = 2;
    static constexpr int THREADS = (4 * NG + 2) * 32;
    static constexpr int A_BYTES = TC_BM * 128, B_BYTES = BNMAX * 128;
    static constexpr int ACC_COLS = BNMAX, TMEM_COLS = 512;
    static constexpr int NBAR = 2 * NRA + 2 * NRB + 2 * NTA + 1;
    static constexpr size_t SMEM = (size_t)NRA * A_BYTES + (size_t)NRB * 2 * B_BYTES + 1024 + 8 * NBAR + 64;
    static_assert(ACC_COLS + NTA * 64 <= 512, "TMEM budget");
};

__global__ void __launch_bounds__(PvCfg::THREADS, 1)
tc_pv_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapW, const __grid_constant__ CUtensorMap mapWlo,
             const TcParams p, const AttnParams ap, const int bn) {
    using Cfg = PvCfg;
    constexpr int NRA = Cfg::NRA, NRB = Cfg::NRB, NTA = Cfg::NTA, NG = Cfg::NG;
    constexpr int PRODUCER_WARP = 4 * NG, MMA_WARP = 4 * NG + 1;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    unsigned char* smemA = smem;
    unsigned char* smemB = smem + (size_t)NRA * Cfg::A_BYTES;
    uint64_t* a_full = reinterpret_cast<uint64_t*>(smemB + (size_t)NRB * 2 * Cfg::B_BYTES);
    uint64_t* a_empty = a_full + NRA;
    uint64_t* b_full = a_empty + NRA;
    uint64_t* b_empty = b_full + NRB;
    uint64_t* ta_ready = b_empty + NRB;
    uint64_t* ta_empty = ta_ready + NTA;
    uint64_t* acc_full = ta_empty + NTA;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int zb = blockIdx.z / p.nh, zh = blockIdx.z % p.nh;
    const int m0 = blockIdx.y * TC_BM;
    const int nkb = (p.seg[0].k_len + TC_BK - 1) / TC_BK;

    if (tid == 0) {
        for (int s = 0; s < NRA; ++s) { mbar_init(&a_full[s], 1); mbar_init(&a_empty[s], 4); }
        for (int s = 0; s < NRB; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], 1); }
        for (int s = 0; s < NTA; ++s) { mbar_init(&ta_ready[s], 4); mbar_init(&ta_empty[s], 1); }
        mbar_init(acc_full, 1);
        mbar_fence_init();
    }
    if (warp == MMA_WARP) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(Cfg::TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t tmem_a0 = tmem_base + (uint32_t)Cfg::ACC_COLS;

    if (warp == PRODUCER_WARP) {
        if (lane == 0) {
            prefetch_tmap(&mapA);
            for (int i = 0; i < nkb; ++i) {
                const int s = i % NRA;
                mbar_wait(&a_empty[s], ((uint32_t)(i / NRA) & 1u) ^ 1u);
                mbar_expect_tx(&a_full[s], Cfg::A_BYTES);
                tma_load_4d(smemA + (size_t)s * Cfg::A_BYTES, &mapA, &a_full[s], i * TC_BK, m0, zh * p.a_mul_h, zb * p.a_mul_b);
            }
        } else if (lane == 1) {
            prefetch_tmap(&mapW);
            prefetch_tmap(&mapWlo);
            const uint32_t bytes = (uint32_t)bn * 128u;
            for (int i = 0; i < nkb; ++i) {
                const int s = i % NRB;
                mbar_wait(&b_empty[s], ((uint32_t)(i / NRB) & 1u) ^ 1u);
                mbar_expect_tx(&b_full[s], ap.f16 ? bytes : 2 * bytes);
                unsigned char* dst = smemB + (size_t)s * 2 * Cfg::B_BYTES;
                tma_load_4d(dst, &mapW, &b_full[s], i * TC_BK, 0, zh * p.w_mul_h, zb * p.w_mul_b);
                if (!ap.f16) tma_load_4d(dst + Cfg::B_BYTES, &mapWlo, &b_full[s], i * TC_BK, 0, zh * p.w_mul_h, zb * p.w_mul_b);
            }
        }
    } else if (warp == MMA_WARP) {
        // running ring counters, descriptors advanced by addition
        const uint32_t idesc = ap.f16 ? make_idesc_f16(TC_BM, bn) : make_idesc_tf32(TC_BM, bn);
        const uint64_t desc0 = make_smem_desc_sw128(smem_u32(smemB));
        constexpr uint64_t STAGE_UNITS = (uint64_t)(2 * Cfg::B_BYTES) >> 4, LO_UNITS = (uint64_t)Cfg::B_BYTES >> 4;
        int sb = 0, sa = 0;
        uint32_t pb = 0, pa = 0;
        for (int i = 0; i < nkb; ++i) {            // (waiting for two slices per iteration was measured slower here: 34.6 -> 42.5 us)
            mbar_wait(&b_full[sb], pb);
            mbar_wait(&ta_ready[sa], pa);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t a_hi = tmem_a0 + (uint32_t)(sa * 64);
            const uint64_t dbh = desc0 + (uint64_t)sb * STAGE_UNITS;
            if (ap.f16) umma_kslice_f16_elect(tmem_base, a_hi, dbh, idesc, i == 0 ? 0u : 1u, smem_u32(&b_empty[sb]), smem_u32(&ta_empty[sa]));
            else umma_kslice_elect(tmem_base, a_hi, a_hi + 32u, dbh, dbh + LO_UNITS, idesc, i == 0 ? 0u : 1u, smem_u32(&b_empty[sb]), smem_u32(&ta_empty[sa]));
            if (++sb == NRB) { sb = 0; pb ^= 1u; }
            if (++sa == NTA) { sa = 0; pa ^= 1u; }
        }
        umma_commit_elect(acc_full);
    } else {
        const int q = warp & 3, grp = warp >> 2, row = q * 32 + lane;
        const int m = m0 + row;
        const float* Fz = ap.Fc ? ap.Fc + (long long)blockIdx.z * ap.ngrp * p.M : nullptr;
        for (int i = grp; i < nkb; i += NG) {
            const int sr = i % NRA, sa = i % NTA;
            const float f = Fz ? ((m < p.M && i < ap.ngrp) ? __ldg(Fz + (long long)i * p.M + m) : 0.f) : 1.f;
            mbar_wait(&a_full[sr], (uint32_t)(i / NRA) & 1u);
            mbar_wait(&ta_empty[sa], ((uint32_t)(i / NTA) & 1u) ^ 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (ap.f16) split_a_slice_to_tmem_f16(smem_u32(smemA + (size_t)sr * Cfg::A_BYTES) + (uint32_t)row * 128u, row,
                                                  tmem_a0 + ((uint32_t)(q * 32) << 16) + (uint32_t)(sa * 64), f * ap.sa);
            else split_a_slice_to_tmem(smem_u32(smemA + (size_t)sr * Cfg::A_BYTES) + (uint32_t)row * 128u, row,
                                       tmem_a0 + ((uint32_t)(q * 32) << 16) + (uint32_t)(sa * 64), f);
            __syncwarp();
            if (lane == 0) { mbar_arrive(&a_empty[sr]); mbar_arrive(&ta_ready[sa]); }
        }
        // ---- epilogue: thread (row, column half) -> global, masked to the N real columns
        mbar_wait(acc_full, 0u);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int half = bn >> 1, c0 = grp * half;
        float* dst = p.C + zb * p.sCb + zh * p.sCh + (long long)m * p.ldc;
        const bool vec = ((reinterpret_cast<uintptr_t>(dst) & 15) == 0);
        uint32_t* irow = ap.img ? ap.img + ((long long)zb * p.M + m) * ap.img_ld : nullptr;
        if (irow && m < p.M && zh == p.nh - 1 && grp == 0) {
            // the K padding of the Wo operand (columns [nh * sCh, img_ld) of the row) belongs to nobody's head: zeros, like the pack pass wrote
            for (int gc = p.nh * (int)p.sCh; gc < (int)ap.img_ld; gc += 4) {
                uint32_t* d = irow + f16x3_word(gc);
                *reinterpret_cast<uint2*>(d) = make_uint2(0u, 0u);
                *reinterpret_cast<uint2*>(d + 16) = make_uint2(0u, 0u);
            }
        }
        if (!ap.direct_store) {
            // Coalesced epilogue through a warp-private staging tile (every MMA has completed — acc_full — so the W ring is idle; see the score
            // kernel's epilogue for why): phase 1, thread = row, stages its `half` columns (scaled, pad columns n >= N as zeros) with a pitch of
            // half + 4 words (conflict-free 16-byte row writes for half = 88); phase 2, consecutive lanes take consecutive 4-column chunks of a
            // row: fp32 mode stores whole float4s of C (a row's 352 bytes leave in ~3 lines instead of 22 scattered pieces), image mode converts
            // the chunk to 2 hi + 2 lo words of the Wo operand image (8 lanes = the 64-byte hi half of a K slice, and its lo half).
            const int pitch = half + 4, nchunk = half >> 2;
            const uint32_t stg = smem_u32(smemB) + (uint32_t)warp * (uint32_t)(32 * (Cfg::BNMAX / 2 + 4) * 4);
            for (int cc = 0; cc < half; cc += 8) {
                uint32_t r[8];
                tmem_ld8(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(c0 + cc), r);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                float v[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) v[e] = (c0 + cc + e < p.N) ? __uint_as_float(r[e]) * p.alpha : 0.f;
                const uint32_t a = stg + (uint32_t)(lane * pitch + cc) * 4u;
                sts128(a, make_float4(v[0], v[1], v[2], v[3]));
                sts128(a + 16u, make_float4(v[4], v[5], v[6], v[7]));
            }
            __syncwarp();
            const int slot = min(bn, (int)p.sCh);                                  // image mode: columns of this head's slot in the row
            float* Cb = p.C + zb * p.sCb + zh * p.sCh;
            for (int f = lane; f < 32 * nchunk; f += 32) {
                const int rr = f / nchunk, ch = f - rr * nchunk;
                const float4 t = lds128(stg + (uint32_t)(rr * pitch + ch * 4) * 4u);
                const int mm = m0 + q * 32 + rr, n = c0 + ch * 4;
                if (mm >= p.M) continue;
                if (ap.img) {
                    if (n >= slot) continue;                                       // columns past the slot belong to the next head's CTA
                    uint32_t hi[2], lo[2];
                    f16x3_split_pair(t.x, t.y, ap.img_scale, hi[0], lo[0]);
                    f16x3_split_pair(t.z, t.w, ap.img_scale, hi[1], lo[1]);
                    uint32_t* d = ap.img + ((long long)zb * p.M + mm) * ap.img_ld + f16x3_word(zh * (int)p.sCh + n);
                    *reinterpret_cast<uint2*>(d) = make_uint2(hi[0], hi[1]);
                    *reinterpret_cast<uint2*>(d + 16) = make_uint2(lo[0], lo[1]);
                } else if (n < p.N) {
                    float* d = Cb + (long long)mm * p.ldc + n;
                    if (n + 3 < p.N && (reinterpret_cast<uintptr_t>(d) & 15) == 0) {
                        *reinterpret_cast<float4*>(d) = t;
                    } else {
                        const float tv[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
                        for (int e = 0; e < 4; ++e)
                            if (n + e < p.N) d[e] = tv[e];
                    }
                }
            }
        } else
        for (int cc = 0; cc < half; cc += 8) {
            uint32_t r[8];
            tmem_ld8(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(c0 + cc), r);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            if (irow) {
                // 2 x 4 columns = 2 x (2 hi words + 2 lo words): a 4-column group never straddles a 32-wide K slice of the Wo operand (the head
                // stride sCh and the column offsets are multiples of 4), 8-byte stores
                if (m < p.M) {
#pragma unroll
                    for (int g4 = 0; g4 < 8; g4 += 4) {
                        const int n = c0 + cc + g4, gc = zh * (int)p.sCh + n;
                        if (n >= bn || n >= (int)p.sCh) continue;                       // columns past the head's slot belong to the next head's CTA
                        uint32_t hi[2], lo[2];
#pragma unroll
                        for (int pr = 0; pr < 2; ++pr) {
                            const float v0 = (n + 2 * pr < p.N) ? __uint_as_float(r[g4 + 2 * pr]) * p.alpha : 0.f;
                            const float v1 = (n + 2 * pr + 1 < p.N) ? __uint_as_float(r[g4 + 2 * pr + 1]) * p.alpha : 0.f;
                            f16x3_split_pair(v0, v1, ap.img_scale, hi[pr], lo[pr]);
                        }
                        uint32_t* d = irow + f16x3_word(gc);
                        *reinterpret_cast<uint2*>(d) = make_uint2(hi[0], hi[1]);
                        *reinterpret_cast<uint2*>(d + 16) = make_uint2(lo[0], lo[1]);
                    }
                }
                continue;
            }
            if (m < p.M) {
#pragma unroll
                for (int jj = 0; jj < 8; jj += 4) {
                    const int n = c0 + cc + jj;
                    if (vec && n + 3 < p.N) {
                        *reinterpret_cast<float4*>(dst + n) = make_float4(__uint_as_float(r[jj]) * p.alpha, __uint_as_float(r[jj + 1]) * p.alpha,
                                                                          __uint_as_float(r[jj + 2]) * p.alpha, __uint_as_float(r[jj + 3]) * p.alpha);
                    } else {
#pragma unroll
                        for (int e = 0; e < 4; ++e)
                            if (n + e < p.N) dst[n + e] = __uint_as_float(r[jj + e]) * p.alpha;
                    }
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == MMA_WARP) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(Cfg::TMEM_COLS) : "memory");
    }
}

// ------------------------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// rank-4 fp32 tensor map {K, rows, heads, batch}; box {32, box_rows, 1, 1}; 128B swizzle; OOB -> 0.
// An axis with stride 0 (operand shared across it) is encoded with extent 1; *mul tells the kernel to pass coordinate 0.
int make_map(CUtensorMap* map, const float* base, long long K, long long rows, long long ld, long long nh, long long s_h, long long nb,
             long long s_b, int box_rows, int* mul_h, int* mul_b) {
    EncodeTiledFn enc = get_encode();
    GVD_REQUIRE(enc, "tcgemm: cuTensorMapEncodeTiled is unavailable in this driver");
    GVD_REQUIRE(((uintptr_t)base & 15) == 0 && ld % 4 == 0 && s_h % 4 == 0 && s_b % 4 == 0, "tcgemm: operand not 16-byte aligned");
    const bool use_h = nh > 1 && s_h != 0, use_b = nb > 1 && s_b != 0;
    *mul_h = use_h ? 1 : 0;
    *mul_b = use_b ? 1 : 0;
    cuuint64_t dims[4] = {(cuuint64_t)K, (cuuint64_t)rows, (cuuint64_t)(use_h ? nh : 1), (cuuint64_t)(use_b ? nb : 1)};
    cuuint64_t strides[3] = {(cuuint64_t)ld * 4, (cuuint64_t)(use_h ? s_h : ld * rows) * 4, (cuuint64_t)(use_b ? s_b : ld * rows) * 4};
    cuuint32_t box[4] = {TC_BK, (cuuint32_t)box_rows, 1, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    GVD_REQUIRE(r == CUDA_SUCCESS, "tcgemm: cuTensorMapEncodeTiled failed (%d) K=%lld rows=%lld ld=%lld", (int)r, K, rows, ld);
    return 0;
}


// =====================================================================================================
// f16ss_kernel — NT GEMM with BOTH operands pre-split into the fp16x3 operand image (gvd_common.cuh): per row and 32-wide K slice 64 B
// of fp16 hi halves | 64 B of fp16 lo halves, i.e. exactly one SWIZZLE_128B row of a K-major tcgen05 operand.  TMA output feeds the MMA
// from shared memory for A and B alike: no conversion warps, no tensor-memory operand slots, a third of the shared-memory traffic per
// K slice of tc2_gemm_kernel (which is bound by it).  Constant weights are packed once (gvd_model_finalize); activations are packed by the
// kernel that produces them (decode step) or by one element-wise pass (gvd_pack_f16x3, prologue: 4 B read + 4 B written per element).
//   warp 0: TMA producer (A and B tile of a stage on one barrier)   warp 1: MMA issuer (6 kind::f16 SS MMAs per slice: lo.hi, hi.lo,
//   hi.hi per 16-wide K step)   warps 2..: accumulator drain (every 2 slices into fp32 registers: the tensor core's accumulate
//   truncates) and the epilogue.
// EPI 0: C[m, n] = act(acc + bias[n]) through a shared-memory staged, coalesced store (prologue GEMMs: M side = activation rows).
// EPI 3: split-K partial, stored transposed part[z][n][m] (decode-step products: M side = weight rows, N = the whole batch, K split over
//        blockIdx.z; the coalesced reductions of gvd_skinny.cu finish the job).
// =====================================================================================================
template <int BN, int EPI> struct SsCfg {
    static constexpr int NST = BN > 128 ? 4 : 6;                     // stages of (A 16 KB + B BN*128 B)
    static constexpr int BUF = BN > 128 ? 256 : 128;                 // TMEM column stride of the two accumulator buffers
    static constexpr int A_BYTES = TC_BM * 128, B_BYTES = BN * 128;
    static constexpr int STAGE = A_BYTES + ((B_BYTES + 1023) / 1024) * 1024;   // B tile starts 1024-aligned (swizzle atom)
    static constexpr int DRAIN_WARPS = (EPI == 3) ? 4 : 8;           // EPI 3: one thread owns a whole weight row (BN <= 128 columns)
    static constexpr int ACC = (EPI == 3) ? BN : BN / 2;
    static constexpr int THREADS = (2 + DRAIN_WARPS) * 32;
    static constexpr int CHUNK = 2;
    static constexpr int TMEM_COLS = 2 * BUF;                        // two accumulator buffers
    static constexpr size_t SMEM = (size_t)NST * STAGE + 1024 + 8 * (2 * NST + 4) + 64;
    static_assert(EPI == 3 || (size_t)NST * STAGE >= (size_t)TC_BM * (BN + 4) * 4, "the epilogue stages the C tile in the pipeline buffers");
};
struct SsParams {
    float* C; long long ldc, plane;        // EPI 0: C[m * ldc + n];  EPI 3: C[z * plane + n * ldc + m]
    int M, N, nslices;                     // rows of the A / B side, 32-wide K slices per CTA
    float oscale;
    const float* bias; const float* scale2; const float* shift2; int act;
    uint32_t* img; long long ld_img; float img_scale;   // persistent kernel: also store the fp16x3 operand image of the (activated) output: the next
                                                        // GEMM streams it directly; C may then be null (output consumed by that GEMM only)
    // persistent kernel, Q|K|V projection of the region encoder (qkv_hp > 0; N = 3 * qkv_hp head-padded columns): columns [0, HP) = Q -> fp32 C;
    // [HP, 2HP) = K -> per-head fp16x3 image k_img[(row * nh + h) * KH + word(c)] (the W operand of the score kernel); [2HP, 3HP) = V -> image
    // of V^T per clip vt_img[(b * HP + c) * Rp + word(r)] (the W operand of the P.V kernel).  Replaces pack_heads / transpose_pack passes.
    int qkv_hp, qkv_hs, qkv_kh, qkv_nh, qkv_R, qkv_Rp;
    uint32_t *k_img, *vt_img;
    float qkv_sk, qkv_sv;
    int chunk;                             // persistent kernel: K slices per TMEM accumulation chunk (the other kernels: SsCfg::CHUNK)
};
template <int BN, int EPI>
__global__ void __launch_bounds__(SsCfg<BN, EPI>::THREADS, 1)
f16ss_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const SsParams p) {
    using Cfg = SsCfg<BN, EPI>;
    constexpr int NST = Cfg::NST, ACC = Cfg::ACC;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)NST * Cfg::STAGE);
    uint64_t* empty = full + NST;
    uint64_t* acc_full = empty + NST;       // [2]
    uint64_t* acc_empty = acc_full + 2;     // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n0 = blockIdx.x * BN, m0 = blockIdx.y * TC_BM, split = blockIdx.z;
    const int nkb = p.nslices, nchunks = (nkb + Cfg::CHUNK - 1) / Cfg::CHUNK;
    if (tid == 0) {
        for (int s = 0; s < NST; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], Cfg::DRAIN_WARPS); }
        mbar_fence_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(Cfg::TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    if (warp == 0) {
        if (lane == 0) {
            prefetch_tmap(&mapA);
            prefetch_tmap(&mapB);
            for (int i = 0; i < nkb; ++i) {
                const int s = i % NST;
                mbar_wait(&empty[s], ((uint32_t)(i / NST) & 1u) ^ 1u);
                unsigned char* st = smem + (size_t)s * Cfg::STAGE;
                mbar_expect_tx(&full[s], Cfg::A_BYTES + Cfg::B_BYTES);
                const int k = (split * nkb + i) * TC_BK;
                tma_load_4d(st, &mapA, &full[s], k, m0, 0, 0);
                tma_load_4d(st + Cfg::A_BYTES, &mapB, &full[s], k, n0, 0, 0);
            }
        }
    } else if (warp == 1) {
        const uint32_t idesc = make_idesc_f16(TC_BM, BN);
        for (int i = 0; i < nkb; ++i) {
            const int s = i % NST;
            const int c = i / Cfg::CHUNK, buf = c & 1;
            const bool first = (i % Cfg::CHUNK) == 0;
            if (first) mbar_wait(&acc_empty[buf], ((uint32_t)(c >> 1) & 1u) ^ 1u);
            mbar_wait(&full[s], (uint32_t)(i / NST) & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t a_addr = smem_u32(smem + (size_t)s * Cfg::STAGE);
            const uint64_t da = make_smem_desc_sw128(a_addr), db = make_smem_desc_sw128(a_addr + Cfg::A_BYTES);
            const uint32_t d_tmem = tmem_base + (uint32_t)(buf * Cfg::BUF);
            // hi halves of K step j at byte 32 j of a row, lo halves at 64 + 32 j: descriptor start address += bytes >> 4
            asm volatile(
                "{\n\t"
                ".reg .pred e, p0, pt;\n\t"
                ".reg .b64 ah1, al0, al1, bh1, bl0, bl1;\n\t"
                "elect.sync _|e, 0xffffffff;\n\t"
                "setp.ne.b32 p0, %4, 0;\n\t"
                "setp.eq.b32 pt, 0, 0;\n\t"
                "add.u64 ah1, %1, 2;\n\t add.u64 al0, %1, 4;\n\t add.u64 al1, %1, 6;\n\t"
                "add.u64 bh1, %2, 2;\n\t add.u64 bl0, %2, 4;\n\t add.u64 bl1, %2, 6;\n\t"
                "@e tcgen05.mma.cta_group::1.kind::f16 [%0], al0, %2, %3, p0;\n\t"
                "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, bl0, %3, pt;\n\t"
                "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, pt;\n\t"
                "@e tcgen05.mma.cta_group::1.kind::f16 [%0], al1, bh1, %3, pt;\n\t"
                "@e tcgen05.mma.cta_group::1.kind::f16 [%0], ah1, bl1, %3, pt;\n\t"
                "@e tcgen05.mma.cta_group::1.kind::f16 [%0], ah1, bh1, %3, pt;\n\t"
                "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%5];\n\t"
                "}\n" ::"r"(d_tmem), "l"(da), "l"(db), "r"(idesc), "r"(first ? 0u : 1u), "r"(smem_u32(&empty[s]))
                : "memory");
            if ((i % Cfg::CHUNK) == Cfg::CHUNK - 1 || i == nkb - 1) umma_commit_elect(&acc_full[buf]);
        }
    } else {
        const int dw = warp - 2;
        const int q = warp & 3;                                               // TMEM lane quarter this warp may access (warp id mod 4)
        const int cbeg = (EPI == 3) ? 0 : (dw >> 2) * ACC;                    // EPI 0: warps 2-5 drain columns [0, BN/2), warps 6-9 the rest
        float acc[ACC];
#pragma unroll
        for (int j = 0; j < ACC; ++j) acc[j] = 0.f;
        for (int c = 0; c < nchunks; ++c) {
            const int buf = c & 1;
            mbar_wait(&acc_full[buf], (uint32_t)(c >> 1) & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            // all tcgen05.ld of a batch are issued back to back and awaited ONCE: a wait after every 16 columns serialises ~4-7 TMEM round
            // trips per chunk and made the drain, not the MMAs, the pace of the whole pipeline
            constexpr int DB = ACC > 64 ? ((ACC / 16 + 1) / 2) * 16 : ACC;            // columns per batch (<= 64 registers in flight)
#pragma unroll
            for (int jb = 0; jb < ACC; jb += DB) {
                uint32_t r[DB];
#pragma unroll
                for (int j0 = 0; j0 < DB; j0 += 16)
                    if (jb + j0 < ACC) tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * Cfg::BUF + cbeg + jb + j0), r + j0);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int e = 0; e < DB; ++e)
                    if (jb + e < ACC) acc[jb + e] = fmaf(__uint_as_float(r[e]), p.oscale, acc[jb + e]);
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[buf]);
        }
        const int row = q * 32 + lane;
        const int m = m0 + row;
        if constexpr (EPI == 3) {
            if (m < p.M) {
                float* dst = p.C + (long long)split * p.plane + m;
#pragma unroll
                for (int j = 0; j < ACC; ++j)
                    if (j < p.N) dst[(long long)j * p.ldc] = acc[j];                // lanes = consecutive m: one 128-byte line per store
            }
        } else {
            // every MMA has completed (the last acc_full was awaited): the pipeline buffers are free to stage the C tile
            constexpr int LDS_ = BN + 4;
            float* Cs = reinterpret_cast<float*>(smem);
#pragma unroll
            for (int j = 0; j < ACC; j += 4) {
                const int n = n0 + cbeg + j;
                float v[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    float x = acc[j + e];
                    const int nn = n + e;
                    if (nn < p.N) {
                        if (p.bias) x += __ldg(p.bias + nn);
                        if (p.act >= GVD_ACT_RELU) x = fmaxf(x, 0.f);
                        if (p.act == GVD_ACT_RELU_AFFINE_RELU) x = fmaxf(fmaf(x, __ldg(p.scale2 + nn), __ldg(p.shift2 + nn)), 0.f);
                    }
                    v[e] = x;
                }
                *reinterpret_cast<float4*>(Cs + row * LDS_ + cbeg + j) = make_float4(v[0], v[1], v[2], v[3]);
            }
            asm volatile("bar.sync 2, %0;" ::"n"(Cfg::DRAIN_WARPS * 32) : "memory");
            constexpr int LANES_PER_ROW = BN / 4;
            constexpr int ROWS_PER_IT = (Cfg::DRAIN_WARPS * 32) / LANES_PER_ROW;
            const int dt = dw * 32 + lane;
            const int rsub = dt / LANES_PER_ROW, c4 = (dt % LANES_PER_ROW) * 4;
            const bool vec_ok = (p.ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.C) & 15) == 0);
#pragma unroll 4
            for (int r0 = 0; r0 < TC_BM; r0 += ROWS_PER_IT) {
                const int rr = r0 + rsub, mm = m0 + rr, n = n0 + c4;
                if (mm < p.M && n < p.N) {
                    const float4 v = *reinterpret_cast<const float4*>(Cs + rr * LDS_ + c4);
                    float* dst = p.C + (long long)mm * p.ldc + n;
                    if (vec_ok && n + 3 < p.N) {
                        *reinterpret_cast<float4*>(dst) = v;
                    } else {
                        const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                        for (int e = 0; e < 4; ++e)
                            if (n + e < p.N) dst[e] = vv[e];
                    }
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(Cfg::TMEM_COLS) : "memory");
    }
}

bool use_v1_static() { static const bool v = getenv("GVD_TC_V1") != nullptr; return v; }
// Cluster TMA-multicast of the activation slice for the skinny (BN = 32) launches.  Measured on the language-LSTM gate GEMM
// (B=100, K=3072, 128 CTAs): cluster 1 -> 60 us, 2 -> 75 us, 4 -> 100 us, 8 -> 250 us: the cluster-scope stage hand-off
// (remote mbarrier arrives from every peer before a stage can be refilled) costs far more than the saved L2 reads, so it
// is OFF by default (GVD_TC_CLUSTER=2|4|8 enables it for experiments).
int tc_cluster_size() { static const int v = getenv("GVD_TC_CLUSTER") ? atoi(getenv("GVD_TC_CLUSTER")) : 1; return v; }

// wide (N = 256) tiles for the big prologue GEMMs — experimental until measured on the device: backend bit 2 (gvd_set_backend(7))
// or GVD_TC_BN256=1
bool tc_bn256() {
    static const bool env = getenv("GVD_TC_BN256") != nullptr && atoi(getenv("GVD_TC_BN256")) != 0;
    return env || (gvd_backend() & 4) != 0;
}

int tc_debug_flags() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("GVD_TC_DEBUG"); v = e ? atoi(e) : 0; }
    return v;
}

// fp32 [N, K] (row pitch ldw) -> the W-operand image of the fp16x3 kernel: per row and 32-wide K slice 16 words of hi pairs then 16 words
// of lo pairs (k = 2p, 2p + 1 in word p), values scaled by GVD_F16_SW; K padded with zeros to a multiple of 32 (row pitch Kp words)
__global__ void pack_f16x3_kernel(const float* __restrict__ W, long long ldw, int N, int K, float sw, uint32_t* __restrict__ out, long long Kp) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;         // (n, slice, pair)
    const long long per_row = Kp / 2;
    if (idx >= (long long)N * per_row) return;
    const long long n = idx / per_row;
    const int r = (int)(idx % per_row), kb = r / 16, pr = r % 16, k = kb * 32 + 2 * pr;
    const float x0 = k < K ? W[n * ldw + k] * sw : 0.f, x1 = k + 1 < K ? W[n * ldw + k + 1] * sw : 0.f;
    const float a0 = tf32_rna(x0), a1 = tf32_rna(x1);
    out[n * Kp + kb * 32 + pr] = pack_h2(a0, a1);
    out[n * Kp + kb * 32 + 16 + pr] = pack_h2(x0 - a0, x1 - a1);
}

template <int BN>
int launch_tc(const CUtensorMap* mA, const CUtensorMap* mW, const TcParams& p_in, dim3 grid, cudaStream_t st) {
    using Cfg = TcCfg<BN>;
    TcParams p = p_in;
    p.dbg = tc_debug_flags();
    if (gvd_gemm_f16()) { p.sa = GVD_F16_SA; p.sw = GVD_F16_SW; p.oscale = 1.f / (GVD_F16_SA * GVD_F16_SW); }   // |activation| <= 16376, |weight| <= 255 after scaling
    else { p.sa = p.sw = 1.f; p.oscale = 0.f; p.wpre = 0; }
    static const int lag = getenv("GVD_TC_LAG") ? atoi(getenv("GVD_TC_LAG")) : TC_LAG;
    p.lag = lag;
    if (use_v1_static()) p.cs = 1;
    static const bool use_v1 = getenv("GVD_TC_V1") != nullptr;
    static bool attr_set = false;
    if (!attr_set) {
        if (use_v1) GVD_CHECK_CUDA(cudaFuncSetAttribute(tc_gemm_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM));
        GVD_CHECK_CUDA(cudaFuncSetAttribute(tc2_gemm_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Tc2Cfg<BN>::SMEM));
        attr_set = true;
    }
    if (p.oscale != 0.f && !use_v1 && p.cs == 1) {      // fp16x3 variant requested (gvd_gemm_f16_scope)
        static bool attr16 = false;
        if (!attr16) {
            GVD_CHECK_CUDA(cudaFuncSetAttribute(tc2_gemm_kernel<BN, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Tc2Cfg<BN, true>::SMEM));
            attr16 = true;
        }
        GVD_CHECK_CUDA(gvd_launch(tc2_gemm_kernel<BN, true>, grid, dim3(Tc2Cfg<BN, true>::THREADS), Tc2Cfg<BN, true>::SMEM, st, mA[0], mA[1], mA[2], mW[0],
                                  mW[1], mW[2], p));
        GVD_CHECK_LAUNCH();
        return 0;
    }
    if (use_v1) tc_gemm_kernel<BN><<<grid, TC_THREADS, Cfg::SMEM, st>>>(mA[0], mA[1], mA[2], mW[0], mW[1], mW[2], p);
    else if (p.cs > 1) {
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = grid; cfg.blockDim = dim3(Tc2Cfg<BN>::THREADS); cfg.dynamicSmemBytes = Tc2Cfg<BN>::SMEM; cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = p.cs; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        GVD_CHECK_CUDA(cudaLaunchKernelEx(&cfg, tc2_gemm_kernel<BN>, mA[0], mA[1], mA[2], mW[0], mW[1], mW[2], p));
    } else tc2_gemm_kernel<BN><<<grid, Tc2Cfg<BN>::THREADS, Tc2Cfg<BN>::SMEM, st>>>(mA[0], mA[1], mA[2], mW[0], mW[1], mW[2], p);
    GVD_CHECK_LAUNCH();
    return 0;
}

}  // namespace

// Short-K (K <= 192) batched product without bias / activation through the A-stationary kernel.
//   W_lo == nullptr : g.W is plain fp32 (split inside the kernel);  else g.W / W_lo are its tf32 hi / lo planes (same strides)
//   F    != nullptr : softmax-numerator epilogue, C = exp((s - mu_group) * smx_scale), F[batch][ceil(N/32)][M] = group factors
// f16: g.W is the fp16x3 image of the streamed operand (K rounded up to 32 words per (row, head)), scale GVD_ATT_SK; the A operand is scaled
// by GVD_ATT_SQ inside the kernel; both are undone through the softmax constant / alpha
#define GVD_ATT_SQ 4.f
#define GVD_ATT_SK 16.f
#define GVD_ATT_SP 1024.f
#define GVD_ATT_SV 16.f
static int launch_astat(const GemmArgs& g, const float* W_lo, float* F, float smx_scale, int batch, cudaStream_t stream, int f16 = 0) {
    GVD_REQUIRE(g.M > 0 && g.N > 0 && g.K > 0 && g.K <= AstatCfg::NTA * TC_BK && g.nh >= 1 && batch % g.nh == 0, "astat gemm: needs K <= %d",
                AstatCfg::NTA * TC_BK);
    GVD_REQUIRE(!g.bias && g.act == GVD_ACT_NONE, "astat gemm: no bias / activation epilogue");
    GVD_REQUIRE(g.K % 4 == 0 && g.lda % 4 == 0 && g.ldw % 4 == 0, "astat gemm: K/lda/ldw must be multiples of 4");
    GVD_REQUIRE(!F || W_lo || f16, "astat gemm: the softmax epilogue is built for pre-split operands");
    const int nb = batch / g.nh;
    CUtensorMap mA, mW, mWl;
    TcParams p{};
    AttnParams ap{};
    p.cs = 1;
    const int Kw = f16 ? (g.K + 31) / 32 * 32 : g.K;          // the image holds whole 32-wide slices
    GVD_TRY(make_map(&mA, g.A, g.K, g.M, g.lda, g.nh, g.sAh, nb, g.sAb, TC_BM, &p.a_mul_h, &p.a_mul_b));
    GVD_TRY(make_map(&mW, g.W, Kw, g.N, g.ldw, g.nh, g.sWh, nb, g.sWb, AstatCfg::BN, &p.w_mul_h, &p.w_mul_b));
    GVD_TRY(make_map(&mWl, (W_lo && !f16) ? W_lo : g.W, Kw, g.N, g.ldw, g.nh, g.sWh, nb, g.sWb, AstatCfg::BN, &p.w_mul_h, &p.w_mul_b));
    p.nseg = 1;
    p.seg[0] = TcSeg{g.K, 0, 0};
    p.M = g.M; p.N = g.N; p.nh = g.nh;
    p.C = g.C; p.ldc = g.ldc; p.sCb = g.sCb; p.sCh = g.sCh; p.alpha = g.alpha;
    ap.F = F; ap.ngrp = gvd_cdiv(g.N, 32); ap.c = smx_scale * 1.4426950408889634f;
    if (f16) { ap.f16 = 1; ap.sa = GVD_ATT_SQ; ap.c *= 1.f / (GVD_ATT_SQ * GVD_ATT_SK); p.alpha *= 1.f / (GVD_ATT_SQ * GVD_ATT_SK); }
    static const bool direct = getenv("GVD_ASTAT_DIRECT") != nullptr;
    ap.direct_store = direct ? 1 : 0;
    p.dbg = tc_debug_flags();
    static bool attr_set = false;
    if (!attr_set) {
        GVD_CHECK_CUDA(cudaFuncSetAttribute(tc_astat_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AstatCfg::SMEM));
        GVD_CHECK_CUDA(cudaFuncSetAttribute(tc_astat_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AstatCfg::SMEM));
        GVD_CHECK_CUDA(cudaFuncSetAttribute(tc_astat_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AstatCfg::SMEM));
        attr_set = true;
    }
    dim3 grid(1, gvd_cdiv(g.M, TC_BM), batch);
    if (F) tc_astat_kernel<true, true><<<grid, AstatCfg::THREADS, AstatCfg::SMEM, stream>>>(mA, mW, mWl, p, ap);
    else if (W_lo || f16) tc_astat_kernel<true, false><<<grid, AstatCfg::THREADS, AstatCfg::SMEM, stream>>>(mA, mW, mWl, p, ap);
    else tc_astat_kernel<false, false><<<grid, AstatCfg::THREADS, AstatCfg::SMEM, stream>>>(mA, mW, mWl, p, ap);
    GVD_CHECK_LAUNCH();
    return 0;
}
int gvd_gemm_nt_astat(const GemmArgs& g, int batch, cudaStream_t stream) { return launch_astat(g, nullptr, nullptr, 0.f, batch, stream); }
int gvd_attn_scores_tc(const GemmArgs& g, const float* W_lo, float* F, float smx_scale, int batch, cudaStream_t stream, int f16) {
    return launch_astat(g, W_lo, F, smx_scale, batch, stream, f16);
}
// O[z] = (F (.) A[z]) W[z]^T with W given as tf32 hi / lo planes, N <= 192 (one column tile), any K;  F [batch][ceil(K/32)][M] or null
int gvd_attn_pv_tc(const GemmArgs& g, const float* W_lo, const float* F, int batch, cudaStream_t stream, int f16, float* img, long long img_ld) {
    GVD_REQUIRE(g.M > 0 && g.N > 0 && g.N <= PvCfg::BNMAX && g.K > 0 && g.nh >= 1 && batch % g.nh == 0 && (W_lo || f16), "attn pv: needs N <= %d and pre-split W",
                PvCfg::BNMAX);
    GVD_REQUIRE(!g.bias && g.act == GVD_ACT_NONE, "attn pv: no bias / activation epilogue");
    GVD_REQUIRE(g.K % 4 == 0 && g.lda % 4 == 0 && g.ldw % 4 == 0, "attn pv: K/lda/ldw must be multiples of 4");
    const int nb = batch / g.nh;
    const int bn = ((g.N + 15) / 16) * 16;
    CUtensorMap mA, mW, mWl;
    TcParams p{};
    AttnParams ap{};
    p.cs = 1;
    GVD_TRY(make_map(&mA, g.A, g.K, g.M, g.lda, g.nh, g.sAh, nb, g.sAb, TC_BM, &p.a_mul_h, &p.a_mul_b));
    const int Kw = f16 ? (g.K + 31) / 32 * 32 : g.K;          // the image holds whole 32-wide slices
    GVD_TRY(make_map(&mW, g.W, Kw, g.N, g.ldw, g.nh, g.sWh, nb, g.sWb, bn, &p.w_mul_h, &p.w_mul_b));
    GVD_TRY(make_map(&mWl, f16 ? g.W : W_lo, Kw, g.N, g.ldw, g.nh, g.sWh, nb, g.sWb, bn, &p.w_mul_h, &p.w_mul_b));
    p.nseg = 1;
    p.seg[0] = TcSeg{g.K, 0, 0};
    p.M = g.M; p.N = g.N; p.nh = g.nh;
    p.C = g.C; p.ldc = g.ldc; p.sCb = g.sCb; p.sCh = g.sCh; p.alpha = g.alpha;
    ap.Fc = F; ap.ngrp = gvd_cdiv(g.K, 32);
    if (f16) { ap.f16 = 1; ap.sa = GVD_ATT_SP; p.alpha *= 1.f / (GVD_ATT_SP * GVD_ATT_SV); }
    static const bool direct = getenv("GVD_PV_DIRECT") != nullptr;              // thread-per-row stores instead of the staged epilogue (measurement aid)
    ap.direct_store = direct ? 1 : 0;
    static_assert(8 * 32 * (PvCfg::BNMAX / 2 + 4) * 4 <= PvCfg::NRB * 2 * PvCfg::B_BYTES, "the staging tiles of the 8 epilogue warps live in the W ring");
    if (img) {
        // every head owns sCh columns of the row (its N real ones + zero pads): together the heads must tile the image row exactly
        GVD_REQUIRE(g.sCh % 4 == 0 && (bn / 2) % 8 == 0 && g.N <= g.sCh && g.sCh <= bn && img_ld % 32 == 0 && img_ld >= (long long)g.nh * g.sCh &&
                    (reinterpret_cast<uintptr_t>(img) & 15) == 0, "attn pv: output image needs 4-column granularity of the head layout");
        ap.img = reinterpret_cast<uint32_t*>(img); ap.img_ld = img_ld; ap.img_scale = GVD_F16_SA;
    }
    static bool attr_set = false;
    if (!attr_set) {
        GVD_CHECK_CUDA(cudaFuncSetAttribute(tc_pv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PvCfg::SMEM));
        attr_set = true;
    }
    dim3 grid(1, gvd_cdiv(g.M, TC_BM), batch);
    tc_pv_kernel<<<grid, PvCfg::THREADS, PvCfg::SMEM, stream>>>(mA, mW, mWl, p, ap, bn);
    GVD_CHECK_LAUNCH();
    return 0;
}

int gvd_pack_f16x3(const float* W, long long ldw, int N, int K, float* out, long long Kp, cudaStream_t st, float scale) {
    GVD_REQUIRE(W && out && Kp % 32 == 0 && Kp >= K, "pack_f16x3: bad arguments");
    const long long n = (long long)N * (Kp / 2);
    pack_f16x3_kernel<<<(unsigned)gvd_cdiv(n, 256), 256, 0, st>>>(W, ldw, N, K, scale, reinterpret_cast<uint32_t*>(out), Kp);
    GVD_CHECK_LAUNCH();
    return 0;
}

// Epilogue store of one thread's output row segment: acc[0..ACC) = columns [ncol0, ncol0 + ACC) of row m (thread <-> row, lane <-> row within the
// warp).  Plain mode: bias / activation, fp32 C and / or the fp16x3 image of the output; Q|K|V mode (p.qkv_hp): Q as fp32, K as the per-head
// image, V as the image of V^T (lane pairs exchange rows with one shuffle per column).
template <int ACC>
__device__ __forceinline__ void ss_store_row(const SsParams& p, const float (&acc)[ACC], const int m, const int ncol0, const int lane, const bool vec_ok) {
    const int n0 = ncol0, cbeg = 0;
    if (p.qkv_hp) {
        // (warp-uniform branches: n is the same for every lane; lane <-> row, so lane ^ 1 holds the other row of an fp16 pair)
        const bool row_ok = m < p.M;
        const int HP = p.qkv_hp, HS = p.qkv_hs, KH = p.qkv_kh;
        const int bclip = m / p.qkv_R, r = m - bclip * p.qkv_R;
        float* dq = p.C + (long long)m * p.ldc;
        uint32_t* dk = p.k_img + (long long)m * p.qkv_nh * KH;
        uint32_t* dv = p.vt_img + (long long)bclip * HP * p.qkv_Rp + f16x3_word(r & ~1) + ((lane & 1) ? 16 : 0);
        const bool last_pair = (r | 1) == p.qkv_R - 1 && (p.qkv_R & 31) != 0;         // this row pair also zeroes the words of rows [R, Rp)
        const int vpad = 16 - ((p.qkv_R & 31) >> 1);
#pragma unroll
        for (int j = 0; j < ACC; j += 4) {
            const int n = n0 + cbeg + j;
            if (n >= p.N) break;
            const float v0 = acc[j], v1 = acc[j + 1], v2 = acc[j + 2], v3 = acc[j + 3];
            if (n < HP) {
                if (row_ok) *reinterpret_cast<float4*>(dq + n) = make_float4(v0, v1, v2, v3);
            } else if (n < 2 * HP) {
                const int kc = n - HP, h = kc / HS, c = kc - h * HS;
                if (row_ok) {
                    uint32_t h0, l0, h1, l1;
                    f16x3_split_pair(v0, v1, p.qkv_sk, h0, l0);
                    f16x3_split_pair(v2, v3, p.qkv_sk, h1, l1);
                    uint32_t* w = dk + h * KH + f16x3_word(c);
                    *reinterpret_cast<uint2*>(w) = make_uint2(h0, h1);
                    *reinterpret_cast<uint2*>(w + 16) = make_uint2(l0, l1);
                    if (c + 4 >= HS && HS < KH) {                        // last group of the head: zero the words of columns [HS, KH)
                        uint32_t* z = dk + h * KH + f16x3_word(HS);
                        for (int i = 0; i < (KH - HS) / 2; ++i) { z[i] = 0u; z[i + 16] = 0u; }
                    }
                }
            } else {
                const int c = n - 2 * HP;
                const float vv[4] = {v0, v1, v2, v3};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float o = __shfl_xor_sync(0xffffffffu, vv[e], 1);
                    uint32_t hi, lo;
                    if (lane & 1) f16x3_split_pair(o, vv[e], p.qkv_sv, hi, lo); else f16x3_split_pair(vv[e], o, p.qkv_sv, hi, lo);
                    if (row_ok) {
                        uint32_t* w = dv + (long long)(c + e) * p.qkv_Rp;      // even lane: hi word, odd lane: lo word of the pair (r & ~1, r | 1)
                        *w = (lane & 1) ? lo : hi;
                        if (last_pair) for (int i = 1; i <= vpad; ++i) w[i] = 0u;
                    }
                }
            }
        }
    } else if (m < p.M) {
        float* dst = p.C ? p.C + (long long)m * p.ldc + n0 + cbeg : nullptr;
        uint32_t* idst = p.img ? p.img + (long long)m * p.ld_img : nullptr;
#pragma unroll
        for (int j = 0; j < ACC; j += 4) {
            const int n = n0 + cbeg + j;
            float v[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                float x = acc[j + e];
                const int nn = n + e;
                if (nn < p.N) {
                    if (p.bias) x += __ldg(p.bias + nn);
                    if (p.act >= GVD_ACT_RELU) x = fmaxf(x, 0.f);
                    if (p.act == GVD_ACT_RELU_AFFINE_RELU) x = fmaxf(fmaf(x, __ldg(p.scale2 + nn), __ldg(p.shift2 + nn)), 0.f);
                } else {
                    x = 0.f;                                        // padding columns of the image are zeros
                }
                v[e] = x;
            }
            if (dst) {
                if (vec_ok && n + 3 < p.N) {
                    *reinterpret_cast<float4*>(dst + j) = make_float4(v[0], v[1], v[2], v[3]);
                } else {
#pragma unroll
                    for (int e = 0; e < 4; ++e)
                        if (n + e < p.N) dst[j + e] = v[e];
                }
            }
            if (idst && n < p.ld_img) {                             // 4 columns = 2 hi words + 2 lo words of one K slice of the next GEMM
                uint32_t h0, l0, h1, l1;
                f16x3_split_pair(v[0], v[1], p.img_scale, h0, l0);
                f16x3_split_pair(v[2], v[3], p.img_scale, h1, l1);
                uint32_t* w = idst + f16x3_word(n);
                *reinterpret_cast<uint2*>(w) = make_uint2(h0, h1);
                *reinterpret_cast<uint2*>(w + 16) = make_uint2(l0, l1);
            }
        }
    }
}

// Warp-private staging tiles of the persistent kernels' epilogue (ss_store_staged): one 32 x 32 fp32 tile per drain warp, placed after the
// barriers, outside the TMA ring (which keeps streaming the next tile while the epilogue runs).
constexpr int SS_STG_OFF = 256, SS_STG_BYTES = 8 * 32 * 128;
template <class Cfg> constexpr size_t ss_persist_smem() {
    static_assert(8 * (2 * Cfg::NST + 4) + 4 <= SS_STG_OFF && Cfg::DRAIN_WARPS * 32 * 128 <= SS_STG_BYTES, "staging tiles after the barriers");
    static_assert(Cfg::SMEM + SS_STG_OFF + SS_STG_BYTES <= 227 * 1024, "ring + staging exceed the 227 KB of shared memory a block may use");
    return Cfg::SMEM + SS_STG_OFF + SS_STG_BYTES;
}

// The plain-mode epilogue of ss_store_row (same values, same destinations) as coalesced stores: a drain warp owns rows [mrow0, mrow0 + 32) x
// columns [ncol0, ncol0 + ACC) (lane <-> row).  Per 32-column block, phase 1: each thread writes its row's accumulators into the warp's 4 KB
// staging tile `stg`, 16-byte chunks XOR-swizzled by the row so that the row-wise writes and the 4-rows-per-instruction reads are both free
// of bank conflicts; phase 2: lane = (row lane / 8 + 4 i, chunk lane % 8) applies bias / activation to its 4 columns and stores them, so 8
// consecutive lanes store one row's 128 bytes of C, or the 64-byte hi and lo halves of its image K slice (a 32-column block is exactly one
// K slice), instead of every store instruction touching 32 lines.
template <int ACC>
__device__ __forceinline__ void ss_store_staged(const SsParams& p, const float (&acc)[ACC], const int mrow0, const int ncol0, const int lane, const bool vec_ok,
                                                const uint32_t stg) {
    const int c = lane & 7;
#pragma unroll
    for (int jb = 0; jb < ACC; jb += 32) {
        const int nb = ncol0 + jb;                    // (warp-uniform)
        if (nb >= p.N) break;
#pragma unroll
        for (int j = 0; j < 32; j += 4)
            sts128(stg + (uint32_t)lane * 128u + (uint32_t)(((j >> 2) ^ (lane & 7)) << 4),
                   make_float4(acc[jb + j], acc[jb + j + 1], acc[jb + j + 2], acc[jb + j + 3]));
        __syncwarp();
        // a lane keeps its 4 columns for the whole block: bias / affine loaded once (the row-owning thread would load all 32)
        const int n = nb + 4 * c;
        float bv[4], sv[4], hv[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const bool ok = n + e < p.N;
            bv[e] = (ok && p.bias) ? __ldg(p.bias + n + e) : 0.f;
            sv[e] = (ok && p.act == GVD_ACT_RELU_AFFINE_RELU) ? __ldg(p.scale2 + n + e) : 0.f;
            hv[e] = (ok && p.act == GVD_ACT_RELU_AFFINE_RELU) ? __ldg(p.shift2 + n + e) : 0.f;
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int rr = i * 4 + (lane >> 3);
            const float4 t = lds128(stg + (uint32_t)rr * 128u + (uint32_t)((c ^ (rr & 7)) << 4));
            const int m = mrow0 + rr;
            if (m >= p.M) continue;
            float v[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {             // the operations of ss_store_row, element by element
                float x = v[e];
                if (n + e < p.N) {
                    if (p.bias) x += bv[e];
                    if (p.act >= GVD_ACT_RELU) x = fmaxf(x, 0.f);
                    if (p.act == GVD_ACT_RELU_AFFINE_RELU) x = fmaxf(fmaf(x, sv[e], hv[e]), 0.f);
                } else {
                    x = 0.f;                          // padding columns of the image are zeros
                }
                v[e] = x;
            }
            if (p.C) {
                float* d = p.C + (long long)m * p.ldc + n;
                if (vec_ok && n + 3 < p.N) {
                    *reinterpret_cast<float4*>(d) = make_float4(v[0], v[1], v[2], v[3]);
                } else {
#pragma unroll
                    for (int e = 0; e < 4; ++e)
                        if (n + e < p.N) d[e] = v[e];
                }
            }
            if (p.img && n < p.ld_img) {
                uint32_t h0, l0, h1, l1;
                f16x3_split_pair(v[0], v[1], p.img_scale, h0, l0);
                f16x3_split_pair(v[2], v[3], p.img_scale, h1, l1);
                uint32_t* w = p.img + (long long)m * p.ld_img + f16x3_word(n);
                *reinterpret_cast<uint2*>(w) = make_uint2(h0, h1);
                *reinterpret_cast<uint2*>(w + 16) = make_uint2(l0, l1);
            }
        }
        __syncwarp();                                 // the next block's phase 1 overwrites the tile
    }
}

// =====================================================================================================
// f16ss_persistent_kernel — f16ss_kernel (EPI 0) as a persistent tile loop: one CTA per SM walks the output tiles (N tiles of one M row
// block consecutively, so the A row block stays in L2), the TMA producer and the MMA issuer run ahead into the next tile while the drain
// warps finish the previous one: the per-CTA set-up (barriers, TMEM allocation, descriptor fetch), the pipeline fill and the epilogue
// no longer sit between two tiles' MMAs (they were ~30 % of a 32-slice tile).  Each drain thread owns one output row x BN/2 columns; the
// plain-mode epilogue (ss_store_staged) goes out through a warp-private staging tile outside the ring, so the ring keeps streaming and the
// stores leave as whole 128-byte lines.  ROWS: thread-per-row stores from registers (ss_store_row: the Q|K|V mode, and the reference the
// staged epilogue is tested against); a separate instantiation, because one kernel holding both epilogues spilled more and ran slower.
// =====================================================================================================
template <int BN, bool ROWS>
__global__ void __launch_bounds__(SsCfg<BN, 0>::THREADS, 1)
f16ss_persistent_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const SsParams p, int tiles_n, int tiles_total) {
    using Cfg = SsCfg<BN, 0>;
    constexpr int NST = Cfg::NST, ACC = Cfg::ACC;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)NST * Cfg::STAGE);
    uint64_t* empty = full + NST;
    uint64_t* acc_full = empty + NST;       // [2]
    uint64_t* acc_empty = acc_full + 2;     // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int CH = p.chunk;                  // K slices accumulated in TMEM between two fp32 register drains
    const int nkb = p.nslices, nchunks = (nkb + CH - 1) / CH;
    if (tid == 0) {
        for (int s = 0; s < NST; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], Cfg::DRAIN_WARPS); }
        mbar_fence_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(Cfg::TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    if (warp == 0) {
        if (lane == 0) {
            prefetch_tmap(&mapA);
            prefetch_tmap(&mapB);
            int i = 0;                                                        // global slice counter: the ring phases run across tiles
            for (int tile = blockIdx.x; tile < tiles_total; tile += gridDim.x) {
                const int m0 = (tile / tiles_n) * TC_BM, n0 = (tile % tiles_n) * BN;
                for (int kb = 0; kb < nkb; ++kb, ++i) {
                    const int s = i % NST;
                    mbar_wait(&empty[s], ((uint32_t)(i / NST) & 1u) ^ 1u);
                    unsigned char* st = smem + (size_t)s * Cfg::STAGE;
                    mbar_expect_tx(&full[s], Cfg::A_BYTES + Cfg::B_BYTES);
                    tma_load_4d(st, &mapA, &full[s], kb * TC_BK, m0, 0, 0);
                    tma_load_4d(st + Cfg::A_BYTES, &mapB, &full[s], kb * TC_BK, n0, 0, 0);
                }
            }
        }
    } else if (warp == 1) {
        const uint32_t idesc = make_idesc_f16(TC_BM, BN);
        int i = 0, c = 0;                                                     // global slice / chunk counters
        for (int tile = blockIdx.x; tile < tiles_total; tile += gridDim.x) {
            for (int kb = 0; kb < nkb; ++kb, ++i) {
                const int s = i % NST;
                const bool first = (kb % CH) == 0;
                const int buf = c & 1;
                if (first) mbar_wait(&acc_empty[buf], ((uint32_t)(c >> 1) & 1u) ^ 1u);
                mbar_wait(&full[s], (uint32_t)(i / NST) & 1u);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t a_addr = smem_u32(smem + (size_t)s * Cfg::STAGE);
                const uint64_t da = make_smem_desc_sw128(a_addr), db = make_smem_desc_sw128(a_addr + Cfg::A_BYTES);
                const uint32_t d_tmem = tmem_base + (uint32_t)(buf * Cfg::BUF);
                asm volatile(
                    "{\n\t"
                    ".reg .pred e, p0, pt;\n\t"
                    ".reg .b64 ah1, al0, al1, bh1, bl0, bl1;\n\t"
                    "elect.sync _|e, 0xffffffff;\n\t"
                    "setp.ne.b32 p0, %4, 0;\n\t"
                    "setp.eq.b32 pt, 0, 0;\n\t"
                    "add.u64 ah1, %1, 2;\n\t add.u64 al0, %1, 4;\n\t add.u64 al1, %1, 6;\n\t"
                    "add.u64 bh1, %2, 2;\n\t add.u64 bl0, %2, 4;\n\t add.u64 bl1, %2, 6;\n\t"
                    "@e tcgen05.mma.cta_group::1.kind::f16 [%0], al0, %2, %3, p0;\n\t"
                    "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, bl0, %3, pt;\n\t"
                    "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, pt;\n\t"
                    "@e tcgen05.mma.cta_group::1.kind::f16 [%0], al1, bh1, %3, pt;\n\t"
                    "@e tcgen05.mma.cta_group::1.kind::f16 [%0], ah1, bl1, %3, pt;\n\t"
                    "@e tcgen05.mma.cta_group::1.kind::f16 [%0], ah1, bh1, %3, pt;\n\t"
                    "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%5];\n\t"
                    "}\n" ::"r"(d_tmem), "l"(da), "l"(db), "r"(idesc), "r"(first ? 0u : 1u), "r"(smem_u32(&empty[s]))
                    : "memory");
                if ((kb % CH) == CH - 1 || kb == nkb - 1) { umma_commit_elect(&acc_full[buf]); ++c; }
            }
        }
    } else {
        const int dw = warp - 2;
        const int q = warp & 3;
        const int cbeg = (dw >> 2) * ACC;
        const int row = q * 32 + lane;
        const bool vec_ok = (p.ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.C) & 15) == 0);
        const uint32_t stg = smem_u32(smem + (size_t)NST * Cfg::STAGE + SS_STG_OFF) + (uint32_t)dw * 4096u;
        int c = 0;
        for (int tile = blockIdx.x; tile < tiles_total; tile += gridDim.x) {
            const int m0 = (tile / tiles_n) * TC_BM, n0 = (tile % tiles_n) * BN;
            float acc[ACC];
#pragma unroll
            for (int j = 0; j < ACC; ++j) acc[j] = 0.f;
            for (int cc = 0; cc < nchunks; ++cc, ++c) {
                const int buf = c & 1;
                mbar_wait(&acc_full[buf], (uint32_t)(c >> 1) & 1u);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                uint32_t r[ACC];
#pragma unroll
                for (int j0 = 0; j0 < ACC; j0 += 16) tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * Cfg::BUF + cbeg + j0), r + j0);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(&acc_empty[buf]);                     // the buffer is free as soon as it sits in registers
#pragma unroll
                for (int e = 0; e < ACC; ++e) acc[e] = fmaf(__uint_as_float(r[e]), p.oscale, acc[e]);
            }
            if constexpr (ROWS) ss_store_row<ACC>(p, acc, m0 + row, n0 + cbeg, lane, vec_ok);
            else ss_store_staged<ACC>(p, acc, m0 + q * 32, n0 + cbeg, lane, vec_ok, stg);
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(Cfg::TMEM_COLS) : "memory");
    }
}

// =====================================================================================================
// f16ss_pair_kernel — the persistent conversion-free GEMM on CTA PAIRS (tcgen05 cta_group::2, thread-block cluster of 2 = one TPC): the pair
// owns a 256 x 256 output tile; each CTA TMA-loads ITS 128 rows of A and ITS 128 of the 256 B rows per K slice (32 KB instead of the 48 KB a
// lone 128 x 256 tile needs), the leader CTA's MMA warp issues M = 256 MMAs that read both CTAs' shared memory and accumulate into both CTAs'
// tensor memory, each CTA drains and stores its own 128 rows.  The single-CTA kernel sits at the L2 -> SM bandwidth (ncu: 11 TB/s of ~12);
// the pair moves 2/3 of the bytes per FLOP.
//   barriers (leader's copy is the one waited on unless noted): full[s]   <- complete_tx of all four TMA loads of the slice (both CTAs)
//                                                                empty[s]  <- tcgen05.commit multicast to BOTH CTAs (each producer waits its own)
//                                                                acc_full  <- tcgen05.commit multicast to BOTH CTAs (each epilogue waits its own)
//                                                                acc_empty <- 8 + 8 drain warps of both CTAs arrive on the LEADER's barrier
// =====================================================================================================
struct PairCfg {
    static constexpr int NST = 6;
    static constexpr int A_BYTES = TC_BM * 128, B_BYTES = 128 * 128, STAGE = A_BYTES + B_BYTES;
    static constexpr int BUF = 256, TMEM_COLS = 512, DRAIN_WARPS = 8, ACC = 128, THREADS = (2 + DRAIN_WARPS) * 32;
    static constexpr size_t SMEM = (size_t)NST * STAGE + 1024 + 8 * (2 * NST + 4) + 64;
};
__device__ __forceinline__ void tma_load_4d_2sm(void* smem_dst, const CUtensorMap* map, uint64_t* leader_bar, int c0, int c1, int c2, int c3) {
    // executed by both CTAs of the pair; the transaction bytes are counted on the LEADER's barrier (CTA rank bit 24 of the cluster address cleared)
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(leader_bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void umma_commit_pair_elect(uint64_t* bar) {          // arrives on `bar` of BOTH CTAs once the MMAs issued so far have completed
    asm volatile(
        "{\n\t"
        ".reg .pred e;\n\t"
        ".reg .b16 m;\n\t"
        "mov.b16 m, 3;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "@e tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], m;\n\t"
        "}\n" ::"r"(smem_u32(bar))
        : "memory");
}
template <bool ROWS>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(PairCfg::THREADS, 1)
f16ss_pair_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const SsParams p, int tiles_n, int tiles_total) {
    using Cfg = PairCfg;
    constexpr int NST = Cfg::NST, ACC = Cfg::ACC;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)NST * Cfg::STAGE);
    uint64_t* empty = full + NST;
    uint64_t* acc_full = empty + NST;       // [2]
    uint64_t* acc_empty = acc_full + 2;     // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = cluster_ctarank();
    const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
    const int CH = p.chunk;
    const int nkb = p.nslices, nchunks = (nkb + CH - 1) / CH;
    if (tid == 0) {
        for (int s = 0; s < NST; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], 2 * Cfg::DRAIN_WARPS); }
        mbar_fence_init();
    }
    __syncthreads();
    cluster_sync_all();                                                          // both CTAs' barriers exist before anything can arrive on them
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(Cfg::TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    cluster_sync_all();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    if (warp == 0) {
        if (lane == 0) {
            prefetch_tmap(&mapA);
            prefetch_tmap(&mapB);
            int i = 0;
            for (int tile = pair; tile < tiles_total; tile += npairs) {
                const int m0 = (tile / tiles_n) * 256 + (int)rank * TC_BM, n0 = (tile % tiles_n) * 256 + (int)rank * 128;
                for (int kb = 0; kb < nkb; ++kb, ++i) {
                    const int s = i % NST;
                    mbar_wait(&empty[s], ((uint32_t)(i / NST) & 1u) ^ 1u);
                    unsigned char* st = smem + (size_t)s * Cfg::STAGE;
                    if (rank == 0) mbar_expect_tx(&full[s], 2 * (Cfg::A_BYTES + Cfg::B_BYTES));
                    tma_load_4d_2sm(st, &mapA, &full[s], kb * TC_BK, m0, 0, 0);
                    tma_load_4d_2sm(st + Cfg::A_BYTES, &mapB, &full[s], kb * TC_BK, n0, 0, 0);
                }
            }
        }
    } else if (warp == 1) {
        if (rank == 0) {
            const uint32_t idesc = make_idesc_f16(256, 256);
            int i = 0, c = 0;
            for (int tile = pair; tile < tiles_total; tile += npairs) {
                for (int kb = 0; kb < nkb; ++kb, ++i) {
                    const int s = i % NST;
                    const bool first = (kb % CH) == 0;
                    const int buf = c & 1;
                    if (first) mbar_wait_cluster(&acc_empty[buf], ((uint32_t)(c >> 1) & 1u) ^ 1u);
                    mbar_wait_cluster(&full[s], (uint32_t)(i / NST) & 1u);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t a_addr = smem_u32(smem + (size_t)s * Cfg::STAGE);
                    const uint64_t da = make_smem_desc_sw128(a_addr), db = make_smem_desc_sw128(a_addr + Cfg::A_BYTES);
                    const uint32_t d_tmem = tmem_base + (uint32_t)(buf * Cfg::BUF);
                    asm volatile(
                        "{\n\t"
                        ".reg .pred e, p0, pt;\n\t"
                        ".reg .b64 ah1, al0, al1, bh1, bl0, bl1;\n\t"
                        ".reg .b16 m;\n\t"
                        "mov.b16 m, 3;\n\t"
                        "elect.sync _|e, 0xffffffff;\n\t"
                        "setp.ne.b32 p0, %4, 0;\n\t"
                        "setp.eq.b32 pt, 0, 0;\n\t"
                        "add.u64 ah1, %1, 2;\n\t add.u64 al0, %1, 4;\n\t add.u64 al1, %1, 6;\n\t"
                        "add.u64 bh1, %2, 2;\n\t add.u64 bl0, %2, 4;\n\t add.u64 bl1, %2, 6;\n\t"
                        "@e tcgen05.mma.cta_group::2.kind::f16 [%0], al0, %2, %3, p0;\n\t"
                        "@e tcgen05.mma.cta_group::2.kind::f16 [%0], %1, bl0, %3, pt;\n\t"
                        "@e tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, pt;\n\t"
                        "@e tcgen05.mma.cta_group::2.kind::f16 [%0], al1, bh1, %3, pt;\n\t"
                        "@e tcgen05.mma.cta_group::2.kind::f16 [%0], ah1, bl1, %3, pt;\n\t"
                        "@e tcgen05.mma.cta_group::2.kind::f16 [%0], ah1, bh1, %3, pt;\n\t"
                        "@e tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%5], m;\n\t"
                        "}\n" ::"r"(d_tmem), "l"(da), "l"(db), "r"(idesc), "r"(first ? 0u : 1u), "r"(smem_u32(&empty[s]))
                        : "memory");
                    if ((kb % CH) == CH - 1 || kb == nkb - 1) { umma_commit_pair_elect(&acc_full[buf]); ++c; }
                }
            }
        }
    } else {
        const int dw = warp - 2;
        const int q = warp & 3;
        const int cbeg = (dw >> 2) * ACC;
        const int row = q * 32 + lane;
        const bool vec_ok = (p.ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.C) & 15) == 0);
        const uint32_t stg = smem_u32(smem + (size_t)NST * Cfg::STAGE + SS_STG_OFF) + (uint32_t)dw * 4096u;
        int c = 0;
        for (int tile = pair; tile < tiles_total; tile += npairs) {
            const int m0 = (tile / tiles_n) * 256 + (int)rank * TC_BM, n0 = (tile % tiles_n) * 256;
            float acc[ACC];
#pragma unroll
            for (int j = 0; j < ACC; ++j) acc[j] = 0.f;
            for (int cc = 0; cc < nchunks; ++cc, ++c) {
                const int buf = c & 1;
                mbar_wait(&acc_full[buf], (uint32_t)(c >> 1) & 1u);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                uint32_t r[ACC];
#pragma unroll
                for (int j0 = 0; j0 < ACC; j0 += 16) tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * Cfg::BUF + cbeg + j0), r + j0);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive_remote(&acc_empty[buf], 0);             // the LEADER's MMA warp owns the buffer hand-off for both CTAs
#pragma unroll
                for (int e = 0; e < ACC; ++e) acc[e] = fmaf(__uint_as_float(r[e]), p.oscale, acc[e]);
            }
            if constexpr (ROWS) ss_store_row<ACC>(p, acc, m0 + row, n0 + cbeg, lane, vec_ok);
            else ss_store_staged<ACC>(p, acc, m0 + q * 32, n0 + cbeg, lane, vec_ok, stg);
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    cluster_sync_all();                                                          // the peer's MMAs / remote arrivals are done with this CTA's memory
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(Cfg::TMEM_COLS) : "memory");
    }
}

// =====================================================================================================
// gru_step_f16_kernel — one time step of one bidirectional GRU layer (model.py:150-154): gh = W_hh h(t-1) on the tensor cores with the
// gate math fused.  The batch (<= 128 clips) is the M side: thread b of the drain warps owns clip b; the N side is a gate-interleaved
// tile of W_hh: rows [r | z | n] of 32 hidden units (three TMA boxes of 32 rows) = 96 columns, so every thread ends up with the r, z and
// n pre-activations of 32 units of ITS clip and finishes the cell alone: no exchange, and every global access of the epilogue is a
// 128-byte run per thread (gi row, previous state, new state, layer output, and the fp16x3 image of the new state = exactly one K slice
// of the next step's A operand).  Both operands arrive pre-split (h image written by the previous step, W_hh image packed once):
// TMA -> tcgen05 SS MMAs, K = G in 32-wide slices, fp32 register drain every 2 slices.   grid (G / 32, 1, 2 directions).
// =====================================================================================================
struct GruStepParams {
    const float* gi;            // [B, T, 6G]  W_ih x + b_ih, direction d at column offset d * 3G
    const float* bhh;           // [2][3G]
    const float* h_prev;        // [2][B][G] fp32
    float* h_new;               // [2][B][G] fp32
    float* h_img_new;           // [2][B][G] words: fp16x3 image of h_new (A operand of the next step)
    float* out;                 // [B, T, 2G]
    const long long* sample_idx;
    int B, T, G, step, nslices;
    float oscale, sa;
};
constexpr int GRU_BN = 96, GRU_NST = 6, GRU_STAGE = TC_BM * 128 + 12 * 1024;      // A 16 KB + B 96 x 128 B
constexpr size_t GRU_SMEM = (size_t)GRU_NST * GRU_STAGE + 1024 + 8 * (2 * GRU_NST + 4) + 64;
__global__ void __launch_bounds__(6 * 32, 1)
gru_step_f16_kernel(const __grid_constant__ CUtensorMap mapH, const __grid_constant__ CUtensorMap mapW, const GruStepParams p) {
    constexpr int NST = GRU_NST, BN = GRU_BN;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)NST * GRU_STAGE);
    uint64_t* empty = full + NST;
    uint64_t* acc_full = empty + NST;
    uint64_t* acc_empty = acc_full + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int u0 = blockIdx.x * 32, d = blockIdx.z, G = p.G;
    const int nkb = p.nslices, nchunks = (nkb + 1) / 2;
    if (tid == 0) {
        for (int s = 0; s < NST; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], 4); }
        mbar_fence_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(256) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    if (tid == 0) pdl_trigger();                  // step t + 1 may be scheduled now: it prefetches its W_hh tiles and waits for our h itself
    if (warp == 0) {
        if (lane == 0) {
            prefetch_tmap(&mapH);
            prefetch_tmap(&mapW);
            // launched with programmatic stream serialization: the W_hh tiles (constant) of the first ring fill stream in while the
            // previous time step is still running; the state image is only touched after griddepcontrol.wait
            const int npre = min(nkb, NST);
            for (int i = 0; i < npre; ++i) {
                unsigned char* st = smem + (size_t)i * GRU_STAGE;
                mbar_expect_tx(&full[i], TC_BM * 128 + BN * 128);
#pragma unroll
                for (int g = 0; g < 3; ++g) tma_load_4d(st + TC_BM * 128 + g * 32 * 128, &mapW, &full[i], i * TC_BK, g * G + u0, 0, d);
            }
            pdl_wait();
            for (int i = 0; i < npre; ++i) tma_load_4d(smem + (size_t)i * GRU_STAGE, &mapH, &full[i], i * TC_BK, 0, 0, d);
            for (int i = npre; i < nkb; ++i) {
                const int s = i % NST;
                mbar_wait(&empty[s], ((uint32_t)(i / NST) & 1u) ^ 1u);
                unsigned char* st = smem + (size_t)s * GRU_STAGE;
                mbar_expect_tx(&full[s], TC_BM * 128 + BN * 128);
                tma_load_4d(st, &mapH, &full[s], i * TC_BK, 0, 0, d);
#pragma unroll
                for (int g = 0; g < 3; ++g) tma_load_4d(st + TC_BM * 128 + g * 32 * 128, &mapW, &full[s], i * TC_BK, g * G + u0, 0, d);
            }
        }
    } else if (warp == 1) {
        const uint32_t idesc = make_idesc_f16(TC_BM, BN);
        for (int i = 0; i < nkb; ++i) {
            const int s = i % NST;
            const int c = i / 2, buf = c & 1;
            const bool first = (i % 2) == 0;
            if (first) mbar_wait(&acc_empty[buf], ((uint32_t)(c >> 1) & 1u) ^ 1u);
            mbar_wait(&full[s], (uint32_t)(i / NST) & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t a_addr = smem_u32(smem + (size_t)s * GRU_STAGE);
            const uint64_t da = make_smem_desc_sw128(a_addr), db = make_smem_desc_sw128(a_addr + TC_BM * 128);
            const uint32_t d_tmem = tmem_base + (uint32_t)(buf * 128);
            asm volatile(
                "{\n\t"
                ".reg .pred e, p0, pt;\n\t"
                ".reg .b64 ah1, al0, al1, bh1, bl0, bl1;\n\t"
                "elect.sync _|e, 0xffffffff;\n\t"
                "setp.ne.b32 p0, %4, 0;\n\t"
                "setp.eq.b32 pt, 0, 0;\n\t"
                "add.u64 ah1, %1, 2;\n\t add.u64 al0, %1, 4;\n\t add.u64 al1, %1, 6;\n\t"
                "add.u64 bh1, %2, 2;\n\t add.u64 bl0, %2, 4;\n\t add.u64 bl1, %2, 6;\n\t"
                "@e tcgen05.mma.cta_group::1.kind::f16 [%0], al0, %2, %3, p0;\n\t"
                "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, bl0, %3, pt;\n\t"
                "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, pt;\n\t"
                "@e tcgen05.mma.cta_group::1.kind::f16 [%0], al1, bh1, %3, pt;\n\t"
                "@e tcgen05.mma.cta_group::1.kind::f16 [%0], ah1, bl1, %3, pt;\n\t"
                "@e tcgen05.mma.cta_group::1.kind::f16 [%0], ah1, bh1, %3, pt;\n\t"
                "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%5];\n\t"
                "}\n" ::"r"(d_tmem), "l"(da), "l"(db), "r"(idesc), "r"(first ? 0u : 1u), "r"(smem_u32(&empty[s]))
                : "memory");
            if ((i % 2) == 1 || i == nkb - 1) umma_commit_elect(&acc_full[buf]);
        }
    } else {
        const int q = warp & 3;
        const int b = q * 32 + lane;                                          // this thread's clip
        float acc[BN];
#pragma unroll
        for (int j = 0; j < BN; ++j) acc[j] = 0.f;
        for (int c = 0; c < nchunks; ++c) {
            const int buf = c & 1;
            mbar_wait(&acc_full[buf], (uint32_t)(c >> 1) & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
            for (int jb = 0; jb < BN; jb += 48) {
                uint32_t r[48];
#pragma unroll
                for (int j0 = 0; j0 < 48; j0 += 16) tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * 128 + jb + j0), r + j0);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int e = 0; e < 48; ++e) acc[jb + e] = fmaf(__uint_as_float(r[e]), p.oscale, acc[jb + e]);
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[buf]);
        }
        pdl_wait();                               // the previous state (and, for step 0, gi) come from predecessor kernels
        if (b < p.B) {
            // gate math: r, z, n order, b_hn inside the r product (torch.nn.GRU); acc[0..32) = W_hr h, [32..64) = W_hz h, [64..96) = W_hn h
            const int t = d ? (p.T - 1 - p.step) : p.step;
            const float* gir = p.gi + ((size_t)b * p.T + t) * (6 * G) + (size_t)d * 3 * G + u0;
            const float* bh = p.bhh + (size_t)d * 3 * G + u0;
            const size_t so = ((size_t)d * p.B + b) * G + u0;
            float hv[32];
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
                const float4 gr = *reinterpret_cast<const float4*>(gir + j), gz = *reinterpret_cast<const float4*>(gir + G + j);
                const float4 gn = *reinterpret_cast<const float4*>(gir + 2 * G + j), hp = *reinterpret_cast<const float4*>(p.h_prev + so + j);
                const float4 br = __ldg(reinterpret_cast<const float4*>(bh + j)), bz = __ldg(reinterpret_cast<const float4*>(bh + G + j));
                const float4 bn = __ldg(reinterpret_cast<const float4*>(bh + 2 * G + j));
                const float grr[4] = {gr.x, gr.y, gr.z, gr.w}, gzz[4] = {gz.x, gz.y, gz.z, gz.w}, gnn[4] = {gn.x, gn.y, gn.z, gn.w};
                const float hpp[4] = {hp.x, hp.y, hp.z, hp.w}, brr[4] = {br.x, br.y, br.z, br.w}, bzz[4] = {bz.x, bz.y, bz.z, bz.w};
                const float bnn[4] = {bn.x, bn.y, bn.z, bn.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float rg = sigmoid_acc(grr[e] + acc[j + e] + brr[e]);
                    const float zg = sigmoid_acc(gzz[e] + acc[32 + j + e] + bzz[e]);
                    const float ng = tanhf(gnn[e] + rg * (acc[64 + j + e] + bnn[e]));
                    hv[j + e] = (1.f - zg) * ng + zg * hpp[e];
                }
            }
            bool keep = true;
            if (p.sample_idx) {
                const long long lo = p.sample_idx[2 * b], hi = p.sample_idx[2 * b + 1];
                keep = !(t < lo || t >= hi);
            }
            float* hn = p.h_new + so;
            float* o = p.out + ((size_t)b * p.T + t) * (2 * G) + (size_t)d * G + u0;
            uint32_t* img = reinterpret_cast<uint32_t*>(p.h_img_new) + so;       // u0 is a multiple of 32: this thread's units are one K slice
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
                *reinterpret_cast<float4*>(hn + j) = make_float4(hv[j], hv[j + 1], hv[j + 2], hv[j + 3]);
                *reinterpret_cast<float4*>(o + j) = keep ? make_float4(hv[j], hv[j + 1], hv[j + 2], hv[j + 3]) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            uint32_t hi_w[16], lo_w[16];
#pragma unroll
            for (int pr = 0; pr < 16; ++pr) f16x3_split_pair(hv[2 * pr], hv[2 * pr + 1], p.sa, hi_w[pr], lo_w[pr]);
#pragma unroll
            for (int j = 0; j < 16; j += 4) {
                *reinterpret_cast<uint4*>(img + j) = make_uint4(hi_w[j], hi_w[j + 1], hi_w[j + 2], hi_w[j + 3]);
                *reinterpret_cast<uint4*>(img + 16 + j) = make_uint4(lo_w[j], lo_w[j + 1], lo_w[j + 2], lo_w[j + 3]);
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(256) : "memory");
    }
}

template <int BN, int EPI>
static int launch_f16ss(const CUtensorMap& mA, const CUtensorMap& mB, const SsParams& p, dim3 grid, cudaStream_t st) {
    static bool attr = false;
    if (!attr) { GVD_CHECK_CUDA(cudaFuncSetAttribute(f16ss_kernel<BN, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SsCfg<BN, EPI>::SMEM)); attr = true; }
    f16ss_kernel<BN, EPI><<<grid, SsCfg<BN, EPI>::THREADS, SsCfg<BN, EPI>::SMEM, st>>>(mA, mB, p);
    GVD_CHECK_LAUNCH();
    return 0;
}

// part[s][b][n] = sum_{k in split s} Wp[n][k] Xp[b][k] with both operands in the fp16x3 image (gvd_pack_f16x3 / the packed activation
// buffers): Wp [Nw, Kp] words, Xp [B, ldx] words; Kp, ldx multiples of 32; nslices = 32-wide K slices per split
int gvd_skinny_f16(const float* Wp, long long ldw, int Nw, const float* Xp, long long ldx, int B, int Ktot, int S, float* part, int ldp,
                   cudaStream_t st) {
    GVD_REQUIRE(Wp && Xp && part && B >= 1 && B <= 128 && S >= 1 && Ktot % (32 * S) == 0 && ldw % 32 == 0 && ldx % 32 == 0 && ldp >= Nw,
                "skinny_f16: bad arguments (Ktot=%d S=%d)", Ktot, S);
    CUtensorMap mA, mB;
    int d0, d1;
    const int bn = B <= 112 ? 112 : 128;
    GVD_TRY(make_map(&mA, Wp, Ktot, Nw, ldw, 1, 0, 1, 0, TC_BM, &d0, &d1));
    GVD_TRY(make_map(&mB, Xp, Ktot, B, ldx, 1, 0, 1, 0, bn, &d0, &d1));
    SsParams p{};
    p.C = part; p.ldc = ldp; p.plane = (long long)B * ldp; p.M = Nw; p.N = B; p.nslices = Ktot / (32 * S);
    p.oscale = 1.f / (GVD_F16_SA * GVD_F16_SW);
    dim3 grid(1, gvd_cdiv(Nw, TC_BM), S);
    return bn == 112 ? launch_f16ss<112, 3>(mA, mB, p, grid, st) : launch_f16ss<128, 3>(mA, mB, p, grid, st);
}

// One bidirectional GRU layer on the tensor cores: T launches of gru_step_f16_kernel with programmatic stream serialization (step t + 1 is
// scheduled while step t runs; only 32 of the 148 SMs are busy per step, so its CTAs start at once, prefetch W_hh and wait for h).
// hstate / h_img: [2 parity][2 dir][B][G] fp32 / fp16x3 words, zero-initialised here.  Whh_img: [2][3G][G] words.  B <= 128, G % 32 == 0.
int gvd_gru_layer_f16(const float* gi, const float* Whh_img, const float* bhh, float* hstate, float* h_img, float* out, const long long* sample_idx, int B,
                      int T, int G, cudaStream_t st) {
    GVD_REQUIRE(gi && Whh_img && bhh && hstate && h_img && out && B >= 1 && B <= 128 && G % 32 == 0, "gru_layer_f16: bad arguments");
    const size_t half = (size_t)2 * B * G;
    GVD_CHECK_CUDA(cudaMemsetAsync(hstate, 0, 2 * half * sizeof(float), st));
    GVD_CHECK_CUDA(cudaMemsetAsync(h_img, 0, 2 * half * sizeof(float), st));
    CUtensorMap mH[2], mW;
    int d0, d1;
    for (int par = 0; par < 2; ++par) GVD_TRY(make_map(&mH[par], h_img + par * half, G, B, G, 1, 0, 2, (long long)B * G, TC_BM, &d0, &d1));
    GVD_TRY(make_map(&mW, Whh_img, G, 3ll * G, G, 1, 0, 2, 3ll * G * G, 32, &d0, &d1));
    static bool attr = false;
    if (!attr) { GVD_CHECK_CUDA(cudaFuncSetAttribute(gru_step_f16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GRU_SMEM)); attr = true; }
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(G / 32, 1, 2); cfg.blockDim = dim3(192); cfg.dynamicSmemBytes = GRU_SMEM; cfg.stream = st;
    cudaLaunchAttribute la[1];
    la[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    la[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = la; cfg.numAttrs = getenv("GVD_GRU_NO_PDL") ? 0 : 1;          // (griddepcontrol is a no-op in a launch without the attribute)
    for (int s = 0; s < T; ++s) {
        const size_t cur = (size_t)(s & 1) * half, nxt = (size_t)((s + 1) & 1) * half;
        GruStepParams p{gi, bhh, hstate + cur, hstate + nxt, h_img + nxt, out, sample_idx, B, T, G, s, G / 32, 1.f / (GVD_F16_SA * GVD_F16_SW), GVD_F16_SA};
        GVD_CHECK_CUDA(cudaLaunchKernelEx(&cfg, gru_step_f16_kernel, mH[s & 1], mW, p));
        gvd_count_launch();
    }
    return 0;
}

// Persistent kernels launch (SM count - reserve) CTAs while a reserve is set: a persistent CTA holds its SM (all of its shared and tensor
// memory) until the last tile, so a concurrent chain of short launches on another stream would otherwise advance one link per GEMM.
// Host-side state of the enqueuing thread (every launch site reads it at enqueue time).
static thread_local int g_sm_reserve = 0;
int gvd_sm_reserve(int n) { const int old = g_sm_reserve; g_sm_reserve = n < 0 ? 0 : n; return old; }

using SsPersistentFn = void (*)(CUtensorMap, CUtensorMap, SsParams, int, int);
template <SsPersistentFn F>
static int launch_ss_persistent(size_t smem, int ctas, int threads, const CUtensorMap& mA, const CUtensorMap& mB, const SsParams& p, int tiles_n, int tiles,
                                cudaStream_t st) {
    static bool a = false;
    if (!a) { GVD_CHECK_CUDA(cudaFuncSetAttribute(F, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); a = true; }
    F<<<ctas, threads, smem, st>>>(mA, mB, p, tiles_n, tiles);
    return 0;
}

// C[M, N] = act(A W^T + bias) with both operands in the fp16x3 image: Ap [M, lda] words (scale GVD_F16_SA), Wp [N, ldw] words (scale
// GVD_F16_SW), lda / ldw multiples of 32 covering K rounded up to 32 (zero padded)
int gvd_gemm_f16ss(const float* Ap, long long lda, const float* Wp, long long ldw, const float* bias, const float* scale2, const float* shift2, int act,
                   float* C, long long ldc, int M, int N, int K, cudaStream_t st, float* img, long long ld_img, const GvdQkvImages* qkv) {
    GVD_REQUIRE(Ap && Wp && (C || img) && M > 0 && N > 0 && K > 0 && lda % 32 == 0 && ldw % 32 == 0, "gemm_f16ss: bad arguments");
    if (qkv) {
        GVD_REQUIRE(C && !img && !bias && act == GVD_ACT_NONE && qkv->k_img && qkv->vt_img, "gemm_f16ss(qkv): plain projection, Q to C, K / V to their images");
        GVD_REQUIRE(N == 3 * qkv->HP && qkv->HP == qkv->nh * qkv->HS && qkv->HS % 4 == 0 && qkv->KH % 32 == 0 && qkv->KH >= qkv->HS && qkv->KH - qkv->HS < 32,
                    "gemm_f16ss(qkv): head layout");
        GVD_REQUIRE(qkv->R % 2 == 0 && M % qkv->R == 0 && qkv->Rp % 32 == 0 && qkv->Rp >= qkv->R && qkv->Rp - qkv->R < 32 && ldc % 4 == 0 &&
                    (reinterpret_cast<uintptr_t>(C) & 15) == 0, "gemm_f16ss(qkv): row layout");
    }
    GVD_REQUIRE(!img || (ld_img % 32 == 0 && ld_img >= N), "gemm_f16ss: the output image needs a 32-multiple pitch >= N");
    const int Kp = (K + 31) / 32 * 32;
    GVD_REQUIRE(lda >= Kp && ldw >= Kp, "gemm_f16ss: operand images must cover K rounded up to 32");
    CUtensorMap mA, mB;
    int d0, d1;
    const long long mt = gvd_cdiv(M, TC_BM);
    static const bool wide = getenv("GVD_SS_BN128") == nullptr;          // 256-column tiles by default: the 128-column kernel sits at the L2 -> SM bandwidth (ncu: 11 TB/s)
    const int bn = (wide && N >= 512 && mt * (N / 256) >= 148) ? 256 : ((mt * gvd_cdiv(N, 128) >= 120) ? 128 : 64);
    GVD_TRY(make_map(&mA, Ap, Kp, M, lda, 1, 0, 1, 0, TC_BM, &d0, &d1));
    GVD_TRY(make_map(&mB, Wp, Kp, N, ldw, 1, 0, 1, 0, bn, &d0, &d1));
    SsParams p{};
    p.C = C; p.ldc = ldc; p.plane = 0; p.M = M; p.N = N; p.nslices = Kp / 32;
    p.oscale = 1.f / (GVD_F16_SA * GVD_F16_SW);
    p.bias = bias; p.scale2 = scale2; p.shift2 = shift2; p.act = act;
    p.img = reinterpret_cast<uint32_t*>(img); p.ld_img = ld_img; p.img_scale = GVD_F16_SA;
    // K slices accumulated inside TMEM between two fp32 register drains.  The tensor core's accumulate truncates: measured max relative error vs fp64
    // (tools/f16ss_err.py, K = 2048, same-sign operands = worst case) 6.0e-7 / 9.2e-7 / 1.8e-6 / 3.9e-6 for 2 / 4 / 8 / 16 slices with a mean signed
    // error of -2.5e-7 / -6.2e-7 / -1.4e-6 / -3.1e-6; step time 25.02 / 24.86 / 24.38 ms for 2 / 4 / 8.  4 keeps the error in the class of an fp32
    // accumulation and lets the MMA warp run 8 slices ahead of the epilogue's store phase.
    static const int ss_chunk = getenv("GVD_SS_CHUNK") ? std::max(1, atoi(getenv("GVD_SS_CHUNK"))) : 4;
    p.chunk = ss_chunk;
    if (qkv) {
        p.qkv_hp = qkv->HP; p.qkv_hs = qkv->HS; p.qkv_kh = qkv->KH; p.qkv_nh = qkv->nh; p.qkv_R = qkv->R; p.qkv_Rp = qkv->Rp;
        p.k_img = reinterpret_cast<uint32_t*>(qkv->k_img); p.vt_img = reinterpret_cast<uint32_t*>(qkv->vt_img);
        p.qkv_sk = qkv->sk; p.qkv_sv = qkv->sv;
    }
    dim3 grid(gvd_cdiv(N, bn), (unsigned)mt, 1);
    static const bool no_persist = getenv("GVD_SS_NO_PERSIST") != nullptr;
    GVD_REQUIRE(!((img || qkv) && no_persist), "gemm_f16ss: the output images are emitted by the persistent kernel only");
    if (!no_persist) {
        static int sms = 0;
        if (!sms) { int dev = 0; GVD_CHECK_CUDA(cudaGetDevice(&dev)); GVD_CHECK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)); }
        const int tiles_n = gvd_cdiv(N, bn);
        const long long tiles = (long long)tiles_n * mt;
        // SMs left free for a concurrent stream (the bi-GRU chain of the frame branch: gvd_sm_reserve, set by the prologue around the region stages)
        const int ctas = (int)std::min<long long>(tiles, std::max(1, sms - g_sm_reserve));
        static const bool no_pair = getenv("GVD_SS_NO_PAIR") != nullptr;
        // thread-per-row epilogue stores (ss_store_row) for the Q|K|V projection (staged, its per-head routing measured slower: interact.qkv_proj
        // 5.6 vs 4.8 ms per step) and under backend bit 11, the reference the staged epilogue is tested against
        const bool rows = qkv || (gvd_backend() & 2048) != 0;
        if (bn == 256 && !no_pair && (gvd_backend() & 1024) != 0 && sms % 2 == 0) {
            // CTA pairs (backend bit 10): 256 x 256 tiles, each CTA streams half of the B tile
            CUtensorMap mB2;
            GVD_TRY(make_map(&mB2, Wp, Kp, N, ldw, 1, 0, 1, 0, 128, &d0, &d1));
            const int tn2 = gvd_cdiv(N, 256);
            const long long tiles2 = (long long)tn2 * gvd_cdiv(M, 256);
            const int ctas2 = (int)std::min<long long>(2 * tiles2, std::max(2, (sms - g_sm_reserve) & ~1));
            GVD_TRY((rows ? launch_ss_persistent<f16ss_pair_kernel<true>> : launch_ss_persistent<f16ss_pair_kernel<false>>)(
                ss_persist_smem<PairCfg>(), ctas2, PairCfg::THREADS, mA, mB2, p, tn2, (int)tiles2, st));
        } else if (bn == 256) {
            GVD_TRY((rows ? launch_ss_persistent<f16ss_persistent_kernel<256, true>> : launch_ss_persistent<f16ss_persistent_kernel<256, false>>)(
                ss_persist_smem<SsCfg<256, 0>>(), ctas, SsCfg<256, 0>::THREADS, mA, mB, p, tiles_n, (int)tiles, st));
        } else if (bn == 128) {
            GVD_TRY((rows ? launch_ss_persistent<f16ss_persistent_kernel<128, true>> : launch_ss_persistent<f16ss_persistent_kernel<128, false>>)(
                ss_persist_smem<SsCfg<128, 0>>(), ctas, SsCfg<128, 0>::THREADS, mA, mB, p, tiles_n, (int)tiles, st));
        } else {
            GVD_TRY((rows ? launch_ss_persistent<f16ss_persistent_kernel<64, true>> : launch_ss_persistent<f16ss_persistent_kernel<64, false>>)(
                ss_persist_smem<SsCfg<64, 0>>(), ctas, SsCfg<64, 0>::THREADS, mA, mB, p, tiles_n, (int)tiles, st));
        }
        GVD_CHECK_LAUNCH();
        return 0;
    }
    GVD_REQUIRE(bn != 256, "gemm_f16ss: 256-column tiles exist in the persistent kernel only");
    return bn == 128 ? launch_f16ss<128, 0>(mA, mB, p, grid, st) : launch_f16ss<64, 0>(mA, mB, p, grid, st);
}

// C = act(alpha * A W^T + bias) with the GemmArgs contract of gvd_gemm.cuh (batched over (b,h))
int gvd_gemm_nt_tc(const GemmArgs& g, int batch, cudaStream_t stream) {
    GVD_REQUIRE(g.M > 0 && g.N > 0 && g.K > 0 && g.nh >= 1 && batch % g.nh == 0, "tcgemm: bad problem");
    GVD_REQUIRE(g.K % 4 == 0 && g.lda % 4 == 0 && g.ldw % 4 == 0, "tcgemm: K/lda/ldw must be multiples of 4");
    const int nb = batch / g.nh;
    // N tile: wide tiles for big problems, narrow ones so that skinny problems still fill 148 SMs
    const long long mt = gvd_cdiv(g.M, TC_BM);
    int BN = 128;
    if (mt * gvd_cdiv(g.N, 128) * batch < 120) BN = 64;
    if (mt * gvd_cdiv(g.N, 64) * batch < 120) BN = 32;
    if (g.force_bn == 32 || g.force_bn == 64 || g.force_bn == 128) BN = g.force_bn;
    // opt-in wide tiles (see Tc2Cfg): whole 256-column tiles through the BN = 256 instantiation, the remaining columns through the
    // regular path (a second launch on the column tail), so that no CTA computes discarded columns
    if (BN == 128 && !g.force_bn && tc_bn256() && g.N >= 256 && mt * (g.N / 256) * batch >= 148 && !use_v1_static()) {
        const int n_main = (g.N / 256) * 256;
        if (n_main < g.N) {
            GemmArgs t = g;
            t.W = g.W + (long long)n_main * g.ldw; t.C = g.C + n_main; t.N = g.N - n_main;
            if (g.bias) t.bias = g.bias + n_main;
            if (g.scale2) t.scale2 = g.scale2 + n_main;
            if (g.shift2) t.shift2 = g.shift2 + n_main;
            GVD_REQUIRE((n_main * g.ldw) % 4 == 0, "tcgemm: tail operand not 16-byte aligned");
            GVD_TRY(gvd_gemm_nt_tc(t, batch, stream));
        }
        GemmArgs m = g;
        m.N = n_main;
        CUtensorMap mA2[3], mW2[3];
        TcParams p2{};
        p2.cs = 1;
        GVD_TRY(make_map(&mA2[0], m.A, m.K, m.M, m.lda, m.nh, m.sAh, nb, m.sAb, TC_BM, &p2.a_mul_h, &p2.a_mul_b));
        GVD_TRY(make_map(&mW2[0], m.W, m.K, m.N, m.ldw, m.nh, m.sWh, nb, m.sWb, 256, &p2.w_mul_h, &p2.w_mul_b));
        mA2[1] = mA2[2] = mA2[0];
        mW2[1] = mW2[2] = mW2[0];
        p2.nseg = 1;
        p2.seg[0] = TcSeg{m.K, 0, 0};
        p2.M = m.M; p2.N = m.N; p2.nh = m.nh;
        p2.C = m.C; p2.ldc = m.ldc; p2.sCb = m.sCb; p2.sCh = m.sCh;
        p2.bias = m.bias; p2.sBb = m.sBb; p2.scale2 = m.scale2; p2.shift2 = m.shift2; p2.act = m.act; p2.alpha = m.alpha;
        p2.mode = 0;
        return launch_tc<256>(mA2, mW2, p2, dim3(m.N / 256, (unsigned)mt, batch), stream);
    }
    CUtensorMap mA[3], mW[3];
    TcParams p{};
    // skinny problems (BN = 32, one m-tile wide N): clusters of 8 CTAs along N share the activation slice by TMA multicast
    const int cs_want = tc_cluster_size();
    p.cs = (BN == 32 && batch == 1 && cs_want > 1 && !use_v1_static() && gvd_cdiv(g.N, 32) >= cs_want) ? cs_want : 1;
    GVD_TRY(make_map(&mA[0], g.A, g.K, g.M, g.lda, g.nh, g.sAh, nb, g.sAb, TC_BM / p.cs, &p.a_mul_h, &p.a_mul_b));
    {
        // fp16x3: a registered constant weight has a pre-split copy (hi | lo halves per 32-wide K slice, gvd_pack_f16x3): stream that one and
        // skip the in-kernel W conversion (half of the shared-memory traffic of a K slice)
        const float* Wp = nullptr;
        long long ldp = 0;
        if (gvd_gemm_f16() && batch == 1 && g.nh == 1 && p.cs == 1 && !use_v1_static() && gvd_packed_lookup(g.W, g.ldw, g.N, g.K, &Wp, &ldp)) {
            GVD_TRY(make_map(&mW[0], Wp, (g.K + 31) / 32 * 32, g.N, ldp, 1, 0, 1, 0, BN, &p.w_mul_h, &p.w_mul_b));
            p.wpre = 1;
        } else {
            GVD_TRY(make_map(&mW[0], g.W, g.K, g.N, g.ldw, g.nh, g.sWh, nb, g.sWb, BN, &p.w_mul_h, &p.w_mul_b));
        }
    }
    mA[1] = mA[2] = mA[0];
    mW[1] = mW[2] = mW[0];
    p.nseg = 1;
    p.seg[0] = TcSeg{g.K, 0, 0};
    p.M = g.M; p.N = g.N; p.nh = g.nh;
    p.C = g.C; p.ldc = g.ldc; p.sCb = g.sCb; p.sCh = g.sCh;
    p.bias = g.bias; p.sBb = g.sBb; p.scale2 = g.scale2; p.shift2 = g.shift2; p.act = g.act; p.alpha = g.alpha;
    p.mode = g.trans_c ? 3 : 0;
    p.pdl = g.pdl;
    GVD_REQUIRE(!g.trans_c || (!g.bias && g.act == GVD_ACT_NONE && !use_v1_static()), "tcgemm: the transposed store takes no bias / activation");
    dim3 grid(gvd_cdiv(g.N, BN), (unsigned)mt, batch);
    if (p.cs > 1) grid.x = (grid.x + p.cs - 1) / p.cs * p.cs;          // whole clusters; the padding CTAs compute discarded columns
    if (BN == 128) return launch_tc<128>(mA, mW, p, grid, stream);
    if (BN == 64) return launch_tc<64>(mA, mW, p, grid, stream);
    return launch_tc<32>(mA, mW, p, grid, stream);
}

// Vocabulary head + greedy pick fused (mode 2): logits = h W^T + b are reduced on the fly, nothing [B,V]-sized is stored.
int gvd_logit_pick_tc(const float* h, long long ldh, const float* W, long long ldw, const float* bias, int B, int V, int K, int unk_idx,
                      float* part, int* ticket, long long* it_out, long long* seq_out, float* logp_out, long long out_stride,
                      const float* embed, float* xt, int E, cudaStream_t stream) {
    GVD_REQUIRE(B >= 1 && B <= TC_BM, "logit_pick: at most %d rows per launch (got %d)", TC_BM, B);
    GVD_REQUIRE(bias && part && ticket && it_out, "logit_pick: null argument");
    GVD_REQUIRE(!use_v1_static(), "logit_pick: not available with the v1 kernel (GVD_TC_V1)");
    CUtensorMap mA[3], mW[3];
    TcParams p{};
    p.cs = 1;
    GVD_TRY(make_map(&mA[0], h, K, B, ldh, 1, 0, 1, 0, TC_BM, &p.a_mul_h, &p.a_mul_b));
    GVD_TRY(make_map(&mW[0], W, K, V, ldw, 1, 0, 1, 0, 32, &p.w_mul_h, &p.w_mul_b));
    mA[1] = mA[2] = mA[0];
    mW[1] = mW[2] = mW[0];
    p.nseg = 1;
    p.seg[0] = TcSeg{K, 0, 0};
    p.M = B; p.N = V; p.nh = 1; p.mode = 2; p.bias = bias; p.alpha = 1.f;
    p.pk_part = part; p.pk_ticket = ticket; p.pk_it = it_out; p.pk_seq = seq_out; p.pk_logp = logp_out; p.pk_stride = out_stride;
    p.pk_unk = unk_idx; p.pk_embed = embed; p.pk_xt = xt; p.pk_E = E;
    dim3 grid(gvd_cdiv(V, 32), 1, 1);
    return launch_tc<32>(mA, mW, p, grid, stream);
}

// LSTMCell step on the tensor cores: same contract as gvd_lstm_step, but segment inputs must be dense
// activation matrices (the caller materialises xt = ReLU(embed[token]) once per step).
int gvd_lstm_step_tc(const LstmArgs& a, cudaStream_t stream) {
    GVD_REQUIRE(a.nseg >= 1 && a.nseg <= 3 && a.H % 8 == 0, "lstm_tc: needs 1..3 segments and H %% 8 == 0");
    CUtensorMap mA[3], mW[3];
    TcParams p{};
    p.nseg = a.nseg;
    const int cs_want = tc_cluster_size();
    p.cs = (cs_want > 1 && !use_v1_static() && a.H / 8 >= cs_want) ? cs_want : 1;
    for (int s = 0; s < 3; ++s) {
        const LstmSeg& sg = a.seg[s < a.nseg ? s : 0];
        GVD_REQUIRE(!sg.gather && !sg.relu, "lstm_tc: gather/ReLU segments must be materialised by the caller");
        int d0, d1;
        GVD_TRY(make_map(&mA[s], sg.x, sg.K, a.B, sg.ldx, 1, 0, 1, 0, TC_BM / p.cs, &d0, &d1));
        GVD_TRY(make_map(&mW[s], sg.w, sg.K, 4ll * a.H, sg.ldw, 1, 0, 1, 0, 8, &d0, &d1));
        if (s < a.nseg) p.seg[s] = TcSeg{sg.K, 0, 0};
    }
    p.M = a.B; p.N = 4 * a.H; p.nh = 1; p.mode = 1; p.H = a.H; p.UJ = 8;
    p.pre = a.pre; p.pre_div = a.pre_div; p.bias1 = a.bias1; p.bias2 = a.bias2; p.c_prev = a.c_prev; p.h_out = a.h_out; p.c_out = a.c_out;
    p.alpha = 1.f;
    dim3 grid(a.H / 8, gvd_cdiv(a.B, TC_BM), 1);
    if (p.cs > 1) grid.x = (grid.x + p.cs - 1) / p.cs * p.cs;          // padding CTAs (j0 >= H) store nothing
    return launch_tc<32>(mA, mW, p, grid, stream);
}
