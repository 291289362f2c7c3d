// Full-precision Linear over many rows on the tcgen05 tensor cores (reference models/sv_layers.py:29-31,
// nn.Linear path of the fp SV models: conv5's 505 -> 512 linear1, the PointNet per-point blocks).
// fp32-level accuracy from bf16 tensor cores: both operands are split EXACTLY into three bf16 planes
// (hi + mid + lo = the fp32 value) and six plane products (h*h, h*m, m*h, m*m, h*l, l*h) are accumulated
// in fp32 tensor memory; the dropped products are < 2^-20 of |a||w| per term.  The summation order differs
// from the CUDA-core kernel's sequential chain (gemm.cu), so this path is tolerance-level (1e-5 relative,
// far inside the 1e-3 / 1e-4 contract of the fp models).  It is chosen by (K, N) only, never by the row count,
// so that a cloud's result does not depend on the batch it is in.
//
//   D[c][r] = sum_k W[c][k] * a[r][k]        M = 128 channels per tile (two accumulators per tile, two tiles per
//                                            CTA: the whole 512-column tensor memory), N = 128 rows, K = 16 per UMMA
//   * weights     : split once per call into [tile][k-chunk 32][plane][k-block 4][128 channels][8 bf16]
//                   (24 KB per chunk), streamed through an mbarrier ring with cp.async.bulk
//   * activations : the CTA's 128 rows are split chunk by chunk into the same layout (double buffered in
//                   shared memory) by the 8 worker warps while the previous chunk's MMAs run
//   * epilogue    : lane = channel -> contiguous stores; colscale / bias / BN / activation as gemm.cu
#include "common.cuh"
#include <stdlib.h>

namespace {

constexpr int TR = 128;                  // rows per CTA (UMMA N)
constexpr int TCH = 128;                 // channels per tile (UMMA M)
constexpr int KC = 32;                   // k per chunk
constexpr int KB_BYTES = 128 * 16;       // one 8-element k-block of 128 rows / channels
constexpr int PLANE_BYTES = (KC / 8) * KB_BYTES;       // 8 KB
constexpr int CHUNK_BYTES = 3 * PLANE_BYTES;           // 24 KB
constexpr int STAGES = 4;
constexpr int NWORK = 256;               // worker threads (warps 0..7): activation staging + epilogue
constexpr int NTH = 320;                 // + warp 8 (MMA issue) + warp 9 (weight producer)
constexpr int MT_MAX = 4;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* b, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(b)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* b)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* b, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t parity)      // bounded: a protocol mistake traps
{
    uint32_t done = 0;
    int spins = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred q;\n\tmbarrier.try_wait.parity.shared::cta.b64 q, [%1], %2;\n\tselp.u32 %0, 1, 0, q;\n\t}\n"
            : "=r"(done)
            : "r"(smem_u32(b)), "r"(parity)
            : "memory");
        if (++spins > (1 << 24)) __trap();
    }
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* b)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(b))
                 : "memory");
}
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes)
{
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* b)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32])
{
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// exact 3-way split of 8 floats into three 16-byte bf16 pieces
__device__ __forceinline__ void split8(const float (&a)[8], uint4& h4, uint4& m4, uint4& l4)
{
    uint32_t hw[4], mw[4], lw[4];
#pragma unroll
    for (int h = 0; h < 4; ++h) {
        uint32_t hh = 0, mm = 0, ll = 0;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const float av = a[h * 2 + e];
            const uint32_t hb = __float_as_uint(av) & 0xFFFF0000u;
            const float r1 = av - __uint_as_float(hb);
            const uint32_t mb = __float_as_uint(r1) & 0xFFFF0000u;
            const float r2 = r1 - __uint_as_float(mb);
            const uint32_t lb = __float_as_uint(r2) & 0xFFFF0000u;
            hh |= (hb >> 16) << (16 * e);
            mm |= (mb >> 16) << (16 * e);
            ll |= (lb >> 16) << (16 * e);
        }
        hw[h] = hh; mw[h] = mm; lw[h] = ll;
    }
    h4 = make_uint4(hw[0], hw[1], hw[2], hw[3]);
    m4 = make_uint4(mw[0], mw[1], mw[2], mw[3]);
    l4 = make_uint4(lw[0], lw[1], lw[2], lw[3]);
}

// W [N][ldw] fp32 -> Wtc [MT][NKC][plane 3][k-block 4][128 channels][8 bf16]
__global__ void gemm_tc3_pack_w_kernel(const float* __restrict__ W, int ldw, int N, int K, int MT, int NKC,
                                       unsigned char* __restrict__ Wtc)
{
    const int total = MT * NKC * 4 * TCH;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int ch = i % TCH, kb = (i / TCH) % 4, kc = (i / (TCH * 4)) % NKC, mt = i / (TCH * 4 * NKC);
        const int c = mt * TCH + ch, k0 = kc * KC + kb * 8;
        float a[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) a[e] = (c < N && k0 + e < K) ? __ldg(W + (long)c * ldw + k0 + e) : 0.0f;
        uint4 h4, m4, l4;
        split8(a, h4, m4, l4);
        unsigned char* d = Wtc + ((size_t)mt * NKC + kc) * CHUNK_BYTES + (size_t)kb * KB_BYTES + ch * 16;
        *reinterpret_cast<uint4*>(d) = h4;
        *reinterpret_cast<uint4*>(d + PLANE_BYTES) = m4;
        *reinterpret_cast<uint4*>(d + 2 * PLANE_BYTES) = l4;
    }
}

struct tc3_args {
    const float* A;
    long lda, rows;
    int K, N, MT, NKC;       // MT = channel tiles handled by one CTA (blockIdx.y selects the group)
    int MT_total;            // channel tiles in the packed weights: the last group may hold fewer than MT
    const unsigned char* Wtc;
    const float* colscale;
    const float* bias;
    const float* bn_a;
    const float* bn_c;
    int act;
    float* C;
    long ldc;
    const float* rowadd;     // optional: + rowadd[(row / rows_per_add) * ld_add + channel] before BN (a per-cloud term)
    long rows_per_add, ld_add;
};

__global__ void __launch_bounds__(NTH, 1) gemm_tc3_kernel(tc3_args p)
{
    extern __shared__ __align__(1024) unsigned char smraw[];
    const int NKC = p.NKC;
    const int mt0 = blockIdx.y * p.MT;                           // first channel tile of this CTA
    // tiles of this CTA: with an odd tile count the last group has one (N = 257..384 at two tiles per CTA); a tile
    // past the last would stream weight chunks from beyond the end of the workspace
    const int MT = min(p.MT, p.MT_total - mt0);
    unsigned char* Bs = smraw;                                   // activations: 2 chunks (double buffer)
    unsigned char* Ring = Bs + 2 * CHUNK_BYTES;                  // weight chunks
    uint64_t* bars = reinterpret_cast<uint64_t*>(Ring + (size_t)STAGES * CHUNK_BYTES);
    uint64_t* full = bars;
    uint64_t* empty = full + STAGES;
    uint64_t* bfull = empty + STAGES;       // [2] activation chunk staged
    uint64_t* bempty = bfull + 2;           // [2] MMAs that read it are complete
    uint64_t* done = bempty + 2;            // all accumulators complete
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);

    const int tid = threadIdx.x, lane = tid & 31, warp = sv_warp_id();
    const long r0 = (long)blockIdx.x * TR;

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); }
        for (int t = 0; t < 2; ++t) { mbar_init(bfull + t, NWORK / 32); mbar_init(bempty + t, 1); }
        mbar_init(done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (warp == 8) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n");
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 9) {
        if (lane == 0) {
            int s = 0, t = 0;
            uint32_t ph = 0;
            for (int kc = 0; kc < NKC; ++kc)
                for (int mt = 0; mt < MT; ++mt, ++t) {
                    if (t >= STAGES) mbar_wait(empty + s, ph ^ 1u);
                    mbar_expect_tx(full + s, CHUNK_BYTES);
                    bulk_g2s(Ring + (size_t)s * CHUNK_BYTES, p.Wtc + ((size_t)(mt0 + mt) * NKC + kc) * CHUNK_BYTES, CHUNK_BYTES, full + s);
                    if (++s == STAGES) { s = 0; ph ^= 1u; }
                }
        }
    } else if (warp == 8) {
        if (lane == 0) {
            // D fp32, A/B bf16, both K-major, N = 128 rows, M = 128 channels
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TR >> 3) << 17) | ((uint32_t)(TCH >> 4) << 24);
            const uint64_t adesc0 = make_desc(smem_u32(Ring), KB_BYTES, 128);
            const uint64_t bdesc0 = make_desc(smem_u32(Bs), KB_BYTES, 128);
            constexpr uint64_t P1 = PLANE_BYTES >> 4, P2 = (2 * PLANE_BYTES) >> 4;
            int s = 0;
            uint32_t ph = 0;
            for (int kc = 0; kc < NKC; ++kc) {
                const int buf = kc & 1;
                mbar_wait(bfull + buf, (uint32_t)((kc >> 1) & 1));
                asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                const uint64_t bd = bdesc0 + (uint64_t)((buf * CHUNK_BYTES) >> 4);
                for (int mt = 0; mt < MT; ++mt) {
                    mbar_wait(full + s, ph);
                    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                    const uint64_t ad = adesc0 + (uint64_t)((s * CHUNK_BYTES) >> 4);
                    // two accumulators per channel tile: the tensor cores truncate when they accumulate, so the
                    // large h*h products get an accumulator of their own (K/16 steps instead of 6K/16) and the five
                    // small products (2^-8 and below) share the other one, where the same truncation is 2^-8 smaller
                    const uint32_t dmain = tmem_base + (uint32_t)(mt * 2 * TR);
                    const uint32_t dsmall = dmain + (uint32_t)TR;
#pragma unroll
                    for (int ks = 0; ks < KC / 16; ++ks) {
                        const uint64_t off = (uint64_t)((2 * ks * KB_BYTES) >> 4);
                        const uint32_t first = (kc == 0 && ks == 0) ? 0u : 1u;
                        // (A = weights, B = activations) small terms: h*l, l*h, m*m, h*m, m*h
                        umma_bf16(dsmall, ad + off, bd + off + P2, idesc, first);
                        umma_bf16(dsmall, ad + off + P2, bd + off, idesc, 1u);
                        umma_bf16(dsmall, ad + off + P1, bd + off + P1, idesc, 1u);
                        umma_bf16(dsmall, ad + off, bd + off + P1, idesc, 1u);
                        umma_bf16(dsmall, ad + off + P1, bd + off, idesc, 1u);
                        umma_bf16(dmain, ad + off, bd + off, idesc, first);
                    }
                    umma_commit(empty + s);
                    if (++s == STAGES) { s = 0; ph ^= 1u; }
                }
                umma_commit(bempty + buf);       // this activation buffer may be overwritten
            }
            umma_commit(done);
        }
    } else {
        // ================= workers: stage the activation chunks, then the epilogue =================
        const bool vec = ((p.lda & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.A) & 15) == 0);
        for (int kc = 0; kc < NKC; ++kc) {
            const int buf = kc & 1;
            if (kc >= 2) mbar_wait(bempty + buf, (uint32_t)(((kc >> 1) - 1) & 1));
            unsigned char* dstc = Bs + (size_t)buf * CHUNK_BYTES;
            for (int i = tid; i < TR * (KC / 8); i += NWORK) {
                const int kb = i & 3, rr = i >> 2;               // consecutive threads: consecutive 32 B of one row
                const long r = r0 + rr;
                const int k0 = kc * KC + kb * 8;
                float a[8];
                if (r < p.rows && vec && k0 + 8 <= p.K) {
                    const float4 x0 = __ldg(reinterpret_cast<const float4*>(p.A + r * p.lda + k0));
                    const float4 x1 = __ldg(reinterpret_cast<const float4*>(p.A + r * p.lda + k0 + 4));
                    a[0] = x0.x; a[1] = x0.y; a[2] = x0.z; a[3] = x0.w; a[4] = x1.x; a[5] = x1.y; a[6] = x1.z; a[7] = x1.w;
                } else {
#pragma unroll
                    for (int e = 0; e < 8; ++e) a[e] = (r < p.rows && k0 + e < p.K) ? __ldg(p.A + r * p.lda + k0 + e) : 0.0f;
                }
                uint4 h4, m4, l4;
                split8(a, h4, m4, l4);
                unsigned char* d = dstc + (size_t)kb * KB_BYTES + rr * 16;
                *reinterpret_cast<uint4*>(d) = h4;
                *reinterpret_cast<uint4*>(d + PLANE_BYTES) = m4;
                *reinterpret_cast<uint4*>(d + 2 * PLANE_BYTES) = l4;
            }
            asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");      // generic-proxy writes -> tensor-core reads
            __syncwarp();
            if (lane == 0) mbar_arrive(bfull + buf);
        }
        mbar_wait(done, 0);
        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
        const int q4 = warp & 3, half = warp >> 2;
        for (int mt = 0; mt < MT; ++mt) {
            const int c = (mt0 + mt) * TCH + q4 * 32 + lane;
            const bool cok = c < p.N;
            const float cs = (cok && p.colscale) ? p.colscale[c] : 1.0f;
            const float bi = (cok && p.bias) ? p.bias[c] : 0.0f;
            const float a1 = (cok && p.bn_a) ? p.bn_a[c] : 1.0f, c1 = (cok && p.bn_a) ? p.bn_c[c] : 0.0f;
            const uint32_t trow = tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(mt * 2 * TR + half * 64);
#pragma unroll
            for (int part = 0; part < 2; ++part) {
                float d[32], ds[32];
                tmem_ld32(trow + (uint32_t)(part * 32), d);
                tmem_ld32(trow + (uint32_t)(TR + part * 32), ds);
#pragma unroll
                for (int j = 0; j < 32; ++j) d[j] += ds[j];
                const long rb = r0 + half * 64 + part * 32;
                if (!cok) continue;
                float* op = p.C + rb * p.ldc + c;
                const int nrow = (int)min(32L, p.rows - rb);
                // row group of the first row and the first row of the next group: one division per 32 rows
                const float* addp = nullptr;
                long next_group = 0;
                if (p.rowadd) {
                    const long g = rb / p.rows_per_add;
                    addp = p.rowadd + g * p.ld_add + c;
                    next_group = (g + 1) * p.rows_per_add;
                }
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    if (j < nrow) {
                        float v = d[j] * cs + bi;            // (colscale == 1 / bias == 0 when absent)
                        if (addp) {
                            while (rb + j >= next_group) { addp += p.ld_add; next_group += p.rows_per_add; }
                            v += __ldg(addp);
                        }
                        v = v * a1 + c1;
                        op[(long)j * p.ldc] = sv_act(v, p.act);
                    }
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if (warp == 8) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"(512));
}

bool tc3_plan(const svnet_gemm_params* p, int* MT, int* NKC, size_t* wbytes, size_t* smem)
{
    const char* on = getenv("SVNET_LINEAR_TC");
    if (on && on[0] == '0') return false;
    if (p->G != 1 || p->sign_w || p->vbn || p->gate || p->c4) return false;     // c4: the float4 table is not this layout
    // The choice must not depend on the number of rows: this path rounds differently from the CUDA-core chain,
    // and a cloud's result has to be the same bits whatever batch (or batch shard) it is part of.
    if (p->M < 1 || p->K < 32 || p->K > 4096 || p->N < 32 || p->N > MT_MAX * TCH) return false;
    *NKC = (p->K + KC - 1) / KC;
    *MT = (p->N + TCH - 1) / TCH;
    *wbytes = (size_t)*MT * *NKC * CHUNK_BYTES;
    *smem = (size_t)(2 + STAGES) * CHUNK_BYTES + (2 * STAGES + 5) * 8 + 16;
    return true;
}

}  // namespace

size_t svnet_linear_tc3_workspace(const svnet_gemm_params* p)
{
    int MT, NKC;
    size_t wb, smem;
    if (!p || !tc3_plan(p, &MT, &NKC, &wb, &smem)) return 0;
    return wb;
}

// svnet_linear_tc3_dispatch with a per-row-group addend (library-internal: the full-precision part-segmentation head adds conv8's per-cloud
// term, rowadd [rows / rows_per_add][ld_add], to every point of the cloud before BN).
int svnet_linear_tc3_rowadd(const svnet_gemm_params* p, const float* rowadd, long rows_per_add, long ld_add, void* workspace,
                            size_t workspace_bytes, cudaStream_t st)
{
    int MT, NKC;
    size_t wb, smem;
    if (!workspace || !tc3_plan(p, &MT, &NKC, &wb, &smem)) return 0;
    if (workspace_bytes < wb || (reinterpret_cast<uintptr_t>(workspace) & 15)) return 0;
    gemm_tc3_pack_w_kernel<<<sv_cdiv((long)MT * NKC * 4 * TCH, 256), 256, 0, st>>>(p->W, p->ldw, p->N, p->K, MT, NKC,
                                                                                  static_cast<unsigned char*>(workspace));
    SV_CHECK_LAUNCH("svnet_linear_rows(pack)");
    tc3_args a;
    // two accumulators per channel tile -> at most two tiles per CTA (512 tensor-memory columns); with few row
    // tiles one channel tile per CTA so that more SMs take part (the activations are staged per CTA)
    const int row_tiles = sv_cdiv(p->M, TR);
    const int mt_per_cta = row_tiles >= 64 ? (MT < 2 ? MT : 2) : 1;
    a.A = p->A; a.lda = p->lda_g; a.rows = p->M; a.K = p->K; a.N = p->N; a.MT = mt_per_cta; a.MT_total = MT; a.NKC = NKC;
    a.Wtc = static_cast<const unsigned char*>(workspace);
    a.colscale = p->colscale; a.bias = p->bias; a.bn_a = p->bn_a; a.bn_c = p->bn_c; a.act = p->act;
    a.C = p->C; a.ldc = p->ldc_g;
    a.rowadd = rowadd; a.rows_per_add = rows_per_add; a.ld_add = ld_add;
    SV_CUDA(cudaFuncSetAttribute(gemm_tc3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    gemm_tc3_kernel<<<dim3(row_tiles, sv_cdiv(MT, mt_per_cta)), NTH, smem, st>>>(a);
    SV_CHECK_LAUNCH("svnet_linear_rows(tcgen05 x3)");
    return 1;
}

// Returns 1 if handled, 0 if the caller should use the CUDA-core kernel, < 0 on error.
int svnet_linear_tc3_dispatch(const svnet_gemm_params* p, void* workspace, size_t workspace_bytes, cudaStream_t st)
{
    return svnet_linear_tc3_rowadd(p, nullptr, 1, 0, workspace, workspace_bytes, st);
}
