// Binarised Linear / Conv1d over packed rows on the tcgen05 tensor cores
// (reference models/sv_layers.py:29-53, :64-78: y = sign(x + beta) . sign(W)^T * scale).
// Same contract as rows.cu:binlinear_rows_kernel -- the dot product of ternary activations
// {-1, 0, +1} (sign / zero-mask words) with +-1 (or, with a non-zero plane, ternary) weights is an exact integer --
// but the products run as
// bf16 UMMAs with fp32 accumulation in tensor memory: every operand value is exactly representable and
// every partial sum is an integer below 2^24, so the result is bit-identical to the XNOR/popcount kernel
// (which is bound by the quarter-rate POPC pipe).
//
//   D[c][r] = sum_k  Wsign[c][k] * t[r][k]            M = 128 output channels, N = 128 rows, K = 16 per UMMA
//   * weights   : expanded once per call into the canonical K-major bf16 layout (chunks of 64 k:
//                 [k-block 8][128 channels][8 bf16] = 16 KB), streamed through an mbarrier ring with
//                 cp.async.bulk
//   * activations: the CTA's 128 rows are expanded from their sign / mask words into the same layout
//                 in shared memory (resident for all channel tiles)
//   * accumulators: 128 x 128 fp32, double buffered in tensor memory; the epilogue (lane = channel, so
//                 the stores of a warp are contiguous) applies scale / bias / BN / activation exactly as the
//                 popcount kernel does.
#include "common.cuh"
#include <stdlib.h>

namespace {

constexpr int TR = 128;                 // rows per CTA (UMMA N)
constexpr int TCH = 128;                // channels per tile (UMMA M)
constexpr int KC = 64;                  // k per chunk
constexpr int KB_BYTES = 128 * 16;      // one 8-element k-block of 128 rows / channels
constexpr int CHUNK_BYTES = (KC / 8) * KB_BYTES;     // 16 KB
constexpr int STAGES = 4;
constexpr int NEPI = 256;               // epilogue threads (warps 0..7)
constexpr int NTH = 320;                // + warp 8 (MMA issue) + warp 9 (producer)
constexpr int KPAD_MAX = 640;

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

// 8 ternary values (bit b of `pos` / `nz`) -> 8 bf16 in one uint4
__device__ __forceinline__ uint4 expand8(uint32_t pos, uint32_t nz)
{
    uint32_t w[4];
#pragma unroll
    for (int h = 0; h < 4; ++h) {
        uint32_t v = 0;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int b = 2 * h + e;
            const uint32_t val = ((nz >> b) & 1u) ? (((pos >> b) & 1u) ? 0x3F80u : 0xBF80u) : 0u;
            v |= val << (16 * e);
        }
        w[h] = v;
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

// sign-bit words W1b [Kw][Cout] -> Wtc [MT][NKC][8 k-blocks][128 channels][8 bf16] (+-1, zero padded).
// TERN: W1nz [Kw][Cout] is the non-zero plane of ternary weights; a zero weight is an exact bf16 0.
template <bool TERN>
__global__ void binlinear_pack_w_kernel(const uint32_t* __restrict__ W1b, int Kw, int K, int Cout, int MT, int NKC,
                                        uint4* __restrict__ Wtc, const uint32_t* __restrict__ W1nz)
{
    const int total = MT * NKC * 8 * TCH;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int ch = i % TCH, kb = (i / TCH) % 8, kc = (i / (TCH * 8)) % NKC, mt = i / (TCH * 8 * NKC);
        const int c = mt * TCH + ch, k0 = kc * KC + kb * 8;
        uint32_t pos = 0, nz = 0;
        if (c < Cout && k0 < K) {
            const uint32_t word = __ldg(W1b + (long)(k0 >> 5) * Cout + c);
            pos = (word >> (k0 & 31)) & 0xFFu;
            const int nvalid = min(8, K - k0);
            nz = (1u << nvalid) - 1u;           // without a plane every real weight is +-1
            if (TERN) nz &= (__ldg(W1nz + (long)(k0 >> 5) * Cout + c) >> (k0 & 31)) & 0xFFu;
        }
        Wtc[i] = expand8(pos, nz);
    }
}

struct bl_args {
    const uint32_t* bits;
    const uint32_t* mask;
    long rows;
    int Kw, Cout, MT, NKC;
    const unsigned char* Wtc;
    const float* scale;
    const float* bias;
    const float* bn_a;
    const float* bn_c;
    int act;
    const int32_t* cloud_dot;
    long rows_per_cloud;
    float* out;
    int ldo;
    int32_t* out_i32;
    float* pool_partial;     // MODE 2: [tile][half][max | sum][Cout]
};

// MODE 0: generic epilogue; 1: scale -> BN -> LeakyReLU stores on full tiles; 2: the same values reduced to
// per-tile column max / sum partials (global pooling fused, nothing else is written)
template <int MODE>
__global__ void __launch_bounds__(NTH, 1) binlinear_tc_kernel(bl_args p)
{
    extern __shared__ __align__(1024) unsigned char smraw[];
    const int NKC = p.NKC, MT = p.MT;
    unsigned char* Bs = smraw;                                   // activations: NKC chunks, resident
    unsigned char* Ring = Bs + (size_t)NKC * CHUNK_BYTES;        // weight chunks
    uint64_t* bars = reinterpret_cast<uint64_t*>(Ring + (size_t)STAGES * CHUNK_BYTES);
    uint64_t* full = bars;
    uint64_t* empty = full + STAGES;
    uint64_t* tfull = empty + STAGES;
    uint64_t* tempty = tfull + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

    const int tid = threadIdx.x, lane = tid & 31, warp = sv_warp_id();
    const long r0 = (long)blockIdx.x * TR;

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); }
        for (int t = 0; t < 2; ++t) { mbar_init(tfull + t, 1); mbar_init(tempty + t, NEPI / 32); }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (warp == 8) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)), "r"(2 * TR));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n");
    }
    // ---- activations of this CTA's rows: sign / mask words -> bf16 {-1, 0, +1}, canonical layout ----
    for (int i = tid; i < TR * NKC * 2; i += NTH) {
        const int rr = i % TR, w = i / TR;                       // w = 32-bit word index (two words per 64-k chunk)
        const long r = r0 + rr;
        uint32_t pos = 0, nz = 0;
        if (r < p.rows && w < p.Kw) { pos = __ldg(p.bits + r * p.Kw + w); nz = __ldg(p.mask + r * p.Kw + w); }
        unsigned char* dst = Bs + (size_t)(w >> 1) * CHUNK_BYTES + (size_t)((w & 1) * 4) * KB_BYTES + rr * 16;
#pragma unroll
        for (int q = 0; q < 4; ++q)
            *reinterpret_cast<uint4*>(dst + q * KB_BYTES) = expand8(pos >> (8 * q), nz >> (8 * q));
    }
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");      // generic-proxy writes -> tensor-core reads
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 9) {
        if (lane == 0) {
            int s = 0;
            uint32_t ph = 0;
            int t = 0;
            for (int mt = 0; mt < MT; ++mt)
                for (int kc = 0; kc < NKC; ++kc, ++t) {
                    if (t >= STAGES) mbar_wait(empty + s, ph ^ 1u);
                    mbar_expect_tx(full + s, CHUNK_BYTES);
                    bulk_g2s(Ring + (size_t)s * CHUNK_BYTES, p.Wtc + ((size_t)mt * NKC + kc) * CHUNK_BYTES, CHUNK_BYTES, full + s);
                    if (++s == STAGES) { s = 0; ph ^= 1u; }
                }
        }
    } else if (warp == 8) {
        if (lane == 0) {
            // D fp32, A/B bf16, both K-major, N = 128 rows, M = 128 channels
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TR >> 3) << 17) | ((uint32_t)(TCH >> 4) << 24);
            const uint64_t adesc0 = make_desc(smem_u32(Ring), KB_BYTES, 128);
            const uint64_t bdesc0 = make_desc(smem_u32(Bs), KB_BYTES, 128);
            int s = 0;
            uint32_t ph = 0;
            for (int mt = 0; mt < MT; ++mt) {
                const int buf = mt & 1;
                if (mt >= 2) mbar_wait(tempty + buf, (uint32_t)(((mt >> 1) - 1) & 1));
                asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                const uint32_t dcol = tmem_base + (uint32_t)(buf * TR);
                for (int kc = 0; kc < NKC; ++kc) {
                    mbar_wait(full + s, ph);
                    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                    const uint64_t ad = adesc0 + (uint64_t)((s * CHUNK_BYTES) >> 4);
                    const uint64_t bd = bdesc0 + (uint64_t)((kc * CHUNK_BYTES) >> 4);
#pragma unroll
                    for (int ks = 0; ks < KC / 16; ++ks) {
                        const uint64_t off = (uint64_t)((2 * ks * KB_BYTES) >> 4);
                        umma_bf16(dcol, ad + off, bd + off, idesc, (kc == 0 && ks == 0) ? 0u : 1u);
                    }
                    umma_commit(empty + s);
                    if (++s == STAGES) { s = 0; ph ^= 1u; }
                }
                umma_commit(tfull + buf);
            }
        }
    } else {
        // ================= epilogue: warps 0..7, lane quarter = warp & 3 (channels), column half = warp >> 2 (rows) =========
        const int q4 = warp & 3, half = warp >> 2;
        for (int mt = 0; mt < MT; ++mt) {
            const int buf = mt & 1;
            const int c = mt * TCH + q4 * 32 + lane;
            const bool cok = c < p.Cout;
            const float sc = (cok && p.scale) ? p.scale[c] : 1.0f;
            const float bi = (cok && p.bias) ? p.bias[c] : 0.0f;
            const float a1 = (cok && p.bn_a) ? p.bn_a[c] : 0.0f, c1 = (cok && p.bn_a) ? p.bn_c[c] : 0.0f;
            mbar_wait(tfull + buf, (uint32_t)((mt >> 1) & 1));
            asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
            const uint32_t trow = tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(buf * TR + half * 64);
            float vmax = -INFINITY, vsum = 0.0f;
#pragma unroll
            for (int part = 0; part < 2; ++part) {
                float d[32];
                tmem_ld32(trow + (uint32_t)(part * 32), d);
                if (part == 1) {
                    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
                    __syncwarp();
                    if (lane == 0) mbar_arrive(tempty + buf);
                }
                const long rb = r0 + half * 64 + part * 32;
                if (MODE == 0) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const long r = rb + j;
                        if (!cok || r >= p.rows) continue;
                        int dot = __float2int_rn(d[j]);
                        if (p.cloud_dot) dot += p.cloud_dot[(r / p.rows_per_cloud) * p.Cout + c];
                        if (p.out_i32) { p.out_i32[r * p.Cout + c] = dot; continue; }
                        float y = __fmul_rn((float)dot, sc);
                        if (p.bias) y = __fadd_rn(y, bi);
                        if (p.bn_a) y = __fadd_rn(__fmul_rn(y, a1), c1);
                        p.out[r * p.ldo + c] = sv_act(y, p.act);
                    }
                } else if (MODE == 2) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        float y = __fadd_rn(__fmul_rn(__fmul_rn(d[j], sc), a1), c1);
                        y = y > 0.0f ? y : __fmul_rn(0.2f, y);
                        vmax = fmaxf(vmax, y);
                        vsum += y;
                    }
                } else {
                    // scale -> BN -> LeakyReLU, full tile: no flags, no bounds checks inside the unrolled loop.
                    // d[j] already holds the exact integer as a float (what (float)dot would give).
                    if (cok) {
                        float* op = p.out + rb * p.ldo + c;
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            float y = __fadd_rn(__fmul_rn(__fmul_rn(d[j], sc), a1), c1);
                            y = y > 0.0f ? y : __fmul_rn(0.2f, y);
                            op[(long)j * p.ldo] = y;
                        }
                    }
                }
            }
            if (MODE == 2 && cok) {
                float* pp = p.pool_partial + ((size_t)blockIdx.x * 2 + half) * 2 * p.Cout;
                pp[c] = vmax;
                pp[p.Cout + c] = vsum;
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if (warp == 8) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"(2 * TR));
}

bool bl_plan(long rows, int K, int Cout, int* MT, int* NKC, size_t* wbytes, size_t* smem)
{
    const char* on = getenv("SVNET_BINLINEAR_TC");
    if (on && on[0] == '0') return false;
    const int Kpad = (K + KC - 1) / KC * KC;
    if (rows < 2048 || K < 64 || Kpad > KPAD_MAX || Cout < 32) return false;
    *NKC = Kpad / KC;
    *MT = (Cout + TCH - 1) / TCH;
    *wbytes = (size_t)*MT * *NKC * CHUNK_BYTES;
    *smem = (size_t)(*NKC + STAGES) * CHUNK_BYTES + (2 * STAGES + 4) * 8 + 16;
    return *smem <= 227 * 1024;
}

// weights -> bf16 operand chunks in the workspace (+-1, or ternary with a non-zero plane)
void bl_pack_w(const uint32_t* W1b, const uint32_t* W1nz, int Kw, int K, int Cout, int MT, int NKC, void* workspace, cudaStream_t st)
{
    const int grid = sv_cdiv((long)MT * NKC * 8 * TCH, 256);
    if (W1nz)
        binlinear_pack_w_kernel<true><<<grid, 256, 0, st>>>(W1b, Kw, K, Cout, MT, NKC, static_cast<uint4*>(workspace), W1nz);
    else
        binlinear_pack_w_kernel<false><<<grid, 256, 0, st>>>(W1b, Kw, K, Cout, MT, NKC, static_cast<uint4*>(workspace), nullptr);
}

}  // namespace


extern "C" size_t svnet_binlinear_workspace_bytes(long rows, int K, int Cout)
{
    int MT, NKC;
    size_t wb, smem;
    if (!bl_plan(rows, K, Cout, &MT, &NKC, &wb, &smem)) return 0;
    return wb;
}

// Returns 1 if handled, 0 if the caller should use the popcount kernel, < 0 on error.
int svnet_binlinear_tc_dispatch(const uint32_t* bits, const uint32_t* mask, long rows, int K, const uint32_t* W1b,
                                const uint32_t* W1nz, int Cout, const float* scale, const float* bias, const float* bn_a,
                                const float* bn_c, int act, const int32_t* cloud_dot, long rows_per_cloud, float* out, int ldo,
                                int32_t* out_i32, void* workspace, size_t workspace_bytes, cudaStream_t st)
{
    int MT, NKC;
    size_t wb, smem;
    if (!workspace || !bl_plan(rows, K, Cout, &MT, &NKC, &wb, &smem)) return 0;
    if (workspace_bytes < wb || (reinterpret_cast<uintptr_t>(workspace) & 15)) return 0;
    // lean epilogue when the call is the common "scale, BN, LeakyReLU on full tiles" shape (2x faster than the
    // popcount kernel at conv5's shape); the generic epilogue is slower than the popcount kernel, so other
    // calls stay there unless SVNET_BINLINEAR_TC=2 forces the tensor-core path (parity tests)
    const bool lean = !cloud_dot && !out_i32 && !bias && bn_a && act == SVNET_ACT_LEAKY && scale && (rows % TR) == 0;
    {
        const char* on = getenv("SVNET_BINLINEAR_TC");
        if (!lean && !(on && on[0] == '2')) return 0;
    }
    const int Kw = (K + 31) / 32;
    bl_pack_w(W1b, W1nz, Kw, K, Cout, MT, NKC, workspace, st);
    SV_CHECK_LAUNCH("svnet_binlinear_rows(pack)");
    bl_args a;
    a.bits = bits; a.mask = mask; a.rows = rows; a.Kw = Kw; a.Cout = Cout; a.MT = MT; a.NKC = NKC;
    a.Wtc = static_cast<const unsigned char*>(workspace);
    a.scale = scale; a.bias = bias; a.bn_a = bn_a; a.bn_c = bn_c; a.act = act;
    a.cloud_dot = cloud_dot; a.rows_per_cloud = rows_per_cloud; a.out = out; a.ldo = ldo; a.out_i32 = out_i32;
    a.pool_partial = nullptr;
    if (lean) {
        SV_CUDA(cudaFuncSetAttribute(binlinear_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        binlinear_tc_kernel<1><<<sv_cdiv(rows, TR), NTH, smem, st>>>(a);
    } else {
        SV_CUDA(cudaFuncSetAttribute(binlinear_tc_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        binlinear_tc_kernel<0><<<sv_cdiv(rows, TR), NTH, smem, st>>>(a);
    }
    SV_CHECK_LAUNCH("svnet_binlinear_rows(tcgen05)");
    return 1;
}

// ---- binarised Linear + BN + LeakyReLU fused with the global max / mean pooling over the rows of a cloud
//      (SV_DGCNN_CLS: conv5's scalar output is only ever pooled, sv_dgcnn_cls.py:68-74) ----
namespace {
__global__ void binlinear_pool_reduce_kernel(const float* __restrict__ partial, int tiles_per_cloud, int Cout, long rows_per_cloud,
                                             float* __restrict__ max_out, float* __restrict__ mean_out, int ldo)
{
    const int b = blockIdx.y;
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= Cout) return;
    const float* p = partial + (size_t)b * tiles_per_cloud * 2 * 2 * Cout;
    float mx = -INFINITY, sm = 0.0f;
    for (int t = 0; t < tiles_per_cloud * 2; ++t) {        // fixed order: tile, then half
        mx = fmaxf(mx, p[(size_t)t * 2 * Cout + c]);
        sm += p[(size_t)t * 2 * Cout + Cout + c];
    }
    if (max_out) max_out[(size_t)b * ldo + c] = mx;
    if (mean_out) mean_out[(size_t)b * ldo + c] = sm / (float)rows_per_cloud;
}
}  // namespace

extern "C" size_t svnet_binlinear_pool_workspace_bytes(long rows, int K, int Cout, long rows_per_cloud)
{
    int MT, NKC;
    size_t wb, smem;
    if (rows_per_cloud < TR || (rows_per_cloud % TR) != 0 || (rows % rows_per_cloud) != 0) return 0;
    if (!bl_plan(rows, K, Cout, &MT, &NKC, &wb, &smem)) return 0;
    return wb + (size_t)(rows / TR) * 2 * 2 * Cout * sizeof(float);
}

extern "C" int svnet_binlinear_pool_nz(const uint32_t* bits, const uint32_t* mask, long rows, int K, const uint32_t* W1b,
                                       const uint32_t* W1nz, int Cout, const float* scale, const float* bn_a, const float* bn_c,
                                       long rows_per_cloud, float* max_out, float* mean_out, int ldo, void* workspace,
                                       size_t workspace_bytes, void* stream)
{
    SV_REQUIRE(bits && mask && W1b && scale && bn_a && bn_c, "svnet_binlinear_pool_ws: null pointer");
    SV_REQUIRE(max_out || mean_out, "svnet_binlinear_pool_ws: no output requested");
    SV_REQUIRE(ldo >= Cout, "svnet_binlinear_pool_ws: ldo too small");
    const size_t need = svnet_binlinear_pool_workspace_bytes(rows, K, Cout, rows_per_cloud);
    SV_REQUIRE(need > 0, "svnet_binlinear_pool_ws: shape not covered (rows %ld, K %d, rows_per_cloud %ld)", rows, K, rows_per_cloud);
    SV_REQUIRE(workspace && workspace_bytes >= need && !(reinterpret_cast<uintptr_t>(workspace) & 15),
               "svnet_binlinear_pool_ws: workspace too small or misaligned");
    int MT, NKC;
    size_t wb, smem;
    bl_plan(rows, K, Cout, &MT, &NKC, &wb, &smem);
    cudaStream_t st = sv_stream(stream);
    const int Kw = (K + 31) / 32;
    bl_pack_w(W1b, W1nz, Kw, K, Cout, MT, NKC, workspace, st);
    SV_CHECK_LAUNCH("svnet_binlinear_pool_ws(pack)");
    bl_args a;
    a.bits = bits; a.mask = mask; a.rows = rows; a.Kw = Kw; a.Cout = Cout; a.MT = MT; a.NKC = NKC;
    a.Wtc = static_cast<const unsigned char*>(workspace);
    a.scale = scale; a.bias = nullptr; a.bn_a = bn_a; a.bn_c = bn_c; a.act = SVNET_ACT_LEAKY;
    a.cloud_dot = nullptr; a.rows_per_cloud = rows_per_cloud; a.out = nullptr; a.ldo = 0; a.out_i32 = nullptr;
    a.pool_partial = reinterpret_cast<float*>(static_cast<unsigned char*>(workspace) + wb);
    SV_CUDA(cudaFuncSetAttribute(binlinear_tc_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    binlinear_tc_kernel<2><<<sv_cdiv(rows, TR), NTH, smem, st>>>(a);
    SV_CHECK_LAUNCH("svnet_binlinear_pool_ws(tcgen05)");
    const int B = (int)(rows / rows_per_cloud);
    binlinear_pool_reduce_kernel<<<dim3(sv_cdiv(Cout, 128), B), 128, 0, st>>>(a.pool_partial, (int)(rows_per_cloud / TR), Cout,
                                                                             rows_per_cloud, max_out, mean_out, ldo);
    SV_CHECK_LAUNCH("svnet_binlinear_pool_ws(reduce)");
    return SVNET_OK;
}

extern "C" int svnet_binlinear_pool_ws(const uint32_t* bits, const uint32_t* mask, long rows, int K, const uint32_t* W1b,
                                       int Cout, const float* scale, const float* bn_a, const float* bn_c,
                                       long rows_per_cloud, float* max_out, float* mean_out, int ldo, void* workspace,
                                       size_t workspace_bytes, void* stream)
{
    return svnet_binlinear_pool_nz(bits, mask, rows, K, W1b, nullptr, Cout, scale, bn_a, bn_c, rows_per_cloud, max_out,
                                   mean_out, ldo, workspace, workspace_bytes, stream);
}
