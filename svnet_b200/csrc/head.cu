// K4 -- classification head, one CTA per cloud: up to three chained layers
//   [binarised Linear (sign-pack + XNOR/popcount) | fp Linear] (+bias) -> BatchNorm affine -> activation
// with the activations kept in shared memory (reference models/sv_dgcnn_cls.py:76-80,
// models/sv_pointnet_cls.py:76-81; Linear: models/sv_layers.py:29-53).
// Binary layers are integer-exact; small fp layers use one sequential fmaf chain per output (the
// oracle's order), large fp layers a warp-per-output shuffle reduction.
#include "common.cuh"
#include <algorithm>

namespace {

constexpr int NT = 512;

// bulk copy global -> shared behind an mbarrier (the binary layers' sign planes are prefetched at kernel start)
__device__ __forceinline__ uint32_t hsmem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void hbar_wait(uint64_t* b, uint32_t parity)      // bounded: a protocol mistake traps
{
    uint32_t done = 0;
    int spins = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred q;\n\tmbarrier.try_wait.parity.shared::cta.b64 q, [%1], %2;\n\tselp.u32 %0, 1, 0, q;\n\t}\n"
            : "=r"(done)
            : "r"(hsmem_u32(b)), "r"(parity)
            : "memory");
        if (++spins > (1 << 24)) __trap();
    }
}

__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(SV_FULL, v, o);
    return v;
}

// non-zero planes of ternary weights, one per layer (NULL: +-1)
struct head_nz {
    const uint32_t* z[3];
};

// prefetch != 0: the sign planes W1b of all binary layers (up to ~150 KB) are fetched into shared memory by cp.async.bulk
// while the input row is loaded and sign-packed (round 2: the popcount loop's dependent-latency weight loads were 40 % of
// the kernel's 31 us, the other threads' barrier waits another 30 %)
// TERN: layers with a non-zero plane (nz.z[l]) count popc(m & z) - 2 popc((a ^ w) & m & z) per word; such calls do not
// prefetch (the cls head's planes, 147 KB, would fill the prefetch area), so those layers read both planes with __ldg
template <bool TERN>
__global__ void __launch_bounds__(NT) head_kernel(svnet_head_params p, int prefetch, head_nz nz)
{
    extern __shared__ __align__(16) float sm[];
    // two ping-pong activation buffers + sign words
    int maxc = p.K0;
    for (int l = 0; l < p.nlayers; ++l) maxc = max(maxc, p.layer[l].Cout);
    float* act0 = sm;
    float* act1 = act0 + maxc;
    uint32_t* bits = reinterpret_cast<uint32_t*>(act1 + maxc);
    const int maxw = (maxc + 31) / 32;
    uint32_t* mask = bits + maxw;
    float* wst = reinterpret_cast<float*>(mask + maxw);      // staged weights of a small fp layer, row stride K + 1
    __shared__ int nvalid_s;
    __shared__ __align__(8) uint64_t wbar;

    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = sv_warp_id();
    // prefetched sign planes live behind the staging area of the fp layer
    size_t wst_floats = 0;
    {
        int Kl = p.K0;
        for (int l = 0; l < p.nlayers; ++l) {
            const svnet_head_layer& L = p.layer[l];
            if (!L.W1b && (long)Kl * L.Cout <= 32768) wst_floats = max(wst_floats, (size_t)L.Cout * (Kl + 1));
            Kl = L.Cout;
        }
    }
    uint32_t* wpre = reinterpret_cast<uint32_t*>(wst + ((wst_floats + 3) & ~(size_t)3));
    if (prefetch && tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(hsmem_u32(&wbar)));
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
        uint32_t total = 0;
        int Kl = p.K0;
        for (int l = 0; l < p.nlayers; ++l) {
            if (p.layer[l].W1b) total += (uint32_t)((Kl + 31) / 32) * p.layer[l].Cout * 4u;
            Kl = p.layer[l].Cout;
        }
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(hsmem_u32(&wbar)), "r"(total) : "memory");
        uint32_t off = 0;
        Kl = p.K0;
        for (int l = 0; l < p.nlayers; ++l) {
            if (p.layer[l].W1b) {
                const uint32_t bytes = (uint32_t)((Kl + 31) / 32) * p.layer[l].Cout * 4u;
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                                 hsmem_u32(wpre) + off),
                             "l"(p.layer[l].W1b), "r"(bytes), "r"(hsmem_u32(&wbar))
                             : "memory");
                off += bytes;
            }
            Kl = p.layer[l].Cout;
        }
    }
    for (int c = tid; c < p.K0; c += NT) act0[c] = p.x[(long)b * p.ldx + c];
    __syncthreads();
    uint32_t pre_off = 0;         // words of the prefetch area consumed by earlier binary layers
    bool pre_ready = false;
    float* cur = act0;
    float* nxt = act1;
    int K = p.K0;
    for (int l = 0; l < p.nlayers; ++l) {
        const svnet_head_layer& L = p.layer[l];
        const int Cout = L.Cout;
        if (L.W1b) {
            // sign(x + beta) -> words (sv_layers.py:36-39)
            const int Kw = (K + 31) / 32;
            if (tid == 0) nvalid_s = 0;
            __syncthreads();
            for (int w = warp; w < Kw; w += NT / 32) {
                const int c = w * 32 + lane;
                const float t = (c < K) ? __fadd_rn(cur[c], L.beta[c]) : 0.0f;
                const unsigned pos = __ballot_sync(SV_FULL, t > 0.0f);
                const unsigned nz = __ballot_sync(SV_FULL, t != 0.0f);
                if (lane == 0) { bits[w] = pos; mask[w] = nz; atomicAdd(&nvalid_s, __popc(nz)); }
            }
            __syncthreads();
            const int nvalid = nvalid_s;
            if (prefetch && !pre_ready) {
                hbar_wait(&wbar, 0);
                pre_ready = true;
            }
            const uint32_t* wsm = wpre + pre_off;
            pre_off += (uint32_t)Kw * Cout;
            const uint32_t* Z = TERN ? nz.z[l] : nullptr;
            for (int o = tid; o < Cout; o += NT) {
                if (TERN && Z) {
                    int dot = 0;
#pragma unroll 16
                    for (int w = 0; w < Kw; ++w) {
                        const uint32_t mz = mask[w] & __ldg(Z + (long)w * Cout + o);
                        dot += __popc(mz) - 2 * __popc((bits[w] ^ __ldg(L.W1b + (long)w * Cout + o)) & mz);
                    }
                    float y = __fmul_rn((float)dot, L.scale ? L.scale[o] : 1.0f);
                    if (L.bias) y = __fadd_rn(y, L.bias[o]);
                    if (L.bn_a) y = __fadd_rn(__fmul_rn(y, L.bn_a[o]), L.bn_c[o]);
                    nxt[o] = sv_act(y, L.act);
                    continue;
                }
                int mism = 0;
                if (prefetch) {
#pragma unroll 8
                    for (int w = 0; w < Kw; ++w) mism += __popc((bits[w] ^ wsm[(size_t)w * Cout + o]) & mask[w]);
                } else {
#pragma unroll 32
                    for (int w = 0; w < Kw; ++w) mism += __popc((bits[w] ^ __ldg(L.W1b + (long)w * Cout + o)) & mask[w]);
                }
                float y = __fmul_rn((float)(nvalid - 2 * mism), L.scale ? L.scale[o] : 1.0f);
                if (L.bias) y = __fadd_rn(y, L.bias[o]);
                if (L.bn_a) y = __fadd_rn(__fmul_rn(y, L.bn_a[o]), L.bn_c[o]);
                nxt[o] = sv_act(y, L.act);
            }
        } else if ((long)K * Cout <= 32768) {
            // small fp layer: one sequential fmaf chain per output (the oracle's order).  The weights are
            // first staged in shared memory by all threads (coalesced, every load in flight); the chains
            // then run from shared memory instead of Cout serial walks over global rows.
            const int ldw = K + 1;                      // odd stride: the Cout chains hit different banks
            for (int i = tid; i < K * Cout; i += NT) {
                const int o = i / K, c = i - o * K;
                float wv = __ldg(L.W + i);
                if (L.sign_w) wv = (wv > 0.0f) ? 1.0f : ((wv < 0.0f) ? -1.0f : 0.0f);
                wst[o * ldw + c] = wv;
            }
            __syncthreads();
            for (int o = tid; o < Cout; o += NT) {
                const float* w = wst + o * ldw;
                float acc = 0.0f;
#pragma unroll 8
                for (int c = 0; c < K; ++c) acc = __fmaf_rn(cur[c], w[c], acc);
                if (L.scale) acc = __fmul_rn(acc, L.scale[o]);
                if (L.bias) acc = __fadd_rn(acc, L.bias[o]);
                if (L.bn_a) acc = __fadd_rn(__fmul_rn(acc, L.bn_a[o]), L.bn_c[o]);
                nxt[o] = sv_act(acc, L.act);
            }
        } else {
            for (int o = warp; o < Cout; o += NT / 32) {
                const float* w = L.W + (long)o * K;
                float acc = 0.0f;
                for (int c = lane; c < K; c += 32) {
                    float wv = __ldg(w + c);
                    if (L.sign_w) wv = (wv > 0.0f) ? 1.0f : ((wv < 0.0f) ? -1.0f : 0.0f);
                    acc = fmaf(cur[c], wv, acc);
                }
                acc = warp_sum(acc);
                if (lane == 0) {
                    if (L.scale) acc *= L.scale[o];
                    if (L.bias) acc += L.bias[o];
                    if (L.bn_a) acc = acc * L.bn_a[o] + L.bn_c[o];
                    nxt[o] = sv_act(acc, L.act);
                }
            }
        }
        __syncthreads();
        float* t = cur; cur = nxt; nxt = t;
        K = Cout;
    }
    for (int c = tid; c < K; c += NT) p.out[(long)b * p.ldo + c] = cur[c];
}

}  // namespace

extern "C" int svnet_head_fwd_nz(const svnet_head_params* p, const uint32_t* const W1nz[3], void* stream)
{
    SV_REQUIRE(p && p->x && p->out, "svnet_head_fwd: null pointer");
    SV_REQUIRE(p->nlayers >= 1 && p->nlayers <= 3 && p->K0 >= 1 && p->B >= 0, "svnet_head_fwd: bad shape");
    int maxc = p->K0, K = p->K0;
    size_t wstage = 0;
    for (int l = 0; l < p->nlayers; ++l) {
        const svnet_head_layer& L = p->layer[l];
        if (!L.W1b && (long)K * L.Cout <= 32768) wstage = std::max(wstage, (size_t)L.Cout * (K + 1));
        SV_REQUIRE(L.Cout >= 1, "svnet_head_fwd: layer %d Cout", l);
        SV_REQUIRE(L.W1b ? (L.beta != nullptr) : (L.W != nullptr), "svnet_head_fwd: layer %d needs W1b+beta or W", l);
        SV_REQUIRE((L.bn_a == nullptr) == (L.bn_c == nullptr), "svnet_head_fwd: layer %d bn_a/bn_c", l);
        maxc = L.Cout > maxc ? L.Cout : maxc;
        K = L.Cout;
    }
    SV_REQUIRE(p->ldx >= p->K0 && p->ldo >= K, "svnet_head_fwd: ldx/ldo too small");
    if (p->B == 0) return SVNET_OK;
    size_t smem = sizeof(float) * ((size_t)2 * maxc + 2 * ((maxc + 31) / 32) + ((wstage + 3) & ~(size_t)3));
    SV_REQUIRE(smem <= 200 * 1024, "svnet_head_fwd: layer too wide");
    // sign planes of the binary layers prefetched into shared memory when they fit and are 16-byte granular
    size_t pre = 0;
    bool pre_ok = true;
    {
        int Kl = p->K0;
        for (int l = 0; l < p->nlayers; ++l) {
            const svnet_head_layer& L = p->layer[l];
            if (L.W1b) {
                const size_t bytes = (size_t)((Kl + 31) / 32) * L.Cout * 4;
                pre += bytes;
                if ((bytes & 15) || (reinterpret_cast<uintptr_t>(L.W1b) & 15)) pre_ok = false;
            }
            Kl = L.Cout;
        }
    }
    head_nz nz = {};
    bool tern = false;
    for (int l = 0; l < p->nlayers && W1nz; ++l) {
        SV_REQUIRE(!W1nz[l] || p->layer[l].W1b, "svnet_head_fwd_nz: layer %d has a non-zero plane but no W1b", l);
        nz.z[l] = W1nz[l];
        tern = tern || W1nz[l] != nullptr;
    }
    if (tern) {
        if (smem > 48 * 1024) SV_CUDA(cudaFuncSetAttribute(head_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        head_kernel<true><<<p->B, NT, smem, sv_stream(stream)>>>(*p, 0, nz);
        SV_CHECK_LAUNCH("svnet_head_fwd_nz");
        return SVNET_OK;
    }
    const int prefetch = (pre > 0 && pre_ok && (smem & 15) == 0 && smem + pre <= 220 * 1024) ? 1 : 0;
    if (prefetch) smem += pre;
    if (smem > 48 * 1024) SV_CUDA(cudaFuncSetAttribute(head_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    head_kernel<false><<<p->B, NT, smem, sv_stream(stream)>>>(*p, prefetch, nz);
    SV_CHECK_LAUNCH("svnet_head_fwd");
    return SVNET_OK;
}

extern "C" int svnet_head_fwd(const svnet_head_params* p, void* stream)
{
    return svnet_head_fwd_nz(p, nullptr, stream);
}
