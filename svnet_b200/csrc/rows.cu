// Per-row building blocks used by conv5, the PointNet per-point blocks, the heads and the
// module-level API: u = [s | v2s(v)] construction with optional sign packing, and the
// XNOR/popcount linear over packed rows.
// Reference: models/sv_layers.py:29-53 (Linear), :64-78 (Conv1d), :111-129 (Vector2Scalar),
//            :185-190 (SVBlock scalar branch), :206-220 (SVFuse).
#include "common.cuh"

namespace {

constexpr int PW = 4;  // warps per CTA in rows_prep

// One warp handles up to three rows at a time: 27 lanes compute the 3x3 frames z (sequential fmaf
// chain over channels == oracle order), then all lanes build u lane-per-channel.
__global__ void __launch_bounds__(PW * 32) rows_prep_kernel(svnet_view in, long rows, const float* __restrict__ Wz,
                                                            const float* __restrict__ zscale,
                                                            const float* __restrict__ z_in,
                                                            const float* __restrict__ beta, float* __restrict__ u_out,
                                                            int ldu, float* __restrict__ z_out,
                                                            uint32_t* __restrict__ bits, uint32_t* __restrict__ mask,
                                                            int32_t* __restrict__ nvalid)
{
    __shared__ float zb_all[PW][28];
    const int lane = threadIdx.x & 31, warp = sv_warp_id();
    float* zb = zb_all[warp];
    const int Cs = in.Cs, Cv = in.Cv;
    const int K = Cs + 3 * Cv, Kw = (K + 31) / 32;
    const long ngroups = (rows + 2) / 3;
    for (long grp = (long)blockIdx.x * PW + warp; grp < ngroups; grp += (long)gridDim.x * PW) {
        const long r0 = grp * 3;
        const int ng = (int)min(3L, rows - r0);
        if (Cv > 0) {
            if (lane < ng * 9) {
                const int g = lane / 9, xm = lane - g * 9, x = xm / 3, m = xm - x * 3;
                float acc = 0.0f;
                if (z_in) {
                    acc = __ldg(z_in + (r0 + g) * 9 + xm);
                } else {
                    const float* vp = in.v + (r0 + g) * in.ldv + x * in.xs;
                    const float* wz = Wz + m * Cv;
#pragma unroll 4
                    for (int c = 0; c < Cv; ++c) acc = __fmaf_rn(__ldg(vp + c), __ldg(wz + c), acc);
                    if (zscale) acc = __fmul_rn(acc, __ldg(zscale + m));
                }
                zb[lane] = acc;
                if (z_out) z_out[(r0 + g) * 9 + xm] = acc;
            }
            __syncwarp();
        }
        for (int g = 0; g < ng; ++g) {
            const long r = r0 + g;
            const float* z = zb + g * 9;
            int nval = 0;
            for (int wd = 0; wd < Kw; ++wd) {
                const int kk = wd * 32 + lane;
                float u = 0.0f;
                if (kk < Cs) u = __ldg(in.s + r * in.lds + kk);
                else if (kk < K) {
                    const int t = kk - Cs, dd = t / 3, m = t - dd * 3;
                    const float* vp = in.v + r * in.ldv + dd;
                    float q = __fmul_rn(__ldg(vp), z[m]);
                    q = __fmaf_rn(__ldg(vp + in.xs), z[3 + m], q);
                    q = __fmaf_rn(__ldg(vp + 2 * in.xs), z[6 + m], q);
                    u = q;
                }
                if (u_out && kk < K) u_out[r * ldu + kk] = u;
                if (bits) {
                    const float t = (kk < K) ? __fadd_rn(u, __ldg(beta + kk)) : 0.0f;
                    const unsigned pos = __ballot_sync(SV_FULL, t > 0.0f);
                    const unsigned nz = __ballot_sync(SV_FULL, t != 0.0f);
                    nval += __popc(nz);
                    if (lane == 0) { bits[r * Kw + wd] = pos; mask[r * Kw + wd] = nz; }
                }
            }
            if (bits && lane == 0) nvalid[r] = nval;
        }
        __syncwarp();
    }
}

// Staged variant: the three rows of a warp's group are first copied to shared memory with cp.async
// (every load of the group in flight at once; the direct version above waits on ~Cv dependent L1/L2
// round trips per row), Wz is CTA-shared; the arithmetic and its order are identical.
__device__ __forceinline__ void rp_cp_async4(void* smem_dst, const void* gsrc)
{
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(d), "l"(gsrc));
}

__global__ void __launch_bounds__(PW * 32) rows_prep_staged_kernel(svnet_view in, long rows, const float* __restrict__ Wz,
                                                                   const float* __restrict__ zscale,
                                                                   const float* __restrict__ beta, float* __restrict__ u_out,
                                                                   int ldu, float* __restrict__ z_out,
                                                                   uint32_t* __restrict__ bits, uint32_t* __restrict__ mask,
                                                                   int32_t* __restrict__ nvalid)
{
    extern __shared__ float rp_smem[];
    const int lane = threadIdx.x & 31, warp = sv_warp_id();
    const int Cs = in.Cs, Cv = in.Cv;
    const int K = Cs + 3 * Cv, Kw = (K + 31) / 32;
    const int V3 = 3 * Cv;                       // vector floats per row
    float* wzs = rp_smem;                        // [3][Cv]
    float* vsm = wzs + V3 + (size_t)warp * (3 * V3 + 28);     // [3 rows][3][Cv]
    float* zb = vsm + 3 * V3;                    // [27]
    for (int i = threadIdx.x; i < V3; i += PW * 32) wzs[i] = __ldg(Wz + i);
    __syncthreads();
    const long ngroups = (rows + 2) / 3;
    for (long grp = (long)blockIdx.x * PW + warp; grp < ngroups; grp += (long)gridDim.x * PW) {
        const long r0 = grp * 3;
        const int ng = (int)min(3L, rows - r0);
        // ---- stage the vectors of the group: [g][x][c], all copies in flight ----
        for (int i = lane; i < V3; i += 32) {
            const int x = i / Cv, c = i - x * Cv;
            const float* src = in.v + r0 * in.ldv + (long)x * in.xs + c;
            for (int g = 0; g < ng; ++g) rp_cp_async4(vsm + g * V3 + i, src + (long)g * in.ldv);
        }
        asm volatile("cp.async.wait_all;\n" ::: "memory");
        __syncwarp();
        // ---- frames: sequential chain over channels == oracle order ----
        if (lane < ng * 9) {
            const int g = lane / 9, xm = lane - g * 9, x = xm / 3, m = xm - x * 3;
            const float* vp = vsm + g * V3 + x * Cv;
            const float* wz = wzs + m * Cv;
            float acc = 0.0f;
#pragma unroll 4
            for (int c = 0; c < Cv; ++c) acc = __fmaf_rn(vp[c], wz[c], acc);
            if (zscale) acc = __fmul_rn(acc, __ldg(zscale + m));
            zb[lane] = acc;
            if (z_out) z_out[(r0 + g) * 9 + xm] = acc;
        }
        __syncwarp();
        for (int g = 0; g < ng; ++g) {
            const long r = r0 + g;
            const float* z = zb + g * 9;
            const float* vr = vsm + g * V3;
            int nval = 0;
            // words that lie entirely in the scalar part: all loads issued before the first use
            // (16 words cover Cs <= 512), compile-time indexing
            const int ws_full = min(Cs >> 5, 16);
            float spre[16];
#pragma unroll
            for (int w = 0; w < 16; ++w) spre[w] = (w < ws_full) ? __ldg(in.s + r * in.lds + w * 32 + lane) : 0.0f;
#pragma unroll
            for (int w = 0; w < 16; ++w) {
                if (w < ws_full) {
                    const int kk = w * 32 + lane;
                    const float u = spre[w];
                    if (u_out) u_out[r * ldu + kk] = u;
                    if (bits) {
                        const float t = __fadd_rn(u, __ldg(beta + kk));
                        const unsigned pos = __ballot_sync(SV_FULL, t > 0.0f);
                        const unsigned nz = __ballot_sync(SV_FULL, t != 0.0f);
                        nval += __popc(nz);
                        if (lane == 0) { bits[r * Kw + w] = pos; mask[r * Kw + w] = nz; }
                    }
                }
            }
#pragma unroll 4
            for (int wd = ws_full; wd < Kw; ++wd) {
                const int kk = wd * 32 + lane;
                float u = 0.0f;
                if (kk < Cs) u = __ldg(in.s + r * in.lds + kk);
                else if (kk < K) {
                    const int t = kk - Cs, dd = t / 3, m = t - dd * 3;
                    float q = __fmul_rn(vr[dd], z[m]);
                    q = __fmaf_rn(vr[Cv + dd], z[3 + m], q);
                    q = __fmaf_rn(vr[2 * Cv + dd], z[6 + m], q);
                    u = q;
                }
                if (u_out && kk < K) u_out[r * ldu + kk] = u;
                if (bits) {
                    const float t = (kk < K) ? __fadd_rn(u, __ldg(beta + kk)) : 0.0f;
                    const unsigned pos = __ballot_sync(SV_FULL, t > 0.0f);
                    const unsigned nz = __ballot_sync(SV_FULL, t != 0.0f);
                    nval += __popc(nz);
                    if (lane == 0) { bits[r * Kw + wd] = pos; mask[r * Kw + wd] = nz; }
                }
            }
            if (bits && lane == 0) nvalid[r] = nval;
        }
        __syncwarp();
    }
}

// 64 rows x 64 outputs per CTA, 4x4 per thread, 16 words per smem chunk.
constexpr int BR = 64, BO = 64, WC = 16;

// TERN: ternary weights, W1nz [Kw][Cout] = non-zero plane.  The count of non-zero products then depends on (row, channel):
// each word adds popc(m & z) - 2 popc((a ^ w) & m & z) to the accumulator, which holds the dot product itself (one
// accumulator per (row, channel), not a count next to a mismatch sum, so the 4x4 tile needs no more registers).
template <bool TERN>
__global__ void __launch_bounds__(256) binlinear_rows_kernel(
    const uint32_t* __restrict__ bits, const uint32_t* __restrict__ mask, const int32_t* __restrict__ nvalid, long rows,
    int Kw, const uint32_t* __restrict__ W1b, int Cout, const float* __restrict__ scale, const float* __restrict__ bias,
    const float* __restrict__ bn_a, const float* __restrict__ bn_c, int act, const int32_t* __restrict__ cloud_dot,
    long rows_per_cloud, float* __restrict__ out, int ldo, int32_t* __restrict__ out_i32, const uint32_t* __restrict__ W1nz)
{
    __shared__ uint32_t As[WC][BR + 1], Ms[WC][BR + 1];
    __shared__ __align__(16) uint32_t Ws[WC][BO];
    __shared__ __align__(16) uint32_t Zs[TERN ? WC : 1][BO];
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
    const long r0 = (long)blockIdx.x * BR;
    const int o0 = blockIdx.y * BO;
    int acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[a][c] = 0;

    for (int w0 = 0; w0 < Kw; w0 += WC) {
        __syncthreads();
        // A/M tile: 64 rows x 16 words; thread -> (row = i / 16, word = i % 16)
        for (int i = tid; i < BR * WC; i += 256) {
            const int rr = i >> 4, ww = i & 15;
            const long r = r0 + rr;
            const int w = w0 + ww;
            uint32_t a = 0u, m = 0u;
            if (r < rows && w < Kw) { a = bits[r * Kw + w]; m = mask[r * Kw + w]; }
            As[ww][rr] = a;
            Ms[ww][rr] = m;
        }
        for (int i = tid; i < WC * BO; i += 256) {
            const int ww = i >> 6, oo = i & 63;
            const int w = w0 + ww, o = o0 + oo;
            Ws[ww][oo] = (w < Kw && o < Cout) ? W1b[(long)w * Cout + o] : 0u;
            if (TERN) Zs[ww][oo] = (w < Kw && o < Cout) ? W1nz[(long)w * Cout + o] : 0u;
        }
        __syncthreads();
        const int wn = min(WC, Kw - w0);
        for (int ww = 0; ww < wn; ++ww) {
            const uint4 wv4 = *reinterpret_cast<const uint4*>(&Ws[ww][tx * 4]);
            const uint32_t wv[4] = {wv4.x, wv4.y, wv4.z, wv4.w};
            if (TERN) {
                const uint4 zv4 = *reinterpret_cast<const uint4*>(&Zs[ww][tx * 4]);
                const uint32_t zv[4] = {zv4.x, zv4.y, zv4.z, zv4.w};
#pragma unroll
                for (int a = 0; a < 4; ++a) {
                    const uint32_t av = As[ww][ty * 4 + a], mv = Ms[ww][ty * 4 + a];
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const uint32_t mz = mv & zv[c];
                        acc[a][c] += __popc(mz) - 2 * __popc((av ^ wv[c]) & mz);
                    }
                }
            } else {
#pragma unroll
                for (int a = 0; a < 4; ++a) {
                    const uint32_t av = As[ww][ty * 4 + a], mv = Ms[ww][ty * 4 + a];
#pragma unroll
                    for (int c = 0; c < 4; ++c) acc[a][c] += __popc((av ^ wv[c]) & mv);
                }
            }
        }
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const long r = r0 + ty * 4 + a;
        if (r >= rows) continue;
        const int nv = TERN ? 0 : nvalid[r];
        const long cb = cloud_dot ? (r / rows_per_cloud) * Cout : 0;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int o = o0 + tx * 4 + c;
            if (o >= Cout) continue;
            int dot = TERN ? acc[a][c] : nv - 2 * acc[a][c];
            if (cloud_dot) dot += cloud_dot[cb + o];
            if (out_i32) { out_i32[r * Cout + o] = dot; continue; }
            float y = __fmul_rn((float)dot, scale ? scale[o] : 1.0f);
            if (bias) y = __fadd_rn(y, bias[o]);
            if (bn_a) y = __fadd_rn(__fmul_rn(y, bn_a[o]), bn_c[o]);
            out[r * ldo + o] = sv_act(y, act);
        }
    }
}

}  // namespace

int svnet_rows_prep_fast_dispatch(const svnet_view* in, long rows, const float* Wz, const float* zscale, const float* beta,
                                  uint32_t* bits, uint32_t* mask, int32_t* nvalid, cudaStream_t st);

extern "C" int svnet_rows_prep(const svnet_view* in, long rows, const float* Wz, const float* zscale, const float* z_in,
                               const float* beta, float* u_out, int ldu, float* z_out, uint32_t* bits, uint32_t* mask, int32_t* nvalid,
                               void* stream)
{
    SV_REQUIRE(in, "svnet_rows_prep: null view");
    SV_REQUIRE(in->Cs + in->Cv >= 1 && rows >= 0, "svnet_rows_prep: bad shape");
    SV_REQUIRE(in->Cs == 0 || in->s, "svnet_rows_prep: null s");
    SV_REQUIRE(in->Cv == 0 || (in->v && (Wz || z_in)), "svnet_rows_prep: null v / Wz");
    SV_REQUIRE(!bits || (mask && nvalid && beta), "svnet_rows_prep: bits output needs mask, nvalid and beta");
    SV_REQUIRE(u_out || bits || z_out, "svnet_rows_prep: no output requested");
    SV_REQUIRE(!u_out || ldu >= in->Cs + 3 * in->Cv, "svnet_rows_prep: ldu too small");
    if (rows == 0) return SVNET_OK;
    if (bits && !u_out && !z_in && !z_out) {      // sign words only: instruction-lean kernel (rows_fast.cu)
        const int handled = svnet_rows_prep_fast_dispatch(in, rows, Wz, zscale, beta, bits, mask, nvalid, sv_stream(stream));
        if (handled != 0) return handled < 0 ? handled : SVNET_OK;
    }
    const long ngroups = (rows + 2) / 3;
    const int grid = (int)min((long)sv_cdiv(ngroups, PW), 148L * 64);
    // staged variant when the group's vectors fit a modest shared-memory slice (conv5 / svfuse / PointNet blocks)
    const size_t staged_smem = sizeof(float) * ((size_t)3 * in->Cv + (size_t)PW * (9 * in->Cv + 28));
    if (in->Cv > 0 && !z_in && staged_smem <= 56 * 1024 && rows >= 1024) {
        SV_CUDA(cudaFuncSetAttribute(rows_prep_staged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)staged_smem));
        rows_prep_staged_kernel<<<grid, PW * 32, staged_smem, sv_stream(stream)>>>(*in, rows, Wz, zscale, beta, u_out, ldu, z_out,
                                                                                     bits, mask, nvalid);
        SV_CHECK_LAUNCH("svnet_rows_prep(staged)");
        return SVNET_OK;
    }
    rows_prep_kernel<<<grid, PW * 32, 0, sv_stream(stream)>>>(*in, rows, Wz, zscale, z_in, beta, u_out, ldu, z_out, bits, mask,
                                                               nvalid);
    SV_CHECK_LAUNCH("svnet_rows_prep");
    return SVNET_OK;
}

int svnet_binlinear_tc_dispatch(const uint32_t* bits, const uint32_t* mask, long rows, int K, const uint32_t* W1b,
                                const uint32_t* W1nz, int Cout, const float* scale, const float* bias, const float* bn_a,
                                const float* bn_c, int act, const int32_t* cloud_dot, long rows_per_cloud, float* out, int ldo,
                                int32_t* out_i32, void* workspace, size_t workspace_bytes, cudaStream_t st);

extern "C" int svnet_binlinear_rows_nz(const uint32_t* bits, const uint32_t* mask, const int32_t* nvalid, long rows, int K,
                                       const uint32_t* W1b, const uint32_t* W1nz, int Cout, const float* scale,
                                       const float* bias, const float* bn_a, const float* bn_c, int act,
                                       const int32_t* cloud_dot, long rows_per_cloud, float* out, int ldo, int32_t* out_i32,
                                       void* workspace, size_t workspace_bytes, void* stream)
{
    SV_REQUIRE(bits && mask && nvalid && W1b, "svnet_binlinear_rows: null pointer");
    SV_REQUIRE(out || out_i32, "svnet_binlinear_rows: no output buffer");
    SV_REQUIRE(rows >= 0 && K >= 1 && Cout >= 1, "svnet_binlinear_rows: bad shape");
    SV_REQUIRE(!out || ldo >= Cout, "svnet_binlinear_rows: ldo too small");
    SV_REQUIRE((bn_a == nullptr) == (bn_c == nullptr), "svnet_binlinear_rows: bn_a/bn_c must come together");
    SV_REQUIRE(!cloud_dot || rows_per_cloud >= 1, "svnet_binlinear_rows: rows_per_cloud");
    if (rows == 0) return SVNET_OK;
    if (workspace) {   // exact bf16 tensor-core path (binlinear_tc.cu) for the shapes it covers
        const int handled = svnet_binlinear_tc_dispatch(bits, mask, rows, K, W1b, W1nz, Cout, scale, bias, bn_a, bn_c, act, cloud_dot,
                                                        rows_per_cloud, out, ldo, out_i32, workspace, workspace_bytes,
                                                        sv_stream(stream));
        if (handled != 0) return handled < 0 ? handled : SVNET_OK;
    }
    dim3 grid(sv_cdiv(rows, BR), sv_cdiv(Cout, BO));
    if (W1nz)
        binlinear_rows_kernel<true><<<grid, 256, 0, sv_stream(stream)>>>(bits, mask, nvalid, rows, (K + 31) / 32, W1b, Cout, scale,
                                                                         bias, bn_a, bn_c, act, cloud_dot, rows_per_cloud, out, ldo,
                                                                         out_i32, W1nz);
    else
        binlinear_rows_kernel<false><<<grid, 256, 0, sv_stream(stream)>>>(bits, mask, nvalid, rows, (K + 31) / 32, W1b, Cout, scale,
                                                                          bias, bn_a, bn_c, act, cloud_dot, rows_per_cloud, out, ldo,
                                                                          out_i32, nullptr);
    SV_CHECK_LAUNCH("svnet_binlinear_rows");
    return SVNET_OK;
}

extern "C" int svnet_binlinear_rows_ws(const uint32_t* bits, const uint32_t* mask, const int32_t* nvalid, long rows, int K,
                                       const uint32_t* W1b, int Cout, const float* scale, const float* bias,
                                       const float* bn_a, const float* bn_c, int act, const int32_t* cloud_dot,
                                       long rows_per_cloud, float* out, int ldo, int32_t* out_i32, void* workspace,
                                       size_t workspace_bytes, void* stream)
{
    return svnet_binlinear_rows_nz(bits, mask, nvalid, rows, K, W1b, nullptr, Cout, scale, bias, bn_a, bn_c, act, cloud_dot,
                                   rows_per_cloud, out, ldo, out_i32, workspace, workspace_bytes, stream);
}

extern "C" int svnet_binlinear_rows(const uint32_t* bits, const uint32_t* mask, const int32_t* nvalid, long rows, int K,
                                    const uint32_t* W1b, int Cout, const float* scale, const float* bias,
                                    const float* bn_a, const float* bn_c, int act, const int32_t* cloud_dot,
                                    long rows_per_cloud, float* out, int ldo, int32_t* out_i32, void* stream)
{
    return svnet_binlinear_rows_ws(bits, mask, nvalid, rows, K, W1b, Cout, scale, bias, bn_a, bn_c, act, cloud_dot,
                                   rows_per_cloud, out, ldo, out_i32, nullptr, 0, stream);
}
