// Small kernels: weight preparation, materialising graph features (module-level parity paths),
// VectorBN on rows, pooling over the rows of a cloud.
#include "common.cuh"
#include <stdarg.h>
#include <string.h>

// ---- error string -------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

void svnet_set_error(const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" int svnet_version(void) { return SVNET_ABI_VERSION; }
extern "C" const char* svnet_last_error(void) { return g_err; }

namespace {

// one warp per (row, word): lane = bit.  NZ: also the non-zero plane (bit set = W != 0; -0.0 is zero as for torch.sign,
// subnormals are not flushed: the library is built without -ftz)
template <bool NZ>
__global__ void pack_sign_kernel(const float* __restrict__ W, int rows, int K, int ldw, uint32_t* __restrict__ bits_t,
                                 uint32_t* __restrict__ nz_t, int* __restrict__ zero_count)
{
    const int Kw = (K + 31) / 32;
    const long gw = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (gw >= (long)rows * Kw) return;
    const int row = (int)(gw / Kw), w = (int)(gw % Kw);
    const int c = w * 32 + lane;
    float v = (c < K) ? W[(long)row * ldw + c] : 0.0f;
    unsigned m = __ballot_sync(SV_FULL, v > 0.0f);
    unsigned z = __ballot_sync(SV_FULL, (c < K) && (v == 0.0f));
    unsigned nz = 0;
    if (NZ) nz = __ballot_sync(SV_FULL, (c < K) && (v != 0.0f));
    if (lane == 0) {
        bits_t[(long)w * rows + row] = m;
        if (NZ) nz_t[(long)w * rows + row] = nz;
        if (z && zero_count) atomicAdd(zero_count, __popc(z));
    }
}

__global__ void fold_bn_kernel(const float* w, const float* b, const float* mean, const float* var, float eps, int C,
                               float* a, float* c)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= C) return;
    float inv = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(var[i], eps)));
    float ai = __fmul_rn(w[i], inv);
    a[i] = ai;
    c[i] = __fsub_rn(b[i], __fmul_rn(mean[i], ai));
}

__global__ void graph_feature_xyz_kernel(const float* __restrict__ xyz, const int64_t* __restrict__ idx, int B, int N,
                                         int k, int nv, float* __restrict__ out)
{
    const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;  // one thread per edge
    if (t >= (long)B * N * k) return;
    const long r = t / k;
    const int b = (int)(r / N);
    const long j = (long)b * N + idx[t];
    const float xi[3] = {xyz[r * 3], xyz[r * 3 + 1], xyz[r * 3 + 2]};
    const float xj[3] = {xyz[j * 3], xyz[j * 3 + 1], xyz[j * 3 + 2]};
    float* o = out + t * 3 * nv;
    for (int a = 0; a < 3; ++a) {
        o[a * nv + 0] = __fsub_rn(xj[a], xi[a]);
        o[a * nv + 1] = xi[a];
    }
    if (nv == 3) {
        o[0 * nv + 2] = __fsub_rn(__fmul_rn(xj[1], xi[2]), __fmul_rn(xj[2], xi[1]));
        o[1 * nv + 2] = __fsub_rn(__fmul_rn(xj[2], xi[0]), __fmul_rn(xj[0], xi[2]));
        o[2 * nv + 2] = __fsub_rn(__fmul_rn(xj[0], xi[1]), __fmul_rn(xj[1], xi[0]));
    }
}

// one warp per edge
__global__ void graph_feature_sv_kernel(const float* __restrict__ s, const float* __restrict__ v,
                                        const int64_t* __restrict__ idx, int B, int N, int k, int Cs, int Cv,
                                        float* __restrict__ sf, float* __restrict__ vf)
{
    const long t = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (t >= (long)B * N * k) return;
    const long r = t / k;
    const int b = (int)(r / N);
    const long j = (long)b * N + idx[t];
    float* so = sf + t * 2 * Cs;
    for (int c = lane; c < Cs; c += 32) {
        float si = s[r * Cs + c];
        so[c] = __fsub_rn(s[j * Cs + c], si);
        so[Cs + c] = si;
    }
    float* vo = vf + t * 6 * Cv;
    for (int q = lane; q < 3 * Cv; q += 32) {
        int a = q / Cv, c = q - a * Cv;
        float vi = v[r * 3 * Cv + q];
        vo[a * 2 * Cv + c] = __fsub_rn(v[j * 3 * Cv + q], vi);
        vo[a * 2 * Cv + Cv + c] = vi;
    }
}

__global__ void vector_bn_rows_kernel(const float* __restrict__ v, long rows, int C, const float* __restrict__ a,
                                      const float* __restrict__ c0, float* __restrict__ out)
{
    const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= rows * C) return;
    const long r = t / C;
    const int c = (int)(t - r * C);
    const float* p = v + r * 3 * C + c;
    const float v0 = p[0], v1 = p[C], v2 = p[2 * C];
    const float n = __fadd_rn(__fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(v0, v0), __fmul_rn(v1, v1)), __fmul_rn(v2, v2))),
                              1e-6f);
    const float nb = __fadd_rn(__fmul_rn(n, a[c]), c0[c]);
    float* o = out + r * 3 * C + c;
    o[0] = __fmul_rn(__fdiv_rn(v0, n), nb);
    o[C] = __fmul_rn(__fdiv_rn(v1, n), nb);
    o[2 * C] = __fmul_rn(__fdiv_rn(v2, n), nb);
}

// CTA per (cloud, 32-column block); 8 row groups x 32 columns, fixed-order combine
__global__ void __launch_bounds__(256) pool_rows_kernel(const float* __restrict__ x, int ld, int C, long rows,
                                                        float* __restrict__ max_out, float* __restrict__ mean_out,
                                                        int ldo)
{
    __shared__ float smax[8][32], ssum[8][32];
    const int b = blockIdx.y;
    const int col = blockIdx.x * 32 + (threadIdx.x & 31);
    const int rg = sv_warp_id();
    float m = -INFINITY, s = 0.0f;
    if (col < C) {
        // eight loads in flight per thread, consumed in row order (the summation order is unchanged)
        const float* p = x + (long)b * rows * ld + col;
        long r = rg;
        for (; r + 56 < rows; r += 64) {
            float t[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) t[u] = __ldg(p + (r + 8 * u) * ld);
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                m = fmaxf(m, t[u]);
                s += t[u];
            }
        }
        for (; r < rows; r += 8) {
            const float t = __ldg(p + r * ld);
            m = fmaxf(m, t);
            s += t;
        }
    }
    smax[rg][threadIdx.x & 31] = m;
    ssum[rg][threadIdx.x & 31] = s;
    __syncthreads();
    if (rg == 0 && col < C) {
        for (int g = 1; g < 8; ++g) { m = fmaxf(m, smax[g][threadIdx.x]); s += ssum[g][threadIdx.x]; }
        if (max_out) max_out[(long)b * ldo + col] = m;
        if (mean_out) mean_out[(long)b * ldo + col] = s / (float)rows;
    }
}

}  // namespace

extern "C" int svnet_pack_sign(const float* W, int rows, int K, int ldw, uint32_t* bits_t, int* zero_count, void* stream)
{
    SV_REQUIRE(W && bits_t, "svnet_pack_sign: null pointer");
    SV_REQUIRE(rows >= 1 && K >= 1 && ldw >= K, "svnet_pack_sign: bad shape rows=%d K=%d ldw=%d", rows, K, ldw);
    cudaStream_t st = sv_stream(stream);
    if (zero_count) SV_CUDA(cudaMemsetAsync(zero_count, 0, sizeof(int), st));
    const long warps = (long)rows * ((K + 31) / 32);
    pack_sign_kernel<false><<<sv_cdiv(warps * 32, 256), 256, 0, st>>>(W, rows, K, ldw, bits_t, nullptr, zero_count);
    SV_CHECK_LAUNCH("svnet_pack_sign");
    return SVNET_OK;
}

extern "C" int svnet_pack_sign_nz(const float* W, int rows, int K, int ldw, uint32_t* bits_t, uint32_t* nz_t, int* zero_count,
                                  void* stream)
{
    SV_REQUIRE(W && bits_t && nz_t, "svnet_pack_sign_nz: null pointer");
    SV_REQUIRE(rows >= 1 && K >= 1 && ldw >= K, "svnet_pack_sign_nz: bad shape rows=%d K=%d ldw=%d", rows, K, ldw);
    cudaStream_t st = sv_stream(stream);
    if (zero_count) SV_CUDA(cudaMemsetAsync(zero_count, 0, sizeof(int), st));
    const long warps = (long)rows * ((K + 31) / 32);
    pack_sign_kernel<true><<<sv_cdiv(warps * 32, 256), 256, 0, st>>>(W, rows, K, ldw, bits_t, nz_t, zero_count);
    SV_CHECK_LAUNCH("svnet_pack_sign_nz");
    return SVNET_OK;
}

extern "C" int svnet_fold_bn(const float* w, const float* b, const float* mean, const float* var, float eps, int C,
                             float* a, float* c, void* stream)
{
    SV_REQUIRE(w && b && mean && var && a && c, "svnet_fold_bn: null pointer");
    SV_REQUIRE(C >= 1, "svnet_fold_bn: C=%d", C);
    fold_bn_kernel<<<sv_cdiv(C, 128), 128, 0, sv_stream(stream)>>>(w, b, mean, var, eps, C, a, c);
    SV_CHECK_LAUNCH("svnet_fold_bn");
    return SVNET_OK;
}

extern "C" int svnet_graph_feature_xyz(const float* xyz, const int64_t* idx, int B, int N, int k, int nv, float* out,
                                       void* stream)
{
    SV_REQUIRE(xyz && idx && out, "svnet_graph_feature_xyz: null pointer");
    SV_REQUIRE(nv == 2 || nv == 3, "svnet_graph_feature_xyz: nv=%d", nv);
    SV_REQUIRE(B >= 0 && N >= 1 && k >= 1, "svnet_graph_feature_xyz: bad shape");
    const long E = (long)B * N * k;
    if (E == 0) return SVNET_OK;
    graph_feature_xyz_kernel<<<sv_cdiv(E, 256), 256, 0, sv_stream(stream)>>>(xyz, idx, B, N, k, nv, out);
    SV_CHECK_LAUNCH("svnet_graph_feature_xyz");
    return SVNET_OK;
}

extern "C" int svnet_graph_feature_sv(const float* s, const float* v, const int64_t* idx, int B, int N, int k, int Cs,
                                      int Cv, float* sf, float* vf, void* stream)
{
    SV_REQUIRE(s && v && idx && sf && vf, "svnet_graph_feature_sv: null pointer");
    SV_REQUIRE(B >= 0 && N >= 1 && k >= 1 && Cs >= 1 && Cv >= 1, "svnet_graph_feature_sv: bad shape");
    const long E = (long)B * N * k;
    if (E == 0) return SVNET_OK;
    graph_feature_sv_kernel<<<sv_cdiv(E * 32, 256), 256, 0, sv_stream(stream)>>>(s, v, idx, B, N, k, Cs, Cv, sf, vf);
    SV_CHECK_LAUNCH("svnet_graph_feature_sv");
    return SVNET_OK;
}

extern "C" int svnet_vector_bn_rows(const float* v, long rows, int C, const float* bn_a, const float* bn_c, float* out,
                                    void* stream)
{
    SV_REQUIRE(v && bn_a && bn_c && out, "svnet_vector_bn_rows: null pointer");
    SV_REQUIRE(rows >= 0 && C >= 1, "svnet_vector_bn_rows: bad shape");
    if (rows == 0) return SVNET_OK;
    vector_bn_rows_kernel<<<sv_cdiv(rows * C, 256), 256, 0, sv_stream(stream)>>>(v, rows, C, bn_a, bn_c, out);
    SV_CHECK_LAUNCH("svnet_vector_bn_rows");
    return SVNET_OK;
}

extern "C" int svnet_pool_rows(const float* x, int ld, int C, int B, long rows, float* max_out, float* mean_out,
                               int ldo, void* stream)
{
    SV_REQUIRE(x && (max_out || mean_out), "svnet_pool_rows: null pointer");
    SV_REQUIRE(C >= 1 && ld >= C && rows >= 1 && B >= 0 && ldo >= C, "svnet_pool_rows: bad shape");
    if (B == 0) return SVNET_OK;
    SV_REQUIRE(B <= 65535 * 1024, "svnet_pool_rows: too many clouds");
    // grid.y is limited to 65535: fold large B (module-level svpool over k uses B*N "clouds")
    const int gx = sv_cdiv(C, 32);
    long done = 0;
    while (done < B) {
        const int nb = (int)((B - done) > 65535 ? 65535 : (B - done));
        dim3 grid(gx, nb);
        pool_rows_kernel<<<grid, 256, 0, sv_stream(stream)>>>(x + done * rows * ld, ld, C, rows,
                                                              max_out ? max_out + done * ldo : nullptr,
                                                              mean_out ? mean_out + done * ldo : nullptr, ldo);
        done += nb;
    }
    SV_CHECK_LAUNCH("svnet_pool_rows");
    return SVNET_OK;
}

// ---- input side of the eval loop (SURVEY.md 8(f) f3): random-rotation transform + (B,N,3)->(B,3,N) ----
namespace {
// out[b][c][n] = sum_d p[b][n][d] * R[b][d][c]   (pytorch3d Rotate.transform_points = points @ R, then
// data.permute(0, 2, 1): reference main_cls_dgcnn.py:229-235)
__global__ void rotate_permute_kernel(const float* __restrict__ pts, const float* __restrict__ R, int B, int N,
                                      float* __restrict__ out)
{
    const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long)B * N) return;
    const int b = (int)(t / N), n = (int)(t - (long)b * N);
    const float p0 = pts[t * 3], p1 = pts[t * 3 + 1], p2 = pts[t * 3 + 2];
    float* o = out + (long)b * 3 * N + n;
    if (R) {
        const float* r = R + (long)b * 9;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            float a = __fmul_rn(p0, r[c]);
            a = __fmaf_rn(p1, r[3 + c], a);
            a = __fmaf_rn(p2, r[6 + c], a);
            o[(long)c * N] = a;
        }
    } else {
        o[0] = p0; o[N] = p1; o[2L * N] = p2;
    }
}
}  // namespace

extern "C" int svnet_rotate_permute(const float* pts, const float* R, int B, int N, float* out, void* stream)
{
    SV_REQUIRE(pts && out, "svnet_rotate_permute: null pointer");
    SV_REQUIRE(B >= 0 && N >= 1, "svnet_rotate_permute: bad shape");
    if (B == 0) return SVNET_OK;
    rotate_permute_kernel<<<sv_cdiv((long)B * N, 256), 256, 0, sv_stream(stream)>>>(pts, R, B, N, out);
    SV_CHECK_LAUNCH("svnet_rotate_permute");
    return SVNET_OK;
}
