// pergauss.cu -- the per-gaussian (HBM-bound) kernels: quat/scale -> covariance, EWA projection,
// spherical harmonics, the fused projection + conic + SH->RGB pass, tile counting / emission and
// the tile-offset encoder.  Compiled with -fmad=false (see gaussmath.cuh).
//
// Reference kernels replaced: csrc/QuatScaleToCovarCUDA.cu:37,211;
// csrc/ProjectionEWA3DGSFused.cu:38-219,376-638; csrc/SphericalHarmonicsCUDA.cu:443-569,785-890,
// 1085-1250 (assemble_proj_features); csrc/IntersectTile.cu:83-464,925-988.
#include <cub/device/device_scan.cuh>

#include "gaussmath.cuh"
#include "rowrec.cuh"

namespace gsb
{
constexpr int kThreads = 256;

// ------------------------------------------------------------------ quat_scale_to_covar_preci
__device__ __forceinline__ void store_sym(float *dst, const M3 &S, bool triu)
{
    if(triu)
    {
        dst[0] = S.m[0], dst[1] = S.m[1], dst[2] = S.m[2], dst[3] = S.m[4], dst[4] = S.m[5], dst[5] = S.m[8];
    }
    else
    {
#pragma unroll
        for(int k = 0; k < 9; ++k)
            dst[k] = S.m[k];
    }
}
__device__ __forceinline__ M3 load_sym_grad(const float *v, bool triu)
{
    M3 G;
    if(triu)
    {
        G.m[0] = v[0];
        G.m[1] = G.m[3] = v[1] * 0.5f;
        G.m[2] = G.m[6] = v[2] * 0.5f;
        G.m[4] = v[3];
        G.m[5] = G.m[7] = v[4] * 0.5f;
        G.m[8] = v[5];
    }
    else
    {
#pragma unroll
        for(int k = 0; k < 9; ++k)
            G.m[k] = v[k];
    }
    return G;
}

__global__ void __launch_bounds__(kThreads) quat_scale_fwd_kernel(
    int64_t N, const float *__restrict__ quats, const float *__restrict__ scales, bool triu, float *__restrict__ covars,
    float *__restrict__ precis
)
{
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if(n >= N)
        return;
    const float q[4] = {quats[n * 4], quats[n * 4 + 1], quats[n * 4 + 2], quats[n * 4 + 3]};
    const float s[3] = {scales[n * 3], scales[n * 3 + 1], scales[n * 3 + 2]};
    const int stride = triu ? 6 : 9;
    if(covars)
        store_sym(covars + n * stride, quat_scale_to_sym<false>(q, s), triu);
    if(precis)
        store_sym(precis + n * stride, quat_scale_to_sym<true>(q, s), triu);
}

__global__ void __launch_bounds__(kThreads) quat_scale_bwd_kernel(
    int64_t N, const float *__restrict__ quats, const float *__restrict__ scales, bool triu,
    const float *__restrict__ v_covars, const float *__restrict__ v_precis, float *__restrict__ v_quats,
    float *__restrict__ v_scales
)
{
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if(n >= N)
        return;
    const float q[4] = {quats[n * 4], quats[n * 4 + 1], quats[n * 4 + 2], quats[n * 4 + 3]};
    const float s[3] = {scales[n * 3], scales[n * 3 + 1], scales[n * 3 + 2]};
    const int stride = triu ? 6 : 9;
    float vq[4] = {0.f, 0.f, 0.f, 0.f}, vs[3] = {0.f, 0.f, 0.f};
    if(v_covars)
        quat_scale_sym_vjp<false>(q, s, load_sym_grad(v_covars + n * stride, triu), vq, vs);
    if(v_precis)
        quat_scale_sym_vjp<true>(q, s, load_sym_grad(v_precis + n * stride, triu), vq, vs);
#pragma unroll
    for(int k = 0; k < 4; ++k)
        v_quats[n * 4 + k] = vq[k];
#pragma unroll
    for(int k = 0; k < 3; ++k)
        v_scales[n * 3 + k] = vs[k];
}

// ------------------------------------------------------------------ projection
__device__ __forceinline__ M3 load_cov6(const float *c6)
{
    M3 S;
    S.m[0] = c6[0];
    S.m[1] = S.m[3] = c6[1];
    S.m[2] = S.m[6] = c6[2];
    S.m[4] = c6[3];
    S.m[5] = S.m[7] = c6[4];
    S.m[8] = c6[5];
    return S;
}

template<int CAM>
__global__ void __launch_bounds__(kThreads) projection_fwd_kernel(
    int64_t B, int64_t C, int64_t N, const float *__restrict__ means, const float *__restrict__ covars,
    const float *__restrict__ quats, const float *__restrict__ scales, const float *__restrict__ opacities,
    const float *__restrict__ viewmats, const float *__restrict__ Ks, uint32_t W, uint32_t H, float eps2d,
    float near_plane, float far_plane, float radius_clip, int32_t *__restrict__ radii, float *__restrict__ means2d,
    float *__restrict__ depths, float *__restrict__ conics, float *__restrict__ compensations
)
{
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if(idx >= B * C * N)
        return;
    const int64_t b = idx / (C * N), c = (idx / N) % C, n = idx % N;
    const int64_t bn = b * N + n;
    const Cam cam = load_cam(viewmats + (b * C + c) * 16, Ks + (b * C + c) * 9);
    const float mean[3] = {means[bn * 3], means[bn * 3 + 1], means[bn * 3 + 2]};
    M3 cov;
    if(covars)
        cov = load_cov6(covars + bn * 6);
    else
    {
        const float q[4] = {quats[bn * 4], quats[bn * 4 + 1], quats[bn * 4 + 2], quats[bn * 4 + 3]};
        const float s[3] = {scales[bn * 3], scales[bn * 3 + 1], scales[bn * 3 + 2]};
        cov = quat_scale_to_sym<false>(q, s);
    }
    float op = 0.f;
    if(opacities)
        op = opacities[bn];
    const Proj p = project_one<CAM>(
        mean, cov, opacities ? &op : nullptr, cam, W, H, eps2d, near_plane, far_plane, radius_clip, compensations != nullptr
    );
    reinterpret_cast<int2 *>(radii)[idx]    = make_int2(p.rx, p.ry);
    reinterpret_cast<float2 *>(means2d)[idx] = make_float2(p.mx, p.my);
    depths[idx]         = p.depth;
    conics[idx * 3]     = p.ca;
    conics[idx * 3 + 1] = p.cb;
    conics[idx * 3 + 2] = p.cc;
    if(compensations)
        compensations[idx] = p.comp;
}

// One thread per (b, n), looping over the C cameras: the per-gaussian sums stay in registers and
// every output row is written exactly once (deterministic, no zero-init, no atomics).
template<int CAM>
__global__ void __launch_bounds__(kThreads) projection_bwd_kernel(
    int64_t B, int64_t C, int64_t N, const float *__restrict__ means, const float *__restrict__ covars,
    const float *__restrict__ quats, const float *__restrict__ scales, const float *__restrict__ viewmats,
    const float *__restrict__ Ks, uint32_t W, uint32_t H, float eps2d, const int32_t *__restrict__ radii,
    const float *__restrict__ conics, const float *__restrict__ compensations, const float *__restrict__ v_means2d,
    int64_t s_m2, const float *__restrict__ v_depths, int64_t s_d, const float *__restrict__ v_conics, int64_t s_c,
    const float *__restrict__ v_compensations, float *__restrict__ v_means, float *__restrict__ v_covars,
    float *__restrict__ v_quats, float *__restrict__ v_scales, float *__restrict__ v_viewmats
)
{
    const int64_t bn   = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool active  = bn < B * N;
    const int64_t b    = active ? bn / N : 0, n = active ? bn % N : 0;
    const unsigned lane = threadIdx.x & 31;
    float mean[3] = {0.f, 0.f, 0.f}, q[4] = {1.f, 0.f, 0.f, 0.f}, s[3] = {1.f, 1.f, 1.f};
    M3 cov;
#pragma unroll
    for(int k = 0; k < 9; ++k)
        cov.m[k] = 0.f;
    if(active)
    {
        mean[0] = means[bn * 3], mean[1] = means[bn * 3 + 1], mean[2] = means[bn * 3 + 2];
        if(covars)
            cov = load_cov6(covars + bn * 6);
        else
        {
#pragma unroll
            for(int k = 0; k < 4; ++k)
                q[k] = quats[bn * 4 + k];
#pragma unroll
            for(int k = 0; k < 3; ++k)
                s[k] = scales[bn * 3 + k];
            cov = quat_scale_to_sym<false>(q, s);
        }
    }
    float v_mean[3] = {0.f, 0.f, 0.f};
    M3 v_cov;
#pragma unroll
    for(int k = 0; k < 9; ++k)
        v_cov.m[k] = 0.f;
    for(int64_t c = 0; c < C; ++c)
    {
        const int64_t idx = (b * C + c) * N + n;
        const bool vis    = active && radii[idx * 2] > 0 && radii[idx * 2 + 1] > 0;
        float vm_part[12];
#pragma unroll
        for(int k = 0; k < 12; ++k)
            vm_part[k] = 0.f;
        if(vis)
        {
            const Cam cam       = load_cam(viewmats + (b * C + c) * 16, Ks + (b * C + c) * 9);
            const float conic[3] = {conics[idx * 3], conics[idx * 3 + 1], conics[idx * 3 + 2]};
            const float vc[3]    = {v_conics[idx * s_c], v_conics[idx * s_c + 1], v_conics[idx * s_c + 2]};
            const bool has_comp  = v_compensations != nullptr;
            const ProjGrad g     = project_one_vjp<CAM>(
                mean, cov, cam, W, H, eps2d, conic, v_means2d[idx * s_m2], v_means2d[idx * s_m2 + 1], v_depths[idx * s_d],
                vc, has_comp, has_comp ? compensations[idx] : 0.f, has_comp ? v_compensations[idx] : 0.f
            );
#pragma unroll
            for(int k = 0; k < 3; ++k)
                v_mean[k] += g.v_mean[k];
#pragma unroll
            for(int k = 0; k < 9; ++k)
                v_cov.m[k] += g.v_cov.m[k];
            if(v_viewmats)
            { // v_R = v_pc mean^T + v_covc R cov^T + v_covc^T R cov ; v_t = v_pc
                const M3 A2 = mul_bt(mul(g.v_covc, cam.R), cov);
                const M3 B2 = mul(mul_at(g.v_covc, cam.R), cov);
#pragma unroll
                for(int i = 0; i < 3; ++i)
                {
#pragma unroll
                    for(int j = 0; j < 3; ++j)
                        vm_part[i * 4 + j] = g.v_pc[i] * mean[j] + A2.m[i * 3 + j] + B2.m[i * 3 + j];
                    vm_part[i * 4 + 3] = g.v_pc[i];
                }
            }
        }
        if(v_viewmats)
        {
            // warp butterfly reduce of the 12 pose-gradient entries, one atomic per owning lane -- valid only when
            // every lane of the warp belongs to the same batch element (a warp straddles a batch boundary when N is
            // not a multiple of 32: those lanes add their own entries)
            const int64_t b0    = __shfl_sync(0xffffffffu, b, 0);
            const bool same_b   = __all_sync(0xffffffffu, !active || b == b0);
            if(same_b)
            {
                Butterfly<12, 16>::run(vm_part, lane);
                const int slot = butterfly_slot<12>(lane);
                if(slot >= 0 && vm_part[0] != 0.f)
                    atomicAdd(v_viewmats + (b0 * C + c) * 16 + slot, vm_part[0]);
            }
            else if(vis)
            {
#pragma unroll
                for(int k = 0; k < 12; ++k)
                    atomicAdd(v_viewmats + (b * C + c) * 16 + k, vm_part[k]);
            }
        }
    }
    if(!active)
        return;
#pragma unroll
    for(int k = 0; k < 3; ++k)
        v_means[bn * 3 + k] = v_mean[k];
    if(covars)
    {
        float *o = v_covars + bn * 6;
        o[0] = v_cov.m[0];
        o[1] = v_cov.m[1] + v_cov.m[3];
        o[2] = v_cov.m[2] + v_cov.m[6];
        o[3] = v_cov.m[4];
        o[4] = v_cov.m[5] + v_cov.m[7];
        o[5] = v_cov.m[8];
    }
    else
    {
        float vq[4] = {0.f, 0.f, 0.f, 0.f}, vs[3] = {0.f, 0.f, 0.f};
        quat_scale_sym_vjp<false>(q, s, v_cov, vq, vs);
#pragma unroll
        for(int k = 0; k < 4; ++k)
            v_quats[bn * 4 + k] = vq[k];
#pragma unroll
        for(int k = 0; k < 3; ++k)
            v_scales[bn * 3 + k] = vs[k];
    }
}

// ------------------------------------------------------------------ spherical harmonics
template<int DEG>
__global__ void __launch_bounds__(kThreads) sh_fwd_kernel(
    int64_t B, int64_t C, int64_t N, int64_t K, int64_t D, const float *__restrict__ means,
    const float *__restrict__ viewmats, const float *__restrict__ coeffs, const uint8_t *__restrict__ masks,
    float *__restrict__ colors
)
{
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if(idx >= B * C * N)
        return;
    const int64_t b = idx / (C * N), c = (idx / N) % C, n = idx % N;
    float *out = colors + idx * D;
    if(masks && !masks[idx])
    {
        for(int64_t d = 0; d < D; ++d)
            out[d] = 0.f;
        return;
    }
    const float mean[3] = {means[(b * N + n) * 3], means[(b * N + n) * 3 + 1], means[(b * N + n) * 3 + 2]};
    float dir[3];
    sh_view_dir(mean, viewmats + (b * C + c) * 16, dir);
    const float inorm = 1.f / sqrtf(dir[0] * dir[0] + dir[1] * dir[1] + dir[2] * dir[2]);
    constexpr int NB  = (DEG + 1) * (DEG + 1);
    Dual<false> Y[NB];
    sh_basis<DEG, false>(dir[0] * inorm, dir[1] * inorm, dir[2] * inorm, Y);
    const float *cf = coeffs + n * K * D;
    for(int64_t d = 0; d < D; ++d)
    {
        float acc = 0.f;
#pragma unroll
        for(int k = 0; k < NB; ++k)
            acc += Y[k].v * cf[k * D + d];
        out[d] = acc;
    }
}

// one thread per (gaussian, channel), looping over images; v_coeffs written once per thread,
// v_means accumulated with atomics (pre-zeroed by the host wrapper).
template<int DEG>
__global__ void __launch_bounds__(kThreads) sh_bwd_kernel(
    int64_t B, int64_t C, int64_t N, int64_t K, int64_t D, const float *__restrict__ means,
    const float *__restrict__ viewmats, const float *__restrict__ coeffs, const uint8_t *__restrict__ masks,
    const float *__restrict__ v_colors, float *__restrict__ v_coeffs, float *__restrict__ v_means,
    float *__restrict__ v_dirsum
)
{
    const int64_t idx  = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool in_range = idx < N * D; // out-of-range threads stay for the warp reduction of v_dirsum
    const int64_t n = in_range ? idx / D : 0, d = in_range ? idx % D : 0;
    const unsigned lane = threadIdx.x & 31;
    constexpr int NB = (DEG + 1) * (DEG + 1);
    float acc[NB];
#pragma unroll
    for(int k = 0; k < NB; ++k)
        acc[k] = 0.f;
    const float *cf = coeffs + n * K * D;
    for(int64_t img = 0; img < B * C; ++img)
    {
        const int64_t b = img / C;
        const int64_t o = img * N + n;
        const bool on   = in_range && !(masks && !masks[o]);
        float vd[3]     = {0.f, 0.f, 0.f};
        if(on)
        {
        const float *mean = means + (b * N + n) * 3;
        float dir[3];
        sh_view_dir(mean, viewmats + img * 16, dir);
        const float inorm = 1.f / sqrtf(dir[0] * dir[0] + dir[1] * dir[1] + dir[2] * dir[2]);
        const float u[3]  = {dir[0] * inorm, dir[1] * inorm, dir[2] * inorm};
        Dual<true> Y[NB];
        sh_basis<DEG, true>(u[0], u[1], u[2], Y);
        const float vc = v_colors[o * D + d];
        float vu[3] = {0.f, 0.f, 0.f};
#pragma unroll
        for(int k = 0; k < NB; ++k)
        {
            acc[k] += Y[k].v * vc;
            const float g = cf[k * D + d] * vc;
            vu[0] += g * Y[k].x;
            vu[1] += g * Y[k].y;
            vu[2] += g * Y[k].z;
        }
        if(DEG >= 1)
        {
            const float dot = vu[0] * u[0] + vu[1] * u[1] + vu[2] * u[2];
#pragma unroll
            for(int j = 0; j < 3; ++j)
                vd[j] = (vu[j] - dot * u[j]) * inorm;
            if(v_means != nullptr)
            {
#pragma unroll
                for(int j = 0; j < 3; ++j)
                    atomicAdd(v_means + (b * N + n) * 3 + j, vd[j]);
            }
        }
        }
        if(v_dirsum != nullptr && DEG >= 1)
        { // per-image sum of the view-direction gradient (for the pose gradient): warp reduce, one atomic per warp
            Butterfly<3, 16>::run(vd, lane);
            const int slot = butterfly_slot<3>(lane);
            if(slot >= 0 && vd[0] != 0.f)
                atomicAdd(v_dirsum + img * 3 + slot, vd[0]);
        }
    }
    if(!in_range)
        return;
    float *vcf = v_coeffs + n * K * D;
#pragma unroll
    for(int k = 0; k < NB; ++k)
        vcf[k * D + d] = acc[k];
    for(int64_t k = NB; k < K; ++k)
        vcf[k * D + d] = 0.f;
}

// ---- SH on packed rows: row i = (batch_ids[i], camera_ids[i], gaussian_ids[i]); the coefficients stay in their
// [N, K, D] table and are indexed in the kernel (no [nnz, K, D] gather as in the reference's packed call,
// rendering.py:1001-1010).  One thread per (row, channel).
template<int DEG>
__global__ void __launch_bounds__(kThreads) sh_rows_fwd_kernel(
    int64_t nnz, int64_t C, int64_t N, int64_t K, int64_t D, const float *__restrict__ means,
    const float *__restrict__ viewmats, const float *__restrict__ coeffs, const int64_t *__restrict__ batch_ids,
    const int64_t *__restrict__ camera_ids, const int64_t *__restrict__ gaussian_ids, float *__restrict__ colors
)
{
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if(idx >= nnz * D)
        return;
    const int64_t i = idx / D, d = idx % D;
    const int64_t b = batch_ids[i], c = camera_ids[i], n = gaussian_ids[i];
    const float mean[3] = {means[(b * N + n) * 3], means[(b * N + n) * 3 + 1], means[(b * N + n) * 3 + 2]};
    float dir[3];
    sh_view_dir(mean, viewmats + (b * C + c) * 16, dir);
    const float inorm = 1.f / sqrtf(dir[0] * dir[0] + dir[1] * dir[1] + dir[2] * dir[2]);
    constexpr int NB  = (DEG + 1) * (DEG + 1);
    Dual<false> Y[NB];
    sh_basis<DEG, false>(dir[0] * inorm, dir[1] * inorm, dir[2] * inorm, Y);
    const float *cf = coeffs + n * K * D;
    float acc       = 0.f;
#pragma unroll
    for(int k = 0; k < NB; ++k)
        acc += Y[k].v * cf[k * D + d];
    colors[idx] = acc;
}

// v_coeffs [N, K, D], v_means [B*N, 3] and v_dirsum [B*C, 3] are zero-initialised by the host and summed with
// atomics (a gaussian seen by several cameras owns several rows).
template<int DEG>
__global__ void __launch_bounds__(kThreads) sh_rows_bwd_kernel(
    int64_t nnz, int64_t C, int64_t N, int64_t K, int64_t D, const float *__restrict__ means,
    const float *__restrict__ viewmats, const float *__restrict__ coeffs, const int64_t *__restrict__ batch_ids,
    const int64_t *__restrict__ camera_ids, const int64_t *__restrict__ gaussian_ids, const float *__restrict__ v_colors,
    float *__restrict__ v_coeffs, float *__restrict__ v_means, float *__restrict__ v_dirsum
)
{
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if(idx >= nnz * D)
        return;
    const int64_t i = idx / D, d = idx % D;
    const int64_t b = batch_ids[i], c = camera_ids[i], n = gaussian_ids[i];
    const float *mean = means + (b * N + n) * 3;
    float dir[3];
    sh_view_dir(mean, viewmats + (b * C + c) * 16, dir);
    const float inorm = 1.f / sqrtf(dir[0] * dir[0] + dir[1] * dir[1] + dir[2] * dir[2]);
    const float u[3]  = {dir[0] * inorm, dir[1] * inorm, dir[2] * inorm};
    constexpr int NB  = (DEG + 1) * (DEG + 1);
    Dual<true> Y[NB];
    sh_basis<DEG, true>(u[0], u[1], u[2], Y);
    const float vc  = v_colors[idx];
    const float *cf = coeffs + n * K * D;
    float *vcf      = v_coeffs + n * K * D;
    float vu[3]     = {0.f, 0.f, 0.f};
#pragma unroll
    for(int k = 0; k < NB; ++k)
    {
        atomicAdd(vcf + k * D + d, Y[k].v * vc);
        const float g = cf[k * D + d] * vc;
        vu[0] += g * Y[k].x;
        vu[1] += g * Y[k].y;
        vu[2] += g * Y[k].z;
    }
    if(DEG >= 1 && (v_means != nullptr || v_dirsum != nullptr))
    {
        const float dot = vu[0] * u[0] + vu[1] * u[1] + vu[2] * u[2];
#pragma unroll
        for(int j = 0; j < 3; ++j)
        {
            const float vd = (vu[j] - dot * u[j]) * inorm;
            if(v_means != nullptr)
                atomicAdd(v_means + (b * N + n) * 3 + j, vd);
            if(v_dirsum != nullptr)
                atomicAdd(v_dirsum + (b * C + c) * 3 + j, vd);
        }
    }
}

// ------------------------------------------------------------------ fused projection + conic + SH -> RGB
// One thread per (camera, gaussian).  SH coefficients of a visible gaussian are fetched with 128-bit
// loads (48 floats = 12 x float4 when K = 16); culled gaussians never touch them.
template<class F>
__device__ __forceinline__ int tiles_of_gaussian(
    float mx, float my, int rx, int ry, const float *conic, const float *opacity, uint32_t tile_size, uint32_t tw,
    uint32_t th, F &&f
); // defined with the tile intersection kernels below

// ROWS: the epilogue also produces what the next two stages would otherwise recompute per row / per intersection --
// the row's tile count and the three totals of gsb200_isect_count_totals (same device function as the emit pass, so the
// counts agree bit for bit), and the 64-byte compositing row record {cull | axis | geom | rgb0} of rowrec.cuh, which
// turns the pack pass into a pure gather.  Only valid when the compositing opacity is the input opacity (no
// antialiasing compensation) -- the host wrapper checks that.
template<int DEG, bool ROWS>
__global__ void __launch_bounds__(kThreads, 4) project_sh_fwd_kernel(
    int64_t C, int64_t N, int64_t K, const float *__restrict__ means, const float *__restrict__ quats,
    const float *__restrict__ scales, const float *__restrict__ opacities, const float *__restrict__ sh,
    const float *__restrict__ viewmats, const float *__restrict__ Ks, uint32_t W, uint32_t H, float eps2d,
    float near_plane, float far_plane, float radius_clip, int32_t *__restrict__ radii, float *__restrict__ means2d,
    float *__restrict__ depths, float *__restrict__ conics, float *__restrict__ compensations,
    float *__restrict__ colors, uint32_t tile_size, uint32_t tile_w, uint32_t tile_h, float4 *__restrict__ rows,
    int32_t *__restrict__ tiles_per_gauss, unsigned long long *__restrict__ totals
)
{
    __shared__ unsigned long long s_tot[3];
    if constexpr(ROWS)
    {
        if(threadIdx.x < 3)
            s_tot[threadIdx.x] = 0ull;
        __syncthreads();
    }
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int cnt           = 0;
    if(idx < C * N)
    {
    const int64_t c = idx / N, n = idx % N;
    const float *vm = viewmats + c * 16;
    const Cam cam   = load_cam(vm, Ks + c * 9);
    const float mean[3] = {means[n * 3], means[n * 3 + 1], means[n * 3 + 2]};
    const float4 q4     = *reinterpret_cast<const float4 *>(quats + n * 4);
    const float q[4]    = {q4.x, q4.y, q4.z, q4.w};
    const float s[3]    = {scales[n * 3], scales[n * 3 + 1], scales[n * 3 + 2]};
    const float op      = opacities[n];
    const M3 cov        = quat_scale_to_sym<false>(q, s);
    const Proj p = project_one(mean, cov, &op, cam, W, H, eps2d, near_plane, far_plane, radius_clip, compensations != nullptr);
    reinterpret_cast<int2 *>(radii)[idx]     = make_int2(p.rx, p.ry);
    reinterpret_cast<float2 *>(means2d)[idx] = make_float2(p.mx, p.my);
    depths[idx]         = p.depth;
    conics[idx * 3]     = p.ca;
    conics[idx * 3 + 1] = p.cb;
    conics[idx * 3 + 2] = p.cc;
    if(compensations)
        compensations[idx] = p.comp;
    float rgb[3] = {0.f, 0.f, 0.f};
    if(p.rx > 0 && p.ry > 0)
    {
        float dir[3];
        sh_view_dir(mean, vm, dir);
        const float inorm = 1.f / sqrtf(dir[0] * dir[0] + dir[1] * dir[1] + dir[2] * dir[2]);
        constexpr int NB  = (DEG + 1) * (DEG + 1);
        const float *cf = sh + n * K * 3;
        float cbuf[NB * 3];
        if(((K * 3) & 3) == 0 && (NB * 3) % 4 == 0)
        { // 16-byte aligned rows: 128-bit read-only loads
            const float4 *cf4 = reinterpret_cast<const float4 *>(cf);
#pragma unroll
            for(int v = 0; v < NB * 3 / 4; ++v)
            {
                const float4 t = ldg_nc_f4(cf4 + v);
                cbuf[4 * v] = t.x, cbuf[4 * v + 1] = t.y, cbuf[4 * v + 2] = t.z, cbuf[4 * v + 3] = t.w;
            }
        }
        else
        {
#pragma unroll
            for(int k = 0; k < NB * 3; ++k)
                cbuf[k] = __ldg(cf + k);
        }
        float acc3[3] = {0.f, 0.f, 0.f};
        sh_visit<DEG, false>(dir[0] * inorm, dir[1] * inorm, dir[2] * inorm, [&](int k, const Dual<false> &Yk) {
#pragma unroll
            for(int d = 0; d < 3; ++d)
                acc3[d] += Yk.v * cbuf[k * 3 + d];
        });
#pragma unroll
        for(int d = 0; d < 3; ++d)
        {
            const float shifted = acc3[d] + 0.5f;
            rgb[d]              = shifted > 0.f ? shifted : 0.f;
        }
    }
    colors[idx * 3] = rgb[0], colors[idx * 3 + 1] = rgb[1], colors[idx * 3 + 2] = rgb[2];
    if constexpr(ROWS)
    {
        if(p.rx > 0 && p.ry > 0)
        {
            float cn[3] = {p.ca, p.cb, p.cc};
            cnt         = tiles_of_gaussian(p.mx, p.my, p.rx, p.ry, cn, &op, tile_size, tile_w, tile_h, [](int64_t) {});
            float4 rc, ra, rg;
            row_record(p.mx, p.my, p.ca, p.cb, p.cc, op, rc, ra, rg);
            rows[idx * 4]     = rc;
            rows[idx * 4 + 1] = ra;
            rows[idx * 4 + 2] = rg;
            rows[idx * 4 + 3] = make_float4(rgb[0], rgb[1], rgb[2], 0.f);
        }
        tiles_per_gauss[idx] = cnt;
    }
    }
    if constexpr(ROWS)
    { // the three totals, as isect_count_totals_kernel forms them
        const int wsum         = __reduce_add_sync(0xffffffffu, cnt);
        const int wmax         = __reduce_max_sync(0xffffffffu, cnt);
        const unsigned nonzero = __ballot_sync(0xffffffffu, cnt > 0);
        if((threadIdx.x & 31) == 0 && nonzero != 0u)
        {
            atomicAdd(&s_tot[0], (unsigned long long)wsum);
            atomicAdd(&s_tot[1], (unsigned long long)__popc(nonzero));
            atomicMax(&s_tot[2], (unsigned long long)wmax);
        }
        __syncthreads();
        if(threadIdx.x < 2 && s_tot[threadIdx.x] != 0ull)
            atomicAdd(&totals[threadIdx.x], s_tot[threadIdx.x]);
        if(threadIdx.x == 2 && s_tot[2] != 0ull)
            atomicMax(&totals[2], s_tot[2]);
    }
}

// One thread per gaussian, looping over cameras: v_means / v_quats / v_scales / v_sh written once.
// ONE_CAM (C == 1: every rank of the view-parallel trainer, any batch-size-1 step): the camera loop is gone at compile
// time, so the 48 SH accumulators die as soon as they are stored -- 80 registers with 36 bytes of spills instead of 128
// with 164, three CTAs per SM instead of two.
template<int DEG, bool ONE_CAM>
__global__ void __launch_bounds__(kThreads, ONE_CAM ? 3 : 2) project_sh_bwd_kernel(
    int64_t C, int64_t N, int64_t K, const float *__restrict__ means, const float *__restrict__ quats,
    const float *__restrict__ scales, const float *__restrict__ sh, const float *__restrict__ viewmats,
    const float *__restrict__ Ks, uint32_t W, uint32_t H, float eps2d, const int32_t *__restrict__ radii,
    const float *__restrict__ conics, const float *__restrict__ compensations, const float *__restrict__ colors,
    const float *__restrict__ v_means2d, int64_t s_m2, const float *__restrict__ v_depths, int64_t s_d,
    const float *__restrict__ v_conics, int64_t s_c, const float *__restrict__ v_colors, int64_t s_col,
    const float *__restrict__ v_compensations, float *__restrict__ v_means, float *__restrict__ v_quats,
    float *__restrict__ v_scales, float *__restrict__ v_sh, uint32_t *__restrict__ seen_bits
)
{
    const int64_t n     = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned lane = threadIdx.x & 31;
    constexpr int NB    = (DEG + 1) * (DEG + 1);
    // Most gaussians are culled in every view: their gradient rows are zeros.  Those rows are written by the whole
    // warp, coalesced (32 consecutive rows = one contiguous block), and their parameters are never loaded.
    bool seen = false;
    if(n < N)
        for(int64_t c = 0; c < (ONE_CAM ? (int64_t)1 : C); ++c)
            seen |= radii[(c * N + n) * 2] > 0 && radii[(c * N + n) * 2 + 1] > 0;
    if(seen)
    {
        const float mean[3] = {means[n * 3], means[n * 3 + 1], means[n * 3 + 2]};
        const float4 q4     = *reinterpret_cast<const float4 *>(quats + n * 4);
        const float q[4]    = {q4.x, q4.y, q4.z, q4.w};
        const float s[3]    = {scales[n * 3], scales[n * 3 + 1], scales[n * 3 + 2]};
        const M3 cov        = quat_scale_to_sym<false>(q, s);
        float v_mean[3] = {0.f, 0.f, 0.f};
        M3 v_cov;
#pragma unroll
        for(int k = 0; k < 9; ++k)
            v_cov.m[k] = 0.f;
        float acc[NB * 3];
#pragma unroll
        for(int k = 0; k < NB * 3; ++k)
            acc[k] = 0.f;
        const float *cf = sh + n * K * 3;
        for(int64_t c = 0; c < (ONE_CAM ? (int64_t)1 : C); ++c)
        {
            const int64_t idx = c * N + n;
            if(!(radii[idx * 2] > 0 && radii[idx * 2 + 1] > 0))
                continue;
            const float *vm      = viewmats + c * 16;
            const Cam cam        = load_cam(vm, Ks + c * 9);
            const float conic[3] = {conics[idx * 3], conics[idx * 3 + 1], conics[idx * 3 + 2]};
            const float vc[3]    = {v_conics[idx * s_c], v_conics[idx * s_c + 1], v_conics[idx * s_c + 2]};
            const bool has_comp  = v_compensations != nullptr;
            const ProjGrad g     = project_one_vjp(
                mean, cov, cam, W, H, eps2d, conic, v_means2d[idx * s_m2], v_means2d[idx * s_m2 + 1], v_depths ? v_depths[idx * s_d] : 0.f,
                vc, has_comp, has_comp ? compensations[idx] : 0.f, has_comp ? v_compensations[idx] : 0.f
            );
#pragma unroll
            for(int k = 0; k < 3; ++k)
                v_mean[k] += g.v_mean[k];
#pragma unroll
            for(int k = 0; k < 9; ++k)
                v_cov.m[k] += g.v_cov.m[k];
            // SH part: relu mask re-derived from the stored post-activation colour
            float vcol[3];
#pragma unroll
            for(int d = 0; d < 3; ++d)
                vcol[d] = colors[idx * 3 + d] > 0.f ? v_colors[idx * s_col + d] : 0.f;
            float dir[3];
            sh_view_dir(mean, vm, dir);
            const float inorm = 1.f / sqrtf(dir[0] * dir[0] + dir[1] * dir[1] + dir[2] * dir[2]);
            const float u[3]  = {dir[0] * inorm, dir[1] * inorm, dir[2] * inorm};
            float vu[3] = {0.f, 0.f, 0.f};
            // the coefficients are visited in address order: with 16-byte aligned rows they are fetched four at a time
            // into a rolling register (12 LDG.128 instead of 48 scalar loads -- the scalar stream stalled on lg_throttle)
            const bool vec4 = ((K * 3) & 3) == 0;
            float4 c4       = make_float4(0.f, 0.f, 0.f, 0.f);
            sh_visit<DEG, true>(u[0], u[1], u[2], [&](int k, const Dual<true> &Yk) {
                float gk = 0.f;
#pragma unroll
                for(int d = 0; d < 3; ++d)
                {
                    acc[k * 3 + d] += Yk.v * vcol[d];
                    const int i = k * 3 + d; // a compile-time constant once sh_visit is unrolled
                    float coef;
                    if(vec4)
                    {
                        if((i & 3) == 0)
                            c4 = ldg_nc_f4(reinterpret_cast<const float4 *>(cf) + (i >> 2));
                        coef = (i & 3) == 0 ? c4.x : ((i & 3) == 1 ? c4.y : ((i & 3) == 2 ? c4.z : c4.w));
                    }
                    else
                        coef = __ldg(cf + i);
                    gk += coef * vcol[d];
                }
                vu[0] += gk * Yk.x;
                vu[1] += gk * Yk.y;
                vu[2] += gk * Yk.z;
            });
            if(DEG >= 1)
            {
                const float dot = vu[0] * u[0] + vu[1] * u[1] + vu[2] * u[2];
#pragma unroll
                for(int j = 0; j < 3; ++j)
                    v_mean[j] += (vu[j] - dot * u[j]) * inorm;
            }
        }
#pragma unroll
        for(int k = 0; k < 3; ++k)
            v_means[n * 3 + k] = v_mean[k];
        float vq[4] = {0.f, 0.f, 0.f, 0.f}, vs[3] = {0.f, 0.f, 0.f};
        quat_scale_sym_vjp<false>(q, s, v_cov, vq, vs);
        *reinterpret_cast<float4 *>(v_quats + n * 4) = make_float4(vq[0], vq[1], vq[2], vq[3]);
#pragma unroll
        for(int k = 0; k < 3; ++k)
            v_scales[n * 3 + k] = vs[k];
        float *vsh = v_sh + n * K * 3;
        if(((K * 3) & 3) == 0 && (NB * 3) % 4 == 0)
        {
#pragma unroll
            for(int v = 0; v < NB * 3 / 4; ++v)
                reinterpret_cast<float4 *>(vsh)[v] = make_float4(acc[4 * v], acc[4 * v + 1], acc[4 * v + 2], acc[4 * v + 3]);
        }
        else
        {
#pragma unroll
            for(int k = 0; k < NB * 3; ++k)
                vsh[k] = acc[k];
        }
        for(int64_t k = NB * 3; k < K * 3; ++k)
            vsh[k] = 0.f;
    }
    else if(n < N)
    {
#pragma unroll
        for(int k = 0; k < 3; ++k)
            v_means[n * 3 + k] = 0.f, v_scales[n * 3 + k] = 0.f;
        *reinterpret_cast<float4 *>(v_quats + n * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    // zero rows of v_sh, warp-cooperatively: lane l writes chunk l, l + 32, ... of the warp's 32-row block
    const unsigned zero_rows = __ballot_sync(0xffffffffu, n < N && !seen);
    if(seen_bits != nullptr)
    { // one bit per gaussian: "has a non-trivial gradient row on this rank" (input of the row-sparse all-reduce)
        const unsigned seen_rows = __ballot_sync(0xffffffffu, seen);
        if(lane == 0 && n < N)
            seen_bits[n >> 5] = seen_rows;
    }
    if(zero_rows != 0u)
    {
        const int64_t row0 = n - lane; // first row of this warp
        const int64_t W3   = K * 3;
        if((W3 & 3) == 0)
        {
            const int per_row = (int)(W3 >> 2);
            float4 *base      = reinterpret_cast<float4 *>(v_sh + row0 * W3);
            for(int f = (int)lane; f < 32 * per_row; f += 32)
                if((zero_rows >> (f / per_row)) & 1u)
                    base[f] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        else
        {
            float *base = v_sh + row0 * W3;
            for(int f = (int)lane; f < 32 * (int)W3; f += 32)
                if((zero_rows >> (f / (int)W3)) & 1u)
                    base[f] = 0.f;
        }
    }
}

// ------------------------------------------------------------------ packed (compacting) projection
// Reference: csrc/ProjectionEWA3DGSPacked.cu:39-284 (two passes over the same kernel: count the visible
// gaussians per block, scan, then write the visible rows back to back), host csrc/Projection.cpp:858-1060.
// Rows come out in ascending (batch, camera, gaussian) order; nothing of size B*C*N is ever allocated.
template<int CAM, bool EMIT>
__global__ void __launch_bounds__(kThreads) projection_packed_kernel(
    int64_t C, int64_t N, const float *__restrict__ means, const float *__restrict__ covars,
    const float *__restrict__ quats, const float *__restrict__ scales, const float *__restrict__ opacities,
    const float *__restrict__ viewmats, const float *__restrict__ Ks, uint32_t W, uint32_t H, float eps2d,
    float near_plane, float far_plane, float radius_clip, bool want_comp, const int32_t *__restrict__ block_accum,
    int32_t *__restrict__ block_cnts, int32_t *__restrict__ indptr, int64_t *__restrict__ batch_ids,
    int64_t *__restrict__ camera_ids, int64_t *__restrict__ gaussian_ids, int32_t *__restrict__ radii,
    float *__restrict__ means2d, float *__restrict__ depths, float *__restrict__ conics, float *__restrict__ compensations
)
{
    __shared__ int warp_cnt[kThreads / 32];
    const int64_t row = blockIdx.y; // (b, c)
    const int64_t b = row / C, c = row % C;
    const int64_t n   = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    Proj p;
    p.rx = p.ry = 0;
    if(n < N)
    {
        const int64_t bn = b * N + n;
        const Cam cam = load_cam(viewmats + row * 16, Ks + row * 9);
        const float mean[3] = {means[bn * 3], means[bn * 3 + 1], means[bn * 3 + 2]};
        M3 cov;
        if(covars)
            cov = load_cov6(covars + bn * 6);
        else
        {
            const float q[4] = {quats[bn * 4], quats[bn * 4 + 1], quats[bn * 4 + 2], quats[bn * 4 + 3]};
            const float s[3] = {scales[bn * 3], scales[bn * 3 + 1], scales[bn * 3 + 2]};
            cov = quat_scale_to_sym<false>(q, s);
        }
        float op = 0.f;
        if(opacities)
            op = opacities[bn];
        p = project_one<CAM>(mean, cov, opacities ? &op : nullptr, cam, W, H, eps2d, near_plane, far_plane, radius_clip, want_comp);
    }
    const bool vis       = p.rx > 0 && p.ry > 0;
    const unsigned ball  = __ballot_sync(0xffffffffu, vis);
    if(lane == 0)
        warp_cnt[warp] = __popc(ball);
    __syncthreads();
    int before = 0, total = 0;
#pragma unroll
    for(int w = 0; w < kThreads / 32; ++w)
    {
        before += (w < (int)warp) ? warp_cnt[w] : 0;
        total += warp_cnt[w];
    }
    const int64_t blk = row * gridDim.x + blockIdx.x;
    if constexpr(!EMIT)
    {
        if(threadIdx.x == 0)
            block_cnts[blk] = total;
    }
    else
    {
        const int32_t base = blk == 0 ? 0 : block_accum[blk - 1];
        if(threadIdx.x == 0)
        {
            if(blockIdx.x == 0)
                indptr[row] = base;
            if(blk == (int64_t)gridDim.x * gridDim.y - 1)
                indptr[gridDim.y] = base + total;
        }
        if(vis)
        {
            const int64_t o = (int64_t)base + before + __popc(ball & ((1u << lane) - 1u));
            batch_ids[o]    = b;
            camera_ids[o]   = c;
            gaussian_ids[o] = n;
            reinterpret_cast<int2 *>(radii)[o]     = make_int2(p.rx, p.ry);
            reinterpret_cast<float2 *>(means2d)[o] = make_float2(p.mx, p.my);
            depths[o]         = p.depth;
            conics[o * 3]     = p.ca;
            conics[o * 3 + 1] = p.cb;
            conics[o * 3 + 2] = p.cc;
            if(compensations)
                compensations[o] = p.comp;
        }
    }
}

// One thread per packed row.  dense_out: gradients are summed into the [B*N, *] tensors with float atomics (rows
// of one gaussian differ only in their camera); otherwise (sparse_grad) every row writes its own [nnz, *] entry.
// Reference: csrc/ProjectionEWA3DGSPacked.cu:385-640.
template<int CAM>
__global__ void __launch_bounds__(kThreads) projection_packed_bwd_kernel(
    int64_t nnz, int64_t C, int64_t N, const float *__restrict__ means, const float *__restrict__ covars,
    const float *__restrict__ quats, const float *__restrict__ scales, const float *__restrict__ viewmats,
    const float *__restrict__ Ks, uint32_t W, uint32_t H, float eps2d, const int64_t *__restrict__ batch_ids,
    const int64_t *__restrict__ camera_ids, const int64_t *__restrict__ gaussian_ids, const float *__restrict__ conics,
    const float *__restrict__ compensations, const float *__restrict__ v_means2d, int64_t s_m2,
    const float *__restrict__ v_depths, int64_t s_d, const float *__restrict__ v_conics, int64_t s_c,
    const float *__restrict__ v_compensations, bool dense_out, float *__restrict__ v_means, float *__restrict__ v_covars,
    float *__restrict__ v_quats, float *__restrict__ v_scales, float *__restrict__ v_viewmats
)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if(i >= nnz)
        return;
    const int64_t b = batch_ids[i], c = camera_ids[i], n = gaussian_ids[i];
    const int64_t bn = b * N + n, row = b * C + c;
    const Cam cam = load_cam(viewmats + row * 16, Ks + row * 9);
    const float mean[3] = {means[bn * 3], means[bn * 3 + 1], means[bn * 3 + 2]};
    float q[4] = {1.f, 0.f, 0.f, 0.f}, s[3] = {1.f, 1.f, 1.f};
    M3 cov;
    if(covars)
        cov = load_cov6(covars + bn * 6);
    else
    {
#pragma unroll
        for(int k = 0; k < 4; ++k)
            q[k] = quats[bn * 4 + k];
#pragma unroll
        for(int k = 0; k < 3; ++k)
            s[k] = scales[bn * 3 + k];
        cov = quat_scale_to_sym<false>(q, s);
    }
    const float conic[3] = {conics[i * 3], conics[i * 3 + 1], conics[i * 3 + 2]};
    const float vc[3]    = {v_conics[i * s_c], v_conics[i * s_c + 1], v_conics[i * s_c + 2]};
    const bool has_comp  = v_compensations != nullptr;
    const ProjGrad g     = project_one_vjp<CAM>(
        mean, cov, cam, W, H, eps2d, conic, v_means2d[i * s_m2], v_means2d[i * s_m2 + 1], v_depths[i * s_d], vc, has_comp,
        has_comp ? compensations[i] : 0.f, has_comp ? v_compensations[i] : 0.f
    );
    const int64_t o = dense_out ? bn : i;
    float out[10];
    int n_out;
    out[0] = g.v_mean[0], out[1] = g.v_mean[1], out[2] = g.v_mean[2];
    if(covars)
    {
        out[3] = g.v_cov.m[0], out[4] = g.v_cov.m[1] + g.v_cov.m[3], out[5] = g.v_cov.m[2] + g.v_cov.m[6];
        out[6] = g.v_cov.m[4], out[7] = g.v_cov.m[5] + g.v_cov.m[7], out[8] = g.v_cov.m[8];
        n_out  = 9;
    }
    else
    {
        float vq[4] = {0.f, 0.f, 0.f, 0.f}, vs[3] = {0.f, 0.f, 0.f};
        quat_scale_sym_vjp<false>(q, s, g.v_cov, vq, vs);
        out[3] = vq[0], out[4] = vq[1], out[5] = vq[2], out[6] = vq[3];
        out[7] = vs[0], out[8] = vs[1], out[9] = vs[2];
        n_out  = 10;
    }
    float *dst[10];
#pragma unroll
    for(int k = 0; k < 3; ++k)
        dst[k] = v_means + o * 3 + k;
    if(covars)
    {
#pragma unroll
        for(int k = 0; k < 6; ++k)
            dst[3 + k] = v_covars + o * 6 + k;
    }
    else
    {
#pragma unroll
        for(int k = 0; k < 4; ++k)
            dst[3 + k] = v_quats + o * 4 + k;
#pragma unroll
        for(int k = 0; k < 3; ++k)
            dst[7 + k] = v_scales + o * 3 + k;
    }
#pragma unroll
    for(int k = 0; k < 10; ++k)
        if(k < n_out)
        {
            if(dense_out)
                atomicAdd(dst[k], out[k]);
            else
                *dst[k] = out[k];
        }
    if(v_viewmats)
    { // v_R = v_pc mean^T + v_covc R cov^T + v_covc^T R cov ; v_t = v_pc
        const M3 A2 = mul_bt(mul(g.v_covc, cam.R), cov);
        const M3 B2 = mul(mul_at(g.v_covc, cam.R), cov);
#pragma unroll
        for(int r = 0; r < 3; ++r)
        {
#pragma unroll
            for(int j = 0; j < 3; ++j)
                atomicAdd(v_viewmats + row * 16 + r * 4 + j, g.v_pc[r] * mean[j] + A2.m[r * 3 + j] + B2.m[r * 3 + j]);
            atomicAdd(v_viewmats + row * 16 + r * 4 + 3, g.v_pc[r]);
        }
    }
}

// ------------------------------------------------------------------ tile intersection
// Enumerates the tiles of one gaussian in the reference's emit order, calling f(tile_id).
// AccuTile / SNUGBOX (csrc/IntersectTile.cu:83-207, 288-373) or the radius AABB (:374-463).
template<class F>
__device__ __forceinline__ int tiles_of_gaussian(
    float mx, float my, int rx, int ry, const float *conic, const float *opacity, uint32_t tile_size, uint32_t tw,
    uint32_t th, F &&f
)
{
    if(rx <= 0 || ry <= 0)
        return 0;
    int count      = 0;
    const float ts = (float)tile_size;
    auto clampi    = [](int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); };
    if(conic != nullptr && opacity != nullptr)
    {
        const float A = conic[0], Bc = conic[1], Cc = conic[2];
        const float disc = Bc * Bc - A * Cc;
        float t          = 2.f * exact_log(*opacity / kAlphaThreshold);
        const float cap  = kGaussianExtend * kGaussianExtend;
        t                = t < cap ? t : cap;
        const float ntd  = -t / disc;
        const float xe = sqrtf(ntd * Cc), ye = sqrtf(ntd * A);
        const float bminx = mx - xe, bminy = my - ye, bmaxx = mx + xe, bmaxy = my + ye;
        const float BxC = Bc * xe / Cc, ByA = Bc * ye / A;
        const float argminx = my + BxC, argminy = mx + ByA, argmaxx = my - BxC, argmaxy = mx - ByA;
        const int rminx = clampi((int)(bminx / ts), 0, (int)tw), rminy = clampi((int)(bminy / ts), 0, (int)th);
        const int rmaxx = clampi((int)(bmaxx / ts + 1.f), 0, (int)tw), rmaxy = clampi((int)(bmaxy / ts + 1.f), 0, (int)th);
        const int ys = rmaxy - rminy, xs = rmaxx - rminx;
        if(ys * xs == 0)
            return 0;
        const bool isY = ys < xs;
        const int ru0 = isY ? rminy : rminx, ru1 = isY ? rmaxy : rmaxx, rv0 = isY ? rminx : rminy, rv1 = isY ? rmaxx : rmaxy;
        const float bminu = isY ? bminy : bminx, bmaxu = isY ? bmaxy : bmaxx;
        const float bminv = isY ? bminx : bminy, bmaxv = isY ? bmaxx : bmaxy;
        const float amin_v = isY ? argminx : argminy, amax_v = isY ? argmaxx : argmaxy;
        const float pu = isY ? my : mx, pv = isY ? mx : my, coeff = isY ? A : Cc;
        auto line = [&](float coord, float &lo, float &hi) {
            const float h  = coord - pu;
            const float sq = sqrtf(disc * h * h + t * coeff);
            lo             = (-Bc * h - sq) / coeff + pv;
            hi             = (-Bc * h + sq) / coeff + pv;
        };
        float maxlo = bmaxv, maxhi = bminv, minlo, minhi;
        float min_line = (float)ru0 * ts;
        if(bminu <= min_line)
            line(min_line, minlo, minhi);
        else
            minlo = maxlo, minhi = maxhi;
        for(int u = ru0; u < ru1; ++u)
        {
            const float max_line = min_line + ts;
            if(max_line <= bmaxu)
                line(max_line, maxlo, maxhi);
            const float emin = (min_line <= amin_v && amin_v < max_line) ? bminv : (minlo < maxlo ? minlo : maxlo);
            const float emax = (min_line <= amax_v && amax_v < max_line) ? bmaxv : (minhi > maxhi ? minhi : maxhi);
            const int e0 = (int)(emin / ts), e1 = (int)(emax / ts + 1.f);
            int v0 = e0 < rv1 ? e0 : rv1;
            v0     = v0 > rv0 ? v0 : rv0;
            int v1 = e1 > rv0 ? e1 : rv0;
            v1     = v1 < rv1 ? v1 : rv1;
            for(int v = v0; v < v1; ++v)
            {
                ++count;
                f(isY ? (int64_t)u * tw + v : (int64_t)v * tw + u);
            }
            minlo = maxlo, minhi = maxhi, min_line = max_line;
        }
    }
    else
    {
        const float trx = (float)rx / ts, try_ = (float)ry / ts, tx = mx / ts, ty = my / ts;
        const int x0 = clampi((int)floorf(tx - trx), 0, (int)tw), y0 = clampi((int)floorf(ty - try_), 0, (int)th);
        const int x1 = clampi((int)ceilf(tx + trx), 0, (int)tw), y1 = clampi((int)ceilf(ty + try_), 0, (int)th);
        for(int i = y0; i < y1; ++i)
            for(int j = x0; j < x1; ++j)
            {
                ++count;
                f((int64_t)i * tw + j);
            }
    }
    return count;
}

// `order` (optional): thread j handles row order[j] (the depth order of gsb200_isect_depth_order) and also
// writes its count to counts_in_order[j], the array the scan runs over.
__global__ void __launch_bounds__(kThreads) isect_count_kernel(
    int64_t total, const float *__restrict__ means2d, const int32_t *__restrict__ radii, const float *__restrict__ conics,
    const float *__restrict__ opacities, const int32_t *__restrict__ order, uint32_t tile_size, uint32_t tw, uint32_t th,
    int32_t *__restrict__ tiles_per_gauss, int32_t *__restrict__ counts_in_order
)
{
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if(j >= total)
        return;
    const int64_t i = order ? (int64_t)order[j] : j;
    const int2 r    = reinterpret_cast<const int2 *>(radii)[i];
    int cnt         = 0;
    if(r.x > 0 && r.y > 0)
    {
        const float2 m = reinterpret_cast<const float2 *>(means2d)[i];
        float cn[3] = {0.f, 0.f, 0.f}, op = 0.f;
        const bool accu = conics != nullptr && opacities != nullptr;
        if(accu)
            cn[0] = conics[i * 3], cn[1] = conics[i * 3 + 1], cn[2] = conics[i * 3 + 2], op = opacities[i];
        cnt = tiles_of_gaussian(m.x, m.y, r.x, r.y, accu ? cn : nullptr, accu ? &op : nullptr, tile_size, tw, th, [](int64_t) {});
    }
    tiles_per_gauss[i] = cnt;
    if(order)
        counts_in_order[j] = cnt;
}

// row-order count + the totals the host reads once: [0] = number of intersections, [1] = rows with tiles,
// [2] = the largest tile count of a row (picks the emit kernel)
__global__ void __launch_bounds__(kThreads) isect_count_totals_kernel(
    int64_t total, const float *__restrict__ means2d, const int32_t *__restrict__ radii, const float *__restrict__ conics,
    const float *__restrict__ opacities, uint32_t tile_size, uint32_t tw, uint32_t th, int32_t *__restrict__ tiles_per_gauss,
    unsigned long long *__restrict__ totals
)
{
    __shared__ unsigned long long s_tot[3];
    if(threadIdx.x < 3)
        s_tot[threadIdx.x] = 0ull;
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int cnt         = 0;
    if(i < total)
    {
        const int2 r = reinterpret_cast<const int2 *>(radii)[i];
        if(r.x > 0 && r.y > 0)
        {
            const float2 m = reinterpret_cast<const float2 *>(means2d)[i];
            float cn[3] = {0.f, 0.f, 0.f}, op = 0.f;
            const bool accu = conics != nullptr && opacities != nullptr;
            if(accu)
                cn[0] = conics[i * 3], cn[1] = conics[i * 3 + 1], cn[2] = conics[i * 3 + 2], op = opacities[i];
            cnt = tiles_of_gaussian(m.x, m.y, r.x, r.y, accu ? cn : nullptr, accu ? &op : nullptr, tile_size, tw, th, [](int64_t) {});
        }
        tiles_per_gauss[i] = cnt;
    }
    const int wsum         = __reduce_add_sync(0xffffffffu, cnt);
    const int wmax         = __reduce_max_sync(0xffffffffu, cnt);
    const unsigned nonzero = __ballot_sync(0xffffffffu, cnt > 0);
    if((threadIdx.x & 31) == 0 && nonzero != 0u)
    {
        atomicAdd(&s_tot[0], (unsigned long long)wsum);
        atomicAdd(&s_tot[1], (unsigned long long)__popc(nonzero));
        atomicMax(&s_tot[2], (unsigned long long)wmax);
    }
    __syncthreads();
    if(threadIdx.x < 2 && s_tot[threadIdx.x] != 0ull)
        atomicAdd(&totals[threadIdx.x], s_tot[threadIdx.x]);
    if(threadIdx.x == 2 && s_tot[2] != 0ull)
        atomicMax(&totals[2], s_tot[2]);
}

// Key of one (gaussian, tile) intersection.  int64_t: the reference's isect id, (image | tile) << 32 | depth bits
// (csrc/IntersectTile.cu:925-988).  uint16_t / uint32_t: the dense tile id image * n_tiles + tile alone -- the rows are
// emitted in depth order already, so the S-sized sort only needs those bits, and moving 2 + 4 instead of 8 + 4 bytes per
// intersection and pass halves its traffic (the 64-bit ids are rebuilt on demand: isect_ids_from_tilekeys_kernel).
template<class KeyT>
struct IsectKey
{
    uint32_t base;
    __device__ __forceinline__ IsectKey(int64_t image, uint32_t, uint32_t, int64_t n_tiles) : base((uint32_t)(image * n_tiles)) {}
    __device__ __forceinline__ KeyT operator()(int64_t tile) const { return (KeyT)(base + (uint32_t)tile); }
};
template<>
struct IsectKey<int64_t>
{
    int64_t hi_db;
    __device__ __forceinline__ IsectKey(int64_t image, uint32_t dbits, uint32_t tile_n_bits, int64_t)
        : hi_db((image << (32 + tile_n_bits)) | (int64_t)dbits)
    {
    }
    __device__ __forceinline__ int64_t operator()(int64_t tile) const { return hi_db | (tile << 32); }
};

// Capacity-bounded emission (gsb200_isect_sorted): the launch covers `total` = capacity row slots and writes into
// capacity-sized outputs, while the real counts sit in device memory (totals[0] intersections, totals[1] rows with
// tiles).  Returns the number of real row slots; the slots between the real intersections and the capacity get padding
// pairs (largest key: the stable sort leaves them behind every real pair; row 0: any valid row).
template<class KeyT>
__device__ __forceinline__ int64_t emit_bounded_rows(
    int64_t j, int64_t n_threads, int64_t total, const int64_t *__restrict__ totals, int64_t cap_isects,
    KeyT *__restrict__ isect_ids, int32_t *__restrict__ flatten_ids
)
{
    const int64_t n_real = totals[0] < cap_isects ? totals[0] : cap_isects;
    for(int64_t s = n_real + j; s < cap_isects; s += n_threads)
    {
        isect_ids[s]   = (KeyT)~(KeyT)0;
        flatten_ids[s] = 0;
    }
    return totals[1] < total ? totals[1] : total;
}

template<class KeyT>
__global__ void __launch_bounds__(kThreads) isect_emit_kernel(
    int64_t total, int64_t N, const float *__restrict__ means2d, const int32_t *__restrict__ radii,
    const float *__restrict__ depths, const float *__restrict__ conics, const float *__restrict__ opacities,
    const int64_t *__restrict__ cum_tiles, const int64_t *__restrict__ image_ids, const int32_t *__restrict__ order,
    uint32_t tile_size, uint32_t tw, uint32_t th, uint32_t tile_n_bits, KeyT *__restrict__ isect_ids,
    int32_t *__restrict__ flatten_ids, const int64_t *__restrict__ totals = nullptr, int64_t cap_isects = 0
)
{
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if(totals != nullptr)
        total = emit_bounded_rows<KeyT>(j, (int64_t)gridDim.x * blockDim.x, total, totals, cap_isects, isect_ids, flatten_ids);
    if(j >= total)
        return;
    if(totals != nullptr && cum_tiles[j] > cap_isects)
        return; // beyond the speculative capacity: the host sees totals[0] > capacity and redoes the stage
    const int64_t i = order ? (int64_t)order[j] : j;
    const int2 r    = reinterpret_cast<const int2 *>(radii)[i];
    if(r.x <= 0 || r.y <= 0)
        return;
    const float2 m = reinterpret_cast<const float2 *>(means2d)[i];
    float cn[3] = {0.f, 0.f, 0.f}, op = 0.f;
    const bool accu = conics != nullptr && opacities != nullptr;
    if(accu)
        cn[0] = conics[i * 3], cn[1] = conics[i * 3 + 1], cn[2] = conics[i * 3 + 2], op = opacities[i];
    int64_t cur         = (j == 0) ? 0 : cum_tiles[j - 1];
    // packed rows carry their image id
    const IsectKey<KeyT> key(image_ids ? image_ids[i] : (i / N), __float_as_uint(depths[i]), tile_n_bits, (int64_t)tw * th);
    tiles_of_gaussian(m.x, m.y, r.x, r.y, accu ? cn : nullptr, accu ? &op : nullptr, tile_size, tw, th, [&](int64_t tile) {
        isect_ids[cur]   = key(tile);
        flatten_ids[cur] = (int32_t)i;
        ++cur;
    });
}

// ---- warp-cooperative emit.  One thread per gaussian with a loop over ITS tiles (isect_emit_kernel) leaves a warp
// waiting for its largest gaussian and writes 8 + 4 byte records at lane-dependent strides: at S = 20 M (large
// screen-space gaussians) it took 444 us for 240 MB of output.  Here a gaussian with more than kSmallTiles tiles is
// handed to its whole warp: the tile interval of every tile row is a closed form of the row index (the incremental
// scheme of tiles_of_gaussian only carries the previous row's far line over as the next row's near line), so lane r
// computes row ru0 + r, a warp scan places the rows, and the lanes then write the tiles round-robin -- consecutive
// lanes, consecutive addresses -- in the same order as the sequential enumeration.
constexpr int kSmallTiles = 64; // measured: below ~2 warps' worth of tiles the per-gaussian warp hand-over costs more than it saves

struct AccuGauss
{
    float mx, my, A, Bc, Cc, disc, t, ts;
    float bminu, bmaxu, bminv, bmaxv, amin_v, amax_v, pu, pv, coeff;
    int ru0, ru1, rv0, rv1;
    bool isY, accu, empty;
    int x0, x1; // AABB path
};

__device__ __forceinline__ AccuGauss accu_setup(
    float mx, float my, int rx, int ry, bool accu, float A, float Bc, float Cc, float opacity, uint32_t tile_size,
    uint32_t tw, uint32_t th
)
{
    AccuGauss g;
    g.mx = mx, g.my = my, g.A = A, g.Bc = Bc, g.Cc = Cc, g.accu = accu, g.ts = (float)tile_size;
    g.empty     = rx <= 0 || ry <= 0;
    g.ru0 = g.ru1 = g.rv0 = g.rv1 = g.x0 = g.x1 = 0;
    g.isY                                        = false;
    auto clampi = [](int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); };
    if(g.empty)
        return g;
    const float ts = g.ts;
    if(accu)
    {
        g.disc          = Bc * Bc - A * Cc;
        float t         = 2.f * exact_log(opacity / kAlphaThreshold);
        const float cap = kGaussianExtend * kGaussianExtend;
        g.t             = t < cap ? t : cap;
        const float ntd = -g.t / g.disc;
        const float xe = sqrtf(ntd * Cc), ye = sqrtf(ntd * A);
        const float bminx = mx - xe, bminy = my - ye, bmaxx = mx + xe, bmaxy = my + ye;
        const float BxC = Bc * xe / Cc, ByA = Bc * ye / A;
        const float argminx = my + BxC, argminy = mx + ByA, argmaxx = my - BxC, argmaxy = mx - ByA;
        const int rminx = clampi((int)(bminx / ts), 0, (int)tw), rminy = clampi((int)(bminy / ts), 0, (int)th);
        const int rmaxx = clampi((int)(bmaxx / ts + 1.f), 0, (int)tw), rmaxy = clampi((int)(bmaxy / ts + 1.f), 0, (int)th);
        const int ys = rmaxy - rminy, xs = rmaxx - rminx;
        if(ys * xs == 0)
        {
            g.empty = true;
            return g;
        }
        g.isY = ys < xs;
        g.ru0 = g.isY ? rminy : rminx, g.ru1 = g.isY ? rmaxy : rmaxx, g.rv0 = g.isY ? rminx : rminy, g.rv1 = g.isY ? rmaxx : rmaxy;
        g.bminu = g.isY ? bminy : bminx, g.bmaxu = g.isY ? bmaxy : bmaxx;
        g.bminv = g.isY ? bminx : bminy, g.bmaxv = g.isY ? bmaxx : bmaxy;
        g.amin_v = g.isY ? argminx : argminy, g.amax_v = g.isY ? argmaxx : argmaxy;
        g.pu = g.isY ? my : mx, g.pv = g.isY ? mx : my, g.coeff = g.isY ? A : Cc;
    }
    else
    {
        const float trx = (float)rx / ts, try_ = (float)ry / ts, tx = mx / ts, ty = my / ts;
        g.x0 = clampi((int)floorf(tx - trx), 0, (int)tw), g.ru0 = clampi((int)floorf(ty - try_), 0, (int)th);
        g.x1 = clampi((int)ceilf(tx + trx), 0, (int)tw), g.ru1 = clampi((int)ceilf(ty + try_), 0, (int)th);
        g.isY = true; // rows are tile rows
        if(g.ru1 <= g.ru0 || g.x1 <= g.x0)
            g.empty = true;
    }
    return g;
}

// tile interval [v0, v1) of row u (ru0 <= u < ru1); identical, bit for bit, to what tiles_of_gaussian enumerates
__device__ __forceinline__ void accu_row(const AccuGauss &g, int u, int &v0, int &v1)
{
    if(!g.accu)
    {
        v0 = g.x0, v1 = g.x1;
        return;
    }
    const float ts = g.ts;
    auto line = [&](float coord, float &lo, float &hi) {
        const float h  = coord - g.pu;
        const float sq = sqrtf(g.disc * h * h + g.t * g.coeff);
        lo             = (-g.Bc * h - sq) / g.coeff + g.pv;
        hi             = (-g.Bc * h + sq) / g.coeff + g.pv;
    };
    const float min_line = (float)u * ts, max_line = min_line + ts;
    float minlo = g.bmaxv, minhi = g.bminv; // the sequential scheme's initial values
    if(u > g.ru0 || g.bminu <= min_line)
        line(min_line, minlo, minhi);
    float maxlo, maxhi;
    if(max_line <= g.bmaxu)
        line(max_line, maxlo, maxhi);
    else if(u > g.ru0)
        maxlo = minlo, maxhi = minhi; // the far line was not computed: the previous one is kept
    else
        maxlo = g.bmaxv, maxhi = g.bminv;
    const float emin = (min_line <= g.amin_v && g.amin_v < max_line) ? g.bminv : (minlo < maxlo ? minlo : maxlo);
    const float emax = (min_line <= g.amax_v && g.amax_v < max_line) ? g.bmaxv : (minhi > maxhi ? minhi : maxhi);
    const int e0 = (int)(emin / ts), e1 = (int)(emax / ts + 1.f);
    v0 = e0 < g.rv1 ? e0 : g.rv1;
    v0 = v0 > g.rv0 ? v0 : g.rv0;
    v1 = e1 > g.rv0 ? e1 : g.rv0;
    v1 = v1 < g.rv1 ? v1 : g.rv1;
    if(v1 < v0)
        v1 = v0;
}

template<class KeyT>
__global__ void __launch_bounds__(kThreads) isect_emit_coop_kernel(
    int64_t total, int64_t N, const float *__restrict__ means2d, const int32_t *__restrict__ radii,
    const float *__restrict__ depths, const float *__restrict__ conics, const float *__restrict__ opacities,
    const int64_t *__restrict__ cum_tiles, const int64_t *__restrict__ image_ids, const int32_t *__restrict__ order,
    uint32_t tile_size, uint32_t tw, uint32_t th, uint32_t tile_n_bits, KeyT *__restrict__ isect_ids,
    int32_t *__restrict__ flatten_ids, const int64_t *__restrict__ totals = nullptr, int64_t cap_isects = 0
)
{
    const int64_t j     = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned lane = threadIdx.x & 31;
    if(totals != nullptr)
        total = emit_bounded_rows<KeyT>(j, (int64_t)gridDim.x * blockDim.x, total, totals, cap_isects, isect_ids, flatten_ids);
    const bool active   = j < total && !(totals != nullptr && cum_tiles[j] > cap_isects);
    const int64_t i     = active ? (order ? (int64_t)order[j] : j) : 0;
    int2 r              = make_int2(0, 0);
    float2 m            = make_float2(0.f, 0.f);
    float cn0 = 0.f, cn1 = 0.f, cn2 = 0.f, op = 0.f;
    const bool accu = conics != nullptr && opacities != nullptr;
    int64_t cur = 0, img = 0;
    uint32_t dbits = 0;
    int cnt = 0;
    if(active)
    {
        r = reinterpret_cast<const int2 *>(radii)[i];
        if(r.x > 0 && r.y > 0)
        {
            m = reinterpret_cast<const float2 *>(means2d)[i];
            if(accu)
                cn0 = conics[i * 3], cn1 = conics[i * 3 + 1], cn2 = conics[i * 3 + 2], op = opacities[i];
            cur   = (j == 0) ? 0 : cum_tiles[j - 1];
            cnt   = (int)(cum_tiles[j] - cur);
            img   = image_ids ? image_ids[i] : (i / N);
            dbits = __float_as_uint(depths[i]);
        }
    }
    // small gaussians: the owning lane writes its few tiles
    if(cnt > 0 && cnt <= kSmallTiles)
    {
        float cn[3] = {cn0, cn1, cn2};
        const IsectKey<KeyT> key(img, dbits, tile_n_bits, (int64_t)tw * th);
        tiles_of_gaussian(m.x, m.y, r.x, r.y, accu ? cn : nullptr, accu ? &op : nullptr, tile_size, tw, th, [&](int64_t tile) {
            isect_ids[cur]   = key(tile);
            flatten_ids[cur] = (int32_t)i;
            ++cur;
        });
    }
    // large gaussians: one at a time, the whole warp
    uint32_t big = __ballot_sync(0xffffffffu, cnt > kSmallTiles);
    while(big)
    {
        const int src = __ffs(big) - 1;
        big &= big - 1;
        const float bmx = __shfl_sync(0xffffffffu, m.x, src), bmy = __shfl_sync(0xffffffffu, m.y, src);
        const int brx = __shfl_sync(0xffffffffu, r.x, src), bry = __shfl_sync(0xffffffffu, r.y, src);
        const float b0 = __shfl_sync(0xffffffffu, cn0, src), b1 = __shfl_sync(0xffffffffu, cn1, src);
        const float b2 = __shfl_sync(0xffffffffu, cn2, src), bop = __shfl_sync(0xffffffffu, op, src);
        const int64_t bcur = __shfl_sync(0xffffffffu, cur, src), bimg = __shfl_sync(0xffffffffu, img, src);
        const uint32_t bdb = __shfl_sync(0xffffffffu, dbits, src);
        const IsectKey<KeyT> bkey(bimg, bdb, tile_n_bits, (int64_t)tw * th);
        const int32_t bi  = (int32_t)__shfl_sync(0xffffffffu, i, src);
        const AccuGauss g = accu_setup(bmx, bmy, brx, bry, accu, b0, b1, b2, bop, tile_size, tw, th);
        if(g.empty)
            continue;
        int64_t base = bcur;
        for(int u0 = g.ru0; u0 < g.ru1; u0 += 32)
        {
            const int u = u0 + (int)lane;
            int v0 = 0, v1 = 0;
            if(u < g.ru1)
                accu_row(g, u, v0, v1);
            const int len = v1 - v0;
            int incl      = len;
#pragma unroll
            for(int o = 1; o < 32; o <<= 1)
            {
                const int up = __shfl_up_sync(0xffffffffu, incl, o);
                if((int)lane >= o)
                    incl += up;
            }
            const int excl  = incl - len;
            const int chunk = __shfl_sync(0xffffffffu, incl, 31);
            // tile k of this 32-row chunk: row = the last row with excl <= k (binary search over the lanes; the loop is
            // warp-uniform so that every shuffle sees all 32 lanes, only the stores are predicated)
            for(int k0 = 0; k0 < chunk; k0 += 32)
            {
                const int k = k0 + (int)lane;
                int row     = 0;
#pragma unroll
                for(int step = 16; step > 0; step >>= 1)
                {
                    const int probe = row + step; // <= 31
                    const int pe    = __shfl_sync(0xffffffffu, excl, probe);
                    if(pe <= k)
                        row = probe;
                }
                const int rex = __shfl_sync(0xffffffffu, excl, row);
                const int rv0 = __shfl_sync(0xffffffffu, v0, row);
                if(k < chunk)
                {
                    const int v        = rv0 + (k - rex);
                    const int uu       = u0 + row;
                    const int64_t tile = g.isY ? (int64_t)uu * tw + v : (int64_t)v * tw + uu;
                    isect_ids[base + k]   = bkey(tile);
                    flatten_ids[base + k] = bi;
                }
            }
            base += chunk;
        }
    }
}

// offsets[(image, tile)] = first sorted index of that tile's run.  One thread per sorted
// intersection; a thread that starts a new run also fills the empty tiles before it.
__global__ void __launch_bounds__(kThreads) isect_offsets_kernel(
    int64_t n_isects, const int64_t *__restrict__ isect_ids, int64_t total_tiles, int64_t n_tiles, uint32_t tile_n_bits,
    int32_t *__restrict__ offsets
)
{
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if(s >= n_isects)
        return;
    const int64_t mask = ((int64_t)1 << tile_n_bits) - 1;
    const int64_t hi   = isect_ids[s] >> 32;
    const int64_t id   = (hi >> tile_n_bits) * n_tiles + (hi & mask);
    int64_t prev       = -1;
    if(s > 0)
    {
        const int64_t hp = isect_ids[s - 1] >> 32;
        prev             = (hp >> tile_n_bits) * n_tiles + (hp & mask);
    }
    for(int64_t k = prev + 1; k <= id; ++k)
        offsets[k] = (int32_t)s;
    if(s == n_isects - 1)
        for(int64_t k = id + 1; k < total_tiles; ++k)
            offsets[k] = (int32_t)n_isects;
}
// ------------------------------------------------------------------ MCMC strategy ops ("next" row, SURVEY 8f.3)
// Relocation, Eq. 9 of "3D Gaussian Splatting as Markov Chain Monte Carlo" (reference:
// csrc/RelocationCUDA.cu:36-80): new opacity 1 - (1 - o)^(1/n) clamped to [min_opacity, 1 - eps]; new scale
// = o / sum_{i=1..n} sum_{k<i} C(i-1,k) (-1)^k / sqrt(k+1) o_new^(k+1) times the old scale.
__global__ void __launch_bounds__(kThreads) relocation_kernel(
    int64_t N, const float *__restrict__ opacities, const float *__restrict__ scales, const int32_t *__restrict__ ratios,
    const float *__restrict__ binoms, int n_max, float min_opacity, float *__restrict__ new_opacities,
    float *__restrict__ new_scales
)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if(i >= N)
        return;
    const int n   = ratios[i];
    const float o = opacities[i];
    float o_new   = 1.0f - powf(1.0f - o, 1.0f / (float)n);
    o_new         = fminf(fmaxf(o_new, min_opacity), 1.0f - 1.1920929e-07f);
    new_opacities[i] = o_new;
    float denom = 0.f;
    for(int r = 1; r <= n; ++r)
    {
        float p = o_new; // o_new^(k+1)
        float sign = 1.f;
        for(int k = 0; k < r; ++k)
        {
            denom += binoms[(r - 1) * n_max + k] * (sign / sqrtf((float)(k + 1))) * p;
            p *= o_new;
            sign = -sign;
        }
    }
    const float coeff = o / denom;
#pragma unroll
    for(int k = 0; k < 3; ++k)
        new_scales[i * 3 + k] = coeff * scales[i * 3 + k];
}

// positions += Sigma * (noise * sigmoid(-k (sigmoid(opacity_logit) - t)) * noise_scale), in place
// (reference: csrc/MCMCPerturbCUDA.cu:28-60).
__global__ void __launch_bounds__(kThreads) mcmc_perturb_kernel(
    int64_t N, float *__restrict__ positions, const float *__restrict__ quats, const float *__restrict__ scales_log,
    const float *__restrict__ opacities_logit, const float *__restrict__ noise, float noise_scale, float t, float k
)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if(i >= N)
        return;
    const float q[4] = {quats[i * 4], quats[i * 4 + 1], quats[i * 4 + 2], quats[i * 4 + 3]};
    const float s[3] = {expf(scales_log[i * 3]), expf(scales_log[i * 3 + 1]), expf(scales_log[i * 3 + 2])};
    const M3 cov     = quat_scale_to_sym<false>(q, s);
    const float dens = 1.f / (1.f + expf(-opacities_logit[i]));
    const float w    = (1.f / (1.f + expf(k * (dens - t)))) * noise_scale;
    const float nz[3] = {noise[i * 3] * w, noise[i * 3 + 1] * w, noise[i * 3 + 2] * w};
#pragma unroll
    for(int r = 0; r < 3; ++r)
        positions[i * 3 + r] += cov.m[r * 3 + 0] * nz[0] + cov.m[r * 3 + 1] * nz[1] + cov.m[r * 3 + 2] * nz[2];
}

// Selective Adam step (no bias correction), in place; rows whose `valid` flag is 0 are left untouched
// (reference: csrc/AdamCUDA.cu:34-70, gsplat/optimizers/selective_adam.py).  One thread per element.
__global__ void __launch_bounds__(kThreads) adam_kernel(
    int64_t total, int64_t D, float *__restrict__ param, const float *__restrict__ grad, float *__restrict__ exp_avg,
    float *__restrict__ exp_avg_sq, const uint8_t *__restrict__ valid, float lr, float b1, float b2, float eps
)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if(i >= total)
        return;
    if(valid != nullptr && !valid[i / D])
        return;
    const float g = grad[i];
    const float m = b1 * exp_avg[i] + (1.0f - b1) * g;
    const float v = b2 * exp_avg_sq[i] + (1.0f - b2) * g * g;
    param[i] += -lr * m / (sqrtf(v) + eps);
    exp_avg[i]    = m;
    exp_avg_sq[i] = v;
}
} // namespace gsb

// =====================================================================================================
// C ABI
using namespace gsb;

extern "C" int gsb200_quat_scale_to_covar_preci_fwd(
    int64_t N, const float *quats, const float *scales, int triu, float *covars, float *precis, void *stream
)
{
    if(N < 0 || (N > 0 && (!quats || !scales)))
        return GSB200_E_INVALID;
    if(N == 0 || (!covars && !precis))
        return GSB200_OK;
    quat_scale_fwd_kernel<<<grid_for(N, kThreads), kThreads, 0, (cudaStream_t)stream>>>(N, quats, scales, triu != 0, covars, precis);
    return check_launch();
}

extern "C" int gsb200_quat_scale_to_covar_preci_bwd(
    int64_t N, const float *quats, const float *scales, int triu, const float *v_covars, const float *v_precis,
    float *v_quats, float *v_scales, void *stream
)
{
    if(N < 0 || (N > 0 && (!quats || !scales || !v_quats || !v_scales)))
        return GSB200_E_INVALID;
    if(N == 0)
        return GSB200_OK;
    quat_scale_bwd_kernel<<<grid_for(N, kThreads), kThreads, 0, (cudaStream_t)stream>>>(
        N, quats, scales, triu != 0, v_covars, v_precis, v_quats, v_scales
    );
    return check_launch();
}

extern "C" int gsb200_projection_fwd(
    int64_t B, int64_t C, int64_t N, const float *means, const float *covars, const float *quats, const float *scales,
    const float *opacities, const float *viewmats, const float *Ks, uint32_t image_width, uint32_t image_height,
    float eps2d, float near_plane, float far_plane, float radius_clip, int camera_model, int32_t *radii, float *means2d,
    float *depths, float *conics, float *compensations, void *stream
)
{
    if(B < 0 || C < 0 || N < 0)
        return GSB200_E_INVALID;
    if(camera_model < 0 || camera_model > 2) // ftheta / lidar are other pipelines (3DGUT), not built
        return GSB200_E_UNSUPPORTED;
    const int64_t total = B * C * N;
    if(total == 0)
        return GSB200_OK;
    if(!means || !viewmats || !Ks || !radii || !means2d || !depths || !conics)
        return GSB200_E_INVALID;
    if(!covars && (!quats || !scales))
        return GSB200_E_INVALID;
#define GSB_LAUNCH(CAM)                                                                                                \
    projection_fwd_kernel<CAM><<<grid_for(total, kThreads), kThreads, 0, (cudaStream_t)stream>>>(                        \
        B, C, N, means, covars, quats, scales, opacities, viewmats, Ks, image_width, image_height, eps2d, near_plane,   \
        far_plane, radius_clip, radii, means2d, depths, conics, compensations                                           \
    )
    if(camera_model == kCamPinhole)
        GSB_LAUNCH(kCamPinhole);
    else if(camera_model == kCamOrtho)
        GSB_LAUNCH(kCamOrtho);
    else
        GSB_LAUNCH(kCamFisheye);
#undef GSB_LAUNCH
    return check_launch();
}

extern "C" int gsb200_projection_bwd(
    int64_t B, int64_t C, int64_t N, const float *means, const float *covars, const float *quats, const float *scales,
    const float *viewmats, const float *Ks, uint32_t image_width, uint32_t image_height, float eps2d, int camera_model,
    const int32_t *radii, const float *conics, const float *compensations, const float *v_means2d,
    int64_t v_means2d_stride, const float *v_depths, int64_t v_depths_stride, const float *v_conics,
    int64_t v_conics_stride, const float *v_compensations, float *v_means, float *v_covars, float *v_quats,
    float *v_scales, float *v_viewmats, void *stream
)
{
    if(B < 0 || C < 0 || N < 0)
        return GSB200_E_INVALID;
    if(camera_model < 0 || camera_model > 2)
        return GSB200_E_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    if(v_viewmats && B * C > 0)
        GSB_CUDA_TRY(cudaMemsetAsync(v_viewmats, 0, sizeof(float) * 16 * (size_t)(B * C), st));
    if(B * N == 0)
        return GSB200_OK;
    if(!means || !viewmats || !Ks || !radii || !conics || !v_means2d || !v_depths || !v_conics || !v_means)
        return GSB200_E_INVALID;
    if(covars ? !v_covars : (!quats || !scales || !v_quats || !v_scales))
        return GSB200_E_INVALID;
    if(v_compensations && !compensations)
        return GSB200_E_INVALID;
#define GSB_LAUNCH(CAM)                                                                                                \
    projection_bwd_kernel<CAM><<<grid_for(B * N, kThreads), kThreads, 0, st>>>(                                          \
        B, C, N, means, covars, quats, scales, viewmats, Ks, image_width, image_height, eps2d, radii, conics,           \
        compensations, v_means2d, v_means2d_stride, v_depths, v_depths_stride, v_conics, v_conics_stride,               \
        v_compensations, v_means, v_covars, v_quats, v_scales, v_viewmats                                               \
    )
    if(camera_model == kCamPinhole)
        GSB_LAUNCH(kCamPinhole);
    else if(camera_model == kCamOrtho)
        GSB_LAUNCH(kCamOrtho);
    else
        GSB_LAUNCH(kCamFisheye);
#undef GSB_LAUNCH
    return check_launch();
}

#define GSB_DEG_SWITCH(deg, CALL)  \
    switch(deg)                    \
    {                              \
    case 0: { CALL(0); } break;    \
    case 1: { CALL(1); } break;    \
    case 2: { CALL(2); } break;    \
    case 3: { CALL(3); } break;    \
    case 4: { CALL(4); } break;    \
    default: return GSB200_E_INVALID; \
    }

extern "C" int gsb200_sh_fwd(
    int64_t B, int64_t C, int64_t N, int64_t K, int64_t D, int degrees_to_use, const float *means,
    const float *viewmats, const float *coeffs, const uint8_t *masks, float *colors, void *stream
)
{
    if(B < 0 || C < 0 || N < 0 || K <= 0 || D <= 0 || degrees_to_use < 0 || degrees_to_use > 4
       || (int64_t)(degrees_to_use + 1) * (degrees_to_use + 1) > K)
        return GSB200_E_INVALID;
    const int64_t total = B * C * N;
    if(total == 0)
        return GSB200_OK;
    if(!means || !viewmats || !coeffs || !colors)
        return GSB200_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
#define CALL(d) sh_fwd_kernel<d><<<grid_for(total, kThreads), kThreads, 0, st>>>(B, C, N, K, D, means, viewmats, coeffs, masks, colors)
    GSB_DEG_SWITCH(degrees_to_use, CALL)
#undef CALL
    return check_launch();
}

extern "C" int gsb200_sh_bwd(
    int64_t B, int64_t C, int64_t N, int64_t K, int64_t D, int degrees_to_use, const float *means,
    const float *viewmats, const float *coeffs, const uint8_t *masks, const float *v_colors, float *v_coeffs,
    float *v_means, float *v_dirsum, void *stream
)
{
    if(B < 0 || C < 0 || N < 0 || K <= 0 || D <= 0 || degrees_to_use < 0 || degrees_to_use > 4
       || (int64_t)(degrees_to_use + 1) * (degrees_to_use + 1) > K)
        return GSB200_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    if(v_means && B * N > 0)
        GSB_CUDA_TRY(cudaMemsetAsync(v_means, 0, sizeof(float) * 3 * (size_t)(B * N), st));
    if(v_dirsum && B * C > 0)
        GSB_CUDA_TRY(cudaMemsetAsync(v_dirsum, 0, sizeof(float) * 3 * (size_t)(B * C), st));
    if(N == 0)
        return GSB200_OK;
    if(!means || !viewmats || !coeffs || !v_colors || !v_coeffs)
        return GSB200_E_INVALID;
#define CALL(d) sh_bwd_kernel<d><<<grid_for(N * D, kThreads), kThreads, 0, st>>>(B, C, N, K, D, means, viewmats, coeffs, masks, v_colors, v_coeffs, v_means, v_dirsum)
    GSB_DEG_SWITCH(degrees_to_use, CALL)
#undef CALL
    return check_launch();
}

extern "C" int gsb200_project_sh_fwd(
    int64_t C, int64_t N, int64_t K, int degrees_to_use, const float *means, const float *quats, const float *scales,
    const float *opacities, const float *sh_coeffs, const float *viewmats, const float *Ks, uint32_t image_width,
    uint32_t image_height, float eps2d, float near_plane, float far_plane, float radius_clip, int calc_compensations,
    int32_t *radii, float *means2d, float *depths, float *conics, float *compensations, float *colors, void *stream
)
{
    if(C < 0 || N < 0 || K <= 0 || degrees_to_use < 0 || degrees_to_use > 4
       || (int64_t)(degrees_to_use + 1) * (degrees_to_use + 1) > K)
        return GSB200_E_INVALID;
    if(C * N == 0)
        return GSB200_OK;
    if(!means || !quats || !scales || !opacities || !sh_coeffs || !viewmats || !Ks || !radii || !means2d || !depths
       || !conics || !colors || (calc_compensations && !compensations))
        return GSB200_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    float *comp     = calc_compensations ? compensations : nullptr;
#define CALL(d)                                                                                                   \
    project_sh_fwd_kernel<d, false><<<grid_for(C * N, kThreads), kThreads, 0, st>>>(                              \
        C, N, K, means, quats, scales, opacities, sh_coeffs, viewmats, Ks, image_width, image_height, eps2d,      \
        near_plane, far_plane, radius_clip, radii, means2d, depths, conics, comp, colors, 0u, 0u, 0u, nullptr,    \
        nullptr, nullptr                                                                                          \
    )
    GSB_DEG_SWITCH(degrees_to_use, CALL)
#undef CALL
    return check_launch();
}

// gsb200_project_sh_fwd (no compensations) + the per-row tile counts / totals of gsb200_isect_count_totals (AccuTile test
// on the row's conic and INPUT opacity) + the 64-byte compositing row records for gsb200_raster_fwd_rows.
// row_records: 64 * C * N bytes, 16-byte aligned; only rows with radii > 0 are written.  totals: int64 [3].
extern "C" int gsb200_project_sh_fwd_rows(
    int64_t C, int64_t N, int64_t K, int degrees_to_use, const float *means, const float *quats, const float *scales,
    const float *opacities, const float *sh_coeffs, const float *viewmats, const float *Ks, uint32_t image_width,
    uint32_t image_height, float eps2d, float near_plane, float far_plane, float radius_clip, uint32_t tile_size,
    uint32_t tile_width, uint32_t tile_height, int32_t *radii, float *means2d, float *depths, float *conics, float *colors,
    void *row_records, int32_t *tiles_per_gauss, int64_t *totals, void *stream
)
{
    if(C < 0 || N < 0 || K <= 0 || degrees_to_use < 0 || degrees_to_use > 4 || tile_size == 0 || !totals
       || (int64_t)(degrees_to_use + 1) * (degrees_to_use + 1) > K)
        return GSB200_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    GSB_CUDA_TRY(cudaMemsetAsync(totals, 0, 3 * sizeof(int64_t), st));
    if(C * N == 0)
        return GSB200_OK;
    if(!means || !quats || !scales || !opacities || !sh_coeffs || !viewmats || !Ks || !radii || !means2d || !depths
       || !conics || !colors || !row_records || !tiles_per_gauss || C * N > 0x7fffffffLL
       || (reinterpret_cast<uintptr_t>(row_records) & 15) != 0)
        return GSB200_E_INVALID;
    if(bits_for_count(C) + bits_for_count((int64_t)tile_width * tile_height) > 32)
        return GSB200_E_KEYBITS;
#define CALL(d)                                                                                                   \
    project_sh_fwd_kernel<d, true><<<grid_for(C * N, kThreads), kThreads, 0, st>>>(                               \
        C, N, K, means, quats, scales, opacities, sh_coeffs, viewmats, Ks, image_width, image_height, eps2d,      \
        near_plane, far_plane, radius_clip, radii, means2d, depths, conics, nullptr, colors, tile_size,           \
        tile_width, tile_height, static_cast<float4 *>(row_records), tiles_per_gauss,                             \
        reinterpret_cast<unsigned long long *>(totals)                                                            \
    )
    GSB_DEG_SWITCH(degrees_to_use, CALL)
#undef CALL
    return check_launch();
}

extern "C" int gsb200_project_sh_bwd(
    int64_t C, int64_t N, int64_t K, int degrees_to_use, const float *means, const float *quats, const float *scales,
    const float *sh_coeffs, const float *viewmats, const float *Ks, uint32_t image_width, uint32_t image_height,
    float eps2d, const int32_t *radii, const float *conics, const float *compensations, const float *colors,
    const float *v_means2d, int64_t v_means2d_stride, const float *v_depths, int64_t v_depths_stride,
    const float *v_conics, int64_t v_conics_stride, const float *v_colors, int64_t v_colors_stride,
    const float *v_compensations, float *v_means, float *v_quats, float *v_scales, float *v_sh_coeffs, uint32_t *seen_bits, void *stream
)
{
    if(C < 0 || N < 0 || K <= 0 || degrees_to_use < 0 || degrees_to_use > 4
       || (int64_t)(degrees_to_use + 1) * (degrees_to_use + 1) > K)
        return GSB200_E_INVALID;
    if(N == 0)
        return GSB200_OK;
    if(!means || !quats || !scales || !sh_coeffs || !viewmats || !Ks || !radii || !conics || !colors || !v_means2d
       || !v_conics || !v_colors || !v_means || !v_quats || !v_scales || !v_sh_coeffs)
        return GSB200_E_INVALID;
    if(v_compensations && !compensations)
        return GSB200_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
#define CALL_ARGS                                                                                                  \
    C, N, K, means, quats, scales, sh_coeffs, viewmats, Ks, image_width, image_height, eps2d, radii, conics,       \
        compensations, colors, v_means2d, v_means2d_stride, v_depths, v_depths_stride, v_conics, v_conics_stride,  \
        v_colors, v_colors_stride, v_compensations, v_means, v_quats, v_scales, v_sh_coeffs, seen_bits
#define CALL(d)                                                                                                    \
    if(C == 1)                                                                                                     \
        project_sh_bwd_kernel<d, true><<<grid_for(N, kThreads), kThreads, 0, st>>>(CALL_ARGS);                     \
    else                                                                                                           \
        project_sh_bwd_kernel<d, false><<<grid_for(N, kThreads), kThreads, 0, st>>>(CALL_ARGS)
    GSB_DEG_SWITCH(degrees_to_use, CALL)
#undef CALL
#undef CALL_ARGS
    return check_launch();
}

// ---- isect
extern "C" size_t gsb200_isect_scan_workspace_bytes(int64_t n_elements)
{
    size_t bytes = 0;
    if(n_elements <= 0)
        return 0;
    cub::DeviceScan::InclusiveSum((void *)nullptr, bytes, (const int32_t *)nullptr, (int64_t *)nullptr, n_elements);
    return ((bytes + 255) & ~(size_t)255) + sizeof(int32_t) * (size_t)n_elements + 256; // + counts in depth order
}

extern "C" int gsb200_isect_count(
    int64_t I, int64_t N, const float *means2d, const int32_t *radii, const float *conics, const float *opacities,
    const int32_t *order, uint32_t tile_size, uint32_t tile_width, uint32_t tile_height, int32_t *tiles_per_gauss,
    int64_t *cum_tiles, void *workspace, size_t workspace_bytes, void *stream
)
{
    if(I < 0 || N < 0 || tile_size == 0)
        return GSB200_E_INVALID;
    const int64_t total = I * N;
    if(total == 0)
        return GSB200_OK;
    if(!means2d || !radii || !tiles_per_gauss || !cum_tiles || !workspace || total > 0x7fffffffLL)
        return GSB200_E_INVALID;
    if(bits_for_count(I) + bits_for_count((int64_t)tile_width * tile_height) > 32)
        return GSB200_E_KEYBITS;
    cudaStream_t st = (cudaStream_t)stream;
    size_t need     = 0;
    cub::DeviceScan::InclusiveSum((void *)nullptr, need, tiles_per_gauss, cum_tiles, total, st);
    const size_t scan_bytes = (need + 255) & ~(size_t)255;
    if(scan_bytes + (order ? sizeof(int32_t) * (size_t)total : 0) > workspace_bytes)
        return GSB200_E_WORKSPACE;
    int32_t *counts_in_order = order ? reinterpret_cast<int32_t *>(static_cast<char *>(workspace) + scan_bytes) : nullptr;
    isect_count_kernel<<<grid_for(total, kThreads), kThreads, 0, st>>>(
        total, means2d, radii, conics, opacities, order, tile_size, tile_width, tile_height, tiles_per_gauss, counts_in_order
    );
    if(int rc = check_launch())
        return rc;
    GSB_CUDA_TRY(cub::DeviceScan::InclusiveSum(workspace, need, order ? counts_in_order : tiles_per_gauss, cum_tiles, total, st));
    return GSB200_OK;
}

extern "C" int gsb200_isect_emit(
    int64_t I, int64_t N, const float *means2d, const int32_t *radii, const float *depths, const float *conics,
    const float *opacities, const int64_t *cum_tiles, const int64_t *image_ids, const int32_t *order, uint32_t tile_size,
    uint32_t tile_width, uint32_t tile_height, int64_t *isect_ids, int32_t *flatten_ids, void *stream
)
{
    if(I < 0 || N < 0 || tile_size == 0)
        return GSB200_E_INVALID;
    // packed layout: N rows in total (image_ids given), I only sizes the key; dense: I * N rows
    const int64_t total = image_ids ? N : I * N;
    if(total == 0)
        return GSB200_OK;
    if(!means2d || !radii || !depths || !cum_tiles || !isect_ids || !flatten_ids)
        return GSB200_E_INVALID;
    const uint32_t tile_bits = bits_for_count((int64_t)tile_width * tile_height);
    if(bits_for_count(I) + tile_bits > 32)
        return GSB200_E_KEYBITS;
    isect_emit_coop_kernel<int64_t><<<grid_for(total, kThreads), kThreads, 0, (cudaStream_t)stream>>>(
        total, N, means2d, radii, depths, conics, opacities, cum_tiles, image_ids, order, tile_size, tile_width, tile_height,
        tile_bits, isect_ids, flatten_ids
    );
    return check_launch();
}

extern "C" int gsb200_isect_count_totals(
    int64_t I, int64_t N, const float *means2d, const int32_t *radii, const float *conics, const float *opacities,
    uint32_t tile_size, uint32_t tile_width, uint32_t tile_height, int32_t *tiles_per_gauss, int64_t *totals, void *stream
)
{
    if(I < 0 || N < 0 || tile_size == 0 || !totals)
        return GSB200_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    GSB_CUDA_TRY(cudaMemsetAsync(totals, 0, 3 * sizeof(int64_t), st));
    const int64_t total = I * N;
    if(total == 0)
        return GSB200_OK;
    if(!means2d || !radii || !tiles_per_gauss || total > 0x7fffffffLL)
        return GSB200_E_INVALID;
    if(bits_for_count(I) + bits_for_count((int64_t)tile_width * tile_height) > 32)
        return GSB200_E_KEYBITS;
    isect_count_totals_kernel<<<grid_for(total, kThreads), kThreads, 0, st>>>(
        total, means2d, radii, conics, opacities, tile_size, tile_width, tile_height, tiles_per_gauss,
        reinterpret_cast<unsigned long long *>(totals)
    );
    return check_launch();
}

namespace gsb
{
template<class KeyT>
static int emit_ordered(
    int64_t I, int64_t N, int64_t n_order, int64_t max_tiles_hint, const float *means2d, const int32_t *radii, const float *depths,
    const float *conics, const float *opacities, const int64_t *cum_tiles, const int64_t *image_ids, const int32_t *order,
    uint32_t tile_size, uint32_t tile_width, uint32_t tile_height, KeyT *keys, int32_t *flatten_ids, void *stream,
    const int64_t *totals = nullptr, int64_t cap_isects = 0
)
{
    if(I < 0 || N < 0 || n_order < 0 || tile_size == 0)
        return GSB200_E_INVALID;
    if(n_order == 0)
        return GSB200_OK;
    if(!means2d || !radii || !depths || !cum_tiles || !order || !keys || !flatten_ids)
        return GSB200_E_INVALID;
    const uint32_t tile_bits = bits_for_count((int64_t)tile_width * tile_height);
    if(bits_for_count(I) + tile_bits > 32)
        return GSB200_E_KEYBITS;
    if(sizeof(KeyT) < 8 && bits_for_count(I * (int64_t)tile_width * tile_height) > 8 * sizeof(KeyT))
        return GSB200_E_KEYBITS;
    // the cooperative kernel pays off when SOME gaussian covers many tiles (one lane looping over thousands of tiles is the
    // tail of the whole launch); when even the largest row has few, the plain one-thread-per-gaussian kernel is leaner
    // (38 vs 45 us at cfg3)
    if(max_tiles_hint > 0 && max_tiles_hint <= 96)
        isect_emit_kernel<KeyT><<<grid_for(n_order, kThreads), kThreads, 0, (cudaStream_t)stream>>>(
            n_order, N, means2d, radii, depths, conics, opacities, cum_tiles, image_ids, order, tile_size, tile_width, tile_height,
            tile_bits, keys, flatten_ids, totals, cap_isects
        );
    else
        isect_emit_coop_kernel<KeyT><<<grid_for(n_order, kThreads), kThreads, 0, (cudaStream_t)stream>>>(
            n_order, N, means2d, radii, depths, conics, opacities, cum_tiles, image_ids, order, tile_size, tile_width, tile_height,
            tile_bits, keys, flatten_ids, totals, cap_isects
        );
    return check_launch();
}

// stage of gsb200_isect_sorted (sort.cu): emission into capacity-sized outputs, real counts in `totals` (device)
int emit_tilekeys_bounded(
    int64_t I, int64_t N, int64_t cap_vis, int64_t max_tiles_hint, const float *means2d, const int32_t *radii, const float *depths,
    const float *conics, const float *opacities, const int64_t *cum_tiles, const int32_t *order, uint32_t tile_size,
    uint32_t tile_width, uint32_t tile_height, int key_bytes, void *keys, int32_t *flatten_ids, const int64_t *totals,
    int64_t cap_isects, cudaStream_t st
)
{
    if(key_bytes == 2)
        return emit_ordered<uint16_t>(
            I, N, cap_vis, max_tiles_hint, means2d, radii, depths, conics, opacities, cum_tiles, nullptr, order, tile_size, tile_width,
            tile_height, static_cast<uint16_t *>(keys), flatten_ids, st, totals, cap_isects
        );
    return emit_ordered<uint32_t>(
        I, N, cap_vis, max_tiles_hint, means2d, radii, depths, conics, opacities, cum_tiles, nullptr, order, tile_size, tile_width,
        tile_height, static_cast<uint32_t *>(keys), flatten_ids, st, totals, cap_isects
    );
}

// offsets[(image, tile)] from sorted dense tile ids (narrow keys): same contract as isect_offsets_kernel
template<class KeyT>
__global__ void __launch_bounds__(kThreads) isect_offsets_tilekeys_kernel(
    int64_t n_isects, const KeyT *__restrict__ keys, int64_t total_tiles, int32_t *__restrict__ offsets,
    const int64_t *__restrict__ totals = nullptr
)
{
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if(totals != nullptr && totals[0] < n_isects)
        n_isects = totals[0]; // capacity-sized launch: the pairs past the real count are padding
    if(s >= n_isects)
        return;
    // Real keys are < total_tiles.  After a capacity miss (gsb200_isect_sorted with a count above its capacity) some
    // slots hold uninitialised pairs: the result is discarded by the caller, but no write may leave the array.
    int64_t id         = (int64_t)keys[s];
    const int64_t prev = s > 0 ? (int64_t)keys[s - 1] : -1;
    id                 = id < total_tiles ? id : total_tiles - 1;
    for(int64_t k = prev + 1; k <= id; ++k)
        offsets[k] = (int32_t)s;
    if(s == n_isects - 1)
        for(int64_t k = id + 1; k < total_tiles; ++k)
            offsets[k] = (int32_t)n_isects;
}

int offsets_tilekeys_bounded(
    int64_t cap_isects, int key_bytes, const void *keys, int64_t total_tiles, int32_t *offsets, const int64_t *totals, cudaStream_t st
)
{
    // no thread writes anything when the real count is 0: start from zeros
    GSB_CUDA_TRY(cudaMemsetAsync(offsets, 0, sizeof(int32_t) * (size_t)total_tiles, st));
    if(cap_isects == 0)
        return GSB200_OK;
    if(key_bytes == 2)
        isect_offsets_tilekeys_kernel<uint16_t><<<grid_for(cap_isects, kThreads), kThreads, 0, st>>>(
            cap_isects, static_cast<const uint16_t *>(keys), total_tiles, offsets, totals
        );
    else
        isect_offsets_tilekeys_kernel<uint32_t><<<grid_for(cap_isects, kThreads), kThreads, 0, st>>>(
            cap_isects, static_cast<const uint32_t *>(keys), total_tiles, offsets, totals
        );
    return check_launch();
}

// the reference's 64-bit intersection ids, rebuilt from the sorted tile ids and the rows' depths
template<class KeyT>
__global__ void __launch_bounds__(kThreads) isect_ids_from_tilekeys_kernel(
    int64_t n_isects, const KeyT *__restrict__ keys, const int32_t *__restrict__ flatten_ids, const float *__restrict__ depths,
    int64_t n_tiles, uint32_t tile_n_bits, int64_t *__restrict__ isect_ids
)
{
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if(s >= n_isects)
        return;
    const int64_t id = (int64_t)keys[s];
    const int64_t image = id / n_tiles, tile = id - image * n_tiles;
    isect_ids[s] = (((image << tile_n_bits) | tile) << 32) | (int64_t)__float_as_uint(depths[flatten_ids[s]]);
}
} // namespace gsb

extern "C" int gsb200_isect_emit_ordered(
    int64_t I, int64_t N, int64_t n_order, int64_t max_tiles_hint, const float *means2d, const int32_t *radii, const float *depths,
    const float *conics, const float *opacities, const int64_t *cum_tiles, const int64_t *image_ids, const int32_t *order,
    uint32_t tile_size, uint32_t tile_width, uint32_t tile_height, int64_t *isect_ids, int32_t *flatten_ids, void *stream
)
{
    return gsb::emit_ordered<int64_t>(
        I, N, n_order, max_tiles_hint, means2d, radii, depths, conics, opacities, cum_tiles, image_ids, order, tile_size, tile_width,
        tile_height, isect_ids, flatten_ids, stream
    );
}

// Narrow-key variant: writes the dense tile id image * n_tiles + tile as a key_bytes-wide (2 or 4) unsigned integer.
extern "C" int gsb200_isect_emit_tilekeys(
    int64_t I, int64_t N, int64_t n_order, int64_t max_tiles_hint, const float *means2d, const int32_t *radii, const float *depths,
    const float *conics, const float *opacities, const int64_t *cum_tiles, const int64_t *image_ids, const int32_t *order,
    uint32_t tile_size, uint32_t tile_width, uint32_t tile_height, int key_bytes, void *tile_keys, int32_t *flatten_ids, void *stream
)
{
    if(key_bytes == 2)
        return gsb::emit_ordered<uint16_t>(
            I, N, n_order, max_tiles_hint, means2d, radii, depths, conics, opacities, cum_tiles, image_ids, order, tile_size,
            tile_width, tile_height, static_cast<uint16_t *>(tile_keys), flatten_ids, stream
        );
    if(key_bytes == 4)
        return gsb::emit_ordered<uint32_t>(
            I, N, n_order, max_tiles_hint, means2d, radii, depths, conics, opacities, cum_tiles, image_ids, order, tile_size,
            tile_width, tile_height, static_cast<uint32_t *>(tile_keys), flatten_ids, stream
        );
    return GSB200_E_INVALID;
}

extern "C" int gsb200_isect_offsets_tilekeys(
    int64_t n_isects, int key_bytes, const void *tile_keys, int64_t I, uint32_t tile_width, uint32_t tile_height, int32_t *offsets,
    void *stream
)
{
    if(n_isects < 0 || I < 0 || (key_bytes != 2 && key_bytes != 4))
        return GSB200_E_INVALID;
    const int64_t total = I * (int64_t)tile_width * tile_height;
    if(total == 0)
        return GSB200_OK;
    if(!offsets)
        return GSB200_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    if(n_isects == 0)
    {
        GSB_CUDA_TRY(cudaMemsetAsync(offsets, 0, sizeof(int32_t) * (size_t)total, st));
        return GSB200_OK;
    }
    if(!tile_keys)
        return GSB200_E_INVALID;
    if(key_bytes == 2)
        isect_offsets_tilekeys_kernel<uint16_t><<<grid_for(n_isects, kThreads), kThreads, 0, st>>>(
            n_isects, static_cast<const uint16_t *>(tile_keys), total, offsets
        );
    else
        isect_offsets_tilekeys_kernel<uint32_t><<<grid_for(n_isects, kThreads), kThreads, 0, st>>>(
            n_isects, static_cast<const uint32_t *>(tile_keys), total, offsets
        );
    return check_launch();
}

extern "C" int gsb200_isect_ids_from_tilekeys(
    int64_t n_isects, int key_bytes, const void *tile_keys, const int32_t *flatten_ids, const float *depths, int64_t I,
    uint32_t tile_width, uint32_t tile_height, int64_t *isect_ids, void *stream
)
{
    if(n_isects < 0 || I < 0 || (key_bytes != 2 && key_bytes != 4))
        return GSB200_E_INVALID;
    if(n_isects == 0)
        return GSB200_OK;
    if(!tile_keys || !flatten_ids || !depths || !isect_ids)
        return GSB200_E_INVALID;
    const int64_t n_tiles = (int64_t)tile_width * tile_height;
    cudaStream_t st       = (cudaStream_t)stream;
    if(key_bytes == 2)
        isect_ids_from_tilekeys_kernel<uint16_t><<<grid_for(n_isects, kThreads), kThreads, 0, st>>>(
            n_isects, static_cast<const uint16_t *>(tile_keys), flatten_ids, depths, n_tiles, bits_for_count(n_tiles), isect_ids
        );
    else
        isect_ids_from_tilekeys_kernel<uint32_t><<<grid_for(n_isects, kThreads), kThreads, 0, st>>>(
            n_isects, static_cast<const uint32_t *>(tile_keys), flatten_ids, depths, n_tiles, bits_for_count(n_tiles), isect_ids
        );
    return check_launch();
}

extern "C" int gsb200_isect_offsets(
    int64_t n_isects, const int64_t *isect_ids, int64_t I, uint32_t tile_width, uint32_t tile_height, int32_t *offsets,
    void *stream
)
{
    if(n_isects < 0 || I < 0)
        return GSB200_E_INVALID;
    const int64_t n_tiles = (int64_t)tile_width * tile_height;
    const int64_t total   = I * n_tiles;
    if(total == 0)
        return GSB200_OK;
    if(!offsets)
        return GSB200_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    if(n_isects == 0)
    {
        GSB_CUDA_TRY(cudaMemsetAsync(offsets, 0, sizeof(int32_t) * (size_t)total, st));
        return GSB200_OK;
    }
    if(!isect_ids)
        return GSB200_E_INVALID;
    isect_offsets_kernel<<<grid_for(n_isects, kThreads), kThreads, 0, st>>>(
        n_isects, isect_ids, total, n_tiles, bits_for_count(n_tiles), offsets
    );
    return check_launch();
}

// ---- MCMC strategy ops
extern "C" int gsb200_relocation(
    int64_t N, const float *opacities, const float *scales, const int32_t *ratios, const float *binoms, int n_max,
    float min_opacity, float *new_opacities, float *new_scales, void *stream
)
{
    if(N < 0 || n_max <= 0)
        return GSB200_E_INVALID;
    if(N == 0)
        return GSB200_OK;
    if(!opacities || !scales || !ratios || !binoms || !new_opacities || !new_scales)
        return GSB200_E_INVALID;
    relocation_kernel<<<grid_for(N, kThreads), kThreads, 0, (cudaStream_t)stream>>>(
        N, opacities, scales, ratios, binoms, n_max, min_opacity, new_opacities, new_scales
    );
    return check_launch();
}

extern "C" int gsb200_mcmc_perturb_positions(
    int64_t N, float *positions, const float *quats, const float *scales_log, const float *opacities_logit,
    const float *noise, float noise_scale, float t, float k, void *stream
)
{
    if(N < 0)
        return GSB200_E_INVALID;
    if(N == 0)
        return GSB200_OK;
    if(!positions || !quats || !scales_log || !opacities_logit || !noise)
        return GSB200_E_INVALID;
    mcmc_perturb_kernel<<<grid_for(N, kThreads), kThreads, 0, (cudaStream_t)stream>>>(
        N, positions, quats, scales_log, opacities_logit, noise, noise_scale, t, k
    );
    return check_launch();
}

extern "C" int gsb200_adam(
    int64_t N, int64_t D, float *param, const float *param_grad, float *exp_avg, float *exp_avg_sq, const uint8_t *valid,
    float lr, float b1, float b2, float eps, void *stream
)
{
    if(N < 0 || D < 0)
        return GSB200_E_INVALID;
    if(N * D == 0)
        return GSB200_OK;
    if(!param || !param_grad || !exp_avg || !exp_avg_sq)
        return GSB200_E_INVALID;
    adam_kernel<<<grid_for(N * D, kThreads), kThreads, 0, (cudaStream_t)stream>>>(
        N * D, D, param, param_grad, exp_avg, exp_avg_sq, valid, lr, b1, b2, eps
    );
    return check_launch();
}

// ---- packed projection (reference ops projection_ewa_3dgs_packed / _bwd, ext.cpp:1065-1077)
extern "C" size_t gsb200_projection_packed_workspace_bytes(int64_t B, int64_t C, int64_t N)
{
    const int64_t blocks = B * C * ((N + kThreads - 1) / kThreads);
    if(blocks <= 0)
        return 0;
    size_t scan = 0;
    cub::DeviceScan::InclusiveSum((void *)nullptr, scan, (const int32_t *)nullptr, (int32_t *)nullptr, blocks);
    return ((scan + 255) & ~(size_t)255) + 2 * (((size_t)blocks * sizeof(int32_t) + 255) & ~(size_t)255) + 256;
}

namespace
{
struct PackedWs
{
    int32_t *cnts, *accum;
    void *scan;
    size_t scan_bytes;
};
PackedWs carve_packed(void *workspace, int64_t blocks)
{
    PackedWs w;
    const size_t seg = ((size_t)blocks * sizeof(int32_t) + 255) & ~(size_t)255;
    char *p          = static_cast<char *>(workspace);
    w.cnts           = reinterpret_cast<int32_t *>(p);
    w.accum          = reinterpret_cast<int32_t *>(p + seg);
    w.scan           = p + 2 * seg;
    w.scan_bytes     = 0;
    cub::DeviceScan::InclusiveSum((void *)nullptr, w.scan_bytes, w.cnts, w.accum, blocks);
    return w;
}
} // namespace

#define GSB_CAM_SWITCH(model, CALL)       \
    if((model) == kCamPinhole)            \
    {                                     \
        CALL(kCamPinhole);                \
    }                                     \
    else if((model) == kCamOrtho)         \
    {                                     \
        CALL(kCamOrtho);                  \
    }                                     \
    else                                  \
    {                                     \
        CALL(kCamFisheye);                \
    }

// Pass 1: per-block visible counts + their inclusive scan in `workspace`; *nnz_dev (device int32) = total.
extern "C" int gsb200_projection_packed_count(
    int64_t B, int64_t C, int64_t N, const float *means, const float *covars, const float *quats, const float *scales,
    const float *opacities, const float *viewmats, const float *Ks, uint32_t image_width, uint32_t image_height,
    float eps2d, float near_plane, float far_plane, float radius_clip, int calc_compensations, int camera_model,
    void *workspace, size_t workspace_bytes, int32_t *nnz_dev, void *stream
)
{
    if(B < 0 || C < 0 || N < 0 || !nnz_dev)
        return GSB200_E_INVALID;
    if(camera_model < 0 || camera_model > 2)
        return GSB200_E_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    if(B * C * N == 0)
    {
        GSB_CUDA_TRY(cudaMemsetAsync(nnz_dev, 0, sizeof(int32_t), st));
        return GSB200_OK;
    }
    if(!means || !viewmats || !Ks || !workspace || (!covars && (!quats || !scales)) || B * C > 65535)
        return GSB200_E_INVALID;
    const int64_t bpr = (N + kThreads - 1) / kThreads, blocks = B * C * bpr;
    if(gsb200_projection_packed_workspace_bytes(B, C, N) > workspace_bytes)
        return GSB200_E_WORKSPACE;
    PackedWs w = carve_packed(workspace, blocks);
    const dim3 grid((unsigned)bpr, (unsigned)(B * C));
#define CALL(CAM)                                                                                                      \
    projection_packed_kernel<CAM, false><<<grid, kThreads, 0, st>>>(                                                    \
        C, N, means, covars, quats, scales, opacities, viewmats, Ks, image_width, image_height, eps2d, near_plane,      \
        far_plane, radius_clip, calc_compensations != 0, nullptr, w.cnts, nullptr, nullptr, nullptr, nullptr, nullptr,  \
        nullptr, nullptr, nullptr, nullptr                                                                              \
    )
    GSB_CAM_SWITCH(camera_model, CALL)
#undef CALL
    if(int rc = check_launch())
        return rc;
    GSB_CUDA_TRY(cub::DeviceScan::InclusiveSum(w.scan, w.scan_bytes, w.cnts, w.accum, blocks, st));
    GSB_CUDA_TRY(cudaMemcpyAsync(nnz_dev, w.accum + blocks - 1, sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
    return GSB200_OK;
}

// Pass 2 (same workspace, untouched since pass 1): the nnz visible rows, ascending (b, c, n); indptr [B*C + 1].
extern "C" int gsb200_projection_packed_emit(
    int64_t B, int64_t C, int64_t N, const float *means, const float *covars, const float *quats, const float *scales,
    const float *opacities, const float *viewmats, const float *Ks, uint32_t image_width, uint32_t image_height,
    float eps2d, float near_plane, float far_plane, float radius_clip, int camera_model, const void *workspace,
    int32_t *indptr, int64_t *batch_ids, int64_t *camera_ids, int64_t *gaussian_ids, int32_t *radii, float *means2d,
    float *depths, float *conics, float *compensations, void *stream
)
{
    if(B < 0 || C < 0 || N < 0 || !indptr)
        return GSB200_E_INVALID;
    if(camera_model < 0 || camera_model > 2)
        return GSB200_E_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    if(B * C * N == 0)
    {
        GSB_CUDA_TRY(cudaMemsetAsync(indptr, 0, sizeof(int32_t) * (size_t)(B * C + 1), st));
        return GSB200_OK;
    }
    if(!means || !viewmats || !Ks || !workspace || (!covars && (!quats || !scales)) || B * C > 65535)
        return GSB200_E_INVALID;
    const int64_t bpr = (N + kThreads - 1) / kThreads, blocks = B * C * bpr;
    PackedWs w = carve_packed(const_cast<void *>(workspace), blocks);
    const dim3 grid((unsigned)bpr, (unsigned)(B * C));
#define CALL(CAM)                                                                                                      \
    projection_packed_kernel<CAM, true><<<grid, kThreads, 0, st>>>(                                                     \
        C, N, means, covars, quats, scales, opacities, viewmats, Ks, image_width, image_height, eps2d, near_plane,      \
        far_plane, radius_clip, compensations != nullptr, w.accum, nullptr, indptr, batch_ids, camera_ids,              \
        gaussian_ids, radii, means2d, depths, conics, compensations                                                     \
    )
    GSB_CAM_SWITCH(camera_model, CALL)
#undef CALL
    return check_launch();
}

// Backward over the nnz rows.  sparse_grad != 0: v_means [nnz,3], v_covars [nnz,6] or v_quats [nnz,4] +
// v_scales [nnz,3] (one entry per row, written); else dense [B*N,*] outputs, zero-initialised here, summed with atomics.
extern "C" int gsb200_projection_packed_bwd(
    int64_t B, int64_t C, int64_t N, int64_t nnz, const float *means, const float *covars, const float *quats,
    const float *scales, const float *viewmats, const float *Ks, uint32_t image_width, uint32_t image_height, float eps2d,
    int camera_model, const int64_t *batch_ids, const int64_t *camera_ids, const int64_t *gaussian_ids,
    const float *conics, const float *compensations, const float *v_means2d, int64_t v_means2d_stride,
    const float *v_depths, int64_t v_depths_stride, const float *v_conics, int64_t v_conics_stride,
    const float *v_compensations, int sparse_grad, float *v_means, float *v_covars, float *v_quats, float *v_scales,
    float *v_viewmats, void *stream
)
{
    if(B < 0 || C < 0 || N < 0 || nnz < 0)
        return GSB200_E_INVALID;
    if(camera_model < 0 || camera_model > 2)
        return GSB200_E_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    if(v_viewmats && B * C > 0)
        GSB_CUDA_TRY(cudaMemsetAsync(v_viewmats, 0, sizeof(float) * 16 * (size_t)(B * C), st));
    if(!v_means || (covars ? !v_covars : (!v_quats || !v_scales)))
        return (B * N == 0 && nnz == 0) ? GSB200_OK : GSB200_E_INVALID;
    if(!sparse_grad && B * N > 0)
    {
        GSB_CUDA_TRY(cudaMemsetAsync(v_means, 0, sizeof(float) * 3 * (size_t)(B * N), st));
        if(covars)
            GSB_CUDA_TRY(cudaMemsetAsync(v_covars, 0, sizeof(float) * 6 * (size_t)(B * N), st));
        else
        {
            GSB_CUDA_TRY(cudaMemsetAsync(v_quats, 0, sizeof(float) * 4 * (size_t)(B * N), st));
            GSB_CUDA_TRY(cudaMemsetAsync(v_scales, 0, sizeof(float) * 3 * (size_t)(B * N), st));
        }
    }
    if(nnz == 0)
        return GSB200_OK;
    if(!means || !viewmats || !Ks || !batch_ids || !camera_ids || !gaussian_ids || !conics || !v_means2d || !v_depths
       || !v_conics || (covars ? false : (!quats || !scales)) || (v_compensations && !compensations))
        return GSB200_E_INVALID;
#define CALL(CAM)                                                                                                      \
    projection_packed_bwd_kernel<CAM><<<grid_for(nnz, kThreads), kThreads, 0, st>>>(                                     \
        nnz, C, N, means, covars, quats, scales, viewmats, Ks, image_width, image_height, eps2d, batch_ids, camera_ids, \
        gaussian_ids, conics, compensations, v_means2d, v_means2d_stride, v_depths, v_depths_stride, v_conics,          \
        v_conics_stride, v_compensations, sparse_grad == 0, v_means, v_covars, v_quats, v_scales, v_viewmats            \
    )
    GSB_CAM_SWITCH(camera_model, CALL)
#undef CALL
    return check_launch();
}

// ---- SH on packed rows (coefficients indexed in place; used by rasterization(packed=True))
extern "C" int gsb200_sh_rows_fwd(
    int64_t nnz, int64_t B, int64_t C, int64_t N, int64_t K, int64_t D, int degrees_to_use, const float *means,
    const float *viewmats, const float *coeffs, const int64_t *batch_ids, const int64_t *camera_ids,
    const int64_t *gaussian_ids, float *colors, void *stream
)
{
    if(nnz < 0 || B < 0 || C < 0 || N < 0 || K <= 0 || D <= 0 || degrees_to_use < 0 || degrees_to_use > 4
       || (int64_t)(degrees_to_use + 1) * (degrees_to_use + 1) > K)
        return GSB200_E_INVALID;
    if(nnz == 0)
        return GSB200_OK;
    if(!means || !viewmats || !coeffs || !batch_ids || !camera_ids || !gaussian_ids || !colors)
        return GSB200_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
#define CALL(d) sh_rows_fwd_kernel<d><<<grid_for(nnz * D, kThreads), kThreads, 0, st>>>(nnz, C, N, K, D, means, viewmats, coeffs, batch_ids, camera_ids, gaussian_ids, colors)
    GSB_DEG_SWITCH(degrees_to_use, CALL)
#undef CALL
    return check_launch();
}

extern "C" int gsb200_sh_rows_bwd(
    int64_t nnz, int64_t B, int64_t C, int64_t N, int64_t K, int64_t D, int degrees_to_use, const float *means,
    const float *viewmats, const float *coeffs, const int64_t *batch_ids, const int64_t *camera_ids,
    const int64_t *gaussian_ids, const float *v_colors, float *v_coeffs, float *v_means, float *v_dirsum, void *stream
)
{
    if(nnz < 0 || B < 0 || C < 0 || N < 0 || K <= 0 || D <= 0 || degrees_to_use < 0 || degrees_to_use > 4
       || (int64_t)(degrees_to_use + 1) * (degrees_to_use + 1) > K || !v_coeffs)
        return GSB200_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    if(N > 0)
        GSB_CUDA_TRY(cudaMemsetAsync(v_coeffs, 0, sizeof(float) * (size_t)(N * K * D), st));
    if(v_means && B * N > 0)
        GSB_CUDA_TRY(cudaMemsetAsync(v_means, 0, sizeof(float) * 3 * (size_t)(B * N), st));
    if(v_dirsum && B * C > 0)
        GSB_CUDA_TRY(cudaMemsetAsync(v_dirsum, 0, sizeof(float) * 3 * (size_t)(B * C), st));
    if(nnz == 0)
        return GSB200_OK;
    if(!means || !viewmats || !coeffs || !batch_ids || !camera_ids || !gaussian_ids || !v_colors)
        return GSB200_E_INVALID;
#define CALL(d) sh_rows_bwd_kernel<d><<<grid_for(nnz * D, kThreads), kThreads, 0, st>>>(nnz, C, N, K, D, means, viewmats, coeffs, batch_ids, camera_ids, gaussian_ids, v_colors, v_coeffs, v_means, v_dirsum)
    GSB_DEG_SWITCH(degrees_to_use, CALL)
#undef CALL
    return check_launch();
}
