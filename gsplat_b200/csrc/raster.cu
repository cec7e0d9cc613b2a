// raster.cu -- rasterize_to_pixels forward / backward for sm_100a.
//
// Replaces (behaviour, not code) the reference kernels
//   csrc/RasterizeToPixels3DGSSerialBatchFwd.cu:41-297   (forward)
//   csrc/RasterizeToPixels3DGSSerialBatchBwd.cu:41-320   (backward)
//   csrc/RasterizeToPixels3DGSDevice.cuh:37-173          (per-pair math)
//
// B200 design (see DESIGN.md section "rasterize"):
//  * a pack pass gathers the depth-sorted per-intersection records ONCE per view into three
//    contiguous float4 streams (cull: mean + conservative half extents of the alpha>=1/255 ellipse,
//    geom: conic + opacity, color), so that every tile's list is a contiguous byte range;
//  * each CTA (one 16x16 tile, 8 warps, a warp owns an 8x4 pixel block) streams its range through a
//    shared-memory ring filled with 1-D TMA bulk copies (cp.async.bulk + mbarrier complete_tx).  For
//    D <= 4 channels the ring has 3 stages and no CTA barrier in the batch loop: every warp works at its
//    own pace and the last warp out of a stage refills it.  For D > 4 the CTA moves through a 2-stage
//    ring in step, with CTA barriers;
//  * inside a batch every lane tests ONE gaussian's extent box against the warp's pixel block and the
//    warp ballots: only gaussians that can reach alpha >= 1/255 inside the block are evaluated
//    (exact: the skipped pairs are `continue`d by the reference too); finished warps drop out by ballot;
//  * the backward walks the same ring back to front with a transposed reduction: per surviving gaussian
//    each lane (= pixel) buffers two scalars, and after 16 survivors each lane (= gaussian) sums its
//    gaussian's gradient record over the warp's pixels and adds it with 128-bit red.global.add.
#include <algorithm>

#include <mutex>

#include "common.cuh"
#include "rowrec.cuh"

namespace gsb
{
constexpr int kBatch  = 128; // gaussians per ring stage
constexpr int kStages = 2;
constexpr int kWarps  = 8;

template<int CDIM, int BATCH = kBatch>
struct RecLayout
{
    static constexpr int kColorVec4 = (CDIM + 3) / 4; // float4 per record for colours
    static constexpr int kStageBytes = BATCH * (16 + 16 + 16 + 16 * kColorVec4);
};

struct RecordStreams
{
    float4 *cull;   // [S] {mx, my, ex, ey}: mean + half extents of the axis-aligned box of {alpha >= 1/255}
    float4 *axis;   // [S] {ux, uy, lu, lv}: unit major-curvature axis and half lengths of its oriented box
    float4 *geom;   // [S] {a, b, c, opacity}
    float4 *color;  // [S * kColorVec4]
    int32_t *order; // [n_tiles] tile indices, longest list first
};

static inline size_t align256(size_t x) { return (x + 255) & ~size_t(255); }

static inline RecordStreams carve_records(void *base, int64_t S, int cvec4)
{
    RecordStreams r;
    char *p = (char *)base;
    r.cull  = (float4 *)p;
    p += align256((size_t)S * 16);
    r.axis = (float4 *)p;
    p += align256((size_t)S * 16);
    r.geom = (float4 *)p;
    p += align256((size_t)S * 16);
    r.color = (float4 *)p;
    p += align256((size_t)S * 16 * (size_t)cvec4);
    r.order = (int32_t *)p;
    return r;
}

// ---------------------------------------------------------------------------------------------
// Longest-list-first tile order.  A tile is one CTA and its list is walked sequentially, so a long list
// that starts late is the tail of the whole launch; CTAs are dispatched in blockIdx order, hence the
// permutation.  One CTA: 256-bin counting sort on (length / 32), descending.
__global__ void __launch_bounds__(1024) tile_order_kernel(
    const int32_t *__restrict__ offsets, const int32_t n_tiles, const int32_t n_isects, int32_t *__restrict__ order
)
{
    __shared__ int32_t hist[256];
    __shared__ int32_t cursor[256];
    for(int i = threadIdx.x; i < 256; i += blockDim.x)
        hist[i] = 0;
    __syncthreads();
    auto bin_of = [&](int t) {
        const int32_t end = (t == n_tiles - 1) ? n_isects : offsets[t + 1];
        const int32_t len = end - offsets[t];
        const int b       = len >> 5;
        return 255 - (b > 255 ? 255 : b); // bin 0 = longest
    };
    for(int t = threadIdx.x; t < n_tiles; t += blockDim.x)
        atomicAdd(&hist[bin_of(t)], 1);
    __syncthreads();
    if(threadIdx.x < 32)
    { // exclusive scan of the 256 bins by one warp: 8 consecutive bins per lane
        const int base = threadIdx.x * 8;
        int32_t local[8], sum = 0;
#pragma unroll
        for(int i = 0; i < 8; ++i)
        {
            local[i] = sum;
            sum += hist[base + i];
        }
        int32_t incl = sum;
#pragma unroll
        for(int o = 1; o < 32; o <<= 1)
        {
            const int32_t up = __shfl_up_sync(0xffffffffu, incl, o);
            if((int)threadIdx.x >= o)
                incl += up;
        }
        const int32_t excl = incl - sum;
#pragma unroll
        for(int i = 0; i < 8; ++i)
            cursor[base + i] = excl + local[i];
    }
    __syncthreads();
    for(int t = threadIdx.x; t < n_tiles; t += blockDim.x)
        order[atomicAdd(&cursor[bin_of(t)], 1)] = t;
}

// ---------------------------------------------------------------------------------------------
// pack: gather sorted records.  One thread per intersection.
template<int CDIM>
__global__ void __launch_bounds__(256) pack_records_kernel(
    const int64_t S, const int32_t *__restrict__ flatten_ids, const float *__restrict__ means2d,
    const float *__restrict__ conics, const float *__restrict__ colors, const float *__restrict__ opacities,
    float4 *__restrict__ cull, float4 *__restrict__ axis, float4 *__restrict__ geom, float4 *__restrict__ color
)
{
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if(s >= S)
        return;
    const int64_t g = flatten_ids[s];
    const float2 m  = *reinterpret_cast<const float2 *>(means2d + g * 2);
    const float a = conics[g * 3], b = conics[g * 3 + 1], c = conics[g * 3 + 2];
    const float op = opacities[g];
    float4 rc, ra, rg;
    row_record(m.x, m.y, a, b, c, op, rc, ra, rg);
    cull[s] = rc;
    axis[s] = ra;
    geom[s] = rg;
    constexpr int CV = RecLayout<CDIM>::kColorVec4;
    float cbuf[CV * 4];
#pragma unroll
    for(int k = 0; k < CV * 4; ++k)
        cbuf[k] = k < CDIM ? colors[g * CDIM + k] : 0.f;
#pragma unroll
    for(int v = 0; v < CV; ++v)
        color[s * CV + v] = make_float4(cbuf[4 * v], cbuf[4 * v + 1], cbuf[4 * v + 2], cbuf[4 * v + 3]);
}

// pack from 64-byte row records {cull | axis | geom | color} written by the fused projection (CDIM <= 4): a pure gather,
// four lanes per intersection, each moving one float4 -- 64 contiguous bytes read per intersection, 128 contiguous bytes
// written per stream and warp.  The id -> row -> store chain is two dependent loads long, so every thread carries
// kPackUnroll independent chains (with one it was latency-bound: 50 us for 236 MB at S = 1.84 M).
constexpr int kPackUnroll = 4;
__global__ void __launch_bounds__(256) pack_rows_kernel(
    const int64_t S, const int32_t *__restrict__ flatten_ids, const float4 *__restrict__ rows, float4 *__restrict__ cull,
    float4 *__restrict__ axis, float4 *__restrict__ geom, float4 *__restrict__ color
)
{
    // a block covers kPackUnroll * 64 consecutive intersections; chain u of a thread handles intersection base + u * 64
    const int part     = (int)(threadIdx.x & 3);
    const int64_t base = (int64_t)blockIdx.x * (kPackUnroll * 64) + (threadIdx.x >> 2);
    float4 *dst        = part == 0 ? cull : (part == 1 ? axis : (part == 2 ? geom : color));
    int32_t g[kPackUnroll];
#pragma unroll
    for(int u = 0; u < kPackUnroll; ++u)
    {
        const int64_t s = base + u * 64;
        g[u]            = s < S ? __ldg(flatten_ids + s) : 0;
    }
    float4 v[kPackUnroll];
#pragma unroll
    for(int u = 0; u < kPackUnroll; ++u)
        v[u] = ldg_nc_f4(rows + (int64_t)g[u] * 4 + part);
#pragma unroll
    for(int u = 0; u < kPackUnroll; ++u)
    {
        const int64_t s = base + u * 64;
        if(s < S)
            dst[s] = v[u];
    }
}

// ---------------------------------------------------------------------------------------------
struct TileGeom
{
    int image_id, tile_id, tile_x, tile_y;
};

__device__ __forceinline__ TileGeom decode_tile(const int32_t *__restrict__ order, uint32_t tw, uint32_t th)
{
    const uint32_t block = order ? (uint32_t)order[blockIdx.x] : blockIdx.x;
    TileGeom t;
    const uint32_t per = tw * th;
    t.image_id         = block / per;
    t.tile_id          = block % per;
    t.tile_x           = t.tile_id % tw;
    t.tile_y           = t.tile_id / tw;
    return t;
}

// the axis stream lies between the cull and geom streams, equally sized: midpoint of the two pointers
__device__ __forceinline__ const float4 *gaxis_from(const float4 *gcull, const float4 *ggeom)
{
    return gcull + ((ggeom - gcull) >> 1);
}

// shared-memory ring: per stage [cull | axis | geom | color] + one full-barrier per stage
template<int CDIM, int BATCH = kBatch, int STAGES = kStages>
struct Ring
{
    static constexpr int CV = RecLayout<CDIM>::kColorVec4;
    static constexpr int kStageBytes = RecLayout<CDIM, BATCH>::kStageBytes;
    unsigned char *base;

    __device__ __forceinline__ void carve(unsigned char *smem) { base = smem; }
    __device__ __forceinline__ float4 *cull(int s) const
    {
        return reinterpret_cast<float4 *>(base + (size_t)s * kStageBytes);
    }
    __device__ __forceinline__ float4 *axis(int s) const { return cull(s) + BATCH; }
    __device__ __forceinline__ float4 *geom(int s) const { return cull(s) + 2 * BATCH; }
    __device__ __forceinline__ float4 *color(int s) const { return cull(s) + 3 * BATCH; }
    __device__ __forceinline__ uint64_t *full(int s) const
    {
        return reinterpret_cast<uint64_t *>(base + (size_t)STAGES * kStageBytes) + s;
    }
    __device__ __forceinline__ int32_t *ids(int s) const
    {
        return reinterpret_cast<int32_t *>(base + (size_t)STAGES * kStageBytes + STAGES * sizeof(uint64_t)) + s * BATCH;
    }
    // one thread: arm the barrier and launch the four bulk copies of records [first, first+count)
    __device__ __forceinline__ void issue(
        int stage, const float4 *gcull, const float4 *ggeom, const float4 *gcolor, int64_t first, int count
    ) const
    {
        // the axis stream sits right behind the cull stream at a fixed distance (see carve_records)
        const uint32_t n16 = (uint32_t)count * 16u;
        mbar_arrive_expect_tx(full(stage), n16 * (3u + CV));
        bulk_g2s(cull(stage), gcull + first, n16, full(stage));
        bulk_g2s(axis(stage), gaxis_from(gcull, ggeom) + first, n16, full(stage));
        bulk_g2s(geom(stage), ggeom + first, n16, full(stage));
        bulk_g2s(color(stage), gcolor + first * CV, n16 * CV, full(stage));
    }
};

template<int CDIM, int BATCH = kBatch, int STAGES = kStages>
constexpr size_t ring_smem_bytes()
{
    // stages | full barriers | per-stage gaussian ids (backward only)
    return (size_t)STAGES * RecLayout<CDIM, BATCH>::kStageBytes + STAGES * sizeof(uint64_t)
         + (size_t)STAGES * BATCH * sizeof(int32_t);
}

// Can the gaussian reach alpha >= 1/255 anywhere in the 8x4 pixel block centred at (cx, cy)?  Conservative:
// its axis-aligned AND its oriented bounding box must both overlap the block (pixel centres span +-3.5, +-1.5).
__device__ __forceinline__ bool block_may_touch(const float4 q, const float4 ax, const float cx, const float cy)
{
    constexpr float hx = 3.5f, hy = 1.5f;
    const float dx = q.x - cx, dy = q.y - cy;
    const float au = fabsf(ax.x), av = fabsf(ax.y);
    return (fabsf(dx) <= q.z + hx) && (fabsf(dy) <= q.w + hy) && (fabsf(dx * ax.x + dy * ax.y) <= ax.z + hx * au + hy * av)
        && (fabsf(dy * ax.x - dx * ax.y) <= ax.w + hx * av + hy * au);
}

// ---------------------------------------------------------------------------------------------
// forward.  PIPE = true: the batch loop has no CTA barrier (same scheme as raster_bwd2_kernel): every warp waits for the
// stage's TMA barrier, works through the batch at its own pace, counts itself off on the stage, and the last warp out
// re-arms the barrier and fetches the batch kPipeStages ahead -- unless every warp of the tile is saturated, in which
// case it publishes the first batch that will NOT arrive (s_stop) and all warps leave when they reach it (the tile-level
// early exit of the barrier version).
constexpr int kPipeStages = 3;

template<int CDIM, bool PIPE = false>
__global__ void __launch_bounds__(kWarps * 32) raster_fwd_kernel(
    const uint32_t I, const int64_t n_isects, const float4 *__restrict__ gcull, const float4 *__restrict__ ggeom,
    const float4 *__restrict__ gcolor, const int32_t *__restrict__ order, const float *__restrict__ backgrounds,
    const uint8_t *__restrict__ masks, const uint32_t W, const uint32_t H, const uint32_t tw, const uint32_t th,
    const int32_t *__restrict__ offsets, float *__restrict__ render_colors, float *__restrict__ render_alphas,
    int32_t *__restrict__ last_ids
)
{
    constexpr int CV = RecLayout<CDIM>::kColorVec4;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int KS = PIPE ? kPipeStages : kStages;
    Ring<CDIM, kBatch, KS> ring;
    ring.carve(smem_raw);

    __shared__ int32_t s_surv[kWarps][32];
    __shared__ int32_t s_cnt[kPipeStages]; // PIPE: warps that are through with the stage's current batch
    __shared__ int32_t s_alive;            // PIPE: warps with an unsaturated pixel
    __shared__ int32_t s_stop;             // PIPE: first batch that will not be fetched (read and written with atomics only)
    const TileGeom tg   = decode_tile(order, tw, th);
    const unsigned tid  = threadIdx.x;
    const unsigned warp = tid >> 5, lane = tid & 31;
    int32_t *surv       = s_surv[warp];
    const uint32_t lanemask_lt = (1u << lane) - 1u;
    // warp -> 8x4 pixel block inside the 16x16 tile
    const int bx0 = tg.tile_x * kTile + (warp & 1) * 8;
    const int by0 = tg.tile_y * kTile + (warp >> 1) * 4;
    const int px_i = bx0 + (lane & 7), py_i = by0 + (lane >> 3);
    const float px = (float)px_i + 0.5f, py = (float)py_i + 0.5f;
    const bool inside = (px_i < (int)W) && (py_i < (int)H);
    const int64_t pix = ((int64_t)tg.image_id * H + py_i) * W + px_i;
    const float *bg   = backgrounds ? backgrounds + (size_t)tg.image_id * CDIM : nullptr;

    const int64_t tile_lin = (int64_t)tg.image_id * tw * th + tg.tile_id;
    if(masks != nullptr && !masks[tile_lin])
    { // masked-off tile: background, zero alpha (reference Fwd.cu:142-160)
        if(inside)
        {
#pragma unroll
            for(int k = 0; k < CDIM; ++k)
                render_colors[pix * CDIM + k] = bg ? bg[k] : 0.f;
            render_alphas[pix] = 0.f;
            last_ids[pix]      = 0;
        }
        return;
    }

    const int32_t range_start = offsets[tile_lin];
    const int32_t range_end   = (tile_lin == (int64_t)I * tw * th - 1) ? (int32_t)n_isects : offsets[tile_lin + 1];
    const int num_batches     = (range_end - range_start + kBatch - 1) / kBatch;

    if(tid == 0)
    {
#pragma unroll
        for(int s = 0; s < KS; ++s)
        {
            mbar_init(ring.full(s), 1);
            s_cnt[s < kPipeStages ? s : 0] = 0;
        }
        s_alive = kWarps;
        s_stop  = 0x7fffffff;
        fence_mbar_init();
    }
    __syncthreads();
    if(tid == 0)
    {
#pragma unroll
        for(int s = 0; s < KS; ++s)
            if(s < num_batches)
            {
                const int64_t first = (int64_t)range_start + (int64_t)s * kBatch;
                const int count     = min(kBatch, (int)(range_end - first));
                ring.issue(s, gcull, ggeom, gcolor, first, count);
            }
    }

    // pixel-block centre extents for the cull test: centres span [bx0+0.5, bx0+7.5] x [by0+0.5, by0+3.5]
    const float cx = (float)bx0 + 4.0f, cy = (float)by0 + 2.0f;

    float T = 1.f;
    float pix_out[CDIM];
#pragma unroll
    for(int k = 0; k < CDIM; ++k)
        pix_out[k] = 0.f;
    int32_t cur_idx = 0;
    uint32_t done   = inside ? 0u : 1u;
    int last_b      = num_batches; // batch at which the tile-level early exit happened

    bool warp_alive = true; // PIPE: this warp still has an unsaturated pixel (uniform in the warp)
    for(int b = 0; b < num_batches; ++b)
    {
        const int stage       = b % KS;
        const uint32_t parity = (uint32_t)(b / KS) & 1u;
        const int32_t first   = range_start + b * kBatch;
        const int count       = min(kBatch, (int)(range_end - first));
        if constexpr(PIPE)
        {
            // lane 0 waits for the batch or for the stop flag; the verdict is broadcast so that the warp leaves as one
            int verdict = 0; // 1 = the batch has landed, 2 = it will never be fetched
            if(lane == 0)
            {
                while(verdict == 0)
                {
                    if(mbar_try_wait(ring.full(stage), parity))
                        verdict = 1;
                    else if(b >= atomicMin(&s_stop, 0x7fffffff)) // atomic read of the flag
                        verdict = 2;
                }
            }
            verdict = __shfl_sync(0xffffffffu, verdict, 0);
            if(verdict == 2)
                break;
            mbar_wait(ring.full(stage), parity); // every lane observes the completed phase itself (returns at once)
        }
        if(!__all_sync(0xffffffffu, done != 0u))
        {
            if constexpr(!PIPE)
                mbar_wait(ring.full(stage), parity);
            const float4 *scull = ring.cull(stage);
            const float4 *saxis = ring.axis(stage);
            const float4 *sgeom = ring.geom(stage);
            const float4 *scol  = ring.color(stage);
            for(int c0 = 0; c0 < count; c0 += 32)
            {
                // Each lane tests one gaussian's extent box against this warp's pixel block; the survivors' batch-local
                // indices are compacted, front to back, into a per-warp list (walking the ballot mask bit by bit cost 10
                // instructions per survivor: FLO, shift, xor, index and address arithmetic; the list costs one LDS)
                const int mine = c0 + (int)lane;
                bool hit       = false;
                if(mine < count)
                    hit = block_may_touch(scull[mine], saxis[mine], cx, cy);
                const uint32_t mask = __ballot_sync(0xffffffffu, hit);
                if(mask == 0u)
                    continue;
                if(hit)
                    surv[__popc(mask & lanemask_lt)] = mine;
                __syncwarp();
                const int n_surv = __popc(mask);
                for(int i = 0; i < n_surv; ++i)
                {
                    const int t     = surv[i];
                    const float4 q  = scull[t];
                    const float4 g  = sgeom[t];
                    const float4 cc = scol[t * CV];
                    const float dx = q.x - px, dy = q.y - py;
                    const float e2    = fmaf(g.x * dx, dx, fmaf(g.z * dy, dy, (g.y * dx) * dy)); // = -sigma * log2(e)
                    const float vis   = fast_ex2(e2);
                    const float alpha = fminf(kMaxAlpha, g.w * vis);
                    if(done == 0u && e2 <= 0.f && alpha >= kAlphaThreshold)
                    {
                        const float next_T = T * (1.0f - alpha);
                        if(next_T <= kTransmittanceThreshold)
                            done = 1u; // this pixel is done: exclusive of the current gaussian
                        else
                        {
                            const float w = alpha * T;
                            pix_out[0] += cc.x * w;
                            if constexpr(CDIM > 1)
                                pix_out[1] += cc.y * w;
                            if constexpr(CDIM > 2)
                                pix_out[2] += cc.z * w;
                            if constexpr(CDIM > 3)
                                pix_out[3] += cc.w * w;
                            if constexpr(CDIM > 4)
                            {
#pragma unroll
                                for(int v = 1; v < CV; ++v)
                                {
                                    const float4 c2 = scol[t * CV + v];
                                    if(4 * v + 0 < CDIM) pix_out[4 * v + 0] += c2.x * w;
                                    if(4 * v + 1 < CDIM) pix_out[4 * v + 1] += c2.y * w;
                                    if(4 * v + 2 < CDIM) pix_out[4 * v + 2] += c2.z * w;
                                    if(4 * v + 3 < CDIM) pix_out[4 * v + 3] += c2.w * w;
                                }
                            }
                            cur_idx = first + t;
                            T       = next_T;
                        }
                    }
                }
                __syncwarp(); // the list is rewritten by the next chunk
                if(__all_sync(0xffffffffu, done != 0u))
                    break; // every pixel of this warp is saturated: drop out of the list
            }
        }
        if constexpr(!PIPE)
        {
            // everyone finished reading this stage; tile-level early exit
            const int n_done = __syncthreads_count(done != 0u);
            if(tid == 0)
                mbar_wait(ring.full(stage), parity); // batch b has landed even if no warp needed it
            if(n_done == kWarps * 32)
            {
                last_b = b;
                break;
            }
            if(tid == 0 && b + KS < num_batches)
            {
                const int64_t nfirst = (int64_t)range_start + (int64_t)(b + KS) * kBatch;
                const int ncount     = min(kBatch, (int)(range_end - nfirst));
                ring.issue(stage, gcull, ggeom, gcolor, nfirst, ncount);
            }
        }
        else
        {
            const bool all_done = __all_sync(0xffffffffu, done != 0u);
            if(lane == 0)
            {
                if(warp_alive && all_done)
                    atomicSub(&s_alive, 1);
                __threadfence_block(); // this warp's reads of the stage are done before it is counted off
                if(atomicAdd(&s_cnt[stage], 1) == kWarps - 1)
                { // last warp out: the stage is free
                    atomicExch(&s_cnt[stage], 0);
                    __threadfence_block();
                    if(b + KS < num_batches)
                    {
                        if(atomicAdd(&s_alive, 0) > 0)
                        {
                            const int64_t nfirst = (int64_t)range_start + (int64_t)(b + KS) * kBatch;
                            const int ncount     = min(kBatch, (int)(range_end - nfirst));
                            ring.issue(stage, gcull, ggeom, gcolor, nfirst, ncount);
                        }
                        else
                            atomicMin(&s_stop, b + KS); // every warp is saturated: batches >= b + KS never arrive
                    }
                }
            }
            if(all_done)
                warp_alive = false;
        }
    }
    if constexpr(!PIPE)
    {
        if(tid == 0)
        { // never retire the CTA with bulk copies still in flight into its shared memory
            for(int b = last_b + 1; b < num_batches && b < last_b + KS; ++b)
                mbar_wait(ring.full(b % KS), (uint32_t)(b / KS) & 1u);
        }
    }

    if(inside)
    {
        render_alphas[pix] = 1.0f - T;
#pragma unroll
        for(int k = 0; k < CDIM; ++k)
            render_colors[pix * CDIM + k] = bg ? (pix_out[k] + T * bg[k]) : pix_out[k];
        last_ids[pix] = cur_idx;
    }
}

// ---------------------------------------------------------------------------------------------
// backward: transposed reduction.
//
// Reducing the 9 (+2) per-pixel partials of every surviving (warp, gaussian) pair across the 32 lanes right away
// (butterfly: 12 shuffles + 12 adds + ~26 selects) costs 50 of 130 instructions per survivor, plus 9 scalar REDs.
// Instead the work is split in two phases per warp:
//   phase A (lane = pixel, sequential over the depth-sorted survivors, as before): per survivor each lane only
//     computes TWO scalars -- f = alpha * T (the weight of the gaussian's colour in this pixel) and
//     o = vis * v_alpha (gated like the reference gates v_sigma) -- and stores them into a per-warp shared
//     [survivor][pixel] buffer.  Everything the 9 gradients need is linear in f and o:
//        v_rgb[k] = sum_p f v_c[k](p),  v_opacity = sum_p o,  v_sigma = -opacity * o  and
//        v_xy / v_conic = sums of v_sigma * {dx, dy, dx^2, dx dy, dy^2}.
//     The colour part of v_alpha needs only the SCALAR sum_{behind} fac_j (c_j . v_c) instead of the reference's
//     per-channel `buffer[k]` (same value, one accumulator).
//   phase B (lane = gaussian, after 16 survivors): each lane walks the 16 pixels of one half of the warp's 8x4
//     block for ITS gaussian and accumulates the 6 moments of o about the half block's centre (pixel offsets are
//     compile-time immediates) and the D colour sums in registers -- no cross-lane traffic; the moments are
//     re-centred on the gaussian's mean once per gaussian, the two halves are combined with one shuffle per
//     value, and the 12-float gradient record is added with three 128-bit REDs instead of nine scalar ones.
// Per survivor: 52 + 18 instructions instead of 130 (SASS counts, DESIGN.md section 3).
struct GradDst
{
    float *means2d, *conics, *colors, *opacities, *abs;
    int64_t s_means2d, s_conics, s_colors, s_opacities, s_abs;
};

constexpr int kBwdBatch = 64; // records per ring stage (smaller than the forward's: the per-warp buffers need the room)
constexpr int kRound    = 16; // survivors per reduction round of a warp
constexpr int kRowF2    = 33; // row stride of the round buffer in float2 units (odd: conflict-free in both phases)

template<int CDIM, bool PIPE = false>
struct Bwd2Smem
{
    static constexpr int CV          = RecLayout<CDIM>::kColorVec4;
    static constexpr int KS          = PIPE ? kPipeStages : kStages;
    static constexpr size_t ring_al  = (ring_smem_bytes<CDIM, kBwdBatch, KS>() + 15) & ~size_t(15);
    static constexpr size_t rbuf     = (size_t)kRound * kRowF2 * sizeof(float2);
    static constexpr size_t meta     = (size_t)kRound * 2 * sizeof(float4);
    static constexpr size_t pixc     = (size_t)32 * CV * sizeof(float4);
    static constexpr size_t slot_t   = (size_t)(kRound + 32) * sizeof(int32_t); // slot -> record index, + the chunk's survivor list
    static constexpr size_t per_warp = rbuf + meta + pixc + slot_t;
    static constexpr size_t total    = ring_al + kWarps * per_warp;
};

__device__ __forceinline__ void red_add_v4(float *addr, float a, float b, float c, float d)
{
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// PIPE = true: no CTA barrier in the batch loop.  Every warp waits for the stage's TMA barrier, works through the
// batch at its own pace and then counts itself off on the stage; the LAST warp to do so re-arms the barrier and issues
// the bulk copies of the batch three ahead.  Warps of a tile differ a lot in survivors per 64-record batch, and with
// two CTA barriers per batch every warp ran at the pace of the slowest one.  The gaussian ids are read from global
// memory when a survivor's data is materialised (no per-batch staging, hence no barrier for it either).
// PIPE = false (D > 4): two CTA barriers per batch, the batch's gaussian ids staged in shared memory.
template<int CDIM, bool ABS, int MINB, bool PIPE = false>
__global__ void __launch_bounds__(kWarps * 32, MINB) raster_bwd2_kernel(
    const uint32_t I, const int64_t n_isects, const float4 *__restrict__ gcull, const float4 *__restrict__ ggeom,
    const float4 *__restrict__ gcolor, const int32_t *__restrict__ order, const int32_t *__restrict__ flatten_ids,
    const float *__restrict__ backgrounds, const uint8_t *__restrict__ masks, const uint32_t W, const uint32_t H,
    const uint32_t tw, const uint32_t th, const int32_t *__restrict__ offsets, const float *__restrict__ render_alphas,
    const int32_t *__restrict__ last_ids, const float *__restrict__ v_render_colors,
    const float *__restrict__ v_render_alphas, const GradDst dst, const uint32_t packed_stride
)
{
    constexpr int CV  = RecLayout<CDIM>::kColorVec4;
    constexpr int NV  = 6 + CDIM + (ABS ? 2 : 0); // [v_xy 2 | v_conic 3 | v_opacity 1 | v_rgb CDIM | abs 2]
    constexpr int NV4 = (NV + 3) / 4;
    using SM          = Bwd2Smem<CDIM, PIPE>;
    constexpr int KS  = SM::KS;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Ring<CDIM, kBwdBatch, KS> ring;
    ring.carve(smem_raw);
    __shared__ int32_t s_tile_bin;
    __shared__ int32_t s_done[kPipeStages]; // PIPE: warps that have finished with the stage's current batch

    const TileGeom tg      = decode_tile(order, tw, th);
    const unsigned tid     = threadIdx.x;
    const unsigned warp    = tid >> 5, lane = tid & 31;
    const int64_t tile_lin = (int64_t)tg.image_id * tw * th + tg.tile_id;
    if(masks != nullptr && !masks[tile_lin])
        return;
    const int32_t range_start = offsets[tile_lin];
    const int32_t range_end0  = (tile_lin == (int64_t)I * tw * th - 1) ? (int32_t)n_isects : offsets[tile_lin + 1];
    if(range_end0 <= range_start)
        return;

    const int bx0 = tg.tile_x * kTile + (warp & 1) * 8;
    const int by0 = tg.tile_y * kTile + (warp >> 1) * 4;
    const int px_i = bx0 + (lane & 7), py_i = by0 + (lane >> 3);
    const float px = (float)px_i + 0.5f, py = (float)py_i + 0.5f;
    const bool inside = (px_i < (int)W) && (py_i < (int)H);
    const int64_t pix = inside ? ((int64_t)tg.image_id * H + py_i) * W + px_i : 0;
    const float *bg   = backgrounds ? backgrounds + (size_t)tg.image_id * CDIM : nullptr;

    const float T_final = inside ? 1.0f - render_alphas[pix] : 1.f;
    float T             = T_final;
    float v_render_c[CV * 4];
    float bg_dot = 0.f;
#pragma unroll
    for(int k = 0; k < CV * 4; ++k)
    {
        v_render_c[k] = (k < CDIM && inside) ? v_render_colors[pix * CDIM + k] : 0.f;
        if(bg && k < CDIM)
            bg_dot += bg[k] * v_render_c[k];
    }
    const float v_render_a       = (inside && v_render_alphas != nullptr) ? v_render_alphas[pix] : 0.f; // null: no gradient on alpha
    const int32_t bin_final      = inside ? last_ids[pix] : -1;
    const int32_t warp_bin_final = __reduce_max_sync(0xffffffffu, bin_final);

    if(tid == 0)
    {
        s_tile_bin = -1;
#pragma unroll
        for(int s = 0; s < KS; ++s)
        {
            mbar_init(ring.full(s), 1);
            s_done[s < kPipeStages ? s : 0] = 0;
        }
        fence_mbar_init();
    }
    __syncthreads();
    if(lane == 0)
        atomicMax(&s_tile_bin, warp_bin_final);
    __syncthreads();
    const int32_t range_end = min(range_end0, s_tile_bin + 1);
    if(range_end <= range_start)
        return;

    // per-warp scratch: round buffer [survivor][pixel] of (f, o), per-survivor gaussian data, per-pixel v_render_c
    unsigned char *wbase = smem_raw + SM::ring_al + (size_t)warp * SM::per_warp;
    float2 *rbuf         = reinterpret_cast<float2 *>(wbase);
    float4 *meta         = reinterpret_cast<float4 *>(wbase + SM::rbuf);
    float4 *pixc         = reinterpret_cast<float4 *>(wbase + SM::rbuf + SM::meta);
    int32_t *slot_t      = reinterpret_cast<int32_t *>(wbase + SM::rbuf + SM::meta + SM::pixc); // batch-local record index per slot
    int32_t *surv        = slot_t + kRound;                                                     // survivors of the current 32-record chunk
    const uint32_t lanemask_gt = lane == 31 ? 0u : (0xffffffffu << (lane + 1));
#pragma unroll
    for(int v = 0; v < CV; ++v)
        pixc[lane * CV + v] = make_float4(v_render_c[4 * v], v_render_c[4 * v + 1], v_render_c[4 * v + 2], v_render_c[4 * v + 3]);

    const int num_batches = (range_end - range_start + kBwdBatch - 1) / kBwdBatch;
    auto batch_first = [&](int b) -> int64_t {
        const int64_t bf = (int64_t)range_end - (int64_t)(b + 1) * kBwdBatch;
        return bf > range_start ? bf : (int64_t)range_start;
    };
    auto batch_count = [&](int b) -> int { return (int)((int64_t)range_end - (int64_t)b * kBwdBatch - batch_first(b)); };
    if(tid == 0)
    {
#pragma unroll
        for(int s = 0; s < KS; ++s)
            if(s < num_batches)
                ring.issue(s, gcull, ggeom, gcolor, batch_first(s), batch_count(s));
    }
    const float cx = (float)bx0 + 4.0f, cy = (float)by0 + 2.0f;
    const float Tf_va = T_final * v_render_a - (bg ? T_final * bg_dot : 0.f); // T_final * (v_render_a - bg . v_render_c)
    float behind      = 0.f; // sum over the contributors behind the current one of fac_j * (c_j . v_render_c)

    // ---- phase B: 16 buffered survivors -> gradient records
    // Per-survivor gaussian data is NOT copied in phase A (that cost 20 instructions per survivor on one lane): the
    // batch-local record index goes into slot_t and slots [ncopied, nslots) are copied from the ring stage to `meta`,
    // one slot per lane, right before they are needed (a flush) or before their stage is recycled (end of a batch).
    int ncopied = 0;
    auto materialise = [&](const int nslots, const float4 *scull, const float4 *sgeom, const int32_t *sid) {
        __syncwarp();
        const int sl = (int)lane;
        if(sl >= ncopied && sl < nslots)
        {
            const int t      = slot_t[sl];
            const float4 q   = scull[t];
            const float4 g   = sgeom[t];
            meta[sl * 2]     = make_float4(q.x, q.y, g.x * kConicUnscaleAC, g.y * kConicUnscaleB);
            meta[sl * 2 + 1] = make_float4(g.z * kConicUnscaleAC, g.w, __int_as_float(sid[t]), 0.f); // PIPE: sid = flatten_ids + first
        }
        ncopied = nslots;
    };
    auto flush = [&](const int nslots) {
        __syncwarp();
        const int gslot   = lane & (kRound - 1);
        const int half    = lane >> 4; // which 8x2 half of the 8x4 pixel block this lane sums
        const float2 *row = rbuf + gslot * kRowF2 + half * 16;
        const float4 *pc  = pixc + half * 16 * CV;
        const float4 m0 = meta[gslot * 2], m1 = meta[gslot * 2 + 1]; // {mx, my, a, b}, {c, opacity, id, -}
        const float Dx = m0.x - cx, Dy = m0.y - (cy - 1.0f + 2.0f * (float)half); // mean relative to the half's centre
        float M0 = 0.f, M1 = 0.f, M2 = 0.f, M3 = 0.f, M4 = 0.f, ax = 0.f, ay = 0.f;
        float rgb[CV * 4];
#pragma unroll
        for(int k = 0; k < CV * 4; ++k)
            rgb[k] = 0.f;
#pragma unroll
        for(int i = 0; i < 16; ++i)
        {
            const float2 fo = row[i];
            const float xi = (float)(i & 7) - 3.5f, eta = (float)(i >> 3) - 0.5f; // pixel centre - half centre
            M0 += fo.y;
            M1 = fmaf(fo.y, xi, M1);
            M2 = fmaf(fo.y, eta, M2);
            M3 = fmaf(fo.y, xi * xi, M3);
            M4 = fmaf(fo.y, xi * eta, M4); // eta is +-0.5: the eta^2 moment is 0.25 * M0
#pragma unroll
            for(int v = 0; v < CV; ++v)
            {
                const float4 c4 = pc[i * CV + v];
                rgb[4 * v]     = fmaf(fo.x, c4.x, rgb[4 * v]);
                rgb[4 * v + 1] = fmaf(fo.x, c4.y, rgb[4 * v + 1]);
                rgb[4 * v + 2] = fmaf(fo.x, c4.z, rgb[4 * v + 2]);
                rgb[4 * v + 3] = fmaf(fo.x, c4.w, rgb[4 * v + 3]);
            }
            if constexpr(ABS)
            { // |v_sigma * d sigma/d mean| is not linear in o: summed per pixel
                const float dxp = Dx - xi, dyp = Dy - eta;
                ax += fabsf(fo.y * (m0.z * dxp + m0.w * dyp));
                ay += fabsf(fo.y * (m0.w * dxp + m1.x * dyp));
            }
        }
        // v_sigma = -opacity * o; moments about the gaussian's mean from the moments about the half's centre
        const float nop = -m1.y;
        const float U0 = nop * M0, U1 = nop * M1, U2 = nop * M2, U3 = nop * M3, U4 = nop * M4, U5 = 0.25f * U0;
        const float Sdx = Dx * U0 - U1, Sdy = Dy * U0 - U2; // sum v_sigma dx, sum v_sigma dy
        float vals[NV4 * 4];
        vals[0] = m0.z * Sdx + m0.w * Sdy;
        vals[1] = m0.w * Sdx + m1.x * Sdy;
        vals[2] = 0.5f * (Dx * (Sdx - U1) + U3);
        vals[3] = Dx * Sdy - Dy * U1 + U4;
        vals[4] = 0.5f * (Dy * (Sdy - U2) + U5);
        vals[5] = M0;
#pragma unroll
        for(int k = 0; k < CDIM; ++k)
            vals[6 + k] = rgb[k];
        if constexpr(ABS)
        {
            vals[6 + CDIM] = m1.y * ax;
            vals[7 + CDIM] = m1.y * ay;
        }
#pragma unroll
        for(int k = NV; k < NV4 * 4; ++k)
            vals[k] = 0.f;
#pragma unroll
        for(int k = 0; k < NV; ++k)
            vals[k] += __shfl_xor_sync(0xffffffffu, vals[k], 16);
        if(gslot < nslots)
        {
            const uint32_t gid = __float_as_uint(m1.z);
            if(packed_stride != 0u)
            { // one 16-byte aligned record per gaussian: 128-bit REDs, alternating between the two halves
                float *rec = dst.means2d + (size_t)(gid * packed_stride);
#pragma unroll
                for(int c = 0; c < NV4; ++c)
                    if((c & 1) == half)
                        red_add_v4(rec + 4 * c, vals[4 * c], vals[4 * c + 1], vals[4 * c + 2], vals[4 * c + 3]);
            }
            else if(half == 0)
            {
                atomicAdd(dst.means2d + (size_t)gid * dst.s_means2d, vals[0]);
                atomicAdd(dst.means2d + (size_t)gid * dst.s_means2d + 1, vals[1]);
                atomicAdd(dst.conics + (size_t)gid * dst.s_conics, vals[2]);
                atomicAdd(dst.conics + (size_t)gid * dst.s_conics + 1, vals[3]);
                atomicAdd(dst.conics + (size_t)gid * dst.s_conics + 2, vals[4]);
                atomicAdd(dst.opacities + (size_t)gid * dst.s_opacities, vals[5]);
#pragma unroll
                for(int k = 0; k < CDIM; ++k)
                    atomicAdd(dst.colors + (size_t)gid * dst.s_colors + k, vals[6 + k]);
                if constexpr(ABS)
                {
                    atomicAdd(dst.abs + (size_t)gid * dst.s_abs, vals[6 + CDIM]);
                    atomicAdd(dst.abs + (size_t)gid * dst.s_abs + 1, vals[7 + CDIM]);
                }
            }
        }
        __syncwarp();
    };

    int nslots = 0;
    for(int b = 0; b < num_batches; ++b)
    {
        const int stage       = b % KS;
        const uint32_t parity = (uint32_t)(b / KS) & 1u;
        const int32_t first   = (int32_t)batch_first(b);
        const int count       = batch_count(b);
        if constexpr(!PIPE)
        {
            if((int)tid < count)
                ring.ids(stage)[tid] = flatten_ids[first + tid];
            __syncthreads();
        }
        else
            mbar_wait(ring.full(stage), parity); // every warp, also one that skips the batch: keeps the stage counters in step
        if(first <= warp_bin_final)
        {
            if constexpr(!PIPE)
                mbar_wait(ring.full(stage), parity);
            const float4 *scull = ring.cull(stage);
            const float4 *saxis = ring.axis(stage);
            const float4 *sgeom = ring.geom(stage);
            const float4 *scol  = ring.color(stage);
            const int32_t *sid  = PIPE ? flatten_ids + first : ring.ids(stage);
            const int lim       = bin_final - first;      // local index of this pixel's last contributor
            const int warp_lim  = warp_bin_final - first; // ... of the warp's
            for(int c1 = count; c1 > 0; c1 -= 32)
            {
                const int c0   = c1 - 32; // chunk covers local [c0, c1); c0 may be negative
                const int mine = c0 + (int)lane;
                bool hit       = false;
                if(mine >= 0 && mine <= warp_lim)
                    hit = block_may_touch(scull[mine], saxis[mine], cx, cy);
                const uint32_t mask = __ballot_sync(0xffffffffu, hit);
                if(mask == 0u)
                    continue;
                // survivors compacted back to front into the per-warp list (one LDS per survivor instead of walking the mask)
                if(hit)
                    surv[__popc(mask & lanemask_gt)] = mine;
                __syncwarp();
                const int n_surv = __popc(mask);
                for(int si = 0; si < n_surv; ++si)
                {
                    const int t    = surv[si];
                    const float4 q = scull[t];
                    const float4 g = sgeom[t];
                    const float dx = q.x - px, dy = q.y - py;
                    const float e2    = fmaf(g.x * dx, dx, fmaf(g.z * dy, dy, (g.y * dx) * dy)); // = -sigma * log2(e)
                    const float vis   = fast_ex2(e2);
                    const float ov    = g.w * vis;
                    const float alpha = fminf(kMaxAlpha, ov);
                    const bool valid  = (t <= lim) && e2 <= 0.f && alpha >= kAlphaThreshold;
                    if(!__any_sync(0xffffffffu, valid))
                        continue;
                    float f = 0.f, o = 0.f;
                    if(valid)
                    {
                        float dot = 0.f;
#pragma unroll
                        for(int v = 0; v < CV; ++v)
                        {
                            const float4 cc = scol[t * CV + v];
                            dot = fmaf(cc.x, v_render_c[4 * v], dot);
                            if(4 * v + 1 < CDIM) dot = fmaf(cc.y, v_render_c[4 * v + 1], dot);
                            if(4 * v + 2 < CDIM) dot = fmaf(cc.z, v_render_c[4 * v + 2], dot);
                            if(4 * v + 3 < CDIM) dot = fmaf(cc.w, v_render_c[4 * v + 3], dot);
                        }
                        const float ra = fast_rcp(fmaxf(kMinOneMinusAlpha, 1.0f - alpha));
                        T *= ra;
                        f                   = alpha * T;
                        const float v_alpha = fmaf(dot, T, ra * (Tf_va - behind));
                        behind              = fmaf(dot, f, behind);
                        if(ov <= kMaxAlpha)
                            o = vis * v_alpha;
                    }
                    rbuf[nslots * kRowF2 + lane] = make_float2(f, o);
                    if(lane == 0)
                        slot_t[nslots] = t;
                    if(++nslots == kRound)
                    {
                        materialise(kRound, scull, sgeom, sid);
                        flush(kRound);
                        nslots = ncopied = 0;
                    }
                }
                __syncwarp(); // the list is rewritten by the next chunk
            }
            if(nslots > ncopied) // pending survivors of this batch: keep their data before the stage is recycled
                materialise(nslots, scull, sgeom, sid);
        }
        if constexpr(!PIPE)
        {
            __syncthreads(); // stage (records + ids) fully consumed
            if(tid == 0)
            {
                mbar_wait(ring.full(stage), parity); // landed even if every warp skipped it
                if(b + KS < num_batches)
                    ring.issue(stage, gcull, ggeom, gcolor, batch_first(b + KS), batch_count(b + KS));
            }
        }
        else
        {
            __syncwarp();
            if(lane == 0)
            {
                __threadfence_block(); // this warp's reads of the stage are done before it is counted off
                if(atomicAdd(&s_done[stage], 1) == kWarps - 1)
                { // last warp out: the stage is free -- re-arm it and fetch the batch KS ahead
                    atomicExch(&s_done[stage], 0);
                    __threadfence_block();
                    if(b + KS < num_batches)
                        ring.issue(stage, gcull, ggeom, gcolor, batch_first(b + KS), batch_count(b + KS));
                }
            }
        }
    }
    if(nslots > 0)
        flush(nslots);
}

// ---------------------------------------------------------------------------------------------
// record streams + tile dispatch order of one view batch (the first stage of the forward; also callable on its own,
// gsb200_raster_pack, for bindings that rebuild the records in their backward instead of keeping them alive)
// The tile dispatch order (one CTA, ~9 us) depends only on the offsets: it runs on a side stream next to the pack pass
// (fork / join by events, one set per device, created on first use).
struct SideLane
{
    cudaStream_t stream = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
};
static std::mutex g_side_mu; // held from fork to join: the event pair of a device is shared by all callers
static SideLane *side_lane()
{
    static SideLane lanes[64];
    int dev = 0;
    if(cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64)
        return nullptr;
    SideLane &l = lanes[dev];
    if(l.stream == nullptr)
    {
        if(cudaStreamCreateWithFlags(&l.stream, cudaStreamNonBlocking) != cudaSuccess
           || cudaEventCreateWithFlags(&l.fork, cudaEventDisableTiming) != cudaSuccess
           || cudaEventCreateWithFlags(&l.join, cudaEventDisableTiming) != cudaSuccess)
        {
            l.stream = nullptr;
            return nullptr;
        }
    }
    return &l;
}

template<int CDIM>
static int launch_pack(
    const float *means2d, const float *conics, const float *colors, const float *opacities, const int32_t *offsets,
    const int32_t *flatten_ids, int64_t S, unsigned n_tiles, void *records, cudaStream_t st, const float4 *rows = nullptr
)
{
    RecordStreams r = carve_records(records, S, RecLayout<CDIM>::kColorVec4);
    const bool want_order = S > 0 && n_tiles >= 2 * 148; // enough tiles for dispatch order to matter
    std::unique_lock<std::mutex> side_lock(g_side_mu, std::defer_lock);
    if(want_order)
        side_lock.lock();
    SideLane *lane = want_order ? side_lane() : nullptr;
    if(lane != nullptr)
    {
        GSB_CUDA_TRY(cudaEventRecord(lane->fork, st));
        GSB_CUDA_TRY(cudaStreamWaitEvent(lane->stream, lane->fork, 0));
        tile_order_kernel<<<1, 1024, 0, lane->stream>>>(offsets, (int32_t)n_tiles, (int32_t)S, r.order);
        if(int rc = check_launch())
            return rc;
        GSB_CUDA_TRY(cudaEventRecord(lane->join, lane->stream));
    }
    if(S > 0)
    {
        if(rows != nullptr && CDIM <= 4) // 64-byte row records from the fused projection: gather only
            pack_rows_kernel<<<grid_for(S, kPackUnroll * 64), 256, 0, st>>>(S, flatten_ids, rows, r.cull, r.axis, r.geom, r.color);
        else
            pack_records_kernel<CDIM><<<grid_for(S, 256), 256, 0, st>>>(
                S, flatten_ids, means2d, conics, colors, opacities, r.cull, r.axis, r.geom, r.color
            );
        if(int rc = check_launch())
            return rc;
    }
    if(lane != nullptr)
        GSB_CUDA_TRY(cudaStreamWaitEvent(st, lane->join, 0));
    else if(want_order)
    {
        tile_order_kernel<<<1, 1024, 0, st>>>(offsets, (int32_t)n_tiles, (int32_t)S, r.order);
        if(int rc = check_launch())
            return rc;
    }
    return GSB200_OK;
}

// ---------------------------------------------------------------------------------------------
template<int CDIM>
static int launch_fwd(
    int64_t I, int64_t N, const float *means2d, const float *conics, const float *colors, const float *opacities,
    const float *backgrounds, const uint8_t *masks, uint32_t W, uint32_t H, uint32_t tw, uint32_t th,
    const int32_t *offsets, const int32_t *flatten_ids, int64_t S, void *records, float *render_colors,
    float *render_alphas, int32_t *last_ids, cudaStream_t st, const float4 *rows = nullptr
)
{
    (void)N;
    const unsigned n_tiles = (unsigned)(I * tw * th);
    if(int rc = launch_pack<CDIM>(means2d, conics, colors, opacities, offsets, flatten_ids, S, n_tiles, records, st, rows))
        return rc;
    RecordStreams r      = carve_records(records, S, RecLayout<CDIM>::kColorVec4);
    const int32_t *order = (S > 0 && n_tiles >= 2 * 148) ? r.order : nullptr;
    // CDIM <= 4: barrier-free ring (0.333 -> 0.304 ms incl. pack at cfg3 on a B200); CDIM > 4: the CTA-barrier ring
    constexpr bool PIPE = CDIM <= 4;
    const size_t smem   = ring_smem_bytes<CDIM, kBatch, PIPE ? kPipeStages : kStages>();
    GSB_CUDA_TRY(cudaFuncSetAttribute(raster_fwd_kernel<CDIM, PIPE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    raster_fwd_kernel<CDIM, PIPE><<<n_tiles, kWarps * 32, smem, st>>>(
        (uint32_t)I, S, r.cull, r.geom, r.color, order, backgrounds, masks, W, H, tw, th, offsets, render_colors,
        render_alphas, last_ids
    );
    return check_launch();
}

template<int CDIM>
static int launch_bwd(
    int64_t I, const float *backgrounds, const uint8_t *masks, uint32_t W, uint32_t H, uint32_t tw, uint32_t th,
    const int32_t *offsets, const int32_t *flatten_ids, int64_t S, const void *records, const float *render_alphas,
    const int32_t *last_ids, const float *v_render_colors, const float *v_render_alphas, const GradDst &dst,
    cudaStream_t st
)
{
    if(S == 0)
        return GSB200_OK; // reference: no launch when there are no intersections (Bwd.cu:350-354)
    RecordStreams r    = carve_records(const_cast<void *>(records), S, RecLayout<CDIM>::kColorVec4);
    const unsigned n_tiles = (unsigned)(I * tw * th);
    const int32_t *order   = (n_tiles >= 2 * 148) ? r.order : nullptr; // written by the forward
    const bool absg        = dst.abs != nullptr;
    // are the five destinations one packed, 16-byte aligned record [v_xy 2 | v_conic 3 | v_opacity 1 | v_rgb D | abs 2]?
    const int64_t P = dst.s_means2d;
    uint32_t packed = 0;
    if(P > 0 && (P % 4) == 0 && P >= 6 + CDIM + (absg ? 2 : 0) && dst.s_conics == P && dst.s_colors == P && dst.s_opacities == P
       && dst.conics == dst.means2d + 2 && dst.opacities == dst.means2d + 5 && dst.colors == dst.means2d + 6
       && (!absg || (dst.s_abs == P && dst.abs == dst.means2d + 6 + CDIM)) && (reinterpret_cast<uintptr_t>(dst.means2d) & 15) == 0)
        packed = (uint32_t)P;
    // CDIM <= 4: barrier-free ring, registers held to 4 CTAs / SM; CDIM > 4: the CTA-barrier ring
    constexpr bool PIPE = CDIM <= 4;
    constexpr int MINB  = CDIM <= 4 ? 4 : 1;
    const size_t smem   = Bwd2Smem<CDIM, PIPE>::total;
    auto launch = [&](auto kernel) -> int {
        GSB_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kernel<<<n_tiles, kWarps * 32, smem, st>>>(
            (uint32_t)I, S, r.cull, r.geom, r.color, order, flatten_ids, backgrounds, masks, W, H, tw, th, offsets,
            render_alphas, last_ids, v_render_colors, v_render_alphas, dst, packed
        );
        return check_launch();
    };
    return absg ? launch(raster_bwd2_kernel<CDIM, true, MINB, PIPE>) : launch(raster_bwd2_kernel<CDIM, false, MINB, PIPE>);
}
} // namespace gsb

// ---------------------------------------------------------------------------------------------
// C ABI
#define GSB_FOR_CHANNELS(X) X(1) X(2) X(3) X(4) X(5) X(8) X(16) X(32)

extern "C" int gsb200_raster_supports_channels(int D)
{
    switch(D)
    {
#define X(n) case n:
        GSB_FOR_CHANNELS(X)
#undef X
        return 1;
    default:
        return 0;
    }
}

extern "C" size_t gsb200_raster_records_bytes(int64_t n_isects, int D, int64_t n_tiles)
{
    if(n_isects < 0 || D <= 0 || n_tiles < 0)
        return 0;
    const size_t cv = (size_t)((D + 3) / 4);
    return 3 * gsb::align256((size_t)n_isects * 16) + gsb::align256((size_t)n_isects * 16 * cv)
         + gsb::align256((size_t)(n_tiles + 1) * 4) + 256;
}

extern "C" int gsb200_raster_pack(
    int64_t I, int D, const float *means2d, const float *conics, const float *colors, const float *opacities,
    uint32_t tile_width, uint32_t tile_height, const int32_t *offsets, const int32_t *flatten_ids, int64_t n_isects,
    void *records, void *stream
)
{
    if(I < 0 || n_isects < 0 || !offsets)
        return GSB200_E_INVALID;
    if(n_isects == 0 || I == 0)
        return GSB200_OK;
    if(!means2d || !conics || !colors || !opacities || !flatten_ids || !records)
        return GSB200_E_INVALID;
    const unsigned n_tiles = (unsigned)(I * tile_width * tile_height);
    cudaStream_t st        = (cudaStream_t)stream;
    switch(D)
    {
#define X(n)                                                                                                         \
    case n:                                                                                                          \
        return gsb::launch_pack<n>(means2d, conics, colors, opacities, offsets, flatten_ids, n_isects, n_tiles, records, st);
        GSB_FOR_CHANNELS(X)
#undef X
    default:
        return GSB200_E_UNSUPPORTED;
    }
}

extern "C" int gsb200_raster_fwd(
    int64_t I, int64_t N, int D, const float *means2d, const float *conics, const float *colors,
    const float *opacities, const float *backgrounds, const uint8_t *masks, uint32_t image_width,
    uint32_t image_height, uint32_t tile_size, uint32_t tile_width, uint32_t tile_height, const int32_t *offsets,
    const int32_t *flatten_ids, int64_t n_isects, void *records, float *render_colors, float *render_alphas,
    int32_t *last_ids, void *stream
)
{
    if(I < 0 || N < 0 || n_isects < 0 || !offsets || !render_colors || !render_alphas || !last_ids)
        return GSB200_E_INVALID;
    if(n_isects > 0 && (!means2d || !conics || !colors || !opacities || !flatten_ids || !records))
        return GSB200_E_INVALID;
    if(tile_size != (uint32_t)gsb::kTile)
        return GSB200_E_UNSUPPORTED;
    if(I == 0 || image_width == 0 || image_height == 0)
        return GSB200_OK;
    if((uint64_t)tile_width * gsb::kTile < image_width || (uint64_t)tile_height * gsb::kTile < image_height)
        return GSB200_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    switch(D)
    {
#define X(n)                                                                                                         \
    case n:                                                                                                          \
        return gsb::launch_fwd<n>(                                                                                   \
            I, N, means2d, conics, colors, opacities, backgrounds, masks, image_width, image_height, tile_width,     \
            tile_height, offsets, flatten_ids, n_isects, records, render_colors, render_alphas, last_ids, st        \
        );
        GSB_FOR_CHANNELS(X)
#undef X
    default:
        return GSB200_E_UNSUPPORTED;
    }
}

// Forward from the 64-byte row records {cull | axis | geom | color} that gsb200_project_sh_fwd_rows wrote (D <= 4).
extern "C" int gsb200_raster_fwd_rows(
    int64_t I, int64_t N, int D, const void *row_records, const float *backgrounds, const uint8_t *masks, uint32_t image_width,
    uint32_t image_height, uint32_t tile_size, uint32_t tile_width, uint32_t tile_height, const int32_t *offsets,
    const int32_t *flatten_ids, int64_t n_isects, void *records, float *render_colors, float *render_alphas,
    int32_t *last_ids, void *stream
)
{
    if(I < 0 || N < 0 || n_isects < 0 || !offsets || !render_colors || !render_alphas || !last_ids)
        return GSB200_E_INVALID;
    if(n_isects > 0 && (!row_records || !flatten_ids || !records || (reinterpret_cast<uintptr_t>(row_records) & 15) != 0))
        return GSB200_E_INVALID;
    if(tile_size != (uint32_t)gsb::kTile || D > 4)
        return GSB200_E_UNSUPPORTED;
    if(I == 0 || image_width == 0 || image_height == 0)
        return GSB200_OK;
    if((uint64_t)tile_width * gsb::kTile < image_width || (uint64_t)tile_height * gsb::kTile < image_height)
        return GSB200_E_INVALID;
    cudaStream_t st  = (cudaStream_t)stream;
    const float4 *rr = static_cast<const float4 *>(row_records);
    switch(D)
    {
#define X(n)                                                                                                         \
    case n:                                                                                                          \
        return gsb::launch_fwd<n>(                                                                                   \
            I, N, nullptr, nullptr, nullptr, nullptr, backgrounds, masks, image_width, image_height, tile_width,    \
            tile_height, offsets, flatten_ids, n_isects, records, render_colors, render_alphas, last_ids, st, rr    \
        );
        X(1) X(2) X(3) X(4)
#undef X
    default:
        return GSB200_E_UNSUPPORTED;
    }
}

extern "C" int gsb200_raster_bwd(
    int64_t I, int64_t N, int D, const float *backgrounds, const uint8_t *masks, uint32_t image_width,
    uint32_t image_height, uint32_t tile_size, uint32_t tile_width, uint32_t tile_height, const int32_t *offsets,
    const int32_t *flatten_ids, int64_t n_isects, const void *records, const float *render_alphas,
    const int32_t *last_ids, const float *v_render_colors, const float *v_render_alphas, float *v_means2d,
    int64_t v_means2d_stride, float *v_conics, int64_t v_conics_stride, float *v_colors, int64_t v_colors_stride,
    float *v_opacities, int64_t v_opacities_stride, float *v_means2d_abs, int64_t v_means2d_abs_stride, void *stream
)
{
    if(I < 0 || N < 0 || n_isects < 0)
        return GSB200_E_INVALID;
    if(tile_size != (uint32_t)gsb::kTile)
        return GSB200_E_UNSUPPORTED;
    if(n_isects == 0 || I == 0)
        return GSB200_OK;
    if(!offsets || !flatten_ids || !records || !render_alphas || !last_ids || !v_render_colors
       || !v_means2d || !v_conics || !v_colors || !v_opacities)
        return GSB200_E_INVALID;
    {   // the kernels address gradient rows with 32-bit element offsets
        const int64_t smax = std::max(std::max(v_means2d_stride, v_conics_stride), std::max(std::max(v_colors_stride, v_opacities_stride), v_means2d_abs ? v_means2d_abs_stride : (int64_t)0));
        if(smax < 0 || (double)I * (double)N * (double)smax >= 4294967296.0)
            return GSB200_E_UNSUPPORTED;
    }
    gsb::GradDst dst;
    dst.means2d = v_means2d, dst.s_means2d = v_means2d_stride;
    dst.conics = v_conics, dst.s_conics = v_conics_stride;
    dst.colors = v_colors, dst.s_colors = v_colors_stride;
    dst.opacities = v_opacities, dst.s_opacities = v_opacities_stride;
    dst.abs = v_means2d_abs, dst.s_abs = v_means2d_abs_stride;
    cudaStream_t st = (cudaStream_t)stream;
    switch(D)
    {
#define X(n)                                                                                                       \
    case n:                                                                                                        \
        return gsb::launch_bwd<n>(                                                                                 \
            I, backgrounds, masks, image_width, image_height, tile_width, tile_height, offsets, flatten_ids,       \
            n_isects, records, render_alphas, last_ids, v_render_colors, v_render_alphas, dst, st                  \
        );
        GSB_FOR_CHANNELS(X)
#undef X
    default:
        return GSB200_E_UNSUPPORTED;
    }
}
