// composite.cu -- stage 3: tile-binned front-to-back alpha compositing on sm_100a.
//
// Replaces the reference's instanced-quad draw + fixed-function blending: vs_main/fs_main
// (gaussian.wgsl:30-66) and PREMULTIPLIED_ALPHA_BLENDING (renderer.rs:63-67).  Per pixel the
// reference computes, over all splats in ascending key order (far -> near),
//     a = p.p, p = (2[v1 v2])^-1 (ndc - c);  discard if a > 2*CUTOFF;
//     b = min(0.99, exp(-a) * alpha);        dst = (rgb*b, b) + dst * (1 - b).
// Here one CTA owns one 16x16 tile and walks the tile's slice of the sorted pair list from
// its END (nearest splat) to its begin, accumulating C += rgb*b*T, T *= (1-b): the same sum,
// associated front-to-back, which allows the early-out once T < 2^-16.
//
//  * each warp owns an 8x4 pixel block; splats are staged 256 at a time into shared memory
//    (decoded from the 20-B f16 record once per tile, not once per pixel);
//  * per 32 staged splats every lane tests one splat's bounding box against the warp's
//    pixel block and a ballot compacts the survivors: a warp only evaluates splats that
//    can touch its 32 pixels (most of a tile's list does not), and skips everything once
//    all of its pixels are saturated (warp-level early-out);
//  * the centre is expressed relative to the tile origin with exact f16 x integer products,
//    so `a` carries ~1e-5 absolute error at 4K instead of ulp(3840);
//  * the per-hit code is branch-free and keeps no `done` flag: a pixel whose transmittance falls below 2^-16 has its
//    T set to exactly 0, after which every further weight is exactly 0 (round 1 tested a flag per hit: 35 SASS
//    instructions per warp x splat hit, 28 now -- the kernel is issue-bound, profiles/r02*_ncu_summary.md).
#include "ws_device.cuh"
#include "ws_kernels.h"

namespace ws {

namespace {

constexpr int CB_THREADS = 256;
constexpr int CB_BATCH = 256;
constexpr float T_EPS = 1.52587890625e-5f;   // 2^-16: early-out once the remaining transmittance cannot move the result by more
constexpr float LOG2E = 1.4426950408889634f;
constexpr float SQRT_LOG2E = 1.2011224087864498f;

__device__ __forceinline__ float hlo(uint32_t w) { __half_raw r; r.x = (unsigned short)(w & 0xffffu); return __half2float(__half(r)); }
__device__ __forceinline__ float hhi(uint32_t w) { __half_raw r; r.x = (unsigned short)(w >> 16); return __half2float(__half(r)); }
// MUFU.EX2: the argument is in [-6.8, 0], far from the denormal range, so .ftz is exact enough
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

struct RawSplat { uint32_t w[5]; };

// staged form of one splat, in pixel coordinates relative to the tile CENTRE (u, v in [-7.5, 7.5]):
//   A = {q0, q1, q2, q3}   B = {q4, q5, alpha, r}   C = {g, b, | cx, cy, ex, ey in D}
// a * log2(e) = q0 + q1 u + q2 v + q3 u^2 + q4 u v + q5 v^2  (five FMAs per pixel); the quadratic form
// is S = log2(e) * Binv^T Binv of the pixel-space map [dx;dy] = Bm p.  Centring on the tile keeps the
// cancellation error of the expanded form below ~6e-5 in `a` even for the smallest footprints
// (sigma^2 = kernel_size), inside the parity tolerance window (DESIGN.md section 5).
__device__ __forceinline__ void decode_splat(const RawSplat &rs, float fw, float fh, float hw, float hh, float ox, float oy,
                                             float4 &A, float4 &B, float4 &C, float4 &D)
{
    const float v1x = hlo(rs.w[0]), v1y = hhi(rs.w[0]), v2x = hlo(rs.w[1]), v2y = hhi(rs.w[1]);
    const float ccx = hlo(rs.w[2]), ccy = hhi(rs.w[2]);
    // pixel-space map  [dx;dy] = Bm p,  Bm = [[W v1x, W v2x],[-H v1y, -H v2y]]  (y down)
    const float b00 = fw * v1x, b01 = fw * v2x, b10 = -(fh * v1y), b11 = -(fh * v2y);   // exact products
    const float det = b00 * b11 - b01 * b10;
    const float inv = SQRT_LOG2E / det;
    const float i00 = b11 * inv, i01 = -b01 * inv, i10 = -b10 * inv, i11 = b00 * inv;  // sqrt(log2 e) * Binv
    const float s00 = i00 * i00 + i10 * i10, s01 = i00 * i01 + i10 * i11, s11 = i01 * i01 + i11 * i11;
    const float cx = ccx * hw + ox;              // centre relative to the tile centre (exact product + 1 rounding)
    const float cy = oy - ccy * hh;
    const float tx = s00 * cx + s01 * cy, ty = s01 * cx + s11 * cy;                    // S c
    A.x = tx * cx + ty * cy;                     // q0 = c^T S c
    A.y = -2.f * tx;                             // q1
    A.z = -2.f * ty;                             // q2
    A.w = s00;                                   // q3
    B.x = 2.f * s01;                             // q4
    B.y = s11;                                   // q5
    B.z = hhi(rs.w[4]);                          // alpha
    B.w = hlo(rs.w[3]);                          // r
    C.x = hhi(rs.w[3]); C.y = hlo(rs.w[4]);      // g, b
    C.z = 0.f; C.w = 0.f;
    D.x = cx; D.y = cy;
    D.z = FOOTPRINT_R * (fw * sqrtf(v1x * v1x + v2x * v2x)) + RECT_PAD;
    D.w = FOOTPRINT_R * (fh * sqrtf(v1y * v1y + v2y * v2y)) + RECT_PAD;
}

// MODE 0: the tile's whole list in one pass.  Occlusion split (two depth slabs, nearest first): MODE 1 walks the near
// slab's list and leaves {r, g, b, T} per pixel plus a per-tile "every pixel saturated" flag; MODE 2 resumes from that
// state over the far slab's list (which holds no pair of splats that only touch saturated tiles) and writes the pixels.
// Per pixel the sequence of blends and early-out tests is exactly that of MODE 0, so the image is bit-identical.
template <int FORMAT, int MODE>
__global__ void __launch_bounds__(CB_THREADS)
composite_kernel(CompositeArgs a)
{
    // double-buffered staging: batch b+1 is fetched (global gathers) while batch b is evaluated.  One 48-B record per
    // splat {A, B, C}: the hit loop addresses it with ONE uniform base (three ULEAs in round 1)
    __shared__ float4 s_abc[2][CB_BATCH * 3];
    __shared__ float4 s_d[2][CB_BATCH];              // bounding box for the per-warp cull (dense: conflict-free LDS.128)

    const unsigned tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint32_t W = a.uniforms->width, H = a.uniforms->height;
    const uint32_t tile_x = blockIdx.x, tile_y = blockIdx.y + a.tile_y0;
    const uint32_t tile = (blockIdx.z * gridDim.y + tile_y) * gridDim.x + tile_x;     // z > 0 only in batches (tile_y0 = 0)
    uint2 range = a.ranges[tile];
    range.y = ~range.y;                                  // stored complemented (atomicMin in the sort's last pass)
    if (range.y <= range.x) range.x = range.y = 0u;      // untouched tile
    const float fw = (float)W, fh = (float)H;
    const float hw = 0.5f * fw, hh = 0.5f * fh;
    const float ox = hw - (float)(tile_x * TILE + TILE / 2), oy = hh - (float)(tile_y * TILE + TILE / 2);   // exact

    // warp's 8x4 pixel block inside the tile
    const uint32_t bx = (warp & 1u) * 8u, by = (warp >> 1) * 4u;
    const uint32_t lx = bx + (lane & 7u), ly = by + (lane >> 3);
    const uint32_t px = tile_x * TILE + lx, py = tile_y * TILE + ly;
    const bool inside = (px < W) && (py < H);
    const float fx = (float)lx - 7.5f, fy = (float)ly - 7.5f;          // pixel centre relative to the tile centre
    const float fxx = fx * fx, fxy = fx * fy, fyy = fy * fy;
    // block bounds in pixel-centre coordinates relative to the tile centre
    const float blo_x = (float)bx - 7.5f, bhi_x = (float)bx - 0.5f;
    const float blo_y = (float)by - 7.5f, bhi_y = (float)by - 4.5f;

    // T == 0 means "saturated" (or outside the frame): nothing can change the pixel any more
    float T = inside ? 1.f : 0.f, cr = 0.f, cg = 0.f, cb = 0.f;
    if (MODE == 2) {
        if (inside) {
            const float4 st = a.state[((size_t)blockIdx.z * H + py) * W + px];
            cr = st.x; cg = st.y; cb = st.z; T = st.w;
        }
        if (a.tile_done[tile]) range.x = range.y = 0u;   // saturated by the near slab: nothing of the far slab can show
    }

    int32_t remaining = (int32_t)(range.y - range.x);
    uint32_t cursor = range.y;           // walk from the end: nearest first

    auto fetch = [&](RawSplat &rs, uint32_t cur, int cnt) {
        if ((int)tid < cnt) {
            const uint32_t slot = __ldg(a.pair_slots + (cur - 1u - tid));
            const uint32_t *sp = a.splats + (size_t)slot * 5u;
#pragma unroll
            for (int q = 0; q < 5; q++) rs.w[q] = __ldg(sp + q);
        }
    };

    RawSplat nxt;
    int cnt = remaining < CB_BATCH ? remaining : CB_BATCH;
    fetch(nxt, cursor, cnt);
    int buf = 0;
    while (remaining > 0) {
        // publish the fetched batch
        if ((int)tid < cnt) {
            float4 A, B, C, D;
            decode_splat(nxt, fw, fh, hw, hh, ox, oy, A, B, C, D);
            float4 *rec = &s_abc[buf][tid * 3];
            rec[0] = A; rec[1] = B; rec[2] = C; s_d[buf][tid] = D;
        }
        const bool warp_done = __all_sync(0xffffffffu, T == 0.f);
        // one barrier per batch: makes the batch visible and agrees on the tile-level early-out.  Buffer
        // `buf` was last read two batches ago, and every warp has passed the previous barrier since.
        if (__syncthreads_and(warp_done ? 1 : 0)) break;
        const int cur_cnt = cnt;
        remaining -= cur_cnt;
        cursor -= (uint32_t)cur_cnt;
        cnt = remaining < CB_BATCH ? remaining : CB_BATCH;
        if (remaining > 0) fetch(nxt, cursor, cnt);          // in flight while this batch is evaluated

        if (!warp_done) {
            const float4 *sabc = s_abc[buf], *sd = s_d[buf];
            // one pixel-splat evaluation, branch-free: 5 FMAs for a*log2(e), MUFU.EX2, weight (0 outside the footprint:
            // a select, so a NaN `a` -- degenerate axes -- contributes nothing), blend, saturation clamp of T
#define WS_EVAL(J)                                                                              \
            {                                                                                   \
                const float4 *rec = sabc + (J) * 3;                                             \
                const float4 A = rec[0];                                                        \
                const float4 B = rec[1];                                                        \
                const float2 C = *reinterpret_cast<const float2 *>(rec + 2);                    \
                float aa = fmaf(A.y, fx, A.x);                                                  \
                aa = fmaf(A.z, fy, aa); aa = fmaf(A.w, fxx, aa); aa = fmaf(B.x, fxy, aa); aa = fmaf(B.y, fyy, aa); \
                float wt = fminf(0.99f, ex2_approx(-aa) * B.z) * T;                             \
                wt = (aa <= TWO_CUTOFF * LOG2E) ? wt : 0.f;                                     \
                cr = fmaf(B.w, wt, cr); cg = fmaf(C.x, wt, cg); cb = fmaf(C.y, wt, cb);         \
                T -= wt;                                          /* T * (1 - w) */             \
                T = (T < T_EPS) ? 0.f : T;                                                      \
            }
            unsigned act = __ballot_sync(0xffffffffu, T != 0.f);        // lanes (pixels) that can still change
            for (int c0 = 0; c0 < cur_cnt; c0 += 32) {
                // cull against the bounding box of the pixels that are still unsaturated, not the whole 8x4 block: a splat that
                // only reaches saturated pixels contributes exactly nothing (their T is 0), so skipping it changes no bit
                float lo_x = blo_x, hi_x = bhi_x, lo_y = blo_y, hi_y = bhi_y;
                if (a.active_cull && act != 0xffffffffu) {
                    const unsigned cols = (act | (act >> 8) | (act >> 16) | (act >> 24)) & 0xffu;      // lane = y * 8 + x
                    const unsigned rows = ((act & 0xffu) ? 1u : 0u) | ((act & 0xff00u) ? 2u : 0u) | ((act & 0xff0000u) ? 4u : 0u) | ((act >> 24) ? 8u : 0u);
                    lo_x = blo_x + (float)(__ffs(cols) - 1); hi_x = blo_x + (float)(31 - __clz(cols));
                    lo_y = blo_y + (float)(__ffs(rows) - 1); hi_y = blo_y + (float)(31 - __clz(rows));
                }
                const int k = c0 + (int)lane;
                bool hit = false;
                if (k < cur_cnt) {
                    const float4 D = sd[k];
                    hit = (D.x + D.z >= lo_x) && (D.x - D.z <= hi_x) && (D.y + D.w >= lo_y) && (D.y - D.w <= hi_y);
                }
                unsigned m = __ballot_sync(0xffffffffu, hit);
                while (m) {                                             // two hits per trip: front-to-back order is kept
                    const int j0 = c0 + (__ffs(m) - 1);
                    m &= m - 1u;
                    WS_EVAL(j0)
                    if (m) {
                        const int j1 = c0 + (__ffs(m) - 1);
                        m &= m - 1u;
                        WS_EVAL(j1)
                    }
                }
                act = __ballot_sync(0xffffffffu, T != 0.f);
                if (act == 0u) break;
            }
#undef WS_EVAL
        }
        buf ^= 1;
    }

    if (MODE == 1) {
        if (inside) a.state[((size_t)blockIdx.z * H + py) * W + px] = make_float4(cr, cg, cb, T);
        const int all_done = __syncthreads_and(T == 0.f ? 1 : 0);
        if (tid == 0) a.tile_done[tile] = (uint8_t)(all_done ? 1 : 0);
        return;
    }
    if (inside) {
        const float r = cr + a.clear[0] * T, g = cg + a.clear[1] * T, b = cb + a.clear[2] * T;
        const float al = (1.f - T) + a.clear[3] * T;
        uint8_t *row = reinterpret_cast<uint8_t *>(a.dst) + blockIdx.z * a.view_stride + (size_t)(py - a.tile_y0 * TILE) * a.row_pitch;
        if (FORMAT == 2) {
            reinterpret_cast<float4 *>(row)[px] = make_float4(r, g, b, al);
        } else if (FORMAT == 1) {
            __half_raw h0 = __float2half_rn(r), h1 = __float2half_rn(g), h2 = __float2half_rn(b), h3 = __float2half_rn(al);
            reinterpret_cast<uint2 *>(row)[px] = make_uint2((uint32_t)h0.x | ((uint32_t)h1.x << 16), (uint32_t)h2.x | ((uint32_t)h3.x << 16));
        } else {
            const uint32_t r8 = __float2uint_rn(__saturatef(r) * 255.f), g8 = __float2uint_rn(__saturatef(g) * 255.f);
            const uint32_t b8 = __float2uint_rn(__saturatef(b) * 255.f), a8 = __float2uint_rn(__saturatef(al) * 255.f);
            reinterpret_cast<uint32_t *>(row)[px] = r8 | (g8 << 8) | (b8 << 16) | (a8 << 24);
        }
    }
    if (a.signal_flag) {
        // sharded rendering: the pixels above went to the ROOT GPU's frame (peer memory); the last CTA
        // of this band raises the band flag there once every store is fenced at system scope
        __threadfence_system();
        __syncthreads();
        if (tid == 0) {
            const uint32_t prev = atomicAdd(a.done_counter, 1u);
            if (prev == gridDim.x * gridDim.y - 1u) { __threadfence_system(); st_release_sys(a.signal_flag, *a.signal_epoch); }
        }
    }
}

}  // namespace

cudaError_t launch_composite(const CompositeArgs &a, uint32_t tiles_x, uint32_t tiles_y, cudaStream_t stream, uint32_t views)
{
    dim3 grid(tiles_x, tiles_y, views);
    if (a.mode == 1) {
        composite_kernel<2, 1><<<grid, CB_THREADS, 0, stream>>>(a);          // no pixels are written: the format is irrelevant
    } else if (a.mode == 2) {
        switch (a.format) {
        case 0: composite_kernel<0, 2><<<grid, CB_THREADS, 0, stream>>>(a); break;
        case 1: composite_kernel<1, 2><<<grid, CB_THREADS, 0, stream>>>(a); break;
        default: composite_kernel<2, 2><<<grid, CB_THREADS, 0, stream>>>(a); break;
        }
    } else {
        switch (a.format) {
        case 0: composite_kernel<0, 0><<<grid, CB_THREADS, 0, stream>>>(a); break;
        case 1: composite_kernel<1, 0><<<grid, CB_THREADS, 0, stream>>>(a); break;
        default: composite_kernel<2, 0><<<grid, CB_THREADS, 0, stream>>>(a); break;
        }
    }
    return cudaGetLastError();
}

}  // namespace ws
