// preprocess.cu -- stage 1 of the splat render path on sm_100a.
//
// Replaces preprocess.wgsl:163-280 / preprocess_compressed.wgsl:206-331 of the reference
// (one thread per Gaussian: cull, 3D->2D covariance, eigen axes, SH colour, f16 pack,
// depth key) and adds what the tile-binned design needs: the per-splat 16x16-tile
// rectangle and the digit histograms of the depth keys for the onesweep that follows.
//
// B200 design notes
//  * three launches: (1) COUNT reads only a 12-B xyz plane, culls, writes the number of
//    survivors of every 256-Gaussian partition and the digit histograms of their depth keys;
//    (2) a one-CTA SCAN turns the counts into slot offsets; (3) MAIN does the projection.
//    Compaction is therefore deterministic (slot order = Gaussian index order; the reference
//    uses one contended global atomic, preprocess.wgsl:262, whose order is not), and MAIN has
//    no inter-CTA dependency at all -- a single-pass chained scan was tried first (r01a/r01b in
//    profiles/): its look-back serialised the prefetch pipeline.  The price is re-reading xyz:
//    +12 B on top of 124 B per Gaussian;
//  * each kernel is one template over <COMPRESSED, BATCH>.  BATCH = false is a single frame: one uniform block and
//    K = 1 view at compile time.  BATCH = true is a batch of K <= MAX_VIEWS views of one cloud (DESIGN.md section 12):
//    the records and SH are read once and every view is culled, projected and compacted from them, into view-major slots;
//  * MAIN is software-pipelined: partitions are assigned round-robin, the 28-B (24-B) AoS
//    records of partition k+1 and -- when at least half of it survives -- its 24-KB SH block
//    are fetched by cp.async.bulk (TMA engine, UBLKCP) into shared-memory rings while
//    partition k is being computed; 3 CTAs x 31 KB per SM are in flight, HBM sees only full bursts;
//    sparse partitions fetch SH with three 256-bit loads per surviving lane instead
//    (one full 32-B sector per request);
//  * records are read from shared memory at a conflict-free 7-word (6-word: 2-way) stride;
//    outputs are staged through shared memory and leave as coalesced streams;
//  * this file is compiled with -fmad=false, so a fused multiply-add happens exactly where fmaf() is
//    written -- the same places as in oracle/ws_oracle.c -- and quotients with a shared divisor are a
//    correctly rounded reciprocal (__frcp_rn: MUFU.RCP + Newton step) times the numerator, again as
//    in the oracle: stage 1 stays bit-identical to the CPU oracle (raw layout) with ~20 % fewer
//    instructions than the round-1 "one rounding per written operation" form (19 IEEE divisions
//    per Gaussian then, 4 reciprocals now; per-frame constants 1/W, 1/H, znear, zfar come from the host).
#include "ws_device.cuh"
#include "ws_kernels.h"

#include <type_traits>

namespace ws {

namespace {

constexpr int PP_THREADS = 256;
constexpr int PP_WARPS = PP_THREADS / 32;

__device__ __forceinline__ float half_lo(uint32_t w) { __half_raw r; r.x = (unsigned short)(w & 0xffffu); return __half2float(__half(r)); }
__device__ __forceinline__ float half_hi(uint32_t w) { __half_raw r; r.x = (unsigned short)(w >> 16); return __half2float(__half(r)); }
__device__ __forceinline__ uint32_t pack2h(float a, float b)
{
    __half_raw ra = __float2half_rn(a), rb = __float2half_rn(b);
    return (uint32_t)ra.x | ((uint32_t)rb.x << 16);
}

struct V3 { float x, y, z; };
__device__ __forceinline__ V3 v3s(float s, V3 a) { return V3{s * a.x, s * a.y, s * a.z}; }
__device__ __forceinline__ V3 v3add(V3 a, V3 b) { return V3{a.x + b.x, a.y + b.y, a.z + b.z}; }
__device__ __forceinline__ V3 v3sub(V3 a, V3 b) { return V3{a.x - b.x, a.y - b.y, a.z - b.z}; }
__device__ __forceinline__ V3 v3fma(float s, V3 a, V3 acc) { return V3{fmaf(s, a.x, acc.x), fmaf(s, a.y, acc.y), fmaf(s, a.z, acc.z)}; }

// SH basis constants, preprocess.wgsl:4-23
#define WS_SH_C0 0.28209479177387814f
#define WS_SH_C1 0.4886025119029199f
#define WS_SH_C2_0 1.0925484305920792f
#define WS_SH_C2_1 (-1.0925484305920792f)
#define WS_SH_C2_2 0.31539156525252005f
#define WS_SH_C2_3 (-1.0925484305920792f)
#define WS_SH_C2_4 0.5462742152960396f
#define WS_SH_C3_0 (-0.5900435899266435f)
#define WS_SH_C3_1 2.890611442640554f
#define WS_SH_C3_2 (-0.4570457994644658f)
#define WS_SH_C3_3 0.3731763325901154f
#define WS_SH_C3_4 (-0.4570457994644658f)
#define WS_SH_C3_5 1.445305721320277f
#define WS_SH_C3_6 (-0.5900435899266435f)

// Coefficient fetchers: k-th RGB triple as f32 (preprocess.wgsl:114-121 / compressed :147-171)
struct ShRaw {
    uint32_t w[24];                 // [[f16;3];16]: half index = k*3 + ch
    __device__ __forceinline__ float h(int i) const { return (i & 1) ? half_hi(w[i >> 1]) : half_lo(w[i >> 1]); }
    __device__ __forceinline__ V3 coef(int k) const { return V3{h(k * 3), h(k * 3 + 1), h(k * 3 + 2)}; }
};
struct ShQuant {
    uint32_t w[12];                 // the entry's (file_deg+1)^2*3 i8 bytes, dc first (io/npz.rs:183-196), zero padded
    const float *lut;               // shared memory: [0..255] dc, [256..511] rest -- dequantised value of every i8 code
    // One table entry = sh_coef() of preprocess_compressed.wgsl:147-171 for that byte: unpack4x8snorm * 127, then
    // dequantizef4 -- the oracle's arithmetic, evaluated 512 times per CTA instead of 48 times per Gaussian (each with
    // an IEEE division by 127: 430 of the ~2300 instructions per Gaussian in round 1).
    static __device__ __forceinline__ float dq(int8_t b, const Quant &q)
    {
        float sn = (float)b / 127.f;            // unpack4x8snorm: max(i/127, -1)
        if (sn < -1.f) sn = -1.f;
        float v = sn * 127.f;
        return (v - (float)q.zero_point) * q.scale;   // dequantizef4
    }
    __device__ __forceinline__ uint32_t byte(int i) const { return (w[i >> 2] >> ((i & 3) * 8)) & 0xffu; }
    __device__ __forceinline__ V3 coef(int k) const
    {
        const float *t = lut + ((k == 0) ? 0 : 256);
        return V3{t[byte(k * 3)], t[byte(k * 3 + 1)], t[byte(k * 3 + 2)]};
    }
    // entry base = sh_idx * ncoef * 3 bytes; degree-3 entries (48 B) are 16-B aligned: three 128-bit loads
    __device__ __forceinline__ void load(const uint8_t *base, uint32_t sh_idx, uint32_t ncoef)
    {
        const uint8_t *p = base + (size_t)sh_idx * ncoef * 3u;
        if (ncoef == 16u) {
            const uint4 *q4 = reinterpret_cast<const uint4 *>(p);
            const uint4 a = __ldg(q4), b = __ldg(q4 + 1), c = __ldg(q4 + 2);
            w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
            w[8] = c.x; w[9] = c.y; w[10] = c.z; w[11] = c.w;
        } else {
#pragma unroll
            for (int i = 0; i < 12; i++) w[i] = 0u;
            const uint32_t nb = ncoef * 3u;                    // 3, 12 or 27 bytes
#pragma unroll
            for (int i = 0; i < 27; i++)                       // static indices keep w[] in registers
                if ((uint32_t)i < nb) w[i >> 2] |= (uint32_t)__ldg(p + i) << ((i & 3) * 8);
        }
    }
};

// evaluate_sh, preprocess.wgsl:124-154: same operation order as oracle/ws_oracle.c
template <class SH>
__device__ __forceinline__ V3 evaluate_sh(float x, float y, float z, const SH &sh, uint32_t deg)
{
    V3 result = v3s(WS_SH_C0, sh.coef(0));
    if (deg > 0u) {
        V3 t = v3s((-WS_SH_C1) * y, sh.coef(1));
        t = v3fma(WS_SH_C1 * z, sh.coef(2), t);
        t = v3fma(-(WS_SH_C1 * x), sh.coef(3), t);
        result = v3add(result, t);
        if (deg > 1u) {
            float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
            V3 u = v3s(WS_SH_C2_0 * xy, sh.coef(4));
            u = v3fma(WS_SH_C2_1 * yz, sh.coef(5), u);
            u = v3fma(WS_SH_C2_2 * (2.0f * zz - xx - yy), sh.coef(6), u);
            u = v3fma(WS_SH_C2_3 * xz, sh.coef(7), u);
            u = v3fma(WS_SH_C2_4 * (xx - yy), sh.coef(8), u);
            result = v3add(result, u);
            if (deg > 2u) {
                V3 w = v3s(WS_SH_C3_0 * y * (3.0f * xx - yy), sh.coef(9));
                w = v3fma(WS_SH_C3_1 * xy * z, sh.coef(10), w);
                w = v3fma(WS_SH_C3_2 * y * (4.0f * zz - xx - yy), sh.coef(11), w);
                w = v3fma(WS_SH_C3_3 * z * (2.0f * zz - 3.0f * xx - 3.0f * yy), sh.coef(12), w);
                w = v3fma(WS_SH_C3_4 * x * (4.0f * zz - xx - yy), sh.coef(13), w);
                w = v3fma(WS_SH_C3_5 * z * (xx - yy), sh.coef(14), w);
                w = v3fma(WS_SH_C3_6 * x * (xx - 3.0f * yy), sh.coef(15), w);
                result = v3add(result, w);
            }
        }
    }
    result.x = result.x + 0.5f; result.y = result.y + 0.5f; result.z = result.z + 0.5f;
    return result;
}

__device__ __forceinline__ void ldg256(const void *p, uint32_t *r)
{
    asm volatile("ld.global.nc.L1::no_allocate.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "l"(p));
}

struct Stage1 {
    uint32_t splat[5];      // v_0, v_1, pos, color_0, color_1 (pointcloud.rs:352-358)
    uint32_t key;
    uint32_t rect_xy;       // x0 | y0 << 16
    uint32_t rect_wh;       // w  | h  << 16  (w == 0: touches no tile)
};

// sort key: preprocess.wgsl:270-273 (f32 bits of zfar - clip.z) / compressed :321-325 (24-bit integer)
template <bool COMPRESSED>
__device__ __forceinline__ uint32_t depth_key(const FrameUniforms &U, float p2)
{
    // znear = -proj[3][2] / proj[2][2], zfar = -proj[3][2] / (proj[2][2] - 1): per-frame constants, divided once on the host
    const float znear = U.znear, zfar = U.zfar;
    if (!COMPRESSED) return __float_as_uint(zfar - p2);
    const float kf = 16777215.f - (p2 - znear) / (zfar - znear) * 16777215.f;
    if (!(kf > 0.f)) return 0u;
    if (kf >= 4294967296.f) return 0xffffffffu;
    return (uint32_t)kf;
}

// Everything after the cull: preprocess.wgsl:194-279 / compressed :235-330.
template <bool COMPRESSED, class SH>
__device__ __forceinline__ void project_tail(const FrameUniforms &U, float x, float y, float z,
                                             float cs0, float cs1, float cs2,
                                             float p0, float p1, float p2, float p3,
                                             const float cov6[6], float opacity, const SH &sh, Stage1 &o)
{
    const float *view = U.cam.view;
    const float fx = U.cam.focal[0], fy = U.cam.focal[1];

    // scale_mod (:196-201)
    float scale_mod = 0.f;
    {
        float ddx = U.rs.center[0] - x, ddy = U.rs.center[1] - y, ddz = U.rs.center[2] - z;
        float dist = sqrtf(fmaf(ddz, ddz, fmaf(ddy, ddy, ddx * ddx)));
        float dd = 5.f * dist * U.inv_scene_extend;
        if (U.rs.walltime > dd) {
            float t = U.rs.walltime - dd;
            t = t < 0.f ? 0.f : (t > 1.f ? 1.f : t);
            scale_mod = t * t * (3.f - 2.f * t);
        }
    }
    const float scaling = U.rs.gaussian_scaling * scale_mod;
    const float c0 = cov6[0] * scaling * scaling, c1 = cov6[1] * scaling * scaling, c2 = cov6[2] * scaling * scaling;
    const float c3 = cov6[3] * scaling * scaling, c4 = cov6[4] * scaling * scaling, c5 = cov6[5] * scaling * scaling;
    const float Vm[3][3] = {{c0, c1, c2}, {c1, c3, c4}, {c2, c4, c5}};

    const float rz = __frcp_rn(cs2), rz2 = rz * rz;
    const float j00 = fx * rz;
    const float j20 = -(fx * cs0) * rz2;
    const float j11 = -(fy * rz);
    const float j21 = (fy * cs1) * rz2;

    float T0[3], T1[3];
#pragma unroll
    for (int i = 0; i < 3; i++) {
        float w0 = view[i * 4 + 0], w1 = view[i * 4 + 1], w2 = view[i * 4 + 2];
        T0[i] = fmaf(w2, j20, w0 * j00);
        T1[i] = fmaf(w2, j21, w1 * j11);
    }
    float A0[3], A1[3];
#pragma unroll
    for (int j = 0; j < 3; j++) {
        float a = T0[0] * Vm[0][j]; a = fmaf(T0[1], Vm[1][j], a); a = fmaf(T0[2], Vm[2][j], a); A0[j] = a;
        float b = T1[0] * Vm[0][j]; b = fmaf(T1[1], Vm[1][j], b); b = fmaf(T1[2], Vm[2][j], b); A1[j] = b;
    }
    float cov00 = A0[0] * T0[0]; cov00 = fmaf(A0[1], T0[1], cov00); cov00 = fmaf(A0[2], T0[2], cov00);
    float cov01 = A1[0] * T0[0]; cov01 = fmaf(A1[1], T0[1], cov01); cov01 = fmaf(A1[2], T0[2], cov01);
    float cov11 = A1[0] * T1[0]; cov11 = fmaf(A1[1], T1[1], cov11); cov11 = fmaf(A1[2], T1[2], cov11);

    const float ks = U.rs.kernel_size;
    if (U.rs.mip_splatting) {                      // :226-236
        float det_0 = cov00 * cov11 - cov01 * cov01;
        det_0 = (det_0 > 1e-6f) ? det_0 : 1e-6f;
        float det_1 = (cov00 + ks) * (cov11 + ks) - cov01 * cov01;
        det_1 = (det_1 > 1e-6f) ? det_1 : 1e-6f;
        float coef = sqrtf(det_0 / (det_1 + 1e-6f) + 1e-6f);
        if (det_0 <= 1e-6f || det_1 <= 1e-6f) coef = 0.0f;
        opacity = opacity * coef;
    }

    const float diagonal1 = cov00 + ks, offDiagonal = cov01, diagonal2 = cov11 + ks;
    const float mid = 0.5f * (diagonal1 + diagonal2);
    const float hx = (diagonal1 - diagonal2) / 2.0f;
    const float radius = sqrtf(fmaf(offDiagonal, offDiagonal, hx * hx));
    float lambda1, lambda2;
    if (!COMPRESSED) {
        lambda1 = mid + radius;
        float l2 = mid - radius;
        lambda2 = (l2 > 0.1f) ? l2 : 0.1f;
    } else {
        float rr = (radius > 0.1f) ? radius : 0.1f;
        lambda1 = mid + rr;
        lambda2 = mid - rr;
    }
    float dvx = offDiagonal, dvy = lambda1 - diagonal1;
    const float rdl = __frcp_rn(sqrtf(fmaf(dvy, dvy, dvx * dvx)));
    dvx = dvx * rdl; dvy = dvy * rdl;
    const float s1 = sqrtf(2.0f * lambda1), s2 = sqrtf(2.0f * lambda2);
    const float v1x = s1 * dvx, v1y = s1 * dvy, v2x = s2 * dvy, v2y = s2 * (-dvx);
    const float rw = __frcp_rn(p3);
    const float vcx = p0 * rw, vcy = p1 * rw;

    const float dx = x - U.cam.view_inv[12], dy = y - U.cam.view_inv[13], dz = z - U.cam.view_inv[14];
    const float rlen = __frcp_rn(sqrtf(fmaf(dz, dz, fmaf(dy, dy, dx * dx))));
    V3 col = evaluate_sh(dx * rlen, dy * rlen, dz * rlen, sh, U.rs.max_sh_deg);
    col.x = (col.x > 0.f) ? col.x : 0.f;
    col.y = (col.y > 0.f) ? col.y : 0.f;
    col.z = (col.z > 0.f) ? col.z : 0.f;

    const float ivw = U.inv_viewport[0], ivh = U.inv_viewport[1];       // 1 / viewport, divided once on the host
    o.splat[0] = pack2h(v1x * ivw, v1y * ivh);
    o.splat[1] = pack2h(v2x * ivw, v2y * ivh);
    o.splat[2] = pack2h(vcx, vcy);
    o.splat[3] = pack2h(col.x, col.y);
    o.splat[4] = pack2h(col.z, opacity);

    o.key = depth_key<COMPRESSED>(U, p2);

    // ---- tile rectangle of the STORED (f16-rounded) splat; must equal oracle wso_tile_rects ----
    {
        const float hv1x = half_lo(o.splat[0]), hv1y = half_hi(o.splat[0]);
        const float hv2x = half_lo(o.splat[1]), hv2y = half_hi(o.splat[1]);
        const float hcx = half_lo(o.splat[2]), hcy = half_hi(o.splat[2]);
        const float fw = (float)U.width, fh = (float)U.height;
        const float ex = FOOTPRINT_R * (fw * sqrtf(hv1x * hv1x + hv2x * hv2x));
        const float ey = FOOTPRINT_R * (fh * sqrtf(hv1y * hv1y + hv2y * hv2y));
        const float pcx = (hcx + 1.f) * 0.5f * fw;
        const float pcy = (1.f - hcy) * 0.5f * fh;
        const float fx0 = floorf((pcx - ex - 0.5f - RECT_PAD) * 0.0625f), fx1 = floorf((pcx + ex - 0.5f + RECT_PAD) * 0.0625f);
        const float fy0 = floorf((pcy - ey - 0.5f - RECT_PAD) * 0.0625f), fy1 = floorf((pcy + ey - 0.5f + RECT_PAD) * 0.0625f);
        o.rect_xy = 0u; o.rect_wh = 0u;
        if (fx0 == fx0 && fx1 == fx1 && fy0 == fy0 && fy1 == fy1) {
            const float mx = (float)(U.tiles_x - 1u), my = (float)(U.tiles_y - 1u);
            const float lx = fx0 < 0.f ? 0.f : fx0, ly = fy0 < 0.f ? 0.f : fy0;
            const float hx1 = fx1 > mx ? mx : fx1, hy1 = fy1 > my ? my : fy1;
            if (!(hx1 < lx || hy1 < ly)) {
                uint32_t x0 = (uint32_t)lx, y0 = (uint32_t)ly, x1 = (uint32_t)hx1, y1 = (uint32_t)hy1;
                o.rect_xy = x0 | (y0 << 16);
                o.rect_wh = (x1 - x0 + 1u) | ((y1 - y0 + 1u) << 16);
            }
        }
    }
}

// Cull + clip-space projection of one record: preprocess.wgsl:177-192 / compressed :223-233.
template <bool COMPRESSED>
__device__ __forceinline__ bool cull_project(const FrameUniforms &U, float x, float y, float z, float cs[4], float pp[4])
{
    // clip box (:177) -- any(xyz < min) || any(xyz > max)
    if (x < U.rs.clip_min[0] || y < U.rs.clip_min[1] || z < U.rs.clip_min[2] ||
        x > U.rs.clip_max[0] || y > U.rs.clip_max[1] || z > U.rs.clip_max[2]) return false;
    const float *view = U.cam.view, *proj = U.cam.proj;
#pragma unroll
    for (int r = 0; r < 4; r++) {
        float acc = view[0 * 4 + r] * x;
        acc = fmaf(view[1 * 4 + r], y, acc);
        acc = fmaf(view[2 * 4 + r], z, acc);
        acc = fmaf(view[3 * 4 + r], 1.f, acc);
        cs[r] = acc;
    }
#pragma unroll
    for (int r = 0; r < 4; r++) {
        float acc = proj[0 * 4 + r] * cs[0];
        acc = fmaf(proj[1 * 4 + r], cs[1], acc);
        acc = fmaf(proj[2 * 4 + r], cs[2], acc);
        acc = fmaf(proj[3 * 4 + r], cs[3], acc);
        pp[r] = acc;
    }
    const float bounds = 1.2f * pp[3];
    const float zz = pp[2] * __frcp_rn(pp[3]);
    if (!COMPRESSED) {
        if (zz <= 0.f || zz >= 1.f || pp[0] < -bounds || pp[0] > bounds || pp[1] < -bounds || pp[1] > bounds) return false;
    } else {
        if (zz < 0.f || zz > 1.f || pp[0] < -bounds || pp[0] > bounds || pp[1] < -bounds || pp[1] > bounds) return false;
    }
    return true;
}

// ---- (1) COUNT: survivors per partition + depth-key digit histograms -----------------------
// BATCH: the K = a.num_views views are culled one after the other against the same positions; part_counts holds
// K x nparts survivor counts (view-major) and part_union the Gaussians of each partition that survive in any view.
template <bool COMPRESSED, bool BATCH>
__global__ void __launch_bounds__(PP_THREADS)
count_kernel(PreprocessArgs a)
{
    __shared__ FrameUniforms s_u[BATCH ? MAX_VIEWS : 1u];
    __shared__ uint32_t s_hist[4 * 256];
    const unsigned tid = threadIdx.x;
    const uint32_t K = BATCH ? a.num_views : 1u;
    {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(a.uniforms);
        uint32_t *dst = reinterpret_cast<uint32_t *>(s_u);
        for (unsigned i = tid; i < K * (uint32_t)(sizeof(FrameUniforms) / 4u); i += PP_THREADS) dst[i] = src[i];
    }
    for (unsigned i = tid; i < 4u * 256u; i += PP_THREADS) s_hist[i] = 0u;
    __syncthreads();
    const uint32_t n = s_u[0].num_points;
    const uint32_t nparts = (n + PP_THREADS - 1u) / PP_THREADS;
    constexpr int NDIG = 4;
    // CNT_UNROLL consecutive partitions per trip: their 3 * CNT_UNROLL loads are issued before the first use, and the
    // block-wide counts (one barrier each) follow back to back -- a single partition per trip left the loads exposed
    // behind every barrier (r01m: long_scoreboard 35 %, 1.9 TB/s)
    constexpr uint32_t CNT_UNROLL = 4;
    for (uint32_t part0 = blockIdx.x * CNT_UNROLL; part0 < nparts; part0 += gridDim.x * CNT_UNROLL) {
        float px[CNT_UNROLL], py[CNT_UNROLL], pz[CNT_UNROLL];
#pragma unroll
        for (uint32_t u = 0; u < CNT_UNROLL; u++) {
            uint32_t idx = (part0 + u) * PP_THREADS + tid;
            idx = idx < n ? idx : n - 1u;                                  // clamped: the loads stay unconditional (n > 0 here)
            const float *p = a.xyz + (size_t)idx * 3u;
            px[u] = __ldg(p); py[u] = __ldg(p + 1); pz[u] = __ldg(p + 2);
        }
        bool any[CNT_UNROLL];                                              // BATCH: survives in at least one view
#pragma unroll
        for (uint32_t u = 0; u < CNT_UNROLL; u++) any[u] = false;
        for (uint32_t v = 0; v < K; v++) {
            const FrameUniforms &U = s_u[v];
            bool keep[CNT_UNROLL];
            uint32_t key[CNT_UNROLL];
#pragma unroll
            for (uint32_t u = 0; u < CNT_UNROLL; u++) {
                float cs[4], pp[4];
                const bool valid = (part0 + u) * PP_THREADS + tid < n;
                keep[u] = cull_project<COMPRESSED>(U, px[u], py[u], pz[u], cs, pp) && valid;
                key[u] = depth_key<COMPRESSED>(U, pp[2]);
                if (BATCH) any[u] = any[u] || keep[u];      // unguarded, it costs the single-view kernel 8 registers
            }
#pragma unroll
            for (uint32_t u = 0; u < CNT_UNROLL; u++) {
                const uint32_t cnt = (uint32_t)__syncthreads_count(keep[u] ? 1 : 0);
                if (tid == 0 && part0 + u < nparts) a.part_counts[v * nparts + part0 + u] = cnt;
            }
            // shared atomics without return sustain ~120 G warp-ops/s on B200 whatever the spread
            // (profiles/microbench/rank_primitives.cu); MATCH-aggregating them was 25x slower
#pragma unroll
            for (uint32_t u = 0; u < CNT_UNROLL; u++) {
                if (keep[u]) {
#pragma unroll
                    for (int d = 0; d < NDIG; d++) atomicAdd(&s_hist[d * 256 + ((key[u] >> (8 * d)) & 255u)], 1u);
                }
            }
        }
        if (BATCH) {
#pragma unroll
            for (uint32_t u = 0; u < CNT_UNROLL; u++) {
                const uint32_t cnt = (uint32_t)__syncthreads_count(any[u] ? 1 : 0);
                if (tid == 0 && part0 + u < nparts) a.part_union[part0 + u] = cnt;
            }
        }
    }
    __syncthreads();
    for (unsigned i = tid; i < (unsigned)NDIG * 256u; i += PP_THREADS) {
        const uint32_t c = s_hist[i];
        if (c) atomicAdd(a.hist + i, c);
    }
}

// ---- (2) SCAN: exclusive scan of the partition counts (one CTA) ------------------------------
// BATCH: one scan over the K x nparts counts gives view-major slot bases, plus the per-view totals V_v
template <bool BATCH>
__global__ void __launch_bounds__(1024)
scan_kernel(PreprocessArgs a)
{
    const uint32_t K = BATCH ? a.num_views : 1u;
    const uint32_t nparts = (a.uniforms->num_points + PP_THREADS - 1u) / PP_THREADS;
    // a single frame has <= N < 2^32 survivors, a batch K * N < 2^30: a 32-bit scan
    const uint32_t total = block_exclusive_scan_1024<uint32_t>(a.part_counts, a.part_bases, K * nparts);
    // the scan ends with a barrier: every base written above is visible to the whole block
    if (BATCH && threadIdx.x < K) {
        const uint32_t v = threadIdx.x;
        const uint32_t b0 = nparts ? a.part_bases[v * nparts] : 0u;
        const uint32_t b1 = (nparts && v + 1u < K) ? a.part_bases[(v + 1u) * nparts] : total;
        a.view_visible[v] = b1 - b0;
    }
    if (threadIdx.x == 0) a.counters->num_visible = total;
}

// ---- (3) MAIN ---------------------------------------------------------------------------------
constexpr int PP_STAGES = 2;                         // ring depth: records and SH of partition k+1 in flight while k is computed
constexpr uint32_t PP_SH_BYTES = PP_THREADS * 96u;   // one partition's SH block
constexpr uint32_t PP_SH_BULK_MIN = 128;             // bulk-stage the SH block when >= half the partition survives

// NU uniform blocks: 1 for a single view, MAX_VIEWS for a batch of views
template <bool COMPRESSED, uint32_t NU = 1>
struct PPSmem {
    static constexpr uint32_t REC = COMPRESSED ? 24u : 28u;
    static constexpr uint32_t REC_BYTES = PP_THREADS * REC;
    static constexpr uint32_t off_rec = 0;
    static constexpr uint32_t off_sh = off_rec + PP_STAGES * REC_BYTES;                        // 128-B aligned (7168, 6144)
    static constexpr uint32_t off_splat = off_sh + (COMPRESSED ? 0u : PP_STAGES * PP_SH_BYTES);
    static constexpr uint32_t off_key = off_splat + PP_THREADS * 20u;
    static constexpr uint32_t off_rect = off_key + PP_THREADS * 4u;
    static constexpr uint32_t off_u = off_rect + PP_THREADS * 8u;
    static constexpr uint32_t off_bar = (off_u + NU * (uint32_t)sizeof(FrameUniforms) + 15u) & ~15u;
    static constexpr uint32_t off_misc = off_bar + 8u * (2 * PP_STAGES);
    static constexpr uint32_t off_lut = off_misc + 64u;                                        // compressed: 2 x 256 dequantised SH codes
    static constexpr uint32_t bytes = off_lut + (COMPRESSED ? 2u * 256u * 4u : 0u);
};
template <bool COMPRESSED, bool BATCH>
using PPLayout = PPSmem<COMPRESSED, BATCH ? MAX_VIEWS : 1u>;

// BATCH: each partition's records and SH are staged once and every view culls, projects and compacts from them in
// turn, with the same cull_project / project_tail as a single frame (this file is built with -fmad=false), so each
// view's halves, keys and rectangles are bit for bit those of the same view rendered alone.  View v's survivors take
// the slots [B_v, B_v + V_v) in Gaussian-index order, and its rectangles are moved down to its rows of the "tall" frame.
template <bool COMPRESSED, bool BATCH>
__global__ void __launch_bounds__(PP_THREADS, 3)
preprocess_kernel(PreprocessArgs a)
{
    using L = PPLayout<COMPRESSED, BATCH>;
    constexpr uint32_t REC = L::REC, REC_WORDS = REC / 4u;
    extern __shared__ __align__(128) uint8_t smem[];
    uint32_t *s_splat = reinterpret_cast<uint32_t *>(smem + L::off_splat);
    uint32_t *s_key = reinterpret_cast<uint32_t *>(smem + L::off_key);
    uint2 *s_rect = reinterpret_cast<uint2 *>(smem + L::off_rect);
    const FrameUniforms *s_u = reinterpret_cast<const FrameUniforms *>(smem + L::off_u);
    uint64_t *s_rbar = reinterpret_cast<uint64_t *>(smem + L::off_bar);
    uint64_t *s_sbar = s_rbar + PP_STAGES;
    uint32_t *s_warp_cnt = reinterpret_cast<uint32_t *>(smem + L::off_misc);      // [8]

    const unsigned tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint32_t K = BATCH ? a.num_views : 1u;
    {   // uniforms -> smem
        const uint32_t *src = reinterpret_cast<const uint32_t *>(a.uniforms);
        uint32_t *dst = reinterpret_cast<uint32_t *>(smem + L::off_u);
        for (unsigned i = tid; i < K * (uint32_t)(sizeof(FrameUniforms) / 4u); i += PP_THREADS) dst[i] = src[i];
    }
    if (tid == 0) {
        for (int i = 0; i < 2 * PP_STAGES; i++) mbar_init(&s_rbar[i], 1);
        fence_mbar_init();
    }
    float *s_lut = reinterpret_cast<float *>(smem + L::off_lut);
    if (COMPRESSED) {
        // s_u is not visible yet: read the two quantisers from global (they belong to the cloud: the same in every view)
        const FrameUniforms *gu = a.uniforms;
        const Quant qd = gu->quant.color_dc, qr = gu->quant.color_rest;
        s_lut[tid] = ShQuant::dq((int8_t)tid, qd);               // index = the byte's bit pattern
        s_lut[256 + tid] = ShQuant::dq((int8_t)tid, qr);
    }
    __syncthreads();
    const uint32_t n = s_u[0].num_points;
    const uint32_t nparts = (n + PP_THREADS - 1u) / PP_THREADS;
    uint32_t max_deg = s_u[0].rs.max_sh_deg;                     // SH is fetched once, for the highest degree of the batch
    for (uint32_t v = 1; v < K; v++) max_deg = s_u[v].rs.max_sh_deg > max_deg ? s_u[v].rs.max_sh_deg : max_deg;
    const bool sh_bulk_ok = !COMPRESSED && max_deg >= 2u;
    const uint32_t *survivors = BATCH ? a.part_union : a.part_counts;     // a batch: survivors in at least one view

    // iteration k of this CTA handles partition blockIdx.x + k * gridDim.x
    auto part_of = [&](uint32_t k) -> uint32_t { return blockIdx.x + k * gridDim.x; };
    auto uses_bulk_sh = [&](uint32_t part) -> bool { return sh_bulk_ok && __ldg(survivors + part) >= PP_SH_BULK_MIN; };
    auto issue = [&](uint32_t k) {                    // thread 0 only: fetch everything partition k needs
        const uint32_t part = part_of(k);
        if (part >= nparts) return;
        const uint32_t s = k % PP_STAGES;
        fence_proxy_async();                          // earlier generic-proxy reads of the slot happen-before the async write
        mbar_arrive_expect_tx(&s_rbar[s], L::REC_BYTES);
        bulk_g2s(smem + L::off_rec + s * L::REC_BYTES, a.gaussians + (size_t)part * L::REC_BYTES, L::REC_BYTES, &s_rbar[s]);
        if (uses_bulk_sh(part)) {
            mbar_arrive_expect_tx(&s_sbar[s], PP_SH_BYTES);
            bulk_g2s(smem + L::off_sh + s * PP_SH_BYTES, a.sh_coefs + (size_t)part * PP_SH_BYTES, PP_SH_BYTES, &s_sbar[s]);
        }
    };

    if (tid == 0) issue(0);
    uint32_t rpar = 0, spar = 0;                      // per-slot mbarrier phase parities (block-uniform)

    for (uint32_t k = 0;; k++) {
        const uint32_t part = part_of(k);
        if (part >= nparts) break;
        const uint32_t s = k % PP_STAGES;
        if (tid == 0) issue(k + 1u);                  // slot (k+1)%2 was last read in iteration k-1 (trailing barrier)

        const bool bulk = uses_bulk_sh(part);
        mbar_wait(&s_rbar[s], (rpar >> s) & 1u); rpar ^= 1u << s;
        if (bulk) { mbar_wait(&s_sbar[s], (spar >> s) & 1u); spar ^= 1u << s; }

        const uint32_t *rec = reinterpret_cast<const uint32_t *>(smem + L::off_rec + s * L::REC_BYTES) + tid * REC_WORDS;
        const uint32_t idx = part * PP_THREADS + tid;
        const float x = __uint_as_float(rec[0]), y = __uint_as_float(rec[1]), z = __uint_as_float(rec[2]);
        // view-independent inputs, loaded at the first view that keeps the Gaussian
        bool loaded = false;
        float opacity = 0.f, cov6[6];
        typename std::conditional<COMPRESSED, ShQuant, ShRaw>::type sh;

        for (uint32_t v = 0; v < K; v++) {
            const FrameUniforms &U = s_u[v];
            bool vis = false;
            Stage1 o;
            o.key = 0u; o.rect_xy = 0u; o.rect_wh = 0u;
            o.splat[0] = o.splat[1] = o.splat[2] = o.splat[3] = o.splat[4] = 0u;
            float cs[4], pp[4];
            if (idx < n && cull_project<COMPRESSED>(U, x, y, z, cs, pp)) {
                vis = true;
                if (!loaded) {
                    loaded = true;
                    if constexpr (!COMPRESSED) {
                        opacity = half_lo(rec[3]);
                        cov6[0] = half_lo(rec[4]); cov6[1] = half_hi(rec[4]); cov6[2] = half_lo(rec[5]);
                        cov6[3] = half_hi(rec[5]); cov6[4] = half_lo(rec[6]); cov6[5] = half_hi(rec[6]);
                        // words beyond a view's degree are never read by evaluate_sh: one fetch serves every view
                        if (bulk) {
                            const uint4 *sp = reinterpret_cast<const uint4 *>(smem + L::off_sh + s * PP_SH_BYTES + tid * 96u);
#pragma unroll
                            for (int q = 0; q < 6; q++) {
                                const uint4 w = sp[q];
                                sh.w[4 * q] = w.x; sh.w[4 * q + 1] = w.y; sh.w[4 * q + 2] = w.z; sh.w[4 * q + 3] = w.w;
                            }
                        } else {
                            const uint8_t *sp = a.sh_coefs + (size_t)idx * 96u;
                            ldg256(sp, sh.w);
                            if (max_deg > 1u) ldg256(sp + 32, sh.w + 8); else {
#pragma unroll
                                for (int i = 8; i < 16; i++) sh.w[i] = 0u;
                            }
                            if (max_deg > 2u) ldg256(sp + 64, sh.w + 16); else {
#pragma unroll
                                for (int i = 16; i < 24; i++) sh.w[i] = 0u;
                            }
                        }
                    } else {
                        const uint32_t os = rec[3];
                        const int8_t q_op = (int8_t)(os & 0xffu), q_sf = (int8_t)((os >> 8) & 0xffu);
                        const uint32_t geo_idx = rec[4], sh_idx = rec[5];
                        opacity = ((float)q_op - (float)U.quant.opacity.zero_point) * U.quant.opacity.scale;
                        const float sfac = expf(((float)q_sf - (float)U.quant.scaling_factor.zero_point) * U.quant.scaling_factor.scale);
                        const float s2 = sfac * sfac;
                        const uint32_t *cw = reinterpret_cast<const uint32_t *>(a.covars + (size_t)geo_idx * 12u);
                        const uint32_t w0 = __ldg(cw), w1 = __ldg(cw + 1), w2 = __ldg(cw + 2);
                        cov6[0] = half_lo(w0) * s2; cov6[1] = half_hi(w0) * s2; cov6[2] = half_lo(w1) * s2;
                        cov6[3] = half_hi(w1) * s2; cov6[4] = half_lo(w2) * s2; cov6[5] = half_hi(w2) * s2;
                        const uint32_t ncoef = (U.file_sh_deg + 1u) * (U.file_sh_deg + 1u);
                        sh.load(a.sh_coefs, sh_idx, ncoef);
                        sh.lut = s_lut;
                    }
                }
                project_tail<COMPRESSED>(U, x, y, z, cs[0], cs[1], cs[2], pp[0], pp[1], pp[2], pp[3], cov6, opacity, sh, o);
                if (BATCH && o.rect_wh) o.rect_xy += (v * U.tiles_y) << 16;      // view v's tile rows in the "tall" frame
            }

            // ---- deterministic compaction: slot = scanned (view, partition) base + rank inside the partition
            const unsigned bal = __ballot_sync(0xffffffffu, vis);
            if (lane == 0) s_warp_cnt[warp] = __popc(bal);
            __syncthreads();
            uint32_t warp_off = 0, total = 0;
#pragma unroll
            for (int w = 0; w < PP_WARPS; w++) {
                uint32_t c = s_warp_cnt[w];
                if (w < (int)warp) warp_off += c;
                total += c;
            }
            const uint32_t local = warp_off + __popc(bal & lanemask_lt());
            if (vis) {
#pragma unroll
                for (int q = 0; q < 5; q++) s_splat[local * 5u + q] = o.splat[q];
                s_key[local] = o.key;
                s_rect[local] = make_uint2(o.rect_xy, o.rect_wh);
            }
            __syncthreads();
            const uint32_t base = __ldg(a.part_bases + v * nparts + part);
            // ---- coalesced output streams ----
            for (uint32_t i = tid; i < total * 5u; i += PP_THREADS) a.splats[(size_t)base * 5u + i] = s_splat[i];
            if (tid < total) {
                a.depth_keys[base + tid] = s_key[tid];
                a.slot_vals[base + tid] = base + tid;           // payload = slot, preprocess.wgsl:274
                a.rects[base + tid] = s_rect[tid];
            }
            __syncthreads();
        }
    }
}

}  // namespace

// The opt-in above 48 KB of dynamic shared memory is a per-device attribute: the C ABI allows several ws_context on
// different devices in one process, so it is tracked per device (and per layout).
template <bool C, bool B>
static cudaError_t pp_prepare()
{
    static bool done[64] = {};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < 64 && done[dev]) return cudaSuccess;
    e = cudaFuncSetAttribute(preprocess_kernel<C, B>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PPLayout<C, B>::bytes);
    if (e == cudaSuccess && dev >= 0 && dev < 64) done[dev] = true;
    return e;
}

template <bool C, bool B>
static cudaError_t pp_launch(const PreprocessArgs &a, int grid_count, int grid_main, cudaStream_t stream)
{
    cudaError_t e = pp_prepare<C, B>();
    if (e != cudaSuccess) return e;
    count_kernel<C, B><<<grid_count, PP_THREADS, 0, stream>>>(a);
    scan_kernel<B><<<1, 1024, 0, stream>>>(a);
    preprocess_kernel<C, B><<<grid_main, PP_THREADS, PPLayout<C, B>::bytes, stream>>>(a);
    return cudaGetLastError();
}

template <bool C, bool B>
static int pp_blocks_per_sm()
{
    int nb = 0;
    if (pp_prepare<C, B>() != cudaSuccess) return 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, preprocess_kernel<C, B>, PP_THREADS, PPLayout<C, B>::bytes);
    return nb > 0 ? nb : 1;
}

cudaError_t launch_preprocess(const PreprocessArgs &a, bool compressed, bool batch, int grid_count, int grid_main, cudaStream_t stream)
{
    if (batch && (a.num_views < 1 || a.num_views > MAX_VIEWS)) return cudaErrorInvalidValue;
    if (compressed) return batch ? pp_launch<true, true>(a, grid_count, grid_main, stream) : pp_launch<true, false>(a, grid_count, grid_main, stream);
    return batch ? pp_launch<false, true>(a, grid_count, grid_main, stream) : pp_launch<false, false>(a, grid_count, grid_main, stream);
}

int preprocess_blocks_per_sm(bool compressed, bool batch)
{
    if (compressed) return batch ? pp_blocks_per_sm<true, true>() : pp_blocks_per_sm<true, false>();
    return batch ? pp_blocks_per_sm<false, true>() : pp_blocks_per_sm<false, false>();
}

}  // namespace ws
