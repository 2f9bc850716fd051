// ws_kernels.h -- host-visible launchers of the sm_100a kernels (internal to the library).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace ws {

struct FrameUniforms;
struct FrameCounters;
struct ShardMailbox;

// ---- stage 1 -----------------------------------------------------------------
struct PreprocessArgs {
    const uint8_t *gaussians;     // N x 28 B (raw) / 24 B (compressed), padded to a multiple of 256 records
    const float *xyz;             // N x 3 f32: position plane for the count kernel (derived at upload)
    const uint8_t *sh_coefs;      // raw: N x 96 B; compressed: i8 entries
    const uint8_t *covars;        // compressed only: 12 B per entry
    const FrameUniforms *uniforms;
    uint32_t *splats;             // out: V x 5 u32 (20-B Splat)
    uint32_t *depth_keys;         // out: V
    uint32_t *slot_vals;          // out: V (iota payload)
    uint2 *rects;                 // out: V x {x0 | y0<<16, w | h<<16}
    uint32_t *part_counts;        // ceil(N/256) (batch: num_views x ceil(N/256), view-major): survivors per partition (count kernel)
    uint32_t *part_bases;         // as part_counts: its exclusive scan (scan kernel)
    uint32_t *hist;               // 4 x 256 depth-key digit histograms (zeroed per frame)
    FrameCounters *counters;
    // read by the batch kernels only (batch = true): `uniforms` then points at num_views view-local blocks
    uint32_t num_views;
    uint32_t *part_union;         // ceil(N/256): Gaussians of the partition that survive in at least one view
    uint32_t *view_visible;       // out: num_views per-view survivor counts V_v
};
constexpr uint32_t MAX_VIEWS = 8;  // views per batch (WS_MAX_VIEWS)
// batch: the kernels of a batch of 1..MAX_VIEWS views of one cloud; otherwise a single frame, which reads one uniform block
cudaError_t launch_preprocess(const PreprocessArgs &a, bool compressed, bool batch, int grid_count, int grid_main, cudaStream_t stream);
int preprocess_blocks_per_sm(bool compressed, bool batch);

// ---- onesweep radix sort of (u32 key, u32 value) pairs ---------------------------
constexpr int SORT_THREADS = 256;
constexpr int SORT_ITEMS = 16;
constexpr int SORT_PART = SORT_THREADS * SORT_ITEMS;   // 4096 pairs per partition
constexpr unsigned SORT_LB_GROUP = 16;                 // partitions per look-back group (two-level look-back)

struct SortPassArgs {
    const uint32_t *keys_in, *vals_in;
    uint32_t *keys_out, *vals_out;   // keys_out may be NULL on the last tile pass (see sort_pass_can_skip_keys)
    const uint32_t *n_ptr;        // device: number of pairs (clamped to n_cap)
    uint32_t n_cap;
    uint32_t *status;             // [ceil(n_cap/4096)][256] look-back words, zeroed before the pass
    uint32_t *gstatus;            // [ceil(parts/16)][256] group-level look-back words, zeroed before the pass
    uint32_t *ticket;             // zeroed before the pass
    const uint32_t *hist;         // 256 digit counts of this pass (over the first min(*n_ptr,n_cap) keys)
    uint32_t shift;               // digit = (key >> shift) & 255
    uint32_t *err;                // optional error word (bit 0: look-back watchdog)
    uint2 *ranges;                // last tile-id pass only: per-tile {begin, ~end}, pre-filled with 0xff; else NULL
};
cudaError_t launch_sort_pass(const SortPassArgs &a, int grid, cudaStream_t stream);
int sort_pass_blocks_per_sm();
bool sort_pass_can_skip_keys();   // the default (TMA-staged) pass accepts keys_out == NULL: the last tile pass then drops the key store
// digit histograms of up to 4 passes (shift 0,8,16,24) in one sweep over the keys; hist zeroed by caller
cudaError_t launch_sort_histogram(const uint32_t *keys, const uint32_t *n_ptr, uint32_t n_cap,
                                  uint32_t *hist /*4x256*/, int passes, int grid, cudaStream_t stream);

// ---- tile binning: expand depth-sorted splats into (tile, slot) pairs ----------------
struct BinningArgs {
    const uint32_t *sorted_slots; // V: payload after the depth sort
    const uint2 *rects;           // per slot
    const FrameUniforms *uniforms;
    FrameCounters *counters;      // reads num_visible, writes num_pairs / pair_overflow
    uint32_t *pair_tiles;         // out: P tile ids
    uint32_t *pair_slots;         // out: P slots
    uint32_t *part_counts;        // ceil(N/1024): pairs per partition (count kernel)
    uint32_t *part_bases;         // ceil(N/1024): exclusive scan (scan kernel)
    uint32_t *hist;               // 4 x 256 tile-id digit histograms (zeroed per frame)
    // occlusion split (DESIGN.md section 4): the depth-sorted splats are binned in two slabs, nearest first
    uint32_t slab;                // 0: all of [0, V);  1: the near slab [split, V);  2: the far slab [0, split),  split = (V - near) & ~3, near = V/4 unless near_pct is set
    const uint8_t *tile_done;     // slab 2: tiles already saturated by the near slab; a splat whose whole rectangle is done emits no pair
    uint32_t *keep4;              // slab 2: ceil(V/2/4) words, one byte per splat: count kernel -> expand kernel
    uint32_t pair_cap;            // capacity of pair_tiles / pair_slots for this launch
    uint32_t *num_pairs_out;      // device counter that receives the number of pairs of this launch
    uint32_t near_pct;            // occlusion split: share of the depth-sorted splats in the near slab, in percent (0 = the default quarter)
    uint32_t num_tiles_hint;      // host-known number of tiles (sizes the shared-memory copy of tile_done); 0 = unknown
    uint32_t done_in_smem;        // set by launch_binning
};
cudaError_t launch_binning(const BinningArgs &a, int grid_count, int grid_expand, cudaStream_t stream);
int binning_blocks_per_sm();

// ---- stage 3 -----------------------------------------------------------------------
struct CompositeArgs {
    const uint32_t *splats;       // V x 5 u32
    const uint32_t *pair_slots;   // sorted
    const uint2 *ranges;          // T x {begin, ~end}; untouched tiles hold 0xffffffff in both words
    const FrameUniforms *uniforms;
    void *dst;                    // device frame
    uint32_t row_pitch;           // bytes
    int format;                   // ws_format
    float clear[4];
    uint32_t tile_y0;             // first tile row to composite (sharded rendering: this rank's band); dst row 0 = that row
    uint32_t *signal_flag;        // optional (peer-mapped): set to signal_epoch by the last CTA once every pixel store is fenced
    const uint32_t *signal_epoch;  // device word holding the frame number to signal (the frame replays as a CUDA graph)
    uint32_t *done_counter;       // with signal_flag: zeroed per frame
    // occlusion split: mode 0 = the whole list in one pass; 1 = near slab, per-pixel state {r,g,b,T} + per-tile
    // "saturated" flag out, no pixels; 2 = far slab, state in, final pixels out
    int mode;
    int active_cull;              // per-warp cull against the bounding box of the still-unsaturated pixels (result-neutral)
    float4 *state;                // W x H per view
    uint8_t *tile_done;           // T
    // batches of views: block z composites view z, whose tiles follow the tiles of views 0..z-1 ("tall" frame of
    // z * tiles_y + y rows), whose state starts at z * W * H and whose pixels start at dst + z * view_stride
    uint64_t view_stride;         // bytes
};
cudaError_t launch_composite(const CompositeArgs &a, uint32_t tiles_x, uint32_t tiles_y, cudaStream_t stream, uint32_t views = 1);

// ---- file-format ingest (ingest.cu) ---------------------------------------------------------------------------
struct PlyConvertArgs {
    const uint8_t *vertices;      // the file's vertex block, uploaded as is
    uint32_t n, stride_bytes, sh_deg, big_endian;
    uint8_t *gaussians;           // out: n x 28 B
    uint8_t *sh_coefs;            // out: n x 96 B
    float *xyz;                   // out: n x 3
    double *sums;                 // out: [9] sum x,y,z, xx,xy,xz,yy,yz,zz (zeroed by the caller)
    uint32_t *minmax;             // out: [6] ordered-int min xyz / max xyz (min = 0xffffffff, max = 0 by the caller)
};
cudaError_t launch_ply_convert(const PlyConvertArgs &a, int grid, cudaStream_t stream);

struct C3dgsArgs {                // device copies of the .npz arrays (io/npz.rs:58-160)
    const uint16_t *xyz_f16;      // n x 3 f16
    const int8_t *opacity;        // n
    const int8_t *scaling_factor; // n or NULL
    const int32_t *gaussian_indices, *feature_indices;   // n or NULL (identity)
    const int8_t *scaling;        // num_covars x 3
    const int8_t *rotation;       // num_covars x 4
    const int8_t *features_dc;    // num_features x 3
    const int8_t *features_rest;  // num_features x (3C - 3)
    uint32_t n, num_covars, num_features, sh_deg;
    float scaling_scale, scaling_zero_point, rotation_scale, rotation_zero_point;
    uint8_t *gaussians;           // out: n x 24 B
    int8_t *sh_out;               // out: num_features x 3C
    uint8_t *covars;              // out: num_covars x 12 B
    float *xyz;                   // out: n x 3
    double *sums; uint32_t *minmax;
};
cudaError_t launch_c3dgs_convert(const C3dgsArgs &a, int max_grid, cudaStream_t stream);
// sets *flag != 0 when a 24-B record's geometry_idx >= num_covars or sh_idx >= num_features (flag zeroed by the caller)
cudaError_t launch_validate_compressed(const uint8_t *gaussians, uint32_t n, uint32_t num_covars, uint32_t num_features,
                                       uint32_t *flag, int max_grid, cudaStream_t stream);

// ---- multi-GPU exchange (shard.cu) ---------------------------------------------------------------
struct RouteArgs {
    const uint32_t *l_splats, *l_keys; const uint2 *l_rects;   // stage-1 output of the local shard (slot order)
    const FrameCounters *counters;                             // num_visible = local V
    uint32_t world, rank;
    uint32_t band_y0[9];                                       // rank d owns tile rows [band_y0[d], band_y0[d+1])
    uint32_t *part_band_counts, *part_band_bases;              // [ceil(V/256)][world]
    uint32_t *totals;                                          // out (pass 2): this rank's row of the G x G count matrix
    const uint32_t *matrix;                                    // in (pass 3): the all-gathered matrix [src][dst]
    uint32_t *peer_splats[8], *peer_keys[8]; uint2 *peer_rects[8];   // destination buffers (peer-mapped for other ranks)
    uint32_t recv_cap;
    uint32_t *err;
    // host-collective-free mode: rows, barrier and band signal go through peer-mapped mailboxes
    ShardMailbox *peer_mail[8];                                // NULL: NCCL mode (matrix/totals are plain buffers)
    const uint32_t *epoch_ptr;                                 // device word: frame number, > 0 (advanced by the frame itself)
    uint32_t *done_counter;                                    // zeroed per frame: last-CTA detection
    uint32_t gated;                                            // 1: flag waits run in one-warp gate kernels in front of the consumers
};
cudaError_t launch_shard_finish_peer(const RouteArgs &a, uint32_t *vals, const uint32_t *keys, uint32_t *hist, int passes,
                                     FrameCounters *counters, int grid, cudaStream_t stream);
cudaError_t launch_wait_bands(const ShardMailbox *mail, uint32_t world, const uint32_t *epoch_ptr, uint32_t *err, cudaStream_t stream);
cudaError_t launch_epoch_advance(uint32_t *epoch, cudaStream_t stream);
cudaError_t launch_route_count(const RouteArgs &a, int grid, cudaStream_t stream);
cudaError_t launch_route_scatter(const RouteArgs &a, int grid, cudaStream_t stream);
cudaError_t launch_shard_finish(const uint32_t *matrix, uint32_t world, uint32_t rank, uint32_t recv_cap,
                                FrameCounters *counters, uint32_t *vals, int grid, cudaStream_t stream);

}  // namespace ws
