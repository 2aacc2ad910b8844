// datum_b200 — launch interface of the prefilter kernels (internal to libdatum_ibl_cuda).
#pragma once

#include "ibl_math.cuh"

#include <cuda_runtime.h>
#include <cstdint>

namespace ibl
{
#ifdef DATUM_IBL_AB_VARIANTS
  // the round-1 first kernel (tools/ab/prefilter.cu): only in the tools build, for A/B timing
  struct PrefilterParams
  {
    uint4 const *records;    // quad records of the SOURCE level (6*ws*hs)
    float4 const *table;     // sample table of this level: (lx, ly, lz, 0.5*lz), decreasing lz
    int table_count;
    uint32_t *dst_words;     // destination level base, rgbe words (may be null)
    float *dst_f32;          // destination level base, fp32 rgb triples before quantisation (may be null)
    int wd, hd;              // destination level size
    int row_begin, row_end;  // slab of the 6*hd face-major rows to compute
    LevelGeom geom;          // source level addressing constants
    Quatf quats[6];          // face rotations, tools/ibl.cpp:253-261
    DecodeMasks masks;       // bit masks of accumulate_tap, passed as parameters so they live in registers
    float norm;              // kAccScale / total weight
    int tiles_x, tiles;      // filled by the launcher
  };
#endif

  // ---- denormal-mantissa kernel (prefilter_dn.cu): every level at least 8 texels wide ----

  constexpr int kMaxPeers = 7;      // one probe split over at most 8 GPUs (one NVSwitch domain)

  // Arrival counters of the GPUs that share a probe: the CTA of a launch that finishes last bumps
  // arrive[k] (a word in peer k's flag block, mapped here) once every store of the launch is out.
  struct PeerSignal
  {
    unsigned int *arrive[kMaxPeers];
    int count;               // 0: nobody to tell
    unsigned int *ticket;    // "CTAs done" counter of this context, zero between launches
  };
  constexpr int kSampleBand = 16;   // entries per band of the banded sample table (ibl_tables.h)
  constexpr int kSectorShare = 4;   // entries per sector and band of the pair kernel's sector tables: bands of 16 (4 sectors) or 32 (8)

  struct PrefilterDnParams
  {
    uint4 const *records;     // quad records of the SOURCE level, words re-laid by pack_dn_word (6*ws*hs)
    float4 const *table;      // banded sample table of this level, every entry scaled by kDnTableScale
    float4 const *table_pairs; // the same entries, last band filled up, two entries interleaved per 32 bytes (ibl_tables.h)
    // the pair kernel's tables, one azimuth sector per warp (ibl_tables.h, build_sector_entries): [0] for 4 warps
    // per tile, [1] for 8.  Projective entries (lx/lz, ly/lz, lz, wh), pair-interleaved; sector_rho[i][w*bands + k] =
    // largest |(lx/lz, ly/lz)| of warp w's share of band k.  Used unless the source level is odd-sized or above
    // 2^22 texels per face (proj_usable): then the one-sample kernel runs.
    float4 const *table_sector[2];
    float const *sector_rho[2];
    int sector_bands[2];
    float const *band_min_lz; // smallest lz of each band (unscaled), decreasing
    int table_count;
    int bands;                // ceil(table_count / kSampleBand)
    uint32_t *dst_words;      // destination level base, rgbe words (may be null)
    float *dst_f32;           // destination level base, fp32 rgb triples before quantisation (may be null)
    uint32_t *peer_words[kMaxPeers]; // the same destination level in the chains of other GPUs (NVLink peer stores)
    int peers;                // how many of them: the epilogue writes every word to dst_words and to each peer
    PeerSignal signal;        // whom to tell when the whole slab is stored
    int wd, hd;               // destination level size
    int row_begin, row_end;   // slab of the 6*hd face-major rows to compute
    LevelGeom geom;           // source level addressing constants
    Quatf quats[6];           // face rotations, tools/ibl.cpp:253-261
    float norm[3];            // per channel: sum -> radiance / total weight (dn_channel_norms)
    uint32_t exp_mul;         // 2^23 (a parameter on purpose, see scale_by_exponent)
    uint32_t red_mul;         // 2^9 (A/B: r mantissa as the high half of word * 2^9)
    int *counters;            // queues+1 tile queue heads, zeroed by launch_build_dn_records
    int blocks_x, tiles;      // filled by the launcher: 4x4-blocked tile numbering
    int queues, chunk, queued;

    // the same level of `probes` chains in one launch (datum_ibl_bake_probes): records of the probes back
    // to back (record_stride each), destination levels dst_stride words apart
    int probes, tiles_per_probe;
    size_t record_stride, dst_stride;

    int no_steal;             // A/B: a group whose chunk and pool are empty leaves instead of helping other SMs

    // frames of the DESTINATION level for the pair kernel (launch_build_frames): nine planes of 6*hd*wd floats
    // — the face-local folded rows T, B, N of every texel (fold_face_row) — followed by the same-face limits
    // of the eight azimuth sectors (sector_rho_limits) per TILE of 8x4 texels: kFrameSectors planes of
    // frame_tile_rows(hd) * frame_tiles_x(wd) floats, each the minimum over the tile's texels.  They depend
    // on the level's geometry alone, so the library keeps them per source size.
    float const *frames;
  };

  inline int frame_tiles_x(int wd) { return (wd + 7) / 8; }
  inline int frame_tile_rows(int hd) { return (6 * hd + 3) / 4; }
  inline size_t frame_floats(int wd, int hd) { return (size_t)9 * 6 * hd * wd + (size_t)kFrameSectors * frame_tile_rows(hd) * frame_tiles_x(wd); }

  constexpr int kWorldFrameFloats = 9;

  // world-space T, B, N of every texel of the wd x hd destination level (what the tail kernel's CTAs need)
  cudaError_t launch_build_world_frames(float *frames, int wd, int hd, Quatf const quats[6], cudaStream_t stream);

  // frames of every texel of the wd x hd destination of a ws x hs source level (proj_usable sizes)
  cudaError_t launch_build_frames(float *frames, int ws, int hs, Quatf const quats[6], cudaStream_t stream);

  // ---- tail levels (prefilter_dn.cu, prefilter_tail_kernel): a few hundred texels ----
  //
  // One CTA per output texel, LANES are samples: the 1024 samples of a texel are one to four steps
  // deep instead of 32, the four footprint words come straight from the source level (no record pass).
  struct PrefilterTailParams
  {
    uint32_t const *src;      // SOURCE level words (6*ws*hs), tools/ibl.cpp layout
    float4 const *table;      // banded sample table of this level scaled by kDnTableScale (any order works)
    float4 const *table_proj; // the same entries as (lx/lz, ly/lz, lz, wh): read instead when proj_usable(ws, hs)
    float const *world_frames; // kWorldFrameFloats planes of 6*hd*wd floats: T, B, N of every destination texel (launch_build_world_frames), or null: computed per CTA
    int table_count;
    uint32_t *dst_words;
    float *dst_f32;
    uint32_t *peer_words[kMaxPeers];
    int peers;
    PeerSignal signal;
    int wd, hd;
    int row_begin, row_end;
    LevelGeom geom;
    Quatf quats[6];
    float norm[3];
    uint32_t exp_mul;
    int probes, texels_per_probe;     // the same level of several chains in one launch
    size_t src_stride, dst_stride;    // words between the probes' source / destination levels
  };

  // slabs up to this many texels go to the tail kernel
  constexpr int kTailTexels = 6144;

  // warps per texel of the tail kernels: enough CTAs to cover the machine first, then depth; never more lanes than samples
  inline int tail_warps(int texels, int table_count)
  {
    if (texels >= 4096 || table_count <= 128)
      return 4;
    if (texels >= 1024 || table_count <= 256)
      return 8;
    if (texels >= 256 || table_count <= 512)
      return 16;
    return 32;
  }

  // Slab-size classes of the pair kernels: slabs of at least kQueuedTexels texels take their tiles from
  // per-SM queues, and of at least kFourWarpTexels run 4 warps per tile instead of 8.  A sample table of more
  // than kBigTableEntries entries (4096-sample bakes) would cost too much shared memory per CTA: it is read
  // through L1.
  constexpr size_t kQueuedTexels = 32u * 148u * 8u;
  constexpr size_t kFourWarpTexels = 160000u;
  constexpr int kBigTableEntries = 1100;

  // Resident CTAs per SM of one kernel for one dynamic shared-memory size (opt-in above 48 KB), remembered
  // per (kernel, device, size) and host thread.
  cudaError_t resident_ctas(void const *kernel, int threads, size_t smem, int *resident);

  // The launch shape of a tiled kernel over a slab (P: PrefilterDnParams or PrefilterFloatParams): 8x4 tiles
  // numbered in 4x4 blocks (tile_texel), the slabs of `probes` probes one after the other; at most one CTA
  // per resident slot; 7/8 of the tiles in per-SM chunks of the tile queues, the rest in the common pool that
  // evens out the end of the launch.
  template<typename P>
  cudaError_t plan_tiles(P &p, void (*kernel)(P), int threads, size_t smem, int probes, int sm_count, int *grid)
  {
    int resident = 0;
    cudaError_t err = resident_ctas((void const*)kernel, threads, smem, &resident);
    if (err != cudaSuccess)
      return err;

    const int tiles_x = (p.wd + 7) / 8, tiles_y = (p.row_end - p.row_begin + 3) / 4;
    p.blocks_x = (tiles_x + 3) / 4;
    p.tiles = p.blocks_x * ((tiles_y + 3) / 4) * 16 * probes;

    *grid = p.tiles < sm_count * resident ? p.tiles : sm_count * resident;
    if (*grid < 1)
      *grid = 1;

    p.queues = sm_count;
    p.chunk = (p.tiles - p.tiles / 8) / sm_count;
    p.queued = p.chunk * sm_count;
    return cudaSuccess;
  }

  cudaError_t launch_prefilter_tail(PrefilterTailParams const &p, int sm_count, cudaStream_t stream);

  // variant 0 = pick by slab size and table size; 50..58 = one sample at a time, fixed <warps per tile,
  // table in shared memory, tile queues>; 70..75 = two samples at a time (prefilter_dp_kernel)
  cudaError_t launch_prefilter_dn(PrefilterDnParams const &p, int variant, int sm_count, cudaStream_t stream, int *launched_grid);

  // the arrival signal alone, for the barrier at the start of a shared bake (one tiny launch)
  cudaError_t launch_peer_signal(PeerSignal const &s, cudaStream_t stream);

  // also zeroes the `ncounters` tile queue heads for the prefilter launch that follows
  cudaError_t launch_build_dn_records(uint32_t const *src, uint4 *rec, int ws, int hs, int probes, size_t src_stride, int *counters, int ncounters, int sm_count, cudaStream_t stream);

  // can the same level of several probes go into one launch (pair kernel usable for a ws x hs source)?
  bool prefilter_batchable(int ws, int hs);

#ifdef DATUM_IBL_AB_VARIANTS
  // variant 0 = pick by slab size; 1..15 = fixed <tile width, texels per lane, warps per tile>
  cudaError_t launch_prefilter_level(PrefilterParams const &p, int variant, int sm_count, cudaStream_t stream, int *launched_grid);

  cudaError_t launch_build_quad_records(uint32_t const *src, uint4 *records, int ws, int hs, int sm_count, cudaStream_t stream);
#endif
}
