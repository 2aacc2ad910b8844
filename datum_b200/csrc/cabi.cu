// datum_b200 — C ABI of libdatum_ibl_cuda (see include/datum_ibl_cuda.h).
//
// Owns the device context: stream, cached per-level sample tables, grow-only
// device scratch (payload chain, quad records, SH9 weight table and partials).
// No CPU fallback exists anywhere in this library: every entry point either runs
// the CUDA kernels or fails with an error string.

#include "../../include/datum_ibl_cuda.h"

#include "ibl_math.cuh"
#include "ibl_tables.h"
#include "prefilter.h"
#include "prefilter_f.h"
#include "sh9.h"
#include "luts.h"
#include "resample.h"

#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "cabi_internal.h"

namespace
{
  thread_local std::string g_last_error;
}

namespace ibl_cabi
{
  int fail(std::string const &what)
  {
    g_last_error = what;
    return 1;
  }

  int fail_cuda(const char *where, cudaError_t err)
  {
    g_last_error = std::string(where) + ": " + cudaGetErrorString(err);
    return 1;
  }
}

namespace
{
  using ibl_cabi::fail;
  using ibl_cabi::fail_cuda;

  struct DeviceTable
  {
    float4 *d_entries = nullptr;
    int count = 0;
    int samples = 0; // the reference's kSamples this table was built for (accepted + rejected)
    float norm = 0;  // kAccScale / total weight
    double total_weight = 0;
    float4 *d_banded = nullptr;  // the entries in banded ring order (ibl_tables.h), scaled by kDnTableScale
    float4 *d_pairs = nullptr;   // the banded entries, last band filled up, interleaved two by two (build_paired_entries)
    float4 *d_sector[2] = { nullptr, nullptr };   // the pair kernel's tables, one azimuth sector per warp, for 4 and 8 warps per tile (ibl_tables.h)
    float *d_sector_rho[2] = { nullptr, nullptr };
    int sector_bands[2] = { 0, 0 };
    float4 *d_banded_proj = nullptr; // d_banded with (lx/lz, ly/lz) in place of (lx, ly): the tail kernel's
    float *d_band_min = nullptr; // smallest lz per band
    int bands = 0;
  };

  template<typename T>
  struct DeviceBuffer
  {
    T *ptr = nullptr;
    size_t capacity = 0;

    cudaError_t reserve(size_t count)
    {
      if (count <= capacity)
        return cudaSuccess;

      if (ptr)
        cudaFree(ptr);

      ptr = nullptr;
      capacity = 0;

      cudaError_t err = cudaMalloc(&ptr, count * sizeof(T));
      if (err == cudaSuccess)
        capacity = count;

      return err;
    }

    void release()
    {
      if (ptr)
        cudaFree(ptr);
      ptr = nullptr;
      capacity = 0;
    }
  };
}

struct datum_ibl_ctx
{
  int device = 0;
  int sm_count = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev_begin = nullptr, ev_end = nullptr;
  bool timed = false;

  uint64_t launches = 0;
  int prefilter_variant = 0;

  ibl::Quatf quats[6];

  std::map<std::pair<int, int>, std::vector<DeviceTable>> tables; // (levels, samples) -> per level

  DeviceBuffer<uint32_t> chain;   // staged payload for the host entry point
  DeviceBuffer<uint32_t> chain2;  // second payload of datum_ibl_bake_probes (double buffering)
  DeviceBuffer<double> batch_sh;  // 28 doubles per probe of a batch
  cudaStream_t copy_in = nullptr, copy_out = nullptr;   // created on first use by datum_ibl_bake_probes
  cudaEvent_t ev_uploaded[2] = { nullptr, nullptr }, ev_computed[2] = { nullptr, nullptr }, ev_downloaded[2] = { nullptr, nullptr };
  cudaEvent_t ev_level[16] = {};  // level L of the current chain is complete (its download starts behind it)
  cudaEvent_t ev_copied[16] = {}; // level L has arrived in host memory (pageable callers: in the pinned staging)
  void *host_stage = nullptr;     // pinned staging between the device and a caller's PAGEABLE payload
  size_t host_stage_bytes = 0;
  DeviceBuffer<uint4> records;    // quad records of the current source level
  DeviceBuffer<unsigned char> float_records; // footprint records of the current source level of a float chain (prefilter_f.h)
  std::map<std::pair<int, int>, float*> frames; // source size -> per-texel frames of the destination level (ibl::launch_build_frames)
  size_t frames_bytes = 0, world_frames_bytes = 0;
  std::map<std::pair<int, int>, float*> world_frames; // destination size -> world-space T, B, N per texel (tail kernel; levels of at most kWorldFrameTexels)
  DeviceBuffer<int> queue_heads;  // per-SM tile queue heads of the prefilter kernel
  int prefilter_no_steal = 0;
  int sh9_kernel = 0, sh9_rows_per_item = 0;   // A/B: 0 = column strips / automatic run length
  int table_order = 0;            // A/B: 0 = bands are rings of the lobe, 1 = compact patches
  DeviceBuffer<unsigned int> peer_ticket; // "CTAs done" counter of launches that signal peers, zero between launches
  bool peer_wait_pending = false; // a stream wait on a peer's arrival is queued: synchronize() watches the clock
  unsigned int *peer_wait_word = nullptr; // the local arrival counters ([2]) those waits look at
  int peer_timeout_ms = 60000;
  DeviceBuffer<float> sh_weights; // solid angle table
  int sh_weights_w = 0, sh_weights_h = 0;
  DeviceBuffer<double> sh_partials; // block partials + 28 result doubles
  DeviceBuffer<unsigned int> sh_counter; // "blocks done" ticket of the projection kernel, zero between launches
  DeviceBuffer<unsigned char> staging; // generic device staging for host entry points
  DeviceBuffer<float> sink;
  DeviceBuffer<float> srgb_lut;   // pow(c/255, 2.2) for the 256 channel values (six-image ingest)

  // CUDA-event ring around the dominant kernel of every chain (the level-1
  // prefilter launch): bench.py's live per-launch duration for the roofline
  static const int kRing = 512;
  std::vector<cudaEvent_t> ring_begin, ring_end;
  int ring_used = 0;            // launches recorded since the last reset (may exceed kRing)
  double ring_texel_samples = 0; // texel-samples of one recorded launch
};

namespace
{
  struct DeviceGuard
  {
    int previous = -1;
    explicit DeviceGuard(int device)
    {
      cudaGetDevice(&previous);
      if (previous != device)
        cudaSetDevice(device);
    }
    ~DeviceGuard()
    {
      if (previous >= 0)
        cudaSetDevice(previous);
    }
  };

  bool valid_chain(int width, int height, int levels)
  {
    if (width < 1 || height < 1 || levels < 1 || levels > 16)
      return false;

    // every level of the chain must have at least one texel, and a level that is
    // convolved needs a source of at least 2x2 (the bilinear footprint of ibl.cpp:40)
    if ((width >> (levels - 1)) < 1 || (height >> (levels - 1)) < 1)
      return false;

    return true;
  }

  void free_table(DeviceTable &t)
  {
    if (t.d_entries) cudaFree(t.d_entries);
    if (t.d_banded) cudaFree(t.d_banded);
    if (t.d_band_min) cudaFree(t.d_band_min);
    if (t.d_pairs) cudaFree(t.d_pairs);
    for(int i = 0; i < 2; ++i)
    {
      if (t.d_sector[i]) cudaFree(t.d_sector[i]);
      if (t.d_sector_rho[i]) cudaFree(t.d_sector_rho[i]);
    }
    if (t.d_banded_proj) cudaFree(t.d_banded_proj);
    t = DeviceTable();
  }

  int get_tables(datum_ibl_ctx *ctx, int levels, int samples, std::vector<DeviceTable> **out)
  {
    auto key = std::make_pair(levels, samples);
    auto it = ctx->tables.find(key);
    if (it == ctx->tables.end())
    {
      std::vector<DeviceTable> built(levels);

      for(int level = 1; level < levels; ++level)
      {
        ibl::LevelSamples host = ibl::build_level_samples(level, levels, samples);

        DeviceTable &t = built[level];
        t.count = host.accepted;
        t.samples = samples;
        t.norm = (float)((double)ibl::kAccScale / host.total_weight);
        t.total_weight = host.total_weight;

        cudaError_t err = cudaMalloc(&t.d_entries, sizeof(float4) * (size_t)(t.count > 0 ? t.count : 1));
        if (err != cudaSuccess)
        {
          for(auto &b : built)
            free_table(b);
          return fail_cuda("cudaMalloc(sample table)", err);
        }

        static_assert(sizeof(ibl::SampleEntry) == sizeof(float4), "table entry layout");

        err = cudaMemcpyAsync(t.d_entries, host.entries.data(), sizeof(float4) * (size_t)t.count, cudaMemcpyHostToDevice, ctx->stream);
        ibl::BandedSamples banded = ibl::build_banded_samples(level, levels, samples, ibl::kSampleBand, ctx->table_order);
        t.bands = (int)banded.band_min_lz.size();

        std::vector<float> paired = ibl::build_paired_entries(banded, ibl::kDnTableScale);
        ibl::SectorTable sector[2] = { ibl::build_sector_entries(host, 4, 4 * ibl::kSectorShare, ibl::kDnTableScale), ibl::build_sector_entries(host, 8, 8 * ibl::kSectorShare, ibl::kDnTableScale) };

        std::vector<ibl::SampleEntry> banded_proj = banded.level.entries;
        for(auto &e : banded_proj)
        {
          e.lx = (float)((double)e.lx / (double)e.lz); e.ly = (float)((double)e.ly / (double)e.lz);
          e.lz *= ibl::kDnTableScale; e.wh *= ibl::kDnTableScale;
        }

        for(auto &e : banded.level.entries)
        {
          e.lx *= ibl::kDnTableScale; e.ly *= ibl::kDnTableScale; e.lz *= ibl::kDnTableScale; e.wh *= ibl::kDnTableScale;
        }

        if (err == cudaSuccess)
          err = cudaMalloc(&t.d_banded, sizeof(float4) * (size_t)(t.count > 0 ? t.count : 1));
        if (err == cudaSuccess)
          err = cudaMalloc(&t.d_band_min, sizeof(float) * (size_t)(t.bands > 0 ? t.bands : 1));
        if (err == cudaSuccess)
          err = cudaMemcpyAsync(t.d_banded, banded.level.entries.data(), sizeof(float4) * (size_t)t.count, cudaMemcpyHostToDevice, ctx->stream);
        if (err == cudaSuccess)
          err = cudaMemcpyAsync(t.d_band_min, banded.band_min_lz.data(), sizeof(float) * (size_t)t.bands, cudaMemcpyHostToDevice, ctx->stream);
        if (err == cudaSuccess)
          err = cudaMalloc(&t.d_pairs, sizeof(float) * (paired.size() > 0 ? paired.size() : 4));
        if (err == cudaSuccess)
          err = cudaMemcpyAsync(t.d_pairs, paired.data(), sizeof(float) * paired.size(), cudaMemcpyHostToDevice, ctx->stream);
        if (err == cudaSuccess)
          err = cudaMalloc(&t.d_banded_proj, sizeof(float4) * (size_t)(t.count > 0 ? t.count : 1));
        if (err == cudaSuccess)
          err = cudaMemcpyAsync(t.d_banded_proj, banded_proj.data(), sizeof(float4) * (size_t)t.count, cudaMemcpyHostToDevice, ctx->stream);
        for(int i = 0; i < 2; ++i)
        {
          t.sector_bands[i] = sector[i].bands;
          if (err == cudaSuccess)
            err = cudaMalloc(&t.d_sector[i], sizeof(float) * sector[i].entries.size());
          if (err == cudaSuccess)
            err = cudaMemcpyAsync(t.d_sector[i], sector[i].entries.data(), sizeof(float) * sector[i].entries.size(), cudaMemcpyHostToDevice, ctx->stream);
          if (err == cudaSuccess)
            err = cudaMalloc(&t.d_sector_rho[i], sizeof(float) * sector[i].rho_max.size());
          if (err == cudaSuccess)
            err = cudaMemcpyAsync(t.d_sector_rho[i], sector[i].rho_max.data(), sizeof(float) * sector[i].rho_max.size(), cudaMemcpyHostToDevice, ctx->stream);
        }

        if (err == cudaSuccess)
          err = cudaStreamSynchronize(ctx->stream); // `host` and `banded` die at the end of this iteration
        if (err != cudaSuccess)
        {
          for(auto &b : built)
            free_table(b);
          return fail_cuda("upload(sample table)", err);
        }
      }

      it = ctx->tables.emplace(key, std::move(built)).first;
    }

    *out = &it->second;
    return 0;
  }

  int begin_dominant(datum_ibl_ctx *ctx, double texel_samples)
  {
    if (ctx->ring_begin.empty())
    {
      ctx->ring_begin.resize(datum_ibl_ctx::kRing);
      ctx->ring_end.resize(datum_ibl_ctx::kRing);
      for(int i = 0; i < datum_ibl_ctx::kRing; ++i)
      {
        cudaEventCreate(&ctx->ring_begin[i]);
        cudaEventCreate(&ctx->ring_end[i]);
      }
    }
    int slot = ctx->ring_used % datum_ibl_ctx::kRing;
    ctx->ring_used += 1;
    ctx->ring_texel_samples = texel_samples;
    cudaEventRecord(ctx->ring_begin[slot], ctx->stream);
    return slot;
  }

  // the GPUs sharing a probe: where this slab's words also go, and whom to tell when all are stored
  struct PeerTargets
  {
    int count = 0;
    uint32_t *words[ibl::kMaxPeers] = {};
    unsigned int *arrive[ibl::kMaxPeers] = {};   // null: no signal from the kernel
  };

  // the same level of several chains in one launch (datum_ibl_bake_probes, datum_ibl_bake_probes_float): chains
  // `stride` texels apart (rgbe words, or texels of a float chain's format)
  struct Batch
  {
    int probes = 1;
    size_t stride = 0;
  };

  int fill_signal(datum_ibl_ctx *ctx, PeerTargets const &peers, ibl::PeerSignal &signal)
  {
    signal = ibl::PeerSignal();
    if (peers.count == 0 || !peers.arrive[0])
      return 0;

    if (!ctx->peer_ticket.ptr)
    {
      cudaError_t err = ctx->peer_ticket.reserve(1);
      if (err == cudaSuccess)
        err = cudaMemsetAsync(ctx->peer_ticket.ptr, 0, sizeof(unsigned int), ctx->stream);
      if (err != cudaSuccess)
        return fail_cuda("cudaMalloc(peer ticket)", err);
    }

    signal.count = peers.count;
    for(int k = 0; k < peers.count; ++k)
      signal.arrive[k] = peers.arrive[k];
    signal.ticket = ctx->peer_ticket.ptr;
    return 0;
  }

  // folded frames and sector limits of the destination level of a ws x hs source (proj_usable sizes), kept
  // per source size: geometry only
  int level_frames(datum_ibl_ctx *ctx, int ws, int hs, float const **out)
  {
    int wd = ws >> 1, hd = hs >> 1;

    auto found = ctx->frames.find(std::make_pair(ws, hs));
    if (found == ctx->frames.end())
    {
      // a process that bakes many different sizes must not collect planes for ever: start over above 1 GiB
      const size_t bytes = sizeof(float) * ibl::frame_floats(wd, hd);
      if (ctx->frames_bytes + bytes > ((size_t)1 << 30) && !ctx->frames.empty())
      {
        cudaStreamSynchronize(ctx->stream);
        for(auto &entry : ctx->frames)
          cudaFree(entry.second);
        ctx->frames.clear();
        ctx->frames_bytes = 0;
      }

      float *built = nullptr;
      cudaError_t err = cudaMalloc(&built, bytes);
      if (err == cudaSuccess)
      {
        err = ibl::launch_build_frames(built, ws, hs, ctx->quats, ctx->stream);
        if (err != cudaSuccess)
          cudaFree(built);
      }
      if (err != cudaSuccess)
        return fail_cuda("build_frames", err);
      ctx->launches += 1;
      ctx->frames_bytes += bytes;
      found = ctx->frames.emplace(std::make_pair(ws, hs), built).first;
    }

    *out = found->second;
    return 0;
  }

  // world-space frames of a wd x hd destination level (tail kernels), kept per size; null for levels above
  // kWorldFrameTexels (the tail kernel then computes a frame per CTA)
  int level_world_frames(datum_ibl_ctx *ctx, int wd, int hd, float const **out)
  {
    *out = nullptr;
    const size_t kWorldFrameTexels = (size_t)1 << 20;
    if ((size_t)6 * wd * hd > kWorldFrameTexels)
      return 0;

    auto found = ctx->world_frames.find(std::make_pair(wd, hd));
    if (found == ctx->world_frames.end())
    {
      // the same bound as for the pair kernel's planes: start over above 256 MiB
      const size_t bytes = sizeof(float) * (size_t)ibl::kWorldFrameFloats * 6 * wd * hd;
      if (ctx->world_frames_bytes + bytes > ((size_t)1 << 28) && !ctx->world_frames.empty())
      {
        cudaStreamSynchronize(ctx->stream);
        for(auto &entry : ctx->world_frames)
          cudaFree(entry.second);
        ctx->world_frames.clear();
        ctx->world_frames_bytes = 0;
      }

      float *built = nullptr;
      cudaError_t err = cudaMalloc(&built, bytes);
      if (err == cudaSuccess)
      {
        err = ibl::launch_build_world_frames(built, wd, hd, ctx->quats, ctx->stream);
        if (err != cudaSuccess)
          cudaFree(built);
      }
      if (err != cudaSuccess)
        return fail_cuda("build_world_frames", err);
      ctx->launches += 1;
      ctx->world_frames_bytes += bytes;
      found = ctx->world_frames.emplace(std::make_pair(wd, hd), built).first;
    }

    *out = found->second;
    return 0;
  }

  // the checks of a slab of destination rows of a ws x hs source level, both chains: 1 after fail(), else 0
  int check_slab(int ws, int hs, int row_begin, int row_end)
  {
    if (ws < 2 || hs < 2)
      return fail("prefilter: source level must be at least 2x2");
    if (row_begin < 0 || row_end > 6 * (hs >> 1) || row_begin > row_end)
      return fail("prefilter: row range outside the destination level");
    return 0;
  }

  // the pair kernels' sector tables (PrefilterDnParams, PrefilterFloatParams)
  template<typename P>
  void set_sector_tables(P &p, DeviceTable const &table)
  {
    for(int i = 0; i < 2; ++i)
    {
      p.table_sector[i] = table.d_sector[i];
      p.sector_rho[i] = table.d_sector_rho[i];
      p.sector_bands[i] = table.sector_bands[i];
    }
  }

  // slabs of more than kTailTexels texels of a level at least a tile wide: denormal-mantissa kernels (prefilter_dn.cu)
  int run_level_dn(datum_ibl_ctx *ctx, uint32_t const *d_src, int ws, int hs, DeviceTable const &table, int row_begin, int row_end, uint32_t *d_dst_words, float *d_dst_f32, bool record_dominant, PeerTargets const &peers, Batch const &batch)
  {
    int wd = ws >> 1, hd = hs >> 1;

    cudaError_t err = ctx->records.reserve((size_t)6 * ws * hs * batch.probes);
    if (err == cudaSuccess)
      err = ctx->queue_heads.reserve((size_t)ctx->sm_count + 1);
    if (err != cudaSuccess)
      return fail_cuda("cudaMalloc(quad records)", err);

    err = ibl::launch_build_dn_records(d_src, ctx->records.ptr, ws, hs, batch.probes, batch.stride, ctx->queue_heads.ptr, ctx->sm_count + 1, ctx->sm_count, ctx->stream);
    if (err != cudaSuccess)
      return fail_cuda("build_dn_records", err);
    ctx->launches += 1;

    // frames of the destination level: geometry only, computed on first use of a source size
    float const *frames = nullptr;
    if (ibl::proj_usable(ws, hs) && level_frames(ctx, ws, hs, &frames))
      return 1;

    ibl::PrefilterDnParams p = {};
    p.frames = frames;
    p.probes = batch.probes;
    p.record_stride = (size_t)6 * ws * hs;
    p.dst_stride = batch.stride;
    p.no_steal = ctx->prefilter_no_steal;
    p.records = ctx->records.ptr;
    p.table = table.d_banded;
    p.table_pairs = table.d_pairs;
    set_sector_tables(p, table);
    p.band_min_lz = table.d_band_min;
    p.table_count = table.count;
    p.bands = table.bands;
    p.dst_words = d_dst_words;
    p.dst_f32 = d_dst_f32;
    p.peers = peers.count;
    for(int k = 0; k < peers.count; ++k)
      p.peer_words[k] = peers.words[k];
    if (fill_signal(ctx, peers, p.signal))
      return 1;
    p.wd = wd;
    p.hd = hd;
    p.row_begin = row_begin;
    p.row_end = row_end;
    p.geom = ibl::make_level_geom(ws, hs);
    for(int f = 0; f < 6; ++f)
      p.quats[f] = ctx->quats[f];
    ibl::dn_channel_norms(table.total_weight, p.norm);
    p.exp_mul = 0x00800000u;
    p.red_mul = 512u;
    p.counters = ctx->queue_heads.ptr;

    int slot = record_dominant ? begin_dominant(ctx, (double)(row_end - row_begin) * wd * (double)table.samples * batch.probes) : -1;

    int grid = 0;
    err = ibl::launch_prefilter_dn(p, ctx->prefilter_variant >= 50 ? ctx->prefilter_variant : 0, ctx->sm_count, ctx->stream, &grid);
    if (err != cudaSuccess)
      return fail_cuda(("prefilter_dn (source " + std::to_string(ws) + "x" + std::to_string(hs) + ", rows " + std::to_string(row_begin) + ".." + std::to_string(row_end) + ", " + std::to_string(batch.probes) + " probe(s), table " + std::to_string(table.count) + ", grid " + std::to_string(grid) + ")").c_str(), err);
    ctx->launches += 1;

    if (slot >= 0)
      cudaEventRecord(ctx->ring_end[slot], ctx->stream);

    return 0;
  }

  // one level on the context's stream: records of the source level, then the prefilter slab
  int run_level(datum_ibl_ctx *ctx, uint32_t const *d_src, int ws, int hs, DeviceTable const &table, int row_begin, int row_end, uint32_t *d_dst_words, float *d_dst_f32, bool record_dominant = false, PeerTargets const &peers = PeerTargets(), Batch const &batch = Batch())
  {
    int wd = ws >> 1, hd = hs >> 1;

    if (check_slab(ws, hs, row_begin, row_end))
      return 1;
    if (row_begin == row_end)
      return 0;

    // Small slabs (a few hundred to a few thousand texels) and levels narrower than the 8x4 tiles of
    // the big kernels: lanes are samples, no record pass.  Variant 80 pins this kernel for every level.
    bool tail = (size_t)(row_end - row_begin) * wd <= (size_t)ibl::kTailTexels || wd < 8;

    if ((ctx->prefilter_variant == 0 && tail) || ctx->prefilter_variant == 80 || (ctx->prefilter_variant >= 50 && wd < 8))
    {
      // world-space frames of the destination level: geometry only, kept per size (small levels only:
      // this kernel runs slabs of at most kTailTexels texels, a bigger level is a shared probe's)
      float const *world_frames = nullptr;
      if (level_world_frames(ctx, wd, hd, &world_frames))
        return 1;

      ibl::PrefilterTailParams p = {};
      p.src = d_src;
      p.world_frames = world_frames;
      p.table_proj = table.d_banded_proj;
      p.table = table.d_banded;
      p.table_count = table.count;
      p.dst_words = d_dst_words;
      p.dst_f32 = d_dst_f32;
      p.peers = peers.count;
      for(int k = 0; k < peers.count; ++k)
        p.peer_words[k] = peers.words[k];
      if (fill_signal(ctx, peers, p.signal))
        return 1;
      p.wd = wd;
      p.hd = hd;
      p.row_begin = row_begin;
      p.row_end = row_end;
      p.geom = ibl::make_level_geom(ws, hs);
      for(int f = 0; f < 6; ++f)
        p.quats[f] = ctx->quats[f];
      ibl::raw_channel_norms(table.total_weight, p.norm);
      p.exp_mul = 0x00800000u;
      p.probes = batch.probes;
      p.src_stride = batch.stride;
      p.dst_stride = batch.stride;

      int slot = record_dominant ? begin_dominant(ctx, (double)(row_end - row_begin) * wd * (double)table.samples * batch.probes) : -1;

      cudaError_t err = ibl::launch_prefilter_tail(p, ctx->sm_count, ctx->stream);
      if (err != cudaSuccess)
        return fail_cuda("prefilter_tail", err);
      ctx->launches += 1;

      if (slot >= 0)
        cudaEventRecord(ctx->ring_end[slot], ctx->stream);

      return 0;
    }

    if (ctx->prefilter_variant == 0 || ctx->prefilter_variant >= 50)
      return run_level_dn(ctx, d_src, ws, hs, table, row_begin, row_end, d_dst_words, d_dst_f32, record_dominant, peers, batch);

#ifdef DATUM_IBL_AB_VARIANTS
    // 10..27 pin a kernel of tools/ab/prefilter.cu (the tools build only, A/B timing)
    if (peers.count > 0 || batch.probes > 1)
      return fail("prefilter: the A/B kernels do not store to peers or take batches");

    cudaError_t err = ctx->records.reserve((size_t)6 * ws * hs);
    if (err != cudaSuccess)
      return fail_cuda("cudaMalloc(quad records)", err);

    err = ibl::launch_build_quad_records(d_src, ctx->records.ptr, ws, hs, ctx->sm_count, ctx->stream);
    if (err != cudaSuccess)
      return fail_cuda("build_quad_records", err);
    ctx->launches += 1;

    ibl::PrefilterParams p = {};
    p.records = ctx->records.ptr;
    p.table = table.d_entries;
    p.table_count = table.count;
    p.dst_words = d_dst_words;
    p.dst_f32 = d_dst_f32;
    p.wd = wd;
    p.hd = hd;
    p.row_begin = row_begin;
    p.row_end = row_end;
    p.geom = ibl::make_level_geom(ws, hs);
    for(int f = 0; f < 6; ++f)
      p.quats[f] = ctx->quats[f];
    p.masks = ibl::make_decode_masks();
    p.norm = table.norm;

    int slot = record_dominant ? begin_dominant(ctx, (double)(row_end - row_begin) * wd * (double)table.samples) : -1;

    err = ibl::launch_prefilter_level(p, ctx->prefilter_variant, ctx->sm_count, ctx->stream, nullptr);
    if (err != cudaSuccess)
      return fail_cuda("prefilter_level", err);
    ctx->launches += 1;

    if (slot >= 0)
      cudaEventRecord(ctx->ring_end[slot], ctx->stream);

    return 0;
#else
    return fail("prefilter: variants 1..49 exist only in the tools build (python -m datum_b200.build --ab)");
#endif
  }

  // data/project.comp:23-106 for a slab of rows, on `stream` (the context's own, or the upload stream of a
  // batch so that the projection of probe i+1 runs under the prefilter kernels of probe i).  The scratch
  // (block partials, ticket) is shared: callers keep their projections on ONE stream at a time.
  int sh9_partial_on(datum_ibl_ctx *ctx, cudaStream_t stream, void const *d_level0, int format, int width, int height, int row_begin, int row_end, double *d_partial, ibl::Sh9Peers const &peers = ibl::Sh9Peers(), int probes = 1, size_t probe_stride = 0)
  {
    if (ctx->sh_weights_w != width || ctx->sh_weights_h != height)
    {
      cudaError_t err = ctx->sh_weights.reserve((size_t)width * height);
      if (err != cudaSuccess)
        return fail_cuda("cudaMalloc(sh9 weights)", err);

      err = ibl::launch_sh9_weights(ctx->sh_weights.ptr, width, height, ctx->stream);
      if (err == cudaSuccess && stream != ctx->stream)
        err = cudaStreamSynchronize(ctx->stream);      // once per face size: the table is built on the context's stream
      if (err != cudaSuccess)
        return fail_cuda("sh9_weights", err);
      ctx->launches += 1;

      ctx->sh_weights_w = width;
      ctx->sh_weights_h = height;
    }

    int blocks = ibl::sh9_partial_blocks(width, height, ctx->sm_count);

    // one ticket per cube of a batch (zeroed once, the kernel leaves them at zero), block partials per cube
    cudaError_t err = ctx->sh_partials.reserve((size_t)blocks * 28 * probes + 28);
    if (err == cudaSuccess && ctx->sh_counter.capacity < (size_t)(probes > 16 ? probes : 16))
    {
      err = cudaStreamSynchronize(stream);             // a projection in flight still owns the old tickets
      if (err == cudaSuccess)
        err = ctx->sh_counter.reserve(probes > 16 ? probes : 16);
      if (err == cudaSuccess)
        err = cudaMemsetAsync(ctx->sh_counter.ptr, 0, ctx->sh_counter.capacity * sizeof(unsigned int), stream);
    }
    if (err != cudaSuccess)
      return fail_cuda("cudaMalloc(sh9 partials)", err);

    err = ibl::launch_sh9_partial(d_level0, format, ctx->sh_weights.ptr, width, height, row_begin, row_end, ctx->sh_partials.ptr, blocks, ctx->sh_counter.ptr, d_partial, peers, ctx->sm_count, stream, ctx->sh9_kernel, ctx->sh9_rows_per_item, probes, probe_stride);
    if (err != cudaSuccess)
      return fail_cuda("sh9_partial", err);
    ctx->launches += 1;

    return 0;
  }

  // ---- arrival counters of the GPUs that share a probe ------------------------------------------
  //
  // Flag block of a rank = two 32-bit counters (zeroed at allocation).  Event e (1, 2, 3, ... in the
  // same order on every rank) uses counter e & 1: every other rank adds 1 to it when its part of the
  // event is stored (the last CTA of the producing launch, or the signal kernel), and the rank's own
  // stream waits until the counter has seen (world - 1) arrivals for each event of that parity so far.
  // Alternating the counters keeps a fast rank's arrival for event e + 1 out of the count of event e
  // (it cannot reach e + 2 before everybody passed e).  The wait is a stream memory operation
  // (cuStreamWaitValue32): no kernel launch, no SM occupied while waiting.
  uint32_t arrivals_expected(uint32_t epoch, int world)
  {
    return ((epoch + (epoch & 1u)) / 2u) * (uint32_t)(world - 1);
  }

  typedef CUresult (*StreamWaitValue32)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);

  StreamWaitValue32 stream_wait_value32()
  {
    static StreamWaitValue32 fn = [] {
      void *ptr = nullptr;
      cudaDriverEntryPointQueryResult found;
      if (cudaGetDriverEntryPoint("cuStreamWaitValue32", &ptr, cudaEnableDefault, &found) != cudaSuccess || found != cudaDriverEntryPointSuccess)
        ptr = nullptr;
      return reinterpret_cast<StreamWaitValue32>(ptr);
    }();
    return fn;
  }

  int wait_for_arrivals(datum_ibl_ctx *ctx, uint32_t *d_own_flags, uint32_t epoch, int world)
  {
    if (world <= 1)
      return 0;

    StreamWaitValue32 wait = stream_wait_value32();
    if (!wait)
      return fail("peer wait: the driver does not export cuStreamWaitValue32");

    CUresult res = wait((CUstream)ctx->stream, (CUdeviceptr)(uintptr_t)(d_own_flags + (epoch & 1u)), arrivals_expected(epoch, world), CU_STREAM_WAIT_VALUE_GEQ);
    if (res != CUDA_SUCCESS)
      return fail("peer wait: cuStreamWaitValue32 failed (" + std::to_string((int)res) + ")");

    ctx->peer_wait_pending = true;
    ctx->peer_wait_word = reinterpret_cast<unsigned int*>(d_own_flags);
    return 0;
  }

  int signal_arrival(datum_ibl_ctx *ctx, int rank, int world, uint32_t *const *d_flags, uint32_t epoch)
  {
    ibl::PeerSignal signal = {};
    for(int r = 0; r < world; ++r)
      if (r != rank)
        signal.arrive[signal.count++] = reinterpret_cast<unsigned int*>(d_flags[r] + (epoch & 1u));

    if (signal.count == 0)
      return 0;

    cudaError_t err = ibl::launch_peer_signal(signal, ctx->stream);
    if (err != cudaSuccess)
      return fail_cuda("peer_signal", err);
    ctx->launches += 1;
    return 0;
  }

  // the copy streams and events of the host entry points, created on first use
  int ensure_pipeline(datum_ibl_ctx *ctx)
  {
    if (ctx->copy_in)
      return 0;

    cudaError_t err = cudaStreamCreateWithFlags(&ctx->copy_in, cudaStreamNonBlocking);
    if (err == cudaSuccess)
      err = cudaStreamCreateWithFlags(&ctx->copy_out, cudaStreamNonBlocking);
    for(int k = 0; k < 2 && err == cudaSuccess; ++k)
    {
      err = cudaEventCreateWithFlags(&ctx->ev_uploaded[k], cudaEventDisableTiming);
      if (err == cudaSuccess)
        err = cudaEventCreateWithFlags(&ctx->ev_computed[k], cudaEventDisableTiming);
      if (err == cudaSuccess)
        err = cudaEventCreateWithFlags(&ctx->ev_downloaded[k], cudaEventDisableTiming);
    }
    for(int k = 0; k < 16 && err == cudaSuccess; ++k)
    {
      err = cudaEventCreateWithFlags(&ctx->ev_level[k], cudaEventDisableTiming);
      if (err == cudaSuccess)
        err = cudaEventCreateWithFlags(&ctx->ev_copied[k], cudaEventDisableTiming);
    }

    if (err != cudaSuccess)
      return fail_cuda("copy streams", err);

    return 0;
  }

  // ---- pageable caller buffers -------------------------------------------------------------------
  //
  // tools/assetbuilder.cpp hands over a plain std::vector<char> (:439, :484).  cudaMemcpyAsync from or to
  // pageable memory is staged by the driver on the calling thread and blocks it: the upload runs at one
  // core's memcpy speed and every level's download stalls the launches behind it (2.17 ms instead of
  // 1.45 ms per 512^2 x 8 bake).  Here pageable payloads go through a pinned staging buffer of the
  // context: the upload in four chunks, each copied by a few host threads and sent while the next one
  // is being copied; the downloads asynchronously like a pinned caller's, each level moved on to the
  // caller's memory as soon as it has arrived, while the later levels are still being computed.

  bool host_is_pinned(void const *ptr)
  {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, ptr) != cudaSuccess)
    {
      cudaGetLastError();
      return false;
    }
    return attr.type == cudaMemoryTypeHost || attr.type == cudaMemoryTypeManaged;
  }

  int reserve_host_stage(datum_ibl_ctx *ctx, size_t bytes)
  {
    if (bytes <= ctx->host_stage_bytes)
      return 0;

    if (ctx->host_stage)
    {
      cudaStreamSynchronize(ctx->stream);
      if (ctx->copy_out)
        cudaStreamSynchronize(ctx->copy_out);
      cudaFreeHost(ctx->host_stage);
      ctx->host_stage = nullptr;
      ctx->host_stage_bytes = 0;
    }

    cudaError_t err = cudaHostAlloc(&ctx->host_stage, bytes, cudaHostAllocDefault);
    if (err != cudaSuccess)
      return fail_cuda("cudaHostAlloc(staging)", err);

    ctx->host_stage_bytes = bytes;
    return 0;
  }

  // memcpy on up to four host threads (one core moves ~10 GB/s, a payload level is megabytes)
  void copy_parallel(void *dst, void const *src, size_t bytes)
  {
    size_t parts = bytes >= ((size_t)2 << 20) ? 4 : (bytes >= ((size_t)512 << 10) ? 2 : 1);
    if (parts == 1)
    {
      std::memcpy(dst, src, bytes);
      return;
    }

    size_t each = (bytes / parts + 63) & ~(size_t)63;
    std::vector<std::thread> helpers;
    for(size_t k = 1; k < parts; ++k)
    {
      size_t begin = k * each, end = std::min(bytes, begin + each);
      if (begin < end)
        helpers.emplace_back([=] { std::memcpy(static_cast<char*>(dst) + begin, static_cast<char const*>(src) + begin, end - begin); });
    }
    std::memcpy(dst, src, std::min(bytes, each));
    for(auto &t : helpers)
      t.join();
  }

  // host -> device on the context's stream; a pageable source goes through `stage` (pinned, at least `bytes`):
  // up to four host threads each own a contiguous share, copy it into the staging in two pieces and queue every
  // piece's DMA behind its copy, so that the copies of one piece run under the DMA of another
  cudaError_t upload_host(datum_ibl_ctx *ctx, void *d_dst, void const *src, size_t bytes, bool pinned, void *stage)
  {
    if (pinned)
      return cudaMemcpyAsync(d_dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream);

    const size_t workers = bytes >= ((size_t)2 << 20) ? 4 : 1;
    const size_t share = ((bytes + workers - 1) / workers + 255) & ~(size_t)255;
    std::vector<cudaError_t> status(workers, cudaSuccess);

    auto work = [&](size_t k)
    {
      cudaSetDevice(ctx->device);
      size_t begin = k * share, end = std::min(bytes, begin + share);
      size_t piece = ((end - begin) / 2 + 255) & ~(size_t)255;
      for(size_t at = begin; at < end && piece > 0; at += piece)
      {
        size_t n = std::min(piece, end - at);
        std::memcpy(static_cast<char*>(stage) + at, static_cast<char const*>(src) + at, n);
        cudaError_t err = cudaMemcpyAsync(static_cast<char*>(d_dst) + at, static_cast<char*>(stage) + at, n, cudaMemcpyHostToDevice, ctx->stream);
        if (err != cudaSuccess)
        {
          status[k] = err;
          return;
        }
      }
    };

    std::vector<std::thread> helpers;
    for(size_t k = 1; k < workers; ++k)
      if (k * share < bytes)
        helpers.emplace_back(work, k);
    work(0);
    for(auto &t : helpers)
      t.join();

    for(auto err : status)
      if (err != cudaSuccess)
        return err;

    return cudaSuccess;
  }

  // levels [first, levels) of a chain have been sent to the staging by run_chain / send_level: move each on
  // to the caller's pageable payload as soon as it has arrived
  int drain_staged_levels(datum_ibl_ctx *ctx, int width, int height, int levels, int first, uint32_t *bits)
  {
    size_t offset = 0;
    for(int level = 0; level < levels; ++level)
    {
      size_t count = (size_t)(width >> level) * (height >> level) * 6;
      if (level >= first)
      {
        cudaError_t err = cudaEventSynchronize(ctx->ev_copied[level]);
        if (err != cudaSuccess)
          return fail_cuda("cudaEventSynchronize(level copied)", err);
        copy_parallel(bits + offset, static_cast<uint32_t*>(ctx->host_stage) + offset, count * sizeof(uint32_t));
      }
      offset += count;
    }
    return 0;
  }

  // one finished level -> host (the caller's pinned payload or the staging), behind the compute stream
  cudaError_t send_level(datum_ibl_ctx *ctx, int level, uint32_t *host_dst, uint32_t const *d_src, size_t count)
  {
    cudaError_t err = cudaEventRecord(ctx->ev_level[level], ctx->stream);
    if (err == cudaSuccess)
      err = cudaStreamWaitEvent(ctx->copy_out, ctx->ev_level[level], 0);
    if (err == cudaSuccess)
      err = cudaMemcpyAsync(host_dst, d_src, count * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->copy_out);
    if (err == cudaSuccess)
      err = cudaEventRecord(ctx->ev_copied[level], ctx->copy_out);
    return err;
  }

  // `host_bits` (optional): the caller's payload; every computed level is copied into it on the
  // download stream as soon as it is complete, under the kernels of the next level.  The caller
  // synchronises ctx->copy_out.
  int run_chain(datum_ibl_ctx *ctx, int width, int height, int levels, int samples, uint32_t *d_bits, float *d_f32, uint32_t *host_bits = nullptr)
  {
    std::vector<DeviceTable> *tables = nullptr;
    if (get_tables(ctx, levels, samples, &tables))
      return 1;

    if (host_bits && ensure_pipeline(ctx))
      return 1;

    cudaEventRecord(ctx->ev_begin, ctx->stream);

    uint32_t *src = d_bits;
    uint32_t *dst = src + (size_t)width * height * 6;

    // tools/ibl.cpp:247-278
    for(int level = 1; level < levels; ++level)
    {
      int hd = height >> 1;

      if (run_level(ctx, src, width, height, (*tables)[level], 0, 6 * hd, dst, d_f32, level == 1))
        return 1;

      size_t outcount = (size_t)(width >> 1) * hd * 6;

      if (host_bits)
      {
        cudaError_t err = send_level(ctx, level, host_bits + (dst - d_bits), dst, outcount);
        if (err != cudaSuccess)
          return fail_cuda("cudaMemcpyAsync(level)", err);
      }

      src += (size_t)width * height * 6;
      dst += outcount;
      if (d_f32)
        d_f32 += 3 * outcount;

      width /= 2;
      height /= 2;
    }

    cudaEventRecord(ctx->ev_end, ctx->stream);
    ctx->timed = true;

    return 0;
  }
}

namespace
{
  // ---- float chains: RGBA16F / RGBA32F levels, no rgbe re-quantisation (prefilter_f.cu) ----

  bool float_format(int format)
  {
    return format == DATUM_IBL_FORMAT_F32 || format == DATUM_IBL_FORMAT_F16;
  }

  // the input range of the float kernels holds up to this many samples (prefilter_f.h, kFloatChainMaxRadiance)
  const int kFloatMaxSamples = 4096;

  // one level of a float chain on the context's stream.  The pair kernel takes slabs above kTailTexels of
  // levels at least a tile wide whose source it can address (proj_usable); everything else runs the tail kernel.
  // A batch computes the level of batch.probes chains in one launch (no d_dst_f32).
  int run_level_float(datum_ibl_ctx *ctx, int format, void const *d_src, int ws, int hs, DeviceTable const &table, int row_begin, int row_end, void *d_dst, float *d_dst_f32, bool record_dominant, Batch const &batch = Batch())
  {
    int wd = ws >> 1, hd = hs >> 1;

    if (check_slab(ws, hs, row_begin, row_end))
      return 1;
    if (row_begin == row_end)
      return 0;

    ibl::PrefilterFloatParams p = {};
    p.format = format;
    p.src = d_src;
    p.table = table.d_banded;
    p.table_proj = table.d_banded_proj;
    set_sector_tables(p, table);
    p.table_count = table.count;
    p.dst = d_dst;
    p.dst_f32 = d_dst_f32;
    p.wd = wd;
    p.hd = hd;
    p.row_begin = row_begin;
    p.row_end = row_end;
    p.geom = ibl::make_level_geom(ws, hs);
    for(int f = 0; f < 6; ++f)
      p.quats[f] = ctx->quats[f];
    p.norm = ibl::float_chain_norm(table.total_weight);
    p.probes = batch.probes;
    p.src_stride = batch.stride;
    p.dst_stride = batch.stride;
    p.record_stride = (size_t)6 * ws * hs;

    const bool tail = (size_t)(row_end - row_begin) * wd <= (size_t)ibl::kTailTexels || wd < 8 || !ibl::proj_usable(ws, hs);
    cudaError_t err = cudaSuccess;

    if (tail)
    {
      if (level_world_frames(ctx, wd, hd, &p.world_frames))
        return 1;
    }
    else
    {
      const size_t record_bytes = format == DATUM_IBL_FORMAT_F16 ? sizeof(ibl::F16Record) : sizeof(ibl::F32Record);
      err = ctx->float_records.reserve((size_t)6 * ws * hs * record_bytes * batch.probes);
      if (err == cudaSuccess)
        err = ctx->queue_heads.reserve((size_t)ctx->sm_count + 1);
      if (err != cudaSuccess)
        return fail_cuda("cudaMalloc(float records)", err);

      err = ibl::launch_build_float_records(format, d_src, ctx->float_records.ptr, ws, hs, batch.probes, batch.stride, ctx->queue_heads.ptr, ctx->sm_count + 1, ctx->sm_count, ctx->stream);
      if (err != cudaSuccess)
        return fail_cuda("build_float_records", err);
      ctx->launches += 1;

      if (level_frames(ctx, ws, hs, &p.frames))
        return 1;
      p.records = ctx->float_records.ptr;
      p.counters = ctx->queue_heads.ptr;
    }

    int slot = record_dominant ? begin_dominant(ctx, (double)(row_end - row_begin) * wd * (double)table.samples * batch.probes) : -1;

    err = tail ? ibl::launch_prefilter_float_tail(p, ctx->stream) : ibl::launch_prefilter_float(p, ctx->sm_count, ctx->stream);
    if (err != cudaSuccess)
      return fail_cuda(("prefilter_float (source " + std::to_string(ws) + "x" + std::to_string(hs) + ", rows " + std::to_string(row_begin) + ".." + std::to_string(row_end) + ", " + std::to_string(batch.probes) + " probe(s))").c_str(), err);
    ctx->launches += 1;

    if (slot >= 0)
      cudaEventRecord(ctx->ring_end[slot], ctx->stream);

    return 0;
  }

  // tools/ibl.cpp:247-278 on a float chain: level L from level L-1 as stored in the chain.  A batch: level L of
  // batch.probes chains (batch.stride texels apart) in one record pass and one prefilter launch.
  int run_chain_float(datum_ibl_ctx *ctx, int format, int width, int height, int levels, int samples, unsigned char *d_chain, float *d_f32, Batch const &batch = Batch())
  {
    std::vector<DeviceTable> *tables = nullptr;
    if (get_tables(ctx, levels, samples, &tables))
      return 1;

    const size_t texel = (size_t)ibl::float_texel_bytes(format);

    cudaEventRecord(ctx->ev_begin, ctx->stream);

    unsigned char *src = d_chain;
    unsigned char *dst = src + (size_t)width * height * 6 * texel;

    for(int level = 1; level < levels; ++level)
    {
      int hd = height >> 1;

      if (run_level_float(ctx, format, src, width, height, (*tables)[level], 0, 6 * hd, dst, d_f32, level == 1, batch))
        return 1;

      size_t outcount = (size_t)(width >> 1) * hd * 6;

      src += (size_t)width * height * 6 * texel;
      dst += outcount * texel;
      if (d_f32)
        d_f32 += 3 * outcount;

      width /= 2;
      height /= 2;
    }

    cudaEventRecord(ctx->ev_end, ctx->stream);
    ctx->timed = true;

    return 0;
  }
}

namespace
{
  // Level 0 is already in ctx->chain (six-image ingest, equirect pack): send it home at once — it travels
  // under the level-1 kernels — then the chain with every level following as soon as it is complete.
  // `bits` receives the whole payload; pageable payloads go through the pinned staging.
  int finish_chain_to_host(datum_ibl_ctx *ctx, int width, int height, int levels, int samples, void *bits, const char *who)
  {
    size_t words = datum_ibl_chain_bytes(width, height, levels) / sizeof(uint32_t);
    size_t level0 = (size_t)width * height * 6;

    if (ensure_pipeline(ctx))
      return 1;

    const bool pinned = host_is_pinned(bits);
    if (!pinned && reserve_host_stage(ctx, words * sizeof(uint32_t)))
      return 1;

    uint32_t *host = pinned ? static_cast<uint32_t*>(bits) : static_cast<uint32_t*>(ctx->host_stage);

    int failed = 0;
    cudaError_t err = send_level(ctx, 0, host, ctx->chain.ptr, level0);
    if (err != cudaSuccess)
      failed = fail_cuda("cudaMemcpyAsync(level 0)", err);

    if (!failed)
      failed = run_chain(ctx, width, height, levels, samples, ctx->chain.ptr, nullptr, host);

    if (!failed && !pinned)
      failed = drain_staged_levels(ctx, width, height, levels, 0, static_cast<uint32_t*>(bits));

    // also after a failure: nothing may stay in flight that writes the caller's payload
    err = cudaStreamSynchronize(ctx->stream);
    cudaError_t err2 = cudaStreamSynchronize(ctx->copy_out);
    if (failed)
      return 1;
    if (err != cudaSuccess || err2 != cudaSuccess)
      return fail_cuda(who, err != cudaSuccess ? err : err2);

    return 0;
  }
}

namespace
{
  // tools/ibl.cpp:247-278 for `probes` chains `stride` words apart, level by level: one record pass and one
  // prefilter launch per level for the whole group
  int run_chain_batch(datum_ibl_ctx *ctx, int width, int height, int levels, int samples, uint32_t *d_base, int probes, size_t stride)
  {
    std::vector<DeviceTable> *tables = nullptr;
    if (get_tables(ctx, levels, samples, &tables))
      return 1;

    Batch batch;
    batch.probes = probes;
    batch.stride = stride;

    cudaEventRecord(ctx->ev_begin, ctx->stream);

    uint32_t *src = d_base;
    uint32_t *dst = src + (size_t)width * height * 6;

    for(int level = 1; level < levels; ++level)
    {
      int hd = height >> 1;

      if (run_level(ctx, src, width, height, (*tables)[level], 0, 6 * hd, dst, nullptr, level == 1, PeerTargets(), batch))
        return 1;

      src += (size_t)width * height * 6;
      dst += (size_t)(width >> 1) * hd * 6;
      width /= 2;
      height /= 2;
    }

    cudaEventRecord(ctx->ev_end, ctx->stream);
    ctx->timed = true;

    return 0;
  }

  // How many probes of a batch share a launch.  Probes of C2's size fill the machine by themselves (and
  // their per-level downloads overlap the next level); smaller ones leave the level-1 grid a few waves
  // deep and the last levels launch-bound, so they are baked 4 to 16 at a time.
  int batch_group(int width, int height, int levels, int count)
  {
    long long level0 = 6ll * width * height;
    long long group = (4ll * 6 * 512 * 512) / (level0 > 0 ? level0 : 1);
    if (group > 16)
      group = 16;
    if (group > count)
      group = count;
    if (group < 2)
      return 1;

    // every level must be able to run on the kernels that take batches
    for(int level = 1; level < levels; ++level)
      if (!ibl::prefilter_batchable(width >> (level - 1), height >> (level - 1)))
        return 1;

    return (int)group;
  }

  // A checked batch of host chains for bake_groups: what the rgbe and the float entries differ in is the texel
  // size, the SH9 format of level 0 and how a group is computed.
  struct BatchJob
  {
    const char *who;            // the entry point, for error strings
    int count, width, height, levels, samples;
    int format;                 // DATUM_IBL_FORMAT_*: what the SH9 projection reads
    size_t texel;               // bytes per texel
    void *const *payloads;      // host chains, level 0 pre-filled
    float *sh;                  // count x float[9][3], or null
  };

  // The pipeline of the batched entries: groups of probes alternate between two device payloads (ctx->chain,
  // ctx->chain2); the uploads of a group run on the upload stream under the kernels of the previous group,
  // with the SH9 of every level 0 behind them; the downloads follow on the download stream.
  // compute(d_base, first, n, levels_sent) queues levels 1.. of probes [first, first + n), chains back to back
  // at d_base, on the context's stream; with levels_sent set it has sent them home itself (on the download
  // stream), else they are copied behind its last kernel.  Synchronous.
  template<typename Compute>
  int bake_groups(datum_ibl_ctx *ctx, BatchJob const &job, int group, Compute compute)
  {
    const std::string who = job.who;
    const size_t chain_bytes = datum_ibl_chain_bytes(job.width, job.height, job.levels) / sizeof(uint32_t) * job.texel;
    const size_t level0 = (size_t)job.width * job.height * 6 * job.texel;
    const size_t slot_words = chain_bytes / sizeof(uint32_t) * group;      // texels of every format are whole words

    cudaError_t err = ctx->chain.reserve(slot_words);
    if (err == cudaSuccess && job.count > group)
      err = ctx->chain2.reserve(slot_words);
    if (err == cudaSuccess && job.sh)
      err = ctx->batch_sh.reserve((size_t)job.count * 28);
    if (err != cudaSuccess)
      return fail_cuda("cudaMalloc(batch)", err);

    if (ensure_pipeline(ctx))
      return 1;

    // sample tables and the solid-angle table are built on the compute stream before the pipeline starts
    std::vector<DeviceTable> *tables = nullptr;
    if (get_tables(ctx, job.levels, job.samples, &tables))
      return 1;

    unsigned char *slots[2] = { reinterpret_cast<unsigned char*>(ctx->chain.ptr), reinterpret_cast<unsigned char*>(ctx->chain2.ptr) };

    // a failure in the middle leaves copies from and to the caller's payloads in flight: drain them first
    auto drain = [ctx](int status)
    {
      cudaStreamSynchronize(ctx->copy_in);
      cudaStreamSynchronize(ctx->stream);
      cudaStreamSynchronize(ctx->copy_out);
      return status;
    };

    // Group sizes: the first upload and the last download cannot hide under any kernel, so a long batch
    // starts and ends with a quarter group (32 probes of 256^2 per GPU: 4 + 16 + 8 + 4 instead of 16 + 16
    // exposes 0.35 ms of copies instead of 1.35 ms).
    const int count = job.count;
    auto group_size = [&](int first)
    {
      int left = count - first;
      int quarter = std::max(1, group / 4);
      if (group >= 4 && count >= group + 2 * quarter)
      {
        if (first == 0)
          return quarter;
        if (left <= quarter)
          return left;
        if (left < group + quarter)
          return left - quarter;          // leave a quarter group for the end
      }
      return std::min(group, left);
    };

    for(int first = 0, g = 0, n = 0; first < count; first += n, ++g)
    {
      int k = g & 1;
      n = group_size(first);
      unsigned char *d_base = slots[k];

      // the uploads of group g wait until the downloads of group g-2 have drained these payloads
      if (g >= 2)
        err = cudaStreamWaitEvent(ctx->copy_in, ctx->ev_downloaded[k], 0);
      for(int j = 0; j < n && err == cudaSuccess; ++j)
        err = cudaMemcpyAsync(d_base + (size_t)j * chain_bytes, job.payloads[first + j], level0, cudaMemcpyHostToDevice, ctx->copy_in);
      if (err == cudaSuccess)
        err = cudaEventRecord(ctx->ev_uploaded[k], ctx->copy_in);
      if (err == cudaSuccess)
        err = cudaStreamWaitEvent(ctx->stream, ctx->ev_uploaded[k], 0);
      if (err != cudaSuccess)
        return drain(fail_cuda((who + ": upload").c_str(), err));

      // the projection reads level 0 only: it runs behind the upload on the upload stream, under the
      // prefilter kernels of the previous group; the next upload into these payloads queues behind it
      if (job.sh && sh9_partial_on(ctx, ctx->copy_in, d_base, job.format, job.width, job.height, 0, 6 * job.height, ctx->batch_sh.ptr + (size_t)first * 28, ibl::Sh9Peers(), ctx->sh9_kernel == 0 ? n : 1, chain_bytes))
        return drain(1);
      for(int j = 1; job.sh && ctx->sh9_kernel != 0 && j < n; ++j)        // the A/B kernel takes one cube per launch
        if (sh9_partial_on(ctx, ctx->copy_in, d_base + (size_t)j * chain_bytes, job.format, job.width, job.height, 0, 6 * job.height, ctx->batch_sh.ptr + (size_t)(first + j) * 28))
          return drain(1);

      bool levels_sent = false;
      if (compute(d_base, first, n, levels_sent))
        return drain(1);

      if (!levels_sent)
      {
        // the group's levels go home behind its last level, under the kernels of the next group
        err = cudaEventRecord(ctx->ev_computed[k], ctx->stream);
        if (err == cudaSuccess)
          err = cudaStreamWaitEvent(ctx->copy_out, ctx->ev_computed[k], 0);
        for(int j = 0; j < n && err == cudaSuccess && chain_bytes > level0; ++j)
          err = cudaMemcpyAsync(static_cast<unsigned char*>(job.payloads[first + j]) + level0, d_base + (size_t)j * chain_bytes + level0, chain_bytes - level0, cudaMemcpyDeviceToHost, ctx->copy_out);
        if (err != cudaSuccess)
          return drain(fail_cuda((who + ": download").c_str(), err));
      }

      err = cudaEventRecord(ctx->ev_downloaded[k], ctx->copy_out);
      if (err != cudaSuccess)
        return drain(fail_cuda((who + ": download").c_str(), err));
    }

    std::vector<double> partials;
    if (job.sh)
    {
      partials.resize((size_t)count * 28);
      // all projections are on the upload stream: read the results behind the last one
      err = cudaMemcpyAsync(partials.data(), ctx->batch_sh.ptr, partials.size() * sizeof(double), cudaMemcpyDeviceToHost, ctx->copy_in);
      if (err == cudaSuccess)
        err = cudaStreamSynchronize(ctx->copy_in);
      if (err != cudaSuccess)
        return drain(fail_cuda((who + ": sh9 download").c_str(), err));
    }

    err = cudaStreamSynchronize(ctx->copy_out);
    if (err == cudaSuccess)
      err = cudaStreamSynchronize(ctx->stream);
    if (err != cudaSuccess)
      return fail_cuda(job.who, err);

    for(int i = 0; job.sh && i < count; ++i)
      datum_ibl_sh9_finish(partials.data() + (size_t)i * 28, job.sh + (size_t)i * 27);

    return 0;
  }
}

extern "C"
{
  const char *datum_ibl_last_error(void) { return g_last_error.c_str(); }

  int datum_ibl_create(int device, datum_ibl_ctx **out)
  {
    if (!out)
      return fail("datum_ibl_create: null out pointer");

    *out = nullptr;

    int count = 0;
    cudaError_t err = cudaGetDeviceCount(&count);
    if (err != cudaSuccess || count == 0)
      return fail(std::string("datum_ibl_create: no CUDA device (") + cudaGetErrorString(err) + "); libdatum_ibl_cuda has no CPU fallback");

    if (device < 0 || device >= count)
      return fail("datum_ibl_create: device index out of range");

    DeviceGuard guard(device);

    cudaDeviceProp prop;
    err = cudaGetDeviceProperties(&prop, device);
    if (err != cudaSuccess)
      return fail_cuda("cudaGetDeviceProperties", err);

    // the library carries sm_100a code only (arch-specific, no PTX fallback): any other device would
    // fail at the first launch with "no kernel image"
    if (prop.major != 10 || prop.minor != 0)
      return fail(std::string("datum_ibl_create: kernels are built for sm_100a (compute capability 10.0) only, device is ") + prop.name + " (" + std::to_string(prop.major) + "." + std::to_string(prop.minor) + ")");

    datum_ibl_ctx *ctx = new datum_ibl_ctx;
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;

    err = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
    if (err == cudaSuccess)
      err = cudaEventCreate(&ctx->ev_begin);
    if (err == cudaSuccess)
      err = cudaEventCreate(&ctx->ev_end);
    if (err != cudaSuccess)
    {
      delete ctx;
      return fail_cuda("datum_ibl_create", err);
    }

    // tools/ibl.cpp:253-261: Quaternion(axis, angle) = (cos(angle/2), axis*sin(angle/2)) in fp32
    const float pi = 3.14159265358979323846f;
    const float angles[6] = { -pi/2, pi/2, -pi/2, pi/2, 0.0f, pi };
    const int axes[6] = { 1, 1, 0, 0, 1, 1 };
    for(int f = 0; f < 6; ++f)
    {
      float c = std::cos(angles[f]/2), s = std::sin(angles[f]/2);
      ctx->quats[f] = ibl::Quatf{ c, axes[f] == 0 ? s : 0.0f, axes[f] == 1 ? s : 0.0f, 0.0f };
    }

    *out = ctx;
    return 0;
  }

  void datum_ibl_destroy(datum_ibl_ctx *ctx)
  {
    if (!ctx)
      return;

    DeviceGuard guard(ctx->device);

    cudaStreamSynchronize(ctx->stream);

    for(auto &entry : ctx->tables)
      for(auto &t : entry.second)
        free_table(t);

    ctx->chain.release();
    ctx->chain2.release();
    ctx->batch_sh.release();
    if (ctx->copy_in)
      cudaStreamDestroy(ctx->copy_in);
    if (ctx->copy_out)
      cudaStreamDestroy(ctx->copy_out);
    for(int k = 0; k < 2; ++k)
    {
      if (ctx->ev_uploaded[k]) cudaEventDestroy(ctx->ev_uploaded[k]);
      if (ctx->ev_computed[k]) cudaEventDestroy(ctx->ev_computed[k]);
      if (ctx->ev_downloaded[k]) cudaEventDestroy(ctx->ev_downloaded[k]);
    }
    for(int k = 0; k < 16; ++k)
    {
      if (ctx->ev_level[k]) cudaEventDestroy(ctx->ev_level[k]);
      if (ctx->ev_copied[k]) cudaEventDestroy(ctx->ev_copied[k]);
    }
    if (ctx->host_stage)
      cudaFreeHost(ctx->host_stage);
    ctx->records.release();
    ctx->float_records.release();
    for(auto &entry : ctx->frames)
      cudaFree(entry.second);
    ctx->frames.clear();
    ctx->frames_bytes = 0;
    for(auto &entry : ctx->world_frames)
      cudaFree(entry.second);
    ctx->world_frames.clear();
    ctx->world_frames_bytes = 0;
    ctx->queue_heads.release();
    ctx->peer_ticket.release();
    ctx->sh_weights.release();
    ctx->sh_partials.release();
    ctx->sh_counter.release();
    ctx->staging.release();
    ctx->sink.release();
    ctx->srgb_lut.release();

    for(auto &e : ctx->ring_begin)
      cudaEventDestroy(e);
    for(auto &e : ctx->ring_end)
      cudaEventDestroy(e);

    cudaEventDestroy(ctx->ev_begin);
    cudaEventDestroy(ctx->ev_end);
    cudaStreamDestroy(ctx->stream);

    delete ctx;
  }

  void *datum_ibl_stream(datum_ibl_ctx *ctx) { return ctx ? (void*)ctx->stream : nullptr; }

  int datum_ibl_synchronize(datum_ibl_ctx *ctx)
  {
    if (!ctx)
      return fail("null context");

    DeviceGuard guard(ctx->device);

    // Waits on peers' arrivals are queued on the stream: a peer that died would hang it for good.
    // Poll with a deadline instead; on expiry satisfy every queued wait from the host (the counters
    // only ever count up to a few thousand: 2^30 passes any GEQ test), let the stream drain and
    // report a recoverable error.
    if (ctx->peer_wait_pending && ctx->peer_timeout_ms > 0)
    {
      auto deadline = std::chrono::steady_clock::now() + std::chrono::milliseconds(ctx->peer_timeout_ms);
      cudaError_t state;
      while ((state = cudaStreamQuery(ctx->stream)) == cudaErrorNotReady)
      {
        std::this_thread::yield();

        if (std::chrono::steady_clock::now() > deadline)
        {
          const unsigned int release[2] = { 0x40000000u, 0x40000000u };
          cudaMemcpy(ctx->peer_wait_word, release, sizeof(release), cudaMemcpyHostToDevice);
          cudaStreamSynchronize(ctx->stream);
          ctx->peer_wait_pending = false;
          return fail("datum_ibl_synchronize: a GPU sharing this probe did not arrive within " + std::to_string(ctx->peer_timeout_ms) + " ms; the waits were released and the results of this bake are invalid");
        }
      }
      ctx->peer_wait_pending = false;
      if (state != cudaSuccess)
        return fail_cuda("cudaStreamQuery", state);
    }

    cudaError_t err = cudaStreamSynchronize(ctx->stream);
    ctx->peer_wait_pending = false;
    return err == cudaSuccess ? 0 : fail_cuda("cudaStreamSynchronize", err);
  }

  int datum_ibl_set_peer_timeout_ms(datum_ibl_ctx *ctx, int milliseconds)
  {
    if (!ctx || milliseconds < 0)
      return fail("datum_ibl_set_peer_timeout_ms: bad argument");

    ctx->peer_timeout_ms = milliseconds;
    return 0;
  }

  uint64_t datum_ibl_launch_count(datum_ibl_ctx *ctx) { return ctx ? ctx->launches : 0; }

  int datum_ibl_set_prefilter_variant(datum_ibl_ctx *ctx, int variant)
  {
    // kernel shape + 10000 * (no tile stealing, A/B); 0 = automatic
    if (!ctx || variant < 0 || variant > 19999 || (variant % 10000) > 99)
      return fail("datum_ibl_set_prefilter_variant: bad argument");

    ctx->prefilter_variant = variant % 100;
    ctx->prefilter_no_steal = variant / 10000;
    return 0;
  }

  int datum_ibl_set_tuning(datum_ibl_ctx *ctx, const char *key, int value)
  {
    if (!ctx || !key || value < 0)
      return fail("datum_ibl_set_tuning: bad argument");

    std::string k = key;
    if (k == "prefilter_variant")
      return datum_ibl_set_prefilter_variant(ctx, value);
    if (k == "table_order" && value <= 1)
    {
      if (value != ctx->table_order)
      {
        // cached tables were built in the other order
        cudaStreamSynchronize(ctx->stream);
        for(auto &entry : ctx->tables)
          for(auto &t : entry.second)
            free_table(t);
        ctx->tables.clear();
      }
      ctx->table_order = value;
    }
    else if (k == "sh9_kernel" && value <= 1)
      ctx->sh9_kernel = value;
    else if (k == "sh9_rows_per_item" && value <= 4096)
      ctx->sh9_rows_per_item = value;
    else
      return fail("datum_ibl_set_tuning: unknown key or value out of range: " + k);

    return 0;
  }

  size_t datum_ibl_chain_bytes(int width, int height, int levels)
  {
    size_t size = 0;
    for(int i = 0; i < levels; ++i)
      size += (size_t)(width >> i) * (size_t)(height >> i) * 6 * sizeof(uint32_t);
    return size;
  }

  int datum_ibl_buildmips_cube_ibl_device(datum_ibl_ctx *ctx, int width, int height, int levels, int samples, uint32_t *d_bits, float *d_f32)
  {
    if (!ctx || !d_bits)
      return fail("datum_ibl_buildmips_cube_ibl_device: null argument");
    if (!valid_chain(width, height, levels) || samples < 1)
      return fail("datum_ibl_buildmips_cube_ibl_device: bad width/height/levels/samples");

    DeviceGuard guard(ctx->device);
    return run_chain(ctx, width, height, levels, samples, d_bits, d_f32);
  }

  int datum_ibl_buildmips_cube_ibl(datum_ibl_ctx *ctx, int width, int height, int levels, int samples, void *bits)
  {
    if (!ctx || !bits)
      return fail("datum_ibl_buildmips_cube_ibl: null argument");
    if (!valid_chain(width, height, levels) || samples < 1)
      return fail("datum_ibl_buildmips_cube_ibl: bad width/height/levels/samples");

    DeviceGuard guard(ctx->device);

    size_t words = datum_ibl_chain_bytes(width, height, levels) / sizeof(uint32_t);
    size_t level0 = (size_t)width * height * 6;

    cudaError_t err = ctx->chain.reserve(words);
    if (err != cudaSuccess)
      return fail_cuda("cudaMalloc(chain)", err);

    if (ensure_pipeline(ctx))
      return 1;

    // a pageable payload (assetbuilder's std::vector<char>) goes through the context's pinned staging
    const bool pinned = host_is_pinned(bits);
    if (!pinned && reserve_host_stage(ctx, words * sizeof(uint32_t)))
      return 1;

    uint32_t *host = pinned ? static_cast<uint32_t*>(bits) : static_cast<uint32_t*>(ctx->host_stage);

    err = upload_host(ctx, ctx->chain.ptr, bits, level0 * sizeof(uint32_t), pinned, ctx->host_stage);
    if (err != cudaSuccess)
    {
      cudaStreamSynchronize(ctx->stream);
      return fail_cuda("cudaMemcpyAsync(level 0)", err);
    }

    int failed = run_chain(ctx, width, height, levels, samples, ctx->chain.ptr, nullptr, host);

    if (!failed && !pinned)
      failed = drain_staged_levels(ctx, width, height, levels, 1, static_cast<uint32_t*>(bits));

    // also after a failure: nothing may stay in flight that reads or writes the caller's payload
    err = cudaStreamSynchronize(ctx->stream);
    if (ctx->copy_out)
    {
      cudaError_t err2 = cudaStreamSynchronize(ctx->copy_out);
      if (err == cudaSuccess)
        err = err2;
    }
    if (failed)
      return 1;
    if (err != cudaSuccess)
      return fail_cuda("datum_ibl_buildmips_cube_ibl", err);

    return 0;
  }

  int datum_ibl_bake_probes(datum_ibl_ctx *ctx, int count, int width, int height, int levels, int samples, void *const *bits, float *sh)
  {
    if (!ctx || (count > 0 && !bits))
      return fail("datum_ibl_bake_probes: null argument");
    if (count < 0 || !valid_chain(width, height, levels) || samples < 1)
      return fail("datum_ibl_bake_probes: bad count/width/height/levels/samples");
    for(int i = 0; i < count; ++i)
      if (!bits[i])
        return fail("datum_ibl_bake_probes: null payload in the batch");
    if (count == 0)
      return 0;

    DeviceGuard guard(ctx->device);

    const size_t words = datum_ibl_chain_bytes(width, height, levels) / sizeof(uint32_t);
    const int group = batch_group(width, height, levels, count);

    BatchJob job = { "datum_ibl_bake_probes", count, width, height, levels, samples, DATUM_IBL_FORMAT_RGBE, sizeof(uint32_t), bits, sh };
    return bake_groups(ctx, job, group, [&](unsigned char *d_base, int first, int n, bool &levels_sent)
    {
      uint32_t *d_words = reinterpret_cast<uint32_t*>(d_base);

      // one probe per launch: every level goes home as soon as it is complete, under the next level's kernels
      if (group == 1)
      {
        levels_sent = true;
        return run_chain(ctx, width, height, levels, samples, d_words, nullptr, (uint32_t*)bits[first]);
      }

      // level L of the whole group in one launch
      return run_chain_batch(ctx, width, height, levels, samples, d_words, n, words);
    });
  }

  int datum_ibl_bake_probes_float(datum_ibl_ctx *ctx, int format, int count, int width, int height, int levels, int samples, void *const *chains, float *sh)
  {
    if (!ctx || (count > 0 && !chains))
      return fail("datum_ibl_bake_probes_float: null argument");
    if (!float_format(format))
      return fail("datum_ibl_bake_probes_float: unknown format " + std::to_string(format) + " (DATUM_IBL_FORMAT_F32 or DATUM_IBL_FORMAT_F16)");
    if (count < 0 || !valid_chain(width, height, levels) || samples < 1 || samples > kFloatMaxSamples)
      return fail("datum_ibl_bake_probes_float: bad count/width/height/levels/samples");
    for(int i = 0; i < count; ++i)
      if (!chains[i])
        return fail("datum_ibl_bake_probes_float: null payload in the batch");
    if (count == 0)
      return 0;

    DeviceGuard guard(ctx->device);

    const size_t texels = datum_ibl_chain_bytes(width, height, levels) / sizeof(uint32_t);
    const int group = batch_group(width, height, levels, count);

    // a group of one runs the single-probe kernels and downloads after its last level like a bigger group
    BatchJob job = { "datum_ibl_bake_probes_float", count, width, height, levels, samples, format, (size_t)ibl::float_texel_bytes(format), chains, sh };
    return bake_groups(ctx, job, group, [&](unsigned char *d_base, int, int n, bool &)
    {
      Batch batch;
      batch.probes = n;
      batch.stride = texels;
      return run_chain_float(ctx, format, width, height, levels, samples, d_base, nullptr, batch);
    });
  }

  int datum_ibl_prefilter_level_device(datum_ibl_ctx *ctx, uint32_t const *d_src, int ws, int hs, int level, int levels, int samples, int row_begin, int row_end, uint32_t *d_dst_words, float *d_dst_f32)
  {
    if (!ctx || !d_src)
      return fail("datum_ibl_prefilter_level_device: null argument");
    if (levels < 2 || levels > 16 || level < 1 || level >= levels || samples < 1)
      return fail("datum_ibl_prefilter_level_device: bad level/levels/samples");

    DeviceGuard guard(ctx->device);

    std::vector<DeviceTable> *tables = nullptr;
    if (get_tables(ctx, levels, samples, &tables))
      return 1;

    return run_level(ctx, d_src, ws, hs, (*tables)[level], row_begin, row_end, d_dst_words, d_dst_f32);
  }

  int datum_ibl_buildmips_cube_float_device(datum_ibl_ctx *ctx, int format, int width, int height, int levels, int samples, void *d_chain, float *d_f32)
  {
    if (!ctx || !d_chain)
      return fail("datum_ibl_buildmips_cube_float_device: null argument");
    if (!float_format(format))
      return fail("datum_ibl_buildmips_cube_float_device: unknown format " + std::to_string(format) + " (DATUM_IBL_FORMAT_F32 or DATUM_IBL_FORMAT_F16)");
    if (!valid_chain(width, height, levels) || samples < 1 || samples > kFloatMaxSamples)
      return fail("datum_ibl_buildmips_cube_float_device: bad width/height/levels/samples");
    if (reinterpret_cast<uintptr_t>(d_chain) % ibl::float_texel_bytes(format) != 0 || reinterpret_cast<uintptr_t>(d_f32) % sizeof(float) != 0)
      return fail("datum_ibl_buildmips_cube_float_device: misaligned chain or d_f32");

    DeviceGuard guard(ctx->device);
    return run_chain_float(ctx, format, width, height, levels, samples, static_cast<unsigned char*>(d_chain), d_f32);
  }

  int datum_ibl_buildmips_cube_float(datum_ibl_ctx *ctx, int format, int width, int height, int levels, int samples, void *chain)
  {
    if (!ctx || !chain)
      return fail("datum_ibl_buildmips_cube_float: null argument");
    if (!float_format(format))
      return fail("datum_ibl_buildmips_cube_float: unknown format " + std::to_string(format) + " (DATUM_IBL_FORMAT_F32 or DATUM_IBL_FORMAT_F16)");
    if (!valid_chain(width, height, levels) || samples < 1 || samples > kFloatMaxSamples)
      return fail("datum_ibl_buildmips_cube_float: bad width/height/levels/samples");

    DeviceGuard guard(ctx->device);

    const size_t texel = (size_t)ibl::float_texel_bytes(format);
    const size_t bytes = datum_ibl_chain_bytes(width, height, levels) / sizeof(uint32_t) * texel;
    const size_t level0 = (size_t)width * height * 6 * texel;

    cudaError_t err = ctx->staging.reserve(bytes);
    if (err != cudaSuccess)
      return fail_cuda("cudaMalloc(chain)", err);

    // a pageable chain goes through the context's pinned staging
    const bool pinned = host_is_pinned(chain);
    if (!pinned && reserve_host_stage(ctx, bytes))
      return 1;

    unsigned char *host = pinned ? static_cast<unsigned char*>(chain) : static_cast<unsigned char*>(ctx->host_stage);

    err = upload_host(ctx, ctx->staging.ptr, chain, level0, pinned, ctx->host_stage);
    if (err != cudaSuccess)
    {
      cudaStreamSynchronize(ctx->stream);
      return fail_cuda("cudaMemcpyAsync(level 0)", err);
    }

    int failed = run_chain_float(ctx, format, width, height, levels, samples, ctx->staging.ptr, nullptr);

    if (!failed && bytes > level0)
    {
      err = cudaMemcpyAsync(host + level0, ctx->staging.ptr + level0, bytes - level0, cudaMemcpyDeviceToHost, ctx->stream);
      if (err != cudaSuccess)
        failed = fail_cuda("cudaMemcpyAsync(levels)", err);
    }

    // also after a failure: nothing may stay in flight that reads or writes the caller's chain
    err = cudaStreamSynchronize(ctx->stream);
    if (failed)
      return 1;
    if (err != cudaSuccess)
      return fail_cuda("datum_ibl_buildmips_cube_float", err);

    if (!pinned && bytes > level0)
      copy_parallel(static_cast<unsigned char*>(chain) + level0, host + level0, bytes - level0);

    return 0;
  }

  int datum_ibl_prefilter_level_float_device(datum_ibl_ctx *ctx, int format, void const *d_src, int ws, int hs, int level, int levels, int samples, int row_begin, int row_end, void *d_dst, float *d_dst_f32)
  {
    if (!ctx || !d_src || !d_dst)
      return fail("datum_ibl_prefilter_level_float_device: null argument");
    if (!float_format(format))
      return fail("datum_ibl_prefilter_level_float_device: unknown format " + std::to_string(format) + " (DATUM_IBL_FORMAT_F32 or DATUM_IBL_FORMAT_F16)");
    if (levels < 2 || levels > 16 || level < 1 || level >= levels || samples < 1 || samples > kFloatMaxSamples)
      return fail("datum_ibl_prefilter_level_float_device: bad level/levels/samples");
    const uintptr_t align = (uintptr_t)ibl::float_texel_bytes(format);
    if (reinterpret_cast<uintptr_t>(d_src) % align != 0 || reinterpret_cast<uintptr_t>(d_dst) % align != 0 || reinterpret_cast<uintptr_t>(d_dst_f32) % sizeof(float) != 0)
      return fail("datum_ibl_prefilter_level_float_device: misaligned source, destination or d_dst_f32");

    DeviceGuard guard(ctx->device);

    std::vector<DeviceTable> *tables = nullptr;
    if (get_tables(ctx, levels, samples, &tables))
      return 1;

    return run_level_float(ctx, format, d_src, ws, hs, (*tables)[level], row_begin, row_end, d_dst, d_dst_f32, false);
  }

  int datum_ibl_prefilter_level_peers(datum_ibl_ctx *ctx, uint32_t const *d_src, int ws, int hs, int level, int levels, int samples, int row_begin, int row_end, int rank, int world, uint32_t *const *d_dst_words, uint32_t *const *d_flags, uint32_t epoch)
  {
    if (!ctx || !d_src || !d_dst_words)
      return fail("datum_ibl_prefilter_level_peers: null argument");
    if (levels < 2 || levels > 16 || level < 1 || level >= levels || samples < 1)
      return fail("datum_ibl_prefilter_level_peers: bad level/levels/samples");
    if (world < 1 || world > DATUM_IBL_MAX_PEERS + 1 || rank < 0 || rank >= world)
      return fail("datum_ibl_prefilter_level_peers: bad rank/world (at most 8 GPUs share a probe)");
    if (d_flags && epoch == 0)
      return fail("datum_ibl_prefilter_level_peers: epochs start at 1");

    PeerTargets peers;
    for(int r = 0; r < world; ++r)
    {
      if (!d_dst_words[r] || (d_flags && !d_flags[r]))
        return fail("datum_ibl_prefilter_level_peers: null pointer for a rank");
      if (r != rank)
      {
        peers.words[peers.count] = d_dst_words[r];
        peers.arrive[peers.count] = d_flags ? reinterpret_cast<unsigned int*>(d_flags[r] + (epoch & 1u)) : nullptr;
        peers.count += 1;
      }
    }

    DeviceGuard guard(ctx->device);

    std::vector<DeviceTable> *tables = nullptr;
    if (get_tables(ctx, levels, samples, &tables))
      return 1;

    if (row_begin == row_end && d_flags)
    {
      // an empty slab still has to arrive
      if (signal_arrival(ctx, rank, world, d_flags, epoch))
        return 1;
    }
    else if (run_level(ctx, d_src, ws, hs, (*tables)[level], row_begin, row_end, d_dst_words[rank], nullptr, false, peers))
      return 1;

    return d_flags ? wait_for_arrivals(ctx, d_flags[rank], epoch, world) : 0;
  }

  int datum_ibl_peer_barrier(datum_ibl_ctx *ctx, int rank, int world, uint32_t *const *d_flags, uint32_t epoch)
  {
    if (!ctx || !d_flags)
      return fail("datum_ibl_peer_barrier: null argument");
    if (world < 1 || world > DATUM_IBL_MAX_PEERS + 1 || rank < 0 || rank >= world || epoch == 0)
      return fail("datum_ibl_peer_barrier: bad rank/world/epoch");

    for(int r = 0; r < world; ++r)
      if (!d_flags[r])
        return fail("datum_ibl_peer_barrier: null flag array");

    DeviceGuard guard(ctx->device);

    if (signal_arrival(ctx, rank, world, d_flags, epoch))
      return 1;

    return wait_for_arrivals(ctx, d_flags[rank], epoch, world);
  }

  int datum_ibl_peer_alloc(datum_ibl_ctx *ctx, size_t bytes, void **d_ptr, void *handle)
  {
    if (!ctx || !d_ptr || !handle || bytes == 0)
      return fail("datum_ibl_peer_alloc: null argument");

    static_assert(sizeof(cudaIpcMemHandle_t) == DATUM_IBL_IPC_HANDLE_BYTES, "IPC handle size");

    DeviceGuard guard(ctx->device);

    void *ptr = nullptr;
    cudaError_t err = cudaMalloc(&ptr, bytes);
    if (err == cudaSuccess)
      err = cudaMemsetAsync(ptr, 0, bytes, ctx->stream);
    if (err == cudaSuccess)
      err = cudaStreamSynchronize(ctx->stream);

    cudaIpcMemHandle_t h;
    if (err == cudaSuccess)
      err = cudaIpcGetMemHandle(&h, ptr);

    if (err != cudaSuccess)
    {
      if (ptr)
        cudaFree(ptr);
      return fail_cuda("datum_ibl_peer_alloc", err);
    }

    std::memcpy(handle, &h, sizeof(h));
    *d_ptr = ptr;
    return 0;
  }

  int datum_ibl_peer_free(datum_ibl_ctx *ctx, void *d_ptr)
  {
    if (!ctx)
      return fail("datum_ibl_peer_free: null argument");
    if (!d_ptr)
      return 0;

    DeviceGuard guard(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    cudaError_t err = cudaFree(d_ptr);
    return err == cudaSuccess ? 0 : fail_cuda("datum_ibl_peer_free", err);
  }

  int datum_ibl_peer_open(datum_ibl_ctx *ctx, void const *handle, void **d_ptr)
  {
    if (!ctx || !handle || !d_ptr)
      return fail("datum_ibl_peer_open: null argument");

    DeviceGuard guard(ctx->device);

    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, sizeof(h));

    void *ptr = nullptr;
    cudaError_t err = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
    if (err != cudaSuccess)
      return fail_cuda("datum_ibl_peer_open (the GPUs must be NVLink/PCIe peers in one node)", err);

    *d_ptr = ptr;
    return 0;
  }

  int datum_ibl_peer_close(datum_ibl_ctx *ctx, void *d_ptr)
  {
    if (!ctx)
      return fail("datum_ibl_peer_close: null argument");
    if (!d_ptr)
      return 0;

    DeviceGuard guard(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    cudaError_t err = cudaIpcCloseMemHandle(d_ptr);
    return err == cudaSuccess ? 0 : fail_cuda("datum_ibl_peer_close", err);
  }

  int datum_ibl_last_prefilter_ms(datum_ibl_ctx *ctx, float *ms)
  {
    if (!ctx || !ms)
      return fail("datum_ibl_last_prefilter_ms: null argument");
    if (!ctx->timed)
      return fail("datum_ibl_last_prefilter_ms: no chain has run yet");

    DeviceGuard guard(ctx->device);

    cudaError_t err = cudaEventSynchronize(ctx->ev_end);
    if (err == cudaSuccess)
      err = cudaEventElapsedTime(ms, ctx->ev_begin, ctx->ev_end);

    return err == cudaSuccess ? 0 : fail_cuda("cudaEventElapsedTime", err);
  }

  int datum_ibl_dominant_kernel_stats(datum_ibl_ctx *ctx, int reset, int *launches, double *avg_ms, double *texel_samples_per_launch)
  {
    if (!ctx || !launches || !avg_ms || !texel_samples_per_launch)
      return fail("datum_ibl_dominant_kernel_stats: null argument");

    DeviceGuard guard(ctx->device);

    cudaError_t err = cudaStreamSynchronize(ctx->stream);
    if (err != cudaSuccess)
      return fail_cuda("datum_ibl_dominant_kernel_stats", err);

    int n = ctx->ring_used < datum_ibl_ctx::kRing ? ctx->ring_used : datum_ibl_ctx::kRing;
    double total = 0;
    for(int i = 0; i < n; ++i)
    {
      float ms = 0;
      err = cudaEventElapsedTime(&ms, ctx->ring_begin[i], ctx->ring_end[i]);
      if (err != cudaSuccess)
        return fail_cuda("cudaEventElapsedTime(ring)", err);
      total += ms;
    }

    *launches = n;
    *avg_ms = n ? total / n : 0.0;
    *texel_samples_per_launch = ctx->ring_texel_samples;

    if (reset)
      ctx->ring_used = 0;

    return 0;
  }

  // ---- SH9 ----------------------------------------------------------------------

  int datum_ibl_sh9_partial_device(datum_ibl_ctx *ctx, void const *d_level0, int format, int width, int height, int row_begin, int row_end, double *d_partial)
  {
    if (!ctx || !d_level0 || !d_partial)
      return fail("datum_ibl_sh9_partial_device: null argument");
    if (width < 1 || height < 1 || (format != DATUM_IBL_FORMAT_RGBE && format != DATUM_IBL_FORMAT_F32 && format != DATUM_IBL_FORMAT_F16))
      return fail("datum_ibl_sh9_partial_device: bad width/height/format");
    if (row_begin < 0 || row_end > 6 * height || row_begin > row_end)
      return fail("datum_ibl_sh9_partial_device: row range outside the cube");

    DeviceGuard guard(ctx->device);

    return sh9_partial_on(ctx, ctx->stream, d_level0, format, width, height, row_begin, row_end, d_partial);
  }

  int datum_ibl_sh9_partial_peers(datum_ibl_ctx *ctx, void const *d_level0, int format, int width, int height, int row_begin, int row_end, int rank, int world, double *const *d_slots, uint32_t *const *d_flags, uint32_t epoch)
  {
    if (!ctx || !d_level0 || !d_slots)
      return fail("datum_ibl_sh9_partial_peers: null argument");
    if (width < 1 || height < 1 || (format != DATUM_IBL_FORMAT_RGBE && format != DATUM_IBL_FORMAT_F32 && format != DATUM_IBL_FORMAT_F16))
      return fail("datum_ibl_sh9_partial_peers: bad width/height/format");
    if (row_begin < 0 || row_end > 6 * height || row_begin > row_end)
      return fail("datum_ibl_sh9_partial_peers: row range outside the cube");
    if (world < 1 || world > DATUM_IBL_MAX_PEERS + 1 || rank < 0 || rank >= world)
      return fail("datum_ibl_sh9_partial_peers: bad rank/world");
    if (d_flags && epoch == 0)
      return fail("datum_ibl_sh9_partial_peers: epochs start at 1");

    ibl::Sh9Peers peers = {};
    for(int r = 0; r < world; ++r)
    {
      if (!d_slots[r] || (d_flags && !d_flags[r]))
        return fail("datum_ibl_sh9_partial_peers: null pointer for a rank");
      if (r != rank)
      {
        peers.slots[peers.count] = d_slots[r] + (size_t)rank * 28;
        peers.arrive[peers.count] = d_flags ? reinterpret_cast<unsigned int*>(d_flags[r] + (epoch & 1u)) : nullptr;
        peers.count += 1;
      }
    }

    DeviceGuard guard(ctx->device);

    if (sh9_partial_on(ctx, ctx->stream, d_level0, format, width, height, row_begin, row_end, d_slots[rank] + (size_t)rank * 28, peers))
      return 1;

    return d_flags ? wait_for_arrivals(ctx, d_flags[rank], epoch, world) : 0;
  }

  void datum_ibl_sh9_finish(double const *partial, float *sh)
  {
    const double pi = 3.1415926535897932384626433832795;
    double scale = 4 * pi / partial[27];
    for(int k = 0; k < 27; ++k)
      sh[k] = (float)(partial[k] * scale);
  }

  int datum_ibl_project_sh9(datum_ibl_ctx *ctx, void const *level0, int format, int width, int height, float *sh)
  {
    if (!ctx || !level0 || !sh)
      return fail("datum_ibl_project_sh9: null argument");
    if (width < 1 || height < 1 || (format != DATUM_IBL_FORMAT_RGBE && format != DATUM_IBL_FORMAT_F32 && format != DATUM_IBL_FORMAT_F16))
      return fail("datum_ibl_project_sh9: bad width/height/format");

    DeviceGuard guard(ctx->device);

    size_t bytes = (size_t)6 * width * height * (format == DATUM_IBL_FORMAT_RGBE ? 4 : (format == DATUM_IBL_FORMAT_F16 ? 8 : 16));

    cudaError_t err = ctx->staging.reserve(bytes + 28 * sizeof(double));
    if (err != cudaSuccess)
      return fail_cuda("cudaMalloc(staging)", err);

    // result slot first so that it stays 8-byte aligned
    double *d_partial = reinterpret_cast<double*>(ctx->staging.ptr);
    unsigned char *d_level0 = ctx->staging.ptr + 28 * sizeof(double);

    err = cudaMemcpyAsync(d_level0, level0, bytes, cudaMemcpyHostToDevice, ctx->stream);
    if (err != cudaSuccess)
      return fail_cuda("cudaMemcpyAsync(level 0)", err);

    if (datum_ibl_sh9_partial_device(ctx, d_level0, format, width, height, 0, 6 * height, d_partial))
      return 1;

    double partial[28];
    err = cudaMemcpyAsync(partial, d_partial, sizeof(partial), cudaMemcpyDeviceToHost, ctx->stream);
    if (err == cudaSuccess)
      err = cudaStreamSynchronize(ctx->stream);
    if (err != cudaSuccess)
      return fail_cuda("datum_ibl_project_sh9", err);

    datum_ibl_sh9_finish(partial, sh);
    return 0;
  }

  int datum_ibl_sh9_irradiance_cube(datum_ibl_ctx *ctx, float const *sh, int width, int height, uint32_t *words, float *f32)
  {
    if (!ctx || !sh || (!words && !f32))
      return fail("datum_ibl_sh9_irradiance_cube: null argument");
    if (width < 1 || height < 1)
      return fail("datum_ibl_sh9_irradiance_cube: bad width/height");

    DeviceGuard guard(ctx->device);

    size_t texels = (size_t)6 * width * height;

    cudaError_t err = ctx->staging.reserve(texels * 16);
    if (err != cudaSuccess)
      return fail_cuda("cudaMalloc(staging)", err);

    float *d_f32 = reinterpret_cast<float*>(ctx->staging.ptr);
    uint32_t *d_words = reinterpret_cast<uint32_t*>(ctx->staging.ptr + texels * 12);

    ibl::Sh9Coefficients coeffs;
    memcpy(coeffs.v, sh, sizeof(coeffs.v));

    err = ibl::launch_sh9_irradiance(coeffs, width, height, words ? d_words : nullptr, f32 ? d_f32 : nullptr, ctx->sm_count, ctx->stream);
    if (err != cudaSuccess)
      return fail_cuda("sh9_irradiance", err);
    ctx->launches += 1;

    if (words)
      err = cudaMemcpyAsync(words, d_words, texels * 4, cudaMemcpyDeviceToHost, ctx->stream);
    if (err == cudaSuccess && f32)
      err = cudaMemcpyAsync(f32, d_f32, texels * 12, cudaMemcpyDeviceToHost, ctx->stream);
    if (err == cudaSuccess)
      err = cudaStreamSynchronize(ctx->stream);

    return err == cudaSuccess ? 0 : fail_cuda("datum_ibl_sh9_irradiance_cube", err);
  }

  // ---- equirect image -> cube (+ chain) -------------------------------------------------

  static int pack_cube_to_device(datum_ibl_ctx *ctx, int imgwidth, int imgheight, float const *pixels, int width, int height, uint32_t *d_level0)
  {
    size_t image_bytes = (size_t)imgwidth * imgheight * sizeof(float4);

    cudaError_t err = ctx->staging.reserve(image_bytes);
    if (err != cudaSuccess)
      return fail_cuda("cudaMalloc(staging)", err);

    // HDRImage::bits is a std::vector: pageable, through the pinned staging in chunks (see upload_host)
    const bool pinned = host_is_pinned(pixels);
    if (!pinned && reserve_host_stage(ctx, image_bytes))
      return 1;

    err = upload_host(ctx, ctx->staging.ptr, pixels, image_bytes, pinned, ctx->host_stage);
    if (err != cudaSuccess)
    {
      cudaStreamSynchronize(ctx->stream);
      return fail_cuda("cudaMemcpyAsync(image)", err);
    }

    ibl::ResampleParams p = {};
    p.image = reinterpret_cast<float4 const *>(ctx->staging.ptr);
    p.imgw = imgwidth;
    p.imgh = imgheight;
    p.width = width;
    p.height = height;
    // tools/hdr.cpp:345
    p.area_x = 1.0f / (float)std::min(4 * width, imgwidth);
    p.area_y = 1.0f / (float)std::min(2 * height, imgheight);
    for(int f = 0; f < 6; ++f)
      p.quats[f] = ctx->quats[f];
    p.dst = d_level0;

    err = ibl::launch_equirect_resample(p, ctx->stream);
    if (err != cudaSuccess)
      return fail_cuda("equirect_resample", err);
    ctx->launches += 1;

    // tools/hdr.cpp:358 -> 322-327 with levels == 1: image_buildmips_rgbe does nothing, then the edge blend
    err = ibl::launch_blend_edges(d_level0, width, height, ctx->stream);
    if (err != cudaSuccess)
      return fail_cuda("blend_edges", err);
    if (width > 1 && height > 1)
      ctx->launches += 1;

    return 0;
  }

  int datum_ibl_pack_cube(datum_ibl_ctx *ctx, int imgwidth, int imgheight, float const *pixels, int width, int height, void *bits)
  {
    if (!ctx || !pixels || !bits)
      return fail("datum_ibl_pack_cube: null argument");
    if (imgwidth < 1 || imgheight < 1 || width < 1 || height < 1)
      return fail("datum_ibl_pack_cube: bad image or cube size");

    DeviceGuard guard(ctx->device);

    size_t level0 = (size_t)width * height * 6;

    cudaError_t err = ctx->chain.reserve(level0);
    if (err != cudaSuccess)
      return fail_cuda("cudaMalloc(chain)", err);

    if (pack_cube_to_device(ctx, imgwidth, imgheight, pixels, width, height, ctx->chain.ptr))
      return 1;

    err = cudaMemcpyAsync(bits, ctx->chain.ptr, level0 * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream);
    if (err == cudaSuccess)
      err = cudaStreamSynchronize(ctx->stream);

    return err == cudaSuccess ? 0 : fail_cuda("datum_ibl_pack_cube", err);
  }

  int datum_ibl_pack_cube_ibl(datum_ibl_ctx *ctx, int imgwidth, int imgheight, float const *pixels, int width, int height, int levels, int samples, void *bits)
  {
    if (!ctx || !pixels || !bits)
      return fail("datum_ibl_pack_cube_ibl: null argument");
    if (imgwidth < 1 || imgheight < 1 || !valid_chain(width, height, levels) || samples < 1)
      return fail("datum_ibl_pack_cube_ibl: bad image size or width/height/levels/samples");

    DeviceGuard guard(ctx->device);

    size_t words = datum_ibl_chain_bytes(width, height, levels) / sizeof(uint32_t);

    cudaError_t err = ctx->chain.reserve(words);
    if (err != cudaSuccess)
      return fail_cuda("cudaMalloc(chain)", err);

    if (!host_is_pinned(bits) && reserve_host_stage(ctx, std::max(words * sizeof(uint32_t), (size_t)imgwidth * imgheight * sizeof(float4))))     // before the upload uses it
      return 1;

    // tools/ibl.cpp:285, 287
    if (pack_cube_to_device(ctx, imgwidth, imgheight, pixels, width, height, ctx->chain.ptr))
      return 1;

    return finish_chain_to_host(ctx, width, height, levels, samples, bits, "datum_ibl_pack_cube_ibl");
  }

  // ---- six ARGB32 face images -> level 0 (+ chain) -------------------------------------

  namespace
  {
    // argb (host) -> ctx->chain level 0 on the context stream
    int ingest_to_device(datum_ibl_ctx *ctx, int width, int height, uint32_t const *argb, uint32_t *d_level0)
    {
      size_t level0 = (size_t)width * height * 6;

      // color.h:103-106, 115-118: the 256 values pow(c/255.0f, 2.2f) a channel can take, computed
      // once on the host with the C library the reference itself would call
      if (!ctx->srgb_lut.ptr)
      {
        float lut[256];
        for(int c = 0; c < 256; ++c)
          lut[c] = std::pow((uint8_t)c / 255.0f, 2.2f);

        cudaError_t err = ctx->srgb_lut.reserve(256);
        if (err == cudaSuccess)
          err = cudaMemcpyAsync(ctx->srgb_lut.ptr, lut, sizeof(lut), cudaMemcpyHostToDevice, ctx->stream);
        if (err == cudaSuccess)
          err = cudaStreamSynchronize(ctx->stream);   // `lut` is a stack array
        if (err != cudaSuccess)
          return fail_cuda("upload(srgb table)", err);
      }

      cudaError_t err = ctx->staging.reserve(level0 * sizeof(uint32_t));
      if (err != cudaSuccess)
        return fail_cuda("cudaMalloc(staging)", err);

      // QImage::bits() is pageable memory: through the pinned staging in chunks (see upload_host)
      const bool pinned = host_is_pinned(argb);
      if (!pinned && reserve_host_stage(ctx, level0 * sizeof(uint32_t)))
        return 1;

      err = upload_host(ctx, ctx->staging.ptr, argb, level0 * sizeof(uint32_t), pinned, ctx->host_stage);
      if (err != cudaSuccess)
      {
        cudaStreamSynchronize(ctx->stream);
        return fail_cuda("cudaMemcpyAsync(argb)", err);
      }

      err = ibl::launch_ingest_argb32((uint32_t const*)ctx->staging.ptr, ctx->srgb_lut.ptr, width, height, d_level0, ctx->sm_count, ctx->stream);
      if (err != cudaSuccess)
        return fail_cuda("ingest_argb32", err);
      ctx->launches += 1;

      return 0;
    }
  }

  int datum_ibl_ingest_cube_argb32(datum_ibl_ctx *ctx, int width, int height, uint32_t const *argb, void *bits)
  {
    if (!ctx || !argb || !bits)
      return fail("datum_ibl_ingest_cube_argb32: null argument");
    if (width < 1 || height < 1)
      return fail("datum_ibl_ingest_cube_argb32: bad width/height");

    DeviceGuard guard(ctx->device);

    size_t level0 = (size_t)width * height * 6;

    cudaError_t err = ctx->chain.reserve(level0);
    if (err != cudaSuccess)
      return fail_cuda("cudaMalloc(chain)", err);

    if (ingest_to_device(ctx, width, height, argb, ctx->chain.ptr))
      return 1;

    err = cudaMemcpyAsync(bits, ctx->chain.ptr, level0 * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream);
    if (err == cudaSuccess)
      err = cudaStreamSynchronize(ctx->stream);

    return err == cudaSuccess ? 0 : fail_cuda("datum_ibl_ingest_cube_argb32", err);
  }

  int datum_ibl_ingest_cube_argb32_ibl(datum_ibl_ctx *ctx, int width, int height, int levels, int samples, uint32_t const *argb, void *bits)
  {
    if (!ctx || !argb || !bits)
      return fail("datum_ibl_ingest_cube_argb32_ibl: null argument");
    if (!valid_chain(width, height, levels) || samples < 1)
      return fail("datum_ibl_ingest_cube_argb32_ibl: bad width/height/levels/samples");

    DeviceGuard guard(ctx->device);

    size_t words = datum_ibl_chain_bytes(width, height, levels) / sizeof(uint32_t);

    cudaError_t err = ctx->chain.reserve(words);
    if (err != cudaSuccess)
      return fail_cuda("cudaMalloc(chain)", err);

    if (!host_is_pinned(bits) && reserve_host_stage(ctx, words * sizeof(uint32_t)))     // before the upload uses it
      return 1;

    // tools/assetbuilder.cpp:443-462, then :465
    if (ingest_to_device(ctx, width, height, argb, ctx->chain.ptr))
      return 1;

    return finish_chain_to_host(ctx, width, height, levels, samples, bits, "datum_ibl_ingest_cube_argb32_ibl");
  }

  // ---- LUTs -----------------------------------------------------------------------

  int datum_ibl_pack_envbrdf(datum_ibl_ctx *ctx, int width, int height, int samples, void *bits)
  {
    if (!ctx || !bits)
      return fail("datum_ibl_pack_envbrdf: null argument");
    if (width < 1 || height < 1 || samples < 1)
      return fail("datum_ibl_pack_envbrdf: bad width/height/samples");

    DeviceGuard guard(ctx->device);

    size_t texels = (size_t)width * height;

    cudaError_t err = ctx->staging.reserve(texels * 4);
    if (err != cudaSuccess)
      return fail_cuda("cudaMalloc(staging)", err);

    uint32_t *d_words = reinterpret_cast<uint32_t*>(ctx->staging.ptr);

    err = ibl::launch_envbrdf(width, height, samples, d_words, nullptr, ctx->stream);
    if (err != cudaSuccess)
      return fail_cuda("envbrdf", err);
    ctx->launches += 1;

    err = cudaMemcpyAsync(bits, d_words, texels * 4, cudaMemcpyDeviceToHost, ctx->stream);
    if (err == cudaSuccess)
      err = cudaStreamSynchronize(ctx->stream);

    return err == cudaSuccess ? 0 : fail_cuda("datum_ibl_pack_envbrdf", err);
  }

  int datum_ibl_pack_watercolor(datum_ibl_ctx *ctx, float const *deepcolor, float const *shallowcolor, float depthscale, float const *fresnelcolor, float fresnelbias, float fresnelpower, int width, int height, void *bits)
  {
    if (!ctx || !bits || !deepcolor || !shallowcolor || !fresnelcolor)
      return fail("datum_ibl_pack_watercolor: null argument");
    if (width < 1 || height < 1)
      return fail("datum_ibl_pack_watercolor: bad width/height");

    DeviceGuard guard(ctx->device);

    size_t texels = (size_t)width * height;

    cudaError_t err = ctx->staging.reserve(texels * 4);
    if (err != cudaSuccess)
      return fail_cuda("cudaMalloc(staging)", err);

    uint32_t *d_words = reinterpret_cast<uint32_t*>(ctx->staging.ptr);

    ibl::WaterColorParams params;
    for(int c = 0; c < 3; ++c)
    {
      params.deep[c] = deepcolor[c];
      params.shallow[c] = shallowcolor[c];
      params.fresnel[c] = fresnelcolor[c];
    }
    params.depthscale = depthscale;
    params.fresnelbias = fresnelbias;
    params.fresnelpower = fresnelpower;

    err = ibl::launch_watercolor(params, width, height, d_words, ctx->stream);
    if (err != cudaSuccess)
      return fail_cuda("watercolor", err);
    ctx->launches += 1;

    err = cudaMemcpyAsync(bits, d_words, texels * 4, cudaMemcpyDeviceToHost, ctx->stream);
    if (err == cudaSuccess)
      err = cudaStreamSynchronize(ctx->stream);

    return err == cudaSuccess ? 0 : fail_cuda("datum_ibl_pack_watercolor", err);
  }

  // ---- measurement ------------------------------------------------------------------

  static int measure_peak(datum_ibl_ctx *ctx, double *tflops, bool packed);

  int datum_ibl_measure_fp32_peak(datum_ibl_ctx *ctx, double *tflops)
  {
    if (!ctx || !tflops)
      return fail("datum_ibl_measure_fp32_peak: null argument");

    return measure_peak(ctx, tflops, false);
  }

  int datum_ibl_measure_fp32x2_peak(datum_ibl_ctx *ctx, double *tflops)
  {
    if (!ctx || !tflops)
      return fail("datum_ibl_measure_fp32x2_peak: null argument");

    return measure_peak(ctx, tflops, true);
  }

  static int measure_peak(datum_ibl_ctx *ctx, double *tflops, bool packed)
  {

    DeviceGuard guard(ctx->device);

    const int threads = 256, blocks = ctx->sm_count * 8, iters = 1 << 15;

    cudaError_t err = ctx->sink.reserve((size_t)threads * blocks);
    if (err != cudaSuccess)
      return fail_cuda("cudaMalloc(sink)", err);

    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);

    double best = 0;

    for(int rep = 0; rep < 5 && err == cudaSuccess; ++rep)
    {
      cudaEventRecord(e0, ctx->stream);
      err = packed ? ibl::launch_fma2_peak(ctx->sink.ptr, blocks, threads, iters, ctx->stream) : ibl::launch_fma_peak(ctx->sink.ptr, blocks, threads, iters, ctx->stream);
      cudaEventRecord(e1, ctx->stream);
      ctx->launches += 1;

      if (err == cudaSuccess)
        err = cudaEventSynchronize(e1);

      float ms = 0;
      if (err == cudaSuccess)
        err = cudaEventElapsedTime(&ms, e0, e1);

      if (err == cudaSuccess && rep > 0 && ms > 0) // rep 0 warms up
      {
        double flops = 2.0 * 16.0 * (double)iters * threads * blocks;
        best = std::max(best, flops / (ms * 1e-3) / 1e12);
      }
    }

    cudaEventDestroy(e0);
    cudaEventDestroy(e1);

    if (err != cudaSuccess)
      return fail_cuda("datum_ibl_measure_fp32_peak", err);

    *tflops = best;
    return 0;
  }
}
