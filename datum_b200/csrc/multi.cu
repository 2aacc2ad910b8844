// datum_b200 — device-list entry points of libdatum_ibl_cuda: several GPUs of one node driven from ONE
// process (see include/datum_ibl_cuda.h, "device list").
//
// The reference's assetbuilder is a single process whose main thread calls image_buildmips_cube_ibl
// once per skybox (tools/assetbuilder.cpp:465, 486, write_core :778): to use more than one GPU it needs
// entry points that take a device list, not one process per GPU.  Everything here sits on top of the
// per-device entry points of cabi.cu:
//
//   one probe split (BASELINE config 3)   every device holds the payload; per level each device computes a
//       slab of rows with datum_ibl_prefilter_level_peers (rgbe) or datum_ibl_prefilter_level_float_peers
//       (F32, F16), whose kernel epilogue stores the slab into all payloads over NVLink (plain peer access
//       inside one process: cudaDeviceEnablePeerAccess, no IPC handles) and whose last CTA bumps the peers'
//       arrival counters; the streams wait on the counters.  The host thread only enqueues: all devices run
//       concurrently, nothing blocks until the end.
//   probe batches (config 4)              probe p on device p % ndev, one host thread per device around
//       datum_ibl_bake_probes or datum_ibl_bake_probes_float; no data-path exchange.
//   SH9 of one cube (config 5)            rows split, 28 partial sums per device added on the host.
//
// A device may appear more than once in the list (two contexts on one GPU): that is how the exchange
// path is exercised on a one-GPU test box.

#include "../../include/datum_ibl_cuda.h"

#include "cabi_internal.h"

#include <cuda_runtime.h>

#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

using ibl_cabi::fail;
using ibl_cabi::fail_cuda;

struct datum_ibl_multi
{
  std::vector<int> devices;
  std::vector<datum_ibl_ctx*> ctx;

  // one shared-probe payload per device: [flag block][chain], grow-only
  std::vector<unsigned char*> shared;
  size_t shared_bytes = 0;
  uint32_t epoch = 0;

  std::vector<unsigned char*> sh_staging;   // per device: 28 doubles + its slab of the cube
  std::vector<size_t> sh_staging_bytes;
};

namespace
{
  // levels of at most this many texels are computed by every device instead of being exchanged (dist.py MIN_SPLIT_TEXELS)
  const long long kMinSplitTexels = 6 * 16 * 16;

  struct DeviceScope
  {
    int previous = -1;
    explicit DeviceScope(int device) { cudaGetDevice(&previous); cudaSetDevice(device); }
    ~DeviceScope() { if (previous >= 0) cudaSetDevice(previous); }
  };

  void release_shared(datum_ibl_multi *m)
  {
    for(size_t d = 0; d < m->shared.size(); ++d)
      if (m->shared[d])
      {
        DeviceScope scope(m->devices[d]);
        cudaFree(m->shared[d]);
        m->shared[d] = nullptr;
      }
    m->shared_bytes = 0;
  }

  // chain bytes of every device's payload (rgbe words or float texels)
  int reserve_shared(datum_ibl_multi *m, size_t bytes)
  {
    if (bytes <= m->shared_bytes)
      return 0;

    // nothing of a previous bake may still be in flight towards the old buffers
    for(auto *c : m->ctx)
      if (datum_ibl_synchronize(c))
        return 1;

    release_shared(m);

    for(size_t d = 0; d < m->devices.size(); ++d)
    {
      DeviceScope scope(m->devices[d]);
      void *ptr = nullptr;
      cudaError_t err = cudaMalloc(&ptr, DATUM_IBL_PEER_FLAG_BYTES + bytes);
      if (err == cudaSuccess)
        err = cudaMemset(ptr, 0, DATUM_IBL_PEER_FLAG_BYTES);
      if (err != cudaSuccess)
      {
        if (ptr)
          cudaFree(ptr);
        release_shared(m);
        return fail_cuda("datum_ibl_multi: cudaMalloc(shared payload)", err);
      }
      m->shared[d] = static_cast<unsigned char*>(ptr);
    }

    m->shared_bytes = bytes;
    m->epoch = 0;
    return 0;
  }

  unsigned char *chain_of(datum_ibl_multi *m, size_t d) { return m->shared[d] + DATUM_IBL_PEER_FLAG_BYTES; }
  uint32_t *flags_of(datum_ibl_multi *m, size_t d) { return reinterpret_cast<uint32_t*>(m->shared[d]); }

  // One probe shared by the devices (BASELINE config 3), rgbe or float chains of `texel` bytes per texel: every
  // device holds the chain; per level each device computes a slab of rows and stores it into every chain (split),
  // or the whole level into its own.  bake_level(d, split, ws, hs, level, row_begin, row_end, src, dst, flags)
  // enqueues device d's part; dst[r] is the destination level in device r's chain, src the source level in d's,
  // flags the devices' flag blocks (epoch m->epoch).
  template<typename BakeLevel>
  int share_probe(datum_ibl_multi *m, const char *who, size_t texel, int width, int height, int levels, void *host, BakeLevel bake_level)
  {
    const int world = (int)m->devices.size();
    const std::string name = who;

    size_t texels = datum_ibl_chain_bytes(width, height, levels) / sizeof(uint32_t);
    size_t level0 = (size_t)width * height * 6;

    if (reserve_shared(m, texels * texel))
      return 1;

    // level 0: every device uploads ONE slice of it over its own PCIe link, then fetches the other slices from its
    // peers over NVLink (one upload to the first device and copies from there took 2.8 ms for the 100 MB of a
    // 2048^2 rgbe cube: 2 ms on one PCIe link + 0.8 ms out of one GPU's NVLink ports)
    std::vector<cudaStream_t> streams(world);
    for(int d = 0; d < world; ++d)
      streams[d] = (cudaStream_t)datum_ibl_stream(m->ctx[d]);

    // slices in texels, multiples of 64
    auto slice_begin = [&](size_t count, int d) { size_t per = ((count + world - 1) / world + 63) & ~(size_t)63; size_t b = per * (size_t)d; return b < count ? b : count; };

    std::vector<cudaEvent_t> uploaded(world, nullptr);
    int failed = 0;

    for(int d = 0; d < world && !failed; ++d)
    {
      DeviceScope scope(m->devices[d]);
      size_t begin = slice_begin(level0, d), end = slice_begin(level0, d + 1);
      cudaError_t err = cudaSuccess;
      if (end > begin)
        err = cudaMemcpyAsync(chain_of(m, d) + begin * texel, static_cast<unsigned char const*>(host) + begin * texel, (end - begin) * texel, cudaMemcpyHostToDevice, streams[d]);
      if (err == cudaSuccess)
        err = cudaEventCreateWithFlags(&uploaded[d], cudaEventDisableTiming);
      if (err == cudaSuccess)
        err = cudaEventRecord(uploaded[d], streams[d]);
      if (err != cudaSuccess)
        failed = fail_cuda((name + ": upload").c_str(), err);
    }

    for(int d = 0; d < world && !failed; ++d)
    {
      DeviceScope scope(m->devices[d]);
      for(int k = 1; k < world && !failed; ++k)
      {
        int s = (d + k) % world;      // every device starts with another peer
        size_t begin = slice_begin(level0, s), end = slice_begin(level0, s + 1);
        if (end <= begin)
          continue;
        cudaError_t err = cudaStreamWaitEvent(streams[d], uploaded[s], 0);
        if (err == cudaSuccess)
          err = cudaMemcpyPeerAsync(chain_of(m, d) + begin * texel, m->devices[d], chain_of(m, s) + begin * texel, m->devices[s], (end - begin) * texel, streams[d]);
        if (err != cudaSuccess)
          failed = fail_cuda((name + ": level 0 from peer").c_str(), err);
      }
    }

    std::vector<uint32_t*> flags(world);
    for(int d = 0; d < world; ++d)
      flags[d] = flags_of(m, d);

    // every device has level 0 before anybody stores level 1 into it, and nobody still reads the previous probe
    if (!failed)
    {
      m->epoch += 1;
      for(int d = 0; d < world && !failed; ++d)
        failed = datum_ibl_peer_barrier(m->ctx[d], d, world, flags.data(), m->epoch);
    }

    // tools/ibl.cpp:247-278, rows of every big level shared out
    size_t src_off = 0, dst_off = level0;
    int ws = width, hs = height;

    for(int level = 1; level < levels && !failed; ++level)
    {
      int wd = ws >> 1, hd = hs >> 1;
      int rows = 6 * hd;
      bool split = rows % world == 0 && (long long)rows * wd > kMinSplitTexels;

      if (split)
        m->epoch += 1;

      std::vector<void*> dst(world);
      for(int r = 0; r < world; ++r)
        dst[r] = chain_of(m, r) + dst_off * texel;

      for(int d = 0; d < world && !failed; ++d)
      {
        int per = rows / world;
        failed = bake_level(d, split, ws, hs, level, split ? d * per : 0, split ? (d + 1) * per : rows, chain_of(m, d) + src_off * texel, dst.data(), flags.data());
      }

      src_off = dst_off;
      dst_off += (size_t)wd * hd * 6;
      ws = wd;
      hs = hd;
    }

    // every device now holds the whole chain: each hands one slice of the baked levels back
    for(int d = 0; d < world && !failed; ++d)
    {
      DeviceScope scope(m->devices[d]);
      size_t begin = level0 + slice_begin(texels - level0, d), end = level0 + slice_begin(texels - level0, d + 1);
      if (end <= begin)
        continue;
      cudaError_t err = cudaMemcpyAsync(static_cast<unsigned char*>(host) + begin * texel, chain_of(m, d) + begin * texel, (end - begin) * texel, cudaMemcpyDeviceToHost, streams[d]);
      if (err != cudaSuccess)
        failed = fail_cuda((name + ": download").c_str(), err);
    }

    // also after a failure: nothing may stay in flight
    std::string first_error = failed ? datum_ibl_last_error() : "";
    for(int d = 0; d < world; ++d)
      if (datum_ibl_synchronize(m->ctx[d]) && !failed)
      {
        failed = 1;
        first_error = datum_ibl_last_error();
      }

    for(cudaEvent_t e : uploaded)
      if (e)
        cudaEventDestroy(e);

    return failed ? fail(first_error) : 0;
  }

  // Probe batches (config 4): probe p on device p % ndev; each device's share is one synchronous batched call
  // bake(ctx, n, payloads, sh) on its own host thread.  One device, or at most one probe: the first device's call.
  template<typename Bake>
  int shard_probes(datum_ibl_multi *m, const char *who, int count, void *const *payloads, float *sh, Bake bake)
  {
    if (!m || (count > 0 && !payloads))
      return fail(std::string(who) + ": null argument");
    if (count < 0)
      return fail(std::string(who) + ": bad count");

    const int world = (int)m->devices.size();

    if (world == 1 || count <= 1)
      return bake(m->ctx[0], count, payloads, sh);

    std::vector<std::vector<void*>> mine(world);
    for(int p = 0; p < count; ++p)
      mine[p % world].push_back(payloads[p]);

    std::vector<std::vector<float>> mine_sh(world);
    std::vector<std::string> errors(world);
    std::vector<std::thread> workers;

    for(int d = 0; d < world; ++d)
    {
      if (sh)
        mine_sh[d].resize(mine[d].size() * 27);

      workers.emplace_back([&, d] {
        if (mine[d].empty())
          return;
        if (bake(m->ctx[d], (int)mine[d].size(), mine[d].data(), sh ? mine_sh[d].data() : nullptr))
          errors[d] = datum_ibl_last_error();       // thread-local text of the worker
      });
    }

    for(auto &w : workers)
      w.join();

    for(int d = 0; d < world; ++d)
      if (!errors[d].empty())
        return fail(std::string(who) + ": device " + std::to_string(m->devices[d]) + ": " + errors[d]);

    for(int p = 0; sh && p < count; ++p)
      std::memcpy(sh + (size_t)p * 27, mine_sh[p % world].data() + (size_t)(p / world) * 27, 27 * sizeof(float));

    return 0;
  }
}

extern "C"
{
  int datum_ibl_multi_create(int ndev, int const *devices, datum_ibl_multi **out)
  {
    if (!out)
      return fail("datum_ibl_multi_create: null out pointer");
    *out = nullptr;
    if (ndev < 1 || ndev > DATUM_IBL_MAX_PEERS + 1 || !devices)
      return fail("datum_ibl_multi_create: 1 to 8 devices");

    datum_ibl_multi *m = new datum_ibl_multi;
    m->devices.assign(devices, devices + ndev);
    m->ctx.assign(ndev, nullptr);
    m->shared.assign(ndev, nullptr);
    m->sh_staging.assign(ndev, nullptr);
    m->sh_staging_bytes.assign(ndev, 0);

    for(int d = 0; d < ndev; ++d)
      if (datum_ibl_create(devices[d], &m->ctx[d]))
      {
        std::string why = datum_ibl_last_error();
        datum_ibl_multi_destroy(m);
        return fail("datum_ibl_multi_create: device " + std::to_string(devices[d]) + ": " + why);
      }

    // plain peer access between every pair of distinct devices (kernels of one store into the memory of the other)
    for(int a = 0; a < ndev; ++a)
      for(int b = 0; b < ndev; ++b)
      {
        if (devices[a] == devices[b])
          continue;

        int can = 0;
        cudaError_t err = cudaDeviceCanAccessPeer(&can, devices[a], devices[b]);
        if (err != cudaSuccess || !can)
        {
          datum_ibl_multi_destroy(m);
          return fail("datum_ibl_multi_create: devices " + std::to_string(devices[a]) + " and " + std::to_string(devices[b]) + " are not peers (NVLink/PCIe peer access is required to share a probe)");
        }

        DeviceScope scope(devices[a]);
        err = cudaDeviceEnablePeerAccess(devices[b], 0);
        if (err == cudaErrorPeerAccessAlreadyEnabled)
          cudaGetLastError();
        else if (err != cudaSuccess)
        {
          datum_ibl_multi_destroy(m);
          return fail_cuda("cudaDeviceEnablePeerAccess", err);
        }
      }

    *out = m;
    return 0;
  }

  void datum_ibl_multi_destroy(datum_ibl_multi *m)
  {
    if (!m)
      return;

    for(auto *c : m->ctx)
      if (c)
        datum_ibl_synchronize(c);

    release_shared(m);

    for(size_t d = 0; d < m->sh_staging.size(); ++d)
      if (m->sh_staging[d])
      {
        DeviceScope scope(m->devices[d]);
        cudaFree(m->sh_staging[d]);
      }

    for(auto *c : m->ctx)
      if (c)
        datum_ibl_destroy(c);

    delete m;
  }

  int datum_ibl_multi_device_count(datum_ibl_multi *m) { return m ? (int)m->devices.size() : 0; }

  datum_ibl_ctx *datum_ibl_multi_context(datum_ibl_multi *m, int index)
  {
    return (m && index >= 0 && index < (int)m->ctx.size()) ? m->ctx[index] : nullptr;
  }

  int datum_ibl_multi_buildmips_cube_ibl(datum_ibl_multi *m, int width, int height, int levels, int samples, void *bits)
  {
    if (!m || !bits)
      return fail("datum_ibl_multi_buildmips_cube_ibl: null argument");

    const int world = (int)m->devices.size();

    if (world == 1)
      return datum_ibl_buildmips_cube_ibl(m->ctx[0], width, height, levels, samples, bits);

    if (width < 1 || height < 1 || levels < 1 || levels > 16 || (width >> (levels - 1)) < 1 || (height >> (levels - 1)) < 1 || samples < 1)
      return fail("datum_ibl_multi_buildmips_cube_ibl: bad width/height/levels/samples");

    return share_probe(m, "datum_ibl_multi_buildmips_cube_ibl", sizeof(uint32_t), width, height, levels, bits,
      [&](int d, bool split, int ws, int hs, int level, int row_begin, int row_end, unsigned char *src, void *const *dst, uint32_t *const *flags)
      {
        if (!split)
          return datum_ibl_prefilter_level_device(m->ctx[d], reinterpret_cast<uint32_t const*>(src), ws, hs, level, levels, samples, row_begin, row_end, static_cast<uint32_t*>(dst[d]), nullptr);

        std::vector<uint32_t*> words(world);
        for(int r = 0; r < world; ++r)
          words[r] = static_cast<uint32_t*>(dst[r]);
        return datum_ibl_prefilter_level_peers(m->ctx[d], reinterpret_cast<uint32_t const*>(src), ws, hs, level, levels, samples, row_begin, row_end, d, world, words.data(), flags, m->epoch);
      });
  }

  int datum_ibl_multi_buildmips_cube_float(datum_ibl_multi *m, int format, int width, int height, int levels, int samples, void *chain)
  {
    if (!m || !chain)
      return fail("datum_ibl_multi_buildmips_cube_float: null argument");

    const int world = (int)m->devices.size();

    if (world == 1)
      return datum_ibl_buildmips_cube_float(m->ctx[0], format, width, height, levels, samples, chain);

    if (format != DATUM_IBL_FORMAT_F32 && format != DATUM_IBL_FORMAT_F16)
      return fail("datum_ibl_multi_buildmips_cube_float: unknown format " + std::to_string(format) + " (DATUM_IBL_FORMAT_F32 or DATUM_IBL_FORMAT_F16)");
    if (width < 1 || height < 1 || levels < 1 || levels > 16 || (width >> (levels - 1)) < 1 || (height >> (levels - 1)) < 1 || samples < 1 || samples > 4096)
      return fail("datum_ibl_multi_buildmips_cube_float: bad width/height/levels/samples");

    const size_t texel = format == DATUM_IBL_FORMAT_F16 ? 8 : 16;

    return share_probe(m, "datum_ibl_multi_buildmips_cube_float", texel, width, height, levels, chain,
      [&](int d, bool split, int ws, int hs, int level, int row_begin, int row_end, unsigned char *src, void *const *dst, uint32_t *const *flags)
      {
        if (!split)
          return datum_ibl_prefilter_level_float_device(m->ctx[d], format, src, ws, hs, level, levels, samples, row_begin, row_end, dst[d], nullptr);
        return datum_ibl_prefilter_level_float_peers(m->ctx[d], format, src, ws, hs, level, levels, samples, row_begin, row_end, d, world, dst, flags, m->epoch);
      });
  }

  int datum_ibl_multi_bake_probes(datum_ibl_multi *m, int count, int width, int height, int levels, int samples, void *const *bits, float *sh)
  {
    return shard_probes(m, "datum_ibl_multi_bake_probes", count, bits, sh, [&](datum_ibl_ctx *ctx, int n, void *const *mine, float *mine_sh)
    {
      return datum_ibl_bake_probes(ctx, n, width, height, levels, samples, mine, mine_sh);
    });
  }

  int datum_ibl_multi_bake_probes_float(datum_ibl_multi *m, int format, int count, int width, int height, int levels, int samples, void *const *chains, float *sh)
  {
    return shard_probes(m, "datum_ibl_multi_bake_probes_float", count, chains, sh, [&](datum_ibl_ctx *ctx, int n, void *const *mine, float *mine_sh)
    {
      return datum_ibl_bake_probes_float(ctx, format, n, width, height, levels, samples, mine, mine_sh);
    });
  }

  int datum_ibl_multi_project_sh9(datum_ibl_multi *m, void const *level0, int format, int width, int height, float *sh)
  {
    if (!m || !level0 || !sh)
      return fail("datum_ibl_multi_project_sh9: null argument");
    if (width < 1 || height < 1 || (format != DATUM_IBL_FORMAT_RGBE && format != DATUM_IBL_FORMAT_F32 && format != DATUM_IBL_FORMAT_F16))
      return fail("datum_ibl_multi_project_sh9: bad width/height/format");

    const int world = (int)m->devices.size();

    if (world == 1)
      return datum_ibl_project_sh9(m->ctx[0], level0, format, width, height, sh);

    const size_t texel = format == DATUM_IBL_FORMAT_RGBE ? 4 : (format == DATUM_IBL_FORMAT_F16 ? 8 : 16);
    const size_t cube_bytes = (size_t)6 * width * height * texel;
    const int rows = 6 * height;

    // Every device receives only its slab, placed where it would sit in the whole cube so that the
    // projection kernel's row addressing needs no offset; the 28 doubles of the result lead the buffer.
    std::vector<double> partial((size_t)world * 28, 0.0);
    int failed = 0;

    for(int d = 0; d < world && !failed; ++d)
    {
      int begin = (int)((long long)rows * d / world), end = (int)((long long)rows * (d + 1) / world);

      DeviceScope scope(m->devices[d]);
      cudaStream_t stream = (cudaStream_t)datum_ibl_stream(m->ctx[d]);

      size_t need = 28 * sizeof(double) + cube_bytes;
      cudaError_t err = cudaSuccess;
      if (m->sh_staging_bytes[d] < need)
      {
        if (m->sh_staging[d])
          cudaFree(m->sh_staging[d]);
        m->sh_staging[d] = nullptr;
        m->sh_staging_bytes[d] = 0;
        void *ptr = nullptr;
        err = cudaMalloc(&ptr, need);
        if (err == cudaSuccess)
        {
          m->sh_staging[d] = static_cast<unsigned char*>(ptr);
          m->sh_staging_bytes[d] = need;
        }
      }

      unsigned char *d_cube = m->sh_staging[d] + 28 * sizeof(double);
      size_t offset = (size_t)begin * width * texel, bytes = (size_t)(end - begin) * width * texel;

      if (err == cudaSuccess && bytes)
        err = cudaMemcpyAsync(d_cube + offset, static_cast<unsigned char const*>(level0) + offset, bytes, cudaMemcpyHostToDevice, stream);
      if (err != cudaSuccess)
      {
        failed = fail_cuda("datum_ibl_multi_project_sh9: upload", err);
        break;
      }

      failed = datum_ibl_sh9_partial_device(m->ctx[d], d_cube, format, width, height, begin, end, reinterpret_cast<double*>(m->sh_staging[d]));

      if (!failed)
      {
        err = cudaMemcpyAsync(partial.data() + (size_t)d * 28, m->sh_staging[d], 28 * sizeof(double), cudaMemcpyDeviceToHost, stream);
        if (err != cudaSuccess)
          failed = fail_cuda("datum_ibl_multi_project_sh9: download", err);
      }
    }

    std::string first_error = failed ? datum_ibl_last_error() : "";
    for(int d = 0; d < world; ++d)
      if (datum_ibl_synchronize(m->ctx[d]) && !failed)
      {
        failed = 1;
        first_error = datum_ibl_last_error();
      }

    if (failed)
      return fail(first_error);

    // slabs added in device order: the same bits whatever the timing
    double total[28] = {};
    for(int d = 0; d < world; ++d)
      for(int k = 0; k < 28; ++k)
        total[k] += partial[(size_t)d * 28 + k];

    datum_ibl_sh9_finish(total, sh);
    return 0;
  }

  // ---- the same with the device list passed per call (a process-wide handle per distinct list) ----

  namespace
  {
    datum_ibl_multi *cached_multi(int ndev, int const *devices)
    {
      static std::vector<datum_ibl_multi*> cache;
      static std::mutex guard;                       // the cache may be reached from several threads; a handle still serves one caller at a time
      std::lock_guard<std::mutex> lock(guard);

      if (ndev < 1 || !devices)
      {
        fail("device list: at least one device");
        return nullptr;
      }

      for(auto *m : cache)
        if ((int)m->devices.size() == ndev && std::memcmp(m->devices.data(), devices, sizeof(int) * ndev) == 0)
          return m;

      datum_ibl_multi *m = nullptr;
      if (datum_ibl_multi_create(ndev, devices, &m))
        return nullptr;

      cache.push_back(m);
      return m;
    }
  }

  int datum_ibl_buildmips_cube_ibl_devices(int ndev, int const *devices, int width, int height, int levels, int samples, void *bits)
  {
    datum_ibl_multi *m = cached_multi(ndev, devices);
    return m ? datum_ibl_multi_buildmips_cube_ibl(m, width, height, levels, samples, bits) : 1;
  }

  int datum_ibl_bake_probes_devices(int ndev, int const *devices, int count, int width, int height, int levels, int samples, void *const *bits, float *sh)
  {
    datum_ibl_multi *m = cached_multi(ndev, devices);
    return m ? datum_ibl_multi_bake_probes(m, count, width, height, levels, samples, bits, sh) : 1;
  }
}
