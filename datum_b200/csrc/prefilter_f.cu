// datum_b200 — GGX prefilter of one level of a FLOAT cube chain, RGBA16F or RGBA32F (sm_100a).
//
// The same level arithmetic as prefilter_dn.cu (tools/ibl.cpp:160-187, 247-278 with the non-seamless
// per-face bilinear Sampler of ibl.cpp:34-88), but a tap is read as the float value the chain stores
// instead of through rgbe_decode, and a level is stored as floats: no 9-bit re-quantisation between
// levels.  Two kernels:
//
//   * prefilter_float_pair_kernel: the projective pair kernel of prefilter_dn.cu (prefilter_dp_kernel,
//     PROJ) with the same sector tables, frame planes, 8x4 tiles and per-SM tile queues.  A lane's
//     footprint comes from a record of the source level (prefilter_f.h): RGBA16F texels verbatim (32 B)
//     or rgb fp32 (48 B).  The rgbe tap decode is replaced by half -> fp32 conversion (F16) or nothing
//     (F32); weights stay fp32, so every tap product is the reference's up to summation order.
//   * prefilter_float_tail_kernel: one CTA per texel, lanes are samples (prefilter_tail_kernel), the four
//     texels of a footprint read straight from the source level.  Small slabs, levels narrower than a
//     tile, and every source the pair kernel cannot address (!proj_usable: odd sizes, faces above 2048^2).
//
// The pair kernel shares its device helpers with prefilter_dn.cu (prefilter_pair.cuh): packed fp32 ops, pair
// entries, projective footprint coordinates, tile hand-out, per-tile frame and same-face band count, CTA
// reduction.  The launchers share resident_ctas, plan_tiles, the slab-size classes and tail_warps (prefilter.h).
//
// Batches (datum_ibl_bake_probes_float): the record pass, the pair kernel and the tail kernel also compute the
// same level of several chains in one launch, like the rgbe kernels, in instantiations of their own (BATCH):
// the single-probe kernels compile none of the batch code.  Launch shapes that decide the order of the sums
// (warps per tile, warps per texel) follow ONE probe's slab, so every probe of a batch gets the bytes of a
// single call; only the tile queues and the grid follow the whole launch.
//
// Shared probes (datum_ibl_prefilter_level_float_peers, datum_ibl_multi_buildmips_cube_float): one probe split
// over up to 8 GPUs by rows, like the rgbe chain's.  The pair kernel and the tail kernel (both forms of PROJ)
// have instantiations of their own (SHARED) whose epilogue stores every texel (8 B for F16, 16 B for F32) into
// this GPU's chain and into every peer's over NVLink, and whose CTAs then run signal_peers_when_last
// (prefilter_pair.cuh): the last one to finish bumps the peers' arrival counters.  One chain, no dst_f32.

#include "prefilter.h"
#include "prefilter_f.h"
#include "prefilter_pair.cuh"
#include "ibl_math.cuh"

#include <cuda_runtime.h>

namespace ibl
{
  namespace
  {
    template<int FMT> struct RecordOf { typedef F32Record type; };
    template<> struct RecordOf<kFloatFormatF16> { typedef F16Record type; };

    // ---- records --------------------------------------------------------------------------

    // BATCH: blockIdx.y = probe, source levels src_stride texels apart, their records back to back
    template<int FMT, bool BATCH>
    __device__ __forceinline__ void build_float_records(void const *__restrict__ src, void *__restrict__ rec, int ws, int hs, size_t src_stride, int *__restrict__ counters, int ncounters)
    {
      // the prefilter launch that follows on the stream takes its tiles from these queues
      if (blockIdx.x == 0 && (!BATCH || blockIdx.y == 0))
        for(int i = threadIdx.x; i < ncounters; i += blockDim.x)
          counters[i] = 0;

      const uint32_t level = 6u * (uint32_t)ws * (uint32_t)hs;

      if (BATCH)
      {
        src = static_cast<unsigned char const*>(src) + (size_t)blockIdx.y * src_stride * float_texel_bytes(FMT);
        rec = static_cast<unsigned char*>(rec) + (size_t)blockIdx.y * level * sizeof(typename RecordOf<FMT>::type);
      }

      for(uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x; idx < level; idx += gridDim.x * blockDim.x)
      {
        uint32_t i = idx % (uint32_t)ws;
        uint32_t j = (idx / (uint32_t)ws) % (uint32_t)hs;
        uint32_t right = (i + 1 < (uint32_t)ws) ? 1u : 0u;
        uint32_t down = (j + 1 < (uint32_t)hs) ? (uint32_t)ws : 0u;
        const uint32_t tap[4] = { idx, idx + right, idx + down, idx + down + right };

        if (FMT == kFloatFormatF16)
        {
          uint2 const *s = reinterpret_cast<uint2 const*>(src);
          uint2 t0 = __ldg(s + tap[0]), t1 = __ldg(s + tap[1]), t2 = __ldg(s + tap[2]), t3 = __ldg(s + tap[3]);
          uint4 *r = reinterpret_cast<uint4*>(rec) + 2 * (size_t)idx;
          r[0] = make_uint4(t0.x, t0.y, t1.x, t1.y);
          r[1] = make_uint4(t2.x, t2.y, t3.x, t3.y);
        }
        else
        {
          float4 const *s = reinterpret_cast<float4 const*>(src);
          float4 t0 = __ldg(s + tap[0]), t1 = __ldg(s + tap[1]), t2 = __ldg(s + tap[2]), t3 = __ldg(s + tap[3]);
          float4 *r = reinterpret_cast<float4*>(rec) + 3 * (size_t)idx;
          r[0] = make_float4(t0.x, t0.y, t0.z, t1.x);
          r[1] = make_float4(t1.y, t1.z, t2.x, t2.y);
          r[2] = make_float4(t2.z, t3.x, t3.y, t3.z);
        }
      }
    }

    // one chain, and the same level of several chains (separate kernels: the single-probe one compiles none of
    // the batch code)
    template<int FMT>
    __global__ void __launch_bounds__(256) build_float_records_kernel(void const *__restrict__ src, void *__restrict__ rec, int ws, int hs, int *__restrict__ counters, int ncounters)
    {
      build_float_records<FMT, false>(src, rec, ws, hs, 0, counters, ncounters);
    }

    template<int FMT>
    __global__ void __launch_bounds__(256) build_float_records_batch_kernel(void const *__restrict__ src, void *__restrict__ rec, int ws, int hs, size_t src_stride, int *__restrict__ counters, int ncounters)
    {
      build_float_records<FMT, true>(src, rec, ws, hs, src_stride, counters, ncounters);
    }

    // ---- taps -----------------------------------------------------------------------------

    // the four texels' rgb of a footprint record: c[k][channel]
    __device__ __forceinline__ void load_footprint(F16Record const *rec, float c[4][3])
    {
      uint4 const *q = reinterpret_cast<uint4 const*>(rec);
      uint4 lo = __ldg(q), hi = __ldg(q + 1);
      const uint32_t w[8] = { lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w };
      #pragma unroll
      for(int k = 0; k < 4; ++k)
      {
        c[k][0] = half_to_float(w[2*k] & 0xFFFFu);
        c[k][1] = half_to_float(w[2*k] >> 16);
        c[k][2] = half_to_float(w[2*k + 1] & 0xFFFFu);
      }
    }

    __device__ __forceinline__ void load_footprint(F32Record const *rec, float c[4][3])
    {
      float4 const *q = reinterpret_cast<float4 const*>(rec);
      float4 a = __ldg(q), b = __ldg(q + 1), d = __ldg(q + 2);
      c[0][0] = a.x; c[0][1] = a.y; c[0][2] = a.z;
      c[1][0] = a.w; c[1][1] = b.x; c[1][2] = b.y;
      c[2][0] = b.z; c[2][1] = b.w; c[2][2] = d.x;
      c[3][0] = d.y; c[3][1] = d.z; c[3][2] = d.w;
    }

    // one texel of the source level itself (tail kernel)
    template<int FMT>
    __device__ __forceinline__ void load_texel(void const *src, uint32_t idx, float c[3])
    {
      if (FMT == kFloatFormatF16)
      {
        uint2 t = __ldg(reinterpret_cast<uint2 const*>(src) + idx);
        c[0] = half_to_float(t.x & 0xFFFFu);
        c[1] = half_to_float(t.x >> 16);
        c[2] = half_to_float(t.y & 0xFFFFu);
      }
      else
      {
        float4 t = __ldg(reinterpret_cast<float4 const*>(src) + idx);
        c[0] = t.x; c[1] = t.y; c[2] = t.z;
      }
    }

    // idx = raw index bits of both samples (what `base` has been moved back by), du/dv = fraction - 0.5;
    // the weights of footprint_weights_diff (ibl.cpp:40 times the sample weight), taps as floats
    template<typename R>
    __device__ __forceinline__ void gather_pair(R const *base, uint32_t idx_a, uint32_t idx_b, f32x2 du, f32x2 dv, PairEntry const &e, Sums &acc)
    {
      float ca[4][3], cb[4][3];
      load_footprint(base + idx_a, ca);
      load_footprint(base + idx_b, cb);

      f32x2 u0 = add2(neg2(du), bcast2(0.5f));
      f32x2 v0 = fma2(neg2(dv), e.lz, e.wh);
      f32x2 v1 = fma2(dv, e.lz, e.wh);
      f32x2 p00 = mul2(u0, v0);
      f32x2 p01 = mul2(u0, v1);

      float wa[4], wb[4];
      unpack2(p00, wa[0], wb[0]);
      unpack2(add2(v0, neg2(p00)), wa[1], wb[1]);
      unpack2(p01, wa[2], wb[2]);
      unpack2(add2(v1, neg2(p01)), wa[3], wb[3]);

      #pragma unroll
      for(int k = 0; k < 4; ++k)
      {
        acc.rg = fma2(pack2(ca[k][0], ca[k][1]), bcast2(wa[k]), acc.rg);
        acc.rg = fma2(pack2(cb[k][0], cb[k][1]), bcast2(wb[k]), acc.rg);
        acc.bb = fma2(pack2(ca[k][2], cb[k][2]), pack2(wa[k], wb[k]), acc.bb);
      }
    }

    // frame rows face-local and folded; `base` = records of the texel's face, moved back by kMagicBits
    template<typename R>
    __device__ __forceinline__ void pair_same_face(PrefilterFloatParams const &p, Frame const &t, R const *base, PairEntry const &e, Sums &acc)
    {
      uint32_t ia, ib;
      f32x2 du, dv;
      pair_taps_same_face(p.geom, t, e, ia, ib, du, dv);
      gather_pair(base, ia, ib, du, dv, e, acc);
    }

    // frame rows in world coordinates; `base` = records moved back by geom.bias_general
    template<typename R>
    __device__ __forceinline__ void pair_general(PrefilterFloatParams const &p, Frame const &t, R const *base, PairEntry const &e, Sums &acc)
    {
      uint32_t ia, ib;
      f32x2 du, dv;
      pair_taps_general(p.geom, t, e, ia, ib, du, dv);
      gather_pair(base, ia, ib, du, dv, e, acc);
    }

    // ---- epilogue ---------------------------------------------------------------------------

    template<int FMT>
    __device__ __forceinline__ void store_texel(PrefilterFloatParams const &p, size_t o, float r, float g, float b)
    {
      if (FMT == kFloatFormatF16)
      {
        uint32_t hr = float_to_half_rn(r), hg = float_to_half_rn(g), hb = float_to_half_rn(b);
        reinterpret_cast<uint2*>(p.dst)[o] = make_uint2(hg << 16 | hr, 0x3C00u << 16 | hb);
        if (p.dst_f32)
        {
          p.dst_f32[3*o + 0] = r;
          p.dst_f32[3*o + 1] = g;
          p.dst_f32[3*o + 2] = b;
        }
      }
      else
      {
        reinterpret_cast<float4*>(p.dst)[o] = make_float4(r, g, b, 1.0f);
        if (p.dst_f32)
        {
          p.dst_f32[3*o + 0] = r;
          p.dst_f32[3*o + 1] = g;
          p.dst_f32[3*o + 2] = b;
        }
      }
    }

    // one probe shared by several GPUs: the texel goes to this GPU's chain and, over NVLink, into every peer's
    template<int FMT>
    __device__ __forceinline__ void store_texel_peers(PrefilterFloatParams const &p, size_t o, float r, float g, float b)
    {
      if (FMT == kFloatFormatF16)
      {
        uint32_t hr = float_to_half_rn(r), hg = float_to_half_rn(g), hb = float_to_half_rn(b);
        const uint2 texel = make_uint2(hg << 16 | hr, 0x3C00u << 16 | hb);
        reinterpret_cast<uint2*>(p.dst)[o] = texel;
        for(int k = 0; k < p.peers; ++k)
          reinterpret_cast<uint2*>(p.peer_dst[k])[o] = texel;
      }
      else
      {
        const float4 texel = make_float4(r, g, b, 1.0f);
        reinterpret_cast<float4*>(p.dst)[o] = texel;
        for(int k = 0; k < p.peers; ++k)
          reinterpret_cast<float4*>(p.peer_dst[k])[o] = texel;
      }
    }

    // ---- the pair kernel ------------------------------------------------------------------------
    //
    // CTA = NW warps sharing one 8x4 tile; warp w reads azimuth sector w of every band of the sector table,
    // its leading bands without face selection as long as they provably stay on the texel's face.
    // BATCH: the same level of p.probes chains, tiles numbered probe by probe (prefilter_dp_kernel's batches).
    // SHARED: one probe shared by several GPUs, a slab stored into every peer's chain and the peers told when it
    // is complete (prefilter_dp_kernel's peer stores).  The single-probe instantiations compile none of either.
    template<int FMT, int NW, int MINB, bool SMEM_TABLE, bool QUEUES, bool BATCH = false, bool SHARED = false>
    __global__ void __launch_bounds__(32 * NW, MINB) prefilter_float_pair_kernel(PrefilterFloatParams p)
    {
      typedef typename RecordOf<FMT>::type R;

      extern __shared__ float4 smem[];
      constexpr int SECTORS = NW == 8 ? 1 : 0;
      const int bands = p.sector_bands[SECTORS];
      constexpr int BAND = kSectorShare * NW;
      const int padded = bands * BAND;
      float4 *s_table = smem;
      float *s_red = reinterpret_cast<float*>(smem + (SMEM_TABLE ? padded : 0));
      int *s_tile = reinterpret_cast<int*>(s_red + NW * 3 * 32);

      const int tid = threadIdx.x;
      const int lane = tid & 31;
      const int warp = tid >> 5;

      if (SMEM_TABLE)
      {
        for(int i = tid; i < padded; i += 32 * NW)
          s_table[i] = __ldg(p.table_sector[SECTORS] + i);
        __syncthreads();
      }

      float4 const *table = SMEM_TABLE ? s_table : p.table_sector[SECTORS];

      uint32_t smid;
      asm("mov.u32 %0, %%smid;" : "=r"(smid));

      constexpr int PER = BAND / NW;
      constexpr int PAIRS = PER / 2;
      constexpr int BAND_UNROLL = PAIRS >= 2 ? 1 : 2;

      R const *biased = opaque(reinterpret_cast<R const*>(p.records) - (size_t)kMagicBits);

      for(int it = 0; ; ++it)
      {
        int tile;
        if (QUEUES)
        {
          if (tid == 0)
            *s_tile = next_tile_plain(p, smid);
          __syncthreads();
          tile = *s_tile;

          if (tile < 0)
          {
            __syncthreads();
            if (warp == 0)
            {
              int stolen = steal_tile(p.counters, p.queues, p.chunk, smid, lane);
              if (lane == 0)
                *s_tile = stolen;
            }
            __syncthreads();
            tile = *s_tile;
          }
        }
        else
        {
          tile = (int)blockIdx.x + it * (int)gridDim.x;
          if (tile >= p.tiles)
            tile = -1;
        }

        if (tile < 0)
          break;

        // a batch: which probe, and the tile within that probe's slab
        int probe = 0, ltile = tile;
        if (BATCH)
        {
          probe = tile / p.tiles_per_probe;
          ltile = tile - probe * p.tiles_per_probe;
        }

        int x, row;
        bool valid = tile_texel(p, ltile, lane, x, row);

        if (__ballot_sync(0xffffffffu, valid) == 0u)
        {
          if (QUEUES)
            __syncthreads();
          continue;
        }

        if (!valid) { x = p.wd >> 1; row = (p.row_begin / p.hd) * p.hd + (p.hd >> 1); }

        int face = row / p.hd;

        Frame st;
        int n_same, n_same_second;
        tile_frame_bands<NW, 1>(p, x, row, warp, lane, bands, st, n_same, n_same_second);

        Sums acc;
        acc.rg = 0ull;
        acc.bb = 0ull;

        float4 const *tw = table + warp * PER;

        // this probe's records (a batch: the probes' records back to back)
        R const *biased_probe = BATCH ? opaque(biased + (size_t)probe * p.record_stride) : biased;

        {
          R const *base = opaque(biased_probe + (size_t)face * p.geom.face_size);

          #pragma unroll BAND_UNROLL
          for(int band = 0; band < n_same; ++band)
          {
            #pragma unroll
            for(int k = 0; k < PAIRS; ++k)
              pair_same_face(p, st, base, load_pair<SMEM_TABLE>(tw + band * BAND + 2 * k), acc);
          }
        }

        if (n_same < bands)
        {
          st.T = from_face_local(face, unfold_face_row(p.geom, st.T));
          st.B = from_face_local(face, unfold_face_row(p.geom, st.B));
          st.N = from_face_local(face, unfold_face_row(p.geom, st.N));

          R const *general = opaque(biased_probe + (size_t)(kMagicBits - p.geom.bias_general));

          #pragma unroll BAND_UNROLL
          for(int band = n_same; band < bands; ++band)
          {
            #pragma unroll
            for(int k = 0; k < PAIRS; ++k)
              pair_general(p, st, general, load_pair<SMEM_TABLE>(tw + band * BAND + 2 * k), acc);
          }
        }

        store_warp_sums(acc, s_red, warp, lane);
        __syncthreads();

        if (warp == 0)
        {
          float sum[3];
          add_warp_sums<NW>(s_red, lane, sum);

          if (valid)
          {
            if (SHARED)
              store_texel_peers<FMT>(p, (size_t)row * p.wd + x, sum[0] * p.norm, sum[1] * p.norm, sum[2] * p.norm);
            else
              store_texel<FMT>(p, (size_t)row * p.wd + x + (BATCH ? (size_t)probe * p.dst_stride : (size_t)0), sum[0] * p.norm, sum[1] * p.norm, sum[2] * p.norm);
          }
        }

        __syncthreads();
      }

      if (SHARED)
        signal_peers_when_last(p.signal);
    }

    // ---- the tail kernel: one CTA per texel, lanes are samples (prefilter_tail_kernel) ----------------
    // BATCH: the same level of p.probes chains, blockIdx.x runs over the texels probe by probe (batches run only
    // where every source is proj_usable, prefilter_batchable: PROJ).  SHARED: one probe's slab stored into every
    // peer's chain, the peers told when it is complete (either form of PROJ: odd sources and faces above 2048^2).
    template<int FMT, int NW, bool PROJ, bool BATCH = false, bool SHARED = false>
    __global__ void __launch_bounds__(32 * NW) prefilter_float_tail_kernel(PrefilterFloatParams p)
    {
      __shared__ float s_red[NW][3];
      __shared__ float s_frame[9];

      const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

      int texel = blockIdx.x, probe = 0;
      if (BATCH)
      {
        probe = texel / p.texels_per_probe;
        texel -= probe * p.texels_per_probe;
      }
      void const *src = BATCH ? static_cast<unsigned char const*>(p.src) + (size_t)probe * p.src_stride * float_texel_bytes(FMT) : p.src;

      const int row = p.row_begin + texel / p.wd;
      const int x = texel - (texel / p.wd) * p.wd;
      const int face = row / p.hd;
      const int y = row - face * p.hd;

      if (p.world_frames)
      {
        if (threadIdx.x < 9)
          s_frame[threadIdx.x] = __ldg(p.world_frames + (size_t)threadIdx.x * ((size_t)6 * p.hd * p.wd) + ((size_t)row * p.wd + x));
      }
      else if (threadIdx.x == 0)
      {
        Vec3f n = texel_normal(p.quats[face], x, y, p.wd, p.hd);
        Vec3f t, b;
        tangent_frame(n, t, b);
        s_frame[0] = t.x; s_frame[1] = t.y; s_frame[2] = t.z;
        s_frame[3] = b.x; s_frame[4] = b.y; s_frame[5] = b.z;
        s_frame[6] = n.x; s_frame[7] = n.y; s_frame[8] = n.z;
      }

      __syncthreads();

      const Vec3f T = { s_frame[0], s_frame[1], s_frame[2] };
      const Vec3f B = { s_frame[3], s_frame[4], s_frame[5] };
      const Vec3f N = { s_frame[6], s_frame[7], s_frame[8] };

      float acc[3] = { 0.0f, 0.0f, 0.0f };

      for(int s = threadIdx.x; s < p.table_count; s += 32 * NW)
      {
        float4 e = __ldg((PROJ ? p.table_proj : p.table) + s);

        float du, dv, w[4];
        uint32_t idx;                 // top-left texel of the footprint; i <= ws-2, j <= hs-2

        if (PROJ)
        {
          float Lx = fmaf(e.x, T.x, fmaf(e.y, B.x, N.x));
          float Ly = fmaf(e.x, T.y, fmaf(e.y, B.y, N.y));
          float Lz = fmaf(e.x, T.z, fmaf(e.y, B.z, N.z));

          uint32_t f;
          idx = cube_footprint_proj(p.geom, Lx, Ly, Lz, du, dv, f);
          idx += f * p.geom.face_size - p.geom.bias_general;
          footprint_weights_diff(du, dv, e.w, e.z, w);
        }
        else
        {
          float Lx = fmaf(e.z, N.x, fmaf(e.y, B.x, e.x * T.x));
          float Ly = fmaf(e.z, N.y, fmaf(e.y, B.y, e.x * T.y));
          float Lz = fmaf(e.z, N.z, fmaf(e.y, B.z, e.x * T.z));

          idx = cube_footprint(p.geom, Lx, Ly, Lz, du, dv);
          footprint_weights(du, dv, e.w, e.z, w);
        }

        const uint32_t tap[4] = { idx, idx + 1, idx + (uint32_t)p.geom.ws, idx + (uint32_t)p.geom.ws + 1 };
        #pragma unroll
        for(int k = 0; k < 4; ++k)
        {
          float c[3];
          load_texel<FMT>(src, tap[k], c);
          float_accumulate_tap(c[0], c[1], c[2], w[k], acc);
        }
      }

      #pragma unroll
      for(int c = 0; c < 3; ++c)
      {
        float v = acc[c];
        #pragma unroll
        for(int offset = 16; offset > 0; offset >>= 1)
          v += __shfl_down_sync(0xffffffffu, v, offset);
        if (lane == 0)
          s_red[warp][c] = v;
      }

      __syncthreads();

      if (threadIdx.x == 0)
      {
        float sum[3] = { 0.0f, 0.0f, 0.0f };
        #pragma unroll
        for(int w = 0; w < NW; ++w)
        {
          #pragma unroll
          for(int c = 0; c < 3; ++c)
            sum[c] += s_red[w][c];
        }

        if (SHARED)
          store_texel_peers<FMT>(p, (size_t)row * p.wd + x, sum[0] * p.norm, sum[1] * p.norm, sum[2] * p.norm);
        else
          store_texel<FMT>(p, (size_t)row * p.wd + x + (BATCH ? (size_t)probe * p.dst_stride : (size_t)0), sum[0] * p.norm, sum[1] * p.norm, sum[2] * p.norm);
      }

      if (SHARED)
        signal_peers_when_last(p.signal);
    }

    template<int FMT, int NW, int MINB, bool SMEM_TABLE, bool QUEUES, bool BATCH, bool SHARED>
    cudaError_t launch_pair(PrefilterFloatParams p, int sm_count, cudaStream_t stream)
    {
      auto kernel = prefilter_float_pair_kernel<FMT, NW, MINB, SMEM_TABLE, QUEUES, BATCH, SHARED>;

      const int table_bands = p.sector_bands[NW == 8 ? 1 : 0];
      size_t smem = (SMEM_TABLE ? (size_t)table_bands * kSectorShare * NW * sizeof(float4) : 0) + (size_t)NW * 3 * 32 * sizeof(float) + sizeof(int);

      int grid = 0;
      cudaError_t err = plan_tiles(p, kernel, 32 * NW, smem, p.probes, sm_count, &grid);
      if (err != cudaSuccess)
        return err;
      p.tiles_per_probe = p.tiles / p.probes;

      kernel<<<grid, 32 * NW, smem, stream>>>(p);
      return cudaGetLastError();
    }

    template<int FMT, int NW, int MINB, bool QUEUES, bool BATCH, bool SHARED>
    cudaError_t launch_pair_table(PrefilterFloatParams const &p, int sm_count, cudaStream_t stream)
    {
      return p.table_count > kBigTableEntries ? launch_pair<FMT, NW, MINB, false, QUEUES, BATCH, SHARED>(p, sm_count, stream) : launch_pair<FMT, NW, MINB, true, QUEUES, BATCH, SHARED>(p, sm_count, stream);
    }

    // The slab-size classes of launch_prefilter_dn.  Warps per tile follow ONE probe's slab (they decide the
    // order of the sums: a batch must give the bytes of single calls), the tile queues the whole launch.
    template<int FMT, bool BATCH, bool SHARED>
    cudaError_t launch_pair_shape(PrefilterFloatParams const &p, int sm_count, cudaStream_t stream)
    {
      const size_t texels = (size_t)(p.row_end - p.row_begin) * p.wd;

      if (texels >= kFourWarpTexels)
        return launch_pair_table<FMT, 4, 8, true, BATCH, SHARED>(p, sm_count, stream);
      if (texels * (size_t)p.probes >= kQueuedTexels)
        return launch_pair_table<FMT, 8, 4, true, BATCH, SHARED>(p, sm_count, stream);
      return launch_pair_table<FMT, 8, 4, false, BATCH, SHARED>(p, sm_count, stream);
    }

    bool shared_probe(PrefilterFloatParams const &p) { return p.peers > 0 || p.signal.count > 0; }

    template<int FMT>
    cudaError_t launch_pair_for(PrefilterFloatParams const &p, int sm_count, cudaStream_t stream)
    {
      if (p.probes > 1)
        return launch_pair_shape<FMT, true, false>(p, sm_count, stream);
      return shared_probe(p) ? launch_pair_shape<FMT, false, true>(p, sm_count, stream) : launch_pair_shape<FMT, false, false>(p, sm_count, stream);
    }

    template<int NW, int FMT, bool PROJ>
    void launch_tail(PrefilterFloatParams const &p, int grid, cudaStream_t stream)
    {
      if (p.probes > 1)
        prefilter_float_tail_kernel<FMT, NW, true, true><<<grid, 32 * NW, 0, stream>>>(p);
      else if (shared_probe(p))
        prefilter_float_tail_kernel<FMT, NW, PROJ, false, true><<<grid, 32 * NW, 0, stream>>>(p);
      else
        prefilter_float_tail_kernel<FMT, NW, PROJ><<<grid, 32 * NW, 0, stream>>>(p);
    }

    // warps per texel (tail_warps) chosen from ONE probe's texels also when a launch carries several
    template<int FMT, bool PROJ>
    cudaError_t launch_tail_for(PrefilterFloatParams const &p, int texels, cudaStream_t stream)
    {
      const int grid = texels * p.probes;
      switch (tail_warps(texels, p.table_count))
      {
        case 4: launch_tail<4, FMT, PROJ>(p, grid, stream); break;
        case 8: launch_tail<8, FMT, PROJ>(p, grid, stream); break;
        case 16: launch_tail<16, FMT, PROJ>(p, grid, stream); break;
        default: launch_tail<32, FMT, PROJ>(p, grid, stream); break;
      }
      return cudaGetLastError();
    }
  }

  cudaError_t launch_build_float_records(int format, void const *src, void *records, int ws, int hs, int probes, size_t src_stride, int *counters, int ncounters, int sm_count, cudaStream_t stream)
  {
    if (probes < 1)
      probes = 1;

    size_t level = (size_t)6 * ws * hs;
    size_t blocks = (level + 255) / 256;
    size_t cap = ((size_t)sm_count * 8 + probes - 1) / probes;
    int grid = (int)(blocks < cap ? blocks : cap);
    if (grid < 1)
      grid = 1;

    const dim3 cubes(grid, probes);
    if (format == kFloatFormatF16 && probes == 1)
      build_float_records_kernel<kFloatFormatF16><<<grid, 256, 0, stream>>>(src, records, ws, hs, counters, ncounters);
    else if (format == kFloatFormatF32 && probes == 1)
      build_float_records_kernel<kFloatFormatF32><<<grid, 256, 0, stream>>>(src, records, ws, hs, counters, ncounters);
    else if (format == kFloatFormatF16)
      build_float_records_batch_kernel<kFloatFormatF16><<<cubes, 256, 0, stream>>>(src, records, ws, hs, src_stride, counters, ncounters);
    else if (format == kFloatFormatF32)
      build_float_records_batch_kernel<kFloatFormatF32><<<cubes, 256, 0, stream>>>(src, records, ws, hs, src_stride, counters, ncounters);
    else
      return cudaErrorInvalidValue;
    return cudaGetLastError();
  }

  cudaError_t launch_prefilter_float(PrefilterFloatParams const &params, int sm_count, cudaStream_t stream)
  {
    PrefilterFloatParams p = params;
    if (p.row_end <= p.row_begin || p.wd <= 0)
      return cudaSuccess;
    if (!proj_usable(p.geom.ws, p.geom.hs) || !p.frames || !p.table_sector[0] || !p.table_sector[1])
      return cudaErrorInvalidValue;
    if (p.probes < 1)
      p.probes = 1;
    if (p.probes > 1 && p.dst_f32)
      return cudaErrorNotSupported;       // batches store the format's texels only
    if (shared_probe(p) && (p.probes > 1 || p.dst_f32))
      return cudaErrorNotSupported;       // a shared probe: one chain, texels of the format

    if (p.format == kFloatFormatF16)
      return launch_pair_for<kFloatFormatF16>(p, sm_count, stream);
    if (p.format == kFloatFormatF32)
      return launch_pair_for<kFloatFormatF32>(p, sm_count, stream);
    return cudaErrorInvalidValue;
  }

  cudaError_t launch_prefilter_float_tail(PrefilterFloatParams const &params, cudaStream_t stream)
  {
    PrefilterFloatParams p = params;
    int texels = (p.row_end - p.row_begin) * p.wd;
    if (texels <= 0)
      return cudaSuccess;

    if (p.probes < 1)
      p.probes = 1;
    p.texels_per_probe = texels;

    const bool proj = proj_usable(p.geom.ws, p.geom.hs);
    if (p.probes > 1 && (p.dst_f32 || !proj))
      return cudaErrorNotSupported;       // batches: texels of the format, proj_usable sources (prefilter_batchable)
    if (shared_probe(p) && (p.probes > 1 || p.dst_f32))
      return cudaErrorNotSupported;       // a shared probe: one chain, texels of the format

    if (p.format == kFloatFormatF16)
      return proj ? launch_tail_for<kFloatFormatF16, true>(p, texels, stream) : launch_tail_for<kFloatFormatF16, false>(p, texels, stream);
    if (p.format == kFloatFormatF32)
      return proj ? launch_tail_for<kFloatFormatF32, true>(p, texels, stream) : launch_tail_for<kFloatFormatF32, false>(p, texels, stream);
    return cudaErrorInvalidValue;
  }
}
