// datum_b200 — GGX prefilter of one cube-map mip level, "denormal mantissa" kernel (sm_100a).
//
// Replaces the triple loop of tools/ibl.cpp:263-272 and the per-texel sample loop of
// tools/ibl.cpp:160-187 (reference paths relative to /root/reference).  This is the kernel the
// library uses for every slab of more than kTailTexels texels; smaller slabs and levels narrower
// than a tile go to prefilter_tail_kernel below.
//
// What one bilinear tap costs decides the speed of this loop (profiles/): the first kernel
// (prefilter.cu) turned each 9-bit mantissa into a float with shift + mask logic, six ALU-pipe ops
// per tap on a half-rate pipe.  Here
//
//   * a quad record still holds the four E5B9G9R9 words of a footprint (16 bytes, one LDG.128),
//     re-laid as r<<23 | g<<14 | b<<5 | E (pack_dn_word);
//   * a mantissa is used as the fp32 number its bits spell under a zero exponent field: a
//     SUBNORMAL, m * 2^-149 times a per-channel power of two.  FFMA consumes subnormal operands
//     exactly and at full rate, so "decode" is one AND (g, b) or one shift (r) and the channel
//     scale moves into the final normalisation;
//   * the shared exponent goes into the tap's bilinear weight: w * 2^E is one integer
//     multiply-add on the weight's exponent field (IMAD, FMA pipe), exact;
//   * no bias accumulator, fp32 weights, exact products: the arithmetic of tools/ibl.cpp:34-41
//     up to summation order.  Four logic ops + one IMAD per tap instead of six logic ops, and
//     six packed FMAs per sample instead of eight.
//
// Around that loop:
//   * the sample table is banded (ibl_tables.h): bands of kSampleBand entries of the lobe-angle
//     order; the warps of a tile each take their share of every band.  For the one-sample kernel
//     (prefilter_dn_kernel) a band is a ring of the lobe walked by azimuth and the same-face test (no
//     cube-face selection needed) is one angle per band and tile; the pair kernel
//     (prefilter_dp_kernel, what the library runs) gives every warp ONE azimuth sector of every band
//     and its own count of same-face bands (ibl_math.cuh, sector_rho_limits);
//   * tiles are numbered in 4x4 blocks and, for big levels, handed out from per-SM queues so that
//     the CTAs resident on one SM work on neighbouring tiles and share the lobe's footprint in L1
//     (measured: L1 hit rate 38 % -> 68 % on the 512^2 -> 256^2 level);
//   * the pair kernel reads a texel's frame and its tile's sector limits from per-level planes
//     (build_frames_kernel) instead of computing them per tile.

#include "prefilter.h"
#include "prefilter_pair.cuh"
#include "ibl_math.cuh"

#include <cuda_runtime.h>

#include <vector>

namespace ibl
{
  namespace
  {
    // bits(w) + E * 2^23 == bits(w * 2^E).  The multiplier arrives as a kernel parameter: as a
    // literal the compiler lowers it to shift + add on the ALU pipe, the pipe this loop is short of.
    __device__ __forceinline__ float scale_by_exponent(float w, uint32_t e, uint32_t emul)
    {
      uint32_t r;
      asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(e), "r"(emul), "r"(f2u(w)));
      return u2f(r);
    }
  }

  // the same on the ALU pipe: LOP3 + LEA.  The pair kernel spreads its taps over both forms so that
  // neither the FMA pipe (IMAD shares it with the packed FMAs) nor the ALU pipe saturates.
  __device__ __forceinline__ float scale_by_exponent_alu(float w, uint32_t word)
  {
    uint32_t e, r;
    asm volatile("and.b32 %0, %1, 31;" : "=r"(e) : "r"(word));
    asm volatile("shl.b32 %0, %1, 23;" : "=r"(r) : "r"(e));
    return u2f(r + f2u(w));
  }

  // r mantissa = word >> 23: a shift on the ALU pipe, or (A/B) the high half of word * 2^9 on the FMA pipe
  template<bool HI>
  __device__ __forceinline__ float red_field(uint32_t word, uint32_t rmul)
  {
    if (!HI)
      return u2f(word >> 23);

    uint32_t r;
    asm("mul.hi.u32 %0, %1, %2;" : "=r"(r) : "r"(word), "r"(rmul));
    return u2f(r);
  }

  template<bool ALU>
  __device__ __forceinline__ float scale_tap(float w, uint32_t word, uint32_t emul)
  {
    return ALU ? scale_by_exponent_alu(w, word) : scale_by_exponent(w, word & kDnMaskE, emul);
  }

  // ---- quad records ----------------------------------------------------------------

  __global__ void __launch_bounds__(256) build_dn_records_kernel(uint32_t const *__restrict__ src, uint4 *__restrict__ rec, int ws, int hs, size_t src_stride, int *__restrict__ counters, int ncounters)
  {
    // the prefilter launch that follows on the stream takes its tiles from these queues
    if (blockIdx.x == 0 && blockIdx.y == 0)
      for(int i = threadIdx.x; i < ncounters; i += blockDim.x)
        counters[i] = 0;

    // blockIdx.y = probe of a batch: source levels `src_stride` words apart, their records back to back
    const uint32_t level = 6u * (uint32_t)ws * (uint32_t)hs;
    src += (size_t)blockIdx.y * src_stride;
    rec += (size_t)blockIdx.y * level;

    for(uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x; idx < level; idx += gridDim.x * blockDim.x)
    {
      uint32_t i = idx % (uint32_t)ws;
      uint32_t j = (idx / (uint32_t)ws) % (uint32_t)hs;
      uint32_t right = (i + 1 < (uint32_t)ws) ? 1u : 0u;           // neighbours clamped inside the face; the clamped
      uint32_t down = (j + 1 < (uint32_t)hs) ? (uint32_t)ws : 0u;  // ones are never addressed (i <= ws-2, j <= hs-2)

      uint32_t const *t = src + idx;

      uint4 r;
      r.x = pack_dn_word(__ldg(t));
      r.y = pack_dn_word(__ldg(t + right));
      r.z = pack_dn_word(__ldg(t + down));
      r.w = pack_dn_word(__ldg(t + down + right));
      rec[idx] = r;
    }
  }


  // ---- "this launch has stored everything" -----------------------------------------------------
  //
  // One probe shared by several GPUs: the epilogues above store every word into the peers' chains.
  // The CTA that finishes LAST (ticket counter) bumps an arrival counter in every peer's flag block
  // with a system-scope release; the peers' streams wait on their own counter (a stream memory
  // operation, no kernel) before the next level reads the words.  Every thread fences its own
  // stores before the ticket, the last CTA fences again behind it (cumulativity).
  __device__ __forceinline__ void signal_peers_when_last(PeerSignal const &s)
  {
    if (s.count <= 0)
      return;

    __threadfence_system();
    __syncthreads();

    if (threadIdx.x == 0)
    {
      unsigned int ticket = atomicAdd(s.ticket, 1u);
      if (ticket == gridDim.x - 1)
      {
        __threadfence_system();
        for(int k = 0; k < s.count; ++k)
          asm volatile("red.release.sys.global.add.u32 [%0], 1;" :: "l"(s.arrive[k]) : "memory");
        *s.ticket = 0;        // ready for the next launch on this stream
      }
    }
  }

  // ---- one sample of one texel -------------------------------------------------------

  struct TexelFrame
  {
    Vec3f T, B, N;      // tangent frame rows: face-local and pre-scaled for the same-face loop, world for the general loop
    uint32_t face_base; // face*face_size - bias
    int face;
  };

  // weights of the 2x2 footprint (tools/ibl.cpp:40 as four products), exponents folded in, taps accumulated
  __device__ __forceinline__ void accumulate(uint4 rec, float du, float dv, float nl, float wh, uint32_t emul, Sums &acc)
  {
    float u0 = 0.5f - du, u1 = 0.5f + du;
    float v0 = fmaf(-dv, nl, wh), v1 = fmaf(dv, nl, wh);

    f32x2 u = pack2(u0, u1);
    float w00, w10, w01, w11;
    unpack2(mul2(u, bcast2(v0)), w00, w10);
    unpack2(mul2(u, bcast2(v1)), w01, w11);

    w00 = scale_by_exponent(w00, rec.x & kDnMaskE, emul);
    w10 = scale_by_exponent(w10, rec.y & kDnMaskE, emul);
    w01 = scale_by_exponent(w01, rec.z & kDnMaskE, emul);
    w11 = scale_by_exponent(w11, rec.w & kDnMaskE, emul);

    acc.rg = fma2(pack2(u2f(rec.x >> 23), u2f(rec.x & kDnMaskG)), bcast2(w00), acc.rg);
    acc.rg = fma2(pack2(u2f(rec.y >> 23), u2f(rec.y & kDnMaskG)), bcast2(w10), acc.rg);
    acc.rg = fma2(pack2(u2f(rec.z >> 23), u2f(rec.z & kDnMaskG)), bcast2(w01), acc.rg);
    acc.rg = fma2(pack2(u2f(rec.w >> 23), u2f(rec.w & kDnMaskG)), bcast2(w11), acc.rg);
    acc.bb = fma2(pack2(u2f(rec.x & kDnMaskB), u2f(rec.y & kDnMaskB)), pack2(w00, w10), acc.bb);
    acc.bb = fma2(pack2(u2f(rec.z & kDnMaskB), u2f(rec.w & kDnMaskB)), pack2(w01, w11), acc.bb);
  }

  // sample whose reflected direction provably stays on the texel's own face: frame rows are in
  // face-local (a, b, m) coordinates with a, b pre-scaled to source texels (face_footprint of ibl_math.cuh,
  // the (a, b) pair carried packed)
  __device__ __forceinline__ void sample_same_face(PrefilterDnParams const &p, TexelFrame const &t, float4 e, Sums &acc)
  {
    f32x2 lab = mul2(bcast2(e.x), pack2(t.T.x, t.T.y));
    lab = fma2(bcast2(e.y), pack2(t.B.x, t.B.y), lab);
    lab = fma2(bcast2(e.z), pack2(t.N.x, t.N.y), lab);
    float lm = fmaf(e.z, t.N.z, fmaf(e.y, t.B.z, e.x * t.T.z));

    float r = rcp_fast(lm);
    f32x2 f = fma2(lab, bcast2(r), pack2(p.geom.hwm, p.geom.hhm));
    f32x2 m = add2(f, bcast2(kMagic));
    f32x2 fi = add2(m, bcast2(-kMagic));
    f32x2 d = fma2(fi, bcast2(-1.0f), f);

    float mu, mv, du, dv;
    unpack2(m, mu, mv);
    unpack2(d, du, dv);

    uint32_t idx = f2u(mv) * (uint32_t)p.geom.ws + f2u(mu) + t.face_base;

    accumulate(__ldg(p.records + idx), du, dv, e.z, e.w, p.exp_mul, acc);
  }

  // any direction: cube face selection of tools/ibl.cpp:43-88 (cube_footprint of ibl_math.cuh)
  __device__ __forceinline__ void sample_general(PrefilterDnParams const &p, TexelFrame const &t, float4 e, Sums &acc)
  {
    float Lx = fmaf(e.z, t.N.x, fmaf(e.y, t.B.x, e.x * t.T.x));
    float Ly = fmaf(e.z, t.N.y, fmaf(e.y, t.B.y, e.x * t.T.y));
    float Lz = fmaf(e.z, t.N.z, fmaf(e.y, t.B.z, e.x * t.T.z));

    float du, dv;
    uint32_t idx = cube_footprint(p.geom, Lx, Ly, Lz, du, dv);

    accumulate(__ldg(p.records + idx), du, dv, e.z, e.w, p.exp_mul, acc);
  }

  // ---- the kernel --------------------------------------------------------------------------
  //
  // CTA = NW warps sharing one tile at a time; warp w takes entries [w*PER, (w+1)*PER) of every
  // band, partial sums meet in shared memory.  Big levels use 4 warps per tile (most CTAs per SM,
  // cheapest reduction), small ones 8, 16 or 32 so that the few tiles still spread over the machine.
  template<int NW, int UNROLL, int MINB, bool SMEM_TABLE, bool QUEUES>
  __global__ void __launch_bounds__(32 * NW, MINB) prefilter_dn_kernel(PrefilterDnParams p)
  {
    extern __shared__ float4 smem[];
    float4 *s_table = smem;
    float *s_red = reinterpret_cast<float*>(smem + (SMEM_TABLE ? p.table_count : 0));
    int *s_tile = reinterpret_cast<int*>(s_red + NW * 3 * 32);

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;

    if (SMEM_TABLE)
    {
      for(int i = tid; i < p.table_count; i += 32 * NW)
        s_table[i] = __ldg(p.table + i);
      __syncthreads();
    }

    float4 const *table = SMEM_TABLE ? s_table : p.table;

    uint32_t smid;
    asm("mov.u32 %0, %%smid;" : "=r"(smid));

    constexpr int PER = kSampleBand / NW > 0 ? kSampleBand / NW : 1;   // entries of a band per warp
    constexpr int SPLIT = kSampleBand / PER;                            // warps that share a band (NW or kSampleBand)
    static_assert(NW % SPLIT == 0, "warps per tile must be a multiple of the band split");

    // with more warps than band entries, consecutive groups of SPLIT warps take alternate bands
    const int lane_warp = warp % SPLIT;
    const int band_first = warp / SPLIT;
    constexpr int BAND_STEP = NW / SPLIT;
    constexpr int BAND_UNROLL = PER >= 4 ? 1 : 4 / PER;

    for(int it = 0; ; ++it)
    {
      int tile;
      if (QUEUES)
      {
        if (tid == 0)
          *s_tile = next_tile_plain(p, smid);
        __syncthreads();
        tile = *s_tile;

        if (tile < 0 && !p.no_steal)
        {
          __syncthreads();                 // everybody has read the empty hand-out
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

      int x, row;
      bool valid = tile_texel(p, tile, lane, x, row);

      // the blocked numbering covers whole 4x4 blocks: a tile past the slab has no work
      if (__ballot_sync(0xffffffffu, valid) == 0u)
      {
        if (QUEUES)
          __syncthreads();   // s_tile is rewritten in the next round
        continue;
      }

      // lanes past the slab still walk the loops (their sums are dropped): park them on a face centre
      if (!valid) { x = p.wd >> 1; row = (p.row_begin / p.hd) * p.hd + (p.hd >> 1); }

      int face = row / p.hd;
      int y = row - face * p.hd;

      TexelFrame st;
      int n_same;
      {
        Vec3f N = texel_normal(p.quats[face], x, y, p.wd, p.hd);
        Vec3f T, B;
        tangent_frame(N, T, B);

        // face-local rows, a and b scaled to source texels (align-corners, ibl.cpp:37-38)
        Vec3f Tl = to_face_local(face, T), Bl = to_face_local(face, B), Nl = to_face_local(face, N);

        float threshold = same_face_threshold(Nl);
        threshold = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(threshold)));

        st.T = Vec3f{ Tl.x * p.geom.hw, Tl.y * p.geom.hh, Tl.z };
        st.B = Vec3f{ Bl.x * p.geom.hw, Bl.y * p.geom.hh, Bl.z };
        st.N = Vec3f{ Nl.x * p.geom.hw, Nl.y * p.geom.hh, Nl.z };
        st.face = face;
        st.face_base = (uint32_t)face * p.geom.face_size - p.geom.bias;

        // number of leading bands (smallest angles) whose samples all stay on every texel's own face
        int lo = 0, hi = p.bands;
        while (lo < hi)
        {
          int mid = (lo + hi) >> 1;
          if (__ldg(p.band_min_lz + mid) > threshold)
            lo = mid + 1;
          else
            hi = mid;
        }
        n_same = lo;
      }

      Sums acc;
      acc.rg = 0ull;
      acc.bb = 0ull;

      const int full_bands = p.table_count / kSampleBand;
      const int same_full = n_same < full_bands ? n_same : full_bands;

      int band = band_first;

      // a warp that owns one or two entries per band gets its independent work from several bands
      #pragma unroll BAND_UNROLL
      for(; band < same_full; band += BAND_STEP)
      {
        float4 const *tb = table + band * kSampleBand + lane_warp * PER;

        #pragma unroll UNROLL
        for(int k = 0; k < PER; ++k)
          sample_same_face(p, st, SMEM_TABLE ? tb[k] : __ldg(tb + k), acc);
      }

      // the short last band, when it also stays on the face
      if (band == full_bands && n_same > full_bands)
      {
        for(int s = band * kSampleBand + lane_warp * PER, k = 0; k < PER && s < p.table_count; ++k, ++s)
          sample_same_face(p, st, SMEM_TABLE ? table[s] : __ldg(table + s), acc);
        band += BAND_STEP;
      }

      if (band < p.bands)
      {
        // back to world coordinates for the samples that may cross a face edge
        st.T = from_face_local(st.face, Vec3f{ st.T.x * p.geom.inv_hw, st.T.y * p.geom.inv_hh, st.T.z });
        st.B = from_face_local(st.face, Vec3f{ st.B.x * p.geom.inv_hw, st.B.y * p.geom.inv_hh, st.B.z });
        st.N = from_face_local(st.face, Vec3f{ st.N.x * p.geom.inv_hw, st.N.y * p.geom.inv_hh, st.N.z });

        #pragma unroll BAND_UNROLL
        for(; band < full_bands; band += BAND_STEP)
        {
          float4 const *tb = table + band * kSampleBand + lane_warp * PER;

          #pragma unroll UNROLL
          for(int k = 0; k < PER; ++k)
            sample_general(p, st, SMEM_TABLE ? tb[k] : __ldg(tb + k), acc);
        }

        if (band == full_bands && band < p.bands)
        {
          for(int s = band * kSampleBand + lane_warp * PER, k = 0; k < PER && s < p.table_count; ++k, ++s)
            sample_general(p, st, SMEM_TABLE ? table[s] : __ldg(table + s), acc);
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
          // sum/totalweight of ibl.cpp:186, then rgbe() of ibl.cpp:269
          float r = sum[0] * p.norm[0], g = sum[1] * p.norm[1], b = sum[2] * p.norm[2];
          size_t o = (size_t)row * p.wd + x;

          if (p.dst_words || p.peers > 0)
          {
            uint32_t word = rgbe_encode(r, g, b);

            if (p.dst_words)
              p.dst_words[o] = word;

            // one probe split over several GPUs: the slab goes straight into every peer's chain
            for(int k = 0; k < p.peers; ++k)
              p.peer_words[k][o] = word;
          }

          if (p.dst_f32)
          {
            p.dst_f32[3*o + 0] = r;
            p.dst_f32[3*o + 1] = g;
            p.dst_f32[3*o + 2] = b;
          }
        }
      }

      __syncthreads();   // s_red and s_tile are reused by the next tile
    }

    signal_peers_when_last(p.signal);
  }

  // ---- per-texel frames of a destination level -----------------------------------------------
  //
  // Normal, tangent frame (exactly rounded divisions and square roots, ~300 instructions), the change to
  // face-local coordinates and the fold depend on the level's geometry alone.  The pair kernel used to
  // redo them per tile in every one of its warps (3.5 % of its instructions on the 512^2 -> 256^2 level);
  // now they are computed once per (source size, context) and read back as ten coalesced planes.
  struct FrameQuats { Quatf q[6]; };

  __global__ void __launch_bounds__(256) build_frames_kernel(float *__restrict__ frames, int wd, int hd, LevelGeom geom, FrameQuats quats)
  {
    const int texels = 6 * wd * hd;
    int o = blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= texels)
      return;

    int x = o % wd, row = o / wd;
    int face = row / hd, y = row - face * hd;

    Vec3f N = texel_normal(quats.q[face], x, y, wd, hd);
    Vec3f T, B;
    tangent_frame(N, T, B);

    Vec3f Tl = to_face_local(face, T), Bl = to_face_local(face, B), Nl = to_face_local(face, N);
    Vec3f Tf = fold_face_row(geom, Tl), Bf = fold_face_row(geom, Bl), Nf = fold_face_row(geom, Nl);

    size_t plane = (size_t)texels;
    frames[0 * plane + o] = Tf.x; frames[1 * plane + o] = Tf.y; frames[2 * plane + o] = Tf.z;
    frames[3 * plane + o] = Bf.x; frames[4 * plane + o] = Bf.y; frames[5 * plane + o] = Bf.z;
    frames[6 * plane + o] = Nf.x; frames[7 * plane + o] = Nf.y; frames[8 * plane + o] = Nf.z;

    // sector limits: minimum over the texels of the 8x4 tile (limits are >= 0: bit order = value order;
    // the planes start out as 0x7f7f7f7f = 3.4e38)
    float limits[kFrameSectors];
    sector_rho_limits(Tl, Bl, Nl, limits);

    const int tiles_x = (wd + 7) / 8, tile_rows = (6 * hd + 3) / 4;
    unsigned int *tile = reinterpret_cast<unsigned int*>(frames + 9 * plane) + (size_t)(row >> 2) * tiles_x + (x >> 3);
    #pragma unroll
    for(int k = 0; k < kFrameSectors; ++k)
      atomicMin(tile + (size_t)k * tile_rows * tiles_x, __float_as_uint(limits[k]));
  }

  __global__ void __launch_bounds__(256) build_world_frames_kernel(float *__restrict__ frames, int wd, int hd, FrameQuats quats)
  {
    const int texels = 6 * wd * hd;
    int o = blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= texels)
      return;

    int x = o % wd, row = o / wd;
    int face = row / hd, y = row - face * hd;

    Vec3f N = texel_normal(quats.q[face], x, y, wd, hd);
    Vec3f T, B;
    tangent_frame(N, T, B);

    size_t plane = (size_t)texels;
    frames[0 * plane + o] = T.x; frames[1 * plane + o] = T.y; frames[2 * plane + o] = T.z;
    frames[3 * plane + o] = B.x; frames[4 * plane + o] = B.y; frames[5 * plane + o] = B.z;
    frames[6 * plane + o] = N.x; frames[7 * plane + o] = N.y; frames[8 * plane + o] = N.z;
  }

  cudaError_t launch_build_world_frames(float *frames, int wd, int hd, Quatf const quats[6], cudaStream_t stream)
  {
    int texels = 6 * wd * hd;
    if (texels <= 0)
      return cudaSuccess;

    FrameQuats q;
    for(int f = 0; f < 6; ++f)
      q.q[f] = quats[f];

    build_world_frames_kernel<<<(texels + 255) / 256, 256, 0, stream>>>(frames, wd, hd, q);
    return cudaGetLastError();
  }

  cudaError_t launch_build_frames(float *frames, int ws, int hs, Quatf const quats[6], cudaStream_t stream)
  {
    int wd = ws >> 1, hd = hs >> 1;
    int texels = 6 * wd * hd;
    if (texels <= 0)
      return cudaSuccess;

    FrameQuats q;
    for(int f = 0; f < 6; ++f)
      q.q[f] = quats[f];

    cudaError_t err = cudaMemsetAsync(frames + (size_t)9 * texels, 0x7f, sizeof(float) * (size_t)kFrameSectors * frame_tile_rows(hd) * frame_tiles_x(wd), stream);
    if (err != cudaSuccess)
      return err;

    build_frames_kernel<<<(texels + 255) / 256, 256, 0, stream>>>(frames, wd, hd, make_level_geom(ws, hs), q);
    return cudaGetLastError();
  }

  // ---- two samples at a time --------------------------------------------------------------
  //
  // The kernel above packs the (a, b) face coordinates of ONE sample into fp32x2 operations; the
  // third coordinate, the bilinear weights and half of the magic-add floor stay scalar.  Packing
  // the SAME quantity of TWO consecutive samples instead makes every per-sample fp32 operation a
  // half-instruction, and the general (cube-face-selecting) path gets the packed direction and floor
  // it never had.  The two b partial sums belong to the two samples of a pair instead of to the tap
  // columns.  The table arrives pair-interleaved with its short shares filled up, so there is no
  // short-band code.
  //
  // Two statements of the per-pair arithmetic follow.  The first (direction_pair, gather_pair,
  // pair_same_face, pair_general: PROJ = false) is round 2's first cut — three-term directions, an
  // integer record index whose bias kMagicBits*(ws+1) is folded into the record pointer, four weight
  // products — kept for the A/B variants of the tools build.  The second (gather_pair_proj with the
  // coordinates of prefilter_pair.cuh: what ships) is the projective form described there.

  // record `idx` (unsigned 32-bit, bias included) of an opaque() `base`
  __device__ __forceinline__ uint4 load_record(uint4 const *base, uint32_t idx)
  {
    return __ldg(base + idx);
  }

  // reflected directions of both samples in the frame's coordinates, the kernel above's operation order
  __device__ __forceinline__ void direction_pair(Frame const &t, PairEntry const &e, f32x2 &x, f32x2 &y, f32x2 &z)
  {
    x = fma2(e.lz, bcast2(t.N.x), fma2(e.ly, bcast2(t.B.x), mul2(e.lx, bcast2(t.T.x))));
    y = fma2(e.lz, bcast2(t.N.y), fma2(e.ly, bcast2(t.B.y), mul2(e.lx, bcast2(t.T.y))));
    z = fma2(e.lz, bcast2(t.N.z), fma2(e.ly, bcast2(t.B.z), mul2(e.lx, bcast2(t.T.z))));
  }

  // (fu, fv) of both samples -> records, weights, taps.  EXP_ALU of the four taps of a sample take their exponent on the ALU pipe.  `base` holds the bias (and the face on the same-face path).
  template<int EXP_ALU, bool RHI>
  __device__ __forceinline__ void gather_pair(PrefilterDnParams const &p, uint4 const *base, uint32_t off_a, uint32_t off_b, f32x2 fu, f32x2 fv, PairEntry const &e, Sums &acc)
  {
    f32x2 mu = add2(fu, bcast2(kMagic));
    f32x2 mv = add2(fv, bcast2(kMagic));
    f32x2 iu = add2(mu, bcast2(-kMagic));
    f32x2 iv = add2(mv, bcast2(-kMagic));
    f32x2 du = fma2(iu, bcast2(-1.0f), fu);
    f32x2 dv = fma2(iv, bcast2(-1.0f), fv);

    float mua, mub, mva, mvb;
    unpack2(mu, mua, mub);
    unpack2(mv, mva, mvb);

    uint4 ra = load_record(base, f2u(mva) * (uint32_t)p.geom.ws + f2u(mua) + off_a);
    uint4 rb = load_record(base, f2u(mvb) * (uint32_t)p.geom.ws + f2u(mub) + off_b);

    // tools/ibl.cpp:40 as four products, times the sample weight: (0.5 -+ du) * (wh -+ dv * nl)
    f32x2 u0 = fma2(du, bcast2(-1.0f), bcast2(0.5f));
    f32x2 u1 = add2(du, bcast2(0.5f));
    f32x2 v0 = fma2(neg2(dv), e.lz, e.wh);
    f32x2 v1 = fma2(dv, e.lz, e.wh);

    float w00a, w00b, w10a, w10b, w01a, w01b, w11a, w11b;
    unpack2(mul2(u0, v0), w00a, w00b);
    unpack2(mul2(u1, v0), w10a, w10b);
    unpack2(mul2(u0, v1), w01a, w01b);
    unpack2(mul2(u1, v1), w11a, w11b);

    const uint32_t emul = p.exp_mul;
    w00a = scale_tap<(EXP_ALU > 0)>(w00a, ra.x, emul);
    w10a = scale_tap<(EXP_ALU > 2)>(w10a, ra.y, emul);
    w01a = scale_tap<(EXP_ALU > 1)>(w01a, ra.z, emul);
    w11a = scale_tap<(EXP_ALU > 3)>(w11a, ra.w, emul);
    w00b = scale_tap<(EXP_ALU > 0)>(w00b, rb.x, emul);
    w10b = scale_tap<(EXP_ALU > 2)>(w10b, rb.y, emul);
    w01b = scale_tap<(EXP_ALU > 1)>(w01b, rb.z, emul);
    w11b = scale_tap<(EXP_ALU > 3)>(w11b, rb.w, emul);

    acc.rg = fma2(pack2(red_field<RHI>(ra.x, p.red_mul), u2f(ra.x & kDnMaskG)), bcast2(w00a), acc.rg);
    acc.rg = fma2(pack2(red_field<RHI>(ra.y, p.red_mul), u2f(ra.y & kDnMaskG)), bcast2(w10a), acc.rg);
    acc.rg = fma2(pack2(red_field<RHI>(ra.z, p.red_mul), u2f(ra.z & kDnMaskG)), bcast2(w01a), acc.rg);
    acc.rg = fma2(pack2(red_field<RHI>(ra.w, p.red_mul), u2f(ra.w & kDnMaskG)), bcast2(w11a), acc.rg);
    acc.rg = fma2(pack2(red_field<RHI>(rb.x, p.red_mul), u2f(rb.x & kDnMaskG)), bcast2(w00b), acc.rg);
    acc.rg = fma2(pack2(red_field<RHI>(rb.y, p.red_mul), u2f(rb.y & kDnMaskG)), bcast2(w10b), acc.rg);
    acc.rg = fma2(pack2(red_field<RHI>(rb.z, p.red_mul), u2f(rb.z & kDnMaskG)), bcast2(w01b), acc.rg);
    acc.rg = fma2(pack2(red_field<RHI>(rb.w, p.red_mul), u2f(rb.w & kDnMaskG)), bcast2(w11b), acc.rg);

    acc.bb = fma2(pack2(u2f(ra.x & kDnMaskB), u2f(rb.x & kDnMaskB)), pack2(w00a, w00b), acc.bb);
    acc.bb = fma2(pack2(u2f(ra.y & kDnMaskB), u2f(rb.y & kDnMaskB)), pack2(w10a, w10b), acc.bb);
    acc.bb = fma2(pack2(u2f(ra.z & kDnMaskB), u2f(rb.z & kDnMaskB)), pack2(w01a, w01b), acc.bb);
    acc.bb = fma2(pack2(u2f(ra.w & kDnMaskB), u2f(rb.w & kDnMaskB)), pack2(w11a, w11b), acc.bb);
  }

  // frame rows in face-local (a, b, m) coordinates, a and b pre-scaled to source texels
  template<int EXP_ALU, bool RHI>
  __device__ __forceinline__ void pair_same_face(PrefilterDnParams const &p, Frame const &t, uint4 const *base, PairEntry const &e, Sums &acc)
  {
    f32x2 la, lb, lm;
    direction_pair(t, e, la, lb, lm);

    float ma, mb;
    unpack2(lm, ma, mb);
    f32x2 r = pack2(rcp_fast(ma), rcp_fast(mb));

    gather_pair<EXP_ALU, RHI>(p, base, 0u, 0u, fma2(la, r, bcast2(p.geom.hwm)), fma2(lb, r, bcast2(p.geom.hhm)), e, acc);
  }

  // frame rows in world coordinates: cube face selection of tools/ibl.cpp:43-88 per sample
  template<int EXP_ALU, bool RHI>
  __device__ __forceinline__ void pair_general(PrefilterDnParams const &p, Frame const &t, uint4 const *base, PairEntry const &e, Sums &acc)
  {
    f32x2 x, y, z;
    direction_pair(t, e, x, y, z);

    float xa, xb, ya, yb, za, zb;
    unpack2(x, xa, xb);
    unpack2(y, ya, yb);
    unpack2(z, za, zb);

    float qua, qva, qub, qvb;
    uint32_t fa, fb;
    cube_select(xa, ya, za, qua, qva, fa);
    cube_select(xb, yb, zb, qub, qvb, fb);

    f32x2 fu = fma2(pack2(qua, qub), bcast2(p.geom.hw), bcast2(p.geom.hwm));
    f32x2 fv = fma2(pack2(qva, qvb), bcast2(p.geom.hh), bcast2(p.geom.hhm));

    // the face offset goes into the 32-bit index (bias + 6 faces cannot wrap, see the launcher)
    gather_pair<EXP_ALU, RHI>(p, base, fa * p.geom.face_size, fb * p.geom.face_size, fu, fv, e, acc);
  }

  // idx = raw index bits of both samples (what `base` has been moved back by), du/dv = fraction - 0.5
  template<int EXP_ALU>
  __device__ __forceinline__ void gather_pair_proj(PrefilterDnParams const &p, uint4 const *base, uint32_t idx_a, uint32_t idx_b, f32x2 du, f32x2 dv, PairEntry const &e, Sums &acc)
  {
    uint4 ra = load_record(base, idx_a);
    uint4 rb = load_record(base, idx_b);

    // tools/ibl.cpp:40 times the sample weight: (0.5 -+ du) * (wh -+ dv * nl), right-hand column by difference
    f32x2 u0 = add2(neg2(du), bcast2(0.5f));
    f32x2 v0 = fma2(neg2(dv), e.lz, e.wh);
    f32x2 v1 = fma2(dv, e.lz, e.wh);
    f32x2 p00 = mul2(u0, v0);
    f32x2 p01 = mul2(u0, v1);

    float w00a, w00b, w10a, w10b, w01a, w01b, w11a, w11b;
    unpack2(p00, w00a, w00b);
    unpack2(p01, w01a, w01b);
    unpack2(add2(v0, neg2(p00)), w10a, w10b);
    unpack2(add2(v1, neg2(p01)), w11a, w11b);

    const uint32_t emul = p.exp_mul;
    w00a = scale_tap<(EXP_ALU > 0)>(w00a, ra.x, emul);
    w10a = scale_tap<(EXP_ALU > 2)>(w10a, ra.y, emul);
    w01a = scale_tap<(EXP_ALU > 1)>(w01a, ra.z, emul);
    w11a = scale_tap<(EXP_ALU > 3)>(w11a, ra.w, emul);
    w00b = scale_tap<(EXP_ALU > 0)>(w00b, rb.x, emul);
    w10b = scale_tap<(EXP_ALU > 2)>(w10b, rb.y, emul);
    w01b = scale_tap<(EXP_ALU > 1)>(w01b, rb.z, emul);
    w11b = scale_tap<(EXP_ALU > 3)>(w11b, rb.w, emul);

    acc.rg = fma2(pack2(u2f(ra.x >> 23), u2f(ra.x & kDnMaskG)), bcast2(w00a), acc.rg);
    acc.rg = fma2(pack2(u2f(ra.y >> 23), u2f(ra.y & kDnMaskG)), bcast2(w10a), acc.rg);
    acc.rg = fma2(pack2(u2f(ra.z >> 23), u2f(ra.z & kDnMaskG)), bcast2(w01a), acc.rg);
    acc.rg = fma2(pack2(u2f(ra.w >> 23), u2f(ra.w & kDnMaskG)), bcast2(w11a), acc.rg);
    acc.rg = fma2(pack2(u2f(rb.x >> 23), u2f(rb.x & kDnMaskG)), bcast2(w00b), acc.rg);
    acc.rg = fma2(pack2(u2f(rb.y >> 23), u2f(rb.y & kDnMaskG)), bcast2(w10b), acc.rg);
    acc.rg = fma2(pack2(u2f(rb.z >> 23), u2f(rb.z & kDnMaskG)), bcast2(w01b), acc.rg);
    acc.rg = fma2(pack2(u2f(rb.w >> 23), u2f(rb.w & kDnMaskG)), bcast2(w11b), acc.rg);

    acc.bb = fma2(pack2(u2f(ra.x & kDnMaskB), u2f(rb.x & kDnMaskB)), pack2(w00a, w00b), acc.bb);
    acc.bb = fma2(pack2(u2f(ra.y & kDnMaskB), u2f(rb.y & kDnMaskB)), pack2(w10a, w10b), acc.bb);
    acc.bb = fma2(pack2(u2f(ra.z & kDnMaskB), u2f(rb.z & kDnMaskB)), pack2(w01a, w01b), acc.bb);
    acc.bb = fma2(pack2(u2f(ra.w & kDnMaskB), u2f(rb.w & kDnMaskB)), pack2(w11a, w11b), acc.bb);
  }

  // frame rows face-local and folded; `base` = records of the texel's face, moved back by kMagicBits
  template<int EXP_ALU>
  __device__ __forceinline__ void pair_same_face_proj(PrefilterDnParams const &p, Frame const &t, uint4 const *base, PairEntry const &e, Sums &acc)
  {
    uint32_t ia, ib;
    f32x2 du, dv;
    pair_taps_same_face(p.geom, t, e, ia, ib, du, dv);
    gather_pair_proj<EXP_ALU>(p, base, ia, ib, du, dv, e, acc);
  }

  // frame rows in world coordinates; `base` = records moved back by geom.bias_general
  template<int EXP_ALU>
  __device__ __forceinline__ void pair_general_proj(PrefilterDnParams const &p, Frame const &t, uint4 const *base, PairEntry const &e, Sums &acc)
  {
    uint32_t ia, ib;
    f32x2 du, dv;
    pair_taps_general(p.geom, t, e, ia, ib, du, dv);
    gather_pair_proj<EXP_ALU>(p, base, ia, ib, du, dv, e, acc);
  }

  template<int NW, int MINB, bool SMEM_TABLE, bool QUEUES, int EXP_ALU, int DEPTH = 1, bool RHI = false, bool PLAIN_QUEUE = false, bool LEAN = false, bool PROJ = true, int VW = 1>
  __global__ void __launch_bounds__(32 * NW, MINB) prefilter_dp_kernel(PrefilterDnParams p)
  {
    extern __shared__ float4 smem[];
    // VW = 2: a warp takes TWO 45-degree sectors of the 8-sector table one after the other, each with its own
    // count of same-face bands, instead of one 90-degree sector of the 4-sector table
    static_assert(VW == 1 || (VW == 2 && NW == 4 && PROJ), "two sectors per warp: four warps per tile, projective form");
    constexpr int SECTORS = NW * VW == 8 ? 1 : 0;                  // which of the two sector tables
    const int bands = PROJ ? p.sector_bands[SECTORS] : p.bands;
    // entries per band: the sector tables hold FOUR entries (two pairs) per sector and band, whatever the number of
    // sectors, so that a round of the sample loops is always two pairs of one band (a loop over one pair of two
    // bands measured 3 % slower); round 2's table for the A/B variants has kSampleBand
    constexpr int BAND = PROJ ? kSectorShare * NW * VW : kSampleBand;
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
        s_table[i] = __ldg((PROJ ? p.table_sector[SECTORS] : p.table_pairs) + i);
      __syncthreads();
    }

    float4 const *table = SMEM_TABLE ? s_table : (PROJ ? p.table_sector[SECTORS] : p.table_pairs);

    uint32_t smid;
    asm("mov.u32 %0, %%smid;" : "=r"(smid));

    constexpr int PER = BAND / (NW * VW);        // entries of a band per warp and pass
    constexpr int PAIRS = PER / 2;
    static_assert(PER >= 2 && PER % 2 == 0, "a warp takes whole pairs of every band");
    constexpr int BAND_UNROLL = (PAIRS >= 2 ? 1 : 2) * DEPTH;     // DEPTH 2: twice the footprint loads in flight per warp (A/B)

    // records, moved back by the bias of the magic-add integers (projective form: of the one fp32 index;
    // the general path's index also carries -hhm*ws, see cube_footprint_proj)
    uint4 const *biased = opaque(p.records - (size_t)(PROJ ? kMagicBits : p.geom.bias));

    for(int it = 0; ; ++it)
    {
      int tile;
      if (QUEUES)
      {
        if (tid == 0)
          *s_tile = next_tile_plain(p, smid);
        __syncthreads();
        tile = *s_tile;

        if (!PLAIN_QUEUE && tile < 0 && !p.no_steal)
        {
          __syncthreads();                 // everybody has read the empty hand-out
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

      // a launch may carry the same level of several probes (datum_ibl_bake_probes): tiles are numbered
      // probe by probe, records and destination levels sit at fixed strides
      int probe = 0, ltile = tile;
      if (!LEAN && p.probes > 1)
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
      int y = row - face * p.hd;

      // this probe's records (a batch: records of the probes back to back)
      uint4 const *biased_probe = LEAN ? biased : opaque(biased + (size_t)probe * p.record_stride);

      Frame st;
      int n_same, n_same_second = 0;
      {
        if (PROJ)
        {
          tile_frame_bands<NW, VW>(p, x, row, warp, lane, bands, st, n_same, n_same_second);
        }
        else
        {
          Vec3f N = texel_normal(p.quats[face], x, y, p.wd, p.hd);
          Vec3f T, B;
          tangent_frame(N, T, B);

          Vec3f Tl = to_face_local(face, T), Bl = to_face_local(face, B), Nl = to_face_local(face, N);

          float threshold = same_face_threshold(Nl);
          threshold = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(threshold)));

          st.T = Vec3f{ Tl.x * p.geom.hw, Tl.y * p.geom.hh, Tl.z };
          st.B = Vec3f{ Bl.x * p.geom.hw, Bl.y * p.geom.hh, Bl.z };
          st.N = Vec3f{ Nl.x * p.geom.hw, Nl.y * p.geom.hh, Nl.z };

          int lo = 0, hi = p.bands;
          while (lo < hi)
          {
            int mid = (lo + hi) >> 1;
            if (__ldg(p.band_min_lz + mid) > threshold)
              lo = mid + 1;
            else
              hi = mid;
          }
          n_same = lo;
        }
      }

      Sums acc;
      acc.rg = 0ull;
      acc.bb = 0ull;

      // entry index == float4 index in the pair-interleaved table
      {
        uint4 const *base = opaque(biased_probe + (size_t)face * p.geom.face_size);

        #pragma unroll 1
        for(int pass = 0; pass < VW; ++pass)
        {
          float4 const *tw = table + (VW * warp + pass) * PER;
          const int count = pass == 0 ? n_same : n_same_second;

          #pragma unroll BAND_UNROLL
          for(int band = 0; band < count; ++band)
          {
            #pragma unroll
            for(int k = 0; k < PAIRS; ++k)
            {
              if (PROJ)
                pair_same_face_proj<EXP_ALU>(p, st, base, load_pair<SMEM_TABLE>(tw + band * BAND + 2 * k), acc);
              else
                pair_same_face<EXP_ALU, RHI>(p, st, base, load_pair<SMEM_TABLE>(tw + band * BAND + 2 * k), acc);
            }
          }
        }
      }

      if (n_same < bands || (VW == 2 && n_same_second < bands))
      {
        // back to world coordinates for the samples that may cross a face edge
        if (PROJ)
        {
          st.T = from_face_local(face, unfold_face_row(p.geom, st.T));
          st.B = from_face_local(face, unfold_face_row(p.geom, st.B));
          st.N = from_face_local(face, unfold_face_row(p.geom, st.N));
        }
        else
        {
          st.T = from_face_local(face, Vec3f{ st.T.x * p.geom.inv_hw, st.T.y * p.geom.inv_hh, st.T.z });
          st.B = from_face_local(face, Vec3f{ st.B.x * p.geom.inv_hw, st.B.y * p.geom.inv_hh, st.B.z });
          st.N = from_face_local(face, Vec3f{ st.N.x * p.geom.inv_hw, st.N.y * p.geom.inv_hh, st.N.z });
        }

        // the general path's index carries kMagicBits - hhm*ws instead of kMagicBits
        uint4 const *general = PROJ ? opaque(biased_probe + (size_t)(kMagicBits - p.geom.bias_general)) : biased_probe;

        #pragma unroll 1
        for(int pass = 0; pass < VW; ++pass)
        {
          float4 const *tw = table + (VW * warp + pass) * PER;

          #pragma unroll BAND_UNROLL
          for(int band = pass == 0 ? n_same : n_same_second; band < bands; ++band)
          {
            #pragma unroll
            for(int k = 0; k < PAIRS; ++k)
            {
              if (PROJ)
                pair_general_proj<EXP_ALU>(p, st, general, load_pair<SMEM_TABLE>(tw + band * BAND + 2 * k), acc);
              else
                pair_general<EXP_ALU, RHI>(p, st, general, load_pair<SMEM_TABLE>(tw + band * BAND + 2 * k), acc);
            }
          }
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
          // sum/totalweight of ibl.cpp:186, then rgbe() of ibl.cpp:269
          float r = sum[0] * p.norm[0], g = sum[1] * p.norm[1], b = sum[2] * p.norm[2];
          size_t o = (size_t)row * p.wd + x + (LEAN ? (size_t)0 : (size_t)probe * p.dst_stride);

          if (p.dst_words || p.peers > 0)
          {
            uint32_t word = rgbe_encode(r, g, b);

            if (p.dst_words)
              p.dst_words[o] = word;

            // one probe split over several GPUs: the slab goes straight into every peer's chain
            for(int k = 0; k < p.peers; ++k)
              p.peer_words[k][o] = word;
          }

          if (p.dst_f32)
          {
            p.dst_f32[3*o + 0] = r;
            p.dst_f32[3*o + 1] = g;
            p.dst_f32[3*o + 2] = b;
          }
        }
      }

      __syncthreads();
    }

    if (!LEAN)
      signal_peers_when_last(p.signal);
  }

  // ---- tail levels: lanes are samples ----------------------------------------------------------
  //
  // The last levels of a chain hold a few hundred texels: with one texel per lane the machine is
  // empty and every warp walks its samples one after the other (level 7 of C2: 3 tiles, 32 samples
  // deep per warp, 14 us for 1e5 texel-samples).  Here a CTA owns ONE texel and its lanes take
  // consecutive table entries: NW*32 samples per step, warp-shuffle + shared-memory reduction at the
  // end.  Every sample goes through the cube-face selection (at these roughnesses almost all leave
  // the face anyway); the four words of a footprint are read from the source level itself (it fits in
  // L1/L2) in the reference's own bit layout (raw_accumulate_tap), so the level needs no record pass: one
  // launch instead of two.  Arithmetic per sample is the one-sample kernel's general path.
  template<int NW, bool PROJ>
  __global__ void __launch_bounds__(32 * NW) prefilter_tail_kernel(PrefilterTailParams p)
  {
    __shared__ float s_red[NW][3];
    __shared__ float s_frame[9];

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    // a launch may carry the same level of several probes: texels are numbered probe by probe
    int texel = blockIdx.x, probe = 0;
    if (p.probes > 1)
    {
      probe = texel / p.texels_per_probe;
      texel -= probe * p.texels_per_probe;
    }
    const int row = p.row_begin + texel / p.wd;
    const int x = texel - (texel / p.wd) * p.wd;
    const int face = row / p.hd;
    const int y = row - face * p.hd;

    // the texel's frame: from the per-level planes (launch_build_world_frames), else computed here once per
    // CTA (exactly rounded divisions and square roots, ~200 dependent instructions by one thread)
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
        // e.x, e.y hold lx/lz, ly/lz (ibl_math.cuh, projective form)
        float Lx = fmaf(e.x, T.x, fmaf(e.y, B.x, N.x));
        float Ly = fmaf(e.x, T.y, fmaf(e.y, B.y, N.y));
        float Lz = fmaf(e.x, T.z, fmaf(e.y, B.z, N.z));

        uint32_t f;
        idx = cube_footprint_proj(p.geom, Lx, Ly, Lz, du, dv, f) + f * p.geom.face_size - p.geom.bias_general;
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

      uint32_t const *t = p.src + (size_t)probe * p.src_stride + idx;
      raw_accumulate_tap(__ldg(t), w[0], p.exp_mul, acc);
      raw_accumulate_tap(__ldg(t + 1), w[1], p.exp_mul, acc);
      raw_accumulate_tap(__ldg(t + p.geom.ws), w[2], p.exp_mul, acc);
      raw_accumulate_tap(__ldg(t + p.geom.ws + 1), w[3], p.exp_mul, acc);
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

      // sum/totalweight of ibl.cpp:186, then rgbe() of ibl.cpp:269
      float r = sum[0] * p.norm[0], g = sum[1] * p.norm[1], b = sum[2] * p.norm[2];
      size_t o = (size_t)row * p.wd + x + (size_t)probe * p.dst_stride;

      if (p.dst_words || p.peers > 0)
      {
        uint32_t word = rgbe_encode(r, g, b);

        if (p.dst_words)
          p.dst_words[o] = word;

        for(int k = 0; k < p.peers; ++k)
          p.peer_words[k][o] = word;
      }

      if (p.dst_f32)
      {
        p.dst_f32[3*o + 0] = r;
        p.dst_f32[3*o + 1] = g;
        p.dst_f32[3*o + 2] = b;
      }
    }

    signal_peers_when_last(p.signal);
  }

  cudaError_t launch_prefilter_tail(PrefilterTailParams const &params, int sm_count, cudaStream_t stream)
  {
    PrefilterTailParams p = params;

    int texels = (p.row_end - p.row_begin) * p.wd;
    if (texels <= 0)
      return cudaSuccess;

    if (p.probes < 1)
      p.probes = 1;
    p.texels_per_probe = texels;

    // warps per texel (tail_warps) chosen from ONE probe's texels also when a launch carries several: the
    // shape decides the order of the sums, and a batch must give the words of single calls
    (void)sm_count;
    int grid = texels * p.probes;
    const bool proj = p.table_proj != nullptr && proj_usable(p.geom.ws, p.geom.hs);
    switch (tail_warps(texels, p.table_count))
    {
      case 4: if (proj) prefilter_tail_kernel<4, true><<<grid, 128, 0, stream>>>(p); else prefilter_tail_kernel<4, false><<<grid, 128, 0, stream>>>(p); break;
      case 8: if (proj) prefilter_tail_kernel<8, true><<<grid, 256, 0, stream>>>(p); else prefilter_tail_kernel<8, false><<<grid, 256, 0, stream>>>(p); break;
      case 16: if (proj) prefilter_tail_kernel<16, true><<<grid, 512, 0, stream>>>(p); else prefilter_tail_kernel<16, false><<<grid, 512, 0, stream>>>(p); break;
      default: if (proj) prefilter_tail_kernel<32, true><<<grid, 1024, 0, stream>>>(p); else prefilter_tail_kernel<32, false><<<grid, 1024, 0, stream>>>(p); break;
    }

    return cudaGetLastError();
  }

  // ---- arrival signal without a producing launch (the barrier at the start of a shared bake) ------
  __global__ void peer_signal_kernel(PeerSignal s)
  {
    __threadfence_system();
    if ((int)threadIdx.x < s.count)
      asm volatile("red.release.sys.global.add.u32 [%0], 1;" :: "l"(s.arrive[threadIdx.x]) : "memory");
  }

  cudaError_t launch_peer_signal(PeerSignal const &s, cudaStream_t stream)
  {
    peer_signal_kernel<<<1, 32, 0, stream>>>(s);
    return cudaGetLastError();
  }

  // ---- host-side launchers ---------------------------------------------------------------

  cudaError_t launch_build_dn_records(uint32_t const *src, uint4 *rec, int ws, int hs, int probes, size_t src_stride, int *counters, int ncounters, int sm_count, cudaStream_t stream)
  {
    if (probes < 1)
      probes = 1;

    size_t level = (size_t)6 * ws * hs;          // < 2^32 for every face size a chain can have (6 * 16384^2 would not fit HBM as records)
    size_t blocks = (level + 255) / 256;
    size_t cap = ((size_t)sm_count * 8 + probes - 1) / probes;
    int grid = (int)(blocks < cap ? blocks : cap);
    if (grid < 1)
      grid = 1;

    build_dn_records_kernel<<<dim3(grid, probes), 256, 0, stream>>>(src, rec, ws, hs, src_stride, counters, ncounters);

    return cudaGetLastError();
  }

  // The occupancy query costs more host time than the launch itself: its answer is remembered per (kernel,
  // device, size).  The kernel's ADDRESS is part of the key (round 1 keyed by size only: a hit recorded by one
  // kernel skipped the opt-in of another).  The dynamic shared-memory opt-in is only ever raised, and only
  // above the 48 KB every kernel may use without it: setting the attribute to a smaller value would LOWER the
  // kernel's limit.
  cudaError_t resident_ctas(void const *kernel, int threads, size_t smem, int *resident)
  {
    struct Entry { void const *kernel; int device; size_t smem; int resident; };
    thread_local static std::vector<Entry> cache;
    struct OptIn { void const *kernel; int device; size_t smem; };
    thread_local static std::vector<OptIn> opted;

    int device = 0;
    cudaError_t err = cudaGetDevice(&device);
    if (err != cudaSuccess)
      return err;

    for(auto const &e : cache)
      if (e.kernel == kernel && e.device == device && e.smem == smem)
      {
        *resident = e.resident;
        return cudaSuccess;
      }

    if (smem > 48 * 1024)
    {
      OptIn *mine = nullptr;
      for(auto &o : opted)
        if (o.kernel == kernel && o.device == device)
          mine = &o;

      if (!mine || mine->smem < smem)
      {
        err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (err != cudaSuccess)
          return err;
        if (mine)
          mine->smem = smem;
        else
          opted.push_back(OptIn{ kernel, device, smem });
      }
    }

    err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(resident, kernel, threads, smem);
    if (err != cudaSuccess)
      return err;
    if (*resident < 1)
      return cudaErrorLaunchOutOfResources;

    if (cache.size() >= 256)
      cache.clear();
    cache.push_back(Entry{ kernel, device, smem, *resident });

    return cudaSuccess;
  }

  namespace
  {
    template<int NW, int UNROLL, int MINB, bool SMEM_TABLE, bool QUEUES>
    cudaError_t launch_dn(PrefilterDnParams p, int sm_count, cudaStream_t stream, int *launched_grid)
    {
      auto kernel = prefilter_dn_kernel<NW, UNROLL, MINB, SMEM_TABLE, QUEUES>;

      size_t smem = (SMEM_TABLE ? (size_t)p.table_count * sizeof(float4) : 0) + (size_t)NW * 3 * 32 * sizeof(float) + sizeof(int);

      int grid = 0;
      cudaError_t err = plan_tiles(p, kernel, 32 * NW, smem, 1, sm_count, &grid);
      if (err != cudaSuccess)
        return err;

      kernel<<<grid, 32 * NW, smem, stream>>>(p);

      if (launched_grid)
        *launched_grid = grid;

      return cudaGetLastError();
    }

    template<int NW, int MINB, bool SMEM_TABLE, bool QUEUES, int EXP_ALU = 0, int DEPTH = 1, bool RHI = false, bool PLAIN_QUEUE = false, bool LEAN = false, bool PROJ = true, int VW = 1>
    cudaError_t launch_dp(PrefilterDnParams p, int sm_count, cudaStream_t stream, int *launched_grid)
    {
      auto kernel = prefilter_dp_kernel<NW, MINB, SMEM_TABLE, QUEUES, EXP_ALU, DEPTH, RHI, PLAIN_QUEUE, LEAN, PROJ, VW>;

      const int table_bands = PROJ ? p.sector_bands[NW * VW == 8 ? 1 : 0] : p.bands;
      const int band_entries = PROJ ? kSectorShare * NW * VW : kSampleBand;
      size_t smem = (SMEM_TABLE ? (size_t)table_bands * band_entries * sizeof(float4) : 0) + (size_t)NW * 3 * 32 * sizeof(float) + sizeof(int);

      // (Cutting the common pool's tiles, or every tile of a slab too small to fill the machine, into 2-8
      // shares of their bands was measured and dropped: profiles/r2_summary.md.)
      if (p.probes < 1)
        p.probes = 1;
      int grid = 0;
      cudaError_t err = plan_tiles(p, kernel, 32 * NW, smem, p.probes, sm_count, &grid);
      if (err != cudaSuccess)
        return err;
      p.tiles_per_probe = p.tiles / p.probes;

      kernel<<<grid, 32 * NW, smem, stream>>>(p);

      if (launched_grid)
        *launched_grid = grid;

      return cudaGetLastError();
    }

    // the pair kernel forms the record index in the fp32 adder (ibl_math.cuh, projective form): even source
    // sizes of at most 2^22 texels per face; everything else runs the one-sample kernel
    bool pair_kernel_usable(PrefilterDnParams const &p)
    {
      return p.table_sector[0] != nullptr && p.table_sector[1] != nullptr && p.frames != nullptr && proj_usable(p.geom.ws, p.geom.hs);
    }
  }

  bool prefilter_batchable(int ws, int hs)
  {
    PrefilterDnParams p = {};
    p.geom = make_level_geom(ws, hs);
    p.table_sector[0] = p.table_sector[1] = reinterpret_cast<float4 const*>(&p);      // any non-null values: only the geometry decides
    p.frames = reinterpret_cast<float const*>(&p);
    return pair_kernel_usable(p);
  }

  cudaError_t launch_prefilter_dn(PrefilterDnParams const &p, int variant, int sm_count, cudaStream_t stream, int *launched_grid)
  {
    int rows = p.row_end - p.row_begin;
    if (rows <= 0 || p.wd <= 0)
      return cudaSuccess;

    // Automatic choice by slab size (measured on C2, tools/level_times.py) and table size (kBigTableEntries).
    if (variant == 0)
    {
      size_t texels = (size_t)rows * p.wd;
      bool big_table = p.table_count > kBigTableEntries;

      // the two biggest classes work on two samples at a time (prefilter_dp_kernel; measured on C2:
      // level 1 885 -> 862 us, level 2 277 -> 262, level 3 96 -> 88); launch_prefilter_dn falls back to
      // the one-sample kernel when the biased record index could wrap
      // Warps per tile follow ONE probe's slab (they decide the order of the sums: a batch must give the
      // words of single calls), the tile queues follow the whole launch.
      // Slabs between the two bounds take 8 warps per tile AND the tile queues: eight 45-degree sectors send fewer
      // warp-samples through the face selection than four of 90 (level 2 of C2: 32 % instead of 38 %; 247 -> 241 us),
      // which on the biggest slabs does not pay for the one-pair loop of that shape (level 1: 780 -> 805 us)
      if (texels >= kFourWarpTexels)
        variant = big_table ? 71 : 70;
      else if (texels >= kQueuedTexels)
        variant = big_table ? 67 : 66;
      else if (texels * (size_t)(p.probes > 1 ? p.probes : 1) >= kQueuedTexels)
        variant = big_table ? 91 : 90;
      else
        variant = big_table ? 73 : 72;      // slabs of at most kTailTexels never get here (prefilter_tail_kernel)
    }

    if (p.probes > 1 && !(((variant >= 70 && variant <= 99) || variant == 66 || variant == 67) && pair_kernel_usable(p)))
      return cudaErrorNotSupported;         // batches run on the pair kernel only (the caller checks prefilter_batchable)

    // two samples at a time; when the biased index could wrap, the same shape one sample at a time
    if (variant >= 81 && variant <= 86 && !pair_kernel_usable(p))
      variant = variant == 83 ? 53 : 51;

    if ((variant == 66 || variant == 67) && !pair_kernel_usable(p))
      variant = variant == 66 ? 53 : 54;

    if (variant >= 70 && variant <= 79 && !pair_kernel_usable(p))
    {
      static const int fallback[10] = { 51, 52, 53, 54, 51, 51, 51, 51, 51, 53 };
      variant = fallback[variant - 70];
    }

    const bool lean = p.probes <= 1 && p.signal.count == 0;

    switch (variant)
    {
      // the shapes the library picks by itself (and the one-sample forms they hand over to)
      //                        NW MINB SMEM  QUEUES
      // LEAN = no batch / peer-signal code in the kernel (single probe on one GPU: the common case; the
      // feature code costs ~1 % of a level through register allocation alone, profiles/r2_summary.md)
      case 70: return lean ? launch_dp<4, 8, true, true, 0, 1, false, false, true>(p, sm_count, stream, launched_grid) : launch_dp<4, 8, true, true>(p, sm_count, stream, launched_grid);
      case 71: return lean ? launch_dp<4, 8, false, true, 0, 1, false, false, true>(p, sm_count, stream, launched_grid) : launch_dp<4, 8, false, true>(p, sm_count, stream, launched_grid);
      case 72: return lean ? launch_dp<8, 4, true, false, 0, 1, false, false, true>(p, sm_count, stream, launched_grid) : launch_dp<8, 4, true, false>(p, sm_count, stream, launched_grid);
      case 73: return lean ? launch_dp<8, 4, false, false, 0, 1, false, false, true>(p, sm_count, stream, launched_grid) : launch_dp<8, 4, false, false>(p, sm_count, stream, launched_grid);
      case 66: return lean ? launch_dp<8, 4, true, true, 0, 1, false, false, true>(p, sm_count, stream, launched_grid) : launch_dp<8, 4, true, true>(p, sm_count, stream, launched_grid);
      case 67: return lean ? launch_dp<8, 4, false, true, 0, 1, false, false, true>(p, sm_count, stream, launched_grid) : launch_dp<8, 4, false, true>(p, sm_count, stream, launched_grid);
      case 90: return launch_dp<8, 4, true, true>(p, sm_count, stream, launched_grid);     // several probes' small slabs in one launch
      case 91: return launch_dp<8, 4, false, true>(p, sm_count, stream, launched_grid);
      //                        NW UNR MINB SMEM  QUEUES
      case 51: return launch_dn<4, 4, 8, true, true>(p, sm_count, stream, launched_grid);
      case 52: return launch_dn<4, 4, 8, false, true>(p, sm_count, stream, launched_grid);
      case 53: return launch_dn<8, 2, 4, true, false>(p, sm_count, stream, launched_grid);
      case 54: return launch_dn<8, 2, 4, false, false>(p, sm_count, stream, launched_grid);

#ifdef DATUM_IBL_AB_VARIANTS
      // A/B shapes of the tuning history (profiles/): only in the tools build (datum_b200.build --ab)
      case 74: return launch_dp<4, 8, true, false>(p, sm_count, stream, launched_grid);
      case 87: return launch_dp<4, 8, true, true, 0, 1, true>(p, sm_count, stream, launched_grid);    // r mantissa through IMAD.HI
      case 88: return launch_dp<8, 4, true, false, 0, 1, true>(p, sm_count, stream, launched_grid);
      case 92: return launch_dp<4, 8, true, true, 0, 1, false, true>(p, sm_count, stream, launched_grid);   // round 1's tile hand-out (one thread, no stealing)
      case 93: return launch_dp<4, 8, true, true, 0, 1, false, true, true>(p, sm_count, stream, launched_grid);   // ... and no batch / peer-signal code
      case 94: return launch_dp<4, 8, true, true, 0, 1, false, false, true>(p, sm_count, stream, launched_grid);  // stealing hand-out, no batch / peer-signal code
      // round 2's arithmetic (three-term directions, integer record index, four weight products) for A/B
      case 95: return launch_dp<4, 8, true, true, 0, 1, false, false, true, false>(p, sm_count, stream, launched_grid);
      case 96: return launch_dp<8, 4, true, false, 0, 1, false, false, true, false>(p, sm_count, stream, launched_grid);
      case 98: return launch_dp<4, 8, true, true, 0, 1, false, false, true, true, 2>(p, sm_count, stream, launched_grid);   // two 45-degree sectors per warp, one after the other
      case 75: return launch_dp<4, 8, true, true, 1, 1, false, false, true>(p, sm_count, stream, launched_grid);
      case 76: return launch_dp<4, 8, true, true, 2, 1, false, false, true>(p, sm_count, stream, launched_grid);
      case 77: return launch_dp<4, 8, true, true, 3, 1, false, false, true>(p, sm_count, stream, launched_grid);
      case 78: return launch_dp<4, 8, true, true, 4, 1, false, false, true>(p, sm_count, stream, launched_grid);
      case 79: return launch_dp<8, 4, true, false, 2>(p, sm_count, stream, launched_grid);
      case 81: return launch_dp<4, 9, true, true, 0, 1, false, false, true>(p, sm_count, stream, launched_grid);
      case 82: return launch_dp<4, 10, true, true, 0, 1, false, false, true>(p, sm_count, stream, launched_grid);
      case 83: return launch_dp<8, 5, true, false>(p, sm_count, stream, launched_grid);
      case 84: return launch_dp<4, 6, true, true, 0, 2, false, false, true>(p, sm_count, stream, launched_grid);
      case 85: return launch_dp<4, 8, true, true, 0, 2, false, false, true>(p, sm_count, stream, launched_grid);
      case 86: return launch_dp<4, 5, true, true, 0, 2, false, false, true>(p, sm_count, stream, launched_grid);
      case 50: return launch_dn<4, 4, 8, true, false>(p, sm_count, stream, launched_grid);
      case 55: return launch_dn<16, 1, 2, true, false>(p, sm_count, stream, launched_grid);
      case 56: return launch_dn<16, 1, 2, false, false>(p, sm_count, stream, launched_grid);
      case 57: return launch_dn<32, 1, 1, true, false>(p, sm_count, stream, launched_grid);
      case 58: return launch_dn<32, 1, 1, false, false>(p, sm_count, stream, launched_grid);
      case 60: return launch_dn<4, 2, 9, true, true>(p, sm_count, stream, launched_grid);
      case 61: return launch_dn<4, 2, 10, true, true>(p, sm_count, stream, launched_grid);
      case 62: return launch_dn<4, 4, 9, true, true>(p, sm_count, stream, launched_grid);
      case 63: return launch_dn<4, 2, 8, true, true>(p, sm_count, stream, launched_grid);
      case 64: return launch_dn<8, 2, 5, true, true>(p, sm_count, stream, launched_grid);
      case 65: return launch_dn<4, 4, 10, true, true>(p, sm_count, stream, launched_grid);
#endif
      default: return cudaErrorInvalidValue;
    }
  }
}
