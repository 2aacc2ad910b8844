// datum_b200 — SH9 irradiance projection of a cube map and its evaluation (sm_100a).
//
// Replaces the single-thread GLSL loop of data/project.comp:23-106 (reference
// paths relative to /root/reference).  The texel solid angle (project.comp:56-60)
// depends only on (x, y), not on the face, and its four-atan form cancels
// catastrophically in fp32 once faces exceed a few hundred texels, so it is
// evaluated ONCE per (x, y) in fp64 into a table that the context caches per
// face size.  The projection itself streams the slab once (16 B/texel RGBA32F):
// a thread owns one column of a face for a run of rows, keeps eight 16-byte loads in
// flight and accumulates six row moments per channel, folded into the 27 sums once per
// run (sh9_columns_kernel); then warp-shuffle and block-reduce in fp64.  Block partials
// are summed in block order by whichever block finishes last, so the result is run-to-run
// deterministic.  The first kernel (row segments, 27 FMAs per texel) stays for A/B.

#include "sh9.h"
#include "ibl_math.cuh"

#include <cuda_runtime.h>
#include <cstdint>

namespace ibl
{
  // ---- solid angle table -------------------------------------------------------

  __device__ __forceinline__ double corner_angle(double x, double y) { return atan2(x * y, sqrt(x * x + y * y + 1.0)); }

  __global__ void __launch_bounds__(256) sh9_weights_kernel(float *__restrict__ weights, int w, int h)
  {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= w * h)
      return;

    int x = idx % w, y = idx / w;

    // project.comp:53, 56-60
    double u = 2 * (x + 0.5) / w - 1;
    double v = 2 * (y + 0.5) / h - 1;
    double x0 = u - 1.0 / w, x1 = u + 1.0 / w;
    double y0 = v - 1.0 / h, y1 = v + 1.0 / h;

    weights[idx] = (float)(corner_angle(x0, y0) - corner_angle(x0, y1) - corner_angle(x1, y0) + corner_angle(x1, y1));
  }

  // ---- projection ----------------------------------------------------------------

  // L2 residency: the texel stream is read once (evict first, do not allocate in L1), the solid-angle
  // table is read once per face and should survive the stream in between (evict last)
  __device__ __forceinline__ unsigned long long l2_policy_evict_first()
  {
    unsigned long long p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
  }

  __device__ __forceinline__ unsigned long long l2_policy_evict_last()
  {
    unsigned long long p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
  }

  __device__ __forceinline__ float4 ldg_stream(float4 const *ptr, unsigned long long policy)
  {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(ptr), "l"(policy));
    return v;
  }

  __device__ __forceinline__ float ldg_keep(float const *ptr, unsigned long long policy)
  {
    float v;
    asm volatile("ld.global.nc.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(v) : "l"(ptr), "l"(policy));
    return v;
  }

  template<int FORMAT>
  __device__ __forceinline__ void load_texel(void const *__restrict__ level0, size_t idx, unsigned long long stream_policy, float &r, float &g, float &b)
  {
    if (FORMAT == 0)
    {
      // color.h:164-172 with the 1/511 folded into the scale (<= 1 ulp from the reference decode)
      uint32_t c = __ldg(reinterpret_cast<uint32_t const *>(level0) + idx);
      float s = u2f((((c >> 27) & 0x1Fu) + 112u) << 23) * (1.0f / 511.0f);
      r = (float)((c >> 0) & 0x1FFu) * s;
      g = (float)((c >> 9) & 0x1FFu) * s;
      b = (float)((c >> 18) & 0x1FFu) * s;
    }
    else if (FORMAT == 1)
    {
      float4 c = ldg_stream(reinterpret_cast<float4 const *>(level0) + idx, stream_policy);
      r = c.x; g = c.y; b = c.z;
    }
    else
    {
      // RGBA16F: one 8-byte load, the halves widened exactly
      uint32_t lo, hi;
      asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.u32 {%0,%1}, [%2], %3;" : "=r"(lo), "=r"(hi) : "l"(reinterpret_cast<uint2 const *>(level0) + idx), "l"(stream_policy));
      asm("{ .reg .b16 x, y; mov.b32 {x, y}, %2; cvt.f32.f16 %0, x; cvt.f32.f16 %1, y; }" : "=f"(r), "=f"(g) : "r"(lo));
      asm("{ .reg .b16 x, y; mov.b32 {x, y}, %1; cvt.f32.f16 %0, x; }" : "=f"(b) : "r"(hi));
    }
  }

  // acc[3*k + c] += weight * color[c] * M_k(ray) with the MONOMIALS
  //     M = 1, y, z, x, xy, yz, z^2, zx, x^2 - y^2
  // of the basis functions of project.comp:64-92; their constant factors (and the "3 z^2 - 1" of
  // Y6) are applied once per block in sh9_basis_from_monomials: 11 multiplies less per texel.
  __device__ __forceinline__ void sh9_accumulate(float acc[28], float wr, float wg, float wb, float rx, float ry, float rz)
  {
    float mono[9];
    mono[0] = 1.0f;
    mono[1] = ry;
    mono[2] = rz;
    mono[3] = rx;
    mono[4] = rx * ry;
    mono[5] = ry * rz;
    mono[6] = rz * rz;
    mono[7] = rz * rx;
    mono[8] = fmaf(rx, rx, -ry * ry);

    acc[0] += wr; acc[1] += wg; acc[2] += wb;

    #pragma unroll
    for(int k = 1; k < 9; ++k)
    {
      acc[3*k + 0] = fmaf(wr, mono[k], acc[3*k + 0]);
      acc[3*k + 1] = fmaf(wg, mono[k], acc[3*k + 1]);
      acc[3*k + 2] = fmaf(wb, mono[k], acc[3*k + 2]);
    }
  }

  // monomial sums -> basis sums (fp64, once per block): project.comp:64-92's constants
  __device__ __forceinline__ double sh9_basis_from_monomials(int k, double const mono[28])
  {
    int band = k / 3, c = k - 3 * band;
    switch (band)
    {
      case 0: return 0.282095 * mono[k];
      case 1: case 2: case 3: return 0.488603 * mono[k];
      case 4: case 5: case 7: return 1.092548 * mono[k];
      case 6: return 0.315392 * (3.0 * mono[k] - mono[c]);
      case 8: return 0.546274 * mono[k];
      default: return mono[k];     // k == 27: the weight sum
    }
  }

  constexpr int kSh9Threads = 256;
  constexpr int kSh9Unroll = 4;                               // texels per thread and work item: four 16-byte loads in flight
  constexpr int kSh9Segment = kSh9Threads * kSh9Unroll;       // texels of one row a CTA takes at a time

  // face rays as in data/convolve.comp:85-100 (equal to project.comp:27-32's quaternions);
  // (a, b, c) = (u, v, 1) / |(u, v, 1)|
  template<int FACE>
  __device__ __forceinline__ void face_ray(float a, float b, float c, float &rx, float &ry, float &rz)
  {
    switch (FACE)
    {
      case 0: rx = c;  ry = b;  rz = a;  break;
      case 1: rx = -c; ry = b;  rz = -a; break;
      case 2: rx = a;  ry = -c; rz = -b; break;
      case 3: rx = a;  ry = c;  rz = b;  break;
      case 4: rx = a;  ry = b;  rz = -c; break;
      default: rx = -a; ry = b; rz = c;  break;
    }
  }

  // One segment of one row of one face: the CTA's threads take texels x0 + j*256 + tid.  All loads of
  // the segment are issued before the arithmetic of the first texel: memory-level parallelism is what
  // keeps this kernel near the HBM roofline (16 B per texel against ~64 instructions).
  template<int FORMAT, int FACE>
  __device__ __forceinline__ void sh9_row_segment(void const *__restrict__ level0, float const *__restrict__ weights, int w, size_t row_offset, int weight_offset, int x0, float v, float vv1, float two_inv_w, float u_bias, unsigned long long stream_policy, unsigned long long keep_policy, float acc[28])
  {
    float r[kSh9Unroll], g[kSh9Unroll], bl[kSh9Unroll], weight[kSh9Unroll];

    #pragma unroll
    for(int j = 0; j < kSh9Unroll; ++j)
    {
      int x = x0 + j * kSh9Threads + (int)threadIdx.x;
      if (x < w)
      {
        load_texel<FORMAT>(level0, row_offset + x, stream_policy, r[j], g[j], bl[j]);

        // the solid angle is symmetric in x (and y, see weight_offset): only one quadrant of the table is ever
        // touched, 17 MB at 4096^2, which the L2 keeps between faces
        int xs = x < w - 1 - x ? x : w - 1 - x;
        weight[j] = ldg_keep(weights + weight_offset + xs, keep_policy);
      }
      else
      {
        r[j] = g[j] = bl[j] = 0.0f;
        weight[j] = 0.0f;          // a texel past the row end adds exact zeros
      }
    }

    #pragma unroll
    for(int j = 0; j < kSh9Unroll; ++j)
    {
      int x = x0 + j * kSh9Threads + (int)threadIdx.x;

      // project.comp:53-54: u = 2 (x + .5) / w - 1, ray = normalize(rot * (u, v, -1))
      float u = fmaf((float)x, two_inv_w, u_bias);
      float inv = rsqrtf(fmaf(u, u, vv1));

      float rx, ry, rz;
      face_ray<FACE>(u * inv, v * inv, inv, rx, ry, rz);

      sh9_accumulate(acc, weight[j] * r[j], weight[j] * g[j], weight[j] * bl[j], rx, ry, rz);
      acc[27] += weight[j];
    }
  }

  template<int FORMAT>
  __global__ void __launch_bounds__(kSh9Threads, 4) sh9_partial_kernel(void const *__restrict__ level0, float const *__restrict__ weights, int w, int h, int row_begin, int row_end, double *__restrict__ block_partials, unsigned int *__restrict__ done_counter, double *__restrict__ partial, Sh9Peers peers)
  {
    float acc[28];
    #pragma unroll
    for(int k = 0; k < 28; ++k)
      acc[k] = 0.0f;

    const float inv_w = 1.0f / (float)w, inv_h = 1.0f / (float)h;
    const float two_inv_w = 2.0f * inv_w, u_bias = inv_w - 1.0f;
    const unsigned long long stream_policy = l2_policy_evict_first(), keep_policy = l2_policy_evict_last();

    // work items: (row of the slab, segment of that row) in row order; rows are face-major, so the
    // slab of a GPU that shares the cube with others is one contiguous range of the level.  (Tried and
    // measured slower on 4096^2 faces, 0.345 ms as is: item order with the six faces of a table stretch
    // side by side, 0.42 ms; the solid angle from a Taylor form instead of the table, 0.38 ms; five row
    // moments per channel folded once per row, 0.40 ms; the texel stream through cp.async.bulk into a
    // four-stage shared-memory ring with mbarriers, 0.41 ms — profiles/r1_summary.md 0.3.)
    const int segments = (w + kSh9Segment - 1) / kSh9Segment;
    const long long items = (long long)(row_end - row_begin) * segments;

    for(long long item = blockIdx.x; item < items; item += gridDim.x)
    {
      int row = row_begin + (int)(item / segments);
      int x0 = (int)(item % segments) * kSh9Segment;
      int face = row / h;
      int y = row - face * h;

      float v = 2.0f * ((float)y + 0.5f) * inv_h - 1.0f;
      float vv1 = fmaf(v, v, 1.0f);
      size_t row_offset = (size_t)row * w;
      int weight_offset = (y < h - 1 - y ? y : h - 1 - y) * w;

      switch (face)
      {
        case 0: sh9_row_segment<FORMAT, 0>(level0, weights, w, row_offset, weight_offset, x0, v, vv1, two_inv_w, u_bias, stream_policy, keep_policy, acc); break;
        case 1: sh9_row_segment<FORMAT, 1>(level0, weights, w, row_offset, weight_offset, x0, v, vv1, two_inv_w, u_bias, stream_policy, keep_policy, acc); break;
        case 2: sh9_row_segment<FORMAT, 2>(level0, weights, w, row_offset, weight_offset, x0, v, vv1, two_inv_w, u_bias, stream_policy, keep_policy, acc); break;
        case 3: sh9_row_segment<FORMAT, 3>(level0, weights, w, row_offset, weight_offset, x0, v, vv1, two_inv_w, u_bias, stream_policy, keep_policy, acc); break;
        case 4: sh9_row_segment<FORMAT, 4>(level0, weights, w, row_offset, weight_offset, x0, v, vv1, two_inv_w, u_bias, stream_policy, keep_policy, acc); break;
        default: sh9_row_segment<FORMAT, 5>(level0, weights, w, row_offset, weight_offset, x0, v, vv1, two_inv_w, u_bias, stream_policy, keep_policy, acc); break;
      }
    }

    // ---- warp shuffle reduction in fp64, then across the block's warps ----
    __shared__ double s_partial[kSh9Threads / 32][28];

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    #pragma unroll
    for(int k = 0; k < 28; ++k)
    {
      double v = (double)acc[k];
      #pragma unroll
      for(int offset = 16; offset > 0; offset >>= 1)
        v += __shfl_down_sync(0xffffffffu, v, offset);

      if (lane == 0)
        s_partial[warp][k] = v;
    }

    __syncthreads();

    __shared__ double s_mono[28];

    if (threadIdx.x < 28)
    {
      double v = 0;
      #pragma unroll
      for(int wi = 0; wi < kSh9Threads / 32; ++wi)
        v += s_partial[wi][threadIdx.x];

      s_mono[threadIdx.x] = v;
    }

    __syncthreads();

    if (threadIdx.x < 28)
      block_partials[(size_t)blockIdx.x * 28 + threadIdx.x] = sh9_basis_from_monomials(threadIdx.x, s_mono);

    // ---- the block that finishes last sums the block partials, in block order: deterministic, and one
    //      launch instead of two (a separate 1-CTA combine kernel cost 7.5 us, as much as a 256^2 cube) ----
    __shared__ bool s_last;

    __threadfence();
    __syncthreads();

    if (threadIdx.x == 0)
    {
      unsigned int ticket = atomicAdd(done_counter, 1u);
      s_last = ticket == gridDim.x - 1;
    }

    __syncthreads();

    if (!s_last)
      return;

    __threadfence();

    // thread (k, part): component k over the blocks part, part + kParts, ...; then the parts in order
    constexpr int kParts = kSh9Threads / 28;              // 9
    __shared__ double s_part[kParts][28];

    if (threadIdx.x < kParts * 28)
    {
      int k = threadIdx.x % 28, part = threadIdx.x / 28;
      double v = 0;

      #pragma unroll 8
      for(int i = part; i < (int)gridDim.x; i += kParts)
        v += __ldcg(block_partials + (size_t)i * 28 + k);

      s_part[part][k] = v;
    }

    __syncthreads();

    if (threadIdx.x < 28)
    {
      double v = 0;
      #pragma unroll
      for(int part = 0; part < kParts; ++part)
        v += s_part[part][threadIdx.x];

      partial[threadIdx.x] = v;

      // a cube shared by several GPUs: the slab's sums go straight into every peer's array
      for(int k = 0; k < peers.count; ++k)
        peers.slots[k][threadIdx.x] = v;
    }

    // ... and the peers' streams are told (they wait on their arrival counter, no kernel in between)
    if (peers.count > 0 && peers.arrive[0])
    {
      __threadfence_system();
      __syncthreads();

      if ((int)threadIdx.x < peers.count)
        asm volatile("red.release.sys.global.add.u32 [%0], 1;" :: "l"(peers.arrive[threadIdx.x]) : "memory");
    }

    if (threadIdx.x == 0)
      *done_counter = 0;      // ready for the next launch on this stream
  }

  // ---- projection, column strips (the kernel in use) ------------------------------------------------
  //
  // The row-segment kernel above spends ~84 instructions per texel (27 accumulating FMAs with three
  // distinct register operands, the monomials, the ray, item bookkeeping every four texels) and sits
  // where the instruction-issue and HBM roofs meet: 0.71 of the measured copy bandwidth with exactly
  // the algorithmic traffic.  Here a thread owns ONE COLUMN x of a face for a run of rows.  With
  // (a, b, c) = (u, v, 1)/|(u, v, 1)| every basis monomial is a product of at most two of a, b, c, and
  // u is a constant of the thread, so per channel six row moments carry everything:
  //     M0 = sum q      M1 = sum q i      M2 = sum q i v      M3 = sum q i^2      M4 = sum q i^2 v      M5 = sum q i^2 v^2
  // (q = solid angle x colour, i = 1/|(u, v, 1)|): 4 products + 5 FMAs + 1 add per channel instead of
  // 8 + 9 FMAs, ~34 instructions per texel.  At the end of a run the 18 moments are folded into the 27
  // monomial sums with the thread's powers of u and the face's axis permutation (once per run, not per
  // texel).  Loads: eight rows of the column in flight per thread before any arithmetic (16-byte texel,
  // 4-byte solid angle), a warp reads 512 contiguous bytes of each row.
  constexpr int kSh9ColThreads = 256;
  constexpr int kSh9ColUnroll = 8;

  // 18 moments + the thread's u -> monomial sums of one channel triple, per face (data/convolve.comp:85-100)
  template<int FACE>
  __device__ __forceinline__ void sh9_fold(float const M[6][3], float u, float acc[28])
  {
    const float uu = u * u;

    #pragma unroll
    for(int ch = 0; ch < 3; ++ch)
    {
      // sums of q times: 1, a, b, c, aa, ab, ac, bb, bc, cc
      float s1 = M[0][ch];
      float sa = u * M[1][ch], sb = M[2][ch], sc = M[1][ch];
      float saa = uu * M[3][ch], sab = u * M[4][ch], sac = u * M[3][ch], sbb = M[5][ch], sbc = M[4][ch], scc = M[3][ch];

      // ray = (rx, ry, rz) as signed picks of (a, b, c); monomials y, z, x, xy, yz, zz, zx, xx - yy
      float y, z, x, xy, yz, zz, zx, xxyy;
      switch (FACE)
      {
        case 0:  x = sc;  y = sb;  z = sa;  xy = sbc;  yz = sab;  zz = saa; zx = sac;  xxyy = scc - sbb; break;   // ( c,  b,  a)
        case 1:  x = -sc; y = sb;  z = -sa; xy = -sbc; yz = -sab; zz = saa; zx = sac;  xxyy = scc - sbb; break;   // (-c,  b, -a)
        case 2:  x = sa;  y = -sc; z = -sb; xy = -sac; yz = sbc;  zz = sbb; zx = -sab; xxyy = saa - scc; break;   // ( a, -c, -b)
        case 3:  x = sa;  y = sc;  z = sb;  xy = sac;  yz = sbc;  zz = sbb; zx = sab;  xxyy = saa - scc; break;   // ( a,  c,  b)
        case 4:  x = sa;  y = sb;  z = -sc; xy = sab;  yz = -sbc; zz = scc; zx = -sac; xxyy = saa - sbb; break;   // ( a,  b, -c)
        default: x = -sa; y = sb;  z = sc;  xy = -sab; yz = sbc;  zz = scc; zx = -sac; xxyy = saa - sbb; break;   // (-a,  b,  c)
      }

      acc[0 + ch] += s1;
      acc[3 + ch] += y;
      acc[6 + ch] += z;
      acc[9 + ch] += x;
      acc[12 + ch] += xy;
      acc[15 + ch] += yz;
      acc[18 + ch] += zz;
      acc[21 + ch] += zx;
      acc[24 + ch] += xxyy;
    }
  }

  __device__ __forceinline__ void sh9_fold_face(int face, float const M[6][3], float u, float acc[28])
  {
    switch (face)
    {
      case 0: sh9_fold<0>(M, u, acc); break;
      case 1: sh9_fold<1>(M, u, acc); break;
      case 2: sh9_fold<2>(M, u, acc); break;
      case 3: sh9_fold<3>(M, u, acc); break;
      case 4: sh9_fold<4>(M, u, acc); break;
      default: sh9_fold<5>(M, u, acc); break;
    }
  }

  template<int FORMAT>
  __global__ void __launch_bounds__(kSh9ColThreads, 2) sh9_columns_kernel(void const *__restrict__ level0, float const *__restrict__ weights, int w, int h, int row_begin, int row_end, int rows_per_item, double *__restrict__ block_partials, unsigned int *__restrict__ done_counter, double *__restrict__ partial, Sh9Peers peers, size_t probe_stride)
  {
    // blockIdx.y = which cube of a batch (datum_ibl_bake_probes): cubes probe_stride bytes apart, their
    // block partials, tickets and results back to back
    level0 = static_cast<unsigned char const*>(level0) + (size_t)blockIdx.y * probe_stride;
    block_partials += (size_t)blockIdx.y * gridDim.x * 28;
    done_counter += blockIdx.y;
    partial += (size_t)blockIdx.y * 28;

    float acc[28];
    #pragma unroll
    for(int k = 0; k < 28; ++k)
      acc[k] = 0.0f;

    const float inv_w = 1.0f / (float)w, inv_h = 1.0f / (float)h;
    const unsigned long long stream_policy = l2_policy_evict_first(), keep_policy = l2_policy_evict_last();

    // work items: (run of rows_per_item rows of the slab, block of 256 columns), column blocks fastest so that
    // the CTAs in flight read neighbouring 4 KB pieces of the same rows
    const int col_blocks = (w + kSh9ColThreads - 1) / kSh9ColThreads;
    const int runs = (row_end - row_begin + rows_per_item - 1) / rows_per_item;
    const long long items = (long long)runs * col_blocks;

    for(long long item = blockIdx.x; item < items; item += gridDim.x)
    {
      const int run = (int)(item / col_blocks);
      const int x = (int)(item - (long long)run * col_blocks) * kSh9ColThreads + (int)threadIdx.x;
      const bool live = x < w;

      // project.comp:53: u = 2 (x + .5) / w - 1
      const float u = live ? 2.0f * ((float)x + 0.5f) * inv_w - 1.0f : 0.0f;
      const float uu1 = fmaf(u, u, 1.0f);
      const int xs = x < w - 1 - x ? x : w - 1 - x;      // the solid angle is symmetric in x and y: one quadrant of the table is ever touched

      int row = row_begin + run * rows_per_item;
      const int run_end = min(row + rows_per_item, row_end);

      // a run may cross into the next face (faces are stacked in the row index): one fold per face piece
      while (row < run_end)
      {
        const int face = row / h;
        const int piece_end = min(run_end, (face + 1) * h);

        float M[6][3];
        #pragma unroll
        for(int k = 0; k < 6; ++k)
          M[k][0] = M[k][1] = M[k][2] = 0.0f;
        float wsum = 0.0f;

        for(; row < piece_end; row += kSh9ColUnroll)
        {
          float r[kSh9ColUnroll], g[kSh9ColUnroll], bl[kSh9ColUnroll], weight[kSh9ColUnroll];

          #pragma unroll
          for(int j = 0; j < kSh9ColUnroll; ++j)
          {
            const int rj = row + j;
            if (live && rj < piece_end)
            {
              const int y = rj - face * h;
              const int ys = y < h - 1 - y ? y : h - 1 - y;
              load_texel<FORMAT>(level0, (size_t)rj * w + x, stream_policy, r[j], g[j], bl[j]);
              weight[j] = ldg_keep(weights + (size_t)ys * w + xs, keep_policy);
            }
            else
            {
              r[j] = g[j] = bl[j] = 0.0f;
              weight[j] = 0.0f;          // a texel past the piece adds exact zeros
            }
          }

          #pragma unroll
          for(int j = 0; j < kSh9ColUnroll; ++j)
          {
            // project.comp:53-54: v = 2 (y + .5) / h - 1, ray = normalize(rot * (u, v, -1))
            const int y = row + j - face * h;
            const float v = 2.0f * ((float)y + 0.5f) * inv_h - 1.0f;
            const float i1 = rsqrtf(fmaf(v, v, uu1));
            const float i1v = i1 * v;
            const float i2 = i1 * i1;
            const float i2v = i2 * v;
            const float i2vv = i2v * v;

            const float q[3] = { weight[j] * r[j], weight[j] * g[j], weight[j] * bl[j] };

            #pragma unroll
            for(int ch = 0; ch < 3; ++ch)
            {
              M[0][ch] += q[ch];
              M[1][ch] = fmaf(q[ch], i1, M[1][ch]);
              M[2][ch] = fmaf(q[ch], i1v, M[2][ch]);
              M[3][ch] = fmaf(q[ch], i2, M[3][ch]);
              M[4][ch] = fmaf(q[ch], i2v, M[4][ch]);
              M[5][ch] = fmaf(q[ch], i2vv, M[5][ch]);
            }
            wsum += weight[j];
          }
        }

        row = piece_end;
        sh9_fold_face(face, M, u, acc);
        acc[27] += wsum;
      }
    }

    // ---- warp shuffle reduction in fp64, then across the block's warps (as in the row-segment kernel) ----
    __shared__ double s_partial[kSh9ColThreads / 32][28];

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    #pragma unroll
    for(int k = 0; k < 28; ++k)
    {
      double v = (double)acc[k];
      #pragma unroll
      for(int offset = 16; offset > 0; offset >>= 1)
        v += __shfl_down_sync(0xffffffffu, v, offset);

      if (lane == 0)
        s_partial[warp][k] = v;
    }

    __syncthreads();

    __shared__ double s_mono[28];

    if (threadIdx.x < 28)
    {
      double v = 0;
      #pragma unroll
      for(int wi = 0; wi < kSh9ColThreads / 32; ++wi)
        v += s_partial[wi][threadIdx.x];

      s_mono[threadIdx.x] = v;
    }

    __syncthreads();

    if (threadIdx.x < 28)
      block_partials[(size_t)blockIdx.x * 28 + threadIdx.x] = sh9_basis_from_monomials(threadIdx.x, s_mono);

    // ---- the block that finishes last sums the block partials, in block order: deterministic, one launch ----
    __shared__ bool s_last;

    __threadfence();
    __syncthreads();

    if (threadIdx.x == 0)
    {
      unsigned int ticket = atomicAdd(done_counter, 1u);
      s_last = ticket == gridDim.x - 1;
    }

    __syncthreads();

    if (!s_last)
      return;

    __threadfence();

    constexpr int kParts = kSh9ColThreads / 28;              // 9
    __shared__ double s_part[kParts][28];

    if (threadIdx.x < kParts * 28)
    {
      int k = threadIdx.x % 28, part = threadIdx.x / 28;
      double v = 0;

      #pragma unroll 8
      for(int i = part; i < (int)gridDim.x; i += kParts)
        v += __ldcg(block_partials + (size_t)i * 28 + k);

      s_part[part][k] = v;
    }

    __syncthreads();

    if (threadIdx.x < 28)
    {
      double v = 0;
      #pragma unroll
      for(int part = 0; part < kParts; ++part)
        v += s_part[part][threadIdx.x];

      partial[threadIdx.x] = v;

      // a cube shared by several GPUs: the slab's sums go straight into every peer's array
      for(int k = 0; k < peers.count; ++k)
        peers.slots[k][threadIdx.x] = v;
    }

    // ... and the peers' streams are told (they wait on their arrival counter, no kernel in between)
    if (peers.count > 0 && peers.arrive[0])
    {
      __threadfence_system();
      __syncthreads();

      if ((int)threadIdx.x < peers.count)
        asm volatile("red.release.sys.global.add.u32 [%0], 1;" :: "l"(peers.arrive[threadIdx.x]) : "memory");
    }

    if (threadIdx.x == 0)
      *done_counter = 0;      // ready for the next launch on this stream
  }

  // ---- irradiance cube from SH9: data/lighting.inc:351-366, 371 ---------------------

  __global__ void __launch_bounds__(256) sh9_irradiance_kernel(Sh9Coefficients sh, int w, int h, uint32_t *__restrict__ words, float *__restrict__ f32)
  {
    size_t total = (size_t)6 * w * h;
    for(size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x)
    {
      int x = (int)(idx % w);
      int y = (int)((idx / w) % h);
      int face = (int)(idx / ((size_t)w * h));

      float u = 2.0f * ((float)x + 0.5f) / (float)w - 1.0f;
      float v = 2.0f * ((float)y + 0.5f) / (float)h - 1.0f;
      float inv = rsqrtf(fmaf(u, u, fmaf(v, v, 1.0f)));
      float a = u * inv, b = v * inv, c = inv;

      float nx, ny, nz;
      switch (face)
      {
        case 0: nx = c;  ny = b;  nz = a;  break;
        case 1: nx = -c; ny = b;  nz = -a; break;
        case 2: nx = a;  ny = -c; nz = -b; break;
        case 3: nx = a;  ny = c;  nz = b;  break;
        case 4: nx = a;  ny = b;  nz = -c; break;
        default: nx = -a; ny = b; nz = c;  break;
      }

      float L[9];
      L[0] = 3.141593f * 0.282095f;
      L[1] = 2.094395f * 0.488603f * ny;
      L[2] = 2.094395f * 0.488603f * nz;
      L[3] = 2.094395f * 0.488603f * nx;
      L[4] = 0.785398f * 1.092548f * nx * ny;
      L[5] = 0.785398f * 1.092548f * ny * nz;
      L[6] = 0.785398f * 0.315392f * (3.0f * nz * nz - 1.0f);
      L[7] = 0.785398f * 1.092548f * nz * nx;
      L[8] = 0.785398f * 0.546274f * (nx * nx - ny * ny);

      float rgb[3] = { 0.0f, 0.0f, 0.0f };
      #pragma unroll
      for(int k = 0; k < 9; ++k)
      {
        rgb[0] = fmaf(L[k], sh.v[3*k + 0], rgb[0]);
        rgb[1] = fmaf(L[k], sh.v[3*k + 1], rgb[1]);
        rgb[2] = fmaf(L[k], sh.v[3*k + 2], rgb[2]);
      }

      rgb[0] = fmaxf(rgb[0], 0.0f); rgb[1] = fmaxf(rgb[1], 0.0f); rgb[2] = fmaxf(rgb[2], 0.0f);

      if (words)
        words[idx] = rgbe_encode(rgb[0], rgb[1], rgb[2]);

      if (f32)
      {
        f32[3*idx + 0] = rgb[0]; f32[3*idx + 1] = rgb[1]; f32[3*idx + 2] = rgb[2];
      }
    }
  }

  // ---- launchers ----------------------------------------------------------------------

  cudaError_t launch_sh9_weights(float *weights, int w, int h, cudaStream_t stream)
  {
    int total = w * h;
    sh9_weights_kernel<<<(total + 255) / 256, 256, 0, stream>>>(weights, w, h);
    return cudaGetLastError();
  }

  int sh9_partial_blocks(int w, int h, int sm_count)
  {
    // upper bound for any slab of the cube and either kernel: up to 4 resident CTAs per SM
    long long items = (long long)6 * h * ((w + kSh9ColThreads - 1) / kSh9ColThreads);
    long long cap = (long long)sm_count * 4;
    return (int)(items < cap ? (items < 1 ? 1 : items) : cap);
  }

  cudaError_t launch_sh9_partial(void const *level0, int format, float const *weights, int w, int h, int row_begin, int row_end, double *block_partials, int blocks, unsigned int *done_counter, double *partial, Sh9Peers const &peers, int sm_count, cudaStream_t stream, int kernel, int rows_per_item, int probes, size_t probe_stride)
  {
    if (probes < 1)
      probes = 1;

    if (kernel == 1)
    {
      // the row-segment kernel (A/B; one cube at a time)
      if (probes != 1)
        return cudaErrorNotSupported;

      if (format == 0)
        sh9_partial_kernel<0><<<blocks, kSh9Threads, 0, stream>>>(level0, weights, w, h, row_begin, row_end, block_partials, done_counter, partial, peers);
      else if (format == 1)
        sh9_partial_kernel<1><<<blocks, kSh9Threads, 0, stream>>>(level0, weights, w, h, row_begin, row_end, block_partials, done_counter, partial, peers);
      else
        sh9_partial_kernel<2><<<blocks, kSh9Threads, 0, stream>>>(level0, weights, w, h, row_begin, row_end, block_partials, done_counter, partial, peers);

      return cudaGetLastError();
    }

    // column strips: two CTAs per SM; runs short enough that the slab makes several items per resident CTA
    // (the fold costs ~60 FMAs per run and thread: at least 8 rows per run keeps it under 8 per texel)
    const int resident = sm_count * 2;
    const int col_blocks = (w + kSh9ColThreads - 1) / kSh9ColThreads;
    const int rows = row_end - row_begin;

    if (rows_per_item <= 0)
    {
      long long want_items = 6ll * resident;
      long long r = ((long long)rows * col_blocks + want_items - 1) / want_items;      // from ONE cube: a batch gives the bits of single calls
      rows_per_item = (int)(r < 8 ? 8 : (r > 64 ? 64 : r));
      rows_per_item = (rows_per_item + kSh9ColUnroll - 1) / kSh9ColUnroll * kSh9ColUnroll;
    }

    long long items = (long long)((rows + rows_per_item - 1) / rows_per_item) * col_blocks;
    int grid = (int)(items < resident ? (items < 1 ? 1 : items) : resident);     // per cube, whatever the batch
    if (grid > blocks)
      grid = blocks;      // the scratch holds `blocks` partial rows per cube

    dim3 cubes(grid, probes);

    if (format == 0)
      sh9_columns_kernel<0><<<cubes, kSh9ColThreads, 0, stream>>>(level0, weights, w, h, row_begin, row_end, rows_per_item, block_partials, done_counter, partial, peers, probe_stride);
    else if (format == 1)
      sh9_columns_kernel<1><<<cubes, kSh9ColThreads, 0, stream>>>(level0, weights, w, h, row_begin, row_end, rows_per_item, block_partials, done_counter, partial, peers, probe_stride);
    else
      sh9_columns_kernel<2><<<cubes, kSh9ColThreads, 0, stream>>>(level0, weights, w, h, row_begin, row_end, rows_per_item, block_partials, done_counter, partial, peers, probe_stride);

    return cudaGetLastError();
  }

  cudaError_t launch_sh9_irradiance(Sh9Coefficients const &sh, int w, int h, uint32_t *words, float *f32, int sm_count, cudaStream_t stream)
  {
    size_t total = (size_t)6 * w * h;
    size_t blocks = (total + 255) / 256;
    size_t cap = (size_t)sm_count * 8;
    int grid = (int)(blocks < cap ? blocks : cap);
    if (grid < 1)
      grid = 1;

    sh9_irradiance_kernel<<<grid, 256, 0, stream>>>(sh, w, h, words, f32);

    return cudaGetLastError();
  }
}
