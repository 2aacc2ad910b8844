// datum_b200 — device helpers of the pair and tail kernels, shared by the rgbe chain (prefilter_dn.cu) and the
// float chains (prefilter_f.cu); internal to libdatum_ibl_cuda.
//
// What both chains compute alike lives here: the packed fp32 ops, the pair table entries and the projective
// footprint coordinates of two samples, the tile hand-out, the per-tile frame, same-face band count and
// CTA reduction, and the arrival signal of a probe shared by several GPUs.  What differs between the chains
// stays in each kernel: the record layout, the tap fetch and decode, the store (peer stores included) and the
// batch addressing (probe strides).  Nothing here depends on which chain calls it.
//
// The rgbe kernels are sensitive to everything compiled into their bodies (DESIGN.md §4.1): these helpers keep
// the statement order of the code they replace, and take output references rather than returning structs,
// so that every kernel of both files compiles to the same SASS as before they were shared.
#pragma once

#include "prefilter.h"
#include "ibl_math.cuh"

#include <cuda_runtime.h>

namespace ibl
{
  // packed two-wide fp32 (fma.rn.f32x2 -> SASS FFMA2/FMUL2/FADD2): same lanes as two scalar
  // ops, one issue slot; every element is rounded exactly like the scalar form
  typedef unsigned long long f32x2;

  __device__ __forceinline__ f32x2 pack2(float lo, float hi) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
  __device__ __forceinline__ void unpack2(f32x2 a, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(a)); }
  __device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
  __device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) { f32x2 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
  __device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) { f32x2 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
  __device__ __forceinline__ f32x2 bcast2(float v) { return pack2(v, v); }

  __device__ __forceinline__ f32x2 neg2(f32x2 a)
  {
    float lo, hi;
    unpack2(a, lo, hi);
    return pack2(-lo, -hi);
  }

  // A record pointer the compiler cannot re-associate: base + idx (unsigned 32-bit, bias included) is then
  // one IMAD.WIDE.U32; otherwise the compiler turns the 64-bit sum into four adds.
  template<typename R>
  __device__ __forceinline__ R const *opaque(R const *ptr)
  {
    asm volatile("" : "+l"(ptr));
    return ptr;
  }

  // ---- two samples at a time ----------------------------------------------------------------

  struct Sums
  {
    f32x2 rg, bb;       // (r, g) and the b sums of the two samples of a pair
  };

  struct PairEntry
  {
    f32x2 lx, ly, lz, wh;   // each: (sample a, sample b)
  };

  template<bool SMEM_TABLE>
  __device__ __forceinline__ PairEntry load_pair(float4 const *t)
  {
    ulonglong2 const *q = reinterpret_cast<ulonglong2 const*>(t);
    ulonglong2 lo = SMEM_TABLE ? q[0] : __ldg(q);
    ulonglong2 hi = SMEM_TABLE ? q[1] : __ldg(q + 1);
    return PairEntry{ lo.x, lo.y, hi.x, hi.y };
  }

  struct Frame
  {
    Vec3f T, B, N;
  };

  // ---- projective form (ibl_math.cuh: face_footprint_proj, cube_footprint_proj, footprint_weights_diff) ----
  //
  // Entries hold (lx/lz, ly/lz): a direction is two packed multiply-adds per component.  On the texel's
  // own face the rows arrive folded (fold_face_row), so integer part and fraction of a texel coordinate
  // are one FFMA2 each straight from the quotient; the record index is formed in the fp32 adder
  // (magic + i + j*ws, exact) and its bits go into IMAD.WIDE as they are.  The right-hand taps' weights
  // are differences (each chain's gather).  Per pair of samples: 32 packed fp32 operations and 10 integer
  // multiply-adds where round 2's form (prefilter_dn.cu, direction_pair) needs 37 and 12.

  __device__ __forceinline__ void direction_pair_proj(Frame const &t, PairEntry const &e, f32x2 &x, f32x2 &y, f32x2 &z)
  {
    x = fma2(e.lx, bcast2(t.T.x), fma2(e.ly, bcast2(t.B.x), bcast2(t.N.x)));
    y = fma2(e.lx, bcast2(t.T.y), fma2(e.ly, bcast2(t.B.y), bcast2(t.N.y)));
    z = fma2(e.lx, bcast2(t.T.z), fma2(e.ly, bcast2(t.B.z), bcast2(t.N.z)));
  }

  // The footprints of both samples of a pair: idx = raw index bits of the top-left records (what the gather's
  // record pointer has been moved back by), du/dv = fraction - 0.5.  Output references, not a returned struct:
  // a struct changes the rgbe pair kernel's register allocation (cuobjdump -sass).

  // frame rows face-local and folded; indices relative to the texel's face, kMagicBits on top
  __device__ __forceinline__ void pair_taps_same_face(LevelGeom const &g, Frame const &t, PairEntry const &e, uint32_t &idx_a, uint32_t &idx_b, f32x2 &du, f32x2 &dv)
  {
    f32x2 la, lb, lm;
    direction_pair_proj(t, e, la, lb, lm);

    float ma, mb;
    unpack2(lm, ma, mb);
    f32x2 r = pack2(rcp_fast(ma), rcp_fast(mb));

    f32x2 mu = fma2(la, r, bcast2(kMagic));
    f32x2 mv = fma2(lb, r, bcast2(kMagic));
    f32x2 niu = add2(neg2(mu), bcast2(kMagic));
    f32x2 niv = add2(neg2(mv), bcast2(kMagic));

    du = fma2(la, r, niu);
    dv = fma2(lb, r, niv);

    float ia, ib;
    unpack2(fma2(niv, bcast2(g.neg_ws), mu), ia, ib);
    idx_a = f2u(ia);
    idx_b = f2u(ib);
  }

  // frame rows in world coordinates: cube face selection of tools/ibl.cpp:43-88 per sample; indices carry the
  // face and g.bias_general
  __device__ __forceinline__ void pair_taps_general(LevelGeom const &g, Frame const &t, PairEntry const &e, uint32_t &idx_a, uint32_t &idx_b, f32x2 &du, f32x2 &dv)
  {
    f32x2 x, y, z;
    direction_pair_proj(t, e, x, y, z);

    float xa, xb, ya, yb, za, zb;
    unpack2(x, xa, xb);
    unpack2(y, ya, yb);
    unpack2(z, za, zb);

    float qua, qva, qub, qvb;
    uint32_t fa, fb;
    cube_select_unshrunk(xa, ya, za, qua, qva, fa);
    cube_select_unshrunk(xb, yb, zb, qub, qvb, fb);

    // the two-ulp shrink of the reciprocal (cube_select) rides in the scale
    f32x2 qu = pack2(qua, qub), qv = pack2(qva, qvb);
    f32x2 mu = fma2(qu, bcast2(g.hw_shrunk), bcast2(g.hwm_magic));
    f32x2 mv = fma2(qv, bcast2(g.hh_shrunk), bcast2(g.hhm_magic));
    f32x2 cu = add2(neg2(mu), bcast2(g.hwm_magic));
    f32x2 cv = add2(neg2(mv), bcast2(g.hhm_magic));

    du = fma2(qu, bcast2(g.hw_shrunk), cu);
    dv = fma2(qv, bcast2(g.hh_shrunk), cv);

    float ia, ib;
    unpack2(fma2(cv, bcast2(g.neg_ws), mu), ia, ib);
    idx_a = fa * g.face_size + f2u(ia);
    idx_b = fb * g.face_size + f2u(ib);
  }

  // ---- tiles ----------------------------------------------------------------------------
  //
  // Tiles of 8x4 texels are numbered in 4x4-blocked order over the slab.  With QUEUES the first
  // `queued` tiles are cut into one contiguous chunk per SM (queue index = %smid) and the rest form
  // a common pool that evens out the tail: a group takes tiles from its SM's chunk, then from the pool.
  //
  // %smid values are not guaranteed to be contiguous, and under MPS limits, green contexts or a
  // concurrent kernel an SM may host no CTA of this launch at all: once its own chunk and the pool are
  // empty (next_tile_plain returns -1) a group therefore looks through every other chunk before it
  // gives up, so every tile is computed whatever the placement of the CTAs.  The look is made by the 32
  // lanes of the group's first warp side by side (148 dependent L2 reads by one thread cost ~20 us per
  // call, measured as +5 % on a whole level; 5 rounds of 32 cost under 1 us), and only then: the common
  // hand-out stays one thread and one or two atomics.  Called by all lanes of warp 0; every lane gets the tile.
  // NOT inlined on purpose: with this code inside the kernel body ptxas schedules the sample loops ~1 % (512^2
  // level) to ~3 % (256^2 level) slower although it only ever runs at the very end of a launch (measured A/B).
  inline __device__ __noinline__ int steal_tile(int *counters, int queues, int chunk, uint32_t smid, int lane)
  {
    const int own = (int)(smid % (uint32_t)queues);

    for(int base = 1; base < queues; base += 32)
    {
      int i = base + lane;
      int q = own + i;
      if (q >= queues)
        q -= queues;

      // a drained chunk costs one read; only chunks that still hold tiles are bumped
      bool holds = i < queues && *(volatile int const *)(counters + q) < chunk;

      for(unsigned candidates = __ballot_sync(0xffffffffu, holds); candidates != 0u; candidates &= candidates - 1u)
      {
        int src = __ffs(candidates) - 1;
        int k = -1;
        if (lane == src)
          k = atomicAdd(counters + q, 1);
        k = __shfl_sync(0xffffffffu, k, src);

        if (k < chunk)
          return __shfl_sync(0xffffffffu, q, src) * chunk + k;
      }
    }

    return -1;
  }

  // the common hand-out, one thread: the SM's own chunk, then the pool; -1 when both are empty
  template<typename P>
  __device__ __forceinline__ int next_tile_plain(P const &p, uint32_t smid)
  {
    if ((int)smid < p.queues)
    {
      int k = atomicAdd(p.counters + smid, 1);
      if (k < p.chunk)
        return (int)smid * p.chunk + k;
    }

    int tile = p.queued + atomicAdd(p.counters + p.queues, 1);
    return tile < p.tiles ? tile : -1;
  }

  // tile number -> texel of this lane; false when the lane's texel is outside the slab
  template<typename P>
  __device__ __forceinline__ bool tile_texel(P const &p, int tile, int lane, int &x, int &row)
  {
    int block = tile >> 4, in = tile & 15;
    int bx = block % p.blocks_x, by = block / p.blocks_x;
    x = (bx * 4 + (in & 3)) * 8 + (lane & 7);
    row = p.row_begin + (by * 4 + (in >> 2)) * 4 + (lane >> 3);
    return x < p.wd && row < p.row_end;
  }

  // ---- per tile ---------------------------------------------------------------------------

  // The texel's folded frame from the per-level planes (launch_build_frames), and this warp's count of leading
  // same-face bands.  A warp reads ONE azimuth sector of every band: how far out its samples may lie before one
  // of them can leave some texel's face is sector_rho_limits, kept as the minimum over the texels of every 8x4
  // tile of the level (a slab that starts between two such tile rows looks at both).  With four warps the eight
  // 45-degree sectors pair up: one 90-degree sector per warp, or with VW == 2 (A/B) both 45-degree sectors one
  // after the other, each with its own count (n_same_second).  sector_rho increases with the band; the lanes
  // look at 32 bands at a time.
  template<int NW, int VW, typename P>
  __device__ __forceinline__ void tile_frame_bands(P const &p, int x, int row, int warp, int lane, int bands, Frame &st, int &n_same, int &n_same_second)
  {
    constexpr int SECTORS = NW * VW == 8 ? 1 : 0;

    float const *f = p.frames + ((size_t)row * p.wd + x);
    const size_t plane = (size_t)6 * p.hd * p.wd;
    st.T = Vec3f{ __ldg(f + 0 * plane), __ldg(f + 1 * plane), __ldg(f + 2 * plane) };
    st.B = Vec3f{ __ldg(f + 3 * plane), __ldg(f + 4 * plane), __ldg(f + 5 * plane) };
    st.N = Vec3f{ __ldg(f + 6 * plane), __ldg(f + 7 * plane), __ldg(f + 8 * plane) };

    float limit, limit_second = 0.0f;
    {
      const int tiles_x = (p.wd + 7) >> 3, tile_rows = (6 * p.hd + 3) >> 2;
      const int top = __shfl_sync(0xffffffffu, row, 0), left = __shfl_sync(0xffffffffu, x, 0);     // lane 0 is always inside the slab
      const int t0 = top >> 2, t1 = min((top + 3) >> 2, tile_rows - 1);
      float const *tile = p.frames + 9 * plane + (left >> 3);
      const size_t sector = (size_t)tile_rows * tiles_x;
      const int first = NW == 8 ? warp : 2 * warp;

      limit = fminf(__ldg(tile + first * sector + (size_t)t0 * tiles_x), __ldg(tile + first * sector + (size_t)t1 * tiles_x));
      if (NW != 8)
      {
        float second = fminf(__ldg(tile + (first + 1) * sector + (size_t)t0 * tiles_x), __ldg(tile + (first + 1) * sector + (size_t)t1 * tiles_x));
        if (VW == 2)
          limit_second = second;
        else
          limit = fminf(limit, second);
      }
    }

    #pragma unroll
    for(int pass = 0; pass < VW; ++pass)
    {
      float const *rho = p.sector_rho[SECTORS] + (VW * warp + pass) * bands;
      const float within_limit = pass == 0 ? limit : limit_second;
      int count = 0;
      for(int base = 0; base < bands; base += 32)
      {
        int k = base + lane;
        unsigned within = __ballot_sync(0xffffffffu, k < bands && __ldg(rho + k) <= within_limit);
        count += __popc(within);
        if (within != 0xffffffffu)
          break;
      }
      if (pass == 0)
        n_same = count;
      else
        n_same_second = count;
    }
  }

  // reduction over the CTA's warps: each warp's sums go to s_red[(warp*3 + c)*32 + lane], then (after a
  // __syncthreads) warp 0 adds them up
  __device__ __forceinline__ void store_warp_sums(Sums const &acc, float *s_red, int warp, int lane)
  {
    float a[4];
    unpack2(acc.rg, a[0], a[1]);
    unpack2(acc.bb, a[2], a[3]);
    a[2] += a[3];

    #pragma unroll
    for(int c = 0; c < 3; ++c)
      s_red[(warp * 3 + c) * 32 + lane] = a[c];
  }

  template<int NW>
  __device__ __forceinline__ void add_warp_sums(float const *s_red, int lane, float sum[3])
  {
    sum[0] = sum[1] = sum[2] = 0.0f;
    #pragma unroll
    for(int w = 0; w < NW; ++w)
    {
      #pragma unroll
      for(int c = 0; c < 3; ++c)
        sum[c] += s_red[(w * 3 + c) * 32 + lane];
    }
  }

  // ---- "this launch has stored everything" -----------------------------------------------------
  //
  // One probe shared by several GPUs: the kernels' epilogues store every texel into the peers' chains.
  // The CTA that finishes LAST (ticket counter) bumps an arrival counter in every peer's flag block
  // with a system-scope release; the peers' streams wait on their own counter (a stream memory
  // operation, no kernel) before the next level reads the texels.  Every thread fences its own
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
}
