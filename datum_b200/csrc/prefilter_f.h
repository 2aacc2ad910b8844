// datum_b200 — GGX prefilter of float cube chains (RGBA16F / RGBA32F): footprint records, per-tap
// arithmetic and launch interface (prefilter_f.cu; internal to libdatum_ibl_cuda).
//
// The record layout and the tap arithmetic are `__host__ __device__` so that tests/emu/prefilter_f_emu.cpp
// compiles the same expressions with g++.
#pragma once

#include "ibl_math.cuh"

#include <cstdint>

#if defined(__CUDACC__)
#include "prefilter.h"

#include <cuda_runtime.h>
#endif

namespace ibl
{
  // texel formats of a float chain (include/datum_ibl_cuda.h: DATUM_IBL_FORMAT_F32, DATUM_IBL_FORMAT_F16)
  constexpr int kFloatFormatF32 = 1;
  constexpr int kFloatFormatF16 = 2;

  IBL_HD int float_texel_bytes(int format) { return format == kFloatFormatF16 ? 8 : 16; }

  // IEEE binary16 -> fp32, exact (subnormals, infinities and NaN included)
  IBL_HD float half_to_float(uint32_t h)
  {
#if defined(__CUDA_ARCH__)
    float f;
    asm("{ .reg .b16 t; cvt.u16.u32 t, %1; cvt.f32.f16 %0, t; }" : "=f"(f) : "r"(h));
    return f;
#else
    uint32_t sign = (h & 0x8000u) << 16, exp = (h >> 10) & 0x1Fu, man = h & 0x3FFu;
    if (exp == 0x1Fu)
      return u2f(sign | 0x7F800000u | (man << 13));
    if (exp == 0)
    {
      float v = (float)man * 5.9604644775390625e-8f;    // man * 2^-24, exact
      return sign ? -v : v;
    }
    return u2f(sign | ((exp + 112u) << 23) | (man << 13));
#endif
  }

  // ---- footprint records ----------------------------------------------------------------
  //
  // Record (i, j) of a source level holds the 2x2 bilinear footprint whose top-left texel is (i, j),
  // neighbours clamped inside the face like build_dn_records_kernel's (the clamped ones are never
  // addressed).  Taps in the order (i, j), (i+1, j), (i, j+1), (i+1, j+1).
  //   F16: the four RGBA16F texels verbatim, 32 bytes: one 32-byte L1 sector per lane and footprint.
  //   F32: the four texels' rgb, 48 bytes (alpha dropped): three 16-byte loads, two sectors.
  struct alignas(32) F16Record
  {
    uint32_t w[8];            // texel k: w[2k] = g<<16 | r, w[2k+1] = a<<16 | b
  };

  struct alignas(16) F32Record
  {
    float c[12];              // texel k: c[3k .. 3k+2] = r, g, b
  };

  IBL_HD void f16_record_tap(F16Record const &r, int k, float &cr, float &cg, float &cb)
  {
    cr = half_to_float(r.w[2*k] & 0xFFFFu);
    cg = half_to_float(r.w[2*k] >> 16);
    cb = half_to_float(r.w[2*k + 1] & 0xFFFFu);
  }

  IBL_HD void f32_record_tap(F32Record const &r, int k, float &cr, float &cg, float &cb)
  {
    cr = r.c[3*k]; cg = r.c[3*k + 1]; cb = r.c[3*k + 2];
  }

  // one tap: acc[c] += w * texel[c], fp32 weight (kDnTableScale included), one rounding per channel
  IBL_HD void float_accumulate_tap(float cr, float cg, float cb, float w, float acc[3])
  {
    acc[0] = fmaf(cr, w, acc[0]);
    acc[1] = fmaf(cg, w, acc[1]);
    acc[2] = fmaf(cb, w, acc[2]);
  }

  // sums -> radiance: the weights carry kDnTableScale (2^64) on top of NdotL
  IBL_HD float float_chain_norm(double total_weight)
  {
    return (float)(1.0 / ((double)kDnTableScale * total_weight));
  }

  // Input range.  A weight is at most 2^63 (0.5 * NdotL * 2^64) and the weights of one texel sum to at
  // most samples * 2^64 (NdotL <= 1), so with level-0 radiance below kFloatChainMaxRadiance no product and
  // no partial sum leaves the fp32 range for samples <= 4096: 2^52 * 4096 * 2^64 = 2^128 is the bound.
  // Every binary16 value (<= 65504) is far inside it.
  constexpr double kFloatChainMaxRadiance = 4503599627370496.0;     // 2^52 = 4.5e15

  // fp32 result -> stored texel of a RGBA16F chain: min(x, 65504) rounded to nearest-even, alpha 1.0
  IBL_HD uint32_t float_to_half_rn(float x)
  {
    x = fminf(x, 65504.0f);
#if defined(__CUDA_ARCH__)
    unsigned short h;
    asm("cvt.rn.f16.f32 %0, %1;" : "=h"(h) : "f"(x));
    return h;
#else
    // x is finite, non-negative and at most 65504 here
    uint32_t u = f2u(x);
    if (u == 0u)
      return 0u;
    int e = (int)(u >> 23) - 127;
    if (e < -25)
      return 0u;
    uint32_t m = (u & 0x7FFFFFu) | 0x800000u;       // 24 significant bits
    int shift = e >= -14 ? 13 : 13 + (-14 - e);      // bits dropped: normal or subnormal half
    uint32_t q = m >> shift, rem = m & ((1u << shift) - 1u), half = 1u << (shift - 1);
    if (rem > half || (rem == half && (q & 1u)))
      ++q;
    if (e >= -14)
      return ((uint32_t)(e + 15) << 10) + (q - 0x400u);   // a carry out of the mantissa bumps the exponent
    return q;                                              // subnormal (q may round up to the smallest normal)
#endif
  }

#if defined(__CUDACC__)
  struct PrefilterFloatParams
  {
    int format;                 // kFloatFormatF32 / kFloatFormatF16
    void const *src;            // SOURCE level (6*ws*hs texels of the format): the tail kernel and the record pass
    void const *records;        // footprint records of the source level (F16Record / F32Record), pair kernel
    float4 const *table;        // banded sample table scaled by kDnTableScale (tail kernel, non-proj sources)
    float4 const *table_proj;   // the same as (lx/lz, ly/lz, lz, wh) (tail kernel, proj_usable sources)
    float4 const *table_sector[2];   // the pair kernel's sector tables for 4 and 8 warps per tile (PrefilterDnParams)
    float const *sector_rho[2];
    int sector_bands[2];
    int table_count;
    float const *frames;        // folded frames + sector limits of the destination level (launch_build_frames)
    float const *world_frames;  // world T, B, N of every destination texel, or null (tail kernel)
    void *dst;                  // destination level base, texels of the format
    float *dst_f32;             // destination level base, fp32 rgb triples before rounding (may be null)
    int wd, hd;                 // destination level size
    int row_begin, row_end;     // slab of the 6*hd face-major rows to compute
    LevelGeom geom;             // source level addressing constants
    Quatf quats[6];
    float norm;                 // float_chain_norm
    int *counters;              // queues+1 tile queue heads, zeroed by launch_build_float_records
    int blocks_x, tiles;        // filled by the launcher
    int queues, chunk, queued;

    // the same level of `probes` chains in one launch (datum_ibl_bake_probes_float); 0 or 1: one chain.
    // Strides in units of the format: src_stride and dst_stride in TEXELS between the probes' source and
    // destination levels, record_stride in RECORDS (F16Record / F32Record) between their record sets
    // (launch_build_float_records writes them back to back: 6*ws*hs).  dst_f32 must be null.
    int probes, tiles_per_probe, texels_per_probe;    // the last two filled by the launchers
    size_t src_stride, record_stride, dst_stride;

    // one probe shared by several GPUs (datum_ibl_prefilter_level_float_peers): the epilogue stores every texel
    // into dst and into the same destination level of each peer's chain; probes == 1 and dst_f32 null
    void *peer_dst[kMaxPeers];
    int peers;
    PeerSignal signal;        // whom to tell when the whole slab is stored
  };

  // records of the ws x hs source levels of `probes` chains (src_stride texels apart; records back to back);
  // also zeroes the `ncounters` tile queue heads
  cudaError_t launch_build_float_records(int format, void const *src, void *records, int ws, int hs, int probes, size_t src_stride, int *counters, int ncounters, int sm_count, cudaStream_t stream);

  // pair kernel (proj_usable sources, slabs above kTailTexels, levels at least 8 wide)
  cudaError_t launch_prefilter_float(PrefilterFloatParams const &p, int sm_count, cudaStream_t stream);

  // one CTA per destination texel, lanes are samples; any source size (a batch: proj_usable sources only).
  // Both launchers run their shared-probe instantiations when p.peers > 0 or p.signal.count > 0.
  cudaError_t launch_prefilter_float_tail(PrefilterFloatParams const &p, cudaStream_t stream);
#endif
}
