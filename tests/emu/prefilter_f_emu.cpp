// TEST INFRASTRUCTURE — host build of the float-chain kernels' per-tap arithmetic.
//
// Compiles datum_b200/csrc/prefilter_f.h, ibl_math.cuh and ibl_tables.cpp with g++ and computes one
// level of a float chain the way prefilter_f.cu does: footprint records laid out like
// build_float_records_kernel's, the sample table scaled by kDnTableScale, cube-face selection and
// footprint of every sample (the tail kernel's general path: projective for proj_usable sources),
// fp32 weights times float taps, float_chain_norm, and the F16 store rounding.  Single-threaded and in
// table order, so the sums differ from the kernels' by summation order only.  tests/test_float_chain_cpu.py
// compares it with the float oracle.  It is NOT a fallback: nothing under datum_b200/ builds, links or
// loads it.

#include "../../datum_b200/csrc/prefilter_f.h"
#include "../../datum_b200/csrc/ibl_tables.h"

#include <cmath>
#include <cstring>
#include <vector>

using namespace ibl;

namespace
{
  // footprint records of a level exactly as build_float_records_kernel lays them out
  template<typename R>
  std::vector<R> build_records(int format, void const *src, int ws, int hs)
  {
    std::vector<R> records((size_t)6 * ws * hs);
    for(size_t idx = 0; idx < records.size(); ++idx)
    {
      int i = (int)(idx % ws), j = (int)((idx / ws) % hs);
      size_t right = (i + 1 < ws) ? 1 : 0, down = (j + 1 < hs) ? (size_t)ws : 0;
      const size_t tap[4] = { idx, idx + right, idx + down, idx + down + right };

      R r;
      std::memset(&r, 0, sizeof(r));
      for(int k = 0; k < 4; ++k)
      {
        if (format == kFloatFormatF16)
        {
          uint32_t const *s = static_cast<uint32_t const*>(src) + 2 * tap[k];
          reinterpret_cast<uint32_t*>(&r)[2*k] = s[0];
          reinterpret_cast<uint32_t*>(&r)[2*k + 1] = s[1];
        }
        else
        {
          float const *s = static_cast<float const*>(src) + 4 * tap[k];
          for(int c = 0; c < 3; ++c)
            reinterpret_cast<float*>(&r)[3*k + c] = s[c];
        }
      }
      records[idx] = r;
    }
    return records;
  }

  inline void record_tap(F16Record const &r, int k, float &cr, float &cg, float &cb) { f16_record_tap(r, k, cr, cg, cb); }
  inline void record_tap(F32Record const &r, int k, float &cr, float &cg, float &cb) { f32_record_tap(r, k, cr, cg, cb); }

  template<typename R>
  void level(int format, void const *src, int ws, int hs, int lvl, int levels, int samples, float *f32, uint16_t *f16)
  {
    LevelSamples table = build_level_samples(lvl, levels, samples);
    LevelGeom geom = make_level_geom(ws, hs);
    const bool proj = proj_usable(ws, hs);
    std::vector<R> records = build_records<R>(format, src, ws, hs);
    const float norm = float_chain_norm(table.total_weight);

    const float kPi = 3.14159265358979323846f;
    float angles[6] = { -kPi/2, kPi/2, -kPi/2, kPi/2, 0.0f, kPi };
    int axes[6] = { 1, 1, 0, 0, 1, 1 };
    Quatf quats[6];
    for(int f = 0; f < 6; ++f)
    {
      float c = std::cos(angles[f]/2), s = std::sin(angles[f]/2);
      quats[f] = Quatf{ c, axes[f] == 0 ? s : 0.0f, axes[f] == 1 ? s : 0.0f, 0.0f };
    }

    int wd = ws >> 1, hd = hs >> 1;

    for(int row = 0; row < 6 * hd; ++row)
    {
      int face = row / hd, y = row % hd;
      for(int x = 0; x < wd; ++x)
      {
        Vec3f N = texel_normal(quats[face], x, y, wd, hd);
        Vec3f T, B;
        tangent_frame(N, T, B);

        float acc[3] = { 0, 0, 0 };

        for(auto const &s : table.entries)
        {
          float du, dv, w[4];
          uint32_t idx;

          if (proj)
          {
            // the tail kernel's projective entry: (lx/lz, ly/lz, lz, wh), the last two scaled
            float ex = (float)((double)s.lx / (double)s.lz), ey = (float)((double)s.ly / (double)s.lz);
            float ez = s.lz * kDnTableScale, ew = s.wh * kDnTableScale;
            float Lx = fmaf(ex, T.x, fmaf(ey, B.x, N.x));
            float Ly = fmaf(ex, T.y, fmaf(ey, B.y, N.y));
            float Lz = fmaf(ex, T.z, fmaf(ey, B.z, N.z));
            uint32_t f;
            idx = cube_footprint_proj(geom, Lx, Ly, Lz, du, dv, f);
            idx += f * geom.face_size - geom.bias_general;
            footprint_weights_diff(du, dv, ew, ez, w);
          }
          else
          {
            float ex = s.lx * kDnTableScale, ey = s.ly * kDnTableScale, ez = s.lz * kDnTableScale, ew = s.wh * kDnTableScale;
            float Lx = fmaf(ez, N.x, fmaf(ey, B.x, ex * T.x));
            float Ly = fmaf(ez, N.y, fmaf(ey, B.y, ex * T.y));
            float Lz = fmaf(ez, N.z, fmaf(ey, B.z, ex * T.z));
            idx = cube_footprint(geom, Lx, Ly, Lz, du, dv);
            footprint_weights(du, dv, ew, ez, w);
          }

          R const &r = records[idx];
          for(int k = 0; k < 4; ++k)
          {
            float cr, cg, cb;
            record_tap(r, k, cr, cg, cb);
            float_accumulate_tap(cr, cg, cb, w[k], acc);
          }
        }

        size_t o = (size_t)row * wd + x;
        for(int c = 0; c < 3; ++c)
        {
          float v = acc[c] * norm;
          f32[3*o + c] = v;
          if (f16)
            f16[4*o + c] = (uint16_t)float_to_half_rn(v);
        }
        if (f16)
          f16[4*o + 3] = 0x3C00;
      }
    }
  }
}

// one level of a float chain from `src` (RGBA float32 for format 1, RGBA binary16 for format 2):
// fp32 rgb into `f32`, and for format 2 the stored RGBA16F texels into `f16` (may be null)
extern "C" void emu_prefilter_level_float(int format, void const *src, int ws, int hs, int level_index, int levels, int samples, float *f32, uint16_t *f16)
{
  if (format == kFloatFormatF16)
    level<F16Record>(format, src, ws, hs, level_index, levels, samples, f32, f16);
  else
    level<F32Record>(format, src, ws, hs, level_index, levels, samples, f32, nullptr);
}

extern "C" float emu_half_to_float(uint32_t h) { return half_to_float(h); }
extern "C" uint32_t emu_float_to_half(float x) { return float_to_half_rn(x); }
