// TEST INFRASTRUCTURE — CPU oracle for the float chains (RGBA32F / RGBA16F).
//
// One level of tools/ibl.cpp:247-278 computed from RGBA fp32 texels taken as they are, instead of from
// rgbe words.  The oracle of the rgbe chain (oracle/ibl_oracle.cpp) is compiled into this translation
// unit unchanged, so that the Hammersley/GGX samples, the texel directions, the face rotations, the
// lerp and fmod2 of the sampler and the thread pool are literally its code.  What is restated here is
// only what fetches a texel: the Sampler of ibl.cpp:16-93 over float texels, and convolve()
// (ibl.cpp:160-187) over that sampler, both written term for term like the rgbe oracle's.
// tests/test_float_chain_cpu.py pins the restatement: fed the decoded words of an rgbe level it gives
// bit for bit the fp32 values the rgbe oracle hands to rgbe().
//
// A RGBA16F level is the same computation on the halves widened to fp32 (exact); the caller rounds.
// Build: g++ -O2 -ffp-contract=off (tests/float_oracle_lib.py), like oracle/Makefile.

#include "../../oracle/ibl_oracle.cpp"

namespace
{
  // ibl.cpp:16-93 over RGBA fp32 texels (alpha ignored by the callers)
  struct FloatSampler
  {
    int width, height;
    float const *faces[6];    // 0 right, 1 left, 2 down, 3 up, 4 forward, 5 back (ibl.cpp:21-26)

    FloatSampler(int w, int h, float const *rgba) : width(w), height(h)
    {
      for(int f = 0; f < 6; ++f)
        faces[f] = rgba + (size_t)4 * f * w * h;
    }

    C4 texel(int face, int i, int j) const
    {
      float const *t = faces[face] + (size_t)4 * (j * width + i);
      return { t[0], t[1], t[2], 1.0f };
    }

    // ibl.cpp:34-41
    C4 sample(int face, float tx, float ty) const
    {
      float i, j;
      float u = std::modf(fmod2(tx, 1.0f) * (width - 1), &i);
      float v = std::modf(fmod2(ty, 1.0f) * (height - 1), &j);

      return lerp4(lerp4(texel(face, (int)i, (int)j), texel(face, (int)i+1, (int)j), u),
                   lerp4(texel(face, (int)i, (int)j+1), texel(face, (int)i+1, (int)j+1), u), v);
    }

    // ibl.cpp:43-88, ties resolved like the rgbe oracle
    C4 sample(V3 const &d) const
    {
      float mx = std::abs(d.x), my = std::abs(d.y), mz = std::abs(d.z);

      if (mx >= std::max(my, mz))
      {
        if (d.x > 0)
          return sample(0, 0.5f + 0.5f*d.z/mx, 0.5f + 0.5f*d.y/mx);
        else
          return sample(1, 0.5f - 0.5f*d.z/mx, 0.5f + 0.5f*d.y/mx);
      }
      else if (my >= mz)
      {
        if (d.y > 0)
          return sample(3, 0.5f + 0.5f*d.x/my, 0.5f + 0.5f*d.z/my);
        else
          return sample(2, 0.5f + 0.5f*d.x/my, 0.5f - 0.5f*d.z/my);
      }
      else
      {
        if (d.z > 0)
          return sample(5, 0.5f - 0.5f*d.x/mz, 0.5f + 0.5f*d.y/mz);
        else
          return sample(4, 0.5f + 0.5f*d.x/mz, 0.5f + 0.5f*d.y/mz);
      }
    }
  };

  // ibl.cpp:160-187 over the float sampler
  inline void convolve_float(float roughness, V3 const &ray, FloatSampler const &envmap, int samples, float out[3])
  {
    V3 N = ray;
    V3 V = ray;

    float sum[3] = { 0, 0, 0 };
    float totalweight = 0;

    for(int i = 0; i < samples; ++i)
    {
      float ux = float(i)/float(samples);
      float uy = radicalinverse_VdC(i);
      V3 H = importancesample_ggx(ux, uy, roughness * roughness, N);
      V3 L = sub3(scale3(2 * dot3(V, H), H), V);

      float NdotL = clampf(dot3(N, L), 0.0f, 1.0f);

      if (NdotL > 0)
      {
        C4 c = envmap.sample(L);

        sum[0] += c.r * NdotL;
        sum[1] += c.g * NdotL;
        sum[2] += c.b * NdotL;

        totalweight += NdotL;
      }
    }

    out[0] = sum[0] / totalweight;
    out[1] = sum[1] / totalweight;
    out[2] = sum[2] / totalweight;
  }
}

extern "C"
{
  // `src` is a (ws x hs x 6) RGBA fp32 level; the (ws/2 x hs/2 x 6) level's fp32 rgb goes to `f32`, rows
  // [row_begin, row_end) of the face-major destination rows, indexed from the start of the level
  void oracle_prefilter_level_rgba32f(float const *src, int ws, int hs, float roughness, int samples, int row_begin, int row_end, float *f32, int threads)
  {
    FloatSampler envmap(ws, hs, src);

    Xform rot[6];
    face_rotations(rot);

    int wd = ws >> 1, hd = hs >> 1;

    parallel_rows(row_begin, row_end, threads, [&](int row)
    {
      int face = row / hd;
      int y = row % hd;

      for(int x = 0; x < wd; ++x)
      {
        float rgb[3];
        convolve_float(roughness, texel_direction(rot[face], x, y, wd, hd), envmap, samples, rgb);

        size_t idx = (size_t)row * wd + x;
        f32[3*idx + 0] = rgb[0];
        f32[3*idx + 1] = rgb[1];
        f32[3*idx + 2] = rgb[2];
      }
    });
  }
}
