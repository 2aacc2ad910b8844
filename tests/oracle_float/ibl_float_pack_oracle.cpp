// TEST INFRASTRUCTURE — CPU oracle of level 0 of a float chain (RGBA32F / RGBA16F) from an equirect HDR image or
// six ARGB32 images.
//
// The rgbe oracle's oracle_image_pack_cube (equirect resample + edge blend, tools/hdr.cpp:331-359, 173-318) and
// oracle_ingest_cube_argb32 (tools/assetbuilder.cpp:443-462) restated as templates over a texel policy that stores
// rgb and reads it back: rgbe words, RGBA32F, RGBA16F (round to nearest-even, clamp at 65504, alpha 1.0).  The rgbe
// oracle (oracle/ibl_oracle.cpp) is compiled into this translation unit unchanged, so Image::sample_dir,
// face_rotations, texel_direction and oracle_srgba_decode are literally its code.  The rgbe instantiation exists
// to pin the restatement: its words equal the rgbe oracle's bit for bit (tests/test_float_pack_cpu.py).
// Build: g++ -O2 -ffp-contract=off (tests/float_pack_oracle_lib.py), like oracle/Makefile.

#include "../../oracle/ibl_oracle.cpp"

namespace
{
  // ---- level 0 of a float chain: equirect image or six ARGB32 images --------------------------------------

  // fp32 -> IEEE binary16 bits, min(x, 65504) rounded to nearest-even; x finite and non-negative.  Written
  // independently of the library's float_to_half_rn: a scaled nearbyint in double (exact: at most 24 bits).
  inline uint16_t half_rn(float x)
  {
    x = std::min(x, 65504.0f);
    if (x == 0.0f)
      return 0;
    if (x < 6.103515625e-05f)                                  // below 2^-14: subnormal units of 2^-24
      return (uint16_t)std::nearbyint((double)x * 16777216.0);  // 1024 is the smallest normal's encoding
    int e;
    std::frexp(x, &e);                                          // x = m * 2^e, m in [0.5, 1)
    int q = (int)std::nearbyint(std::ldexp((double)x, 11 - e));    // 1024..2048 units of 2^(e-11)
    return (uint16_t)(((e + 14) << 10) + (q - 1024));          // q == 2048 carries into the exponent
  }

  inline float half_widen(uint16_t h)
  {
    int exp = (h >> 10) & 0x1F, man = h & 0x3FF;
    return exp == 0 ? std::ldexp((float)man, -24) : std::ldexp((float)(man | 0x400), exp - 25);
  }

  struct RgbeStore
  {
    typedef uint32_t Word;
    static Word encode(float r, float g, float b) { return rgbe_encode(r, g, b); }
    static C4 decode(Word w) { return rgbe_decode(w); }
  };

  struct F32Store
  {
    struct Word { float c[4]; };
    static Word encode(float r, float g, float b) { return { { r, g, b, 1.0f } }; }
    static C4 decode(Word w) { return { w.c[0], w.c[1], w.c[2], w.c[3] }; }
  };

  struct F16Store
  {
    struct Word { uint16_t c[4]; };
    static Word encode(float r, float g, float b) { return { { half_rn(r), half_rn(g), half_rn(b), 0x3C00 } }; }
    static C4 decode(Word w) { return { half_widen(w.c[0]), half_widen(w.c[1]), half_widen(w.c[2]), half_widen(w.c[3]) }; }
  };

  // the rgbe oracle's blend3 with the codec swapped for the store
  template<typename S>
  typename S::Word blend3_as(typename S::Word a, typename S::Word b, typename S::Word c)
  {
    C4 ca = S::decode(a), cb = S::decode(b), cc = S::decode(c);
    return S::encode(0.3f * ca.r + 0.4f * cb.r + 0.3f * cc.r, 0.3f * ca.g + 0.4f * cb.g + 0.3f * cc.g, 0.3f * ca.b + 0.4f * cb.b + 0.3f * cc.b);
  }

  // oracle_image_blend_edges on one level of texels of the store, the same twelve loops in the same order
  template<typename S>
  void blend_edges_as(int w, int h, typename S::Word *img)
  {
    typedef typename S::Word Word;
    if (w <= 1 || h <= 1)
      return;

    auto tex = [=](int x, int y, int z) -> Word& { return img[(size_t)z*w*h + (size_t)y*w + x]; };

    auto run = [&](int count, auto coords)
    {
      for(int k = 0; k < count; ++k)
      {
        int c[4][3];
        coords(k, c);
        Word a = tex(c[0][0], c[0][1], c[0][2]), b = tex(c[1][0], c[1][1], c[1][2]);
        Word cc = tex(c[2][0], c[2][1], c[2][2]), d = tex(c[3][0], c[3][1], c[3][2]);
        tex(c[1][0], c[1][1], c[1][2]) = blend3_as<S>(a, b, cc);
        tex(c[2][0], c[2][1], c[2][2]) = blend3_as<S>(b, cc, d);
      }
    };

    int ring[4][2] = { { 4, 0 }, { 0, 5 }, { 5, 1 }, { 1, 4 } };
    for(auto &seam : ring)
    {
      int fa = seam[0], fb = seam[1];
      run(h, [=](int k, int c[4][3]) {
        int v[4][3] = { { w - 2, k, fa }, { w - 1, k, fa }, { 0, k, fb }, { 1, k, fb } };
        memcpy(c, v, sizeof(v));
      });
    }

    run(w, [=](int k, int c[4][3]) { int v[4][3] = { { k, h - 2, 4 }, { k, h - 1, 4 }, { k, 0, 3 }, { k, 1, 3 } }; memcpy(c, v, sizeof(v)); });
    run(w, [=](int k, int c[4][3]) { int v[4][3] = { { k, h - 2, 3 }, { k, h - 1, 3 }, { w - 1 - k, h - 1, 5 }, { w - 1 - k, h - 2, 5 } }; memcpy(c, v, sizeof(v)); });
    run(w, [=](int k, int c[4][3]) { int v[4][3] = { { k, 1, 5 }, { k, 0, 5 }, { w - 1 - k, 0, 2 }, { w - 1 - k, 1, 2 } }; memcpy(c, v, sizeof(v)); });
    run(w, [=](int k, int c[4][3]) { int v[4][3] = { { k, h - 2, 2 }, { k, h - 1, 2 }, { k, 0, 4 }, { k, 1, 4 } }; memcpy(c, v, sizeof(v)); });

    int m = std::min(w, h);
    run(m, [=](int k, int c[4][3]) { int v[4][3] = { { k, h - 2, 0 }, { k, h - 1, 0 }, { w - 1, k, 3 }, { w - 2, k, 3 } }; memcpy(c, v, sizeof(v)); });
    run(m, [=](int k, int c[4][3]) { int v[4][3] = { { 1, k, 3 }, { 0, k, 3 }, { w - 1 - k, h - 1, 1 }, { w - 1 - k, h - 2, 1 } }; memcpy(c, v, sizeof(v)); });
    run(m, [=](int k, int c[4][3]) { int v[4][3] = { { k, 1, 1 }, { k, 0, 1 }, { 0, k, 2 }, { 1, k, 2 } }; memcpy(c, v, sizeof(v)); });
    run(m, [=](int k, int c[4][3]) { int v[4][3] = { { w - 2, k, 2 }, { w - 1, k, 2 }, { w - 1 - k, 0, 0 }, { w - 1 - k, 1, 0 } }; memcpy(c, v, sizeof(v)); });
  }

  // oracle_image_pack_cube with levels == 1 (the IBL path) into texels of the store
  template<typename S>
  void pack_cube_as(int imgw, int imgh, float const *pixels, int width, int height, void *out)
  {
    typename S::Word *level0 = static_cast<typename S::Word*>(out);
    Image image = { imgw, imgh, reinterpret_cast<C4 const *>(pixels) };

    Xform rot[6];
    face_rotations(rot);

    float ax = 1.0f / std::min(4 * width, imgw);
    float ay = 1.0f / std::min(2 * height, imgh);

    parallel_rows(0, 6 * height, 0, [&](int row)
    {
      int face = row / height;
      int y = row % height;

      for(int x = 0; x < width; ++x)
      {
        C4 c = image.sample_dir(texel_direction(rot[face], x, y, width, height), ax, ay);

        level0[(size_t)row * width + x] = S::encode(c.r, c.g, c.b);
      }
    });

    blend_edges_as<S>(width, height, level0);
  }

  // oracle_ingest_cube_argb32 into texels of the store
  template<typename S>
  void ingest_as(uint32_t const *argb, int width, int height, void *out)
  {
    typename S::Word *level0 = static_cast<typename S::Word*>(out);
    size_t face_size = (size_t)width * height;

    for(int face = 0; face < 6; ++face)
    {
      for(int y = 0; y < height; ++y)
      {
        for(int x = 0; x < width; ++x)
        {
          float rgba[4];
          oracle_srgba_decode(argb[face * face_size + (size_t)y * width + x], rgba);

          level0[face * face_size + (size_t)(height - 1 - y) * width + x] = S::encode(rgba[0], rgba[1], rgba[2]);
        }
      }
    }
  }
}

extern "C"
{
  // `format`: 0 rgbe words, 1 RGBA32F, 2 RGBA16F (include/datum_ibl_cuda.h); returns non-zero for others
  int oracle_float_pack_cube(int format, int imgw, int imgh, float const *pixels, int width, int height, void *level0)
  {
    switch(format)
    {
      case 0: pack_cube_as<RgbeStore>(imgw, imgh, pixels, width, height, level0); return 0;
      case 1: pack_cube_as<F32Store>(imgw, imgh, pixels, width, height, level0); return 0;
      case 2: pack_cube_as<F16Store>(imgw, imgh, pixels, width, height, level0); return 0;
    }
    return 1;
  }

  int oracle_float_ingest_cube_argb32(int format, uint32_t const *argb, int width, int height, void *level0)
  {
    switch(format)
    {
      case 0: ingest_as<RgbeStore>(argb, width, height, level0); return 0;
      case 1: ingest_as<F32Store>(argb, width, height, level0); return 0;
      case 2: ingest_as<F16Store>(argb, width, height, level0); return 0;
    }
    return 1;
  }

  void oracle_half_rn_array(float const *x, size_t count, uint16_t *out)
  {
    for(size_t i = 0; i < count; ++i)
      out[i] = half_rn(x[i]);
  }
}
