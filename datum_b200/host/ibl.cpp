// datum_b200 host shim — drop-in replacement for the reference's tools/ibl.cpp.
//
// Keeps the four signatures of tools/ibl.h:9-15 and forwards plain pointers and
// sizes to libdatum_ibl_cuda (include/datum_ibl_cuda.h).  The reference functions
// return void and cannot fail; here a failing CUDA call becomes
// std::runtime_error, which assetbuilder's main() already catches and reports
// (tools/assetbuilder.cpp:968-982).  There is no CPU fallback.

// In the reference tree: copy this file over tools/ibl.cpp and define
// DATUM_IBL_IN_REFERENCE_TREE; "ibl.h" then resolves to the reference's own header
// (tools/ibl.h -> tools/hdr.h -> datum/math.h) and tools/hdr.cpp keeps providing
// load_hdr / image_pack_cube.  Stand-alone (this repository): "ibl.h" is
// datum_b200/host/ibl.h with the same declarations.

#include "ibl.h"

#include "datum_ibl_cuda.h"

#ifdef DATUM_IBL_IN_REFERENCE_TREE
void image_project_sh9_cube(int width, int height, void const *level0_rgbe, float *sh);
void image_pack_cube_faces_ibl(unsigned int const *argb, int width, int height, int levels, void *bits);
void image_pack_cube_float_ibl(HDRImage const &image, int width, int height, int levels, int format, void *chain);
void image_set_ibl_samples(int samples);
void image_buildmips_cube_ibl_batch(int count, int width, int height, int levels, void *const *bits, float *sh);
void image_pack_irradiance_sh9(int width, int height, void const *level0_rgbe, void *bits);
void image_pack_irradiance_cube(void const *sh9_bits, int width, int height, void *bits);
#endif

#include <cstdint>
#include <cstdlib>
#include <mutex>
#include <stdexcept>
#include <string>
#include <vector>

namespace
{
  int g_samples = 1024; // tools/ibl.cpp:162

  // One lazily created device set per process, like the reference's stateless free functions: callers
  // never see it.  DATUM_IBL_DEVICES="0,1,2,3" lists the GPUs this process may use (default: the one
  // device DATUM_IBL_DEVICE names, else device 0).  With several devices a batch is spread probe by probe,
  // and ONE probe of at least DATUM_IBL_SPLIT_MIN_FACE texels per face (default 1024 x 1024) is shared by
  // all of them, rows of every level split (datum_ibl_multi_*); smaller probes run on the first device.
  struct Devices
  {
    datum_ibl_multi *multi = nullptr;
    datum_ibl_ctx *first = nullptr;
    int count = 0;
    long long split_min_face = 1024LL * 1024LL;
  };

  Devices &devices()
  {
    static Devices set;
    static std::once_flag once;
    static std::string error;

    std::call_once(once, [] {
      std::vector<int> list;
      if (const char *env = std::getenv("DATUM_IBL_DEVICES"))
      {
        for(const char *p = env; *p; )
        {
          char *end = nullptr;
          long v = std::strtol(p, &end, 10);
          if (end == p)
            break;
          list.push_back((int)v);
          p = (*end == ',') ? end + 1 : end;
        }
      }
      if (list.empty())
      {
        const char *env = std::getenv("DATUM_IBL_DEVICE");
        list.push_back(env ? std::atoi(env) : 0);
      }
      if (const char *env = std::getenv("DATUM_IBL_SPLIT_MIN_FACE"))
        set.split_min_face = std::atoll(env);

      if (datum_ibl_multi_create((int)list.size(), list.data(), &set.multi))
        error = datum_ibl_last_error();
      else
      {
        set.first = datum_ibl_multi_context(set.multi, 0);
        set.count = (int)list.size();
      }
    });

    if (!set.multi)
      throw std::runtime_error("datum ibl: " + error);

    return set;
  }

  datum_ibl_ctx *context() { return devices().first; }

  void check(int status)
  {
    if (status)
      throw std::runtime_error(std::string("datum ibl: ") + datum_ibl_last_error());
  }
}

///////////////////////// image_buildmips_cube_ibl //////////////////////////
void image_buildmips_cube_ibl(int width, int height, int levels, void *bits)
{
  Devices &set = devices();

  if (set.count > 1 && (long long)width * height >= set.split_min_face)
    check(datum_ibl_multi_buildmips_cube_ibl(set.multi, width, height, levels, g_samples, bits));
  else
    check(datum_ibl_buildmips_cube_ibl(set.first, width, height, levels, g_samples, bits));
}

///////////////////////// image_pack_cube_ibl ///////////////////////////////
void image_pack_cube_ibl(HDRImage const &image, int width, int height, int levels, void *bits)
{
  static_assert(sizeof(lml::Color4) == 4 * sizeof(float), "HDRImage::bits must be packed RGBA fp32");

  check(datum_ibl_pack_cube_ibl(context(), image.width, image.height, &image.bits[0].r, width, height, levels, g_samples, bits));
}

///////////////////////// image_pack_envbrdf ////////////////////////////////
void image_pack_envbrdf(int width, int height, void *bits)
{
  check(datum_ibl_pack_envbrdf(context(), width, height, 1024, bits)); // tools/ibl.cpp:191
}

///////////////////////// image_pack_watercolor /////////////////////////////
void image_pack_watercolor(lml::Color3 const &deepcolor, lml::Color3 const &shallowcolor, float depthscale, lml::Color3 const &fresnelcolor, float fresnelbias, float fresnelpower, int width, int height, void *bits)
{
  float deep[3] = { deepcolor.r, deepcolor.g, deepcolor.b };
  float shallow[3] = { shallowcolor.r, shallowcolor.g, shallowcolor.b };
  float fresnel[3] = { fresnelcolor.r, fresnelcolor.g, fresnelcolor.b };

  check(datum_ibl_pack_watercolor(context(), deep, shallow, depthscale, fresnel, fresnelbias, fresnelpower, width, height, bits));
}

///////////////////////// extensions ////////////////////////////////////////
void image_project_sh9_cube(int width, int height, void const *level0_rgbe, float *sh)
{
  Devices &set = devices();

  if (set.count > 1 && (long long)width * height >= set.split_min_face)
    check(datum_ibl_multi_project_sh9(set.multi, level0_rgbe, DATUM_IBL_FORMAT_RGBE, width, height, sh));
  else
    check(datum_ibl_project_sh9(set.first, level0_rgbe, DATUM_IBL_FORMAT_RGBE, width, height, sh));
}

void image_pack_cube_faces_ibl(unsigned int const *argb, int width, int height, int levels, void *bits)
{
  check(datum_ibl_ingest_cube_argb32_ibl(context(), width, height, levels, g_samples, argb, bits));
}

void image_pack_cube_float_ibl(HDRImage const &image, int width, int height, int levels, int format, void *chain)
{
  check(datum_ibl_pack_cube_float_ibl(context(), format, image.width, image.height, &image.bits[0].r, width, height, levels, g_samples, chain));
}

void image_buildmips_cube_ibl_batch(int count, int width, int height, int levels, void *const *bits, float *sh)
{
  check(datum_ibl_multi_bake_probes(devices().multi, count, width, height, levels, g_samples, bits, sh));
}

void image_pack_irradiance_sh9(int width, int height, void const *level0_rgbe, void *bits)
{
  // payload of a 3 x 9 x 1 f32 image == float L[9][3]
  check(datum_ibl_project_sh9(context(), level0_rgbe, DATUM_IBL_FORMAT_RGBE, width, height, static_cast<float*>(bits)));
}

void image_pack_irradiance_cube(void const *sh9_bits, int width, int height, void *bits)
{
  check(datum_ibl_sh9_irradiance_cube(context(), static_cast<float const*>(sh9_bits), width, height, static_cast<uint32_t*>(bits), nullptr));
}

void image_set_ibl_samples(int samples)
{
  if (samples < 1)
    throw std::runtime_error("datum ibl: samples must be positive");

  g_samples = samples;
}

///////////////////////// image_pack_cube ///////////////////////////////////
// declared in hdr.h; lives here so that the shim has a single context.  Inside the
// reference tree tools/hdr.cpp keeps its own (CPU) definition for other callers.
#ifndef DATUM_IBL_IN_REFERENCE_TREE
void image_pack_cube(HDRImage const &image, int width, int height, int levels, void *bits)
{
  if (levels != 1)
    throw std::runtime_error("datum ibl: image_pack_cube is offered for levels == 1 only (the IBL path, tools/ibl.cpp:285)");

  check(datum_ibl_pack_cube(context(), image.width, image.height, &image.bits[0].r, width, height, bits));
}
#endif
