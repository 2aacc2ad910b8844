// TEST INFRASTRUCTURE — the .hdr flow of write_skybox_asset (tools/assetbuilder.cpp:473-491) producing a float
// probe through the C++ host shim (datum_b200/host/ibl.h): load_hdr, then image_pack_cube_float_ibl.
//
//   float_pack_driver hdr_float FILE.hdr W H LEVELS FORMAT out.bin    FORMAT 1 = RGBA32F, 2 = RGBA16F

#include "ibl.h"

#include <cstdint>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <stdexcept>
#include <string>
#include <vector>

static size_t chain_texels(int w, int h, int levels) // the levels of tools/assetpacker.cpp:488-497, 6 faces
{
  size_t texels = 0;
  for(int i = 0; i < levels; ++i)
    texels += (size_t)(w >> i) * (h >> i) * 6;
  return texels;
}

int main(int argc, char **argv)
{
  try
  {
    if (argc == 8 && std::string(argv[1]) == "hdr_float")
    {
      int w = atoi(argv[3]), h = atoi(argv[4]), levels = atoi(argv[5]), format = atoi(argv[6]);
      HDRImage image = load_hdr(argv[2]);
      std::vector<char> chain(chain_texels(w, h, levels) * (format == 2 ? 8 : 16));
      image_pack_cube_float_ibl(image, w, h, levels, format, chain.data());
      std::ofstream(argv[7], std::ios::binary).write(chain.data(), (std::streamsize)chain.size());
      return 0;
    }

    std::cerr << "usage: float_pack_driver hdr_float FILE.hdr W H LEVELS FORMAT out.bin" << std::endl;
    return 2;
  }
  catch(std::exception &e)
  {
    std::cout << "Critical Error: " << e.what() << std::endl; // tools/assetbuilder.cpp:978
    return 1;
  }
}
