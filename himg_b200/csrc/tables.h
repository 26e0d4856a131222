// Host-side codec tables for the B200 HIMG path (product code).
//
// Everything here is a few hundred bytes of integer work per (quality, colour-space) pair, so it
// stays on the host exactly as in the reference; the results travel to the device as kernel
// parameters / small LUT uploads and in-band in the .himg container (LMAP/QCFG/FMAP chunks).
//
// Reference behaviour restated: quantize.cpp:72-125 (shift tables), mapper.cpp:75-97,193-223
// (mapping tables), mapper.cpp:105-157 (mapping-function serialisation), mapper.cpp:159-182
// (MapTo8Bit, including its top/tie quirks), encoder.cpp:111-184,222-256 (container headers).
#ifndef HIMG_B200_TABLES_H_
#define HIMG_B200_TABLES_H_

#include <cstdint>
#include <vector>

namespace himgcu {

constexpr int kNumSymbols = 261;
constexpr int kFullMapLutSize = 7616;  // magnitudes >= 7608 all map to 127 (mapper.cpp:170-181)

struct EncodeTables {
  uint8_t shift_luma[64];
  uint8_t shift_chroma[64];
  uint16_t low_table[128];    // LowResMapper magnitudes for this quality
  uint16_t full_table[128];   // FullResMapper magnitudes (quality independent)
  uint8_t low_map_lut[256];   // |delta| (0..255) -> magnitude code 0..127
  bool ycbcr;
  int quality;
};

void BuildEncodeTables(int quality, bool ycbcr, EncodeTables *t);

// |x| -> code magnitude for an arbitrary monotone table (mapper.cpp:159-182).
int MapMagnitude(const uint16_t table[128], int a);

// The 7616-entry full-res LUT (|x| -> code magnitude).
const uint8_t *FullMapLut();

// Mapping-function bytes (mapper.cpp:105-125).
std::vector<uint8_t> SerializeMapFun(const uint16_t table[128]);

// Parse mapping-function bytes into unmap[code byte] (mapper.cpp:127-157). false = reject.
bool ParseMapFun(const uint8_t *in, int size, int16_t unmap[256]);

// Everything of the container that precedes the LRES payload and everything between the LRES
// and FRES payloads, for one (shape, quality, colour-space): SURVEY A.1.
struct ContainerTemplate {
  std::vector<uint8_t> head;  // "RIFF" size "HIMG" FRMT LMAP "LRES" size   (sizes patched on device)
  std::vector<uint8_t> mid;   // QCFG FMAP "FRES" size
  // offset in `head` of the FRMT width and height (u32 each): "RIFF" size "HIMG", "FRMT" size, version byte
  static constexpr int kDimsAt = 12 + 8 + 1;
};
void BuildContainerTemplate(const EncodeTables &t, int width, int height, int nch,
                            ContainerTemplate *out);

}  // namespace himgcu

#endif  // HIMG_B200_TABLES_H_
