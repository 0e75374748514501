// binfileutils containers (snarkjs .r1cs / .ptau / .zkey): the section-table reader and the output writer shared by the
// setup entry points (setup.cu `zkey new`, ptau.cu `powersoftau prepare phase2`).
#pragma once
#include "api_util.cuh"

namespace nzcp {

static inline uint32_t rd32u(const uint8_t* p) { uint32_t v; memcpy(&v, p, 4); return v; }
static inline uint64_t rd64u(const uint8_t* p) { uint64_t v; memcpy(&v, p, 8); return v; }

struct Sect { const uint8_t* p = nullptr; uint64_t len = 0; };

// secs[id] = first section with that id, for id <= max_id; later duplicates are ignored.
static inline void parse_bin(const uint8_t* b, size_t len, const char* magic, Sect* secs, int max_id) {
  if (len < 12 || memcmp(b, magic, 4) != 0) throw ApiError(NZCP_E_FORMAT, std::string(magic) + " file: Invalid File format");
  if (rd32u(b + 4) > 1) throw ApiError(NZCP_E_FORMAT, "Version not supported");
  size_t pos = 12;
  for (uint32_t i = 0, n = rd32u(b + 8); i < n; i++) {
    if (pos + 12 > len) throw ApiError(NZCP_E_FORMAT, "truncated section table");
    const uint32_t id = rd32u(b + pos);
    const uint64_t sl = rd64u(b + pos + 4);
    pos += 12;
    if (sl > len - pos) throw ApiError(NZCP_E_FORMAT, "section exceeds file size");
    if (id <= (uint32_t)max_id && !secs[id].p) { secs[id].p = b + pos; secs[id].len = sl; }
    pos += sl;
  }
}

struct Writer {
  uint8_t* p;
  size_t cap, pos = 0;
  Writer(uint8_t* b, size_t c) : p(b), cap(c) {}
  void need(size_t n) { if (pos + n > cap) throw ApiError(NZCP_E_ARG, "output buffer too small"); }
  void u32(uint32_t v) { need(4); memcpy(p + pos, &v, 4); pos += 4; }
  void u64(uint64_t v) { need(8); memcpy(p + pos, &v, 8); pos += 8; }
  void raw(const void* s, size_t n) { need(n); memcpy(p + pos, s, n); pos += n; }
  void zeros(size_t n) { need(n); memset(p + pos, 0, n); pos += n; }
  uint8_t* reserve(size_t n) { need(n); uint8_t* q = p + pos; pos += n; return q; }
  void section(uint32_t id, uint64_t len) { u32(id); u64(len); }
};

}  // namespace nzcp
