// binfileutils containers (snarkjs .r1cs / .ptau / .zkey): the section-table reader, the output writer and the point check
// shared by the setup entry points (setup.cu `zkey new`, ptau.cu `powersoftau prepare phase2`, contribute.cu `zkey
// contribute` / `zkey beacon`).
#pragma once
#include <algorithm>
#include <thread>

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

// Every point of a section of n affine points must be the (0,0) marker or have canonical coordinates and lie on the curve
// y^2 = x^3 + b.  Scanned by all host threads; throws NZCP_E_RANGE naming the first offending point ("<what>: section
// <sec> point <i> ...").
template <class F>
void check_points(const char* what, const uint8_t* p, uint64_t n, int sec, const F& b) {
  // first offending point of each thread's chunk; 1 = coordinate >= q, 2 = off the curve
  const unsigned nt = std::max(1u, std::min(64u, std::thread::hardware_concurrency()));
  const uint64_t chunk = (n + nt - 1) / nt;
  std::vector<uint64_t> first(nt, UINT64_MAX);
  std::vector<int> kind(nt, 0);
  auto scan = [&](unsigned t) {
    for (uint64_t i = t * chunk; i < std::min(n, (t + 1) * chunk); i++) {
      Affine<F> a;
      memcpy(&a, p + i * sizeof(Affine<F>), sizeof(Affine<F>));
      bool inf;
      if (a.is_inf()) continue;
      const int k = !(CoordCanon<F>::ok(a.x) && CoordCanon<F>::ok(a.y)) ? 1 : !point_ok(a, b, &inf) ? 2 : 0;
      if (k) { first[t] = i; kind[t] = k; return; }
    }
  };
  if (n < 4096) {
    for (unsigned t = 0; t < nt; t++) scan(t);
  } else {
    std::vector<std::thread> th;
    for (unsigned t = 0; t < nt; t++) th.emplace_back(scan, t);
    for (auto& t : th) t.join();
  }
  for (unsigned t = 0; t < nt; t++)
    if (kind[t])
      throw ApiError(NZCP_E_RANGE, std::string(what) + ": section " + std::to_string(sec) + " point " + std::to_string(first[t]) +
                                       (kind[t] == 1 ? " has a coordinate >= q" : " is not on the curve"));
}

}  // namespace nzcp
