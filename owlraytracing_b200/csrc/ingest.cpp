// ingest.cpp — fast point-file ingest and neighbour writer (SURVEY.md §8f rank 2), host only.
//
// The reference reads its input with a serial getline + stringstream + push_back loop
// (samples/s01-trueknn/hostCode.cpp:83-104) and never writes neighbours (the dump at :312-319 is
// commented out).  Here the file is mmap-ed, cut into line-aligned chunks parsed in parallel with
// std::from_chars, and stitched under the SAME grammar: lines are consumed while n*dim floats are
// still owed (the last line read is consumed whole), floats are separated by ',' and/or blanks, a
// token that is not a float ends its line, and the flat float list is chunked by dim (dim 2 => z = 0).
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <charconv>
#include <cstdio>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../../include/trueknn.h"

namespace {

struct Chunk {
  std::vector<float> vals;
  std::vector<uint32_t> per_line;  // floats on each line of the chunk
};

inline bool is_blank(char c) { return c == ' ' || c == '\t' || c == '\r' || c == '\v' || c == '\f'; }

void parse_chunk(const char* p, const char* end, Chunk& out) {
  while (p < end) {
    const char* eol = static_cast<const char*>(memchr(p, '\n', (size_t)(end - p)));
    if (!eol) eol = end;
    uint32_t cnt = 0;
    const char* s = p;
    while (s < eol) {
      while (s < eol && is_blank(*s)) ++s;
      if (s >= eol) break;
      const char* t = s;
      if (*t == '+') ++t;  // operator>> accepts a leading '+', from_chars does not
      float v;
      auto r = std::from_chars(t, eol, v);
      if (r.ec != std::errc() || r.ptr == t) break;  // not a float: the rest of the line is dropped
      out.vals.push_back(v);
      ++cnt;
      s = r.ptr;
      if (s < eol && *s == ',') ++s;
    }
    out.per_line.push_back(cnt);
    p = eol + 1;
  }
}

}  // namespace

extern "C" {

// Reads up to n points of `dim` (2|3) coordinates from a text file (or raw little-endian float32 rows
// when the name ends in ".f32") into xyz_out (n_cap rows of 3 floats).  *n_out = points read.  The last line read
// is consumed whole (hostCode.cpp:92), so a file with several points per line can yield more than n rows: when they
// do not fit, the call returns TKNN_EINVAL with *n_out = the rows it needs (0 for every other failure).
TKNN_API int tknn_read_points(const char* path, uint64_t n, int dim, float* xyz_out, uint64_t n_cap, uint64_t* n_out) {
  if (!path || !xyz_out || !n_out || (dim != 2 && dim != 3)) return TKNN_EINVAL;
  *n_out = 0;
  const int fd = open(path, O_RDONLY);
  if (fd < 0) return TKNN_EINVAL;
  struct stat st;
  if (fstat(fd, &st) != 0) { close(fd); return TKNN_EINVAL; }
  const size_t size = (size_t)st.st_size;
  if (size == 0) { close(fd); return TKNN_OK; }
  const char* data = static_cast<const char*>(mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0));
  close(fd);
  if (data == MAP_FAILED) return TKNN_ENOMEM;
  int rc = TKNN_OK;
  const size_t plen = strlen(path);
  if (plen > 4 && strcmp(path + plen - 4, ".f32") == 0) {
    const uint64_t rows = std::min<uint64_t>(n, size / (sizeof(float) * (size_t)dim));
    if (rows > n_cap) { *n_out = rows; rc = TKNN_EINVAL; }
    else {
      const float* f = reinterpret_cast<const float*>(data);
      for (uint64_t i = 0; i < rows; ++i) {
        xyz_out[3 * i] = f[dim * i];
        xyz_out[3 * i + 1] = f[dim * i + 1];
        xyz_out[3 * i + 2] = dim == 3 ? f[dim * i + 2] : 0.0f;
      }
      *n_out = rows;
    }
    munmap(const_cast<char*>(data), size);
    return rc;
  }
  unsigned nt = std::max(1u, std::thread::hardware_concurrency());
  nt = (unsigned)std::min<size_t>(nt, std::max<size_t>(1, size / (1 << 20)));
  std::vector<size_t> cut(nt + 1, size);
  cut[0] = 0;
  for (unsigned t = 1; t < nt; ++t) {  // chunk borders snap forward to the next line start
    size_t pos = size * t / nt;
    const char* nl = static_cast<const char*>(memchr(data + pos, '\n', size - pos));
    cut[t] = nl ? (size_t)(nl - data) + 1 : size;
  }
  std::vector<Chunk> chunks(nt);
  std::vector<std::thread> th;
  for (unsigned t = 0; t < nt; ++t)
    th.emplace_back([&, t]() { if (cut[t] < cut[t + 1]) parse_chunk(data + cut[t], data + cut[t + 1], chunks[t]); });
  for (auto& x : th) x.join();
  munmap(const_cast<char*>(data), size);
  // stitch: consume whole lines while floats are still owed (hostCode.cpp:92: `while (getline && count > 0)`)
  const uint64_t want = n * (uint64_t)dim;
  std::vector<float> flat;
  flat.reserve((size_t)std::min<uint64_t>(want + 16, (uint64_t)1 << 33));
  uint64_t have = 0;
  for (unsigned t = 0; t < nt && have < want; ++t) {
    size_t off = 0;
    for (uint32_t c : chunks[t].per_line) {
      if (have >= want) break;
      flat.insert(flat.end(), chunks[t].vals.begin() + (long)off, chunks[t].vals.begin() + (long)(off + c));
      off += c;
      have += c;
    }
  }
  if (flat.size() % (size_t)dim) return TKNN_EINVAL;  // the reference throws std::out_of_range here
  const uint64_t rows = flat.size() / (size_t)dim;
  if (rows > n_cap) { *n_out = rows; return TKNN_EINVAL; }  // *n_out names the capacity a retry needs
  for (uint64_t i = 0; i < rows; ++i) {
    xyz_out[3 * i] = flat[dim * i];
    xyz_out[3 * i + 1] = flat[dim * i + 1];
    xyz_out[3 * i + 2] = dim == 3 ? flat[dim * i + 2] : 0.0f;
  }
  *n_out = rows;
  return TKNN_OK;
}

// Writes `query,neighbourIndex,distance` lines (the format commented out at hostCode.cpp:316), or raw
// int32 / float32 arrays when binary != 0 (path + ".idx.i32" / ".dist.f32").
TKNN_API int tknn_write_neighbours(const char* path, const int32_t* idx, const float* dist, uint64_t n, int k, int binary) {
  if (!path || !idx || !dist || k < 1) return TKNN_EINVAL;
  if (binary) {
    const std::string pi = std::string(path) + ".idx.i32", pd = std::string(path) + ".dist.f32";
    FILE* fi = fopen(pi.c_str(), "wb");
    FILE* fd = fopen(pd.c_str(), "wb");
    bool ok = fi && fd && fwrite(idx, sizeof(int32_t), (size_t)n * k, fi) == (size_t)n * k &&
              fwrite(dist, sizeof(float), (size_t)n * k, fd) == (size_t)n * k;
    if (fi) fclose(fi);
    if (fd) fclose(fd);
    return ok ? TKNN_OK : TKNN_EINVAL;
  }
  unsigned nt = std::max(1u, std::thread::hardware_concurrency());
  nt = (unsigned)std::min<uint64_t>(nt, std::max<uint64_t>(1, n / 4096));
  std::vector<std::string> parts(nt);
  std::vector<std::thread> th;
  for (unsigned t = 0; t < nt; ++t)
    th.emplace_back([&, t]() {
      const uint64_t a = n * t / nt, b = n * (t + 1) / nt;
      std::string& s = parts[t];
      s.reserve((size_t)(b - a) * (size_t)k * 28);
      char buf[96];
      for (uint64_t q = a; q < b; ++q)
        for (int i = 0; i < k; ++i) {
          const int m = snprintf(buf, sizeof(buf), "%llu,%d,%.9g\n", (unsigned long long)q, idx[q * k + i], (double)dist[q * k + i]);
          s.append(buf, (size_t)m);
        }
    });
  for (auto& x : th) x.join();
  FILE* f = fopen(path, "w");
  if (!f) return TKNN_EINVAL;
  bool ok = true;
  for (auto& s : parts) ok = ok && fwrite(s.data(), 1, s.size(), f) == s.size();
  fclose(f);
  return ok ? TKNN_OK : TKNN_EINVAL;
}

// The CSR rows of tknn_radius_search / _query: `query,neighbourIndex,distance` lines (`query,neighbourIndex` without dist),
// or raw arrays when binary != 0 (path + ".off.u64" / ".idx.i32" / ".dist.f32").
TKNN_API int tknn_write_neighbour_lists(const char* path, const uint64_t* offsets, const int32_t* idx, const float* dist,
                                        uint64_t nq, int binary) {
  if (!path || !offsets) return TKNN_EINVAL;
  const uint64_t total = offsets[nq];
  if (total && !idx) return TKNN_EINVAL;
  if (binary) {
    const std::string po = std::string(path) + ".off.u64", pi = std::string(path) + ".idx.i32",
                      pd = std::string(path) + ".dist.f32";
    FILE* fo = fopen(po.c_str(), "wb");
    FILE* fi = fopen(pi.c_str(), "wb");
    FILE* fd = dist ? fopen(pd.c_str(), "wb") : nullptr;
    bool ok = fo && fi && (!dist || fd) && fwrite(offsets, sizeof(uint64_t), (size_t)nq + 1, fo) == (size_t)nq + 1 &&
              fwrite(idx, sizeof(int32_t), (size_t)total, fi) == (size_t)total &&
              (!dist || fwrite(dist, sizeof(float), (size_t)total, fd) == (size_t)total);
    if (fo) fclose(fo);
    if (fi) fclose(fi);
    if (fd) fclose(fd);
    return ok ? TKNN_OK : TKNN_EINVAL;
  }
  unsigned nt = std::max(1u, std::thread::hardware_concurrency());
  nt = (unsigned)std::min<uint64_t>(nt, std::max<uint64_t>(1, total / 65536));
  std::vector<std::string> parts(nt);
  std::vector<std::thread> th;
  for (unsigned t = 0; t < nt; ++t)
    th.emplace_back([&, t]() {
      // rows split so that every thread writes about the same number of entries
      const uint64_t lo = total * t / nt, hi = total * (t + 1) / nt;
      const uint64_t a = (uint64_t)(std::upper_bound(offsets, offsets + nq + 1, lo) - offsets) - 1;
      const uint64_t b = t + 1 == nt ? nq : (uint64_t)(std::upper_bound(offsets, offsets + nq + 1, hi) - offsets) - 1;
      std::string& s = parts[t];
      s.reserve((size_t)(offsets[b] - offsets[a]) * 28);
      char buf[96];
      for (uint64_t q = (t == 0 ? 0 : a); q < b; ++q)
        for (uint64_t e = offsets[q]; e < offsets[q + 1]; ++e) {
          const int m = dist ? snprintf(buf, sizeof(buf), "%llu,%d,%.9g\n", (unsigned long long)q, idx[e], (double)dist[e])
                             : snprintf(buf, sizeof(buf), "%llu,%d\n", (unsigned long long)q, idx[e]);
          s.append(buf, (size_t)m);
        }
    });
  for (auto& x : th) x.join();
  FILE* f = fopen(path, "w");
  if (!f) return TKNN_EINVAL;
  bool ok = true;
  for (auto& s : parts) ok = ok && fwrite(s.data(), 1, s.size(), f) == s.size();
  fclose(f);
  return ok ? TKNN_OK : TKNN_EINVAL;
}

}  // extern "C"
