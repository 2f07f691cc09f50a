// host_util.cc -- host-only parts of libzipc_b200: messages, checksum combines, DOS time,
// ZIP central-directory parsing / archive layout.  (The synthetic workload generators live in synth.cc.)
//
// The archive code restates the *layout rules* of the reference's src/zipc.ml (cited per function);
// payload bytes are produced elsewhere (GPU codecs) and only placed here.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "common.cuh"

namespace zb {
uint32_t gf_mul_host(uint32_t a, uint32_t b);
}  // namespace zb

extern "C" {

const char *zipc_b200_version(void) { return "zipc_b200 0.1.0 (sm_100a)"; }

const char *zipc_b200_strerror(int st) {
  switch (st) {
  case ZIPC_OK: return "";
  case ZIPC_ERR_CORRUPTED: return "Corrupted data stream";
  case ZIPC_ERR_SIZE_EXCEEDED: return "Expected decompression size exceeded";
  case ZIPC_ERR_ZLIB_METHOD: return "Unknown compression method (%d)";
  case ZIPC_ERR_ZLIB_WINDOW: return "Window size too large";
  case ZIPC_ERR_ZLIB_DICT: return "Preset dictionary unsupported";
  case ZIPC_ERR_CHECKSUM: return "Checksum mismatch, expected %lx found %lx)";
  case ZIPC_ERR_NOMEM: return "Out of memory";
  case ZIPC_ERR_INVALID_ARG: return "Invalid argument";
  case ZIPC_ERR_CUDA: return "CUDA failure";
  case ZIPC_ERR_NO_DEVICE: return "No CUDA device";
  case ZIPC_ERR_DST_TOO_SMALL: return "Output arena too small";
  case ZIPC_ERR_ZIP_ZIP64: return "ZIP64 archives are not supported";
  case ZIPC_ERR_ZIP_MULTIPART: return "Multipart archives are not supported";
  case ZIPC_ERR_ZIP_EOCD: return "Corrupted end of central directory record";
  case ZIPC_ERR_ZIP_NO_EOCD: return "Likely not a ZIP archive: no end of central directory record found";
  case ZIPC_ERR_ZIP_SHORT: return "File too short to be a ZIP archive";
  case ZIPC_ERR_ZIP_TRUNC_CD: return "Truncated central directory";
  case ZIPC_ERR_ZIP_CDFH: return "Corrupted central directory file header";
  case ZIPC_ERR_ZIP_LFH: return "Corrupted local file header";
  case ZIPC_ERR_ZIP_COUNT: return "Maximum ZIP member count 65535 exceeded (%d)";
  case ZIPC_ERR_ZIP_PATH_LEN: return "Maximum ZIP path length 65535 exceeded (%d)";
  case ZIPC_ERR_ZIP_SIZE:
    return "Maximum ZIP byte size 4294967295 exceeded by compressed (%d) or decompressed (%d) file size";
  case ZIPC_ERR_ZIP_ENCRYPTED: return "Encrypted file not supported";
  case ZIPC_ERR_ZIP_FORMAT: return "Compression %a not supported";
  case ZIPC_ERR_ZIP_CD_OFFSET: return "Maximum ZIP central directory offset 4294967295 exceeded (%d)";
  case ZIPC_ERR_ZIP_CD_SIZE: return "Maximum ZIP central directory size 4294967295 exceeded (%d)";
  default: return "Unknown error";
  }
}

void zipc_b200_free(void *p) { std::free(p); }

// ---- checksum combines (gather step of the multi-GPU / multi-call path) --------------------------
// crc(A||B) = crc(A) * x^(8|B|) + crc(B) in GF(2)[x]/P; init and final xor cancel.
uint32_t zipc_b200_crc32_combine(uint32_t crc_a, uint32_t crc_b, uint64_t len_b) {
  return zb::gf_mul_host(crc_a, zb::gf_xpow8(len_b)) ^ crc_b;
}
// RFC 1950 only: s1 = s1a + s1b - 1, s2 = s2a + s2b + |B| (s1a - 1)   (mod 65521)
uint32_t zipc_b200_adler32_combine(uint32_t a, uint32_t b, uint64_t len_b) {
  const uint64_t M = 65521;
  uint64_t rem = len_b % M;
  uint64_t s1a = a & 0xffff, s2a = (a >> 16) & 0xffff, s1b = b & 0xffff, s2b = (b >> 16) & 0xffff;
  uint64_t s1 = (s1a + s1b + M - 1) % M;
  uint64_t s2 = (s2a + s2b + rem * ((s1a + M - 1) % M)) % M;
  return (uint32_t)((s2 << 16) | s1);
}

// ---- Zipc.Ptime (zipc.ml:64-125) ----------------------------------------------------------------
static const int64_t kDosEpoch = 315532800;  // 1980-01-01 in POSIX time

static void civil_of_ptime(int64_t t, int &y, int &mo, int &d, int &hh, int &mm, int &ss) {  // zipc.ml:67-86
  int64_t jd = t / 86400 + 2440588, r = t % 86400;
  hh = (int)(r / 3600);
  mm = (int)(r % 3600 / 60);
  ss = (int)(r % 3600 % 60);
  int64_t a = jd + 32044, b = (4 * a + 3) / 146097, c = a - 146097 * b / 4;
  int64_t dd = (4 * c + 3) / 1461, e = c - 1461 * dd / 4, m = (5 * e + 2) / 153;
  d = (int)(e - (153 * m + 2) / 5 + 1);
  mo = (int)(m + 3 - 12 * (m / 10));
  y = (int)(100 * b + dd - 4800 + m / 10);
}

void zipc_b200_ptime_to_dos(int64_t t, int *dos_date, int *dos_time) {  // zipc.ml:115-124
  int y, mo, d, hh, mm, ss;
  civil_of_ptime(t, y, mo, d, hh, mm, ss);
  if (y < 1980) { y = 1980; mo = 1; d = 1; hh = mm = ss = 0; }
  else if (y > 2107) { y = 2107; mo = 12; d = 31; hh = 23; mm = 59; ss = 59; }
  *dos_date = d | (mo << 5) | ((y - 1980) << 9);
  *dos_time = (ss / 2) | (mm << 5) | (hh << 11);
}

int64_t zipc_b200_ptime_of_dos(int dos_date, int dos_time) {  // zipc.ml:96-113
  if (dos_date < 0x21) return kDosEpoch;
  int hh = dos_time >> 11, mm = (dos_time >> 5) & 0x3F, ss = (dos_time & 0x1F) * 2;
  int year = ((dos_date >> 9) & 0x7F) + 1980, month = (dos_date >> 5) & 0xF, day = dos_date & 0x1F;
  int64_t a = (14 - month) / 12, y = year + 4800 - a, m = month + 12 * a - 3;
  int64_t jd = day + (153 * m + 2) / 5 + 365 * y + y / 4 - y / 100 + y / 400 - 32045;
  return (jd - 2440588) * 86400 + hh * 3600 + mm * 60 + ss;
}

// ---- little-endian field access --------------------------------------------------------------------
static inline unsigned rd16(const uint8_t *b, size_t o) { return b[o] | (unsigned)b[o + 1] << 8; }
static inline uint32_t rd32(const uint8_t *b, size_t o) { return rd16(b, o) | (uint32_t)rd16(b, o + 2) << 16; }

static inline bool path_less(const zipc_b200_member &a, const zipc_b200_member &b) {  // String.compare
  size_t n = std::min(a.path_len, b.path_len);
  int c = n ? std::memcmp(a.path, b.path, n) : 0;
  return c ? c < 0 : a.path_len < b.path_len;
}
static inline bool path_eq(const zipc_b200_member &a, const zipc_b200_member &b) {
  return a.path_len == b.path_len && (a.path_len == 0 || std::memcmp(a.path, b.path, a.path_len) == 0);
}
// String_map semantics: increasing path order, the last of equal paths wins (zipc.ml:301-308).
static std::vector<size_t> map_order(const zipc_b200_member *ms, size_t n) {
  std::vector<size_t> idx(n);
  for (size_t i = 0; i < n; i++) idx[i] = i;
  std::stable_sort(idx.begin(), idx.end(), [&](size_t a, size_t b) { return path_less(ms[a], ms[b]); });
  std::vector<size_t> out;
  out.reserve(n);
  for (size_t i = 0; i < n; i++)
    if (i + 1 == n || !path_eq(ms[idx[i]], ms[idx[i + 1]])) out.push_back(idx[i]);
  return out;
}

static inline uint64_t rd64(const uint8_t *b, size_t o) { return rd32(b, o) | (uint64_t)rd32(b, o + 4) << 32; }

// ZIP64 extended information extra field (header id 0x0001, APPNOTE 4.5.3) of a central directory entry: the 64-bit
// values stand in the fixed order uncompressed size, compressed size, local header offset, and only those whose 32-bit
// field holds 0xFFFFFFFF are present.  false: field missing or too short.
static bool zip64_cd_extra(const uint8_t *x, size_t xlen, uint64_t &usize, uint64_t &csize, uint64_t &lfh) {
  const bool wu = usize == 0xFFFFFFFFull, wc = csize == 0xFFFFFFFFull, wl = lfh == 0xFFFFFFFFull;
  if (!wu && !wc && !wl) return true;
  for (size_t o = 0; o + 4 <= xlen;) {
    const unsigned id = rd16(x, o), sz = rd16(x, o + 2);
    if (o + 4 + sz > xlen) return false;
    if (id == 1) {
      size_t q = o + 4;
      const size_t end = q + sz;
      if (wu) { if (q + 8 > end) return false; usize = rd64(x, q); q += 8; }
      if (wc) { if (q + 8 > end) return false; csize = rd64(x, q); q += 8; }
      if (wl) { if (q + 8 > end) return false; lfh = rd64(x, q); q += 8; }
      return true;
    }
    o += 4 + sz;
  }
  return false;
}

// ---- Zipc.of_binary_string (zipc.ml:400-438) ------------------------------------------------------
// One parser for host and device bytes.  It looks at an archive through the few pieces it needs: the window at the end
// where the EOCD is searched, the ZIP64 end record, the central directory, and four fields of each member's local header.
// zipc_b200_zip_parse_ex finds them all in host memory; zipc_b200_zip_parse_dev (zip_api.cu) copies the first three from
// device memory and reads the local headers with one kernel.  The checks are made in the sequential parser's order: member
// k's local header is checked before member k + 1's directory entry.
}  // extern "C"

namespace zb {

// The end of central directory record, searched in tail = bytes [tail_at, len) (zipc.ml:415-425).  tail_at must be at most
// len - kZipTailWindow (or 0).  A ZIP64 end record to read next is reported in e.rec64 (else ~0).
int zip_find_end(const uint8_t *tail, uint64_t tail_at, uint64_t len, unsigned flags, ZipEnd &e) {
  const bool z64 = (flags & ZIPC_ZIP_ALLOW_ZIP64) != 0;
  if (len < 22) return ZIPC_ERR_ZIP_SHORT;
  auto r16 = [&](uint64_t o) { return rd16(tail, (size_t)(o - tail_at)); };   // (only offsets >= tail_at are read)
  auto r32 = [&](uint64_t o) { return rd32(tail, (size_t)(o - tail_at)); };
  int64_t at = (int64_t)len - 22, lowest = (int64_t)len - 65535 - 22;
  for (;; at--) {
    if (at < lowest || at < 0) return ZIPC_ERR_ZIP_NO_EOCD;
    if (r32((uint64_t)at) == 0x06054b50u) break;
  }
  const uint64_t o = (uint64_t)at;
  e.count = r16(o + 10);
  e.cd_size = r32(o + 12);
  e.cd_start = r32(o + 16);
  e.rec64 = ~0ull;
  if (z64 && o >= 20 && r32(o - 20) == 0x07064b50u) {               // ZIP64 EOCD locator (APPNOTE 4.3.15)
    if (r32(o - 16) != 0 || r32(o - 4) > 1) return ZIPC_ERR_ZIP_MULTIPART;
    const uint64_t r = r32(o - 12) | (uint64_t)r32(o - 8) << 32;
    if (r > len || len - r < 56) return ZIPC_ERR_ZIP_EOCD;
    e.rec64 = r;
    return ZIPC_OK;
  }
  if (r16(o + 4) == 0xFFFF) return ZIPC_ERR_ZIP_ZIP64;               // zipc.ml:404
  if (r16(o + 4) != 0 || r16(o + 6) != 0) return ZIPC_ERR_ZIP_MULTIPART;
  return zip_check_cd_range(len, e);
}

// The 56 bytes of the ZIP64 end of central directory record at e.rec64 (APPNOTE 4.3.14).
int zip_read_end64(const uint8_t *r, uint64_t len, ZipEnd &e) {
  if (rd32(r, 0) != 0x06064b50u) return ZIPC_ERR_ZIP_EOCD;
  if (rd32(r, 16) != 0 || rd32(r, 20) != 0) return ZIPC_ERR_ZIP_MULTIPART;
  if (rd64(r, 24) != rd64(r, 32)) return ZIPC_ERR_ZIP_MULTIPART;
  e.count = rd64(r, 32);
  e.cd_size = rd64(r, 40);
  e.cd_start = rd64(r, 48);
  if (e.cd_size > len || e.count > e.cd_size / 46) return ZIPC_ERR_ZIP_EOCD;  // (a count no directory of that size can hold)
  return zip_check_cd_range(len, e);
}

int zip_check_cd_range(uint64_t len, const ZipEnd &e) {
  if (e.cd_start > len || e.cd_size > len - e.cd_start) return ZIPC_ERR_ZIP_EOCD;
  return ZIPC_OK;
}

// The central directory (cd: its e.cd_size bytes) entry by entry, up to the first error, whose status is returned.  ms / lfh
// receive the members before it (paths point into cd); lfh[k].off is member k's local header offset (directories: unused).
int zip_walk_cd(const uint8_t *cd, uint64_t len, unsigned flags, const ZipEnd &e, std::vector<zipc_b200_member> &ms,
                std::vector<ZipLfh> &lfh) {
  const bool z64 = (flags & ZIPC_ZIP_ALLOW_ZIP64) != 0;
  ms.clear();
  lfh.clear();
  ms.reserve((size_t)e.count);
  lfh.reserve((size_t)e.count);
  const uint8_t *s = cd;
  const int64_t cd_max = (int64_t)e.cd_size - 1;
  int64_t i = 0;
  for (uint64_t k = 0; k < e.count; k++) {
    if (i > cd_max) return ZIPC_ERR_ZIP_TRUNC_CD;                     // zipc.ml:394
    if (i + 45 > cd_max || rd32(s, (size_t)i) != 0x02014b50u) return ZIPC_ERR_ZIP_CDFH;
    const size_t o = (size_t)i;
    const unsigned plen = rd16(s, o + 28);
    const int64_t next = i + 46 + plen + rd16(s, o + 30) + rd16(s, o + 32);
    if (next - 1 > cd_max) return ZIPC_ERR_ZIP_CDFH;
    zipc_b200_member m;
    std::memset(&m, 0, sizeof m);
    m.path = reinterpret_cast<const char *>(s + o + 46);
    m.path_len = plen;
    m.mtime = zipc_b200_ptime_of_dos((int)rd16(s, o + 14), (int)rd16(s, o + 12));
    const unsigned hi = rd16(s, o + 40);                               // zipc.ml:360-369
    if (hi) { m.is_dir = (hi & 070000) == 040000; m.mode = (int32_t)(hi & 07777); }
    else if (s[o + 38] & 0x10) { m.is_dir = 1; m.mode = 0755; }
    else { m.is_dir = 0; m.mode = 0644; }
    ZipLfh f;
    std::memset(&f, 0, sizeof f);
    if (!m.is_dir) {
      m.compression = (int32_t)rd16(s, o + 10);
      m.version_made_by = (int32_t)rd16(s, o + 4);
      m.version_needed = (int32_t)rd16(s, o + 6);
      m.gp_flags = (int32_t)rd16(s, o + 8);
      m.compressed_size = rd32(s, o + 20);
      m.decompressed_size = rd32(s, o + 24);
      m.crc32 = rd32(s, o + 16);
      uint64_t off = rd32(s, o + 42);
      if (z64 && !zip64_cd_extra(s + o + 46 + plen, rd16(s, o + 30), m.decompressed_size, m.compressed_size, off)) return ZIPC_ERR_ZIP_CDFH;
      if (off >= len) return ZIPC_ERR_ZIP_CDFH;                       // zipc.ml:380
      f.off = off;
    }
    ms.push_back(m);
    lfh.push_back(f);
    i = next;
  }
  return ZIPC_OK;
}

// The local header checks of the members zip_walk_cd returned, in order, then cd_status (the walk's); on success the members
// sorted by path, a later duplicate winning, into one allocation.  lfh[k]'s fields are read when lfh[k].off + 30 <= len.
// Payloads are at `bytes` + start.  With cd_copy, the directory's cd_size bytes are copied behind the members and the paths
// point there (they pointed into cd).
int zip_parse_finish(std::vector<zipc_b200_member> &ms, const std::vector<ZipLfh> &lfh, int cd_status, uint64_t len,
                     const uint8_t *bytes, const uint8_t *cd, uint64_t cd_size, bool cd_copy, zipc_b200_member **members,
                     size_t *n_out) {
  for (size_t k = 0; k < ms.size(); k++) {
    zipc_b200_member &m = ms[k];
    if (m.is_dir) continue;
    const ZipLfh &f = lfh[k];
    if (f.off + 30 > len || f.sig != 0x04034b50u) return ZIPC_ERR_ZIP_LFH;
    const uint64_t data = f.off + 30 + f.name_len + f.extra_len;
    if (data > len || m.compressed_size > len - data) return ZIPC_ERR_ZIP_LFH;  // zipc.ml:335
    if (m.crc32 == 0) m.crc32 = f.crc;                                // zipc.ml:382-385
    m.compressed_bytes = bytes;
    m.start = data;
  }
  if (cd_status) return cd_status;
  std::vector<size_t> ord = map_order(ms.data(), ms.size());
  const size_t head = sizeof(zipc_b200_member) * (ord.size() ? ord.size() : 1);
  zipc_b200_member *res = static_cast<zipc_b200_member *>(std::malloc(head + (cd_copy ? (size_t)cd_size : 0)));
  if (!res) return ZIPC_ERR_NOMEM;
  const char *names = reinterpret_cast<const char *>(cd);
  if (cd_copy) {
    char *copy = reinterpret_cast<char *>(res) + head;
    if (cd_size) std::memcpy(copy, cd, (size_t)cd_size);
    names = copy;
  }
  for (size_t k = 0; k < ord.size(); k++) {
    res[k] = ms[ord[k]];
    res[k].path = names + (res[k].path - reinterpret_cast<const char *>(cd));
  }
  *members = res;
  *n_out = ord.size();
  return ZIPC_OK;
}

}  // namespace zb

extern "C" {

int zipc_b200_zip_parse(const void *bytes, size_t len, zipc_b200_member **members, size_t *n_out) {
  return zipc_b200_zip_parse_ex(bytes, len, ZIPC_ZIP_REFERENCE, members, n_out);
}

// flags = ZIPC_ZIP_REFERENCE: the reference's behaviour (ZIP64 rejected, zipc.ml:404).  ZIPC_ZIP_ALLOW_ZIP64 (SURVEY.md
// 8f-4, beyond the reference): a ZIP64 end of central directory locator in front of the EOCD is followed, and central
// directory entries take their 64-bit sizes / offsets from the ZIP64 extra field.
int zipc_b200_zip_parse_ex(const void *bytes, size_t len, unsigned flags, zipc_b200_member **members, size_t *n_out) {
  if (!members || !n_out || (!bytes && len)) return ZIPC_ERR_INVALID_ARG;
  *members = nullptr;
  *n_out = 0;
  const uint8_t *s = static_cast<const uint8_t *>(bytes);
  zb::ZipEnd e;
  if (int st = zb::zip_find_end(s, 0, len, flags, e)) return st;
  if (e.rec64 != ~0ull)
    if (int st = zb::zip_read_end64(s + e.rec64, len, e)) return st;
  std::vector<zipc_b200_member> ms;
  std::vector<zb::ZipLfh> lfh;
  const int cd_status = zb::zip_walk_cd(s + e.cd_start, len, flags, e, ms, lfh);
  for (size_t k = 0; k < ms.size(); k++)
    if (!ms[k].is_dir && lfh[k].off + 30 <= len) zb::zip_lfh_fields(s + lfh[k].off, lfh[k]);
  return zb::zip_parse_finish(ms, lfh, cd_status, len, s, s + e.cd_start, e.cd_size, false, members, n_out);
}

// ---- Zipc.encoding_size / to_binary_string (zipc.ml:447-588) -----------------------------------------
uint64_t zipc_b200_zip_encoding_size(const zipc_b200_member *ms, size_t n) {
  uint64_t acc = 22;
  for (size_t k : map_order(ms, n))
    acc += 30 + ms[k].path_len + (ms[k].is_dir ? 0 : ms[k].compressed_size) + 46 + ms[k].path_len;
  return acc;
}

}  // extern "C"

namespace zb {
ZipHdr zip_hdr(const zipc_b200_member &m, const Layout &L, size_t j) {
  ZipHdr h;
  std::memset(&h, 0, sizeof h);
  int date, time;
  zipc_b200_ptime_to_dos(m.mtime, &date, &time);
  h.date = (uint16_t)date;
  h.time = (uint16_t)time;
  if (m.is_dir) { h.made_by = 0x314; h.needed = 20; h.flags = 0x800; h.method = 0; h.crc = 0; h.csize = h.usize = 0; }
  else {
    h.made_by = (uint16_t)m.version_made_by;
    h.needed = (uint16_t)m.version_needed;
    h.flags = (uint16_t)(m.gp_flags & ~8);  // data-descriptor bit is never written (zipc.ml:442-445)
    h.method = (uint16_t)m.compression;
    h.crc = m.crc32;
    h.csize = m.compressed_size;
    h.usize = m.decompressed_size;
  }
  h.ext_attr = (m.is_dir ? 0x10u : 0u) | ((m.is_dir ? 040000u : 0100000u) | ((unsigned)m.mode & 07777u)) << 16;
  h.path_len = m.path_len;
  h.lfh_at = L.lfh_at[j];
  h.cd_at = L.cd_at[j];
  h.big = L.big[j];
  return h;
}

constexpr uint64_t k32 = 0xFFFFFFFFull;
int make_layout(const zipc_b200_member *ms, size_t n, const char *first, unsigned flags, Layout &L) {
  if (!first) first = "mimetype";
  const size_t flen = std::strlen(first);
  const bool allow = (flags & (ZIPC_ZIP_ALLOW_ZIP64 | ZIPC_ZIP_FORCE_ZIP64)) != 0, force = (flags & ZIPC_ZIP_FORCE_ZIP64) != 0;
  L.ord = map_order(ms, n);
  if (L.ord.size() > 0xFFFF && !allow) return ZIPC_ERR_ZIP_COUNT;     // zipc.ml:574
  for (size_t k = 0; k < L.ord.size(); k++) {                          // `first` leads (zipc.ml:575-580)
    const zipc_b200_member &m = ms[L.ord[k]];
    if (m.path_len == flen && std::memcmp(m.path, first, flen) == 0) {
      size_t f = L.ord[k];
      L.ord.erase(L.ord.begin() + (long)k);
      L.ord.insert(L.ord.begin(), f);
      break;
    }
  }
  L.lfh_at.resize(L.ord.size());
  L.cd_at.resize(L.ord.size());
  L.big.assign(L.ord.size(), 0);
  uint64_t pos = 0;
  for (size_t j = 0; j < L.ord.size(); j++) {
    const zipc_b200_member &m = ms[L.ord[j]];
    const uint64_t cs = m.is_dir ? 0 : m.compressed_size, us = m.is_dir ? 0 : m.decompressed_size;
    if (m.path_len > 0xFFFF) return ZIPC_ERR_ZIP_PATH_LEN;
    if (cs >= k32 || us >= k32) {
      if (!allow) return ZIPC_ERR_ZIP_SIZE;                            // zipc.ml:130-133 (File.make refuses these)
      L.big[j] |= 1;
    }
    if (force) L.big[j] |= 3;
    if (pos >= k32) L.big[j] |= 2;  // (only reachable with ZIP64 allowed: without it the directory offset check fails below)
    L.lfh_at[j] = pos;
    pos += zip_lfh_size(m.path_len, L.big[j]) + cs;
  }
  L.cd_start = pos;
  for (size_t j = 0; j < L.ord.size(); j++) {
    L.cd_at[j] = pos;
    pos += zip_cdfh_size(ms[L.ord[j]].path_len, L.big[j]);
  }
  L.cd_size = pos - L.cd_start;
  if (L.ord.empty()) L.cd_start = L.cd_size = 0;                       // zipc.ml:571-572
  L.eocd64 = force || L.ord.size() > 0xFFFF || L.cd_start >= k32 || L.cd_size >= k32;
  if (!allow) {
    if (L.cd_start > k32) return ZIPC_ERR_ZIP_CD_OFFSET;               // zipc.ml:550
    if (L.cd_size > k32) return ZIPC_ERR_ZIP_CD_SIZE;                  // zipc.ml:551
    L.eocd64 = false;
  }
  L.total = pos + zip_end_size(zip_tail(L));
  return ZIPC_OK;
}

std::vector<uint64_t> payload_offsets(const std::vector<zipc_b200_member> &ms, const Layout &L) {
  std::vector<uint64_t> off(ms.size(), ~0ull);
  for (size_t j = 0; j < L.ord.size(); j++) off[L.ord[j]] = L.lfh_at[j] + zip_lfh_size(ms[L.ord[j]].path_len, L.big[j]);
  return off;
}

// Archive layout engine behind zipc_b200_zip_assemble.  out_v == nullptr: compute *out_len only.
// copy_payload == false: payloads are already in place (the pipelined archive call put them there).
int zip_assemble_impl(const zipc_b200_member *ms, size_t n, const char *first, void *out_v, size_t out_cap,
                      size_t *out_len, bool copy_payload, unsigned flags) {
  if (!out_len || (!ms && n)) return ZIPC_ERR_INVALID_ARG;
  Layout L;
  if (int st = make_layout(ms, n, first, flags, L)) return st;
  const std::vector<size_t> &ord = L.ord;
  if (!out_v) { *out_len = (size_t)L.total; return ZIPC_OK; }
  if (L.total > out_cap) { *out_len = (size_t)L.total; return ZIPC_ERR_DST_TOO_SMALL; }
  uint8_t *b = static_cast<uint8_t *>(out_v);
  for (size_t j = 0; j < ord.size(); j++) {  // headers (common.cuh: the same writers as zip_headers_kernel) and payloads
    const zipc_b200_member &m = ms[ord[j]];
    const ZipHdr h = zip_hdr(m, L, j);
    zip_write_lfh(b + h.lfh_at, h, m.path);
    zip_write_cdfh(b + h.cd_at, h, m.path);
    if (copy_payload && !m.is_dir && m.compressed_size)
      std::memcpy(b + h.lfh_at + zip_lfh_size(h.path_len, h.big), m.compressed_bytes + m.start, m.compressed_size);
  }
  zip_write_end(b + L.cd_start + L.cd_size, zip_tail(L));
  *out_len = (size_t)L.total;
  return ZIPC_OK;
}
}  // namespace zb

extern "C" {

int zipc_b200_zip_assemble(const zipc_b200_member *ms, size_t n, const char *first, void *out_v, size_t out_cap,
                           size_t *out_len) {
  if (!out_v) return ZIPC_ERR_INVALID_ARG;
  return zb::zip_assemble_impl(ms, n, first, out_v, out_cap, out_len, true, ZIPC_ZIP_REFERENCE);
}

int zipc_b200_zip_assemble_ex(const zipc_b200_member *ms, size_t n, const char *first, unsigned flags, void *out_v,
                              size_t out_cap, size_t *out_len) {
  if (!out_v) return ZIPC_ERR_INVALID_ARG;
  return zb::zip_assemble_impl(ms, n, first, out_v, out_cap, out_len, true, flags);
}

// Zipc.encoding_size for an archive that may need ZIP64 structures (their presence depends on the offsets, hence `first`).
// 0 if the members cannot be encoded under `flags`.
uint64_t zipc_b200_zip_encoding_size_ex(const zipc_b200_member *ms, size_t n, const char *first, unsigned flags) {
  size_t total = 0;
  if (zb::zip_assemble_impl(ms, n, first, nullptr, 0, &total, false, flags)) return 0;
  return total;
}

}  // extern "C"
