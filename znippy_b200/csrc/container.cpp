// `.znippy` v0.7 container in C++ (no Arrow library): footer, manifest and sub-index reader + writer.
//
// First "next" row of SURVEY.md §8(f): the container is the step on both sides of the hot path — it supplies every
// batch descriptor (blob_offset, blob_size, compressed, uncompressed_size, checksum, fdata_offset).  Restates
//   znippy-common/src/index.rs:43-54    sub-index schema (8 base columns, all non-nullable; plugin columns may follow)
//   znippy-common/src/index.rs:245-277  "ZNPYMIDX" + LE u64 footer
//   znippy-common/src/index.rs:279-367  manifest (pkg_type, repo, module_name, index_offset, index_len, row_count)
//   znippy-common/src/index.rs:374-441  read_znippy_index: footer -> manifest -> every sub-index, rows concatenated
//   znippy-common/src/meta_sink.rs:71-118  writer tail: sub-index(es) -> manifest -> magic + offset
// The sub-indexes and the manifest are Arrow IPC *streams* (encapsulated messages: 0xFFFFFFFF, metadata length,
// Message flatbuffer, 8-byte aligned body).  Only what this schema needs of Arrow is implemented: Schema and
// RecordBatch messages; Utf8, Int/UInt 8-64, Bool, FixedSizeBinary columns; no dictionaries, no body compression.
// Parity: pyarrow reads what this writes and this reads what pyarrow writes (tests/test_container_native.py).
#include <dirent.h>
#include <fcntl.h>
#include <sys/resource.h>
#include <sys/stat.h>
#include <unistd.h>

#include <cstdint>
#include <cstdio>
#include <algorithm>
#include <atomic>
#include <cctype>
#include <condition_variable>
#include <cstring>
#include <deque>
#include <functional>
#include <list>
#include <map>
#include <mutex>
#include <string>
#include <string_view>
#include <thread>
#include <unordered_map>
#include <unordered_set>
#include <vector>

#include "../../include/znippy_cuda.h"
#include "codec_word.h"

namespace {
constexpr uint64_t kMaxRowBytes = 1ull << 32;  // blobs / slices of 4 GiB or more are unsupported (include/znippy_cuda.h)

// ------------------------------------------------------------------------------------------------ flatbuffer reading
struct Span {
  const uint8_t* p;
  size_t n;
};

struct FbErr {};

inline void need(const Span& s, size_t off, size_t len) {
  if (off > s.n || len > s.n - off) throw FbErr();
}
template <typename T>
inline T rd(const Span& s, size_t off) {
  need(s, off, sizeof(T));
  T v;
  memcpy(&v, s.p + off, sizeof(T));
  return v;
}
// position of field `id` inside table at `tbl`, 0 when absent
inline size_t fb_field(const Span& s, size_t tbl, int id) {
  const int32_t so = rd<int32_t>(s, tbl);
  const size_t vt = (size_t)((int64_t)tbl - so);
  const uint16_t vts = rd<uint16_t>(s, vt);
  const size_t slot = 4 + 2 * (size_t)id;
  if (slot + 2 > vts) return 0;
  const uint16_t fo = rd<uint16_t>(s, vt + slot);
  return fo ? tbl + fo : 0;
}
template <typename T>
inline T fb_scalar(const Span& s, size_t tbl, int id, T def) {
  const size_t f = fb_field(s, tbl, id);
  return f ? rd<T>(s, f) : def;
}
inline size_t fb_indirect(const Span& s, size_t tbl, int id) {  // table / vector / string position, 0 when absent
  const size_t f = fb_field(s, tbl, id);
  return f ? f + rd<uint32_t>(s, f) : 0;
}
inline std::string fb_string(const Span& s, size_t pos) {
  if (!pos) return std::string();
  const uint32_t n = rd<uint32_t>(s, pos);
  need(s, pos + 4, n);
  return std::string((const char*)s.p + pos + 4, n);
}

enum ArrowType { T_INT = 2, T_FLOAT = 3, T_BINARY = 4, T_UTF8 = 5, T_BOOL = 6, T_FSB = 15, T_LBINARY = 19, T_LUTF8 = 20 };

struct FieldInfo {
  std::string name;
  int type = 0;
  int bit_width = 0;   // Int
  int byte_width = 0;  // FixedSizeBinary
  int n_buffers = 0;
};

struct Column {  // one decoded column of one record batch (views into the file image)
  const uint8_t* data = nullptr;
  uint64_t data_len = 0;
  const uint8_t* offsets = nullptr;  // utf8
  uint64_t offsets_len = 0;
};

struct IndexImpl {
  uint64_t rows = 0;        // rows held here (all of the archive's, or the groups a ranged open asked for)
  uint64_t row_base = 0;    // archive row number of local row 0
  uint64_t rows_total = 0;  // rows of the whole archive (manifest)
  std::vector<uint64_t> col[4];  // blob_offset, blob_size, fdata_offset, uncompressed_size
  std::vector<uint32_t> chunk_seq;
  std::vector<uint8_t> compressed;
  std::vector<uint8_t> comp_eff;  // what the batch calls get: 4 (enveloped) instead of 1 when the archive declares an envelope
  bool seekable = false;          // znippy_seekable = "zstd": zstd payloads may end in a seek table (ZN_CODEC_SEEKABLE)
  std::vector<uint8_t> checksums;
  std::vector<uint64_t> path_off;  // rows + 1
  std::string paths;
  struct Group {
    int8_t pkg_type;
    std::string repo, module_name;
    uint64_t index_offset, index_len, row_count;
  };
  std::vector<Group> groups;
  std::map<std::string, std::string> metadata;
  std::vector<std::string> field_names;
};

struct Msg {
  int header_type;
  size_t header;  // position of the header table inside meta
  Span meta;
  Span body;
};

// Iterates the encapsulated messages of one IPC stream; returns false at end-of-stream.
bool next_message(const Span& stream, size_t* pos, Msg* m) {
  if (*pos + 8 > stream.n) return false;
  uint32_t cont = rd<uint32_t>(stream, *pos);
  int32_t mlen;
  size_t hdr = 8;
  if (cont == 0xFFFFFFFFu) mlen = rd<int32_t>(stream, *pos + 4);
  else { mlen = (int32_t)cont; hdr = 4; }  // pre-0.15 framing without the continuation marker
  if (mlen == 0) return false;
  if (mlen < 0) throw FbErr();
  need(stream, *pos + hdr, (size_t)mlen);
  m->meta = Span{stream.p + *pos + hdr, (size_t)mlen};
  const size_t root = rd<uint32_t>(m->meta, 0);
  m->header_type = fb_scalar<uint8_t>(m->meta, root, 1, 0);
  m->header = fb_indirect(m->meta, root, 2);
  const int64_t blen = fb_scalar<int64_t>(m->meta, root, 3, 0);
  if (blen < 0) throw FbErr();
  need(stream, *pos + hdr + (size_t)mlen, (size_t)blen);
  m->body = Span{stream.p + *pos + hdr + (size_t)mlen, (size_t)blen};
  *pos += hdr + (size_t)mlen + (size_t)blen;
  return true;
}

void parse_schema(const Msg& m, std::vector<FieldInfo>* fields, std::map<std::string, std::string>* kv) {
  const Span& s = m.meta;
  const size_t fv = fb_indirect(s, m.header, 1);
  if (!fv) throw FbErr();
  const uint32_t nf = rd<uint32_t>(s, fv);
  for (uint32_t i = 0; i < nf; i++) {
    const size_t slot = fv + 4 + 4 * (size_t)i;
    const size_t ft = slot + rd<uint32_t>(s, slot);
    FieldInfo f;
    f.name = fb_string(s, fb_indirect(s, ft, 0));
    f.type = fb_scalar<uint8_t>(s, ft, 2, 0);
    const size_t tt = fb_indirect(s, ft, 3);
    if (fb_indirect(s, ft, 4)) throw FbErr();  // dictionary-encoded columns are not part of this format
    switch (f.type) {
      case T_INT: f.bit_width = tt ? fb_scalar<int32_t>(s, tt, 0, 0) : 0; f.n_buffers = 2; break;
      case T_FLOAT: f.n_buffers = 2; break;
      case T_BOOL: f.n_buffers = 2; break;
      case T_FSB: f.byte_width = tt ? fb_scalar<int32_t>(s, tt, 0, 0) : 0; f.n_buffers = 2; break;
      case T_UTF8: case T_BINARY: case T_LUTF8: case T_LBINARY: f.n_buffers = 3; break;
      default: throw FbErr();
    }
    fields->push_back(f);
  }
  if (kv) {
    const size_t mv = fb_indirect(s, m.header, 2);
    if (mv) {
      const uint32_t nk = rd<uint32_t>(s, mv);
      for (uint32_t i = 0; i < nk; i++) {
        const size_t slot = mv + 4 + 4 * (size_t)i;
        const size_t t = slot + rd<uint32_t>(s, slot);
        (*kv)[fb_string(s, fb_indirect(s, t, 0))] = fb_string(s, fb_indirect(s, t, 1));
      }
    }
  }
}

// Columns of one RecordBatch message, in schema order.  Returns the row count.
uint64_t parse_batch(const Msg& m, const std::vector<FieldInfo>& fields, std::vector<Column>* cols) {
  const Span& s = m.meta;
  const int64_t length = fb_scalar<int64_t>(s, m.header, 0, 0);
  if (fb_indirect(s, m.header, 3)) throw FbErr();  // body compression
  const size_t nodes = fb_indirect(s, m.header, 1), bufs = fb_indirect(s, m.header, 2);
  if (length < 0 || !nodes || !bufs) throw FbErr();
  const uint32_t nn = rd<uint32_t>(s, nodes), nb = rd<uint32_t>(s, bufs);
  if (nn != fields.size()) throw FbErr();
  uint32_t bi = 0;
  cols->assign(fields.size(), Column());
  for (size_t f = 0; f < fields.size(); f++) {
    const int64_t flen = rd<int64_t>(s, nodes + 4 + 16 * f), nulls = rd<int64_t>(s, nodes + 4 + 16 * f + 8);
    if (flen != length || nulls < 0) throw FbErr();
    if (bi + (uint32_t)fields[f].n_buffers > nb) throw FbErr();
    auto buf = [&](uint32_t k, const uint8_t** p, uint64_t* n) {
      const int64_t off = rd<int64_t>(s, bufs + 4 + 16 * (size_t)(bi + k)), len = rd<int64_t>(s, bufs + 4 + 16 * (size_t)(bi + k) + 8);
      if (off < 0 || len < 0) throw FbErr();
      need(m.body, (size_t)off, (size_t)len);
      *p = m.body.p + off;
      *n = (uint64_t)len;
    };
    Column& c = (*cols)[f];
    if (fields[f].n_buffers == 3) { buf(1, &c.offsets, &c.offsets_len); buf(2, &c.data, &c.data_len); }
    else buf(1, &c.data, &c.data_len);
    bi += (uint32_t)fields[f].n_buffers;
  }
  return (uint64_t)length;
}

int find_field(const std::vector<FieldInfo>& f, const char* name) {
  for (size_t i = 0; i < f.size(); i++)
    if (f[i].name == name) return (int)i;
  return -1;
}

uint64_t get_uint(const Column& c, int bits, uint64_t i) {
  switch (bits) {
    case 8: return c.data[i];
    case 16: { uint16_t v; memcpy(&v, c.data + 2 * i, 2); return v; }
    case 32: { uint32_t v; memcpy(&v, c.data + 4 * i, 4); return v; }
    default: { uint64_t v; memcpy(&v, c.data + 8 * i, 8); return v; }
  }
}

// Appends the rows of one sub-index stream to `ix` (columns looked up by NAME, as the reference does).
void read_subindex(const Span& stream, IndexImpl* ix, bool first, bool schema_only = false) {
  size_t pos = 0;
  Msg m;
  if (!next_message(stream, &pos, &m) || m.header_type != 1) throw FbErr();
  std::vector<FieldInfo> fields;
  parse_schema(m, &fields, first ? &ix->metadata : nullptr);
  if (first)
    for (auto& f : fields) ix->field_names.push_back(f.name);
  if (schema_only) return;
  static const char* u64names[4] = {"blob_offset", "blob_size", "fdata_offset", "uncompressed_size"};
  int fi_u64[4], fi_path = find_field(fields, "relative_path"), fi_seq = find_field(fields, "chunk_seq"),
                 fi_comp = find_field(fields, "compressed"), fi_sum = find_field(fields, "checksum");
  auto int_width_ok = [](const FieldInfo& f) { return f.type == T_INT && (f.bit_width == 8 || f.bit_width == 16 || f.bit_width == 32 || f.bit_width == 64); };
  for (int k = 0; k < 4; k++) {
    fi_u64[k] = find_field(fields, u64names[k]);
    if (fi_u64[k] < 0 || !int_width_ok(fields[fi_u64[k]])) throw FbErr();
  }
  if (fi_path < 0 || fi_seq < 0 || fi_comp < 0 || fi_sum < 0) throw FbErr();
  if (fields[fi_path].type != T_UTF8 || fields[fi_comp].type != T_BOOL || fields[fi_sum].type != T_FSB ||
      fields[fi_sum].byte_width != 32 || !int_width_ok(fields[fi_seq]))
    throw FbErr();
  std::vector<Column> cols;
  while (next_message(stream, &pos, &m)) {
    if (m.header_type != 3) continue;  // only record batches carry rows
    const uint64_t n = parse_batch(m, fields, &cols);
    for (int k = 0; k < 4; k++) {
      const Column& c = cols[fi_u64[k]];
      const int bits = fields[fi_u64[k]].bit_width;
      if (n > c.data_len / (uint64_t)(bits / 8)) throw FbErr();
      for (uint64_t i = 0; i < n; i++) ix->col[k].push_back(get_uint(c, bits, i));
    }
    {
      const Column& c = cols[fi_seq];
      const int bits = fields[fi_seq].bit_width;
      if (n > c.data_len / (uint64_t)(bits / 8)) throw FbErr();
      for (uint64_t i = 0; i < n; i++) ix->chunk_seq.push_back((uint32_t)get_uint(c, bits, i));
    }
    {
      const Column& c = cols[fi_comp];
      if (c.data_len < (n + 7) / 8) throw FbErr();
      for (uint64_t i = 0; i < n; i++) ix->compressed.push_back((c.data[i >> 3] >> (i & 7)) & 1);
    }
    {
      const Column& c = cols[fi_sum];
      if (n > c.data_len / 32) throw FbErr();
      ix->checksums.insert(ix->checksums.end(), c.data, c.data + n * 32);
    }
    {
      const Column& c = cols[fi_path];
      if (n >= c.offsets_len / 4) throw FbErr();
      for (uint64_t i = 0; i < n; i++) {
        int32_t a, b;
        memcpy(&a, c.offsets + 4 * i, 4);
        memcpy(&b, c.offsets + 4 * (i + 1), 4);
        if (a < 0 || b < a || (uint64_t)b > c.data_len) throw FbErr();
        ix->paths.append((const char*)c.data + a, (size_t)(b - a));
        ix->path_off.push_back(ix->paths.size());
      }
    }
    ix->rows += n;
  }
}

void read_manifest(const Span& stream, IndexImpl* ix) {
  size_t pos = 0;
  Msg m;
  if (!next_message(stream, &pos, &m) || m.header_type != 1) throw FbErr();
  std::vector<FieldInfo> fields;
  parse_schema(m, &fields, nullptr);
  const int f_pkg = find_field(fields, "pkg_type"), f_repo = find_field(fields, "repo"), f_mod = find_field(fields, "module_name"),
            f_off = find_field(fields, "index_offset"), f_len = find_field(fields, "index_len"), f_rows = find_field(fields, "row_count");
  if (f_pkg < 0 || f_repo < 0 || f_mod < 0 || f_off < 0 || f_len < 0 || f_rows < 0) throw FbErr();
  // exact types (index.rs manifest schema): Int8, Utf8, Utf8, UInt64 x3 — anything else is not this format
  if (fields[f_pkg].type != T_INT || fields[f_pkg].bit_width != 8 || fields[f_repo].type != T_UTF8 || fields[f_mod].type != T_UTF8)
    throw FbErr();
  for (int f : {f_off, f_len, f_rows})
    if (fields[f].type != T_INT || fields[f].bit_width != 64) throw FbErr();
  std::vector<Column> cols;
  while (next_message(stream, &pos, &m)) {
    if (m.header_type != 3) continue;
    const uint64_t n = parse_batch(m, fields, &cols);
    if (n > cols[f_pkg].data_len) throw FbErr();
    for (int f : {f_off, f_len, f_rows})
      if (n > cols[f].data_len / 8) throw FbErr();
    for (int f : {f_repo, f_mod})
      if (n >= cols[f].offsets_len / 4) throw FbErr();
    auto str = [&](int f, uint64_t i) {
      const Column& c = cols[f];
      int32_t a, b;
      if (c.offsets_len < (i + 2) * 4) throw FbErr();
      memcpy(&a, c.offsets + 4 * i, 4);
      memcpy(&b, c.offsets + 4 * (i + 1), 4);
      if (a < 0 || b < a || (uint64_t)b > c.data_len) throw FbErr();
      return std::string((const char*)c.data + a, (size_t)(b - a));
    };
    for (uint64_t i = 0; i < n; i++) {
      IndexImpl::Group g;
      g.pkg_type = (int8_t)get_uint(cols[f_pkg], 8, i);
      g.repo = str(f_repo, i);
      g.module_name = str(f_mod, i);
      g.index_offset = get_uint(cols[f_off], 64, i);
      g.index_len = get_uint(cols[f_len], 64, i);
      g.row_count = get_uint(cols[f_rows], 64, i);
      ix->groups.push_back(g);
    }
  }
}

bool read_range(int fd, uint64_t off, uint64_t len, std::vector<uint8_t>* out) {
  out->resize(len);
  uint64_t done = 0;
  while (done < len) {
    const ssize_t r = pread(fd, out->data() + done, len - done, (off_t)(off + done));
    if (r <= 0) return false;
    done += (uint64_t)r;
  }
  return true;
}

void set_err(char* err, size_t cap, const std::string& m) {
  if (err && cap) snprintf(err, cap, "%s", m.c_str());
}

// ------------------------------------------------------------------------------------------------ flatbuffer writing
// Forward builder: a table is written as [vtable][table] and its children after it, so every uoffset is positive.
struct FbW {
  std::vector<uint8_t> b;
  void align(size_t a) { while (b.size() % a) b.push_back(0); }
  template <typename T>
  void put(T v) { const size_t n = b.size(); b.resize(n + sizeof(T)); memcpy(b.data() + n, &v, sizeof(T)); }
  template <typename T>
  void patch(size_t pos, T v) { memcpy(b.data() + pos, &v, sizeof(T)); }
  // points the uoffset slot at `slot` to the current (aligned) end of the buffer
  void point_here(size_t slot, size_t a = 4) { align(a); patch<uint32_t>(slot, (uint32_t)(b.size() - slot)); }
  size_t string(const std::string& s) {  // returns position
    align(4);
    const size_t p = b.size();
    put<uint32_t>((uint32_t)s.size());
    b.insert(b.end(), s.begin(), s.end());
    b.push_back(0);
    return p;
  }
};

// Table with explicit field layout: each field = (id, size, alignment).  Returns table position; slot positions of the
// fields are returned through `slots` (absolute).  All fields are present.
struct FieldSpec {
  int id, size;
};
size_t fb_table(FbW& w, const std::vector<FieldSpec>& fs, std::vector<size_t>* slots) {
  int max_id = -1;
  for (auto& f : fs) max_id = f.id > max_id ? f.id : max_id;
  // object layout: soffset (4) then fields in descending size order (keeps natural alignment)
  std::vector<FieldSpec> order = fs;
  for (size_t i = 0; i < order.size(); i++)
    for (size_t j = i + 1; j < order.size(); j++)
      if (order[j].size > order[i].size) std::swap(order[i], order[j]);
  std::vector<uint16_t> foff((size_t)max_id + 1, 0);
  size_t obj = 4, maxal = 4;
  for (auto& f : order) {
    const size_t al = (size_t)f.size;
    if (al > maxal) maxal = al;
  }
  // the object starts (soffset word) at a position aligned to the widest field; fields are padded relative to it
  for (auto& f : order) {
    const size_t al = (size_t)f.size;
    while (obj % al) obj++;
    foff[(size_t)f.id] = (uint16_t)obj;
    obj += (size_t)f.size;
  }
  const size_t vts = 4 + 2 * ((size_t)max_id + 1);
  // place vtable so that the table that follows is aligned to maxal
  w.align(2);
  while ((w.b.size() + vts) % maxal) w.b.push_back(0);
  const size_t vt = w.b.size();
  w.put<uint16_t>((uint16_t)vts);
  w.put<uint16_t>((uint16_t)obj);
  for (int i = 0; i <= max_id; i++) w.put<uint16_t>(foff[(size_t)i]);
  const size_t tbl = w.b.size();
  w.put<int32_t>((int32_t)(tbl - vt));
  w.b.resize(tbl + obj, 0);
  slots->assign((size_t)max_id + 1, 0);
  for (auto& f : fs) (*slots)[(size_t)f.id] = tbl + foff[(size_t)f.id];
  return tbl;
}

struct ColSpec {
  const char* name;
  int type;   // ArrowType
  int bits;   // Int
  bool sign;  // Int
  int width;  // FixedSizeBinary
};

// Schema message (metadata only, no body)
std::vector<uint8_t> schema_message(const std::vector<ColSpec>& cols, const std::vector<std::pair<std::string, std::string>>& kv) {
  FbW w;
  w.put<uint32_t>(0);  // root uoffset, patched below
  std::vector<size_t> ms;
  // Message: version(0) i16, header_type(1) u8, header(2) off, bodyLength(3) i64
  w.align(8);
  const size_t msg = fb_table(w, {{0, 2}, {1, 1}, {2, 4}, {3, 8}}, &ms);
  w.patch<uint32_t>(0, (uint32_t)msg);
  w.patch<int16_t>(ms[0], 4);  // MetadataVersion V5
  w.patch<uint8_t>(ms[1], 1);  // Schema
  w.patch<int64_t>(ms[3], 0);
  // Schema: endianness(0) i16, fields(1) off, custom_metadata(2) off
  std::vector<size_t> ss;
  const bool has_kv = !kv.empty();
  w.align(4);
  {
    std::vector<FieldSpec> spec = {{0, 2}, {1, 4}};
    if (has_kv) spec.push_back({2, 4});
    const size_t pos_before = w.b.size();
    (void)pos_before;
    const size_t sch = fb_table(w, spec, &ss);
    w.patch<uint32_t>(ms[2], (uint32_t)(sch - ms[2]));
    w.patch<int16_t>(ss[0], 0);  // little endian
  }
  // fields vector
  w.point_here(ss[1]);
  w.put<uint32_t>((uint32_t)cols.size());
  const size_t fvec = w.b.size();
  for (size_t i = 0; i < cols.size(); i++) w.put<uint32_t>(0);
  for (size_t i = 0; i < cols.size(); i++) {
    const ColSpec& c = cols[i];
    std::vector<size_t> fsl;
    // Field: name(0) off, nullable(1) u8, type_type(2) u8, type(3) off, children(5) off
    w.align(4);
    const size_t ft = fb_table(w, {{0, 4}, {1, 1}, {2, 1}, {3, 4}, {5, 4}}, &fsl);
    w.patch<uint32_t>(fvec + 4 * i, (uint32_t)(ft - (fvec + 4 * i)));
    w.patch<uint8_t>(fsl[1], 0);
    w.patch<uint8_t>(fsl[2], (uint8_t)c.type);
    const size_t np = w.string(c.name);
    w.patch<uint32_t>(fsl[0], (uint32_t)(np - fsl[0]));
    // type table
    std::vector<size_t> tsl;
    w.align(4);
    size_t tt;
    if (c.type == T_INT) {
      tt = fb_table(w, {{0, 4}, {1, 1}}, &tsl);
      w.patch<int32_t>(tsl[0], c.bits);
      w.patch<uint8_t>(tsl[1], c.sign ? 1 : 0);
    } else if (c.type == T_FSB) {
      tt = fb_table(w, {{0, 4}}, &tsl);
      w.patch<int32_t>(tsl[0], c.width);
    } else {
      tt = fb_table(w, {}, &tsl);  // Utf8 / Bool: empty table
    }
    w.patch<uint32_t>(fsl[3], (uint32_t)(tt - fsl[3]));
    w.point_here(fsl[5]);
    w.put<uint32_t>(0);  // children: empty vector
  }
  if (has_kv) {
    w.point_here(ss[2]);
    w.put<uint32_t>((uint32_t)kv.size());
    const size_t kvec = w.b.size();
    for (size_t i = 0; i < kv.size(); i++) w.put<uint32_t>(0);
    for (size_t i = 0; i < kv.size(); i++) {
      std::vector<size_t> ks;
      w.align(4);
      const size_t kt = fb_table(w, {{0, 4}, {1, 4}}, &ks);
      w.patch<uint32_t>(kvec + 4 * i, (uint32_t)(kt - (kvec + 4 * i)));
      const size_t k = w.string(kv[i].first);
      w.patch<uint32_t>(ks[0], (uint32_t)(k - ks[0]));
      const size_t v = w.string(kv[i].second);
      w.patch<uint32_t>(ks[1], (uint32_t)(v - ks[1]));
    }
  }
  w.align(8);
  return w.b;
}

// RecordBatch message metadata for `length` rows with the given buffers (offset, length pairs; one FieldNode per column)
std::vector<uint8_t> batch_message(uint64_t length, size_t ncols, const std::vector<std::pair<uint64_t, uint64_t>>& buffers,
                                   uint64_t body_len) {
  FbW w;
  w.put<uint32_t>(0);
  std::vector<size_t> ms;
  w.align(8);
  const size_t msg = fb_table(w, {{0, 2}, {1, 1}, {2, 4}, {3, 8}}, &ms);
  w.patch<uint32_t>(0, (uint32_t)msg);
  w.patch<int16_t>(ms[0], 4);
  w.patch<uint8_t>(ms[1], 3);  // RecordBatch
  w.patch<int64_t>(ms[3], (int64_t)body_len);
  std::vector<size_t> rs;
  w.align(8);
  const size_t rb = fb_table(w, {{0, 8}, {1, 4}, {2, 4}}, &rs);
  w.patch<uint32_t>(ms[2], (uint32_t)(rb - ms[2]));
  w.patch<int64_t>(rs[0], (int64_t)length);
  // nodes: vector of struct {length i64, null_count i64}: the elements must be 8-aligned, the length word sits before
  w.align(8);
  w.put<uint32_t>(0);  // pad so that (len word at 8k+4) -> elements at 8(k+1)
  w.patch<uint32_t>(rs[1], (uint32_t)(w.b.size() - rs[1]));
  w.put<uint32_t>((uint32_t)ncols);
  for (size_t i = 0; i < ncols; i++) { w.put<int64_t>((int64_t)length); w.put<int64_t>(0); }
  w.align(8);
  w.put<uint32_t>(0);
  w.patch<uint32_t>(rs[2], (uint32_t)(w.b.size() - rs[2]));
  w.put<uint32_t>((uint32_t)buffers.size());
  for (auto& b : buffers) { w.put<int64_t>((int64_t)b.first); w.put<int64_t>((int64_t)b.second); }
  w.align(8);
  return w.b;
}

void append_message(std::vector<uint8_t>* out, const std::vector<uint8_t>& meta, const std::vector<uint8_t>& body) {
  const uint32_t cont = 0xFFFFFFFFu;
  const int32_t mlen = (int32_t)meta.size();  // already a multiple of 8
  out->insert(out->end(), (const uint8_t*)&cont, (const uint8_t*)&cont + 4);
  out->insert(out->end(), (const uint8_t*)&mlen, (const uint8_t*)&mlen + 4);
  out->insert(out->end(), meta.begin(), meta.end());
  out->insert(out->end(), body.begin(), body.end());
}
void append_eos(std::vector<uint8_t>* out) {
  const uint32_t e[2] = {0xFFFFFFFFu, 0};
  out->insert(out->end(), (const uint8_t*)e, (const uint8_t*)e + 8);
}

struct BodyW {
  std::vector<uint8_t> b;
  std::vector<std::pair<uint64_t, uint64_t>> bufs;
  void add(const void* p, uint64_t n) {
    bufs.push_back({b.size(), n});
    b.insert(b.end(), (const uint8_t*)p, (const uint8_t*)p + n);
    while (b.size() % 8) b.push_back(0);
  }
  void add_empty() { bufs.push_back({b.size(), 0}); }  // absent validity bitmap (no nulls)
};

bool write_all(int fd, const void* p, size_t n, uint64_t off) {
  size_t done = 0;
  while (done < n) {
    const ssize_t r = pwrite(fd, (const uint8_t*)p + done, n - done, (off_t)(off + done));
    if (r <= 0) return false;
    done += (size_t)r;
  }
  return true;
}

}  // namespace

// ================================================================================================ C ABI: reader
struct zn_index {
  IndexImpl ix;
};

// Opens the index; only the sub-indexes that hold archive rows [want_lo, want_hi) are parsed (a GPU shard of a large
// archive needs its own groups, not all of them: 1.3 M rows cost ~0.25 s to parse).  Local row r = archive row
// row_base + r.  The first sub-index's schema is always read (metadata, field names).
static zn_index* index_open_range(const char* path, uint64_t want_lo, uint64_t want_hi, char* err, size_t errcap) {
  const int fd = open(path, O_RDONLY);
  if (fd < 0) { set_err(err, errcap, "cannot open archive"); return nullptr; }
  zn_index* h = new zn_index();
  try {
    struct stat st;
    if (fstat(fd, &st) != 0 || st.st_size < 16) throw std::string("not a znippy archive (too small)");
    const uint64_t flen = (uint64_t)st.st_size;
    std::vector<uint8_t> tail;
    if (!read_range(fd, flen - 16, 16, &tail)) throw std::string("read error");
    if (memcmp(tail.data(), "ZNPYMIDX", 8) != 0) throw std::string("v0.6 archives are not supported");  // index.rs:387-389
    uint64_t moff;
    memcpy(&moff, tail.data() + 8, 8);
    if (moff > flen - 16) throw std::string("manifest offset outside file");
    std::vector<uint8_t> mbytes;
    if (!read_range(fd, moff, flen - 16 - moff, &mbytes)) throw std::string("read error");
    read_manifest(Span{mbytes.data(), mbytes.size()}, &h->ix);
    bool first = true;
    std::vector<uint8_t> sub;
    uint64_t g_lo = 0;
    for (auto& g : h->ix.groups) {
      if (g.index_offset > flen || g.index_len > flen - g.index_offset) throw std::string("sub-index outside file");
      const uint64_t g_hi = g_lo + g.row_count;
      const bool wanted = g_hi > want_lo && g_lo < want_hi;
      if (wanted || first) {
        if (!read_range(fd, g.index_offset, g.index_len, &sub)) throw std::string("read error");
        const uint64_t before = h->ix.rows;
        read_subindex(Span{sub.data(), sub.size()}, &h->ix, first, !wanted);
        if (wanted && h->ix.rows - before != g.row_count) throw std::string("sub-index row count differs from the manifest");
      }
      if (!wanted && h->ix.rows == 0) h->ix.row_base = g_hi;  // still in front of the first wanted group
      first = false;
      g_lo = g_hi;
    }
    h->ix.rows_total = g_lo;
    if (h->ix.rows == 0) h->ix.row_base = std::min(want_lo, g_lo);
    h->ix.path_off.insert(h->ix.path_off.begin(), 0);
    // Index columns come from the file: every blob must lie inside the payload region (before the first sub-index)
    // and both sizes stay below the 4 GiB the batch calls support, so that no later sum of them can wrap.
    h->ix.comp_eff = h->ix.compressed;
    {
      auto it = h->ix.metadata.find("znippy_envelope");
      if (it != h->ix.metadata.end()) {
        if (it->second != "ZNB1") throw std::string("archive declares an unknown blob envelope: " + it->second);
        for (auto& c : h->ix.comp_eff) c = c ? 4 : 0;
      }
      it = h->ix.metadata.find("znippy_seekable");
      if (it != h->ix.metadata.end()) {
        if (it->second != "zstd") throw std::string("archive declares an unknown seekable format: " + it->second);
        h->ix.seekable = true;
      }
    }
    uint64_t payload_end = moff;
    for (auto& g : h->ix.groups) payload_end = std::min(payload_end, g.index_offset);
    for (uint64_t r = 0; r < h->ix.rows; r++) {
      const uint64_t bo = h->ix.col[0][r], bs = h->ix.col[1][r], fo = h->ix.col[2][r], us = h->ix.col[3][r];
      if (bs >= kMaxRowBytes || us >= kMaxRowBytes) throw std::string("index row " + std::to_string(r) + ": blob of 4 GiB or more");
      if (bo > payload_end || bs > payload_end - bo) throw std::string("index row " + std::to_string(r) + ": blob outside the payload region");
      if (fo > (1ull << 62)) throw std::string("index row " + std::to_string(r) + ": file offset out of range");
    }
  } catch (const std::string& m) {
    set_err(err, errcap, m);
    delete h;
    h = nullptr;
  } catch (const FbErr&) {
    set_err(err, errcap, "malformed Arrow IPC metadata in archive index");
    delete h;
    h = nullptr;
  } catch (const std::exception& e) {
    set_err(err, errcap, e.what());
    delete h;
    h = nullptr;
  }
  close(fd);
  return h;
}

extern "C" zn_index* zn_index_open(const char* path, char* err, size_t errcap) { return index_open_range(path, 0, ~0ull, err, errcap); }

extern "C" void zn_index_close(zn_index* h) { delete h; }
extern "C" uint64_t zn_index_rows(const zn_index* h) { return h ? h->ix.rows : 0; }
extern "C" const uint64_t* zn_index_u64(const zn_index* h, int col) { return (h && col >= 0 && col < 4) ? h->ix.col[col].data() : nullptr; }
extern "C" const uint32_t* zn_index_chunk_seq(const zn_index* h) { return h ? h->ix.chunk_seq.data() : nullptr; }
extern "C" const uint8_t* zn_index_compressed(const zn_index* h) { return h ? h->ix.compressed.data() : nullptr; }
extern "C" const uint8_t* zn_index_checksums(const zn_index* h) { return h ? h->ix.checksums.data() : nullptr; }
extern "C" const char* zn_index_path(const zn_index* h, uint64_t row, uint32_t* len) {
  if (!h || row >= h->ix.rows) return nullptr;
  if (len) *len = (uint32_t)(h->ix.path_off[row + 1] - h->ix.path_off[row]);
  return h->ix.paths.data() + h->ix.path_off[row];
}
extern "C" uint64_t zn_index_groups(const zn_index* h) { return h ? h->ix.groups.size() : 0; }
extern "C" int zn_index_group(const zn_index* h, uint64_t g, int8_t* pkg_type, const char** repo, uint64_t* index_offset,
                              uint64_t* index_len, uint64_t* row_count) {
  if (!h || g >= h->ix.groups.size()) return ZN_E_ARG;
  const auto& G = h->ix.groups[g];
  if (pkg_type) *pkg_type = G.pkg_type;
  if (repo) *repo = G.repo.c_str();
  if (index_offset) *index_offset = G.index_offset;
  if (index_len) *index_len = G.index_len;
  if (row_count) *row_count = G.row_count;
  return ZN_OK;
}
extern "C" const char* zn_index_metadata(const zn_index* h, const char* key) {
  if (!h || !key) return nullptr;
  auto it = h->ix.metadata.find(key);
  return it == h->ix.metadata.end() ? nullptr : it->second.c_str();
}
extern "C" uint32_t zn_index_field_count(const zn_index* h) { return h ? (uint32_t)h->ix.field_names.size() : 0; }
extern "C" const char* zn_index_field_name(const zn_index* h, uint32_t i) {
  return (h && i < h->ix.field_names.size()) ? h->ix.field_names[i].c_str() : nullptr;
}

// ================================================================================================ C ABI: writer
struct zn_index_writer {
  int fd;
  uint64_t cursor;
  std::vector<IndexImpl::Group> groups;
  std::vector<std::pair<std::string, std::string>> kv;
};

extern "C" zn_index_writer* zn_index_writer_create(int fd, uint64_t blob_end) {
  zn_index_writer* w = new zn_index_writer();
  w->fd = fd;
  w->cursor = blob_end;
  return w;
}
extern "C" int zn_index_writer_metadata(zn_index_writer* w, const char* key, const char* value) {
  if (!w || !key || !value) return ZN_E_ARG;
  w->kv.push_back({key, value});
  return ZN_OK;
}

// One sub-index (one record batch) for a (pkg_type, repo) group: index.rs:131-191 + meta_sink.rs:71-101
extern "C" int zn_index_writer_push_group(zn_index_writer* w, int8_t pkg_type, const char* repo, uint64_t n,
                                          const char* const* paths, const uint32_t* chunk_seq, const uint64_t* fdata_offset,
                                          const uint8_t* compressed, const uint64_t* uncompressed_size,
                                          const uint64_t* blob_offset, const uint64_t* blob_size, const uint8_t* checksums) {
  if (!w || (n && (!paths || !chunk_seq || !fdata_offset || !compressed || !uncompressed_size || !blob_offset || !blob_size || !checksums)))
    return ZN_E_ARG;
  static const std::vector<ColSpec> cols = {
      {"relative_path", T_UTF8, 0, false, 0}, {"chunk_seq", T_INT, 32, false, 0}, {"fdata_offset", T_INT, 64, false, 0},
      {"compressed", T_BOOL, 0, false, 0},    {"uncompressed_size", T_INT, 64, false, 0}, {"blob_offset", T_INT, 64, false, 0},
      {"blob_size", T_INT, 64, false, 0},     {"checksum", T_FSB, 0, false, 32}};
  std::vector<uint8_t> out;
  append_message(&out, schema_message(cols, w->kv), {});
  BodyW body;
  {
    std::vector<int32_t> offs(n + 1, 0);
    std::string data;
    for (uint64_t i = 0; i < n; i++) { data += paths[i]; offs[i + 1] = (int32_t)data.size(); }
    body.add_empty(); body.add(offs.data(), (n + 1) * 4); body.add(data.data(), data.size());
  }
  body.add_empty(); body.add(chunk_seq, n * 4);
  body.add_empty(); body.add(fdata_offset, n * 8);
  {
    std::vector<uint8_t> bits((n + 7) / 8, 0);
    for (uint64_t i = 0; i < n; i++) if (compressed[i]) bits[i >> 3] |= (uint8_t)(1u << (i & 7));
    body.add_empty(); body.add(bits.data(), bits.size());
  }
  body.add_empty(); body.add(uncompressed_size, n * 8);
  body.add_empty(); body.add(blob_offset, n * 8);
  body.add_empty(); body.add(blob_size, n * 8);
  body.add_empty(); body.add(checksums, n * 32);
  append_message(&out, batch_message(n, cols.size(), body.bufs, body.b.size()), body.b);
  append_eos(&out);
  if (!write_all(w->fd, out.data(), out.size(), w->cursor)) return ZN_E_ARG;
  IndexImpl::Group g;
  g.pkg_type = pkg_type;
  g.repo = repo ? repo : "";
  g.index_offset = w->cursor;
  g.index_len = out.size();
  g.row_count = n;
  w->groups.push_back(g);
  w->cursor += out.size();
  return ZN_OK;
}

// manifest + footer + fsync (meta_sink.rs:103-118); destroys the writer
extern "C" int zn_index_writer_finish(zn_index_writer* w) {
  if (!w) return ZN_E_ARG;
  static const std::vector<ColSpec> cols = {{"pkg_type", T_INT, 8, true, 0},      {"repo", T_UTF8, 0, false, 0},
                                            {"module_name", T_UTF8, 0, false, 0}, {"index_offset", T_INT, 64, false, 0},
                                            {"index_len", T_INT, 64, false, 0},   {"row_count", T_INT, 64, false, 0}};
  const uint64_t n = w->groups.size();
  std::vector<uint8_t> out;
  append_message(&out, schema_message(cols, {}), {});
  BodyW body;
  std::vector<int8_t> pk(n);
  std::vector<uint64_t> io(n), il(n), rc(n);
  std::vector<int32_t> ro(n + 1, 0), mo(n + 1, 0);
  std::string rd_, md_;
  for (uint64_t i = 0; i < n; i++) {
    pk[i] = w->groups[i].pkg_type; io[i] = w->groups[i].index_offset; il[i] = w->groups[i].index_len; rc[i] = w->groups[i].row_count;
    rd_ += w->groups[i].repo; ro[i + 1] = (int32_t)rd_.size();
    md_ += w->groups[i].module_name; mo[i + 1] = (int32_t)md_.size();
  }
  body.add_empty(); body.add(pk.data(), n);
  body.add_empty(); body.add(ro.data(), (n + 1) * 4); body.add(rd_.data(), rd_.size());
  body.add_empty(); body.add(mo.data(), (n + 1) * 4); body.add(md_.data(), md_.size());
  body.add_empty(); body.add(io.data(), n * 8);
  body.add_empty(); body.add(il.data(), n * 8);
  body.add_empty(); body.add(rc.data(), n * 8);
  append_message(&out, batch_message(n, cols.size(), body.bufs, body.b.size()), body.b);
  append_eos(&out);
  int rcode = ZN_OK;
  if (!write_all(w->fd, out.data(), out.size(), w->cursor)) rcode = ZN_E_ARG;
  uint8_t footer[16];
  memcpy(footer, "ZNPYMIDX", 8);
  memcpy(footer + 8, &w->cursor, 8);
  if (rcode == ZN_OK && !write_all(w->fd, footer, 16, w->cursor + out.size())) rcode = ZN_E_ARG;
  if (rcode == ZN_OK && ftruncate(w->fd, (off_t)(w->cursor + out.size() + 16)) != 0) rcode = ZN_E_ARG;
  if (rcode == ZN_OK) fsync(w->fd);
  delete w;
  return rcode;
}

// ================================================================================================ native decompress_archive
extern "C" int zn_decompress_rows_ex(zn_ctx* c, int archive_fd, uint64_t row_lo, uint64_t row_hi, const uint64_t* blob_offset,
                                     const uint64_t* blob_size, const uint64_t* fdata_offset, const uint8_t* compressed,
                                     const uint64_t* uncompressed_size, const uint8_t* checksums, const int* out_fd,
                                     size_t batch_bytes, int io_threads, uint64_t* corrupt_rows_out, zn_verify_stats* stats,
                                     const char* out_root, const char* paths, const uint64_t* path_off);  // znippy_cuda.cu

// decompress.rs:39-222 end to end: index -> (pre-create output files) -> zn_decompress_rows -> VerifyReport.
extern "C" int zn_archive_decompress(zn_ctx* ctx, const char* index_path, int save_data, const char* out_dir, uint64_t row_lo,
                                     uint64_t row_hi, size_t batch_bytes, int io_threads, zn_verify_report* report, char* err,
                                     size_t errcap) {
  if (!ctx || !index_path || !report) return ZN_E_ARG;
  memset(report, 0, sizeof *report);
  zn_index* h = index_open_range(index_path, row_lo, row_hi, err, errcap);  // this shard's groups only
  if (!h) return ZN_E_ARG;
  const IndexImpl& ix = h->ix;
  // from here on rows are LOCAL to the parsed groups (a file's rows never leave its group, so every neighbour the
  // shard logic below looks at is present)
  if (row_hi > ix.rows_total) row_hi = ix.rows_total;
  if (row_lo > row_hi) row_lo = row_hi;
  row_lo = row_lo >= ix.row_base ? row_lo - ix.row_base : 0;
  row_hi = row_hi >= ix.row_base ? row_hi - ix.row_base : 0;
  if (row_hi > ix.rows) row_hi = ix.rows;
  if (row_lo > row_hi) row_lo = row_hi;
  std::unordered_set<std::string_view> uniq;
  uniq.reserve((size_t)(row_hi - row_lo) * 2);
  int rc = ZN_OK;
  for (uint64_t r = row_lo; r < row_hi; r++) uniq.insert(std::string_view(ix.paths.data() + ix.path_off[r], ix.path_off[r + 1] - ix.path_off[r]));
  // decompress.rs:74-101 keeps one fd per path for the whole run.  With 100 000 small files that needs a raised
  // RLIMIT_NOFILE, so here the row range is worked off in windows of at most `max_open` distinct paths (rows of a
  // file are adjacent in the index): same files, same bytes, any descriptor limit.
  size_t max_open = 4096;
  {
    struct rlimit rl;
    if (getrlimit(RLIMIT_NOFILE, &rl) == 0) {
      if (rl.rlim_cur < rl.rlim_max) { rl.rlim_cur = rl.rlim_max; setrlimit(RLIMIT_NOFILE, &rl); getrlimit(RLIMIT_NOFILE, &rl); }
      const size_t lim = rl.rlim_cur == RLIM_INFINITY ? 65536 : (size_t)rl.rlim_cur;
      max_open = std::max<size_t>(16, std::min<size_t>(lim > 128 ? (lim - 64) / 2 : 16, 16384));
    }
    if (const char* e = getenv("ZN_MAX_OPEN_FILES")) max_open = std::max(1, atoi(e));  // tests: force several windows
  }
  const int afd = open(index_path, O_RDONLY);
  if (afd < 0) { set_err(err, errcap, "cannot open archive"); rc = ZN_E_ARG; }
  zn_verify_stats total;
  memset(&total, 0, sizeof total);
  std::vector<int> fds;
  if (save_data) fds.assign(ix.rows, -1);
  std::vector<uint64_t> corrupt(row_hi - row_lo + 1);
  std::unordered_set<std::string> created;  // a path met again in a later window is re-opened without truncation
  std::unordered_set<std::string> made_dirs;  // directories known to exist (100 000 files in 100 directories: 100 mkdir walks)
  const std::string root = out_dir ? out_dir : ".";
  // helper threads for the per-file system calls of a window (open / ftruncate / close): 100 000 small files are 300 000 of
  // them, and issued from one thread they took longer than decoding and writing the files did
  auto for_each_parallel = [&](size_t n, const std::function<void(size_t)>& f) {
    const int nt = n >= 64 ? std::max(1, std::min(io_threads, 16)) : 1;
    if (nt == 1) { for (size_t i = 0; i < n; i++) f(i); return; }
    std::atomic<size_t> cur{0};
    std::vector<std::thread> ts;
    for (int t = 0; t < nt; t++)
      ts.emplace_back([&] { for (size_t i; (i = cur.fetch_add(1)) < n;) f(i); });
    for (auto& t : ts) t.join();
  };
  struct OutFile {
    std::string_view rel;
    uint64_t first_row;
    int fd = -1;
    int err = 0;  // 1 open failed, 2 ftruncate failed
  };
  for (uint64_t w_lo = row_lo; w_lo < row_hi && rc == ZN_OK;) {
    std::vector<OutFile> open_files;
    uint64_t w_hi = w_lo;
    if (save_data) {
      // 1. the window: rows up to max_open distinct paths (rows of a file are adjacent, so a path that differs from its
      //    predecessor's is looked up, every other row reuses the previous answer)
      std::unordered_map<std::string_view, uint32_t> at;
      std::vector<uint32_t> row_file;
      std::vector<std::string_view> lazy_dirs;  // paths of this window's one-row files (their directories must exist)
      uint32_t prev = ~0u;
      auto path_of = [&](uint64_t r) { return std::string_view(ix.paths.data() + ix.path_off[r], ix.path_off[r + 1] - ix.path_off[r]); };
      for (; w_hi < row_hi; w_hi++) {
        const std::string_view rel = path_of(w_hi);
        // a file that is exactly this one row needs no descriptor here: the writer thread that holds the row opens, writes
        // and closes it (zn_decompress_rows_ex); only multi-row files count against the descriptor window
        if ((w_hi == 0 || path_of(w_hi - 1) != rel) && (w_hi + 1 >= ix.rows || path_of(w_hi + 1) != rel) && !created.count(std::string(rel))) {
          lazy_dirs.push_back(rel);
          row_file.push_back(~0u);
          prev = ~0u;
          continue;
        }
        uint32_t fi;
        if (prev != ~0u && open_files[prev].rel == rel) fi = prev;
        else {
          auto it = at.find(rel);
          if (it != at.end()) fi = it->second;
          else {
            if (open_files.size() >= max_open) break;
            fi = (uint32_t)open_files.size();
            OutFile of;
            of.rel = rel;
            of.first_row = w_hi;
            open_files.push_back(of);
            at.emplace(rel, fi);
          }
        }
        row_file.push_back(fi);
        prev = fi;
      }
      // 2. directories (serial: few; out_dir itself first), 3. open / size the files (parallel)
      if (made_dirs.insert("").second) {
        for (size_t p = 1; p <= root.size(); p++)
          if (p == root.size() || root[p] == '/') mkdir(root.substr(0, p).c_str(), 0755);
      }
      auto ensure_dir = [&](std::string_view rel) {
        const size_t slash = rel.find_last_of('/');
        if (slash == std::string_view::npos) return;
        const std::string dir(rel.substr(0, slash));
        if (!made_dirs.insert(dir).second) return;
        const std::string full = root + "/" + dir;
        for (size_t p = root.size() + 1; p <= full.size(); p++)
          if (p == full.size() || full[p] == '/') mkdir(full.substr(0, p).c_str(), 0755);
      };
      {
        std::string_view last_dir;
        for (const std::string_view rel : lazy_dirs) {  // consecutive files share their directory: one set lookup per change
          const size_t slash = rel.find_last_of('/');
          const std::string_view dir = slash == std::string_view::npos ? std::string_view() : rel.substr(0, slash);
          if (dir == last_dir) continue;
          last_dir = dir;
          ensure_dir(rel);
        }
      }
      for (const OutFile& of : open_files) ensure_dir(of.rel);
      for_each_parallel(open_files.size(), [&](size_t k) {
        OutFile& of = open_files[k];
        const std::string rel(of.rel);
        const std::string full = root + "/" + rel;
        const bool again = created.count(rel) != 0;  // (read-only here; the set is updated after the parallel part)
        // A file whose rows straddle [row_lo, row_hi) is also written by the neighbouring shard (another process or
        // GPU): truncating it here could destroy chunks that shard has already written.  It is opened without
        // O_TRUNC and sized to its full length from the index instead (idempotent, never cuts live data).
        auto same_path = [&](uint64_t r) {
          return ix.path_off[r + 1] - ix.path_off[r] == rel.size() && memcmp(ix.paths.data() + ix.path_off[r], rel.data(), rel.size()) == 0;
        };
        const bool shared = (row_lo > 0 && same_path(row_lo - 1)) || (row_hi < ix.rows && same_path(row_hi));
        of.fd = open(full.c_str(), O_CREAT | O_WRONLY | (again || shared ? 0 : O_TRUNC), 0644);
        if (of.fd < 0) { of.err = 1; return; }
        if (shared && !again) {
          uint64_t a = of.first_row, b = of.first_row, size = 0;
          while (a > 0 && same_path(a - 1)) a--;
          while (b + 1 < ix.rows && same_path(b + 1)) b++;
          for (uint64_t r = a; r <= b; r++) size = std::max(size, ix.col[2][r] + ix.col[3][r]);
          if (ftruncate(of.fd, (off_t)size) != 0) of.err = 2;
        }
      });
      for (const OutFile& of : open_files) {
        created.insert(std::string(of.rel));
        if (of.err && rc == ZN_OK) {
          set_err(err, errcap, std::string(of.err == 1 ? "failed to open output file " : "failed to size output file ") + root + "/" + std::string(of.rel));
          rc = ZN_E_ARG;
        }
      }
      for (uint64_t r = w_lo; r < w_hi; r++) fds[r] = row_file[r - w_lo] == ~0u ? -2 : open_files[row_file[r - w_lo]].fd;
      for (const std::string_view rel : lazy_dirs) created.insert(std::string(rel));
    } else {
      w_hi = row_hi;
    }
    if (rc == ZN_OK) {
      zn_verify_stats st;
      rc = zn_decompress_rows_ex(ctx, afd, w_lo, w_hi, ix.col[0].data(), ix.col[1].data(), ix.col[2].data(), ix.comp_eff.data(),
                                 ix.col[3].data(), ix.checksums.data(), save_data ? fds.data() : nullptr, batch_bytes, io_threads,
                                 corrupt.data(), &st, root.c_str(), ix.paths.data(), ix.path_off.data());
      if (rc != ZN_OK) set_err(err, errcap, zn_last_error(ctx));
      total.corrupt_rows += st.corrupt_rows;
      total.total_written_bytes += st.total_written_bytes;
      total.verified_bytes += st.verified_bytes;
      total.corrupt_bytes += st.corrupt_bytes;
      total.total_chunks += st.total_chunks;
    }
    for_each_parallel(open_files.size(), [&](size_t k) { if (open_files[k].fd >= 0) close(open_files[k].fd); });
    w_lo = w_hi;
  }
  if (rc == ZN_OK) {
    report->total_files = uniq.size();
    report->corrupt_files = total.corrupt_rows;  // the reference counts corrupt ROWS here (decompress.rs:210)
    report->verified_files = report->total_files > report->corrupt_files ? report->total_files - report->corrupt_files : 0;
    report->total_bytes = total.total_written_bytes;
    report->verified_bytes = total.verified_bytes;
    report->corrupt_bytes = total.corrupt_bytes;
    report->chunks = total.total_chunks;
  }
  if (afd >= 0) close(afd);
  zn_index_close(h);
  return rc;
}

// ================================================================================================ native write pipeline
// compress_stream (znippy-compress/src/stream_packer.rs:58-372) as a C++ object: entries are cut into <= 8 MiB rounds
// (:169-202) straight into a pinned staging slot (the Magazine slot of slotpool.rs:93-130); a full slot is ONE
// zn_compress_batch (blake3 + frame per slice, the barrel body :217-232) plus one zn_hash_batch for the store-as-is
// rounds (:222-227); the writer step pwrites the payloads at a running cursor (:252-285); finish() sorts the blob
// metas by (file_index, chunk_seq), groups them by (pkg_type, repo) in BTreeMap order and emits sub-indexes, manifest
// and footer (:293-346, meta_sink.rs:71-118).
extern "C" void* zn_ctx_pinned_alloc(size_t bytes);
extern "C" void zn_ctx_pinned_free(void* p);

namespace {
constexpr uint64_t kSliceSize = 8ull * 1024 * 1024;  // stream_packer.rs:31

bool should_skip_compression(const std::string& path) {  // index.rs:470-488: last extension only, case-insensitive
  static const char* ext[] = {"zip", "gz", "bz2", "xz", "lz", "lzma", "7z", "rar", "cab", "jar", "war", "ear", "zst", "sz",
                              "lz4", "tgz", "txz", "tbz", "apk", "dmg", "deb", "rpm", "arrow", "mpeg", "mpg", "jpeg", "jpg",
                              "gif", "bmp", "png", "crate", "znippy", "zdata", "parquet", "webp", "webm"};
  const size_t slash = path.find_last_of('/');
  const std::string base = slash == std::string::npos ? path : path.substr(slash + 1);
  const size_t dot = base.find_last_of('.');
  if (dot == std::string::npos) return false;
  std::string e = base.substr(dot + 1);
  for (auto& ch : e) ch = (char)tolower((unsigned char)ch);
  for (const char* x : ext)
    if (e == x) return true;
  return false;
}

struct Round {
  uint64_t file_index, fdata_offset, stage_off, len;
  uint32_t chunk_seq;
  bool skip;
};
struct BlobMetaRow {
  uint64_t file_index, fdata_offset, usize, blob_offset, blob_size;
  uint32_t chunk_seq;
  bool compressed;
  uint8_t checksum[32];
};
struct EntryInfo {
  std::string path, repo;
  int8_t pkg_type;
  bool skip;
};
}  // namespace

// The Magazine (slotpool.rs:93-227) as a three-stage pipeline over `kSlots` pinned slots:
//   fill     the caller (zn_archive_writer_add) or the directory readers (zn_archive_compress_dir) copy source bytes
//            into the slot they hold; a full slot is published
//   gpu      one thread: ONE zn_compress_batch per slot (blake3 + frame per slice, the barrel body
//            stream_packer.rs:217-232 / slot_packer.rs:551-572) + one zn_hash_batch for its store-as-is rounds
//   write    one thread (the reference's writer thread, stream_packer.rs:252-285): pwrite of the payloads at the running
//            cursor, blob metas, report counters; then the slot is free again (Ejector::release_one)
// so that filling slot k+2, compressing slot k+1 and writing slot k overlap.  The zn_ctx is used by the gpu thread
// only, for as long as the writer lives.
struct WSlot {
  uint8_t* stage = nullptr;  // pinned: source slices
  uint8_t* outb = nullptr;   // pinned: compressed frames
  uint64_t outb_cap = 0, used = 0;
  std::vector<Round> rounds;
  std::vector<uint64_t> d_off, c_out;
  std::vector<uint8_t> c_dig, s_dig;
  std::atomic<uint32_t> pending{0};  // directory readers still copying into this slot
};

struct zn_archive_writer {
  static constexpr int kSlots = 3;
  zn_ctx* ctx;
  int fd;
  bool no_skip;
  int level, codec;       // codec: the word without ZN_CODEC_ENVELOPE, as zn_compress_batch takes it
  zn::CodecWord cw;       // its parts; cw.envelope: blobs of compressed rows are ZNB1 envelopes (store-if-incompressible)
  uint64_t slot_bytes, out_cursor = 0;
  WSlot slots[kSlots];
  WSlot* cur = nullptr;  // the slot being filled
  std::mutex mu;
  std::condition_variable cv;
  std::deque<WSlot*> free_q, gpu_q, write_q;
  bool closing = false;
  int rc = ZN_OK;  // first failure of any stage (sticky)
  std::thread gpu_thread, write_thread;
  std::vector<BlobMetaRow> metas;
  std::vector<EntryInfo> entries;
  zn_compression_report rep;
  std::string err;
};

namespace {
void writer_fail(zn_archive_writer* w, int rc, const std::string& msg) {
  std::lock_guard<std::mutex> g(w->mu);
  if (w->rc == ZN_OK) { w->rc = rc; w->err = msg; }
}

// gpu stage of one slot
int slot_compress(zn_archive_writer* w, WSlot* s) {
  const size_t n = s->rounds.size();
  std::vector<uint64_t> c_off, c_len, s_off, s_len;
  s->d_off.clear();
  uint64_t dcur = 0;
  for (size_t i = 0; i < n; i++) {
    const Round& r = s->rounds[i];
    if (r.skip) { s_off.push_back(r.stage_off); s_len.push_back(r.len); }
    else {
      c_off.push_back(r.stage_off); c_len.push_back(r.len);
      s->d_off.push_back(dcur);
      dcur += (zn_compress_bound(r.len, w->codec) + 15) & ~15ull;
    }
  }
  s->d_off.push_back(dcur);
  if (dcur > s->outb_cap) {
    if (s->outb) zn_ctx_pinned_free(s->outb);
    s->outb = (uint8_t*)zn_ctx_pinned_alloc(dcur + 4096);
    s->outb_cap = s->outb ? dcur + 4096 : 0;
    if (!s->outb) { writer_fail(w, ZN_E_NOMEM, "pinned output allocation failed"); return ZN_E_NOMEM; }
  }
  s->c_out.assign(c_off.size(), 0);
  s->c_dig.assign(c_off.size() * 32, 0);
  s->s_dig.assign(s_off.size() * 32, 0);
  std::vector<uint32_t> c_st(c_off.size());
  if (!c_off.empty()) {
    const int rc = zn_compress_batch(w->ctx, s->stage, c_off.data(), c_len.data(), (uint32_t)c_off.size(), w->level, w->codec, s->outb,
                                     s->d_off.data(), s->c_out.data(), s->c_dig.data(), c_st.data());
    if (rc != ZN_OK) { writer_fail(w, rc, zn_last_error(w->ctx)); return rc; }
    for (uint32_t st : c_st)
      if (st != ZN_S_OK) { writer_fail(w, ZN_E_ARG, "compress failed for a slice"); return ZN_E_ARG; }  // `?` propagates, stream_packer.rs:230
  }
  if (!s_off.empty()) {
    const int rc = zn_hash_batch(w->ctx, s->stage, s_off.data(), s_len.data(), (uint32_t)s_off.size(), s->s_dig.data());
    if (rc != ZN_OK) { writer_fail(w, rc, zn_last_error(w->ctx)); return rc; }
  }
  return ZN_OK;
}

// writer stage of one slot, in round order (stream_packer.rs:252-285)
int slot_write(zn_archive_writer* w, WSlot* s) {
  size_t ci = 0, si = 0;
  // payloads of consecutive rounds are gathered into runs so that 100 000 small blobs are not 100 000 pwrite calls
  std::vector<uint8_t> run;
  uint64_t run_at = w->out_cursor;
  auto flush_run = [&]() -> bool {
    const bool ok = run.empty() || write_all(w->fd, run.data(), run.size(), run_at);
    run.clear();
    return ok;
  };
  for (size_t i = 0; i < s->rounds.size(); i++) {
    const Round& r = s->rounds[i];
    BlobMetaRow m;
    m.file_index = r.file_index; m.chunk_seq = r.chunk_seq; m.fdata_offset = r.fdata_offset; m.usize = r.len;
    m.compressed = !r.skip; m.blob_offset = w->out_cursor;
    const uint8_t* payload;
    uint8_t hdr[ZN_ENVELOPE_ZNB1_MAX_HEADER];
    size_t hl = 0;
    if (r.skip) { payload = s->stage + r.stage_off; m.blob_size = r.len; memcpy(m.checksum, s->s_dig.data() + 32 * si, 32); si++; }
    else {
      payload = s->outb + s->d_off[ci]; m.blob_size = s->c_out[ci]; memcpy(m.checksum, s->c_dig.data() + 32 * ci, 32); ci++;
      if (w->cw.envelope) {
        // store-if-incompressible (deferred in the reference, TODO_NOW.md:37-38): a frame that did not shrink the slice
        // is dropped for the raw bytes; the row stays `compressed` and the envelope says RAW
        uint32_t pc = w->cw.base == ZN_CODEC_LZ4 ? ZN_PAYLOAD_LZ4_FRAME : ZN_PAYLOAD_ZSTD;
        if (m.blob_size >= r.len) { pc = ZN_PAYLOAD_RAW; payload = s->stage + r.stage_off; m.blob_size = r.len; }
        hl = zn_envelope_znb1_header(pc, r.len, hdr, sizeof hdr);
      }
    }
    const uint64_t total = hl + m.blob_size;
    if (total <= (256u << 10)) {
      if (run.empty()) run_at = w->out_cursor;
      run.insert(run.end(), hdr, hdr + hl);
      run.insert(run.end(), payload, payload + m.blob_size);
      if (run.size() >= (8u << 20) && !flush_run()) { writer_fail(w, ZN_E_ARG, "pwrite failed"); return ZN_E_ARG; }
    } else {
      if (!flush_run() || (hl && !write_all(w->fd, hdr, hl, w->out_cursor)) ||
          !write_all(w->fd, payload, m.blob_size, w->out_cursor + hl)) { writer_fail(w, ZN_E_ARG, "pwrite failed"); return ZN_E_ARG; }
    }
    m.blob_size = total;
    w->out_cursor += total;
    w->metas.push_back(m);
    w->rep.chunks++;
    w->rep.total_bytes_in += r.len;
    w->rep.total_bytes_out += total;
    if (r.skip) w->rep.uncompressed_bytes += r.len; else w->rep.compressed_bytes += r.len;
  }
  if (!flush_run()) { writer_fail(w, ZN_E_ARG, "pwrite failed"); return ZN_E_ARG; }
  return ZN_OK;
}

void gpu_loop(zn_archive_writer* w) {
  for (;;) {
    WSlot* s;
    {
      std::unique_lock<std::mutex> l(w->mu);
      w->cv.wait(l, [&] { return !w->gpu_q.empty() || w->closing; });
      if (w->gpu_q.empty()) break;
      s = w->gpu_q.front();
      w->gpu_q.pop_front();
    }
    while (s->pending.load(std::memory_order_acquire)) std::this_thread::yield();  // directory readers still copying
    bool ok;
    { std::lock_guard<std::mutex> g(w->mu); ok = w->rc == ZN_OK; }
    if (ok) slot_compress(w, s);
    {
      std::lock_guard<std::mutex> g(w->mu);
      w->write_q.push_back(s);
    }
    w->cv.notify_all();
  }
  {
    std::lock_guard<std::mutex> g(w->mu);
    w->write_q.push_back(nullptr);  // end marker
  }
  w->cv.notify_all();
}

void write_loop(zn_archive_writer* w) {
  for (;;) {
    WSlot* s;
    {
      std::unique_lock<std::mutex> l(w->mu);
      w->cv.wait(l, [&] { return !w->write_q.empty(); });
      s = w->write_q.front();
      w->write_q.pop_front();
    }
    if (!s) break;
    bool ok;
    { std::lock_guard<std::mutex> g(w->mu); ok = w->rc == ZN_OK; }
    if (ok) slot_write(w, s);
    s->rounds.clear();
    s->used = 0;
    {
      std::lock_guard<std::mutex> g(w->mu);
      w->free_q.push_back(s);
    }
    w->cv.notify_all();
  }
}

WSlot* writer_acquire(zn_archive_writer* w) {
  std::unique_lock<std::mutex> l(w->mu);
  w->cv.wait(l, [&] { return !w->free_q.empty(); });
  WSlot* s = w->free_q.front();
  w->free_q.pop_front();
  return s;
}

void writer_publish(zn_archive_writer* w) {
  if (!w->cur) return;
  {
    std::lock_guard<std::mutex> g(w->mu);
    w->gpu_q.push_back(w->cur);
  }
  w->cur = nullptr;
  w->cv.notify_all();
}

// Reserves room for one round in the current slot (publishing it first when full); returns where its bytes go.
uint8_t* writer_reserve(zn_archive_writer* w, uint64_t file_index, uint32_t seq, uint64_t fdata_offset, uint64_t n, bool skip,
                        WSlot** slot_out) {
  if (w->cur && w->cur->used + n > w->slot_bytes) writer_publish(w);
  if (!w->cur) w->cur = writer_acquire(w);
  WSlot* s = w->cur;
  Round r;
  r.file_index = file_index; r.chunk_seq = seq; r.fdata_offset = fdata_offset; r.stage_off = s->used; r.len = n; r.skip = skip;
  s->rounds.push_back(r);
  uint8_t* dst = s->stage + s->used;
  s->used += (n + 15) & ~15ull;
  if (slot_out) *slot_out = s;
  return dst;
}

uint64_t writer_new_entry(zn_archive_writer* w, const char* relative_path, int has_pkg_type, int8_t pkg_type, const char* repo, bool* skip) {
  EntryInfo e;
  e.path = relative_path;
  e.repo = repo ? repo : "";
  e.pkg_type = has_pkg_type ? pkg_type : 0;
  e.skip = !w->no_skip && should_skip_compression(e.path);
  *skip = e.skip;
  w->entries.push_back(e);
  w->rep.total_files++;
  if (e.skip) w->rep.uncompressed_files++; else w->rep.compressed_files++;
  return w->entries.size() - 1;
}
}  // namespace

extern "C" zn_archive_writer* zn_archive_writer_create(zn_ctx* ctx, const char* output_path, int no_skip, int level, int codec,
                                                       size_t slot_bytes) {
  if (!ctx || !output_path) return nullptr;
  zn::CodecWord cw;
  if (zn::codec_split(codec, level, true, &cw)) return nullptr;
  if (slot_bytes < 2 * kSliceSize) slot_bytes = 2 * kSliceSize;
  const int fd = open(output_path, O_CREAT | O_RDWR | O_TRUNC, 0644);
  if (fd < 0) return nullptr;
  zn_archive_writer* w = new zn_archive_writer();
  w->ctx = ctx; w->fd = fd; w->no_skip = no_skip != 0; w->level = level; w->codec = codec & ~ZN_CODEC_ENVELOPE;
  w->slot_bytes = slot_bytes;
  w->cw = cw;
  memset(&w->rep, 0, sizeof w->rep);
  for (auto& s : w->slots) {
    s.stage = (uint8_t*)zn_ctx_pinned_alloc(slot_bytes + 4096);
    if (!s.stage) {
      for (auto& t : w->slots) if (t.stage) zn_ctx_pinned_free(t.stage);
      close(fd); delete w; return nullptr;
    }
    w->free_q.push_back(&s);
  }
  w->gpu_thread = std::thread(gpu_loop, w);
  w->write_thread = std::thread(write_loop, w);
  return w;
}

extern "C" const char* zn_archive_writer_error(const zn_archive_writer* w) { return w ? w->err.c_str() : "null writer"; }

extern "C" int zn_archive_writer_add(zn_archive_writer* w, const char* relative_path, const uint8_t* data, uint64_t len,
                                     int has_pkg_type, int8_t pkg_type, const char* repo) {
  if (!w || !relative_path || (len && !data)) return ZN_E_ARG;
  bool skip;
  const uint64_t fi = writer_new_entry(w, relative_path, has_pkg_type, pkg_type, repo, &skip);
  uint64_t off = 0;
  uint32_t seq = 0;
  do {  // an empty entry still yields one zero-length round (stream_packer.rs:169-183)
    const uint64_t n = len - off < kSliceSize ? len - off : kSliceSize;
    uint8_t* dst = writer_reserve(w, fi, seq++, off, n, skip, nullptr);
    if (n) memcpy(dst, data + off, n);
    off += n;
  } while (off < len);
  std::lock_guard<std::mutex> g(w->mu);
  return w->rc;
}

extern "C" int zn_archive_writer_finish(zn_archive_writer* w, zn_compression_report* report) {
  if (!w) return ZN_E_ARG;
  writer_publish(w);
  {
    std::lock_guard<std::mutex> g(w->mu);
    w->closing = true;
  }
  w->cv.notify_all();
  w->gpu_thread.join();
  w->write_thread.join();
  int rc = w->rc;
  if (rc == ZN_OK) {
    std::stable_sort(w->metas.begin(), w->metas.end(), [](const BlobMetaRow& a, const BlobMetaRow& b) {
      return a.file_index != b.file_index ? a.file_index < b.file_index : a.chunk_seq < b.chunk_seq;
    });
    std::map<std::pair<int8_t, std::string>, std::vector<const BlobMetaRow*>> groups;  // BTreeMap order
    for (auto& m : w->metas) groups[{w->entries[m.file_index].pkg_type, w->entries[m.file_index].repo}].push_back(&m);
    if (groups.empty()) groups[{0, ""}];
    zn_index_writer* iw = zn_index_writer_create(w->fd, w->out_cursor);
    {  // config echoed into the schema metadata (index.rs:73-85)
      const long cores = sysconf(_SC_NPROCESSORS_ONLN) > 0 ? sysconf(_SC_NPROCESSORS_ONLN) : 1;
      zn_index_writer_metadata(iw, "znippy_format_version", "3");
      zn_index_writer_metadata(iw, "max_core_in_flight", std::to_string((cores * 9 + 9) / 10).c_str());
      zn_index_writer_metadata(iw, "max_core_in_compress", std::to_string(cores).c_str());
      zn_index_writer_metadata(iw, "max_mem_allowed", "0");
      zn_index_writer_metadata(iw, "min_free_memory_ratio", "0.1");
      zn_index_writer_metadata(iw, "file_split_block_size", "10485760");
      zn_index_writer_metadata(iw, "max_chunks", "128");
      zn_index_writer_metadata(iw, "compression_level", "19");
      zn_index_writer_metadata(iw, "zstd_output_buffer_size", "1048576");
      if (w->cw.envelope) zn_index_writer_metadata(iw, "znippy_envelope", "ZNB1");  // readers resolve compressed rows through zn_envelope_parse
      if (w->cw.seekable) zn_index_writer_metadata(iw, "znippy_seekable", "zstd");  // range reads use the seek tables
    }
    for (auto& kv : groups) {
      const auto& rows = kv.second;
      const uint64_t n = rows.size();
      std::vector<const char*> paths(n);
      std::vector<uint32_t> seq(n);
      std::vector<uint64_t> fo(n), us(n), bo(n), bs(n);
      std::vector<uint8_t> cp(n), ck(n * 32);
      for (uint64_t i = 0; i < n; i++) {
        const BlobMetaRow* m = rows[i];
        paths[i] = w->entries[m->file_index].path.c_str();
        seq[i] = m->chunk_seq; fo[i] = m->fdata_offset; us[i] = m->usize; bo[i] = m->blob_offset; bs[i] = m->blob_size;
        cp[i] = m->compressed ? 1 : 0;
        memcpy(ck.data() + 32 * i, m->checksum, 32);
      }
      const int prc = zn_index_writer_push_group(iw, kv.first.first, kv.first.second.c_str(), n, paths.data(), seq.data(), fo.data(),
                                                 cp.data(), us.data(), bo.data(), bs.data(), ck.data());
      if (prc != ZN_OK && rc == ZN_OK) rc = prc;
    }
    const int frc = zn_index_writer_finish(iw);
    if (frc != ZN_OK && rc == ZN_OK) rc = frc;
  }
  if (report) *report = w->rep;
  close(w->fd);
  for (auto& s : w->slots) {
    if (s.stage) zn_ctx_pinned_free(s.stage);
    if (s.outb) zn_ctx_pinned_free(s.outb);
  }
  delete w;
  return rc;
}

// compress_dir (znippy-compress: walk -> readers -> Magazine -> workers -> writer, slot_packer.rs:329-609) natively:
// the directory is walked once (sorted, so the archive is deterministic), every file is cut into rounds that are
// ASSIGNED a place in a slot right away (sizes come from stat), and `io_threads` readers pread the file bytes into
// those places in parallel; a slot goes to the GPU stage when its last reader is done.  No per-file call crosses the
// language boundary.
namespace {
struct DirFile {
  std::string rel, full;
  uint64_t size;
};
void walk_dir(const std::string& root, const std::string& rel, std::vector<DirFile>* out) {
  const std::string dir = rel.empty() ? root : root + "/" + rel;
  DIR* d = opendir(dir.c_str());
  if (!d) return;
  std::vector<std::string> names;
  while (dirent* e = readdir(d)) {
    if (!strcmp(e->d_name, ".") || !strcmp(e->d_name, "..")) continue;
    names.push_back(e->d_name);
  }
  closedir(d);
  std::sort(names.begin(), names.end());
  for (auto& n : names) {
    const std::string r = rel.empty() ? n : rel + "/" + n, full = root + "/" + r;
    struct stat st;
    if (lstat(full.c_str(), &st) != 0) continue;
    if (S_ISDIR(st.st_mode)) walk_dir(root, r, out);
    else if (S_ISREG(st.st_mode)) out->push_back({r, full, (uint64_t)st.st_size});
  }
}
struct ReadJob {
  const DirFile* f;
  uint64_t off, len;
  uint8_t* dst;
  WSlot* slot;
};
}  // namespace

extern "C" int zn_archive_compress_dir(zn_ctx* ctx, const char* input_dir, const char* output_path, int no_skip, int level, int codec,
                                       size_t slot_bytes, int io_threads, zn_compression_report* report, char* err, size_t errcap) {
  if (!ctx || !input_dir || !output_path) return ZN_E_ARG;
  zn::CodecWord cw;
  if (const char* why = zn::codec_split(codec, level, true, &cw)) {
    set_err(err, errcap, why);
    return ZN_E_ARG;
  }
  std::vector<DirFile> files;
  walk_dir(input_dir, "", &files);
  zn_archive_writer* w = zn_archive_writer_create(ctx, output_path, no_skip, level, codec, slot_bytes ? slot_bytes : (256u << 20));
  if (!w) { set_err(err, errcap, "cannot create the output archive"); return ZN_E_ARG; }
  if (io_threads < 1) io_threads = 1;
  std::mutex jm;
  std::condition_variable jcv;
  std::deque<ReadJob> jobs;
  bool jobs_done = false;
  std::atomic<int> io_err{0};
  std::vector<std::thread> readers;
  for (int t = 0; t < io_threads; t++)
    readers.emplace_back([&] {
      int fd = -1;
      const DirFile* open_for = nullptr;
      for (;;) {
        ReadJob j;
        {
          std::unique_lock<std::mutex> l(jm);
          jcv.wait(l, [&] { return !jobs.empty() || jobs_done; });
          if (jobs.empty()) break;
          j = jobs.front();
          jobs.pop_front();
        }
        if (j.len) {
          if (open_for != j.f) {
            if (fd >= 0) close(fd);
            fd = open(j.f->full.c_str(), O_RDONLY);
            open_for = j.f;
          }
          uint64_t done = 0;
          while (fd >= 0 && done < j.len) {
            const ssize_t r = pread(fd, j.dst + done, j.len - done, (off_t)(j.off + done));
            if (r <= 0) break;
            done += (uint64_t)r;
          }
          if (done < j.len) { io_err = 1; memset(j.dst + done, 0, j.len - done); }
        }
        j.slot->pending.fetch_sub(1, std::memory_order_release);
      }
      if (fd >= 0) close(fd);
    });
  for (const DirFile& f : files) {
    bool skip;
    const uint64_t fi = writer_new_entry(w, f.rel.c_str(), 0, 0, "", &skip);
    uint64_t off = 0;
    uint32_t seq = 0;
    do {
      const uint64_t n = f.size - off < kSliceSize ? f.size - off : kSliceSize;
      WSlot* s;
      uint8_t* dst = writer_reserve(w, fi, seq++, off, n, skip, &s);
      s->pending.fetch_add(1, std::memory_order_relaxed);
      {
        std::lock_guard<std::mutex> g(jm);
        jobs.push_back({&f, off, n, dst, s});
      }
      jcv.notify_one();
      off += n;
    } while (off < f.size);
  }
  {
    std::lock_guard<std::mutex> g(jm);
    jobs_done = true;
  }
  jcv.notify_all();
  for (auto& t : readers) t.join();
  if (io_err) writer_fail(w, ZN_E_ARG, "failed to read an input file");
  std::string msg;
  { std::lock_guard<std::mutex> g(w->mu); msg = w->err; }
  const int rc = zn_archive_writer_finish(w, report);
  if (rc != ZN_OK) set_err(err, errcap, msg.empty() ? "compress_dir failed" : msg);
  return rc;
}

// ================================================================================================ native random access
// ZnippyArchive (znippy-common/src/archive.rs:46-168): open = index + per-file chunk lists sorted by fdata_offset
// (:68-136); extract_files (:27-29) = every chunk of every requested file in ONE zn_decode_verify_batch, no digest
// compare (extract_file does not verify, :144-168), chunks concatenated in fdata_offset order.
struct zn_archive {
  zn_index* index = nullptr;
  int fd = -1;
  struct FileEntry {
    uint64_t size = 0;
    std::vector<uint64_t> rows;  // sorted by fdata_offset
  };
  std::map<std::string, FileEntry> files;
  std::vector<std::map<std::string, FileEntry>::const_iterator> order;  // first-seen order for listing
  // LRU of decoded slices (SURVEY §8f-2): an artifact server asks for the same hot files again and again; a slice that was
  // decoded once is answered from host memory afterwards.  Keyed by index row, bounded by bytes, off until a budget is set.
  struct Cache {
    std::mutex mu;
    uint64_t budget = 0, used = 0, hits = 0, misses = 0, evictions = 0;
    std::list<std::pair<uint64_t, std::vector<uint8_t>>> lru;  // front = most recent
    std::unordered_map<uint64_t, std::list<std::pair<uint64_t, std::vector<uint8_t>>>::iterator> at;
  } cache;
};

extern "C" zn_archive* zn_archive_open(const char* path, char* err, size_t errcap) {
  zn_index* ix = zn_index_open(path, err, errcap);
  if (!ix) return nullptr;
  const int fd = open(path, O_RDONLY);
  if (fd < 0) { set_err(err, errcap, "cannot open archive"); zn_index_close(ix); return nullptr; }
  zn_archive* a = new zn_archive();
  a->index = ix;
  a->fd = fd;
  const IndexImpl& I = ix->ix;
  for (uint64_t r = 0; r < I.rows; r++) {
    const std::string p(I.paths.data() + I.path_off[r], I.path_off[r + 1] - I.path_off[r]);
    auto ins = a->files.emplace(p, zn_archive::FileEntry());
    if (ins.second) a->order.push_back(ins.first);
    ins.first->second.size += I.col[3][r];
    ins.first->second.rows.push_back(r);
  }
  for (auto& kv : a->files)
    std::stable_sort(kv.second.rows.begin(), kv.second.rows.end(), [&](uint64_t x, uint64_t y) { return I.col[2][x] < I.col[2][y]; });
  return a;
}
extern "C" void zn_archive_close(zn_archive* a) {
  if (!a) return;
  if (a->fd >= 0) close(a->fd);
  zn_index_close(a->index);
  delete a;
}
extern "C" uint64_t zn_archive_file_count(const zn_archive* a) { return a ? a->order.size() : 0; }
extern "C" const char* zn_archive_file_name(const zn_archive* a, uint64_t i, uint64_t* size) {
  if (!a || i >= a->order.size()) return nullptr;
  if (size) *size = a->order[i]->second.size;
  return a->order[i]->first.c_str();
}
extern "C" int zn_archive_file_size(const zn_archive* a, const char* path, uint64_t* size) {  // contains + file_size
  if (!a || !path) return 0;
  auto it = a->files.find(path);
  if (it == a->files.end()) return 0;
  if (size) *size = it->second.size;
  return 1;
}

extern "C" int zn_archive_set_cache(zn_archive* a, uint64_t budget_bytes) {
  if (!a) return ZN_E_ARG;
  std::lock_guard<std::mutex> g(a->cache.mu);
  a->cache.budget = budget_bytes;
  while (a->cache.used > budget_bytes && !a->cache.lru.empty()) {
    a->cache.used -= a->cache.lru.back().second.size();
    a->cache.at.erase(a->cache.lru.back().first);
    a->cache.lru.pop_back();
    a->cache.evictions++;
  }
  return ZN_OK;
}
extern "C" int zn_archive_cache_stats(zn_archive* a, uint64_t stats[5]) {
  if (!a || !stats) return ZN_E_ARG;
  std::lock_guard<std::mutex> g(a->cache.mu);
  stats[0] = a->cache.hits; stats[1] = a->cache.misses; stats[2] = a->cache.evictions; stats[3] = a->cache.used; stats[4] = a->cache.lru.size();
  return ZN_OK;
}

// file_status[i]: 0 ok, 1 not in archive, 2 a chunk failed to decode (first failing chunk's per-blob status in the high half)
extern "C" int zn_archive_extract_files(zn_ctx* ctx, zn_archive* a, const char* const* paths, uint32_t n, uint8_t* out_base,
                                        const uint64_t* out_off, uint32_t* file_status) {
  if (!ctx || !a || (n && (!paths || !out_base || !out_off || !file_status))) return ZN_E_ARG;
  const IndexImpl& I = a->index->ix;
  std::vector<uint64_t> rows, bo, bl, ol, oo;
  std::vector<uint8_t> cf;
  std::vector<uint32_t> owner;
  uint64_t in_cur = 0;
  zn_archive::Cache& K = a->cache;
  for (uint32_t k = 0; k < n; k++) {
    auto it = a->files.find(paths[k]);
    if (it == a->files.end()) { file_status[k] = 1; continue; }
    file_status[k] = 0;
    uint64_t pos = out_off[k];
    for (uint64_t r : it->second.rows) {
      if (K.budget) {  // a cached slice is answered from host memory and never reaches the batch
        std::lock_guard<std::mutex> g(K.mu);
        auto c = K.at.find(r);
        if (c != K.at.end()) {
          K.lru.splice(K.lru.begin(), K.lru, c->second);
          memcpy(out_base + pos, c->second->second.data(), c->second->second.size());
          pos += I.col[3][r];
          K.hits++;
          continue;
        }
        K.misses++;
      }
      rows.push_back(r);
      bo.push_back(in_cur); bl.push_back(I.col[1][r]); cf.push_back(I.comp_eff[r]); ol.push_back(I.col[3][r]); oo.push_back(pos);
      owner.push_back(k);
      in_cur += (I.col[1][r] + 15) & ~15ull;
      pos += I.col[3][r];
    }
  }
  if (rows.empty()) return ZN_OK;
  if (rows.size() > 0xFFFFFFF0ull) return ZN_E_ARG;  // row sizes were bounded by zn_index_open, so in_cur cannot wrap
  uint8_t* stage = (uint8_t*)zn_ctx_pinned_alloc(in_cur + 4096);
  if (!stage) return ZN_E_NOMEM;
  std::atomic<int> io_err{0};
  {
    std::atomic<size_t> cur{0};
    auto body = [&] {
      for (;;) {
        const size_t i = cur.fetch_add(1);
        if (i >= rows.size()) break;
        uint64_t done = 0;
        const uint64_t len = bl[i], off = I.col[0][rows[i]];
        while (done < len) {
          const ssize_t r = pread(a->fd, stage + bo[i] + done, len - done, (off_t)(off + done));
          if (r <= 0) { io_err = 1; return; }
          done += (uint64_t)r;
        }
      }
    };
    std::vector<std::thread> ts;
    const int nt = rows.size() >= 16 ? 4 : 1;
    for (int t = 1; t < nt; t++) ts.emplace_back(body);
    body();
    for (auto& t : ts) t.join();
  }
  int rc = io_err ? ZN_E_ARG : ZN_OK;
  if (rc == ZN_OK) {
    std::vector<uint32_t> st(rows.size());
    rc = zn_decode_verify_batch(ctx, stage, bo.data(), bl.data(), cf.data(), ol.data(), nullptr, out_base, oo.data(),
                                (uint32_t)rows.size(), st.data(), nullptr);
    if (rc == ZN_OK)
      for (size_t i = 0; i < rows.size(); i++)
        if (st[i] != ZN_S_OK && file_status[owner[i]] == 0) file_status[owner[i]] = 2u | (st[i] << 16);
    if (rc == ZN_OK && K.budget) {
      std::lock_guard<std::mutex> g(K.mu);
      for (size_t i = 0; i < rows.size(); i++) {
        if (st[i] != ZN_S_OK || ol[i] > K.budget || K.at.count(rows[i])) continue;
        while (K.used + ol[i] > K.budget && !K.lru.empty()) {  // evict from the cold end
          K.used -= K.lru.back().second.size();
          K.at.erase(K.lru.back().first);
          K.lru.pop_back();
          K.evictions++;
        }
        K.lru.emplace_front(rows[i], std::vector<uint8_t>(out_base + oo[i], out_base + oo[i] + ol[i]));
        K.at[rows[i]] = K.lru.begin();
        K.used += ol[i];
      }
    }
  }
  zn_ctx_pinned_free(stage);
  return rc;
}

// envelope.cpp: zn_envelope_parse over the first `head` bytes of a blob of `len` bytes
extern "C" int zn_envelope_parse_head(const uint8_t* blob, size_t head, size_t len, zn_envelope* e);

// Windowed decode of znippy_cuda.cu (declared in host_api.h, which needs the CUDA headers this file is built without).
extern "C" int zn_decode_windows_checked(zn_ctx* c, const uint8_t* blobs_base, const uint64_t* blob_off, const uint64_t* blob_len,
                                         const uint8_t* compressed, const uint64_t* out_len, const uint64_t* stop, uint32_t n,
                                         const uint32_t* win_row, const uint64_t* win_off, const uint64_t* win_len, uint32_t n_win,
                                         const uint32_t* ck_row, const uint64_t* ck_off, const uint64_t* ck_len,
                                         const uint32_t* ck_sum, uint32_t n_ck, uint8_t* pack, uint32_t* status, uint64_t* produced);

namespace {
struct PinnedBuf {  // pinned host buffer from the process-wide cache, returned on scope exit
  uint8_t* p = nullptr;
  ~PinnedBuf() { if (p) zn_ctx_pinned_free(p); }
};
bool pread_all(int fd, uint8_t* dst, uint64_t len, uint64_t off) {
  uint64_t done = 0;
  while (done < len) {
    const ssize_t r = pread(fd, dst + done, len - done, (off_t)(off + done));
    if (r <= 0) return false;
    done += (uint64_t)r;
  }
  return true;
}

// One frame of a seekable zstd payload (ZN_CODEC_SEEKABLE): compressed bytes [c, c + cs) of the payload decode to
// content bytes [d, d + ds) of the row, whose XXH64 has the low 32 bits `sum`.
struct SeekFrame {
  uint64_t c, d;
  uint32_t cs, ds, sum;
};
constexpr uint64_t kSeekBlock = 128u << 10;  // frame size of this library's writer (cz::kZstdCBlock)
uint32_t ld32(const uint8_t* p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24; }

// The seek table at the end of a zstd payload of plen bytes at archive offset po that decodes to ul bytes (the Zstandard
// seekable format: skippable frame 0x184D2A5E, 12-byte entries with checksums, footer {N, 0x80, 0x8F92EAB1}).  The
// writer's frame count is tried first, then the footer's.  False when the table is absent or inconsistent with the
// payload or the index: the row is then decoded from its start.
bool read_seek_table(int fd, uint64_t po, uint64_t plen, uint64_t ul, std::vector<SeekFrame>* fr, uint64_t* bytes_read) {
  uint64_t nf = ul ? (ul + kSeekBlock - 1) / kSeekBlock : 1;
  std::vector<uint8_t> t;
  for (int attempt = 0;; attempt++) {
    const uint64_t tl = 12 * nf + 17;
    if (tl > plen) return false;
    t.resize(tl);
    if (!pread_all(fd, t.data(), tl, po + plen - tl)) return false;
    *bytes_read += tl;
    const uint8_t* f = t.data() + tl - 9;
    if (ld32(f + 5) != 0x8F92EAB1u) return false;
    if (ld32(f) == nf) break;
    if (attempt == 1) return false;
    nf = ld32(f);
  }
  const uint8_t desc = t[t.size() - 5];
  if (!(desc & 0x80) || (desc & 0x7C)) return false;  // checksums present, reserved bits clear
  if (ld32(t.data()) != 0x184D2A5Eu || ld32(t.data() + 4) != 12 * nf + 9) return false;
  fr->resize(nf);
  uint64_t c = 0, d = 0;
  for (uint64_t k = 0; k < nf; k++) {
    const uint8_t* e = t.data() + 8 + 12 * k;
    (*fr)[k] = {c, d, ld32(e), ld32(e + 4), ld32(e + 8)};
    c += ld32(e);
    d += ld32(e + 4);
  }
  return c + t.size() == plen && d == ul;
}
}  // namespace

// Byte ranges (include/znippy_cuda.h): each request is cut into pieces, one per index row it overlaps; the distinct rows
// are answered from the LRU, pread in part (store-as-is rows, RAW payloads) or decoded, full rows in full and edge rows
// up to the furthest byte any piece needs (zn_decode_windows).  Pieces are written only once every row of their request
// is known to be good.
extern "C" int zn_archive_read_ranges(zn_ctx* ctx, zn_archive* a, const char* const* paths, const uint64_t* offset,
                                      const uint64_t* length, uint32_t n, uint8_t* out_base, const uint64_t* out_off,
                                      uint64_t* got, uint32_t* file_status, zn_range_stats* stats) {
  if (!ctx || !a || (n && (!paths || !offset || !length || !out_base || !out_off || !got || !file_status))) return ZN_E_ARG;
  zn_range_stats S;
  memset(&S, 0, sizeof S);
  const IndexImpl& I = a->index->ix;
  struct Piece {
    uint32_t req, row;     // row: index into `rows` below
    uint64_t s, e, dst;    // bytes [s, e) of the row go to out_base + dst
    uint64_t at;           // where the bytes wait: offset in `cached` or in the decode pack
    uint32_t unit = 0;     // decode rows: the decode unit (below) that holds the bytes
  };
  struct Row {
    uint64_t r, need = 0;  // index row; bytes [0, need) of it are needed
    int kind = 0;          // 0 decode, 1 pread (store-as-is or RAW payload), 2 cache, 3 failed before any decode
    uint64_t raw_off = 0;  // kind 1: archive offset of the row's first content byte
    uint32_t status = 0, flag = 0;
    uint64_t payload_off = 0, payload_len = 0;
  };
  std::vector<Piece> pieces;
  std::vector<Row> rows;
  std::unordered_map<uint64_t, uint32_t> row_at;
  for (uint32_t k = 0; k < n; k++) {
    got[k] = 0;
    file_status[k] = 0;
    auto it = a->files.find(paths[k]);
    if (it == a->files.end()) { file_status[k] = 1; continue; }
    const zn_archive::FileEntry& F = it->second;
    if (length[k] == 0 || offset[k] >= F.size) continue;
    const uint64_t lo = offset[k], hi = lo + std::min(length[k], F.size - lo);
    got[k] = hi - lo;
    // the last row starting at or before lo, then forward while rows start before hi
    auto rit = std::upper_bound(F.rows.begin(), F.rows.end(), lo, [&](uint64_t v, uint64_t r) { return v < I.col[2][r]; });
    if (rit != F.rows.begin()) --rit;
    for (; rit != F.rows.end() && I.col[2][*rit] < hi; ++rit) {
      const uint64_t r = *rit, fo = I.col[2][r], s = std::max(lo, fo), e = std::min(hi, fo + I.col[3][r]);
      if (s >= e) continue;
      auto ins = row_at.emplace(r, (uint32_t)rows.size());
      if (ins.second) { rows.emplace_back(); rows.back().r = r; }
      Row& R = rows[ins.first->second];
      R.need = std::max(R.need, e - fo);
      pieces.push_back({k, ins.first->second, s - fo, e - fo, out_off[k] + (s - lo), 0});
    }
  }
  // cached rows: the bytes of their pieces are copied out under the lock (a later insertion may evict the row)
  std::vector<uint8_t> cached;
  zn_archive::Cache& K = a->cache;
  if (K.budget && !rows.empty()) {
    std::lock_guard<std::mutex> g(K.mu);
    for (Row& R : rows) {
      auto c = K.at.find(R.r);
      if (c == K.at.end()) { K.misses++; continue; }
      K.lru.splice(K.lru.begin(), K.lru, c->second);
      K.hits++;
      R.kind = 2;
      S.rows_from_cache++;
    }
    for (Piece& P : pieces) {
      if (rows[P.row].kind != 2) continue;
      const std::vector<uint8_t>& v = K.at[rows[P.row].r]->second;
      P.at = cached.size();
      cached.insert(cached.end(), v.begin() + (long)P.s, v.begin() + (long)P.e);
    }
  }
  // envelopes and store-as-is rows: which rows reach a decoder, and with which payload
  static const uint8_t flag_of[5] = {0, 1, 3, 1, 2};  // ZN_PAYLOAD_* -> compressed value of a bare payload
  for (Row& R : rows) {
    if (R.kind == 2) continue;
    const uint64_t bo = I.col[0][R.r], bl = I.col[1][R.r], ul = I.col[3][R.r];
    const uint8_t ce = I.comp_eff[R.r];
    R.payload_off = 0;
    R.payload_len = bl;
    R.flag = ce;
    if (ce == 4) {
      // ZNB1 and bare frames are parsed from their first bytes; a foreign envelope, and a bare zstd blob that ends in
      // a seek table (its size is the table's sum), get the whole blob
      std::vector<uint8_t> head((size_t)std::min<uint64_t>(bl, 64));
      if (!pread_all(a->fd, head.data(), head.size(), bo)) return ZN_E_ARG;
      S.blob_bytes_read += head.size();
      uint32_t magic = 0, tail = 0;
      if (head.size() >= 4) memcpy(&magic, head.data(), 4);
      if (magic == 0xFD2FB528u && bl > head.size()) {
        uint8_t t[4];
        if (!pread_all(a->fd, t, 4, bo + bl - 4)) return ZN_E_ARG;
        S.blob_bytes_read += 4;
        tail = ld32(t);
      }
      const bool header_only = magic == 0x31424E5Au /* "ZNB1" */ || (magic == 0xFD2FB528u && tail != 0x8F92EAB1u) ||
                               magic == 0x184D2204u || (magic & 0xFFFFFFF0u) == 0x184D2A50u;
      if (!header_only && head.size() < bl) {
        head.resize(bl);
        if (!pread_all(a->fd, head.data(), bl, bo)) return ZN_E_ARG;
        S.blob_bytes_read += bl;
      }
      zn_envelope e;
      const int erc = zn_envelope_parse_head(head.data(), head.size(), bl, &e);
      if (erc != ZN_OK || (e.out_len != ~0ull && e.out_len != ul)) {
        R.kind = 3;
        R.status = erc != ZN_OK ? ZN_S_UNSUPPORTED : ZN_S_SIZE_MISMATCH;
        continue;
      }
      R.payload_off = e.payload_off;
      R.payload_len = e.payload_len;
      R.flag = flag_of[e.codec];
    }
    if (R.flag == 0) {
      if (R.payload_len != ul) { R.kind = 3; R.status = ZN_S_SIZE_MISMATCH; continue; }  // as zn_decode_verify_batch
      R.kind = 1;
      R.raw_off = bo + R.payload_off;
    }
  }
  // decode units: a decode row whole, up to its `need` (the prefix path), or, for a seekable row read in part, each run
  // of adjacent frames its pieces touch, decoded whole and checked frame by frame against the seek table
  struct Unit {
    uint32_t row;
    uint64_t rd_off, rd_len;  // archive bytes pread for the unit
    uint64_t in_off, in_len;  // decoder input: bytes [in_off, + in_len) of what was pread
    uint64_t d_off, d_len;    // content bytes [d_off, + d_len) of the row
    uint64_t stop;            // decode up to here (d_len: whole)
    bool seek = false;
  };
  std::vector<Unit> units;
  std::vector<uint32_t> ck_row, ck_sum;
  std::vector<uint64_t> ck_off, ck_len;
  std::vector<std::vector<uint32_t>> pieces_of(rows.size());
  for (uint32_t p = 0; p < (uint32_t)pieces.size(); p++) pieces_of[pieces[p].row].push_back(p);
  // the seek tables of the seekable zstd rows read in part (their pieces leave a byte uncovered), pread in parallel
  std::vector<uint32_t> seek_rows;
  for (uint32_t j = 0; I.seekable && j < (uint32_t)rows.size(); j++) {
    const Row& R = rows[j];
    if (R.kind != 0 || R.flag != 1) continue;
    std::vector<std::pair<uint64_t, uint64_t>> iv;
    for (uint32_t p : pieces_of[j]) iv.emplace_back(pieces[p].s, pieces[p].e);
    std::sort(iv.begin(), iv.end());
    uint64_t covered = 0;
    for (auto& v : iv) if (v.first <= covered) covered = std::max(covered, v.second);
    if (covered < I.col[3][R.r]) seek_rows.push_back(j);
  }
  std::vector<std::vector<SeekFrame>> tables(rows.size());
  std::vector<uint8_t> has_table(rows.size(), 0);
  {
    std::atomic<size_t> next{0};
    std::atomic<uint64_t> table_bytes{0};
    auto body = [&] {
      for (size_t k; (k = next.fetch_add(1)) < seek_rows.size();) {
        const uint32_t j = seek_rows[k];
        const Row& R = rows[j];
        uint64_t got = 0;
        has_table[j] = read_seek_table(a->fd, I.col[0][R.r] + R.payload_off, R.payload_len, I.col[3][R.r], &tables[j], &got);
        table_bytes += got;
      }
    };
    std::vector<std::thread> ts;
    for (int t = 1; t < (seek_rows.size() >= 16 ? 4 : 1); t++) ts.emplace_back(body);
    body();
    for (auto& t : ts) t.join();
    S.blob_bytes_read += table_bytes;
  }
  uint32_t rows_dec = 0;
  for (uint32_t j = 0; j < (uint32_t)rows.size(); j++) {
    Row& R = rows[j];
    if (R.kind != 0) continue;
    rows_dec++;
    const uint64_t bo = I.col[0][R.r], ul = I.col[3][R.r];
    const std::vector<SeekFrame>& fr = tables[j];
    if (!has_table[j]) {
      units.push_back({j, bo, I.col[1][R.r], R.payload_off, R.payload_len, 0, ul, R.need});
      for (uint32_t p : pieces_of[j]) pieces[p].unit = (uint32_t)units.size() - 1;
      continue;
    }
    std::vector<uint8_t> touched(fr.size(), 0);
    auto frame_of = [&](uint64_t x) {  // the frame holding content byte x
      return (size_t)(std::upper_bound(fr.begin(), fr.end(), x, [](uint64_t v, const SeekFrame& f) { return v < f.d; }) - fr.begin()) - 1;
    };
    for (uint32_t p : pieces_of[j])
      for (size_t f = frame_of(pieces[p].s); f < fr.size() && fr[f].d < pieces[p].e; f++) touched[f] = 1;
    const uint32_t first_unit = (uint32_t)units.size();
    for (size_t f = 0; f < fr.size();) {
      if (!touched[f]) { f++; continue; }
      size_t g = f;
      while (g < fr.size() && touched[g]) g++;
      const uint64_t c0 = fr[f].c, c1 = fr[g - 1].c + fr[g - 1].cs, d0 = fr[f].d, d1 = fr[g - 1].d + fr[g - 1].ds;
      const uint32_t u = (uint32_t)units.size();
      units.push_back({j, bo + R.payload_off + c0, c1 - c0, 0, c1 - c0, d0, d1 - d0, d1 - d0, true});
      for (size_t k = f; k < g; k++) {
        ck_row.push_back(u); ck_off.push_back(fr[k].d - d0); ck_len.push_back(fr[k].ds); ck_sum.push_back(fr[k].sum);
      }
      f = g;
    }
    for (uint32_t p : pieces_of[j]) {  // every piece lies inside one run: the frames it touches are adjacent
      uint32_t u = first_unit;
      while (u + 1 < units.size() && units[u + 1].d_off <= pieces[p].s) u++;
      pieces[p].unit = u;
    }
  }
  // units into pinned staging, 16 bytes apart (room for the magic of a magicless zstd payload)
  uint64_t in_cur = 0;
  for (const Unit& U : units) in_cur += 16 + ((U.rd_len + 15) & ~15ull);
  std::vector<uint8_t> full_row(units.size(), 0);  // a row decoded in full (and so a candidate for the cache)
  std::vector<uint32_t> unit_status(units.size(), 0);
  PinnedBuf pack;  // the decoded bytes of every piece of a decode row
  if (!units.empty()) {
    const uint32_t nd = (uint32_t)units.size();
    std::vector<uint64_t> bo(nd), bl(nd), ol(nd), stop(nd), prod(nd), w_off, w_len;
    std::vector<uint8_t> cf(nd);
    std::vector<uint32_t> st(nd), w_row;
    PinnedBuf stage_buf;
    uint8_t* stage = stage_buf.p = (uint8_t*)zn_ctx_pinned_alloc(in_cur + 4096);
    if (!stage) return ZN_E_NOMEM;
    std::vector<uint64_t> rd_at(nd);
    uint64_t cur = 0;
    for (uint32_t j = 0; j < nd; j++) {
      const Unit& U = units[j];
      const Row& R = rows[U.row];
      rd_at[j] = cur + 16;
      bo[j] = cur + 16 + U.in_off;
      bl[j] = U.in_len;
      cf[j] = U.seek ? 1 : (uint8_t)R.flag;
      ol[j] = U.d_len;
      stop[j] = U.stop;
      full_row[j] = !U.seek && (R.need >= ol[j] || R.flag == 2);
      cur += 16 + ((U.rd_len + 15) & ~15ull);
    }
    {
      std::atomic<size_t> next{0};
      std::atomic<int> io_err{0};
      auto body = [&] {
        for (size_t j; (j = next.fetch_add(1)) < nd;)
          if (!pread_all(a->fd, stage + rd_at[j], units[j].rd_len, units[j].rd_off)) io_err = 1;
      };
      std::vector<std::thread> ts;
      for (int t = 1; t < (nd >= 16 ? 4 : 1); t++) ts.emplace_back(body);
      body();
      for (auto& t : ts) t.join();
      if (io_err) return ZN_E_ARG;
    }
    for (uint32_t j = 0; j < nd; j++) {
      S.blob_bytes_read += units[j].rd_len;
      if (cf[j] == 3) {  // magicless zstd payload: decoded as magic + payload
        static const uint8_t magic[4] = {0x28, 0xB5, 0x2F, 0xFD};
        bo[j] -= 4;
        bl[j] += 4;
        memcpy(stage + bo[j], magic, 4);
        cf[j] = 1;
      }
    }
    // windows: one per piece, plus the whole row where a full row goes into the cache
    uint64_t packed = 0;
    for (Piece& P : pieces) {
      if (rows[P.row].kind != 0) continue;
      w_row.push_back(P.unit); w_off.push_back(P.s - units[P.unit].d_off); w_len.push_back(P.e - P.s);
      P.at = packed;
      packed += P.e - P.s;
    }
    std::vector<uint64_t> whole_at(nd, ~0ull);
    if (K.budget)
      for (uint32_t j = 0; j < nd; j++)
        if (full_row[j] && ol[j] <= K.budget) {
          w_row.push_back(j); w_off.push_back(0); w_len.push_back(ol[j]);
          whole_at[j] = packed;
          packed += ol[j];
        }
    if (!(pack.p = (uint8_t*)zn_ctx_pinned_alloc(packed + 64))) return ZN_E_NOMEM;
    const int rc = zn_decode_windows_checked(ctx, stage, bo.data(), bl.data(), cf.data(), ol.data(), stop.data(), nd, w_row.data(),
                                     w_off.data(), w_len.data(), (uint32_t)w_row.size(), ck_row.data(), ck_off.data(),
                                     ck_len.data(), ck_sum.data(), (uint32_t)ck_row.size(), pack.p, st.data(), prod.data());
    if (rc != ZN_OK) return rc;
    S.rows_decoded += rows_dec;
    for (uint32_t j = 0; j < nd; j++) {
      unit_status[j] = st[j];
      S.bytes_decoded += prod[j];
    }
    if (K.budget) {
      std::lock_guard<std::mutex> g(K.mu);
      for (uint32_t j = 0; j < nd; j++) {
        const uint64_t r = rows[units[j].row].r;
        if (whole_at[j] == ~0ull || st[j] != ZN_S_OK || K.at.count(r)) continue;
        while (K.used + ol[j] > K.budget && !K.lru.empty()) {  // evict from the cold end
          K.used -= K.lru.back().second.size();
          K.at.erase(K.lru.back().first);
          K.lru.pop_back();
          K.evictions++;
        }
        K.lru.emplace_front(r, std::vector<uint8_t>(pack.p + whole_at[j], pack.p + whole_at[j] + ol[j]));
        K.at[r] = K.lru.begin();
        K.used += ol[j];
      }
    }
  }
  // request statuses: the first failing row (or decode unit) of each request, in file order
  for (const Piece& P : pieces) {
    const Row& R = rows[P.row];
    const uint32_t status = R.kind == 0 ? unit_status[P.unit] : R.status;
    if (status != ZN_S_OK && file_status[P.req] == 0) {
      file_status[P.req] = 2u | (status << 16);
      got[P.req] = 0;
    }
  }
  // the bytes of good requests: decoded and cached pieces, and store-as-is / RAW bytes pread straight into place
  for (const Piece& P : pieces) {
    if (file_status[P.req] != 0) continue;
    const Row& R = rows[P.row];
    if (R.kind == 0) memcpy(out_base + P.dst, pack.p + P.at, P.e - P.s);
    if (R.kind == 2) memcpy(out_base + P.dst, cached.data() + P.at, P.e - P.s);
    if (R.kind == 1) {
      if (!pread_all(a->fd, out_base + P.dst, P.e - P.s, R.raw_off + P.s)) return ZN_E_ARG;
      S.blob_bytes_read += P.e - P.s;
    }
  }
  if (stats) *stats = S;
  return ZN_OK;
}
