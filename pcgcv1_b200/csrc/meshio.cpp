// Host mesh reader of libpcgc_b200.so: OBJ, OFF and PLY (ascii / binary_little_endian) triangle meshes for the training-set
// generator (pcgcv1_b200/dataset.py).  Every polygon becomes the fan (v0, v_i, v_{i+1}) in file order.  Contract in
// include/pcgc_b200.h (pcgc_mesh_parse).
#include <stdint.h>
#include <string.h>

#include <charconv>
#include <string>
#include <vector>

#include "../../include/pcgc_b200.h"

namespace {

struct ParseError {
  int code;
};
[[noreturn]] void corrupt() { throw ParseError{PCGC_ERR_CORRUPT}; }

inline bool is_ws(char c) { return c == ' ' || c == '\t' || c == '\r' || c == '\v' || c == '\f'; }

// Whitespace-separated tokens of one line [p, e) (no '\n' inside).
struct Line {
  const char* p;
  const char* e;
  bool next(const char** b, const char** t) {
    while (p < e && is_ws(*p)) ++p;
    if (p == e) return false;
    *b = p;
    while (p < e && !is_ws(*p)) ++p;
    *t = p;
    return true;
  }
};

// Splits [data, data + n) into lines; next() returns false at the end.
struct Lines {
  const char* p;
  const char* end;
  bool next(Line* l) {
    if (p >= end) return false;
    const char* q = (const char*)memchr(p, '\n', (size_t)(end - p));
    const char* le = q ? q : end;
    *l = Line{p, le};
    p = q ? q + 1 : end;
    return true;
  }
};

double to_double(const char* b, const char* e) {
  if (b < e && *b == '+') ++b;
  double v = 0.0;
  const auto r = std::from_chars(b, e, v);
  if (r.ec != std::errc() || r.ptr != e) corrupt();
  return v;
}

int64_t to_int(const char* b, const char* e) {
  if (b < e && *b == '+') ++b;
  int64_t v = 0;
  const auto r = std::from_chars(b, e, v);
  if (r.ec != std::errc() || r.ptr != e) corrupt();
  return v;
}

bool token_is(const char* b, const char* e, const char* s) {
  const size_t n = strlen(s);
  return (size_t)(e - b) == n && memcmp(b, s, n) == 0;
}

struct Mesh {
  std::vector<double> v;     // [nv*3]
  std::vector<int32_t> t;    // [nt*3]
  int64_t nv() const { return (int64_t)v.size() / 3; }
  void fan(const std::vector<int64_t>& poly) {
    if (poly.size() < 3) corrupt();
    for (size_t i = 1; i + 1 < poly.size(); ++i) {
      t.push_back((int32_t)poly[0]); t.push_back((int32_t)poly[i]); t.push_back((int32_t)poly[i + 1]);
    }
  }
  void check_indices() const {
    const int64_t n = nv();
    for (int32_t i : t)
      if (i < 0 || i >= n) corrupt();
  }
};

// ---- OBJ -------------------------------------------------------------------------------------------------------------------
void parse_obj(const char* data, int64_t nbytes, Mesh& m) {
  Lines lines{data, data + nbytes};
  Line l;
  std::vector<int64_t> poly;
  while (lines.next(&l)) {
    const char *b, *e;
    if (!l.next(&b, &e) || *b == '#') continue;
    if (token_is(b, e, "v")) {
      for (int k = 0; k < 3; ++k) {
        if (!l.next(&b, &e)) corrupt();
        m.v.push_back(to_double(b, e));
      }
    } else if (token_is(b, e, "f")) {
      poly.clear();
      const int64_t nv = m.nv();
      while (l.next(&b, &e)) {
        const char* s = (const char*)memchr(b, '/', (size_t)(e - b));
        int64_t i = to_int(b, s ? s : e);
        if (i == 0) corrupt();
        i = i > 0 ? i - 1 : nv + i;      // negative: relative to the vertices read so far
        if (i < 0 || i > INT32_MAX) corrupt();
        poly.push_back(i);
      }
      m.fan(poly);
    } else if (!(token_is(b, e, "vt") || token_is(b, e, "vn") || token_is(b, e, "g") || token_is(b, e, "o") ||
                 token_is(b, e, "s") || token_is(b, e, "usemtl") || token_is(b, e, "mtllib") || token_is(b, e, "l") ||
                 token_is(b, e, "p"))) {
      corrupt();
    }
  }
  m.check_indices();
}

// ---- OFF -------------------------------------------------------------------------------------------------------------------
// Next line with a token, '#' comments stripped.
bool off_line(Lines& lines, Line* l) {
  while (lines.next(l)) {
    const char* h = (const char*)memchr(l->p, '#', (size_t)(l->e - l->p));
    if (h) l->e = h;
    Line probe = *l;
    const char *b, *e;
    if (probe.next(&b, &e)) return true;
  }
  return false;
}

void parse_off(const char* data, int64_t nbytes, Mesh& m) {
  Lines lines{data, data + nbytes};
  Line l;
  const char *b, *e;
  if (!off_line(lines, &l) || !l.next(&b, &e)) corrupt();
  // "OFF" / "COFF", possibly with the counts glued on ("OFF490 518 0")
  const char* hdr = (size_t)(e - b) >= 4 && memcmp(b, "COFF", 4) == 0 ? b + 4 : (size_t)(e - b) >= 3 && memcmp(b, "OFF", 3) == 0 ? b + 3 : nullptr;
  if (!hdr) corrupt();
  Line counts{hdr, l.e};
  if (!Line(counts).next(&b, &e)) {
    if (!off_line(lines, &counts)) corrupt();
  }
  int64_t c[2];
  for (int k = 0; k < 2; ++k) {
    if (!counts.next(&b, &e)) corrupt();
    c[k] = to_int(b, e);
  }
  if (c[0] < 0 || c[1] < 0 || c[0] > INT32_MAX) corrupt();
  m.v.reserve((size_t)c[0] * 3);
  for (int64_t i = 0; i < c[0]; ++i) {
    if (!off_line(lines, &l)) corrupt();
    for (int k = 0; k < 3; ++k) {
      if (!l.next(&b, &e)) corrupt();
      m.v.push_back(to_double(b, e));
    }
  }
  std::vector<int64_t> poly;
  for (int64_t f = 0; f < c[1]; ++f) {
    if (!off_line(lines, &l) || !l.next(&b, &e)) corrupt();
    const int64_t n = to_int(b, e);
    if (n < 0) corrupt();
    poly.clear();
    for (int64_t k = 0; k < n; ++k) {
      if (!l.next(&b, &e)) corrupt();
      const int64_t i = to_int(b, e);
      if (i < 0 || i >= c[0]) corrupt();
      poly.push_back(i);
    }
    m.fan(poly);                          // colour values after the indices are ignored
  }
}

// ---- PLY -------------------------------------------------------------------------------------------------------------------
enum Scalar { S_I8, S_U8, S_I16, S_U16, S_I32, S_U32, S_F32, S_F64 };

Scalar scalar_of(const char* b, const char* e) {
  static const struct { const char* name; Scalar s; } kTypes[] = {
      {"char", S_I8},   {"int8", S_I8},    {"uchar", S_U8}, {"uint8", S_U8},     {"short", S_I16},  {"int16", S_I16},
      {"ushort", S_U16}, {"uint16", S_U16}, {"int", S_I32},  {"int32", S_I32},    {"uint", S_U32},   {"uint32", S_U32},
      {"float", S_F32}, {"float32", S_F32}, {"double", S_F64}, {"float64", S_F64}};
  for (const auto& t : kTypes)
    if (token_is(b, e, t.name)) return t.s;
  corrupt();
}

int size_of(Scalar s) { return s == S_I8 || s == S_U8 ? 1 : s == S_I16 || s == S_U16 ? 2 : s == S_F64 ? 8 : 4; }

struct Property {
  bool list = false;
  Scalar count, type;
  std::string name;
};

struct Element {
  std::string name;
  int64_t n;
  std::vector<Property> props;
};

// Reads the body values one by one, from ASCII tokens or from little-endian binary.
struct Body {
  bool binary;
  const char* p;
  const char* end;
  Lines lines{nullptr, nullptr};
  Line line{nullptr, nullptr};

  double value(Scalar s) {
    if (!binary) {
      const char *b, *e;
      while (!line.next(&b, &e))
        if (!lines.next(&line)) corrupt();
      return s == S_F32 || s == S_F64 ? to_double(b, e) : (double)to_int(b, e);
    }
    const int n = size_of(s);
    if (end - p < n) corrupt();
    double v = 0.0;
    switch (s) {
      case S_I8: { int8_t x; memcpy(&x, p, 1); v = x; break; }
      case S_U8: { uint8_t x; memcpy(&x, p, 1); v = x; break; }
      case S_I16: { int16_t x; memcpy(&x, p, 2); v = x; break; }
      case S_U16: { uint16_t x; memcpy(&x, p, 2); v = x; break; }
      case S_I32: { int32_t x; memcpy(&x, p, 4); v = x; break; }
      case S_U32: { uint32_t x; memcpy(&x, p, 4); v = x; break; }
      case S_F32: { float x; memcpy(&x, p, 4); v = x; break; }
      case S_F64: { memcpy(&v, p, 8); break; }
    }
    p += n;
    return v;
  }
};

int64_t as_index(double v) {
  if (!(v >= 0.0 && v <= (double)INT32_MAX) || v != (double)(int64_t)v) corrupt();
  return (int64_t)v;
}

int parse_ply(const char* data, int64_t nbytes, Mesh& m) {
  Lines lines{data, data + nbytes};
  Line l;
  const char *b, *e;
  if (!lines.next(&l) || !l.next(&b, &e) || !token_is(b, e, "ply")) corrupt();
  int fmt = -1;       // 0 ascii, 1 binary_little_endian
  std::vector<Element> elems;
  bool ended = false;
  while (!ended && lines.next(&l)) {
    if (!l.next(&b, &e)) continue;
    if (token_is(b, e, "format")) {
      if (!l.next(&b, &e)) corrupt();
      if (token_is(b, e, "ascii")) fmt = 0;
      else if (token_is(b, e, "binary_little_endian")) fmt = 1;
      else return PCGC_ERR_BAD_ARG;                      // binary_big_endian or unknown: not supported
      if (!l.next(&b, &e) || !token_is(b, e, "1.0")) return PCGC_ERR_BAD_ARG;
    } else if (token_is(b, e, "element")) {
      Element el;
      if (!l.next(&b, &e)) corrupt();
      el.name.assign(b, e);
      if (!l.next(&b, &e)) corrupt();
      el.n = to_int(b, e);
      if (el.n < 0) corrupt();
      elems.push_back(el);
    } else if (token_is(b, e, "property")) {
      if (elems.empty() || !l.next(&b, &e)) corrupt();
      Property pr;
      if (token_is(b, e, "list")) {
        pr.list = true;
        if (!l.next(&b, &e)) corrupt();
        pr.count = scalar_of(b, e);
        if (pr.count == S_F32 || pr.count == S_F64) corrupt();
        if (!l.next(&b, &e)) corrupt();
      }
      pr.type = scalar_of(b, e);
      if (!l.next(&b, &e)) corrupt();
      pr.name.assign(b, e);
      elems.back().props.push_back(pr);
    } else if (token_is(b, e, "end_header")) {
      ended = true;
    } else if (!(token_is(b, e, "comment") || token_is(b, e, "obj_info"))) {
      corrupt();
    }
  }
  if (!ended || fmt < 0) corrupt();
  Body body{fmt == 1, lines.p, data + nbytes};
  if (!body.binary) body.lines = Lines{lines.p, data + nbytes};
  bool have_v = false, have_f = false;
  std::vector<int64_t> poly;
  for (const Element& el : elems) {
    const bool is_v = el.name == "vertex", is_f = el.name == "face";
    int xyz[3] = {-1, -1, -1}, idx = -1;
    for (size_t k = 0; k < el.props.size(); ++k) {
      const Property& pr = el.props[k];
      if (is_v && !pr.list)
        for (int d = 0; d < 3; ++d)
          if (pr.name == std::string(1, (char)('x' + d))) xyz[d] = (int)k;
      if (is_f && pr.list && (pr.name == "vertex_indices" || pr.name == "vertex_index")) idx = (int)k;
      if (body.binary && pr.list && !is_v && !is_f) corrupt();       // other elements are skipped by size: scalar properties only
    }
    if (is_v) {
      if (xyz[0] < 0 || xyz[1] < 0 || xyz[2] < 0 || el.n > INT32_MAX) corrupt();
      m.v.reserve((size_t)el.n * 3);
      have_v = true;
    }
    if (is_f) {
      if (idx < 0) corrupt();
      have_f = true;
    }
    if (!is_v && !is_f && body.binary) {                            // skip the whole element at once
      int64_t row = 0;
      for (const Property& pr : el.props) row += size_of(pr.type);
      if (el.n > 0 && (body.end - body.p) / el.n < row) corrupt();
      body.p += el.n * row;
      continue;
    }
    for (int64_t i = 0; i < el.n; ++i) {
      double xv[3] = {0.0, 0.0, 0.0};
      for (size_t k = 0; k < el.props.size(); ++k) {
        const Property& pr = el.props[k];
        if (!pr.list) {
          const double v = body.value(pr.type);
          for (int d = 0; d < 3; ++d)
            if ((int)k == xyz[d]) xv[d] = v;
          continue;
        }
        const int64_t n = as_index(body.value(pr.count));
        if ((int)k == idx && is_f) poly.clear();
        for (int64_t j = 0; j < n; ++j) {
          const double v = body.value(pr.type);
          if ((int)k == idx && is_f) poly.push_back(as_index(v));
        }
        if ((int)k == idx && is_f) m.fan(poly);
      }
      if (is_v) for (int d = 0; d < 3; ++d) m.v.push_back(xv[d]);
    }
  }
  if (!have_v || !have_f) corrupt();
  m.check_indices();
  return PCGC_OK;
}

}  // namespace

extern "C" {

int pcgc_mesh_parse(const char* data, int64_t nbytes, int format, double* verts, int64_t vcap, int32_t* tris, int64_t tcap, int64_t* nv,
                    int64_t* nt) {
  if ((!data && nbytes) || nbytes < 0 || !nv || !nt || vcap < 0 || tcap < 0 || (!verts && vcap) || (!tris && tcap)) return PCGC_ERR_BAD_ARG;
  if (format != PCGC_MESH_OBJ && format != PCGC_MESH_OFF && format != PCGC_MESH_PLY) return PCGC_ERR_BAD_ARG;
  Mesh m;
  try {
    int rc = PCGC_OK;
    if (format == PCGC_MESH_OBJ) parse_obj(data, nbytes, m);
    else if (format == PCGC_MESH_OFF) parse_off(data, nbytes, m);
    else rc = parse_ply(data, nbytes, m);
    if (rc != PCGC_OK) return rc;
  } catch (const ParseError& err) {
    return err.code;
  } catch (const std::bad_alloc&) {
    return PCGC_ERR_OOM;
  }
  *nv = m.nv();
  *nt = (int64_t)m.t.size() / 3;
  if (*nv > vcap || *nt > tcap) return PCGC_ERR_OVERFLOW;
  if (!m.v.empty()) memcpy(verts, m.v.data(), m.v.size() * sizeof(double));
  if (!m.t.empty()) memcpy(tris, m.t.data(), m.t.size() * sizeof(int32_t));
  return PCGC_OK;
}

}  // extern "C"
