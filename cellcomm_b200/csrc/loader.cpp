// 10x MatrixMarket (.mtx) loader -> compact-index CSR with the reference's pandas semantics.
//
// Replaces load_matrix(), src/cell_type_training.py:9-17:
//     df = pd.read_csv(file, header=None, skiprows=3, delim_whitespace=True,
//                      names=['gene', 'barcode', 'p'])
//     df = df.pivot_table(index='barcode', columns='gene', values='p', fill_value=0)
// i.e. (SURVEY.md App. A.1) skip exactly 3 lines (the dims line is ignored), rows are the
// distinct barcode ids ascending, columns the distinct gene ids ascending (absent ids are
// dropped), duplicate (gene, barcode) entries are averaged in float64, explicit zeros keep
// their row/column alive, input order is irrelevant.
//
// Host-only C++ (no CUDA): the text parse is chunked over std::threads, the CSR is built with
// a counting sort over rows and a per-row sort over columns.
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <cerrno>
#include <cmath>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <memory>
#include <ctime>
#include <string>
#include <thread>
#include <vector>

#include "../../include/cellcomm_b200.h"

namespace cc {
void set_error(const char* fmt, ...);
}

struct cc_csr {
  int64_t rows = 0, cols = 0;
  std::vector<int64_t> rowptr;
  std::vector<int32_t> colidx;
  std::vector<float> values;
  std::vector<double> values64;
  std::vector<int64_t> row_ids, col_ids;
};

namespace {

// CC_LOADER_TIMING=1: stage timings on stderr
struct StageTimer {
  bool on;
  double t0;
  static double now() {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec + 1e-9 * ts.tv_nsec;
  }
  StageTimer() : on(getenv("CC_LOADER_TIMING") != nullptr), t0(now()) {}
  void lap(const char* what) {
    if (!on) return;
    const double t = now();
    fprintf(stderr, "cc loader: %-28s %8.1f ms\n", what, (t - t0) * 1e3);
    t0 = t;
  }
};


inline bool is_space(char c) { return c == ' ' || c == '\t' || c == '\r'; }

// parse one whitespace-separated field as a number; integers take the fast path
inline bool parse_number(const char*& p, const char* end, double* out, bool* is_int, int64_t* iv) {
  while (p < end && is_space(*p)) ++p;
  if (p >= end || *p == '\n') return false;
  const char* s = p;
  bool neg = false;
  if (*p == '-' || *p == '+') {
    neg = (*p == '-');
    ++p;
  }
  int64_t v = 0;
  int digits = 0;
  while (p < end && *p >= '0' && *p <= '9') {
    v = v * 10 + (*p - '0');
    ++p;
    ++digits;
  }
  if (digits > 0 && digits <= 18 && (p >= end || is_space(*p) || *p == '\n')) {
    *iv = neg ? -v : v;
    *out = (double)*iv;
    *is_int = true;
    return true;
  }
  // general float: find the field end and use strtod on a bounded copy
  const char* q = s;
  while (q < end && !is_space(*q) && *q != '\n') ++q;
  char buf[64];
  size_t len = (size_t)(q - s);
  if (len == 0 || len >= sizeof(buf)) return false;
  memcpy(buf, s, len);
  buf[len] = 0;
  char* e = nullptr;
  errno = 0;
  double d = strtod(buf, &e);
  if (e != buf + len) return false;
  *out = d;
  *is_int = false;
  *iv = (int64_t)d;
  p = q;
  return true;
}

// parse lines in [p, end) into the caller's slices (capacity >= number of newlines + 1);
// returns the number of entries, or -1 (with the line text) on a malformed line
int64_t parse_chunk(const char* p, const char* end, int64_t* gene, int64_t* barcode, double* val,
                    std::string* err) {
  int64_t n = 0;
  while (p < end) {
    // skip blank lines (pandas skip_blank_lines=True)
    const char* ls = p;
    while (p < end && is_space(*p)) ++p;
    if (p >= end) break;
    if (*p == '\n') {
      ++p;
      continue;
    }
    double g, b, v;
    bool gi, bi, vi;
    int64_t giv, biv, viv;
    bool ok = parse_number(p, end, &g, &gi, &giv) && parse_number(p, end, &b, &bi, &biv) &&
              parse_number(p, end, &v, &vi, &viv) && gi && bi;
    if (ok) {
      while (p < end && is_space(*p)) ++p;
      ok = (p >= end || *p == '\n');
    }
    if (!ok) {
      const char* le = ls;
      while (le < end && *le != '\n') ++le;
      *err = std::string(ls, std::min<size_t>((size_t)(le - ls), 80));
      return -1;
    }
    gene[n] = giv;
    barcode[n] = biv;
    val[n] = v;
    ++n;
    if (p < end) ++p;  // newline
  }
  return n;
}

inline int64_t count_newlines(const char* p, const char* end) {
  int64_t n = 0;
  while (p < end) {
    const char* nl = (const char*)memchr(p, '\n', (size_t)(end - p));
    if (!nl) break;
    ++n;
    p = nl + 1;
  }
  return n;
}

template <typename F>
void parallel_ranges(int64_t n, unsigned nt, F f) {
  if (nt <= 1 || n < 2) {
    f(0, n, 0u);
    return;
  }
  std::vector<std::thread> th;
  for (unsigned t = 0; t < nt; ++t) {
    const int64_t lo = n * t / nt, hi = n * (t + 1) / nt;
    th.emplace_back([=] { f(lo, hi, t); });
  }
  for (auto& x : th) x.join();
}

unsigned worker_threads() {
  unsigned nt = std::thread::hardware_concurrency();
  if (nt == 0) nt = 4;
  if (nt > 32) nt = 32;
  return nt;
}

// ids -> (sorted distinct ids, compact index of every element)
void compact_ids(const int64_t* ids, int64_t n, std::vector<int64_t>* distinct,
                 std::vector<int32_t>* index) {
  index->resize((size_t)n);
  distinct->clear();
  if (n == 0) return;
  int64_t lo = ids[0], hi = ids[0];
  for (int64_t i = 1; i < n; ++i) {
    lo = std::min(lo, ids[i]);
    hi = std::max(hi, ids[i]);
  }
  const int64_t range = hi - lo + 1;
  if (range <= std::max<int64_t>(4 * n, 1 << 20)) {
    const unsigned nt = n > (1 << 18) ? worker_threads() : 1;
    std::vector<int32_t> lut((size_t)range, -1);
    // (threads may mark the same id: every writer stores the same value)
    parallel_ranges(n, nt, [&](int64_t a, int64_t b, unsigned) {
      for (int64_t i = a; i < b; ++i) lut[(size_t)(ids[i] - lo)] = 0;
    });
    int32_t next = 0;
    for (int64_t k = 0; k < range; ++k)
      if (lut[(size_t)k] == 0) {
        lut[(size_t)k] = next++;
        distinct->push_back(lo + k);
      }
    parallel_ranges(n, nt, [&](int64_t a, int64_t b, unsigned) {
      for (int64_t i = a; i < b; ++i) (*index)[(size_t)i] = lut[(size_t)(ids[i] - lo)];
    });
  } else {
    std::vector<int64_t> s(ids, ids + n);
    std::sort(s.begin(), s.end());
    s.erase(std::unique(s.begin(), s.end()), s.end());
    *distinct = s;
    for (int64_t i = 0; i < n; ++i)
      (*index)[(size_t)i] =
          (int32_t)(std::lower_bound(s.begin(), s.end(), ids[i]) - s.begin());
  }
}

int build_csr(const int64_t* gene, const int64_t* barcode, const double* val, int64_t nnz,
              cc_csr** out) {
  cc_csr* c = new cc_csr();
  StageTimer tm;
  std::vector<int32_t> ri, ci;
  compact_ids(barcode, nnz, &c->row_ids, &ri);
  compact_ids(gene, nnz, &c->col_ids, &ci);
  tm.lap("compact ids");
  c->rows = (int64_t)c->row_ids.size();
  c->cols = (int64_t)c->col_ids.size();
  struct Ent {
    int32_t col;
    double v;
  };
  std::vector<int64_t> start((size_t)c->rows + 1, 0);
  std::unique_ptr<Ent[]> ents_mem(new Ent[(size_t)nnz > 0 ? (size_t)nnz : 1]);  // uninitialised
  Ent* const ents = ents_mem.get();
  // 10x files are barcode-major: when the compact row index never decreases the entries are
  // already grouped by row in file order and only need copying (in parallel); otherwise a
  // counting sort by row (stable: duplicates keep file order)
  bool grouped = true;
  for (int64_t i = 1; i < nnz; ++i)
    if (ri[(size_t)i] < ri[(size_t)i - 1]) {
      grouped = false;
      break;
    }
  for (int64_t i = 0; i < nnz; ++i) ++start[(size_t)ri[(size_t)i] + 1];
  for (int64_t r = 0; r < c->rows; ++r) start[(size_t)r + 1] += start[(size_t)r];
  if (grouped) {
    parallel_ranges(nnz, nnz > (1 << 18) ? worker_threads() : 1, [&](int64_t a, int64_t b, unsigned) {
      for (int64_t i = a; i < b; ++i) ents[(size_t)i] = Ent{ci[(size_t)i], val[(size_t)i]};
    });
  } else {
    std::vector<int64_t> pos(start.begin(), start.end() - 1);
    for (int64_t i = 0; i < nnz; ++i) {
      int64_t& p = pos[(size_t)ri[(size_t)i]];
      ents[(size_t)p++] = Ent{ci[(size_t)i], val[(size_t)i]};
    }
  }
  tm.lap(grouped ? "group by row (already grouped)" : "counting sort by row");
  // per-row: sort by column (stable, so duplicates keep file order), average duplicates.
  // Rows are independent: pass A sorts (skipped when the row is already strictly ascending, the
  // normal case of a 10x file) and counts the distinct columns, pass B writes the CSR arrays.
  const unsigned nt = nnz > (1 << 16) ? worker_threads() : 1;
  c->rowptr.assign((size_t)c->rows + 1, 0);
  parallel_ranges(c->rows, nt, [&](int64_t r0, int64_t r1, unsigned) {
    for (int64_t r = r0; r < r1; ++r) {
      Ent* b = ents + start[(size_t)r];
      Ent* e = ents + start[(size_t)r + 1];
      bool ascending = true;
      for (Ent* q = b + 1; q < e; ++q)
        if (q->col <= (q - 1)->col) {
          ascending = false;
          break;
        }
      int64_t distinct = e - b;
      if (!ascending) {
        std::stable_sort(b, e, [](const Ent& x, const Ent& y) { return x.col < y.col; });
        distinct = (e > b) ? 1 : 0;
        for (Ent* q = b + 1; q < e; ++q) distinct += (q->col != (q - 1)->col);
      }
      c->rowptr[(size_t)r + 1] = distinct;
    }
  });
  for (int64_t r = 0; r < c->rows; ++r) c->rowptr[(size_t)r + 1] += c->rowptr[(size_t)r];
  const size_t out_nnz = (size_t)c->rowptr[(size_t)c->rows];
  c->colidx.resize(out_nnz);
  c->values64.resize(out_nnz);
  c->values.resize(out_nnz);
  parallel_ranges(c->rows, nt, [&](int64_t r0, int64_t r1, unsigned) {
    for (int64_t r = r0; r < r1; ++r) {
      const Ent* e = ents + start[(size_t)r + 1];
      size_t o = (size_t)c->rowptr[(size_t)r];
      for (const Ent* q = ents + start[(size_t)r]; q < e;) {
        const Ent* g = q;
        double sum = 0.0;
        int64_t cnt = 0;
        while (g < e && g->col == q->col) {
          sum += g->v;
          ++cnt;
          ++g;
        }
        const double v = cnt == 1 ? sum : sum / (double)cnt;
        c->colidx[o] = q->col;
        c->values64[o] = v;
        c->values[o] = (float)v;
        ++o;
        q = g;
      }
    }
  });
  tm.lap("row sort + dedup (threads)");
  *out = c;
  return 0;
}

}  // namespace

extern "C" int cc_coo_to_csr(const int64_t* gene, const int64_t* barcode, const double* val,
                             int64_t nnz, cc_csr** out) {
  if (out == nullptr || nnz < 0) {
    cc::set_error("cc_coo_to_csr: bad arguments");
    return -1;
  }
  return build_csr(gene, barcode, val, nnz, out);
}

// The file's triplets in FILE ORDER (1-based ids as written), parsed by all host threads.
struct Triplets {
  std::unique_ptr<int64_t[]> gene, barcode;
  std::unique_ptr<double[]> val;
  int64_t nnz = 0;
};

static int parse_mtx_file(const char* path, Triplets* t_out, StageTimer& tm) {
  int fd = open(path, O_RDONLY);
  if (fd < 0) {
    cc::set_error("cc_mtx_load: cannot open %s: %s", path, strerror(errno));
    return -1;
  }
  struct stat sb;
  if (fstat(fd, &sb) != 0) {
    close(fd);
    cc::set_error("cc_mtx_load: fstat failed on %s", path);
    return -1;
  }
  const size_t size = (size_t)sb.st_size;
  const char* data = nullptr;
  if (size > 0) {
    data = (const char*)mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0);
    if (data == MAP_FAILED) {
      close(fd);
      cc::set_error("cc_mtx_load: mmap failed on %s", path);
      return -1;
    }
  }
  // skip exactly 3 lines (skiprows=3): banner, comment, dims
  const char* p = data;
  const char* end = data + size;
  for (int l = 0; l < 3 && p < end; ++l) {
    const char* nl = (const char*)memchr(p, '\n', (size_t)(end - p));
    p = nl ? nl + 1 : end;
  }
  // chunk the body at line boundaries
  unsigned nt = worker_threads();
  const size_t body = (size_t)(end - p);
  if (body < (1u << 20)) nt = 1;
  std::vector<const char*> cut(nt + 1);
  cut[0] = p;
  cut[nt] = end;
  for (unsigned t = 1; t < nt; ++t) {
    const char* q = p + body / nt * t;
    if (q < cut[t - 1]) q = cut[t - 1];
    const char* nl = (const char*)memchr(q, '\n', (size_t)(end - q));
    cut[t] = nl ? nl + 1 : end;
  }
  // pass 1: an upper bound of every chunk's entry count (newlines + 1) gives each thread its
  // slice of the triplet arrays; pass 2 parses straight into the slices (no per-thread vectors,
  // no concatenation)
  std::vector<int64_t> cap(nt, 0), off(nt + 1, 0), got(nt, 0);
  {
    std::vector<std::thread> threads;
    for (unsigned t = 0; t < nt; ++t)
      threads.emplace_back([&, t] { cap[t] = count_newlines(cut[t], cut[t + 1]) + 1; });
    for (auto& th : threads) th.join();
  }
  for (unsigned t = 0; t < nt; ++t) off[t + 1] = off[t] + cap[t];
  // (uninitialised: every used element is written by the parser)
  const size_t cap_total = (size_t)off[nt] > 0 ? (size_t)off[nt] : 1;
  std::unique_ptr<int64_t[]> gene_mem(new int64_t[cap_total]), barcode_mem(new int64_t[cap_total]);
  std::unique_ptr<double[]> val_mem(new double[cap_total]);
  int64_t* const gene = gene_mem.get();
  int64_t* const barcode = barcode_mem.get();
  double* const val = val_mem.get();
  std::vector<std::string> errs(nt);
  {
    std::vector<std::thread> threads;
    for (unsigned t = 0; t < nt; ++t)
      threads.emplace_back([&, t] {
        got[t] = parse_chunk(cut[t], cut[t + 1], gene + off[t], barcode + off[t],
                             val + off[t], &errs[t]);
      });
    for (auto& th : threads) th.join();
  }
  tm.lap("count + parse (threads)");
  if (data) munmap((void*)data, size);
  close(fd);
  for (unsigned t = 0; t < nt; ++t)
    if (got[t] < 0) {
      cc::set_error("cc_mtx_load: malformed line in %s: '%s'", path, errs[t].c_str());
      return -1;
    }
  // close the gaps blank lines / the +1 left between the slices (normally a few elements)
  int64_t nnz = got[0];
  for (unsigned t = 1; t < nt; ++t) {
    if (off[t] != nnz && got[t] > 0) {
      memmove(gene + nnz, gene + off[t], (size_t)got[t] * sizeof(int64_t));
      memmove(barcode + nnz, barcode + off[t], (size_t)got[t] * sizeof(int64_t));
      memmove(val + nnz, val + off[t], (size_t)got[t] * sizeof(double));
    }
    nnz += got[t];
  }
  tm.lap("close gaps");
  t_out->gene = std::move(gene_mem);
  t_out->barcode = std::move(barcode_mem);
  t_out->val = std::move(val_mem);
  t_out->nnz = nnz;
  return 0;
}

extern "C" int cc_mtx_load_csr(const char* path, cc_csr** out) {
  if (path == nullptr || out == nullptr) {
    cc::set_error("cc_mtx_load_csr: bad arguments");
    return -1;
  }
  StageTimer tm;
  Triplets t;
  if (int rc = parse_mtx_file(path, &t, tm)) return rc;
  return build_csr(t.gene.get(), t.barcode.get(), t.val.get(), t.nnz, out);
}

// ---- triplets in file order (the cells / genes importer groups on first appearance) ----
struct cc_coo {
  Triplets t;
};

extern "C" int cc_mtx_load_coo(const char* path, cc_coo** out) {
  if (path == nullptr || out == nullptr) {
    cc::set_error("cc_mtx_load_coo: bad arguments");
    return -1;
  }
  StageTimer tm;
  std::unique_ptr<cc_coo> c(new cc_coo);
  if (int rc = parse_mtx_file(path, &c->t, tm)) return rc;
  *out = c.release();
  return 0;
}
extern "C" void cc_coo_destroy(cc_coo* coo) { delete coo; }
extern "C" int64_t cc_coo_nnz(const cc_coo* c) { return c->t.nnz; }
extern "C" const int64_t* cc_coo_gene(const cc_coo* c) { return c->t.gene.get(); }
extern "C" const int64_t* cc_coo_barcode(const cc_coo* c) { return c->t.barcode.get(); }
extern "C" const double* cc_coo_value(const cc_coo* c) { return c->t.val.get(); }
extern "C" int cc_coo_build_csr(const cc_coo* c, cc_csr** out) {
  if (c == nullptr || out == nullptr) {
    cc::set_error("cc_coo_build_csr: bad arguments");
    return -1;
  }
  return build_csr(c->t.gene.get(), c->t.barcode.get(), c->t.val.get(), c->t.nnz, out);
}

// ---- writer: host CSR -> 10x .mtx (the loader's counterpart) ----
namespace {

// integer-valued and printable as int64 (NaN / inf / |v| >= 2^63 are not)
inline bool int_valued(double v) { return v == std::nearbyint(v) && std::fabs(v) < 9.2e18; }

// decimal digits of a signed integer; returns the end of the text
inline char* put_int(char* p, int64_t v) {
  uint64_t u = v < 0 ? (uint64_t)0 - (uint64_t)v : (uint64_t)v;
  if (v < 0) *p++ = '-';
  char tmp[24];
  int n = 0;
  do {
    tmp[n++] = (char)('0' + u % 10);
    u /= 10;
  } while (u);
  while (n) *p++ = tmp[--n];
  return p;
}

// one "gene barcode value\n" line: at most 20 + 1 + 20 + 1 + 25 + 1 bytes
constexpr size_t kMaxLine = 72;

}  // namespace

extern "C" int cc_mtx_write(const char* path, int64_t rows, int64_t cols, int64_t nnz,
                            const int64_t* rowptr, const int32_t* colidx, const double* values,
                            const int64_t* row_ids, const int64_t* col_ids) {
  if (path == nullptr || rows < 0 || cols < 0 || nnz < 0 || rowptr == nullptr ||
      (rows > 0 && row_ids == nullptr) || (cols > 0 && col_ids == nullptr) ||
      (nnz > 0 && (colidx == nullptr || values == nullptr))) {
    cc::set_error("cc_mtx_write: bad arguments");
    return -1;
  }
  if (rowptr[0] != 0 || rowptr[rows] != nnz) {
    cc::set_error("cc_mtx_write: rowptr runs from %lld to %lld, expected 0 to nnz = %lld",
                  (long long)rowptr[0], (long long)rowptr[rows], (long long)nnz);
    return -1;
  }
  for (int64_t r = 0; r < rows; ++r)
    if (rowptr[r + 1] < rowptr[r]) {
      cc::set_error("cc_mtx_write: rowptr decreases at row %lld", (long long)r);
      return -1;
    }
  const unsigned nt = nnz > (1 << 16) ? worker_threads() : 1;
  std::vector<char> bad(nt, 0), real(nt, 0);
  parallel_ranges(nnz, nt, [&](int64_t a, int64_t b, unsigned t) {
    for (int64_t e = a; e < b; ++e) {
      if (colidx[e] < 0 || colidx[e] >= cols) bad[t] = 1;
      if (!int_valued(values[e])) real[t] = 1;
    }
  });
  for (unsigned t = 0; t < nt; ++t)
    if (bad[t]) {
      cc::set_error("cc_mtx_write: a column index lies outside [0, %lld)", (long long)cols);
      return -1;
    }
  const bool is_real = std::find(real.begin(), real.end(), 1) != real.end();

  FILE* f = fopen(path, "wb");
  if (f == nullptr) {
    cc::set_error("cc_mtx_write: cannot open %s: %s", path, strerror(errno));
    return -1;
  }
  bool ok = fprintf(f, "%%%%MatrixMarket matrix coordinate %s general\n%%\n%lld %lld %lld\n",
                    is_real ? "real" : "integer", (long long)cols, (long long)rows,
                    (long long)nnz) > 0;
  // blocks of entries: the threads format their slices of a block in parallel, then the
  // slices are written in order (bounded memory, file order = CSR order)
  const int64_t kBlock = 1 << 20;
  std::vector<std::vector<char>> text(nt, std::vector<char>());
  std::vector<size_t> used(nt, 0);
  for (int64_t e0 = 0; ok && e0 < nnz; e0 += kBlock) {
    const int64_t e1 = std::min(nnz, e0 + kBlock);
    parallel_ranges(e1 - e0, nt, [&](int64_t a, int64_t b, unsigned t) {
      a += e0;
      b += e0;
      std::vector<char>& buf = text[t];
      if (buf.size() < (size_t)(b - a) * kMaxLine) buf.resize((size_t)(b - a) * kMaxLine);
      char* p = buf.data();
      // the row of entry a: last r with rowptr[r] <= a (rows may be empty)
      int64_t r = (int64_t)(std::upper_bound(rowptr, rowptr + rows + 1, a) - rowptr) - 1;
      for (int64_t e = a; e < b; ++e) {
        while (rowptr[r + 1] <= e) ++r;
        p = put_int(p, col_ids[colidx[e]]);
        *p++ = ' ';
        p = put_int(p, row_ids[r]);
        *p++ = ' ';
        const double v = values[e];
        if (int_valued(v))
          p = put_int(p, (int64_t)v);
        else
          p += snprintf(p, 32, "%.17g", v);
        *p++ = '\n';
      }
      used[t] = (size_t)(p - buf.data());
    });
    const unsigned parts = (e1 - e0) >= 2 ? nt : 1;   // parallel_ranges' own split
    for (unsigned t = 0; ok && t < parts; ++t)
      ok = fwrite(text[t].data(), 1, used[t], f) == used[t];
  }
  if (fclose(f) != 0) ok = false;
  if (!ok) {
    cc::set_error("cc_mtx_write: writing %s failed: %s", path, strerror(errno));
    return -1;
  }
  return 0;
}

extern "C" void cc_csr_destroy(cc_csr* csr) { delete csr; }
extern "C" int64_t cc_csr_rows(const cc_csr* c) { return c->rows; }
extern "C" int64_t cc_csr_cols(const cc_csr* c) { return c->cols; }
extern "C" int64_t cc_csr_nnz(const cc_csr* c) { return (int64_t)c->colidx.size(); }
extern "C" const int64_t* cc_csr_rowptr(const cc_csr* c) { return c->rowptr.data(); }
extern "C" const int32_t* cc_csr_colidx(const cc_csr* c) { return c->colidx.data(); }
extern "C" const float* cc_csr_values(const cc_csr* c) { return c->values.data(); }
extern "C" const double* cc_csr_values64(const cc_csr* c) { return c->values64.data(); }
extern "C" const int64_t* cc_csr_row_ids(const cc_csr* c) { return c->row_ids.data(); }
extern "C" const int64_t* cc_csr_col_ids(const cc_csr* c) { return c->col_ids.data(); }
