// grimb_text.cpp -- host-side text pipeline of libgrimb200.so (see include/grimb200.h, "Text
// pipeline").  Multi-threaded C++: line split, GL-string tokenising, race -> prior matrices,
// and the six output texts with Python's str(float) layout.  Behaviour mirrors, line for line,
// grim/imputation/impute.py:_process/_encode_gl/_prior_matrix/_format_subject of this package,
// which in turn follow the reference (nmdp-bioinformatics/py-graph-imputation,
// grim/imputation/impute.py:24-118,246-272,1844-1975,1985-2155).  No CUDA calls in this file
// except through grimb_impute_host.
#include <algorithm>
#include <cerrno>
#include <charconv>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <string>
#include <string_view>
#include <thread>
#include <unordered_map>
#include <vector>
#include <unistd.h>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif

#include "../../include/grimb200.h"

extern "C" void* grimb_pinned_alloc(size_t bytes);  // grimb200.cu: cudaMallocHost or nullptr
extern "C" void grimb_pinned_free(void* p);
extern "C" void grimb_set_error(const char* msg);   // grimb200.cu: the message grimb_last_error() returns
extern "C" const char* grimb_last_error(void);

namespace {

using sv = std::string_view;

// Append-only byte buffer of the formatter.  The six outputs are built from some 40 short pieces per row;
// std::string pays a capacity check, a memcpy call and a terminator store for each.  Here the capacity check is
// one compare against a slack the buffer always keeps, and pieces up to 16 bytes (allele names, ids, digits) are
// copied with two overlapping word moves.
struct OutStr {
  char* p = nullptr;
  size_t n = 0, cap = 0;
  OutStr() = default;
  OutStr(const OutStr&) = delete;
  OutStr& operator=(const OutStr&) = delete;
  OutStr(OutStr&& o) noexcept : p(o.p), n(o.n), cap(o.cap) { o.p = nullptr; o.n = o.cap = 0; }
  OutStr& operator=(OutStr&& o) noexcept {
    if (this != &o) {
      free(p);
      p = o.p; n = o.n; cap = o.cap;
      o.p = nullptr; o.n = o.cap = 0;
    }
    return *this;
  }
  ~OutStr() { free(p); }
  size_t size() const { return n; }
  bool empty() const { return n == 0; }
  const char* data() const { return p; }
  void clear() { n = 0; }
  void grow(size_t need) {
    size_t c = cap ? cap * 2 : 4096;
    while (c < n + need + 64) c *= 2;
    char* q = (char*)realloc(p, c);
    if (!q) throw std::bad_alloc();
    p = q;
    cap = c;
  }
  inline void room(size_t need) {
    if (n + need + 64 > cap) grow(need);
  }
  inline OutStr& operator+=(char c) {
    room(1);
    p[n++] = c;
    return *this;
  }
  inline void append(const char* s, size_t len) {
    room(len);
    char* d = p + n;
    if (len <= 16) {
      if (len >= 8) {
        uint64_t a, b;
        memcpy(&a, s, 8);
        memcpy(&b, s + len - 8, 8);
        memcpy(d, &a, 8);
        memcpy(d + len - 8, &b, 8);
      } else if (len >= 4) {
        uint32_t a, b;
        memcpy(&a, s, 4);
        memcpy(&b, s + len - 4, 4);
        memcpy(d, &a, 4);
        memcpy(d + len - 4, &b, 4);
      } else {
        for (size_t i = 0; i < len; ++i) d[i] = s[i];
      }
    } else {
      memcpy(d, s, len);
    }
    n += len;
  }
  inline OutStr& operator+=(sv x) {
    append(x.data(), x.size());
    return *this;
  }
  inline OutStr& operator+=(const std::string& x) {
    append(x.data(), x.size());
    return *this;
  }
};

int tfail(int code, const std::string& m) {
  grimb_set_error(m.c_str());
  return code;
}

enum { H_OK = 0, H_PROBLEM = 1, H_FAULT = 2 };

struct Unknown {
  uint8_t locus;
  uint16_t id;
  std::string name;
};

struct Line {
  sv raw, sid, race1, race2;
  bool has_race = false;
  bool no_fields = false;  // rejected by the field-count check (IndexError in the reference's parser)
  uint8_t hclass = H_OK;
  uint16_t mask = 0;
  uint16_t counts[GRIMB_MAX_LOCI * 2];
  uint32_t ids_off = 0, ids_cnt = 0;   // into the owning thread's id vector
  uint32_t unk_off = 0, unk_cnt = 0;   // into the owning thread's Unknown vector
  uint32_t thread = 0;
  uint32_t prior = 0;
};

struct SvHash {
  size_t operator()(sv s) const { return std::hash<sv>()(s); }
};

inline bool py_space(unsigned char c) { return (c >= 0x09 && c <= 0x0d) || (c >= 0x1c && c <= 0x20); }

void split(sv s, char d, std::vector<sv>& out) {
  out.clear();
  size_t b = 0;
  for (;;) {
    size_t e = s.find(d, b);
    if (e == sv::npos) {
      out.push_back(s.substr(b));
      return;
    }
    out.push_back(s.substr(b, e - b));
    b = e + 1;
  }
}

// Python's repr(float) / str(float): shortest round-trip digits, fixed notation iff
// -4 < decpt <= 16 (Python/pystrtod.c format_float_short, mode 'r').  Writes at most 32 bytes.
int py_float_buf(double x, char* out) {
  char* o = out;
  auto lit = [&](const char* t) {
    size_t n = strlen(t);
    memcpy(o, t, n);
    return (int)n;
  };
  if (x == 0.0) return lit(std::signbit(x) ? "-0.0" : "0.0");
  if (std::isnan(x)) return lit("nan");
  if (std::isinf(x)) return lit(x < 0 ? "-inf" : "inf");
  char buf[48];
  auto r = std::to_chars(buf, buf + sizeof(buf), x, std::chars_format::scientific);
  const char* s = buf;
  size_t n = (size_t)(r.ptr - buf);
  if (s[0] == '-') {
    *o++ = '-';
    ++s;
    --n;
  }
  size_t e = 0;
  while (s[e] != 'e') ++e;
  int exp10 = 0;
  std::from_chars(s + e + 1 + (s[e + 1] == '+' ? 1 : 0), s + n, exp10);
  char digits[24];
  int nd = 0;
  for (size_t i = 0; i < e; ++i)
    if (s[i] != '.') digits[nd++] = s[i];
  const int decpt = exp10 + 1;
  if (decpt <= -4 || decpt > 16) {
    *o++ = digits[0];
    if (nd > 1) {
      *o++ = '.';
      memcpy(o, digits + 1, (size_t)(nd - 1));
      o += nd - 1;
    }
    *o++ = 'e';
    int ex = decpt - 1;
    *o++ = ex < 0 ? '-' : '+';
    if (ex < 0) ex = -ex;
    char eb[8];
    int k = 0;
    do {
      eb[k++] = (char)('0' + ex % 10);
      ex /= 10;
    } while (ex);
    if (k < 2) eb[k++] = '0';
    while (k) *o++ = eb[--k];
  } else if (decpt <= 0) {
    *o++ = '0';
    *o++ = '.';
    memset(o, '0', (size_t)(-decpt));
    o += -decpt;
    memcpy(o, digits, (size_t)nd);
    o += nd;
  } else if (decpt >= nd) {
    memcpy(o, digits, (size_t)nd);
    o += nd;
    memset(o, '0', (size_t)(decpt - nd));
    o += decpt - nd;
    *o++ = '.';
    *o++ = '0';
  } else {
    memcpy(o, digits, (size_t)decpt);
    o += decpt;
    *o++ = '.';
    memcpy(o, digits + decpt, (size_t)(nd - decpt));
    o += nd - decpt;
  }
  return (int)(o - out);
}

void py_float(double x, OutStr& out) {
  out.room(40);
  out.n += (size_t)py_float_buf(x, out.p + out.n);
}

void put_uint(uint64_t v, OutStr& out) {
  out.room(24);
  if (v < 10) {   // the rank column: mostly one digit
    out.p[out.n++] = (char)('0' + v);
    return;
  }
  auto r = std::to_chars(out.p + out.n, out.p + out.n + 24, v);
  out.n = (size_t)(r.ptr - out.p);
}

struct PriorKey {
  bool has;
  std::string r1, r2;
  bool operator==(const PriorKey& o) const { return has == o.has && r1 == o.r1 && r2 == o.r2; }
};
struct PriorKeyHash {
  size_t operator()(const PriorKey& k) const {
    return std::hash<std::string>()(k.r1) * 1000003u ^ std::hash<std::string>()(k.r2) ^ (k.has ? 0x9e3779b9u : 0u);
  }
};

}  // namespace

struct GrimbText {
  int L = 0, P = 0, n_threads = 1;
  std::vector<std::string> loci, pops;
  std::vector<std::vector<std::string>> alleles;              // [L][n]
  std::vector<std::unordered_map<sv, uint16_t, SvHash>> ids;  // [L] name -> id
  std::unordered_map<sv, int, SvHash> locus_index;
  std::unordered_map<sv, int, SvHash> pop_index;
  std::vector<double> count_by_prob;
  double alpha = 0, eta = 0, beta = 0, gamma = 0, delta = 0;
  bool mr = true;
  int key_bits[GRIMB_MAX_LOCI];
  int shift[GRIMB_MAX_LOCI];
  // priors (memoised across calls)
  std::unordered_map<PriorKey, uint32_t, PriorKeyHash> prior_index;
  std::vector<double> priors;
  // fast name lookup of the tokeniser: every table allele of every locus in one open-addressing table
  struct NameEnt {
    uint64_t h;
    uint64_t w0, w1;   // the name's first 16 bytes, zero padded (names of up to 16 bytes compare by these alone)
    const char* s;
    uint16_t len, id;
    uint8_t locus;
  };
  std::vector<NameEnt> name_ent;
  std::vector<uint32_t> name_slot;   // entry index + 1, 0 = empty
  uint32_t name_mask = 0;
  bool fast_path = true;             // GRIMB_TEXT_FAST=0: every line through the general parser (A/B, tests)
  bool packed_ok = true;             // GRIMB_TEXT_PACKED=0: never the packed batch form (A/B, tests)
  std::vector<uint8_t> type_allowed; // Plan_A_Matrix: [1 << L] typed-locus patterns that are matrix rows (empty: no matrix)
  // pinned staging (grow-only)
  struct HostBuf {
    void* p = nullptr;
    size_t cap = 0;
    bool pinned = false;
    void* reserve(size_t bytes) {
      if (bytes <= cap && p) return p;
      release();
      size_t want = bytes + bytes / 4 + 4096;
      p = grimb_pinned_alloc(want);
      pinned = p != nullptr;
      if (!p) p = malloc(want);
      cap = p ? want : 0;
      return p;
    }
    void release() {
      if (p) {
        if (pinned) grimb_pinned_free(p);
        else free(p);
      }
      p = nullptr;
      cap = 0;
    }
    ~HostBuf() { release(); }
  };
  // State of one chunk of input in flight: the single-call entry points use slot0, the file pipeline
  // (grimb_impute_file) keeps several so that tokenising, the GPU, formatting and file writes overlap.
  struct Slot {
    const char* text = nullptr;   // the chunk's bytes (string_views of `lines` point into them)
    size_t text_len = 0;
    std::string own;              // private copy when the caller's buffer may go away
    int64_t first_index = 0;
    std::vector<Line> lines;
    // one per tokeniser thread, each on its own cache line: push_back rewrites the vector's end pointer, and with
    // the 24-byte headers packed side by side every thread invalidated its neighbours' lines on every allele id
    // (the tokeniser ran SLOWER on 4 threads than on 1)
    struct alignas(64) IdVec : std::vector<uint16_t> {};
    struct alignas(64) UnkVec : std::vector<Unknown> {};
    std::vector<IdVec> t_ids;
    std::vector<UnkVec> t_unk;
    std::vector<uint16_t> b_typed, b_counts, b_alleles;
    std::vector<uint32_t> b_off, b_prior;
    std::vector<uint64_t> b_keys;    // packed form of the batch (include/grimb200.h): [S][2] keys ...
    std::vector<uint16_t> b_flags;   // ... and [S] flag words
    std::vector<double> priors;   // snapshot of the memoised prior matrices at tokenise time
    GrimbBatch batch;
    HostBuf hb_compact, hb_words, hb_general, hb_hap, hb_pop;
    std::vector<GrimbCompact> m_compact;      // merged results when a workspace tier overflowed
    std::vector<uint64_t> m_words;
    std::vector<GrimbSubjectResult> m_general;
    std::vector<GrimbHapRow> m_hap;
    std::vector<GrimbPopRow> m_pop;
    GrimbResults fin;
    int64_t totals[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    int64_t retries = 0;
    int64_t chunk_id = 0;         // grimb_impute_file_sharded: index of the input chunk
    int fmt_threads = 0;          // pieces per output in fmt_parts (thread order)
    std::vector<OutStr> fmt_parts;   // per-thread pieces of the six outputs (capacity reused)
    std::string out[6];
    int64_t out_size[6] = {0, 0, 0, 0, 0, 0};
    int64_t plan_count[4] = {0, 0, 0, 0};
    double sec_tok = 0, sec_gpu = 0, sec_fmt = 0;
  };
  Slot slot0;
  std::vector<std::unique_ptr<Slot>> pipe;   // slots of the file pipeline (grimb_impute_file)
  std::string file_acc[6];                   // outputs of grimb_impute_file that are kept in memory
  double per_subject[4] = {0.5, 0.05, 0.3, 0.3};   // words, general records, hap rows, pop rows (adaptive capacities)

  // Worker threads of one calling thread (the tokeniser, the formatter and the GPU stage of the file pipeline
  // each call parallel() from their own thread, concurrently): created on first use, parked on a condition
  // variable between regions -- a region costs a wake-up instead of n thread creations and joins.
  struct Pool {
    std::vector<std::thread> th;
    std::mutex m;
    std::condition_variable cv_go, cv_done;
    const std::function<void(int)>* job = nullptr;
    uint64_t gen = 0;
    int active = 0, pending = 0;
    bool stop = false;
    pid_t owner = getpid();
    // after fork() the child has this object but none of its threads: forget them (the handles are leaked on
    // purpose -- joining or destroying a std::thread whose thread does not exist in this process is undefined)
    void forget_if_forked() {
      if (getpid() == owner) return;
      new std::vector<std::thread>(std::move(th));
      th.clear();
      // the parent's parked workers were waiting on these: their internal waiter state is meaningless here
      new (&m) std::mutex();
      new (&cv_go) std::condition_variable();
      new (&cv_done) std::condition_variable();
      owner = getpid();
      job = nullptr;
      gen = 0;
      active = pending = 0;
    }
    void worker(int t) {
      uint64_t seen = 0;
      for (;;) {
        const std::function<void(int)>* j = nullptr;
        {
          std::unique_lock<std::mutex> g(m);
          cv_go.wait(g, [&] { return stop || gen != seen; });
          if (stop) return;
          seen = gen;
          if (t < active) j = job;
        }
        if (j) {
          (*j)(t);
          std::lock_guard<std::mutex> g(m);
          if (--pending == 0) cv_done.notify_one();
        }
      }
    }
    void run(int nt, const std::function<void(int)>& f) {
      forget_if_forked();
      while ((int)th.size() < nt - 1) {
        const int t = (int)th.size() + 1;   // the calling thread is worker 0
        th.emplace_back([this, t]() { worker(t); });
      }
      {
        std::lock_guard<std::mutex> g(m);
        job = &f;
        active = nt;
        pending = nt - 1;
        ++gen;
      }
      cv_go.notify_all();
      f(0);
      std::unique_lock<std::mutex> g(m);
      cv_done.wait(g, [&] { return pending == 0; });
      job = nullptr;
    }
    ~Pool() {
      forget_if_forked();
      {
        std::lock_guard<std::mutex> g(m);
        stop = true;
      }
      cv_go.notify_all();
      for (auto& x : th) x.join();
    }
  };

  template <class F>
  void parallel(size_t n, F f) const {
    int nt = n_threads;
    if ((size_t)nt > n) nt = (int)(n ? n : 1);
    if (nt <= 1) {
      f(0, (size_t)0, n);
      return;
    }
    const size_t per = (n + nt - 1) / nt;
    const std::function<void(int)> body = [&](int t) {
      const size_t lo = std::min(n, per * (size_t)t), hi = std::min(n, per * (size_t)(t + 1));
      f(t, lo, hi);
    };
    static const bool use_pool = !(getenv("GRIMB_POOL") && getenv("GRIMB_POOL")[0] == '0');
    if (use_pool) {
      tls_pool().run(nt, body);
      return;
    }
    std::vector<std::thread> th;   // GRIMB_POOL=0: a thread per slice, created and joined per region
    for (int t = 1; t < nt; ++t) th.emplace_back([&body, t]() { body(t); });
    body(0);
    for (auto& x : th) x.join();
  }
  static Pool& tls_pool() {   // one pool per calling thread, whatever the region (not one per template instance)
    static thread_local Pool pool;
    return pool;
  }

  // calc_priority_matrix (reference impute.py:1844-1924), same operation order
  void prior_matrix(const std::vector<int>& r1, const std::vector<int>& r2, std::vector<double>& M) const {
    const int n = P;
    M.assign((size_t)n * n, 0.0);
    std::vector<double> T((size_t)n * n), U((size_t)n * n);
    for (int a : r1)
      for (int b : r2) {
        if (a < 0 && b < 0) continue;
        std::fill(T.begin(), T.end(), 0.0);
        if (a < 0 || b < 0) {
          const int r = a < 0 ? b : a;
          for (int i = 0; i < n; ++i) T[(size_t)r * n + i] = T[(size_t)r * n + i] + gamma * 2;
          for (int i = 0; i < n; ++i)
            for (int j = 0; j < n; ++j) U[(size_t)i * n + j] = T[(size_t)i * n + j] + T[(size_t)j * n + i];
          T.swap(U);
          T[(size_t)r * n + r] -= gamma * 2;
        } else {
          for (int i = 0; i < n; ++i) {
            T[(size_t)a * n + i] = T[(size_t)a * n + i] + gamma;
            T[(size_t)i * n + b] = T[(size_t)i * n + b] + gamma;
          }
          T[(size_t)a * n + b] -= gamma;
          T[(size_t)a * n + b] = T[(size_t)a * n + b] + alpha;
          if (a != b) {
            for (int i = 0; i < n; ++i)
              for (int j = 0; j < n; ++j) U[(size_t)i * n + j] = T[(size_t)i * n + j] + T[(size_t)j * n + i];
            T.swap(U);
            T[(size_t)a * n + a] -= gamma;
            T[(size_t)b * n + b] -= gamma;
          }
          T[(size_t)a * n + a] += delta;
          if (a != b) T[(size_t)b * n + b] += delta;
        }
        for (int i = 0; i < n; ++i)
          for (int j = 0; j < n; ++j) {
            const double e = (i == j) ? 1.0 : 0.0;
            const double v = (eta * 1.0 + T[(size_t)i * n + j]) + beta * e;
            M[(size_t)i * n + j] += v;
          }
      }
    double total = 0.0;
    bool first = true;
    for (int i = 0; i < n; ++i)
      for (int j = 0; j < n; ++j) {
        double& m = M[(size_t)i * n + j];
        m = m * count_by_prob[i] * count_by_prob[j];
        if (first) {
          total = m;
          first = false;
        } else {
          total += m;
        }
      }
    for (double& m : M) m = m / total;
  }

  // consecutive lines mostly repeat the race fields: remember the last key
  bool last_has_race = false, last_valid = false;
  sv last_r1, last_r2;
  uint32_t last_prior = 0;

  uint32_t prior_for(const Line& ln) {
    if (last_valid && ln.has_race == last_has_race && ln.race1 == last_r1 && ln.race2 == last_r2) return last_prior;
    const uint32_t idx = prior_lookup(ln);
    last_valid = true;
    last_has_race = ln.has_race;
    last_r1 = ln.race1;      // views into this call's text buffer: reset by grimb_text_tokenise
    last_r2 = ln.race2;
    last_prior = idx;
    return idx;
  }

  std::mutex prior_m;   // the memo is shared by the tokeniser's worker threads
  uint32_t prior_lookup_locked(const Line& ln) {
    std::lock_guard<std::mutex> g(prior_m);
    return prior_lookup(ln);
  }

  uint32_t prior_lookup(const Line& ln) {
    PriorKey k{ln.has_race, std::string(ln.race1), std::string(ln.race2)};
    auto it = prior_index.find(k);
    if (it != prior_index.end()) return it->second;
    std::vector<double> M((size_t)P * P, mr ? 1.0 : 0.0);
    if (!mr)
      for (int i = 0; i < P; ++i) M[(size_t)i * P + i] = 1.0;
    if (ln.has_race && (!ln.race1.empty() || !ln.race2.empty())) {
      bool known = false;
      std::vector<sv> parts;
      std::vector<int> r1, r2;
      split(ln.race1, ';', parts);
      for (sv p : parts) {
        auto f = pop_index.find(p);
        r1.push_back(f == pop_index.end() ? -1 : f->second);
        known = known || f != pop_index.end();
      }
      split(ln.race2, ';', parts);
      for (sv p : parts) {
        auto f = pop_index.find(p);
        r2.push_back(f == pop_index.end() ? -1 : f->second);
        known = known || f != pop_index.end();
      }
      if (known) prior_matrix(r1, r2, M);
    }
    uint32_t idx = (uint32_t)(priors.size() / ((size_t)P * P));
    priors.insert(priors.end(), M.begin(), M.end());
    prior_index.emplace(std::move(k), idx);
    return idx;
  }

  // ---- fast name lookup
  static uint64_t name_hash(const char* s, size_t n) {
    uint64_t h = 0x9E3779B97F4A7C15ull ^ (uint64_t)n;
    while (n >= 8) {
      uint64_t w;
      memcpy(&w, s, 8);
      h = (h ^ w) * 0xff51afd7ed558ccdULL;
      h ^= h >> 32;
      s += 8;
      n -= 8;
    }
    if (n) {
      uint64_t w = 0;
      memcpy(&w, s, n);
      h = (h ^ w) * 0xff51afd7ed558ccdULL;
      h ^= h >> 32;
    }
    return h;
  }

  void build_name_table() {
    size_t n = 0;
    for (auto& a : alleles) n += a.size();
    uint32_t sz = 16;
    while (sz < n * 2 + 2) sz <<= 1;
    name_mask = sz - 1;
    name_slot.assign(sz, 0);
    name_ent.clear();
    name_ent.reserve(n);
    for (int l = 0; l < L; ++l)
      for (size_t i = 0; i < alleles[l].size(); ++i) {
        const std::string& nm = alleles[l][i];
        // the general parser decides the locus from the prefix before '*': only names that carry their own
        // locus prefix may take the fast path
        if (nm.size() > 0xFFFF || sv(nm).substr(0, nm.find('*')) != sv(loci[l])) continue;
        NameEnt e;
        e.h = name_hash(nm.data(), nm.size());
        e.w0 = e.w1 = 0;
        memcpy(&e.w0, nm.data(), std::min<size_t>(8, nm.size()));
        if (nm.size() > 8) memcpy(&e.w1, nm.data() + 8, std::min<size_t>(8, nm.size() - 8));
        e.s = nm.data();
        e.len = (uint16_t)nm.size();
        e.id = (uint16_t)(i + 1);
        e.locus = (uint8_t)l;
        uint32_t h = (uint32_t)e.h & name_mask;
        bool dup = false;
        while (name_slot[h]) {
          const NameEnt& o = name_ent[name_slot[h] - 1];
          if (o.h == e.h && o.len == e.len && memcmp(o.s, e.s, e.len) == 0) dup = true;   // same name under two loci
          h = (h + 1) & name_mask;
        }
        if (dup) {
          fast_path = false;
          continue;
        }
        name_ent.push_back(e);
        name_slot[h] = (uint32_t)name_ent.size();
      }
  }

  // `wide`: 16 bytes are readable at s (the name is not within 16 bytes of the end of the text buffer)
  const NameEnt* find_name(const char* s, size_t n, bool wide) const {
    if (wide && n <= 16 && n > 0) {
      // the name as two zero-padded words: they feed the same hash as name_hash() and are the comparison
      uint64_t w0, w1;
      memcpy(&w0, s, 8);
      memcpy(&w1, s + 8, 8);
      if (n < 8) {
        w0 &= ~0ull >> (8 * (8 - n));
        w1 = 0;
      } else if (n < 16) {
        w1 = n == 8 ? 0 : (w1 & (~0ull >> (8 * (16 - n))));
      }
      uint64_t hv = 0x9E3779B97F4A7C15ull ^ (uint64_t)n;
      hv = (hv ^ w0) * 0xff51afd7ed558ccdULL;
      hv ^= hv >> 32;
      if (n > 8) {
        hv = (hv ^ w1) * 0xff51afd7ed558ccdULL;
        hv ^= hv >> 32;
      }
      uint32_t h = (uint32_t)hv & name_mask;
      for (;;) {
        const uint32_t k = name_slot[h];
        if (!k) return nullptr;
        const NameEnt& e = name_ent[k - 1];
        if (e.w0 == w0 && e.w1 == w1 && e.len == n) return &e;
        h = (h + 1) & name_mask;
      }
    }
    const uint64_t hv = name_hash(s, n);
    uint32_t h = (uint32_t)hv & name_mask;
    for (;;) {
      const uint32_t k = name_slot[h];
      if (!k) return nullptr;
      const NameEnt& e = name_ent[k - 1];
      if (e.h == hv && e.len == n && memcmp(e.s, s, n) == 0) return &e;
      h = (h + 1) & name_mask;
    }
  }

  // first character at or after q (before lim) that is not a plain name character: a delimiter of the GL grammar
  // or one of 'g' 'L' 'U'; `wide_end`: last address from which 16 bytes may be read
  static inline const char* scan_name(const char* q, const char* lim, const char* wide_end) {
#if defined(__SSE2__)
    while (q < lim && q <= wide_end) {
      const __m128i v = _mm_loadu_si128(reinterpret_cast<const __m128i*>(q));
      __m128i m = _mm_cmpeq_epi8(v, _mm_set1_epi8('/'));
      m = _mm_or_si128(m, _mm_cmpeq_epi8(v, _mm_set1_epi8('+')));
      m = _mm_or_si128(m, _mm_cmpeq_epi8(v, _mm_set1_epi8('^')));
      m = _mm_or_si128(m, _mm_cmpeq_epi8(v, _mm_set1_epi8('g')));
      m = _mm_or_si128(m, _mm_cmpeq_epi8(v, _mm_set1_epi8('L')));
      m = _mm_or_si128(m, _mm_cmpeq_epi8(v, _mm_set1_epi8('U')));
      const unsigned bits = (unsigned)_mm_movemask_epi8(m);
      if (bits) {
        const char* f = q + __builtin_ctz(bits);
        return f < lim ? f : lim;
      }
      q += 16;
    }
    if (q > lim) return lim;
#endif
    while (q < lim && kCharClass.c[(unsigned char)*q] == 0) ++q;
    return q;
  }

  // Fast path of the tokeniser: one pass over a line of the regular shape
  //     id,LOC*a[/LOC*b...]+LOC*c[/...]^LOC2*...+...[,race1,race2[,...]]
  // with the loci in ascending loci_map order, every listed allele a table allele carrying its locus prefix,
  // and none of the characters clean_up_gl (impute.py:105-118) reacts to ('g', 'L', 'U').  For such a line
  // the general parser below does exactly this: the per-side sorts (gl2haps, impute.py:271) are no-ops
  // because every string starts with its locus prefix and the prefixes ascend, the locus of a chunk is
  // that of its first name, and ids are listed locus by locus, side 0 then side 1, duplicates dropped.
  // Anything else returns false with nothing changed, and the general parser takes the line.
  struct CharClass {   // 0 name character, 1 delimiter of the GL grammar, 2 'g' / 'L' / 'U'
    uint8_t c[256];
    CharClass() {
      memset(c, 0, sizeof(c));
      c[(unsigned char)'/'] = c[(unsigned char)'+'] = c[(unsigned char)'^'] = 1;
      c[(unsigned char)'g'] = c[(unsigned char)'L'] = c[(unsigned char)'U'] = 2;
    }
  };
  static inline const CharClass kCharClass{};

  bool parse_fast(Slot& S, sv raw_line, Line& ln, int thread) const {
    size_t e = raw_line.size();
    while (e > 0 && py_space((unsigned char)raw_line[e - 1])) --e;
    const char* p = raw_line.data();
    const char* end = p + e;
    const char* c1 = (const char*)memchr(p, ',', e);
    if (!c1) return false;
    const char* g0 = c1 + 1;
    const char* c2 = (const char*)memchr(g0, ',', (size_t)(end - g0));
    const char* g1 = c2 ? c2 : end;
    sv race1, race2;
    if (c2) {
      const char* r1 = c2 + 1;
      const char* c3 = (const char*)memchr(r1, ',', (size_t)(end - r1));
      if (!c3) return false;   // exactly three fields: the reference's parser raises
      const char* r2 = c3 + 1;
      const char* c4 = (const char*)memchr(r2, ',', (size_t)(end - r2));
      race1 = sv(r1, (size_t)(c3 - r1));
      race2 = sv(r2, (size_t)((c4 ? c4 : end) - r2));
    }
    if (g0 == g1) return false;
    // 16-byte loads are allowed up to here (the line lies inside the slot's text buffer)
    const char* wide_end = S.text_len >= 16 ? S.text + S.text_len - 16 : nullptr;
    std::vector<uint16_t>& idv = S.t_ids[thread];
    const size_t ids_off = idv.size();
    uint16_t counts[GRIMB_MAX_LOCI * 2];
    memset(counts, 0, sizeof(counts));
    uint32_t mask = 0;
    int last_l = -1;
    const char* q = g0;
    for (;;) {   // one locus chunk: side '+' side
      int l = -1;
      for (int side = 0; side < 2; ++side) {
        const size_t lst = idv.size();
        for (;;) {   // one allele name
          const char* n0 = q;
          q = scan_name(q, g1, wide_end);
          if (q < g1 && kCharClass.c[(unsigned char)*q] == 2) goto slow;   // a character clean_up_gl reacts to
          if (q == n0) goto slow;
          const NameEnt* ne = find_name(n0, (size_t)(q - n0), n0 <= wide_end);
          if (!ne) goto slow;
          if (l < 0) {
            l = ne->locus;
            if (l <= last_l) goto slow;
          } else if (ne->locus != l) {
            goto slow;
          }
          bool seen = false;
          for (size_t k = lst; k < idv.size(); ++k) seen = seen || idv[k] == ne->id;
          if (!seen) idv.push_back(ne->id);
          if (q < g1 && *q == '/') {
            ++q;
            continue;
          }
          break;
        }
        counts[2 * l + side] = (uint16_t)(idv.size() - lst);
        if (side == 0) {
          if (q >= g1 || *q != '+') goto slow;
          ++q;
        }
      }
      mask |= 1u << l;
      last_l = l;
      if (q == g1) break;
      if (*q != '^') goto slow;   // e.g. a third side
      ++q;
      if (q == g1) goto slow;     // trailing '^'
    }
    ln = Line();
    ln.raw = sv(p, e);
    ln.sid = sv(p, (size_t)(c1 - p));
    ln.has_race = c2 != nullptr;
    ln.race1 = race1;
    ln.race2 = race2;
    ln.no_fields = false;
    ln.hclass = H_OK;
    ln.thread = (uint32_t)thread;
    ln.mask = (uint16_t)mask;
    memcpy(ln.counts, counts, sizeof(counts));
    ln.ids_off = (uint32_t)ids_off;
    ln.ids_cnt = (uint32_t)(idv.size() - ids_off);
    ln.unk_off = (uint32_t)S.t_unk[thread].size();
    ln.unk_cnt = 0;
    return true;
  slow:
    idv.resize(ids_off);
    return false;
  }

  // one input line -> Line (reference impute.py:2022-2036 + clean_up_gl + gl2haps)
  void parse_line(Slot& S, sv raw_line, Line& ln, int thread, bool planb, std::string& clean, std::vector<sv>& f1,
                  std::vector<sv>& f2, std::vector<sv>& t1, std::vector<sv>& t2, std::vector<sv>& names,
                  std::vector<uint16_t>& scr) {
    size_t e = raw_line.size();
    while (e > 0 && py_space((unsigned char)raw_line[e - 1])) --e;
    sv raw = raw_line.substr(0, e);
    ln = Line();
    ln.raw = raw;
    ln.thread = (uint32_t)thread;
    split(raw, raw.find(',') != sv::npos ? ',' : '%', f1);
    ln.sid = f1[0];
    if (f1.size() < 2 || f1.size() == 3) {
      ln.hclass = H_FAULT;  // IndexError in the reference's line parser
      ln.no_fields = true;
      return;
    }
    sv gl = f1[1];
    if (f1.size() > 2) {
      ln.has_race = true;
      ln.race1 = f1[2];
      ln.race2 = f1[3];
    }
    if (gl.empty()) {
      ln.hclass = H_PROBLEM;
      return;
    }
    // clean_up_gl: drop every 'g' and 'L', then loci that start or end with 'U'
    clean.clear();
    for (char c : gl)
      if (c != 'g' && c != 'L') clean += c;
    split(sv(clean), '^', f2);
    size_t w = 0;
    for (sv p : f2)
      if (!(!p.empty() && (p.front() == 'U' || p.back() == 'U'))) f2[w++] = p;
    f2.resize(w);
    if (f2.empty() || (f2.size() == 1 && (f2[0].empty() || f2[0] == " "))) {
      ln.hclass = H_PROBLEM;
      return;
    }
    t1.clear();
    t2.clear();
    for (sv chunk : f2) {
      if (chunk.empty()) {
        ln.hclass = H_FAULT;  // IndexError on chunk[0]
        return;
      }
      if (chunk[0] == '+') chunk.remove_prefix(1);
      size_t p = chunk.find('+');
      if (p == sv::npos) {
        if (chunk.empty()) continue;
        ln.hclass = H_PROBLEM;  // a locus without '+': gl2haps returns []
        return;
      }
      sv rest = chunk.substr(p + 1);
      size_t q = rest.find('+');
      t1.push_back(chunk.substr(0, p));
      t2.push_back(q == sv::npos ? rest : rest.substr(0, q));
    }
    if (t1.empty()) {
      ln.hclass = H_FAULT;  // 2 ** (0 - 1) phases
      return;
    }
    std::sort(t1.begin(), t1.end());
    std::sort(t2.begin(), t2.end());
    std::vector<uint16_t>& idv = S.t_ids[thread];
    std::vector<Unknown>& unk = S.t_unk[thread];
    const uint32_t ids_off = (uint32_t)idv.size(), unk_off = (uint32_t)unk.size();
    // the id lists of this line, built in a reused scratch vector: [off, off + cnt) per locus and side
    scr.clear();
    uint32_t per_off[GRIMB_MAX_LOCI][2] = {{0}}, per_cnt[GRIMB_MAX_LOCI][2] = {{0}};
    bool used[GRIMB_MAX_LOCI] = {false};
    auto foreign = [&]() {
      idv.resize(ids_off);
      unk.resize(unk_off);
      ln.hclass = planb ? H_FAULT : H_OK;  // mask stays 0: nothing is imputed
      ln.mask = 0;
    };
    if (!type_allowed.empty()) {
      // Plan_A_Matrix: input_type (impute.py:1574-1579) looks every typed locus up before anything else --
      // an unknown locus raises (raw line in .problem); a repeated locus gives a pattern that is no matrix row
      bool repeated = false;
      bool seen_l[GRIMB_MAX_LOCI] = {false};
      for (size_t k = 0; k < t1.size(); ++k) {
        sv first = t1[k].substr(0, t1[k].find('/'));
        auto li = locus_index.find(first.substr(0, first.find('*')));
        if (li == locus_index.end()) {
          ln.hclass = H_FAULT;
          return;
        }
        repeated = repeated || seen_l[li->second];
        seen_l[li->second] = true;
      }
      if (repeated) {
        ln.hclass = H_PROBLEM;
        return;
      }
    }
    for (size_t k = 0; k < t1.size(); ++k) {
      sv first = t1[k].substr(0, t1[k].find('/'));
      sv prefix = first.substr(0, first.find('*'));
      auto li = locus_index.find(prefix);
      if (li == locus_index.end() || used[li->second]) return foreign();
      const int l = li->second;
      used[l] = true;
      const int n_tab = (int)alleles[l].size();
      const int cap = (1 << key_bits[l]) - 1;
      std::vector<std::pair<sv, uint16_t>> local;
      for (int x = 0; x < 2; ++x) {
        split(x ? t2[k] : t1[k], '/', names);
        const uint32_t lst_off = (uint32_t)scr.size();
        per_off[l][x] = lst_off;
        for (sv name : names) {
          if (name.substr(0, name.find('*')) != sv(loci[l])) return foreign();
          uint16_t id = 0;
          auto it = ids[l].find(name);
          if (it != ids[l].end()) id = it->second;
          else {
            for (auto& pr : local)
              if (pr.first == name) id = pr.second;
            if (!id) {
              int nid = n_tab + 1 + (int)local.size();
              if (nid > cap) {
                idv.resize(ids_off);
                unk.resize(unk_off);
                ln.hclass = H_FAULT;
                return;
              }
              id = (uint16_t)nid;
              local.emplace_back(name, id);
              unk.push_back(Unknown{(uint8_t)l, id, std::string(name)});
            }
          }
          if (std::find(scr.begin() + lst_off, scr.end(), id) == scr.end()) scr.push_back(id);
        }
        per_cnt[l][x] = (uint32_t)scr.size() - lst_off;
      }
    }
    memset(ln.counts, 0, sizeof(ln.counts));
    for (int l = 0; l < L; ++l)
      if (used[l]) {
        ln.mask |= (uint16_t)(1u << l);
        for (int x = 0; x < 2; ++x) {
          ln.counts[l * 2 + x] = (uint16_t)per_cnt[l][x];
          idv.insert(idv.end(), scr.begin() + per_off[l][x], scr.begin() + per_off[l][x] + per_cnt[l][x]);
        }
      }
    ln.ids_off = ids_off;
    ln.ids_cnt = (uint32_t)idv.size() - ids_off;
    ln.unk_off = unk_off;
    ln.unk_cnt = (uint32_t)unk.size() - unk_off;
  }

  sv allele_name(const Slot& S, int l, uint32_t id, const Line& ln) const {
    if (id >= 1 && id <= alleles[l].size()) return alleles[l][id - 1];
    const std::vector<Unknown>& u = S.t_unk[ln.thread];
    for (uint32_t i = 0; i < ln.unk_cnt; ++i)
      if (u[ln.unk_off + i].locus == l && u[ln.unk_off + i].id == id) return u[ln.unk_off + i].name;
    return "?";
  }

  // allele id of locus l inside a packed key (GRIMB_KEY_WORDS little-endian 64-bit words)
#if GRIMB_KEY_WORDS == 1
  typedef uint64_t keyref;
  uint32_t field(keyref key, int l) const { return (uint32_t)((key >> shift[l]) & ((1ull << key_bits[l]) - 1ull)); }
#else
  typedef const uint64_t* keyref;
  uint32_t field(keyref key, int l) const {
    const unsigned __int128 k = (unsigned __int128)key[0] | ((unsigned __int128)key[1] << 64);
    return (uint32_t)((uint64_t)(k >> shift[l]) & ((1ull << key_bits[l]) - 1ull));
  }
#endif

  void put_hap(const Slot& S, keyref key, const Line& ln, OutStr& o) const {
    bool first = true;
    for (int l = 0; l < L; ++l) {
      uint32_t id = field(key, l);
      if (!id) continue;
      if (!first) o += '~';
      first = false;
      o += allele_name(S, l, id, ln);
    }
  }

  sv pop_name(uint16_t p) const { return p == 0xFFFF ? sv("all_pops") : sv(pops[p]); }

  static void put_row_tail(double prob, uint32_t k, OutStr& s) {
    s += ',';
    py_float(prob, s);
    s += ',';
    put_uint(k, s);
    s += '\n';
  }

  // a probability with its text (most rows of a subject of the single-population path repeat one value)
  struct ProbText {
    double v;
    char t[40];
    int n;
  };
  static void put_row_tail(const ProbText& pt, double prob, uint32_t k, OutStr& s) {
    if (dbits_equal(prob, pt.v)) {
      s += ',';
      s.append(pt.t, (size_t)pt.n);
      s += ',';
      put_uint(k, s);
      s += '\n';
    } else {
      put_row_tail(prob, k, s);
    }
  }
  static bool dbits_equal(double a, double b) { return memcmp(&a, &b, 8) == 0; }

  void put_pop_row(sv sid, sv x, sv y, double prob, uint32_t k, bool sorted, OutStr& s,
                   const ProbText* pt = nullptr) const {
    if (sorted && y < x) std::swap(x, y);
    s += sid;
    s += ',';
    s += x;
    s += ',';
    s += y;
    if (pt) put_row_tail(*pt, prob, k, s);
    else put_row_tail(prob, k, s);
  }

  // Rows of a subject the warp-per-subject kernels finished (GRIMB_KIND_SIMPLE / GRIMB_KIND_TYPED, ABI v4):
  // every locus typed with one allele per side, so the single UMUG genotype is the subject's own allele
  // pairs and a PMUG row's haplotypes follow from its phase id (bit m: locus m takes its side-2 allele in
  // the first haplotype).  Same row order and text as the general layout below.
  void format_compact(const Slot& S, const Line& ln, const GrimbCompact& c, const uint64_t* words, const GrimbConfig* cfg,
                      OutStr* o) const {
    const uint16_t* ids = S.t_ids[ln.thread].data() + ln.ids_off;   // [L][2]
    const uint32_t kind = c.kind_flags & 3u;
    uint32_t n_pmug = c.kind_flags >> 4;
    const bool has = (c.kind_flags & GRIMB_KIND_HAS_RESULTS) != 0;
    const uint64_t* w = words + c.off;
    uint32_t n_pops = 0;
    uint32_t phase[16];
    const uint64_t* pmug_prob = nullptr;   // nullptr: the single PMUG row carries `total`
    const uint64_t* pop_prob = nullptr;
    const uint64_t* pop_code = nullptr;
    if (kind == GRIMB_KIND_SIMPLE && n_pmug == 15u) {
      // long form (more than four PMUG rows): a count word, a word of phase ids, then the probabilities
      n_pmug = (uint32_t)w[0] > 16u ? 16u : (uint32_t)w[0];
      for (uint32_t k = 0; k < n_pmug; ++k) phase[k] = (uint32_t)(w[1] >> (4 * k)) & 15u;
      pmug_prob = w + 2;
      n_pops = (has && cfg->n_pop_results >= 1) ? 1u : 0u;
    } else if (kind == GRIMB_KIND_SIMPLE) {
      for (uint32_t k = 0; k < n_pmug; ++k) phase[k] = (c.phases >> (4 * k)) & 15u;
      if (c.kind_flags & GRIMB_KIND_WORDS) pmug_prob = w;
      n_pops = (has && cfg->n_pop_results >= 1) ? 1u : 0u;
    } else {
      const uint64_t hdr = w[0];
      n_pops = (uint32_t)(hdr & 0xFFFFu);
      for (uint32_t k = 0; k < n_pmug; ++k) phase[k] = (uint32_t)(hdr >> (16 + 12 * k)) & 0xFFFu;
      pmug_prob = w + 1;
      pop_prob = w + 1 + n_pmug;
      pop_code = pop_prob + n_pops;
    }
    auto dbl = [](uint64_t u) {
      double d;
      memcpy(&d, &u, 8);
      return d;
    };
    ProbText pt;
    pt.v = c.total;
    pt.n = py_float_buf(c.total, pt.t);
    auto pop_pair = [&](uint32_t k, sv& x, sv& y, double& p) {
      if (!pop_code) {
        x = y = sv(pops[0]);
        p = c.total;
        return;
      }
      const uint32_t code = (uint32_t)(pop_code[k >> 2] >> (16 * (k & 3u))) & 0xFFFFu;
      x = sv(pops[code >> 8]);
      y = sv(pops[code & 0xFFu]);
      p = dbl(pop_prob[k]);
    };
    if (cfg->output_pmug) {
      for (uint32_t k = 0; k < n_pmug; ++k) {
        OutStr& s = o[GRIMB_OUT_PMUG];
        s += ln.sid;
        s += ',';
        for (int side = 0; side < 2; ++side) {
          if (side) s += '+';
          for (int l = 0; l < L; ++l) {
            if (l) s += '~';
            s += allele_name(S, l, ids[2 * l + (int)(((phase[k] >> l) & 1u) ^ (uint32_t)side)], ln);
          }
        }
        put_row_tail(pt, pmug_prob ? dbl(pmug_prob[k]) : c.total, k, s);
      }
      for (uint32_t k = 0; k < n_pops; ++k) {
        sv x, y;
        double p;
        pop_pair(k, x, y, p);
        put_pop_row(ln.sid, x, y, p, k, false, o[GRIMB_OUT_PMUG_POPS], &pt);
      }
    }
    if (cfg->output_umug && has) {
      if (cfg->n_results >= 1) {
        OutStr& s = o[GRIMB_OUT_UMUG];
        s += ln.sid;
        s += ',';
        for (int l = 0; l < L; ++l) {
          sv x = allele_name(S, l, ids[2 * l], ln), y = allele_name(S, l, ids[2 * l + 1], ln);
          if (y < x) std::swap(x, y);
          if (l) s += '^';
          s += x;
          s += '+';
          s += y;
        }
        put_row_tail(pt, c.total, 0, s);
      }
      for (uint32_t k = 0; k < n_pops; ++k) {
        sv x, y;
        double p;
        pop_pair(k, x, y, p);
        put_pop_row(ln.sid, x, y, p, k, true, o[GRIMB_OUT_UMUG_POPS], &pt);
      }
    }
  }

  void format_subject(const Slot& S, const Line& ln, const GrimbSubjectResult& r, const GrimbHapRow* hr, const GrimbPopRow* pr,
                      const GrimbConfig* cfg, OutStr* o) const {
    if (cfg->output_pmug) {
      for (uint32_t k = 0; k < r.n_pmug; ++k) {
        const GrimbHapRow& row = hr[r.hap_off + r.n_umug + k];
        OutStr& s = o[GRIMB_OUT_PMUG];
        s += ln.sid;
        s += ',';
        put_hap(S, row.a, ln, s);
        s += '+';
        put_hap(S, row.b, ln, s);
        put_row_tail(row.prob, k, s);
      }
      for (uint32_t k = 0; k < r.n_pmug_pops; ++k) {
        const GrimbPopRow& row = pr[r.pop_off + r.n_umug_pops + k];
        put_pop_row(ln.sid, pop_name(row.pop_a), pop_name(row.pop_b), row.prob, k, false, o[GRIMB_OUT_PMUG_POPS]);
      }
    }
    if (cfg->output_umug) {
      for (uint32_t k = 0; k < r.n_umug; ++k) {
        const GrimbHapRow& row = hr[r.hap_off + k];
        OutStr& s = o[GRIMB_OUT_UMUG];
        s += ln.sid;
        s += ',';
        bool first = true;
        for (int l = 0; l < L; ++l) {
          uint32_t a = field(row.a, l), b = field(row.b, l);
          if (!a) continue;
          sv x = allele_name(S, l, a, ln), y = allele_name(S, l, b, ln);
          if (y < x) std::swap(x, y);
          if (!first) s += '^';
          first = false;
          s += x;
          s += '+';
          s += y;
        }
        put_row_tail(row.prob, k, s);
      }
      const bool planc_empty = r.plan_umug == GRIMB_PLAN_C && r.tot_umug == 0;
      for (uint32_t k = 0; k < r.n_umug_pops; ++k) {
        const GrimbPopRow& row = pr[r.pop_off + k];
        OutStr& s = o[GRIMB_OUT_UMUG_POPS];
        sv x = pop_name(row.pop_a), y = pop_name(row.pop_b);
        if (y < x) std::swap(x, y);
        s += ln.sid;
        s += ',';
        s += x;
        s += ',';
        s += y;
        s += ',';
        if (planc_empty) s += '0';  // sum() of an empty dict is the int 0 (reference impute.py:1376)
        else py_float(row.prob, s);
        s += ',';
        put_uint(k, s);
        s += '\n';
      }
    }
  }
};

extern "C" int grimb_text_create(const GrimbTextDesc* d, GrimbText** out) {
  if (!d || !out || d->n_loci < 1 || d->n_loci > GRIMB_MAX_LOCI || d->n_pops < 1) return tfail(GRIMB_E_ARG, "bad text descriptor");
  GrimbText* t = new GrimbText();
  t->L = d->n_loci;
  t->P = d->n_pops;
  t->n_threads = d->n_threads > 0 ? d->n_threads : (int)std::max(1u, std::thread::hardware_concurrency());
  size_t pos = 0;
  int sh = 0;
  t->alleles.resize(t->L);
  t->ids.resize(t->L);
  for (int l = 0; l < t->L; ++l) {
    t->loci.emplace_back(d->locus_names[l]);
    t->key_bits[l] = d->key_bits[l];
    t->shift[l] = sh;
    sh += d->key_bits[l];
    t->alleles[l].reserve((size_t)d->allele_counts[l]);
    for (int i = 0; i < d->allele_counts[l]; ++i) t->alleles[l].emplace_back(d->allele_names[pos++]);
  }
  for (int l = 0; l < t->L; ++l) {
    t->locus_index.emplace(sv(t->loci[l]), l);
    for (size_t i = 0; i < t->alleles[l].size(); ++i) t->ids[l].emplace(sv(t->alleles[l][i]), (uint16_t)(i + 1));
  }
  for (int p = 0; p < t->P; ++p) t->pops.emplace_back(d->pop_names[p]);
  for (int p = 0; p < t->P; ++p) t->pop_index.emplace(sv(t->pops[p]), p);  // first occurrence wins, like list.index
  t->count_by_prob.assign(d->count_by_prob, d->count_by_prob + t->P);
  t->alpha = d->alpha;
  t->eta = d->eta;
  t->beta = d->beta;
  t->gamma = d->gamma;
  t->delta = d->delta;
  t->mr = d->unk_priors_mr != 0;
  if (d->type_allowed) t->type_allowed.assign(d->type_allowed, d->type_allowed + ((size_t)1 << t->L));
  if (const char* fp = getenv("GRIMB_TEXT_FAST"))
    if (fp[0] == '0') t->fast_path = false;
  if (const char* pk = getenv("GRIMB_TEXT_PACKED"))
    if (pk[0] == '0') t->packed_ok = false;
  // the fast path relies on the loci ascending in loci_map order == ascending string order of "LOC*"
  for (int l = 1; l < t->L; ++l)
    if (!(t->loci[l - 1] + "*" < t->loci[l] + "*")) t->fast_path = false;
  t->build_name_table();
  *out = t;
  return GRIMB_OK;
}

// sizeof of the ABI structs as this library was compiled (bindings check their own layouts against it):
// 0 GrimbConfig, 1 GrimbTableDesc, 2 GrimbTextDesc, 3 GrimbBatch, 4 GrimbResults, 5 GrimbTextOut, 6 GrimbFileStats,
// 7 GrimbTableInfo
extern "C" int64_t grimb_struct_size(int32_t which) {
  switch (which) {
    case 0: return (int64_t)sizeof(GrimbConfig);
    case 1: return (int64_t)sizeof(GrimbTableDesc);
    case 2: return (int64_t)sizeof(GrimbTextDesc);
    case 3: return (int64_t)sizeof(GrimbBatch);
    case 4: return (int64_t)sizeof(GrimbResults);
    case 5: return (int64_t)sizeof(GrimbTextOut);
    case 6: return (int64_t)sizeof(GrimbFileStats);
    case 7: return (int64_t)sizeof(GrimbTableInfo);
    case 8: return (int64_t)sizeof(GrimbRows);
    default: return -1;
  }
}

extern "C" int grimb_text_free(GrimbText* t) {
  delete t;
  return GRIMB_OK;
}

namespace {

using Slot = GrimbText::Slot;
using clk = std::chrono::steady_clock;
inline double secs(clk::time_point a, clk::time_point b) { return std::chrono::duration<double>(b - a).count(); }

// input bytes -> Lines + the GrimbBatch arrays of the slot.  `borrow`: the caller keeps `text` alive until
// the slot has been formatted; otherwise the slot takes a private copy.
int tokenise_slot(GrimbText* t, Slot& S, const GrimbConfig* cfg, const char* text, int64_t len, int64_t first_line_index,
                  bool borrow) {
  auto t0 = clk::now();
  if (borrow) {
    S.text = text;
  } else {
    S.own.assign(text, (size_t)len);
    S.text = S.own.data();
  }
  S.text_len = (size_t)len;
  S.first_index = first_line_index;
  const char* p = S.text;
  const size_t n = S.text_len;
  const int nt = t->n_threads;
  // line boundaries (Python file iteration: split on '\n', a final line without '\n' counts): every thread
  // counts the newlines of its byte range, then parses the lines that START in its range
  std::vector<size_t> cut((size_t)nt + 1, 0), nl((size_t)nt + 1, 0);
  for (int k = 0; k <= nt; ++k) cut[k] = n * (size_t)k / (size_t)nt;
  // a range starts at the first line start at or after cut[k]
  for (int k = 1; k < nt; ++k) {
    size_t b0 = cut[k];
    if (b0 > 0 && b0 < n && p[b0 - 1] != '\n') {
      const void* q = memchr(p + b0, '\n', n - b0);
      b0 = q ? (size_t)((const char*)q - p) + 1 : n;
    }
    cut[k] = b0;
  }
  for (int k = 1; k <= nt; ++k)
    if (cut[k] < cut[k - 1]) cut[k] = cut[k - 1];
  t->parallel((size_t)nt, [&](int, size_t lo, size_t hi) {
    for (size_t k = lo; k < hi; ++k) {
      size_t c = 0;
      const char* q = p + cut[k];
      const char* e = p + cut[k + 1];
      while (q < e) {
        const void* f = memchr(q, '\n', (size_t)(e - q));
        ++c;   // a line (terminated here, or the unterminated tail of the range)
        if (!f) break;
        q = (const char*)f + 1;
      }
      nl[k + 1] = c;
    }
  });
  for (int k = 0; k < nt; ++k) nl[k + 1] += nl[k];
  const size_t NS = nl[nt];
  auto tA = clk::now();
  S.lines.resize(NS);   // every Line is reset by the parser that fills it
  S.t_ids.resize((size_t)nt);
  S.t_unk.resize((size_t)nt);
  for (auto& v : S.t_ids) v.clear();
  for (auto& v : S.t_unk) v.clear();
  const bool planb = cfg->planb != 0;
  const bool fast = t->fast_path;
  const int L = t->L;
  S.b_typed.resize(NS);
  S.b_off.resize(NS + 1);
  S.b_prior.resize(NS);
  std::vector<size_t> r_ids((size_t)nt + 1, 0);
  std::vector<uint8_t> r_multi((size_t)nt, 0), r_prior((size_t)nt, 0), r_part((size_t)nt, 0);
  const uint32_t full_mask = (1u << L) - 1u;
  // parse: every range its own lines; b_off is written relative to the range and re-based below
  t->parallel((size_t)nt, [&](int, size_t klo, size_t khi) {
    std::string clean;
    std::vector<sv> f1, f2, t1, t2, names;
    std::vector<uint16_t> scr;
    for (size_t k = klo; k < khi; ++k) {
      size_t i = nl[k];
      const char* q = p + cut[k];
      const char* e = p + cut[k + 1];
      // consecutive lines mostly repeat the race fields: remember the last key of this range
      bool lv = false, l_has = false;
      sv l_r1, l_r2;
      uint32_t l_prior = 0;
      size_t run = 0;
      bool multi = false, other_prior = false, partial = false;
      while (q < e) {
        const void* f = memchr(q, '\n', (size_t)(e - q));
        const char* le = f ? (const char*)f + 1 : e;
        const sv line(q, (size_t)(le - q));
        Line& ln = S.lines[i];
        if (!(fast && t->parse_fast(S, line, ln, (int)k)))
          t->parse_line(S, line, ln, (int)k, planb, clean, f1, f2, t1, t2, names, scr);
        if (!t->type_allowed.empty() && ln.hclass == H_OK && ln.mask && !t->type_allowed[ln.mask]) {
          // Plan_A_Matrix: the typed-locus pattern is no matrix row (impute.py:1592-1596) -> .problem "i,id"
          S.t_ids[k].resize(ln.ids_off);
          S.t_unk[k].resize(ln.unk_off);
          ln.hclass = H_PROBLEM;
          ln.mask = 0;
        }
        if (!ln.no_fields) {   // the reference computes the prior before looking at the GL
          if (!(lv && ln.has_race == l_has && ln.race1 == l_r1 && ln.race2 == l_r2)) {
            l_prior = t->prior_lookup_locked(ln);
            lv = true;
            l_has = ln.has_race;
            l_r1 = ln.race1;
            l_r2 = ln.race2;
          }
          ln.prior = l_prior;
        }
        S.b_prior[i] = ln.prior;
        other_prior = other_prior || ln.prior != 0;
        S.b_off[i] = (uint32_t)run;
        const bool valid = ln.hclass == H_OK && ln.mask;
        S.b_typed[i] = valid ? ln.mask : (uint16_t)0;
        if (valid) {
          run += ln.ids_cnt;
          multi = multi || ln.ids_cnt != 2u * (uint32_t)__builtin_popcount(ln.mask);
          partial = partial || ln.mask != full_mask;
        }
        ++i;
        q = le;
      }
      r_ids[k + 1] = run;   // == S.t_ids[k].size(): only valid lines leave ids behind
      r_multi[k] = multi;
      r_prior[k] = other_prior;
      r_part[k] = partial;
    }
  });
  auto tB = clk::now();
  bool all_single = true, one_prior = true, all_full = true;
  for (int k = 0; k < nt; ++k) {
    r_ids[k + 1] += r_ids[k];
    all_single = all_single && !r_multi[k];
    one_prior = one_prior && !r_prior[k];
    all_full = all_full && !r_part[k];
  }
  // packed form (ABI v4): every imputable line is typed at every locus with one allele per side -> the
  // subject travels as its two packed keys + a flag word (18 bytes) instead of mask, offset and 2L ids
  const bool packed = GRIMB_KEY_WORDS == 1 && L <= 5 && all_single && all_full && t->packed_ok;
  const size_t total = r_ids[nt];
  S.b_off[NS] = (uint32_t)total;
  {
    std::lock_guard<std::mutex> g(t->prior_m);
    if (t->priors.empty()) {   // no line carried fields: the kernels still expect matrix 0
      Line dummy;
      t->prior_lookup(dummy);
    }
    S.priors = t->priors;   // snapshot: a later chunk may add matrices while this one is still on the GPU
  }
  auto tC = clk::now();
  S.b_alleles.resize(total ? total : 1);
  // ABI v4: the counts travel only when some subject lists several alleles on a side (every typed side
  // lists at least one), the prior indices only when more than one prior matrix is in use
  if (!all_single) S.b_counts.assign(NS * (size_t)L * 2, 0);
  if (packed) {
    S.b_keys.resize(NS * 2 + 2);
    S.b_flags.resize(NS + 1);
  }
  t->parallel((size_t)nt, [&](int, size_t klo, size_t khi) {
    for (size_t k = klo; k < khi; ++k) {
      const uint32_t base = (uint32_t)r_ids[k];
      if (!S.t_ids[k].empty()) memcpy(&S.b_alleles[base], S.t_ids[k].data(), S.t_ids[k].size() * 2);
      for (size_t i = nl[k]; i < nl[k + 1]; ++i) {
        if (packed) {
          const Line& ln = S.lines[i];
          uint64_t k0 = 0, k1 = 0;
          uint32_t fl = 0x8000u;   // skip
          if (ln.hclass == H_OK && ln.mask) {
            const uint16_t* ids = S.t_ids[k].data() + ln.ids_off;
            fl = 0;
            for (int l = 0; l < L; ++l) {
              const uint32_t a0 = ids[2 * l], a1 = ids[2 * l + 1];
              k0 |= (uint64_t)a0 << t->shift[l];
              k1 |= (uint64_t)a1 << t->shift[l];
              const uint32_t ntab = (uint32_t)t->alleles[l].size();
              fl |= (a0 != a1 ? 1u : 0u) << l;
              fl |= (a0 > ntab ? 1u : 0u) << (5 + l);
              fl |= (a1 > ntab ? 1u : 0u) << (10 + l);
            }
          }
          S.b_keys[2 * i] = k0;
          S.b_keys[2 * i + 1] = k1;
          S.b_flags[i] = (uint16_t)fl;
        }
        S.b_off[i] += base;
        if (!all_single) {
          const Line& ln = S.lines[i];
          if (ln.hclass == H_OK && ln.mask)
            for (int q = 0; q < L * 2; ++q) S.b_counts[i * (size_t)L * 2 + q] = ln.counts[q];
        }
      }
    }
  });
  GrimbBatch& b = S.batch;
  b.n_subjects = (int64_t)NS;
  b.typed_mask = S.b_typed.data();
  b.counts = all_single ? nullptr : S.b_counts.data();
  b.allele_off = S.b_off.data();
  b.alleles = S.b_alleles.data();
  b.n_alleles_total = (int64_t)total;
  b.prior_index = one_prior ? nullptr : S.b_prior.data();
  b.priors = S.priors.data();
  b.n_priors = (int32_t)(S.priors.size() / ((size_t)t->P * t->P));
  b.phase_mask = nullptr;   // default phase enumeration; masks are served by the numpy host front end
  b.packed_keys = packed ? S.b_keys.data() : nullptr;
  b.packed_flags = packed ? S.b_flags.data() : nullptr;
  S.sec_tok = secs(t0, clk::now());
  if (getenv("GRIMB_TEXT_TRACE") && getenv("GRIMB_TEXT_TRACE")[0] == '2')
    fprintf(stderr, "tokenise: count %.1f ms, parse %.1f ms, seq %.1f ms, fill %.1f ms\n", secs(t0, tA) * 1e3, secs(tA, tB) * 1e3,
            secs(tB, tC) * 1e3, secs(tC, clk::now()) * 1e3);
  return GRIMB_OK;
}

// results of the slot's batch -> the six texts (S.out / S.out_size), plan histogram
// `concat` false (file pipeline): the per-thread pieces stay as they are (S.fmt_parts, thread order) and the writer
// streams them out one after the other -- one copy of every output byte less
int format_slot(GrimbText* t, Slot& S, const GrimbConfig* cfg, const GrimbResults* res, bool concat = true) {
  auto t0 = clk::now();
  const size_t NS = S.lines.size();
  const int nt = t->n_threads;
  std::vector<OutStr>& parts = S.fmt_parts;
  parts.resize((size_t)nt * 6);
  for (auto& ps : parts) ps.clear();
  std::vector<int64_t> plans((size_t)nt * 4, 0);
  static const GrimbSubjectResult kNoRecord = {};   // a skipped subject: nothing was computed
  // Plan_A_Matrix with Plan B on: a subject that leaves Plan A empty-handed would enter the reference's Plan B,
  // which is not well defined under a matrix (DESIGN.md section 7) -> the call fails
  const bool guard_planb = cfg->plan_a_only && cfg->planb;
  std::vector<int64_t> undefined_first((size_t)nt, -1), undefined_n((size_t)nt, 0);
  t->parallel(NS, [&](int th, size_t lo, size_t hi) {
    OutStr* o = &parts[(size_t)th * 6];
    int64_t my_plans[4] = {0, 0, 0, 0};   // (a shared array of counters, one slot per thread, is a false-sharing trap)
    for (size_t i = lo; i < hi; ++i) {
      const Line& ln = S.lines[i];
      const uint64_t idx = (uint64_t)S.first_index + i;
      if (ln.hclass == H_PROBLEM) {
        put_uint(idx, o[GRIMB_OUT_PROBLEM]);
        o[GRIMB_OUT_PROBLEM] += ',';
        o[GRIMB_OUT_PROBLEM] += ln.sid;
        o[GRIMB_OUT_PROBLEM] += '\n';
        continue;
      }
      if (ln.hclass == H_FAULT) {
        o[GRIMB_OUT_PROBLEM] += ln.raw;
        o[GRIMB_OUT_PROBLEM] += '\n';
        continue;
      }
      const GrimbCompact& c = res->compact[i];
      if (c.status == GRIMB_ST_FAULT) {
        o[GRIMB_OUT_PROBLEM] += ln.raw;
        o[GRIMB_OUT_PROBLEM] += '\n';
        continue;
      }
      if (c.status == GRIMB_ST_NO_PHASES) {
        // nothing opens: the reference returns its defaults and the PMUG writer then raises
        if (cfg->output_pmug) {
          o[GRIMB_OUT_PROBLEM] += ln.raw;
          o[GRIMB_OUT_PROBLEM] += '\n';
        }
        continue;
      }
      const uint32_t kind = c.kind_flags & 3u;
      if (kind != GRIMB_KIND_GENERAL) {
        my_plans[GRIMB_PLAN_A] += 1;
        if (guard_planb && !(c.kind_flags & GRIMB_KIND_HAS_RESULTS)) {
          if (undefined_n[(size_t)th]++ == 0) undefined_first[(size_t)th] = (int64_t)i;
        }
        if (cfg->output_pmug && !(c.kind_flags & GRIMB_KIND_HAS_RESULTS)) {
          put_uint(idx, o[GRIMB_OUT_MISS]);
          o[GRIMB_OUT_MISS] += ',';
          o[GRIMB_OUT_MISS] += ln.sid;
          o[GRIMB_OUT_MISS] += '\n';
        }
        t->format_compact(S, ln, c, res->words, cfg, o);
        continue;
      }
      const GrimbSubjectResult& r = c.off == 0xFFFFFFFFu ? kNoRecord : res->general[c.off];
      my_plans[(cfg->output_umug ? r.plan_umug : r.plan_pmug) & 3] += 1;
      const bool pm_empty = cfg->output_pmug ? r.tot_pmug == 0 : false;
      if (guard_planb && c.status == GRIMB_ST_OK && c.off != 0xFFFFFFFFu &&
          ((cfg->output_umug && r.tot_umug == 0) || (cfg->output_pmug && r.tot_pmug == 0))) {
        if (undefined_n[(size_t)th]++ == 0) undefined_first[(size_t)th] = (int64_t)i;
      }
      if (pm_empty && r.tot_umug == 0) {
        put_uint(idx, o[GRIMB_OUT_MISS]);
        o[GRIMB_OUT_MISS] += ',';
        o[GRIMB_OUT_MISS] += ln.sid;
        o[GRIMB_OUT_MISS] += '\n';
      }
      t->format_subject(S, ln, r, res->hap_rows, res->pop_rows, cfg, o);
    }
    for (int k = 0; k < 4; ++k) plans[(size_t)th * 4 + k] = my_plans[k];
  });
  auto tR = clk::now();
  // concatenate the pieces of every output in thread order, the copies themselves in parallel
  std::vector<size_t> offs((size_t)nt * 6, 0);
  for (int k = 0; k < 6; ++k) {
    size_t n = 0;
    for (int th = 0; th < nt; ++th) {
      offs[(size_t)th * 6 + k] = n;
      n += parts[(size_t)th * 6 + k].size();
    }
    if (concat && S.out[k].size() < n) S.out[k].resize(n);   // grow-only buffer; out_size[k] carries the valid length
    S.out_size[k] = (int64_t)n;
  }
  S.fmt_threads = nt;
  if (concat)
    t->parallel((size_t)nt, [&](int, size_t lo, size_t hi) {
      for (size_t th = lo; th < hi; ++th)
        for (int k = 0; k < 6; ++k) {
          const OutStr& ps = parts[th * 6 + k];
          if (!ps.empty()) memcpy(&S.out[k][offs[th * 6 + k]], ps.data(), ps.size());
        }
    });
  for (int k = 0; k < 4; ++k) S.plan_count[k] = 0;
  for (int th = 0; th < nt; ++th)
    for (int k = 0; k < 4; ++k) S.plan_count[k] += plans[(size_t)th * 4 + k];
  S.sec_fmt = secs(t0, clk::now());
  if (getenv("GRIMB_TEXT_TRACE") && getenv("GRIMB_TEXT_TRACE")[0] == '2')
    fprintf(stderr, "format: rows %.1f ms, concatenate %.1f ms\n", secs(t0, tR) * 1e3, secs(tR, clk::now()) * 1e3);
  {
    int64_t n_undef = 0, first = -1;
    for (int th = 0; th < nt; ++th) {
      n_undef += undefined_n[(size_t)th];
      if (first < 0 && undefined_first[(size_t)th] >= 0) first = undefined_first[(size_t)th];
    }
    if (n_undef) {
      const Line& ln = S.lines[(size_t)first];
      return tfail(GRIMB_E_UNDEFINED, std::to_string(n_undef) + " subject(s) leave Plan A without a result under a Plan_A_Matrix (first: line " +
                                          std::to_string((uint64_t)S.first_index + (uint64_t)first) + ", id " + std::string(ln.sid) +
                                          "): the reference's Plan B is not well defined there; set \"planb\": false to write them to the .miss file");
    }
  }
  return GRIMB_OK;
}

// One ABI call per workspace tier.  Tier 0 takes the whole batch and its results are used straight from
// the pinned staging buffers; only when some subject overflowed its workspace (rare) are the tiers'
// results merged into one set of arrays first.  Leaves S.fin / S.totals[4] (pair evaluations) / S.retries.
int run_slot(GrimbText* t, Slot& S, GrimbEngine* const* engines, int32_t n_engines, const GrimbConfig* cfg) {
  auto t0 = clk::now();
  const GrimbBatch& b = S.batch;
  const size_t NS = (size_t)b.n_subjects;
  const int L = t->L;
  S.m_compact.clear();
  S.m_words.clear();
  S.m_general.clear();
  S.m_hap.clear();
  S.m_pop.clear();
  std::vector<uint32_t> todo;
  int64_t evals = 0;
  int64_t tot[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  S.retries = 0;
  S.totals[6] = S.totals[7] = S.totals[8] = 0;
  memset(&S.fin, 0, sizeof(S.fin));
  int rc = GRIMB_OK;
  for (int tier = 0; tier < n_engines && (tier == 0 || !todo.empty()); ++tier) {
    // gather the sub-batch (tier 0: the whole batch as is)
    GrimbBatch sb = b;
    std::vector<uint16_t> g_typed, g_counts, g_all;
    std::vector<uint32_t> g_off, g_prior;
    const size_t n = tier == 0 ? NS : todo.size();
    if (tier > 0) {
      g_typed.resize(n);
      g_counts.resize(n * (size_t)L * 2);
      g_off.resize(n + 1);
      g_prior.resize(n);
      size_t tot_al = 0;
      for (size_t k = 0; k < n; ++k) {
        const uint32_t s = todo[k];
        g_typed[k] = b.typed_mask[s];
        g_prior[k] = b.prior_index ? b.prior_index[s] : 0u;
        if (b.counts) memcpy(&g_counts[k * (size_t)L * 2], b.counts + (size_t)s * L * 2, (size_t)L * 4);
        g_off[k] = (uint32_t)tot_al;
        tot_al += b.allele_off[s + 1] - b.allele_off[s];
      }
      g_off[n] = (uint32_t)tot_al;
      g_all.resize(tot_al ? tot_al : 1);
      for (size_t k = 0; k < n; ++k) {
        const uint32_t s = todo[k];
        std::copy(b.alleles + b.allele_off[s], b.alleles + b.allele_off[s + 1], g_all.begin() + g_off[k]);
      }
      sb.n_subjects = (int64_t)n;
      sb.typed_mask = g_typed.data();
      sb.counts = b.counts ? g_counts.data() : nullptr;
      sb.allele_off = g_off.data();
      sb.alleles = g_all.data();
      sb.n_alleles_total = (int64_t)tot_al;
      sb.prior_index = g_prior.data();
      sb.packed_keys = nullptr;    // the re-issued subjects travel in the general form
      sb.packed_flags = nullptr;
    }
    // pinned, grow-only staging; capacities follow what the previous call needed per subject (+25 %)
    GrimbCompact* rc_ = (GrimbCompact*)S.hb_compact.reserve((n + 1) * sizeof(GrimbCompact));
    int64_t cap[4];
    for (int k = 0; k < 4; ++k) cap[k] = std::max<int64_t>(1024, (int64_t)((double)n * t->per_subject[k] * 1.25) + 64);
    GrimbResults r;
    for (;;) {
      r.compact = rc_;
      r.words = (uint64_t*)S.hb_words.reserve((size_t)cap[0] * 8);
      r.word_capacity = cap[0];
      r.general = (GrimbSubjectResult*)S.hb_general.reserve((size_t)cap[1] * sizeof(GrimbSubjectResult));
      r.general_capacity = cap[1];
      r.hap_rows = (GrimbHapRow*)S.hb_hap.reserve((size_t)cap[2] * sizeof(GrimbHapRow));
      r.hap_capacity = cap[2];
      r.pop_rows = (GrimbPopRow*)S.hb_pop.reserve((size_t)cap[3] * sizeof(GrimbPopRow));
      r.pop_capacity = cap[3];
      r.totals = tot;
      if (!rc_ || !r.words || !r.general || !r.hap_rows || !r.pop_rows) return tfail(GRIMB_E_NOMEM, "host staging allocation failed");
      rc = grimb_impute_host(engines[tier], cfg, &sb, &r);
      if (rc == GRIMB_E_CAPACITY) {
        for (int k = 0; k < 4; ++k) cap[k] = std::max(cap[k], tot[k]);
        continue;
      }
      if (rc) return rc;
      break;
    }
    if (tier == 0 && n > 0)
      for (int k = 0; k < 4; ++k) t->per_subject[k] = std::max(k == 1 ? 0.01 : 0.1, (double)tot[k] / (double)n);
    evals += tot[4];
    for (int k = 6; k < 9; ++k) S.totals[k] += tot[k];
    // subjects whose workspace overflowed (found in parallel: the records are only 16 bytes each)
    std::vector<std::vector<uint32_t>> again_t((size_t)t->n_threads);
    t->parallel(n, [&](int th, size_t lo, size_t hi) {
      for (size_t k = lo; k < hi; ++k)
        if (rc_[k].status == GRIMB_ST_WORKSPACE) again_t[th].push_back(tier == 0 ? (uint32_t)k : todo[k]);
    });
    std::vector<uint32_t> again;
    for (auto& v : again_t) again.insert(again.end(), v.begin(), v.end());
    if (tier == 0 && again.empty()) {
      S.fin = r;   // the usual case: format from the staging buffers
      break;
    }
    // merge this tier into the slot's arrays, re-basing the offsets
    if (tier == 0) S.m_compact.assign(rc_, rc_ + n);
    const uint32_t wbase = (uint32_t)S.m_words.size(), gbase = (uint32_t)S.m_general.size();
    const uint64_t hbase = S.m_hap.size(), pbase = S.m_pop.size();
    S.m_words.insert(S.m_words.end(), r.words, r.words + tot[0]);
    for (int64_t k = 0; k < tot[1]; ++k) {
      GrimbSubjectResult o = r.general[k];
      o.hap_off += hbase;
      o.pop_off += pbase;
      S.m_general.push_back(o);
    }
    S.m_hap.insert(S.m_hap.end(), r.hap_rows, r.hap_rows + tot[2]);
    S.m_pop.insert(S.m_pop.end(), r.pop_rows, r.pop_rows + tot[3]);
    for (size_t k = 0; k < n; ++k) {
      GrimbCompact c = rc_[k];
      if (c.status == GRIMB_ST_WORKSPACE) continue;
      if ((c.kind_flags & 3u) == GRIMB_KIND_GENERAL) {
        if (c.off != 0xFFFFFFFFu) c.off += gbase;
      } else {
        c.off += wbase;
      }
      S.m_compact[tier == 0 ? k : todo[k]] = c;
    }
    S.retries += (int64_t)again.size();
    todo.swap(again);
    S.fin.compact = S.m_compact.data();
    S.fin.words = S.m_words.data();
    S.fin.general = S.m_general.data();
    S.fin.hap_rows = S.m_hap.data();
    S.fin.pop_rows = S.m_pop.data();
  }
  if (!todo.empty()) return tfail(GRIMB_E_NOMEM, "a subject exceeds the largest workspace tier");
  S.totals[4] = evals;
  S.fin.totals = S.totals;
  S.sec_gpu = secs(t0, clk::now());
  return GRIMB_OK;
}

void fill_out(const Slot& S, GrimbTextOut* out) {
  for (int k = 0; k < 6; ++k) {
    out->data[k] = S.out[k].data();
    out->size[k] = S.out_size[k];
  }
  out->n_lines = (int64_t)S.lines.size();
  for (int k = 0; k < 4; ++k) out->plan_count[k] = S.plan_count[k];
}

}  // namespace

extern "C" int grimb_text_tokenise(GrimbText* t, const GrimbConfig* cfg, const char* text, int64_t len,
                                   int64_t first_line_index, GrimbBatch* b) {
  if (!t || !cfg || !text || !b || len < 0) return tfail(GRIMB_E_ARG, "null argument");
  int rc = tokenise_slot(t, t->slot0, cfg, text, len, first_line_index, false);
  if (rc) return rc;
  *b = t->slot0.batch;
  return GRIMB_OK;
}

extern "C" int grimb_text_format(GrimbText* t, const GrimbConfig* cfg, const GrimbResults* res, GrimbTextOut* out) {
  if (!t || !cfg || !res || !out || !res->compact) return tfail(GRIMB_E_ARG, "null argument");
  int rc = format_slot(t, t->slot0, cfg, res);
  if (rc) return rc;
  fill_out(t->slot0, out);
  out->pair_evals = res->totals ? res->totals[4] : 0;
  return GRIMB_OK;
}

extern "C" int grimb_impute_text(GrimbText* t, GrimbEngine* const* engines, int32_t n_engines, const GrimbConfig* cfg,
                                 const char* text, int64_t len, int64_t first_line_index, GrimbTextOut* out) {
  if (!t || !engines || n_engines < 1 || !cfg || !text || !out || len < 0) return tfail(GRIMB_E_ARG, "null argument");
  Slot& S = t->slot0;
  int rc = tokenise_slot(t, S, cfg, text, len, first_line_index, true);   // `text` outlives this call
  if (rc) return rc;
  rc = run_slot(t, S, engines, n_engines, cfg);
  if (rc) return rc;
  rc = format_slot(t, S, cfg, &S.fin);
  if (rc) return rc;
  fill_out(S, out);
  out->pair_evals = S.totals[4];
  out->workspace_retries = S.retries;
  out->seconds_tokenise = S.sec_tok;
  out->seconds_gpu = S.sec_gpu;
  out->seconds_format = S.sec_fmt;
  return GRIMB_OK;
}

// ------------------------------------------------------------------------------------------
// File pipeline: what Imputation.impute_file (reference impute.py:1985-2155) does for a whole
// input file, as four overlapped stages over chunks of lines -- tokenise(c+1) | GPU(c) |
// format(c-1) | write(c-2) -- each on its own host thread (the tokeniser and the formatter fan out
// over worker threads themselves).  The input is memory-mapped, never copied.
// ------------------------------------------------------------------------------------------
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <condition_variable>
#include <deque>
#include <memory>
#include <mutex>

namespace {

struct Channel {   // a small blocking queue of slot indices; -1 closes it
  std::mutex m;
  std::condition_variable cv;
  std::deque<int> q;
  void push(int v) {
    {
      std::lock_guard<std::mutex> g(m);
      q.push_back(v);
    }
    cv.notify_one();
  }
  int pop() {
    std::unique_lock<std::mutex> g(m);
    cv.wait(g, [&] { return !q.empty(); });
    int v = q.front();
    q.pop_front();
    return v;
  }
};

bool write_all(int fd, const char* p, size_t n) {
  while (n) {
    ssize_t w = write(fd, p, n);
    if (w < 0) {
      if (errno == EINTR) continue;
      return false;
    }
    p += w;
    n -= (size_t)w;
  }
  return true;
}

// first line start at or after `pos` (a line starts at 0 or right after a '\n')
size_t line_start_at(const char* p, size_t n, size_t pos) {
  if (pos == 0) return 0;
  if (pos >= n) return n;
  const void* q = memchr(p + pos - 1, '\n', n - (pos - 1));
  return q ? (size_t)((const char*)q - p) + 1 : n;
}

// ---- sharing one input file between the ranks of a host (grimb_impute_file_sharded) ------------------------
// The ranks take the input's chunks round-robin (chunk c -> rank c % world) and meet on a small board in a
// memory-mapped file: per chunk its line count (published after tokenising: the formatter of a later chunk needs
// the global index of its first line for the .miss / .problem rows) and the sizes of its six output pieces
// (published after formatting: the writer of a later chunk needs its file offsets).  Every rank streams its
// pieces straight into the final files with pwrite -- nothing is accumulated, gathered or written afterwards.
struct Board {
  int64_t* p = nullptr;
  size_t bytes = 0;
  int64_t n_chunks = 0;
  int rank = 0, world = 1;
  static constexpr int64_t MAGIC = 0x4752494d42424f41ll;
  enum { HDR = 8, ENT = 16, F_LINES_READY = 0, F_LINES = 1, F_SIZES_READY = 2, F_SIZE0 = 3 };
  int64_t* ent(int64_t c) const { return p + HDR + ENT * c; }
  void fail() const { __atomic_store_n(p + 2, (int64_t)1, __ATOMIC_RELEASE); }
  bool failed() const { return __atomic_load_n(p + 2, __ATOMIC_ACQUIRE) != 0; }
  void publish(int64_t c, int ready_field) const { __atomic_store_n(ent(c) + ready_field, (int64_t)1, __ATOMIC_RELEASE); }
  // waits until chunk c has published `ready_field`; false: another rank failed, or nothing happened for 10 minutes
  bool wait(int64_t c, int ready_field) const {
    auto t0 = clk::now();
    for (unsigned spin = 0;; ++spin) {
      if (__atomic_load_n(ent(c) + ready_field, __ATOMIC_ACQUIRE) != 0) return true;
      if (failed()) return false;
      if (spin > 200) {
        std::this_thread::sleep_for(std::chrono::microseconds(50));
        if ((spin & 1023) == 0 && secs(t0, clk::now()) > 600.0) return false;
      }
    }
  }
};

bool pwrite_all(int fd, const char* p, size_t n, int64_t off) {
  while (n) {
    ssize_t w = pwrite(fd, p, n, (off_t)off);
    if (w < 0) {
      if (errno == EINTR) continue;
      return false;
    }
    p += w;
    n -= (size_t)w;
    off += w;
  }
  return true;
}

int impute_file_impl(GrimbText* t, GrimbEngine* const* engines, int32_t n_engines, const GrimbConfig* cfg, const char* in_path,
                     int64_t byte_lo, int64_t byte_hi, int64_t first_line_index, const char* const* out_paths, int64_t chunk_bytes,
                     GrimbTextOut* out, GrimbFileStats* stats, const Board* board);

}  // namespace

extern "C" int grimb_file_count_lines(const char* path, int64_t byte_lo, int64_t byte_hi, int32_t n_threads,
                                      int64_t* n_lines, int64_t* lo_adj, int64_t* hi_adj) {
  if (!path || !n_lines) return tfail(GRIMB_E_ARG, "null argument");
  int fd = open(path, O_RDONLY);
  if (fd < 0) return tfail(GRIMB_E_ARG, std::string("cannot open ") + path);
  struct stat st;
  if (fstat(fd, &st) != 0) {
    close(fd);
    return tfail(GRIMB_E_ARG, "fstat failed");
  }
  const size_t n = (size_t)st.st_size;
  *n_lines = 0;
  if (lo_adj) *lo_adj = 0;
  if (hi_adj) *hi_adj = 0;
  if (n == 0) {
    close(fd);
    return GRIMB_OK;
  }
  const char* p = (const char*)mmap(nullptr, n, PROT_READ, MAP_PRIVATE, fd, 0);
  close(fd);
  if (p == MAP_FAILED) return tfail(GRIMB_E_NOMEM, "mmap failed");
  const size_t lo = line_start_at(p, n, (size_t)std::max<int64_t>(0, byte_lo));
  const size_t hi = byte_hi < 0 || (size_t)byte_hi >= n ? n : line_start_at(p, n, (size_t)byte_hi);
  int nt = n_threads > 0 ? n_threads : (int)std::max(1u, std::thread::hardware_concurrency());
  std::vector<int64_t> cnt((size_t)nt, 0);
  std::vector<std::thread> th;
  for (int k = 0; k < nt; ++k)
    th.emplace_back([&, k]() {
      const size_t a = lo + (hi - lo) * (size_t)k / (size_t)nt, b = lo + (hi - lo) * (size_t)(k + 1) / (size_t)nt;
      int64_t c = 0;
      const char* q = p + a;
      const char* e = p + b;
      while (q < e) {
        const void* f = memchr(q, '\n', (size_t)(e - q));
        if (!f) break;
        ++c;
        q = (const char*)f + 1;
      }
      cnt[k] = c;
    });
  for (auto& x : th) x.join();
  int64_t total = 0;
  for (int64_t c : cnt) total += c;
  if (hi > lo && p[hi - 1] != '\n') ++total;   // an unterminated last line
  munmap((void*)p, n);
  *n_lines = total;
  if (lo_adj) *lo_adj = (int64_t)lo;
  if (hi_adj) *hi_adj = (int64_t)hi;
  return GRIMB_OK;
}

extern "C" int grimb_file_write_at(const char* path, int64_t offset, const void* data, int64_t size) {
  if (!path || (!data && size) || offset < 0 || size < 0) return tfail(GRIMB_E_ARG, "bad argument");
  int fd = open(path, O_WRONLY | O_CREAT, 0644);
  if (fd < 0) return tfail(GRIMB_E_ARG, std::string("cannot open ") + path);
  const char* p = (const char*)data;
  int64_t done = 0;
  while (done < size) {
    ssize_t w = pwrite(fd, p + done, (size_t)(size - done), (off_t)(offset + done));
    if (w < 0) {
      if (errno == EINTR) continue;
      close(fd);
      return tfail(GRIMB_E_ARG, std::string("write failed: ") + path);
    }
    done += w;
  }
  close(fd);
  return GRIMB_OK;
}

extern "C" int grimb_impute_file(GrimbText* t, GrimbEngine* const* engines, int32_t n_engines, const GrimbConfig* cfg,
                                 const char* in_path, int64_t byte_lo, int64_t byte_hi, int64_t first_line_index,
                                 const char* const* out_paths, int64_t chunk_bytes, GrimbTextOut* out, GrimbFileStats* stats) {
  return impute_file_impl(t, engines, n_engines, cfg, in_path, byte_lo, byte_hi, first_line_index, out_paths, chunk_bytes, out,
                          stats, nullptr);
}

// Size of the board file for an input of `file_bytes` cut into chunks of `chunk_bytes`; rank 0 creates the file
// zero-filled before the ranks call grimb_impute_file_sharded.
extern "C" int64_t grimb_file_board_bytes(int64_t file_bytes, int64_t chunk_bytes) {
  if (chunk_bytes <= 0) chunk_bytes = 16 << 20;
  const int64_t n = (file_bytes + chunk_bytes - 1) / chunk_bytes;
  return (int64_t)sizeof(int64_t) * (Board::HDR + Board::ENT * (n > 0 ? n : 1));
}

extern "C" int grimb_impute_file_sharded(GrimbText* t, GrimbEngine* const* engines, int32_t n_engines, const GrimbConfig* cfg,
                                         const char* in_path, const char* const* out_paths, int64_t chunk_bytes, int32_t rank,
                                         int32_t world, const char* board_path, GrimbFileStats* stats) {
  if (!board_path || !out_paths || rank < 0 || world < 1 || rank >= world || !stats) return tfail(GRIMB_E_ARG, "bad shard arguments");
  if (chunk_bytes <= 0) chunk_bytes = 16 << 20;
  int fd = open(board_path, O_RDWR);
  if (fd < 0) return tfail(GRIMB_E_ARG, std::string("cannot open the board ") + board_path);
  struct stat st;
  if (fstat(fd, &st) != 0 || (size_t)st.st_size < sizeof(int64_t) * (Board::HDR + Board::ENT)) {
    close(fd);
    return tfail(GRIMB_E_ARG, "board file too small");
  }
  Board b;
  b.bytes = (size_t)st.st_size;
  b.p = (int64_t*)mmap(nullptr, b.bytes, PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
  close(fd);
  if (b.p == MAP_FAILED) return tfail(GRIMB_E_NOMEM, "mmap of the board failed");
  b.rank = rank;
  b.world = world;
  GrimbTextOut out;
  int rc = impute_file_impl(t, engines, n_engines, cfg, in_path, 0, -1, 0, out_paths, chunk_bytes, &out, stats, &b);
  if (rc != GRIMB_OK) b.fail();
  munmap(b.p, b.bytes);
  return rc;
}

namespace {
int impute_file_impl(GrimbText* t, GrimbEngine* const* engines, int32_t n_engines, const GrimbConfig* cfg, const char* in_path,
                     int64_t byte_lo, int64_t byte_hi, int64_t first_line_index, const char* const* out_paths, int64_t chunk_bytes,
                     GrimbTextOut* out, GrimbFileStats* stats, const Board* board) {
  if (!t || !engines || n_engines < 1 || !cfg || !in_path || !out || !stats) return tfail(GRIMB_E_ARG, "null argument");
  auto t_begin = clk::now();
  memset(stats, 0, sizeof(*stats));
  memset(out, 0, sizeof(*out));
  int fd = open(in_path, O_RDONLY);
  if (fd < 0) return tfail(GRIMB_E_ARG, std::string("cannot open ") + in_path);
  struct stat st;
  if (fstat(fd, &st) != 0) {
    close(fd);
    return tfail(GRIMB_E_ARG, "fstat failed");
  }
  const size_t fsize = (size_t)st.st_size;
  const char* base = nullptr;
  if (fsize) {
    base = (const char*)mmap(nullptr, fsize, PROT_READ, MAP_PRIVATE, fd, 0);
    if (base == MAP_FAILED) {
      close(fd);
      return tfail(GRIMB_E_NOMEM, "mmap of the input failed");
    }
    madvise((void*)base, fsize, MADV_SEQUENTIAL);
  }
  close(fd);
  const size_t lo = fsize ? line_start_at(base, fsize, (size_t)std::max<int64_t>(0, byte_lo)) : 0;
  const size_t hi = !fsize ? 0 : (byte_hi < 0 || (size_t)byte_hi >= fsize ? fsize : line_start_at(base, fsize, (size_t)byte_hi));
  // outputs: a path = streamed to that file (created / truncated here); NULL = kept in memory and returned
  int ofd[6];
  // An output file left by an earlier run is moved aside and deleted in the background: truncating a large
  // file in place frees its page-cache pages synchronously (0.3 s for the 1.4 GB of a 4M-subject run).
  std::vector<std::string> old_files;
  for (int k = 0; k < 6; ++k) {
    ofd[k] = -1;
    t->file_acc[k].clear();
    if (board && out_paths && out_paths[k]) {
      ofd[k] = open(out_paths[k], O_WRONLY);
      if (ofd[k] < 0) {
        for (int j = 0; j < k; ++j)
          if (ofd[j] >= 0) close(ofd[j]);
        if (fsize) munmap((void*)base, fsize);
        return tfail(GRIMB_E_ARG, std::string("cannot open ") + out_paths[k]);
      }
      continue;
    }
    if (out_paths && out_paths[k]) {
      struct stat ost;
      if (stat(out_paths[k], &ost) == 0 && S_ISREG(ost.st_mode) && ost.st_size > (1 << 20) && ost.st_nlink == 1) {
        std::string aside = std::string(out_paths[k]) + ".old." + std::to_string((long long)getpid());
        if (rename(out_paths[k], aside.c_str()) == 0) old_files.push_back(aside);
      }
      ofd[k] = open(out_paths[k], O_WRONLY | O_CREAT | O_TRUNC, 0644);
      if (ofd[k] < 0) {
        for (int j = 0; j < k; ++j)
          if (ofd[j] >= 0) close(ofd[j]);
        if (fsize) munmap((void*)base, fsize);
        for (const std::string& f : old_files) unlink(f.c_str());
        return tfail(GRIMB_E_ARG, std::string("cannot create ") + out_paths[k]);
      }
    }
  }
  if (chunk_bytes <= 0) chunk_bytes = 16 << 20;
  constexpr int NSLOT = 4;
  if (t->pipe.size() < (size_t)NSLOT)
    for (size_t k = t->pipe.size(); k < (size_t)NSLOT; ++k) t->pipe.emplace_back(new Slot());
  Channel free_q, to_gpu, to_fmt, to_write;
  for (int k = 0; k < NSLOT; ++k) free_q.push(k);
  std::mutex err_m;
  int err_rc = GRIMB_OK;
  std::string err_msg;
  auto set_err = [&](int rc) {
    std::lock_guard<std::mutex> g(err_m);
    if (err_rc == GRIMB_OK) {
      err_rc = rc;
      err_msg = grimb_last_error();   // the failing thread's message
    }
    if (board) board->fail();         // the other ranks stop waiting for this one's chunks
  };
  auto failed = [&]() {
    std::lock_guard<std::mutex> g(err_m);
    return err_rc != GRIMB_OK;
  };
  double s_tok = 0, s_gpu = 0, s_fmt = 0, s_wr = 0;
  std::thread th_old([&]() {
    for (const std::string& f : old_files) unlink(f.c_str());
  });
  const int64_t n_chunks = board ? (int64_t)((fsize + (size_t)chunk_bytes - 1) / (size_t)chunk_bytes) : 0;
  if (board && (int64_t)(board->bytes / sizeof(int64_t)) < Board::HDR + Board::ENT * (n_chunks > 0 ? n_chunks : 1)) {
    for (int k = 0; k < 6; ++k)
      if (ofd[k] >= 0) close(ofd[k]);
    if (fsize) munmap((void*)base, fsize);
    return tfail(GRIMB_E_ARG, "board file too small for this input / chunk size");
  }
  std::thread th_tok([&]() {
    if (board) {
      // chunk c = bytes [c * chunk_bytes, (c + 1) * chunk_bytes), both ends moved to the next line start
      for (int64_t c = board->rank; c < n_chunks && !failed() && !board->failed(); c += board->world) {
        const size_t pos = line_start_at(base, fsize, (size_t)c * (size_t)chunk_bytes);
        const size_t e = c + 1 >= n_chunks ? fsize : line_start_at(base, fsize, (size_t)(c + 1) * (size_t)chunk_bytes);
        if (e <= pos) {   // a line longer than a chunk: nothing starts here
          int64_t* en = board->ent(c);
          for (int q = 0; q < Board::ENT; ++q) en[q] = 0;
          board->publish(c, Board::F_LINES_READY);
          board->publish(c, Board::F_SIZES_READY);
          continue;
        }
        const int k = free_q.pop();
        Slot& S = *t->pipe[(size_t)k];
        int rc = tokenise_slot(t, S, cfg, base + pos, (int64_t)(e - pos), 0, true);
        if (rc) {
          set_err(rc);
          free_q.push(k);
          break;
        }
        S.chunk_id = c;
        board->ent(c)[Board::F_LINES] = (int64_t)S.lines.size();
        board->publish(c, Board::F_LINES_READY);
        s_tok += S.sec_tok;
        to_gpu.push(k);
      }
      to_gpu.push(-1);
      return;
    }
    size_t pos = lo;
    int64_t first = first_line_index;
    while (pos < hi && !failed()) {
      size_t e = pos + (size_t)chunk_bytes;
      e = e >= hi ? hi : line_start_at(base, fsize, e);
      if (e > hi) e = hi;
      const int k = free_q.pop();
      Slot& S = *t->pipe[(size_t)k];
      int rc = tokenise_slot(t, S, cfg, base + pos, (int64_t)(e - pos), first, true);
      if (rc) {
        set_err(rc);
        free_q.push(k);
        break;
      }
      s_tok += S.sec_tok;
      first += (int64_t)S.lines.size();
      pos = e;
      to_gpu.push(k);
    }
    to_gpu.push(-1);
  });
  std::thread th_gpu([&]() {
    for (;;) {
      const int k = to_gpu.pop();
      if (k < 0) break;
      Slot& S = *t->pipe[(size_t)k];
      if (!failed()) {
        int rc = run_slot(t, S, engines, n_engines, cfg);
        if (rc) set_err(rc);
        s_gpu += S.sec_gpu;
      }
      to_fmt.push(k);
    }
    to_fmt.push(-1);
  });
  std::thread th_fmt([&]() {
    int64_t line_cursor = 0, next_c = 0;   // board: lines of the chunks [0, next_c)
    for (;;) {
      const int k = to_fmt.pop();
      if (k < 0) break;
      Slot& S = *t->pipe[(size_t)k];
      if (!failed()) {
        if (board) {
          for (; next_c < S.chunk_id && !failed(); ++next_c) {
            if (!board->wait(next_c, Board::F_LINES_READY)) {
              tfail(GRIMB_E_ARG, "another rank failed (or stalled) before publishing its line counts");
              set_err(GRIMB_E_ARG);
              break;
            }
            line_cursor += board->ent(next_c)[Board::F_LINES];
          }
          S.first_index = line_cursor;
          line_cursor += (int64_t)S.lines.size();
          next_c = S.chunk_id + 1;
        }
        if (!failed()) {
          int rc = format_slot(t, S, cfg, &S.fin, false);
          if (rc) set_err(rc);
          s_fmt += S.sec_fmt;
        }
        if (board && !failed()) {
          for (int o = 0; o < 6; ++o) board->ent(S.chunk_id)[Board::F_SIZE0 + o] = S.out_size[o];
          board->publish(S.chunk_id, Board::F_SIZES_READY);
        }
      }
      to_write.push(k);
    }
    to_write.push(-1);
  });
  std::thread th_wr([&]() {
    int64_t off_cursor[6] = {0, 0, 0, 0, 0, 0}, next_c = 0;   // board: output bytes of the chunks [0, next_c)
    for (;;) {
      const int k = to_write.pop();
      if (k < 0) break;
      Slot& S = *t->pipe[(size_t)k];
      if (board && !failed()) {
        for (; next_c < S.chunk_id && !failed(); ++next_c) {
          if (!board->wait(next_c, Board::F_SIZES_READY)) {
            tfail(GRIMB_E_ARG, "another rank failed (or stalled) before publishing its output sizes");
            set_err(GRIMB_E_ARG);
            break;
          }
          for (int o = 0; o < 6; ++o) off_cursor[o] += board->ent(next_c)[Board::F_SIZE0 + o];
        }
      }
      if (!failed()) {
        auto w0 = clk::now();
        // the six outputs of the chunk in parallel: streamed to their files, or appended in memory
        std::vector<std::thread> ws;
        bool ok[6] = {true, true, true, true, true, true};
        for (int o = 0; o < 6; ++o) {
          if (S.out_size[o] == 0) continue;
          ws.emplace_back([&, o]() {
            int64_t at = off_cursor[o];
            for (int th = 0; th < S.fmt_threads && ok[o]; ++th) {   // the formatter's pieces, in thread order
              const OutStr& ps = S.fmt_parts[(size_t)th * 6 + o];
              if (ps.empty()) continue;
              if (board && ofd[o] >= 0) ok[o] = pwrite_all(ofd[o], ps.data(), ps.size(), at);
              else if (ofd[o] >= 0) ok[o] = write_all(ofd[o], ps.data(), ps.size());
              else t->file_acc[o].append(ps.data(), ps.size());
              at += (int64_t)ps.size();
            }
          });
        }
        for (auto& x : ws) x.join();
        for (int o = 0; o < 6; ++o)
          if (!ok[o]) {
            tfail(GRIMB_E_ARG, "write to an output file failed");
            set_err(GRIMB_E_ARG);
          }
        stats->n_lines += (int64_t)S.lines.size();
        stats->pair_evals += S.totals[4];
        stats->workspace_retries += S.retries;
        for (int q = 0; q < 4; ++q) stats->plan_count[q] += S.plan_count[q];
        for (int o = 0; o < 6; ++o) stats->out_bytes[o] += S.out_size[o];
        stats->n_chunks += 1;
        s_wr += secs(w0, clk::now());
        if (board) {
          for (int o = 0; o < 6; ++o) off_cursor[o] += S.out_size[o];
          next_c = S.chunk_id + 1;
        }
      }
      free_q.push(k);
    }
  });
  th_tok.join();
  th_gpu.join();
  th_fmt.join();
  th_wr.join();
  th_old.join();
  for (int k = 0; k < 6; ++k)
    if (ofd[k] >= 0) close(ofd[k]);
  if (fsize) munmap((void*)base, fsize);
  if (err_rc != GRIMB_OK) return tfail(err_rc, err_msg);
  for (int k = 0; k < 6; ++k) {
    out->data[k] = t->file_acc[k].data();
    out->size[k] = ofd[k] >= 0 ? 0 : (int64_t)t->file_acc[k].size();
  }
  out->n_lines = stats->n_lines;
  out->pair_evals = stats->pair_evals;
  out->workspace_retries = stats->workspace_retries;
  for (int q = 0; q < 4; ++q) out->plan_count[q] = stats->plan_count[q];
  out->seconds_tokenise = stats->seconds_tokenise = s_tok;
  out->seconds_gpu = stats->seconds_gpu = s_gpu;
  out->seconds_format = stats->seconds_format = s_fmt;
  stats->seconds_write = s_wr;
  stats->in_bytes = (int64_t)(hi - lo);
  stats->seconds_total = secs(t_begin, clk::now());
  if (getenv("GRIMB_TEXT_TRACE"))
    fprintf(stderr, "impute_file: %lld lines, %lld chunks, %.3f s wall; busy: tokenise %.3f, gpu %.3f, format %.3f, write %.3f s\n",
            (long long)stats->n_lines, (long long)stats->n_chunks, stats->seconds_total, s_tok, s_gpu, s_fmt, s_wr);
  return GRIMB_OK;
}
}  // namespace
