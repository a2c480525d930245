// grimb200.cu -- libgrimb200.so: C ABI (include/grimb200.h), device table build (K0) and the
// imputation kernel launcher.  Compile for sm_100a with -fmad=false (FP64 operation order must
// match the reference's Python floats; see grimb_subject.h).
#include <cuda_runtime.h>
#include <cub/cub.cuh>

#include <chrono>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "grimb_plan.h"

using namespace grimb;

// ------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------
static thread_local std::string g_err;
static int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define CK(call)                                                                          \
  do {                                                                                    \
    cudaError_t e_ = (call);                                                              \
    if (e_ != cudaSuccess)                                                                \
      return fail(GRIMB_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));      \
  } while (0)

extern "C" int grimb_abi_version(void) { return GRIMB_ABI_VERSION; }

// page-locked host staging for the text pipeline (internal; nullptr when there is no device)
extern "C" void* grimb_pinned_alloc(size_t bytes) {
  void* p = nullptr;
  if (cudaMallocHost(&p, bytes) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return p;
}
extern "C" void grimb_pinned_free(void* p) {
  if (p) cudaFreeHost(p);
}
extern "C" const char* grimb_last_error(void) { return g_err.c_str(); }
// the text pipeline (grimb_text.cpp) reports through the same per-thread message
extern "C" void grimb_set_error(const char* msg) { g_err = msg ? msg : ""; }

// ------------------------------------------------------------------------------------------
// table image: one device allocation = header + arrays (so one broadcast replicates it)
// ------------------------------------------------------------------------------------------
struct ImageHeader {
  uint64_t magic;
  int32_t L, P;
  uint32_t n_nodes, n_full;
  uint8_t shift[9];
  uint8_t width[9];
  uint32_t n_alleles[9];
  uint64_t n_toplinks, n_conn_edges, n_slots, bytes;
  // byte offsets from the image base
  uint64_t o_label_first, o_label_count, o_ht_off, o_ht_mask, o_slots, o_node_key, o_freq, o_tl_start,
      o_tl_cnt, o_tl_adj, o_cn_start, o_cn_cnt, o_cn_adj;
};
static const uint64_t IMAGE_MAGIC = 0x4752494d42323030ULL + (GRIMB_KW - 1);  // "GRIMB200" (+1: 128-bit keys)

struct GrimbTables {
  int device;
  char* image;  // device
  ImageHeader h;
  TablesView view;
  int build_launches = 0;   // kernel launches of grimb_tables_build (0 for a table made from an image)
  float build_ms = 0.0f;    // device time of the build after the inputs were staged (CUDA events on the build's stream)
#if GRIMB_KW == 1
  char* fidx_mem = nullptr;   // FastIndex keys + fslot (derived from the image; tables the fast path serves only)
  uint64_t fidx_bytes = 0;
  FastIndex fidx = {nullptr, nullptr, 0};
#endif
};

static void make_view(GrimbTables* t) {
  const ImageHeader& h = t->h;
  TablesView& v = t->view;
  v.L = h.L;
  v.P = h.P;
  v.n_nodes = h.n_nodes;
  v.n_full = h.n_full;
  memcpy(v.shift, h.shift, 9);
  memcpy(v.width, h.width, 9);
  memcpy(v.n_alleles, h.n_alleles, sizeof(h.n_alleles));
  char* b = t->image;
  v.label_first = (const uint32_t*)(b + h.o_label_first);
  v.label_count = (const uint32_t*)(b + h.o_label_count);
  v.ht_off = (const uint64_t*)(b + h.o_ht_off);
  v.ht_mask = (const uint32_t*)(b + h.o_ht_mask);
  v.slots = (const HSlot*)(b + h.o_slots);
  v.node_key = (const hkey*)(b + h.o_node_key);
  v.freq = (const double*)(b + h.o_freq);
  v.tl_start = (const uint32_t*)(b + h.o_tl_start);
  v.tl_cnt = (const uint32_t*)(b + h.o_tl_cnt);
  v.tl_adj = (const uint32_t*)(b + h.o_tl_adj);
  v.cn_start = (const uint32_t*)(b + h.o_cn_start);
  v.cn_cnt = (const uint32_t*)(b + h.o_cn_cnt);
  v.cn_adj = (const uint32_t*)(b + h.o_cn_adj);
}

// ------------------------------------------------------------------------------------------
// K0: table build kernels
// ------------------------------------------------------------------------------------------
__global__ void k_pack_full(const uint16_t* al, int L, const uint8_t* shift, uint64_t n, hkey* keys) {
  uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  hkey k = 0;
  for (int l = 0; l < L; ++l) k |= (hkey)al[i * L + l] << shift[l];
  keys[i] = k;
}

__global__ void k_full_nodes(const hkey* keys, const double* full_freq, uint32_t n, int P, hkey* node_key,
                             double* freq, uint32_t* tl_start, uint32_t* tl_cnt) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  node_key[i] = keys[i];
  tl_start[i] = 0;
  tl_cnt[i] = 0;
  for (int p = 0; p < P; ++p) freq[(uint64_t)i * P + p] = full_freq[(uint64_t)i * P + p];
}

__global__ void k_init_slots(HSlot* s, uint64_t n) {
  uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  HSlot e;
  memset(&e, 0, sizeof(e));
  e.key = ~(hkey)0;
  e.node = GRIMB_NONE;
  s[i] = e;
}

static inline unsigned nblk(uint64_t n, unsigned t = 256) { return (unsigned)((n + t - 1) / t); }

#if GRIMB_KW == 1
// FastIndex insert: one thread per full haplotype (node ids [0, n_full): the full label comes first).
// A key takes the first empty slot from its home sector on; one stored past its home sector sets the
// home sector's flag.  Sectors never empty again, so every sector between a key's home and its slot is
// full: a lookup may stop at the first sector with an empty slot.
__global__ void k_fast_index(const hkey* __restrict__ node_key, const double* __restrict__ freq, uint32_t n,
                             unsigned long long* keys, double* fslot, uint32_t sec_mask) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double f = freq[i];   // P == 1
  if (!(f > 0)) return;       // the fast path treats f == 0 as absent
  const unsigned long long key = node_key[i];
  const uint32_t home = hash_key(key) & sec_mask;
  for (uint32_t sec = home;; sec = (sec + 1) & sec_mask) {
    unsigned long long* w = keys + 4ull * sec;
    for (int j = 0; j < 4; ++j) {
      // the first word of a sector may carry the flag: it is empty with the flag either way
      unsigned long long flag = 0, old;
      while ((old = atomicCAS(w + j, flag, flag | key)) != flag) {
        if (j != 0 || (old & ~FIDX_FLAG) != 0) break;   // taken
        flag = old;                                      // only the flag was set meanwhile
      }
      if (old == flag) {
        fslot[4ull * sec + j] = f;
        if (sec != home) atomicOr(keys + 4ull * home, FIDX_FLAG);
        return;
      }
    }
  }
}

// Builds t->fidx for a table the single-population fast path serves (L <= 5, P == 1); nothing otherwise.
// GRIMB_FAST_INDEX_MULT (2..16) sets the slots per full haplotype.  Default 4: on B200 the 1M-haplotype table's
// probe kernel takes the same time with 4 (32 MB of keys) as with 8 (64 MB), at half the memory.
static cudaError_t build_fast_index(GrimbTables* t, int* launches) {
  const ImageHeader& h = t->h;
  if (h.L > 5 || h.P != 1) return cudaSuccess;
  if (h.n_full > (1u << 30)) return cudaErrorInvalidValue;   // slot positions are 32-bit, load <= 1/2
  uint64_t mult = 4;
  if (const char* m = getenv("GRIMB_FAST_INDEX_MULT")) {
    const long v = atol(m);
    if (v >= 2 && v <= 16) mult = (uint64_t)v;
  }
  uint64_t n_slots = 4;
  while (n_slots < mult * h.n_full && n_slots < (1ull << 31)) n_slots <<= 1;
  cudaError_t e = cudaMalloc((void**)&t->fidx_mem, n_slots * 16);
  if (e != cudaSuccess) {
    t->fidx_mem = nullptr;
    return e;
  }
  t->fidx_bytes = n_slots * 16;
  unsigned long long* keys = (unsigned long long*)t->fidx_mem;
  double* fslot = (double*)(t->fidx_mem + n_slots * 8);
  t->fidx.keys = (const uint64_t*)keys;
  t->fidx.fslot = fslot;
  t->fidx.sec_mask = (uint32_t)(n_slots / 4 - 1);
  e = cudaMemsetAsync(keys, 0, n_slots * 8, 0);
  if (e != cudaSuccess) return e;
  if (h.n_full) {
    k_fast_index<<<nblk(h.n_full), 256>>>(t->view.node_key, t->view.freq, h.n_full, keys, fslot, t->fidx.sec_mask);
    if (launches) ++*launches;
  }
  return cudaGetLastError();
}
#endif

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    cudaError_t e = cudaMalloc(&p, bytes ? bytes : 16);
    if (e == cudaSuccess) cap = bytes;
    return e;
  }
  ~DevBuf() {
    if (p) cudaFree(p);
  }
};

static std::vector<uint32_t> label_order(int L) {
  // full label, then subsets of decreasing size in itertools.combinations order
  // (generate_neo4j_multi_hpf.py:105-110)
  std::vector<uint32_t> out;
  out.push_back((1u << L) - 1u);
  for (int r = L - 1; r >= 1; --r) {
    std::vector<int> c(r);
    for (int i = 0; i < r; ++i) c[i] = i;
    for (;;) {
      uint32_t m = 0;
      for (int i = 0; i < r; ++i) m |= 1u << c[i];
      out.push_back(m);
      int i = r - 1;
      while (i >= 0 && c[i] == L - r + i) --i;
      if (i < 0) break;
      ++c[i];
      for (int j = i + 1; j < r; ++j) c[j] = c[j - 1] + 1;
    }
  }
  return out;
}

// reference quirk: the closing CSR sentinel is len(Vertices) (networkx_graph.py:195-196)
static uint32_t sentinel_count(uint64_t own, uint64_t n_edges, uint64_t n_vertices) {
  uint64_t start = n_edges - own;
  if (n_vertices <= start) return 0;
  if (n_vertices > n_edges) return GRIMB_ADJ_FAULT;
  return (uint32_t)(n_vertices - start);
}

// ------------------------------------------------------------------------------------------
// K0: table build, batched over labels.  All marginal labels are grouped with ONE stable sort-by-key:
// element (label li, full haplotype i) carries the composite key  li || projected haplotype  (the
// projection re-packed at minimal field widths so that the composite usually fits 64 bits; two LSD
// passes over 64-bit words otherwise).  Equal keys stay in hpf order, so a segment's first member is
// the node's first appearance, its members in sorted order are its top links (ascending full id), and
// the ordered segmented sum adds the members' frequency vectors exactly as
// generate_neo4j_multi_hpf.py:405 does.  Node ids follow from a second sort of the segments by
// (label, first member).  Connectors are grouped the same way, one element per (parent label B, dropped
// locus l, node of B).  Large tables are processed in groups of labels / pairs of bounded size.
// ------------------------------------------------------------------------------------------
struct CompactLayout {
  uint8_t cshift[9];
  uint8_t cwidth[9];
  int32_t cbits;
};

typedef unsigned __int128 u128;

__device__ __forceinline__ u128 compact_of(hkey key, const uint8_t* shift, const uint8_t* width, const CompactLayout& C, int L,
                                           uint32_t label) {
  u128 c = 0;
  for (int l = 0; l < L; ++l)
    if (label >> l & 1u) c |= (u128)((uint64_t)(key >> shift[l]) & ((1ull << width[l]) - 1ull)) << C.cshift[l];
  return c;
}

struct K0Meta {   // small per-build tables, device resident
  uint32_t label_mask[512];   // label index (build order) -> locus mask
};

// elements of one group of labels [li0, li0 + nl): e -> (li0 + e / N, e % N)
__global__ void k0_make_keys(const hkey* __restrict__ full_keys, TablesView T, CompactLayout C, const uint32_t* __restrict__ label_mask,
                             uint32_t li0, uint64_t N, uint64_t E, uint64_t* lo, uint64_t* hi, uint32_t* val) {
  const uint64_t e = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (e >= E) return;
  const uint32_t li = li0 + (uint32_t)(e / N);
  const uint32_t i = (uint32_t)(e % N);
  const u128 c = ((u128)li << C.cbits) | compact_of(full_keys[i], T.shift, T.width, C, T.L, label_mask[li]);
  lo[e] = (uint64_t)c;
  if (hi) hi[e] = (uint64_t)(c >> 64);
  val[e] = i;
}

__global__ void k0_gather64(const uint64_t* in, const uint32_t* pos, uint64_t n, uint64_t* out) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i < n) out[i] = in[pos[i]];
}
__global__ void k0_gather32(const uint32_t* in, const uint32_t* pos, uint64_t n, uint32_t* out) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i < n) out[i] = in[pos[i]];
}
__global__ void k0_iota(uint32_t* a, uint64_t n) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i < n) a[i] = (uint32_t)i;
}

__global__ void k0_heads(const uint64_t* lo, const uint64_t* hi, uint64_t n, uint32_t* flag) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  flag[i] = (i == 0 || lo[i] != lo[i - 1] || (hi && hi[i] != hi[i - 1])) ? 1u : 0u;
}

// per segment head of a label group: position, ordering key (label, first member) and the label's node count
__global__ void k0_seg_heads(const uint32_t* flag, const uint32_t* seg_of, const uint32_t* val, uint64_t E, uint64_t N, uint32_t li0,
                             uint64_t pos_base, uint32_t seg_base, uint64_t* head_pos, uint64_t* seg_key, uint32_t* lcount) {
  const uint64_t e = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (e >= E || !flag[e]) return;
  const uint32_t s = seg_base + seg_of[e];
  const uint32_t li = li0 + (uint32_t)(e / N);
  head_pos[s] = pos_base + e;
  seg_key[s] = ((uint64_t)li << 32) | (uint64_t)val[e];
  atomicAdd(&lcount[li], 1u);
}

// node r (r-th segment by (label, first member)): key, top-link range and the SEQUENTIAL sum of the members'
// frequency vectors in hpf order (generate_neo4j_multi_hpf.py:405)
__global__ void k0_label_nodes(const uint32_t* seg_by_rank, const uint64_t* head_pos, uint32_t nseg, uint64_t E_total, uint64_t N,
                               const uint32_t* sorted_val, const hkey* full_keys, const double* full_freq, int P,
                               const uint32_t* label_mask, TablesView T, hkey* node_key, double* freq, uint32_t* tl_start,
                               uint32_t* tl_cnt) {
  const uint64_t q = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (q >= (uint64_t)nseg * (uint64_t)P) return;
  const uint32_t r = (uint32_t)(q / P), p = (uint32_t)(q % P);
  const uint32_t s = seg_by_rank[r];
  const uint64_t b0 = head_pos[s], b1 = (s + 1 < nseg) ? head_pos[s + 1] : E_total;
  double acc = 0.0 + full_freq[(uint64_t)sorted_val[b0] * P + p];
  for (uint64_t i = b0 + 1; i < b1; ++i) acc = acc + full_freq[(uint64_t)sorted_val[i] * P + p];
  const uint32_t node = (uint32_t)N + r;
  freq[(uint64_t)node * P + p] = acc;
  if (p == 0) {
    const uint32_t li = 1u + (uint32_t)(b0 / N);
    node_key[node] = full_keys[sorted_val[b0]] & key_mask_of(T, label_mask[li]);
    tl_start[node] = (uint32_t)b0;
    tl_cnt[node] = (uint32_t)(b1 - b0);
  }
}

// hash insert of every node: the label (= region) of a node follows from the label's node-id range
__global__ void k0_insert(HSlot* slots, const uint64_t* ht_off, const uint32_t* ht_mask, const hkey* node_key, uint32_t n_nodes,
                          const uint32_t* label_first_by_index, const uint32_t* label_mask, int n_labels) {
  const uint32_t node = blockIdx.x * blockDim.x + threadIdx.x;
  if (node >= n_nodes) return;
  int lo = 0, hi = n_labels - 1;   // largest label index whose first node id <= node
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (label_first_by_index[mid] <= node) lo = mid; else hi = mid - 1;
  }
  const uint32_t m = label_mask[lo];
  const hkey key = node_key[node];
  const uint32_t mask = ht_mask[m];
  HSlot* base = slots + ht_off[m];
  uint32_t h = ht_home(key, mask);
  for (;;) {
    const unsigned int old = atomicCAS(&base[h].node, GRIMB_NONE, node);
    if (old == GRIMB_NONE) {
      base[h].key = key;
      return;
    }
    h = (h + 1) & mask;
  }
}

// connector elements of one group of (parent label, dropped locus) pairs: e -> (pair, node of the parent label)
__global__ void k0_conn_keys(TablesView T, CompactLayout C, const uint64_t* __restrict__ pair_off, const uint32_t* __restrict__ pair_child,
                             const uint32_t* __restrict__ pair_first, uint32_t pi0, uint32_t npairs, uint64_t e0, uint64_t E,
                             uint64_t* lo, uint64_t* hi, uint32_t* val) {
  const uint64_t e = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (e >= E) return;
  const uint64_t ge = e0 + e;
  uint32_t a = pi0, b = pi0 + npairs - 1;   // largest pair with pair_off <= ge
  while (a < b) {
    const uint32_t mid = (a + b + 1) >> 1;
    if (pair_off[mid] <= ge) a = mid; else b = mid - 1;
  }
  const uint32_t node = pair_first[a] + (uint32_t)(ge - pair_off[a]);
  const u128 c = ((u128)a << C.cbits) | compact_of(T.node_key[node], T.shift, T.width, C, T.L, pair_child[a]);
  lo[e] = (uint64_t)c;
  if (hi) hi[e] = (uint64_t)(c >> 64);
  val[e] = node;
}

// head of a connector group -> CSR entry of (child node, added locus)
__global__ void k0_conn_heads(const uint32_t* flag, const uint32_t* next_head, const uint32_t* sorted_node, uint64_t E, uint64_t e0,
                              TablesView T, const uint64_t* __restrict__ pair_off, const uint32_t* __restrict__ pair_child,
                              const uint8_t* __restrict__ pair_locus, uint32_t pi0, uint32_t npairs, uint32_t* cn_start,
                              uint32_t* cn_cnt, unsigned int* n_conn) {
  const uint64_t e = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (e >= E || !flag[e]) return;
  const uint64_t ge = e0 + e;
  uint32_t a = pi0, b = pi0 + npairs - 1;
  while (a < b) {
    const uint32_t mid = (a + b + 1) >> 1;
    if (pair_off[mid] <= ge) a = mid; else b = mid - 1;
  }
  const uint32_t A = pair_child[a];
  const hkey ck = T.node_key[sorted_node[e]] & key_mask_of(T, A);
  const uint32_t child = ht_lookup(T, A, ck);
  if (child == GRIMB_NONE) return;  // cannot happen: every projection of a node is a node
  cn_start[(uint64_t)child * T.L + pair_locus[a]] = (uint32_t)ge;
  cn_cnt[(uint64_t)child * T.L + pair_locus[a]] = next_head[e] - (uint32_t)e;
  atomicAdd(n_conn, 1u);
}

// next_head[i] for head positions: position of the following head (or n)
__global__ void k0_next_head(const uint32_t* flag, uint64_t n, uint32_t* next_head) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= n || !flag[i]) return;
  uint64_t j = i + 1;
  while (j < n && !flag[j]) ++j;
  next_head[i] = (uint32_t)j;
}

// Stable sort of n composite keys (lo, optional hi) with their 32-bit values; results in lo_out / hi_out / val_out.
struct K0Sorter {
  DevBuf tmp, pos0, pos1, pos2, g64;
  cudaError_t reserve(uint64_t n, bool two) {
    size_t t1 = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, t1, (uint64_t*)nullptr, (uint64_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr, (int)n);
    size_t t2 = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, t2, (uint32_t*)nullptr, (uint32_t*)nullptr, (int)n);
    cudaError_t e = tmp.reserve((t1 > t2 ? t1 : t2) + 64);
    if (two) {
      if (e == cudaSuccess) e = pos0.reserve(n * 4);
      if (e == cudaSuccess) e = pos1.reserve(n * 4);
      if (e == cudaSuccess) e = pos2.reserve(n * 4);
      if (e == cudaSuccess) e = g64.reserve(n * 8);
    }
    return e;
  }
  cudaError_t sort(const uint64_t* lo, const uint64_t* hi, const uint32_t* val, uint64_t* lo_out, uint64_t* hi_out, uint32_t* val_out,
                   uint64_t n, int bits, int* launches) {
    if (n == 0) return cudaSuccess;
    size_t tb = tmp.cap;
    const unsigned g = nblk(n);
    if (!hi) {
      *launches += 1 + (bits + 7) / 8;
      return cub::DeviceRadixSort::SortPairs(tmp.p, tb, lo, lo_out, val, val_out, (int)n, 0, bits < 64 ? bits : 64);
    }
    // LSD over the two 64-bit words, carrying a position permutation
    k0_iota<<<g, 256>>>((uint32_t*)pos0.p, n);
    cudaError_t e = cub::DeviceRadixSort::SortPairs(tmp.p, tb, lo, lo_out, (const uint32_t*)pos0.p, (uint32_t*)pos1.p, (int)n, 0, 64);
    if (e != cudaSuccess) return e;
    k0_gather64<<<g, 256>>>(hi, (const uint32_t*)pos1.p, n, (uint64_t*)g64.p);
    tb = tmp.cap;
    e = cub::DeviceRadixSort::SortPairs(tmp.p, tb, (const uint64_t*)g64.p, hi_out, (const uint32_t*)pos1.p, (uint32_t*)pos2.p, (int)n, 0,
                                        bits - 64);
    if (e != cudaSuccess) return e;
    k0_gather64<<<g, 256>>>(lo, (const uint32_t*)pos2.p, n, lo_out);
    k0_gather32<<<g, 256>>>(val, (const uint32_t*)pos2.p, n, val_out);
    *launches += 5 + 9 + (bits - 64 + 7) / 8 + 1;
    return cudaGetLastError();
  }
};

extern "C" int grimb_tables_build(const GrimbTableDesc* d, GrimbTables** out) {
  if (!d || !out) return fail(GRIMB_E_ARG, "null argument");
  const int L = d->n_loci, P = d->n_pops;
  if (L < 1 || L > GRIMB_MAX_LOCI || P < 1) return fail(GRIMB_E_ARG, "bad n_loci / n_pops");
  if (d->n_full < 0 || d->n_full > 0x7FFFFFF0ll) return fail(GRIMB_E_ARG, "bad n_full");
  int bits = 0;
  for (int l = 0; l < L; ++l) {
    if (d->key_bits[l] < 1 || d->key_bits[l] > 16) return fail(GRIMB_E_LAYOUT, "key_bits must be 1..16");
    if ((1ll << d->key_bits[l]) <= d->n_alleles[l]) return fail(GRIMB_E_LAYOUT, "allele ids do not fit key_bits");
    bits += d->key_bits[l];
  }
  if (bits > 64 * GRIMB_KW - 1)
    return fail(GRIMB_E_LAYOUT, GRIMB_KW == 1 ? "packed key exceeds 63 bits (use libgrimb200w.so: 128-bit keys)"
                                              : "packed key exceeds 127 bits");
  CK(cudaSetDevice(d->device));
  const uint64_t N = (uint64_t)d->n_full;
  const uint32_t NL = 1u << L;
  // labels of the store: every locus subset in the reference's order, or (Plan_A_Matrix) the caller's list
  std::vector<uint32_t> order = label_order(L);
  const bool restricted = d->label_masks != nullptr;
  if (restricted) {
    if (d->n_labels < 2 || d->n_labels > (int32_t)(NL - 1) || d->n_plan_a_labels < 2 || d->n_plan_a_labels > d->n_labels)
      return fail(GRIMB_E_ARG, "bad label list");
    order.assign(d->label_masks, d->label_masks + d->n_labels);
    std::vector<uint8_t> seen(NL, 0);
    for (uint32_t m : order) {
      if (m == 0 || m >= NL || seen[m]) return fail(GRIMB_E_ARG, "label list: masks must be distinct locus subsets");
      seen[m] = 1;
    }
    if (order[0] != NL - 1) return fail(GRIMB_E_ARG, "label list: the full label comes first");
  }
  const uint32_t n_labels = (uint32_t)order.size();   // full label + marginals
  const uint32_t n_csr_labels = restricted ? (uint32_t)d->n_plan_a_labels : n_labels;   // labels whose nodes are CSR vertices
  // 32-bit offsets everywhere (tl_start, cn_start, row indices): reject what would not fit
  if (N * (uint64_t)(n_labels - 1) > 0xFFFFFFF0ull) return fail(GRIMB_E_ARG, "too many top links (n_full x marginal labels >= 2^32)");

  GrimbTables* t = new GrimbTables();
  t->device = d->device;
  t->image = nullptr;
  ImageHeader& h = t->h;
  memset(&h, 0, sizeof(h));
  h.magic = IMAGE_MAGIC;
  h.L = L;
  h.P = P;
  h.n_full = (uint32_t)N;
  CompactLayout CL;
  memset(&CL, 0, sizeof(CL));
  int sh = 0, csh = 0;
  for (int l = 0; l < L; ++l) {
    h.shift[l] = (uint8_t)sh;
    h.width[l] = (uint8_t)d->key_bits[l];
    h.n_alleles[l] = (uint32_t)d->n_alleles[l];
    sh += d->key_bits[l];
    int w = 1;
    while ((1ll << w) <= d->n_alleles[l]) ++w;   // minimal width for the table ids 1..n
    CL.cshift[l] = (uint8_t)csh;
    CL.cwidth[l] = (uint8_t)w;
    csh += w;
  }
  CL.cbits = csh;
  int launches = 0;
  std::vector<void*> owned;   // device allocations released on every exit path
  unsigned int* d_nconn = nullptr;
  auto cleanup = [&](bool ok) {
    for (void* p : owned) cudaFree(p);
    if (d_nconn) cudaFree(d_nconn);
    if (!ok) {
      if (t->image) cudaFree(t->image);
#if GRIMB_KW == 1
      if (t->fidx_mem) cudaFree(t->fidx_mem);
#endif
      delete t;
    }
  };
  cudaError_t e;
#define CKT(call)                                                                   \
  do {                                                                              \
    e = (call);                                                                     \
    if (e != cudaSuccess) {                                                         \
      cleanup(false);                                                               \
      return fail(e == cudaErrorMemoryAllocation ? GRIMB_E_NOMEM : GRIMB_E_CUDA,    \
                  std::string(#call) + ": " + cudaGetErrorString(e));               \
    }                                                                               \
  } while (0)
  auto dalloc = [&](void** p, size_t bytes) -> cudaError_t {
    cudaError_t r = cudaMalloc(p, bytes ? bytes : 16);
    if (r == cudaSuccess) owned.push_back(*p);
    return r;
  };

  // ---- stage inputs
  uint16_t* d_al = nullptr;
  double* d_ff = nullptr;
  hkey* d_keys = nullptr;
  uint8_t* d_shift = nullptr;
  uint32_t* d_lmask = nullptr;
  CKT(dalloc((void**)&d_al, N * L * 2));
  CKT(dalloc((void**)&d_ff, N * P * 8));
  CKT(dalloc((void**)&d_keys, N * sizeof(hkey)));
  CKT(dalloc((void**)&d_shift, 16));
  CKT(dalloc((void**)&d_lmask, 512 * 4));
  CKT(cudaMemcpy(d_al, d->full_alleles, N * L * 2, cudaMemcpyHostToDevice));
  CKT(cudaMemcpy(d_ff, d->full_freqs, N * P * 8, cudaMemcpyHostToDevice));
  CKT(cudaMemcpy(d_shift, h.shift, 9, cudaMemcpyHostToDevice));
  {
    std::vector<uint32_t> lm(512, 0);
    for (uint32_t li = 0; li < n_labels; ++li) lm[li] = order[li];
    CKT(cudaMemcpy(d_lmask, lm.data(), 512 * 4, cudaMemcpyHostToDevice));
  }
  cudaEvent_t ev_b0 = nullptr, ev_b1 = nullptr;
  cudaEventCreate(&ev_b0);
  cudaEventCreate(&ev_b1);
  cudaEventRecord(ev_b0, 0);
  if (N) {
    k_pack_full<<<nblk(N), 256>>>(d_al, L, d_shift, N, d_keys);
    ++launches;
  }
  CKT(cudaGetLastError());
  // a view good enough for key_mask_of / compact_of before the image exists
  TablesView pv;
  memset(&pv, 0, sizeof(pv));
  pv.L = L;
  pv.P = P;
  memcpy(pv.shift, h.shift, 9);
  memcpy(pv.width, h.width, 9);

  // ---- pass 1: group the marginal labels (bounded groups of labels)
  int lbits = 1;
  while ((1u << lbits) < n_labels) ++lbits;
  const int tot_bits = CL.cbits + lbits;
  const bool two = tot_bits > 64;
  const uint64_t E_total = N * (uint64_t)(n_labels - 1);
  uint64_t budget = 1ull << 28;   // elements per group
  if (const char* gb = getenv("GRIMB_K0_GROUP")) {
    const long long v = atoll(gb);
    if (v >= 1024) budget = (uint64_t)v;
  }
  uint32_t labels_per_group = N ? (uint32_t)std::max<uint64_t>(1, budget / N) : n_labels;
  if (labels_per_group > n_labels - 1) labels_per_group = n_labels > 1 ? n_labels - 1 : 1;
  const uint64_t Eg = N * (uint64_t)labels_per_group;   // largest group
  uint64_t *g_lo = nullptr, *g_hi = nullptr, *s_lo = nullptr, *s_hi = nullptr, *d_head_pos = nullptr, *d_seg_key = nullptr;
  uint32_t *g_val = nullptr, *d_sorted_val = nullptr, *d_flag = nullptr, *d_seg = nullptr, *d_lcount = nullptr;
  K0Sorter sorter;
  std::vector<uint32_t> lcount_i(n_labels, 0);   // nodes per label index
  uint32_t nseg_total = 0;
  if (E_total) {
    CKT(dalloc((void**)&g_lo, Eg * 8));
    CKT(dalloc((void**)&s_lo, Eg * 8));
    if (two) {
      CKT(dalloc((void**)&g_hi, Eg * 8));
      CKT(dalloc((void**)&s_hi, Eg * 8));
    }
    CKT(dalloc((void**)&g_val, Eg * 4));
    CKT(dalloc((void**)&d_sorted_val, E_total * 4));     // becomes tl_adj
    CKT(dalloc((void**)&d_flag, Eg * 4));
    CKT(dalloc((void**)&d_seg, Eg * 4));
    CKT(dalloc((void**)&d_head_pos, (E_total + 1) * 8)); // worst case: every element its own segment
    CKT(dalloc((void**)&d_seg_key, (E_total + 1) * 8));
    CKT(dalloc((void**)&d_lcount, 512 * 4));
    CKT(cudaMemset(d_lcount, 0, 512 * 4));
    CKT(sorter.reserve(Eg > E_total ? E_total : Eg, two));
    for (uint32_t li0 = 1; li0 < n_labels; li0 += labels_per_group) {
      const uint32_t nl = std::min(labels_per_group, n_labels - li0);
      const uint64_t E = N * (uint64_t)nl, pos_base = N * (uint64_t)(li0 - 1);
      k0_make_keys<<<nblk(E), 256>>>(d_keys, pv, CL, d_lmask, li0, N, E, g_lo, g_hi, g_val);
      CKT(sorter.sort(g_lo, g_hi, g_val, s_lo, s_hi, d_sorted_val + pos_base, E, tot_bits, &launches));
      k0_heads<<<nblk(E), 256>>>(s_lo, s_hi, E, d_flag);
      size_t tb = sorter.tmp.cap;
      CKT(cub::DeviceScan::ExclusiveSum(sorter.tmp.p, tb, d_flag, d_seg, (int)E));
      k0_seg_heads<<<nblk(E), 256>>>(d_flag, d_seg, d_sorted_val + pos_base, E, N, li0, pos_base, nseg_total, d_head_pos,
                                     d_seg_key, d_lcount);
      launches += 5;
      // segments of this group (one small read-back per GROUP of labels, not per label)
      uint32_t last_flag = 0, last_seg = 0;
      CKT(cudaMemcpy(&last_flag, d_flag + (E - 1), 4, cudaMemcpyDeviceToHost));
      CKT(cudaMemcpy(&last_seg, d_seg + (E - 1), 4, cudaMemcpyDeviceToHost));
      if ((uint64_t)nseg_total + last_seg + last_flag > 0x7FFFFFF0ull) {
        cleanup(false);
        return fail(GRIMB_E_ARG, "too many nodes");
      }
      nseg_total += last_seg + last_flag;
    }
    CKT(cudaMemcpy(lcount_i.data(), d_lcount, n_labels * 4, cudaMemcpyDeviceToHost));
  }
  lcount_i[0] = (uint32_t)N;
  const uint64_t n_nodes = N + nseg_total;
  if (n_nodes > 0x7FFFFFF0ull) {
    cleanup(false);
    return fail(GRIMB_E_ARG, "too many nodes");
  }
  h.n_nodes = (uint32_t)n_nodes;
  h.n_toplinks = E_total;

  // ---- label ranges, hash region sizes, connector pairs
  std::vector<uint32_t> lfirst(NL, 0), lcount(NL, 0), hmask(NL, 1), lfirst_i(n_labels, 0);
  std::vector<uint64_t> hoff(NL, 0);
  {
    uint32_t nb = 0;
    for (uint32_t li = 0; li < n_labels; ++li) {
      lfirst[order[li]] = nb;
      lfirst_i[li] = nb;
      lcount[order[li]] = lcount_i[li];
      nb += lcount_i[li];
    }
    uint64_t so = 0;
    for (uint32_t m = 0; m < NL; ++m) {
      // load factor <= 0.5; <= 0.125 for the full-haplotype label, which takes the bulk of the
      // probes (2^L per fully typed subject, mostly misses: a miss scans until an empty slot)
      uint64_t full_mult = 8;   // slots per full haplotype (GRIMB_FULL_LOAD_MULT overrides, for A/B runs)
      if (const char* fm = getenv("GRIMB_FULL_LOAD_MULT")) {
        const long v = atol(fm);
        if (v >= 2 && v <= 64) full_mult = (uint64_t)v;
      }
      const uint64_t want = (m == NL - 1 ? full_mult : 2ull) * (uint64_t)lcount[m];
      uint32_t sz = 2;
      while (sz < want) sz <<= 1;
      hmask[m] = sz - 1;
      hoff[m] = so;
      so += sz;
    }
    h.n_slots = so;
  }
  // pairs (parent label B, dropped locus l) in the order the reference scans edges.csv
  std::vector<uint64_t> pair_off;
  std::vector<uint32_t> pair_child, pair_first;
  std::vector<uint8_t> pair_locus;
  uint64_t n_cn = 0;
  for (uint32_t li = 0; li < n_labels && !restricted; ++li) {   // a restricted store serves Plan A only: no connectors
    const uint32_t B = order[li];
    if (__builtin_popcount(B) < 2 || lcount[B] == 0) continue;
    for (int l = 0; l < L; ++l) {
      if (!(B >> l & 1u)) continue;
      pair_off.push_back(n_cn);
      pair_child.push_back(B & ~(1u << l));
      pair_first.push_back(lfirst[B]);
      pair_locus.push_back((uint8_t)l);
      n_cn += lcount[B];
    }
  }
  const uint32_t n_pairs = (uint32_t)pair_off.size();
  pair_off.push_back(n_cn);
  h.n_conn_edges = n_cn;
  if (n_cn + n_nodes * (uint64_t)L > 0xFFFFFFF0ull || n_nodes * (uint64_t)P > (1ull << 40)) {
    cleanup(false);
    return fail(GRIMB_E_ARG, "table too large for 32-bit connector offsets");
  }

  // ---- image layout
  auto al16 = [](uint64_t x) { return (x + 255ull) & ~255ull; };
  uint64_t o = al16(sizeof(ImageHeader));
  h.o_label_first = o; o = al16(o + (uint64_t)NL * 4);
  h.o_label_count = o; o = al16(o + (uint64_t)NL * 4);
  h.o_ht_off = o; o = al16(o + (uint64_t)NL * 8);
  h.o_ht_mask = o; o = al16(o + (uint64_t)NL * 4);
  h.o_slots = o; o = al16(o + h.n_slots * sizeof(HSlot));
  h.o_node_key = o; o = al16(o + n_nodes * sizeof(hkey));
  h.o_freq = o; o = al16(o + n_nodes * P * 8);
  h.o_tl_start = o; o = al16(o + n_nodes * 4);
  h.o_tl_cnt = o; o = al16(o + n_nodes * 4);
  h.o_tl_adj = o; o = al16(o + (h.n_toplinks ? h.n_toplinks : 1) * 4);
  h.o_cn_start = o; o = al16(o + n_nodes * L * 4);
  h.o_cn_cnt = o; o = al16(o + n_nodes * L * 4);
  h.o_cn_adj = o; o = al16(o + (n_cn ? n_cn : 1) * 4);
  h.bytes = o;
  e = cudaMalloc((void**)&t->image, h.bytes);
  if (e != cudaSuccess) {
    t->image = nullptr;
    cleanup(false);
    return fail(GRIMB_E_NOMEM, std::string("table image: ") + cudaGetErrorString(e));
  }
  make_view(t);
  TablesView& v = t->view;
  // everything except the slots (initialised below) and the arrays written in full starts at zero
  CKT(cudaMemsetAsync(t->image, 0, h.o_slots, 0));
  CKT(cudaMemsetAsync((char*)t->image + h.o_tl_start, 0, h.o_tl_adj - h.o_tl_start, 0));
  CKT(cudaMemsetAsync((char*)t->image + h.o_cn_start, 0, h.o_cn_adj - h.o_cn_start, 0));
  CKT(cudaMemcpy((void*)v.label_first, lfirst.data(), (size_t)NL * 4, cudaMemcpyHostToDevice));
  CKT(cudaMemcpy((void*)v.label_count, lcount.data(), (size_t)NL * 4, cudaMemcpyHostToDevice));
  CKT(cudaMemcpy((void*)v.ht_off, hoff.data(), (size_t)NL * 8, cudaMemcpyHostToDevice));
  CKT(cudaMemcpy((void*)v.ht_mask, hmask.data(), (size_t)NL * 4, cudaMemcpyHostToDevice));

  // ---- pass 2: node ids (segments by (label, first member)), node arrays, top links
  if (N) {
    k_full_nodes<<<nblk(N), 256>>>(d_keys, d_ff, (uint32_t)N, P, (hkey*)v.node_key, (double*)v.freq, (uint32_t*)v.tl_start,
                                   (uint32_t*)v.tl_cnt);
    ++launches;
  }
  if (nseg_total) {
    uint64_t* d_seg_key2 = nullptr;
    uint32_t *d_iota = nullptr, *d_by_rank = nullptr;
    CKT(dalloc((void**)&d_seg_key2, (uint64_t)nseg_total * 8));
    CKT(dalloc((void**)&d_iota, (uint64_t)nseg_total * 4));
    CKT(dalloc((void**)&d_by_rank, (uint64_t)nseg_total * 4));
    k0_iota<<<nblk(nseg_total), 256>>>(d_iota, nseg_total);
    K0Sorter s2;
    CKT(s2.reserve(nseg_total, false));
    CKT(s2.sort(d_seg_key, nullptr, d_iota, d_seg_key2, nullptr, d_by_rank, nseg_total, 32 + lbits, &launches));
    k0_label_nodes<<<nblk((uint64_t)nseg_total * P), 256>>>(d_by_rank, d_head_pos, nseg_total, E_total, N, d_sorted_val, d_keys, d_ff,
                                                           P, d_lmask, pv, (hkey*)v.node_key, (double*)v.freq,
                                                           (uint32_t*)v.tl_start, (uint32_t*)v.tl_cnt);
    CKT(cudaMemcpyAsync((void*)v.tl_adj, d_sorted_val, E_total * 4, cudaMemcpyDeviceToDevice, 0));
    launches += 3;
  }
  CKT(cudaGetLastError());

  // ---- hash insert: one launch over all nodes
  uint32_t* d_lfirst_i = nullptr;
  CKT(dalloc((void**)&d_lfirst_i, 512 * 4));
  CKT(cudaMemcpy(d_lfirst_i, lfirst_i.data(), n_labels * 4, cudaMemcpyHostToDevice));
  k_init_slots<<<nblk(h.n_slots), 256>>>((HSlot*)v.slots, h.n_slots);
  if (n_nodes)
    k0_insert<<<nblk(n_nodes), 256>>>((HSlot*)v.slots, v.ht_off, v.ht_mask, v.node_key, (uint32_t)n_nodes, d_lfirst_i, d_lmask,
                                      (int)n_labels);
  launches += 2;
  CKT(cudaGetLastError());

  // ---- connectors: for every label B (>= 2 loci) and locus l in B, group B's nodes by B \ l
  CKT(cudaMalloc(&d_nconn, 4));
  CKT(cudaMemset(d_nconn, 0, 4));
  if (n_cn) {
    uint64_t* d_pair_off = nullptr;
    uint32_t *d_pair_child = nullptr, *d_pair_first = nullptr, *d_next = nullptr;
    uint8_t* d_pair_locus = nullptr;
    CKT(dalloc((void**)&d_pair_off, (n_pairs + 1) * 8));
    CKT(dalloc((void**)&d_pair_child, n_pairs * 4));
    CKT(dalloc((void**)&d_pair_first, n_pairs * 4));
    CKT(dalloc((void**)&d_pair_locus, n_pairs));
    CKT(cudaMemcpy(d_pair_off, pair_off.data(), (n_pairs + 1) * 8, cudaMemcpyHostToDevice));
    CKT(cudaMemcpy(d_pair_child, pair_child.data(), n_pairs * 4, cudaMemcpyHostToDevice));
    CKT(cudaMemcpy(d_pair_first, pair_first.data(), n_pairs * 4, cudaMemcpyHostToDevice));
    CKT(cudaMemcpy(d_pair_locus, pair_locus.data(), n_pairs, cudaMemcpyHostToDevice));
    int pbits = 1;
    while ((1u << pbits) < n_pairs) ++pbits;
    const int cbits_tot = CL.cbits + pbits;
    const bool ctwo = cbits_tot > 64;
    // groups of consecutive pairs with a bounded number of elements (a pair is never split)
    uint64_t gmax = 0;
    {
      uint32_t a = 0;
      while (a < n_pairs) {
        uint32_t b = a + 1;
        while (b < n_pairs && pair_off[b + 1] - pair_off[a] <= budget) ++b;
        gmax = std::max(gmax, pair_off[b] - pair_off[a]);
        a = b;
      }
    }
    // the label-pass buffers are reused when they are large enough
    uint64_t *c_lo = g_lo, *c_hi = g_hi, *cs_lo = s_lo, *cs_hi = s_hi;
    uint32_t *c_val = g_val, *c_flag = d_flag;
    if (gmax > Eg || (ctwo && !two)) {
      CKT(dalloc((void**)&c_lo, gmax * 8));
      CKT(dalloc((void**)&cs_lo, gmax * 8));
      CKT(dalloc((void**)&c_val, gmax * 4));
      CKT(dalloc((void**)&c_flag, gmax * 4));
      if (ctwo) {
        CKT(dalloc((void**)&c_hi, gmax * 8));
        CKT(dalloc((void**)&cs_hi, gmax * 8));
      }
    }
    if (!ctwo) c_hi = cs_hi = nullptr;
    CKT(dalloc((void**)&d_next, gmax * 4));
    K0Sorter cs;
    CKT(cs.reserve(gmax, ctwo));
    uint32_t a = 0;
    while (a < n_pairs) {
      uint32_t b = a + 1;
      while (b < n_pairs && pair_off[b + 1] - pair_off[a] <= budget) ++b;
      const uint64_t e0 = pair_off[a], E = pair_off[b] - pair_off[a];
      if (E) {
        k0_conn_keys<<<nblk(E), 256>>>(v, CL, d_pair_off, d_pair_child, d_pair_first, a, b - a, e0, E, c_lo, c_hi, c_val);
        CKT(cs.sort(c_lo, c_hi, c_val, cs_lo, cs_hi, (uint32_t*)v.cn_adj + e0, E, cbits_tot, &launches));
        k0_heads<<<nblk(E), 256>>>(cs_lo, cs_hi, E, c_flag);
        k0_next_head<<<nblk(E), 256>>>(c_flag, E, d_next);
        k0_conn_heads<<<nblk(E), 256>>>(c_flag, d_next, (const uint32_t*)v.cn_adj + e0, E, e0, v, d_pair_off, d_pair_child,
                                       d_pair_locus, a, b - a, (uint32_t*)v.cn_start, (uint32_t*)v.cn_cnt, d_nconn);
        launches += 4;
      }
      a = b;
    }
  }
  CKT(cudaGetLastError());
  CKT(cudaDeviceSynchronize());
  unsigned int n_conn = 0;
  CKT(cudaMemcpy(&n_conn, d_nconn, 4, cudaMemcpyDeviceToHost));

  // ---- reference CSR sentinel quirk (networkx_graph.py:195-196; SURVEY trap T1)
  if (n_nodes > N && N > 0) {
    // vertices of the reference's CSR: every node, or (restricted) the nodes of the Plan-A labels, which come first
    uint64_t n_vertices = n_nodes;
    if (restricted) n_vertices = (uint64_t)lfirst_i[n_csr_labels - 1] + lcount_i[n_csr_labels - 1];
    const uint32_t last = (uint32_t)n_vertices - 1;
    uint32_t deg = 0;
    CKT(cudaMemcpy(&deg, v.tl_cnt + last, 4, cudaMemcpyDeviceToHost));
    uint32_t nc = sentinel_count(deg, N * (uint64_t)(n_csr_labels - 1), n_vertices);
    CKT(cudaMemcpy((uint32_t*)v.tl_cnt + last, &nc, 4, cudaMemcpyHostToDevice));
    if (L >= 2 && !restricted) {
      int pl_locus = d->last_parent_locus >= 0 ? d->last_parent_locus : L - 2;
      uint64_t idx = (uint64_t)last * L + pl_locus;
      CKT(cudaMemcpy(&deg, v.cn_cnt + idx, 4, cudaMemcpyDeviceToHost));
      nc = sentinel_count(deg, (uint64_t)n_conn + n_cn, n_nodes + n_conn);
      CKT(cudaMemcpy((uint32_t*)v.cn_cnt + idx, &nc, 4, cudaMemcpyHostToDevice));
    }
  }
  CKT(cudaMemcpy(t->image, &h, sizeof(h), cudaMemcpyHostToDevice));
#if GRIMB_KW == 1
  CKT(build_fast_index(t, &launches));
#endif
  cudaEventRecord(ev_b1, 0);
  CKT(cudaDeviceSynchronize());
  if (ev_b0 && ev_b1) cudaEventElapsedTime(&t->build_ms, ev_b0, ev_b1);
  if (ev_b0) cudaEventDestroy(ev_b0);
  if (ev_b1) cudaEventDestroy(ev_b1);
  t->build_launches = launches;
  cleanup(true);
  *out = t;
  return GRIMB_OK;
#undef CKT
}


extern "C" int grimb_tables_free(GrimbTables* t) {
  if (!t) return GRIMB_OK;
  cudaSetDevice(t->device);
  cudaFree(t->image);
#if GRIMB_KW == 1
  cudaFree(t->fidx_mem);
#endif
  delete t;
  return GRIMB_OK;
}

extern "C" int64_t grimb_tables_build_launches(const GrimbTables* t) { return t ? t->build_launches : 0; }
extern "C" double grimb_tables_build_ms(const GrimbTables* t) { return t ? (double)t->build_ms : 0.0; }

extern "C" int grimb_tables_info(const GrimbTables* t, GrimbTableInfo* info) {
  if (!t || !info) return fail(GRIMB_E_ARG, "null argument");
  info->n_loci = t->h.L;
  info->n_pops = t->h.P;
  info->n_nodes = t->h.n_nodes;
  info->n_full = t->h.n_full;
  info->n_toplinks = (int64_t)t->h.n_toplinks;
  info->n_conn_edges = (int64_t)t->h.n_conn_edges;
  info->n_slots = (int64_t)t->h.n_slots;
  info->device_bytes = (int64_t)t->h.bytes;
#if GRIMB_KW == 1
  info->device_bytes += (int64_t)t->fidx_bytes;
#endif
  return GRIMB_OK;
}

extern "C" int grimb_tables_export(const GrimbTables* t, uint64_t* node_key, double* node_freq, uint32_t* tl_start,
                                   uint32_t* tl_cnt, uint32_t* tl_adj, uint32_t* cn_start, uint32_t* cn_cnt,
                                   uint32_t* cn_adj, uint32_t* label_first, uint32_t* label_count) {
  if (!t) return fail(GRIMB_E_ARG, "null argument");
  CK(cudaSetDevice(t->device));
  const ImageHeader& h = t->h;
  const TablesView& v = t->view;
  const uint64_t n = h.n_nodes;
  if (node_key) CK(cudaMemcpy(node_key, v.node_key, n * sizeof(hkey), cudaMemcpyDeviceToHost));
  if (node_freq) CK(cudaMemcpy(node_freq, v.freq, n * h.P * 8, cudaMemcpyDeviceToHost));
  if (tl_start) CK(cudaMemcpy(tl_start, v.tl_start, n * 4, cudaMemcpyDeviceToHost));
  if (tl_cnt) CK(cudaMemcpy(tl_cnt, v.tl_cnt, n * 4, cudaMemcpyDeviceToHost));
  if (tl_adj) CK(cudaMemcpy(tl_adj, v.tl_adj, h.n_toplinks * 4, cudaMemcpyDeviceToHost));
  if (cn_start) CK(cudaMemcpy(cn_start, v.cn_start, n * h.L * 4, cudaMemcpyDeviceToHost));
  if (cn_cnt) CK(cudaMemcpy(cn_cnt, v.cn_cnt, n * h.L * 4, cudaMemcpyDeviceToHost));
  if (cn_adj) CK(cudaMemcpy(cn_adj, v.cn_adj, h.n_conn_edges * 4, cudaMemcpyDeviceToHost));
  if (label_first) CK(cudaMemcpy(label_first, v.label_first, (size_t)(1u << h.L) * 4, cudaMemcpyDeviceToHost));
  if (label_count) CK(cudaMemcpy(label_count, v.label_count, (size_t)(1u << h.L) * 4, cudaMemcpyDeviceToHost));
  return GRIMB_OK;
}

extern "C" int grimb_tables_image_size(const GrimbTables* t, int64_t* bytes) {
  if (!t || !bytes) return fail(GRIMB_E_ARG, "null argument");
  *bytes = (int64_t)t->h.bytes;
  return GRIMB_OK;
}

extern "C" int grimb_tables_image_ptr(const GrimbTables* t, void** dev_ptr) {
  if (!t || !dev_ptr) return fail(GRIMB_E_ARG, "null argument");
  *dev_ptr = t->image;
  return GRIMB_OK;
}

extern "C" int grimb_tables_image_copy(const GrimbTables* t, void* dst) {
  if (!t || !dst) return fail(GRIMB_E_ARG, "null argument");
  CK(cudaSetDevice(t->device));
  CK(cudaMemcpy(dst, t->image, t->h.bytes, cudaMemcpyDefault));
  return GRIMB_OK;
}

extern "C" int grimb_tables_from_image(const void* dev_image, int64_t bytes, int device, GrimbTables** out) {
  if (!dev_image || !out || bytes < (int64_t)sizeof(ImageHeader)) return fail(GRIMB_E_ARG, "bad image");
  CK(cudaSetDevice(device));
  GrimbTables* t = new GrimbTables();
  t->device = device;
  t->image = nullptr;
  cudaError_t e = cudaMemcpy(&t->h, dev_image, sizeof(ImageHeader), cudaMemcpyDefault);
  if (e != cudaSuccess || t->h.magic != IMAGE_MAGIC || (int64_t)t->h.bytes != bytes) {
    delete t;
    return fail(GRIMB_E_ARG, "not a grimb200 table image");
  }
  e = cudaMalloc((void**)&t->image, (size_t)bytes);
  if (e != cudaSuccess) {
    delete t;
    return fail(GRIMB_E_NOMEM, cudaGetErrorString(e));
  }
  e = cudaMemcpy(t->image, dev_image, (size_t)bytes, cudaMemcpyDefault);
  if (e != cudaSuccess) {
    cudaFree(t->image);
    delete t;
    return fail(GRIMB_E_CUDA, cudaGetErrorString(e));
  }
  make_view(t);
#if GRIMB_KW == 1
  e = build_fast_index(t, nullptr);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    cudaFree(t->fidx_mem);
    cudaFree(t->image);
    delete t;
    return fail(e == cudaErrorMemoryAllocation ? GRIMB_E_NOMEM : GRIMB_E_CUDA,
                std::string("fast-path index: ") + cudaGetErrorString(e));
  }
#endif
  *out = t;
  return GRIMB_OK;
}

// ------------------------------------------------------------------------------------------
// imputation kernel: persistent CTAs, one subject per CTA at a time, dynamic work fetch
// ------------------------------------------------------------------------------------------
// Work for the general kernel is handed out heaviest first (longest-processing-time order): a
// classify pass sorts the pending subjects into GRIMB_BUCKETS cost buckets, and the persistent
// CTAs draw tickets that walk bucket 0 (heaviest) to bucket 3.  Without it a 50 ms subject that
// happens to sit at the end of the batch becomes the tail of the whole launch.
constexpr int GRIMB_BUCKETS = 4;

__global__ void k_classify(GrimbBatch B, int L, const uint32_t* list, const unsigned int* list_n, uint32_t* buckets,
                           unsigned int* bucket_n, uint64_t stride) {
  const uint64_t n = list ? (uint64_t)*list_n : (uint64_t)B.n_subjects;
  for (uint64_t w = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; w < n; w += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t s = list ? list[w] : (uint32_t)w;
    const uint32_t typed = batch_typed(B, s, (1u << L) - 1u);
    // candidates per phase ~ product of the listed alleles; phases = 2^(typed-1); an untyped
    // locus multiplies the hits (top links / whole-label scans in Plan B)
    float a = 1.f, b = 1.f;
    int nt = 0;
    for (int l = 0; l < L; ++l)
      if (typed >> l & 1u) {
        a *= (float)batch_count(B, s, L, l, 0);
        b *= (float)batch_count(B, s, L, l, 1);
        ++nt;
      }
    float cost = (a + b) * (float)(1u << (nt > 0 ? nt - 1 : 0));
    if (nt < L) cost *= 16.f;
    const int k = cost >= 32768.f ? 0 : cost >= 2048.f ? 1 : cost >= 128.f ? 2 : 3;
    buckets[(uint64_t)k * stride + atomicAdd(&bucket_n[k], 1u)] = s;
  }
}

#ifndef KI_MIN_BLOCKS
#define KI_MIN_BLOCKS 2   /* x MAXT = 512 threads: 64 registers, i.e. 8 CTAs of 128 threads per SM; measured 13-18 % faster on C4 than 124 registers / 4 CTAs */
#endif

static __device__ __forceinline__ void init_subject(Subject& S, Shared& sh, const TablesView& T, const GrimbConfig* cfg,
                                                    const double* ones, char* arena, uint64_t arena_per_cta) {
  S.g.tid = threadIdx.x;
  S.g.n = blockDim.x;
  S.g.scratch = sh.scratch;
  S.sh = &sh;
  S.T = T;
  S.cfg = cfg;
  S.ones = ones;
  S.ar_base = arena + (uint64_t)blockIdx.x * arena_per_cta;
  S.ar_cap = arena_per_cta;
  S.pre = nullptr;
  S.pre_j = 0xFFFFFFFFu;
}

// Cooperative CTA group for the heaviest subjects (cost bucket 0 of k_classify: long allele lists,
// Cartesian products of up to number_of_options_threshold candidates per phase and side).  The unit of
// work of this kernel is one (subject, phase, side) slot, drawn from a global ticket counter, so up to
// 2^L CTAs open, probe and reduce the slots of ONE subject at the same time (open_phases + adjs_query +
// convert_list_to_one_dim, impute.py:914-989, nxg.py:253-278, impute.py:424-442); k_impute, launched next,
// starts such a subject from the finished top-K lists instead of walking its slots one after the other.
// (It is the same entry point as k_impute, launched with mode = 1: ptxas 12.9 crashes when the per-subject
// routines are reachable from two different kernels.)
static __device__ __forceinline__ void impute_slots(Subject& S, Shared& sh, const TablesView& T, const GrimbConfig* __restrict__ cfg,
                                                    const GrimbBatch& B, const OutArrays& O, unsigned long long* ticket,
                                                    const uint32_t* buckets, const unsigned int* bucket_n, const PreView& pv) {
  uint32_t nheavy = bucket_n[0];
  if (nheavy > pv.max_subjects) nheavy = pv.max_subjects;
  if (nheavy == 0) return;   // uniform over the grid
  const uint64_t items = (uint64_t)nheavy * pv.slots_per_subject;
  for (;;) {
    __syncthreads();
    if (threadIdx.x == 0) {
      const unsigned long long w = atomicAdd(ticket, 1ull);
      sh.work = (uint32_t)(w < items ? w : 0xFFFFFFFFull);
    }
    __syncthreads();
    const uint32_t w = sh.work;
    if (w == 0xFFFFFFFFu) break;
    const uint32_t j = w / pv.slots_per_subject;
    const int slot = (int)(w % pv.slots_per_subject);
    const uint64_t s = buckets[j];   // bucket 0
    run_slot_item(S, B, O, s, j, slot, pv);
  }
}

__global__ void __launch_bounds__(MAXT, KI_MIN_BLOCKS)
k_impute(TablesView T, const GrimbConfig* __restrict__ cfg, GrimbBatch B, OutArrays O, char* arena, uint64_t arena_per_cta,
         const double* ones, unsigned long long* work, const uint32_t* buckets, const unsigned int* bucket_n,
         uint64_t stride, PreView pv, int mode) {
  __shared__ Shared sh;
  Subject S;
  init_subject(S, sh, T, cfg, ones, arena, arena_per_cta);
  const PreView pvl = pv;   // a local copy: the subject keeps a pointer to it
  if ((mode & 3) == 1) {    // cooperative slot pass over the heaviest subjects (`work` = its ticket counter)
    impute_slots(S, sh, T, cfg, B, O, work, buckets, bucket_n, pvl);
    return;
  }
  S.pre = &pvl;
  uint64_t bound[GRIMB_BUCKETS + 1];
  bound[0] = 0;
  for (int k = 0; k < GRIMB_BUCKETS; ++k) bound[k + 1] = bound[k] + bucket_n[k];
  if (bound[GRIMB_BUCKETS] == 0) return;   // nothing was handed to the general kernel (uniform over the grid)
  // mode 0: every bucket.  mode 2 + 16 * hb: the heavy buckets [0, hb) only; mode 3 + 16 * hb: the others
  // (launch_tail runs the heavy buckets first, on wide CTAs and with the SMs to themselves)
  const int hb = mode >> 4;
  const uint64_t w_lo = (mode & 3) == 3 ? bound[hb] : 0, w_hi = (mode & 3) == 2 ? bound[hb] : bound[GRIMB_BUCKETS];
  for (;;) {
    __syncthreads();
    if (threadIdx.x == 0) sh.work = (uint32_t)atomicAdd(work, 1ull);
    __syncthreads();
    const uint64_t w = w_lo + sh.work;
    if (w >= w_hi) break;
    int k = 0;
    while (w >= bound[k + 1]) ++k;
    // the heaviest subjects come first: bucket 0, entry w -> its lists from the cooperative slot kernel
    S.pre_j = (k == 0 && w < pv.max_subjects && pv.top != nullptr) ? (uint32_t)w : 0xFFFFFFFFu;
    run_subject(S, B, O, (uint64_t)buckets[(uint64_t)k * stride + (w - bound[k])]);
  }
}

// ------------------------------------------------------------------------------------------
// Fast path: one WARP per subject for the common case of BASELINE config 2 -- every locus
// typed, one allele per chromosome side, one population (L <= 5 so the 2^L side haplotypes map
// onto the 32 lanes).  Lane v probes the haplotype that takes side bit_l(v) at locus l; phase i
// (lane i < 2^(L-1)) pairs lane i with lane 2^L-1-i (gen_phases, impute.py:274-303).  The epsilon
// schedule (impute.py:1658-1693) is a loop of ballots over the same 16 registers; sums run in
// phase order, ranks by (probability desc, phase asc), exactly as the general kernel does.
// Subjects that are not of this shape, or for which Plan A finds nothing (-> Plan B/C), are
// appended to `worklist` and handled by k_impute.  Result rows are allocated with one atomicAdd
// per CTA (8 subjects).
// ------------------------------------------------------------------------------------------
#if GRIMB_KW == 1
constexpr int FAST_WARPS = 8;
constexpr int FAST_MAX_ROUNDS = 40;
#ifndef FAST_MIN_BLOCKS
#define FAST_MIN_BLOCKS 4
#endif

// accept test of calc_haps_pairs (impute.py:458-491) for one candidate pair with P == 1:
//   x = eps / f1;  f2 >= x  and  m > 0  and  m*f2 >= x (x2 if the two haplotypes are equal)
// <=> m > 0 and fl(eps/f1) <= t with t = min(f2, m*f2 [/2]).  With b = fl(f1*t): eps <= b(1-2^-50)
// proves it and eps >= b(1+2^-50) refutes it, so the FP64 division only runs inside that band.
struct FastPair {
  double f, f2, y, lo, hi;
  bool same, mpos;
  __device__ __forceinline__ bool accept(double e) const {
    if (!mpos) return false;
    if (e <= lo) return true;
    if (e >= hi) return false;
    const double x = e / f;
    return f2 >= x && (same ? (y >= x * 2) : (y >= x));
  }
};

// Inputs of one subject, loaded one loop iteration ahead so that the dependent chain
// allele_off -> alleles and prior_index -> prior overlaps the previous subject's work.  Lane l < L of
// the half-warp holds locus l (its allele pair and listed counts); every lane holds the scalars.
struct FastIn {
  uint32_t typed, c, pair;
  double m;
};

__device__ __forceinline__ void fast_load(FastIn& in, const GrimbBatch& B, uint64_t s, int L, int i, const TablesView& T) {
  if (B.packed_keys) {   // packed form: lane l takes the two alleles of locus l out of the subject's keys
    const uint32_t fl = B.packed_flags[s];
    in.typed = (fl & 0x8000u) ? 0u : ((1u << L) - 1u);
    in.c = 0x00010001u;
    in.pair = 0;
    if (i < L) {
      const uint64_t k0 = B.packed_keys[2 * s], k1 = B.packed_keys[2 * s + 1];
      in.pair = (uint32_t)key_field(T, k0, i) | ((uint32_t)key_field(T, k1, i) << 16);
    }
    in.m = __ldg(B.priors + batch_prior(B, s));
    return;
  }
  in.typed = B.typed_mask[s];
  const uint32_t off = B.allele_off[s];
  // the listed counts of one subject are 2L uint16 = L aligned uint32; every count must be 1
  in.c = 0x00010001u;
  if (B.counts && i < L) in.c = reinterpret_cast<const uint32_t*>(B.counts + s * (uint64_t)L * 2)[i];
  in.pair = 0;
  // only inside the subject's own range: a subject that lists fewer than 2L alleles is not of this shape
  if (i < L && 2u * (uint32_t)i + 2u <= B.allele_off[s + 1] - off) {
    const uint16_t* al = B.alleles + off + 2 * i;
    in.pair = (off & 1u) ? ((uint32_t)al[0] | ((uint32_t)al[1] << 16)) : *reinterpret_cast<const uint32_t*>(al);
  }
  in.m = __ldg(B.priors + batch_prior(B, s));
}

// Two independent probes of the full-label region; the first sector of each is requested before
// either is examined (the common case resolves both in that one round trip).
__device__ __forceinline__ void ht_lookup2(const HSlot* __restrict__ base, uint32_t mask, uint64_t k1, bool p1, uint64_t k2,
                                           bool p2, uint32_t& n1, uint32_t& n2) {
  uint32_t h1 = ht_home(k1, mask), h2 = ht_home(k2, mask);
  n1 = n2 = GRIMB_NONE;
  HSlot a0, a1, b0, b1;
  a0.node = a1.node = b0.node = b1.node = GRIMB_NONE;
  a0.key = a1.key = b0.key = b1.key = 0;
  if (p1) load_sector(base + h1, a0, a1);
  if (p2) load_sector(base + h2, b0, b1);
  bool more1 = false, more2 = false;
  if (p1) {
    if (a0.node == GRIMB_NONE) {}
    else if (a0.key == k1) n1 = a0.node;
    else if (a1.node == GRIMB_NONE) {}
    else if (a1.key == k1) n1 = a1.node;
    else more1 = true;
  }
  if (p2) {
    if (b0.node == GRIMB_NONE) {}
    else if (b0.key == k2) n2 = b0.node;
    else if (b1.node == GRIMB_NONE) {}
    else if (b1.key == k2) n2 = b1.node;
    else more2 = true;
  }
  while (more1) {
    h1 = (h1 + 2) & mask;
    load_sector(base + h1, a0, a1);
    more1 = false;
    if (a0.node == GRIMB_NONE) {}
    else if (a0.key == k1) n1 = a0.node;
    else if (a1.node == GRIMB_NONE) {}
    else if (a1.key == k1) n1 = a1.node;
    else more1 = true;
  }
  while (more2) {
    h2 = (h2 + 2) & mask;
    load_sector(base + h2, b0, b1);
    more2 = false;
    if (b0.node == GRIMB_NONE) {}
    else if (b0.key == k2) n2 = b0.node;
    else if (b1.node == GRIMB_NONE) {}
    else if (b1.key == k2) n2 = b1.node;
    else more2 = true;
  }
}

// One 32-byte sector of the FastIndex (four keys) with one 256-bit load (sm_100: LDG.E.256).
__device__ __forceinline__ void fidx_sector(const uint64_t* p, uint64_t (&w)[4]) {
  uint32_t r0, r1, r2, r3, r4, r5, r6, r7;
  asm volatile("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3), "=r"(r4), "=r"(r5), "=r"(r6), "=r"(r7)
               : "l"(p));
  w[0] = (uint64_t)r0 | ((uint64_t)r1 << 32);
  w[1] = (uint64_t)r2 | ((uint64_t)r3 << 32);
  w[2] = (uint64_t)r4 | ((uint64_t)r5 << 32);
  w[3] = (uint64_t)r6 | ((uint64_t)r7 << 32);
}

// Examines sector `sec` of a probe for `key` (never 0): sets pos to the slot on a hit; returns true when
// the next sector is needed -- no hit, no empty slot, and (home sector) the overflow flag set.
__device__ __forceinline__ bool fidx_step(const uint64_t (&w)[4], uint64_t key, uint32_t sec, bool home, uint32_t& pos) {
  const uint64_t w0 = w[0] & ~FIDX_FLAG;
  if (w0 == key) pos = 4 * sec;
  else if (w[1] == key) pos = 4 * sec + 1;
  else if (w[2] == key) pos = 4 * sec + 2;
  else if (w[3] == key) pos = 4 * sec + 3;
  else return !(w0 == 0 || w[1] == 0 || w[2] == 0 || w[3] == 0) && (!home || (w[0] & FIDX_FLAG));
  return false;
}

// Two independent FastIndex probes; the home sector of each is requested before either is examined (the
// common case resolves both in that one round trip).  n1 / n2: slot positions, GRIMB_NONE when absent.
__device__ __forceinline__ void fidx_lookup2(const FastIndex& X, uint64_t k1, bool p1, uint64_t k2, bool p2, uint32_t& n1,
                                             uint32_t& n2) {
  uint32_t h1 = hash_key(k1) & X.sec_mask, h2 = hash_key(k2) & X.sec_mask;
  n1 = n2 = GRIMB_NONE;
  uint64_t a[4] = {0, 0, 0, 0}, b[4] = {0, 0, 0, 0};
  if (p1) fidx_sector(X.keys + 4ull * h1, a);
  if (p2) fidx_sector(X.keys + 4ull * h2, b);
  bool more1 = p1 && fidx_step(a, k1, h1, true, n1);
  bool more2 = p2 && fidx_step(b, k2, h2, true, n2);
  while (more1) {
    h1 = (h1 + 1) & X.sec_mask;
    fidx_sector(X.keys + 4ull * h1, a);
    more1 = fidx_step(a, k1, h1, false, n1);
  }
  while (more2) {
    h2 = (h2 + 1) & X.sec_mask;
    fidx_sector(X.keys + 4ull * h2, b);
    more2 = fidx_step(b, k2, h2, false, n2);
  }
}

__device__ __forceinline__ uint64_t half_or64(uint32_t hmask, uint64_t v) {
  const uint32_t lo = __reduce_or_sync(hmask, (uint32_t)v), hi = __reduce_or_sync(hmask, (uint32_t)(v >> 32));
  return (uint64_t)lo | ((uint64_t)hi << 32);
}

// Row space is claimed per HALF-WARP in chunks (one global atomicAdd per FAST_CHUNK rows), so the
// kernel has no CTA barrier and no per-subject global atomic; the unused tail of a chunk is a
// hole in the row arrays (offsets are explicit per subject, so holes are harmless).
#ifndef GRIMB_FAST_CHUNK
#define GRIMB_FAST_CHUNK 32
#endif
constexpr uint32_t FAST_CHUNK = GRIMB_FAST_CHUNK;

// Half-warp per subject: lane i (0..15) of a half owns phase i and probes both of its haplotypes
// (side choice i and its complement), so a warp imputes two subjects at once.  Keys are built
// cooperatively: lane l < L shifts the two alleles of locus l into place, two OR-reductions give
// k0 (all side-0 alleles) and k1 (all side-1 alleles), and phase i's haplotypes are
// k0 ^ (D & M_i) and its complement, with D = k0 ^ k1 and M_i the field mask of the loci i flips
// (a per-lane constant).  All votes / reductions use the half's lane mask.
template <bool LIST>
__global__ void __launch_bounds__(FAST_WARPS * 32, FAST_MIN_BLOCKS)
k_impute_fast(TablesView T, const GrimbConfig* __restrict__ cfg, GrimbBatch B, OutArrays O, uint32_t* worklist,
              unsigned int* worklist_n, const uint32_t* __restrict__ list, const unsigned int* __restrict__ list_n,
              uint32_t s_begin) {
  __shared__ double s_chain[FAST_MAX_ROUNDS];
  __shared__ int s_nchain;
  if (LIST && *list_n == 0u) return;   // empty overflow list (the usual case): nothing to set up
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int half = lane >> 4, i = lane & 15, hbase = half << 4;
  const uint32_t hmask = 0xFFFFu << hbase;
  const int L = T.L;
  const uint32_t full = (1u << L) - 1u;
  const int nphase = 1 << (L - 1);
  GrimbResults& R = O.r;
  const bool want_u = cfg->output_umug != 0, want_p = cfg->output_pmug != 0, planb = cfg->planb != 0;
  const uint32_t lim_r = (uint32_t)cfg->n_results, lim_p = (uint32_t)cfg->n_pop_results;
  if (threadIdx.x == 0) {
    // epsilon chain of call_comp_phase_prob (impute.py:1665-1673): repeated FP64 /= 10
    double e = cfg->epsilon;
    int n = 0;
    while (e > 0 && n < FAST_MAX_ROUNDS) {
      e /= 10;
      if (e < 1.0e-9) e = 0.0;
      s_chain[n++] = e;
    }
    s_nchain = (e > 0) ? -1 : n;  // -1: schedule too long for this kernel -> general kernel
  }
  __syncthreads();
  const int nchain = s_nchain;
  // per-lane constants: this lane's locus (shift, dictionary size) and its phase's flip mask
  const uint32_t my_shift = i < L ? T.shift[i] : 0u;
  const uint32_t my_nal = i < L ? T.n_alleles[i] : 0u;
  uint64_t Mi = 0;
  for (int l = 0; l < L; ++l)
    if ((i >> l) & 1) Mi |= ((1ull << T.width[l]) - 1ull) << T.shift[l];
  const uint64_t Mlast = ((1ull << T.width[L - 1]) - 1ull) << T.shift[L - 1];
  const uint32_t ht_mask = T.ht_mask[full];
  const HSlot* __restrict__ ht_base = T.slots + T.ht_off[full];
  // with `list` the kernel serves the listed subjects only (overflow of the split fast path)
  const uint64_t S = LIST ? (uint64_t)*list_n : (uint64_t)B.n_subjects;
  const uint64_t stride = (uint64_t)gridDim.x * FAST_WARPS * 2;
  uint64_t hap_base = 0, pop_base = 0;   // this half-warp's current chunks (uniform within the half)
  uint32_t hap_left = 0, pop_left = 0;
  // without a list the kernel serves the subjects [s_begin, n_subjects)
  uint64_t s = (LIST ? 0ull : (uint64_t)s_begin) + ((uint64_t)blockIdx.x * FAST_WARPS + warp) * 2 + half;
  FastIn nxt;
  uint64_t sx_next = 0;
  if (s < S) {
    sx_next = LIST ? (uint64_t)list[s] : s;
    fast_load(nxt, B, sx_next, L, i, T);
  }
  for (; s < S; s += stride) {   // the two halves may leave the loop one iteration apart
    const FastIn in = nxt;
    const uint64_t sx = sx_next;   // the subject this iteration serves
    if (s + stride < S) {
      sx_next = LIST ? (uint64_t)list[s + stride] : s + stride;
      fast_load(nxt, B, sx_next, L, i, T);
    }
    bool done = false;  // finished here (rows, an empty result, or a skipped subject)
    uint32_t acc = 0, rank = 0, n_acc = 0, evals = 0, gsel = 0;
    uint64_t key = 0, key2 = 0, D = 0;
    double prob = 0.0, total = 0.0;
    const uint32_t typed = in.typed;
    bool shape = typed == full && nchain >= 0;
    shape = __all_sync(hmask, in.c == 0x00010001u) && shape;
    if (shape) {
      const uint32_t a0 = in.pair & 0xffffu, a1 = in.pair >> 16;   // lanes >= L hold 0, 0
      const uint64_t k0 = half_or64(hmask, (uint64_t)a0 << my_shift);
      const uint64_t k1 = half_or64(hmask, (uint64_t)a1 << my_shift);
      const uint32_t unk0 = (__ballot_sync(hmask, i < L && (a0 - 1u) >= my_nal) >> hbase) & 0xFFFFu;
      const uint32_t unk1 = (__ballot_sync(hmask, i < L && (a1 - 1u) >= my_nal) >> hbase) & 0xFFFFu;
      const uint32_t het = (__ballot_sync(hmask, a0 != a1) >> hbase) & 0xFFFFu;
      gsel = (__ballot_sync(hmask, a0 > a1) >> hbase) & 0xFFFFu;
      D = k0 ^ k1;
      key = k0 ^ (D & Mi);    // side 1 of phase i takes the side-1 allele at the loci i flips
      key2 = key ^ D;
      const uint32_t ib = (uint32_t)i;
      const bool known1 = ((unk0 & ~ib) | (unk1 & ib)) == 0, known2 = ((unk1 & ~ib) | (unk0 & ib)) == 0;
      const uint32_t low = het & ((uint32_t)nphase - 1u);
      const bool last_het = (het >> (L - 1)) & 1u;
      // the last locus never flips: phases are i < 2^(L-1); homozygous loci collapse phases
      const bool kept = i < nphase && !(ib & ~low) && (last_het || ib <= (low ^ ib));
      // side 2 is only probed when side 1 exists (comp_phase_prob_*: `if len(Prob1) > 0`); probing
      // both at once returns the same lists
      uint32_t n1, n2;
      ht_lookup2(ht_base, ht_mask, key, kept && known1, key2, kept && known2, n1, n2);
      FastPair pr;
      pr.f = n1 != GRIMB_NONE ? __ldg(T.freq + n1) : 0.0;   // P == 1
      pr.f2 = n2 != GRIMB_NONE ? __ldg(T.freq + n2) : 0.0;
      const bool cand = kept && pr.f > 0 && pr.f2 > 0;
      const uint32_t ncand = __popc(__ballot_sync(hmask, cand));
      const double m = in.m;
      pr.same = D == 0;
      pr.mpos = m > 0;
      pr.y = m * pr.f2;
      {
        const double t = fmin(pr.f2, pr.same ? pr.y * 0.5 : pr.y);
        const double b = pr.f * t;
        const bool tiny = !(b > 1.0e-280);
        pr.lo = tiny ? -1.0 : b * (1.0 - 0x1p-50);
        pr.hi = tiny ? __longlong_as_double(0x7ff0000000000000LL) : b * (1.0 + 0x1p-50);
      }
      if (cand) {
        prob = pr.f * pr.f2 * m;
        if (!pr.same) prob = prob * 2;
      }
      // first round of the schedule at which this pair is accepted (acceptance is monotone in eps)
      uint32_t r_mine = 99;
      if (cand && pr.mpos) {
        // rounds whose epsilon is above the proven band are rejections; the exact test only runs
        // for an epsilon inside the band
        int r = 0;
        while (r < nchain && s_chain[r] >= pr.hi) ++r;
        while (r < nchain && !pr.accept(s_chain[r])) ++r;
        if (r < nchain) r_mine = (uint32_t)r;
      }
      const uint32_t r_star = __reduce_min_sync(hmask, r_mine);
      if (r_star == 99) {
        evals = ncand * (uint32_t)nchain;
      } else {
        evals = ncand * (r_star + 1);
        bool a = r_mine <= r_star;
        if (s_chain[r_star] > 0) {
          // MaxProb of that round -> epsilon = MaxProb / 100000, one more evaluation (impute.py:1683-1693)
          const uint32_t hi = a ? (uint32_t)__double2hiint(prob) : 0u;
          const uint32_t mh = __reduce_max_sync(hmask, hi);
          const uint32_t lo = (a && hi == mh) ? (uint32_t)__double2loint(prob) : 0u;
          const uint32_t ml = __reduce_max_sync(hmask, lo);
          const double eps = __hiloint2double((int)mh, (int)ml) / 100000;
          a = cand && pr.accept(eps);
          evals += ncand;
        }
        acc = (__ballot_sync(hmask, a) >> hbase) & 0xFFFFu;
      }
      if (acc == 0 && planb) {
        shape = false;  // Plan B / C: general kernel
      } else {
        done = true;
        n_acc = __popc(acc);
        // += in phase order; rank by (probability desc, phase asc)
        bool first = true;
        for (uint32_t mm = acc; mm; mm &= mm - 1) {
          const int j = __ffs(mm) - 1;
          const double pj = __shfl_sync(hmask, prob, hbase + j);
          if (first) {
            total = pj;
            first = false;
          } else {
            total = total + pj;
          }
          if (pj > prob || (pj == prob && j < i)) ++rank;
        }
        if (want_u && want_p) evals *= 2;  // the reference evaluates once per output kind
      }
    }
    if (!shape) {
      if (typed != 0) {
        if (i == 0) worklist[atomicAdd(worklist_n, 1u)] = (uint32_t)sx;
      } else {
        done = true;  // GRIMB_ST_SKIPPED
      }
    }
    if (!done) continue;
    const bool rows = typed != 0 && n_acc != 0;
    const uint32_t nu = (rows && want_u) ? (lim_r < 1u ? lim_r : 1u) : 0u;
    const uint32_t np = (rows && want_p) ? (n_acc < lim_r ? n_acc : lim_r) : 0u;
    const uint32_t nup = (rows && want_u) ? (lim_p < 1u ? lim_p : 1u) : 0u;
    const uint32_t npp = (rows && want_p) ? (lim_p < 1u ? lim_p : 1u) : 0u;
    const uint32_t nh = nu + np, npop = nup + npp;
    if (nh > hap_left) {  // uniform within the half: refill its chunk
      unsigned long long b = 0;
      const uint32_t take = nh > FAST_CHUNK ? nh : FAST_CHUNK;
      if (i == 0) b = atomicAdd(O.hap_counter, (unsigned long long)take);
      hap_base = __shfl_sync(hmask, b, hbase);
      hap_left = take;
    }
    if (npop > pop_left) {
      unsigned long long b = 0;
      const uint32_t take = npop > FAST_CHUNK ? npop : FAST_CHUNK;
      if (i == 0) b = atomicAdd(O.pop_counter, (unsigned long long)take);
      pop_base = __shfl_sync(hmask, b, hbase);
      pop_left = take;
    }
    const uint64_t hb = hap_base, pb = pop_base;
    hap_base += nh;
    hap_left -= nh;
    pop_base += npop;
    pop_left -= npop;
    if (i == 0) {
      if (!typed) {
        R.compact[sx] = make_compact(GRIMB_ST_SKIPPED, GRIMB_KIND_GENERAL, 0, 0xFFFFFFFFu, 0.0);
      } else {
        GrimbSubjectResult o;
        o.status = GRIMB_ST_OK;
        o.plan_umug = want_u ? GRIMB_PLAN_A : GRIMB_PLAN_NONE;
        o.plan_pmug = want_p ? GRIMB_PLAN_A : GRIMB_PLAN_NONE;
        o.reserved = 0;
        o.n_umug = nu;
        o.n_pmug = np;
        o.n_umug_pops = nup;
        o.n_pmug_pops = npp;
        o.tot_umug = (want_u && n_acc) ? 1u : 0u;
        o.tot_pmug = want_p ? n_acc : 0u;
        o.pair_evals = evals;
        o.hap_off = hb;
        o.pop_off = pb;
        publish_general(O, sx, o);
      }
    }
    if ((int64_t)(hb + nh) <= R.hap_capacity) {
      // the single UMUG genotype, per-locus (min, max) of the two typed alleles: the lane whose
      // phase flips exactly the loci with a0 > a1 already holds it, up to the last locus
      if (nu && (uint32_t)i == (gsel & ((uint32_t)nphase - 1u))) {
        const uint64_t fix = ((gsel >> (L - 1)) & 1u) ? (D & Mlast) : 0ull;
        GrimbHapRow o;
        o.a = key ^ fix;
        o.b = key2 ^ fix;
        o.prob = total;
        R.hap_rows[hb] = o;
      }
      if ((acc >> i & 1u) && rank < np) {
        GrimbHapRow o;
        o.a = key;
        o.b = key2;
        o.prob = prob;
        R.hap_rows[hb + nu + rank] = o;
      }
    }
    if ((int64_t)(pb + npop) <= R.pop_capacity && i < (int)npop) {
      GrimbPopRow o;
      o.pop_a = 0;
      o.pop_b = 0;
      o.pad = 0;
      o.prob = total;
      R.pop_rows[pb + i] = o;
    }
  }
}


// ------------------------------------------------------------------------------------------
// Split form of the fast path: k_fast_probe (half-warp per subject: keys, FastIndex probes) hands the
// few phases whose two haplotypes are both in the table to k_fast_score (one LANE per subject: frequency
// loads, epsilon schedule, sums, ranks, result record and rows).  The probe kernel carries no FP64
// state, so it fits more warps per SM, and the scoring work -- which used 16 lanes per subject for
// what is typically one or two candidate phases -- shrinks to a few instructions per subject.
// Hand-over record: 48 bytes per subject in a device buffer owned by the engine.
// ------------------------------------------------------------------------------------------
constexpr int FAST_CMAX = 4;    // candidate phases k_fast_score keeps in registers (the usual subject has one or two)
constexpr int FAST_CALL = 16;   // candidate phases a hand-over record holds (= every phase of a 5-locus subject)

// A candidate is the FastIndex slot positions (p1, p2) of its two haplotypes; k_fast_score reads their
// frequencies from FastIndex.fslot.  The record is split: a dense array of 16-byte heads (flags and the
// first candidate), which is all the usual subject (one candidate phase) touches, and a 32-byte record for
// candidates 2..4.  A subject with more than FAST_CMAX candidate phases (rare) keeps them in a side
// record claimed from `extra`.
struct __align__(16) FastHead {
  uint32_t flags;        // bits 0-1 state (0 not for k_fast_score, 1 ready), 2-6 ncand, 7 both haplotypes equal,
                         // 16-31 candidate mask (bit i: phase i; candidates are stored in ascending phase order)
  uint32_t extra;        // ncand > FAST_CMAX: index of the subject's FastExtra
  uint2 p0;              // (p1, p2) of the first candidate phase
};
struct __align__(32) FastMore {
  uint2 p[FAST_CMAX - 1];   // candidates 2..FAST_CMAX (ncand <= FAST_CMAX)
  uint2 pad;
};
struct FastMid {
  FastHead* head;
  FastMore* more;
};
struct __align__(32) FastExtra {
  uint2 p[FAST_CALL];
};

#ifndef FASTPROBE_MIN_BLOCKS
#define FASTPROBE_MIN_BLOCKS 6   /* 40 registers, 48 warps/SM: 0.373 ms vs 0.385 at 5 CTAs (48 registers), 0.418 at 7 */
#endif

// inputs of the probe kernel (no prior: k_fast_score reads it).  Every typed locus side lists at least
// one allele (GrimbBatch.counts >= 1, include/grimb200.h), so "one allele per side at every locus" is
// allele_off[s+1] - allele_off[s] == 2L and the counts need not be read.
struct ProbeIn {
  uint32_t typed, nall, pair;
  uint64_t k0, k1;   // packed form only
};

// PACKED (include/grimb200.h): the subject is its two packed haplotype keys and a flag word -- no cooperative
// key build, no cross-lane reduction before the probes
template <bool PACKED>
__device__ __forceinline__ void probe_load(ProbeIn& in, const GrimbBatch& B, uint32_t s, int L, int i) {
  if (PACKED) {
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(B.packed_keys) + s);   // the same 16 bytes for the half-warp
    in.k0 = (uint64_t)v.x | ((uint64_t)v.y << 32);
    in.k1 = (uint64_t)v.z | ((uint64_t)v.w << 32);
    in.typed = B.packed_flags[s];
    in.nall = in.pair = 0;
    return;
  }
  in.k0 = in.k1 = 0;
  in.typed = B.typed_mask[s];
  const uint32_t off = B.allele_off[s];
  in.nall = B.allele_off[s + 1] - off;
  in.pair = 0;
  if (i < L && 2u * (uint32_t)i + 2u <= in.nall) {   // only inside the subject's own range
    const uint16_t* al = B.alleles + off + 2 * i;
    in.pair = (off & 1u) ? ((uint32_t)al[0] | ((uint32_t)al[1] << 16)) : *reinterpret_cast<const uint32_t*>(al);
  }
}

template <bool PACKED>
__global__ void __launch_bounds__(FAST_WARPS * 32, FASTPROBE_MIN_BLOCKS)
k_fast_probe(TablesView T, const FastIndex X, GrimbBatch B, OutArrays O, FastMid mid, uint32_t* worklist,
             unsigned int* worklist_n, FastExtra* __restrict__ extra, unsigned int* extra_n, uint32_t extra_cap, int nchain_ok,
             uint32_t s_begin) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int half = lane >> 4, i = lane & 15, hbase = half << 4;
  const uint32_t hmask = 0xFFFFu << hbase;
  const int L = T.L;
  const uint32_t full = (1u << L) - 1u;
  const int nphase = 1 << (L - 1);
  const uint32_t my_shift = i < L ? T.shift[i] : 0u;
  const uint32_t my_nal = i < L ? T.n_alleles[i] : 0u;
  uint64_t Mi = 0;
  for (int l = 0; l < L; ++l)
    if ((i >> l) & 1) Mi |= ((1ull << T.width[l]) - 1ull) << T.shift[l];
  const uint32_t S = (uint32_t)B.n_subjects;               // subject indices fit 32 bits (worklists are uint32)
  const uint32_t stride = gridDim.x * FAST_WARPS * 2;
  uint32_t s = s_begin + (blockIdx.x * FAST_WARPS + warp) * 2 + half;   // subjects [s_begin, n_subjects)
  ProbeIn nxt;
  if (s < S) probe_load<PACKED>(nxt, B, s, L, i);
  for (; s < S; s += stride) {
    const ProbeIn in = nxt;
    if (s + stride < S && s + stride > s) probe_load<PACKED>(nxt, B, s + stride, L, i);
    // packed form: in.typed is the flag word (bit 15 = skip); every subject that is not skipped has the shape
    const uint32_t typed = PACKED ? ((in.typed & 0x8000u) ? 0u : full) : in.typed;
    const bool shape = typed == full && nchain_ok && (PACKED || in.nall == 2u * (uint32_t)L);   // uniform in the half-warp
    uint32_t state = 0, ncand = 0, same = 0, xslot = 0, phases = 0;
    if (shape) {
      uint64_t k0, k1;
      uint32_t unk0, unk1, het;
      if (PACKED) {
        k0 = in.k0;
        k1 = in.k1;
        het = in.typed & 31u;
        unk0 = (in.typed >> 5) & 31u;
        unk1 = (in.typed >> 10) & 31u;
      } else {
        const uint32_t a0 = in.pair & 0xffffu, a1 = in.pair >> 16;
        k0 = half_or64(hmask, (uint64_t)a0 << my_shift);
        k1 = half_or64(hmask, (uint64_t)a1 << my_shift);
        // three per-locus flags in one OR-reduction: byte k of `packed` is the locus mask of flag k
        uint32_t bits = 0;
        if (i < L)
          bits = ((((a0 - 1u) >= my_nal) ? 1u : 0u) | (((a1 - 1u) >= my_nal) ? 0x100u : 0u) | ((a0 != a1) ? 0x10000u : 0u)) << i;
        const uint32_t packed = __reduce_or_sync(hmask, bits);
        unk0 = packed & 0xFFu;
        unk1 = (packed >> 8) & 0xFFu;
        het = (packed >> 16) & 0xFFu;
      }
      same = het == 0u ? 1u : 0u;
      const uint64_t D = k0 ^ k1;
      const uint64_t key = k0 ^ (D & Mi), key2 = key ^ D;
      const uint32_t ib = (uint32_t)i;
      const bool known1 = ((unk0 & ~ib) | (unk1 & ib)) == 0, known2 = ((unk1 & ~ib) | (unk0 & ib)) == 0;
      const uint32_t low = het & ((uint32_t)nphase - 1u);
      const bool last_het = (het >> (L - 1)) & 1u;
      const bool kept = i < nphase && !(ib & ~low) && (last_het || ib <= (low ^ ib));
      uint32_t n1, n2;
      fidx_lookup2(X, key, kept && known1, key2, kept && known2, n1, n2);
      const bool cand = kept && n1 != GRIMB_NONE && n2 != GRIMB_NONE;   // the index holds the haplotypes with f > 0
      const uint32_t cmask = (__ballot_sync(hmask, cand) >> hbase) & 0xFFFFu;
      ncand = __popc(cmask);
      state = 1;
      phases = cmask;   // the candidates' phase ids: k_fast_score reads them off the mask (q-th set bit)
      uint2* dst = nullptr;      // the side record of a long-form subject
      if (ncand > FAST_CMAX) {   // rare: a side record (uniform in the half-warp)
        unsigned int x = 0;
        if (i == 0) x = atomicAdd(extra_n, 1u);
        x = __shfl_sync(hmask, x, hbase);
        xslot = x;
        if (x >= extra_cap) {    // no side record left: the general kernel serves the subject
          state = 0;
          if (i == 0) worklist[atomicAdd(worklist_n, 1u)] = s;
        }
        dst = extra[x < extra_cap ? x : 0].p;
      }
      if (cand && state) {
        const uint32_t slot = __popc(cmask & ((1u << i) - 1u));
        const uint2 v = make_uint2(n1, n2);
        if (dst) dst[slot] = v;
        else if (slot == 0) mid.head[s].p0 = v;
        else mid.more[s].p[slot - 1] = v;
      }
    }
    if (!shape && typed != 0) {
      if (i == 0) worklist[atomicAdd(worklist_n, 1u)] = s;
    }
    if (i == 0) {
      if (typed == 0)   // GRIMB_ST_SKIPPED: finished here
        O.r.compact[s] = make_compact(GRIMB_ST_SKIPPED, GRIMB_KIND_GENERAL, 0, 0xFFFFFFFFu, 0.0);
      uint2 h1;   // header: state and candidate bookkeeping (p0 is written by the first candidate's lane)
      h1.x = state | (ncand << 2) | (same << 7) | (phases << 16);
      h1.y = xslot;
      *reinterpret_cast<uint2*>(mid.head + s) = h1;
    }
  }
}

// ---- two-level form of k_fast_probe (packed batches; the default, GRIMB_FAST_PROBE=1 selects the kernel above).
// A phase is a candidate only when BOTH of its haplotypes are in the table, and the usual first haplotype is not
// (DESIGN §4: 1.5 of ~14 eligible phases per subject hit).  Level 1 probes the first haplotype of every eligible
// phase; each hit appends (second key, p1, subject, phase) to a per-warp queue in shared memory, and the queue is
// drained 32 entries at a time, one second probe per lane, with its loads in flight together with the next
// iteration's level-1 loads.  The hand-over record is the one k_fast_probe writes, bit for bit.
// Warp-uniform by construction: the loop runs while the warp's first subject is < S, every lane takes every
// branch that holds a __shfl / __ballot / __match_any / __syncwarp, and lanes of subjects >= S only mask.
#ifndef FASTPROBE2_MIN_BLOCKS
#define FASTPROBE2_MIN_BLOCKS 4   /* 63 registers, 0 spills, 32 warps/SM: 0.146 ms vs 0.196 at 5 CTAs (48 registers,
                                     130 B spilled), 0.282 at 6 (40 registers, 238 B spilled) */
#endif
constexpr uint32_t PQ_CAP = 128;   // queue entries per warp (a power of two; the bound is argued at the drain)
constexpr uint32_t PQ_DRAIN = 32;  // a drain serves at most one entry per lane
constexpr uint32_t PQ_HIGH = 64;   // after an iteration's enqueue the warp drains (without overlap) while >= this

struct ProbeQueue {
  uint64_t key[PQ_CAP];   // the second haplotype of the phase
  uint32_t p1[PQ_CAP];    // FastIndex slot of the first haplotype
  uint32_t s[PQ_CAP];     // subject
  uint8_t ph[PQ_CAP];     // phase
};

// one queue entry per lane, its second probe's home sector requested (what the entry holds besides the key is
// read again from the queue when the sector has arrived)
struct Drain {
  uint64_t key, w[4];
  uint32_t sec;
  bool v;
};

// Entries [qh, qh + min(qn, 32)) of the ring, less the entries of the subject that continues past the window:
// entries of one subject are contiguous and at most 16, so a drain of a queue holding more than 32 entries
// takes at least 17 and only whole subjects.  Reads stay within the qn <= 110 live entries (see the loop).
__device__ __forceinline__ void drain_issue(const ProbeQueue& q, const FastIndex& X, uint32_t qh, uint32_t qn, int lane,
                                            Drain& d) {
  const uint32_t e = (qh + (uint32_t)lane) & (PQ_CAP - 1u);
  d.v = (uint32_t)lane < qn;   // lane < 32
  if (qn > PQ_DRAIN && q.s[e] == q.s[(qh + PQ_DRAIN) & (PQ_CAP - 1u)]) d.v = false;   // entry 32 is live when qn > 32
  d.key = q.key[e];
  d.sec = hash_key(d.key) & X.sec_mask;
  d.w[0] = d.w[1] = d.w[2] = d.w[3] = 0;
  if (d.v) fidx_sector(X.keys + 4ull * d.sec, d.w);
}

// The second probes of a drain resolved; each subject of the window gets its hand-over record (same layout and
// values as k_fast_probe).  Returns the entries consumed.  Called by all 32 lanes.
__device__ __forceinline__ uint32_t drain_finish(const ProbeQueue& q, Drain& d, const FastIndex& X, uint32_t qh, FastMid mid,
                                                 uint32_t* worklist, unsigned int* worklist_n, FastExtra* __restrict__ extra,
                                                 unsigned int* extra_n, uint32_t extra_cap, int lane) {
  const uint32_t FULL = 0xFFFFFFFFu;
  uint32_t p2 = GRIMB_NONE;
  bool more = d.v && fidx_step(d.w, d.key, d.sec, true, p2);
  while (more) {   // continuation sectors (rare; per lane, no warp collective inside)
    d.sec = (d.sec + 1) & X.sec_mask;
    fidx_sector(X.keys + 4ull * d.sec, d.w);
    more = fidx_step(d.w, d.key, d.sec, false, p2);
  }
  const uint32_t e = (qh + (uint32_t)lane) & (PQ_CAP - 1u);
  // subject indices are < S <= 2^32 - 1: the invalid lanes' marker never equals a valid lane's subject
  const uint32_t s = d.v ? q.s[e] : 0xFFFFFFFFu;
  const bool cand = d.v && p2 != GRIMB_NONE;
  const uint32_t taken = __ballot_sync(FULL, d.v);
  const uint32_t grp = __match_any_sync(FULL, s);   // the lanes of my subject: contiguous (invalid lanes: the tail)
  const uint32_t cb = __ballot_sync(FULL, cand) & grp;
  const int leader = __ffs(grp) - 1;
  const uint32_t ncand = __popc(cb);
  // phase mask of the subject's candidates: segmented OR over the group (contiguous, <= 16 lanes)
  uint32_t cm = cand ? (1u << q.ph[e]) : 0u;
#pragma unroll
  for (int k = 1; k < 16; k <<= 1) {
    const uint32_t t = __shfl_down_sync(FULL, cm, k);
    if (((grp >> lane) >> k) & 1u) cm |= t;   // lane + k is in my group (0 past lane 31)
  }
  const bool lead = d.v && lane == leader;
  const bool longf = ncand > (uint32_t)FAST_CMAX;   // uniform in the group
  unsigned int x = 0;
  if (lead && longf) x = atomicAdd(extra_n, 1u);
  x = __shfl_sync(FULL, x, leader);
  const bool ok = !longf || x < extra_cap;   // no side record left: the general kernel serves the subject
  if (cand && ok) {
    const uint32_t slot = __popc(cb & ((1u << lane) - 1u));
    const uint2 v = make_uint2(q.p1[e], p2);
    if (longf) extra[x].p[slot] = v;
    else if (slot == 0) mid.head[s].p0 = v;
    else mid.more[s].p[slot - 1] = v;
  }
  if (lead) {
    if (!ok) worklist[atomicAdd(worklist_n, 1u)] = s;
    uint2 h1;
    h1.x = (ok ? 1u : 0u) | (ncand << 2) | (cm << 16);   // same = 0: homozygous subjects never enter the queue
    h1.y = longf ? x : 0u;
    *reinterpret_cast<uint2*>(mid.head + s) = h1;
  }
  return __popc(taken);
}

__global__ void __launch_bounds__(FAST_WARPS * 32, FASTPROBE2_MIN_BLOCKS)
k_fast_probe2(TablesView T, const FastIndex X, GrimbBatch B, OutArrays O, FastMid mid, uint32_t* worklist,
              unsigned int* worklist_n, FastExtra* __restrict__ extra, unsigned int* extra_n, uint32_t extra_cap,
              int nchain_ok, uint32_t s_begin) {
  __shared__ ProbeQueue s_q[FAST_WARPS];
  const uint32_t FULL = 0xFFFFFFFFu;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int half = lane >> 4, i = lane & 15;
  ProbeQueue& q = s_q[warp];
  const int L = T.L;
  const int nphase = 1 << (L - 1);
  uint64_t Mi = 0;
  for (int l = 0; l < L; ++l)
    if ((i >> l) & 1) Mi |= ((1ull << T.width[l]) - 1ull) << T.shift[l];
  const uint32_t ib = (uint32_t)i;
  const uint32_t lt = (1u << lane) - 1u;
  const uint32_t S = (uint32_t)B.n_subjects;   // subject indices fit 32 bits (worklists are uint32)
  const uint32_t stride = gridDim.x * FAST_WARPS * 4;
  // the warp serves subjects s0 .. s0+3 per iteration: lane (half h, phase i) owns phase i of s0+h and s0+2+h.
  // s0 < S in the loop, so "s0 + k < S" is written S - s0 > k (no 32-bit overflow)
  uint32_t s0 = s_begin + (blockIdx.x * FAST_WARPS + warp) * 4;
  uint32_t qh = 0, qn = 0;   // ring head and fill (warp-uniform)
  uint4 nk[2];
  uint32_t nf[2];
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    nk[u] = make_uint4(0u, 0u, 0u, 0u);
    nf[u] = 0x8000u;
    if (s0 < S && S - s0 > (uint32_t)(2 * u + half)) {
      nk[u] = __ldg(reinterpret_cast<const uint4*>(B.packed_keys) + s0 + 2 * u + half);
      nf[u] = B.packed_flags[s0 + 2 * u + half];
    }
  }
  Drain d;
  while (s0 < S) {
    // level 1: phase i's first haplotype, for both subjects of the lane; both sectors requested before either is examined
    uint64_t key[2], key2[2], w[2][4];
    uint32_t sec[2], cf[2];
    bool pr[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const uint32_t fl = cf[u] = nf[u];
      const bool shape = S - s0 > (uint32_t)(2 * u + half) && !(fl & 0x8000u) && nchain_ok;   // packed: not skipped = shape
      const uint64_t k0 = (uint64_t)nk[u].x | ((uint64_t)nk[u].y << 32), k1 = (uint64_t)nk[u].z | ((uint64_t)nk[u].w << 32);
      const uint32_t het = fl & 31u, unk0 = (fl >> 5) & 31u, unk1 = (fl >> 10) & 31u;
      const uint64_t D = k0 ^ k1;
      key[u] = k0 ^ (D & Mi);
      key2[u] = key[u] ^ D;
      const bool known1 = ((unk0 & ~ib) | (unk1 & ib)) == 0, known2 = ((unk1 & ~ib) | (unk0 & ib)) == 0;
      const uint32_t low = het & ((uint32_t)nphase - 1u);
      const bool last_het = (het >> (L - 1)) & 1u;
      const bool kept = i < nphase && !(ib & ~low) && (last_het || ib <= (low ^ ib));
      // a phase with an unknown allele on either side cannot be a candidate: not probed at all
      pr[u] = shape && kept && known1 && known2;
      sec[u] = hash_key(key[u]) & X.sec_mask;
      w[u][0] = w[u][1] = w[u][2] = w[u][3] = 0;
      if (pr[u]) fidx_sector(X.keys + 4ull * sec[u], w[u]);
    }
    // level 2, overlapped: a queue holding 32 or more entries is drained with this iteration's level-1 loads in flight
    const bool drain_now = qn >= PQ_DRAIN;
    if (drain_now) drain_issue(q, X, qh, qn, lane, d);
    uint32_t p1[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      p1[u] = GRIMB_NONE;
      bool more = pr[u] && fidx_step(w[u], key[u], sec[u], true, p1[u]);
      while (more) {
        sec[u] = (sec[u] + 1) & X.sec_mask;
        fidx_sector(X.keys + 4ull * sec[u], w[u]);
        more = fidx_step(w[u], key[u], sec[u], false, p1[u]);
      }
    }
    // the next iteration's inputs, requested once the level-1 sectors are consumed (fewer registers at the peak)
    const bool last = stride >= S - s0;
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      nf[u] = 0x8000u;
      if (!last && S - s0 - stride > (uint32_t)(2 * u + half)) {
        nk[u] = __ldg(reinterpret_cast<const uint4*>(B.packed_keys) + s0 + stride + 2 * u + half);
        nf[u] = B.packed_flags[s0 + stride + 2 * u + half];
      }
    }
    if (drain_now) {
      const uint32_t n = drain_finish(q, d, X, qh, mid, worklist, worklist_n, extra, extra_n, extra_cap, lane);
      qh += n;
      qn -= n;
      __syncwarp();   // the drained entries were read before this iteration's enqueue may reuse their slots
    }
    // level-1 results.  Homozygous subjects (both haplotypes one key) are decided here, as are subjects without a
    // level-1 hit; the others enqueue one entry per hit phase, subject by subject (ballot order: s0, s0+1, s0+2, s0+3)
    uint32_t base = qh + qn;
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const uint32_t s = s0 + 2 * u + half;
      const uint32_t fl = cf[u];
      const bool inb = S - s0 > (uint32_t)(2 * u + half);
      const bool shape = inb && !(fl & 0x8000u) && nchain_ok;
      const bool same = (fl & 31u) == 0u;
      const bool hit = p1[u] != GRIMB_NONE;   // pr[u] implied
      const uint32_t enq = __ballot_sync(FULL, hit && !same);
      const uint32_t hh = (enq >> (half << 4)) & 0xFFFFu;   // the level-1 hits of a heterozygous subject
      if (hit && !same) {
        // bound: qn <= 46 after the drain above (see below), plus at most 64 entries this iteration: <= 110 < PQ_CAP
        const uint32_t e = (base + __popc(enq & lt)) & (PQ_CAP - 1u);
        q.key[e] = key2[u];
        q.p1[e] = p1[u];
        q.s[e] = s;
        q.ph[e] = (uint8_t)i;
      }
      base += __popc(enq);
      if (i == 0 && inb) {
        if (!shape) {
          if (fl & 0x8000u)   // GRIMB_ST_SKIPPED: finished here
            O.r.compact[s] = make_compact(GRIMB_ST_SKIPPED, GRIMB_KIND_GENERAL, 0, 0xFFFFFFFFu, 0.0);
          else
            worklist[atomicAdd(worklist_n, 1u)] = s;
          mid.head[s] = FastHead{0u, 0u, make_uint2(0u, 0u)};
        } else if (same) {   // phase 0 only; its second haplotype is its first
          mid.head[s] = FastHead{1u | (hit ? (1u << 2) | (1u << 16) : 0u) | (1u << 7), 0u, make_uint2(p1[u], p1[u])};
        } else if (hh == 0u) {
          mid.head[s] = FastHead{1u, 0u, make_uint2(0u, 0u)};
        }
      }
    }
    qn = base - qh;
    __syncwarp();   // the enqueued entries are visible to every lane of the next drain
    // bound: qn <= 110 here.  Each drain of more than 32 entries takes at least 17, so this leaves qn <= 63, the
    // overlapped drain of the next iteration leaves qn <= 46 (or <= 31 when it does not run) and the next
    // enqueue adds <= 64.  Adversarial batches only: on the benchmark's batch the queue peaks at 56 entries and
    // this loop never runs (tools/probe_queue_sim.py)
    while (qn >= PQ_HIGH) {
      drain_issue(q, X, qh, qn, lane, d);
      const uint32_t n = drain_finish(q, d, X, qh, mid, worklist, worklist_n, extra, extra_n, extra_cap, lane);
      qh += n;
      qn -= n;
      __syncwarp();
    }
    if (last) break;
    s0 += stride;
  }
  while (qn > 0) {   // flush: every entry left belongs to a whole subject
    drain_issue(q, X, qh, qn, lane, d);
    const uint32_t n = drain_finish(q, d, X, qh, mid, worklist, worklist_n, extra, extra_n, extra_cap, lane);
    qh += n;
    qn -= n;
    __syncwarp();
  }
}

// ---- more than FAST_CMAX candidate phases (rare): the WARP serves such a subject together, lane q = candidate q
// (ascending phase), each lane reading its own (p1, p2) from the subject's side record and their frequencies once.
// Same schedule as the per-lane path below: first accepting round per candidate, minimum over the candidates,
// MaxProb / 100000, one more evaluation, += in phase order, ranks by (probability desc, phase asc).
struct LongCand {
  FastPair pr;
  double p;
  bool valid;
};

__device__ __forceinline__ void long_cand(LongCand& c, const FastExtra* ex, const double* __restrict__ fslot, uint32_t q,
                                          uint32_t ncand, double m, bool same) {
  c.valid = q < ncand;
  double2 v = make_double2(0.0, 0.0);
  if (c.valid) {
    const uint2 pp = ex->p[q];
    v.x = __ldg(fslot + pp.x);
    v.y = __ldg(fslot + pp.y);
  }
  c.pr.f = v.x;
  c.pr.f2 = v.y;
  c.pr.same = same;
  c.pr.mpos = c.valid && m > 0;
  c.pr.y = m * c.pr.f2;
  const double t = fmin(c.pr.f2, same ? c.pr.y * 0.5 : c.pr.y);
  const double b = c.pr.f * t;
  const bool tiny = !(b > 1.0e-280);
  c.pr.lo = tiny ? -1.0 : b * (1.0 - 0x1p-50);
  c.pr.hi = tiny ? __longlong_as_double(0x7ff0000000000000LL) : b * (1.0 + 0x1p-50);
  c.p = v.x * v.y * m;
  if (!same) c.p = c.p * 2;
}

__device__ __forceinline__ double shfl_double(double v, int src) {
  const long long b = __double_as_longlong(v);
  const int lo = __shfl_sync(0xFFFFFFFFu, (int)(b & 0xFFFFFFFFll), src), hi = __shfl_sync(0xFFFFFFFFu, (int)(b >> 32), src);
  return __longlong_as_double(((long long)hi << 32) | (unsigned int)lo);
}

struct ScoreLong {
  double total, e_fin;
  uint32_t n_acc, evals;
};

// called by all 32 lanes; every lane returns the same values
__device__ __noinline__ void score_long_eval(const FastExtra* ex, const double* fslot, uint32_t ncand, double m, bool same,
                                             const double* chain, int nchain, ScoreLong& o) {
  const int lane = threadIdx.x & 31;
  LongCand c;
  long_cand(c, ex, fslot, (uint32_t)lane, ncand, m, same);
  uint32_t rq = 99;
  if (c.pr.mpos) {
    int r = 0;
    while (r < nchain && chain[r] >= c.pr.hi) ++r;
    while (r < nchain && !c.pr.accept(chain[r])) ++r;
    if (r < nchain) rq = (uint32_t)r;
  }
  const uint32_t rs = __reduce_min_sync(0xFFFFFFFFu, rq);
  o.total = 0.0;
  o.e_fin = 0.0;
  o.n_acc = 0;
  if (rs == 99) {
    o.evals = ncand * (uint32_t)nchain;
    return;
  }
  o.evals = ncand * (rs + 1);
  bool acc = rq <= rs;
  if (chain[rs] > 0) {   // MaxProb of that round -> epsilon = MaxProb / 100000, one more evaluation
    double mx = acc ? c.p : 0.0;   // probabilities are >= 0: the larger value has the larger bit pattern
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      const double y = shfl_double(mx, lane ^ d);
      mx = y > mx ? y : mx;
    }
    o.e_fin = mx / 100000;
    acc = c.pr.accept(o.e_fin);
    o.evals += ncand;
  }
  uint32_t am = __ballot_sync(0xFFFFFFFFu, acc);
  o.n_acc = (uint32_t)__popc(am);
  bool first = true;
  while (am) {   // += in phase order
    const int j = __ffs(am) - 1;
    am &= am - 1;
    const double pj = shfl_double(c.p, j);
    o.total = first ? pj : o.total + pj;
    first = false;
  }
}

// rows of the long form: words[0] = number of rows, words[1] = their phase ids (rank order), words[2 + k] = probability
__device__ __noinline__ void score_long_rows(const FastExtra* ex, const double* fslot, uint32_t ncand, double m, bool same,
                                             double e_fin, uint32_t cmask, uint32_t np, uint64_t* words) {
  const int lane = threadIdx.x & 31;
  LongCand c;
  long_cand(c, ex, fslot, (uint32_t)lane, ncand, m, same);
  const bool acc = c.pr.accept(e_fin);
  uint32_t am = __ballot_sync(0xFFFFFFFFu, acc);
  uint32_t rank = 0;   // by (probability desc, phase asc)
  while (am) {
    const int j = __ffs(am) - 1;
    am &= am - 1;
    const double pj = shfl_double(c.p, j);
    if (pj > c.p || (pj == c.p && j < lane)) ++rank;
  }
  uint32_t lo = 0, hi = 0;
  if (acc && rank < np) {
    const uint32_t id = __fns(cmask, 0, lane + 1) & 15u;   // phase of candidate `lane`: the lane-th set bit
    if (rank < 8) lo = id << (4 * rank);
    else hi = id << (4 * (rank - 8));
    words[2 + rank] = (uint64_t)__double_as_longlong(c.p);
  }
  lo = __reduce_or_sync(0xFFFFFFFFu, lo);
  hi = __reduce_or_sync(0xFFFFFFFFu, hi);
  if (lane == 0) {
    words[0] = (uint64_t)np;
    words[1] = (uint64_t)lo | ((uint64_t)hi << 32);
  }
}

#ifndef FASTSCORE_MIN_BLOCKS
#define FASTSCORE_MIN_BLOCKS 8   /* 64 registers (a few spilled words): 0.046 ms per 2^20 subjects vs 0.048 at 6 CTAs, 0.052 unbounded (96) */
#endif
__global__ void __launch_bounds__(128, FASTSCORE_MIN_BLOCKS)
k_fast_score(TablesView T, const FastIndex X, const GrimbConfig* __restrict__ cfg, GrimbBatch B, OutArrays O,
             const FastMid mid, const FastExtra* __restrict__ extra, uint32_t* worklist, unsigned int* worklist_n,
             uint32_t s_begin) {
  __shared__ double s_chain[FAST_MAX_ROUNDS];
  __shared__ int s_nchain;
  const int lane = threadIdx.x & 31;
  GrimbResults& R = O.r;
  const bool want_u = cfg->output_umug != 0, want_p = cfg->output_pmug != 0, planb = cfg->planb != 0;
  const uint32_t lim_r = (uint32_t)cfg->n_results;
  if (threadIdx.x == 0) {
    double e = cfg->epsilon;
    int n = 0;
    while (e > 0 && n < FAST_MAX_ROUNDS) {
      e /= 10;
      if (e < 1.0e-9) e = 0.0;
      s_chain[n++] = e;
    }
    s_nchain = (e > 0) ? -1 : n;
  }
  __syncthreads();
  const int nchain = s_nchain;
  const uint64_t S = (uint64_t)B.n_subjects;
  const uint64_t nthreads = (uint64_t)gridDim.x * blockDim.x;
  unsigned long long evals_sum = 0;
  // whole warps iterate together (the word-space claim is a warp scan)
  // subjects [s_begin, n_subjects); s_begin is a multiple of 32
  for (uint64_t s0 = (uint64_t)s_begin + ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) - lane; s0 < S; s0 += nthreads) {
    const uint64_t s = s0 + lane;
    bool ready = false;
    double m = 0.0;
    uint32_t fl = 0, xslot = 0;
    uint32_t cmask = 0;    // candidate phases (bit i: phase i); candidate q is the q-th set bit
    uint2 p0 = make_uint2(0u, 0u);
    if (s < S) {
      // the prior (P == 1: one double per subject) does not depend on the header: requested with it
      const uint4 h1 = *reinterpret_cast<const uint4*>(mid.head + s);   // p0 is garbage unless ncand >= 1
      const uint32_t pi = batch_prior(B, s);
      m = __ldg(B.priors + pi);
      fl = h1.x;
      xslot = h1.y;
      p0 = make_uint2(h1.z, h1.w);
      cmask = fl >> 16;
      ready = (fl & 3u) == 1u;
    }
    const uint32_t ncand_all = ready ? ((fl >> 2) & 31u) : 0u;
    const bool long_form = ncand_all > (uint32_t)FAST_CMAX;   // rare: more candidate phases than the register path keeps
    const uint32_t ncand = long_form ? 0u : ncand_all;
    const bool same = (fl >> 7) & 1u;
    const bool mpos = m > 0;
    ScoreLong sl;   // long form: the warp serves its long-form subjects one after the other
    sl.total = sl.e_fin = 0.0;
    sl.n_acc = sl.evals = 0;
    for (uint32_t lm = __ballot_sync(0xFFFFFFFFu, long_form); lm; lm &= lm - 1) {
      const int o = __ffs(lm) - 1;
      ScoreLong r;
      score_long_eval(extra + __shfl_sync(0xFFFFFFFFu, xslot, o), X.fslot, __shfl_sync(0xFFFFFFFFu, ncand_all, o), shfl_double(m, o),
                      __shfl_sync(0xFFFFFFFFu, (int)same, o) != 0, s_chain, nchain, r);
      if (lane == o) sl = r;
    }
    double pf[FAST_CMAX], pf2[FAST_CMAX], prob[FAST_CMAX];
    uint32_t rq[FAST_CMAX];
    bool acc[FAST_CMAX];
    uint32_t r_star = 99;
    // the candidates' frequencies: every load is issued before any is used
    uint2 pp[FAST_CMAX];
    pp[0] = p0;
#pragma unroll
    for (int q = 1; q < FAST_CMAX; ++q) pp[q] = (uint32_t)q < ncand ? mid.more[s].p[q - 1] : make_uint2(0u, 0u);
#pragma unroll
    for (int q = 0; q < FAST_CMAX; ++q) {
      pf[q] = pf2[q] = 0.0;
      if ((uint32_t)q < ncand) {
        pf[q] = __ldg(X.fslot + pp[q].x);
        pf2[q] = __ldg(X.fslot + pp[q].y);
      }
    }
#pragma unroll
    for (int q = 0; q < FAST_CMAX; ++q) {
      prob[q] = 0.0;
      rq[q] = 99;
      acc[q] = false;
      if ((uint32_t)q < ncand) {
        const double2 v = make_double2(pf[q], pf2[q]);
        FastPair pr;
        pr.f = v.x;
        pr.f2 = v.y;
        pr.same = same;
        pr.mpos = mpos;
        pr.y = m * pr.f2;
        const double t = fmin(pr.f2, same ? pr.y * 0.5 : pr.y);
        const double b = pr.f * t;
        const bool tiny = !(b > 1.0e-280);
        pr.lo = tiny ? -1.0 : b * (1.0 - 0x1p-50);
        pr.hi = tiny ? __longlong_as_double(0x7ff0000000000000LL) : b * (1.0 + 0x1p-50);
        double p = v.x * v.y * m;
        if (!same) p = p * 2;
        prob[q] = p;
        if (mpos) {
          int r = 0;
          while (r < nchain && s_chain[r] >= pr.hi) ++r;
          while (r < nchain && !pr.accept(s_chain[r])) ++r;
          if (r < nchain) rq[q] = (uint32_t)r;
        }
        r_star = rq[q] < r_star ? rq[q] : r_star;
      }
    }
    uint32_t evals = 0, n_acc = 0;
    if (r_star == 99) {
      evals = ncand * (uint32_t)nchain;
    } else {
      evals = ncand * (r_star + 1);
      if (s_chain[r_star] > 0) {
        // MaxProb of that round -> epsilon = MaxProb / 100000, one more evaluation (impute.py:1683-1693)
        double mx = 0.0;
#pragma unroll
        for (int q = 0; q < FAST_CMAX; ++q)
          if (rq[q] <= r_star && prob[q] > mx) mx = prob[q];
        const double eps = mx / 100000;
#pragma unroll
        for (int q = 0; q < FAST_CMAX; ++q)
          if ((uint32_t)q < ncand) {
            FastPair pr;
            pr.f = pf[q];
            pr.f2 = pf2[q];
            pr.same = same;
            pr.mpos = mpos;
            pr.y = m * pr.f2;
            const double t = fmin(pr.f2, same ? pr.y * 0.5 : pr.y);
            const double b = pr.f * t;
            const bool tiny = !(b > 1.0e-280);
            pr.lo = tiny ? -1.0 : b * (1.0 - 0x1p-50);
            pr.hi = tiny ? __longlong_as_double(0x7ff0000000000000LL) : b * (1.0 + 0x1p-50);
            acc[q] = pr.accept(eps);
          }
        evals += ncand;
      } else {
#pragma unroll
        for (int q = 0; q < FAST_CMAX; ++q) acc[q] = rq[q] <= r_star;
      }
    }
    double total = 0.0;
    bool first = true;
#pragma unroll
    for (int q = 0; q < FAST_CMAX; ++q)
      if (acc[q]) {   // += in phase order
        total = first ? prob[q] : total + prob[q];
        first = false;
        ++n_acc;
      }
    if (long_form) {
      total = sl.total;
      n_acc = sl.n_acc;
      evals = sl.evals;
    }
    if (want_u && want_p) evals *= 2;
    bool done = ready;
    if (ready && n_acc == 0 && planb) {   // Plan B / C: general kernel (which counts its own evaluations)
      worklist[atomicAdd(worklist_n, 1u)] = (uint32_t)s;
      done = false;
    }
    if (done) evals_sum += evals;
    const uint32_t np = (done && n_acc != 0 && want_p) ? (n_acc < lim_r ? n_acc : lim_r) : 0u;
    // PMUG probabilities travel as 8-byte words only when several phases were accepted (with one accepted
    // phase the row's probability is `total`); one claim of word space per warp, and none at all for the
    // usual warp whose subjects all have a single accepted phase
    // (long form: a count word, a word of phase ids, then the probabilities)
    const uint32_t nw = long_form ? (np ? np + 2u : 0u) : ((np != 0u && n_acc >= 2u) ? np : 0u);
    uint32_t sc = nw;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t a = __shfl_up_sync(0xFFFFFFFFu, sc, d);
      if (lane >= d) sc += a;
    }
    const uint32_t wtot = __shfl_sync(0xFFFFFFFFu, sc, 31);
    unsigned long long wb = 0;
    if (wtot) {
      if (lane == 31) wb = atomicAdd(O.word_counter, (unsigned long long)wtot);
      wb = __shfl_sync(0xFFFFFFFFu, wb, 31);
    }
    const uint64_t my = wb + (sc - nw);
    const bool fits = (int64_t)(wb + wtot) <= R.word_capacity;
    for (uint32_t lm = __ballot_sync(0xFFFFFFFFu, long_form && done && np && fits); lm; lm &= lm - 1) {
      const int o = __ffs(lm) - 1;
      const uint32_t ph = __shfl_sync(0xFFFFFFFFu, cmask, o);
      const uint64_t at = (uint64_t)__shfl_sync(0xFFFFFFFFu, (uint32_t)my, o) |
                          ((uint64_t)__shfl_sync(0xFFFFFFFFu, (uint32_t)(my >> 32), o) << 32);
      score_long_rows(extra + __shfl_sync(0xFFFFFFFFu, xslot, o), X.fslot, __shfl_sync(0xFFFFFFFFu, ncand_all, o), shfl_double(m, o),
                      __shfl_sync(0xFFFFFFFFu, (int)same, o) != 0, shfl_double(sl.e_fin, o), ph, __shfl_sync(0xFFFFFFFFu, np, o),
                      R.words + at);
    }
    if (!done) continue;
    uint32_t phases = 0;
    uint32_t mm = cmask;
#pragma unroll
    for (int q = 0; q < FAST_CMAX; ++q) {
      const uint32_t pid = (uint32_t)(__ffs(mm) - 1) & 15u;   // phase id of candidate q
      mm &= mm - 1;
      if (acc[q]) {
        // rank by (probability desc, phase asc); candidates are stored in ascending phase order
        uint32_t rank = 0;
#pragma unroll
        for (int j = 0; j < FAST_CMAX; ++j)
          if (acc[j] && (prob[j] > prob[q] || (prob[j] == prob[q] && j < q))) ++rank;
        if (rank < np) {
          phases |= pid << (4 * rank);
          if (nw && fits) R.words[my + rank] = (uint64_t)__double_as_longlong(prob[q]);
        }
      }
    }
    // the UMUG genotype and the two haplotypes of every PMUG row follow from the subject's own alleles and
    // the phase ids (include/grimb200.h, GRIMB_KIND_SIMPLE): one 16-byte store per subject
    const GrimbCompact c = make_compact(GRIMB_ST_OK, GRIMB_KIND_SIMPLE | (n_acc ? GRIMB_KIND_HAS_RESULTS : 0u) |
                                        (nw ? GRIMB_KIND_WORDS : 0u) | ((long_form ? (np ? 15u : 0u) : np) << 4), phases,
                                        (uint32_t)my, total);
    *reinterpret_cast<uint4*>(R.compact + s) = *reinterpret_cast<const uint4*>(&c);
  }
  // pair evaluations of the subjects finished here: one atomic per warp for the whole launch
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) evals_sum += __shfl_xor_sync(0xFFFFFFFFu, evals_sum, d);
  if (lane == 0 && evals_sum) atomicAdd(O.evals_counter, evals_sum);
}

#endif  // GRIMB_KW == 1

// ------------------------------------------------------------------------------------------
// Typed path: one WARP per subject for fully typed, unambiguous, heterozygous subjects with any
// number of populations P <= 32, any number of loci and either key width (BASELINE configs 3
// and 5).  What the general kernel does with CTA-wide barriers over a global-memory arena is done
// here with the 32 lanes and ~6-10 KB of shared memory per warp:
//   probes      16 phases per pass: lane v < 16 probes the side-1 haplotype of phase base+v, lane
//               16+v its complement (gen_phases, impute.py:274-303; adjs_query, nxg.py:253-278)
//   side lists  lane j = population j: (f, pop) with f > 0, ranked by f*M[j][j] descending, ties by
//               population (convert_list_to_one_dim, impute.py:424-442), capped at K
//   pair test   lane k = position in the side-2 list, loop over h: x = eps / f1[h]; the `break` of
//               the k loop (impute.py:464,545-546) is a prefix-minimum of f2 compared with x
//   schedule    rounds of call_comp_phase_prob (impute.py:1658-1693) until one accepts, MaxProb/1e5
//   sums        hap_total / per-phase PMUG sums in (phase, h, k) order; population-pair sums in
//               shared memory (within one h step the pairs are distinct, so lanes add in parallel and
//               steps are sequential: the reference's += order)
// Subjects of any other shape -- or with more than TY_VP phases whose two haplotypes are both in
// the table, or for which Plan A finds nothing -- go to `worklist` for k_impute.  geno_seen
// de-duplication only matters for a fully homozygous subject (one phase, both haplotypes equal):
// distinct kept phases of a heterozygous subject are distinct unordered haplotype pairs.
// ------------------------------------------------------------------------------------------
constexpr int TY_WARPS = 8;
constexpr int TY_VP = 4;
#ifndef TY_MIN_BLOCKS
#define TY_MIN_BLOCKS 4   /* 64 registers, 32 warps/SM (shared memory allows 4 CTAs at P = 21): 83 M vs 61 M subjects/s at 3 */
#endif
constexpr int TY_MAX_ROUNDS = 40;

struct __align__(16) TyLists {
  uint16_t ph[TY_VP];     // phase id of the kept phase (bit m: locus m takes its side-2 allele in haplotype 1)
  uint16_t ph_pad[4];
  double f1s[TY_VP][32];
  double f2s[TY_VP][32];
  double pm2[TY_VP][32];
  double xs[32];
  uint8_t p1s[TY_VP][32];
  uint8_t p2s[TY_VP][32];
  uint8_t n1[TY_VP], n2[TY_VP];
};

static inline size_t ty_bytes_per_warp(int P) {
  const size_t G = (size_t)P * (P + 1) / 2;
  return (sizeof(TyLists) + G * 12 + 15) & ~(size_t)15;
}

__global__ void __launch_bounds__(TY_WARPS * 32, TY_MIN_BLOCKS)
k_impute_typed(TablesView T, const GrimbConfig* __restrict__ cfg, GrimbBatch B, OutArrays O, uint32_t* worklist,
               unsigned int* worklist_n, uint32_t per_warp, uint32_t s_begin) {
  extern __shared__ __align__(16) unsigned char ty_smem[];
  __shared__ double s_chain[TY_MAX_ROUNDS];
  __shared__ int s_nchain;
  const uint32_t FULLM = 0xFFFFFFFFu;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int L = T.L, P = T.P;
  const int G = P * (P + 1) / 2;
  TyLists& W = *reinterpret_cast<TyLists*>(ty_smem + (size_t)warp * per_warp);
  double* gsum = reinterpret_cast<double*>(ty_smem + (size_t)warp * per_warp + sizeof(TyLists));
  uint16_t* gslot = reinterpret_cast<uint16_t*>(gsum + G);
  uint16_t* gpair = gslot + G;
  GrimbResults& R = O.r;
  const bool want_u = cfg->output_umug != 0, want_p = cfg->output_pmug != 0;
  const uint32_t lim_r = (uint32_t)cfg->n_results, lim_p = (uint32_t)cfg->n_pop_results;
  const int K = cfg->max_haps_in_phase;
  if (threadIdx.x == 0) {
    double e = cfg->epsilon;   // epsilon chain of call_comp_phase_prob (impute.py:1665-1673)
    int n = 0;
    while (e > 0 && n < TY_MAX_ROUNDS) {
      e /= 10;
      if (e < 1.0e-9) e = 0.0;
      s_chain[n++] = e;
    }
    s_nchain = (e > 0) ? -1 : n;
  }
  __syncthreads();
  const int nchain = s_nchain;
  const uint32_t full = (1u << L) - 1u;
  const uint32_t nphase = 1u << (L - 1);
  const uint64_t S = (uint64_t)B.n_subjects;
  unsigned long long evals_sum = 0;   // pair evaluations of the subjects this warp finishes (warp-uniform)
  unsigned long long n_probes = 0, n_hits = 0, n_vecs = 0;   // of every subject this warp looked at (warp-uniform)
  for (uint64_t s = (uint64_t)s_begin + (uint64_t)blockIdx.x * TY_WARPS + warp; s < S; s += (uint64_t)gridDim.x * TY_WARPS) {
    const uint32_t typed = batch_typed(B, s, full);
    if (typed == 0) {   // GRIMB_ST_SKIPPED
      if (lane == 0) R.compact[s] = make_compact(GRIMB_ST_SKIPPED, GRIMB_KIND_GENERAL, 0, 0xFFFFFFFFu, 0.0);
      continue;
    }
    // one allele per side at every locus: every typed side lists >= 1 allele, so the total says it all
    const bool is_packed = B.packed_keys != nullptr;
    const uint32_t al_off = is_packed ? 0u : B.allele_off[s];
    const bool shape = typed == full && nchain >= 0 && (is_packed || B.allele_off[s + 1] - al_off == 2u * (uint32_t)L);
    uint32_t pairs[GRIMB_MAX_LOCI];
    uint32_t het = 0;
    if (shape) {
      const uint16_t* al = B.alleles + al_off;
#if GRIMB_KW == 1
      const uint64_t pk0 = is_packed ? B.packed_keys[2 * s] : 0ull, pk1 = is_packed ? B.packed_keys[2 * s + 1] : 0ull;
#endif
#pragma unroll
      for (int l = 0; l < GRIMB_MAX_LOCI; ++l) {
        pairs[l] = 0;
        if (l < L) {
#if GRIMB_KW == 1
          const uint32_t a0 = is_packed ? (uint32_t)key_field(T, pk0, l) : al[2 * l];
          const uint32_t a1 = is_packed ? (uint32_t)key_field(T, pk1, l) : al[2 * l + 1];
#else
          const uint32_t a0 = al[2 * l], a1 = al[2 * l + 1];
#endif
          pairs[l] = a0 | (a1 << 16);
          if (a0 != a1) het |= 1u << l;
        }
      }
    }
    // het == 0: one phase whose two haplotypes are equal.  Its two side lists are identical, pair
    // (h, k) and pair (k, h) are the same unordered {(hap,pop),(hap,pop)} and geno_seen keeps the
    // first one met (impute.py:508-513); equal haplotypes are not doubled and need m*f2 >= 2x.
    const bool same = het == 0;
    int nvp = 0;
    bool punt = !shape;
    const double* M = B.priors + (uint64_t)batch_prior(B, s) * P * P;
    if (!punt) {
      const double mdiag = lane < P ? __ldg(M + lane * P + lane) : 0.0;
      const uint32_t low = het & (nphase - 1u);
      const bool last_het = (het >> (L - 1)) & 1u;
      for (uint32_t base = 0; base < nphase && !punt; base += 16) {
        const uint32_t v = lane & 15, side = lane >> 4, i = base + v;
        const bool kept = i < nphase && !(i & ~low) && (last_het || i <= (low ^ i));
        hkey key = 0;
        bool known = true;
#pragma unroll
        for (int l = 0; l < GRIMB_MAX_LOCI; ++l)
          if (l < L) {
            const uint32_t a0 = pairs[l] & 0xffffu, a1 = pairs[l] >> 16;
            const uint32_t a = (((i >> l) & 1u) ^ side) ? a1 : a0;   // the last locus never flips
            known = known && (a - 1u) < T.n_alleles[l];
            key |= (hkey)a << T.shift[l];
          }
        const uint32_t node = (kept && known) ? ht_lookup(T, full, key) : GRIMB_NONE;
        const uint32_t hits = __ballot_sync(FULLM, node != GRIMB_NONE);
        n_probes += __popc(__ballot_sync(FULLM, kept && known));
        n_hits += __popc(hits);
        uint32_t both = hits & (hits >> 16) & 0xFFFFu;
        while (both) {
          const int b = __ffs(both) - 1;
          both &= both - 1;
          if (nvp == TY_VP) {
            punt = true;
            break;
          }
          const uint32_t nd1 = __shfl_sync(FULLM, node, b), nd2 = __shfl_sync(FULLM, node, 16 + b);
          n_vecs += 2;
          double f1 = 0.0, f2 = 0.0;
          if (lane < P) {
            f1 = __ldg(T.freq + (uint64_t)nd1 * P + lane);
            f2 = __ldg(T.freq + (uint64_t)nd2 * P + lane);
          }
          const double w1 = f1 * mdiag, w2 = f2 * mdiag;
          const bool v1 = f1 > 0, v2 = f2 > 0;
          const uint32_t vm1 = __ballot_sync(FULLM, v1), vm2 = __ballot_sync(FULLM, v2);
          int n1 = __popc(vm1), n2 = __popc(vm2);
          n1 = n1 < K ? n1 : K;
          n2 = n2 < K ? n2 : K;
          if (n1 == 0 || n2 == 0) continue;   // the phase yields no pairs
          int r1 = 0, r2 = 0;
          for (int j = 0; j < P; ++j) {
            const double u1 = __shfl_sync(FULLM, w1, j), u2 = __shfl_sync(FULLM, w2, j);
            if (((vm1 >> j) & 1u) && (u1 > w1 || (u1 == w1 && j < lane))) ++r1;
            if (((vm2 >> j) & 1u) && (u2 > w2 || (u2 == w2 && j < lane))) ++r2;
          }
          if (v1 && r1 < n1) {
            W.f1s[nvp][r1] = f1;
            W.p1s[nvp][r1] = (uint8_t)lane;
          }
          if (v2 && r2 < n2) {
            W.f2s[nvp][r2] = f2;
            W.p2s[nvp][r2] = (uint8_t)lane;
          }
          if (lane == 0) W.ph[nvp] = (uint16_t)(base + (uint32_t)b);
          __syncwarp();
          double pmv = lane < n2 ? W.f2s[nvp][lane] : 0.0;
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) {
            const double o = __shfl_up_sync(FULLM, pmv, d);
            if (lane >= d && o < pmv) pmv = o;
          }
          if (lane < n2) W.pm2[nvp][lane] = pmv;
          if (lane == 0) {
            W.n1[nvp] = (uint8_t)n1;
            W.n2[nvp] = (uint8_t)n2;
          }
          ++nvp;
        }
      }
      __syncwarp();
      if (nvp == 0) punt = true;   // Plan A has no candidates: Plan B / C
    }
    // ---- epsilon schedule: rounds until one accepts (impute.py:1665-1681)
    uint32_t evals = 0;
    double eps_final = 0.0;
    bool count_final = false;
    if (!punt) {
      int rstar = -1;
      double mx = 0.0;
      for (int r = 0; r < nchain && rstar < 0; ++r) {
        const double eps = s_chain[r];
        bool any = false;
        double lmx = 0.0;
        for (int vp = 0; vp < nvp; ++vp) {
          const int n1 = W.n1[vp], n2 = W.n2[vp];
          __syncwarp();
          if (lane < n1) W.xs[lane] = eps / W.f1s[vp][lane];
          __syncwarp();
          const double f2 = lane < n2 ? W.f2s[vp][lane] : 0.0;
          const double pm = lane < n2 ? W.pm2[vp][lane] : -1.0;
          const uint32_t p2 = W.p2s[vp][lane];
          for (int h = 0; h < n1; ++h) {
            const double x = W.xs[h];
            const bool reach = pm >= x;
            const int cnt = __popc(__ballot_sync(FULLM, reach));
            evals += cnt < n2 ? cnt + 1 : n2;
            if (reach) {
              const double m = __ldg(M + (uint32_t)W.p1s[vp][h] * P + p2);
              if (m > 0 && m * f2 >= (same ? x * 2 : x)) {
                bool dup = false;
                if (same && lane < h) {   // the mirror pair (k, h) comes first: accepted -> this one is a duplicate
                  const double xk = W.xs[lane];
                  const double mk = __ldg(M + p2 * P + (uint32_t)W.p1s[vp][h]);
                  dup = W.pm2[vp][h] >= xk && mk > 0 && mk * W.f2s[vp][h] >= xk * 2;
                }
                if (!dup) {
                  any = true;
                  double pr = W.f1s[vp][h] * f2 * m;
                  if (!same) pr = pr * 2;
                  if (pr > lmx) lmx = pr;
                }
              }
            }
          }
        }
        if (__any_sync(FULLM, any)) {
          rstar = r;
#pragma unroll
          for (int d = 16; d > 0; d >>= 1) {
            const double o = __shfl_xor_sync(FULLM, lmx, d);
            lmx = o > lmx ? o : lmx;
          }
          mx = lmx;
        }
      }
      if (rstar < 0) punt = true;
      else if (s_chain[rstar] > 0) {
        eps_final = mx / 100000;   // impute.py:1683-1693: one more evaluation at MaxProb / 100000
        count_final = true;
      }
    }
    // ---- final evaluation with accumulation in (phase, h, k) order
    uint32_t E = 0, ng = 0, nrows = 0;
    double total = 0.0, my_sum = 0.0;
    int my_vp = 0;
    if (!punt) {
      for (int g = lane; g < G; g += 32) gslot[g] = 0xFFFFu;
      bool have_total = false;
      for (int vp = 0; vp < nvp; ++vp) {
        const int n1 = W.n1[vp], n2 = W.n2[vp];
        __syncwarp();
        if (lane < n1) W.xs[lane] = eps_final / W.f1s[vp][lane];
        __syncwarp();
        const double f2 = lane < n2 ? W.f2s[vp][lane] : 0.0;
        const double pm = lane < n2 ? W.pm2[vp][lane] : -1.0;
        const uint32_t p2 = W.p2s[vp][lane];
        double psum = 0.0;
        bool have_p = false;
        for (int h = 0; h < n1; ++h) {
          const double x = W.xs[h];
          const bool reach = pm >= x;
          if (count_final) {
            const int cnt = __popc(__ballot_sync(FULLM, reach));
            evals += cnt < n2 ? cnt + 1 : n2;
          }
          const uint32_t p1 = W.p1s[vp][h];
          bool a = false;
          double pr = 0.0;
          if (reach) {
            const double m = __ldg(M + p1 * P + p2);
            if (m > 0 && m * f2 >= (same ? x * 2 : x)) {
              bool dup = false;
              if (same && lane < h) {
                const double xk = W.xs[lane];
                const double mk = __ldg(M + p2 * P + p1);
                dup = W.pm2[vp][h] >= xk && mk > 0 && mk * W.f2s[vp][h] >= xk * 2;
              }
              if (!dup) {
                a = true;
                pr = W.f1s[vp][h] * f2 * m;
                if (!same) pr = pr * 2;
              }
            }
          }
          const uint32_t A = __ballot_sync(FULLM, a);
          if (A) {
            E += __popc(A);
            // population pair sums (impute.py:535-543): pairs of one h step are distinct
            uint32_t g = 0, slot = 0;
            bool fresh = false;
            if (a) {
              const uint32_t lo = p1 < p2 ? p1 : p2, hi = p1 < p2 ? p2 : p1;
              g = hi * (hi + 1) / 2 + lo;
              slot = gslot[g];
              fresh = slot == 0xFFFFu;
            }
            const uint32_t Fm = __ballot_sync(FULLM, fresh);
            if (a) {
              if (fresh) {
                slot = ng + __popc(Fm & ((1u << lane) - 1u));
                gslot[g] = (uint16_t)slot;
                gsum[slot] = pr;
                gpair[slot] = (uint16_t)((p1 << 8) | p2);
              } else {
                gsum[slot] = gsum[slot] + pr;
              }
            }
            ng += __popc(Fm);
            // hap_total (impute.py:529-533) and the per-phase haplotype-pair sum, k ascending
            for (uint32_t mm = A; mm; mm &= mm - 1) {
              const int j = __ffs(mm) - 1;
              const double pj = __shfl_sync(FULLM, pr, j);
              total = have_total ? total + pj : pj;
              have_total = true;
              psum = have_p ? psum + pj : pj;
              have_p = true;
            }
            __syncwarp();
          }
        }
        if (have_p) {
          if (lane == (int)nrows) {
            my_sum = psum;
            my_vp = vp;
          }
          ++nrows;
        }
      }
      if (E == 0) punt = true;   // nothing survives MaxProb / 100000: Plan B
    }
    if (punt) {
      if (lane == 0) worklist[atomicAdd(worklist_n, 1u)] = (uint32_t)s;
      continue;
    }
    // ---- publish (include/grimb200.h, GRIMB_KIND_TYPED): record + header word, PMUG probabilities,
    // population-pair probabilities in rank order, their pair codes four per word.  The UMUG genotype and
    // the haplotypes of the PMUG rows follow from the subject's alleles and the phase ids.
    const uint32_t np = want_p ? (nrows < lim_r ? nrows : lim_r) : 0u;
    const uint32_t npg = ng < lim_p ? ng : lim_p;
    const uint32_t nwords = 1u + np + npg + ((npg + 3u) >> 2);
    unsigned long long wb = 0;
    if (lane == 0) wb = atomicAdd(O.word_counter, (unsigned long long)nwords);
    wb = __shfl_sync(FULLM, wb, 0);
    if (want_u && want_p) evals *= 2;   // the reference evaluates once per output kind
    evals_sum += evals;                 // warp-uniform
    const bool fits = (int64_t)(wb + nwords) <= R.word_capacity;
    // PMUG rows: one per phase with accepted pairs, by (sum desc, phase asc)
    uint32_t rank = 0;
    for (uint32_t j = 0; j < nrows; ++j) {
      const double sj = __shfl_sync(FULLM, my_sum, (int)j);
      if (sj > my_sum || (sj == my_sum && (int)j < lane)) ++rank;
    }
    const bool my_row = lane < (int)nrows && rank < np;
    uint64_t hdr = my_row ? ((uint64_t)W.ph[my_vp] << (16 + 12 * rank)) : 0ull;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) hdr |= __shfl_xor_sync(FULLM, hdr, d);
    if (fits) {
      if (lane == 0) R.words[wb] = hdr | (uint64_t)npg;
      if (my_row) R.words[wb + 1 + rank] = (uint64_t)__double_as_longlong(my_sum);
    }
    if (lane == 0)
      R.compact[s] = make_compact(GRIMB_ST_OK, GRIMB_KIND_TYPED | GRIMB_KIND_HAS_RESULTS | (np << 4), 0, (uint32_t)wb, total);
    __syncwarp();
    if (npg) {
      // population rows by (sum desc, first encounter asc); the same rows serve both output kinds.  Each
      // lane ranks up to 4 groups per sweep over the list (one shared-memory read per comparand); the
      // group-lookup table is free by now and takes the pair codes in rank order.
      uint16_t* codes = gslot;
      for (uint32_t t0 = lane; t0 < ng; t0 += 128) {
        double vt[4];
        uint32_t rk[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const uint32_t t = t0 + 32u * q;
          vt[q] = t < ng ? gsum[t] : 0.0;
          rk[q] = 0;
        }
        for (uint32_t u = 0; u < ng; ++u) {
          const double vu = gsum[u];
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (vu > vt[q] || (vu == vt[q] && u < t0 + 32u * q)) ++rk[q];
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const uint32_t t = t0 + 32u * q;
          if (t < ng && rk[q] < npg) {
            codes[rk[q]] = gpair[t];
            if (fits) R.words[wb + 1 + np + rk[q]] = (uint64_t)__double_as_longlong(vt[q]);
          }
        }
      }
      __syncwarp();
      if (fits)
        for (uint32_t w = lane; w < ((npg + 3u) >> 2); w += 32) {
          uint64_t v = 0;
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (4 * w + q < npg) v |= (uint64_t)codes[4 * w + q] << (16 * q);
          R.words[wb + 1 + np + npg + w] = v;
        }
    }
    __syncwarp();
  }
  if (lane == 0) {
    if (evals_sum) atomicAdd(O.evals_counter, evals_sum);
    if (n_probes) atomicAdd(O.probe_counters + 0, n_probes);
    if (n_hits) atomicAdd(O.probe_counters + 1, n_hits);
    if (n_vecs) atomicAdd(O.probe_counters + 2, n_vecs);
  }
}

constexpr int GRIMB_MAX_CHUNKS = 64;

// The counters of a chunk reach the host through mapped pinned memory, written by this one-warp kernel on the
// compute stream: a cudaMemcpyAsync there would queue behind the copy-out stream's large transfers on the
// device-to-host copy engine and stall the kernels that follow it.
// the records of the subjects on a hand-over list, gathered for one small copy-out
__global__ void k_gather_compact(const uint32_t* __restrict__ list, uint32_t n, const GrimbCompact* __restrict__ compact,
                                 GrimbCompact* __restrict__ out, uint32_t* __restrict__ out_idx) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t s = list[i];
  out[i] = compact[s];
  out_idx[i] = s;
}

__global__ void k_snapshot(const unsigned long long* __restrict__ cnt, unsigned long long* out, int n) {
  if ((int)threadIdx.x < n) out[threadIdx.x] = cnt[threadIdx.x];
  __threadfence_system();
}

// Device counters of one call (unsigned long long each).  The first eight are per launch group (one
// chunk of a host batch) and are cleared between chunks; the rest keep running across the chunks of one
// ABI call, so the rows / words / records of a chunk occupy one contiguous range of their arrays.
enum {
  CNT_WORK = 0,       // tickets of the general kernel's persistent CTAs
  CNT_WORKLIST = 1,   // (u32) subjects handed from a warp-per-subject kernel to the general kernel
  CNT_BUCKETS = 2,    // (4 x u32) cost buckets of the general kernel's work
  CNT_OVERFLOW = 4,   // (u32) side records claimed by subjects with more candidate phases than a hand-over record holds
  CNT_SLOT_TICKET = 5,   // tickets of the cooperative slot kernel
  CNT_WORK2 = 6,      // tickets of the second general-kernel launch when the heavy buckets run first
  CNT_CHUNK_END = 8,
  CNT_HAP = 8,
  CNT_POP = 9,
  CNT_WORDS = 10,
  CNT_GENERAL = 11,
  CNT_EVALS = 12,
  CNT_PROBES = 13,    // probes issued, probes answered, frequency vectors read (general and typed kernels)
  CNT_N = 16
};

struct GrimbEngine {
  const GrimbTables* tables;
  int device;
  int threads;
  int threads_fixed = 0;          // GRIMB_THREADS given: no switching
  int64_t wide_cta_below = 2048;  // general-kernel lists up to this length run MAXT threads per CTA (GRIMB_WIDE_CTA_BELOW)
  int split_heavy = 0;            // longer lists: cost buckets [0, split_heavy) run first, on wide CTAs (GRIMB_SPLIT_HEAVY; 0 off)
  int n_ctas;
  uint64_t arena_per_cta;
  char* arena = nullptr;
  double* ones = nullptr;
  GrimbConfig* d_cfg = nullptr;
  unsigned long long* d_counters = nullptr;  // [CNT_N]
  cudaStream_t stream = nullptr;
  cudaStream_t s_in = nullptr, s_out = nullptr;   // copy-in / copy-out streams of the pipelined host call
  cudaEvent_t ev_in[GRIMB_MAX_CHUNKS], ev_k[GRIMB_MAX_CHUNKS];
  unsigned long long* h_cnt = nullptr;            // pinned + mapped: counters after every chunk [GRIMB_MAX_CHUNKS + 1][CNT_N]
  unsigned long long* h_cnt_dev = nullptr;        // its device address
  int64_t host_chunk = 262144;                    // subjects per pipeline chunk (GRIMB_HOST_CHUNK)
  GrimbConfig cfg_host;                           // the configuration d_cfg holds (valid when cfg_sent)
  GrimbConfig cfg_dev;                            // ... as the kernels see it
  int cfg_sent = 0;
  unsigned long long* h_tail = nullptr;           // pinned: the counters as read by the device-pointer call
  cudaStream_t pending_stream = nullptr;          // grimb_impute_device_async: stream of the call in flight
  int pending = 0;
  cudaEvent_t ev_done = nullptr;                  // ... recorded behind its last operation
  int tail_queued = 0;                            // ... the tail kernels were queued with it
  int tail_expected = 0;                          // the previous call of this engine handed subjects on
  GrimbBatch pend_batch;                          // ... its batch / result views (for the tail, if one is needed)
  GrimbResults pend_res;
  int64_t launches = 0;
  // staging for the host-pointer form (grow-only)
  DevBuf in[6], outb[5], in_mask;
  DevBuf worklist;   // subjects the fast kernel hands to the general kernel
  DevBuf buckets;    // the general kernel's work, by cost bucket (heaviest first)
  DevBuf gather;              // records of handed-on subjects, gathered for the copy-out of the host form
  void* h_gather = nullptr;   // ... their pinned landing buffer
  size_t h_gather_cap = 0;
  DevBuf pre_top, pre_meta;   // Plan A side lists of the heaviest subjects (cooperative slot kernel)
  uint32_t pre_max = 0;       // subjects the buffers hold (GRIMB_GROUP_SUBJECTS; 0 disables the slot kernel)
  int pre_K = 0;
  int sm_count = 0;
  int fast_path = 1; // GRIMB_FAST=0 disables the warp-per-subject kernel (debugging / A-B runs)
  int fast_split = 1; // k_fast_probe + k_fast_score (default); GRIMB_FAST_SPLIT=0: the fused k_impute_fast
  int fast_probe = 2; // packed batches: k_fast_probe2 (default); GRIMB_FAST_PROBE=1: the one-level k_fast_probe
  int last_probe = -1; // last split fast-path launch: 2 k_fast_probe2, 1 k_fast_probe (packed), 0 k_fast_probe (general form)
  int timing = 1;     // CUDA events around the kernels in the device-pointer form (GRIMB_KERNEL_EVENTS=0: none)
  int timing_host = 0;   // ... in the chunked host-pointer form (GRIMB_HOST_EVENTS=1)
  DevBuf mid;         // hand-over records of the split fast path
  DevBuf overflow;    // side records (FastExtra) of subjects with more candidate phases than a hand-over record holds
  cudaEvent_t ev_score[2] = {nullptr, nullptr};
  int ev_score_valid = 0;
  cudaEvent_t ev_slots[2] = {nullptr, nullptr};
  int ev_slots_valid = 0;
  // CUDA events around the last launch of k_impute_fast [0,1], k_impute [2,3], k_impute_typed [4,5]
  cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  int ev_valid[3] = {0, 0, 0};
  double last_worklist = -1; // subjects the last call handed from a warp-per-subject kernel to k_impute
  int typed_ctas = 0;        // resident CTAs of k_impute_typed on this device (0: P > 32, kernel unused)
  uint32_t typed_per_warp = 0;
  // grimb_batch_from_genotypes (the batch it returns lives here) and grimb_results_rows; grow-only
  DevBuf geno_keys, geno_flags, geno_mask, geno_off, geno_alleles, geno_small, scan_tmp;
  unsigned long long* h_small = nullptr;   // pinned: the read-backs of both calls
  cudaEvent_t ev_geno[4] = {nullptr, nullptr, nullptr, nullptr};   // [0,1] k_geno_encode, [2,3] scan + k_geno_fill
  int ev_geno_valid = 0;                   // bit 0 / bit 1: pair recorded by the last call
  cudaEvent_t ev_rows[4] = {nullptr, nullptr, nullptr, nullptr};   // [0,1] count + scans, [2,3] k_rows_fill
  int ev_rows_valid = 0;
  // grimb_batch_from_genotype_lists (the batch it returns lives here); grow-only
  DevBuf gl_in_off, gl_stage, gl_mask, gl_counts, gl_off, gl_alleles;
  cudaEvent_t ev_gl[4] = {nullptr, nullptr, nullptr, nullptr};     // [0,1] k_gl_count + scan, [2,3] dedup, scan, fill
  int ev_gl_valid = 0;
};

extern "C" int grimb_engine_free(GrimbEngine* e);

// A probe wants ONE 32-byte sector, but the memory side works in 64-byte units: ncu of k_fast_probe shows 32.1 M
// read requests from the SMs looked up as 70.5 M sectors at the L2 (+ 30.7 M again on the far die's slices for the
// half homed there: the "2.9x algorithmic" lts__t_sectors of the round-1 review) and DRAM reading 64 B per missing
// request.  cudaLimitMaxL2FetchGranularity = 32 is the documented knob; on B200 it changed nothing
// (0.2507 ms with 32, 0.2508 ms with 64), so it is only applied on request (GRIMB_L2_FETCH=32|64|128).
static void set_l2_fetch_granularity() {
  const char* v = getenv("GRIMB_L2_FETCH");
  if (!v) return;
  const long x = atol(v);
  if (x != 32 && x != 64 && x != 128) return;
  if (cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)x) != cudaSuccess) cudaGetLastError();
}

extern "C" int grimb_engine_create(const GrimbTables* t, int64_t workspace_bytes_per_cta, GrimbEngine** out) {
  if (!t || !out || workspace_bytes_per_cta < (1 << 16)) return fail(GRIMB_E_ARG, "bad engine arguments");
  CK(cudaSetDevice(t->device));
  set_l2_fetch_granularity();
  GrimbEngine* e = new GrimbEngine();
  for (int i = 0; i < GRIMB_MAX_CHUNKS; ++i) e->ev_in[i] = e->ev_k[i] = nullptr;
  e->tables = t;
  e->device = t->device;
  e->threads = 128;
  // every failure below releases what was created so far
#define CKE(call)                                                                          \
  do {                                                                                     \
    cudaError_t e_ = (call);                                                               \
    if (e_ != cudaSuccess) {                                                               \
      grimb_engine_free(e);                                                                \
      return fail(GRIMB_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));       \
    }                                                                                      \
  } while (0)
  cudaDeviceProp prop;
  CKE(cudaGetDeviceProperties(&prop, t->device));
  int per_sm = 0;
  CKE(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_impute, e->threads, 0));
  if (per_sm < 1) per_sm = 1;
  size_t free_b = 0, total_b = 0;
  CKE(cudaMemGetInfo(&free_b, &total_b));
  int64_t n = (int64_t)prop.multiProcessorCount * per_sm;
  e->arena_per_cta = ((uint64_t)workspace_bytes_per_cta + 255ull) & ~255ull;
  while (n > prop.multiProcessorCount && (uint64_t)n * e->arena_per_cta > free_b / 2) n -= prop.multiProcessorCount;
  while (n > 1 && (uint64_t)n * e->arena_per_cta > free_b / 2) n /= 2;
  e->n_ctas = (int)n;
  cudaError_t ce = cudaMalloc((void**)&e->arena, (uint64_t)e->n_ctas * e->arena_per_cta);
  if (ce != cudaSuccess) {
    grimb_engine_free(e);
    return fail(GRIMB_E_NOMEM, std::string("engine arena: ") + cudaGetErrorString(ce));
  }
  const int P = t->h.P;
  std::vector<double> one((size_t)P * P, 1.0);
  CKE(cudaMalloc((void**)&e->ones, one.size() * 8));
  CKE(cudaMemcpy(e->ones, one.data(), one.size() * 8, cudaMemcpyHostToDevice));
  CKE(cudaMalloc((void**)&e->d_cfg, sizeof(GrimbConfig)));
  CKE(cudaMalloc((void**)&e->d_counters, CNT_N * sizeof(unsigned long long)));
  CKE(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
  CKE(cudaStreamCreateWithFlags(&e->s_in, cudaStreamNonBlocking));
  CKE(cudaStreamCreateWithFlags(&e->s_out, cudaStreamNonBlocking));
  for (int i = 0; i < GRIMB_MAX_CHUNKS; ++i) {
    CKE(cudaEventCreateWithFlags(&e->ev_in[i], cudaEventDisableTiming));
    CKE(cudaEventCreateWithFlags(&e->ev_k[i], cudaEventDisableTiming));
  }
  CKE(cudaHostAlloc((void**)&e->h_cnt, (GRIMB_MAX_CHUNKS + 1) * CNT_N * sizeof(unsigned long long), cudaHostAllocMapped));
  CKE(cudaHostGetDevicePointer((void**)&e->h_cnt_dev, e->h_cnt, 0));
  CKE(cudaMallocHost((void**)&e->h_tail, CNT_N * sizeof(unsigned long long)));
  if (const char* hc = getenv("GRIMB_HOST_CHUNK")) {
    const long long v = atoll(hc);
    if (v >= 1024) e->host_chunk = v;
  }
  for (int i = 0; i < 6; ++i) CKE(cudaEventCreate(&e->ev[i]));
  e->sm_count = prop.multiProcessorCount;
  if (P <= 32) {
    e->typed_per_warp = (uint32_t)ty_bytes_per_warp(P);
    const size_t dyn = (size_t)e->typed_per_warp * TY_WARPS;
    // the attribute is per function, not per engine: always allow the largest layout (P = 32)
    CKE(cudaFuncSetAttribute(k_impute_typed, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)(ty_bytes_per_warp(32) * TY_WARPS)));
    int tb = 0;
    CKE(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&tb, k_impute_typed, TY_WARPS * 32, dyn));
    e->typed_ctas = (tb < 1 ? 1 : tb) * prop.multiProcessorCount;
  }
  const char* fp = getenv("GRIMB_FAST");
  if (fp && fp[0] == '0') e->fast_path = 0;
  const char* fsp = getenv("GRIMB_FAST_SPLIT");
  if (fsp && fsp[0] == '0') e->fast_split = 0;
  const char* fpr = getenv("GRIMB_FAST_PROBE");
  if (fpr && fpr[0] == '1') e->fast_probe = 1;
  const char* kev = getenv("GRIMB_KERNEL_EVENTS");
  if (kev && kev[0] == '0') e->timing = 0;
  const char* hev = getenv("GRIMB_HOST_EVENTS");
  if (hev && hev[0] == '1') e->timing_host = 1;
  for (int i = 0; i < 2; ++i) CKE(cudaEventCreate(&e->ev_score[i]));
  for (int i = 0; i < 2; ++i) CKE(cudaEventCreate(&e->ev_slots[i]));
  CKE(cudaEventCreateWithFlags(&e->ev_done, cudaEventDisableTiming));
  for (int i = 0; i < 4; ++i) CKE(cudaEventCreate(&e->ev_geno[i]));
  for (int i = 0; i < 4; ++i) CKE(cudaEventCreate(&e->ev_rows[i]));
  for (int i = 0; i < 4; ++i) CKE(cudaEventCreate(&e->ev_gl[i]));
  CKE(cudaMallocHost((void**)&e->h_small, 8 * sizeof(unsigned long long)));
  e->pre_max = 4096;
  if (const char* gs = getenv("GRIMB_GROUP_SUBJECTS")) {
    const long long v = atoll(gs);
    if (v >= 0 && v <= (1 << 20)) e->pre_max = (uint32_t)v;
  }
  const char* th = getenv("GRIMB_THREADS");
  if (th) {
    int v = atoi(th);
    if (v >= 32 && v <= MAXT && v % 32 == 0) {
      e->threads = v;
      e->threads_fixed = 1;
    }
  }
  if (const char* wc = getenv("GRIMB_WIDE_CTA_BELOW")) e->wide_cta_below = atoll(wc);
  if (const char* sh = getenv("GRIMB_SPLIT_HEAVY")) {
    const int v = atoi(sh);
    if (v >= 0 && v < GRIMB_BUCKETS) e->split_heavy = v;
  }
#undef CKE
  *out = e;
  return GRIMB_OK;
}

extern "C" int grimb_engine_free(GrimbEngine* e) {
  if (!e) return GRIMB_OK;
  cudaSetDevice(e->device);
  if (e->stream) cudaStreamSynchronize(e->stream);
  cudaFree(e->arena);
  cudaFree(e->ones);
  cudaFree(e->d_cfg);
  cudaFree(e->d_counters);
  if (e->stream) cudaStreamDestroy(e->stream);
  if (e->s_in) cudaStreamDestroy(e->s_in);
  if (e->s_out) cudaStreamDestroy(e->s_out);
  for (int i = 0; i < GRIMB_MAX_CHUNKS; ++i) {
    if (e->ev_in[i]) cudaEventDestroy(e->ev_in[i]);
    if (e->ev_k[i]) cudaEventDestroy(e->ev_k[i]);
  }
  for (int i = 0; i < 6; ++i)
    if (e->ev[i]) cudaEventDestroy(e->ev[i]);
  for (int i = 0; i < 2; ++i)
    if (e->ev_score[i]) cudaEventDestroy(e->ev_score[i]);
  for (int i = 0; i < 2; ++i)
    if (e->ev_slots[i]) cudaEventDestroy(e->ev_slots[i]);
  if (e->ev_done) cudaEventDestroy(e->ev_done);
  for (int i = 0; i < 4; ++i) {
    if (e->ev_geno[i]) cudaEventDestroy(e->ev_geno[i]);
    if (e->ev_rows[i]) cudaEventDestroy(e->ev_rows[i]);
    if (e->ev_gl[i]) cudaEventDestroy(e->ev_gl[i]);
  }
  if (e->h_small) cudaFreeHost(e->h_small);
  if (e->h_gather) cudaFreeHost(e->h_gather);
  if (e->h_cnt) cudaFreeHost(e->h_cnt);
  if (e->h_tail) cudaFreeHost(e->h_tail);
  cudaGetLastError();
  delete e;
  return GRIMB_OK;
}

extern "C" int64_t grimb_engine_launches(const GrimbEngine* e) { return e ? e->launches : 0; }

// Device time (CUDA events on the launching stream) of the last launch of k_fast_probe / k_impute_fast
// (which = 0), k_impute (1), k_impute_typed (2), k_fast_score (4); valid after the call that launched it
// has finished.  < 0 if not launched.  which = 3: subjects the last call handed on to k_impute.
extern "C" double grimb_engine_kernel_ms(const GrimbEngine* e, int which) {
  if (e && which == 3) return e->last_worklist;
  if (e && which == 6) return (double)e->last_probe;
  if (e && which >= 7 && which <= 9) {   // sum of the event pairs the last grimb_batch_from_genotypes / _results_rows /
                                          // grimb_batch_from_genotype_lists recorded
    const cudaEvent_t* ev = which == 7 ? e->ev_geno : which == 8 ? e->ev_rows : e->ev_gl;
    const int valid = which == 7 ? e->ev_geno_valid : which == 8 ? e->ev_rows_valid : e->ev_gl_valid;
    if (!valid) return -1.0;
    double sum = 0.0;
    for (int k = 0; k < 2; ++k) {
      float ms = 0.f;
      if (!(valid & (1 << k))) continue;
      if (cudaEventElapsedTime(&ms, ev[2 * k], ev[2 * k + 1]) != cudaSuccess) {
        cudaGetLastError();
        return -1.0;
      }
      sum += ms;
    }
    return sum;
  }
  if (e && which == 5) {   // k_impute_slots
    float ms5 = -1.f;
    if (!e->ev_slots_valid || cudaEventElapsedTime(&ms5, e->ev_slots[0], e->ev_slots[1]) != cudaSuccess) {
      cudaGetLastError();
      return -1.0;
    }
    return (double)ms5;
  }
  if (e && which == 4) {
    float ms4 = -1.f;
    if (!e->ev_score_valid || cudaEventElapsedTime(&ms4, e->ev_score[0], e->ev_score[1]) != cudaSuccess) {
      cudaGetLastError();
      return -1.0;
    }
    return (double)ms4;
  }
  if (!e || which < 0 || which > 2 || !e->ev_valid[which]) return -1.0;
  float ms = -1.f;
  if (cudaEventElapsedTime(&ms, e->ev[2 * which], e->ev[2 * which + 1]) != cudaSuccess) {
    cudaGetLastError();
    return -1.0;
  }
  return (double)ms;
}

static int check_cfg(const GrimbConfig* c, const GrimbTables* t) {
  if (!(c->epsilon > 0)) return fail(GRIMB_E_ARG, "epsilon must be > 0");
  if (c->max_haps_in_phase < 1 || c->max_haps_in_phase > 512) return fail(GRIMB_E_ARG, "max_haps_in_phase must be 1..512");
  if (c->n_results < 0 || c->n_pop_results < 0) return fail(GRIMB_E_ARG, "negative result limits");
  if (c->options_threshold < 1 || c->options_threshold > (1ll << 31)) return fail(GRIMB_E_ARG, "options_threshold out of range");
  if (c->n_rows < 0 || c->n_rows > GRIMB_MAX_ROWS) return fail(GRIMB_E_ARG, "too many Plan_B_Matrix rows");
  for (int r = 0; r < c->n_rows; ++r)
    if (c->row_blocks[r] < 0 || c->row_blocks[r] > GRIMB_MAX_BLOCKS) return fail(GRIMB_E_ARG, "too many blocks in a row");
  (void)t;
  return GRIMB_OK;
}

// The configuration lives in device memory for the kernels; it is uploaded only when it differs from
// the copy the engine last sent (a pageable-memory copy per call otherwise costs more than a launch).
static int upload_cfg(GrimbEngine* e, const GrimbConfig* cfg, cudaStream_t st) {
  if (e->cfg_sent && memcmp(&e->cfg_host, cfg, sizeof(GrimbConfig)) == 0) return GRIMB_OK;
  e->cfg_sent = 0;
  CK(cudaStreamSynchronize(e->stream));   // an earlier call on the engine stream may still read d_cfg
  e->cfg_host = *cfg;
  e->cfg_dev = *cfg;
  if (cfg->plan_a_only) e->cfg_dev.planb = 0;   // a restricted store serves Plan A only (include/grimb200.h)
  CK(cudaMemcpyAsync(e->d_cfg, &e->cfg_dev, sizeof(GrimbConfig), cudaMemcpyHostToDevice, st));
  CK(cudaStreamSynchronize(st));
  e->cfg_sent = 1;
  return GRIMB_OK;
}

static OutArrays out_arrays(GrimbEngine* e, const GrimbResults& r) {
  OutArrays O;
  O.r = r;
  O.hap_counter = e->d_counters + CNT_HAP;
  O.pop_counter = e->d_counters + CNT_POP;
  O.word_counter = e->d_counters + CNT_WORDS;
  O.general_counter = e->d_counters + CNT_GENERAL;
  O.evals_counter = e->d_counters + CNT_EVALS;
  O.probe_counters = e->d_counters + CNT_PROBES;
  return O;
}

// The kernels of one call come in two parts.  launch_warp: the warp-per-subject kernels over the subjects
// [s_begin, s_end) of the batch (device pointers) -- what they cannot finish is appended to the engine's
// hand-over lists, which keep growing across the ranges of one call.  launch_tail, once per call after the
// last range: the fused kernel over the overflow list, the cost classification, the cooperative slot pass
// and the general kernel over everything that was handed on (or over the whole batch when no
// warp-per-subject kernel serves this table / mode).  No synchronisation in either.
static bool warp_kernels_apply(const GrimbEngine* e, const GrimbConfig* cfg, const GrimbBatch* batch) {
  // the warp-per-subject kernels implement the default phase enumeration and row layout only
  if (!(e->fast_path && (!batch->phase_mask || batch->packed_keys) && !cfg->hap_pop_pair && !cfg->encounter_order)) return false;
  const TablesView& tv = e->tables->view;
#if GRIMB_KW == 1
  if (tv.L <= 5 && tv.P == 1) return true;
#endif
  return e->typed_ctas > 0;
}

static int launch_warp(GrimbEngine* e, const GrimbConfig* cfg, const GrimbBatch* batch, const OutArrays& O, cudaStream_t st,
                       bool tm, int64_t s_begin, int64_t s_end) {
  const int64_t n = s_end - s_begin;
  if (n <= 0 || !warp_kernels_apply(e, cfg, batch)) return GRIMB_OK;
  const TablesView& tv = e->tables->view;
  GrimbBatch rb = *batch;
  rb.n_subjects = s_end;   // the kernels walk [s_begin, n_subjects)
  CK(e->worklist.reserve((size_t)batch->n_subjects * 4 + 16));
  unsigned int* cnt = (unsigned int*)(e->d_counters + CNT_WORKLIST);
#if GRIMB_KW == 1
  if (tv.L <= 5 && tv.P == 1) {
    const uint64_t groups = ((uint64_t)n + FAST_WARPS * 2 - 1) / (FAST_WARPS * 2);
    if (e->fast_split) {
      const FastIndex& fidx = e->tables->fidx;
      if (!fidx.keys) return fail(GRIMB_E_ARG, "table has no fast-path index");
      CK(e->mid.reserve((size_t)batch->n_subjects * (sizeof(FastHead) + sizeof(FastMore)) + 256));
      FastMid midv;
      midv.head = (FastHead*)e->mid.p;
      midv.more = (FastMore*)((char*)e->mid.p + (((size_t)batch->n_subjects * sizeof(FastHead) + 127) & ~(size_t)127));
      double eps = cfg->epsilon;
      int nr = 0;
      while (eps > 0 && nr < FAST_MAX_ROUNDS) {
        eps /= 10;
        if (eps < 1.0e-9) eps = 0.0;
        ++nr;
      }
      uint64_t fgp = (uint64_t)e->sm_count * FASTPROBE_MIN_BLOCKS;
      if (fgp > groups) fgp = groups;
      const uint32_t extra_cap = (uint32_t)(batch->n_subjects / 16 + 1024);   // side records for subjects with > 4 candidate phases
      CK(e->overflow.reserve((size_t)extra_cap * sizeof(FastExtra) + 64));
      unsigned int* ovf_n = (unsigned int*)(e->d_counters + CNT_OVERFLOW);
      if (tm) CK(cudaEventRecord(e->ev[0], st));
      if (batch->packed_keys && e->fast_probe == 2) {
        uint64_t g2 = (uint64_t)e->sm_count * FASTPROBE2_MIN_BLOCKS;
        const uint64_t quads = ((uint64_t)n + FAST_WARPS * 4 - 1) / (FAST_WARPS * 4);
        if (g2 > quads) g2 = quads;
        k_fast_probe2<<<(unsigned)g2, FAST_WARPS * 32, 0, st>>>(tv, fidx, rb, O, midv, (uint32_t*)e->worklist.p, cnt,
                                                             (FastExtra*)e->overflow.p, ovf_n, extra_cap, eps > 0 ? 0 : 1,
                                                             (uint32_t)s_begin);
        e->last_probe = 2;
      } else if (batch->packed_keys) {
        k_fast_probe<true><<<(unsigned)fgp, FAST_WARPS * 32, 0, st>>>(tv, fidx, rb, O, midv, (uint32_t*)e->worklist.p, cnt,
                                                                    (FastExtra*)e->overflow.p, ovf_n, extra_cap, eps > 0 ? 0 : 1, (uint32_t)s_begin);
        e->last_probe = 1;
      } else {
        k_fast_probe<false><<<(unsigned)fgp, FAST_WARPS * 32, 0, st>>>(tv, fidx, rb, O, midv, (uint32_t*)e->worklist.p, cnt,
                                                                     (FastExtra*)e->overflow.p, ovf_n, extra_cap, eps > 0 ? 0 : 1, (uint32_t)s_begin);
        e->last_probe = 0;
      }
      CK(cudaGetLastError());
      if (tm) CK(cudaEventRecord(e->ev[1], st));
      uint64_t sg = ((uint64_t)n + 127) / 128;
      if (sg > (uint64_t)e->sm_count * 16) sg = (uint64_t)e->sm_count * 16;
      if (tm) CK(cudaEventRecord(e->ev_score[0], st));
      k_fast_score<<<(unsigned)sg, 128, 0, st>>>(tv, fidx, e->d_cfg, rb, O, midv, (const FastExtra*)e->overflow.p,
                                                (uint32_t*)e->worklist.p, cnt, (uint32_t)s_begin);
      CK(cudaGetLastError());
      if (tm) CK(cudaEventRecord(e->ev_score[1], st));
      e->ev_score_valid = tm;
      e->ev_valid[0] = tm;
      e->launches += 2;
    } else {
      uint64_t fg = (uint64_t)e->sm_count * FAST_MIN_BLOCKS;  // resident CTAs only: each warp strides over subjects
      if (fg > groups) fg = groups;
      if (tm) CK(cudaEventRecord(e->ev[0], st));
      k_impute_fast<false><<<(unsigned)fg, FAST_WARPS * 32, 0, st>>>(tv, e->d_cfg, rb, O, (uint32_t*)e->worklist.p, cnt, nullptr,
                                                                    nullptr, (uint32_t)s_begin);
      CK(cudaGetLastError());
      if (tm) CK(cudaEventRecord(e->ev[1], st));
      e->ev_valid[0] = tm;
      e->launches += 1;
    }
    return GRIMB_OK;
  }
#endif
  // warp-per-subject kernel for fully typed unambiguous subjects, any P <= 32 / L / key width
  uint64_t tg = ((uint64_t)n + TY_WARPS - 1) / TY_WARPS;
  if (tg > (uint64_t)e->typed_ctas) tg = (uint64_t)e->typed_ctas;
  if (tm) CK(cudaEventRecord(e->ev[4], st));
  k_impute_typed<<<(unsigned)tg, TY_WARPS * 32, (size_t)e->typed_per_warp * TY_WARPS, st>>>(
      tv, e->d_cfg, rb, O, (uint32_t*)e->worklist.p, cnt, e->typed_per_warp, (uint32_t)s_begin);
  CK(cudaGetLastError());
  if (tm) CK(cudaEventRecord(e->ev[5], st));
  e->ev_valid[2] = tm;
  e->launches += 1;
  return GRIMB_OK;
}

// n_tail: subjects the general kernel will serve when the caller knows (the whole batch without warp kernels, the
// length of the hand-over list once it has been read back), -1 otherwise.
static int launch_tail(GrimbEngine* e, const GrimbConfig* cfg, const GrimbBatch* batch, const OutArrays& O, cudaStream_t st,
                       bool tm, int64_t n_tail = -1) {
  if (batch->n_subjects <= 0) return GRIMB_OK;
  const TablesView& tv = e->tables->view;
  const bool warp = warp_kernels_apply(e, cfg, batch);
  const uint32_t* wl = warp ? (const uint32_t*)e->worklist.p : nullptr;
  unsigned int* cnt = (unsigned int*)(e->d_counters + CNT_WORKLIST);
  const unsigned int* wl_n = warp ? cnt : nullptr;
  const uint64_t stride = (uint64_t)batch->n_subjects;
  CK(e->buckets.reserve((size_t)stride * 4 * GRIMB_BUCKETS + 16));
  unsigned int* bucket_n = (unsigned int*)(e->d_counters + CNT_BUCKETS);
  {
    uint64_t cg = (stride + 255) / 256;
    if (cg > (uint64_t)e->sm_count * 4) cg = (uint64_t)e->sm_count * 4;
    if (wl) cg = cg < 64 ? cg : 64;   // a hand-over list is short (or empty)
    k_classify<<<(unsigned)cg, 256, 0, st>>>(*batch, tv.L, wl, wl_n, (uint32_t*)e->buckets.p, bucket_n, stride);
    CK(cudaGetLastError());
    e->launches += 1;
  }
  int grid = e->n_ctas;
  if ((int64_t)grid > batch->n_subjects) grid = (int)batch->n_subjects;
  // A small batch is bound by its slowest subjects, each alone on one CTA at a few per cent of the SM's issue
  // rate: twice the threads per CTA halve that subject's time (53 -> 26 ms for the slowest of the C4 messy
  // set) at the price of half the resident CTAs, which a short list does not fill anyway (cross-over measured
  // near 3,000 subjects: 250 / 1,000 / 2,000 / 4,000 messy subjects take 45 / 59 / 95 / 179 ms at 256 threads,
  // 53 / 66 / 112 / 162 ms at 128).
  int threads = e->threads;
  if (!e->threads_fixed && n_tail >= 0 && n_tail <= e->wide_cta_below && e->n_ctas >= 4) {
    // 256 threads, or 512 for a very short list (an eighth of the threshold: 256 subjects)
    threads = n_tail <= e->wide_cta_below / 8 ? 512 : 256;
    const int div = threads / 128;
    if (grid > e->n_ctas / div) grid = e->n_ctas / div;
  }
  // cooperative slot kernel for the heaviest subjects (bucket 0), then the general kernel
  PreView pv;
  memset(&pv, 0, sizeof(pv));
  if (e->pre_max > 0 && (!batch->phase_mask || batch->packed_keys)) {
    const uint32_t spp = 1u << tv.L;
    const uint32_t K = (uint32_t)cfg->max_haps_in_phase;
    uint64_t fit = e->pre_max;
    const uint64_t budget = 1ull << 31;   // bytes of top lists
    const uint64_t per_subject = (uint64_t)spp * K * sizeof(TopItem);
    if (fit * per_subject > budget) fit = budget / per_subject;
    if ((int64_t)fit > batch->n_subjects) fit = (uint64_t)batch->n_subjects;
    if (fit > 0) {
      CK(e->pre_top.reserve(fit * per_subject + 16));
      CK(e->pre_meta.reserve(fit * spp * 12 + 16));
      pv.top = (TopItem*)e->pre_top.p;
      pv.n = (uint32_t*)e->pre_meta.p;
      pv.ne = pv.n + fit * spp;
      pv.ready = pv.ne + fit * spp;
      pv.max_subjects = (uint32_t)fit;
      pv.slots_per_subject = spp;
      pv.K = K;
      if (tm) CK(cudaEventRecord(e->ev_slots[0], st));
      k_impute<<<grid, threads, 0, st>>>(tv, e->d_cfg, *batch, O, e->arena, e->arena_per_cta, e->ones,
                                        e->d_counters + CNT_SLOT_TICKET, (const uint32_t*)e->buckets.p, bucket_n, stride, pv, 1);
      CK(cudaGetLastError());
      if (tm) CK(cudaEventRecord(e->ev_slots[1], st));
      e->ev_slots_valid = tm;
      e->launches += 1;
    }
  }
  if (tm) CK(cudaEventRecord(e->ev[2], st));
  if (e->split_heavy > 0 && threads == e->threads && !e->threads_fixed && e->n_ctas >= 2) {
    // a long list: its heavy buckets first, alone on the GPU and on wide CTAs, then the rest
    const int hb = e->split_heavy;
    int gh = e->n_ctas / 2;
    if ((int64_t)gh > batch->n_subjects) gh = (int)batch->n_subjects;
    k_impute<<<gh, 256, 0, st>>>(tv, e->d_cfg, *batch, O, e->arena, e->arena_per_cta, e->ones, e->d_counters + CNT_WORK,
                                (const uint32_t*)e->buckets.p, bucket_n, stride, pv, 2 + 16 * hb);
    CK(cudaGetLastError());
    k_impute<<<grid, threads, 0, st>>>(tv, e->d_cfg, *batch, O, e->arena, e->arena_per_cta, e->ones, e->d_counters + CNT_WORK2,
                                      (const uint32_t*)e->buckets.p, bucket_n, stride, pv, 3 + 16 * hb);
    e->launches += 1;
  } else {
    k_impute<<<grid, threads, 0, st>>>(tv, e->d_cfg, *batch, O, e->arena, e->arena_per_cta, e->ones, e->d_counters + CNT_WORK,
                                      (const uint32_t*)e->buckets.p, bucket_n, stride, pv, 0);
  }
  CK(cudaGetLastError());
  if (tm) CK(cudaEventRecord(e->ev[3], st));
  e->ev_valid[1] = tm;
  e->launches += 1;
  return GRIMB_OK;
}

static void reset_event_flags(GrimbEngine* e) {
  e->ev_valid[0] = e->ev_valid[1] = e->ev_valid[2] = 0;
  e->ev_score_valid = 0;
  e->ev_slots_valid = 0;
}

static int check_batch(const GrimbBatch* b, const GrimbTables* t) {
  if (b->n_subjects < 0 || b->n_subjects > 0x7FFFFFF0ll) return fail(GRIMB_E_ARG, "bad n_subjects");
  if (b->n_subjects == 0) return GRIMB_OK;
  if (b->packed_keys) {
    if (GRIMB_KW != 1 || t->h.L > 5) return fail(GRIMB_E_ARG, "packed batches need the 64-bit-key build and L <= 5");
    if (!b->packed_flags || !b->priors) return fail(GRIMB_E_ARG, "packed batch: packed_flags / priors missing");
    return GRIMB_OK;
  }
  if (!b->typed_mask || !b->allele_off || !b->alleles || !b->priors) return fail(GRIMB_E_ARG, "batch arrays missing");
  return GRIMB_OK;
}

static int check_results(const GrimbResults* r) {
  if (!r->compact || !r->totals) return fail(GRIMB_E_ARG, "GrimbResults.compact / totals missing");
  if (r->word_capacity < 0 || r->general_capacity < 0 || r->hap_capacity < 0 || r->pop_capacity < 0)
    return fail(GRIMB_E_ARG, "negative result capacity");
  return GRIMB_OK;
}

static int totals_from(const unsigned long long* c, double handed, const GrimbResults* r) {
  int64_t* t = r->totals;
  t[0] = (int64_t)c[CNT_WORDS];
  t[1] = (int64_t)c[CNT_GENERAL];
  t[2] = (int64_t)c[CNT_HAP];
  t[3] = (int64_t)c[CNT_POP];
  t[4] = (int64_t)c[CNT_EVALS];
  t[5] = (int64_t)handed;
  t[6] = (int64_t)c[CNT_PROBES];
  t[7] = (int64_t)c[CNT_PROBES + 1];
  t[8] = (int64_t)c[CNT_PROBES + 2];
  if (t[0] > r->word_capacity || t[1] > r->general_capacity || t[2] > r->hap_capacity || t[3] > r->pop_capacity)
    return fail(GRIMB_E_CAPACITY, "result buffers too small (see GrimbResults.totals)");
  return GRIMB_OK;
}

// Asynchronous device-pointer form.  The call enqueues the warp-per-subject kernels (and a copy of the
// counters into pinned memory) and returns; grimb_impute_finish waits for THIS call (an event, not the
// stream: other engines' calls queued behind it on the same stream keep running), and only if something was
// handed on -- or no warp-per-subject kernel serves the table / mode -- launches the tail (overflow list,
// classification, cooperative slot pass, general kernel) and waits for it.  The usual batch of BASELINE
// config 2 therefore costs two kernels.  One call may be in flight per engine; a caller that wants batch
// k+1 queued while batch k runs alternates between two engines.
extern "C" int grimb_impute_device_async(GrimbEngine* e, const GrimbConfig* cfg, const GrimbBatch* batch,
                                         const GrimbResults* res, void* cuda_stream) {
  if (!e || !cfg || !batch || !res) return fail(GRIMB_E_ARG, "null argument");
  if (e->pending) return fail(GRIMB_E_ARG, "a call is in flight on this engine: grimb_impute_finish first");
  int rc = check_cfg(cfg, e->tables);
  if (rc) return rc;
  rc = check_results(res);
  if (rc) return rc;
  rc = check_batch(batch, e->tables);
  if (rc) return rc;
  CK(cudaSetDevice(e->device));
  cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : e->stream;
  rc = upload_cfg(e, cfg, st);
  if (rc) return rc;
  CK(cudaMemsetAsync(e->d_counters, 0, CNT_N * sizeof(unsigned long long), st));
  reset_event_flags(e);
  const OutArrays O = out_arrays(e, *res);
  rc = launch_warp(e, cfg, batch, O, st, e->timing != 0, 0, batch->n_subjects);
  if (rc) return rc;
  // the tail is queued right away when the previous call of this engine needed one (a steady stream of
  // batches with a few handed-on subjects each then never waits twice); otherwise it is left to finish
  e->tail_queued = e->tail_expected || !warp_kernels_apply(e, cfg, batch);
  if (e->tail_queued) {
    rc = launch_tail(e, cfg, batch, O, st, e->timing != 0, warp_kernels_apply(e, cfg, batch) ? -1 : batch->n_subjects);
    if (rc) return rc;
  }
  CK(cudaMemcpyAsync(e->h_tail, e->d_counters, CNT_N * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
  CK(cudaEventRecord(e->ev_done, st));
  e->pending_stream = st;
  e->pend_batch = *batch;
  e->pend_res = *res;
  e->pending = 1;
  return GRIMB_OK;
}

extern "C" int grimb_impute_finish(GrimbEngine* e, const GrimbResults* res) {
  if (!e || !res || !res->totals) return fail(GRIMB_E_ARG, "null argument");
  if (!e->pending) return fail(GRIMB_E_ARG, "no call in flight");
  CK(cudaSetDevice(e->device));
  e->pending = 0;
  CK(cudaEventSynchronize(e->ev_done));
  const bool warp = warp_kernels_apply(e, &e->cfg_host, &e->pend_batch);
  const unsigned long long handed = e->h_tail[CNT_WORKLIST] & 0xFFFFFFFFull;
  e->tail_expected = handed > 0;
  if (!e->tail_queued && (!warp || handed > 0)) {
    cudaStream_t st = e->pending_stream;
    int rc = launch_tail(e, &e->cfg_host, &e->pend_batch, out_arrays(e, e->pend_res), st, e->timing != 0,
                         warp ? (int64_t)handed : e->pend_batch.n_subjects);
    if (rc) return rc;
    CK(cudaMemcpyAsync(e->h_tail, e->d_counters, CNT_N * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CK(cudaEventRecord(e->ev_done, st));
    CK(cudaEventSynchronize(e->ev_done));
  }
  e->last_worklist = (double)(unsigned int)(e->h_tail[CNT_WORKLIST] & 0xFFFFFFFFull);
  return totals_from(e->h_tail, e->last_worklist, res);
}

extern "C" int grimb_impute_device(GrimbEngine* e, const GrimbConfig* cfg, const GrimbBatch* batch, GrimbResults* res,
                                   void* cuda_stream) {
  int rc = grimb_impute_device_async(e, cfg, batch, res, cuda_stream);
  if (rc) return rc;
  return grimb_impute_finish(e, res);
}

// Host-pointer form.  Large batches are pipelined in chunks over three streams: while chunk c is
// imputed, chunk c+1 is copied in and the results of chunk c-1 are copied out (PCIe is full duplex),
// so the call costs about max(H2D, kernels, D2H) instead of their sum.  What one chunk appends to each
// result array is one contiguous range (launches of one stream serialise and the counters keep
// running), so each chunk's D2H is a handful of plain copies once its counters are known.
extern "C" int grimb_impute_host(GrimbEngine* e, const GrimbConfig* cfg, const GrimbBatch* b, GrimbResults* r) {
  if (!e || !cfg || !b || !r) return fail(GRIMB_E_ARG, "null argument");
  int rc = check_cfg(cfg, e->tables);
  if (rc) return rc;
  rc = check_results(r);
  if (rc) return rc;
  rc = check_batch(b, e->tables);
  if (rc) return rc;
  using hclk = std::chrono::steady_clock;
  const auto h0 = hclk::now();
  double hmark[6] = {0, 0, 0, 0, 0, 0};
  auto mark = [&](int k) { hmark[k] = std::chrono::duration<double, std::milli>(hclk::now() - h0).count(); };
  CK(cudaSetDevice(e->device));
  const int L = e->tables->h.L, P = e->tables->h.P;
  const int64_t S = b->n_subjects;
  cudaStream_t st = e->stream;
  const bool packed = b->packed_keys != nullptr;   // in[0]: flags, in[3]: keys
  const size_t in_bytes[6] = {(size_t)S * 2, (b->counts && !packed) ? (size_t)S * L * 2 * 2 : 0, packed ? 0 : (size_t)(S + 1) * 4,
                              packed ? (size_t)S * 16 : (size_t)b->n_alleles_total * 2, b->prior_index ? (size_t)S * 4 : 0,
                              (size_t)b->n_priors * P * P * 8};
  for (int i = 0; i < 6; ++i) CK(e->in[i].reserve(in_bytes[i] + 64));
  if (b->phase_mask && !packed) CK(e->in_mask.reserve((size_t)S * 2 + 16));
  const size_t ob[5] = {(size_t)S * sizeof(GrimbCompact), (size_t)r->word_capacity * 8,
                        (size_t)r->general_capacity * sizeof(GrimbSubjectResult),
                        (size_t)r->hap_capacity * sizeof(GrimbHapRow), (size_t)r->pop_capacity * sizeof(GrimbPopRow)};
  for (int i = 0; i < 5; ++i) CK(e->outb[i].reserve(ob[i] + 16));
  GrimbResults dr = *r;
  dr.compact = (GrimbCompact*)e->outb[0].p;
  dr.words = (uint64_t*)e->outb[1].p;
  dr.general = (GrimbSubjectResult*)e->outb[2].p;
  dr.hap_rows = (GrimbHapRow*)e->outb[3].p;
  dr.pop_rows = (GrimbPopRow*)e->outb[4].p;
  // chunking: the ~15 API calls per chunk become the critical path when chunks are small, the pipeline
  // fill / drain (first copy-in, last copy-out not overlapped) when they are large
  int64_t chunk = e->host_chunk;
  if (S > chunk * GRIMB_MAX_CHUNKS) chunk = (S + GRIMB_MAX_CHUNKS - 1) / GRIMB_MAX_CHUNKS;
  chunk = (chunk + 31) & ~(int64_t)31;   // the warp-per-lane kernel starts its ranges on warp boundaries
  int64_t bound[GRIMB_MAX_CHUNKS + 1];
  int nch = 0;
  bound[0] = 0;
  while (bound[nch] < S) {
    bound[nch + 1] = bound[nch] + chunk < S ? bound[nch] + chunk : S;
    ++nch;
  }
  rc = upload_cfg(e, cfg, st);
  if (rc) return rc;
  // GRIMB_HOST_TRACE=1: timeline of the pipeline (CUDA events per chunk; diagnostic only)
  static const bool trace = getenv("GRIMB_HOST_TRACE") != nullptr;
  std::vector<cudaEvent_t> tev;
  if (trace) {
    tev.resize(1 + 3 * (size_t)nch);
    for (auto& x : tev) CK(cudaEventCreate(&x));
    CK(cudaEventRecord(tev[0], st));
    if (nch > 1) {
      CK(cudaStreamWaitEvent(e->s_in, tev[0], 0));
    }
  }
  CK(cudaMemsetAsync(e->d_counters, 0, CNT_N * sizeof(unsigned long long), st));
  if (in_bytes[5]) CK(cudaMemcpyAsync(e->in[5].p, b->priors, in_bytes[5], cudaMemcpyHostToDevice, st));
  // Per chunk: the 16-byte records of its subjects and the words its warp kernels appended (one contiguous
  // range: the counters keep running).  After the last chunk the tail runs once (launch_tail); what it wrote
  // -- general records, their rows, and the records of the subjects it served -- is copied out at the end.
  unsigned long long words_prev = 0, end[CNT_N];
  memset(end, 0, sizeof(end));
  const unsigned long long wcap = (unsigned long long)r->word_capacity;
  auto copy_out = [&](int c) -> int {
    const int64_t s0 = bound[c], n = bound[c + 1] - s0;
    CK(cudaEventSynchronize(e->ev_k[c]));
    const unsigned long long* hc = e->h_cnt + (size_t)CNT_N * c;
    cudaStream_t so = nch > 1 ? e->s_out : st;
    CK(cudaMemcpyAsync(r->compact + s0, dr.compact + s0, (size_t)n * sizeof(GrimbCompact), cudaMemcpyDeviceToHost, so));
    const unsigned long long hi = hc[CNT_WORDS] < wcap ? hc[CNT_WORDS] : wcap;
    if (hi > words_prev) {
      CK(cudaMemcpyAsync(r->words + words_prev, dr.words + words_prev, (size_t)(hi - words_prev) * 8, cudaMemcpyDeviceToHost, so));
      words_prev = hi;
    }
    if (trace) CK(cudaEventRecord(tev[3 + 3 * c], so));
    return GRIMB_OK;
  };
  // copy-in of every chunk is queued first (nothing on the device holds it back), so the in-stream streams
  // the whole batch back to back while the kernels and the copy-out trail one chunk behind
  for (int c = 0; c < nch; ++c) {
    const int64_t s0 = bound[c], s1 = bound[c + 1], n = s1 - s0;
    cudaStream_t si = nch > 1 ? e->s_in : st;
    if (packed) {
      CK(cudaMemcpyAsync((uint64_t*)e->in[3].p + 2 * s0, b->packed_keys + 2 * s0, (size_t)n * 16, cudaMemcpyHostToDevice, si));
      CK(cudaMemcpyAsync((uint16_t*)e->in[0].p + s0, b->packed_flags + s0, (size_t)n * 2, cudaMemcpyHostToDevice, si));
      if (b->prior_index)
        CK(cudaMemcpyAsync((uint32_t*)e->in[4].p + s0, b->prior_index + s0, (size_t)n * 4, cudaMemcpyHostToDevice, si));
      if (nch > 1) CK(cudaEventRecord(e->ev_in[c], si));
      if (trace) CK(cudaEventRecord(tev[1 + 3 * c], si));
      continue;
    }
    const uint32_t a0 = b->allele_off[s0], a1 = b->allele_off[s1];
    CK(cudaMemcpyAsync((uint16_t*)e->in[0].p + s0, b->typed_mask + s0, (size_t)n * 2, cudaMemcpyHostToDevice, si));
    if (b->counts)
      CK(cudaMemcpyAsync((uint16_t*)e->in[1].p + s0 * L * 2, b->counts + s0 * L * 2, (size_t)n * L * 4, cudaMemcpyHostToDevice, si));
    CK(cudaMemcpyAsync((uint32_t*)e->in[2].p + s0, b->allele_off + s0, (size_t)(n + 1) * 4, cudaMemcpyHostToDevice, si));
    if (a1 > a0)
      CK(cudaMemcpyAsync((uint16_t*)e->in[3].p + a0, b->alleles + a0, (size_t)(a1 - a0) * 2, cudaMemcpyHostToDevice, si));
    if (b->prior_index)
      CK(cudaMemcpyAsync((uint32_t*)e->in[4].p + s0, b->prior_index + s0, (size_t)n * 4, cudaMemcpyHostToDevice, si));
    if (b->phase_mask)
      CK(cudaMemcpyAsync((uint16_t*)e->in_mask.p + s0, b->phase_mask + s0, (size_t)n * 2, cudaMemcpyHostToDevice, si));
    if (nch > 1) CK(cudaEventRecord(e->ev_in[c], si));
  }
  mark(0);   // copy-in of every chunk queued
  // the batch as the kernels see it: device arrays of the whole call, subjects addressed by their index in it
  GrimbBatch db = *b;
  db.typed_mask = (const uint16_t*)e->in[0].p;
  db.counts = (b->counts && !packed) ? (const uint16_t*)e->in[1].p : nullptr;
  db.allele_off = (const uint32_t*)e->in[2].p;
  db.alleles = (const uint16_t*)e->in[3].p;
  if (packed) {
    db.packed_keys = (const uint64_t*)e->in[3].p;
    db.packed_flags = (const uint16_t*)e->in[0].p;
    db.typed_mask = nullptr;
    db.allele_off = nullptr;
    db.alleles = nullptr;
  }
  db.prior_index = b->prior_index ? (const uint32_t*)e->in[4].p : nullptr;
  db.priors = (const double*)e->in[5].p;
  db.phase_mask = (b->phase_mask && !packed) ? (const uint16_t*)e->in_mask.p : nullptr;
  const OutArrays O = out_arrays(e, dr);
  const bool tm = e->timing_host != 0;
  reset_event_flags(e);
  const bool warp = warp_kernels_apply(e, cfg, &db);
  for (int c = 0; c < nch; ++c) {
    if (nch > 1) CK(cudaStreamWaitEvent(st, e->ev_in[c], 0));
    if (warp) {
      rc = launch_warp(e, cfg, &db, O, st, tm, bound[c], bound[c + 1]);
      if (rc) return rc;
      k_snapshot<<<1, 32, 0, st>>>(e->d_counters, e->h_cnt_dev + (size_t)CNT_N * c, CNT_N);
      CK(cudaEventRecord(e->ev_k[c], st));
      if (trace) CK(cudaEventRecord(tev[2 + 3 * c], st));
      // with chunk c in the queue, hand chunk c-1 to the copy-out stream
      if (c > 0) {
        rc = copy_out(c - 1);
        if (rc) return rc;
      }
    }
  }
  mark(1);   // warp kernels of every chunk queued, copy-out of all but the last chunk handed over
  // the tail, once: everything the warp kernels handed on (or the whole batch when none serves it).  The length
  // of the hand-over list is read first (the last chunk's counters, through mapped memory): an empty list needs no
  // tail at all, a short one runs on wide CTAs (launch_tail).  The last chunk's copy-out is queued BEHIND the
  // tail: with a single chunk it shares the compute stream, and ahead of the tail it would hold the kernels back
  // (and block this thread when the caller's buffers are pageable).
  int64_t n_tail = warp ? -1 : (int64_t)S;
  if (warp && nch > 0) {
    CK(cudaEventSynchronize(e->ev_k[nch - 1]));
    n_tail = (int64_t)(e->h_cnt[(size_t)CNT_N * (nch - 1) + CNT_WORKLIST] & 0xFFFFFFFFull);
  }
  if (!(warp && n_tail == 0)) {
    rc = launch_tail(e, cfg, &db, O, st, tm, n_tail);
    if (rc) return rc;
  }
  k_snapshot<<<1, 32, 0, st>>>(e->d_counters, e->h_cnt_dev + (size_t)CNT_N * GRIMB_MAX_CHUNKS, CNT_N);
  CK(cudaGetLastError());
  if (warp && nch > 0) {
    rc = copy_out(nch - 1);
    if (rc) return rc;
  }
  mark(2);   // tail queued, last chunk handed to the copy-out stream
  CK(cudaStreamSynchronize(st));
  mark(3);   // compute stream idle
  memcpy(end, e->h_cnt + (size_t)CNT_N * GRIMB_MAX_CHUNKS, sizeof(end));
  const double wl = (double)(unsigned int)(end[CNT_WORKLIST] & 0xFFFFFFFFull);
  {
    const unsigned long long tail_subjects = end[CNT_WORKLIST] & 0xFFFFFFFFull;
    // records written by the tail: every subject's when no warp kernel ran, else those of the handed-on ones
    // (scattered: the array is copied again as a whole, 16 bytes per subject)
    if (!warp || tail_subjects > (unsigned long long)S / 8) {
      CK(cudaMemcpyAsync(r->compact, dr.compact, (size_t)S * sizeof(GrimbCompact), cudaMemcpyDeviceToHost, st));
    } else if (tail_subjects > 0) {
      // few subjects: their records are gathered on the device and scattered into place here
      const uint32_t nw = (uint32_t)(end[CNT_WORKLIST] & 0xFFFFFFFFull), no = 0u;
      const size_t nt = (size_t)nw + no, bytes = nt * (sizeof(GrimbCompact) + 4);
      CK(e->gather.reserve(bytes + 64));
      if (e->h_gather_cap < bytes) {
        if (e->h_gather) cudaFreeHost(e->h_gather);
        e->h_gather = nullptr;
        e->h_gather_cap = 0;
        CK(cudaMallocHost(&e->h_gather, bytes * 2 + 4096));
        e->h_gather_cap = bytes * 2 + 4096;
      }
      GrimbCompact* gc = (GrimbCompact*)e->gather.p;
      uint32_t* gi = (uint32_t*)(gc + nt);
      if (nw) k_gather_compact<<<nblk(nw), 256, 0, st>>>((const uint32_t*)e->worklist.p, nw, dr.compact, gc, gi);
      CK(cudaMemcpyAsync(e->h_gather, e->gather.p, bytes, cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
      const GrimbCompact* hc = (const GrimbCompact*)e->h_gather;
      const uint32_t* hi = (const uint32_t*)(hc + nt);
      if (nch > 1) CK(cudaStreamSynchronize(e->s_out));   // the per-chunk copies of the same records come first
      for (size_t k = 0; k < nt; ++k) r->compact[hi[k]] = hc[k];
    }
    const unsigned long long whi = end[CNT_WORDS] < wcap ? end[CNT_WORDS] : wcap;
    if (whi > words_prev)
      CK(cudaMemcpyAsync(r->words + words_prev, dr.words + words_prev, (size_t)(whi - words_prev) * 8, cudaMemcpyDeviceToHost, st));
    const unsigned long long ng = std::min<unsigned long long>(end[CNT_GENERAL], (unsigned long long)r->general_capacity);
    const unsigned long long nh = std::min<unsigned long long>(end[CNT_HAP], (unsigned long long)r->hap_capacity);
    const unsigned long long np = std::min<unsigned long long>(end[CNT_POP], (unsigned long long)r->pop_capacity);
    if (ng) CK(cudaMemcpyAsync(r->general, dr.general, (size_t)ng * sizeof(GrimbSubjectResult), cudaMemcpyDeviceToHost, st));
    if (nh) CK(cudaMemcpyAsync(r->hap_rows, dr.hap_rows, (size_t)nh * sizeof(GrimbHapRow), cudaMemcpyDeviceToHost, st));
    if (np) CK(cudaMemcpyAsync(r->pop_rows, dr.pop_rows, (size_t)np * sizeof(GrimbPopRow), cudaMemcpyDeviceToHost, st));
  }
  if (nch > 1) CK(cudaStreamSynchronize(e->s_out));
  CK(cudaStreamSynchronize(st));
  mark(4);
  if (trace) {
    fprintf(stderr, "impute_host host clock (ms since entry): copy-in queued %.3f, chunks queued %.3f, tail queued %.3f, compute idle %.3f, all done %.3f\n",
            hmark[0], hmark[1], hmark[2], hmark[3], hmark[4]);
    fprintf(stderr, "impute_host trace (ms after the call's first event): chunk: copy-in done / kernels done / copy-out done\n");
    for (int c = 0; c < nch; ++c) {
      float a = -1, k = -1, o = -1;
      if (packed) cudaEventElapsedTime(&a, tev[0], tev[1 + 3 * c]);
      if (warp) cudaEventElapsedTime(&k, tev[0], tev[2 + 3 * c]);
      if (warp) cudaEventElapsedTime(&o, tev[0], tev[3 + 3 * c]);
      fprintf(stderr, "  %d: %.3f / %.3f / %.3f\n", c, a, k, o);
    }
    cudaGetLastError();
    for (auto& x : tev) cudaEventDestroy(x);
  }
  e->last_worklist = wl;
  return totals_from(end, wl, r);
}

// ------------------------------------------------------------------------------------------
// Device-resident genotype interface (include/grimb200.h): genotype tensor -> GrimbBatch, and the
// results of a finished call -> ragged rows.  Integer work only; probabilities are copied as bits.
// ------------------------------------------------------------------------------------------
enum { GENO_PARTIAL = 0, GENO_ALLELES = 1 };   // geno_small counters: valid subjects typed at some loci only, allele ids

// Small per-call parameters of k_geno_encode, in device memory (indexed per locus / pattern).
struct GenoParams {
  uint32_t allow[16];           // bit m: typed-locus pattern m is a Plan_A_Matrix row (all ones without a matrix)
  uint32_t n_alleles[GRIMB_MAX_LOCI];
  uint8_t shift[GRIMB_MAX_LOCI], width[GRIMB_MAX_LOCI];
};

// Per-locus validation of both genotype encoders.  n0 / n1: ids listed on side 0 / side 1; lo / hi: the smallest /
// largest of them; cap: the largest id the locus's key field holds.  Both sides empty = untyped; exactly one side
// empty, an id 0 or an id wider than the key field = a bad subject (GRIMB_ST_SKIPPED).
enum { GENO_UNTYPED = 0, GENO_TYPED = 1, GENO_BAD = 2 };
__device__ __forceinline__ int geno_locus(uint32_t n0, uint32_t n1, uint32_t lo, uint32_t hi, uint32_t cap) {
  if ((n0 | n1) == 0u) return GENO_UNTYPED;
  return (n0 == 0u || n1 == 0u || lo == 0u || hi > cap) ? GENO_BAD : GENO_TYPED;
}
// The subject's typed-locus pattern: at least one locus, and a Plan_A_Matrix row when a matrix is in force.
__device__ __forceinline__ bool geno_pattern_ok(const GenoParams* gp, uint32_t mask) {
  return mask != 0u && ((gp->allow[mask >> 5] >> (mask & 31u)) & 1u);
}

static GenoParams geno_params(const TablesView& tv, const uint8_t* type_allowed) {
  GenoParams gp;
  memset(&gp, 0, sizeof(gp));
  for (uint32_t m = 0; m < (1u << tv.L); ++m)
    if (!type_allowed || type_allowed[m]) gp.allow[m >> 5] |= 1u << (m & 31u);
  for (int l = 0; l < tv.L; ++l) {
    gp.n_alleles[l] = tv.n_alleles[l];
    gp.shift[l] = tv.shift[l];
    gp.width[l] = tv.width[l];
  }
  return gp;
}

// One thread per subject: validate, write typed_mask and the allele count (scanned into allele_off later),
// and -- when the packed form may serve this build -- the two packed keys and the flag word.
template <bool PACK>
__global__ void __launch_bounds__(256) k_geno_encode(const uint32_t* __restrict__ ids, int64_t S, int L,
                                                     const GenoParams* __restrict__ gp, uint16_t* __restrict__ typed_mask,
                                                     uint32_t* __restrict__ count, uint64_t* __restrict__ keys,
                                                     uint16_t* __restrict__ flags, unsigned long long* __restrict__ small) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t typed = 0;
  if (s < S) {
    uint32_t mask = 0;
    bool bad = false;
    uint64_t k0 = 0, k1 = 0;
    uint32_t fl = 0;
    const uint32_t* p = ids + s * L;
    for (int l = 0; l < L; ++l) {
      const uint32_t v = __ldg(p + l);
      const uint32_t a0 = v & 0xFFFFu, a1 = v >> 16;
      const uint32_t sh = gp->shift[l], cap = (1u << gp->width[l]) - 1u;
      const int st = geno_locus(a0 != 0u, a1 != 0u, min(a0, a1), max(a0, a1), cap);
      if (st == GENO_UNTYPED) continue;
      if (st == GENO_BAD) bad = true;
      mask |= 1u << l;
      if (PACK) {
        k0 |= (uint64_t)a0 << sh;
        k1 |= (uint64_t)a1 << sh;
        fl |= (a0 != a1 ? 1u : 0u) << l;
        fl |= (a0 > gp->n_alleles[l] ? 1u : 0u) << (5 + l);
        fl |= (a1 > gp->n_alleles[l] ? 1u : 0u) << (10 + l);
      }
    }
    if (!geno_pattern_ok(gp, mask)) bad = true;
    typed = bad ? 0u : mask;
    typed_mask[s] = (uint16_t)typed;
    count[s] = 2u * (uint32_t)__popc(typed);
    if (PACK) {
      const bool full = typed == (1u << L) - 1u;
      keys[2 * s] = full ? k0 : 0ull;
      keys[2 * s + 1] = full ? k1 : 0ull;
      flags[s] = (uint16_t)(full ? fl : 0x8000u);
    }
  }
  // warp-aggregated counters: subjects the packed form cannot carry, allele ids of the general form
  const bool partial = typed != 0u && typed != (1u << L) - 1u;
  const unsigned int np = __popc(__ballot_sync(0xFFFFFFFFu, partial));
  unsigned int na = 2u * (unsigned int)__popc(typed);
  for (int o = 16; o > 0; o >>= 1) na += __shfl_xor_sync(0xFFFFFFFFu, na, o);
  if ((threadIdx.x & 31u) == 0u) {
    if (np) atomicAdd(small + GENO_PARTIAL, (unsigned long long)np);
    if (na) atomicAdd(small + GENO_ALLELES, (unsigned long long)na);
  }
}

// General form: the typed loci's ids, side 0 then side 1, at the subject's scanned offset.
__global__ void __launch_bounds__(256) k_geno_fill(const uint32_t* __restrict__ ids, int64_t S, int L,
                                                   const uint16_t* __restrict__ typed_mask, const uint32_t* __restrict__ off,
                                                   uint16_t* __restrict__ alleles) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  const uint32_t typed = typed_mask[s];
  uint32_t o = off[s];
  const uint32_t* p = ids + s * L;
  for (int l = 0; l < L; ++l) {
    if (!((typed >> l) & 1u)) continue;
    const uint32_t v = __ldg(p + l);
    alleles[o] = (uint16_t)(v & 0xFFFFu);
    alleles[o + 1] = (uint16_t)(v >> 16);
    o += 2;
  }
}

extern "C" int grimb_batch_from_genotypes(GrimbEngine* e, const uint16_t* ids, int64_t n_subjects, const uint32_t* prior_index,
                                          const double* priors, int32_t n_priors, const uint8_t* type_allowed, GrimbBatch* out,
                                          void* cuda_stream) {
  if (!e || !out || !priors || n_priors < 1) return fail(GRIMB_E_ARG, "null argument");
  if (n_subjects < 0 || n_subjects > 0x7FFFFFF0ll) return fail(GRIMB_E_ARG, "bad n_subjects");
  if (n_subjects > 0 && (!ids || ((uintptr_t)ids & 3u))) return fail(GRIMB_E_ARG, "ids must be a 4-byte aligned device array");
  CK(cudaSetDevice(e->device));
  const TablesView& tv = e->tables->view;
  const int L = tv.L;
  const int64_t S = n_subjects;
  cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : e->stream;
  const GenoParams gp = geno_params(tv, type_allowed);
  const bool packable = GRIMB_KW == 1 && L <= 5;
  CK(e->geno_mask.reserve((size_t)S * 2 + 16));
  CK(e->geno_off.reserve((size_t)(S + 1) * 4 + 16));
  CK(e->geno_small.reserve(64 + sizeof(GenoParams)));
  if (packable) {
    CK(e->geno_keys.reserve((size_t)S * 16 + 16));
    CK(e->geno_flags.reserve((size_t)S * 2 + 16));
  }
  unsigned long long* small = (unsigned long long*)e->geno_small.p;
  GenoParams* d_gp = (GenoParams*)((char*)e->geno_small.p + 64);
  CK(cudaMemsetAsync(small, 0, 64, st));
  CK(cudaMemcpyAsync(d_gp, &gp, sizeof(gp), cudaMemcpyHostToDevice, st));
  uint32_t* off = (uint32_t*)e->geno_off.p;
  CK(cudaMemsetAsync(off + S, 0, 4, st));
  e->ev_geno_valid = 0;
  if (S > 0) {
    if (e->timing) CK(cudaEventRecord(e->ev_geno[0], st));
    const unsigned g = nblk((uint64_t)S);
    if (packable)
      k_geno_encode<true><<<g, 256, 0, st>>>((const uint32_t*)ids, S, L, d_gp, (uint16_t*)e->geno_mask.p, off,
                                            (uint64_t*)e->geno_keys.p, (uint16_t*)e->geno_flags.p, small);
    else
      k_geno_encode<false><<<g, 256, 0, st>>>((const uint32_t*)ids, S, L, d_gp, (uint16_t*)e->geno_mask.p, off, nullptr, nullptr,
                                             small);
    CK(cudaGetLastError());
    if (e->timing) CK(cudaEventRecord(e->ev_geno[1], st));
    e->ev_geno_valid = e->timing ? 1 : 0;
    e->launches += 1;
  }
  CK(cudaMemcpyAsync(e->h_small, small, 16, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  const unsigned long long partial = e->h_small[GENO_PARTIAL], n_ids = e->h_small[GENO_ALLELES];
  GrimbBatch b;
  memset(&b, 0, sizeof(b));
  b.n_subjects = S;
  b.prior_index = prior_index;
  b.priors = priors;
  b.n_priors = n_priors;
  if (packable && partial == 0) {
    b.packed_keys = (const uint64_t*)e->geno_keys.p;
    b.packed_flags = (const uint16_t*)e->geno_flags.p;
    *out = b;
    return GRIMB_OK;
  }
  if (n_ids > 0xFFFFFFF0ull) return fail(GRIMB_E_ARG, "more than 2^32 allele ids in one batch");
  CK(e->geno_alleles.reserve((size_t)n_ids * 2 + 16));
  if (S > 0) {
    size_t tb = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, tb, off, off, (int)(S + 1), st));
    CK(e->scan_tmp.reserve(tb + 16));
    if (e->timing) CK(cudaEventRecord(e->ev_geno[2], st));
    CK(cub::DeviceScan::ExclusiveSum(e->scan_tmp.p, tb, off, off, (int)(S + 1), st));
    k_geno_fill<<<nblk((uint64_t)S), 256, 0, st>>>((const uint32_t*)ids, S, L, (const uint16_t*)e->geno_mask.p, off,
                                                  (uint16_t*)e->geno_alleles.p);
    CK(cudaGetLastError());
    if (e->timing) CK(cudaEventRecord(e->ev_geno[3], st));
    e->ev_geno_valid |= e->timing ? 2 : 0;
    e->launches += 2;
  }
  b.typed_mask = (const uint16_t*)e->geno_mask.p;
  b.counts = nullptr;
  b.allele_off = off;
  b.alleles = (const uint16_t*)e->geno_alleles.p;
  b.n_alleles_total = (int64_t)n_ids;
  *out = b;
  return GRIMB_OK;
}

// ---- ragged allele lists (grimb_batch_from_genotype_lists) ----

// One thread per subject: the number of ids the subject lists, i.e. its share of the caller's `alleles` (64-bit, so
// that no sum of counts can wrap onto the caller's n_alleles); scanned into the input offsets.
__global__ void __launch_bounds__(256) k_gl_count(const uint16_t* __restrict__ counts, int64_t S, int L,
                                                  unsigned long long* __restrict__ in_off) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  const uint16_t* c = counts + s * 2 * L;
  unsigned long long n = 0;
  for (int i = 0; i < 2 * L; ++i) n += __ldg(c + i);
  in_off[s] = n;
}

// One thread per subject: validate (geno_locus, geno_pattern_ok), drop repeated ids of each side's list (the first
// occurrence stays, as the host tokenisers do), and write the kept ids to `stage` at the subject's input offset,
// the de-duplicated counts, the typed mask and the subject's kept total (scanned into allele_off next).  A bad
// subject gets typed mask 0, counts 0 and total 0.  Lists may be long (40+ ids on a side): the repeat test walks
// the side's earlier ids in the input, no fixed-size table.
__global__ void __launch_bounds__(256) k_gl_dedup(const uint16_t* __restrict__ counts, const uint16_t* __restrict__ alleles,
                                                  const unsigned long long* __restrict__ in_off, int64_t S, int L,
                                                  const GenoParams* __restrict__ gp, uint16_t* __restrict__ stage,
                                                  uint16_t* __restrict__ typed_mask, uint16_t* __restrict__ dcounts,
                                                  uint32_t* __restrict__ dtot) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  const uint16_t* c = counts + s * 2 * L;
  uint16_t* dc = dcounts + s * 2 * L;
  const unsigned long long base = in_off[s];
  const uint16_t* src = alleles + base;
  uint16_t* dst = stage + base;
  uint32_t pos = 0, kept = 0, mask = 0;
  bool bad = false;
  for (int l = 0; l < L; ++l) {
    const uint32_t n0 = __ldg(c + 2 * l), n1 = __ldg(c + 2 * l + 1);
    uint32_t lo = 0xFFFFu, hi = 0u;
    for (int x = 0; x < 2; ++x) {
      const uint32_t n = x ? n1 : n0, first = pos;
      uint32_t k = 0;
      for (; pos < first + n; ++pos) {
        const uint32_t v = __ldg(src + pos);
        lo = min(lo, v);
        hi = max(hi, v);
        bool dup = false;
        for (uint32_t j = first; j < pos && !dup; ++j) dup = __ldg(src + j) == v;
        if (!dup) dst[kept + k++] = (uint16_t)v;
      }
      dc[2 * l + x] = (uint16_t)k;
      kept += k;
    }
    const int st = geno_locus(n0, n1, lo, hi, (1u << gp->width[l]) - 1u);
    if (st == GENO_BAD) bad = true;
    if (st != GENO_UNTYPED) mask |= 1u << l;
  }
  if (!geno_pattern_ok(gp, mask)) bad = true;
  if (bad) {
    for (int i = 0; i < 2 * L; ++i) dc[i] = 0;
    mask = kept = 0;
  }
  typed_mask[s] = (uint16_t)mask;
  dtot[s] = kept;
}

// One thread per subject: the kept ids from the subject's input offset to its de-duplicated offset.
__global__ void __launch_bounds__(256) k_gl_fill(const uint16_t* __restrict__ stage, const unsigned long long* __restrict__ in_off,
                                                 const uint32_t* __restrict__ off, int64_t S, uint16_t* __restrict__ alleles) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  const uint16_t* src = stage + in_off[s];
  const uint32_t o = off[s], n = off[s + 1] - o;
  for (uint32_t i = 0; i < n; ++i) alleles[o + i] = src[i];
}

extern "C" int grimb_batch_from_genotype_lists(GrimbEngine* e, const uint16_t* counts, const uint16_t* alleles, int64_t n_alleles,
                                               int64_t n_subjects, const uint32_t* prior_index, const double* priors,
                                               int32_t n_priors, const uint16_t* phase_mask, const uint8_t* type_allowed,
                                               GrimbBatch* out, void* cuda_stream) {
  if (!e || !out || !priors || n_priors < 1) return fail(GRIMB_E_ARG, "null argument");
  if (n_subjects < 0 || n_subjects > 0x7FFFFFF0ll) return fail(GRIMB_E_ARG, "bad n_subjects");
  if (n_alleles < 0 || n_alleles > 0xFFFFFFF0ll) return fail(GRIMB_E_ARG, "bad n_alleles (at most 2^32 - 16 ids)");
  if (n_subjects > 0 && !counts) return fail(GRIMB_E_ARG, "counts missing");
  if (n_alleles > 0 && !alleles) return fail(GRIMB_E_ARG, "alleles missing");
  CK(cudaSetDevice(e->device));
  const TablesView& tv = e->tables->view;
  const int L = tv.L;
  const int64_t S = n_subjects;
  cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : e->stream;
  const GenoParams gp = geno_params(tv, type_allowed);
  CK(e->gl_in_off.reserve((size_t)(S + 1) * 8 + 16));
  CK(e->gl_mask.reserve((size_t)S * 2 + 16));
  CK(e->gl_counts.reserve((size_t)S * L * 4 + 16));
  CK(e->gl_off.reserve((size_t)(S + 1) * 4 + 16));
  CK(e->geno_small.reserve(64 + sizeof(GenoParams)));
  unsigned long long* small = (unsigned long long*)e->geno_small.p;
  GenoParams* d_gp = (GenoParams*)((char*)e->geno_small.p + 64);
  unsigned long long* in_off = (unsigned long long*)e->gl_in_off.p;
  uint32_t* off = (uint32_t*)e->gl_off.p;
  CK(cudaMemcpyAsync(d_gp, &gp, sizeof(gp), cudaMemcpyHostToDevice, st));
  CK(cudaMemsetAsync(in_off + S, 0, 8, st));
  CK(cudaMemsetAsync(off + S, 0, 4, st));
  e->ev_gl_valid = 0;
  // pass 1 reads the counts only: the caller's lengths are checked before any kernel reads `alleles`
  size_t tb = 0, tb32 = 0;
  if (S > 0) {
    CK(cub::DeviceScan::ExclusiveSum(nullptr, tb, in_off, in_off, (int)(S + 1), st));
    CK(cub::DeviceScan::ExclusiveSum(nullptr, tb32, off, off, (int)(S + 1), st));
    CK(e->scan_tmp.reserve((tb > tb32 ? tb : tb32) + 16));
    if (e->timing) CK(cudaEventRecord(e->ev_gl[0], st));
    k_gl_count<<<nblk((uint64_t)S), 256, 0, st>>>(counts, S, L, in_off);
    CK(cudaGetLastError());
    CK(cub::DeviceScan::ExclusiveSum(e->scan_tmp.p, tb, in_off, in_off, (int)(S + 1), st));
    if (e->timing) CK(cudaEventRecord(e->ev_gl[1], st));
    e->ev_gl_valid = e->timing ? 1 : 0;
    e->launches += 2;
  }
  CK(cudaMemcpyAsync(e->h_small, in_off + S, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if ((long long)e->h_small[0] != n_alleles || e->h_small[0] > 0xFFFFFFF0ull)
    return fail(GRIMB_E_ARG, "the counts list a different number of ids than n_alleles");
  CK(e->gl_stage.reserve((size_t)n_alleles * 2 + 16));
  CK(e->gl_alleles.reserve((size_t)n_alleles * 2 + 16));
  if (S > 0) {
    if (e->timing) CK(cudaEventRecord(e->ev_gl[2], st));
    k_gl_dedup<<<nblk((uint64_t)S), 256, 0, st>>>(counts, alleles, in_off, S, L, d_gp, (uint16_t*)e->gl_stage.p,
                                                 (uint16_t*)e->gl_mask.p, (uint16_t*)e->gl_counts.p, off);
    CK(cudaGetLastError());
    CK(cub::DeviceScan::ExclusiveSum(e->scan_tmp.p, tb32, off, off, (int)(S + 1), st));
    k_gl_fill<<<nblk((uint64_t)S), 256, 0, st>>>((const uint16_t*)e->gl_stage.p, in_off, off, S, (uint16_t*)e->gl_alleles.p);
    CK(cudaGetLastError());
    if (e->timing) CK(cudaEventRecord(e->ev_gl[3], st));
    e->ev_gl_valid |= e->timing ? 2 : 0;
    e->launches += 3;
  }
  // the de-duplicated total, for n_alleles_total
  CK(cudaMemcpyAsync(e->h_small + 1, off + S, 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  GrimbBatch b;
  memset(&b, 0, sizeof(b));
  b.n_subjects = S;
  b.typed_mask = (const uint16_t*)e->gl_mask.p;
  b.counts = (const uint16_t*)e->gl_counts.p;
  b.allele_off = off;
  b.alleles = (const uint16_t*)e->gl_alleles.p;
  b.n_alleles_total = (int64_t)(uint32_t)e->h_small[1];
  b.prior_index = prior_index;
  b.priors = priors;
  b.n_priors = n_priors;
  b.phase_mask = phase_mask;
  *out = b;
  return GRIMB_OK;
}

// What the row decoder needs of the configuration, by value.
struct RowsCfg {
  int32_t L, out_u, out_p, n_results, n_pop_results, hap_pop_pair;
};

// Per-subject view of a result record (GrimbCompact + its words or its GrimbSubjectResult), the one place
// that reads the record layout of include/grimb200.h for the decoder.
struct RowsRec {
  uint32_t status, kind, has, n[4];        // rows per kind (GRIMB_ROWS_*), gated by status and configuration
  uint32_t plan_u, plan_p, tot_u, tot_p;
  uint32_t n_pm;                           // SIMPLE / TYPED: PMUG rows of the record
  uint64_t phases;                         // SIMPLE: 4 bits per row; TYPED: the header (12 bits per row from bit 16)
  const uint64_t* pm_prob;                 // SIMPLE / TYPED: PMUG probabilities (nullptr: `total`)
  const uint64_t* pop_prob;                // TYPED: population-pair probabilities, then their codes
  const uint64_t* pop_code;
  double total;
  const GrimbSubjectResult* g;             // GENERAL (nullptr: no record)
};

__device__ __forceinline__ RowsRec rows_record(const GrimbResults& R, const RowsCfg& c, uint64_t s) {
  RowsRec r;
  const GrimbCompact cp = R.compact[s];
  r.status = cp.status;
  r.kind = cp.kind_flags & 3u;
  r.has = (cp.kind_flags & GRIMB_KIND_HAS_RESULTS) ? 1u : 0u;
  r.total = cp.total;
  r.g = nullptr;
  r.pm_prob = r.pop_prob = r.pop_code = nullptr;
  r.phases = 0;
  r.n_pm = 0;
  r.n[0] = r.n[1] = r.n[2] = r.n[3] = 0;
  r.plan_u = r.plan_p = r.tot_u = r.tot_p = 0;
  const bool ok = r.status == GRIMB_ST_OK;
  if (r.kind == GRIMB_KIND_GENERAL) {
    if (cp.off != 0xFFFFFFFFu && (int64_t)cp.off < R.general_capacity) {
      r.g = R.general + cp.off;
      const GrimbSubjectResult& g = *r.g;
      r.plan_u = g.plan_umug;
      r.plan_p = g.plan_pmug;
      r.tot_u = g.tot_umug;
      r.tot_p = g.tot_pmug;
      if (ok) {
        r.n[0] = c.out_u ? g.n_umug : 0u;
        r.n[1] = c.out_p ? g.n_pmug : 0u;
        r.n[2] = c.out_u ? g.n_umug_pops : 0u;
        r.n[3] = c.out_p ? g.n_pmug_pops : 0u;
      }
    }
    return r;
  }
  const uint64_t* w = R.words + cp.off;
  uint32_t n_pm = cp.kind_flags >> 4, n_pops;
  if (r.kind == GRIMB_KIND_SIMPLE && n_pm == 15u) {   // long form: a count word, a word of phase ids, the probabilities
    n_pm = w[0] > 16u ? 16u : (uint32_t)w[0];
    r.phases = w[1];
    r.pm_prob = w + 2;
    n_pops = (r.has && c.n_pop_results >= 1) ? 1u : 0u;
  } else if (r.kind == GRIMB_KIND_SIMPLE) {
    r.phases = cp.phases;
    r.pm_prob = (cp.kind_flags & GRIMB_KIND_WORDS) ? w : nullptr;
    n_pops = (r.has && c.n_pop_results >= 1) ? 1u : 0u;
  } else {
    r.phases = w[0];
    n_pops = (uint32_t)(w[0] & 0xFFFFu);
    r.pm_prob = w + 1;
    r.pop_prob = w + 1 + n_pm;
    r.pop_code = r.pop_prob + n_pops;
  }
  r.n_pm = n_pm;
  r.plan_u = c.out_u ? GRIMB_PLAN_A : GRIMB_PLAN_NONE;
  r.plan_p = c.out_p ? GRIMB_PLAN_A : GRIMB_PLAN_NONE;
  r.tot_u = (r.has && c.out_u) ? 1u : 0u;
  r.tot_p = c.out_p ? (r.has ? (n_pm > 1u ? n_pm : 1u) : 0u) : 0u;
  if (ok) {
    r.n[0] = (c.out_u && r.has && c.n_results >= 1) ? 1u : 0u;
    r.n[1] = c.out_p ? n_pm : 0u;
    r.n[2] = (c.out_u && r.has) ? n_pops : 0u;
    r.n[3] = c.out_p ? n_pops : 0u;
  }
  return r;
}

__global__ void __launch_bounds__(256) k_rows_count(GrimbResults R, RowsCfg c, int64_t S, GrimbRows O) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  const RowsRec r = rows_record(R, c, (uint64_t)s);
  uint32_t fl = r.has ? GRIMB_ROWS_HAS_RESULTS : 0u;
  if (r.status == GRIMB_ST_OK && c.out_p && r.tot_p == 0u && r.tot_u == 0u) fl |= GRIMB_ROWS_MISS;
  if (r.status == GRIMB_ST_SKIPPED || r.status == GRIMB_ST_FAULT || (r.status == GRIMB_ST_NO_PHASES && c.out_p))
    fl |= GRIMB_ROWS_PROBLEM;
  O.status[s] = (uint8_t)r.status;
  O.plan_umug[s] = (uint8_t)r.plan_u;
  O.plan_pmug[s] = (uint8_t)r.plan_p;
  O.flags[s] = (uint8_t)fl;
  O.tot_umug[s] = r.tot_u;
  O.tot_pmug[s] = r.tot_p;
  for (int k = 0; k < 4; ++k) O.off[k][s] = (int64_t)r.n[k];
}

// the packed key of a hap row (GRIMB_KEY_WORDS little-endian words)
__device__ __forceinline__ hkey row_key_a(const GrimbHapRow& h) {
#if GRIMB_KW == 1
  return h.a;
#else
  return (hkey)h.a[0] | ((hkey)h.a[1] << 64);
#endif
}
__device__ __forceinline__ hkey row_key_b(const GrimbHapRow& h) {
#if GRIMB_KW == 1
  return h.b;
#else
  return (hkey)h.b[0] | ((hkey)h.b[1] << 64);
#endif
}

__global__ void __launch_bounds__(256) k_rows_fill(GrimbResults R, RowsCfg c, int64_t S, GrimbBatch B, TablesView T, GrimbRows O) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  const RowsRec r = rows_record(R, c, (uint64_t)s);
  if ((r.n[0] | r.n[1] | r.n[2] | r.n[3]) == 0u) return;
  const int L = c.L;
  int64_t o[4];
  for (int k = 0; k < 4; ++k) o[k] = O.off[k][s];
  uint16_t* um = O.rows[GRIMB_ROWS_UMUG] + o[0] * 2 * L;
  uint16_t* pm = O.rows[GRIMB_ROWS_PMUG] + o[1] * 2 * L;
  double* ump = O.prob[GRIMB_ROWS_UMUG] + o[0];
  double* pmp = O.prob[GRIMB_ROWS_PMUG] + o[1];
  if (r.g) {
    const GrimbSubjectResult& g = *r.g;
    for (uint32_t q = 0; q < r.n[0]; ++q) {
      const GrimbHapRow h = R.hap_rows[g.hap_off + q];
      const hkey a = row_key_a(h), b = row_key_b(h);
      for (int l = 0; l < L; ++l) {
        const uint32_t x = (uint32_t)key_field(T, a, l), y = (uint32_t)key_field(T, b, l);
        um[(q * L + l) * 2] = (uint16_t)(x < y ? x : y);
        um[(q * L + l) * 2 + 1] = (uint16_t)(x < y ? y : x);
      }
      ump[q] = h.prob;
    }
    for (uint32_t q = 0; q < r.n[1]; ++q) {
      const GrimbHapRow h = R.hap_rows[g.hap_off + g.n_umug + q];
      const hkey a = row_key_a(h), b = row_key_b(h);
      for (int l = 0; l < L; ++l) {
        pm[(q * 2) * L + l] = (uint16_t)key_field(T, a, l);
        pm[(q * 2 + 1) * L + l] = (uint16_t)key_field(T, b, l);
      }
      pmp[q] = h.prob;
    }
    if (c.hap_pop_pair) {   // the companion pop row of PMUG row q, after the UMUG and PMUG pop rows
      const GrimbPopRow* cp = R.pop_rows + g.pop_off + g.n_umug_pops + g.n_pmug_pops;
      for (uint32_t q = 0; q < r.n[1]; ++q) {
        const GrimbPopRow p = cp[q];
        O.pmug_pairs[(o[1] + q) * 2] = p.pop_a;
        O.pmug_pairs[(o[1] + q) * 2 + 1] = p.pop_b;
      }
    }
    for (int k = 2; k < 4; ++k) {
      const uint64_t base = g.pop_off + (k == 3 ? g.n_umug_pops : 0u);
      for (uint32_t q = 0; q < r.n[k]; ++q) {
        const GrimbPopRow p = R.pop_rows[base + q];
        O.rows[k][(o[k] + q) * 2] = p.pop_a;
        O.rows[k][(o[k] + q) * 2 + 1] = p.pop_b;
        O.prob[k][o[k] + q] = p.prob;
      }
    }
    return;
  }
  // SIMPLE / TYPED: every locus typed with one allele per side; the rows follow from the subject's own alleles
  hkey k0 = 0, k1 = 0;   // side-0 / side-1 alleles in the key layout (registers, not an indexed array)
  if (B.packed_keys) {
    k0 = (hkey)B.packed_keys[2 * s];
    k1 = (hkey)B.packed_keys[2 * s + 1];
  } else {
    const uint16_t* a = B.alleles + B.allele_off[s];
    for (int l = 0; l < L; ++l) {
      k0 |= (hkey)a[2 * l] << T.shift[l];
      k1 |= (hkey)a[2 * l + 1] << T.shift[l];
    }
  }
  if (r.n[0]) {
    for (int l = 0; l < L; ++l) {
      const uint32_t x = (uint32_t)key_field(T, k0, l), y = (uint32_t)key_field(T, k1, l);
      um[2 * l] = (uint16_t)(x < y ? x : y);
      um[2 * l + 1] = (uint16_t)(x < y ? y : x);
    }
    ump[0] = r.total;
  }
  const bool typed = r.kind == GRIMB_KIND_TYPED;
  for (uint32_t q = 0; q < r.n[1]; ++q) {
    const uint32_t ph = typed ? (uint32_t)(r.phases >> (16 + 12 * q)) & 0xFFFu : (uint32_t)(r.phases >> (4 * q)) & 15u;
    for (int l = 0; l < L; ++l) {
      const uint32_t x = (uint32_t)key_field(T, k0, l), y = (uint32_t)key_field(T, k1, l);
      const bool flip = (ph >> l) & 1u;
      pm[(q * 2) * L + l] = (uint16_t)(flip ? y : x);
      pm[(q * 2 + 1) * L + l] = (uint16_t)(flip ? x : y);
    }
    pmp[q] = r.pm_prob ? __longlong_as_double((long long)r.pm_prob[q]) : r.total;
  }
  for (int k = 2; k < 4; ++k) {
    for (uint32_t q = 0; q < r.n[k]; ++q) {
      uint32_t pa = 0, pb = 0;
      double p = r.total;
      if (r.pop_code) {
        const uint32_t code = (uint32_t)(r.pop_code[q >> 2] >> (16 * (q & 3u))) & 0xFFFFu;
        pa = code >> 8;
        pb = code & 0xFFu;
        p = __longlong_as_double((long long)r.pop_prob[q]);
      }
      O.rows[k][(o[k] + q) * 2] = (uint16_t)pa;
      O.rows[k][(o[k] + q) * 2 + 1] = (uint16_t)pb;
      O.prob[k][o[k] + q] = p;
    }
  }
}

extern "C" int grimb_results_rows(GrimbEngine* e, const GrimbConfig* cfg, const GrimbBatch* batch, const GrimbResults* res,
                                  const GrimbRows* rows, void* cuda_stream) {
  if (!e || !cfg || !batch || !res || !rows || !rows->totals) return fail(GRIMB_E_ARG, "null argument");
  if (cfg->hap_pop_pair && !rows->pmug_pairs) return fail(GRIMB_E_ARG, "GrimbRows.pmug_pairs is required under hap_pop_pair");
  const int64_t S = batch->n_subjects;
  if (S < 0 || S > 0x7FFFFFF0ll) return fail(GRIMB_E_ARG, "bad n_subjects");
  for (int k = 0; k < 4; ++k)
    if (!rows->off[k] || rows->capacity[k] < 0) return fail(GRIMB_E_ARG, "GrimbRows.off / capacity");
  if (S > 0) {
    if (!res->compact) return fail(GRIMB_E_ARG, "GrimbResults.compact missing");
    if (!rows->status || !rows->plan_umug || !rows->plan_pmug || !rows->flags || !rows->tot_umug || !rows->tot_pmug)
      return fail(GRIMB_E_ARG, "GrimbRows per-subject arrays missing");
    if (!batch->packed_keys && (!batch->allele_off || !batch->alleles)) return fail(GRIMB_E_ARG, "batch arrays missing");
  }
  CK(cudaSetDevice(e->device));
  cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : e->stream;
  const TablesView& tv = e->tables->view;
  RowsCfg c;
  c.L = tv.L;
  c.out_u = cfg->output_umug ? 1 : 0;
  c.out_p = cfg->output_pmug ? 1 : 0;
  c.n_results = cfg->n_results;
  c.n_pop_results = cfg->n_pop_results;
  c.hap_pop_pair = cfg->hap_pop_pair ? 1 : 0;
  e->ev_rows_valid = 0;
  for (int k = 0; k < 4; ++k) CK(cudaMemsetAsync(rows->off[k] + S, 0, 8, st));
  CK(e->geno_small.reserve(64 + sizeof(GenoParams)));
  unsigned long long* small = (unsigned long long*)e->geno_small.p;
  if (S > 0) {
    size_t tb = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, tb, rows->off[0], rows->off[0], (int)(S + 1), st));
    CK(e->scan_tmp.reserve(tb + 16));
    if (e->timing) CK(cudaEventRecord(e->ev_rows[0], st));
    k_rows_count<<<nblk((uint64_t)S), 256, 0, st>>>(*res, c, S, *rows);
    CK(cudaGetLastError());
    for (int k = 0; k < 4; ++k) CK(cub::DeviceScan::ExclusiveSum(e->scan_tmp.p, tb, rows->off[k], rows->off[k], (int)(S + 1), st));
    if (e->timing) CK(cudaEventRecord(e->ev_rows[1], st));
    e->ev_rows_valid = e->timing ? 1 : 0;
    e->launches += 5;
  }
  for (int k = 0; k < 4; ++k) CK(cudaMemcpyAsync(small + k, rows->off[k] + S, 8, cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(e->h_small, small, 32, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  bool over = false;
  for (int k = 0; k < 4; ++k) {
    rows->totals[k] = (int64_t)e->h_small[k];
    if (rows->totals[k] > rows->capacity[k]) over = true;
    if (rows->totals[k] > 0 && (!rows->rows[k] || !rows->prob[k])) return fail(GRIMB_E_ARG, "GrimbRows row arrays missing");
  }
  if (over) return fail(GRIMB_E_CAPACITY, "row buffers too small (see GrimbRows.totals)");
  if (S > 0 && (rows->totals[0] | rows->totals[1] | rows->totals[2] | rows->totals[3])) {
    if (e->timing) CK(cudaEventRecord(e->ev_rows[2], st));
    k_rows_fill<<<nblk((uint64_t)S), 256, 0, st>>>(*res, c, S, *batch, tv, *rows);
    CK(cudaGetLastError());
    if (e->timing) CK(cudaEventRecord(e->ev_rows[3], st));
    e->ev_rows_valid |= e->timing ? 2 : 0;
    e->launches += 1;
  }
  CK(cudaStreamSynchronize(st));
  return GRIMB_OK;
}
