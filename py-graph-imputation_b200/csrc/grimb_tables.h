// grimb_tables.h -- device view of the frequency store and the probe primitives.
//
// Layout in HBM (DESIGN.md "Data layout"):
//   slots      open-addressing hash table, one region per locus-subset label (the full-label
//              region of a 1M-haplotype table is 128 MB at load 1/8, larger than the L2; the
//              single-population fast path probes the FastIndex below instead);
//              16-byte slots {packed key, node id}, load factor <= 0.5, linear probing, one
//              128-bit load per probe (two slots per 32-byte sector); 32-byte slots when the
//              packed key is 128 bits wide (GRIMB_KW = 2).
//   node_key   packed allele ids of node i (0 in the fields of absent loci)
//   freq       [n_nodes][P] FP64 frequency vectors, reference node-id order
//   tl_*       CSR: partial node -> full nodes containing it (ascending id)   [adjs_query]
//   cn_*       CSR: (child node, added locus) -> parents one locus longer     [adjs_query_by_color]
//   label_*    node-id range of every label                                   [haps_by_label]
#pragma once
#include "grimb_group.h"

namespace grimb {

#define GRIMB_NONE 0xFFFFFFFFu
#define GRIMB_ADJ_FAULT 0xFFFFFFFFu  // tl_cnt/cn_cnt: the reference raises IndexError here (T1)

#if GRIMB_KW == 1
struct HSlot {   // 16 bytes: two slots per 32-byte sector
  hkey key;
  uint32_t node;
  uint32_t pad;
};
#else
struct HSlot {   // 32 bytes: one slot per sector
  hkey key;
  uint32_t node;
  uint32_t pad[3];
};
#endif

struct TablesView {
  int32_t L, P;
  uint32_t n_nodes, n_full;
  uint8_t shift[9];
  uint8_t width[9];
  uint32_t n_alleles[9];
  const uint32_t* label_first;  // [1<<L]
  const uint32_t* label_count;  // [1<<L]
  const uint64_t* ht_off;       // [1<<L] first slot of the label's region
  const uint32_t* ht_mask;      // [1<<L] region size - 1 (power of two)
  const HSlot* slots;
  const hkey* node_key;
  const double* freq;
  const uint32_t* tl_start;
  const uint32_t* tl_cnt;
  const uint32_t* tl_adj;
  const uint32_t* cn_start;     // [n_nodes][L]
  const uint32_t* cn_cnt;
  const uint32_t* cn_adj;
};

#if GRIMB_KW == 1
// Key-only index of the full haplotypes with freq > 0, for the single-population fast path
// (k_fast_probe / k_fast_score; L <= 5, P == 1).  Derived from the image on every device that holds
// one (grimb_tables_build, grimb_tables_from_image), never stored in it.
//   keys   [sec_mask + 1][4] packed keys, four to a 32-byte sector, 0 = empty (every field of a full
//          key is >= 1).  Home sector hash_key(key) & sec_mask, linear probing by sector.  Bit 63 of a
//          sector's first word (keys have <= 63 bits) is set when a key whose home is this sector is
//          stored further on: a miss reads one sector unless it is set.  At 4 slots per haplotype the
//          1M-haplotype table's keys are 32 MB, inside the L2.
//   fslot  frequency of the key in the same slot (k_fast_score reads it; the probe kernel never does)
struct FastIndex {
  const uint64_t* keys;
  const double* fslot;
  uint32_t sec_mask;
};
#define FIDX_FLAG (1ull << 63)
#endif

GD uint64_t key_field(const TablesView& T, hkey key, int locus) {
  return (uint64_t)(key >> T.shift[locus]) & ((1ull << T.width[locus]) - 1ull);
}

GD hkey key_mask_of(const TablesView& T, uint32_t label) {
  hkey m = 0;
  for (int l = 0; l < T.L; ++l)
    if (label >> l & 1u) m |= (hkey)((1ull << T.width[l]) - 1ull) << T.shift[l];
  return m;
}

GD HSlot load_slot(const HSlot* p) {
#if GRIMB_DEVICE
  HSlot s;
#if GRIMB_KW == 1
  uint4 v = __ldg(reinterpret_cast<const uint4*>(p));
  s.key = (uint64_t)v.x | ((uint64_t)v.y << 32);
  s.node = v.z;
  s.pad = v.w;
#else
  // a 32-byte slot is one sector: one 256-bit load (sm_100: LDG.E.256)
  uint32_t r0, r1, r2, r3, r4, r5, r6, r7;
  asm volatile("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3), "=r"(r4), "=r"(r5), "=r"(r6), "=r"(r7)
               : "l"(p));
  s.key = (hkey)((uint64_t)r0 | ((uint64_t)r1 << 32)) | ((hkey)((uint64_t)r2 | ((uint64_t)r3 << 32)) << 64);
  s.node = r4;
  s.pad[0] = s.pad[1] = s.pad[2] = 0;
  (void)r5; (void)r6; (void)r7;
#endif
  return s;
#else
  return *p;
#endif
}

#if GRIMB_KW == 1
// Both slots of a 32-byte sector with ONE 256-bit load (sm_100: LDG.E.256); p must be sector aligned.
GD void load_sector(const HSlot* p, HSlot& s0, HSlot& s1) {
#if GRIMB_DEVICE
  uint32_t r0, r1, r2, r3, r4, r5, r6, r7;
  asm volatile("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3), "=r"(r4), "=r"(r5), "=r"(r6), "=r"(r7)
               : "l"(p));
  s0.key = (uint64_t)r0 | ((uint64_t)r1 << 32);
  s0.node = r2;
  s0.pad = r3;
  s1.key = (uint64_t)r4 | ((uint64_t)r5 << 32);
  s1.node = r6;
  s1.pad = r7;
#else
  s0 = p[0];
  s1 = p[1];
#endif
}
#endif

// Home slot of a key: always the first slot of a 32-byte sector (two 16-byte slots), so a probe
// reads whole sectors -- both slots of a sector come with ONE 256-bit load (load_sector: LDG.E.256).
#if GRIMB_KW == 1
GD uint32_t ht_home(hkey key, uint32_t mask) { return hash_key(key) & mask & ~1u; }

// One probe: hash, then linear scan, a sector (two slots) per step, until the key or an empty slot.
GD uint32_t ht_lookup(const TablesView& T, uint32_t label, hkey key) {
  const uint32_t mask = T.ht_mask[label];
  const HSlot* base = T.slots + T.ht_off[label];
  uint32_t h = ht_home(key, mask);
  for (;;) {
    HSlot s0, s1;
    load_sector(base + h, s0, s1);
    if (s0.node == GRIMB_NONE) return GRIMB_NONE;
    if (s0.key == key) return s0.node;
    if (s1.node == GRIMB_NONE) return GRIMB_NONE;
    if (s1.key == key) return s1.node;
    h = (h + 2) & mask;
  }
}
#else
GD uint32_t ht_home(hkey key, uint32_t mask) { return hash_key(key) & mask; }

// One probe: hash, then linear scan, a sector (one 32-byte slot) per step.
GD uint32_t ht_lookup(const TablesView& T, uint32_t label, hkey key) {
  const uint32_t mask = T.ht_mask[label];
  const HSlot* base = T.slots + T.ht_off[label];
  uint32_t h = ht_home(key, mask);
  for (;;) {
    const HSlot s0 = load_slot(base + h);
    if (s0.node == GRIMB_NONE) return GRIMB_NONE;
    if (s0.key == key) return s0.node;
    h = (h + 1) & mask;
  }
}
#endif

}  // namespace grimb
