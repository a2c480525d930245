/*
 * grimb200.h -- C ABI of libgrimb200.so, the B200 (sm_100a) implementation of the GRIM
 * per-subject imputation hot path.
 *
 * The reference (nmdp-bioinformatics/py-graph-imputation) has no FFI: its seams are Python
 * call signatures.  Each entry point below names the reference interface it stands in for
 * (paths relative to the reference root).  The Python host in
 * py-graph-imputation_b200/grim/ binds these with ctypes; INTEGRATION.md shows the stub a
 * maintainer of the reference would add.
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on success or a
 * negative GRIMB_E_* code (text via grimb_last_error()); no C++ exception crosses the
 * boundary; per-subject failures are status codes in the result arrays, never call failures.
 * The caller owns every buffer it passes; the library owns GrimbTables and GrimbEngine.
 */
#ifndef GRIMB200_H
#define GRIMB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GRIMB_ABI_VERSION 5
#define GRIMB_MAX_LOCI 9
#define GRIMB_MAX_ROWS 16
#define GRIMB_MAX_BLOCKS 9

/* error codes */
#define GRIMB_OK 0
#define GRIMB_E_ARG (-1)      /* bad argument */
#define GRIMB_E_CUDA (-2)     /* CUDA runtime error (no device, launch failure, ...) */
#define GRIMB_E_NOMEM (-3)
#define GRIMB_E_LAYOUT (-4)   /* allele ids do not fit the packed key */
#define GRIMB_E_CAPACITY (-5) /* caller-provided result buffers too small; see grimb_impute_* */
#define GRIMB_E_UNDEFINED (-6) /* the reference has no defined behaviour for this input (Plan B under a Plan_A_Matrix) */

/* per-subject status (GrimbResults.status) */
#define GRIMB_ST_OK 0          /* rows written (possibly zero rows: reference writes .miss) */
#define GRIMB_ST_FAULT 2       /* the reference raises inside this subject -> raw line in .problem */
#define GRIMB_ST_WORKSPACE 3   /* per-CTA workspace too small: re-issue with a bigger workspace */
#define GRIMB_ST_SKIPPED 4     /* not processed (host marked it unparsable: .problem "i,id") */
#define GRIMB_ST_NO_PHASES 5   /* nothing opens after both reductions (impute.py:1620-1629): the reference
                                  returns its defaults; the host reproduces the writer's behaviour */

/* plan that produced the rows (impute.py:216,1638,1702), per output kind */
#define GRIMB_PLAN_NONE 0
#define GRIMB_PLAN_A 1
#define GRIMB_PLAN_B 2
#define GRIMB_PLAN_C 3

typedef struct GrimbTables GrimbTables; /* device-resident frequency store (one per device) */
typedef struct GrimbEngine GrimbEngine; /* per-device workspaces + stream for imputation    */

/* ------------------------------------------------------------------------------------------
 * Frequency store.  Replaces graph_generation/generate_neo4j_multi_hpf.py:209-486
 * (generate_graph: marginal nodes, sequential sums, top links, parent edges) and
 * grim/imputation/networkx_graph.py:42-213 (Graph.build_graph: dicts + CSR), including the
 * CSR sentinel quirk at networkx_graph.py:195-196.  Node ids equal the reference's
 * haplotypeId column.  Input = the unique full haplotypes of hpf.csv after trimming, in
 * first-appearance order, as allele ids (1-based per locus, locus order = loci_map index).
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t n_loci;                         /* L, 1..GRIMB_MAX_LOCI                             */
  int32_t n_pops;                         /* P                                                */
  int64_t n_full;                         /* number of full haplotypes                        */
  const uint16_t* full_alleles;           /* [n_full][L] host, ids 1..n_alleles[l]            */
  const double* full_freqs;               /* [n_full][P] host                                 */
  int32_t n_alleles[GRIMB_MAX_LOCI];      /* table alleles per locus                          */
  int32_t key_bits[GRIMB_MAX_LOCI];       /* packed-key field width per locus (sum <= 63)     */
  int32_t last_parent_locus;              /* locus whose connector is created last (T1), or -1 to derive L-2 */
  int32_t device;                         /* CUDA device ordinal                              */
  /* "Plan_A_Matrix" (generate_neo4j_multi_hpf.py:101-192, networkx_graph.py:32-66): NULL = every locus subset.
   * Else the labels to build, as locus bit masks in node-id order, the full label first: the first
   * n_plan_a_labels are the matrix rows (the vertices of the reference's Plan-A CSR, sentinel quirk included),
   * the rest are labels kept for look-ups only (the single-locus labels the allele-existence checks read).  A
   * restricted store has no connectors: it serves Plan A, which is all the reference computes reliably under
   * a matrix (DESIGN.md section 7). */
  const uint32_t* label_masks;            /* [n_labels] or NULL                               */
  int32_t n_labels;
  int32_t n_plan_a_labels;
} GrimbTableDesc;

int grimb_abi_version(void);
const char* grimb_last_error(void);
/* sizeof of an ABI struct as the library was compiled, for bindings to check their mirror of it: 0 GrimbConfig,
 * 1 GrimbTableDesc, 2 GrimbTextDesc, 3 GrimbBatch, 4 GrimbResults, 5 GrimbTextOut, 6 GrimbFileStats,
 * 7 GrimbTableInfo, 8 GrimbRows; -1 otherwise. */
int64_t grimb_struct_size(int32_t which);

int grimb_tables_build(const GrimbTableDesc* desc, GrimbTables** out);
int grimb_tables_free(GrimbTables* t);

/* Sizes, for tests / export / broadcast: n_nodes, n_full, n_toplinks, n_conn_edges, n_slots */
typedef struct {
  int32_t n_loci, n_pops;
  int64_t n_nodes, n_full, n_toplinks, n_conn_edges, n_slots, device_bytes;
} GrimbTableInfo;
int grimb_tables_info(const GrimbTables* t, GrimbTableInfo* info);
/* Kernel launches grimb_tables_build issued for this table (0 for a table made from an image): the build is
 * batched over labels, about 60 launches for a 5-locus table whatever its size. */
int64_t grimb_tables_build_launches(const GrimbTables* t);
/* Device time of that build in ms, from the staged inputs to the finished image (CUDA events; 0 for an image). */
double grimb_tables_build_ms(const GrimbTables* t);

/* Copies table arrays to host buffers (any pointer may be NULL).  node_key: packed alleles of
 * node id i; node_freq [n_nodes][P]; tl_start/tl_cnt [n_nodes] and tl_adj [n_toplinks] = top
 * links (networkx_graph.py:253-278 view); cn_start/cn_cnt [n_nodes][L] and cn_adj = connector
 * parents for (child node, added locus) (networkx_graph.py:280-307 view); label_first/count
 * [1<<L] node-id range per locus-subset mask (haps_by_label, networkx_graph.py:215-236). */
int grimb_tables_export(const GrimbTables* t, uint64_t* node_key, double* node_freq,
                        uint32_t* tl_start, uint32_t* tl_cnt, uint32_t* tl_adj,
                        uint32_t* cn_start, uint32_t* cn_cnt, uint32_t* cn_adj,
                        uint32_t* label_first, uint32_t* label_count);

/* Raw device image of the tables for replication across GPUs (one ncclBroadcast of this
 * buffer per peer; SURVEY 8(e)): size, then copy out / build from an image on another device. */
int grimb_tables_image_size(const GrimbTables* t, int64_t* bytes);
int grimb_tables_image_ptr(const GrimbTables* t, void** dev_ptr);        /* device pointer */
int grimb_tables_image_copy(const GrimbTables* t, void* dst);            /* dst: host or device, image_size bytes */
int grimb_tables_from_image(const void* image, int64_t bytes, int device, GrimbTables** out); /* image: host or device */

/* ------------------------------------------------------------------------------------------
 * Imputation.  Replaces Imputation.impute_one / comp_cand and everything below them
 * (grim/imputation/impute.py:1584-1724, 1940-1983) for a batch of already-tokenised subjects,
 * plus the top-N selection of write_best_prob / write_best_prob_genotype (impute.py:24-76).
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  /* run_impute_def.py:63-129 keys */
  double epsilon;                     /* "epsilon"                                            */
  double factor_missing_pow[GRIMB_MAX_LOCI + 1]; /* factor_missing_data ** k, k = 0..L (host pow) */
  int64_t options_threshold;          /* "number_of_options_threshold"                        */
  int32_t max_haps_in_phase;          /* "max_haplotypes_number_in_phase" (<= 512)            */
  int32_t n_results;                  /* "number_of_results"                                  */
  int32_t n_pop_results;              /* "number_of_pop_results"                              */
  int32_t planb;                      /* "planb"                                              */
  int32_t output_umug;                /* "output_MUUG"                                        */
  int32_t output_pmug;                /* "output_haplotypes"                                  */
  int32_t save_space;                 /* "save_space_mode"                                    */
  int32_t compensated_sum;            /* 1: Python's sum() of floats is Neumaier-compensated (CPython >= 3.12),
                                         0: plain left-to-right adds (older CPython); affects
                                         allel_to_SR (impute.py:1260-1262) and save-space pruning (:1053) */
  /* "Plan_B_Matrix": rows of blocks, each block a locus bitmask (bit l = loci_map index l+1) */
  int32_t n_rows;
  int32_t row_blocks[GRIMB_MAX_ROWS];
  uint16_t block_mask[GRIMB_MAX_ROWS][GRIMB_MAX_BLOCKS];
  uint8_t row_is_plan_a[GRIMB_MAX_ROWS]; /* impute.py:1118: block 0 == list(set(loci indices)) */
  /* EM-facing modes (SURVEY 8f-4) */
  int32_t hap_pop_pair;               /* grim.impute(hap_pop_pair=True) / impute_file(em_mr=True), impute.py:79-99,
                                         2079-2088: the PMUG rows are the n_results best single (haplotype;pop,
                                         haplotype;pop) pairs, not merged; each PMUG hap row k has a companion
                                         GrimbPopRow with its two populations at
                                         pop_rows[pop_off + n_umug_pops + n_pmug_pops + k]; one PMUG pop row   */
  int32_t em;                         /* impute_file(em=True): no Plan C for the haplotype output (impute.py:1648) */
  int32_t plan_a_only;                /* "Plan_A_Matrix" in force (tables built from a label list): the kernels run
                                         Plan A only whatever `planb` says.  With planb set, the text pipeline
                                         fails with GRIMB_E_UNDEFINED when a subject leaves Plan A without a result:
                                         the reference's Plan B is not well defined under a matrix (DESIGN.md 7) */
  int32_t encounter_order;            /* 1: rows are not ranked -- they come in the order the reference's traversal
                                         first meets them (the insertion order of its result dicts and lists), which
                                         is what Imputation.impute_one returns (impute.py:1940-1983); with hap_pop_pair
                                         the PMUG rows are then the un-merged accepted pairs.  General kernel only. */
} GrimbConfig;

/* A batch of subjects, tokenised by the host (replaces the string handling of
 * clean_up_gl / gl2haps, impute.py:105-118,246-272).  All pointers are DEVICE pointers for
 * grimb_impute_device and HOST pointers for grimb_impute_host. */
typedef struct {
  int64_t n_subjects;
  const uint16_t* typed_mask;   /* [S] bit l set = locus l typed; 0 = skip subject (GRIMB_ST_SKIPPED) */
  const uint16_t* counts;       /* [S][L][2] alleles listed per locus and chromosome side; >= 1 for
                                   every typed locus (an empty side is one unknown allele), 0 otherwise.
                                   NULL (ABI v4) = every typed locus side of every subject of this batch
                                   lists exactly one allele (saves 4L of the ~10L bytes per subject)  */
  const uint32_t* allele_off;   /* [S+1] offset of the subject's allele ids in `alleles`            */
  const uint16_t* alleles;      /* ids, per subject: locus ascending, side 0 then 1; ids > n_alleles[l]
                                   are subject-local names of alleles absent from the table        */
  int64_t n_alleles_total;      /* allele_off[S]                                                    */
  const uint32_t* prior_index;  /* [S] row of `priors`; NULL (ABI v4) = row 0 for every subject         */
  const double* priors;         /* [n_priors][P][P] prior matrices (impute.py:1844-1924,1956-1959)  */
  int32_t n_priors;
  const uint16_t* phase_mask;   /* optional [S] (NULL = none): bit m set = the m-th TYPED locus may switch
                                   sides when phases are enumerated (bin_imputation_in_file,
                                   impute.py:277-290,2001-2005,2030-2032)                              */
  /* ABI v4, PACKED form (optional; 64-bit-key build, L <= 5): for a batch in which every subject is typed
   * at every locus with exactly one allele per chromosome side -- or is to be skipped -- the subject is
   * 18 bytes: packed_keys[s] = {k0, k1}, its side-0 / side-1 alleles packed with the tables' key layout
   * (field of locus l at bit sum(key_bits[0..l)); subject-local ids of unknown alleles included), and
   * packed_flags[s]: bits 0..4 locus heterozygous (a0 != a1), bits 5..9 side-0 allele not a table allele,
   * bits 10..14 side-1 allele not a table allele, bit 15 skip the subject (GRIMB_ST_SKIPPED).  When
   * packed_keys is non-NULL, typed_mask / counts / allele_off / alleles / phase_mask are ignored (may be
   * NULL) and n_alleles_total is 0. */
  const uint64_t* packed_keys;  /* [S][2] or NULL                                                    */
  const uint16_t* packed_flags; /* [S]                                                               */
} GrimbBatch;

/* Result rows.  A hap row is two packed keys + probability: for UMUG the per-locus (min id,
 * max id) pair of the genotype (impute.py:497-504; the host orders each pair as strings), for
 * PMUG the two haplotypes in first-seen orientation (impute.py:28-38,651). */
#ifndef GRIMB_KEY_WORDS
#define GRIMB_KEY_WORDS 1   /* 1: libgrimb200.so (packed key <= 63 bits); 2: libgrimb200w.so (<= 127 bits) */
#endif
#if GRIMB_KEY_WORDS == 1
typedef struct { uint64_t a, b; double prob; } GrimbHapRow;
#else
typedef struct { uint64_t a[2], b[2]; double prob; } GrimbHapRow; /* little-endian words: [0] = low 64 bits */
#endif
typedef struct { uint16_t pop_a, pop_b; uint32_t pad; double prob; } GrimbPopRow;

/* Record of a GENERAL subject (48 bytes, 16-byte aligned: written with three 128-bit stores); its
 * rows are hap_rows[hap_off ...] / pop_rows[pop_off ...]. */
typedef struct {
  uint8_t status;        /* GRIMB_ST_*                                                   */
  uint8_t plan_umug;     /* GRIMB_PLAN_*                                                 */
  uint8_t plan_pmug;
  uint8_t reserved;
  uint32_t n_umug;       /* rows written (<= n_results)                                  */
  uint32_t n_pmug;
  uint32_t n_umug_pops;  /* rows written (<= n_pop_results)                              */
  uint32_t n_pmug_pops;
  uint32_t tot_umug;     /* len(res_muugs["Haps"]) before top-N (the count the reference prints) */
  uint32_t tot_pmug;     /* len(res_haps["Haps"])                                        */
  uint32_t pair_evals;   /* iterations reaching impute.py:464/573 (metric numerator; saturates) */
  uint64_t hap_off;      /* first UMUG row in hap_rows; the PMUG rows follow             */
  uint64_t pop_off;      /* first UMUG pop row in pop_rows; the PMUG pop rows follow     */
} GrimbSubjectResult;

/* ABI v4: ONE 16-byte record per subject, in input order.  Subjects that the warp-per-subject kernels
 * finish -- every locus typed, one allele per chromosome side, Plan A (the bulk of BASELINE configs 2, 3
 * and 5) -- are described completely by this record plus a few 8-byte words: their single UMUG genotype is
 * the subject's own allele pairs and the two haplotypes of a PMUG row follow from the subject's alleles and
 * the row's phase id (gen_phases, impute.py:274-303: bit m of the id = locus m takes its side-2 allele in
 * the first haplotype), so no packed keys travel back.  Everything else (ambiguity, missing loci, Plan B /
 * C, EM modes) keeps the 48-byte GrimbSubjectResult + row arrays above, appended to `general`.
 *   kind_flags: bits 0-1 GRIMB_KIND_*, bit 2 GRIMB_KIND_WORDS, bit 3 "has results" (else the reference
 *               writes .miss), bits 4-7 n_pmug = PMUG rows written (SIMPLE / TYPED: <= 4)
 *   GENERAL: off = index of the subject's GrimbSubjectResult in `general` (0xFFFFFFFF: none, skipped subject)
 *   SIMPLE : one population.  total = probability of the UMUG genotype = the population row's value;
 *            phases = phase ids of the PMUG rows in rank order, 4 bits each; with GRIMB_KIND_WORDS
 *            words[off + k] = probability of PMUG row k, without it (a single accepted phase) the one
 *            PMUG row's probability is `total`.  n_pmug == 15 marks the long form (more than four PMUG
 *            rows): words[off] = number of rows, words[off + 1] = their phase ids (4 bits each, rank order),
 *            words[off + 2 + k] = probability of row k
 *   TYPED  : P <= 32 populations.  words[off] = header: n_pops (bits 0-15), then the PMUG rows' phase ids,
 *            12 bits each from bit 16; words[off + 1 + k] = probability of PMUG row k; then n_pops
 *            probabilities of the population-pair rows in rank order (the same rows serve .umug.pops and
 *            .pmug.pops), then their pair codes, one uint16 each ((first-seen pop_a << 8) | pop_b), packed
 *            four per word. */
#define GRIMB_KIND_GENERAL 0
#define GRIMB_KIND_SIMPLE 1
#define GRIMB_KIND_TYPED 2
#define GRIMB_KIND_WORDS 4        /* SIMPLE: the PMUG probabilities are words[off ...] */
#define GRIMB_KIND_HAS_RESULTS 8
typedef struct {
  uint8_t status;        /* GRIMB_ST_*                                                   */
  uint8_t kind_flags;
  uint16_t phases;
  uint32_t off;
  double total;
} GrimbCompact;

typedef struct {
  GrimbCompact* compact;        /* [S]                                                   */
  uint64_t* words;        int64_t word_capacity;      /* rows of SIMPLE / TYPED subjects          */
  GrimbSubjectResult* general;  int64_t general_capacity;  /* records of GENERAL subjects, appended */
  GrimbHapRow* hap_rows;  int64_t hap_capacity;       /* rows of GENERAL subjects                 */
  GrimbPopRow* pop_rows;  int64_t pop_capacity;
  /* totals written by the call (host memory, always): entries needed; > capacity => GRIMB_E_CAPACITY.
   * [0] words, [1] general records, [2] hap rows, [3] pop rows, [4] pair evaluations of the whole batch
   * (iterations reaching impute.py:464/573, the metric's second numerator), [5] subjects the
   * warp-per-subject kernels handed on to the general kernel, [6] hash probes issued, [7] probes answered
   * with a node, [8] frequency vectors read by the probes' expansions (general and typed kernels; the
   * single-population fast path issues two probes per kept phase and is not instrumented).  9 entries. */
  int64_t* totals;
} GrimbResults;

int grimb_engine_create(const GrimbTables* t, int64_t workspace_bytes_per_cta, GrimbEngine** out);
int grimb_engine_free(GrimbEngine* e);

/* Device-pointer form: batch and result arrays already in HBM.  grimb_impute_device_async enqueues the
 * warp-per-subject kernels on `cuda_stream` (a cudaStream_t, 0 = engine stream) and returns without
 * synchronising; grimb_impute_finish waits for that call (an event: work of other engines queued behind it
 * on the same stream keeps running), launches the tail kernels (overflow list, cost classification,
 * cooperative slot pass, general kernel) only if some subject was handed on -- or if no warp-per-subject
 * kernel serves this table / mode -- and fills res->totals.  One call may be in flight per engine: a caller
 * that wants batch k+1 queued while batch k runs alternates between two engines.  The batch, result and
 * configuration structs are copied by the async call; the arrays they point at must stay valid until finish.
 * grimb_impute_device = the two together. */
int grimb_impute_device_async(GrimbEngine* e, const GrimbConfig* cfg, const GrimbBatch* batch,
                              const GrimbResults* res, void* cuda_stream);
int grimb_impute_finish(GrimbEngine* e, const GrimbResults* res);
int grimb_impute_device(GrimbEngine* e, const GrimbConfig* cfg, const GrimbBatch* batch,
                        GrimbResults* res, void* cuda_stream);

/* Host-pointer form: copies the batch in, runs, copies the results out (pinned staging owned
 * by the engine).  This is the call the Python drop-in makes per chunk of input lines. */
int grimb_impute_host(GrimbEngine* e, const GrimbConfig* cfg, const GrimbBatch* batch,
                      GrimbResults* res);

/* Number of kernel launches issued by this engine so far (bench.py's gpu_launches). */
int64_t grimb_engine_launches(const GrimbEngine* e);
/* Device time in ms (CUDA events on the launching stream) of the last launch of: which = 0 the
 * single-population probe kernel (k_fast_probe; k_impute_fast when GRIMB_FAST_SPLIT=0), 1 k_impute,
 * 2 k_impute_typed, 4 k_fast_score; negative if that kernel was not launched.  which = 3
 * (diagnostic): number of subjects the warp-per-subject kernels of the last call handed on to
 * k_impute.  which = 6 (diagnostic): the probe kernel of the engine's last split fast-path launch,
 * 2 the two-level k_fast_probe2 (packed batch), 1 k_fast_probe on a packed batch, 0 k_fast_probe on
 * the general batch form, -1 none yet.  which = 7: the last grimb_batch_from_genotypes (k_geno_encode, plus the
 * allele-offset scan and k_geno_fill when it built the general form); which = 8: the last grimb_results_rows
 * (k_rows_count, the row-offset scans and k_rows_fill; the host read-back between them is not counted); which = 9:
 * the last grimb_batch_from_genotype_lists (k_gl_count and the input-offset scan, then k_gl_dedup, the
 * allele-offset scan and k_gl_fill; the read-back between them is not counted). */
double grimb_engine_kernel_ms(const GrimbEngine* e, int which);

/* ------------------------------------------------------------------------------------------
 * Device-resident genotype interface: a genotype tensor in, ranked result rows out, both encoded and
 * decoded on the device, so a caller holding typed genotypes in HBM needs neither the text pipeline nor
 * the packed batch / GrimbCompact encodings.
 * ------------------------------------------------------------------------------------------ */

/* ids: DEVICE [n_subjects][L][2] allele ids in the tables' dictionary (id = position in the locus's sorted allele
 * list + 1; side 0 = the allele written before the '+'), 4-byte aligned; 0/0 = locus untyped; ids past the table
 * are subject-local names of alleles absent from it (n_l + 1, n_l + 2).  prior_index (DEVICE [S] or NULL) and
 * priors (DEVICE [n_priors][P][P]) pass through to the batch.  type_allowed: HOST [1 << L] or NULL, as in
 * GrimbTextDesc (Plan_A_Matrix).  A subject with one side of a locus 0, an id wider than its locus's key field,
 * no typed locus, or (type_allowed) a typed-locus pattern that is no matrix row is skipped (GRIMB_ST_SKIPPED, no
 * rows); the call does not fail for it.  *out gets a batch in buffers the engine owns (valid until the engine's
 * next call of this function): the PACKED form when the build has 64-bit keys, L <= 5 and every subject is fully
 * typed or skipped, else the general form (counts = NULL, allele_off by a device scan).  The call waits for one
 * 16-byte read-back (which form applies, and the allele total) on `cuda_stream` (0 = engine stream). */
int grimb_batch_from_genotypes(GrimbEngine* e, const uint16_t* ids, int64_t n_subjects, const uint32_t* prior_index,
                               const double* priors, int32_t n_priors, const uint8_t* type_allowed, GrimbBatch* out,
                               void* cuda_stream);

/* The same for subjects with allele ambiguity: ragged allele lists in, always the general batch form out.
 * counts: DEVICE [n_subjects][L][2], the number of ids listed on side x of locus l (0/0 = locus untyped);
 * alleles: DEVICE [n_alleles], the ids concatenated subject-major, locus ascending, side 0 then side 1, each list in
 * the order it was written (the layout of GrimbBatch.alleles); ids as in grimb_batch_from_genotypes.  phase_mask
 * (DEVICE [S] or NULL) passes through to GrimbBatch.phase_mask; prior_index, priors and type_allowed as above.
 * A repeated id inside one side's list is dropped, the first occurrence kept (as the text tokenisers do).  A
 * subject with exactly one side of a locus listing nothing, an id 0, an id wider than its locus's key field, no
 * typed locus, or (type_allowed) a typed-locus pattern that is no matrix row is skipped (GRIMB_ST_SKIPPED, no rows).
 * If the counts sum to anything but n_alleles the call returns GRIMB_E_ARG: it reads the counts first and checks
 * their sum (one read-back) before any kernel reads `alleles`.  *out gets the general form with de-duplicated
 * counts (non-NULL), allele_off and compacted alleles, in buffers the engine owns (valid until the engine's next
 * call of this function); subjects with one allele per side at every locus still take the warp-per-subject kernels
 * when no phase mask and no hap_pop_pair apply.  The call waits for two small read-backs on `cuda_stream`
 * (0 = engine stream): the input total, then the de-duplicated total (n_alleles_total). */
int grimb_batch_from_genotype_lists(GrimbEngine* e, const uint16_t* counts, const uint16_t* alleles, int64_t n_alleles,
                                    int64_t n_subjects, const uint32_t* prior_index, const double* priors, int32_t n_priors,
                                    const uint16_t* phase_mask, const uint8_t* type_allowed, GrimbBatch* out,
                                    void* cuda_stream);

/* Result rows of a finished device call (grimb_impute_device, or _async + finish), decoded on the device.  Every
 * pointer is a DEVICE pointer except `totals`.  Per subject [S]: status, plans and the counts the reference prints
 * (tot_umug, tot_pmug), flags (GRIMB_ROWS_*).  Four row kinds, each with its own offsets off[k] [S+1] and rows in
 * rank order; a subject has rows only with status GRIMB_ST_OK, and only for the outputs the configuration enables:
 *   GRIMB_ROWS_UMUG      rows[0] [n][L][2] per-locus allele pairs (min id, max id), 0/0 at an untyped locus
 *   GRIMB_ROWS_PMUG      rows[1] [n][2][L] haplotype 1 then haplotype 2 in first-seen orientation, 0 = no allele
 *   GRIMB_ROWS_UMUG_POPS rows[2] [n][2] population indices (0xFFFF = all_pops) as the kernels recorded them (the
 *   GRIMB_ROWS_PMUG_POPS rows[3] [n][2]  .umug.pops text sorts the two names; these rows do not)
 * prob[k] [n]: probabilities, copied bit for bit.  Table alleles keep their dictionary ids (id order = the
 * reference's string order); an unknown allele keeps its subject-local id.  totals (HOST [4]) get the rows needed
 * per kind; if one exceeds capacity[k] the call returns GRIMB_E_CAPACITY and writes no rows.  Under
 * cfg->hap_pop_pair, pmug_pairs [capacity[GRIMB_ROWS_PMUG]][2] gets the populations of haplotype 1 and haplotype 2
 * of each PMUG row (its companion pop row, see GrimbConfig.hap_pop_pair); it is then required
 * (NULL: GRIMB_E_ARG) and ignored otherwise. */
#define GRIMB_ROWS_UMUG 0
#define GRIMB_ROWS_PMUG 1
#define GRIMB_ROWS_UMUG_POPS 2
#define GRIMB_ROWS_PMUG_POPS 3
#define GRIMB_ROWS_HAS_RESULTS 1  /* flags bit 0: the subject has result rows                          */
#define GRIMB_ROWS_MISS 2         /* flags bit 1: the reference writes the subject to .miss (OK status, haplotype
                                     output on, no UMUG and no PMUG row; nothing when the haplotype output is off) */
#define GRIMB_ROWS_PROBLEM 4      /* flags bit 2: .problem: SKIPPED, FAULT, or NO_PHASES with the haplotype output on */
typedef struct {
  uint8_t* status;              /* [S] GRIMB_ST_*                                                     */
  uint8_t* plan_umug;           /* [S] GRIMB_PLAN_*                                                   */
  uint8_t* plan_pmug;           /* [S]                                                                */
  uint8_t* flags;               /* [S] GRIMB_ROWS_HAS_RESULTS | GRIMB_ROWS_MISS | GRIMB_ROWS_PROBLEM   */
  uint32_t* tot_umug;           /* [S]                                                                */
  uint32_t* tot_pmug;           /* [S]                                                                */
  int64_t* off[4];              /* [S+1] per row kind                                                 */
  uint16_t* rows[4];            /* per row kind, see above                                            */
  double* prob[4];              /* [capacity[k]]                                                      */
  int64_t capacity[4];          /* rows each kind's arrays hold                                       */
  int64_t* totals;              /* HOST [4]: rows needed per kind                                     */
  uint16_t* pmug_pairs;         /* [capacity[GRIMB_ROWS_PMUG]][2] under hap_pop_pair, else unused     */
} GrimbRows;

/* cfg: the configuration of the call that produced `res`; batch: its batch (SIMPLE / TYPED rows take the
 * subject's own alleles from it), any form; res: its GrimbResults (device arrays).  Synchronous on `cuda_stream`
 * (0 = engine stream) for the 32-byte read-back of the totals. */
int grimb_results_rows(GrimbEngine* e, const GrimbConfig* cfg, const GrimbBatch* batch, const GrimbResults* res,
                       const GrimbRows* rows, void* cuda_stream);

/* ------------------------------------------------------------------------------------------
 * Text pipeline (host C++, multi-threaded): the steps either side of the kernels.  Replaces the
 * per-line work of Imputation.impute_file (impute.py:2019-2144): line split, clean_up_gl /
 * gl2haps tokenising (:105-118,246-272), the race -> prior matrix step (:1956-1975,1844-1924),
 * the .miss / .problem classification (:2061-2068,2141-2144) and the row text of
 * write_best_prob / write_best_prob_genotype (:24-76) with Python's str(float) layout.
 * ------------------------------------------------------------------------------------------ */
typedef struct GrimbText GrimbText;

typedef struct {
  int32_t n_loci, n_pops;
  const char* const* locus_names;    /* [L] in loci_map index order                               */
  const char* const* allele_names;   /* table alleles, locus 0 first; id = position in its locus + 1 */
  const int32_t* allele_counts;      /* [L]                                                       */
  const char* const* pop_names;      /* [P] "populations"                                         */
  const double* count_by_prob;       /* [P] column 3 of pops_count_file, or ones (impute.py:205-212) */
  double alpha, eta, beta, gamma, delta; /* "priority"                                            */
  int32_t unk_priors_mr;             /* "UNK_priors" == "MR" (ones) else identity                 */
  int32_t key_bits[GRIMB_MAX_LOCI];  /* the tables' packed-key layout                             */
  int32_t n_threads;                 /* 0 = hardware concurrency                                  */
  const uint8_t* type_allowed;       /* "Plan_A_Matrix": [1 << L], non-zero where the typed-locus pattern (bit l =
                                        locus l typed) is a matrix row -- other subjects go to .problem
                                        (impute.py:1592-1596); NULL = no matrix                                  */
} GrimbTextDesc;

/* the six output texts of one call; pointers stay valid until the next call on the same GrimbText */
#define GRIMB_OUT_UMUG 0
#define GRIMB_OUT_UMUG_POPS 1
#define GRIMB_OUT_PMUG 2
#define GRIMB_OUT_PMUG_POPS 3
#define GRIMB_OUT_MISS 4
#define GRIMB_OUT_PROBLEM 5
typedef struct {
  const char* data[6];
  int64_t size[6];
  int64_t n_lines, pair_evals, workspace_retries;
  int64_t plan_count[4];
  double seconds_tokenise, seconds_gpu, seconds_format;
} GrimbTextOut;

int grimb_text_create(const GrimbTextDesc* d, GrimbText** out);
int grimb_text_free(GrimbText* t);

/* Two host-only halves (no CUDA calls; also what the CPU tests drive):
 *   tokenise: input lines -> a GrimbBatch (host arrays owned by `t`) + per-line bookkeeping
 *   format  : GrimbResults for that batch -> the six texts                                   */
int grimb_text_tokenise(GrimbText* t, const GrimbConfig* cfg, const char* text, int64_t len,
                        int64_t first_line_index, GrimbBatch* batch_out);
int grimb_text_format(GrimbText* t, const GrimbConfig* cfg, const GrimbResults* res, GrimbTextOut* out);

/* tokenise -> grimb_impute_host (subjects that overflow a workspace tier are re-issued on the
 * next engine of `engines`) -> format.  This is what grim.grim.impute() calls per chunk of the
 * input file. */
int grimb_impute_text(GrimbText* t, GrimbEngine* const* engines, int32_t n_engines, const GrimbConfig* cfg,
                      const char* text, int64_t len, int64_t first_line_index, GrimbTextOut* out);

/* ------------------------------------------------------------------------------------------
 * File pipeline.  Replaces Imputation.impute_file (impute.py:1985-2155) for a whole input file (or
 * the byte range [byte_lo, byte_hi) of it: the lines that START in the range; byte_hi < 0 = to the
 * end): the input is memory-mapped and cut into chunks of about chunk_bytes (0 = default) at line
 * boundaries, and four host threads overlap tokenise(c+1) | GPU(c) | format(c-1) | write(c-2).
 * out_paths[k] (GRIMB_OUT_* order) non-NULL: that output is streamed to the file (created /
 * truncated); NULL (or out_paths == NULL): it is kept in memory and returned through `out` (valid
 * until the next call on the same GrimbText) -- what a multi-process caller needs to place its
 * rows at an offset of a shared file with grimb_file_write_at.  first_line_index: number of the
 * first line of the range in the whole input (.miss / .problem rows carry line numbers).
 * grimb_file_count_lines: lines starting in the byte range (multi-threaded) and the range adjusted
 * to line boundaries.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int64_t n_lines, n_chunks, in_bytes, pair_evals, workspace_retries;
  int64_t plan_count[4];
  int64_t out_bytes[6];
  double seconds_total;                 /* wall clock of the call                              */
  double seconds_tokenise, seconds_gpu, seconds_format, seconds_write;   /* busy time per stage */
} GrimbFileStats;

int grimb_impute_file(GrimbText* t, GrimbEngine* const* engines, int32_t n_engines, const GrimbConfig* cfg,
                      const char* in_path, int64_t byte_lo, int64_t byte_hi, int64_t first_line_index,
                      const char* const* out_paths, int64_t chunk_bytes, GrimbTextOut* out, GrimbFileStats* stats);
int grimb_file_count_lines(const char* path, int64_t byte_lo, int64_t byte_hi, int32_t n_threads,
                           int64_t* n_lines, int64_t* lo_adj, int64_t* hi_adj);
int grimb_file_write_at(const char* path, int64_t offset, const void* data, int64_t size);

/* One input file shared by the ranks of a host (one process per GPU).  The ranks take the input's chunks
 * round-robin (chunk c -> rank c % world) and stream their rows straight into the SAME six final files: a board
 * in a small memory-mapped file carries every chunk's line count (for the global line indices of the .miss /
 * .problem rows) and the sizes of its six output pieces (for the file offsets), so nothing is accumulated in
 * memory, gathered between the ranks or written after the computation.  Rank 0 creates the six output files
 * (empty) and the board file (grimb_file_board_bytes() zero bytes) before any rank calls; all ranks pass the same
 * chunk_bytes.  A rank that fails marks the board and the others return an error instead of waiting. */
int64_t grimb_file_board_bytes(int64_t file_bytes, int64_t chunk_bytes);
int grimb_impute_file_sharded(GrimbText* t, GrimbEngine* const* engines, int32_t n_engines, const GrimbConfig* cfg,
                              const char* in_path, const char* const* out_paths, int64_t chunk_bytes, int32_t rank,
                              int32_t world, const char* board_path, GrimbFileStats* stats);

#ifdef __cplusplus
}
#endif
#endif /* GRIMB200_H */
