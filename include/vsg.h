/* include/vsg.h — C ABI of libvsg.so, the B200-native (sm_100a CUDA) implementation of the
 * vsearch hot path: the 16-bit affine-gap global aligner `search16` and the k-mer candidate
 * ranker `search_topscores`, batched over many queries.
 *
 * Plain pointers and sizes only; no C++ or torch types cross this boundary.  Every entry point
 * names the reference interface it replaces (reference = torognes/vsearch v2.31.0, paths relative
 * to its src/).  Errors: functions return 0 on success or a negative VSG_E* code and leave a
 * message retrievable with vsg_last_error(); nothing throws (the reference is built
 * -fno-exceptions, Makefile.am:53) and nothing falls back to a CPU path: without a CUDA device
 * vsg_ctx_create fails with VSG_ENODEVICE.
 *
 * In-band "cannot align this pair" is signalled exactly as the reference does it: score ==
 * VSG_SCORE_SENTINEL (SHRT_MAX), zero statistics, empty CIGAR (core/align_simd.cpp:1463-1479,
 * 1838-1846, 1871-1881); the caller re-aligns such pairs with its linear-memory aligner
 * (core/searchcore.cpp:806-832).
 */
#ifndef VSG_H
#define VSG_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VSG_OK 0
#define VSG_ENODEVICE (-1) /* no CUDA device / driver */
#define VSG_ECUDA (-2)     /* a CUDA call failed */
#define VSG_EINVAL (-3)    /* bad argument */
#define VSG_ENOMEM (-4)    /* host or device allocation failed */
#define VSG_ECAP (-5)      /* caller-provided output buffer too small */

#define VSG_SCORE_SENTINEL 32767

typedef struct vsg_ctx vsg_ctx;       /* one per host thread; owns a CUDA stream + scratch  */
typedef struct vsg_seqset vsg_seqset; /* a set of sequences resident in HBM                 */
typedef struct vsg_index vsg_index;   /* k-mer postings index resident in HBM               */

/* Scores/penalties in search16_init's own argument order (core/align_simd.hpp:76-91):
 * v[0]=match v[1]=mismatch, v[2..7]=gap open {query_left,target_left,query_interior,
 * target_interior,query_right,target_right}, v[8..13]=gap extension in the same order.
 * "open" excludes the first extension, i.e. the values vsearch_apply_defaults_fixups leaves
 * in Parameters (vsearch.cc:250-259). */
typedef struct vsg_scoring {
  int64_t v[14];
  int32_t n_mismatch; /* opt_n_mismatch */
} vsg_scoring;

const char * vsg_last_error(void);
const char * vsg_version(void);
/* number of kernels this library has launched in the calling process (bench "gpu_launches") */
int64_t vsg_launch_count(void);

/* ---- context: replaces search16_init / search16_exit (core/align_simd.cpp:1282-1403) ---- */
int vsg_ctx_create(int device, const vsg_scoring * scoring, vsg_ctx ** out);
void vsg_ctx_destroy(vsg_ctx * ctx);
/* the CUDA stream (cudaStream_t) all work of this context is enqueued on */
void * vsg_ctx_stream(vsg_ctx * ctx);
int vsg_ctx_sync(vsg_ctx * ctx);

/* ---- pairs the 16-bit aligner cannot take (score == VSG_SCORE_SENTINEL): the reference re-aligns
 *      them with its scalar LinearMemoryAligner (core/searchcore.cpp:806-832,
 *      commands/allpairs_global.cpp:447-473).  That routine stays on the host side of the boundary:
 *      the embedding application registers it here and vsg_search_batch / vsg_allpairs call it for
 *      exactly those pairs.  query/target are indices into the sequence sets of the call, strand is
 *      1 when the query is to be reverse-complemented.  out[10] = {nwscore, alignment length,
 *      matches, mismatches, gaps, trim_q_left, trim_t_left, trim_q_right, trim_t_right, forbidden}
 *      (trims as in vsg_align_pairs).  `forbidden` (preset to 0) is the application's verdict of
 *      alignment_uses_forbidden_gap (core/searchcore.cpp:612-660): non-zero iff the alignment uses a
 *      gap class whose penalty was given as '*'; such a hit is rejected exactly as
 *      search_acceptable_aligned does (:677-680).  '*' penalties reach the library as values that do
 *      not fit a 16-bit cell, which defers every pair to this callback (align_simd.cpp:1463-1479).
 *      Return 0 on success.  Called from the library's worker threads, possibly
 *      concurrently.  Without a callback such a pair makes the call fail with VSG_EINVAL. ---- */
typedef int (*vsg_fallback_fn)(void * user, int64_t query, int32_t strand, int64_t target, int64_t * out);
int vsg_ctx_set_fallback(vsg_ctx * ctx, vsg_fallback_fn fn, void * user);

/* ---- sequences: replaces Database::add / getsequence / getsequencelen
 *      (core/db.hpp:137-201, core/db.cpp:170-226).  ASCII, one byte per nucleotide, any case,
 *      IUPAC allowed; offsets index into `cat`. `host` selects where cat/off/len live
 *      (1 = host memory; 0 = device memory of ctx's device, e.g. after an NCCL broadcast).  Either way the
 *      data is COPIED (encoded into the library's own symbol buffer): the caller may free its arrays when
 *      the call returns.  A seqset / index belongs to the device of the context that made it; passing it to
 *      a context of another device is an error (VSG_EINVAL). ---- */
int vsg_seqset_create(vsg_ctx * ctx, const char * cat, const int64_t * off, const int32_t * len,
                      int64_t n, int host, vsg_seqset ** out);
void vsg_seqset_destroy(vsg_seqset * s);
int64_t vsg_seqset_count(const vsg_seqset * s);
/* DUST soft-masking in place on the device: replaces dust() / dust_all() (core/mask.cpp:79-188;
 * default --qmask dust / --dbmask dust).  Afterwards lower case marks exactly the regions the
 * reference would have masked; pass mask_lower = 1 to vsg_index_create / vsg_rank / vsg_search_batch. */
int vsg_seqset_dust(vsg_ctx * ctx, vsg_seqset * s);
/* the symbol bytes as stored in HBM (bits 0-3 = 4-bit nucleotide code, bit 4 = lower case), in the
 * order and at the offsets given to vsg_seqset_create; cap >= total sequence bytes.  For tools/tests. */
int vsg_seqset_symbols(vsg_ctx * ctx, const vsg_seqset * s, uint8_t * out, int64_t cap);
/* the reverse complements of sequences [q0, q0 + n) of `src` as a new set of n sequences (entry i = the reverse
 * complement of sequence q0 + i): replaces reverse_complement (utils/reverse_complement.cpp:71-84).  Case, and so
 * the soft mask, is kept; non-IUPAC symbols become 'N'.  E.g. the CIGAR of a strand-1 clustering record is
 * vsg_align_pairs(revcomp set, set) of that sequence against its centroid.  Free with vsg_seqset_destroy. */
int vsg_seqset_revcomp(vsg_ctx * ctx, const vsg_seqset * src, int64_t q0, int64_t n, vsg_seqset ** out);

/* ---- batched alignment: replaces search16_qprep + search16 (core/align_simd.cpp:1406-2060)
 *      for npairs (query,target) pairs at once.  qidx[i] indexes `queries`, tidx[i] indexes
 *      `targets`.  Outputs are caller-allocated arrays of npairs elements, identical in meaning
 *      to search16's pscores/paligned/pmatches/pmismatches/pgaps.
 *      trims (optional, may be NULL): 4 x int32 per pair {trim_q_left, trim_t_left, trim_q_right,
 *      trim_t_right} = run length of a leading / trailing D resp. I CIGAR op, before the
 *      "covers the whole alignment" fix-up of align_trim (core/searchcore.cpp:357-417).
 *      CIGARs (optional): if cigar_buf != NULL the NUL-terminated CIGAR of pair i is written at
 *      cigar_buf + cigar_off[i] (cigar_off is an OUTPUT, npairs+1 entries, dense); cigar_cap is
 *      the buffer size; VSG_ECAP if it does not fit (a capacity of sum(qlen+dlen+1) always fits).
 *      All pointers are HOST pointers; the sequences themselves are already resident in HBM
 *      (vsg_seqset_create), only the pair list goes up and the fixed-size results come back. ---- */
int vsg_align_pairs(vsg_ctx * ctx, const vsg_seqset * queries, const vsg_seqset * targets,
                    int64_t npairs, const uint32_t * qidx, const uint32_t * tidx,
                    int16_t * score, uint16_t * aligned, uint16_t * matches,
                    uint16_t * mismatches, uint16_t * gaps, int32_t * trims,
                    char * cigar_buf, int64_t cigar_cap, int64_t * cigar_off);

/* Layout of the per-pair statistics record the kernels produce (8 x int32, device side);
 * exposed so that tools reading the raw buffers agree on it. */
#define VSG_STAT_SCORE 0
#define VSG_STAT_ALIGNED 1
#define VSG_STAT_MATCHES 2
#define VSG_STAT_MISMATCHES 3
#define VSG_STAT_GAPS 4
#define VSG_STAT_TRIM_LEFT 5  /* +run: leading D (gap in target) ; -run: leading I ; 0: leading M */
#define VSG_STAT_TRIM_RIGHT 6 /* same for the trailing op */
#define VSG_STAT_CIGARLEN 7   /* strlen of the CIGAR */
#define VSG_STAT_WORDS 8

/* Cumulative device-side profile of this context since the last vsg_profile_reset: DP cells
 * (sum qlen*dlen of the pairs that went through a forward kernel), forward / traceback / ranker
 * kernel time (cudaEvents on the context's stream, ms), pair counts per kernel and the number of
 * forward launches.  bench.py computes its roofline from these. */
typedef struct vsg_profile {
  int64_t cells;
  int64_t fast_pairs;
  int64_t exact_pairs;
  int64_t fwd_launches;
  float fwd_ms;
  float traceback_ms;
  float rank_ms;
  float reserved;
  int64_t tb_skipped;   /* pairs whose walk back was skipped by traceback on demand (vsg_search_batch; their DP was computed) */
} vsg_profile;
int vsg_profile_reset(vsg_ctx * ctx);
int vsg_profile_get(vsg_ctx * ctx, vsg_profile * out);
/* Measured integer issue peak of this device: thread-instructions per second of an even mix of packed 16x2 DPX
 * (ALU pipe) and 32-bit multiply-add (FMA pipe) instructions with no memory traffic — each processes the two
 * packed cells of a register, so 2 x this / (instructions per cell pair) is the DP roofline's denominator. */
int vsg_measure_int_peak(vsg_ctx * ctx, double * packed_lane_ops_per_s);

/* ---- k-mer index: replaces Dbindex::prepare + add_all_sequences + the getters
 *      (core/dbindex.hpp:79-120, core/dbindex.cpp:121-255).  mask_lower != 0 means soft-masked
 *      (lower-case) symbols do not seed k-mers (unique.cpp:198-199). ---- */
int vsg_index_create(vsg_ctx * ctx, const vsg_seqset * db, int wordlength, int mask_lower,
                     vsg_index ** out);
void vsg_index_destroy(vsg_index * ix);
/* wordlength 3..15, as the reference (cli.cc --wordlength).  3..10: list heads for all 4^k words per shard of 32 766
 * targets, targets de-duplicated through a bitmap (unique_count_bitmap, core/unique.cpp:155-240).  11..15: only the
 * words that occur get a list, found by sorting (what unique_count_hash's table finds, core/unique.cpp:243-334),
 * looked up by binary search. */

/* ---- candidate ranking: replaces unique_count + search_topscores + minheap
 *      (core/unique.cpp:337-353, core/searchcore.cpp:260-340, core/minheap.cpp) for every query
 *      of `queries` in [q0, q0+nq).  For query q the best-first list (count desc, target length
 *      asc, target number asc) of at most tophits targets with count >= min(minwordmatches,
 *      number of distinct query k-mers) is written to cand_seqno/cand_count[(q-q0)*tophits ...],
 *      its length to ncand[q-q0].  Host pointers.  Any tophits >= 1: up to 1 024 one ranking pass with
 *      the list in shared memory; beyond, two counting passes and a segmented sort (any list length,
 *      up to the whole database). ---- */
int vsg_rank(vsg_ctx * ctx, const vsg_index * ix, const vsg_seqset * queries, int64_t q0,
             int64_t nq, int minwordmatches, int tophits, int mask_lower,
             uint32_t * cand_seqno, uint32_t * cand_count, int32_t * ncand);

/* ---- whole-path search: replaces search_batch (core/search.hpp:135-145, search.cpp:511-593) /
 *      the body of search_thread_run (commands/usearch_global.cpp:376-497) for plus-strand (and
 *      optionally minus-strand) queries with the reference's default pre-alignment filters.
 *      result layout mirrors search_result_s (core/search.hpp:67-80). ---- */
typedef struct vsg_search_opts {
  double id;              /* --id                         */
  double weak_id;         /* --weak_id (10.0 = default)   */
  int32_t maxaccepts;     /* --maxaccepts (default 1)     */
  int32_t maxrejects;     /* --maxrejects (default 32)    */
  int32_t wordlength;     /* --wordlength (default 8)     */
  int32_t minwordmatches; /* <0: reference default table  */
  int32_t iddef;          /* --iddef (default 2)          */
  int32_t strand_both;    /* --strand both                */
  int32_t mask_lower;     /* queries are soft-masked      */
  int32_t lazy;           /* 0 (default): align exactly the groups of <= 8 candidates the reference
                             hands to search16; 1: align a candidate only when the replay is about to
                             examine it (same decisions and hit tables, fewer DP cells)           */
  /* optional accept/reject filters, reference defaults from vsg_search_opts_default():
     before alignment (search_acceptable_unaligned, core/searchcore.cpp:573-587) */
  double minqt, maxqt;    /* --minqt / --maxqt : query/target length ratio          */
  double minsl, maxsl;    /* --minsl / --maxsl : shorter/longer length ratio        */
  /* after alignment (search_acceptable_aligned, core/searchcore.cpp:671-699) */
  double maxid;           /* --maxid  (1.0)                */
  double mid;             /* --mid    (0.0)                */
  double query_cov;       /* --query_cov (0.0)             */
  double target_cov;      /* --target_cov (0.0)            */
  int64_t maxsubs;        /* --maxsubs  (INT_MAX)          */
  int64_t maxgaps;        /* --maxgaps  (INT_MAX)          */
  int64_t mincols;        /* --mincols  (0)                */
  int64_t maxdiffs;       /* --maxdiffs (INT_MAX)          */
  int32_t leftjust;       /* --leftjust                    */
  int32_t rightjust;      /* --rightjust                   */
  /* the remaining pre-alignment filters of search_acceptable_unaligned (core/searchcore.cpp:561-608);
     vsg_search_batch only (vsg_allpairs ignores them, as allpairs_global's defaults do) */
  int64_t maxqsize;       /* --maxqsize (INT64_MAX): query abundance <= maxqsize           */
  int64_t mintsize;       /* --mintsize (0):         target abundance >= mintsize          */
  double minsizeratio;    /* --minsizeratio (0.0):   query abundance >= ratio * target's   */
  double maxsizeratio;    /* --maxsizeratio (DBL_MAX)                                      */
  int32_t idprefix;       /* --idprefix (0): first n nucleotides identical (compared on the device) */
  int32_t idsuffix;       /* --idsuffix (0): last n nucleotides identical                   */
  int32_t self;           /* --self:   reject a target whose label equals the query's      */
  int32_t selfid;         /* --selfid: reject a target whose sequence equals the query's   */
  int32_t qmask_dust;     /* --qmask dust with --strand both: the caller has DUST-masked `queries`
                             (vsg_seqset_dust); the reverse complements made inside the call are masked
                             on their own, as search_batch_worker_fn does per strand (core/search.cpp:437-449) */
  int32_t unoise;         /* --cluster_unoise acceptance (searchcore.cpp:700-717): a hit that passes the filters is accepted
                             iff it has no mismatch or query abundance / target abundance <= 1 / 2^(unoise_alpha * mismatches + 1),
                             instead of the --id test; needs query_sizes / target_sizes */
  const int64_t * query_sizes;   /* abundance of query q0+i at [i]; NULL = 1 everywhere (db.getabundance / qsize) */
  const int64_t * target_sizes;  /* abundance of target t at [t];   NULL = 1 everywhere                     */
  const int64_t * query_labels;  /* --self: label identities, [i] for query q0+i resp. [t] for target t; two  */
  const int64_t * target_labels; /*         sequences carry the same header iff their identities are equal  */
  double unoise_alpha;    /* --unoise_alpha (2.0) */
  int32_t sizeorder;      /* --sizeorder (vsg_cluster_fast / sessions, with maxaccepts > 1): among the accepted hits the centroid of
                             highest abundance wins, then identity, then the earlier one (search_findbest2_bysize,
                             searchcore.cpp:182-240, 994-1025) instead of identity first; needs target_sizes */
  int32_t reserved1;
} vsg_search_opts;

typedef struct vsg_search_result {
  int32_t target;
  int32_t matches;
  int32_t mismatches;
  int32_t gaps;
  int32_t alignment_length;
  int32_t query_length;
  int32_t target_length;
  int32_t accepted;
  int32_t strand;
  int32_t nwscore;
  double id;
  int32_t internal_alignment_length;   /* alignment columns / gap opens without the terminal gaps that align_trim   */
  int32_t internal_gaps;               /* removes (core/searchcore.cpp:409-463): the --blast6out columns 4 and 6     */
} vsg_search_result;

void vsg_search_opts_default(vsg_search_opts * o);
/* results[(q)*max_results + j], counts[q]; work (optional, 4 x int64): {pairs, DP cells} the
 * reference's driver hands to search16 for the same queries, then {pairs, DP cells} actually
 * aligned here (identical unless opts->lazy).  Any maxaccepts / maxrejects (0 = all, as the command
 * line clamps them to the database size): candidate lists longer than 1 024 are ranked in two passes
 * and searched in pieces of bounded candidate volume. */
int vsg_search_batch(vsg_ctx * ctx, const vsg_index * ix, const vsg_seqset * db,
                     const vsg_seqset * queries, int64_t q0, int64_t nq,
                     const vsg_search_opts * opts, vsg_search_result * results, int max_results,
                     int32_t * counts, int64_t * work);

/* ---- all-against-all: replaces the per-query body of allpairs_thread_run
 *      (commands/allpairs_global.cpp:340-549) for query rows [row0, row0+nrows) of `set`: every
 *      target j > i is aligned (no k-mer filter, default pre-alignment filters), a pair is kept iff
 *      search_acceptable_aligned accepts it (id >= opts->id under opts->iddef), kept pairs of a
 *      query are ordered by (id desc, target asc) as allpairs_hit_compare does, queries ascending.
 *      hits: caller-allocated, `cap` records; *nhits receives the number produced (VSG_ECAP if it
 *      exceeds cap).  Rows are independent, so N GPUs take disjoint row ranges (SURVEY.md §8e).
 *      work (optional, 2 x int64): pairs and DP cells aligned. ---- */
typedef struct vsg_pair_hit {
  int32_t query;
  int32_t target;
  int32_t matches;
  int32_t mismatches;
  int32_t gaps;
  int32_t alignment_length;
  int32_t nwscore;
  int32_t internal_alignment_length;
  double id;
} vsg_pair_hit;
/* Row ranges of equal DP work for `nparts` workers (GPUs): bounds[p] .. bounds[p+1] are the rows of
 * part p, chosen so that every part has about the same sum over its rows i of len[i] * (sum of len[j],
 * j > i) — the triangle balancing SURVEY.md §8(e) asks for; equal row counts would give the first
 * GPU almost twice the work of the average.  Pure host arithmetic; bounds has nparts+1 entries. */
int vsg_allpairs_partition(const int32_t * len, int64_t n, int nparts, int64_t * bounds);
int vsg_allpairs(vsg_ctx * ctx, const vsg_seqset * set, int64_t row0, int64_t nrows,
                 const vsg_search_opts * opts, vsg_pair_hit * hits, int64_t cap, int64_t * nhits,
                 int64_t * work);

/* ---- greedy centroid clustering: replaces cluster_core_parallel / cluster_core_serial with cluster_query_core,
 *      evaluate_extra_hits and Dbindex::add_sequence (core/cluster.cpp:162-189, 601-856, 877-1115;
 *      core/dbindex.cpp:121-148) for --cluster_fast-style clustering of `set` IN THE ORDER GIVEN (the reference
 *      sorts by decreasing length first, core/db.cpp:433-449; mask the set with vsg_seqset_dust and pass
 *      opts->mask_lower = 1 for the default --qmask dust).  round_size = the reference's --threads: sequences are
 *      searched in rounds of that many against the centroids found so far and then resolved one by one, centroids
 *      of the same round included (cluster.cpp:881-882, 946-1025) — the assignments depend on it, so compare
 *      with `vsearch --cluster_fast --threads round_size`.  results[i] for sequence i: its cluster number
 *      (creation order of the centroids) and either centroid = -1 (it founded the cluster: an "S" record of
 *      --uc) or the sequence number of the centroid it matched plus that alignment's statistics and identity
 *      (an "H" record; the CIGAR is one vsg_align_pairs call away).  NOTE the reference's default --maxrejects for
 *      --cluster_fast is 8, not 32 (cli.cc:4163-4172): set opts->maxrejects accordingly.  opts: id, iddef, maxaccepts, maxrejects,
 *      wordlength, minwordmatches, mask_lower, strand_both, the length / abundance / post-alignment filters
 *      (target_sizes and target_labels are per sequence of `set`).  work (optional, 2 x int64): pairs and DP cells
 *      handed to the aligner, both strands counted.
 *      strand_both (--strand both, cluster.cpp:162-189, 946-1025): each sequence is also searched as the reverse
 *      complement of the sequence AS STORED, so its soft mask is mirrored and not computed again (unlike
 *      vsg_search_batch with qmask_dust, which masks each strand on its own).  Each strand has its own candidate
 *      list, counters and hit list; the best hit is taken over the plus hits, then the minus hits, ties going to plus.
 *      results[i].strand = 1 when the sequence matched its centroid as the reverse complement: identity and
 *      statistics are those of the reverse complement aligned to the centroid, and so is the CIGAR
 *      (vsg_seqset_revcomp, then vsg_align_pairs).  New centroids are always indexed as stored (strand 0).  A
 *      deferred pair reaches the fallback callback with the sequence's number in `set` and its strand.  The set is
 *      mirrored once at setup into a device copy holding every sequence and its reverse complement (twice the
 *      set's symbol bytes). ---- */
typedef struct vsg_cluster_result {
  int32_t cluster;
  int32_t centroid;
  int32_t matches;
  int32_t mismatches;
  int32_t gaps;
  int32_t alignment_length;
  int32_t nwscore;
  int32_t strand;
  double id;
} vsg_cluster_result;
int vsg_cluster_fast(vsg_ctx * ctx, const vsg_seqset * set, const vsg_search_opts * opts, int round_size,
                     vsg_cluster_result * results, int64_t * nclusters, int64_t * work);

/* ---- the same clustering as a SESSION that is fed ranges of the set: replaces cluster_session_init /
 *      cluster_assign_single / cluster_assign_batch / cluster_session_cleanup (core/cluster.hpp:78-118,
 *      core/cluster.cpp:1633-1930).  The session owns the device index of the centroids found so far and the cluster
 *      numbers; `set` (already masked and sorted, as for vsg_cluster_fast), the context and the arrays `opts` points
 *      to must outlive it.  vsg_cluster_session_assign handles the sequences [start, start + count) in rounds of
 *      round_size (cluster_assign_batch: the caller's --threads; cluster_assign_single: count = round_size = 1);
 *      ranges must be ascending and contiguous (cluster.hpp:104-111), results[i] belongs to sequence start + i.
 *      A session fed the whole set in one call gives vsg_cluster_fast's results.  The set's contents must not change
 *      after vsg_cluster_session_create (no vsg_seqset_dust in between): with strand_both the session reads its
 *      queries, both strands, from the mirror it copied at create. ---- */
typedef struct vsg_cluster_session vsg_cluster_session;
int vsg_cluster_session_create(vsg_ctx * ctx, const vsg_seqset * set, const vsg_search_opts * opts, vsg_cluster_session ** out);
int vsg_cluster_session_assign(vsg_cluster_session * session, int64_t start, int64_t count, int round_size,
                               vsg_cluster_result * results);
int64_t vsg_cluster_session_clusters(const vsg_cluster_session * session);
void vsg_cluster_session_destroy(vsg_cluster_session * session);

/* ---- several GPUs behind one process (SURVEY.md §8e; the reference is a single process, LIBRARY_API.md:138-156):
 *      vsg_group_create uploads the database ONCE (to devices[0]; dust_db != 0 also DUST-masks it there,
 *      core/mask.cpp dust_all), copies the packed sequences device to device over NVLink to every other GPU and
 *      builds the k-mer index on each.  vsg_group_search shards the queries (host arrays, as for
 *      vsg_seqset_create) into contiguous ranges of equal nucleotide count, one per device, and runs
 *      vsg_search_batch on all devices concurrently; results land in the caller's arrays in query order.
 *      vsg_group_allpairs shards the rows of the group's own sequence set with vsg_allpairs_partition.  No
 *      collective is involved beyond the one-to-all copy of the database.  stats: ms3 = {upload+mask on the first
 *      device, device-to-device copies, index builds}, bytes copied between devices. ---- */
typedef struct vsg_group vsg_group;
int vsg_group_create(const int * devices, int ndev, const vsg_scoring * scoring, const char * cat,
                     const int64_t * off, const int32_t * len, int64_t n, int wordlength, int mask_lower,
                     int dust_db, vsg_group ** out);
void vsg_group_destroy(vsg_group * g);
int vsg_group_size(const vsg_group * g);
vsg_ctx * vsg_group_ctx(vsg_group * g, int i);
vsg_seqset * vsg_group_db(vsg_group * g, int i);
vsg_index * vsg_group_index(vsg_group * g, int i);
int vsg_group_stats(const vsg_group * g, double * ms3, int64_t * broadcast_bytes);
int vsg_group_set_fallback(vsg_group * g, vsg_fallback_fn fn, void * user);
int vsg_group_search(vsg_group * g, const char * qcat, const int64_t * qoff, const int32_t * qlen, int64_t nq,
                     int dust_queries, const vsg_search_opts * opts, vsg_search_result * results, int max_results,
                     int32_t * counts, int64_t * work);
int vsg_group_allpairs(vsg_group * g, const vsg_search_opts * opts, vsg_pair_hit * hits, int64_t cap,
                       int64_t * nhits, int64_t * work);

/* ---- streaming --usearch_global driver (SURVEY.md §8 f1): replaces the query loop of search_thread_run /
 *      search_output_results (commands/usearch_global.cpp:150-300, 376-534) for FASTA in, --blast6out out
 *      (core/results.cpp:221-271).  Three stages run concurrently on batches of batch_queries sequences:
 *      a reader thread parses the FASTA file (headers cut at the first blank unless notrunclabels), the calling
 *      thread runs vsg_group_search on every GPU of the group (query upload, optional DUST, ranking, alignment,
 *      accept/reject, hit table download), a writer thread formats the rows of min(maxhits, hits) per query IN INPUT
 *      ORDER (the reference's order with --threads 1); no other bound on the rows of a query (--maxaccepts 0 may
 *      report the whole database).  target_labels: the database headers as the reference would
 *      print them.  output_no_hits != 0: the "*" row for queries without a hit.  stats (optional) receives counts and
 *      the busy seconds of each stage. ---- */
typedef struct vsg_stream_stats {
  int64_t queries, matched, rows, batches, nucleotides;
  double parse_s, search_s, write_s, wall_s;
} vsg_stream_stats;
int vsg_usearch_stream(vsg_group * g, const char * const * target_labels, const char * query_fasta,
                       const vsg_search_opts * opts, int qmask_dust, int notrunclabels, int batch_queries,
                       int64_t maxhits, int output_no_hits, const char * blast6out_path, vsg_stream_stats * stats);

/* ---- UDB database files (SURVEY.md §8 f3): replaces udb_detect_isudb and udb_read (core/udb.cpp:120-175, 196-578).
 *      vsg_udb_detect: 1 if the file starts with the UDB signature, 0 if not, < 0 on error.  vsg_udb_open parses and
 *      validates the whole file on the host (no GPU needed; every "Invalid UDB file" check of udb_read, as VSG_EINVAL);
 *      the accessors hand out views that live until vsg_udb_close: the sequences (ASCII, back to back; case carries
 *      the masking the file was made with), the NUL-terminated headers, the stored word index (kmercount[4^k], then
 *      the ascending sequence numbers of every word).  vsg_udb_load makes the device-resident database: sequences
 *      uploaded, the device index built at the file's word length and CHECKED against the stored one (per word, the
 *      number of sequences holding it); *mask_lower (optional) receives whether the stored index excludes lower-case
 *      symbols (--dbmask dust/soft when the file was made) — pass it on as the index's masking.  A file whose stored
 *      counts match neither convention is rejected.  vsg_group_create_udb: the same for a vsg_group. ---- */
typedef struct vsg_udb vsg_udb;
typedef struct vsg_udb_info {
  int64_t sequences, nucleotides, header_chars, index_entries, longest_header;
  int32_t wordlength, dbaccel, shortest, longest;
} vsg_udb_info;
int vsg_udb_detect(const char * path);
int vsg_udb_open(const char * path, vsg_udb ** out);
void vsg_udb_close(vsg_udb * udb);
int vsg_udb_info_get(const vsg_udb * udb, vsg_udb_info * out);
int vsg_udb_sequences(const vsg_udb * udb, const char ** cat, const int64_t ** off, const int32_t ** len);
const char * vsg_udb_header(const vsg_udb * udb, int64_t i);
int vsg_udb_words(const vsg_udb * udb, const uint32_t ** kmercount, const uint32_t ** kmerindex);
int vsg_udb_load(vsg_ctx * ctx, const vsg_udb * udb, vsg_seqset ** db, vsg_index ** index, int * mask_lower);
int vsg_group_create_udb(const int * devices, int ndev, const vsg_scoring * scoring, const vsg_udb * udb, vsg_group ** out);

#ifdef __cplusplus
}
#endif
#endif /* VSG_H */
