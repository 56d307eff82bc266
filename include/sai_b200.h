/*
 * sai_b200.h -- C ABI of the B200-native U / Q sliding-window scoring path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch types.  A
 * reference-side binding (ctypes; see INTEGRATION.md) calls these from the
 * reference's batched entry point `ChunkPreprocessor.run(chr_name, start, end)`
 * (sai/preprocessors/chunk_preprocessor.py:105-147), replacing the per-window
 * Python loop
 *     WindowGenerator._window_generator   sai/generators/window_generator.py:150-247
 *     FeaturePreprocessor.run             sai/preprocessors/feature_preprocessor.py:63-191
 *     UStatistic.compute                  sai/stats/u_statistic.py:37-99
 *     QStatistic.compute                  sai/stats/q_statistic.py:37-104
 *     compute_matching_loci / calc_freq   sai/stats/stat_utils.py:55-168 / :26-52
 * The reference has no FFI of its own (pure Python + numpy); every entry point
 * below names the reference interface it replaces.
 *
 * All functions return 0 on success or a negative SAI_E_* code; device entry
 * points are stream-ordered and never synchronise the host.  `stream` is a
 * cudaStream_t passed as void* (0 = legacy default stream).
 *
 * ---------------------------------------------------------------------------
 * Packed genotype layout ("tiled bit-planes")
 * ---------------------------------------------------------------------------
 * Input encoding replaced: per-population int64 matrices of per-individual
 * allele sums, `reshape_genotypes(is_phased=False)` sai/utils/utils.py:405-410.
 *
 *  - An individual's value v (sum of its alleles; any v < 0 = missing call) is
 *    stored in `bits` = B bit-planes as the binary code of v; the all-ones code
 *    (2^B - 1) means missing.  B = 2 covers haploid/diploid data (0,1,2,missing); B up to 8
 *    holds every int8 value (multi-allelic GT indices are not recoded by the reference, and a
 *    flipped missing allele counts 2: sai/utils/utils.py:119-135, :555).  The genotype pass is
 *    at the HBM roofline for B = 2..4; B = 5..8 take a plain per-word path (DD included:
 *    sai_site_hist / sai_window_dd).
 *  - 32 individuals of one population form a *group*: B consecutive 32-bit
 *    words (plane 0 .. plane B-1), bit i of a word = individual 32*g + i.
 *    Unused individuals of the last group are coded missing.
 *  - The words of a population (groups * B of them) are laid out in 8-byte
 *    *pairs* (padded with one zero word when odd).  A site's column is the
 *    concatenation of its populations' pairs: `pairs_per_site` pairs.
 *  - Sites are grouped in *tiles* of 32.  A tile is stored as
 *        pair_t tile[pairs_per_site][32 sites]          (8-byte elements)
 *    so that the 32 lanes of a warp read 256 contiguous bytes per pair index
 *    and each lane owns one site.  Tiles are contiguous:
 *        byte offset(tile T, pair p, site s) = ((T*pairs_per_site + p)*32 + s)*8
 *    Sites beyond n_sites in the last tile are coded all-missing.
 */
#ifndef SAI_B200_H
#define SAI_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SAI_MAX_POPS 16  /* populations in one packed matrix          */
#define SAI_MAX_SRC 8    /* source populations of one job             */
#define SAI_MAX_JOBS 8   /* (ref,tgt) jobs fused into one genotype pass */
#define SAI_TILE_SITES 32
#define SAI_MAX_BITS 8    /* bit-planes per population: values 0..254, i.e. all of int8 */

enum {
  SAI_OK = 0,
  SAI_E_ARG = -1,      /* invalid argument (maps to the reference's ValueError) */
  SAI_E_CUDA = -2,     /* CUDA runtime error; see sai_last_error()              */
  SAI_E_DOMAIN = -3,   /* genotype value does not fit the bit-planes            */
  SAI_E_CAPACITY = -4, /* candidate buffers too small; totals were written      */
  SAI_E_NOMEM = -5,
  SAI_E_CORRUPT = -6,  /* a bgzip block inflated on the device is corrupt; see sai_last_error() */
  SAI_E_ORDER = -7     /* genome ingest: a chromosome's records resume after another chromosome's */
};

/* comparator of a source population, `"=", "<", ">", "<=", ">="`
 * (sai/stats/stat_utils.py:133-139, parsed at sai/configs/stat_config.py:159-207) */
enum { SAI_OP_EQ = 0, SAI_OP_LT = 1, SAI_OP_GT = 2, SAI_OP_LE = 3, SAI_OP_GE = 4 };

typedef struct {
  int32_t n_samples; /* individuals in the population                     */
  int32_t ploidy;    /* configured ploidy: frequency denominator factor   */
  int32_t bits;      /* bit-planes B (2..SAI_MAX_BITS)                    */
  int32_t pair_off;  /* first pair of this population in a site column    */
  int32_t n_pairs;   /* pairs owned by this population                    */
  int32_t n_groups;  /* ceil(n_samples / 32)                              */
} sai_pop_layout;

typedef struct {
  int32_t n_pops;
  int32_t pairs_per_site;
  sai_pop_layout pop[SAI_MAX_POPS];
} sai_layout;

/* One condition block = the arguments of compute_matching_loci
 * (sai/stats/stat_utils.py:55-63) that are not genotypes. */
typedef struct {
  double w;                      /* ref_freq < w                               */
  double y[SAI_MAX_SRC];         /* thresholds, one per source population      */
  double one_minus_y[SAI_MAX_SRC]; /* host-computed Python-float `1 - y`
                                    (stat_utils.py:149)                       */
  int32_t op[SAI_MAX_SRC];       /* SAI_OP_*                                   */
  int32_t enabled;               /* 0: statistic not requested                 */
  int32_t pad_;
} sai_cond;

/* One job = one (ref_pop, tgt_pop, src_combination) of the population product
 * (sai/generators/window_generator.py:164-166) with the U and Q parameters
 * FeaturePreprocessor.run hands to the statistic classes
 * (sai/preprocessors/feature_preprocessor.py:163-186). */
typedef struct {
  int32_t ref_pop;               /* index into sai_layout.pop                  */
  int32_t tgt_pop;
  int32_t n_src;
  int32_t src_pop[SAI_MAX_SRC];
  int32_t anc_allele_available;  /* 0: also try 1-y and invert (stat_utils.py:146-160) */
  sai_cond u;                    /* UStatistic: w, y_list                      */
  double x;                      /* UStatistic: tgt_freq > x  (u_statistic.py:92) */
  sai_cond q;                    /* QStatistic: w, y_list                      */
  double quantile;               /* QStatistic: quantile (q_statistic.py:100)  */
} sai_job;

/* ---- library ------------------------------------------------------------ */
const char* sai_version(void);
const char* sai_last_error(void); /* thread-local message of the last failure */

/* ---- layout / host encode (replaces reshape_genotypes, utils.py:405-410) -- */
/* Fills offsets for `n_pops` populations; bits[i] <= 0 selects the smallest B
 * that holds 0..ploidy plus the missing code. */
int sai_layout_init(sai_layout* lay, int32_t n_pops, const int32_t* n_samples,
                    const int32_t* ploidy, const int32_t* bits);
/* bits needed for values 0..max_value plus the missing code */
int32_t sai_bits_for_max_value(int32_t max_value);
int64_t sai_num_tiles(int64_t n_sites);
uint64_t sai_packed_bytes(const sai_layout* lay, int64_t n_sites);

/* Packs population `pop` of sites [0, n_sites) from a row-major int8 matrix of
 * per-individual allele sums (`gt[site*row_stride + individual]`, negative =
 * missing) into `packed` (host memory, sai_packed_bytes() long, all
 * populations share it).  Call once per population.  Returns SAI_E_DOMAIN if a
 * value exceeds the population's bit-planes.  `n_threads` <= 0: hardware
 * concurrency. */
int sai_pack_i8(const sai_layout* lay, int32_t pop, const int8_t* gt,
                int64_t n_sites, int64_t row_stride, uint8_t* packed,
                int32_t n_threads);
/* All populations in one pass, site by site: when the matrices are column blocks of one row-major
 * matrix (what a VCF parse leaves behind) the input is read as one sequential stream. */
int sai_pack_i8_all(const sai_layout* lay, const int8_t* const* gt, const int64_t* row_stride, int64_t n_sites,
                    uint8_t* packed, int32_t n_threads);
/* The vector path the packer selected on this CPU: "avx512gfni" (AVX-512 + GFNI + VBMI: 8x8
 * bit-matrix transposes), "avx512bw", "avx2", "sse2" or "portable"; sai_pack_i8_isa forces one
 * (1 portable, 2 sse2, 3 avx2, 4 avx512bw, 5 avx512gfni; 0 = best; an unavailable choice falls
 * back to the best) -- all paths produce identical bytes (tests). */
const char* sai_pack_isa(void);
int sai_pack_i8_isa(const sai_layout* lay, int32_t pop, const int8_t* gt, int64_t n_sites,
                    int64_t row_stride, uint8_t* packed, int32_t n_threads, int32_t isa);
/* Inverse of sai_pack_i8 for sites [site0, site0+n): missing decodes to -1. */
int sai_unpack_i8(const sai_layout* lay, int32_t pop, const uint8_t* packed,
                  int64_t n_sites_total, int64_t site0, int64_t n, int8_t* gt,
                  int64_t row_stride);

/* Negative-value table of one int8 population matrix (the side table of DD, see "N4" below):
 * every entry v < 0, row-major -> (site, individual, value).  Returns the number of entries;
 * nothing is written when cap is 0 (counting call) or smaller than that number. */
int64_t sai_neg_table_i8(const int8_t* gt, int64_t n_sites, int32_t n_samples, int64_t row_stride,
                         int32_t* site, int32_t* ind, int32_t* val, int64_t cap, int32_t n_threads);

/* ---- host VCF ingest (replaces read_geno_data + check_anc_allele + flip_snps +
 * reshape_genotypes(is_phased=False), sai/utils/utils.py:78-186, 492-555, 405-410) */
/* One pass over VCF text (complete lines are consumed; *bytes_consumed tells
 * where the next call has to start).  For every record of `chrom` with
 * start <= POS <= end (no region filter when start > end) that survives the
 * ancestral-allele table (n_anc == 0: no table; entries: sorted anc_pos[i] with
 * the allele in anc_allele + 8*i, NUL padded) writes out_pos[row] and, for every
 * requested output column o, out_gt[row*row_stride + o] = sum of the first
 * sample_ploidy[o] alleles of VCF sample column sample_column[o] ("." and
 * absent alleles = -1; flipped records: every allele a -> |a - 1|).
 * Returns the number of rows written (<= rows_cap) or a negative SAI_E_* code. */
int64_t sai_vcf_parse_gt(const char* text, int64_t len, const char* chrom, int64_t start,
                         int64_t end, const int32_t* sample_column, const int32_t* sample_ploidy,
                         int32_t n_out, const int32_t* anc_pos, const char* anc_allele,
                         int64_t n_anc, int32_t* out_pos, int8_t* out_gt, int64_t row_stride,
                         int64_t rows_cap, int64_t* bytes_consumed, int32_t n_threads);

/* First / last POS (file order) and number of records of `chrom` among the complete lines of
 * `text` (replaces the pysam loop of ChunkGenerator.__init__, chunk_generator.py:64-76).
 * *first = *last = -1 when the chromosome does not occur. */
int sai_vcf_chrom_span(const char* text, int64_t len, const char* chrom, int64_t* first,
                       int64_t* last, int64_t* n_records, int64_t* bytes_consumed,
                       int32_t n_threads);

/* BGZF (bgzip) input: a .vcf.gz written by bgzip is a sequence of independent gzip members of
 * <= 64 KB.  sai_bgzf_scan indexes the complete blocks at the start of `data` (at most
 * max_blocks, stopping before the uncompressed total exceeds max_out_bytes unless it is the
 * first block): block_off[i] = offset of block i, out_off[i] = offset of its text,
 * out_off[n] = total text bytes, *consumed = compressed bytes covered; returns n.
 * sai_bgzf_inflate inflates those blocks in parallel (CRC checked) into `out`. */
int32_t sai_is_bgzf(const uint8_t* data, int64_t len);
int64_t sai_bgzf_scan(const uint8_t* data, int64_t len, int64_t max_blocks, int64_t max_out_bytes,
                      int64_t* block_off, int64_t* out_off, int64_t* consumed);
int sai_bgzf_inflate(const uint8_t* data, const int64_t* block_off, const int64_t* out_off,
                     int64_t n_blocks, uint8_t* out, int32_t n_threads);
/* Fused bgzip read: blocks [0, n_blocks) as indexed by sai_bgzf_scan over the WHOLE rest of the
 * file, inflated in groups and parsed by the thread that inflated them while the text is still
 * in its cache -- the text never exists in memory as a whole.  `skip` = text offset of the first
 * record (the byte behind the "#CHROM" line); the other arguments and the rows written are those
 * of sai_vcf_parse_gt over the same text (a last line without a newline is complete).  Returns
 * the number of rows, SAI_E_CAPACITY when rows_cap is too small (nothing is resumable: size the
 * output from the text size, out_off[n_blocks] / (2 * n_out) rows are always enough), or another
 * negative SAI_E_* code.  group_blocks <= 0: 16 blocks (~1 MB of text) per group. */
int64_t sai_bgzf_parse_gt(const uint8_t* data, const int64_t* block_off, const int64_t* out_off,
                          int64_t n_blocks, int64_t skip, const char* chrom, int64_t start,
                          int64_t end, const int32_t* sample_column, const int32_t* sample_ploidy,
                          int32_t n_out, const int32_t* anc_pos, const char* anc_allele,
                          int64_t n_anc, int32_t* out_pos, int8_t* out_gt, int64_t row_stride,
                          int64_t rows_cap, int32_t group_blocks, int32_t n_threads);
/* A plain single-member gzip file (not bgzip) into `out` in one call with the same decoder:
 * returns the text length (= the trailer's ISIZE), SAI_E_CAPACITY when out_cap is smaller,
 * SAI_E_DOMAIN when the file is not what the fast path handles -- several members, more than
 * 4 GB of text, or corrupt: read it with a streaming gzip reader instead -- or SAI_E_ARG. */
int64_t sai_gzip_inflate(const uint8_t* data, int64_t len, uint8_t* out, int64_t out_cap);
/* The block decoder and checksum sai_bgzf_inflate uses (tests, tools): raw deflate stream
 * (RFC 1951) of known inflated size -> 1 on success, 0 on anything unexpected (sai_bgzf_inflate
 * then repeats the block with zlib); CRC-32 == zlib's crc32(0, data, len) (isa: 0 = PCLMULQDQ
 * when the CPU has it, 1 = slicing tables). */
int32_t sai_inflate_raw(const uint8_t* in, int64_t in_len, uint8_t* out, int64_t out_len);
uint32_t sai_crc32(const uint8_t* data, int64_t len, int32_t isa);

/* Device inflate of BGZF blocks (all of RFC 1951, CRC-32 checked).  One descriptor per block,
 * built on the host from sai_bgzf_scan's table: the raw deflate payload of comp_bytes bytes at
 * d_comp + comp_off (behind the gzip header, FEXTRA included), inflated into exactly isize (<= 65536)
 * bytes at d_out + text_off, whose CRC-32 must equal crc (the member's trailer).  Stream-ordered,
 * never synchronises the host.  d_status[i] = 0 when block i decoded to exactly isize bytes with a
 * matching CRC; 1 an invalid stream, 2 too much or too little output, 3 a CRC mismatch -- and then
 * its output range holds '\n' bytes only.  Blocks never write outside their own output range. */
typedef struct {
  int64_t comp_off;   /* payload offset in the device compressed buffer */
  int64_t text_off;   /* offset of the block's text in the device output */
  int32_t comp_bytes; /* payload bytes (the member minus header and the 8-byte trailer) */
  int32_t isize;      /* text bytes (the trailer's ISIZE) */
  uint32_t crc;       /* expected CRC-32 of the text (the trailer's CRC32) */
  int32_t pad_;
} sai_bgzf_block;
int sai_bgzf_inflate_device(const uint8_t* d_comp, const sai_bgzf_block* d_blocks, int64_t n_blocks,
                            uint8_t* d_out, int32_t* d_status, void* stream);
/* The descriptors of blocks [0, n_blocks) of a sai_bgzf_scan table (HOST data, block_off, out_off)
 * when the members from block_off[0] on are copied, as they lie, to d_comp + comp_base and the text
 * of block 0 goes to d_out + text_base: the payload offset from the gzip header walk (FEXTRA may
 * hold more than BC), isize = out_off[j + 1] - out_off[j], crc from the member's trailer. */
int sai_bgzf_descriptors(const uint8_t* data, const int64_t* block_off, const int64_t* out_off, int64_t n_blocks,
                         int64_t comp_base, int64_t text_base, sai_bgzf_block* out);

/* ---- device VCF ingest: VCF text in HBM -> tiled bit-planes ----------------
 * The same records and values as sai_vcf_parse_gt (the host parser is the specification), written
 * straight into the packed layout: population p of `lay` takes its n_samples individuals from the
 * VCF sample columns sample_column[first_p .. first_p + n_samples), first_p = sum of the earlier
 * populations' n_samples, with the population's ploidy.  Values are coded in the population's
 * bit-planes (negative = missing); a value that does not fit is recorded in vmax and the call still
 * succeeds -- sai_vcf_state tells the caller to repeat with a wider layout. */
typedef struct {
  sai_layout lay;
  const int32_t* sample_column; /* DEVICE, one VCF sample column per individual (see above) */
  const int32_t* anc_pos;       /* DEVICE, sorted; n_anc == 0: no ancestral-allele table   */
  const char* anc_allele;       /* DEVICE, 8 bytes per entry, NUL padded                    */
  int64_t n_anc;
  int64_t start, end;           /* start <= POS <= end; no region filter when start > end   */
  int32_t max_column;           /* largest entry of sample_column                          */
  int32_t chrom_len;            /* 1..255                                                  */
  char chrom[256];
} sai_vcf_query;

/* Device-side running state of one parse (zero it before the first slice). */
typedef struct {
  int64_t n_sites;              /* sites found so far: slice k numbers its records from here  */
  int32_t overflow;             /* 1: more sites than site_cap (those beyond it not written) */
  int32_t pad_;
  int32_t vmax[SAI_MAX_POPS];   /* largest value above the population's ploidy, else 0     */
} sai_vcf_state;

/* Device scratch one slice of `len` bytes needs (bytes, 256-byte aligned base). */
uint64_t sai_vcf_scratch_bytes(const sai_vcf_query* q, int64_t len);
/* Parses one slice of complete lines d_text[0, len) (16-byte aligned, len < 2^31), stream-ordered:
 * kept records become sites d_state->n_sites, d_state->n_sites + 1, ... of d_tiles (tile 0 based,
 * site_cap sites = a multiple of 32) and d_pos; the sites behind the last one, to the end of its
 * tile, are coded all-missing, so after every call the tiles equal sai_pack_i8_all's over the
 * sites so far.  Never synchronises the host. */
int sai_vcf_tiles_device(const sai_vcf_query* q, const char* d_text, int64_t len, void* d_scratch,
                         uint64_t scratch_bytes, void* d_tiles, int32_t* d_pos, int64_t site_cap,
                         sai_vcf_state* d_state, void* stream);

/* ---- K1: site counts (replaces calc_freq's passes, stat_utils.py:45-49) --- */
/* For tiles [tile0, tile0+n_tiles): per population p and site s
 *     num[p*stride + s]    = sum of called values      (stat_utils.py:48)
 *     called[p*stride + s] = number of called individuals (stat_utils.py:46)
 * d_packed points at tile 0.  `variant` must be 0 (carry-save popcount, 8 streaming loads in
 * flight per lane, 4 blocks/SM); other values select A/B variants that exist only in
 * -DSAI_EXPERIMENTS builds (tools/, profiles/round1_notes.md) and are rejected with SAI_E_ARG. */
int sai_site_counts(const sai_layout* lay, const void* d_packed, int64_t tile0,
                    int64_t n_tiles, int32_t* d_num, int32_t* d_called,
                    int64_t stride, int32_t variant, void* stream);

/* ---- K1 fused: counts + per-site U/Q conditions in one genotype pass ------ */
/* Per job j and tile T writes the 32-bit masks
 *     d_mask_u[j*n_tiles_total + T], d_mask_q[j*n_tiles_total + T]
 * (bit s = site 32*T+s satisfies the U resp. Q condition: stat_utils.py:166,
 * u_statistic.py:92) and, for Q-flagged sites, the (possibly inverted) target
 * frequency d_qval[j*qval_stride + site] (q_statistic.py:92).  Optionally also
 * stores the counts (d_num/d_called may be NULL). */
int sai_site_flags(const sai_layout* lay, const void* d_packed, int64_t tile0,
                   int64_t n_tiles, int64_t n_tiles_total, const sai_job* jobs,
                   int32_t n_jobs, uint32_t* d_mask_u, uint32_t* d_mask_q,
                   double* d_qval, int64_t qval_stride, int32_t* d_num,
                   int32_t* d_called, int64_t count_stride, int32_t variant,
                   void* stream);

/* Same outputs computed from cached counts (threshold sweeps never re-read the
 * genotypes). */
int sai_flags_from_counts(const sai_layout* lay, const int32_t* d_num,
                          const int32_t* d_called, int64_t count_stride,
                          int64_t n_sites, const sai_job* jobs, int32_t n_jobs,
                          uint32_t* d_mask_u, uint32_t* d_mask_q, double* d_qval,
                          int64_t qval_stride, void* stream);

/* ---- K4: windows (one launch) --------------------------------------------- */
/* Per job j and window i (inclusive [win_start[i], win_end[i]],
 * window_generator.py:173-174) over sorted unique positions d_pos[n_sites]:
 *     nsnps[j*W+i]    number of sites in the window   (feature_preprocessor.py:127)
 *     u[j*W+i]        U count                          (u_statistic.py:94-96)
 *     q[j*W+i]        Q value, NaN if no site matches  (q_statistic.py:96-100)
 *     q_cnt[j*W+i]    number of Q candidate positions  (q_statistic.py:101)
 *     u_start/q_start[j*W+i]  where the window's candidate positions start in
 *                     d_u_cand + j*cap_u / d_q_cand + j*cap_q; a window's list
 *                     is contiguous and in genome order (u[..] resp. q_cnt[..]
 *                     entries); the order of windows inside the buffer is
 *                     arbitrary (space is reserved with one atomic per window)
 *     totals[j*2+0/1] candidates of job j (U / Q).  Lists that do not fit
 *                     cap_u / cap_q are clipped: call again with larger buffers
 *                     when a total exceeds its capacity. */
int sai_window_stats(const int32_t* d_pos, int64_t n_sites, const int64_t* d_win_start,
                     const int64_t* d_win_end, int64_t n_windows, const sai_job* jobs,
                     int32_t n_jobs, const uint32_t* d_mask_u, const uint32_t* d_mask_q,
                     const double* d_qval, int64_t qval_stride, int32_t* d_nsnps,
                     int64_t* d_u, double* d_q, int32_t* d_q_cnt, int64_t* d_u_start,
                     int64_t* d_q_start, int64_t* d_totals, int32_t* d_u_cand, int64_t cap_u,
                     int32_t* d_q_cand, int64_t cap_q, void* stream);

/* Several chromosomes (or chromosome pieces) in ONE launch: the pieces' tiles and positions are
 * concatenated (every piece starts on a tile boundary; positions sorted inside a piece) and window
 * i is searched only among the sites [d_win_first_site[i], d_win_last_site[i]) of its own piece.
 * This is how one GPU scores its share of a whole-genome run -- the window ranges of
 * ChunkGenerator._split_windows_ranges (sai/generators/chunk_generator.py:111-142) over the
 * flattened (chromosome, window) list -- with one genotype pass and one window launch instead of
 * one pair per chromosome.  Everything else as sai_window_stats. */
int sai_window_stats_pieces(const int32_t* d_pos, int64_t n_sites, const int64_t* d_win_start,
                            const int64_t* d_win_end, const int32_t* d_win_first_site,
                            const int32_t* d_win_last_site, int64_t n_windows, const sai_job* jobs,
                            int32_t n_jobs, const uint32_t* d_mask_u, const uint32_t* d_mask_q,
                            const double* d_qval, int64_t qval_stride, int32_t* d_nsnps,
                            int64_t* d_u, double* d_q, int32_t* d_q_cnt, int64_t* d_u_start,
                            int64_t* d_q_start, int64_t* d_totals, int32_t* d_u_cand, int64_t cap_u,
                            int32_t* d_q_cand, int64_t cap_q, void* stream);

/* ---- N1: genome-wide outlier threshold (sai/sai.py:192-214) ------------------------------- */
/* Linear quantile `q` (pandas Series.quantile -> numpy 'linear') of the non-NaN values of each of
 * n_cols score columns, exact (radix select on the float64 bit patterns, numpy's separately
 * rounded lerp).  A column is the union of n_chunks pieces of `len` doubles:
 *     value(col, chunk, i) = d_vals[chunk*chunk_stride + col*col_stride + i]     (NaN = no value)
 * -- the layout ONE all_gather_into_tensor of the per-GPU score arrays produces, so the
 * multi-GPU threshold needs no host copy and no sort.  d_out[col*4 + 0..3] = threshold (NaN when
 * the column is empty or holds a single distinct value: the reference then writes an empty
 * table, sai.py:195-207), number of values, minimum, maximum. */
int sai_column_quantiles(const double* d_vals, int32_t n_cols, int32_t n_chunks, int64_t chunk_stride,
                         int64_t col_stride, int64_t len, double q, double* d_out, void* stream);

/* ---- N3: site-pattern sums for Danc / Dplus / df / fd ------------------------ */
/* From the cached counts of sai_site_counts: for every source population k and
 * window i the seven sums d_sums[(k*W + i)*7 + t], t = abba, baba, baaa, abaa,
 * bbaa, abba_d, baba_d (calc_pattern_sum, sai/stats/stat_utils.py:220-272; the
 * _d sums use max(tgt, src), sai/stats/fd_statistic.py:78-81).  out_pop < 0 =
 * no outgroup (frequency 0, stat_utils.py:212-213).  The statistics are
 *   Danc  = (baaa - abaa) / (baaa + abaa)                 danc_statistic.py:74-80
 *   Dplus = (abba - baba + baaa - abaa) / (abba + baba + baaa + abaa)   dplus_statistic.py:76-83
 *   df    = (abba - baba) / (abba + baba + 2 bbaa)         df_statistic.py:75-81
 *   fd    = (abba - baba) / (abba_d - baba_d)              fd_statistic.py:83-86
 * (NaN when the denominator is 0), formed by the caller.  The sums are accumulated in the order
 * of numpy's pairwise summation (np.sum of a contiguous float64 vector), so they are bit-identical
 * to the reference's. */
int sai_window_patterns(const sai_layout* lay, const int32_t* d_pos, int64_t n_sites,
                        const int64_t* d_win_start, const int64_t* d_win_end, int64_t n_windows,
                        const int32_t* d_num, const int32_t* d_called, int64_t count_stride,
                        int32_t ref_pop, int32_t tgt_pop, int32_t out_pop, const int32_t* src_pops,
                        int32_t n_src, double* d_sums, void* stream);

/* ---- N4: DD (sai/stats/dd_statistic.py:62-77) ------------------------------- */
/* DD = mean_a( mean_j sum_sites |src_a - ref_j|  -  mean_j sum_sites |src_a - tgt_j| ) uses the RAW
 * allele sums, missing calls included with their negative value (cdist cityblock,
 * dd_statistic.py:70-71).  The bit-planes keep a single missing code, so DD takes a
 * *negative-value table* next to the packed matrix: for population p the entries
 * neg_off[p] .. neg_off[p+1]-1 of (neg_site = site index, neg_ind = individual index
 * inside the population, neg_val = raw value < 0), sorted by (site, individual).
 * neg_off is host memory ([n_pops + 1], neg_off[0] = 0).
 *
 * sai_site_hist: one genotype pass over the listed populations; row r of population
 * pops[q] (rows of earlier populations first, sai_hist_rows() in total: 2^bits - 1 rows for
 * bits <= 4, 16 rows for bits 5..8)
 *     d_hist[r*stride + site] = number of individuals whose called value is r   (r <= 14),
 * and for bits 5..8 row 15 = number of *wide* calls (called values >= 15), which
 * sai_window_dd reads back from the bit-planes.
 * d_missing[q] (optional) = missing calls of pops[q] over sites < n_sites, padding excluded.
 *
 * sai_window_dd: d_hist must hold {ref_pop, tgt_pop} in this order.  Per source population k,
 * window i and source individual a (exact integers)
 *     d_ref_sum[(k*W + i)*m_max + a] = sum_j sum_sites |src_a - ref_j|        (tgt likewise)
 * *d_err is set to 1 if a missing source call has no table entry.  Per-site distances are int32:
 * ref and tgt may hold at most 8 454 660 individuals each (254 per individual and site).
 * The caller forms
 *     DD_k = mean_a( ref_sum/n_ref - tgt_sum/n_tgt )           dd_statistic.py:74-77 */
int64_t sai_hist_rows(const sai_layout* lay, const int32_t* pops, int32_t n);
int sai_site_hist(const sai_layout* lay, const void* d_packed, int64_t n_sites, const int32_t* pops,
                  int32_t n_hist_pops, int32_t* d_hist, int64_t stride, uint64_t* d_missing,
                  void* stream);
int sai_window_dd(const sai_layout* lay, const void* d_packed, const int32_t* d_pos, int64_t n_sites,
                  const int64_t* d_win_start, const int64_t* d_win_end, int64_t n_windows,
                  const int32_t* d_hist, int64_t stride, int32_t ref_pop, int32_t tgt_pop,
                  const int32_t* src_pops, int32_t n_src, const int64_t* neg_off,
                  const int32_t* d_neg_site, const int32_t* d_neg_ind, const int32_t* d_neg_val,
                  int64_t* d_ref_sum, int64_t* d_tgt_sum, int32_t m_max, int32_t* d_err,
                  void* stream);

/* ---- zt: zero-suppressed tiles, the host->device wire format --------------- */
/* End to end the path is bound by the PCIe copy of the packed tiles, and most of a genotype
 * matrix is the hom-ref code 0.  The zt stream holds, per tile (P = pairs_per_site rows of 32
 * pairs), at byte offset tile_off[T] & ~SAI_ZT_RAW (8-byte aligned):
 *     u32 n1        non-zero pairs of the tile
 *     u32 nz[P]     bit s of nz[r]: pair (row r, site s) is non-zero
 *     u8  mask[n1]  per non-zero pair in (r, s) order: bit k = byte k of the pair is non-zero
 *     u8  data[..]  the non-zero bytes in the same order, ascending k
 * where "pair" = stored pair XOR the row's padding constant (ones for the unused individuals
 * of a population's last group).  A tile that would not shrink is stored as its P*256 raw
 * bytes, flagged by SAI_ZT_RAW in tile_off[T]; tile_off[n_tiles] = stream length.
 * Lossless: sai_zt_decode(sai_zt_encode(x)) == x bit for bit. */
#define SAI_ZT_RAW (1ull << 63)
uint64_t sai_zt_bound(const sai_layout* lay, int64_t n_sites); /* upper bound of the stream length */
/* Host: packed tiles -> stream + tile_off[n_tiles + 1].  Returns the stream length or a
 * negative SAI_E_* code (SAI_E_CAPACITY: out_cap too small). */
int64_t sai_zt_encode(const sai_layout* lay, const uint8_t* packed, int64_t n_sites, uint8_t* out,
                      uint64_t out_cap, uint64_t* tile_off, int32_t n_threads);
/* The encoder's vector path on this CPU: "avx512vbmi2" (vpcompressb) or "portable";
 * sai_zt_encode_isa forces one (0 = best, 1 = portable) -- identical bytes (tests). */
const char* sai_zt_isa(void);
int64_t sai_zt_encode_isa(const sai_layout* lay, const uint8_t* packed, int64_t n_sites, uint8_t* out,
                          uint64_t out_cap, uint64_t* tile_off, int32_t n_threads, int32_t isa);
/* Host: int8 matrices (arguments as sai_pack_i8_all) -> the same stream and directory as
 * sai_zt_encode(sai_pack_i8_all(...)), byte for byte, without the dense tiles ever leaving the
 * packers' L1 caches (the int8 pipeline's encoder; also the fast way to build a compressed
 * on-disk cache).  Returns the stream length or a negative SAI_E_* code (SAI_E_DOMAIN: a value
 * does not fit the layout's bit-planes; SAI_E_CAPACITY: out_cap too small -- sai_zt_bound is
 * always enough). */
int64_t sai_zt_pack_i8(const sai_layout* lay, const int8_t* const* gt, const int64_t* row_stride,
                       int64_t n_sites, uint8_t* out, uint64_t out_cap, uint64_t* tile_off,
                       int32_t n_threads);
/* Host decoder (tests, tools). */
int sai_zt_decode_host(const sai_layout* lay, const uint8_t* stream, const uint64_t* tile_off,
                       int64_t n_sites, uint8_t* packed);
/* Device: rebuilds dense tiles [tile0, tile0 + n_tiles) of d_packed (tile 0 based) from the
 * stream resident at d_stream (offset 0 based, 8-byte aligned, stream_bytes = tile_off[n_tiles_total]
 * long: the decoder never loads beyond it) and its directory d_tile_off. */
int sai_zt_decode(const sai_layout* lay, const void* d_stream, uint64_t stream_bytes,
                  const uint64_t* d_tile_off, int64_t tile0, int64_t n_tiles, void* d_packed,
                  void* stream);

/* ---- host-buffer engine (replaces ChunkPreprocessor.run's inner loop) ----- */
typedef struct sai_engine sai_engine;
int sai_engine_create(int32_t device, sai_engine** out);
void sai_engine_destroy(sai_engine* e);

typedef struct {
  int32_t* nsnps;   /* [n_jobs*W]     */
  int64_t* u;       /* [n_jobs*W]     */
  double* q;        /* [n_jobs*W]     */
  int32_t* q_cnt;   /* [n_jobs*W]     */
  int64_t* u_start; /* [n_jobs*W]     */
  int64_t* q_start; /* [n_jobs*W]     */
  int64_t* totals;  /* [n_jobs*2]     */
  int32_t* u_cand;  /* [n_jobs*cap_u] */
  int32_t* q_cand;  /* [n_jobs*cap_q] */
  int64_t cap_u, cap_q;
} sai_host_results;

/* HOST pointers in, HOST results out: copies the packed tiles to the GPU in
 * slices that overlap with the genotype pass, runs the window kernel, copies
 * the results back and synchronises.  Returns SAI_E_CAPACITY (everything but
 * the candidate lists is valid, totals say what is needed) when cap_u / cap_q
 * were too small. */
int sai_engine_score_host(sai_engine* e, const sai_layout* lay, const uint8_t* packed,
                          const int32_t* pos, int64_t n_sites, const int64_t* win_start,
                          const int64_t* win_end, int64_t n_windows, const sai_job* jobs,
                          int32_t n_jobs, sai_host_results* out);

/* Same as sai_engine_score_host with the tiles in zt form (HOST stream + HOST directory):
 * the stream is copied in ~32 MB slices, each slice is expanded to dense tiles on the device
 * and flagged while the next slice is on the wire. */
int sai_engine_score_host_zt(sai_engine* e, const sai_layout* lay, const uint8_t* zt_stream,
                             const uint64_t* zt_tile_off, const int32_t* pos, int64_t n_sites,
                             const int64_t* win_start, const int64_t* win_end, int64_t n_windows,
                             const sai_job* jobs, int32_t n_jobs, sai_host_results* out);

/* Same as sai_engine_score_host straight from the reference-side representation: gt[p] is the
 * row-major int8 matrix of population p's per-individual allele sums
 * (gt[p][site * row_stride[p] + individual], negative = missing; what reshape_genotypes leaves
 * in memory, sai/utils/utils.py:405-410, narrowed to int8), ordinary pageable host memory.
 * A pool of host threads (sai_engine_set_host_threads; default: all cores) packs 32 MB slices
 * of tiles into a ring of pinned staging buffers with the CPU's vector unit (sai_pack_isa) --
 * by default as zt records encoded while a tile is still in the packer's L1 (sai_zt_isa,
 * sai_engine_set_i8_wire); each finished slice is copied to the GPU, expanded and flagged while
 * the following slices are being packed, so the call costs about max(pack, copy) instead of
 * pack + copy.  Returns SAI_E_DOMAIN when a
 * value does not fit the layout's bit-planes (retry with a wider layout). */
int sai_engine_score_host_i8(sai_engine* e, const sai_layout* lay, const int8_t* const* gt,
                             const int64_t* row_stride, const int32_t* pos, int64_t n_sites,
                             const int64_t* win_start, const int64_t* win_end, int64_t n_windows,
                             const sai_job* jobs, int32_t n_jobs, sai_host_results* out);
/* Wire format of the int8 pipeline.  2 = zt records: every packer turns the tile it has just
 * packed into a zt record while it is still in its L1 and only the records cross host memory and
 * PCIe (k_zt_decode rebuilds the dense tiles in HBM) -- the packers are bound by the host's
 * memory system, so the bytes not written and not read back by the copy engine are throughput.
 * 1 = dense tiles (data known not to compress: no hom-ref majority).  0 (default) = auto: zt
 * when this CPU has the vector record encoder (sai_zt_isa() != "portable"), else dense.
 * Results are identical.
 * sai_engine_i8_wire_bytes: tile bytes the last sai_engine_score_host_i8 call copied. */
int sai_engine_set_i8_wire(sai_engine* e, int32_t mode);
uint64_t sai_engine_i8_wire_bytes(const sai_engine* e);
/* Host threads the int8 pipeline may use (<= 0: hardware concurrency).  One engine per GPU:
 * with several ranks on a box give each its share of the cores. */
int sai_engine_set_host_threads(sai_engine* e, int32_t n_threads);

/* Another batch of jobs over the chunk of the last sai_engine_score_host* call, whose tiles,
 * positions and windows are still resident on the device: genotype pass + window kernel, no host
 * to device traffic.  This is how a population product of more than SAI_MAX_JOBS combinations
 * (sai/generators/window_generator.py:164-166) is scored with ONE upload. */
int sai_engine_score_resident(sai_engine* e, const sai_job* jobs, int32_t n_jobs, sai_host_results* out);

/* After SAI_E_CAPACITY: re-runs only the window kernel on the flags still
 * resident on the device, with the (larger) buffers of `out`. */
int sai_engine_rescore_windows(sai_engine* e, sai_host_results* out);

/* Site-pattern sums (see sai_window_patterns) for the chunk of the last
 * sai_engine_score_host call, whose packed tiles, positions and windows are
 * still resident on the device: runs the counting genotype pass + the pattern
 * kernel and copies sums[n_src][W][7] to the host.  The pattern kernel runs once per piece
 * (sai_engine_score_loaded_pieces), a piece's window i landing at sums[k][w0 + i] for its first
 * window w0; a chunk scored whole is the one piece of W windows from window 0 and all sites from
 * site 0.  The DD sums below walk the pieces the same way. */
int sai_engine_pattern_sums(sai_engine* e, const sai_layout* lay, int32_t ref_pop, int32_t tgt_pop,
                            int32_t out_pop, const int32_t* src_pops, int32_t n_src, double* sums);

/* DD sums (see sai_window_dd) for the chunk of the last sai_engine_score_host call; the
 * negative-value table is HOST memory, one row of offsets (neg_off[n_pops + 1]), copied to the
 * device per call.  The chunk is one piece (see sai_engine_pattern_sums); tiles scored in pieces
 * are refused (sai_engine_dd_sums_loaded takes them).  Fails with SAI_E_ARG when the table does not
 * cover every missing call of ref_pop / tgt_pop / the source populations.
 * ref_sum / tgt_sum: host, [n_src][W][m_max]. */
int sai_engine_dd_sums(sai_engine* e, const sai_layout* lay, int32_t ref_pop, int32_t tgt_pop,
                       const int32_t* src_pops, int32_t n_src, const int64_t* neg_off,
                       const int32_t* neg_site, const int32_t* neg_ind, const int32_t* neg_val,
                       int64_t* ref_sum, int64_t* tgt_sum, int32_t m_max);

/* ---- engine ingest session: a VCF parsed on the device, tiles left resident -------------------
 * sai_engine_vcf_begin: populations of `lay` as in sai_vcf_query (sample_column, n_out = sum of
 * n_samples, HOST), the ancestral-allele table (HOST, as sai_vcf_parse_gt), n_file_samples = sample
 * columns of the #CHROM line and text_bytes_hint = text bytes expected (0: unknown) size the tile
 * buffer (records are >= 2 * n_file_samples + 18 bytes; it grows with the text fed), min_sites = a
 * lower bound of its capacity (a repeat after SAI_E_CAPACITY).
 * sai_engine_vcf_feed: host text of any size; the complete lines are consumed (*consumed), the
 * rest is the caller's to carry -- the contract of a `_scan_text` on_lines callback.  Host threads
 * copy slices of complete lines into a ring of pinned buffers; each slice goes to the device with
 * cudaMemcpyAsync on the copy stream and is parsed on the compute stream while the next ones are
 * staged.  Returns once the bytes are staged.
 * sai_engine_vcf_finish: synchronises once; *n_sites, max_value[p] = max(ploidy, largest value of
 * population p), positions copied to pos_out when pos_cap >= *n_sites.  SAI_E_DOMAIN: a value does
 * not fit its population's bit-planes (begin again with bits = sai_bits_for_max_value(max_value[p]));
 * SAI_E_CAPACITY: more records than the tile buffer held (begin again with min_sites = *n_sites).
 * sai_engine_score_loaded: K1 + K4 on the tiles the session left resident; afterwards
 * sai_engine_score_resident / _rescore_windows / _pattern_sums work on them unchanged. */
int sai_engine_vcf_begin(sai_engine* e, const sai_layout* lay, const char* chrom, int64_t start, int64_t end,
                         const int32_t* sample_column, int32_t n_out, const int32_t* anc_pos,
                         const char* anc_allele, int64_t n_anc, int32_t n_file_samples, int64_t text_bytes_hint,
                         int64_t min_sites);
int sai_engine_vcf_feed(sai_engine* e, const char* text, int64_t len, int64_t* consumed);
/* The bgzip counterpart: blocks [0, n_blocks) as indexed by sai_bgzf_scan over the whole rest of the
 * file (out_off[0] = 0), records from text offset `skip` on (the byte behind the #CHROM line).  The
 * staging threads inflate groups of blocks (CRC checked, sai_bgzf_inflate) straight into the pinned
 * ring slots -- the text never exists as a whole -- and the incomplete last line of a slot is carried
 * into the next one; a last line without a newline is complete. */
int sai_engine_vcf_feed_bgzf(sai_engine* e, const uint8_t* data, const int64_t* block_off, const int64_t* out_off,
                             int64_t n_blocks, int64_t skip);
/* The same with the blocks inflated on the device (sai_bgzf_inflate_device): the staging threads copy
 * each group's compressed members (whole-file reads and region reads alike: block_off may index any
 * contiguous run of blocks, out_off[0] = 0) into a pinned ring, one cudaMemcpyAsync moves them to the
 * device, and the kernel inflates them into the slot that is parsed.  The host inflates only a group's
 * last block(s) to find its last newline; the incomplete line behind it travels in front of the next
 * group.  A group without any newline is staged with host inflate.  at_eof != 0: the blocks end the
 * file, so a last line without a newline is complete; otherwise that line is dropped (a region read
 * that stops inside the file).  A corrupt block makes sai_engine_vcf_finish return SAI_E_CORRUPT and
 * name the first one (its index in block_off) in sai_last_error(). */
int sai_engine_vcf_feed_bgzf_device(sai_engine* e, const uint8_t* data, const int64_t* block_off,
                                    const int64_t* out_off, int64_t n_blocks, int64_t skip, int32_t at_eof);
int sai_engine_vcf_finish(sai_engine* e, int64_t* n_sites, int32_t* max_value, int32_t* pos_out, int64_t pos_cap);
int sai_engine_score_loaded(sai_engine* e, const int64_t* win_start, const int64_t* win_end, int64_t n_windows,
                            const sai_job* jobs, int32_t n_jobs, sai_host_results* out);
/* Slice size (bytes, >= 64) and ring depth (>= 2) of the ingest session; <= 0 keeps the default
 * (32 MB, 4).  Tests use tiny slices to make records and tiles straddle slices.
 * sai_engine_vcf_slices: slices the last session parsed (tests). */
int sai_engine_set_vcf_slicing(sai_engine* e, int64_t slice_bytes, int32_t ring);
int64_t sai_engine_vcf_slices(const sai_engine* e);
/* Stages of the last finished session: out[0] host seconds staging / inflating into the ring, [1] host
 * seconds waiting for a free slot, [2] H2D and [3] parse seconds summed over the slices (CUDA events),
 * [4] seconds from the first slice's H2D start to the last slice's parse end (events), [5] slices,
 * [6] text bytes, [7] host seconds finish waited for the device, [8] host seconds enqueueing copies and
 * kernels, [9] host seconds inside the feed calls (all of the above host times and the slicing),
 * [10] device inflate seconds summed over the slices (CUDA events), [11] compressed bytes copied for
 * device inflate (descriptors included), [12] host seconds inflating the boundary blocks of
 * device-inflated groups, [13] slices inflated on the device.  n <= 14 values are written. */
int sai_engine_vcf_stats(const sai_engine* e, double* out, int32_t n);
/* The resident tiles of the finished session (sai_packed_bytes(lay, n_sites) bytes) into HOST `out`. */
int sai_engine_loaded_tiles(sai_engine* e, uint8_t* out, uint64_t cap);

/* ---- genome ingest: every chromosome of a table from one pass over a multi-chromosome VCF ------
 * sai_engine_vcf_genome_begin: as sai_engine_vcf_begin, with n_chrom (1..SAI_VCF_MAX_CHROMS) distinct
 * chromosome names (names[name_off[c] .. name_off[c + 1]), 1..255 bytes each, HOST) instead of one
 * name and no region, and the ancestral-allele tables of all of them concatenated: chromosome c's
 * entries are anc_pos / anc_allele [anc_off[c], anc_off[c + 1]) (HOST; n_anc = anc_off[n_chrom];
 * anc_off == NULL: no table, nothing is filtered).  A record's CHROM is hashed into a table in shared
 * memory and compared once, so a record costs the same whatever n_chrom is.  The session is fed with
 * sai_engine_vcf_feed / _feed_bgzf / _feed_bgzf_device.  Kept records become sites in file order, and
 * each chromosome's first site lies on a tile boundary (the genome layout of sai_window_stats_pieces):
 * the sites between a chromosome's last site and the next boundary are coded all-missing, so a
 * chromosome's tiles equal sai_pack_i8_all's over that chromosome alone.
 * sai_engine_vcf_genome_finish: as sai_engine_vcf_finish (*n_sites counts the padding sites, and so
 * does the SAI_E_CAPACITY retry), plus chroms[c] for every chromosome of the table.  SAI_E_ORDER: a
 * chromosome's kept records resume after another chromosome's (the tiles are not usable; read such a
 * file one chromosome at a time). */
#define SAI_VCF_MAX_CHROMS 1024
typedef struct {
  int64_t first_pos, last_pos; /* POS of the first / last record in file order (sai_vcf_chrom_span's  */
  int64_t n_records;           /* semantics, every record: before the ancestral-allele filter); 0 none */
  int64_t first_site, n_sites; /* kept sites [first_site, first_site + n_sites); first_site -1: none  */
} sai_vcf_chrom;
int sai_engine_vcf_genome_begin(sai_engine* e, const sai_layout* lay, const char* names, const int32_t* name_off,
                                int32_t n_chrom, const int32_t* sample_column, int32_t n_out, const int32_t* anc_pos,
                                const char* anc_allele, const int64_t* anc_off, int32_t n_file_samples,
                                int64_t text_bytes_hint, int64_t min_sites);
int sai_engine_vcf_genome_finish(sai_engine* e, int64_t* n_sites, int32_t* max_value, sai_vcf_chrom* chroms,
                                 int32_t* pos_out, int64_t pos_cap);
/* sai_engine_score_loaded over pieces of the resident tiles: piece p = pieces[3p .. 3p + 2] = (number of
 * windows, first site (a multiple of 32), number of sites); the windows are given piece after piece.
 * One genotype pass over all tiles, one sai_window_stats_pieces launch.  Afterwards
 * sai_engine_score_resident / _rescore_windows / _pattern_sums (one sai_window_patterns per piece) work
 * on the same pieces; sai_engine_dd_sums is refused (sai_engine_dd_sums_loaded is not). */
int sai_engine_score_loaded_pieces(sai_engine* e, const int64_t* win_start, const int64_t* win_end,
                                   const int64_t* pieces, int32_t n_pieces, const sai_job* jobs, int32_t n_jobs,
                                   sai_host_results* out);

/* ---- negative-value table of an ingest session (DD without a host copy) --------------------------
 * sai_engine_set_vcf_neg_table: on != 0 makes the ingest sessions that follow (sai_engine_vcf_begin /
 * _genome_begin) also keep the N4 negative-value table of their populations: the genotype pass keeps
 * the raw value of every missing call it parses.  Its capacity is unknown until the text has been
 * read: min_entries (0..2^31 - 1) is a lower bound of it (a repeat), and the finish returns
 * SAI_E_CAPACITY when the text holds more entries; sai_engine_loaded_neg_table then returns how many.
 * sai_engine_loaded_neg_table: the table of the last finished session into HOST memory, the entries of
 * chromosome c (0 for a single-chromosome session) and population p at
 *     neg_off[c * (n_pops + 1) + p] .. neg_off[c * (n_pops + 1) + p + 1] - 1
 * of site / ind / val, sorted by (site, individual), site counted from the chromosome's first site --
 * for every chromosome exactly sai_neg_table_i8 of its own int8 matrices.  neg_off (optional,
 * [n_chrom][n_pops + 1]) is always written; the entries only when cap >= their number.  Returns that
 * number (after SAI_E_CAPACITY: the number a repeat needs) or a negative SAI_E_* code.
 * sai_engine_dd_sums_loaded: sai_engine_dd_sums on the resident tiles and the resident table (no copy
 * to the device) after sai_engine_score_loaded or _score_loaded_pieces: one sai_site_hist +
 * sai_window_dd per piece (see sai_engine_pattern_sums), which must be a chromosome of the session and
 * reads that chromosome's row of the table (a single-chromosome session: its one row), its results at
 * ref_sum[k][w0 + i].  Fails with SAI_E_ARG when a population's missing calls and its table entries
 * differ. */
int sai_engine_set_vcf_neg_table(sai_engine* e, int32_t on, int64_t min_entries);
int64_t sai_engine_loaded_neg_table(sai_engine* e, int64_t* neg_off, int32_t* site, int32_t* ind, int32_t* val,
                                    int64_t cap);
int sai_engine_dd_sums_loaded(sai_engine* e, int32_t ref_pop, int32_t tgt_pop, const int32_t* src_pops, int32_t n_src,
                              int64_t* ref_sum, int64_t* tgt_sum, int32_t m_max);

/* ---- score file text on the device (score(..., write="device")) ------------------------------------
 * The rows of the score file and of the .U.log / .Q.log files, byte for byte what the host writer
 * (sai_b200.preprocessors.write_items) prints from the item dicts, formatted in HBM.  Rows come in
 * blocks: block b is one (chromosome, combination) run of windows, rows block_rows[b] ..
 * block_rows[b + 1] - 1, and holds two strings of `strings`: its chromosome (block_str[4b], length
 * block_str[4b + 1]) and "Ref\tTgt\tSrc\tOutgroup" (block_str[4b + 2], length block_str[4b + 3]).
 * A score row is
 *     chrom \t start \t end \t Ref \t Tgt \t Src \t Outgroup \t nsnps \t field_0 \t ... \t field_{n-1} \n
 * field[f] = SAI_FMT_U (the integer u), SAI_FMT_Q (the float64 q) or a column k of vals[row][n_vals];
 * every field of a row with nsnps == 0 prints "nan", a float64 prints as Python's repr(float).  A log
 * row is "chrom \t start \t end \t " followed by "NA" or the window's candidate positions as
 * "chrom:pos" joined by ",": u[row] positions from u_cand[u_start[row]] (none when nsnps == 0), and
 * q_cnt[row] from q_cand[q_start[row]] (none when nsnps == 0 or q is NaN).  The .U.log text exists
 * when a field is SAI_FMT_U (u, u_start, u_cand are then read), the .Q.log text likewise.
 * sai_engine_format_scores copies the inputs to the device, formats the three texts there (a length
 * pass, a scan of the lengths, a write pass) and keeps them resident; sizes[0..2] = bytes of the
 * rows, the .U.log and the .Q.log text (0 for one that does not exist).  sai_engine_format_text
 * copies text `which` (0..2) of the last call into HOST memory (cap >= its size).
 * sai_engine_format_stats: seconds of the last call (CUDA events): input copy, length + scan
 * kernels, write kernels.
 * sai_format_double / sai_format_doubles: repr(float(x)) on the host (the device's code), the
 * length returned; the batch writes 32 NUL-padded bytes per value.  sai_engine_format_doubles: the
 * same batch formatted by the device in one launch (tests). */
#define SAI_FMT_U (-1)
#define SAI_FMT_Q (-2)
typedef struct {
  int64_t n_blocks, n_rows;
  const int64_t* block_rows; /* [n_blocks + 1] */
  const int64_t* block_str;  /* [n_blocks][4]  */
  const char* strings;
  int64_t strings_len;
  const int64_t* start;      /* [n_rows] window bounds */
  const int64_t* end;
  const int32_t* nsnps;
  const int64_t* u;          /* [n_rows], with u_start: NULL without SAI_FMT_U */
  const int64_t* u_start;
  const double* q;           /* [n_rows], with q_start, q_cnt: NULL without SAI_FMT_Q */
  const int64_t* q_start;
  const int32_t* q_cnt;
  const int32_t* u_cand;     /* [n_u_cand] */
  const int32_t* q_cand;     /* [n_q_cand] */
  int64_t n_u_cand, n_q_cand;
  const int32_t* field;      /* [n_fields] */
  const double* vals;        /* [n_rows][n_vals] */
  int32_t n_fields, n_vals;
} sai_format_input;
int sai_engine_format_scores(sai_engine* e, const sai_format_input* in, int64_t* sizes);
int sai_engine_format_text(sai_engine* e, int32_t which, char* out, int64_t cap);
int sai_engine_format_stats(const sai_engine* e, double* out, int32_t n);
int sai_engine_format_doubles(sai_engine* e, const double* x, int64_t n, char* out);
int32_t sai_format_double(double x, char* out);
int sai_format_doubles(const double* x, int64_t n, char* out);

/* ---- outlier tables on the device (outlier(..., text="device")) ---------------------------------
 * The tables of `sai outlier` (sai_b200.outlier.outlier) built from a score file in HBM, byte for byte
 * what the host path prints after pandas.read_csv(sep="\t", na_values=["nan"], index_col=False).
 * sai_engine_table_load copies the file (header line + data rows, '\n'-terminated, the last one
 * optionally not) to the device, finds its lines and every data cell of n_cols (the header's field
 * count, at most SAI_TABLE_MAX_COLS), and ORs the classes of the cells (SAI_CELL_*, as
 * sai_classify_cells gives them) per column and per chunk of chunk_rows rows -- the rows pandas' C
 * parser infers one dtype for.  info = {data rows, chunks, SAI_TABLE_* flags of what the device path
 * does not reproduce}.  sai_engine_table_classes copies the masks, [chunks][n_cols] uint32.
 * sai_engine_table_parse takes the dtype of every column (SAI_TABLE_TEXT / _INT / _FLOAT) and the
 * columns first_metric.., Chrom, Start, End (int64): it writes the metric columns as float64 into
 * the DEVICE array d_vals[n_metric][rows] (NaN for NA; what sai_column_quantiles reads), the first
 * value of each metric column in file order into first_val (NaN when it has none), and the number of
 * runs of equal Chrom text into *n_runs; sai_engine_table_runs gives each run's Chrom as a byte
 * offset and length within the file.  sai_engine_table_order sorts the rows stably on (run_rank of
 * the row's run, Start, End).  sai_engine_table_build makes one table per metric column m: the
 * header line, then the sorted rows with value > thr[m] (strict[m] != 0) or >= thr[m] (NaN is never
 * kept; thr NaN keeps nothing), printed as ScoreTable.format_cell prints them; table m is
 * offsets[m] .. offsets[m + 1] of one text that sai_engine_table_text copies into HOST memory.
 * sai_engine_table_stats: seconds of the last calls (CUDA events): copy in, tokenise + classify,
 * parse, sort, format, copy back.
 * sai_parse_doubles: pandas' precise_xstrtod of each string text[offs[i] .. offs[i + 1]) on the host
 * (the device's code); ok[i] = 1 where pandas reads it as a float.  sai_engine_parse_doubles: the
 * same on the device (tests).  sai_classify_cells: the class of each string as a score-file cell. */
#define SAI_TABLE_MAX_COLS 128
#define SAI_TABLE_TEXT 0
#define SAI_TABLE_INT 1
#define SAI_TABLE_FLOAT 2
#define SAI_CELL_INT 1
#define SAI_CELL_FLOAT 2
#define SAI_CELL_NA 4
#define SAI_CELL_TEXT 8
#define SAI_CELL_UNSURE 16
#define SAI_CELL_BIGINT 32  /* with SAI_CELL_INT: |value| > 2^53, or more than 17 digits */
#define SAI_CELL_NEGZERO 64 /* with SAI_CELL_INT: a negative zero ("-0") */
#define SAI_TABLE_QUOTE_CR 1
#define SAI_TABLE_HIGH_BYTE 2
#define SAI_TABLE_BLANK_LINE 4
#define SAI_TABLE_RAGGED 8
#define SAI_TABLE_LONG_LINE 16 /* a line longer than 65535 bytes */
int sai_engine_table_load(sai_engine* e, const char* text, int64_t n_bytes, int32_t n_cols, int64_t chunk_rows,
                          int64_t* info);
int sai_engine_table_classes(sai_engine* e, uint32_t* out, int64_t cap);
int sai_engine_table_parse(sai_engine* e, const int32_t* kinds, int32_t first_metric, int32_t chrom, int32_t start,
                           int32_t end, double* d_vals, double* first_val, int64_t* n_runs);
int sai_engine_table_runs(sai_engine* e, int64_t* off, int64_t* len, int64_t cap);
int sai_engine_table_order(sai_engine* e, const int32_t* run_rank, int64_t n_runs);
int sai_engine_table_build(sai_engine* e, const double* thr, const int32_t* strict, int64_t* offsets);
int sai_engine_table_text(sai_engine* e, char* out, int64_t cap);
int sai_engine_table_stats(const sai_engine* e, double* out, int32_t n);
int sai_engine_parse_doubles(sai_engine* e, const char* text, const int64_t* offs, int64_t n, double* out, uint8_t* ok);
int sai_parse_doubles(const char* text, const int64_t* offs, int64_t n, double* out, uint8_t* ok);
int sai_classify_cells(const char* text, const int64_t* offs, int64_t n, uint8_t* cls);

/* ---- synthetic genotypes (bench / tests only) ---------------------------- */
/* Fills tiles [tile0, tile0+n_tiles) of a packed matrix directly on the device
 * with the synthetic model of DESIGN.md (counter-based RNG, reproducible from
 * `seed`).  role[p]: 0 = ref-like, 1 = tgt-like, 2 = src-like population. */
int sai_synth_fill(const sai_layout* lay, void* d_packed, int64_t tile0, int64_t n_tiles,
                   int64_t n_sites, const int32_t* role, uint64_t seed,
                   double missing_rate, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SAI_B200_H */
