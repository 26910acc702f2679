/* xcltk_b200.h -- C-ABI of the B200-native basefc / baf counting paths.
 *
 * The reference (hxj5/xcltk v0.5.2) is pure Python and has NO plugin / FFI boundary
 * (SURVEY.md section 8b); the seam this library sits behind is the per-worker counting core
 *   basefc: fc_features()  xcltk/rdr/fc/core.py:69-148  (fc_fet1 :151-178, check_read :46-62)
 *   baf:    fc_features()  xcltk/baf/fc/core.py:42-139  (fc_fet1 :143-194, plp_snp :198-247)
 * together with the pysam calls underneath it (AlignmentFile.fetch, AlignedSegment fields;
 * call sites listed in SURVEY.md section 8c).  Every entry point below names the reference
 * code it replaces.  INTEGRATION.md shows the ctypes stub a maintainer adds to
 * xcltk/rdr/fc/main.py:fc_core and xcltk/baf/fc/main.py:afc_core.
 *
 * Conventions: plain pointers + sizes, little-endian, no exceptions across the boundary.
 * Return 0 on success, a negative code on error (mirrors the reference's "errcode -N"
 * convention, xcltk/rdr/fc/main.py:283-292); xg_last_error() gives the message.
 * There is NO CPU fallback: device entry points fail with XG_E_CUDA when no B200 is present.
 * One xg_ctx per GPU; a context is not thread-safe, distinct contexts may be used from
 * distinct host threads concurrently.
 */
#ifndef XCLTK_B200_H
#define XCLTK_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define XG_OK 0
#define XG_E_ARG (-1)     /* bad argument                                            */
#define XG_E_IO (-2)      /* file cannot be read / is not a BAM                      */
#define XG_E_FORMAT (-3)  /* corrupt BGZF/BAM, or BAM not coordinate sorted          */
#define XG_E_NOMEM (-4)
#define XG_E_CUDA (-5)    /* CUDA error or no device: the product path has no CPU fallback */
#define XG_E_LIMIT (-6)   /* an internal capacity (32-bit offsets ...) would overflow */
#define XG_E_UNSUPPORTED (-7) /* xg_decode_bams_device: file layout / keys need the host decoder */

/* ---- string keys -------------------------------------------------------------------
 * Cell barcodes, UMIs and query names are compared by exact string equality in the
 * reference (dict / set of Python str: rdr/fc/mcount.py:34-43,119-127, baf/fc/mcount.py:109-127).
 * The device works on lossless 64-bit keys:
 *   bit63 = 0: the string itself, bit-packed MSB first, 3 bits per character
 *              (A=1 C=2 G=3 T=4 N=5 '-'=6, 7 = escape followed by a 4-bit decimal digit),
 *              zero padded; fits e.g. "ACGTACGTACGTACGT-1" and any [ACGTN]{0,21};
 *   bit63 = 1: (1<<63) | id, id = index of the string in the keyspace's intern table.
 * Equal strings <=> equal keys within one keyspace.                                     */
#define XG_KEY_EMPTY 0ULL                       /* tag present, empty string (falsy in Python) */
#define XG_KEY_NONE 0xFFFFFFFFFFFFFFFFULL       /* tag absent (has_tag() false)              */
#define XG_KEY_NOMATCH 0xFFFFFFFFFFFFFFFEULL    /* tag present but not a string: equals no barcode */

typedef struct xg_keyspace xg_keyspace;
xg_keyspace *xg_keyspace_create(void);
void xg_keyspace_destroy(xg_keyspace *ks);
uint64_t xg_key_encode(xg_keyspace *ks, const char *s, int64_t len);
/* Writes the string of `key` into buf (no NUL); returns its length, or -1 if unknown. */
int64_t xg_key_decode(xg_keyspace *ks, uint64_t key, char *buf, int64_t cap);
int64_t xg_keyspace_n_interned(xg_keyspace *ks);

/* ---- read records: flat structure-of-arrays -------------------------------------------
 * What pysam exposes per AlignedSegment to the two paths (SURVEY.md A.3), one entry per
 * BAM record that lies on a contig some feature/SNP refers to, in (BAM-list index, file)
 * order -- the order fetch() yields them in (baf first-read-wins needs it, B4/B5).      */
typedef struct {
    int32_t bam_idx;    /* index in the BAM list (= sample column in sample-ID mode)   */
    int32_t gid;        /* caller's contig id (see tid_map of xg_decode_bams)          */
    int64_t rec_beg;    /* records [rec_beg, rec_end) are this BAM's reads on this contig, */
    int64_t rec_end;    /*   sorted by pos (file order)                                */
} xg_run;

#define XG_TILE 1024    /* max records per tile; tiles never straddle runs */
typedef struct {
    int64_t rec_beg;    /* first record of the tile                                    */
    int32_t n_rec;      /* 1..XG_TILE records                                          */
    int32_t run;        /* the run all of them belong to                               */
    int32_t first_pos;  /* pos of the tile's first record                              */
    int32_t max_end;    /* max bam_endpos over the tile's records                      */
} xg_tile;

typedef struct {
    int64_t n_reads;
    int64_t n_cigar;        /* words in `cigar`                                         */
    int64_t n_seq_words;    /* words in `seq` (0 when decoded without sequences)        */
    int32_t n_runs;
    int32_t n_tiles;        /* sum over runs of ceil(run length / XG_TILE)              */
    int32_t max_aln_len;    /* max over reads of sum(M,=,X) -- sizes the include table  */
    int32_t max_span;       /* max over reads of end - pos                              */
    int64_t n_records_seen; /* all BAM records scanned, incl. dropped contigs/unmapped  */
    /* per read */
    const int32_t *pos_end;   /* [2*n] pos (0-based), end = htslib bam_endpos()          */
    const uint32_t *fmq;      /* flag | mapq<<16 | ncw<<24, ncw = CIGAR words stored:    */
                              /*   0 = "simple" read (one M/=/X op of length end-pos,     */
                              /*   nothing stored), 1..254 ops, 255 = true count is in    */
                              /*   the word before cig_off                                */
    const uint32_t *cig_off;  /* [n+1] first CIGAR word of the read in `cigar`; non-       */
                              /*   decreasing; cig_off[n] = n_cigar                         */
    const uint64_t *keys;     /* [2*n] cell key, UMI key (UMI tag, or query name)        */
    const uint32_t *seq_off;  /* first word of the read's 4-bit sequence (NULL if none)  */
    /* streams */
    const uint32_t *cigar;    /* BAM CIGAR words (len<<4|op) of the non-simple reads; a  */
                              /*   record without CIGAR stores one 0-length P op         */
    const uint32_t *seq;      /* BAM 4-bit bases, 8 per word, each read word-aligned;    */
                              /*   byte order as in the BAM record                       */
    const xg_run *runs;
    const xg_tile *tiles;
} xg_reads;

/* BAM header access (replaces pysam.AlignmentFile(fn).references; used by the host side to
 * resolve feature / SNP contig names the way sam_fetch does, xcltk/utils/sam.py:85-118).  */
typedef struct xg_bam_header xg_bam_header;
int xg_bam_header_read(const char *path, xg_bam_header **out);
int32_t xg_bam_header_n_ref(const xg_bam_header *h);
const char *xg_bam_header_ref_name(const xg_bam_header *h, int32_t tid);
int64_t xg_bam_header_ref_len(const xg_bam_header *h, int32_t tid);
void xg_bam_header_free(xg_bam_header *h);

/* Decode BAMs into one xg_reads (replaces pysam.AlignmentFile + AlignedSegment accessors:
 * rdr/fc/core.py:73-76,154; utils/sam.py:21-27; BGZF inflate is multi-threaded).
 *   tid_map[b][tid] = caller's contig id (gid) or -1 to drop the contig's reads;
 *   cell_tag / umi_tag: 2-char tag or NULL; umi_tag NULL => UMI key = query name
 *   (rdr/fc/mcount.py:36-41); want_seq: also emit 4-bit sequences (baf).
 * The result is library-owned (pinned host memory when a CUDA device is present).       */
int xg_decode_bams(int32_t n_bams, const char *const *paths, const int32_t *const *tid_map,
                   const int32_t *tid_map_len, const char *cell_tag, const char *umi_tag,
                   int32_t want_seq, int32_t n_threads, xg_keyspace *ks, xg_reads **out);
void xg_reads_free(xg_reads *r);
const char *xg_host_last_error(void);

/* Matrix-Market text of a CSR result, byte-identical to merge_mtx (rdr/fc/utils.py:54-94):
 * header, "%%", "nrow\tncol\tnnz", then 1-based "row\tcol\tval" lines.  row_ptr spans all
 * n_rows_in input rows; out_row[r] = 1-based output row of input row r, 0 = not emitted (the
 * row must then be empty) -- the renumbering over emitted features of fc_features' emit loop
 * (rdr/fc/core.py:109-124).  Multi-threaded formatting, ordered write.                     */
int xg_write_mtx(const char *path, int32_t n_rows_in, const int64_t *row_ptr, const int32_t *out_row,
                 int32_t n_rows_out, int32_t n_cols, const int32_t *col, const int32_t *val,
                 int32_t n_threads);
/* Same text from rows located by (row_beg, row_cnt) -- the XG_LAYOUT_ROWS layout of xg_coo.  */
int xg_write_mtx_rows(const char *path, int32_t n_rows_in, const int64_t *row_beg, const int32_t *row_cnt,
                      const int32_t *out_row, int32_t n_rows_out, int32_t n_cols, const int32_t *col,
                      const int32_t *val, int32_t n_threads);
/* ... and from the XG_LAYOUT_ROWS_NARROW layout (colval16 + side list of large counts).       */
int xg_write_mtx_rows16(const char *path, int32_t n_rows_in, const int64_t *row_beg, const int32_t *row_cnt,
                        const int32_t *out_row, int32_t n_rows_out, int32_t n_cols, const uint32_t *colval16,
                        int64_t n_over, const int64_t *over_idx, const int32_t *over_val, int32_t n_threads);
/* ... and from the XG_LAYOUT_ROWS_TINY layout (coldelta16 + side list, see xg_coo).           */
int xg_write_mtx_rows_tiny(const char *path, int32_t n_rows_in, const int64_t *row_beg, const int32_t *row_cnt,
                           const int32_t *out_row, int32_t n_rows_out, int32_t n_cols, const uint16_t *coldelta16,
                           int64_t n_over, const int64_t *over_idx, const int32_t *over_col, const int32_t *over_val,
                           int32_t n_threads);

/* ---- device side --------------------------------------------------------------------- */
typedef struct xg_ctx xg_ctx;
typedef struct xg_dreads xg_dreads;      /* read records resident in HBM */

int xg_create(int32_t device, xg_ctx **out);
void xg_destroy(xg_ctx *ctx);
const char *xg_last_error(xg_ctx *ctx);
/* Options: "stream_priority" 1: the context's stream is recreated with the device's greatest
 * priority (a context whose short kernels run beside another context's long ones).            */
int xg_set_option(xg_ctx *ctx, const char *name, int64_t value);

/* Host -> HBM copy of a decoded batch (the only cross-device traffic of the path).      */
int xg_upload_reads(xg_ctx *ctx, const xg_reads *host, xg_dreads **out);
/* Zero-copy variant for the baf pileup: pos/end are copied to HBM, every other array is read
 * by the kernels from the (pinned) host arrays of `host`, which must outlive the result.
 * The pileup touches flag / keys / CIGAR / sequence of the reads that cover a SNP only, so
 * ~8 B per read cross PCIe instead of ~84 B.  XG_E_ARG if the arrays are not pinned.           */
int xg_map_reads(xg_ctx *ctx, const xg_reads *host, xg_dreads **out);
/* Device decoder: BGZF inflate + BAM record parse on the GPU; the compressed files cross PCIe
 * once and the batch is left in HBM, array for array what xg_decode_bams + xg_upload_reads
 * produce.  Replaces pysam.AlignmentFile + fetch() (xcltk/rdr/fc/core.py:75,100;
 * xcltk/baf/fc/core.py:60,99).  Arguments as xg_decode_bams; the files go through the device in
 * windows, so device memory is bounded by a window plus the batch.  Cell / UMI values that do
 * not pack into 63 bits (query names with `--UMItag None`, free-text barcodes, integer tags) are
 * gathered on the device and interned by `ks` on the host; with ks == NULL such input is declined.
 * Returns XG_E_UNSUPPORTED -- and the caller falls back to xg_decode_bams + xg_upload_reads --
 * when a BAM's records cross BGZF block boundaries (htslib-written files never do, unless a
 * record exceeds 64 KiB), for float-typed UMI tags, or when a window or the batch does not fit
 * the device.  n_records_seen may be NULL.                                                    */
int xg_decode_bams_device(xg_ctx *ctx, int32_t n_bams, const char *const *paths,
                          const int32_t *const *tid_map, const int32_t *tid_map_len,
                          const char *cell_tag, const char *umi_tag, int32_t want_seq,
                          xg_keyspace *ks, xg_dreads **out, int64_t *n_records_seen);
/* The same for a byte range of every file: only the BGZF blocks in [range_lo[b], range_hi[b]) of BAM b are inflated
 * and parsed (range_hi[b] = 0: the whole file); both offsets must be block starts (xg_bgzf_block_index) and the block
 * at range_lo[b] must begin with a record (htslib's layout).  This is how one library is split between GPUs: every
 * GPU decodes the blocks of its genomic chunk (+ halo) only.                                              */
int xg_decode_bams_device_range(xg_ctx *ctx, int32_t n_bams, const char *const *paths,
                                const int32_t *const *tid_map, const int32_t *tid_map_len,
                                const char *cell_tag, const char *umi_tag, int32_t want_seq, xg_keyspace *ks,
                                const int64_t *range_lo, const int64_t *range_hi, xg_dreads **out,
                                int64_t *n_records_seen);
/* The same for a list of ranges per file: BAM b decodes the ranges r = range_ptr[b] .. range_ptr[b + 1] - 1, ascending
 * and disjoint.  range_lo[r] is the BGZF virtual offset of the range's first record (block offset << 16 | offset in
 * the inflated block, as a .bai gives it), range_hi[r] the file offset of the block after the range (or the file's
 * end); the walk of the range's first block starts at that record.  An empty list decodes nothing of that BAM,
 * range_ptr = NULL every file whole.  The ranges of a BAM go through one staging / window pipeline one after the
 * other (the bytes between them are never read); runs and the sort check are stitched across them as across windows.
 * *n_records_seen counts the records walked, *bytes_read (may be NULL) the compressed bytes read from the files,
 * headers included.  Records that cross blocks: XG_E_UNSUPPORTED, as for the whole file; so is, when a BAM is read
 * in ranges, a record that does not parse or is out of order (a range that does not start at a record): the caller
 * then decodes the whole files on the host, which reports what is wrong with them.  The ranges come from
 * xg_bam_index_ranges.                                                                                          */
int xg_decode_bams_device_ranges(xg_ctx *ctx, int32_t n_bams, const char *const *paths,
                                 const int32_t *const *tid_map, const int32_t *tid_map_len,
                                 const char *cell_tag, const char *umi_tag, int32_t want_seq, xg_keyspace *ks,
                                 const int64_t *range_ptr, const int64_t *range_lo, const int64_t *range_hi,
                                 xg_dreads **out, int64_t *n_records_seen, int64_t *bytes_read);

/* ---- BAM index (.bai, SAMv1 section 5.2) ---------------------------------------------
 * xg_bam_index_open looks for <bam>.bai, then <bam without .bam>.bai.  Neither there: XG_OK with *out = NULL (the
 * file is read whole; a .csi is not read).  An index that is there but cannot be trusted returns XG_E_FORMAT with the
 * reason in xg_host_last_error(): not a BAI or truncated, n_ref differs from the BAM header, an offset beyond the BAM,
 * older than the BAM.  Release with xg_bam_index_free.                                                          */
typedef struct xg_bam_index xg_bam_index;
int xg_bam_index_open(const char *bam_path, xg_bam_index **out);
void xg_bam_index_free(xg_bam_index *idx);
int32_t xg_bam_index_n_ref(const xg_bam_index *idx);
/* The index of contig tid as read (pointers into idx): n_bins bins ascending (the pseudo-bin left out), the chunks of
 * bin i as (beg, end) virtual-offset pairs chunks[2k], chunks[2k + 1] for k in [bin_ptr[i], bin_ptr[i + 1]), and
 * the n_intv offsets of the 16 kb linear index.                                                                  */
int xg_bam_index_ref(const xg_bam_index *idx, int32_t tid, int64_t *n_bins, const uint32_t **bins,
                     const int64_t **bin_ptr, const uint64_t **chunks, int64_t *n_intv, const uint64_t **linear);
/* The ranges of the BAM that hold every record overlapping one of the n 0-based half-open intervals
 * (tid[i], beg[i], end[i]): the chunks htslib's bam_itr_queryi visits (the bins of reg2bins, less the chunks that end
 * at or before the linear-index offset of the interval's start), merged, then widened to the end of whole BGZF
 * blocks -- a range ends at the block after its last chunk's end -- and merged again when fewer than
 * XG_BAM_INDEX_MERGE_GAP bytes lie between them (reading the gap costs less than one more range).  *ranges: 2 *
 * *n_ranges entries lo, hi, ascending, lo the virtual offset of the range's first record, hi a file offset (release
 * with xg_free_array); the form xg_decode_bams_device_ranges takes.  Unknown tids and empty intervals add nothing.
 * XG_E_FORMAT when an offset is not a BGZF block start of the BAM or lies beyond its block (an index of another
 * file): the caller then reads the file whole.                                                                   */
#define XG_BAM_INDEX_MERGE_GAP (256 << 10)
int xg_bam_index_ranges(const xg_bam_index *idx, int64_t n, const int32_t *tid, const int64_t *beg, const int64_t *end,
                        int64_t **ranges, int64_t *n_ranges);

/* Host helpers for choosing the ranges (what the .bai linear index gives pysam's fetch, computed from the file):
 * offsets of all BGZF blocks (n + 1 entries, the last = file size; release with xg_free_array), the block in which
 * the first record starts (*aligned = 1: exactly at its beginning, as htslib writes), and the (tid, pos) of the
 * record at the beginning of the block at `offset` (tid -2: empty / too short a block).                       */
int xg_bgzf_block_index(const char *path, int64_t **offsets, int64_t *n_blocks, int64_t *first_record_block,
                        int32_t *aligned);
void xg_free_array(void *p);
int xg_bam_block_probe(const char *path, int64_t offset, int32_t *tid, int32_t *pos);

/* Validation entry: inflate a whole BGZF file on the device into out[0, cap).  With out == NULL
 * (or cap too small) only *n_out, the inflated size, is set.                               */
int xg_bgzf_inflate_device(xg_ctx *ctx, const char *path, uint8_t *out, int64_t cap, int64_t *n_out);
/* HBM -> host copy (tests: run the oracle on device-generated records).                 */
int xg_download_reads(xg_ctx *ctx, const xg_dreads *d, xg_reads **out);
void xg_dreads_free(xg_ctx *ctx, xg_dreads *d);
int64_t xg_dreads_n(const xg_dreads *d);
/* out[0..7] = n_reads, n_cigar, n_seq_words, n_runs, n_tiles, max_aln_len, max_span, bytes in HBM */
void xg_dreads_info(const xg_dreads *d, int64_t out[8]);
/* Host copies of the batch's run and tile index (n_runs / n_tiles entries; either may be NULL). */
void xg_dreads_index(const xg_dreads *d, xg_run *runs_out, xg_tile *tiles_out);

/* Read filters = check_read(), rdr/fc/core.py:46-62 == baf/fc/core.py:18-34.            */
typedef struct {
    int32_t min_mapq;      /* ceil(conf.min_mapq): mapq < x  <=>  mapq < ceil(x)          */
    int32_t min_len;       /* len(read.positions) >= min_len                              */
    uint32_t incl_flag;    /* 0 disables                                                  */
    uint32_t excl_flag;    /* 0 disables                                                  */
    int32_t no_orphan;     /* drop PAIRED & !PROPER_PAIR                                  */
    int32_t use_cell_tag;  /* barcode mode: cell key must be present and listed           */
    int32_t need_umi_tag;  /* conf.umi_tag set: has_tag(umi) required                     */
    /* include test, rdr/fc/core.py:160-165 (basefc only):
     * keep iff m >= min_incl_tab[n] (n = aligned length) when the table is given
     * (fraction mode; built by the caller with the reference's own float expression),
     * else iff m >= min_incl_len.                                                        */
    const int32_t *min_incl_tab;
    int32_t min_incl_tab_len;
    int32_t min_incl_len;
} xg_params;

/* Features (basefc) / regions (baf): 0-based half-open [beg, end) on contig gid,
 * gid < 0 or end <= beg => never fetched (unknown contig, start <= 0: utils/sam.py:105-118). */
typedef struct {
    int32_t n;
    const int32_t *gid;
    const int32_t *beg;
    const int32_t *end;
} xg_features;

/* Cell barcodes (barcode mode): keys of conf.samples in column order; n = 0 => sample-ID
 * mode, column = xg_run.bam_idx (rdr/fc/core.py:166-170).                                */
typedef struct {
    int32_t n;
    const uint64_t *keys;
    int32_t n_samples;     /* number of columns (= n in barcode mode, #BAMs otherwise)    */
} xg_barcodes;

/* Sparse result, 0-based; library-owned pinned host memory, valid until xg_coo_free() (which
 * must be called before the context is destroyed).  The layout is chosen by the `layout` argument
 * of xg_basefc / xg_basefc_host; every other entry point returns XG_LAYOUT_CSR.              */
#define XG_LAYOUT_CSR 0         /* sorted by (row, col): row_ptr, col, val                             */
#define XG_LAYOUT_ROWS 1        /* rows in the order the device completed them -- each row contiguous and
                                 * sorted by col -- located by row_beg / row_cnt, entries in col / val;
                                 * copied to the host while the later reads are still being counted   */
#define XG_LAYOUT_ROWS_NARROW 2 /* the same, entries in colval16; with more than 65536 columns, or too
                                 * many large counts for the side list, the call returns XG_LAYOUT_ROWS */
#define XG_LAYOUT_ROWS_TINY 3   /* the same, entries in coldelta16; with too many entries for the side
                                 * list the call returns XG_LAYOUT_ROWS                                */
typedef struct {
    int64_t nnz;
    int32_t n_rows, n_cols;
    const int32_t *col;       /* NULL in the packed layouts */
    const int32_t *val;
    const int64_t *row_ptr;   /* XG_LAYOUT_CSR: CSR offsets, n_rows + 1; else NULL */
    const int64_t *row_beg;   /* rows layouts: first entry of every row, n_rows; else NULL */
    const int32_t *row_cnt;   /* rows layouts: entries of every row, n_rows; else NULL */
    /* XG_LAYOUT_ROWS_NARROW: entry k is colval16[k] = column | count << 16; a count field of 65535 means
     * "look entry k up in the side list" (over_idx ascending is not guaranteed; n_over entries).  Half the
     * bytes per entry.                                                                                  */
    const uint32_t *colval16;
    int64_t n_over;
    const int64_t *over_idx;
    const int32_t *over_val;
    /* XG_LAYOUT_ROWS_TINY: entry k is the 16-bit word
     * coldelta16[k] = (column - previous column of the row - 1) << 4 | count  (count 1..15, gap <= 4095 columns);
     * the word 0 means "look entry k up in the side list": over_idx / over_col / over_val, n_over entries in no
     * particular order -- always the first entry of a row, else entries whose gap or count does not fit.
     * A quarter of the bytes of (col, val): the result copy is what a host shared by several GPUs runs out of. */
    const uint16_t *coldelta16;
    const int32_t *over_col;
} xg_coo;
void xg_coo_free(xg_coo *m);

/* basefc (needs a batch from xg_upload_reads, not xg_map_reads): replaces the per-feature loop fc_features()/fc_fet1() (rdr/fc/core.py:96-124,151-178)
 * and MCount/SCount (rdr/fc/mcount.py): out[row f, col c] = number of distinct UMI keys among
 * the reads of cell c that overlap feature f and pass check_read + the include test.
 * layout: one of XG_LAYOUT_*, the layout of *out (see xg_coo).                              */
int xg_basefc(xg_ctx *ctx, const xg_dreads *reads, const xg_features *feats,
              const xg_barcodes *cells, const xg_params *par, int32_t layout, xg_coo **out);

/* Same from a pinned host batch (xg_decode_bams output): the records are copied to HBM epoch
 * by epoch on a copy stream while the previous epochs are being counted, so that the call
 * costs about max(H2D, kernels) instead of their sum.  This is the end-to-end entry point. */
int xg_basefc_host(xg_ctx *ctx, const xg_reads *host, const xg_features *feats,
                   const xg_barcodes *cells, const xg_params *par, int32_t layout, xg_coo **out);
/* Matrix-Market text written on the device (SURVEY.md 8f N2; replaces merge_mtx, rdr/fc/utils.py:54-94): when the LAST
 * xg_basefc call of this context produced a rows layout, its rows are still in its staging area; they are formatted
 * there (one warp per row, rows placed in input order by a scan) and the text leaves through pinned buffers that writer threads pwrite() in parallel.  The same bytes as the
 * writers above (out_row[r]: 1-based output row of input row r, 0 = not emitted; n_rows_in = rows of that call). */
int xg_basefc_write_mtx_device(xg_ctx *ctx, const char *path, int32_t n_rows_in, const int32_t *out_row,
                               int32_t n_rows_out, int32_t n_threads);
/* Read-assignment summary of basefc (what htseq-count's special counters and featureCounts' .summary report; the
 * reference has no counterpart).  It counts RECORDS, not UMIs: a record is in range iff it overlaps some feature that
 * fetch() would query (gid >= 0, beg >= 0, end > beg) with sam.fetch's rule pos < end && bam_endpos > beg
 * (utils/sam.py:85-118); records in range of no feature are not counted (the reference never sees them).  Row: the
 * column of the record's cell key if that key is listed, else row n_samples ("__no_cell": tag missing or barcode not
 * listed); sample-ID mode: the BAM's column (row n_samples stays 0).  Fate: the first that applies, in check_read's
 * order (rdr/fc/core.py:46-62) --
 *   0 mapq < min_mapq   1 excl_flag hit, incl_flag missed or orphan   2 need_umi_tag and the UMI tag missing or
 *   empty (such a record never reaches the matrix)   3 aligned length < min_len   then the include test
 *   (rdr/fc/core.py:160-165, as xg_basefc applies it) for every feature the record overlaps:
 *   4 fails for all   5 passes for exactly one   6 passes for two or more (counted once in each, SURVEY.md A.1 R9).
 * out: (n_samples + 1) x 7 counters, row-major.  own: NULL, or the half-open range [(own[0], own[1]), (own[2],
 * own[3])) of record start keys (gid, pos) that the call counts (one library split between GPUs: every record is
 * counted by the GPU whose cut holds its start).  Works on batches from xg_upload_reads, the device decoder and
 * xg_map_reads (flags, keys and CIGAR are read for the records in range only); XG_E_ARG when keys are not 16-byte,
 * pos_end not 8-byte or the other record arrays not 4-byte aligned.  Uses the interval index of the
 * context's last xg_basefc call when the features are the same; never touches the staging area that
 * xg_basefc_write_mtx_device formats.  xg_last_timing: [0] / [1] the kernel (ms)  [2] launches  [12] host ms. */
int xg_basefc_summary(xg_ctx *ctx, const xg_dreads *reads, const xg_features *feats, const xg_barcodes *cells,
                      const xg_params *par, const int32_t *own, int64_t *out);

/* baf phase 1: replaces plp_snp() up to mcnt.stat() (baf/fc/core.py:198-237; first-read-wins
 * per (SNP, cell, UMI): baf/fc/mcount.py:109-127; allele: :39-60 + utils/sam.py:4-40).
 * totals[5*i .. 5*i+4] = A,C,G,T,N bucket counts of SNP i over all listed cells.          */
typedef struct {
    int32_t n;
    const int32_t *gid;
    const int32_t *pos;        /* 0-based */
} xg_snps;
typedef struct xg_baf_state xg_baf_state;
int xg_baf_pileup(xg_ctx *ctx, const xg_dreads *reads, const xg_snps *snps,
                  const xg_barcodes *cells, const xg_params *par,
                  int64_t *totals /* may be NULL: not copied out */, xg_baf_state **state);
/* baf phase 2: replaces fc_fet1() aggregation + emit (baf/fc/core.py:143-194, 84-113).
 *   hap_of[8*i + code] for SNP i and base code (0..4 = A,C,G,T,N; 5 = other / IUPAC) is the
 *   region haplotype index 0 / 1, or 2 for "other allele", as SNP.get_region_allele_index
 *   gives (baf/fc/gfeature.py:38-39); keep[i] = 0 drops the SNP (plp_snp filter :238-246,
 *   evaluated by the caller in Python for float exactness);
 *   region r's SNPs are reg_snp[reg_ptr[r] .. reg_ptr[r+1]).
 * Outputs AD / DP / OTH as in fc_features' emit loop (rows = regions, cols = cells).      */
int xg_baf_count(xg_ctx *ctx, xg_baf_state *state, int32_t n_regions, const int64_t *reg_ptr,
                 const int32_t *reg_snp, const uint8_t *hap_of, const uint8_t *keep,
                 int32_t no_dup_hap, xg_coo **ad, xg_coo **dp, xg_coo **oth);
void xg_baf_state_free(xg_ctx *ctx, xg_baf_state *state);
/* baf, one call: xg_baf_pileup -> plp_snp's SNP filter ON THE DEVICE -> xg_baf_count; what one fc_features worker
 * of the reference does for its regions (baf/fc/core.py:42-247).  The filter (baf/fc/core.py:238-246): SNP i is
 * skipped iff  sum(tcount) < min_count  or  min(tcount[ref_idx[i]], tcount[alt_idx[i]]) < sum(tcount) * min_maf,
 * evaluated in IEEE double exactly as Python evaluates int-with-float (counts < 2^53); ref_idx / alt_idx are
 * MCount.base_idx of the SNP's alleles (0..4 = A,C,G,T,N; baf/fc/mcount.py:178).  The per-SNP totals never leave
 * the device unless `totals` (n_snps x 5 int64) is given; `keep_out` (n_snps bytes) receives the filter if given.
 * Same results as the three-step sequence with the filter evaluated by the caller; two host synchronisations
 * and 8 MB of D2H less per call.                                                                             */
typedef struct {
    const uint8_t *ref_idx, *alt_idx;
    double min_count, min_maf;
} xg_snp_filter;
int xg_baf_fc(xg_ctx *ctx, const xg_dreads *reads, const xg_snps *snps, const xg_barcodes *cells,
              const xg_params *par, const xg_snp_filter *filt, int32_t n_regions, const int64_t *reg_ptr,
              const int32_t *reg_snp, const uint8_t *hap_of, int32_t no_dup_hap, int64_t *totals,
              uint8_t *keep_out, xg_coo **ad, xg_coo **dp, xg_coo **oth);
/* SNP-level allele counting: the per-SNP x cell counts of the candidate SNPs themselves (what cellsnp-lite's
 * cellSNP.tag.{AD,DP,OTH}.mtx hold), with the pileup of plp_snp (baf/fc/core.py:198-247; first read wins per
 * (SNP, cell, UMI), a None allele included: baf/fc/mcount.py:39-60,109-150) and its filter as in xg_baf_fc.  Each SNP
 * counts as a region of one SNP with GT 0|1 (baf/fc/core.py:143-194): over the winning UMIs of SNP i in cell c whose
 * allele is not None,  AD = UMIs whose base is the ALT (base index alt_idx[i]),  DP = UMIs whose base is REF or ALT,
 * OTH = the others (IUPAC codes and '=' match neither; REF == ALT counts as ALT).  Rows are all snps->n SNPs in
 * input order -- a SNP removed by the filter has empty rows, keep_out reports it -- columns cells->n_samples
 * (< 2^24, else XG_E_LIMIT); XG_LAYOUT_CSR.  Works on batches from xg_upload_reads, the device decoder and
 * xg_map_reads.  xg_last_timing: [0] device span  [1] scan  [2] launches  [4] result D2H  [6] (read, SNP) pairs
 * [7] winners reduced  [8..10] host milestones (ms since entry: pileup, kernels queued, end)
 * [14] / [15] SNPs reduced by one warp / by a whole CTA.                                                      */
int xg_snp_pileup(xg_ctx *ctx, const xg_dreads *reads, const xg_snps *snps, const xg_barcodes *cells,
                  const xg_params *par, const xg_snp_filter *filt, int64_t *totals /* may be NULL */,
                  uint8_t *keep_out /* may be NULL */, xg_coo **ad, xg_coo **dp, xg_coo **oth);

/* SNP discovery (cellsnp-lite's mode without a candidate list; the reference has no such mode): every 0-based
 * position p in [beg, end) of every target (targets->n entries {gid, beg, end}; gid < 0 or end <= beg: skipped;
 * targets of one contig must not overlap, else XG_E_ARG) is a possible site.  Its totals are exactly plp_snp's for a
 * SNP at p (baf/fc/core.py:198-247), i.e. what xg_baf_pileup writes: check_read, a listed cell (or the BAM's column in
 * sample mode), a UMI key, the first read per (cell, UMI) in file order wins even when its allele is None, and the
 * winners with an allele count into A / C / G / T / N.  REF is the A..T bucket with the largest count, ALT the one
 * with the second largest (ties to the lower index in A < C < G < T; N is never REF or ALT).  A site is kept iff
 * ALT >= 1, sum >= min_count and ALT >= sum * min_maf (plp_snp's filter, baf/fc/core.py:238-246, in IEEE double).
 * The reads' aligned bases are first counted per position without the UMI collapse; positions whose raw counts
 * cannot pass (raw sum < min_count, or fewer than two A..T buckets with max(1, min_count * min_maf) bases) are
 * dropped, the others go through xg_baf_pileup (in slices when one slice exceeds its limits) and the filter.
 * *out: the kept sites in target order, then by position, with their totals (n x 5: A C G T N) and the allele
 * indices (0..3 = A C G T); library-owned host memory, release with xg_sites_free.
 * xg_last_timing: [0] device span  [1] raw scan  [2] launches  [3] exact stage  [5] windows with reads
 * [6] positions scanned (the positions of those windows)  [7] raw candidates  [11] pileup slices
 * [12] host ms of the call  [13] (read, window) entries  [14] kept sites.
 * xg_set_option(ctx, "discover_slice", n): at most n candidates per pileup slice (0: the default, 2^22).        */
typedef struct {
    double min_count, min_maf;
} xg_discover_filter;
typedef struct {
    int64_t n;
    const int32_t *gid;
    const int32_t *pos;        /* 0-based */
    const uint8_t *ref;
    const uint8_t *alt;
    const int64_t *totals;     /* n x 5 */
} xg_sites;
int xg_snp_discover(xg_ctx *ctx, const xg_dreads *reads, const xg_features *targets, const xg_barcodes *cells,
                    const xg_params *par, const xg_discover_filter *filter, xg_sites **out);
void xg_sites_free(xg_sites *sites);

/* Local phasing of long regions (the pre-step of `xcltk baf`; xcltk/baf/fc/phasing.py:13-78 over
 * xcltk/baf/localphase.py:14-243, as xcltk_b200/baf/fc/phasing.py:reg_local_phasing and baf/localphase.py compute it
 * region by region on the host).  Per region, one CTA: the SNPs with no depth leave the region's list (keep_out), the
 * counts are oriented by ref_idx (1: DP - AD), then up to 50 rounds of {cells with aggregated BAF in [0.45, 0.55]
 * leave; two-component EM (min 10, max 1000 iterations, convergence 1e-3) with the posteriors smoothed by the
 * row-normalised kernel exp(-(x_j - x_i)^2 / 20000^2); flip = Z1 >= Z0; re-orient} until a round after the fifth
 * flips all or none.  A round in which the live cells give some SNP no depth makes the reference's EM all NaN: it
 * flips nothing.  No live cell left: the region failed (status 0), nothing flips.  Otherwise (status 1) the final
 * flips are inverted when more than half flip, written to flip_out and applied to ref_idx (in/out, 0 / 1 per SNP).
 * Status 2: as 1, but some flip (|Z1 - Z0| < 1e-6) or convergence test (|dll - 1e-3| < 1e-9 max(1, |ll|)) was a
 * tie that the reference's own rounding decides; the caller re-decides the region and reruns the later waves.
 * Regions arrive in wave order (wave_ptr): regions of one wave share no SNP, and a region reads ref_idx as the
 * earlier waves left it; the waves run in order on the context's stream without a host synchronisation.
 * Entries are the (SNP slot, cell) pairs with DP > 0 of each region, given SNP-major (slot_ent_ptr: per slot, local
 * cell id, AD = UMIs with ALT, DP = UMIs with REF or ALT) and cell-major (cell_ent_ptr: per local cell, local SNP
 * index in the region's list) -- the same entries of region r in both.  FP64, fixed summation order: the same
 * input gives the same bytes.  xg_last_timing: [0] device span  [1] EM kernels  [2] waves  [3] regions
 * [4] inner EM iterations  [5] longest region (ms, one CTA)  [6] its share of [1]  [7] entries  [8] status-2
 * regions  [12] host ms.                                                                                        */
typedef struct {
    int32_t n_regions, n_waves;
    const int32_t *wave_ptr;        /* n_waves + 1: regions of wave w are [wave_ptr[w], wave_ptr[w + 1])     */
    const int64_t *reg_snp_ptr;     /* n_regions + 1: SNP slots of region r                                 */
    const int32_t *reg_snp;         /* per slot: SNP index (< n_snps), the region's order (sorted by position) */
    const int64_t *slot_ent_ptr;    /* slots + 1: SNP-major entries of each slot                             */
    const int32_t *sm_cell, *sm_ad, *sm_dp;
    const int64_t *reg_cell_ptr;    /* n_regions + 1: local cells of region r                               */
    const int64_t *cell_ent_ptr;    /* cells + 1: cell-major entries of each local cell                      */
    const int32_t *cm_snp, *cm_ad, *cm_dp;
} xg_phase_regions;
int xg_local_phase(xg_ctx *ctx, int32_t n_snps, const int32_t *snp_pos, uint8_t *ref_idx, const xg_phase_regions *regs,
                   uint8_t *keep_out /* per slot */, uint8_t *flip_out /* per slot */, int8_t *status_out /* per region */);

/* Synthetic 10x-style records generated directly in HBM (bench / tests; no reference
 * counterpart -- SURVEY.md 8(d) C3 allows device-side generation for kernel-only runs).  */
typedef struct {
    int64_t n_reads;
    int32_t n_cells;          /* listed barcodes; 5% of molecules carry an unlisted one   */
    int32_t read_len;
    int32_t want_seq;
    uint64_t seed;
    /* reads are spread uniformly over the union of these spans (sorted, disjoint), per contig */
    int32_t n_spans;
    const int32_t *span_gid;
    const int32_t *span_beg;
    const int32_t *span_end;
    /* optional SNP table so that bases at SNPs are haplotype consistent */
    int32_t n_snps;
    const int32_t *snp_gid;
    const int32_t *snp_pos;
    const uint8_t *snp_ref;   /* base codes 0..3 */
    const uint8_t *snp_alt;
    const uint8_t *snp_ref_hap;
    /* total_reads > 0: generate only reads [first_read, first_read + n_reads) of a library of total_reads
     * (every field of read i depends on i, seed and the library size only), so that several GPUs can each
     * hold one genomic chunk of ONE library                                                   */
    int64_t first_read;
    int64_t total_reads;
    /* pseudo_ref != 0: aligned bases away from the SNP table are a seeded pseudo-reference base of (gid, pos), each
     * replaced by one of the other three bases with probability ref_error (so that SNP discovery has a background
     * to find sites in); 0: pseudo-random bases, as without these fields                                       */
    int32_t pseudo_ref;
    double ref_error;
} xg_synth_params;
int xg_synth_reads(xg_ctx *ctx, const xg_synth_params *p, xg_dreads **out, uint64_t *barcode_keys);
/* Index of the first read at or after (gid, pos) in the library of p->n_reads reads (host only). */
int64_t xg_synth_read_index(const xg_synth_params *p, int32_t gid, int32_t pos);

/* The inverse of the decoders (bench / tests; no reference counterpart): a coordinate-sorted, htslib-layout BAM
 * holding exactly the records of `reads` (one BAM, runs in contig order; contig gid becomes tid gid): pos, flag, mapq,
 * CIGAR, the 4-bit sequence if the batch has one (else pseudo-random bases of the right length), CB / UB tags
 * spelled from the keys (cell_tag / umi_tag NULL: not written), query name "r<index>" or -- name_from_umi -- the
 * UMI key's text (records of a molecule then share their name, like mates).  Host only.                   */
int xg_write_bam(const char *path, const xg_reads *reads, int32_t n_gid, const char *const *gid_names,
                 const int64_t *gid_lens, xg_keyspace *ks, const char *cell_tag, const char *umi_tag,
                 int32_t name_from_umi, int32_t level, int32_t n_threads);

/* Timing of the last xg_basefc / xg_baf_* call (CUDA events on the library's streams, ms):
 * [0] device span of the call  [1] sum of the dominant counting kernel's launches
 * [2] kernel launches          [3] span of the epoch loop + gather (basefc)
 * [4] result D2H               [5] epochs (basefc)   [6] pool bytes / pairs   [7] staging entries
 * [8..11] host phases of xg_basefc (ms): index build; windows and epoch plan (device kernels) until the plan's
 * summary is back; allocation of the pool and the staging area; uploads (filters, barcode table); [12] whole call;
 * [13] bytes copied host -> device (xg_basefc_host); [14] / [15] features counted in segments / in sets.
 * xg_baf_*: [8..10] host milestones of the call (ms since entry).                                   */
void xg_last_timing(xg_ctx *ctx, double out[16]);
/* Route counters of the segment finalize in the last xg_basefc / xg_basefc_host call: [0..3] ordinary CTAs,
 * [4..7] big CTAs, each {heavy features, careful column ranges, fast ranges that overflowed, sub-partition doublings}. */
int xg_basefc_finalize_stats(xg_ctx *ctx, int64_t out[8]);

const char *xg_version(void);

#ifdef __cplusplus
}
#endif
#endif
