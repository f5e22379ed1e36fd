/* breakmer_b200 -- C ABI of the B200-native BreaKmer k-mer assembly hot path.
 *
 * The reference (ccgd-profile/BreaKmer) has no FFI: its boundary for this path is
 * a set of plain Python call sites (SURVEY.md section 8.3).  Each entry point
 * below names the reference interface it stands in for; the Python shims in
 * breakmer_b200/ (olc.py, utils.py, sv_assembly.py, sv_processor.py) keep the
 * reference's function names and argument meaning and call these through ctypes.
 *
 * Conventions
 *   - plain pointers and sizes; no torch / CUDA types in any signature;
 *   - inputs are caller-owned HOST buffers; they are copied to the device inside
 *     the call (the *_dev timing entry points are the only exception);
 *   - outputs returned through `const T**` live in library-owned pinned host
 *     arenas and stay valid until the next call on the same handle or
 *     bk_destroy; outputs passed as plain `T*` are caller-owned buffers;
 *   - every function returns 0 on success or a negative BK_ERR_* code, and
 *     bk_last_error(h) gives the message;
 *   - one handle = one CUDA device + one stream; calls on one handle must not
 *     overlap; distinct handles may be used from distinct host threads
 *     (one handle per GPU is the multi-GPU model: regions are sharded by the
 *     caller, there is no collective).
 *   - sequences are ASCII; A/C/G/T (either case for counting) are bases, any
 *     other byte behaves like 'N'.
 */
#ifndef BREAKMER_B200_H
#define BREAKMER_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BK_OK 0
#define BK_ERR_CUDA (-1)
#define BK_ERR_ARG (-2)
#define BK_ERR_NOMEM (-3)
#define BK_ERR_CAPACITY (-4)  /* a device-side hard limit is exceeded (a read or contig above 4095 bases inside the
                                  batched assembler of bk_compare_kmers_batch, above 65535 bases in that of
                                  bk_compare_kmers_long; bk_nw_batch itself has no length limit) */
#define BK_ERR_EMPTY_SEQ (-5) /* olc.nw raises NameError on an empty sequence (olc.py:86-87) */
#define BK_ERR_FORMAT (-6)    /* malformed FASTQ record (FastqFile raises, utils.py:704-719) */
#define BK_ERR_IO (-7)        /* an input file cannot be read */

typedef struct bk_handle_s* bk_handle_t;

int bk_version(void);
int bk_device_count(void);
int bk_create(int device, bk_handle_t* out);
int bk_destroy(bk_handle_t h);
const char* bk_last_error(bk_handle_t h);

/* ---- olc.nw (olc.py:40-107; call sites sv_assembly.py:451-452) ----------------
 * For pair p: seq1 = sequence pair_a[p], seq2 = sequence pair_b[p] of the
 * concatenated `seqs` (seq_off has n_seq+1 entries).
 * out[p*10 + 0..4] = fields [2:7] of nw(seq1, seq2): prej, j, prei, i, max_i
 * out[p*10 + 5..9] = the same five fields of nw(seq2, seq1) (computed in the same
 *                    sweep; check_align always needs both).
 * If want_aln != 0, align1/align2 of nw(seq1, seq2) (tuple fields [0:2]) are
 * written to aln1/aln2 at aln_off[p] (capacity len(seq1)+len(seq2) each) and
 * their common length to aln_len[p].
 * Like olc.nw (olc.py:40-52) the call has no length limit: pairs with a sequence above 4095 bases
 * (the packed-cell warp kernels' range) are run by a 32-bit anti-diagonal kernel, one thread block
 * per direction (csrc/nw_long.cuh); memory is O(m+n) per pair, (m+1)(n+1) bytes more with want_aln. */
int bk_nw_batch(bk_handle_t h, const char* seqs, const int64_t* seq_off, int64_t n_seq,
                const int32_t* pair_a, const int32_t* pair_b, int64_t n_pairs, int32_t* out,
                int want_aln, char* aln1, char* aln2, const int64_t* aln_off, int32_t* aln_len);

/* ---- read redundancy (SURVEY.md section 8.7 f.4; sv_assembly_mm2.py:64-94, 290-355) ----------
 * read_batch.check_mer_read (call site: contig.check_read, sv_assembly_mm2.py:478) for whole
 * batches.  Batch b = reads batch_off[b] .. batch_off[b+1]-1 of the concatenated `seqs`, in the
 * order the assembler meets them; its first read opens the batch (read_batch.__init__, :290-294);
 * mer_pos[r] = offset of the seed k-mer in read r (the `pos` argument of check_mer_read).
 * subseq_frac = the subseq() identity threshold (0.90 in sv_assembly_mm2.py:77, 0.85 in
 * sv_assembly.py:80).  The alignments the decision chains need are computed ahead of the decisions
 * for all batches together (every read against its 4 predecessors in one olc.nw launch; a further
 * launch per round for chains that dropped more reads in a row), and the chains are replayed on the
 * host.  Outputs (caller-owned, n_reads bytes each): check[r] = what check_mer_read returned for
 * read r (1 for an opener); flags[r] = BK_DEDUP_ADDED (1, appended to batch_reads) |
 * BK_DEDUP_REDUNDANT (2, b_read.redundant) | BK_DEDUP_DELETED (4, id in read_batch.delete).
 * n_pairs_out / n_launches_out (optional) = alignments computed (each one sweep that yields both
 * directions) and kernel launches made.  An empty sequence in a batch of two or more reads ->
 * BK_ERR_EMPTY_SEQ (olc.nw raises NameError). */
#define BK_DEDUP_ADDED 1
#define BK_DEDUP_REDUNDANT 2
#define BK_DEDUP_DELETED 4
int bk_dedup_reads(bk_handle_t h, const char* seqs, const int64_t* seq_off, int64_t n_reads, const int32_t* mer_pos,
                   const int64_t* batch_off, int64_t n_batches, double subseq_frac, uint8_t* check, uint8_t* flags,
                   int64_t* n_pairs_out, int32_t* n_launches_out);

/* ---- run_jellyfish + load_kmers (utils.py:151-179, 287-297) --------------------
 * Strand-specific k-mer occurrence counts over n_rec records (`bases`
 * concatenated, rec_off has n_rec+1 entries, rec_mult optional per-record
 * multiplicity).  Returns the distinct k-mers in ascending 2-bit code order
 * (A<C<G<T, first base most significant) with their counts.  1 <= k <= 31. */
int bk_count_kmers(bk_handle_t h, const char* bases, const int64_t* rec_off, int64_t n_rec,
                   const uint32_t* rec_mult, int k,
                   const uint64_t** mers, const uint32_t** counts, int64_t* n_out);

/* ---- the set algebra of target.compare_kmers (sv_processor.py:621-622, 630-631)
 * plus normal-sample subtraction (SURVEY.md K4).  Inputs are sorted unique k-mer
 * arrays as bk_count_kmers returns them; normal may be null/0.
 * Result: sample_only = (case & case_sc) - ref - normal, counts taken from case. */
int bk_sample_only(bk_handle_t h, int k,
                   const uint64_t* case_mers, const uint32_t* case_counts, int64_t n_case,
                   const uint64_t* sc_mers, int64_t n_sc,
                   const uint64_t* ref_mers, int64_t n_ref,
                   const uint64_t* normal_mers, int64_t n_normal,
                   const uint64_t** mers, const uint32_t** counts, int64_t* n_out);

/* ---- the whole hot path for a batch of target regions -----------------------------
 * target.compare_kmers (sv_processor.py:609-645) for n_regions targets at once:
 * k-mer counting of the four inputs, sample-only selection, grouping of identical
 * reads (utils.py:239-244), and init_assembly (sv_assembly.py:30-63).
 *
 * Per-region record ranges: region r owns records [x_reg_off[r], x_reg_off[r+1]).
 * read_flags[i] bit0 = fq_read.indel_only of record i.
 * If have_mers != 0 the k-mer stage is skipped and in_mers/in_counts/in_mers_off
 * give each region's sample-only k-mers (ascending) -- this is the shape of
 * init_assembly(mers, fq_recs, kmer_len, rc_thresh, read_len) itself.
 * read_len may be null (then max record length per region, utils.py:236). */
typedef struct bk_batch_input {
  int32_t n_regions;
  int32_t k;
  int32_t rc_thresh;
  int32_t have_mers;
  const char* ref_bases;   const int64_t* ref_off;                         /* n_regions+1 */
  const char* read_bases;  const int64_t* read_off;  const int64_t* read_reg_off;  const uint8_t* read_flags;
  const char* sc_bases;    const int64_t* sc_off;    const int64_t* sc_reg_off;
  const char* normal_bases; const int64_t* normal_off; const int64_t* normal_reg_off;   /* optional */
  const uint64_t* in_mers; const uint32_t* in_counts; const int64_t* in_mers_off;      /* have_mers */
  const int32_t* read_len;                                                             /* optional */
} bk_batch_input;

/* All arrays are library-owned (valid until the next call on the handle).
 * Contig c of region r: c in [ctg_reg_off[r], ctg_reg_off[r+1]), acceptance order.
 * Each ctg_*_off table holds an (offset, length) PAIR per contig: X_off[2c] is the
 * start in the payload array(s), X_off[2c+1] the element count (payload arrays are
 * in device completion order, only these tables are ordered).
 *   sequence       ctg_seq[off .. off+len)          via ctg_seq_off
 *   kmer_locs      ctg_kmer_locs[off .. off+len)    via ctg_seq_off, one int per base
 *   count vectors  ctg_indel_only / ctg_others      via ctg_cnt_off (their length can
 *                  differ from the sequence length, SURVEY Q17)
 *   reads          ctg_reads                        via ctg_reads_off = record index
 *                  (into the input read arrays) of the representative (first) record
 *                  of each unique read in contig.reads
 *   k-mer tuples   ctg_kmer_mer/pos/lth/dist/order  via ctg_kmers_off ; order
 *                  0='for' 1='rev' 2='mid' (sv_assembly.py:130,142)
 * With the "rejected_contigs" option the ctg_*_off tables also hold, after the n_contigs
 * accepted contigs, those the acceptance test dropped (bk_rejected_contigs).
 * Unique reads (fq_recs keys, insertion order): region r owns
 * [uniq_reg_off[r], uniq_reg_off[r+1]); uniq_rec = representative record index,
 * uniq_mult = len(fq_recs[seq]). */
typedef struct bk_batch_result {
  int32_t n_regions;
  int64_t n_contigs;
  const int64_t* so_off;  const uint64_t* so_mers;  const uint32_t* so_counts;
  const int64_t* uniq_reg_off; const int32_t* uniq_rec; const uint32_t* uniq_mult;
  const int64_t* ctg_reg_off;
  const int64_t* ctg_seq_off;   const char* ctg_seq;   const int32_t* ctg_kmer_locs;
  const int64_t* ctg_cnt_off;   const int32_t* ctg_indel_only; const int32_t* ctg_others;
  const int64_t* ctg_reads_off; const int32_t* ctg_reads;
  const int64_t* ctg_kmers_off; const uint64_t* ctg_kmer_mer; const int32_t* ctg_kmer_pos;
  const int32_t* ctg_kmer_lth;  const int32_t* ctg_kmer_dist; const int32_t* ctg_kmer_order;
  const int32_t* region_status;      /* 0 or BK_ERR_CAPACITY per region (the cause: bk_region_report) */
  /* work counters of this call (for roofline arithmetic) */
  int64_t n_check_align;             /* contig.check_align calls (each = two olc.nw) */
  int64_t n_dp_cells;                /* sum over those of len(contig)*len(read) (one sweep each).  With the
                                        "long_regions" option both count all device work of the call, including the
                                        abandoned first attempt of a region the long assembler took over */
  int64_t n_kmer_occurrences;        /* k-mer windows of all inputs (reference forward + reverse, reads, soft clips, normal) */
  double  gpu_ms;                    /* device time of the call, CUDA events */
  int64_t n_sorted_keys;             /* windows that went through the sort (the sample's; the rest are streamed past) */
  const int64_t* region_dp_cells;    /* per region: its share of n_dp_cells (cost models for sharding, shard.py); with
                                        "long_regions", that of the pass that produced the region's result */
  double host_wait_ms;               /* bk_batch_wait: time blocked on the device ... */
  double host_post_ms;               /* ... and time spent building the result tables on the host */
} bk_batch_result;

int bk_compare_kmers_batch(bk_handle_t h, const bk_batch_input* in, bk_batch_result* out);

/* The same call for regions beyond the limits of bk_compare_kmers_batch's assembler: reads and contigs up to 65535
 * bases (a region with a longer read, or whose contig would grow longer, or that starts more than 65535 contigs, is
 * reported through region_status as BK_ERR_CAPACITY, with no contigs in the result; the other regions are unaffected).
 * Same inputs, outputs and k-mer stage; it is the "long_regions" pass (bk_set_option) with every region given to the
 * long assembler, which runs one 256-thread CTA per region, without speculation, and aligns pairs above 4095 bases
 * with the anti-diagonal sweep of bk_nw_batch's long pairs.  Synchronous; meant for the few regions the batched call
 * reports as BK_ERR_CAPACITY, not as a replacement for it. */
int bk_compare_kmers_long(bk_handle_t h, const bk_batch_input* in, bk_batch_result* out);

/* The same call in two halves, for callers that keep several batches in flight from ONE host thread (the region loop
 * of sv_processor.py:185-201 turned into a pipeline; one handle per batch in flight, several handles per GPU):
 * bk_batch_submit copies the inputs and enqueues the whole device pass on the handle's stream without waiting for
 * the device at any point (every intermediate size stays in device memory), then returns; bk_batch_wait blocks until
 * that pass is done and fills `out`.  in == NULL submits the batch uploaded with bk_batch_upload.  The input arrays
 * must stay valid and unchanged until bk_batch_submit returns (page-locked inputs, e.g. from bk_ingest_*: until
 * bk_batch_wait returns).  One batch in flight per handle.  A region holding a read longer than 4095 bases is left
 * out of the device pass and reported through region_status (BK_ERR_CAPACITY); the other regions are unaffected
 * (the handle's "long_regions" option, bk_set_option, assembles such regions in the same pass). */
int bk_batch_submit(bk_handle_t h, const bk_batch_input* in);
int bk_batch_wait(bk_handle_t h, bk_batch_result* out);

/* ---- timing support for bench.py ------------------------------------------------------
 * bk_batch_upload copies a batch to the device once; bk_compare_kmers_resident then runs
 * the whole device pipeline on the resident copy (no host->device input traffic in the
 * call; results still come back).  bk_kernel_times returns the accumulated device time
 * (ms, CUDA events on the handle's stream) and launch count per kernel family since the
 * last bk_kernel_times_reset; names is a ';'-separated list in the same order. */
int bk_batch_upload(bk_handle_t h, const bk_batch_input* in);
/* ---- persistent reference k-mer cache ------------------------------------------------------
 * The GPU analogue of the reference's marker-file cache of the target reference dumps
 * (utils.py:157 skips jellyfish when the dump exists; preset_ref_data, sv_processor.py:108-162):
 * the forward and reverse-complement k-mers of every target window are counted once and kept on
 * the device.  A later bk_compare_kmers_batch / bk_batch_upload on this handle whose ref_bases and
 * ref_off are NULL uses the cache instead (same n_regions, same k, regions in the same order). */
int bk_ref_cache_build(bk_handle_t h, const char* ref_bases, const int64_t* ref_off, int32_t n_regions, int32_t k);
int bk_ref_cache_clear(bk_handle_t h);

/* Options of a handle.  "spec_width" = 0 | 1 | 2 | 4 | 8: warps per region in the assembler (how many
 * reads are aligned speculatively at once).  0 (default) = 4, one aligning warp per SM
 * sub-partition.  "blocking_sync" = 0 | 1: host threads waiting for the handle's stream spin (default, lowest
 * latency) or sleep on a blocking event (for hosts with fewer cores than handles in flight).  Results never
 * depend on either.
 * "long_regions" = 0 | 1 changes which regions get results.  0 (default): the batched entries report a region with a
 * read or contig above 4095 bases as BK_ERR_CAPACITY, as described above.  1: bk_compare_kmers_batch,
 * bk_batch_submit / bk_batch_wait and bk_batch_upload + bk_compare_kmers_resident assemble such regions in the same
 * device pass, up to 65535 bases, with the results bk_compare_kmers_long gives them: a region with a longer read is
 * left out and reported as BK_ERR_CAPACITY, and so is a region the long assembler cannot finish either (its contig
 * would grow past 65535 bases); such a region has no contigs in the result.  Contigs of a region's abandoned first
 * attempt never appear.  The option is read when the inputs are uploaded (bk_batch_submit with inputs,
 * bk_compare_kmers_batch, bk_batch_upload): a batch in flight or already uploaded keeps the mode it was uploaded
 * with.  It costs device memory per call (scratch of the long assembler, about 11 MB per CTA for at least 4 CTAs)
 * and two small launches; with 0 nothing extra is allocated or launched.
 * "rejected_contigs" = 0 | 1 adds to a result the contigs the assembler grows completely and then drops in its
 * acceptance test (sv_assembly.py:53-59): total read support below rc_thresh, or not longer than read_len.  0
 * (default): a result holds the accepted contigs only.  1: the rejected contigs are written out exactly as accepted
 * ones are and follow them in the ctg_*_off tables, at indices n_contigs and up; bk_rejected_contigs tells which
 * region and reason each one has.  Accepted contigs, n_contigs, ctg_reg_off and the files of bk_write_contigs /
 * bk_write_sample_kmers are the same either way.  A contig only set up (its first read already used) is never grown or
 * tested, so it is not one of them, and a region reported as BK_ERR_CAPACITY has none.  Read when the inputs are
 * uploaded, as "long_regions" is; bk_compare_kmers_long honours it too.  The rejected contigs take room in the
 * output arena like accepted ones. */
int bk_set_option(bk_handle_t h, const char* name, int64_t value);

/* ---- per-region report: why a region's assembly stopped and what the assembler did ----------------------------
 * One row of BK_RR_FIELDS int32 per region, in the order of the call's regions:
 *   BK_RR_REASON        why the region has no result (region_status BK_ERR_CAPACITY), BK_RR_OK (0) when it has one:
 *                       BK_RR_READ_TOO_LONG     a read above the mode's limit (4095 bases, 65535 in the long modes):
 *                                               the region was left out at upload
 *                       BK_RR_CONTIG_TOO_LONG   a contig would grow past the assembler's limit
 *                       BK_RR_KMER_LIST_FULL    a contig holds more k-mer tuples than 2 x that limit
 *                       BK_RR_TOO_MANY_CONTIGS  the region started more contigs than the assembler can tag
 *                                               (2^20 in the batched assembler, 2^16 in the long one)
 *   BK_RR_PASS          which assembler produced the result: BK_RR_PASS_NONE (0, left out at upload),
 *                       BK_RR_PASS_BATCHED (1, the batched assembler), BK_RR_PASS_LONG (2, the long assembler)
 *   BK_RR_FIRST_REASON  for a region the long assembler took over under the "long_regions" option: why the batched
 *                       assembler did not keep it -- BK_RR_READ_TOO_LONG (a read above 4095 bases, routed at upload),
 *                       one of the codes above, or BK_RR_OUTPUT_ARENA (its contigs did not fit the output arena).
 *                       0 for every other region, and for every region of bk_compare_kmers_long.
 *   BK_RR_SEEDS         seeds taken (akmers.has_mers iterations, sv_assembly.py:43-45)
 *   BK_RR_FIND_READS    find_reads calls
 *   BK_RR_CHECK_ALIGN   contig.check_align calls
 *   BK_RR_GROWN         contigs taken from buffer.contigs, grown and tested for acceptance (sv_assembly.py:50-59)
 *   BK_RR_REJ_SUPPORT   of those, rejected because their total read support is below rc_thresh
 *   BK_RR_REJ_LENGTH    of those, rejected because they are not longer than read_len (support tested first)
 * The counters are those of the pass that produced the result (BK_RR_PASS).  For a region with BK_RR_REASON 0,
 * BK_RR_GROWN = its contigs in the result + BK_RR_REJ_SUPPORT + BK_RR_REJ_LENGTH. */
#define BK_RR_REASON 0
#define BK_RR_PASS 1
#define BK_RR_FIRST_REASON 2
#define BK_RR_SEEDS 3
#define BK_RR_FIND_READS 4
#define BK_RR_CHECK_ALIGN 5
#define BK_RR_GROWN 6
#define BK_RR_REJ_SUPPORT 7
#define BK_RR_REJ_LENGTH 8
#define BK_RR_FIELDS 9

#define BK_RR_OK 0
#define BK_RR_READ_TOO_LONG 1
#define BK_RR_CONTIG_TOO_LONG 2
#define BK_RR_KMER_LIST_FULL 3
#define BK_RR_TOO_MANY_CONTIGS 4
#define BK_RR_OUTPUT_ARENA 5

#define BK_RR_PASS_NONE 0
#define BK_RR_PASS_BATCHED 1
#define BK_RR_PASS_LONG 2

/* The per-region report of the last result on the handle (bk_compare_kmers_batch, bk_compare_kmers_long,
 * bk_compare_kmers_resident, bk_batch_wait): n_regions rows of *n_fields int32, row-major, library-owned,
 * valid until the next call on the handle.  Copied from the device on request (nothing is copied when it
 * is not asked for).  BK_ERR_ARG while a batch is in flight or before any result. */
int bk_region_report(bk_handle_t h, const int32_t** table, int32_t* n_fields);

/* ---- rejected contigs of the last result (the "rejected_contigs" option) ------------------------------------------
 * Rejected contig j of region r has j in [reg_off[r], reg_off[r+1]) (n_regions + 1 offsets), in the order the
 * assembler grew them, and reason[j] = BK_REJ_SUPPORT (its total read support is below rc_thresh, tested first) or
 * BK_REJ_LENGTH (it is not longer than read_len).  Its sequence, kmer_locs, count vectors, reads and k-mer tuples are
 * those of contig n_contigs + j of the result's ctg_*_off tables.  For every region with a result,
 * reg_off[r+1] - reg_off[r] = BK_RR_REJ_SUPPORT + BK_RR_REJ_LENGTH of bk_region_report.  *n = reg_off[n_regions].
 * The arrays are library-owned host memory, valid until the next call on the handle.  BK_ERR_ARG while a batch is in
 * flight, before any result, after another call reused the result's memory, and for a result of a batch uploaded with
 * the option off. */
#define BK_REJ_SUPPORT 1
#define BK_REJ_LENGTH 2
int bk_rejected_contigs(bk_handle_t h, const int64_t** reg_off, const int32_t** reason, int64_t* n);

int bk_compare_kmers_resident(bk_handle_t h, bk_batch_result* out);
int bk_kernel_times(bk_handle_t h, const char** names, const double** ms, const int64_t** launches, int32_t* n);
int bk_kernel_times_reset(bk_handle_t h, int enable);

/* ---- ingest: text -> bk_batch_input (SURVEY.md section 8.7, row f.1) ----------------------------
 * Stands in for the readers on the way INTO target.compare_kmers:
 *   FastqFile / fq_read            utils.py:681-720   cleaned FASTQ -> (header, seq, qual) records
 *   get_fastq_reads                utils.py:203-246   records -> fq_recs + read_len (the sv_reads
 *                                                     filter of :213-236 stays with the caller, who
 *                                                     passes the filtered text)
 *   the readers of `jellyfish count`  utils.py:160    FASTA / FASTQ inputs of the three k-mer sets
 * For each of n_regions targets the caller gives up to four texts (in memory, or as file paths):
 * the reference window FASTA (files['target_ref_fn'][0]; its first record is used), the cleaned
 * reads FASTQ (files['cleaned_fq']), the soft-clip FASTA (files['sv_sc_unmapped_fa']) and
 * optionally a normal-sample FASTQ/FASTA.  A NULL list, NULL entry or empty path means "no
 * records".  The texts are parsed on n_threads host threads (0 = all cores) straight into ONE
 * host buffer owned by the ingest object -- page-locked when pinned != 0, so that
 * bk_compare_kmers_batch copies from it by DMA -- and `in` is filled with pointers into it
 * (k, rc_thresh, have_mers are left 0 for the caller; read_len = max record length per region,
 * utils.py:236; read_flags = the "_1" suffix fq_line writes, utils.py:436-443, and may be
 * overwritten in place through text->read_flags).  `text` (optional) gives the record ids and
 * quality strings needed to rebuild fq_read objects lazily.  Everything stays valid until the
 * next bk_ingest_* call on the object or bk_ingest_destroy.  Malformed FASTQ -> BK_ERR_FORMAT.
 * Host code only: no device work, usable without a GPU when pinned == 0. */
typedef struct bk_ingest_s* bk_ingest_t;
typedef struct bk_text { const char* p; int64_t n; } bk_text;
typedef struct bk_ingest_text {
  const char* id_bytes;   const int64_t* id_off;      /* n_reads + 1 */
  const char* qual_bytes; const int64_t* qual_off;    /* n_reads + 1 */
  int64_t n_reads;
  uint8_t* read_flags;                                /* mutable view of in->read_flags */
} bk_ingest_text;
int bk_ingest_create(int n_threads, int pinned, bk_ingest_t* out);
int bk_ingest_destroy(bk_ingest_t g);
const char* bk_ingest_last_error(bk_ingest_t g);
int bk_ingest_buffers(bk_ingest_t g, int32_t n_regions, const bk_text* ref_fa, const bk_text* reads_fq,
                      const bk_text* sc_fa, const bk_text* normal_fq, bk_batch_input* in, bk_ingest_text* text);
int bk_ingest_files(bk_ingest_t g, int32_t n_regions, const char* const* ref_fa, const char* const* reads_fq,
                    const char* const* sc_fa, const char* const* normal_fq, bk_batch_input* in, bk_ingest_text* text);

/* ---- contig hand-off (SURVEY.md section 8.7, row f.3) --------------------------------------------
 * The files sv_processor.contig.setup writes for every contig before blat
 * (sv_processor.py:749-782), for ALL contigs of a batch result on the ingest object's host threads:
 *   <contigs_dir[r]>/contig<n>/contig<n>.fq   write_read_fq   (:767-772)  id, seq, "+", qual per read
 *   <contigs_dir[r]>/contig<n>/contig<n>.fa   write_contig_fa (:776-781)  ">contig1\n" + sequence
 *   <cluster_fn[r]>                           write_cluster_file (:758-763) of the target's LAST contig
 *                                             (the reference reopens the file with 'w' for every contig)
 * n = 1.. in acceptance order (resolve_sv, sv_processor.py:649-653).  `res` is the result of the
 * bk_compare_kmers_batch call made with `in`; `in` and `text` come from bk_ingest_* (in->k set).
 * contigs_dir[r] NULL/"" skips region r; cluster_fn may be NULL.  Reads are written in ctg_reads
 * order (the reference iterates a Python set: no defined order). */
int bk_write_contigs(bk_ingest_t g, const bk_batch_result* res, const bk_batch_input* in, const bk_ingest_text* text,
                     const char* const* contigs_dir, const char* const* cluster_fn, int64_t* n_files);
/* The "<name>_sample_kmers.out" file of every target (sv_processor.py:625-632): "<mer>\t<case count>\n" per
 * sample-only k-mer, ascending mer order (the reference walks a Python set).  paths[r] NULL/"" skips region r. */
int bk_write_sample_kmers(bk_ingest_t g, const bk_batch_result* res, int32_t k, const char* const* paths, int64_t* n_files);

#ifdef __cplusplus
}
#endif
#endif /* BREAKMER_B200_H */
