/*
 * ssq.h — C-ABI of libssq.so, the B200-native implementation of the `speedseq align` hot path.
 *
 * The reference's drop-in boundary for this path is a PROCESS boundary, not an FFI:
 * bin/speedseq sources speedseq.config (/root/reference/bin/speedseq:15-24,361) and interpolates
 * $BWA and $SAMBLASTER into the pipeline text at /root/reference/bin/speedseq:437-449 (interleaved)
 * and :467-479 (two files); the index is made by `$BWA index` at :389.  libssq.so is what the two
 * replacement executables (speedseq_b200/bin/bwa, speedseq_b200/bin/samblaster) link; its entry
 * points are the batch forms of the functions those tools spend their time in (SURVEY.md §8a).
 * Each declaration cites the reference call site it serves and names the upstream routine it
 * replaces (upstream sources are NOT vendored in the reference tree: .SUBMODULES.json:23-29,51-57).
 *
 * Conventions: plain pointers and sizes, caller-owned HOST buffers unless a name ends in _dev,
 * int return code (0 = ok, <0 = SSQ_E*), no global state other than the CUDA context, one CUDA
 * stream per handle.  Every entry point fails with SSQ_ENOGPU when no sm_100 device is usable —
 * there is no CPU fallback inside this library.
 */
#ifndef SSQ_H
#define SSQ_H
#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSQ_OK        0
#define SSQ_ENOGPU   (-1)  /* no CUDA device / wrong architecture */
#define SSQ_EIO      (-2)  /* index files missing or malformed */
#define SSQ_ENOMEM   (-3)
#define SSQ_EINVAL   (-4)
#define SSQ_ECAP     (-5)  /* caller buffer too small; required size returned through *needed */
#define SSQ_ECUDA    (-6)  /* a CUDA call failed; see ssq_last_error() */
#define SSQ_ELEN     (-7)  /* a read is longer than SSQ_MAX_READ_LEN */
#define SSQ_EFORMAT  (-8)  /* FASTQ text the device tokeniser does not take (see ssq_aligner_upload_fastq); use the host tokeniser */

#define SSQ_MAX_READ_LEN 255

const char *ssq_last_error(void);
int ssq_device_count(void);

/* ---------------------------------------------------------------- options ----
 * Scoring/heuristic parameters of `bwa mem`; speedseq passes none of them on the command line
 * (/root/reference/bin/speedseq:438), so ssq_opts_default() is what the pipeline runs with.
 * Replaces upstream mem_opt_init(). */
typedef struct {
	int32_t a, b, o_del, e_del, o_ins, e_ins;
	int32_t pen_unpaired, pen_clip5, pen_clip3, w, zdrop, T;
	int32_t min_seed_len, split_width, max_occ, max_chain_gap, max_mem_intv;
	int32_t min_chain_weight, max_chain_extend, max_ins, max_matesw, max_XA_hits;
	float split_factor, mask_level, drop_ratio, XA_drop_ratio, mask_level_redun;
	int32_t mapQ_coef_len, mapQ_coef_fac;
	int32_t n_threads; /* host threads for the per-pair bookkeeping and SAM formatting (`bwa mem -t`); does not change any result */
} ssq_opts_t;
void ssq_opts_default(ssq_opts_t *o);

/* ------------------------------------------------------------------ index ----
 * Device-resident FM index + packed reference.  ssq_index_load replaces upstream bwa_idx_load()
 * (start of `$BWA mem`, /root/reference/bin/speedseq:438): reads PREFIX.{bwt,sa,pac,ann,amb} in the
 * on-disk format of the reference's goldens (/root/reference/example/data/ *.fasta.{amb,ann,pac,bwt,sa})
 * and uploads them to `device`. */
typedef struct ssq_index ssq_index_t;
/* `$BWA index $REF` (/root/reference/bin/speedseq:389): FASTA (plain or gz) -> PREFIX.{amb,ann,pac,bwt,sa}, byte-identical
 * to the reference's goldens for example/data; suffix sorting, BWT, occ checkpoints and SA sampling run on `device`.
 * References beyond the device sort's 2^31 - 2 suffixes (1.07 Gbp; a whole human genome has 6.2 G) are indexed on the host
 * instead — induced sorting with 5-byte entries, same files, no GPU touched (about 15 bytes of host memory per base pair:
 * 45 GB and 51 min for a 3.1 Gbp reference on 8 cores).
 * prefix == NULL means prefix = fasta.  Replaces upstream bwa_idx_build(). */
int ssq_index_build(const char *fasta, const char *prefix, int device);
int ssq_index_load(const char *prefix, int device, ssq_index_t **out);
void ssq_index_free(ssq_index_t *idx);
/* what: 0 l_pac, 1 seq_len(=2*l_pac), 2 primary, 3 n_seqs, 4 bwt words, 5 n_sa, 6 device bytes, 7 bytes per rank query (32|64),
 * 8 bytes per SA sample read (4|8), 9 SA sampling interval in device memory (on disk: 32; the loader derives a denser sample) */
uint64_t ssq_index_info(const ssq_index_t *idx, int what);

/* ----------------------------------------------------- kernel-level batches ----
 * Reads are passed as one byte per base (0=A 1=C 2=G 3=T 4=N), concatenated, with read_off[n+1]. */

/* SMEM seeding, all three passes, per read.  Replaces upstream mem_collect_intv() →
 * bwt_smem1a / bwt_seed_strategy1 / bwt_extend / bwt_2occ4 (inside `$BWA mem`, speedseq:438).
 * Output intervals of read i are out[out_off[i] .. out_off[i+1]) sorted by (qbeg<<32|qend). */
typedef struct { uint64_t k, l, s; uint32_t qbeg, qend; } ssq_smem_t;
int ssq_smem_batch(const ssq_index_t *idx, const ssq_opts_t *opt, int n_reads, const uint8_t *seq, const uint64_t *read_off,
                   ssq_smem_t *out, uint64_t out_cap, uint64_t *out_off, uint64_t *needed);

/* Suffix-array lookup of BWT rows.  Replaces upstream bwt_sa() / bwt_invPsi() (speedseq:438). */
int ssq_sa_lookup_batch(const ssq_index_t *idx, uint64_t n, const uint64_t *rows, uint64_t *pos);

/* Banded affine-gap seed extension.  Replaces upstream ksw_extend2() as called from
 * mem_chain2aln() (speedseq:438).  Sequences are one byte per base in qbuf/tbuf.
 * Each task needs 1 <= qlen <= SSQ_MAX_READ_LEN, h0 >= 1 and h0 + qlen * opt->a <= 65535: the DP row keeps H and E in
 * 16 bits each, so a larger possible score fails the call with SSQ_EINVAL (the pipeline's own extensions stay far below). */
typedef struct { uint64_t q_off, t_off; int32_t qlen, tlen, h0, w, end_bonus, zdrop; } ssq_sw_task_t;
typedef struct { int32_t score, qle, tle, gtle, gscore, max_off; } ssq_sw_result_t;
int ssq_sw_extend_batch(const ssq_opts_t *opt, int device, uint64_t n, const ssq_sw_task_t *tasks,
                        const uint8_t *qbuf, uint64_t qbuf_len, const uint8_t *tbuf, uint64_t tbuf_len, ssq_sw_result_t *out);

/* Local alignment in the evaluation order of the reference's striped SSE2 kernel.  Replaces upstream ksw_align2() as called from
 * mem_matesw() (mate rescue inside `$BWA mem`, speedseq:438): xtra = KSW_XSUBO|KSW_XSTART|(KSW_XBYTE if qlen*a < 250)|minsc.
 * One warp per problem, the SSE lanes mapped onto warp lanes (csrc/ssq_warp.cuh). */
typedef struct { uint64_t q_off, t_off; int32_t qlen, tlen, xtra, pad; } ssq_swl_task_t;
typedef struct { int32_t score, te, qe, score2, te2, tb, qb; } ssq_swl_result_t;
#define SSQ_KSW_XBYTE  0x10000
#define SSQ_KSW_XSTOP  0x20000
#define SSQ_KSW_XSUBO  0x40000
#define SSQ_KSW_XSTART 0x80000
int ssq_sw_local_batch(const ssq_opts_t *opt, int device, uint64_t n, const ssq_swl_task_t *tasks, const uint8_t *qbuf, uint64_t qbuf_len,
                       const uint8_t *tbuf, uint64_t tbuf_len, ssq_swl_result_t *out);

/* Chains after seeding + SA lookup + chaining + chain filter.  Replaces upstream mem_chain() +
 * mem_chain_flt() (speedseq:438).  Flattened: read i owns chains [read_chain_off[i], read_chain_off[i+1]),
 * chain c owns seeds [chain_seed_off[c], chain_seed_off[c+1]). */
typedef struct { int64_t rbeg; int32_t qbeg, len; } ssq_seed_t;
int ssq_chain_batch(const ssq_index_t *idx, const ssq_opts_t *opt, int n_reads, const uint8_t *seq, const uint64_t *read_off,
                    ssq_seed_t *seeds, uint64_t seed_cap, uint64_t *chain_seed_off, uint64_t chain_cap, uint64_t *read_chain_off,
                    uint64_t *n_chains, uint64_t *n_seeds);

/* Duplicate marking over pair signatures, first occurrence in input order is kept.  Replaces the
 * signature hash sets of samblaster's markDupsDiscordants() (`$SAMBLASTER`, speedseq:439).
 * valid==0 entries (both ends unmapped) are never duplicates. */
typedef struct { uint64_t pos1, pos2; uint8_t strand1, strand2, valid, pad[5]; } ssq_dupsig_t;
int ssq_dupmark_batch(int device, uint64_t n, const ssq_dupsig_t *sig, uint8_t *is_dup);

/* Streaming form for inputs that arrive in pieces (the `samblaster` shim): the set remembers every signature it has seen,
 * so "first occurrence wins" holds across calls as if all batches had been one. */
typedef struct ssq_dupset ssq_dupset_t;
int ssq_dupset_create(int device, ssq_dupset_t **out);
int ssq_dupset_mark(ssq_dupset_t *set, uint64_t n, const ssq_dupsig_t *sig, uint8_t *is_dup);
uint64_t ssq_dupset_size(const ssq_dupset_t *set);
void ssq_dupset_free(ssq_dupset_t *set);

/* Device-pointer form used by the multi-GPU exchange (speedseq_b200/dist.py): keys already sit in HBM (received by an NCCL
 * all-to-all), element order = first-seen order, key = (5' position << 1 | strand) of the canonically ordered ends. */
int ssq_dupmark_keys_dev(int device, uint64_t n, const uint64_t *d_key1, const uint64_t *d_key2, const uint8_t *d_valid, uint8_t *d_is_dup, void *stream);

/* ------------------------------------------------- the alignment pipeline ----
 * Seeding → SA lookup → chaining → chain filter → seed extension → alignment regions, all on the
 * device (the single-end core of `$BWA mem`, upstream mem_align1_core() up to and including
 * mem_chain2aln(); stage 1 adds mem_sort_dedup_patch()).  Regions of read i are
 * out[out_off[i] .. out_off[i+1]) in the order the reference produces them. */
typedef struct {
	int64_t rb, re;
	int32_t qb, qe, rid, score, truesc, w, seedcov, seedlen0;
	float frac_rep;
	int32_t read_id;
} ssq_alnreg_t;

/* one-shot, HOST buffers in and out: regions only (parity tests of the seed -> extend half; the CLI shim and bench.py drive ssq_aligner_*) */
int ssq_align_batch(const ssq_index_t *idx, const ssq_opts_t *opt, int n_reads, const uint8_t *seq, const uint64_t *read_off,
                    int stage, ssq_alnreg_t *out, uint64_t out_cap, uint64_t *out_off, uint64_t *needed);

/* staged form: upload once, run the kernels any number of times with everything resident in HBM
 * (`value` in bench.py), fetch results when wanted */
typedef struct ssq_batch ssq_batch_t;
int ssq_batch_create(const ssq_index_t *idx, const ssq_opts_t *opt, int n_reads, const uint8_t *seq, const uint64_t *read_off, ssq_batch_t **out);
/* (re)load a batch object with new reads; device buffers are kept and grown, so one object serves a stream of batches.
 * ssq_batch_create(..., read_off == NULL) makes an empty object to be filled by ssq_batch_upload(). */
int ssq_batch_upload(ssq_batch_t *b, int n_reads, const uint8_t *seq, const uint64_t *read_off);
int ssq_batch_run(ssq_batch_t *b);                 /* all kernels of the path on the batch's stream; returns when the last is queued */
int ssq_batch_sync(ssq_batch_t *b);
int ssq_batch_fetch(ssq_batch_t *b, ssq_alnreg_t *out, uint64_t out_cap, uint64_t *out_off, uint64_t *needed);
void *ssq_batch_stream(ssq_batch_t *b);            /* cudaStream_t, for event timing on the launching stream */
int ssq_batch_set_stream(ssq_batch_t *b, void *stream); /* make several batch objects share one caller-owned stream */
/* per-run work counters measured on the device: what: 0 occ blocks read by seeding, 1 occ blocks read by SA walks,
 * 2 SA samples read, 3 SW extension calls, 4 SW cells, 5 SW algorithmic bytes, 6 kernels launched per run, 7 seeds, 8 regions */
uint64_t ssq_batch_counter(const ssq_batch_t *b, int what);
/* milliseconds of the last run per stage (CUDA events on the batch stream): 0 smem, 1 sa, 2 chain, 3 extend, 4 finalize */
float ssq_batch_stage_ms(const ssq_batch_t *b, int stage);
void ssq_batch_free(ssq_batch_t *b);

/* ------------------------------------------------------- `bwa mem` for one batch ----
 * What the `bwa` shim calls per batch of reads (upstream mem_process_seqs(); `$BWA mem`, speedseq:438,468): reads as ASCII
 * strings (names already stripped of /1 /2), paired = adjacent reads are mates.  n_processed = global ordinal of reads[0]
 * (tie-breaking hashes use it).  pes0 != NULL overrides the per-batch insert-size statistics (`-I`).  Returns the SAM
 * records of the batch in input order as one malloc'd string (free with ssq_free).  Seeding, chaining, all Smith-Waterman
 * variants and CIGAR/NM/MD generation run on the device; pairing, MAPQ and text formatting on the host. */
typedef struct { int32_t low, high, failed, pad; double avg, std; } ssq_pestat_t;
int ssq_mem_batch_sam(const ssq_index_t *idx, const ssq_opts_t *opt, int n_reads, const char *const *names, const char *const *seqs, const char *const *quals,
                      const char *const *comments, int64_t n_processed, int paired, const ssq_pestat_t *pes0, const char *rg_id, int verbose, char **sam_out, size_t *sam_len,
                      size_t *read_sam_off /* optional [n_reads+1]: byte range of each read's lines */);
void ssq_free(void *p);

/* ----------------------------------------- `bwa mem | samblaster`, HBM-resident ----
 * The whole pipe of /root/reference/bin/speedseq:438-439 (interleaved) / :468-469 (two files) for one batch of reads:
 * `$BWA mem -t T [-p] [-C] [-I ..] -R RG REF FQ.. | $SAMBLASTER [--excludeDups] --addMateTags --maxSplitCount C
 * --minNonOverlap M --splitterFile F --discordantFile F`.  Reads go in as the FASTQ fields (concatenated, with offsets), the three
 * SAM record streams come out (main, splitters, discordants; headers are the caller's business: they depend on argv).  Between
 * the two copies everything stays on the device: alignment (upstream mem_process_seqs incl. mem_pestat's batch coupling — only
 * its histogram reduction runs on the host), pairing, MAPQ, CIGAR/NM/MD, samblaster's signature / discordant / splitter tests,
 * first-seen-wins duplicate marking against every earlier batch of the same aligner object, and the SAM text itself.
 * With sb == NULL or sb->enabled == 0 only text[0] is produced and it is exactly `bwa mem`'s records (what ssq_mem_batch_sam
 * returns).  One aligner object = one `bwa mem | samblaster` run: create, run batch after batch in input order, free. */
typedef struct {
	int32_t enabled;            /* 0: plain `bwa mem` records */
	int32_t exclude_dups;       /* --excludeDups: duplicates stay out of the splitter / discordant streams (speedseq:241) */
	int32_t add_mate_tags;      /* --addMateTags: MC:Z / MQ:i on every record of a pair (speedseq:439) */
	int32_t max_split_count;    /* --maxSplitCount (speedseq:242) */
	int32_t min_non_overlap;    /* --minNonOverlap (speedseq:243) */
	int32_t min_indel_size, max_unmapped_bases; /* samblaster defaults 50 / 50 */
	int32_t remove_dups;        /* --removeDups */
	int32_t want_split, want_disc; /* --splitterFile / --discordantFile given */
} ssq_sb_opts_t;
void ssq_sb_opts_default(ssq_sb_opts_t *o);

typedef struct {
	int32_t n_reads, paired;              /* paired: adjacent reads are mates (`-p` after smart pairing, or two files interleaved) */
	const char *seq; const uint64_t *seq_off;   /* bases as in the FASTQ (ASCII, any case), concatenated; seq_off[n_reads + 1] */
	const char *qual;                     /* qualities at the same offsets; NULL = none (FASTA input) */
	const char *name; const uint32_t *name_off; /* names without the /1 /2 suffix, concatenated, no terminators; name_off[n_reads + 1] */
	const char *comment; const uint32_t *comment_off; /* FASTQ comments for `-C`; NULL = none */
	int64_t n_processed;                  /* global ordinal of reads[0] (tie-breaking hashes use it) */
} ssq_reads_t;

typedef struct {
	const char *text[3]; size_t len[3];   /* 0 main SAM records, 1 splitters, 2 discordants; owned by the aligner, valid until its next run */
	const uint64_t *read_off;             /* [n_reads + 1]: byte range of each read's records in text[0] */
	uint64_t n_ids, n_dup;                /* QNAME blocks seen / marked duplicate in this batch */
	ssq_pestat_t pes[4];                  /* the insert-size statistics the batch was paired with */
} ssq_sam_t;

typedef struct ssq_aligner ssq_aligner_t;
int ssq_aligner_create(const ssq_index_t *idx, const ssq_opts_t *opt, const ssq_sb_opts_t *sb, const char *rg_id, ssq_aligner_t **out);
/* pes0 != NULL overrides the per-batch insert-size statistics (`-I`); verbose: mem_pestat's log lines on stderr like bwa */
int ssq_aligner_run(ssq_aligner_t *al, const ssq_reads_t *reads, const ssq_pestat_t *pes0, int verbose, ssq_sam_t *out);
/* the three phases of ssq_aligner_run, separately (bench.py times `compute` with the reads resident in HBM) */
int ssq_aligner_upload(ssq_aligner_t *al, const ssq_reads_t *reads);
int ssq_aligner_compute(ssq_aligner_t *al, const ssq_pestat_t *pes0, int verbose);
/* FASTQ ingest on the device instead of ssq_aligner_upload (upstream bseq_read -> kseq_read inside `$BWA mem`, speedseq:438,468;
 * tokenisation rules of /root/reference/src/samtools-1.3.1/htslib-1.3.1/htslib/kseq.h:189-231).  fq1 / fq2: raw, uncompressed text of
 * the FASTQ input(s) from a record boundary on (fq2 == NULL: one file; interleaved: adjacent records are mates, `-p`); final: no
 * more text follows.  The device finds the records, closes the batch where bwa would (bases >= chunk_bases and an even number of
 * reads), strips /1 /2, and packs names, bases, qualities and (keep_comment, `-C`) comments into the aligner's batch buffers;
 * *used1 / *used2 = bytes of each text the batch covers (the caller keeps the rest for the next call).  *need_more: no complete
 * batch in the text and more text exists -> call again with more.  SSQ_EFORMAT: not the four-lines-per-record layout (multi-line
 * records, FASTA, unpaired reads in an interleaved file, files of different lengths): nothing was consumed, tokenise on the host. */
int ssq_aligner_upload_fastq(ssq_aligner_t *al, const char *fq1, size_t len1, int final1, const char *fq2, size_t len2, int final2, int interleaved, int keep_comment,
                             int64_t chunk_bases, int64_t n_processed, size_t *used1, size_t *used2, int *n_reads, int *need_more);
void *ssq_host_alloc(size_t bytes); /* page-locked host memory for the text buffers (full-rate host->device copies) */
void ssq_host_free(void *p);
int ssq_aligner_fetch(ssq_aligner_t *al, ssq_sam_t *out);
int ssq_aligner_reset_dups(ssq_aligner_t *al);     /* forget every signature seen so far (a new run) */
/* several aligner objects (one host thread + stream each) can work on consecutive batches of ONE run: they share a dup-set, and
 * each batch is given its turn number (0, 1, 2, ... since the last reset) so that "first seen wins" still follows input order */
int ssq_aligner_share_dupset(ssq_aligner_t *al, ssq_dupset_t *set);
int ssq_aligner_set_turn(ssq_aligner_t *al, long long turn); /* -1 (default): no ordering (a single aligner runs its batches in order anyway) */
void *ssq_aligner_stream(ssq_aligner_t *al);       /* cudaStream_t of the object, for event timing on the launching stream */
/* milliseconds of the last batch per stage (CUDA events): 0 upload, 1 seed..extend, 2 sort/dedup/patch, 3 insert-size statistics,
 * 4 mate rescue, 5 pairing/MAPQ/planning, 6 CIGAR/NM/MD, 7 samblaster + dup-set, 8 text, 9 fetch; 10.. = ssq_batch_stage_ms(0..4) */
float ssq_aligner_stage_ms(const ssq_aligner_t *al, int stage);
/* what < 100: ssq_batch_counter of the alignment stage; 100 alignments written (CIGAR tasks), 101-103 bytes of the three streams, 104 dup-set size,
 * 105 pairs that went through mate rescue, 106 alignments that needed the banded global DP for their CIGAR,
 * 107 local-SW passes run by the mate rescue, 108 their cells, 109 bases / 110 reads of the batch in the aligner */
uint64_t ssq_aligner_counter(const ssq_aligner_t *al, int what);
void ssq_aligner_free(ssq_aligner_t *al);

/* ----------------------------------------------------------------- BAM records ----
 * The downstream half of the pipe turns the SAM text straight back into BAM (`sambamba view -S -f bam -l 0 | sambamba sort`,
 * speedseq:440-441, :444-448).  With ssq_aligner_set_bam(al, 1, ..) the aligner additionally encodes the records of the three
 * streams as BAM on the device, straight from its structured alignments (layout: htslib sam.c:443-467, bin: hts.h:580-586),
 * coordinate-sorted within the batch by (reference, position, strand) with equal keys in input order — what sambamba's sort
 * produces (tests/golden/ex_bam_*: written by the reference's own sambamba, matched byte for byte).  blank_side_streams: the
 * splitter / discordant records carry no SEQ / QUAL, like after speedseq's gawk step (speedseq:443,446).
 * ssq_bam_header + ssq_bgzf_compress (host: zlib) make a complete .bam out of header and records; ssq_bam_merge_runs merges the
 * sorted runs of the batches of a run into the order `sambamba sort` gives the whole input. */
int ssq_aligner_set_bam(ssq_aligner_t *al, int enable, int blank_side_streams);
int ssq_aligner_fetch_bam(ssq_aligner_t *al, int stream, const void **records, size_t *len); /* after ssq_aligner_compute; owned by the aligner */
/* the SAM text of one stream alone (0 main, 1 splitters, 2 discordants), for callers that take the main records as BAM and only
 * want the side streams as text (speedseq:443,446 run them through gawk); after ssq_aligner_compute; owned by the aligner */
int ssq_aligner_fetch_text(ssq_aligner_t *al, int stream, const char **text, size_t *len);
int ssq_bam_header(const ssq_index_t *idx, const char *sam_header_text, int sorted, void **out, size_t *out_len); /* free with ssq_free */
/* the header text alone: sorted != 0 rewrites it the way `sambamba view -S | sambamba sort` does (@HD SO:coordinate first, sambamba's
 * tag order inside @SQ / @RG / @PG lines); free with ssq_free */
int ssq_bam_header_text(const char *sam_header_text, int sorted, char **out);
int ssq_bgzf_compress(const void *in, size_t n, int level, int with_eof, void **out, size_t *out_len);           /* free with ssq_free */
/* the sorted runs of consecutive batches -> one sorted record stream (stable: equal keys keep batch order); free with ssq_free */
int ssq_bam_merge_runs(int n_runs, const void *const *runs, const size_t *lens, void **out, size_t *out_len);

/* ------------------------------------------------------------------ several GPUs ----
 * Batches are dealt to the ranks round-robin with the index replicated (no collective); "first pair seen with a signature is
 * kept" (`$SAMBLASTER`, speedseq:439) stays global through one exchange per round, in C over NCCL: signatures go to the owner rank
 * hash(signature) mod N (grouped ncclSend/ncclRecv, 16 B per pair), the owner marks them against everything it has owned so far,
 * one byte per pair comes back (csrc/ssq_dist.cu).  One process per GPU: rank 0 makes the id, every rank creates its communicator
 * and hands it to its aligner object(s); ssq_aligner_compute then performs the round inside its duplicate stage (a collective: all
 * ranks run the same number of batches, empty ones included). */
typedef struct ssq_comm ssq_comm_t;
int ssq_comm_unique_id(void *id128);  /* 128 bytes, to be broadcast to the other ranks by whatever launched them */
int ssq_comm_create(const void *id128, int rank, int world, int device, ssq_comm_t **out);
int ssq_aligner_set_comm(ssq_aligner_t *al, ssq_comm_t *comm);
/* one round on explicit device arrays (key = 5' position << 1 | strand of the canonically ordered ends, array order = input order) */
int ssq_comm_mark_round(ssq_comm_t *comm, uint64_t n, const uint64_t *d_key1, const uint64_t *d_key2, const uint8_t *d_valid, uint8_t *d_is_dup, void *stream);
ssq_dupset_t *ssq_comm_dupset(ssq_comm_t *comm);            /* the signatures this rank owns (reset it on every rank to start a new run) */
uint64_t ssq_comm_counter(const ssq_comm_t *comm, int what); /* 0 bytes sent to other ranks, 1 bytes received back, 2 rounds */
void ssq_comm_free(ssq_comm_t *comm);

/* streaming dup-set on device pointers (what the aligner uses; also the owner-side step of the multi-GPU exchange) */
int ssq_dupset_mark_dev(ssq_dupset_t *set, uint64_t n, const uint64_t *d_key1, const uint64_t *d_key2, const uint8_t *d_valid, uint8_t *d_is_dup, void *stream);
int ssq_dupset_reset(ssq_dupset_t *set);
/* contig table for the SAM header: name/length of contig i (0 <= i < ssq_index_info(idx,3)) */
const char *ssq_index_contig(const ssq_index_t *idx, int i, int64_t *len);

#ifdef __cplusplus
}
#endif
#endif
