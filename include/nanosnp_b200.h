/*
 * nanosnp_b200 -- C ABI of the B200-native NanoSNP pileup-model hot path (stages s1 + s2).
 *
 * NanoSNP itself has no FFI: its stages are coupled by CLIs and files (SURVEY.md section 8b).  Every
 * entry point below therefore cites the reference *program or function* whose work it replaces.
 * A maintainer binds this library from Python with ctypes (INTEGRATION.md shows the stub); there are
 * no torch / C++ types in any signature: plain pointers, sizes, a cudaStream_t passed as void*.
 *
 * Conventions
 *   - every function returns 0 on success and a negative NSNP_E_* code on failure; nothing throws,
 *     nothing aborts, nothing falls back to the CPU.  nsnp_last_error() gives a thread-local message.
 *   - "dev" pointers are device memory owned by the caller (torch tensors in the Python host code);
 *     the library never allocates device memory: workspaces are sized by nsnp_*_workspace_bytes().
 *   - positions are 0-based on the contig inside this ABI; VCF / .tensor text is 1-based.
 *   - kernels are enqueued on the caller's stream and do not synchronise unless stated.
 */
#ifndef NANOSNP_B200_H
#define NANOSNP_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NSNP_ABI_VERSION 2

/* error codes */
#define NSNP_OK               0
#define NSNP_E_INVALID       -1   /* bad argument (null pointer, negative size, unsorted reads ...) */
#define NSNP_E_CUDA          -2   /* a CUDA runtime call failed; see nsnp_last_error() */
#define NSNP_E_WORKSPACE     -3   /* caller workspace too small */
#define NSNP_E_OVERFLOW      -4   /* a device-side capacity was exceeded (> 16383 reads over one 1024-bp tile, candidate buffer) */
#define NSNP_E_NO_DEVICE     -5   /* no CUDA device: there is deliberately no CPU fallback */
#define NSNP_E_UNSUPPORTED   -6   /* e.g. a CIGAR with P pads or unmerged adjacent I I / D D ops (nsnp_bam_fill merges them) */

/* channel order of the count tensor: reference dna_sv_tensor/src/common/tensor.hpp:6-26 */
enum {
    NSNP_CH_A = 0, NSNP_CH_C, NSNP_CH_G, NSNP_CH_T, NSNP_CH_I, NSNP_CH_I1, NSNP_CH_D, NSNP_CH_D1,
    NSNP_CH_STAR, NSNP_CH_a, NSNP_CH_c, NSNP_CH_g, NSNP_CH_t, NSNP_CH_i, NSNP_CH_i1, NSNP_CH_d,
    NSNP_CH_d1, NSNP_CH_POUND, NSNP_CHANNELS /* = 18 */
};
#define NSNP_FLANK       16      /* make_predict_data.sh:119 FLANKING_BASES */
#define NSNP_WINDOW      33      /* make_candidate_snp_tensor/main.cpp:126 */
#define NSNP_MAX_INDEL   60      /* tensor_maker.cpp:5 kMaxIndelSize */
#define NSNP_GT_CLASSES  21      /* PileupModel/options.py:8-28 */
#define NSNP_ZY_CLASSES  3       /* PileupModel/options.py:30 */

/* bits of the per-position flag byte written by nsnp_pileup_counts */
#define NSNP_F_COVERED   1       /* an mpileup row exists for this position (SURVEY appendix B.2) */
#define NSNP_F_GATE      2       /* refbase in ACGT && pass_af && depth >= min_coverage (main.cpp:196) */

/*
 * Aligned reads of ONE contig region as flat packed arrays (what a host BAM decoder produces;
 * replaces the BAM -> `samtools mpileup` text hand-off of make_predict_data.sh:117,151).
 * Reads must be sorted by pos (coordinate-sorted BAM order); ties keep file order.
 * CIGARs must be canonical: adjacent ops of the same indel type merged ("1D2D" -> "3D", as htslib reports them), no P ops;
 * anything else is refused with NSNP_E_UNSUPPORTED.  Leading / trailing / adjacent I-D ops, N skips, S/H clips and =/X are
 * handled as `samtools mpileup` reports them (SURVEY appendix B.2; hand-worked cases in tests/golden/cigar_cases.txt).
 */
typedef struct nsnp_reads {
    int64_t         n_reads;
    const int32_t*  pos;        /* [n] 0-based leftmost reference position (BAM pos) */
    const uint16_t* flag;       /* [n] SAM flag; reads with (flag & excl_flags) are dropped */
    const uint8_t*  mapq;       /* [n] reads with mapq < min_mapq are dropped */
    const int64_t*  cigar_off;  /* [n+1] index of the read's first op in cigar[] */
    const uint32_t* cigar;      /* BAM encoding: len<<4 | op, op = MIDNSHP=X -> 0..8 (uint16 words when cigar_bits == 16) */
    const int64_t*  seq_off;    /* [n] index (in bases) of the read's first SEQ base in seq2/nmask */
    const uint8_t*  seq2;       /* 2-bit bases A0 C1 G2 T3: base k lives in byte k>>2, bits 2*(k&3) */
    const uint8_t*  nmask;      /* optional (may be NULL): bit (k&7) of byte k>>3 set => base k is N */
    const uint8_t*  qual;       /* optional, unused: s1/s2 run with --min-BQ 0 and never read qualities */
    int64_t         n_cigar;    /* total ops  (= cigar_off[n]) */
    int64_t         n_bases;    /* capacity of seq2/nmask in bases */
    int32_t         cigar_bits; /* 32 (or 0): cigar[] holds uint32 words; 16: the same values as uint16 (every length < 4096) --
                                   what a host decoder ships when it can: halves the CIGAR bytes on the wire */
    int32_t         reserved;
} nsnp_reads_t;

/* s1 parameters; defaults = make_predict_data.sh:117-125 */
typedef struct nsnp_params {
    double   snp_min_af;     /* 0.12 */
    double   indel_min_af;   /* 0.12 */
    int32_t  min_coverage;   /* 6 */
    int32_t  min_mapq;       /* 20   (--min-MQ) */
    uint32_t excl_flags;     /* 2316 (--excl-flags) */
    int32_t  max_depth;      /* 144  (--max-depth): htslib's streaming depth cap, SURVEY appendix B.3; <= 0 disables it */
} nsnp_params_t;

void        nsnp_default_params(nsnp_params_t* p);
int         nsnp_abi_version(void);
const char* nsnp_last_error(void);
int         nsnp_device_count(void);          /* 0 when no GPU is visible (library still loads) */

/* ---- s1, step A: pileup counts ------------------------------------------------------------------
 * Replaces `samtools mpileup` + TensorMaker::make_tensor (tensor_maker.cpp:61-249) for the region
 * [region_start, region_start + region_len) of one contig.
 *   ref_dev      [contig_len]      ASCII reference of the whole contig (raw case)
 *   counts_dev   [region_len][18]  int32, final values incl. the reference-channel overwrite
 *   flags_dev    [region_len]      NSNP_F_COVERED | NSNP_F_GATE
 *   status_dev   [4] int32         device-side status words (0 = ok); read with nsnp_check_status
 * reads may include reads that do not overlap the region (they are skipped).
 */
size_t nsnp_pileup_workspace_bytes(int64_t n_reads, int64_t n_cigar, int64_t region_len);
int nsnp_pileup_counts(const nsnp_reads_t* reads_dev, const uint8_t* ref_dev, int64_t contig_len,
                       int64_t region_start, int64_t region_len, const nsnp_params_t* params,
                       int32_t* counts_dev, uint8_t* flags_dev,
                       void* workspace_dev, size_t workspace_bytes, int32_t* status_dev, void* stream);

/* ---- s1, step B: candidate selection ------------------------------------------------------------
 * Replaces the gate + 33-row contiguity rule of create_pileup_tensor (main.cpp:174-217).
 * Emits, in ascending order, every 0-based position c in [emit_start, emit_end) with the GATE bit set
 * and COVERED set on all of [c-16, c+16].  flags_dev covers [region_start, region_start+region_len).
 *   recompute_gate != 0: ignore the GATE bit and recompute it from counts_dev + ref_dev
 *   pos_dev [capacity] int32 (contig coordinates); n_dev [1] int32 receives the total count
 *   (which may exceed capacity: then only the first `capacity` are written and NSNP_E_OVERFLOW is
 *    reported through status_dev).
 */
size_t nsnp_select_workspace_bytes(int64_t region_len);
int nsnp_select_candidates(const int32_t* counts_dev, uint8_t* flags_dev, const uint8_t* ref_dev,
                           int64_t contig_len, int64_t region_start, int64_t region_len,
                           int64_t emit_start, int64_t emit_end, const nsnp_params_t* params,
                           int recompute_gate, int32_t* pos_dev, int64_t capacity, int32_t* n_dev,
                           void* workspace_dev, size_t workspace_bytes, int32_t* status_dev, void* stream);

/* ---- s1, steps A and B restricted to target intervals ------------------------------------------------
 * An extension of this library with no reference counterpart (NanoSNP calls whole contigs).
 * targets: n_targets half-open [start, end) int32 pairs in contig coordinates, in HOST memory, non-empty,
 * ascending and disjoint (adjacent is allowed), inside [region_start, region_start + region_len); anything
 * else returns NSNP_E_INVALID.  The library copies them to its workspace and derives on the device
 *   - pileup: the tiles holding any position of [start - 16, end + 16); only those are computed.  Flags of
 *     every other position are written as 0 and their count rows are left unwritten.  Count rows and flags
 *     of computed positions equal those of nsnp_pileup_counts on the same reads.  The read pre-pass and the
 *     depth cap still run over every read passed.
 *   - select: a position is a candidate iff it is one of nsnp_select_candidates AND lies in an interval.
 * n_targets == 0 is valid: no tile is computed, no site is selected.
 */
size_t nsnp_pileup_targets_workspace_bytes(int64_t n_reads, int64_t n_cigar, int64_t region_len, int64_t n_targets);
int nsnp_pileup_counts_targets(const nsnp_reads_t* reads_dev, const uint8_t* ref_dev, int64_t contig_len,
                               int64_t region_start, int64_t region_len, const int32_t* targets, int64_t n_targets,
                               const nsnp_params_t* params, int32_t* counts_dev, uint8_t* flags_dev,
                               void* workspace_dev, size_t workspace_bytes, int32_t* status_dev, void* stream);
size_t nsnp_select_targets_workspace_bytes(int64_t region_len, int64_t n_targets);
int nsnp_select_candidates_targets(const int32_t* counts_dev, uint8_t* flags_dev, const uint8_t* ref_dev,
                                   int64_t contig_len, int64_t region_start, int64_t region_len,
                                   int64_t emit_start, int64_t emit_end, const int32_t* targets, int64_t n_targets,
                                   const nsnp_params_t* params, int recompute_gate, int32_t* pos_dev, int64_t capacity,
                                   int32_t* n_dev, void* workspace_dev, size_t workspace_bytes, int32_t* status_dev,
                                   void* stream);

/* ---- s1, step C: window gather ------------------------------------------------------------------
 * Replaces the ring-buffer window emit (main.cpp:220-251), DNA_CreatePredictData
 * (make_predict_data/main.cpp:76-127) and make_bin_predict_data.py:35-55: writes position_matrix
 * [n][33][18] directly in the PileupModel input layout.  Either output may be NULL.
 *   x_i32_dev int32 [n][33][18]   (PredictDataset.position_matrix, dataset.py:121)
 *   x_f32_dev float [n][33][18]   (predict.py:49 .type(FloatTensor))
 *   refbase_dev u8 [n]            upper-cased centre reference base (dataset.py:133 ord(seq[16]))
 */
int nsnp_gather_windows(const int32_t* counts_dev, const uint8_t* ref_dev, int64_t region_start,
                        int64_t region_len, const int32_t* pos_dev, const int32_t* n_dev, int64_t n_max,
                        int32_t* x_i32_dev, float* x_f32_dev, uint8_t* refbase_dev, void* stream);

/* ---- s2: PileupModel forward ----------------------------------------------------------------------
 * Replaces LSTMNetwork.predict (PileupModel/model.py:114-119): 2-layer BiLSTM(18->64) + output_proj
 * + dense/tanh @t=16 + genotype/zygosity heads + softmax.  Weights are the fp32 tensors of the
 * reference checkpoint (utils.py:67-77), packed by nsnp_model_pack_weights into one device blob.
 */
typedef struct nsnp_model_weights {      /* host pointers, PyTorch layouts, gate order i,f,g,o */
    const float* w_ih[2][2];   /* [layer][dir]  [256][18] / [256][128] */
    const float* w_hh[2][2];   /*               [256][64] */
    const float* b_ih[2][2];   /*               [256] */
    const float* b_hh[2][2];   /*               [256] */
    const float* proj_w;  const float* proj_b;    /* [128][128], [128] */
    const float* dense_w; const float* dense_b;   /* [256][128], [256] */
    const float* gt_w;    const float* gt_b;      /* [21][256], [21] */
    const float* zy_w;    const float* zy_b;      /* [3][256], [3] */
} nsnp_model_weights_t;

size_t nsnp_model_blob_bytes(void);
/* packs into host_blob (caller copies it to the device once) */
int nsnp_model_pack_weights(const nsnp_model_weights_t* w, void* host_blob, size_t blob_bytes);
size_t nsnp_model_workspace_bytes(int64_t n_sites);
/* x: exactly one of x_i32_dev / x_f32_dev non-NULL, [n][33][18].  n_dev (optional) overrides n. */
int nsnp_pileup_model_forward(const void* blob_dev, const int32_t* x_i32_dev, const float* x_f32_dev,
                              int64_t n, const int32_t* n_dev, float* gt_prob_dev, float* zy_prob_dev,
                              void* workspace_dev, size_t workspace_bytes, int precision, void* stream);
/* Same network, reading each site's window straight from the count tensor of its region: a window is the contiguous row span
 * counts[pos - 16 .. pos + 16] (create_pileup_tensor, main.cpp:220-251), so the [n][33][18] tensor of the dataset seam need not
 * be materialised between s1 and s2 (saves one 4.7 KB/site gather and its read-back).  NSNP_PREC_F16X3 / F16X1 only. */
int nsnp_pileup_model_forward_sites(const void* blob_dev, const int32_t* counts_dev, int64_t region_start, int64_t region_len,
                                    const int32_t* pos_dev, int64_t n, const int32_t* n_dev, float* gt_prob_dev, float* zy_prob_dev,
                                    void* workspace_dev, size_t workspace_bytes, int precision, void* stream);
#define NSNP_PREC_FP32    0   /* fp32 FFMA everywhere (parity path) */
#define NSNP_PREC_F16X3   1   /* tcgen05 tensor-core path: fp16 hi/lo split operands (3 MMAs per product), fp32 accumulate */
#define NSNP_PREC_F16X1   2   /* opt-in: ONE fp16 MMA per product (operands rounded to fp16, fp32 accumulate), then every site whose
                                 top-2 margin is below 0.02 in either head is re-evaluated with NSNP_PREC_F16X3 (<= 4096 per call), so
                                 the genotype / zygosity calls are those of NSNP_PREC_F16X3; other sites: |dp| < 5e-3 (observed 3e-3),
                                 QUAL may move by up to ~0.06.  Batches of <= 16384 sites run NSNP_PREC_F16X3 directly. */
/* NSNP_PREC_F16X1 keeps two counters in the first bytes of the model workspace: the low-margin sites the LAST forward call
 * found and their maximum over all calls since nsnp_model_f16x1_reset (call it once on a fresh workspace).
 * nsnp_model_f16x1_reevaluated returns the former (synchronises the stream) and NSNP_E_OVERFLOW when ANY call since the reset
 * found more than the 4096 that are re-evaluated. */
int nsnp_model_f16x1_reset(void* workspace_dev, void* stream);
int nsnp_model_f16x1_reevaluated(const void* workspace_dev, int64_t* count_out, void* stream);

/* debug aid for the tensor-core path: raw gate pre-activations [m][256] (TMEM column order) of the FIRST step of one
 * (layer, direction); cg = 1 or 2 CTAs per MMA.  Used by the GPU tests to validate operand layouts. */
int nsnp_debug_lstm_tc_gates(const void* blob_dev, const int32_t* x_i32_dev, int layer, int dir, int cg, const void* h0_dev,
                             float* gates_out_dev, int64_t m, void* stream);

/* ---- BASELINE configs[4]: HaplotypeModel s5 (csrc/haplotype.cu) ---------------------------------------------------------
 * nsnp_hap_features replaces get_frequency_feature + the reference-code row (HaplotypeModel/dataset_dev.py:11-87,337-349):
 *   seq / bq / mq / hp  int32 [n][depth][L]  read x position matrices as write_to_bins.py:15-63 stores them
 *                       (base 1..4, deletion -1, absent 0, pad rows -2; HP tag 1 / 2, untagged 3)
 *   refcode             int32 [n][L]         A1 C2 G3 T4, everything else 0 (dataset_dev.py:104-118)
 *   out                 float [n][105][L]    bit-identical to the reference's float64 features after `.type(FloatTensor)`
 * nsnp_hap_model_forward replaces LSTMNetwork.predict (HaplotypeModel/model_dev.py:133-143): x_pileup [n][105][33],
 * x_haplotype [n][105][11] -> softmaxed genotype [n][10] / zygosity [n][3].  fp32.  Weights: PyTorch layouts, gate order i,f,g,o;
 * index [encoder 0 pileup / 1 haplotype][layer 0..2][direction]. */
typedef struct nsnp_hap_weights {
    const float* w_ih[2][3][2];    /* [1024][105] (layer 0) / [1024][512] */
    const float* w_hh[2][3][2];    /* [1024][256] */
    const float* b_ih[2][3][2];    /* [1024] */
    const float* b_hh[2][3][2];
    const float* proj_w[2]; const float* proj_b[2];      /* output_proj [256][512], [256] */
    const float* dense_w;  const float* dense_b;         /* [256][512], [256] */
    const float* gt_w;     const float* gt_b;            /* [10][256], [10] */
    const float* zy_w;     const float* zy_b;            /* [3][256], [3] */
} nsnp_hap_weights_t;
int nsnp_hap_features(const int32_t* seq_dev, const int32_t* bq_dev, const int32_t* mq_dev, const int32_t* hp_dev, const int32_t* refcode_dev,
                      int64_t n, int32_t depth, int32_t L, float* out_dev, void* stream);
size_t nsnp_hap_model_blob_bytes(void);
int nsnp_hap_model_pack_weights(const nsnp_hap_weights_t* w, void* host_blob, size_t blob_bytes);
size_t nsnp_hap_model_workspace_bytes(int64_t n);
int nsnp_hap_model_forward(const void* blob_dev, const float* xp_dev, const float* xh_dev, int64_t n, float* gt_prob_dev, float* zy_prob_dev,
                           void* workspace_dev, size_t workspace_bytes, void* stream);
/* Opt-in tensor-core version of nsnp_hap_model_forward (csrc/haplotype_tc.cu): same inputs and outputs, its own packed blob and
 * workspace.  Precision f16x3: tcgen05 MMAs with hi/lo split operands (three MMAs per product), fp32 accumulation -- tf32 hi/lo
 * for the layer-0 input channels (unbounded feature values), fp16 hi/lo for h and the layer outputs.  Probabilities stay within
 * 5e-5 of a float64 evaluation of the network, as NSNP_PREC_F16X3 does for the PileupModel; nsnp_hap_model_forward (fp32) stays
 * the parity reference.  A site's result does not depend on the batch it is in. */
size_t nsnp_hap_model_tc_blob_bytes(void);
int nsnp_hap_model_tc_pack_weights(const nsnp_hap_weights_t* w, void* host_blob, size_t blob_bytes);
size_t nsnp_hap_model_tc_workspace_bytes(int64_t n);
int nsnp_hap_model_tc_forward(const void* blob_dev, const float* xp_dev, const float* xh_dev, int64_t n, float* gt_prob_dev, float* zy_prob_dev,
                              void* workspace_dev, size_t workspace_bytes, void* stream);
/* test aid, like nsnp_debug_lstm_tc_gates: the layer-0 gate pre-activations (input part + bias, h = 0) of the FIRST step of one
 * (encoder 0 pileup / 1 haplotype, direction), [m][1024] in PyTorch gate order.  x_dev: that encoder's features [m][105][L]. */
int nsnp_debug_hap_tc_gates(const void* blob_dev, const float* x_dev, int encoder, int dir, float* gates_out_dev, int64_t m, void* stream);

/* ---- BASELINE configs[4]: HaplotypeModel s4, read x position matrices (csrc/hap_groups.cu) -----------------------------
 * Replaces single_group_pileup_haplotype_feature (HaplotypeModel/create_pileup_haplotype.py:23-216): the two pysam pileup
 * sweeps + pandas of one sub-group.  reads_dev: one contig, file order; reads->qual (optional) holds the base qualities at the
 * same base index as seq2.  hp_dev [n_reads]: HP tag (1 / 2, 0 = untagged).  end_dev / end_pm_dev [n_reads]: exclusive reference
 * end of every alignment (nsnp_hap_read_ends) and its running maximum.  checkpoints_dev (optional, 8-byte aligned):
 * 2 x nsnp_hap_checkpoint_count() int32, the (reference, query) position every 32 CIGAR ops, also written by nsnp_hap_read_ends:
 * lets the kernel jump to a column instead of walking there.  dup_prev_dev / dup_next_dev [n_reads] (both or NULL):
 * previous / next alignment with the same query name among the alignments pysam's stepper keeps, -1 = none -- the reference
 * keys its rows by query name (:107-121).  gpos_dev [n_groups][n_hap]: 1-based ascending positions, centre = candidate.
 * fetch_lo_dev [n_groups]: `start` of the pysam sweep the group belongs to (alignments with end <= start are not fetched).
 * flank < 0: first sweep (:39-46) -- only n_cols_dev [n_groups][n_hap] (pileupcolumn.n of the hap sites), depth_dev (rows) and
 * flags_dev are written, hap_dev / pile_dev are NULL.  flank >= 0: second sweep (:93-205) -- n_cols_dev
 * [n_groups][n_hap + 2*flank+1], and hap_dev[4] / pile_dev[4] = {sequences, hap, baseq, mapq} int32 [n_groups][cap][n_hap] /
 * [n_groups][cap][2*flank+1], rows ordered by the centre's HP tag, padded with -2 (write_to_bins.py:14-30).
 * flags_dev bit 0: a SEQ letter outside ACGT on a column of interest (KeyError at :123 -> the reference drops the sub-group);
 * bit 1: more rows than cap. */
int64_t nsnp_hap_checkpoint_count(int64_t n_reads, int64_t n_cigar);
int nsnp_hap_read_ends(const nsnp_reads_t* reads_dev, int32_t* end_dev, int32_t* checkpoints_dev, void* stream);
int nsnp_hap_group_matrices(const nsnp_reads_t* reads_dev, const uint8_t* hp_dev, const int32_t* end_dev, const int32_t* end_pm_dev,
                            const int32_t* checkpoints_dev,
                            const int32_t* dup_prev_dev, const int32_t* dup_next_dev, const int32_t* gpos_dev,
                            const int32_t* fetch_lo_dev, int64_t n_groups, int32_t n_hap, int32_t flank, int32_t cap,
                            int32_t* n_cols_dev, int32_t* depth_dev, int32_t* flags_dev, int32_t* const* hap_dev,
                            int32_t* const* pile_dev, void* stream);

/* ---- per-kernel timing (bench.py) ---------------------------------------------------------------
 * When enabled, every kernel launch of this library is bracketed by cudaEventRecord on the launching stream.
 * nsnp_profile_read synchronises, adds the elapsed times per kernel slot into ms_out[NSNP_PROF_SLOTS] and
 * launches_out[NSNP_PROF_SLOTS], and clears the pending events.  Slots: */
enum { NSNP_PROF_READ_SCAN = 0, NSNP_PROF_PILEUP_TILE, NSNP_PROF_SELECT, NSNP_PROF_GATHER, NSNP_PROF_LSTM0, NSNP_PROF_LSTM1,
       NSNP_PROF_TAIL, NSNP_PROF_RECORDS, NSNP_PROF_VCF_TEXT, NSNP_PROF_SLOTS };
void nsnp_profile_enable(int on);
int  nsnp_profile_read(double* ms_out, int64_t* launches_out);

/* ---- status / utilities ----------------------------------------------------------------------- */
/* copies status_dev[0..3] to the host (synchronises the stream), maps it to an NSNP_E_* code and, after an error, clears it */
int nsnp_check_status(int32_t* status_dev, void* stream);

/* ---- s2 host side: VCF record formatting ----------------------------------------------------------
 * Replaces the per-site loop of PileupModel/predict.py:66-194 for ONE batch (<= batch_size sites of
 * one contig file), including its order-dependent quirks (SURVEY section 8a, row P13).  Host memory.
 *   cov8 float[n][8] = centre counts of channels [A C G T a c g t] (predict.py:63)
 * Returns the number of bytes written to out (or the negative of the required capacity).
 */
int64_t nsnp_vcf_format_batch(const char* contig, int64_t n, const int32_t* pos1, const uint8_t* refbase,
                              const float* gt_prob, const float* zy_prob, const float* cov8,
                              char* out, int64_t out_capacity);

/* ---- s2: compact site records (numeric half of predict.py:54-88 on the GPU) ---------------------------------- */
typedef struct nsnp_site_record {        /* 32 bytes */
    uint8_t gt, zy, flags, ref;          /* argmax of the two heads, NSNP_REC_* flags, centre reference base */
    int32_t pos1;                        /* 1-based position */
    int32_t q100_gt, q100_zy;            /* round(QUAL * 100) of the genotype / zygosity probability */
    int32_t depth;                       /* DP */
    int32_t af_q;                        /* AF * 1e6 rounded like '%f', or NSNP_AF_ONE / NSNP_AF_NAN / NSNP_AF_NEG_INF / negative code */
    float   p_gt, p_zy;                  /* the max probabilities (host recomputes flagged rounding ties) */
} nsnp_site_record_t;
#define NSNP_REC_DROP    1               /* predict.py would raise for this site: no record */
#define NSNP_REC_TIE_GT  2               /* QUAL within 1e-6 of a rounding tie: recompute on the host */
#define NSNP_REC_TIE_ZY  4
#define NSNP_AF_ONE      1000001
#define NSNP_AF_NAN      (-1)
#define NSNP_AF_NEG_INF  (-2)            /* '%f' of -inf (positive support over a depth of -0.0) */
/* af_q <= -3: a negative quotient (negative support: impossible for gate-passing counts, the ABI accepts any x);
 * -(af_q + 3) = |AF| * 1e6 rounded like '%f', printed with a leading '-' */
int nsnp_site_records(const float* gt_prob_dev, const float* zy_prob_dev, const int32_t* x_i32_dev, const uint8_t* refbase_dev,
                      const int32_t* pos_dev, int64_t n, const int32_t* n_dev, nsnp_site_record_t* rec_dev, void* stream);
/* the same records with the centre row read from the count tensor and the reference base from the contig (no window tensor) */
int nsnp_site_records_sites(const float* gt_prob_dev, const float* zy_prob_dev, const int32_t* counts_dev, int64_t region_start,
                            const uint8_t* ref_dev, const int32_t* pos_dev, int64_t n, const int32_t* n_dev, nsnp_site_record_t* rec_dev,
                            void* stream);
/* host: text of all records of consecutive batch_size-site batches from compact records (same bytes as the two below) */
int64_t nsnp_vcf_format_contig_records(const char* contig, int64_t n, const nsnp_site_record_t* rec, int64_t batch_size,
                                       int n_threads, char* out, int64_t out_capacity);

/* ---- s2: VCF record TEXT on the GPU (csrc/vcf_dev.cu) ---------------------------------------------------------------
 * Replaces the text half of predict.py:66-194 for records [first_index, first_index + n) of one contig file; the bytes are
 * those of nsnp_vcf_format_contig_records.  `gt_output[ti]` (predict.py:106,119) reads the genotype argmax of the first ten
 * sites of the record's batch_size-site batch:
 *   heads_dev == NULL: first_index must be a multiple of batch_size and the batch heads are taken from rec_dev itself
 *   heads_dev != NULL: u8 [n_batches][10] table of the contig (255 = the batch has no such site), filled by
 *                      nsnp_vcf_batch_heads by whoever owns those sites (multi-GPU: completed with one MIN all-reduce)
 * text_len_dev [1] int64 receives the text length (> text_capacity: nothing usable was written).  Records whose QUAL the
 * device flagged as a 2-decimal rounding tie are listed in the workspace (nsnp_vcf_text_ties); after copying text and list to
 * the host, nsnp_vcf_text_patch_ties re-evaluates them with libc -- the result is byte-identical to the host formatter. */
size_t  nsnp_vcf_text_workspace_bytes(int64_t n);
int64_t nsnp_vcf_text_capacity(int64_t n, const char* contig);     /* upper bound of the text of n records */
int nsnp_vcf_text_records(const char* contig, const nsnp_site_record_t* rec_dev, int64_t n, const int32_t* n_dev, int64_t first_index,
                          int64_t batch_size, const uint8_t* heads_dev, char* text_dev, int64_t text_capacity, int64_t* text_len_dev,
                          void* workspace_dev, size_t workspace_bytes, void* stream);
int nsnp_vcf_text_ties(const void* workspace_dev, int64_t n, const void** count_dev, const void** entries_dev, int32_t* capacity);
/* Deferred batch heads (multi-GPU streaming): the text of a region is made as soon as its records exist -- record lengths do not
 * depend on the heads -- with the one ALT character of every "fix-up" record (predict.py:101-131) left as '?' and listed
 * (16-byte entries: int64 text offset, int32 record index, u8 zygosity, u8 ref base); once the contig's batch-head table is
 * complete the host writes those characters (nsnp_vcf_text_patch_heads), then applies the tie fix-up with the table
 * (nsnp_vcf_text_patch_ties_at).  The result is byte-identical to nsnp_vcf_text_records with the table. */
int nsnp_vcf_text_records_deferred(const char* contig, const nsnp_site_record_t* rec_dev, int64_t n, const int32_t* n_dev, char* text_dev,
                                   int64_t text_capacity, int64_t* text_len_dev, void* workspace_dev, size_t workspace_bytes, void* stream);
int nsnp_vcf_text_fixups(const void* workspace_dev, int64_t n, const void** count_dev, const void** entries_dev);
int nsnp_vcf_text_patch_heads(char* text_host, int64_t text_len, const void* fix_host, int32_t n_fix, int64_t first_index, int64_t batch_size,
                              const uint8_t* heads_table, int32_t* n_drop);
int64_t nsnp_vcf_text_patch_ties_at(const char* contig, char* text_host, int64_t text_len, int64_t text_capacity, const void* ties_host,
                                    int32_t n_ties, int64_t first_index, int64_t batch_size, const uint8_t* heads_table);
int nsnp_vcf_batch_heads(const nsnp_site_record_t* rec_dev, int64_t n, const int32_t* n_dev, int64_t first_index, int64_t batch_size,
                         uint8_t* heads_dev, void* stream);
int64_t nsnp_vcf_text_patch_ties(const char* contig, char* text_host, int64_t text_len, int64_t text_capacity, const void* ties_host,
                                 int32_t n_ties);
/* host twin of the device formatter (same source compiled for the host; tests, fall-backs of the callers) */
int64_t nsnp_vcf_format_records_at(const char* contig, const nsnp_site_record_t* rec, int64_t n, int64_t first_index, int64_t batch_size,
                                   const uint8_t* heads, char* out, int64_t out_capacity);

/* Whole contig file: consecutive batches of batch_size sites (predict.py:43 DataLoader(batch_size, shuffle=False)),
 * formatted on n_threads host threads with hand-rolled number formatting (same bytes as nsnp_vcf_format_batch). */
int64_t nsnp_vcf_format_contig(const char* contig, int64_t n, const int32_t* pos1, const uint8_t* refbase,
                               const float* gt_prob, const float* zy_prob, const float* cov8, int64_t batch_size,
                               int n_threads, char* out, int64_t out_capacity);

/* ---- host: BAM records -> flat packed arrays (replaces the BAM reading samtools does for mpileup) ------------
 * `data` is the UNCOMPRESSED BAM stream (the caller inflates BGZF with zlib); first_record_offset points past the
 * header and reference list.  Two passes: count, then fill caller-allocated arrays.  Return the read count or -1. */
int64_t nsnp_bam_count(const uint8_t* data, int64_t n_bytes, int64_t first_record_offset, int32_t ref_id,
                       int64_t* n_cigar, int64_t* n_bases_padded);
int64_t nsnp_bam_fill(const uint8_t* data, int64_t n_bytes, int64_t first_record_offset, int32_t ref_id,
                      int32_t* pos, uint16_t* flag, uint8_t* mapq, int64_t* cigar_off, uint32_t* cigar, int64_t* seq_off,
                      uint8_t* seq2, uint8_t* nmask);

/* ---- host: streaming BAM reader (csrc/bam_stream.cu) -------------------------------------------------------------
 * BGZF blocks are inflated on n_threads host threads, <= 32 MB at a time, while the previous batch is parsed; records
 * are decoded contig by contig (file order) or, with a .bai next to the file, region by region through the linear
 * index, so a rank of a multi-GPU run only inflates the byte range of its own regions.  CIGAR runs of one op type are
 * merged ("1D2D" -> "3D"), '=' / IUPAC bases count as N.  The reader owns the arrays of the contig / region it decoded
 * last; nsnp_bam_take copies them into caller buffers sized from the returned counts (seq2: n_bases_padded / 4 + 16
 * bytes, nmask: n_bases_padded / 8 + 16, cigar_off: n_reads + 1).  Errors: NULL / negative return + nsnp_last_error(). */
typedef struct nsnp_bam_reader nsnp_bam_reader_t;
nsnp_bam_reader_t* nsnp_bam_open(const char* path, int n_threads);
void        nsnp_bam_close(nsnp_bam_reader_t* r);
int32_t     nsnp_bam_n_ref(const nsnp_bam_reader_t* r);
const char* nsnp_bam_ref_name(const nsnp_bam_reader_t* r, int32_t i);
int64_t     nsnp_bam_ref_len(const nsnp_bam_reader_t* r, int32_t i);
int         nsnp_bam_has_index(const nsnp_bam_reader_t* r);
int64_t     nsnp_bam_inflated_bytes(const nsnp_bam_reader_t* r);
/* next reference (file order) that has reads and whose want[ref_id] != 0 (want may be NULL = all): returns its id, -1 at
 * the end of the file, -2 on a malformed file */
int32_t nsnp_bam_next_contig(nsnp_bam_reader_t* r, const int8_t* want, int64_t* n_reads, int64_t* n_cigar, int64_t* n_bases_padded);
/* reads of ref_id that start before `end` and overlap [beg, end) (needs the .bai); returns ref_id or -2 */
int32_t nsnp_bam_fetch(nsnp_bam_reader_t* r, int32_t ref_id, int64_t beg, int64_t end, int64_t* n_reads, int64_t* n_cigar,
                       int64_t* n_bases_padded);
/* reads of ref_id that overlap any of the n ranges [beg, end) (int64 pairs, ascending and disjoint; needs the .bai), each
 * once, in file order.  Seeks through the linear index only when a range's first offset lies past what is already inflated,
 * so each needed BGZF block is inflated once.  Returns ref_id or -2. */
int32_t nsnp_bam_fetch_ranges(nsnp_bam_reader_t* r, int32_t ref_id, const int64_t* ranges, int64_t n, int64_t* n_reads,
                              int64_t* n_cigar, int64_t* n_bases_padded);
int nsnp_bam_take(nsnp_bam_reader_t* r, int32_t* pos, uint16_t* flag, uint8_t* mapq, int64_t* cigar_off, uint32_t* cigar,
                  int64_t* seq_off, uint8_t* seq2, uint8_t* nmask, int32_t* any_n);
/* HaplotypeModel s4 inputs: with keep != 0 the reader also keeps, for every record it decodes from then on, the base
 * qualities (one byte per base at the read's seq_off, 0xFF = absent), the HP:i tag (0 = none) and a 64-bit FNV-1a hash of the
 * query name; nsnp_bam_take_aux copies them out (qual: n_bases_padded bytes; hp, qname_hash: n_reads). */
int nsnp_bam_keep_aux(nsnp_bam_reader_t* r, int keep);
int nsnp_bam_take_aux(nsnp_bam_reader_t* r, uint8_t* qual, uint8_t* hp, uint64_t* qname_hash);

/* ---- synthetic inputs (bench / tests; SURVEY section 8d) --------------------------------------- */
typedef struct nsnp_synth_cfg {
    uint64_t seed_ref, seed_var, seed_reads;
    int64_t  contig_len;
    int64_t  n_reads;
    uint32_t sub_thr, ins_thr, del_thr;        /* per-base probabilities * 2^32 */
    uint32_t snp_thr;                          /* planted variant density * 2^32 */
    uint32_t lowmapq_thr, secondary_thr, supp_thr, nbase_thr, softclip_thr, long_indel_thr;
    int32_t  len_min;
    int32_t  ref_n_period, ref_n_len;          /* every period bp, a run of N in the reference (0 = none) */
    int32_t  ref_lower_period, ref_lower_len;  /* soft-masked (lower-case) runs */
    int32_t  gap_period, gap_len;              /* coverage gaps: no passing read overlaps them */
    int32_t  use_eqx;                          /* 1: emit =/X ops instead of M */
    const int32_t*  len_quantiles;             /* [1025] read reference-span quantiles */
    const uint32_t* mrun_cdf;                  /* [256]  P(match-run <= k+1) * 2^32 */
    const uint32_t* indel_cdf;                 /* [60]   P(indel len <= k+1) * 2^32 */
} nsnp_synth_cfg_t;

/* host generator (plain C loops; used by CPU tests and small cases) */
int nsnp_synth_ref_host(const nsnp_synth_cfg_t* cfg, uint8_t* ref_out);
int nsnp_synth_count_host(const nsnp_synth_cfg_t* cfg, int32_t* pos, uint16_t* flag, uint8_t* mapq,
                          int32_t* n_ops, int32_t* n_query);
int nsnp_synth_fill_host(const nsnp_synth_cfg_t* cfg, const int64_t* cigar_off, const int64_t* seq_off,
                         uint32_t* cigar, uint8_t* seq2, uint8_t* nmask);
/* device generator: same arithmetic, one thread per read (tables in cfg must be device pointers) */
int nsnp_synth_ref_dev(const nsnp_synth_cfg_t* cfg, uint8_t* ref_dev, void* stream);
int nsnp_synth_count_dev(const nsnp_synth_cfg_t* cfg, int32_t* pos, uint16_t* flag, uint8_t* mapq,
                         int32_t* n_ops, int32_t* n_query, void* stream);
int nsnp_synth_fill_dev(const nsnp_synth_cfg_t* cfg, const int64_t* cigar_off, const int64_t* seq_off,
                        uint32_t* cigar, uint8_t* seq2, uint8_t* nmask, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NANOSNP_B200_H */
