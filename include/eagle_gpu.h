/*
 * eagle_gpu.h -- C ABI of libeaglegpu.so, the B200 (sm_100a) implementation of the genome-scan
 * hot path of Eagle / WMAM v1.0.3.  This library replaces the nvblas / Makevars.gpu route
 * (reference: MyPackage/Makevars.gpu:1-2, nvblas.conf, ReadMe_GPU:57-71).  Plain pointers and
 * sizes only; no R, Rcpp, Eigen or torch types.  INTEGRATION.md shows the Rcpp glue that binds it.
 *
 * Reference paths below are relative to /root/reference/MyPackage/Eagle/.
 *
 * Conventions
 *   - every function returns EG_OK (0) or an EG_ERR_* code; eg_last_error() holds the text of the
 *     last failure on the calling thread (what the Rcpp glue passes to Rcpp::stop);
 *   - matrices crossing the ABI on the host side are column-major doubles, exactly the memory of
 *     an R numeric matrix / Eigen::MatrixXd (RcppExports.cpp:61-62 Eigen::Map is zero-copy);
 *   - `selected_loci` follows the reference: 0-based indices as doubles, element 0 == NA_real_
 *     (any NaN) means "none" (calculateMMt_rcpp.cpp:88, calculate_a_and_vara_rcpp.cpp:79);
 *   - `max_memory_in_Gbytes` and `num_cores` are accepted and ignored: GPU residency of the int8
 *     genotypes (1 byte/genotype instead of 8) replaces the host row-blocking they drive.  When the
 *     genotypes of the input file do not fit in device memory even after the path cache has been
 *     evicted, calculateMMt_rcpp, calculate_a_and_vara_rcpp, extract_geno_rcpp and createMt_ASCII_rcpp
 *     stream the file through the device piece by piece instead (eg_store_stream_file; one GPU only;
 *     nothing is cached; a non-quiet call says so) -- the reference's blocked branches, with the same
 *     results as the resident run.  A multi-GPU set, ReshapeM_rcpp, calculate_reduced_a_rcpp and
 *     the packed container still fail with EG_ERR_ALLOC then;
 *   - there is NO CPU fallback: without a usable CUDA device every compute entry point fails
 *     with EG_ERR_CUDA.
 */
#ifndef EAGLE_GPU_H_INCLUDED
#define EAGLE_GPU_H_INCLUDED

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EG_OK 0
#define EG_ERR_CUDA 1     /* CUDA runtime / cuBLAS failure, or no device */
#define EG_ERR_OPEN 2     /* "ERROR: Could not open <file>" (ReadBlock.cpp:42-45) */
#define EG_ERR_FORMAT 3   /* byte outside {'0','1','2'} or wrong line pitch (reference: undefined behaviour) */
#define EG_ERR_ARG 4      /* bad argument (null pointer, negative size, index out of range) */
#define EG_ERR_ALLOC 5    /* out of device / host memory */

/* message(...) callback of the reference's exports (Rcpp::Function message); called only on the
 * calling thread.  May be NULL. */
typedef void (*eg_message_fn)(void* ctx, const char* text);

/* ---------------------------------------------------------------- lifecycle */
int eg_init(int device);            /* bind this process/thread to one GPU; idempotent */
/* The reference's `ngpu` argument made live (R/AM.R:185-196; forced to 0 at R/AM.R:214): ONE process, one host thread per
 * GPU, NCCL (ncclCommInitAll; libnccl.so.2 is bound at run time, so single-GPU users do not depend on it).  devs == NULL:
 * devices 0 .. ngpu-1.  After this call the genotype stores built by the entry points below are sharded by markers over the
 * GPUs -- columns of M.ascii, rows of Mt.ascii, 128-aligned contiguous ranges -- and calculateMMt_rcpp,
 * calculate_a_and_vara_rcpp, extract_geno_rcpp and the eg_store_* calls work on the shards internally: every GPU decodes and
 * contracts its own markers, the partial M.Mt is summed by ONE int32 all-reduce over NVLink, S and V are uploaded once (a
 * 1/ngpu slice per GPU, exchanged over NVLink), the scan's outputs go from every GPU straight into the caller's vectors.
 * Results are bit-identical to the single-GPU ones.  Ingest, ReshapeM, the packed container and the n x n algebra run on
 * the first GPU of the set.  ngpu == 1 is eg_init(devs ? devs[0] : 0). */
int eg_init_multi(int ngpu, const int* devs);
int eg_gpu_count(void);             /* GPUs of the current set (0 before eg_init / eg_init_multi) */
int eg_shutdown(void);              /* frees every cached genotype store and workspace */
const char* eg_last_error(void);
int eg_abi_version(void);
int eg_device_count(void);          /* 0 when no CUDA device is usable */
void eg_cache_clear(void);          /* drop device-resident genotype stores keyed by file path */

/* ================================================================ reference-facing entry points
 * One per Rcpp export on the hot path; same argument order and meaning. */

/* ReadBlock(asciifname, start_row, numcols, numrows_in_block)          src/ReadBlock.cpp:16-68
 * out: numrows_in_block x numcols doubles, column-major, values -1/0/1. */
int eg_ReadBlock(const char* asciifname, int64_t start_row, int64_t numcols, int64_t numrows_in_block,
                 double* out_colmajor);

/* calculateMMt_rcpp(...)                                           src/calculateMMt_rcpp.cpp:19-185
 * dims = (n, L) of M.ascii.  out_MMt: n x n doubles (exact integers, exactly symmetric). */
int eg_calculateMMt_rcpp(const char* f_name_ascii, double max_memory_in_Gbytes, int num_cores,
                         const double* selected_loci, int64_t n_selected_loci, const int64_t* dims, int quiet,
                         eg_message_fn message, void* message_ctx, double* out_MMt);

/* calculate_a_and_vara_rcpp(...)                           src/calculate_a_and_vara_rcpp.cpp:22-241
 * f_name_ascii = Mt.ascii, dims = (L, n) of Mt.  inv_MMt_sqrt, dim_reduced_vara: n x n; a: n.
 * out_a, out_vara: L doubles each (the reference's List(a = Lx1, vara = Lx1)). */
int eg_calculate_a_and_vara_rcpp(const char* f_name_ascii, const double* selected_loci, int64_t n_selected_loci,
                                 const double* inv_MMt_sqrt, const double* dim_reduced_vara,
                                 double max_memory_in_Gbytes, const int64_t* dims, const double* a, int quiet,
                                 eg_message_fn message, void* message_ctx, double* out_a, double* out_vara);

/* calculate_reduced_a_rcpp(...)                             src/calculate_reduced_a_rcpp.cpp:20-171
 * f_name_ascii = Mt.ascii, dims = (n, L) of M (sic, :37,:71).  P: n x n, y: n.  out_ar: L doubles
 * = varG * Mt * (P * y). */
int eg_calculate_reduced_a_rcpp(const char* f_name_ascii, double varG, const double* P, const double* y,
                                double max_memory_in_Gbytes, const int64_t* dims, const double* selected_loci,
                                int64_t n_selected_loci, int quiet, eg_message_fn message, void* message_ctx,
                                double* out_ar);

/* extract_geno_rcpp(...)                                          src/extract_geno_rcpp.cpp:17-86
 * dims = (n, L) of M.ascii; selected_locus 0-based.  out: n ints in {-1,0,1}. */
int eg_extract_geno_rcpp(const char* f_name_ascii, double max_memory_in_Gbytes, int64_t selected_locus,
                         const int64_t* dims, int32_t* out);

/* ---------------------------------------------------------------- ingest (SURVEY.md section 8(f) rank 3)
 * createM_ASCII_rcpp(f_name, f_name_ascii, type, AA, AB, BB, max_memory_in_Gbytes, dims, quiet, message, missing)
 *                                                  src/createM_ASCII_rcpp.cpp:19-106, src/CreateASCIInospace.cpp:17-164
 * Whitespace-separated genotype text -> the no-space ASCII file, tokenised on the device (csrc/ingest.cu).  *ok is the
 * reference's bool: 0 after the reference's messages for an unreadable input, a token that is none of BB / AB / AA /
 * missing, or a row whose token count is not dims[1] (rows before the offending one have been written, as in the
 * reference).
 * type "PLINK": src/CreateASCIInospace_PLINK.cpp:16-248, dims = (rows, 6 + 2 * nsnp) of the ped file; the per-SNP allele
 * state machine runs on the device too.  *ok = 0 after the reference's messages for a line with a wrong token count or a
 * third allele at a locus; missing alleles ('0', '-') become heterozygotes with the reference's warning.  One deviation:
 * allele tokens longer than one character, which the reference misreads character by character (:88-93), are
 * EG_ERR_FORMAT. */
int eg_createM_ASCII_rcpp(const char* f_name, const char* f_name_ascii, const char* type, const char* AA, const char* AB,
                          const char* BB, double max_memory_in_Gbytes, const int64_t* dims, int quiet,
                          eg_message_fn message, void* message_ctx, const char* missing, int* ok);
/* createMt_ASCII_rcpp(f_name, f_name_ascii, type, max_memory_in_Gbytes, dims, quiet, message)
 *                                                                          src/createMt_ASCII_rcpp.cpp:15-245
 * f_name = M.ascii with dims = (n, L); writes its transpose Mt.ascii (L lines of n characters) to f_name_ascii: decode,
 * transpose and re-encode on the device.  Both stores stay resident under their file names, so the calculateMMt_rcpp /
 * calculate_a_and_vara_rcpp calls that follow upload nothing.  A missing input is EG_ERR_OPEN with the reference's
 * Rcpp::stop text. */
int eg_createMt_ASCII_rcpp(const char* f_name, const char* f_name_ascii, const char* type, double max_memory_in_Gbytes,
                           const int64_t* dims, int quiet, eg_message_fn message, void* message_ctx);

/* ReshapeM_rcpp(fnameM, fnameMt, indxNA, dims)                                    src/ReshapeM_rcpp.cpp:16-117
 * dims = (n, L) of M.ascii; indxNA: 0-based individuals whose trait is NA, in decreasing order as R passes them.  Writes
 * <fnameM>tmp without those lines and <fnameMt>tmp with those characters erased from every line (erased one after the
 * other, as the reference does); newdims[0] = lines kept, newdims[1] = L.  A row / column gather of the resident stores
 * and the ASCII encoder; the reshaped stores stay resident under the two new file names.  A missing file is EG_ERR_OPEN
 * with the reference's Rcpp::stop text. */
int eg_ReshapeM_rcpp(const char* fnameM, const char* fnameMt, const int64_t* indxNA, int64_t n_indx, const int64_t* dims,
                     int64_t* newdims);
/* getRowColumn(fname)                                                              src/getRowColumn.cpp:19-72
 * dimen[0] = lines of the file (an unterminated last line counts), dimen[1] = whitespace-separated tokens of line 1. */
int eg_getRowColumn(const char* fname, int64_t* dimen);

/* ================================================================ resident genotype stores
 * A store is a decoded genotype matrix held in HBM as int8, `rows` x `cols`, holding the NEGATED reference value
 * 1 - code (AA = +1, AB = 0, BB = -1; csrc/decode.cu explains why: power); every entry point that returns genotypes or
 * signed projections undoes the sign.  It is laid out in one of
 * two layouts:
 *   row-major  (Mt orientation: markers as rows; what the scan reads): row pitch `pitch` bytes
 *              (multiple of 128, > cols; the tail of every row is zero);
 *   K-blocked  (M orientation: individuals as rows; what M.Mt streams): [ceil(cols/128)][rows][128]
 *              bytes, i.e. all rows of one 128-marker block are contiguous; eg_store_info reports
 *              pitch == 0 for it.
 * eg_store_from_host_ascii / eg_store_from_file build the K-blocked layout, eg_store_from_host_ascii_rows
 * and eg_store_transpose the row-major one.  The entry points above keep stores in a cache keyed by
 * (path, size, mtime, dims, layout); these calls manage them explicitly (host buffers in, handles out). */
typedef struct eg_store eg_store_t;

/* `image` is a byte-exact no-space ASCII file image in host memory (CreateASCIInospace.cpp:119-122):
 * `rows` lines of `cols` chars + '\n'.  Only columns [col0, col1) are transferred and decoded (a
 * marker shard when the image is M.ascii); pass 0, cols for everything. */
int eg_store_from_host_ascii(const uint8_t* image, int64_t rows, int64_t cols, int64_t col0, int64_t col1,
                             eg_store_t** out);
int eg_store_from_file(const char* path, int64_t rows, int64_t cols, int64_t col0, int64_t col1, eg_store_t** out);
/* rows [row0,row1) of the image (a marker shard when the image is Mt.ascii) */
int eg_store_from_host_ascii_rows(const uint8_t* image, int64_t rows, int64_t cols, int64_t row0, int64_t row1,
                                  eg_store_t** out);
int eg_store_transpose(const eg_store_t* in, eg_store_t** out); /* replaces createMt_ASCII_rcpp.cpp:99 on device */
/* SURVEY.md section 8(f) rank 2: the packed 2-bit container of the pre-CRAN code (RcppFunctions.cpp.gpu:224-345,
 * CreatePackedBinary): per row ceil(cols/32) little-endian uint64, genotype k in bits 2(k%32).. of word k/32, codes 0/1/2
 * as in the ASCII file.  4x fewer bytes over PCIe / from disk than the ASCII image.  csrc/pack2.cu. */
/* SURVEY.md section 8(f) rank 3 (half of it): ReshapeM as a device mask instead of rewriting both ASCII files
 * (src/ReshapeM_rcpp.cpp:59-109).  idx: 0-based individuals to drop -- rows of an M store (individuals_are_rows != 0) or
 * columns of a row-major Mt store. */
int eg_store_drop_individuals(const eg_store_t* in, const int64_t* idx, int64_t k, int individuals_are_rows, eg_store_t** out);
int eg_dev_gather_rows(const int8_t* d_in, int64_t in_rows, int64_t cols, int64_t in_pitch, const int64_t* d_map, int64_t out_rows,
                       int8_t* d_out, int64_t out_pitch, void* stream);
int eg_dev_gather_cols(const int8_t* d_in, int64_t rows, int64_t in_pitch, const int64_t* d_map, int64_t out_cols, int8_t* d_out,
                       int64_t out_pitch, void* stream);
int64_t eg_packed_words_per_row(int64_t cols);
int eg_store_from_host_packed(const uint64_t* words, int64_t rows, int64_t cols, int kblocked, eg_store_t** out);
int eg_store_to_host_packed(const eg_store_t* s, uint64_t* out_words);
int eg_dev_pack_2bit(const int8_t* d_store, int64_t rows, int64_t cols, int64_t pitch, uint64_t* d_words, void* stream);
int eg_dev_unpack_2bit(const uint64_t* d_words, int64_t rows, int64_t cols, int8_t* d_store, int64_t pitch, int32_t* d_err,
                       void* stream);
/* PLINK 1 binary genotypes: a .bed file (with its .bim, one line per SNP, and .fam, one line per individual) straight into
 * a store, 4 genotypes per byte over PCIe instead of 1 (csrc/bed.cu).  The format read:
 *   header    0x6C 0x1B 0x01 (SNP-major).  Refused with EG_ERR_FORMAT: mode byte 0x00 (individual-major), any other magic,
 *             and (files) a size that is not exactly 3 + L * ceil(n/4);
 *   layout    SNP j in bytes 3 + j*bpr .. 3 + (j+1)*bpr - 1, bpr = ceil(n/4); individual i of it is
 *             v = (byte[i/4] >> 2*(i%4)) & 3.  The bits past individual n-1 in a SNP's last byte are ignored;
 *   values    v = 0 homozygous for the first .bim allele (A1) -> code 0 (AA, store +1); v = 2 heterozygous -> code 1 (AB,
 *             store 0); v = 3 homozygous A2 -> code 2 (BB, store -1); v = 1 missing -> code 1, a heterozygote, as missing
 *             text tokens and ped alleles are read.  Swapping A1 / A2 of a SNP negates its column: M.Mt, var(a) and the
 *             picks do not change, a and extracted genotypes change sign.
 * n and L come from the line counts of .fam and .bim (eg_getRowColumn); names and positions stay with the map file.
 * SNPs [snp0, snp1) make the store (a marker shard; 0, L for everything); kblocked != 0: the K-blocked M store
 * (n x (snp1 - snp0)), else the row-major Mt store ((snp1 - snp0) x n).  *n_missing (may be NULL): missing genotypes read.
 * Header, size and ranges are checked before any device work.  The bytes go through the page-locked staging ring in
 * pieces (pread for the file), each piece decoded while the next is copied; with eg_init_multi every GPU pulls and decodes
 * only its own SNP range (one contiguous byte range of the file).  `image` is the whole file image, header included. */
int eg_store_from_bed(const char* path, int64_t n, int64_t L, int64_t snp0, int64_t snp1, int kblocked, int64_t* n_missing,
                      eg_store_t** out);
int eg_store_from_host_bed(const uint8_t* image, int64_t n, int64_t L, int64_t snp0, int64_t snp1, int kblocked,
                           int64_t* n_missing, eg_store_t** out);
/* A .bed file -> M.ascii (n lines of L characters) and Mt.ascii (L lines of n), byte-identical to what the text readers
 * write for the same genotypes; both stores stay in the path cache under those names, so the calculateMMt_rcpp /
 * calculate_a_and_vara_rcpp calls that follow upload nothing.  How an R user brings a .bed file to AM(). */
int eg_bed_to_ascii(const char* bed_path, int64_t n, int64_t L, const char* M_ascii, const char* Mt_ascii);
/* Streamed stores: genotype sets larger than device memory.  The handle holds the source and no genotype bytes on the
 * device; every call that reads it stages the source in pieces of whole 128-marker blocks (EAGLE_INGEST_PIECE_BYTES source
 * bytes at most, 256 MB by default) through the page-locked ring and decodes each piece while the next is copied, with the
 * same decoders as the resident uploads.  Results are bit-identical to the resident store's.
 *   source       eg_store_stream_file: M.ascii (kblocked != 0, rows = n, cols = L) or Mt.ascii (kblocked == 0, rows = L,
 *                cols = n), checked as eg_store_from_file checks it; _bed / _host_bed: SNPs [snp0, snp1) of a .bed file or
 *                image, checked as eg_store_from_bed / eg_store_from_host_bed check them, in either orientation.  A file
 *                stays open for the handle's life; a host image must outlive the handle.
 *   accepted     eg_store_info (device_ptr == NULL; rows, cols and pitch of the resident store), eg_store_mmt and
 *                eg_store_extract_col on M (kblocked), eg_store_a_and_vara on Mt (the slices of U are made once per call,
 *                and eg_last_scan_kernel reports the sum over the pieces).  An ASCII format error in any piece is
 *                EG_ERR_FORMAT with the resident upload's text.  Its "near row, column" names the decoder unit that
 *                saw the byte: the same position as the resident upload for Mt.ascii; for M.ascii, whose column pieces
 *                are decoded in other units than the resident upload's whole rows, a unit that holds the byte too.
 *   refused      eg_store_transpose, eg_store_drop_individuals, eg_store_to_host_packed: EG_ERR_ARG.
 *   one GPU      under eg_init_multi with more than one GPU the constructors return EG_ERR_ARG. */
int eg_store_stream_file(const char* path, int64_t rows, int64_t cols, int kblocked, eg_store_t** out);
int eg_store_stream_bed(const char* path, int64_t n, int64_t L, int64_t snp0, int64_t snp1, int kblocked, eg_store_t** out);
int eg_store_stream_host_bed(const uint8_t* image, int64_t n, int64_t L, int64_t snp0, int64_t snp1, int kblocked,
                             eg_store_t** out);
int eg_store_free(eg_store_t* s);
int eg_store_info(const eg_store_t* s, int64_t* rows, int64_t* cols, int64_t* pitch, void** device_ptr);

/* M.Mt of a store holding M (n x L_shard), with optional zeroed columns (store-local indices).
 * out_MMt_host: n x n doubles. */
int eg_store_mmt(const eg_store_t* M, const int64_t* zero_cols, int64_t n_zero, double* out_MMt_host);
/* a / vara scan of a store holding Mt (L_shard x n); zero_rows are store-local. */
int eg_store_a_and_vara(const eg_store_t* Mt, const int64_t* zero_rows, int64_t n_zero, const double* inv_MMt_sqrt,
                        const double* dim_reduced_vara, const double* a, double* out_a, double* out_vara);
int eg_store_extract_col(const eg_store_t* M, int64_t col, int32_t* out);

/* ================================================================ device-level entry points
 * Device pointers + a CUDA stream (cudaStream_t passed as void*, NULL = default stream).  Used by
 * the host-level calls above, by bench.py (inputs resident in HBM) and by the multi-GPU
 * plumbing, which owns the buffers and runs the NCCL all-reduce between eg_dev_syrk_i8 and
 * eg_dev_mmt_finalize. */

/* K1: ASCII bytes -> int8.  src byte (r,c) at src + r*src_pitch + c; writes dst[r*dst_pitch + c] = byte - '1'
 * for c < cols and 0 for cols <= c < dst_pitch.  src must be readable up to src_bytes_avail (>= the
 * last needed byte, ideally +32).  d_err: 4 ints, [0] != 0 when a byte outside {'0','1','2'} was seen. */
int eg_dev_decode(const uint8_t* d_src, int64_t src_pitch, int64_t src_bytes_avail, int64_t rows, int64_t cols,
                  int8_t* d_dst, int64_t dst_pitch, int32_t* d_err, void* stream);
int eg_dev_transpose_i8(const int8_t* d_in, int64_t rows, int64_t cols, int64_t in_pitch, int8_t* d_out,
                        int64_t out_pitch, void* stream);
/* K-blocked variants: the store is [ceil(cols/128)][kb_rows][128] bytes; decode fills rows [row0, row0+rows). */
int eg_dev_decode_kb(const uint8_t* d_src, int64_t src_pitch, int64_t src_bytes_avail, int64_t rows, int64_t cols,
                     int8_t* d_dst, int64_t kb_rows, int64_t row0, int32_t* d_err, void* stream);
/* .bed SNP rows -> store (format: eg_store_from_bed).  d_snps: nsnp rows of ceil(n/4) bytes at any alignment; they become
 * markers [m0, m0 + nsnp) of a store of dst_rows_or_L markers, pads written as eg_dev_decode / eg_dev_decode_kb write them.
 * dst_pitch > 0: row-major Mt store (row pitch, multiple of 128, >= n); dst_pitch == 0: K-blocked M store
 * [ceil(L/128)][n][128] with L = dst_rows_or_L, where m0 is a multiple of 128 and nsnp is one too unless the piece ends at
 * L.  *d_missing (may be NULL) += the missing genotypes of the piece. */
int eg_dev_decode_bed(const uint8_t* d_snps, int64_t n, int64_t nsnp, int8_t* d_dst, int64_t dst_rows_or_L, int64_t dst_pitch,
                      int64_t m0, uint64_t* d_missing, void* stream);
int eg_dev_transpose_kb_i8(const int8_t* d_in_kb, int64_t rows, int64_t cols, int8_t* d_out, int64_t out_pitch,
                           void* stream);
int eg_dev_syrk_i8_kb(const int8_t* d_Mkb, int64_t n, int64_t kcols, int32_t* d_C, int64_t ldc, void* stream);
/* K2: C (int32, n x n row-major, ld = ldc, must be zeroed by the caller) += M * M^T over columns
 * [0, kcols) of M (int8 n x kcols, row pitch multiple of 128 and padded with zeros).  Only entries
 * with col >= row are complete.  M holds genotypes in {-1, 0, +1}: by default both entry points copy
 * it to E2M1 (a pool block of half its bytes) for the block-scaled FP4 kernel; EAGLE_MMT_MODE=i8
 * contracts the int8 bytes themselves. */
int eg_dev_syrk_i8(const int8_t* d_M, int64_t n, int64_t kcols, int64_t pitch, int32_t* d_C, int64_t ldc,
                   void* stream);
/* C[r][c] -= sum_s M[r][zero_cols[s]] * M[c][zero_cols[s]]  (calculateMMt_rcpp.cpp:88-92 as a rank-k fix) */
int eg_dev_syrk_zero_cols(const int8_t* d_M, int64_t n, int64_t pitch, const int64_t* h_zero_cols, int64_t n_zero,
                          int32_t* d_C, int64_t ldc, void* stream);
/* mirror the upper triangle and convert: out (n x n doubles, column-major == row-major, symmetric) */
int eg_dev_mmt_finalize(const int32_t* d_C, int64_t n, int64_t ldc, double* d_out, void* stream);

/* K3 pre-products (calculate_a_and_vara_rcpp.cpp:90, 97-98): v = S*a; W = S*(V*S); packed for K3.
 * d_S, d_V: n x n column-major doubles; d_a: n.  d_Wp: eg_scan_wp_elems(n) doubles;
 * d_tmp: n*n doubles scratch. */
int64_t eg_scan_wp_elems(int64_t n);
int eg_dev_scan_prepare(const double* d_S, const double* d_V, const double* d_a, int64_t n, double* d_tmp,
                        double* d_Wp, void* stream);
/* The same in steps, for marker-sharded multi-GPU runs: each rank computes the columns [col0,col1) of W
 * (d_tmp: n*(col1-col0) doubles; d_Wp zeroed by the caller), the column blocks are exchanged between the
 * ranks (broadcast / all-gather of contiguous ranges of d_Wp: column c starts at d_Wp + c*round_up(n,32)),
 * then every rank folds the complete W.  When S and V are symmetric (eg_dev_inputs_symmetric: to 1e-13 of
 * their largest entry -- always the case under AM()) W is symmetric and `upper_only` / `w_is_upper` restrict
 * the second product to rows 0..col1-1 (3 n^3 instead of 4 n^3 flops). */
/* 1 when the n^3 pre-products of symmetric inputs run as exact int8 digit-slice products (deterministic for any column
 * split), 0 when they are two library DGEMMs (n < 512, or EAGLE_PREP_MODE=f64): sharded callers split the columns of W only
 * in the first case. */
int eg_prep_uses_i8(int64_t n);
int eg_dev_symmetry(const double* d_A, int64_t n, double* max_abs, double* max_asym, void* stream);
int eg_dev_inputs_symmetric(const double* d_S, const double* d_V, int64_t n, int* yes, void* stream);
int eg_dev_scan_prepare_cols(const double* d_S, const double* d_V, int64_t n, int64_t col0, int64_t col1,
                             int upper_only, double* d_tmp, double* d_Wp, void* stream);
int eg_dev_scan_fold(const double* d_S, const double* d_a, int64_t n, int w_is_upper, double* d_Wp, void* stream);
/* K3: a = Mt*v, vara_j = (Mt*W)_j . Mt_j for marker rows of an Mt store (L x n int8, pitch >=
 * round_up(n+1,128)); zero rows get a = vara = 0. */
int eg_dev_scan(const int8_t* d_Mt, int64_t L, int64_t n, int64_t pitch, const double* d_Wp,
                const int64_t* h_zero_rows, int64_t n_zero, double* d_a, double* d_vara, void* stream);
/* K5: tsq = a^2/vara; maximum ignoring NaN and lowest index attaining it (find_qtl.R:71-80).
 * d_out: {max tsq (double), index (int64 bits in a double slot)}; index -1 if all NaN. */
int eg_dev_argmax_tsq(const double* d_a, const double* d_vara, int64_t L, double* d_best, int64_t* d_best_idx,
                      void* stream);
/* y = scale * Mt * x  (calculate_reduced_a_rcpp.cpp:82-84 second product) */
int eg_dev_gemv_i8(const int8_t* d_Mt, int64_t L, int64_t n, int64_t pitch, const double* d_x, double scale,
                   double* d_y, void* stream);
/* pitch == 0 selects the K-blocked layout in the two calls below (and in eg_dev_syrk_zero_cols) */
int eg_dev_extract_col(const int8_t* d_M, int64_t n, int64_t pitch, int64_t col, int32_t* d_out, void* stream);

/* Tokeniser of CreateASCIInospace.cpp:67-125 on a text resident in HBM.  d_text: nbytes of text at a 16-byte aligned
 * address, readable for 32 bytes beyond nbytes.  Work is cut into eg_tokenise_chunks(nbytes) chunks of
 * eg_tokenise_chunk_bytes() bytes.  _scan: d_counts = 2 * chunks uint32 of scratch; d_prefix = 2 * (chunks + 1) int64:
 * (tokens, '\n' bytes) before each chunk, the last pair = totals.  _emit: d_out = out_rows * (cols + 1) bytes; *d_err_pos
 * (set to UINT64_MAX by the caller) receives the smallest byte position of an error event: the start of a token that is
 * none of the codes, or the '\n' (nbytes for an unterminated last line) that closes a row without exactly `cols` tokens. */
int64_t eg_tokenise_chunks(int64_t nbytes);
int64_t eg_tokenise_chunk_bytes(void);
int eg_dev_tokenise_scan(const uint8_t* d_text, int64_t nbytes, uint32_t* d_counts, int64_t* d_prefix, void* stream);
int eg_dev_tokenise_emit(const uint8_t* d_text, int64_t nbytes, const int64_t* d_prefix, int64_t cols, const char* AA,
                         const char* AB, const char* BB, const char* missing, uint8_t* d_out, int64_t out_rows,
                         uint64_t* d_err_pos, void* stream);
/* PLINK ped files (CreateASCIInospace_PLINK.cpp:78-196) in two stages.  _alleles: token 6 + k of every line (ncols = 6 +
 * 2 * nsnp tokens per line) -> d_alleles[row * (ncols - 6) + k]; *d_err_pos as above (a line whose token count is not
 * ncols, or an allele token longer than one character).  _genotypes: the per-SNP allele state machine over `rows` rows ->
 * rows * (nsnp + 1) bytes of no-space ASCII; d_state = 2 * nsnp bytes carried between the pieces of a file (first_piece
 * != 0 initialises it from row 0); d_keys = 2 x uint64 set to UINT64_MAX by the caller: [0] the smallest
 * (row_base + row) * nsnp + snp at which a third allele appears, [1] the same for the first missing allele. */
int eg_dev_ped_alleles(const uint8_t* d_text, int64_t nbytes, const int64_t* d_prefix, int64_t ncols, uint8_t* d_alleles,
                       int64_t out_rows, uint64_t* d_err_pos, void* stream);
int eg_dev_ped_genotypes(const uint8_t* d_alleles, int64_t rows, int64_t nsnp, int first_piece, int64_t row_base,
                         uint8_t* d_state, uint8_t* d_out, uint64_t* d_keys, void* stream);
/* Rows [row0, row0 + nrows) of a row-major int8 store as no-space ASCII ('0' + code, '\n' after each row):
 * nrows * (cols + 1) bytes at d_out (16-byte aligned).  The writer of createMt_ASCII_rcpp.cpp:104-118. */
int eg_dev_encode_ascii(const int8_t* d_store, int64_t pitch, int64_t cols, int64_t row0, int64_t nrows, uint8_t* d_out,
                        void* stream);

/* Bench / test utility: write a synthetic M.ascii image (rows x (cols+1) bytes, Binomial(2,p_j)
 * genotypes from a counter-based hash; same bytes as eagleeverything_b200/synth.py) into device memory.
 * Column c is marker col_offset + c, row r is individual row_offset + r of an n_total-individual data set. */
int eg_dev_synth_ascii(uint8_t* d_img, int64_t rows, int64_t cols, int64_t col_offset, int64_t n_total,
                       int64_t row_offset, uint64_t seed, void* stream);

/* ------------------------------------------------------------------------------------------------
 * SURVEY.md section 8(f) rank 1: the n x n FP64 algebra between two scans (base-R LAPACK/BLAS in the
 * reference).  Matrices are n x n column-major doubles as R holds them; X is n x q.  csrc/algebra.cu.
 * ------------------------------------------------------------------------------------------------ */
/* R/calculateMMt_sqrt_and_sqrtinv.R:1-52.  *ok = 0 after the reference's messages when MMt is not positive
 * definite (R returns NULL); an asymmetric MMt is an error as in matrixcalc::is.positive.definite. */
int eg_calculateMMt_sqrt_and_sqrtinv(const double* MMt, int64_t n, int checkres, eg_message_fn message, void* message_ctx,
                                     double* out_sqrt, double* out_invsqrt, int* ok);
/* R/calculateH.R:1-38: H = varE I + varG MMt; *ok = 0 with the reference's message for a negative variance. */
int eg_calculateH(const double* MMt, int64_t n, double varE, double varG, eg_message_fn message, void* message_ctx,
                  double* out_H, int* ok);
/* R/calculateP.R:1-32 */
int eg_calculateP(const double* H, const double* X, int64_t n, int q, double* out_P);
/* R/calculate_reduced_a.R:1-35: varG * MMtsqrt %*% P %*% y */
int eg_calculate_reduced_a(double varG, const double* P, const double* MMtsqrt, const double* y, int64_t n, double* out_a);
/* R/calculate_reduced_vara.R:1-38 (invMMt is only used for its dimension there: pass n) */
int eg_calculate_reduced_vara(const double* X, int64_t n, int q, double varE, double varG, const double* MMtsqrt, double* out_V);
/* EMMA's eigendecompositions (the rcppMagmaSYEVD hooks the reference left commented out):
 * R/emma_eigen_L_wo_Z.R:9 -- eigen(K, symmetric=TRUE), values decreasing; out_vectors may be NULL;
 * R/emma_eigen_R_wo_Z.R:4-20 -- eigen(S (K+I) S): values[1:(n-q)] - 1 and the first n-q vectors (n x (n-q)).
 * Eigenvectors are determined up to sign (and up to rotation inside a repeated eigenvalue), as in LAPACK. */
int eg_emma_eigen_L_wo_Z(const double* K, int64_t n, double* out_values, double* out_vectors);
int eg_emma_eigen_R_wo_Z(const double* K, const double* X, int64_t n, int q, double* out_values, double* out_vectors);
/* device-level forms (device pointers, caller-provided scratch; see csrc/algebra.cu for the sizes) */
int eg_dev_eigen_sym(double* d_A, int64_t n, double* d_values, void* stream);
int eg_dev_emma_SKS(const double* d_K, const double* d_X, int64_t n, int q, double* d_out, double* d_tmp, double* d_small,
                    void* stream);
/* emma.eigen.R.wo.Z with everything resident: d_U (n x n) <- eigenvectors of S (K + I) S (R keeps the first n - q),
 * d_values[0, n-q) <- eigenvalues - 1, and d_etas[0, n-q) <- U[, 1:(n-q)]^T y when d_y / d_etas are given (both or
 * neither).  d_w1, d_w2: n*n doubles of scratch each; d_small: 2*n*q + 2*q*q doubles. */
int eg_dev_emma_eigen_R_wo_Z(const double* d_K, const double* d_X, const double* d_y, int64_t n, int q, double* d_values,
                             double* d_etas, double* d_U, double* d_w1, double* d_w2, double* d_small, void* stream);
int eg_dev_sqrt_and_sqrtinv(const double* d_K, int64_t n, double* d_sqrt, double* d_invsqrt, double* d_tmp, int* not_pd,
                            double* trace_check, void* stream);
int eg_dev_calculateH(const double* d_K, int64_t n, double varE, double varG, double* d_H, void* stream);
int eg_dev_calculateP(const double* d_H, const double* d_X, int64_t n, int q, double* d_P, double* d_small, void* stream);
int eg_dev_calculate_reduced_a(double varG, const double* d_P, const double* d_sqrt, const double* d_y, int64_t n,
                               double* d_tmp_n, double* d_out, void* stream);
int eg_dev_calculate_reduced_vara(const double* d_X, int q, double varE, double varG, const double* d_sqrt, int64_t n,
                                  double* d_V, double* d_D, double* d_small, void* stream);

/* ------------------------------------------------------------------------------------------------
 * The same algebra in the basis of eigen(K), csrc/eigbasis.cu + csrc/secular.cuh.  K = MMt/max(MMt) + 0.95 I is fixed after
 * the first forward iteration (R/AM.R:414-423): with K = U diag(xi) U^T computed once (eg_dev_eigen_sym), H^-1, K^+-1/2 and
 * D^-1 are diagonal in U and P, V are diagonal + rank q, so an iteration costs O(q n^2) + ONE n^3 product instead of the
 * reference's dense eigendecomposition, three dense inversions and ~10 n^3 products.
 * ------------------------------------------------------------------------------------------------ */
/* emma.eigen.R.wo.Z (R/emma_eigen_R_wo_Z.R:7-20) followed by etas = t(vectors) %*% y (R/emma_REMLE.R:40), given
 * xi[n] = eigen(K)$values (any order), Xt = U^T X (n x q column-major) and yt = U^T y in the same order: the n - q
 * non-trivial eigenvalues of S (K + I) S minus 1 (decreasing) and the matching etas (up to sign), by q rank-one
 * compressions of the diagonal solved through their secular equations on the device -- O(q n^2), no n x n matrix.
 * Host pointers.  stats4 (may be NULL): compressions done, poles deflated, worst root-finder iteration count, roots. */
int eg_emma_eigen_R_wo_Z_eigbasis(const double* xi, const double* Xt, const double* yt, int64_t n, int q, double* out_values,
                                  double* out_etas, int64_t* stats4);
/* seconds of the calling thread's last secular solve: [0] inside the device back end, [1] the whole call */
int eg_last_secular_times(double* out2);
int eg_dev_transpose_f64(const double* d_in, int64_t n, double* d_out, void* stream);
/* d_out (n x r) = U^T d_in (to_eigenbasis != 0) or U d_in */
int eg_dev_eigbasis_apply(const double* d_U, int64_t n, const double* d_in, int r, int to_eigenbasis, double* d_out, void* stream);
/* The scan's right-hand side (what eg_dev_scan_prepare builds from S, V, a) from eigenbasis quantities:
 * W = U diag(w) U^T - E E^T with E = U Et (n x q, q may be 0), folded into d_Wp; v = U vt into its column n.
 * d_Ut = U^T (eg_dev_transpose_f64).  d_work: n * max(q,1) doubles; d_work2: n*n doubles, only read when the product runs
 * in FP64 (n < 512, or the digit slices do not fit) and may be NULL otherwise. */
int eg_dev_scan_prepare_eig(const double* d_U, const double* d_Ut, int64_t n, const double* d_w, const double* d_Et, int q,
                            const double* d_vt, double* d_work, double* d_work2, double* d_Wp, void* stream);

/* The scan from a cached projection (am.AM_resident's bcache route): K is fixed for the whole search, so B = M^T U (U the
 * eigenvectors of K; L x n doubles, row pitch ldb) is computed ONCE by the int8 digit-slice contraction in projection mode
 * (one rounding per entry); afterwards var(a)_j = sum_k w_k B_jk^2 - sum_c e_cj^2 with e_c = Mt E_c (eg_dev_gemv_i8) is one
 * HBM-bound pass over B instead of the n^2 L contraction per forward iteration.  d_e: q x L row-major; d_tmp_L: L doubles. */
int eg_dev_project_i8(const int8_t* d_Mt, int64_t L, int64_t n, int64_t pitch, const double* d_U, double* d_B, int64_t ldb,
                      void* stream);
int eg_dev_bscan(const double* d_B, int64_t L, int64_t n, int64_t ldb, const double* d_w, const double* d_e, int q,
                 double* d_tmp_L, double* d_vara, void* stream);

/* How var(a) is contracted (same result within the stated tolerance, both deterministic):
 *   1  exact int8 slices of U on the tcgen05 int8 tensor cores, scan_i8.cu -- the default;
 *   0  FP64 tensor cores (DMMA), scan_f64.cu (also: environment EAGLE_SCAN_MODE=f64). */
int eg_set_scan_mode(int mode);
int eg_get_scan_mode(void);
/* Digits (balanced base-256, int8) that mode 1 keeps of every column of the folded matrix U:
 *   7 (default)  the full significand of the column's largest entry, one rounding per entry of Mt U: more accurate than the
 *       FP64 accumulation it replaces;
 *   6 (EAGLE_SCAN_DIGITS=6)  47 bits + sign: truncation <= 2^(e_k - 48) per entry, exact accumulation and recombination --
 *       inside an FP64 GEMM's worst-case bound, five orders of magnitude inside the 1e-9 tolerance, 5 % faster. */
int eg_set_scan_digits(int digits);
int eg_get_scan_digits(void);
/* Device time of the dominant kernel of the last eg_dev_scan (scan_i8_kernel or scan_f64_kernel),
 * measured with CUDA events on its stream, and the arithmetic operations it executed. */
int eg_last_scan_kernel(double* ms, double* ops);

/* Device time (CUDA events) and executed int8 operations of the prep_i8_kernel launches of the last
 * eg_dev_scan_prepare / eg_dev_scan_prepare_cols; ms = 0 when the cuBLAS path ran. */
int eg_last_prep_kernels(double* ms, double* ops);
/* Kernels launched by this library in this process so far (bench.py reports the difference over its timed region). */
long long eg_launch_count(void);

/* timing of the last host-level call, milliseconds per stage (h2d, decode, syrk, finalize, d2h,
 * prepare, scan); n_out entries written. */
int eg_last_timing(double* out_ms, int n_out);

#ifdef __cplusplus
}
#endif
#endif /* EAGLE_GPU_H_INCLUDED */
