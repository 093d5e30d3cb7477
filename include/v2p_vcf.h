/*
 * v2p_vcf.h -- VCF sample columns on the device: plain VCF text in, the FORMAT/BCSQ mask matrix out.
 *
 * The matrix is the `masks[record][sample][word]` input of v2p_sites_from_masks (include/v2p_taskgen.h),
 * v2p_pipeline_run_masks (include/v2p_pipeline.h) and v2p_cohort_run_masks (include/v2p_cohort.h); pass it with
 * V2P_FLAG_DEVICE_PTRS (pipeline: mask_flags; cohort: V2P_COHORT_DEVICE_MASKS).  It replaces the reference's per-cell
 * text parse (readers.rs, get_bit_mask in text_parser.rs:163-194) and the per-sample transpose in front of the mask
 * decode (get_patient_fields, vcf_ds.rs:126-213).
 *
 * The work has two phases, and the host does its per-record work between them on its own copy of the text:
 *   v2p_vcf_load         upload (or borrow) the text and index it: line table, the #CHROM line, where each data line's
 *                        sample cells begin.  Columns 1-9 of a data line are text[line_begin, cells_begin): the host
 *                        reads INFO/BCSQ there, keeps the records it supports and maps their consequences to catalogue
 *                        sites (per record, not per sample).
 *   v2p_vcf_parse_masks  parse the sample cells of the chosen data lines into the mask matrix.
 * A bgzip'd file (.vcf.gz) goes in through v2p_vcf_load_bgzf (include/v2p_vcf_bgzf.h) instead of v2p_vcf_load: it is
 * inflated on the device, and the host gets columns 1-9 of every data line back, since it has no text of its own.
 *
 * Dialect (the minimal VCF the reference reads, SURVEY.md section 8c):
 *   - Lines end at '\n'; a '\r' that ends a line is not part of it; a last line without '\n' counts.
 *   - Lines starting with '#' are headers; the first line starting with "#CHROM" defines n_samples = its columns after
 *     FORMAT (the 9th column).  A text without a #CHROM line is V2P_ERR_VCF_PARSE.  Empty lines are skipped.
 *   - Every other line is a data line.  Its cells are the tab-separated columns 10 onwards.
 *   - The mask of a cell is its last ':'-separated field, or the whole cell when it has no ':'.  A mask is one or more
 *     ','-separated words; a word is one or more ASCII digits with a value <= 2^32-1.
 *   - A selected data line is V2P_ERR_VCF_PARSE when it has a number of cells other than n_samples, or a mask with an
 *     empty word, a word with any other character ('.', a sign, a space) or a word that overflows.  The message names
 *     the 1-based line number of the file and the 1-based sample column; of several errors the first in file order
 *     (lowest line, then lowest sample column) is reported, whatever the thread timing.
 *   The reference's own handling of malformed cells is not pinned by anything this project can run, so the library
 *   refuses such cells and says where they are instead of guessing a meaning for them.  Lines that are not selected are
 *   never read past their 9th column.
 *
 * Threading: one call at a time per object (like a catalogue); objects on different devices are independent.
 */
#ifndef V2P_VCF_H
#define V2P_VCF_H

#include <stddef.h>
#include <stdint.h>

#include "v2p_engine.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct v2p_vcf v2p_vcf;

int v2p_vcf_create(int cuda_device, v2p_vcf** out);
void v2p_vcf_destroy(v2p_vcf* v);
/* Message of the last failure on this object ("" if none).  Valid until the next call on `v`. */
const char* v2p_vcf_last_error(v2p_vcf* v);

typedef struct {
    uint64_t n_samples;                 /* columns after FORMAT on the #CHROM line                               */
    uint64_t header_begin, header_end;  /* byte range of the #CHROM line (the host splits out the sample names)   */
    uint64_t n_lines;                   /* data lines: non-empty lines that do not start with '#', in file order  */
    const uint64_t* line_begin;         /* host memory owned by v, n_lines: offset of the line's first byte       */
    const uint64_t* cells_begin;        /* offset of its first sample cell (after the 9th tab); the line end if it
                                           has fewer columns.  text[line_begin, cells_begin) = columns 1-9         */
    uint64_t h2d_bytes;                 /* bytes uploaded (0 for device text)                                      */
    float h2d_ms, index_ms;             /* device time of the upload and of the index kernels (CUDA events)        */
} v2p_vcf_lines;

/* Upload the text (host memory; pinned for the full PCIe rate, as for `out` elsewhere in the ABI) or borrow it
 * (flags = V2P_FLAG_DEVICE_PTRS: device memory on v's device, 16-byte aligned, valid until the next load / destroy),
 * then index it.  Errors: V2P_ERR_VCF_PARSE (no #CHROM line), V2P_ERR_INVALID_ARG, V2P_ERR_CUDA. */
int v2p_vcf_load(v2p_vcf* v, const uint8_t* text, uint64_t n_bytes, uint32_t flags, v2p_vcf_lines* out);

typedef struct {
    const uint32_t* masks;      /* device, [n_records][n_samples][words_per_cell], owned by v until the next call */
    uint64_t n_records, n_samples;
    uint32_t words_per_cell;    /* widest cell among the selected lines (>= 1); narrower cells are zero-padded,
                                   which decodes exactly as the single-word cell would (MaskDecoder.rs:95-153)  */
    float parse_ms;             /* device time of the parse (CUDA events)                                       */
} v2p_vcf_masks;

/* rec_line[n_records] (host): row r of the matrix is data line rec_line[r] of the last load; any order, repeats allowed;
 * lines not named are never read past their 9th column.  flags: 0.  Errors: V2P_ERR_INVALID_ARG (an entry >= n_lines,
 * no text loaded), V2P_ERR_VCF_PARSE (see the dialect above), V2P_ERR_CUDA.  After any error the object stays usable. */
int v2p_vcf_parse_masks(v2p_vcf* v, uint64_t n_records, const uint64_t* rec_line, uint32_t flags, v2p_vcf_masks* out);

#ifdef __cplusplus
}
#endif
#endif /* V2P_VCF_H */
