/*
 * v2p_vcf_bgzf.h -- bgzip'd VCF (.vcf.gz) into the device VCF reader of include/v2p_vcf.h: the BGZF blocks are inflated
 * on the device and indexed as v2p_vcf_load indexes plain text; v2p_vcf_parse_masks then works unchanged.
 *
 * With plain text the host reads columns 1-9 from its own copy.  With a compressed file it has none, so the load also
 * hands back the header lines (`head`) and columns 1-9 of every data line (`fixed`); the sample columns, the bulk of
 * the file, stay on the device.
 *
 * BGZF (SAM spec section 4.1), what v2p_vcf_load_bgzf accepts:
 *   - A sequence of gzip members (blocks), each with ID1 31, ID2 139, CM 8, FLG 4 (FEXTRA alone), XLEN >= 6 holding a
 *     "BC" subfield with SLEN 2 among any others, BSIZE + 1 <= the bytes left, and a trailer of CRC32 and ISIZE with
 *     ISIZE <= 65536.  Blocks with ISIZE 0 may appear anywhere; the 28-byte EOF block is optional (htslib only warns).
 *   - The data of a block is raw DEFLATE (RFC 1951) that reaches the end of its final block inside the data; bytes
 *     after that and before the trailer are ignored (htslib's bgzf_uncompress; zlib.decompressobj(-15) with eof set).
 *   - Huffman codes as zlib's inftrees.c takes them: an over-subscribed set is invalid; an incomplete set is invalid
 *     except a lit/len or distance set whose only code has length 1; the lit/len code must code symbol 256.
 *     Lit/len symbols 286-287 and distance symbols 30-31 are invalid, and so is a code-length repeat with no previous
 *     length or running past HLIT + HDIST, a stored block with LEN != ~NLEN, BTYPE 3, and a distance reaching before
 *     the start of the block (blocks are independent).
 *   - The inflated text must have ISIZE bytes and the trailer's CRC-32.
 * An error is V2P_ERR_BGZF with the message "BGZF block <k> at byte <offset>: <class>" for the first bad block in file
 * order (k from 0, offset = the block's first byte), whatever the thread timing.  Within one block the classes rank
 *   1 "bad BGZF block header (<why>)"   2 "invalid DEFLATE data"   3 "inflated size differs from the trailer's ISIZE"
 *   4 "CRC-32 differs from the trailer's"
 * A bad header ends the walk, but the blocks before it are still inflated and checked, and an error there comes first.
 * A plain gzip file (no BC subfield) or plain text is refused as a bad header "(not BGZF: recompress with bgzip)": the
 * input is never sniffed, and v2p_vcf_load never inflates.
 *
 * Threading: as include/v2p_vcf.h (one call at a time per object).
 */
#ifndef V2P_VCF_BGZF_H
#define V2P_VCF_BGZF_H

#include "v2p_vcf.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct {
    uint64_t n_blocks;            /* BGZF blocks walked, the empty EOF block included                                  */
    uint64_t text_bytes;          /* inflated size = sum of the blocks' ISIZE                                           */
    const uint8_t* text;          /* device, the inflated text, owned by v until the next load / destroy                */
    const uint8_t* head;          /* host, owned by v: text[0, header_end) -- every line up to and including #CHROM     */
    const uint8_t* fixed;         /* host, owned by v: columns 1-9 of every data line, file order, concatenated          */
    const uint64_t* fixed_begin;  /* host, n_lines + 1: fixed[fixed_begin[l], fixed_begin[l+1]) == text[line_begin[l], cells_begin[l]) */
    float inflate_ms, fixed_ms;   /* device time of the inflate and of the columns 1-9 gather + copy-back (CUDA events) */
} v2p_vcf_bgzf;

/* BGZF (host memory; pinned for the full PCIe rate) -> inflated text on the device -> the same index v2p_vcf_load builds.
 * `out` is filled exactly as v2p_vcf_load fills it for the inflated text (offsets are into the inflated text;
 * h2d_bytes = compressed bytes).  flags: 0 (V2P_FLAG_DEVICE_PTRS is INVALID_ARG).  Afterwards v2p_vcf_parse_masks
 * works unchanged.  Errors: V2P_ERR_BGZF, V2P_ERR_VCF_PARSE, V2P_ERR_INVALID_ARG, V2P_ERR_CUDA.  After any error the
 * object stays usable. */
int v2p_vcf_load_bgzf(v2p_vcf* v, const uint8_t* data, uint64_t n_bytes, uint32_t flags, v2p_vcf_lines* out,
                      v2p_vcf_bgzf* bz);

#ifdef __cplusplus
}
#endif
#endif /* V2P_VCF_BGZF_H */
