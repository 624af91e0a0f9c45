/* jxlfront.h -- C ABI of libjxlfront.so, the host front end of the decoder (SURVEY.md 8f-1).
 *
 * The reference decodes everything on the caller's thread in Java.  The north star keeps the sequential half there
 * (container demux, headers, ANS / prefix / LZ77 entropy decoding, MA-tree traversal); this image has no JVM, so that
 * half is restated in C++ (jxlatte_b200/frontend/) behind this ABI.  It replaces, for the purpose of feeding real .jxl
 * files to libjxlb200.so:
 *   J/io/Demuxer.java, J/io/Bitreader.java, J/entropy/*.java, J/bundle/ImageHeader.java (+ the bundle/ and color/ header
 *   classes), J/frame/FrameHeader.java, J/frame/Frame.java:129-200 (TOC) and :271-462 (decode flow), J/frame/LFGlobal.java,
 *   J/frame/group/{LFGroup,Pass,PassGroup}.java (constructors), J/frame/modular/{MATree,ModularChannel.decode,ModularStream
 *   ctor}.java, J/frame/vardct/{LFCoefficients,HFMetadata,HFBlockContext,HFPass,HFGlobal ctor,HFCoefficients ctor}.java
 * It runs no reconstruction: its output is exactly the argument list of jxlb200_vardct_reconstruct() / jxlb200_modular_*()
 * (include/jxlb200.h).  Pure host code, no CUDA.
 *
 * Status codes: 0 OK, -1 internal / invalid argument, -2 invalid bitstream (InvalidBitstreamException),
 * -3 valid but unsupported by this build (UnsupportedOperationException).  On a non-zero status the image handle is
 * still returned so jxlf_error() and whatever was parsed so far can be read; free it with jxlf_free().
 */
#ifndef JXLFRONT_H
#define JXLFRONT_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct jxlf_image jxlf_image;

#define JXLF_HOST_TRANSFORMS 1 /* also undo the frame-level Modular transforms on the host (tests / cross-checks only) */
#define JXLF_HEADERS_ONLY 2    /* stop after the first frame header + TOC */
/* Parse every frame up to its LF image: LfGlobal and, in each LF group, the LF coefficients and the LF-group Modular channels.
 * HF metadata, HfGlobal and the pass groups are skipped unread.  "lf", "lf_quant" and "lf_extra_precision" are what the full
 * parse gives; the HF arrays ("qcoeff", "dct_select", "block_origin", "hf_mul", "sharpness", "x_from_y", "b_from_y") are
 * not found; jxlf_describe adds "lf_only": true and leaves out the HfGlobal fields "quant_all_default" / "quant_params".
 * Modular channels that pass groups fill stay empty, so JXLF_HOST_TRANSFORMS cannot be combined with it (status -1). */
#define JXLF_LF_ONLY 4

/* JXLDecoder(InputStream) + decode() up to the end of the codestream (J/JXLCodestreamDecoder.java:547-626): every frame is
 * entropy-decoded; nothing is rendered. */
int32_t jxlf_decode(const uint8_t *data, uint64_t size, int32_t flags, jxlf_image **out);
void jxlf_free(jxlf_image *image);
const char *jxlf_error(const jxlf_image *image);
/* All header fields (ImageHeader, per-frame FrameHeader / LFGlobal / HFGlobal parameters, the frame-level modular
 * stream's channel list and transform list) as one JSON document; owned by the image. */
const char *jxlf_describe(const jxlf_image *image);
/* Arrays by name; *ptr stays owned by the image.  dtype: 0 int32, 1 float32, 2 uint8.
 *   "qcoeff", "lf"            index = channel (X, Y, B); frame-level planes, passes summed
 *   "lf_quant"                index = channel (X, Y, B); the quantised LF before LFCoefficients' arithmetic, (hb >> sy) x (wb >> sx)
 *   "lf_extra_precision"      one byte per LF group
 *   "dct_select", "block_origin", "hf_mul", "sharpness", "x_from_y", "b_from_y"
 *   "modular"                 index = channel of the frame-level modular stream (before its transforms are undone)
 *   "qraw"                    index = 3 * parameter set + channel (MODE_RAW quant tables)
 *   "icc"                     the still-encoded ICC stream (frame ignored) */
int32_t jxlf_array(const jxlf_image *image, int32_t frame, const char *name, int32_t index, const void **ptr, int64_t *count, int32_t *dtype);
/* The number of OpenMP threads the calling thread's later jxlf_decode calls spread a frame's sections over (omp_set_num_threads:
 * the setting belongs to the calling thread, so threads that parse files side by side can each take a share of the cores).
 * n < 1 is ignored. */
void jxlf_set_threads(int32_t n);

#ifdef __cplusplus
}
#endif
#endif
