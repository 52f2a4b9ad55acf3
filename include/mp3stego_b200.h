/*
 * mp3stego_b200.h -- C ABI of libmp3stego_b200.so, the B200 (sm_100a) implementation of the
 * per-granule codec hot path of mp3stego (tomershay100/mp3-steganography-lib 1.1.8).
 *
 * The reference has no FFI of its own: the hot path sits behind two Python methods,
 *   MP3Parser.parse_file()   mp3stego/decoder/MP3_Parser.py:57-85   (MP3 -> PCM + reveal bits)
 *   MP3Encoder.encode()      mp3stego/encoder/MP3_Encoder.py:596-621 (PCM -> MP3, optional hide)
 * and this header declares exactly what those two methods would bind (ctypes; see INTEGRATION.md).
 * Everything is plain C: pointers + sizes, int status returns, no exceptions, no torch types.
 *
 * Conventions
 *   - Every call returns M3S_OK (0) or a negative M3S_ERR_*; m3s_last_error() gives the text.
 *   - `mem` arguments say where the caller's bulk buffers live: M3S_MEM_HOST (pageable or pinned host
 *     memory; the library stages through the device inside the call) or M3S_MEM_DEVICE (device
 *     pointers, e.g. torch tensors' data_ptr(); nothing crosses PCIe).
 *     Small per-file descriptor arrays (offsets, counts, status) are ALWAYS host memory.
 *     Device buffers must be READY when a call starts -- the library works on its own streams (or the one given to
 *     m3s_set_stream) and is not ordered with whatever else the caller has queued, e.g. the kernel that produced an
 *     input or the fill of a freshly allocated output; results are complete when the call returns.
 *   - A handle owns one CUDA stream (or borrows one via m3s_set_stream) and grow-only device
 *     workspaces; calls on one handle are serialised and block until their results are readable,
 *     except where a function says it is asynchronous.  Handles are not thread-safe.
 *   - Supported streams: MPEG-1 Layer III, 32/44.1/48 kHz, mono or stereo, CBR or VBR, with or
 *     without CRC -- the domain in which the reference itself works (FrameHeader.py:125-143).
 */
#ifndef MP3STEGO_B200_H
#define MP3STEGO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define M3S_API __attribute__((visibility("default")))
#else
#define M3S_API
#endif

typedef struct m3s_ctx *m3s_handle_t;

enum {
    M3S_OK = 0,
    M3S_ERR_CUDA = -1,        /* a CUDA runtime call or kernel failed */
    M3S_ERR_ARG = -2,         /* bad argument */
    M3S_ERR_STATE = -3,       /* call order violated (e.g. decode_run without decode_scan) */
    M3S_ERR_NO_DEVICE = -4,   /* no CUDA device / not an sm_100 part */
    M3S_ERR_CAPACITY = -5     /* output buffer too small */
};

enum { M3S_MEM_HOST = 0, M3S_MEM_DEVICE = 1 };

/* per-file status written by m3s_decode_scan (mirrors where MP3Parser stops or raises) */
enum {
    M3S_FILE_OK = 0,
    M3S_FILE_NO_SYNC = 1,        /* first audio bytes are not 0xFF 0xEx: MP3Parser.__valid False (MP3_Parser.py:36-44) */
    M3S_FILE_UNSUPPORTED = 2,    /* a frame header outside MPEG-1 Layer III / reserved sample rate or bitrate index 15 */
    M3S_FILE_TRAILING_JUNK = 4,  /* parsing stopped at a bad sync word; the last frame's PCM is repeated once (MP3_Parser.py:68-79) */
    M3S_FILE_CHANNEL_SWITCH = 16,/* mono and stereo frames in one file: MP3Parser.parse_file raises ValueError when it stacks PCM rows of
                                    different widths (MP3_Parser.py:83); the PCM this library writes for such a file is unspecified */
    M3S_FILE_BAD_SIDEINFO = 32,  /* a granule with big_values > 288 or region0_count + region1_count + 2 > 22: the reference raises
                                    IndexError (Frame.py:461-478); this library clamps and flags the file */
    M3S_FILE_STATE_CARRY = 8     /* some granule takes scalefactors from EARLIER frames through the reference's persistent arrays: a mixed
                                    block (scale_fac_s[..][0..2], Frame.py:387-403 vs :198) or scfsi over a short-block granule 0
                                    (Frame.py:419-437).  A frame-range shard of such a file needs the whole prefix as its halo. */
};

/* flags for m3s_decode_run */
enum {
    M3S_DEC_PCM_FLOAT = 1,       /* pcm buffer is float32 (pre-int16 samples) instead of int16 */
    M3S_DEC_EXACT = 2            /* run requantize..synthesis in float64 like the reference (Frame.py is float64 end to end):
                                    int16 PCM then equals the reference's sample for sample in practice, which the hide / clear
                                    composites need to reproduce the reference's MP3 bytes; the default FP32 path is within 1 LSB */
};

/* ---------------------------------------------------------------- lifetime */
M3S_API int m3s_create(int device, m3s_handle_t *out);
M3S_API int m3s_destroy(m3s_handle_t h);
M3S_API const char *m3s_last_error(m3s_handle_t h);
/* Borrow a caller-owned cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream); NULL restores the handle's own. */
M3S_API int m3s_set_stream(m3s_handle_t h, void *cuda_stream);
/* Block until everything queued on the handle's stream has finished. */
M3S_API int m3s_synchronize(m3s_handle_t h);
/* Number of kernel launches issued by this handle since creation (bench.py's gpu_launches). */
M3S_API int64_t m3s_launch_count(m3s_handle_t h);
/* Library/ABI version: major*10000 + minor*100 + patch. */
M3S_API int m3s_version(void);

/* ------------------------------------------------------------------ decode
 * Replaces MP3Parser.__init__ + the frame walk of MP3Parser.parse_file (MP3_Parser.py:21-85),
 * FrameHeader.init_header_params (FrameHeader.py:51-192), Frame.set_frame_size (Frame.py:288-316),
 * FrameSideInformation.set_side_info (FrameSideInformation.py:39-137) and the reveal-bit rule
 * Frame.__get_frame_huffman_tables + util.bit_from_huffman_tables (Frame.py:676-685, util.py:67-81)
 * for a BATCH of files laid end to end in `bytes`.
 *
 *   bytes        all files concatenated (host or device per `mem`)
 *   file_off     [n_files+1] host: byte offset of each file in `bytes`; file i = [file_off[i], file_off[i+1])
 *   audio_start  [n_files] host or NULL: offset of the first audio byte inside each file (ID3v2 skip,
 *                decoder.py:29-33); NULL = 0 for every file
 * outputs (host arrays of n_files entries, any may be NULL):
 *   n_frames     frames parsed                      (parse_file's return value)
 *   pcm_rows     PCM rows the file decodes to = 1152 * (n_frames + 1 if trailing junk)
 *   sample_rate, channels, bitrate_bps   of the LAST frame, as MP3Parser.get_bitrate / Frame.sampling_rate report
 *   status       M3S_FILE_* bits
 * The scan result stays in the handle for m3s_decode_reveal / m3s_decode_run.
 */
M3S_API int m3s_decode_scan(m3s_handle_t h, const uint8_t *bytes, int mem, const int64_t *file_off,
                            const int64_t *audio_start, int32_t n_files, int64_t *n_frames, int64_t *pcm_rows,
                            int32_t *sample_rate, int32_t *channels, int32_t *bitrate_bps, int32_t *status);

/* Reveal outputs of the last scan (the `reveal` half of decode+reveal; needs no Huffman decode).
 *   table_ids    [total_frames*12] per frame the 12 table ids in (ch, gr, region) order incl. the stale
 *                region-2 id of window-switched granules (Frame.py:676-685); mono frames fill 6. May be NULL.
 *   reveal_bits  ['0'/'1' chars] file i's string starts at 12 * (sum of n_frames of files < i); May be NULL.
 *   reveal_len   [n_files] host: number of chars of each file's string (MP3Parser.output_bits). */
M3S_API int m3s_decode_reveal(m3s_handle_t h, uint8_t *table_ids, uint8_t *reveal_bits, int mem, int64_t *reveal_len);

/* Byte position of every frame of the last scan, relative to the start of its file: [total_frames] host array, file i's frames
 * at [sum of n_frames of files < i, ...).  What Frame.set_frame_size accumulates into MP3Parser's offset (MP3_Parser.py:75,
 * Frame.py:288-316); a host that splits one long file into frame ranges for several GPUs cuts the byte stream here. */
M3S_API int m3s_decode_frame_pos(m3s_handle_t h, int64_t *frame_pos);

/* Huffman decode -> requantize -> stereo -> reorder/alias -> IMDCT/overlap -> polyphase synthesis of the
 * last scanned batch: Frame.init_frame_params (Frame.py:244-286) for every frame, then
 * MP3Parser.write_to_wav's float->int16 conversion (MP3_Parser.py:87-91).
 *   pcm       interleaved samples, file i at element offset pcm_off[i]; rows*channels elements per file
 *   pcm_off   [n_files] host element offsets, or NULL for back-to-back
 *   spectra   optional parity tap (device or host per mem): int16 [total_frames][gr][ch][576] integer spectra
 *             as Frame.__unpack_samples leaves them (Frame.py:443-559); NULL to skip */
M3S_API int m3s_decode_run(m3s_handle_t h, void *pcm, int mem, const int64_t *pcm_off, int16_t *spectra,
                           uint32_t flags);

/* Frame-range decode of one file of the last scan (a long file split across several GPUs, SURVEY.md 8e): frames
 * [first_frame, first_frame + frame_count) of file `file_index` into `pcm` (host or device per mem), *rows_out = PCM rows written
 * (1152 per frame, + 1152 when the range holds the last frame of a file that ends in junk).  The library decodes one warm-up
 * frame in front of the range (overlap-add tail + synthesis fifo, Frame.py:81-92,150-153) and compacts the <= 9 frames of bit
 * reservoir it may reach into (Frame.py:306-309,337-356); the ranges of all ranks, concatenated, equal the whole-file decode. */
M3S_API int m3s_decode_run_range(m3s_handle_t h, int32_t file_index, int64_t first_frame, int64_t frame_count, void *pcm, int mem,
                                 int64_t *rows_out, uint32_t flags);

/* The batch call: everything above in ONE call that pipelines itself -- MP3Parser.parse_file + write_to_wav's conversion
 * (MP3_Parser.py:57-91) for n_files files.  The library cuts the batch into waves of whole files and overlaps, on its own
 * streams, the upload of wave k+1 (host buffers), the scan of wave k+1, the Huffman + synthesis kernels of wave k and the
 * download of wave k-1 (host buffers); the host thread waits once per wave and the call returns when every output is readable.
 *   bytes, mem, file_off, audio_start, n_files   as m3s_decode_scan
 *   pcm            interleaved samples of all files back to back (int16, or float32 with M3S_DEC_PCM_FLOAT); host or device per mem
 *   pcm_capacity   elements `pcm` can hold; M3S_ERR_CAPACITY if the batch decodes to more (m3s_decode_bound sizes it)
 *   pcm_off        [n_files+1] host, OUT (may be NULL): element offset of every file in pcm, and the total
 *   table_ids, reveal_bits   as m3s_decode_reveal (host or device per mem; either may be NULL); frames_capacity = frames they hold
 *   reveal_len, n_frames, sample_rate, channels, bitrate_bps, status   [n_files] host, OUT, any may be NULL
 *   flags          M3S_DEC_* */
M3S_API int m3s_decode(m3s_handle_t h, const uint8_t *bytes, int mem, const int64_t *file_off, const int64_t *audio_start,
                       int32_t n_files, void *pcm, int64_t pcm_capacity, int64_t *pcm_off, uint8_t *table_ids, uint8_t *reveal_bits,
                       int64_t frames_capacity, int64_t *reveal_len, int64_t *n_frames, int32_t *sample_rate, int32_t *channels,
                       int32_t *bitrate_bps, int32_t *status, uint32_t flags);
/* Host-only sizing aid for m3s_decode with HOST bytes: frames each file can hold according to its first frame header (exact
 * for constant-bitrate files, which is all the reference's own encoder writes; a VBR file may decode to more and then makes
 * m3s_decode return M3S_ERR_CAPACITY -- size from m3s_decode_scan's pcm_rows instead).  Returns the PCM elements to reserve
 * (stereo assumed) and the frame count through *frames_bound; < 0 on bad arguments. */
M3S_API int64_t m3s_decode_bound(const uint8_t *bytes_host, const int64_t *file_off, const int64_t *audio_start, int32_t n_files,
                                 int64_t *frames_bound);

/* ------------------------------------------------------------------ encode
 * Replaces MP3Encoder.__init__ + MP3Encoder.encode (MP3_Encoder.py:462-650): analysis filterbank + MDCT
 * (:652-758), rate loop with the stego table swap (:760-1264) and bitstream formatting (:1266-1552),
 * for a BATCH of 16-bit stereo clips.
 *   pcm           interleaved int16 stereo, clip i at element offset pcm_off[i], 2*n_samples[i] elements
 *   n_samples     [n_clips] host: samples per channel; must be a multiple of 1152 (the reference raises otherwise)
 *   payload_bits  '0'/'1' chars of all payloads concatenated (host), clip i = [payload_off[i], payload_off[i+1]);
 *                 NULL or empty range = plain encode (no swap)
 *   mp3_out       output bytes, clip i at mp3_off[i]; capacity mp3_cap[i] >= m3s_encode_bound()
 *   out_len       [n_clips] host: bytes written (a multiple of 4, MP3_Encoder.py:1370-1392,1549-1552)
 *   hide_str_offset_out  [n_clips] host: MP3Encoder.hide_str_offset after the last frame
 * A granule whose step search would quantise at a step above 0 (loud high-frequency input at low bitrates, e.g. a
 * full-scale Nyquist-rate square at 44.1 kHz / 32 kbps) would make the reference read its 128-entry step table past
 * the end (SURVEY A.E13); there is no defined output for it.  The kernels stop that search at step 0, and the call
 * returns M3S_ERR_ARG with an m3s_last_error text naming the first such clip and frame ("clip %d frame %d: ... runs
 * past the end of the step table").  The whole batch fails: no clip's output or hide_str_offset is valid, and the
 * handle stays usable for the next call.
 */
M3S_API int64_t m3s_encode_bound(int64_t n_samples, int32_t sample_rate, int32_t bitrate_kbps);
/* Exact number of bytes MP3Encoder emits for a clip of n_samples per channel: the sum of the padded frame sizes
 * (slot-lag recurrence, MP3_Encoder.py:504-513,630-632) rounded DOWN to whole 32-bit words (:1370-1392). <0 on bad arguments. */
M3S_API int64_t m3s_encode_size(int64_t n_samples, int32_t sample_rate, int32_t bitrate_kbps);
M3S_API int m3s_encode(m3s_handle_t h, const int16_t *pcm, int mem, const int64_t *pcm_off, const int64_t *n_samples,
                       int32_t n_clips, int32_t sample_rate, int32_t bitrate_kbps, const uint8_t *payload_bits,
                       const int64_t *payload_off, uint8_t *mp3_out, const int64_t *mp3_off, const int64_t *mp3_cap,
                       int64_t *out_len, int64_t *hide_str_offset_out);
/* m3s_encode with a rate pair per clip: clips of different sample rates and bitrates in ONE call (a mixed MP3 collection
 * re-encoded at each file's own rates needs no grouping by the caller).
 *   sample_rate   [n_clips] host: 32000, 44100 or 48000 per clip
 *   bitrate_kbps  [n_clips] host: one of the 14 MPEG-1 Layer III bitrates per clip
 * Everything else as m3s_encode, per clip: clip i's bytes, out_len and hide_str_offset are what m3s_encode gives for it at its own
 * pair.  A clip with an unsupported rate fails the call with M3S_ERR_ARG before anything is queued, the text naming the clip
 * ("clip %d: sample rate ..." / "clip %d: bitrate ...").  The step-table failure above names the caller's clip index and frame.
 * m3s_encode_taps works after a single-chunk call, frames in the caller's clip order.  m3s_encode is this function with its two
 * rates broadcast to every clip. */
M3S_API int m3s_encode_mixed(m3s_handle_t h, const int16_t *pcm, int mem, const int64_t *pcm_off, const int64_t *n_samples,
                             int32_t n_clips, const int32_t *sample_rate, const int32_t *bitrate_kbps, const uint8_t *payload_bits,
                             const int64_t *payload_off, uint8_t *mp3_out, const int64_t *mp3_off, const int64_t *mp3_cap,
                             int64_t *out_len, int64_t *hide_str_offset_out);
/* hide_str_offset of many candidate payloads per clip, without writing MP3 bytes: how much of a message fits in a clip, answered
 * for every prefix at once.  The analysis and the rate loop's probe of every payload variant run once per clip; only the offset
 * chain runs per candidate, so the call costs about one encode without the quantisation and the bit packing.
 *   pcm, mem, pcm_off, n_samples, n_clips, sample_rate, bitrate_kbps   as m3s_encode_mixed (pcm host or device per mem)
 *   body          host bytes; clip i's body is body[body_off[i] .. body_off[i+1])
 *   body_off      [n_clips+1] host
 *   cand_off      [n_clips+1] host, cand_off[0] = 0: the candidates of clip i are c in [cand_off[i], cand_off[i+1]); a clip may have none
 *   head          host bytes; candidate c's head is head[head_off[c] .. head_off[c+1]), at most 32 bytes
 *   head_off      [n_cand+1] host, n_cand = cand_off[n_clips]
 *   body_len      [n_cand] host: candidate c hides the MSB-first bits of its head followed by the first body_len[c] bytes of its
 *                 clip's body.  (The facade frames message[:n] as head "<n>#" and body = the message's utf-8 bytes.)
 *   hide_str_offset_out  [n_cand] host: what m3s_encode_mixed returns as clip i's hide_str_offset with that payload as '0'/'1'
 *                 chars; an empty payload gets the plain encode's offset.
 * The clip checks of m3s_encode_mixed apply; a head over 32 bytes, a body_len past the clip's body or bad offsets fail with
 * M3S_ERR_ARG before anything is queued, the text naming the clip and the candidate.  A step-table overrun (see m3s_encode) under
 * any candidate fails the whole call, the text naming the caller's clip, the candidate and the frame ("clip %d candidate %lld
 * frame %d: ... runs past the end of the step table"); the handle stays usable.  m3s_encode_taps fails after this call. */
M3S_API int m3s_encode_offsets(m3s_handle_t h, const int16_t *pcm, int mem, const int64_t *pcm_off, const int64_t *n_samples,
                               int32_t n_clips, const int32_t *sample_rate, const int32_t *bitrate_kbps,
                               const uint8_t *body, const int64_t *body_off, const int64_t *cand_off,
                               const uint8_t *head, const int64_t *head_off, const int64_t *body_len,
                               int64_t *hide_str_offset_out);
/* Parity taps of the last m3s_encode / m3s_encode_mixed call (host buffers): mdct int32 [frames][ch][gr][576] (MP3_Encoder.py:652),
 * ix int32 [frames][ch][gr][576] signed as written (:1272-1276), info int32 [frames][gr][ch][16]:
 * part2_3_length, big_values, count1, global_gain, table_select[3], region0_count, region1_count,
 * count1table_select, address1..3, quantizerStepSize, padding, hide_str_offset-after-frame. */
M3S_API int m3s_encode_taps(m3s_handle_t h, int32_t *mdct, int32_t *ix, int32_t *info, int32_t *scfsi);

/* ---------------------------------------------------------------- timing
 * Optional per-kernel device timing used by bench.py's roofline line: when enabled every kernel launch of
 * the handle is bracketed by a cudaEvent pair on the launching stream.  m3s_timing_get synchronises the
 * stream and returns the accumulated device milliseconds and launch count of kernel `kernel_id`
 * (launch counts are kept even while timing is disabled). m3s_timing_enable(…, on) also resets both. */
enum {
    M3S_K_WALK = 0,      /* D0a frame walk (one warp per file, speculative 32-frame windows) */
    M3S_K_FSCAN,         /* D0a' per-file scans: payload prefix, carried table_select[2], reveal offsets */
    M3S_K_SIDEINFO,      /* D0b side-info parse + D4 reveal bits (one thread per frame) */
    M3S_K_STRIP,         /* main-data compaction through the bit reservoir */
    M3S_K_HUFF,          /* D1 scalefactor + Huffman decode */
    M3S_K_SPEC_EXPORT,   /* parity tap */
    M3S_K_HYBRID,        /* D2+D3 requantize .. polyphase synthesis .. int16 */
    M3S_K_ENC_ANALYSIS,  /* E1 polyphase analysis + MDCT + alias (fixed point) */
    M3S_K_ENC_RATE,      /* E2 per-granule rate loop incl. table selection + stego swap, every payload variant of a granule (k_enc_probe) */
    M3S_K_ENC_RESOLVE,   /* E2b per-clip sequential offset scan over granule variants */
    M3S_K_ENC_PACK,      /* E3 side-info + main-data bit packing */
    M3S_K_ENC_AUX,       /* E2c quantisation at the chosen step (k_enc_emit) */
    M3S_K_ENC_OFFSETS,   /* E2d m3s_encode_offsets: the offset chains of many candidate payloads per clip (k_enc_offsets) */
    M3S_K_COUNT
};
M3S_API int m3s_timing_enable(m3s_handle_t h, int on);
M3S_API int m3s_timing_get(m3s_handle_t h, int kernel_id, double *total_ms, int64_t *launches);
M3S_API const char *m3s_kernel_name(int kernel_id);

/* ------------------------------------------------------------- diagnostics */
/* sha-free table export used by tests/test_tables.py: copies table `which` (see m3s_table_id) into out. */
enum {
    M3S_TAB_HUFF_PACKED = 0, M3S_TAB_HUFF_BOOK_OFF, M3S_TAB_HUFF_DIM, M3S_TAB_HUFF_LINBITS, M3S_TAB_SFB_LONG,
    M3S_TAB_SFB_SHORT, M3S_TAB_SFW_SHORT, M3S_TAB_SLEN, M3S_TAB_PRETAB, M3S_TAB_SYNTH_WINDOW, M3S_TAB_ENWINDOW,
    M3S_TAB_ENC_FL, M3S_TAB_ENC_COSL, M3S_TAB_ENC_STEPTABI, M3S_TAB_ENC_STEPTAB, M3S_TAB_ENC_INT2IDX,
    M3S_TAB_ENC_CA, M3S_TAB_ENC_CS, M3S_TAB_SUBDV, M3S_TAB_STEGO_PAIR, M3S_TAB_ALIAS_CS, M3S_TAB_ALIAS_CA,
    M3S_TAB_H0_MASK, M3S_TAB_COUNT
};
/* Returns the element count (or <0); if out != NULL copies min(count, cap) elements widened to double. */
M3S_API int64_t m3s_table_export(int which, double *out, int64_t cap);

#ifdef __cplusplus
}
#endif
#endif /* MP3STEGO_B200_H */
