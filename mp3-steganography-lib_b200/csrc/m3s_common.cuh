// m3s_common.cuh -- shared declarations of libmp3stego_b200 (host context, device record layouts).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "../../include/mp3stego_b200.h"

// ------------------------------------------------------------------------------------------------
// device-side record layouts (HBM-resident, SoA across frames; see DESIGN.md "Data layout")
// ------------------------------------------------------------------------------------------------

// One per input file, built on the host after the frame walk.
struct M3sFileRec {
    int64_t begin;        // first byte of the file in the batch buffer
    int64_t end;          // one past the last byte
    int64_t audio;        // first audio byte (after ID3v2)
    int64_t frame_base;   // global index of the file's first frame
    int64_t s_base;       // byte offset of the file's header-stripped main-data stream in S
    int64_t pcm_base;     // element offset of the file's PCM in the output buffer
    int32_t n_frames;
    int32_t flags;        // M3S_FILE_* bits
    int32_t channels;
    int32_t pad;
    int64_t tmp_base;     // first slot of the file in the walk's temporary frame-position array
};

// Written by the walk kernel, one per file.
struct M3sFileOut {
    int64_t payload_total;  // bytes of main data (sum of frame payloads)
    int32_t n_frames;
    int32_t status;         // M3S_FILE_* bits
    int32_t sample_rate;
    int32_t channels;
    int32_t bitrate;
    int32_t reveal_len;
};

// frame meta word (fr_meta)
#define M3S_META_PAYLOAD_MASK 0x7FFu      // [0:11)  payload bytes present in the file (frame_size - header - side info - crc, clipped)
#define M3S_META_CRC (1u << 11)           // CRC word present (protection bit 0)
#define M3S_META_MODE_SHIFT 12            // [12:14) channel mode
#define M3S_META_MS (1u << 14)            // joint stereo with mode_extension bit 0x20 (Frame.py:273)
#define M3S_META_SR_SHIFT 15              // [15:17) sampling_frequency index
#define M3S_META_MONO (1u << 17)
#define M3S_META_FIRST (1u << 18)         // first frame of its file
#define M3S_META_DUP (1u << 19)           // last frame of a file that ends in junk: its PCM is emitted twice
#define M3S_META_HDR_SHIFT 20             // [20:26) header + crc + side-info bytes (36/38/21/23)

// One per granule-channel ("unit"), 4 slots per frame: slot = 2*gr + ch.
struct __align__(16) M3sUnitRec {
    uint64_t bit_start;   // absolute bit position in S where part2 (scalefactors) starts
    int32_t limit_bits;   // bits readable from bit_start before the frame's assembled main data ends (may be <= 0)
    uint32_t a;           // part2_3_length[0:12) big_values[12:21) global_gain[21:29) window_switching[29] block_type[30:32)
    uint32_t b;           // scalefac_compress[0:4) mixed[4] table_select0[5:10) 1[10:15) 2[15:20) region0[20:24) region1[24:27)
                          // preflag[27] scalefac_scale[28] count1table[29] ms[30] mono[31]
    uint32_t c;           // subblock_gain0[0:3) 1[3:6) 2[6:9) scfsi[9:13) sr_idx[13:15) gr[15] ch[16] valid[17] first_frame[18]
    uint32_t frame;       // global frame index
    uint32_t pad;
};

#define M3S_UA_P23(a) ((a) & 0xFFFu)
#define M3S_UA_BV(a) (((a) >> 12) & 0x1FFu)
#define M3S_UA_GG(a) (((a) >> 21) & 0xFFu)
#define M3S_UA_WS(a) (((a) >> 29) & 1u)
#define M3S_UA_BT(a) (((a) >> 30) & 3u)
#define M3S_UB_SFC(b) ((b) & 0xFu)
#define M3S_UB_MIXED(b) (((b) >> 4) & 1u)
#define M3S_UB_TS(b, r) (((b) >> (5 + 5 * (r))) & 0x1Fu)
#define M3S_UB_R0(b) (((b) >> 20) & 0xFu)
#define M3S_UB_R1(b) (((b) >> 24) & 0x7u)
#define M3S_UB_PREFLAG(b) (((b) >> 27) & 1u)
#define M3S_UB_SFSCALE(b) (((b) >> 28) & 1u)
#define M3S_UB_C1SEL(b) (((b) >> 29) & 1u)
#define M3S_UB_MS(b) (((b) >> 30) & 1u)
#define M3S_UB_MONO(b) (((b) >> 31) & 1u)
#define M3S_UC_SBG(c, w) (((c) >> (3 * (w))) & 7u)
#define M3S_UC_SCFSI(c) (((c) >> 9) & 0xFu)
#define M3S_UC_SR(c) (((c) >> 13) & 3u)
#define M3S_UC_GR(c) (((c) >> 15) & 1u)
#define M3S_UC_CH(c) (((c) >> 16) & 1u)
#define M3S_UC_VALID(c) (((c) >> 17) & 1u)
#define M3S_UC_FIRST(c) (((c) >> 18) & 1u)

// scalefactor bytes per unit: long [0..21], short [22 + 13*win + sfb]
#define M3S_SF_STRIDE 64
#define M3S_SF_SHORT 22

// Huffman decode LUT (built on the host at m3s_create, see m3s_context.cu):
//   entry uint16: leaf      0 | len[8:13) | x[4:8) | y[0:4)
//                 internal  0x8000 | nbits[11:15) | (sub offset >> 1)[0:11)
//   per table id: desc = l1_base[0:13) | l1_bits[13:17) | linbits[17:21);  sub = absolute index of the book's sub-table area
#define M3S_HUFF_L1_BITS 8
struct M3sDevTables {
    uint16_t huff_lut[8192];
    uint32_t huff_desc[32];
    uint32_t huff_sub[32];
    uint8_t count1_lut[64];      // table A: len[4:8) | v w x y [0:4)
    uint16_t sfb_long[3][23];
    uint16_t sfb_short[3][14];
    uint8_t sfw_short[3][12];
    uint8_t slen[16][2];
    uint8_t pretab[22];
    uint8_t long_sfb_of[3][576];   // sample index -> long sfb
    uint8_t short_sfw_of[3][576];  // sample index (pre-reorder) -> sfb*3 + window
    uint16_t reorder_dst[3][576];  // short-block reorder: source index -> destination index (Frame.py:574-602)
    float pow43[256];              // |x|^(4/3) for small |x| (double-rounded)
    float quarter[4];              // 2^(0/4) .. 2^(3/4)
    float imdct_cos36[36][18];
    float imdct_cos12[12][8];      // padded rows
    float sine_block[4][36];
    float synth_n[64][32];
    float synth_d[512];
    float alias_cs[8], alias_ca[8];
    // encoder
    int32_t enwindow[512];
    int32_t enc_fl[32][64];
    int32_t enc_cosl[18][36];
    int32_t enc_ca[8], enc_cs[8];
    int32_t steptabi[128];
    double steptab[128];
    int32_t int2idx[10000];
    uint8_t subdv[23][2];
    uint8_t pair[32][2];
    uint32_t enc_hpacked[1410];    // (code << 8) | len
    uint16_t enc_hoff[34];
    uint8_t enc_hdim[34];
    uint8_t enc_linbits[34];
    uint16_t enc_linmax[34];
};

// float64 copies of the hybrid-synthesis tables for the `exact` decode instantiation (M3S_DEC_EXACT)
struct M3sDevTablesD {
    double pow43[256];
    double quarter[4];
    double imdct_cos36[36][18];
    double imdct_cos12[12][8];
    double sine_block[4][36];
    double synth_n[64][32];
    double synth_d[512];
    double alias_cs[8], alias_ca[8];
};

// ------------------------------------------------------------------------------------------------
// host context
// ------------------------------------------------------------------------------------------------
struct M3sBuf {
    void *p = nullptr;
    size_t cap = 0;
};

// One CTA's run of frames in k_hybrid_fast.
struct M3sWork {
    int64_t g_first;   // first frame whose PCM this CTA emits
    int32_t count;     // frames to emit
    int32_t warm;      // 1: decode frame g_first-1 first without emitting
    int64_t pcm_elem;  // element offset of frame g_first's first sample in the PCM buffer
    int32_t channels;
    int32_t pad;
};

// Written by k_layout, one per scan: the wave's totals.
struct M3sLayout {
    int64_t total_frames;
    int64_t s_bytes;        // bytes of the header-stripped stream S the wave needs
    int64_t irregular;      // frames past the ninth of a file whose bit reservoir is assembled explicitly (see k_sideinfo)
    int32_t overflow;       // total_frames exceeded the set's capacity: the scan stopped after the walk
    int32_t pad;
};

// One wave's scan state: D0 (frame walk, per-frame records, unit records) and D4 (table ids, reveal chars).
struct M3sScanSet {
    M3sBuf files, fouts, tmp_pos, fr_pos, fr_P, fr_meta, fr_carry, fr_reveal, fr_file, units, tabids, reveal, layout, irr;
    // per-file results and the totals reach the host through MAPPED pinned memory (kernel stores), not copy-engine commands: a scan
    // is then never queued behind a bulk PCM transfer
    M3sFileOut *fouts_mapped = nullptr, *fouts_mdev = nullptr;
    M3sLayout *lay_mapped = nullptr, *lay_mdev = nullptr;
    size_t fouts_cap = 0;
    int64_t frames_cap = 0;            // frames the per-frame buffers hold
    int32_t n_files = 0;
    int64_t total_frames = 0, s_bytes = 0, total_bytes = 0, irregular = 0;
    const uint8_t *d_bytes = nullptr;  // device pointer to the wave's bytes (caller's or staged)
    std::vector<M3sFileRec> files_h;
    std::vector<M3sFileOut> fouts_h;
    void *pin = nullptr;               // pinned staging of the file records
    size_t pin_cap = 0;
};

// One encode chunk's intermediates: MDCT spectra, granule statistics, quantised values, side info, scfsi, and the per-granule
// variant records / summaries of the parallel rate loop (k_enc_probe -> k_enc_resolve).
struct M3sEncSet {
    M3sBuf mdct, gran, ix, info, scfsi, var, sum;
};

struct m3s_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t own_stream = nullptr;
    // copy streams + events of the host-buffer pipelines (created on first use): PCIe transfers of chunk k+1 / k-1 overlap the kernels of chunk k
    cudaStream_t copy_in = nullptr, copy_out = nullptr;
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr};
    cudaEvent_t ev_pace[3] = {nullptr, nullptr, nullptr};   // m3s_copy_paced
    // encoder: the analysis of chunk k+1 runs on `aux` next to the rate loop of chunk k (ev_ana[buf] = its spectra are ready)
    cudaStream_t aux = nullptr, launch_stream = nullptr;   // launch_stream: where the kernel being timed is launched (NULL = stream)
    cudaEvent_t ev_ana[2] = {nullptr, nullptr}, ev_pack[2] = {nullptr, nullptr};
    std::string err;
    int64_t launches = 0;
    // ---- optional per-kernel device timing (m3s_timing_enable): cudaEvent pairs on the launching stream
    bool timing = false;
    struct Timed { int id; cudaEvent_t e0, e1; };
    std::vector<Timed> timed;
    std::vector<cudaEvent_t> ev_pool;
    double k_ms[M3S_K_COUNT] = {0};
    int64_t k_launches[M3S_K_COUNT] = {0};
    M3sDevTables *d_tab = nullptr;
    M3sDevTablesD *d_tab_f64 = nullptr;
    int sm_count = 148;

    // ---- decode state.  A scan set holds one wave's D0 + D4 results (valid between a scan and the next scan on that set); the pipelined
    //      batch call m3s_decode alternates between the two sets so that wave k+1 is scanned while wave k is in the big kernels.
    M3sScanSet ss[2];
    M3sScanSet *cur = &ss[0];          // the set m3s_decode_reveal / m3s_decode_frame_pos / m3s_decode_run work on
    bool scanned = false;
    double dec_bpf_guess = 0.0;        // bytes per frame seen by earlier scans of device-resident input (sizes the next scan's workspaces)
    int64_t dec_wave_bytes = 0;        // M3S_DEC_WAVE_BYTES override of the pipelined call's wave size (0 = default)
    M3sBuf b_stage_in[2], b_pcm_stage[2];
    M3sBuf b_sf, b_S, b_spec, b_work, b_spec_export;
    void *work_pin[2] = {nullptr, nullptr};   // pinned staging of the hybrid kernel's work lists
    size_t work_pin_cap[2] = {0, 0};
    std::vector<M3sWork> work_h[2];
    cudaEvent_t ev_d_h2d[2] = {nullptr, nullptr}, ev_d_scan[2] = {nullptr, nullptr}, ev_d_comp[2] = {nullptr, nullptr},
                ev_d_out[2] = {nullptr, nullptr};
    uint8_t *rev_mapped = nullptr, *rev_dev = nullptr;   // m3s_decode_reveal to host memory: mapped pinned staging filled by a copy KERNEL
    size_t rev_cap = 0;
    // ---- encode state.  The per-chunk intermediates exist twice: chunk k uses set k & 1, so that the analysis writes ahead.
    M3sEncSet es[2];
    M3sBuf e_cand;   // m3s_encode_offsets: candidate records, work items, heads and bodies
    M3sBuf e_pcm, e_clips, e_out, e_payload, e_misc, e_pad, e_tabs, e_state, e_lastix, e_work;
    bool enc_taps_ok = false;
    int64_t enc_chunk_budget = 0;   // frames of intermediates kept per chunk (0 = default; M3S_ENC_CHUNK_FRAMES overrides)
    int64_t enc_total_frames = 0;
    std::vector<int64_t> enc_tap_runs;   // last encode: (device frame, caller frame, frames) triples, the taps' way back to the caller's clip order
};

int m3s_fail(m3s_ctx *h, int code, const char *fmt, ...);
void m3s_time_begin(m3s_ctx *h, int id);
void m3s_time_end(m3s_ctx *h);
int m3s_buf_reserve(m3s_ctx *h, M3sBuf &b, size_t bytes);
int m3s_pipeline_init(m3s_ctx *h);   // creates copy_in / copy_out and their events
int m3s_sync_streams(m3s_ctx *h);    // waits for the main stream and, once created, copy_in / copy_out / aux
// M3S_TRACE set: host-clock stage marks and per-chunk / per-wave device timelines of the pipelined calls on stderr (diagnostic)
extern const bool m3s_trace;
double m3s_now_ms();
// a batch of (dst, src, bytes) row copies on one stream: one cudaMemcpy2DAsync when the rows are equally long and equally spaced
struct M3sRow { char *dst; const char *src; size_t bytes; };
// blocking-call flavour: at most two pieces are queued at a time, so copies of OTHER handles (whose host threads wait on them)
// interleave within a millisecond instead of queueing behind the whole transfer -- copy engines serve commands in submission order
int m3s_copy_paced(m3s_ctx *h, void *dst, const void *src, size_t bytes, cudaMemcpyKind kind);
cudaError_t m3s_copy_bulk(void *dst, const void *src, size_t bytes, cudaMemcpyKind kind, cudaStream_t s);   // in bounded pieces
cudaError_t m3s_copy_rows(const std::vector<M3sRow> &rows, cudaMemcpyKind kind, cudaStream_t s);
int m3s_upload_fast_const();  // m3s_decode.cu: the fast transforms' twiddles in constant memory of the current device

// launches on `s` are timed on `s` (m3s_time_begin records on launch_stream); restored when the scope ends, error returns included
struct M3sLaunchOn {
    m3s_ctx *h;
    cudaStream_t saved;
    M3sLaunchOn(m3s_ctx *h_, cudaStream_t s) : h(h_), saved(h_->launch_stream) { h->launch_stream = s; }
    ~M3sLaunchOn() { h->launch_stream = saved; }
};

#define M3S_CUDA(h, call)                                                                             \
    do {                                                                                              \
        cudaError_t e__ = (call);                                                                     \
        if (e__ != cudaSuccess)                                                                       \
            return m3s_fail((h), M3S_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), \
                            __FILE__, __LINE__);                                                      \
    } while (0)

// M3S_KBEGIN(h, id); kernel<<<...>>>(...); M3S_LAUNCH_CHECK(h);
#define M3S_KBEGIN(h, id)                  \
    do {                                   \
        (h)->k_launches[id]++;             \
        if ((h)->timing) m3s_time_begin((h), (id)); \
    } while (0)

#define M3S_LAUNCH_CHECK(h)                                                                           \
    do {                                                                                              \
        (h)->launches++;                                                                              \
        if ((h)->timing) m3s_time_end(h);                                                                              \
        cudaError_t e__ = cudaGetLastError();                                                         \
        if (e__ != cudaSuccess)                                                                       \
            return m3s_fail((h), M3S_ERR_CUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(e__), \
                            __FILE__, __LINE__);                                                      \
    } while (0)
