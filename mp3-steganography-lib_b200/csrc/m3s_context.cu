// m3s_context.cu -- handle lifetime, device table construction, error plumbing.
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <chrono>

#include "m3s_common.cuh"
#include "m3s_tables_data.h"

int m3s_fail(m3s_ctx *h, int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (h) h->err = buf;
    return code;
}

const bool m3s_trace = getenv("M3S_TRACE") != nullptr;

double m3s_now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

int m3s_sync_streams(m3s_ctx *h)
{
    M3S_CUDA(h, cudaStreamSynchronize(h->stream));
    if (h->copy_in) {
        M3S_CUDA(h, cudaStreamSynchronize(h->copy_in));
        M3S_CUDA(h, cudaStreamSynchronize(h->copy_out));
        M3S_CUDA(h, cudaStreamSynchronize(h->aux));
    }
    return M3S_OK;
}

int m3s_buf_reserve(m3s_ctx *h, M3sBuf &b, size_t bytes)
{
    if (bytes <= b.cap) return M3S_OK;
    if (b.p) {
        // the helper streams of the pipelines may still reference the buffer (e.g. after an early error return)
        const int rc = m3s_sync_streams(h);
        if (rc) return rc;
        M3S_CUDA(h, cudaFree(b.p));
        b.p = nullptr;
        b.cap = 0;
    }
    size_t cap = bytes + bytes / 8 + 256;
    cap = (cap + 255) & ~(size_t)255;
    M3S_CUDA(h, cudaMalloc(&b.p, cap));
    b.cap = cap;
    return M3S_OK;
}

// ------------------------------------------------------------------------------------------------
// Huffman decode LUT: two-level, 8-bit first level (ISO 11172-3 Table B.7 code books; every book is a
// complete prefix code, so a LUT walk is equivalent to the reference's first-prefix-match scan,
// Frame.py:491-517 -- tests/test_parity_decode.py checks that against the oracle's linear search).
// ------------------------------------------------------------------------------------------------
static int build_huff_lut(M3sDevTables *T)
{
    int next = 0;
    int base_of_book[34];
    int sub_of_book[34];
    int l1bits_of_book[34];
    for (int t = 0; t < 34; t++) base_of_book[t] = -1;
    memset(T->huff_lut, 0, sizeof T->huff_lut);
    for (int t = 1; t < 32; t++) {
        int dim = M3S_HUFF_DIM[t];
        T->huff_desc[t] = 0;
        T->huff_sub[t] = 0;
        if (dim == 0) continue;
        int off = M3S_HUFF_BOOK_OFF[t];
        int owner = -1;
        for (int u = 1; u < t; u++)
            if (M3S_HUFF_DIM[u] && M3S_HUFF_BOOK_OFF[u] == off) { owner = u; break; }
        if (owner < 0) {
            int n = dim * dim, maxlen = 0;
            for (int i = 0; i < n; i++) { int l = M3S_HUFF_PACKED[off + i] & 0xFF; if (l > maxlen) maxlen = l; }
            int l1 = maxlen < M3S_HUFF_L1_BITS ? maxlen : M3S_HUFF_L1_BITS;
            int l1base = next;
            next += 1 << l1;
            if (next & 1) next++;
            int subbase = next;
            // pass 1: short codes fill the first level; long codes record the deepest length per prefix
            int subbits[256];
            int suboff[256];
            for (int i = 0; i < 256; i++) { subbits[i] = 0; suboff[i] = -1; }
            for (int i = 0; i < n; i++) {
                uint32_t code = M3S_HUFF_PACKED[off + i] >> 8;
                int len = M3S_HUFF_PACKED[off + i] & 0xFF;
                int x = i / dim, y = i % dim;
                if (len <= l1) {
                    uint32_t lo = code << (l1 - len);
                    for (uint32_t k = 0; k < (1u << (l1 - len)); k++)
                        T->huff_lut[l1base + lo + k] = (uint16_t)((len << 8) | (x << 4) | y);
                } else {
                    uint32_t p = code >> (len - l1);
                    if (len - l1 > subbits[p]) subbits[p] = len - l1;
                }
            }
            int sub_next = 0;
            for (int p = 0; p < (1 << l1); p++)
                if (subbits[p]) {
                    suboff[p] = sub_next;
                    sub_next += 1 << subbits[p];
                    if (sub_next & 1) sub_next++;
                    if (suboff[p] >= 4096) return -1;
                    T->huff_lut[l1base + p] = (uint16_t)(0x8000 | (subbits[p] << 11) | (suboff[p] >> 1));
                }
            for (int i = 0; i < n; i++) {
                uint32_t code = M3S_HUFF_PACKED[off + i] >> 8;
                int len = M3S_HUFF_PACKED[off + i] & 0xFF;
                int x = i / dim, y = i % dim;
                if (len > l1) {
                    uint32_t p = code >> (len - l1);
                    int nb = subbits[p];
                    uint32_t rest = code & ((1u << (len - l1)) - 1);
                    uint32_t lo = rest << (nb - (len - l1));
                    for (uint32_t k = 0; k < (1u << (nb - (len - l1))); k++)
                        T->huff_lut[subbase + suboff[p] + lo + k] = (uint16_t)((len << 8) | (x << 4) | y);
                }
            }
            next = subbase + sub_next;
            if (next & 1) next++;
            if (next > 8192) return -1;
            base_of_book[t] = l1base;
            sub_of_book[t] = subbase;
            l1bits_of_book[t] = l1;
            owner = t;
        }
        T->huff_desc[t] = (uint32_t)base_of_book[owner] | ((uint32_t)l1bits_of_book[owner] << 13) |
                          ((uint32_t)M3S_HUFF_LINBITS[t] << 17);
        T->huff_sub[t] = (uint32_t)sub_of_book[owner];
        base_of_book[t] = base_of_book[owner];
        sub_of_book[t] = sub_of_book[owner];
        l1bits_of_book[t] = l1bits_of_book[owner];
    }
    // count1 table A: 6-bit LUT
    int off = M3S_HUFF_BOOK_OFF[32];
    for (int e = 0; e < 16; e++) {
        uint32_t code = M3S_HUFF_PACKED[off + e] >> 8;
        int len = M3S_HUFF_PACKED[off + e] & 0xFF;
        uint32_t lo = code << (6 - len);
        for (uint32_t k = 0; k < (1u << (6 - len)); k++) T->count1_lut[lo + k] = (uint8_t)((len << 4) | e);
    }
    return next;
}

// requantize / IMDCT / synthesis constants, generated in double with the reference's formulas and stored as R
template <typename TAB, typename R>
static void build_hybrid_tables(TAB *T)
{
    const double PI = 3.141592653589793;
    for (int i = 0; i < 256; i++) T->pow43[i] = (R)pow((double)i, 4.0 / 3.0);
    for (int i = 0; i < 4; i++) T->quarter[i] = (R)pow(2.0, i / 4.0);
    for (int i = 0; i < 36; i++)
        for (int k = 0; k < 18; k++) T->imdct_cos36[i][k] = (R)cos(PI / 72.0 * (2 * i + 1 + 18) * (2 * k + 1));
    for (int i = 0; i < 12; i++)
        for (int k = 0; k < 8; k++) T->imdct_cos12[i][k] = k < 6 ? (R)cos(PI / 24.0 * (2 * i + 1 + 6) * (2 * k + 1)) : (R)0;
    double sb[4][36];  // Frame.py:32-62
    memset(sb, 0, sizeof sb);
    for (int i = 0; i < 36; i++) sb[0][i] = sin(PI / 36.0 * (i + 0.5));
    for (int i = 0; i < 18; i++) sb[1][i] = sin(PI / 36.0 * (i + 0.5));
    for (int i = 18; i < 24; i++) sb[1][i] = 1.0;
    for (int i = 24; i < 30; i++) sb[1][i] = sin(PI / 12.0 * (i - 18.0 + 0.5));
    for (int i = 30; i < 36; i++) sb[1][i] = 1.0;  // sic: the reference's start window ends in ones
    for (int i = 0; i < 12; i++) sb[2][i] = sin(PI / 12.0 * (i + 0.5));
    for (int i = 6; i < 12; i++) sb[3][i] = sin(PI / 12.0 * (i - 6.0 + 0.5));
    for (int i = 12; i < 18; i++) sb[3][i] = 1.0;
    for (int i = 18; i < 36; i++) sb[3][i] = sin(PI / 36.0 * (i + 0.5));
    for (int b = 0; b < 4; b++)
        for (int i = 0; i < 36; i++) T->sine_block[b][i] = (R)sb[b][i];
    for (int i = 0; i < 64; i++)
        for (int j = 0; j < 32; j++) T->synth_n[i][j] = (R)cos((16.0 + i) * (2.0 * j + 1.0) * (PI / 64.0));
    for (int i = 0; i < 512; i++) T->synth_d[i] = (R)M3S_SYNTH_WINDOW[i];
    for (int i = 0; i < 8; i++) { T->alias_cs[i] = (R)M3S_ALIAS_CS[i]; T->alias_ca[i] = (R)M3S_ALIAS_CA[i]; }
}

static void build_tables(M3sDevTables *T)
{
    for (int s = 0; s < 3; s++) {
        for (int i = 0; i < 23; i++) T->sfb_long[s][i] = M3S_SFB_LONG[23 * s + i];
        for (int i = 0; i < 14; i++) T->sfb_short[s][i] = M3S_SFB_SHORT[14 * s + i];
        for (int i = 0; i < 12; i++) T->sfw_short[s][i] = M3S_SFW_SHORT[12 * s + i];
        int sfb = 0;
        for (int i = 0; i < 576; i++) {  // Frame.py:202-204
            if (i == T->sfb_long[s][sfb + 1]) sfb++;
            T->long_sfb_of[s][i] = (uint8_t)sfb;
        }
        int idx = 0;  // Frame.py:186-194
        for (int b = 0; b < 12; b++)
            for (int w = 0; w < 3; w++)
                for (int i = 0; i < T->sfw_short[s][b]; i++) T->short_sfw_of[s][idx++] = (uint8_t)(b * 3 + w);
        int total = 0, start = 0, block = 0;  // Frame.py:574-602
        for (int b = 0; b < 12; b++) {
            int w = T->sfw_short[s][b];
            for (int ss = 0; ss < w; ss++) {
                T->reorder_dst[s][total + ss + w * 0] = (uint16_t)(start + block + 0);
                T->reorder_dst[s][total + ss + w * 1] = (uint16_t)(start + block + 6);
                T->reorder_dst[s][total + ss + w * 2] = (uint16_t)(start + block + 12);
                if (block != 0 && block % 5 == 0) { start += 18; block = 0; }
                else block++;
            }
            total += 3 * w;
        }
        // The 12 short bands cover only `total` (< 576) samples: the reference's reorder drops the rest and leaves the
        // destinations it never wrote at zero (Frame.py:584,586-602).  Give every dropped source one of those holes and
        // flag it (0x8000 = "store zero"), so that the scatter is a full permutation and needs no separate clear.
        {
            bool covered[576];
            for (int i = 0; i < 576; i++) covered[i] = false;
            for (int i = 0; i < total; i++) covered[T->reorder_dst[s][i]] = true;
            int hole = 0;
            for (int i = total; i < 576; i++) {
                while (covered[hole]) hole++;
                T->reorder_dst[s][i] = (uint16_t)(hole | 0x8000);
                covered[hole] = true;
            }
            for (int i = idx; i < 576; i++) T->short_sfw_of[s][i] = 36;  // past the last band: sfb 12, window 0 (scalefactor 0)
        }
    }
    for (int i = 0; i < 16; i++) { T->slen[i][0] = M3S_SLEN[2 * i]; T->slen[i][1] = M3S_SLEN[2 * i + 1]; }
    for (int i = 0; i < 22; i++) T->pretab[i] = M3S_PRETAB[i];
    build_hybrid_tables<M3sDevTables, float>(T);
    // encoder
    memcpy(T->enwindow, M3S_ENWINDOW, sizeof T->enwindow);
    memcpy(T->enc_fl, M3S_ENC_FL, sizeof T->enc_fl);
    memcpy(T->enc_cosl, M3S_ENC_COSL, sizeof T->enc_cosl);
    memcpy(T->enc_ca, M3S_ENC_ALIAS_CA, sizeof T->enc_ca);
    memcpy(T->enc_cs, M3S_ENC_ALIAS_CS, sizeof T->enc_cs);
    memcpy(T->steptabi, M3S_ENC_STEPTABI, sizeof T->steptabi);
    for (int i = 0; i < 128; i++) { int e = 127 - i; T->steptab[i] = ldexp(M3S_ENC_QUARTER[e % 4], e / 4); }
    for (int i = 0; i < 10000; i++)  // MP3_Encoder.py:577-579 (sqrt is correctly rounded everywhere)
        T->int2idx[i] = (int32_t)(sqrt(sqrt((double)i) * (double)i) - 0.0946 + 0.5);
    for (int i = 0; i < 23; i++) { T->subdv[i][0] = M3S_SUBDV[2 * i]; T->subdv[i][1] = M3S_SUBDV[2 * i + 1]; }
    for (int i = 0; i < 32; i++) { T->pair[i][0] = M3S_STEGO_PAIR[2 * i]; T->pair[i][1] = M3S_STEGO_PAIR[2 * i + 1]; }
    memcpy(T->enc_hpacked, M3S_HUFF_PACKED, sizeof T->enc_hpacked);
    for (int i = 0; i < 34; i++) {
        T->enc_hoff[i] = M3S_HUFF_BOOK_OFF[i];
        T->enc_hdim[i] = M3S_HUFF_DIM[i];
        T->enc_linbits[i] = M3S_HUFF_LINBITS[i];
        T->enc_linmax[i] = M3S_HUFF_LINMAX[i];
    }
}

static_assert(sizeof(M3S_HUFF_PACKED) / sizeof(uint32_t) == 1410, "packed code book size");

extern "C" int m3s_version(void) { return 400; }

extern "C" int m3s_create(int device, m3s_handle_t *out)
{
    if (!out) return M3S_ERR_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return M3S_ERR_NO_DEVICE;
    m3s_ctx *h = new m3s_ctx();
    h->device = device;
    cudaDeviceProp prop;
    if (cudaSetDevice(device) != cudaSuccess || cudaGetDeviceProperties(&prop, device) != cudaSuccess) {
        delete h;
        return M3S_ERR_NO_DEVICE;
    }
    if (prop.major < 10) {  // kernels are built for sm_100a only; there is no fallback path
        delete h;
        return M3S_ERR_NO_DEVICE;
    }
    h->sm_count = prop.multiProcessorCount;
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);   // the main stream outranks the helper streams (aux analysis, copies)
    if (cudaStreamCreateWithPriority(&h->own_stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess) {
        delete h;
        return M3S_ERR_CUDA;
    }
    h->stream = h->own_stream;
    if (const char *cb = getenv("M3S_ENC_CHUNK_FRAMES")) h->enc_chunk_budget = atoll(cb);
    if (const char *cb = getenv("M3S_DEC_WAVE_BYTES")) h->dec_wave_bytes = atoll(cb);
    M3sDevTables *T = new M3sDevTables();
    memset(T, 0, sizeof *T);
    build_tables(T);
    if (build_huff_lut(T) < 0) {
        delete T;
        cudaStreamDestroy(h->own_stream);
        delete h;
        return M3S_ERR_STATE;
    }
    cudaError_t e = cudaMalloc(&h->d_tab, sizeof(M3sDevTables));
    if (e == cudaSuccess) e = cudaMemcpy(h->d_tab, T, sizeof(M3sDevTables), cudaMemcpyHostToDevice);
    delete T;
    if (e == cudaSuccess) {
        M3sDevTablesD *TD = new M3sDevTablesD();
        build_hybrid_tables<M3sDevTablesD, double>(TD);
        e = cudaMalloc(&h->d_tab_f64, sizeof(M3sDevTablesD));
        if (e == cudaSuccess) e = cudaMemcpy(h->d_tab_f64, TD, sizeof(M3sDevTablesD), cudaMemcpyHostToDevice);
        delete TD;
    }
    if (e == cudaSuccess && m3s_upload_fast_const() != 0) e = cudaErrorUnknown;
    if (e != cudaSuccess) {
        if (h->d_tab) cudaFree(h->d_tab);
        if (h->d_tab_f64) cudaFree(h->d_tab_f64);
        cudaStreamDestroy(h->own_stream);
        delete h;
        return M3S_ERR_CUDA;
    }
    *out = h;
    return M3S_OK;
}

static void timing_resolve(m3s_ctx *h);

int m3s_pipeline_init(m3s_ctx *h)
{
    if (h->copy_in) return M3S_OK;
    M3S_CUDA(h, cudaStreamCreateWithFlags(&h->copy_in, cudaStreamNonBlocking));
    M3S_CUDA(h, cudaStreamCreateWithFlags(&h->copy_out, cudaStreamNonBlocking));
    M3S_CUDA(h, cudaStreamCreateWithFlags(&h->aux, cudaStreamNonBlocking));
    for (int i = 0; i < 2; i++) {
        M3S_CUDA(h, cudaEventCreateWithFlags(&h->ev_ana[i], cudaEventDisableTiming));
        M3S_CUDA(h, cudaEventCreateWithFlags(&h->ev_pack[i], cudaEventDisableTiming));
    }
    for (int i = 0; i < 2; i++) {
        M3S_CUDA(h, cudaEventCreateWithFlags(&h->ev_in[i], cudaEventDisableTiming));
        M3S_CUDA(h, cudaEventCreateWithFlags(&h->ev_free[i], cudaEventDisableTiming));
    }
    return M3S_OK;
}

// Bulk PCIe transfers are issued in pieces of at most M3S_COPY_PIECE bytes: a copy engine serves one command at a time,
// so a multi-GB command would hold back every small descriptor copy (and the host thread waiting on it) of this and of
// other handles for tens of milliseconds; with bounded pieces those slot in within about a millisecond.
#define M3S_COPY_PIECE ((size_t)16 << 20)

cudaError_t m3s_copy_bulk(void *dst, const void *src, size_t bytes, cudaMemcpyKind kind, cudaStream_t s)
{
    for (size_t o = 0; o < bytes; o += M3S_COPY_PIECE) {
        const size_t n = bytes - o < M3S_COPY_PIECE ? bytes - o : M3S_COPY_PIECE;
        const cudaError_t e = cudaMemcpyAsync((char *)dst + o, (const char *)src + o, n, kind, s);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

int m3s_copy_paced(m3s_ctx *h, void *dst, const void *src, size_t bytes, cudaMemcpyKind kind)
{
    for (int i = 0; i < 3; i++)
        if (!h->ev_pace[i]) M3S_CUDA(h, cudaEventCreateWithFlags(&h->ev_pace[i], cudaEventDisableTiming));
    int i = 0;
    for (size_t o = 0; o < bytes; o += M3S_COPY_PIECE, i++) {
        const size_t n = bytes - o < M3S_COPY_PIECE ? bytes - o : M3S_COPY_PIECE;
        if (i >= 2) M3S_CUDA(h, cudaEventSynchronize(h->ev_pace[(i - 2) % 3]));
        M3S_CUDA(h, cudaMemcpyAsync((char *)dst + o, (const char *)src + o, n, kind, h->stream));
        M3S_CUDA(h, cudaEventRecord(h->ev_pace[i % 3], h->stream));
    }
    return M3S_OK;
}

cudaError_t m3s_copy_rows(const std::vector<M3sRow> &rows, cudaMemcpyKind kind, cudaStream_t s)
{
    const size_t n = rows.size();
    if (n == 0) return cudaSuccess;
    bool regular = n > 1 && rows[0].bytes > 0;
    ptrdiff_t dp = 0, sp = 0;
    if (regular) {
        dp = rows[1].dst - rows[0].dst;
        sp = rows[1].src - rows[0].src;
        regular = dp >= (ptrdiff_t)rows[0].bytes && sp >= (ptrdiff_t)rows[0].bytes && dp <= 0x7FFFFFFF && sp <= 0x7FFFFFFF;
        for (size_t i = 1; regular && i < n; i++)
            regular = rows[i].bytes == rows[0].bytes && rows[i].dst - rows[i - 1].dst == dp && rows[i].src - rows[i - 1].src == sp;
    }
    if (regular) {
        size_t per = M3S_COPY_PIECE / rows[0].bytes;   // rows per 2-D command
        if (per < 1) per = 1;
        for (size_t i = 0; i < n; i += per) {
            const size_t h = n - i < per ? n - i : per;
            const cudaError_t e = cudaMemcpy2DAsync(rows[i].dst, (size_t)dp, rows[i].src, (size_t)sp, rows[0].bytes, h, kind, s);
            if (e != cudaSuccess) return e;
        }
        return cudaSuccess;
    }
    for (const M3sRow &r : rows)
        if (r.bytes) {
            const cudaError_t e = m3s_copy_bulk(r.dst, r.src, r.bytes, kind, s);
            if (e != cudaSuccess) return e;
        }
    return cudaSuccess;
}

static void free_buf(M3sBuf &b)
{
    if (b.p) cudaFree(b.p);
    b.p = nullptr;
    b.cap = 0;
}

extern "C" int m3s_destroy(m3s_handle_t h)
{
    if (!h) return M3S_ERR_ARG;
    cudaSetDevice(h->device);
    m3s_sync_streams(h);
    M3sBuf *bufs[] = {&h->b_stage_in[0], &h->b_stage_in[1], &h->b_pcm_stage[0], &h->b_pcm_stage[1],
                      &h->b_sf, &h->b_S, &h->b_spec,
                      &h->b_work, &h->b_spec_export, &h->e_pcm, &h->e_clips, &h->e_out, &h->e_payload, &h->e_misc, &h->e_pad,
                      &h->e_tabs, &h->e_state, &h->e_lastix, &h->e_work, &h->e_cand};
    for (M3sBuf *b : bufs) free_buf(*b);
    for (M3sEncSet &es : h->es)
        for (M3sBuf *b : {&es.mdct, &es.gran, &es.ix, &es.info, &es.scfsi, &es.var, &es.sum}) free_buf(*b);
    for (M3sScanSet &ss : h->ss) {
        M3sBuf *sb[] = {&ss.files, &ss.fouts, &ss.tmp_pos, &ss.fr_pos, &ss.fr_P, &ss.fr_meta, &ss.fr_carry, &ss.fr_reveal, &ss.fr_file,
                        &ss.units, &ss.tabids, &ss.reveal, &ss.layout, &ss.irr};
        for (M3sBuf *b : sb) free_buf(*b);
        if (ss.fouts_mapped) cudaFreeHost(ss.fouts_mapped);
        if (ss.pin) cudaFreeHost(ss.pin);
    }
    for (int i = 0; i < 2; i++) {
        if (h->work_pin[i]) cudaFreeHost(h->work_pin[i]);
        if (h->ev_d_h2d[i]) { cudaEventDestroy(h->ev_d_h2d[i]); cudaEventDestroy(h->ev_d_scan[i]); cudaEventDestroy(h->ev_d_comp[i]); cudaEventDestroy(h->ev_d_out[i]); }
    }
    if (h->rev_mapped) cudaFreeHost(h->rev_mapped);
    timing_resolve(h);
    for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
    if (h->d_tab) cudaFree(h->d_tab);
    if (h->d_tab_f64) cudaFree(h->d_tab_f64);
    if (h->copy_in) cudaStreamDestroy(h->copy_in);
    if (h->copy_out) cudaStreamDestroy(h->copy_out);
    if (h->aux) cudaStreamDestroy(h->aux);
    for (int i = 0; i < 2; i++)
        if (h->ev_ana[i]) { cudaEventDestroy(h->ev_ana[i]); cudaEventDestroy(h->ev_pack[i]); }
    for (int i = 0; i < 2; i++) {
        if (h->ev_in[i]) cudaEventDestroy(h->ev_in[i]);
        if (h->ev_free[i]) cudaEventDestroy(h->ev_free[i]);
    }
    for (int i = 0; i < 3; i++)
        if (h->ev_pace[i]) cudaEventDestroy(h->ev_pace[i]);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    delete h;
    return M3S_OK;
}

extern "C" const char *m3s_last_error(m3s_handle_t h) { return h ? h->err.c_str() : "null handle"; }

extern "C" int m3s_set_stream(m3s_handle_t h, void *cuda_stream)
{
    if (!h) return M3S_ERR_ARG;
    cudaStreamSynchronize(h->stream);
    h->stream = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
    return M3S_OK;
}

extern "C" int m3s_synchronize(m3s_handle_t h)
{
    if (!h) return M3S_ERR_ARG;
    M3S_CUDA(h, cudaSetDevice(h->device));
    M3S_CUDA(h, cudaStreamSynchronize(h->stream));
    return M3S_OK;
}

extern "C" int64_t m3s_launch_count(m3s_handle_t h) { return h ? h->launches : -1; }

// ------------------------------------------------------------------------------------------------
// per-kernel device timing (bench.py roofline): event pairs on the launching stream, resolved lazily
// ------------------------------------------------------------------------------------------------
static cudaEvent_t take_event(m3s_ctx *h)
{
    if (!h->ev_pool.empty()) {
        cudaEvent_t e = h->ev_pool.back();
        h->ev_pool.pop_back();
        return e;
    }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}

void m3s_time_begin(m3s_ctx *h, int id)
{
    m3s_ctx::Timed t;
    t.id = id;
    t.e0 = take_event(h);
    t.e1 = take_event(h);
    cudaEventRecord(t.e0, h->launch_stream ? h->launch_stream : h->stream);
    h->timed.push_back(t);
}

void m3s_time_end(m3s_ctx *h)
{
    if (!h->timed.empty()) cudaEventRecord(h->timed.back().e1, h->launch_stream ? h->launch_stream : h->stream);
}

static void timing_resolve(m3s_ctx *h)
{
    cudaStreamSynchronize(h->stream);
    if (h->aux) { cudaStreamSynchronize(h->aux); cudaStreamSynchronize(h->copy_out); }
    for (auto &t : h->timed) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, t.e0, t.e1) == cudaSuccess) h->k_ms[t.id] += ms;
        h->ev_pool.push_back(t.e0);
        h->ev_pool.push_back(t.e1);
    }
    h->timed.clear();
}

extern "C" int m3s_timing_enable(m3s_handle_t h, int on)
{
    if (!h) return M3S_ERR_ARG;
    M3S_CUDA(h, cudaSetDevice(h->device));
    timing_resolve(h);
    for (int i = 0; i < M3S_K_COUNT; i++) { h->k_ms[i] = 0; h->k_launches[i] = 0; }
    h->timing = on != 0;
    return M3S_OK;
}

extern "C" int m3s_timing_get(m3s_handle_t h, int kernel_id, double *total_ms, int64_t *launches)
{
    if (!h || kernel_id < 0 || kernel_id >= M3S_K_COUNT) return M3S_ERR_ARG;
    M3S_CUDA(h, cudaSetDevice(h->device));
    timing_resolve(h);
    if (total_ms) *total_ms = h->k_ms[kernel_id];
    if (launches) *launches = h->k_launches[kernel_id];
    return M3S_OK;
}

extern "C" const char *m3s_kernel_name(int kernel_id)
{
    static const char *names[M3S_K_COUNT] = {"k_walk", "k_fscan", "k_sideinfo", "k_strip", "k_huff", "k_spec_export", "k_hybrid",
                                             "k_enc_analysis", "k_enc_rate", "k_enc_resolve", "k_enc_pack", "k_enc_emit",
                                             "k_enc_offsets"};
    return kernel_id >= 0 && kernel_id < M3S_K_COUNT ? names[kernel_id] : "?";
}

// ------------------------------------------------------------------------------------------------
// table export for tests/test_tables.py (host-only, needs no GPU)
// ------------------------------------------------------------------------------------------------
template <typename T>
static int64_t export_arr(const T *src, int64_t n, double *out, int64_t cap)
{
    if (out)
        for (int64_t i = 0; i < n && i < cap; i++) out[i] = (double)src[i];
    return n;
}

extern "C" int64_t m3s_table_export(int which, double *out, int64_t cap)
{
    static M3sDevTables *T = nullptr;
    if (!T) {
        T = new M3sDevTables();
        memset(T, 0, sizeof *T);
        build_tables(T);
        build_huff_lut(T);
    }
    switch (which) {
    case M3S_TAB_HUFF_PACKED: return export_arr(M3S_HUFF_PACKED, 1410, out, cap);
    case M3S_TAB_HUFF_BOOK_OFF: return export_arr(M3S_HUFF_BOOK_OFF, 34, out, cap);
    case M3S_TAB_HUFF_DIM: return export_arr(M3S_HUFF_DIM, 34, out, cap);
    case M3S_TAB_HUFF_LINBITS: return export_arr(M3S_HUFF_LINBITS, 34, out, cap);
    case M3S_TAB_SFB_LONG: return export_arr(&T->sfb_long[0][0], 69, out, cap);
    case M3S_TAB_SFB_SHORT: return export_arr(&T->sfb_short[0][0], 42, out, cap);
    case M3S_TAB_SFW_SHORT: return export_arr(&T->sfw_short[0][0], 36, out, cap);
    case M3S_TAB_SLEN: return export_arr(&T->slen[0][0], 32, out, cap);
    case M3S_TAB_PRETAB: return export_arr(T->pretab, 21, out, cap);
    case M3S_TAB_SYNTH_WINDOW: return export_arr(M3S_SYNTH_WINDOW, 512, out, cap);
    case M3S_TAB_ENWINDOW: return export_arr(T->enwindow, 512, out, cap);
    case M3S_TAB_ENC_FL: return export_arr(&T->enc_fl[0][0], 2048, out, cap);
    case M3S_TAB_ENC_COSL: return export_arr(&T->enc_cosl[0][0], 648, out, cap);
    case M3S_TAB_ENC_STEPTABI: return export_arr(T->steptabi, 128, out, cap);
    case M3S_TAB_ENC_STEPTAB: return export_arr(T->steptab, 128, out, cap);
    case M3S_TAB_ENC_INT2IDX: return export_arr(T->int2idx, 10000, out, cap);
    case M3S_TAB_ENC_CA: return export_arr(T->enc_ca, 8, out, cap);
    case M3S_TAB_ENC_CS: return export_arr(T->enc_cs, 8, out, cap);
    case M3S_TAB_SUBDV: return export_arr(&T->subdv[0][0], 46, out, cap);
    case M3S_TAB_STEGO_PAIR: return export_arr(&T->pair[0][0], 64, out, cap);
    case M3S_TAB_ALIAS_CS: return export_arr(M3S_ALIAS_CS, 8, out, cap);
    case M3S_TAB_ALIAS_CA: return export_arr(M3S_ALIAS_CA, 8, out, cap);
    case M3S_TAB_H0_MASK: { uint32_t m = M3S_H0_MASK; return export_arr(&m, 1, out, cap); }
    default: return -1;
    }
}
