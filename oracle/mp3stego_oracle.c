/*
 * mp3stego_oracle.c -- CPU ORACLE (test infrastructure, NOT product code).
 *
 * A plain-C, single-threaded restatement of the reference's per-granule codec hot path
 * (tomershay100/mp3-steganography-lib, package mp3stego 1.1.8), kept deliberately sequential and
 * stateful in the same way the reference is, so that its quirks (stale side-info fields, count-down
 * table search, 4-byte flush truncation, ...) are reproduced rather than "fixed".
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load
 * this library.  The CUDA product path never links or calls it.
 *
 * Parity pin: tests/test_oracle_golden.py checks this file against golden vectors produced by running
 * the unmodified Python reference in the development container (tests/golden/make_golden.py).
 *
 * Each function cites the reference file:line it follows (paths relative to /root/reference/mp3stego).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "oracle_tables.h"

#define ORA_API __attribute__((visibility("default")))

/* ------------------------------------------------------------------------------------------------
 * small helpers
 * ---------------------------------------------------------------------------------------------- */

typedef struct {
    const uint8_t *p;
    int64_t len;
} bytes_t;

/* decoder/util.py:22-64 get_bits: MSB-first, bytes beyond the buffer read as zero, slice_len <= 32 */
static uint32_t get_bits(const uint8_t *buf, int64_t len, int64_t start_bit, int n)
{
    uint32_t r = 0;
    for (int i = 0; i < n; i++) {
        int64_t b = start_bit + i;
        int64_t byte = b >> 3;
        uint32_t bit = 0;
        if (byte < len) bit = (buf[byte] >> (7 - (b & 7))) & 1u;
        r = (r << 1) | bit;
    }
    return r;
}

/* growable byte vector */
typedef struct {
    uint8_t *p;
    int64_t n, cap;
} vec_t;
static void vec_push(vec_t *v, const uint8_t *src, int64_t n)
{
    if (n <= 0) return;
    if (v->n + n > v->cap) {
        int64_t c = v->cap ? v->cap * 2 : 4096;
        while (c < v->n + n) c *= 2;
        v->p = (uint8_t *)realloc(v->p, (size_t)c);
        v->cap = c;
    }
    memcpy(v->p + v->n, src, (size_t)n);
    v->n += n;
}

/* Python list slicing a[lo:hi] (step 1) incl. negative-index wrap, appended to v (Frame.py:348-356) */
static void py_slice_push(vec_t *v, const uint8_t *a, int64_t len, int64_t lo, int64_t hi)
{
    if (lo < 0) { lo += len; if (lo < 0) lo = 0; }
    if (hi < 0) { hi += len; if (hi < 0) hi = 0; }
    if (lo > len) lo = len;
    if (hi > len) hi = len;
    if (hi > lo) vec_push(v, a + lo, hi - lo);
}

/* ================================================================================================
 * DECODER
 * ============================================================================================== */

typedef struct {
    /* FrameHeader.py */
    int layer, crc /* protection bit: 1 = no CRC */, bit_rate, sampling_rate, padding, channel_mode, channels;
    int mode_ext0, mode_ext1, sr_index;
    const int *long_win, *short_idx, *short_w;
    /* FrameSideInformation.py (persistent across frames: MP3_Parser.py:23, Frame.py:232) */
    int main_data_begin;
    int scfsi[2][4];
    int part2_3_length[2][2], big_value[2][2], global_gain[2][2], scale_fac_compress[2][2];
    int window_switching[2][2], block_type[2][2], mixed_block_flag[2][2];
    int table_select[2][2][3], sub_block_gain[2][2][3], region0_count[2][2], region1_count[2][2];
    int pre_flag[2][2], scale_fac_scale[2][2], count1table_select[2][2];
    int scale_fac_l[2][2][22], scale_fac_s[2][2][3][13];
    /* Frame.py */
    double prev_frame_size[9];
    int frame_size;
    double prev_samples[2][32][18];
    double fifo[2][1024];
    double samples[2][2][576];
    double pcm[1152][2];
    vec_t main_data;
    double sine_block[4][36];
    double synth_n[64][32];
    double cos36[36][18], cos12[12][6];
} dec_t;

typedef struct ora_dec_result {
    int64_t n_frames;
    int64_t n_pcm_rows;
    int channels, sampling_rate, bit_rate, status;
    double *pcm;      /* [n_pcm_rows][channels] */
    int32_t *spectra; /* [n_frames][gr][ch][576] integer spectra after Huffman decode */
    uint8_t *tables;  /* [n_frames][12] (ch, gr, region) */
    char *bits;       /* reveal bit string, NUL terminated */
    int64_t n_bits;
    int32_t *side;    /* [n_frames][gr][ch][ORA_SIDE_FIELDS] */
    int64_t *frame_off; /* [n_frames] byte offset of each frame header */
    int32_t *frame_mdb; /* [n_frames] main_data_begin */
    double *xr;       /* [n_frames][gr][ch][576] after requantize+stereo+reorder/alias (hybrid input) */
} ora_dec_result;

#define ORA_SIDE_FIELDS 20

/* FrameHeader.py:51-192.  Returns 0 if ok, <0 when the stream leaves the supported domain
 * (MPEG-1 Layer III, 32/44.1/48 kHz, bitrate index != 15), where the reference raises or mis-sizes. */
static int dec_header(dec_t *d, const uint8_t *b)
{
    int ver_bits = (b[1] >> 3) & 3; /* FrameHeader.py:70-81 */
    if (ver_bits != 3) return -2;
    d->layer = 4 - ((b[1] >> 1) & 3); /* :83-91 */
    if (d->layer != 3) return -3;
    d->crc = b[1] & 1; /* :93-97 */
    int sri = (b[2] >> 2) & 3; /* :110-123 */
    if (sri == 3) return -4;
    static const int rates[3] = {44100, 48000, 32000};
    d->sampling_rate = rates[sri];
    d->sr_index = sri;
    d->long_win = ORA_SFB_LONG + 23 * sri; /* :125-143 */
    d->short_idx = ORA_SFB_SHORT + 14 * sri;
    d->short_w = ORA_SFW_SHORT + 12 * sri;
    d->channel_mode = (b[3] >> 6) & 3; /* :145-154 */
    d->channels = d->channel_mode == 3 ? 1 : 2;
    d->mode_ext0 = b[3] & 0x20; /* :156-161 */
    d->mode_ext1 = b[3] & 0x10;
    d->padding = (b[2] & 2) ? 1 : 0; /* :163-167 */
    static const int br[14] = {32, 40, 48, 56, 64, 80, 96, 112, 128, 160, 192, 224, 256, 320};
    int bi = (b[2] >> 4) - 1; /* :169-192; index -1 wraps to the last entry in Python */
    if (bi == 14) return -5;
    if (bi < 0) bi = 13;
    d->bit_rate = br[bi] * 1000;
    return 0;
}

/* Frame.py:288-316 */
static void dec_set_frame_size(dec_t *d)
{
    for (int i = 8; i > 0; i--) d->prev_frame_size[i] = d->prev_frame_size[i - 1];
    d->prev_frame_size[0] = d->frame_size;
    d->frame_size = (int)(((1152.0 / 8.0) * d->bit_rate) / d->sampling_rate);
    if (d->padding) d->frame_size += 1;
}

/* FrameSideInformation.py:39-137 */
static void dec_side_info(dec_t *d, const uint8_t *buf, int64_t len)
{
    int64_t off = 0;
    d->main_data_begin = (int)get_bits(buf, len, 0, 9);
    off += 9;
    off += d->channel_mode == 3 ? 5 : 3;
    for (int ch = 0; ch < d->channels; ch++)
        for (int b = 0; b < 4; b++) d->scfsi[ch][b] = get_bits(buf, len, off++, 1) != 0;
    for (int gr = 0; gr < 2; gr++)
        for (int ch = 0; ch < d->channels; ch++) {
            d->part2_3_length[gr][ch] = get_bits(buf, len, off, 12); off += 12;
            d->big_value[gr][ch] = get_bits(buf, len, off, 9); off += 9;
            d->global_gain[gr][ch] = get_bits(buf, len, off, 8); off += 8;
            d->scale_fac_compress[gr][ch] = get_bits(buf, len, off, 4); off += 4;
            d->window_switching[gr][ch] = get_bits(buf, len, off, 1) == 1; off += 1;
            if (d->window_switching[gr][ch]) {
                d->block_type[gr][ch] = get_bits(buf, len, off, 2); off += 2;
                d->mixed_block_flag[gr][ch] = get_bits(buf, len, off, 1) == 1; off += 1;
                d->region0_count[gr][ch] = d->block_type[gr][ch] == 2 ? 8 : 7;
                d->region1_count[gr][ch] = 20 - d->region0_count[gr][ch];
                for (int r = 0; r < 2; r++) { d->table_select[gr][ch][r] = get_bits(buf, len, off, 5); off += 5; }
                for (int w = 0; w < 3; w++) { d->sub_block_gain[gr][ch][w] = get_bits(buf, len, off, 3); off += 3; }
            } else {
                d->block_type[gr][ch] = 0;
                d->mixed_block_flag[gr][ch] = 0;
                for (int r = 0; r < 3; r++) { d->table_select[gr][ch][r] = get_bits(buf, len, off, 5); off += 5; }
                d->region0_count[gr][ch] = get_bits(buf, len, off, 4); off += 4;
                d->region1_count[gr][ch] = get_bits(buf, len, off, 3); off += 3;
            }
            d->pre_flag[gr][ch] = get_bits(buf, len, off, 1); off += 1;
            d->scale_fac_scale[gr][ch] = get_bits(buf, len, off, 1); off += 1;
            d->count1table_select[gr][ch] = get_bits(buf, len, off, 1); off += 1;
        }
}

/* Frame.py:365-441 */
static int64_t dec_unpack_scale_fac(dec_t *d, int gr, int ch, int64_t bit)
{
    const uint8_t *md = d->main_data.p;
    int64_t ml = d->main_data.n;
    int sl0 = ORA_SLEN[2 * d->scale_fac_compress[gr][ch]];
    int sl1 = ORA_SLEN[2 * d->scale_fac_compress[gr][ch] + 1];
    if (d->block_type[gr][ch] == 2 && d->window_switching[gr][ch]) {
        if (d->mixed_block_flag[gr][ch] == 1) {
            for (int sfb = 0; sfb < 8; sfb++) { d->scale_fac_l[gr][ch][sfb] = get_bits(md, ml, bit, sl0); bit += sl0; }
            for (int sfb = 3; sfb < 6; sfb++)
                for (int w = 0; w < 3; w++) { d->scale_fac_s[gr][ch][w][sfb] = get_bits(md, ml, bit, sl0); bit += sl0; }
        } else {
            for (int sfb = 0; sfb < 6; sfb++)
                for (int w = 0; w < 3; w++) { d->scale_fac_s[gr][ch][w][sfb] = get_bits(md, ml, bit, sl0); bit += sl0; }
        }
        for (int sfb = 6; sfb < 12; sfb++)
            for (int w = 0; w < 3; w++) { d->scale_fac_s[gr][ch][w][sfb] = get_bits(md, ml, bit, sl1); bit += sl1; }
        for (int w = 0; w < 3; w++) d->scale_fac_s[gr][ch][w][12] = 0;
    } else {
        if (gr == 0) {
            for (int sfb = 0; sfb < 11; sfb++) { d->scale_fac_l[gr][ch][sfb] = get_bits(md, ml, bit, sl0); bit += sl0; }
            for (int sfb = 11; sfb < 21; sfb++) { d->scale_fac_l[gr][ch][sfb] = get_bits(md, ml, bit, sl1); bit += sl1; }
        } else {
            static const int SB[4] = {6, 11, 16, 21}, PSB[4] = {0, 6, 11, 16};
            for (int i = 0; i < 4; i++) {
                int sl = i < 2 ? sl0 : sl1;
                for (int sfb = PSB[i]; sfb < SB[i]; sfb++) {
                    if (d->scfsi[ch][i]) d->scale_fac_l[gr][ch][sfb] = d->scale_fac_l[0][ch][sfb];
                    else { d->scale_fac_l[gr][ch][sfb] = get_bits(md, ml, bit, sl); bit += sl; }
                }
            }
        }
        d->scale_fac_l[gr][ch][21] = 0;
    }
    return bit;
}

/* Frame.py:443-559 */
static void dec_unpack_samples(dec_t *d, int gr, int ch, int64_t bit, int64_t max_bit)
{
    const uint8_t *md = d->main_data.p;
    int64_t ml = d->main_data.n;
    double *s = d->samples[gr][ch];
    for (int i = 0; i < 576; i++) s[i] = 0;
    int region0, region1;
    if (d->window_switching[gr][ch] && d->block_type[gr][ch] == 2) { region0 = 36; region1 = 576; }
    else {
        region0 = d->long_win[d->region0_count[gr][ch] + 1];
        /* index can reach 23 for region0+region1 = 15+7; numpy would raise -- clamp to the last entry */
        int idx = d->region0_count[gr][ch] + 1 + d->region1_count[gr][ch] + 1;
        if (idx > 22) idx = 22;
        region1 = d->long_win[idx];
    }
    int sample = 0;
    while (sample < d->big_value[gr][ch] * 2 && sample + 1 < 576 + 2) {
        if (sample >= 576) break; /* reference would raise IndexError; stop */
        int tn;
        if (sample < region0) tn = d->table_select[gr][ch][0];
        else if (sample < region1) tn = d->table_select[gr][ch][1];
        else tn = d->table_select[gr][ch][2];
        if (tn == 0) { s[sample] = 0; sample += 2; continue; }
        int mx = ORA_HUFF_MAX[tn];
        uint32_t bs = get_bits(md, ml, bit, 32);
        int found = 0;
        for (int row = 0; row < mx && !found; row++)
            for (int col = 0; col < mx; col++) {
                int e = ORA_HUFF_OFF[tn] + mx * row + col;
                uint32_t code = ORA_HUFF_CODE_L[e];
                int size = ORA_HUFF_LEN[e];
                if ((code >> (32 - size)) == (bs >> (32 - size))) {
                    bit += size;
                    int v[2] = {row, col};
                    for (int i = 0; i < 2; i++) {
                        int linbit = 0;
                        if (ORA_HUFF_LINBITS[tn] != 0 && v[i] == mx - 1) {
                            linbit = (int)get_bits(md, ml, bit, ORA_HUFF_LINBITS[tn]);
                            bit += ORA_HUFF_LINBITS[tn];
                        }
                        int sign = 1;
                        if (v[i] > 0) { sign = get_bits(md, ml, bit, 1) > 0 ? -1 : 1; bit += 1; }
                        s[sample + i] = (double)(sign * (v[i] + linbit));
                    }
                    found = 1;
                    break;
                }
            }
        sample += 2;
    }
    while (bit < max_bit && sample + 4 < 576) {
        int v[4] = {0, 0, 0, 0};
        if (d->count1table_select[gr][ch] == 1) {
            uint32_t bs = get_bits(md, ml, bit, 4);
            bit += 4;
            v[0] = (bs & 8) ? 0 : 1; v[1] = (bs & 4) ? 0 : 1; v[2] = (bs & 2) ? 0 : 1; v[3] = (bs & 1) ? 0 : 1;
        } else {
            uint32_t bs = get_bits(md, ml, bit, 32);
            for (int e = 0; e < 16; e++) {
                uint32_t code = ORA_QUAD_CODE_L[e];
                int size = ORA_QUAD_LEN[e];
                if ((code >> (32 - size)) == (bs >> (32 - size))) {
                    bit += size;
                    v[0] = (e >> 3) & 1; v[1] = (e >> 2) & 1; v[2] = (e >> 1) & 1; v[3] = e & 1;
                    break;
                }
            }
        }
        for (int i = 0; i < 4; i++)
            if (v[i] > 0) { if (get_bits(md, ml, bit, 1) == 1) v[i] = -v[i]; bit += 1; }
        for (int i = 0; i < 4; i++) s[sample + i] = v[i];
        sample += 4;
    }
}

/* Frame.py:318-363 */
static void dec_set_main_data(dec_t *d, const uint8_t *file, int64_t flen, int64_t curr)
{
    int constant = d->channel_mode == 3 ? 21 : 36;
    if (d->crc == 0) constant += 2;
    if (d->main_data_begin == 0) {
        d->main_data.n = 0;
        py_slice_push(&d->main_data, file + curr, flen - curr, constant, d->frame_size);
    } else {
        double bound = 0;
        for (int frame = 0; frame < 9; frame++) {
            bound += d->prev_frame_size[frame] - constant;
            if (d->main_data_begin < bound) {
                double ptr_offset = d->main_data_begin + frame * constant;
                double part[9] = {0};
                part[frame] = d->main_data_begin;
                for (int i = 0; i < frame; i++) { part[i] = d->prev_frame_size[i] - constant; part[frame] -= part[i]; }
                d->main_data.n = 0;
                int64_t loc = (int64_t)(curr - ptr_offset);
                py_slice_push(&d->main_data, file, flen, loc, loc + (int64_t)part[frame]);
                ptr_offset -= part[frame] + constant;
                for (int i = frame - 1; i >= 0; i--) {
                    loc = (int64_t)(curr - ptr_offset);
                    py_slice_push(&d->main_data, file, flen, loc, loc + (int64_t)part[i]);
                    ptr_offset -= part[i] + constant;
                }
                py_slice_push(&d->main_data, file + curr, flen - curr, constant, d->frame_size);
                break;
            }
        }
        /* no window matched: main_data stays stale (A.D9) */
    }
}

/* Frame.py:157-218 */
static void dec_requantize(dec_t *d, int gr, int ch)
{
    int window = 0, sfb = 0, sample = 0, i = 0;
    double mult = d->scale_fac_scale[gr][ch] == 0 ? 0.5 : 1.0;
    double *s = d->samples[gr][ch];
    while (sample < 576) {
        double exp1, exp2;
        if (d->block_type[gr][ch] == 2 || (d->mixed_block_flag[gr][ch] && sfb >= 8)) {
            int swv = sfb < 12 ? d->short_w[sfb] : 0;
            if (i == swv) {
                i = 0;
                if (window == 2) { window = 0; sfb += 1; }
                else window += 1;
            }
            exp1 = d->global_gain[gr][ch] - 210.0 - 8.0 * d->sub_block_gain[gr][ch][window];
            /* scale_fac_s has 13 columns; numba does not bounds-check, keep the index in range */
            exp2 = mult * d->scale_fac_s[gr][ch][window][sfb < 13 ? sfb : 12];
        } else {
            if (sample == d->long_win[sfb + 1]) sfb += 1;
            exp1 = d->global_gain[gr][ch] - 210.0;
            int pt = sfb < 21 ? ORA_PRETAB[sfb] : 0;
            exp2 = mult * (d->scale_fac_l[gr][ch][sfb] + d->pre_flag[gr][ch] * pt);
        }
        double sign = s[sample] < 0 ? -1.0 : 1.0;
        double a = pow(fabs(s[sample]), 4.0 / 3.0);
        double b = pow(2.0, exp1 / 4.0);
        double c = pow(2.0, -exp2);
        s[sample] = sign * a * b * c;
        sample += 1;
        i += 1;
    }
}

/* Frame.py:561-572 */
static void dec_ms_stereo(dec_t *d, int gr)
{
    const double SQRT2 = sqrt(2.0);
    for (int i = 0; i < 576; i++) {
        double m = d->samples[gr][0][i], s = d->samples[gr][1][i];
        d->samples[gr][0][i] = (m + s) / SQRT2;
        d->samples[gr][1][i] = (m - s) / SQRT2;
    }
}

/* Frame.py:574-602 */
static void dec_reorder(dec_t *d, int gr, int ch)
{
    int total = 0, start = 0, block = 0;
    double tmp[576 + 32];
    memset(tmp, 0, sizeof tmp);
    double *s = d->samples[gr][ch];
    for (int sb = 0; sb < 12; sb++) {
        int w = d->short_w[sb];
        for (int ss = 0; ss < w; ss++) {
            tmp[start + block + 0] = s[total + ss + w * 0];
            tmp[start + block + 6] = s[total + ss + w * 1];
            tmp[start + block + 12] = s[total + ss + w * 2];
            if (block != 0 && block % 5 == 0) { start += 18; block = 0; }
            else block += 1;
        }
        total += w * 3;
    }
    for (int i = 0; i < 576; i++) s[i] = tmp[i];
}

/* Frame.py:604-622 */
static void dec_alias(dec_t *d, int gr, int ch)
{
    double *s = d->samples[gr][ch];
    int sb_max = d->mixed_block_flag[gr][ch] ? 2 : 32;
    for (int sb = 1; sb < sb_max; sb++)
        for (int k = 0; k < 8; k++) {
            int o1 = 18 * sb - k - 1, o2 = 18 * sb + k;
            double s1 = s[o1], s2 = s[o2];
            s[o1] = s1 * ORA_ALIAS_CS[k] - s2 * ORA_ALIAS_CA[k];
            s[o2] = s2 * ORA_ALIAS_CS[k] + s1 * ORA_ALIAS_CA[k];
        }
}

/* Frame.py:106-154 */
static void dec_imdct(dec_t *d, int gr, int ch)
{
    double sb36[36], tmp[36];
    int bt = d->block_type[gr][ch];
    int n = bt == 2 ? 12 : 36, half = n / 2, sample = 0;
    double *s = d->samples[gr][ch];
    for (int block = 0; block < 32; block++) {
        for (int k = 0; k < 36; k++) sb36[k] = 0; /* np.zeros(36) once; entries are fully rewritten below */
        for (int win = 0; win < (bt == 2 ? 3 : 1); win++)
            for (int i = 0; i < n; i++) {
                double xi = 0.0;
                for (int k = 0; k < half; k++) {
                    double v = s[18 * block + half * win + k];
                    xi += v * (n == 36 ? d->cos36[i][k] : d->cos12[i][k]);
                }
                sb36[win * n + i] = xi * d->sine_block[bt][i];
            }
        if (bt == 2) {
            memcpy(tmp, sb36, sizeof tmp);
            for (int i = 0; i < 6; i++) sb36[i] = 0;
            for (int i = 6; i < 12; i++) sb36[i] = tmp[i - 6];
            for (int i = 12; i < 18; i++) sb36[i] = tmp[i - 6] + tmp[12 + i - 12];
            for (int i = 18; i < 24; i++) sb36[i] = tmp[12 + i - 12] + tmp[24 + i - 18];
            for (int i = 24; i < 30; i++) sb36[i] = tmp[24 + i - 18];
            for (int i = 30; i < 36; i++) sb36[i] = 0;
        }
        for (int i = 0; i < 18; i++) {
            s[sample + i] = sb36[i] + d->prev_samples[ch][block][i];
            d->prev_samples[ch][block][i] = sb36[18 + i];
        }
        sample += 18;
    }
}

/* Frame.py:624-631 */
static void dec_freq_inversion(dec_t *d, int gr, int ch)
{
    for (int sb = 1; sb < 18; sb += 2)
        for (int i = 1; i < 32; i += 2) d->samples[gr][ch][i * 18 + sb] *= -1;
}

/* Frame.py:65-103 */
static void dec_synth(dec_t *d, int gr, int ch)
{
    double s[32], u[512], w[512], pcm[576];
    double *fifo = d->fifo[ch];
    for (int sb = 0; sb < 18; sb++) {
        for (int i = 0; i < 32; i++) s[i] = d->samples[gr][ch][i * 18 + sb];
        for (int i = 1023; i > 63; i--) fifo[i] = fifo[i - 64];
        for (int i = 0; i < 64; i++) {
            fifo[i] = 0.0;
            for (int j = 0; j < 32; j++) fifo[i] += s[j] * d->synth_n[i][j];
        }
        for (int i = 0; i < 8; i++)
            for (int j = 0; j < 32; j++) {
                u[i * 64 + j] = fifo[i * 128 + j];
                u[i * 64 + j + 32] = fifo[i * 128 + j + 96];
            }
        for (int i = 0; i < 512; i++) w[i] = u[i] * ORA_SYNTH_WINDOW[i];
        for (int i = 0; i < 32; i++) {
            double sum = 0;
            for (int j = 0; j < 16; j++) sum += w[j * 32 + i];
            pcm[32 * sb + i] = sum;
        }
    }
    memcpy(d->samples[gr][ch], pcm, sizeof pcm);
}

static void dec_init(dec_t *d)
{
    memset(d, 0, sizeof *d);
    const double PI = 3.141592653589793;
    for (int i = 0; i < 64; i++) /* Frame.py:16-29 */
        for (int j = 0; j < 32; j++) d->synth_n[i][j] = cos((16.0 + i) * (2.0 * j + 1.0) * (PI / 64.0));
    for (int i = 0; i < 36; i++) d->sine_block[0][i] = sin(PI / 36.0 * (i + 0.5)); /* Frame.py:32-62 */
    for (int i = 0; i < 18; i++) d->sine_block[1][i] = sin(PI / 36.0 * (i + 0.5));
    for (int i = 18; i < 24; i++) d->sine_block[1][i] = 1.0;
    for (int i = 24; i < 30; i++) d->sine_block[1][i] = sin(PI / 12.0 * (i - 18.0 + 0.5));
    for (int i = 30; i < 36; i++) d->sine_block[1][i] = 1.0;
    for (int i = 0; i < 12; i++) d->sine_block[2][i] = sin(PI / 12.0 * (i + 0.5));
    for (int i = 0; i < 6; i++) d->sine_block[3][i] = 0.0;
    for (int i = 6; i < 12; i++) d->sine_block[3][i] = sin(PI / 12.0 * (i - 6.0 + 0.5));
    for (int i = 12; i < 18; i++) d->sine_block[3][i] = 1.0;
    for (int i = 18; i < 36; i++) d->sine_block[3][i] = sin(PI / 36.0 * (i + 0.5));
    /* Frame.py:128: math.cos(math.pi / (2 * n) * (2 * i + 1 + half_n) * (2 * k + 1)), same evaluation order */
    for (int i = 0; i < 36; i++)
        for (int k = 0; k < 18; k++) d->cos36[i][k] = cos(PI / (2 * 36) * (2 * i + 1 + 18) * (2 * k + 1));
    for (int i = 0; i < 12; i++)
        for (int k = 0; k < 6; k++) d->cos12[i][k] = cos(PI / (2 * 12) * (2 * i + 1 + 6) * (2 * k + 1));
}

/* MP3_Parser.py:21-85 + Frame.py:244-286.  `offset` = first audio byte (after ID3). */
ORA_API ora_dec_result *ora_decode(const uint8_t *file, int64_t flen, int64_t offset, int want_taps)
{
    ora_dec_result *r = (ora_dec_result *)calloc(1, sizeof *r);
    dec_t *d = (dec_t *)malloc(sizeof *d);
    dec_init(d);
    int valid = 0;
    if (flen - offset >= 2 && file[offset] == 0xFF && file[offset + 1] >= 0xE0) {
        valid = 1;
        int st = dec_header(d, file + offset);
        if (st < 0) { r->status = st; valid = 0; }
        else dec_set_frame_size(d);
    } else r->status = -1;
    int64_t cap = 0;
    vec_t bits = {0};
    while (valid && flen > offset + 4) {
        const uint8_t *buf = file + offset;
        int64_t blen = flen - offset;
        if (buf[0] == 0xFF && buf[1] >= 0xE0) {
            int st = dec_header(d, buf);
            if (st < 0) { r->status = st; break; }
        } else valid = 0;
        if (r->n_pcm_rows / 1152 + 1 > cap) {
            cap = cap ? cap * 2 : 64;
            r->pcm = (double *)realloc(r->pcm, sizeof(double) * cap * 1152 * 2);
            r->tables = (uint8_t *)realloc(r->tables, cap * 12);
            r->frame_off = (int64_t *)realloc(r->frame_off, sizeof(int64_t) * cap);
            r->frame_mdb = (int32_t *)realloc(r->frame_mdb, sizeof(int32_t) * cap);
            if (want_taps) {
                r->spectra = (int32_t *)realloc(r->spectra, sizeof(int32_t) * cap * 4 * 576);
                r->side = (int32_t *)realloc(r->side, sizeof(int32_t) * cap * 4 * ORA_SIDE_FIELDS);
                r->xr = (double *)realloc(r->xr, sizeof(double) * cap * 4 * 576);
            }
        }
        if (valid) {
            int64_t f = r->n_frames;
            dec_set_frame_size(d);
            memset(d->pcm, 0, sizeof d->pcm);
            int si = d->crc == 0 ? 6 : 4;
            dec_side_info(d, buf + (si < blen ? si : blen), blen - si > 0 ? blen - si : 0);
            /* Frame.py:676-685 table list, (ch, gr, region) order */
            int t = 0;
            memset(r->tables + 12 * f, 0, 12);
            for (int ch = 0; ch < d->channels; ch++)
                for (int gr = 0; gr < 2; gr++)
                    for (int rg = 0; rg < 3; rg++) r->tables[12 * f + t++] = (uint8_t)d->table_select[gr][ch][rg];
            r->frame_off[f] = offset;
            r->frame_mdb[f] = d->main_data_begin;
            dec_set_main_data(d, file, flen, offset);
            int64_t bit = 0;
            for (int gr = 0; gr < 2; gr++)
                for (int ch = 0; ch < d->channels; ch++) {
                    int64_t max_bit = bit + d->part2_3_length[gr][ch];
                    int64_t b0 = bit;
                    bit = dec_unpack_scale_fac(d, gr, ch, bit);
                    dec_unpack_samples(d, gr, ch, bit, max_bit);
                    if (want_taps) {
                        int32_t *sp = r->spectra + ((f * 2 + gr) * 2 + ch) * 576;
                        for (int i = 0; i < 576; i++) sp[i] = (int32_t)d->samples[gr][ch][i];
                        int32_t *sd = r->side + ((f * 2 + gr) * 2 + ch) * ORA_SIDE_FIELDS;
                        sd[0] = d->part2_3_length[gr][ch]; sd[1] = d->big_value[gr][ch];
                        sd[2] = d->global_gain[gr][ch]; sd[3] = d->scale_fac_compress[gr][ch];
                        sd[4] = d->window_switching[gr][ch]; sd[5] = d->block_type[gr][ch];
                        sd[6] = d->mixed_block_flag[gr][ch];
                        sd[7] = d->table_select[gr][ch][0]; sd[8] = d->table_select[gr][ch][1];
                        sd[9] = d->table_select[gr][ch][2];
                        sd[10] = d->sub_block_gain[gr][ch][0]; sd[11] = d->sub_block_gain[gr][ch][1];
                        sd[12] = d->sub_block_gain[gr][ch][2];
                        sd[13] = d->region0_count[gr][ch]; sd[14] = d->region1_count[gr][ch];
                        sd[15] = d->pre_flag[gr][ch]; sd[16] = d->scale_fac_scale[gr][ch];
                        sd[17] = d->count1table_select[gr][ch];
                        sd[18] = (int32_t)b0; sd[19] = (int32_t)(bit - b0);
                    }
                    bit = max_bit;
                }
            /* when mono, the unused channel taps stay zero */
            if (want_taps && d->channels == 1)
                for (int gr = 0; gr < 2; gr++) {
                    memset(r->spectra + ((f * 2 + gr) * 2 + 1) * 576, 0, sizeof(int32_t) * 576);
                    memset(r->side + ((f * 2 + gr) * 2 + 1) * ORA_SIDE_FIELDS, 0, sizeof(int32_t) * ORA_SIDE_FIELDS);
                }
            for (int gr = 0; gr < 2; gr++) {
                for (int ch = 0; ch < d->channels; ch++) dec_requantize(d, gr, ch);
                if (d->channel_mode == 1 && d->mode_ext0) dec_ms_stereo(d, gr);
                for (int ch = 0; ch < d->channels; ch++) {
                    if (d->block_type[gr][ch] == 2 || d->mixed_block_flag[gr][ch]) dec_reorder(d, gr, ch);
                    else dec_alias(d, gr, ch);
                    if (want_taps) memcpy(r->xr + ((f * 2 + gr) * 2 + ch) * 576, d->samples[gr][ch], sizeof(double) * 576);
                    dec_imdct(d, gr, ch);
                    dec_freq_inversion(d, gr, ch);
                    dec_synth(d, gr, ch);
                }
            }
            for (int gr = 0; gr < 2; gr++) /* Frame.py:633-640 */
                for (int s = 0; s < 576; s++)
                    for (int ch = 0; ch < d->channels; ch++) d->pcm[s + 576 * gr][ch] = d->samples[gr][ch][s];
            /* decoder/util.py:67-81 */
            for (int k = 0; k < 12; k++) {
                int x = r->tables[12 * f + k];
                if (k >= 6 * d->channels) break;
                if (x == 0) continue;
                uint8_t c = ((ORA_H0_MASK >> x) & 1u) ? '0' : '1';
                vec_push(&bits, &c, 1);
            }
            r->n_frames += 1;
            offset += d->frame_size;
        }
        /* MP3_Parser.py:79: the current frame's pcm is appended even when the sync check just failed */
        for (int s = 0; s < 1152; s++)
            for (int ch = 0; ch < d->channels; ch++)
                r->pcm[(r->n_pcm_rows + s) * d->channels + ch] = d->pcm[s][ch];
        r->n_pcm_rows += 1152;
    }
    uint8_t z = 0;
    r->n_bits = bits.n;
    vec_push(&bits, &z, 1);
    r->bits = (char *)bits.p;
    r->channels = d->channels;
    r->sampling_rate = d->sampling_rate;
    r->bit_rate = d->bit_rate;
    free(d->main_data.p);
    free(d);
    return r;
}

ORA_API void ora_dec_free(ora_dec_result *r)
{
    if (!r) return;
    free(r->pcm); free(r->spectra); free(r->tables); free(r->bits); free(r->side);
    free(r->frame_off); free(r->frame_mdb); free(r->xr);
    free(r);
}

/* MP3_Parser.py:91 `(pcm * 32767).astype(np.int16)`: C cast of the double to int32, then low 16 bits (A.D8) */
ORA_API void ora_pcm_to_int16(const double *pcm, int64_t n, int16_t *out)
{
    for (int64_t i = 0; i < n; i++) {
        double v = pcm[i] * 32767;
        int32_t t;
        if (v >= 2147483648.0 || v < -2147483648.0 || v != v) t = (int32_t)0x80000000; /* x86 cvttsd2si */
        else t = (int32_t)v;
        out[i] = (int16_t)(uint16_t)(t & 0xFFFF);
    }
}

/* ================================================================================================
 * ENCODER (reference: encoder/MP3_Encoder.py, a port of Shine)
 * ============================================================================================== */

typedef struct {
    int table_select[3];
    int part2_3_length, big_values, count1, global_gain, scale_fac_compress, region0_count, region1_count;
    int preflag, scale_fac_scale, count1table_select, part2_length, address1, address2, address3;
    int quantizerStepSize;
} grinfo_t;

typedef struct {
    /* config */
    int nch, samplerate, bitrate, sr_index, bitrate_index;
    const int16_t *buffer;
    int64_t buffer_len, buffer_pos[2];
    /* mpeg */
    int padding, bits_per_frame, whole_slots_per_frame, mean_bits, side_info_len;
    double frac_slots_per_frame, slot_lag;
    /* state */
    int32_t off[2], x[2][512];
    int32_t l3_sb_sample[2][3][18][32];
    int32_t mdct_freq[2][2][576];
    int32_t l3_enc[2][2][576];
    int32_t xrsq[576], xrabs[576], xrmax;
    const int32_t *xr;
    int32_t en_tot[2], en[2][21], xm[2][21], xrmaxl[2];
    int scfsi[2][4];
    grinfo_t gi[2][2]; /* [gr][ch] */
    double resv_size;
    int resv_max;
    /* bitstream (MP3_Encoder.py:1362-1392) */
    uint32_t cache;
    int cache_bits;
    vec_t out;
    /* stego */
    const char *hide_str;
    int64_t hide_len, hide_off;
    int32_t int2idx[10000];
} enc_t;

typedef struct ora_enc_result {
    uint8_t *data;
    int64_t n_bytes, n_frames, hide_str_offset;
    int32_t *mdct; /* [n_frames][ch][gr][576] */
    int32_t *ix;   /* [n_frames][ch][gr][576] signed, as written */
    int32_t *info; /* [n_frames][gr][ch][ORA_ENC_FIELDS] */
    int32_t *scfsi; /* [n_frames][ch][4] */
    int status;     /* 0; -1 mono; -2 bad rate; -3 step table overrun (A.E13): no bytes, n_frames = that frame */
} ora_enc_result;
#define ORA_ENC_FIELDS 16

static inline int32_t e_mul(int32_t a, int32_t b) { return (int32_t)(((int64_t)a * (int64_t)b) >> 32); }
static inline int32_t e_mulr(int32_t a, int32_t b) { return (int32_t)((((int64_t)a * (int64_t)b) + 2147483648LL) >> 32); }
static inline int32_t e_mulsr(int32_t a, int32_t b) { return (int32_t)((((int64_t)a * (int64_t)b) + 1073741824LL) >> 31); }
static inline int32_t wadd(int32_t a, int32_t b) { return (int32_t)((uint32_t)a + (uint32_t)b); }

/* MP3_Encoder.py:1362-1392 */
static void put_bits(enc_t *e, uint32_t val, int N)
{
    if (N == 0) return; /* every zero-width call in the reference carries val == 0: a no-op there too */
    if (e->cache_bits > N) {
        e->cache_bits -= N;
        e->cache |= (uint32_t)(val << e->cache_bits);
    } else {
        N -= e->cache_bits;
        e->cache |= (N < 32 ? (val >> N) : 0);
        uint8_t b[4] = {(uint8_t)(e->cache >> 24), (uint8_t)(e->cache >> 16), (uint8_t)(e->cache >> 8), (uint8_t)e->cache};
        vec_push(&e->out, b, 4);
        e->cache_bits = 32 - N;
        if (N != 0) e->cache = (uint32_t)(val << e->cache_bits);
        else e->cache = 0;
    }
}
static int64_t bits_count(enc_t *e) { return e->out.n * 8 + 32 - e->cache_bits; }

/* MP3_Encoder.py:751-758 */
static void replace_samples(enc_t *e, int ch)
{
    for (int i = 31; i >= 0; i--) {
        int64_t p = e->buffer_pos[ch];
        int32_t v = p < e->buffer_len ? e->buffer[p] : 0; /* reference raises IndexError past the end */
        e->x[ch][i + e->off[ch]] = (int32_t)((uint32_t)v << 16);
        e->buffer_pos[ch] += 2;
    }
}

/* MP3_Encoder.py:322-370 */
static void window_filter_sub_band(enc_t *e, int32_t *s, int ch)
{
    int32_t tmp[64];
    for (int i = 63; i >= 0; i--) {
        int32_t v = 0;
        for (int k = 0; k < 8; k++)
            v = wadd(v, e_mul(e->x[ch][(e->off[ch] + i + (k << 6)) & 511], ORA_ENWINDOW[i + (k << 6)]));
        tmp[i] = v;
    }
    e->off[ch] = (e->off[ch] + 480) & 511;
    for (int i = 31; i >= 0; i--) {
        int32_t v = 0;
        for (int j = 63; j >= 0; j--) v = wadd(v, e_mul(ORA_ENC_FL[i * 64 + j], tmp[j]));
        s[i] = v;
    }
}

/* MP3_Encoder.py:652-749 */
static void mdct_sub(enc_t *e)
{
    int32_t in[36];
    for (int ch = e->nch - 1; ch >= 0; ch--) {
        for (int gr = 0; gr < 2; gr++) {
            for (int k = 0; k < 18; k += 2) {
                replace_samples(e, ch);
                window_filter_sub_band(e, e->l3_sb_sample[ch][gr + 1][k], ch);
                replace_samples(e, ch);
                window_filter_sub_band(e, e->l3_sb_sample[ch][gr + 1][k + 1], ch);
                for (int band = 1; band < 32; band += 2)
                    e->l3_sb_sample[ch][gr + 1][k + 1][band] = (int32_t)(0u - (uint32_t)e->l3_sb_sample[ch][gr + 1][k + 1][band]);
            }
            int32_t(*mf)[18] = (int32_t(*)[18])e->mdct_freq[ch][gr];
            for (int band = 0; band < 32; band++) {
                for (int k = 17; k >= 0; k--) {
                    in[k] = e->l3_sb_sample[ch][gr][k][band];
                    in[k + 18] = e->l3_sb_sample[ch][gr + 1][k][band];
                }
                for (int k = 17; k >= 0; k--) {
                    int32_t vm = 0;
                    for (int j = 35; j >= 0; j--) vm = wadd(vm, e_mul(in[j], ORA_ENC_COSL[k * 36 + j]));
                    mf[band][k] = vm;
                }
                if (band != 0)
                    for (int k = 0; k < 8; k++) { /* util.cmuls, util.py:145-155 */
                        int64_t are = mf[band][k], aim = mf[band - 1][17 - k];
                        int64_t bre = ORA_ENC_CS[k], bim = ORA_ENC_CA[k];
                        int32_t tre = (int32_t)((are * bre - aim * bim) >> 31);
                        int32_t dim = (int32_t)((are * bim + aim * bre) >> 31);
                        mf[band][k] = tre;
                        mf[band - 1][17 - k] = dim;
                    }
            }
        }
        memcpy(e->l3_sb_sample[ch][0], e->l3_sb_sample[ch][2], sizeof e->l3_sb_sample[ch][0]);
    }
}

/* MP3_Encoder.py:374-415 */
static int quantize(enc_t *e, int32_t *ix, int step_size)
{
    int ix_max = 0;
    int32_t scalei = ORA_ENC_STEPTABI[step_size + 127];
    if (e_mulr(e->xrmax, scalei) > 165140) return 16384;
    for (int i = 0; i < 576; i++) {
        int64_t ab = e->xr[i] < 0 ? -(int64_t)e->xr[i] : (int64_t)e->xr[i];
        int32_t ln = (int32_t)((ab * (int64_t)scalei + 2147483648LL) >> 32);
        if (ln < 10000) ix[i] = e->int2idx[ln];
        else {
            double scale = ORA_ENC_STEPTAB[step_size + 127];
            double dbl = (double)e->xrabs[i] * scale * 4.656612875e-10;
            ix[i] = (int32_t)sqrt(sqrt(dbl) * dbl);
        }
        if (ix_max < ix[i]) ix_max = ix[i];
    }
    return ix_max;
}

/* MP3_Encoder.py:266-291 */
static void calc_run_len(const int32_t *ix, grinfo_t *ci)
{
    int i = 576;
    while (i > 1) {
        if (ix[i - 1] == 0 && ix[i - 2] == 0) i -= 2;
        else break;
    }
    ci->count1 = 0;
    while (i > 3) {
        if (ix[i - 1] <= 1 && ix[i - 2] <= 1 && ix[i - 3] <= 1 && ix[i - 4] <= 1) { ci->count1 += 1; i -= 4; }
        else break;
    }
    ci->big_values = i >> 1;
}

/* MP3_Encoder.py:171-211 */
static int count1_bit_count(const int32_t *ix, grinfo_t *ci)
{
    int i = ci->big_values << 1, sum0 = 0, sum1 = 0;
    for (int k = 0; k < ci->count1; k++) {
        int v = ix[i], w = ix[i + 1], x = ix[i + 2], y = ix[i + 3];
        int p = v + (w << 1) + (x << 2) + (y << 3);
        int sb = (v != 0) + (w != 0) + (x != 0) + (y != 0);
        sum0 += sb; sum1 += sb;
        sum0 += ORA_ENC_HLEN[ORA_ENC_OFF[32] + p];
        sum1 += ORA_ENC_HLEN[ORA_ENC_OFF[33] + p];
        i += 4;
    }
    if (sum0 < sum1) { ci->count1table_select = 0; return sum0; }
    ci->count1table_select = 1;
    return sum1;
}

/* MP3_Encoder.py:214-263 */
static int count_bit(const int32_t *ix, int start, int end, int table)
{
    if (table == 0) return 0;
    int sum = 0, ylen = ORA_ENC_YLEN[table], lin = ORA_ENC_LINBITS[table];
    const uint8_t *hl = ORA_ENC_HLEN + ORA_ENC_OFF[table];
    if (table > 15) {
        for (int i = start; i < end; i += 2) {
            int x = ix[i], y = ix[i + 1];
            if (x > 14) { x = 15; sum += lin; }
            if (y > 14) { y = 15; sum += lin; }
            sum += hl[x * ylen + y];
            if (x) sum += 1;
            if (y) sum += 1;
        }
    } else {
        for (int i = start; i < end; i += 2) {
            int x = ix[i], y = ix[i + 1];
            sum += hl[x * ylen + y];
            if (x != 0) sum += 1;
            if (y != 0) sum += 1;
        }
    }
    return sum;
}

/* MP3_Encoder.py:998-1036 */
static void subdivide(enc_t *e, grinfo_t *ci)
{
    if (ci->big_values == 0) { ci->region0_count = 0; ci->region1_count = 0; return; }
    const int *sf = ORA_SFB_LONG + 23 * e->sr_index;
    int bvr = 2 * ci->big_values;
    int anz = 0;
    while (sf[anz] < bvr) anz++;
    int tc = ORA_SUBDV[2 * anz];
    while (tc > 0) { if (sf[tc + 1] <= bvr) break; tc--; }
    ci->region0_count = tc;
    ci->address1 = sf[tc + 1];
    sf += tc + 1;
    tc = ORA_SUBDV[2 * anz + 1];
    while (tc > 0) { if (sf[tc + 1] <= bvr) break; tc--; }
    ci->region1_count = tc;
    ci->address2 = sf[tc + 1];
    ci->address3 = bvr;
}

/* MP3_Encoder.py:1170-1264 */
static int new_choose_table(enc_t *e, const int32_t *ix, int begin, int end, int64_t idx)
{
    int ix_max = 0;
    for (int i = begin; i < end; i++) if (ix[i] > ix_max) ix_max = ix[i];
    if (ix_max == 0) return 0;
    int choice0 = 0, choice1 = 0, sum0, sum1;
    if (ix_max < 15) {
        for (int i = 13; i >= 0; i--) if (ORA_ENC_XLEN[i] > ix_max) { choice0 = i; break; }
        sum0 = count_bit(ix, begin, end, choice0);
        switch (choice0) { /* only the 13 arm is reachable (A.E4); the others are restated for completeness */
        case 2: sum1 = count_bit(ix, begin, end, 3); if (sum1 <= sum0) choice0 = 3; break;
        case 5: sum1 = count_bit(ix, begin, end, 6); if (sum1 <= sum0) choice0 = 6; break;
        case 7:
            sum1 = count_bit(ix, begin, end, 8); if (sum1 <= sum0) choice0 = 8;
            sum1 = count_bit(ix, begin, end, 9); if (sum1 <= sum0) choice0 = 9; break;
        case 10:
            sum1 = count_bit(ix, begin, end, 11); if (sum1 <= sum0) choice0 = 11;
            sum1 = count_bit(ix, begin, end, 12); if (sum1 <= sum0) choice0 = 12; break;
        case 13: sum1 = count_bit(ix, begin, end, 15); if (sum1 <= sum0) choice0 = 15; break;
        default: break;
        }
    } else {
        ix_max -= 15;
        for (int i = 15; i < 24; i++) if (ORA_ENC_LINMAX[i] >= ix_max) { choice0 = i; break; }
        for (int i = 24; i < 32; i++) if (ORA_ENC_LINMAX[i] >= ix_max) { choice1 = i; break; }
        sum0 = count_bit(ix, begin, end, choice0);
        sum1 = count_bit(ix, begin, end, choice1);
        if (sum1 < sum0) choice0 = choice1;
    }
    if (e->hide_len > 0) {
        if (idx < e->hide_len) return ORA_PAIR[choice0 * 2 + (e->hide_str[idx] == '1' ? 1 : 0)];
        return choice0;
    }
    return choice0;
}

/* MP3_Encoder.py:1147-1168 */
static void big_v_tab_select(enc_t *e, const int32_t *ix, grinfo_t *ci)
{
    int64_t idx = e->hide_off;
    ci->table_select[0] = ci->address1 <= 0 ? 0 : new_choose_table(e, ix, 0, ci->address1, e->hide_off);
    if (ci->table_select[0] > 0) idx += 1;
    ci->table_select[1] = ci->address2 <= ci->address1 ? 0 : new_choose_table(e, ix, ci->address1, ci->address2, idx);
    if (ci->table_select[1] > 0) idx += 1;
    ci->table_select[2] = (ci->big_values << 1) <= ci->address2 ? 0 : new_choose_table(e, ix, ci->address2, ci->big_values << 1, idx);
}

/* MP3_Encoder.py:294-318 */
static int big_v_bit_count(const int32_t *ix, const grinfo_t *ci)
{
    int bits = 0;
    if (ci->table_select[0]) bits += count_bit(ix, 0, ci->address1, ci->table_select[0]);
    if (ci->table_select[1]) bits += count_bit(ix, ci->address1, ci->address2, ci->table_select[1]);
    if (ci->table_select[2]) bits += count_bit(ix, ci->address2, ci->address3, ci->table_select[2]);
    return bits;
}

static int probe_bits(enc_t *e, int32_t *ix, grinfo_t *ci)
{
    calc_run_len(ix, ci);
    int bits = count1_bit_count(ix, ci);
    subdivide(e, ci);
    big_v_tab_select(e, ix, ci);
    bits += big_v_bit_count(ix, ci);
    return bits;
}

/* MP3_Encoder.py:958-996 */
static int bin_search_step_size(enc_t *e, int desired, int32_t *ix, grinfo_t *ci)
{
    int next = -120, count = 120;
    do {
        int half = count / 2, bit;
        if (quantize(e, ix, next + half) > 8192) bit = 100000;
        else bit = probe_bits(e, ix, ci);
        if (bit < desired) count = half;
        else { next += half; count -= half; }
    } while (count > 1);
    return next;
}

/* MP3_Encoder.py:1064-1095 */
/* Returns -1 instead of a bit count when the search would quantise at a step above 0: quantize() would read steptabi[128],
 * past the end of the 128-entry table, and the reference has no defined output there (SURVEY A.E13). */
static int inner_loop(enc_t *e, int32_t *ix, int max_bits, grinfo_t *ci)
{
    int bits;
    if (max_bits < 0) ci->quantizerStepSize -= 1;
    do {
        while (ci->quantizerStepSize < 0 && quantize(e, ix, ci->quantizerStepSize + 1) > 8192) ci->quantizerStepSize += 1;
        if (ci->quantizerStepSize >= 0) return -1;
        ci->quantizerStepSize += 1;
        bits = probe_bits(e, ix, ci);
    } while (bits > max_bits);
    return bits;
}

/* MP3_Encoder.py:817-892 */
static void calc_scfsi(enc_t *e, int ch, int gr)
{
    static const int band[5] = {0, 6, 11, 16, 21};
    const int *sf = ORA_SFB_LONG + 23 * e->sr_index;
    int condition = 0;
    e->xrmaxl[gr] = e->xrmax;
    int32_t temp = 0;
    for (int i = 575; i >= 0; i--) temp = wadd(temp, e->xrsq[i] >> 10);
    if (temp) e->en_tot[gr] = (int32_t)(log((double)temp * 4.768371584e-7) / 0.69314718);
    else e->en_tot[gr] = 0;
    for (int sfb = 20; sfb >= 0; sfb--) {
        temp = 0;
        for (int i = sf[sfb]; i < sf[sfb + 1]; i++) temp = wadd(temp, e->xrsq[i] >> 10);
        if (temp) e->en[gr][sfb] = (int32_t)(log((double)temp * 4.768371584e-7) / 0.69314718);
        else e->en[gr][sfb] = 0;
        e->xm[gr][sfb] = 0;
    }
    if (gr == 1) {
        for (int g2 = 1; g2 >= 0; g2--) { if (e->xrmaxl[g2]) condition++; condition++; }
        if (abs(e->en_tot[0] - e->en_tot[1]) < 10) condition++;
        int tp = 0;
        for (int sfb = 20; sfb >= 0; sfb--) tp += abs(e->en[0][sfb] - e->en[1][sfb]);
        if (tp < 100) condition++;
        if (condition == 6) {
            for (int b = 0; b < 4; b++) {
                int sum0 = 0, sum1 = 0;
                for (int sfb = band[b]; sfb < band[b + 1]; sfb++) {
                    sum0 += abs(e->en[0][sfb] - e->en[1][sfb]);
                    sum1 += abs(e->xm[0][sfb] - e->xm[1][sfb]);
                }
                e->scfsi[ch][b] = (sum0 < 10 && sum1 < 10) ? 1 : 0;
            }
        } else
            for (int b = 0; b < 4; b++) e->scfsi[ch][b] = 0;
    }
}

/* MP3_Encoder.py:1097-1145 */
static void resv_frame_end(enc_t *e)
{
    if (e->nch == 2 && (e->mean_bits & 1)) e->resv_size += 1;
    double over = e->resv_size - e->resv_max;
    if (over < 0) over = 0;
    e->resv_size -= over;
    double stuffing = over;
    over = fmod(e->resv_size, 8.0);
    if (over < 0) over += 8.0; /* Python float % */
    if (over != 0) { stuffing += over; e->resv_size -= over; }
    if (stuffing != 0) {
        grinfo_t *gi = &e->gi[0][0];
        if (gi->part2_3_length + stuffing < 4095) gi->part2_3_length += (int)stuffing;
        else {
            for (int gr = 0; gr < 2; gr++)
                for (int ch = 0; ch < e->nch; ch++) {
                    gi = &e->gi[gr][ch];
                    if (stuffing == 0) break;
                    double extra = 4095 - gi->part2_3_length;
                    double t = extra < stuffing ? extra : stuffing;
                    gi->part2_3_length += (int)t;
                    stuffing -= t;
                }
        }
    }
}

/* MP3_Encoder.py:760-815 */
/* Returns 0, or -1 when a granule's step search runs past the step table (inner_loop). */
static int iteration_loop(enc_t *e)
{
    for (int ch = 0; ch < e->nch; ch++)
        for (int gr = 0; gr < 2; gr++) {
            int32_t *ix = e->l3_enc[ch][gr];
            e->xr = e->mdct_freq[ch][gr];
            e->xrmax = 0;
            for (int i = 575; i >= 0; i--) {
                e->xrsq[i] = e_mulsr(e->xr[i], e->xr[i]);
                int64_t ab = e->xr[i] < 0 ? -(int64_t)e->xr[i] : (int64_t)e->xr[i];
                e->xrabs[i] = (int32_t)ab;
                if (e->xrabs[i] > e->xrmax) e->xrmax = e->xrabs[i];
            }
            grinfo_t *ci = &e->gi[gr][ch];
            calc_scfsi(e, ch, gr);
            int mean = e->mean_bits / e->nch; /* floor div of non-negative ints */
            int max_bits = mean > 4095 ? 4095 : mean;
            ci->part2_3_length = 0; ci->big_values = 0; ci->count1 = 0; ci->scale_fac_compress = 0;
            ci->table_select[0] = ci->table_select[1] = ci->table_select[2] = 0;
            ci->region0_count = 0; ci->region1_count = 0; ci->part2_length = 0; ci->preflag = 0;
            ci->scale_fac_scale = 0; ci->count1table_select = 0;
            if (e->xrmax) {
                /* __outer_loop, MP3_Encoder.py:933-956 (part2_length is always 0: scale_fac_compress == 0) */
                ci->quantizerStepSize = bin_search_step_size(e, max_bits, ix, ci);
                ci->part2_length = 0;
                int bits = inner_loop(e, ix, max_bits - ci->part2_length, ci);
                if (bits < 0) return -1;
                ci->part2_3_length = ci->part2_length + bits;
                e->hide_off += (ci->table_select[0] > 0) + (ci->table_select[1] > 0) + (ci->table_select[2] > 0);
            }
            e->resv_size += ((double)e->mean_bits / e->nch) - ci->part2_3_length;
            ci->global_gain = ci->quantizerStepSize + 210;
        }
    resv_frame_end(e);
    return 0;
}

/* MP3_Encoder.py:1448-1513 */
static void huffman_code(enc_t *e, int table, int x, int y)
{
    int sx = 0, sy = 0;
    if (!(x > 0)) { x = -x; sx = 1; } /* util.abs_and_sign: zero gets sign 1, never written */
    if (!(y > 0)) { y = -y; sy = 1; }
    int ylen = ORA_ENC_YLEN[table];
    const uint32_t *code_t = ORA_ENC_CODE + ORA_ENC_OFF[table];
    const uint8_t *hl = ORA_ENC_HLEN + ORA_ENC_OFF[table];
    if (table > 15) {
        uint32_t ext = 0;
        int xbits = 0, lbx = 0, lby = 0, lin = ORA_ENC_LINBITS[table];
        if (x > 14) { lbx = x - 15; x = 15; }
        if (y > 14) { lby = y - 15; y = 15; }
        int idx = x * ylen + y;
        uint32_t code = code_t[idx];
        int cbits = hl[idx];
        if (x > 14) { ext |= (uint32_t)lbx; xbits += lin; }
        if (x != 0) { ext <<= 1; ext |= (uint32_t)sx; xbits += 1; }
        if (y > 14) { ext <<= lin; ext |= (uint32_t)lby; xbits += lin; }
        if (y != 0) { ext <<= 1; ext |= (uint32_t)sy; xbits += 1; }
        put_bits(e, code, cbits);
        put_bits(e, ext, xbits);
    } else {
        int idx = x * ylen + y;
        uint32_t code = code_t[idx];
        int cbits = hl[idx];
        if (x != 0) { code = (code << 1) | (uint32_t)sx; cbits += 1; }
        if (y != 0) { code = (code << 1) | (uint32_t)sy; cbits += 1; }
        put_bits(e, code, cbits);
    }
}

/* MP3_Encoder.py:1394-1446, :1515-1547 */
static void huffman_code_bits(enc_t *e, int gr, int ch)
{
    const int *sf = ORA_SFB_LONG + 23 * e->sr_index;
    grinfo_t *gi = &e->gi[gr][ch];
    int64_t bits0 = bits_count(e);
    int big_values = gi->big_values << 1;
    int sfi = gi->region0_count + 1;
    int r1 = sf[sfi];
    sfi += gi->region1_count + 1;
    int r2 = sf[sfi];
    const int32_t *ix = e->l3_enc[ch][gr];
    for (int i = 0; i < big_values; i += 2) {
        int idx = (i >= r1) + (i >= r2);
        int t = gi->table_select[idx];
        if (t != 0) huffman_code(e, t, ix[i], ix[i + 1]);
    }
    int ht = gi->count1table_select + 32;
    int c1end = big_values + (gi->count1 << 2);
    for (int i = big_values; i < c1end; i += 4) {
        int v = ix[i], w = ix[i + 1], x = ix[i + 2], y = ix[i + 3];
        int sv = 0, sw = 0, sx = 0, sy = 0;
        if (!(v > 0)) { v = -v; sv = 1; }
        if (!(w > 0)) { w = -w; sw = 1; }
        if (!(x > 0)) { x = -x; sx = 1; }
        if (!(y > 0)) { y = -y; sy = 1; }
        int p = v + (w << 1) + (x << 2) + (y << 3);
        put_bits(e, ORA_ENC_CODE[ORA_ENC_OFF[ht] + p], ORA_ENC_HLEN[ORA_ENC_OFF[ht] + p]);
        uint32_t code = 0;
        int cbits = 0;
        if (v) { code = (uint32_t)sv; cbits = 1; }
        if (w) { code = (code << 1) | (uint32_t)sw; cbits += 1; }
        if (x) { code = (code << 1) | (uint32_t)sx; cbits += 1; }
        if (y) { code = (code << 1) | (uint32_t)sy; cbits += 1; }
        put_bits(e, code, cbits);
    }
    int64_t bits = bits_count(e) - bits0;
    bits = gi->part2_3_length - gi->part2_length - bits;
    if (bits > 0) { /* Python `if bits:`; a negative count would loop forever there */
        int64_t words = bits / 32, rem = bits % 32;
        while (words) { put_bits(e, 0xFFFFFFFFu, 32); words--; }
        if (rem) put_bits(e, (uint32_t)((1ull << rem) - 1), (int)rem);
    }
}

/* MP3_Encoder.py:1266-1360 */
static void format_bitstream(enc_t *e)
{
    for (int ch = 0; ch < e->nch; ch++)
        for (int gr = 0; gr < 2; gr++)
            for (int i = 0; i < 576; i++)
                if (e->mdct_freq[ch][gr][i] < 0 && e->l3_enc[ch][gr][i] > 0) e->l3_enc[ch][gr][i] *= -1;
    put_bits(e, 0x7ff, 11);
    put_bits(e, 3, 2);  /* version: MPEG-I */
    put_bits(e, 1, 2);  /* layer III */
    put_bits(e, 1, 1);  /* no crc */
    put_bits(e, e->bitrate_index, 4);
    put_bits(e, e->sr_index % 3, 2);
    put_bits(e, e->padding, 1);
    put_bits(e, 0, 1);
    put_bits(e, e->nch == 1 ? 3 : 0, 2);
    put_bits(e, 0, 2);
    put_bits(e, 0, 1);  /* copyright */
    put_bits(e, 1, 1);  /* original */
    put_bits(e, 0, 2);  /* emphasis */
    put_bits(e, 0, 9);
    put_bits(e, 0, e->nch == 2 ? 3 : 5);
    for (int ch = 0; ch < e->nch; ch++)
        for (int b = 0; b < 4; b++) put_bits(e, e->scfsi[ch][b], 1);
    for (int gr = 0; gr < 2; gr++)
        for (int ch = 0; ch < e->nch; ch++) {
            grinfo_t *gi = &e->gi[gr][ch];
            put_bits(e, gi->part2_3_length, 12);
            put_bits(e, gi->big_values, 9);
            put_bits(e, gi->global_gain, 8);
            put_bits(e, gi->scale_fac_compress, 4);
            put_bits(e, 0, 1);
            for (int r = 0; r < 3; r++) put_bits(e, gi->table_select[r], 5);
            put_bits(e, gi->region0_count, 4);
            put_bits(e, gi->region1_count, 3);
            put_bits(e, gi->preflag, 1);
            put_bits(e, gi->scale_fac_scale, 1);
            put_bits(e, gi->count1table_select, 1);
        }
    for (int gr = 0; gr < 2; gr++)
        for (int ch = 0; ch < e->nch; ch++) huffman_code_bits(e, gr, ch); /* scalefactors: slen == 0, nothing written */
}

/* MP3_Encoder.py:462-526 (constructor), :596-650 (encode loop).
 * pcm: interleaved int16 as WAV_Reader.py:108 holds it; n_samples: per channel (WAV_Reader.py:93). */
ORA_API ora_enc_result *ora_encode(const int16_t *pcm, int64_t pcm_len, int64_t n_samples, int nch, int samplerate,
                                   int bitrate_kbps, const char *hide_bits, int64_t hide_len, int want_taps)
{
    ora_enc_result *r = (ora_enc_result *)calloc(1, sizeof *r);
    if (nch != 2) { r->status = -1; return r; } /* mono is broken in the reference (A.E1) */
    int sri = samplerate == 44100 ? 0 : samplerate == 48000 ? 1 : samplerate == 32000 ? 2 : -1;
    static const int br[16] = {-1, 32, 40, 48, 56, 64, 80, 96, 112, 128, 160, 192, 224, 256, 320, -1};
    int bri = -1;
    for (int i = 0; i < 16; i++) if (br[i] == bitrate_kbps) { bri = i; break; }
    if (sri < 0 || bri < 0) { r->status = -2; return r; }
    enc_t *e = (enc_t *)calloc(1, sizeof *e);
    e->nch = nch; e->samplerate = samplerate; e->bitrate = bitrate_kbps; e->sr_index = sri; e->bitrate_index = bri;
    e->buffer = pcm; e->buffer_len = pcm_len; e->buffer_pos[0] = 0; e->buffer_pos[1] = 1;
    e->hide_str = hide_bits; e->hide_len = hide_len;
    e->cache = 0; e->cache_bits = 32;
    for (int i = 0; i < 10000; i++) /* MP3_Encoder.py:577-579 */
        e->int2idx[i] = (int32_t)(sqrt(sqrt((double)i) * (double)i) - 0.0946 + 0.5);
    double avg = (2.0 * 576 / (double)samplerate) * (1000 * (double)bitrate_kbps / 8.0); /* :504-505 */
    e->whole_slots_per_frame = (int)avg;
    e->frac_slots_per_frame = avg - (double)e->whole_slots_per_frame;
    e->slot_lag = -e->frac_slots_per_frame;
    e->padding = 0;
    e->side_info_len = 8 * (4 + 32);
    int64_t total = n_samples * nch, per_pass = 1152 * nch;
    int64_t count = total / per_pass + ((total % per_pass) ? 1 : 0);
    if (want_taps) {
        r->mdct = (int32_t *)calloc((size_t)(count ? count : 1) * 4 * 576, sizeof(int32_t));
        r->ix = (int32_t *)calloc((size_t)(count ? count : 1) * 4 * 576, sizeof(int32_t));
        r->info = (int32_t *)calloc((size_t)(count ? count : 1) * 4 * ORA_ENC_FIELDS, sizeof(int32_t));
        r->scfsi = (int32_t *)calloc((size_t)(count ? count : 1) * 8, sizeof(int32_t));
    }
    for (int64_t f = 0; f < count; f++) { /* __encode_buffer_internal, :623-650 */
        if (e->frac_slots_per_frame != 0) {
            e->padding = e->slot_lag <= (e->frac_slots_per_frame - 1.0) ? 1 : 0;
            e->slot_lag += e->padding - e->frac_slots_per_frame;
        }
        e->bits_per_frame = 8 * (e->whole_slots_per_frame + e->padding);
        e->mean_bits = (int)((e->bits_per_frame - e->side_info_len) / 2.0);
        mdct_sub(e);
        if (iteration_loop(e)) { /* step table overrun: no bytes, n_frames = the frame it happened in */
            r->status = -3;
            r->n_frames = f;
            free(e->out.p); free(e);
            return r;
        }
        format_bitstream(e);
        if (want_taps) {
            memcpy(r->mdct + f * 4 * 576, e->mdct_freq, sizeof e->mdct_freq);
            memcpy(r->ix + f * 4 * 576, e->l3_enc, sizeof e->l3_enc);
            for (int gr = 0; gr < 2; gr++)
                for (int ch = 0; ch < 2; ch++) {
                    int32_t *o = r->info + ((f * 2 + gr) * 2 + ch) * ORA_ENC_FIELDS;
                    grinfo_t *gi = &e->gi[gr][ch];
                    o[0] = gi->part2_3_length; o[1] = gi->big_values; o[2] = gi->count1; o[3] = gi->global_gain;
                    o[4] = gi->table_select[0]; o[5] = gi->table_select[1]; o[6] = gi->table_select[2];
                    o[7] = gi->region0_count; o[8] = gi->region1_count; o[9] = gi->count1table_select;
                    o[10] = gi->address1; o[11] = gi->address2; o[12] = gi->address3; o[13] = gi->quantizerStepSize;
                    o[14] = e->padding; o[15] = (int32_t)e->hide_off;
                }
            for (int ch = 0; ch < 2; ch++)
                for (int b = 0; b < 4; b++) r->scfsi[f * 8 + ch * 4 + b] = e->scfsi[ch][b];
        }
    }
    r->n_frames = count;
    r->data = e->out.p; /* whole 32-bit words only; the partial cache word is never flushed (A.E8) */
    r->n_bytes = e->out.n;
    r->hide_str_offset = e->hide_off;
    free(e);
    return r;
}

ORA_API void ora_enc_free(ora_enc_result *r)
{
    if (!r) return;
    free(r->data); free(r->mdct); free(r->ix); free(r->info); free(r->scfsi);
    free(r);
}

/* accessors for ctypes */
ORA_API int ora_side_fields(void) { return ORA_SIDE_FIELDS; }
ORA_API int ora_enc_fields(void) { return ORA_ENC_FIELDS; }

/* SURVEY.md A.E10 known answers for the fixed-point primitives (encoder/util.py:123-172), measured on the reference.
 * Returns 0 when all hold, else the 1-based index of the first failing one. */
ORA_API int ora_fixed_kat(void)
{
    if (e_mul(-1, 1) != -1) return 1;
    if (e_mul(2147483647, 2147483647) != 1073741823) return 2;
    if (e_mul((int32_t)(-2147483647 - 1), 2147483647) != -1073741824) return 3;
    if (e_mulr(-3, 2147483647) != -1) return 4;
    if (e_mulr(3, 2147483647) != 1) return 5;
    if (e_mulsr((int32_t)(-2147483647 - 1), (int32_t)(-2147483647 - 1)) != (int32_t)(-2147483647 - 1)) return 6;
    if (e_mulsr(46341, 46341) != 1) return 7;
    if (e_mulsr(-7, 3) != 0) return 8;
    {
        int64_t are = -5, aim = 7, bre = 2147483647, bim = -1073741824;
        int32_t tre = (int32_t)((are * bre - aim * bim) >> 31);
        int32_t dim = (int32_t)((are * bim + aim * bre) >> 31);
        if (tre != -2 || dim != 9) return 9;
    }
    if (ORA_ENC_CA[0] != -1104871221 || ORA_ENC_CA[7] != -7945635 || ORA_ENC_CS[0] != 1841452035 || ORA_ENC_CS[7] != 2147468947) return 10;
    return 0;
}
