// m3s_encode.cu -- encode half of the hot path (reference: mp3stego/encoder/MP3_Encoder.py, a port of Shine).
//
//   E1 k_enc_analysis_fold  polyphase analysis + MDCT + alias butterflies, exact 32-bit fixed point; also the per-granule
//                      spectral statistics the rate loop and scfsi need (xrmax, en_tot, en[21]).           (:322-370, :652-758, :817-861)
//                      Equal truncated products are computed once (generated straight-line code, m3s_enc_fold_gen.cuh).
//   E2 the per-granule quantisation / rate loop with table selection and the stego table swap (:760-1264), in three kernels:
//      k_enc_probe    one warp per granule-channel and NO chain between granules: the reference's step search is walked for every
//                     payload variant the granule can meet (the <= 3 payload bits at its hide_str_offset: 15 cases), the
//                     payload-independent part of a probe computed once per distinct step;
//      k_enc_resolve  one warp per clip turns offsets into variants in the reference's order (frame, ch, gr) on registers,
//                     and redoes the few granules that read the slot's stale address1/2/3 (SURVEY A.E5/A.E6);
//      k_enc_emit     one warp per granule-channel quantises at the chosen step.
//   E3 k_enc_pack      header, side info and Huffman bit packing, one warp per frame (frames are self-contained:
//                      main_data_begin = 0 and every frame is filled to its nominal size by stuffing).            (:1266-1552)
//
// All arithmetic is integer and bit-exact with the reference; the only floating point is the reference's own
// double-precision fallback in quantize (:401-407) and the padding recurrence (:504-513, :630-632) done on the host.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <functional>
#include <vector>

#include "m3s_common.cuh"

// ------------------------------------------------------------------------------------------------
// device records
// ------------------------------------------------------------------------------------------------
struct M3sEncClip {
    int64_t pcm_base;      // element offset of the clip's first sample (interleaved int16 stereo)
    int64_t frame_base;    // global frame index of the clip's first frame (in the whole batch)
    int64_t out_base;      // byte offset of the clip's MP3 in the output buffer
    int64_t out_len;       // bytes the reference's bit writer emits (whole 32-bit words only, A.E8)
    int64_t payload_base;  // first payload char
    int64_t payload_len;   // number of payload chars ('0'/'1'); 0 = plain encode
    int32_t n_frames;
    int32_t pad_base;      // first entry of the clip's frame byte offsets in the padding tables of the call (one table per rate pair)
    int32_t whole_slots;   // whole bytes of a frame at the clip's rate pair (a padded frame has one more)
    int16_t sr_idx;        // 0 = 44.1, 1 = 48, 2 = 32 kHz (the header's sampling_frequency field)
    int16_t bitrate_idx;   // the header's bitrate_index, 1..14
};

struct M3sEncState {       // E2 state carried from chunk to chunk (and between frames inside the kernel)
    int64_t hide_off;      // MP3Encoder.hide_str_offset
    int32_t a1[4], a2[4], a3[4], step[4];  // per (gr, ch) slot: address1..3 (stale when big_values == 0, A.E6), quantizerStepSize
    int32_t src[4];        // per slot: 1 + clip frame of the latest non-silent granule (0 = none yet); l3_enc keeps ITS values while silent
    int32_t overrun;       // 1 + clip frame of the first granule whose step search runs past the step table (0 = none; SURVEY A.E13)
    int32_t pad;
};

struct __align__(16) M3sEncStats {  // per granule-channel, written by E1
    int32_t xrmax;
    int8_t en_tot;
    int8_t en[21];
    int8_t pad[6];
};

struct M3sEncWork {        // E1 work item: a run of granules of one clip
    int32_t clip;
    int32_t g_first;       // first granule (2 * frame + gr) whose MDCT this CTA emits
    int32_t count;
    int32_t ch;            // channel this CTA transforms
};

#define ENC_INFO_FIELDS 16

struct EncTables {         // small read-only tables of E2/E3, built on the host once per handle
    uint32_t hl4[256];     // code lengths of books 13 | 15 << 8 | 16 << 16 | 24 << 24 at [x * 16 + y]
    uint32_t en_thresh[32];  // smallest temp with en(temp) >= j - 20  (calc_scfsi's truncated log, :836-857)
    uint8_t hlc1[2][16];   // count1 tables A / B code lengths
};

__device__ __forceinline__ int32_t mulr32(int32_t a, int32_t b)  // util.mulr (util.py:129-133)
{
    return (int32_t)(((int64_t)a * (int64_t)b + 0x80000000LL) >> 32);
}
__device__ __forceinline__ int32_t mulsr32(int32_t a, int32_t b)  // util.mulsr (util.py:135-139)
{
    return (int32_t)(((int64_t)a * (int64_t)b + 0x40000000LL) >> 31);
}

// ================================================================================================
// E1: analysis filterbank + MDCT, folded.  Every product is the reference's mul(a, b) = (a * b) >> 32 truncated on its own
// (util.py:121-127), so no algebraic folding of the SUMS is exact: done directly, that is 66,816 IMAD.HI per granule-channel on a pipe
// that issues 29 lanes/clk/SM (tools/ubench_pipes.cu).
//
// The matrixing's 32 x 64 matrix holds cosines of a 128-point grid: a column carries at most 16 distinct magnitudes (920 distinct
// (|v|, j) pairs for 2,025 non-zero entries), and  mul(-v, y) = -mul(v, y) - [(v y) mod 2^32 != 0].  So ONE truncated product per
// distinct magnitude serves every band that uses +v or -v, exactly, as long as the correction bit is known -- it is 1 whenever the
// low 26 bits of y are not all zero (tz(v) <= 6 for every entry).  tools/gen_enc_fold.py turns the tables into straight-line code
// (m3s_enc_fold_gen.cuh: products once, then signed adds into accumulators whose start values carry the corrections); where a y
// breaks the assumption (silence, mostly) the missing [(v y) mod 2^32 == 0] terms are added afterwards.  The MDCT's 18 x 36 table
// folds the same way (488 distinct of 648).  Truncated products per granule-channel: 66,816 -> 9,216 + 16,560 + 15,616 = 41,392.
//
// Sharing products needs one thread to own ALL outputs of its inputs with the coefficient pattern known at compile time, so the
// roles turn round: in the filterbank lane = time slot (the filterbank is stateless per slot: the CTA walks its run of granules as
// a STREAM of slots, one per thread and block, and cuts the 18-slot granules from a ring of subband samples as they complete), in
// the MDCT lane = band and warp = granule.  Straight-line code is big (~90 KB, far beyond the 32 KB instruction cache of an SM), so
// the instruction fetches must be shared: every warp of the CTA runs the SAME code at the same time, and the CTAs are large.
// Measured (kernel ms per 1.378 M frames; direct form 60.1): one column subset per warp, i.e. four code streams per 4-warp CTA: 94.2
// (10 of 11 stall cycles "no instruction"); all columns per thread, 4 warps x 4 CTAs per SM: 51.5 (still 3.4 of 10.4); 8 warps x
// 2 CTAs: **46.4** (0.14); 16 warps x 1 CTA: 52.6 (nothing left to cover the barriers).  Barriers inside the straight-line code
// to keep the warps aligned did not help (47.6 - 51.2).
// ================================================================================================
__constant__ int32_t c_enc_cos[18][36];   // MP3Encoder.__cos_l (:557-566), window folded in, for the MDCT's correction pass

#define M3S_FOLD_FN __device__ __forceinline__
#define M3S_FOLD_MULHI(a, b) __mulhi((a), (b))
#include "m3s_enc_fold_gen.cuh"

__constant__ int32_t c_enc_fl[32][64];    // MP3Encoder filter matrix (:544-555) and analysis window (tables.py:34-78) for the
__constant__ int32_t c_enc_win[512];      // correction pass of a slot whose fast path reported `bad`

#define ANA3_WARPS 8   // warps per CTA = 32-slot groups per block (8 warps x 2 CTAs per SM, see above)
struct Ana3Smem {
    static constexpr int SLOTS = 32 * ANA3_WARPS;   // slots per block: one per thread
    static constexpr int XP = 15 + SLOTS;      // columns of the sample tile: 15 slots of history + the block's slots; odd: conflict-free fills
    static constexpr int RING = (SLOTS + 35 + 17) / 18 * 18;   // subband-sample ring: a granule reaches back 36 slots from its end, a block adds
                                                               // SLOTS more; a multiple of 18, so that the rows of a granule never wrap
    static constexpr int RUN = SLOTS * 9 / 18 - 1;   // granules per CTA: with the warm-up granule 9 blocks exactly
    int32_t xT[32][XP];                // sample 32 u + r of this channel at [r][u - u0], as int16 << 16
    int32_t sb[RING + 18][33];         // [ring row][band] subband samples; rows RING.. stay zero (the granule in front of a clip)
    int32_t mf[ANA3_WARPS][576];       // per warp: [band * 18 + k] MDCT lines of the granule it works on
    uint32_t bins[ANA3_WARPS][24];     // per warp: 0..20 band energies, 21 total, 22 xrmax
    uint32_t en_thresh[32];
    uint8_t sfb[576];
    int32_t ca[8], cs[8];
};

template <int ANA3_XP>
struct Ana3LoadX {   // sample k of input j of the windowing: x[32 t + 31 - j - 64 k] of this lane's slot t (p = &xT[0][column of t])
    const int32_t *p;
    __device__ __forceinline__ int32_t operator()(int j, int k) const
    {
        return j < 32 ? p[(31 - j) * ANA3_XP - 2 * k] : p[(63 - j) * ANA3_XP - 2 * k - 1];
    }
};
struct Ana3LoadSb {  // input j of the MDCT: slot j of the previous granule (j < 18) or slot j - 18 of the current one, band = lane
    const int32_t *prev, *cur;   // the two granules' first ring rows at this lane's band
    __device__ __forceinline__ int32_t operator()(int j) const { return j < 18 ? prev[j * 33] : cur[(j - 18) * 33]; }
};

// `zero` (always 0) is added to every shared product (guard 0 of m3s_enc_fold_gen.cuh): ptxas cannot see through it, so it keeps
// each product once instead of recomputing it per use, and the add folds into the multiply's addend
__global__ void __launch_bounds__(32 * ANA3_WARPS, 2)
k_enc_analysis_fold(const int16_t *__restrict__ pcm, const M3sEncClip *__restrict__ clips, const M3sEncWork *__restrict__ work,
                    const M3sDevTables *__restrict__ T, const EncTables *__restrict__ ET, int64_t chunk_frame0,
                    int32_t *__restrict__ mdct, M3sEncStats *__restrict__ stats, const uint32_t zero)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    typedef Ana3Smem Smem;
    constexpr int ANA3_THREADS = 32 * ANA3_WARPS, ANA3_SLOTS = Smem::SLOTS, ANA3_XP = Smem::XP, ANA3_RING = Smem::RING;
    Smem &S = *reinterpret_cast<Smem *>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const M3sEncWork wk = work[blockIdx.x];
    const M3sEncClip cl = clips[wk.clip];
    const int ch = wk.ch;
    for (int i = tid; i < 576; i += ANA3_THREADS) S.sfb[i] = T->long_sfb_of[cl.sr_idx][i];
    if (tid < 8) { S.ca[tid] = T->enc_ca[tid]; S.cs[tid] = T->enc_cs[tid]; }
    if (tid < 32) S.en_thresh[tid] = ET->en_thresh[tid];
    if (tid < 24 * ANA3_WARPS) (&S.bins[0][0])[tid] = 0u;
    for (int i = tid; i < 18 * 33; i += ANA3_THREADS) (&S.sb[ANA3_RING][0])[i] = 0;

    const uint32_t *pcm32 = (const uint32_t *)(pcm + cl.pcm_base);  // one stereo sample per word (pcm_base is even)
    const int sh = ch ? 0 : 16;                                     // channel 0 = low half of the word
    const int g_end = wk.g_first + wk.count;
    const int t_begin = wk.g_first > 0 ? 18 * (wk.g_first - 1) : 0; // first slot of the stream: one warm-up granule in front of the run
    const int t_stop = 18 * g_end;                                  // slots of the run end here
    const int64_t s_end = (int64_t)g_end * 576;                     // ... and so do the samples it may read (clip / chunk staging)
    const int n_blocks = (t_stop - t_begin + ANA3_SLOTS - 1) / ANA3_SLOTS;
    int g_next = wk.g_first;
    for (int k = 0; k < n_blocks; k++) {
        const int t0 = t_begin + ANA3_SLOTS * k;
        // ---- sample tile: slots t0 - 15 .. t0 + ANA3_SLOTS - 1, transposed (row = sample within its slot, column = slot)
        {
            const int64_t n0 = ((int64_t)t0 - 15) * 32;
            constexpr int NLD = (32 * ANA3_XP + ANA3_THREADS - 1) / ANA3_THREADS;
            uint32_t w[NLD];
#pragma unroll
            for (int q = 0; q < NLD; q++) {   // every load of the tile in flight at once: one DRAM latency per block, not one per batch
                const int i = tid + ANA3_THREADS * q;
                const int64_t n = n0 + i;
                w[q] = (i < 32 * ANA3_XP && n >= 0 && n < s_end) ? __ldg(pcm32 + n) : 0u;
            }
#pragma unroll
            for (int q = 0; q < NLD; q++) {
                const int i = tid + ANA3_THREADS * q;
                if (i < 32 * ANA3_XP) S.xT[i & 31][i >> 5] = (int32_t)((w[q] << sh) & 0xFFFF0000u);
            }
        }
        __syncthreads();   // also: every warp has left the MDCT phase of the previous block, the ring rows below are free
        if (k + 1 < n_blocks) {   // the next block's new samples on their way into L2 while this block is in the arithmetic
            const int64_t n = ((int64_t)t0 + ANA3_SLOTS) * 32 + 32 * tid;   // one 128-byte line per thread: 32 * SLOTS samples in all
            if (n < s_end) asm volatile("prefetch.global.L2 [%0];" ::"l"(pcm32 + n));
        }
        // ---- windowing + matrixing of slot t0 + tid: y_j = sum_k mul(x[32 t + 31 - j - 64 k], enwindow[j + 64 k])   (:337-356),
        //      s_b = sum_j mul(fl[b][j], y_j); odd bands of odd slots negated   (:358-368, :678-679)
        if (t0 + 32 * warp < t_stop) {   // warp-uniform
            uint32_t acc[32], bad, any;
            const Ana3LoadX<ANA3_XP> ld{&S.xT[0][15 + tid]};
            m3s_matrix_fold<0>(ld, zero, acc, bad, any);
            if (bad) {   // some y has 26 zero low bits: its negative uses were charged a correction they may not owe
                if (any == 0u) {
#pragma unroll
                    for (int b = 0; b < 32; b++) acc[b] = 0u;
                } else {
#pragma unroll 1
                    for (int j = 0; j < 64; j++) {
                        const int32_t *xp = j < 32 ? ld.p + (31 - j) * ANA3_XP : ld.p + (63 - j) * ANA3_XP - 1;
                        uint32_t ys = 0u;
#pragma unroll
                        for (int kk = 0; kk < 8; kk++) ys += (uint32_t)__mulhi(xp[-2 * kk], c_enc_win[j + 64 * kk]);
                        if ((ys & M3S_MATRIX_FOLD_YMASK) != 0u) continue;
#pragma unroll
                        for (int b = 0; b < 32; b++) {
                            const int32_t v = c_enc_fl[b][j];
                            acc[b] += (uint32_t)(v < 0 && (uint32_t)v * ys == 0u);
                        }
                    }
                }
            }
            int32_t *row = &S.sb[(ANA3_SLOTS * k + tid) % ANA3_RING][0];
            const uint32_t odd = 0u - (uint32_t)(lane & 1);   // t_begin and the block size are even: slot parity = lane parity
#pragma unroll
            for (int b = 0; b < 32; b++) row[b] = (int32_t)((b & 1) ? (acc[b] ^ odd) - odd : acc[b]);
        }
        __syncthreads();
        // ---- every granule whose 18 slots are now in the ring: one warp per granule, lane = band
        int g_hi = (t0 + ANA3_SLOTS) / 18;
        if (g_hi > g_end) g_hi = g_end;
        for (int G = g_next + warp; G < g_hi; G += ANA3_WARPS) {
            int32_t *mf = S.mf[warp];
            uint32_t *bins = S.bins[warp];
            // ---- MDCT   (:683-701)
            {
                uint32_t acc[18], bad, any;
                const Ana3LoadSb ld{&S.sb[G == 0 ? ANA3_RING : (18 * (G - 1) - t_begin) % ANA3_RING][lane], &S.sb[(18 * G - t_begin) % ANA3_RING][lane]};
                m3s_mdct_fold<0>(ld, zero, acc, bad, any);
                if (bad) {
                    if (any == 0u) {
#pragma unroll
                        for (int q = 0; q < 18; q++) acc[q] = 0u;
                    } else {
#pragma unroll 1
                        for (int j = 0; j < 36; j++) {
                            const uint32_t v = (uint32_t)(j < 18 ? ld.prev[j * 33] : ld.cur[(j - 18) * 33]);
                            if ((v & M3S_MDCT_FOLD_YMASK) != 0u) continue;
#pragma unroll
                            for (int q = 0; q < 18; q++) {
                                const int32_t c = c_enc_cos[q][j];
                                acc[q] += (uint32_t)(c < 0 && (uint32_t)c * v == 0u);
                            }
                        }
                    }
                }
#pragma unroll
                for (int q = 0; q < 18; q++) mf[lane * 18 + q] = (int32_t)acc[q];
            }
            __syncwarp();
            // ---- alias butterflies between neighbouring bands, cmuls with >> 31   (:704-744, util.py:145-155)
            for (int r = lane; r < 248; r += 32) {
                const int band = 1 + (r >> 3), kk = r & 7;
                const int64_t are = mf[band * 18 + kk], aim = mf[(band - 1) * 18 + 17 - kk];
                const int64_t bre = S.cs[kk], bim = S.ca[kk];
                mf[band * 18 + kk] = (int32_t)((are * bre - aim * bim) >> 31);
                mf[(band - 1) * 18 + 17 - kk] = (int32_t)((are * bim + aim * bre) >> 31);
            }
            __syncwarp();
            // ---- store + statistics: xrmax, en_tot, en[sfb]   (:772-776, :836-857)
            const int frame = G >> 1, gr = G & 1;
            const int64_t gslot = (((int64_t)(cl.frame_base + frame) - chunk_frame0) * 2 + ch) * 2 + gr;
            uint32_t tot = 0u, mx = 0u;
            for (int i = lane; i < 576; i += 32) {
                const int32_t v = mf[i];
                mdct[gslot * 576 + i] = v;
                const uint32_t e = (uint32_t)(mulsr32(v, v) >> 10);
                const int sfb = S.sfb[i];
                if (sfb < 21 && e) atomicAdd(&bins[sfb], e);
                tot += e;
                mx = max(mx, v < 0 ? (uint32_t)(-(int64_t)v) : (uint32_t)v);
            }
            tot = __reduce_add_sync(0xFFFFFFFFu, tot);
            mx = __reduce_max_sync(0xFFFFFFFFu, mx);
            __syncwarp();
            if (lane < 22) {
                const uint32_t temp = lane == 21 ? tot : bins[lane];
                int en = 0;
                if (temp) {
                    en = -21;
                    for (int j = 0; j < 31; j++) en += S.en_thresh[j] <= temp;
                }
                M3sEncStats *st = stats + gslot;
                if (lane == 21) { st->en_tot = (int8_t)en; st->xrmax = (int32_t)mx; }
                else st->en[lane] = (int8_t)en;
            }
            __syncwarp();
            if (lane < 21) bins[lane] = 0u;
            __syncwarp();
        }
        g_next = g_hi > g_next ? g_hi : g_next;
    }
}

// ================================================================================================
// E2, shared pieces: the reference's step search on shared-memory tables (the slow path of k_enc_resolve, the quantiser of k_enc_emit)
// ================================================================================================
struct RateSmem {
    uint16_t i2i[10000];
    uint2 hlc[256];        // .x = hl4 (code lengths of books 13 | 15 << 8 | 16 << 16 | 24 << 24), .y = signs | escapes << 16 of the pair
    int32_t steptabi[128];
    double steptab[128];
    uint16_t sfb[24];
    uint16_t linmax[32];
    uint8_t linbits[32];
    uint8_t subdv[23][2];
    uint8_t pair[32][2];
    uint8_t hlc1[2][16];
};

struct GranInfo {  // the reference's gr_info fields the probes rewrite (MP3_Encoder.py:76-104)
    int bv, count1, c1sel, r0, r1, ts0, ts1, ts2;
};

// the reference's double-precision fallback of quantize() for ln >= 10000 (:401-407); rare, kept out of line so that
// the 18 call sites of the unrolled quantiser stay small
__device__ __noinline__ int quant_slow(int32_t xabs, double scale)
{
    const double dbl = __dmul_rn(__dmul_rn((double)xabs, scale), 4.656612875e-10);
    return (int)__dsqrt_rn(__dmul_rn(__dsqrt_rn(dbl), dbl));
}

// quantize() of the single largest coefficient: decides `quantize(...) > 8192` without touching the other 575
// (ix is monotone in |xr| for a fixed step, and an overflowing probe's ix is never read again).   (:374-415)
__device__ __forceinline__ int quant_max(const RateSmem &S, int32_t xrmax, int step)
{
    const int32_t scalei = S.steptabi[step + 127];
    const int32_t ln = mulr32(xrmax, scalei);
    if (ln > 165140) return 16384;
    if (ln < 10000) return S.i2i[ln];
    return quant_slow(xrmax, S.steptab[step + 127]);
}

__device__ __forceinline__ int table_cost(const RateSmem &S, int t, uint32_t lo, uint32_t hi, uint32_t cnt)
{
    // count_bit() of table t over a region from the region's pooled sums   (:215-263)
    const int nsign = cnt & 0xFFFF, n15 = cnt >> 16;
    if (t == 0) return 0;
    if (t == 13) return (int)(lo & 0xFFFF) + nsign;
    if (t == 15) return (int)(hi & 0xFFFF) + nsign;
    return (int)(t < 24 ? (lo >> 16) : (hi >> 16)) + nsign + (int)S.linbits[t] * n15;
}

// new_choose_table (:1170-1264) on pooled sums; `k` = payload bits already consumed by earlier regions of this probe
__device__ __forceinline__ int choose_table(const RateSmem &S, int mx, uint32_t lo, uint32_t hi, uint32_t cnt, bool hiding,
                                            int k, int hn, uint32_t hb)
{
    if (mx == 0) return 0;
    int choice;
    if (mx < 15) {
        choice = 13;  // the count-down search always stops at 13 (A.E4); only its 13-vs-15 arm is live
        if (table_cost(S, 15, lo, hi, cnt) <= table_cost(S, 13, lo, hi, cnt)) choice = 15;
    } else {
        // first table of 15..23 / 24..31 whose lin_max (0,1,3,7,15,63,255,1023,8191 / 15,31,63,127,255,511,2047,8191) covers mx - 15:
        // a function of the bit length of mx - 15 (<= 13 bits since mx <= 8192 here)
        const int nb = 32 - __clz(mx - 15);
        const int c0 = 15 + (int)((0x88877665543210ULL >> (4 * nb)) & 15);
        const int c1 = 24 + (int)((0x77665432100000ULL >> (4 * nb)) & 15);
        choice = c0;
        if (table_cost(S, c1, lo, hi, cnt) < table_cost(S, c0, lo, hi, cnt)) choice = c1;
    }
    if (hiding && k < hn) choice = S.pair[choice][(hb >> k) & 1u];
    return choice;
}

// Everything a probe derives from the quantised values WITHOUT looking at the payload bits: run lengths, count1 bits, region
// bounds and, per region, the maximum and the pooled code-length / sign / escape sums.  The table choice (with the stego swap)
// and the bit count follow from it in a few scalar steps (probe_tables).
struct Pooled {
    int c1bits, c1sel, bv, count1, r0, r1, a1, a2, a3;
    uint32_t m0, m1, m2, lo0, hi0, cn0, lo1, hi1, cn1, lo2, hi2, cn2;
};

// calc_run_len + count1_bit_count + subdivide + the pooled sums of big_v_tab_select / big_v_bit_count for the quantised values
// held pair-interleaved in the warp (lane L holds pairs 32 j + L).  a1..a3 come in as the slot's current addresses.
__device__ __forceinline__ void probe_pool(const RateSmem &S, const uint32_t (&qx)[9], const uint32_t (&qy)[9], int lane, int a1, int a2,
                                           int a3, Pooled &P)
{
    GranInfo gi;
    const uint32_t FULL = 0xFFFFFFFFu;
    // ---- calc_run_len (:266-291)
    uint32_t lastnz = 0, lastbig = 0, nzmask = 0;
#pragma unroll
    for (int j = 0; j < 9; j++) {
        const uint32_t p = 32 * j + lane;
        if (qx[j] | qy[j]) lastnz = p + 1;
        if (qx[j] > 1) lastbig = 2 * p + 1;
        if (qy[j] > 1) lastbig = 2 * p + 2;
        nzmask |= (uint32_t)(qx[j] != 0) << (2 * j) | (uint32_t)(qy[j] != 0) << (2 * j + 1);
    }
    lastnz = __reduce_max_sync(FULL, lastnz);
    lastbig = __reduce_max_sync(FULL, lastbig);
    const int i_end = 2 * (int)lastnz;
    gi.count1 = (i_end - (int)lastbig) >> 2;
    gi.bv = (i_end - 4 * gi.count1) >> 1;
    // ---- count1_bit_count (:171-211): quads start at pair bv; the partner pair lives in the next lane
    const uint32_t nb = __shfl_sync(FULL, nzmask, (lane + 1) & 31);
    uint32_t c1s = 0;
#pragma unroll
    for (int j = 0; j < 9; j++) {
        const int rel = 32 * j + lane - gi.bv;
        if (rel >= 0 && rel < 2 * gi.count1 && !(rel & 1)) {
            const uint32_t me = (nzmask >> (2 * j)) & 3u;
            const uint32_t nx = lane < 31 ? (nb >> (2 * j)) & 3u : (nb >> (2 * j + 2)) & 3u;
            const uint32_t idx = me | (nx << 2);  // v + 2 w + 4 x + 8 y
            const uint32_t nn = __popc(idx);
            // code lengths: table A = {1,4,4,5,4,6,5,6,4,5,5,6,5,6,6,6} (one nibble each), table B = 4 everywhere
            c1s += ((uint32_t)((0x6665655465645441ULL >> (4 * idx)) & 15) + nn) | ((4u + nn) << 16);
        }
    }
    c1s = __reduce_add_sync(FULL, c1s);
    int bits;
    if ((c1s & 0xFFFF) < (c1s >> 16)) { gi.c1sel = 0; bits = c1s & 0xFFFF; }
    else { gi.c1sel = 1; bits = c1s >> 16; }
    // ---- subdivide (:998-1036); with big_values == 0 the addresses keep their old values (A.E6)
    if (gi.bv == 0) { gi.r0 = 0; gi.r1 = 0; }
    else {
        const int bvr = 2 * gi.bv;
        const int anz = __popc(__ballot_sync(FULL, lane < 23 && (int)S.sfb[lane] < bvr));
        int tc = S.subdv[anz][0];
        while (tc > 0 && (int)S.sfb[tc + 1] > bvr) tc--;
        gi.r0 = tc;
        a1 = S.sfb[tc + 1];
        const int base = tc + 1;
        tc = S.subdv[anz][1];
        while (tc > 0 && (int)S.sfb[min(base + tc + 1, 23)] > bvr) tc--;
        gi.r1 = tc;
        a2 = S.sfb[min(base + tc + 1, 23)];
        a3 = bvr;
    }
    // ---- pooled region sums: [0, a1) [a1, a2) [a2, 2 bv)   (:1147-1168, :294-318)
    const int e2 = 2 * gi.bv;
    uint32_t lo0 = 0, hi0 = 0, cn0 = 0, lo1 = 0, hi1 = 0, cn1 = 0, lo2 = 0, hi2 = 0, cn2 = 0, m0 = 0, m1 = 0, m2 = 0;
#pragma unroll
    for (int j = 0; j < 9; j++) {
        const int e = 2 * (32 * j + lane);
        const uint32_t x = qx[j], y = qy[j];
        const uint2 w2 = S.hlc[min(x, 15u) * 16 + min(y, 15u)];
        const uint32_t wl = w2.x & 0x00FF00FFu, wh = (w2.x >> 8) & 0x00FF00FFu;
        const uint32_t cn = w2.y;   // (x != 0) + (y != 0) + (((x > 14) + (y > 14)) << 16)
        const uint32_t mx = max(x, y);
        if (e < a1) { lo0 += wl; hi0 += wh; cn0 += cn; m0 = max(m0, mx); }
        else if (e < a2) { lo1 += wl; hi1 += wh; cn1 += cn; m1 = max(m1, mx); }
        else if (e < e2) { lo2 += wl; hi2 += wh; cn2 += cn; m2 = max(m2, mx); }
    }
    m0 = __reduce_max_sync(FULL, m0); m1 = __reduce_max_sync(FULL, m1); m2 = __reduce_max_sync(FULL, m2);
    lo0 = __reduce_add_sync(FULL, lo0); hi0 = __reduce_add_sync(FULL, hi0); cn0 = __reduce_add_sync(FULL, cn0);
    lo1 = __reduce_add_sync(FULL, lo1); hi1 = __reduce_add_sync(FULL, hi1); cn1 = __reduce_add_sync(FULL, cn1);
    lo2 = __reduce_add_sync(FULL, lo2); hi2 = __reduce_add_sync(FULL, hi2); cn2 = __reduce_add_sync(FULL, cn2);
    P.c1bits = bits; P.c1sel = gi.c1sel; P.bv = gi.bv; P.count1 = gi.count1; P.r0 = gi.r0; P.r1 = gi.r1; P.a1 = a1; P.a2 = a2; P.a3 = a3;
    P.m0 = m0; P.m1 = m1; P.m2 = m2; P.lo0 = lo0; P.hi0 = hi0; P.cn0 = cn0; P.lo1 = lo1; P.hi1 = hi1; P.cn1 = cn1;
    P.lo2 = lo2; P.hi2 = hi2; P.cn2 = cn2;
}

// big_v_tab_select with the stego swap (the payload index advances past non-zero tables only) + big_v_bit_count   (:1147-1168, :294-318)
__device__ __forceinline__ int probe_tables(const RateSmem &S, const Pooled &P, bool hiding, int hn, uint32_t hb, GranInfo &gi)
{
    gi.bv = P.bv; gi.count1 = P.count1; gi.c1sel = P.c1sel; gi.r0 = P.r0; gi.r1 = P.r1;
    const int e2 = 2 * P.bv;
    int k = 0;
    gi.ts0 = P.a1 <= 0 ? 0 : choose_table(S, (int)P.m0, P.lo0, P.hi0, P.cn0, hiding, k, hn, hb);
    if (gi.ts0 > 0) k++;
    gi.ts1 = P.a2 <= P.a1 ? 0 : choose_table(S, (int)P.m1, P.lo1, P.hi1, P.cn1, hiding, k, hn, hb);
    if (gi.ts1 > 0) k++;
    gi.ts2 = e2 <= P.a2 ? 0 : choose_table(S, (int)P.m2, P.lo2, P.hi2, P.cn2, hiding, k, hn, hb);
    return P.c1bits + table_cost(S, gi.ts0, P.lo0, P.hi0, P.cn0) + table_cost(S, gi.ts1, P.lo1, P.hi1, P.cn1) +
           table_cost(S, gi.ts2, P.lo2, P.hi2, P.cn2);
}

// quantize() of all 576 values (:374-415); callers know from quant_max() that the maximum is <= 8192
__device__ __forceinline__ void quantize_all(const RateSmem &S, const uint32_t (&ax)[9], const uint32_t (&ay)[9], int step,
                                             uint32_t (&qx)[9], uint32_t (&qy)[9])
{
    const int32_t scalei = S.steptabi[step + 127];
    uint32_t big = 0;
#pragma unroll
    for (int j = 0; j < 9; j++) {
        const int32_t lx = mulr32((int32_t)ax[j], scalei), ly = mulr32((int32_t)ay[j], scalei);
        qx[j] = S.i2i[min(lx, 9999)];
        qy[j] = S.i2i[min(ly, 9999)];
        big |= (uint32_t)(lx >= 10000) << (2 * j) | (uint32_t)(ly >= 10000) << (2 * j + 1);
    }
    if (__any_sync(0xFFFFFFFFu, big != 0)) {
        const double scale = S.steptab[step + 127];
#pragma unroll
        for (int j = 0; j < 9; j++) {
            if ((big >> (2 * j)) & 1u) qx[j] = (uint32_t)quant_slow((int32_t)ax[j], scale);
            if ((big >> (2 * j + 1)) & 1u) qy[j] = (uint32_t)quant_slow((int32_t)ay[j], scale);
        }
    }
}

// the shared-memory tables of k_enc_resolve and k_enc_emit; the band bounds S.sfb depend on the sample rate and only the
// resolve kernel reads them (it loads them itself, once per sample-rate group)
__device__ __forceinline__ void rate_tables_load(RateSmem &S, const M3sDevTables *__restrict__ T, const EncTables *__restrict__ ET,
                                                 int tid, int nthr)
{
    for (int i = tid; i < 10000; i += nthr) S.i2i[i] = (uint16_t)T->int2idx[i];
    for (int i = tid; i < 256; i += nthr) {
        const uint32_t x = i >> 4, y = i & 15;
        S.hlc[i] = make_uint2(ET->hl4[i], (uint32_t)(x != 0) + (uint32_t)(y != 0) + (((uint32_t)(x > 14) + (uint32_t)(y > 14)) << 16));
    }
    for (int i = tid; i < 128; i += nthr) { S.steptabi[i] = T->steptabi[i]; S.steptab[i] = T->steptab[i]; }
    if (tid < 32) {
        S.linmax[tid] = T->enc_linmax[tid];
        S.linbits[tid] = T->enc_linbits[tid];
        S.pair[tid][0] = T->pair[tid][0];
        S.pair[tid][1] = T->pair[tid][1];
    }
    if (tid < 23) { S.subdv[tid][0] = T->subdv[tid][0]; S.subdv[tid][1] = T->subdv[tid][1]; }
    if (tid < 16) { S.hlc1[0][tid] = ET->hlc1[0][tid]; S.hlc1[1][tid] = ET->hlc1[1][tid]; }
}

// ================================================================================================
// E2: k_enc_probe -> k_enc_resolve -> k_enc_emit
//
// A granule depends on its predecessors only through (a) the <= 3 payload bits at its hide_str_offset -- i.e. through one of
// 15 "variants": three bits (8), two (4) or one (2) left before the payload ends, or none -- and (b) the slot's stale
// address1..3, which are read only by probes that find big_values == 0 among non-zero values (A.E6).  So
//   k_enc_probe    one warp per granule-channel, NO chain: lane v walks the reference's step search for variant v; the
//                  payload-independent part of a probe (quantise, run lengths, pooled code-length sums: `Pooled`) is computed
//                  once per distinct step by the whole warp and cached in shared memory -- on the tone+noise corpus the eight
//                  3-bit variants visit 7 distinct steps together, one fewer than the 8 probes of a single sequential run;
//   k_enc_resolve  one warp per clip walks the granules in the reference's order with nothing but register arithmetic per
//                  granule (offset -> variant -> bits consumed), 32 granules per batch; granules that did depend on the
//                  stale addresses (flagged by the probe kernel) are redone here with the true state;
//   k_enc_emit     one warp per granule quantises at the chosen step and writes the values the packer reads.
// ================================================================================================
#define PROBE_WARPS 8        // warps per CTA of k_enc_probe, two CTAs per SM (128 registers a thread)
#define PROBE_G 8            // granules per warp of k_enc_probe (amortises the CTA's table staging)
#define PROBE_CACHE 24       // distinct steps cached per granule; more than that (never seen) sends the granule to the resolve kernel
#define VAR_SILENT 0x80000000u
#define VAR_SLOW 0x40000000u
#define VAR_OVERRUN (VAR_SLOW | VAR_SILENT)   // the walk needs step 1 (steptabi[128]): the resolve kernel's search finds it again and records it
#define VAR_NONE 0xFFFFFFFFu

// What a probe (one step of one granule) leaves for the variant walks: everything but the payload bits.  The table the
// reference would choose for a region BEFORE the swap does not depend on the payload, nor does the payload index of a region
// (the number of earlier regions with a non-zero table, and a swapped table is non-zero iff the original is); so the bit count
// of a variant is  c1bits + sum over regions of cost[region][mode]  with mode = no swap / swap by a '0' / swap by a '1'.
struct ProbeRow {
    int32_t c1bits;
    uint32_t geo;             // big_values[0:9) count1[9:17) count1table[17] region0[18:22) region1[22:25) table0 != 0 [25] table1 != 0 [26]
    uint32_t addr;            // address1 | address2 << 10 | address3 << 20 after this probe
    uint32_t tag;             // the addresses the sums were pooled over when the probe read them (big_values == 0, A.E6), else VAR_NONE
    uint16_t cost[3][4];      // [region][mode] count_bit() of the region under table tab[region][mode]
    uint8_t tab[3][4];
    uint32_t lt, le;          // bit v: variant v's bit count of this probe is < / <= max_bits (the two decisions the step search takes)
};
struct ProbeWarpSmem {
    ProbeRow row[PROBE_CACHE];
    uint8_t slotmap[128];    // step + 120 -> cache row (0xFF = not computed yet)
};
// variant v <-> (bits left, their values): 0..7 three bits, 8..11 two, 12..13 one, 14 none (also: plain encode)
__device__ __forceinline__ void variant_bits(int v, int &hn, uint32_t &hb)
{
    if (v < 8) { hn = 3; hb = (uint32_t)v; }
    else if (v < 12) { hn = 2; hb = (uint32_t)(v - 8); }
    else if (v < 14) { hn = 1; hb = (uint32_t)(v - 12); }
    else { hn = 0; hb = 0u; }
}
__device__ __forceinline__ int variant_index(int hn, uint32_t hb)
{
    return hn == 3 ? (int)hb : (hn == 2 ? 8 + (int)hb : (hn == 1 ? 12 + (int)hb : 14));
}

__device__ __forceinline__ void load_granule(const int32_t *__restrict__ mdct_g, int lane, uint32_t (&ax)[9], uint32_t (&ay)[9], uint32_t &sg)
{
    const int2 *xr = (const int2 *)mdct_g;
    sg = 0;
#pragma unroll
    for (int j = 0; j < 9; j++) {
        const int2 v = __ldg(xr + 32 * j + lane);
        ax[j] = v.x < 0 ? (uint32_t)(-(int64_t)v.x) : (uint32_t)v.x;
        ay[j] = v.y < 0 ? (uint32_t)(-(int64_t)v.y) : (uint32_t)v.y;
        sg |= (uint32_t)(v.x < 0) << (2 * j) | (uint32_t)(v.y < 0) << (2 * j + 1);
    }
}

// max_bits of frame f of clip `cl` (its own rate pair); `byteoff` = the padding tables of the call
__device__ __forceinline__ int frame_max_bits(const uint32_t *__restrict__ byteoff, const M3sEncClip &cl, int f, int &padding, int &mean_bits)
{
    const uint32_t *bo = byteoff + cl.pad_base;
    padding = (int)(bo[f + 1] - bo[f]) - cl.whole_slots;
    const int bits_per_frame = 8 * (cl.whole_slots + padding);
    mean_bits = (bits_per_frame - 288) / 2;                  // :634-636 (side info 8 * (4 + 32) bits)
    return min(mean_bits / 2, 4095);                         // :894-912 with the reservoir never enabled (A.E7)
}

// Shared-memory tables of k_enc_probe.  The quantiser table carries, next to int2idx[ln], what the passes after it would
// otherwise re-derive per value: the value clamped to 15 in BOTH nibble positions of a Huffman-table index byte and the
// "non-zero" / "above one" flags in both positions of a pair's flag group, so that one LOP3 merges the two values of a pair
// into (index byte, flag group):  M = (ex & XROLE) | (ey & ~XROLE).
#define I2X_XROLE 0x05F00000u   // bits an entry contributes as the FIRST value of a pair: index nibble [20:24), non-zero [24], above-one [26]
struct ProbeTab {
    uint32_t i2x[10000];     // q | min(q,15) << 16 | min(q,15) << 20 | (q != 0) * 0x03000000 | (q > 1) * 0x0C000000
    uint2 hlc[256];          // .x = code lengths of books 13 | 15 << 8 | 16 << 16 | 24 << 24 at [x * 16 + y], .y = signs | escapes << 16
    int32_t steptabi[128];
    double steptab[128];
    uint16_t sfb[24];
    uint8_t linbits[32];
    uint8_t subdv[23][2];
    uint8_t pair[32][2];
    uint32_t subdiv[289];    // subdivide() by big_values: region0_count | region1_count << 4 | address1 << 8 | address2 << 18
    uint32_t c1cost[256];    // count1 quads two at a time: sum over the byte's two 4-bit patterns of (table A bits | table B bits << 16)
};
struct ProbeSmem {
    ProbeTab T;
    ProbeWarpSmem W[PROBE_WARPS];
};

__device__ __forceinline__ uint32_t i2x_entry(uint32_t q)
{
    const uint32_t c = min(q, 15u);
    return q | c << 16 | c << 20 | (q != 0 ? 0x03000000u : 0u) | (q > 1 ? 0x0C000000u : 0u);
}

// quantize() of one value (:374-415) as a table entry
__device__ __forceinline__ uint32_t quant_entry(const ProbeTab &T, uint32_t a, int32_t scalei, double scale)
{
    const int32_t ln = mulr32((int32_t)a, scalei);
    if (ln < 10000) return T.i2x[ln];
    return i2x_entry((uint32_t)quant_slow((int32_t)a, scale));
}

// quantize() > 8192 for the granule's largest coefficient (ix is monotone in |xr|)
__device__ __forceinline__ bool quant_overflows(const ProbeTab &T, int32_t xrmax, int step)
{
    const int32_t ln = mulr32(xrmax, T.steptabi[step + 127]);
    if (ln > 165140) return true;
    if (ln < 10000) return false;   // int2idx stays below 1000
    return quant_slow(xrmax, T.steptab[step + 127]) > 8192;
}

// bit count of a probe under variant (hn, hb): the payload index of a region is the number of earlier regions with a table
__device__ __forceinline__ int row_bits(const ProbeRow &R, int hn, uint32_t hb, int &mode0, int &mode1, int &mode2)
{
    const uint32_t geo = R.geo;
    const int k1 = (int)((geo >> 25) & 1u), k2 = k1 + (int)((geo >> 26) & 1u);
    mode0 = 0 < hn ? 1 + (int)(hb & 1u) : 0;
    mode1 = k1 < hn ? 1 + (int)((hb >> k1) & 1u) : 0;
    mode2 = k2 < hn ? 1 + (int)((hb >> k2) & 1u) : 0;
    return R.c1bits + (int)R.cost[0][mode0] + (int)R.cost[1][mode1] + (int)R.cost[2][mode2];
}

// One probe = quantize + calc_run_len + count1_bit_count + subdivide + the table choice and bit count of every region under
// "no swap / swap by 0 / swap by 1", for step `sc`; written to row R by lanes 0..2.  Returns false when the probe reads the
// slot's stale addresses that only the resolve kernel knows (big_values == 0 among non-zero values before any probe of this walk
// had big values, A.E6).
__device__ __forceinline__ bool probe_row(const ProbeTab &T, const uint32_t (&ax)[9], const uint32_t (&ay)[9], int32_t xrmax, int sc, int lane,
                                          int lhave, uint32_t lla, int max_bits, int vhn, uint32_t vhb, ProbeRow &R)
{
    const uint32_t FULL = 0xFFFFFFFFu;
    const int32_t scalei = T.steptabi[sc + 127];
    uint32_t M[9], X[9], accA = 0, accB = 0;
    // ---- quantize (:374-415): M = index byte + flag group of the pair, X = the larger entry (entries are monotone in the value)
    if (mulr32(xrmax, scalei) < 10000) {
#pragma unroll
        for (int j = 0; j < 9; j++) {
            const uint32_t ex = T.i2x[mulr32((int32_t)ax[j], scalei)], ey = T.i2x[mulr32((int32_t)ay[j], scalei)];
            M[j] = (ex & I2X_XROLE) | (ey & ~I2X_XROLE);
            X[j] = max(ex, ey);
        }
    } else {
        const double scale = T.steptab[sc + 127];
#pragma unroll
        for (int j = 0; j < 9; j++) {
            const uint32_t ex = quant_entry(T, ax[j], scalei, scale), ey = quant_entry(T, ay[j], scalei, scale);
            M[j] = (ex & I2X_XROLE) | (ey & ~I2X_XROLE);
            X[j] = max(ex, ey);
        }
    }
    // flag groups {x != 0, y != 0, x > 1, y > 1} of my pairs: pair j at accA[4j : 4j + 4), pair 8 in accB
#pragma unroll
    for (int j = 0; j < 8; j++) accA |= j < 6 ? (M[j] & 0x0F000000u) >> (24 - 4 * j) : (M[j] & 0x0F000000u) << (4 * j - 24);
    accB = (M[8] >> 24) & 15u;
    // ---- calc_run_len (:266-291)
    uint32_t lastnz = 0, lastbig = 0;
    {
        const uint32_t nzA = accA & 0x33333333u, bgA = accA & 0xCCCCCCCCu;
        if (accB & 3u) lastnz = 256 + lane + 1;
        else if (nzA) lastnz = 32 * ((31 - __clz(nzA)) >> 2) + lane + 1;
        if (accB & 12u) lastbig = 2 * (256 + lane) + 1 + ((accB >> 3) & 1u);
        else if (bgA) {
            const int pos = 31 - __clz(bgA);
            lastbig = 2 * (32 * (pos >> 2) + lane) + 1 + (pos & 1);
        }
    }
    lastnz = __reduce_max_sync(FULL, lastnz);
    lastbig = __reduce_max_sync(FULL, lastbig);
    const int i_end = 2 * (int)lastnz;
    const int count1 = (i_end - (int)lastbig) >> 2;
    const int bv = (i_end - 4 * count1) >> 1;
    // ---- count1_bit_count (:171-211): quads start at pair bv; the partner pair lives in the next lane (lane 31: lane 0, next row).
    //      A lane's pairs all have the parity of (lane - bv), so it either starts a quad at each of its in-range pairs or at none; the
    //      quads' 4-bit patterns v + 2 w + 4 x + 8 y are looked up two at a time, out-of-range ones zeroed and their cost taken back
    int c1bits, c1sel;
    {
        uint32_t nbA = __shfl_sync(FULL, accA, (lane + 1) & 31), nbB = __shfl_sync(FULL, accB, (lane + 1) & 31);
        if (lane == 31) { nbA = (nbA >> 4) | (nbB << 28); nbB = 0; }
        const uint32_t idxA = (accA & 0x33333333u) | ((nbA & 0x33333333u) << 2), idxB = (accB & 3u) | ((nbB & 3u) << 2);
        const int d = bv - lane, e = bv + 2 * count1 - lane;
        int jlo = d <= 0 ? 0 : (d + 31) >> 5, jhi = e <= 0 ? 0 : min(9, (e + 31) >> 5);
        if ((lane - bv) & 1) { jlo = 0; jhi = 0; }
        const int n_in = max(0, jhi - jlo), ja = min(jlo, 8), jb = min(jhi, 8);
        const uint32_t ma = (jb >= 8 ? 0xFFFFFFFFu : (1u << (4 * jb)) - 1u) & ~(ja >= 8 ? 0xFFFFFFFFu : (1u << (4 * ja)) - 1u);
        const uint32_t w = idxA & ma, w8 = (jlo <= 8 && jhi == 9) ? idxB : 0u;
        uint32_t c1s = T.c1cost[w & 0xFFu] + T.c1cost[(w >> 8) & 0xFFu] + T.c1cost[(w >> 16) & 0xFFu] + T.c1cost[w >> 24] + T.c1cost[w8];
        c1s -= (uint32_t)(10 - n_in) * (1u | 4u << 16);   // ten patterns were looked up; the empty ones cost 1 | 4 bits each
        c1s = __reduce_add_sync(FULL, c1s);
        if ((c1s & 0xFFFF) < (c1s >> 16)) { c1sel = 0; c1bits = (int)(c1s & 0xFFFF); }
        else { c1sel = 1; c1bits = (int)(c1s >> 16); }
    }
    // ---- subdivide (:998-1036); with big_values == 0 the addresses keep their old values (A.E6)
    int a1 = (int)(lla & 1023u), a2 = (int)((lla >> 10) & 1023u), a3 = (int)((lla >> 20) & 1023u), r0 = 0, r1 = 0;
    const bool uses_addr = bv == 0 && count1 > 0;
    if (uses_addr && !lhave) return false;
    if (bv != 0) {
        const uint32_t sd = T.subdiv[bv];
        r0 = (int)(sd & 15u); r1 = (int)((sd >> 4) & 15u); a1 = (int)((sd >> 8) & 1023u); a2 = (int)((sd >> 18) & 1023u); a3 = 2 * bv;
    }
    // ---- pooled region sums over pairs [0, a1/2) [a1/2, a2/2) [a2/2, bv)   (:1147-1168, :294-318); per lane a region holds at
    //      most 9 pairs of code length <= 19, so the four books' sums travel as the four bytes of the table word
    uint32_t A0 = 0, A1 = 0, A2 = 0, C0 = 0, C1 = 0, C2 = 0, m0 = 0, m1 = 0, m2 = 0;
    {
        const int h1 = a1 >> 1, h2 = a2 >> 1;          // region bounds are even (scalefactor band edges)
        const int pend = max(bv, max(h1, h2));
#pragma unroll
        for (int j = 0; j < 9; j++) {
            if (32 * j >= pend) break;   // warp-uniform: no pair of this row or a later one lies in a region
            const int p = 32 * j + lane;
            const uint2 w2 = T.hlc[(M[j] >> 16) & 0xFFu];
            const bool p0 = p < h1, p1 = !p0 && p < h2, p2 = !p0 && !p1 && p < bv;
            A0 += p0 ? w2.x : 0u; C0 += p0 ? w2.y : 0u; m0 = max(m0, p0 ? X[j] : 0u);
            A1 += p1 ? w2.x : 0u; C1 += p1 ? w2.y : 0u; m1 = max(m1, p1 ? X[j] : 0u);
            A2 += p2 ? w2.x : 0u; C2 += p2 ? w2.y : 0u; m2 = max(m2, p2 ? X[j] : 0u);
        }
    }
    // lanes 0..2 end up with the totals of region `lane`: every lane contributes to all three reductions
    uint32_t lo = 0, hi = 0, cn = 0, mx = 0;
    {
        const uint32_t l0 = __reduce_add_sync(FULL, A0 & 0x00FF00FFu), h0 = __reduce_add_sync(FULL, (A0 >> 8) & 0x00FF00FFu);
        const uint32_t l1 = __reduce_add_sync(FULL, A1 & 0x00FF00FFu), h1_ = __reduce_add_sync(FULL, (A1 >> 8) & 0x00FF00FFu);
        const uint32_t l2 = __reduce_add_sync(FULL, A2 & 0x00FF00FFu), h2_ = __reduce_add_sync(FULL, (A2 >> 8) & 0x00FF00FFu);
        const uint32_t c0 = __reduce_add_sync(FULL, C0), c1 = __reduce_add_sync(FULL, C1), c2 = __reduce_add_sync(FULL, C2);
        const uint32_t x0 = __reduce_max_sync(FULL, m0), x1 = __reduce_max_sync(FULL, m1), x2 = __reduce_max_sync(FULL, m2);
        const int r = lane == 0 ? 0 : (lane == 1 ? 1 : 2);
        lo = r == 0 ? l0 : (r == 1 ? l1 : l2); hi = r == 0 ? h0 : (r == 1 ? h1_ : h2_);
        cn = r == 0 ? c0 : (r == 1 ? c1 : c2); mx = (r == 0 ? x0 : (r == 1 ? x1 : x2)) & 0xFFFFu;
    }
    // ---- new_choose_table (:1170-1264) before the swap, and the cost of the region under the choice and under either swap
    {
        const int r = lane == 0 ? 0 : (lane == 1 ? 1 : 2);
        const bool exists = r == 0 ? a1 > 0 : (r == 1 ? a2 > a1 : 2 * bv > a2);
        // count_bit() (:215-263) of the four code books the search can reach, from the pooled sums
        const int nsign = (int)(cn & 0xFFFFu), n15 = (int)(cn >> 16);
        const int c13 = (int)(lo & 0xFFFFu) + nsign, c15 = (int)(hi & 0xFFFFu) + nsign, b16 = (int)(lo >> 16) + nsign, b24 = (int)(hi >> 16) + nsign;
        auto cost_of = [&](int t) {   // linbits is zero below table 16: one select chain, no branch
            const int base = t == 0 ? 0 : (t == 13 ? c13 : (t == 15 ? c15 : (t < 24 ? b16 : b24)));
            return base + (int)T.linbits[t] * n15;
        };
        int ch0 = 0;
        if (exists && mx != 0) {
            if (mx < 15) {
                ch0 = c15 <= c13 ? 15 : 13;   // the count-down search always stops at 13 (A.E4); only its 13-vs-15 arm is live
            } else {
                // first table of 15..23 / 24..31 whose lin_max covers mx - 15: a function of the bit length of mx - 15 (<= 13 bits)
                const int nb = 32 - __clz((int)mx - 15);
                const int c0 = 15 + (int)((0x88877665543210ULL >> (4 * nb)) & 15);
                const int c1 = 24 + (int)((0x77665432100000ULL >> (4 * nb)) & 15);
                ch0 = cost_of(c1) < cost_of(c0) ? c1 : c0;
            }
        }
        const int t0 = T.pair[ch0][0], t1 = T.pair[ch0][1];
        const uint32_t nz = __ballot_sync(FULL, ch0 > 0);
        if (lane < 3) {
            R.cost[r][0] = (uint16_t)cost_of(ch0);
            R.cost[r][1] = (uint16_t)cost_of(t0);
            R.cost[r][2] = (uint16_t)cost_of(t1);
            R.tab[r][0] = (uint8_t)ch0; R.tab[r][1] = (uint8_t)t0; R.tab[r][2] = (uint8_t)t1;
        }
        if (lane == 0) {
            R.c1bits = c1bits;
            R.geo = (uint32_t)bv | (uint32_t)count1 << 9 | (uint32_t)c1sel << 17 | (uint32_t)r0 << 18 | (uint32_t)r1 << 22 | (nz & 3u) << 25;
            R.addr = (uint32_t)a1 | (uint32_t)a2 << 10 | (uint32_t)a3 << 20;
            R.tag = uses_addr ? lla : VAR_NONE;
        }
    }
    __syncwarp();
    {   // the two decisions the step search can take on this probe, for every variant at once (lane = variant)
        int m0, m1, m2;
        const int b = row_bits(R, vhn, vhb, m0, m1, m2);
        const uint32_t lt = __ballot_sync(FULL, b < max_bits), le = __ballot_sync(FULL, b <= max_bits);
        if (lane == 0) { R.lt = lt; R.le = le; }
    }
    __syncwarp();
    return true;
}

__global__ void __launch_bounds__(32 * PROBE_WARPS, 2)
k_enc_probe(const M3sEncClip *__restrict__ clips, const int32_t *__restrict__ frame_clip, const M3sDevTables *__restrict__ DT,
            const EncTables *__restrict__ ET, const uint32_t *__restrict__ byteoff, int sr_idx, int64_t g_begin, int64_t g_end,
            const int32_t *__restrict__ mdct, const M3sEncStats *__restrict__ stats, uint4 *__restrict__ var,
            uint32_t *__restrict__ sum, uint8_t *__restrict__ scfsi_out)
{   // granule slots [g_begin, g_end) of the chunk: the frames of the clips at sample rate sr_idx (their tables are per CTA)
    extern __shared__ __align__(16) unsigned char smem_raw[];
    ProbeSmem &PS = *reinterpret_cast<ProbeSmem *>(smem_raw);
    ProbeTab &T = PS.T;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t FULL = 0xFFFFFFFFu;
    ProbeWarpSmem &W = PS.W[warp];
    for (int i = tid; i < 10000; i += 32 * PROBE_WARPS) T.i2x[i] = i2x_entry((uint32_t)DT->int2idx[i]);
    for (int i = tid; i < 256; i += 32 * PROBE_WARPS) {
        const uint32_t x = i >> 4, y = i & 15;
        T.hlc[i] = make_uint2(ET->hl4[i], (uint32_t)(x != 0) + (uint32_t)(y != 0) + (((uint32_t)(x > 14) + (uint32_t)(y > 14)) << 16));
    }
    for (int i = tid; i < 128; i += 32 * PROBE_WARPS) { T.steptabi[i] = DT->steptabi[i]; T.steptab[i] = DT->steptab[i]; }
    if (tid < 24) T.sfb[tid] = tid < 23 ? DT->sfb_long[sr_idx][tid] : 576;
    if (tid < 32) { T.linbits[tid] = DT->enc_linbits[tid]; T.pair[tid][0] = DT->pair[tid][0]; T.pair[tid][1] = DT->pair[tid][1]; }
    if (tid < 23) { T.subdv[tid][0] = DT->subdv[tid][0]; T.subdv[tid][1] = DT->subdv[tid][1]; }
    for (int i = tid; i < 256; i += 32 * PROBE_WARPS) {
        uint32_t v = 0;
        for (int h = 0; h < 2; h++) {
            const uint32_t idx = (i >> (4 * h)) & 15u, nn = __popc(idx);
            // code lengths: table A = {1,4,4,5,4,6,5,6,4,5,5,6,5,6,6,6} (one nibble each), table B = 4 everywhere
            v += ((uint32_t)((0x6665655465645441ULL >> (4 * idx)) & 15) + nn) | ((4u + nn) << 16);
        }
        T.c1cost[i] = v;
    }
    __syncthreads();
    for (int bvv = tid; bvv < 289; bvv += 32 * PROBE_WARPS) {   // subdivide (:998-1036) for every big_values
        uint32_t v = 0;
        if (bvv > 0) {
            const int bvr = 2 * bvv;
            int anz = 0;
            while ((int)T.sfb[anz] < bvr) anz++;
            int tc = T.subdv[anz][0];
            while (tc > 0 && (int)T.sfb[tc + 1] > bvr) tc--;
            const int r0 = tc, a1 = T.sfb[tc + 1], base = tc + 1;
            tc = T.subdv[anz][1];
            while (tc > 0 && (int)T.sfb[min(base + tc + 1, 23)] > bvr) tc--;
            v = (uint32_t)r0 | (uint32_t)tc << 4 | (uint32_t)a1 << 8 | (uint32_t)T.sfb[min(base + tc + 1, 23)] << 18;
        }
        T.subdiv[bvv] = v;
    }
    __syncthreads();
    int vhn;
    uint32_t vhb;
    variant_bits(lane, vhn, vhb);
    // one tile of PROBE_WARPS * PROBE_G granules per CTA: warp w takes granules w, w + PROBE_WARPS, ... of tile blockIdx.x
#pragma unroll 1
    for (int it = 0; it < PROBE_G; it++) {
        const int64_t gs = g_begin + (int64_t)blockIdx.x * (PROBE_WARPS * PROBE_G) + warp + it * PROBE_WARPS;
        if (gs >= g_end) break;
        const int64_t fl_ = gs >> 2;
        const int q = (int)(gs & 3);                         // position in the reference's order: (ch0,gr0) (ch0,gr1) (ch1,gr0) (ch1,gr1)
        const int c = frame_clip[fl_];
        const int64_t payload_len = clips[c].payload_len;
        const int f = (int)(fl_ - clips[c].frame_base);      // frame index inside the clip
        int padding, mean_bits;
        const int max_bits = frame_max_bits(byteoff, clips[c], f, padding, mean_bits);
        const int32_t xrmax = stats[gs].xrmax;
        if (q & 1) {
            // ---- calc_scfsi (:862-892) of this channel: needs the statistics of both granules
            const M3sEncStats *s0 = stats + gs - 1, *s1 = stats + gs;
            const int d = lane < 21 ? abs((int)s0->en[lane] - (int)s1->en[lane]) : 0;
            const int tp = __reduce_add_sync(FULL, d);
            int condition = 2 + (s0->xrmax != 0) + (s1->xrmax != 0);
            if (abs((int)s0->en_tot - (int)s1->en_tot) < 10) condition++;
            if (tp < 100) condition++;
            const int b0 = __reduce_add_sync(FULL, lane < 6 ? d : 0), b1 = __reduce_add_sync(FULL, lane >= 6 && lane < 11 ? d : 0);
            const int b2 = __reduce_add_sync(FULL, lane >= 11 && lane < 16 ? d : 0), b3 = __reduce_add_sync(FULL, lane >= 16 ? d : 0);
            if (lane < 4) {
                const int sum0 = lane == 0 ? b0 : (lane == 1 ? b1 : (lane == 2 ? b2 : b3));
                scfsi_out[(fl_ * 2 + (q >> 1)) * 4 + lane] = (condition == 6 && sum0 < 10) ? 1 : 0;   // xm[] is all zero: sum1 = 0
            }
        }
        if (!xrmax) {
            if (lane == 0) sum[gs] = VAR_SILENT;
            continue;
        }
        uint32_t ax[9], ay[9], sg;
        load_granule(mdct + gs * 576, lane, ax, ay, sg);
        // which variants can occur: the offset in front of this granule is at most 3 bits per earlier granule of the clip
        const bool hiding = payload_len > 0;
        const bool sure3 = payload_len - 3 * (4 * (int64_t)f + q) >= 3;
        __syncwarp();   // the previous granule's lanes have finished reading this warp's rows and slot map
        ((uint32_t *)W.slotmap)[lane] = 0xFFFFFFFFu;
        // quantize(step) > 8192 holds exactly for the steps below s_min (the quantised maximum shrinks as the step grows)
        int s_min = -120;
        if (quant_overflows(T, xrmax, -120)) {
            int n = 0;
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const int st = -120 + 32 * k + lane;
                n += __popc(__ballot_sync(FULL, st <= 0 && quant_overflows(T, xrmax, st)));
            }
            s_min = -120 + n;
        }
        __syncwarp();
        // ---- bin_search_step_size (:958-996) then inner_loop (:1064-1095).  The variants nearly always take the same decisions, so
        //      the walk runs ONCE, warp-uniform, on the per-probe decision masks, for as long as the active variants agree ...
        const uint32_t act = hiding ? (sure3 ? 0xFFu : 0x7FFFu) : 0x4000u;
        int next = -120, count = 120, step = 0, s = 0, nslots = 0, have = 0;
        uint32_t la = 0;
        bool in_bin = true, slow = false, diverged = false, overrun = false;
        for (;;) {
            int half = 0, nstep = step;
            bool ovf = false;
            if (in_bin) {
                half = count / 2;
                s = next + half;
                ovf = s < s_min;
            } else {
                nstep = max(step, s_min - 1) + 1;   // while quantize(step + 1) > 8192: step += 1; then step += 1
                if (nstep > 0) { overrun = true; break; }   // the step table ends at step 0
                s = nstep;
            }
            uint32_t lt = 0, le = 0, geo = 0, addr = 0;   // an overflowing probe counts 100000 bits: neither < nor <= max_bits
            if (!ovf) {
                int slot = W.slotmap[s + 120];
                if (slot == 0xFF) {
                    if (nslots == PROBE_CACHE) { slow = true; break; }
                    if (!probe_row(T, ax, ay, xrmax, s, lane, have, la, max_bits, vhn, vhb, W.row[nslots])) { slow = true; break; }
                    slot = nslots++;
                    if (lane == 0) W.slotmap[s + 120] = (uint8_t)slot;
                    __syncwarp();
                }
                const ProbeRow &R = W.row[slot];
                if (R.tag != VAR_NONE && (!have || R.tag != la)) { slow = true; break; }   // a revisited probe pooled over older addresses
                lt = R.lt & act; le = R.le & act; geo = R.geo; addr = R.addr;
            }
            if (in_bin) {
                if (lt == act) count = half;
                else if (lt == 0) { next += half; count -= half; }
                else { diverged = true; break; }
                if (geo & 0x1FFu) { have = 1; la = addr; }
                if (count <= 1) { in_bin = false; step = next; }
            } else {
                if (le != act && le != 0) { diverged = true; break; }
                step = nstep;
                if (geo & 0x1FFu) { have = 1; la = addr; }
                if (le == act) break;
            }
        }
        // ---- ... and per lane from the first probe on which they disagree (that probe is taken again, lane by lane)
        if (diverged && !slow) {
            bool done = !((act >> lane) & 1u), lane_over = false;
            for (;;) {
                int half = 0;
                bool ovf = false;
                if (!done) {
                    if (in_bin) {
                        half = count / 2;
                        s = next + half;
                        ovf = s < s_min;
                    } else {
                        step = max(step, s_min - 1) + 1;
                        s = step;
                        if (step > 0) { lane_over = true; done = true; }   // the step table ends at step 0
                    }
                }
                // every step some lane needs and the cache lacks is probed once, by the whole warp
                for (;;) {
                    const bool need = !done && !ovf && W.slotmap[s + 120] == 0xFF;
                    const uint32_t m = __ballot_sync(FULL, need);
                    if (!m) break;
                    if (nslots == PROBE_CACHE) { slow = true; break; }
                    const int ldr = __ffs(m) - 1;
                    const int sc = __shfl_sync(FULL, s, ldr);
                    // a probe that finds big_values == 0 among non-zero values pools over the addresses of the latest probe with big
                    // values (A.E6): the requesting lane's own, if its walk has met one in this granule -- else the slot's stale ones
                    const int lhave = __shfl_sync(FULL, have, ldr);
                    const uint32_t lla = __shfl_sync(FULL, la, ldr);
                    if (!probe_row(T, ax, ay, xrmax, sc, lane, lhave, lla, max_bits, vhn, vhb, W.row[nslots])) { slow = true; break; }
                    if (lane == 0) W.slotmap[sc + 120] = (uint8_t)nslots;
                    nslots++;
                    __syncwarp();
                }
                if (slow) break;
                bool stray = false;
                if (!done) {
                    int bits = 100000;
                    if (!ovf) {
                        const ProbeRow &R = W.row[W.slotmap[s + 120]];
                        const uint32_t tag = R.tag;
                        stray = tag != VAR_NONE && (!have || tag != la);   // pooled over another walk's addresses
                        int m0, m1, m2;
                        bits = row_bits(R, vhn, vhb, m0, m1, m2);
                        if (R.geo & 0x1FFu) { have = 1; la = R.addr; }
                    }
                    if (in_bin) {
                        if (bits < max_bits) count = half;
                        else { next += half; count -= half; }
                        if (count <= 1) { in_bin = false; step = next; }
                    } else if (bits <= max_bits) done = true;
                }
                if (__any_sync(FULL, stray)) { slow = true; break; }
                if (__all_sync(FULL, done)) break;
            }
            overrun = __any_sync(FULL, lane_over);
        }
        if (slow || overrun) {
            if (lane == 0) sum[gs] = slow ? VAR_SLOW : VAR_OVERRUN;
            continue;
        }
        uint32_t cntw = 0;
        if ((act >> lane) & 1u) {   // the last probe of the walk is the accepted one: its row, under this variant's modes
            const ProbeRow &R = W.row[W.slotmap[s + 120]];
            const uint32_t geo = R.geo;
            int mode0, mode1, mode2;
            const int bits = row_bits(R, vhn, vhb, mode0, mode1, mode2);
            const int ts0 = R.tab[0][mode0], ts1 = R.tab[1][mode1], ts2 = R.tab[2][mode2];
            const int cnt = (ts0 > 0) + (ts1 > 0) + (ts2 > 0);   // :808-809
            cntw = (uint32_t)cnt << (2 * lane);
            uint4 r;
            r.x = (uint32_t)bits | (geo & 0x1FFu) << 12 | ((geo >> 9) & 0xFFu) << 21 | ((geo >> 17) & 1u) << 29;
            r.y = (uint32_t)(step + 128) | (uint32_t)ts0 << 8 | (uint32_t)ts1 << 13 | (uint32_t)ts2 << 18 | ((geo >> 18) & 15u) << 23 |
                  ((geo >> 22) & 7u) << 27 | (uint32_t)have << 30;
            r.z = la;
            r.w = 0u;
            var[gs * 16 + lane] = r;
        }
        cntw = __reduce_or_sync(FULL, cntw);
        if (lane == 0) sum[gs] = cntw;
    }
}


// The reference's own sequential search for ONE granule with the true state (the slow path of k_enc_resolve).
// Returns false, with step 0 and an empty granule, when the search would quantise at a step above 0 (steptabi[128], past the
// end of the table: the reference has no defined output there, SURVEY A.E13).
__device__ __noinline__ bool search_granule(const RateSmem &S, const int32_t *__restrict__ mdct_g, int32_t xrmax, int max_bits, int hn,
                                            uint32_t hb, int lane, int &a1, int &a2, int &a3, int &step, GranInfo &gi, int &part23)
{
    uint32_t ax[9], ay[9], qx[9], qy[9], sg;
    load_granule(mdct_g, lane, ax, ay, sg);
    gi.bv = 0; gi.count1 = 0; gi.c1sel = 0; gi.r0 = 0; gi.r1 = 0; gi.ts0 = 0; gi.ts1 = 0; gi.ts2 = 0;
    int next = -120, count = 120, half = 0, bits = 0, s = 0;
    bool in_bin = true;
    for (;;) {
        bool ovf = false;
        if (in_bin) {
            half = count / 2;
            s = next + half;
            ovf = quant_max(S, xrmax, s) > 8192;
        } else {
            while (step < 0 && quant_max(S, xrmax, step + 1) > 8192) step++;
            if (step >= 0) {
                gi.bv = 0; gi.count1 = 0; gi.c1sel = 0; gi.r0 = 0; gi.r1 = 0; gi.ts0 = 0; gi.ts1 = 0; gi.ts2 = 0;
                step = 0;
                part23 = 0;
                return false;
            }
            step++;
            s = step;
        }
        bits = 100000;
        if (!ovf) {
            Pooled P;
            quantize_all(S, ax, ay, s, qx, qy);
            probe_pool(S, qx, qy, lane, a1, a2, a3, P);
            a1 = P.a1; a2 = P.a2; a3 = P.a3;
            bits = probe_tables(S, P, true, hn, hb, gi);
        }
        if (in_bin) {
            if (bits < max_bits) count = half;
            else { next += half; count -= half; }
            if (count <= 1) { in_bin = false; step = next; }
        } else if (bits <= max_bits) break;
    }
    part23 = bits;
    return true;
}

// "latest value at or before my lane among the lanes of my slot" (lanes 4 apart), VAR_NONE where a lane has nothing to say
__device__ __forceinline__ uint32_t slot_scan(uint32_t v, int lane)
{
#pragma unroll
    for (int d = 4; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, v, d);
        if (lane >= d && v == VAR_NONE) v = t;
    }
    return v;
}

#define RESOLVE_WARPS 2
__global__ void __launch_bounds__(32 * RESOLVE_WARPS)
k_enc_resolve(const M3sEncClip *__restrict__ clips, int c_begin, int c_end, M3sEncState *__restrict__ states, const M3sDevTables *__restrict__ T,
              const EncTables *__restrict__ ET, const uint32_t *__restrict__ byteoff, const uint8_t *__restrict__ payload, int sr_idx,
              int32_t chunk_first, int32_t chunk_frames, const int32_t *__restrict__ mdct,
              const M3sEncStats *__restrict__ stats, const uint4 *__restrict__ var, uint32_t *__restrict__ sum, int32_t *__restrict__ info)
{   // clips [c_begin, c_end): the clips at sample rate sr_idx
    extern __shared__ __align__(16) unsigned char smem_raw[];
    RateSmem &S = *reinterpret_cast<RateSmem *>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t FULL = 0xFFFFFFFFu;
    rate_tables_load(S, T, ET, tid, 32 * RESOLVE_WARPS);
    if (tid < 24) S.sfb[tid] = tid < 23 ? T->sfb_long[sr_idx][tid] : 576;
    __syncthreads();
    const int c = c_begin + blockIdx.x * RESOLVE_WARPS + warp;
    if (c >= c_end) return;
    const M3sEncClip cl = clips[c];
    const int f_end = min(cl.n_frames, chunk_first + chunk_frames);
    if (f_end <= chunk_first) return;
    const int ng = 4 * (f_end - chunk_first);
    const bool hiding = cl.payload_len > 0;
    M3sEncState *sp = states + c;
    int64_t off = sp->hide_off;
    const int q = lane & 3, slot = 2 * (q & 1) + (q >> 1);   // my position in the reference's order; the (gr, ch) slot it belongs to
    // carried slot state, replicated in every lane of the slot
    uint32_t car_a = (uint32_t)sp->a1[slot] | (uint32_t)sp->a2[slot] << 10 | (uint32_t)sp->a3[slot] << 20;
    uint32_t car_step = (uint32_t)(sp->step[slot] + 128);    // steps travel as step + 128 (8..128) so that none collides with VAR_NONE
    uint32_t car_src = (uint32_t)sp->src[slot];
    int32_t overrun = sp->overrun;
#pragma unroll 1
    for (int gb = 0; gb < ng; gb += 32) {
        const int i = gb + lane;
        const bool valid = i < ng;
        const int f = chunk_first + (i >> 2);
        const int64_t fl_ = cl.frame_base + f;
        const int64_t gs = fl_ * 4 + q;
        const uint32_t wsum = valid ? sum[gs] : VAR_SILENT;
        // payload window: the 128 chars from `off` on (a batch consumes at most 96)
        const int64_t woff = off;
        uint32_t w0 = 0, w1 = 0, w2 = 0, w3 = 0;
        if (hiding) {
            const uint8_t *pp = payload + cl.payload_base;
            const int64_t i0 = woff + lane;
            w0 = __ballot_sync(FULL, i0 < cl.payload_len && __ldg(pp + i0) == '1');
            w1 = __ballot_sync(FULL, i0 + 32 < cl.payload_len && __ldg(pp + i0 + 32) == '1');
            w2 = __ballot_sync(FULL, i0 + 64 < cl.payload_len && __ldg(pp + i0 + 64) == '1');
            w3 = __ballot_sync(FULL, i0 + 96 < cl.payload_len && __ldg(pp + i0 + 96) == '1');
        }
        auto bits_at = [&](int64_t o, int &hn, uint32_t &hb) {
            const int64_t left = cl.payload_len - o;
            hn = !hiding ? 0 : (left > 3 ? 3 : (left < 0 ? 0 : (int)left));
            const int rel = (int)(o - woff), k = rel >> 5;
            const uint32_t lo = k == 0 ? w0 : (k == 1 ? w1 : (k == 2 ? w2 : w3));
            const uint32_t hi = k == 0 ? w1 : (k == 1 ? w2 : (k == 2 ? w3 : 0u));
            hb = __funnelshift_r(lo, hi, rel & 31) & ((1u << hn) - 1u);
        };
        // per-lane results of my granule
        int r_p23 = 0, r_bv = 0, r_c1 = 0, r_c1sel = 0, r_ts0 = 0, r_ts1 = 0, r_ts2 = 0, r_r0 = 0, r_r1 = 0, r_cnt = 0;
        uint32_t r_a = 0, r_step = 0, r_src = 0;
        int64_t my_off = 0;
        int i0 = 0;
        while (i0 < 32) {
            // ---- sequential part: offset -> variant -> bits consumed, registers only
            int my_v = 14, stop = 32;
#pragma unroll 1
            for (int j = i0; j < 32; j++) {
                const uint32_t ws = __shfl_sync(FULL, wsum, j);
                if (ws & VAR_SLOW) { stop = j; break; }
                int v = 14, cnt = 0;
                if (!(ws & VAR_SILENT)) {
                    int hn;
                    uint32_t hb;
                    bits_at(off, hn, hb);
                    v = variant_index(hn, hb);
                    cnt = (int)((ws >> (2 * v)) & 3u);
                }
                if (lane == j) { my_v = v; my_off = off; r_cnt = cnt; }
                off += cnt;
            }
            // ---- parallel part: lanes [i0, stop) fetch the chosen variant's record
            const bool mine = lane >= i0 && lane < stop && valid;
            const bool live = mine && !(wsum & VAR_SILENT);
            uint32_t va = VAR_NONE, vs = VAR_NONE, vsrc = VAR_NONE;
            if (live) {
                const uint4 r = var[gs * 16 + my_v];
                r_p23 = (int)(r.x & 0xFFFu); r_bv = (int)((r.x >> 12) & 0x1FFu); r_c1 = (int)((r.x >> 21) & 0xFFu); r_c1sel = (int)((r.x >> 29) & 1u);
                vs = r.y & 0xFFu;
                r_ts0 = (int)((r.y >> 8) & 31u); r_ts1 = (int)((r.y >> 13) & 31u); r_ts2 = (int)((r.y >> 18) & 31u);
                r_r0 = (int)((r.y >> 23) & 15u); r_r1 = (int)((r.y >> 27) & 7u);
                if ((r.y >> 30) & 1u) va = r.z;
                vsrc = (uint32_t)(f + 1);
            }
            va = slot_scan(va, lane); vs = slot_scan(vs, lane); vsrc = slot_scan(vsrc, lane);
            if (va == VAR_NONE) va = car_a;
            if (vs == VAR_NONE) vs = car_step;
            if (vsrc == VAR_NONE) vsrc = car_src;
            if (mine) { r_a = va; r_step = vs; r_src = vsrc; }
            car_a = __shfl_sync(FULL, va, 28 + q); car_step = __shfl_sync(FULL, vs, 28 + q); car_src = __shfl_sync(FULL, vsrc, 28 + q);
            if (stop == 32) break;
            // ---- granule `stop` depends on the slot's stale addresses: the reference's own search with the true state
            {
                const int j = stop, jq = j & 3;
                const uint32_t sa = __shfl_sync(FULL, car_a, jq);
                int a1 = (int)(sa & 1023u), a2 = (int)((sa >> 10) & 1023u), a3 = (int)((sa >> 20) & 1023u);
                int step = (int)__shfl_sync(FULL, car_step, jq) - 128;
                const int fj = chunk_first + ((gb + j) >> 2);
                const int64_t gsj = (cl.frame_base + fj) * 4 + jq;
                int padding, mean_bits, hn, part23 = 0;
                uint32_t hb;
                const int max_bits = frame_max_bits(byteoff, cl, fj, padding, mean_bits);
                bits_at(off, hn, hb);
                GranInfo gi;
                if (!search_granule(S, mdct + gsj * 576, stats[gsj].xrmax, max_bits, hn, hb, lane, a1, a2, a3, step, gi, part23) && !overrun)
                    overrun = fj + 1;
                const int cnt = (gi.ts0 > 0) + (gi.ts1 > 0) + (gi.ts2 > 0);
                const uint32_t na = (uint32_t)a1 | (uint32_t)a2 << 10 | (uint32_t)a3 << 20;
                if (lane == j) {
                    my_off = off; r_cnt = cnt; r_p23 = part23; r_bv = gi.bv; r_c1 = gi.count1; r_c1sel = gi.c1sel;
                    r_ts0 = gi.ts0; r_ts1 = gi.ts1; r_ts2 = gi.ts2; r_r0 = gi.r0; r_r1 = gi.r1;
                    r_a = na; r_step = (uint32_t)(step + 128); r_src = (uint32_t)(fj + 1);
                }
                if (q == jq) { car_a = na; car_step = (uint32_t)(step + 128); car_src = (uint32_t)(fj + 1); }
                off += cnt;
                i0 = j + 1;
            }
        }
        // ---- per frame (4 lanes): resv_frame_end (:1097-1145) -- every unused bit of the frame becomes stuffing -- and the records
        {
            int padding = 0, mean_bits = 0;
            if (valid) frame_max_bits(byteoff, cl, f, padding, mean_bits);
            const int base = lane & ~3;
            // part2_3_length in the order gr0ch0, gr0ch1, gr1ch0, gr1ch1 = my positions 0, 2, 1, 3
            int p23[4];
            p23[0] = __shfl_sync(FULL, r_p23, base); p23[1] = __shfl_sync(FULL, r_p23, base + 2);
            p23[2] = __shfl_sync(FULL, r_p23, base + 1); p23[3] = __shfl_sync(FULL, r_p23, base + 3);
            const int64_t off_after = __shfl_sync(FULL, my_off + r_cnt, base + 3);
            int stuffing = 0;
#pragma unroll
            for (int k = 0; k < 4; k++) stuffing += mean_bits / 2 - p23[k];   // :812 (mean_bits is even)
            if (stuffing > 0) {
                if (p23[0] + stuffing < 4095) p23[0] += stuffing;
                else {
#pragma unroll
                    for (int k = 0; k < 4; k++) {
                        const int t = min(4095 - p23[k], max(stuffing, 0));
                        p23[k] += t;
                        stuffing -= t;
                    }
                }
            }
            if (valid) {
                const int mine23 = slot == 0 ? p23[0] : (slot == 1 ? p23[1] : (slot == 2 ? p23[2] : p23[3]));
                const int step = (int)r_step - 128;
                int4 *r = (int4 *)(info + (fl_ * 4 + slot) * ENC_INFO_FIELDS);
                r[0] = make_int4(mine23, r_bv, r_c1, step + 210);
                r[1] = make_int4(r_ts0, r_ts1, r_ts2, r_r0);
                r[2] = make_int4(r_r1, r_c1sel, (int)(r_a & 1023u), (int)((r_a >> 10) & 1023u));
                r[3] = make_int4((int)((r_a >> 20) & 1023u), step, padding, (int)off_after);
                sum[gs] = r_src;   // the summary word has been consumed: the emit kernel finds the source frame of a silent granule here
            }
        }
    }
    // ---- hand the state to the next chunk
    if (lane < 4) {
        sp->a1[slot] = (int32_t)(car_a & 1023u); sp->a2[slot] = (int32_t)((car_a >> 10) & 1023u); sp->a3[slot] = (int32_t)((car_a >> 20) & 1023u);
        sp->step[slot] = (int32_t)car_step - 128;
        sp->src[slot] = (int32_t)car_src;
        if (lane == 0) { sp->hide_off = off; sp->overrun = overrun; }
    }
}

// ================================================================================================
// E2 for many payloads: k_enc_offsets (m3s_encode_offsets).  hide_str_offset of up to 32 candidate payloads of ONE clip per warp,
// lane = candidate, against the one probe pass of the clip: per granule every lane reads the same summary word, takes the <= 3
// bits at its own offset, and adds the count of its variant.  It writes nothing but the candidates' carried state: `sum` and
// `var` are read by every warp of the clip.
// ================================================================================================
struct M3sOffCand {        // candidate payload: the MSB-first bits of head[0 .. head_len) followed by body[body_base .. body_base + body_len)
    int64_t body_base;     // first body byte in the call's body buffer
    int64_t nbits;         // 8 * (head_len + body_len)
    int32_t head_base;     // first head byte in the call's head buffer
    int32_t head_len;      // <= 32
};
struct M3sOffWork {        // one warp: candidates [cand_first, cand_first + count) of library clip `clip`, count <= 32
    int32_t clip;
    int32_t count;
    int64_t cand_first;
};

#define OFFSETS_WARPS 2
__global__ void __launch_bounds__(32 * OFFSETS_WARPS)
k_enc_offsets(const M3sEncClip *__restrict__ clips, const M3sOffWork *__restrict__ work, int w_begin, int w_end,
              const M3sOffCand *__restrict__ cands, const uint8_t *__restrict__ head, const uint8_t *__restrict__ body,
              M3sEncState *__restrict__ states, const M3sDevTables *__restrict__ T, const EncTables *__restrict__ ET,
              const uint32_t *__restrict__ byteoff, int sr_idx, int32_t chunk_first, int32_t chunk_frames,
              const int32_t *__restrict__ mdct, const M3sEncStats *__restrict__ stats, const uint4 *__restrict__ var,
              const uint32_t *__restrict__ sum)
{   // work items [w_begin, w_end): the candidates of the clips at sample rate sr_idx
    extern __shared__ __align__(16) unsigned char smem_raw[];
    RateSmem &S = *reinterpret_cast<RateSmem *>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t FULL = 0xFFFFFFFFu;
    rate_tables_load(S, T, ET, tid, 32 * OFFSETS_WARPS);
    if (tid < 24) S.sfb[tid] = tid < 23 ? T->sfb_long[sr_idx][tid] : 576;
    __syncthreads();
    const int w = w_begin + blockIdx.x * OFFSETS_WARPS + warp;
    if (w >= w_end) return;
    const M3sOffWork wk = work[w];
    const M3sEncClip cl = clips[wk.clip];
    const int f_end = min(cl.n_frames, chunk_first + chunk_frames);
    if (f_end <= chunk_first) return;
    const bool mine = lane < wk.count;
    const int64_t ci = wk.cand_first + (mine ? lane : 0);
    const M3sOffCand cd = cands[ci];
    M3sEncState *sp = states + ci;
    int64_t off = sp->hide_off;
    uint32_t car_a[4];
    int car_step[4];
#pragma unroll
    for (int s = 0; s < 4; s++) {
        car_a[s] = (uint32_t)sp->a1[s] | (uint32_t)sp->a2[s] << 10 | (uint32_t)sp->a3[s] << 20;
        car_step[s] = sp->step[s];
    }
    int32_t overrun = sp->overrun;
    // the payload bits [wbase, wbase + 64) MSB first; a granule reads 3 bits at `off`, so the window moves every ~20 granules
    const int64_t nbytes = cd.nbits >> 3;
    uint64_t win = 0;
    int64_t wbase = INT64_MIN / 2;
    auto bits_at = [&](int64_t o, int &hn, uint32_t &hb) {   // hb bit j = payload bit o + j, as k_enc_resolve's payload window
        const int64_t left = cd.nbits - o;
        hn = left > 3 ? 3 : (left < 0 ? 0 : (int)left);
        hb = 0u;
        if (hn == 0) return;
        if (o + 3 > wbase + 64) {
            wbase = o & ~(int64_t)7;
            win = 0;
#pragma unroll 1
            for (int b = 0; b < 8; b++) {
                const int64_t k = (wbase >> 3) + b;
                const uint32_t v = k >= nbytes ? 0u : (k < cd.head_len ? __ldg(head + cd.head_base + k) : __ldg(body + cd.body_base + k - cd.head_len));
                win |= (uint64_t)v << (56 - 8 * b);
            }
        }
        const int rel = (int)(o - wbase);
        const uint32_t top = (uint32_t)(win >> (61 - rel)) & 7u;   // bits rel, rel + 1, rel + 2 as b0 b1 b2 (MSB first)
        hb = (((top >> 2) & 1u) | (top & 2u) | ((top & 1u) << 2)) & ((1u << hn) - 1u);
    };
#pragma unroll 1
    for (int f = chunk_first; f < f_end; f++) {
        const int64_t fl_ = cl.frame_base + f;
        const uint4 ws4 = *(const uint4 *)(sum + fl_ * 4);   // the frame's four summary words, the same for every lane
#pragma unroll
        for (int q = 0; q < 4; q++) {   // the reference's order (ch0,gr0) (ch0,gr1) (ch1,gr0) (ch1,gr1); slot = 2 gr + ch
            const int slot = 2 * (q & 1) + (q >> 1);
            const int64_t gs = fl_ * 4 + q;
            const uint32_t ws = q == 0 ? ws4.x : (q == 1 ? ws4.y : (q == 2 ? ws4.z : ws4.w));
            int hn;
            uint32_t hb;
            if (ws & VAR_SLOW) {
                // the probe could not settle this granule (stale addresses, or the step table's end): the reference's search with each
                // lane's true state, served one lane at a time by the whole warp
                bits_at(off, hn, hb);
                int padding, mean_bits;
                const int max_bits = frame_max_bits(byteoff, cl, f, padding, mean_bits);
                const int32_t xrmax = stats[gs].xrmax;
                uint32_t new_a = car_a[slot];
                int new_step = car_step[slot], cnt = 0;
                bool over = false;
                for (uint32_t pend = __ballot_sync(FULL, mine); pend; pend &= pend - 1) {
                    const int src = __ffs(pend) - 1;
                    const uint32_t sa = __shfl_sync(FULL, car_a[slot], src);
                    int step = __shfl_sync(FULL, car_step[slot], src);
                    const int lhn = __shfl_sync(FULL, hn, src);
                    const uint32_t lhb = __shfl_sync(FULL, hb, src);
                    int a1 = (int)(sa & 1023u), a2 = (int)((sa >> 10) & 1023u), a3 = (int)((sa >> 20) & 1023u), part23 = 0;
                    GranInfo gi;
                    const bool ok = search_granule(S, mdct + gs * 576, xrmax, max_bits, lhn, lhb, lane, a1, a2, a3, step, gi, part23);
                    if (lane == src) {
                        new_a = (uint32_t)a1 | (uint32_t)a2 << 10 | (uint32_t)a3 << 20;
                        new_step = step;
                        cnt = (gi.ts0 > 0) + (gi.ts1 > 0) + (gi.ts2 > 0);
                        over = !ok;
                    }
                }
                car_a[slot] = new_a;
                car_step[slot] = new_step;
                if (over && !overrun) overrun = f + 1;
                off += cnt;
            } else if (!(ws & VAR_SILENT)) {
                bits_at(off, hn, hb);
                const int v = variant_index(hn, hb);
                off += (ws >> (2 * v)) & 3u;
                const uint4 r = var[gs * 16 + v];   // k_enc_probe's record of the variant: .y = step + 128 | ... | have << 30, .z = addresses
                car_step[slot] = (int)(r.y & 0xFFu) - 128;
                if ((r.y >> 30) & 1u) car_a[slot] = r.z;
            }
        }
    }
    if (mine) {
#pragma unroll
        for (int s = 0; s < 4; s++) {
            sp->a1[s] = (int32_t)(car_a[s] & 1023u); sp->a2[s] = (int32_t)((car_a[s] >> 10) & 1023u); sp->a3[s] = (int32_t)((car_a[s] >> 20) & 1023u);
            sp->step[s] = car_step[s];
        }
        sp->hide_off = off;
        sp->overrun = overrun;
    }
}

// One warp per granule-channel: quantise at the chosen step and write the signed values format_bitstream codes (:1272-1276).
// A silent granule keeps what l3_enc held for its slot (never coded: big_values = count1 = 0): the values of the latest
// non-silent granule of the slot, re-derived from that granule's spectra, or read from `last_in` when it lies in an earlier chunk.
#define EMIT_WARPS 8
#define EMIT_G 8
__global__ void __launch_bounds__(32 * EMIT_WARPS, 3)
k_enc_emit(const M3sEncClip *__restrict__ clips, const int32_t *__restrict__ frame_clip, const M3sDevTables *__restrict__ T,
           const EncTables *__restrict__ ET, int32_t chunk_first, int32_t chunk_frames, int64_t n_gran,
           const int32_t *__restrict__ mdct, const M3sEncStats *__restrict__ stats, const uint32_t *__restrict__ srcs,
           const int32_t *__restrict__ info, uint32_t *__restrict__ ixout, const uint32_t *__restrict__ last_in,
           uint32_t *__restrict__ last_out)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    RateSmem &S = *reinterpret_cast<RateSmem *>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    rate_tables_load(S, T, ET, tid, 32 * EMIT_WARPS);
    __syncthreads();
    const int64_t g0 = (int64_t)blockIdx.x * (EMIT_WARPS * EMIT_G) + warp;
#pragma unroll 1
    for (int it = 0; it < EMIT_G; it++) {
        const int64_t gs = g0 + (int64_t)it * EMIT_WARPS;
        if (gs >= n_gran) break;
        const int64_t fl_ = gs >> 2;
        const int q = (int)(gs & 3), slot = 2 * (q & 1) + (q >> 1);
        const int c = frame_clip[fl_];
        const int f = (int)(fl_ - clips[c].frame_base);
        const int n_frames = clips[c].n_frames;
        const int src = (int)srcs[gs] - 1;                   // clip frame whose values this slot holds (-1: none yet)
        uint32_t out[9];
        if (src < 0) {
#pragma unroll
            for (int j = 0; j < 9; j++) out[j] = 0u;
        } else if (src < chunk_first) {
            const uint32_t *lp = last_in + ((int64_t)c * 4 + q) * 288;
#pragma unroll
            for (int j = 0; j < 9; j++) out[j] = lp[32 * j + lane];
        } else {
            const int64_t back = f - src;                    // 0 for a granule that was coded itself
            const int step = info[((fl_ - back) * 4 + slot) * ENC_INFO_FIELDS + 13];
            uint32_t ax[9], ay[9], qx[9], qy[9], sg;
            load_granule(mdct + (gs - 4 * back) * 576, lane, ax, ay, sg);
            quantize_all(S, ax, ay, step, qx, qy);
#pragma unroll
            for (int j = 0; j < 9; j++) {
                const int vx = ((sg >> (2 * j)) & 1u) ? -(int)qx[j] : (int)qx[j];
                const int vy = ((sg >> (2 * j + 1)) & 1u) ? -(int)qy[j] : (int)qy[j];
                out[j] = ((uint32_t)vx & 0xFFFFu) | ((uint32_t)vy << 16);
            }
        }
        uint32_t *ixd = ixout + gs * 288;
#pragma unroll
        for (int j = 0; j < 9; j++) ixd[32 * j + lane] = out[j];
        const int f_end = min(n_frames, chunk_first + chunk_frames);
        if (f == f_end - 1 && f_end < n_frames) {            // what the slot holds when the next chunk starts
            uint32_t *lp = last_out + ((int64_t)c * 4 + q) * 288;
#pragma unroll
            for (int j = 0; j < 9; j++) lp[32 * j + lane] = out[j];
        }
    }
}

// ================================================================================================
// E3: bit packing, one warp per frame
// ================================================================================================
#define PACK_WARPS 2
#define PACK_WORDS 364   // >= 1441 bytes (320 kbps at 32 kHz, padded)

struct PackSmem {
    uint32_t code[1410];
    uint16_t hoff[34];
    uint8_t linbits[34];
    uint16_t sfb[3][24];     // per sample rate: the two warps of a CTA may pack frames of clips at different rates
    uint32_t frame[PACK_WARPS][PACK_WORDS];
    uint32_t ix[PACK_WARPS][288];
};

// append `n` (<= 32) bits of `v` at bit position `pos` of a big-endian word buffer (bit 0 = MSB of word 0)
__device__ __forceinline__ void put_bits_at(uint32_t *buf, int pos, uint32_t v, int n)
{
    if (n == 0) return;
    const int w = pos >> 5, o = pos & 31;
    const uint64_t x = ((uint64_t)(n < 32 ? (v & ((1u << n) - 1u)) : v)) << (64 - n - o);
    atomicOr(&buf[w], (uint32_t)(x >> 32));
    if ((uint32_t)x) atomicOr(&buf[w + 1], (uint32_t)x);
}

__global__ void __launch_bounds__(32 * PACK_WARPS)
k_enc_pack(const M3sEncClip *__restrict__ clips, const int32_t *__restrict__ frame_clip, const M3sDevTables *__restrict__ T,
           const uint32_t *__restrict__ byteoff, int64_t chunk_frame0, int64_t chunk_total_frames, const uint32_t *__restrict__ ixin,
           const int32_t *__restrict__ info, const uint8_t *__restrict__ scfsi, uint8_t *__restrict__ out)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    PackSmem &S = *reinterpret_cast<PackSmem *>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t FULL = 0xFFFFFFFFu;
    for (int i = tid; i < 1410; i += 32 * PACK_WARPS) S.code[i] = T->enc_hpacked[i];
    if (tid < 34) { S.hoff[tid] = T->enc_hoff[tid]; S.linbits[tid] = T->enc_linbits[tid]; }
    for (int i = tid; i < 3 * 24; i += 32 * PACK_WARPS) S.sfb[i / 24][i % 24] = i % 24 < 23 ? T->sfb_long[i / 24][i % 24] : 576;
    __syncthreads();
    const int64_t fl_ = (int64_t)blockIdx.x * PACK_WARPS + warp;
    if (fl_ >= chunk_total_frames) return;
    const int c = frame_clip[fl_];
    const M3sEncClip cl = clips[c];
    const int f = (int)(chunk_frame0 + fl_ - cl.frame_base);
    const uint32_t *bo = byteoff + cl.pad_base;
    const uint16_t *sfb = S.sfb[cl.sr_idx];
    const int fbytes = (int)(bo[f + 1] - bo[f]);
    const int padding = fbytes - cl.whole_slots;
    uint32_t *buf = S.frame[warp];
    for (int i = lane; i < PACK_WORDS; i += 32) buf[i] = 0u;
    __syncwarp();
    const int32_t *inf = info + fl_ * 4 * ENC_INFO_FIELDS;
    // ---- header + side info: 288 bits = words 0..8   (:1281-1337)
    if (lane == 0) {
        int pos = 0;
        auto put = [&](uint32_t v, int n) { put_bits_at(buf, pos, v, n); pos += n; };
        put(0x7ff, 11); put(3, 2); put(1, 2); put(1, 1); put((uint32_t)cl.bitrate_idx, 4); put((uint32_t)cl.sr_idx, 2);
        put((uint32_t)padding, 1); put(0, 1); put(0, 2); put(0, 2); put(0, 1); put(1, 1); put(0, 2);
        put(0, 9); put(0, 3);
        for (int ch = 0; ch < 2; ch++)
            for (int b = 0; b < 4; b++) put(scfsi[(fl_ * 2 + ch) * 4 + b], 1);
        for (int gr = 0; gr < 2; gr++)
            for (int ch = 0; ch < 2; ch++) {
                const int32_t *r = inf + (2 * gr + ch) * ENC_INFO_FIELDS;
                put((uint32_t)r[0], 12); put((uint32_t)r[1], 9); put((uint32_t)r[3], 8); put(0, 4); put(0, 1);
                put((uint32_t)r[4], 5); put((uint32_t)r[5], 5); put((uint32_t)r[6], 5); put((uint32_t)r[7], 4); put((uint32_t)r[8], 3);
                put(0, 1); put(0, 1); put((uint32_t)r[9], 1);
            }
    }
    // ---- main data: (gr0,ch0) (gr0,ch1) (gr1,ch0) (gr1,ch1), each exactly part2_3_length bits   (:1339-1446)
    int start = 288;
    for (int gr = 0; gr < 2; gr++)
        for (int ch = 0; ch < 2; ch++) {
            const int32_t *r = inf + (2 * gr + ch) * ENC_INFO_FIELDS;
            const int part23 = r[0], bv = r[1], count1 = r[2], ts[3] = {r[4], r[5], r[6]}, c1sel = r[9];
            const int r1 = sfb[r[7] + 1], r2 = sfb[min(r[7] + 1 + r[8] + 1, 23)];
            const uint32_t *src = ixin + ((fl_ * 2 + ch) * 2 + gr) * 288;
            uint32_t *ix = S.ix[warp];
            for (int j = 0; j < 9; j++) ix[32 * j + lane] = __ldg(src + 32 * j + lane);
            __syncwarp();
            int pos = start;
            // big values: pair p carries code(+signs) or code, linbits, signs   (:1448-1513)
            for (int j = 0; j < 9; j++) {
                const int p = 32 * j + lane;
                uint64_t bitsv = 0;
                int nb = 0;
                if (p < bv) {
                    const int e = 2 * p;
                    const int t = ts[(e >= r1) + (e >= r2)];
                    if (t) {
                        const uint32_t wv = ix[p];
                        int x = (int)(int16_t)(wv & 0xFFFFu), y = (int)(int16_t)(wv >> 16);
                        const uint32_t sx = x > 0 ? 0u : 1u, sy = y > 0 ? 0u : 1u;
                        x = x < 0 ? -x : x;
                        y = y < 0 ? -y : y;
                        if (t > 15) {
                            const int lin = S.linbits[t];
                            uint32_t ext = 0;
                            int xbits = 0, lbx = 0, lby = 0;
                            if (x > 14) { lbx = x - 15; x = 15; }
                            if (y > 14) { lby = y - 15; y = 15; }
                            const uint32_t cw = S.code[S.hoff[t] + x * 16 + y];
                            if (x > 14) { ext |= (uint32_t)lbx; xbits += lin; }
                            if (x != 0) { ext = (ext << 1) | sx; xbits += 1; }
                            if (y > 14) { ext = (ext << lin) | (uint32_t)lby; xbits += lin; }
                            if (y != 0) { ext = (ext << 1) | sy; xbits += 1; }
                            bitsv = ((uint64_t)(cw >> 8) << xbits) | ext;
                            nb = (int)(cw & 0xFF) + xbits;
                        } else {
                            const int dim = t < 2 ? 2 : (t < 4 ? 3 : (t < 7 ? 4 : (t < 10 ? 6 : (t < 13 ? 8 : 16))));
                            const uint32_t cw = S.code[S.hoff[t] + x * dim + y];
                            uint32_t code = cw >> 8;
                            nb = (int)(cw & 0xFF);
                            if (x != 0) { code = (code << 1) | sx; nb++; }
                            if (y != 0) { code = (code << 1) | sy; nb++; }
                            bitsv = code;
                        }
                    }
                }
                int inc = nb;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const int v = __shfl_up_sync(FULL, inc, d);
                    if (lane >= d) inc += v;
                }
                const int at = pos + inc - nb;
                if (nb > 32) { put_bits_at(buf, at, (uint32_t)(bitsv >> 32), nb - 32); put_bits_at(buf, at + nb - 32, (uint32_t)bitsv, 32); }
                else put_bits_at(buf, at, (uint32_t)bitsv, nb);
                pos += __shfl_sync(FULL, inc, 31);
                if (32 * (j + 1) >= bv) break;
            }
            // count1 quads (:1515-1547): p = v + 2 w + 4 x + 8 y on magnitudes, then the signs of the non-zero ones
            for (int m0 = 0; m0 < count1; m0 += 32) {
                const int m = m0 + lane;
                uint32_t code = 0;
                int nb = 0;
                if (m < count1) {
                    const uint32_t w0 = ix[bv + 2 * m], w1 = ix[bv + 2 * m + 1];
                    int q[4] = {(int)(int16_t)(w0 & 0xFFFFu), (int)(int16_t)(w0 >> 16), (int)(int16_t)(w1 & 0xFFFFu), (int)(int16_t)(w1 >> 16)};
                    uint32_t sgn = 0, idx = 0;
                    int ns = 0;
#pragma unroll
                    for (int z = 0; z < 4; z++) {
                        const int a = q[z] < 0 ? -q[z] : q[z];
                        idx |= (uint32_t)(a & 1) << z;   // magnitudes are 0 or 1 in the count1 region
                        if (a) { sgn = (sgn << 1) | (q[z] > 0 ? 0u : 1u); ns++; }
                    }
                    const uint32_t cw = S.code[S.hoff[32 + c1sel] + idx];
                    code = ((cw >> 8) << ns) | sgn;
                    nb = (int)(cw & 0xFF) + ns;
                }
                int inc = nb;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const int v = __shfl_up_sync(FULL, inc, d);
                    if (lane >= d) inc += v;
                }
                put_bits_at(buf, pos + inc - nb, code, nb);
                pos += __shfl_sync(FULL, inc, 31);
            }
            // stuffing with one-bits up to part2_3_length (:1433-1446)
            const int end = start + part23;
            for (int b = pos + 32 * lane; b < end; b += 32 * 32) put_bits_at(buf, b, 0xFFFFFFFFu, min(32, end - b));
            start = end;
            __syncwarp();
        }
    __syncwarp();
    // ---- copy out, clipped to what the reference's word-granular writer emits for the whole clip (A.E8)
    const int64_t fo = bo[f];
    const uint8_t *bb = (const uint8_t *)buf;
    for (int i = lane; i < fbytes; i += 32)
        if (fo + i < cl.out_len) out[cl.out_base + fo + i] = bb[i ^ 3];   // big-endian words -> byte stream
}

// ================================================================================================
// host orchestration
// ================================================================================================
// clip index of every chunk-local frame slot (what the per-granule / per-frame kernels of E2 / E3 map a slot back with), written on
// the device: the host only sends one (first slot, count) pair per clip and chunk instead of one entry per frame
__global__ void __launch_bounds__(128)
k_enc_frame_clip(const int64_t *__restrict__ first, const int32_t *__restrict__ count, int n_clips, int32_t *__restrict__ frame_clip)
{
    const int64_t f0 = first[blockIdx.x];
    const int n = count[blockIdx.x], clip = (int)(blockIdx.x % (unsigned)n_clips);
    for (int q = threadIdx.x; q < n; q += 128) frame_clip[f0 + q] = clip;
}

static const int kBitrates[16] = {-1, 32, 40, 48, 56, 64, 80, 96, 112, 128, 160, 192, 224, 256, 320, -1};

static int sr_index_of(int sr) { return sr == 44100 ? 0 : sr == 48000 ? 1 : sr == 32000 ? 2 : -1; }
static int br_index_of(int br)
{
    for (int i = 1; i < 15; i++)
        if (kBitrates[i] == br) return i;
    return -1;
}

// byte offset of every frame of a clip: whole_slots + padding, padding from the reference's float64 slot-lag recurrence (:504-513, :630-632)
static void padding_prefix(int sample_rate, int bitrate_kbps, int64_t n_frames, std::vector<uint32_t> &off, int &whole)
{
    const double avg = (2.0 * 576 / (double)sample_rate) * (1000 * (double)bitrate_kbps / 8.0);
    whole = (int)avg;
    const double frac = avg - (double)whole;
    double slot_lag = -frac;
    off.assign((size_t)n_frames + 1, 0u);
    int padding = 0;
    for (int64_t f = 0; f < n_frames; f++) {
        if (frac != 0) {
            padding = slot_lag <= (frac - 1.0) ? 1 : 0;
            slot_lag += padding - frac;
        }
        off[f + 1] = off[f] + (uint32_t)(whole + padding);
    }
}

extern "C" int64_t m3s_encode_bound(int64_t n_samples, int32_t sample_rate, int32_t bitrate_kbps)
{
    if (n_samples < 0 || sample_rate <= 0) return -1;
    int64_t frames = (n_samples + 1151) / 1152;
    int64_t fs = (144000LL * bitrate_kbps) / sample_rate + 1;
    return frames * fs + 8;
}

extern "C" int64_t m3s_encode_size(int64_t n_samples, int32_t sample_rate, int32_t bitrate_kbps)
{
    if (n_samples < 0 || n_samples % 1152 || sr_index_of(sample_rate) < 0 || br_index_of(bitrate_kbps) < 0) return -1;
    std::vector<uint32_t> off;
    int whole = 0;
    padding_prefix(sample_rate, bitrate_kbps, n_samples / 1152, off, whole);
    return (int64_t)(off.back() / 4) * 4;
}

static void build_enc_tables(const M3sDevTables *T, EncTables *E)
{
    memset(E, 0, sizeof *E);
    const int books[4] = {13, 15, 16, 24};
    for (int i = 0; i < 256; i++) {
        uint32_t w = 0;
        for (int b = 0; b < 4; b++) w |= (T->enc_hpacked[T->enc_hoff[books[b]] + i] & 0xFFu) << (8 * b);
        E->hl4[i] = w;
    }
    for (int i = 0; i < 16; i++) {
        E->hlc1[0][i] = (uint8_t)(T->enc_hpacked[T->enc_hoff[32] + i] & 0xFF);
        E->hlc1[1][i] = (uint8_t)(T->enc_hpacked[T->enc_hoff[33] + i] & 0xFF);
    }
    // en(temp) = (int32)(log(temp * 4.768371584e-7) / 0.69314718) is monotone in temp: tabulate where it steps (host libm,
    // the same one the reference's numbers come from) so that the device needs no log at all
    auto en_of = [](uint32_t temp) { return (int)(log((double)temp * 4.768371584e-7) / 0.69314718); };
    for (int j = 0; j < 32; j++) {
        const int target = j - 20;
        uint32_t lo = 1, hi = 0x7FFFFFFFu;
        if (en_of(hi) < target) { E->en_thresh[j] = 0xFFFFFFFFu; continue; }
        while (lo < hi) {
            const uint32_t mid = lo + (hi - lo) / 2;
            if (en_of(mid) >= target) hi = mid;
            else lo = mid + 1;
        }
        E->en_thresh[j] = lo;
    }
}

// The candidate payloads of m3s_encode_offsets (see the header).
struct EncOffsets {
    const uint8_t *body;
    const int64_t *body_off, *cand_off;
    const uint8_t *head;
    const int64_t *head_off, *body_len;
};

// The clip arguments every encode entry point takes (see the header), with one rate pair per clip.
struct EncClips {
    const int16_t *pcm;
    int mem;
    const int64_t *pcm_off, *n_samples;
    int32_t n_clips;
    const int32_t *sample_rate, *bitrate_kbps;
};

#define M3S_ENC_MARK(tag) do { if (m3s_trace) { const double t__ = m3s_now_ms(); fprintf(stderr, "[m3s enc] %-22s +%.2f ms\n", tag, t__ - tr_t); tr_t = t__; } } while (0)

// The checks every entry point starts with; `outputs`: the entry point's own required pointers are set.
static int check_call(m3s_ctx *h, const EncClips &a, bool outputs)
{
    if (!h) return M3S_ERR_ARG;
    h->enc_taps_ok = false;
    if (!a.pcm || !a.n_samples || a.n_clips <= 0 || !a.sample_rate || !a.bitrate_kbps || !outputs)
        return m3s_fail(h, M3S_ERR_ARG, "encode: null argument");
    if ((uintptr_t)a.pcm & 3) return m3s_fail(h, M3S_ERR_ARG, "encode: pcm must be 4-byte aligned (one stereo sample per word)");
    return M3S_OK;
}

// The checks of caller clip j, run by every entry point in the caller's order before anything is queued.
static int check_clip(m3s_ctx *h, const EncClips &a, int j)
{
    if (sr_index_of(a.sample_rate[j]) < 0) return m3s_fail(h, M3S_ERR_ARG, "encode: clip %d: sample rate %d is not an MPEG-1 rate", j, a.sample_rate[j]);
    if (br_index_of(a.bitrate_kbps[j]) < 0)
        return m3s_fail(h, M3S_ERR_ARG, "encode: clip %d: bitrate %d is not an MPEG-1 Layer III rate (WAV_Reader.py:112-114)", j, a.bitrate_kbps[j]);
    if (a.n_samples[j] < 0 || a.n_samples[j] % 1152) return m3s_fail(h, M3S_ERR_ARG, "encode: clip %d has %lld samples per channel, not a multiple of 1152 (the reference raises IndexError, MP3_Encoder.py:611-614)", j, (long long)a.n_samples[j]);
    if (a.pcm_off && (a.pcm_off[j] & 1)) return m3s_fail(h, M3S_ERR_ARG, "encode: pcm_off must be even (stereo samples)");
    return M3S_OK;
}

// The host-side layout of a call.  The library's clip order groups the clips by sample rate (stable), so that in every chunk the
// frame slots of one sample rate are contiguous and the kernels that stage per-rate tables once per CTA (probe, resolve) run once
// per group.  Clip i of that order is the caller's clip order[i]; every output goes back by the caller's index.
struct EncLayout {
    std::vector<int> order, inv;
    int grp[4];                      // clips of sample rate index s: [grp[s], grp[s + 1])
    std::vector<M3sEncClip> clips;   // in the library's order; the payload and output fields are the entry point's to fill
    std::vector<uint32_t> byteoff;   // the padding tables
    int64_t total_frames = 0, max_frames = 0;
    // chunking: all clips advance together through windows of `cf` frames so that the intermediates (MDCT spectra 9.2 KB/frame,
    // quantised values 4.6 KB/frame) stay bounded while every clip keeps its warp busy; chunk_cap = frame slots of the fullest chunk
    int64_t cf = 0, n_chunks = 0, chunk_cap = 0;
};

static int enc_layout(m3s_ctx *h, const EncClips &a, EncLayout &L)
{
    const int n_clips = a.n_clips;
    L.order.resize(n_clips);
    L.inv.resize(n_clips);
    for (int i = 0; i < n_clips; i++) L.order[i] = i;
    std::stable_sort(L.order.begin(), L.order.end(), [&](int x, int y) { return sr_index_of(a.sample_rate[x]) < sr_index_of(a.sample_rate[y]); });
    for (int i = 0; i < n_clips; i++) L.inv[L.order[i]] = i;
    for (int s = 0, i = 0; s < 4; s++) {
        while (s < 3 && i < n_clips && sr_index_of(a.sample_rate[L.order[i]]) < s) i++;
        L.grp[s] = s < 3 ? i : n_clips;
    }
    // ---- clip table
    L.clips.resize(n_clips);
    for (int i = 0; i < n_clips; i++) {
        const int j = L.order[i];
        M3sEncClip &c = L.clips[i];
        c.pcm_base = a.pcm_off ? a.pcm_off[j] : 0;
        c.n_frames = (int32_t)(a.n_samples[j] / 1152);
        c.frame_base = L.total_frames;
        c.sr_idx = (int16_t)sr_index_of(a.sample_rate[j]);
        c.bitrate_idx = (int16_t)br_index_of(a.bitrate_kbps[j]);
        L.total_frames += c.n_frames;
        L.max_frames = std::max<int64_t>(L.max_frames, c.n_frames);
    }
    if (!a.pcm_off) {   // back to back in the caller's order
        int64_t e = 0;
        for (int j = 0; j < n_clips; j++) { L.clips[L.inv[j]].pcm_base = e; e += 2 * a.n_samples[j]; }
    }
    // ---- padding tables: one per rate pair of the batch, sized to its longest clip, back to back
    int64_t pair_frames[3][16];
    for (auto &r : pair_frames) for (int64_t &v : r) v = -1;
    for (const M3sEncClip &c : L.clips) pair_frames[c.sr_idx][c.bitrate_idx] = std::max<int64_t>(pair_frames[c.sr_idx][c.bitrate_idx], c.n_frames);
    static const int kRates[3] = {44100, 48000, 32000};
    std::vector<uint32_t> tab;
    int pair_base[3][16] = {}, pair_whole[3][16] = {};
    for (int s = 0; s < 3; s++)
        for (int b = 1; b < 15; b++) {
            if (pair_frames[s][b] < 0) continue;
            padding_prefix(kRates[s], kBitrates[b], pair_frames[s][b], tab, pair_whole[s][b]);
            if (L.byteoff.size() + tab.size() > (size_t)INT32_MAX) return m3s_fail(h, M3S_ERR_ARG, "encode: too many frames in one call");
            pair_base[s][b] = (int)L.byteoff.size();
            L.byteoff.insert(L.byteoff.end(), tab.begin(), tab.end());
        }
    for (M3sEncClip &c : L.clips) {
        c.pad_base = pair_base[c.sr_idx][c.bitrate_idx];
        c.whole_slots = pair_whole[c.sr_idx][c.bitrate_idx];
        c.out_len = (int64_t)(L.byteoff[(size_t)c.pad_base + c.n_frames] / 4) * 4;
    }
    if (L.max_frames == 0) return M3S_OK;   // nothing to encode, no chunk
    // host buffers: smaller chunks, because nothing runs before the first chunk's PCM has crossed PCIe (measured: 10.1 -> 10.5 M frames/s e2e)
    const int64_t budget_frames = h->enc_chunk_budget > 0 ? h->enc_chunk_budget : (a.mem == M3S_MEM_HOST ? (1 << 17) : (1 << 19));
    L.cf = std::min(std::max<int64_t>(1, budget_frames / n_clips), L.max_frames);
    for (const M3sEncClip &c : L.clips) L.chunk_cap += std::min<int64_t>(L.cf, c.n_frames);
    L.n_chunks = (L.max_frames + L.cf - 1) / L.cf;
    return M3S_OK;
}

// What the kernels that follow the probe read in chunk k: frames [c0, c0 + cf) of every clip.
struct EncChunk {
    int64_t k, c0, slots;        // slots: the chunk's frame slots
    const M3sEncClip *clips;     // chunk-local clip records (device)
    const int32_t *frame_clip;   // clip index of every frame slot of the chunk (device)
    const int64_t *grp_slot;     // frame slots of sample rate index s: [grp_slot[s], grp_slot[s + 1])
    const M3sEncSet &set;        // the chunk's intermediates
};

// Runs every chunk of a call: analysis, probe, then `after_probe` on the main stream.  With host buffers the PCM is staged in and,
// when mp3_out is given, each chunk's MP3 bytes go back to it from e_out.  The carried states start at zero; `states` receives them.
static int enc_pipeline(m3s_ctx *h, const EncClips &a, const EncLayout &L, std::vector<M3sEncState> &states, uint8_t *mp3_out,
                        double tr_t, const std::function<int(const EncChunk &)> &after_probe)
{
    int rc;
    const int n_clips = a.n_clips;
    const std::vector<M3sEncClip> &clips = L.clips;
    const int64_t cf = L.cf, n_chunks = L.n_chunks;
    // ---- encoder constant tables (once per handle)
    if (!h->e_tabs.p) {
        std::vector<uint8_t> hostT(sizeof(M3sDevTables));
        M3S_CUDA(h, cudaMemcpy(hostT.data(), h->d_tab, sizeof(M3sDevTables), cudaMemcpyDeviceToHost));
        EncTables E;
        build_enc_tables((const M3sDevTables *)hostT.data(), &E);
        if ((rc = m3s_buf_reserve(h, h->e_tabs, sizeof(EncTables)))) return rc;
        M3S_CUDA(h, cudaMemcpy(h->e_tabs.p, &E, sizeof E, cudaMemcpyHostToDevice));
        M3S_CUDA(h, cudaMemcpyToSymbol(c_enc_cos, ((const M3sDevTables *)hostT.data())->enc_cosl, sizeof(int32_t) * 18 * 36));
        M3S_CUDA(h, cudaMemcpyToSymbol(c_enc_fl, ((const M3sDevTables *)hostT.data())->enc_fl, sizeof(int32_t) * 32 * 64));
        M3S_CUDA(h, cudaMemcpyToSymbol(c_enc_win, ((const M3sDevTables *)hostT.data())->enwindow, sizeof(int32_t) * 512));
    }
    // ---- inputs.  Host buffers are streamed: the PCM of chunk k+1 crosses PCIe on `copy_in` while chunk k is in the
    //      kernels, and the MP3 bytes of chunk k-1 go back on `copy_out` (see the chunk loop below)
    const bool host = a.mem == M3S_MEM_HOST;
    if ((rc = m3s_pipeline_init(h))) return rc;
    if ((rc = m3s_buf_reserve(h, h->e_pad, sizeof(uint32_t) * L.byteoff.size()))) return rc;
    M3S_CUDA(h, cudaMemcpyAsync(h->e_pad.p, L.byteoff.data(), sizeof(uint32_t) * L.byteoff.size(), cudaMemcpyHostToDevice, h->stream));
    if ((rc = m3s_buf_reserve(h, h->e_state, sizeof(M3sEncState) * states.size()))) return rc;
    M3S_CUDA(h, cudaMemsetAsync(h->e_state.p, 0, sizeof(M3sEncState) * states.size(), h->stream));
    const size_t cap = (size_t)L.chunk_cap;
    for (int q = 0; q < (n_chunks > 1 ? 2 : 1); q++) {   // with several chunks, chunk k uses set k & 1
        M3sEncSet &es = h->es[q];
        if ((rc = m3s_buf_reserve(h, es.mdct, cap * 4 * 576 * 4))) return rc;
        if ((rc = m3s_buf_reserve(h, es.gran, cap * 4 * sizeof(M3sEncStats)))) return rc;
        if ((rc = m3s_buf_reserve(h, es.scfsi, cap * 8))) return rc;
        if ((rc = m3s_buf_reserve(h, es.var, cap * 4 * 16 * sizeof(uint4)))) return rc;
        if ((rc = m3s_buf_reserve(h, es.sum, cap * 4 * sizeof(uint32_t)))) return rc;
    }
    M3S_CUDA(h, cudaFuncSetAttribute(k_enc_probe, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ProbeSmem)));
    M3S_CUDA(h, cudaFuncSetAttribute(k_enc_probe, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    M3S_CUDA(h, cudaFuncSetAttribute(k_enc_analysis_fold, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Ana3Smem)));
    M3S_CUDA(h, cudaFuncSetAttribute(k_enc_analysis_fold, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    const int64_t ana_run = Ana3Smem::RUN;   // granules per analysis work item
    auto frames_in_chunk = [&](int i, int64_t c0) { return std::max<int64_t>(0, std::min<int64_t>(cf, clips[i].n_frames - c0)); };
    // host staging: per chunk every clip owns a region of cf * 1152 + 1056 stereo samples (1056 = the analysis history the
    // first granule of the chunk reaches back to: 480 window taps + one warm-up granule), two region sets for double buffering
    const int64_t region = cf * 1152 + 1056;
    const size_t stage_bytes = host ? (size_t)n_clips * (size_t)region * 4 : 0;
    if (host && (rc = m3s_buf_reserve(h, h->e_pcm, 2 * stage_bytes + 16))) return rc;
    M3S_ENC_MARK("buffers");
    std::vector<M3sRow> rows;
    bool free_recorded[2] = {false, false};
    struct ChunkEv { cudaEvent_t c0, c1, a0, a1, r1, p1, o1; };   // M3S_TRACE: copy in, analysis, rate loop, pack, copy out of every chunk
    std::vector<ChunkEv> tev;
    if (m3s_trace) tev.assign((size_t)n_chunks, ChunkEv{});
    auto tmark = [&](cudaEvent_t &e, cudaStream_t st) { if (m3s_trace) { cudaEventCreate(&e); cudaEventRecord(e, st); } };
    auto stage_chunk = [&](int64_t k) -> cudaError_t {   // H2D of the PCM that chunk k reads, into staging set k & 1
        const int64_t c0 = k * cf;
        const int pb = (int)(k & 1);
        rows.clear();
        for (int i = 0; i < n_clips; i++) {
            const int64_t nfc = frames_in_chunk(i, c0);
            if (nfc == 0) continue;
            const int64_t first = c0 * 1152 - 1056, s0 = std::max<int64_t>(first, 0), s1 = (c0 + nfc) * 1152;
            M3sRow r;
            r.dst = (char *)h->e_pcm.p + (size_t)pb * stage_bytes + ((size_t)i * region + (size_t)(s0 - first)) * 4;
            r.src = (const char *)a.pcm + clips[i].pcm_base * 2 + s0 * 4;
            r.bytes = (size_t)(s1 - s0) * 4;
            rows.push_back(r);
        }
        cudaError_t e = cudaSuccess;
        if (free_recorded[pb]) e = cudaStreamWaitEvent(h->copy_in, h->ev_free[pb], 0);
        if (m3s_trace) tmark(tev[k].c0, h->copy_in);
        if (e == cudaSuccess) e = m3s_copy_rows(rows, cudaMemcpyHostToDevice, h->copy_in);
        if (e == cudaSuccess) e = cudaEventRecord(h->ev_in[pb], h->copy_in);
        if (m3s_trace) tmark(tev[k].c1, h->copy_in);
        return e;
    };
    // the first chunk's PCM starts crossing PCIe now, under the host work below (descriptors of every chunk); the descriptors' own
    // upload queues behind it on the copy engine, so the second chunk is staged after them
    if (host) M3S_CUDA(h, stage_chunk(0));
    // ---- descriptors of ALL chunks go up once, so that the chunk loop below issues no small copy (a pageable copy blocks the host
    //      until its stream gets there, which would serialise the streams of the pipeline)
    std::vector<M3sEncWork> work;          // E1 work items, chunk k = [work_off[k], work_off[k+1])
    std::vector<int64_t> fc_first((size_t)n_clips * n_chunks);   // frame slots of clip i in chunk k: [fc_first, fc_first + fc_count) of the
    std::vector<int32_t> fc_count((size_t)n_clips * n_chunks);   // frame_clip array, whose chunk k is [slot_off[k], slot_off[k+1])
    std::vector<M3sEncClip> cclips((size_t)n_clips * n_chunks);   // chunk-local clip records
    std::vector<int64_t> work_off(n_chunks + 1, 0), slot_off(n_chunks + 1, 0);
    std::vector<int64_t> grp_slot((size_t)n_chunks * 4);   // chunk k: the frame slots of sample rate index s are [grp_slot[4k + s], grp_slot[4k + s + 1])
    for (int64_t k = 0; k < n_chunks; k++) {
        const int64_t c0 = k * cf;
        int64_t base = 0;
        for (int i = 0; i < n_clips; i++) {
            for (int s = 0; s < 4; s++)
                if (L.grp[s] == i) grp_slot[(size_t)k * 4 + s] = base;
            const int64_t nfc = frames_in_chunk(i, c0);
            M3sEncClip &cc = cclips[(size_t)k * n_clips + i];
            cc = clips[i];
            // chunk-local frame slot of clip frame f is  base + (f - c0)  ==  (frame_base' + f) - chunk_frame0 with frame_base' = base - c0, chunk_frame0 = 0
            cc.frame_base = base - c0;
            // staged PCM: sample t of the clip sits at  region * i + t - (c0 * 1152 - 1056)  of this chunk's staging set
            if (host) cc.pcm_base = 2 * ((int64_t)i * region - (c0 * 1152 - 1056));
            for (int64_t g = 2 * c0; g < 2 * (c0 + nfc); g += ana_run) {
                M3sEncWork w;
                w.clip = i; w.g_first = (int32_t)g; w.count = (int32_t)std::min<int64_t>(ana_run, 2 * (c0 + nfc) - g);
                w.ch = 0; work.push_back(w);
                w.ch = 1; work.push_back(w);
            }
            fc_first[(size_t)k * n_clips + i] = slot_off[k] + base;
            fc_count[(size_t)k * n_clips + i] = (int32_t)nfc;
            base += nfc;
        }
        for (int s = 0; s < 4; s++)
            if (L.grp[s] == n_clips) grp_slot[(size_t)k * 4 + s] = base;
        work_off[k + 1] = (int64_t)work.size();
        slot_off[k + 1] = slot_off[k] + base;
    }
    M3S_ENC_MARK("descriptors built");
    if ((rc = m3s_buf_reserve(h, h->e_work, sizeof(M3sEncWork) * work.size()))) return rc;
    const size_t fc_bytes = ((size_t)slot_off[n_chunks] * sizeof(int32_t) + 15) / 16 * 16;   // frame_clip, then the (first, count) pairs
    if ((rc = m3s_buf_reserve(h, h->e_misc, fc_bytes + fc_first.size() * 12))) return rc;
    if ((rc = m3s_buf_reserve(h, h->e_clips, sizeof(M3sEncClip) * cclips.size()))) return rc;
    M3S_CUDA(h, cudaMemcpyAsync(h->e_work.p, work.data(), sizeof(M3sEncWork) * work.size(), cudaMemcpyHostToDevice, h->stream));
    M3S_CUDA(h, cudaMemcpyAsync((char *)h->e_misc.p + fc_bytes, fc_first.data(), fc_first.size() * 8, cudaMemcpyHostToDevice, h->stream));
    M3S_CUDA(h, cudaMemcpyAsync((char *)h->e_misc.p + fc_bytes + fc_first.size() * 8, fc_count.data(), fc_count.size() * 4, cudaMemcpyHostToDevice, h->stream));
    M3S_KBEGIN(h, M3S_K_ENC_AUX);
    k_enc_frame_clip<<<(unsigned)fc_first.size(), 128, 0, h->stream>>>((const int64_t *)((char *)h->e_misc.p + fc_bytes),
        (const int32_t *)((char *)h->e_misc.p + fc_bytes + fc_first.size() * 8), n_clips, (int32_t *)h->e_misc.p);
    M3S_LAUNCH_CHECK(h);
    M3S_CUDA(h, cudaMemcpyAsync(h->e_clips.p, cclips.data(), sizeof(M3sEncClip) * cclips.size(), cudaMemcpyHostToDevice, h->stream));
    M3S_CUDA(h, cudaStreamSynchronize(h->stream));   // everything uploaded so far (payload, padding table, state, descriptors) is visible to every stream
    M3S_ENC_MARK("descriptors uploaded");

    // E1 of chunk k on the aux stream; ev_ana[k & 1] = spectra + statistics of the chunk are ready
    auto launch_analysis = [&](int64_t k) -> int {
        const int pb = (int)(k & 1);
        const int64_t nw = work_off[k + 1] - work_off[k];
        if (nw == 0) return M3S_OK;
        const int16_t *k_pcm = a.pcm;
        if (host) {
            k_pcm = (const int16_t *)((const char *)h->e_pcm.p + (size_t)pb * stage_bytes);
            M3S_CUDA(h, cudaStreamWaitEvent(h->aux, h->ev_in[pb], 0));
        }
        // chunk k-2 has left this spectra set (rate loop read it, frames packed).  Waiting for its PACK -- the last kernel in front of
        // the rate loop of chunk k-1 on the main stream -- also lets that rate loop's CTAs take their SM slots first: the analysis
        // then fills what is left instead of crowding the critical chain out
        if (k >= 2) M3S_CUDA(h, cudaStreamWaitEvent(h->aux, h->ev_pack[pb], 0));
        M3sLaunchOn on_aux(h, h->aux);   // timing events of this launch go to the aux stream; restored on every return path
        if (m3s_trace) tmark(tev[k].a0, h->aux);
        M3S_KBEGIN(h, M3S_K_ENC_ANALYSIS);
        k_enc_analysis_fold<<<(unsigned)nw, 32 * ANA3_WARPS, sizeof(Ana3Smem), h->aux>>>(
            k_pcm, (const M3sEncClip *)h->e_clips.p + (size_t)k * n_clips, (const M3sEncWork *)h->e_work.p + work_off[k], h->d_tab,
            (const EncTables *)h->e_tabs.p, 0, (int32_t *)h->es[pb].mdct.p, (M3sEncStats *)h->es[pb].gran.p, 0u);
        M3S_LAUNCH_CHECK(h);
        if (m3s_trace) tmark(tev[k].a1, h->aux);
        M3S_CUDA(h, cudaEventRecord(h->ev_ana[pb], h->aux));
        if (host) {
            M3S_CUDA(h, cudaEventRecord(h->ev_free[pb], h->aux));   // the staging set may be refilled once the analysis has read it
            free_recorded[pb] = true;
        }
        return M3S_OK;
    };
    // ---- software pipeline over the chunks (frames [k cf, (k+1) cf) of every clip); nothing in the loop blocks the host:
    //        copy_in   PCM of chunk k+2                       (host buffers only)
    //        aux       analysis of chunk k+1                  queued behind the packing of chunk k
    //        stream    rate loop + packing of chunk k         the critical path: back to back, chunk after chunk
    //        copy_out  MP3 bytes of chunk k                   (host buffers only)
    //      The probe and resolve kernels stage per-sample-rate tables once per CTA: they run once per sample rate present in the
    //      chunk, over its frame slots / clips.  The other kernels read the rate from the clip record and run once per chunk.
    if (host && n_chunks > 1) M3S_CUDA(h, stage_chunk(1));
    if ((rc = launch_analysis(0))) return rc;
    for (int64_t k = 0; k < n_chunks; k++) {
        const int64_t c0 = k * cf;
        const int pb = (int)(k & 1);
        const int64_t chunk_total = slot_off[k + 1] - slot_off[k];
        if (chunk_total == 0) break;
        const M3sEncSet &es = h->es[pb];
        const EncChunk chunk{k, c0, chunk_total, (const M3sEncClip *)h->e_clips.p + (size_t)k * n_clips,
                             (const int32_t *)h->e_misc.p + slot_off[k], &grp_slot[(size_t)k * 4], es};
        M3S_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_ana[pb], 0));
        for (int s = 0; s < 3; s++) {
            const int64_t g0 = 4 * chunk.grp_slot[s], g1 = 4 * chunk.grp_slot[s + 1];
            if (g1 == g0) continue;
            M3S_KBEGIN(h, M3S_K_ENC_RATE);
            k_enc_probe<<<(unsigned)((g1 - g0 + PROBE_WARPS * PROBE_G - 1) / (PROBE_WARPS * PROBE_G)), 32 * PROBE_WARPS, sizeof(ProbeSmem), h->stream>>>(
                chunk.clips, chunk.frame_clip, h->d_tab, (const EncTables *)h->e_tabs.p, (const uint32_t *)h->e_pad.p,
                s, g0, g1, (const int32_t *)es.mdct.p, (const M3sEncStats *)es.gran.p, (uint4 *)es.var.p,
                (uint32_t *)es.sum.p, (uint8_t *)es.scfsi.p);
            M3S_LAUNCH_CHECK(h);
        }
        if (m3s_trace) tmark(tev[k].r1, h->stream);
        if (host && k + 2 < n_chunks) M3S_CUDA(h, stage_chunk(k + 2));
        if ((rc = after_probe(chunk))) return rc;
        if (m3s_trace) tmark(tev[k].p1, h->stream);
        M3S_CUDA(h, cudaEventRecord(h->ev_pack[pb], h->stream));
        // the rate loop and the analysis are both issue-bound: the next chunk's analysis waits for this chunk's packing (measured:
        // overlapping them gains nothing and stretches the analysis kernel's own time)
        if (k + 1 < n_chunks) {
            M3S_CUDA(h, cudaStreamWaitEvent(h->aux, h->ev_pack[pb], 0));
            if ((rc = launch_analysis(k + 1))) return rc;
        }
        if (host && mp3_out) {   // this chunk's bytes of every clip go home behind the pack kernel
            M3S_CUDA(h, cudaStreamWaitEvent(h->copy_out, h->ev_pack[pb], 0));
            rows.clear();
            for (int i = 0; i < n_clips; i++) {
                const int64_t nfc = frames_in_chunk(i, c0);
                if (nfc == 0) continue;
                const uint32_t *bo = L.byteoff.data() + clips[i].pad_base;
                const int64_t b0 = bo[c0], b1 = std::min<int64_t>(bo[c0 + nfc], clips[i].out_len);
                if (b1 <= b0) continue;
                M3sRow r;
                r.dst = (char *)mp3_out + clips[i].out_base + b0;
                r.src = (const char *)h->e_out.p + clips[i].out_base + b0;
                r.bytes = (size_t)(b1 - b0);
                rows.push_back(r);
            }
            M3S_CUDA(h, m3s_copy_rows(rows, cudaMemcpyDeviceToHost, h->copy_out));
            if (m3s_trace) tmark(tev[k].o1, h->copy_out);
        }
    }
    M3S_ENC_MARK("chunks queued");
    if ((rc = m3s_sync_streams(h))) return rc;
    M3S_ENC_MARK("streams drained");
    if (m3s_trace && host) {   // timeline of the call, ms since the first copy was queued
        auto at = [&](cudaEvent_t e) { float ms = -1.f; if (e) cudaEventElapsedTime(&ms, tev[0].c0, e); return ms; };
        for (int64_t k = 0; k < n_chunks; k++) {
            if (k < 6 || k >= n_chunks - 3)
                fprintf(stderr, "[m3s enc] chunk %3lld  copy_in %7.2f..%7.2f  analysis %7.2f..%7.2f  rate ..%7.2f  pack ..%7.2f  copy_out ..%7.2f\n", (long long)k,
                        at(tev[k].c0), at(tev[k].c1), at(tev[k].a0), at(tev[k].a1), at(tev[k].r1), at(tev[k].p1), at(tev[k].o1));
        }
        for (int64_t k = 0; k < n_chunks; k++)
            for (cudaEvent_t e : {tev[k].c0, tev[k].c1, tev[k].a0, tev[k].a1, tev[k].r1, tev[k].p1, tev[k].o1}) if (e) cudaEventDestroy(e);
    }
    M3S_CUDA(h, cudaMemcpyAsync(states.data(), h->e_state.p, sizeof(M3sEncState) * states.size(), cudaMemcpyDeviceToHost, h->stream));
    M3S_CUDA(h, cudaStreamSynchronize(h->stream));
    return M3S_OK;
}

// An error return may leave work of the call on the handle's streams: they are drained before the caller reuses its buffers.
static int drain_on_error(m3s_ctx *h, int rc)
{
    if (rc != M3S_OK && h) { const std::string keep = h->err; m3s_sync_streams(h); h->err = keep; }
    return rc;
}

// m3s_encode and m3s_encode_mixed: MP3 bytes, out_len and hide_str_offset of every clip
static int encode_mp3(m3s_ctx *h, const EncClips &a, const uint8_t *payload_bits, const int64_t *payload_off, uint8_t *mp3_out,
                      const int64_t *mp3_off, const int64_t *mp3_cap, int64_t *out_len, int64_t *hide_str_offset_out)
{
    double tr_t = m3s_trace ? m3s_now_ms() : 0.0;
    int rc;
    if ((rc = check_call(h, a, mp3_out && mp3_off))) return rc;
    for (int j = 0; j < a.n_clips; j++)
        if ((rc = check_clip(h, a, j))) return rc;
    M3S_CUDA(h, cudaSetDevice(h->device));
    EncLayout L;
    if ((rc = enc_layout(h, a, L))) return rc;
    const int n_clips = a.n_clips;
    int64_t out_total = 0, pay_total = 0;
    for (int j = 0; j < n_clips; j++) {
        M3sEncClip &c = L.clips[L.inv[j]];
        c.out_base = mp3_off[j];
        c.payload_base = payload_bits && payload_off ? payload_off[j] : 0;
        c.payload_len = payload_bits && payload_off ? payload_off[j + 1] - payload_off[j] : 0;
        out_total = std::max(out_total, c.out_base + c.out_len);
        pay_total = std::max(pay_total, c.payload_base + c.payload_len);
        if (mp3_cap && mp3_cap[j] < c.out_len) return m3s_fail(h, M3S_ERR_CAPACITY, "encode: clip %d needs %lld output bytes, capacity %lld", j, (long long)c.out_len, (long long)mp3_cap[j]);
        if (out_len) out_len[j] = c.out_len;
        if (hide_str_offset_out) hide_str_offset_out[j] = 0;
    }
    if (L.total_frames == 0) return M3S_OK;
    M3S_ENC_MARK("clip table");
    uint8_t *d_out = mp3_out;
    if (a.mem == M3S_MEM_HOST) {
        if ((rc = m3s_buf_reserve(h, h->e_out, (size_t)out_total + 16))) return rc;
        d_out = (uint8_t *)h->e_out.p;
    }
    if ((rc = m3s_buf_reserve(h, h->e_payload, (size_t)pay_total + 16))) return rc;
    if (pay_total > 0) M3S_CUDA(h, cudaMemcpyAsync(h->e_payload.p, payload_bits, (size_t)pay_total, cudaMemcpyHostToDevice, h->stream));
    const size_t lastix_bytes = (size_t)n_clips * 4 * 288 * 4;
    if ((rc = m3s_buf_reserve(h, h->e_lastix, 2 * lastix_bytes))) return rc;   // two sets: chunk k reads set k & 1 and writes the other
    for (int q = 0; q < (L.n_chunks > 1 ? 2 : 1); q++) {
        if ((rc = m3s_buf_reserve(h, h->es[q].ix, (size_t)L.chunk_cap * 4 * 288 * 4))) return rc;
        if ((rc = m3s_buf_reserve(h, h->es[q].info, (size_t)L.chunk_cap * 4 * ENC_INFO_FIELDS * 4))) return rc;
    }
    M3S_CUDA(h, cudaFuncSetAttribute(k_enc_resolve, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RateSmem)));
    M3S_CUDA(h, cudaFuncSetAttribute(k_enc_emit, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RateSmem)));
    M3S_CUDA(h, cudaFuncSetAttribute(k_enc_pack, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(PackSmem)));
    std::vector<M3sEncState> states(n_clips);
    rc = enc_pipeline(h, a, L, states, mp3_out, tr_t, [&](const EncChunk &c) -> int {
        const M3sEncSet &es = c.set;
        for (int s = 0; s < 3; s++) {
            if (c.grp_slot[s + 1] == c.grp_slot[s]) continue;   // no clip of this sample rate has a frame in the chunk
            M3S_KBEGIN(h, M3S_K_ENC_RESOLVE);
            k_enc_resolve<<<(unsigned)((L.grp[s + 1] - L.grp[s] + RESOLVE_WARPS - 1) / RESOLVE_WARPS), 32 * RESOLVE_WARPS, sizeof(RateSmem), h->stream>>>(
                c.clips, L.grp[s], L.grp[s + 1], (M3sEncState *)h->e_state.p, h->d_tab, (const EncTables *)h->e_tabs.p, (const uint32_t *)h->e_pad.p,
                (const uint8_t *)h->e_payload.p, s, (int32_t)c.c0, (int32_t)L.cf, (const int32_t *)es.mdct.p,
                (const M3sEncStats *)es.gran.p, (const uint4 *)es.var.p, (uint32_t *)es.sum.p, (int32_t *)es.info.p);
            M3S_LAUNCH_CHECK(h);
        }
        const int64_t n_gran = 4 * c.slots;
        M3S_KBEGIN(h, M3S_K_ENC_AUX);
        k_enc_emit<<<(unsigned)((n_gran + EMIT_WARPS * EMIT_G - 1) / (EMIT_WARPS * EMIT_G)), 32 * EMIT_WARPS, sizeof(RateSmem), h->stream>>>(
            c.clips, c.frame_clip, h->d_tab, (const EncTables *)h->e_tabs.p, (int32_t)c.c0, (int32_t)L.cf,
            n_gran, (const int32_t *)es.mdct.p, (const M3sEncStats *)es.gran.p, (const uint32_t *)es.sum.p,
            (const int32_t *)es.info.p, (uint32_t *)es.ix.p,
            (const uint32_t *)((const char *)h->e_lastix.p + (size_t)(c.k & 1) * lastix_bytes),
            (uint32_t *)((char *)h->e_lastix.p + (size_t)((c.k + 1) & 1) * lastix_bytes));
        M3S_LAUNCH_CHECK(h);
        // packing stays on the rate loop's stream
        M3S_KBEGIN(h, M3S_K_ENC_PACK);
        k_enc_pack<<<(unsigned)((c.slots + PACK_WARPS - 1) / PACK_WARPS), 32 * PACK_WARPS, sizeof(PackSmem), h->stream>>>(
            c.clips, c.frame_clip, h->d_tab, (const uint32_t *)h->e_pad.p, 0, c.slots,
            (const uint32_t *)es.ix.p, (const int32_t *)es.info.p, (const uint8_t *)es.scfsi.p, d_out);
        M3S_LAUNCH_CHECK(h);
        return M3S_OK;
    });
    if (rc) return rc;
    // ---- results, by the caller's clip index
    if (hide_str_offset_out)
        for (int j = 0; j < n_clips; j++) hide_str_offset_out[j] = states[L.inv[j]].hide_off;
    for (int j = 0; j < n_clips; j++)
        if (states[L.inv[j]].overrun)
            return m3s_fail(h, M3S_ERR_ARG, "encode: clip %d frame %d: the step search runs past the end of the step table (quantize would "
                            "read steptabi[128]; the reference has no defined output for this input, SURVEY A.E13)", j, states[L.inv[j]].overrun - 1);
    // taps: the device holds the frames in the library's clip order; (device frame, caller frame, frames) runs map them back
    h->enc_tap_runs.clear();
    std::vector<int64_t> caller_fb(n_clips + 1, 0);
    for (int j = 0; j < n_clips; j++) caller_fb[j + 1] = caller_fb[j] + a.n_samples[j] / 1152;
    for (int i = 0; i < n_clips; i++) {
        const int64_t src = L.clips[i].frame_base, dst = caller_fb[L.order[i]], n = L.clips[i].n_frames;
        std::vector<int64_t> &R = h->enc_tap_runs;
        if (n == 0) continue;
        if (!R.empty() && R[R.size() - 3] + R.back() == src && R[R.size() - 2] + R.back() == dst) R.back() += n;
        else R.insert(R.end(), {src, dst, n});
    }
    h->enc_taps_ok = L.n_chunks == 1;
    h->enc_total_frames = L.total_frames;
    return M3S_OK;
}

extern "C" int m3s_encode(m3s_handle_t h, const int16_t *pcm, int mem, const int64_t *pcm_off, const int64_t *n_samples,
                          int32_t n_clips, int32_t sample_rate, int32_t bitrate_kbps, const uint8_t *payload_bits,
                          const int64_t *payload_off, uint8_t *mp3_out, const int64_t *mp3_off, const int64_t *mp3_cap,
                          int64_t *out_len, int64_t *hide_str_offset_out)
{
    if (!h) return M3S_ERR_ARG;
    h->enc_taps_ok = false;
    if (sr_index_of(sample_rate) < 0) return m3s_fail(h, M3S_ERR_ARG, "encode: sample rate %d is not an MPEG-1 rate", sample_rate);
    if (br_index_of(bitrate_kbps) < 0)
        return m3s_fail(h, M3S_ERR_ARG, "encode: bitrate %d is not an MPEG-1 Layer III rate (WAV_Reader.py:112-114)", bitrate_kbps);
    // the batch's one rate pair, broadcast to every clip
    const std::vector<int32_t> srs((size_t)std::max(n_clips, 0), sample_rate), brs((size_t)std::max(n_clips, 0), bitrate_kbps);
    return drain_on_error(h, encode_mp3(h, EncClips{pcm, mem, pcm_off, n_samples, n_clips, srs.data(), brs.data()}, payload_bits,
                                        payload_off, mp3_out, mp3_off, mp3_cap, out_len, hide_str_offset_out));
}

extern "C" int m3s_encode_mixed(m3s_handle_t h, const int16_t *pcm, int mem, const int64_t *pcm_off, const int64_t *n_samples,
                                int32_t n_clips, const int32_t *sample_rate, const int32_t *bitrate_kbps, const uint8_t *payload_bits,
                                const int64_t *payload_off, uint8_t *mp3_out, const int64_t *mp3_off, const int64_t *mp3_cap,
                                int64_t *out_len, int64_t *hide_str_offset_out)
{
    return drain_on_error(h, encode_mp3(h, EncClips{pcm, mem, pcm_off, n_samples, n_clips, sample_rate, bitrate_kbps}, payload_bits,
                                        payload_off, mp3_out, mp3_off, mp3_cap, out_len, hide_str_offset_out));
}

// The payload length k_enc_probe prunes the variants of caller clip j with (`sure3`).  It is the shortest hiding candidate's: with a
// longer one the probe would skip end-of-payload variants that a shorter candidate meets.  An empty candidate next to hiding ones
// needs variant 14 (no bits left) at every granule, which only a payload shorter than 3 bits keeps active.  0 when no candidate hides.
static int64_t offsets_probe_len(const EncOffsets &ox, int j)
{
    int64_t shortest = INT64_MAX;
    bool empty = false;
    for (int64_t c = ox.cand_off[j]; c < ox.cand_off[j + 1]; c++) {
        const int64_t nbits = 8 * (ox.head_off[c + 1] - ox.head_off[c] + ox.body_len[c]);
        if (nbits == 0) empty = true;
        else shortest = std::min(shortest, nbits);
    }
    if (shortest == INT64_MAX) return 0;
    return empty ? 1 : shortest;
}

// m3s_encode_offsets: analysis and probe as for an encode, then k_enc_offsets instead of resolve, emit and pack;
// hide_str_offset_out is indexed by candidate
static int encode_offsets(m3s_ctx *h, const EncClips &a, const EncOffsets &ox, int64_t *hide_str_offset_out)
{
    double tr_t = m3s_trace ? m3s_now_ms() : 0.0;
    int rc;
    if ((rc = check_call(h, a, ox.body_off && ox.cand_off && ox.head_off && ox.body_len && hide_str_offset_out))) return rc;
    if (ox.cand_off[0] != 0) return m3s_fail(h, M3S_ERR_ARG, "encode_offsets: cand_off[0] is %lld, not 0", (long long)ox.cand_off[0]);
    for (int j = 0; j < a.n_clips; j++) {
        if ((rc = check_clip(h, a, j))) return rc;
        const int64_t c0 = ox.cand_off[j], c1 = ox.cand_off[j + 1], b0 = ox.body_off[j], b1 = ox.body_off[j + 1];
        if (c1 < c0) return m3s_fail(h, M3S_ERR_ARG, "encode_offsets: clip %d: cand_off decreases (%lld -> %lld)", j, (long long)c0, (long long)c1);
        if (b0 < 0 || b1 < b0) return m3s_fail(h, M3S_ERR_ARG, "encode_offsets: clip %d: bad body range [%lld, %lld)", j, (long long)b0, (long long)b1);
        if (b1 > b0 && !ox.body) return m3s_fail(h, M3S_ERR_ARG, "encode_offsets: clip %d: body is NULL", j);
        for (int64_t c = c0; c < c1; c++) {
            const int64_t h0 = ox.head_off[c], h1 = ox.head_off[c + 1], bl = ox.body_len[c];
            if (h0 < 0 || h1 < h0) return m3s_fail(h, M3S_ERR_ARG, "encode_offsets: clip %d candidate %lld: bad head range [%lld, %lld)", j, (long long)c, (long long)h0, (long long)h1);
            if (h1 - h0 > 32) return m3s_fail(h, M3S_ERR_ARG, "encode_offsets: clip %d candidate %lld: head of %lld bytes, more than 32", j, (long long)c, (long long)(h1 - h0));
            if (h1 > h0 && !ox.head) return m3s_fail(h, M3S_ERR_ARG, "encode_offsets: clip %d candidate %lld: head is NULL", j, (long long)c);
            if (bl < 0 || bl > b1 - b0)
                return m3s_fail(h, M3S_ERR_ARG, "encode_offsets: clip %d candidate %lld: body_len %lld outside the clip's body of %lld bytes", j, (long long)c, (long long)bl, (long long)(b1 - b0));
        }
    }
    M3S_CUDA(h, cudaSetDevice(h->device));
    EncLayout L;
    if ((rc = enc_layout(h, a, L))) return rc;
    const int n_clips = a.n_clips;
    for (int j = 0; j < n_clips; j++) L.clips[L.inv[j]].payload_len = offsets_probe_len(ox, j);
    const int64_t n_cand = ox.cand_off[n_clips];
    for (int64_t c = 0; c < n_cand; c++) hide_str_offset_out[c] = 0;
    if (L.total_frames == 0 || n_cand == 0) return M3S_OK;
    M3S_ENC_MARK("clip table");
    // the candidates, k_enc_offsets' work items (32 candidates of one clip each, in the library's clip order, so that the items of
    // one sample rate are [ogrp[s], ogrp[s + 1])), the heads and the bodies, in one buffer
    std::vector<M3sOffCand> cands((size_t)n_cand);
    std::vector<M3sOffWork> owork;
    int ogrp[4] = {0, 0, 0, 0};
    int64_t body_total = 0;
    for (int i = 0; i < n_clips; i++) {
        const int j = L.order[i];
        for (int s = 0; s < 4; s++)
            if (L.grp[s] == i) ogrp[s] = (int)owork.size();
        body_total = std::max(body_total, ox.body_off[j + 1]);
        for (int64_t c = ox.cand_off[j]; c < ox.cand_off[j + 1]; c++) {
            M3sOffCand &d = cands[(size_t)c];
            d.head_base = (int32_t)ox.head_off[c];
            d.head_len = (int32_t)(ox.head_off[c + 1] - ox.head_off[c]);
            d.body_base = ox.body_off[j];
            d.nbits = 8 * (d.head_len + ox.body_len[c]);
            if ((c - ox.cand_off[j]) % 32 == 0) owork.push_back(M3sOffWork{i, (int32_t)std::min<int64_t>(32, ox.cand_off[j + 1] - c), c});
        }
    }
    for (int s = 0; s < 4; s++)
        if (L.grp[s] == n_clips) ogrp[s] = (int)owork.size();
    const int64_t head_total = ox.head_off[n_cand];
    if (head_total > INT32_MAX || owork.size() > (size_t)INT32_MAX) return m3s_fail(h, M3S_ERR_ARG, "encode_offsets: too many candidates in one call");
    auto al16 = [](size_t b) { return (b + 15) / 16 * 16; };
    const size_t o_work = al16(sizeof(M3sOffCand) * cands.size()), o_head = o_work + al16(sizeof(M3sOffWork) * owork.size());
    const size_t o_body = o_head + al16((size_t)head_total);
    if ((rc = m3s_buf_reserve(h, h->e_cand, o_body + (size_t)body_total + 16))) return rc;
    char *base = (char *)h->e_cand.p;
    M3S_CUDA(h, cudaMemcpyAsync(base, cands.data(), sizeof(M3sOffCand) * cands.size(), cudaMemcpyHostToDevice, h->stream));
    M3S_CUDA(h, cudaMemcpyAsync(base + o_work, owork.data(), sizeof(M3sOffWork) * owork.size(), cudaMemcpyHostToDevice, h->stream));
    if (head_total > 0) M3S_CUDA(h, cudaMemcpyAsync(base + o_head, ox.head, (size_t)head_total, cudaMemcpyHostToDevice, h->stream));
    if (body_total > 0) M3S_CUDA(h, cudaMemcpyAsync(base + o_body, ox.body, (size_t)body_total, cudaMemcpyHostToDevice, h->stream));
    const M3sOffCand *d_cands = (const M3sOffCand *)base;
    const M3sOffWork *d_owork = (const M3sOffWork *)(base + o_work);
    const uint8_t *d_head = (const uint8_t *)(base + o_head), *d_body = (const uint8_t *)(base + o_body);
    M3S_CUDA(h, cudaFuncSetAttribute(k_enc_offsets, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RateSmem)));
    std::vector<M3sEncState> states((size_t)n_cand);   // the carried state is per candidate
    rc = enc_pipeline(h, a, L, states, nullptr, tr_t, [&](const EncChunk &c) -> int {
        for (int s = 0; s < 3; s++) {
            if (c.grp_slot[s + 1] == c.grp_slot[s] || ogrp[s + 1] == ogrp[s]) continue;
            M3S_KBEGIN(h, M3S_K_ENC_OFFSETS);
            k_enc_offsets<<<(unsigned)((ogrp[s + 1] - ogrp[s] + OFFSETS_WARPS - 1) / OFFSETS_WARPS), 32 * OFFSETS_WARPS, sizeof(RateSmem), h->stream>>>(
                c.clips, d_owork, ogrp[s], ogrp[s + 1], d_cands, d_head, d_body, (M3sEncState *)h->e_state.p, h->d_tab,
                (const EncTables *)h->e_tabs.p, (const uint32_t *)h->e_pad.p, s, (int32_t)c.c0, (int32_t)L.cf, (const int32_t *)c.set.mdct.p,
                (const M3sEncStats *)c.set.gran.p, (const uint4 *)c.set.var.p, (const uint32_t *)c.set.sum.p);
            M3S_LAUNCH_CHECK(h);
        }
        return M3S_OK;
    });
    if (rc) return rc;
    // ---- results, by the caller's candidate index
    for (int64_t c = 0; c < n_cand; c++) hide_str_offset_out[c] = states[(size_t)c].hide_off;
    for (int j = 0; j < n_clips; j++)
        for (int64_t c = ox.cand_off[j]; c < ox.cand_off[j + 1]; c++)
            if (states[(size_t)c].overrun)
                return m3s_fail(h, M3S_ERR_ARG, "encode_offsets: clip %d candidate %lld frame %d: the step search runs past the end of the step "
                                "table (quantize would read steptabi[128]; the reference has no defined output for this input, SURVEY A.E13)",
                                j, (long long)c, states[(size_t)c].overrun - 1);
    return M3S_OK;
}

extern "C" int m3s_encode_offsets(m3s_handle_t h, const int16_t *pcm, int mem, const int64_t *pcm_off, const int64_t *n_samples,
                                  int32_t n_clips, const int32_t *sample_rate, const int32_t *bitrate_kbps, const uint8_t *body,
                                  const int64_t *body_off, const int64_t *cand_off, const uint8_t *head, const int64_t *head_off,
                                  const int64_t *body_len, int64_t *hide_str_offset_out)
{
    return drain_on_error(h, encode_offsets(h, EncClips{pcm, mem, pcm_off, n_samples, n_clips, sample_rate, bitrate_kbps},
                                            EncOffsets{body, body_off, cand_off, head, head_off, body_len}, hide_str_offset_out));
}

extern "C" int m3s_encode_taps(m3s_handle_t h, int32_t *mdct, int32_t *ix, int32_t *info, int32_t *scfsi)
{
    if (!h) return M3S_ERR_ARG;
    if (!h->enc_taps_ok) return m3s_fail(h, M3S_ERR_STATE, "encode_taps: the last m3s_encode ran in several chunks (or failed); taps need a single-chunk batch");
    M3S_CUDA(h, cudaSetDevice(h->device));
    const int64_t nf = h->enc_total_frames;
    const std::vector<int64_t> &R = h->enc_tap_runs;   // (device frame, caller frame, frames): one run when the order is the caller's
    const size_t NM = 4 * 576, NI = 4 * ENC_INFO_FIELDS;   // values per frame
    for (size_t r = 0; r < R.size(); r += 3) {
        if (mdct) M3S_CUDA(h, cudaMemcpyAsync(mdct + R[r + 1] * NM, (const int32_t *)h->es[0].mdct.p + R[r] * NM, R[r + 2] * NM * 4, cudaMemcpyDeviceToHost, h->stream));
        if (info) M3S_CUDA(h, cudaMemcpyAsync(info + R[r + 1] * NI, (const int32_t *)h->es[0].info.p + R[r] * NI, R[r + 2] * NI * 4, cudaMemcpyDeviceToHost, h->stream));
    }
    std::vector<int16_t> ix16;
    std::vector<uint8_t> sc8;
    if (ix) {
        ix16.resize((size_t)nf * NM);
        M3S_CUDA(h, cudaMemcpyAsync(ix16.data(), h->es[0].ix.p, ix16.size() * 2, cudaMemcpyDeviceToHost, h->stream));
    }
    if (scfsi) {
        sc8.resize((size_t)nf * 8);
        M3S_CUDA(h, cudaMemcpyAsync(sc8.data(), h->es[0].scfsi.p, sc8.size(), cudaMemcpyDeviceToHost, h->stream));
    }
    M3S_CUDA(h, cudaStreamSynchronize(h->stream));
    for (size_t r = 0; r < R.size(); r += 3) {
        if (ix) for (size_t i = 0; i < (size_t)R[r + 2] * NM; i++) ix[R[r + 1] * NM + i] = ix16[R[r] * NM + i];
        if (scfsi) for (size_t i = 0; i < (size_t)R[r + 2] * 8; i++) scfsi[R[r + 1] * 8 + i] = sc8[R[r] * 8 + i];
    }
    return M3S_OK;
}
