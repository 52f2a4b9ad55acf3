// m3s_hybrid_fast.cuh -- D2 + D3 of the decoder, k_hybrid_fast in FP32 (the default path) or float64 (M3S_DEC_EXACT):
// requantize -> MS stereo -> reorder / alias -> IMDCT + window + overlap -> frequency inversion -> polyphase synthesis -> int16.
// (Frame.py:157-218 re_quantize, :561-572, :574-602, :604-622, :106-154 imdct, :624-631, :65-103 synth_filter_bank,
//  :633-640 interleave, MP3_Parser.py:91 int16 conversion)
//
// One CTA (8 warps) walks a run of consecutive frames of one file; a run that does not start its file first decodes one warm-up
// frame whose PCM is dropped (SURVEY.md 8e).  A frame costs three CTA barriers; within a phase the warps take different roles:
//
//   phase A   warps 0-1  IMDCT of frame f: lane = subband, warp = channel, both granules in turn -- the overlap (second half of the
//                        previous granule) never leaves the thread's registers; alias butterflies are applied while the 18 inputs
//                        are loaded (each output depends on one neighbour value, read from the still unmodified spectrum); the
//                        36-point IMDCT is an 18-point DCT-IV in registers (m3s_fast_transforms.cuh)
//             warps 2-7  requantize + MS + reorder of frame f + 1 into the other half of the double-buffered spectrum
//             all        slide the V history, store the PCM of frame f - 1 from its staging tile (32-bit L/R words, coalesced)
//   phase B   warps 0-2  matrixing: one THREAD per (granule, channel, slot) runs a 32-point Lee DCT in registers on its row
//             warps 3-7  fetch frame f + 2: integer spectra by cp.async, per-band requantisation factors, block types
//   phase C   warps 0-7  windowing: warp = (granule, channel, slot parity), lane = output sample; the nine slots of one parity
//                        share their V rows, so 32 loads feed 144 multiply-adds; results go to the PCM staging tile as int16
//
// Shared-memory rows are padded (19 floats per subband, 36 per 32-wide row) so that thread-per-row accesses are conflict-free.
#pragma once
#include "m3s_fast_transforms.cuh"

#define HF_THREADS 256
#define HF_XS 608   // floats per (granule, channel) spectrum: 32 subbands x 19
#define HF_ROW 36   // floats per 32-wide row of tt / v

template <typename OUT, typename R>
struct HybFastSmem {
    uint4 spec[288];                   // integer spectra of ONE frame: [pair] = (x, y) int16 of slots 0..3 (slot = 2 gr + ch)
    R xr[2][2][2][HF_XS];          // [buffer][gr][ch]: requantised spectrum, sample s at s + s / 18
    R tt[2][2][18][HF_ROW];        // [gr][ch][slot][subband]: IMDCT output = matrixing input
    R v[2][51][HF_ROW];            // [ch][row]: per slot the 32 distinct matrixing outputs; 15 rows of history + 2 x 18 new
    OUT stage[2][1152];                // PCM of one frame, channel-major (interleaved when it is stored)
    R wcoef[16][32];               // windowing: per lane its 8 + 8 signed window coefficients (see the kernel)
    R pow43[256];
    R scale[4][64];                // per slot: 2^(e4/4) of long sfb 0..21 | short (sfb * 3 + window) at 22..60
    R sine[4][36];
    R cos12[12][8];
    R cs[8], ca[8];
    R quarter[4];
    uint32_t info[4][4];               // ring over frames (g & 3) x slot: block_type [0:2) | mixed [2]
    uint16_t reorder[576];             // short-block scatter: padded destination | 0x8000 = store zero
    uint8_t band2[2][288];             // pair -> scale index: [0] long sfb, [1] 22 + short sfb * 3 + window
    uint8_t pretab[24];
    int sr_loaded;
};

__device__ __forceinline__ float hf_pow2i(int e)
{
    e = e < -126 ? -126 : (e > 127 ? 127 : e);
    return __int_as_float((e + 127) << 23);
}
// the pieces that differ between the FP32 instantiation and the float64 one (M3S_DEC_EXACT)
__device__ __forceinline__ float hf_scale(float quarter, int e4) { return quarter * hf_pow2i(e4 >> 2); }
__device__ __forceinline__ double hf_scale(double quarter, int e4) { return quarter * scalbn(1.0, e4 >> 2); }
__device__ __forceinline__ float hf_pow43_big(float, int ax) { return (float)ax * cbrtf((float)ax); }
__device__ __forceinline__ double hf_pow43_big(double, int ax) { return pow((double)ax, 4.0 / 3.0); }
__device__ __forceinline__ float hf_signed(float m, int x) { return __int_as_float(__float_as_int(m) | (x & 0x80000000)); }   // m >= 0: OR in the sign of x
__device__ __forceinline__ double hf_signed(double m, int x) { return x < 0 ? -m : m; }
// v -> int32 as numpy's astype does it on x86 (cvttss2si / cvttsd2si): truncation toward zero, and 0x80000000 for v >= 2^31,
// v < -2^31 or NaN, where __float2int_rz / __double2int_rz would saturate (A.D8).  2^31 is exact in both types.
__device__ __forceinline__ int hf_to_int(float o) { return o >= -2147483648.0f && o < 2147483648.0f ? __float2int_rz(o) : (int)0x80000000; }
__device__ __forceinline__ int hf_to_int(double o) { return o >= -2147483648.0 && o < 2147483648.0 ? __double2int_rz(o) : (int)0x80000000; }

// Packed FP32 (Blackwell FFMA2, PTX fma.rn.f32x2): two independent round-to-nearest FMAs per instruction -- the same results as two
// fmaf, half the issue slots.  The windowing's two accumulator chains per output sample (even / odd history rows) run as one.
__device__ __forceinline__ uint64_t hf_pack2(float lo, float hi)
{
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ uint64_t hf_fma2(uint64_t a, uint64_t b, uint64_t c)
{
    uint64_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ float hf_sum2(uint64_t v)
{
    float lo, hi;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
    return lo + hi;
}

// x[i] of the 36-point IMDCT from the 18 DCT-IV values (the index folds once the caller's loop is unrolled)
template <typename R>
__device__ __forceinline__ R hf_imdct_at(const R (&c)[18], int i)
{
    return i < 9 ? c[i + 9] : (i <= 26 ? -c[26 - i] : -c[i - 27]);
}

// The channel count is a template parameter (the host launches the stereo and the mono runs of a wave separately): no register
// for it, no per-sample tests.
// R = float: the default path (<= 1 LSB).  R = double (M3S_DEC_EXACT): the same kernel in float64 -- the int16 samples then equal the
// reference's (which is float64 end to end) on every golden stream; TF holds the hybrid tables in precision R.
template <typename OUT, bool FLOAT_OUT, int nch, typename R, typename TAB>
__global__ void __launch_bounds__(HF_THREADS, sizeof(R) == 4 ? 3 : 1)
k_hybrid_fast(const uint32_t *__restrict__ spec, const M3sUnitRec *__restrict__ units, const uint8_t *__restrict__ sfin,
              const uint32_t *__restrict__ fr_meta, const M3sWork *__restrict__ work, const M3sDevTables *__restrict__ T,
              const TAB *__restrict__ TF, void *__restrict__ pcm_out)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    HybFastSmem<OUT, R> &sm = *reinterpret_cast<HybFastSmem<OUT, R> *>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const M3sWork wk = work[blockIdx.x];
    // (frame indices are wave-relative and fit 32 bits: they stay `int` to keep the loop-carried state small)
    const int g_begin = (int)wk.g_first - (wk.warm ? 1 : 0);
    const int g_end = (int)wk.g_first + wk.count;
    const uint4 *spec4 = (const uint4 *)spec;

    // ---- one-time table staging
    for (int i = tid; i < 12 * 8; i += HF_THREADS) (&sm.cos12[0][0])[i] = (&TF->imdct_cos12[0][0])[i];
    for (int i = tid; i < 4 * 36; i += HF_THREADS) (&sm.sine[0][0])[i] = (&TF->sine_block[0][0])[i];
    for (int i = tid; i < 256; i += HF_THREADS) sm.pow43[i] = TF->pow43[i];
    if (tid < 8) { sm.cs[tid] = TF->alias_cs[tid]; sm.ca[tid] = TF->alias_ca[tid]; }
    if (tid < 4) sm.quarter[tid] = TF->quarter[tid];
    if (tid < 22) sm.pretab[tid] = T->pretab[tid];
    if (tid == 0) sm.sr_loaded = -1;
    if (tid < 16) (&sm.info[0][0])[tid] = 0u;
    for (int i = tid; i < 2 * 51 * HF_ROW; i += HF_THREADS) (&sm.v[0][0][0])[i] = (R)0;
    // windowing (Frame.py:89-101): pcm[32 t + i] = sum_m V_{t-2m}[i] D[64 m + i] + V_{t-2m-1}[32 + i] D[64 m + 32 + i].  A V row holds the 32
    // distinct values W[l] = D[16 + l] (l < 16), W[l] = D[l - 16] (l >= 16) of the slot's 32-point DCT D; lane i reads
    // V[i] = +W[i] | 0 | -W[32 - i] and V[32 + i] = -W[0] | -W[32 - i] | -W[i]; the signs are folded into its 16 window coefficients.
    for (int e = tid; e < 16 * 32; e += HF_THREADS) {
        const int m = e >> 5, i = e & 31;
        const R sA = i < 16 ? (R)1 : (i == 16 ? (R)0 : (R)-1);
        // (the FP32 int16 path folds MP3Parser.write_to_wav's factor 32767 into the coefficients: one multiply per sample less; the
        //  float64 path multiplies the finished sample, as the reference does)
        const R k16 = (FLOAT_OUT || sizeof(R) == 8) ? (R)1 : (R)32767;
        sm.wcoef[m][i] = k16 * (m < 8 ? sA * TF->synth_d[64 * m + i] : -TF->synth_d[64 * (m - 8) + 32 + i]);
    }
    R ovl[18];   // IMDCT warps: windowed second half of the previous granule of (channel = warp, subband = lane)
#pragma unroll
    for (int i = 0; i < 18; i++) ovl[i] = (R)0;

    // ---- per-frame staging: spectra, requantisation factors and block types of frame g, by threads [t0, t0 + nt)
    auto fetch_frame = [&](int g, int t0, int nt) {
        const int tr = tid - t0;
        if (tr < 0 || tr >= nt) return;
        for (int p = tr; p < 288; p += nt) {
            const unsigned dst = (unsigned)__cvta_generic_to_shared(&sm.spec[p]);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(spec4 + (int64_t)g * 288 + p) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        const int sr = (int)((fr_meta[g] >> M3S_META_SR_SHIFT) & 3u);
        if (sm.sr_loaded != sr) {   // uniform over the fetching threads: sr_loaded only changes behind a barrier
            for (int i = tr; i < 576; i += nt) {
                const uint32_t d = T->reorder_dst[sr][i];
                const uint32_t dd = d & 0x3FFu;
                sm.reorder[i] = (uint16_t)((dd + dd / 18u) | (d & 0x8000u));
            }
            for (int p = tr; p < 288; p += nt) {
                sm.band2[0][p] = T->long_sfb_of[sr][2 * p];
                sm.band2[1][p] = (uint8_t)(22 + T->short_sfw_of[sr][2 * p]);
            }
        }
        // requantisation factors: the four slots go to the first four warps of the fetching threads (nt >= 128), two band entries per
        // lane; the unit-record fields are warp-uniform loads
        if (tr < 128 && !(nch == 1 && (tr & 32))) {   // (a mono frame has no slots 1 and 3: their records are placeholders, their scalefactors unwritten)
            const int slot = tr >> 5;
            const M3sUnitRec *r = units + 4 * (int64_t)g + slot;
            const uint32_t a = r->a, b = r->b, c = r->c;
            const uint8_t *sf = sfin + (4 * (int64_t)g + slot) * M3S_SF_STRIDE;
            const int gg = M3S_UA_GG(a), mult4 = M3S_UB_SFSCALE(b) ? 4 : 2, pre = (int)M3S_UB_PREFLAG(b);
#pragma unroll
            for (int it = 0; it < 2; it++) {
                const int idx = (tr & 31) + 32 * it;
                int e4 = 0;
                if (idx < 22) e4 = gg - 210 - mult4 * ((int)sf[idx] + pre * (int)sm.pretab[idx]);
                else if (idx < 61) {
                    const int q = idx - 22, sfb = q / 3, wnd = q - 3 * sfb;
                    e4 = gg - 210 - 8 * (int)M3S_UC_SBG(c, wnd) - mult4 * (int)sf[M3S_SF_SHORT + 13 * wnd + sfb];
                }
                sm.scale[slot][idx] = hf_scale(sm.quarter[e4 & 3], e4);
            }
            if ((tr & 31) == 0) sm.info[g & 3][slot] = M3S_UA_BT(a) | (M3S_UB_MIXED(b) << 2);
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");
    };
    // (sr_loaded is updated by one thread after the barrier that follows a fetch)

    // ---- requantize + MS + reorder of frame g into xr[buf] (Frame.py:157-218, :561-572, :574-602) by the 192 threads [t0, t0 + 192):
    //      96 threads per granule, three pairs each; everything that depends on the granule only is hoisted out of the pair loop
    auto requant_pair = [&](uint32_t wv, R sc, R &vx, R &vy) {
        const int x = (int)(int16_t)(wv & 0xFFFFu), y = (int)wv >> 16;
        const int ax = x < 0 ? -x : x, ay = y < 0 ? -y : y;
        R mx, my;
        if ((ax | ay) < 256) { mx = sm.pow43[ax]; my = sm.pow43[ay]; }
        else {
            mx = ax < 256 ? sm.pow43[ax] : hf_pow43_big((R)0, ax);
            my = ay < 256 ? sm.pow43[ay] : hf_pow43_big((R)0, ay);
        }
        vx = hf_signed(mx * sc, x);   // sign(x) |x|^(4/3) 2^(e4/4)
        vy = hf_signed(my * sc, y);
    };
    auto requant_store = [&](R *X, bool reord, int p, R v0, R v1) {
        if (reord) {
            const uint32_t d01 = ((const uint32_t *)sm.reorder)[p];
            const uint32_t d0 = d01 & 0xFFFFu, d1 = d01 >> 16;
            X[d0 & 0x3FFu] = (d0 & 0x8000u) ? (R)0 : v0;
            X[d1 & 0x3FFu] = (d1 & 0x8000u) ? (R)0 : v1;
        } else {
            const int pos = 2 * p + p / 9;   // samples 2 p and 2 p + 1 lie in the same subband; 19 floats per subband
            X[pos] = v0;
            X[pos + 1] = v1;
        }
    };
    auto requant_frame = [&](int g, int buf, int t0) {
        const int tr = tid - t0;
        if (tr < 0 || tr >= 192) return;
        const int gr = tr >= 96, t = tr - 96 * gr;
        const bool ms = (fr_meta[g] & M3S_META_MS) != 0 && nch == 2;
        const uint32_t inf0 = sm.info[g & 3][2 * gr], inf1 = sm.info[g & 3][2 * gr + 1];
        const bool sh0 = (inf0 & 3u) == 2u, sh1 = (inf1 & 3u) == 2u;
        const bool re0 = sh0 || (inf0 & 4u), re1 = sh1 || (inf1 & 4u);
        const uint8_t *band0 = sm.band2[sh0], *band1 = sm.band2[sh1];
        const R *sc0 = sm.scale[2 * gr], *sc1 = sm.scale[2 * gr + 1];
        R *X0 = sm.xr[buf][gr][0], *X1 = sm.xr[buf][gr][1];
#pragma unroll
        for (int j = 0; j < 3; j++) {
            const int p = t + 96 * j;
            const uint2 w2 = ((const uint2 *)&sm.spec[p])[gr];
            R a0, a1, b0 = (R)0, b1 = (R)0;
            requant_pair(w2.x, sc0[band0[p]], a0, a1);
            if (nch == 2) requant_pair(w2.y, sc1[band1[p]], b0, b1);
            if (ms) {   // (M + S) / SQRT2, (M - S) / SQRT2 (Frame.py:568-572)
                const R m0 = a0, m1 = a1, rs2 = (R)0.70710678118654752;
                a0 = (m0 + b0) * rs2; b0 = (m0 - b0) * rs2;
                a1 = (m1 + b1) * rs2; b1 = (m1 - b1) * rs2;
            }
            requant_store(X0, re0, p, a0, a1);
            if (nch == 2) requant_store(X1, re1, p, b0, b1);
        }
    };

    // ---- prologue: frame g_begin requantised, frame g_begin + 1 fetched
    __syncthreads();
    fetch_frame(g_begin, 0, HF_THREADS);
    __syncthreads();
    if (tid == 0) sm.sr_loaded = (int)((fr_meta[g_begin] >> M3S_META_SR_SHIFT) & 3u);
    requant_frame(g_begin, 0, 0);
    __syncthreads();
    if (g_begin + 1 < g_end) fetch_frame(g_begin + 1, 0, HF_THREADS);
    __syncthreads();
    if (tid == 0 && g_begin + 1 < g_end) sm.sr_loaded = (int)((fr_meta[g_begin + 1] >> M3S_META_SR_SHIFT) & 3u);

    int staged = -1;            // >= 0: the staging tile holds emitted frame number `staged` of the run, still to be stored
    auto store_staged = [&](int t0, int nt) {   // by threads [t0, t0 + nt); every thread keeps `staged` in step
        if (staged < 0) return;
        const int tr = tid - t0;
        if (tr < 0 || tr >= nt) { staged = -1; return; }
        const int n_el = 1152 * nch;
        const M3sWork *w = work + blockIdx.x;   // re-read here rather than held in registers across the frame loop
        const int reps = (fr_meta[w->g_first + staged] & M3S_META_DUP) ? 2 : 1;
        for (int rep = 0; rep < reps; rep++) {
            OUT *dst = (OUT *)pcm_out + w->pcm_elem + (int64_t)(staged + rep) * n_el;
            if (nch == 2) {   // interleave L / R on the way out: every thread stores whole 32-bit (int16) or 64-bit (float) L/R words
                if constexpr (FLOAT_OUT) {
                    float2 *d2 = (float2 *)dst;    // stereo offsets are even: 8-byte aligned
                    for (int i = tr; i < 1152; i += nt) d2[i] = make_float2((float)sm.stage[0][i], (float)sm.stage[1][i]);
                } else {
                    const uint32_t *sl = (const uint32_t *)sm.stage[0], *sr_ = (const uint32_t *)sm.stage[1];
                    const bool al8 = ((uintptr_t)dst & 7) == 0;
                    for (int i = tr; i < 576; i += nt) {   // samples 2 i and 2 i + 1
                        const uint32_t l2 = sl[i], r2 = sr_[i];
                        const uint32_t w0 = __byte_perm(l2, r2, 0x5410), w1 = __byte_perm(l2, r2, 0x7632);
                        if (al8) ((uint2 *)dst)[i] = make_uint2(w0, w1);
                        else { ((uint32_t *)dst)[2 * i] = w0; ((uint32_t *)dst)[2 * i + 1] = w1; }
                    }
                }
            } else {
                for (int i = tr; i < 1152; i += nt) dst[i] = sm.stage[0][i];
            }
        }
        staged = -1;
    };

    const int n_run = g_end - g_begin, warm = wk.warm ? 1 : 0;
    for (int f = 0; f < n_run; f++) {
        const int g = g_begin + f;
        const int buf = f & 1;
        const bool emit = f >= warm;
        // ================================================================ phase A
        if (g > g_begin && tid >= 64) {   // slide the V history: rows 36..50 -> 0..14 (nobody else touches V in this phase; the IMDCT
                                          // warps, the phase's critical path, are left out of it)
            constexpr int CH16 = 15 * HF_ROW * (int)sizeof(R) / 16;   // 16-byte chunks per channel
            for (int idx = tid - 64; idx < nch * CH16; idx += HF_THREADS - 64) {
                const int ch = idx >= CH16, r_ = idx - ch * CH16;
                ((uint4 *)&sm.v[ch][0][0])[r_] = ((const uint4 *)&sm.v[ch][36][0])[r_];
            }
        }
        if (warp < 2) {
            const int ch = warp, sb = lane;
            if (ch < nch) {
#pragma unroll 1
                for (int gr = 0; gr < 2; gr++) {
                    const uint32_t inf = sm.info[g & 3][2 * gr + ch];
                    const int bt = (int)(inf & 3u);
                    const R *X = sm.xr[buf][gr][ch];
                    R *ttc = &sm.tt[gr][ch][0][sb];
                    R x[18];
#pragma unroll
                    for (int k = 0; k < 18; k++) x[k] = X[19 * sb + k];
                    if (bt != 2) {
                        if (!(inf & 4u)) {   // alias reduction (Frame.py:604-622): skipped for short and mixed granules
                            if (sb >= 1) {
#pragma unroll
                                for (int i = 0; i < 8; i++) x[i] = x[i] * sm.cs[i] + X[19 * (sb - 1) + 17 - i] * sm.ca[i];
                            }
                            if (sb <= 30) {
#pragma unroll
                                for (int i = 0; i < 8; i++) x[17 - i] = x[17 - i] * sm.cs[i] - X[19 * (sb + 1) + i] * sm.ca[i];
                            }
                        }
                        R c[18];
                        dct4_18<R>(x, c);
                        const R *w = sm.sine[bt];
#pragma unroll
                        for (int i = 0; i < 18; i++) {
                            R o = m3s_fma(hf_imdct_at(c, i), w[i], ovl[i]);
                            if ((i & 1) && (sb & 1)) o = -o;       // frequency inversion (Frame.py:624-631)
                            ttc[HF_ROW * i] = o;
                            ovl[i] = hf_imdct_at(c, 18 + i) * w[18 + i];
                        }
                    } else {
                        // three 12-point IMDCTs, windowed and placed at 6 / 12 / 18 with overlap (Frame.py:135-148)
#pragma unroll
                        for (int i = 0; i < 18; i++) {
                            R acc = (R)0;
                            if (i >= 6) {
                                const int w_hi = (i - 6) / 6, i_hi = i - 6 - 6 * w_hi;
                                if (w_hi < 3) {
                                    R a2 = (R)0;
#pragma unroll
                                    for (int k = 0; k < 6; k++) a2 = m3s_fma(x[6 * w_hi + k], sm.cos12[i_hi][k], a2);
                                    acc += a2 * sm.sine[2][i_hi];
                                }
                                const int w_lo = w_hi - 1;
                                if (w_lo >= 0) {
                                    R a2 = (R)0;
#pragma unroll
                                    for (int k = 0; k < 6; k++) a2 = m3s_fma(x[6 * w_lo + k], sm.cos12[i_hi + 6][k], a2);
                                    acc += a2 * sm.sine[2][i_hi + 6];
                                }
                            }
                            R o = acc + ovl[i];
                            if ((i & 1) && (sb & 1)) o = -o;
                            ttc[HF_ROW * i] = o;
                        }
                        // second half -> the next granule's overlap (every ovl[i] was consumed above)
#pragma unroll
                        for (int i = 18; i < 36; i++) {
                            R acc = (R)0;
                            if (i < 30) {
                                const int w_hi = (i - 6) / 6, i_hi = i - 6 - 6 * w_hi;
                                if (w_hi < 3) {
                                    R a2 = (R)0;
#pragma unroll
                                    for (int k = 0; k < 6; k++) a2 = m3s_fma(x[6 * w_hi + k], sm.cos12[i_hi][k], a2);
                                    acc += a2 * sm.sine[2][i_hi];
                                }
                                const int w_lo = w_hi - 1;
                                R a2 = (R)0;
#pragma unroll
                                for (int k = 0; k < 6; k++) a2 = m3s_fma(x[6 * w_lo + k], sm.cos12[i_hi + 6][k], a2);
                                acc += a2 * sm.sine[2][i_hi + 6];
                            }
                            ovl[i - 18] = acc;
                        }
                    }
                }
            }
        } else if (g + 1 < g_end) {
            requant_frame(g + 1, buf ^ 1, 64);
        }
        __syncthreads();
        // ================================================================ phase B
        if (tid < nch * 36) {   // matrixing: thread = (granule, channel, slot), a 32-point DCT-II in registers (Frame.py:81-87)
            const int t = tid % 18, gc = tid / 18, ch = gc % nch, gr = gc / nch;
            R S[32];
            const R *row = sm.tt[gr][ch][t];
            R *vo = sm.v[ch][15 + 18 * gr + t];
            if constexpr (sizeof(R) == 4) {
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    const float4 q = ((const float4 *)row)[j];
                    S[4 * j] = q.x; S[4 * j + 1] = q.y; S[4 * j + 2] = q.z; S[4 * j + 3] = q.w;
                }
            } else {
#pragma unroll
                for (int j = 0; j < 16; j++) {
                    const double2 q = ((const double2 *)row)[j];
                    S[2 * j] = q.x; S[2 * j + 1] = q.y;
                }
            }
            dct2_lee<32, R>(S);
            if constexpr (sizeof(R) == 4) {
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    ((float4 *)vo)[j] = make_float4(S[16 + 4 * j], S[17 + 4 * j], S[18 + 4 * j], S[19 + 4 * j]);
                    ((float4 *)vo)[4 + j] = make_float4(S[4 * j], S[4 * j + 1], S[4 * j + 2], S[4 * j + 3]);
                }
            } else {
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    ((double2 *)vo)[j] = make_double2(S[16 + 2 * j], S[17 + 2 * j]);
                    ((double2 *)vo)[8 + j] = make_double2(S[2 * j], S[2 * j + 1]);
                }
            }
        }
        if (warp >= 3) {   // frame f - 1's PCM goes out of its staging tile, frame f + 2 comes in
            if (g + 2 < g_end) fetch_frame(g + 2, 96, HF_THREADS - 96);
        }
        store_staged(96, HF_THREADS - 96);
        __syncthreads();
        if (tid == 0 && g + 2 < g_end) sm.sr_loaded = (int)((fr_meta[g + 2] >> M3S_META_SR_SHIFT) & 3u);
        // ================================================================ phase C
        if (emit) {   // windowing: warp = (granule, channel, slot parity), lane = sample of the slot
            const int gr = warp >> 2, ch = (warp >> 1) & 1, par = warp & 1;
            if (ch < nch) {
                const int idxA = lane < 16 ? lane : (lane == 16 ? 0 : 32 - lane);
                const int idxB = lane == 0 ? 0 : (lane < 16 ? 32 - lane : lane);
                const R *va = &sm.v[ch][1 + 18 * gr + par][idxA], *vb = &sm.v[ch][18 * gr + par][idxB];
                R a[16], b[16], dA[8], dB[8];
#pragma unroll
                for (int m = 0; m < 8; m++) { dA[m] = sm.wcoef[m][lane]; dB[m] = sm.wcoef[8 + m][lane]; }
#pragma unroll
                for (int d = 0; d < 16; d++) { a[d] = va[2 * HF_ROW * d]; b[d] = vb[2 * HF_ROW * d]; }
                uint64_t ab2[16], d2[8];   // FP32: (a, b) and (dA, dB) as register pairs for FFMA2
                if constexpr (sizeof(R) == 4) {
#pragma unroll
                    for (int m = 0; m < 8; m++) d2[m] = hf_pack2((float)dA[m], (float)dB[m]);
#pragma unroll
                    for (int d = 0; d < 16; d++) ab2[d] = hf_pack2((float)a[d], (float)b[d]);
                }
#pragma unroll
                for (int q = 0; q < 9; q++) {
                    R o;
                    if constexpr (sizeof(R) == 4) {
                        uint64_t acc = 0ull;   // (+0.0f, +0.0f)
#pragma unroll
                        for (int m = 0; m < 8; m++) acc = hf_fma2(ab2[q - m + 7], d2[m], acc);
                        o = (R)hf_sum2(acc);
                    } else {
                        R acc0 = (R)0, acc1 = (R)0;
#pragma unroll
                        for (int m = 0; m < 8; m++) {
                            acc0 = m3s_fma(a[q - m + 7], dA[m], acc0);
                            acc1 = m3s_fma(b[q - m + 7], dB[m], acc1);
                        }
                        o = acc0 + acc1;
                    }
                    OUT *so = &sm.stage[ch][gr * 576 + 32 * par + lane];
                    // (pcm * 32767).astype(int16): truncate to int32 (0x80000000 outside it), keep the low 16 bits (A.D8); FP32 carries
                    // the factor in its window coefficients
                    if (FLOAT_OUT) so[64 * q] = (OUT)o;
                    else if constexpr (sizeof(R) == 8) so[64 * q] = (OUT)(int16_t)hf_to_int(o * (R)32767);
                    else so[64 * q] = (OUT)(int16_t)hf_to_int(o);
                }
            }
            staged = f - warm;
        }
        __syncthreads();
    }
    store_staged(0, HF_THREADS);
}
