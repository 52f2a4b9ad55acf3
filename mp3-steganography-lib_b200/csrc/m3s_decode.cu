// m3s_decode.cu -- decode half of the hot path: D0 frame walk + side-info scan (+ reveal bits),
// main-data compaction, D1 Huffman/scalefactor decode, D2+D3 fused requantize -> stereo -> reorder/alias ->
// IMDCT/overlap -> polyphase synthesis -> int16.   Reference: mp3stego/decoder/{MP3_Parser,Frame,
// FrameHeader,FrameSideInformation,util}.py (cited per kernel below).
#include <string.h>

#include <algorithm>

#include "m3s_common.cuh"
#include "m3s_tables_data.h"

// ================================================================================================
// small device helpers
// ================================================================================================
__device__ __forceinline__ uint32_t ldb(const uint8_t *bytes, int64_t p, int64_t fend)
{
    return p < fend ? (uint32_t)__ldg(bytes + p) : 0u;  // util.get_bits pads with zeros past the buffer (util.py:41-43)
}

// n <= 16 bits at bit offset `bitoff` from byte position `base`, MSB first, file-clipped
__device__ __forceinline__ uint32_t bits_at(const uint8_t *bytes, int64_t base, int64_t fend, int bitoff, int n)
{
    int64_t p = base + (bitoff >> 3);
    uint32_t w = (ldb(bytes, p, fend) << 16) | (ldb(bytes, p + 1, fend) << 8) | ldb(bytes, p + 2, fend);
    return (w >> (24 - (bitoff & 7) - n)) & ((1u << n) - 1u);
}

struct M3sHdr {
    int frame_size, hdrlen, mono, crc_present, mode, ms, sr_idx, bitrate, sr;
};

// FrameHeader.init_header_params (FrameHeader.py:51-192) + Frame.set_frame_size (Frame.py:288-316).
// Returns 0, or <0 outside the supported domain (MPEG-1 Layer III, non-reserved rate, bitrate index != 15).
__device__ __forceinline__ int parse_header(uint32_t b1, uint32_t b2, uint32_t b3, M3sHdr &h)
{
    if (((b1 >> 3) & 3) != 3) return -2;
    if (((b1 >> 1) & 3) != 1) return -3;
    int sri = (b2 >> 2) & 3;
    if (sri == 3) return -4;
    int bi = (int)(b2 >> 4);
    if (bi == 15) return -5;
    const int br_tab[14] = {32, 40, 48, 56, 64, 80, 96, 112, 128, 160, 192, 224, 256, 320};
    bi = bi == 0 ? 13 : bi - 1;  // index 0 -> rates[-1] in the reference (FrameHeader.py:180-181)
    h.bitrate = br_tab[bi] * 1000;
    h.sr = sri == 0 ? 44100 : (sri == 1 ? 48000 : 32000);
    h.sr_idx = sri;
    h.crc_present = (b1 & 1) ? 0 : 1;
    h.mode = (b3 >> 6) & 3;
    h.mono = h.mode == 3;
    h.ms = (h.mode == 1) && (b3 & 0x20);
    h.frame_size = (144 * h.bitrate) / h.sr + ((b2 >> 1) & 1);  // == int((1152/8*bit_rate)/sampling_rate) + padding
    h.hdrlen = 4 + (h.crc_present ? 2 : 0) + (h.mono ? 17 : 32);
    return 0;
}

// ================================================================================================
// D0a: frame walk, one WARP per file (MP3_Parser.py:57-85).  The chain offset -> header -> frame size ->
// next offset is serial, so the warp hides the memory latency by speculation: lane k prefetches a 64-byte
// window where frame k of the next 32 is expected for a constant frame size (its start can only drift by
// the <= 31 padding bytes of the frames before it), then the 32 headers are resolved from shared memory
// with no further global round trip.  A header outside its window (VBR, bitrate change) is fetched
// directly.  Writes file-relative frame positions to a temporary array and per-file totals.
// ================================================================================================
#define WALK_WARPS 4
#define WALK_WIN 64
#define WALK_STRIDE 17  // words per lane window (64 B + 4 B pad: conflict-free)

__device__ __forceinline__ uint4 load16_clipped(const uint8_t *bytes, int64_t p, int64_t fend, int64_t total_bytes)
{
    // 16 bytes at p (p + addr 16-aligned); bytes at or beyond fend read as zero; never touches memory beyond total_bytes
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (p >= fend) return v;
    if (p >= 0 && p + 16 <= total_bytes) {
        v = __ldg((const uint4 *)(bytes + p));
        if (p + 16 > fend) {
            uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int i = 0; i < 4; i++) {
                int64_t q = p + 4 * i;
                if (q >= fend) w[i] = 0u;
                else if (q + 4 > fend) w[i] &= 0xFFFFFFFFu >> (8 * (int)(q + 4 - fend));
            }
            v = make_uint4(w[0], w[1], w[2], w[3]);
        }
    } else {
        uint32_t w[4] = {0u, 0u, 0u, 0u};
        for (int i = 0; i < 16; i++) {
            int64_t q = p + i;
            if (q >= 0 && q < fend) w[i >> 2] |= (uint32_t)__ldg(bytes + q) << (8 * (i & 3));
        }
        v = make_uint4(w[0], w[1], w[2], w[3]);
    }
    return v;
}

__global__ void __launch_bounds__(32 * WALK_WARPS)
k_walk(const uint8_t *__restrict__ bytes, int64_t total_bytes, const M3sFileRec *__restrict__ files, M3sFileOut *fouts,
       int n_files, uint32_t *__restrict__ tmp_pos)
{
    __shared__ uint32_t s_win[WALK_WARPS][32 * WALK_STRIDE];
    const int lane = threadIdx.x & 31, wip = threadIdx.x >> 5;
    const int f = blockIdx.x * WALK_WARPS + wip;
    if (f >= n_files) return;
    const M3sFileRec fr = files[f];
    int64_t off = fr.audio;
    const int64_t fend = fr.end;
    M3sFileOut o;
    o.payload_total = 0; o.n_frames = 0; o.status = 0; o.sample_rate = 0; o.channels = 0; o.bitrate = 0; o.reveal_len = 0;
    if (!(fend - off >= 2 && ldb(bytes, off, fend) == 0xFF && ldb(bytes, off + 1, fend) >= 0xE0)) {
        o.status = M3S_FILE_NO_SYNC;
        if (lane == 0) fouts[f] = o;
        return;
    }
    uint32_t *win = s_win[wip];
    const uint8_t *winb = (const uint8_t *)win;
    const int64_t align_fix = (int64_t)((uintptr_t)bytes & 15);  // windows are aligned in the address space
    int fs_guess = 0;
    {
        M3sHdr h0;
        if (parse_header(ldb(bytes, off + 1, fend), ldb(bytes, off + 2, fend), ldb(bytes, off + 3, fend), h0) == 0)
            fs_guess = (144 * h0.bitrate) / h0.sr;
    }
    int64_t P = 0;
    int n = 0;
    bool done = false;
    while (!done) {
        // ---- speculative prefetch
        const int64_t want = off + (int64_t)lane * fs_guess;
        const int64_t wbase = ((want + align_fix) & ~(int64_t)15) - align_fix;  // <= want, 16-aligned address
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const uint4 v = load16_clipped(bytes, wbase + 16 * q, fend, total_bytes);
            uint32_t *d = win + lane * WALK_STRIDE + 4 * q;
            d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
        }
        __syncwarp();
        // ---- resolve up to 32 frames (uniform control flow)
        uint32_t mypos = 0;
        int got = 0, k0 = 0;
        // Fast path for runs of frames that repeat the batch's first header up to the padding bit (every constant-bitrate file): frame k
        // then starts at off + k * fs + (padding bits of frames 0 .. k-1), i.e. at one of k + 1 positions of lane k's window.  Each lane
        // tests ITS candidates in parallel (match mask, padding mask); the serial part of the chain shrinks to a shuffle, two bit
        // tests and a few adds per frame.  The first frame that does not match falls back to the general step below.
        {
            const int d0 = (int)(off - __shfl_sync(0xFFFFFFFFu, wbase, 0));
            M3sHdr hr;
            uint32_t r1 = 0, r2 = 0, r3 = 0;
            bool fast = fend > off + 4 && d0 >= 0 && d0 + 4 <= WALK_WIN;
            if (fast) {
                const uint8_t *q = winb + d0;
                r1 = q[1]; r2 = q[2]; r3 = q[3];
                fast = q[0] == 0xFF && r1 >= 0xE0 && parse_header(r1, r2, r3, hr) == 0 && (144 * hr.bitrate) / hr.sr == fs_guess;
            }
            if (fast) {
                const int fs0 = fs_guess, dmin = (int)(want - wbase);   // candidate c of lane k sits at window byte dmin + c, c <= k
                uint32_t mm = 0, pm = 0;
                const uint32_t *ww = win + lane * WALK_STRIDE;
                for (int c = 0; c <= lane; c++) {
                    const int d = dmin + c;
                    const uint32_t v = __funnelshift_r(ww[d >> 2], ww[(d >> 2) + 1], 8 * (d & 3));   // bytes d .. d + 3, little-endian
                    const bool ok = (v & 0xC0FCFFFFu) == (0xFFu | r1 << 8 | (r2 & 0xFCu) << 16 | (r3 & 0xC0u) << 24);
                    mm |= (uint32_t)ok << c;
                    pm |= ((v >> 17) & 1u) << c;
                }
                int c = 0;
                for (; k0 < 32; k0++) {
                    if (!(fend > off + 4)) { done = true; break; }
                    const uint32_t m = __shfl_sync(0xFFFFFFFFu, mm, k0), pbits = __shfl_sync(0xFFFFFFFFu, pm, k0);
                    if (!((m >> c) & 1u)) break;
                    const int pad = (int)((pbits >> c) & 1u), fs = fs0 + pad;
                    const int64_t avail = fend - off;
                    int payload = (fs < avail ? fs : (int)avail) - hr.hdrlen;
                    if (payload < 0) payload = 0;
                    if (lane == k0) mypos = (uint32_t)(off - fr.begin);
                    got++;
                    P += payload;
                    off += fs;
                    c += pad;
                }
                if (got) { o.sample_rate = hr.sr; o.channels = hr.mono ? 1 : 2; o.bitrate = hr.bitrate; }
            }
        }
        for (int k = k0; k < 32 && !done; k++) {
            if (!(fend > off + 4)) { done = true; break; }
            const int64_t kbase = __shfl_sync(0xFFFFFFFFu, wbase, k);
            uint32_t b0, b1, b2, b3;
            const int64_t d = off - kbase;
            if (d >= 0 && d + 4 <= WALK_WIN) {
                const uint8_t *q = winb + k * (4 * WALK_STRIDE) + d;
                b0 = q[0]; b1 = q[1]; b2 = q[2]; b3 = q[3];
            } else {
                b0 = ldb(bytes, off, fend); b1 = ldb(bytes, off + 1, fend); b2 = ldb(bytes, off + 2, fend); b3 = ldb(bytes, off + 3, fend);
            }
            if (!(b0 == 0xFF && b1 >= 0xE0)) { o.status |= M3S_FILE_TRAILING_JUNK; done = true; break; }
            M3sHdr h;
            if (parse_header(b1, b2, b3, h) < 0) { o.status |= M3S_FILE_UNSUPPORTED; done = true; break; }
            const int64_t avail = fend - off;
            const int fs = h.frame_size < avail ? h.frame_size : (int)avail;
            int payload = fs - h.hdrlen;
            if (payload < 0) payload = 0;
            if (lane == k) mypos = (uint32_t)(off - fr.begin);
            got++;
            P += payload;
            o.sample_rate = h.sr;
            o.channels = h.mono ? 1 : 2;
            o.bitrate = h.bitrate;
            fs_guess = (144 * h.bitrate) / h.sr;
            off += h.frame_size;
        }
        if (lane < got) tmp_pos[fr.tmp_base + n + lane] = mypos;
        n += got;
        __syncwarp();
    }
    o.n_frames = n;
    o.payload_total = P;
    if (lane == 0) fouts[f] = o;
}

// ================================================================================================
// D0a'': the wave's layout, one CTA: exclusive prefix sums over the files of the frame counts (global frame index of each file's
// first frame) and of the main-data bytes (position of each file's header-stripped stream in S), written into the device file
// records -- the host does not have to see the walk's result before the per-frame kernels can be launched.  Each file's stream is
// preceded by M3S_APX_BYTES of assembly slots for its first nine frames (see resv_plan) and 512 zero bytes.
// ================================================================================================
#define M3S_APX_SLOTS 9
#define M3S_APX_SLOT_BYTES 2048
#define M3S_APX_BYTES (M3S_APX_SLOTS * M3S_APX_SLOT_BYTES)
#define M3S_META_IRR (1u << 26)           // fr_meta: the frame's main data is assembled explicitly into a slot (k_reservoir_fix)

__global__ void __launch_bounds__(256)
k_layout(M3sFileRec *__restrict__ files, const M3sFileOut *__restrict__ fouts, int n_files, int64_t frames_cap, M3sLayout *lay)
{
    __shared__ int64_t s_fr[256], s_sb[256];
    __shared__ int64_t carry_fr, carry_sb;
    const int tid = threadIdx.x;
    if (tid == 0) { carry_fr = 0; carry_sb = 0; }
    __syncthreads();
    for (int base = 0; base < n_files; base += 256) {
        const int f = base + tid;
        int64_t nfr = 0, sbytes = 0;
        if (f < n_files) {
            nfr = fouts[f].n_frames;
            sbytes = M3S_APX_BYTES + 512 + ((fouts[f].payload_total + 15) & ~(int64_t)15) + 64;
        }
        s_fr[tid] = nfr; s_sb[tid] = sbytes;
        __syncthreads();
        for (int d = 1; d < 256; d <<= 1) {
            int64_t a = 0, b = 0;
            if (tid >= d) { a = s_fr[tid - d]; b = s_sb[tid - d]; }
            __syncthreads();
            s_fr[tid] += a; s_sb[tid] += b;
            __syncthreads();
        }
        if (f < n_files) {
            files[f].frame_base = carry_fr + s_fr[tid] - nfr;
            files[f].s_base = carry_sb + s_sb[tid] - sbytes + M3S_APX_BYTES + 512;
            files[f].n_frames = (int32_t)nfr;
            files[f].flags = fouts[f].status;
            files[f].channels = fouts[f].channels;
        }
        __syncthreads();
        if (tid == 255) { carry_fr += s_fr[255]; carry_sb += s_sb[255]; }
        __syncthreads();
    }
    if (tid == 0) {
        lay->total_frames = carry_fr;
        lay->s_bytes = carry_sb + 64;
        lay->irregular = 0;
        lay->overflow = carry_fr > frames_cap ? 1 : 0;
        lay->pad = 0;
    }
}

// ================================================================================================
// D0a': per-file scans over the frames found by the walk, one warp per file, one frame per lane:
// payload prefix (position in the header-stripped stream), the carried table_select[2] of window-switched
// granules (A.D3: FrameSideInformation.py:104-107 parses only two selects, the third keeps its old value)
// and the reveal-bit offset (number of non-zero table ids in earlier frames, util.py:67-81).
// ================================================================================================
#define FSCAN_STRIDE 17  // words per lane (64-byte window + pad: conflict-free)

__device__ __forceinline__ uint32_t sbits(const uint8_t *w, int bitoff, int n)  // n <= 16, MSB first, from a staged window
{
    const uint8_t *q = w + (bitoff >> 3);
    uint32_t v = ((uint32_t)q[0] << 16) | ((uint32_t)q[1] << 8) | (uint32_t)q[2];
    return (v >> (24 - (bitoff & 7) - n)) & ((1u << n) - 1u);
}

__global__ void __launch_bounds__(32 * WALK_WARPS)
k_fscan(const uint8_t *__restrict__ bytes, int64_t total_bytes, const M3sFileRec *__restrict__ files, M3sFileOut *fouts,
        int n_files, const uint32_t *__restrict__ tmp_pos, int64_t *__restrict__ fr_pos, uint32_t *__restrict__ fr_P,
        uint32_t *__restrict__ fr_meta, uint32_t *__restrict__ fr_carry, uint32_t *__restrict__ fr_reveal,
        int32_t *__restrict__ fr_file, const M3sLayout *__restrict__ lay)
{
    __shared__ uint32_t s_win[WALK_WARPS][32 * FSCAN_STRIDE + 4];
    const int lane = threadIdx.x & 31, wip = threadIdx.x >> 5;
    const int f = blockIdx.x * WALK_WARPS + wip;
    if (f >= n_files || lay->overflow) return;   // overflow: the per-frame arrays are too small, the host grows them and rescans
    const M3sFileRec fr = files[f];
    const int64_t fend = fr.end;
    const int64_t align_fix = (int64_t)((uintptr_t)bytes & 15);
    uint32_t *win = s_win[wip] + lane * FSCAN_STRIDE;
    const bool junk = (fr.flags & M3S_FILE_TRAILING_JUNK) != 0;
    uint32_t carry_in = 0;   // 5 bits per (gr, ch) slot
    uint32_t P_in = 0, reveal_in = 0;
    bool state_carry = false;   // a granule inherits scalefactors from earlier frames (M3S_FILE_STATE_CARRY)
    uint32_t seen_mono = 0, seen_stereo = 0;
    for (int n0 = 0; n0 < fr.n_frames; n0 += 32) {
        const int n = n0 + lane;
        const bool valid = n < fr.n_frames;
        uint32_t payload = 0, meta = 0, nzfix = 0, t2pack = 0, wsmask = 0xFu;
        int64_t pos = 0;
        uint32_t nz01 = 0;
        if (valid) {
            pos = fr.begin + (int64_t)tmp_pos[fr.tmp_base + n];
            const int64_t wbase = ((pos + align_fix) & ~(int64_t)15) - align_fix;
#pragma unroll
            for (int q = 0; q < 4; q++) {  // 64 bytes from wbase always cover header + CRC + side info (pos - wbase <= 15, <= 38 bytes)
                const uint4 v = load16_clipped(bytes, wbase + 16 * q, fend, total_bytes);
                win[4 * q + 0] = v.x; win[4 * q + 1] = v.y; win[4 * q + 2] = v.z; win[4 * q + 3] = v.w;
            }
        }
        __syncwarp();
        if (valid) {
            const int64_t wbase = ((pos + align_fix) & ~(int64_t)15) - align_fix;
            const int d = (int)(pos - wbase);
            const uint8_t *wb = (const uint8_t *)win + d;
            M3sHdr h;
            parse_header(wb[1], wb[2], wb[3], h);  // validated by the walk
            const int64_t avail = fend - pos;
            const int fs = h.frame_size < avail ? h.frame_size : (int)avail;
            int pl = fs - h.hdrlen;
            if (pl < 0) pl = 0;
            payload = (uint32_t)pl;
            meta = (uint32_t)pl | (h.crc_present ? M3S_META_CRC : 0) | ((uint32_t)h.mode << M3S_META_MODE_SHIFT) |
                   (h.ms ? M3S_META_MS : 0) | ((uint32_t)h.sr_idx << M3S_META_SR_SHIFT) | (h.mono ? M3S_META_MONO : 0) |
                   (n == 0 ? M3S_META_FIRST : 0) | ((uint32_t)h.hdrlen << M3S_META_HDR_SHIFT) |
                   ((junk && n == fr.n_frames - 1) ? M3S_META_DUP : 0);
            const int si = 4 + (h.crc_present ? 2 : 0);
            int rb = h.mono ? 18 : 20;
            wsmask = 0xFu;
            const uint32_t scfsi_all = h.mono ? sbits(wb + si, 14, 4) << 4 : sbits(wb + si, 12, 8);   // ch0 in the high nibble
            for (int gr = 0; gr < 2; gr++)
                for (int ch = 0; ch < (h.mono ? 1 : 2); ch++) {
                    const int slot = 2 * gr + ch;
                    uint32_t ws, t0, t1, t2 = 0;
                    const uint8_t *sp = wb + si;
                    ws = sbits(sp, rb + 33, 1);
                    if (ws && sbits(sp, rb + 34, 2) == 2) {   // short block: mixed, or granule 0 under a non-zero scfsi of its channel
                        if (sbits(sp, rb + 36, 1)) state_carry = true;
                        if (gr == 0 && ((scfsi_all >> (ch ? 0 : 4)) & 15u)) state_carry = true;
                    }
                    if (ws) { t0 = sbits(sp, rb + 37, 5); t1 = sbits(sp, rb + 42, 5); }
                    else { t0 = sbits(sp, rb + 34, 5); t1 = sbits(sp, rb + 39, 5); t2 = sbits(sp, rb + 44, 5); }
                    nz01 += (t0 != 0) + (t1 != 0);
                    if (!ws) { wsmask &= ~(1u << slot); t2pack |= t2 << (5 * slot); }
                    rb += 59;
                }
            nzfix = h.mono ? 0x5u : 0xFu;  // slots that exist in this frame
        }
        seen_mono |= __ballot_sync(0xFFFFFFFFu, valid && (meta & M3S_META_MONO));
        seen_stereo |= __ballot_sync(0xFFFFFFFFu, valid && !(meta & M3S_META_MONO));
        // ---- carry scan: carry after frame k, slot s = t2 of the latest frame <= k that parsed slot s without window switching
        uint32_t carry = 0;
        uint32_t nz = nz01;
#pragma unroll
        for (int s = 0; s < 4; s++) {
            const uint32_t upd = __ballot_sync(0xFFFFFFFFu, valid && !((wsmask >> s) & 1u));
            const uint32_t le = upd & (0xFFFFFFFFu >> (31 - lane));
            const int src = le ? 31 - __clz(le) : 0;
            const uint32_t v = __shfl_sync(0xFFFFFFFFu, (t2pack >> (5 * s)) & 31u, src);
            const uint32_t c = le ? v : (carry_in >> (5 * s)) & 31u;
            carry |= c << (5 * s);
            if (valid && ((nzfix >> s) & 1u)) nz += c != 0;  // effective region-2 id of the slot: own value or the stale one
        }
        // ---- prefix sums of payload and non-zero table count
        uint32_t pP = payload, pR = nz;
#pragma unroll
        for (int dlt = 1; dlt < 32; dlt <<= 1) {
            const uint32_t a = __shfl_up_sync(0xFFFFFFFFu, pP, dlt), b = __shfl_up_sync(0xFFFFFFFFu, pR, dlt);
            if (lane >= dlt) { pP += a; pR += b; }
        }
        if (valid) {
            const int64_t g = fr.frame_base + n;
            fr_pos[g] = pos;
            fr_P[g] = P_in + pP - payload;
            fr_meta[g] = meta;
            fr_carry[g] = carry;
            fr_reveal[g] = reveal_in + pR - nz;
            fr_file[g] = f;
        }
        carry_in = __shfl_sync(0xFFFFFFFFu, carry, 31);  // lanes past the last frame update nothing: same carry as the last frame
        P_in += __shfl_sync(0xFFFFFFFFu, pP, 31);
        reveal_in += __shfl_sync(0xFFFFFFFFu, pR, 31);
        __syncwarp();
    }
    state_carry = __any_sync(0xFFFFFFFFu, state_carry);
    if (lane == 0) {
        fouts[f].reveal_len = (int32_t)reveal_in;
        if (state_carry) fouts[f].status |= M3S_FILE_STATE_CARRY;
        if (seen_mono && seen_stereo) fouts[f].status |= M3S_FILE_CHANNEL_SWITCH;
    }
}

// ================================================================================================
// Bit reservoir, the reference's way (Frame.py:318-363).  A frame's main data is the `main_data_begin` bytes in front of its header,
// skipping the headers + side infos of the frames in between, then its own payload.  On the header-stripped stream S that is plain
// addressing (start = sum of earlier payloads - main_data_begin) -- as long as every byte comes out of an earlier frame's payload.
// The reference does NOT require that; it applies its formula to whatever lies in front of the frame:
//   * it remembers the sizes of 9 earlier frames, the list starting (A.D9) with a phantom copy of frame 0 in front of the file
//     (MP3Parser.__init__ calls set_frame_size once more than there are frames), then zeros;
//   * it takes the CURRENT frame's header + side-info length C for every earlier frame (mono / stereo or CRC changes shift the cut);
//   * the window search `main_data_begin < bound` may fail within the first 8 frames of a file: main_data then stays what the
//     PREVIOUS frame assembled (a cut stream whose first frames still point into the missing part);
//   * bytes "of the phantom frame" are the bytes physically in front of frame 0 (an ID3 tag), with Python's slice rules when the
//     position is negative.
// resv_plan() decides which of the three a frame is; the irregular ones get their main data assembled byte by byte into a slot
// (k_reservoir_fix) and their unit records point there.
// ================================================================================================
struct M3sResvPlan {
    int kind;        // 0: regular (S addressing)   1: assembled from the segments below + own payload   2: stale (no window matched)
    int nseg;
    int total;       // bytes of the segments (without the own payload)
    int64_t lo[10];  // absolute batch positions
    int len[10];
};

__device__ __forceinline__ void py_slice(int64_t a, int64_t b, int64_t n, int64_t &lo, int64_t &len)   // list[a:b] of a list of n
{
    if (a < 0) { a += n; if (a < 0) a = 0; }
    if (b < 0) { b += n; if (b < 0) b = 0; }
    if (a > n) a = n;
    if (b > n) b = n;
    lo = a;
    len = b > a ? b - a : 0;
}

__device__ __forceinline__ int nominal_frame_size(const uint8_t *bytes, int64_t pos, int64_t fend)
{
    M3sHdr h;
    if (parse_header(ldb(bytes, pos + 1, fend), ldb(bytes, pos + 2, fend), ldb(bytes, pos + 3, fend), h) < 0) return 0;
    return h.frame_size;
}

// g: global frame index, n: its index inside the file, mdb > 0
__device__ __noinline__ void resv_plan(const uint8_t *__restrict__ bytes, const M3sFileRec &fr, const int64_t *__restrict__ fr_pos,
                                       const uint32_t *fr_meta, int64_t g, int n, int mdb, M3sResvPlan &pl)
{
    const int C = (int)((fr_meta[g] >> M3S_META_HDR_SHIFT) & 63u);
    pl.nseg = 0;
    pl.total = 0;
    // ---- regular: every byte comes out of the payload of a real earlier frame with the same C
    {
        int acc = 0;
        const int lim = n < 9 ? n : 9;
        for (int i = 1; i <= lim; i++) {
            if ((int)((fr_meta[g - i] >> M3S_META_HDR_SHIFT) & 63u) != C) break;
            acc += (int)(fr_pos[g - i + 1] - fr_pos[g - i]) - C;
            if (mdb <= acc) { pl.kind = 0; return; }
        }
    }
    // ---- the reference's search, literally
    int prev[9];
    for (int i = 0; i < 9; i++) {
        if (i < n) prev[i] = (int)(fr_pos[g - i] - fr_pos[g - 1 - i]);
        else if (i == n) prev[i] = nominal_frame_size(bytes, fr_pos[g - n], fr.end);
        else prev[i] = 0;
    }
    const int64_t curr = fr_pos[g] - fr.begin, flen = fr.end - fr.begin;
    int bound = 0;
    for (int frame = 0; frame < 9; frame++) {
        bound += prev[frame] - C;
        if (mdb < bound) {
            int part[9];
            part[frame] = mdb;
            for (int i = 0; i < frame; i++) { part[i] = prev[i] - C; part[frame] -= part[i]; }
            int64_t ptr = (int64_t)mdb + (int64_t)frame * C;
            for (int i = frame; i >= 0; i--) {
                const int64_t loc = curr - ptr;
                int64_t lo, len;
                py_slice(loc, loc + part[i], flen, lo, len);
                pl.lo[pl.nseg] = fr.begin + lo;
                pl.len[pl.nseg] = (int)len;
                pl.total += (int)len;
                pl.nseg++;
                ptr -= part[i] + C;
            }
            pl.kind = 1;
            return;
        }
    }
    pl.kind = 2;
}

// ================================================================================================
// D0b + D4: side-info parse, one thread per frame (FrameSideInformation.py:39-137), bit cursors through
// the reservoir (Frame.py:318-363 restated on the header-stripped stream S), table ids and reveal chars
// (Frame.py:676-685, util.py:67-81).
// ================================================================================================
__global__ void k_sideinfo(const uint8_t *__restrict__ bytes, const M3sFileRec *__restrict__ files, M3sLayout *lay,
                           const int64_t *__restrict__ fr_pos, const uint32_t *__restrict__ fr_P,
                           uint32_t *fr_meta, const uint32_t *__restrict__ fr_carry,
                           const uint32_t *__restrict__ fr_reveal, const int32_t *__restrict__ fr_file, M3sUnitRec *units,
                           uint8_t *tabids, uint8_t *reveal, uint32_t *irr, M3sFileOut *fouts)
{
    int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (lay->overflow || g >= lay->total_frames) return;
    int f = fr_file[g];
    const M3sFileRec fr = files[f];
    uint32_t meta = fr_meta[g];
    int mono = (meta & M3S_META_MONO) != 0;
    int64_t fend = fr.end;
    int64_t si = fr_pos[g] + 4 + ((meta & M3S_META_CRC) ? 2 : 0);
    uint32_t carry = fr_carry[g];
    uint32_t mdb = bits_at(bytes, si, fend, 0, 9);
    uint32_t scfsi_all = mono ? bits_at(bytes, si, fend, 14, 4) << 4 : bits_at(bytes, si, fend, 12, 8);
    int rb = mono ? 18 : 20;
    int payload = meta & M3S_META_PAYLOAD_MASK;
    int64_t cur = 8 * (fr.s_base + (int64_t)fr_P[g] - (int64_t)mdb);
    int64_t limit = 8 * (fr.s_base + (int64_t)fr_P[g] + payload);
    if (mdb) {
        const int n = (int)(g - fr.frame_base);
        M3sResvPlan pl;
        resv_plan(bytes, fr, fr_pos, fr_meta, g, n, (int)mdb, pl);
        if (pl.kind != 0) {
            int64_t k = g;          // the frame whose assembled main data this frame reads
            int kn = n;
            uint32_t kmdb = mdb;
            while (pl.kind == 2 && kn > 0) {   // stale: what the previous frame assembled (at most 7 steps, first frames of a file only)
                k--; kn--;
                const uint32_t km = fr_meta[k];
                kmdb = bits_at(bytes, fr_pos[k] + 4 + ((km & M3S_META_CRC) ? 2 : 0), fend, 0, 9);
                if (kmdb == 0) { pl.kind = 0; break; }
                resv_plan(bytes, fr, fr_pos, fr_meta, k, kn, (int)kmdb, pl);
            }
            const int kpayload = (int)(fr_meta[k] & M3S_META_PAYLOAD_MASK);
            if (pl.kind == 2) {            // frame 0 found no window either: main_data is still the empty list
                cur = 8 * fr.s_base;
                limit = cur;
            } else if (pl.kind == 0) {
                cur = 8 * (fr.s_base + (int64_t)fr_P[k] - (int64_t)kmdb);
                limit = 8 * (fr.s_base + (int64_t)fr_P[k] + kpayload);
            } else {
                int64_t slot_addr;
                if (kn < M3S_APX_SLOTS) {
                    slot_addr = fr.s_base - 512 - M3S_APX_BYTES + (int64_t)kn * M3S_APX_SLOT_BYTES;
                    if (k == g) { meta |= M3S_META_IRR; fr_meta[g] = meta; }
                } else {   // only reached with k == g: the stale chain never leaves the first 8 frames
                    const unsigned long long slot = atomicAdd((unsigned long long *)&lay->irregular, 1ULL);
                    irr[slot] = (uint32_t)g;
                    slot_addr = lay->s_bytes + (int64_t)slot * M3S_APX_SLOT_BYTES;
                }
                cur = 8 * slot_addr;
                limit = 8 * (slot_addr + pl.total + kpayload);
            }
        }
    }
    uint8_t ids[12];
#pragma unroll
    for (int i = 0; i < 12; i++) ids[i] = 0;
    M3sUnitRec inval;
    inval.bit_start = 0; inval.limit_bits = 0; inval.a = 0; inval.b = 0; inval.frame = (uint32_t)g; inval.pad = 0;
    inval.c = (meta & M3S_META_FIRST) ? (1u << 18) : 0;   // the backward walks for stale scalefactors stop at a file's first frame
    if (mono) { units[4 * g + 1] = inval; units[4 * g + 3] = inval; }
    for (int gr = 0; gr < 2; gr++)
        for (int ch = 0; ch < (mono ? 1 : 2); ch++) {
            int slot = 2 * gr + ch;
            uint32_t p23 = bits_at(bytes, si, fend, rb, 12);
            uint32_t bv = bits_at(bytes, si, fend, rb + 12, 9);
            uint32_t gg = bits_at(bytes, si, fend, rb + 21, 8);
            uint32_t sfc = bits_at(bytes, si, fend, rb + 29, 4);
            uint32_t ws = bits_at(bytes, si, fend, rb + 33, 1);
            uint32_t bt = 0, mixed = 0, t0, t1, t2, r0, r1, sbg = 0;
            if (ws) {
                bt = bits_at(bytes, si, fend, rb + 34, 2);
                mixed = bits_at(bytes, si, fend, rb + 36, 1);
                t0 = bits_at(bytes, si, fend, rb + 37, 5);
                t1 = bits_at(bytes, si, fend, rb + 42, 5);
                t2 = (carry >> (5 * slot)) & 31u;  // stale region-2 id (A.D3)
                sbg = bits_at(bytes, si, fend, rb + 47, 3) | (bits_at(bytes, si, fend, rb + 50, 3) << 3) |
                      (bits_at(bytes, si, fend, rb + 53, 3) << 6);
                r0 = bt == 2 ? 8 : 7;
                r1 = 20 - r0;  // kept in 4 bits below; only used when not (ws && bt == 2)
            } else {
                t0 = bits_at(bytes, si, fend, rb + 34, 5);
                t1 = bits_at(bytes, si, fend, rb + 39, 5);
                t2 = bits_at(bytes, si, fend, rb + 44, 5);
                r0 = bits_at(bytes, si, fend, rb + 49, 4);
                r1 = bits_at(bytes, si, fend, rb + 53, 3);
            }
            uint32_t pre = bits_at(bytes, si, fend, rb + 56, 1);
            uint32_t sfs = bits_at(bytes, si, fend, rb + 57, 1);
            uint32_t c1 = bits_at(bytes, si, fend, rb + 58, 1);
            M3sUnitRec u;
            u.bit_start = (uint64_t)cur;
            int64_t lb = limit - cur;
            u.limit_bits = lb > 0x7FFFFFFF ? 0x7FFFFFFF : (lb < -0x7FFFFFFF ? -0x7FFFFFFF : (int32_t)lb);
            u.a = p23 | (bv << 12) | (gg << 21) | (ws << 29) | (bt << 30);
            // region1 of a window-switched granule (12 or 13) does not fit 3 bits: store region0+region1+2 capped to 22 instead
            uint32_t r01 = r0 + r1 + 2;
            if (bv > 288 || r01 > 22) atomicOr(&fouts[f].status, M3S_FILE_BAD_SIDEINFO);   // the reference raises IndexError here; k_huff clamps
            if (r01 > 22) r01 = 22;
            u.b = sfc | (mixed << 4) | (t0 << 5) | (t1 << 10) | (t2 << 15) | (r0 << 20) | ((uint32_t)(meta & M3S_META_MS ? 1 : 0) << 30) |
                  ((uint32_t)mono << 31) | (pre << 27) | (sfs << 28) | (c1 << 29);
            uint32_t scfsi = ch == 0 ? (scfsi_all >> 4) & 15u : scfsi_all & 15u;
            u.c = sbg | (scfsi << 9) | (((meta >> M3S_META_SR_SHIFT) & 3u) << 13) | ((uint32_t)gr << 15) | ((uint32_t)ch << 16) |
                  (1u << 17) | ((meta & M3S_META_FIRST) ? (1u << 18) : 0) | (r01 << 19);
            u.frame = (uint32_t)g;
            u.pad = 0;
            units[4 * g + slot] = u;
            ids[ch * 6 + gr * 3 + 0] = (uint8_t)t0;
            ids[ch * 6 + gr * 3 + 1] = (uint8_t)t1;
            ids[ch * 6 + gr * 3 + 2] = (uint8_t)t2;
            cur += p23;
            rb += 59;
        }
    uint8_t *rv = reveal + 12 * fr.frame_base + fr_reveal[g];
    int j = 0;
#pragma unroll
    for (int i = 0; i < 12; i++) {
        tabids[12 * g + i] = ids[i];
        if (ids[i]) rv[j++] = ((M3S_H0_MASK >> ids[i]) & 1u) ? '0' : '1';
    }
}

// ================================================================================================
// main-data compaction: copy every frame's payload (bytes after header/CRC/side info, clipped to the
// file) to its position in the header-stripped stream S, one warp per frame.
// ================================================================================================
__global__ void k_strip(const uint8_t *__restrict__ bytes, int64_t total_bytes, const M3sFileRec *__restrict__ files,
                        int64_t g_lo, int64_t g_hi, const int64_t *__restrict__ fr_pos, const uint32_t *__restrict__ fr_P,
                        const uint32_t *__restrict__ fr_meta, const int32_t *__restrict__ fr_file, uint8_t *S)
{
    int64_t g = g_lo + (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    int lane = threadIdx.x & 31;
    if (g >= g_hi) return;
    uint32_t meta = fr_meta[g];
    int n = meta & M3S_META_PAYLOAD_MASK;
    int64_t src = fr_pos[g] + ((meta >> M3S_META_HDR_SHIFT) & 63);
    int64_t dst = files[fr_file[g]].s_base + fr_P[g];
    int head = (int)((4 - (dst & 3)) & 3);
    if (head > n) head = n;
    if (lane < head) S[dst + lane] = bytes[src + lane];
    int nwords = (n - head) >> 2;
    const uint8_t *sp = bytes + src + head;
    uint32_t *dp = (uint32_t *)(S + dst + head);
    uintptr_t sa = (uintptr_t)sp;
    int sh = (int)(sa & 3);
    const uint32_t *sw = (const uint32_t *)(sa - sh);
    // the aligned two-word read may touch up to 7 bytes past the last payload byte: keep it inside the batch buffer
    int64_t safe_words = (total_bytes - (src + head) - 8) >> 2;
    const int nfast = (int)(safe_words < 0 ? 0 : (safe_words < nwords ? safe_words : nwords));   // words the two-word reads may serve
    int wi = lane;
    for (; wi + 96 < nfast; wi += 128) {   // four words per lane with all eight loads in flight: the kernel waits on DRAM latency, not on bandwidth
        uint32_t lo[4], hi[4];
#pragma unroll
        for (int q = 0; q < 4; q++) { lo[q] = __ldg(sw + wi + 32 * q); hi[q] = __ldg(sw + wi + 32 * q + 1); }
#pragma unroll
        for (int q = 0; q < 4; q++) dp[wi + 32 * q] = __funnelshift_r(lo[q], hi[q], 8 * sh);
    }
    for (; wi < nfast; wi += 32) dp[wi] = __funnelshift_r(__ldg(sw + wi), __ldg(sw + wi + 1), 8 * sh);
    for (int wt = nfast + lane; wt < nwords; wt += 32) {   // the last words of the batch buffer, byte by byte
        const uint8_t *q = sp + 4 * wt;
        dp[wt] = (uint32_t)q[0] | ((uint32_t)q[1] << 8) | ((uint32_t)q[2] << 16) | ((uint32_t)q[3] << 24);
    }
    int tail = n - head - 4 * nwords;
    if (lane < tail) S[dst + head + 4 * nwords + lane] = bytes[src + head + 4 * nwords + lane];
    // the readers fetch whole 32-bit words and mask what lies beyond a frame's limit: give the word after a file's last payload byte
    // defined contents (S is not cleared)
    const M3sFileRec &fl = files[fr_file[g]];
    if (g == fl.frame_base + fl.n_frames - 1 && lane < 8) S[dst + n + lane] = 0;
}

// ================================================================================================
// Irregular bit reservoirs (see resv_plan): one warp per candidate frame -- the first nine frames of every file (flagged
// M3S_META_IRR by k_sideinfo) and the frames k_sideinfo listed in `irr` -- copies the segments the reference would assemble,
// then the frame's own payload, into the frame's slot.
// ================================================================================================
__global__ void k_reservoir_fix(const uint8_t *__restrict__ bytes, const M3sFileRec *__restrict__ files, int n_files,
                                const int64_t *__restrict__ fr_pos, const uint32_t *__restrict__ fr_meta,
                                const int32_t *__restrict__ fr_file, const uint32_t *__restrict__ irr, int64_t n_irr,
                                int64_t apx2_base, uint8_t *S)
{
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    int64_t g, slot_addr;
    int n;
    if (w < (int64_t)n_files * M3S_APX_SLOTS) {
        const int f = (int)(w / M3S_APX_SLOTS);
        n = (int)(w - (int64_t)f * M3S_APX_SLOTS);
        if (n >= files[f].n_frames) return;
        g = files[f].frame_base + n;
        if (!(fr_meta[g] & M3S_META_IRR)) return;
        slot_addr = files[f].s_base - 512 - M3S_APX_BYTES + (int64_t)n * M3S_APX_SLOT_BYTES;
    } else {
        const int64_t k = w - (int64_t)n_files * M3S_APX_SLOTS;
        if (k >= n_irr) return;
        g = irr[k];
        n = (int)(g - files[fr_file[g]].frame_base);
        slot_addr = apx2_base + k * M3S_APX_SLOT_BYTES;
    }
    const M3sFileRec fr = files[fr_file[g]];
    const uint32_t meta = fr_meta[g];
    const int64_t si = fr_pos[g] + 4 + ((meta & M3S_META_CRC) ? 2 : 0);
    const int mdb = (int)bits_at(bytes, si, fr.end, 0, 9);
    M3sResvPlan pl;
    resv_plan(bytes, fr, fr_pos, fr_meta, g, n, mdb, pl);
    if (pl.kind != 1) return;
    int64_t dst = slot_addr;
    for (int sg = 0; sg < pl.nseg; sg++) {
        for (int i = lane; i < pl.len[sg]; i += 32) S[dst + i] = bytes[pl.lo[sg] + i];
        dst += pl.len[sg];
    }
    const int own = (int)(meta & M3S_META_PAYLOAD_MASK);
    const int64_t src = fr_pos[g] + ((meta >> M3S_META_HDR_SHIFT) & 63);
    for (int i = lane; i < own; i += 32) S[dst + i] = bytes[src + i];
    if (lane < 8) S[dst + own + lane] = 0;   // (the word the readers fetch and mask at the end of the slot's contents)
}

// end of a scan: per-file results and the totals -> mapped host memory
__global__ void k_scan_publish(const M3sFileOut *__restrict__ fouts, int n_files, const M3sLayout *__restrict__ lay,
                               M3sFileOut *__restrict__ fouts_host, M3sLayout *__restrict__ lay_host)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_files) fouts_host[i] = fouts[i];
    if (i == 0) *lay_host = *lay;
}

// ================================================================================================
// D1: scalefactor + Huffman decode, one thread per granule-channel (Frame.py:365-559).
// ================================================================================================
struct BitReader {
    const uint32_t *w;  // word-aligned base in S
    int lim;            // bits readable relative to w (reads at or beyond read as zero)
    int pos;            // current bit position relative to w
    int idx;
    uint32_t hi, lo, nx;   // words idx, idx + 1 and idx + 2: the third one is fetched a whole word ahead of its first use, so its
                           // latency hides under the pairs decoded in between
    __device__ __forceinline__ uint32_t load(int wi) const
    {
        if (wi < (lim >> 5)) return __byte_perm(__ldg(w + wi), 0, 0x0123);   // whole word inside the limit: the common case
        const int b = wi * 32;
        if (b >= lim) return 0u;
        const uint32_t v = __byte_perm(__ldg(w + wi), 0, 0x0123);
        return v & ~(0xFFFFFFFFu >> (lim - b));
    }
    __device__ __forceinline__ void init(const uint8_t *S, uint64_t bit_start, int limit_bits)
    {
        uint64_t wbase = bit_start >> 5;
        w = (const uint32_t *)S + wbase;
        pos = (int)(bit_start & 31);
        lim = limit_bits > 0x7FFFFF00 ? 0x7FFFFF00 : limit_bits + pos;
        idx = 0;
        hi = load(0);
        lo = load(1);
        nx = load(2);
    }
    __device__ __forceinline__ uint32_t peek() const { return __funnelshift_l(lo, hi, pos & 31); }
    __device__ __forceinline__ void skip(int n)  // n <= 32
    {
        pos += n;
        int ni = pos >> 5;
        if (ni != idx) {
            hi = lo;
            lo = nx;
            nx = load(ni + 2);
            idx = ni;
        }
    }
    __device__ __forceinline__ uint32_t get(int n)  // n <= 16
    {
        if (n == 0) return 0u;
        uint32_t v = peek() >> (32 - n);
        skip(n);
        return v;
    }
};

// arbitrary-position read used by the rare stale-scalefactor paths (A.D4, scfsi from a non-long gr0)
__device__ __noinline__ uint32_t read_bits_at(const uint8_t *S, const M3sUnitRec &d, int rel_bit, int n)
{
    if (n == 0) return 0u;
    BitReader r;
    r.init(S, d.bit_start, d.limit_bits);
    // advance in <=32-bit steps
    int to = rel_bit;
    while (to > 0) { int s = to > 32 ? 32 : to; r.skip(s); to -= s; }
    return r.get(n);
}

// scale_fac_l[0][ch][sfb] as the reference's persistent array holds it when granule 1 copies it (Frame.py:419-437):
// the latest frame <= this one whose gr0 wrote that band.
__device__ __noinline__ uint32_t fetch_gr0_long_sf(const uint8_t *S, const M3sUnitRec *units, const M3sDevTables *T,
                                                   int64_t u_gr0, int sfb)
{
    for (int64_t u = u_gr0;; u -= 4) {
        const M3sUnitRec d = units[u];
        if (M3S_UC_VALID(d.c)) {   // not the placeholder of a mono frame's second channel: that frame wrote nothing to this slot
            uint32_t sl0 = T->slen[M3S_UB_SFC(d.b)][0], sl1 = T->slen[M3S_UB_SFC(d.b)][1];
            bool is_short = M3S_UA_BT(d.a) == 2 && M3S_UA_WS(d.a);
            if (!is_short) return read_bits_at(S, d, sfb < 11 ? sfb * sl0 : 11 * sl0 + (sfb - 11) * sl1, sfb < 11 ? sl0 : sl1);
            if (M3S_UB_MIXED(d.b) && sfb < 8) return read_bits_at(S, d, sfb * sl0, sl0);
        }
        if (M3S_UC_FIRST(d.c)) return 0u;
    }
}

// scale_fac_s[gr][ch][win][sfb<3] left behind by the latest earlier pure-short granule in the same slot (A.D4)
__device__ __noinline__ uint32_t fetch_stale_short_sf(const uint8_t *S, const M3sUnitRec *units, const M3sDevTables *T,
                                                      int64_t u_self, int win, int sfb)
{
    if (M3S_UC_FIRST(units[u_self].c)) return 0u;
    for (int64_t u = u_self - 4;; u -= 4) {
        const M3sUnitRec d = units[u];
        if (M3S_UC_VALID(d.c) && M3S_UA_BT(d.a) == 2 && M3S_UA_WS(d.a) && !M3S_UB_MIXED(d.b)) {
            uint32_t sl0 = T->slen[M3S_UB_SFC(d.b)][0];
            return read_bits_at(S, d, (sfb * 3 + win) * sl0, sl0);
        }
        if (M3S_UC_FIRST(d.c)) return 0u;
    }
}

#define HUFF_THREADS 256

// Bit reader of the Huffman loops: a 64-bit window whose top bit is the next unread bit, refilled 32 bits at a time from words that
// were loaded two refills earlier (a lane streams through its own granule; the latency of its loads hides under the pairs decoded in
// between).  After every consume() the window holds more than 32 valid bits, so one peek serves a whole code (<= 19 bits) plus
// both sign bits, or both linbits fields + signs (<= 28).  (A queue of 128-bit loads halved the load stalls but cost 47 % more
// instructions for its bookkeeping and was slower: the kernel is bound by instruction issue.)
struct BitWindow {
    const uint32_t *w;   // word-aligned base in S
    int lim;             // bits readable relative to w (reads at or beyond read as zero, util.get_bits, util.py:41-43)
    int pos;             // bits consumed relative to w
    int have;            // valid bits in win
    int nextw;           // index of the word held in n1
    uint64_t win;
    uint32_t n1, n2;     // word nextw (ready to use) and word nextw + 1 AS LOADED: its byte swap and tail mask wait until it moves into
                         // n1, one refill later -- done right behind the load they would stall on it, which is what the prefetch is there to avoid
    __device__ __forceinline__ uint32_t load_raw(int wi) const { return wi * 32 < lim ? __ldg(w + wi) : 0u; }
    __device__ __forceinline__ uint32_t fix(int wi, uint32_t raw) const   // big-endian word wi with the bits at or beyond lim cleared
    {
        const uint32_t v = __byte_perm(raw, 0, 0x0123);
        const int left = lim - wi * 32;                      // > 0 whenever raw was loaded; raw == 0 otherwise
        return left < 32 ? v & ~(0xFFFFFFFFu >> (left > 0 ? left : 0)) : v;
    }
    __device__ __forceinline__ uint32_t load(int wi) const { return fix(wi, load_raw(wi)); }
    __device__ __forceinline__ void init(const BitReader &r)   // continue where the scalefactor reader stopped
    {
        w = r.w; lim = r.lim; pos = r.pos;
        const int wi = pos >> 5, sh = pos & 31;
        win = (((uint64_t)load(wi) << 32) | (uint64_t)load(wi + 1)) << sh;
        have = 64 - sh;
        nextw = wi + 2;
        n1 = load(nextw);
        n2 = load_raw(nextw + 1);
    }
    __device__ __forceinline__ uint32_t peek() const { return (uint32_t)(win >> 32); }
    __device__ __forceinline__ void consume(int n)   // n <= 32
    {
        win <<= n;
        have -= n;
        pos += n;
        if (have <= 32) {
            win |= (uint64_t)n1 << (32 - have);
            have += 32;
            nextw++;
            n1 = fix(nextw, n2);
            n2 = load_raw(nextw + 1);
        }
    }
};

// One thread per granule-channel.  The three parts of a granule's spectrum -- big-value pairs, count1 quads, zeros -- run as three
// loops, so that the lanes of a warp (whose granules have different big_values) stay on the same code path within each loop.
__global__ void __launch_bounds__(HUFF_THREADS)
k_huff(const uint8_t *__restrict__ S, const M3sUnitRec *__restrict__ units, int64_t u_lo, int64_t u_hi,
       const M3sDevTables *__restrict__ T, uint32_t *__restrict__ spec, uint8_t *__restrict__ sfout)
{
    __shared__ uint16_t s_lut[8192];
    __shared__ uint32_t s_desc[32], s_sub[32];
    __shared__ uint8_t s_c1[64];
    __shared__ uint32_t s_sf[HUFF_THREADS][17];   // this thread's 64 scalefactor bytes (17-word rows: conflict-free); dynamically indexed
    for (int i = threadIdx.x; i < 4096; i += HUFF_THREADS) ((uint32_t *)s_lut)[i] = ((const uint32_t *)T->huff_lut)[i];
    if (threadIdx.x < 32) { s_desc[threadIdx.x] = T->huff_desc[threadIdx.x]; s_sub[threadIdx.x] = T->huff_sub[threadIdx.x]; }
    if (threadIdx.x < 64) s_c1[threadIdx.x] = T->count1_lut[threadIdx.x];
    __syncthreads();
    int64_t u = u_lo + (int64_t)blockIdx.x * HUFF_THREADS + threadIdx.x;
    if (u >= u_hi) return;
    const M3sUnitRec rec = units[u];
    uint32_t *out = spec + (u >> 2) * (288 * 4) + (u & 3);
    if (!M3S_UC_VALID(rec.c)) {   // the second channel of a mono frame: zero spectrum, zero scalefactors
        for (int k = 0; k < 288; k++) out[4 * k] = 0u;
        uint4 *so = (uint4 *)(sfout + u * M3S_SF_STRIDE);
        so[0] = so[1] = so[2] = so[3] = make_uint4(0u, 0u, 0u, 0u);
        return;
    }
    const uint32_t a = rec.a, b = rec.b, c = rec.c;
    const int gr = M3S_UC_GR(c), sr = M3S_UC_SR(c);
    const bool is_short = M3S_UA_BT(a) == 2 && M3S_UA_WS(a);
    BitReader br;
    br.init(S, rec.bit_start, rec.limit_bits);
    const int pos0 = br.pos;
    // ---------------------------------------------------------------- scalefactors (Frame.py:365-441)
    uint32_t *sfw = s_sf[threadIdx.x];
#pragma unroll
    for (int i = 0; i < 16; i++) sfw[i] = 0;
    uint8_t *sfb8 = (uint8_t *)sfw;
    {
        const int sl0 = T->slen[M3S_UB_SFC(b)][0], sl1 = T->slen[M3S_UB_SFC(b)][1];
        if (is_short) {
            if (M3S_UB_MIXED(b)) {
                br.skip(8 * sl0 > 32 ? 32 : 8 * sl0);  // scale_fac_l[0..7] are parsed but never used by the short requantize path (A.D2)
                for (int sfb = 0; sfb < 3; sfb++)
                    for (int w = 0; w < 3; w++) sfb8[M3S_SF_SHORT + 13 * w + sfb] = (uint8_t)fetch_stale_short_sf(S, units, T, u, w, sfb);
                for (int sfb = 3; sfb < 6; sfb++)
                    for (int w = 0; w < 3; w++) sfb8[M3S_SF_SHORT + 13 * w + sfb] = (uint8_t)br.get(sl0);
            } else {
                for (int sfb = 0; sfb < 6; sfb++)
                    for (int w = 0; w < 3; w++) sfb8[M3S_SF_SHORT + 13 * w + sfb] = (uint8_t)br.get(sl0);
            }
            for (int sfb = 6; sfb < 12; sfb++)
                for (int w = 0; w < 3; w++) sfb8[M3S_SF_SHORT + 13 * w + sfb] = (uint8_t)br.get(sl1);
        } else if (gr == 0) {
            for (int sfb = 0; sfb < 11; sfb++) sfb8[sfb] = (uint8_t)br.get(sl0);
            for (int sfb = 11; sfb < 21; sfb++) sfb8[sfb] = (uint8_t)br.get(sl1);
        } else {
            const uint32_t scfsi = M3S_UC_SCFSI(c);
            const int lo_[4] = {0, 6, 11, 16}, hi_[4] = {6, 11, 16, 21};
            for (int i = 0; i < 4; i++) {
                int sl = i < 2 ? sl0 : sl1;
                for (int sfb = lo_[i]; sfb < hi_[i]; sfb++) {
                    if ((scfsi >> (3 - i)) & 1u) sfb8[sfb] = (uint8_t)fetch_gr0_long_sf(S, units, T, u - 2, sfb);
                    else sfb8[sfb] = (uint8_t)br.get(sl);
                }
            }
        }
    }
    {
        uint4 *so = (uint4 *)(sfout + u * M3S_SF_STRIDE);
        so[0] = make_uint4(sfw[0], sfw[1], sfw[2], sfw[3]);
        so[1] = make_uint4(sfw[4], sfw[5], sfw[6], sfw[7]);
        so[2] = make_uint4(sfw[8], sfw[9], sfw[10], sfw[11]);
        so[3] = make_uint4(sfw[12], sfw[13], sfw[14], sfw[15]);
    }
    // ---------------------------------------------------------------- big values (Frame.py:443-519)
    int bv = M3S_UA_BV(a);
    if (bv > 288) bv = 288;  // the reference raises IndexError beyond 576 samples
    int r0p, r1p;
    if (is_short) { r0p = 18; r1p = 288; }
    else {
        r0p = T->sfb_long[sr][M3S_UB_R0(b) + 1] >> 1;
        r1p = T->sfb_long[sr][(c >> 19) & 31u] >> 1;
    }
    const uint32_t d0 = s_desc[M3S_UB_TS(b, 0)], d1 = s_desc[M3S_UB_TS(b, 1)], d2 = s_desc[M3S_UB_TS(b, 2)];
    const uint32_t sb0 = s_sub[M3S_UB_TS(b, 0)], sb1 = s_sub[M3S_UB_TS(b, 1)], sb2 = s_sub[M3S_UB_TS(b, 2)];
    BitWindow bw;
    bw.init(br);
    int k = 0;
    for (; k < bv; k++) {
        const uint32_t desc = k < r0p ? d0 : (k < r1p ? d1 : d2);
        const uint32_t sub = k < r0p ? sb0 : (k < r1p ? sb1 : sb2);
        const int l1b = (desc >> 13) & 15;
        uint32_t o = 0;
        if (l1b) {  // tables 0, 4 and 14 carry no codes: zeros, no bits consumed (A.D6)
            uint32_t wv = bw.peek();
            uint32_t e = s_lut[(desc & 0x1FFF) + (wv >> (32 - l1b))];
            if (e & 0x8000u) {
                const int nb = (e >> 11) & 15;
                e = s_lut[sub + ((e & 0x7FFu) << 1) + ((wv << l1b) >> (32 - nb))];
            }
            const int len = (e >> 8) & 31;
            int x = (e >> 4) & 15, y = e & 15;
            const int lb = (desc >> 17) & 15;
            int used;
            if (lb) {   // escape tables: code, then per value [linbits if 15] [sign if non-zero] (Frame.py:503-513)
                bw.consume(len);
                wv = bw.peek();
                used = 0;
                if (x == 15) { x += wv >> (32 - lb); wv <<= lb; used += lb; }
                if (x) { if (wv >> 31) x = -x; wv <<= 1; used++; }
                if (y == 15) { y += wv >> (32 - lb); wv <<= lb; used += lb; }
                if (y) { if (wv >> 31) y = -y; used++; }
            } else {
                wv <<= len;
                used = len;
                if (x) { if (wv >> 31) x = -x; wv <<= 1; used++; }
                if (y) { if (wv >> 31) y = -y; used++; }
            }
            bw.consume(used);
            o = ((uint32_t)x & 0xFFFFu) | ((uint32_t)y << 16);
        }
        out[4 * k] = o;
    }
    // ---------------------------------------------------------------- count1 quads (Frame.py:521-559): `while bit < max_bit and sample + 4 < 576`
    const bool c1b = M3S_UB_C1SEL(b);
    const int max_pos = pos0 + (int)M3S_UA_P23(a);
    while (bw.pos < max_pos && 2 * k + 4 < 576) {
        uint32_t wv = bw.peek();
        uint32_t q;  // v w x y in bits 3..0
        int used;
        if (c1b) { q = (~wv >> 28) & 15u; used = 4; }
        else { const uint32_t e = s_c1[wv >> 26]; q = e & 15u; used = e >> 4; }
        wv <<= used;
        int v0 = (q >> 3) & 1, v1 = (q >> 2) & 1, v2 = (q >> 1) & 1, v3 = q & 1;
        if (v0) { if (wv >> 31) v0 = -1; wv <<= 1; used++; }
        if (v1) { if (wv >> 31) v1 = -1; wv <<= 1; used++; }
        if (v2) { if (wv >> 31) v2 = -1; wv <<= 1; used++; }
        if (v3) { if (wv >> 31) v3 = -1; used++; }
        bw.consume(used);
        out[4 * k] = ((uint32_t)v0 & 0xFFFFu) | ((uint32_t)v1 << 16);
        out[4 * k + 4] = ((uint32_t)v2 & 0xFFFFu) | ((uint32_t)v3 << 16);
        k += 2;
    }
    // ---------------------------------------------------------------- the rest is zero
    for (; k < 288; k++) out[4 * k] = 0u;
}

// int16 [frame][gr][ch][576] parity tap from the pair-major spectra layout
__global__ void k_spec_export(const uint32_t *__restrict__ spec, int64_t total_frames, int16_t *__restrict__ out)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // one thread per (frame, pair, slot)
    if (i >= total_frames * 288 * 4) return;
    int slot = (int)(i & 3);
    int64_t r = i >> 2;
    int k = (int)(r % 288);
    int64_t g = r / 288;
    uint32_t v = spec[i];
    int16_t *o = out + ((g * 4 + slot) * 576 + 2 * k);
    o[0] = (int16_t)(v & 0xFFFF);
    o[1] = (int16_t)(v >> 16);
}

// ================================================================================================
// D2 + D3: requantize, MS stereo, reorder / alias, IMDCT + window + overlap, frequency inversion,
// polyphase synthesis, int16 pack: k_hybrid_fast (m3s_hybrid_fast.cuh).  One CTA walks a run of consecutive
// frames of one file; a run that does not start its file first re-decodes one warm-up frame (SURVEY.md 8e)
// whose PCM is discarded.
// (Frame.py:157-218 re_quantize, :561-572, :574-602, :604-622, :106-154 imdct, :624-631, :65-103 synth,
//  :633-640 interleave, MP3_Parser.py:91 int16 conversion)
// ================================================================================================
#include "m3s_hybrid_fast.cuh"

int m3s_upload_fast_const()
{
    M3sFastConst fc;   // twiddles of the fast transforms, in both precisions
    m3s_fast_const_build(fc);
    if (cudaMemcpyToSymbol(c_fast, &fc, sizeof fc) != cudaSuccess) return -1;
    M3sFastConstD fcd;
    m3s_fast_const_build(fcd);
    if (cudaMemcpyToSymbol(c_fast_d, &fcd, sizeof fcd) != cudaSuccess) return -1;
    return 0;
}

// ================================================================================================
// host orchestration
// ================================================================================================
#include <chrono>
static const bool g_trace = getenv("M3S_TRACE") != nullptr;   // host-clock stage timing of the decode calls (diagnostic)
static inline double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
#define M3S_TRACE_MARK(tag) do { if (g_trace) { const double t__ = now_ms(); fprintf(stderr, "[m3s %p] %-18s +%.2f ms\n", (void *)h, tag, t__ - tr_t); tr_t = t__; } } while (0)

static inline int64_t round_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

static int sync_all_streams(m3s_ctx *h)
{
    M3S_CUDA(h, cudaStreamSynchronize(h->stream));
    if (h->copy_in) {
        M3S_CUDA(h, cudaStreamSynchronize(h->copy_in));
        M3S_CUDA(h, cudaStreamSynchronize(h->copy_out));
        M3S_CUDA(h, cudaStreamSynchronize(h->aux));
    }
    return M3S_OK;
}

// grow-only reserve that is safe while other streams of the handle may still use the buffer
static int reserve_quiet(m3s_ctx *h, M3sBuf &b, size_t bytes)
{
    if (bytes <= b.cap) return M3S_OK;
    int rc = sync_all_streams(h);
    if (rc) return rc;
    return m3s_buf_reserve(h, b, bytes);
}

// small pinned staging areas (file records, work lists): an asynchronous copy out of PAGEABLE memory would first wait for the
// stream to drain, i.e. for the previous wave's kernels
static int pin_reserve(m3s_ctx *h, void *&p, size_t &cap, size_t bytes)
{
    if (bytes <= cap) return M3S_OK;
    int rc = sync_all_streams(h);
    if (rc) return rc;
    if (p) M3S_CUDA(h, cudaFreeHost(p));
    p = nullptr;
    cap = 0;
    const size_t want = bytes + bytes / 4 + 4096;
    M3S_CUDA(h, cudaHostAlloc(&p, want, cudaHostAllocDefault));
    cap = want;
    return M3S_OK;
}

// frames a file of `len` audio bytes can hold when its first header says `first4`; <= 0: no usable header
static int64_t frames_by_first_header(const uint8_t *p, int64_t len)
{
    if (len < 4 || p[0] != 0xFF || p[1] < 0xE0) return 0;
    const uint32_t b1 = p[1], b2 = p[2];
    if (((b1 >> 3) & 3) != 3 || ((b1 >> 1) & 3) != 1) return 0;
    const int sri = (b2 >> 2) & 3;
    int bi = (int)(b2 >> 4);
    if (sri == 3 || bi == 15) return 0;
    static const int br_tab[14] = {32, 40, 48, 56, 64, 80, 96, 112, 128, 160, 192, 224, 256, 320};
    bi = bi == 0 ? 13 : bi - 1;
    const int sr = sri == 0 ? 44100 : (sri == 1 ? 48000 : 32000);
    const int fs = 144 * br_tab[bi] * 1000 / sr;
    return len / fs + 2;
}

static int scan_reserve_frames(m3s_ctx *h, M3sScanSet &ss, int64_t frames)
{
    if (frames <= ss.frames_cap) return M3S_OK;
    const int64_t nf = frames + frames / 16 + 64;
    int rc;
    if ((rc = reserve_quiet(h, ss.fr_pos, sizeof(int64_t) * (nf + 1)))) return rc;
    if ((rc = reserve_quiet(h, ss.fr_P, sizeof(uint32_t) * nf))) return rc;
    if ((rc = reserve_quiet(h, ss.fr_meta, sizeof(uint32_t) * nf))) return rc;
    if ((rc = reserve_quiet(h, ss.fr_carry, sizeof(uint32_t) * nf))) return rc;
    if ((rc = reserve_quiet(h, ss.fr_reveal, sizeof(uint32_t) * nf))) return rc;
    if ((rc = reserve_quiet(h, ss.fr_file, sizeof(int32_t) * nf))) return rc;
    if ((rc = reserve_quiet(h, ss.irr, sizeof(uint32_t) * nf))) return rc;
    if ((rc = reserve_quiet(h, ss.units, sizeof(M3sUnitRec) * 4 * nf))) return rc;
    if ((rc = reserve_quiet(h, ss.tabids, 12 * nf))) return rc;
    if ((rc = reserve_quiet(h, ss.reveal, 12 * nf))) return rc;
    ss.frames_cap = nf;
    return M3S_OK;
}

// Queue the scan of one wave on stream `s` (no host synchronisation): walk -> layout -> per-file scans -> side info -> publish.
// `hint` (host copy of the wave's bytes, or NULL) sizes the per-frame arrays from every file's first header; device-resident input is
// sized from the bytes per frame earlier scans saw.  scan_finish() reads the result once `s` has passed this point.
static int scan_enqueue(m3s_ctx *h, M3sScanSet &ss, cudaStream_t s, const uint8_t *d_bytes, const uint8_t *hint, const int64_t *file_off,
                        const int64_t *audio_start, int32_t n_files, bool relaunch_only = false)
{
    int rc;
    M3sLaunchOn on(h, s);
    const int wg = (n_files + WALK_WARPS - 1) / WALK_WARPS;
    if (!relaunch_only) {
        const int64_t base = file_off[0];
        const int64_t total_bytes = file_off[n_files] - base;
        ss.n_files = n_files;
        ss.d_bytes = d_bytes;
        ss.total_bytes = total_bytes;
        ss.files_h.assign(n_files, M3sFileRec());
        ss.fouts_h.assign(n_files, M3sFileOut());
        int64_t tb = 0, est = 0;
        for (int i = 0; i < n_files; i++) {
            M3sFileRec &f = ss.files_h[i];
            f.begin = file_off[i] - base;
            f.end = file_off[i + 1] - base;
            f.audio = f.begin + (audio_start ? audio_start[i] : 0);
            if (f.audio > f.end) f.audio = f.end;
            f.frame_base = 0; f.s_base = 0; f.pcm_base = 0; f.n_frames = 0; f.flags = 0; f.channels = 0; f.pad = 0;
            if (f.end - f.begin > 0xFFFFFFFFLL) return m3s_fail(h, M3S_ERR_ARG, "decode: file %d exceeds 4 GiB", i);
            f.tmp_base = tb;
            tb += (f.end - f.audio) / 96 + 2;   // the walk's temporary position array is sized by the smallest legal frame (96 bytes)
            if (hint) est += frames_by_first_header(hint + f.audio, f.end - f.audio);
            else est += (int64_t)((double)(f.end - f.audio) / (h->dec_bpf_guess > 0 ? h->dec_bpf_guess : 417.0)) + 2;
        }
        if ((rc = reserve_quiet(h, ss.files, sizeof(M3sFileRec) * n_files))) return rc;
        if ((rc = reserve_quiet(h, ss.fouts, sizeof(M3sFileOut) * n_files))) return rc;
        if ((rc = reserve_quiet(h, ss.layout, sizeof(M3sLayout)))) return rc;
        if ((rc = reserve_quiet(h, ss.tmp_pos, sizeof(uint32_t) * (size_t)(tb + 32)))) return rc;
        if ((rc = scan_reserve_frames(h, ss, est + 8))) return rc;
        if ((size_t)n_files > ss.fouts_cap) {
            if ((rc = sync_all_streams(h))) return rc;
            if (ss.fouts_mapped) M3S_CUDA(h, cudaFreeHost(ss.fouts_mapped));
            ss.fouts_mapped = nullptr;
            ss.fouts_cap = 0;
            const size_t cap = (size_t)n_files + 64;
            M3S_CUDA(h, cudaHostAlloc((void **)&ss.fouts_mapped, sizeof(M3sFileOut) * cap + sizeof(M3sLayout), cudaHostAllocMapped));
            M3S_CUDA(h, cudaHostGetDevicePointer((void **)&ss.fouts_mdev, ss.fouts_mapped, 0));
            ss.lay_mapped = (M3sLayout *)(ss.fouts_mapped + cap);
            ss.lay_mdev = (M3sLayout *)(ss.fouts_mdev + cap);
            ss.fouts_cap = cap;
        }
        if ((rc = pin_reserve(h, ss.pin, ss.pin_cap, sizeof(M3sFileRec) * n_files))) return rc;
        memcpy(ss.pin, ss.files_h.data(), sizeof(M3sFileRec) * n_files);
        M3S_CUDA(h, cudaMemcpyAsync(ss.files.p, ss.pin, sizeof(M3sFileRec) * n_files, cudaMemcpyHostToDevice, s));
        M3S_KBEGIN(h, M3S_K_WALK);
        k_walk<<<wg, 32 * WALK_WARPS, 0, s>>>(ss.d_bytes, ss.total_bytes, (const M3sFileRec *)ss.files.p, (M3sFileOut *)ss.fouts.p,
                                               n_files, (uint32_t *)ss.tmp_pos.p);
        M3S_LAUNCH_CHECK(h);
    }
    // the reveal chars of a file fill only the first reveal_len bytes of its 12-bytes-per-frame area: clear the rest, it is copied out too
    M3S_CUDA(h, cudaMemsetAsync(ss.reveal.p, 0, (size_t)12 * (size_t)ss.frames_cap, s));
    M3S_KBEGIN(h, M3S_K_FSCAN);
    k_layout<<<1, 256, 0, s>>>((M3sFileRec *)ss.files.p, (const M3sFileOut *)ss.fouts.p, n_files, ss.frames_cap, (M3sLayout *)ss.layout.p);
    M3S_LAUNCH_CHECK(h);
    M3S_KBEGIN(h, M3S_K_FSCAN);
    k_fscan<<<wg, 32 * WALK_WARPS, 0, s>>>(ss.d_bytes, ss.total_bytes, (const M3sFileRec *)ss.files.p, (M3sFileOut *)ss.fouts.p, n_files,
                                            (const uint32_t *)ss.tmp_pos.p, (int64_t *)ss.fr_pos.p, (uint32_t *)ss.fr_P.p,
                                            (uint32_t *)ss.fr_meta.p, (uint32_t *)ss.fr_carry.p, (uint32_t *)ss.fr_reveal.p,
                                            (int32_t *)ss.fr_file.p, (const M3sLayout *)ss.layout.p);
    M3S_LAUNCH_CHECK(h);
    M3S_KBEGIN(h, M3S_K_SIDEINFO);
    k_sideinfo<<<(unsigned)((ss.frames_cap + 127) / 128), 128, 0, s>>>(
        ss.d_bytes, (const M3sFileRec *)ss.files.p, (M3sLayout *)ss.layout.p, (const int64_t *)ss.fr_pos.p, (const uint32_t *)ss.fr_P.p,
        (uint32_t *)ss.fr_meta.p, (const uint32_t *)ss.fr_carry.p, (const uint32_t *)ss.fr_reveal.p, (const int32_t *)ss.fr_file.p,
        (M3sUnitRec *)ss.units.p, (uint8_t *)ss.tabids.p, (uint8_t *)ss.reveal.p, (uint32_t *)ss.irr.p, (M3sFileOut *)ss.fouts.p);
    M3S_LAUNCH_CHECK(h);
    M3S_KBEGIN(h, M3S_K_SIDEINFO);
    k_scan_publish<<<(n_files + 255) / 256, 256, 0, s>>>((const M3sFileOut *)ss.fouts.p, n_files, (const M3sLayout *)ss.layout.p,
                                                          ss.fouts_mdev, ss.lay_mdev);
    M3S_LAUNCH_CHECK(h);
    return M3S_OK;
}

// After stream `s` has run the scan: read the results; when the per-frame arrays were too small (VBR files, a wrong guess) grow them
// and run the per-frame part again (synchronously -- the rare slow path).
static int scan_finish(m3s_ctx *h, M3sScanSet &ss, cudaStream_t s, const int64_t *file_off, const int64_t *audio_start)
{
    for (int attempt = 0;; attempt++) {
        const M3sLayout lay = *ss.lay_mapped;
        if (!lay.overflow) {
            memcpy(ss.fouts_h.data(), ss.fouts_mapped, sizeof(M3sFileOut) * ss.n_files);
            ss.total_frames = lay.total_frames;
            ss.s_bytes = lay.s_bytes;
            ss.irregular = lay.irregular;
            break;
        }
        if (attempt > 0) return m3s_fail(h, M3S_ERR_STATE, "decode: scan overflow persists");
        int rc = scan_reserve_frames(h, ss, lay.total_frames);
        if (rc) return rc;
        if ((rc = scan_enqueue(h, ss, s, ss.d_bytes, nullptr, file_off, audio_start, ss.n_files, true))) return rc;
        M3S_CUDA(h, cudaStreamSynchronize(s));
    }
    int64_t fb = 0, sb = 0, audio_bytes = 0;
    for (int i = 0; i < ss.n_files; i++) {   // the same layout k_layout computed on the device
        M3sFileRec &f = ss.files_h[i];
        const M3sFileOut &o = ss.fouts_h[i];
        f.frame_base = fb;
        f.n_frames = o.n_frames;
        f.flags = o.status;
        f.channels = o.channels;
        fb += f.n_frames;
        sb += M3S_APX_BYTES + 512;
        f.s_base = sb;
        sb += round_up(o.payload_total, 16) + 64;
        audio_bytes += f.end - f.audio;
    }
    if (fb != ss.total_frames || sb + 64 != ss.s_bytes) return m3s_fail(h, M3S_ERR_STATE, "decode: host and device layouts disagree");
    if (fb > 0) h->dec_bpf_guess = 0.97 * (double)audio_bytes / (double)fb;
    return M3S_OK;
}

static int decode_events_init(m3s_ctx *h)
{
    int rc = m3s_pipeline_init(h);
    if (rc) return rc;
    for (int i = 0; i < 2; i++) {
        if (h->ev_d_h2d[i]) continue;
        M3S_CUDA(h, cudaEventCreateWithFlags(&h->ev_d_h2d[i], cudaEventDisableTiming));
        M3S_CUDA(h, cudaEventCreateWithFlags(&h->ev_d_scan[i], cudaEventDisableTiming));
        M3S_CUDA(h, cudaEventCreateWithFlags(&h->ev_d_comp[i], cudaEventDisableTiming));
        M3S_CUDA(h, cudaEventCreateWithFlags(&h->ev_d_out[i], cudaEventDisableTiming));
    }
    return M3S_OK;
}

extern "C" int m3s_decode_scan(m3s_handle_t h, const uint8_t *bytes, int mem, const int64_t *file_off,
                               const int64_t *audio_start, int32_t n_files, int64_t *n_frames, int64_t *pcm_rows,
                               int32_t *sample_rate, int32_t *channels, int32_t *bitrate_bps, int32_t *status)
{
    if (!h) return M3S_ERR_ARG;
    h->scanned = false;
    if (!bytes || !file_off || n_files <= 0) return m3s_fail(h, M3S_ERR_ARG, "decode_scan: bytes/file_off/n_files");
    M3S_CUDA(h, cudaSetDevice(h->device));
    double tr_t = g_trace ? now_ms() : 0.0;
    for (int i = 0; i < n_files; i++)
        if (file_off[i + 1] < file_off[i] || (audio_start && (audio_start[i] < 0)))
            return m3s_fail(h, M3S_ERR_ARG, "decode_scan: file_off must be non-decreasing, audio_start >= 0");
    const int64_t total_bytes = file_off[n_files] - file_off[0];
    M3sScanSet &ss = h->ss[0];
    h->cur = &ss;
    int rc;
    const uint8_t *d_bytes = bytes + file_off[0];
    // ---- stage the bytes on the device when they are host memory
    if (mem == M3S_MEM_HOST) {
        if ((rc = m3s_buf_reserve(h, h->b_stage_in[0], (size_t)total_bytes + 16))) return rc;
        if ((rc = m3s_copy_paced(h, h->b_stage_in[0].p, bytes + file_off[0], (size_t)total_bytes, cudaMemcpyHostToDevice))) return rc;
        d_bytes = (const uint8_t *)h->b_stage_in[0].p;
    }
    M3S_TRACE_MARK("scan.h2d_submitted");
    if ((rc = scan_enqueue(h, ss, h->stream, d_bytes, mem == M3S_MEM_HOST ? bytes + file_off[0] : nullptr, file_off, audio_start, n_files)))
        return rc;
    M3S_TRACE_MARK("scan.launched");
    M3S_CUDA(h, cudaStreamSynchronize(h->stream));
    if ((rc = scan_finish(h, ss, h->stream, file_off, audio_start))) return rc;
    M3S_TRACE_MARK("scan.synced");
    for (int i = 0; i < n_files; i++) {
        const M3sFileOut &o = ss.fouts_h[i];
        if (n_frames) n_frames[i] = o.n_frames;
        if (pcm_rows) pcm_rows[i] = 1152LL * (o.n_frames + ((o.status & M3S_FILE_TRAILING_JUNK) && o.n_frames > 0 ? 1 : 0));
        if (sample_rate) sample_rate[i] = o.sample_rate;
        if (channels) channels[i] = o.channels;
        if (bitrate_bps) bitrate_bps[i] = o.bitrate;
        if (status) status[i] = o.status;
    }
    h->scanned = true;
    return M3S_OK;
}

// device -> mapped host memory by SM stores (one 32-bit word per thread, coalesced): the reveal outputs are small and the host
// thread waits for them, so they must not queue behind another handle's bulk PCM transfer in the copy engine
__global__ void k_words_out(const uint32_t *__restrict__ a, const uint32_t *__restrict__ b, int64_t n_words, uint32_t *__restrict__ out_a,
                            uint32_t *__restrict__ out_b)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_words) return;
    if (out_a) out_a[i] = a[i];
    if (out_b) out_b[i] = b[i];
}

extern "C" int m3s_decode_reveal(m3s_handle_t h, uint8_t *table_ids, uint8_t *reveal_bits, int mem, int64_t *reveal_len)
{
    if (!h) return M3S_ERR_ARG;
    if (!h->scanned) return m3s_fail(h, M3S_ERR_STATE, "decode_reveal: call m3s_decode_scan first");
    M3S_CUDA(h, cudaSetDevice(h->device));
    M3sScanSet &ss = *h->cur;
    if (reveal_len)
        for (int i = 0; i < ss.n_files; i++) reveal_len[i] = ss.fouts_h[i].reveal_len;
    const size_t nb = (size_t)12 * (size_t)ss.total_frames;   // bytes of each output (a multiple of 4)
    if (nb == 0 || (!table_ids && !reveal_bits)) return M3S_OK;
    if (mem != M3S_MEM_HOST) {
        if (table_ids) M3S_CUDA(h, cudaMemcpyAsync(table_ids, ss.tabids.p, nb, cudaMemcpyDeviceToDevice, h->stream));
        if (reveal_bits) M3S_CUDA(h, cudaMemcpyAsync(reveal_bits, ss.reveal.p, nb, cudaMemcpyDeviceToDevice, h->stream));
        M3S_CUDA(h, cudaStreamSynchronize(h->stream));
        return M3S_OK;
    }
    if (2 * nb > h->rev_cap) {
        M3S_CUDA(h, cudaStreamSynchronize(h->stream));
        if (h->rev_mapped) M3S_CUDA(h, cudaFreeHost(h->rev_mapped));
        h->rev_mapped = nullptr;
        h->rev_cap = 0;
        const size_t cap = 2 * nb + (1 << 16);
        M3S_CUDA(h, cudaHostAlloc((void **)&h->rev_mapped, cap, cudaHostAllocMapped));
        M3S_CUDA(h, cudaHostGetDevicePointer((void **)&h->rev_dev, h->rev_mapped, 0));
        h->rev_cap = cap;
    }
    const int64_t nw = (int64_t)(nb / 4);
    M3S_KBEGIN(h, M3S_K_SIDEINFO);
    k_words_out<<<(unsigned)((nw + 255) / 256), 256, 0, h->stream>>>((const uint32_t *)ss.tabids.p, (const uint32_t *)ss.reveal.p, nw,
                                                                       table_ids ? (uint32_t *)h->rev_dev : nullptr,
                                                                       reveal_bits ? (uint32_t *)(h->rev_dev + nb) : nullptr);
    M3S_LAUNCH_CHECK(h);
    M3S_CUDA(h, cudaStreamSynchronize(h->stream));
    if (table_ids) memcpy(table_ids, h->rev_mapped, nb);
    if (reveal_bits) memcpy(reveal_bits, h->rev_mapped + nb, nb);
    return M3S_OK;
}

extern "C" int m3s_decode_frame_pos(m3s_handle_t h, int64_t *frame_pos)
{
    if (!h) return M3S_ERR_ARG;
    if (!h->scanned) return m3s_fail(h, M3S_ERR_STATE, "decode_frame_pos: call m3s_decode_scan first");
    if (!frame_pos) return m3s_fail(h, M3S_ERR_ARG, "decode_frame_pos: null output");
    M3sScanSet &ss = *h->cur;
    if (ss.total_frames == 0) return M3S_OK;
    M3S_CUDA(h, cudaSetDevice(h->device));
    M3S_CUDA(h, cudaMemcpyAsync(frame_pos, ss.fr_pos.p, sizeof(int64_t) * (size_t)ss.total_frames, cudaMemcpyDeviceToHost, h->stream));
    M3S_CUDA(h, cudaStreamSynchronize(h->stream));
    for (int i = 0; i < ss.n_files; i++)   // wave positions -> file-relative
        for (int64_t g = ss.files_h[i].frame_base; g < ss.files_h[i].frame_base + ss.files_h[i].n_frames; g++) frame_pos[g] -= ss.files_h[i].begin;
    return M3S_OK;
}

// frames per CTA run of k_hybrid_fast.  Every run pays the CTA's table staging and one warm-up frame (together ~9 % of a 32-frame
// run), so large batches use long runs; small batches keep runs short enough to fill the SMs (3 CTAs per SM, >= 8 waves of them).
static int hybrid_run_length(int64_t total_frames, int sm_count)
{
    const int64_t want = total_frames / ((int64_t)sm_count * 3 * 8);
    return (int)std::max<int64_t>(16, std::min<int64_t>(128, want));
}

// Queue D1-D3 of a scanned wave on the handle's compute stream: main-data compaction (+ irregular reservoirs), Huffman decode,
// hybrid synthesis into d_pcm.  files_h[].pcm_base must hold each file's element offset inside d_pcm.
static int run_enqueue(m3s_ctx *h, M3sScanSet &ss, void *d_pcm, int16_t *d_spectra, uint32_t flags, int wb, int range_file = -1,
                       int64_t range_first = 0, int64_t range_count = 0)
{
    std::vector<M3sWork> &work = h->work_h[wb];
    const int64_t nf = ss.total_frames;
    if (nf == 0) return M3S_OK;
    // frames [g_lo, g_hi) go through Huffman decode + synthesis; [s_lo, g_hi) through the main-data compaction
    int64_t g_lo = 0, g_hi = nf, s_lo = 0;
    const bool fl = (flags & M3S_DEC_PCM_FLOAT) != 0;
    int rc;
    cudaStream_t s = h->stream;
    work.clear();
    if (range_file >= 0) {
        // one file's frames [first, first + count): the frame in front is the warm-up frame (its PCM is dropped; overlap-add tail and
        // the 15 V vectors of the synthesis fifo, Frame.py:81-92,150-153), and its main data may reach 511 bytes = at most 9 frames
        // back (Frame.py:306-309); a file whose granules inherit scalefactors from arbitrarily old frames needs its whole prefix in S
        const M3sFileRec &f = ss.files_h[range_file];
        const int run = hybrid_run_length(range_count, h->sm_count);
        g_lo = f.frame_base + std::max<int64_t>(range_first - 1, 0);
        g_hi = f.frame_base + range_first + range_count;
        s_lo = (f.flags & M3S_FILE_STATE_CARRY) ? f.frame_base : std::max<int64_t>(g_lo - 9, f.frame_base);
        for (int64_t k = range_first; k < range_first + range_count; k += run) {
            M3sWork w;
            w.g_first = f.frame_base + k;
            w.count = (int32_t)std::min<int64_t>(run, range_first + range_count - k);
            w.warm = k > 0 ? 1 : 0;
            w.pcm_elem = (k - range_first) * 1152 * f.channels;
            w.channels = f.channels;
            w.pad = 0;
            work.push_back(w);
        }
    } else {
        const int run = hybrid_run_length(nf, h->sm_count);
        for (int i = 0; i < ss.n_files; i++) {
            const M3sFileRec &f = ss.files_h[i];
            for (int64_t k = 0; k < f.n_frames; k += run) {
                M3sWork w;
                w.g_first = f.frame_base + k;
                w.count = (int32_t)std::min<int64_t>(run, f.n_frames - k);
                w.warm = k > 0 ? 1 : 0;
                w.pcm_elem = f.pcm_base + k * 1152 * f.channels;
                w.channels = f.channels;
                w.pad = 0;
                work.push_back(w);
            }
        }
    }
    if (work.empty()) return M3S_OK;
    const size_t n_stereo = (size_t)(std::stable_partition(work.begin(), work.end(), [](const M3sWork &w) { return w.channels == 2; }) - work.begin());
    const int64_t s_total = ss.s_bytes + ss.irregular * M3S_APX_SLOT_BYTES;
    if ((rc = reserve_quiet(h, h->b_S, (size_t)s_total))) return rc;
    if ((rc = reserve_quiet(h, h->b_spec, (size_t)nf * 288 * 4 * 4))) return rc;
    if ((rc = reserve_quiet(h, h->b_sf, (size_t)nf * 4 * M3S_SF_STRIDE))) return rc;
    if ((rc = reserve_quiet(h, h->b_work, sizeof(M3sWork) * work.size()))) return rc;
    if ((rc = pin_reserve(h, h->work_pin[wb], h->work_pin_cap[wb], sizeof(M3sWork) * work.size()))) return rc;
    memcpy(h->work_pin[wb], work.data(), sizeof(M3sWork) * work.size());
    M3S_CUDA(h, cudaMemcpyAsync(h->b_work.p, h->work_pin[wb], sizeof(M3sWork) * work.size(), cudaMemcpyHostToDevice, s));
    // (S needs no clearing: every reader is confined to [start, limit) of a frame's assembled main data -- regular frames start at or
    //  after their file's first payload byte by construction of resv_plan, irregular ones read a slot that k_reservoir_fix has written
    //  in full, and BitReader / BitWindow return zeros at or beyond the limit without touching memory)
    M3S_KBEGIN(h, M3S_K_STRIP);
    k_strip<<<(unsigned)(((g_hi - s_lo) * 32 + 255) / 256), 256, 0, s>>>(
        ss.d_bytes, ss.total_bytes, (const M3sFileRec *)ss.files.p, s_lo, g_hi, (const int64_t *)ss.fr_pos.p,
        (const uint32_t *)ss.fr_P.p, (const uint32_t *)ss.fr_meta.p, (const int32_t *)ss.fr_file.p, (uint8_t *)h->b_S.p);
    M3S_LAUNCH_CHECK(h);
    {   // irregular reservoirs: candidates are the first nine frames of every file + the listed frames (a no-op launch for clean input)
        const int64_t warps = (int64_t)ss.n_files * M3S_APX_SLOTS + ss.irregular;
        M3S_KBEGIN(h, M3S_K_STRIP);
        k_reservoir_fix<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, s>>>(
            ss.d_bytes, (const M3sFileRec *)ss.files.p, ss.n_files, (const int64_t *)ss.fr_pos.p, (const uint32_t *)ss.fr_meta.p,
            (const int32_t *)ss.fr_file.p, (const uint32_t *)ss.irr.p, ss.irregular, ss.s_bytes, (uint8_t *)h->b_S.p);
        M3S_LAUNCH_CHECK(h);
    }
    M3S_KBEGIN(h, M3S_K_HUFF);
    k_huff<<<(unsigned)((4 * (g_hi - g_lo) + HUFF_THREADS - 1) / HUFF_THREADS), HUFF_THREADS, 0, s>>>(
        (const uint8_t *)h->b_S.p, (const M3sUnitRec *)ss.units.p, 4 * g_lo, 4 * g_hi, h->d_tab, (uint32_t *)h->b_spec.p, (uint8_t *)h->b_sf.p);
    M3S_LAUNCH_CHECK(h);
    if (d_spectra) {
        M3S_KBEGIN(h, M3S_K_SPEC_EXPORT);
        k_spec_export<<<(unsigned)((nf * 288 * 4 + 255) / 256), 256, 0, s>>>((const uint32_t *)h->b_spec.p, nf, d_spectra);
        M3S_LAUNCH_CHECK(h);
    }
    const bool exact = (flags & M3S_DEC_EXACT) != 0;
#define M3S_LAUNCH_HYBRID_FAST1(OUT, FL, NCH, R, TAB, tabptr, first, count)                                                 \
    do {                                                                                                                      \
        const size_t smem = sizeof(HybFastSmem<OUT, R>);                                                                      \
        M3S_CUDA(h, cudaFuncSetAttribute(k_hybrid_fast<OUT, FL, NCH, R, TAB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        M3S_KBEGIN(h, M3S_K_HYBRID);                                                                                          \
        k_hybrid_fast<OUT, FL, NCH, R, TAB><<<(unsigned)(count), HF_THREADS, smem, s>>>(                                      \
            (const uint32_t *)h->b_spec.p, (const M3sUnitRec *)ss.units.p, (const uint8_t *)h->b_sf.p,                        \
            (const uint32_t *)ss.fr_meta.p, (const M3sWork *)h->b_work.p + (first), h->d_tab, (tabptr), d_pcm);               \
        M3S_LAUNCH_CHECK(h);                                                                                                  \
    } while (0)
    // the work list holds the stereo runs first, then the mono ones (see above): one launch per channel count that occurs
#define M3S_LAUNCH_HYBRID_FAST(OUT, FL, R, TAB, tabptr)                                                                       \
    do {                                                                                                                      \
        if (n_stereo > 0) M3S_LAUNCH_HYBRID_FAST1(OUT, FL, 2, R, TAB, tabptr, 0, n_stereo);                                   \
        if (work.size() > n_stereo) M3S_LAUNCH_HYBRID_FAST1(OUT, FL, 1, R, TAB, tabptr, n_stereo, work.size() - n_stereo);    \
    } while (0)
    if (exact) {
        if (fl) M3S_LAUNCH_HYBRID_FAST(float, true, double, M3sDevTablesD, h->d_tab_f64);
        else M3S_LAUNCH_HYBRID_FAST(int16_t, false, double, M3sDevTablesD, h->d_tab_f64);
    } else {
        if (fl) M3S_LAUNCH_HYBRID_FAST(float, true, float, M3sDevTables, h->d_tab);
        else M3S_LAUNCH_HYBRID_FAST(int16_t, false, float, M3sDevTables, h->d_tab);
    }
    return M3S_OK;
}

static inline int64_t file_pcm_elems(const M3sFileRec &f)
{
    const int64_t rows = 1152LL * (f.n_frames + ((f.flags & M3S_FILE_TRAILING_JUNK) && f.n_frames > 0 ? 1 : 0));
    return rows * std::max(f.channels, 1);
}

extern "C" int m3s_decode_run(m3s_handle_t h, void *pcm, int mem, const int64_t *pcm_off, int16_t *spectra, uint32_t flags)
{
    if (!h) return M3S_ERR_ARG;
    if (!h->scanned) return m3s_fail(h, M3S_ERR_STATE, "decode_run: call m3s_decode_scan first");
    if (!pcm) return m3s_fail(h, M3S_ERR_ARG, "decode_run: pcm is NULL");
    M3S_CUDA(h, cudaSetDevice(h->device));
    M3sScanSet &ss = *h->cur;
    const int64_t nf = ss.total_frames;
    if (nf == 0) return M3S_OK;
    double tr_t = g_trace ? now_ms() : 0.0;
    const bool fl = (flags & M3S_DEC_PCM_FLOAT) != 0;
    const size_t esz = fl ? 4 : 2;
    int rc;
    // ---- PCM layout: the caller's offsets, or back to back
    int64_t total_elems = 0;
    std::vector<int64_t> user_base(ss.n_files);
    for (int i = 0; i < ss.n_files; i++) {
        M3sFileRec &f = ss.files_h[i];
        const int64_t elems = file_pcm_elems(f);
        user_base[i] = pcm_off ? pcm_off[i] : total_elems;
        if (f.channels == 2 && !fl && (user_base[i] & 1)) return m3s_fail(h, M3S_ERR_ARG, "decode_run: stereo pcm_off must be even");
        // host buffers are staged back to back on the device and copied out file by file (gaps the caller left stay untouched)
        f.pcm_base = mem == M3S_MEM_HOST ? total_elems + (total_elems & 1) : user_base[i];
        if (mem == M3S_MEM_HOST) total_elems = f.pcm_base + elems;
        else total_elems = std::max(total_elems, f.pcm_base + elems);
    }
    void *d_pcm = pcm;
    if (mem == M3S_MEM_HOST) {
        if ((rc = m3s_buf_reserve(h, h->b_pcm_stage[0], (size_t)total_elems * esz + 16))) return rc;
        d_pcm = h->b_pcm_stage[0].p;
    }
    int16_t *d_sp = spectra;
    if (spectra && mem == M3S_MEM_HOST) {
        if ((rc = m3s_buf_reserve(h, h->b_spec_export, (size_t)nf * 4 * 576 * 2))) return rc;
        d_sp = (int16_t *)h->b_spec_export.p;
    }
    if ((rc = run_enqueue(h, ss, d_pcm, d_sp, flags, 0))) return rc;
    if (spectra && mem == M3S_MEM_HOST)
        M3S_CUDA(h, m3s_copy_bulk(spectra, d_sp, (size_t)nf * 4 * 576 * 2, cudaMemcpyDeviceToHost, h->stream));
    M3S_TRACE_MARK("run.launched");
    if (g_trace) { cudaStreamSynchronize(h->stream); M3S_TRACE_MARK("run.kernels_done"); }
    if (mem == M3S_MEM_HOST) {
        bool dense = true;   // one paced transfer when the caller's layout is the staging layout
        for (int i = 0; i < ss.n_files; i++) dense = dense && user_base[i] == ss.files_h[i].pcm_base;
        if (dense) {
            if ((rc = m3s_copy_paced(h, pcm, d_pcm, (size_t)total_elems * esz, cudaMemcpyDeviceToHost))) return rc;
        } else {
            std::vector<M3sRow> rows;
            for (int i = 0; i < ss.n_files; i++) {
                const M3sFileRec &f = ss.files_h[i];
                rows.push_back(M3sRow{(char *)pcm + user_base[i] * esz, (const char *)d_pcm + f.pcm_base * esz, (size_t)file_pcm_elems(f) * esz});
            }
            M3S_CUDA(h, m3s_copy_rows(rows, cudaMemcpyDeviceToHost, h->stream));
        }
    }
    M3S_CUDA(h, cudaStreamSynchronize(h->stream));
    M3S_TRACE_MARK("run.d2h_done");
    return M3S_OK;
}

// ================================================================================================
// m3s_decode: the whole of MP3Parser.parse_file + write_to_wav's conversion (MP3_Parser.py:57-91) for a batch, as ONE call that
// pipelines itself.  The files are cut into waves; four streams keep both PCIe directions and the SMs busy at once:
//
//      copy_in   MP3 bytes of wave k+1            (host buffers only)
//      aux       scan of wave k+1                 (walk, layout, per-file scans, side info + reveal: latency-bound, tiny)
//      stream    compaction, Huffman, hybrid of wave k
//      copy_out  PCM + table ids + reveal chars of wave k-1   (host buffers only)
//
// The host waits once per wave, for the scan of the NEXT wave, while the current wave's kernels are already queued; there is no
// other synchronisation until the end of the call.
// ================================================================================================
extern "C" int64_t m3s_decode_bound(const uint8_t *bytes_host, const int64_t *file_off, const int64_t *audio_start, int32_t n_files,
                                    int64_t *frames_bound)
{
    if (!bytes_host || !file_off || n_files <= 0) return -1;
    int64_t frames = 0;
    for (int i = 0; i < n_files; i++) {
        int64_t a = file_off[i] + (audio_start ? audio_start[i] : 0);
        if (a > file_off[i + 1]) a = file_off[i + 1];
        frames += frames_by_first_header(bytes_host + a, file_off[i + 1] - a);
    }
    if (frames_bound) *frames_bound = frames;
    return frames * 1152 * 2;
}

extern "C" int m3s_decode(m3s_handle_t h, const uint8_t *bytes, int mem, const int64_t *file_off, const int64_t *audio_start,
                          int32_t n_files, void *pcm, int64_t pcm_capacity, int64_t *pcm_off, uint8_t *table_ids, uint8_t *reveal_bits,
                          int64_t frames_capacity, int64_t *reveal_len, int64_t *n_frames, int32_t *sample_rate, int32_t *channels,
                          int32_t *bitrate_bps, int32_t *status, uint32_t flags)
{
    if (!h) return M3S_ERR_ARG;
    h->scanned = false;
    if (!bytes || !file_off || n_files <= 0 || !pcm) return m3s_fail(h, M3S_ERR_ARG, "decode: bytes/file_off/n_files/pcm");
    for (int i = 0; i < n_files; i++)
        if (file_off[i + 1] < file_off[i] || (audio_start && (audio_start[i] < 0)))
            return m3s_fail(h, M3S_ERR_ARG, "decode: file_off must be non-decreasing, audio_start >= 0");
    M3S_CUDA(h, cudaSetDevice(h->device));
    int rc;
    if ((rc = decode_events_init(h))) return rc;
    const bool host = mem == M3S_MEM_HOST;
    const bool fl = (flags & M3S_DEC_PCM_FLOAT) != 0;
    const size_t esz = fl ? 4 : 2;
    // ---- waves of whole files
    // host buffers: waves small enough that the pipeline fills / drains in a few percent of the call; device-resident input: waves
    // large enough that the tail of each wave's last CTAs (the kernels of consecutive waves do not overlap) stays small
    const int64_t wave_bytes = h->dec_wave_bytes > 0 ? h->dec_wave_bytes : (host ? ((int64_t)256 << 20) : ((int64_t)1 << 30));
    std::vector<int> wave_first;
    for (int i = 0; i < n_files;) {
        wave_first.push_back(i);
        int64_t acc = 0;
        do { acc += file_off[i + 1] - file_off[i]; i++; } while (i < n_files && acc + (file_off[i + 1] - file_off[i]) <= wave_bytes);
    }
    const int W = (int)wave_first.size();
    wave_first.push_back(n_files);
    int64_t frames_before = 0, elems_before = 0;
    // M3S_TRACE=1: a timeline of the call (timing events on every stream; printed at the end, relative to the first upload)
    struct WaveEv { cudaEvent_t h2d0, h2d1, scan1, comp0, comp1, out0, out1; double host_scan_wait_ms; };
    std::vector<WaveEv> tev;
    auto mark = [&](cudaEvent_t &e, cudaStream_t st) { if (g_trace) { cudaEventCreate(&e); cudaEventRecord(e, st); } };
    if (g_trace) { tev.assign(W, WaveEv()); }
    int err = M3S_OK;
    for (int k = 0; k <= W && err == M3S_OK; k++) {
        // ------------------------------------------------------------ A(k): bytes of wave k up, scan of wave k
        if (k < W) {
            const int b = k & 1, f0 = wave_first[k], nfl = wave_first[k + 1] - f0;
            M3sScanSet &ss = h->ss[b];
            const int64_t nbytes = file_off[f0 + nfl] - file_off[f0];
            const uint8_t *d_bytes = bytes + file_off[f0];
            if (host) {
                if ((err = reserve_quiet(h, h->b_stage_in[b], (size_t)nbytes + 16))) break;
                d_bytes = (const uint8_t *)h->b_stage_in[b].p;
            }
            if (k >= 2) {   // set b's previous wave (k - 2) must be through the kernels (they read its bytes and records) and copied out
                M3S_CUDA(h, cudaStreamWaitEvent(h->copy_in, h->ev_d_comp[b], 0));
                M3S_CUDA(h, cudaStreamWaitEvent(h->aux, h->ev_d_comp[b], 0));
                if (host) M3S_CUDA(h, cudaStreamWaitEvent(h->aux, h->ev_d_out[b], 0));
            }
            if (host) {
                if (g_trace) mark(tev[k].h2d0, h->copy_in);
                M3S_CUDA(h, cudaMemcpyAsync((void *)d_bytes, bytes + file_off[f0], (size_t)nbytes, cudaMemcpyHostToDevice, h->copy_in));
                if (g_trace) mark(tev[k].h2d1, h->copy_in);
                M3S_CUDA(h, cudaEventRecord(h->ev_d_h2d[b], h->copy_in));
                M3S_CUDA(h, cudaStreamWaitEvent(h->aux, h->ev_d_h2d[b], 0));
            }
            if ((err = scan_enqueue(h, ss, h->aux, d_bytes, host ? bytes + file_off[f0] : nullptr, file_off + f0,
                                    audio_start ? audio_start + f0 : nullptr, nfl)))
                break;
            if (g_trace) mark(tev[k].scan1, h->aux);
            M3S_CUDA(h, cudaEventRecord(h->ev_d_scan[b], h->aux));
        }
        // ------------------------------------------------------------ B(k - 1): kernels of wave k - 1, results home
        if (k >= 1) {
            const int j = k - 1, b = j & 1, f0 = wave_first[j];
            M3sScanSet &ss = h->ss[b];
            const double tw0 = g_trace ? now_ms() : 0.0;
            M3S_CUDA(h, cudaEventSynchronize(h->ev_d_scan[b]));
            if (g_trace) tev[j].host_scan_wait_ms = now_ms() - tw0;
            if ((err = scan_finish(h, ss, h->aux, file_off + f0, audio_start ? audio_start + f0 : nullptr))) break;
            int64_t wave_elems = 0;
            for (int i = 0; i < ss.n_files; i++) {
                M3sFileRec &f = ss.files_h[i];
                const M3sFileOut &o = ss.fouts_h[i];
                const int64_t elems = file_pcm_elems(f);
                f.pcm_base = (host ? 0 : elems_before) + wave_elems;
                if (pcm_off) pcm_off[f0 + i] = elems_before + wave_elems;
                wave_elems += elems;
                if (n_frames) n_frames[f0 + i] = o.n_frames;
                if (sample_rate) sample_rate[f0 + i] = o.sample_rate;
                if (channels) channels[f0 + i] = o.channels;
                if (bitrate_bps) bitrate_bps[f0 + i] = o.bitrate;
                if (status) status[f0 + i] = o.status;
                if (reveal_len) reveal_len[f0 + i] = o.reveal_len;
            }
            if (elems_before + wave_elems > pcm_capacity) {
                err = m3s_fail(h, M3S_ERR_CAPACITY, "decode: pcm holds %lld elements, files up to %d need %lld", (long long)pcm_capacity,
                               f0 + ss.n_files - 1, (long long)(elems_before + wave_elems));
                break;
            }
            if ((table_ids || reveal_bits) && frames_before + ss.total_frames > frames_capacity) {
                err = m3s_fail(h, M3S_ERR_CAPACITY, "decode: table_ids / reveal_bits hold %lld frames, files up to %d need %lld",
                               (long long)frames_capacity, f0 + ss.n_files - 1, (long long)(frames_before + ss.total_frames));
                break;
            }
            void *d_pcm = pcm;
            if (host) {
                if ((err = reserve_quiet(h, h->b_pcm_stage[b], (size_t)wave_elems * esz + 16))) break;
                d_pcm = h->b_pcm_stage[b].p;
                if (j >= 2) M3S_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_d_out[b], 0));   // the staging buffer's previous wave is home
            }
            M3S_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_d_scan[b], 0));
            if (g_trace) mark(tev[j].comp0, h->stream);
            if ((err = run_enqueue(h, ss, d_pcm, nullptr, flags, b))) break;
            if (g_trace) mark(tev[j].comp1, h->stream);
            const size_t nb = (size_t)12 * (size_t)ss.total_frames;
            if (!host && nb) {
                if (table_ids) M3S_CUDA(h, cudaMemcpyAsync(table_ids + 12 * frames_before, ss.tabids.p, nb, cudaMemcpyDeviceToDevice, h->stream));
                if (reveal_bits) M3S_CUDA(h, cudaMemcpyAsync(reveal_bits + 12 * frames_before, ss.reveal.p, nb, cudaMemcpyDeviceToDevice, h->stream));
            }
            M3S_CUDA(h, cudaEventRecord(h->ev_d_comp[b], h->stream));
            if (host) {
                // the reveal outputs only need the scan; they go first so that they never wait behind the PCM
                if (nb && table_ids) M3S_CUDA(h, cudaMemcpyAsync(table_ids + 12 * frames_before, ss.tabids.p, nb, cudaMemcpyDeviceToHost, h->copy_out));
                if (nb && reveal_bits) M3S_CUDA(h, cudaMemcpyAsync(reveal_bits + 12 * frames_before, ss.reveal.p, nb, cudaMemcpyDeviceToHost, h->copy_out));
                M3S_CUDA(h, cudaStreamWaitEvent(h->copy_out, h->ev_d_comp[b], 0));
                if (g_trace) mark(tev[j].out0, h->copy_out);
                if (wave_elems)
                    M3S_CUDA(h, cudaMemcpyAsync((char *)pcm + elems_before * esz, d_pcm, (size_t)wave_elems * esz, cudaMemcpyDeviceToHost, h->copy_out));
                if (g_trace) mark(tev[j].out1, h->copy_out);
                M3S_CUDA(h, cudaEventRecord(h->ev_d_out[b], h->copy_out));
            }
            frames_before += ss.total_frames;
            elems_before += wave_elems;
        }
    }
    if (err == M3S_OK && pcm_off) pcm_off[n_files] = elems_before;
    const std::string keep = h->err;
    const int rc2 = sync_all_streams(h);
    if (g_trace && err == M3S_OK && host && W > 0) {
        auto rel = [&](cudaEvent_t e) { float ms = 0.f; if (e) cudaEventElapsedTime(&ms, tev[0].h2d0, e); return ms; };
        fprintf(stderr, "[m3s_decode] %d waves; per wave (ms since the first upload): h2d [start end] scan_end comp [start end] d2h [start end] | host wait for the scan\n", W);
        for (int k = 0; k < W; k++)
            fprintf(stderr, "  wave %3d  h2d %7.2f %7.2f  scan %7.2f  comp %7.2f %7.2f  d2h %7.2f %7.2f | %.2f\n", k, rel(tev[k].h2d0), rel(tev[k].h2d1),
                    rel(tev[k].scan1), rel(tev[k].comp0), rel(tev[k].comp1), rel(tev[k].out0), rel(tev[k].out1), tev[k].host_scan_wait_ms);
        for (auto &w : tev)
            for (cudaEvent_t e : {w.h2d0, w.h2d1, w.scan1, w.comp0, w.comp1, w.out0, w.out1})
                if (e) cudaEventDestroy(e);
    }
    if (err != M3S_OK) { h->err = keep; return err; }
    return rc2;
}


// Frame-range decode of ONE file of the last scan (SURVEY.md 8e: a long file split across GPUs).  Every rank scans the whole file
// (the reference never resynchronises: frame positions, bit-reservoir cursors, reveal bits and the carried table ids come from there),
// then runs Huffman decode + synthesis only on frames [first, first + count) plus ONE warm-up frame in front, and compacts the main
// data of at most 9 more frames for that frame's bit reservoir -- all cut from the bytes already on the device.
extern "C" int m3s_decode_run_range(m3s_handle_t h, int32_t file_index, int64_t first_frame, int64_t frame_count, void *pcm, int mem,
                                    int64_t *rows_out, uint32_t flags)
{
    if (!h) return M3S_ERR_ARG;
    if (!h->scanned) return m3s_fail(h, M3S_ERR_STATE, "decode_run_range: call m3s_decode_scan first");
    M3sScanSet &ss = *h->cur;
    if (file_index < 0 || file_index >= ss.n_files) return m3s_fail(h, M3S_ERR_ARG, "decode_run_range: file_index");
    const M3sFileRec &f = ss.files_h[file_index];
    if (first_frame < 0 || frame_count < 0 || first_frame + frame_count > f.n_frames) return m3s_fail(h, M3S_ERR_ARG, "decode_run_range: frame range");
    if (!pcm && frame_count) return m3s_fail(h, M3S_ERR_ARG, "decode_run_range: pcm is NULL");
    M3S_CUDA(h, cudaSetDevice(h->device));
    const bool fl = (flags & M3S_DEC_PCM_FLOAT) != 0;
    const size_t esz = fl ? 4 : 2;
    const bool last = first_frame + frame_count == f.n_frames;
    const int64_t rows = 1152LL * (frame_count + (last && frame_count > 0 && (f.flags & M3S_FILE_TRAILING_JUNK) ? 1 : 0));
    if (rows_out) *rows_out = rows;
    if (frame_count == 0) return M3S_OK;
    const int64_t elems = rows * std::max(f.channels, 1);
    int rc;
    void *d_pcm = pcm;
    if (mem == M3S_MEM_HOST) {
        if ((rc = m3s_buf_reserve(h, h->b_pcm_stage[0], (size_t)elems * esz + 16))) return rc;
        d_pcm = h->b_pcm_stage[0].p;
    }
    if ((rc = run_enqueue(h, ss, d_pcm, nullptr, flags, 0, file_index, first_frame, frame_count))) return rc;
    if (mem == M3S_MEM_HOST)
        if ((rc = m3s_copy_paced(h, pcm, d_pcm, (size_t)elems * esz, cudaMemcpyDeviceToHost))) return rc;
    M3S_CUDA(h, cudaStreamSynchronize(h->stream));
    return M3S_OK;
}
