// Audio ingest in front of the log-mel: raw PCM -> fp32, channel mean, polyphase sinc resampling to 16 kHz, for many songs
// in one launch (reference etude/data/extractor.py:180-184: torchaudio.load -> torch.mean(wave, dim=0) ->
// torchaudio.transforms.Resample(sr, 16000) with torchaudio's defaults: sinc_interp_hann, lowpass_filter_width 6,
// rolloff 0.99; SURVEY.md section 8 row f-2).
//
//     y[i * new + p] = sum_k kern[p][k] * xm[i * orig + k - width],   xm = channel mean (zero outside the clip)
//
// orig / new are the rates divided by their gcd (441 / 160 for 44.1 kHz), K = 2 width + orig taps per phase (475).  Only a
// span of each row is non-zero (34 taps at 44.1 kHz): the sinc argument is clamped to +-6 where the Hann window is 0.
//
// Conversion to fp32 follows FFmpeg's sample-format rules (what torchaudio.load returns through TorchCodec): u8
// (x - 128) 2^-7, s16 x 2^-15, s24 x 2^-23, s32 (float)x 2^-31 (round to nearest), f32 as is, f64 rounded.  The mean is
// s = 0, s += x_c in channel order, s / C for C > 1, once per input frame.
//
// Bit-exactness with the full 475-tap chain: every output is one fmaf chain in ascending k from +0.  The accumulator
// never becomes -0, so a skipped tap of value +-0 on a finite sample changes nothing; zero samples outside the clip are
// identities as well.  A non-finite sample is spread over the full row (0 * inf = NaN, as torchaudio's conv does): a tile
// whose staged input holds one runs the full-row loop.
//
// Work layout (resampling, staged path).  Outputs are grouped into super-periods of P = lcm(new, 4) outputs (P / new
// input periods, sp_in input frames); a super-period is nb = P / 4 blocks of 4 consecutive outputs.  One thread computes
// one block: the union of its 4 trimmed windows (W taps) is one run of staged samples, and the block table holds the 4
// taps of every window position as a float4, so each sample loaded from shared memory feeds 4 FMAs.  The 32 lanes of a
// warp take the same block of 32 consecutive super-periods: the table load is a broadcast, the sample loads stride by
// sp_in (441 at 44.1 kHz: conflict-free).  A CTA stages S super-periods of converted, channel-averaged input and keeps
// the block tables of the current song in shared memory across the tiles it visits.
#pragma once
#include "common.cuh"

namespace etude {

enum PcmFormat { PCM_U8 = 1, PCM_S16 = 2, PCM_S24 = 3, PCM_S32 = 4, PCM_F32 = 5, PCM_F64 = 6 };

struct PcmSongDev {         // one song of an ingest launch (kernel parameter: no device buffer of the handle is used)
    const uint8_t* src;     // frame 0, channel 0
    float* out;             // n_out samples
    const float* kern;      // full table [nw][K]; nullptr: same rate (channel mean only)
    const float4* btab;     // block tables [nb][W]
    const int* bstart;      // [nb] first window position of every block, relative to the super-period's k = 0
    int64_t n_frames, n_out, frame_stride, chan_stride;   // strides in bytes
    int fmt, channels, orig, nw, width, K;
    int P, nb, W, sp_in;
    int S;                  // super-periods per tile (a multiple of 32); 0: unstaged (every output reads global memory)
    int tile0, n_tiles;     // this song's CTAs-tiles [tile0, tile0 + n_tiles) of the launch
};

constexpr int kIngestThreads = 256;
constexpr int kIngestMaxSongs = 24;          // descriptors per launch: below the 4 KB kernel-parameter limit
constexpr int kIngestFlatTile = 1024;        // outputs per tile of the same-rate and unstaged paths
constexpr int kIngestSmemBudget = 160 * 1024;

struct IngestLaunch {
    PcmSongDev song[kIngestMaxSongs];
    int n_songs;
};
static_assert(sizeof(IngestLaunch) <= 4096, "ingest descriptors exceed the kernel-parameter limit");

__device__ __forceinline__ float pcm_sample(const uint8_t* p, int fmt) {
    switch (fmt) {
        case PCM_U8: return (float)((int)*p - 128) * 0.0078125f;
        case PCM_S16: return (float)*(const int16_t*)p * (1.f / 32768.f);
        case PCM_S24: return (float)((int)((uint32_t)p[0] << 8 | (uint32_t)p[1] << 16 | (uint32_t)p[2] << 24) >> 8) * (1.f / 8388608.f);
        case PCM_S32: return __int2float_rn(*(const int32_t*)p) * (1.f / 2147483648.f);
        case PCM_F32: return *(const float*)p;
        default: return (float)*(const double*)p;   // PCM_F64, round to nearest
    }
}

// channel mean of input frame g (0 outside the clip)
__device__ __forceinline__ float pcm_frame(const PcmSongDev& s, int64_t g) {
    if (g < 0 || g >= s.n_frames) return 0.f;
    const uint8_t* f = s.src + g * s.frame_stride;
    float acc = 0.f;
    for (int c = 0; c < s.channels; ++c) acc += pcm_sample(f + c * s.chan_stride, s.fmt);
    return s.channels > 1 ? acc / (float)s.channels : acc;
}

// Converted, channel-averaged input frames [x_lo, x_lo + n) into xs.  Each thread converts 8 frames at a time with the
// loads of all 8 issued before any is used: one frame after another would leave the loop waiting on HBM latency.
template <int FMT>
__device__ __forceinline__ int stage_frames(const PcmSongDev& s, float* xs, int64_t x_lo, int n) {
    constexpr int B = 8;
    int bad = 0;
    for (int m0 = threadIdx.x; m0 < n; m0 += B * kIngestThreads) {
        float acc[B];
        const uint8_t* f[B];
        bool in[B];
#pragma unroll
        for (int u = 0; u < B; ++u) {
            const int64_t g = x_lo + m0 + u * kIngestThreads;
            in[u] = m0 + u * kIngestThreads < n && g >= 0 && g < s.n_frames;
            f[u] = s.src + (in[u] ? g : 0) * s.frame_stride;
            acc[u] = 0.f;
        }
        for (int c = 0; c < s.channels; ++c) {
#pragma unroll
            for (int u = 0; u < B; ++u)
                if (in[u]) acc[u] += pcm_sample(f[u] + c * s.chan_stride, FMT);
        }
#pragma unroll
        for (int u = 0; u < B; ++u) {
            const int m = m0 + u * kIngestThreads;
            if (m < n) {
                const float v = in[u] ? (s.channels > 1 ? acc[u] / (float)s.channels : acc[u]) : 0.f;
                xs[m] = v;
                bad |= !isfinite(v);
            }
        }
    }
    return bad;
}

// the whole row of phase j % nw from +0 in ascending k: the reference chain, for tiles with a non-finite sample and for
// rates whose tiles do not fit in shared memory.  x(k) is the channel mean at input frame (j / nw) * orig - width + k.
template <class X>
__device__ __forceinline__ float full_row(const PcmSongDev& s, int64_t j, X x) {
    const int64_t i = j / s.nw;
    const int ph = (int)(j - i * s.nw);
    const float* __restrict__ kr = s.kern + (size_t)ph * s.K;
    const int64_t base = i * s.orig - s.width;
    float acc = 0.f;
    for (int k = 0; k < s.K; ++k) acc = fmaf(__ldg(kr + k), x(base + k), acc);
    return acc;
}

__global__ void __launch_bounds__(kIngestThreads) ingest_pcm_kernel(const __grid_constant__ IngestLaunch L) {
    extern __shared__ __align__(16) uint8_t ingest_smem[];
    int cur = -1;   // song whose block tables are in shared memory
    for (int t = blockIdx.x;; t += gridDim.x) {
        int si = 0;
        while (si < L.n_songs && t >= L.song[si].tile0 + L.song[si].n_tiles) ++si;
        if (si >= L.n_songs) break;
        const PcmSongDev& s = L.song[si];
        const int64_t tile = t - s.tile0;

        if (s.kern == nullptr || s.S == 0) {   // same rate, or a rate whose tiles do not fit: one thread per output
            for (int r = threadIdx.x; r < kIngestFlatTile; r += kIngestThreads) {
                const int64_t j = tile * kIngestFlatTile + r;
                if (j >= s.n_out) break;
                s.out[j] = s.kern == nullptr ? pcm_frame(s, j) : full_row(s, j, [&](int64_t g) { return pcm_frame(s, g); });
            }
            continue;
        }

        float4* tb = reinterpret_cast<float4*>(ingest_smem);
        int* bs = reinterpret_cast<int*>(tb + (size_t)s.nb * s.W);
        float* xs = reinterpret_cast<float*>(bs + ((s.nb + 3) & ~3));
        __syncthreads();   // the previous tile is done with shared memory
        if (si != cur) {
            for (int e = threadIdx.x; e < s.nb * s.W; e += kIngestThreads) tb[e] = __ldg(s.btab + e);
            for (int e = threadIdx.x; e < s.nb; e += kIngestThreads) bs[e] = __ldg(s.bstart + e);
            cur = si;
        }
        const int64_t sp0 = tile * s.S;
        const int64_t x_lo = sp0 * s.sp_in - s.width;
        const int n_x = s.S * s.sp_in - s.orig + s.K;   // every input frame the full rows of the tile's outputs visit
        int bad;
        switch (s.fmt) {
            case PCM_U8: bad = stage_frames<PCM_U8>(s, xs, x_lo, n_x); break;
            case PCM_S16: bad = stage_frames<PCM_S16>(s, xs, x_lo, n_x); break;
            case PCM_S24: bad = stage_frames<PCM_S24>(s, xs, x_lo, n_x); break;
            case PCM_S32: bad = stage_frames<PCM_S32>(s, xs, x_lo, n_x); break;
            case PCM_F32: bad = stage_frames<PCM_F32>(s, xs, x_lo, n_x); break;
            default: bad = stage_frames<PCM_F64>(s, xs, x_lo, n_x); break;
        }
        for (int m = n_x + threadIdx.x; m < n_x + s.W; m += kIngestThreads) xs[m] = 0.f;   // read by zero taps of short blocks
        const int any_bad = __syncthreads_or(bad);
        const int64_t j_tile = sp0 * s.P;

        if (any_bad) {
            const int n = s.S * s.P;
            for (int r = threadIdx.x; r < n; r += kIngestThreads) {
                const int64_t j = j_tile + r;
                if (j >= s.n_out) break;
                s.out[j] = full_row(s, j, [&](int64_t g) { return xs[g - x_lo]; });
            }
            continue;
        }

        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        const int chunks = s.S >> 5;                   // 32-super-period chunks per tile
        for (int g = warp; g < chunks * s.nb; g += kIngestThreads / 32) {
            const int b = g / chunks;
            const int sp = (g - b * chunks) * 32 + lane;
            const int64_t j = j_tile + (int64_t)sp * s.P + 4 * b;
            if (j >= s.n_out) continue;
            const float* xw = xs + sp * s.sp_in + bs[b];
            const float4* tw = tb + (size_t)b * s.W;
            float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 4
            for (int u = 0; u < s.W; ++u) {
                const float x = xw[u];
                const float4 w = tw[u];
                a0 = fmaf(w.x, x, a0);
                a1 = fmaf(w.y, x, a1);
                a2 = fmaf(w.z, x, a2);
                a3 = fmaf(w.w, x, a3);
            }
            float* o = s.out + j;
            if (j + 4 <= s.n_out && ((uintptr_t)o & 15) == 0) {
                *reinterpret_cast<float4*>(o) = make_float4(a0, a1, a2, a3);
            } else {
                o[0] = a0;
                if (j + 1 < s.n_out) o[1] = a1;
                if (j + 2 < s.n_out) o[2] = a2;
                if (j + 3 < s.n_out) o[3] = a3;
            }
        }
    }
}

}  // namespace etude
