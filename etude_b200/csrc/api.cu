// libetude_b200.so: handle, weight packing, launch orchestration and the C ABI of include/etude_b200.h.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <map>
#include <vector>

#include "../../include/etude_b200.h"
#include "../../include/etude_b200_kernels.h"
#include "attention2.cuh"
#include "attention4.cuh"
#include "attn_qkv.cuh"
#include "attn_pair.cuh"
#include "chain3.cuh"
#include "embed2.cuh"
#include "gemm.cuh"
#include "logmel.cuh"
#include "logmel2.cuh"
#include "ingest.cuh"
#include "notes.cuh"
#include "pairmma.cuh"
#ifdef ETUDE_DEV_BUILD   // libetude_b200_dev.so (tests only): micro-benchmarks, kernel timelines, the generic GEMM epilogues
#include "mmabench.cuh"
#endif

using namespace etude;

// ------------------------------------------------------------------------------------------------ errors
static thread_local std::string g_err;
static int fail(const char* fmt, ...) {
    char buf[4096];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return -1;
}
#define CUDA_OK(expr)                                                                              \
    do {                                                                                           \
        cudaError_t e_ = (expr);                                                                   \
        if (e_ != cudaSuccess) return fail("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

extern "C" const char* etude_last_error(void) { return g_err.c_str(); }
extern "C" const char* etude_version(void) { return "etude_b200 0.1 (sm_100a, tcgen05/TMEM/TMA)"; }

// ------------------------------------------------------------------------------------------------ tensor maps
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// Row-major [rows, ld] matrix of bf16 (elem_bytes 2) or fp32 (4); box = box_cols x box_rows with the swizzle whose span
// equals the box's inner extent in bytes (128 B -> SWIZZLE_128B, 64 B -> SWIZZLE_64B).
static int make_tmap_ex(CUtensorMap* m, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows,
                        uint32_t box_cols, int elem_bytes) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return fail("cuTensorMapEncodeTiled entry point not available");
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {ld * (uint64_t)elem_bytes};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    const uint32_t inner = box_cols * elem_bytes;
    if (inner != 128 && inner != 64) return fail("make_tmap: unsupported box inner extent %u B", inner);
    CUresult r = fn(m, elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base),
                    dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    inner == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled failed (%d) rows=%llu cols=%llu ld=%llu box=%ux%u", (int)r,
                                       (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld, box_cols, box_rows);
    return 0;
}
// bf16 [d2][d1][256] tensor as a 3-D map (innermost = 256 channels): box = 64 channels (128 B, SW128) x b1 x b2.  Used for
// stores whose rows are strided (embed2: 128 frames of one bin) or must be clipped per sequence.
static int make_tmap_3d(CUtensorMap* m, const void* base, uint64_t d1, uint64_t d2, uint32_t b1, uint32_t b2) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return fail("cuTensorMapEncodeTiled entry point not available");
    cuuint64_t dims[3] = {256, d1, d2};
    cuuint64_t strides[2] = {256 * 2, d1 * 256 * 2};
    cuuint32_t box[3] = {64, b1, b2};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled (3-D) failed (%d) d1=%llu d2=%llu box=%ux%u", (int)r, (unsigned long long)d1,
                                       (unsigned long long)d2, b1, b2);
    return 0;
}
// bf16 operand map: box = 64 columns (128 B, one swizzle atom) x box_rows rows.
static int make_tmap(CUtensorMap* m, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows) {
    return make_tmap_ex(m, base, rows, cols, ld, box_rows, 64, 2);
}

// ------------------------------------------------------------------------------------------------ handle
struct Linear {  // bf16 weight [n, k] + fp32 bias [n] on the device
    __nv_bfloat16* w = nullptr;
    float* b = nullptr;
    int n = 0, k = 0;
};
struct LayerW {
    float *ln_g = nullptr, *ln_b = nullptr;
    Linear qkv;       // self-attention Q|K|V  [768,256]
    Linear qkv_hm;    // the same, head-major: row h * 192 + {0..63 Q_h, 64..127 K_h, 128..191 V_h} (attn_qkv.cuh)
    Linear o;         // self-attention fc_o
    Linear cq, co;    // cross-attention fc_q, fc_o
    Linear f1, f2;    // FFN
};

enum ProfClass { PC_LOGMEL = 0, PC_EMBED, PC_GEMM_BIAS, PC_GEMM_LN, PC_GEMM_HEADS, PC_ATTN, PC_NOTES, PC_TRANSPOSE, PC_CHAIN, PC_ATTN_FUSED, PC_INGEST, PC_COUNT };
static const char* kProfNames[PC_COUNT] = {"logmel", "embed", "gemm_bias", "gemm_ln", "gemm_heads", "attention", "notes", "transpose", "chain", "attention_fused",
                                           "ingest"};

// Launch accounting (always on) and optional CUDA-event timing of every launch, per kernel class.
struct Profile {
    bool timing = false;
    int64_t launches[PC_COUNT] = {0};
    double flops[PC_COUNT] = {0};   // algorithmic FLOPs of the launches (2MNK; 4*Lq*Lk*64 per head for attention)
    double bytes[PC_COUNT] = {0};   // algorithmic HBM bytes (front-end only)
    std::vector<cudaEvent_t> pool;  // event pairs, reused
    std::vector<int> pair_class;
    size_t used = 0;
    cudaEvent_t begin(int cls, cudaStream_t st, double fl, double by) {
        launches[cls]++; flops[cls] += fl; bytes[cls] += by;
        if (!timing) return nullptr;
        if (used + 2 > pool.size()) {
            cudaEvent_t a, b;
            cudaEventCreate(&a); cudaEventCreate(&b);
            pool.push_back(a); pool.push_back(b);
        }
        pair_class.push_back(cls);
        cudaEventRecord(pool[used], st);
        used += 2;
        return pool[used - 1];
    }
    void end(cudaEvent_t e, cudaStream_t st) { if (e) cudaEventRecord(e, st); }
};

struct etude_handle {
    Profile prof;
    int device = 0;
    int num_sms = 148;
    int64_t notes_last_total = 0;   // records of the last etude_notes_begin call (still in d_sorted)
    int frames = kFrames;  // frames per window: 512 (AMT-APC extractor) or 128 (HFT_Transformer), from the weight count
    std::vector<void*> allocs;
    // front-end tables
    struct ResampleTable {   // polyphase kernel + the block tables of ingest_pcm_kernel (ingest.cuh)
        float* d_kern; float4* d_btab; int* d_bstart;
        int orig, nw, width, K, P, nb, W, sp_in, S;
    };
    std::map<std::pair<int, int>, ResampleTable> resample_tabs;  // (sr_in, sr_out) -> polyphase kernel (etude_ingest)
    LogmelTables tab{};
    float2* tw32x32 = nullptr;  // [32 k1][32 n2] W_1024^(n2 k1) (logmel2.cuh)
    LogmelSong* d_songs = nullptr;
    int max_songs = 4096;
    // embedding
    float *w16 = nullptr, *posb = nullptr;
    __nv_bfloat16* w_embed_bf16 = nullptr;  // [256][64] taps 0..63 of W16 (embed2.cuh)
    float* w64 = nullptr;                   // [256] tap 64
    LayerW enc[3], dec0, dec[2], tim[3];
    Linear kv_all;  // the three cross-attention K|V projections [1536,256]
    __nv_bfloat16* q0 = nullptr;  // fc_q(pos_embedding_freq) of layer zero, [128,256] (rows >= 88 zero)
    float* pos_freq = nullptr;    // decoder.pos_embedding_freq [88,256] (+ wrap rows)
    __nv_bfloat16* pos_freq_bf16 = nullptr;  // the same table, bf16, three times over [264,256]: chain residual, row % 88
    float* pos_time = nullptr;    // decoder.pos_embedding_time [512,256]
    Linear heads_f, heads_t;      // [144,256]: onset, offset, mpe, velocity[128], zero padding
    int64_t* d_win_row = nullptr;  // [ETUDE_MAX_WINDOWS]
    int64_t* d_out_row = nullptr;
    // notes scratch (notes_reserve)
    NotesSong* d_nsongs = nullptr;
    int64_t* d_counts = nullptr;      // [max_songs * 88]
    float* notes_scratch = nullptr;   // pitch-major copies of the three fp32 rolls
    void* d_notes = nullptr;          // note slabs: one record slot per (frame, pitch)
    double* d_onsets = nullptr;       // their onset keys
    void* d_sorted = nullptr;         // sorted notes of the last etude_notes call
    int32_t* d_chunk_tab = nullptr;   // first_on | first_kept | first_off | chunk_count
    int64_t notes_rows_cap = 0, notes_chunks_cap = 0;
    int notes_songs_cap = 0;
    int64_t* d_song_base = nullptr;   // [max_songs] first sorted record of every song
    int64_t* d_song_total = nullptr;  // [max_songs + 1] notes per song, grand total
    int64_t* h_song_total = nullptr;  // pinned copy
    void* h_notes_pinned = nullptr;   // pinned D2H staging of the sorted notes = the library-owned result of etude_notes
    int64_t h_notes_cap = 0;
};

template <class T>
static int dev_upload(etude_handle* h, T** dst, const T* src, size_t n) {
    CUDA_OK(cudaMalloc((void**)dst, n * sizeof(T)));
    h->allocs.push_back(*dst);
    if (src) CUDA_OK(cudaMemcpy(*dst, src, n * sizeof(T), cudaMemcpyHostToDevice));
    return 0;
}

static int upload_linear(etude_handle* h, Linear* L, const std::vector<float>& w, const std::vector<float>& b, int n, int k) {
    std::vector<__nv_bfloat16> wb((size_t)n * k);
    for (size_t i = 0; i < wb.size(); ++i) wb[i] = __float2bfloat16(w[i]);
    L->n = n;
    L->k = k;
    if (dev_upload(h, &L->w, wb.data(), wb.size())) return -1;
    return dev_upload(h, &L->b, b.data(), b.size());
}

struct Blob {
    const float* base;
    size_t pos, total;
    const float* take(size_t n) {
        const float* p = base + pos;
        pos += n;
        return p;
    }
};
struct RawLinear {
    const float *w, *b;
};
struct RawMha {
    RawLinear q, k, v, o;
};
static RawLinear take_linear(Blob& bl, int n, int k) {
    RawLinear r;
    r.w = bl.take((size_t)n * k);
    r.b = bl.take(n);
    return r;
}
static RawMha take_mha(Blob& bl) {
    RawMha m;
    m.q = take_linear(bl, 256, 256);
    m.k = take_linear(bl, 256, 256);
    m.v = take_linear(bl, 256, 256);
    m.o = take_linear(bl, 256, 256);
    return m;
}
static void append(std::vector<float>& dst, const float* src, size_t n) { dst.insert(dst.end(), src, src + n); }

static int upload_raw(etude_handle* h, Linear* L, const RawLinear& r, int n, int k) {
    std::vector<float> w(r.w, r.w + (size_t)n * k), b(r.b, r.b + n);
    return upload_linear(h, L, w, b, n, k);
}
static int upload_qkv(etude_handle* h, Linear* L, const RawMha& m) {
    std::vector<float> w, b;
    append(w, m.q.w, 65536); append(w, m.k.w, 65536); append(w, m.v.w, 65536);
    append(b, m.q.b, 256); append(b, m.k.b, 256); append(b, m.v.b, 256);
    return upload_linear(h, L, w, b, 768, 256);
}
// Q|K|V weights regrouped by head for the fused projection + attention kernel: row h * 192 + {Q_h | K_h | V_h}
static int upload_qkv_head_major(etude_handle* h, Linear* L, const RawMha& m) {
    std::vector<float> w((size_t)768 * 256), b(768);
    const RawLinear* src[3] = {&m.q, &m.k, &m.v};
    for (int hd = 0; hd < 4; ++hd)
        for (int part = 0; part < 3; ++part) {
            memcpy(&w[((size_t)hd * 192 + part * 64) * 256], src[part]->w + (size_t)hd * 64 * 256, (size_t)64 * 256 * sizeof(float));
            memcpy(&b[hd * 192 + part * 64], src[part]->b + hd * 64, 64 * sizeof(float));
        }
    return upload_linear(h, L, w, b, 768, 256);
}
static int upload_heads(etude_handle* h, Linear* L, const RawLinear& on, const RawLinear& off, const RawLinear& mpe, const RawLinear& vel) {
    std::vector<float> w((size_t)144 * 256, 0.f), b(144, 0.f);
    memcpy(&w[0], on.w, 1024); memcpy(&w[256], off.w, 1024); memcpy(&w[512], mpe.w, 1024);
    memcpy(&w[768], vel.w, (size_t)128 * 1024);
    b[0] = on.b[0]; b[1] = off.b[0]; b[2] = mpe.b[0];
    memcpy(&b[3], vel.b, 512);
    return upload_linear(h, L, w, b, 144, 256);
}

// torchaudio.functional.melscale_fbanks(1025, 0, 8000, 256, 16000, norm="slaney", mel_scale="htk"), in double.
static void build_mel(std::vector<int>& start, std::vector<int>& count, std::vector<int>& offset, std::vector<float>& weight) {
    const int nf = kFreqs, nm = kBins;
    auto hz2mel = [](double f) { return 2595.0 * std::log10(1.0 + f / 700.0); };
    auto mel2hz = [](double m) { return 700.0 * (std::pow(10.0, m / 2595.0) - 1.0); };
    std::vector<double> fpts(nm + 2);
    const double m0 = hz2mel(0.0), m1 = hz2mel(8000.0);
    for (int i = 0; i < nm + 2; ++i) fpts[i] = mel2hz(m0 + (m1 - m0) * i / (nm + 1));
    start.assign(nm, 0); count.assign(nm, 0); offset.assign(nm, 0);
    weight.clear();
    for (int m = 0; m < nm; ++m) {
        const double enorm = 2.0 / (fpts[m + 2] - fpts[m]);
        int first = -1, last = -1;
        std::vector<float> wv(nf, 0.f);
        for (int k = 0; k < nf; ++k) {
            const double f = 8000.0 * k / (nf - 1);
            const double down = (f - fpts[m]) / (fpts[m + 1] - fpts[m]);
            const double up = (fpts[m + 2] - f) / (fpts[m + 2] - fpts[m + 1]);
            const double v = std::max(0.0, std::min(down, up)) * enorm;
            wv[k] = (float)v;
            if (wv[k] > 0.f) {
                if (first < 0) first = k;
                last = k;
            }
        }
        start[m] = first < 0 ? 0 : first;
        count[m] = first < 0 ? 0 : last - first + 1;
        offset[m] = (int)weight.size();
        for (int k = 0; k < count[m]; ++k) weight.push_back(wv[start[m] + k]);
    }
}

static int set_func_attrs_once();

extern "C" int etude_create(int device, const float* weights_host, size_t n_floats, etude_handle_t** out) {
    if (!out || !weights_host) return fail("etude_create: null argument");
    // the two architectures on the path differ only in decoder.pos_embedding_time [n_frame, 256]
    int frames = 0;
    if (n_floats == (size_t)ETUDE_N_WEIGHT_FLOATS) frames = 512;
    else if (n_floats == (size_t)ETUDE_N_WEIGHT_FLOATS_HFT) frames = 128;
    else return fail("etude_create: expected %d (ExtractorConfig, 512-frame windows) or %d (HFTConfig, 128-frame windows) weight floats, got %zu",
                     ETUDE_N_WEIGHT_FLOATS, ETUDE_N_WEIGHT_FLOATS_HFT, n_floats);
    int n_dev = 0;
    CUDA_OK(cudaGetDeviceCount(&n_dev));
    if (device < 0 || device >= n_dev) return fail("etude_create: device %d not present (%d devices)", device, n_dev);
    cudaDeviceProp prop;
    CUDA_OK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail("etude_create: device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
    CUDA_OK(cudaSetDevice(device));
    if (!get_encode_fn()) return fail("etude_create: driver lacks cuTensorMapEncodeTiled");

    etude_handle* h = new etude_handle();
    h->device = device;
    h->num_sms = prop.multiProcessorCount;
    h->frames = frames;
    int rc = 0;
    auto guard = [&](int r) { if (r) rc = -1; return r; };

    // ---- front-end tables
    {
        std::vector<float2> tw1(1024), tw2(1025);
        for (int i = 0; i < 1024; ++i) tw1[i] = make_float2((float)std::cos(-2.0 * M_PI * i / 1024.0), (float)std::sin(-2.0 * M_PI * i / 1024.0));
        for (int i = 0; i <= 1024; ++i) tw2[i] = make_float2((float)std::cos(-2.0 * M_PI * i / 2048.0), (float)std::sin(-2.0 * M_PI * i / 2048.0));
        std::vector<float> win(kNfft);
        for (int i = 0; i < kNfft; ++i) win[i] = (float)(0.5 - 0.5 * std::cos(2.0 * M_PI * i / kNfft));
        std::vector<int> ms, mc, mo;
        std::vector<float> mw;
        build_mel(ms, mc, mo, mw);
        float2 *d1, *d2; float *dw, *dmw; int *dms, *dmc, *dmo;
        if (guard(dev_upload(h, &d1, tw1.data(), tw1.size())) || guard(dev_upload(h, &d2, tw2.data(), tw2.size())) ||
            guard(dev_upload(h, &dw, win.data(), win.size())) || guard(dev_upload(h, &dms, ms.data(), ms.size())) ||
            guard(dev_upload(h, &dmc, mc.data(), mc.size())) || guard(dev_upload(h, &dmo, mo.data(), mo.size())) ||
            guard(dev_upload(h, &dmw, mw.data(), mw.size()))) { etude_destroy(h); return rc; }
        h->tab = LogmelTables{d1, d2, dw, dms, dmc, dmo, dmw};
        std::vector<float2> tw3(32 * 32);
        for (int k1 = 0; k1 < 32; ++k1)
            for (int n2 = 0; n2 < 32; ++n2)
                tw3[k1 * 32 + n2] = make_float2((float)std::cos(-2.0 * M_PI * (k1 * n2) / 1024.0), (float)std::sin(-2.0 * M_PI * (k1 * n2) / 1024.0));
        if (guard(dev_upload(h, &h->tw32x32, tw3.data(), tw3.size()))) { etude_destroy(h); return rc; }
        if (guard(dev_upload<LogmelSong>(h, &h->d_songs, nullptr, h->max_songs)) ||
            guard(dev_upload<NotesSong>(h, &h->d_nsongs, nullptr, h->max_songs)) ||
            guard(dev_upload<int64_t>(h, &h->d_counts, nullptr, (size_t)h->max_songs * kNotes)) ||
            guard(dev_upload<int64_t>(h, &h->d_song_base, nullptr, (size_t)h->max_songs)) ||
            guard(dev_upload<int64_t>(h, &h->d_song_total, nullptr, (size_t)h->max_songs + 1)) ||
            guard(dev_upload<int64_t>(h, &h->d_win_row, nullptr, 4 * ETUDE_MAX_WINDOWS)) ||
            guard(dev_upload<int64_t>(h, &h->d_out_row, nullptr, 4 * ETUDE_MAX_WINDOWS))) { etude_destroy(h); return rc; }
    }

    // ---- model weights (order: etude_b200/weights.py::STATE_DICT_LAYOUT)
    Blob bl{weights_host, 0, n_floats};
    const float* conv_w = bl.take(20);   // [4,1,1,5]
    const float* conv_b = bl.take(4);
    RawLinear tok = take_linear(bl, 256, 244);
    const float* pos_enc = bl.take(65536);
    {
        // fold conv(1x5, 4 ch) into the 244 -> 256 linear: one 65-tap filter per hidden channel (SURVEY.md A4)
        std::vector<float> w16((size_t)256 * kProc, 0.f), posb((size_t)256 * 256);
        for (int hh = 0; hh < 256; ++hh) {
            double beff = tok.b[hh];
            for (int c = 0; c < 4; ++c)
                for (int pp = 0; pp < 61; ++pp) {
                    const double wt = tok.w[(size_t)hh * 244 + c * 61 + pp];
                    beff += wt * conv_b[c];
                    for (int k = 0; k < 5; ++k) w16[(size_t)hh * kProc + pp + k] += (float)(16.0 * wt * conv_w[c * 5 + k]);
                }
            for (int b = 0; b < 256; ++b) posb[(size_t)b * 256 + hh] = (float)(16.0 * beff + pos_enc[(size_t)b * 256 + hh]);
        }
        if (guard(dev_upload(h, &h->w16, w16.data(), w16.size())) || guard(dev_upload(h, &h->posb, posb.data(), posb.size()))) { etude_destroy(h); return rc; }
        // tensor-core embedding (embed2.cuh): taps 0..63 as a bf16 [256][64] MMA operand, tap 64 stays fp32
        std::vector<__nv_bfloat16> wb((size_t)256 * 64);
        std::vector<float> w64(256);
        for (int hh = 0; hh < 256; ++hh) {
            for (int t = 0; t < 64; ++t) wb[(size_t)hh * 64 + t] = __float2bfloat16(w16[(size_t)hh * kProc + t]);
            w64[hh] = w16[(size_t)hh * kProc + 64];
        }
        if (guard(dev_upload(h, &h->w_embed_bf16, wb.data(), wb.size())) || guard(dev_upload(h, &h->w64, w64.data(), w64.size()))) { etude_destroy(h); return rc; }
    }
    auto take_ln = [&](LayerW& L) -> int {
        const float* g = bl.take(256);
        const float* b = bl.take(256);
        return dev_upload(h, &L.ln_g, g, 256) || dev_upload(h, &L.ln_b, b, 256);
    };
    auto take_ffn = [&](LayerW& L) -> int {
        RawLinear f1 = take_linear(bl, 512, 256);
        RawLinear f2 = take_linear(bl, 256, 512);
        return upload_raw(h, &L.f1, f1, 512, 256) || upload_raw(h, &L.f2, f2, 256, 512);
    };
    std::vector<float> kvw, kvb;  // cross-attention K|V of the three decoder layers
    auto take_cross = [&](LayerW& L, RawMha* keep) -> int {
        RawMha m = take_mha(bl);
        append(kvw, m.k.w, 65536); append(kvw, m.v.w, 65536);
        append(kvb, m.k.b, 256); append(kvb, m.v.b, 256);
        if (keep) *keep = m;
        return upload_raw(h, &L.cq, m.q, 256, 256) || upload_raw(h, &L.co, m.o, 256, 256);
    };
    for (int i = 0; i < 3 && !rc; ++i) {
        if (guard(take_ln(h->enc[i]))) break;
        RawMha m = take_mha(bl);
        if (guard(upload_qkv(h, &h->enc[i].qkv, m)) || guard(upload_qkv_head_major(h, &h->enc[i].qkv_hm, m)) ||
            guard(upload_raw(h, &h->enc[i].o, m.o, 256, 256)) || guard(take_ffn(h->enc[i]))) break;
    }
    const float* pos_dec = bl.take((size_t)kNotes * 256);
    RawMha zero_cross{};
    if (!rc) guard(take_ln(h->dec0) || take_cross(h->dec0, &zero_cross) || take_ffn(h->dec0));
    for (int i = 0; i < 2 && !rc; ++i) {
        if (guard(take_ln(h->dec[i]))) break;
        RawMha m = take_mha(bl);
        if (guard(upload_qkv(h, &h->dec[i].qkv, m)) || guard(upload_raw(h, &h->dec[i].o, m.o, 256, 256)) ||
            guard(take_cross(h->dec[i], nullptr)) || guard(take_ffn(h->dec[i]))) break;
    }
    RawLinear on_f = take_linear(bl, 1, 256), off_f = take_linear(bl, 1, 256), mpe_f = take_linear(bl, 1, 256), vel_f = take_linear(bl, 128, 256);
    const float* pos_time = bl.take((size_t)frames * 256);
    for (int i = 0; i < 3 && !rc; ++i) {
        if (guard(take_ln(h->tim[i]))) break;
        RawMha m = take_mha(bl);
        if (guard(upload_qkv(h, &h->tim[i].qkv, m)) || guard(upload_raw(h, &h->tim[i].o, m.o, 256, 256)) || guard(take_ffn(h->tim[i]))) break;
    }
    RawLinear on_t = take_linear(bl, 1, 256), off_t = take_linear(bl, 1, 256), mpe_t = take_linear(bl, 1, 256), vel_t = take_linear(bl, 128, 256);
    if (!rc && bl.pos != n_floats) rc = fail("etude_create: weight layout consumed %zu of %zu floats", bl.pos, n_floats);
    if (!rc) guard(upload_linear(h, &h->kv_all, kvw, kvb, 1536, 256));
    if (!rc) guard(upload_heads(h, &h->heads_f, on_f, off_f, mpe_f, vel_f) || upload_heads(h, &h->heads_t, on_t, off_t, mpe_t, vel_t));
    if (!rc) {
        // decoder.pos_embedding_freq followed by a copy of its first 32 rows: the LN epilogue's 32-row residual boxes start
        // at row % 88 and must not run off the table
        std::vector<float> wrapped((size_t)(kNotes + 32) * 256);
        memcpy(wrapped.data(), pos_dec, (size_t)kNotes * 1024);
        memcpy(wrapped.data() + (size_t)kNotes * 256, pos_dec, (size_t)32 * 1024);
        guard(dev_upload(h, &h->pos_freq, wrapped.data(), wrapped.size()) || dev_upload(h, &h->pos_time, pos_time, (size_t)frames * 256));
        std::vector<__nv_bfloat16> wb((size_t)3 * kNotes * 256);
        for (int r = 0; r < 3 * kNotes; ++r)
            for (int c = 0; c < 256; ++c) wb[(size_t)r * 256 + c] = __float2bfloat16(pos_dec[(size_t)(r % kNotes) * 256 + c]);
        if (!rc) guard(dev_upload(h, &h->pos_freq_bf16, wb.data(), wb.size()));
    }
    if (!rc) {
        // layer-zero queries are input independent: Q0 = fc_q(pos_embedding_freq)  (amt_apc.py:168-175, 342)
        std::vector<__nv_bfloat16> q0((size_t)128 * 256, __float2bfloat16(0.f));
        for (int n = 0; n < kNotes; ++n)
            for (int o = 0; o < 256; ++o) {
                double acc = zero_cross.q.b[o];
                for (int k = 0; k < 256; ++k) acc += (double)pos_dec[(size_t)n * 256 + k] * zero_cross.q.w[(size_t)o * 256 + k];
                q0[(size_t)n * 256 + o] = __float2bfloat16((float)acc);
            }
        guard(dev_upload(h, &h->q0, q0.data(), q0.size()));
    }
    if (!rc && set_func_attrs_once()) rc = -1;
    if (rc) { etude_destroy(h); return rc; }
    if (cudaHostAlloc((void**)&h->h_song_total, sizeof(int64_t) * (h->max_songs + 1), cudaHostAllocDefault) != cudaSuccess) {
        etude_destroy(h);
        return fail("etude_create: pinned host allocation failed");
    }
    *out = h;
    return 0;
}

extern "C" void etude_destroy(etude_handle_t* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    for (cudaEvent_t e : h->prof.pool) cudaEventDestroy(e);
    for (void* p : h->allocs) cudaFree(p);
    for (void* p : {(void*)h->notes_scratch, h->d_notes, (void*)h->d_onsets, h->d_sorted, (void*)h->d_chunk_tab})
        if (p) cudaFree(p);
    if (h->h_notes_pinned) cudaFreeHost(h->h_notes_pinned);
    if (h->h_song_total) cudaFreeHost(h->h_song_total);
    delete h;
}

// ------------------------------------------------------------------------------------------------ launchers
// ETUDE_SYNC_DEBUG=1: synchronise after every launch and name the kernel that failed (debugging aid; off by default)
static int debug_sync(const char* what, cudaStream_t st) {
    static const bool on = getenv("ETUDE_SYNC_DEBUG") != nullptr;
    if (!on) return 0;
    static unsigned long long* host_report = nullptr;
    if (!host_report) {  // host-mapped words the bounded waits fill in before they trap
        if (cudaHostAlloc((void**)&host_report, 256, cudaHostAllocMapped) == cudaSuccess) {
            memset(host_report, 0, 256);
            unsigned long long* dptr = nullptr;
            cudaHostGetDevicePointer((void**)&dptr, host_report, 0);
            cudaMemcpyToSymbol(g_hang_report, &dptr, sizeof dptr);
        }
    }
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) {
        if (host_report && host_report[0]) {
            std::string msg;
            for (unsigned long long i = 0; i < std::min<unsigned long long>(host_report[0], 24); ++i) {
                const unsigned long long v = host_report[1 + i];
                char b[96];
                snprintf(b, sizeof b, " [tag %llu blk %llu warp %llu info %llu par %llu]", v >> 56, (v >> 40) & 0xFFFF, (v >> 32) & 0xFF,
                         (v >> 1) & 0x7FFFFFFF, v & 1);
                msg += b;
            }
            return fail("%s: %s; bounded waits that gave up:%s", what, cudaGetErrorString(e), msg.c_str());
        }
        return fail("%s: %s", what, cudaGetErrorString(e));
    }
    return 0;
}
static int set_func_attrs_once() {
    static bool done_dev[64] = {false};
    static int status_dev[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    dev &= 63;
    bool& done = done_dev[dev];
    int& status = status_dev[dev];
    if (done) return status;
    done = true;
    cudaError_t e = cudaSuccess;
    auto set_smem = [&](const void* fn, size_t bytes) { if (e == cudaSuccess) e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes); };
#ifdef ETUDE_DEV_BUILD
    set_smem((const void*)gemm_tcgen05_kernel<256, EPI_BIAS>, gemm_smem_bytes<256, EPI_BIAS>());
    set_smem((const void*)gemm_tcgen05_kernel<256, EPI_BIAS_RELU>, gemm_smem_bytes<256, EPI_BIAS_RELU>());
    set_smem((const void*)gemm_tcgen05_kernel<256, EPI_RESID_LN>, gemm_smem_bytes<256, EPI_RESID_LN>());
#endif
    set_smem((const void*)gemm_tcgen05_kernel<144, EPI_HEADS>, gemm_smem_bytes<144, EPI_HEADS>());
    set_smem((const void*)gemm_bstat_kernel, kGemmBsSmemBytes);
    set_smem((const void*)attention2_kernel<256>, kAttn2SmemBytes);
    set_smem((const void*)attention2_kernel<96>, kAttn2SmemBytes);
    set_smem((const void*)attention4_kernel<128>, kAttn4SmemBytes);
    set_smem((const void*)attention4_kernel<96>, kAttn4SmemBytes);
#ifdef ETUDE_HAVE_ATTN_QKV_CTA1
    set_smem((const void*)attn_qkv_kernel, kAttnQkvSmemBytes);
#endif
    set_smem((const void*)attn_pair_kernel, kAttnPairSmemBytes);
    set_smem((const void*)chain3_kernel<true>, kChain3SmemBytes);
    set_smem((const void*)chain3_kernel<false>, kChain3SmemBytes);
    set_smem((const void*)embed2_kernel, kEmbed2SmemBytes);
    set_smem((const void*)ingest_pcm_kernel, kIngestSmemBudget);
    // The note-decoding kernels (and the ingest of extract_files) run on other streams beside the model kernels.  An SM has ONE L1 / shared
    // memory split at a time: with the default (L1-heavy) carve-out a resident notes block keeps every model CTA (which
    // needs the 227 KB split) off its SM until it finishes, and the statically partitioned model kernel waits for it.
    auto max_smem_carveout = [&](const void* fn) {
        if (e == cudaSuccess) e = cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
    };
    for (const void* fn : {(const void*)ingest_pcm_kernel, (const void*)notes_transpose_kernel, (const void*)notes_scan_kernel, (const void*)notes_walk_kernel,
                           (const void*)notes_compact_kernel, (const void*)notes_bases_kernel, (const void*)notes_rank_kernel})
        max_smem_carveout(fn);
    set_smem((const void*)logmel2_kernel, kLogmel2SmemBytes);
    if (e != cudaSuccess) status = fail("cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
    return status;
}

static int num_sms_cached() {
    static int n = 0;
    if (!n) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

struct GemmIO {  // global buffers the epilogue touches through TMA
    __nv_bfloat16* out_bf16 = nullptr;
    int ld_out = 0;            // row stride of out_bf16 (elements)
    float* out_f32 = nullptr;  // LN only, [M,256]
    const float* resid = nullptr;  // LN only, fp32 [resid_rows,256]
    int64_t resid_rows = 0;
};

template <int BLOCK_N, int EPI>
static int launch_gemm(const void* a, const void* w, GemmParams p, const GemmIO& io, cudaStream_t st, Profile* prof = nullptr) {
    if (p.K % kBlockK) return fail("gemm: K=%d not a multiple of %d", p.K, kBlockK);
    if (p.N % BLOCK_N) return fail("gemm: N=%d not a multiple of the tile width %d", p.N, BLOCK_N);
    CUtensorMap ta, tb, tob, tof, tr;
    if (make_tmap(&ta, a, (uint64_t)p.M, (uint64_t)p.K, (uint64_t)p.K, kBlockM)) return -1;
    if (make_tmap(&tb, w, (uint64_t)p.N, (uint64_t)p.K, (uint64_t)p.K, BLOCK_N)) return -1;
    tob = ta; tof = ta; tr = ta;  // unused maps must still be valid descriptors
    if (EPI == EPI_BIAS || EPI == EPI_BIAS_RELU) {
        if (!io.out_bf16) return fail("gemm: missing bf16 output");
        if (make_tmap_ex(&tob, io.out_bf16, (uint64_t)p.M, (uint64_t)p.N, (uint64_t)io.ld_out, 32, 64, 2)) return -1;
    } else if (EPI == EPI_RESID_LN) {
        if (!io.out_bf16 || !io.out_f32 || !io.resid) return fail("gemm: LayerNorm epilogue needs out_bf16, out_f32 and resid");
        if (make_tmap_ex(&tob, io.out_bf16, (uint64_t)p.M, 256, 256, 32, 32, 2)) return -1;
        if (make_tmap_ex(&tof, io.out_f32, (uint64_t)p.M, 256, 256, 32, 32, 4)) return -1;
        if (make_tmap_ex(&tr, io.resid, (uint64_t)io.resid_rows, 256, 256, 32, 32, 4)) return -1;
    }
    p.num_m_tiles = (p.M + kBlockM - 1) / kBlockM;
    p.num_n_tiles = p.N / BLOCK_N;
    const int tiles = p.num_m_tiles * p.num_n_tiles;
    const int grid = std::min(tiles, num_sms_cached());
    const int cls = EPI == EPI_RESID_LN ? PC_GEMM_LN : (EPI == EPI_HEADS ? PC_GEMM_HEADS : PC_GEMM_BIAS);
    const int n_alg = EPI == EPI_HEADS ? 3 + kVel : p.N;
    cudaEvent_t ev = prof ? prof->begin(cls, st, 2.0 * p.M * (double)n_alg * p.K, 0.0) : nullptr;
    gemm_tcgen05_kernel<BLOCK_N, EPI><<<grid, kGemmThreads, gemm_smem_bytes<BLOCK_N, EPI>(), st>>>(ta, tb, tob, tof, tr, p);
    if (prof) prof->end(ev, st);
    CUDA_OK(cudaGetLastError());
    {
        char what[96];
        snprintf(what, sizeof what, "gemm epi=%d M=%d N=%d K=%d", EPI, p.M, p.N, p.K);
        if (debug_sync(what, st)) return -1;
    }
    return 0;
}

// K = 256 projection with the W slice resident in smem (gemm_bstat_kernel)
static int launch_gemm_bstat(const void* a, const void* w, const float* bias, int M, int N, __nv_bfloat16* out, cudaStream_t st, Profile* prof) {
    if (N % 256) return fail("gemm_bstat: N=%d not a multiple of 256", N);
    CUtensorMap ta, tb, to;
    if (make_tmap(&ta, a, (uint64_t)M, 256, 256, kBlockM)) return -1;
    if (make_tmap(&tb, w, (uint64_t)N, 256, 256, 256)) return -1;
    if (make_tmap_ex(&to, out, (uint64_t)M, (uint64_t)N, (uint64_t)N, 32, 64, 2)) return -1;
    GemmParams p{};
    p.M = M; p.N = N; p.K = 256; p.bias = bias;
    p.num_m_tiles = (M + kBlockM - 1) / kBlockM;
    p.num_n_tiles = N / 256;
    const int grid = std::max(1, num_sms_cached() / p.num_n_tiles) * p.num_n_tiles;
    cudaEvent_t ev = prof ? prof->begin(PC_GEMM_BIAS, st, 2.0 * M * (double)N * 256.0, 0.0) : nullptr;
    gemm_bstat_kernel<<<grid, kBsThreads, kGemmBsSmemBytes, st>>>(ta, tb, to, p);
    if (prof) prof->end(ev, st);
    CUDA_OK(cudaGetLastError());
    {
        char what[96];
        snprintf(what, sizeof what, "gemm_bstat M=%d N=%d", M, N);
        if (debug_sync(what, st)) return -1;
    }
    return 0;
}

// Every bias-only projection of the model is K = 256, N a multiple of 256: the B-stationary kernel.
static int gemm_bias(const void* a, const Linear& L, int M, __nv_bfloat16* out, cudaStream_t st, Profile* prof) {
    if (L.k != 256 || L.n % 256 != 0) return fail("gemm_bias: unsupported projection shape N=%d K=%d", L.n, L.k);
    return launch_gemm_bstat(a, L.w, L.b, M, L.n, out, st, prof);
}

// Debug timeline of the chain / attention kernels (dev build only: tests/gpu_diag.py chain_trace, attn_trace): device
// buffer of 3 roles x kChTraceSlots (id, clock) pairs (= 6 roles x 256 tiles for attention4).  Always null in the product.
static long long* g_chain_trace = nullptr;

// Persistent pipelined attention: attention4.cuh (128-key blocks, four TMEM buffers); the probabilities output of the
// 9-tuple API runs on attention2.cuh (one 256-key block per row, P also written to HBM).
static int launch_attention(const void* q, int64_t q_rows, int q_ld, int q_col0, int q_seq_stride, const void* kv, int kv_ld,
                            int k_col0, int v_col0, int n_seq, int Lq, int Lk, __nv_bfloat16* out, float* probs, cudaStream_t st,
                            Profile* prof = nullptr) {
    const int gen = probs != nullptr ? 2 : 4;
    Attn2Params p{};
    int kb;
    if (Lk == 88) kb = 96;
    else if (Lk == 128) kb = 128;
    else if (Lk == 256 || Lk == 512) kb = gen == 4 ? 128 : 256;
    else return fail("attention: unsupported key length %d", Lk);
    if (Lq > 512 || Lq < 1) return fail("attention: unsupported query length %d", Lq);
    p.Lq = Lq; p.Lk = Lk; p.n_items = n_seq * kHeads; p.q_seq_stride = q_seq_stride;
    p.QT = (Lq + 127) / 128;
    p.NKV = (Lk + kb - 1) / kb;
    if (probs && (p.NKV != 1 || kb == 128)) return fail("attention: the probabilities output is built for one block of 88 or 256 keys");
    if (gen == 4 ? (2 * p.NKV > kA4KvSlots) : (2 * p.NKV + 1 > kA2KvSlots || p.NKV > 2))
        return fail("attention: %d KV blocks exceed the smem ring", p.NKV);
    p.q_col0 = q_col0; p.k_col0 = k_col0; p.v_col0 = v_col0;
    p.out = out; p.probs = probs;
    p.trace = g_chain_trace;  // debug timeline buffer (etude_debug_chain_trace), normally null
    p.scale_log2e = 1.4426950408889634f / 8.0f;
    CUtensorMap tq, tkv;
    if (make_tmap(&tq, q, (uint64_t)q_rows, (uint64_t)q_ld, (uint64_t)q_ld, 128)) return -1;
    if (make_tmap(&tkv, kv, (uint64_t)n_seq * Lk, (uint64_t)kv_ld, (uint64_t)kv_ld, kb)) return -1;
    const int grid = std::min(p.n_items, num_sms_cached());
    cudaEvent_t ev = prof ? prof->begin(PC_ATTN, st, 4.0 * n_seq * kHeads * (double)Lq * Lk * kHeadDim, 0.0) : nullptr;
    if (gen == 2) {
        if (kb == 256) attention2_kernel<256><<<grid, kAttn2Threads, kAttn2SmemBytes, st>>>(tq, tkv, p);
        else attention2_kernel<96><<<grid, kAttn2Threads, kAttn2SmemBytes, st>>>(tq, tkv, p);
    } else {
        if (kb == 128) attention4_kernel<128><<<grid, kAttn4Threads, kAttn4SmemBytes, st>>>(tq, tkv, p);
        else attention4_kernel<96><<<grid, kAttn4Threads, kAttn4SmemBytes, st>>>(tq, tkv, p);
    }
    if (prof) prof->end(ev, st);
    CUDA_OK(cudaGetLastError());
    {
        char what[96];
        snprintf(what, sizeof what, "attention gen%d n_seq=%d Lq=%d Lk=%d", gen, n_seq, Lq, Lk);
        if (debug_sync(what, st)) return -1;
    }
    return 0;
}

#ifdef ETUDE_DEV_BUILD
extern "C" int etude_debug_mma_bench(int mode, int n, int iters, int n_bufs, int grid, int64_t* host_out) {
    long long* d = nullptr;
    CUDA_OK(cudaMalloc((void**)&d, 16));
    CUDA_OK(cudaFuncSetAttribute((const void*)mma_bench_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 210 * 1024));
    mma_bench_kernel<<<grid, 128, 210 * 1024>>>(mode, n, iters, n_bufs, d);
    CUDA_OK(cudaDeviceSynchronize());
    CUDA_OK(cudaMemcpy(host_out, d, 16, cudaMemcpyDeviceToHost));
    cudaFree(d);
    return 0;
}

extern "C" int etude_debug_mma_mix(int ts, int iters, int n_ld, int st_too, int grid, int64_t* host_out) {
    long long* d = nullptr;
    CUDA_OK(cudaMalloc((void**)&d, 32));
    CUDA_OK(cudaMemset(d, 0, 32));
    CUDA_OK(cudaFuncSetAttribute((const void*)mma_mix_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 140 * 1024));
    mma_mix_kernel<<<grid, 768, 140 * 1024>>>(ts, iters, n_ld, st_too, d);
    CUDA_OK(cudaDeviceSynchronize());
    CUDA_OK(cudaMemcpy(host_out, d, 16, cudaMemcpyDeviceToHost));
    cudaFree(d);
    return 0;
}

extern "C" int etude_debug_tmem_bench(int mode, int n_warps, int iters, int grid, int64_t* host_out) {
    long long* d = nullptr;
    CUDA_OK(cudaMalloc((void**)&d, 32));
    CUDA_OK(cudaMemset(d, 0, 32));
    tmem_bench_kernel<<<grid, 32 * n_warps>>>(mode, iters, d, reinterpret_cast<float*>(d + 2));
    CUDA_OK(cudaDeviceSynchronize());
    CUDA_OK(cudaMemcpy(host_out, d, 8, cudaMemcpyDeviceToHost));
    cudaFree(d);
    return 0;
}

// Debug timeline control: enable allocates + zeroes the buffer, a later call with host_out reads it back.
extern "C" int etude_debug_chain_trace(int enable, int64_t* host_out, int n_values) {
    const size_t bytes = (size_t)64 * 1024;   // 3 roles x 512 (id, clock) pairs (chain) / 8 x 192 x 2 (attention4) / 8 x 64 x 8 (attn_qkv)
    if (host_out && g_chain_trace) {
        CUDA_OK(cudaDeviceSynchronize());
        CUDA_OK(cudaMemcpy(host_out, g_chain_trace, std::min(bytes, (size_t)n_values * sizeof(int64_t)), cudaMemcpyDeviceToHost));
    }
    if (enable && !g_chain_trace) {
        CUDA_OK(cudaMalloc((void**)&g_chain_trace, bytes));
    } else if (!enable && g_chain_trace) {
        cudaFree(g_chain_trace);
        g_chain_trace = nullptr;
    }
    if (g_chain_trace) CUDA_OK(cudaMemset(g_chain_trace, 0, bytes));
    return 0;
}
// cta_group::2 self-test (pairmma.cuh): A bf16 [256, 64], B bf16 [128, 64], VT bf16 [64, 128] -> D fp32 [256, 128] = A B^T,
// O fp32 [256, 64] = bf16(D) VT^T.  One cluster of two CTAs.
extern "C" int etude_debug_pairmma(const void* a, const void* b, const void* vt, float* d, float* o) {
    const size_t smem = 16384 + 8192 + 8192 + 64;
    CUDA_OK(cudaFuncSetAttribute((const void*)pairmma_test_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    pairmma_test_kernel<<<2, 128, smem>>>((const __nv_bfloat16*)a, (const __nv_bfloat16*)b, (const __nv_bfloat16*)vt, d, o);
    CUDA_OK(cudaGetLastError());
    CUDA_OK(cudaDeviceSynchronize());
    return 0;
}
// cta_group::2 MMA rate (pairmma.cuh): host_out[0] = issue clocks, [1] = clocks until completion, of `iters` M256 x n x K16 MMAs
extern "C" int etude_debug_pairmma_bench(int ts, int n, int iters, int alt, int grid, int64_t* host_out) {
    long long* d = nullptr;
    CUDA_OK(cudaMalloc((void**)&d, 16));
    const size_t smem = 192 * 1024;
    CUDA_OK(cudaFuncSetAttribute((const void*)pairmma_bench_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    pairmma_bench_kernel<<<grid, 128, smem>>>(ts, n, iters, alt, d);
    CUDA_OK(cudaGetLastError());
    CUDA_OK(cudaDeviceSynchronize());
    CUDA_OK(cudaMemcpy(host_out, d, 16, cudaMemcpyDeviceToHost));
    cudaFree(d);
    return 0;
}
#endif  // ETUDE_DEV_BUILD

// Self-attention with the Q|K|V projection fused in (attn_qkv.cuh): x bf16 [n_seq * 256, 256] -> context bf16 [n_seq * 256, 256].
// w_hm / bias_hm are head-major (upload_qkv_head_major).  One cluster of two CTAs per sequence of 256 tokens.
// pair = true: attn_pair.cuh (CTA-pair MMAs: the product); false: attn_qkv.cuh (cta_group::1; test-only library and
// -DETUDE_ATTN_PAIR=0 A/B builds)
static int launch_attn_qkv(const void* x, const __nv_bfloat16* w_hm, const float* bias_hm, int n_seq, __nv_bfloat16* out, cudaStream_t st,
                           Profile* prof, bool pair = ETUDE_ATTN_PAIR != 0) {
    if (n_seq < 1) return fail("attn_qkv: n_seq=%d", n_seq);
    CUtensorMap tx, tw;
    if (make_tmap(&tx, x, (uint64_t)n_seq * 256, 256, 256, 128)) return -1;
    if (make_tmap(&tw, w_hm, 768, 256, 256, 96)) return -1;
    AttnQkvParams p{};
    p.n_seq = n_seq; p.bias = bias_hm; p.out = out;
    p.scale_log2e = 1.4426950408889634f / 8.0f;
    p.trace = g_chain_trace;
    const int clusters = std::min(n_seq, num_sms_cached() / 2);
    const double fl = 2.0 * n_seq * 256.0 * 768.0 * 256.0 + 4.0 * n_seq * kHeads * 256.0 * 256.0 * kHeadDim;
    cudaEvent_t ev = prof ? prof->begin(PC_ATTN_FUSED, st, fl, 0.0) : nullptr;
    if (pair) {
        attn_pair_kernel<<<2 * clusters, kAqThreads, kAttnPairSmemBytes, st>>>(tx, tw, p);
    } else {
#ifdef ETUDE_HAVE_ATTN_QKV_CTA1
        attn_qkv_kernel<<<2 * clusters, kAqThreads, kAttnQkvSmemBytes, st>>>(tx, tw, p);
#else
        return fail("attn_qkv: the cta_group::1 kernel is not in this build");
#endif
    }
    if (prof) prof->end(ev, st);
    CUDA_OK(cudaGetLastError());
    {
        char what[64];
        snprintf(what, sizeof what, "attn_qkv n_seq=%d", n_seq);
        if (debug_sync(what, st)) return -1;
    }
    return 0;
}

// Fused fc_o + residual + LN (+ FFN + residual + LN) over 128-token tiles (chain3.cuh).  `resid` is bf16 [M,256], or with
// resid_mod > 0 a bf16 table of at least resid_mod + 127 rows whose row r holds entry r % resid_mod.  out may alias resid.
static int launch_chain(const void* ctx, const Linear& o, const Linear* f1, const Linear* f2, const float* gamma, const float* beta,
                        const void* resid, int resid_mod, int64_t resid_rows, __nv_bfloat16* out, int M, cudaStream_t st, Profile* prof) {
    const bool ffn = f1 != nullptr;
    if (o.n != 256 || o.k != 256 || (ffn && (f1->n != 512 || f1->k != 256 || !f2 || f2->n != 256 || f2->k != 512)))
        return fail("chain: unexpected layer shapes");
    // clusters of two sharing the weight stream (chain3.cuh)
    CUtensorMap tc, two, tw1, tw2, tr, tout;
    if (make_tmap(&tc, ctx, (uint64_t)M, 256, 256, 128)) return -1;
    if (make_tmap(&tout, out, (uint64_t)M, 256, 256, 128)) return -1;
    if (make_tmap(&two, o.w, 256, 256, 256, kC3PartRows)) return -1;
    tw1 = two; tw2 = two;
    if (ffn) {
        if (make_tmap(&tw1, f1->w, 512, 256, 256, kC3PartRows)) return -1;
        if (make_tmap(&tw2, f2->w, 256, 512, 512, kC3PartRows)) return -1;
    }
    if (make_tmap(&tr, resid, (uint64_t)resid_rows, 256, 256, 128)) return -1;
    ChainParams p{};
    p.M = M; p.num_tiles = (M + 127) / 128; p.resid_mod = resid_mod;
    p.bo = o.b; p.b1 = ffn ? f1->b : o.b; p.b2 = ffn ? f2->b : o.b; p.gamma = gamma; p.beta = beta;
    p.trace = g_chain_trace;
    const int n_pairs = (p.num_tiles + kC3Cluster - 1) / kC3Cluster;
    const int grid = std::min(n_pairs, num_sms_cached() / kC3Cluster) * kC3Cluster;
    cudaEvent_t ev = prof ? prof->begin(PC_CHAIN, st, 2.0 * M * 256.0 * 256.0 + (ffn ? 4.0 * M * 512.0 * 256.0 : 0.0), 0.0) : nullptr;
    if (ffn) chain3_kernel<true><<<grid, kC3Threads, kChain3SmemBytes, st>>>(tc, two, tw1, tw2, tr, tout, p);
    else chain3_kernel<false><<<grid, kC3Threads, kChain3SmemBytes, st>>>(tc, two, tw1, tw2, tr, tout, p);
    if (prof) prof->end(ev, st);
    CUDA_OK(cudaGetLastError());
    {
        char what[96];
        snprintf(what, sizeof what, "chain3 ffn=%d M=%d resid_mod=%d", (int)ffn, M, resid_mod);
        if (debug_sync(what, st)) return -1;
    }
    return 0;
}

// ------------------------------------------------------------------------------------------------ kernel-level ABI
extern "C" int etude_k_gemm(const void* a, const void* w, const float* bias, int M, int N, int K, int epilogue, void* out_bf16,
                            const float* resid, int resid_mod, const float* gamma, const float* beta, float* out_f32, void* stream) {
    if (set_func_attrs_once()) return -1;
    cudaStream_t st = (cudaStream_t)stream;
    if (epilogue == EPI_BIAS && K == 256 && N % 256 == 0) return launch_gemm_bstat(a, w, bias, M, N, (__nv_bfloat16*)out_bf16, st, nullptr);
#ifdef ETUDE_DEV_BUILD   // the generic tile GEMM with its other epilogues is not on the product path (tests keep exercising it)
    GemmParams p{};
    p.M = M; p.N = N; p.K = K; p.bias = bias;
    p.resid_mod = resid_mod; p.ln_gamma = gamma; p.ln_beta = beta;
    GemmIO io;
    io.out_bf16 = (__nv_bfloat16*)out_bf16; io.ld_out = N; io.out_f32 = out_f32; io.resid = resid;
    io.resid_rows = resid_mod ? resid_mod + 32 : M;
    switch (epilogue) {
        case EPI_BIAS: return launch_gemm<256, EPI_BIAS>(a, w, p, io, st);
        case EPI_BIAS_RELU: return launch_gemm<256, EPI_BIAS_RELU>(a, w, p, io, st);
        case EPI_RESID_LN:
            if (N != 256) return fail("gemm: LayerNorm epilogue needs N == 256");
            return launch_gemm<256, EPI_RESID_LN>(a, w, p, io, st);
        default: return fail("gemm: unknown epilogue %d", epilogue);
    }
#else
    (void)resid; (void)resid_mod; (void)gamma; (void)beta; (void)out_f32;
    return fail("etude_k_gemm: only the bias epilogue with K == 256 and N %% 256 == 0 is built into the product library "
                "(epilogue %d, N=%d, K=%d needs libetude_b200_dev.so)", epilogue, N, K);
#endif
}

extern "C" int etude_k_attention(const void* q, int64_t q_rows, int q_ld, int q_col0, int q_seq_stride, const void* kv, int kv_ld,
                                 int k_col0, int v_col0, int n_seq, int Lq, int Lk, void* out, float* probs, void* stream) {
    if (set_func_attrs_once()) return -1;
    return launch_attention(q, q_rows, q_ld, q_col0, q_seq_stride, kv, kv_ld, k_col0, v_col0, n_seq, Lq, Lk, (__nv_bfloat16*)out,
                            probs, (cudaStream_t)stream);
}

extern "C" int etude_k_attn_qkv(const void* x, const void* w_hm, const float* bias_hm, int n_seq, void* out, void* stream) {
    if (!x || !w_hm || !bias_hm || !out) return fail("etude_k_attn_qkv: null argument");
    if (set_func_attrs_once()) return -1;
    return launch_attn_qkv(x, (const __nv_bfloat16*)w_hm, bias_hm, n_seq, (__nv_bfloat16*)out, (cudaStream_t)stream, nullptr);
}

#ifdef ETUDE_DEV_BUILD
// the cta_group::1 implementation of the same operator (attn_qkv.cuh): the cross-check partner of the product kernel
extern "C" int etude_debug_attn_qkv_cta1(const void* x, const void* w_hm, const float* bias_hm, int n_seq, void* out, void* stream) {
    if (!x || !w_hm || !bias_hm || !out) return fail("etude_debug_attn_qkv_cta1: null argument");
    if (set_func_attrs_once()) return -1;
    return launch_attn_qkv(x, (const __nv_bfloat16*)w_hm, bias_hm, n_seq, (__nv_bfloat16*)out, (cudaStream_t)stream, nullptr, false);
}
#endif

extern "C" int etude_k_chain(const void* ctx, const void* wo, const float* bo, const void* w1, const float* b1, const void* w2,
                             const float* b2, const float* gamma, const float* beta, const void* resid, int resid_mod,
                             int64_t resid_rows, void* out, int M, void* stream) {
    if (set_func_attrs_once()) return -1;
    Linear o, f1, f2;
    o.w = (__nv_bfloat16*)wo; o.b = (float*)bo; o.n = 256; o.k = 256;
    f1.w = (__nv_bfloat16*)w1; f1.b = (float*)b1; f1.n = 512; f1.k = 256;
    f2.w = (__nv_bfloat16*)w2; f2.b = (float*)b2; f2.n = 256; f2.k = 512;
    return launch_chain(ctx, o, w1 ? &f1 : nullptr, w1 ? &f2 : nullptr, gamma, beta, resid, resid_mod, resid_rows, (__nv_bfloat16*)out, M,
                        (cudaStream_t)stream, nullptr);
}

// ------------------------------------------------------------------------------------------------ front-end
static int64_t igcd(int64_t a, int64_t b) { while (b) { const int64_t t = a % b; a = b; b = t; } return a; }

extern "C" int64_t etude_resampled_length(int64_t n_in, int sr_in, int sr_out) {
    if (n_in < 0 || sr_in <= 0 || sr_out <= 0) return -1;
    if (sr_in == sr_out) return n_in;
    const int64_t g = igcd(sr_in, sr_out), orig = sr_in / g, nw = sr_out / g;
    return (int64_t)std::ceil((double)(nw * n_in) / (double)orig);   // torchaudio: ceil(new_freq * length / orig_freq)
}

// torchaudio.functional._get_sinc_resample_kernel (sinc_interp_hann, lowpass_filter_width 6, rolloff 0.99): indices in
// float64, the phase term -p / new rounded to float32 first (an int64 tensor divided by an int is float32 in torch).
// Besides the full [new][K] table: each phase's non-zero span and the 4-output block tables of ingest_pcm_kernel.
static int build_resample_table(etude_handle* h, int sr_in, int sr_out, etude_handle::ResampleTable* out) {
    auto it = h->resample_tabs.find({sr_in, sr_out});
    if (it != h->resample_tabs.end()) { *out = it->second; return 0; }
    const int g = (int)igcd(sr_in, sr_out), orig = sr_in / g, nw = sr_out / g;
    const double base_freq = std::min(orig, nw) * 0.99;
    const int width = (int)std::ceil(6.0 * orig / base_freq), K = 2 * width + orig;
    if ((int64_t)nw * K > (int64_t)64 << 20) return fail("etude_ingest: %d -> %d Hz needs a %d x %d tap table", sr_in, sr_out, nw, K);
    std::vector<float> kern((size_t)nw * K);
    const double scale = base_freq / orig;
    for (int p = 0; p < nw; ++p) {
        const double phase = (double)((float)(-p) / (float)nw);
        for (int k = 0; k < K; ++k) {
            double t = (phase + (double)(k - width) / orig) * base_freq;
            t = std::max(-6.0, std::min(6.0, t));
            const double c = std::cos(t * M_PI / 6.0 / 2.0), window = c * c;
            t *= M_PI;
            const double v = (t == 0.0) ? 1.0 : std::sin(t) / t;
            kern[(size_t)p * K + k] = (float)(v * window * scale);
        }
    }
    etude_handle::ResampleTable tab{};
    tab.orig = orig; tab.nw = nw; tab.width = width; tab.K = K;
    std::vector<int> lo(nw, 0), hi(nw, 0);   // non-zero span [lo, hi) of every phase
    for (int p = 0; p < nw; ++p) {
        const float* r = &kern[(size_t)p * K];
        int a = 0, b = K;
        while (a < K && r[a] == 0.f) ++a;
        while (b > a && r[b - 1] == 0.f) --b;
        lo[p] = a < b ? a : 0;
        hi[p] = a < b ? b : 0;
    }
    // blocks of 4 consecutive outputs over a super-period of P = lcm(nw, 4) outputs: window = union of the 4 spans
    tab.P = (int)((int64_t)nw * 4 / igcd(nw, 4));
    tab.nb = tab.P / 4;
    tab.sp_in = tab.P / nw * orig;
    std::vector<int> bstart(tab.nb), bend(tab.nb);
    for (int b = 0; b < tab.nb; ++b) {
        int st = INT32_MAX, en = 0;
        for (int r = 0; r < 4; ++r) {
            const int j = 4 * b + r, p = j % nw, rel = j / nw * orig;
            st = std::min(st, rel + lo[p]);
            en = std::max(en, rel + hi[p]);
        }
        bstart[b] = st;
        bend[b] = std::max(en, st);
        tab.W = std::max(tab.W, bend[b] - st);
    }
    const int64_t tab_bytes = (int64_t)tab.nb * tab.W * 16 + (int64_t)((tab.nb + 3) & ~3) * 4;
    auto smem = [&](int64_t S) { return tab_bytes + 4 * (S * tab.sp_in - orig + K + tab.W); };
    tab.S = smem(32) <= kIngestSmemBudget ? 32 : 0;     // unstaged when 32 super-periods do not fit
    while (tab.S && (int64_t)tab.S * tab.nb < 1024 && smem(2 * tab.S) <= 80 * 1024) tab.S *= 2;   // >= 4 blocks per thread
    if (tab.S) {
        std::vector<float4> bt((size_t)tab.nb * tab.W, make_float4(0.f, 0.f, 0.f, 0.f));
        for (int b = 0; b < tab.nb; ++b)
            for (int r = 0; r < 4; ++r) {
                const int j = 4 * b + r, p = j % nw, rel = j / nw * orig;
                for (int k = lo[p]; k < hi[p]; ++k) (&bt[(size_t)b * tab.W + rel + k - bstart[b]].x)[r] = kern[(size_t)p * K + k];
            }
        if (dev_upload(h, &tab.d_btab, bt.data(), bt.size()) || dev_upload(h, &tab.d_bstart, bstart.data(), bstart.size())) return -1;
    }
    if (dev_upload(h, &tab.d_kern, kern.data(), kern.size())) return -1;
    h->resample_tabs[{sr_in, sr_out}] = tab;
    *out = tab;
    return 0;
}

extern "C" int etude_ingest_reserve(etude_handle_t* h, const int* sample_rates, int n, int sr_out) {
    if (!h || (n > 0 && !sample_rates) || n < 0 || sr_out <= 0) return fail("etude_ingest_reserve: bad argument");
    CUDA_OK(cudaSetDevice(h->device));
    for (int i = 0; i < n; ++i) {
        if (sample_rates[i] <= 0) return fail("etude_ingest_reserve: sample rate %d", sample_rates[i]);
        etude_handle::ResampleTable tab;
        if (sample_rates[i] != sr_out && build_resample_table(h, sample_rates[i], sr_out, &tab)) return -1;
    }
    return 0;
}

static int pcm_container_bytes(int fmt) {
    switch (fmt) {
        case ETUDE_PCM_U8: return 1;
        case ETUDE_PCM_S16: return 2;
        case ETUDE_PCM_S24: return 3;
        case ETUDE_PCM_S32: case ETUDE_PCM_F32: return 4;
        case ETUDE_PCM_F64: return 8;
        default: return 0;
    }
}

extern "C" int etude_ingest_pcm(etude_handle_t* h, const void* pcm_dev, const etude_pcm_song_t* songs, int n_songs, int sr_out,
                                float* wave_out_dev, void* stream) {
    if (!h || !pcm_dev || !songs || !wave_out_dev) return fail("etude_ingest_pcm: null argument");
    if (n_songs < 1 || sr_out <= 0) return fail("etude_ingest_pcm: n_songs=%d, sr_out=%d", n_songs, sr_out);
    static_assert(ETUDE_PCM_U8 == PCM_U8 && ETUDE_PCM_S16 == PCM_S16 && ETUDE_PCM_S24 == PCM_S24 && ETUDE_PCM_S32 == PCM_S32 &&
                  ETUDE_PCM_F32 == PCM_F32 && ETUDE_PCM_F64 == PCM_F64, "format codes");
    CUDA_OK(cudaSetDevice(h->device));
    std::vector<PcmSongDev> dev(n_songs);
    std::vector<double> flops(n_songs), bytes(n_songs);
    for (int i = 0; i < n_songs; ++i) {   // everything is checked before the first launch
        const etude_pcm_song_t& s = songs[i];
        const int cb = pcm_container_bytes(s.format);
        if (!cb) return fail("etude_ingest_pcm: song %d: unknown format %d", i, s.format);
        if (s.channels < 1 || s.channels > 64) return fail("etude_ingest_pcm: song %d: %d channels (1..64)", i, s.channels);
        if (s.n_frames < 1 || s.sample_rate <= 0) return fail("etude_ingest_pcm: song %d: %lld frames at %d Hz", i, (long long)s.n_frames, s.sample_rate);
        if (s.byte_offset < 0 || s.dst_offset < 0 || s.frame_stride < cb || (s.channels > 1 && s.channel_stride < cb))
            return fail("etude_ingest_pcm: song %d: bad offsets or strides (offset %lld, frame stride %lld, channel stride %lld, dst %lld)", i,
                        (long long)s.byte_offset, (long long)s.frame_stride, (long long)s.channel_stride, (long long)s.dst_offset);
        const int al = cb == 3 ? 1 : cb;
        if (((uintptr_t)pcm_dev + s.byte_offset) % al || s.frame_stride % al || s.channel_stride % al)
            return fail("etude_ingest_pcm: song %d: offset / strides not aligned to its %d-byte samples", i, cb);
        PcmSongDev& d = dev[i];
        d = PcmSongDev{};
        d.src = (const uint8_t*)pcm_dev + s.byte_offset;
        d.out = wave_out_dev + s.dst_offset;
        d.n_frames = s.n_frames;
        d.n_out = etude_resampled_length(s.n_frames, s.sample_rate, sr_out);
        d.frame_stride = s.frame_stride;
        d.chan_stride = s.channels > 1 ? s.channel_stride : 0;
        d.fmt = s.format;
        d.channels = s.channels;
        if (d.n_out < 1) return fail("etude_ingest_pcm: song %d: empty output", i);
        int64_t taps = 0;
        if (s.sample_rate != sr_out) {
            etude_handle::ResampleTable tab;
            if (build_resample_table(h, s.sample_rate, sr_out, &tab)) return -1;
            d.kern = tab.d_kern; d.btab = tab.d_btab; d.bstart = tab.d_bstart;
            d.orig = tab.orig; d.nw = tab.nw; d.width = tab.width; d.K = tab.K;
            d.P = tab.P; d.nb = tab.nb; d.W = tab.W; d.sp_in = tab.sp_in; d.S = tab.S;
            taps = tab.S ? (int64_t)tab.W : (int64_t)tab.K;   // per output, as visited
        }
        if (d.kern && d.S) {
            const int64_t n_sp = (d.n_out + d.P - 1) / d.P;
            d.n_tiles = (int)((n_sp + d.S - 1) / d.S);
        } else {
            d.n_tiles = (int)((d.n_out + kIngestFlatTile - 1) / kIngestFlatTile);
        }
        flops[i] = 2.0 * (double)taps * (double)d.n_out;
        bytes[i] = (double)s.n_frames * s.channels * cb + 4.0 * (double)d.n_out;
    }
    if (set_func_attrs_once()) return -1;
    cudaStream_t st = (cudaStream_t)stream;
    int per_sm = 0;
    for (int a = 0; a < n_songs; a += kIngestMaxSongs) {
        IngestLaunch L{};
        L.n_songs = std::min(kIngestMaxSongs, n_songs - a);
        int tiles = 0;
        size_t smem = 0;
        double fl = 0, by = 0;
        for (int i = 0; i < L.n_songs; ++i) {
            PcmSongDev& d = dev[a + i];
            d.tile0 = tiles;
            tiles += d.n_tiles;
            if (d.kern && d.S)
                smem = std::max(smem, (size_t)d.nb * d.W * 16 + (size_t)((d.nb + 3) & ~3) * 4 + 4 * (size_t)(d.S * d.sp_in - d.orig + d.K + d.W));
            fl += flops[a + i];
            by += bytes[a + i];
            L.song[i] = d;
        }
        CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ingest_pcm_kernel, kIngestThreads, smem));
        const int grid = std::max(1, std::min(tiles, h->num_sms * std::max(per_sm, 1)));
        cudaEvent_t ev = h->prof.begin(PC_INGEST, st, fl, by);
        ingest_pcm_kernel<<<grid, kIngestThreads, smem, st>>>(L);
        h->prof.end(ev, st);
        CUDA_OK(cudaGetLastError());
    }
    return 0;
}

// One planar fp32 song through ingest_pcm_kernel.
extern "C" int etude_ingest(etude_handle_t* h, const float* pcm, int channels, int64_t n_in, int sr_in, int sr_out, float* wave_out,
                            void* stream) {
    if (!h || !pcm || !wave_out) return fail("etude_ingest: null argument");
    if (channels < 1 || channels > 64 || n_in < 1 || sr_in <= 0 || sr_out <= 0) return fail("etude_ingest: bad shape (channels=%d, n=%lld, %d -> %d Hz)", channels, (long long)n_in, sr_in, sr_out);
    etude_pcm_song_t s{};
    s.n_frames = n_in;
    s.frame_stride = 4;
    s.channel_stride = 4 * n_in;
    s.channels = channels;
    s.sample_rate = sr_in;
    s.format = ETUDE_PCM_F32;
    return etude_ingest_pcm(h, pcm, &s, 1, sr_out, wave_out, stream);
}

extern "C" int64_t etude_feature_rows(int64_t n_samples) {
    const int64_t t = 1 + n_samples / kHop;
    const int64_t t_pad = (t + kFrames - 1) / kFrames * kFrames;
    return t_pad + 2 * kMargin;
}

extern "C" int etude_logmel_layout(etude_handle_t* h, const float* wave, const int64_t* wave_off, const int64_t* n_samples, int n_songs,
                                   float* feat, const int64_t* feat_row_off, const int64_t* feat_rows, int front_rows, float pad_value,
                                   int pad_reflect, void* stream) {
    if (!h || !wave || !feat || !wave_off || !n_samples || !feat_row_off || !feat_rows) return fail("etude_logmel: null argument");
    if (n_songs <= 0 || n_songs > h->max_songs) return fail("etude_logmel: n_songs=%d out of range (1..%d)", n_songs, h->max_songs);
    if (front_rows < 0) return fail("etude_logmel: front_rows=%d", front_rows);
    CUDA_OK(cudaSetDevice(h->device));
    std::vector<LogmelSong> songs(n_songs);
    int64_t max_rows = 0;
    for (int s = 0; s < n_songs; ++s) {
        // torch.stft needs the reflect padding (n_fft / 2 per side) to be shorter than the signal; constant padding does not
        if (n_samples[s] < 1 || (pad_reflect && n_samples[s] <= kNfft / 2))
            return fail("etude_logmel: song %d has %lld samples; reflect padding needs more than %d", s, (long long)n_samples[s], kNfft / 2);
        songs[s].wave_off = wave_off[s];
        songs[s].n_samples = n_samples[s];
        songs[s].row_off = feat_row_off[s];
        songs[s].n_rows = feat_rows[s];
        songs[s].n_frames = 1 + n_samples[s] / kHop;
        songs[s].front_rows = front_rows;
        if (feat_rows[s] < front_rows + songs[s].n_frames)
            return fail("etude_logmel: song %d: %lld rows cannot hold %d pad rows + %lld frames", s, (long long)feat_rows[s], front_rows, (long long)songs[s].n_frames);
        max_rows = std::max(max_rows, songs[s].n_rows);
    }
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_OK(cudaMemcpyAsync(h->d_songs, songs.data(), sizeof(LogmelSong) * n_songs, cudaMemcpyHostToDevice, st));
    if (set_func_attrs_once()) return -1;
    const int rows_per_cta = kL2RowsPerCta;
    dim3 grid((unsigned)((max_rows + rows_per_cta - 1) / rows_per_cta), (unsigned)n_songs);
    double alg_bytes = 0;  // SURVEY 8(d): 4 B per sample in + 4 B x 256 per frame out
    for (int s = 0; s < n_songs; ++s) alg_bytes += 4.0 * n_samples[s] + 4.0 * kBins * songs[s].n_frames;
    cudaEvent_t ev = h->prof.begin(PC_LOGMEL, st, 0.0, alg_bytes);
    logmel2_kernel<<<grid, kL2Threads, kLogmel2SmemBytes, st>>>(wave, h->d_songs, h->tab, h->tw32x32, feat, pad_value, 1e-8f, pad_reflect);
    h->prof.end(ev, st);
    CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int etude_logmel(etude_handle_t* h, const float* wave, const int64_t* wave_off, const int64_t* n_samples, int n_songs,
                            float* feat, const int64_t* feat_row_off, void* stream) {
    if (!n_samples || n_songs <= 0) return fail("etude_logmel: null argument");
    std::vector<int64_t> rows(n_songs);
    for (int s = 0; s < n_songs; ++s) rows[s] = etude_feature_rows(n_samples[s]);
    return etude_logmel_layout(h, wave, wave_off, n_samples, n_songs, feat, feat_row_off, rows.data(), kMargin, -18.0f, 1, stream);
}

// ------------------------------------------------------------------------------------------------ model forward
struct Workspace {  // every activation is bf16 [tokens, width]; nothing fp32 between kernels
    __nv_bfloat16* x; __nv_bfloat16* qkv; __nv_bfloat16* ctx; __nv_bfloat16* kv;
    __nv_bfloat16* d; __nv_bfloat16* dqkv; __nv_bfloat16* dctx; __nv_bfloat16* dq; __nv_bfloat16* t;
};
static size_t carve(Workspace* ws, uint8_t* base, int nw, int frames) {
    const size_t NT = (size_t)nw * frames * kBins, ND = (size_t)nw * frames * kNotes;
    size_t off = 0;
    auto take = [&](size_t bytes) { uint8_t* p = base ? base + off : nullptr; off += (bytes + 1023) & ~size_t(1023); return p; };
    Workspace w;
    w.x = (__nv_bfloat16*)take(NT * 256 * 2);
    w.qkv = (__nv_bfloat16*)take(NT * 768 * 2);
    w.ctx = (__nv_bfloat16*)take(NT * 256 * 2);
    w.kv = (__nv_bfloat16*)take(NT * 1536 * 2);
    w.d = (__nv_bfloat16*)take(ND * 256 * 2);
    w.dqkv = (__nv_bfloat16*)take(ND * 768 * 2);
    w.dctx = (__nv_bfloat16*)take(ND * 256 * 2);
    w.dq = (__nv_bfloat16*)take(ND * 256 * 2);
    w.t = (__nv_bfloat16*)take(ND * 256 * 2);
    if (ws) *ws = w;
    return off;
}

// windows per call: the same token budget for both window lengths (64 x 512 frames = 256 x 128 frames)
static int max_windows_of(const etude_handle_t* h) { return ETUDE_MAX_WINDOWS * (kFrames / h->frames); }

extern "C" int etude_n_frame(const etude_handle_t* h) { return h ? h->frames : 0; }
extern "C" int etude_max_windows(const etude_handle_t* h) { return h ? max_windows_of(h) : 0; }

extern "C" size_t etude_workspace_bytes(const etude_handle_t* h, int max_windows) {
    if (!h) return 0;
    if (max_windows < 1) max_windows = 1;
    if (max_windows > max_windows_of(h)) max_windows = max_windows_of(h);
    return carve(nullptr, nullptr, max_windows, h->frames) + 1024;
}

// x = LN(x + MHA(x)); x = LN(x + FFN(x)) over n_seq sequences of L tokens   (EncoderLayer, amt_apc.py:244-259):
// Q|K|V projection GEMM, fused attention, then everything after the attention core in one chain kernel (x in place).
static int self_layer(const LayerW& L, __nv_bfloat16* x, __nv_bfloat16* qkv, __nv_bfloat16* ctx, int n_seq, int len, cudaStream_t st,
                      Profile* prof) {
    const int M = n_seq * len;
    if (gemm_bias(x, L.qkv, M, qkv, st, prof)) return -1;
    if (launch_attention(qkv, M, 768, 0, len, qkv, 768, 256, 512, n_seq, len, len, ctx, nullptr, st, prof)) return -1;
    return launch_chain(ctx, L.o, &L.f1, &L.f2, L.ln_g, L.ln_b, x, 0, M, x, M, st, prof);
}

// Token embedding over nw windows (h->d_win_row already holds their first padded rows): out bf16 [nw * frames * 256, 256].
static int launch_embed(etude_handle_t* h, const float* feat, int nw, __nv_bfloat16* out, cudaStream_t st, Profile* prof, int no_store = 0) {
    const int NF = nw * h->frames;
    CUtensorMap tw, tout;
    if (make_tmap(&tw, h->w_embed_bf16, 256, 64, 64, 256)) return -1;
    if (make_tmap_3d(&tout, out, kBins, (uint64_t)NF, 1, 32)) return -1;
    cudaEvent_t ev_embed = prof ? prof->begin(PC_EMBED, st, 2.0 * NF * 256.0 * 256.0 * kProc, 0.0) : nullptr;
    Embed2Params ep{feat, h->d_win_row, h->w64, h->posb, nw, h->frames / 128, no_store};
    const int n_jobs = nw * ep.fblocks * (kBins / kE2BinsPerJob);
    embed2_kernel<<<std::min(n_jobs, num_sms_cached()), kE2Threads, kEmbed2SmemBytes, st>>>(tw, tout, ep);
    if (prof) prof->end(ev_embed, st);
    CUDA_OK(cudaGetLastError());
    return debug_sync("embed", st);
}

extern "C" int etude_k_embed(etude_handle_t* h, const float* feat, const int64_t* win_row, int nw, void* out_bf16, int variant, void* stream) {
    if (!h || !feat || !win_row || !out_bf16) return fail("etude_k_embed: null argument");
    if (nw < 1 || nw > max_windows_of(h)) return fail("etude_k_embed: n_windows=%d out of range", nw);
    if (set_func_attrs_once()) return -1;
    CUDA_OK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_OK(cudaMemcpyAsync(h->d_win_row, win_row, sizeof(int64_t) * nw, cudaMemcpyHostToDevice, st));
    return launch_embed(h, feat, nw, (__nv_bfloat16*)out_bf16, st, nullptr, variant >= 16 ? variant - 16 : 0);
}

static int check_rolls(const char* who, void* const rolls[4], const char* name) {
    if (rolls)
        for (int i = 0; i < 4; ++i)
            if (!rolls[i]) return fail("%s: %s[%d] is null (pass %s = NULL to skip those heads)", who, name, i, name);
    return 0;
}

// The heads GEMM of forward_impl alone, on caller-supplied weights (the epilogue is the only place the rolls are written).
extern "C" int etude_k_heads(etude_handle_t* h, const void* x_bf16, const void* w_bf16, const float* bias, int nw, int time_major,
                             const int64_t* out_row, int keep0, int keepn, void* const rolls[4], float* vel_logits, void* stream) {
    if (!h || !x_bf16 || !w_bf16 || !bias || !out_row || !rolls) return fail("etude_k_heads: null argument");
    if (check_rolls("etude_k_heads", rolls, "rolls")) return -1;
    if (nw < 1 || nw > max_windows_of(h)) return fail("etude_k_heads: n_windows=%d out of range (1..%d)", nw, max_windows_of(h));
    if (keep0 < 0 || keepn < 1 || keep0 + keepn > h->frames)
        return fail("etude_k_heads: kept frames [%d, %d) outside the %d-frame window", keep0, keep0 + keepn, h->frames);
    if (set_func_attrs_once()) return -1;
    CUDA_OK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_OK(cudaMemcpyAsync(h->d_out_row, out_row, sizeof(int64_t) * nw, cudaMemcpyHostToDevice, st));
    GemmParams p{};
    p.M = nw * h->frames * kNotes; p.N = 144; p.K = 256; p.bias = bias; p.heads_time_major = time_major ? 1 : 0; p.heads_row0 = h->d_out_row;
    p.roll_onset = (float*)rolls[0]; p.roll_offset = (float*)rolls[1]; p.roll_mpe = (float*)rolls[2];
    p.roll_velocity = (int8_t*)rolls[3]; p.vel_logits = vel_logits;
    p.frames = h->frames; p.keep0 = keep0; p.keepn = keepn;
    return launch_gemm<144, EPI_HEADS>(x_bf16, w_bf16, p, GemmIO{}, st, nullptr);
}

// The decoder's time-axis transpose of forward_impl alone, with the handle's pos_time table and window length.
extern "C" int etude_k_transpose_time(etude_handle_t* h, const void* in_bf16, int nw, void* out_bf16, void* stream) {
    if (!h || !in_bf16 || !out_bf16) return fail("etude_k_transpose_time: null argument");
    if (nw < 1 || nw > max_windows_of(h)) return fail("etude_k_transpose_time: n_windows=%d out of range (1..%d)", nw, max_windows_of(h));
    CUDA_OK(cudaSetDevice(h->device));
    const int ND = nw * h->frames * kNotes;
    transpose_time_kernel<<<(ND + 7) / 8, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)in_bf16, h->pos_time, 16.f, ND, h->frames,
                                                                         (__nv_bfloat16*)out_bf16);
    CUDA_OK(cudaGetLastError());
    return debug_sync("transpose_time", (cudaStream_t)stream);
}

// What one pass over nw windows reads and writes; the public entry points below are thin views of it.
struct ForwardIO {
    const float* feat = nullptr;        // padded feature blocks (encoder input) ...
    const int64_t* win_row = nullptr;   //   ... and the first padded row of every window
    const float* enc_in = nullptr;      // or: the encoder output fp32 [nw * frames * 256, 256] (decode only)
    float* enc_out = nullptr;           // encode only: the encoder output, fp32
    const int64_t* out_row = nullptr;   // first roll row of every window
    void* const* rolls_A = nullptr;     // frequency-axis heads (optional)
    void* const* rolls_B = nullptr;     // time-axis heads (optional: without them the time-axis layers are skipped)
    float* vel_logits_A = nullptr;
    float* vel_logits_B = nullptr;
    float* attention = nullptr;
    int keep0 = 0, keepn = 0;           // window frames that reach the rolls (0, frames = all)
};

static int forward_impl(etude_handle_t* h, const ForwardIO& io, int nw, void* workspace, size_t workspace_bytes, cudaStream_t st) {
    const int F = h->frames;
    CUDA_OK(cudaSetDevice(h->device));
    if (set_func_attrs_once()) return -1;
    uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 1023) & ~uintptr_t(1023));
    Workspace ws;
    const size_t need = carve(&ws, base, nw, F) + (size_t)(base - (uint8_t*)workspace);
    if (need > workspace_bytes) return fail("etude: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
    if (io.win_row) CUDA_OK(cudaMemcpyAsync(h->d_win_row, io.win_row, sizeof(int64_t) * nw, cudaMemcpyHostToDevice, st));
    if (io.out_row) CUDA_OK(cudaMemcpyAsync(h->d_out_row, io.out_row, sizeof(int64_t) * nw, cudaMemcpyHostToDevice, st));

    const int NF = nw * F;               // frames
    const int NT = NF * kBins;           // encoder tokens
    const int ND = NF * kNotes;          // decoder tokens
    Profile* prof = &h->prof;
    const size_t enc_n8 = (size_t)NT * kHid / 8;
    // --- encoder: embedding + 3 frequency-axis layers (Encoder_SPEC2MIDI.forward, amt_apc.py:74-120)
    if (io.enc_in) {
        cvt_f32_to_bf16_kernel<<<(unsigned)((enc_n8 + 255) / 256), 256, 0, st>>>(io.enc_in, ws.x, enc_n8);
        CUDA_OK(cudaGetLastError());
    } else {
        if (launch_embed(h, io.feat, nw, ws.x, st, prof)) return -1;
        for (int l = 0; l < 3; ++l) {   // EncoderLayer (amt_apc.py:244-259): fused Q|K|V projection + attention, then the chain
            const LayerW& L = h->enc[l];
            if (launch_attn_qkv(ws.x, L.qkv_hm.w, L.qkv_hm.b, NF, ws.ctx, st, prof)) return -1;
            if (launch_chain(ws.ctx, L.o, &L.f1, &L.f2, L.ln_g, L.ln_b, ws.x, 0, NT, ws.x, NT, st, prof)) return -1;
        }
    }
    if (io.enc_out) {
        cvt_bf16_to_f32_kernel<<<(unsigned)((enc_n8 + 255) / 256), 256, 0, st>>>(ws.x, io.enc_out, enc_n8);
        CUDA_OK(cudaGetLastError());
    }
    if (!io.rolls_A && !io.rolls_B) return 0;   // encode only
    // --- decoder, frequency -> note (Decoder_SPEC2MIDI.forward part 1, amt_apc.py:159-183)
    if (gemm_bias(ws.x, h->kv_all, NT, ws.kv, st, prof)) return -1;  // K|V of all three cross-attentions
    // layer zero: cross-attention with the input-independent queries, then fc_o + LN + FFN + LN (residual = the query embedding)
    if (launch_attention(h->q0, 128, 256, 0, 0, ws.kv, 1536, 0, 256, NF, kNotes, kBins, ws.dctx, nullptr, st, prof)) return -1;
    if (launch_chain(ws.dctx, h->dec0.co, &h->dec0.f1, &h->dec0.f2, h->dec0.ln_g, h->dec0.ln_b, h->pos_freq_bf16, kNotes, 3 * kNotes, ws.d, ND,
                     st, prof)) return -1;
    for (int l = 0; l < 2; ++l) {
        const LayerW& L = h->dec[l];
        if (gemm_bias(ws.d, L.qkv, ND, ws.dqkv, st, prof)) return -1;
        if (launch_attention(ws.dqkv, ND, 768, 0, kNotes, ws.dqkv, 768, 256, 512, NF, kNotes, kNotes, ws.dctx, nullptr, st, prof)) return -1;
        if (launch_chain(ws.dctx, L.o, nullptr, nullptr, L.ln_g, L.ln_b, ws.d, 0, ND, ws.d, ND, st, prof)) return -1;
        if (gemm_bias(ws.d, L.cq, ND, ws.dq, st, prof)) return -1;
        if (launch_attention(ws.dq, ND, 256, 0, kNotes, ws.kv, 1536, (l + 1) * 512, (l + 1) * 512 + 256, NF, kNotes, kBins, ws.dctx,
                             (l == 1) ? io.attention : nullptr, st, prof)) return -1;
        if (launch_chain(ws.dctx, L.co, &L.f1, &L.f2, L.ln_g, L.ln_b, ws.d, 0, ND, ws.d, ND, st, prof)) return -1;
    }
    auto heads = [&](const Linear& W, const __nv_bfloat16* src, void* const* rolls, float* logits, int time_major) -> int {
        GemmParams p{};
        p.M = ND; p.N = 144; p.K = 256; p.bias = W.b; p.heads_time_major = time_major; p.heads_row0 = h->d_out_row;
        p.roll_onset = (float*)rolls[0]; p.roll_offset = (float*)rolls[1]; p.roll_mpe = (float*)rolls[2];
        p.roll_velocity = (int8_t*)rolls[3]; p.vel_logits = logits;
        p.frames = F; p.keep0 = io.keep0; p.keepn = io.keepn;
        return launch_gemm<144, EPI_HEADS>(src, W.w, p, GemmIO{}, st, prof);
    };
    // heads_freq (amt_apc.py:186-189): dead for extract(), kept for _transcript / the 9-tuple
    if (io.rolls_A && heads(h->heads_f, ws.d, io.rolls_A, io.vel_logits_A, 0)) return -1;
    if (!io.rolls_B) return 0;   // frequency-axis outputs only (_transcript(mode != "combination"))
    {   // the single global transpose: (window, frame, note) -> (window, note, frame), *16 + pos_time (amt_apc.py:203-205)
        cudaEvent_t ev = prof->begin(PC_TRANSPOSE, st, 0.0, (double)ND * 256 * (2 + 2));
        transpose_time_kernel<<<(ND + 7) / 8, 256, 0, st>>>(ws.d, h->pos_time, 16.f, ND, F, ws.t);
        prof->end(ev, st);
        CUDA_OK(cudaGetLastError());
    }
    // --- decoder, time axis (amt_apc.py:203-220): 3 layers over the window's frames, batch = windows x 88 notes
    for (int l = 0; l < 3; ++l)
        if (self_layer(h->tim[l], ws.t, ws.dqkv, ws.dctx, nw * kNotes, F, st, prof)) return -1;
    return heads(h->heads_t, ws.t, io.rolls_B, io.vel_logits_B, 1);
}

extern "C" int etude_forward_windows(etude_handle_t* h, const float* feat, const int64_t* win_row, const int64_t* out_row, int nw,
                                     void* const rolls_A[4], void* const rolls_B[4], float* vel_logits_A, float* vel_logits_B,
                                     float* attention, void* workspace, size_t workspace_bytes, void* stream) {
    if (!h || !feat || !win_row || !out_row || !workspace) return fail("etude_forward_windows: null argument");
    if (nw < 1 || nw > max_windows_of(h)) return fail("etude_forward_windows: n_windows=%d out of range (1..%d)", nw, max_windows_of(h));
    if (!rolls_A && !rolls_B) return fail("etude_forward_windows: both rolls_A and rolls_B are null");
    if (check_rolls("etude_forward_windows", rolls_A, "rolls_A") || check_rolls("etude_forward_windows", rolls_B, "rolls_B")) return -1;
    if (vel_logits_A && !rolls_A) return fail("etude_forward_windows: vel_logits_A needs rolls_A");
    if ((vel_logits_B || attention) && !rolls_B && !rolls_A) return fail("etude_forward_windows: model-level outputs need the rolls");
    if (vel_logits_B && !rolls_B) return fail("etude_forward_windows: vel_logits_B needs rolls_B");
    ForwardIO io;
    io.feat = feat; io.win_row = win_row; io.out_row = out_row; io.rolls_A = rolls_A; io.rolls_B = rolls_B;
    io.vel_logits_A = vel_logits_A; io.vel_logits_B = vel_logits_B; io.attention = attention; io.keep0 = 0; io.keepn = h->frames;
    return forward_impl(h, io, nw, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int etude_forward_windows_stride(etude_handle_t* h, const float* feat, const int64_t* win_row, const int64_t* out_row, int nw,
                                            void* const rolls_A[4], void* const rolls_B[4], int keep_first, int keep_count,
                                            void* workspace, size_t workspace_bytes, void* stream) {
    if (!h || !feat || !win_row || !out_row || !workspace) return fail("etude_forward_windows_stride: null argument");
    if (nw < 1 || nw > max_windows_of(h)) return fail("etude_forward_windows_stride: n_windows=%d out of range (1..%d)", nw, max_windows_of(h));
    if (!rolls_A && !rolls_B) return fail("etude_forward_windows_stride: both rolls_A and rolls_B are null");
    if (check_rolls("etude_forward_windows_stride", rolls_A, "rolls_A") || check_rolls("etude_forward_windows_stride", rolls_B, "rolls_B")) return -1;
    if (keep_first < 0 || keep_count < 1 || keep_first + keep_count > h->frames)
        return fail("etude_forward_windows_stride: kept frames [%d, %d) outside the %d-frame window", keep_first, keep_first + keep_count, h->frames);
    ForwardIO io;
    io.feat = feat; io.win_row = win_row; io.out_row = out_row; io.rolls_A = rolls_A; io.rolls_B = rolls_B;
    io.keep0 = keep_first; io.keepn = keep_count;
    return forward_impl(h, io, nw, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int etude_encode_windows(etude_handle_t* h, const float* feat, const int64_t* win_row, int nw, float* enc_out, void* workspace,
                                    size_t workspace_bytes, void* stream) {
    if (!h || !feat || !win_row || !enc_out || !workspace) return fail("etude_encode_windows: null argument");
    if (nw < 1 || nw > max_windows_of(h)) return fail("etude_encode_windows: n_windows=%d out of range (1..%d)", nw, max_windows_of(h));
    ForwardIO io;
    io.feat = feat; io.win_row = win_row; io.enc_out = enc_out;
    return forward_impl(h, io, nw, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int etude_decode_windows(etude_handle_t* h, const float* enc_in, const int64_t* out_row, int nw, void* const rolls_A[4],
                                    void* const rolls_B[4], float* vel_logits_A, float* vel_logits_B, float* attention, void* workspace,
                                    size_t workspace_bytes, void* stream) {
    if (!h || !enc_in || !out_row || !workspace) return fail("etude_decode_windows: null argument");
    if (nw < 1 || nw > max_windows_of(h)) return fail("etude_decode_windows: n_windows=%d out of range (1..%d)", nw, max_windows_of(h));
    if (!rolls_A && !rolls_B) return fail("etude_decode_windows: both rolls_A and rolls_B are null");
    if (check_rolls("etude_decode_windows", rolls_A, "rolls_A") || check_rolls("etude_decode_windows", rolls_B, "rolls_B")) return -1;
    if ((vel_logits_A && !rolls_A) || (vel_logits_B && !rolls_B)) return fail("etude_decode_windows: velocity logits need their rolls");
    ForwardIO io;
    io.enc_in = enc_in; io.out_row = out_row; io.rolls_A = rolls_A; io.rolls_B = rolls_B;
    io.vel_logits_A = vel_logits_A; io.vel_logits_B = vel_logits_B; io.attention = attention; io.keep0 = 0; io.keepn = h->frames;
    return forward_impl(h, io, nw, workspace, workspace_bytes, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------ profiling
extern "C" int etude_profile_classes(void) { return PC_COUNT; }
extern "C" const char* etude_profile_class_name(int cls) { return (cls >= 0 && cls < PC_COUNT) ? kProfNames[cls] : ""; }

extern "C" int etude_profile_reset(etude_handle_t* h, int enable_timing) {
    if (!h) return fail("etude_profile_reset: null handle");
    Profile& p = h->prof;
    p.timing = enable_timing != 0;
    for (int c = 0; c < PC_COUNT; ++c) { p.launches[c] = 0; p.flops[c] = 0; p.bytes[c] = 0; }
    p.used = 0;
    p.pair_class.clear();
    return 0;
}

extern "C" int etude_profile_read(etude_handle_t* h, double* ms, int64_t* launches, double* flops, double* bytes) {
    if (!h || !ms || !launches || !flops || !bytes) return fail("etude_profile_read: null argument");
    CUDA_OK(cudaSetDevice(h->device));
    CUDA_OK(cudaDeviceSynchronize());
    Profile& p = h->prof;
    for (int c = 0; c < PC_COUNT; ++c) { ms[c] = 0; launches[c] = p.launches[c]; flops[c] = p.flops[c]; bytes[c] = p.bytes[c]; }
    for (size_t i = 0; i < p.pair_class.size(); ++i) {
        float t = 0.f;
        CUDA_OK(cudaEventElapsedTime(&t, p.pool[2 * i], p.pool[2 * i + 1]));
        ms[p.pair_class[i]] += t;
    }
    return 0;
}

// Per-launch timeline of the profiled pass: start (ms after the first profiled launch began) and duration of launch i,
// in recording order; returns the number of launches written (<= cap).  Shows the idle time BETWEEN kernels.
extern "C" int etude_profile_timeline(etude_handle_t* h, double* start_ms, double* dur_ms, int32_t* cls, int cap) {
    if (!h || !start_ms || !dur_ms || !cls) return fail("etude_profile_timeline: null argument");
    CUDA_OK(cudaSetDevice(h->device));
    CUDA_OK(cudaDeviceSynchronize());
    Profile& p = h->prof;
    const int n = (int)std::min<size_t>(p.pair_class.size(), (size_t)std::max(cap, 0));
    for (int i = 0; i < n; ++i) {
        float t0 = 0.f, t = 0.f;
        CUDA_OK(cudaEventElapsedTime(&t0, p.pool[0], p.pool[2 * i]));
        CUDA_OK(cudaEventElapsedTime(&t, p.pool[2 * i], p.pool[2 * i + 1]));
        start_ms[i] = t0; dur_ms[i] = t; cls[i] = p.pair_class[i];
    }
    return n;
}

// ------------------------------------------------------------------------------------------------ notes
// Device scratch of the note stage, sized by (roll rows, songs) of one call: pitch-major roll copies, note slabs (one record
// slot per frame and pitch: the worst case), their sorted copy, the per-chunk tables.  Grown here, never inside the kernels'
// critical section; etude_notes_reserve lets the caller do it once, up front.
static int notes_reserve(etude_handle* h, int64_t rows, int n_songs) {
    if (rows <= h->notes_rows_cap && n_songs <= h->notes_songs_cap) return 0;
    const int64_t new_rows = std::max(rows, h->notes_rows_cap), cells = new_rows * kNotes;
    const int new_songs = std::max(n_songs, h->notes_songs_cap);
    const int64_t chunks = (new_rows / kNoteChunk + new_songs) * kNotes;   // sum over songs of ceil(rows_s / chunk) <= rows / chunk + songs
    CUDA_OK(cudaDeviceSynchronize());   // nothing may still be using the old buffers
    for (void** pp : {(void**)&h->notes_scratch, (void**)&h->d_notes, (void**)&h->d_onsets, (void**)&h->d_sorted, (void**)&h->d_chunk_tab})
        if (*pp) { cudaFree(*pp); *pp = nullptr; }
    h->notes_rows_cap = 0; h->notes_songs_cap = 0;
    CUDA_OK(cudaMalloc((void**)&h->notes_scratch, 3 * cells * sizeof(float)));
    CUDA_OK(cudaMalloc((void**)&h->d_notes, cells * sizeof(NoteRec)));
    CUDA_OK(cudaMalloc((void**)&h->d_onsets, cells * sizeof(double)));
    CUDA_OK(cudaMalloc((void**)&h->d_sorted, cells * sizeof(NoteRec)));
    CUDA_OK(cudaMalloc((void**)&h->d_chunk_tab, 4 * chunks * sizeof(int32_t)));
    h->notes_rows_cap = new_rows; h->notes_songs_cap = new_songs; h->notes_chunks_cap = chunks;
    return 0;
}

extern "C" int etude_notes_reserve(etude_handle_t* h, int64_t max_rows, int max_songs) {
    if (!h) return fail("etude_notes_reserve: null handle");
    if (max_rows < 1 || max_songs < 1 || max_songs > h->max_songs) return fail("etude_notes_reserve: bad sizes (rows=%lld, songs=%d)", (long long)max_rows, max_songs);
    CUDA_OK(cudaSetDevice(h->device));
    return notes_reserve(h, max_rows, max_songs);
}

// Kernels + the per-song counts (one host round trip); the sorted records stay on the device (h->d_sorted).
extern "C" int etude_notes_begin(etude_handle_t* h, const float* onset, const float* offset, const float* mpe, const int8_t* velocity,
                                 const int64_t* song_row_off, const int64_t* song_rows, int n_songs, int note_min, double hop_sec,
                                 double thred_onset, double thred_offset, double thred_mpe, int mode_velocity, int mode_offset,
                                 int64_t* n_notes, void* stream) {
    if (!h || !onset || !offset || !mpe || !velocity || !song_row_off || !song_rows || !n_notes)
        return fail("etude_notes: null argument");
    if (n_songs <= 0 || n_songs > h->max_songs) return fail("etude_notes: n_songs=%d out of range (1..%d)", n_songs, h->max_songs);
    static_assert(sizeof(etude_note_t) == sizeof(NoteRec), "note record layout");
    CUDA_OK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    std::vector<NotesSong> songs(n_songs);
    int64_t max_rows = 0, rows = 0;
    int chunks = 0, max_items = 0;
    for (int s = 0; s < n_songs; ++s) {
        if (song_rows[s] < 1 || song_row_off[s] < 0) return fail("etude_notes: song %d has an empty or negative row range", s);
        const int nc = (int)((song_rows[s] + kNoteChunk - 1) / kNoteChunk);
        songs[s] = NotesSong{song_row_off[s], song_rows[s], rows, chunks * kNotes, nc};   // scratch is indexed relative to this call
        rows += song_rows[s];
        chunks += nc;
        max_rows = std::max(max_rows, song_rows[s]);
        max_items = std::max(max_items, nc * kNotes);
    }
    if (notes_reserve(h, rows, n_songs)) return -1;
    CUDA_OK(cudaMemcpyAsync(h->d_nsongs, songs.data(), sizeof(NotesSong) * n_songs, cudaMemcpyHostToDevice, st));
    const int64_t cells = h->notes_rows_cap * kNotes;
    float* t_on = h->notes_scratch; float* t_off = t_on + cells; float* t_mpe = t_off + cells;
    NotesParams p{};
    p.onset = t_on; p.offset = t_off; p.mpe = t_mpe; p.velocity = velocity; p.songs = h->d_nsongs; p.n_songs = n_songs;
    p.note_min = note_min; p.hop_sec = hop_sec;
    p.thr_onset = (float)thred_onset; p.thr_offset = (float)thred_offset; p.thr_mpe = (float)thred_mpe;  // NEP 50: float32 compares
    p.mode_velocity = mode_velocity; p.mode_offset = mode_offset;
    p.first_on = h->d_chunk_tab; p.first_kept = p.first_on + h->notes_chunks_cap; p.first_off = p.first_kept + h->notes_chunks_cap;
    p.chunk_count = p.first_off + h->notes_chunks_cap;
    p.counts = h->d_counts; p.notes = (NoteRec*)h->d_notes; p.onsets = h->d_onsets;
    cudaEvent_t ev = h->prof.begin(PC_NOTES, st, 0.0, 0.0);
    notes_transpose_kernel<<<dim3((unsigned)((max_rows + 31) / 32), (unsigned)n_songs, 3), 256, 0, st>>>(onset, offset, mpe, h->d_nsongs,
                                                                                                  t_on, t_off, t_mpe);
    const dim3 item_grid((unsigned)((max_items + 63) / 64), (unsigned)n_songs);   // small blocks: the walks are latency-bound, spread them over the SMs
    notes_scan_kernel<<<item_grid, 64, 0, st>>>(p);
    notes_walk_kernel<<<item_grid, 64, 0, st>>>(p);
    notes_compact_kernel<<<(n_songs * kNotes * 32 + 127) / 128, 128, 0, st>>>(p);
    notes_bases_kernel<<<1, 256, 0, st>>>(h->d_counts, n_songs, h->d_song_base, h->d_song_total);
    // the counts are not known on the host: enough blocks for four notes per thread in the worst case (one note per frame and
    // pitch), i.e. about one per thread at the densities seen; a thread's 87 binary searches are dependent L2 loads
    const unsigned rank_blocks = (unsigned)std::max<int64_t>(1, (max_rows * kNotes + 4 * 256 - 1) / (4 * 256));
    notes_rank_kernel<<<dim3(rank_blocks, (unsigned)n_songs), 256, 0, st>>>((const NoteRec*)h->d_notes, h->d_onsets, h->d_nsongs, h->d_counts,
                                                                    h->d_song_base, (NoteRec*)h->d_sorted);
    h->prof.end(ev, st);
    h->prof.launches[PC_NOTES] += 5;   // six kernels under one event pair
    CUDA_OK(cudaGetLastError());
    // the one host round trip of the call, after the last kernel: per-song counts, then exactly `total` sorted records
    CUDA_OK(cudaMemcpyAsync(h->h_song_total, h->d_song_total, sizeof(int64_t) * (n_songs + 1), cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaStreamSynchronize(st));
    for (int s = 0; s < n_songs; ++s) n_notes[s] = h->h_song_total[s];
    h->notes_last_total = h->h_song_total[n_songs];
    return 0;
}

// Second half of the round trip: exactly the records of the last etude_notes_begin call, into caller-owned host memory
// (pinned memory makes it one DMA transfer; pageable memory works too).
extern "C" int etude_notes_fetch(etude_handle_t* h, etude_note_t* dst_host, int64_t n_records, void* stream) {
    if (!h || (!dst_host && n_records > 0)) return fail("etude_notes_fetch: null argument");
    if (n_records < 0 || n_records > h->notes_last_total)
        return fail("etude_notes_fetch: %lld records asked, the last call produced %lld", (long long)n_records, (long long)h->notes_last_total);
    CUDA_OK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (n_records > 0) {
        CUDA_OK(cudaMemcpyAsync(dst_host, h->d_sorted, n_records * sizeof(NoteRec), cudaMemcpyDeviceToHost, st));
        CUDA_OK(cudaStreamSynchronize(st));
    }
    return 0;
}

extern "C" int etude_notes(etude_handle_t* h, const float* onset, const float* offset, const float* mpe, const int8_t* velocity,
                           const int64_t* song_row_off, const int64_t* song_rows, int n_songs, int note_min, double hop_sec,
                           double thred_onset, double thred_offset, double thred_mpe, int mode_velocity, int mode_offset,
                           const etude_note_t** notes_out, int64_t* n_notes, void* stream) {
    if (!notes_out) return fail("etude_notes: null argument");
    if (etude_notes_begin(h, onset, offset, mpe, velocity, song_row_off, song_rows, n_songs, note_min, hop_sec, thred_onset, thred_offset,
                          thred_mpe, mode_velocity, mode_offset, n_notes, stream))
        return -1;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t total = h->notes_last_total;
    if (total > h->h_notes_cap) {   // pinned staging of the result (grows geometrically; library-owned)
        if (h->h_notes_pinned) cudaFreeHost(h->h_notes_pinned);
        h->h_notes_pinned = nullptr; h->h_notes_cap = 0;
        const int64_t cap = total + total / 2 + 4096;
        CUDA_OK(cudaHostAlloc(&h->h_notes_pinned, cap * sizeof(NoteRec), cudaHostAllocDefault));
        h->h_notes_cap = cap;
    }
    if (total > 0) {
        CUDA_OK(cudaMemcpyAsync(h->h_notes_pinned, h->d_sorted, total * sizeof(NoteRec), cudaMemcpyDeviceToHost, st));
        CUDA_OK(cudaStreamSynchronize(st));
    }
    *notes_out = (const etude_note_t*)h->h_notes_pinned;
    return 0;
}
