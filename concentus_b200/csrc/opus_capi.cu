// opus_capi.cu — kernels and the C ABI of libconcentus_b200.so (declared in include/opus_b200.h).
//
// Boundary: libopus's public decoder API (opus-fix/include/opus.h:406-512) plus our batch / span calls.
// Host side = argument checks, ctl, state residency and copies; everything from TOC parsing and ec_dec_init down runs on
// the device as a two-stage pipeline: parse_kernel (one thread per run of packets: range decoder, allocation, PVQ band
// loop -> IR in HBM) and synth_kernel (one warp per stream: energies, anti-collapse, IMDCT, post-filter, de-emphasis,
// all persistent state).  Time chunks are double-buffered so stage A of chunk c+1 overlaps stage B of chunk c.
// There is NO CPU path: if CUDA is unusable every codec call returns OPUS_INTERNAL_ERROR.
#define CB_SMALL_CODE 1   // celt_simt.cuh: real calls for the medium-sized helpers and no loop unrolling — the decoder stages were 50-55 % instruction-fetch stalled with everything inlined (profiles/r1_dec_*), +30 % throughput
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <unordered_set>
#include <vector>

#include "../../include/opus_b200.h"
#include "host_runtime.h"
#include "opus_decoder_dev.cuh"
#include "opus_multistream.h"

using namespace cb;

// ------------------------------------------------------------------------------------------------
// Caller-visible state block.  Pointer-free and memcpy-able like the reference's (tests/test_opus_decode.c:84-95):
// `st` is the authoritative serialised state whenever host_current != 0; after a batch/span call the
// authoritative copy is the HBM slot (slot, gen) and host_current == 0 until the next sync.
// ------------------------------------------------------------------------------------------------
struct OpusDecoder {
    uint32_t magic;
    int32_t slot;          // device pool slot or -1
    uint64_t gen;          // generation of the slot contents this block refers to
    int32_t host_current;  // 1: `st` below is up to date
    int32_t device;        // the device whose pool `slot` refers to
    CbDecState st;
};
static const uint32_t kDecMagic = 0x0B200DECu;

// ------------------------------------------------------------------------------------------------
// Kernels (DESIGN.md §3)
// ------------------------------------------------------------------------------------------------
#ifndef CB_PARSE_THREADS
#define CB_PARSE_THREADS 128   // stage A block
#endif
#ifndef CB_PARSE_MINBLOCKS
#define CB_PARSE_MINBLOCKS 8   // stage A: min resident blocks per SM (register cap 64; 4/6/8/10 measured within 3 %, 8 best)
#endif
#ifndef CB_WPB
#define CB_WPB 4               // stage B: warps (= streams) per block
#endif
#ifndef CB_SYNTH_MINBLOCKS
#define CB_SYNTH_MINBLOCKS 8
#endif

struct IrView {
    CbPacketIR *pk;      // [n * Fc]
    CbFrameIR *fr;       // [n * Fc * kmax]
    int16_t *X;          // [n * Fc * xstride]
    int *sig;            // [n * Fc * sigstride] staged post-filter signal for stage C (channel-major per packet)
    CbSigRange *range;   // [n * Fc]
    int kmax;
    int xstride;         // int16 per packet
    int sigstride;       // int32 per packet = cap48 * 2
    int Fc;              // packets per stream in this chunk buffer
};

// Stage A — parse + PVQ, one THREAD per run of R consecutive packets of one stream.  Frames are independent given the
// fold seed (= final range of the previous frame), which each thread recovers for the start of its run by re-parsing the
// packet before it; inside the run the seed chains naturally.  No decoder state is written here (st->rng is read once per
// launch for the very first packet of a stream).
__global__ void __launch_bounds__(CB_PARSE_THREADS, CB_PARSE_MINBLOCKS)
parse_kernel(const CbCallCtx *call_ctx, const uint8_t *data, const int64_t *offs, const int32_t *lens, int n, int F,
             int f0, int f1, int call_f0, int R, int cap, int decode_fec, IrView ir) {
    const int runs = (f1 - f0 + R - 1) / R;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * runs) return;
    const int s = t / runs, r = t - s * runs;
    // Thread-local working set (5.6 KB of local memory: lane-interleaved, write-back in L1).  As per-thread rows of a global
    // array the same data made every 2-byte store a 32-byte write-through to L2: 251 GB of L1->L2 writes per 2.4 GB of output,
    // the L1->crossbar request path 52 % busy (profiles/r1_dec_v4_parse_kernel); local: parse 186 -> 114 ms per chunk.
    ParseScratch ps;
    const int first = f0 + r * R;
    const int last = first + R < f1 ? first + R : f1;
    opus_parse_run(call_ctx[s], data, offs + (size_t)s * F, lens + (size_t)s * F, call_f0, first, last, cap, decode_fec, ir.kmax, ir.xstride,
                   ir.pk + (size_t)s * ir.Fc, ir.fr + (size_t)s * ir.Fc * ir.kmax, ir.X + (size_t)s * ir.Fc * ir.xstride, f0, ps);
}

// Snapshot of what stage A needs of every stream's state, taken once per call before any stage runs (see CbCallCtx).
__global__ void call_ctx_kernel(const CbDecState *pool, const int *slots, CbCallCtx *out, int n) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < n) call_ctx_from_state(out[s], pool + slots[s]);
}

// Stage B — synthesis, one warp per stream, packets f0..f1 in order.  PCM row of packet (s,f) starts at
// pcm[(s*pcm_F + (f-pcm_f0)) * row]: row = cap * channels for a call of uniform channel count, cap * 2 when mono and stereo
// streams share one staging layout (multistream calls).
__global__ void __launch_bounds__(CB_WPB * 32, CB_SYNTH_MINBLOCKS)
synth_kernel(CbDecState *pool, const int *slots, IrView ir, int16_t *pcm, int n, int F, int f0, int f1, int pcm_F, int pcm_f0,
             int cap, int row, int *rets, PlcScratch *plc) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int s = blockIdx.x * CB_WPB + warp;
    if (s >= n) return;
    SynthScratch &S = *(reinterpret_cast<SynthScratch *>(smem) + warp);
    CbDecState *st = pool + slots[s];
    WarpTeam tm{lane};
    for (int f = f0; f < f1; f++) {
        const size_t slot = (size_t)s * ir.Fc + (f - f0);
        int16_t *out = pcm + ((size_t)s * pcm_F + f - pcm_f0) * row;
        int r = opus_synth_packet(tm, st, S, plc[s], ir.pk[slot], ir.fr + slot * ir.kmax, ir.X + slot * ir.xstride, out, cap,
                                  ir.sig + slot * ir.sigstride, ir.range + slot);
        if (lane == 0) rets[(size_t)s * F + f] = r;
        __syncwarp();
    }
}

// Stage C — de-emphasis + decode gain + PCM store, one THREAD per (stream, channel): the 1-pole IIR is order dependent
// along time but independent across streams and channels, so 32 of them fill a warp.  For the common stereo / 48 kHz case the
// two channel threads of a stream (an even/odd lane pair) swap halves of each 8-sample batch with shuffles so that each
// writes 16 contiguous bytes of interleaved PCM instead of eight scattered 2-byte stores.
__device__ __forceinline__ int deemph_pair_stereo(const int *x, int n, int16_t *pcm_lr, int c, int m, int gain, unsigned pairmask) {
    // x: this channel's samples (16-byte aligned), pcm_lr: interleaved L/R output (16-byte aligned), n % 8 == 0
    for (int j = 0; j < n; j += 8) {
        const int4 a = *reinterpret_cast<const int4 *>(x + j);
        const int4 b = *reinterpret_cast<const int4 *>(x + j + 4);
        const int xs[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        unsigned w[4];
#pragma unroll
        for (int u = 0; u < 8; u++) {
            int t = wadd(xs[u], m);
            m = mul16_32_q15(kPreemphCoef0, t);
            int v = sig2word16(t);
            if (gain >= 0) { int g = mul16_32_p16(v, gain); v = g > 32767 ? 32767 : (g < -32767 ? -32767 : g); }
            if (u & 1) w[u >> 1] |= (unsigned)(v & 0xffff) << 16;
            else w[u >> 1] = (unsigned)(v & 0xffff);
        }
        // even lane (L) keeps samples 0..3 and needs R0..R3; odd lane (R) keeps samples 4..7 and needs L4..L7
        const unsigned o0 = __shfl_xor_sync(pairmask, c == 0 ? w[2] : w[0], 1);
        const unsigned o1 = __shfl_xor_sync(pairmask, c == 0 ? w[3] : w[1], 1);
        const unsigned l0 = c == 0 ? w[0] : o0, l1 = c == 0 ? w[1] : o1;   // two L samples per word
        const unsigned r0 = c == 0 ? o0 : w[2], r1 = c == 0 ? o1 : w[3];   // two R samples per word
        uint4 out;
        out.x = __byte_perm(l0, r0, 0x5410);   // L_k   | R_k   << 16
        out.y = __byte_perm(l0, r0, 0x7632);   // L_k+1 | R_k+1 << 16
        out.z = __byte_perm(l1, r1, 0x5410);
        out.w = __byte_perm(l1, r1, 0x7632);
        *reinterpret_cast<uint4 *>(pcm_lr + (j + (c == 0 ? 0 : 4)) * 2) = out;
    }
    return m;
}

__global__ void __launch_bounds__(128)
deemph_kernel(CbDecState *pool, const int *slots, IrView ir, int16_t *pcm, int n, int f0, int f1, int pcm_F, int pcm_f0, int cap, int row) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int s = t >> 1, c = t & 1;
    if (s >= n) return;
    CbDecState *st = pool + slots[s];
    const int channels = st->channels;
    if (c >= channels) return;
    const int ds = st->downsample;
    const int gain = st->decode_gain ? celt_exp2(s16(mul16_16_p15(21771, st->decode_gain))) : -1;   // QCONST16(6.48814081e-4f, 25); -1 = no gain stage (a very negative gain gives 0 = silence, opus_decoder.c:700-711)
    const unsigned pairmask = 3u << ((threadIdx.x & 31) & ~1);
    const bool paired = channels == 2 && ds == 1;
    int m = st->preemph_memD[c];
    for (int f = f0; f < f1; f++) {
        const size_t slot = (size_t)s * ir.Fc + (f - f0);
        int16_t *out = pcm + ((size_t)s * pcm_F + (f - pcm_f0)) * row;
        const CbSigRange rg = ir.range[slot];
        if (rg.end <= rg.begin) continue;
        const int *x = ir.sig + slot * ir.sigstride + c * (cap * ds) + rg.begin;
        const int cnt = rg.end - rg.begin;
        int16_t *y0 = out + (rg.begin / ds) * channels;
        // the two lanes of a stereo pair must take the same path (the paired one shuffles): x of channel 1 is offset by cap*ds
        // ints, so its alignment can differ from channel 0's — combine the per-lane predicates over the pair
        bool vec_ok = paired && (cnt & 7) == 0 && ((((uintptr_t)x) | ((uintptr_t)y0)) & 15) == 0;
        if (paired) vec_ok = __all_sync(pairmask, vec_ok);
        if (vec_ok)
            m = deemph_pair_stereo(x, cnt, y0, c, m, gain, pairmask);
        else
            m = deemphasis_channel(x, cnt, y0 + c, channels, ds, m, gain);
    }
    st->preemph_memD[c] = m;
}

// ---- multistream (DESIGN.md §3): a call over n multistream decoders of S streams is one pipeline call over the n*S embedded
// decoders, elementary decoder e = m*S + s.  ms_split_kernel turns the multistream packets into elementary ones before it,
// ms_gather_kernel turns each chunk's elementary PCM into multistream rows after it.

// End of the furthest packet of a device-resident span (the size of the split's scratch copy of the input).
__global__ void ms_extent_kernel(const int64_t *offs, const int32_t *lens, int N, unsigned long long *extent) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < N && lens[t] > 0) atomicMax(extent, (unsigned long long)(offs[t] + lens[t]));
}

// One thread per multistream packet (m,f): validation and undelimiting (ms_split_packet) into `blob`, a copy of `data` followed by
// the reject marker at `reject_off`; fills the elementary offsets / lengths [(m*S+s)*F + f] and the packet's own error code (0 = none).
__global__ void ms_split_kernel(const uint8_t *data, const int64_t *offs, const int32_t *lens, int n, int F, int S, int Fs, int frame_size,
                                uint8_t *blob, int64_t reject_off, int64_t *eoffs, int32_t *elens, int *ms_err) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t == 0) ms_write_reject_marker(blob + reject_off);   // read only by the stages after this kernel
    if (t >= n * F) return;
    const int m = t / F, f = t - m * F;
    const int len = lens[t];
    const int64_t off = len > 0 ? offs[t] : 0;
    const size_t e0 = (size_t)m * S * F + f;
    const int r = ms_split_packet(data + off, len, S, Fs, frame_size, blob + off, off, eoffs + e0, elens + e0, (size_t)F, reject_off);
    ms_err[t] = r < 0 ? r : 0;
}

// One block per multistream packet of the chunk [f0, f1): output channel c of sample i is stream channel mapping[c] of the
// elementary rows (coupled stream s: channels 2s / 2s+1, interleaved in a stereo row; mono stream s: channel coupled + s), a
// channel mapped to 255 and the row tail past the packet's samples are zero.  ret = the packet's split error, else the first
// elementary error in stream order, else the sample count; a packet with an error gets an all-zero row.
// epcm: elementary row (e, f) at ((e * e_F) + f - f0) * erow; out: row (m, f) at ((m * out_F) + f - out_f0) * frame_size * channels.
__global__ void __launch_bounds__(256)
ms_gather_kernel(const int16_t *epcm, int e_F, int erow, const int *erets, const int *ms_err, const uint8_t *mapping, int16_t *out,
                 int out_F, int out_f0, int F, int f0, int f1, int S, int coupled, int channels, int frame_size, int *ret) {
    __shared__ int s_ret;
    __shared__ uint8_t s_map[256];
    const int nf = f1 - f0;
    const int m = blockIdx.x / nf, f = f0 + (blockIdx.x - m * nf);
    for (int c = threadIdx.x; c < channels; c += blockDim.x) s_map[c] = mapping[(size_t)m * channels + c];
    if (threadIdx.x == 0) {
        int r = ms_err[(size_t)m * F + f];
        if (r == 0) {
            r = erets[((size_t)m * S) * F + f];
            for (int s = 1; s < S && r >= 0; s++) {
                const int e = erets[((size_t)m * S + s) * F + f];
                if (e < 0) r = e;
            }
        }
        s_ret = r;
        ret[(size_t)m * F + f] = r;
    }
    __syncthreads();
    const int r = s_ret > 0 ? s_ret : 0;
    const int16_t *ebase = epcm + ((size_t)m * S * e_F + (f - f0)) * erow;
    const size_t estride = (size_t)e_F * erow;   // from stream s to s+1 of the same multistream decoder
    int16_t *o = out + ((size_t)m * out_F + (f - out_f0)) * frame_size * channels;
    for (int i = threadIdx.x; i < frame_size; i += blockDim.x) {
        for (int c = 0; c < channels; c++) {
            const int k = s_map[c];
            int16_t v = 0;
            if (i < r && k != 255) {
                if (k < 2 * coupled) v = ebase[(size_t)(k >> 1) * estride + 2 * i + (k & 1)];
                else v = ebase[(size_t)(k - coupled) * estride + i];
            }
            o[(size_t)i * channels + c] = v;
        }
    }
}

// state staging <-> pool
__global__ void scatter_states_kernel(CbDecState *pool, const int *slots, const CbDecState *stage, int n) {
    const int words = sizeof(CbDecState) / 4;
    for (int k = blockIdx.x; k < n; k += gridDim.x) {
        const int *src = reinterpret_cast<const int *>(stage + k);
        int *dst = reinterpret_cast<int *>(pool + slots[k]);
        for (int i = threadIdx.x; i < words; i += blockDim.x) dst[i] = src[i];
    }
}
__global__ void gather_states_kernel(const CbDecState *pool, const int *slots, CbDecState *stage, int n) {
    const int words = sizeof(CbDecState) / 4;
    for (int k = blockIdx.x; k < n; k += gridDim.x) {
        const int *src = reinterpret_cast<const int *>(pool + slots[k]);
        int *dst = reinterpret_cast<int *>(stage + k);
        for (int i = threadIdx.x; i < words; i += blockDim.x) dst[i] = src[i];
    }
}

// ------------------------------------------------------------------------------------------------
// Runtime context
// ------------------------------------------------------------------------------------------------
namespace {

typedef CbSlotInfo SlotInfo;
typedef CbDevBuf DevBuf;
typedef CbPinBuf PinBuf;

struct Ctx {
    std::mutex mu;
    bool tried = false, ok = false;
    int device = 0;
    cudaStream_t stream = nullptr, copy_stream = nullptr, parse_stream = nullptr, synth_stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_chunk[2] = {nullptr, nullptr}, ev_copy[2] = {nullptr, nullptr};
    cudaEvent_t ev_parse[2] = {nullptr, nullptr}, ev_synth[2] = {nullptr, nullptr}, ev_deemph[2] = {nullptr, nullptr}, ev_call = nullptr;
    CbDecState *pool = nullptr;
    int pool_cap = 0;
    std::vector<SlotInfo> reg;
    std::vector<int> free_slots;
    DevBuf d_slots, d_data, d_offs, d_lens, d_pcm[2], d_rets, d_stage;
    DevBuf d_irpk[2], d_irfr[2], d_irx[2], d_sig[2], d_range[2], d_plc, d_callctx;
    // multistream calls: the split's copy of the input, elementary offsets / lengths / returns, per-packet split errors, channel
    // mappings, elementary PCM of a chunk (double-buffered), the input extent of a device-resident span
    DevBuf d_blob, d_eoffs, d_elens, d_erets, d_mserr, d_map, d_epcm[2], d_extent;
    cudaEvent_t ev_gather[2] = {nullptr, nullptr};
    size_t ir_budget = (size_t)16 << 30;  // bytes of IR + staging per chunk buffer (env CB200_IR_MB)
    // Host-buffer calls copy each chunk's PCM out while the next chunk decodes; the last chunk's copy overlaps nothing, so
    // they run on smaller chunks (measured: e2e 108 K -> 126 K x realtime; the device-resident path keeps the large ones)
    size_t ir_budget_host = (size_t)6 << 30;   // env CB200_IR_HOST_MB (4 / 6 / 8 GB measured: 119 K / 126 K / 116 K)
    int run_len = 3;                      // packets per stage-A thread (env CB200_RUN)
    int parse_wave_blocks = 0;            // blocks of parse_kernel resident at once on this device (occupancy x SMs)
    int max_waves = 1;                    // stage-A waves per chunk (env CB200_WAVES; 0: what the IR budget allows).  Measured at 4,096 streams x 60 s: 1 wave (108-frame chunks) 157.7 K x, 2 waves 147.4 K x, 3 (the 16 GB budget) 145.4 K x: more, shorter chunks pipeline the three stages better
    PinBuf h_stage, h_slots, h_misc;
    long long launches = 0;
    float last_ms = 0.f;
    // per-stage timing: one event pair per launch, folded into the totals at synchronize time
    struct Timed { cudaEvent_t a, b; int stage; };
    std::vector<Timed> timed;
    std::vector<cudaEvent_t> ev_pool;
    double stage_ms[5] = {0, 0, 0, 0, 0};   // parse, synth, de-emphasis, multistream split, multistream gather
    long long stage_launches[5] = {0, 0, 0, 0, 0};
    int smem_per_block = 0;
    // slots of this device's pool whose owners moved to another device: released by the next call here (see release_elsewhere)
    std::mutex deferred_mu;
    std::vector<std::pair<int, const void *>> deferred;
};
// One context per device; a thread works on the device it selected with opus_b200_init (host_runtime.h).
Ctx g_ctxs[kCbMaxDevices];
thread_local int tl_device = -1;
int g_default_device = -1;
inline int cur_device() {
    const int d = tl_device >= 0 ? tl_device : g_default_device;
    return d < 0 || d >= kCbMaxDevices ? 0 : d;
}
#define g (g_ctxs[cur_device()])

enum { kStageStates = 4096 };   // states per upload / download slice: one copy, one kernel, one synchronisation for a whole batch

void release_slot_locked(OpusDecoder *d);
bool ctx_init_locked() {
    if (g.tried) {
        if (g.ok) {
            cudaSetDevice(g.device);
            if (!g.deferred.empty()) {
                std::lock_guard<std::mutex> lk(g.deferred_mu);
                for (auto &pr : g.deferred)
                    if (pr.first >= 0 && pr.first < g.pool_cap && g.reg[pr.first].owner == pr.second) {
                        g.reg[pr.first].owner = nullptr;
                        g.reg[pr.first].gen++;
                        g.free_slots.push_back(pr.first);
                    }
                g.deferred.clear();
            }
        }
        return g.ok;
    }
    g.tried = true;
    g.device = cur_device();
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
        fprintf(stderr, "concentus_b200: no CUDA device available — this library has no CPU path\n");
        return false;
    }
    if (g.device >= ndev) return false;
    if (cudaSetDevice(g.device) != cudaSuccess) return false;
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    // Measured on B200: giving stages B/C priority interleaves their blocks into the stage A grid and is ~13 % SLOWER
    // (cache interference); plain FIFO between the streams is the default, CB200_PRIO=1 re-enables the experiment.
    if (!getenv("CB200_PRIO")) prio_hi = prio_lo;
    if (cudaStreamCreateWithPriority(&g.stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess) return false;
    if (cudaStreamCreateWithPriority(&g.copy_stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess) return false;
    if (cudaStreamCreateWithPriority(&g.parse_stream, cudaStreamNonBlocking, prio_lo) != cudaSuccess) return false;
    if (cudaStreamCreateWithPriority(&g.synth_stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess) return false;
    cudaEventCreate(&g.ev0);
    cudaEventCreate(&g.ev1);
    for (int i = 0; i < 2; i++) {
        cudaEventCreateWithFlags(&g.ev_chunk[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&g.ev_copy[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&g.ev_parse[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&g.ev_synth[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&g.ev_deemph[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&g.ev_gather[i], cudaEventDisableTiming);
    }
    cudaEventCreateWithFlags(&g.ev_call, cudaEventDisableTiming);
    if (const char *e = getenv("CB200_IR_MB")) g.ir_budget = (size_t)atol(e) << 20;
    if (const char *e = getenv("CB200_IR_HOST_MB")) g.ir_budget_host = (size_t)atol(e) << 20;
    if (const char *e = getenv("CB200_RUN")) g.run_len = atoi(e) > 0 ? atoi(e) : 5;
    if (const char *e = getenv("CB200_WAVES")) g.max_waves = atoi(e);
    {
        int per_sm = 0, dev = 0, sms = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, parse_kernel, CB_PARSE_THREADS, 0) == cudaSuccess)
            g.parse_wave_blocks = per_sm * sms;
        if (getenv("CB200_NO_WAVE_SIZING")) g.parse_wave_blocks = 0;
    }
    {
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && g.ir_budget > free_b / 10) g.ir_budget = free_b / 10;
    }
    g.smem_per_block = (int)(CB_WPB * sizeof(SynthScratch));
    cudaFuncSetAttribute(synth_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, g.smem_per_block);
    cudaFuncSetAttribute(parse_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 0);   // stage A wants L1, not shared
    if (!g.h_stage.reserve(sizeof(CbDecState) * 64)) return false;
    if (!g.d_stage.reserve(sizeof(CbDecState) * 64)) return false;
    g.ok = (cudaGetLastError() == cudaSuccess);
    return g.ok;
}

bool pool_reserve_locked(int need_total) {
    if (need_total <= g.pool_cap) return true;
    int ncap = g.pool_cap ? g.pool_cap : 64;
    while (ncap < need_total) ncap *= 2;
    CbDecState *np = nullptr;
    if (cudaMalloc(&np, sizeof(CbDecState) * (size_t)ncap) != cudaSuccess) return false;
    if (g.pool) {
        cudaMemcpyAsync(np, g.pool, sizeof(CbDecState) * (size_t)g.pool_cap, cudaMemcpyDeviceToDevice, g.stream);
        cudaStreamSynchronize(g.stream);
        cudaFree(g.pool);
    }
    for (int i = ncap - 1; i >= g.pool_cap; i--) g.free_slots.push_back(i);
    g.reg.resize(ncap, SlotInfo{nullptr, 0});
    g.pool = np;
    g.pool_cap = ncap;
    return true;
}

inline bool resident(const OpusDecoder *d) {
    return d->device == g.device && d->slot >= 0 && d->slot < g.pool_cap && g.reg[d->slot].owner == d && g.reg[d->slot].gen == d->gen;
}
// the block's slot lives in another device's pool: that device's next call gives it back
void release_elsewhere(OpusDecoder *d) {
    if (d->slot >= 0 && d->device >= 0 && d->device < kCbMaxDevices && d->device != g.device) {
        Ctx &o = g_ctxs[d->device];
        std::lock_guard<std::mutex> lk(o.deferred_mu);
        o.deferred.emplace_back(d->slot, (const void *)d);
        d->slot = -1;
    }
}

// Bring the host copy of `d` up to date (download from its slot when the slot holds the newer state).
int make_host_current_locked(OpusDecoder *d) {
    if (d->host_current) return OPUS_OK;
    // stale host block: the state it refers to must still be in its slot with the same generation
    // (this also covers a block that was memcpy'd while its original was device-resident).  A state resident on ANOTHER device
    // has to be synchronised by a thread of that device first (opus_decoder_sync): OPUS_INVALID_STATE here.
    if (d->device != g.device || d->slot < 0 || d->slot >= g.pool_cap || g.reg[d->slot].gen != d->gen) return OPUS_INVALID_STATE;
    if (cudaMemcpyAsync(&d->st, g.pool + d->slot, sizeof(CbDecState), cudaMemcpyDeviceToHost, g.stream) != cudaSuccess)
        return OPUS_INTERNAL_ERROR;
    if (cudaStreamSynchronize(g.stream) != cudaSuccess) return OPUS_INTERNAL_ERROR;
    d->host_current = 1;
    return OPUS_OK;
}

void release_slot_locked(OpusDecoder *d) {
    release_elsewhere(d);
    if (d->slot >= 0 && d->slot < g.pool_cap && g.reg[d->slot].owner == d) {
        g.reg[d->slot].owner = nullptr;
        g.reg[d->slot].gen++;
        g.free_slots.push_back(d->slot);
    }
    d->slot = -1;
}

// Make every state resident in the pool; fills h_slots[0..n).  Uploads go through a pinned staging buffer.
int make_resident_locked(OpusDecoder **st, int n, int *h_slots) {
    int need_new = 0;
    for (int i = 0; i < n; i++) {
        OpusDecoder *d = st[i];
        if (!d || d->magic != kDecMagic) return OPUS_BAD_ARG;
        if (!resident(d)) need_new++;
    }
    // the same state twice in one batch would race two warps on it
    if (n > 1) {
        std::unordered_set<const void *> seen;
        seen.reserve((size_t)n * 2);
        for (int i = 0; i < n; i++)
            if (!seen.insert(st[i]).second) return OPUS_BAD_ARG;
    }
    int in_use = g.pool_cap - (int)g.free_slots.size();
    if (!pool_reserve_locked(in_use + need_new)) return OPUS_ALLOC_FAIL;
    std::vector<int> up_idx;
    for (int i = 0; i < n; i++) {
        OpusDecoder *d = st[i];
        if (resident(d)) {
            if (d->host_current) up_idx.push_back(i);   // host block is authoritative (e.g. after a ctl): refresh slot
        } else {
            if (!d->host_current) {
                int rc = make_host_current_locked(d);
                if (rc != OPUS_OK) return rc;
            }
            release_elsewhere(d);
            d->slot = g.free_slots.back();
            g.free_slots.pop_back();
            d->device = g.device;
            g.reg[d->slot].owner = d;
            d->gen = ++g.reg[d->slot].gen;
            up_idx.push_back(i);
        }
        h_slots[i] = d->slot;
    }
    {
        const size_t slice = up_idx.size() < (size_t)kStageStates ? up_idx.size() : (size_t)kStageStates;
        if (slice > 0 && (!g.h_stage.reserve(sizeof(CbDecState) * slice) || !g.d_stage.reserve(sizeof(CbDecState) * slice))) return OPUS_ALLOC_FAIL;
    }
    CbDecState *hs = (CbDecState *)g.h_stage.p;
    for (size_t base = 0; base < up_idx.size(); base += kStageStates) {
        int cnt = (int)((up_idx.size() - base) < (size_t)kStageStates ? (up_idx.size() - base) : kStageStates);
        std::vector<int> sl(cnt);
        for (int k = 0; k < cnt; k++) {
            OpusDecoder *d = st[up_idx[base + k]];
            memcpy(&hs[k], &d->st, sizeof(CbDecState));
            sl[k] = d->slot;
        }
        if (!g.d_slots.reserve(sizeof(int) * (size_t)(n > kStageStates ? n : kStageStates))) return OPUS_ALLOC_FAIL;
        cudaMemcpyAsync(g.d_stage.p, hs, sizeof(CbDecState) * (size_t)cnt, cudaMemcpyHostToDevice, g.stream);
        cudaMemcpyAsync(g.d_slots.p, sl.data(), sizeof(int) * (size_t)cnt, cudaMemcpyHostToDevice, g.stream);
        scatter_states_kernel<<<cnt < 2048 ? cnt : 2048, 256, 0, g.stream>>>(g.pool, (const int *)g.d_slots.p, (const CbDecState *)g.d_stage.p, cnt);
        if (cudaStreamSynchronize(g.stream) != cudaSuccess) return OPUS_INTERNAL_ERROR;
    }
    return OPUS_OK;
}

// After a launch: the slot now holds a newer state than the host block.
void mark_device_newer_locked(OpusDecoder **st, int n) {
    for (int i = 0; i < n; i++) {
        OpusDecoder *d = st[i];
        d->gen = ++g.reg[d->slot].gen;
        d->host_current = 0;
    }
}

int sync_states_locked(OpusDecoder **st, int n, bool release) {
    std::vector<int> idx;
    for (int i = 0; i < n; i++) {
        OpusDecoder *d = st[i];
        if (!d || d->magic != kDecMagic) return OPUS_BAD_ARG;
        if (!d->host_current) {
            if (!resident(d)) {
                int rc = make_host_current_locked(d);
                if (rc != OPUS_OK) return rc;
            } else {
                idx.push_back(i);
            }
        }
    }
    {
        const size_t slice = idx.size() < (size_t)kStageStates ? idx.size() : (size_t)kStageStates;
        if (slice > 0 && (!g.h_stage.reserve(sizeof(CbDecState) * slice) || !g.d_stage.reserve(sizeof(CbDecState) * slice))) return OPUS_ALLOC_FAIL;
    }
    CbDecState *hs = (CbDecState *)g.h_stage.p;
    for (size_t base = 0; base < idx.size(); base += kStageStates) {
        int cnt = (int)((idx.size() - base) < (size_t)kStageStates ? (idx.size() - base) : kStageStates);
        std::vector<int> sl(cnt);
        for (int k = 0; k < cnt; k++) sl[k] = st[idx[base + k]]->slot;
        if (!g.d_slots.reserve(sizeof(int) * (size_t)cnt)) return OPUS_ALLOC_FAIL;
        cudaMemcpyAsync(g.d_slots.p, sl.data(), sizeof(int) * (size_t)cnt, cudaMemcpyHostToDevice, g.stream);
        gather_states_kernel<<<cnt < 2048 ? cnt : 2048, 256, 0, g.stream>>>(g.pool, (const int *)g.d_slots.p, (CbDecState *)g.d_stage.p, cnt);
        cudaMemcpyAsync(hs, g.d_stage.p, sizeof(CbDecState) * (size_t)cnt, cudaMemcpyDeviceToHost, g.stream);
        if (cudaStreamSynchronize(g.stream) != cudaSuccess) return OPUS_INTERNAL_ERROR;
        for (int k = 0; k < cnt; k++) {
            OpusDecoder *d = st[idx[base + k]];
            memcpy(&d->st, &hs[k], sizeof(CbDecState));
            d->host_current = 1;
        }
    }
    if (release)
        for (int i = 0; i < n; i++) release_slot_locked(st[i]);
    return OPUS_OK;
}

cudaEvent_t timing_event() {
    if (!g.ev_pool.empty()) { cudaEvent_t e = g.ev_pool.back(); g.ev_pool.pop_back(); return e; }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}
void timing_begin(int stage, cudaStream_t s) {
    Ctx::Timed t{timing_event(), timing_event(), stage};
    cudaEventRecord(t.a, s);
    g.timed.push_back(t);
}
void timing_end(cudaStream_t s) { cudaEventRecord(g.timed.back().b, s); }
void timing_fold() {   // call only when all streams are idle
    for (auto &t : g.timed) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, t.a, t.b) == cudaSuccess) { g.stage_ms[t.stage] += ms; g.stage_launches[t.stage]++; }
        g.ev_pool.push_back(t.a);
        g.ev_pool.push_back(t.b);
    }
    g.timed.clear();
}

// Geometry of one call: chunking of the time axis and the IR buffers behind it.
struct Plan {
    int n, F, cap, fec, kmax, xstride, sigstride, Fc, nchunks, R;
};

bool plan_call(Plan &pl, int n, int F, int cap, int fec, int Fs, bool host_io) {
    pl.n = n; pl.F = F; pl.cap = cap; pl.fec = fec;
    int k = cap / (Fs / 400);
    pl.kmax = k < 1 ? 1 : (k > 48 ? 48 : k);
    pl.xstride = (cap * (48000 / Fs) * 2 + 7) & ~7;   // stage A stores bands with up to 16-byte vectors (store_band): every packet's spectrum must start 16-byte aligned
    pl.sigstride = cap * (48000 / Fs) * 2;
    pl.R = g.run_len;
    const size_t per_packet = sizeof(CbPacketIR) + (size_t)pl.kmax * sizeof(CbFrameIR) + (size_t)pl.xstride * sizeof(int16_t) +
                              (size_t)pl.sigstride * sizeof(int) + sizeof(CbSigRange);
    size_t budget = host_io && g.ir_budget_host < g.ir_budget ? g.ir_budget_host : g.ir_budget;
    size_t fc = budget / (per_packet * (size_t)n);
    if (fc < 1) fc = 1;
    if (fc > (size_t)F) fc = (size_t)F;
    if (fc > (size_t)pl.R) fc -= fc % pl.R;
    // Stage A is a latency-bound kernel of equal-cost threads: its blocks run in waves of `parse_wave_blocks`, and a chunk a few
    // blocks over a whole number of waves pays for another wave (measured: 114-frame chunks of 4,096 streams = 1,216 blocks on
    // 1,184 slots decode at 140 K x, 90-frame chunks at 149 K x).  So a chunk holds whole waves: k * floor(W * threads / n) runs.
    if (g.parse_wave_blocks > 0) {
        const size_t runs_per_wave = (size_t)g.parse_wave_blocks * CB_PARSE_THREADS / (size_t)n;
        if (runs_per_wave >= 1) {
            size_t k = fc / (runs_per_wave * pl.R);                       // whole waves the IR budget allows
            if (g.max_waves > 0) {
                // ... of which `max_waves` are used, but never chunks shorter than ~96 packets (very large batches: a wave of
                // 65,536 streams is 6 packets, and stages B / C pay per launch)
                size_t want = (size_t)g.max_waves, floor_k = (96 + runs_per_wave * pl.R - 1) / (runs_per_wave * pl.R);
                if (want < floor_k) want = floor_k;
                if (k > want) k = want;
            }
            if (k >= 1) fc = k * runs_per_wave * pl.R;
        }
    }
    // equal chunks (a multiple of the run length) instead of full ones plus a remnant
    const size_t nch = ((size_t)F + fc - 1) / fc;
    size_t eq = ((size_t)F + nch - 1) / nch;
    eq = (eq + pl.R - 1) / pl.R * pl.R;
    if (eq < fc) fc = eq;
    pl.Fc = (int)fc;
    pl.nchunks = (F + pl.Fc - 1) / pl.Fc;
    const int nb = pl.nchunks > 1 ? 2 : 1;
    const size_t slots = (size_t)n * pl.Fc;
    for (int b = 0; b < nb; b++) {
        if (!g.d_irpk[b].reserve(slots * sizeof(CbPacketIR)) || !g.d_irfr[b].reserve(slots * pl.kmax * sizeof(CbFrameIR)) ||
            !g.d_irx[b].reserve(slots * pl.xstride * sizeof(int16_t)) || !g.d_sig[b].reserve(slots * pl.sigstride * sizeof(int)) ||
            !g.d_range[b].reserve(slots * sizeof(CbSigRange)))
            return false;
    }
    if (!g.d_callctx.reserve((size_t)n * sizeof(CbCallCtx))) return false;
    return g.d_plc.reserve((size_t)n * sizeof(PlcScratch));   // concealment scratch, one per stream (lost frames only)
}

IrView ir_view(const Plan &pl, int b) {
    IrView v;
    v.pk = (CbPacketIR *)g.d_irpk[b].p; v.fr = (CbFrameIR *)g.d_irfr[b].p; v.X = (int16_t *)g.d_irx[b].p;
    v.sig = (int *)g.d_sig[b].p; v.range = (CbSigRange *)g.d_range[b].p;
    v.kmax = pl.kmax; v.xstride = pl.xstride; v.sigstride = pl.sigstride; v.Fc = pl.Fc;
    return v;
}

// Enqueue stage A for chunk c on the parse stream and stage B on the main stream.  PCM goes to pcm_dst laid out with
// pcm_F packets per stream starting at packet pcm_f0, `row` int16 per packet (the caller decides: whole-call buffer or a chunk
// buffer).
void enqueue_chunk(const Plan &pl, int c, const int *d_slots, const uint8_t *d_data, const int64_t *d_offs, const int32_t *d_lens,
                   int16_t *pcm_dst, int pcm_F, int pcm_f0, int row, int *d_rets, cudaEvent_t pcm_free = nullptr) {
    const int b = c & 1;
    const int f0 = c * pl.Fc, f1 = (f0 + pl.Fc < pl.F) ? f0 + pl.Fc : pl.F;
    const int runs = (f1 - f0 + pl.R - 1) / pl.R;
    const long long threads = (long long)pl.n * runs;
    IrView v = ir_view(pl, b);
    // stage A(c) may start once stage B(c-2) has drained IR buffer b, and (first chunk) once earlier calls are done
    if (c == 0) {
        cudaStreamWaitEvent(g.parse_stream, g.ev_call, 0);
        cudaStreamWaitEvent(g.synth_stream, g.ev_call, 0);
    }
    if (c >= 2) cudaStreamWaitEvent(g.parse_stream, g.ev_synth[b], 0);
    timing_begin(0, g.parse_stream);
    parse_kernel<<<(unsigned)((threads + CB_PARSE_THREADS - 1) / CB_PARSE_THREADS), CB_PARSE_THREADS, 0, g.parse_stream>>>(
        (const CbCallCtx *)g.d_callctx.p, d_data, d_offs, d_lens, pl.n, pl.F, f0, f1, 0, pl.R, pl.cap, pl.fec, v);
    timing_end(g.parse_stream);
    cudaEventRecord(g.ev_parse[b], g.parse_stream);
    // stage B(c): after A(c); its staging buffer b must have been drained by C(c-2)
    cudaStreamWaitEvent(g.synth_stream, g.ev_parse[b], 0);
    if (c >= 2) cudaStreamWaitEvent(g.synth_stream, g.ev_deemph[b], 0);
    if (pcm_free) cudaStreamWaitEvent(g.synth_stream, pcm_free, 0);   // stage B writes PCM too (leading zero frames)
    timing_begin(1, g.synth_stream);
    synth_kernel<<<(pl.n + CB_WPB - 1) / CB_WPB, CB_WPB * 32, g.smem_per_block, g.synth_stream>>>(g.pool, d_slots, v, pcm_dst, pl.n, pl.F, f0,
                                                                                                  f1, pcm_F, pcm_f0, pl.cap, row, d_rets, (PlcScratch *)g.d_plc.p);
    timing_end(g.synth_stream);
    cudaEventRecord(g.ev_synth[b], g.synth_stream);
    // stage C(c) on the main stream (the one the caller synchronises / times)
    cudaStreamWaitEvent(g.stream, g.ev_synth[b], 0);
    timing_begin(2, g.stream);
    deemph_kernel<<<(2 * pl.n + 127) / 128, 128, 0, g.stream>>>(g.pool, d_slots, v, pcm_dst, pl.n, f0, f1, pcm_F, pcm_f0, pl.cap, row);
    timing_end(g.stream);
    cudaEventRecord(g.ev_deemph[b], g.stream);
    g.launches += 3;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// C ABI — runtime
// ------------------------------------------------------------------------------------------------
extern "C" {

// Select the device the CALLING THREAD codes on (and initialise its context).  The first call of the process also sets the device
// of threads that never call this.
int opus_b200_init(int device) {
    if (device < 0 || device >= kCbMaxDevices) return OPUS_BAD_ARG;
    tl_device = device;
    if (g_default_device < 0) g_default_device = device;
    std::lock_guard<std::mutex> lk(g.mu);
    return ctx_init_locked() ? OPUS_OK : OPUS_INTERNAL_ERROR;
}
int opus_b200_current_device(void) { return cur_device(); }
// The device this process codes on (initialises the runtime); -1 when CUDA is unusable.  Used by the encoder half
// (opus_enc_capi.cu) so both halves share one device selection.
int opus_b200_device_index(void) {
    std::lock_guard<std::mutex> lk(g.mu);
    return ctx_init_locked() ? g.device : -1;
}
int opus_b200_synchronize(void) {
    std::lock_guard<std::mutex> lk(g.mu);
    if (!ctx_init_locked()) return OPUS_INTERNAL_ERROR;
    if (cudaStreamSynchronize(g.stream) != cudaSuccess) return OPUS_INTERNAL_ERROR;
    if (cudaStreamSynchronize(g.copy_stream) != cudaSuccess) return OPUS_INTERNAL_ERROR;
    if (cudaStreamSynchronize(g.parse_stream) != cudaSuccess || cudaStreamSynchronize(g.synth_stream) != cudaSuccess) return OPUS_INTERNAL_ERROR;
    if (g.launches > 0) cudaEventElapsedTime(&g.last_ms, g.ev0, g.ev1);   // last call (events on g.stream)
    timing_fold();
    return OPUS_OK;
}
void *opus_b200_stream(void) {
    std::lock_guard<std::mutex> lk(g.mu);
    if (!ctx_init_locked()) return nullptr;
    return (void *)g.stream;
}
long long opus_b200_kernel_launches(void) { return g.launches; }
// Accumulated device time (ms, CUDA events around every launch on its own stream) and launch count per pipeline stage
// (0 = parse, 1 = synth, 2 = de-emphasis) since the last reset.  Folded in at synchronisation points.
int opus_b200_stage_times(double ms[3], long long launches[3], int reset) {
    std::lock_guard<std::mutex> lk(g.mu);
    for (int i = 0; i < 3; i++) {
        if (ms) ms[i] = g.stage_ms[i];
        if (launches) launches[i] = g.stage_launches[i];
        if (reset) { g.stage_ms[i] = 0; g.stage_launches[i] = 0; }
    }
    return OPUS_OK;
}
// The same for the two multistream stages (0 = split, 1 = gather).
int opus_b200_ms_stage_times(double ms[2], long long launches[2], int reset) {
    std::lock_guard<std::mutex> lk(g.mu);
    for (int i = 0; i < 2; i++) {
        if (ms) ms[i] = g.stage_ms[3 + i];
        if (launches) launches[i] = g.stage_launches[3 + i];
        if (reset) { g.stage_ms[3 + i] = 0; g.stage_launches[3 + i] = 0; }
    }
    return OPUS_OK;
}
float opus_b200_last_kernel_ms(void) {
    std::lock_guard<std::mutex> lk(g.mu);
    return g.last_ms;
}

const char *opus_strerror(int error) {
    static const char *const s[8] = {"success", "invalid argument", "buffer too small", "internal error", "corrupted stream",
                                     "request not implemented", "invalid state", "memory allocation failed"};
    if (error > 0 || error < -7) return "unknown error";
    return s[-error];
}
const char *opus_get_version_string(void) { return "libopus 1.1.2-fixed (concentus_b200, sm_100a CELT engine)"; }

// ---- packet helpers (host) ----
int opus_packet_parse(const unsigned char *data, opus_int32 len, unsigned char *out_toc, const unsigned char *frames[48],
                      opus_int16 size[48], int *payload_offset) {
    if (size == nullptr || len < 0) return OPUS_BAD_ARG;
    int off = 0;
    int count = pkt_parse(data, len, 0, out_toc, size, &off, nullptr);
    if (count < 0) return count;
    if (payload_offset) *payload_offset = off;
    if (frames) {
        const unsigned char *p = data + off;
        for (int i = 0; i < count; i++) {
            frames[i] = p;
            p += size[i];
        }
    }
    return count;
}
int opus_packet_get_bandwidth(const unsigned char *data) { return pkt_bandwidth(data); }
int opus_packet_get_samples_per_frame(const unsigned char *data, opus_int32 Fs) { return pkt_samples_per_frame(data, Fs); }
int opus_packet_get_nb_channels(const unsigned char *data) { return pkt_nb_channels(data); }
int opus_packet_get_nb_frames(const unsigned char packet[], opus_int32 len) {
    if (len < 1) return OPUS_BAD_ARG;
    int count = packet[0] & 0x3;
    if (count == 0) return 1;
    if (count != 3) return 2;
    if (len < 2) return OPUS_INVALID_PACKET;
    return packet[1] & 0x3F;
}
int opus_packet_get_nb_samples(const unsigned char packet[], opus_int32 len, opus_int32 Fs) {
    int count = opus_packet_get_nb_frames(packet, len);
    if (count < 0) return count;
    int samples = count * pkt_samples_per_frame(packet, Fs);
    if (samples * 25 > Fs * 3) return OPUS_INVALID_PACKET;
    return samples;
}
int opus_decoder_get_nb_samples(const OpusDecoder *dec, const unsigned char packet[], opus_int32 len) {
    return opus_packet_get_nb_samples(packet, len, dec->st.Fs);
}

// ---- decoder lifecycle ----
int opus_decoder_get_size(int channels) {
    if (channels < 1 || channels > 2) return 0;
    return (int)sizeof(OpusDecoder);
}
int opus_decoder_init(OpusDecoder *st, opus_int32 Fs, int channels) {
    if ((Fs != 48000 && Fs != 24000 && Fs != 16000 && Fs != 12000 && Fs != 8000) || (channels != 1 && channels != 2))
        return OPUS_BAD_ARG;
    {   // re-initialising a live block in place (the reference's tests do): give its pool slot back first
        std::lock_guard<std::mutex> lk(g.mu);
        if (g.ok && st->magic == kDecMagic && st->slot >= 0) release_slot_locked(st);
    }
    memset(st, 0, sizeof(OpusDecoder));
    st->magic = kDecMagic;
    st->slot = -1;
    st->gen = 0;
    st->host_current = 1;
    st->device = -1;
    if (dec_state_init(&st->st, Fs, channels) != 0) return OPUS_BAD_ARG;
    return OPUS_OK;
}
OpusDecoder *opus_decoder_create(opus_int32 Fs, int channels, int *error) {
    if ((Fs != 48000 && Fs != 24000 && Fs != 16000 && Fs != 12000 && Fs != 8000) || (channels != 1 && channels != 2)) {
        if (error) *error = OPUS_BAD_ARG;
        return nullptr;
    }
    OpusDecoder *st = (OpusDecoder *)malloc(sizeof(OpusDecoder));
    if (!st) {
        if (error) *error = OPUS_ALLOC_FAIL;
        return nullptr;
    }
    int ret = opus_decoder_init(st, Fs, channels);
    if (error) *error = ret;
    if (ret != OPUS_OK) {
        free(st);
        st = nullptr;
    }
    return st;
}
void opus_decoder_destroy(OpusDecoder *st) {
    if (!st) return;
    {
        std::lock_guard<std::mutex> lk(g.mu);
        if (g.ok && st->magic == kDecMagic) release_slot_locked(st);
    }
    free(st);
}

int opus_decoder_ctl(OpusDecoder *st, int request, ...) {
    int ret = OPUS_OK;
    va_list ap;
    va_start(ap, request);
    // any ctl that reads or writes codec state needs the host block current
    {
        std::lock_guard<std::mutex> lk(g.mu);
        if (!st->host_current) {
            if (!ctx_init_locked()) { va_end(ap); return OPUS_INTERNAL_ERROR; }
            int rc = make_host_current_locked(st);
            if (rc != OPUS_OK) { va_end(ap); return rc; }
        }
    }
    CbDecState *s = &st->st;
    switch (request) {
    case OPUS_GET_BANDWIDTH_REQUEST: {
        opus_int32 *v = va_arg(ap, opus_int32 *);
        if (!v) { ret = OPUS_BAD_ARG; break; }
        *v = s->bandwidth;
    } break;
    case OPUS_GET_FINAL_RANGE_REQUEST: {
        opus_uint32 *v = va_arg(ap, opus_uint32 *);
        if (!v) { ret = OPUS_BAD_ARG; break; }
        *v = s->rangeFinal;
    } break;
    case OPUS_RESET_STATE: {
        std::lock_guard<std::mutex> lk(g.mu);
        dec_state_reset(s);
        // host block is now authoritative; a resident slot is refreshed on the next batch call
    } break;
    case OPUS_GET_SAMPLE_RATE_REQUEST: {
        opus_int32 *v = va_arg(ap, opus_int32 *);
        if (!v) { ret = OPUS_BAD_ARG; break; }
        *v = s->Fs;
    } break;
    case OPUS_GET_PITCH_REQUEST: {
        opus_int32 *v = va_arg(ap, opus_int32 *);
        if (!v) { ret = OPUS_BAD_ARG; break; }
        *v = s->prev_mode == CB_MODE_CELT_ONLY ? s->postfilter_period : 0;
    } break;
    case OPUS_GET_GAIN_REQUEST: {
        opus_int32 *v = va_arg(ap, opus_int32 *);
        if (!v) { ret = OPUS_BAD_ARG; break; }
        *v = s->decode_gain;
    } break;
    case OPUS_SET_GAIN_REQUEST: {
        opus_int32 v = va_arg(ap, opus_int32);
        if (v < -32768 || v > 32767) { ret = OPUS_BAD_ARG; break; }
        s->decode_gain = v;
    } break;
    case OPUS_GET_LAST_PACKET_DURATION_REQUEST: {
        opus_uint32 *v = va_arg(ap, opus_uint32 *);
        if (!v) { ret = OPUS_BAD_ARG; break; }
        *v = (opus_uint32)s->last_packet_duration;
    } break;
    default:
        ret = OPUS_UNIMPLEMENTED;
        break;
    }
    va_end(ap);
    return ret;
}

// ---- decode ----
int opus_decode_span_device(OpusDecoder **st, int n, int F, const unsigned char *d_data, const int64_t *d_offs,
                            const opus_int32 *d_len, opus_int16 *d_pcm, int frame_size, int *d_ret) {
    if (!st || n <= 0 || F <= 0 || frame_size <= 0) return OPUS_BAD_ARG;
    std::lock_guard<std::mutex> lk(g.mu);
    if (!ctx_init_locked()) return OPUS_INTERNAL_ERROR;
    // the IR / staging geometry of a call is sized from one (Fs, channels): every stream must share it
    for (int i = 0; i < n; i++) {
        if (!st[i] || st[i]->magic != kDecMagic) return OPUS_BAD_ARG;
        if (st[i]->st.channels != st[0]->st.channels || st[i]->st.Fs != st[0]->st.Fs) return OPUS_BAD_ARG;
    }
    if (!g.h_slots.reserve(sizeof(int) * (size_t)n)) return OPUS_ALLOC_FAIL;
    int *hsl = (int *)g.h_slots.p;
    int rc = make_resident_locked(st, n, hsl);
    if (rc != OPUS_OK) return rc;
    if (!g.d_slots.reserve(sizeof(int) * (size_t)n)) return OPUS_ALLOC_FAIL;
    Plan pl;
    if (!plan_call(pl, n, F, frame_size, 0, st[0]->st.Fs, false)) return OPUS_ALLOC_FAIL;
    cudaMemcpyAsync(g.d_slots.p, hsl, sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, g.stream);
    cudaEventRecord(g.ev0, g.stream);
    call_ctx_kernel<<<(n + 127) / 128, 128, 0, g.stream>>>(g.pool, (const int *)g.d_slots.p, (CbCallCtx *)g.d_callctx.p, n);
    g.launches++;
    cudaEventRecord(g.ev_call, g.stream);
    for (int c = 0; c < pl.nchunks; c++)
        enqueue_chunk(pl, c, (const int *)g.d_slots.p, d_data, d_offs, d_len, d_pcm, F, 0, frame_size * st[0]->st.channels, d_ret);
    cudaEventRecord(g.ev1, g.stream);
    mark_device_newer_locked(st, n);
    if (cudaGetLastError() != cudaSuccess) return OPUS_INTERNAL_ERROR;
    return OPUS_OK;
}

// Host-buffer span decode.  The packet bytes go up in one copy; the kernel then runs in time chunks whose
// PCM is copied back on a second stream while the next chunk decodes (double-buffered).
static int decode_span_host_locked(OpusDecoder **st, int n, int F, const unsigned char *data, int64_t data_bytes,
                                   const int64_t *offs, const opus_int32 *len, opus_int16 *pcm, int frame_size,
                                   int decode_fec, int *ret, bool keep_resident) {
    if (!ctx_init_locked()) return OPUS_INTERNAL_ERROR;
    if (!st[0] || st[0]->magic != kDecMagic) return OPUS_BAD_ARG;
    const int channels = st[0]->st.channels;
    for (int i = 0; i < n; i++) {
        if (!st[i] || st[i]->magic != kDecMagic) return OPUS_BAD_ARG;
        // the IR / staging geometry of a call is sized from one (Fs, channels): every stream must share it
        if (st[i]->st.channels != channels || st[i]->st.Fs != st[0]->st.Fs) return OPUS_BAD_ARG;
    }
    if (!g.h_slots.reserve(sizeof(int) * (size_t)n)) return OPUS_ALLOC_FAIL;
    int *hsl = (int *)g.h_slots.p;
    int rc = make_resident_locked(st, n, hsl);
    if (rc != OPUS_OK) return rc;
    const size_t NF = (size_t)n * F;
    if (!g.d_slots.reserve(sizeof(int) * (size_t)n) || !g.d_data.reserve((size_t)data_bytes + 16) ||
        !g.d_offs.reserve(sizeof(int64_t) * NF) || !g.d_lens.reserve(sizeof(int32_t) * NF) || !g.d_rets.reserve(sizeof(int) * NF))
        return OPUS_ALLOC_FAIL;
    // time chunking follows the IR plan; PCM of a chunk is copied back while the next chunk is decoded
    Plan pl;
    if (!plan_call(pl, n, F, frame_size, decode_fec, st[0]->st.Fs, true)) return OPUS_ALLOC_FAIL;
    const size_t row = (size_t)frame_size * channels * sizeof(int16_t);
    const int Fc = pl.Fc, nchunks = pl.nchunks;
    const size_t chunk_bytes = (size_t)n * Fc * row;
    if (!g.d_pcm[0].reserve(chunk_bytes) || (nchunks > 1 && !g.d_pcm[1].reserve(chunk_bytes))) return OPUS_ALLOC_FAIL;
    cudaMemcpyAsync(g.d_slots.p, hsl, sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, g.stream);
    if (data_bytes > 0) cudaMemcpyAsync(g.d_data.p, data, (size_t)data_bytes, cudaMemcpyHostToDevice, g.stream);
    cudaMemcpyAsync(g.d_offs.p, offs, sizeof(int64_t) * NF, cudaMemcpyHostToDevice, g.stream);
    cudaMemcpyAsync(g.d_lens.p, len, sizeof(int32_t) * NF, cudaMemcpyHostToDevice, g.stream);
    cudaEventRecord(g.ev0, g.stream);
    call_ctx_kernel<<<(n + 127) / 128, 128, 0, g.stream>>>(g.pool, (const int *)g.d_slots.p, (CbCallCtx *)g.d_callctx.p, n);
    g.launches++;
    cudaEventRecord(g.ev_call, g.stream);
    for (int c = 0; c < nchunks; c++) {
        const int b = c & 1;
        const int f0 = c * Fc, f1 = (f0 + Fc < F) ? f0 + Fc : F;
        if (c >= 2) cudaStreamWaitEvent(g.stream, g.ev_copy[b], 0);   // PCM buffer b drained?
        enqueue_chunk(pl, c, (const int *)g.d_slots.p, (const uint8_t *)g.d_data.p, (const int64_t *)g.d_offs.p,
                      (const int32_t *)g.d_lens.p, (int16_t *)g.d_pcm[b].p, Fc, f0, frame_size * channels, (int *)g.d_rets.p,
                      c >= 2 ? g.ev_copy[b] : nullptr);
        cudaEventRecord(g.ev_chunk[b], g.stream);
        cudaStreamWaitEvent(g.copy_stream, g.ev_chunk[b], 0);
        // rows of (f1-f0) packets per stream: device pitch Fc*row, host pitch F*row
        cudaMemcpy2DAsync((char *)pcm + (size_t)f0 * row, (size_t)F * row, g.d_pcm[b].p, (size_t)Fc * row, (size_t)(f1 - f0) * row,
                          (size_t)n, cudaMemcpyDeviceToHost, g.copy_stream);
        cudaEventRecord(g.ev_copy[b], g.copy_stream);
    }
    cudaEventRecord(g.ev1, g.stream);
    cudaMemcpyAsync(ret, g.d_rets.p, sizeof(int) * NF, cudaMemcpyDeviceToHost, g.stream);
    mark_device_newer_locked(st, n);
    if (cudaStreamSynchronize(g.stream) != cudaSuccess || cudaStreamSynchronize(g.copy_stream) != cudaSuccess ||
        cudaStreamSynchronize(g.parse_stream) != cudaSuccess || cudaStreamSynchronize(g.synth_stream) != cudaSuccess) {
        fprintf(stderr, "concentus_b200: CUDA failure in decode span: %s\n", cudaGetErrorString(cudaGetLastError()));
        return OPUS_INTERNAL_ERROR;
    }
    cudaEventElapsedTime(&g.last_ms, g.ev0, g.ev1);
    timing_fold();
    if (!keep_resident) return sync_states_locked(st, n, true);
    return OPUS_OK;
}

int opus_decode_span(OpusDecoder **st, int n, int F, const unsigned char *data, const int64_t *offs, const opus_int32 *len,
                     opus_int16 *pcm, int frame_size, int *ret) {
    if (!st || n <= 0 || F <= 0 || frame_size <= 0 || !offs || !len || !pcm || !ret) return OPUS_BAD_ARG;
    int64_t bytes = 0;
    const size_t NF = (size_t)n * F;
    for (size_t i = 0; i < NF; i++) {
        if (len[i] < 0 || offs[i] < 0) return OPUS_BAD_ARG;
        int64_t e = offs[i] + len[i];
        if (len[i] > 0 && e > bytes) bytes = e;
    }
    std::lock_guard<std::mutex> lk(g.mu);
    return decode_span_host_locked(st, n, F, data, bytes, offs, len, pcm, frame_size, 0, ret, true);
}

int opus_decode_batch(OpusDecoder **st, const unsigned char *const *data, const opus_int32 *len, opus_int16 *const *pcm,
                      int frame_size, int decode_fec, int *ret, int n) {
    if (!st || !len || !pcm || !ret || n <= 0) return OPUS_BAD_ARG;
    if (frame_size <= 0) {
        for (int i = 0; i < n; i++) ret[i] = OPUS_BAD_ARG;
        return OPUS_OK;
    }
    std::lock_guard<std::mutex> lk(g.mu);
    if (!ctx_init_locked()) return OPUS_INTERNAL_ERROR;
    // group by (Fs, channel count): the span kernels want a uniform PCM row size and one IR geometry per call
    static const int kRates[5] = {48000, 24000, 16000, 12000, 8000};
    for (int grp = 0; grp < 10; grp++) {
        const int pass = 1 + (grp & 1), rate = kRates[grp >> 1];
        std::vector<int> idx;
        for (int i = 0; i < n; i++)
            if (st[i] && st[i]->magic == kDecMagic && st[i]->st.channels == pass && st[i]->st.Fs == rate) idx.push_back(i);
        if (idx.empty()) continue;
        const int m = (int)idx.size();
        std::vector<OpusDecoder *> sts(m);
        std::vector<int64_t> offs(m);
        std::vector<int32_t> lens(m);
        std::vector<int> rets(m);
        int64_t total = 0;
        for (int k = 0; k < m; k++) {
            int i = idx[k];
            sts[k] = st[i];
            int l = (data && data[i]) ? len[i] : 0;
            if (len[i] < 0 && data && data[i]) l = -1;
            lens[k] = l;
            offs[k] = total;
            if (l > 0) total += l;
        }
        std::vector<unsigned char> blob((size_t)total + 1);
        for (int k = 0; k < m; k++)
            if (lens[k] > 0) memcpy(blob.data() + offs[k], data[idx[k]], (size_t)lens[k]);
        std::vector<int16_t> out((size_t)m * frame_size * pass);
        // negative len is a scalar-API argument error: report per stream, do not launch for it
        bool any_neg = false;
        for (int k = 0; k < m; k++) any_neg |= lens[k] < 0;
        if (any_neg) {
            for (int k = 0; k < m; k++) if (lens[k] < 0) { ret[idx[k]] = OPUS_BAD_ARG; lens[k] = 0; sts[k] = nullptr; }
            std::vector<OpusDecoder *> s2; std::vector<int> map2;
            std::vector<int64_t> o2; std::vector<int32_t> l2;
            for (int k = 0; k < m; k++) if (sts[k]) { s2.push_back(sts[k]); map2.push_back(idx[k]); o2.push_back(offs[k]); l2.push_back(lens[k]); }
            if (s2.empty()) continue;
            std::vector<int> r2(s2.size());
            int rc = decode_span_host_locked(s2.data(), (int)s2.size(), 1, blob.data(), total, o2.data(), l2.data(), out.data(),
                                             frame_size, decode_fec, r2.data(), true);
            if (rc != OPUS_OK) return rc;
            for (size_t k = 0; k < s2.size(); k++) {
                ret[map2[k]] = r2[k];
                if (r2[k] > 0) memcpy(pcm[map2[k]], out.data() + k * (size_t)frame_size * pass, (size_t)r2[k] * pass * sizeof(int16_t));
            }
            continue;
        }
        int rc = decode_span_host_locked(sts.data(), m, 1, blob.data(), total, offs.data(), lens.data(), out.data(), frame_size,
                                         decode_fec, rets.data(), true);
        if (rc != OPUS_OK) return rc;
        for (int k = 0; k < m; k++) {
            ret[idx[k]] = rets[k];
            if (rets[k] > 0) memcpy(pcm[idx[k]], out.data() + (size_t)k * frame_size * pass, (size_t)rets[k] * pass * sizeof(int16_t));
        }
    }
    for (int i = 0; i < n; i++)
        if (!st[i] || st[i]->magic != kDecMagic) ret[i] = OPUS_BAD_ARG;
    return OPUS_OK;
}

int opus_decoder_sync(OpusDecoder **st, int n) {
    if (!st || n <= 0) return OPUS_BAD_ARG;
    std::lock_guard<std::mutex> lk(g.mu);
    if (!ctx_init_locked()) return OPUS_INTERNAL_ERROR;
    return sync_states_locked(st, n, true);
}

// Scalar call = batch of one; the host block is left current (write-back) so it stays memcpy-able.
int opus_decode(OpusDecoder *st, const unsigned char *data, opus_int32 len, opus_int16 *pcm, int frame_size, int decode_fec) {
    if (frame_size <= 0) return OPUS_BAD_ARG;
    if (!st || st->magic != kDecMagic || !pcm) return OPUS_BAD_ARG;
    if (decode_fec < 0 || decode_fec > 1) return OPUS_BAD_ARG;
    if (len < 0 && data != nullptr) return OPUS_BAD_ARG;   // a NULL packet is a lost packet whatever its length says (opus_decoder.c:611-629)
    std::lock_guard<std::mutex> lk(g.mu);
    if (!ctx_init_locked()) return OPUS_INTERNAL_ERROR;
    const int channels = st->st.channels;
    // clamp the capacity handed to the kernel: a packet never carries more than 120 ms
    int cap = frame_size;
    const int max_cap = st->st.Fs / 25 * 3;
    if (cap > max_cap && !(decode_fec || len == 0 || data == nullptr)) cap = max_cap;
    if (cap > 4 * max_cap) return OPUS_BAD_ARG;
    int64_t off = 0;
    int32_t l = (data == nullptr) ? 0 : len;
    int r = 0;
    std::vector<int16_t> out((size_t)cap * channels);
    OpusDecoder *one = st;
    int rc = decode_span_host_locked(&one, 1, 1, data, l, &off, &l, out.data(), cap, decode_fec, &r, false);
    if (rc != OPUS_OK) return rc;
    if (r > 0) memcpy(pcm, out.data(), (size_t)r * channels * sizeof(int16_t));
    return r;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// Multistream decoder (libopus opus_multistream.h; layout and packet format RFC 7845 §5.1.1, RFC 6716 Appendix B).  The block
// is a header followed by `streams` ordinary OpusDecoder blocks (coupled streams first, stereo; then mono), so residency,
// write-back, memcpy and the duplicate check of the embedded decoders are exactly those of single-stream decoders.
// ------------------------------------------------------------------------------------------------
struct OpusMSDecoder {
    uint32_t magic;
    int32_t Fs, channels, streams, coupled;
    uint8_t mapping[255];   // output channel c = stream channel mapping[c]; 255 = silence
};
static const uint32_t kMsDecMagic = 0x0B2005DCu;
static const size_t kMsHeader = (sizeof(OpusMSDecoder) + 63) & ~(size_t)63;

static inline OpusDecoder *ms_stream(OpusMSDecoder *st, int s) {
    return reinterpret_cast<OpusDecoder *>(reinterpret_cast<char *>(st) + kMsHeader + (size_t)s * sizeof(OpusDecoder));
}

// Multistream span over host or device buffers (device_io).  n decoders sharing (Fs, channels, streams, coupled); packet (m,f) at
// data[offs[m*F+f] ..][0 .. len[m*F+f]), its PCM at pcm + (m*F+f)*frame_size*channels, ret[m*F+f] = what the scalar call returns.
// data_bytes: extent of the host input (ignored for device_io, where it is measured on the device).
static int ms_decode_span_locked(OpusMSDecoder **st, int n, int F, const unsigned char *data, int64_t data_bytes, const int64_t *offs,
                                 const opus_int32 *len, opus_int16 *pcm, int frame_size, int decode_fec, int *ret, bool device_io,
                                 bool keep_resident) {
    if (!ctx_init_locked()) return OPUS_INTERNAL_ERROR;
    for (int i = 0; i < n; i++) {
        if (!st[i] || st[i]->magic != kMsDecMagic) return OPUS_BAD_ARG;
        // one IR geometry and one elementary layout per call
        if (st[i]->Fs != st[0]->Fs || st[i]->channels != st[0]->channels || st[i]->streams != st[0]->streams ||
            st[i]->coupled != st[0]->coupled)
            return OPUS_BAD_ARG;
    }
    const int Fs = st[0]->Fs, channels = st[0]->channels, S = st[0]->streams, coupled = st[0]->coupled;
    const int E = n * S;
    const size_t NF = (size_t)n * F, EF = (size_t)E * F;
    std::vector<OpusDecoder *> el((size_t)E);
    for (int m = 0; m < n; m++)
        for (int s = 0; s < S; s++) el[(size_t)m * S + s] = ms_stream(st[m], s);
    if (!g.h_slots.reserve(sizeof(int) * (size_t)E)) return OPUS_ALLOC_FAIL;
    int *hsl = (int *)g.h_slots.p;
    int rc = make_resident_locked(el.data(), E, hsl);
    if (rc != OPUS_OK) return rc;
    // opus_multistream_decode clamps the room per channel to 120 ms: what a lost packet conceals; rows keep frame_size
    const int cap = frame_size < Fs / 25 * 3 ? frame_size : Fs / 25 * 3;
    if (!g.d_slots.reserve(sizeof(int) * (size_t)E) || !g.d_eoffs.reserve(sizeof(int64_t) * EF) || !g.d_elens.reserve(sizeof(int32_t) * EF) ||
        !g.d_erets.reserve(sizeof(int) * EF) || !g.d_mserr.reserve(sizeof(int) * NF) || !g.d_map.reserve((size_t)n * channels) ||
        !g.d_extent.reserve(sizeof(unsigned long long)) || !g.h_misc.reserve(sizeof(unsigned long long)))
        return OPUS_ALLOC_FAIL;
    const uint8_t *d_in;
    const int64_t *d_offs;
    const int32_t *d_lens;
    if (device_io) {
        d_in = data; d_offs = offs; d_lens = len;
        cudaMemsetAsync(g.d_extent.p, 0, sizeof(unsigned long long), g.stream);
        ms_extent_kernel<<<(unsigned)((NF + 255) / 256), 256, 0, g.stream>>>(offs, len, (int)NF, (unsigned long long *)g.d_extent.p);
        g.launches++;
        cudaMemcpyAsync(g.h_misc.p, g.d_extent.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost, g.stream);
        if (cudaStreamSynchronize(g.stream) != cudaSuccess) return OPUS_INTERNAL_ERROR;
        data_bytes = (int64_t)*(unsigned long long *)g.h_misc.p;
    } else {
        if (!g.d_data.reserve((size_t)data_bytes + 16) || !g.d_offs.reserve(sizeof(int64_t) * NF) || !g.d_lens.reserve(sizeof(int32_t) * NF) ||
            !g.d_rets.reserve(sizeof(int) * NF))
            return OPUS_ALLOC_FAIL;
        if (data_bytes > 0) cudaMemcpyAsync(g.d_data.p, data, (size_t)data_bytes, cudaMemcpyHostToDevice, g.stream);
        cudaMemcpyAsync(g.d_offs.p, offs, sizeof(int64_t) * NF, cudaMemcpyHostToDevice, g.stream);
        cudaMemcpyAsync(g.d_lens.p, len, sizeof(int32_t) * NF, cudaMemcpyHostToDevice, g.stream);
        d_in = (const uint8_t *)g.d_data.p; d_offs = (const int64_t *)g.d_offs.p; d_lens = (const int32_t *)g.d_lens.p;
    }
    if (!g.d_blob.reserve((size_t)data_bytes + 16)) return OPUS_ALLOC_FAIL;   // the input, then the reject marker at data_bytes
    Plan pl;
    if (!plan_call(pl, E, F, cap, decode_fec, Fs, !device_io)) return OPUS_ALLOC_FAIL;
    const int Fc = pl.Fc, nchunks = pl.nchunks, erow = cap * 2;   // elementary rows sized for stereo: mono and stereo share them
    const size_t orow = (size_t)frame_size * channels * sizeof(int16_t);
    for (int b = 0; b < (nchunks > 1 ? 2 : 1); b++) {
        if (!g.d_epcm[b].reserve((size_t)E * Fc * erow * sizeof(int16_t))) return OPUS_ALLOC_FAIL;
        if (!device_io && !g.d_pcm[b].reserve((size_t)n * Fc * orow)) return OPUS_ALLOC_FAIL;
    }
    {
        std::vector<uint8_t> maps((size_t)n * channels);
        for (int m = 0; m < n; m++) memcpy(maps.data() + (size_t)m * channels, st[m]->mapping, (size_t)channels);
        cudaMemcpyAsync(g.d_map.p, maps.data(), maps.size(), cudaMemcpyHostToDevice, g.stream);
        cudaMemcpyAsync(g.d_slots.p, hsl, sizeof(int) * (size_t)E, cudaMemcpyHostToDevice, g.stream);
        cudaStreamSynchronize(g.stream);   // `maps` is pageable and goes out of scope
    }
    cudaEventRecord(g.ev0, g.stream);
    if (data_bytes > 0) cudaMemcpyAsync(g.d_blob.p, d_in, (size_t)data_bytes, cudaMemcpyDeviceToDevice, g.stream);
    timing_begin(3, g.stream);
    ms_split_kernel<<<(unsigned)((NF + 127) / 128), 128, 0, g.stream>>>(d_in, d_offs, d_lens, n, F, S, Fs, frame_size, (uint8_t *)g.d_blob.p,
                                                                      data_bytes, (int64_t *)g.d_eoffs.p, (int32_t *)g.d_elens.p, (int *)g.d_mserr.p);
    timing_end(g.stream);
    call_ctx_kernel<<<(E + 127) / 128, 128, 0, g.stream>>>(g.pool, (const int *)g.d_slots.p, (CbCallCtx *)g.d_callctx.p, E);
    g.launches += 2;
    cudaEventRecord(g.ev_call, g.stream);
    int *d_ret = device_io ? ret : (int *)g.d_rets.p;
    for (int c = 0; c < nchunks; c++) {
        const int b = c & 1;
        const int f0 = c * Fc, f1 = (f0 + Fc < F) ? f0 + Fc : F;
        if (!device_io && c >= 2) cudaStreamWaitEvent(g.stream, g.ev_copy[b], 0);   // output staging b drained?
        // elementary staging b is free once the gather of chunk c-2 has read it
        enqueue_chunk(pl, c, (const int *)g.d_slots.p, (const uint8_t *)g.d_blob.p, (const int64_t *)g.d_eoffs.p, (const int32_t *)g.d_elens.p,
                      (int16_t *)g.d_epcm[b].p, Fc, f0, erow, (int *)g.d_erets.p, c >= 2 ? g.ev_gather[b] : nullptr);
        int16_t *out = device_io ? (int16_t *)pcm : (int16_t *)g.d_pcm[b].p;
        timing_begin(4, g.stream);
        ms_gather_kernel<<<(unsigned)(n * (f1 - f0)), 256, 0, g.stream>>>((const int16_t *)g.d_epcm[b].p, Fc, erow, (const int *)g.d_erets.p,
                                                                          (const int *)g.d_mserr.p, (const uint8_t *)g.d_map.p, out,
                                                                          device_io ? F : Fc, device_io ? 0 : f0, F, f0, f1, S, coupled,
                                                                          channels, frame_size, d_ret);
        timing_end(g.stream);
        g.launches++;
        cudaEventRecord(g.ev_gather[b], g.stream);
        if (!device_io) {
            cudaEventRecord(g.ev_chunk[b], g.stream);
            cudaStreamWaitEvent(g.copy_stream, g.ev_chunk[b], 0);
            cudaMemcpy2DAsync((char *)pcm + (size_t)f0 * orow, (size_t)F * orow, g.d_pcm[b].p, (size_t)Fc * orow, (size_t)(f1 - f0) * orow,
                              (size_t)n, cudaMemcpyDeviceToHost, g.copy_stream);
            cudaEventRecord(g.ev_copy[b], g.copy_stream);
        }
    }
    cudaEventRecord(g.ev1, g.stream);
    mark_device_newer_locked(el.data(), E);
    if (device_io) return cudaGetLastError() == cudaSuccess ? OPUS_OK : OPUS_INTERNAL_ERROR;
    cudaMemcpyAsync(ret, g.d_rets.p, sizeof(int) * NF, cudaMemcpyDeviceToHost, g.stream);
    if (cudaStreamSynchronize(g.stream) != cudaSuccess || cudaStreamSynchronize(g.copy_stream) != cudaSuccess ||
        cudaStreamSynchronize(g.parse_stream) != cudaSuccess || cudaStreamSynchronize(g.synth_stream) != cudaSuccess) {
        fprintf(stderr, "concentus_b200: CUDA failure in multistream decode: %s\n", cudaGetErrorString(cudaGetLastError()));
        return OPUS_INTERNAL_ERROR;
    }
    cudaEventElapsedTime(&g.last_ms, g.ev0, g.ev1);
    timing_fold();
    if (!keep_resident) return sync_states_locked(el.data(), E, true);
    return OPUS_OK;
}

extern "C" {

int opus_multistream_decoder_get_size(int streams, int coupled_streams) {
    if (streams < 1 || coupled_streams > streams || coupled_streams < 0) return 0;
    return (int)(kMsHeader + (size_t)streams * sizeof(OpusDecoder));
}

int opus_multistream_decoder_init(OpusMSDecoder *st, opus_int32 Fs, int channels, int streams, int coupled_streams,
                                  const unsigned char *mapping) {
    if (channels > 255 || channels < 1 || coupled_streams > streams || streams < 1 || coupled_streams < 0 || streams > 255 - coupled_streams)
        return OPUS_BAD_ARG;
    if (!mapping) return OPUS_BAD_ARG;
    for (int c = 0; c < channels; c++)
        if (mapping[c] >= streams + coupled_streams && mapping[c] != 255) return OPUS_BAD_ARG;
    // re-initialising a live block in place: the embedded decoders give their pool slots back (opus_decoder_init)
    const bool live = st->magic == kMsDecMagic;
    const int old_streams = live ? st->streams : 0;
    for (int s = 0; s < streams; s++) {
        OpusDecoder *d = ms_stream(st, s);
        if (!(live && s < old_streams)) d->magic = 0;   // not a live decoder: nothing to release
        const int ret = opus_decoder_init(d, Fs, s < coupled_streams ? 2 : 1);
        if (ret != OPUS_OK) return ret;
    }
    st->magic = kMsDecMagic;
    st->Fs = Fs;
    st->channels = channels;
    st->streams = streams;
    st->coupled = coupled_streams;
    memset(st->mapping, 255, sizeof(st->mapping));
    memcpy(st->mapping, mapping, (size_t)channels);
    return OPUS_OK;
}

OpusMSDecoder *opus_multistream_decoder_create(opus_int32 Fs, int channels, int streams, int coupled_streams, const unsigned char *mapping,
                                               int *error) {
    if (channels > 255 || channels < 1 || coupled_streams > streams || streams < 1 || coupled_streams < 0 || streams > 255 - coupled_streams) {
        if (error) *error = OPUS_BAD_ARG;
        return nullptr;
    }
    OpusMSDecoder *st = (OpusMSDecoder *)malloc((size_t)opus_multistream_decoder_get_size(streams, coupled_streams));
    if (!st) {
        if (error) *error = OPUS_ALLOC_FAIL;
        return nullptr;
    }
    st->magic = 0;
    const int ret = opus_multistream_decoder_init(st, Fs, channels, streams, coupled_streams, mapping);
    if (error) *error = ret;
    if (ret != OPUS_OK) {
        opus_multistream_decoder_destroy(st);
        st = nullptr;
    }
    return st;
}

void opus_multistream_decoder_destroy(OpusMSDecoder *st) {
    if (!st) return;
    if (st->magic == kMsDecMagic) {
        std::lock_guard<std::mutex> lk(g.mu);
        if (g.ok)
            for (int s = 0; s < st->streams; s++) {
                OpusDecoder *d = ms_stream(st, s);
                if (d->magic == kDecMagic) release_slot_locked(d);
            }
    }
    free(st);
}

int opus_multistream_decoder_ctl(OpusMSDecoder *st, int request, ...) {
    if (!st || st->magic != kMsDecMagic) return OPUS_BAD_ARG;
    int ret = OPUS_OK;
    va_list ap;
    va_start(ap, request);
    switch (request) {
    case OPUS_GET_BANDWIDTH_REQUEST:
    case OPUS_GET_SAMPLE_RATE_REQUEST:
    case OPUS_GET_GAIN_REQUEST:
    case OPUS_GET_LAST_PACKET_DURATION_REQUEST: {   // answered by the first stream
        void *v = va_arg(ap, void *);
        ret = opus_decoder_ctl(ms_stream(st, 0), request, v);
    } break;
    case OPUS_GET_FINAL_RANGE_REQUEST: {   // XOR of every stream's final range
        opus_uint32 *v = va_arg(ap, opus_uint32 *);
        if (!v) { ret = OPUS_BAD_ARG; break; }
        opus_uint32 acc = 0, r = 0;
        for (int s = 0; s < st->streams && ret == OPUS_OK; s++) {
            ret = opus_decoder_ctl(ms_stream(st, s), OPUS_GET_FINAL_RANGE_REQUEST, &r);
            acc ^= r;
        }
        if (ret == OPUS_OK) *v = acc;
    } break;
    case OPUS_RESET_STATE:
        for (int s = 0; s < st->streams && ret == OPUS_OK; s++) ret = opus_decoder_ctl(ms_stream(st, s), OPUS_RESET_STATE);
        break;
    case OPUS_SET_GAIN_REQUEST: {
        const opus_int32 v = va_arg(ap, opus_int32);
        for (int s = 0; s < st->streams && ret == OPUS_OK; s++) ret = opus_decoder_ctl(ms_stream(st, s), OPUS_SET_GAIN_REQUEST, v);
    } break;
    case OPUS_MULTISTREAM_GET_DECODER_STATE_REQUEST: {
        const opus_int32 id = va_arg(ap, opus_int32);
        OpusDecoder **v = va_arg(ap, OpusDecoder **);
        if (id < 0 || id >= st->streams) { ret = OPUS_BAD_ARG; break; }
        *v = ms_stream(st, id);
    } break;
    default:
        ret = OPUS_UNIMPLEMENTED;
        break;
    }
    va_end(ap);
    return ret;
}

int opus_multistream_decode_span(OpusMSDecoder **st, int n, int F, const unsigned char *data, const int64_t *offs, const opus_int32 *len,
                                 opus_int16 *pcm, int frame_size, int *ret) {
    if (!st || n <= 0 || F <= 0 || frame_size <= 0 || !offs || !len || !pcm || !ret) return OPUS_BAD_ARG;
    int64_t bytes = 0;
    const size_t NF = (size_t)n * F;
    for (size_t i = 0; i < NF; i++) {
        if (len[i] > 0 && offs[i] < 0) return OPUS_BAD_ARG;
        const int64_t e = offs[i] + len[i];
        if (len[i] > 0 && e > bytes) bytes = e;
    }
    std::lock_guard<std::mutex> lk(g.mu);
    return ms_decode_span_locked(st, n, F, data, bytes, offs, len, pcm, frame_size, 0, ret, false, true);
}

int opus_multistream_decode_span_device(OpusMSDecoder **st, int n, int F, const unsigned char *d_data, const int64_t *d_offs,
                                        const opus_int32 *d_len, opus_int16 *d_pcm, int frame_size, int *d_ret) {
    if (!st || n <= 0 || F <= 0 || frame_size <= 0) return OPUS_BAD_ARG;
    std::lock_guard<std::mutex> lk(g.mu);
    return ms_decode_span_locked(st, n, F, d_data, 0, d_offs, d_len, d_pcm, frame_size, 0, d_ret, true, true);
}

int opus_multistream_decoder_sync(OpusMSDecoder **st, int n) {
    if (!st || n <= 0) return OPUS_BAD_ARG;
    std::vector<OpusDecoder *> el;
    for (int m = 0; m < n; m++) {
        if (!st[m] || st[m]->magic != kMsDecMagic) return OPUS_BAD_ARG;
        for (int s = 0; s < st[m]->streams; s++) el.push_back(ms_stream(st[m], s));
    }
    std::lock_guard<std::mutex> lk(g.mu);
    if (!ctx_init_locked()) return OPUS_INTERNAL_ERROR;
    return sync_states_locked(el.data(), (int)el.size(), true);
}

// Scalar call = span of one; the embedded blocks are left current (write-back) so the decoder stays memcpy-able.
int opus_multistream_decode(OpusMSDecoder *st, const unsigned char *data, opus_int32 len, opus_int16 *pcm, int frame_size, int decode_fec) {
    if (frame_size <= 0) return OPUS_BAD_ARG;
    if (!st || st->magic != kMsDecMagic || !pcm) return OPUS_BAD_ARG;
    if (decode_fec < 0 || decode_fec > 1) return OPUS_BAD_ARG;
    if (data == nullptr) len = 0;   // a NULL packet is a lost packet
    if (len < 0) return OPUS_BAD_ARG;
    // a row of the clamped size holds whatever the call can return (ms_decode_span_locked: at most 120 ms)
    const int cap = frame_size < st->Fs / 25 * 3 ? frame_size : st->Fs / 25 * 3;
    std::lock_guard<std::mutex> lk(g.mu);
    std::vector<int16_t> out((size_t)cap * st->channels);
    int64_t off = 0;
    int32_t l = len;
    int r = 0;
    OpusMSDecoder *one = st;
    const int rc = ms_decode_span_locked(&one, 1, 1, data, l, &off, &l, out.data(), cap, decode_fec, &r, false, false);
    if (rc != OPUS_OK) return rc;
    if (r > 0) memcpy(pcm, out.data(), (size_t)r * st->channels * sizeof(int16_t));
    return r;
}

}  // extern "C"
