// opus_enc_capi.cu — encoder kernels and the encoder half of the C ABI of libconcentus_b200.so (include/opus_b200.h).
//
// Boundary: libopus's public encoder API (opus-fix/include/opus.h:171-328, src/opus_encoder.c:150-252,2007-2507) plus our
// batch / span calls.  Host side = argument checks, ctl, state residency and copies; everything from the Opus-layer rate
// decisions down to ec_enc_done runs on the device, one warp per stream, F frames per launch (the frames of a stream are
// serially dependent through the encoder state; streams are independent).
// There is NO CPU path: if CUDA is unusable every codec call returns OPUS_INTERNAL_ERROR.
#if !defined(CB_NO_PHASE_SYNC) && !defined(CB_PHASE_SYNC)
#define CB_PHASE_SYNC 1      // see the block-shape note below
#endif
#define CB_SMALL_CODE 1   // see celt_simt.cuh: the encoder kernel is instruction-cache bound when everything is inlined
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <unordered_set>
#include <vector>

#include "../../include/opus_b200.h"
#include "enc_pipe_host.h"
#include "host_runtime.h"
#include "opus_encoder_dev.cuh"
#include "opus_ms_encoder.h"
#include "opus_multistream.h"

using namespace cb;

extern "C" int opus_b200_device_index(void);   // opus_capi.cu: the device opus_b200_init selected (initialises the runtime)

// Caller-visible state block: pointer-free and memcpy-able like the reference's (tests/test_opus_encode.c:198,214).
// Same residency protocol as OpusDecoder (opus_capi.cu).
struct OpusEncoder {
    uint32_t magic;
    int32_t slot;
    uint64_t gen;
    int32_t host_current;
    int32_t device;        // the device whose pool `slot` refers to
    CbEncState st;
};
static const uint32_t kEncMagic = 0x0B200E4Cu;

// Block shape (measured on B200, profiles/r1_enc_*): ONE block of 14 warps per SM, the warps phase-synchronised
// (celt_simt.cuh WarpTeam::phase).  The kernel is ~250 KB of SASS against a 32 KB L1.5 instruction cache: with free-running
// warps 35-70 % of the issue slots were lost to instruction fetch; letting the 14 streams of an SM walk the frame in step
// doubled the throughput.  2,072 streams are resident per B200, so 4,096 streams are two full waves.
#ifndef CB_ENC_WPB
#define CB_ENC_WPB 14         // warps (= streams) per block
#endif
#ifndef CB_ENC_MINBLOCKS
#define CB_ENC_MINBLOCKS 1
#endif
#if !defined(CB_NO_PHASE_SYNC) && !defined(CB_PHASE_SYNC)
#define CB_PHASE_SYNC 1
#endif

// Shared memory of one warp: the frame working set plus the head of the stream's state (scalars + band-energy histories),
// which stays on chip for the whole span and is written back once at the end.
struct EncWarpSmem {
    EncShared S;
    int head[CB_ENC_HEAD_BYTES / 4];
};

// The one-kernel path: takes every stream the frame-synchronous pipeline (opus_enc_pipe.cu) does not (OPUS_APPLICATION_AUDIO,
// 40 / 60 ms frames, "PLC frame" budgets) — and everything when CB200_ENC_PIPE=0.
// One warp per stream, frames 0..F-1 in order.  PCM of frame (s,f): pcm[(s*F+f)*frame_size*channels]; packet slot:
// data[(s*F+f)*stride], at most max_bytes are written; rets[s*F+f] = packet length or error.  One launch codes frames [f0, f1).
// ctl (nullable): per-frame control of the multistream encoder, ctl[s*F+f] = {budget, bitrate, bitrate2, -}: the frame is coded
// with `budget` in place of max_bytes after OPUS_SET_BITRATE(bitrate) and OPUS_SET_BITRATE(bitrate2) (0 = none: enc_ctl refuses
// it).  A budget <= 0 returns OPUS_BAD_ARG with the state untouched, which is how a frame is skipped.  kCtl = (ctl != nullptr):
// a separate instantiation, so that the single-stream kernel's code, registers and spills stay what they were.
template <bool kCtl>
__global__ void __launch_bounds__(CB_ENC_WPB * 32, CB_ENC_MINBLOCKS)
encode_span_kernel(CbEncState *pool, const int *slots, const int *sidx, EncGlobal *scratch, const int16_t *pcm, uint8_t *data, int *rets,
                   unsigned *ranges, int n, int F, int f0, int f1, int frame_size, int max_bytes, int stride, const int4 *ctl) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int s = blockIdx.x * CB_ENC_WPB + warp;
    if (s >= n) {
#if defined(CB_PHASE_SYNC)
        {
            WarpTeam idle{lane};
            for (int f = 0; f < (f1 - f0) * kEncPhases; f++) idle.phase();   // keep the block's phase barriers balanced
        }
#endif
        return;
    }
    EncWarpSmem &W = reinterpret_cast<EncWarpSmem *>(smem_raw)[warp];
    CbEncState *gst = pool + slots[s];
    for (int i = lane; i < CB_ENC_HEAD_BYTES / 4; i += 32) W.head[i] = reinterpret_cast<const int *>(gst)[i];
    __syncwarp();
    CbEncState *st = reinterpret_cast<CbEncState *>(W.head);   // only the head fields are valid through this pointer
    EncGlobal &G = scratch[s];
    const int channels = st->channels;
    WarpTeam tm{lane};
    const int srow = sidx ? sidx[s] : s;   // the stream's row of PCM / packets / rets (a launch may cover a subset of a call's streams)
    for (int f = f0; f < f1; f++) {
        const size_t k = (size_t)srow * F + f;
        int budget = max_bytes;
        if (kCtl) {
            const int4 c = ctl[k];
            budget = c.x;
            if (lane == 0) {
                int unused;
                enc_ctl(st, 4002, c.y, &unused);   // OPUS_SET_BITRATE
                enc_ctl(st, 4002, c.z, &unused);
            }
            __syncwarp();
        }
        const int r = opus_encode_frame(tm, st, gst, W.S, G, pcm + k * frame_size * channels, frame_size, data + k * stride, budget);
        if (lane == 0) {
            rets[k] = r;
            if (ranges) ranges[k] = st->rangeFinal;   // OPUS_GET_FINAL_RANGE after this frame (what opus_demo stores per packet)
        }
        __syncwarp();
    }
    for (int i = lane; i < CB_ENC_HEAD_BYTES / 4; i += 32) reinterpret_cast<int *>(gst)[i] = W.head[i];
}

__global__ void enc_scatter_states_kernel(CbEncState *pool, const int *slots, const CbEncState *stage, int n) {
    const int words = sizeof(CbEncState) / 4;
    for (int k = blockIdx.x; k < n; k += gridDim.x) {
        const int *src = reinterpret_cast<const int *>(stage + k);
        int *dst = reinterpret_cast<int *>(pool + slots[k]);
        for (int i = threadIdx.x; i < words; i += blockDim.x) dst[i] = src[i];
    }
}
__global__ void enc_gather_states_kernel(const CbEncState *pool, const int *slots, CbEncState *stage, int n) {
    const int words = sizeof(CbEncState) / 4;
    for (int k = blockIdx.x; k < n; k += gridDim.x) {
        const int *src = reinterpret_cast<const int *>(pool + slots[k]);
        int *dst = reinterpret_cast<int *>(stage + k);
        for (int i = threadIdx.x; i < words; i += blockDim.x) dst[i] = src[i];
    }
}

// ---- multistream (DESIGN.md §3): a call over n multistream encoders of S streams codes the n·S embedded encoders, coupled
// (stereo) streams and mono streams in two groups of uniform channel count.  Group row g of stream s of encoder m:
// m*coupled + s (coupled), m*(S-coupled) + s - coupled (mono); PCM, packets, returns and per-frame control of row g, frame f
// are at index g*F + f of the group's arrays, as the single-stream launches lay them out.
__device__ __forceinline__ int ms_group_row(int m, int s, int S, int coupled) { return s < coupled ? m * coupled + s : m * (S - coupled) + s - coupled; }

// One block per multistream frame (m,f): input row pcm[(m*F+f)*frame_size*channels] -> the stereo rows of its coupled streams and
// the mono rows of its mono streams.  src[m*K + k] (K = S + coupled) is the input channel of stream channel k (the first one
// mapped to it).  A row that fits is staged in shared memory with 16-byte loads.
enum { kMsRouteSmem = 32 * 1024 };
__global__ void __launch_bounds__(256)
ms_route_kernel(const int16_t *pcm, const int *src, int F, int channels, int frame_size, int S, int coupled, int16_t *st_pcm,
                int16_t *mono_pcm) {
    __shared__ __align__(16) int16_t row[kMsRouteSmem / 2];
    __shared__ int s_src[512];
    const int m = blockIdx.x / F, f = blockIdx.x - m * F;
    const int K = S + coupled, mono = S - coupled;
    for (int k = threadIdx.x; k < K; k += blockDim.x) s_src[k] = src[(size_t)m * K + k];
    const size_t nsmp = (size_t)frame_size * channels;
    const int16_t *in = pcm + ((size_t)m * F + f) * nsmp;
    const bool staged = nsmp * 2 <= kMsRouteSmem && (nsmp & 7) == 0 && ((uintptr_t)in & 15) == 0;
    if (staged) {
        const int4 *in4 = reinterpret_cast<const int4 *>(in);
        int4 *row4 = reinterpret_cast<int4 *>(row);
        for (int i = threadIdx.x; i < (int)(nsmp / 8); i += blockDim.x) row4[i] = in4[i];
    }
    __syncthreads();
    const int16_t *x = staged ? row : in;
    for (int i = threadIdx.x; i < frame_size; i += blockDim.x) {
        const int16_t *xi = x + (size_t)i * channels;
        for (int s = 0; s < coupled; s++) {
            int16_t *o = st_pcm + ((size_t)(m * coupled + s) * F + f) * frame_size * 2;
            o[2 * i] = xi[s_src[2 * s]];
            o[2 * i + 1] = xi[s_src[2 * s + 1]];
        }
        for (int j = 0; j < mono; j++) mono_pcm[((size_t)(m * mono + j) * F + f) * frame_size + i] = xi[s_src[2 * coupled + j]];
    }
}

// Per-encoder parameters of a multistream call: {max_data_bytes after the CBR cap, CBR (stream 0 not VBR), the last stream's
// allocated rate, -}.
// ms_budget_kernel: one thread per multistream frame (m,f), before the pass over stream s: the control of (m,s,f) for
// encode_span_kernel from the bytes the earlier streams took (tot) — a budget of 0 skips the frame when an earlier stream of
// it failed (err); CBR's last stream is set to its allocated rate, then to the rate of its budget (opus_multistream_encode_native).
__global__ void ms_budget_kernel(const int4 *prm, const int *tot, const int *err, int n, int F, int S, int coupled, int s, int Fs,
                                 int frame_size, int4 *ctl) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * F) return;
    const int m = t / F, f = t - m * F;
    const int4 p = prm[m];
    const bool last_cbr = p.y && s == S - 1;
    int4 c = make_int4(0, last_cbr ? p.z : 0, 0, 0);
    if (err[t] == 0) {
        const int curr_max = ms_stream_budget(p.x, tot[t], S, s);
        c.x = curr_max < 1276 ? curr_max : 1276;   // the single-stream encoder's clamp (opus_encode)
        if (last_cbr) c.z = ms_cbr_last_bitrate(curr_max, Fs, frame_size);
    }
    ctl[(size_t)ms_group_row(m, s, S, coupled) * F + f] = c;
}

// One thread per multistream frame (m,f): streams [s0, s1) of it are framed (ms_pack_packet) into the caller's slot
// data + (m*F+f)*slot after the tot bytes the streams before s0 took.  The first error in stream order stops the packet
// (err); with `final`, ret = err or the packet length.
__global__ void ms_pack_kernel(const int4 *prm, const uint8_t *epkt_st, const uint8_t *epkt_mono, const int *erets_st, const int *erets_mono,
                               int estride, int n, int F, int S, int coupled, int s0, int s1, uint8_t *data, int slot, int *tot, int *err,
                               int *ret, int final) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * F) return;
    const int m = t / F, f = t - m * F;
    const int4 p = prm[m];
    int e = err[t], used = tot[t];
    uint8_t *out = data + (size_t)t * slot;
    for (int s = s0; s < s1 && e == 0; s++) {
        const size_t k = (size_t)ms_group_row(m, s, S, coupled) * F + f;
        const int r = s < coupled ? erets_st[k] : erets_mono[k];
        if (r < 0) { e = r; break; }
        const uint8_t *pk = (s < coupled ? epkt_st : epkt_mono) + k * estride;
        const int len = ms_pack_packet(pk, r, s < S - 1, p.y && s == S - 1, out + used, p.x - used);
        if (len < 0) { e = len; break; }
        used += len;
    }
    err[t] = e;
    tot[t] = used;
    if (final) ret[t] = e ? e : used;
}

// OPUS_SET_BITRATE on resident embedded encoders: pairs (slot, value)
__global__ void ms_set_bitrate_kernel(CbEncState *pool, const int *pairs, int K) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K) return;
    int unused;
    enc_ctl(pool + pairs[2 * k], 4002, pairs[2 * k + 1], &unused);
}

namespace {

inline int hmin(int a, int b) { return a < b ? a : b; }

typedef CbSlotInfo SlotInfo;
typedef CbDevBuf DevBuf;
typedef CbPinBuf PinBuf;

struct EncCtx {
    std::mutex mu;
    bool tried = false, ok = false;
    cudaStream_t stream = nullptr, copy_stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    enum { kMaxSub = 8 };
    cudaEvent_t ev_in[kMaxSub] = {}, ev_done[kMaxSub] = {}, ev_prev = nullptr;
    CbEncState *pool = nullptr;
    int pool_cap = 0;
    std::vector<SlotInfo> reg;
    std::vector<int> free_slots;
    DevBuf d_slots, d_pcm, d_data, d_rets, d_ranges, d_stage, d_scratch, d_split;
    PinBuf h_stage, h_slots, h_split[4];
    cudaStream_t legacy_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_legacy = nullptr;
    int use_pipe = 1;
    unsigned split_seq = 0;
    long long pipe_streams = 0, legacy_streams = 0;
    long long launches = 0;
    float last_ms = 0.f;
    double total_ms = 0;
    int device = 0;
    std::mutex deferred_mu;
    std::vector<std::pair<int, const void *>> deferred;   // slots of this pool whose owners moved to another device
    // multistream calls: routed PCM (stereo rows, mono rows), elementary packets / returns (stereo group, then mono group),
    // per-frame control, per-packet bytes used and first error, the call's upload of indices and parameters (a ring of pinned
    // host buffers, as for split_span), the last stream's control read back in CBR, and device time per stage (route, budget, pack)
    DevBuf d_ms_pcm[2], d_ms_pkt, d_ms_rets, d_ms_ctl, d_ms_tot, d_ms_err, d_ms_idx;
    PinBuf h_ms[4], h_ms_ctl;
    unsigned ms_seq = 0;
    struct Timed { cudaEvent_t a, b; int stage; };
    std::vector<Timed> ms_timed;
    std::vector<cudaEvent_t> ms_ev_pool;
    double ms_stage_ms[3] = {0, 0, 0};
    long long ms_stage_launches[3] = {0, 0, 0};
};
// one context per device; the calling thread's device is the one it selected with opus_b200_init (host_runtime.h)
EncCtx e_ctxs[kCbMaxDevices];
#define e (e_ctxs[opus_b200_current_device()])
enum { kStageStates = 4096 };   // states per upload / download slice

bool ctx_init_locked() {
    if (e.tried) {
        if (e.ok) {
            cudaSetDevice(e.device);
            if (!e.deferred.empty()) {
                std::lock_guard<std::mutex> lk(e.deferred_mu);
                for (auto &pr : e.deferred)
                    if (pr.first >= 0 && pr.first < e.pool_cap && e.reg[pr.first].owner == pr.second) {
                        e.reg[pr.first].owner = nullptr;
                        e.reg[pr.first].gen++;
                        e.free_slots.push_back(pr.first);
                    }
                e.deferred.clear();
            }
        }
        return e.ok;
    }
    e.tried = true;
    const int dev = opus_b200_device_index();
    if (dev < 0) return false;
    e.device = dev;
    if (cudaSetDevice(dev) != cudaSuccess) return false;
    if (cudaStreamCreateWithFlags(&e.stream, cudaStreamNonBlocking) != cudaSuccess) return false;
    if (cudaStreamCreateWithFlags(&e.copy_stream, cudaStreamNonBlocking) != cudaSuccess) return false;
    cudaEventCreate(&e.ev0);
    cudaEventCreate(&e.ev1);
    for (int i = 0; i < EncCtx::kMaxSub; i++) {
        cudaEventCreateWithFlags(&e.ev_in[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&e.ev_done[i], cudaEventDisableTiming);
    }
    cudaEventCreateWithFlags(&e.ev_prev, cudaEventDisableTiming);
    if (cudaStreamCreateWithFlags(&e.legacy_stream, cudaStreamNonBlocking) != cudaSuccess) return false;
    cudaEventCreateWithFlags(&e.ev_fork, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&e.ev_legacy, cudaEventDisableTiming);
    if (const char *v = getenv("CB200_ENC_PIPE")) e.use_pipe = atoi(v);
    if (!e.h_stage.reserve(sizeof(CbEncState) * 64) || !e.d_stage.reserve(sizeof(CbEncState) * 64)) return false;
    for (auto k : {encode_span_kernel<false>, encode_span_kernel<true>})
        cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(CB_ENC_WPB * sizeof(EncWarpSmem)));
#ifndef CB_ENC_CARVEOUT
#define CB_ENC_CARVEOUT 70   // % of the 228 KB: the block needs 157 KB of shared memory; the rest stays L1 for stacks and tables
#endif
    for (auto k : {encode_span_kernel<false>, encode_span_kernel<true>})
        cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, CB_ENC_CARVEOUT);
    e.ok = cudaGetLastError() == cudaSuccess;
    return e.ok;
}

bool pool_reserve_locked(int need_total) {
    if (need_total <= e.pool_cap) return true;
    int ncap = e.pool_cap ? e.pool_cap : 64;
    while (ncap < need_total) ncap *= 2;
    CbEncState *np = nullptr;
    if (cudaMalloc(&np, sizeof(CbEncState) * (size_t)ncap) != cudaSuccess) return false;
    if (e.pool) {
        cudaMemcpyAsync(np, e.pool, sizeof(CbEncState) * (size_t)e.pool_cap, cudaMemcpyDeviceToDevice, e.stream);
        cudaStreamSynchronize(e.stream);
        cudaFree(e.pool);
    }
    for (int i = ncap - 1; i >= e.pool_cap; i--) e.free_slots.push_back(i);
    e.reg.resize(ncap, SlotInfo{nullptr, 0});
    e.pool = np;
    e.pool_cap = ncap;
    return true;
}

inline bool resident(const OpusEncoder *d) {
    return d->device == e.device && d->slot >= 0 && d->slot < e.pool_cap && e.reg[d->slot].owner == d && e.reg[d->slot].gen == d->gen;
}
// the block's slot lives in another device's pool: that device's next call gives it back
void release_elsewhere(OpusEncoder *d) {
    if (d->slot >= 0 && d->device >= 0 && d->device < kCbMaxDevices && d->device != e.device) {
        EncCtx &o = e_ctxs[d->device];
        std::lock_guard<std::mutex> lk(o.deferred_mu);
        o.deferred.emplace_back(d->slot, (const void *)d);
        d->slot = -1;
    }
}

int make_host_current_locked(OpusEncoder *d) {
    if (d->host_current) return OPUS_OK;
    // (a state resident on another device has to be synchronised by a thread of that device: OPUS_INVALID_STATE here)
    if (d->device != e.device || d->slot < 0 || d->slot >= e.pool_cap || e.reg[d->slot].gen != d->gen) return OPUS_INVALID_STATE;
    if (cudaMemcpyAsync(&d->st, e.pool + d->slot, sizeof(CbEncState), cudaMemcpyDeviceToHost, e.stream) != cudaSuccess) return OPUS_INTERNAL_ERROR;
    if (cudaStreamSynchronize(e.stream) != cudaSuccess) return OPUS_INTERNAL_ERROR;
    d->host_current = 1;
    return OPUS_OK;
}

void release_slot_locked(OpusEncoder *d) {
    release_elsewhere(d);
    if (d->slot >= 0 && d->slot < e.pool_cap && e.reg[d->slot].owner == d) {
        e.reg[d->slot].owner = nullptr;
        e.reg[d->slot].gen++;
        e.free_slots.push_back(d->slot);
    }
    d->slot = -1;
}

int make_resident_locked(OpusEncoder **st, int n, int *h_slots) {
    int need_new = 0;
    for (int i = 0; i < n; i++) {
        OpusEncoder *d = st[i];
        if (!d || d->magic != kEncMagic) return OPUS_BAD_ARG;
        if (!resident(d)) need_new++;
    }
    if (n > 1) {   // the same state twice in one batch would race two warps on it
        std::unordered_set<const void *> seen;
        seen.reserve((size_t)n * 2);
        for (int i = 0; i < n; i++)
            if (!seen.insert(st[i]).second) return OPUS_BAD_ARG;
    }
    const int in_use = e.pool_cap - (int)e.free_slots.size();
    if (!pool_reserve_locked(in_use + need_new)) return OPUS_ALLOC_FAIL;
    std::vector<int> up_idx;
    for (int i = 0; i < n; i++) {
        OpusEncoder *d = st[i];
        if (resident(d)) {
            if (d->host_current) up_idx.push_back(i);
        } else {
            if (!d->host_current) {
                int rc = make_host_current_locked(d);
                if (rc != OPUS_OK) return rc;
            }
            release_elsewhere(d);
            d->slot = e.free_slots.back();
            e.free_slots.pop_back();
            d->device = e.device;
            e.reg[d->slot].owner = d;
            d->gen = ++e.reg[d->slot].gen;
            up_idx.push_back(i);
        }
        h_slots[i] = d->slot;
    }
    {
        const size_t slice = up_idx.size() < (size_t)kStageStates ? up_idx.size() : (size_t)kStageStates;
        if (slice > 0 && (!e.h_stage.reserve(sizeof(CbEncState) * slice) || !e.d_stage.reserve(sizeof(CbEncState) * slice))) return OPUS_ALLOC_FAIL;
    }
    CbEncState *hs = (CbEncState *)e.h_stage.p;
    if (!e.d_slots.reserve(sizeof(int) * (size_t)(n > kStageStates ? n : kStageStates))) return OPUS_ALLOC_FAIL;
    for (size_t base = 0; base < up_idx.size(); base += kStageStates) {
        const int cnt = (int)((up_idx.size() - base) < (size_t)kStageStates ? (up_idx.size() - base) : kStageStates);
        std::vector<int> sl(cnt);
        for (int k = 0; k < cnt; k++) {
            OpusEncoder *d = st[up_idx[base + k]];
            memcpy(&hs[k], &d->st, sizeof(CbEncState));
            sl[k] = d->slot;
        }
        cudaMemcpyAsync(e.d_stage.p, hs, sizeof(CbEncState) * (size_t)cnt, cudaMemcpyHostToDevice, e.stream);
        cudaMemcpyAsync(e.d_slots.p, sl.data(), sizeof(int) * (size_t)cnt, cudaMemcpyHostToDevice, e.stream);
        enc_scatter_states_kernel<<<cnt < 2048 ? cnt : 2048, 256, 0, e.stream>>>(e.pool, (const int *)e.d_slots.p, (const CbEncState *)e.d_stage.p, cnt);
        if (cudaStreamSynchronize(e.stream) != cudaSuccess) return OPUS_INTERNAL_ERROR;
    }
    return OPUS_OK;
}

void mark_device_newer_locked(OpusEncoder **st, int n) {
    for (int i = 0; i < n; i++) {
        OpusEncoder *d = st[i];
        d->gen = ++e.reg[d->slot].gen;
        d->host_current = 0;
    }
}

int sync_states_locked(OpusEncoder **st, int n, bool release) {
    std::vector<int> idx;
    for (int i = 0; i < n; i++) {
        OpusEncoder *d = st[i];
        if (!d || d->magic != kEncMagic) return OPUS_BAD_ARG;
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
        if (slice > 0 && (!e.h_stage.reserve(sizeof(CbEncState) * slice) || !e.d_stage.reserve(sizeof(CbEncState) * slice))) return OPUS_ALLOC_FAIL;
    }
    CbEncState *hs = (CbEncState *)e.h_stage.p;
    if (!e.d_slots.reserve(sizeof(int) * (size_t)kStageStates)) return OPUS_ALLOC_FAIL;
    for (size_t base = 0; base < idx.size(); base += kStageStates) {
        const int cnt = (int)((idx.size() - base) < (size_t)kStageStates ? (idx.size() - base) : kStageStates);
        std::vector<int> sl(cnt);
        for (int k = 0; k < cnt; k++) sl[k] = st[idx[base + k]]->slot;
        cudaMemcpyAsync(e.d_slots.p, sl.data(), sizeof(int) * (size_t)cnt, cudaMemcpyHostToDevice, e.stream);
        enc_gather_states_kernel<<<cnt < 2048 ? cnt : 2048, 256, 0, e.stream>>>(e.pool, (const int *)e.d_slots.p, (CbEncState *)e.d_stage.p, cnt);
        cudaMemcpyAsync(hs, e.d_stage.p, sizeof(CbEncState) * (size_t)cnt, cudaMemcpyDeviceToHost, e.stream);
        if (cudaStreamSynchronize(e.stream) != cudaSuccess) return OPUS_INTERNAL_ERROR;
        for (int k = 0; k < cnt; k++) {
            OpusEncoder *d = st[idx[base + k]];
            memcpy(&d->st, &hs[k], sizeof(CbEncState));
            d->host_current = 1;
        }
    }
    if (release)
        for (int i = 0; i < n; i++) release_slot_locked(st[i]);
    return OPUS_OK;
}

// Common checks of a span call; all streams must share Fs / channels, and frame_size must be the size every stream actually
// codes: opus_encode runs frame_size_select (opus_encoder.c:807-826,2007-2025) first, so a stream whose
// OPUS_SET_EXPERT_FRAME_DURATION selects another size, or a size that is no Opus frame, is an argument error here (the kernel
// would otherwise walk PCM rows of the wrong length).  The ctl-visible configuration never changes on the device, so a stale host
// block still holds it.
int check_span(OpusEncoder **st, int n, int frame_size) {
    for (int i = 0; i < n; i++) {
        if (!st[i] || st[i]->magic != kEncMagic) return OPUS_BAD_ARG;
        if (st[i]->st.channels != st[0]->st.channels || st[i]->st.Fs != st[0]->st.Fs) return OPUS_BAD_ARG;
        if (frame_size_select(frame_size, st[i]->st.variable_duration, st[i]->st.Fs) != frame_size) return OPUS_BAD_ARG;
    }
    return OPUS_OK;
}

// How a call's streams are divided between the two encoder paths (device arrays in e.d_split).
struct SpanSplit {
    int n_pipe = 0, n_legacy = 0;
    const int *d_pslots = nullptr, *d_psidx = nullptr, *d_lslots = nullptr, *d_lsidx = nullptr;
};

// Decide per stream (host side, ctl-visible configuration only) and upload the two index lists.
bool split_span(OpusEncoder **st, const int *h_slots, int n, int frame_size, int max_bytes, SpanSplit &sp) {
    PinBuf &hb = e.h_split[e.split_seq++ & 3];   // a small ring: an earlier call's upload may still be in flight
    if (!hb.reserve(sizeof(int) * 4 * (size_t)n) || !e.d_split.reserve(sizeof(int) * 4 * (size_t)n)) return false;
    int *h = (int *)hb.p;
    int *pslots = h, *psidx = h + n, *lslots = h + 2 * n, *lsidx = h + 3 * n;
    for (int i = 0; i < n; i++) {
        if (e.use_pipe && enc_pipe_takes(&st[i]->st, frame_size, max_bytes)) { pslots[sp.n_pipe] = h_slots[i]; psidx[sp.n_pipe++] = i; }
        else { lslots[sp.n_legacy] = h_slots[i]; lsidx[sp.n_legacy++] = i; }
    }
    cudaMemcpyAsync(e.d_split.p, h, sizeof(int) * 4 * (size_t)n, cudaMemcpyHostToDevice, e.stream);
    const int *d = (const int *)e.d_split.p;
    sp.d_pslots = d; sp.d_psidx = d + n; sp.d_lslots = d + 2 * n; sp.d_lsidx = d + 3 * n;
    e.pipe_streams += sp.n_pipe;
    e.legacy_streams += sp.n_legacy;
    return true;
}

// d_ctl (multistream calls, see encode_span_kernel): only with sp.n_pipe == 0, the pipeline takes no per-frame control.
int launch_frames(const SpanSplit &sp, const int16_t *d_pcm, uint8_t *d_data, int *d_rets, int F, int f0, int f1, int frame_size, int channels, int Fs,
                  int max_bytes, int stride, unsigned *d_ranges = nullptr, const int4 *d_ctl = nullptr) {
    if (sp.n_legacy > 0) {
        // the one-kernel path runs beside the pipeline on its own stream
        if (!e.d_scratch.reserve(sizeof(EncGlobal) * (size_t)sp.n_legacy)) return OPUS_ALLOC_FAIL;
        cudaStream_t ls = sp.n_pipe > 0 ? e.legacy_stream : e.stream;
        if (sp.n_pipe > 0) {
            cudaEventRecord(e.ev_fork, e.stream);
            cudaStreamWaitEvent(ls, e.ev_fork, 0);
        }
        (d_ctl ? encode_span_kernel<true> : encode_span_kernel<false>)<<<(sp.n_legacy + CB_ENC_WPB - 1) / CB_ENC_WPB, CB_ENC_WPB * 32,
                                                                       CB_ENC_WPB * sizeof(EncWarpSmem), ls>>>(
            e.pool, sp.d_lslots, sp.d_lsidx, (EncGlobal *)e.d_scratch.p, d_pcm, d_data, d_rets, d_ranges, sp.n_legacy, F, f0, f1, frame_size, max_bytes,
            stride, d_ctl);
        e.launches++;
        if (sp.n_pipe > 0) cudaEventRecord(e.ev_legacy, ls);
    }
    if (sp.n_pipe > 0) {
        EncPipeCall c;
        c.pool = e.pool; c.d_slots = sp.d_pslots; c.d_sidx = sp.d_psidx; c.n = sp.n_pipe;
        c.F = F; c.f0 = f0; c.f1 = f1; c.frame_size = frame_size; c.channels = channels; c.Fs = Fs;
        c.max_bytes = max_bytes; c.stride = stride;
        c.d_pcm = d_pcm; c.d_data = d_data; c.d_rets = d_rets; c.d_ranges = d_ranges;
        const int r = enc_pipe_enqueue(c, e.stream);
        if (r < 0) return r;
        e.launches += r;
        if (sp.n_legacy > 0) cudaStreamWaitEvent(e.stream, e.ev_legacy, 0);
    }
    return OPUS_OK;
}
int launch_span(const SpanSplit &sp, const int16_t *d_pcm, uint8_t *d_data, int *d_rets, int F, int frame_size, int channels, int Fs, int max_bytes,
                int stride, unsigned *d_ranges = nullptr) {
    cudaEventRecord(e.ev0, e.stream);
    const int rc = launch_frames(sp, d_pcm, d_data, d_rets, F, 0, F, frame_size, channels, Fs, max_bytes, stride, d_ranges);
    cudaEventRecord(e.ev1, e.stream);
    return rc;
}

int encode_span_host_locked(OpusEncoder **st, int n, int F, const int16_t *pcm, int frame_size, uint8_t *data, int max_bytes, int stride,
                            int *ret, bool keep_resident, uint32_t *ranges = nullptr) {
    if (!ctx_init_locked()) return OPUS_INTERNAL_ERROR;
    int rc = check_span(st, n, frame_size);
    if (rc != OPUS_OK) return rc;
    const int channels = st[0]->st.channels;
    if (!e.h_slots.reserve(sizeof(int) * (size_t)n)) return OPUS_ALLOC_FAIL;
    int *hsl = (int *)e.h_slots.p;
    rc = make_resident_locked(st, n, hsl);
    if (rc != OPUS_OK) return rc;
    const size_t NF = (size_t)n * F;
    const size_t pcm_bytes = NF * frame_size * channels * sizeof(int16_t);
    if (!e.d_pcm.reserve(pcm_bytes) || !e.d_data.reserve(NF * stride) || !e.d_rets.reserve(sizeof(int) * NF) ||
        (ranges && !e.d_ranges.reserve(sizeof(uint32_t) * NF)))
        return OPUS_ALLOC_FAIL;
    unsigned *d_ranges = ranges ? (unsigned *)e.d_ranges.p : nullptr;
    SpanSplit sp;
    if (!split_span(st, hsl, n, frame_size, max_bytes, sp)) return OPUS_ALLOC_FAIL;
    const int Fs = st[0]->st.Fs;
    // Large spans are cut into up to kMaxSub sub-spans of frames: the PCM of sub-span k+1 goes up and the packets of sub-span
    // k-1 come down on the copy stream while sub-span k is coded (the state stays resident between the launches).
    int nsub = 1;
    if (pcm_bytes >= ((size_t)32 << 20)) nsub = F / 8 < 1 ? 1 : (F / 8 > 5 ? 5 : F / 8);
    const size_t row_pcm = (size_t)frame_size * channels * sizeof(int16_t);   // one frame of one stream
    if (nsub == 1) {
        cudaMemcpyAsync(e.d_pcm.p, pcm, pcm_bytes, cudaMemcpyHostToDevice, e.stream);
        rc = launch_span(sp, (const int16_t *)e.d_pcm.p, (uint8_t *)e.d_data.p, (int *)e.d_rets.p, F, frame_size, channels, Fs, max_bytes, stride, d_ranges);
        if (rc != OPUS_OK) return rc;
        cudaMemcpyAsync(data, e.d_data.p, NF * stride, cudaMemcpyDeviceToHost, e.stream);
    } else {
        cudaEventRecord(e.ev_prev, e.stream);                 // earlier work on the device buffers (previous call) is done
        cudaStreamWaitEvent(e.copy_stream, e.ev_prev, 0);
        const int per = (F + nsub - 1) / nsub;
        for (int k = 0; k < nsub; k++) {
            const int f0 = k * per, f1 = hmin(F, f0 + per);
            cudaMemcpy2DAsync((char *)e.d_pcm.p + f0 * row_pcm, F * row_pcm, (const char *)pcm + f0 * row_pcm, F * row_pcm, (f1 - f0) * row_pcm,
                              (size_t)n, cudaMemcpyHostToDevice, e.copy_stream);
            cudaEventRecord(e.ev_in[k], e.copy_stream);
        }
        cudaEventRecord(e.ev0, e.stream);
        for (int k = 0; k < nsub; k++) {
            const int f0 = k * per, f1 = hmin(F, f0 + per);
            cudaStreamWaitEvent(e.stream, e.ev_in[k], 0);
            rc = launch_frames(sp, (const int16_t *)e.d_pcm.p, (uint8_t *)e.d_data.p, (int *)e.d_rets.p, F, f0, f1, frame_size, channels, Fs, max_bytes,
                               stride, d_ranges);
            if (rc != OPUS_OK) return rc;
            cudaEventRecord(e.ev_done[k], e.stream);
            cudaStreamWaitEvent(e.copy_stream, e.ev_done[k], 0);
            cudaMemcpy2DAsync(data + (size_t)f0 * stride, (size_t)F * stride, (const uint8_t *)e.d_data.p + (size_t)f0 * stride, (size_t)F * stride,
                              (size_t)(f1 - f0) * stride, (size_t)n, cudaMemcpyDeviceToHost, e.copy_stream);
        }
        cudaEventRecord(e.ev1, e.stream);
    }
    cudaMemcpyAsync(ret, e.d_rets.p, sizeof(int) * NF, cudaMemcpyDeviceToHost, e.stream);
    if (ranges) cudaMemcpyAsync(ranges, d_ranges, sizeof(uint32_t) * NF, cudaMemcpyDeviceToHost, e.stream);
    mark_device_newer_locked(st, n);
    if (cudaStreamSynchronize(e.stream) != cudaSuccess || cudaStreamSynchronize(e.copy_stream) != cudaSuccess) {
        fprintf(stderr, "concentus_b200: CUDA failure in encode span: %s\n", cudaGetErrorString(cudaGetLastError()));
        return OPUS_INTERNAL_ERROR;
    }
    cudaEventElapsedTime(&e.last_ms, e.ev0, e.ev1);
    e.total_ms += e.last_ms;
    if (!keep_resident) return sync_states_locked(st, n, true);
    return OPUS_OK;
}

}  // namespace

extern "C" {

long long opus_b200_enc_kernel_launches(void) { return e.launches; }
// streams x calls coded by the frame-synchronous pipeline / by the one-kernel path since start (tests check which path ran)
void opus_b200_enc_path_counts(long long *pipe, long long *legacy) {
    if (pipe) *pipe = e.pipe_streams;
    if (legacy) *legacy = e.legacy_streams;
}
// split band loop statistics (opus_enc_pipe.cu): leaves the exact chain searched itself / leaves the speculative chain listed
void opus_b200_enc_band_stats(long long *misses, long long *leaves) {
    std::lock_guard<std::mutex> lk(e.mu);
    if (e.ok) cudaDeviceSynchronize();
    enc_pipe_stats(misses, leaves);
}
// 1 (default): streams the pipeline takes go through it; 0: everything through the one-kernel path.  Returns the previous setting.
int opus_b200_enc_set_pipeline(int on) {
    std::lock_guard<std::mutex> lk(e.mu);
    if (!ctx_init_locked()) return OPUS_INTERNAL_ERROR;
    const int prev = e.use_pipe;
    e.use_pipe = on != 0;
    return prev;
}
#if defined(CB_PHASE_PROF)
// dev build only: cycles per phase slot of stream 0 (own work, then barrier wait); reset != 0 clears the counters
int opus_b200_enc_phase_prof(long long *cycles, long long *wait, int reset) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(cycles, cb::g_phase_cycles, sizeof(long long) * 64);
    cudaMemcpyFromSymbol(wait, cb::g_phase_wait, sizeof(long long) * 64);
    if (reset) {
        long long z[64] = {0};
        int zi = 0;
        cudaMemcpyToSymbol(cb::g_phase_cycles, z, sizeof(z));
        cudaMemcpyToSymbol(cb::g_phase_wait, z, sizeof(z));
        cudaMemcpyToSymbol(cb::g_phase_idx, &zi, sizeof(zi));
    }
    return 0;
}
#endif
void *opus_b200_enc_stream(void) {
    std::lock_guard<std::mutex> lk(e.mu);
    if (!ctx_init_locked()) return nullptr;
    return (void *)e.stream;
}
float opus_b200_enc_last_kernel_ms(void) {
    std::lock_guard<std::mutex> lk(e.mu);
    return e.last_ms;
}
int opus_b200_enc_synchronize(void) {
    std::lock_guard<std::mutex> lk(e.mu);
    if (!ctx_init_locked()) return OPUS_INTERNAL_ERROR;
    if (cudaStreamSynchronize(e.stream) != cudaSuccess) return OPUS_INTERNAL_ERROR;
    if (e.launches > 0) cudaEventElapsedTime(&e.last_ms, e.ev0, e.ev1);
    return OPUS_OK;
}

// ---- lifecycle (opus_encoder.c:150-252,482-510) ----
int opus_encoder_get_size(int channels) {
    if (channels < 1 || channels > 2) return 0;
    return (int)sizeof(OpusEncoder);
}
int opus_encoder_init(OpusEncoder *st, opus_int32 Fs, int channels, int application) {
    if ((Fs != 48000 && Fs != 24000 && Fs != 16000 && Fs != 12000 && Fs != 8000) || (channels != 1 && channels != 2) ||
        (application != OPUS_APPLICATION_VOIP && application != OPUS_APPLICATION_AUDIO && application != OPUS_APPLICATION_RESTRICTED_LOWDELAY))
        return OPUS_BAD_ARG;
    {   // re-initialising a live block in place: give its pool slot back first
        std::lock_guard<std::mutex> lk(e.mu);
        if (e.ok && st->magic == kEncMagic && st->slot >= 0) release_slot_locked(st);
    }
    memset(st, 0, sizeof(OpusEncoder));
    st->magic = kEncMagic;
    st->slot = -1;
    st->gen = 0;
    st->host_current = 1;
    st->device = -1;
    if (enc_state_init(&st->st, Fs, channels, application) != 0) return OPUS_BAD_ARG;
    return OPUS_OK;
}
OpusEncoder *opus_encoder_create(opus_int32 Fs, int channels, int application, int *error) {
    if ((Fs != 48000 && Fs != 24000 && Fs != 16000 && Fs != 12000 && Fs != 8000) || (channels != 1 && channels != 2) ||
        (application != OPUS_APPLICATION_VOIP && application != OPUS_APPLICATION_AUDIO && application != OPUS_APPLICATION_RESTRICTED_LOWDELAY)) {
        if (error) *error = OPUS_BAD_ARG;
        return nullptr;
    }
    OpusEncoder *st = (OpusEncoder *)malloc(sizeof(OpusEncoder));
    if (!st) {
        if (error) *error = OPUS_ALLOC_FAIL;
        return nullptr;
    }
    int ret = opus_encoder_init(st, Fs, channels, application);
    if (error) *error = ret;
    if (ret != OPUS_OK) {
        free(st);
        st = nullptr;
    }
    return st;
}
void opus_encoder_destroy(OpusEncoder *st) {
    if (!st) return;
    {
        std::lock_guard<std::mutex> lk(e.mu);
        if (e.ok && st->magic == kEncMagic) release_slot_locked(st);
    }
    free(st);
}

// opus_encoder_ctl (opus_encoder.c:2031-2507): every supported request carries one opus_int32 or one pointer to it
int opus_encoder_ctl(OpusEncoder *st, int request, ...) {
    va_list ap;
    va_start(ap, request);
    {
        std::lock_guard<std::mutex> lk(e.mu);
        if (!st->host_current) {
            if (!ctx_init_locked()) { va_end(ap); return OPUS_INTERNAL_ERROR; }
            int rc = make_host_current_locked(st);
            if (rc != OPUS_OK) { va_end(ap); return rc; }
        }
    }
    int ret;
    if (request == 10024) {
        // OPUS_SET_LFE (celt.h:113, opus_encoder.c:2455): the multistream encoder's switch for a low-frequency-effects channel.  The
        // default (0) is accepted; the LFE analysis path itself is part of the multistream scope that is not built.
        ret = va_arg(ap, opus_int32) == 0 ? OPUS_OK : OPUS_UNIMPLEMENTED;
    } else if (request == 10026) {
        // OPUS_SET_ENERGY_MASK (celt.h:116, opus_encoder.c:2462): a surround masking curve; only "none" (NULL) is accepted
        ret = va_arg(ap, void *) == nullptr ? OPUS_OK : OPUS_UNIMPLEMENTED;
    } else if (request == OPUS_RESET_STATE) {
        ret = enc_ctl(&st->st, request, 0, nullptr);
    } else if (enc_ctl_is_get(request)) {
        opus_int32 *p = va_arg(ap, opus_int32 *);
        if (!p) ret = OPUS_BAD_ARG;
        else {
            int v = 0;
            ret = enc_ctl(&st->st, request, 0, &v);
            if (ret == OPUS_OK) *p = v;
        }
    } else {
        opus_int32 v = va_arg(ap, opus_int32);
        int dummy = 0;
        ret = enc_ctl(&st->st, request, v, &dummy);
    }
    va_end(ap);
    return ret;
}

// ---- encode ----
int opus_encode_span_device(OpusEncoder **st, int n, int F, const opus_int16 *d_pcm, int frame_size, unsigned char *d_data,
                            opus_int32 max_data_bytes, opus_int32 *d_ret) {
    if (!st || n <= 0 || F <= 0 || frame_size <= 0 || max_data_bytes <= 0) return OPUS_BAD_ARG;
    std::lock_guard<std::mutex> lk(e.mu);
    if (!ctx_init_locked()) return OPUS_INTERNAL_ERROR;
    int rc = check_span(st, n, frame_size);
    if (rc != OPUS_OK) return rc;
    if (!e.h_slots.reserve(sizeof(int) * (size_t)n)) return OPUS_ALLOC_FAIL;
    int *hsl = (int *)e.h_slots.p;
    rc = make_resident_locked(st, n, hsl);
    if (rc != OPUS_OK) return rc;
    SpanSplit sp;
    if (!split_span(st, hsl, n, frame_size, hmin(max_data_bytes, 1276), sp)) return OPUS_ALLOC_FAIL;
    rc = launch_span(sp, d_pcm, d_data, d_ret, F, frame_size, st[0]->st.channels, st[0]->st.Fs, hmin(max_data_bytes, 1276), max_data_bytes);
    if (rc != OPUS_OK) return rc;
    mark_device_newer_locked(st, n);
    if (cudaGetLastError() != cudaSuccess) return OPUS_INTERNAL_ERROR;
    return OPUS_OK;
}

int opus_encode_span(OpusEncoder **st, int n, int F, const opus_int16 *pcm, int frame_size, unsigned char *data, opus_int32 max_data_bytes,
                     opus_int32 *ret) {
    if (!st || n <= 0 || F <= 0 || frame_size <= 0 || max_data_bytes <= 0 || !pcm || !data || !ret) return OPUS_BAD_ARG;
    std::lock_guard<std::mutex> lk(e.mu);
    return encode_span_host_locked(st, n, F, pcm, frame_size, data, hmin(max_data_bytes, 1276), max_data_bytes, ret, true);
}

int opus_encode_span_ranges(OpusEncoder **st, int n, int F, const opus_int16 *pcm, int frame_size, unsigned char *data,
                            opus_int32 max_data_bytes, opus_int32 *ret, opus_uint32 *final_range) {
    if (!st || n <= 0 || F <= 0 || frame_size <= 0 || max_data_bytes <= 0 || !pcm || !data || !ret || !final_range) return OPUS_BAD_ARG;
    std::lock_guard<std::mutex> lk(e.mu);
    return encode_span_host_locked(st, n, F, pcm, frame_size, data, hmin(max_data_bytes, 1276), max_data_bytes, ret, true, final_range);
}

int opus_encode_batch(OpusEncoder **st, const opus_int16 *const *pcm, int frame_size, unsigned char *const *data, opus_int32 max_data_bytes,
                      opus_int32 *ret, int n) {
    if (!st || !pcm || !data || !ret || n <= 0) return OPUS_BAD_ARG;
    if (frame_size <= 0 || max_data_bytes <= 0) {
        for (int i = 0; i < n; i++) ret[i] = OPUS_BAD_ARG;
        return OPUS_OK;
    }
    std::lock_guard<std::mutex> lk(e.mu);
    if (!ctx_init_locked()) return OPUS_INTERNAL_ERROR;
    const int stride = hmin(max_data_bytes, 1276);
    for (int i = 0; i < n; i++)
        if (!st[i] || st[i]->magic != kEncMagic || !pcm[i] || !data[i]) ret[i] = OPUS_BAD_ARG;
    // group by (Fs, channels): the span kernel wants uniform rows
    std::vector<char> done(n, 0);
    for (int i = 0; i < n; i++) {
        if (done[i] || !st[i] || st[i]->magic != kEncMagic || !pcm[i] || !data[i]) continue;
        std::vector<int> idx;
        for (int j = i; j < n; j++)
            if (!done[j] && st[j] && st[j]->magic == kEncMagic && pcm[j] && data[j] && st[j]->st.channels == st[i]->st.channels &&
                st[j]->st.Fs == st[i]->st.Fs) {
                idx.push_back(j);
                done[j] = 1;
            }
        const int m = (int)idx.size(), ch = st[i]->st.channels;
        // OPUS_SET_EXPERT_FRAME_DURATION: the frame actually coded (opus_encode -> compute_frame_size, opus_encoder.c:2007-2025).
        // Streams of one group that select different sizes are launched separately.
        std::vector<int> fsz(m);
        for (int k = 0; k < m; k++) {
            if (!st[idx[k]]->host_current && st[idx[k]]->st.variable_duration != 5000) { /* config never changes on the device */ }
            fsz[k] = frame_size_select(frame_size, st[idx[k]]->st.variable_duration, st[idx[k]]->st.Fs);
        }
        std::vector<char> sub_done(m, 0);
        for (int k0 = 0; k0 < m; k0++) {
            if (sub_done[k0]) continue;
            if (fsz[k0] < 0) { ret[idx[k0]] = OPUS_BAD_ARG; sub_done[k0] = 1; continue; }
            std::vector<int> sub;
            for (int k = k0; k < m; k++)
                if (!sub_done[k] && fsz[k] == fsz[k0]) { sub.push_back(idx[k]); sub_done[k] = 1; }
            const int q = (int)sub.size(), fs = fsz[k0];
            std::vector<OpusEncoder *> sts(q);
            std::vector<int16_t> in((size_t)q * fs * ch);
            std::vector<uint8_t> out((size_t)q * stride);
            std::vector<int> rets(q);
            for (int k = 0; k < q; k++) {
                sts[k] = st[sub[k]];
                memcpy(in.data() + (size_t)k * fs * ch, pcm[sub[k]], (size_t)fs * ch * sizeof(int16_t));
            }
            int rc = encode_span_host_locked(sts.data(), q, 1, in.data(), fs, out.data(), stride, stride, rets.data(), true);
            if (rc != OPUS_OK) return rc;
            for (int k = 0; k < q; k++) {
                ret[sub[k]] = rets[k];
                if (rets[k] > 0) memcpy(data[sub[k]], out.data() + (size_t)k * stride, (size_t)rets[k]);
            }
        }
    }
    return OPUS_OK;
}

int opus_encoder_sync(OpusEncoder **st, int n) {
    if (!st || n <= 0) return OPUS_BAD_ARG;
    std::lock_guard<std::mutex> lk(e.mu);
    if (!ctx_init_locked()) return OPUS_INTERNAL_ERROR;
    return sync_states_locked(st, n, true);
}

// Scalar call = batch of one; the host block is left current so it stays memcpy-able (opus_encoder.c:2007-2025).
opus_int32 opus_encode(OpusEncoder *st, const opus_int16 *pcm, int analysis_frame_size, unsigned char *data, opus_int32 max_data_bytes) {
    if (!st || st->magic != kEncMagic || !pcm || !data) return OPUS_BAD_ARG;
    if (max_data_bytes <= 0) return OPUS_BAD_ARG;
    std::lock_guard<std::mutex> lk(e.mu);
    if (!ctx_init_locked()) return OPUS_INTERNAL_ERROR;
    // the ctl-visible configuration never changes on the device, so a stale host block still holds it
    const int frame_size = frame_size_select(analysis_frame_size, st->st.variable_duration, st->st.Fs);
    if (frame_size < 0) return OPUS_BAD_ARG;
    const int stride = hmin(max_data_bytes, 1276);
    std::vector<uint8_t> out((size_t)stride);
    int r = 0;
    OpusEncoder *one = st;
    int rc = encode_span_host_locked(&one, 1, 1, pcm, frame_size, out.data(), stride, stride, &r, false);
    if (rc != OPUS_OK) return rc;
    if (r > 0) memcpy(data, out.data(), (size_t)r);
    return r;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// Multistream encoder (libopus opus_multistream.h; the encode loop of src/opus_multistream_encoder.c is restated in
// opus_ms_encoder.h).  The block is a header followed by `streams` ordinary OpusEncoder blocks (coupled streams first, stereo;
// then mono), so residency, write-back, memcpy and the duplicate check of the embedded encoders are exactly those of
// single-stream encoders.
// ------------------------------------------------------------------------------------------------
struct OpusMSEncoder {
    uint32_t magic;
    int32_t Fs, channels, streams, coupled, application;
    int32_t bitrate;        // OPUS_SET_BITRATE of the multistream encoder (OPUS_AUTO after init)
    uint8_t mapping[255];   // input channel c feeds stream channel mapping[c]; 255 = ignored
};
static const uint32_t kMsEncMagic = 0x0B2005ECu;
static const size_t kMsEncHeader = (sizeof(OpusMSEncoder) + 63) & ~(size_t)63;

static inline OpusEncoder *ms_enc_stream(OpusMSEncoder *st, int s) {
    return reinterpret_cast<OpusEncoder *>(reinterpret_cast<char *>(st) + kMsEncHeader + (size_t)s * sizeof(OpusEncoder));
}

namespace {

void ms_timing_begin(int stage) {
    EncCtx::Timed t;
    for (cudaEvent_t *ev : {&t.a, &t.b}) {
        if (!e.ms_ev_pool.empty()) { *ev = e.ms_ev_pool.back(); e.ms_ev_pool.pop_back(); }
        else cudaEventCreate(ev);
    }
    t.stage = stage;
    cudaEventRecord(t.a, e.stream);
    e.ms_timed.push_back(t);
}
void ms_timing_end() { cudaEventRecord(e.ms_timed.back().b, e.stream); }
void ms_timing_fold() {   // call only when e.stream is idle
    for (auto &t : e.ms_timed) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, t.a, t.b) == cudaSuccess) { e.ms_stage_ms[t.stage] += ms; e.ms_stage_launches[t.stage]++; }
        e.ms_ev_pool.push_back(t.a);
        e.ms_ev_pool.push_back(t.b);
    }
    e.ms_timed.clear();
}

// Offsets into a call's index upload of one launch's split (see SpanSplit).
struct MsSplit {
    int n_pipe = 0, n_legacy = 0;
    size_t pslots = 0, psidx = 0, lslots = 0, lsidx = 0;
    SpanSplit at(const int *d) const {
        SpanSplit sp;
        sp.n_pipe = n_pipe; sp.n_legacy = n_legacy;
        sp.d_pslots = d + pslots; sp.d_psidx = d + psidx; sp.d_lslots = d + lslots; sp.d_lsidx = d + lsidx;
        return sp;
    }
};
// Appends the split of encoders enc[i] (pool slot slot[i], group row row[i]) to h; allow_pipe = false keeps all of them on the
// one-kernel path (per-frame control).
MsSplit ms_add_split(std::vector<int> &h, const std::vector<OpusEncoder *> &enc, const std::vector<int> &slot, const std::vector<int> &row,
                     bool allow_pipe, int frame_size) {
    std::vector<int> ps, pr, ls, lr;
    for (size_t i = 0; i < enc.size(); i++) {
        if (allow_pipe && e.use_pipe && enc_pipe_takes(&enc[i]->st, frame_size, 1276)) { ps.push_back(slot[i]); pr.push_back(row[i]); }
        else { ls.push_back(slot[i]); lr.push_back(row[i]); }
    }
    MsSplit sp;
    sp.n_pipe = (int)ps.size();
    sp.n_legacy = (int)ls.size();
    sp.pslots = h.size(); h.insert(h.end(), ps.begin(), ps.end());
    sp.psidx = h.size(); h.insert(h.end(), pr.begin(), pr.end());
    sp.lslots = h.size(); h.insert(h.end(), ls.begin(), ls.end());
    sp.lsidx = h.size(); h.insert(h.end(), lr.begin(), lr.end());
    e.pipe_streams += sp.n_pipe;
    e.legacy_streams += sp.n_legacy;
    return sp;
}

// Multistream span over host or device buffers (device_io): n encoders sharing (Fs, channels, streams, coupled); input frame (m,f)
// at pcm + (m*F+f)*frame_size*channels, its packet at data + (m*F+f)*max_data_bytes, ret[m*F+f] = what the scalar call returns.
//
// Two schedules (DESIGN.md §3).  Merged: when every embedded encoder is OPUS_APPLICATION_RESTRICTED_LOWDELAY and VBR / CVBR and
// max_data_bytes >= 1278·S − 2, every stream's budget is the single-stream clamp of 1276 whatever the earlier streams took and no
// stream can fail, so all coupled streams are coded in one launch, all mono streams in another, and the packets are framed after.
// Ordered (everything else): S passes by stream index, each preceded by ms_budget_kernel and followed by ms_pack_kernel, which
// reproduces the budgets, the CBR bitrate of the last stream and the stop at the first failing stream exactly.
int ms_encode_span_locked(OpusMSEncoder **st, int n, int F, const int16_t *pcm, int frame_size, uint8_t *data, int max_data_bytes, int *ret,
                          bool device_io, bool keep_resident) {
    for (int m = 0; m < n; m++) {
        if (!st[m] || st[m]->magic != kMsEncMagic) return OPUS_BAD_ARG;
        if (st[m]->Fs != st[0]->Fs || st[m]->channels != st[0]->channels || st[m]->streams != st[0]->streams || st[m]->coupled != st[0]->coupled)
            return OPUS_BAD_ARG;
    }
    const int Fs = st[0]->Fs, channels = st[0]->channels, S = st[0]->streams, cpl = st[0]->coupled, mono = S - cpl;
    const int E = n * S, K = S + cpl;
    // embedded encoders in group order: the coupled group (row m*cpl+s), then the mono group (row m*mono+j)
    std::vector<OpusEncoder *> el((size_t)E);
    for (int m = 0; m < n; m++)
        for (int s = 0; s < S; s++) el[s < cpl ? (size_t)m * cpl + s : (size_t)n * cpl + (size_t)m * mono + (s - cpl)] = ms_enc_stream(st[m], s);
    auto el_of = [&](int m, int s) { return s < cpl ? (size_t)m * cpl + s : (size_t)n * cpl + (size_t)m * mono + (s - cpl); };
    // the ctl-visible configuration never changes on the device, so a stale host block still holds it
    for (int i = 0; i < E; i++)
        if (frame_size_select(frame_size, el[i]->st.variable_duration, Fs) != frame_size) return OPUS_BAD_ARG;
    if (max_data_bytes < ms_enc_min_bytes(S)) return OPUS_BUFFER_TOO_SMALL;
    if (!ctx_init_locked()) return OPUS_INTERNAL_ERROR;
    if (!e.h_slots.reserve(sizeof(int) * (size_t)E)) return OPUS_ALLOC_FAIL;
    int *hsl = (int *)e.h_slots.p;
    int rc = make_resident_locked(el.data(), E, hsl);
    if (rc != OPUS_OK) return rc;

    // per-encoder parameters, the rate allocation applied to every stream (host block and, where it changes, the resident slot)
    std::vector<int> h((size_t)n * 4 + (size_t)n * K);
    std::vector<int> pairs;
    std::vector<int32_t> rate((size_t)S);
    bool merged = max_data_bytes >= 1278 * S - 2, any_cbr = false;
    for (int m = 0; m < n; m++) {
        ms_rate_allocation(st[m]->bitrate, channels, S, cpl, Fs, frame_size, rate.data());
        const int cbr = !ms_enc_stream(st[m], 0)->st.use_vbr;
        any_cbr |= cbr != 0;
        h[(size_t)m * 4 + 0] = cbr ? ms_cbr_max_bytes(max_data_bytes, st[m]->bitrate, Fs, frame_size) : max_data_bytes;
        h[(size_t)m * 4 + 1] = cbr;
        h[(size_t)m * 4 + 2] = rate[S - 1];
        h[(size_t)m * 4 + 3] = 0;
        for (int k = 0; k < K; k++) h[(size_t)n * 4 + (size_t)m * K + k] = ms_enc_source_channel(st[m]->mapping, channels, k);
        for (int s = 0; s < S; s++) {
            const size_t i = el_of(m, s);
            CbEncState &es = el[i]->st;
            const int before = es.user_bitrate_bps;
            int unused;
            enc_ctl(&es, 4002, rate[s], &unused);
            if (es.user_bitrate_bps != before) { pairs.push_back(hsl[i]); pairs.push_back(es.user_bitrate_bps); }
            if (es.application != kAppLowdelay || !es.use_vbr) merged = false;
        }
    }
    const size_t off_pairs = h.size();
    h.insert(h.end(), pairs.begin(), pairs.end());
    std::vector<MsSplit> splits;
    {
        std::vector<OpusEncoder *> enc;
        std::vector<int> slot, row;
        auto group = [&](int s0, int s1) {   // streams [s0, s1) of every encoder
            enc.clear(); slot.clear(); row.clear();
            for (int m = 0; m < n; m++)
                for (int s = s0; s < s1; s++) {
                    const size_t i = el_of(m, s);
                    enc.push_back(el[i]); slot.push_back(hsl[i]);
                    row.push_back(s < cpl ? m * cpl + s : m * mono + s - cpl);
                }
        };
        if (merged) {
            group(0, cpl); splits.push_back(ms_add_split(h, enc, slot, row, true, frame_size));
            group(cpl, S); splits.push_back(ms_add_split(h, enc, slot, row, true, frame_size));
        } else {
            for (int s = 0; s < S; s++) { group(s, s + 1); splits.push_back(ms_add_split(h, enc, slot, row, false, frame_size)); }
        }
    }
    const size_t NF = (size_t)n * F;
    const size_t st_rows = (size_t)n * cpl * F, mono_rows = (size_t)n * mono * F;
    if (!e.d_ms_idx.reserve(sizeof(int) * h.size()) || !e.d_ms_pcm[0].reserve(st_rows * frame_size * 2 * sizeof(int16_t) + 16) ||
        !e.d_ms_pcm[1].reserve(mono_rows * frame_size * sizeof(int16_t) + 16) || !e.d_ms_pkt.reserve((st_rows + mono_rows) * 1276) ||
        !e.d_ms_rets.reserve(sizeof(int) * (st_rows + mono_rows)) || !e.d_ms_tot.reserve(sizeof(int) * NF) || !e.d_ms_err.reserve(sizeof(int) * NF) ||
        (!merged && !e.d_ms_ctl.reserve(sizeof(int4) * (st_rows + mono_rows))))
        return OPUS_ALLOC_FAIL;
    const size_t pcm_bytes = NF * frame_size * channels * sizeof(int16_t);
    if (!device_io && (!e.d_pcm.reserve(pcm_bytes) || !e.d_data.reserve(NF * (size_t)max_data_bytes) || !e.d_rets.reserve(sizeof(int) * NF)))
        return OPUS_ALLOC_FAIL;
    PinBuf &hb = e.h_ms[e.ms_seq++ & 3];   // an earlier call's upload may still be in flight
    if (!hb.reserve(sizeof(int) * h.size())) return OPUS_ALLOC_FAIL;
    memcpy(hb.p, h.data(), sizeof(int) * h.size());
    const int *d_idx = (const int *)e.d_ms_idx.p;
    const int4 *d_prm = (const int4 *)d_idx;
    int16_t *st_pcm = (int16_t *)e.d_ms_pcm[0].p, *mono_pcm = (int16_t *)e.d_ms_pcm[1].p;
    uint8_t *pkt_st = (uint8_t *)e.d_ms_pkt.p, *pkt_mono = pkt_st + st_rows * 1276;
    int *rets_st = (int *)e.d_ms_rets.p, *rets_mono = rets_st + st_rows;
    int4 *ctl_st = (int4 *)e.d_ms_ctl.p, *ctl_mono = ctl_st + st_rows;
    int *tot = (int *)e.d_ms_tot.p, *err = (int *)e.d_ms_err.p;
    const int16_t *d_pcm = device_io ? pcm : (const int16_t *)e.d_pcm.p;
    uint8_t *d_data = device_io ? data : (uint8_t *)e.d_data.p;
    int *d_ret = device_io ? ret : (int *)e.d_rets.p;

    if (!device_io) cudaMemcpyAsync(e.d_pcm.p, pcm, pcm_bytes, cudaMemcpyHostToDevice, e.stream);
    cudaEventRecord(e.ev0, e.stream);
    cudaMemcpyAsync(e.d_ms_idx.p, hb.p, sizeof(int) * h.size(), cudaMemcpyHostToDevice, e.stream);
    const int npairs = (int)(pairs.size() / 2);
    if (npairs > 0) {
        ms_set_bitrate_kernel<<<(npairs + 127) / 128, 128, 0, e.stream>>>(e.pool, d_idx + off_pairs, npairs);
        e.launches++;
    }
    cudaMemsetAsync(tot, 0, sizeof(int) * NF, e.stream);
    cudaMemsetAsync(err, 0, sizeof(int) * NF, e.stream);
    ms_timing_begin(0);
    ms_route_kernel<<<(unsigned)NF, 256, 0, e.stream>>>(d_pcm, d_idx + (size_t)n * 4, F, channels, frame_size, S, cpl, st_pcm, mono_pcm);
    ms_timing_end();
    e.launches++;
    const unsigned pk_blocks = (unsigned)((NF + 127) / 128);
    if (merged) {
        if (cpl > 0) rc = launch_frames(splits[0].at(d_idx), st_pcm, pkt_st, rets_st, F, 0, F, frame_size, 2, Fs, 1276, 1276);
        if (rc == OPUS_OK && mono > 0) rc = launch_frames(splits[1].at(d_idx), mono_pcm, pkt_mono, rets_mono, F, 0, F, frame_size, 1, Fs, 1276, 1276);
        if (rc != OPUS_OK) return rc;
        ms_timing_begin(2);
        ms_pack_kernel<<<pk_blocks, 128, 0, e.stream>>>(d_prm, pkt_st, pkt_mono, rets_st, rets_mono, 1276, n, F, S, cpl, 0, S, d_data,
                                                        max_data_bytes, tot, err, d_ret, 1);
        ms_timing_end();
        e.launches++;
    } else {
        for (int s = 0; s < S; s++) {
            ms_timing_begin(1);
            ms_budget_kernel<<<pk_blocks, 128, 0, e.stream>>>(d_prm, tot, err, n, F, S, cpl, s, Fs, frame_size, s < cpl ? ctl_st : ctl_mono);
            ms_timing_end();
            rc = s < cpl ? launch_frames(splits[s].at(d_idx), st_pcm, pkt_st, rets_st, F, 0, F, frame_size, 2, Fs, 1276, 1276, nullptr, ctl_st)
                         : launch_frames(splits[s].at(d_idx), mono_pcm, pkt_mono, rets_mono, F, 0, F, frame_size, 1, Fs, 1276, 1276, nullptr, ctl_mono);
            if (rc != OPUS_OK) return rc;
            ms_timing_begin(2);
            ms_pack_kernel<<<pk_blocks, 128, 0, e.stream>>>(d_prm, pkt_st, pkt_mono, rets_st, rets_mono, 1276, n, F, S, cpl, s, s + 1, d_data,
                                                            max_data_bytes, tot, err, d_ret, s == S - 1);
            ms_timing_end();
            e.launches += 2;
        }
    }
    cudaEventRecord(e.ev1, e.stream);
    mark_device_newer_locked(el.data(), E);
    if (!merged && any_cbr) {
        // CBR changed the last stream's bitrate frame by frame on the device: the host block takes the value its last frame left
        const int4 *src = (S - 1 < cpl ? ctl_st + (size_t)(S - 1) * F : ctl_mono + (size_t)(mono - 1) * F);
        const size_t pitch = (size_t)(S - 1 < cpl ? cpl : mono) * F * sizeof(int4);
        if (!e.h_ms_ctl.reserve(NF * sizeof(int4))) return OPUS_ALLOC_FAIL;
        cudaMemcpy2DAsync(e.h_ms_ctl.p, (size_t)F * sizeof(int4), src, pitch, (size_t)F * sizeof(int4), (size_t)n, cudaMemcpyDeviceToHost, e.stream);
        if (cudaStreamSynchronize(e.stream) != cudaSuccess) return OPUS_INTERNAL_ERROR;
        const int4 *c = (const int4 *)e.h_ms_ctl.p;
        for (int m = 0; m < n; m++) {
            if (!h[(size_t)m * 4 + 1]) continue;
            CbEncState &es = el[el_of(m, S - 1)]->st;
            int unused;
            for (int f = 0; f < F; f++) {
                enc_ctl(&es, 4002, c[(size_t)m * F + f].y, &unused);
                enc_ctl(&es, 4002, c[(size_t)m * F + f].z, &unused);
            }
        }
    }
    if (device_io) {
        if (e.ms_timed.size() > 4096 && cudaStreamSynchronize(e.stream) == cudaSuccess) ms_timing_fold();
        return cudaGetLastError() == cudaSuccess ? OPUS_OK : OPUS_INTERNAL_ERROR;
    }
    cudaMemcpyAsync(data, e.d_data.p, NF * (size_t)max_data_bytes, cudaMemcpyDeviceToHost, e.stream);
    cudaMemcpyAsync(ret, e.d_rets.p, sizeof(int) * NF, cudaMemcpyDeviceToHost, e.stream);
    if (cudaStreamSynchronize(e.stream) != cudaSuccess) {
        fprintf(stderr, "concentus_b200: CUDA failure in multistream encode: %s\n", cudaGetErrorString(cudaGetLastError()));
        return OPUS_INTERNAL_ERROR;
    }
    cudaEventElapsedTime(&e.last_ms, e.ev0, e.ev1);
    e.total_ms += e.last_ms;
    ms_timing_fold();
    if (!keep_resident) return sync_states_locked(el.data(), E, true);
    return OPUS_OK;
}

int ms_check_args(int channels, int streams, int coupled) {
    return (channels > 255 || channels < 1 || coupled > streams || streams < 1 || coupled < 0 || streams > 255 - coupled) ? OPUS_BAD_ARG : OPUS_OK;
}

}  // namespace

extern "C" {

int opus_multistream_encoder_get_size(int streams, int coupled_streams) {
    if (streams < 1 || coupled_streams > streams || coupled_streams < 0) return 0;
    return (int)(kMsEncHeader + (size_t)streams * sizeof(OpusEncoder));
}

int opus_multistream_encoder_init(OpusMSEncoder *st, opus_int32 Fs, int channels, int streams, int coupled_streams, const unsigned char *mapping,
                                  int application) {
    if (ms_check_args(channels, streams, coupled_streams) != OPUS_OK || !mapping) return OPUS_BAD_ARG;
    if (ms_enc_check_layout(channels, streams, coupled_streams, mapping) != 0) return OPUS_BAD_ARG;
    // re-initialising a live block in place: the embedded encoders give their pool slots back (opus_encoder_init)
    const bool live = st->magic == kMsEncMagic;
    const int old_streams = live ? st->streams : 0;
    if (live && old_streams > streams) {
        std::lock_guard<std::mutex> lk(e.mu);
        for (int s = streams; s < old_streams; s++) {
            OpusEncoder *d = ms_enc_stream(st, s);
            if (e.ok && d->magic == kEncMagic && d->slot >= 0) release_slot_locked(d);
        }
    }
    st->magic = 0;
    for (int s = 0; s < streams; s++) {
        OpusEncoder *d = ms_enc_stream(st, s);
        if (!(live && s < old_streams)) d->magic = 0;   // not a live encoder: nothing to release
        const int ret = opus_encoder_init(d, Fs, s < coupled_streams ? 2 : 1, application);
        if (ret != OPUS_OK) return ret;
    }
    st->magic = kMsEncMagic;
    st->Fs = Fs;
    st->channels = channels;
    st->streams = streams;
    st->coupled = coupled_streams;
    st->application = application;
    st->bitrate = OPUS_AUTO;
    memset(st->mapping, 255, sizeof(st->mapping));
    memcpy(st->mapping, mapping, (size_t)channels);
    return OPUS_OK;
}

OpusMSEncoder *opus_multistream_encoder_create(opus_int32 Fs, int channels, int streams, int coupled_streams, const unsigned char *mapping,
                                               int application, int *error) {
    if (ms_check_args(channels, streams, coupled_streams) != OPUS_OK) {
        if (error) *error = OPUS_BAD_ARG;
        return nullptr;
    }
    OpusMSEncoder *st = (OpusMSEncoder *)malloc((size_t)opus_multistream_encoder_get_size(streams, coupled_streams));
    if (!st) {
        if (error) *error = OPUS_ALLOC_FAIL;
        return nullptr;
    }
    st->magic = 0;
    const int ret = opus_multistream_encoder_init(st, Fs, channels, streams, coupled_streams, mapping, application);
    if (error) *error = ret;
    if (ret != OPUS_OK) {
        opus_multistream_encoder_destroy(st);
        st = nullptr;
    }
    return st;
}

void opus_multistream_encoder_destroy(OpusMSEncoder *st) {
    if (!st) return;
    if (st->magic == kMsEncMagic) {
        std::lock_guard<std::mutex> lk(e.mu);
        if (e.ok)
            for (int s = 0; s < st->streams; s++) {
                OpusEncoder *d = ms_enc_stream(st, s);
                if (d->magic == kEncMagic) release_slot_locked(d);
            }
    }
    free(st);
}

opus_int32 opus_multistream_surround_encoder_get_size(int channels, int mapping_family) {
    int streams = 0, coupled = 0;
    uint8_t mapping[255];
    if (ms_surround_layout(channels, mapping_family, &streams, &coupled, mapping) != 0) return 0;
    return opus_multistream_encoder_get_size(streams, coupled);
}

int opus_multistream_surround_encoder_init(OpusMSEncoder *st, opus_int32 Fs, int channels, int mapping_family, int *streams, int *coupled_streams,
                                           unsigned char *mapping, int application) {
    if (!streams || !coupled_streams || !mapping) return OPUS_BAD_ARG;
    const int rc = ms_surround_layout(channels, mapping_family, streams, coupled_streams, mapping);
    if (rc != 0) return rc;
    return opus_multistream_encoder_init(st, Fs, channels, *streams, *coupled_streams, mapping, application);
}

OpusMSEncoder *opus_multistream_surround_encoder_create(opus_int32 Fs, int channels, int mapping_family, int *streams, int *coupled_streams,
                                                       unsigned char *mapping, int application, int *error) {
    const int size = opus_multistream_surround_encoder_get_size(channels, mapping_family);
    if (!size || !streams || !coupled_streams || !mapping) {
        if (error) *error = (channels > 255 || channels < 1 || !streams || !coupled_streams || !mapping) ? OPUS_BAD_ARG : OPUS_UNIMPLEMENTED;
        return nullptr;
    }
    OpusMSEncoder *st = (OpusMSEncoder *)malloc((size_t)size);
    if (!st) {
        if (error) *error = OPUS_ALLOC_FAIL;
        return nullptr;
    }
    st->magic = 0;
    const int ret = opus_multistream_surround_encoder_init(st, Fs, channels, mapping_family, streams, coupled_streams, mapping, application);
    if (error) *error = ret;
    if (ret != OPUS_OK) {
        opus_multistream_encoder_destroy(st);
        st = nullptr;
    }
    return st;
}

// opus_multistream_encoder_ctl (opus_multistream_encoder.c): the multistream bitrate is the encoder's own; OPUS_GET_BITRATE sums
// the streams' bitrates, OPUS_GET_FINAL_RANGE XORs their final ranges; reset and the other SETs go to every stream (stopping at
// the first error), the other GETs are answered by stream 0.
int opus_multistream_encoder_ctl(OpusMSEncoder *st, int request, ...) {
    if (!st || st->magic != kMsEncMagic) return OPUS_BAD_ARG;
    int ret = OPUS_OK;
    va_list ap;
    va_start(ap, request);
    switch (request) {
    case OPUS_SET_BITRATE_REQUEST: {
        const opus_int32 v = va_arg(ap, opus_int32);
        if (v < 0 && v != OPUS_AUTO && v != OPUS_BITRATE_MAX) { ret = OPUS_BAD_ARG; break; }
        st->bitrate = v;
    } break;
    case OPUS_GET_BITRATE_REQUEST:
    case OPUS_GET_FINAL_RANGE_REQUEST: {
        opus_int32 *v = va_arg(ap, opus_int32 *);
        if (!v) { ret = OPUS_BAD_ARG; break; }
        opus_int32 acc = 0, r = 0;
        for (int s = 0; s < st->streams && ret == OPUS_OK; s++) {
            ret = opus_encoder_ctl(ms_enc_stream(st, s), request, &r);
            acc = request == OPUS_GET_BITRATE_REQUEST ? acc + r : (opus_int32)((opus_uint32)acc ^ (opus_uint32)r);
        }
        if (ret == OPUS_OK) *v = acc;
    } break;
    case OPUS_GET_LSB_DEPTH_REQUEST: case OPUS_GET_VBR_REQUEST: case OPUS_GET_APPLICATION_REQUEST: case OPUS_GET_BANDWIDTH_REQUEST:
    case OPUS_GET_VBR_CONSTRAINT_REQUEST: case OPUS_GET_COMPLEXITY_REQUEST: case OPUS_GET_PACKET_LOSS_PERC_REQUEST: case OPUS_GET_DTX_REQUEST:
    case OPUS_GET_SIGNAL_REQUEST: case OPUS_GET_LOOKAHEAD_REQUEST: case OPUS_GET_SAMPLE_RATE_REQUEST:
    case OPUS_GET_INBAND_FEC_REQUEST: case OPUS_GET_FORCE_CHANNELS_REQUEST: case OPUS_GET_PREDICTION_DISABLED_REQUEST:
    case OPUS_GET_EXPERT_FRAME_DURATION_REQUEST: {
        opus_int32 *v = va_arg(ap, opus_int32 *);
        ret = opus_encoder_ctl(ms_enc_stream(st, 0), request, v);
    } break;
    case OPUS_SET_LSB_DEPTH_REQUEST: case OPUS_SET_COMPLEXITY_REQUEST: case OPUS_SET_VBR_REQUEST: case OPUS_SET_VBR_CONSTRAINT_REQUEST:
    case OPUS_SET_MAX_BANDWIDTH_REQUEST: case OPUS_SET_BANDWIDTH_REQUEST: case OPUS_SET_SIGNAL_REQUEST: case OPUS_SET_APPLICATION_REQUEST:
    case OPUS_SET_INBAND_FEC_REQUEST: case OPUS_SET_PACKET_LOSS_PERC_REQUEST: case OPUS_SET_DTX_REQUEST: case OPUS_SET_FORCE_MODE_REQUEST:
    case OPUS_SET_FORCE_CHANNELS_REQUEST: case OPUS_SET_PREDICTION_DISABLED_REQUEST: case OPUS_SET_EXPERT_FRAME_DURATION_REQUEST: {
        const opus_int32 v = va_arg(ap, opus_int32);
        for (int s = 0; s < st->streams && ret == OPUS_OK; s++) ret = opus_encoder_ctl(ms_enc_stream(st, s), request, v);
    } break;
    case OPUS_RESET_STATE:
        for (int s = 0; s < st->streams && ret == OPUS_OK; s++) ret = opus_encoder_ctl(ms_enc_stream(st, s), OPUS_RESET_STATE);
        break;
    case OPUS_MULTISTREAM_GET_ENCODER_STATE_REQUEST: {
        const opus_int32 id = va_arg(ap, opus_int32);
        OpusEncoder **v = va_arg(ap, OpusEncoder **);
        if (id < 0 || id >= st->streams || !v) { ret = OPUS_BAD_ARG; break; }
        *v = ms_enc_stream(st, id);
    } break;
    default:
        ret = OPUS_UNIMPLEMENTED;
        break;
    }
    va_end(ap);
    return ret;
}

int opus_multistream_encode_span(OpusMSEncoder **st, int n, int F, const opus_int16 *pcm, int frame_size, unsigned char *data,
                                 opus_int32 max_data_bytes, opus_int32 *ret) {
    if (!st || n <= 0 || F <= 0 || frame_size <= 0 || max_data_bytes <= 0 || !pcm || !data || !ret) return OPUS_BAD_ARG;
    std::lock_guard<std::mutex> lk(e.mu);
    return ms_encode_span_locked(st, n, F, pcm, frame_size, data, max_data_bytes, ret, false, true);
}

int opus_multistream_encode_span_device(OpusMSEncoder **st, int n, int F, const opus_int16 *d_pcm, int frame_size, unsigned char *d_data,
                                        opus_int32 max_data_bytes, opus_int32 *d_ret) {
    if (!st || n <= 0 || F <= 0 || frame_size <= 0 || max_data_bytes <= 0) return OPUS_BAD_ARG;
    std::lock_guard<std::mutex> lk(e.mu);
    return ms_encode_span_locked(st, n, F, d_pcm, frame_size, d_data, max_data_bytes, d_ret, true, true);
}

int opus_multistream_encoder_sync(OpusMSEncoder **st, int n) {
    if (!st || n <= 0) return OPUS_BAD_ARG;
    std::vector<OpusEncoder *> el;
    for (int m = 0; m < n; m++) {
        if (!st[m] || st[m]->magic != kMsEncMagic) return OPUS_BAD_ARG;
        for (int s = 0; s < st[m]->streams; s++) el.push_back(ms_enc_stream(st[m], s));
    }
    std::lock_guard<std::mutex> lk(e.mu);
    if (!ctx_init_locked()) return OPUS_INTERNAL_ERROR;
    return sync_states_locked(el.data(), (int)el.size(), true);
}

// Scalar call = span of one; the embedded blocks are left current (write-back) so the encoder stays memcpy-able.
opus_int32 opus_multistream_encode(OpusMSEncoder *st, const opus_int16 *pcm, int frame_size, unsigned char *data, opus_int32 max_data_bytes) {
    if (!st || st->magic != kMsEncMagic || !pcm || !data || frame_size <= 0 || max_data_bytes <= 0) return OPUS_BAD_ARG;
    std::lock_guard<std::mutex> lk(e.mu);
    std::vector<uint8_t> out((size_t)max_data_bytes);
    int r = 0;
    OpusMSEncoder *one = st;
    const int rc = ms_encode_span_locked(&one, 1, 1, pcm, frame_size, out.data(), max_data_bytes, &r, false, false);
    if (rc != OPUS_OK) return rc;
    if (r > 0) memcpy(data, out.data(), (size_t)r);
    return r;
}

// Device time of the multistream encoder's own kernels (0 route, 1 budget, 2 pack) in ms and launches, since the last reset.
int opus_b200_ms_enc_stage_times(double ms[3], long long launches[3], int reset) {
    std::lock_guard<std::mutex> lk(e.mu);
    if (e.ok) {
        if (cudaStreamSynchronize(e.stream) != cudaSuccess) return OPUS_INTERNAL_ERROR;
        ms_timing_fold();
    }
    for (int i = 0; i < 3; i++) {
        if (ms) ms[i] = e.ms_stage_ms[i];
        if (launches) launches[i] = e.ms_stage_launches[i];
        if (reset) { e.ms_stage_ms[i] = 0; e.ms_stage_launches[i] = 0; }
    }
    return OPUS_OK;
}

}  // extern "C"
