// Waveform ingest on the device: what ``Nomad.load_processing`` (reference nomad.py:192-212) does on the host
// between ``torchaudio.load`` and the model -- samples -> float (U8, S16, S24, S32, F32 or F64, decoded exactly as the
// host path ``audio.load_wav`` does, see include/nomad_b200.h), mean of the first two channels when the file has more
// than one (nomad.py:199-200), ``torchaudio.transforms.Resample(sr, 16000)`` when the rates differ (nomad.py:203-205;
// torchaudio's default sinc-Hann kernel, lowpass_filter_width 6, rolloff 0.99), optional trim to 10 s (nomad.py:208-210).
// The bytes that cross PCIe are the file's own data bytes at the file's own rate.
//
// Resampling follows torchaudio/functional/functional.py (_get_sinc_resample_kernel / _apply_sinc_resample_kernel):
// with o = sr / gcd, n = target / gcd, width = ceil(6 o / (0.99 min(o, n))), K = 2 width + o, output sample
// j = m n + p is  sum_k h[p][k] xpad[m o + k],  xpad = x padded by `width` zeros on the left.  The table h is built
// on the host in float64 exactly as torchaudio builds it (including the float32 rounding of -p / n that its
// int64-arange / int division produces) and cast to float32.
//
// A batch of files takes one launch for the items already at the target rate and one per distinct other rate: every
// block of a launch works on 256 consecutive output samples of one item, found through a block -> item map that
// travels with the descriptor table into the caller's workspace.
#include <array>
#include <cmath>
#include <cstring>
#include <map>
#include <mutex>
#include <vector>

#include "../../include/nomad_b200.h"
#include "common.cuh"

namespace nb {

struct ResampleTable {
    int o = 0, n = 0, width = 0, K = 0;
    float* dev = nullptr;  // [n][K]
    int2* range = nullptr; // [n]: first and one-past-last tap of phase p that is not (numerically) zero
};

static long long gcd_ll(long long a, long long b) {
    while (b) {
        const long long t = a % b;
        a = b;
        b = t;
    }
    return a;
}

static int get_table(int sr, int target, ResampleTable* out) {
    static std::mutex mu;
    static std::map<std::pair<int, long long>, ResampleTable> cache;  // per (device, rates)
    int dev = 0;
    NB_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(mu);
    const std::pair<int, long long> key(dev, ((long long)sr << 32) | (unsigned)target);
    auto it = cache.find(key);
    if (it != cache.end()) {
        *out = it->second;
        return 0;
    }
    const long long g = gcd_ll(sr, target);
    ResampleTable t;
    t.o = (int)(sr / g);
    t.n = (int)(target / g);
    const double lpw = 6.0, rolloff = 0.99;
    const double base = (double)(t.o < t.n ? t.o : t.n) * rolloff;
    t.width = (int)std::ceil(lpw * t.o / base);
    t.K = 2 * t.width + t.o;
    NB_CHECK((long long)t.n * t.K < (1LL << 26), "resample %d -> %d Hz needs a %d x %d filter bank: unsupported rate pair", sr,
             target, t.n, t.K);
    std::vector<float> h((size_t)t.n * t.K);
    const double scale = base / t.o;
    for (int p = 0; p < t.n; ++p) {
        const double tp = (double)(float)((double)(-p) / (double)t.n);  // torch: int64 arange / int -> float32
        for (int k = 0; k < t.K; ++k) {
            double tt = (tp + (double)(k - t.width) / (double)t.o) * base;
            tt = tt < -lpw ? -lpw : (tt > lpw ? lpw : tt);
            const double c = std::cos(tt * M_PI / lpw / 2.0);
            const double window = c * c;
            tt *= M_PI;
            const double s = tt == 0.0 ? 1.0 : std::sin(tt) / tt;
            h[(size_t)p * t.K + k] = (float)(s * window * scale);
        }
    }
    // Outside |t| < 6 the Hann window is cos^2(pi / 2): ~1e-33 in float64, never visible in an fp32 sum.  For
    // 44.1 kHz that leaves ~34 live taps of 475 per phase.
    std::vector<int2> rng(t.n);
    for (int p = 0; p < t.n; ++p) {
        int lo = 0, hi = t.K;
        while (lo < hi && std::fabs(h[(size_t)p * t.K + lo]) < 1e-30f) ++lo;
        while (hi > lo && std::fabs(h[(size_t)p * t.K + hi - 1]) < 1e-30f) --hi;
        rng[p] = make_int2(lo, hi);
    }
    NB_CUDA(cudaMalloc((void**)&t.dev, h.size() * sizeof(float)));
    NB_CUDA(cudaMemcpy(t.dev, h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice));
    NB_CUDA(cudaMalloc((void**)&t.range, rng.size() * sizeof(int2)));
    NB_CUDA(cudaMemcpy(t.range, rng.data(), rng.size() * sizeof(int2), cudaMemcpyHostToDevice));
    cache[key] = t;
    *out = t;
    return 0;
}

// One item of a launch as the kernels see it: pointers already offset, block0 = its first block in the launch's grid.
struct DevItem {
    const unsigned char* src;
    float* out;
    long long n_in, n_out;
    int channels, format, block0, pad;
};

// The items of one launch: a device table plus a block -> item map, or (one-item calls) the item itself.
struct ItemTable {
    const DevItem* items;    // nullptr: `one` is the only item
    const int* block_item;   // [gridDim.x] index into items
    DevItem one;
};

__device__ __forceinline__ DevItem item_of_block(const ItemTable& t, long long* blk) {
    if (t.items == nullptr) {
        *blk = blockIdx.x;
        return t.one;
    }
    const DevItem it = t.items[__ldg(t.block_item + blockIdx.x)];
    *blk = (long long)blockIdx.x - it.block0;
    return it;
}

// sample s (frame * channels + channel) of the raw data bytes p, as audio.load_wav decodes it; every case is exact in
// fp32 or the single round-to-nearest numpy does
template <int FMT>
__device__ __forceinline__ float decode(const unsigned char* __restrict__ p, long long s) {
    if constexpr (FMT == NOMAD_B200_WAV_U8) {
        return (float)((int)p[s] - 128) * (1.0f / 128.0f);
    } else if constexpr (FMT == NOMAD_B200_WAV_S16) {
        return (float)reinterpret_cast<const int16_t*>(p)[s] * (1.0f / 32768.0f);
    } else if constexpr (FMT == NOMAD_B200_WAV_S24) {
        const unsigned char* q = p + 3 * s;
        const int v = (int)(((unsigned)q[0] | ((unsigned)q[1] << 8) | ((unsigned)q[2] << 16)) << 8) >> 8;
        return (float)v * (1.0f / 8388608.0f);
    } else if constexpr (FMT == NOMAD_B200_WAV_S32) {
        return __int2float_rn(reinterpret_cast<const int*>(p)[s]) * (1.0f / 2147483648.0f);
    } else if constexpr (FMT == NOMAD_B200_WAV_F32) {
        return reinterpret_cast<const float*>(p)[s];
    } else {
        return __double2float_rn(reinterpret_cast<const double*>(p)[s]);
    }
}

// mono frame i: one channel as is, more: (ch0 + ch1) * 0.5 in fp32 (nomad.py:199-200)
template <int FMT>
__device__ __forceinline__ float mono(const unsigned char* __restrict__ p, long long i, int channels) {
    const long long s = i * channels;
    return channels == 1 ? decode<FMT>(p, s) : (decode<FMT>(p, s) + decode<FMT>(p, s + 1)) * 0.5f;
}

template <int FMT>
__device__ __forceinline__ void to_mono_item(const DevItem& it, long long i) {
    it.out[i] = mono<FMT>(it.src, i, it.channels);
}

// items already at the target rate: one output sample per thread
__global__ void __launch_bounds__(256) to_mono_kernel(const ItemTable tab) {
    long long blk;
    const DevItem it = item_of_block(tab, &blk);
    const long long i = blk * 256 + threadIdx.x;
    if (i >= it.n_out) return;
    switch (it.format) {
        case NOMAD_B200_WAV_U8: to_mono_item<NOMAD_B200_WAV_U8>(it, i); break;
        case NOMAD_B200_WAV_S16: to_mono_item<NOMAD_B200_WAV_S16>(it, i); break;
        case NOMAD_B200_WAV_S24: to_mono_item<NOMAD_B200_WAV_S24>(it, i); break;
        case NOMAD_B200_WAV_S32: to_mono_item<NOMAD_B200_WAV_S32>(it, i); break;
        case NOMAD_B200_WAV_F32: to_mono_item<NOMAD_B200_WAV_F32>(it, i); break;
        default: to_mono_item<NOMAD_B200_WAV_F64>(it, i); break;
    }
}

template <int FMT>
__device__ __forceinline__ void stage_window(const DevItem& it, long long first, int win, float* xs) {
    for (int i = threadIdx.x; i < win; i += 256) {
        const long long s = first + i;
        xs[i] = (s >= 0 && s < it.n_in) ? mono<FMT>(it.src, s, it.channels) : 0.f;
    }
}

// One block = 256 consecutive output samples of one item.  The input window they need is staged in shared memory as
// mono float (decoded once per block); each thread then runs its phase's K taps over it.  All items of a launch share
// the source rate (and so the filter bank).
__global__ void __launch_bounds__(256) resample_kernel(const ItemTable tab, const float* __restrict__ h,
                                                       const int2* __restrict__ range, int o, int n, int width, int K,
                                                       int win_cap) {
    extern __shared__ float xs[];
    long long blk;
    const DevItem it = item_of_block(tab, &blk);
    const long long n_out = it.n_out;
    const long long j0 = blk * 256;
    const long long m0 = j0 / n;                                  // first input group of the block
    const long long j_last = min(j0 + 255, n_out - 1);
    const long long m1 = j_last / n;
    const long long first = m0 * o - width;                        // input index of xs[0]
    const int win = (int)min((m1 - m0) * o + K, (long long)win_cap);
    switch (it.format) {
        case NOMAD_B200_WAV_U8: stage_window<NOMAD_B200_WAV_U8>(it, first, win, xs); break;
        case NOMAD_B200_WAV_S16: stage_window<NOMAD_B200_WAV_S16>(it, first, win, xs); break;
        case NOMAD_B200_WAV_S24: stage_window<NOMAD_B200_WAV_S24>(it, first, win, xs); break;
        case NOMAD_B200_WAV_S32: stage_window<NOMAD_B200_WAV_S32>(it, first, win, xs); break;
        case NOMAD_B200_WAV_F32: stage_window<NOMAD_B200_WAV_F32>(it, first, win, xs); break;
        default: stage_window<NOMAD_B200_WAV_F64>(it, first, win, xs); break;
    }
    __syncthreads();
    const long long j = j0 + threadIdx.x;
    if (j >= n_out) return;
    const long long m = j / n;
    const int p = (int)(j - m * n);
    const float* hp = h + (long long)p * K;
    const float* x = xs + (m - m0) * o;
    const int2 kr = __ldg(range + p);
    float acc = 0.f;
    for (int k = kr.x; k < kr.y; ++k) acc = fmaf(__ldg(hp + k), x[k], acc);
    it.out[j] = acc;
}

// One launch over `blocks` blocks of items at source rate `sr`.
static int launch_group(int sr, int target_sr, const ItemTable& tab, long long blocks, cudaStream_t st) {
    NB_CHECK(blocks > 0 && blocks < (1LL << 31), "ingest: %lld blocks in one launch", blocks);
    if (sr == target_sr) {
        to_mono_kernel<<<(unsigned)blocks, 256, 0, st>>>(tab);
        NB_LAUNCHED();
        return 0;
    }
    ResampleTable t;
    NB_TRY(get_table(sr, target_sr, &t));
    // input window of one block: the groups its 256 outputs touch, plus the filter length
    const int win_cap = (256 / t.n + 2) * t.o + t.K;
    const size_t smem = (size_t)win_cap * sizeof(float);
    NB_CHECK(smem <= 200 * 1024, "ingest: resampling %d -> %d Hz needs %zu bytes of shared memory per block", sr, target_sr, smem);
    static size_t smem_set_dev[64] = {0};  // the attribute is per device
    int cur_dev = 0;
    if (cudaGetDevice(&cur_dev) != cudaSuccess || cur_dev < 0 || cur_dev >= 64) cur_dev = 0;
    size_t& smem_set = smem_set_dev[cur_dev];
    if (smem > 48 * 1024 && smem > smem_set) {
        NB_CUDA(cudaFuncSetAttribute(resample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        smem_set = smem;
    }
    resample_kernel<<<(unsigned)blocks, 256, smem, st>>>(tab, t.dev, t.range, t.o, t.n, t.width, t.K, win_cap);
    NB_LAUNCHED();
    return 0;
}

static int format_bytes(int format) {
    switch (format) {
        case NOMAD_B200_WAV_U8: return 1;
        case NOMAD_B200_WAV_S16: return 2;
        case NOMAD_B200_WAV_S24: return 3;
        case NOMAD_B200_WAV_S32: return 4;
        case NOMAD_B200_WAV_F32: return 4;
        case NOMAD_B200_WAV_F64: return 8;
    }
    return 0;
}

// The launches of a batch: items grouped by source rate (the target rate first), each group's blocks numbered from 0.
struct IngestPlan {
    struct Group {
        int sr;
        long long first_block, blocks;
    };
    std::vector<DevItem> items;
    std::vector<int> block_item;
    std::vector<Group> groups;
    size_t table_bytes() const { return (items.size() * sizeof(DevItem) + 255) / 256 * 256; }
    size_t workspace_bytes() const { return table_bytes() + block_item.size() * sizeof(int) + 256; }
};

static int plan_ingest(const void* src, const nomad_b200_ingest_item* items, int64_t n, int target_sr, float* out,
                       IngestPlan* plan) {
    NB_CHECK(n >= 0 && (n == 0 || items) && target_sr > 0, "ingest_batch: bad arguments");
    std::map<int, std::vector<int64_t>> by_rate;  // the target rate first, then ascending
    for (int64_t i = 0; i < n; ++i) {
        const nomad_b200_ingest_item& it = items[i];
        const int bytes = format_bytes(it.format);
        const int align = it.format == NOMAD_B200_WAV_S24 ? 1 : bytes;
        NB_CHECK(bytes > 0, "ingest_batch: item %lld: unknown sample format %d", (long long)i, it.format);
        NB_CHECK(it.channels >= 1 && it.sample_rate > 0 && it.n_frames >= 0 && it.byte_offset >= 0 && it.out_offset >= 0,
                 "ingest_batch: item %lld: bad descriptor", (long long)i);
        NB_CHECK(it.byte_offset % align == 0, "ingest_batch: item %lld: byte offset %lld is not aligned to %d bytes",
                 (long long)i, (long long)it.byte_offset, align);
        const int64_t full = nomad_b200_ingest_out_samples(it.n_frames, it.sample_rate, target_sr, 0);
        NB_CHECK(it.out_samples >= 0 && it.out_samples <= full, "ingest_batch: item %lld: %lld output samples, at most %lld",
                 (long long)i, (long long)it.out_samples, (long long)full);
        if (it.out_samples > 0) by_rate[it.sample_rate == target_sr ? 0 : it.sample_rate].push_back(i);
    }
    for (const auto& kv : by_rate) {
        IngestPlan::Group g;
        g.sr = kv.first == 0 ? target_sr : kv.first;
        g.first_block = (long long)plan->block_item.size();
        long long block0 = 0;
        for (int64_t i : kv.second) {
            const nomad_b200_ingest_item& it = items[i];
            DevItem d;
            d.src = src ? (const unsigned char*)src + it.byte_offset : nullptr;
            d.out = out ? out + it.out_offset : nullptr;
            d.n_in = it.n_frames;
            d.n_out = it.out_samples;
            d.channels = it.channels;
            d.format = it.format;
            d.block0 = (int)block0;
            d.pad = 0;
            const long long nb = (it.out_samples + 255) / 256;
            NB_CHECK(block0 + nb < (1LL << 31), "ingest_batch: too many output samples at %d Hz in one call", g.sr);
            plan->block_item.insert(plan->block_item.end(), (size_t)nb, (int)plan->items.size());
            plan->items.push_back(d);
            block0 += nb;
        }
        g.blocks = block0;
        plan->groups.push_back(g);
    }
    return 0;
}

// Host -> device copy of a descriptor table through a small pinned ring per device (the caller's table may be pageable
// and temporary): a slot is reused once the copy that last read it has completed, so nothing waits per call.
static int upload_table(const void* host, size_t bytes, void* dst_dev, cudaStream_t st) {
    struct Slot {
        char* host = nullptr;
        size_t cap = 0;
        cudaEvent_t ev = nullptr;
    };
    static std::mutex mu;
    static std::map<int, std::pair<int, std::array<Slot, 4>>> rings;
    int dev = 0;
    NB_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(mu);
    auto& ring = rings[dev];
    ring.first = (ring.first + 1) % 4;
    Slot& s = ring.second[ring.first];
    if (s.ev == nullptr) NB_CUDA(cudaEventCreateWithFlags(&s.ev, cudaEventDisableTiming));
    NB_CUDA(cudaEventSynchronize(s.ev));  // no-op unless this slot's previous copy is still in flight
    if (s.cap < bytes) {
        if (s.host) NB_CUDA(cudaFreeHost(s.host));
        s.cap = bytes < (64u << 10) ? (64u << 10) : bytes + bytes / 4;
        NB_CUDA(cudaMallocHost((void**)&s.host, s.cap));
    }
    memcpy(s.host, host, bytes);
    NB_CUDA(cudaMemcpyAsync(dst_dev, s.host, bytes, cudaMemcpyHostToDevice, st));
    NB_CUDA(cudaEventRecord(s.ev, st));
    return 0;
}

}  // namespace nb

using namespace nb;

extern "C" {

int64_t nomad_b200_ingest_out_samples(int64_t n_frames, int sr, int target_sr, int trim) {
    if (n_frames < 0 || sr <= 0 || target_sr <= 0) return -1;
    int64_t n = n_frames;
    if (sr != target_sr) {
        const long long g = gcd_ll(sr, target_sr);
        const long long o = sr / g, nn = target_sr / g;
        n = (nn * n_frames + o - 1) / o;  // ceil(new * length / orig)
    }
    if (trim && n > (int64_t)target_sr * 10) n = (int64_t)target_sr * 10;
    return n;
}

int nomad_b200_ingest_pcm16(const int16_t* pcm_dev, int64_t n_frames, int channels, int sr, int target_sr, int trim,
                            float* out_dev, void* stream) {
    NB_CHECK(pcm_dev && out_dev && n_frames >= 0 && channels >= 1 && sr > 0 && target_sr > 0, "ingest: bad arguments");
    const int64_t n_out = nomad_b200_ingest_out_samples(n_frames, sr, target_sr, trim);
    if (n_out == 0) return 0;
    ItemTable tab;
    tab.items = nullptr;
    tab.block_item = nullptr;
    tab.one.src = (const unsigned char*)pcm_dev;
    tab.one.out = out_dev;
    tab.one.n_in = n_frames;
    tab.one.n_out = n_out;
    tab.one.channels = channels;
    tab.one.format = NOMAD_B200_WAV_S16;
    tab.one.block0 = tab.one.pad = 0;
    return launch_group(sr, target_sr, tab, (n_out + 255) / 256, (cudaStream_t)stream);
}

size_t nomad_b200_ingest_workspace_bytes(const nomad_b200_ingest_item* items, int64_t n, int target_sr) {
    IngestPlan plan;
    if (plan_ingest(nullptr, items, n, target_sr, nullptr, &plan) != 0) return 0;
    return plan.workspace_bytes();
}

int nomad_b200_ingest_batch(const void* src_dev, const nomad_b200_ingest_item* items, int64_t n, int target_sr,
                            float* out_dev, void* workspace_dev, size_t workspace_bytes, void* stream) {
    IngestPlan plan;
    NB_TRY(plan_ingest(src_dev, items, n, target_sr, out_dev, &plan));
    if (plan.groups.empty()) return 0;
    NB_CHECK(src_dev && out_dev && workspace_dev, "ingest_batch: bad arguments");
    NB_CHECK(workspace_bytes >= plan.workspace_bytes(), "ingest_batch: workspace of %zu bytes, needs %zu", workspace_bytes,
             plan.workspace_bytes());
    // [item table | block -> item map] in one copy; the device copy starts at a 256-byte boundary of the workspace
    char* ws = (char*)(((uintptr_t)workspace_dev + 255) / 256 * 256);
    const size_t tb = plan.table_bytes(), mb = plan.block_item.size() * sizeof(int);
    std::vector<char> blob(tb + mb, 0);
    memcpy(blob.data(), plan.items.data(), plan.items.size() * sizeof(DevItem));
    memcpy(blob.data() + tb, plan.block_item.data(), mb);
    cudaStream_t st = (cudaStream_t)stream;
    NB_TRY(upload_table(blob.data(), blob.size(), ws, st));
    for (const IngestPlan::Group& g : plan.groups) {
        ItemTable tab;
        memset(&tab, 0, sizeof(tab));
        tab.items = (const DevItem*)ws;
        tab.block_item = (const int*)(ws + tb) + g.first_block;
        NB_TRY(launch_group(g.sr, target_sr, tab, g.blocks, st));
    }
    return 0;
}

}  // extern "C"
