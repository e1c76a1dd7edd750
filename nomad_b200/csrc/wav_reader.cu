// Native reader of PCM and IEEE-float RIFF/WAVE files: the decode step of ``Nomad.load_processing`` (reference
// nomad.py:192-212, ``torchaudio.load``) for the common corpus formats, done by a few host threads straight into the
// caller's (pinned) staging buffer.  Python's ``wave`` module costs ~0.25 ms of interpreter time per file, which is what
// held ``nomad.predict`` from files at 31 k utterance-seconds per second against 50 k from memory (profiles/
// r02_final_bench_files.json).  Host code only (no CUDA).  The reader moves raw data bytes; the device ingest
// (ingest.cu) decodes them.  Files it does not handle (u-law, A-law, ADPCM, RIFX, other widths, a ``data`` chunk before
// ``fmt ``) are reported with frames = -1 and take the Python path.
#include <atomic>
#include <cstdio>
#include <cstring>
#include <thread>
#include <vector>

#include "../../include/nomad_b200.h"
#include "common.cuh"

namespace nb {

struct WavInfo {
    int sr = 0, channels = 0, format = 0;
    long long frames = -1, data_offset = 0;
};

static uint32_t rd32(const unsigned char* p) { return p[0] | (p[1] << 8) | (p[2] << 16) | ((uint32_t)p[3] << 24); }
static uint16_t rd16(const unsigned char* p) { return (uint16_t)(p[0] | (p[1] << 8)); }

// Bytes 4..15 of KSDATAFORMAT_SUBTYPE_PCM / _IEEE_FLOAT ({0000000X-0000-0010-8000-00AA00389B71}, little-endian); the
// first four bytes carry the format tag.
static const unsigned char kGuidTail[12] = {0x00, 0x00, 0x10, 0x00, 0x80, 0x00, 0x00, 0xAA, 0x00, 0x38, 0x9B, 0x71};

// sample format of (format tag, container bits), 0 when not handled
static int sample_format(int tag, int bits) {
    if (tag == 1) {
        switch (bits) {
            case 8: return NOMAD_B200_WAV_U8;
            case 16: return NOMAD_B200_WAV_S16;
            case 24: return NOMAD_B200_WAV_S24;
            case 32: return NOMAD_B200_WAV_S32;
        }
    } else if (tag == 3) {
        if (bits == 32) return NOMAD_B200_WAV_F32;
        if (bits == 64) return NOMAD_B200_WAV_F64;
    }
    return 0;
}

// Parse the RIFF header.  frames = -1 (format 0) when the file is not one of the handled encodings; sample rate and
// channels are still reported when the ``fmt `` chunk could be read.
static WavInfo probe_one(const char* path) {
    WavInfo w;
    FILE* f = fopen(path, "rb");
    if (!f) return w;
    unsigned char h[12];
    if (fread(h, 1, 12, f) != 12 || memcmp(h, "RIFF", 4) != 0 || memcmp(h + 8, "WAVE", 4) != 0) {
        fclose(f);
        return w;
    }
    int format = 0, block_align = 0;
    long long pos = 12;
    for (;;) {
        unsigned char ch[8];
        if (fseek(f, (long)pos, SEEK_SET) != 0 || fread(ch, 1, 8, f) != 8) break;
        const uint32_t size = rd32(ch + 4);
        if (memcmp(ch, "fmt ", 4) == 0) {
            unsigned char fm[40];
            const size_t n = size < 40 ? size : 40;
            if (n < 16 || fread(fm, 1, n, f) != n) break;
            int tag = rd16(fm);
            w.channels = rd16(fm + 2);
            w.sr = (int)rd32(fm + 4);
            block_align = rd16(fm + 12);
            const int bits = rd16(fm + 14);  // container width; WAVE_FORMAT_EXTENSIBLE's valid-bits field is ignored
            if (tag == 0xFFFE) {             // WAVE_FORMAT_EXTENSIBLE: the whole sub-format GUID decides
                const uint32_t sub = n >= 40 ? rd32(fm + 24) : 0;
                tag = (sub == 1 || sub == 3) && memcmp(fm + 28, kGuidTail, 12) == 0 ? (int)sub : 0;
            }
            format = sample_format(tag, bits);
            if (format == 0 || w.channels < 1 || w.sr <= 0 || block_align != w.channels * (bits / 8)) {
                format = 0;
                break;
            }
        } else if (memcmp(ch, "data", 4) == 0) {
            if (format != 0) {
                fseek(f, 0, SEEK_END);
                const long long file_size = ftell(f);
                long long bytes = size;
                if (pos + 8 + bytes > file_size) bytes = file_size - (pos + 8);  // truncated file / streaming header
                w.data_offset = pos + 8;
                w.frames = bytes / block_align;
                w.format = format;
            }
            break;
        }
        pos += 8 + (long long)size + (size & 1);
    }
    fclose(f);
    return w;
}

template <typename F>
static void parallel_for(long long n, int threads, F fn) {
    if (threads <= 0) threads = (int)std::thread::hardware_concurrency();
    if (threads < 1) threads = 1;
    if (threads > n) threads = (int)(n > 0 ? n : 1);
    std::atomic<long long> next{0};
    auto work = [&] {
        for (long long i = next.fetch_add(1); i < n; i = next.fetch_add(1)) fn(i);
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < threads; ++t) pool.emplace_back(work);
    work();
    for (auto& t : pool) t.join();
}

}  // namespace nb

extern "C" {

int nomad_b200_wav_probe_format(const char* const* paths, int64_t n, int32_t* sample_rate, int32_t* channels,
                                int64_t* frames, int64_t* data_offset, int32_t* format, int threads) {
    NB_CHECK(n >= 0 && (n == 0 || (paths && sample_rate && channels && frames && data_offset && format)),
             "wav_probe_format: bad arguments");
    nb::parallel_for(n, threads, [&](long long i) {
        const nb::WavInfo w = nb::probe_one(paths[i]);
        sample_rate[i] = w.sr;
        channels[i] = w.channels;
        frames[i] = w.frames;
        data_offset[i] = w.data_offset;
        format[i] = w.format;
    });
    return 0;
}

int nomad_b200_wav_probe(const char* const* paths, int64_t n, int32_t* sample_rate, int32_t* channels, int64_t* frames,
                         int64_t* data_offset, int threads) {
    NB_CHECK(n >= 0 && (n == 0 || (paths && sample_rate && channels && frames && data_offset)), "wav_probe: bad arguments");
    std::vector<int32_t> format((size_t)n);
    NB_TRY(nomad_b200_wav_probe_format(paths, n, sample_rate, channels, frames, data_offset, format.data(), threads));
    for (int64_t i = 0; i < n; ++i) {
        if (format[i] != NOMAD_B200_WAV_S16) {
            frames[i] = -1;
            data_offset[i] = 0;
        }
    }
    return 0;
}

int nomad_b200_wav_read(const char* const* paths, int64_t n, const int64_t* src_offset, const int64_t* n_bytes,
                        const int64_t* dst_offset, void* dst, int threads) {
    NB_CHECK(n >= 0 && (n == 0 || (paths && src_offset && n_bytes && dst_offset && dst)), "wav_read: bad arguments");
    std::atomic<long long> failed{-1};
    nb::parallel_for(n, threads, [&](long long i) {
        if (n_bytes[i] <= 0) return;
        FILE* f = fopen(paths[i], "rb");
        bool ok = f != nullptr && fseek(f, (long)src_offset[i], SEEK_SET) == 0 &&
                  fread((char*)dst + dst_offset[i], 1, (size_t)n_bytes[i], f) == (size_t)n_bytes[i];
        if (f) fclose(f);
        if (!ok) failed.store(i);
    });
    NB_CHECK(failed.load() < 0, "wav_read: short read on %s", paths[failed.load()]);
    return 0;
}

int nomad_b200_wav_read_pcm16(const char* const* paths, int64_t n, const int64_t* data_offset, const int64_t* n_samples,
                              const int64_t* dst_offset, int16_t* dst, int threads) {
    NB_CHECK(n >= 0 && (n == 0 || (paths && data_offset && n_samples && dst_offset && dst)), "wav_read_pcm16: bad arguments");
    std::vector<int64_t> n_bytes((size_t)n), dst_bytes((size_t)n);
    for (int64_t i = 0; i < n; ++i) {
        n_bytes[i] = 2 * n_samples[i];
        dst_bytes[i] = 2 * dst_offset[i];
    }
    return nomad_b200_wav_read(paths, n, data_offset, n_bytes.data(), dst_bytes.data(), dst, threads);
}

}  // extern "C"
