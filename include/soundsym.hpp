// soundsym.hpp — C++17 host mirror of the reference crate's public API for the hot path, on top of the C ABI
// (soundsym_b200.h). The reference is compiled Rust and Rust is not installed in this image, so this header plays the
// role of the `extern "C"` shim of INTEGRATION.md: same type names, method names, argument meaning and error behaviour
// as src/lib.rs / src/sound.rs. Header-only; link with -lsoundsym_b200. All numerics run in the library on the GPU.
//
//   Sound            src/sound.rs:71-213      SoundDictionary  src/sound.rs:288-371
//   SoundSequence    src/sound.rs:373-484     Partitioner      src/lib.rs:62-151      CosError  src/lib.rs:181-198
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <filesystem>
#include <fstream>
#include <limits>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <vector>

#include "soundsym_b200.h"

namespace soundsym {

constexpr size_t NCOEFFS = SS_NCOEFFS, NCLUSTERS = SS_NCLUSTERS, HOP = SS_HOP, BIN = SS_BIN;  // src/lib.rs:22-25

/// CosError (src/lib.rs:181-198): a message plus the C ABI status it came from.
struct CosError : std::runtime_error {
    int code;
    CosError(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

/// one ss_ctx per process and device (the crate is single-threaded; so is a context)
class Context {
   public:
    explicit Context(int device = 0) {
        const int rc = ss_ctx_create(device, &h_);
        if (rc != SS_OK) throw CosError(rc, ss_last_error(nullptr));
    }
    ~Context() { ss_ctx_destroy(h_); }
    Context(const Context&) = delete;
    Context& operator=(const Context&) = delete;
    ss_ctx* get() const { return h_; }
    void check(int rc) const {
        if (rc != SS_OK) throw CosError(rc, ss_last_error(h_));
    }
    static Context& global() {
        static Context ctx(0);
        return ctx;
    }

   private:
    ss_ctx* h_ = nullptr;
};

/// GaussianMixtureModel as train_model returns it (src/lib.rs:44-54)
struct GaussianMixtureModel {
    int ncomp = 0, ncoeffs = 0;
    std::vector<double> means, covs, weights;
    ss_gmm view() const { return ss_gmm{ncomp, ncoeffs, means.data(), covs.data(), weights.data()}; }
    /// binary dump: i32 ncomp, i32 ncoeffs, then means, covs, weights as f64
    static GaussianMixtureModel load(const std::string& path) {
        std::ifstream f(path, std::ios::binary);
        if (!f) throw CosError(SS_ERR_INVALID, "cannot open model file " + path);
        GaussianMixtureModel m;
        int32_t hdr[2];
        f.read(reinterpret_cast<char*>(hdr), 8);
        m.ncomp = hdr[0];
        m.ncoeffs = hdr[1];
        m.means.resize((size_t)m.ncomp * m.ncoeffs);
        m.covs.resize((size_t)m.ncomp * m.ncoeffs * m.ncoeffs);
        m.weights.resize(m.ncomp);
        f.read(reinterpret_cast<char*>(m.means.data()), m.means.size() * 8);
        f.read(reinterpret_cast<char*>(m.covs.data()), m.covs.size() * 8);
        f.read(reinterpret_cast<char*>(m.weights.data()), m.weights.size() * 8);
        if (!f) throw CosError(SS_ERR_INVALID, "short model file " + path);
        return m;
    }
};

class Sound {
   public:
    std::optional<std::string> name;

    /// Sound::from_samples (src/sound.rs:92-112): MFCC + max_power + mean in one device pass
    static Sound from_samples(std::vector<double> samples, double sample_rate, std::optional<std::vector<double>> mfccs = std::nullopt,
                              std::optional<std::string> name = std::nullopt, Context& ctx = Context::global()) {
        Sound s;
        s.ctx_ = &ctx;
        s.name = std::move(name);
        s.sample_rate_ = sample_rate;
        size_t frames = 0;
        ss_frame_count(samples.size(), &frames);
        std::vector<double> out(frames * NCOEFFS);
        s.mean_mfccs_.assign(NCOEFFS, 0.0);
        ctx.check(ss_sound_analyze(ctx.get(), samples.data(), samples.size(), sample_rate, (int)NCOEFFS, out.data(), &frames, &s.max_power_,
                                   s.mean_mfccs_.data()));
        if (mfccs) {  // the reference computes and discards its own analysis here (src/sound.rs:94)
            s.mfccs_ = std::move(*mfccs);
            s.mean_mfccs_ = mean_of(s.mfccs_);
        } else {
            s.mfccs_ = std::move(out);
        }
        s.samples_ = std::move(samples);
        return s;
    }

    /// Sound::from_path (src/sound.rs:116-126): mono integer-PCM WAV; the int -> f64 conversion runs on the GPU
    static Sound from_path(const std::string& path, Context& ctx = Context::global()) {
        int bits = 0;
        double sr = 0;
        std::vector<int32_t> pcm = read_wav_pcm(path, &bits, &sr);
        std::vector<double> samples(pcm.size());
        ctx.check(ss_decode_pcm(ctx.get(), pcm.data(), pcm.size(), bits, samples.data()));
        std::string stem = path.substr(path.find_last_of('/') == std::string::npos ? 0 : path.find_last_of('/') + 1);
        stem = stem.substr(0, stem.find_last_of('.'));
        return from_samples(std::move(samples), sr, std::nullopt, stem, ctx);
    }

    /// Sound::push_samples (src/sound.rs:145-164), including its `(old*n0 + new*n1) * 0.5` mean rule
    void push_samples(const std::vector<double>& new_samples) {
        const size_t initial = num_frames();
        samples_.insert(samples_.end(), new_samples.begin(), new_samples.end());
        const double* tail = samples_.data() + initial * HOP;
        const size_t n = samples_.size() - initial * HOP;
        size_t frames = 0;
        ss_frame_count(n, &frames);
        std::vector<double> out(frames * NCOEFFS), mean(NCOEFFS);
        double mp = 0;
        ctx_->check(ss_sound_analyze(ctx_->get(), tail, n, sample_rate_, (int)NCOEFFS, out.data(), &frames, &mp, mean.data()));
        mfccs_.insert(mfccs_.end(), out.begin(), out.end());
        const size_t nf = num_frames() - initial;
        for (size_t k = 0; k < NCOEFFS; k++) mean_mfccs_[k] = (mean_mfccs_[k] * (double)initial + mean[k] * (double)nf) * 0.5;
        max_power_ = std::fmax(max_power_, mp);
    }

    double max_power() const { return max_power_; }
    const std::vector<double>& samples() const { return samples_; }
    double sample_rate() const { return sample_rate_; }
    const std::vector<double>& mfccs() const { return mfccs_; }
    const std::vector<double>& mean_mfccs() const { return mean_mfccs_; }
    size_t num_frames() const { return mfccs_.size() / NCOEFFS; }
    Context& context() const { return *ctx_; }

    /// a cut of a longer sound that carries the parent's MFCC rows (add_segments / reconstruction.rs:77-81):
    /// Sound::from_samples(samp, sr, Some(mfccs), None) without re-running the discarded analysis
    /// max_power = analyze_max_power of the cut (src/sound.rs:95), computed by the caller for all cuts in one launch
    static Sound from_cut(std::vector<double> samples, double sample_rate, std::vector<double> mfccs, double max_power, Context& ctx) {
        Sound s;
        s.ctx_ = &ctx;
        s.sample_rate_ = sample_rate;
        s.samples_ = std::move(samples);
        s.mfccs_ = std::move(mfccs);
        s.mean_mfccs_ = mean_of(s.mfccs_);
        s.max_power_ = max_power;
        return s;
    }

    /// the segment cuts of a longer sound, each carrying the parent's MFCC rows - the loop of add_segments
    /// (src/sound.rs:330-343) and of examples/reconstruction.rs:77-81: segment i takes seg_i samples and (seg_i / HOP) *
    /// NCOEFFS MFCC values. Every cut's max power (Sound::from_samples runs analyze_max_power on it, src/sound.rs:95)
    /// comes from ONE batched launch.
    static std::vector<std::shared_ptr<Sound>> cut(const Sound& sound, const std::vector<size_t>& segments, Context& ctx) {
        std::vector<uint64_t> bounds(segments.size() + 1, 0), foff(segments.size() + 1, 0);
        for (size_t i = 0; i < segments.size(); i++) bounds[i + 1] = std::min<uint64_t>(bounds[i] + segments[i], sound.samples().size());
        std::vector<double> power(segments.size(), 0.0);
        if (!segments.empty())
            ctx.check(ss_sound_analyze_batch(ctx.get(), sound.samples().data(), bounds.data(), segments.size(), sound.sample_rate(), (int)NCOEFFS,
                                             nullptr, foff.data(), power.data(), nullptr));
        std::vector<std::shared_ptr<Sound>> out;
        size_t spos = 0, fpos = 0, i = 0;
        for (size_t seg : segments) {
            const size_t ns = std::min(seg, sound.samples().size() - std::min(spos, sound.samples().size()));
            const size_t nv = std::min(seg / HOP * NCOEFFS, sound.mfccs().size() - std::min(fpos, sound.mfccs().size()));
            std::vector<double> samp(sound.samples().begin() + spos, sound.samples().begin() + spos + ns);
            std::vector<double> m(sound.mfccs().begin() + fpos, sound.mfccs().begin() + fpos + nv);
            spos += ns;
            fpos += nv;
            out.push_back(std::make_shared<Sound>(Sound::from_cut(std::move(samp), sound.sample_rate(), std::move(m), power[i++], ctx)));
        }
        return out;
    }

    /// many sounds analysed in ONE device pass (ss_sound_analyze_batch): what SoundDictionary::from_path and
    /// SoundSequence::from_timestamps build their Sounds from. All sounds share sample_rate.
    static std::vector<std::shared_ptr<Sound>> from_samples_batch(std::vector<std::vector<double>> cuts, double sample_rate,
                                                                  const std::vector<std::optional<std::string>>& names, Context& ctx) {
        std::vector<uint64_t> off(cuts.size() + 1, 0), foff(cuts.size() + 1, 0);
        std::vector<double> flat;
        size_t frames = 0;
        for (size_t i = 0; i < cuts.size(); i++) {
            off[i + 1] = off[i] + cuts[i].size();
            flat.insert(flat.end(), cuts[i].begin(), cuts[i].end());
            size_t f = 0;
            ss_frame_count(cuts[i].size(), &f);
            frames += f;
        }
        std::vector<double> mfcc(frames * NCOEFFS), mp(cuts.size(), 0.0), mean(cuts.size() * NCOEFFS, 0.0);
        ctx.check(ss_sound_analyze_batch(ctx.get(), flat.data(), off.data(), cuts.size(), sample_rate, (int)NCOEFFS, mfcc.data(), foff.data(),
                                         mp.data(), mean.data()));
        std::vector<std::shared_ptr<Sound>> out;
        for (size_t i = 0; i < cuts.size(); i++) {
            auto s = std::make_shared<Sound>();
            s->ctx_ = &ctx;
            s->name = i < names.size() ? names[i] : std::nullopt;
            s->sample_rate_ = sample_rate;
            s->samples_ = std::move(cuts[i]);
            s->mfccs_.assign(mfcc.begin() + foff[i] * NCOEFFS, mfcc.begin() + foff[i + 1] * NCOEFFS);
            s->mean_mfccs_.assign(mean.begin() + i * NCOEFFS, mean.begin() + (i + 1) * NCOEFFS);
            s->max_power_ = mp[i];
            out.push_back(std::move(s));
        }
        return out;
    }
    /// a mono integer-PCM WAV as f64 samples, s / (i32::MAX >> (32 - bits)) (src/sound.rs:117-120), on the host
    static std::vector<double> read_wav_samples(const std::string& path, double* sr) {
        int bits = 0;
        std::vector<int32_t> pcm = read_wav_pcm(path, &bits, sr);
        const double denom = (double)(INT32_MAX >> (32 - bits));
        std::vector<double> out(pcm.size());
        for (size_t i = 0; i < pcm.size(); i++) out[i] = (double)pcm[i] / denom;
        return out;
    }
    /// Sound::write_file (src/sound.rs:129-143): 32-bit integer PCM, (sample * i32::MAX) as i32
    void write_file(const std::string& path) const { write_wav_i32(path, samples_.data(), samples_.size(), sample_rate_); }
    static void write_wav_i32(const std::string& path, const double* s, size_t n, double sample_rate) {
        std::ofstream f(path, std::ios::binary);
        if (!f) throw CosError(SS_ERR_INVALID, "cannot create " + path);
        const uint32_t bytes = (uint32_t)(n * 4), riff = 36 + bytes, sixteen = 16, rate = (uint32_t)sample_rate, brate = rate * 4;
        const uint16_t pcm = 1, ch = 1, align = 4, bits = 32;
        f.write("RIFF", 4), f.write((const char*)&riff, 4), f.write("WAVEfmt ", 8), f.write((const char*)&sixteen, 4);
        f.write((const char*)&pcm, 2), f.write((const char*)&ch, 2), f.write((const char*)&rate, 4), f.write((const char*)&brate, 4);
        f.write((const char*)&align, 2), f.write((const char*)&bits, 2), f.write("data", 4), f.write((const char*)&bytes, 4);
        std::vector<int32_t> q(n);
        for (size_t i = 0; i < n; i++) {  // Rust's `as i32`: truncate toward zero, saturate, NaN -> 0
            const double v = s[i] * 2147483647.0;
            q[i] = v != v ? 0 : (v >= 2147483647.0 ? INT32_MAX : (v <= -2147483648.0 ? INT32_MIN : (int32_t)v));
        }
        f.write((const char*)q.data(), bytes);
    }

   private:
    static std::vector<double> mean_of(const std::vector<double>& m) {  // analyze_mean_mfccs, src/sound.rs:271-286
        std::vector<double> out(NCOEFFS, 0.0);
        const size_t frames = m.size() / NCOEFFS;
        for (size_t f = 0; f < frames; f++)
            for (size_t k = 0; k < NCOEFFS; k++) out[k] += m[f * NCOEFFS + k];
        for (size_t k = 0; k < NCOEFFS; k++) out[k] = out[k] / (double)frames;
        return out;
    }
    /// integer-PCM RIFF/WAVE only (what hound::WavReader yields at src/sound.rs:117): format tag 1 or 0xFFFE with the PCM
    /// sub-format, 8 (unsigned, offset 128) / 16 / 24 / 32 bits, fmt before data, every chunk inside the file
    static std::vector<int32_t> read_wav_pcm(const std::string& path, int* bits, double* sr) {
        std::ifstream f(path, std::ios::binary);
        if (!f) throw CosError(SS_ERR_INVALID, "cannot open " + path);
        std::vector<char> d((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
        if (d.size() < 12 || memcmp(d.data(), "RIFF", 4) || memcmp(d.data() + 8, "WAVE", 4)) throw CosError(SS_ERR_INVALID, "not a WAVE file: " + path);
        size_t pos = 12;
        std::vector<int32_t> pcm;
        bool have_fmt = false, have_data = false;
        while (pos + 8 <= d.size()) {
            uint32_t size;
            memcpy(&size, d.data() + pos + 4, 4);
            const char* body = d.data() + pos + 8;
            const size_t avail = std::min<size_t>(size, d.size() - pos - 8);
            if (!memcmp(d.data() + pos, "fmt ", 4)) {
                if (avail < 16) throw CosError(SS_ERR_INVALID, "truncated fmt chunk: " + path);
                uint16_t tag, b;
                uint32_t rate;
                memcpy(&tag, body, 2);
                memcpy(&rate, body + 4, 4);
                memcpy(&b, body + 14, 2);
                if (tag == 0xFFFE) {
                    if (avail < 26) throw CosError(SS_ERR_INVALID, "truncated extensible fmt chunk: " + path);
                    memcpy(&tag, body + 24, 2);
                }
                if (tag != 1) throw CosError(SS_ERR_INVALID, "unsupported WAV format tag (integer PCM only): " + path);
                if (b != 8 && b != 16 && b != 24 && b != 32) throw CosError(SS_ERR_INVALID, "unsupported bits per sample: " + path);
                *sr = rate;
                *bits = b;
                have_fmt = true;
            } else if (!memcmp(d.data() + pos, "data", 4) && !have_data) {
                if (!have_fmt) throw CosError(SS_ERR_INVALID, "data chunk before fmt chunk: " + path);
                const int bytes = *bits / 8;
                pcm.resize(avail / bytes);
                for (size_t i = 0; i < pcm.size(); i++) {
                    int32_t v = 0;
                    memcpy(&v, body + i * bytes, bytes);
                    if (bytes == 1) v = (v & 0xFF) - 128;
                    else if (bytes < 4) v = (int32_t)((uint32_t)v << (32 - *bits)) >> (32 - *bits);  // sign-extend
                    pcm[i] = v;
                }
                have_data = true;
            }
            pos += 8 + (size_t)size + (size & 1);
        }
        if (!have_fmt || !have_data) throw CosError(SS_ERR_INVALID, "no fmt / data chunk: " + path);
        return pcm;
    }
    Context* ctx_ = nullptr;
    double max_power_ = 0, sample_rate_ = 44100;
    std::vector<double> samples_, mfccs_, mean_mfccs_;
};

class SoundDictionary {
   public:
    std::vector<std::shared_ptr<Sound>> sounds;
    int mode = SS_COSINE_REF;  // SS_DTW selects the DTW extension
    uint32_t dtw_band = 0;     // Sakoe-Chiba radius of the SS_DTW distance and of align() (ss_dict_set_dtw_band; 0 = no band)

    explicit SoundDictionary(Context& ctx = Context::global()) : ctx_(&ctx) {}
    ~SoundDictionary() { ss_dict_destroy(dev_); }
    SoundDictionary(const SoundDictionary&) = delete;
    SoundDictionary& operator=(const SoundDictionary&) = delete;

    /// SoundDictionary::add_segments (src/sound.rs:330-343)
    void add_segments(const Sound& sound, const std::vector<size_t>& segments) {
        for (auto& c : Sound::cut(sound, segments, *ctx_)) sounds.push_back(std::move(c));
        ss_dict_destroy(dev_);
        dev_ = nullptr;
    }
    /// SoundDictionary::from_path (src/sound.rs:304-320): every *.wav directly inside `dir` becomes one Sound (sorted by
    /// name: read_dir's order is platform-defined). Files are decoded on the host and analysed together, one
    /// ss_sound_analyze_batch per distinct sample rate.
    static std::unique_ptr<SoundDictionary> from_path(const std::string& dir, Context& ctx = Context::global()) {
        namespace fs = std::filesystem;
        std::vector<std::string> files;
        for (const auto& e : fs::directory_iterator(dir))
            if (e.is_regular_file() && e.path().extension() == ".wav") files.push_back(e.path().string());
        std::sort(files.begin(), files.end());
        auto d = std::make_unique<SoundDictionary>(ctx);
        d->sounds.resize(files.size());
        std::vector<double> rates(files.size());
        std::vector<std::vector<double>> samples(files.size());
        for (size_t i = 0; i < files.size(); i++) samples[i] = Sound::read_wav_samples(files[i], &rates[i]);
        std::vector<bool> done(files.size(), false);
        for (size_t i = 0; i < files.size(); i++) {
            if (done[i]) continue;
            std::vector<size_t> sel;
            std::vector<std::vector<double>> cuts;
            std::vector<std::optional<std::string>> names;
            for (size_t j = i; j < files.size(); j++)
                if (!done[j] && rates[j] == rates[i]) {
                    sel.push_back(j);
                    cuts.push_back(std::move(samples[j]));
                    names.push_back(fs::path(files[j]).stem().string());
                    done[j] = true;
                }
            auto snds = Sound::from_samples_batch(std::move(cuts), rates[i], names, ctx);
            for (size_t k = 0; k < sel.size(); k++) d->sounds[sel[k]] = std::move(snds[k]);
        }
        return d;
    }
    static std::unique_ptr<SoundDictionary> from_segments(const Sound& sound, const std::vector<size_t>& segments, Context& ctx = Context::global()) {
        auto d = std::make_unique<SoundDictionary>(ctx);
        d->add_segments(sound, segments);
        return d;
    }

    /// batched at_distance: (indices, distances) for every query; targets empty -> 1.0 (match_sound)
    void match_indices(const std::vector<std::shared_ptr<Sound>>& queries, const std::vector<double>& targets, int k, std::vector<uint32_t>* idx,
                       std::vector<double>* dist) {
        ss_dict* d = device();
        std::vector<uint64_t> off(queries.size() + 1, 0);
        std::vector<double> flat;
        for (size_t i = 0; i < queries.size(); i++) {
            off[i + 1] = off[i] + queries[i]->num_frames();
            flat.insert(flat.end(), queries[i]->mfccs().begin(), queries[i]->mfccs().end());
        }
        idx->assign(queries.size() * k, 0);
        dist->assign(queries.size() * k, 0.0);
        ctx_->check(ss_dict_match(d, flat.data(), off.data(), queries.size(), mode, targets.empty() ? nullptr : targets.data(), k, idx->data(),
                                  dist->data()));
    }
    /// SoundDictionary::at_distance (src/sound.rs:351-370); always Some for a non-empty dictionary
    std::shared_ptr<Sound> at_distance(double distance, const std::shared_ptr<Sound>& other) {
        std::vector<uint32_t> idx;
        std::vector<double> dist;
        match_indices({other}, {distance}, 1, &idx, &dist);
        return sounds[idx[0]];
    }
    /// SoundSequence::from_distances' chain for SS_COSINE_REF on the device (ss_dict_walk): step t matches the sound step
    /// t - 1 returned (step 0: start) at distances[t]
    void walk(const Sound& start, const std::vector<double>& distances, std::vector<uint32_t>* idx, std::vector<double>* dist) {
        ss_dict* d = device();
        idx->assign(distances.size(), 0);
        dist->assign(distances.size(), 0.0);
        ctx_->check(ss_dict_walk(d, start.mfccs().data(), start.num_frames(), distances.data(), distances.size(), idx->data(), dist->data()));
    }
    /// DTW warping path (ss_dict_align) of queries[p] against sounds[indices[p]] (indices as match_indices returns them;
    /// 0xFFFFFFFF -> empty path, inf): (*paths)[p] holds (frame of the query, frame of the dictionary sound) pairs in order.
    /// Works in either mode: the path is the SS_DTW one whatever matcher chose the indices.
    void align(const std::vector<std::shared_ptr<Sound>>& queries, const std::vector<uint32_t>& indices,
               std::vector<std::vector<std::pair<uint32_t, uint32_t>>>* paths, std::vector<double>* dist) {
        if (indices.size() != queries.size()) ctx_->check(SS_ERR_INVALID);
        ss_dict* d = device();
        std::vector<uint64_t> off(queries.size() + 1, 0);
        std::vector<double> flat;
        size_t cap = 0;
        for (size_t i = 0; i < queries.size(); i++) {
            off[i + 1] = off[i] + queries[i]->num_frames();
            flat.insert(flat.end(), queries[i]->mfccs().begin(), queries[i]->mfccs().end());
            if (indices[i] < sounds.size() && queries[i]->num_frames() && sounds[indices[i]]->num_frames())
                cap += queries[i]->num_frames() + sounds[indices[i]]->num_frames() - 1;
        }
        std::vector<uint32_t> cells(2 * std::max<size_t>(cap, 1));
        std::vector<uint64_t> poff(queries.size() + 1);
        dist->assign(queries.size(), 0.0);
        ctx_->check(ss_dict_align(d, flat.data(), off.data(), queries.size(), indices.data(), cells.data(), cap, poff.data(), dist->data()));
        paths->assign(queries.size(), {});
        for (size_t p = 0; p < queries.size(); p++)
            for (uint64_t e = poff[p]; e < poff[p + 1]; e++) (*paths)[p].emplace_back(cells[2 * e], cells[2 * e + 1]);
    }
    /// SoundDictionary::match_sound (src/sound.rs:346-348)
    std::shared_ptr<Sound> match_sound(const std::shared_ptr<Sound>& other) { return at_distance(1.0, other); }
    Context& context() const { return *ctx_; }

   private:
    ss_dict* device() {
        if (!dev_) {
            std::vector<uint64_t> off(sounds.size() + 1, 0);
            std::vector<double> flat;
            for (size_t i = 0; i < sounds.size(); i++) {
                off[i + 1] = off[i] + sounds[i]->num_frames();
                flat.insert(flat.end(), sounds[i]->mfccs().begin(), sounds[i]->mfccs().end());
            }
            ctx_->check(ss_dict_create(ctx_->get(), flat.data(), off.data(), sounds.size(), (int)NCOEFFS, 0, &dev_));
        }
        if (ss_dict_dtw_band(dev_) != dtw_band) ctx_->check(ss_dict_set_dtw_band(dev_, dtw_band));  // (add_segments drops dev_)
        return dev_;
    }
    Context* ctx_;
    ss_dict* dev_ = nullptr;
};

class SoundSequence {
   public:
    /// SoundSequence::new (src/sound.rs:392-401): consecutive angular distances of the mean MFCCs
    explicit SoundSequence(std::vector<std::shared_ptr<Sound>> sounds, Context& ctx = Context::global()) : sounds_(std::move(sounds)), ctx_(&ctx) {
        if (sounds_.size() >= 2) {
            std::vector<double> rows;
            for (auto& s : sounds_) rows.insert(rows.end(), s->mean_mfccs().begin(), s->mean_mfccs().end());
            distances_.assign(sounds_.size() - 1, 0.0);
            ctx.check(ss_sequence_distances(ctx.get(), rows.data(), sounds_.size(), (int)NCOEFFS, distances_.data()));
        }
    }
    const std::vector<std::shared_ptr<Sound>>& sounds() const { return sounds_; }
    const std::vector<double>& distances() const { return distances_; }

    /// SoundSequence::clone_from_dictionary (src/sound.rs:451-472) + to_sound (:475-483): ONE batched match, then the
    /// pad / truncate / concatenate on the GPU. Returns the assembled Sound.
    Sound clone_from_dictionary_to_sound(SoundDictionary& dict, std::vector<uint32_t>* out_idx = nullptr) {
        std::vector<uint32_t> idx;
        std::vector<double> dist;
        dict.match_indices(sounds_, {}, 1, &idx, &dist);
        std::vector<uint64_t> doff(dict.sounds.size() + 1, 0), tlen(sounds_.size());
        std::vector<double> dsamples;
        for (size_t i = 0; i < dict.sounds.size(); i++) {
            doff[i + 1] = doff[i] + dict.sounds[i]->samples().size();
            dsamples.insert(dsamples.end(), dict.sounds[i]->samples().begin(), dict.sounds[i]->samples().end());
        }
        uint64_t total = 0;
        for (size_t i = 0; i < sounds_.size(); i++) total += (tlen[i] = sounds_[i]->samples().size());
        std::vector<double> out(total);
        ctx_->check(ss_resynth(ctx_->get(), dsamples.data(), doff.data(), dict.sounds.size(), idx.data(), tlen.data(), sounds_.size(), out.data()));
        if (out_idx) *out_idx = idx;
        const double sr = sounds_.empty() ? 44100.0 : sounds_[0]->sample_rate();
        return Sound::from_samples(std::move(out), sr, std::nullopt, std::nullopt, *ctx_);
    }

    /// SoundSequence::from_timestamps (src/sound.rs:419-430): one new Sound per (start, end, label), cut at
    /// round(start * sr) ..= round(end * sr); all cuts analysed in one batch
    static SoundSequence from_timestamps(const std::shared_ptr<Sound>& sound, const std::vector<struct Timestamp>& timestamps);

    /// SoundSequence::morph_to (src/sound.rs:440-449), batched
    SoundSequence morph_to(const std::vector<double>& distances, SoundDictionary& dict) {
        const size_t n = std::min(sounds_.size(), distances.size());
        std::vector<std::shared_ptr<Sound>> q(sounds_.begin(), sounds_.begin() + n), out;
        std::vector<uint32_t> idx;
        std::vector<double> dist;
        dict.match_indices(q, std::vector<double>(distances.begin(), distances.begin() + n), 1, &idx, &dist);
        for (uint32_t i : idx) out.push_back(dict.sounds[i]);
        return SoundSequence(std::move(out), *ctx_);
    }
    /// SoundSequence::from_distances (src/sound.rs:405-417): a chain, step t matches the sound step t - 1 returned.
    /// SS_COSINE_REF runs it on the device in one call; SS_DTW (whose at_distance ignores the target) keeps the nq = 1 loop.
    static SoundSequence from_distances(const std::vector<double>& distances, std::shared_ptr<Sound> start, SoundDictionary& dict) {
        std::vector<std::shared_ptr<Sound>> sounds{std::move(start)};
        if (!distances.empty() && dict.mode == SS_COSINE_REF) {
            std::vector<uint32_t> idx;
            std::vector<double> dist;
            dict.walk(*sounds[0], distances, &idx, &dist);
            for (uint32_t i : idx) sounds.push_back(dict.sounds[i]);
        } else {
            for (double d : distances) sounds.push_back(dict.at_distance(d, sounds.back()));
        }
        return SoundSequence(std::move(sounds), dict.context());
    }

   private:
    std::vector<std::shared_ptr<Sound>> sounds_;
    std::vector<double> distances_;
    Context* ctx_;
};

class Partitioner {
   public:
    std::shared_ptr<Sound> sound;
    size_t depth = 5, threshold = 4;  // Partitioner::new defaults, src/lib.rs:75-82
    std::optional<GaussianMixtureModel> model;

    explicit Partitioner(std::shared_ptr<Sound> s) : sound(std::move(s)) {}
    /// Partitioner::from_path (src/lib.rs:85-88)
    static Partitioner from_path(const std::string& path, Context& ctx = Context::global()) {
        return Partitioner(std::make_shared<Sound>(Sound::from_path(path, ctx)));
    }
    Partitioner& set_depth(size_t d) { return depth = d, *this; }
    Partitioner& set_threshold(size_t t) { return threshold = t, *this; }
    /// Partitioner::train (src/lib.rs:101-107). EM training is not on the data-parallel path (the reference's is randomly
    /// seeded, so parity is only defined GIVEN a model): the caller supplies one.
    void train(GaussianMixtureModel m) { model = std::move(m); }
    /// the same on the GPU (ss_gmm_train): 26 components, 5 EM rounds, Regularized(0.1); seeded instead of thread_rng,
    /// retried with the next seed when a component collapses (the reference's `while let Err` loop, src/lib.rs:50-52)
    void train(uint64_t seed = 0) {
        Context& ctx = sound->context();
        GaussianMixtureModel m;
        m.ncomp = (int)NCLUSTERS;
        m.ncoeffs = (int)NCOEFFS;
        m.means.resize(NCLUSTERS * NCOEFFS);
        m.covs.resize(NCLUSTERS * NCOEFFS * NCOEFFS);
        m.weights.resize(NCLUSTERS);
        int rc = SS_OK;
        for (int attempt = 0; attempt < 64; attempt++) {
            rc = ss_gmm_train(ctx.get(), sound->mfccs().data(), sound->num_frames(), m.ncoeffs, m.ncomp, 5, 0.1, seed + attempt,
                              m.means.data(), m.covs.data(), m.weights.data());
            if (rc != SS_ERR_INVALID) break;
        }
        ctx.check(rc);
        model = std::move(m);
    }

    /// Partitioner::partition_other (src/lib.rs:112-144): segment lengths in samples
    std::vector<size_t> partition_other(const Sound& other) const {
        Context& ctx = other.context();
        std::vector<uint64_t> lens(std::max<size_t>(other.num_frames(), 1));
        size_t nseg = 0;
        ss_gmm view{};
        if (model) view = model->view();
        ctx.check(ss_partition(ctx.get(), other.mfccs().data(), other.num_frames(), model ? &view : nullptr, (int)depth, (int)threshold, lens.data(), &nseg));
        return std::vector<size_t>(lens.begin(), lens.begin() + nseg);
    }
    std::vector<size_t> partition() const { return partition_other(*sound); }
};

/// Timestamp (src/sound.rs:508)
struct Timestamp {
    double start = 0, end = 0;
    std::optional<std::string> label;
};

/// audacity_labels_to_timestamps (src/sound.rs:511-531): `start<TAB>end<TAB>label` per line; a missing or unparsable number is
/// 0.0, a missing label is none
inline std::vector<Timestamp> audacity_labels_to_timestamps(const std::string& path) {
    std::ifstream f(path);
    if (!f) throw CosError(SS_ERR_INVALID, "cannot open " + path);
    auto num = [](const std::string& t) {
        try {
            size_t used = 0;
            const double v = std::stod(t, &used);
            return used == t.size() ? v : 0.0;
        } catch (...) {
            return 0.0;
        }
    };
    std::vector<Timestamp> out;
    std::string line;
    while (std::getline(f, line)) {
        const size_t a = line.find_first_not_of(" \t\r\n"), b = line.find_last_not_of(" \t\r\n");
        line = a == std::string::npos ? std::string() : line.substr(a, b - a + 1);
        std::vector<std::string> parts;
        size_t pos = 0;
        for (;;) {
            const size_t tab = line.find('\t', pos);
            parts.push_back(line.substr(pos, tab == std::string::npos ? std::string::npos : tab - pos));
            if (tab == std::string::npos) break;
            pos = tab + 1;
        }
        Timestamp t;
        if (parts.size() > 0) t.start = num(parts[0]);
        if (parts.size() > 1) t.end = num(parts[1]);
        if (parts.size() > 2) t.label = parts[2];
        out.push_back(std::move(t));
    }
    return out;
}

inline SoundSequence SoundSequence::from_timestamps(const std::shared_ptr<Sound>& sound, const std::vector<Timestamp>& timestamps) {
    const double sr = sound->sample_rate();
    std::vector<std::vector<double>> cuts;
    std::vector<std::optional<std::string>> names;
    for (const Timestamp& t : timestamps) {
        const long long a = std::llround(t.start * sr), b = std::llround(t.end * sr);
        if (a < 0 || b + 1 > (long long)sound->samples().size() || a > b + 1) throw CosError(SS_ERR_INVALID, "timestamp outside the sound");
        cuts.emplace_back(sound->samples().begin() + a, sound->samples().begin() + b + 1);
        names.push_back(t.label);
    }
    return SoundSequence(Sound::from_samples_batch(std::move(cuts), sr, names, sound->context()), sound->context());
}

/// write_splits (src/lib.rs:155-178): consecutive cuts of `sound` as `<out>/<idx:05>_<len>.wav`, 32-bit integer PCM
inline void write_splits(const Sound& sound, const std::vector<size_t>& splits, const std::string& out_path) {
    size_t pos = 0;
    for (size_t idx = 0; idx < splits.size(); idx++) {
        const size_t n = std::min(splits[idx], sound.samples().size() - std::min(pos, sound.samples().size()));
        char name[64];
        snprintf(name, sizeof(name), "/%05zu_%zu.wav", idx, splits[idx]);
        Sound::write_wav_i32(out_path + name, sound.samples().data() + pos, n, sound.sample_rate());
        pos += n;
    }
}

}  // namespace soundsym
