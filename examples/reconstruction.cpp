// examples/reconstruction.cpp — the flow of the reference's examples/reconstruction.rs (and, with --partition-only,
// examples/partition.rs) written against include/soundsym.hpp:
//   -s source.wav  -t target.wav  -o out.wav  -m model.bin  [--depth 3] [--threshold 4] [--dtw | --dtw-target] [--warp] [--partition-only]
//   --matcher dict_dir query_dir [--dtw] [--locate]
// Partitioner::from_path(source).threshold(4).depth(3) -> train (model supplied) -> partition -> SoundDictionary::from_segments
// -> partition the target with the source's model -> clone_from_dictionary -> to_sound -> write_file. --warp fits every matched
// sound to its target segment's timing along the DTW warping path (ss_resynth_warped) instead of zero-padding or cutting it.
// --dtw-target matches in SS_DTW_TARGET mode; with --morph its target distances are DTW distances, spread over the range the
// flow's own nearest-match distances span.
// Prints one JSON line with the segment counts, the match indices and checksums so that a test can compare it with the
// golden fixtures.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <string>

#include "soundsym.hpp"

using namespace soundsym;

int main(int argc, char** argv) {
    std::string src, tgt, out, model_path;
    size_t depth = 3, threshold = 4;  // examples/reconstruction.rs:44-45
    bool dtw = false, dtw_target = false, partition_only = false, morph = false, matcher_loop = false, warp = false, locate = false;
    size_t chain = 6;
    std::string dict_dir, query_dir, splits_dir;  // --matcher <dictionary dir> <query dir>: the flow of examples/matcher.rs
    for (int i = 1; i < argc; i++) {
        const std::string a = argv[i];
        auto next = [&]() { return i + 1 < argc ? std::string(argv[++i]) : std::string(); };
        if (a == "-s") src = next();
        else if (a == "-t") tgt = next();
        else if (a == "-o") out = next();
        else if (a == "-m") model_path = next();
        else if (a == "--depth") depth = std::stoul(next());
        else if (a == "--threshold") threshold = std::stoul(next());
        else if (a == "--dtw") dtw = true;
        else if (a == "--dtw-target") dtw_target = true;
        else if (a == "--warp") warp = true;
        else if (a == "--partition-only") partition_only = true;
        else if (a == "--matcher") dict_dir = next(), query_dir = next();
        else if (a == "--matcher-loop") dict_dir = next(), query_dir = next(), matcher_loop = true;
        else if (a == "--locate") locate = true;
        else if (a == "--morph") morph = true;
        else if (a == "--chain") chain = std::stoul(next());
        else if (a == "--write-splits") splits_dir = next();
    }
    try {
        if (matcher_loop) {
            // examples/matcher.rs:18-56 literally: ONE match_sound (nq = 1) per query file, silence below max_power 0.03, the
            // matched samples zero-padded / truncated to the query's length and scaled by i16::MAX * 4^max_power
            auto dictionary = SoundDictionary::from_path(dict_dir);
            dictionary->mode = dtw ? SS_DTW : SS_COSINE_REF;
            auto queries = SoundDictionary::from_path(query_dir);  // the directory listing + Sound::from_path of every file
            std::vector<int16_t> concat;
            printf("{\"matches\": [");
            bool first = true;
            for (auto& phoneme : queries->sounds) {
                if (phoneme->max_power() < 0.03) {
                    concat.insert(concat.end(), phoneme->samples().size(), 0);
                    continue;
                }
                auto sound = dictionary->match_sound(phoneme);
                const std::vector<double>& smp = sound->samples();
                const double gain = 32767.0 * std::pow(4.0, phoneme->max_power());
                for (size_t i = 0; i < phoneme->samples().size(); i++) {
                    const double v = (i < smp.size() ? smp[i] : 0.0) * gain;  // `as i16`: truncate toward zero, saturate, NaN -> 0
                    concat.push_back(v != v ? 0 : (v >= 32767.0 ? 32767 : (v <= -32768.0 ? -32768 : (int16_t)v)));
                }
                printf("%s[\"%s\", \"%s\"]", first ? "" : ",", phoneme->name.value_or("").c_str(), sound->name.value_or("").c_str());
                first = false;
            }
            long long sum = 0;
            for (int16_t v : concat) sum += v;
            printf("], \"concat_len\": %zu, \"concat_sum\": %lld}\n", concat.size(), sum);
            return 0;
        }
        if (!dict_dir.empty() && locate) {
            // --matcher <dictionary dir> <query dir> --locate: where inside the dictionary files every query file occurs
            // (SoundDictionary::locate, k = 1), as [query, dictionary sound, first frame, last frame, cost]
            auto dictionary = SoundDictionary::from_path(dict_dir);
            auto queries = SoundDictionary::from_path(query_dir);
            std::vector<uint32_t> idx, first, last;
            std::vector<double> cost;
            dictionary->locate(queries->sounds, 1, &idx, &first, &last, &cost);
            printf("{\"located\": [");
            for (size_t i = 0; i < queries->sounds.size(); i++)
                printf("%s[\"%s\", \"%s\", %u, %u, %.17g]", i ? "," : "", queries->sounds[i]->name.value_or("").c_str(),
                       idx[i] < dictionary->sounds.size() ? dictionary->sounds[idx[i]]->name.value_or("").c_str() : "", first[i], last[i], cost[i]);
            printf("]}\n");
            return 0;
        }
        if (!dict_dir.empty()) {
            // examples/matcher.rs:19-52: a dictionary of whole files, every query file matched against it unless it is
            // quieter than 0.03 (then silence); here the queries are matched in ONE batched call
            auto dictionary = SoundDictionary::from_path(dict_dir);
            dictionary->mode = dtw ? SS_DTW : SS_COSINE_REF;
            auto queries = SoundDictionary::from_path(query_dir);
            std::vector<std::shared_ptr<Sound>> loud;
            for (auto& q : queries->sounds)
                if (!(q->max_power() < 0.03)) loud.push_back(q);
            std::vector<uint32_t> idx;
            std::vector<double> dist;
            if (!loud.empty()) dictionary->match_indices(loud, {}, 1, &idx, &dist);
            printf("{\"dictionary\": %zu, \"queries\": %zu, \"silent\": %zu, \"matches\": [", dictionary->sounds.size(), queries->sounds.size(),
                   queries->sounds.size() - loud.size());
            for (size_t i = 0; i < loud.size(); i++)
                printf("%s[\"%s\", \"%s\"]", i ? "," : "", loud[i]->name.value_or("").c_str(), dictionary->sounds[idx[i]]->name.value_or("").c_str());
            printf("]}\n");
            return 0;
        }
        auto source = std::make_shared<Sound>(Sound::from_path(src));
        Partitioner partitioner(source);
        partitioner.set_threshold(threshold).set_depth(depth);
        if (!model_path.empty()) partitioner.train(GaussianMixtureModel::load(model_path));
        const std::vector<size_t> splits = partitioner.partition();  // "Must first train model" without -m
        if (!splits_dir.empty()) write_splits(*source, splits, splits_dir);  // examples/partition.rs:76
        if (partition_only) {
            printf("{\"source_frames\": %zu, \"max_power\": %.17g, \"nsplits\": %zu, \"splits\": [", source->num_frames(), source->max_power(), splits.size());
            for (size_t i = 0; i < splits.size(); i++) printf("%s%zu", i ? "," : "", splits[i]);
            printf("]}\n");
            return 0;
        }
        auto dictionary = SoundDictionary::from_segments(*source, splits);
        dictionary->mode = dtw_target ? SS_DTW_TARGET : (dtw ? SS_DTW : SS_COSINE_REF);

        auto target = std::make_shared<Sound>(Sound::from_path(tgt));
        partitioner.sound = target;
        const std::vector<size_t> tsplits = partitioner.partition();
        std::vector<std::shared_ptr<Sound>> segments = Sound::cut(*target, tsplits, target->context());  // examples/reconstruction.rs:77-81
        SoundSequence sequence(segments);
        if (morph) {
            // SoundSequence::morph_to (src/sound.rs:440-449) with target distances spread over the similarity range, and
            // SoundSequence::from_distances (:405-417): a chain of `chain` nq = 1 matches starting from the first segment
            auto index_of = [&](const std::shared_ptr<Sound>& s) {
                for (size_t i = 0; i < dictionary->sounds.size(); i++)
                    if (dictionary->sounds[i] == s) return (long long)i;
                return -1ll;
            };
            std::vector<double> distances(segments.size());
            for (size_t i = 0; i < distances.size(); i++) distances[i] = -1e-4 + 2e-4 * (double)i / (double)std::max<size_t>(distances.size() - 1, 1);
            std::vector<double> steps(chain);
            for (size_t i = 0; i < chain; i++) steps[i] = (i % 2 ? -1.0 : 1.0) * 5e-5 * (double)(i + 1) / (double)chain;
            if (dtw_target) {
                // DTW distances from [lo, 2 hi], lo / hi the smallest / largest nearest-match distance of the target's segments
                std::vector<uint32_t> nidx;
                std::vector<double> ndist;
                dictionary->match_indices(segments, {}, 1, &nidx, &ndist);
                double lo = INFINITY, hi = 0.0;
                for (double v : ndist)
                    if (std::isfinite(v)) lo = std::min(lo, v), hi = std::max(hi, v);
                if (!(lo <= hi)) lo = hi = 0.0;
                for (size_t i = 0; i < distances.size(); i++) distances[i] = lo + (2.0 * hi - lo) * (double)i / (double)std::max<size_t>(distances.size() - 1, 1);
                for (size_t i = 0; i < chain; i++) steps[i] = lo + (2.0 * hi - lo) * (double)(i + 1) / (double)chain;
            }
            SoundSequence morphed = sequence.morph_to(distances, *dictionary);
            SoundSequence chained = SoundSequence::from_distances(steps, segments.at(0), *dictionary);
            printf("{");
            if (dtw_target) {
                printf("\"targets\": [");
                for (size_t i = 0; i < distances.size(); i++) printf("%s%.17g", i ? "," : "", distances[i]);
                printf("], \"steps\": [");
                for (size_t i = 0; i < chain; i++) printf("%s%.17g", i ? "," : "", steps[i]);
                printf("], ");
            }
            printf("\"morph\": [");
            for (size_t i = 0; i < morphed.sounds().size(); i++) printf("%s%lld", i ? "," : "", index_of(morphed.sounds()[i]));
            printf("], \"chain\": [");
            for (size_t i = 1; i < chained.sounds().size(); i++) printf("%s%lld", i > 1 ? "," : "", index_of(chained.sounds()[i]));
            printf("], \"chain_distances\": [");
            for (size_t i = 0; i < chained.distances().size(); i++) printf("%s%.17g", i ? "," : "", chained.distances()[i]);
            printf("]}\n");
            return 0;
        }
        std::vector<uint32_t> idx;
        Sound result = sequence.clone_from_dictionary_to_sound(*dictionary, &idx, warp);
        if (!out.empty()) result.write_file(out);
        double sum = 0;
        for (double s : result.samples()) sum += s;
        printf("{\"nsplits\": %zu, \"ntarget\": %zu, \"out_samples\": %zu, \"out_sum\": %.17g, \"out_frames\": %zu, \"idx\": [", splits.size(),
               tsplits.size(), result.samples().size(), sum, result.num_frames());
        for (size_t i = 0; i < idx.size(); i++) printf("%s%u", i ? "," : "", idx[i]);
        printf("]}\n");
    } catch (const CosError& e) {
        printf("{\"error\": \"%s\", \"code\": %d}\n", e.what(), e.code);
        return 1;
    }
    return 0;
}
