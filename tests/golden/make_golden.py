"""Generates the committed golden fixtures under tests/golden/ from the reference's own WAV fixtures.

Run HERE (the build container), where /root/reference exists:  python tests/golden/make_golden.py
The GPU box has no /root/reference; tests read only the .npz / .json files this script writes.

What pins what:
  kats.json            known answers taken from the reference's own tests / call sites (src/lib.rs:258 decode KAT,
                       src/sound.rs:612-615 angular KAT, vox_box dct KAT quoted in SURVEY.md §8a-5, frame-count rule)
  section71.npz        tests/Section_7_1.wav PCM + oracle outputs for every stage of config 2 (MFCC, max_power, mean,
                       seeded model, symbols, votes, splits)
  sample_excerpt.npz   first 12 s of tests/sample.wav (24-bit) + oracle outputs, incl. config 1's matches against the
                       Section_7_1 dictionary in both matcher modes
  synthetic_small.npz  seeded synthetic dictionary x queries (config-3 generator, small) with oracle top-k
Each oracle output was cross-checked against oracle/numpy_twin.py by tests/test_oracle.py before being trusted.
"""
import json
import os
import sys
import zipfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import numpy_twin as T  # noqa: E402
from oracle import oracle as O  # noqa: E402
from soundsym_b200 import synth  # noqa: E402

REF = "/root/reference/tests"
OUT = os.path.dirname(os.path.abspath(__file__))


def savez_lzma(path, **arrays):
    """np.savez with LZMA-compressed members, which np.load reads like any .npz: the PCM of the two WAV fixtures
    compresses to under 1 MB per file this way (deflate leaves sample_excerpt.npz at 1.2 MB)."""
    with zipfile.ZipFile(path, "w", zipfile.ZIP_LZMA) as z:
        for name, a in arrays.items():
            with z.open(name + ".npy", "w", force_zip64=True) as f:
                np.lib.format.write_array(f, np.asanyarray(a))


def cut(mfcc, seg_lens_samples, hop=256):
    """SoundDictionary::add_segments (src/sound.rs:330-343): segment i takes seg_i/HOP frames of the MFCC stream."""
    frames = (np.asarray(seg_lens_samples, dtype=np.uint64) // np.uint64(hop)).astype(np.uint64)
    off = np.zeros(len(frames) + 1, dtype=np.uint64)
    off[1:] = np.cumsum(frames)
    return mfcc[: int(off[-1])], off


def main():
    O.set_threads(8)
    # ---- Section_7_1.wav : config 2 -------------------------------------------------------------------------------
    s71, sr71, bits71, pcm71 = T.read_wav(os.path.join(REF, "Section_7_1.wav"))
    m71 = O.mfcc(s71, sr71)
    z71, _, _ = O.standardize(m71)
    model = O.gmm_train(z71, seed=0)  # train_model (src/lib.rs:44-54), seeded
    sym71 = O.symbols(m71, *model)
    g = dict(pcm=pcm71.astype(np.int16), bits=np.int32(bits71), sample_rate=np.float64(sr71), mfcc=m71,
             max_power=np.float64(O.max_power(s71)), mean_mfccs=O.mean_mfccs(m71),
             gmm_means=model[0], gmm_covs=model[1], gmm_weights=model[2], symbols=sym71)
    for depth, thr in ((3, 4), (4, 3), (5, 4)):  # reconstruction.rs:44-45, partition.rs:65-68, Partitioner::new defaults
        votes = O.cast_votes(sym71, depth)
        g["votes_d%d" % depth] = votes
        g["splits_d%dt%d" % (depth, thr)] = O.split(votes, len(sym71), thr) * np.uint64(256)
    savez_lzma(os.path.join(OUT, "section71.npz"), **g)

    # ---- sample.wav excerpt : config 1 ----------------------------------------------------------------------------
    s, sr, bits, pcm = T.read_wav(os.path.join(REF, "sample.wav"))
    full_max_abs = float(np.abs(s).max())
    full_max_power = O.max_power(s)
    full_frames = O.frame_count(len(s))
    n_ex = 12 * 44100
    s_ex, pcm_ex = s[:n_ex], pcm[:n_ex]
    m_ex = O.mfcc(s_ex, sr)
    sym_ex = O.symbols(m_ex, *model)  # partition_other with the source's model (reconstruction.rs:71-77)
    splits_ex = O.split(O.cast_votes(sym_ex, 3), len(sym_ex), 4) * np.uint64(256)
    dict_mfcc, dict_off = cut(m71, g["splits_d3t4"])
    q_mfcc, q_off = cut(m_ex, splits_ex)
    # matcher.rs:40 gates silent queries with max_power < 0.03
    q_pow = np.array([O.max_power(s_ex[int(a) * 256:int(b) * 256]) for a, b in zip(q_off[:-1], q_off[1:])])
    cos_idx, cos_dist = O.cosine_match(dict_mfcc, dict_off, q_mfcc, q_off, 12)
    dtw_idx, dtw_dist = O.dtw_topk(dict_mfcc, dict_off, q_mfcc, q_off, 12, k=4)
    # resynthesis (clone_from_dictionary + to_sound) with the cosine-ref matches
    samp_off = np.zeros(len(g["splits_d3t4"]) + 1, dtype=np.uint64)
    samp_off[1:] = np.cumsum(g["splits_d3t4"])
    resyn = O.resynth(s71, samp_off, cos_idx, splits_ex)
    savez_lzma(os.path.join(OUT, "sample_excerpt.npz"), pcm=pcm_ex.astype(np.int32), bits=np.int32(bits),
               sample_rate=np.float64(sr), mfcc=m_ex, max_power=np.float64(O.max_power(s_ex)), symbols=sym_ex,
               splits_d3t4=splits_ex, q_max_power=q_pow, cos_idx=cos_idx, cos_dist=cos_dist, dtw_idx=dtw_idx,
               dtw_dist=dtw_dist, resynth_head=resyn[:65536], resynth_sum=np.float64(resyn.sum()),
               resynth_len=np.uint64(len(resyn)))

    # ---- synthetic small : config-3 generator ----------------------------------------------------------------------
    d, doff = synth.segments(600, 13, seed=1234)
    q, qoff = synth.segments(48, 13, seed=5678)
    di, dd = O.dtw_topk(d, doff, q, qoff, 13, k=4)
    ci, cd = O.cosine_match(d, doff, q, qoff, 13)
    savez_lzma(os.path.join(OUT, "synthetic_small.npz"), dtw_idx=di, dtw_dist=dd, cos_idx=ci, cos_dist=cd,
               dict_checksum=np.float64(d.sum()), q_checksum=np.float64(q.sum()))

    kats = {
        "decode_24bit_max_abs_sample_wav": {"value": full_max_abs, "expected": 0.6503654301602161, "tol": 1e-9,
                                            "source": "src/lib.rs:258"},
        "max_power_sample_wav_head_constants": {"value": full_max_power, "expected": 0.3263162680772736, "tol": 1e-12,
                                                "source": "src/sound.rs:244-256 evaluated at HEAD constants (SURVEY §4; the "
                                                          "value pinned at src/lib.rs:259 is stale)"},
        "frames_sample_wav": {"value": full_frames, "expected": 4540, "source": "SURVEY §8 size table"},
        "frames_section71": {"value": int(m71.shape[0]), "expected": 1978, "source": "SURVEY §8 size table"},
        "angular_kat": {"value": O.cosine_sim_angular([.1, .4, .2, .8] + [0.] * 8, [.1, .4, .2, .8] + [0.] * 8),
                        "expected": 0.0, "source": "src/sound.rs:612-615"},
        "dct_kat": {"value": list(O.dct([.2, .3, .4, .3])), "expected": [2.4, -0.26131, -0.28284, 0.10823], "tol": 1e-5,
                    "source": "vox_box dct test vector, SURVEY §8a-5"},
        "mel_bins_c12": {"value": [int(b) for b in O.mel_bins(12)],
                         "expected": [2, 6, 11, 17, 24, 33, 45, 58, 75, 95, 119, 149, 185, 230], "source": "SURVEY §8a-5"},
        "mel_bins_c13": {"value": [int(b) for b in O.mel_bins(13)],
                         "expected": [2, 6, 10, 15, 22, 30, 39, 50, 64, 80, 100, 123, 152, 185, 226], "source": "SURVEY §8a-5"},
    }
    with open(os.path.join(OUT, "kats.json"), "w") as f:
        json.dump(kats, f, indent=1)
    for k, v in kats.items():
        print(k, v["value"], "expected", v["expected"])
    print("dict segs", len(dict_off) - 1, "queries", len(q_off) - 1, "non-silent", int((q_pow >= 0.03).sum()),
          "max dict len", int(np.diff(dict_off).max()), "max q len", int(np.diff(q_off).max()))


if __name__ == "__main__":
    main()
