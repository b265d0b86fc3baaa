"""ORACLE helper (authoring container only): writes tests/golden/*.npz from the REFERENCE'S OWN code
(imported by oracle/ref_import.py from /root/reference/src) and from the oracle networks.

    python oracle/make_golden.py

Fixtures
  cluster_traces.npz   speaker maps + centroid digests produced by the reference's
                       OnlineSpeakerClustering on the seeded streams of oracle/synth_cluster.py
  functional_kats.npz  overlapped_speech_penalty / OverlappedSpeechPenalty(normalize) /
                       normalize_embeddings known answers from reference functional.py, blocks/embedding.py
  nets.npz             segmentation scores and unit-norm embeddings of the oracle networks, computed
                       THROUGH the reference's SpeakerSegmentation / OverlapAwareSpeakerEmbedding blocks
  net_layers.npz       per-layer fingerprints (mean, std, |max|, 32 samples) of PyanNet / XVectorSincNet / the powerset
                       PyanNet / WeSpeakerResNet34 on one seeded chunk (SURVEY.md 8(c) golden kind 1); needs no reference tree:
                       python oracle/make_golden.py --layers
  reference_blocks.npz what the reference's own OnlineSpeakerClustering, DelayedAggregation, Binarize,
                       TemporalFeatureFormatter, AdjustVolume and Resample return on seeded inputs: per-chunk digests of the
                       clustering, full aggregation outputs, seeded samples of the waveform outputs; alone:
                       python oracle/make_golden.py --reference-blocks
"""
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from diart_b200 import synth  # noqa: E402
from diart_b200.core import SlidingWindow, SlidingWindowFeature  # noqa: E402
from oracle import nets, ref_import  # noqa: E402
from oracle.synth_cluster import make_stream  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
CLUSTER_CONFIGS = [  # (seed, max_speakers, sigma, delta, tau, rho, K, n_chunks)
    (0, 20, 1.2, 1.0, 0.6, 0.3, 3, 400), (1, 4, 1.2, 1.0, 0.6, 0.3, 3, 400), (2, 20, 2.5, 0.8, 0.5, 0.3, 3, 400),
    (3, 6, 3.0, 0.7, 0.6, 0.2, 3, 400), (4, 3, 1.0, 1.0, 0.6, 0.3, 3, 400), (5, 20, 0.5, 0.3, 0.6, 0.3, 3, 400),
    (6, 20, 1.5, 0.9, 0.6, 0.3, 4, 400), (7, 5, 2.0, 0.9, 0.55, 0.25, 4, 400),
]


def digest(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def fingerprint(t: torch.Tensor) -> np.ndarray:
    a = t.detach().double().reshape(-1)
    idx = torch.linspace(0, a.numel() - 1, 32).long()
    return np.concatenate([[a.mean().item(), a.std().item(), a.abs().max().item()], a[idx].numpy()])


def layer_fingerprints() -> dict:
    """{tap name: fingerprint} of the four oracle networks on window 0 of synth_audio(seed=1234)"""
    x = torch.from_numpy(synth.windows(synth.synth_audio(80000 + 8000, seed=1234), 1))[:, None, :]
    w = torch.rand(1, 293, generator=torch.Generator().manual_seed(7))
    out = {}
    with torch.no_grad():
        taps = {}
        out["seg/out"] = fingerprint(nets.make_segmentation()(x, taps))
        out.update({f"seg/{k}": fingerprint(v) for k, v in taps.items()})
        taps = {}
        emb = nets.make_embedding()
        trunk = emb.trunk(x, taps)
        out.update({f"emb/{k}": fingerprint(v) for k, v in taps.items()})
        out["emb/out_weighted"] = fingerprint(emb.embedding(emb.stats_pool(trunk, w)))
        taps = {}
        nets.make_powerset_segmentation()(x, taps)
        out["powerset/log_probabilities"] = fingerprint(taps["log_probabilities"])
        wes = nets.make_wespeaker()
        fb = wes.compute_fbank(x)
        out["wespeaker/fbank"] = fingerprint(fb)
        out["wespeaker/maps"] = fingerprint(wes.resnet.maps(fb))
        out["wespeaker/out_weighted"] = fingerprint(wes(x, w))
    return out


# ---- reference_blocks.npz: each function below takes the classes to run (the reference's or this project's), so the
# golden file and tests/test_oracle_vs_reference.py evaluate exactly the same inputs
CLASS_CONFIGS = [(20, 1.2, 1.0, 0.6, 0.3), (4, 1.2, 1.0, 0.6, 0.3), (6, 3.0, 0.7, 0.6, 0.2), (20, 0.5, 0.3, 0.6, 0.3)]
CLASS_CHUNKS = 250          # config i = (max_speakers, sigma, delta, tau, rho) clusters make_stream(CLASS_CHUNKS, 100 + i, sigma)
WAVEFORM_SAMPLES = 1024     # values kept per waveform output (in full, the six are ~0.5 MB of incompressible floats)


def value_digest(a) -> np.ndarray:
    """first 16 bytes of sha256 over the shape and the float64 values of an array (-0.0 counted as 0.0); None -> digest of b''"""
    h = hashlib.sha256()
    if a is not None:
        a = np.ascontiguousarray(a, dtype=np.float64) + 0.0
        h.update(str(a.shape).encode())
        h.update(a.tobytes())
    return np.frombuffer(h.digest()[:16], dtype=np.uint8)


def waveform_sample(a: np.ndarray) -> np.ndarray:
    """a fixed, seeded sample of WAVEFORM_SAMPLES values of a flattened output"""
    a = np.asarray(a).reshape(-1)
    return a[np.random.default_rng(17).choice(a.size, min(WAVEFORM_SAMPLES, a.size), replace=False)]


def clustering_trace(make, call) -> dict:
    """every chunk of the CLASS_CONFIGS streams through make(tau, rho, delta, "cosine", M); call(clustering, seg, emb) returns
    the permuted scores.  Per chunk: digests of the permuted scores and of the centers, the active centers as a bit mask"""
    out, centers, active = [], [], []
    for i, (M, sigma, delta, tau, rho) in enumerate(CLASS_CONFIGS):
        seg, emb = make_stream(CLASS_CHUNKS, 100 + i, sigma=sigma)
        clu = make(tau, rho, delta, "cosine", M)
        for s, e in zip(seg, emb):
            out.append(value_digest(call(clu, s, e)))
            centers.append(value_digest(clu.centers))
            active.append(sum(1 << int(c) for c in clu.active_centers))
    return {"cluster_out": np.stack(out), "cluster_centers": np.stack(centers), "cluster_active": np.array(active, np.int64)}


def aggregation_outputs(delayed_aggregation, binarize) -> dict:
    """DelayedAggregation(step 0.5) over seeded score buffers: data, output window (start, step), number of overlapping windows,
    and the RTTM text of Binarize(0.6) of the aggregate"""
    rng = np.random.default_rng(3)
    res = 5 / 293
    cases = []
    for latency, n_buf in [(0.5, 1), (2.0, 4), (5.0, 10)]:
        for first in (0, 7):
            cases.append((f"hamming_loose_{latency:g}_{first}", (latency, "hamming", "loose"), n_buf, 5, first))
    cases += [("mean_strict_1.5_3", (1.5, "mean", "strict"), 3, 2, 3), ("first_center_1.5_3", (1.5, "first", "center"), 3, 2, 3)]
    out = {}
    for name, (latency, strategy, mode), n_buf, K, first in cases:
        agg = delayed_aggregation(0.5, latency, strategy, mode)
        bufs = [SlidingWindowFeature(rng.random((293, K)), SlidingWindow(start=0.5 * (first + i), duration=res, step=res))
                for i in range(n_buf)]
        a = agg(bufs)
        out[f"agg_{name}_data"] = a.data
        out[f"agg_{name}_window"] = np.array([a.sliding_window.start, a.sliding_window.step])
        out[f"agg_{name}_num_windows"] = np.array(agg.num_overlapping_windows)
        out[f"agg_{name}_rttm"] = np.array(binarize(0.6)(a).to_rttm())
    return out


def formatter_outputs(formatter) -> dict:
    """TemporalFeatureFormatter: cast of a seeded SlidingWindowFeature, output window of restore_type"""
    f = formatter()
    swf = SlidingWindowFeature(np.random.default_rng(11).random((50, 3)), SlidingWindow(start=1.5, duration=0.1, step=0.1))
    cast = f.cast(swf)
    restored = f.restore_type(torch.ones(1, 25, 2))
    return {"formatter_cast": cast.numpy(), "formatter_restored_window": np.array([restored.sliding_window.start,
                                                                                  restored.sliding_window.step])}


def preprocessing_outputs(adjust_volume, resample) -> dict:
    """AdjustVolume and Resample on seeded waveforms: shape and waveform_sample of every output, Resample's output window"""
    rng = np.random.default_rng(5)
    batch = torch.from_numpy(rng.standard_normal((3, 8000, 1)).astype(np.float32) * 0.05)
    full = {}
    for target in (-20.0, 3.0):
        for level, x in (("quiet", batch), ("loud", batch * 100)):
            full[f"volume_{target:g}_{level}"] = adjust_volume(target)(x).numpy()
    swf = SlidingWindowFeature(batch[0].numpy(), SlidingWindow(start=1.5, duration=1 / 8000, step=1 / 8000))
    up = resample(8000, 16000)(swf)
    full["resample_up"] = up.data
    full["resample_down"] = resample(16000, 8000)(batch).numpy()
    out = {"resample_up_window": np.array([up.sliding_window.start, up.sliding_window.step])}
    for name, a in full.items():
        out[f"{name}_shape"] = np.array(a.shape)
        out[f"{name}_sample"] = waveform_sample(a)
    return out


def reference_blocks(ref) -> dict:
    import importlib

    sw = SlidingWindow(start=0, duration=5 / 293, step=5 / 293)
    utils = importlib.import_module("diart.blocks.utils")
    out = clustering_trace(ref.clustering.OnlineSpeakerClustering,
                           lambda clu, s, e: clu(SlidingWindowFeature(s, sw), torch.from_numpy(e)).data)
    out.update(aggregation_outputs(importlib.import_module("diart.blocks.aggregation").DelayedAggregation, utils.Binarize))
    out.update(formatter_outputs(ref.features.TemporalFeatureFormatter))
    out.update(preprocessing_outputs(utils.AdjustVolume, utils.Resample))
    return out


def main():
    if "--layers" in sys.argv:
        np.savez_compressed(os.path.join(OUT, "net_layers.npz"), **{k.replace("/", "__"): v for k, v in layer_fingerprints().items()})
        print("golden written: net_layers.npz")
        return
    ref = ref_import.load()
    os.makedirs(OUT, exist_ok=True)
    np.savez_compressed(os.path.join(OUT, "reference_blocks.npz"), **reference_blocks(ref))
    if "--reference-blocks" in sys.argv:
        print("golden written: reference_blocks.npz")
        return
    torch.set_num_threads(8)
    # ---- clustering traces from the reference class
    out = {"configs": np.array(CLUSTER_CONFIGS, dtype=np.float64)}
    sw = SlidingWindow(start=0, duration=5 / 293, step=5 / 293)
    for cfg in CLUSTER_CONFIGS:
        seed, M, sigma, delta, tau, rho, K, n = cfg
        seg, emb = make_stream(n, seed, K=K, sigma=sigma)
        clu = ref.clustering.OnlineSpeakerClustering(tau, rho, delta, "cosine", M)
        maps = -np.ones((n, K), dtype=np.int8)
        for i in range(n):
            m = clu.identify(SlidingWindowFeature(seg[i], sw), torch.from_numpy(emb[i]))
            for s, t in zip(*m.valid_assignments()):
                maps[i, s] = t
        out[f"maps_{seed}"] = maps
        out[f"centers_sha_{seed}"] = np.array(digest(clu.centers))
        out[f"centers_head_{seed}"] = clu.centers[:, :4].copy()
        out[f"active_{seed}"] = np.array(sorted(clu.active_centers), dtype=np.int32)
    np.savez_compressed(os.path.join(OUT, "cluster_traces.npz"), **out)
    # ---- functional KATs
    rng = np.random.default_rng(7)
    seg = rng.random((3, 40, 3)).astype(np.float32)
    seg[0, :5] = 1e-4                       # clamp branch
    seg[1, :, 1] = 1e-4                     # whole column clamps to 1e-8: min == max -> NaN -> 1e-8 under normalize
    emb = rng.standard_normal((3, 3, 16)).astype(np.float32)
    F = ref.functional
    kat = {"seg": seg, "emb": emb,
           "osp_3_10": F.overlapped_speech_penalty(torch.from_numpy(seg), 3, 10).numpy(),
           "osp_2_5": F.overlapped_speech_penalty(torch.from_numpy(seg), 2, 5).numpy(),
           "osp_2p5_7": F.overlapped_speech_penalty(torch.from_numpy(seg), 2.5, 7).numpy(),
           "osp_norm": ref.embedding.OverlappedSpeechPenalty(3, 10, normalize=True)(torch.from_numpy(seg)).numpy(),
           "normalize_1": F.normalize_embeddings(torch.from_numpy(emb), 1).numpy(),
           "normalize_2p5": F.normalize_embeddings(torch.from_numpy(emb), 2.5).numpy()}
    np.savez_compressed(os.path.join(OUT, "functional_kats.npz"), **kat)
    # ---- networks through the reference's own blocks (oracle nets behind the loader API)
    seg_net, emb_net = nets.make_segmentation(), nets.make_embedding()
    stream = synth.synth_audio(80000 + 8000 * 7, seed=1234)
    x = synth.windows(stream, 8)[:2]
    seg_block = ref.segmentation.SpeakerSegmentation(ref.models.SegmentationModel(lambda: seg_net), torch.device("cpu"))
    emb_block = ref.embedding.OverlapAwareSpeakerEmbedding(ref.models.EmbeddingModel(lambda: emb_net), 3, 10, 1,
                                                           False, torch.device("cpu"))
    batch = torch.from_numpy(x)[:, :, None]              # (batch, samples, channels) as diarization.py:177 builds it
    s = seg_block(batch)
    e = emb_block(batch, s)
    np.savez_compressed(os.path.join(OUT, "nets.npz"), seg=s.numpy(), emb=e.numpy(),
                        note=np.array("reference SpeakerSegmentation / OverlapAwareSpeakerEmbedding over oracle nets; "
                                      "audio = synth_audio(seed=1234) windows 0..1"))
    print("golden written:", os.listdir(OUT))


if __name__ == "__main__":
    main()
