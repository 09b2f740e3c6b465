"""Mint the golden fixtures under tests/golden/ (run in the authoring container, where /root/reference and
torchaudio are present; the GPU box has neither the reference checkout nor a need for it).

The reference ships no golden vectors (SURVEY.md §4, "parity unpinned").  What is pinned here:
  fbank_wavs.npz   int16 samples of the reference's bundled wavs (dataset/a_1,a_2,b_1,b_2.wav and a 3 s crop of
                   test_long.wav) + torchaudio.compliance.kaldi.fbank(sample_frequency=16000, num_mel_bins=80)
                   of the [-1,1)-scaled samples -- the upstream implementation paddleaudio's kaldi.fbank mirrors.
  fbank_synth.npz  seeded synthetic [4,48000] batch -> torchaudio fbank, and the oracle's AudioFeaturizer output
                   with a lens-ratio mask.
  ecapa_seed1000.npz  oracle (fp64) ECAPA-TDNN embeddings for seeded weights / inputs, B=3, T in {98, 298}.
  head_seed1000.npz   AAM loss / gradients (torch autograd, fp64) and a 17x23 cosine matrix.
Usage:  python tests/golden/make_golden.py
"""
import os
import sys
import wave

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import campplus, ecapa, eres2net, fbank, head, resnet_se  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"


def read_wav_int16(path):
    with wave.open(path) as w:
        assert w.getsampwidth() == 2 and w.getnchannels() == 1 and w.getframerate() == 16000
        return np.frombuffer(w.readframes(w.getnframes()), dtype=np.int16).copy()


def savez_lzma(path, arrays):
    """np.savez with LZMA-compressed members (np.load reads them as usual): the int16 PCM and float32 features pack ~9 % tighter
    than with deflate, which keeps fbank_wavs.npz under 1 MB."""
    import io
    import zipfile
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_LZMA) as z:
        for k, a in arrays.items():
            buf = io.BytesIO()
            np.lib.format.write_array(buf, np.asanyarray(a))
            z.writestr(k + ".npy", buf.getvalue())


def ta_fbank(x):
    import torchaudio.compliance.kaldi as K
    return K.fbank(torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32))[None], sample_frequency=16000.0,
                   num_mel_bins=80).numpy()


def main():
    # ---- bundled wavs
    d = {}
    for name in ["a_1", "a_2", "b_1", "b_2"]:
        s = read_wav_int16(f"{REF}/dataset/{name}.wav")
        d[name + "_pcm"] = s
        d[name + "_fbank"] = ta_fbank(s.astype(np.float32) / 32768.0)
    s = read_wav_int16(f"{REF}/dataset/test_long.wav")[160000:160000 + 48000]
    d["long3s_pcm"] = s
    d["long3s_fbank"] = ta_fbank(s.astype(np.float32) / 32768.0)
    savez_lzma(f"{OUT}/fbank_wavs.npz", d)
    print({k: v.shape for k, v in d.items()})

    # ---- synthetic batch (SURVEY.md §8d config 2 recipe, 4 utterances)
    g = torch.Generator().manual_seed(1000)
    x = (0.1 * torch.randn(4, 48000, generator=g)).clamp(-1, 1).numpy()
    ref = np.stack([ta_fbank(u) for u in x])
    ratio = np.array([1.0, 0.75, 0.5, 0.3], dtype=np.float32)
    feat = fbank.audio_featurizer_fbank(x, ratio, dtype=np.float64, n_mels=80)
    np.savez_compressed(f"{OUT}/fbank_synth.npz", fbank=ref.astype(np.float32), ratio=ratio,
                        featurizer_masked=feat.astype(np.float32))

    # ---- ECAPA embeddings (fp64 oracle)
    W = ecapa.make_ecapa_weights(seed=1000, dtype=torch.float64)
    e = {}
    for T in (98, 298):
        gi = torch.Generator().manual_seed(1000 + T)
        f = torch.randn(3, T, 80, generator=gi, dtype=torch.float64)
        f = f - f.mean(1, keepdim=True)
        taps = {}
        emb = ecapa.ecapa_forward(f, W, taps=taps)
        e[f"emb_T{T}"] = emb.numpy()
        for k, v in taps.items():
            e[f"tap_{k}_T{T}_absmean"] = np.array(v.abs().mean().item())
    np.savez_compressed(f"{OUT}/ecapa_seed1000.npz", **e)
    print({k: (v.shape, float(np.abs(v).mean())) for k, v in e.items()})

    # ---- ResNetSE embeddings (fp64 oracle)
    Wr = resnet_se.make_resnet_se_weights(seed=1000, dtype=torch.float64)
    r = {}
    for T in (64, 149):
        gi = torch.Generator().manual_seed(2000 + T)
        f = torch.randn(2, T, 80, generator=gi, dtype=torch.float64)
        f = f - f.mean(1, keepdim=True)
        r[f"emb_T{T}"] = resnet_se.resnet_se_forward(f, Wr).numpy()
    np.savez_compressed(f"{OUT}/resnetse_seed1000.npz", **r)

    # ---- ERes2Net embeddings (fp64 oracle)
    We = eres2net.make_eres2net_weights(seed=1000, dtype=torch.float64)
    r = {}
    for T in (64, 149):
        gi = torch.Generator().manual_seed(3000 + T)
        f = torch.randn(2, T, 80, generator=gi, dtype=torch.float64)
        f = f - f.mean(1, keepdim=True)
        r[f"emb_T{T}"] = eres2net.eres2net_forward(f, We).numpy()
    np.savez_compressed(f"{OUT}/eres2net_seed1000.npz", **r)

    # ---- CAM++ embeddings (fp64 oracle)
    Wc_ = campplus.make_campplus_weights(seed=1000, dtype=torch.float64)
    r = {}
    for T in (64, 298, 451):
        gi = torch.Generator().manual_seed(4000 + T)
        f = torch.randn(2, T, 80, generator=gi, dtype=torch.float64)
        f = f - f.mean(1, keepdim=True)
        r[f"emb_T{T}"] = campplus.campplus_forward(f, Wc_).numpy()
    np.savez_compressed(f"{OUT}/campplus_seed1000.npz", **r)

    # ---- head: AAM + cosine
    g = torch.Generator().manual_seed(1000)
    B, D, S = 8, 192, 157
    emb = torch.randn(B, D, generator=g, dtype=torch.float64)
    Wc = (torch.rand(D, S, generator=g, dtype=torch.float64) * 2 - 1) * (6.0 / (D + S)) ** 0.5
    labels = torch.randint(0, S, (B,), generator=g)
    # make two rows nearly aligned with their class centre so the th / mmm branch and phi branch are both hit
    emb[0] = Wc[:, labels[0]] * 3 + 0.05 * emb[0]
    emb[1] = -Wc[:, labels[1]] * 3 + 0.01 * emb[1]
    h = {"emb": emb.numpy(), "W": Wc.numpy(), "labels": labels.numpy()}
    for margin, ls in [(0.0, 0.0), (0.2, 0.0), (0.3, 0.1)]:
        e_ = emb.clone().requires_grad_(True)
        w_ = Wc.clone().requires_grad_(True)
        logits = head.cosine_logits(e_, w_)
        loss = head.aam_loss(logits, labels, margin=margin, scale=32.0, label_smoothing=ls)
        loss.backward()
        tag = f"m{margin}_ls{ls}"
        h[f"logits"] = logits.detach().numpy()
        h[f"loss_{tag}"] = np.array(loss.item())
        h[f"demb_{tag}"] = e_.grad.numpy()
        h[f"dW_{tag}"] = w_.grad.numpy().astype(np.float32)
    A = torch.randn(17, 192, generator=g, dtype=torch.float64).numpy()
    Bm = torch.randn(23, 192, generator=g, dtype=torch.float64).numpy()
    h["cos_A"], h["cos_B"], h["cos_AB"] = A, Bm, head.cosine_matrix(A, Bm)
    np.savez_compressed(f"{OUT}/head_seed1000.npz", **h)

    # ---- EER / minDCF: produced by the REFERENCE's own ppvector/metric/metrics.py (pure numpy, importable here)
    import importlib.util
    spec = importlib.util.spec_from_file_location("ref_metrics", f"{REF}/ppvector/metric/metrics.py")
    ref_metrics = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref_metrics)
    rng = np.random.default_rng(1000)
    scores = rng.standard_normal(5000).astype(np.float32) * 0.2
    labels = (rng.random(5000) < 0.05).astype(np.int32)
    scores[labels == 1] += 0.45
    fnr, fpr, thr = ref_metrics.compute_fnr_fpr(scores, labels)
    eer, eer_thr = ref_metrics.compute_eer(fnr, fpr, scores)
    np.savez_compressed(f"{OUT}/metrics_ref.npz", scores=scores, labels=labels, eer=float(eer), threshold=float(eer_thr),
                        min_dcf=float(ref_metrics.compute_dcf(fnr, fpr)), fnr_head=fnr[:50], fpr_tail=fpr[-50:])
    print("losses", {k: float(v) for k, v in h.items() if k.startswith("loss")})


if __name__ == "__main__":
    main()
