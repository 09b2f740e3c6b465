"""Mint reference-derived fixtures: run the reference's OWN model / loss / scheduler code (imported unmodified
from /root/reference under tests/paddle_shim) on seeded weights and inputs, in fp64, and record what it computes.

Runs only in the authoring container (needs /root/reference).  Output: tests/golden/ref_*.npz, consumed by
tests/test_oracle_vs_reference.py on any machine.  The files hold reference OUTPUTS only; weights and inputs are
re-derived from seeds by the consumer (oracle.make_*_weights and `feats()` below), so agreement also pins
parameter names and shapes (set_state_dict refuses missing / extra / mis-shaped keys).

Usage:  python tests/golden/make_ref_fixtures.py            (rewrites the fixtures and ref_digests.json)
        python tests/golden/make_ref_fixtures.py --check    (recomputes and compares with the committed files)
ref_digests.json records a SHA-256 of every array the reference's code computed; tests/test_oracle_vs_reference.py checks
the committed fixtures against it without needing the reference.
"""
import hashlib
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("PPV_REFERENCE", "/root/reference")
sys.path[:0] = [os.path.join(ROOT, "tests", "paddle_shim"), REF, ROOT]
torch.set_default_dtype(torch.float64)

import paddle  # noqa: E402  (the shim)
from ppvector.loss.aamloss import AAMLoss  # noqa: E402  (the REFERENCE's files from here on)
from ppvector.loss.amloss import AMLoss  # noqa: E402
from ppvector.loss.armloss import ARMLoss  # noqa: E402
from ppvector.loss.celoss import CELoss  # noqa: E402
from ppvector.loss.sphereface2 import SphereFace2  # noqa: E402
from ppvector.loss.subcenterloss import SubCenterLoss  # noqa: E402
from ppvector.models.campplus import CAMPPlus  # noqa: E402
from ppvector.models.ecapa_tdnn import EcapaTdnn  # noqa: E402
from ppvector.models.eres2net import ERes2Net, ERes2NetV2  # noqa: E402
from ppvector.models.fc import SpeakerIdentification  # noqa: E402
from ppvector.models.resnet_se import ResNetSE  # noqa: E402
from ppvector.optimizer.scheduler import MarginScheduler, cosine_decay_with_warmup  # noqa: E402

import ppvector  # noqa: E402

assert os.path.realpath(ppvector.__file__).startswith(os.path.realpath(REF)), ppvector.__file__

from oracle import campplus as o_campplus  # noqa: E402
from oracle import ecapa as o_ecapa  # noqa: E402
from oracle import eres2net as o_eres2net  # noqa: E402
from oracle import resnet_se as o_resnet  # noqa: E402

SEEDS = {"ecapa": 1000, "resnetse": 2000, "eres2net": 3000, "campplus": 4000}


def feats(model, T, B=2):
    """Seeded, time-mean-subtracted features [B,T,80] (same recipe as tests/golden/make_golden.py)."""
    g = torch.Generator().manual_seed(SEEDS[model] + T)
    f = torch.randn(B, T, 80, generator=g, dtype=torch.float64)
    return f - f.mean(1, keepdim=True)


def tap_slice(t):
    """A small deterministic view of an intermediate activation (keeps the fixture files small)."""
    t = t.detach()
    idx = tuple(slice(0, min(n, 6)) for n in t.shape)
    return np.concatenate([t[idx].reshape(-1).numpy(), [float(t.abs().mean()), float(t.sum())]])


def hook_taps(model, names):
    taps = {}
    mods = dict(model.named_modules())
    hs = [mods[n].register_forward_hook(lambda m, i, o, n=n: taps.__setitem__(n, o)) for n in names]
    return taps, hs


def run(model, W, x, tap_names=(), **kw):
    model.set_state_dict(W)
    model.eval()
    taps, hs = hook_taps(model, tap_names)
    with torch.no_grad():
        emb = model(paddle.to_tensor(x), **kw)
    for h in hs:
        h.remove()
    return emb.numpy(), {k: tap_slice(v) for k, v in taps.items()}


def models_fixture():
    d = {}
    # ---- ECAPA-TDNN (ecapa_tdnn.py:145-276), all pooling heads, lengths, global_context off, a shortcut-conv variant
    W = o_ecapa.make_ecapa_weights(seed=1000, dtype=torch.float64)
    tap_names = ["blocks.0", "blocks.1.tdnn1", "blocks.1.res2net_block", "blocks.1.tdnn2", "blocks.1", "blocks.2", "blocks.3", "mfa", "asp"]
    for T in (98, 298):
        emb, taps = run(EcapaTdnn(input_size=80), W, feats("ecapa", T), tap_names)
        d[f"ecapa_T{T}_emb"] = emb
        for k, v in taps.items():
            d[f"ecapa_T{T}_tap_{k}"] = v
    lens = torch.tensor([1.0, 0.6])
    d["ecapa_T98_lengths_emb"], _ = run(EcapaTdnn(input_size=80), W, feats("ecapa", 98), lengths=paddle.to_tensor(lens))
    # pooling_type SAP / TAP / TSP: the reference's EcapaTdnn.forward un-squeezes twice (pooling.py:24,46,65 return [N,C,1],
    # ecapa_tdnn.py:272 un-squeezes again) and then calls Conv1d on a 4-D tensor, which raises in Paddle (F.pad 'NCL' needs 3-D,
    # conv1d needs 3-D) -- and under the shim.  Recorded as "raises"; the pooling MODULES themselves are pinned standalone below.
    from ppvector.models.pooling import SelfAttentivePooling, TemporalAveragePooling, TemporalStatisticsPooling
    g = torch.Generator().manual_seed(515)
    xp = torch.randn(2, 1536, 50, generator=g, dtype=torch.float64)
    d["pool_x_seed515_checksum"] = np.array(float(xp.sum()))
    for pt, cls in (("SAP", lambda: SelfAttentivePooling(1536, 128)), ("TAP", TemporalAveragePooling), ("TSP", TemporalStatisticsPooling)):
        Wp = o_ecapa.make_ecapa_weights(seed=1000, dtype=torch.float64, pooling_type=pt)
        try:
            run(EcapaTdnn(input_size=80, pooling_type=pt), Wp, feats("ecapa", 98))
            d[f"ecapa_{pt}_raises"] = np.array(0)
        except Exception as e:  # noqa: BLE001
            print(f"reference EcapaTdnn(pooling_type={pt}) raises {type(e).__name__}: {str(e)[:80]}")
            d[f"ecapa_{pt}_raises"] = np.array(1)
        m = cls()
        m.set_state_dict({k[len("asp."):]: v for k, v in Wp.items() if k.startswith("asp.")})
        m.eval()
        with torch.no_grad():
            d[f"pool_{pt}_out"] = m(paddle.to_tensor(xp)).numpy()
    # ResNetSE with a non-ASP head feeds [N,C,1] into nn.Linear(cat_channels, ...) (resnet_se.py:137): raises as well
    try:
        with torch.no_grad():
            ResNetSE(input_size=80, pooling_type="TAP").eval()(paddle.to_tensor(feats("resnetse", 40)))
        d["resnetse_TAP_raises"] = np.array(0)
    except Exception as e:  # noqa: BLE001
        print(f"reference ResNetSE(pooling_type=TAP) raises {type(e).__name__}: {str(e)[:80]}")
        d["resnetse_TAP_raises"] = np.array(1)
    # ASP with global_context=False (pooling.py:77-78, 108-109)
    Wg = o_ecapa.make_ecapa_weights(seed=1000, dtype=torch.float64, global_context=False)
    d["ecapa_T98_noctx_emb"], _ = run(EcapaTdnn(input_size=80, global_context=False), Wg, feats("ecapa", 98))
    ch = dict(channels=(256, 384, 384, 384, 1152))  # in != out at blocks.1 -> shortcut conv (ecapa_tdnn.py:125-131)
    Ws = o_ecapa.make_ecapa_weights(seed=1000, dtype=torch.float64, **ch)
    d["ecapa_T98_shortcut_emb"], _ = run(EcapaTdnn(input_size=80, channels=list(ch["channels"])), Ws, feats("ecapa", 98))

    # ---- ResNetSE (resnet_se.py:66-139)
    W = o_resnet.make_resnet_se_weights(seed=1000, dtype=torch.float64)
    for T in (98, 298):
        emb, taps = run(ResNetSE(input_size=80), W, feats("resnetse", T), ["relu", "layer1", "layer2", "layer3", "layer4", "pooling"])
        d[f"resnetse_T{T}_emb"] = emb
        for k, v in taps.items():
            d[f"resnetse_T{T}_tap_{k}"] = v
    # ---- ERes2Net (eres2net.py:173-263)
    W = o_eres2net.make_eres2net_weights(seed=1000, dtype=torch.float64)
    for T in (98, 298):
        emb, taps = run(ERes2Net(input_size=80), W, feats("eres2net", T),
                        ["layer1", "layer2", "layer3", "layer4", "fuse_mode12", "fuse_mode123", "fuse_mode1234", "pooling"])
        d[f"eres2net_T{T}_emb"] = emb
        for k, v in taps.items():
            d[f"eres2net_T{T}_tap_{k}"] = v
    # ---- ERes2NetV2 (eres2net.py:266-462): base_width 26 (widths 13 / 26 / 52 / 104), layer3_ds + fuse34
    W = o_eres2net.make_eres2net_weights(seed=1000, dtype=torch.float64, base_width=26, version=2)
    for T in (98, 298):
        emb, taps = run(ERes2NetV2(input_size=80), W, feats("eres2net", T), ["layer1", "layer2", "layer3", "layer4", "fuse34", "pooling"])
        d[f"eres2netv2_T{T}_emb"] = emb
        for k, v in taps.items():
            d[f"eres2netv2_T{T}_tap_{k}"] = v
    # ---- CAM++ (campplus.py:284-335); embd_dim 192 as configs/cam++.yml sets it
    W = o_campplus.make_campplus_weights(seed=1000, dtype=torch.float64)
    for T in (98, 298):
        emb, taps = run(CAMPPlus(input_size=80, embd_dim=192), W, feats("campplus", T),
                        ["head", "xvector.tdnn", "xvector.block1", "xvector.transit1", "xvector.block2", "xvector.transit2",
                         "xvector.block3", "xvector.transit3", "xvector.stats"])
        d[f"campplus_T{T}_emb"] = emb
        for k, v in taps.items():
            d[f"campplus_T{T}_tap_{k}"] = v
    return d


def head_fixture():
    """SpeakerIdentification (fc.py:41-53) + AAMLoss (aamloss.py:28-53) forward / backward through torch autograd."""
    g = torch.Generator().manual_seed(1000)
    B, D, S = 8, 192, 157
    emb = torch.randn(B, D, generator=g, dtype=torch.float64)
    Wc = (torch.rand(D, S, generator=g, dtype=torch.float64) * 2 - 1) * (6.0 / (D + S)) ** 0.5
    labels = torch.randint(0, S, (B,), generator=g)
    emb[0] = Wc[:, labels[0]] * 3 + 0.05 * emb[0]      # phi branch
    emb[1] = -Wc[:, labels[1]] * 3 + 0.01 * emb[1]     # c - mmm branch
    d = {"emb": emb.numpy(), "W": Wc.numpy(), "labels": labels.numpy()}
    clf = SpeakerIdentification(input_dim=D, num_speakers=S)
    clf.set_state_dict({"weight": Wc})
    for margin, ls, easy in [(0.0, 0.0, False), (0.2, 0.0, False), (0.3, 0.1, False), (0.2, 0.0, True)]:
        e = paddle.to_tensor(emb)
        e.requires_grad_(True)
        clf.weight.grad = None
        out = clf(e)
        crit = AAMLoss(margin=margin, scale=32, easy_margin=easy, label_smoothing=ls)
        loss = crit(out, paddle.to_tensor(labels))
        loss.backward()
        tag = f"m{margin}_ls{ls}_easy{int(easy)}"
        d["logits"] = out["logits"].numpy()
        d[f"loss_{tag}"] = np.array(float(loss))
        d[f"demb_{tag}"] = e.grad.numpy()
        d[f"dW_{tag}"] = clf.weight.grad.detach().numpy().copy()
    # the other softmax heads on the same logits: AMLoss (amloss.py), ARMLoss (armloss.py), CELoss (celoss.py)
    for name, crit in [("AM_m0.2_ls0.0", AMLoss(margin=0.2, scale=30, label_smoothing=0.0)), ("AM_m0.35_ls0.1", AMLoss(margin=0.35, scale=30, label_smoothing=0.1)),
                       ("ARM_m0.2_ls0.0", ARMLoss(margin=0.2, scale=30, label_smoothing=0.0)), ("ARM_m0.1_ls0.1", ARMLoss(margin=0.1, scale=30, label_smoothing=0.1)),
                       ("CE_m0.0_ls0.0", CELoss(label_smoothing=0.0)), ("CE_m0.0_ls0.1", CELoss(label_smoothing=0.1))]:
        e = paddle.to_tensor(emb)
        e.requires_grad_(True)
        clf.weight.grad = None
        loss = crit(clf(e), paddle.to_tensor(labels))
        loss.backward()
        d[f"loss_{name}"] = np.array(float(loss))
        d[f"demb_{name}"] = e.grad.numpy()
        d[f"dW_{name}"] = clf.weight.grad.detach().numpy().copy()
    # SubCenterLoss (subcenterloss.py) over a classifier with K sub-centres per class (fc.py:33): the first 156 columns of W as 52 x 3 / 78 x 2
    for K, margin, ls, easy in [(3, 0.2, 0.0, False), (3, 0.3, 0.1, False), (2, 0.2, 0.0, True)]:
        Sk = 156 // K
        clfk = SpeakerIdentification(input_dim=D, num_speakers=Sk, K=K)
        clfk.set_state_dict({"weight": Wc[:, :156].clone()})
        lab = labels % Sk
        e = paddle.to_tensor(emb)
        e.requires_grad_(True)
        loss = SubCenterLoss(margin=margin, scale=32, easy_margin=easy, K=K, label_smoothing=ls)(clfk(e), paddle.to_tensor(lab))
        loss.backward()
        tag = f"SUB_K{K}_m{margin}_ls{ls}_easy{int(easy)}"
        d[f"loss_{tag}"] = np.array(float(loss))
        d[f"demb_{tag}"] = e.grad.numpy()
        d[f"dW_{tag}"] = clfk.weight.grad.detach().numpy().copy()
    # SphereFace2 (sphereface2.py): both margin types
    for mt, margin, lam, t in [("C", 0.2, 0.7, 3), ("A", 0.15, 0.7, 3), ("C", 0.3, 0.5, 2)]:
        e = paddle.to_tensor(emb)
        e.requires_grad_(True)
        clf.weight.grad = None
        loss = SphereFace2(margin=margin, scale=32.0, lanbuda=lam, t=t, margin_type=mt)(clf(e), paddle.to_tensor(labels))
        loss.backward()
        tag = f"SF2{mt}_m{margin}_l{lam}_t{t}"
        d[f"loss_{tag}"] = np.array(float(loss))
        d[f"demb_{tag}"] = e.grad.numpy()
        d[f"dW_{tag}"] = clf.weight.grad.detach().numpy().copy()
    # AAMLoss.update (aamloss.py:48-53) == constructing with that margin
    crit = AAMLoss(margin=0.0, scale=32)
    crit.update(margin=0.25)
    d["update_0.25"] = np.array([crit.cos_m, crit.sin_m, crit.th, crit.mmm])
    for k in [k for k in d if k.startswith("dW_")]:
        d["dWspan_" + k[len("dW_"):]] = span_coefficients(d["emb"], d["W"], d.pop(k))
    return d


def span_coefficients(emb, W, dW):
    """Every head here is a function of the cosine logits, so column j of the classifier's gradient is
    (I - w_j w_j^T / |w_j|^2) / |w_j| * sum_b dlogit_bj * x_b / |x_b|: it lies in the span of the B embedding rows and w_j.
    Store those B + 1 coefficients per column instead of its D entries (the fixture stays under 1 MB); the tests rebuild
    dW = emb^T c[:-1] + W * c[-1] (conftest.py, fixture `ref_head`), checked here against the reference's dW."""
    B, S = emb.shape[0], dW.shape[1]
    c = np.empty((B + 1, S))
    for j in range(S):
        c[:, j] = np.linalg.lstsq(np.concatenate([emb.T, W[:, j:j + 1]], axis=1), dW[:, j], rcond=None)[0]
    err = np.abs(emb.T @ c[:-1] + W[:, :S] * c[-1] - dW).max() / np.abs(dW).max()
    assert err < 1e-13, err
    return c


def train_fixture():
    """One TRAIN-mode step of the reference graph (trainer.py:206-229): ECAPA-TDNN forward with batch statistics,
    classifier, AAMLoss, backward (torch autograd through the shim).  Records loss, a few gradients, updated running stats."""
    W = o_ecapa.make_ecapa_weights(seed=1000, dtype=torch.float64)
    g = torch.Generator().manual_seed(77)
    B, T, S = 4, 61, 37
    f = torch.randn(B, T, 80, generator=g, dtype=torch.float64)
    f = f - f.mean(1, keepdim=True)
    labels = torch.randint(0, S, (B,), generator=g)
    Wc = (torch.rand(192, S, generator=g, dtype=torch.float64) * 2 - 1) * (6.0 / (192 + S)) ** 0.5
    model = EcapaTdnn(input_size=80)
    model.set_state_dict(W)
    clf = SpeakerIdentification(input_dim=192, num_speakers=S)
    clf.set_state_dict({"weight": Wc})
    model.train()
    out = clf(model(paddle.to_tensor(f)))
    crit = AAMLoss(margin=0.2, scale=32, label_smoothing=0.0)
    loss = crit(out, paddle.to_tensor(labels))
    loss.backward()
    d = {"feats": f.numpy(), "labels": labels.numpy(), "Wcls": Wc.numpy(), "loss": np.array(float(loss)),
         "logits": out["logits"].numpy()}
    params = dict(model.named_parameters())
    for k in ["blocks.0.conv.conv.weight", "blocks.0.norm.norm.weight", "blocks.2.res2net_block.blocks.3.conv.conv.weight",
              "blocks.3.se_block.conv1.conv.bias", "mfa.conv.conv.weight", "asp.tdnn.conv.conv.weight", "asp.conv.conv.weight",
              "asp_bn.norm.bias", "fc.conv.weight"]:
        d["grad_" + k] = tap_slice(params[k].grad)
        d["gradnorm_" + k] = np.array(float(params[k].grad.norm()))
    d["grad_classifier.weight"] = clf.weight.grad.numpy().copy()
    sd = model.state_dict()
    for k in ["blocks.0.norm.norm._mean", "blocks.0.norm.norm._variance", "mfa.norm.norm._variance", "asp_bn.norm._mean"]:
        d["stat_" + k] = sd[k].numpy().copy()
    return d


def sched_fixture():
    d = {}
    # cosine_decay_with_warmup (scheduler.py:6-40): the lr the optimizer sees at step 0,1,2,...
    for name, kw in {"a": dict(learning_rate=1e-3, step_per_epoch=7, fix_epoch=6, warmup_epoch=2, min_lr=1e-5),
                     "b": dict(learning_rate=0.01, step_per_epoch=3, fix_epoch=10, warmup_epoch=5, min_lr=0.0)}.items():
        s = cosine_decay_with_warmup(**kw)
        vals = []
        for _ in range(kw["step_per_epoch"] * kw["fix_epoch"] + 5):
            vals.append(s.get_lr())
            s.step()
        d["lr_" + name] = np.array(vals)

    class Crit:
        def update(self, margin):
            self.m = margin

    for name, kw in {"exp": dict(increase_start_epoch=3, fix_epoch=7, step_per_epoch=5, initial_margin=0.0, final_margin=0.3),
                     "lin": dict(increase_start_epoch=2, fix_epoch=4, step_per_epoch=4, initial_margin=0.1, final_margin=0.5,
                                 increase_type="linear")}.items():
        ms = MarginScheduler(criterion=Crit(), **kw)
        vals = []
        for _ in range(kw["fix_epoch"] * kw["step_per_epoch"] + 3):
            ms.step()
            vals.append(ms.get_margin())
        d["margin_" + name] = np.array(vals)
    return d


FIXTURES = {"ref_models.npz": models_fixture, "ref_head.npz": head_fixture, "ref_train.npz": train_fixture,
            "ref_sched.npz": sched_fixture}
DIGESTS = os.path.join(HERE, "ref_digests.json")


def array_digest(a):
    """dtype, shape and SHA-256 of the bytes of one array (same recipe in tests/test_oracle_vs_reference.py)."""
    a = np.ascontiguousarray(a)
    return {"dtype": a.dtype.str, "shape": list(a.shape), "sha256": hashlib.sha256(a.tobytes()).hexdigest()}


def main():
    check = "--check" in sys.argv
    bad = 0
    digests = {}
    for fn, make in FIXTURES.items():
        d = make()
        digests[fn] = {k: array_digest(d[k]) for k in sorted(d)}  # written with the fixtures; --check compares values instead
        path = os.path.join(HERE, fn)
        if check:
            old = np.load(path)
            assert sorted(old.files) == sorted(d), (fn, set(old.files) ^ set(d))
            err = max(float(np.abs(old[k] - d[k]).max()) for k in d)
            print(f"{fn}: {len(d)} arrays, max |committed - recomputed| = {err:.3e}")
            bad += err > 1e-12
        else:
            np.savez_compressed(path, **d)
            print(f"wrote {fn}: {len(d)} arrays, {os.path.getsize(path)} bytes")
    if not check:
        with open(DIGESTS, "w") as f:
            json.dump(digests, f, indent=1, sort_keys=True)
            f.write("\n")
        print(f"wrote {os.path.basename(DIGESTS)}")
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
