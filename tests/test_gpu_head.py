"""GPU: cosine scoring and the AAM head vs the oracle / golden vectors."""
import numpy as np
import pytest
import torch

from oracle import head as oh
from ppvector.loss.aamloss import AAMLoss
from ppvector.metric.cosine import cosine_matrix, cosine_pairlist
from ppvector.models.fc import SpeakerIdentification

pytestmark = pytest.mark.gpu

SCORE_TOL = 1e-4  # SURVEY.md §8(d) config 5: scores within 1e-4 absolute of the oracle


def test_cosine_matrix_golden(cuda, golden_dir):
    g = np.load(f"{golden_dir}/head_seed1000.npz")
    out = cosine_matrix(torch.from_numpy(g["cos_A"]).float().to(cuda), torch.from_numpy(g["cos_B"]).float().to(cuda))
    assert out.shape == (17, 23)
    assert np.abs(out.cpu().numpy() - g["cos_AB"]).max() < 1e-5


@pytest.mark.parametrize("M,N,D", [(1, 1, 192), (3, 1000, 192), (1000, 1000, 192), (257, 129, 256), (64, 50, 100)])
def test_cosine_matrix_shapes(cuda, M, N, D):
    g = torch.Generator().manual_seed(M + N + D)
    A, B = torch.randn(M, D, generator=g), torch.randn(N, D, generator=g) * 5
    out = cosine_matrix(A.to(cuda), B.to(cuda)).cpu().numpy()
    ref = oh.cosine_matrix(A.numpy(), B.numpy())
    assert np.abs(out - ref).max() < 1e-5 < SCORE_TOL


def test_cosine_properties_full_size(cuda):
    """config 5 size: 1000 x 1000 = 1e6 scores; self-similarity is 1, matrix is symmetric, scale invariant."""
    g = torch.Generator().manual_seed(5)
    E = torch.randn(1000, 192, generator=g).to(cuda)
    S = cosine_matrix(E, E)
    # split-bf16 (hi*hi + lo*hi + hi*lo) drops the lo*lo term: ~2^-18 relative, systematic on self-products
    assert (S.diagonal() - 1).abs().max().item() < 1e-5
    assert (S - S.t()).abs().max().item() < 1e-5
    S2 = cosine_matrix(E * 3.7, E * 0.01)
    assert (S - S2).abs().max().item() < 1e-5
    assert S.abs().max().item() <= 1 + 1e-5


def test_pairlist(cuda):
    g = torch.Generator().manual_seed(11)
    E = torch.randn(10000, 192, generator=g)
    idx = torch.randint(0, 10000, (100003, 2), generator=g, dtype=torch.int32)
    out = cosine_pairlist(E.to(cuda), idx).cpu().numpy()
    ref = oh.cosine_pairlist(E.numpy(), idx.numpy().astype(np.int64))
    assert np.abs(out - ref).max() < 2e-6
    assert cosine_pairlist(E.to(cuda), idx[:0]).numel() == 0
    # agrees with the matrix form
    Mx = cosine_matrix(E[:50].to(cuda), E[:50].to(cuda)).cpu().numpy()
    ii = np.stack(np.meshgrid(np.arange(50), np.arange(50), indexing="ij"), -1).reshape(-1, 2)
    pl = cosine_pairlist(E[:50].to(cuda), torch.from_numpy(ii.astype(np.int32))).cpu().numpy().reshape(50, 50)
    assert np.abs(pl - Mx).max() < 1e-5


@pytest.mark.parametrize("margin,ls", [(0.0, 0.0), (0.2, 0.0), (0.3, 0.1)])
def test_aam_golden(cuda, golden_dir, margin, ls):
    g = np.load(f"{golden_dir}/head_seed1000.npz")
    emb = torch.from_numpy(g["emb"]).float().to(cuda).requires_grad_(True)
    head = SpeakerIdentification(192, 157).to(cuda)
    with torch.no_grad():
        head.weight.copy_(torch.from_numpy(g["W"]).float())
    loss_fn = AAMLoss(margin=margin, scale=32, label_smoothing=ls)
    out = head(emb)
    assert np.abs(out["logits"].detach().cpu().numpy() - g["logits"]).max() < 2e-6
    loss = loss_fn(out, torch.from_numpy(g["labels"]).to(cuda))
    tag = f"m{margin}_ls{ls}"
    assert abs(loss.item() - float(g[f"loss_{tag}"])) < 2e-5 * max(1.0, abs(float(g[f"loss_{tag}"])))
    loss.backward()
    de, dw = emb.grad.cpu().numpy(), head.weight.grad.cpu().numpy()
    assert np.abs(de - g[f"demb_{tag}"]).max() < 1e-5 * max(1.0, np.abs(g[f"demb_{tag}"]).max())
    assert np.abs(dw - g[f"dW_{tag}"]).max() < 1e-5 * max(1.0, np.abs(g[f"dW_{tag}"]).max())


def test_aam_config_size_vs_autograd(cuda):
    """configs/*.yml: B=64, S=2796, D=192, margin scheduled up to 0.3, scale 32."""
    g = torch.Generator().manual_seed(1000)
    B, D, S = 64, 192, 2796
    emb = torch.randn(B, D, generator=g, dtype=torch.float64)
    W = (torch.rand(D, S, generator=g, dtype=torch.float64) * 2 - 1) * 0.05
    labels = torch.randint(0, S, (B,), generator=g)
    e_, w_ = emb.clone().requires_grad_(True), W.clone().requires_grad_(True)
    ref = oh.aam_loss(oh.cosine_logits(e_, w_), labels, margin=0.3, scale=32.0)
    ref.backward()
    head = SpeakerIdentification(D, S).to(cuda)
    with torch.no_grad():
        head.weight.copy_(W.float())
    x = emb.float().to(cuda).requires_grad_(True)
    loss = AAMLoss(margin=0.3, scale=32)(head(x), labels.to(cuda))
    loss.backward()
    assert abs(loss.item() - ref.item()) < 2e-5 * ref.item()
    assert (x.grad.cpu().double() - e_.grad).abs().max().item() < 1e-5 * e_.grad.abs().max().item() + 1e-9
    assert (head.weight.grad.cpu().double() - w_.grad).abs().max().item() < 1e-5 * w_.grad.abs().max().item() + 1e-9


@pytest.mark.parametrize("kind,margin,ls", [("AM", 0.2, 0.0), ("AM", 0.35, 0.1), ("ARM", 0.2, 0.0), ("ARM", 0.1, 0.1), ("CE", 0.0, 0.0), ("CE", 0.0, 0.1)])
def test_other_softmax_heads_match_the_reference_code(cuda, ref_head, kind, margin, ls):
    """AMLoss / ARMLoss / CELoss (ppvector/loss/amloss.py, armloss.py, celoss.py) on the fused CUDA head against what the REFERENCE's
    own loss classes computed (tests/golden/ref_head.npz, made by tests/golden/make_ref_fixtures.py): loss and both gradients."""
    from ppvector.loss import AMLoss, ARMLoss, CELoss
    from ppvector.models.fc import SpeakerIdentification
    g = ref_head
    emb = torch.from_numpy(g["emb"]).float().to(cuda).requires_grad_(True)
    clf = SpeakerIdentification(input_dim=192, num_speakers=g["W"].shape[1]).to(cuda)
    with torch.no_grad():
        clf.weight.copy_(torch.from_numpy(g["W"]).float())
    crit = {"AM": lambda: AMLoss(margin=margin, scale=30, label_smoothing=ls), "ARM": lambda: ARMLoss(margin=margin, scale=30, label_smoothing=ls),
            "CE": lambda: CELoss(label_smoothing=ls)}[kind]()
    loss = crit(clf(emb), torch.from_numpy(g["labels"]).to(cuda))
    loss.backward()
    tag = f"{kind}_m{margin}_ls{ls}"
    assert abs(loss.item() - float(g[f"loss_{tag}"])) < 2e-5 * max(1.0, abs(float(g[f"loss_{tag}"])))
    for got, want in ((emb.grad, g[f"demb_{tag}"]), (clf.weight.grad, g[f"dW_{tag}"])):
        want = torch.from_numpy(want)
        rel = (got.double().cpu() - want).norm() / want.norm()
        assert rel < 5e-5, (tag, rel)


@pytest.mark.parametrize("K,margin,ls,easy", [(3, 0.2, 0.0, False), (3, 0.3, 0.1, False), (2, 0.2, 0.0, True)])
def test_subcenter_loss_matches_the_reference_code(cuda, ref_head, K, margin, ls, easy):
    """SubCenterLoss (ppvector/loss/subcenterloss.py:33-54; classifier with K sub-centres per class, fc.py:33) on the fused CUDA head against
    the REFERENCE's own class (tests/golden/ref_head.npz): a class's cosine is the max over its K adjacent columns, the AAM margin rule on top,
    and only the winning sub-centre column receives the class's gradient."""
    from ppvector.loss import SubCenterLoss
    from ppvector.models.fc import SpeakerIdentification
    g = ref_head
    Sk = 156 // K
    emb = torch.from_numpy(g["emb"]).float().to(cuda).requires_grad_(True)
    clf = SpeakerIdentification(input_dim=192, num_speakers=Sk, K=K).to(cuda)
    with torch.no_grad():
        clf.weight.copy_(torch.from_numpy(g["W"][:, :156].copy()).float())
    crit = SubCenterLoss(margin=margin, scale=32, easy_margin=easy, K=K, label_smoothing=ls)
    loss = crit(clf(emb), (torch.from_numpy(g["labels"]) % Sk).to(cuda))
    loss.backward()
    tag = f"SUB_K{K}_m{margin}_ls{ls}_easy{int(easy)}"
    assert abs(loss.item() - float(g[f"loss_{tag}"])) < 2e-5 * max(1.0, abs(float(g[f"loss_{tag}"])))
    for got, want in ((emb.grad, g[f"demb_{tag}"]), (clf.weight.grad, g[f"dW_{tag}"])):
        want = torch.from_numpy(want)
        rel = (got.double().cpu() - want).norm() / want.norm()
        assert rel < 5e-5, (tag, rel)


@pytest.mark.parametrize("mt,margin,lam,t", [("C", 0.2, 0.7, 3), ("A", 0.15, 0.7, 3), ("C", 0.3, 0.5, 2)])
def test_sphereface2_matches_the_reference_code(cuda, ref_head, mt, margin, lam, t):
    """SphereFace2 (ppvector/loss/sphereface2.py:44-70: per-entry binary logistic loss over g(z) = 2 ((z+1)/2)^t - 1, margin types 'C' and 'A')
    on the fused CUDA head against the REFERENCE's own class (tests/golden/ref_head.npz): loss and both gradients."""
    from ppvector.loss import SphereFace2
    from ppvector.models.fc import SpeakerIdentification
    g = ref_head
    emb = torch.from_numpy(g["emb"]).float().to(cuda).requires_grad_(True)
    clf = SpeakerIdentification(input_dim=192, num_speakers=g["W"].shape[1]).to(cuda)
    with torch.no_grad():
        clf.weight.copy_(torch.from_numpy(g["W"]).float())
    loss = SphereFace2(margin=margin, scale=32.0, lanbuda=lam, t=t, margin_type=mt)(clf(emb), torch.from_numpy(g["labels"]).to(cuda))
    loss.backward()
    tag = f"SF2{mt}_m{margin}_l{lam}_t{t}"
    assert abs(loss.item() - float(g[f"loss_{tag}"])) < 2e-5 * max(1.0, abs(float(g[f"loss_{tag}"])))
    for got, want in ((emb.grad, g[f"demb_{tag}"]), (clf.weight.grad, g[f"dW_{tag}"])):
        want = torch.from_numpy(want)
        rel = (got.double().cpu() - want).norm() / want.norm()
        assert rel < 5e-5, (tag, rel)
