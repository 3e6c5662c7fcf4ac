"""CPU: the oracle restatement (oracle/dvc_oracle.py) against the vectors generated from the real
reference (tests/golden/*.npz, written by oracle/make_golden.py).  In the container that generated
them the agreement is bit-exact (tests/golden/PIN_REPORT.txt), and it is demanded wherever torch runs the same CPU
kernels; elsewhere the CPU's conv/GEMM kernels may differ in summation order, so the gate is the fp32-noise-floor
metric of SURVEY.md §8c."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import dvc_oracle as O
from oracle.make_golden import contextual_loss_maps

CASES = ["small_32x48", "padbranch_40x64", "softmax_32x64", "softmax5_48x48", "batch2_32x32"]


def _run(sds, g):
    IA, IB, last = (torch.from_numpy(g[k]) for k in ("IA_lab", "IB_lab", "IA_last_lab"))
    ex = {}
    with torch.no_grad():
        fB = O.exemplar_features(sds["vgg"], IB)
        ab, warped, sim, fA = O.frame_colorization(sds, IA, IB, last, fB, temperature=float(g["temperature"]), extras=ex)
    return ab, warped, sim, fA, fB, ex


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_reference_vectors(sds, name):
    g = load_golden(name)
    ab, warped, sim, fA, fB, ex = _run(sds, g)
    floor = np.abs(g["ab32"].astype(np.float64) - g["ab64"]).max()
    err = np.abs(ab.numpy().astype(np.float64) - g["ab64"]).max()
    assert err <= max(1e-3, 2.0 * floor), (err, floor)
    assert np.abs(sim.numpy()[:, :, ::4, ::4] - g["sim32"]).max() < 2e-5
    if float(g["temperature"]) < 1e-9:
        # one-hot warp: identical argmax wherever the fp64 top-2 gap is not a numerical tie
        clear = g["gap64"] > 1e-5
        assert (ex["argmax"].numpy()[clear] == g["argmax64"][clear]).all()
        B, _, h, w = g["warped32"].shape
        mine = warped.numpy()[:, :, ::4, ::4].reshape(B, 3, -1)
        ref = g["warped32"].reshape(B, 3, -1)
        m = np.broadcast_to(clear[:, None, :], mine.shape)
        assert np.array_equal(mine[m], ref[m])
    else:
        assert np.abs(warped.numpy()[:, :, ::4, ::4] - g["warped64"]).max() < 5e-3


def test_oracle_intermediates_small(sds):
    g = load_golden("small_32x48")
    ab, warped, sim, fA, fB, ex = _run(sds, g)
    for i, k in enumerate(["r12", "r22", "r32", "r42", "r52"]):
        for side, f in (("A", fA), ("B", fB)):
            ref = g[f"{side}_{k}"]
            assert np.abs(f[i].numpy() - ref).max() <= 1e-4 * np.abs(ref).max() + 1e-12
    assert np.abs(ex["theta_hat"].numpy() - g["theta_hat32"]).max() < 1e-5
    assert np.abs(ex["phi_hat"].numpy() - g["phi_hat32"]).max() < 1e-5
    assert np.abs(ex["V"].numpy() - g["V32"]).max() < 1e-5


def test_oracle_clip_recurrence(sds):
    """test.py:76-96: with teacher forcing (the reference's own previous prediction as `last`) every frame
    matches; the free-running recurrence is chaotic with random weights (see DESIGN.md) and is checked
    only for plumbing (first frame starts from zeros)."""
    g = load_golden("clip3_32x48")
    frames, IB, ref = torch.from_numpy(g["frames_lab"]), torch.from_numpy(g["IB_lab"]), torch.from_numpy(g["ab32"])
    with torch.no_grad():
        fB = O.exemplar_features(sds["vgg"], IB)
        last = torch.zeros_like(frames[0:1])
        for t in range(frames.shape[0]):
            ab, _, _, _ = O.frame_colorization(sds, frames[t:t + 1], IB, last, fB)
            assert (ab - ref[t:t + 1]).abs().max() < 5e-3
            last = torch.cat((frames[t:t + 1, 0:1], ref[t:t + 1]), 1)


def test_chunked_correlation_equals_unchunked():
    g = torch.Generator().manual_seed(3)
    th = torch.nn.functional.normalize(torch.randn(1, 256, 300, generator=g), dim=1)
    ph = torch.nn.functional.normalize(torch.randn(1, 256, 280, generator=g), dim=1)
    V = torch.randn(1, 280, 3, generator=g)
    for T in (1e-10, 0.01):
        y1, s1 = O.corr_softmax_warp(th, ph, V, T, row_chunk=4096)
        y2, s2 = O.corr_softmax_warp(th, ph, V, T, row_chunk=64)
        assert torch.allclose(y1, y2, atol=1e-5) and torch.allclose(s1, s2, atol=1e-6)


@pytest.fixture
def golden_arithmetic():
    """torch's CPU kernels as oracle/make_golden.py ran them: 8 intra-op threads, AVX-512 kernels.  The reference's fp32
    outputs are reproduced bit for bit only with the same split of every sum."""
    if torch.backends.cpu.get_cpu_capability() != "AVX512":
        pytest.skip("bit-exact comparison needs the AVX-512 CPU kernels the golden vectors were computed with")
    n = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize("name", CASES)
def test_oracle_bit_exact_against_reference_outputs(sds, golden_arithmetic, name):
    """The restatement runs the reference's torch ops in the reference's order: its fp32 outputs equal the stored fp32
    outputs of the unmodified reference (ab in full, warped colour and similarity on the stored 4x subsample)."""
    g = load_golden(name)
    ab, warped, sim, fA, fB, ex = _run(sds, g)
    assert np.array_equal(ab.numpy(), g["ab32"])
    assert np.array_equal(warped.numpy()[:, :, ::4, ::4], g["warped32"])
    assert np.array_equal(sim.numpy()[:, :, ::4, ::4], g["sim32"])


def test_lab_to_rgb8_oracle_anchors():
    """The float64 output conversion (utils/util.py:140-151) has no pinned reference here (skimage is absent), so it is
    anchored on (a) closed-form values and (b) the reference's own fp32 torch twin `tensor_lab2rgb` (util.py:379-414),
    which the golden vectors pin bit-exactly: same formula, so the uint8 results agree up to one level where the fp32
    and float64 evaluations straddle a truncation boundary."""
    l = torch.tensor([-50.0, 0.0, 50.0, 3.0]).view(4, 1, 1, 1)
    ab = torch.zeros(4, 2, 1, 1)
    got = O.lab_to_rgb8(l, ab)[:, 0, 0, :]
    assert got[0].tolist() == [0, 0, 0]              # L = 0: black
    assert min(got[2].tolist()) >= 254               # L = 100: white (a channel just below 1.0 truncates to 254)
    assert got[1].tolist() == [118, 118, 118]        # L = 50: Y = 0.1842 -> sRGB 0.4663 -> 118.9
    g = torch.Generator().manual_seed(5)
    l = torch.rand(2, 1, 24, 40, generator=g) * 100 - 50
    ab = (torch.rand(2, 2, 24, 40, generator=g) * 2 - 1) * 100
    twin = O.tensor_lab2rgb(torch.cat((l + 50.0, ab), 1))  # [n,3,h,w] in [0,1]
    twin8 = (twin.clamp(0, 1) * 255).to(torch.uint8).permute(0, 2, 3, 1)
    d = (O.lab_to_rgb8(l, ab).int() - twin8.int()).abs()
    assert int(d.max()) <= 1 and float((d > 0).float().mean()) < 2e-2


def test_rgb8_to_lab_oracle_anchors():
    """Closed-form anchors of the (unpinned, skimage-restating) ingest conversion and its inverse."""
    rgb = torch.tensor([[0, 0, 0], [255, 255, 255], [255, 0, 0]], dtype=torch.uint8).view(1, 1, 3, 3)
    lab = O.rgb8_to_lab(rgb)[0, :, 0, :]  # [3 channels, 3 pixels]
    assert abs(float(lab[0, 0]) + 50.0) < 1e-4 and abs(float(lab[1, 0])) < 1e-4            # black: L = 0
    assert abs(float(lab[0, 1]) - 50.0) < 1e-2 and abs(float(lab[1, 1])) < 1e-2            # white: L = 100, a = b = 0
    assert abs(float(lab[0, 2]) + 50.0 - 53.24) < 0.02 and abs(float(lab[1, 2]) - 80.09) < 0.05  # sRGB red: (53.24, 80.09, 67.20)
    assert abs(float(lab[2, 2]) - 67.20) < 0.05
    g = torch.Generator().manual_seed(8)
    rgb = torch.randint(0, 256, (1, 20, 30, 3), generator=g, dtype=torch.uint8)
    lab = O.rgb8_to_lab(rgb)
    back = O.lab_to_rgb8(lab[:, 0:1], lab[:, 1:3])
    assert int((back.int() - rgb.int()).abs().max()) <= 1


def test_contextual_loss_restatement_is_the_reference(golden_arithmetic):
    """oracle.contextual_loss_forward == models/ContextualLoss.py: ContextualLoss_forward of the unmodified reference, bit for
    bit (same torch ops in the same order), on seeded feature maps of several depths.  tests/golden/contextual_loss.npz holds
    the reference's values; they were written through this restatement, unchanged since it last matched the reference
    module bit for bit (oracle/make_golden.py writes them from the module itself)."""
    gold = load_golden("contextual_loss")
    for key, X, Y, centering in contextual_loss_maps():
        with torch.no_grad():
            mine = O.contextual_loss_forward(X, Y, 0.1, centering)
        assert np.array_equal(mine.numpy(), gold[key]), (key, mine, gold[key])
