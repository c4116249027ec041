"""CPU: oracle/io_oracle.py (input pipeline, evaluate / predict tails) against the fixtures generated from the
reference itself by tests/golden/make_golden_io.py, plus the host-side argument logic of unetb200.data /
unetb200.eval_tail.  Never needs the reference, no compute calls into the CUDA library."""
import os

import numpy as np
import pytest
import torch

from oracle import io_oracle as IO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def gio():
    from gpu_io_checks import load_golden_io
    return load_golden_io()


def test_pipeline_matches_reference_arrays(gio):
    assert len(gio["pipeline"]) == 16
    for c in gio["pipeline"]:
        img, msk = IO.make_batch([c["img"].numpy()], [c["msk"].numpy()], [c["k"]])
        assert img.dtype == torch.float32 and msk.dtype == torch.int64
        assert torch.equal(img[0], c["out_img"]), (c["tag"], c["k"])
        assert torch.equal(msk[0], c["out_msk"]), (c["tag"], c["k"])
    # the /255 branch is data dependent (data_loading.py:86): an image without a value > 1 is NOT scaled
    lo = [c for c in gio["pipeline"] if c["tag"] == "gray_binary_24x24"][0]
    assert lo["out_img"].max().item() == 1.0 and set(lo["out_img"].unique().tolist()) <= {0.0, 1.0}


def test_rotation_is_counter_clockwise_quarter_turns():
    a = np.arange(6, dtype=np.uint8).reshape(2, 3)
    assert IO.rotate(a, 1).tolist() == [[2, 5], [1, 4], [0, 3]]
    assert IO.rotate(a, 2).tolist() == [[5, 4, 3], [2, 1, 0]]
    assert IO.rotate(a, 3).tolist() == [[3, 0], [4, 1], [5, 2]]


def test_evaluate_tails(gio):
    for c in gio["eval_mc"]:
        idx, dice, counts = IO.eval_multiclass(c["logits"], c["true"], c["c"])
        assert torch.equal(idx, c["idx"]) and torch.equal(dice, c["dice"]), c["tag"]
        assert counts.shape == (c["logits"].shape[0], 3)
    empty = [c for c in gio["eval_mc"] if c["tag"] == "mc_empty"][0]
    assert empty["dice"].item() == 1.0                     # sets_sum == 0 -> inter -> eps/eps
    for c in gio["eval_bin"]:
        binary, dice, _ = IO.eval_binary(c["logits"], c["true"])
        assert torch.equal(binary, c["binary"]) and torch.equal(dice, c["dice"]), c["tag"]
    with pytest.raises(AssertionError):
        IO.eval_binary(torch.zeros(1, 1, 4, 4), torch.full((1, 4, 4), 5.0))


def test_predict_tail(gio):
    for c in gio["predict"]:
        assert torch.equal(IO.predict_tail(c["logits"], c["size"]), c["idx"]), c["tag"]
        ex = IO.resize_argmax_exact(c["logits"], c["size"])
        agree = (ex == c["idx"]).float().mean().item()
        assert agree >= (1.0 if c["tag"].startswith("same") else 0.999), (c["tag"], agree)


def test_host_argument_logic():
    from unetb200 import data, eval_tail
    assert data.check_rotations(None, 2, 4, 6) == (None, False)
    assert data.check_rotations([1, 3], 2, 4, 6) == ([1, 3], True)
    assert data.check_rotations([0, 2], 2, 4, 6) == ([0, 2], False)
    assert data.check_rotations([0, 1, 6, 7], 4, 8, 8) == ([0, 1, 2, 3], False)      # square: any mix stacks
    with pytest.raises(ValueError):
        data.check_rotations([0, 1], 2, 4, 6)
    with pytest.raises(ValueError):
        data.check_rotations([0], 2, 4, 4)
    with pytest.raises(ValueError):
        data._as_u8_batch([np.zeros((4, 4), np.uint8), np.zeros((4, 5), np.uint8)], "t")
    with pytest.raises(ValueError):
        data._as_u8_batch(np.zeros((1, 4, 4), np.float32), "t")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        data.preprocess_batch([np.zeros((4, 4), np.uint8)], device="cpu")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        eval_tail.argmax_class_dice(torch.zeros(1, 3, 4, 4), torch.zeros(1, 4, 4))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        eval_tail.resize_argmax(torch.zeros(1, 3, 4, 4), (8, 8))
    with pytest.raises(ValueError):
        eval_tail.binary_dice(torch.zeros(1, 2, 4, 4), torch.zeros(1, 4, 4))


def test_evaluate_host_logic(monkeypatch):
    """unetb200.eval_tail.evaluate's control flow (per-batch scores, post-processing leg, min rule, return triple,
    eval()/train() switching) with the device tails replaced by the oracle: it must reproduce evaluate.py:12-173."""
    from unetb200 import eval_tail, losses

    def fake_mc(mask_pred, mask_true, c=2, index_dtype=torch.int64, epsilon=1e-6):
        idx, dice, counts = IO.eval_multiclass(mask_pred.float(), mask_true.float(), c)
        return idx.to(index_dtype), dice, counts

    def fake_bin(mask_pred, mask_true, index_dtype=torch.uint8, epsilon=1e-6):
        binary, dice, counts = IO.eval_binary(mask_pred.float(), mask_true.float())
        return binary.to(index_dtype), dice, counts
    monkeypatch.setattr(eval_tail, "argmax_class_dice", fake_mc)
    monkeypatch.setattr(eval_tail, "binary_dice", fake_bin)
    monkeypatch.setattr(losses, "dice_coeff", IO.dice_coeff)

    class Net(torch.nn.Module):
        def __init__(self, n_classes):
            super().__init__()
            self.n_classes = n_classes
            self.conv = torch.nn.Conv2d(1, n_classes, 3, padding=1)

        def forward(self, x):
            return self.conv(x)

    def erode(m):                                   # a stand-in for utils.post_process.postprocess_mask
        out = m.copy()
        out[::2] = 0
        return out

    dev = torch.device("cpu")
    for ncls in (3, 1):
        torch.manual_seed(ncls)
        net = Net(ncls).train()
        g = torch.Generator().manual_seed(5)
        batches = [{"image": torch.rand(2, 1, 16, 16, generator=g),
                    "mask": torch.randint(0, 3 if ncls > 1 else 4, (2, 16, 16), generator=g)} for _ in range(3)]
        # literal restatement of the reference loop
        orig, post = [], []
        with torch.inference_mode():
            net.eval()
            for b in batches:
                lg = net(b["image"])
                if ncls == 1:
                    binary, d, _ = IO.eval_binary(lg, b["mask"].float())
                    orig.append(d.item())
                    pp = torch.stack([torch.from_numpy((erode(m.numpy().astype(np.uint8) * 255) // 255).astype(np.float32))
                                      for m in binary])
                    true = b["mask"].float() // 2
                    post.append(IO.dice_coeff(pp, true, reduce_batch_first=False).item())
                else:
                    idx, d, _ = IO.eval_multiclass(lg, b["mask"].float(), 2)
                    orig.append(d.item())
                    pp = torch.stack([torch.from_numpy(erode(m.numpy().astype(np.uint8))) for m in idx])
                    post.append(IO.dice_coeff((pp == 2).float(), (b["mask"] == 2).float(), reduce_batch_first=False).item())
            net.train()
        got = eval_tail.evaluate(net, batches, dev, amp=False, postprocess=True, postprocess_fn=erode)
        assert net.training
        assert abs(got[0] - sum(orig) / 3) < 1e-6 and abs(got[1] - sum(post) / 3) < 1e-6
        want_min = min(min(o, p) for o, p in zip(orig, post)) if ncls == 1 else min(orig)     # evaluate.py:85 vs :121
        assert abs(got[2] - want_min) < 1e-6
        got = eval_tail.evaluate(net, batches, dev, amp=False, postprocess=False)
        assert got[1] == got[0] and abs(got[2] - min(orig)) < 1e-6                            # evaluate.py:169-170
    assert eval_tail.evaluate(Net(3), [], dev, amp=False) == (0, 0, 10)
    with pytest.raises(ValueError):
        eval_tail.evaluate(Net(3), [], dev, amp=False, postprocess=True)
    # epoch_pred_dir: the PNGs of evaluate.py:92-107 / :146-166 (0 / 128 / 255 for classes 0 / 1 / 2; 0 / 255 binary)
    import tempfile
    from PIL import Image
    for ncls in (3, 1):
        torch.manual_seed(ncls)
        net = Net(ncls)
        with tempfile.TemporaryDirectory() as td:
            eval_tail.evaluate(net, batches, dev, amp=False, epoch_pred_dir=td, postprocess=True, postprocess_fn=erode)
            names = sorted(os.listdir(td))
            assert names == ["postprocessed"] + [f"pred_batch{b}_sample{i}.png" for b in range(3) for i in range(2)]
            assert sorted(os.listdir(os.path.join(td, "postprocessed"))) == names[1:]
            with torch.inference_mode():
                lg = net.eval()(batches[1]["image"])
            want = (torch.sigmoid(lg[1, 0]) > 0.5).numpy().astype(np.uint8) * 255 if ncls == 1 else \
                np.array([0, 128, 255], dtype=np.uint8)[lg[1].argmax(0).numpy()]
            assert np.array_equal(np.asarray(Image.open(os.path.join(td, "pred_batch1_sample1.png"))), want)


def test_oracle_properties():
    """Size-independent properties the GPU full-size gates rely on, checked on the oracle itself."""
    rng = np.random.default_rng(1)
    a = rng.integers(0, 256, size=(5, 7, 3), dtype=np.uint8)
    for k in range(4):
        assert np.array_equal(IO.rotate(IO.rotate(a, k), 4 - k), a)
        assert np.array_equal(IO.rotate(a, k + 4), IO.rotate(a, k))
    imgs = rng.integers(0, 256, size=(4, 6, 6), dtype=np.uint8)
    msks = np.array([0, 128, 255], dtype=np.uint8)[rng.integers(0, 3, size=(4, 6, 6))]
    base_i, base_m = IO.make_batch(list(imgs), list(msks), [0] * 4)
    rot_i, rot_m = IO.make_batch(list(imgs), list(msks), [0, 1, 2, 3])
    for b in range(4):
        assert torch.equal(rot_i[b], torch.rot90(base_i[b], b, dims=(1, 2)))
        assert torch.equal(rot_m[b], torch.rot90(base_m[b], b, dims=(0, 1)))
    assert base_i.max() <= 1.0 and set(base_m.unique().tolist()) <= {0, 1, 2}
    g = torch.Generator().manual_seed(2)
    lg = torch.randn(3, 4, 9, 11, generator=g)
    true = lg.argmax(1).float()
    idx, dice, counts = IO.eval_multiclass(lg, true, 2)
    assert abs(dice.item() - 1.0) < 1e-6                        # prediction == truth
    assert (counts[:, 0] <= counts[:, 1]).all() and (counts[:, 0] <= counts[:, 2]).all()
    assert torch.equal(IO.resize_argmax_exact(lg, (9, 11)), idx)  # identity resize is the plain argmax
    assert torch.equal(IO.predict_tail(lg, (9, 11)), idx)
