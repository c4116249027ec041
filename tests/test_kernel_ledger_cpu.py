"""Without a GPU: (a) the kernel ledger names exactly the in-scope kernels of the built library, and its cases are
consistent with it; (b) the elementwise comparator of tests/kernel_ledger.py flags local faults of a convolution that
the older max-abs metric lets through, and passes honest rounding."""
import os
import shutil
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import kernel_ledger as KL  # noqa: E402

LIB = os.path.join(KL.PKG, "unetb200", "libunetb200.so")


def _cuobjdump():
    p = shutil.which("cuobjdump")
    if p is None and os.path.isfile("/usr/local/cuda/bin/cuobjdump"):
        p = "/usr/local/cuda/bin/cuobjdump"
    return p


@pytest.mark.skipif(_cuobjdump() is None or shutil.which("c++filt") is None or not os.path.isfile(LIB),
                    reason="needs cuobjdump, c++filt and a built libunetb200.so")
def test_ledger_names_every_in_scope_kernel_of_the_library():
    sass = subprocess.run([_cuobjdump(), "-sass", LIB], capture_output=True, text=True, check=True).stdout
    mangled = [ln.split("Function :", 1)[1].strip() for ln in sass.splitlines() if "Function :" in ln]
    names = subprocess.run(["c++filt"], input="\n".join(mangled), capture_output=True, text=True,
                           check=True).stdout.splitlines()
    names = {KL.normalise(n) for n in names}
    unclassified = sorted(n for n in names if KL.base(n) not in KL.SCOPE_BASES | KL.OUT_OF_SCOPE_BASES)
    assert not unclassified, f"kernels of a new kind: add them to SCOPE_BASES (and the ledger) or OUT_OF_SCOPE_BASES: {unclassified}"
    lib_in = {n for n in names if KL.in_scope(n)}
    missing = sorted(lib_in - set(KL.LEDGER))
    stale = sorted(set(KL.LEDGER) - lib_in)
    assert not missing, f"instantiations without a ledger entry: {missing}"
    assert not stale, f"ledger entries the library does not contain: {stale}"
    kinds = {"cases": 0, "env": 0, "unreachable": 0}
    for e in KL.LEDGER.values():
        kinds[KL.entry_kind(e)] += 1
    print(f"\n{len(lib_in)} in-scope kernel instantiations of {len(names)}: {kinds}")


def test_ledger_and_cases_agree():
    ids = {c.id: c for c in KL.CASES}
    assert len(ids) == len(KL.CASES), "case ids must be unique"
    listed = set()
    for k, e in KL.LEDGER.items():
        kind = KL.entry_kind(e)
        assert KL.in_scope(k), k
        if kind == "unreachable":
            assert isinstance(e[1], str) and e[1], k
            continue
        cases = KL.entry_cases(e)
        assert cases, f"{k}: no case"
        for cid in cases:
            assert cid in ids, f"{k}: unknown case {cid}"
            listed.add(cid)
            if kind == "env":
                assert ids[cid].env != "default" and KL.ENV_SETS[ids[cid].env] == e[1], \
                    f"{k}: case {cid} does not run under the switches {e[1]}"
        if kind == "cases":
            assert any(ids[c].env == "default" for c in cases), f"{k}: reachable without switches needs a default case"
    # every case launches at least one in-scope kernel, so each one is named by the ledger
    assert set(ids) == listed, f"cases the ledger does not name: {sorted(set(ids) - listed)}"


# ------------------------------------------------------------------------------------------------
# (b) the comparator on synthetic faults of an fp64 reference
# ------------------------------------------------------------------------------------------------
def _tf32(t):
    """round fp32 to TF32 (10 explicit mantissa bits), to nearest"""
    v = t.float().contiguous().view(torch.int32)
    return ((v + 0x1000) & ~0x1FFF).view(torch.float32)


def _conv_case(seed=0, B=2, Ci=128, Co=16, H=20, W=18):
    g = torch.Generator().manual_seed(seed)
    x = KL.rq(torch.randn(B, Ci, H, W, generator=g), torch.bfloat16)
    w = KL.rq(torch.randn(Co, Ci, 3, 3, generator=g) / (3 * Ci ** 0.5), torch.bfloat16)
    ref, A = KL.ref_conv3x3(x, w)
    return x, w, ref, A, 9 * Ci


def _faults():
    x, w, ref, A, K = _conv_case()
    B, Co, H, W = ref.shape
    out = {}
    # one tap dropped for one input channel at a border pixel (row 0, column 5: the tap above reads padding, the
    # one to the left is in the image); the channel whose product there is largest -- a product below the output's
    # rounding unit is invisible to any comparison of a bf16 result
    d = ref.clone()
    c = int((x[1, :, 0, 4].double() * w[3, :, 1, 0].double()).abs().argmax())
    d[1, 3, 0, 5] -= x[1, c, 0, 4].double() * w[3, c, 1, 0].double()
    out["tap_dropped_at_border"] = (d, ref, A, K, "bf16")
    # the halo row of the last 16-row tile read one row too high: tap dy = -1 of output row 16 reads input row 14
    d = ref.clone()
    wrong = F.conv2d(x[:, :, 14:15].double(), w[:, :, 0:1].double(), padding=(0, 1))
    right = F.conv2d(x[:, :, 15:16].double(), w[:, :, 0:1].double(), padding=(0, 1))
    d[:, :, 16:17] += wrong - right
    out["last_tile_halo_row_shifted"] = (d, ref, A, K, "bf16")
    # the last 64-channel chunk of the reduction left out of the accumulation
    xc = x.clone()
    xc[:, -64:] = 0
    d = F.conv2d(xc.double(), w.double(), padding=1)
    out["last_channel_chunk_zeroed"] = (d, ref, A, K, "bf16")
    # one pixel missing from the BatchNorm statistics
    y = KL.rq(ref.float(), torch.bfloat16)
    s, sA = KL.ref_stats(y)
    ym = y.clone()
    ym[1, :, H - 1, W - 1] = 0
    out["stats_pixel_missing"] = (KL.ref_stats(ym)[0], s, sA, B * H * W, "acc32")
    # two OutConv classes swapped
    g = torch.Generator().manual_seed(1)
    xo = KL.rq(torch.relu(torch.randn(2, 64, 9, 7, generator=g)), torch.bfloat16)
    wo = KL.rq(torch.randn(5, 64, generator=g) * 0.3, torch.bfloat16)
    bo = KL.rq(torch.randn(5, generator=g), torch.bfloat16)
    lo, lA = KL.ref_outconv(xo, wo, bo)
    out["outconv_classes_swapped"] = (lo[:, [0, 1, 3, 2, 4]], lo, lA, 65, "bf16")
    return out


def test_comparator_flags_local_faults():
    let_through = []
    for name, (dev, ref, A, K, comp) in _faults().items():
        e = KL.err_over_bound(dev, ref, A, K, comp)
        assert e > 1.0, f"{name}: err/bound {e:.3g} not flagged"
        if KL.rel(dev, ref) <= KL.REL_TOL[comp]:
            let_through.append(name)
    print(f"\nfaults the max-abs metric rel() lets through at its tolerance: {let_through}")


def test_comparator_passes_honest_rounding():
    x, w, ref, A, K = _conv_case(seed=3)
    # bf16 storage of an exact fp32-accumulated result
    assert KL.err_over_bound(KL.rq(ref.float(), torch.bfloat16), ref, A, K, "bf16") <= 1.0
    # TF32 operands (fp32 tensors), fp32 storage
    g = torch.Generator().manual_seed(4)
    xf, wf = torch.randn(2, 64, 12, 10, generator=g), torch.randn(32, 64, 3, 3, generator=g) / 24
    r32, A32 = KL.ref_conv3x3(xf, wf)
    dev = F.conv2d(_tf32(xf).double(), _tf32(wf).double(), padding=1).float()
    assert KL.err_over_bound(dev, r32, A32, 9 * 64, "tf32") <= 1.0
    # fp32 accumulation in a different order (wgrad: K = B*H*W products per element)
    gy = KL.rq(torch.randn(2, 32, 12, 10, generator=g), torch.bfloat16)
    xb = KL.rq(xf, torch.bfloat16)
    dw, dA = KL.ref_wgrad3x3(xb, gy)
    dev = torch.nn.grad.conv2d_weight(xb, dw.shape, gy, padding=1)            # fp32
    assert KL.err_over_bound(dev, dw, dA, 2 * 12 * 10, "acc32") <= 1.0
