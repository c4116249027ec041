"""nn.SyncBatchNorm on the UNet (unetb200.ddp peer groups, csrc/bn_sync.cu).

CPU: convert_sync_batchnorm keeps the state_dict surface, the statistics arena counts the converted layers, and the
process-group / momentum validation.  GPU: a converted model without a group of more than one rank runs the per-replica
path bit for bit with no exchange launch; with two GPUs tests/syncbn_worker.py checks the synchronised path."""
import os
import socket
import subprocess
import sys

import pytest
import torch
import torch.distributed as dist
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))


def _converted(*args):
    import unet
    torch.manual_seed(0)
    return nn.SyncBatchNorm.convert_sync_batchnorm(unet.UNet(*args))


def test_converted_model_keeps_its_state_dict_keys():
    import unet
    torch.manual_seed(0)
    plain = unet.UNet(1, 3)
    conv = _converted(1, 3)
    assert list(conv.state_dict()) == list(plain.state_dict()) and len(conv.state_dict()) == 118
    assert sum(isinstance(m, nn.SyncBatchNorm) for m in conv.modules()) == 18
    assert not any(type(m) is nn.BatchNorm2d for m in conv.modules())
    for k, v in plain.state_dict().items():
        assert torch.equal(conv.state_dict()[k], v), k


def test_statistics_arena_counts_converted_layers():
    import unet
    torch.manual_seed(0)
    n = unet.UNet(1, 3).bn_arena_doubles()
    assert n == 2 * sum(2 * c for c in (64, 128, 256, 512, 1024, 512, 256, 128, 64))
    assert _converted(1, 3).bn_arena_doubles() == n


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.fixture
def gloo_world1():
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(_free_port())
    dist.init_process_group("gloo", rank=0, world_size=1)
    try:
        yield
    finally:
        dist.destroy_process_group()


def test_process_group_and_momentum_validation(gloo_world1):
    from unetb200 import ddp
    from unetb200 import functional as UF
    m = _converted(1, 2)
    assert ddp.sync_bn_process_group(m, training=True) == (18, None)
    other = dist.new_group([0])
    m.up2.conv.double_conv[1].process_group = other
    with pytest.raises(ValueError, match="same process group"):
        ddp.sync_bn_process_group(m)
    for mod in m.modules():
        if isinstance(mod, nn.SyncBatchNorm):
            mod.process_group = other
    assert ddp.sync_bn_process_group(m) == (18, other)
    m.inc.double_conv[4].momentum = None
    assert ddp.sync_bn_process_group(m, training=False) == (18, other)
    with pytest.raises(ValueError, match="momentum=None"):
        ddp.sync_bn_process_group(m, training=True)
    # a group of one rank, eval mode and BatchNorm2d holders all take the per-replica path
    bn = m.inc.double_conv[1]
    cpu = torch.device("cpu")
    assert UF.sync_peer(bn, True, cpu) is None and UF.sync_peer(bn, False, cpu) is None
    assert UF.sync_peer(nn.BatchNorm2d(4), True, cpu) is None
    assert not ddp._PEER_GROUPS


@pytest.mark.gpu
def test_converted_model_without_group_is_bit_identical():
    """No process group: the converted model computes exactly what the BatchNorm2d model computes, with the same
    launches (no exchange)."""
    import unet
    from oracle import unet_oracle as O
    from unetb200 import losses as UL
    from unetb200 import ops
    assert not (dist.is_available() and dist.is_initialized())
    dev = torch.device("cuda:0")
    st = O.build_state(1, 3, False, seed=0)
    img, msk = O.synthetic_batch(2, 1, 3, 64, 64)
    x = img.to(dev).contiguous(memory_format=torch.channels_last)
    t = msk.to(dev)
    out = {}
    for name in ("plain", "sync"):
        torch.manual_seed(0)
        m = unet.UNet(1, 3)
        if name == "sync":
            m = nn.SyncBatchNorm.convert_sync_batchnorm(m)
        m.load_state_dict(st)
        m = m.to(dev).to(memory_format=torch.channels_last).train()
        with ops.profile() as rec:
            with torch.autocast("cuda"):
                logits = m(x)
                loss = UL.training_criterion(logits, t, boundary_coeff=0.2)
            loss.backward()
        torch.cuda.synchronize()
        m.eval()
        with torch.no_grad():
            ev = m(x)
        torch.cuda.synchronize()
        out[name] = (logits.detach().clone(), {k: p.grad.clone() for k, p in m.named_parameters()},
                     {k: v.clone() for k, v in m.state_dict().items()}, [r[0] for r in rec], ev)
    a, b = out["plain"], out["sync"]
    assert torch.equal(a[0], b[0])
    assert a[1].keys() == b[1].keys() and all(torch.equal(a[1][k], b[1][k]) for k in a[1])
    assert a[2].keys() == b[2].keys() and all(torch.equal(a[2][k], b[2][k]) for k in a[2])
    assert a[3] == b[3] and not any("sync" in n for n in b[3])
    assert torch.equal(a[4], b[4])


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_syncbn_world2():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(_free_port()), os.path.join(HERE, "syncbn_worker.py")]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    sys.stdout.write(p.stdout[-6000:])
    sys.stderr.write(p.stderr[-6000:])
    assert p.returncode == 0, "SyncBatchNorm worker failed"
    assert "RANK 0: OK" in p.stdout and "RANK 1: OK" in p.stdout
